"""Import the REAL reference's NumPy modules (path (iii) + the sampler) with tensorflow / igraph stubbed.

Only usable where OPENEA_REFERENCE names a checkout of the original project.  Used by tests/golden/make_golden.py
and by CPU tests run with OPENEA_REFERENCE set to record the golden results the tests compare with
(tests/helpers.ReferenceRecord).  TEST INFRASTRUCTURE ONLY.
"""
import importlib
import os
import sys
import types

REF_SRC = os.path.join(os.environ.get("OPENEA_REFERENCE", ""), "src")


def available():
    return bool(os.environ.get("OPENEA_REFERENCE")) and os.path.isdir(os.path.join(REF_SRC, "openea"))


def load():
    """Returns a namespace with the reference modules: similarity, alignment, evaluation, batch, finder, read, util."""
    if not available():
        raise RuntimeError("set OPENEA_REFERENCE to a checkout of the original OpenEA")
    saved = {k: sys.modules.get(k) for k in ("tensorflow", "igraph", "openea")}
    saved_sub = {k: v for k, v in sys.modules.items() if k.startswith("openea.")}
    for k in saved_sub:
        del sys.modules[k]
    sys.modules["tensorflow"] = types.ModuleType("tensorflow")
    sys.modules["igraph"] = types.ModuleType("igraph")
    pkg = types.ModuleType("openea")          # namespace stub: skips openea/__init__.py (imports TF models)
    pkg.__path__ = [os.path.join(REF_SRC, "openea")]
    sys.modules["openea"] = pkg
    try:
        ns = types.SimpleNamespace(
            similarity=importlib.import_module("openea.modules.finding.similarity"),
            alignment=importlib.import_module("openea.modules.finding.alignment"),
            evaluation=importlib.import_module("openea.modules.finding.evaluation"),
            batch=importlib.import_module("openea.modules.train.batch"),
            finder=importlib.import_module("openea.modules.bootstrapping.alignment_finder"),
            read=importlib.import_module("openea.modules.load.read"),
            util=importlib.import_module("openea.modules.utils.util"),
        )
    finally:
        # leave no trace: the repo's own `openea` drop-in package must stay importable afterwards
        for k in [k for k in sys.modules if k == "openea" or k.startswith("openea.")]:
            del sys.modules[k]
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
            else:
                sys.modules.pop(k, None)
        sys.modules.update(saved_sub)
    return ns
