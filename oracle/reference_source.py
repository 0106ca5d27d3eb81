"""TEST INFRASTRUCTURE: pure-Python / NumPy / pandas helper functions of the reference compiled from its own source
(selected top-level definitions only, so TensorFlow is never imported).  Available only where OPENEA_REFERENCE names a
checkout of the original project: tests call it to record their golden results.  Nothing under openea_b200/ imports this."""
import ast
import os

REF_ROOT = os.path.join(os.environ.get("OPENEA_REFERENCE", ""), "src", "openea")


def extract(rel_path, names, namespace):
    """Compile the top-level functions / classes `names` of REF_ROOT/rel_path into `namespace`; None if absent."""
    path = os.path.join(REF_ROOT, rel_path)
    if not os.environ.get("OPENEA_REFERENCE") or not os.path.exists(path):
        return None
    with open(path) as f:
        tree = ast.parse(f.read())
    keep = [n for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and n.name in set(names)]
    ns = dict(namespace)
    exec(compile(ast.Module(body=keep, type_ignores=[]), path, "exec"), ns)
    return ns


def iptranse_helpers():
    """generate_2steps_path, generate_newly_triples, generate_triples_of_latent_ents, generate_neg_triples_w,
    generate_neg_paths of approaches/iptranse.py:21-121."""
    import random
    import numpy as np
    import pandas as pd
    quiet = lambda *a, **k: None
    return extract("approaches/iptranse.py",
                   ["generate_2steps_path", "generate_newly_triples", "generate_triples_of_latent_ents",
                    "generate_neg_triples_w", "generate_neg_paths"],
                   {"np": np, "pd": pd, "random": random, "print": quiet, "KGs": object})


def bootea_helpers():
    """update_labeled_alignment_x / _y, generate_supervised_triples, generate_newly_triples, generate_pos_batch,
    calculate_likelihood_mat of approaches/bootea.py:35-137 (pure Python; the diagnostics print is silenced)."""
    import gc
    import time
    import numpy as np
    return extract("approaches/bootea.py",
                   ["update_labeled_alignment_x", "update_labeled_alignment_y", "generate_supervised_triples",
                    "generate_newly_triples", "generate_pos_batch", "calculate_likelihood_mat"],
                   {"np": np, "gc": gc, "time": time, "print": lambda *a, **k: None,
                    "check_new_alignment": lambda *a, **k: None})
