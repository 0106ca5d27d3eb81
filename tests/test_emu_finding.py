"""CPU: the kernels of path (iii) (openea_b200/csrc/oea_sim.cu: tiled similarity with top-k / rank / store epilogues,
CSLS on the stored matrix, row / column top-k means, radix selection of the k nearest, rank statistics) executed from
their SOURCE on the warp emulator (all warps of a block concurrent, real __syncthreads) through the
product's own host layer (openea_b200/finding.py over CPU tensors), against the golden vectors the reference itself
produced (tests/golden/finding_golden.npz).  The same checks run on the B200 in tests/test_finding_gpu.py."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from openea_b200 import lib as L
from tests.emu import build_emu

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "finding_golden.npz"))


@pytest.fixture()
def finding_cpu(monkeypatch):
    so = build_emu.build()
    if so is None:
        pytest.skip("no CUDA headers for the emulator build")
    lib = C.CDLL(so)
    for name, (res, args) in L.SIGNATURES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    from openea_b200 import engine as eng
    from openea_b200 import finding
    monkeypatch.setattr(L, "load", lambda: lib)
    monkeypatch.setattr(finding, "_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(finding, "_stream_ptr", lambda: C.c_void_p(0))
    monkeypatch.setattr(eng, "_stream_ptr", lambda: C.c_void_p(0))
    return finding


@pytest.mark.parametrize("tag,metric,norm", [("b", "inner", 0), ("b", "inner", 1), ("b", "cosine", 0), ("b", "euclidean", 0),
                                             ("b", "manhattan", 0), ("a", "inner", 0)])
def test_emulated_sim_matrix_and_csls_equal_the_reference_golden(finding_cpu, tag, metric, norm):
    e1, e2 = GOLD[tag + "_e1"], GOLD[tag + "_e2"]
    key = "%s_%s_%d" % (tag, metric, norm)
    rows = GOLD[tag + "_sim_rows"]
    got = finding_cpu.sim(e1, e2, metric, bool(norm), 0).numpy()
    np.testing.assert_allclose(got[rows], GOLD[key + "_sim"], rtol=2e-5, atol=3e-5)
    got = finding_cpu.sim(e1, e2, metric, bool(norm), 10).numpy()
    np.testing.assert_allclose(got[rows], GOLD[key + "_csls"], rtol=2e-5, atol=1e-4)


@pytest.mark.parametrize("materialize", [True, False])
@pytest.mark.parametrize("metric,norm,csls_k", [("inner", 0, 0), ("inner", 1, 10), ("manhattan", 0, 10), ("euclidean", 0, 0)])
def test_emulated_greedy_alignment_equals_the_reference_golden(finding_cpu, monkeypatch, capsys, metric, norm, csls_k, materialize):
    if not materialize:
        monkeypatch.setattr(finding_cpu, "MATERIALIZE_MAX_BYTES", 0)       # the streaming strategy (no stored matrix)
    e1, e2 = GOLD["b_e1"], GOLD["b_e2"]
    key = "b_%s_%d_k%d" % (metric, norm, csls_k)
    pairs, hits1, mr, mrr = finding_cpu.greedy_alignment(e1, e2, [1, 5, 10, 50], 4, metric, bool(norm), csls_k, True)
    assert {(int(i), int(j)) for i, j in pairs} == {tuple(p) for p in GOLD[key + "_pairs"].tolist()}
    h1, wmr, wmrr = GOLD[key + "_stats"]
    assert hits1 == pytest.approx(h1, abs=1e-9) and mr == pytest.approx(wmr, rel=1e-9) and mrr == pytest.approx(wmrr, rel=1e-9)


def test_emulated_neighbour_search_and_bootstrap_filter_equal_the_reference_golden(finding_cpu):
    tag = "b"
    e2 = GOLD[tag + "_e2"]
    en = e2 / np.linalg.norm(e2, axis=1, keepdims=True)
    k = int(GOLD[tag + "_neigh_k"][0])
    ents = (np.arange(e2.shape[0]) * 2 + 1).astype(np.int32)
    got = finding_cpu.find_neighbours_device(en, ents, k, row_block=100).numpy()
    want = GOLD[tag + "_neigh"]
    assert got.shape == want.shape
    assert all(set(got[i].tolist()) == set(want[i].tolist()) for i in range(len(got)))
    rows, cols, vals = finding_cpu.find_alignment_device(GOLD[tag + "_e1"], e2, 0.7, 10)
    assert set(zip(rows.numpy().tolist(), cols.numpy().tolist())) == {tuple(p) for p in GOLD[tag + "_find_alignment"].tolist()}
