"""GPU parity of path (iii): K3 kernels (through the C-ABI) against the golden vectors produced by the
reference itself and against the NumPy oracle.  Index outputs (alignment pairs, ranks, neighbour sets) must
be bit-exact except on near-ties, which are counted and bounded; similarity values are fp32 within 2e-5."""
import os

import numpy as np
import pytest
import torch

from oracle import finding as orf

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "finding_golden.npz"))
METRICS = [("inner", 0), ("inner", 1), ("cosine", 0), ("euclidean", 0), ("manhattan", 0)]


def F():
    from openea_b200 import finding
    return finding


@pytest.mark.parametrize("tag", ["a", "b"])
@pytest.mark.parametrize("metric,norm", METRICS)
def test_sim_matrix_and_csls_vs_reference_golden(cuda_device, tag, metric, norm):
    e1, e2 = GOLD[tag + "_e1"], GOLD[tag + "_e2"]
    key = "%s_%s_%d" % (tag, metric, norm)
    rows = GOLD[tag + "_sim_rows"]
    got = F().sim(e1, e2, metric, bool(norm), 0).cpu().numpy()
    np.testing.assert_allclose(got[rows], GOLD[key + "_sim"], rtol=2e-5, atol=3e-5)
    got = F().sim(e1, e2, metric, bool(norm), 10).cpu().numpy()
    np.testing.assert_allclose(got[rows], GOLD[key + "_csls"], rtol=2e-5, atol=1e-4)


@pytest.mark.parametrize("tag", ["a", "b"])
@pytest.mark.parametrize("metric,norm", METRICS)
@pytest.mark.parametrize("csls_k", [0, 10])
def test_greedy_alignment_vs_reference_golden(cuda_device, capsys, monkeypatch, tag, metric, norm, csls_k):
    if tag == "b":   # tag "a" runs the default (materialised CSLS); tag "b" forces the streaming strategy
        monkeypatch.setattr(F(), "MATERIALIZE_MAX_BYTES", 0)
    e1, e2 = GOLD[tag + "_e1"], GOLD[tag + "_e2"]
    key = "%s_%s_%d_k%d" % (tag, metric, norm, csls_k)
    pairs, hits1, mr, mrr = F().greedy_alignment(e1, e2, [1, 5, 10, 50], 4, metric, bool(norm), csls_k, True)
    want = {tuple(p) for p in GOLD[key + "_pairs"].tolist()}
    assert {(int(i), int(j)) for i, j in pairs} == want      # bit-exact alignment indices
    h1, wmr, wmrr = GOLD[key + "_stats"]
    assert hits1 == pytest.approx(h1, abs=1e-9) and mr == pytest.approx(wmr, rel=1e-9) and mrr == pytest.approx(wmrr, rel=1e-9)
    out = capsys.readouterr().out
    assert ("accurate results with csls: csls=10, hits@[1, 5, 10, 50] = [" in out) if csls_k else ("accurate results: hits@[1, 5, 10, 50] = [" in out)


@pytest.mark.parametrize("n1,n2,d,metric,csls_k", [(2000, 2000, 100, "inner", 0), (2000, 2000, 100, "inner", 10),
                                                   (1500, 2300, 200, "manhattan", 10), (700, 3001, 75, "euclidean", 10),
                                                   (129, 127 + 128, 300, "inner", 10)])
@pytest.mark.parametrize("materialize", [False, True])
def test_rank_and_top1_vs_oracle_seeded(cuda_device, n1, n2, d, metric, csls_k, materialize):
    """SURVEY §7 (5): identical (i, argmax) sets and Hits@k on seeded inputs; tie/near-tie disagreements reported."""
    rng = np.random.default_rng(n1 + n2 + d)
    e2 = rng.standard_normal((n2, d)).astype(np.float32)
    e1 = (e2[:n1] + 0.5 * rng.standard_normal((n1, d))).astype(np.float32)
    norm = metric == "inner"
    # both CSLS strategies: streaming (3 fused tile passes, nothing stored) and materialised (1 pass + 3 streaming reads)
    top1, rk, hits, mr, mrr = F().eval_alignment(e1, e2, [1, 5, 10, 50], metric, norm, csls_k, materialize=materialize)
    s = orf.sim(e1, e2, metric, norm, csls_k)
    wtop1, wrank = orf.rank_rows(s)
    whits, wmr, wmrr = orf.metrics_from_ranks(wrank, [1, 5, 10, 50])
    top1, rk = top1.cpu().numpy(), rk.cpu().numpy()
    n_bad = int((top1 != wtop1).sum()) + int((rk != wrank).sum())
    assert n_bad <= max(1, n1 // 1000), "index disagreements beyond near-ties: %d" % n_bad
    if n_bad == 0:
        assert hits == whits and mr == pytest.approx(wmr) and mrr == pytest.approx(wmrr)


def test_topk_values_indices_and_means(cuda_device):
    rng = np.random.default_rng(8)
    e1 = rng.standard_normal((333, 100)).astype(np.float32)
    e2 = rng.standard_normal((1000, 100)).astype(np.float32)
    f = F()
    d1, d = f.to_device_rows(e1, True)
    d2, _ = f.to_device_rows(e2, True)
    for k in (1, 10, 32):
        res = f.topk(d1, d2, d, "inner", k)
        s = orf.sim(e1, e2, "inner", True, 0)
        wv, wi = orf.topk_rows(s, k)
        np.testing.assert_array_equal(res["idx"].cpu().numpy(), wi)
        np.testing.assert_allclose(res["val"].cpu().numpy(), wv, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(res["mean"].cpu().numpy(), orf.nearest_k_mean(s, k), rtol=1e-5, atol=1e-6)


def test_duplicate_rows_tie_rule(cuda_device):
    """Exact ties (duplicated columns): the lower column index wins in argmax, rank and top-k order."""
    rng = np.random.default_rng(4)
    base = rng.standard_normal((50, 64)).astype(np.float32)
    e2 = np.concatenate([base, base], 0)          # column j and j+50 are identical
    e1 = base.copy()
    f = F()
    top1, rk, hits, _, _ = f.eval_alignment(e1, e2, [1], "inner", False, 0)
    assert (top1.cpu().numpy() == np.arange(50)).all() and (rk.cpu().numpy() == 0).all() and hits == [100.0]
    gold = torch.arange(50, 100, dtype=torch.int32)
    top1, rk, _, _, _ = f.eval_alignment(e1, e2, [1], "inner", False, 0, gold=gold.cuda())
    assert (rk.cpu().numpy() == 1).all()          # the identical lower-index column ranks first


@pytest.mark.parametrize("tag", ["a", "b"])
def test_neighbour_search_and_bootstrap_filter_vs_reference_golden(cuda_device, tag):
    e2 = GOLD[tag + "_e2"]
    en = e2 / np.linalg.norm(e2, axis=1, keepdims=True)
    k = int(GOLD[tag + "_neigh_k"][0])
    ents = (np.arange(e2.shape[0]) * 2 + 1).astype(np.int32)
    got = F().find_neighbours_device(en, ents, k, row_block=100).cpu().numpy()
    want = GOLD[tag + "_neigh"]
    assert got.shape == want.shape
    assert all(set(got[i].tolist()) == set(want[i].tolist()) for i in range(len(got)))
    rows, cols, vals = F().find_alignment_device(GOLD[tag + "_e1"], e2, 0.7, 10)
    got_pairs = set(zip(rows.cpu().numpy().tolist(), cols.cpu().numpy().tolist()))
    assert got_pairs == {tuple(p) for p in GOLD[tag + "_find_alignment"].tolist()}


def test_large_k_select_properties(cuda_device):
    """Full-size shape (15K × 15K, k = 1500): size-independent properties of the ε-truncated search."""
    rng = np.random.default_rng(5)
    n, d, k = 15000, 100, 1500
    e = rng.standard_normal((n, d)).astype(np.float32)
    e /= np.linalg.norm(e, axis=1, keepdims=True)
    ents = np.arange(n, dtype=np.int32) * 2
    out = F().find_neighbours_device(e, ents, k).cpu().numpy()
    assert out.shape == (n, k)
    rows = rng.choice(n, 40, replace=False)
    s = e[rows] @ e.T
    for r, row in enumerate(rows):
        got = out[row] // 2
        assert len(set(got.tolist())) == k, "no duplicates"
        kth = np.partition(-s[r], k - 1)[k - 1] * -1
        assert (s[r][got] >= kth - 1e-6).all(), "every selected entity is at least as similar as the k-th best"
        assert row in got, "an entity is its own nearest neighbour"


def test_rdgcn_get_neg_matches_cdist_argsort(cuda_device):
    """rdgcn.py:75-87: k nearest by cityblock distance (the seed itself first), against scipy's cdist + argsort."""
    from scipy.spatial.distance import cdist
    from openea_b200.approaches.rdgcn_ops import get_neg
    rng = np.random.default_rng(12)
    emb = rng.standard_normal((1500, 300)).astype(np.float32)
    ill = rng.choice(1500, 200, replace=False)
    k = 10
    got = get_neg(ill, emb, k).cpu().numpy().reshape(200, k)
    sim = cdist(emb[ill], emb, metric="cityblock")
    want = np.argsort(sim, axis=1, kind="stable")[:, :k]
    assert (got[:, 0] == ill).all()
    assert (got == want).mean() > 0.999          # fp32 vs fp64 distances: only near-ties may swap


@pytest.mark.parametrize("d", [3, 12, 75, 100, 104])
@pytest.mark.parametrize("metric", ["inner", "euclidean", "manhattan"])
def test_resident_panel_store_kernel_is_bit_identical_to_streaming_kernel(cuda_device, monkeypatch, d, metric):
    """k_sim_store_shortk (A panel resident, two half-K stages per column tile) accumulates in the same ascending-k
    order as k_sim_tile, so the stored matrix — plain and with CSLS offsets — is bit-identical; shapes cover ragged
    row/column tiles and several column splits."""
    rng = np.random.default_rng(1000 + d)
    n1, n2 = 389, 1301
    e1 = rng.standard_normal((n1, d)).astype(np.float32)
    e2 = rng.standard_normal((n2, d)).astype(np.float32)
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("OEA_SIM_NO_SHORTK", mode)
        out[mode] = (F().sim(e1, e2, metric, False, 0).cpu().numpy(), F().sim(e1, e2, metric, False, 5).cpu().numpy())
    assert np.array_equal(out["0"][0], out["1"][0])
    assert np.array_equal(out["0"][1], out["1"][1])
    want = orf.sim(e1, e2, metric, False)
    np.testing.assert_allclose(out["0"][0], want, rtol=2e-5, atol=3e-5)


@pytest.mark.parametrize("n_rows,n_cols", [(700, 1301), (70, 37), (2100, 129)])
@pytest.mark.parametrize("k", [1, 3, 8, 10, 16, 25, 32])
def test_matrix_column_and_row_topk_mean_every_list_size(cuda_device, n_rows, n_cols, k):
    """oea_matrix_topk_mean on a stored matrix: register-list column kernel (every KCAP instantiation, ragged last
    column group, padded leading dimension holding garbage) + partial merge, and the row kernel, against NumPy."""
    import ctypes as C
    from openea_b200 import lib as L
    from openea_b200.engine import _ptr, _stream_ptr
    lib = L.load()
    rng = np.random.default_rng(k * 1000 + n_cols)
    m = rng.standard_normal((n_rows, n_cols)).astype(np.float32)
    m[rng.integers(0, n_rows, 50), rng.integers(0, n_cols, 50)] = 3.5      # ties among the largest
    ld = (n_cols + 3) // 4 * 4
    dev = torch.full((n_rows, ld), 1e30, dtype=torch.float32, device="cuda")   # padding must never be read as data
    dev[:, :n_cols] = torch.from_numpy(m).cuda()
    for by_col in (0, 1):
        n_out = n_cols if by_col else n_rows
        if k > (n_rows if by_col else n_cols):
            continue
        out = torch.empty(n_out, dtype=torch.float32, device="cuda")
        nbytes = lib.oea_matrix_topk_mean_workspace_bytes(n_rows, n_cols, k, by_col)
        ws = torch.empty(max(16, nbytes), dtype=torch.uint8, device="cuda")
        L.check(lib.oea_matrix_topk_mean(_ptr(dev), ld, n_rows, n_cols, k, by_col, _ptr(out), _ptr(ws), nbytes, _stream_ptr()))
        a = m.T if by_col else m
        want = -np.sort(-a, axis=1)[:, :k].astype(np.float64).mean(1)
        np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-5, atol=1e-6)


def test_rank_stats_kernel_matches_numpy(cuda_device):
    rng = np.random.default_rng(3)
    rk = np.minimum(rng.geometric(0.05, 10500) - 1, 10499).astype(np.int32)
    hits, mr, mrr = F().rank_stats(torch.from_numpy(rk).cuda(), [1, 5, 10, 50])
    want_hits = [round(float((rk < k).sum()) / len(rk) * 100, 3) for k in [1, 5, 10, 50]]
    assert hits == want_hits
    assert mr == pytest.approx(float((rk + 1).mean()), rel=1e-12)
    assert mrr == pytest.approx(float((1.0 / (rk + 1)).mean()), rel=1e-12)
    hits9, _, _ = F().rank_stats(torch.from_numpy(rk).cuda(), list(range(1, 12)))    # more than 8 thresholds: two launches
    assert hits9 == [round(float((rk < k).sum()) / len(rk) * 100, 3) for k in range(1, 12)]
