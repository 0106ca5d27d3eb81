"""CPU: pin the NumPy oracle for path (iii) against golden vectors generated FROM THE REFERENCE ITSELF
(tests/golden/make_golden.py) and against results the reference functions returned on a further seed."""
import ast
import contextlib
import io
import os

import numpy as np
import pytest

from oracle import finding as orf
from oracle import ref_adapter
from tests.helpers import ReferenceRecord

REC = ReferenceRecord("reference_oracle_finding")
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "finding_golden.npz"))
METRICS = [("inner", 0), ("inner", 1), ("cosine", 0), ("euclidean", 0), ("manhattan", 0)]


@pytest.mark.parametrize("tag", ["a", "b"])
@pytest.mark.parametrize("metric,norm", METRICS)
def test_sim_and_csls_match_reference(tag, metric, norm):
    e1, e2 = GOLD[tag + "_e1"], GOLD[tag + "_e2"]
    key = "%s_%s_%d" % (tag, metric, norm)
    rows = GOLD[tag + "_sim_rows"]
    s = orf.sim(e1, e2, metric, bool(norm), 0)
    np.testing.assert_allclose(s[rows], GOLD[key + "_sim"], rtol=2e-5, atol=2e-5)
    sc = orf.sim(e1, e2, metric, bool(norm), 10)
    np.testing.assert_allclose(sc[rows], GOLD[key + "_csls"], rtol=2e-5, atol=6e-5)


@pytest.mark.parametrize("tag", ["a", "b"])
@pytest.mark.parametrize("metric,norm", METRICS)
@pytest.mark.parametrize("csls_k", [0, 10])
def test_greedy_alignment_matches_reference(tag, metric, norm, csls_k):
    e1, e2 = GOLD[tag + "_e1"], GOLD[tag + "_e2"]
    key = "%s_%s_%d_k%d" % (tag, metric, norm, csls_k)
    pairs, hits, mr, mrr = orf.greedy_alignment(e1, e2, [1, 5, 10, 50], metric, bool(norm), csls_k)
    want_pairs = {tuple(p) for p in GOLD[key + "_pairs"].tolist()}
    assert pairs == want_pairs          # bit-exact alignment indices
    h1, wmr, wmrr = GOLD[key + "_stats"]
    assert hits[0] == pytest.approx(h1, abs=1e-9)
    assert mr == pytest.approx(wmr, rel=1e-12) and mrr == pytest.approx(wmrr, rel=1e-12)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_neighbours_and_find_alignment_match_reference(tag):
    e2 = GOLD[tag + "_e2"]
    en = e2 / np.linalg.norm(e2, axis=1, keepdims=True)
    k = int(GOLD[tag + "_neigh_k"][0])
    ents = np.arange(e2.shape[0]) * 2 + 1
    got = orf.find_neighbours(en, en, ents, k)
    want = GOLD[tag + "_neigh"]
    assert all(got[i] == set(want[i].tolist()) for i in range(len(got)))
    s = orf.sim(GOLD[tag + "_e1"], e2, "inner", True, 0)
    pairs = orf.find_alignment(s, 0.7, 10) or set()
    assert pairs == {tuple(p) for p in GOLD[tag + "_find_alignment"].tolist()}


def test_rank_tie_rule_and_metrics_known_answer():
    s = np.array([[0.9, 0.9, 0.1, 0.0],     # gold 0 tied with col 1 → lower index wins → rank 0
                  [0.5, 0.5, 0.7, 0.5],     # gold 1: one better (col 2), tie with col 0 before it → rank 2
                  [0.1, 0.2, 0.3, 0.4],     # gold 2: one better → rank 1
                  [0.0, 0.0, 0.0, 1.0]], dtype=np.float32)
    top1, rank = orf.rank_rows(s)
    assert top1.tolist() == [0, 2, 3, 3] and rank.tolist() == [0, 2, 1, 0]
    hits, mr, mrr = orf.metrics_from_ranks(rank, [1, 2])
    assert hits == [50.0, 75.0] and mr == pytest.approx(7 / 4) and mrr == pytest.approx((1 + 1 / 3 + 1 / 2 + 1) / 4)


def test_csls_known_answer_3x4():
    s = np.array([[1, 2, 3, 4], [4, 3, 2, 1], [0, 0, 5, 5]], dtype=np.float32)
    r = np.array([3.5, 3.5, 5.0]); c = np.array([2.5, 2.5, 4.0, 4.5])   # top-2 means of rows / columns
    want = 2 * s - r[:, None] - c[None, :]
    np.testing.assert_allclose(orf.csls_sim(s, 2), want)


def test_live_reference_agrees_on_fresh_seed():
    ref = ref_adapter.load() if REC.live else None
    rng = np.random.default_rng(2024)
    e2 = rng.standard_normal((150, 64)).astype(np.float32)
    e1 = (e2[:120] + 0.4 * rng.standard_normal((120, 64))).astype(np.float32)
    for metric, norm, k in (("inner", True, 10), ("manhattan", False, 5), ("euclidean", False, 0)):
        def reference():
            with contextlib.redirect_stdout(io.StringIO()):
                want, h1, mr, mrr = ref.alignment.greedy_alignment(e1, e2, [1, 5], 1, metric, norm, k, True)
            return np.array(sorted(want), dtype=np.float64).reshape(-1), np.array([h1, mr, mrr], dtype=np.float64)
        key = "%s-%d-%d" % (metric, norm, k)
        want = REC.array(key + "/pairs", lambda: reference()[0]).astype(np.int64).reshape(-1, 2)
        h1, mr, mrr = REC.array(key + "/stats", lambda: reference()[1])
        got, hits, gmr, gmrr = orf.greedy_alignment(e1, e2, [1, 5], metric, norm, k)
        assert got == {(int(i), int(j)) for i, j in want} and hits[0] == pytest.approx(h1)
        assert gmr == pytest.approx(mr) and gmrr == pytest.approx(mrr)
