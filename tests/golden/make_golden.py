"""Generate golden vectors from the REFERENCE ITSELF (its NumPy modules imported with TF stubbed).

Run with a checkout of the original project:  OPENEA_REFERENCE=/path/to/OpenEA python tests/golden/make_golden.py
The .npz file it writes is committed; the tests read it and need no reference.  The similarity and CSLS matrices are
stored for a seeded sample of rows (`<tag>_sim_rows`, first and last row included) to keep the file under 1 MB; the
alignments, ranks and neighbour lists derived from the full matrices are stored whole.
"""
import contextlib
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_adapter  # noqa: E402


def embeds(seed, n1, n2, d, noise=0.35):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((n2, d)).astype(np.float32)
    e2 = base
    e1 = (base[:n1] + noise * rng.standard_normal((n1, d))).astype(np.float32)
    return e1, e2


SIM_ROWS = {"a": 32, "b": 24}


def sim_rows(tag, n1):
    rows = np.random.default_rng(0).choice(np.arange(1, n1 - 1), SIM_ROWS[tag] - 2, replace=False)
    return np.sort(np.concatenate([[0, n1 - 1], rows])).astype(np.int64)


def main():
    ref = ref_adapter.load()
    out = {}
    quiet = io.StringIO()
    cases = [("a", 11, 257, 300, 100), ("b", 12, 130, 130, 75)]
    for tag, seed, n1, n2, d in cases:
        e1, e2 = embeds(seed, n1, n2, d)
        out["%s_e1" % tag], out["%s_e2" % tag] = e1, e2
        rows = out["%s_sim_rows" % tag] = sim_rows(tag, n1)
        for metric, norm in (("inner", False), ("inner", True), ("cosine", False), ("euclidean", False), ("manhattan", False)):
            with contextlib.redirect_stdout(quiet):
                s = ref.similarity.sim(e1, e2, metric=metric, normalize=norm, csls_k=0)
                sc = ref.similarity.sim(e1, e2, metric=metric, normalize=norm, csls_k=10)
            key = "%s_%s_%d" % (tag, metric, int(norm))
            out[key + "_sim"] = s[rows].astype(np.float32)
            out[key + "_csls"] = sc[rows].astype(np.float32)
            for csls_k in (0, 10):
                with contextlib.redirect_stdout(quiet):
                    pairs, hits1, mr, mrr = ref.alignment.greedy_alignment(e1, e2, [1, 5, 10, 50], 1, metric, norm, csls_k, True)
                pr = np.array(sorted(pairs), dtype=np.int32)
                out["%s_k%d_pairs" % (key, csls_k)] = pr
                out["%s_k%d_stats" % (key, csls_k)] = np.array([hits1, mr, mrr], dtype=np.float64)
        # large-k neighbour search (batch.py:145-165) on normalised rows, k = 10 % of the list
        en = e2 / np.linalg.norm(e2, axis=1, keepdims=True)
        ents = (np.arange(n2) * 2 + 1).astype(np.int64)
        k = max(3, n2 // 10)
        dic = ref.batch.generate_neighbours_single_thread(en, ents.tolist(), k, 3)
        out["%s_neigh_k" % tag] = np.array([k])
        out["%s_neigh" % tag] = np.array([sorted(dic[int(e)]) for e in ents], dtype=np.int64)
        # bootstrapping filter ∧ top-k (alignment_finder.py:28-51)
        with contextlib.redirect_stdout(quiet):
            s = ref.similarity.sim(e1, e2, metric="inner", normalize=True, csls_k=0)
            pairs = ref.finder.find_alignment(s, 0.7, 10)
        out["%s_find_alignment" % tag] = np.array(sorted(pairs) if pairs else [], dtype=np.int64).reshape(-1, 2)
    # host logic: task_divide, batch slicing, id assignment
    td = [ref.util.task_divide(list(range(n)), t) for n, t in ((10, 3), (7, 7), (5, 8), (0, 2), (12, 4))]
    out["task_divide"] = np.array([str(td)])
    tl1 = [(i, 0, i + 1) for i in range(23)]
    tl2 = [(100 + i, 1, 101 + i) for i in range(11)]
    slices = []
    for step in range(5):
        b = ref.batch.generate_pos_batch(tl1, tl2, 8, step)
        slices.append(b)
    out["pos_batch_slices"] = np.array([str(slices)])
    t1 = {("a", "r1", "b"), ("a", "r1", "c"), ("b", "r2", "c")}
    t2 = {("x", "s1", "y"), ("y", "s1", "z"), ("z", "s2", "x"), ("y", "s2", "w"), ("w", "s1", "v")}
    ids1, ids2 = ref.read.generate_mapping_id(t1, {"a", "b", "c"}, t2, {"x", "y", "z", "w", "v"}, ordered=True)
    out["mapping_id"] = np.array([str(sorted(ids1.items())), str(sorted(ids2.items()))])
    ids1, ids2 = ref.read.generate_sharing_id([("a", "y")], t1, {"a", "b", "c"}, t2, {"x", "y", "z", "w", "v"}, ordered=True)
    out["sharing_id"] = np.array([str(sorted(ids1.items())), str(sorted(ids2.items()))])
    np.savez_compressed(os.path.join(HERE, "finding_golden.npz"), **out)
    print("wrote", os.path.join(HERE, "finding_golden.npz"), len(out), "arrays")


if __name__ == "__main__":
    main()
