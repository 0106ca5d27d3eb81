"""CPU: the tensor versions of BootEA's bootstrapping step (openea_b200/modules/bootstrapping/device.py) against the
set / dict functions of approaches/bootea.py and alignment_finder.py that mirror the reference — same matching, same
label edits, same swap triples — on random inputs (CPU tensors; the product runs the same code on CUDA tensors)."""
import contextlib
import io

import numpy as np
import pytest
import torch

from openea_b200.approaches import bootea as host
from openea_b200.modules.bootstrapping import alignment_finder as af
from openea_b200.modules.bootstrapping import device as boot


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


@pytest.mark.parametrize("seed", range(6))
def test_greedy_matching_equals_sequential_greedy(seed):
    rng = np.random.default_rng(seed)
    n1, n2, e = 60, 50, 400
    pairs = np.unique(np.stack([rng.integers(0, n1, e), rng.integers(0, n2, e)], 1), axis=0)
    vals = rng.random(len(pairs)).astype(np.float32)
    if seed % 2:                                  # ties among the weights: earlier edge first, as the stable sort does
        vals = np.round(vals, 1)
    sel = boot.greedy_matching(torch.as_tensor(pairs[:, 0]), torch.as_tensor(pairs[:, 1]), torch.as_tensor(vals), n1, n2)
    got = {tuple(p) for p in pairs[sel.numpy()].tolist()}
    weights = {tuple(p): float(v) for p, v in zip(pairs.tolist(), vals)}
    want = af.mwgm_scipy([tuple(p) for p in pairs.tolist()], weights)
    assert got == want
    assert len({i for i, _ in got}) == len(got) == len({j for _, j in got})


def test_greedy_matching_degenerate_inputs():
    empty = torch.zeros(0, dtype=torch.int64)
    assert boot.greedy_matching(empty, empty, torch.zeros(0), 5, 5).numel() == 0
    one = boot.greedy_matching(torch.tensor([2]), torch.tensor([3]), torch.tensor([0.5]), 5, 5)
    assert one.tolist() == [True]
    star = boot.greedy_matching(torch.tensor([0, 0, 0]), torch.tensor([0, 1, 2]), torch.tensor([0.1, 0.9, 0.5]), 1, 3)
    assert star.tolist() == [False, True, False]


@pytest.mark.parametrize("seed", range(5))
def test_label_edits_equal_the_host_set_functions(seed):
    rng = np.random.default_rng(100 + seed)
    n, d = 80, 16
    e1 = torch.nn.functional.normalize(torch.as_tensor(rng.standard_normal((n, d)), dtype=torch.float32), dim=1)
    e2 = torch.nn.functional.normalize(e1 + 0.8 * torch.as_tensor(rng.standard_normal((n, d)), dtype=torch.float32), dim=1)
    sim = host.PairSim(e1, e2)
    # previous labels: a partial one-to-one assignment (what update_y leaves behind)
    pi, pj = rng.permutation(n)[:30], rng.permutation(n)[:30]
    labeled = set(zip(pi.tolist(), pj.tolist()))
    label = torch.full((n,), -1, dtype=torch.int64)
    label[torch.as_tensor(pi)] = torch.as_tensor(pj)
    # a new matching that overlaps the old labels on both sides
    mi, mj = rng.permutation(n)[:40], rng.permutation(n)[:40]
    curr = set(zip(mi.tolist(), mj.tolist()))
    want = _quiet(host.update_labeled_alignment_x, labeled, curr, sim)
    got = _quiet(boot.edit_labels_x, label, torch.as_tensor(mi), torch.as_tensor(mj), e1, e2)
    as_set = lambda lab: {(int(i), int(lab[i])) for i in torch.nonzero(lab >= 0).flatten()}
    assert as_set(got) == want
    want = _quiet(host.update_labeled_alignment_y, want, sim)
    got = _quiet(boot.edit_labels_y, got, e1, e2)
    assert as_set(got) == want
    js = [j for _, j in want]
    assert len(js) == len(set(js))


def test_bootstrap_pass_equals_host_bootstrapping(monkeypatch):
    """bootstrap_labels (matching + both edits) from given candidates == the host pipeline from the same candidates."""
    rng = np.random.default_rng(9)
    n, d, k, th = 70, 12, 4, 0.2
    e1 = torch.nn.functional.normalize(torch.as_tensor(rng.standard_normal((n, d)), dtype=torch.float32), dim=1)
    e2 = torch.nn.functional.normalize(e1 + 0.6 * torch.as_tensor(rng.standard_normal((n, d)), dtype=torch.float32), dim=1)
    s = e1 @ e2.t()
    val, idx = s.topk(k, dim=1)
    keep = val > th
    rows = torch.arange(n)[:, None].expand_as(keep)[keep]
    cand = (rows, idx[keep], val[keep])
    label = torch.full((n,), -1, dtype=torch.int64)
    labeled = set()
    sim = host.PairSim(e1, e2)
    for _ in range(2):                                      # two passes: the second one edits existing labels
        pairs = set(zip(cand[0].tolist(), cand[1].tolist()))
        curr = af.mwgm_scipy(list(pairs), sim.values(list(pairs)))
        labeled = _quiet(host.update_labeled_alignment_x, labeled, curr, sim)
        labeled = _quiet(host.update_labeled_alignment_y, labeled, sim)
        _, i, j = _quiet(boot.bootstrap_labels, e1, e2, label, cand)
        assert set(zip(i.tolist(), j.tolist())) == labeled
        e2 = torch.nn.functional.normalize(e2 + 0.3 * torch.as_tensor(rng.standard_normal((n, d)), dtype=torch.float32), dim=1)
        sim = host.PairSim(e1, e2)
        s = e1 @ e2.t()
        val, idx = s.topk(k, dim=1)
        keep = val > th
        cand = (torch.arange(n)[:, None].expand_as(keep)[keep], idx[keep], val[keep])
    assert _quiet(boot.bootstrap_labels, e1, e2, label.clone(), None)[1].numel() == len(labeled)


def test_swap_triples_and_batches_equal_the_host_functions():
    rng = np.random.default_rng(3)
    n_ent, n_rel = 50, 4
    tri = np.unique(np.stack([rng.integers(0, n_ent, 300), rng.integers(0, n_rel, 300), rng.integers(0, n_ent, 300)], 1), axis=0)
    rt, hr = {}, {}
    for h, r, t in tri.tolist():
        rt.setdefault(h, set()).add((r, t))
        hr.setdefault(t, set()).add((h, r))
    src, dst = rng.permutation(n_ent)[:12], rng.permutation(n_ent)[:12]
    want1, _ = _quiet(host.generate_supervised_triples, rt, hr, {}, {}, src.tolist(), dst.tolist())
    got = boot.swap_triples(torch.as_tensor(tri.astype(np.int32)), torch.as_tensor(src), torch.as_tensor(dst), n_ent)
    assert sorted(map(tuple, got.tolist())) == sorted(want1)
    # batching: same slice arithmetic as generate_pos_batch
    a = torch.as_tensor(rng.integers(0, 9, (23, 3)).astype(np.int32))
    b = torch.as_tensor(rng.integers(0, 9, (31, 3)).astype(np.int32))
    for step in range(5):
        h1, h2 = host.generate_pos_batch(a.tolist(), b.tolist(), step, 16)
        want = np.asarray(h1 + h2, dtype=np.int32).reshape(-1, 3).T
        assert np.array_equal(boot.pos_batch(a, b, step, 16).numpy(), want)


def test_bootea_device_iteration_methods_on_cpu_tensors(monkeypatch):
    """BootEA.bootstrap_on_device + train_alignment_device wired end to end on CPU tensors: the candidate search is
    replaced by a torch top-k stand-in (the K3 kernel needs a GPU) and the alignment trainer by a recorder; every
    swap triple of the labelled pairs reaches the trainer exactly once, in fed-scorer layout."""
    from types import SimpleNamespace
    from openea_b200 import finding as F
    rng = np.random.default_rng(5)
    n_ent, d = 120, 10
    ref1, ref2 = list(range(0, 60, 2)), list(range(1, 60, 2))            # 30 reference entities per KG
    emb = torch.nn.functional.normalize(torch.as_tensor(rng.standard_normal((n_ent, d)), dtype=torch.float32), dim=1)
    emb[ref2] = torch.nn.functional.normalize(emb[ref1] + 0.3 * torch.as_tensor(rng.standard_normal((30, d)), dtype=torch.float32), dim=1)

    def topk_standin(e1, e2, sim_th, k, metric, normalize):
        val, idx = (e1 @ e2.t()).topk(k, dim=1)
        keep = val > sim_th
        rows = torch.arange(e1.shape[0], dtype=torch.int32)[:, None].expand_as(keep)[keep]
        return rows, idx[keep].to(torch.int32), val[keep]
    monkeypatch.setattr(F, "find_alignment_device", topk_standin)

    tri = lambda lo: np.unique(np.stack([rng.integers(lo, lo + 60, 200), rng.integers(0, 3, 200),
                                         rng.integers(lo, lo + 60, 200)], 1), axis=0).astype(np.int32)
    t1, t2 = tri(0), tri(0)
    seen = []
    model = object.__new__(host.BootEA)
    model.args = SimpleNamespace(sim_th=0.5, k=3, batch_size=64)
    model.ref_ent1, model.ref_ent2 = ref1, ref2
    model.ent_embeds = SimpleNamespace(device=torch.device("cpu"), dim=d)
    model.eval_ref_sim_mat = lambda: host.PairSim(emb[ref1], emb[ref2])
    model.kgs = SimpleNamespace(entities_num=n_ent, kg1=SimpleNamespace(local_relation_triples_array=t1),
                                kg2=SimpleNamespace(local_relation_triples_list=[tuple(x) for x in t2.tolist()]))
    model.alignment_trainer = SimpleNamespace(score_fed=lambda pos: seen.append(pos.clone()), apply=lambda: None,
                                              read_loss=lambda: 1.0)
    ents1, ents2 = _quiet(model.bootstrap_on_device)
    assert ents1.numel() > 10 and ents1.numel() == ents2.numel()
    assert set(ents1.tolist()) <= set(ref1) and set(ents2.tolist()) <= set(ref2)
    right = sum(int(a) + 1 == int(b) for a, b in zip(ents1.tolist(), ents2.tolist()))
    assert right >= 0.8 * ents1.numel()                     # the noisy copies are each other's nearest neighbours
    _quiet(model.train_alignment_device, ents1, ents2, 1)
    fed = torch.cat(seen, 1).t().tolist()
    want = boot.swap_triples(torch.as_tensor(t1), ents1, ents2, n_ent).tolist() + \
        boot.swap_triples(torch.as_tensor(t2), ents2, ents1, n_ent).tolist()
    assert sorted(map(tuple, fed)) == sorted(map(tuple, want)) and all(p.dtype == torch.int32 and p.shape[0] == 3 for p in seen)
    ents1b, _ = _quiet(model.bootstrap_on_device)             # second pass edits the existing labels
    assert ents1b.numel() >= ents1.numel()


def test_host_and_device_functions_equal_the_reference_source():
    """The label-editing, swap-triple and batch-slicing functions of BootEA, executed from the reference's own source
    (approaches/bootea.py:35-137) and recorded, against this package's host functions and the tensor versions."""
    import collections
    import contextlib
    import io
    from openea_b200.approaches import bootea as host
    from openea_b200.modules.bootstrapping import device as dev
    from oracle import reference_source
    from tests.helpers import ReferenceRecord
    rec = ReferenceRecord("reference_bootea")
    ref = reference_source.bootea_helpers() if rec.live else None
    rng = np.random.default_rng(3)
    n = 40
    for trial in range(5):
        e1 = torch.nn.functional.normalize(torch.as_tensor(rng.standard_normal((n, 8)), dtype=torch.float32), dim=1)
        e2 = torch.nn.functional.normalize(torch.as_tensor(rng.standard_normal((n, 8)), dtype=torch.float32), dim=1)
        sim, pair_sim = (e1 @ e2.t()).numpy(), host.PairSim(e1, e2)      # the reference indexes a matrix, this package pairs
        pre = {(int(i), int(j)) for i, j in zip(rng.permutation(n)[:15], rng.integers(0, n, 15))}
        cur = {(int(i), int(j)) for i, j in zip(rng.permutation(n)[:20], rng.permutation(n)[:20])}     # a matching
        with contextlib.redirect_stdout(io.StringIO()):
            got_x = host.update_labeled_alignment_x(set(pre), set(cur), pair_sim)
            assert rec.equal("update_labeled_alignment_x/%d" % trial, got_x,
                             lambda: ref["update_labeled_alignment_x"](set(pre), set(cur), sim))
            assert rec.equal("update_labeled_alignment_y/%d" % trial, host.update_labeled_alignment_y(set(got_x), pair_sim),
                             lambda: ref["update_labeled_alignment_y"](set(got_x), sim))
    # swap triples: dict walk of the reference vs host mirror vs masked gathers on tensors
    tri = np.unique(np.stack([rng.integers(0, 30, 200), rng.integers(0, 5, 200), rng.integers(0, 30, 200)], 1), axis=0)
    tri2 = np.unique(np.stack([rng.integers(30, 60, 200), rng.integers(0, 5, 200), rng.integers(30, 60, 200)], 1), axis=0)

    def dicts(t):
        rt, hr = collections.defaultdict(set), collections.defaultdict(set)
        for h, r, tt in t:
            rt[int(h)].add((int(r), int(tt)))
            hr[int(tt)].add((int(h), int(r)))
        return rt, hr
    rt1, hr1 = dicts(tri)
    rt2, hr2 = dicts(tri2)
    e1 = [int(x) for x in rng.permutation(30)[:12]]
    e2 = [int(x) for x in 30 + rng.permutation(30)[:12]]
    with contextlib.redirect_stdout(io.StringIO()):
        g1, g2 = host.generate_supervised_triples(rt1, hr1, rt2, hr2, e1, e2)

        def reference():
            w1, w2 = ref["generate_supervised_triples"](rt1, hr1, rt2, hr2, e1, e2)
            return sorted(w1), sorted(w2)
        assert rec.equal("generate_supervised_triples", (sorted(g1), sorted(g2)), reference)
    t1 = dev.swap_triples(torch.as_tensor(tri.astype(np.int32)), torch.as_tensor(e1), torch.as_tensor(e2), 60)
    t2 = dev.swap_triples(torch.as_tensor(tri2.astype(np.int32)), torch.as_tensor(e2), torch.as_tensor(e1), 60)
    assert sorted(map(tuple, t1.tolist())) == sorted(g1) and sorted(map(tuple, t2.tolist())) == sorted(g2)
    # batch slices
    a, b = [tuple(x) for x in tri.tolist()], [tuple(x) for x in tri2.tolist()]
    for step in range(0, 9):
        want = host.generate_pos_batch(a, b, step, 64)
        assert rec.equal("generate_pos_batch/%d" % step, want, lambda: ref["generate_pos_batch"](a, b, step, 64))
        got = dev.pos_batch(torch.as_tensor(tri.astype(np.int32)), torch.as_tensor(tri2.astype(np.int32)), step, 64)
        assert [tuple(x) for x in got.t().tolist()] == list(want[0]) + list(want[1])
