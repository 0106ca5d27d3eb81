"""CPU: IPTransE's host / index layer (openea_b200/approaches/iptranse.py) — the two-step path table against a
brute-force statement of iptranse.py:98-121 and against recorded results of the reference's own pandas source, the
triples of latent aligned entities against the reference's dict walk, and the whole approach
(PTransE epochs + an alignment epoch) on the CPU warp emulator."""
import collections
import re

import numpy as np
import pytest
import torch

from openea_b200.approaches import iptranse as ipt
from oracle import reference_source as ref_src
from tests.helpers import ReferenceRecord
from tests.test_emu_triple_core import cpu_engine      # noqa: F401  (fixture: the engine over the emulated library)

REC = ReferenceRecord("reference_iptranse")


def random_kg(rng, n_ent, n_rel, n_tri):
    t = np.stack([rng.integers(0, n_ent, n_tri), rng.integers(0, n_rel, n_tri), rng.integers(0, n_ent, n_tri)], 1)
    return np.unique(t, axis=0)


def brute_paths(tri):
    size = collections.Counter((h, r) for h, r, _ in tri)
    by_head = collections.defaultdict(list)
    direct = collections.defaultdict(list)
    for h, r, t in tri:
        by_head[h].append((r, t))
        direct[(h, t)].append(r)
    rows = []
    for h, rx, m in tri:
        for ry, t in by_head[m]:
            w = size[(h, rx)] * size[(m, ry)]
            if w < 101:
                rows.extend((rx, ry, r, float(w)) for r in direct[(h, t)])
    return collections.Counter(rows)


@pytest.mark.parametrize("seed,n_ent,n_rel,n_tri", [(0, 12, 3, 60), (1, 40, 6, 300), (2, 5, 2, 40)])
def test_two_step_paths_equal_a_brute_force_join(seed, n_ent, n_rel, n_tri):
    tri = random_kg(np.random.default_rng(seed), n_ent, n_rel, n_tri)
    for chunk in (7, 4_000_000):
        rows, w = ipt.two_step_paths(tri, chunk=chunk)
        got = collections.Counter((int(a), int(b), int(c), float(x)) for (a, b, c), x in zip(rows, w))
        assert got == brute_paths([tuple(int(v) for v in t) for t in tri])
    assert ipt.two_step_paths(np.zeros((0, 3), np.int64))[0].shape == (0, 3)


def test_two_step_paths_and_latent_triples_equal_the_reference_source():
    ref = ref_src.iptranse_helpers() if REC.live else None
    rng = np.random.default_rng(5)
    tri = random_kg(rng, 60, 7, 500)
    rows, w = ipt.two_step_paths(tri)
    assert REC.equal("generate_2steps_path",
                     collections.Counter((int(a), int(b), int(c), float(x)) for (a, b, c), x in zip(rows, w)),
                     lambda: collections.Counter((int(a), int(b), int(c), float(w)) for a, b, c, w in
                                                 ref["generate_2steps_path"]([tuple(int(v) for v in t) for t in tri])))

    # triples of latent aligned entities: kg1 over ids 0..59, kg2 over 60..119; several kg1 entities may share a partner
    tri2 = random_kg(rng, 60, 7, 400) + np.array([60, 0, 60])
    class KG:
        def __init__(self, t):
            self.rt_dict, self.hr_dict = collections.defaultdict(set), collections.defaultdict(set)
            for h, r, tt in t:
                self.rt_dict[int(h)].add((int(r), int(tt)))
                self.hr_dict[int(tt)].add((int(h), int(r)))
    class KGs:
        kg1, kg2 = KG(tri), KG(tri2)
    ents1 = rng.choice(60, 25, replace=False)
    ents2 = rng.integers(60, 120, 25)
    ws = rng.random(25).astype(np.float32)
    t1, t2 = torch.as_tensor(tri.astype(np.int32)), torch.as_tensor(tri2.astype(np.int32))
    e1, e2, w = torch.as_tensor(ents1), torch.as_tensor(ents2), torch.as_tensor(ws)
    a, wa = ipt.latent_triples(ipt._by_column(t1, 0, 120), ipt._by_column(t1, 2, 120), e1, e2, w)
    b, wb = ipt.latent_triples(ipt._by_column(t2, 0, 120), ipt._by_column(t2, 2, 120), e2, e1, w)
    got_t, got_w = ipt.distinct_weighted(torch.cat([a, b]), torch.cat([wa, wb]), 120, 7)
    got = {(int(h), int(r), int(t), float(x)) for (h, r, t), x in zip(got_t.tolist(), got_w.tolist())}
    assert REC.equal("generate_triples_of_latent_ents", got, lambda: ref["generate_triples_of_latent_ents"](
        KGs, [int(e) for e in ents1], [int(e) for e in ents2], [float(x) for x in ws]))
    assert len(got) == got_t.shape[0]


def test_iptranse_lifecycle_on_the_emulator(cpu_engine, monkeypatch, tmp_path, capsys):
    """init / run of IPTransE on a 40-entity synthetic dataset with the kernels' sources on the CPU emulator: PTransE
    epochs (sampled triple scorer + weighted path scorer, one Adagrad step), then an alignment epoch on the triples of
    latent aligned entities.  The candidate search (a K3 kernel, GPU only) is stood in by a dense matmul."""
    from openea_b200 import finding, presets
    from openea_b200.approaches import IPTransE
    from openea_b200.modules.base import initializers
    from openea_b200.modules.load.kgs import read_kgs_from_folder
    from openea_b200.synth import write_dataset
    monkeypatch.setattr(initializers, "_make", lambda values, norm, optimizer=None: cpu_engine.EmbeddingTable(
        values, bool(norm), optimizer or "Adagrad", "cpu"))
    monkeypatch.setattr(ipt, "load_session", lambda: None)

    def candidates(e1, e2, sim_th, k, metric, normalize):
        s = e1 @ e2.t()
        vals, cols = s.max(1)
        keep = vals > sim_th
        return torch.arange(e1.shape[0], dtype=torch.int32)[keep], cols[keep].to(torch.int32), vals[keep]
    monkeypatch.setattr(finding, "find_alignment_device", candidates)
    folder = write_dataset(str(tmp_path) + "/micro/", "micro")
    args = presets.iptranse("15K")
    args.training_data, args.output = folder, str(tmp_path) + "/out/"
    args.batch_size, args.max_epoch, args.start_valid, args.dim, args.bp_freq, args.sim_th = 64, 4, 1000, 16, 2, 0.05
    kgs = read_kgs_from_folder(folder, args.dataset_division, "sharing", args.ordered)
    model = IPTransE()
    model.set_args(args)
    model.set_kgs(kgs)
    model.init()
    assert model.paths1.shape[0] > 0 and model.paths2.shape[0] > 0
    pos, neg, w = model._path_batch(20)
    assert pos.shape == neg.shape == (3, 20) and w.shape == (20,)
    assert torch.equal(pos[:2], neg[:2])                                    # only the direct relation is replaced
    rels1 = set(kgs.kg1.relations_list)
    n1 = int(model.paths1.shape[0] / (model.paths1.shape[0] + model.paths2.shape[0]) * 20)
    assert set(neg[2, :n1].tolist()) <= rels1
    before = model.ent_embeds.weight.clone(), model.rel_embeds.weight.clone()
    acc_before = model.alignment_trainer.ent.state1.clone()
    model.run()
    out = capsys.readouterr().out
    losses = [float(x) for x in re.findall(r"avg\. triple loss: ([0-9.]+)", out)]
    assert len(losses) == 3 and all(np.isfinite(losses)) and losses[0] > 0          # epochs 1 .. max_epoch − 1
    assert "newly triples:" in out and re.search(r"epoch 2, alignment loss: [0-9.]+", out)
    assert not torch.equal(before[0], model.ent_embeds.weight) and not torch.equal(before[1], model.rel_embeds.weight)
    assert torch.isfinite(model.ent_embeds.weight).all()
    # the alignment optimiser owns its Adagrad accumulators
    assert not torch.equal(acc_before, model.alignment_trainer.ent.state1)
    assert model.alignment_trainer.ent.weight.data_ptr() == model.ent_embeds.weight.data_ptr()
