"""CPU tests of the host-side mirror of the reference interface: args, task_divide, batch slicing, id
assignment, dataset loading (against goldens generated from the reference: stored vectors and recorded results of its
read_kgs_from_folder), the host sampler's rules, Gale-Shapley, early_stop, and the `openea` drop-in import surface."""
import ast
import contextlib
import io
import json
import os
import random

import numpy as np
import pytest

from oracle import ref_adapter
from tests.helpers import ReferenceRecord

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "finding_golden.npz"))
REC = ReferenceRecord("reference_host_modules")


def test_args_loader(tmp_path):
    from openea_b200.modules.args.args_hander import load_args, check_args
    p = tmp_path / "a.json"
    p.write_text(json.dumps({"dim": 100, "embedding_module": "TransE", "neg_triple_num": 1, "top_k": [1, 5]}))
    with contextlib.redirect_stdout(io.StringIO()):
        a = load_args(str(p))
    assert a.dim == 100 and a.top_k == [1, 5]
    check_args(a)
    a.neg_triple_num = 2
    with pytest.raises(AssertionError):
        check_args(a)


def test_task_divide_golden():
    from openea_b200.modules.utils.util import task_divide, merge_dic
    want = ast.literal_eval(str(GOLD["task_divide"][0]))
    got = [task_divide(list(range(n)), t) for n, t in ((10, 3), (7, 7), (5, 8), (0, 2), (12, 4))]
    assert got == want
    assert merge_dic({1: 2}, {1: 3, 4: 5}) == {1: 3, 4: 5}


def test_pos_batch_slices_golden():
    from openea_b200.modules.train.batch import generate_pos_batch
    tl1 = [(i, 0, i + 1) for i in range(23)]
    tl2 = [(100 + i, 1, 101 + i) for i in range(11)]
    want = ast.literal_eval(str(GOLD["pos_batch_slices"][0]))
    assert [generate_pos_batch(tl1, tl2, 8, step) for step in range(5)] == want


def test_id_assignment_golden():
    from openea_b200.modules.load import read as rd
    t1 = {("a", "r1", "b"), ("a", "r1", "c"), ("b", "r2", "c")}
    t2 = {("x", "s1", "y"), ("y", "s1", "z"), ("z", "s2", "x"), ("y", "s2", "w"), ("w", "s1", "v")}
    i1, i2 = rd.generate_mapping_id(t1, {"a", "b", "c"}, t2, {"x", "y", "z", "w", "v"}, ordered=True)
    assert [str(sorted(i1.items())), str(sorted(i2.items()))] == GOLD["mapping_id"].tolist()
    # hand check of the interleaving: KG1 rank i → 2i, KG2 rank i → 2i+1, KG2 overflow continues after 2·n1
    assert i1 == {"c": 0, "b": 2, "a": 4} or set(i1.values()) == {0, 2, 4}
    assert sorted(i2.values()) == [1, 3, 5, 6, 7]
    i1, i2 = rd.generate_sharing_id([("a", "y")], t1, {"a", "b", "c"}, t2, {"x", "y", "z", "w", "v"}, ordered=True)
    assert [str(sorted(i1.items())), str(sorted(i2.items()))] == GOLD["sharing_id"].tolist()
    assert i2["y"] == i1["a"]


def test_host_sampler_rules():
    """generate_neg_triples_fast: k negatives per positive, same relation, exactly one side corrupted per
    negative, candidates from the neighbour list when present, known triples filtered (except last try)."""
    from openea_b200.modules.train.batch import generate_neg_triples_fast, generate_relation_triple_batch
    random.seed(1); np.random.seed(1)
    ents = list(range(0, 200, 2))
    triples = [(random.choice(ents), random.randrange(5), random.choice(ents)) for _ in range(300)]
    tset = set(triples)
    neigh = {e: random.sample(ents, 12) for e in ents[:50]}
    pos = triples[:64]
    neg = generate_neg_triples_fast(pos, tset, ents, 10, neighbor=neigh)
    assert len(neg) == 640
    for i, (h, r, t) in enumerate(pos):
        block = neg[10 * i:10 * i + 10]
        for nh, nr, nt in block:
            assert nr == r and ((nh == h) != (nt == t) or (nh, nr, nt) == (h, r, t))
            if nh != h and h in neigh:
                assert nh in neigh[h]
            if nt != t and t in neigh:
                assert nt in neigh[t]
    assert sum(1 for x in neg if x in tset) <= 2
    p, n = generate_relation_triple_batch(triples[:100], triples[100:], tset, tset, ents, ents, 40, 1, None, None, 3)
    assert len(n) == 3 * len(p) and len(p) == 40


def test_galeshapley_and_early_stop():
    from openea_b200.modules.finding.alignment import galeshapley
    from openea_b200.modules.finding.evaluation import early_stop
    suitors = {"x_0": ["y_0", "y_1"], "x_1": ["y_0", "y_1"]}
    reviewers = {"y_0": ["x_1", "x_0"], "y_1": ["x_0", "x_1"]}
    assert galeshapley(suitors, reviewers, 100) == {"x_1": "y_0", "x_0": "y_1"}
    with contextlib.redirect_stdout(io.StringIO()):
        assert early_stop(0.5, 0.4, 0.3) == (0.4, 0.3, True)
        assert early_stop(0.3, 0.4, 0.5) == (0.4, 0.5, False)
        assert early_stop(-1, -1, 0.2) == (-1, 0.2, False)


def test_calculate_rank_host_helper_matches_oracle():
    from openea_b200.modules.finding.alignment import calculate_rank
    from oracle import finding as orf
    rng = np.random.default_rng(0)
    s = rng.standard_normal((40, 60)).astype(np.float32)
    mr, mrr, hits, pairs = calculate_rank(list(range(40)), s, [1, 5], True, 40)
    top1, rank = orf.rank_rows(s)
    assert pairs == {(i, int(j)) for i, j in enumerate(top1)}
    assert hits == [int((rank < 1).sum()), int((rank < 5).sum())]
    assert mr == pytest.approx((rank + 1).mean()) and mrr == pytest.approx((1 / (rank + 1)).mean())


def test_openea_dropin_import_surface():
    """Every import of the reference's run/main_from_args.py:5-35 resolves, and `openea.*` aliases `openea_b200.*`."""
    import importlib
    import sys
    import openea  # noqa: F401
    for mod, names in (("openea.modules.args.args_hander", ["check_args", "load_args", "ARGs"]),
                       ("openea.modules.load.kgs", ["read_kgs_from_folder", "KGs"]),
                       ("openea.modules.load.kg", ["KG"]),
                       ("openea.modules.base.losses", ["get_loss_func", "margin_loss", "positive_loss", "limited_loss", "logistic_loss", "mapping_loss"]),
                       ("openea.modules.base.initializers", ["init_embeddings"]),
                       ("openea.modules.base.optimizers", ["generate_optimizer", "get_optimizer"]),
                       ("openea.modules.base.mapping", ["add_mapping_variables", "add_mapping_module"]),
                       ("openea.modules.train.batch", ["generate_relation_triple_batch", "generate_neg_triples_fast", "generate_neighbours_single_thread", "find_neighbours"]),
                       ("openea.modules.finding.similarity", ["sim", "csls_sim"]),
                       ("openea.modules.finding.alignment", ["greedy_alignment", "stable_alignment", "calculate_rank"]),
                       ("openea.modules.finding.evaluation", ["valid", "test", "early_stop"]),
                       ("openea.modules.bootstrapping.alignment_finder", ["find_alignment", "find_potential_alignment_mwgm", "find_potential_alignment_greedily", "search_nearest_k", "check_new_alignment"]),
                       ("openea.models.basic_model", ["BasicModel"]),
                       ("openea.models.trans", ["TransD", "TransE", "TransH", "TransR"]),
                       ("openea.models.semantic", ["DistMult", "HolE", "SimplE", "RotatE"]),
                       ("openea.models.neural", ["ConvE", "ProjE"]),
                       ("openea.approaches", ["AlignE", "BootEA", "JAPE", "Attr2Vec", "MTransE", "IPTransE", "GCN_Align", "AttrE", "IMUSE", "SEA", "MultiKE", "RSN4EA", "GMNN", "KDCoE", "RDGCN", "BootEA_RotatE", "BootEA_TransH", "AliNet"])):
        m = importlib.import_module(mod)
        for n in names:
            assert hasattr(m, n), "%s.%s" % (mod, n)
    assert sys.modules["openea.models.basic_model"] is sys.modules["openea_b200.models.basic_model"]
    from openea.models.basic_model import BasicModel
    for meth in ("set_args", "set_kgs", "init", "run", "valid", "test", "save", "retest", "predict"):
        assert callable(getattr(BasicModel, meth))
    from openea.approaches import KDCoE          # out-of-scope classes stay importable and say so when used
    with pytest.raises(NotImplementedError):
        KDCoE().init()


def _reference_kgs(folder, modes):
    """read_kgs_from_folder of the live reference (TensorFlow stubbed) for the given id modes."""
    if not REC.live:
        return None
    import importlib
    import sys
    import types
    saved = {k: v for k, v in sys.modules.items() if k == "openea" or k.startswith("openea.")}
    for k in saved:
        del sys.modules[k]
    sys.modules["tensorflow"] = types.ModuleType("tensorflow")
    pkg = types.ModuleType("openea")
    pkg.__path__ = [os.path.join(ref_adapter.REF_SRC, "openea")]
    sys.modules["openea"] = pkg
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            rk = importlib.import_module("openea.modules.load.kgs")
            return {m: rk.read_kgs_from_folder(folder, "721_5fold/1/", m, True) for m in modes}
    finally:
        for k in [k for k in sys.modules if k == "openea" or k.startswith("openea.")]:
            del sys.modules[k]
        sys.modules.pop("tensorflow", None)
        sys.modules.update(saved)


@pytest.mark.parametrize("loader", ["arrays", "containers", "arrays-cached"])
def test_dataset_loading_equals_live_reference(tmp_path, monkeypatch, loader):
    """Full read_kgs_from_folder equivalence with the reference on a synthetic folder, in all three id modes, for
    the array-backed loader (fresh parse and binary cache) and the container-based loader: id dicts, triple sets and
    lists incl. swap triples, every derived dict, vocabularies, counts, links, URI-level KGs."""
    from openea_b200.modules.load import fast
    from openea_b200.modules.load.kgs import read_kgs_from_folder
    from openea_b200.synth import write_dataset
    folder = str(tmp_path) + "/"
    write_dataset(folder, "tiny")
    monkeypatch.setenv("OEA_CACHE_DIR", str(tmp_path) + "/cache")
    if loader == "containers":
        monkeypatch.setenv("OEA_LOADER", "containers")
    modes = ("swapping", "mapping", "sharing")
    with contextlib.redirect_stdout(io.StringIO()) as log:
        mine = {m: read_kgs_from_folder(folder, "721_5fold/1/", m, True) for m in modes}
        if loader == "arrays-cached":
            mine = {m: read_kgs_from_folder(folder, "721_5fold/1/", m, True) for m in modes}
    if loader == "arrays-cached":
        assert log.getvalue().count("loaded from cache") == 3
    assert isinstance(mine["mapping"], fast.ArrayKGs) == (loader != "containers")
    theirs = _reference_kgs(folder, modes)

    def facts(k):
        f = {"nums": (k.entities_num, k.relations_num, k.attributes_num)}
        for side in ("kg1", "kg2", "uri_kg1", "uri_kg2"):
            g = getattr(k, side)
            names = ["relation_triples_set", "attribute_triples_set", "local_relation_triples_set", "rt_dict", "hr_dict",
                     "av_dict", "entity_relations_dict", "entity_attributes_dict", "entities_set", "relations_set",
                     "attributes_set", "entities_num", "relations_num", "attributes_num", "relation_triples_num",
                     "local_relation_triples_num", "attribute_triples_num", "local_attribute_triples_num"]
            if not side.startswith("uri"):
                names += ["entities_id_dict", "relations_id_dict", "attributes_id_dict", "sup_relation_triples_set",
                          "sup_attribute_triples_set"]
            for name in names:
                f[side + "." + name] = getattr(g, name)
            for lst in ("relation_triples_list", "local_relation_triples_list", "attribute_triples_list",
                        "local_attribute_triples_list", "entities_list", "relations_list", "attributes_list"):
                f[side + "." + lst] = (len(getattr(g, lst)), set(getattr(g, lst)))
        for part in ("train", "valid", "test"):
            for name in (part + "_links", part + "_entities1", "uri_%s_links" % part):
                f[name] = getattr(k, name)
        f["useful_entities_list1"] = set(k.useful_entities_list1)
        return f
    for m in mine:
        want = facts(theirs[m]) if REC.live else None
        for key, val in facts(mine[m]).items():
            assert REC.equal("tiny/%s/%s" % (m, key), val, lambda: want[key]), (m, key)


@pytest.mark.parametrize("case", ["clean", "dirty"])
def test_array_loader_edge_cases_equal_live_reference(tmp_path, monkeypatch, case):
    """Hand-written folder: duplicate lines, padded fields, values with a trailing '.', an entity that only carries
    attributes, a link naming an unknown entity, KGs of different sizes (id overflow branch), equal-frequency ties.
    'clean' stays on the array path; 'dirty' adds attribute lines with too few / too many fields, which the array
    path must hand to the container-based loader (same result as the reference either way)."""
    from openea_b200.modules.load import fast
    from openea_b200.modules.load.kgs import read_kgs_from_folder
    folder = str(tmp_path) + "/"
    os.makedirs(folder + "721_5fold/1")
    w = lambda name, text: open(folder + name, "w", encoding="utf8").write(text)
    w("rel_triples_1", "a\tp\tb\na\tp\tb\n b \tq\tc\nc\tp\ta\nd\tq\td\ne\tp\ta\nf\tr\tg\n")
    w("rel_triples_2", "x\tP\ty\ny\tQ\tz\nz\tP\tx\nx\tQ\tz\n")
    w("attr_triples_1", "a\tname\t\"Alice\" .\nb\tname\tBob.\nh\tage\t 42 \na\tname\t\"Alice\" .\n"
      + ("a\tonly-two-fields\n\nb\tnote\tx\ty z\n" if case == "dirty" else ""))
    w("attr_triples_2", "x\tlabel\tex\ny\tlabel\twhy.\n")
    w("ent_links", "a\tx\nb\ty\nc\tz\n")
    w("721_5fold/1/train_links", "a\tx\n")
    w("721_5fold/1/valid_links", "b\ty\n")
    w("721_5fold/1/test_links", "c\tz\nnobody\tz\n")
    monkeypatch.setenv("OEA_NO_DATASET_CACHE", "1")
    modes = ("swapping", "mapping", "sharing")
    with contextlib.redirect_stdout(io.StringIO()) as log:
        mine = {m: read_kgs_from_folder(folder, "721_5fold/1/", m, True) for m in modes}
    assert isinstance(mine["mapping"], fast.ArrayKGs) == (case == "clean")
    assert ("array-backed loader not applicable" in log.getvalue()) == (case == "dirty")
    theirs = _reference_kgs(folder, modes)

    def facts(k):
        f = {"nums": (k.entities_num, k.relations_num, k.attributes_num)}
        for side in ("kg1", "kg2"):
            for name in ("entities_id_dict", "relations_id_dict", "attributes_id_dict", "relation_triples_set",
                         "attribute_triples_set", "sup_relation_triples_set", "sup_attribute_triples_set", "rt_dict",
                         "hr_dict", "av_dict", "entity_attributes_dict", "entities_set"):
                f[side + "." + name] = getattr(getattr(k, side), name)
        for name in ("train_links", "valid_links", "test_links"):
            f[name] = getattr(k, name)
        return f
    for m in modes:
        want = facts(theirs[m]) if REC.live else None
        for key, val in facts(mine[m]).items():
            assert REC.equal("edge-%s/%s/%s" % (case, m, key), val, lambda: want[key]), (m, key)


def test_array_loader_refuses_what_only_the_container_loader_covers(tmp_path):
    from openea_b200.modules.load import fast
    from openea_b200.synth import write_dataset
    folder = write_dataset(str(tmp_path) + "/d/", "micro")
    with pytest.raises(fast.Unsupported):
        fast.load(folder, "721_5fold/1/", "mapping", False)                  # unordered ids: Python set iteration order
    with pytest.raises(fast.Unsupported):
        fast.load(folder, "721_5fold/1/", "mapping", True, remove_unlinked=True)
    rows = np.array([[3, 1, 2], [3, 1, 2], [0, 0, 0], [3, 1, 1]], dtype=np.int32)
    assert fast.unique_int_rows(rows).tolist() == [[3, 1, 2], [0, 0, 0], [3, 1, 1]]


@pytest.mark.parametrize("seed", range(8))
def test_array_loader_equals_container_loader_on_random_folders(tmp_path, monkeypatch, seed):
    """Random small datasets with everything that stresses the id assignment: equal occurrence counts (ties broken by
    name), non-ASCII and prefix-related names, KGs of very different sizes, entities that occur only in attribute
    triples, repeated lines.  Both loaders must agree on every id and every triple in all three id modes (the container
    loader is the line-by-line mirror of the reference, pinned above)."""
    from openea_b200.modules.load import fast
    from openea_b200.modules.load.kgs import read_kgs_from_folder
    rng = np.random.default_rng(seed)
    names = ["e%d" % i for i in range(12)] + ["é%d" % i for i in range(6)] + ["e1%d" % i for i in range(6)] + ["实体%d" % i for i in range(4)]
    folder = str(tmp_path) + "/"
    os.makedirs(folder + "721_5fold/1")
    sizes = [(int(rng.integers(8, 28)), int(rng.integers(20, 90))), (int(rng.integers(4, 12)), int(rng.integers(6, 40)))]
    ents = []
    for side, (n_e, n_t) in zip(("1", "2"), sizes):
        e = ["kg%s:%s" % (side, x) for x in rng.permutation(names)[:n_e]]
        ents.append(e)
        rels = ["kg%s:p%d" % (side, i) for i in range(int(rng.integers(1, 5)))]
        with open(folder + "rel_triples_" + side, "w", encoding="utf8") as f:
            for _ in range(n_t):
                f.write("%s\t%s\t%s\n" % (e[rng.integers(n_e)], rels[rng.integers(len(rels))], e[rng.integers(n_e)]))
        with open(folder + "attr_triples_" + side, "w", encoding="utf8") as f:
            for _ in range(int(rng.integers(3, 30))):
                who = e[rng.integers(n_e)] if rng.random() < 0.8 else "kg%s:attr-only%d" % (side, rng.integers(3))
                f.write("%s\tkg%s:a%d\t\"v %d\" .\n" % (who, side, rng.integers(4), rng.integers(6)))
    n_links = min(len(ents[0]), len(ents[1]))
    pairs = list(zip(rng.permutation(ents[0])[:n_links], rng.permutation(ents[1])[:n_links]))
    # only entities that occur in relation / attribute triples can be linked (the reference raises KeyError otherwise)
    with contextlib.redirect_stdout(io.StringIO()):
        monkeypatch.setenv("OEA_LOADER", "containers")
        known1 = {h for h, _, t in _quiet_read(folder + "rel_triples_1")} | {t for _, _, t in _quiet_read(folder + "rel_triples_1")}
        known2 = {h for h, _, t in _quiet_read(folder + "rel_triples_2")} | {t for _, _, t in _quiet_read(folder + "rel_triples_2")}
    pairs = [(a, b) for a, b in pairs if a in known1 and b in known2]
    if len(pairs) < 3:
        pytest.skip("degenerate draw")
    cut = max(1, len(pairs) // 3)
    for name, part in (("train", pairs[:cut]), ("valid", pairs[cut:2 * cut]), ("test", pairs[2 * cut:])):
        with open(folder + "721_5fold/1/%s_links" % name, "w", encoding="utf8") as f:
            f.writelines("%s\t%s\n" % p for p in part)
    monkeypatch.setenv("OEA_NO_DATASET_CACHE", "1")
    for mode in ("mapping", "sharing", "swapping"):
        with contextlib.redirect_stdout(io.StringIO()):
            monkeypatch.setenv("OEA_LOADER", "containers")
            want = read_kgs_from_folder(folder, "721_5fold/1/", mode, True)
            monkeypatch.setenv("OEA_LOADER", "arrays")
            got = read_kgs_from_folder(folder, "721_5fold/1/", mode, True)
        assert isinstance(got, fast.ArrayKGs) and not isinstance(want, fast.ArrayKGs)
        assert (got.entities_num, got.relations_num, got.attributes_num) == (want.entities_num, want.relations_num, want.attributes_num)
        for side in ("kg1", "kg2"):
            a, b = getattr(got, side), getattr(want, side)
            for name in ("entities_id_dict", "relations_id_dict", "attributes_id_dict", "relation_triples_set",
                         "attribute_triples_set", "sup_relation_triples_set", "sup_attribute_triples_set", "rt_dict",
                         "hr_dict", "av_dict", "entity_relations_dict", "entity_attributes_dict", "entities_set"):
                assert getattr(a, name) == getattr(b, name), (mode, side, name)
        assert got.train_links == want.train_links and got.valid_links == want.valid_links and got.test_links == want.test_links


def _quiet_read(path):
    from openea_b200.modules.load import read as rd
    with contextlib.redirect_stdout(io.StringIO()):
        return rd.read_relation_triples(path)[0]


def test_mwgm_exact_is_optimal_where_greedy_is_not():
    """alignment_finder.mwgm_igraph's counterpart (exact maximum-weight bipartite matching via the doubled-graph
    assignment) against brute force on random small candidate graphs; greedy (graph-tool heuristic's counterpart) is a
    1/2-approximation and differs on the textbook case."""
    import itertools
    from openea_b200.modules.bootstrapping import alignment_finder as af
    sim = {(0, 0): 0.9, (0, 1): 0.85, (1, 0): 0.85}
    assert af.mwgm_greedy(list(sim), sim) == {(0, 0)}
    assert af.mwgm_exact(list(sim), sim) == {(0, 1), (1, 0)} == af.mwgm(list(sim), sim, af.mwgm_igraph)
    rng = np.random.default_rng(0)
    for _ in range(150):
        n1, n2 = rng.integers(2, 7, 2)
        edges = [(i, j) for i in range(n1) for j in range(n2) if rng.random() < 0.5]
        if not edges:
            continue
        w = {e: float(rng.random() * 0.5 + 0.5) for e in edges}
        got = af.mwgm_exact(edges, w)
        assert len({a for a, _ in got}) == len(got) == len({b for _, b in got}) and got <= set(edges)
        best = max(sum(w[e] for e in sub) for r in range(min(n1, n2) + 1) for sub in itertools.combinations(edges, r)
                   if len({a for a, _ in sub}) == r and len({b for _, b in sub}) == r)
        assert abs(sum(w[e] for e in got) - best) < 1e-9
        assert sum(w[e] for e in af.mwgm_greedy(edges, w)) >= 0.5 * best - 1e-9


def test_pair_set_behaves_like_the_reference_set():
    """finding.PairSet (what greedy_alignment returns instead of a 70 000-tuple Python set) against a real set."""
    from openea_b200.finding import PairSet
    top1 = np.array([3, 0, 0, 2], dtype=np.int32)
    ps, real = PairSet(top1), {(0, 3), (1, 0), (2, 0), (3, 2)}
    assert len(ps) == 4 and set(ps) == real and ps == real and real == ps
    assert (1, 0) in ps and (1, 1) not in ps and (9, 0) not in ps and "x" not in ps
    assert ps - {(0, 3)} == real - {(0, 3)} and ps | {(7, 7)} == real | {(7, 7)} and ps & {(2, 0), (5, 5)} == {(2, 0)}
    assert sorted(ps) == sorted(real) and [(i, j) for i, j in ps][0] == (0, 3)


def test_galeshapley_port_equals_the_reference_function():
    """The host restatement of galeshapley against the reference's own function (recorded with TF stubbed) on
    random preference structures, including max_iteration cut-offs that stop before everybody is matched."""
    import copy
    from openea_b200.modules.finding.alignment import arg_sort, galeshapley
    ref = ref_adapter.load().alignment if REC.live else None
    rng = np.random.default_rng(5)
    for n1, n2, cut in ((12, 12, 100), (20, 15, 100), (15, 20, 3), (30, 30, 2)):
        s = rng.standard_normal((n1, n2)).astype(np.float32)
        a = arg_sort(list(range(n1)), s, "x_", "y_"); b = arg_sort(list(range(n2)), s.T, "y_", "x_")
        if n1 > n2 and cut >= n2:
            continue      # more suitors than reviewers and unlimited rounds: the reference runs lists empty (IndexError)
        got = galeshapley(copy.deepcopy(a), copy.deepcopy(b), cut)
        assert REC.equal("galeshapley/%d-%d-%d" % (n1, n2, cut), got,
                         lambda: ref.galeshapley(copy.deepcopy(a), copy.deepcopy(b), cut)), (n1, n2, cut)
