"""Generates tests/golden/path_i_reference_graphs.npz by EXECUTING the reference's own graph-definition code for path
(i) — `_define_variables`, `_define_embed_graph`, `_define_alignment_graph`, the mapping module, and
`session.run([loss, optimizer], feed_dict)` — on oracle/tf1_shim.py (a TensorFlow-1 graph interpreter on torch float64;
TensorFlow itself is not installable here).  Runs with OPENEA_REFERENCE set to a checkout of the original project; the
fixture it writes is what travels.  Per case: the variables' start values, every run's feeds, the fetched loss of every run and all variables
after the last run.

    OPENEA_REFERENCE=/path/to/OpenEA python scripts/make_golden_path_i.py
"""
import importlib
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # never write into the reference checkout
from oracle import tf1_shim  # noqa: E402

REF_SRC = os.path.join(os.environ.get("OPENEA_REFERENCE", ""), "src")
OUT = os.path.join(ROOT, "tests", "golden", "path_i_reference_graphs.npz")
N_ENT, N_REL = 40, 6


class _Stub(types.ModuleType):
    def __getattr__(self, key):
        if key.startswith("__"):
            raise AttributeError(key)
        return lambda *a, **kw: None


def _accept_np_matrix():
    """The reference passes np.matrix to sklearn.preprocessing.normalize (initializers.py:49), which current scikit-learn
    rejects: convert on the way in (environment compatibility only — the values are overwritten by the goldens)."""
    from sklearn import preprocessing
    if not getattr(preprocessing.normalize, "_oea_wrapped", False):
        orig = preprocessing.normalize
        wrapped = lambda X, *a, **kw: orig(np.asarray(X), *a, **kw)
        wrapped._oea_wrapped = True
        preprocessing.normalize = wrapped


def import_reference(name):
    """Import a reference module with `tensorflow` = the shim and absent third-party packages stubbed."""
    sys.modules["tensorflow"] = tf1_shim
    _accept_np_matrix()
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    for _ in range(40):
        try:
            return importlib.import_module(name)
        except ModuleNotFoundError as exc:
            sys.modules[exc.name] = _Stub(exc.name)
    raise RuntimeError("could not import " + name)


BASE = dict(dim=12, init="normal", ent_l2_norm=True, rel_l2_norm=True, loss_norm="L2", learning_rate=0.01,
            optimizer="Adagrad", batch_size=16, neg_triple_num=3, margin=1.5, pos_margin=0.01, neg_margin=2.0,
            neg_margin_balance=0.2, alpha=5, loss="limited", path_parm=0.1, alpha_1=2.5, alpha_2=0.25, sub_epoch=1)

# case → (module, class, args overrides, graph-definition calls, runs); a run is (kind, number of negatives per positive)
CASES = {
    "aligne_limited": ("openea.approaches.aligne", "AlignE", {}, ["_define_variables", "_define_embed_graph"],
                       [("triple", 3), ("triple", 3)]),
    "bootea": ("openea.approaches.bootea", "BootEA", {},
               ["_define_variables", "_define_embed_graph", "_define_alignment_graph"],
               [("triple", 3), ("align", 0), ("triple", 3), ("align", 0)]),
    "mtranse": ("openea.approaches.mtranse", "MTransE", dict(init="unit"),
                ["_define_variables", "_define_mapping_variables", "_define_embed_graph", "_define_mapping_graph"],
                [("triple", 0), ("mapping", 0), ("triple", 0), ("mapping", 0)]),
    "transe_margin_l1_sgd": ("openea.models.trans.transe", "TransE", dict(loss="margin-based", loss_norm="L1", optimizer="SGD"),
                             ["_define_variables", "_define_embed_graph"], [("triple", 1), ("triple", 1)]),
    "transe_margin_adam": ("openea.models.trans.transe", "TransE", dict(loss="margin-based", optimizer="Adam"),
                           ["_define_variables", "_define_embed_graph"], [("triple", 1), ("triple", 1), ("triple", 1)]),
    "transe_logistic_adadelta_nonorm": ("openea.models.trans.transe", "TransE",
                                        dict(loss="logistic", optimizer="Adadelta", ent_l2_norm=False, rel_l2_norm=False,
                                             learning_rate=1.0),
                                        ["_define_variables", "_define_embed_graph"], [("triple", 2), ("triple", 2)]),
    "transe_limited_d75": ("openea.models.trans.transe", "TransE", dict(dim=75), ["_define_variables", "_define_embed_graph"],
                           [("triple", 3), ("triple", 3)]),
    "transh": ("openea.models.trans.transh", "TransH", dict(loss="margin-based"), ["_define_variables", "_define_embed_graph"],
               [("triple", 1), ("triple", 1)]),
    "transd": ("openea.models.trans.transd", "TransD", dict(loss="margin-based"), ["_define_variables", "_define_embed_graph"],
               [("triple", 1), ("triple", 1)]),
    "distmult": ("openea.models.semantic.distmult", "DistMult", {}, ["_define_variables", "_define_embed_graph"],
                 [("label", 2), ("label", 2)]),
    "simple": ("openea.models.semantic.simple", "SimplE", {}, ["_define_variables", "_define_embed_graph"],
               [("triple", 2), ("triple", 2)]),
    "bootea_transh": ("openea.approaches.bootea_transh", "BootEA_TransH", {},
                      ["_define_variables", "_define_embed_graph", "_define_alignment_graph"],
                      [("triple", 3), ("align", 0), ("triple", 3)]),
    "jape": ("openea.approaches.jape", "JAPE", dict(neg_alpha=0.1), ["_define_variables", "_define_embed_graph"],
             [("triple", 2), ("triple", 2)]),
    "iptranse": ("openea.approaches.iptranse", "IPTransE", dict(neg_triple_num=1),
                 ["_define_variables", "_define_embed_graph", "_define_alignment_graph"],
                 [("ptranse", 1), ("ipt_align", 1), ("ptranse", 1)]),
    "sea": ("openea.approaches.sea", "SEA", dict(loss="margin-based", optimizer="Adam", neg_triple_num=1),
            ["_define_variables", "_define_embed_graph"], [("triple", 1), ("sea_map", 0), ("triple", 1), ("sea_map", 0)]),
    "imuse": ("openea.approaches.imuse", "IMUSE", dict(loss="margin-based", optimizer="SGD", neg_triple_num=1),
              ["_define_variables", "_define_embed_graph"], [("triple", 1), ("imuse_align", 0), ("triple", 1)]),
}


def triple_batch(rng, n, k):
    pos = np.stack([rng.integers(0, N_ENT, n), rng.integers(0, N_REL, n), rng.integers(0, N_ENT, n)]).astype(np.int32)
    if k == 0:
        return pos, None
    neg = np.repeat(pos, k, axis=1)
    side = rng.random(n * k) < 0.5
    neg[0, side] = rng.integers(0, N_ENT, int(side.sum()))
    neg[2, ~side] = rng.integers(0, N_ENT, int((~side).sum()))
    return pos, neg


def make_run(kind, k, rng, model):
    """→ (fetch attribute names, {placeholder attribute: array})."""
    n = 16
    if kind == "triple":
        pos, neg = triple_batch(rng, n, k)
        feed = {"pos_hs": pos[0], "pos_rs": pos[1], "pos_ts": pos[2]}
        if neg is not None:
            feed.update({"neg_hs": neg[0], "neg_rs": neg[1], "neg_ts": neg[2]})
        return ("triple_loss", "triple_optimizer"), feed
    if kind == "label":
        pos, neg = triple_batch(rng, n, k)
        both = np.concatenate([pos, neg], 1)
        label = np.concatenate([np.ones(n), -np.ones(n * k)]).astype(np.float32)
        return ("triple_loss", "triple_optimizer"), {"hs": both[0], "rs": both[1], "ts": both[2], "label": label}
    if kind == "align":
        pos, _ = triple_batch(rng, n, 0)
        return ("alignment_loss", "alignment_optimizer"), {"new_h": pos[0], "new_r": pos[1], "new_t": pos[2]}
    if kind == "mapping":
        return ("mapping_loss", "mapping_optimizer"), {"seed_entities1": rng.integers(0, N_ENT, 9).astype(np.int32),
                                                       "seed_entities2": rng.integers(0, N_ENT, 9).astype(np.int32)}
    if kind == "ptranse":
        pos, neg = triple_batch(rng, n, 1)
        m = 11
        path = rng.integers(0, N_REL, (3, m)).astype(np.int32)
        npath = path.copy()
        npath[2] = rng.integers(0, N_REL, m)
        feed = {"pos_hs": pos[0], "pos_rs": pos[1], "pos_ts": pos[2], "neg_hs": neg[0], "neg_rs": neg[1], "neg_ts": neg[2],
                "pos_rx": path[0], "pos_ry": path[1], "pos_r": path[2], "neg_rx": npath[0], "neg_ry": npath[1],
                "neg_r": npath[2], "path_weight": rng.integers(1, 100, m).astype(np.float32)}
        return ("train_loss", "optimizer"), feed
    if kind == "ipt_align":
        pos, neg = triple_batch(rng, n, 1)
        return ("alignment_loss", "alignment_optimizer"), {
            "new_ph": pos[0], "new_pr": pos[1], "new_pt": pos[2], "new_nh": neg[0], "new_nr": neg[1], "new_nt": neg[2],
            "tr_weight": (rng.random(n) * 0.3 + 0.7).astype(np.float32)}
    if kind == "sea_map":
        ids = lambda m: rng.integers(0, N_ENT, m).astype(np.int32)
        return ("mapping_loss", "mapping_optimizer"), {"labeled_entities1": ids(7), "labeled_entities2": ids(7),
                                                       "unlabeled_entities1": ids(10), "unlabeled_entities2": ids(10)}
    if kind == "imuse_align":
        return ("align_loss", "align_optimizer"), {"aligned_ents1": rng.integers(0, N_ENT, 8).astype(np.int32),
                                                   "aligned_ents2": rng.integers(0, N_ENT, 8).astype(np.int32)}
    raise ValueError(kind)


def generate():
    out, meta = {}, {}
    for case, (module, cls, overrides, defines, runs) in CASES.items():
        tf1_shim.reset_default_graph()
        mod = import_reference(module)
        args = dict(BASE)
        args.update(overrides)
        model = getattr(mod, cls)()
        model.args = types.SimpleNamespace(**args)
        model.kgs = types.SimpleNamespace(entities_num=N_ENT, relations_num=N_REL)
        for name in defines:
            getattr(model, name)()
        session = tf1_shim.Session()
        rng = np.random.default_rng(sum(map(ord, case)))
        variables = tf1_shim.trainable_variables()
        names = [v.name for v in variables]
        assert len(set(names)) == len(names), names
        for v in variables:
            shape = tuple(v.value.shape)
            if v.name.startswith("mapping_matrix"):
                start = np.linalg.qr(rng.standard_normal(shape))[0]
            else:
                start = rng.standard_normal(shape) * 2.0 / np.sqrt(shape[1])
            start = start.astype(np.float32).astype(np.float64)          # exactly representable in the engine's fp32
            v.assign_numpy(start)
            out["%s/var0/%s" % (case, v.name)] = start
        run_meta = []
        for i, (kind, k) in enumerate(runs):
            fetch, feed = make_run(kind, k, rng, model)
            loss, _ = session.run([getattr(model, fetch[0]), getattr(model, fetch[1])],
                                  feed_dict={getattr(model, key): val for key, val in feed.items()})
            out["%s/run%d/loss" % (case, i)] = np.float64(loss)
            for key, val in feed.items():
                out["%s/run%d/feed/%s" % (case, i, key)] = val
            run_meta.append({"kind": kind, "k": k, "fetch": list(fetch)})
        for v in variables:
            out["%s/var_final/%s" % (case, v.name)] = v.value.detach().numpy().copy()
        meta[case] = {"class": module + "." + cls, "args": args, "defines": defines, "runs": run_meta, "variables": names}
        print("%-34s %s  losses %s" % (case, names, ["%.6g" % float(out["%s/run%d/loss" % (case, i)]) for i in range(len(runs))]))
    out["meta"] = np.frombuffer(json.dumps(meta, sort_keys=True).encode(), dtype=np.uint8)
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


def generate_attre():
    """AttrE (approaches/attre.py:109-188): the structure loss, the character-level loss over composed literal vectors
    (n-gram compositional function with its tf.while_loop) and the joint loss, each with its own SGD optimiser.
    → tests/golden/path_i_attre.npz"""
    mod = import_reference("openea.approaches.attre")
    tf = tf1_shim
    tf.reset_default_graph()
    rng = np.random.default_rng(41)
    n_attr, n_val, n_char, lit, batch, dim = 5, 30, 9, 4, 8, 12
    chars = rng.integers(0, n_char, (n_val, lit))
    chars[rng.random((n_val, lit)) < 0.15] = 0                    # padding / rare characters
    model = mod.AttrE()
    model.args = types.SimpleNamespace(**dict(BASE, loss="margin-based", optimizer="SGD", neg_triple_num=1, batch_size=batch,
                                              literal_len=lit, attr_l2_norm=True, char_l2_norm=True, dim=dim))
    model.kgs = types.SimpleNamespace(entities_num=N_ENT, relations_num=N_REL, attributes_num=n_attr)
    model.value_id_char_ids, model.char_list_size = chars.tolist(), n_char
    model._define_variables()
    model._define_embed_graph()
    variables = tf.trainable_variables()
    out = {"chars": chars.astype(np.int32), "dims": np.array([n_attr, n_val, n_char, lit, batch, dim])}
    for v in variables:
        start = (rng.standard_normal(tuple(v.value.shape)) * 2.0 / np.sqrt(dim)).astype(np.float32).astype(np.float64)
        v.assign_numpy(start)
        out["var0/" + v.name] = start
    session = tf.Session()
    kinds = ["triple", "ce", "joint", "ce", "triple", "joint"]
    for i, kind in enumerate(kinds):
        if kind == "triple":
            fetch, feed = make_run("triple", 1, rng, model)
        elif kind == "ce":
            pos = np.stack([rng.integers(0, N_ENT, batch), rng.integers(0, n_attr, batch), rng.integers(0, n_val, batch)])
            neg = pos.copy()
            neg[0] = rng.integers(0, N_ENT, batch)
            fetch = ("triple_loss_ce", "triple_optimizer_ce")
            feed = {"pos_es": pos[0], "pos_as": pos[1], "pos_vs": pos[2], "neg_es": neg[0], "neg_as": neg[1], "neg_vs": neg[2]}
        else:
            fetch, feed = ("joint_loss", "optimizer_joint"), {"joint_ents": rng.permutation(N_ENT)[:25]}
        loss, _ = session.run([getattr(model, fetch[0]), getattr(model, fetch[1])],
                              feed_dict={getattr(model, key): np.asarray(val) for key, val in feed.items()})
        out["run%d/loss" % i] = np.float64(loss)
        out["run%d/kind" % i] = np.frombuffer(kind.encode(), dtype=np.uint8)
        for key, val in feed.items():
            out["run%d/feed/%s" % (i, key)] = np.asarray(val).astype(np.int32)
    for v in variables:
        out["var_final/" + v.name] = v.value.detach().numpy().copy()
    print("attre: losses %s" % ["%.6g" % float(out["run%d/loss" % i]) for i in range(len(kinds))], [v.name for v in variables])
    path = os.path.join(ROOT, "tests", "golden", "path_i_attre.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def generate_gcn_align():
    """Path (ii), GCN-Align: the reference's GCN_Align_Unit (gcn_align.py:498-539) for the structure branch (featureless,
    l2-normalised entity table) and the attribute branch (sparse features · weights), its align_loss and its
    GradientDescentOptimizer, fed through GCN_Utils.construct_feed_dict exactly as train_embeddings does (:737-757).
    → tests/golden/path_ii_gcn_align.npz"""
    import scipy.sparse as sp
    mod = import_reference("openea.approaches.gcn_align")
    tf = tf1_shim
    rng = np.random.default_rng(11)
    n, n_feat, dim, t, k = 30, 9, 8, 7, 3
    a = sp.random(n, n, density=0.12, random_state=3, format="coo")
    a = a + a.T + sp.eye(n)
    deg = np.asarray(a.sum(1)).ravel()
    a = sp.coo_matrix(sp.diags(deg ** -0.5) @ a @ sp.diags(deg ** -0.5))
    support = [(np.vstack((a.row, a.col)).transpose(), a.data.astype(np.float32).astype(np.float64), a.shape)]
    feat = sp.coo_matrix((rng.random((n, n_feat)) < 0.3).astype(np.float64))
    features = (np.vstack((feat.row, feat.col)).transpose(), feat.data, feat.shape)
    ill = np.stack([rng.permutation(n)[:t], rng.permutation(n)[:t]], 1)
    args = types.SimpleNamespace(learning_rate=8.0, gamma=3.0, neg_triple_num=k, dropout=0.0, support_number=1)
    out = {"support/coords": support[0][0], "support/values": support[0][1], "features/coords": features[0],
           "features/values": features[1], "ill": ill,
           "dims": np.array([n, n_feat, dim, t, k]), "gamma": np.float64(args.gamma), "lr": np.float64(args.learning_rate)}
    for branch, featureless in (("se", True), ("ae", False)):
        tf.reset_default_graph()
        ph = {"support": [tf.sparse_placeholder(tf.float32)],
              "features": tf.placeholder(tf.float32) if featureless else tf.sparse_placeholder(tf.float32),
              "dropout": tf.placeholder_with_default(0., shape=()),
              "num_features_nonzero": tf.placeholder_with_default(0, shape=())}
        model = mod.GCN_Align_Unit(args, ph, input_dim=n if featureless else n_feat, output_dim=dim, ILL=ill,
                                   sparse_inputs=not featureless, featureless=featureless, logging=False)
        (var,) = tf.trainable_variables()
        start = (rng.standard_normal(tuple(var.value.shape)) * 0.5).astype(np.float32).astype(np.float64)
        var.assign_numpy(start)
        out[branch + "/var0"] = start
        session = tf.Session()
        for step in range(3):
            neg = {key: rng.integers(0, n, t * k) for key in ("neg_left", "neg_right", "neg2_left", "neg2_right")}
            feed = mod.GCN_Utils.construct_feed_dict(1. if featureless else features, support, ph)
            feed.update({ph["dropout"]: args.dropout})
            feed.update({key + ":0": val for key, val in neg.items()})
            loss, _ = session.run([model.loss, model.opt_op], feed_dict=feed)
            out["%s/run%d/loss" % (branch, step)] = np.float64(loss)
            for key, val in neg.items():
                out["%s/run%d/%s" % (branch, step, key)] = val.astype(np.int32)
        out[branch + "/var_final"] = var.value.detach().numpy().copy()
        out[branch + "/outputs_final"] = session.run(model.outputs, feed_dict=feed)
        print("gcn_align %s: losses %s" % (branch, ["%.6g" % float(out["%s/run%d/loss" % (branch, i)]) for i in range(3)]))
    path = os.path.join(ROOT, "tests", "golden", "path_ii_gcn_align.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


RDGCN_NAMES = ["X0", "self.W", "self.f1.w", "self.f1.b", "self.f2.w", "self.f2.b", "sp1.w", "sp1.b", "dual.W", "dual.b",
               "dual.f1.w", "dual.f1.b", "dual.f2.w", "dual.f2.b", "sp2.w", "sp2.b", "diag1.w", "hw1.W", "hw1.b",
               "diag2.w", "hw2.W", "hw2.b"]       # the reference's variables in creation order (rdgcn.py:317-338)


def generate_rdgcn():
    """Path (ii), RDGCN: the reference's Layer.build() (rdgcn.py:160-338: dual relation graph, self / dual attention,
    per-edge relation attention, diagonal GCN layers, highway gates, L1 alignment loss) and its AdamOptimizer.
    → tests/golden/path_ii_rdgcn.npz"""
    mod = import_reference("openea.approaches.rdgcn")
    tf = tf1_shim
    rng = np.random.default_rng(21)
    n_ent, n_rel, dim, t, k = 24, 4, 8, 5, 3
    tri1 = np.unique(np.stack([rng.integers(0, 12, 30), rng.integers(0, n_rel, 30), rng.integers(0, 12, 30)], 1), axis=0)
    tri2 = np.unique(np.stack([rng.integers(12, 24, 30), rng.integers(0, n_rel, 30), rng.integers(12, 24, 30)], 1), axis=0)
    as_list = lambda a: [tuple(int(v) for v in row) for row in a]
    links = [(int(a), int(b)) for a, b in zip(rng.permutation(12)[:t], 12 + rng.permutation(12)[:t])]
    kgs = types.SimpleNamespace(train_links=links, relations_num=n_rel, entities_num=n_ent,
                                kg1=types.SimpleNamespace(relation_triples_list=as_list(tri1)),
                                kg2=types.SimpleNamespace(relation_triples_list=as_list(tri2)))
    args = types.SimpleNamespace(dim=dim, dropout=0.0, gamma=1.0, neg_triple_num=k, alpha=0.1, beta=0.3, learning_rate=0.01)
    embedding = (rng.standard_normal((n_ent, dim)) * 0.5).astype(np.float32)
    layer = mod.Layer(args, kgs, embedding)
    output, loss = layer.build()
    train_op = tf.train.AdamOptimizer(args.learning_rate).minimize(loss)
    variables = tf.trainable_variables()
    assert len(variables) == len(RDGCN_NAMES), [v.name for v in variables]
    out = {"triples1": tri1.astype(np.int32), "triples2": tri2.astype(np.int32), "links": np.asarray(links, dtype=np.int32),
           "dims": np.array([n_ent, n_rel, dim, t, k]), "alpha": np.float64(args.alpha), "beta": np.float64(args.beta),
           "gamma": np.float64(args.gamma), "lr": np.float64(args.learning_rate)}
    for v, name in zip(variables, RDGCN_NAMES):
        shape = tuple(v.value.shape)
        if name.startswith("diag"):
            start = 1.0 + 0.1 * rng.standard_normal(shape)
        elif name.endswith(".b"):
            start = 0.05 * rng.standard_normal(shape)
        elif name == "X0":
            start = embedding
        else:
            start = rng.standard_normal(shape) * 0.4
        start = np.asarray(start, dtype=np.float32).astype(np.float64)
        v.assign_numpy(start)
        out["var0/" + name] = start
    session = tf.Session()
    for step in range(3):
        feed = {key + ":0": rng.integers(0, n_ent, t * k) for key in ("neg_left", "neg_right", "neg2_left", "neg2_right")}
        val, _ = session.run([loss, train_op], feed_dict=feed)
        out["run%d/loss" % step] = np.float64(val)
        for key, ids in feed.items():
            out["run%d/%s" % (step, key[:-2])] = ids.astype(np.int32)
    for v, name in zip(variables, RDGCN_NAMES):
        out["var_final/" + name] = v.value.detach().numpy().copy()
    out["outputs_final"] = session.run(output, feed_dict=feed)
    print("rdgcn: losses %s" % ["%.6g" % float(out["run%d/loss" % i]) for i in range(3)],
          [tuple(v.value.shape) for v in variables])
    path = os.path.join(ROOT, "tests", "golden", "path_ii_rdgcn.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def generate_alinet():
    """Path (ii), AliNet: the reference's _get_variable / _generate_rel_graph (alinet.py:779-883: batch-normalised GCN
    layers over the one-hop adjacency, edge-softmax attention over the two-hop adjacency, highway gates, the
    normalised concatenation of all layers, contrastive alignment loss + relation loss) and its AdamOptimizer.
    → tests/golden/path_ii_alinet.npz"""
    import scipy.sparse as sp
    mod = import_reference("openea.approaches.alinet")
    tf = tf1_shim
    tf.reset_default_graph()
    rng = np.random.default_rng(31)
    n, dims, win = 26, [12, 8, 8], 3

    def adjacency(density, seed):
        a = sp.random(n, n, density=density, random_state=seed, format="coo")
        a = sp.coo_matrix(((a + a.T) > 0).astype(np.float64)) + sp.eye(n)
        deg = np.asarray(a.sum(1)).ravel()
        a = sp.coo_matrix(sp.diags(deg ** -0.5) @ a @ sp.diags(deg ** -0.5))
        return (np.vstack((a.row, a.col)).transpose(), a.data.astype(np.float32).astype(np.float64), a.shape)
    one, two = adjacency(0.10, 5), adjacency(0.18, 6)
    model = mod.AliNet()
    model.kgs = types.SimpleNamespace(entities_num=n)
    model.args = types.SimpleNamespace(layer_dims=dims, num_features_nonzero=0, dropout=0.0, neg_margin=1.5,
                                       neg_margin_balance=0.1, rel_param=0.01, learning_rate=0.001)
    model.adj = [one, two]
    model.rel_win_size = win
    model._get_variable()
    model._generate_rel_graph()
    variables = tf.trainable_variables()
    names = [v.name for v in variables]
    out = {"one/coords": one[0], "one/values": one[1], "two/coords": two[0], "two/values": two[1],
           "dims": np.array([n] + dims + [win]), "neg_margin": np.float64(1.5), "balance": np.float64(0.1),
           "rel_param": np.float64(0.01), "lr": np.float64(0.001)}
    for v in variables:
        shape = tuple(v.value.shape)
        if v.name.endswith("/gamma"):
            start = 1.0 + 0.1 * rng.standard_normal(shape)
        elif v.name.endswith(("/beta", "_bias")):
            start = 0.05 * rng.standard_normal(shape)
        else:
            start = rng.standard_normal(shape) * (0.6 / np.sqrt(shape[0]) if v.name != "init_embedding" else 0.5)
        start = np.asarray(start, dtype=np.float32).astype(np.float64)
        v.assign_numpy(start)
        out["var0/" + v.name] = start
    session = tf.Session()
    for step in range(3):
        pos = np.stack([rng.integers(0, n, 6), rng.integers(0, n, 6), np.zeros(6, dtype=np.int64)], 1)
        neg = rng.integers(0, n, (14, 2))
        hs, ts = rng.integers(0, n, 4 * win), rng.integers(0, n, 4 * win)
        feed = {model.rel_pos_links: pos, model.rel_neg_links: neg, model.hs: hs, model.ts: ts}
        res = session.run({"loss": model.loss, "optimizer": model.optimizer}, feed_dict=feed)
        out["run%d/loss" % step] = np.float64(res["loss"])
        for key, val in (("pos", pos), ("neg", neg), ("hs", hs), ("ts", ts)):
            out["run%d/%s" % (step, key)] = val.astype(np.int32)
    for v in variables:
        out["var_final/" + v.name] = v.value.detach().numpy().copy()
    for i, node in enumerate(model.output_embeds_list):
        out["outputs_final/%d" % i] = session.run(node)
    print("alinet: losses %s" % ["%.6g" % float(out["run%d/loss" % i]) for i in range(3)], names)
    path = os.path.join(ROOT, "tests", "golden", "path_ii_alinet.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if not os.path.isdir(REF_SRC):
        sys.exit("set OPENEA_REFERENCE to a checkout of the original OpenEA: the goldens are generated from it")
    generate()
    generate_attre()
    generate_gcn_align()
    generate_rdgcn()
    generate_alinet()
