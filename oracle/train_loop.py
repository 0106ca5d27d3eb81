"""CPU ORACLE end-to-end training loop for path (i) — TEST INFRASTRUCTURE ONLY.

Restates BasicModel.run / launch_triple_training_1epo (models/basic_model.py:211-290) and the AlignE / BootEA
configuration on the CPU: the reference's own Python sampler (modules/train/batch.py, imported from the checkout
OPENEA_REFERENCE names, otherwise the behavioural port in openea_b200.modules.train.batch), the C oracle
step (dense TF semantics) and the NumPy evaluation.  Used to calibrate end-to-end accuracy (Hits@1) of the
engine on the same synthetic KG: parity here is statistical (different RNG streams), not bit-wise.
"""
import math
import random

import numpy as np

from oracle import finding as orf
from oracle import ref_adapter
from oracle import triple as orc


def _batch_module():
    if ref_adapter.available():
        return ref_adapter.load().batch
    from openea_b200.modules.train import batch
    return batch


def train_triples(arr, dim, batch_size, neg_per_pos, epochs, loss="limited", lr=0.01, margin=0.01, neg_margin=2.0,
                  balance=0.2, truncated_eps=None, truncated_freq=10, seed=0, init="normal", log=None, on_epoch=None):
    """arr: dict from openea_b200.synth.synth_id_arrays.  Returns the final DenseState."""
    bat = _batch_module()
    random.seed(seed)
    np.random.seed(seed)
    rng = np.random.default_rng(seed)
    n_ent, n_rel = arr["n_ent"], arr["n_rel"]
    std = 1.0 / math.sqrt(dim)
    def trunc(shape):
        # tf.initializers.truncated_normal: values beyond ±2σ are RE-DRAWN, not clipped (the raw row norm sets
        # the effective angular step through the l2_normalize Jacobian, so this matters for learning speed)
        x = rng.standard_normal(shape)
        bad = np.abs(x) > 2
        while bad.any():
            x[bad] = rng.standard_normal(int(bad.sum()))
            bad = np.abs(x) > 2
        return (x * std).astype(np.float32)
    if init == "normal":
        ent, rel = trunc((n_ent, dim)), trunc((n_rel, dim))
    else:
        ent = rng.standard_normal((n_ent, dim)).astype(np.float32)
        ent /= np.linalg.norm(ent, axis=1, keepdims=True)
        rel = rng.standard_normal((n_rel, dim)).astype(np.float32)
        rel /= np.linalg.norm(rel, axis=1, keepdims=True)
    st = orc.DenseState(ent, rel, "Adagrad")
    t1 = [tuple(x) for x in arr["triples1"].tolist()]
    t2 = [tuple(x) for x in arr["triples2"].tolist()]
    s1, s2 = set(t1), set(t2)
    e1, e2 = arr["entities1"].tolist(), arr["entities2"].tolist()
    steps = int(math.ceil((len(t1) + len(t2)) / batch_size))
    nb1 = nb2 = None
    for epoch in range(1, epochs + 1):
        tot, cnt = 0.0, 0
        for step in range(steps):
            if neg_per_pos > 0:
                pos, neg = bat.generate_relation_triple_batch(t1, t2, s1, s2, e1, e2, batch_size, step, nb1, nb2, neg_per_pos)
            else:
                pos, neg = bat.generate_pos_batch(t1, t2, batch_size, step), None
            if not pos:
                continue
            p = np.asarray(pos, dtype=np.int32).T.copy()
            n = None if neg is None else np.asarray(neg, dtype=np.int32).T.copy()
            tot += orc.step(st, p, n, loss, "L2", True, True, lr, margin=margin, neg_margin=neg_margin, balance=balance)
            cnt += len(pos)
        random.shuffle(t1)
        random.shuffle(t2)
        if log:
            log("epoch %d, avg. triple loss: %.4f" % (epoch, tot / max(1, cnt)))
        if on_epoch is not None:
            on_epoch(epoch, st)
        if truncated_eps is not None and epoch % truncated_freq == 0:
            en = orc.l2_normalize(st.ent)
            k1, k2 = int((1 - truncated_eps) * len(e1)), int((1 - truncated_eps) * len(e2))
            nb1 = dict(zip(e1, [list(s) for s in orf.find_neighbours(en[e1], en[e1], e1, k1)]))
            nb2 = dict(zip(e2, [list(s) for s in orf.find_neighbours(en[e2], en[e2], e2, k2)]))
    return st


def test_hits(st, arr, metric="inner", normalize=False, csls_k=0, top_k=(1, 5, 10, 50)):
    en = orc.l2_normalize(st.ent)
    links = arr["test_links"]
    _, hits, mr, mrr = orf.greedy_alignment(en[links[:, 0]], en[links[:, 1]], list(top_k), metric, normalize, csls_k)
    return hits, mr, mrr
