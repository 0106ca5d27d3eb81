"""Shared test helpers: float64 torch-autograd statement of the triple-scoring graph (an independent
derivation used to check the C oracle's hand-written backward), seeded batch generators, and the recorded results of
the original OpenEA functions the host ports are compared with."""
import hashlib
import json
import numbers
import os
from collections.abc import Mapping, Set

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def canonical(x):
    """Text form of a result that is equal for two results exactly when Python's == holds between them (dicts and sets
    in sorted order, integral floats as ints, NumPy scalars and arrays as Python values)."""
    if isinstance(x, Mapping):
        return "{" + ",".join(sorted(canonical(k) + ":" + canonical(v) for k, v in x.items())) + "}"
    if isinstance(x, Set):
        return "set(" + ",".join(sorted(canonical(e) for e in x)) + ")"
    if isinstance(x, tuple):
        return "(" + ",".join(canonical(e) for e in x) + ")"
    if isinstance(x, (list, np.ndarray)):
        return "[" + ",".join(canonical(e) for e in x) + "]"
    if isinstance(x, (bool, np.bool_)):
        return repr(bool(x))
    if isinstance(x, numbers.Integral):
        return str(int(x))
    if isinstance(x, numbers.Real):
        f = float(x)
        return str(int(f)) if f.is_integer() else repr(f)
    if isinstance(x, str) or x is None:
        return repr(x)
    raise TypeError("no canonical form for %r" % type(x))


def digest(x):
    return hashlib.sha256(canonical(x).encode("utf8")).hexdigest()


class ReferenceRecord:
    """What the original OpenEA functions returned on a test's inputs, stored as tests/golden/<name>.json (SHA-256 of
    the canonical form of results compared with ==) and tests/golden/<name>.npz (arrays compared with a tolerance).

    With OPENEA_REFERENCE set to a checkout of the original project, `reference` callables are run live, the test's
    comparison is made against the live result, and the record is rewritten; otherwise the stored record is used."""

    def __init__(self, name):
        self.json_path = os.path.join(GOLDEN, name + ".json")
        self.npz_path = os.path.join(GOLDEN, name + ".npz")
        self.live = bool(os.environ.get("OPENEA_REFERENCE"))
        self.digests, self.arrays = {}, {}
        if os.path.exists(self.json_path):
            with open(self.json_path) as f:
                self.digests = json.load(f)
        if os.path.exists(self.npz_path):
            with np.load(self.npz_path) as z:
                self.arrays = {k: z[k] for k in z.files}

    def equal(self, key, mine, reference):
        """mine == the reference's result (`reference()` is only called when recording)."""
        if self.live:
            want = reference()
            self.digests[key] = digest(want)
            with open(self.json_path, "w") as f:
                json.dump(self.digests, f, indent=0, sort_keys=True)
            return mine == want
        return digest(mine) == self.digests[key]

    def array(self, key, reference):
        """The reference's numeric result as an array (`reference()` is only called when recording)."""
        if self.live:
            self.arrays[key] = np.asarray(reference())
            np.savez_compressed(self.npz_path, **self.arrays)
        return self.arrays[key]


def torch_triple_loss(ent, rel, pos, neg, loss, loss_norm, ent_norm, rel_norm, margin=0.0, neg_margin=0.0,
                      balance=1.0, dtype=torch.float64):
    """Formulas of modules/base/losses.py + initializers.py:26 in torch; returns (loss, g_ent, g_rel, scores)."""
    E = torch.tensor(np.asarray(ent), dtype=dtype, requires_grad=True)
    R = torch.tensor(np.asarray(rel), dtype=dtype, requires_grad=True)

    def l2n(x):
        ss = (x * x).sum(1, keepdim=True)
        return x * torch.rsqrt(torch.clamp(ss, min=1e-12))

    Eh = l2n(E) if ent_norm else E
    Rh = l2n(R) if rel_norm else R

    def score(hrt):
        hrt = torch.as_tensor(np.asarray(hrt), dtype=torch.long)
        u = Eh[hrt[0]] + Rh[hrt[1]] - Eh[hrt[2]]
        return u.abs().sum(1) if loss_norm == "L1" else (u * u).sum(1)

    sp = score(pos)
    sn = score(neg) if neg is not None and np.asarray(neg).size else torch.zeros(0, dtype=dtype)
    relu = torch.nn.functional.relu
    if loss == "margin-based":
        val = relu(margin + sp - sn).sum()
    elif loss == "limited":
        val = relu(sp - margin).sum() + balance * relu(neg_margin - sn).sum()
    elif loss == "logistic":
        val = torch.log(1 + torch.exp(sp)).sum() + torch.log(1 + torch.exp(-sn)).sum()
    elif loss == "positive":
        val = sp.sum()
    elif loss == "logsigmoid":
        val = -torch.log(torch.sigmoid(-sp)).sum()
    else:
        raise ValueError(loss)
    val.backward()
    g_e = E.grad if E.grad is not None else torch.zeros_like(E)
    g_r = R.grad if R.grad is not None else torch.zeros_like(R)
    return float(val.detach()), g_e.numpy(), g_r.numpy(), torch.cat([sp, sn]).detach().numpy()


def make_tables(rng, n_ent, n_rel, d, scale=1.0):
    ent = (rng.standard_normal((n_ent, d)) * scale / np.sqrt(d)).astype(np.float32)
    rel = (rng.standard_normal((n_rel, d)) * scale / np.sqrt(d)).astype(np.float32)
    return ent, rel


def make_batch(rng, n_ent, n_rel, n_pos, k, hot=True):
    """Index batch with repeated rows (a few hot entities/relations) as Zipf-like KGs produce."""
    def ents(n):
        e = rng.integers(0, n_ent, size=n)
        if hot and n > 4:
            m = rng.random(n) < 0.3
            e[m] = rng.integers(0, max(1, min(5, n_ent)), size=int(m.sum()))
        return e
    pos = np.stack([ents(n_pos), rng.integers(0, n_rel, size=n_pos), ents(n_pos)]).astype(np.int32)
    if k == 0:
        return pos, None
    neg = np.repeat(pos, k, axis=1)
    side = rng.random(n_pos * k) < 0.5
    repl = ents(n_pos * k)
    neg[0, side] = repl[side]
    neg[2, ~side] = repl[~side]
    return pos, neg.astype(np.int32)
