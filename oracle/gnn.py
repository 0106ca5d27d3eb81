"""CPU ORACLE for path (ii) (GCN-Align aggregation + L1 alignment loss) — TEST INFRASTRUCTURE ONLY.

PARITY: the GCN-Align unit below reproduces the reference's own GCN_Align_Unit executed on oracle/tf1_shim.py
(tests/test_reference_graph_goldens.py, 1e-9); the engine's AliNet model and RDGCN layer are held to such goldens
directly.  TF's op / optimiser semantics (restated in that interpreter) stay unpinned: TensorFlow 1.x is absent here.
This restates it with torch-CPU autograd at the reference's call sites:
  GraphConvolution._call  gcn_align.py:239-267   (featureless first layer, weight-less second layer)
  trunc_normal + l2_normalize(·, 1)  gcn_align.py:52-56
  align_loss  gcn_align.py:298-320
  GradientDescentOptimizer  gcn_align.py:511
The adjacency builders ARE pinned: `reference_gcn_utils()` executes the reference's own GCN_Utils / load_attr
source (pure NumPy/SciPy, extracted from the file because the module itself imports TensorFlow).
"""
import ast
import os

import numpy as np
import scipy.sparse as sp
import torch

REF_DIR = os.path.join(os.environ.get("OPENEA_REFERENCE", ""), "src", "openea", "approaches")
REF_FILE = os.path.join(REF_DIR, "gcn_align.py")


def reference_gcn_utils():
    """(GCN_Utils class, load_attr function) compiled from the reference source; None if it is not present."""
    if not os.environ.get("OPENEA_REFERENCE") or not os.path.exists(REF_FILE):
        return None
    with open(REF_FILE) as f:
        tree = ast.parse(f.read())
    keep = [n for n in tree.body if (isinstance(n, ast.ClassDef) and n.name == "GCN_Utils")
            or (isinstance(n, ast.FunctionDef) and n.name == "load_attr")]
    ns = {"np": np, "sp": sp, "merge_dic": lambda a, b: {**a, **b}, "eigsh": None, "print": lambda *a, **k: None}
    exec(compile(ast.Module(body=keep, type_ignores=[]), REF_FILE, "exec"), ns)
    return ns["GCN_Utils"], ns["load_attr"]


def _sparse(mat, dtype):
    m = sp.coo_matrix(mat)
    idx = torch.tensor(np.vstack([m.row, m.col]), dtype=torch.long)
    return torch.sparse_coo_tensor(idx, torch.tensor(m.data, dtype=dtype), m.shape).coalesce()


def l2n(x):
    return x * torch.rsqrt(torch.clamp((x * x).sum(1, keepdim=True), min=1e-12))


def unit_forward(support, W, features=None, dtype=torch.float32):
    """OUT = A·relu(A·pre), pre = l2n(W) (featureless) or X_attr·l2n(W)."""
    A = _sparse(support, dtype)
    Wn = l2n(W)
    pre = Wn if features is None else torch.sparse.mm(_sparse(features, dtype), Wn)
    h1 = torch.relu(torch.sparse.mm(A, pre))
    return torch.sparse.mm(A, h1)


def align_loss(out, ill, gamma, k, neg_left, neg_right, neg2_left, neg2_right):
    left, right = torch.as_tensor(ill[:, 0], dtype=torch.long), torch.as_tensor(ill[:, 1], dtype=torch.long)
    t = len(ill)
    a = (out[left] - out[right]).abs().sum(1)
    d = (a + gamma).reshape(t, 1)
    tot = 0.0
    for nl, nr in ((neg_left, neg_right), (neg2_left, neg2_right)):
        b = (out[torch.as_tensor(nl, dtype=torch.long)] - out[torch.as_tensor(nr, dtype=torch.long)]).abs().sum(1)
        tot = tot + torch.relu(-b.reshape(t, k) + d).sum()
    return tot / (2.0 * k * t)


def unit_train_step(support, W0, features, ill, gamma, k, negs, lr, dtype=torch.float32):
    """One session.run([loss, opt_op]) of a GCN_Align_Unit: returns (loss, updated W, outputs)."""
    W = torch.tensor(np.asarray(W0), dtype=dtype, requires_grad=True)
    out = unit_forward(support, W, features, dtype)
    loss = align_loss(out, np.asarray(ill), gamma, k, *negs)
    loss.backward()
    with torch.no_grad():
        W_new = W - lr * W.grad
    return float(loss.detach()), W_new.numpy(), out.detach().numpy()


# ---- AliNet (approaches/alinet.py) — torch-CPU restatement with dense-free sparse ops (TF semantics unpinned) ----
ALINET_REF_FILE = os.path.join(REF_DIR, "alinet.py")


def reference_alinet_builders():
    """Namespace with the reference's own pure-Python/NumPy/pandas builders (AKG, enhance_triples, no_weighted_adj,
    generate_2hop_triples, remove_unlinked_triples, generate_rel_ht, …) compiled from its source; None if absent."""
    if not os.environ.get("OPENEA_REFERENCE") or not os.path.exists(ALINET_REF_FILE):
        return None
    import math
    import time
    import pandas as pd
    with open(ALINET_REF_FILE) as f:
        tree = ast.parse(f.read())
    want = {"sparse_to_tuple", "normalize_adj", "preprocess_adj", "no_weighted_adj", "remove_unlinked_triples",
            "generate_2hop_triples", "enhance_triples", "generate_rel_ht", "AKG"}
    keep = [n for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and n.name in want]
    ns = {"np": np, "sp": sp, "pd": pd, "math": math, "time": time, "print": lambda *a, **k: None}
    exec(compile(ast.Module(body=keep, type_ignores=[]), ALINET_REF_FILE, "exec"), ns)
    return ns


def edge_softmax_aggregate(adj, s1, s2, M, slope=0.2):
    """Σ_j softmax_j(leaky_relu(a_ij (s1_i + s2_j))) M_j over the non-zeros of `adj` (scipy), with torch autograd."""
    m = sp.coo_matrix(adj)
    row = torch.as_tensor(m.row, dtype=torch.long)
    col = torch.as_tensor(m.col, dtype=torch.long)
    a = torch.as_tensor(m.data, dtype=M.dtype)
    logit = torch.nn.functional.leaky_relu(a * (s1[row] + s2[col]), slope)
    mx = torch.full((m.shape[0],), -1e30, dtype=M.dtype).scatter_reduce(0, row, logit, "amax")
    ex = torch.exp(logit - mx[row])
    den = torch.zeros(m.shape[0], dtype=M.dtype).index_add(0, row, ex)
    alpha = ex / den[row]
    return torch.zeros(m.shape[0], M.shape[1], dtype=M.dtype).index_add(0, row, alpha[:, None] * M[col])


def alinet_forward(params, adj1, adj2, n_layers, dtype=torch.float64):
    """Same graph as openea_b200.approaches.alinet.AliNetModel.forward with torch.sparse / scatter ops."""
    import math
    bn = lambda x, g, b: x * (g / math.sqrt(1.0 + 1e-3)) + b
    A1 = _sparse(adj1, dtype)
    x = params["init_embedding"]
    outs = []
    for i in range(n_layers):
        xb = bn(x, params["gcn%d.bn_gamma" % i], params["gcn%d.bn_beta" % i])
        one = torch.tanh(torch.sparse.mm(A1, xb @ params["gcn%d.kernel" % i]) + params["gcn%d.bias" % i])
        if i < n_layers - 1:
            xg = bn(x, params["gat%d.bn_gamma" % i], params["gat%d.bn_beta" % i])
            mapped = xg @ params["gat%d.kernel" % i]
            s1 = torch.tanh(((xg @ params["gat%d.kernel1" % i]) * xg).sum(1))
            s2 = torch.tanh(((xg @ params["gat%d.kernel2" % i]) * xg).sum(1))
            two = torch.tanh(edge_softmax_aggregate(adj2, s1, s2, mapped))
            g1 = bn(two, params["hw%d.bn_gamma" % i], params["hw%d.bn_beta" % i])
            g2 = bn(one, params["hw%d.bn_gamma" % i], params["hw%d.bn_beta" % i])
            gate = torch.relu(torch.tanh(g1 @ params["hw%d.kernel" % i]))
            x = torch.tanh(g2 * (1 - gate) + g1 * gate)
        else:
            x = one
        outs.append(x)
    return outs


def alinet_loss(params, outs, pos, neg, neg_margin, balance, hs, ts, rel_win, rel_param):
    emb = l2n(torch.cat([l2n(o) for o in outs + [params["init_embedding"]]], dim=1))
    tl = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.long)
    pos, neg = tl(pos), tl(neg)
    total = ((emb[pos[:, 0]] - emb[pos[:, 1]]) ** 2).sum()
    total = total + balance * torch.relu(neg_margin - ((emb[neg[:, 0]] - emb[neg[:, 1]]) ** 2).sum(1)).sum()
    if rel_param > 0:
        diff = emb[tl(hs)] - emb[tl(ts)]
        r = l2n(diff.reshape(-1, rel_win, emb.shape[1]).mean(1, keepdim=True).expand(-1, rel_win, -1).reshape(-1, emb.shape[1]))
        total = total + rel_param * ((diff - r) ** 2).sum()
    return total


# ---- RDGCN (approaches/rdgcn.py) — torch-CPU restatement (TF semantics unpinned) -------------------------------
RDGCN_REF_FILE = os.path.join(REF_DIR, "rdgcn.py")


def reference_rdgcn_builders():
    """get_mat / rfunc of the reference compiled from its source (tf.SparseTensor stubbed to a tuple)."""
    if not os.environ.get("OPENEA_REFERENCE") or not os.path.exists(RDGCN_REF_FILE):
        return None
    import math
    import types
    with open(RDGCN_REF_FILE) as f:
        tree = ast.parse(f.read())
    keep = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in ("rfunc", "get_mat")]
    tf_stub = types.SimpleNamespace(SparseTensor=lambda indices, values, dense_shape: (indices, values, dense_shape))
    ns = {"np": np, "math": math, "tf": tf_stub}
    exec(compile(ast.Module(body=keep, type_ignores=[]), RDGCN_REF_FILE, "exec"), ns)
    return ns


def rdgcn_forward(P, M, head_avg, tail_avg, dual_A, tri, alpha, beta, dtype=torch.float64, slope=0.2):
    """Layer.build (rdgcn.py:317-338) with torch.sparse / scatter ops.  P: dict of float64 tensors named as in
    openea_b200.approaches.rdgcn.RDGCNLayer; tri: [T, 3] int array (one r_mat entry per triple)."""
    Ms, Hs, Ts = _sparse(M, dtype), _sparse(head_avg, dtype), _sparse(tail_avg, dtype)
    A = torch.as_tensor(dual_A, dtype=dtype)
    bias = -1e9 * (1.0 - (A > 0).to(dtype))
    vec = lambda n: (P[n + ".w"][:, :1], P[n + ".b"][:, :1])
    row = torch.as_tensor(tri[:, 0], dtype=torch.long); col = torch.as_tensor(tri[:, 2], dtype=torch.long)
    rel = torch.as_tensor(tri[:, 1], dtype=torch.long)
    E = M.shape[0]

    def dual_input(x):
        return torch.cat([torch.sparse.mm(Hs, x), torch.sparse.mm(Ts, x)], 1)

    def att(fts, values, f1, f2):
        (w1, b1), (w2, b2) = vec(f1), vec(f2)
        logits = (fts @ w1 + b1) + (fts @ w2 + b2).t()
        return torch.relu(torch.softmax(torch.nn.functional.leaky_relu(A * logits, slope) + bias, 1) @ values)

    def sparse_att(x, dual_h, name):
        w, b = vec(name)
        logit = torch.nn.functional.leaky_relu((dual_h @ w + b).reshape(-1)[rel], slope)
        mx = torch.full((E,), -1e30, dtype=dtype).scatter_reduce(0, row, logit, "amax")
        ex = torch.exp(logit - mx[row])
        den = torch.zeros(E, dtype=dtype).index_add(0, row, ex)
        return torch.relu(torch.zeros(E, x.shape[1], dtype=dtype).index_add(0, row, (ex / den[row])[:, None] * x[col]))

    def highway(l1, l2, name):
        g = torch.sigmoid(l1 @ P[name + ".W"] + P[name + ".b"])
        return g * l2 + (1 - g) * l1

    x0 = P["X0"]
    dx1 = dual_input(x0)
    dh1 = att(dx1 @ P["self.W"], dx1, "self.f1", "self.f2")
    x1 = x0 + alpha * sparse_att(x0, dh1, "sp1")
    dx2 = dual_input(x1)
    dh2 = att(dx2 @ P["dual.W"] + P["dual.b"], dh1, "dual.f1", "dual.f2")
    x2 = x0 + beta * sparse_att(x1, dh2, "sp2")
    g1 = highway(x2, torch.relu(torch.sparse.mm(Ms, x2 * P["diag1.w"])), "hw1")
    return highway(g1, torch.relu(torch.sparse.mm(Ms, g1 * P["diag2.w"])), "hw2")
