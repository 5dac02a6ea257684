"""CPU oracle for the TorchRecSys collaborative-filtering hot path (numpy, fp32).

TEST INFRASTRUCTURE ONLY.  Nothing in ``torchrecsys_b200/`` may import this module;
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / reference
arm do.  It is a restatement, in plain numpy, of what the reference computes on its
``use_cuda=False`` path.  Every function cites the reference lines it follows
(paths relative to ``/root/reference``; ``torch:`` = the installed torch 2.11 tree,
where the reference's arithmetic actually lives -- the reference pins no torch
version, ``setup.py:7``).

Parity pin: the reference's own tests hold no numeric golden vectors for this path
(SURVEY.md §8c), so this oracle is pinned against the *live reference* run in the
build container: ``oracle/make_golden.py`` imports ``/root/reference`` unmodified,
records inputs/outputs into ``tests/golden/*.npz`` and ``tests/test_oracle_golden.py``
checks this file against them.

Conventions
-----------
* parameters are float32 numpy arrays keyed by the reference ``state_dict`` names
  (without the ``net.`` prefix): Linear ``user.weight item.weight user_bias.weight
  item_bias.weight metadata.{f}.weight``; FM ``user.weight item.weight
  linear_user.weight linear_item.weight metadata.{f}.weight
  linear_metadata.{f}.weight``; MLP ``user.weight item.weight
  metadata_embeddings.{f}.weight fcs.{l}.weight fcs.{l}.bias bns.{l}.*
  output_layer.weight output_layer.bias``.
* a batch is ``dict(user[B], pos[B], neg[B], pos_meta[B,F], neg_meta[B,F])`` of int64;
  one id per metadata feature (SURVEY.md D7: the reference only ever reads bag
  element 0 of each feature).
* "rows" of a sparse gradient are summed per table in lookup order after a stable
  sort by row index -- the order ``coalesce()`` produces.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import numpy as np

F32 = np.float32


# --------------------------------------------------------------------------------------
# a1  embeddings: row gather (+ sum-pool over metadata features)
# --------------------------------------------------------------------------------------
def gather_rows(table: np.ndarray, idx: np.ndarray) -> np.ndarray:
    """``nn.Embedding.forward`` == row gather (embeddings/init_embeddings.py:5,53;
    torch: nn/functional.py embedding -> index_select).  Bit-exact copy."""
    return table[idx]


def gather_sum(item_table, item_idx, meta_tables=(), meta_idx=None) -> np.ndarray:
    """Item vector of the Linear scorer: ``item[i] += meta_f[m[:, f]]`` in feature
    order (collaborative/linear.py:67-75)."""
    out = item_table[item_idx].astype(F32, copy=True)
    for f, t in enumerate(meta_tables):
        out = (out + t[meta_idx[:, f]]).astype(F32)
    return out


def scaled_embedding_init(rng: np.random.Generator, n: int, d: int) -> np.ndarray:
    """``ScaledEmbedding.reset_parameters``: N(0, 1/D) i.e. std = 1/D
    (embeddings/init_embeddings.py:43-50)."""
    return (rng.standard_normal((n, d)) / d).astype(F32)


# --------------------------------------------------------------------------------------
# a2/a3  scorers
# --------------------------------------------------------------------------------------
def _meta_tables(params: Dict[str, np.ndarray], prefix: str) -> List[np.ndarray]:
    out, f = [], 0
    while f"{prefix}.{f}.weight" in params:
        out.append(params[f"{prefix}.{f}.weight"])
        f += 1
    return out


def linear_scores(params, user, item, meta=None) -> np.ndarray:
    """``Linear.forward`` (collaborative/linear.py:54-80): dot(u, v + sum_f m_f) + b_u + b_i.
    Returns shape (B, 1) like the reference."""
    u = params["user.weight"][user]
    v = gather_sum(params["item.weight"], item, _meta_tables(params, "metadata"), meta)
    s = (u * v).sum(axis=1, dtype=F32)
    s = s + params["user_bias.weight"][user, 0] + params["item_bias.weight"][item, 0]
    return s.astype(F32).reshape(-1, 1)


def _fm_fields(params, user, item, meta):
    embs = [params["user.weight"][user], params["item.weight"][item]]
    lins = [params["linear_user.weight"][user, 0], params["linear_item.weight"][item, 0]]
    for f, t in enumerate(_meta_tables(params, "metadata")):
        embs.append(t[meta[:, f]])
        lins.append(params[f"linear_metadata.{f}.weight"][meta[:, f], 0])
    return embs, lins


def fm_logits(params, user, item, meta=None) -> np.ndarray:
    """Pre-sigmoid FM activation (collaborative/fm.py:70-97)."""
    embs, lins = _fm_fields(params, user, item, meta)
    e = np.stack(embs, axis=1)  # (B, K, D)
    power_of_sum = e.sum(axis=1, dtype=F32) ** 2
    sum_of_power = (e ** 2).sum(axis=1, dtype=F32)
    pair = (power_of_sum - sum_of_power).sum(axis=1, dtype=F32) * F32(0.5)
    lin = np.stack(lins, axis=1).sum(axis=1, dtype=F32)
    return (lin + pair).astype(F32)


def sigmoid(z: np.ndarray) -> np.ndarray:
    z = z.astype(F32)
    return (F32(1.0) / (F32(1.0) + np.exp(-z, dtype=F32))).astype(F32)


def fm_scores(params, user, item, meta=None) -> np.ndarray:
    """``FM.forward`` (collaborative/fm.py:60-101); shape (B,)."""
    return sigmoid(fm_logits(params, user, item, meta))


# --------------------------------------------------------------------------------------
# a5  loss, a10 pairwise "auc"
# --------------------------------------------------------------------------------------
def hinge_loss(pos: np.ndarray, neg: np.ndarray) -> np.float32:
    """``mean(clamp(neg - pos + 1, 0))`` (helper/loss.py:5-9)."""
    h = np.maximum(neg.astype(F32) - pos.astype(F32) + F32(1.0), F32(0.0))
    return F32(h.mean(dtype=F32))


def pairwise_auc(pos: np.ndarray, neg: np.ndarray) -> np.float32:
    """``(pos > neg).sum() / len(pos)`` (evaluate/metrics.py:23-31); strict ``>``."""
    return F32((pos.reshape(-1) > neg.reshape(-1)).sum() / F32(pos.shape[0]))


def roc_auc(pos: np.ndarray, neg: np.ndarray) -> float:
    """Sort-based ROC-AUC over {pos: label 1, neg: label 0}, ties get average rank
    (Mann-Whitney U).  Not in the reference (SURVEY.md D11); checked against
    sklearn.metrics.roc_auc_score in tests."""
    s = np.concatenate([pos.reshape(-1), neg.reshape(-1)]).astype(np.float64)
    order = np.argsort(s, kind="stable")
    ranks = np.empty(len(s), dtype=np.float64)
    ss = s[order]
    i = 0
    while i < len(ss):
        j = i
        while j + 1 < len(ss) and ss[j + 1] == ss[i]:
            j += 1
        ranks[order[i : j + 1]] = 0.5 * (i + j) + 1.0
        i = j + 1
    n1, n0 = pos.size, neg.size
    return float((ranks[:n1].sum() - n1 * (n1 + 1) / 2.0) / (n1 * n0))


# --------------------------------------------------------------------------------------
# a7  closed-form gradients of  mean_b max(0, s-_b - s+_b + 1)
# --------------------------------------------------------------------------------------
def hinge_weights(pos, neg) -> np.ndarray:
    """d loss / d (neg - pos): 1/B where the hinge is active; ``clamp`` passes the
    gradient at exactly 0 (SURVEY.md a5, probed), hence ``>=``."""
    B = pos.shape[0]
    h = neg.reshape(-1).astype(F32) - pos.reshape(-1).astype(F32) + F32(1.0)
    return np.where(h >= 0, F32(1.0) / F32(B), F32(0.0)).astype(F32)


SparseGrad = Tuple[np.ndarray, np.ndarray]  # (row indices [n], values [n, W])


def linear_grads(params, batch) -> Tuple[np.float32, Dict[str, SparseGrad]]:
    """Loss and per-lookup sparse gradients of the Linear scorer (autograd of
    collaborative/linear.py:64-78 under helper/loss.py:7-9).  d u = g (v- - v+),
    d v+ = -g u, d v- = +g u, metadata rows as the item rows, d b_i = -/+ g,
    d b_u = 0 (it cancels between the two passes, SURVEY.md D12)."""
    user, pos, neg = batch["user"], batch["pos"], batch["neg"]
    pm, nm = batch.get("pos_meta"), batch.get("neg_meta")
    sp = linear_scores(params, user, pos, pm)
    sn = linear_scores(params, user, neg, nm)
    loss = hinge_loss(sp, sn)
    g = hinge_weights(sp, sn)[:, None]
    u = params["user.weight"][user]
    metas = _meta_tables(params, "metadata")
    vp = gather_sum(params["item.weight"], pos, metas, pm)
    vn = gather_sum(params["item.weight"], neg, metas, nm)
    grads: Dict[str, SparseGrad] = {}
    grads["user.weight"] = (np.concatenate([user, user]),
                            np.concatenate([-g * vp, g * vn]).astype(F32))
    gi = np.concatenate([-g * u, g * u]).astype(F32)
    grads["item.weight"] = (np.concatenate([pos, neg]), gi)
    grads["user_bias.weight"] = (np.concatenate([user, user]),
                                 np.concatenate([-g, g]).astype(F32))
    grads["item_bias.weight"] = (np.concatenate([pos, neg]), np.concatenate([-g, g]).astype(F32))
    for f in range(len(metas)):
        grads[f"metadata.{f}.weight"] = (np.concatenate([pm[:, f], nm[:, f]]), gi.copy())
    return loss, grads


def fm_grads(params, batch) -> Tuple[np.float32, Dict[str, SparseGrad]]:
    """Loss and sparse gradients of the FM scorer (autograd of collaborative/fm.py:70-99).
    With S = sum_k e_k and delta = -/+ g sigma (1 - sigma):  d e_k = delta (S - e_k),
    d w_k = delta."""
    user, pos, neg = batch["user"], batch["pos"], batch["neg"]
    pm, nm = batch.get("pos_meta"), batch.get("neg_meta")
    sp = fm_scores(params, user, pos, pm)
    sn = fm_scores(params, user, neg, nm)
    loss = hinge_loss(sp, sn)
    g = hinge_weights(sp, sn)
    dp = (-g * sp * (F32(1.0) - sp)).astype(F32)[:, None]
    dn = (g * sn * (F32(1.0) - sn)).astype(F32)[:, None]
    ep, _ = _fm_fields(params, user, pos, pm)
    en, _ = _fm_fields(params, user, neg, nm)
    Sp = np.sum(np.stack(ep, 1), axis=1, dtype=F32)
    Sn = np.sum(np.stack(en, 1), axis=1, dtype=F32)
    grads: Dict[str, SparseGrad] = {}
    uu = np.concatenate([user, user])
    ii = np.concatenate([pos, neg])
    grads["user.weight"] = (uu, np.concatenate([dp * (Sp - ep[0]), dn * (Sn - en[0])]).astype(F32))
    grads["item.weight"] = (ii, np.concatenate([dp * (Sp - ep[1]), dn * (Sn - en[1])]).astype(F32))
    grads["linear_user.weight"] = (uu, np.concatenate([dp, dn]).astype(F32))
    grads["linear_item.weight"] = (ii, np.concatenate([dp, dn]).astype(F32))
    for f in range(len(ep) - 2):
        mm = np.concatenate([pm[:, f], nm[:, f]])
        grads[f"metadata.{f}.weight"] = (
            mm, np.concatenate([dp * (Sp - ep[2 + f]), dn * (Sn - en[2 + f])]).astype(F32))
        grads[f"linear_metadata.{f}.weight"] = (mm, np.concatenate([dp, dn]).astype(F32))
    return loss, grads


def coalesce(idx: np.ndarray, vals: np.ndarray) -> SparseGrad:
    """``grad.coalesce()`` (torch: optim/_functional.py:44, optim/adagrad.py:364): unique
    sorted rows, duplicates summed in lookup order (stable sort)."""
    order = np.argsort(idx, kind="stable")
    si, sv = idx[order], vals[order].astype(F32)
    heads = np.ones(len(si), dtype=bool)
    heads[1:] = si[1:] != si[:-1]
    rows = si[heads]
    out = np.zeros((len(rows),) + sv.shape[1:], dtype=F32)
    seg = np.cumsum(heads) - 1
    for k in range(len(si)):  # sequential fp32 accumulation, like the CPU kernel
        out[seg[k]] = (out[seg[k]] + sv[k]).astype(F32)
    return rows, out


# --------------------------------------------------------------------------------------
# a7  row-wise optimizers on touched rows
# --------------------------------------------------------------------------------------
class OptSpec:
    """kind in {'sgd', 'adagrad', 'sparse_adam'} with torch's default hyper-parameters."""

    def __init__(self, kind, lr=None, betas=(0.9, 0.999), eps=None, lr_decay=0.0):
        self.kind = kind
        self.lr = lr if lr is not None else {"sgd": 1e-3, "adagrad": 1e-2, "sparse_adam": 1e-3}[kind]
        self.betas = betas
        self.eps = eps if eps is not None else {"sgd": 0.0, "adagrad": 1e-10, "sparse_adam": 1e-8}[kind]
        self.lr_decay = lr_decay


def init_opt_state(params: Dict[str, np.ndarray], spec: OptSpec) -> Dict[str, Dict[str, np.ndarray]]:
    st = {}
    for k, p in params.items():
        if spec.kind == "adagrad":
            st[k] = {"sum": np.zeros_like(p)}
        elif spec.kind == "sparse_adam":
            st[k] = {"exp_avg": np.zeros_like(p), "exp_avg_sq": np.zeros_like(p)}
        else:
            st[k] = {}
    return st


def adam_step_size(spec: OptSpec, step: int) -> float:
    """torch: optim/_functional.py:80-82 (python double arithmetic)."""
    b1, b2 = spec.betas
    return spec.lr * math.sqrt(1 - b2 ** step) / (1 - b1 ** step)


def adagrad_clr(spec: OptSpec, step: int) -> float:
    """torch: optim/adagrad.py:361."""
    return spec.lr / (1 + (step - 1) * spec.lr_decay)


def apply_rows(p, state, rows, g, spec: OptSpec, step: int) -> None:
    """In-place update of ``p[rows]`` with coalesced gradient rows ``g``.

    sparse_adam: torch: optim/_functional.py:65-84; adagrad: torch: optim/adagrad.py:363-373;
    sgd: torch: optim/sgd.py (_single_tensor_sgd: ``param.add_(grad, alpha=-lr)``).
    Every product is rounded before its sum, as torch on CUDA does; tests/test_train_exact.py states this contract and
    checks the kernels and torch's CUDA optimizers against this function bit for bit."""
    g = g.astype(F32)
    if spec.kind == "sgd":
        p[rows] = (p[rows] + F32(-spec.lr) * g).astype(F32)
    elif spec.kind == "adagrad":
        G = state["sum"]
        G[rows] = (G[rows] + g * g).astype(F32)
        std = (np.sqrt(G[rows], dtype=F32) + F32(spec.eps)).astype(F32)
        p[rows] = (p[rows] + F32(-adagrad_clr(spec, step)) * (g / std).astype(F32)).astype(F32)
    elif spec.kind == "sparse_adam":
        b1, b2 = spec.betas
        m, v = state["exp_avg"], state["exp_avg_sq"]
        m_old, v_old = m[rows].copy(), v[rows].copy()
        um = ((g - m_old).astype(F32) * F32(1 - b1)).astype(F32)
        m[rows] = (m_old + um).astype(F32)
        uv = (((g * g).astype(F32) - v_old).astype(F32) * F32(1 - b2)).astype(F32)
        v[rows] = (v_old + uv).astype(F32)
        numer = (um + m_old).astype(F32)
        denom = (np.sqrt((uv + v_old).astype(F32), dtype=F32) + F32(spec.eps)).astype(F32)
        p[rows] = (p[rows] + F32(-adam_step_size(spec, step)) * (numer / denom).astype(F32)).astype(F32)
    else:
        raise ValueError(spec.kind)


def train_step(net_type: str, params, opt_state, batch, spec: OptSpec, step: int) -> np.float32:
    """One iteration of the reference ``fit`` loop body for the sparse scorers
    (model.py:274-284): two forwards, hinge, backward, optimizer.step().
    ``step`` is the 1-based per-parameter step count.  Mutates params/opt_state."""
    loss, grads = (linear_grads if net_type == "linear" else fm_grads)(params, batch)
    for name, (idx, vals) in grads.items():
        rows, g = coalesce(idx, vals)
        apply_rows(params[name], opt_state[name], rows, g, spec, step)
    return loss


# --------------------------------------------------------------------------------------
# a4  MLP tower (fp32 oracle), batch norm with per-pass statistics
# --------------------------------------------------------------------------------------
BN_EPS = 1e-5
BN_MOMENTUM = 0.1


def mlp_n_layers(params) -> int:
    n = 0
    while f"fcs.{n}.weight" in params:
        n += 1
    return n


def mlp_input(params, user, item, meta=None) -> np.ndarray:
    """concat[u, v, meta_f...] (collaborative/mlp.py:93-104)."""
    cols = [params["user.weight"][user], params["item.weight"][item]]
    for f, t in enumerate(_meta_tables(params, "metadata_embeddings")):
        cols.append(t[meta[:, f]])
    return np.concatenate(cols, axis=1).astype(F32)


def mlp_forward(params, x, train: bool, use_bn: bool = True, cache: Optional[list] = None):
    """(Linear -> BN -> ReLU) x n, then Linear(->1) (collaborative/mlp.py:106-113).
    In train mode BN uses this pass's batch statistics (biased variance) and updates the
    running statistics with the unbiased variance, momentum 0.1 (torch BatchNorm1d defaults,
    collaborative/mlp.py:82).  Returns (B,1)."""
    h = x.astype(F32)
    for l in range(mlp_n_layers(params)):
        W, b = params[f"fcs.{l}.weight"], params[f"fcs.{l}.bias"]
        z = (h @ W.T + b).astype(F32)
        if use_bn:
            gamma, beta = params[f"bns.{l}.weight"], params[f"bns.{l}.bias"]
            if train:
                mu = z.mean(axis=0, dtype=F32)
                var = z.var(axis=0, dtype=F32)
                n = z.shape[0]
                params[f"bns.{l}.running_mean"] = ((1 - BN_MOMENTUM) * params[f"bns.{l}.running_mean"]
                                                   + BN_MOMENTUM * mu).astype(F32)
                params[f"bns.{l}.running_var"] = ((1 - BN_MOMENTUM) * params[f"bns.{l}.running_var"]
                                                  + BN_MOMENTUM * var * (n / max(n - 1, 1))).astype(F32)
                params[f"bns.{l}.num_batches_tracked"] = params[f"bns.{l}.num_batches_tracked"] + 1
            else:
                mu, var = params[f"bns.{l}.running_mean"], params[f"bns.{l}.running_var"]
            rstd = (F32(1.0) / np.sqrt(var + F32(BN_EPS), dtype=F32)).astype(F32)
            xhat = ((z - mu) * rstd).astype(F32)
            y = (xhat * gamma + beta).astype(F32)
        else:
            xhat, rstd, y = None, None, z
        a = np.maximum(y, F32(0))
        if cache is not None:
            cache.append((h, xhat, rstd, y))
        h = a
    out = (h @ params["output_layer.weight"].T + params["output_layer.bias"]).astype(F32)
    if cache is not None:
        cache.append((h,))
    return out


def mlp_backward(params, cache, dout, use_bn: bool = True):
    """Backward of mlp_forward (train mode).  Returns (dx, dict of dense grads)."""
    grads = {}
    (h_last,) = cache[-1]
    grads["output_layer.weight"] = (dout.T @ h_last).astype(F32)
    grads["output_layer.bias"] = dout.sum(axis=0, dtype=F32)
    dh = (dout @ params["output_layer.weight"]).astype(F32)
    for l in reversed(range(mlp_n_layers(params))):
        h_in, xhat, rstd, y = cache[l]
        dy = np.where(y > 0, dh, F32(0)).astype(F32)
        if use_bn:
            gamma = params[f"bns.{l}.weight"]
            grads[f"bns.{l}.weight"] = (dy * xhat).sum(axis=0, dtype=F32)
            grads[f"bns.{l}.bias"] = dy.sum(axis=0, dtype=F32)
            n = F32(dy.shape[0])
            dxhat = (dy * gamma).astype(F32)
            dz = (rstd / n * (n * dxhat - dxhat.sum(axis=0, dtype=F32)
                              - xhat * (dxhat * xhat).sum(axis=0, dtype=F32))).astype(F32)
        else:
            dz = dy
        grads[f"fcs.{l}.weight"] = (dz.T @ h_in).astype(F32)
        grads[f"fcs.{l}.bias"] = dz.sum(axis=0, dtype=F32)
        dh = (dz @ params[f"fcs.{l}.weight"]).astype(F32)
    return dh, grads


def mlp_scores(params, user, item, meta=None, train=False, use_bn=True) -> np.ndarray:
    return mlp_forward(params, mlp_input(params, user, item, meta), train, use_bn)


def mlp_grads(params, batch, use_bn=True):
    """Loss, sparse embedding grads and dense grads for one MLP training step
    (model.py:171-185 two passes -> BN statistics and running stats per pass)."""
    user, pos, neg = batch["user"], batch["pos"], batch["neg"]
    pm, nm = batch.get("pos_meta"), batch.get("neg_meta")
    cp, cn = [], []
    sp = mlp_forward(params, mlp_input(params, user, pos, pm), True, use_bn, cp)
    sn = mlp_forward(params, mlp_input(params, user, neg, nm), True, use_bn, cn)
    loss = hinge_loss(sp, sn)
    g = hinge_weights(sp, sn)[:, None]
    dxp, gp = mlp_backward(params, cp, -g, use_bn)
    dxn, gn = mlp_backward(params, cn, g, use_bn)
    dense = {k: (gp[k] + gn[k]).astype(F32) for k in gp}
    D = params["user.weight"].shape[1]
    sparse: Dict[str, SparseGrad] = {
        "user.weight": (np.concatenate([user, user]), np.concatenate([dxp[:, :D], dxn[:, :D]])),
        "item.weight": (np.concatenate([pos, neg]), np.concatenate([dxp[:, D:2 * D], dxn[:, D:2 * D]])),
    }
    for f in range(len(_meta_tables(params, "metadata_embeddings"))):
        sl = slice((2 + f) * D, (3 + f) * D)
        sparse[f"metadata_embeddings.{f}.weight"] = (
            np.concatenate([pm[:, f], nm[:, f]]), np.concatenate([dxp[:, sl], dxn[:, sl]]))
    return loss, sparse, dense


def apply_dense(p, state, g, spec: OptSpec, step: int) -> None:
    """Dense Adagrad / SGD on the MLP weights (torch: optim/adagrad.py:380-385, sgd.py)."""
    if spec.kind == "sgd":
        p += (F32(-spec.lr) * g).astype(F32)
    elif spec.kind == "adagrad":
        state["sum"] += (g * g).astype(F32)
        std = np.sqrt(state["sum"], dtype=F32) + F32(spec.eps)
        p += (F32(-adagrad_clr(spec, step)) * (g / std)).astype(F32)
    else:
        raise ValueError("dense params need sgd or adagrad (SparseAdam rejects dense grads, SURVEY D2)")


def mlp_train_step(params, opt_state, batch, spec: OptSpec, step: int, use_bn=True) -> np.float32:
    loss, sparse, dense = mlp_grads(params, batch, use_bn)
    for name, (idx, vals) in sparse.items():
        rows, g = coalesce(idx, vals)
        apply_rows(params[name], opt_state[name], rows, g, spec, step)
    for name, g in dense.items():
        apply_dense(params[name], opt_state[name], g, spec, step)
    return loss


# --------------------------------------------------------------------------------------
# a9  negative sampling (Philox4x32-10, counter = global sample index)
# --------------------------------------------------------------------------------------
_PH_M0, _PH_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_PH_W0, _PH_W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al. 2011, Random123 reference constants) on uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint32).copy() for c in (c0, c1, c2, c3))
    k0, k1 = np.uint32(k0), np.uint32(k1)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _PH_M0 * c0.astype(np.uint64)
            p1 = _PH_M1 * c2.astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & _MASK32).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & _MASK32).astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0 = np.uint32((int(k0) + int(_PH_W0)) & 0xFFFFFFFF)
            k1 = np.uint32((int(k1) + int(_PH_W1)) & 0xFFFFFFFF)
    return c0, c1, c2, c3


def philox_negatives(seed: int, first_index: int, pos: np.ndarray, n_items: int) -> np.ndarray:
    """Dynamic negatives: uniform over [0, n_items) re-drawn while equal to the positive
    (dataset/dataset.py:435-447), drawn from Philox instead of numpy's global RNG.
    Sample j uses counter (lo32(idx), hi32(idx), block, 0) with idx = first_index + j and key
    (lo32(seed), hi32(seed)); candidate t (t = 0,1,2,...) is word t%4 of block t//4 mapped to
    [0, n_items) by ``(word * n_items) >> 32``.  Bit-exact against the CUDA kernel."""
    n = len(pos)
    idx = np.uint64(first_index) + np.arange(n, dtype=np.uint64)
    lo, hi = (idx & _MASK32).astype(np.uint32), (idx >> np.uint64(32)).astype(np.uint32)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    neg = np.full(n, -1, dtype=np.int64)
    todo = np.arange(n)
    block = 0
    while len(todo):
        words = philox4x32_10(lo[todo], hi[todo], np.full(len(todo), block, np.uint32),
                              np.zeros(len(todo), np.uint32), k0, k1)
        for w in words:
            cand = ((w.astype(np.uint64) * np.uint64(n_items)) >> np.uint64(32)).astype(np.int64)
            open_ = neg[todo] < 0
            ok = open_ & (cand != pos[todo])
            neg[todo[ok]] = cand[ok]
        todo = todo[neg[todo] < 0]
        block += 1
    return neg


# --------------------------------------------------------------------------------------
# a11  predict: all-item scores + top-k
# --------------------------------------------------------------------------------------
def topk_desc(scores: np.ndarray, k: int) -> np.ndarray:
    """Indices of the k largest scores, descending; ties -> lower item index first
    (== torch.sort(stable=True, descending=True)[:k]; the reference's sort at model.py:447
    is unstable, SURVEY.md D10, so this is the stated tie-break)."""
    order = np.argsort(-scores.astype(np.float64), kind="stable")
    return order[:k].astype(np.int64)


def predict_scores(net_type: str, params, user_id: int, n_items: int) -> np.ndarray:
    """Scores of one user against all items, as ``predict`` builds them chunk by chunk
    (model.py:383-443; metadata-free, SURVEY.md D8)."""
    users = np.full(n_items, user_id, dtype=np.int64)
    items = np.arange(n_items, dtype=np.int64)
    if net_type == "linear":
        return linear_scores(params, users, items).reshape(-1)
    if net_type == "fm":
        return fm_scores(params, users, items)
    return mlp_scores(params, users, items, train=False).reshape(-1)


def predict_topk(net_type: str, params, user_id: int, k: int) -> np.ndarray:
    n_items = params["item.weight"].shape[0]
    return topk_desc(predict_scores(net_type, params, user_id, n_items), k)
