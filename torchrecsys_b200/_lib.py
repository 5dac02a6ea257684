"""ctypes binding of include/trs.h (libtrs_b200.so).

There is no CPU fallback: if the library is missing or a call fails this module raises.  torch is
used only for device memory (``data_ptr()``) and the current CUDA stream."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

MAX_META = 8
NET_LINEAR, NET_FM = 0, 1
OPT_SGD, OPT_ADAGRAD, OPT_SPARSE_ADAM = 0, 1, 2

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtrs_b200.so")

# every symbol include/trs.h declares (tests/test_abi.py checks the .so exports them all)
SYMBOLS = [
    "trs_abi_version", "trs_last_error", "trs_device_info", "trs_embed_gather_sum", "trs_scores",
    "trs_philox_negatives", "trs_validate_ids", "trs_plan_bytes", "trs_plan_tmp_bytes",
    "trs_plan_build", "trs_train_workspace_bytes", "trs_train_steps", "trs_eval_pairwise",
    "trs_gemm_bf16_tn", "trs_mlp_forward_workspace_bytes", "trs_mlp_forward",
    "trs_mlp_train_workspace_bytes", "trs_mlp_train_steps", "trs_predict_topk_workspace_bytes",
    "trs_predict_topk", "trs_shard_stage_bytes", "trs_shard_plan_bytes", "trs_shard_plan_tmp_bytes",
    "trs_shard_plan_build", "trs_shard_workspace_bytes", "trs_shard_train_steps", "trs_ipc_export",
    "trs_ipc_open", "trs_ipc_close", "trs_scores_backward", "trs_sort_workspace_bytes", "trs_sorted_auc",
    "trs_epoch_shuffle", "trs_gather_rows_i64", "trs_predict_topk_reuse", "trs_shard_eval_pairwise",
    "trs_shard_gather_rows", "trs_shard_topk_exact_workspace_bytes", "trs_shard_topk_exact",
    "trs_shard_topk_merge_sorted",
]


class Table(C.Structure):
    _fields_ = [("emb", C.c_void_p), ("emb_s0", C.c_void_p), ("emb_s1", C.c_void_p),
                ("lin", C.c_void_p), ("lin_s0", C.c_void_p), ("lin_s1", C.c_void_p),
                ("n_rows", C.c_int64)]


class Model(C.Structure):
    _fields_ = [("net", C.c_int32), ("dim", C.c_int32), ("n_meta", C.c_int32), ("reserved", C.c_int32),
                ("user", Table), ("item", Table), ("meta", Table * MAX_META)]


class Epoch(C.Structure):
    _fields_ = [("user", C.c_void_p), ("pos", C.c_void_p), ("neg", C.c_void_p),
                ("pos_meta", C.c_void_p), ("neg_meta", C.c_void_p),
                ("n_samples", C.c_int64), ("batch", C.c_int32), ("reserved", C.c_int32)]


class Optim(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("step_scale", C.c_void_p)]


class GemmArgs(C.Structure):
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("lda", C.c_int64), ("ldb", C.c_int64),
                ("m", C.c_int64), ("n", C.c_int64), ("k", C.c_int64), ("out", C.c_void_p),
                ("ldc", C.c_int64), ("split_stride", C.c_int64), ("out_bf16", C.c_int32),
                ("splits", C.c_int32), ("a_mn", C.c_int32), ("b_mn", C.c_int32), ("bias", C.c_void_p), ("col_sum", C.c_void_p),
                ("col_sumsq", C.c_void_p), ("rows_per_half", C.c_int64), ("rows_valid", C.c_int64)]


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m torchrecsys_b200.build` "
                "(there is no CPU / eager fallback for the hot path)")
        L = C.CDLL(LIB_PATH)
        L.trs_last_error.restype = C.c_char_p
        for name in ("trs_plan_bytes", "trs_plan_tmp_bytes", "trs_train_workspace_bytes", "trs_shard_stage_bytes",
                     "trs_shard_plan_bytes", "trs_shard_plan_tmp_bytes", "trs_shard_workspace_bytes",
                     "trs_sort_workspace_bytes", "trs_shard_topk_exact_workspace_bytes"):
            getattr(L, name).restype = C.c_size_t
        if L.trs_abi_version() != 1:
            raise RuntimeError("libtrs_b200.so ABI version mismatch")
        _lib = L
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError(f"libtrs_b200: {lib().trs_last_error().decode()} (status {rc})")


def _ptr(t: Optional[torch.Tensor], dtype=None) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libtrs_b200 takes CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("tensor must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"expected {dtype}, got {t.dtype}")
    return t.data_ptr()


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def make_table(emb, emb_s0=None, emb_s1=None, lin=None, lin_s0=None, lin_s1=None) -> Table:
    f32 = torch.float32
    return Table(_ptr(emb, f32), _ptr(emb_s0, f32), _ptr(emb_s1, f32), _ptr(lin, f32),
                 _ptr(lin_s0, f32), _ptr(lin_s1, f32), emb.shape[0])


def make_model(net: int, dim: int, user: Table, item: Table, metas: Sequence[Table]) -> Model:
    if len(metas) > MAX_META:
        raise RuntimeError(f"at most {MAX_META} metadata features are supported")
    m = Model(net, dim, len(metas), 0, user, item)
    for f, t in enumerate(metas):
        m.meta[f] = t
    return m


def make_epoch(user, pos, neg, pos_meta=None, neg_meta=None, batch: int = 512) -> Epoch:
    i64 = torch.int64
    return Epoch(_ptr(user, i64), _ptr(pos, i64), _ptr(neg, i64), _ptr(pos_meta, i64),
                 _ptr(neg_meta, i64), user.shape[0], batch, 0)


def device_info():
    sm, grid, block = C.c_int(), C.c_int(), C.c_int()
    _check(lib().trs_device_info(C.byref(sm), C.byref(grid), C.byref(block)))
    return sm.value, grid.value, block.value


def embed_gather_sum(table, idx, meta_tables=(), meta_idx=None) -> torch.Tensor:
    n, dim = idx.shape[0], table.shape[1]
    out = torch.empty((n, dim), dtype=torch.float32, device=table.device)
    ptrs = (C.c_void_p * max(len(meta_tables), 1))(*[_ptr(t, torch.float32) for t in meta_tables])
    _check(lib().trs_embed_gather_sum(C.c_void_p(_ptr(table, torch.float32)), dim,
                                      C.c_void_p(_ptr(idx, torch.int64)), C.c_int64(n), ptrs,
                                      C.c_void_p(_ptr(meta_idx, torch.int64)), len(meta_tables),
                                      C.c_void_p(_ptr(out)), _stream()))
    return out


def scores(model: Model, user, item, meta=None) -> torch.Tensor:
    n = user.shape[0]
    out = torch.empty(n, dtype=torch.float32, device=user.device)
    _check(lib().trs_scores(C.byref(model), C.c_void_p(_ptr(user, torch.int64)),
                            C.c_void_p(_ptr(item, torch.int64)), C.c_void_p(_ptr(meta, torch.int64)),
                            C.c_int64(n), C.c_void_p(_ptr(out)), _stream()))
    return out


def philox_negatives(seed: int, first_index: int, pos, n_items: int, item_meta=None):
    n = pos.shape[0]
    neg = torch.empty_like(pos)
    n_meta = 0 if item_meta is None else item_meta.shape[1]
    neg_meta = None if item_meta is None else torch.empty((n, n_meta), dtype=torch.int64, device=pos.device)
    _check(lib().trs_philox_negatives(C.c_uint64(seed), C.c_uint64(first_index),
                                      C.c_void_p(_ptr(pos, torch.int64)), C.c_int64(n),
                                      C.c_int64(n_items), C.c_void_p(_ptr(item_meta, torch.int64)),
                                      n_meta, C.c_void_p(_ptr(neg)), C.c_void_p(_ptr(neg_meta)), _stream()))
    return neg, neg_meta


def count_bad_ids(ids, n_rows: int, counter: torch.Tensor) -> None:
    _check(lib().trs_validate_ids(C.c_void_p(_ptr(ids, torch.int64)), C.c_int64(ids.numel()),
                                  C.c_int64(n_rows), C.c_void_p(_ptr(counter, torch.int32)), _stream()))


def _grown(buf, nbytes: int, device) -> torch.Tensor:
    """A uint8 device buffer of at least nbytes: `buf` if it is big enough, else a new one."""
    if buf is not None and buf.numel() >= nbytes and buf.device == torch.device(device):
        return buf
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)


def plan_build(model: Model, epoch: Epoch, device, plan=None, tmp=None) -> torch.Tensor:
    """Builds the epoch's sort plan; `plan` / `tmp` are reused when they are large enough."""
    L = lib()
    nbytes = L.trs_plan_bytes(C.byref(model), C.byref(epoch))
    tbytes = L.trs_plan_tmp_bytes(C.byref(model), C.byref(epoch))
    plan = _grown(plan, nbytes, device)
    tmp = _grown(tmp, tbytes, device)
    _check(L.trs_plan_build(C.byref(model), C.byref(epoch), C.c_void_p(plan.data_ptr()),
                            C.c_size_t(plan.numel()), C.c_void_p(tmp.data_ptr()), C.c_size_t(tmp.numel()), _stream()))
    return plan


def train_buffer_bytes(model: Model, epoch: Epoch):
    """(plan, plan scratch, training workspace) sizes in bytes for an epoch of this shape."""
    L = lib()
    return (L.trs_plan_bytes(C.byref(model), C.byref(epoch)), L.trs_plan_tmp_bytes(C.byref(model), C.byref(epoch)),
            L.trs_train_workspace_bytes(C.byref(model), C.byref(epoch)))


def train_workspace(model: Model, epoch: Epoch, device) -> torch.Tensor:
    nbytes = lib().trs_train_workspace_bytes(C.byref(model), C.byref(epoch))
    if nbytes == 0:
        raise RuntimeError(f"libtrs_b200: {lib().trs_last_error().decode()}")
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def train_steps(model: Model, epoch: Epoch, optim: Optim, plan, workspace, first_step: int,
                n_steps: int, loss_out: torch.Tensor) -> None:
    _check(lib().trs_train_steps(C.byref(model), C.byref(epoch), C.byref(optim),
                                 C.c_void_p(plan.data_ptr()), C.c_void_p(workspace.data_ptr()),
                                 C.c_size_t(workspace.numel()), first_step, n_steps,
                                 C.c_void_p(_ptr(loss_out, torch.float32)), _stream()))


def eval_pairwise(model: Model, epoch: Epoch, want_scores: bool = False):
    n = epoch.n_samples
    nb = (n + epoch.batch - 1) // epoch.batch
    dev = torch.device("cuda", torch.cuda.current_device())
    loss = torch.empty(nb, dtype=torch.float32, device=dev)
    auc = torch.empty(nb, dtype=torch.float32, device=dev)
    pos = torch.empty(n, dtype=torch.float32, device=dev) if want_scores else None
    neg = torch.empty(n, dtype=torch.float32, device=dev) if want_scores else None
    _check(lib().trs_eval_pairwise(C.byref(model), C.byref(epoch), C.c_void_p(_ptr(loss)),
                                   C.c_void_p(_ptr(auc)), C.c_void_p(_ptr(pos)), C.c_void_p(_ptr(neg)),
                                   _stream()))
    return loss, auc, pos, neg


def gemm_bf16_tn(a, b, out, bias=None, splits: int = 1, col_sum=None, col_sumsq=None,
                 rows_per_half: int = 0, rows_valid: int = 0, a_mn: bool = False, b_mn: bool = False) -> None:
    """out[m, n] = sum_k a[m, k] * b[n, k] (+ bias[n]); a, b bf16 row-major (last dim contiguous);
    with a_mn / b_mn the operand is passed as stored [k, m] / [k, n].
    out fp32 or bf16 ([m, n], or [splits, m, n] fp32 partials when splits > 1)."""
    bf = torch.bfloat16
    for t in (a, b):
        if t.dtype != bf or t.dim() != 2 or t.stride(1) != 1 or not t.is_cuda:
            raise RuntimeError("gemm_bf16_tn takes 2-D bf16 CUDA operands with a contiguous last dimension")
    k, m = a.shape if a_mn else a.shape[::-1]
    kb, n = b.shape if b_mn else b.shape[::-1]
    if kb != k:
        raise RuntimeError("gemm_bf16_tn: k mismatch")
    o2 = out if splits == 1 else out[0]
    if tuple(o2.shape) != (m, n) or o2.stride(1) != 1 or out.dtype not in (bf, torch.float32):
        raise RuntimeError("gemm_bf16_tn: bad output")
    args = GemmArgs(a.data_ptr(), b.data_ptr(), a.stride(0), b.stride(0), m, n, k, out.data_ptr(),
                    o2.stride(0), out.stride(0) if splits > 1 else 0, int(out.dtype == bf), splits,
                    int(a_mn), int(b_mn), _ptr(bias, torch.float32), _ptr(col_sum, torch.float32), _ptr(col_sumsq, torch.float32),
                    rows_per_half, rows_valid)
    _check(lib().trs_gemm_bf16_tn(C.byref(args), _stream()))


# ---- MLP tower (include/trs.h: trs_mlp) -------------------------------------------------------------
MAX_LAYERS = 8
NET_MLP = 2
_PL = C.c_void_p * MAX_LAYERS


class Mlp(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("use_bn", C.c_int32), ("hidden", C.c_int32 * MAX_LAYERS),
                ("W", _PL), ("b", _PL), ("gamma", _PL), ("beta", _PL), ("running_mean", _PL),
                ("running_var", _PL), ("w_out", C.c_void_p), ("b_out", C.c_void_p),
                ("dW", _PL), ("db", _PL), ("dgamma", _PL), ("dbeta", _PL), ("dw_out", C.c_void_p),
                ("db_out", C.c_void_p), ("s0W", _PL), ("s0b", _PL), ("s0gamma", _PL), ("s0beta", _PL),
                ("s0w_out", C.c_void_p), ("s0b_out", C.c_void_p)]


def mlp_forward(model: Model, mlp: Mlp, user, item, meta=None, batch_stats: bool = False) -> torch.Tensor:
    """Scores of n (user, item[, meta]) rows through the tower; eval-mode BatchNorm unless batch_stats."""
    L = lib()
    L.trs_mlp_forward_workspace_bytes.restype = C.c_size_t
    n = user.shape[0]
    out = torch.empty(n, dtype=torch.float32, device=user.device)
    chunk = n if batch_stats else 1 << 16  # eval mode is row-independent: bound the activation workspace
    ws = None
    for lo in range(0, n, max(chunk, 1)):
        hi = min(n, lo + chunk)
        nbytes = L.trs_mlp_forward_workspace_bytes(C.byref(model), C.byref(mlp), C.c_int64(hi - lo))
        if nbytes == 0:
            raise RuntimeError(f"libtrs_b200: {L.trs_last_error().decode()}")
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=user.device)
        m = None if meta is None else meta[lo:hi]
        _check(L.trs_mlp_forward(C.byref(model), C.byref(mlp), C.c_void_p(_ptr(user[lo:hi], torch.int64)),
                                 C.c_void_p(_ptr(item[lo:hi], torch.int64)), C.c_void_p(_ptr(m, torch.int64)),
                                 C.c_int64(hi - lo), int(batch_stats), C.c_void_p(out[lo:hi].data_ptr()),
                                 C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), _stream()))
    return out


def mlp_train_workspace(model: Model, mlp: Mlp, epoch: Epoch, device) -> torch.Tensor:
    L = lib()
    L.trs_mlp_train_workspace_bytes.restype = C.c_size_t
    nbytes = L.trs_mlp_train_workspace_bytes(C.byref(model), C.byref(mlp), C.byref(epoch))
    if nbytes == 0:
        raise RuntimeError(f"libtrs_b200: {L.trs_last_error().decode()}")
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def mlp_train_steps(model: Model, mlp: Mlp, epoch: Epoch, optim: Optim, plan, workspace, first_step: int,
                    n_steps: int, loss_out: torch.Tensor) -> None:
    _check(lib().trs_mlp_train_steps(C.byref(model), C.byref(mlp), C.byref(epoch), C.byref(optim),
                                     C.c_void_p(plan.data_ptr()), C.c_void_p(workspace.data_ptr()),
                                     C.c_size_t(workspace.numel()), first_step, n_steps,
                                     C.c_void_p(_ptr(loss_out, torch.float32)), _stream()))


class TopkCache:
    """Keeps the predict workspace -- with the prepared bf16 item operand inside -- between calls.  ``key`` is whatever
    the caller uses to say "the item tables have not changed" (model.py: tensor versions + the fused runners'
    update counter); a different key, query count or k rebuilds."""

    def __init__(self):
        self.ws, self.key = None, None


def predict_topk(model: Model, users, k: int, item_meta=None, item_offset: int = 0, cache: Optional[TopkCache] = None,
                 cache_key=None):
    """Top-k items for each user id in ``users`` against all items of ``model.item``.
    Returns (idx int64 [n, k], score fp32 [n, k], overflow int32 [n])."""
    L = lib()
    L.trs_predict_topk_workspace_bytes.restype = C.c_size_t
    n = users.shape[0]
    dev = users.device
    idx = torch.empty((n, k), dtype=torch.int64, device=dev)
    score = torch.empty((n, k), dtype=torch.float32, device=dev)
    over = torch.empty(n, dtype=torch.int32, device=dev)
    if n == 0:
        return idx, score, over
    nbytes = L.trs_predict_topk_workspace_bytes(C.byref(model), C.c_int64(n), k)
    if nbytes == 0:
        raise RuntimeError(f"libtrs_b200: {L.trs_last_error().decode()}")
    key = (cache_key, n, k, int(model.item.emb or 0), nbytes, str(dev))
    reuse = cache is not None and cache.ws is not None and cache.key == key and cache_key is not None
    if reuse:
        ws = cache.ws
    else:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        if cache is not None:
            cache.ws, cache.key = ws, key
    _check(L.trs_predict_topk_reuse(C.byref(model), C.c_void_p(_ptr(users, torch.int64)), C.c_int64(n),
                                    C.c_void_p(_ptr(item_meta, torch.int64)), k, C.c_int64(item_offset),
                                    C.c_void_p(idx.data_ptr()), C.c_void_p(score.data_ptr()),
                                    C.c_void_p(over.data_ptr()), C.c_void_p(ws.data_ptr()),
                                    C.c_size_t(nbytes), int(reuse), _stream()))
    return idx, score, over


# ---- row-sharded training over peer-mapped shards (include/trs.h: trs_shard) ---------------------------
MAX_RANKS = 8
SHARD_SYNC_BYTES = 4096


class Shard(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("dim", C.c_int32), ("reserved", C.c_int32),
                ("n_users", C.c_int64), ("n_items", C.c_int64), ("user", Table * MAX_RANKS),
                ("item", Table * MAX_RANKS), ("stage", C.c_void_p * MAX_RANKS), ("sync", C.c_void_p * MAX_RANKS)]


def table_at(base: int, emb_off, s0_off, s1_off, lin_off, lin_s0_off, lin_s1_off, n_rows: int) -> Table:
    """A trs_table from raw device addresses: ``base`` + byte offsets (None = absent)."""
    at = lambda o: None if o is None else base + o
    return Table(at(emb_off), at(s0_off), at(s1_off), at(lin_off), at(lin_s0_off), at(lin_s1_off), n_rows)


def shard_stage_bytes(dim: int, global_batch: int) -> int:
    return lib().trs_shard_stage_bytes(dim, global_batch)


def shard_plan_build(shard: Shard, epoch: Epoch, device, plan=None, tmp=None) -> torch.Tensor:
    L = lib()
    plan = _grown(plan, L.trs_shard_plan_bytes(C.byref(epoch)), device)
    tmp = _grown(tmp, L.trs_shard_plan_tmp_bytes(C.byref(epoch)), device)
    _check(L.trs_shard_plan_build(C.byref(shard), C.byref(epoch), C.c_void_p(plan.data_ptr()), C.c_size_t(plan.numel()),
                                  C.c_void_p(tmp.data_ptr()), C.c_size_t(tmp.numel()), _stream()))
    return plan


def shard_train_steps(shards: Sequence[Shard], epoch: Epoch, optim: Optim, plans: Sequence[torch.Tensor],
                      first_step: int, n_steps: int, sync_epoch: int, loss_sums: Sequence[torch.Tensor],
                      status: torch.Tensor, workspace=None, timeout_ms: int = 20000) -> torch.Tensor:
    """One persistent launch for the local ranks (1 in production, the whole group when one GPU emulates it).
    Returns the workspace so the caller can keep it for the next call."""
    L = lib()
    n = len(shards)
    arr = (Shard * n)(*shards)
    nbytes = L.trs_shard_workspace_bytes(C.byref(epoch), n)
    if nbytes == 0:
        raise RuntimeError("libtrs_b200: bad shard workspace query")
    workspace = _grown(workspace, nbytes, status.device)
    plan_ptrs = (C.c_void_p * n)(*[p.data_ptr() for p in plans])
    loss_ptrs = (C.c_void_p * n)(*[_ptr(t, torch.float32) for t in loss_sums])
    _check(L.trs_shard_train_steps(arr, n, C.byref(epoch), C.byref(optim), plan_ptrs, C.c_void_p(workspace.data_ptr()),
                                   C.c_size_t(workspace.numel()), first_step, n_steps, C.c_uint64(sync_epoch), loss_ptrs,
                                   C.c_void_p(_ptr(status, torch.int32)), timeout_ms, _stream()))
    return workspace


def shard_eval_pairwise(shard: Shard, epoch: Epoch, first_batch: int, n_batches: int, loss, auc, pos=None,
                        neg=None) -> None:
    """Batches [first_batch, first_batch + n_batches) of the global epoch, every row read from its owner: loss / auc
    [>= n_batches] and the optional scores pos / neg [>= the range's samples] are written from index 0."""
    f32 = torch.float32
    _check(lib().trs_shard_eval_pairwise(C.byref(shard), C.byref(epoch), C.c_int64(first_batch), C.c_int64(n_batches),
                                         C.c_void_p(_ptr(loss, f32)), C.c_void_p(_ptr(auc, f32)),
                                         C.c_void_p(_ptr(pos, f32)), C.c_void_p(_ptr(neg, f32)), _stream()))


def shard_gather_rows(shard: Shard, table: int, ids, device):
    """(rows [n, dim], biases [n, 1]) of global ids of the user (0) or item (1) table, copied from their owners."""
    n = ids.shape[0]
    emb = torch.empty((n, shard.dim), dtype=torch.float32, device=device)
    lin = torch.empty((n, 1), dtype=torch.float32, device=device)
    _check(lib().trs_shard_gather_rows(C.byref(shard), table, C.c_void_p(_ptr(ids, torch.int64)), C.c_int64(n),
                                       C.c_void_p(emb.data_ptr()), C.c_void_p(lin.data_ptr()), _stream()))
    return emb, lin


def shard_topk_exact(shard: Shard, user_emb, user_lin, k: int, excl_ptr=None, excl_ids=None, workspace=None):
    """Exact top-k of rank ``shard.rank``'s own item shard for the query rows user_emb [Q, dim] / user_lin [Q] ->
    (global idx int64 [Q, k], score fp32 [Q, k], workspace to keep), -1 / -inf padded.  excl_ptr [Q + 1] / excl_ids:
    per query position, the sorted local item ids of this shard to leave out."""
    L = lib()
    n = user_emb.shape[0]
    dev = user_emb.device
    idx = torch.empty((n, k), dtype=torch.int64, device=dev)
    score = torch.empty((n, k), dtype=torch.float32, device=dev)
    nbytes = L.trs_shard_topk_exact_workspace_bytes(C.byref(shard), C.c_int64(n), k)
    if nbytes == 0:
        raise RuntimeError(f"libtrs_b200: {L.trs_last_error().decode()}")
    workspace = _grown(workspace, nbytes, dev)
    i64 = torch.int64
    _check(L.trs_shard_topk_exact(C.byref(shard), C.c_void_p(_ptr(user_emb, torch.float32)),
                                  C.c_void_p(_ptr(user_lin, torch.float32)), C.c_int64(n), k,
                                  C.c_void_p(_ptr(excl_ptr, i64)), C.c_void_p(_ptr(excl_ids, i64)),
                                  C.c_void_p(idx.data_ptr()), C.c_void_p(score.data_ptr()),
                                  C.c_void_p(workspace.data_ptr()), C.c_size_t(workspace.numel()), _stream()))
    return idx, score, workspace


def topk_merge_sorted(score, idx, k: int, excl_ptr=None, excl_ids=None):
    """Sorted lists score / idx [n_lists, n_query, k_in] -> merged (idx [n_query, k], score [n_query, k]) by (score
    desc, id asc), -1 / -inf padded; excl_ptr [n_query + 1] / excl_ids drop the given ids of each query."""
    n_lists, nq, k_in = score.shape
    out_idx = torch.empty((nq, k), dtype=torch.int64, device=score.device)
    out_score = torch.empty((nq, k), dtype=torch.float32, device=score.device)
    i64 = torch.int64
    _check(lib().trs_shard_topk_merge_sorted(C.c_void_p(_ptr(score, torch.float32)), C.c_void_p(_ptr(idx, i64)),
                                             n_lists, C.c_int64(nq), k_in, k, C.c_void_p(_ptr(excl_ptr, i64)),
                                             C.c_void_p(_ptr(excl_ids, i64)), C.c_void_p(out_idx.data_ptr()),
                                             C.c_void_p(out_score.data_ptr()), _stream()))
    return out_idx, out_score


def ipc_export(t: torch.Tensor):
    """(64-byte handle, offset) of the CUDA allocation that holds tensor ``t`` -- for a peer process to map."""
    handle = (C.c_ubyte * 64)()
    off = C.c_uint64()
    _check(lib().trs_ipc_export(C.c_void_p(t.data_ptr()), handle, C.byref(off)))
    return bytes(handle), int(off.value)


def ipc_open(handle: bytes) -> int:
    base = C.c_void_p()
    buf = (C.c_ubyte * 64).from_buffer_copy(handle)
    _check(lib().trs_ipc_open(buf, C.byref(base)))
    return int(base.value)


def ipc_close(base: int) -> None:
    _check(lib().trs_ipc_close(C.c_void_p(base)))


# ---- autograd-visible forward, sorted AUC, epoch shuffle (csrc/extra.cu) ---------------------------------
def scores_backward(model: Model, user, item, meta, grad_out, with_lin_user: bool, with_lin_item: bool,
                    meta_lin: Sequence[bool]):
    """Per-lookup gradient rows of ``scores``: (g_user [n, D], g_item [n, D], [g_meta_f], g_lin_user, g_lin_item,
    [g_lin_meta_f]); absent companions are None."""
    n, dim, F = user.shape[0], model.dim, model.n_meta
    dev = user.device
    f32 = torch.float32
    row = lambda: torch.empty((n, dim), dtype=f32, device=dev)
    vec = lambda: torch.empty(n, dtype=f32, device=dev)
    g_user, g_item = row(), row()
    g_meta = [row() for _ in range(F)]
    g_lu = vec() if with_lin_user else None
    g_li = vec() if with_lin_item else None
    g_lm = [vec() if (f < len(meta_lin) and meta_lin[f]) else None for f in range(F)]
    pm = (C.c_void_p * max(F, 1))(*[t.data_ptr() for t in g_meta])
    plm = (C.c_void_p * max(F, 1))(*[None if t is None else t.data_ptr() for t in g_lm])
    _check(lib().trs_scores_backward(C.byref(model), C.c_void_p(_ptr(user, torch.int64)),
                                     C.c_void_p(_ptr(item, torch.int64)), C.c_void_p(_ptr(meta, torch.int64)),
                                     C.c_int64(n), C.c_void_p(_ptr(grad_out, f32)), C.c_void_p(g_user.data_ptr()),
                                     C.c_void_p(g_item.data_ptr()), pm, C.c_void_p(_ptr(g_lu)), C.c_void_p(_ptr(g_li)),
                                     plm, _stream()))
    return g_user, g_item, g_meta, g_lu, g_li, g_lm


def _sort_ws(n: int, device) -> torch.Tensor:
    return torch.empty(lib().trs_sort_workspace_bytes(C.c_int64(n)), dtype=torch.uint8, device=device)


def sorted_auc(pos: torch.Tensor, neg: torch.Tensor) -> torch.Tensor:
    """ROC-AUC of positive vs negative scores (fp32 CUDA tensors) -> device float64 scalar tensor [1]."""
    pos, neg = pos.reshape(-1).contiguous(), neg.reshape(-1).contiguous()
    dev = pos.device
    out = torch.empty(1, dtype=torch.float64, device=dev)
    n = pos.numel() + neg.numel()
    ws = _sort_ws(n, dev)
    _check(lib().trs_sorted_auc(C.c_void_p(_ptr(pos, torch.float32) if pos.numel() else None), C.c_int64(pos.numel()),
                                C.c_void_p(_ptr(neg, torch.float32) if neg.numel() else None), C.c_int64(neg.numel()),
                                C.c_void_p(out.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), _stream()))
    return out


def epoch_shuffle(seed: int, n: int, device) -> torch.Tensor:
    """A Philox-keyed permutation of [0, n) as an int64 device tensor."""
    perm = torch.empty(n, dtype=torch.int64, device=device)
    if n:
        ws = _sort_ws(n, device)
        _check(lib().trs_epoch_shuffle(C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), C.c_int64(n), C.c_void_p(perm.data_ptr()),
                                       C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), _stream()))
    return perm


def gather_rows(columns: Sequence[torch.Tensor], perm: torch.Tensor):
    """[col[perm] for col in columns] for int64 id columns ([n] or [n, w]) in ONE launch."""
    n = perm.shape[0]
    outs = [torch.empty((n,) + tuple(c.shape[1:]), dtype=torch.int64, device=perm.device) for c in columns]
    k = len(columns)
    if n == 0 or k == 0:
        return outs
    src = (C.c_void_p * k)(*[_ptr(c, torch.int64) for c in columns])
    dst = (C.c_void_p * k)(*[o.data_ptr() for o in outs])
    width = (C.c_int32 * k)(*[int(c.numel() // max(c.shape[0], 1)) for c in columns])
    _check(lib().trs_gather_rows_i64(src, dst, width, k, C.c_void_p(_ptr(perm, torch.int64)), C.c_int64(n), _stream()))
    return outs
