"""Multi-GPU paths for tables that do not fit (or should not be replicated on) one GPU -- SURVEY.md §8e.
The reference is single-device (model.py:74, README.md:3); this is new design: one process per GPU,
``torch.distributed`` (NCCL; gloo in the CPU tests) for rendezvous, the per-epoch id all-gather and the loss
all-reduce -- and NO collective on the step path:

Row-sharded training (BASELINE configs[3], Linear 50M x 5M, dim 128)  -- ``ShardedLinearTrainer``
    owner(row) = row % G, local row = row // G  (uniform load under any id skew).
    Every rank holds its shards, their optimizer state, a gradient staging buffer and a page of barrier words in
    ONE device allocation (the *arena*) and maps every peer's arena into its own address space by CUDA IPC.
    ``train_epoch`` takes the GLOBAL epoch (every rank's samples in loader order, identical on all ranks) and runs
    it as one persistent kernel per rank (csrc/shard.cu): a rank runs the samples whose user row it owns, reads
    item rows straight from their owner's HBM over NVLink, stores each lookup's gradient row straight into its
    owner's staging buffer, and every owner coalesces + updates its own rows -- two flag barriers per step.
    ``state_dict()`` / ``load_state_dict()`` gather / scatter the shards (parameters AND optimizer state) in the
    reference's single-process layout and key names, so checkpoints interchange with ``TorchRecSys``.
    ``evaluate`` / ``eval_pairwise`` / ``lookup`` serve the model where it lives: their kernels
    (csrc/shard_serve.cu) read every row from its owner through the same peer mappings, nothing is gathered.
    ``recommend`` (and ``predict_topk``, its narrower form) ranks each rank's own item shard (csrc/shard_topk.cu)
    and merges the ranks' sorted lists with trs_shard_topk_merge_sorted.
    One GPU can host the whole group (``emulate_world=G``): the parity tests run that way on a 1-GPU box.

Item-sharded predict (BASELINE configs[4])
    contiguous item blocks per rank (global id = offset + local id, so the single-GPU tie-break "lower item id
    first" carries over), user rows replicated; each rank runs trs_predict_topk on its block, each user's
    sorted (score, id)[k] lists go to one merger rank by all_to_all, are merged there by
    trs_shard_topk_merge_sorted, and the results are all-gathered."""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from .engine import OptBinding, step_scales

_KINDS = {"sgd": 0, "adagrad": 1, "sparse_adam": 2}
_STATE_KEYS = {"sgd": (), "adagrad": ("sum",), "sparse_adam": ("exp_avg", "exp_avg_sq")}


def shard_rows(n: int, rank: int, world: int) -> int:
    """Rows r of a table of n with r % world == rank."""
    return (n - rank + world - 1) // world if n > rank else 0


class _ArenaLayout:
    """Byte offsets inside a rank's arena -- the same on every rank (shards are sized for ceil(n / world) rows)."""

    def __init__(self, n_users: int, n_items: int, dim: int, n_state: int, world: int, stage_bytes: int, sync_bytes: int):
        off = 0

        def take(nbytes: int) -> int:
            nonlocal off
            o = off
            off += (nbytes + 255) // 256 * 256
            return o

        self.rows = {"user": -(-n_users // world), "item": -(-n_items // world)}
        self.emb, self.emb_state, self.lin, self.lin_state = {}, {}, {}, {}
        for name in ("user", "item"):
            r = max(self.rows[name], 1)
            self.emb[name] = take(r * dim * 4)
            self.emb_state[name] = [take(r * dim * 4) for _ in range(n_state)]
            self.lin[name] = take(r * 4)
            self.lin_state[name] = [take(r * 4) for _ in range(n_state)]
        self.stage = take(stage_bytes)
        self.sync = take(sync_bytes)
        self.total = off


class ShardedLinearTrainer:
    """Linear scorer (collaborative/linear.py:8-80) with user / item tables row-sharded over the ranks of ``group``.

    ``global_batch`` is the largest step (samples over ALL ranks) ``train_epoch`` will be asked to run: it sizes
    the staging buffers, which are part of the peer-mapped arena.  ``emulate_world=G`` builds all G ranks inside
    this process on the current GPU (no torch.distributed needed)."""

    def __init__(self, n_users: int, n_items: int, dim: int, global_batch: int, optimizer: str = "sparse_adam",
                 lr: float = 1e-3, device=None, group=None, betas=(0.9, 0.999), eps: Optional[float] = None,
                 lr_decay: float = 0.0, emulate_world: Optional[int] = None, timeout_ms: int = 20000):
        from . import _lib
        self._lib = _lib
        self.group = group
        if emulate_world:
            self.world, self.local_ranks = int(emulate_world), list(range(int(emulate_world)))
            self.rank = 0
        else:
            self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
            self.local_ranks = [self.rank]
        if not 1 <= self.world <= _lib.MAX_RANKS:
            raise ValueError(f"world size {self.world} outside 1..{_lib.MAX_RANKS}")
        if dim % 4 or dim <= 0 or dim > 512:
            raise ValueError("row-sharded training needs n_factors to be a multiple of 4 (<= 512)")
        if optimizer not in _KINDS:
            raise ValueError(f"optimizer must be one of {sorted(_KINDS)}")
        self.dim, self.n_users, self.n_items = dim, n_users, n_items
        self.global_batch = int(global_batch)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.kind = optimizer
        eps = eps if eps is not None else (1e-8 if optimizer == "sparse_adam" else 1e-10)
        self.binding = OptBinding(_KINDS[optimizer], _STATE_KEYS[optimizer], float(lr), float(betas[0]),
                                  float(betas[1]), float(eps), float(lr_decay), 0)
        self.timeout_ms = timeout_ms
        self.sync_epoch = 0   # cross-rank barriers the group has passed (2 per step), identical on every rank
        n_state = len(_STATE_KEYS[optimizer])
        self.layout = _ArenaLayout(n_users, n_items, dim, n_state, self.world,
                                   _lib.shard_stage_bytes(dim, self.global_batch), _lib.SHARD_SYNC_BYTES)
        # one allocation per local rank; barrier words zeroed once, tables initialised like the reference's
        # ScaledEmbedding / ZeroEmbedding (embeddings/init_embeddings.py:43-50, 90-97): N(0, 1/dim), zero biases
        self.arenas: Dict[int, torch.Tensor] = {}
        self.tables: Dict[int, Dict[str, Tuple[torch.Tensor, torch.Tensor]]] = {}
        self.state: Dict[int, Dict[str, List[Tuple[torch.Tensor, torch.Tensor]]]] = {}
        L = self.layout
        for r in self.local_ranks:
            arena = torch.empty(L.total, dtype=torch.uint8, device=self.device)
            arena[L.sync:L.sync + _lib.SHARD_SYNC_BYTES].zero_()
            self.arenas[r] = arena
            self.tables[r], self.state[r] = {}, {}
            for name, n in (("user", n_users), ("item", n_items)):
                rows = shard_rows(n, r, self.world)
                view = lambda off, cols: arena[off:off + rows * cols * 4].view(torch.float32).view(rows, cols)
                emb, lin = view(L.emb[name], dim), view(L.lin[name], 1)
                emb.normal_(0.0, 1.0 / dim)
                lin.zero_()
                self.tables[r][name] = (emb, lin)
                self.state[r][name] = []
                for i in range(n_state):
                    s_e, s_l = view(L.emb_state[name][i], dim), view(L.lin_state[name][i], 1)
                    s_e.zero_()
                    s_l.zero_()
                    self.state[r][name].append((s_e, s_l))
        self._map_peers()
        self._plans: Dict[int, torch.Tensor] = {}
        self._plan_tmp = None
        self._ws = None
        self._inv_counts = None
        self._h2d = None          # train_epoch_host: two device id buffers + the copy stream
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.launches = 0
        self._state_version = 0   # bumped by load_state_dict: with sync_epoch, says whether the tables changed
        self._topk_caches: Dict[int, object] = {}   # per local rank: predict's prepared bf16 item-shard operand
        # users the last predict_topk / recommend re-ranked exactly on this process's shards because the tensor-core
        # top-k flagged their candidate set as overflowing
        self.last_predict_overflow = 0
        self.last_recommend_paths: Dict[int, str] = {}   # local rank -> "tensor core" / "exact" of the last recommend

    # ---- peer mapping -----------------------------------------------------------------------------
    def _map_peers(self) -> None:
        """bases[q] = address of rank q's arena in THIS process."""
        _lib = self._lib
        self._opened: List[int] = []
        if self.device.type != "cuda":  # host-logic tests: checkpoints work on CPU arenas, training does not
            self.bases = None
            return
        if len(self.local_ranks) == self.world:
            self.bases = [self.arenas[q].data_ptr() for q in range(self.world)]
            return
        handle, off = _lib.ipc_export(self.arenas[self.rank])
        everyone: List = [None] * self.world
        dist.all_gather_object(everyone, (handle, off), group=self.group)
        self.bases = []
        for q, (h, o) in enumerate(everyone):
            if q == self.rank:
                self.bases.append(self.arenas[q].data_ptr())
            else:
                base = _lib.ipc_open(h)
                self._opened.append(base)
                self.bases.append(base + o)
        dist.barrier(group=self.group)  # every arena is initialised and mapped before anyone trains

    def close(self) -> None:
        for base in getattr(self, "_opened", []):
            self._lib.ipc_close(base)
        self._opened = []

    def _shard_struct(self, r: int):
        """trs_shard of local rank r: every rank's tables / staging / barrier words at their mapped addresses."""
        _lib, L = self._lib, self.layout
        sh = _lib.Shard()
        sh.rank, sh.world, sh.dim = r, self.world, self.dim
        sh.n_users, sh.n_items = self.n_users, self.n_items
        pick = lambda offs, i: offs[i] if i < len(offs) else None
        for q in range(self.world):
            for name, arr, n in (("user", sh.user, self.n_users), ("item", sh.item, self.n_items)):
                es, ls = L.emb_state[name], L.lin_state[name]
                arr[q] = _lib.table_at(self.bases[q], L.emb[name], pick(es, 0), pick(es, 1), L.lin[name], pick(ls, 0),
                                       pick(ls, 1), shard_rows(n, q, self.world))
            sh.stage[q] = self.bases[q] + L.stage
            sh.sync[q] = self.bases[q] + L.sync
        return sh

    # ---- training -----------------------------------------------------------------------------------
    def train_epoch(self, user: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, global_batch: Optional[int] = None,
                    check: bool = True, timing: bool = False, _scales: Optional[torch.Tensor] = None) -> torch.Tensor:
        """user / pos / neg: the GLOBAL epoch (int64 device tensors, identical on every rank), step s = samples
        [s*B, (s+1)*B) with B = ``global_batch``.  Returns the per-step batch-mean hinge losses (device, [n_steps]) --
        what ``loss.item()`` returns at model.py:200.  ``check=False`` skips the status read-back (no host sync);
        call ``check_status()`` later.  ``timing=True`` brackets the plan build and the persistent kernel with CUDA
        events (``self.events = (plan0, plan1, kernel0, kernel1)``, bench.py's roofline)."""
        _lib = self._lib
        if self.bases is None:
            raise RuntimeError("torchrecsys_b200 has no CPU fallback: row-sharded training needs CUDA devices")
        B = int(global_batch or self.global_batch)
        if B > self.global_batch:
            raise ValueError(f"global batch {B} exceeds the {self.global_batch} the staging buffers were sized for")
        n = user.shape[0]
        n_steps = -(-n // B)
        if n_steps == 0:
            return torch.empty(0, device=self.device)
        epoch = _lib.make_epoch(user, pos, neg, None, None, B)
        shards = [self._shard_struct(r) for r in self.local_ranks]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timing else None
        if ev:
            ev[0].record()
        for r, sh in zip(self.local_ranks, shards):
            self._plans[r] = _lib.shard_plan_build(sh, epoch, self.device, self._plans.get(r), self._plan_tmp)
        scales = self._step_scales(n_steps) if _scales is None else _scales
        b = self.binding
        optim = _lib.Optim(b.kind, 0, b.beta1, b.beta2, b.eps, scales.data_ptr())
        sums = torch.zeros((len(self.local_ranks), n_steps), dtype=torch.float32, device=self.device)
        if ev:
            ev[1].record()
            ev[2].record()
        self._ws = _lib.shard_train_steps(shards, epoch, optim, [self._plans[r] for r in self.local_ranks], 0, n_steps,
                                          self.sync_epoch, [sums[i] for i in range(len(shards))], self.status,
                                          self._ws, self.timeout_ms)
        if ev:
            ev[3].record()
            self.events = tuple(ev)
        self.sync_epoch += 2 * n_steps
        self.launches += 1 + len(self.local_ranks) * self.plan_launches()
        b.step0 += n_steps
        total = sums[0] if len(self.local_ranks) == 1 else sums.sum(0)
        if len(self.local_ranks) < self.world:
            dist.all_reduce(total, group=self.group)
        key = (n, B)
        if self._inv_counts is None or self._inv_counts[0] != key:  # 1 / samples per step, cached per epoch shape;
            last = 1.0 / (n - (n_steps - 1) * B)                    # built on the device: no copy that would wait
            c = torch.full((n_steps,), 1.0 / B, dtype=torch.float64, device=self.device)   # for the running kernel
            if n % B:
                c[-1:].fill_(last)                                  # (c[-1] = x would go through a host tensor)
            self._inv_counts = (key, c.to(torch.float32))
        if check:
            self.check_status()
        return total * self._inv_counts[1]

    def _step_scales(self, n_steps: int) -> torch.Tensor:
        """trs_optim.step_scale of the next ``n_steps`` steps on the device (python doubles, as torch computes them)."""
        scales = torch.tensor(step_scales(self.binding, n_steps), dtype=torch.float64).to(torch.float32)
        return scales.pin_memory().to(self.device, non_blocking=True)   # pinned: the copy does not wait for the stream

    def plan_launches(self) -> int:
        """CUDA kernels one trs_shard_plan_build launches for one rank (bench.py's gpu_launches)."""
        passes = lambda rows: max(1, -(-max(1, (max(rows, 2) - 1).bit_length()) // 8))
        # per id space: count + scatter + 2 per radix pass; then the item filter, the three flag kernels, the compaction;
        # one rank: the single item rows' flags and phase B's item pairs (count + scatter)
        return 2 * (2 + passes(-(-self.n_users // self.world)) + passes(-(-self.n_items // self.world))) + 5 + \
            2 * (self.world == 1)

    def check_status(self) -> None:
        if int(self.status.item()) != 0:
            raise RuntimeError("row-sharded training: a peer rank did not reach a step barrier within "
                               f"{self.timeout_ms} ms; the tables are in an undefined state")

    def gather_epoch(self, local: torch.Tensor) -> List[torch.Tensor]:
        """The loaders' exchange: ``local`` is THIS rank's [n_steps, k, B] int64 ids (k columns: user, positive, ...);
        returns the k columns of the GLOBAL epoch, int64 [n_steps * world * B], step-major and rank-major inside a
        step -- what ``train_epoch`` takes.  One NCCL all-gather; ids travel as int32 when every table has fewer
        than 2^31 rows (half the NVLink bytes) and are widened by the same pass that reorders them."""
        n_steps, k, B = local.shape
        W = self.world
        if len(self.local_ranks) == W:
            if W != 1:
                raise ValueError("gather_epoch with emulated ranks: stack the ranks' outputs yourself")
            return [local[:, j].reshape(-1) for j in range(k)]
        narrow = max(self.n_users, self.n_items) < 2 ** 31
        part = local.to(torch.int32) if narrow else local.contiguous()
        allr = torch.empty((W * n_steps, k, B), dtype=part.dtype, device=part.device)
        dist.all_gather_into_tensor(allr, part, group=self.group)
        cols = torch.empty((k, n_steps, W, B), dtype=torch.int64, device=part.device)
        cols.copy_(allr.view(W, n_steps, k, B).permute(2, 1, 0, 3))
        return [cols[j].view(-1) for j in range(k)]

    @staticmethod
    def host_chunks(n_steps: int, chunk_steps: Optional[int] = None) -> Tuple[int, List[int]]:
        """Chunk boundaries of a host-fed epoch: (largest chunk, [0, ..., n_steps]).  A short first chunk (its copy is
        the one nothing hides), then four times longer each time (copying a step's ids takes 10-20 % of the time the step
        takes to train) up to ``chunk_steps``: n/16, n/4, the rest for an epoch of up to ~3000 steps.  Few chunks: each
        costs 0.2 ms (one GPU) to ~1 ms (eight) of exchange / plan / launch ramp."""
        chunk_steps = int(chunk_steps or min(2048, max(64, -(-11 * n_steps // 16))))
        bounds, size = [0], max(8, min(chunk_steps, -(-n_steps // 16)))
        while bounds[-1] < n_steps:
            bounds.append(min(n_steps, bounds[-1] + size))
            size = min(chunk_steps, 4 * size)
        return chunk_steps, bounds

    def train_epoch_host(self, ids_host: torch.Tensor, draw_negatives: Callable[[torch.Tensor, int], torch.Tensor],
                         loss_host: Optional[torch.Tensor] = None, chunk_steps: Optional[int] = None) -> torch.Tensor:
        """A whole epoch straight from THIS rank's loader output in (pinned) host memory: ``ids_host`` is int64
        [n_steps, 2, B] (user, positive).  The epoch is cut into chunks of steps; chunk i+1 is copied to the device on a
        side stream (two device buffers) while chunk i trains, so the host-to-device copy leaves the critical path
        (chunks grow from a sixteenth of the epoch to ``chunk_steps`` steps: only the short first copy is exposed).
        Per chunk: id exchange (``gather_epoch``), ``draw_negatives(positives_global, first_global_sample)`` (device
        int64, e.g. the Philox kernel), plan, one persistent launch.  Per-step losses are also copied into ``loss_host``
        (pinned) if given.  No host synchronisation; call ``check_status()`` afterwards."""
        if self.bases is None:
            raise RuntimeError("torchrecsys_b200 has no CPU fallback: row-sharded training needs CUDA devices")
        if len(self.local_ranks) != 1:
            raise ValueError("train_epoch_host drives one rank per process")
        n_steps, k, B = ids_host.shape
        if n_steps == 0:
            return torch.empty(0, device=self.device)
        Bg = B * self.world
        chunk_steps, bounds = self.host_chunks(n_steps, chunk_steps)
        if self._h2d is None or tuple(self._h2d[0][0].shape) != (chunk_steps, k, B):
            self._h2d = ([torch.empty((chunk_steps, k, B), dtype=torch.int64, device=self.device) for _ in range(2)],
                         torch.cuda.Stream(self.device))
        bufs, side = self._h2d
        main = torch.cuda.current_stream(self.device)
        side.wait_stream(main)                    # the buffers may still feed the previous call's last chunks
        free = [None, None]                       # event: the chunk that last used the buffer has trained

        def stage(i):
            lo, hi = bounds[i], bounds[i + 1]
            buf = bufs[i % 2][:hi - lo]
            with torch.cuda.stream(side):
                if free[i % 2] is not None:
                    side.wait_event(free[i % 2])
                buf.copy_(ids_host[lo:hi], non_blocking=True)
                landed = torch.cuda.Event()
                landed.record(side)
            return buf, landed

        # every step's optimizer scalar up front: a pinned allocation inside the loop would wait for the running kernel
        scales = self._step_scales(n_steps)
        losses = []
        nxt = stage(0)
        for i in range(len(bounds) - 1):
            buf, landed = nxt
            if i + 2 < len(bounds):
                nxt = stage(i + 1)                # queued before this chunk's work: the copy engine starts right away
            main.wait_event(landed)
            cols = self.gather_epoch(buf)
            neg = draw_negatives(cols[1], bounds[i] * Bg)
            loss = self.train_epoch(cols[0], cols[1], neg, Bg, check=False, _scales=scales[bounds[i]:bounds[i + 1]])
            if loss_host is not None:
                loss_host[bounds[i]:bounds[i + 1]].copy_(loss, non_blocking=True)
            free[i % 2] = torch.cuda.Event()
            free[i % 2].record(main)
            losses.append(loss)
        return losses[0] if len(losses) == 1 else torch.cat(losses)

    def train_step(self, user: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor) -> torch.Tensor:
        """Convenience: THIS rank's samples of one step; the global batch is the all-gather over ranks (rank-major).
        Returns the global batch-mean hinge (device scalar)."""
        if len(self.local_ranks) < self.world:
            user, pos, neg = self.gather_epoch(torch.stack([user, pos, neg]).unsqueeze(0))
        return self.train_epoch(user, pos, neg, user.shape[0])[0]

    # ---- checkpoints: the reference's single-process layout (state_dict keys of collaborative/linear.py) --------
    _KEYS = (("user", "user.weight", "user_bias.weight"), ("item", "item.weight", "item_bias.weight"))

    def _gather(self, pieces: Dict[int, torch.Tensor], n: int) -> torch.Tensor:
        """Interleave per-rank shards [rows_q, C] into the full [n, C] table (row r = shard r % G, row r // G)."""
        G = self.world
        cols = next(iter(pieces.values())).shape[1]
        rows = -(-n // G)
        pad = lambda t: torch.cat([t, t.new_zeros((rows - t.shape[0], cols))]) if t.shape[0] < rows else t
        if len(self.local_ranks) == G:
            stack = [pad(pieces[q]) for q in range(G)]
        else:
            mine = pad(pieces[self.rank]).contiguous()
            stack = [torch.empty_like(mine) for _ in range(G)]
            dist.all_gather(stack, mine, group=self.group)
        return torch.stack(stack, 1).reshape(rows * G, cols)[:n].contiguous()

    def state_dict(self) -> Dict[str, torch.Tensor]:
        out = {}
        for name, wkey, bkey in self._KEYS:
            n = self.n_users if name == "user" else self.n_items
            out[wkey] = self._gather({r: self.tables[r][name][0] for r in self.local_ranks}, n)
            out[bkey] = self._gather({r: self.tables[r][name][1] for r in self.local_ranks}, n)
        return out

    def optimizer_state_dict(self) -> Dict[str, Dict[str, torch.Tensor]]:
        """{parameter key: {torch's state name: full tensor, "step": t}} -- torch.optim's per-parameter state."""
        out: Dict[str, Dict[str, torch.Tensor]] = {}
        for name, wkey, bkey in self._KEYS:
            n = self.n_users if name == "user" else self.n_items
            out[wkey], out[bkey] = {"step": self.binding.step0}, {"step": self.binding.step0}
            for i, sname in enumerate(_STATE_KEYS[self.kind]):
                out[wkey][sname] = self._gather({r: self.state[r][name][i][0] for r in self.local_ranks}, n)
                out[bkey][sname] = self._gather({r: self.state[r][name][i][1] for r in self.local_ranks}, n)
        return out

    def load_state_dict(self, params: Dict[str, torch.Tensor],
                        optimizer_state: Optional[Dict[str, Dict[str, torch.Tensor]]] = None) -> None:
        """Scatter full tables (a ``Linear``/``TorchRecSys.net`` state_dict, or ``state_dict()`` of another group
        size) onto the shards: every rank keeps rows rank::world."""
        G = self.world
        for name, wkey, bkey in self._KEYS:
            for r in self.local_ranks:
                emb, lin = self.tables[r][name]
                emb.copy_(params[wkey][r::G].to(self.device))
                lin.copy_(params[bkey][r::G].to(self.device).view(-1, 1))
                if optimizer_state is not None:
                    for i, sname in enumerate(_STATE_KEYS[self.kind]):
                        self.state[r][name][i][0].copy_(optimizer_state[wkey][sname][r::G].to(self.device))
                        self.state[r][name][i][1].copy_(optimizer_state[bkey][sname][r::G].to(self.device).view(-1, 1))
        if optimizer_state is not None:
            self.binding.step0 = int(optimizer_state["user.weight"].get("step", 0))
        self._state_version += 1
        if len(self.local_ranks) < G:
            if self.device.type == "cuda":
                torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)  # peers read these rows: nobody trains before everyone has loaded

    # ---- serving on the shards: lookup / eval_pairwise / evaluate / predict_topk, nothing gathered ------------------
    # Ordering rule.  In a real group a rank must not train while another rank still reads its rows.
    #  * Reads after training are safe: every training launch ends waiting for every rank's last arrival (csrc/shard.cu,
    #    the cross_wait after the step loop), and load_state_dict ends with a barrier.
    #  * Reads before the next training: each method below that launches a peer-reading kernel ends with a group
    #    collective on this rank's stream before it returns -- eval_pairwise the all-gather, recommend / predict_topk
    #    the all_to_all merger's all-gather, lookup a one-element all-reduce.  This rank's next training kernel is
    #    queued behind that collective, and the collective cannot complete before every rank's reads have finished: no
    #    host synchronisation is needed.
    # In a real group these methods are collective: every rank calls them with the same arguments.
    TOPK_MAX_FACTORS = 239   # predict_batch's kernel path (csrc/topk.cu: check_topk); k in 1..128 likewise

    def _require_cuda(self) -> None:
        if self.bases is None:
            raise RuntimeError("torchrecsys_b200 has no CPU fallback: the row-sharded tables need CUDA devices")

    def _device_ids(self, ids, n: int, what: str) -> torch.Tensor:
        """int64 ids on this device; IndexError outside [0, n), as TorchRecSys raises."""
        ids = torch.as_tensor(ids, dtype=torch.int64).reshape(-1)
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= n):
            raise IndexError(f"{what} ids must lie in [0, {n})")
        return ids.to(self.device).contiguous()

    def lookup(self, name: str, ids) -> Tuple[torch.Tensor, torch.Tensor]:
        """Rows of global ``ids`` of the ``"user"`` or ``"item"`` table and their biases, (emb [n, D], bias [n, 1]),
        copied from their owners bit for bit."""
        self._require_cuda()
        if name not in ("user", "item"):
            raise ValueError(f"table must be 'user' or 'item', got {name!r}")
        ids = self._device_ids(ids, self.n_users if name == "user" else self.n_items, name)
        out = self._lib.shard_gather_rows(self._shard_struct(self.local_ranks[0]), int(name == "item"), ids, self.device)
        if len(self.local_ranks) < self.world:
            dist.all_reduce(torch.zeros(1, device=self.device), group=self.group)   # the ordering rule above
        return out

    def eval_pairwise(self, user: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, batch_size: int = 512,
                      want_scores: bool = False):
        """``_lib.eval_pairwise`` on the shards -> (loss [nb], auc [nb], pos scores, neg scores; None unless
        ``want_scores``), bit-identical to it on the gathered model.  user / pos / neg: the GLOBAL test epoch (int64
        device tensors, identical on every rank).  Rank q evaluates the whole batches [q P, (q + 1) P), P = ceil(nb / W):
        a batch is never divided between ranks, so its mean hinge keeps its association."""
        self._require_cuda()
        _lib, W, B = self._lib, self.world, int(batch_size)
        n = user.shape[0]
        nb = -(-n // B)
        P = -(-nb // W)
        L = len(self.local_ranks)
        # [rank, (loss, auc), batch] and [rank, (pos, neg), sample], each rank's block at its batch range
        stats = torch.empty((L, 2, P), dtype=torch.float32, device=self.device)
        scores = torch.empty((L, 2, P * B), dtype=torch.float32, device=self.device) if want_scores else None
        if nb:
            epoch = _lib.make_epoch(user, pos, neg, None, None, B)
            for i, r in enumerate(self.local_ranks):
                lo = min(r * P, nb)
                _lib.shard_eval_pairwise(self._shard_struct(r), epoch, lo, min(nb, lo + P) - lo, stats[i, 0], stats[i, 1],
                                         *((scores[i, 0], scores[i, 1]) if want_scores else ()))
            if L < W:   # every rank takes part, also one whose range is empty (the ordering rule above)
                parts = [stats] + ([scores] if want_scores else [])
                full = [torch.empty((W,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device) for t in parts]
                for f, t in zip(full, parts):
                    dist.all_gather_into_tensor(f, t, group=self.group)
                stats, scores = full[0], (full[1] if want_scores else None)
        # fresh tensors, as _lib.eval_pairwise returns: a torch reduction's association follows its input's alignment
        loss, auc = (stats[:, j].reshape(-1)[:nb].clone() for j in (0, 1))
        if not want_scores:
            return loss, auc, None, None
        return loss, auc, scores[:, 0].reshape(-1)[:n].clone(), scores[:, 1].reshape(-1)[:n].clone()

    def evaluate(self, user: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, batch_size: int = 512,
                 eval_metrics=("loss", "auc")) -> Dict[str, float]:
        """``TorchRecSys.evaluate``'s metrics on the shards, returned rather than printed: ``loss`` / ``auc`` the mean
        over batches of ``eval_pairwise``, ``roc_auc`` the sort-based ROC-AUC of the whole split, 0 for an unknown name.
        ``neg`` is the caller's negatives (e.g. those ``TorchRecSys._with_negatives`` draws)."""
        from .model import TorchRecSys
        loss, auc, ps, ns = self.eval_pairwise(user, pos, neg, batch_size, want_scores="roc_auc" in eval_metrics)
        results, out = {"loss": loss, "auc": auc}, {}
        for metric in eval_metrics:
            if metric in results:
                out[metric] = float(results[metric].mean().item())
            elif metric == "roc_auc":
                out[metric] = TorchRecSys._roc_auc(ps, ns)
            else:
                out[metric] = 0
        return out

    def predict_topk(self, users, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k items of each user against the whole catalogue -> (idx int64 [Q, min(k, n_items)], score fp32), on the
        device and the same on every rank; equal to ``_lib.predict_topk`` / ``TorchRecSys.predict_batch`` on the gathered
        model (best first, ties towards the lower item id).  ``recommend(users, k)`` under predict_batch's limits:
        1 <= k <= 128 and n_factors <= 239, which keep every shard on the tensor-core top-k."""
        self._require_cuda()
        if not 1 <= int(k) <= 128:
            raise ValueError(f"top_k must be in 1..128 on the row-sharded tables (got {k})")
        if self.dim > self.TOPK_MAX_FACTORS:
            raise ValueError(f"predict_topk on the row-sharded tables needs n_factors <= {self.TOPK_MAX_FACTORS}")
        return self.recommend(users, k)   # raises IndexError for bad ids

    RECOMMEND_MAX_K = 1024   # trs_shard_topk_exact

    EXACT_CHUNK = 32768   # query users per trs_shard_topk_exact call: its workspace stays <= ~0.5 GB at k = 1024

    def _exact_topk(self, r: int, u_emb, u_lin, k: int, excl_ptr=None, excl_ids=None):
        """trs_shard_topk_exact on local rank r's item shard -> (global idx [Q, k], score [Q, k]), in chunks of
        EXACT_CHUNK query users; the workspace lives for this call only."""
        sh, u_lin, Q = self._shard_struct(r), u_lin.reshape(-1), u_emb.shape[0]
        if Q <= self.EXACT_CHUNK:
            return self._lib.shard_topk_exact(sh, u_emb, u_lin, k, excl_ptr, excl_ids)[:2]
        idx = torch.empty((Q, k), dtype=torch.int64, device=self.device)
        score = torch.empty((Q, k), dtype=torch.float32, device=self.device)
        ws = None
        for lo in range(0, Q, self.EXACT_CHUNK):
            hi = min(Q, lo + self.EXACT_CHUNK)
            ptr = ids = None
            if excl_ptr is not None:   # the chunk's rows of the CSR, re-based
                ptr = (excl_ptr[lo:hi + 1] - excl_ptr[lo]).contiguous()
                ids = excl_ids[int(excl_ptr[lo]):int(excl_ptr[hi])].contiguous()
            i, s, ws = self._lib.shard_topk_exact(sh, u_emb[lo:hi], u_lin[lo:hi], k, ptr, ids, ws)
            idx[lo:hi], score[lo:hi] = i, s
        return idx, score

    def _exclusion_csr(self, r: int, users: torch.Tensor, ex_user: torch.Tensor, ex_item: torch.Tensor):
        """(row pointers [Q + 1], sorted unique local item ids) of rank r's excluded items per query position, and the
        most any query position has."""
        W = self.world
        on = ex_item % W == r
        rows = max(shard_rows(self.n_items, r, W), 1)
        key = torch.unique(ex_user[on] * rows + ex_item[on] // W)   # sorted: by user, then local id
        pair_user, pair_local = key // rows, key % rows
        start = torch.searchsorted(pair_user, users, right=False)
        count = torch.searchsorted(pair_user, users, right=True) - start
        ptr = torch.zeros(users.numel() + 1, dtype=torch.int64, device=self.device)
        torch.cumsum(count, 0, out=ptr[1:])
        total = int(ptr[-1])
        most = int(count.max()) if count.numel() else 0
        within = torch.arange(total, device=self.device) - torch.repeat_interleave(ptr[:-1], count, output_size=total)
        ids = pair_local[torch.repeat_interleave(start, count, output_size=total) + within]
        return ptr, ids.contiguous(), most

    def recommend(self, users, k: int, exclude=None, _force_exact: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k items of each user against the whole catalogue, leaving out ``exclude = (user_ids, item_ids)`` pairs
        (any order, duplicates allowed, pairs of users not queried ignored) -> (idx int64 [Q, min(k, n_items)], score
        fp32), on the device and the same on every rank, best first, ties towards the lower item id; rows with fewer
        than k remaining items end in -1 / -inf.  Scores equal ``trs_scores`` on the gathered model bit for bit.
        1 <= k <= 1024, any n_factors.  Each rank ranks its own item shard: with the tensor-core top-k
        (``predict_topk``'s) when n_factors <= 239 and k plus the most items one query user has excluded on the shard
        is <= 128 -- it over-requests that many and drops the excluded ones -- else with the exact fp32 kernel."""
        self._require_cuda()
        if not 1 <= int(k) <= self.RECOMMEND_MAX_K:
            raise ValueError(f"k must be in 1..{self.RECOMMEND_MAX_K} for recommend on the row-sharded tables (got {k})")
        _lib, W, k = self._lib, self.world, int(k)
        users = self._device_ids(users, self.n_users, "user")
        if exclude is not None:
            ex_user, ex_item = exclude
            ex_user, ex_item = (t.reshape(-1) if torch.is_tensor(t) else torch.as_tensor(np.asarray(t)).reshape(-1)
                                for t in (ex_user, ex_item))
            if ex_user.numel() != ex_item.numel():
                raise ValueError(f"exclude needs as many user ids as item ids (got {ex_user.numel()} and "
                                 f"{ex_item.numel()})")
            ex_user = self._device_ids(ex_user, self.n_users, "exclude user")
            ex_item = self._device_ids(ex_item, self.n_items, "exclude item")
        Q, kk = users.numel(), min(k, self.n_items)
        self.last_predict_overflow = 0
        if Q == 0:
            return (torch.empty((0, kk), dtype=torch.int64, device=self.device),
                    torch.empty((0, kk), dtype=torch.float32, device=self.device))
        u_emb, u_lin = _lib.shard_gather_rows(self._shard_struct(self.local_ranks[0]), 0, users, self.device)
        queries = torch.arange(Q, device=self.device)
        key = (self.sync_epoch, self._state_version)   # unchanged tables: the prepared item operand is reused

        def local_topk(r: int):
            """(global idx, score) [Q, k] of rank r's item shard with its excluded items left out, -1 / -inf padded."""
            ptr, ids, most = (self._exclusion_csr(r, users, ex_user, ex_item) if exclude is not None
                              else (None, None, 0))
            rows = shard_rows(self.n_items, r, W)
            exact = _force_exact or rows == 0 or self.dim > self.TOPK_MAX_FACTORS or k + most > 128
            self.last_recommend_paths[r] = "exact" if exact else "tensor core"
            if exact:
                return self._exact_topk(r, u_emb, u_lin, k, ptr, ids)
            emb, lin = self.tables[r]["item"]
            model = _lib.make_model(_lib.NET_LINEAR, self.dim, _lib.make_table(u_emb, lin=u_lin),
                                    _lib.make_table(emb, lin=lin), [])
            kq = k + most
            idx, score, over = _lib.predict_topk(model, queries, kq,
                                                 cache=self._topk_caches.setdefault(r, _lib.TopkCache()), cache_key=key)
            over = torch.nonzero(over).flatten()
            if over.numel():   # candidate set did not fit: rank those users exactly
                idx[over], score[over] = self._exact_topk(r, u_emb[over], u_lin[over], kq)
                idx[over] = torch.where(idx[over] >= 0, idx[over] // W, idx[over])   # back to local ids
                self.last_predict_overflow += over.numel()
            if ptr is not None:   # drops the excluded
                idx, score = _lib.topk_merge_sorted(score[None], idx[None], k, ptr, ids)
            # local order is global order within a shard: (score desc, local id asc) merges as (score desc, global id asc)
            return torch.where(idx >= 0, idx * W + r, idx), score

        if len(self.local_ranks) == W:
            lists = [local_topk(r) for r in self.local_ranks]
            idx, score = lists[0] if W == 1 else merge_topk_lists(torch.stack([s for _, s in lists]),
                                                                  torch.stack([i for i, _ in lists]), k)
        else:   # the all_to_all merger; its all_gather is the closing collective (the ordering rule above)
            idx, score = sharded_predict_topk(lambda u, kq, offset: local_topk(self.rank), users, k, self.n_items,
                                              self.group)
        return idx[:, :kk].contiguous(), score[:, :kk].contiguous()

    # ---- the bridge to TorchRecSys(net_type='linear'): shard a model + its torch optimizer, and hand them back ------
    @classmethod
    def from_model(cls, net: torch.nn.Module, optimizer: torch.optim.Optimizer, global_batch: int, device=None,
                   group=None, emulate_world: Optional[int] = None, timeout_ms: int = 20000) -> "ShardedLinearTrainer":
        """``net`` is a ``Linear`` scorer without metadata (``TorchRecSys(...).net``), ``optimizer`` the torch optimizer
        bound to its parameters (SparseAdam / Adam, Adagrad, plain SGD -- the ones with a row-wise kernel, read the way
        ``engine.bind_optimizer`` reads them).  Tables, optimizer state and step count move onto the shards; training
        continues exactly where ``fit`` would (same update arithmetic: tested bit-for-bit against the fused kernel)."""
        sd = {k: v.detach() for k, v in net.state_dict().items()}
        extra = set(sd) - {"user.weight", "item.weight", "user_bias.weight", "item_bias.weight"}
        if extra or getattr(net, "use_metadata", False):
            raise ValueError(f"row-sharded training covers the Linear scorer without metadata (got {sorted(extra)})")
        name = type(optimizer).__name__
        g = optimizer.param_groups[0]
        if any(any(pg.get(k) != g.get(k) for k in ("lr", "betas", "eps", "lr_decay")) for pg in optimizer.param_groups):
            raise NotImplementedError("the row-wise update needs identical hyper-parameters in every param group")
        if name in ("SparseAdam", "Adam"):
            if g.get("weight_decay") or g.get("amsgrad") or g.get("maximize"):
                raise NotImplementedError(f"{name}: weight_decay / amsgrad / maximize are not supported on sparse tables")
            kw = dict(optimizer="sparse_adam", lr=g["lr"], betas=tuple(g["betas"]), eps=g["eps"])
        elif name == "Adagrad":
            if g.get("weight_decay") or g.get("maximize"):
                raise NotImplementedError("Adagrad: weight_decay is not compatible with sparse gradients (as in torch)")
            kw = dict(optimizer="adagrad", lr=g["lr"], eps=g["eps"], lr_decay=g.get("lr_decay", 0.0))
        elif name == "SGD":
            if g.get("momentum") or g.get("weight_decay") or g.get("nesterov") or g.get("maximize"):
                raise NotImplementedError("SGD: momentum / weight_decay / nesterov are not row-sparse")
            kw = dict(optimizer="sgd", lr=g["lr"])
        else:
            raise NotImplementedError(f"optimizer {name} has no row-wise update; use SparseAdam, Adagrad or plain SGD")
        n_users, dim = sd["user.weight"].shape
        tr = cls(n_users, sd["item.weight"].shape[0], dim, global_batch, device=device, group=group,
                 emulate_world=emulate_world, timeout_ms=timeout_ms, **kw)
        state = None
        named = dict(net.named_parameters())
        if all(len(optimizer.state.get(named[k], {})) for k in sd) and _STATE_KEYS[tr.kind]:
            state = {}
            for k in sd:
                st = optimizer.state[named[k]]
                step = st.get("step", 0)
                state[k] = {"step": int(step.item()) if torch.is_tensor(step) else int(step)}
                for sname in _STATE_KEYS[tr.kind]:
                    state[k][sname] = st[sname].detach()
        tr.load_state_dict(sd, state)
        return tr

    def to_model(self, net: torch.nn.Module, optimizer: Optional[torch.optim.Optimizer] = None) -> None:
        """Gather the shards back into ``net`` (and the optimizer's per-parameter state into ``optimizer``, in torch's own
        names and step convention) -- for ``evaluate`` / ``predict`` / ``torch.save`` on one device.  Collective: every
        rank of the group calls it and ends up with the full model."""
        sd = self.state_dict()
        with torch.no_grad():
            for k, p in net.named_parameters():
                p.copy_(sd[k].to(p.device))
        if hasattr(net, "_trs_version"):
            net._trs_version += 1
        if optimizer is None or not _STATE_KEYS[self.kind]:
            return
        osd = self.optimizer_state_dict()
        tensor_step = type(optimizer).__name__ != "SparseAdam"     # torch keeps an int there for SparseAdam only
        for k, p in net.named_parameters():
            st = optimizer.state[p]
            st["step"] = torch.tensor(float(self.binding.step0)) if tensor_step else int(self.binding.step0)
            for sname in _STATE_KEYS[self.kind]:
                st[sname] = osd[k][sname].to(p.device).view_as(p).clone()

    def gather_full(self, name: str) -> Tuple[torch.Tensor, torch.Tensor]:
        sd = self.state_dict()
        return sd[f"{name}.weight"], sd[f"{name}_bias.weight"]


# ------------------------------------------------------------------------------------------------------
# item-sharded predict
# ------------------------------------------------------------------------------------------------------
def item_block(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous item block [lo, hi) of a rank."""
    per = (n_items + world - 1) // world
    return min(rank * per, n_items), min((rank + 1) * per, n_items)


def merge_topk_lists(scores: torch.Tensor, idx: torch.Tensor, k: int, merge: Optional[Callable] = None):
    """scores / idx [G, Q, k_in], each row sorted by (score desc, id asc) with idx < 0 padding at the end -> (idx [Q, k],
    score [Q, k]) in the same order, -1 / -inf padded.  ``merge`` replaces trs_shard_topk_merge_sorted (CPU tests)."""
    if merge is not None:
        return merge(scores, idx, k)
    from . import _lib
    return _lib.topk_merge_sorted(scores.contiguous(), idx.contiguous(), k)


def sharded_predict_topk(local_topk: Callable, users: torch.Tensor, k: int, n_items: int, group=None,
                         merge: Optional[Callable] = None):
    """``local_topk(users, k, item_offset) -> (idx [Q, k] global ids, score [Q, k])`` on this rank's item block, each
    row sorted by (score desc, id asc) and -1 / -inf padded, as trs_predict_topk writes it; returns the merged global
    top-k on every rank.

    The per-rank candidate lists are exchanged with an all_to_all that sends each user's candidates to ONE merger rank
    (users split evenly over the ranks): every rank merges Q / G users x G lists instead of all Q users -- G times less
    merge work and traffic than all-gathering the lists -- and the merged [Q / G, k] results are all-gathered."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, _ = item_block(n_items, rank, world)
    idx, score = local_topk(users, k, lo)
    Q = idx.shape[0]
    if world == 1:   # one sorted list is its own merge
        return idx, score
    Qc = -(-Q // world)                                   # users per merger rank
    pad = Qc * world - Q
    if pad:
        idx = torch.cat([idx, idx.new_full((pad, k), -1)])
        score = torch.cat([score, score.new_full((pad, k), float("-inf"))])
    got_idx, got_score = torch.empty_like(idx), torch.empty_like(score)   # [world, Qc, k]: every rank's list for MY users
    dist.all_to_all_single(got_idx, idx.contiguous(), group=group)
    dist.all_to_all_single(got_score, score.contiguous(), group=group)
    m_idx, m_score = merge_topk_lists(got_score.view(world, Qc, k), got_idx.view(world, Qc, k), k, merge)
    out_idx = torch.empty((world * Qc, k), dtype=m_idx.dtype, device=m_idx.device)
    out_score = torch.empty((world * Qc, k), dtype=m_score.dtype, device=m_score.device)
    dist.all_gather_into_tensor(out_idx, m_idx.contiguous(), group=group)
    dist.all_gather_into_tensor(out_score, m_score.contiguous(), group=group)
    return out_idx[:Q], out_score[:Q]
