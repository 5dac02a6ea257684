#!/usr/bin/env python
"""bench.py -- headline benchmark of the TorchRecSys hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference|torch_cuda] [--workload NAME]

A "step" is one training step of the named workload: forward x2 + hinge + backward + sparse optimizer update
over one batch (reference model.py:274-284).

Default workload ("c4") = BASELINE.json configs[3], the large-table config north_star scales: Linear 50M users x
5M items, dim 128, SparseAdam, batch 16384 PER GPU (weak scaling: the global batch is 16384 * N), through the
ROW-SHARDED persistent kernel (csrc/shard.cu) at every N:
  N = 1   a group of one rank: the whole tables (84.5 GB with optimizer state) on one GPU.
  N > 1   (under torchrun, one rank per GPU) row r lives on rank r % N; every rank maps its peers' shards (CUDA
          IPC) and one persistent kernel per rank reads item rows from / stores gradient rows into the owners'
          HBM over NVLink.  NCCL carries the per-epoch id all-gather and the loss all-reduce; nothing per step.
The other BASELINE configs ride along in the same JSON line under "other_workloads" (N = 1: C2 FM, C3 MLP, C5
predict, and the SAME C4 tables through fit()'s fused single-GPU kernel, csrc/train.cu; N > 1: item-sharded C5
predict).  `--workload c2_fm`,
`c3_mlp`, `c5_predict`, `c1_linear`, `c4_fused`, `c4_linear` select one of them as the headline instead.

  value      whole-job samples/s, every input already resident in HBM, CUDA events, max over ranks.  The timed
             region is exactly K steps, one epoch (one persistent launch unless K x global batch exceeds
             SAMPLE_CAP), and contains EVERYTHING a step needs: (N > 1: the id all-gather,) Philox negatives, the
             sort plan (coalesce's sort) and the persistent kernel.  The epoch's fixed cost (plan build, launch:
             about 0.5 ms on one B200 at 1000 W) is spread over K steps, so the rate of a long epoch wants K in
             the thousands.  (The fused single-GPU workloads repeat their K-step block `config.repeats` times so
             that the region lasts >= --min-ms.)
  --dump-outputs DIR  writes what the K timed steps computed as DIR/<name>.npy: the per-step losses and the user /
             item rows their last step updated (a seeded sample of at most 8192 per table).  The inputs are
             seeded, so two builds run with the same arguments can be compared array for array.
  e2e        the same blocks with the ids starting in pinned HOST memory (H2D inside the timed region) and the
             per-step losses read back to the host (D2H inside).
  roofline   the persistent kernel alone: algorithmic HBM bytes (SURVEY.md §8d: ids + each unique touched row's
             param+state read once and written once) / its CUDA-event duration, against the measured HBM peak of
             MEASURED_PEAKS.json; N > 1 adds the NVLink figure (bytes that must cross / 770 GB/s per direction).
  cpu_baseline  the reference's CPU op stream (oracle/torch_port.py, kind "port": /root/reference is not on the
             GPU box) on a bounded sample of the same workload on the host cores (N = 1 only).

--impl reference runs only that CPU arm and prints it as the main line.  --impl torch_cuda (secondary baseline,
SURVEY.md §2.1) runs the same port with its tables on the GPU: the stock ATen CUDA kernels the reference's
use_cuda=True path would launch.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: net, users, items, dim, n_categories (0 = no metadata), batch, optimizer, dynamic negs
    "c2_fm": dict(net="fm", n_users=1_000_000, n_items=200_000, dim=64, n_cat=100, batch=8192,
                  opt="sparse_adam", lr=1e-3, desc="BASELINE configs[1]: FM + product_category(100), "
                  "dynamic negatives, 1M users x 200k items, dim 64, batch 8192, SparseAdam"),
    "c1_linear": dict(net="linear", n_users=3000, n_items=1000, dim=80, n_cat=0, batch=1024,
                      opt="sparse_adam", lr=1e-3, desc="BASELINE configs[0] shape: linear 3k x 1k, dim 80, batch 1024"),
    "c3_mlp": dict(net="mlp", n_users=1_000_000, n_items=200_000, dim=64, n_cat=0, batch=16384, opt="adagrad",
                   lr=1e-2, hidden=[512, 256, 128], desc="BASELINE configs[2]: MLP [512,256,128] + batch norm, bf16 "
                   "tensor-core GEMMs, 1M users x 200k items, dim 64, batch 16384, Adagrad"),
    "c5_predict": dict(net="linear", n_users=1_000_000, n_items=5_000_000, dim=128, n_cat=0, batch=148 * 128, k=100,
                       opt=None, lr=0.0, predict=True, desc="BASELINE configs[4]: batched predict top-100 against a "
                       "5M-item table (linear scorer, dim 128); a step = 18944 users (148 user tiles)"),
    "c4_fused": dict(net="linear", n_users=50_000_000, n_items=5_000_000, dim=128, n_cat=0, batch=16384,
                     opt="sparse_adam", lr=1e-3,
                     desc="BASELINE configs[3]: linear 50M x 5M, dim 128, batch 16384/GPU, SparseAdam"),
    "c4_linear": dict(net="linear", n_users=50_000_000, n_items=5_000_000, dim=128, n_cat=0, batch=16384,
                      opt="sparse_adam", lr=1e-3, sharded=True,
                      desc="BASELINE configs[3]: linear 50M x 5M, dim 128, batch 16384/GPU, SparseAdam"),
}
C4_DESC = "BASELINE configs[3]: linear 50M x 5M, dim 128, batch 16384/GPU, SparseAdam"
NVLINK_GBS = 770.0  # measured peer copy per direction on this pool (B200_PROFILING.md); 900 nominal


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_cuda"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS) + ["c4"])
    ap.add_argument("--users", type=int, default=0, help="override the workload's user count (memory-bound hosts)")
    ap.add_argument("--items", type=int, default=0, help="override the workload's item count")
    ap.add_argument("--batch", type=int, default=0, help="override the workload's batch size (per GPU)")
    ap.add_argument("--dim", type=int, default=0, help="override the workload's n_factors")
    ap.add_argument("--zipf", type=float, default=0.0, help="draw training ids from Zipf(A), A > 1, instead of uniformly")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the CPU baseline sample")
    ap.add_argument("--min-ms", type=float, default=100.0,
                    help="fused single-GPU workloads: the K-step block is repeated until the timed region lasts this long")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the other_workloads sub-results")
    ap.add_argument("--shard-it", type=int, default=0, help="tuning: 16-byte chunks per lane of the sharded kernel (1 or 2)")
    ap.add_argument("--shard-remote-hint", type=int, default=None, help="tuning: L2 policy on stores into peer memory (1) or local only (0)")
    ap.add_argument("--shard-overlap", type=int, default=None, help="tuning: force the early first pass of phase A on (1) / off (0)")
    ap.add_argument("--emulate-world", type=int, default=0,
                    help="c4_linear on ONE GPU: host a group of this many ranks in one launch (structure check, no NVLink)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="c4 / c4_linear: after the timed steps, write what they computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload not in ("c4", "c4_linear") or args.impl != "b200"):
        ap.error("--dump-outputs covers the row-sharded workload (c4, c4_linear), whose timed steps are exactly --steps")
    return args


# ------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md §8d): uniform ids, rng seed 1234, category(item) = item mod n_cat
# ------------------------------------------------------------------------------------------------
def synth_ids(wl, n, seed=1234):
    """Uniform i.i.d. ids (SURVEY.md §8d), or with --zipf A: rank-frequency Zipf(A) ids (hot rows, many duplicates)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    a = wl.get("zipf", 0.0)
    if a > 1.0:
        user = ((rng.zipf(a, n) - 1) % wl["n_users"]).astype(np.int64)
        pos = ((rng.zipf(a, n) - 1) % wl["n_items"]).astype(np.int64)
        return user, pos
    user = rng.integers(0, wl["n_users"], n, dtype=np.int64)
    pos = rng.integers(0, wl["n_items"], n, dtype=np.int64)
    return user, pos


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------
# baseline arms: the reference's op stream on the host cores (or, --impl torch_cuda, on the GPU)
# ------------------------------------------------------------------------------------------------
def port_reference(wl, steps, warmup, budget_s, device="cpu"):
    """Times oracle/torch_port.py (the ATen ops of the reference's scorer + hinge + torch optimizer) on a bounded
    sample: `steps` steps of the workload's batch size.  CPU: thread count swept, best kept."""
    import numpy as np
    import torch
    from oracle import cf_oracle as O
    from oracle import torch_port as TP
    B = wl["batch"]
    cap_note = ""
    if device == "cpu" and wl["n_users"] > 5_000_000:  # host RAM: 50M x 128 fp32 + SparseAdam state would be 77 GB
        wl = dict(wl, n_users=5_000_000)
        cap_note = " (user table cut to 5M rows on the host: 25.6 GB + optimizer state does not fit; row access stays random)"
    n = (steps + warmup) * B
    user, pos = synth_ids(wl, n)
    neg = O.philox_negatives(1234, 0, pos, wl["n_items"])
    dev = torch.device(device)
    ids = {k: torch.from_numpy(v).to(dev) for k, v in (("user", user), ("pos", pos), ("neg", neg))}
    batch_of = lambda s: {k: v[s * B:(s + 1) * B] for k, v in ids.items()}
    metas = [wl["n_cat"]] if wl["n_cat"] else []
    ncores = len(os.sched_getaffinity(0))
    threads = sorted({1, 2, 4, 8, 16, 32, ncores} & set(range(1, ncores + 1))) if device == "cpu" else [ncores]
    torch.manual_seed(1234)
    kw = dict(hidden=wl["hidden"], batch_norm=True) if wl["net"] == "mlp" else {}
    net = TP.make_net(wl["net"], wl["n_users"], wl["n_items"], metas, wl["dim"], **kw).to(dev)
    net.train()
    opt = TP.make_optimizer(wl["opt"], net, wl["lr"])

    def run(s):
        b = batch_of(s)
        if metas:
            b["pos_meta"] = (b["pos"] % wl["n_cat"]).view(-1, 1)
            b["neg_meta"] = (b["neg"] % wl["n_cat"]).view(-1, 1)
        return TP.train_step(net, opt, b)

    sync = torch.cuda.synchronize if device != "cpu" else (lambda: None)
    best, tried = None, {}
    t_start = time.time()
    for nt in threads:
        if time.time() - t_start > budget_s and best is not None:
            break
        if device == "cpu":
            torch.set_num_threads(nt)
        for s in range(warmup):
            run(s)
        sync()
        t0 = time.perf_counter()
        done = 0
        for s in range(warmup, warmup + steps):
            run(s)
            done += 1
            if time.perf_counter() - t0 > budget_s / max(len(threads), 1) and done >= 2:
                break
        sync()
        dt = time.perf_counter() - t0
        tried[nt] = done * B / dt
        if best is None or tried[nt] > best[0]:
            best = (tried[nt], nt, done, dt)
    value, nt, done, dt = best
    where = (f"torch {torch.__version__} CPU, threads swept { {k: round(v) for k, v in tried.items()} } on {ncores} "
             "cores, best kept") if device == "cpu" else \
        f"torch {torch.__version__} stock ATen CUDA kernels on {torch.cuda.get_device_name(0)} (per-step loss.item() as the reference)"
    return {"value": value, "unit": "samples/s", "cores": nt, "kind": "port",
            "sample": f"{done} steps of batch {B} ({done * B} samples) of the same workload after "
                      f"{warmup} warm-up steps, {where}" + cap_note,
            "ms_per_step": dt / done * 1e3, "steps": done}


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (NVML, ~2 ms period)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            # NVML queries take a driver lock: dense at first (short timed regions still get a few samples), sparse
            # afterwards (a long region with many launches is not disturbed)
            time.sleep(0.002 if len(self.samples) < 6 else 0.01)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s), "sm_mhz_min": s[0] if s else None}


def clock_ramp(dev, seconds=0.3):
    """Not steps: keep the GPU busy so the timed region does not start at idle clocks."""
    import torch
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    t0 = time.time()
    while time.time() - t0 < seconds:
        scratch.copy_(scratch.flip(0))
        torch.cuda.synchronize()
    del scratch


def pick_repeats(probe_ms, min_ms, world, dev):
    """How often the K-step block runs inside a timed region so that it lasts >= min_ms (same on every rank)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([probe_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return int(max(1, min(200, math.ceil(min_ms / max(float(t.item()), 1e-3)))))


SAMPLE_CAP = 1 << 26  # samples (over all ranks) of one timed launch: bounds the id / plan buffers


def split_repeats(R, samples_per_block):
    """The K-step block is replayed R times; r_in replays go into ONE epoch (one plan build, one persistent launch --
    what a real epoch of thousands of steps looks like), as many as the sample cap allows; the rest as further
    launches.  Returns (replays per launch, launches)."""
    r_in = max(1, min(R, SAMPLE_CAP // max(samples_per_block, 1)))
    return r_in, -(-R // r_in)


def traffic_of(workload, K):
    """dram bytes of the dominant kernel per launch, from the committed ncu --set full capture (STATIC: it is not
    measured by this run; profiles/traffic.json holds bytes per step, one launch = K steps)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return None, None
    v = t.get(workload)
    return (v * K if v else None), t.get("_source", "profiles/traffic.json")


# ------------------------------------------------------------------------------------------------
# single-GPU training through the fused persistent kernel (and N independent replicas of it)
# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(wl, user, pos, neg, n_steps, B, S):
    """SURVEY.md §8d: 8 B per id consumed + per unique touched row (param + S state tensors) read once
    and written once, embedding row (dim floats) and its width-1 companion.  From the actual batches."""
    import torch
    D, F = wl["dim"], 1 if wl["n_cat"] else 0
    row_bytes = 4 * (D + (0 if wl["net"] == "mlp" else 1)) * (2 + 2 * S)  # MLP tables have no width-1 companion
    total = 0
    for s in range(n_steps):
        sl = slice(s * B, (s + 1) * B)
        uu = torch.unique(user[sl]).numel()
        items = torch.cat([pos[sl], neg[sl]])
        ui = torch.unique(items).numel()
        um = torch.unique(items % wl["n_cat"]).numel() if F else 0
        meta_row = row_bytes if wl["net"] == "fm" else 4 * D * (2 + 2 * S)
        total += 8 * (3 * B + 2 * B * F) + (uu + ui) * row_bytes + um * meta_row
    return total


def gpu_bench(args, wl, name):
    import torch
    import torch.distributed as dist
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.collaborative.fm import FM
    from torchrecsys_b200.collaborative.linear import Linear
    from torchrecsys_b200.collaborative.mlp import MLP
    from torchrecsys_b200.engine import EpochRunner, MlpEpochRunner, advance_steps, step_scales

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    K, W, B = args.steps, max(args.warmup, 3), wl["batch"]
    F = 1 if wl["n_cat"] else 0

    torch.manual_seed(1234 + rank)
    is_mlp = wl["net"] == "mlp"
    if is_mlp:
        net = MLP(wl["n_users"], wl["n_items"], {}, wl["dim"], use_metadata=False, use_batch_norm=True,
                  hidden_layers=wl["hidden"], use_cuda=True).to(dev).train()
    else:
        cls = FM if wl["net"] == "fm" else Linear
        with torch.device(dev):  # the big tables are created on the device (50M x 128 does not visit the host)
            net = cls(wl["n_users"], wl["n_items"], {"product_category": wl["n_cat"]} if F else {}, wl["dim"],
                      use_metadata=bool(F), use_cuda=True)
        net = net.to(dev)
    if wl["opt"] == "sparse_adam":
        opt = torch.optim.SparseAdam(list(net.parameters()), lr=wl["lr"])
        S = 2
    else:
        opt = torch.optim.Adagrad(net.parameters(), lr=wl["lr"])
        S = 1
    runner = (MlpEpochRunner if is_mlp else EpochRunner)(net, opt)

    n = (K + W) * B
    user_h, pos_h = synth_ids(wl, n, seed=1234 + rank)
    user_h, pos_h = torch.from_numpy(user_h).pin_memory(), torch.from_numpy(pos_h).pin_memory()
    user, pos = user_h.to(dev), pos_h.to(dev)
    item_meta = (torch.arange(wl["n_items"], device=dev) % wl["n_cat"]).view(-1, 1).contiguous() if F else None

    def step_block(u, p, first):
        """Everything the steps need, device side: negatives -> plan -> fused kernel."""
        neg, neg_meta = _lib.philox_negatives(1234, first, p, wl["n_items"], item_meta)
        smp = {"user": u, "pos": p, "neg": neg}
        if F:
            smp["pos_meta"] = item_meta[p]  # category of the positive (torch gather: loader-side plumbing)
            smp["neg_meta"] = neg_meta
        return runner.run(smp, B)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    sync_all = (lambda: (torch.cuda.synchronize(), dist.barrier(), torch.cuda.synchronize())) if world > 1 \
        else torch.cuda.synchronize
    clock_ramp(dev)

    # W warm-up steps, then the memory pool: an epoch of K steps needs other buffer sizes than the W warm-up steps
    # did.  Reserve them now, so that the timed region measures the steps and not torch's first cudaMalloc of each
    # size (in a real fit() every epoch has the same shape and reuses the blocks of the one before)
    loss_w = step_block(user[:W * B], pos[:W * B], 0)
    sync_all()
    first_loss = float(loss_w[0].item())
    if hasattr(runner, "reserve"):
        runner.reserve(K * B, B)
    uK, pK = user[W * B:], pos[W * B:]
    uK_h, pK_h = user_h[W * B:], pos_h[W * B:]
    seen = [W * B]

    def run_block(u, p, n_samples, loss_host=None):
        loss = step_block(u, p, seen[0])
        seen[0] += n_samples
        if loss_host is not None:
            loss_host.copy_(loss, non_blocking=True)
        return loss

    def timed(fn, n):
        e0, e1 = ev(), ev()
        sync_all()
        e0.record()
        for _ in range(n):
            loss = fn()
        e1.record()
        sync_all()
        return e0.elapsed_time(e1), loss

    # how many replays of the K-step block make a timed region of >= min_ms: probe one block, then put the replays
    # into ONE epoch (r_in x K steps: one plan build, one persistent launch) as far as the sample cap allows
    run_block(uK, pK, K * B)
    probe_ms, _ = timed(lambda: run_block(uK, pK, K * B), 1)
    R = pick_repeats(probe_ms, args.min_ms, world, dev)
    r_in, n_launch = split_repeats(R, K * B)
    R = r_in * n_launch
    uR, pR = uK.repeat(r_in), pK.repeat(r_in)
    uR_h, pR_h = uK_h.repeat(r_in).pin_memory(), pK_h.repeat(r_in).pin_memory()
    loss_host = torch.empty(r_in * K, dtype=torch.float32).pin_memory()
    if hasattr(runner, "reserve"):
        runner.reserve(r_in * K * B, B)
    resident_block = lambda: run_block(uR, pR, r_in * K * B)
    e2e_block = lambda: run_block(uR_h.to(dev, non_blocking=True), pR_h.to(dev, non_blocking=True), r_in * K * B, loss_host)
    # both regions are warmed the same way: one untimed block each (allocator sizes), then the timed ones
    resident_block()
    e2e_block()
    launches0 = runner.launches
    with ClockSampler(local) as clocks:
        ms, loss = timed(resident_block, n_launch)
    launches = (runner.launches - launches0) // n_launch + 1  # per launch of r_in x K steps; + the Philox kernel
    mean_loss = float(loss.mean().item())
    e2e_ms, _ = timed(e2e_block, n_launch)

    # ---- the fused kernel alone (roofline): the same K steps once more ----
    neg, neg_meta = _lib.philox_negatives(1234, seen[0], pK, wl["n_items"], item_meta)
    smp = {"user": uK, "pos": pK, "neg": neg}
    if F:
        smp["pos_meta"], smp["neg_meta"] = item_meta[pK], neg_meta
    b = runner.binding
    model = net.abi_model(opt.state, b.keys)
    epoch = _lib.make_epoch(smp["user"], smp["pos"], smp["neg"], smp.get("pos_meta"), smp.get("neg_meta"), B)
    scales = torch.tensor(step_scales(b, K), dtype=torch.float64).float().to(dev)
    optim_c = _lib.Optim(b.kind, 0, b.beta1, b.beta2, b.eps, scales.data_ptr())
    p0, p1, k0, k1 = ev(), ev(), ev(), ev()
    torch.cuda.synchronize()
    p0.record()
    plan = _lib.plan_build(model, epoch, dev)
    p1.record()
    loss2 = torch.empty(K, device=dev)
    if is_mlp:
        mlp_c = net.abi_mlp(runner.grads, opt.state if b.keys[0] else None, b.keys[0])
        ws = _lib.mlp_train_workspace(model, mlp_c, epoch, dev)
        k0.record()
        _lib.mlp_train_steps(model, mlp_c, epoch, optim_c, plan, ws, 0, K, loss2)
        k1.record()
    else:
        ws = _lib.train_workspace(model, epoch, dev)
        k0.record()
        _lib.train_steps(model, epoch, optim_c, plan, ws, 0, K, loss2)
        k1.record()
    torch.cuda.synchronize()
    advance_steps(opt, runner.params, b, K)
    kernel_ms, plan_ms = k0.elapsed_time(k1), p0.elapsed_time(p1)
    alg_bytes = algorithmic_bytes(wl, uK, pK, neg, K, B, S)

    times = torch.tensor([ms, e2e_ms, kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms, kernel_ms = (float(x) for x in times.cpu())

    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "kernel": "trs::train_kernel (one persistent launch, K steps)",
                "kernel_ms_per_step": kernel_ms / K, "plan_ms_per_step": plan_ms / K,
                "algorithmic_bytes_per_step": alg_bytes / K,
                "whole_step_frac": alg_bytes / (ms / R * 1e-3) / 1e9 / peak,
                "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650"}
    if is_mlp:
        # the tower's GEMMs bound this workload (SURVEY.md §8d): 3 x 2 x MACs per row, 2 rows per sample
        width, macs = wl["dim"] * 2, 0
        for h in wl["hidden"]:
            macs += width * h
            width = h
        flops_step = 3 * 2 * (macs + width) * 2 * B
        tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        tach = flops_step * K / (kernel_ms * 1e-3) / 1e12
        roofline = {"bound": "tensor", "achieved": tach, "peak": tpeak, "unit": "TFLOP/s", "frac": tach / tpeak,
                    "kernel": "trs::gemm_tn_kernel (tcgen05 GEMMs) timed inside the whole fused step: "
                              "every kernel of trs_mlp_train_steps is in the denominator",
                    "kernel_ms_per_step": kernel_ms / K, "plan_ms_per_step": plan_ms / K,
                    "algorithmic_flops_per_step": flops_step,
                    "embedding_bytes_per_step": alg_bytes / K,
                    "peak_source": "measured sustained bf16 (MEASURED_PEAKS.json)" if peaks else "fallback 1400"}
    traffic, traffic_src = traffic_of(name, K)
    roofline["traffic"] = traffic
    roofline["traffic_source"] = f"static: {traffic_src} (ncu capture of an earlier run, not measured here)" if traffic else None
    out = {
        "metric": "train samples/sec (fwd+bwd+sparse update)", "value": world * R * K * B / (ms * 1e-3),
        "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / (R * K),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if is_mlp else "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "name": name, "batch_per_gpu": B, "global_batch": B * world,
                   "optimizer": wl["opt"], "repeats": R, "steps_per_launch": r_in * K, "launches": n_launch,
                   "l2": "inputs larger than L2: tables+optimizer state "
                   f"{(wl['n_users'] + wl['n_items']) * (wl['dim'] + 1) * 4 * (1 + S) / 1e9:.2f} GB, rows hit at random",
                   "timed_region": ("Philox negatives + sort plan + fused MLP steps (one C call per launch); the K-step "
                                    "block replayed `repeats` times, `steps_per_launch` steps per epoch call"
                                    if is_mlp else
                                    "Philox negatives + sort plan + persistent fused train kernel; the K-step block "
                                    "replayed `repeats` times, `steps_per_launch` steps per plan build + kernel launch"),
                   "parallelism": (f"{world} INDEPENDENT REPLICAS of a single-GPU workload (no data-path collective: "
                                   "not a scaling result)") if world > 1 else "single GPU",
                   "clock_ramp": "0.3 s of device copies before the warm-up steps",
                   "memory_pool": "buffer sizes of a K-step epoch reserved before the timed region (no cudaMalloc inside)",
                   "first_step_loss": first_loss, "mean_loss_last_block": mean_loss,
                   "loss_note": "the K-step block is replayed `repeats` times (fresh negatives each time): the model "
                                "memorises its few samples, the hinge goes to 0; the work per step does not change"},
        "e2e": {"value": world * R * K * B / (e2e_ms * 1e-3), "unit": "samples/s",
                "h2d_bytes_per_step": 16 * B, "d2h_bytes_per_step": 4,
                "note": "user+positive ids from pinned host memory; metadata ids and negatives are derived on the device"},
        "gpu_launches": launches,
        "roofline": roofline,
        "clocks": clocks.summary(),
    }
    del runner, opt, net, plan, ws
    torch.cuda.empty_cache()
    return out, rank


# ------------------------------------------------------------------------------------------------
# predict / top-k (BASELINE configs[4])
# ------------------------------------------------------------------------------------------------
def cpu_predict(wl, budget_s):
    """The reference's predict (model.py:341-452: score every item for one user, sort, slice) on the host
    cores through oracle/torch_port.py (same ATen ops, without the per-chunk pandas frame)."""
    import torch
    from oracle import torch_port as TP
    ncores = len(os.sched_getaffinity(0))
    torch.set_num_threads(ncores)
    torch.manual_seed(1234)
    net = TP.make_net("linear", 1024, wl["n_items"], [], wl["dim"]).eval()
    t0, done = time.perf_counter(), 0
    while done < 3 or (time.perf_counter() - t0 < budget_s and done < 64):
        TP.predict_topk(net, done % 1024, wl["n_items"], wl["k"], chunk=1 << 20)
        done += 1
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "users/s", "cores": ncores, "kind": "port",
            "sample": f"{done} users x all {wl['n_items']} items, top-{wl['k']}, torch {torch.__version__} CPU, "
                      f"{ncores} threads (user table cut to 1024 rows: it is not on the path)",
            "ms_per_step": dt / done * 1e3, "steps": done}


def predict_bench(args, wl, name, K=None, W=None):
    import numpy as np
    import torch
    import torch.distributed as dist
    from torchrecsys_b200 import _lib
    from torchrecsys_b200 import sharded as S
    from torchrecsys_b200.collaborative.linear import Linear
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    K = K or args.steps
    W = W or max(args.warmup, 3)
    B, k = wl["batch"], wl["k"]
    torch.manual_seed(1234)
    # N > 1: the item table is cut into contiguous blocks, one per rank; user rows are replicated
    lo_item, hi_item = S.item_block(wl["n_items"], rank, world)
    with torch.device(dev):
        net = Linear(wl["n_users"], hi_item - lo_item, {}, wl["dim"], use_metadata=False, use_cuda=True)
    net = net.to(dev).eval()
    with torch.no_grad():
        net.item_bias.weight.normal_(0, 0.01)
    model = net.abi_model()
    cache = _lib.TopkCache()  # the item tables do not change between the steps: the bf16 item operand is prepared once
    if world > 1:
        def local_topk(u, kk, offset):
            idx, score, over = _lib.predict_topk(model, u, kk, item_offset=offset, cache=cache, cache_key="static")
            return idx, score

        def predict(u):
            idx, score = S.sharded_predict_topk(local_topk, u, k, wl["n_items"])
            return idx, score, torch.zeros(1, dtype=torch.int32, device=dev)
    else:
        predict = lambda u: _lib.predict_topk(model, u, k, cache=cache, cache_key="static")
    rng = np.random.default_rng(1234)
    users_h = torch.from_numpy(rng.integers(0, wl["n_users"], (K + W) * B)).pin_memory()
    users = users_h.to(dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    clock_ramp(dev)
    for s in range(W):
        predict(users[s * B:(s + 1) * B])
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    with ClockSampler(dev.index) as clocks:
        e0.record()
        for s in range(W, W + K):
            idx, score, over = predict(users[s * B:(s + 1) * B])
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    n_over = int(over.sum())
    x0, x1 = ev(), ev()
    out_h = torch.empty((B, k), dtype=torch.int64).pin_memory()
    x0.record()
    for s in range(W, W + K):
        u = users_h[s * B:(s + 1) * B].to(dev, non_blocking=True)
        idx, score, over = predict(u)
        out_h.copy_(idx, non_blocking=True)
    x1.record()
    torch.cuda.synchronize()
    e2e_ms = x0.elapsed_time(x1)
    peaks = load_peaks()
    tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    flops = 2.0 * wl["n_items"] * wl["dim"] * B * K
    if world > 1:
        t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = (float(x) for x in t.cpu())
    tach = flops / (ms * 1e-3) / 1e12 / world   # per GPU
    traffic, traffic_src = traffic_of(name, 1)
    del net
    torch.cuda.empty_cache()
    return {
        "metric": "predict top-k users/sec", "value": K * B / (ms * 1e-3), "unit": "users/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl["desc"], "name": name, "users_per_step": B, "top_k": k,
                   "parallelism": (f"item table in {world} contiguous blocks, local top-k per rank (the same users on "
                                   "every rank), a user's candidate lists go to ONE merger rank (all_to_all), k-way merge "
                                   "of its share of the users there, results all-gathered") if world > 1 else "single GPU",
                   "l2": "inputs larger than L2: bf16 item operand 1.44 GB streamed per user wave",
                   "timed_region": "user operand preparation + tcgen05 score/top-k kernel + exact fp32 re-scoring, every "
                                   "step; the bf16 item operand is prepared once while the tables are unchanged (first "
                                   "warm-up step)", "overflow_users_last_step": n_over},
        "e2e": {"value": K * B / (e2e_ms * 1e-3), "unit": "users/s", "h2d_bytes_per_step": 8 * B,
                "d2h_bytes_per_step": 8 * B * k},
        "gpu_launches": 7 * K,
        "roofline": {"bound": "tensor", "achieved": tach, "peak": tpeak, "unit": "TFLOP/s", "frac": tach / tpeak,
                     "traffic": traffic,
                     "traffic_source": f"static: {traffic_src} (not measured here)" if traffic else None,
                     "kernel": "trs::topk_score_kernel, timed inside the whole predict call "
                     "(preparation and re-scoring are in the denominator)",
                     "algorithmic_flops_per_step": flops / K,
                     "peak_source": "measured sustained bf16 (MEASURED_PEAKS.json)" if peaks else "fallback 1400"},
        "clocks": clocks.summary(),
    }


# ------------------------------------------------------------------------------------------------
# row-sharded large-table training (BASELINE configs[3]) -- torchrun, one rank per GPU
# ------------------------------------------------------------------------------------------------
def shard_parity_check(dev, world, rank):
    """Before anything is timed: a small problem through the SAME multi-rank path (IPC-mapped shards, NVLink loads
    and stores, flag barriers) against the fused single-GPU kernel on the same ids and initial tables.  The fused
    kernel is pinned to the reference by tests/ (golden vectors); this closes the loop for the sharded path on the
    box the numbers come from."""
    import numpy as np
    import torch
    from torchrecsys_b200.collaborative.linear import Linear
    from torchrecsys_b200.engine import EpochRunner
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    U, I, D, B, steps = 20011, 3001, 128, 2048, 4
    rng = np.random.default_rng(77)
    full = {"user.weight": rng.normal(0, .3, (U, D)).astype(np.float32),
            "item.weight": rng.normal(0, .3, (I, D)).astype(np.float32),
            "user_bias.weight": np.zeros((U, 1), np.float32),
            "item_bias.weight": rng.normal(0, .1, (I, 1)).astype(np.float32)}
    full = {k: torch.from_numpy(v) for k, v in full.items()}
    ids = [torch.from_numpy(rng.integers(0, m, B * steps)).to(dev) for m in (U, I, I)]
    tr = ShardedLinearTrainer(U, I, D, global_batch=B, optimizer="sparse_adam", lr=0.01, device=dev)
    tr.load_state_dict(full)
    loss_s = tr.train_epoch(*ids, B)
    sd = tr.state_dict()
    out = {"ok": True}
    if rank == 0:
        net = Linear(U, I, {}, D, use_metadata=False, use_cuda=True)
        net.load_state_dict(full)
        net = net.to(dev)
        opt = torch.optim.SparseAdam(list(net.parameters()), lr=0.01)
        loss_f = EpochRunner(net, opt).run({"user": ids[0], "pos": ids[1], "neg": ids[2]}, B)
        dl = float((loss_s - loss_f).abs().max())
        dw = max(float((sd[k] - v).abs().max()) for k, v in net.state_dict().items())
        out = {"ok": bool(dl < 1e-5 and dw < 2e-4), "max_abs_loss_diff": dl, "max_abs_param_diff": dw,
               "what": f"{steps} SparseAdam steps of a {U}x{I} dim-{D} Linear, batch {B}, on {world} ranks over "
                       "IPC-mapped shards vs the fused single-GPU kernel (same ids, same initial tables)"}
        del net, opt
    tr.close()
    del tr
    torch.cuda.empty_cache()
    return out


DUMP_ROWS = 8192        # rows per table that --dump-outputs writes
DUMP_BYTES = 64 << 20


def shard_outputs(tr, loss, users, items):
    """What a caller of the timed epoch receives: its per-step losses, and the user / item rows (embedding and bias)
    that its last step updated -- all of them up to DUMP_ROWS per table, else a fixed, seeded sample; only the rows this
    process holds.  Row ids are stored as float64 (exact below 2^53)."""
    import numpy as np
    import torch
    out = {"loss": loss.float().cpu().numpy()}
    G = tr.world
    for name, ids in (("user", users), ("item", items)):
        rows = np.unique(ids.cpu().numpy())
        rows = rows[np.isin(rows % G, tr.local_ranks)]
        if len(rows) > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(1234).choice(rows, DUMP_ROWS, replace=False))
        weight = np.empty((len(rows), tr.dim), np.float32)
        bias = np.empty(len(rows), np.float32)
        for q in tr.local_ranks:
            mine = rows % G == q
            local = torch.from_numpy(rows[mine] // G).to(tr.device)
            emb, lin = tr.tables[q][name]
            weight[mine] = emb.index_select(0, local).cpu().numpy()
            bias[mine] = lin.index_select(0, local).view(-1).cpu().numpy()
        out[f"{name}_ids"] = rows.astype(np.float64)
        out[f"{name}_weight"] = weight
        out[f"{name}_bias"] = bias
    return out


def write_outputs(path, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES} byte budget")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def sharded_bench(args, wl, name):
    import numpy as np
    import torch
    import torch.distributed as dist
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    emu = args.emulate_world if world == 1 else 0
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    if args.shard_it:
        _lib.lib().trs_debug_shard_chunks_per_lane(args.shard_it)
    if args.shard_overlap is not None:
        _lib.lib().trs_debug_shard_overlap(args.shard_overlap)
    if args.shard_remote_hint is not None:
        _lib.lib().trs_debug_shard_remote_hint(args.shard_remote_hint)
    G = emu or world                       # ranks of the group
    K, W, B = args.steps, max(args.warmup, 3), wl["batch"]
    Bg = B * G
    D = wl["dim"]
    parity = shard_parity_check(dev, world, rank) if world > 1 else None
    torch.manual_seed(1234 + rank)         # the tables' N(0, 1/dim) initialisation: the same inputs on every run
    tr = ShardedLinearTrainer(wl["n_users"], wl["n_items"], D, global_batch=Bg, optimizer=wl["opt"], lr=wl["lr"],
                              device=dev, emulate_world=emu or (1 if world == 1 else None))
    # every rank's loader output: (K + W) steps of its own B samples, stored [step, {user, positive}, B] so that a
    # run of steps is one contiguous block (in emulation this process holds all G ranks' outputs)
    mine = list(range(G)) if world == 1 else [rank]

    def loader_output(q):
        import numpy as np
        u, p = synth_ids(wl, (K + W) * B, seed=1234 + q)
        return torch.from_numpy(np.stack([u.reshape(K + W, B), p.reshape(K + W, B)], 1)).pin_memory()

    ids_h = {q: loader_output(q) for q in mine}
    ids_d = {q: t.to(dev) for q, t in ids_h.items()}

    def global_epoch(src, lo_step, n_steps):
        """All ranks' samples of steps [lo_step, lo_step + n_steps) in loader order: step-major, rank-major inside a
        step.  ONE all-gather per epoch (NCCL) -- the only collective besides the loss all-reduce."""
        if world > 1:
            part = src[rank][lo_step:lo_step + n_steps]
            if not part.is_cuda:
                part = part.to(dev, non_blocking=True)
            return tuple(tr.gather_epoch(part))     # ids cross NVLink as int32, widened while reordering
        allr = torch.stack([src[q][lo_step:lo_step + n_steps].to(dev, non_blocking=True) for q in mine])
        cols = allr.permute(2, 1, 0, 3).contiguous()     # [G, steps, 2, B] -> [2, steps, G, B]
        return cols[0].view(-1), cols[1].view(-1)

    seen = [0]

    def block(src, lo_step, n_steps, timing=False, loss_host=None):
        gu, gp = global_epoch(src, lo_step, n_steps)
        neg, _ = _lib.philox_negatives(1234, seen[0], gp, wl["n_items"])
        seen[0] += n_steps * Bg
        loss = tr.train_epoch(gu, gp, neg, Bg, check=False, timing=timing)
        if loss_host is not None:
            loss_host.copy_(loss, non_blocking=True)
        return loss, (gu, gp, neg)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    sync_all = (lambda: (torch.cuda.synchronize(), dist.barrier(), torch.cuda.synchronize())) if world > 1 \
        else torch.cuda.synchronize
    clock_ramp(dev)
    loss_w = block(ids_d, 0, W)[0]
    sync_all()
    tr.check_status()
    first_loss = float(loss_w[0].item())

    def timed(fn):
        e0, e1 = ev(), ev()
        sync_all()
        e0.record()
        out = fn()
        e1.record()
        sync_all()
        return e0.elapsed_time(e1), out

    # the K timed steps (loader steps [W, W + K)) are ONE epoch: one id all-gather, one plan build, one persistent
    # launch per rank -- cut into several launches only where K x global batch exceeds the sample cap
    n_launch = -(-K * Bg // SAMPLE_CAP)
    per_launch = -(-K // n_launch)
    loss_host = torch.empty(K, dtype=torch.float32).pin_memory()

    def resident_epoch():
        """The K steps from ids already in HBM; per launch: its losses, the events around its plan build and kernel,
        and its (user, positive, negative) ids."""
        launches = []
        for s in range(0, K, per_launch):
            loss, step_ids = block(ids_d, W + s, min(per_launch, K - s), timing=True)
            launches.append((loss, tr.events, step_ids))
        return launches

    if emu:
        def e2e_epoch():
            return torch.cat([block(ids_h, W + s, min(per_launch, K - s), loss_host=loss_host[s:s + per_launch])[0]
                              for s in range(0, K, per_launch)])
    else:   # the trainer's own host-fed epoch: chunks copied on a side stream while the previous chunk trains
        def draw(gp, first):
            neg, _ = _lib.philox_negatives(1234, seen[0] + first, gp, wl["n_items"])
            return neg

        def e2e_epoch():
            loss = tr.train_epoch_host(ids_h[rank][W:], draw, loss_host)
            seen[0] += K * Bg
            return loss
    # both timed epochs are run once untimed first, on the same steps: the plan, workspace and allocator blocks of a
    # K-step epoch exist before the timed region (no cudaMalloc inside it)
    resident_epoch()
    e2e_epoch()
    sync_all()
    tr.check_status()
    launches0 = tr.launches
    with ClockSampler(local) as clocks:
        ms, timed_launches = timed(resident_epoch)
    loss = torch.cat([l for l, _, _ in timed_launches])
    events = [e for _, e, _ in timed_launches]
    gu, gp, neg = (torch.cat(c) for c in zip(*(i for _, _, i in timed_launches)))
    launches = (tr.launches - launches0) // n_launch + 1   # per launch; + the Philox kernel
    tr.check_status()
    mean_loss = float(loss.mean().item())
    outputs = shard_outputs(tr, loss, gu[-Bg:], torch.cat([gp[-Bg:], neg[-Bg:]])) if args.dump_outputs else None
    e2e_ms, _ = timed(e2e_epoch)
    tr.check_status()
    kernel_ms = sum(k0.elapsed_time(k1) for _, _, k0, k1 in events)     # per K steps
    plan_ms = sum(p0.elapsed_time(p1) for p0, p1, _, _ in events)
    times = torch.tensor([ms, e2e_ms, kernel_ms, plan_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms, kernel_ms, plan_ms = (float(x) for x in times.cpu())

    S_ = {"sgd": 0, "adagrad": 1, "sparse_adam": 2}[wl["opt"]]
    alg = algorithmic_bytes(wl, gu, gp, neg, K, Bg, S_)        # of the GLOBAL batch; every rank owns 1/G of the rows
    # bytes that must cross NVLink per rank and direction: item rows (+ bias) whose owner is not the sample's rank,
    # read in phase A and their gradient rows (+ bias gradient) stored back; a rank serves as much as it asks for
    remote = int(((gp % G) != (gu % G)).sum() + ((neg % G) != (gu % G)).sum())
    nvl_dir = 2.0 * remote * (4 * D + 4) / G
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ach = alg / G / (kernel_ms * 1e-3) / 1e9
    nvl_ach = nvl_dir / (kernel_ms * 1e-3) / 1e9
    t_hbm, t_nvl = alg / G / (peak * 1e9), nvl_dir / (NVLINK_GBS * 1e9)
    out = {
        "metric": "train samples/sec (fwd+bwd+sparse update)", "value": K * Bg / (ms * 1e-3), "unit": "samples/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "name": name, "batch_per_gpu": B, "global_batch": Bg, "optimizer": wl["opt"],
                   "steps_per_launch": per_launch, "launches": n_launch,
                   "parallelism": (f"user / item tables ROW-SHARDED over {G} ranks (row % {G}); samples run on their "
                                   "user row's owner; item rows read from and gradient rows stored into the owner's "
                                   "HBM over NVLink by one persistent kernel per rank (CUDA-IPC mapped shards, flag "
                                   "barriers); NCCL: id all-gather per epoch + loss all-reduce")
                   + (f" [EMULATED: all {G} ranks hosted by one launch on ONE GPU, no NVLink]" if emu else ""),
                   "l2": f"inputs larger than L2: {(wl['n_users'] + wl['n_items']) * (D + 1) * 4 * (1 + S_) / G / 1e9:.1f} "
                         "GB of tables + optimizer state per rank, rows hit at random",
                   "timed_region": "id all-gather (NCCL) + Philox negatives + routing / sort plan + persistent sharded "
                                   "kernel + loss all-reduce; exactly K steps, `steps_per_launch` steps per all-gather + plan "
                                   "build + kernel launch (max over ranks); each timed epoch also ran once untimed on "
                                   "the same steps",
                   "clock_ramp": "0.3 s of device copies before the warm-up steps",
                   "first_step_loss": first_loss, "mean_loss_last_block": mean_loss,
                   "loss_note": "mean over the K timed steps, the third pass over their samples (fresh negatives "
                                "each time)"},
        "e2e": {"value": K * Bg / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": 16 * B,
                "d2h_bytes_per_step": 4,
                "note": "ShardedLinearTrainer.train_epoch_host: each rank's user+positive ids from pinned host memory in "
                        "chunks of >= 64 steps, chunk i+1 copied on a side stream while chunk i trains; negatives are "
                        "drawn on the device; per-step losses back to pinned host memory"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": traffic_of(name, K)[0],
                     "traffic_source": "static: profiles/shard_r2.md (ncu --set full of a 1-rank launch on 4M x 1M tables; "
                                       "per step, times K; not measured by this run)",
                     "kernel": "trs::shard_train_kernel (one persistent launch per rank)",
                     "kernel_time_source": "CUDA events around the persistent launches INSIDE the timed region, "
                                           "summed over its launches, max over ranks",
                     "kernel_ms_per_step": kernel_ms / K, "plan_ms_per_step": plan_ms / K,
                     "algorithmic_bytes_per_step": alg / K / G,
                     "whole_step_frac": alg / G / (ms * 1e-3) / 1e9 / peak,
                     "nvlink": {"bytes_per_step_per_direction": nvl_dir / K, "achieved": nvl_ach, "peak": NVLINK_GBS,
                                "unit": "GB/s per direction per GPU", "frac": nvl_ach / NVLINK_GBS,
                                "peak_source": "measured peer copy on this pool (B200_PROFILING.md); 900 nominal"},
                     "limiter": "nvlink" if t_nvl > t_hbm else "hbm",
                     "frac_of_binding_roofline": max(t_hbm, t_nvl) / (kernel_ms * 1e-3),
                     "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650"},
        "clocks": clocks.summary(),
    }
    if parity is not None:
        out["parity_check"] = parity
    tr.close()
    del tr
    torch.cuda.empty_cache()
    return out, outputs


# ------------------------------------------------------------------------------------------------
# BASELINE configs[0] as a user runs it (README.md:53-80): TorchRecSys(...).fit(optimizer, epochs=5, batch_size=1024)
# ------------------------------------------------------------------------------------------------
def c1_fit_bench(with_cpu: bool):
    """Wall time of the public ``fit`` on the README shape (linear, 3k users x 1k items, 100k interactions, D = 80,
    80 000 training rows, batch 1024, 5 epochs, SparseAdam -- README's Adam cannot run, SURVEY D2), host to host:
    includes the device loader's shuffles, negatives, plan, kernel and the per-epoch loss read-back.  Beside it the
    reference's loop body (oracle/torch_port.py) over the same number of batches on the host cores."""
    import contextlib
    import io
    import numpy as np
    import pandas as pd
    import torch
    from torchrecsys.model import TorchRecSys
    rng = np.random.default_rng(1234)
    df = pd.DataFrame({"user": rng.choice(3000, 100_000), "item": rng.choice(1000, 100_000)})
    np.random.seed(1234)
    torch.manual_seed(1234)
    with contextlib.redirect_stdout(io.StringIO()):
        model = TorchRecSys(df, "user", "item", n_factors=80, net_type="linear", use_cuda=True)
        opt = torch.optim.SparseAdam(list(model.parameters()), lr=1e-3)
        model.fit(opt, epochs=1, batch_size=1024)        # first call: allocator, module load
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.fit(opt, epochs=5, batch_size=1024)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    n_train = int(model.data_processor.train_data["user_id"].numel())
    out = {"workload": "BASELINE configs[0]: README quickstart, TorchRecSys(net_type='linear').fit(SparseAdam, epochs=5, "
                       "batch_size=1024) on 3k users x 1k items, 100k interactions",
           "fit_wall_s": wall, "value": 5 * n_train / wall, "unit": "samples/s", "train_rows": n_train,
           "steps": 5 * -(-n_train // 1024)}
    if with_cpu:
        from oracle import torch_port as TP
        torch.set_num_threads(min(4, len(os.sched_getaffinity(0))))   # SURVEY.md §6: 4 threads are this shape's best
        net = TP.make_net("linear", model.n_users, model.n_items, [], 80)
        popt = TP.make_optimizer("sparse_adam", net, 1e-3)
        tr = model.data_processor.train_data
        ids = {"user": tr["user_id"], "pos": tr["pos_item_id"], "neg": tr["neg_item_id"]}
        t0 = time.perf_counter()
        for _ in range(5):
            perm = torch.randperm(n_train)
            for lo in range(0, n_train, 1024):
                sel = perm[lo:lo + 1024]
                TP.train_step(net, popt, {k: v[sel] for k, v in ids.items()})
        cpu_wall = time.perf_counter() - t0
        out["cpu_port"] = {"fit_wall_s": cpu_wall, "value": 5 * n_train / cpu_wall, "threads": torch.get_num_threads(),
                           "what": "the reference's loop body (forward x2, hinge, backward, SparseAdam.step, loss.item) "
                                   "over the same 5 x 79 batches, torch CPU"}
    return out


# ------------------------------------------------------------------------------------------------
def brief(line):
    """The part of a full bench line that other_workloads keeps."""
    r = line.get("roofline", {})
    return {"metric": line["metric"], "value": line["value"], "unit": line["unit"], "ms_per_step": line["ms_per_step"],
            "steps": line["steps"], "repeats": line["config"].get("repeats"), "workload": line["config"]["workload"],
            "parallelism": line["config"].get("parallelism"), "e2e": line["e2e"]["value"],
            "roofline": {k: r.get(k) for k in ("bound", "achieved", "peak", "unit", "frac", "kernel_ms_per_step",
                                               "plan_ms_per_step", "limiter", "frac_of_binding_roofline") if k in r},
            "gpu_launches": line.get("gpu_launches"), "clocks": line.get("clocks")}


def resolve(args):
    name = args.workload
    if name == "c4":
        name = "c4_linear"   # every N runs the row-sharded kernel (N = 1: a group of one rank)
    wl = dict(WORKLOADS[name])
    if args.batch:
        wl["batch"] = args.batch
    if args.users:
        wl["n_users"] = args.users
        wl["desc"] += f" [users overridden: {args.users}]"
    if args.items:
        wl["n_items"] = args.items
        wl["desc"] += f" [items overridden: {args.items}]"
    if args.dim:
        wl["dim"] = args.dim
        wl["desc"] += f" [n_factors overridden: {args.dim}]"
    if args.zipf:
        wl["zipf"] = args.zipf
        wl["desc"] += f" [ids drawn from Zipf({args.zipf})]"
    return name, wl


def reference_line(args, wl, name, device):
    impl = "reference" if device == "cpu" else "torch_cuda"
    if wl.get("predict"):
        r = cpu_predict(wl, max(args.cpu_seconds, 20.0) * 3)
        metric, unit, W = "predict top-k users/sec", "users/s", 0
    else:
        W = max(1, min(args.warmup, 3))
        r = port_reference(wl, max(1, args.steps), W, budget_s=max(args.cpu_seconds, 20.0) * 3, device=device)
        metric, unit = "train samples/sec (fwd+bwd+sparse update)", "samples/s"
    return {"impl": impl, "metric": metric, "value": r["value"], "unit": unit, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": W, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "name": name, "batch_per_gpu": wl["batch"]},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def main():
    args = parse_args()
    name, wl = resolve(args)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl in ("reference", "torch_cuda"):
        if rank == 0:
            print(json.dumps(reference_line(args, wl, name, "cpu" if args.impl == "reference" else "cuda")))
        return
    outputs = None
    if wl.get("predict"):
        out = predict_bench(args, wl, name)
    elif wl.get("sharded"):
        out, outputs = sharded_bench(args, wl, name)
    else:
        out, _ = gpu_bench(args, wl, name)
    # ---- the other BASELINE configs, in the same line ----
    others = {}
    if args.workload == "c4" and not args.no_others:
        import copy
        import gc
        import torch
        sub = copy.copy(args)
        gc.collect()
        torch.cuda.empty_cache()
        try:
            if world == 1 and not args.emulate_world:
                sub.steps, sub.warmup = max(args.steps, 20), max(args.warmup, 5)
                others["c2_fm"] = brief(gpu_bench(sub, dict(WORKLOADS["c2_fm"]), "c2_fm")[0])
                others["c3_mlp"] = brief(gpu_bench(sub, dict(WORKLOADS["c3_mlp"]), "c3_mlp")[0])
                others["c5_predict"] = brief(predict_bench(sub, dict(WORKLOADS["c5_predict"]), "c5_predict", K=5, W=3))
                others["c1_fit"] = c1_fit_bench(with_cpu=not args.no_cpu_baseline)
                sub.steps, sub.warmup = args.steps, args.warmup
                others["c4_fused_fit_kernel"] = brief(gpu_bench(sub, dict(WORKLOADS["c4_fused"]), "c4_fused")[0])
            elif world > 1:
                others["c5_predict"] = brief(predict_bench(sub, dict(WORKLOADS["c5_predict"]), "c5_predict", K=5, W=3))
        except Exception as e:  # a sub-result must never cost the headline line
            others["error"] = f"{type(e).__name__}: {e}"
    if world > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    if rank != 0:
        return
    if others:
        out["other_workloads"] = others
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if args.gpus == 1 and not args.no_cpu_baseline:
        r = cpu_predict(wl, args.cpu_seconds) if wl.get("predict") else \
            port_reference(wl, steps=8, warmup=1, budget_s=args.cpu_seconds)
        out["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
