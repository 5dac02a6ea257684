"""Phase timeline of trs::shard_train_kernel on the C4 shape: per step, when the slowest / average CTA finishes
phase A, leaves barrier 1, finishes phase B, and how long the next phase A waits for the step's end (globaltimer stamps,
trs_debug_shard_trace).
    python tools/shard_phases.py [--world 1] [--users 50000000] [--items 5000000] [--steps 12] [--it 2]   # one GPU
        [--one-pass 0]   # one rank: the two-phase kernel instead of the one-pass one (trs_debug_shard_one_pass)
    torchrun --nproc-per-node N tools/shard_phases.py ...                                                 # real peers"""
import argparse
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from torchrecsys_b200 import _lib  # noqa: E402
from torchrecsys_b200.sharded import ShardedLinearTrainer  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--world", type=int, default=1)
ap.add_argument("--users", type=int, default=50_000_000)
ap.add_argument("--items", type=int, default=5_000_000)
ap.add_argument("--dim", type=int, default=128)
ap.add_argument("--batch", type=int, default=16384)
ap.add_argument("--steps", type=int, default=12)
ap.add_argument("--it", type=int, default=1)
ap.add_argument("--overlap", type=int, default=-1)
ap.add_argument("--one-pass", type=int, default=1)
a = ap.parse_args()
real = "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
rank = 0
if real:
    dist.init_process_group("nccl", device_id=dev)
    rank, a.world = dist.get_rank(), dist.get_world_size()
L = _lib.lib()
L.trs_debug_shard_chunks_per_lane(a.it)
L.trs_debug_shard_overlap(a.overlap)
L.trs_debug_shard_one_pass(a.one_pass)
G, B = a.world, a.batch * a.world
tr = ShardedLinearTrainer(a.users, a.items, a.dim, global_batch=B, device=dev, emulate_world=None if real else G)
rng = np.random.default_rng(0)
n = a.steps * B
ids = [torch.from_numpy(rng.integers(0, m, n)).to(dev) for m in (a.users, a.items, a.items)]
tr.train_epoch(*ids, B)  # warm
sm = _lib.device_info()[0]
n_local = 1 if real else G
cpr = sm // n_local
buf = torch.zeros(n_local * a.steps * cpr * 8, dtype=torch.int64, device=dev)
L.trs_debug_shard_trace(C.c_void_p(buf.data_ptr()))
if real:
    torch.cuda.synchronize()
    dist.barrier()
tr.train_epoch(*ids, B)
torch.cuda.synchronize()
L.trs_debug_shard_trace(None)
t = buf.cpu().numpy().reshape(n_local, a.steps, cpr, 8).astype(np.float64) / 1e3  # us
names = ["A done", "bar1 left", "B done", "arrived at end"]
if rank == 0:
    print(f"world {G}{' (real peers)' if real else ' (one GPU)'}, {cpr} CTAs per rank, batch/rank {a.batch}, "
          f"{a.it} chunks per lane, {'one-pass' if L.trs_debug_shard_last_one_pass() == 1 else 'two-phase'} kernel; "
          "microseconds from the step's earliest start")
for r in range(n_local):
    if rank == 0:
        for s in range(max(2, a.steps - 4), a.steps):
            t0 = t[r, s, :, 0].min()
            row = [f"start max {t[r, s, :, 0].max() - t0:5.1f}"]
            for j, nm in enumerate(names, 1):
                x = t[r, s, :, j] - t0
                row.append(f"{nm}: avg {x.mean():5.1f} max {x.max():5.1f}")
            print(f"rank {r} step {s}: " + " | ".join(row))
    d = t[r, 2:, :, :]
    step = np.mean(d[1:, :, 0].min(axis=1) - d[:-1, :, 0].min(axis=1))
    who = rank if real else r
    # the wait for the barrier that ends step s sits inside step s + 1's phase A, after its first pass (stamps 5, 6)
    wait = np.mean(d[1:, :, 6] - d[1:, :, 5])
    print(f"rank {who} mean over steps (avg CTA): A {np.mean(d[:, :, 1] - d[:, :, 0]):.1f} (first pass "
          f"{np.mean(d[1:, :, 5] - d[1:, :, 0]):.1f}, wait for the previous step's end {wait:.1f})  "
          f"bar1 {np.mean(d[:, :, 2] - d[:, :, 1]):.1f}  B {np.mean(d[:, :, 3] - d[:, :, 2]):.1f}  "
          f"arrive {np.mean(d[:, :, 4] - d[:, :, 3]):.1f}  step {step:.1f}", flush=True)
if real:
    dist.barrier()
    tr.close()
    dist.destroy_process_group()
