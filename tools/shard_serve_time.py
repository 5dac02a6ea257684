"""Times serving on the row-sharded tables at the benchmark's shape (50M users x 5M items, D = 128, SparseAdam state
allocated), with CUDA events; prints one JSON line per measurement (rank 0).

    python tools/shard_serve_time.py                       # one GPU (W = 1)
    torchrun --nproc-per-node=N tools/shard_serve_time.py  # N GPUs, real peers

  * evaluate (loss + auc) on a 2^20-sample split at batch 512 and 16384, samples/s;
  * at W = 1, trs_eval_pairwise on the same tables (the shard IS the whole table there);
  * predict_topk of 18944 users at top-100, users/s, first call (prepares the bf16 item operand) and a cached call;
  * for comparison, what to_model + predict_batch cost: the gather of the tables (state_dict, the part of to_model that
    moves data) followed by trs_predict_topk on the gathered model, with the peak device memory above the trainer's.
The tables are read from HBM (several GB; far beyond the 126 MB L2)."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from torchrecsys_b200 import _lib  # noqa: E402
from torchrecsys_b200.sharded import ShardedLinearTrainer  # noqa: E402


def timed(fn, reps):
    """(median ms, all ms) of fn() over reps runs, CUDA events around each, after one warm-up run."""
    fn()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return sorted(out)[len(out) // 2], out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=50_000_000)
    ap.add_argument("--items", type=int, default=5_000_000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--samples", type=int, default=1 << 20)
    ap.add_argument("--queries", type=int, default=18944)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-gather", action="store_true", help="skip the to_model + predict_batch comparison")
    a = ap.parse_args()
    real = "WORLD_SIZE" in os.environ and int(os.environ["WORLD_SIZE"]) > 1
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if real:
        dist.init_process_group("nccl", device_id=dev)
    W = dist.get_world_size() if real else 1
    lead = not real or dist.get_rank() == 0
    props = torch.cuda.get_device_properties(dev)
    tr = ShardedLinearTrainer(a.users, a.items, a.dim, global_batch=16384, optimizer="sparse_adam", lr=1e-3,
                              device=dev, emulate_world=None if real else 1)
    for r in tr.local_ranks:
        for name in ("user", "item"):
            tr.tables[r][name][1].normal_(0, .1)
    g = torch.Generator(device=dev).manual_seed(7)        # the same split on every rank
    user = torch.randint(0, a.users, (a.samples,), device=dev, generator=g)
    pos = torch.randint(0, a.items, (a.samples,), device=dev, generator=g)
    neg = torch.randint(0, a.items, (a.samples,), device=dev, generator=g)
    head = {"gpu": props.name, "world": W, "users": a.users, "items": a.items, "dim": a.dim}
    out = []
    for B in (512, 16384):
        ms, runs = timed(lambda: tr.evaluate(user, pos, neg, B), a.reps)
        out.append(dict(head, what="evaluate", batch=B, samples=a.samples, ms=ms, runs_ms=runs,
                        samples_per_s=a.samples / ms * 1e3))
        if W == 1:
            emb_u, lin_u = tr.tables[0]["user"]
            emb_i, lin_i = tr.tables[0]["item"]
            model = _lib.make_model(_lib.NET_LINEAR, a.dim, _lib.make_table(emb_u, lin=lin_u),
                                    _lib.make_table(emb_i, lin=lin_i), [])
            ep = _lib.make_epoch(user, pos, neg, None, None, B)
            ms, runs = timed(lambda: _lib.eval_pairwise(model, ep), a.reps)
            out.append(dict(head, what="trs_eval_pairwise", batch=B, samples=a.samples, ms=ms, runs_ms=runs,
                            samples_per_s=a.samples / ms * 1e3))
            ms, runs = timed(lambda: tr.eval_pairwise(user, pos, neg, B), a.reps)
            out.append(dict(head, what="eval_pairwise", batch=B, samples=a.samples, ms=ms, runs_ms=runs,
                            samples_per_s=a.samples / ms * 1e3))
    q = torch.randint(0, a.users, (a.queries,), device=dev, generator=g)
    firsts = []
    for _ in range(a.reps):
        tr._state_version += 1                          # as a load_state_dict would: the item operand is rebuilt
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tr.predict_topk(q, 100)
        e1.record()
        torch.cuda.synchronize()
        firsts.append(e0.elapsed_time(e1))
    ms = sorted(firsts)[len(firsts) // 2]
    out.append(dict(head, what="predict_topk first call", queries=a.queries, k=100, ms=ms, runs_ms=firsts,
                    users_per_s=a.queries / ms * 1e3, overflow=tr.last_predict_overflow))
    ms, runs = timed(lambda: tr.predict_topk(q, 100), a.reps)
    out.append(dict(head, what="predict_topk cached", queries=a.queries, k=100, ms=ms, runs_ms=runs,
                    users_per_s=a.queries / ms * 1e3))
    if not a.no_gather:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sd = tr.state_dict()
        model = _lib.make_model(_lib.NET_LINEAR, a.dim, _lib.make_table(sd["user.weight"], lin=sd["user_bias.weight"]),
                                _lib.make_table(sd["item.weight"], lin=sd["item_bias.weight"]), [])
        _lib.predict_topk(model, q, 100)
        e1.record()
        torch.cuda.synchronize()
        out.append(dict(head, what="gather (state_dict) + trs_predict_topk", queries=a.queries, k=100,
                        ms=e0.elapsed_time(e1), users_per_s=a.queries / e0.elapsed_time(e1) * 1e3,
                        peak_extra_gib=(torch.cuda.max_memory_allocated(dev) - base) / 2 ** 30))
    if lead:
        for o in out:
            print(json.dumps(o))
    tr.close()
    if real:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
