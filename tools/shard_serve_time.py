"""Times serving on the row-sharded tables at the benchmark's shape (50M users x 5M items, D = 128, SparseAdam state
allocated), with CUDA events; prints one JSON line per measurement (rank 0).

    python tools/shard_serve_time.py                       # one GPU (W = 1)
    torchrun --nproc-per-node=N tools/shard_serve_time.py  # N GPUs, real peers

  * evaluate (loss + auc) on a 2^20-sample split at batch 512 and 16384, samples/s;
  * at W = 1, trs_eval_pairwise on the same tables (the shard IS the whole table there);
  * predict_topk of 18944 users at top-100, users/s, first call (prepares the bf16 item operand) and a cached call;
  * for comparison, what to_model + predict_batch cost: the gather of the tables (state_dict, the part of to_model that
    moves data) followed by trs_predict_topk on the gathered model, with the peak device memory above the trainer's.
The tables are read from HBM (several GB; far beyond the 126 MB L2).

    python tools/shard_serve_time.py --recommend           # recommend cases only (one GPU)

  * recommend of 18944 users at D = 128: k = 100 with about 20 excluded items per user (tensor-core path) and k = 1000
    (exact kernel), with the exact path's share of its FP32-FMA bound; at D = 256 (SGD state, so that it fits) k = 100
    (exact kernel); what a user does today for k = 1000 -- gather the tables, then TorchRecSys._predict_exact's trs_scores
    over every item + a stable sort per user -- for a sample of users, per user.
  The card's name, power limit and clocks are read with nvidia-smi in the same run."""
import argparse
import json
import os
import subprocess
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


# FP32 FMA on CUDA cores: 148 SMs x 128 lanes x 2 FLOP x 1.965 GHz (max SM clock); derived, the card may clock lower
FMA_BOUND_FLOPS = 148 * 128 * 2 * 1.965e9


def card():
    """name, power limit and clocks as nvidia-smi reports them now."""
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout
    except (OSError, subprocess.SubprocessError) as e:
        return {"nvidia_smi": f"unavailable: {e}"}
    return dict(zip(q.split(","), (v.strip() for v in line.strip().split(","))))


def recommend_cases(a, dev):
    out = []
    g = torch.Generator(device=dev).manual_seed(11)
    head = {"gpu": torch.cuda.get_device_properties(dev).name, "world": 1, "users": a.users, "items": a.items}
    for D, opt in ((128, "sparse_adam"), (256, "sgd")):
        tr = ShardedLinearTrainer(a.users, a.items, D, global_batch=16384, optimizer=opt, lr=1e-3, device=dev,
                                  emulate_world=1)
        for name in ("user", "item"):
            tr.tables[0][name][1].normal_(0, .1)
        # distinct users: a user drawn twice would have 40 excluded items and push k + 40 past the tensor-core limit
        q = torch.randperm(a.users, device=dev, generator=g)[:a.queries]
        ex_user = q.repeat_interleave(20)
        ex_item = torch.randint(0, a.items, (ex_user.numel(),), device=dev, generator=g)
        h = dict(head, dim=D, optimizer=opt, queries=a.queries)
        cases = [(100, (ex_user, ex_item), "exclude ~20 per user")] if D == 128 else []
        cases += [(1000, None, "no exclusion")] if D == 128 else [(100, None, "no exclusion")]
        for k, ex, label in cases:
            ms, runs = timed(lambda: tr.recommend(q, k, exclude=ex), a.reps)
            row = dict(h, what=f"recommend k={k}, {label}", k=k, ms=ms, runs_ms=runs, users_per_s=a.queries / ms * 1e3)
            row.update(path=tr.last_recommend_paths[0])   # the path recommend took
            if row["path"] == "exact":   # 2 D FLOP per (user, item)
                flop = 2.0 * D * a.items * a.queries
                row.update(tflops=flop / ms / 1e9, fma_bound_ms=flop / FMA_BOUND_FLOPS * 1e3,
                           share_of_fma_bound=flop / FMA_BOUND_FLOPS * 1e3 / ms)
            out.append(row)
        if D == 128:   # today's k = 1000: gather the tables, then trs_scores over every item + stable sort per user
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sd = tr.state_dict()
            model = _lib.make_model(_lib.NET_LINEAR, D, _lib.make_table(sd["user.weight"], lin=sd["user_bias.weight"]),
                                    _lib.make_table(sd["item.weight"], lin=sd["item_bias.weight"]), [])
            e1.record()
            torch.cuda.synchronize()
            gather_ms = e0.elapsed_time(e1)
            items = torch.arange(a.items, device=dev)

            def exact_one(u):
                s = _lib.scores(model, torch.full_like(items, u), items)
                return torch.sort(s, descending=True, stable=True)[1][:1000].cpu()

            sample = q[:a.sample_users].tolist()
            exact_one(sample[0])
            torch.cuda.synchronize()
            e0.record()
            for u in sample:
                exact_one(u)
            e1.record()
            torch.cuda.synchronize()
            per = e0.elapsed_time(e1) / len(sample)
            out.append(dict(h, what="gather + _predict_exact per user, k=1000", k=1000, gather_ms=gather_ms,
                            sampled_users=len(sample), ms_per_user=per,
                            ms_for_all_queries_estimated=per * a.queries + gather_ms))
            del sd, model
        tr.close()
        del tr
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=50_000_000)
    ap.add_argument("--items", type=int, default=5_000_000)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--samples", type=int, default=1 << 20)
    ap.add_argument("--queries", type=int, default=18944)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-gather", action="store_true", help="skip the to_model + predict_batch comparison")
    ap.add_argument("--recommend", action="store_true", help="only the recommend cases (one GPU)")
    ap.add_argument("--sample-users", type=int, default=16)
    a = ap.parse_args()
    if a.recommend:
        dev = torch.device("cuda", 0)
        c = card()
        for o in recommend_cases(a, dev):
            print(json.dumps(dict(o, card=c)))
        return
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
