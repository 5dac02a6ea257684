"""torchrun worker: evaluation, prediction and row lookups on the row-sharded tables over REAL peers (CUDA-IPC mapped
shards read over NVLink; torchrecsys_b200/sharded.py + csrc/shard_serve.cu, recommend with exclusions), each against the single-GPU kernels on
the gathered model, bit for bit.  Training runs between the serving calls, so the ordering of peer reads against the
owners' next updates is exercised too.  Prints SHARD SERVE CHECK OK on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from torchrecsys_b200 import _lib, sharded as S  # noqa: E402


def want_topk(model, users, k):
    """trs_predict_topk on the gathered model, overflowing users ranked by trs_scores + stable sort (predict_batch)."""
    idx, score, over = _lib.predict_topk(model, users, k)
    items = torch.arange(model.item.n_rows, device=users.device)
    for q in torch.nonzero(over).flatten().tolist():
        s, order = torch.sort(_lib.scores(model, torch.full_like(items, int(users[q])), items), descending=True,
                              stable=True)
        idx[q], score[q] = order[:k], s[:k]
    return idx, score


def gathered(tr):
    sd = tr.state_dict()
    model = _lib.make_model(_lib.NET_LINEAR, tr.dim, _lib.make_table(sd["user.weight"], lin=sd["user_bias.weight"]),
                            _lib.make_table(sd["item.weight"], lin=sd["item_bias.weight"]), [])
    return model, sd


def main():
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    U, I, D, B = 3001, 1777, 64, 512
    rng = np.random.default_rng(5)                         # same seed on every rank: the global epoch is identical
    full = {"user.weight": rng.normal(0, .5, (U, D)).astype(np.float32),
            "item.weight": rng.normal(0, .5, (I, D)).astype(np.float32),
            "user_bias.weight": rng.normal(0, .1, (U, 1)).astype(np.float32),
            "item_bias.weight": rng.normal(0, .1, (I, 1)).astype(np.float32)}
    tr = S.ShardedLinearTrainer(U, I, D, global_batch=B, optimizer="sparse_adam", lr=0.05, device=dev)
    tr.load_state_dict({k: torch.from_numpy(v) for k, v in full.items()})
    epoch = lambda n: [torch.from_numpy(rng.integers(0, m, n)).to(dev) for m in (U, I, I)]
    users = torch.arange(0, U, 5, device=dev)
    for rnd in range(3):
        tr.train_epoch(*epoch(4 * B), B)                   # serving reads, then the owners update again
        model, keep = gathered(tr)
        for n, bs in ((20 * B - 11, B), (B // 2, B), (3 * B, 64)):
            user, pos, neg = epoch(n)
            got = tr.eval_pairwise(user, pos, neg, bs, want_scores=True)
            want = _lib.eval_pairwise(model, _lib.make_epoch(user, pos, neg, None, None, bs), want_scores=True)
            for name, g, w in zip(("loss", "auc", "pos", "neg"), got, want):
                assert torch.equal(g, w), (rnd, n, bs, name)
            m = tr.evaluate(user, pos, neg, bs, eval_metrics=("loss", "auc", "roc_auc"))
            assert m["loss"] == float(want[0].mean().item()) and m["auc"] == float(want[1].mean().item()), (rnd, m)
        for k in (1, 10, 100, 128):
            idx, score = tr.predict_topk(users, k)
            w_idx, w_score = want_topk(model, users, k)
            assert torch.equal(idx, w_idx) and torch.equal(score, w_score), (rnd, k)
        ex_user = rng.integers(0, U, 20000)               # ~7 excluded items per user, duplicates included
        ex_item = rng.integers(0, I, ex_user.size)
        codes = torch.from_numpy(np.unique(ex_user * I + ex_item)).to(dev)
        items = torch.arange(I, device=dev)
        for k in (10, 100, 1000):                          # tensor-core path, then the exact kernel
            for exact in (False, True):
                idx, score = tr.recommend(users, k, exclude=(ex_user, ex_item), _force_exact=exact)
                for q, u in enumerate(users[:64].tolist()):
                    s, o = torch.sort(_lib.scores(model, torch.full_like(items, u), items), descending=True, stable=True)
                    keep_ = ~torch.isin(u * I + o, codes)
                    o, s = o[keep_][:k], s[keep_][:k]
                    m = o.numel()
                    assert torch.equal(idx[q, :m], o) and torch.equal(score[q, :m], s), (rnd, k, exact, u)
                    assert bool((idx[q, m:] == -1).all()), (rnd, k, exact, u)
        ids = torch.from_numpy(rng.integers(0, U, 1000)).to(dev)
        emb, bias = tr.lookup("user", ids)
        assert torch.equal(emb, keep["user.weight"][ids]) and torch.equal(bias, keep["user_bias.weight"][ids])
    tr.close()
    dist.barrier()
    if rank == 0:
        print("SHARD SERVE CHECK OK", world, "ranks")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
