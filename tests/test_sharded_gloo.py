"""Host logic of the item-sharded predict (torchrecsys_b200/sharded.py: sharded_predict_topk) on the CPU: world size
2, gloo, with torch stand-ins for the local top-k and the list merge.  Checks that the all_to_all merger returns the
global stable top-k."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

U, I, D, WORLD = 41, 29, 8, 2


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        from torchrecsys_b200 import sharded as S
        torch.set_num_threads(1)
        rng = np.random.default_rng(7)
        user_w = rng.normal(0, .5, (U, D)).astype(np.float32)
        item_w = rng.normal(0, .5, (I, D)).astype(np.float32)
        item_b = rng.normal(0, .1, (I, 1)).astype(np.float32)
        # item-sharded predict: local top-k on a contiguous block, each user's lists to one merger rank, merge, all-gather
        k = 7
        scores_full = torch.from_numpy(user_w[:5] @ item_w.T + item_b.T)
        scores_full = (scores_full * 4).round() / 4  # force ties

        def local_topk(users, kk, offset):
            lo, hi = S.item_block(I, rank, WORLD)
            v, o = torch.sort(scores_full[users, lo:hi], dim=1, descending=True, stable=True)
            return (o[:, :kk] + offset).contiguous(), v[:, :kk].contiguous()

        def merge(sc, ix, kk):  # torch stand-in of trs_shard_topk_merge_sorted: (score desc, id asc)
            Q = sc.shape[1]
            s2, i2 = sc.permute(1, 0, 2).reshape(Q, -1), ix.permute(1, 0, 2).reshape(Q, -1)
            o = torch.argsort(i2, dim=1, stable=True)
            s2, i2 = s2.gather(1, o), i2.gather(1, o)
            o = torch.sort(s2, dim=1, descending=True, stable=True)[1]
            return i2.gather(1, o)[:, :kk], s2.gather(1, o)[:, :kk]

        idx, _ = S.sharded_predict_topk(local_topk, torch.arange(5), k, I, merge=merge)
        want = torch.sort(scores_full, dim=1, descending=True, stable=True)[1][:, :k]
        assert torch.equal(idx, want)
        q.put((rank, "ok"))
    except Exception as e:  # surface the failure in the parent
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_item_sharded_predict_merge_world_size_2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, port, q)) for r in range(WORLD)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, msg in results:
        assert msg == "ok", f"rank {rank}:\n{msg}"
