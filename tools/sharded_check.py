"""torchrun worker: the row-sharded Linear trainer over REAL peers (CUDA-IPC mapped shards, NVLink loads / stores,
flag barriers; torchrecsys_b200/sharded.py + csrc/shard.cu) and the item-sharded predict over NCCL -- each against
the numpy oracle's single-process results on the global batch.
Prints SHARDED CHECK OK on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import cf_oracle as O  # noqa: E402
from torchrecsys_b200 import _lib, sharded as S  # noqa: E402
from torchrecsys_b200.collaborative.linear import Linear  # noqa: E402


def main():
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    U, I, D, B, steps = 3001, 1777, 64, 512, 4
    rng = np.random.default_rng(5)
    full = {"user.weight": rng.normal(0, .5, (U, D)).astype(np.float32),
            "item.weight": rng.normal(0, .5, (I, D)).astype(np.float32),
            "user_bias.weight": np.zeros((U, 1), np.float32),
            "item_bias.weight": rng.normal(0, .1, (I, 1)).astype(np.float32)}
    for kind, tol in (("sgd", 2e-6), ("adagrad", 2e-5), ("sparse_adam", 2e-4)):
        spec = O.OptSpec(kind, lr=0.05)
        # ---- the product path: peer-mapped shards, one persistent kernel per rank ----
        tr = S.ShardedLinearTrainer(U, I, D, global_batch=world * B, optimizer=kind, lr=0.05, device=dev)
        tr.load_state_dict({k: torch.from_numpy(v) for k, v in full.items()})
        params = {k: v.copy() for k, v in full.items()}
        state = O.init_opt_state(params, spec)
        brng = np.random.default_rng(11)
        batches = [{k: brng.integers(0, n, world * B) for k, n in (("user", U), ("pos", I), ("neg", I))}
                   for _ in range(steps)]
        glob = {k: torch.from_numpy(np.concatenate([b[k] for b in batches])).to(dev) for k in ("user", "pos", "neg")}
        loss = tr.train_epoch(glob["user"], glob["pos"], glob["neg"], world * B).cpu().numpy()
        want = [O.train_step("linear", params, state, b, spec, s + 1) for s, b in enumerate(batches)]
        np.testing.assert_allclose(loss, np.array(want), rtol=1e-4, atol=1e-5, err_msg=f"peer-mapped {kind} loss")
        sd = tr.state_dict()
        for k in params:
            np.testing.assert_allclose(sd[k].cpu().numpy(), params[k], rtol=1e-4, atol=tol, err_msg=f"peer-mapped {kind} {k}")
        # one more step through the per-rank convenience entry (all-gathers the ranks' samples)
        b = {k: brng.integers(0, n, world * B) for k, n in (("user", U), ("pos", I), ("neg", I))}
        sl = slice(rank * B, (rank + 1) * B)
        l1 = tr.train_step(*(torch.from_numpy(b[k][sl]).to(dev) for k in ("user", "pos", "neg")))
        w1 = O.train_step("linear", params, state, b, spec, steps + 1)
        assert abs(float(l1) - float(w1)) < 1e-4, (kind, float(l1), float(w1))
        tr.close()
    # item-sharded predict: each rank holds a contiguous item block of the (replicated-user) Linear model
    k, Q = 50, 200
    lo, hi = S.item_block(I, rank, world)
    net = Linear(U, hi - lo, {}, D, use_metadata=False, use_cuda=True)
    net.load_state_dict({"user.weight": torch.from_numpy(params["user.weight"]),
                         "user_bias.weight": torch.from_numpy(params["user_bias.weight"]),
                         "item.weight": torch.from_numpy(params["item.weight"][lo:hi]),
                         "item_bias.weight": torch.from_numpy(params["item_bias.weight"][lo:hi])})
    net = net.to(dev).eval()
    users = torch.arange(Q, device=dev)

    def local_topk(u, kk, offset):
        idx, score, over = _lib.predict_topk(net.abi_model(), u, kk, item_offset=offset)
        assert int(over.sum()) == 0
        return idx, score

    idx, score = S.sharded_predict_topk(local_topk, users, k, I)
    for u in (0, 57, 199):
        np.testing.assert_array_equal(idx[u].cpu().numpy(), O.predict_topk("linear", params, u, k))
    dist.barrier()
    if rank == 0:
        print("SHARDED CHECK OK", world, "ranks")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
