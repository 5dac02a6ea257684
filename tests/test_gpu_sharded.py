"""The multi-GPU paths on one B200 (``-m gpu``): the merge of sorted top-k lists against a stable sort in torch, and,
when the box has >= 2 GPUs, the row-sharded trainer and the item-sharded predict over NCCL against the numpy oracle's
single-process results on the global batch."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def test_sorted_merge_orders_by_score_then_lower_id(dev):
    """trs_shard_topk_merge_sorted on lists sorted by (score desc, id asc), as every caller passes them."""
    from torchrecsys_b200 import _lib
    g = torch.Generator().manual_seed(0)
    G_, Q, k = 8, 37, 100
    score = (torch.randn((G_, Q, k), generator=g) * 2).round() / 2      # heavy ties
    idx = torch.stack([torch.randperm(1000, generator=g)[:G_ * k].view(G_, k) for _ in range(Q)], 1)
    idx[3, :, 90:] = -1                                                   # a shard with only 90 items
    score[3, :, 90:] = float("-inf")
    o = torch.argsort(idx, dim=2, stable=True)                            # each list by (score desc, id asc),
    score, idx = score.gather(2, o), idx.gather(2, o)                     # its padding last
    o = torch.sort(score, dim=2, descending=True, stable=True)[1]
    score, idx = score.gather(2, o), idx.gather(2, o)
    out_idx, out_score = _lib.topk_merge_sorted(score.to(dev).contiguous(), idx.to(dev).contiguous(), k)
    s2, i2 = score.permute(1, 0, 2).reshape(Q, -1), idx.permute(1, 0, 2).reshape(Q, -1)
    s2 = torch.where(i2 < 0, torch.full_like(s2, float("-inf")), s2)
    big = torch.where(i2 < 0, torch.full_like(i2, 1 << 40), i2)
    o = torch.argsort(big, dim=1, stable=True)
    s2, i2 = s2.gather(1, o), i2.gather(1, o)
    o = torch.sort(s2, dim=1, descending=True, stable=True)[1][:, :k]
    assert torch.equal(out_idx.cpu(), i2.gather(1, o))
    assert torch.equal(out_score.cpu(), s2.gather(1, o))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_row_sharded_training_over_nccl_matches_the_oracle():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    n = min(torch.cuda.device_count(), 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tools", "sharded_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SHARDED CHECK OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
