"""The multi-GPU building blocks on one B200 (``-m gpu``): owner-side coalesce + row update, the Linear step on
gathered rows, the top-k list merge -- each against the numpy oracle -- and, when the box has >= 2 GPUs, the
row-sharded trainer over NCCL against the oracle's single-process step on the global batch."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import cf_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.mark.parametrize("kind", ["sgd", "adagrad", "sparse_adam"])
@pytest.mark.parametrize("dim", [16, 64, 128, 6])
def test_sparse_row_update_matches_coalesce_then_optimizer(dev, kind, dim):
    from torchrecsys_b200 import _lib
    rng = np.random.default_rng(dim)
    n_rows, n = 500, 3000  # many duplicates, some rows hit 20+ times
    p = rng.normal(0, .3, (n_rows, dim)).astype(np.float32)
    b = rng.normal(0, .3, (n_rows, 1)).astype(np.float32)
    ids = np.concatenate([rng.integers(0, n_rows, n - 200), rng.integers(0, 5, 200)])
    g = rng.normal(0, 1, (n, dim)).astype(np.float32)
    gb = rng.normal(0, 1, (n, 1)).astype(np.float32)
    spec = O.OptSpec(kind, lr=0.05)
    step = 3
    params = {"e": p.copy(), "b": b.copy()}
    state = O.init_opt_state(params, spec)
    for k in state:
        for s in state[k].values():
            s += rng.random(s.shape).astype(np.float32) * 0.1   # non-trivial optimizer state
    state0 = {k: {n_: v.copy() for n_, v in st.items()} for k, st in state.items()}
    for name, vals in (("e", g), ("b", gb)):
        rows, gs = O.coalesce(ids, vals)
        O.apply_rows(params[name], state[name], rows, gs, spec, step)
    t = lambda a: torch.from_numpy(a).to(dev).contiguous()
    names = {"adagrad": ["sum"], "sparse_adam": ["exp_avg", "exp_avg_sq"], "sgd": []}[kind]
    emb, bias = t(p), t(b)
    es = [t(state0["e"][k]) for k in names] + [None, None]
    bs = [t(state0["b"][k]) for k in names] + [None, None]
    table = _lib.make_table(emb, es[0], es[1], bias, bs[0], bs[1])
    scale = {"sgd": spec.lr, "adagrad": O.adagrad_clr(spec, step), "sparse_adam": O.adam_step_size(spec, step)}[kind]
    scales = torch.tensor([0.0, 0.0, scale], dtype=torch.float64).float().to(dev)
    optim = _lib.Optim({"sgd": 0, "adagrad": 1, "sparse_adam": 2}[kind], 0, 0.9, 0.999, spec.eps, scales.data_ptr())
    _lib.sparse_row_update(table, dim, t(ids), t(g), t(gb[:, 0]), optim, 2)
    torch.cuda.synchronize()
    np.testing.assert_allclose(emb.cpu().numpy(), params["e"], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(bias.cpu().numpy(), params["b"], rtol=1e-5, atol=2e-6)
    for i, k in enumerate(names):
        np.testing.assert_allclose(es[i].cpu().numpy(), state["e"][k], rtol=1e-5, atol=2e-6)
    untouched = np.setdiff1d(np.arange(n_rows), ids)
    assert np.array_equal(emb.cpu().numpy()[untouched], p[untouched])


@pytest.mark.parametrize("dim", [16, 128, 80])
def test_linear_rows_step_matches_oracle_gradients(dev, dim):
    from torchrecsys_b200 import _lib
    rng = np.random.default_rng(3)
    U, I, B = 50, 40, 777
    params = {"user.weight": rng.normal(0, .5, (U, dim)).astype(np.float32),
              "item.weight": rng.normal(0, .5, (I, dim)).astype(np.float32),
              "user_bias.weight": rng.normal(0, .1, (U, 1)).astype(np.float32),
              "item_bias.weight": rng.normal(0, .1, (I, 1)).astype(np.float32)}
    batch = {"user": rng.integers(0, U, B), "pos": rng.integers(0, I, B), "neg": rng.integers(0, I, B)}
    loss, grads = O.linear_grads(params, batch)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    u, vp, vn = (t(params[k][batch[b]]) for k, b in (("user.weight", "user"), ("item.weight", "pos"), ("item.weight", "neg")))
    bu, bp, bn = (t(params[k][batch[b]][:, 0]) for k, b in (("user_bias.weight", "user"), ("item_bias.weight", "pos"),
                                                            ("item_bias.weight", "neg")))
    g_u, g_vp, g_vn, g_bp, g_bn, hsum = _lib.linear_rows_step(u, vp, vn, bu, bp, bn, 1.0 / B)
    assert abs(float(hsum) / B - float(loss)) < 1e-5
    gi = grads["item.weight"][1]
    gu = grads["user.weight"][1]
    np.testing.assert_allclose(g_vp.cpu().numpy(), gi[:B], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(g_vn.cpu().numpy(), gi[B:], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(g_u.cpu().numpy(), gu[:B] + gu[B:], rtol=1e-5, atol=1e-7)
    gb = grads["item_bias.weight"][1][:, 0]
    np.testing.assert_array_equal(g_bp.cpu().numpy(), gb[:B])
    np.testing.assert_array_equal(g_bn.cpu().numpy(), gb[B:])


def test_topk_merge_orders_by_score_then_lower_id(dev):
    from torchrecsys_b200 import _lib
    g = torch.Generator().manual_seed(0)
    G_, Q, k = 8, 37, 100
    score = (torch.randn((G_, Q, k), generator=g) * 2).round() / 2      # heavy ties
    idx = torch.stack([torch.randperm(1000, generator=g)[:G_ * k].view(G_, k) for _ in range(Q)], 1)
    idx[3, :, 90:] = -1                                                   # a shard with only 90 items
    score[3, :, 90:] = float("-inf")
    out_idx, out_score = _lib.topk_merge(score.to(dev).contiguous(), idx.to(dev).contiguous(), k)
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
