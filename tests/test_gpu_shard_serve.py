"""Evaluation, prediction and row lookups on the row-sharded tables where they live (csrc/shard_serve.cu,
ShardedLinearTrainer.eval_pairwise / evaluate / predict_topk / lookup), on ONE B200 (``-m gpu``): the group is emulated
in one process (``emulate_world``), so every "peer" row is read through the same trs_shard pointers a real group maps.

Oracle: the single-GPU functions (trs_eval_pairwise, trs_predict_topk, trs_scores) on the gathered model, compared
bit for bit (``torch.equal``)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _skewed(rng, n_rows, n):
    hot = rng.integers(0, 3, n)
    warm = rng.integers(0, min(n_rows, 64), n)
    cold = rng.integers(0, n_rows, n)
    pick = rng.random(n)
    return np.where(pick < 0.10, hot, np.where(pick < 0.35, warm, cold)).astype(np.int64)


def _ids(rng, kind, n_rows, n):
    return rng.integers(0, n_rows, n, dtype=np.int64) if kind == "uniform" else _skewed(rng, n_rows, n)


def _to(dev, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _trained(dev, world, U, I, D, seed, ids="uniform", steps=3, B=256):
    """A trainer whose tables went through a few SparseAdam steps (biases included), not the initial ones."""
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    rng = np.random.default_rng(seed)
    tr = ShardedLinearTrainer(U, I, D, global_batch=B, optimizer="sparse_adam", lr=0.05, device=dev,
                              emulate_world=world, timeout_ms=5000)
    tr.load_state_dict({"user.weight": torch.from_numpy(rng.normal(0, .4, (U, D)).astype(np.float32)),
                        "item.weight": torch.from_numpy(rng.normal(0, .4, (I, D)).astype(np.float32)),
                        "user_bias.weight": torch.from_numpy(rng.normal(0, .1, (U, 1)).astype(np.float32)),
                        "item_bias.weight": torch.from_numpy(rng.normal(0, .1, (I, 1)).astype(np.float32))})
    n = steps * B
    tr.train_epoch(*(_to(dev, _ids(rng, ids, m, n)) for m in (U, I, I)), B)
    return tr


def _gathered(tr):
    """(trs_model of the gathered tables, the tensors it points into -- keep them alive)."""
    from torchrecsys_b200 import _lib
    sd = tr.state_dict()
    model = _lib.make_model(_lib.NET_LINEAR, tr.dim, _lib.make_table(sd["user.weight"], lin=sd["user_bias.weight"]),
                            _lib.make_table(sd["item.weight"], lin=sd["item_bias.weight"]), [])
    return model, sd


def _want_topk(model, users, k):
    """trs_predict_topk on the gathered model; users it flags as overflowing ranked as TorchRecSys does: trs_scores
    over every item and a stable descending sort."""
    from torchrecsys_b200 import _lib
    idx, score, over = _lib.predict_topk(model, users, k)
    items = torch.arange(model.item.n_rows, device=users.device)
    for q in torch.nonzero(over).flatten().tolist():
        s, order = torch.sort(_lib.scores(model, torch.full_like(items, int(users[q])), items), descending=True,
                              stable=True)
        m = min(k, items.numel())
        idx[q, :m], score[q, :m] = order[:m], s[:m]
    return idx, score


def _eval_equal(tr, user, pos, neg, B):
    from torchrecsys_b200 import _lib
    got = tr.eval_pairwise(user, pos, neg, B, want_scores=True)
    model, _keep = _gathered(tr)
    want = _lib.eval_pairwise(model, _lib.make_epoch(user, pos, neg, None, None, B), want_scores=True)
    for name, g, w in zip(("loss", "auc", "pos", "neg"), got, want):
        assert g.shape == w.shape and torch.equal(g, w), name


# every row shape of pick_row_shape at a multiple of 4 -- (G lanes, IT chunks) = (4,1) at 4 and 12 (partial), (8,1) at 20
# (partial), (16,1) at 36 (partial) and 64, (32,1) at 100 (partial) and 128, (32,2) at 132 (partial), (32,4) at 260
# (partial) and 512
_DIMS = (4, 12, 20, 36, 64, 100, 128, 132, 260, 512)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("dim", _DIMS)
def test_eval_pairwise_equals_the_gathered_model(dev, world, dim):
    """Uniform ids on half of the (world, dim) grid, skewed ids on the other half; a ragged last batch."""
    U, I, B = 3001, 701, 512
    ids = "skewed" if (dim // 4 + world) % 2 else "uniform"
    tr = _trained(dev, world, U, I, dim, seed=dim * 10 + world, ids=ids)
    rng = np.random.default_rng(dim + world)
    n = 9 * B - 37
    user, pos, neg = (_to(dev, _ids(rng, ids, m, n)) for m in (U, I, I))
    _eval_equal(tr, user, pos, neg, B)


@pytest.mark.parametrize("world", [3, 8])
@pytest.mark.parametrize("n,B", [(100, 512), (512, 512), (3 * 512 - 5, 512), (7 * 64 + 1, 64)])
def test_eval_pairwise_batch_splits(dev, world, n, B):
    """One batch in all, fewer batches than ranks (ranks with an empty range), a last batch of one sample."""
    tr = _trained(dev, world, 1000, 300, 64, seed=n + world)
    rng = np.random.default_rng(n)
    user, pos, neg = (_to(dev, rng.integers(0, m, n)) for m in (1000, 300, 300))
    _eval_equal(tr, user, pos, neg, B)
    loss, auc, p, q = tr.eval_pairwise(user, pos, neg, B)
    assert loss.shape == (-(-n // B),) and p is None and q is None


def test_torchrecsys_fit_then_evaluate_and_predict_on_three_ranks(dev):
    """A fitted TorchRecSys(net_type='linear') moved onto 3 ranks evaluates and predicts exactly as the model does."""
    import contextlib
    import io
    import pandas as pd
    from torchrecsys_b200.model import TorchRecSys
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    rng = np.random.default_rng(7)
    n_u, n_i, n_int, D, B = 400, 150, 8000, 16, 256
    df = pd.DataFrame({"user": np.r_[np.arange(n_u), rng.integers(0, n_u, n_int - n_u)],
                       "item": np.r_[np.arange(n_i), rng.integers(0, n_i, n_int - n_i)]})
    torch.manual_seed(3)
    metrics = ["loss", "auc", "roc_auc"]
    with contextlib.redirect_stdout(io.StringIO()):
        model = TorchRecSys(df, "user", "item", n_factors=D, net_type="linear", dynamic_neg_sampling=True,
                            use_cuda=True)
        opt = torch.optim.SparseAdam(list(model.parameters()), lr=1e-2)
        model.fit(opt, epochs=1, batch_size=B)
        model.evaluate(batch_size=B, eval_metrics=metrics)
    test = model._device_split("test_data")
    test = model._with_negatives(test, (1 << 40) + model._epochs_seen * test["user"].shape[0])
    tr = ShardedLinearTrainer.from_model(model.net, opt, B, device=dev, emulate_world=3)
    got = tr.evaluate(test["user"], test["pos"], test["neg"], batch_size=B, eval_metrics=metrics + ["mrr"])
    assert got == dict(model.last_eval, mrr=0)
    users = torch.arange(0, n_u, 3)
    idx, score = tr.predict_topk(users, 10)
    assert torch.equal(idx.cpu(), model.predict_batch(users, 10))


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("dim", [16, 64, 128, 200])
def test_predict_topk_equals_the_gathered_model(dev, world, dim):
    from torchrecsys_b200 import _lib
    U, I = 2000, 1500
    tr = _trained(dev, world, U, I, dim, seed=dim + 100 * world, ids="skewed")
    model, _keep = _gathered(tr)
    users = _to(dev, np.r_[np.arange(0, U, 7), [U - 1, 0, 0]])
    for k in (1, 10, 100, 128):
        idx, score = tr.predict_topk(users, k)
        w_idx, w_score = _want_topk(model, users, k)
        assert torch.equal(idx, w_idx) and torch.equal(score, w_score), k


@pytest.mark.parametrize("world,n_items", [(8, 37), (3, 130), (8, 700)])
def test_predict_topk_small_shards_and_catalogues(dev, world, n_items):
    """Shards with fewer than k items; a catalogue smaller than k gives [Q, n_items]."""
    from torchrecsys_b200 import _lib
    tr = _trained(dev, world, 500, n_items, 32, seed=n_items)
    model, _keep = _gathered(tr)
    users = torch.arange(500, device=dev)
    for k in (5, 100, 128):
        idx, score = tr.predict_topk(users, k)
        kk = min(k, n_items)
        w_idx, w_score = _want_topk(model, users, k)
        assert idx.shape == (500, kk)
        assert torch.equal(idx, w_idx[:, :kk]) and torch.equal(score, w_score[:, :kk]), k
        assert bool((idx >= 0).all())


def test_predict_topk_ties_across_owners_prefer_the_lower_id(dev):
    """Items 3j .. 3j+2 share one row and bias and live on three different owners: ties everywhere, lower id first."""
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    U, I, D = 300, 900, 32
    rng = np.random.default_rng(4)
    item = np.repeat(rng.normal(0, .5, (I // 3, D)).astype(np.float32), 3, axis=0)
    bias = np.repeat(rng.normal(0, .1, (I // 3, 1)).astype(np.float32), 3, axis=0)
    params = {"user.weight": torch.from_numpy(rng.normal(0, .5, (U, D)).astype(np.float32)),
              "user_bias.weight": torch.zeros(U, 1), "item.weight": torch.from_numpy(item),
              "item_bias.weight": torch.from_numpy(bias)}
    tr = ShardedLinearTrainer(U, I, D, global_batch=64, device=dev, emulate_world=3)
    tr.load_state_dict(params)
    model, _keep = _gathered(tr)
    users = torch.arange(U, device=dev)
    idx, score = tr.predict_topk(users, 30)
    w_idx, w_score = _want_topk(model, users, 30)
    assert torch.equal(idx, w_idx) and torch.equal(score, w_score)
    assert torch.equal(idx[:, 0] % 3, torch.zeros_like(idx[:, 0]))
    assert torch.equal(idx[:, 1], idx[:, 0] + 1) and torch.equal(idx[:, 2], idx[:, 0] + 2)


def test_predict_topk_overflow_ranks_exactly(dev):
    """Every item row and bias equal: each user's candidates overflow, and the exact path gives the stable sort."""
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    U, I, D, k = 64, 3000, 16, 50
    rng = np.random.default_rng(8)
    params = {"user.weight": torch.from_numpy(rng.normal(0, .5, (U, D)).astype(np.float32)),
              "user_bias.weight": torch.from_numpy(rng.normal(0, .1, (U, 1)).astype(np.float32)),
              "item.weight": torch.from_numpy(np.tile(rng.normal(0, .5, (1, D)).astype(np.float32), (I, 1))),
              "item_bias.weight": torch.full((I, 1), 0.25)}
    tr = ShardedLinearTrainer(U, I, D, global_batch=64, device=dev, emulate_world=3)
    tr.load_state_dict(params)
    users = torch.arange(0, U, 5, device=dev)
    idx, score = tr.predict_topk(users, k)
    assert tr.last_predict_overflow > 0
    model, _keep = _gathered(tr)
    items = torch.arange(I, device=dev)
    for q, u in enumerate(users.tolist()):
        s = _lib.scores(model, torch.full_like(items, u), items)
        w_score, w_idx = torch.sort(s, descending=True, stable=True)
        assert torch.equal(idx[q], w_idx[:k]) and torch.equal(score[q], w_score[:k]), u


def test_predict_after_training_and_loading_sees_the_new_tables(dev):
    """The prepared item operand is reused only while the tables are unchanged: a training step or a load rebuilds it."""
    from torchrecsys_b200 import _lib
    U, I, D, B = 1000, 800, 64, 256
    tr = _trained(dev, 3, U, I, D, seed=5)
    users = torch.arange(0, U, 3, device=dev)

    def check():
        model, _keep = _gathered(tr)
        w_idx, w_score = _want_topk(model, users, 20)
        idx, score = tr.predict_topk(users, 20)
        assert torch.equal(idx, w_idx) and torch.equal(score, w_score)
        return idx

    first = check()
    assert torch.equal(check(), first)          # unchanged: the cached operand
    rng = np.random.default_rng(6)
    tr.train_epoch(*(_to(dev, rng.integers(0, m, B)) for m in (U, I, I)), B)
    check()
    sd = tr.state_dict()
    sd["item.weight"] = sd["item.weight"].flip(0).contiguous()
    tr.load_state_dict(sd)
    assert not torch.equal(check(), first)


def test_lookup_and_argument_errors(dev):
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    U, I = 1000, 300
    tr = _trained(dev, 3, U, I, 32, seed=9)
    sd = tr.state_dict()
    ids = torch.tensor([0, 1, 2, 999, 500, 500, 3], device=dev)
    for name, n in (("user", U), ("item", I)):
        emb, bias = tr.lookup(name, ids % n)
        assert torch.equal(emb, sd[f"{name}.weight"][ids % n]) and torch.equal(bias, sd[f"{name}_bias.weight"][ids % n])
        with pytest.raises(IndexError):
            tr.lookup(name, [n])
        with pytest.raises(IndexError):
            tr.lookup(name, [-1])
    e, b = tr.lookup("item", torch.empty(0, dtype=torch.int64))
    assert e.shape == (0, 32) and b.shape == (0, 1)
    with pytest.raises(IndexError):
        tr.predict_topk([U], 10)
    for k in (0, 129):
        with pytest.raises(ValueError):
            tr.predict_topk([0], k)
    wide = ShardedLinearTrainer(100, 50, 240, global_batch=16, device=dev, emulate_world=2)
    with pytest.raises(ValueError):
        wide.predict_topk([0], 10)


def _free_gib():
    free, _ = torch.cuda.mem_get_info()
    return free / 2 ** 30


@pytest.mark.parametrize("world", [1, 3])
def test_benchmark_tables(dev, world):
    """50M x 5M at D = 128 with SGD (bench.py's tables): at one rank the user shard holds more than 2^32 floats.
    Compared with the single-GPU kernels on tables compacted by indexing the shard tensors in torch."""
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    if _free_gib() < 30:
        pytest.skip(f"needs about 30 GiB of free device memory, {_free_gib():.1f} GiB free")
    U, I, D, n, B = 50_000_000, 5_000_000, 128, 65536, 512
    tr = ShardedLinearTrainer(U, I, D, global_batch=B, optimizer="sgd", lr=0.05, device=dev, emulate_world=world)
    for r in tr.local_ranks:                                   # non-zero biases
        for name in ("user", "item"):
            tr.tables[r][name][1].normal_(0, .1)
    rng = np.random.default_rng(world)
    user = _to(dev, np.r_[rng.integers(0, U, n - 2), [U - 1, U - 2]])
    pos, neg = (_to(dev, rng.integers(0, I, n)) for _ in range(2))

    def compact(name, ids):
        uniq, inv = torch.unique(ids, return_inverse=True)
        emb = torch.empty((uniq.numel(), D), device=dev)
        lin = torch.empty((uniq.numel(), 1), device=dev)
        for r in tr.local_ranks:
            sel = uniq % world == r
            e, b = tr.tables[r][name]
            emb[sel], lin[sel] = e[uniq[sel] // world], b[uniq[sel] // world]
        return emb, lin, inv

    ue, ul, uinv = compact("user", user)
    ie, il, iinv = compact("item", torch.cat([pos, neg]))
    model = _lib.make_model(_lib.NET_LINEAR, D, _lib.make_table(ue, lin=ul), _lib.make_table(ie, lin=il), [])
    pinv, ninv = iinv[:n].contiguous(), iinv[n:].contiguous()
    want = _lib.eval_pairwise(model, _lib.make_epoch(uinv, pinv, ninv, None, None, B), want_scores=True)
    got = tr.eval_pairwise(user, pos, neg, B, want_scores=True)
    for name, g, w in zip(("loss", "auc", "pos", "neg"), got, want):
        assert torch.equal(g, w), name
    del ie, il, model

    q_users = user[:256]
    qe, ql = ue[uinv[:256]], ul[uinv[:256]]
    if world == 1:
        item_emb, item_lin = tr.tables[0]["item"]
    else:
        item_emb, item_lin = torch.empty((I, D), device=dev), torch.empty((I, 1), device=dev)
        for r in tr.local_ranks:
            item_emb[r::world], item_lin[r::world] = tr.tables[r]["item"]
    model = _lib.make_model(_lib.NET_LINEAR, D, _lib.make_table(qe, lin=ql), _lib.make_table(item_emb, lin=item_lin), [])
    w_idx, w_score = _want_topk(model, torch.arange(256, device=dev), 100)
    idx, score = tr.predict_topk(q_users, 100)
    assert torch.equal(idx, w_idx) and torch.equal(score, w_score)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_serving_over_real_peers_matches_the_gathered_model():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    n = min(torch.cuda.device_count(), 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tools", "shard_serve_check.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SHARD SERVE CHECK OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
