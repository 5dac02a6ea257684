"""ShardedLinearTrainer.recommend (csrc/shard_topk.cu: trs_shard_topk_exact / trs_shard_topk_merge_sorted) on ONE B200
(``-m gpu``): the group is emulated in one process (``emulate_world``).

Oracle: trs_scores on the gathered model over every item, a stable descending sort, the excluded items dropped, the
first k, -1 / -inf padding -- compared bit for bit (``torch.equal``)."""
import numpy as np
import pytest
import torch

from tests.test_gpu_shard_serve import _DIMS, _free_gib, _gathered, _ids, _to, _trained

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _oracle(model, users, k, excluded=None):
    """(idx [Q, k], score [Q, k]) ranked as TorchRecSys does; ``excluded[q]`` a set of item ids left out of row q.
    ``users`` index model.user."""
    from torchrecsys_b200 import _lib
    I = model.item.n_rows
    dev = users.device
    Q = users.numel()
    idx = torch.full((Q, k), -1, dtype=torch.int64, device=dev)
    score = torch.full((Q, k), float("-inf"), device=dev)
    items = torch.arange(I, device=dev)
    for q0 in range(0, Q, 64):
        uq = users[q0:q0 + 64]
        s = _lib.scores(model, uq.repeat_interleave(I), items.repeat(uq.numel())).view(uq.numel(), I)
        s, order = torch.sort(s, dim=1, descending=True, stable=True)
        for j in range(uq.numel()):
            q = q0 + j
            o, v = order[j], s[j]
            if excluded is not None and excluded[q]:
                keep = ~torch.isin(o, torch.tensor(sorted(excluded[q]), dtype=torch.int64, device=dev))
                o, v = o[keep], v[keep]
            m = min(k, o.numel())
            idx[q, :m], score[q, :m] = o[:m], v[:m]
    return idx, score


def _check(tr, model, users, k, exclude=None, excluded=None, paths=("tc", "exact")):
    kk = min(k, tr.n_items)
    w_idx, w_score = _oracle(model, users, k, excluded)
    outs = []
    for path in paths:
        idx, score = tr.recommend(users, k, exclude=exclude, _force_exact=path == "exact")
        assert idx.shape == (users.numel(), kk) and idx.dtype == torch.int64 and score.dtype == torch.float32
        assert torch.equal(idx, w_idx[:, :kk]) and torch.equal(score, w_score[:, :kk]), (path, k)
        outs.append((idx, score))
    return outs


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("dim", _DIMS)
def test_recommend_equals_the_gathered_model(dev, world, dim):
    """Every row shape; uniform ids on half of the grid, skewed on the other; k across the tensor-core and exact paths."""
    U, I = 900, 1500
    ids = "skewed" if (dim // 4 + world) % 2 else "uniform"
    tr = _trained(dev, world, U, I, dim, seed=dim * 7 + world, ids=ids)
    model, _keep = _gathered(tr)
    users = _to(dev, np.r_[np.arange(0, U, 37), [U - 1, 0, 0]])
    for k in (1, 100, 129, 1000, 1024):
        _check(tr, model, users, k, paths=("tc", "exact") if k <= 128 else ("tc",))


@pytest.mark.parametrize("world,n_items", [(8, 5), (8, 37), (3, 130), (2, 1100), (8, 3000)])
def test_recommend_small_shards_and_catalogues(dev, world, n_items):
    """Fewer items than ranks, shards and catalogues smaller than k: [Q, min(k, n_items)]."""
    tr = _trained(dev, world, 300, n_items, 32, seed=n_items + world)
    model, _keep = _gathered(tr)
    users = torch.arange(0, 300, 7, device=dev)
    for k in (3, 100, 500, 1024):
        _check(tr, model, users, k)


@pytest.mark.parametrize("world,dim", [(1, 64), (3, 128), (8, 200)])
def test_recommend_equals_predict_topk(dev, world, dim):
    tr = _trained(dev, world, 2000, 1500, dim, seed=world + dim, ids="skewed")
    users = _to(dev, np.r_[np.arange(0, 2000, 11), [1999, 0, 0]])
    for k in (1, 10, 100, 128):
        got, want = tr.recommend(users, k), tr.predict_topk(users, k)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), k


def _excluded_sets(users, ex_user, ex_item):
    by_user = {}
    for u, i in zip(ex_user.tolist(), ex_item.tolist()):
        by_user.setdefault(u, set()).add(i)
    return [by_user.get(u, set()) for u in users.tolist()]


@pytest.mark.parametrize("world", [1, 3, 8])
def test_recommend_excludes_pairs(dev, world):
    """Random pairs with duplicates and in any order, pairs of users not queried, a user queried twice; exclusions all
    on one owner; a user with every item excluded; a user left with exactly k - 1 items.  The tensor-core path (small
    k) and the exact kernel agree."""
    U, I, D = 400, 600, 48
    tr = _trained(dev, world, U, I, D, seed=11 * world)
    model, _keep = _gathered(tr)
    rng = np.random.default_rng(world)
    users = _to(dev, np.r_[[5, 17, 17, 250, 399, 0, 1, 2], np.arange(20, 400, 23)])
    k = 40
    ex_user = rng.integers(0, U - 1, 6000)
    ex_user = ex_user[ex_user != 250]   # 250 and 399 get exactly their own pairs below
    ex_item = rng.integers(0, I, ex_user.size)
    ex_user = np.r_[ex_user, ex_user[:500], np.full(I, 250), np.full(I - k + 1, 399), np.full(60, 17)]
    ex_item = np.r_[ex_item, ex_item[:500], np.arange(I), rng.permutation(I)[:I - k + 1],
                    (rng.integers(0, I // world, 60) * world)]   # user 17: extra items all on owner 0
    perm = rng.permutation(ex_user.size)
    ex_user, ex_item = ex_user[perm], ex_item[perm]
    excluded = _excluded_sets(users.cpu(), ex_user, ex_item)
    for kq in (k, 5, 300):
        outs = _check(tr, model, users, kq, exclude=(ex_user, ex_item), excluded=excluded)
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    idx, score = tr.recommend(users, k, exclude=(torch.from_numpy(ex_user), torch.from_numpy(ex_item)))
    q250, q399 = 3, 4
    assert bool((idx[q250] == -1).all()) and bool(torch.isinf(score[q250]).all())
    assert bool((idx[q399, :k - 1] >= 0).all()) and int(idx[q399, k - 1]) == -1


def test_recommend_exact_kernel_in_query_chunks(dev):
    """Queries split into several trs_shard_topk_exact calls (the exclusion CSR re-based per chunk) give the one-call
    result; the path taken is reported per rank."""
    U, I, D, world, k = 300, 700, 32, 3, 50
    tr = _trained(dev, world, U, I, D, seed=31)
    rng = np.random.default_rng(31)
    users = torch.arange(0, U, 2, device=dev)
    ex = (rng.integers(0, U, 3000), rng.integers(0, I, 3000))
    whole = tr.recommend(users, k, exclude=ex, _force_exact=True)
    assert tr.last_recommend_paths == {r: "exact" for r in range(world)}
    tr.EXACT_CHUNK = 7
    chunked = tr.recommend(users, k, exclude=ex, _force_exact=True)
    assert torch.equal(whole[0], chunked[0]) and torch.equal(whole[1], chunked[1])
    tr.recommend(users, 10)
    assert tr.last_recommend_paths == {r: "tensor core" for r in range(world)}


def test_recommend_small_k_tensor_core_path_with_exclusion(dev):
    """A few excluded items per user: k + excluded <= 128 takes the tensor-core path, which drops them in the merge."""
    U, I, D, world = 500, 2000, 64, 3
    tr = _trained(dev, world, U, I, D, seed=21)
    model, _keep = _gathered(tr)
    rng = np.random.default_rng(3)
    users = torch.arange(0, U, 4, device=dev)
    # each queried user's own current top 10 excluded: the over-request must reach past them
    top, _ = tr.recommend(users, 10)
    ex_user = users.repeat_interleave(10).cpu().numpy()
    ex_item = top.reshape(-1).cpu().numpy()
    ex_user = np.r_[ex_user, rng.integers(0, U, 300)]
    ex_item = np.r_[ex_item, rng.integers(0, I, 300)]
    excluded = _excluded_sets(users.cpu(), ex_user, ex_item)
    outs = _check(tr, model, users, 20, exclude=(ex_user, ex_item), excluded=excluded)
    assert torch.equal(outs[0][0], outs[1][0])


def test_recommend_fitted_torchrecsys_excludes_seen_items(dev):
    """A fitted TorchRecSys(net_type='linear') on 3 ranks: recommend(exclude=train pairs) == predict_batch(exclude_seen)."""
    import contextlib
    import io
    import pandas as pd
    from torchrecsys_b200.model import TorchRecSys
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    rng = np.random.default_rng(7)
    n_u, n_i, n_int, D, B = 400, 300, 12000, 16, 256
    df = pd.DataFrame({"user": np.r_[np.arange(n_u), rng.integers(0, n_u, n_int - n_u)],
                       "item": np.r_[np.arange(n_i), rng.integers(0, n_i, n_int - n_i)]})
    torch.manual_seed(3)
    with contextlib.redirect_stdout(io.StringIO()):
        model = TorchRecSys(df, "user", "item", n_factors=D, net_type="linear", dynamic_neg_sampling=True,
                            use_cuda=True)
        opt = torch.optim.SparseAdam(list(model.parameters()), lr=1e-2)
        model.fit(opt, epochs=1, batch_size=B)
    tr = ShardedLinearTrainer.from_model(model.net, opt, B, device=dev, emulate_world=3)
    users = torch.arange(0, n_u, 3)
    train = (model.data_processor.train_data["user_id"], model.data_processor.train_data["pos_item_id"])
    for k in (10, 200):
        idx, _ = tr.recommend(users, k, exclude=train)
        assert torch.equal(idx.cpu(), model.predict_batch(users, k, exclude_seen=True)), k


def test_recommend_ties_prefer_the_lower_id(dev):
    """Identical item rows and biases everywhere: every score ties, ids come out ascending across owners."""
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    U, I, D = 64, 3000, 16
    rng = np.random.default_rng(8)
    params = {"user.weight": torch.from_numpy(rng.normal(0, .5, (U, D)).astype(np.float32)),
              "user_bias.weight": torch.from_numpy(rng.normal(0, .1, (U, 1)).astype(np.float32)),
              "item.weight": torch.from_numpy(np.tile(rng.normal(0, .5, (1, D)).astype(np.float32), (I, 1))),
              "item_bias.weight": torch.full((I, 1), 0.25)}
    tr = ShardedLinearTrainer(U, I, D, global_batch=64, device=dev, emulate_world=3)
    tr.load_state_dict(params)
    model, _keep = _gathered(tr)
    users = torch.arange(0, U, 5, device=dev)
    for k in (50, 1000):
        idx, score = _check(tr, model, users, k)[0]
        assert torch.equal(idx, torch.arange(k, device=dev).expand_as(idx))


def test_recommend_sees_training_and_loading(dev):
    U, I, D, B = 1000, 800, 64, 256
    tr = _trained(dev, 3, U, I, D, seed=5)
    users = torch.arange(0, U, 3, device=dev)

    def check():
        model, _keep = _gathered(tr)
        return _check(tr, model, users, 20)[0][0]

    first = check()
    rng = np.random.default_rng(6)
    tr.train_epoch(*(_to(dev, rng.integers(0, m, B)) for m in (U, I, I)), B)
    check()
    sd = tr.state_dict()
    sd["item.weight"] = sd["item.weight"].flip(0).contiguous()
    tr.load_state_dict(sd)
    assert not torch.equal(check(), first)


def test_recommend_argument_errors(dev):
    U, I = 1000, 300
    tr = _trained(dev, 3, U, I, 32, seed=9)
    for k in (0, 1025):
        with pytest.raises(ValueError, match="1024"):
            tr.recommend([0], k)
    with pytest.raises(IndexError):
        tr.recommend([U], 10)
    with pytest.raises(IndexError):
        tr.recommend([0], 10, exclude=([U], [0]))
    with pytest.raises(IndexError):
        tr.recommend([0], 10, exclude=([0], [I]))
    with pytest.raises(ValueError):
        tr.recommend([0], 10, exclude=([0, 1], [0]))
    idx, score = tr.recommend(torch.empty(0, dtype=torch.int64), 10)
    assert idx.shape == (0, 10) and score.shape == (0, 10)


@pytest.mark.parametrize("world", [1, 3])
def test_recommend_benchmark_tables(dev, world):
    """50M x 5M at D = 128 with SGD: a few users at k = 1000 with exclusions.  The oracle takes the query users' rows
    from lookup() and only the item table gathered: the user table is never gathered."""
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    if _free_gib() < 40:
        pytest.skip(f"needs about 40 GiB of free device memory, {_free_gib():.1f} GiB free")
    U, I, D, k = 50_000_000, 5_000_000, 128, 1000
    tr = ShardedLinearTrainer(U, I, D, global_batch=512, optimizer="sgd", lr=0.05, device=dev, emulate_world=world)
    for r in tr.local_ranks:
        for name in ("user", "item"):
            tr.tables[r][name][1].normal_(0, .1)
    rng = np.random.default_rng(world)
    users = _to(dev, np.r_[rng.integers(0, U, 3), [U - 1]])
    ue, ul = tr.lookup("user", users)
    if world == 1:
        item_emb, item_lin = tr.tables[0]["item"]
    else:
        item_emb, item_lin = torch.empty((I, D), device=dev), torch.empty((I, 1), device=dev)
        for r in tr.local_ranks:
            item_emb[r::world], item_lin[r::world] = tr.tables[r]["item"]
    model = _lib.make_model(_lib.NET_LINEAR, D, _lib.make_table(ue, lin=ul), _lib.make_table(item_emb, lin=item_lin), [])
    want_plain, _ = _oracle(model, torch.arange(4, device=dev), 50)
    ex_user = np.r_[np.repeat(users.cpu().numpy(), 50), rng.integers(0, U, 1000)]
    ex_item = np.r_[want_plain.reshape(-1).cpu().numpy(), rng.integers(0, I, 1000)]   # each user's top 50
    excluded = _excluded_sets(users.cpu(), ex_user, ex_item)
    w_idx, w_score = _oracle(model, torch.arange(4, device=dev), k, excluded)
    idx, score = tr.recommend(users, k, exclude=(ex_user, ex_item))
    assert torch.equal(idx, w_idx) and torch.equal(score, w_score)
