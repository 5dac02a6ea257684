"""Row-sharded Linear training over peer-mapped shards (csrc/shard.cu, torchrecsys_b200/sharded.py) on ONE B200
(``-m gpu``): a single cooperative launch hosts all G ranks of the group (the SMs are split between them), so the
whole multi-rank path -- sample placement by user owner, loads from / gradient stores into "peer" arenas, the flag
barriers, owner-side coalesce + update -- runs on a 1-GPU box exactly as it does over NVLink, minus the wires.

Oracle: the numpy restatement's single-process step on the GLOBAL batch (oracle/cf_oracle.py: train_step), i.e.
model.py:274-284 of the reference.  Tolerances as tests/test_gpu_train_shapes.py (fp32; the order of a duplicate
row's summands differs from numpy's for rows with many lookups)."""
import numpy as np
import pytest
import torch

from oracle import cf_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _skewed(rng, n_rows, n):
    hot = rng.integers(0, 3, n)
    warm = rng.integers(0, min(n_rows, 64), n)
    cold = rng.integers(0, n_rows, n)
    pick = rng.random(n)
    return np.where(pick < 0.10, hot, np.where(pick < 0.35, warm, cold)).astype(np.int64)


def _full_params(rng, U, I, D):
    return {"user.weight": rng.normal(0, .4, (U, D)).astype(np.float32),
            "item.weight": rng.normal(0, .4, (I, D)).astype(np.float32),
            "user_bias.weight": rng.normal(0, .1, (U, 1)).astype(np.float32),
            "item_bias.weight": rng.normal(0, .1, (I, 1)).astype(np.float32)}


def _trainer(dev, world, U, I, D, B, opt, lr, params):
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    tr = ShardedLinearTrainer(U, I, D, global_batch=B, optimizer=opt, lr=lr, device=dev, emulate_world=world,
                              timeout_ms=5000)
    tr.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    return tr


def _to(dev, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


@pytest.fixture
def shard_hooks():
    """The sharded kernel's tuning hooks are process-wide settings: whoever changes one gets the defaults back
    afterwards (chunks per lane 1, overlap automatic, remote L2 hint on), also when the test fails."""
    from torchrecsys_b200 import _lib
    L = _lib.lib()
    yield L
    L.trs_debug_shard_chunks_per_lane(1)
    L.trs_debug_shard_overlap(-1)
    L.trs_debug_shard_remote_hint(1)


def _train_vs_oracle(dev, world, opt, lr, B, params, user, pos, neg):
    """Train the epoch (user, pos, neg) on ``world`` ranks and compare losses, tables and optimizer state with the
    oracle's single-process steps on the global batch; rows nobody looked up must be bit-identical to ``params``.
    Returns the trainer, the losses and the numbers of untouched user / item rows."""
    U, dim = params["user.weight"].shape
    I = params["item.weight"].shape[0]
    init = {k: v.copy() for k, v in params.items()}
    tr = _trainer(dev, world, U, I, dim, B, opt, lr, params)
    loss = tr.train_epoch(_to(dev, user), _to(dev, pos), _to(dev, neg), B).cpu().numpy()

    spec = O.OptSpec(opt, lr=lr)
    ref = {k: v.copy() for k, v in params.items()}
    state = O.init_opt_state(ref, spec)
    want = []
    for s in range(-(-len(user) // B)):
        batch = {"user": user[s * B:(s + 1) * B], "pos": pos[s * B:(s + 1) * B], "neg": neg[s * B:(s + 1) * B]}
        want.append(O.train_step("linear", ref, state, batch, spec, s + 1))
    np.testing.assert_allclose(loss[0], want[0], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(loss, np.array(want), rtol=2e-5 if opt == "sgd" else 5e-4, atol=2e-6)
    tol = dict(rtol=2e-3, atol=2e-3 * lr * 20) if opt == "sparse_adam" else dict(rtol=1e-4, atol=2e-5)
    got = {k: v.cpu().numpy() for k, v in tr.state_dict().items()}
    for k in ref:
        np.testing.assert_allclose(got[k], ref[k], err_msg=k, **tol)
    gst = tr.optimizer_state_dict()
    for k in ref:
        for sname, want_s in state[k].items():
            if k == "user_bias.weight":
                continue  # its gradient is exactly 0 (SURVEY D12): state stays 0 here; the oracle decays nothing either
            np.testing.assert_allclose(gst[k][sname].cpu().numpy(), want_s, err_msg=f"{k}.{sname}", **tol)
    # rows nobody looked up are bit-identical to the initial tables: embedding and bias, user and item
    untouched = {"user": np.setdiff1d(np.arange(U), user), "item": np.setdiff1d(np.arange(I), np.concatenate([pos, neg]))}
    for name, rows in untouched.items():
        for k in (f"{name}.weight", f"{name}_bias.weight"):
            assert np.array_equal(got[k][rows], init[k][rows]), k
    return tr, loss, len(untouched["user"]), len(untouched["item"])


def _steps_match_the_oracle(dev, world, dim, opt):
    U, I, steps = 3001, 701, 4
    B = 1500 if opt == "sgd" else 1024   # power-of-two batch: g = 1/B sums exactly (see test_gpu_train_shapes)
    lr = 0.05
    rng = np.random.default_rng(dim * 11 + world)
    params = _full_params(rng, U, I, dim)
    n = B * steps - (37 if opt == "sgd" else 0)   # SGD: short last batch
    items = np.setdiff1d(np.arange(I), rng.choice(I, 40, replace=False))   # 40 item rows nobody looks up
    user = _skewed(rng, U, n)
    pos, neg = items[_skewed(rng, len(items), n)], items[_skewed(rng, len(items), n)]
    _, _, n_user_rows, n_item_rows = _train_vs_oracle(dev, world, opt, lr, B, params, user, pos, neg)
    assert n_user_rows and n_item_rows >= 40


# dims 16, 64, 128 and 256 give the row shapes (G lanes, IT chunks per lane) = (4,1), (16,1), (32,1), (32,2), each
# filled by dim / 4 chunks.  These add the other default shapes, (8,1) at 20 and (32,4) at 260-512, and partial rows,
# where dim / 4 is not a multiple of G: 4, 12 (4,1), 20 (8,1), 36 (16,1), 100 (32,1), 132 (32,2), 260 and 384 (32,4)
_NEW_DIMS = (4, 12, 20, 36, 100, 132, 260, 384, 512)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("dim", sorted((16, 64, 128, 256) + _NEW_DIMS))
@pytest.mark.parametrize("opt", ["sgd", "adagrad", "sparse_adam"])
def test_sharded_steps_match_the_oracle_on_the_global_batch(dev, world, dim, opt):
    if opt != "sparse_adam" and (world != 3 if dim in _NEW_DIMS else (dim in (16, 256) or world in (3, 8))):
        pytest.skip("optimizer variants are covered on the other shapes")
    _steps_match_the_oracle(dev, world, dim, opt)


@pytest.mark.parametrize("world", [1, 3])
@pytest.mark.parametrize("dim", [32, 48, 64, 100, 128])
@pytest.mark.parametrize("opt", ["sgd", "sparse_adam"])
def test_two_chunks_per_lane_match_the_oracle(dev, shard_hooks, world, dim, opt):
    """trs_debug_shard_chunks_per_lane(2): (G, IT) = (4,2), (8,2) with a partial row, (8,2), (16,2) partial, (16,2) --
    shapes only this setting reaches, and the ones without the item-row prefetch region.  Against the oracle, not bit
    for bit against one chunk per lane: a lane sums its IT chunks before the lanes are added, so the dot products'
    association differs."""
    shard_hooks.trs_debug_shard_chunks_per_lane(2)
    _steps_match_the_oracle(dev, world, dim, opt)


def test_group_sizes_agree_bit_for_bit_and_split_launches_equal_one(dev):
    """The result does not depend on how many ranks share the work (every sum has a fixed association: slot order)
    nor on where an epoch is cut into launches."""
    U, I, D, B, steps = 2000, 500, 64, 512, 6
    rng = np.random.default_rng(3)
    params = _full_params(rng, U, I, D)
    n = B * steps
    user, pos, neg = (_to(dev, _skewed(rng, m, n)) for m in (U, I, I))
    ref = None
    for world in (1, 2, 4):
        tr = _trainer(dev, world, U, I, D, B, "sparse_adam", 0.05, params)
        loss = tr.train_epoch(user, pos, neg, B)
        sd = tr.state_dict()
        tr2 = _trainer(dev, world, U, I, D, B, "sparse_adam", 0.05, params)
        h = (steps // 2) * B
        l2 = torch.cat([tr2.train_epoch(user[:h], pos[:h], neg[:h], B), tr2.train_epoch(user[h:], pos[h:], neg[h:], B)])
        sd2 = tr2.state_dict()
        assert torch.equal(loss, l2)
        for k in sd:
            assert torch.equal(sd[k], sd2[k]), k
        if ref is None:
            ref = sd
        else:
            for k in sd:
                assert torch.equal(sd[k], ref[k]), (world, k)


def _plan_words(plan, n, B):
    """The plan's arrays (uint32 words at 256-byte aligned offsets, csrc/shard.cu: shard_plan_layout)."""
    words = plan.cpu().numpy().view(np.uint32)
    steps, off, out = -(-n // B), 0, {}
    for name, cnt in (("samp_cnt", steps), ("own_cnt", 2 * steps), ("samp", n), ("ukey", n), ("uval", n),
                      ("ikey", 2 * n), ("ival", 2 * n)):
        out[name] = words[off // 4: off // 4 + cnt]
        off += (cnt * 4 + 255) // 256 * 256
    return out


def _check_shard_plan(dev, user, pos, neg, B, n_users, n_items, world):
    """Every rank's plan (csrc/shard.cu: trs_shard_plan_build) against a numpy restatement, entry by entry:
      samp_cnt / samp   the samples whose user the rank owns (user % W == rank), their positions in ascending order;
      ukey / uval       (local row user // W, index in the rank's list), stably sorted by row, rows the step looks up
                        once dropped (phase A finishes those: every lookup of a user is on its owner); own_cnt[2s]
      ikey / ival       (local row id // W, lookup j) of the owned item lookups j < 2 B_s (j < B_s: positive of sample j,
                        else negative of sample j - B_s), stably sorted by row; own_cnt[2s + 1]
    Only the first own_cnt entries of a step's segment are compared: the rest is scratch.
    Flags of the samp entries: phase A runs a sample BEFORE the previous step's owners are done unless the plan flags one
    of its three rows as updated by that step (bits 28 / 30 / 31).  A flag may be set needlessly (the filter is hashed
    for large tables), it must never be missing; bit 27 marks the users with one lookup in the step, bit 29 is unused."""
    from torchrecsys_b200 import _lib
    n = len(user)
    steps = -(-n // B)
    ids = [_to(dev, a) for a in (user, pos, neg)]          # make_epoch takes addresses: the tensors must stay alive
    epoch = _lib.make_epoch(*ids, None, None, B)
    needless = total = 0
    for rank in range(world):
        sh = _lib.Shard()
        sh.rank, sh.world, sh.dim, sh.n_users, sh.n_items = rank, world, 64, n_users, n_items
        P = _plan_words(_lib.shard_plan_build(sh, epoch, dev), n, B)
        torch.cuda.synchronize()
        for s in range(steps):
            lo, hi = s * B, min(n, (s + 1) * B)
            u_s, p_s, n_s = user[lo:hi], pos[lo:hi], neg[lo:hi]
            mine = np.flatnonzero(u_s % world == rank)
            cnt = int(P["samp_cnt"][s])
            assert cnt == len(mine), (rank, s)
            ent = P["samp"][lo:lo + cnt]
            np.testing.assert_array_equal(ent & 0x07FFFFFF, mine)        # the rank's samples, in batch order
            u, p_, n_ = u_s[mine], p_s[mine], n_s[mine]
            uniq, c = np.unique(u_s, return_counts=True)
            single = np.isin(u, uniq[c == 1])
            np.testing.assert_array_equal((ent >> 27) & 1, single.astype(np.uint32))
            assert not ((ent >> 29) & 1).any()

            key = u // world
            order = np.argsort(key, kind="stable")
            kept = order[~single[order]]
            nu = int(P["own_cnt"][2 * s])
            assert nu == len(kept), (rank, s)
            np.testing.assert_array_equal(P["ukey"][lo:lo + nu], key[kept])
            np.testing.assert_array_equal(P["uval"][lo:lo + nu], kept)    # bit 31 (done in phase A) clear

            both = np.concatenate([p_s, n_s])
            j = np.flatnonzero(both % world == rank)
            order = np.argsort(both[j] // world, kind="stable")
            ni = int(P["own_cnt"][2 * s + 1])
            assert ni == len(j), (rank, s)
            np.testing.assert_array_equal(P["ikey"][2 * lo:2 * lo + ni], both[j[order]] // world)
            np.testing.assert_array_equal(P["ival"][2 * lo:2 * lo + ni], j[order])

            f_user, f_pos, f_neg = (((ent >> k) & 1).astype(bool) for k in (28, 30, 31))
            if s == 0:                                     # nothing is known about the step before the plan
                assert f_user.all() and f_pos.all() and f_neg.all()
                continue
            plo = lo - B
            items_prev = np.union1d(pos[plo:lo], neg[plo:lo])
            up, cp = np.unique(user[plo:lo], return_counts=True)
            must = (np.isin(u, up[cp > 1]), np.isin(p_, items_prev), np.isin(n_, items_prev))
            for flag, need in zip((f_user, f_pos, f_neg), must):
                assert not (need & ~flag).any()
                needless += int((flag & ~need).sum())
                total += len(flag)
    assert needless <= 0.04 * total


@pytest.mark.parametrize("world,n_items", [(1, 3000), (4, 3000), (2, 3_000_000), (8, 3_000_000)])
def test_plan_flags_never_miss_a_row_the_previous_step_updates(dev, world, n_items):
    """The whole plan (_check_shard_plan) with an exact item filter (3000 items) and a hashed one (3M)."""
    U, B, steps = 4000, 1024, 5
    rng = np.random.default_rng(world + n_items)
    n = B * steps - 100                                   # a ragged last step
    user, pos, neg = _skewed(rng, U, n), _skewed(rng, n_items, n), rng.integers(0, n_items, n)
    _check_shard_plan(dev, user, pos, neg, B, U, n_items, world)


def _ids(rng, kind, n_rows, n):
    """Uniform ids, or _skewed's mix with half of it mirrored to the top of the table (hot rows at both ends)."""
    if kind == "uniform":
        return rng.integers(0, n_rows, n, dtype=np.int64)
    x = _skewed(rng, n_rows, n)
    return np.where(rng.random(n) < 0.5, x, n_rows - 1 - x)


@pytest.mark.parametrize("ids", ["uniform", "skewed"])
@pytest.mark.parametrize("n_users,n_items,world,B", [   # radix passes of the user / item sort on every rank
    (1000, 200, 4, 1000),                               # 1 / 1
    (3001, 701, 8, 1000),                               # 2 / 1
    (50_000_000, 5_000_000, 1, 16384),                  # 4 / 3: the benchmark's workload (C4) on one GPU
    (50_000_000, 5_000_000, 8, 131072),                 # 3 / 3: C4 on eight GPUs (16384 samples per rank and step)
    (2 ** 32 - 1, 2 ** 32 - 1, 3, 16384),               # 4 / 4: ids >= 2^31, a group size that is not a power of two
])
def test_shard_plan_matches_its_numpy_restatement(dev, n_users, n_items, world, B, ids):
    """The plan at the benchmark's table sizes and batches: odd pass counts start the sort in the scratch buffer, a
    step spans many route tiles (2048 lookups each) and many 1024-pair chunks of the in-place user compaction."""
    rng = np.random.default_rng(n_users % 1000 + world + (ids == "skewed"))
    n = 3 * B - B // 3 - 1                                # a ragged last step
    user, pos, neg = (_ids(rng, ids, m, n) for m in (n_users, n_items, n_items))
    _check_shard_plan(dev, user, pos, neg, B, n_users, n_items, world)


def test_host_fed_epoch_in_chunks_equals_one_resident_epoch(dev):
    """train_epoch_host copies chunk i+1 on a side stream while chunk i trains: same tables, same losses as one
    train_epoch over device-resident ids (chunks are split launches; negatives keyed by the global sample index)."""
    from torchrecsys_b200 import _lib
    U, I, D, B, steps = 3000, 800, 32, 256, 150
    rng = np.random.default_rng(11)
    params = _full_params(rng, U, I, D)
    ids_host = torch.from_numpy(np.stack([_skewed(rng, U, steps * B).reshape(steps, B),
                                          _skewed(rng, I, steps * B).reshape(steps, B)], 1)).pin_memory()
    draw = lambda pos, first: _lib.philox_negatives(99, first, pos, I)[0]
    a = _trainer(dev, 1, U, I, D, B, "adagrad", 0.05, params)
    loss_host = torch.zeros(steps).pin_memory()
    la = a.train_epoch_host(ids_host, draw, loss_host, chunk_steps=64)      # 10 + 40 + 64 + 36 steps
    a.check_status()
    b = _trainer(dev, 1, U, I, D, B, "adagrad", 0.05, params)
    user, pos = ids_host[:, 0].reshape(-1).to(dev), ids_host[:, 1].reshape(-1).to(dev)
    lb = b.train_epoch(user, pos, draw(pos, 0), B)
    torch.cuda.synchronize()
    assert torch.equal(la, lb) and torch.equal(loss_host, lb.cpu())
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    # and again: the buffers of the first call are reused
    la2 = a.train_epoch_host(ids_host, draw, None, chunk_steps=64)
    lb2 = b.train_epoch(user, pos, draw(pos, 0), B)
    assert torch.equal(la2, lb2)


def test_sharded_training_equals_the_fused_single_gpu_kernel(dev):
    """Same ids, same init: the peer-mapped path and trs_train_steps (one GPU, whole tables) end in the same
    tables up to the order of duplicate sums."""
    from torchrecsys_b200.collaborative.linear import Linear
    from torchrecsys_b200.engine import EpochRunner
    U, I, D, B, steps = 5000, 900, 128, 1024, 5
    rng = np.random.default_rng(9)
    params = _full_params(rng, U, I, D)
    n = B * steps
    user, pos, neg = (_to(dev, rng.integers(0, m, n)) for m in (U, I, I))
    net = Linear(U, I, {}, D, use_metadata=False, use_cuda=True)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    net = net.to(dev)
    opt = torch.optim.SparseAdam(list(net.parameters()), lr=0.01)
    loss_f = EpochRunner(net, opt).run({"user": user, "pos": pos, "neg": neg}, B)
    tr = _trainer(dev, 4, U, I, D, B, "sparse_adam", 0.01, params)
    loss_s = tr.train_epoch(user, pos, neg, B)
    np.testing.assert_allclose(loss_s.cpu().numpy(), loss_f.cpu().numpy(), rtol=1e-5, atol=1e-6)
    sd = tr.state_dict()
    for k, v in net.state_dict().items():
        np.testing.assert_allclose(sd[k].cpu().numpy(), v.cpu().numpy(), rtol=2e-3, atol=2e-4, err_msg=k)


def test_a_fitted_model_moves_onto_shards_and_back(dev):
    """fit (fused kernel, torch SparseAdam) -> from_model -> a sharded epoch -> to_model -> fit again, against the fused
    kernel running all three epochs: the optimizer's moments and step count travel both ways."""
    import copy
    from torchrecsys_b200.collaborative.linear import Linear
    from torchrecsys_b200.engine import EpochRunner
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    U, I, D, B, steps = 3000, 700, 64, 512, 4
    rng = np.random.default_rng(21)
    n = B * steps
    epochs = [{k: _to(dev, rng.integers(0, m, n)) for k, m in (("user", U), ("pos", I), ("neg", I))} for _ in range(3)]
    torch.manual_seed(5)
    net_a = Linear(U, I, {}, D, use_metadata=False, use_cuda=True).to(dev)
    net_b = copy.deepcopy(net_a)
    opt_a = torch.optim.SparseAdam(list(net_a.parameters()), lr=0.02)
    opt_b = torch.optim.SparseAdam(list(net_b.parameters()), lr=0.02)
    for e in epochs:                                                   # a: the fused kernel all the way
        EpochRunner(net_a, opt_a).run(e, B)
    EpochRunner(net_b, opt_b).run(epochs[0], B)                        # b: fused, sharded over 2 ranks, fused
    tr = ShardedLinearTrainer.from_model(net_b, opt_b, B, device=dev, emulate_world=2)
    assert tr.binding.step0 == steps
    tr.train_epoch(epochs[1]["user"], epochs[1]["pos"], epochs[1]["neg"], B)
    tr.to_model(net_b, opt_b)
    assert opt_b.state[net_b.user.weight]["step"] == 2 * steps
    EpochRunner(net_b, opt_b).run(epochs[2], B)
    for (k, p), (_, q) in zip(net_a.named_parameters(), net_b.named_parameters()):
        np.testing.assert_allclose(q.detach().cpu().numpy(), p.detach().cpu().numpy(), rtol=2e-3, atol=2e-4, err_msg=k)
        for name in ("exp_avg", "exp_avg_sq"):
            np.testing.assert_allclose(opt_b.state[q][name].cpu().numpy(), opt_a.state[p][name].cpu().numpy(),
                                       rtol=2e-3, atol=1e-6, err_msg=f"{k} {name}")


def test_checkpoint_moves_between_group_sizes_and_the_single_gpu_model(dev):
    """state_dict() / optimizer_state_dict() are in the reference's single-process layout: train on 2 ranks, reload on
    3 ranks (parameters AND SparseAdam moments), continue -- equals 4 uninterrupted steps on 1 rank."""
    U, I, D, B = 1200, 300, 32, 256
    rng = np.random.default_rng(5)
    params = _full_params(rng, U, I, D)
    n = B * 4
    user, pos, neg = (_to(dev, _skewed(rng, m, n)) for m in (U, I, I))
    one = _trainer(dev, 1, U, I, D, B, "sparse_adam", 0.05, params)
    one.train_epoch(user, pos, neg, B)
    a = _trainer(dev, 2, U, I, D, B, "sparse_adam", 0.05, params)
    h = 2 * B
    a.train_epoch(user[:h], pos[:h], neg[:h], B)
    b = _trainer(dev, 3, U, I, D, B, "sparse_adam", 0.05, params)
    b.load_state_dict(a.state_dict(), a.optimizer_state_dict())
    assert b.binding.step0 == 2
    b.train_epoch(user[h:], pos[h:], neg[h:], B)
    for k, v in one.state_dict().items():
        assert torch.equal(b.state_dict()[k], v), k
    so, sb = one.optimizer_state_dict(), b.optimizer_state_dict()
    for k in so:
        for name in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(so[k][name], sb[k][name]), (k, name)
    # and into the single-GPU module of the drop-in API
    from torchrecsys_b200.collaborative.linear import Linear
    net = Linear(U, I, {}, D, use_metadata=False, use_cuda=True)
    net.load_state_dict(b.state_dict())
    assert torch.equal(net.item.weight.detach().cpu(), one.state_dict()["item.weight"].cpu())


def test_bad_arguments_raise(dev):
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    with pytest.raises(ValueError):
        ShardedLinearTrainer(10, 10, 6, global_batch=8, device=dev, emulate_world=2)      # dim % 4
    tr = ShardedLinearTrainer(100, 50, 8, global_batch=16, device=dev, emulate_world=2)
    ids = torch.zeros(64, dtype=torch.int64, device=dev)
    with pytest.raises(ValueError):
        tr.train_epoch(ids, ids, ids, 32)                                                  # batch > staging size
