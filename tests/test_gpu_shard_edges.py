"""Row-sharded Linear training (csrc/shard.cu) at its edges, on ONE B200 (``-m gpu``, all ranks of a group hosted by
one launch as in test_gpu_shard_train.py): tuning hooks that must not change a bit, degenerate batches and placements,
and the benchmark's own table sizes (50M x 5M rows, a user shard beyond 2^32 floats)."""
import numpy as np
import pytest
import torch

from oracle import cf_oracle as O
from tests.test_gpu_shard_train import (_full_params, _plan_words, _skewed, _to, _train_vs_oracle, _trainer,
                                        shard_hooks)  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _equal_runs(a, b):
    (la, sa, oa), (lb, sb, ob) = a, b
    assert torch.equal(la, lb)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
        for name, t in oa[k].items():
            if torch.is_tensor(t):
                assert torch.equal(t, ob[k][name]), (k, name)


# ---- C: tuning hooks that must be bit-neutral ----------------------------------------------------------------------
@pytest.mark.parametrize("hook,value,world", [("overlap", 1, 1), ("overlap", 0, 2), ("overlap", 0, 4),
                                              ("remote_hint", 0, 4)])
def test_tuning_hooks_do_not_change_a_bit(dev, shard_hooks, hook, value, world):
    """Phase A's early pass (on by default only with W > 1) and the L2 policy on stores into peer memory decide WHEN
    and HOW rows move, never what is summed in which order: losses, tables and optimizer state are identical."""
    U, I, D, B, steps = 3000, 20000, 64, 1024, 6
    rng = np.random.default_rng(7 * world + value)
    params = _full_params(rng, U, I, D)
    n = B * steps - 100
    user, pos, neg = (_to(dev, _skewed(rng, m, n)) for m in (U, I, I))
    runs = []
    for forced in (False, True):
        if forced:
            getattr(shard_hooks, f"trs_debug_shard_{hook}")(value)
        tr = _trainer(dev, world, U, I, D, B, "sparse_adam", 0.05, params)
        loss = tr.train_epoch(user, pos, neg, B)
        runs.append((loss, tr.state_dict(), tr.optimizer_state_dict()))
        # skewed ids: the plan flags some samples of every later step and leaves others to the early pass
        P = _plan_words(tr._plans[0], n, B)
        for s in range(1, steps):
            ent = P["samp"][s * B:s * B + int(P["samp_cnt"][s])]
            dirty = (ent & np.uint32(0xD0000000)) != 0
            assert dirty.any() and not dirty.all(), s
    _equal_runs(*runs)


# ---- D: edge batches -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [1, 3, 8])
@pytest.mark.parametrize("opt", ["adagrad", "sparse_adam"])
def test_pos_equal_neg_gives_exactly_zero_update(dev, world, opt):
    """Distinct users and items, pos == neg in every sample, fresh optimizer state: every hinge is exactly 1, every
    gradient row exactly 0 (the user's cancels in the difference, the item's between its two lookups), so the tables and
    the state do not move by a bit -- the sharded twin of test_gpu_parity's test of the same name."""
    U, I, D, B, steps = 3000, 2000, 64, 256, 3
    rng = np.random.default_rng(world)
    params = _full_params(rng, U, I, D)
    n = B * steps
    user = rng.permutation(U)[:n]
    item = rng.permutation(I)[:n]
    tr = _trainer(dev, world, U, I, D, B, opt, 0.05, params)
    before = (None, tr.state_dict(), tr.optimizer_state_dict())
    loss = tr.train_epoch(_to(dev, user), _to(dev, item), _to(dev, item), B)
    assert torch.equal(loss.cpu(), torch.ones(steps))
    _equal_runs((loss, *before[1:]), (loss, tr.state_dict(), tr.optimizer_state_dict()))


@pytest.mark.parametrize("world", [1, 3, 8])
def test_an_exact_hinge_tie_passes_the_gradient(dev, world):
    """h = s- - s+ + 1 == 0 exactly: zero user rows, user bias 0.5, positives' bias 0.75, negatives' -0.25 (all exact in
    fp32).  torch's clamp passes the gradient at 0 (the oracle's hinge_weights: >=), so the users move by g (v- - v+)
    and the item biases by -/+ g.  Every step draws fresh users and items, so each of its samples ties exactly; users
    repeat within a step (their rows go through the owners' staging buffers) and some occur once (updated in phase A)."""
    U, I, D, B, steps = 4000, 3000, 32, 256, 2
    rng = np.random.default_rng(40 + world)
    params = _full_params(rng, U, I, D)
    upool = rng.permutation(U)[:steps * 200].reshape(steps, 200)
    ipool = rng.permutation(I)[:steps * 240].reshape(steps, 2, 120)
    user = np.concatenate([rng.choice(upool[s], B) for s in range(steps)])
    pos = np.concatenate([rng.choice(ipool[s, 0], B) for s in range(steps)])
    neg = np.concatenate([rng.choice(ipool[s, 1], B) for s in range(steps)])
    params["user.weight"][user] = 0.0
    params["user_bias.weight"][user] = 0.5
    params["item_bias.weight"][pos] = 0.75
    params["item_bias.weight"][neg] = -0.25
    for s in range(steps):
        sl = slice(s * B, (s + 1) * B)
        h = O.linear_scores(params, user[sl], neg[sl]) - O.linear_scores(params, user[sl], pos[sl]) + np.float32(1)
        assert not h.any()
    tr, loss, _, _ = _train_vs_oracle(dev, world, "sgd", 0.05, B, params, user, pos, neg)
    assert not loss.any()
    sd = tr.state_dict()
    assert (sd["user.weight"].cpu().numpy()[user] != 0).any(axis=1).all()            # every tied user moved
    assert (sd["item_bias.weight"].cpu().numpy()[pos] > 0.75).all()


@pytest.mark.parametrize("world", [1, 3, 8])
def test_a_batch_smaller_than_the_group_and_a_last_step_of_one_sample(dev, world):
    """B = 2 global samples per step (fewer than the ranks) and a last step of 1: ranks that own no sample, ranks that
    own no pair, a step whose owners see one sample in all.  A power-of-two batch: g = 1/B sums exactly, so the user
    bias's gradient (-g + g per sample) is exactly 0 in the oracle too."""
    U, I, D, B = 50, 20, 36, 2
    rng = np.random.default_rng(60 + world)
    params = _full_params(rng, U, I, D)
    n = 6 * B + 1
    user, pos, neg = (rng.integers(0, m, n) for m in (U, I, I))
    _train_vs_oracle(dev, world, "sparse_adam", 0.05, B, params, user, pos, neg)


@pytest.mark.parametrize("world", [1, 3, 8])
def test_one_rank_runs_all_of_phase_a(dev, world):
    """Every user of the epoch is a multiple of W: rank 0 places every sample, the others only update the item rows
    they own (and receive gradient rows from rank 0)."""
    U, I, D, B, steps = 3000, 700, 64, 512, 3
    rng = np.random.default_rng(70 + world)
    params = _full_params(rng, U, I, D)
    n = B * steps
    user = world * _skewed(rng, U // world, n)
    pos, neg = _skewed(rng, I, n), _skewed(rng, I, n)
    _train_vs_oracle(dev, world, "adagrad", 0.05, B, params, user, pos, neg)


@pytest.mark.parametrize("world", [1, 3, 8])
def test_one_user_row_and_one_item_row_take_every_lookup(dev, world):
    """One user in every sample (phase B walks a run of B staged rows) and one item as every positive: step 0 also
    makes it every negative (a run of 2B), step 1 half of them, step 2 none.  SGD: in step 0 the user's gradient is
    exactly 0 in the kernel, which forms v- - v+ per sample, but a rounding residual in torch's order (every -g v+
    term, then every +g v-); Adagrad and Adam would turn that residual into a step of +-lr, SGD into lr times it."""
    U, I, D, B, steps = 1000, 500, 64, 1024, 3
    rng = np.random.default_rng(80 + world)
    params = _full_params(rng, U, I, D)
    n = B * steps
    u0, i0 = 997, 499
    user = np.full(n, u0)
    pos = np.full(n, i0)
    neg = rng.integers(0, I, n)
    neg[:B] = i0
    neg[B:2 * B:2] = i0
    tr, loss, _, _ = _train_vs_oracle(dev, world, "sgd", 0.05, B, params, user, pos, neg)
    assert loss[0] == 1.0


# ---- E: the benchmark's table sizes ----------------------------------------------------------------------------
def _gather_rows(tr, ids):
    """{param key: rows} and {param key: {state name: rows}} of the global ids ``ids[name]`` ("user" / "item"), read
    from their owners' shards (row r: rank r % W, local row r // W) -- never the whole table."""
    from torchrecsys_b200.sharded import _STATE_KEYS
    W = tr.world

    def pick(rows, get):
        out = None
        for q in range(W):
            m = rows % W == q
            if m.any():
                part = get(q)[torch.from_numpy(rows[m] // W).to(tr.device)].cpu().numpy()
                if out is None:
                    out = np.empty((len(rows), part.shape[1]), np.float32)
                out[m] = part
        return out

    params, state = {}, {}
    for name, wkey, bkey in tr._KEYS:
        rows = ids[name]
        params[wkey] = pick(rows, lambda q: tr.tables[q][name][0])
        params[bkey] = pick(rows, lambda q: tr.tables[q][name][1])
        state[wkey], state[bkey] = {}, {}
        for i, sname in enumerate(_STATE_KEYS[tr.kind]):
            state[wkey][sname] = pick(rows, lambda q: tr.state[q][name][i][0])
            state[bkey][sname] = pick(rows, lambda q: tr.state[q][name][i][1])
    return params, state


@pytest.mark.parametrize("dim,opt,world", [
    (128, "sgd", 1),          # C4's tables on one GPU: the user shard holds 6.4e9 floats, beyond 2^32
    (16, "sparse_adam", 2),   # 25M user rows per rank (a 4-pass sort) with optimizer state
])
def test_benchmark_sized_tables_match_the_oracle_on_the_rows_they_touch(dev, dim, opt, world):
    """ShardedLinearTrainer(50M, 5M) for 3 steps of 16384 samples against the oracle on COMPACTED tables: the sorted
    touched ids of each table, ids remapped by searchsorted (monotone: coalesce's order and every row's update are
    unchanged).  Forced into the ids: rows 0, U - 1, I - 1 and the last row of every shard, with U - 1 and I - 1 hot
    (several lookups per step: phase B, not phase A, updates a row that lies beyond 2^32 floats).  A seeded sample of
    untouched rows -- the touched rows' neighbours and the last rows of every bias shard among them (the kernel reads
    a bias 16 bytes at a time) -- must be bit-identical before and after."""
    from torchrecsys_b200 import _lib
    from torchrecsys_b200.sharded import ShardedLinearTrainer, _ArenaLayout, _STATE_KEYS, shard_rows
    U, I, B, steps = 50_000_000, 5_000_000, 16384, 3
    lr = {"sgd": 1000.0, "sparse_adam": 0.01}[opt]   # SGD: large enough that every update shows at fp32 precision
    need = world * _ArenaLayout(U, I, dim, len(_STATE_KEYS[opt]), world, _lib.shard_stage_bytes(dim, B),
                                _lib.SHARD_SYNC_BYTES).total
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(dev)[0]
    if free < need + (4 << 30):
        pytest.skip(f"needs {need / 2 ** 30:.1f} GiB of device memory + 4 GiB margin, {free / 2 ** 30:.1f} GiB free")

    rng = np.random.default_rng(dim)
    n = B * steps
    user, pos, neg = rng.integers(0, U, n), rng.integers(0, I, n), rng.integers(0, I, n)
    tops = {m: [(shard_rows(m, q, world) - 1) * world + q for q in range(world)] for m in (U, I)}
    for s in range(steps):
        at = s * B + rng.choice(B, 64, replace=False)
        user[at[:16]] = U - 1                     # hot: 16 lookups per step
        pos[at[16:32]] = I - 1
        neg[at[32:40]] = I - 1
        user[at[40:40 + world]] = tops[U]
        pos[at[48:48 + world]] = tops[I]
        if s == 0:
            user[at[60]], pos[at[61]] = 0, 0
    touched = {"user": np.unique(user), "item": np.unique(np.concatenate([pos, neg]))}

    def untouched_sample(n_rows, rows):
        cand = [rng.integers(0, n_rows, 4096), rows - 1, rows + 1]
        for q in range(world):
            cand.append(tops[n_rows][q] - world * np.arange(8))   # the last 8 rows of every shard
        c = np.concatenate(cand)
        return np.setdiff1d(c[(c >= 0) & (c < n_rows)], rows)
    others = {"user": untouched_sample(U, touched["user"]), "item": untouched_sample(I, touched["item"])}

    torch.manual_seed(dim)
    tr = ShardedLinearTrainer(U, I, dim, global_batch=B, optimizer=opt, lr=lr, device=dev, emulate_world=world)
    try:
        for q in range(world):                    # biases: non-zero everywhere, so that a stray write shows
            for name in ("user", "item"):
                tr.tables[q][name][1].normal_(0.0, 0.1)
        params, state = _gather_rows(tr, touched)
        others_before, others_state_before = _gather_rows(tr, others)
        ids = [_to(dev, a) for a in (user, pos, neg)]
        loss = tr.train_epoch(*ids, B).cpu().numpy()
        got, got_state = _gather_rows(tr, touched)
        others_after, others_state_after = _gather_rows(tr, others)
    finally:
        del tr
        torch.cuda.empty_cache()

    init = {k: v.copy() for k, v in params.items()}
    ids_of = {"user.weight": touched["user"], "item.weight": touched["item"], "item_bias.weight": touched["item"]}
    spec = O.OptSpec(opt, lr=lr)
    uc = np.searchsorted(touched["user"], user)
    pc, nc = np.searchsorted(touched["item"], pos), np.searchsorted(touched["item"], neg)
    want = []
    for s in range(steps):
        sl = slice(s * B, (s + 1) * B)
        want.append(O.train_step("linear", params, state, {"user": uc[sl], "pos": pc[sl], "neg": nc[sl]}, spec, s + 1))
    np.testing.assert_allclose(loss[0], want[0], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(loss, np.array(want), rtol=2e-5 if opt == "sgd" else 5e-4, atol=2e-6)
    tol = dict(rtol=2e-3, atol=2e-3 * lr * 20) if opt == "sparse_adam" else dict(rtol=1e-4, atol=2e-5)
    for k in params:
        np.testing.assert_allclose(got[k], params[k], err_msg=k, **tol)
        if k != "user_bias.weight":               # its gradient is exactly 0 (SURVEY D12)
            for sname in state[k]:
                np.testing.assert_allclose(got_state[k][sname], state[k][sname], err_msg=f"{k}.{sname}", **tol)
    for k, row in (("user.weight", U - 1), ("item.weight", I - 1), ("item_bias.weight", I - 1)):
        r = np.searchsorted(ids_of[k], row)
        assert not np.array_equal(got[k][r], init[k][r]), k          # the hot rows' updates are visible
    for k in others_before:
        assert np.array_equal(others_after[k], others_before[k]), k
        for sname in others_state_before[k]:
            assert np.array_equal(others_state_after[k][sname], others_state_before[k][sname]), (k, sname)
