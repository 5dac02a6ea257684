"""The one-pass kernel of the row-sharded trainer (csrc/shard.cu, one rank, one chunk per lane): phase A also updates
the item rows a step looks up once, phase B only runs the rows with several lookups.  It must compute bit for bit what
the two-phase kernel computes (trs_debug_shard_one_pass(0) forces that one), and the plan arrays it reads (iflag,
ikeyB / ivalB, cntB) must match a numpy restatement."""
import numpy as np
import pytest
import torch

from tests.test_gpu_shard_train import _full_params, _ids, _to, _trainer

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture
def one_pass_hook():
    """trs_debug_shard_one_pass is a process-wide setting: back to its default (on) afterwards, also on failure."""
    from torchrecsys_b200 import _lib
    L = _lib.lib()
    yield L
    L.trs_debug_shard_one_pass(1)
    L.trs_debug_shard_chunks_per_lane(1)


def _run(L, dev, one, world, opt, params, B, user, pos, neg):
    """Train the epoch with the one-pass kernel allowed (one=1) or not; returns losses, tables, optimizer state and
    which kernel the launch ran."""
    U, D = params["user.weight"].shape
    I = params["item.weight"].shape[0]
    L.trs_debug_shard_one_pass(one)
    tr = _trainer(dev, world, U, I, D, B, opt, 0.05, params)
    loss = tr.train_epoch(*(_to(dev, a) for a in (user, pos, neg)), B)
    return loss, tr.state_dict(), tr.optimizer_state_dict(), L.trs_debug_shard_last_one_pass()


def _same(a, b):
    (la, sa, oa, _), (lb, sb, ob, _) = a, b
    assert torch.equal(la, lb)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
        for name, t in oa[k].items():
            if torch.is_tensor(t):
                assert torch.equal(t, ob[k][name]), (k, name)


def _one_vs_two(L, dev, opt, params, B, user, pos, neg):
    one = _run(L, dev, 1, 1, opt, params, B, user, pos, neg)
    two = _run(L, dev, 0, 1, opt, params, B, user, pos, neg)
    assert one[3] == 1 and two[3] == 0
    _same(one, two)


@pytest.mark.parametrize("ids", ["uniform", "skewed"])
@pytest.mark.parametrize("dim", [4, 16, 64, 100, 128])
@pytest.mark.parametrize("opt", ["sgd", "adagrad", "sparse_adam"])
def test_one_pass_equals_two_phase(dev, one_pass_hook, opt, dim, ids):
    """Uniform ids (almost every item row single) and skewed ones (runs of duplicates, hot rows), every tenth sample
    with pos == neg, a ragged last step; dims 4 .. 128 give the row shapes (4,1), (16,1), (32,1) and a partial row."""
    U, I, B, steps = 3000, 20000, 1024, 5
    rng = np.random.default_rng(dim * 3 + len(ids) + len(opt))
    params = _full_params(rng, U, I, dim)
    n = B * steps - 300
    user, pos, neg = (_ids(rng, ids, m, n) for m in (U, I, I))
    neg[::10] = pos[::10]
    _one_vs_two(one_pass_hook, dev, opt, params, B, user, pos, neg)


@pytest.mark.parametrize("opt", ["adagrad", "sparse_adam"])
def test_a_single_row_read_again_next_step_and_a_row_taking_a_whole_step(dev, one_pass_hook, opt):
    """Item 7 is looked up once in step 0 (phase A updates it) and again in step 1, which must read the update;
    in step 2 item 9 takes every lookup (phase B sums all 2 B of them)."""
    U, I, D, B = 500, 4000, 64, 256
    rng = np.random.default_rng(11)
    params = _full_params(rng, U, I, D)
    user = rng.integers(0, U, 4 * B)
    pos, neg = rng.integers(10, I, 4 * B), rng.integers(10, I, 4 * B)
    pos[3], pos[B + 5], neg[B + 100] = 7, 7, 7
    pos[2 * B:3 * B] = neg[2 * B:3 * B] = 9
    _one_vs_two(one_pass_hook, dev, opt, params, B, user, pos, neg)


def test_the_benchmark_shape_runs_the_one_pass_kernel(dev, one_pass_hook):
    """D = 128 (one chunk per lane), SparseAdam, B = 16384 on one rank: the one-pass kernel runs and agrees with the
    two-phase one.  Two ranks, or two chunks per lane, keep the two-phase kernel."""
    U, I, D, B = 200_000, 100_000, 128, 16384
    rng = np.random.default_rng(5)
    params = _full_params(rng, U, I, D)
    n = 3 * B
    user, pos, neg = (rng.integers(0, m, n) for m in (U, I, I))
    _one_vs_two(one_pass_hook, dev, "sparse_adam", params, B, user, pos, neg)
    small = {k: v[:4000] for k, v in params.items()}
    u, p, q = user[:4096] % 4000, pos[:4096] % 4000, neg[:4096] % 4000
    assert _run(one_pass_hook, dev, 1, 2, "sparse_adam", small, 1024, u, p, q)[3] == 0
    one_pass_hook.trs_debug_shard_chunks_per_lane(2)
    assert _run(one_pass_hook, dev, 1, 1, "sparse_adam", small, 1024, u, p, q)[3] == 0


def _plan_arrays(plan, n, B):
    """The plan's arrays (csrc/shard.cu: shard_plan_layout), the one-rank ones after the seven shared ones."""
    raw = plan.cpu().numpy()
    words = raw.view(np.uint32)
    steps, off, out = -(-n // B), 0, {}
    for name, cnt in (("samp_cnt", steps), ("own_cnt", 2 * steps), ("samp", n), ("ukey", n), ("uval", n),
                      ("ikey", 2 * n), ("ival", 2 * n), ("cntB", 2 * steps), ("iflag", -(-2 * n // 4)),
                      ("ikeyB", 2 * n), ("ivalB", 2 * n)):
        out[name] = raw[off:off + 2 * n] if name == "iflag" else words[off // 4: off // 4 + cnt]
        off += (cnt * 4 + 255) // 256 * 256
    return out


@pytest.mark.parametrize("ids", ["uniform", "skewed"])
@pytest.mark.parametrize("n_users,n_items,B", [(1000, 200, 1000), (3001, 701, 1024), (50_000_000, 5_000_000, 16384)])
def test_one_rank_plan_arrays_match_their_numpy_restatement(dev, n_users, n_items, B, ids):
    """iflag: 1 exactly where the lookup's item row has no other lookup in the step; ikeyB / ivalB: the sorted item
    pairs of the other rows, in the same (stable) order; cntB: the user count of own_cnt and their number."""
    from torchrecsys_b200 import _lib
    rng = np.random.default_rng(n_items + len(ids))
    n = 3 * B - B // 3 - 1                                # a ragged last step
    user, pos, neg = (_ids(rng, ids, m, n) for m in (n_users, n_items, n_items))
    t = [_to(dev, a) for a in (user, pos, neg)]          # make_epoch takes addresses: the tensors must stay alive
    epoch = _lib.make_epoch(*t, None, None, B)
    sh = _lib.Shard()
    sh.rank, sh.world, sh.dim, sh.n_users, sh.n_items = 0, 1, 64, n_users, n_items
    P = _plan_arrays(_lib.shard_plan_build(sh, epoch, dev), n, B)
    torch.cuda.synchronize()
    n_single = 0
    for s in range(-(-n // B)):
        lo, hi = s * B, min(n, (s + 1) * B)
        both = np.concatenate([pos[lo:hi], neg[lo:hi]])
        _, inv, cnt = np.unique(both, return_inverse=True, return_counts=True)
        single = cnt[inv] == 1
        np.testing.assert_array_equal(P["iflag"][2 * lo:2 * lo + len(both)], single.astype(np.uint8))
        order = np.argsort(both, kind="stable")
        kept = order[~single[order]]
        assert int(P["cntB"][2 * s]) == int(P["own_cnt"][2 * s]), s
        nb = int(P["cntB"][2 * s + 1])
        assert nb == len(kept), s
        np.testing.assert_array_equal(P["ikeyB"][2 * lo:2 * lo + nb], both[kept])
        np.testing.assert_array_equal(P["ivalB"][2 * lo:2 * lo + nb], kept)
        n_single += int(single.sum())
    assert n_single > 0 or n_items < 1000
