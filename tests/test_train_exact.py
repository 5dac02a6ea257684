"""The training kernels, bit for bit, against an exact restatement of torch's optimizer step.

Why bit for bit is possible here
--------------------------------
Every other training test compares within a tolerance: with random fp32 tables a hot row's gradient is a sum whose
rounding depends on the order of its terms, and the kernels sum in another order than numpy or torch.  This file builds
fixtures on which that order cannot matter.  The scorer is Linear (with and without metadata tables); its parameters
are small integers, or dyadic values on a coarse grid, and every step's sample count is a power of two, so that the
hinge weight g = 1 / B_s is exact.  Then every score, hinge, per-lookup gradient, coalesced gradient row and loss is a
multiple of a known power of two, and ``exact_step`` PROVES, per fixture and per step, that each sum stays below 2^24
grid units counting the absolute values of its terms.  Every fp32 partial sum, in any order and any association, is
then exact.  A fixture that fails the proof is refused (``NotExact``): no test here falls back to a tolerance.  The
margins are integers, so ties (h == 0, where the hinge passes its gradient) and inactive samples both occur often.

What the kernels must compute (the contract of csrc/train.cuh: opt_update)
-------------------------------------------------------------------------
G is the exact coalesced gradient of a row, t the 1-based step, every op an fp32 op, correctly rounded, none fused
(torch: optim/_functional.py sparse_adam, optim/adagrad.py _single_tensor_adagrad, optim/sgd.py):

  SGD         p <- p + f32(-lr) * G
  Adagrad     s <- s + G * G;   std <- sqrt(s) + f32(eps);   p <- p + f32(-clr_t) * (G / std)
              clr_t = lr / (1 + (t - 1) lr_decay) in doubles
  SparseAdam  m' <- m + (G - m) * f32(1 - b1);   v' <- v + (G * G - v) * f32(1 - b2)
              p <- p + f32(-step_t) * (m' / (sqrt(v') + f32(eps)))
              step_t = lr sqrt(1 - b2^t) / (1 - b1^t) in doubles

A product followed by a sum rounds twice.  ``oracle/cf_oracle.py: apply_rows`` states exactly this stream; the
reference here is apply_rows applied to the exact G of every row a step looks up.  That includes rows whose G is 0
(looked up only by inactive samples, or with cancelling lookups): SparseAdam still decays their moments and moves them.
Not included is ``user_bias``: its gradient is -g + g = 0 per sample, and the kernels never touch that table or its
state (SURVEY D12).  The tests load zero state for it, on which torch's own step leaves it unchanged as well.

How torch itself is pinned (``test_torch_cuda_optimizers_follow_the_reference``, on the GPU)
-----------------------------------------------------------------------------------------
torch.optim.{SGD, Adagrad, SparseAdam} on CUDA tensors, fed the per-lookup (uncoalesced) gradient an
``nn.Embedding(sparse=True)`` backward produces, step the same fixture.  Their results equal the reference bit for bit:
on CUDA, ``dense.add_(sparse, alpha=a)`` with a sparse tensor not flagged coalesced -- what Adagrad's ``_make_sparse``
builds -- computes ``values.mul(a)`` and then ``index_add_``: two roundings, as above.  torch's CUDA sqrt and
division are correctly rounded.  torch on the CPU deviates in two places, and the CPU self-checks below only compare
what those do not reach.  Its dense += alpha * sparse is an axpy, a fused multiply-add with one rounding.  Its in-place
fp32 ``sqrt_`` is not correctly rounded: about 0.7 % of inputs come out 1 ulp off.  The kernels keep the stream above.

SGD agrees with torch bit for bit only where every product and partial sum is exact: torch applies each lookup's
-lr * g on its own, in an order it does not fix, while the kernels add -lr * G once per row.  On these fixtures lr is
a power of two (or B_s), so both are exact.  With any other lr the two agree to rounding.

Where it runs
-------------
fused trainer (csrc/train.cu through EpochRunner; both plan builders), row-sharded trainer (csrc/shard.cu: one-pass
and two-phase kernels, 1 to 8 emulated ranks, two chunks per lane), and the autograd backward (trs_scores_backward).
Three kinds of test: one step from random optimizer state (every rounding of the update); SGD over eight and more
steps in one launch and split over launches (a stale read of a row changes an integer score, not a last bit); and two
Adagrad / SparseAdam steps from fresh state, where step 1 moves every entry by exactly +-lr or 0."""
import numpy as np
import pytest
import torch

from oracle import cf_oracle as O

F32 = np.float32
BASE_KEYS = ("user.weight", "item.weight", "user_bias.weight", "item_bias.weight")


# --------------------------------------------------------------------------------------------------------------------
# fixtures: ids that take every reduce path, integer tables
# --------------------------------------------------------------------------------------------------------------------
def lookup_ids(rng, n, n_rows, hot_row=None, carry=()):
    """``n`` lookups into a table of ``n_rows`` rows: one hot row with more than 8 lookups (a whole CTA reduces it),
    rows with 2..8 lookups, and rows looked up once (phase A updates those), shuffled.  ``carry``: rows of the
    previous step, some of which come back as single lookups (step s + 1 must read what step s wrote)."""
    perm = rng.permutation(n_rows)
    if hot_row is not None:
        perm = np.concatenate([[hot_row], perm[perm != hot_row]])
    ids, nxt = [], 0
    if n >= 24:
        ids += [perm[0]] * max(9, n // 8)
        nxt = 1
    while len(ids) < n // 2:
        ids += [perm[nxt]] * int(rng.integers(2, 9))
        nxt += 1
    ids = ids[:n]
    fresh = perm[nxt:]
    back = [r for r in carry if r not in set(ids)][: (n - len(ids)) // 4]
    fresh = fresh[~np.isin(fresh, back)]
    ids += list(back) + list(fresh[: n - len(ids) - len(back)])
    assert len(ids) == n, "table too small for the lookups of a step"
    return rng.permutation(np.array(ids, dtype=np.int64))


def make_ids(rng, steps, U, I, pattern="mixed"):
    """Global epoch (user, pos, neg) of the given step sizes.  ``mixed``: lookup_ids per id space, every 16th sample
    with pos == neg.  ``one_user``: one user row and one positive item row take every user / positive lookup of the
    step."""
    user, pos, neg = [], [], []
    carry_u, carry_i = (), ()
    hot_u, hot_i = int(rng.integers(U)), int(rng.integers(I))
    for Bs in steps:
        u = lookup_ids(rng, Bs, U, hot_u, carry_u)
        both = lookup_ids(rng, 2 * Bs, I, hot_i, carry_i)
        p, q = both[:Bs], both[Bs:].copy()
        q[::16] = p[::16]
        if pattern == "one_user":
            u, p = np.full(Bs, hot_u), np.full(Bs, hot_i)
        user.append(u), pos.append(p), neg.append(q)
        carry_u, carry_i = tuple(u[:Bs // 2]), tuple(np.concatenate([p, q])[:Bs])
    return (np.concatenate(user).astype(np.int64), np.concatenate(pos).astype(np.int64),
            np.concatenate(neg).astype(np.int64))


def make_params(rng, U, I, D, meta_sizes=(), dense_users=0.5, item_vals=2, meta_vals=1, bias_vals=3):
    """Integer tables.  A user row is dense (entries in [-2, 2]) or has one to three entries of +-1 / +-2: dense rows
    give varied gradients, sparse ones small margins and many exact ties."""
    user = rng.integers(-2, 3, (U, D))
    sparse = rng.random(U) >= dense_users
    user[sparse] = 0
    for r in np.flatnonzero(sparse):
        k = int(rng.integers(1, 4))
        user[r, rng.choice(D, k, replace=False)] = rng.choice([-2, -1, 1, 2], k)
    p = {f"metadata.{f}.weight": rng.integers(-meta_vals, meta_vals + 1, (C, D)) for f, C in enumerate(meta_sizes)}
    p.update({"user.weight": user, "item.weight": rng.integers(-item_vals, item_vals + 1, (I, D)),
              "user_bias.weight": rng.integers(-bias_vals, bias_vals + 1, (U, 1)),
              "item_bias.weight": rng.integers(-bias_vals, bias_vals + 1, (I, 1))})
    return {k: v.astype(F32) for k, v in p.items()}


def item_meta(rng, I, meta_sizes):
    """Per-item metadata ids: feature 0 from a small table (every row hot), feature 1 a permutation of the items (the
    multiplicities of the item table, in another table)."""
    cols = [rng.integers(0, meta_sizes[0], I)] if meta_sizes else []
    if len(meta_sizes) > 1:
        assert meta_sizes[1] == I
        cols.append(rng.permutation(I))
    return np.stack(cols, 1).astype(np.int64) if cols else np.zeros((I, 0), np.int64)


def random_state(rng, params, kind, eps):
    """torch-layout optimizer state of any value: exp_avg of either sign over ten decades, exp_avg_sq / sum positive
    over thirteen, some of them near eps and near eps^2 (where sqrt(s) ~ eps).  user_bias keeps zero state (D12)."""
    st = {}
    for k, p in params.items():
        def pos():
            x = 10.0 ** rng.uniform(-12, 1, p.shape)
            pick = rng.random(p.shape)
            x = np.where(pick < 0.1, eps * rng.uniform(0.5, 2, p.shape), x)
            x = np.where(pick > 0.9, eps * eps * rng.uniform(0.5, 4, p.shape), x)
            return x.astype(F32)
        if kind == "adagrad":
            st[k] = {"sum": pos()}
        elif kind == "sparse_adam":
            m = (rng.choice([-1.0, 1.0], p.shape) * 10.0 ** rng.uniform(-9, 1, p.shape)).astype(F32)
            st[k] = {"exp_avg": m, "exp_avg_sq": pos()}
        else:
            st[k] = {}
        if k == "user_bias.weight":
            st[k] = {n: np.zeros_like(v) for n, v in st[k].items()}
    return st


# --------------------------------------------------------------------------------------------------------------------
# the exact step: gradients with a proof of exactness, then apply_rows
# --------------------------------------------------------------------------------------------------------------------
class NotExact(AssertionError):
    """A fixture on which some fp32 sum of the step could round: the test refuses it."""


def grid_exponent(params):
    """The least e >= 0 with every parameter a multiple of 2^-e."""
    for e in range(0, 41):
        if all(np.all(np.floor(v.astype(np.float64) * 2.0 ** e) == v.astype(np.float64) * 2.0 ** e)
               for v in params.values()):
            return e
    raise NotExact("parameters are not on a dyadic grid")


def _bound(abs_sum, e, what):
    """Every term a multiple of 2^-e and the sum of their absolute values below 2^24 grid units: every partial sum,
    in any order, is an exact fp32 value."""
    worst = float(np.max(abs_sum, initial=0.0)) * 2.0 ** e
    if not worst < 2.0 ** 24:
        raise NotExact(f"{what}: {worst:.0f} grid units of 2^-{e} (limit 2^24)")


def exact_step(params, batch):
    """Loss and coalesced gradient of one step of the Linear scorer, in float64, with the proof that fp32 computes
    the same values in any summation order.  Returns (loss, {key: (rows, G)}, coverage counts, {key: (ids, g)});
    rows are the unique rows the step looks up, G their exact gradient (zero rows included, as torch's coalesced
    gradient has them), ids / g the per-lookup gradient an nn.Embedding(sparse=True) backward emits."""
    user, pos, neg = batch["user"], batch["pos"], batch["neg"]
    Bs = len(user)
    if Bs & (Bs - 1):
        raise NotExact(f"step of {Bs} samples: 1/B is not a power of two")
    lb = Bs.bit_length() - 1
    n_meta = sum(k.startswith("metadata.") for k in params)
    P = {k: v.astype(np.float64) for k, v in params.items()}
    e = grid_exponent(params)

    def item_vec(items, meta):
        parts = [P["item.weight"][items]] + [P[f"metadata.{f}.weight"][meta[:, f]] for f in range(n_meta)]
        return sum(parts), sum(np.abs(x) for x in parts)

    u = P["user.weight"][user]
    vp, vpa = item_vec(pos, batch.get("pos_meta"))
    vn, vna = item_vec(neg, batch.get("neg_meta"))
    _bound(np.maximum(vpa, vna), e, "item + metadata vector")
    bu, bp, bn = P["user_bias.weight"][user, 0], P["item_bias.weight"][pos, 0], P["item_bias.weight"][neg, 0]
    # both scores and the hinge, every product and bias counted: covers any association of dot, biases and margin
    _bound((np.abs(u) * (vpa + vna)).sum(1) + 2 * np.abs(bu) + np.abs(bp) + np.abs(bn) + 1, 2 * e, "hinge")
    sp = (u * vp).sum(1) + bu + bp
    sn = (u * vn).sum(1) + bu + bn
    h = sn - sp + 1
    act = (h >= 0).astype(np.float64)
    _bound(np.abs(h).sum(), 2 * e, "loss sum")
    loss = float(np.maximum(h, 0).sum()) / Bs
    g = act / Bs
    ge = e + lb                                           # grid of the embedding gradients: params * 2^-lb
    per_lookup = {
        "user.weight": (np.concatenate([user, user]), np.concatenate([-g[:, None] * vp, g[:, None] * vn]),
                        np.concatenate([g[:, None] * vpa, g[:, None] * vna]), ge),
        "item.weight": (np.concatenate([pos, neg]), np.concatenate([-g[:, None] * u, g[:, None] * u]),
                        np.concatenate([g[:, None] * np.abs(u)] * 2), ge),
        "user_bias.weight": (np.concatenate([user, user]), np.concatenate([-g, g])[:, None],
                             np.concatenate([g, g])[:, None], lb),
        "item_bias.weight": (np.concatenate([pos, neg]), np.concatenate([-g, g])[:, None],
                             np.concatenate([g, g])[:, None], lb),
    }
    for f in range(n_meta):
        ids = np.concatenate([batch["pos_meta"][:, f], batch["neg_meta"][:, f]])
        per_lookup[f"metadata.{f}.weight"] = (ids,) + per_lookup["item.weight"][1:]
    grads, lookups = {}, {}
    cover = {"ties": int((h == 0).sum()), "inactive": int((h < 0).sum()), "pos_eq_neg": int((pos == neg).sum())}
    for k, (ids, vals, absv, gk) in per_lookup.items():
        lookups[k] = (ids, vals.astype(F32))             # each term is exact: it is part of the bounded sum below
        rows, inv, cnt = np.unique(ids, return_inverse=True, return_counts=True)
        G = np.zeros((len(rows), vals.shape[1]))
        A = np.zeros_like(G)
        np.add.at(G, inv, vals)
        np.add.at(A, inv, absv)
        _bound(A, gk, f"coalesced gradient of {k}")
        G32 = G.astype(F32)
        if not np.array_equal(G32.astype(np.float64), G):
            raise NotExact(f"{k}: a gradient row is not an fp32 value")
        grads[k] = (rows, G32)
        if k in ("user.weight", "item.weight"):
            cnt = cnt // 2 if k == "user.weight" else cnt   # the kernels reduce a user row once per sample
            live = np.zeros(len(rows))
            np.add.at(live, inv, np.concatenate([act, act]))
            cover[k] = {"single": int((cnt == 1).sum()), "2..8": int(((cnt > 1) & (cnt <= 8)).sum()),
                        ">8": int((cnt > 8).sum()), "inactive only": int((live == 0).sum()), "max": int(cnt.max())}
    return F32(loss), grads, cover, lookups


def ref_step(params, state, batch, spec, t):
    """One step of the contract (module docstring) on the exact gradient; mutates params / state, returns the loss."""
    loss, grads = exact_step(params, batch)[:2]
    for k, (rows, G) in grads.items():
        if k != "user_bias.weight":                      # never touched (SURVEY D12), its gradient is 0
            O.apply_rows(params[k], state[k], rows, G, spec, t)
    return loss


def batches(user, pos, neg, steps, meta=None):
    out, lo = [], 0
    for Bs in steps:
        b = {"user": user[lo:lo + Bs], "pos": pos[lo:lo + Bs], "neg": neg[lo:lo + Bs]}
        if meta is not None and meta.shape[1]:
            b["pos_meta"], b["neg_meta"] = meta[b["pos"]], meta[b["neg"]]
        out.append(b)
        lo += Bs
    return out


def ref_epoch(params, state, bs, spec, t0):
    """The reference over consecutive steps from step count t0 (steps already taken); returns the losses."""
    return np.array([ref_step(params, state, b, spec, t0 + i + 1) for i, b in enumerate(bs)], dtype=F32)


def copy_tree(d):
    return {k: (copy_tree(v) if isinstance(v, dict) else v.copy()) for k, v in d.items()}


# --------------------------------------------------------------------------------------------------------------------
# the cases
# --------------------------------------------------------------------------------------------------------------------
# one step from random state: non-default hyper-parameters, lr not a power of two, a random step count
HP = {"sgd": dict(lr=0.25), "adagrad": dict(lr=0.0123, eps=3e-9, lr_decay=0.013),
      "sparse_adam": dict(lr=0.0123, betas=(0.85, 0.995), eps=2e-7)}
# two steps from fresh state: step 1 moves every entry by exactly +-lr or 0 (see test_two_steps_from_fresh_state)
HP2 = {"adagrad": dict(lr=0.5, eps=2.0 ** -100), "sparse_adam": dict(lr=0.5, betas=(0.5, 0.75), eps=2.0 ** -100)}


def spec_of(kind, hp):
    return O.OptSpec(kind, lr=hp["lr"], betas=hp.get("betas", (0.9, 0.999)), eps=hp.get("eps"),
                     lr_decay=hp.get("lr_decay", 0.0))


def one_step_case(seed, D, F, kind, pattern="mixed", B=256):
    """(params, state, t0, (user, pos, neg), item_meta, steps): one step of B samples from random state, F metadata
    tables (7 rows, and one as large as the item table)."""
    rng = np.random.default_rng(seed)
    U, I = 6 * B, 10 * B
    sizes = (7, I)[:F]
    params = make_params(rng, U, I, D, sizes)
    meta = item_meta(rng, I, sizes)
    ids = make_ids(rng, [B], U, I, pattern)
    state = random_state(rng, params, kind, spec_of(kind, HP[kind]).eps)
    t0 = int(rng.integers(0, 5000))
    return params, state, t0, ids, meta, [B]


def sgd_case(seed, D, F=0, B=64, n_steps=9):
    """SGD with lr = B over n_steps steps (the last one B / 4): lr * g = +-1 per active lookup, integer tables stay
    integer.  Sparse, small tables keep eight and more steps of growth inside the exactness proof."""
    rng = np.random.default_rng(seed)
    U, I = 6 * B, 10 * B
    sizes = (61, I)[:F]                                 # not 7 rows: hot metadata rows would outgrow the proof
    params = make_params(rng, U, I, D, sizes, dense_users=0.0, item_vals=1, bias_vals=2)
    sparse_items = rng.random(I) < 0.75
    params["item.weight"][sparse_items] *= (rng.random((int(sparse_items.sum()), D)) < 4.0 / D)
    for f in range(len(sizes)):
        params[f"metadata.{f}.weight"] *= (rng.random(params[f"metadata.{f}.weight"].shape) < 2.0 / D)
    meta = item_meta(rng, I, sizes)
    steps = [B] * (n_steps - 1) + [B // 4]
    ids = make_ids(rng, steps, U, I)
    # one step where a single user row and item row take every lookup (pos == neg: gradients cancel)
    k = n_steps // 2
    lo = k * B
    ids[0][lo:lo + B], ids[1][lo:lo + B], ids[2][lo:lo + B] = ids[0][lo], ids[1][lo], ids[1][lo]
    return params, {k2: {} for k2 in params}, 0, ids, meta, steps


def two_step_case(seed, D, F, kind, B=256):
    rng = np.random.default_rng(seed)
    U, I = 6 * B, 10 * B
    sizes = (7, I)[:F]
    params = make_params(rng, U, I, D, sizes)
    meta = item_meta(rng, I, sizes)
    steps = [B, B // 4]
    ids = make_ids(rng, steps, U, I)
    return params, O.init_opt_state(params, spec_of(kind, HP2[kind])), 0, ids, meta, steps


def expected(case, spec):
    params, state, t0, (user, pos, neg), meta, steps = case
    p, s = copy_tree(params), copy_tree(state)
    loss = ref_epoch(p, s, batches(user, pos, neg, steps, meta), spec, t0)
    return loss, p, s


# --------------------------------------------------------------------------------------------------------------------
# CPU: the fixtures and the reference
# --------------------------------------------------------------------------------------------------------------------
FUSED_DIMS = (4, 6, 32, 64, 80, 128, 256, 500)          # every row shape of the fused kernel
SHARD_DIMS = (4, 12, 20, 36, 64, 100, 128, 132, 256, 260, 512)
ONE_USER_DIMS = (20, 128, 260)                            # sharded dims that run the "one_user" pattern
SHARD_SGD_DIMS = (4, 64, 128, 260)
TWO_STEP_DIMS = (4, 64, 256)


def _fused_cases():
    out = []
    for i, D in enumerate(FUSED_DIMS):
        for kind in ("sgd", "adagrad", "sparse_adam"):
            out.append((kind, D, (0, 2)[(i + len(kind)) % 2], "one_user" if i % 3 == 2 else "mixed"))
    return out


def _shard_cases():
    """Every dim at one rank on both kernels and on a group (2, 3, 4, 8 in turn); two chunks per lane where that
    changes the row shape (32 <= dim <= 128)."""
    out = []
    for i, D in enumerate(SHARD_DIMS):
        for kind in ("sgd", "adagrad", "sparse_adam"):
            out += [(kind, D, 1, 1, 1), (kind, D, 1, 0, 1), (kind, D, (2, 3, 4, 8)[(i + len(kind)) % 4], 1, 1)]
            if 32 <= D <= 128:
                out.append((kind, D, 1 + 2 * (i % 2), 1, 2))
    return out


def _sgd_cases():
    """(dim, metadata tables) of the fused SGD runs: metadata where its growth over nine steps stays in the proof."""
    return [(4, 2), (64, 2), (132, 0), (260, 0)]


def fused_case(kind, D, F, pattern):
    return one_step_case(D * 13 + F, D, F, kind, pattern)


def shard_case(kind, D, world):
    return one_step_case(D * 17 + world, D, 0, kind, "one_user" if D in ONE_USER_DIMS else "mixed")


def fused_sgd_case(D, F):
    return sgd_case(D * 5 + F, D, F)


def shard_sgd_case(D):
    return sgd_case(D * 7, D)


def two_step_fused_case(kind, D, F):
    return two_step_case(D * 19 + F, D, F, kind)


def two_step_shard_case(kind, D):
    return two_step_case(D * 23, D, 0, kind)


def _cover_ok(case):
    """The first step reaches single rows, rows with 2..8 and with more than 8 lookups in both id spaces, item rows
    only inactive samples look up, ties, inactive samples and pos == neg."""
    params, _, _, ids, meta, steps = case
    cover = exact_step(params, batches(*ids, steps, meta)[0])[2]
    for table in ("user.weight", "item.weight"):
        c = cover[table]
        assert c["single"] and c["2..8"] and c[">8"], (table, c)
    assert cover["item.weight"]["inactive only"] > 0 and cover["ties"] > 0 and cover["pos_eq_neg"] > 0, cover
    assert 0 < cover["inactive"] < len(ids[0]), cover
    return cover


def test_fixtures_pass_their_exactness_proof_and_take_every_reduce_path():
    """Every fixture the GPU tests of this file run: the proof holds at every step of the reference, and the ids take
    every reduce path (_cover_ok; the "one_user" pattern: one user row takes every user lookup of the step)."""
    for kind, D, F, pattern in _fused_cases():
        case = fused_case(kind, D, F, pattern)
        if pattern == "mixed":
            _cover_ok(case)
        else:
            assert exact_step(case[0], batches(*case[3], case[5], case[4])[0])[2]["user.weight"]["max"] == 256
        expected(case, spec_of(kind, HP[kind]))
    for kind, D, world, _, _ in _shard_cases():
        case = shard_case(kind, D, world)
        if D not in ONE_USER_DIMS:
            _cover_ok(case)
        expected(case, spec_of(kind, HP[kind]))
    for kind in HP2:
        for D in TWO_STEP_DIMS:
            for F in (0, 2):
                _cover_ok(two_step_fused_case(kind, D, F))
                expected(two_step_fused_case(kind, D, F), spec_of(kind, HP2[kind]))
            expected(two_step_shard_case(kind, D), spec_of(kind, HP2[kind]))
    sgd = [fused_sgd_case(D, F) for D, F in _sgd_cases()] + [shard_sgd_case(D) for D in SHARD_SGD_DIMS]
    for case in sgd:
        _cover_ok(case)
        loss, p, _ = expected(case, O.OptSpec("sgd", lr=float(case[5][0])))
        assert all(np.array_equal(np.round(v), v) for v in p.values())
        assert (loss > 0).all() and len(case[5]) >= 9


def test_a_fixture_that_could_round_is_refused():
    rng = np.random.default_rng(0)
    params = make_params(rng, 64, 64, 16)
    b = {"user": np.arange(8), "pos": np.arange(8), "neg": np.arange(8, 16)}
    exact_step(params, b)
    with pytest.raises(NotExact):
        exact_step(params, {k: v[:6] for k, v in b.items()})          # 1/6 is not dyadic
    big = {k: v * F32(2.0 ** 12) for k, v in params.items()}
    with pytest.raises(NotExact):
        exact_step(big, b)                                               # products beyond 2^24
    off = {k: v.copy() for k, v in params.items()}
    off["item.weight"][0, 0] = F32(0.1)
    with pytest.raises(NotExact):
        exact_step(off, b)                                               # not on a dyadic grid


def _port(params, F, dev="cpu"):
    from oracle.torch_port import LinearPort
    U, D = params["user.weight"].shape
    sizes = [params[f"metadata.{f}.weight"].shape[0] for f in range(F)]
    net = LinearPort(U, params["item.weight"].shape[0], sizes, D)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    return net.to(dev)


def _port_grads(net, b, F, dev="cpu"):
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in b.items()}
    from oracle.torch_port import hinge
    sp = net(t["user"], t["pos"], t.get("pos_meta"))
    sn = net(t["user"], t["neg"], t.get("neg_meta"))
    loss = hinge(sp, sn)
    net.zero_grad()
    loss.backward()
    return loss, {k: p.grad for k, p in net.named_parameters()}


@pytest.mark.parametrize("F", [0, 2])
@pytest.mark.parametrize("D", [4, 64, 500])
def test_exact_gradients_equal_torch_autograd(D, F):
    """The reference's loss and coalesced gradients equal LinearPort's (nn.Embedding(sparse=True) + autograd on
    the CPU) bit for bit."""
    params, _, _, ids, meta, steps = one_step_case(D * 3 + F, D, F, "sgd")
    b = batches(*ids, steps, meta)[0]
    loss, grads = exact_step(params, b)[:2]
    tl, tg = _port_grads(_port(params, F), b, F)
    assert tl.item() == float(loss)
    for k, (rows, G) in grads.items():
        c = tg[k].coalesce()
        assert np.array_equal(c.indices()[0].numpy(), rows), k
        assert np.array_equal(c.values().numpy(), G), k


def _torch_opt(kind, hp, params):
    if kind == "sgd":
        return torch.optim.SGD(params, lr=hp["lr"])
    if kind == "adagrad":
        return torch.optim.Adagrad(params, lr=hp["lr"], eps=hp["eps"], lr_decay=hp.get("lr_decay", 0.0))
    return torch.optim.SparseAdam(list(params), lr=hp["lr"], betas=hp["betas"], eps=hp["eps"])


def torch_step(case, kind, hp, dev):
    """torch.optim's own step of the case (first step only) on ``dev``: parameters, state and step count loaded,
    each table's gradient the per-lookup sparse tensor of the exact gradients, as the embedding backward emits it."""
    params, state, t0, ids, meta, steps = case
    b = batches(*ids, steps, meta)[0]
    lookups = exact_step(params, b)[3]
    ts = {k: torch.nn.Parameter(torch.from_numpy(v.copy()).to(dev)) for k, v in params.items()}
    opt = _torch_opt(kind, hp, list(ts.values()))
    for k, p in ts.items():
        for n, v in state[k].items():
            opt.state[p][n] = torch.from_numpy(v.copy()).to(dev)
        if kind == "adagrad":
            opt.state[p]["step"] = torch.tensor(float(t0))
        elif kind == "sparse_adam":
            opt.state[p]["step"] = t0
    for k, p in ts.items():
        ids, g = lookups[k]
        p.grad = torch.sparse_coo_tensor(torch.from_numpy(ids)[None].to(dev), torch.from_numpy(g).to(dev), p.shape,
                                         check_invariants=False)
    opt.step()
    return {k: p.detach().cpu().numpy() for k, p in ts.items()}, \
        {k: {n: v.cpu().numpy() for n, v in opt.state[p].items() if torch.is_tensor(v) and v.dim()} for k, p in ts.items()}


def test_reference_sgd_equals_torch_cpu_sgd():
    """Power-of-two lr: torch's per-lookup products and sums and the reference's single row update are exact alike."""
    for D, F in ((4, 0), (64, 2), (500, 2)):
        case = one_step_case(D + 5, D, F, "sgd")
        _, p, _ = expected(case, spec_of("sgd", HP["sgd"]))
        b = batches(*case[3], case[5], case[4])[0]
        net = _port(case[0], F)
        opt = torch.optim.SGD(net.parameters(), lr=HP["sgd"]["lr"])
        _port_grads(net, b, F)
        opt.step()
        for k, v in net.state_dict().items():
            assert np.array_equal(v.numpy(), p[k]), k


@pytest.mark.parametrize("kind", ["adagrad", "sparse_adam"])
def test_reference_state_equals_torch_cpu_state(kind):
    """From random state: the reference's sum / exp_avg / exp_avg_sq equal torch CPU's bit for bit (no sqrt, no
    fused product on that path).  The parameters are not compared: torch CPU's sqrt_ and axpy deviate (docstring)."""
    for D, F in ((4, 0), (64, 2), (500, 2)):
        case = one_step_case(D + 7, D, F, kind)
        _, _, s = expected(case, spec_of(kind, HP[kind]))
        _, ts = torch_step(case, kind, HP[kind], "cpu")
        for k in s:
            for n in s[k]:
                assert np.array_equal(ts[k][n], s[k][n]), (k, n)


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


def _to(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _assert_tables(got_p, got_s, want_p, want_s, init_p, what):
    """Every table and state tensor bit for bit; user_bias and its (zero) state untouched (SURVEY D12)."""
    for k in want_p:
        assert np.array_equal(got_p[k], want_p[k]), f"{what}: {k} ({int((got_p[k] != want_p[k]).sum())} entries differ)"
        if k == "user_bias.weight":
            assert np.array_equal(got_p[k], init_p[k]), f"{what}: user_bias must stay untouched"
        for n, w in want_s[k].items():
            g = got_s[k][n]
            assert np.array_equal(g, w), f"{what}: {k}.{n} ({int((g != w).sum())} entries differ)"
            if k == "user_bias.weight":
                assert not g.any(), f"{what}: user_bias state must stay 0"


def run_fused(case, kind, hp, tiled, monkeypatch, calls=1, max_steps=None):
    """EpochRunner on a Linear module loaded with the case's tables and optimizer state (optimizer.state + step):
    returns (losses, tables, state).  ``calls`` run() calls; ``max_steps``: launches of at most that many steps."""
    from torchrecsys_b200 import engine
    from torchrecsys_b200.collaborative.linear import Linear
    params, state, t0, (user, pos, neg), meta, steps = case
    dev = _dev()
    U, D = params["user.weight"].shape
    F = sum(k.startswith("metadata.") for k in params)
    sizes = {f"m{f}": params[f"metadata.{f}.weight"].shape[0] for f in range(F)}
    net = Linear(U, params["item.weight"].shape[0], sizes, D, use_metadata=F > 0, use_cuda=True)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    net = net.to(dev)
    opt = _torch_opt(kind, hp, net.parameters())
    for k, p in net.named_parameters():
        for n, v in state[k].items():
            opt.state[p][n] = _to(v, dev)
        if kind == "adagrad":
            opt.state[p]["step"] = torch.tensor(float(t0))
        elif kind == "sparse_adam":
            opt.state[p]["step"] = t0
    smp = {"user": user, "pos": pos, "neg": neg}
    if F:
        smp["pos_meta"], smp["neg_meta"] = meta[pos], meta[neg]
    smp = {k: _to(v, dev) for k, v in smp.items()}
    monkeypatch.setenv("TRS_PLAN_TILED", "1" if tiled else "0")
    if max_steps:
        monkeypatch.setattr(engine, "MAX_STEPS_PER_CALL", max_steps)
    B = steps[0]
    runner = engine.EpochRunner(net, opt)
    cut = (len(steps) // 2) * B if calls == 2 else len(user)
    loss = [runner.run({k: v[:cut] for k, v in smp.items()}, B)]
    if cut < len(user):
        loss.append(runner.run({k: v[cut:] for k, v in smp.items()}, B))
    torch.cuda.synchronize()
    names = dict(net.named_parameters())
    got_s = {k: {n: opt.state[names[k]][n].cpu().numpy() for n in state[k]} for k in params}
    return (torch.cat(loss).cpu().numpy(), {k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}, got_s)


@pytest.fixture
def shard_hooks():
    """The sharded kernel's settings are process-wide: back to their defaults afterwards, also on failure."""
    from torchrecsys_b200 import _lib
    L = _lib.lib()
    yield L
    L.trs_debug_shard_one_pass(1)
    L.trs_debug_shard_chunks_per_lane(1)


def run_sharded(case, kind, hp, world, L, one_pass=1, chunks=1, calls=1):
    """ShardedLinearTrainer on ``world`` emulated ranks, loaded through load_state_dict(params, optimizer_state);
    returns (losses, tables, state, whether the one-pass kernel ran)."""
    from torchrecsys_b200.sharded import ShardedLinearTrainer
    params, state, t0, (user, pos, neg), _, steps = case
    dev = _dev()
    U, D = params["user.weight"].shape
    L.trs_debug_shard_one_pass(one_pass)
    L.trs_debug_shard_chunks_per_lane(chunks)
    B = steps[0]
    tr = ShardedLinearTrainer(U, params["item.weight"].shape[0], D, global_batch=B, optimizer=kind, lr=hp["lr"],
                              device=dev, betas=hp.get("betas", (0.9, 0.999)), eps=hp.get("eps"),
                              lr_decay=hp.get("lr_decay", 0.0), emulate_world=world, timeout_ms=5000)
    ost = None if kind == "sgd" else {k: dict({n: torch.from_numpy(v) for n, v in state[k].items()}, step=t0)
                                      for k in BASE_KEYS}
    tr.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, ost)
    u, p, q = (_to(a, dev) for a in (user, pos, neg))
    cut = (len(steps) // 2) * B if calls == 2 else len(user)
    loss = [tr.train_epoch(u[:cut], p[:cut], q[:cut], B)]
    if cut < len(user):
        loss.append(tr.train_epoch(u[cut:], p[cut:], q[cut:], B))
    ran_one = L.trs_debug_shard_last_one_pass()
    gs = tr.optimizer_state_dict()
    got_s = {k: {n: gs[k][n].cpu().numpy().reshape(params[k].shape) for n in state[k]} for k in BASE_KEYS}
    got_p = {k: v.cpu().numpy().reshape(params[k].shape) for k, v in tr.state_dict().items()}
    tr.close()
    return torch.cat(loss).cpu().numpy(), got_p, got_s, ran_one


def _check(case, kind, hp, got, what):
    want_l, want_p, want_s = expected(case, spec_of(kind, hp))
    assert np.array_equal(got[0], want_l), f"{what}: losses {got[0]} != {want_l}"
    _assert_tables(got[1], got[2], want_p, want_s, case[0], what)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sgd", "adagrad", "sparse_adam"])
def test_torch_cuda_optimizers_follow_the_reference(kind):
    """torch.optim on CUDA steps the fixture from random state exactly as the reference does (module docstring): this
    pins which products torch rounds before the sum (Adagrad's add_(sparse, alpha=-clr) included) and that its CUDA
    sqrt and division are correctly rounded."""
    for D, F in ((4, 0), (64, 2), (500, 2)):
        case = one_step_case(D + 11, D, F, kind)
        _, want_p, want_s = expected(case, spec_of(kind, HP[kind]))
        got_p, got_s = torch_step(case, kind, HP[kind], _dev())
        for k in want_p:
            assert np.array_equal(got_p[k], want_p[k]), f"{k}: {int((got_p[k] != want_p[k]).sum())} entries differ"
            for n in want_s[k]:
                assert np.array_equal(got_s[k][n], want_s[k][n]), (k, n)


@pytest.mark.gpu
@pytest.mark.parametrize("tiled", [0, 1])
@pytest.mark.parametrize("kind,D,F,pattern", _fused_cases())
def test_fused_step_from_any_state_is_exact(kind, D, F, pattern, tiled, monkeypatch):
    """One step of the fused kernel (csrc/train.cu) from random optimizer state, every table and state tensor
    compared with torch.equal, rows nobody looked up included; both plan builders."""
    case = fused_case(kind, D, F, pattern)
    got = run_fused(case, kind, HP[kind], tiled, monkeypatch)
    _check(case, kind, HP[kind], got, f"fused {kind} D={D} F={F} {pattern} tiled={tiled}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,D,world,one_pass,chunks", _shard_cases())
def test_sharded_step_from_any_state_is_exact(kind, D, world, one_pass, chunks, shard_hooks):
    """One step of the row-sharded kernel (csrc/shard.cu) from random optimizer state, loaded through
    load_state_dict(params, optimizer_state): the one-pass kernel (one rank, dim <= 128), the two-phase kernel, and
    two chunks per lane -- bit-comparable with the reference, and so with each other, on these fixtures."""
    case = shard_case(kind, D, world)
    got = run_sharded(case, kind, HP[kind], world, shard_hooks, one_pass, chunks)
    assert got[3] == int(one_pass == 1 and world == 1 and chunks == 1 and D <= 128)
    _check(case, kind, HP[kind], got[:3], f"sharded {kind} D={D} world={world} one_pass={one_pass} chunks={chunks}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sgd", "adagrad", "sparse_adam"])
def test_sharded_batch_smaller_than_the_group(kind, shard_hooks):
    """Eight ranks, steps of 4 and 1 samples: most ranks own no sample of a step and still update their rows."""
    rng = np.random.default_rng(3)
    U, I, D = 40, 60, 36
    params = make_params(rng, U, I, D)
    ids = make_ids(rng, [4, 4, 1], U, I)
    case = (params, random_state(rng, params, kind, spec_of(kind, HP[kind]).eps), 7, ids, None, [4, 4, 1])
    # each step launched on its own from the same tables and state: after a step from random state the tables leave
    # the grid, so only a first step is exact
    for s in range(3):
        sub = (case[0], case[1], case[2], tuple(a[4 * s:4 * s + case[5][s]] for a in ids), None, [case[5][s]])
        got = run_sharded(sub, kind, HP[kind], 8, shard_hooks)
        _check(sub, kind, HP[kind], got[:3], f"world 8, batch {sub[5][0]}")




@pytest.mark.gpu
@pytest.mark.parametrize("D,F", _sgd_cases())
def test_fused_sgd_many_steps_are_exact(D, F, monkeypatch):
    """Nine SGD steps with lr = B: one launch (both plan builders), launches of four steps, two run() calls -- all
    equal to the reference.  A row read before the previous step's update is visible changes an integer score."""
    case = fused_sgd_case(D, F)
    hp = dict(lr=float(case[5][0]))
    for tiled, calls, max_steps in ((0, 1, None), (1, 1, None), (0, 1, 4), (1, 2, None)):
        got = run_fused(case, "sgd", hp, tiled, monkeypatch, calls, max_steps)
        _check(case, "sgd", hp, got, f"fused sgd D={D} F={F} tiled={tiled} calls={calls} max_steps={max_steps}")


@pytest.mark.gpu
@pytest.mark.parametrize("D", SHARD_SGD_DIMS)
def test_sharded_sgd_many_steps_are_exact(D, shard_hooks):
    """The row-sharded kernels over nine SGD steps (lr = B): one rank on both kernels, two and eight ranks, two
    chunks per lane, and the epoch in two train_epoch calls."""
    case = shard_sgd_case(D)
    hp = dict(lr=float(case[5][0]))
    runs = [(1, 1, 1, 1), (1, 0, 1, 1), (3, 1, 1, 1), (8, 1, 1, 1), (1, 1, 1, 2), (2, 1, 1, 2)]
    if 32 <= D <= 128:
        runs.append((1, 1, 2, 1))
    for world, one_pass, chunks, calls in runs:
        got = run_sharded(case, "sgd", hp, world, shard_hooks, one_pass, chunks, calls)
        _check(case, "sgd", hp, got[:3], f"sharded sgd D={D} world={world} one_pass={one_pass} chunks={chunks} "
                                          f"calls={calls}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["adagrad", "sparse_adam"])
@pytest.mark.parametrize("D", TWO_STEP_DIMS)
def test_two_steps_from_fresh_state(kind, D, shard_hooks, monkeypatch):
    """Fresh state, eps = 2^-100, lr = 1/2 (SparseAdam: betas (0.5, 0.75), |G| with at most 12 significant bits):
    step 1 moves every entry by exactly +-lr or 0, so step 2's scores are exact again and step 2 -- which reads the
    state and the rows step 1 wrote -- is compared bit for bit.  Fused kernel (F = 0 and 2) and sharded kernels."""
    hp = HP2[kind]
    for F in (0, 2):
        case = two_step_fused_case(kind, D, F)
        params, _, _, ids, meta, steps = case
        b1 = batches(*ids, steps, meta)[0]
        for rows, G in exact_step(params, b1)[1].values():
            m, _ = np.frexp(G[G != 0].astype(np.float64) * 2.0 ** 40)
            assert np.array_equal(np.round(m * 2.0 ** 12), m * 2.0 ** 12), "|G| has more than 12 significant bits"
        got = run_fused(case, kind, hp, F, monkeypatch)
        _check(case, kind, hp, got, f"fused {kind} D={D} F={F}")
    case = two_step_shard_case(kind, D)
    for world, one_pass in ((1, 1), (1, 0), (4, 1)):
        got = run_sharded(case, kind, hp, world, shard_hooks, one_pass)
        _check(case, kind, hp, got[:3], f"sharded {kind} D={D} world={world} one_pass={one_pass}")


@pytest.mark.gpu
@pytest.mark.parametrize("F", [0, 2])
@pytest.mark.parametrize("D", [4, 64, 500])
def test_autograd_backward_equals_the_cpu_port(D, F):
    """trs_scores_backward through the autograd-visible forward: the loss and the coalesced sparse gradient of every
    table equal LinearPort's on the CPU bit for bit."""
    from torchrecsys_b200.collaborative.linear import Linear
    from torchrecsys_b200.helper.loss import hinge_loss
    params, _, _, ids, meta, steps = one_step_case(D * 29 + F, D, F, "sgd")
    b = batches(*ids, steps, meta)[0]
    dev = _dev()
    U, _ = params["user.weight"].shape
    sizes = {f"m{f}": params[f"metadata.{f}.weight"].shape[0] for f in range(F)}
    net = Linear(U, params["item.weight"].shape[0], sizes, D, use_metadata=F > 0, use_cuda=True)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()})
    net = net.to(dev)
    t = {k: _to(v, dev) for k, v in b.items()}
    sp = net.forward(t, "user", "pos", "pos_meta" if F else None)
    sn = net.forward(t, "user", "neg", "neg_meta" if F else None)
    loss = hinge_loss(sp, sn)
    loss.backward()
    want_l, want_g = _port_grads(_port(params, F), b, F)
    assert loss.item() == want_l.item()
    for k, p in net.named_parameters():
        g, w = p.grad.coalesce().cpu(), want_g[k].coalesce()
        assert torch.equal(g.indices(), w.indices()), k
        assert torch.equal(g.values(), w.values()), k
