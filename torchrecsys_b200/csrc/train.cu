// train.cu -- fused forward + hinge + backward + segmented reduce + row-wise optimizer for the
// Linear and FM scorers, as ONE persistent cooperative kernel over many steps.
//
// Per step (reference model.py:274-284):
//   phase A  one row group per sample: gather u, v+, v- (+ metadata rows), both scores, hinge,
//            closed-form gradient rows (SURVEY.md a7).  A user / item row that this step looks up exactly
//            ONCE (plan.cuh: single_*; >90 % of the lookups under uniform ids) has no other reader or writer
//            in the step, so the sample's own row group applies the optimizer update to it right here:
//            parameter and optimizer-state rows are fetched together with the gather, updated in registers
//            and written once.  Every other gradient row goes to an L2-resident staging buffer.
//   grid barrier (staged rows complete; every score of the step was computed from pre-update parameters)
//   phase B  long segments (rows with > LONG_SEG_T lookups: the small metadata tables, hot rows) are reduced
//            by a whole CTA -- its row groups sum strided subsets of the staged rows, the partial sums are
//            added in group order through shared memory, one group updates the row; short segments (2..T
//            lookups, and every metadata row) stream through a per-thread cp.async ring: param + state rows
//            fetched before the barrier, staged gradient rows after it, duplicates summed in lookup order.
//            Right after its phase A every row group starts copying the rows (parameters AND optimizer state)
//            of its NEXT step's samples into shared memory -- all but the rows this step itself looks up
//            (plan flag bit 1), which are read after the step's last barrier.
//   grid barrier
// HBM traffic per step is ids + (param+state read, param+state write) per unique touched row; staging and plan
// are served from L2.  Nothing depends on the order in which CTAs or row groups run: every floating-point sum
// has a fixed association (deterministic results).
//
// NET == TRS_NET_MLP: phase A is skipped -- the gradient rows were staged by the tower's backward (mlp.cu).
#include <stdlib.h>

#include "plan.cuh"
#include "ptx.cuh"
#include "scorer.cuh"
#include "train.cuh"

namespace trs {

constexpr int MF = 1;  // metadata features whose rows are kept in registers between fwd and bwd

struct PlanPtrs {
    const uint32_t *user_key, *user_perm, *item_key, *item_perm;
    const uint32_t* meta_key[TRS_MAX_META];
    const uint32_t* meta_perm[TRS_MAX_META];
    const uint32_t* item_cnt;
    const uint32_t* long_cnt;
    const uint8_t* single_user;
    const uint8_t* single_item;
    const uint4* items;
    const uint4* long_segs;
    int item_cap, long_cap;
};

struct Stage {
    float* gU;                 // [B, dim]
    float* gI;                 // [2B, dim]
    float* gM[TRS_MAX_META];   // FM / MLP: [2B, dim]
    float* gbU;                // FM only: [B]
    float* gbI;                // [2B]  (FM: also the gradient of linear_metadata, d w_k = delta)
    float* loss_part;          // [n_steps, gridDim.x]
    unsigned* barrier;         // [1] monotonically increasing arrival counter
    unsigned long long* trace; // debug (TRS_DEBUG_SKIP & 64): [n_steps, gridDim.x, 16] globaltimer stamps
};

struct StageLayout {
    size_t gU, gI, gM[TRS_MAX_META], gbU, gbI, loss_part, sync_words, trace, total;
    size_t sync_bytes;
};

static StageLayout stage_layout(const trs_model* m, const trs_epoch* ep, int grid) {
    StageLayout L;
    size_t off = 0;
    auto take = [&](size_t n_floats) {
        size_t o = off;
        off += (n_floats * sizeof(float) + 255) / 256 * 256;
        return o;
    };
    const size_t B = (size_t)ep->batch, D = (size_t)m->dim;
    L.gU = take(B * D);
    L.gI = take(2 * B * D);
    for (int f = 0; f < TRS_MAX_META; ++f) L.gM[f] = (m->net != TRS_NET_LINEAR && f < m->n_meta) ? take(2 * B * D) : 0;
    L.gbU = take(B);
    L.gbI = take(2 * B);
    L.loss_part = take((size_t)n_steps_of(ep) * grid);
    L.sync_words = off;  // barrier[1] (+ padding); zeroed before every launch
    L.sync_bytes = 64 * sizeof(unsigned);
    off += (L.sync_bytes + 255) / 256 * 256;
    L.trace = take((size_t)n_steps_of(ep) * grid * 16 * 2);
    L.total = off;
    return L;
}

// ---- small device helpers -------------------------------------------------------------------
template <int V, int G, int IT>
__device__ __forceinline__ void prefetch_row(const float* base, int nch, int gl) {
#pragma unroll
    for (int i = 0; i < IT; ++i) {
        const int c = gl + i * G;
        if (c < nch) prefetch_l2(base + (size_t)c * V);
    }
}
template <int V, int IT>
__device__ __forceinline__ Row<V, IT> row_scaled_diff(float a, const Row<V, IT>& x,
                                                      const Row<V, IT>& y) {  // a*(x-y)
    Row<V, IT> r;
#pragma unroll
    for (int i = 0; i < IT; ++i)
#pragma unroll
        for (int k = 0; k < V; ++k) r.c[i][k] = a * (x.c[i][k] - y.c[i][k]);
    return r;
}
template <int V, int IT>
__device__ __forceinline__ Row<V, IT> row_scaled(float a, const Row<V, IT>& x) {
    Row<V, IT> r;
#pragma unroll
    for (int i = 0; i < IT; ++i)
#pragma unroll
        for (int k = 0; k < V; ++k) r.c[i][k] = a * x.c[i][k];
    return r;
}

// Grid-wide barrier for a cooperative launch (all CTAs resident).  `counter` only ever grows:
// after the g-th barrier it holds g * gridDim.x.  One release fence on the way in (bar.sync before it: the stores of
// the whole CTA happen before the fence), a relaxed add, relaxed polling, one acquire load on the way out -- acq_rel
// fences instead of the sequentially-consistent __threadfence() (= fence.sc.gpu), which measured ~1 us more per
// barrier on the row-sharded kernel (csrc/shard.cu).
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& target) {
    __syncthreads();
    target += gridDim.x;
    if (threadIdx.x == 0) {
        fence_acq_rel_gpu();
        red_relaxed_gpu(counter);
        while ((int)(ld_relaxed_gpu(counter) - target) < 0) {
        }
        (void)ld_acquire_gpu(counter);
    }
    __syncthreads();
}

// Which arrays an id space (0 user, 1 item, 2+f metadata f) reduces from / updates.
struct SpaceRef {
    const trs_table* t;
    const uint32_t* K;
    const uint32_t* P;
    const float* stage;
    const float* stage_lin;
};

template <int NET>
__device__ __forceinline__ SpaceRef resolve_space(int space, const trs_model& m, const PlanPtrs& plan,
                                                  const Stage& st, int64_t lo) {
    SpaceRef r;
    if (space == 0) {
        r = {&m.user, plan.user_key + lo, plan.user_perm + lo, st.gU, NET == TRS_NET_FM ? st.gbU : nullptr};
    } else if (space == 1) {
        r = {&m.item, plan.item_key + 2 * lo, plan.item_perm + 2 * lo, st.gI, st.gbI};
    } else {
        const int f = space - 2;
        r = {&m.meta[f], plan.meta_key[f] + 2 * lo, plan.meta_perm[f] + 2 * lo,
             NET != TRS_NET_LINEAR ? st.gM[f] : st.gI, NET == TRS_NET_FM ? st.gbI : nullptr};
    }
    if (!r.t->lin) r.stage_lin = nullptr;
    return r;
}

// the width-1 companion of a row (bias / first-order weight), one thread
__device__ __forceinline__ void update_lin(const trs_table& t, uint32_t key, const OptScalars& o, float scale, float g) {
    float pl = __ldcg(t.lin + key), l0 = 0.f, l1 = 0.f;
    if (o.kind != TRS_OPT_SGD) l0 = __ldcg(t.lin_s0 + key);
    if (o.kind == TRS_OPT_SPARSE_ADAM) l1 = __ldcg(t.lin_s1 + key);
    update_store_lin(t, key, o, scale, g, pl, l0, l1);
}

// ---- cp.async ring: per-thread prefetch slots in shared memory (V == 4 only) -------------------
// Every lane copies only the 16-byte chunks it will itself consume, so no cross-thread
// synchronisation is needed: cp.async.wait_group makes a thread's own copies visible to it.
constexpr int RING = 4;
#ifndef TRS_TRAIN_T1
#define TRS_TRAIN_T1 512  // threads per CTA for rows of <= 32 chunks (tuning hook: -DTRS_TRAIN_T1=256|384|512)
#endif
template <int V, int IT>
constexpr int train_threads() { return V == 1 ? 256 : (IT == 1 ? TRS_TRAIN_T1 : (IT == 2 ? 256 : 128)); }
template <int V, int IT>
constexpr size_t ring_smem_bytes() {
    return V == 1 ? 0 : (size_t)train_threads<V, IT>() * (2 * RING * 16 + RING * 4 * IT * 16);
}
// Linear / FM use the same region for the early fetch of the NEXT step's rows instead (the ring only serves
// the MLP tower's staged mode there): PF samples per row group x 9 rows (param, s0, s1 of user / pos / neg),
// thread-private 16-byte slots like the ring's.
constexpr int MLIN_CAP = 2048;  // a metadata first-order table up to this many rows is cached in shared memory
constexpr int PF = 2;
constexpr int PF_ROWS = 11;  // 0-8: {param, s0, s1} x {user, positive item, negative item}; 9, 10: metadata rows
template <int V, int IT>
constexpr size_t front_smem_bytes() {
    const size_t pf = V == 1 ? 0 : (size_t)train_threads<V, IT>() * PF * PF_ROWS * IT * 16;
    return pf > ring_smem_bytes<V, IT>() ? pf : ring_smem_bytes<V, IT>();
}
// + the partial sums of a CTA-cooperative long-segment reduce: one row slice per thread, one scalar per group
template <int V, int IT>
constexpr size_t train_smem_bytes() {
    return front_smem_bytes<V, IT>() + (size_t)train_threads<V, IT>() * (IT * V * 4 + 4) + MLIN_CAP * 4;
}

template <int NT, int IT>
struct Ring {
    uint4* desc;   // [2*RING][NT]
    float4* rows;  // [RING][4 fields: p, s0, s1, grad][IT][NT]
    __device__ __forceinline__ uint4* d(int n) const { return desc + (n % (2 * RING)) * NT + threadIdx.x; }
    __device__ __forceinline__ float4* r(int n, int f, int i) const {
        return rows + (((n % RING) * 4 + f) * IT + i) * NT + threadIdx.x;
    }
};

// ids of one sample, as 32-bit row numbers (every table has < 2^32 rows, checked by plan_build)
struct SampleIds {
    uint32_t u, ip, in, pm[MF], nm[MF];
};
__device__ __forceinline__ SampleIds load_ids(const trs_epoch& ep, int64_t smp, int F) {
    SampleIds r;
    r.u = (uint32_t)ep.user[smp];
    r.ip = (uint32_t)ep.pos[smp];
    r.in = (uint32_t)ep.neg[smp];
#pragma unroll
    for (int f = 0; f < MF; ++f) {
        r.pm[f] = f < F ? (uint32_t)ep.pos_meta[smp * F + f] : 0u;
        r.nm[f] = f < F ? (uint32_t)ep.neg_meta[smp * F + f] : 0u;
    }
    return r;
}

// ids and plan flags of one sample.  fl: byte 0 user flags, byte 1 positive item, byte 2 negative item.
struct SampleRec {
    uint32_t u, ip, in, pm, nm, fl;
};
constexpr int REC_WORDS = 6;
// word f of the record of sample b of the step starting at lo
__device__ __forceinline__ uint32_t load_rec_word(const trs_epoch& ep, const uint8_t* single_user,
                                                  const uint8_t* single_item, int64_t lo, int Bs, int b, int F, int f) {
    const int64_t smp = lo + b;
    switch (f) {
        case 0: return (uint32_t)ep.user[smp];
        case 1: return (uint32_t)ep.pos[smp];
        case 2: return (uint32_t)ep.neg[smp];
        case 3: return F ? (uint32_t)ep.pos_meta[smp * F] : 0u;
        case 4: return F ? (uint32_t)ep.neg_meta[smp * F] : 0u;
        default:
            return (uint32_t)single_user[lo + b] | ((uint32_t)single_item[2 * lo + b] << 8) |
                   ((uint32_t)single_item[2 * lo + Bs + b] << 16);
    }
}

// optimizer state of a row that phase A updates itself (zeros where the optimizer has none / not fused)
template <int V, int G, int IT>
__device__ __forceinline__ void load_state_rows(const trs_table& t, size_t roff, int nch, int gl, int kind, bool fused,
                                                Row<V, IT>& s0, Row<V, IT>& s1) {
    row_zero(s0);
    row_zero(s1);
    if (fused && kind != TRS_OPT_SGD) s0 = load_row_cg<V, G, IT>(t.emb_s0 + roff, nch, gl);
    if (fused && kind == TRS_OPT_SPARSE_ADAM) s1 = load_row_cg<V, G, IT>(t.emb_s1 + roff, nch, gl);
}

// ---- the kernel -------------------------------------------------------------------------------
template <int NET, int V, int G, int IT>
__global__ void __launch_bounds__((train_threads<V, IT>()), 1)
train_kernel(const __grid_constant__ trs_model m, const __grid_constant__ trs_epoch ep,
             const __grid_constant__ OptScalars opt, const __grid_constant__ PlanPtrs plan,
             const __grid_constant__ Stage st, const int first_step, const int n_steps,
             float* __restrict__ loss_out, const int dbg) {
    constexpr int NT = train_threads<V, IT>();
    constexpr bool RINGED = (V == 4) && NET == TRS_NET_MLP;   // cp.async ring for the short segments
    constexpr bool PFETCH = (V == 4) && NET != TRS_NET_MLP;   // early shared-memory fetch of the next step's rows
    __shared__ float s_loss[NT / 32];
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Ring<NT, IT> ring;
    ring.desc = reinterpret_cast<uint4*>(smem_raw);
    ring.rows = reinterpret_cast<float4*>(smem_raw + (size_t)2 * RING * NT * sizeof(uint4));
    float* s_part = reinterpret_cast<float*>(smem_raw + front_smem_bytes<V, IT>());  // [GPB][IT][G][V]
    float* s_part_lin = s_part + (size_t)NT * IT * V;                                // [GPB]
    // FM: every sample reads linear_metadata.0 -- a table of a few cache lines that the whole GPU would hammer
    // at once; each CTA takes one coalesced copy per step instead
    float* s_mlin = s_part_lin + NT;                                                 // [MLIN_CAP]
    const bool mlin_cached = NET == TRS_NET_FM && m.n_meta > 0 && m.meta[0].lin != nullptr &&
                             m.meta[0].n_rows <= MLIN_CAP && (m.meta[0].n_rows & 3) == 0;

    const int dim = m.dim, nch = dim / V, F = m.n_meta;
    const int gl = threadIdx.x % G;
    constexpr int GPW = 32 / G;                        // groups per warp
    constexpr int GPB = NT / G;                        // groups per block
    const int g_in_cta = threadIdx.x / G;
    const int gid = blockIdx.x * GPB + g_in_cta;
    const int ngroups = gridDim.x * GPB;
    const int gid_warp0 = gid - (gid % GPW);           // first group of my warp
    const int kind = opt.kind;
    unsigned bar_target = 0;
    float4* pf_base = reinterpret_cast<float4*>(smem_raw);
    // slot of (sample k of this group, row r: 3*table + {param, s0, s1}, chunk a) in the early-fetch region
    auto pf_slot = [&](int k, int r, int a) { return pf_base + (((k * PF_ROWS + r) * IT + a) * NT + threadIdx.x); };
    auto pf_issue = [&](int k, int r, const float* row) {
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int c = gl + a * G;
            if (c < nch) cp_async16(pf_slot(k, r, a), row + (size_t)c * 4);
        }
    };
    auto pf_row = [&](int k, int r) {
        Row<V, IT> x;
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int c = gl + a * G;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < nch) v = *pf_slot(k, r, a);
            x.c[a][0] = v.x; x.c[a][V > 1 ? 1 : 0] = v.y; x.c[a][V > 2 ? 2 : 0] = v.z; x.c[a][V > 3 ? 3 : 0] = v.w;
        }
        return x;
    };
    // The records (ids + flags) of my group's first PF samples are held one WORD PER LANE (lane w % G keeps word
    // w of the PF * REC_WORDS words) and broadcast by shuffles: they cross the step barrier in a single register.
    constexpr int WPL = (PF * REC_WORDS + G - 1) / G;
    auto rec_load = [&](uint32_t (&w)[WPL], int64_t lo_, int Bs_) {
#pragma unroll
        for (int i = 0; i < WPL; ++i) {
            const int idx = gl + i * G;
            w[i] = 0u;
            if (idx < PF * REC_WORDS && Bs_ > 0) {
                const int k = idx / REC_WORDS;
                w[i] = load_rec_word(ep, plan.single_user, plan.single_item, lo_, Bs_, min(gid + k * ngroups, Bs_ - 1), F,
                                     idx % REC_WORDS);
            }
        }
    };
    auto rec_get = [&](const uint32_t (&w)[WPL], int k) {   // every lane of the warp must call this
        uint32_t f[REC_WORDS];
#pragma unroll
        for (int q = 0; q < REC_WORDS; ++q) {
            const int idx = k * REC_WORDS + q;
            uint32_t v = w[0];
#pragma unroll
            for (int i = 1; i < WPL; ++i) v = (idx / G == i) ? w[i] : v;
            f[q] = __shfl_sync(0xffffffffu, v, idx % G, G);
        }
        SampleRec r = {f[0], f[1], f[2], f[3], f[4], f[5]};
        return r;
    };
    unsigned have = 0;  // bit 3k+t: the param (+ state, if fused) row of table t of my sample k sits in shared memory

    // ---- ring stages (phase B), item n of this group = global item n*ngroups + gid ----
    auto issue_desc = [&](const uint4* items, int n_items, int n) {
        const int i = n * ngroups + gid;
        if (RINGED && i < n_items) cp_async16(ring.d(n), items + i);
    };
    auto issue_state = [&](int n_items, int n, int64_t lo) {   // needs desc n landed
        const int i = n * ngroups + gid;
        if (!RINGED || i >= n_items) return;
        const uint4 it = *ring.d(n);
        const SpaceRef sp = resolve_space<NET>((int)(it.x & 0xffu), m, plan, st, lo);
        const size_t roff = (size_t)it.z * dim;
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int c = gl + a * G;
            if (c < nch) {
                cp_async16(ring.r(n, 0, a), sp.t->emb + roff + (size_t)c * 4);
                if (kind != TRS_OPT_SGD) cp_async16(ring.r(n, 1, a), sp.t->emb_s0 + roff + (size_t)c * 4);
                if (kind == TRS_OPT_SPARSE_ADAM) cp_async16(ring.r(n, 2, a), sp.t->emb_s1 + roff + (size_t)c * 4);
            }
        }
    };
    auto issue_grad = [&](int n_items, int n, int64_t lo) {    // after the barrier: staged gradient row
        const int i = n * ngroups + gid;
        if (!RINGED || i >= n_items) return;
        const uint4 it = *ring.d(n);
        const SpaceRef sp = resolve_space<NET>((int)(it.x & 0xffu), m, plan, st, lo);
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int c = gl + a * G;
            if (c < nch) cp_async16(ring.r(n, 3, a), sp.stage + (size_t)it.w * dim + (size_t)c * 4);
        }
    };
    auto consume = [&](const uint4* items, int n_items, int n, int64_t lo, float scale) {
        const int i = n * ngroups + gid;
        if (i >= n_items) return;
        uint4 it;
        Row<V, IT> p, s0, s1, g;
        row_zero(s0);
        row_zero(s1);
        if (RINGED) {
            it = *ring.d(n);
#pragma unroll
            for (int a = 0; a < IT; ++a) {
                const int c = gl + a * G;
                if (c < nch) {
                    const float4 vp = *ring.r(n, 0, a), vg = *ring.r(n, 3, a);
                    p.c[a][0] = vp.x; p.c[a][V > 1 ? 1 : 0] = vp.y; p.c[a][V > 2 ? 2 : 0] = vp.z; p.c[a][V > 3 ? 3 : 0] = vp.w;
                    g.c[a][0] = vg.x; g.c[a][V > 1 ? 1 : 0] = vg.y; g.c[a][V > 2 ? 2 : 0] = vg.z; g.c[a][V > 3 ? 3 : 0] = vg.w;
                    if (kind != TRS_OPT_SGD) {
                        const float4 v0 = *ring.r(n, 1, a);
                        s0.c[a][0] = v0.x; s0.c[a][V > 1 ? 1 : 0] = v0.y; s0.c[a][V > 2 ? 2 : 0] = v0.z; s0.c[a][V > 3 ? 3 : 0] = v0.w;
                    }
                    if (kind == TRS_OPT_SPARSE_ADAM) {
                        const float4 v1 = *ring.r(n, 2, a);
                        s1.c[a][0] = v1.x; s1.c[a][V > 1 ? 1 : 0] = v1.y; s1.c[a][V > 2 ? 2 : 0] = v1.z; s1.c[a][V > 3 ? 3 : 0] = v1.w;
                    }
                } else {
                    p.c[a] = Vec<V>::zero();
                    g.c[a] = Vec<V>::zero();
                }
            }
        } else {
            it = items[i];
        }
        const SpaceRef sp = resolve_space<NET>((int)(it.x & 0xffu), m, plan, st, lo);
        const size_t roff = (size_t)it.z * dim;
        if (!RINGED) {
            g = load_row_cg<V, G, IT>(sp.stage + (size_t)it.w * dim, nch, gl);
            p = load_row_cg<V, G, IT>(sp.t->emb + roff, nch, gl);
            if (kind != TRS_OPT_SGD) s0 = load_row_cg<V, G, IT>(sp.t->emb_s0 + roff, nch, gl);
            if (kind == TRS_OPT_SPARSE_ADAM) s1 = load_row_cg<V, G, IT>(sp.t->emb_s1 + roff, nch, gl);
        }
        const int c = (int)((it.x >> 8) & 0xffu);
        for (int q = 1; q < c; ++q) {  // duplicates, in lookup order
            const uint32_t j = sp.P[it.y + q];
            row_acc(g, load_row_cg<V, G, IT>(sp.stage + (size_t)j * dim, nch, gl));
        }
        update_store_row<V, G, IT>(*sp.t, roff, nch, gl, opt, scale, p, s0, s1, g);
    };

    // ---- prologue: what step `first_step` needs before its phase A ----
    int n_items_cur = 0, n_long_cur = 0;
    uint32_t curw[WPL], nxtw[WPL];  // record words of the current / next step (see rec_load)
#pragma unroll
    for (int i = 0; i < WPL; ++i) curw[i] = nxtw[i] = 0u;
    {
        const int64_t s0i = first_step;
        const int64_t lo0 = s0i * (int64_t)ep.batch;
        const int Bs0 = (int)min((int64_t)ep.batch, ep.n_samples - lo0);
        n_items_cur = min((int)plan.item_cnt[s0i], plan.item_cap);
        n_long_cur = min((int)plan.long_cnt[s0i], plan.long_cap);
        if (NET != TRS_NET_MLP) rec_load(curw, lo0, Bs0);
        const uint4* items0 = plan.items + (size_t)s0i * plan.item_cap;
        for (int n = 0; n < 2 * RING; ++n) issue_desc(items0, n_items_cur, n);
        cp_async_commit();
    }

    for (int si = 0; si < n_steps; ++si) {
        const int64_t s = first_step + si;
        const int64_t lo = s * (int64_t)ep.batch;
        const int Bs = (int)min((int64_t)ep.batch, ep.n_samples - lo);
        const float invB = 1.0f / (float)Bs;
        const uint4* items = plan.items + (size_t)s * plan.item_cap;
        const int n_items = n_items_cur, n_long = n_long_cur;
        const float scale = opt.step_scale[s];
        // what the next step will need (loaded now, used after two barriers)
        int n_items_next = 0, n_long_next = 0;
        const int64_t lo2 = lo + ep.batch;
        const int Bs2 = (si + 1 < n_steps) ? (int)min((int64_t)ep.batch, ep.n_samples - lo2) : 0;
        if (si + 1 < n_steps) {
            n_items_next = min((int)plan.item_cnt[s + 1], plan.item_cap);
            n_long_next = min((int)plan.long_cnt[s + 1], plan.long_cap);
            if (NET != TRS_NET_MLP) rec_load(nxtw, lo2, Bs2);
        }
        // width-1 companion work of this thread (phase B): descriptor fetched now
        const int lin_i = threadIdx.x * gridDim.x + blockIdx.x;  // every CTA gets every gridDim-th item
        uint4 lin_it = make_uint4(0, 0, 0, 0);
        if (lin_i < n_items) lin_it = items[lin_i];

        // debug trace: slots 0-7 by thread 0, 8-15 by thread NT/2
        const bool tracing = (dbg & 64) && threadIdx.x == 0;
        unsigned long long* tr = st.trace + ((size_t)si * gridDim.x + blockIdx.x) * 16;
        if (tracing) tr[0] = global_ns();
        // ------------------------------ phase A ------------------------------------------
        float hsum = 0.f;
        if (mlin_cached) {
            for (int i = threadIdx.x * 4; i < (int)m.meta[0].n_rows; i += NT * 4)
                *reinterpret_cast<float4*>(s_mlin + i) = __ldcg(reinterpret_cast<const float4*>(m.meta[0].lin + i));
        }
        if (PFETCH) {
            cp_async_wait(0);  // my own copies of this step's rows (issued during the last phase B)
            // the metadata rows of my first two samples (updated by every step: L2-hot) -> shared memory,
            // issued together so that the second sample does not wait for them again
            if (F > 0 && NET != TRS_NET_MLP) {
#pragma unroll
                for (int k = 0; k < PF; ++k) {
                    const SampleRec r = rec_get(curw, k);
                    if (gid + k * ngroups < Bs) {
                        pf_issue(k, 9, m.meta[0].emb + (size_t)r.pm * dim);
                        pf_issue(k, 10, m.meta[0].emb + (size_t)r.nm * dim);
                    }
                }
                cp_async_commit();
            }
        }
        if (mlin_cached) __syncthreads();
        if (tracing) tr[8] = global_ns();
        if constexpr (NET != TRS_NET_MLP)
        if (!(dbg & 1))
        for (int b0 = gid_warp0, kk = 0; b0 < Bs; b0 += ngroups, ++kk) {   // warp-uniform trip count
            const int b_raw = b0 + (gid - gid_warp0);
            const bool valid = b_raw < Bs;
            const int b = valid ? b_raw : Bs - 1;
            const int64_t smp = lo + b;
            SampleRec rec;
            if (kk < PF) {
                rec = rec_get(curw, kk);
            } else {
                rec.u = (uint32_t)ep.user[smp];
                rec.ip = (uint32_t)ep.pos[smp];
                rec.in = (uint32_t)ep.neg[smp];
                rec.pm = F ? (uint32_t)ep.pos_meta[smp * F] : 0u;
                rec.nm = F ? (uint32_t)ep.neg_meta[smp * F] : 0u;
                rec.fl = load_rec_word(ep, plan.single_user, plan.single_item, lo, Bs, b, F, 5);
            }
            SampleIds id;
            id.u = rec.u; id.ip = rec.ip; id.in = rec.in; id.pm[0] = rec.pm; id.nm[0] = rec.nm;
            const int64_t* pm = F ? ep.pos_meta + smp * F : nullptr;
            const int64_t* nm = F ? ep.neg_meta + smp * F : nullptr;
            // rows this sample alone touches in this step (flag bit 0): updated right here
            const bool fu = valid && !(dbg & 128) && (rec.fl & 1u);
            const bool fp = valid && !(dbg & 128) && (rec.fl & 0x100u);
            const bool fn = valid && !(dbg & 128) && (rec.fl & 0x10000u);
            const size_t ou = (size_t)id.u * dim, op = (size_t)id.ip * dim, on = (size_t)id.in * dim;
            // rows already sitting in shared memory (fetched during the previous step's phase B)
            const bool hu = PFETCH && kk < PF && valid && ((have >> (3 * kk + 0)) & 1u);
            const bool hp = PFETCH && kk < PF && valid && ((have >> (3 * kk + 1)) & 1u);
            const bool hn = PFETCH && kk < PF && valid && ((have >> (3 * kk + 2)) & 1u);
            // every load of the sample issued back to back (L2 only: rows are rewritten by other SMs)
            Row<V, IT> ru = hu ? pf_row(kk, 0) : load_row_cg<V, G, IT>(m.user.emb + ou, nch, gl);
            Row<V, IT> rp = hp ? pf_row(kk, 3) : load_row_cg<V, G, IT>(m.item.emb + op, nch, gl);
            Row<V, IT> rn = hn ? pf_row(kk, 6) : load_row_cg<V, G, IT>(m.item.emb + on, nch, gl);
            // scalar loads first (they are in flight while the shared-memory copies are awaited below)
            float wp = 0.f, wn = 0.f;  // FM: sum of the metadata first-order weights
            if (NET == TRS_NET_FM) {
#pragma unroll
                for (int f = 0; f < MF; ++f) {
                    if (f < F && m.meta[f].lin) {
                        wp += (f == 0 && mlin_cached) ? s_mlin[id.pm[f]] : __ldcg(m.meta[f].lin + id.pm[f]);
                        wn += (f == 0 && mlin_cached) ? s_mlin[id.nm[f]] : __ldcg(m.meta[f].lin + id.nm[f]);
                    }
                }
            }
            const float bu = m.user.lin ? __ldcg(m.user.lin + id.u) : 0.f;
            const float bip = m.item.lin ? __ldcg(m.item.lin + id.ip) : 0.f;
            const float bin = m.item.lin ? __ldcg(m.item.lin + id.in) : 0.f;
            Row<V, IT> mp[MF], mn[MF];
#pragma unroll
            for (int f = 0; f < MF; ++f) {
                if (f < F) {
                    if (PFETCH && kk < PF && valid) {
                        cp_async_wait(0);
                        mp[f] = pf_row(kk, 9);
                        mn[f] = pf_row(kk, 10);
                    } else {
                        mp[f] = load_row_cg<V, G, IT>(m.meta[f].emb + (size_t)id.pm[f] * dim, nch, gl);
                        mn[f] = load_row_cg<V, G, IT>(m.meta[f].emb + (size_t)id.nm[f] * dim, nch, gl);
                    }
                } else {
                    row_zero(mp[f]);
                    row_zero(mn[f]);
                }
            }
            // Optimizer state of the rows updated here is NOT held in registers across the scorer math: rows
            // fetched early already sit in shared memory; the others are copied there asynchronously now
            // (samples with a slot) or hinted into L2, and read right before their update.
            const bool slot = PFETCH && kk < PF;
            if (kind != TRS_OPT_SGD) {
                const bool need[3] = {fu && !hu, fp && !hp, fn && !hn};
                const size_t offs[3] = {ou, op, on};
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    if (!need[t]) continue;
                    const trs_table& tb = t ? m.item : m.user;
                    if (slot) {
                        pf_issue(kk, 3 * t + 1, tb.emb_s0 + offs[t]);
                        if (kind == TRS_OPT_SPARSE_ADAM) pf_issue(kk, 3 * t + 2, tb.emb_s1 + offs[t]);
                    } else {
                        prefetch_row<V, G, IT>(tb.emb_s0 + offs[t], nch, gl);
                        if (kind == TRS_OPT_SPARSE_ADAM) prefetch_row<V, G, IT>(tb.emb_s1 + offs[t], nch, gl);
                    }
                }
                if (slot) cp_async_commit();
            }
            // width-1 companions of the rows updated here: lane 0 takes the user's, lane 1 the positive
            // item's, lane 2 the negative item's -- one code path, state fetched now, update at the end
            const bool lf = gl == 0 ? (fu && NET == TRS_NET_FM) : (gl == 1 ? fp : (gl == 2 ? fn : false));
            const trs_table& ltab = gl == 0 ? m.user : m.item;
            const uint32_t lkey = gl == 0 ? id.u : (gl == 1 ? id.ip : id.in);
            const bool ldo = lf && ltab.lin != nullptr && !(dbg & 256);
            float lin_s0 = 0.f, lin_s1 = 0.f;
            if (ldo && kind != TRS_OPT_SGD) lin_s0 = __ldcg(ltab.lin_s0 + lkey);
            if (ldo && kind == TRS_OPT_SPARSE_ADAM) lin_s1 = __ldcg(ltab.lin_s1 + lkey);
            // optimizer state of the shared rows -> L2, for phase B's ring refills
            if (kind != TRS_OPT_SGD && valid && !(dbg & 16)) {
                if (!fu) prefetch_row<V, G, IT>(m.user.emb_s0 + ou, nch, gl);
                if (!fp) prefetch_row<V, G, IT>(m.item.emb_s0 + op, nch, gl);
                if (!fn) prefetch_row<V, G, IT>(m.item.emb_s0 + on, nch, gl);
                if (kind == TRS_OPT_SPARSE_ADAM) {
                    if (!fu) prefetch_row<V, G, IT>(m.user.emb_s1 + ou, nch, gl);
                    if (!fp) prefetch_row<V, G, IT>(m.item.emb_s1 + op, nch, gl);
                    if (!fn) prefetch_row<V, G, IT>(m.item.emb_s1 + on, nch, gl);
                }
            }
            // pooled sums over the fields beyond MF (rare): Sx = sum of rows, Qx = sum of squares
            Row<V, IT> Sp_x, Sn_x, Qp_x, Qn_x;
            row_zero(Sp_x); row_zero(Sn_x); row_zero(Qp_x); row_zero(Qn_x);
            for (int f = MF; f < F; ++f) {
                const Row<V, IT> a = load_row_cg<V, G, IT>(m.meta[f].emb + (size_t)pm[f] * dim, nch, gl);
                const Row<V, IT> c = load_row_cg<V, G, IT>(m.meta[f].emb + (size_t)nm[f] * dim, nch, gl);
#pragma unroll
                for (int i = 0; i < IT; ++i)
#pragma unroll
                    for (int k = 0; k < V; ++k) {
                        Sp_x.c[i][k] += a.c[i][k];
                        Sn_x.c[i][k] += c.c[i][k];
                        Qp_x.c[i][k] = fmaf(a.c[i][k], a.c[i][k], Qp_x.c[i][k]);
                        Qn_x.c[i][k] = fmaf(c.c[i][k], c.c[i][k], Qn_x.c[i][k]);
                    }
                if (NET == TRS_NET_FM && m.meta[f].lin) {
                    wp += __ldcg(m.meta[f].lin + pm[f]);
                    wn += __ldcg(m.meta[f].lin + nm[f]);
                }
            }

            if (tracing && kk == 0) tr[9] = global_ns() + (unsigned long long)(__float_as_uint(ru.c[0][0] + mp[0].c[0][0] + bu + bip + bin) & 1u);
            Row<V, IT> gu, gp, gn;   // gradient rows of the user / positive / negative lookups
            float gbu = 0.f, gbp, gbn;  // and of their width-1 companions
            if (NET == TRS_NET_LINEAR) {
                // v = item + sum_f meta_f (feature order), s = <u, v> + b_u + b_i
                Row<V, IT> vp = rp, vn = rn;
#pragma unroll
                for (int f = 0; f < MF; ++f) {
                    row_add(vp, mp[f]);
                    row_add(vn, mn[f]);
                }
                row_add(vp, Sp_x);
                row_add(vn, Sn_x);
                const float sp = (group_sum<G>(row_dot_partial(ru, vp)) + bu) + bip;
                const float sn = (group_sum<G>(row_dot_partial(ru, vn)) + bu) + bin;
                const float h = __fadd_rn(__fsub_rn(sn, sp), 1.0f);
                const float g = (h >= 0.f) ? invB : 0.f;
                if (valid && gl == 0) hsum += fmaxf(h, 0.f);
                gu = row_scaled_diff(g, vn, vp);
                gp = row_scaled(-g, ru);
                gn = row_scaled(g, ru);
                gbp = -g;
                gbn = g;
            } else {
                // S = sum_k e_k, Q = sum_k e_k^2 over fields user, item, meta_f
                Row<V, IT> Sp, Sn;
                float pp = 0.f, pn = 0.f;
#pragma unroll
                for (int i = 0; i < IT; ++i)
#pragma unroll
                    for (int k = 0; k < V; ++k) {
                        const float a = ru.c[i][k], x = rp.c[i][k], y = rn.c[i][k];
                        float sp_ = a + x, sn_ = a + y;
                        float qp_ = a * a + x * x, qn_ = a * a + y * y;
#pragma unroll
                        for (int f = 0; f < MF; ++f) {
                            sp_ += mp[f].c[i][k];
                            sn_ += mn[f].c[i][k];
                            qp_ = fmaf(mp[f].c[i][k], mp[f].c[i][k], qp_);
                            qn_ = fmaf(mn[f].c[i][k], mn[f].c[i][k], qn_);
                        }
                        sp_ += Sp_x.c[i][k];
                        sn_ += Sn_x.c[i][k];
                        qp_ += Qp_x.c[i][k];
                        qn_ += Qn_x.c[i][k];
                        Sp.c[i][k] = sp_;
                        Sn.c[i][k] = sn_;
                        pp += sp_ * sp_ - qp_;
                        pn += sn_ * sn_ - qn_;
                    }
                const float zp = ((bu + bip) + wp) + group_sum<G>(pp) * 0.5f;
                const float zn = ((bu + bin) + wn) + group_sum<G>(pn) * 0.5f;
                const float sp = sigmoidf_acc(zp), sn = sigmoidf_acc(zn);
                const float h = __fadd_rn(__fsub_rn(sn, sp), 1.0f);
                const float g = (h >= 0.f) ? invB : 0.f;
                const float dp = -g * sp * (1.0f - sp);
                const float dn = g * sn * (1.0f - sn);
                if (valid && gl == 0) hsum += fmaxf(h, 0.f);
#pragma unroll
                for (int i = 0; i < IT; ++i)
#pragma unroll
                    for (int k = 0; k < V; ++k)
                        // two separately rounded products, like the reference's two lookups: when
                        // pos == neg they cancel to an exact 0 (an FMA would leave a ~1e-10 residue
                        // that Adagrad/Adam's g/(|g|+eps) blows up into a step of ~lr)
                        gu.c[i][k] = __fadd_rn(__fmul_rn(dp, Sp.c[i][k] - ru.c[i][k]),
                                               __fmul_rn(dn, Sn.c[i][k] - ru.c[i][k]));
                gp = row_scaled_diff(dp, Sp, rp);
                gn = row_scaled_diff(dn, Sn, rn);
                gbu = dp + dn;
                gbp = dp;
                gbn = dn;
                if (valid) {  // metadata rows are always reduced in phase B
#pragma unroll
                    for (int f = 0; f < MF; ++f) {
                        if (f < F) {
                            store_row<V, G, IT>(st.gM[f] + (size_t)b * dim, nch, gl, row_scaled_diff(dp, Sp, mp[f]));
                            store_row<V, G, IT>(st.gM[f] + (size_t)(Bs + b) * dim, nch, gl, row_scaled_diff(dn, Sn, mn[f]));
                        }
                    }
                    for (int f = MF; f < F; ++f) {
                        Row<V, IT> r = load_row_cg<V, G, IT>(m.meta[f].emb + (size_t)pm[f] * dim, nch, gl);
                        store_row<V, G, IT>(st.gM[f] + (size_t)b * dim, nch, gl, row_scaled_diff(dp, Sp, r));
                        r = load_row_cg<V, G, IT>(m.meta[f].emb + (size_t)nm[f] * dim, nch, gl);
                        store_row<V, G, IT>(st.gM[f] + (size_t)(Bs + b) * dim, nch, gl, row_scaled_diff(dn, Sn, r));
                    }
                }
            }
            if (tracing && kk == 0) tr[10] = global_ns() + (unsigned long long)(__float_as_uint(gu.c[0][0] + gp.c[0][0]) & 1u);
            if (valid) {
                if (slot) cp_async_wait(0);  // my state-row copies of this sample
                auto fused = [&](const trs_table& tb, size_t off, int t, Row<V, IT>& p, const Row<V, IT>& g) {
                    Row<V, IT> s0, s1;
                    row_zero(s0);
                    row_zero(s1);
                    if (kind != TRS_OPT_SGD)
                        s0 = slot ? pf_row(kk, 3 * t + 1) : load_row_cg<V, G, IT>(tb.emb_s0 + off, nch, gl);
                    if (kind == TRS_OPT_SPARSE_ADAM)
                        s1 = slot ? pf_row(kk, 3 * t + 2) : load_row_cg<V, G, IT>(tb.emb_s1 + off, nch, gl);
                    update_store_row<V, G, IT>(tb, off, nch, gl, opt, scale, p, s0, s1, g);
                };
                // user row
                if (fu) {
                    fused(m.user, ou, 0, ru, gu);
                } else {
                    store_row<V, G, IT>(st.gU + (size_t)b * dim, nch, gl, gu);
                    if (NET == TRS_NET_FM && gl == 0) st.gbU[b] = gbu;
                }
                // Linear pools the metadata rows into the item row: their gradient IS the item row's, so
                // it stays staged for the metadata reduce even when the item row itself is updated here
                const bool stage_items = (NET == TRS_NET_LINEAR && F > 0);
                // FM: d linear_metadata = delta, the same scalar as d linear_item -> always staged
                const bool meta_lin = (NET == TRS_NET_FM && F > 0);
                if (fp) fused(m.item, op, 1, rp, gp);
                if (!fp || stage_items) store_row<V, G, IT>(st.gI + (size_t)b * dim, nch, gl, gp);
                if ((!fp || meta_lin) && gl == 0) st.gbI[b] = gbp;
                if (fn) fused(m.item, on, 2, rn, gn);
                if (!fn || stage_items) store_row<V, G, IT>(st.gI + (size_t)(Bs + b) * dim, nch, gl, gn);
                if ((!fn || meta_lin) && gl == 0) st.gbI[Bs + b] = gbn;
                if (tracing && kk == 0) tr[11] = global_ns();
                if (ldo) {  // lanes 0..2: the width-1 companions, state already in registers
                    const float pl = gl == 0 ? bu : (gl == 1 ? bip : bin);
                    const float gg = gl == 0 ? gbu : (gl == 1 ? gbp : gbn);
                    update_store_lin(ltab, lkey, opt, scale, gg, pl, lin_s0, lin_s1);
                }
            }
        }
        // The next step's rows.  My first PF samples: parameter rows (+ optimizer state where the row will be
        // updated in phase A) are copied into shared memory NOW, asynchronously -- before the step's first
        // barrier, so the copies fly during both barriers and phase B -- unless this step looks the row up
        // itself (flag bit 1: some CTA updates it in this step; it is read after the step's last barrier
        // instead).  My own phase A is over: its shared-memory slots are free.
        have = 0;
        if (PFETCH && si + 1 < n_steps && !(dbg & 16)) {
#pragma unroll
            for (int k = 0; k < PF; ++k) {
                const SampleRec nr = rec_get(nxtw, k);   // warp-wide shuffles: before any divergence
                const int b = gid + k * ngroups;
                if (b >= Bs2) continue;
                const uint32_t rows[3] = {nr.u, nr.ip, nr.in};
                const unsigned tf[3] = {nr.fl & 0xffu, (nr.fl >> 8) & 0xffu, (nr.fl >> 16) & 0xffu};

#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    if (tf[t] & 2u) continue;  // updated below by some CTA: not safe to copy yet
                    const trs_table& tb = t ? m.item : m.user;
                    const size_t ro = (size_t)rows[t] * dim;
                    pf_issue(k, 3 * t, tb.emb + ro);
                    if ((tf[t] & 1u) && kind != TRS_OPT_SGD) pf_issue(k, 3 * t + 1, tb.emb_s0 + ro);
                    if ((tf[t] & 1u) && kind == TRS_OPT_SPARSE_ADAM) pf_issue(k, 3 * t + 2, tb.emb_s1 + ro);
                    have |= 1u << (3 * k + t);
                }
                // width-1 companions (+ their optimizer state where updated in phase A) -> L2: lane t takes table t
                const unsigned tfl = gl == 0 ? tf[0] : (gl == 1 ? tf[1] : tf[2]);
                if (gl < 3 && !(tfl & 2u)) {
                    const trs_table& tb = gl ? m.item : m.user;
                    const uint32_t row = gl == 0 ? nr.u : (gl == 1 ? nr.ip : nr.in);
                    if (tb.lin) {
                        prefetch_l2(tb.lin + row);
                        if ((tfl & 1u) && kind != TRS_OPT_SGD && tb.lin_s0) prefetch_l2(tb.lin_s0 + row);
                        if ((tfl & 1u) && kind == TRS_OPT_SPARSE_ADAM && tb.lin_s1) prefetch_l2(tb.lin_s1 + row);
                    }
                }
            }
            cp_async_commit();
        }
        // samples beyond the shared-memory budget (large batches): L2 prefetch hints
        if (si + 1 < n_steps && !(dbg & 16) && NET != TRS_NET_MLP) {
            for (int b = gid + (PFETCH ? PF : 0) * ngroups; b < Bs2; b += ngroups) {
                const uint32_t u = (uint32_t)ep.user[lo2 + b], ip = (uint32_t)ep.pos[lo2 + b],
                               in = (uint32_t)ep.neg[lo2 + b];
                prefetch_row<V, G, IT>(m.user.emb + (size_t)u * dim, nch, gl);
                prefetch_row<V, G, IT>(m.item.emb + (size_t)ip * dim, nch, gl);
                prefetch_row<V, G, IT>(m.item.emb + (size_t)in * dim, nch, gl);
                if (kind != TRS_OPT_SGD) {
                    prefetch_row<V, G, IT>(m.user.emb_s0 + (size_t)u * dim, nch, gl);
                    prefetch_row<V, G, IT>(m.item.emb_s0 + (size_t)ip * dim, nch, gl);
                    prefetch_row<V, G, IT>(m.item.emb_s0 + (size_t)in * dim, nch, gl);
                }
                if (kind == TRS_OPT_SPARSE_ADAM) {
                    prefetch_row<V, G, IT>(m.user.emb_s1 + (size_t)u * dim, nch, gl);
                    prefetch_row<V, G, IT>(m.item.emb_s1 + (size_t)ip * dim, nch, gl);
                    prefetch_row<V, G, IT>(m.item.emb_s1 + (size_t)in * dim, nch, gl);
                }
            }
        }
        // the step's first ring items: their descriptors landed long ago; fetch param + state rows
        // now (nothing in phase A writes them: they are not single-lookup rows), so only the staged
        // gradients wait for the barrier
        if (tracing) tr[12] = global_ns();
        if (RINGED) {
            cp_async_wait(0);
            if (!(dbg & 4)) {
                for (int n = 0; n < RING; ++n) issue_state(n_items, n, lo);
            }
            cp_async_commit();
        }
        // my CTA's first long segment: its descriptor and this group's first lookup ids are plan data --
        // fetched before the barrier so that only the staged rows wait for it
        constexpr int U = 6;  // staged rows in flight per group (one batch covers 6 * groups-per-CTA lookups)
        uint4 seg_pre = make_uint4(0, 0, 0, 0);
        uint32_t j_pre[U] = {0, 0, 0, 0, 0, 0};
        if ((int)blockIdx.x < n_long && !(dbg & 2)) {
            seg_pre = plan.long_segs[(size_t)s * plan.long_cap + blockIdx.x];
            const SpaceRef sp = resolve_space<NET>((int)seg_pre.x, m, plan, st, lo);
#pragma unroll
            for (int z = 0; z < U; ++z)
                if (g_in_cta + z * GPB < (int)seg_pre.z) j_pre[z] = sp.P[seg_pre.y + g_in_cta + z * GPB];
        }

        if (tracing) tr[13] = global_ns() + (j_pre[0] & 1u);
        if (NET != TRS_NET_MLP) {
            hsum = warp_sum(hsum);
            if ((threadIdx.x & 31) == 0) s_loss[threadIdx.x >> 5] = hsum;
            __syncthreads();
            if (threadIdx.x == 0) {
                float H = 0.f;
#pragma unroll
                for (int w = 0; w < NT / 32; ++w) H += s_loss[w];
                st.loss_part[(size_t)si * gridDim.x + blockIdx.x] = H;
            }
        }
        if (tracing) tr[1] = global_ns();
        if (!(dbg & 8)) grid_barrier(st.barrier, bar_target);
        if (tracing) tr[2] = global_ns();

        // ------------------------------ phase B ------------------------------------------
        if (RINGED) {
            if (!(dbg & 4)) {
                for (int n = 0; n < RING; ++n) issue_grad(n_items, n, lo);
            }
            cp_async_commit();
        }
        if (tracing) tr[4] = global_ns();
        // width-1 companions (biases / first-order weights) of the short segments: one THREAD per segment;
        // the loads are issued here and consumed after the long segments below
        float lin_p = 0.f, lin_0 = 0.f, lin_1 = 0.f, lin_g = 0.f;
        bool lin_live = false;
        SpaceRef lin_sp = {};
        if (!(dbg & 32) && lin_i < n_items) {
            lin_sp = resolve_space<NET>((int)(lin_it.x & 0xffu), m, plan, st, lo);
            lin_live = lin_sp.stage_lin != nullptr;
            if (lin_live) {
                const trs_table& t = *lin_sp.t;
                lin_p = __ldcg(t.lin + lin_it.z);
                if (kind != TRS_OPT_SGD) lin_0 = __ldcg(t.lin_s0 + lin_it.z);
                if (kind == TRS_OPT_SPARSE_ADAM) lin_1 = __ldcg(t.lin_s1 + lin_it.z);
                lin_g = __ldcg(lin_sp.stage_lin + lin_it.w);
            }
        }
        if (tracing) tr[5] = global_ns();
        // long segments: one CTA per segment, every row group sums a strided subset of its lookups
        if (!(dbg & 2)) {
            for (int sg = blockIdx.x; sg < n_long; sg += gridDim.x) {   // block-uniform trip count
                const bool first = sg == (int)blockIdx.x;
                const uint4 seg = first ? seg_pre : plan.long_segs[(size_t)s * plan.long_cap + sg];  // space, start, length, row
                const SpaceRef sp = resolve_space<NET>((int)seg.x, m, plan, st, lo);
                const uint32_t* P = sp.P + seg.y;
                const int c = (int)seg.z;
                const uint32_t key = seg.w;
                const size_t roff = (size_t)key * dim;
                // the updating group fetches the row's parameter + state while the sums are formed
                Row<V, IT> p, s0, s1;
                row_zero(p); row_zero(s0); row_zero(s1);
                if (g_in_cta == 0) {
                    p = load_row_cg<V, G, IT>(sp.t->emb + roff, nch, gl);
                    if (kind != TRS_OPT_SGD) s0 = load_row_cg<V, G, IT>(sp.t->emb_s0 + roff, nch, gl);
                    if (kind == TRS_OPT_SPARSE_ADAM) s1 = load_row_cg<V, G, IT>(sp.t->emb_s1 + roff, nch, gl);
                }
                Row<V, IT> acc;
                row_zero(acc);
                float accl = 0.f;
                for (int q0 = g_in_cta; q0 < c; q0 += U * GPB) {
                    uint32_t j[U];
#pragma unroll
                    for (int z = 0; z < U; ++z)
                        j[z] = (first && q0 == g_in_cta) ? j_pre[z] : ((q0 + z * GPB < c) ? P[q0 + z * GPB] : 0u);
                    Row<V, IT> r[U];
                    float l[U];
#pragma unroll
                    for (int z = 0; z < U; ++z) {
                        if (q0 + z * GPB < c) {
                            r[z] = load_row_cg<V, G, IT>(sp.stage + (size_t)j[z] * dim, nch, gl);
                            l[z] = (sp.stage_lin && gl == 0) ? __ldcg(sp.stage_lin + j[z]) : 0.f;
                        }
                    }
#pragma unroll
                    for (int z = 0; z < U; ++z) {
                        if (q0 + z * GPB < c) {
                            row_acc(acc, r[z]);
                            accl = __fadd_rn(accl, l[z]);
                        }
                    }
                }
                // partial sums -> shared memory, [group][chunk of the row][lane][V]
#pragma unroll
                for (int a = 0; a < IT; ++a)
#pragma unroll
                    for (int k = 0; k < V; ++k) s_part[((g_in_cta * IT + a) * G + gl) * V + k] = acc.c[a][k];
                if (gl == 0) s_part_lin[g_in_cta] = accl;
                __syncthreads();
                if (g_in_cta == 0) {
                    Row<V, IT> g;
                    row_zero(g);
                    float g_lin = 0.f;
                    const int ng = min(GPB, c);  // groups that summed at least one row, in group order
                    for (int q = 0; q < ng; ++q) {
#pragma unroll
                        for (int a = 0; a < IT; ++a)
#pragma unroll
                            for (int k = 0; k < V; ++k)
                                g.c[a][k] = __fadd_rn(g.c[a][k], s_part[((q * IT + a) * G + gl) * V + k]);
                        g_lin = __fadd_rn(g_lin, s_part_lin[q]);
                    }
                    update_store_row<V, G, IT>(*sp.t, roff, nch, gl, opt, scale, p, s0, s1, g);
                    if (sp.stage_lin && gl == 0) update_lin(*sp.t, key, opt, scale, g_lin);
                }
                __syncthreads();
            }
        }
        // finish the width-1 companion items
        if (lin_live) {
            const int c = (int)((lin_it.x >> 8) & 0xffu);
            for (int q = 1; q < c; ++q) lin_g = __fadd_rn(lin_g, __ldcg(lin_sp.stage_lin + lin_sp.P[lin_it.y + q]));
            update_store_lin(*lin_sp.t, lin_it.z, opt, scale, lin_g, lin_p, lin_0, lin_1);
        }
        if (!(dbg & 32)) {  // more short segments than threads: the rest, one at a time
            for (int i = lin_i + NT * (int)gridDim.x; i < n_items; i += NT * (int)gridDim.x) {
                const uint4 it = items[i];
                const SpaceRef sp = resolve_space<NET>((int)(it.x & 0xffu), m, plan, st, lo);
                if (!sp.stage_lin) continue;
                float g_lin = __ldcg(sp.stage_lin + it.w);
                const int c = (int)((it.x >> 8) & 0xffu);
                for (int q = 1; q < c; ++q) g_lin = __fadd_rn(g_lin, __ldcg(sp.stage_lin + sp.P[it.y + q]));
                update_lin(*sp.t, it.z, opt, scale, g_lin);
            }
        }
        if (tracing) tr[6] = global_ns();
        // short segments through the ring
        if (!(dbg & 4)) {
            if (RINGED) cp_async_wait(0);
            const int my_items = n_items > gid ? (n_items - gid + ngroups - 1) / ngroups : 0;
            for (int n = 0; n < my_items; ++n) {
                if (RINGED && n >= RING) cp_async_wait(RING - 1);
                consume(items, n_items, n, lo, scale);
                if (RINGED) {
                    issue_state(n_items, n + RING, lo);
                    issue_grad(n_items, n + RING, lo);
                    issue_desc(items, n_items, n + 2 * RING);
                    cp_async_commit();
                }
            }
            if (RINGED) cp_async_wait(0);
        }
        if (tracing) tr[7] = global_ns();
        // descriptors of the next step's first work items
        if (RINGED) {
            if (si + 1 < n_steps) {
                const uint4* items2 = plan.items + (size_t)(s + 1) * plan.item_cap;
                for (int n = 0; n < 2 * RING; ++n) issue_desc(items2, n_items_next, n);
            }
            cp_async_commit();
        }
        n_items_cur = n_items_next;
        n_long_cur = n_long_next;
#pragma unroll
        for (int i = 0; i < WPL; ++i) curw[i] = nxtw[i];
        if (tracing) tr[3] = global_ns();
        if (!(dbg & 8)) grid_barrier(st.barrier, bar_target);
    }
    cp_async_wait(0);

    // batch-mean hinge per step, summed over CTAs in a fixed order (deterministic)
    if (NET != TRS_NET_MLP && blockIdx.x == 0) {
        for (int si = threadIdx.x; si < n_steps; si += NT) {
            const int64_t lo = (first_step + (int64_t)si) * ep.batch;
            const int Bs = (int)min((int64_t)ep.batch, ep.n_samples - lo);
            float H = 0.f;
            for (unsigned c = 0; c < gridDim.x; ++c) H += __ldcg(st.loss_part + (size_t)si * gridDim.x + c);
            loss_out[si] = H / (float)Bs;
        }
    }
}

template <int V, int G, int IT>
static void launch_train(const trs_model* m, const trs_epoch* ep, const OptScalars* opt,
                         const PlanPtrs* plan, const Stage* st, int first_step, int n_steps,
                         float* loss, int grid, cudaStream_t stream, cudaError_t* err) {
    // Timing experiments only (results are wrong), compiled in with -DTRS_DEBUG and then read from the environment:
    // TRS_DEBUG_SKIP bits 1 phase A, 2 long segments, 4 ring, 8 grid barriers, 16 L2 prefetches, 32 width-1
    // companions, 64 phase trace, 128 no phase-A updates.  A production build ignores the variable.
    int dbg = 0;
#ifdef TRS_DEBUG
    const char* dbg_env = getenv("TRS_DEBUG_SKIP");
    dbg = dbg_env ? atoi(dbg_env) : 0;
#endif
    void* args[] = {(void*)m, (void*)ep, (void*)opt, (void*)plan, (void*)st,
                    (void*)&first_step, (void*)&n_steps, (void*)&loss, (void*)&dbg};
    const void* fn = m->net == TRS_NET_LINEAR ? (const void*)train_kernel<TRS_NET_LINEAR, V, G, IT>
                     : m->net == TRS_NET_FM   ? (const void*)train_kernel<TRS_NET_FM, V, G, IT>
                                              : (const void*)train_kernel<TRS_NET_MLP, V, G, IT>;
    const size_t smem = train_smem_bytes<V, IT>();
    if (smem > 48 * 1024) {
        *err = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (*err != cudaSuccess) return;
    }
    *err = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(train_threads<V, IT>()), args, smem, stream);
}

// one CTA per SM: the ring takes most of the SM's shared memory
static int train_grid_for(const trs_model*, const RowShape&) { return device_props().sm_count; }

}  // namespace trs

using namespace trs;

extern "C" int trs_device_info(int* sm_count_host, int* train_grid_host, int* train_block_host) {
    if (sm_count_host) *sm_count_host = device_props().sm_count;
    if (train_block_host) *train_block_host = train_threads<4, 1>();
    if (train_grid_host) *train_grid_host = device_props().sm_count;
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

// debug hook (not part of trs.h): byte offset of the phase trace inside the train workspace
extern "C" size_t trs_debug_trace_offset(const trs_model* model, const trs_epoch* epoch) {
    RowShape shape;
    if (!model || !epoch || epoch->batch <= 0 || check_model(model, &shape)) return 0;
    return stage_layout(model, epoch, train_grid_for(model, shape)).trace;
}

extern "C" size_t trs_train_workspace_bytes(const trs_model* model, const trs_epoch* epoch) {
    RowShape shape;
    if (!model || !epoch || epoch->batch <= 0 || check_model(model, &shape)) return 0;
    return stage_layout(model, epoch, train_grid_for(model, shape)).total;
}

namespace trs {
StagePtrs stage_pointers(const trs_model* model, const trs_epoch* ep, void* workspace) {
    RowShape shape;
    StagePtrs r = {};
    if (!pick_row_shape(model->dim, &shape)) return r;
    const StageLayout SL = stage_layout(model, ep, train_grid_for(model, shape));
    char* W = (char*)workspace;
    r.gU = (float*)(W + SL.gU);
    r.gI = (float*)(W + SL.gI);
    for (int f = 0; f < model->n_meta; ++f) r.gM[f] = (float*)(W + SL.gM[f]);
    return r;
}
}  // namespace trs

extern "C" int trs_train_steps(const trs_model* model, const trs_epoch* ep, const trs_optim* optim,
                               const void* plan, void* workspace, size_t workspace_bytes,
                               int first_step, int n_steps, float* loss, trs_stream_t stream) {
    TRS_REQUIRE(model && model->net != TRS_NET_MLP, "trs_train_steps: use trs_mlp_train_steps for net_type mlp");
    return trs::run_train_steps(model, ep, optim, plan, workspace, workspace_bytes, first_step, n_steps, loss,
                                (cudaStream_t)stream);
}

int trs::run_train_steps(const trs_model* model, const trs_epoch* ep, const trs_optim* optim,
                         const void* plan, void* workspace, size_t workspace_bytes,
                         int first_step, int n_steps, float* loss, cudaStream_t stream) {
    RowShape shape;
    int rc = check_model(model, &shape);
    if (rc) return rc;
    TRS_REQUIRE(ep && ep->user && ep->pos && ep->neg, "epoch ids are NULL");
    TRS_REQUIRE(ep->batch > 0, "batch must be positive");
    TRS_REQUIRE(model->n_meta == 0 || (ep->pos_meta && ep->neg_meta), "metadata ids are NULL");
    TRS_REQUIRE(optim && optim->step_scale, "optimizer / step_scale is NULL");
    TRS_REQUIRE(optim->kind >= TRS_OPT_SGD && optim->kind <= TRS_OPT_SPARSE_ADAM, "unknown optimizer kind %d", optim->kind);
    TRS_REQUIRE(plan && workspace && (loss || model->net == TRS_NET_MLP), "plan / workspace / loss is NULL");
    const int64_t steps = n_steps_of(ep);
    TRS_REQUIRE(first_step >= 0 && n_steps >= 0 && first_step + (int64_t)n_steps <= steps,
                "steps [%d, %d) outside the epoch's %lld steps", first_step, first_step + n_steps, (long long)steps);
    if (n_steps == 0) return TRS_OK;

    auto need_state = [&](const trs_table& t, const char* name) -> int {
        const bool lin_learns = t.lin && !(model->net == TRS_NET_LINEAR && &t == &model->user);
        if (optim->kind != TRS_OPT_SGD) {
            TRS_REQUIRE(t.emb_s0 && (!lin_learns || t.lin_s0), "%s: optimizer state s0 is NULL", name);
        }
        if (optim->kind == TRS_OPT_SPARSE_ADAM) {
            TRS_REQUIRE(t.emb_s1 && (!lin_learns || t.lin_s1), "%s: optimizer state s1 is NULL", name);
        }
        return TRS_OK;
    };
    if ((rc = need_state(model->user, "user"))) return rc;
    if ((rc = need_state(model->item, "item"))) return rc;
    for (int f = 0; f < model->n_meta; ++f)
        if ((rc = need_state(model->meta[f], "metadata"))) return rc;

    const int grid = train_grid_for(model, shape);
    TRS_REQUIRE(grid > 0, "no launch configuration for n_factors %d", model->dim);
    const StageLayout SL = stage_layout(model, ep, grid);
    if (workspace_bytes < SL.total) {
        set_error("train workspace too small: %zu < %zu", workspace_bytes, SL.total);
        return TRS_ERR_WORKSPACE;
    }
    const PlanLayout PL = plan_layout(ep->n_samples, ep->batch, model->n_meta);
    char* W = (char*)workspace;
    Stage st = {};
    st.gU = (float*)(W + SL.gU);
    st.gI = (float*)(W + SL.gI);
    for (int f = 0; f < model->n_meta; ++f) st.gM[f] = (float*)(W + SL.gM[f]);
    st.gbU = (float*)(W + SL.gbU);
    st.gbI = (float*)(W + SL.gbI);
    st.loss_part = (float*)(W + SL.loss_part);
    st.barrier = (unsigned*)(W + SL.sync_words);
    st.trace = (unsigned long long*)(W + SL.trace);
    TRS_CUDA(cudaMemsetAsync(W + SL.sync_words, 0, SL.sync_bytes, stream));

    const char* P = (const char*)plan;
    PlanPtrs pp = {};
    pp.user_key = (const uint32_t*)(P + PL.user_key);
    pp.user_perm = (const uint32_t*)(P + PL.user_perm);
    pp.item_key = (const uint32_t*)(P + PL.item_key);
    pp.item_perm = (const uint32_t*)(P + PL.item_perm);
    for (int f = 0; f < model->n_meta; ++f) {
        pp.meta_key[f] = (const uint32_t*)(P + PL.meta_key[f]);
        pp.meta_perm[f] = (const uint32_t*)(P + PL.meta_perm[f]);
    }
    pp.item_cnt = (const uint32_t*)(P + PL.item_cnt);
    pp.long_cnt = (const uint32_t*)(P + PL.long_cnt);
    pp.single_user = (const uint8_t*)(P + PL.single_user);
    pp.single_item = (const uint8_t*)(P + PL.single_item);
    pp.items = (const uint4*)(P + PL.items);
    pp.long_segs = (const uint4*)(P + PL.long_segs);
    pp.item_cap = PL.item_cap;
    pp.long_cap = PL.long_cap;

    const OptScalars os = make_opt_scalars(optim);
    cudaError_t err = cudaSuccess;
    TRS_DISPATCH_ROW_SHAPE(shape, launch_train, model, ep, &os, &pp, &st, first_step, n_steps, loss,
                           grid, stream, &err);
    TRS_CUDA(err);
    return TRS_OK;
}
