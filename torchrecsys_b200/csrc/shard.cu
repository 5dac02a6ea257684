// shard.cu -- row-sharded training of the Linear scorer over PEER-MAPPED table shards (SURVEY.md §8e, BASELINE
// configs[3]: 50M users x 5M items, dim 128, 1/2/4/8 GPUs).  Reference semantics: model.py:274-284 on ONE global
// batch per step (forward x2, hinge_loss, backward, optimizer.step()); the reference itself is single-device.
//
// Row r of a table lives on rank r % W at local row r / W.  Every rank maps every peer's shard, gradient staging
// buffer and barrier words (CUDA IPC) and runs ONE persistent cooperative kernel for K steps -- the exchange step
// of the sharded path is the kernel's own loads and stores over NVLink, there is no collective call per step:
//
//   phase A  the samples PLACED on this rank (those whose user row it owns: user rows never cross NVLink; the
//            step's global batch is the same set of samples whichever rank runs which).  A row group (dim/4
//            lanes) per sample.  The two item rows of a group's first 7 samples sit in a per-group region of shared
//            memory that bulk async copies (cp.async.bulk + one mbarrier per group) fill A STEP AHEAD, straight from
//            the owner's HBM -- local or peer -- while the owners update; rows the previous step updates (plan
//            flag) are fetched after the barrier instead.  User rows (+ optimizer state) come by cp.async into
//            thread-private slots, four samples at a time.  Both scores, the hinge with g = [h >= 0] / B_global; a
//            user row looked up once in the step is updated in place, every other gradient row goes straight into
//            its OWNER's staging buffer at slot = the lookup's position in the global batch (remote store, L2
//            policy evict_last: the owner reads it once, with evict_first).
//            With W > 1 phase A runs in two passes: the samples none of whose rows the previous step updates run
//            BEFORE the rank waits for the barrier that ends that step (the staging buffers exist twice, for even
//            and odd steps), the flagged ones after it.
//   cross-rank barrier: a monotonic arrival counter per rank -- one release fence (system scope after stores into
//            peer memory), a relaxed add to every rank's counter, relaxed polling of the own counter, one acquire
//            load.  The barrier after phase B is split into arrive (there) and wait (inside the next phase A).
//   phase B  every owner walks the (local row, slot) pairs of the lookups it owns and phase A did not finish --
//            stably sorted by row: the plan, built once per epoch -- sums the staged rows of a row in slot order
//            (what coalesce() gives, deterministic, independent of W), applies SGD / Adagrad / SparseAdam to
//            parameter + state rows of ITS shard.
//   cross-rank barrier (updates visible before the next step's reads).
//
// HBM per step and rank: each owned touched row's parameter + state read once and written once, the staged
// gradient rows written (by NVLink or locally) and read once, ids.  NVLink per step and rank: 2 item rows in and
// 2 gradient rows out per sample whose item lives elsewhere ((W-1)/W of them).
//
// One GPU can host all W ranks of a group in ONE cooperative launch (n_local = W, the SMs split between the
// ranks): that is how the parity tests run on a single-GPU box -- kernels that wait on each other must never be
// separate launches on one device.
//
// Two kernels run this step, built from the same step pieces (StepThread): shard_train_kernel, the two-phase kernel
// above, at any group size and row shape; and shard_train_one_pass_kernel, for one rank in one launch with one chunk
// per lane (the default benchmark), whose phase A also updates the item rows a step looks up once and leaves phase B
// only the rows with several lookups.  Both give the same results bit for bit.
#include <cuda.h>
#include <string.h>

#include "plan.cuh"
#include "ptx.cuh"
#include "scorer.cuh"
#include "train.cuh"

namespace trs {

// ------------------------------------------------------------------------------------------------------------
// plan: sample placement + the owner's sorted (local row, slot) pairs
// ------------------------------------------------------------------------------------------------------------
struct ShardPlanLayout {
    size_t samp_cnt;  // [steps]      samples placed on this rank
    size_t own_cnt;   // [steps][2]   lookups this rank owns: user space, item space
    size_t samp;      // [n]          step s at s*B: position b of each placed sample in the step, ascending
    size_t ukey, uval;  // [n]        sorted (local row, slot) pairs of the owned user lookups; step s at s*B
    size_t ikey, ival;  // [2n]       ... item lookups (slot b: positive of sample b, B_s + b: its negative); 2*s*B
    // one rank only (item_single_*_kernel), for the one-pass kernel:
    size_t cntB;        // [steps][2] own_cnt with the item count of ikeyB / ivalB
    size_t iflag;       // [2n] bytes 1: the item row of lookup slot j is looked up once in the step; 2*s*B
    size_t ikeyB, ivalB;  // [2n]     the pairs of ikey / ival whose row the step looks up more than once; 2*s*B
    size_t total;
};
static ShardPlanLayout shard_plan_layout(int64_t n, int B) {
    ShardPlanLayout L;
    size_t off = 0;
    auto take = [&](size_t n_elems) {
        size_t o = off;
        off += (n_elems * sizeof(uint32_t) + 255) / 256 * 256;
        return o;
    };
    const int64_t steps = (n + B - 1) / B;
    L.samp_cnt = take((size_t)steps);
    L.own_cnt = take((size_t)2 * steps);
    L.samp = take((size_t)n);
    L.ukey = take((size_t)n);
    L.uval = take((size_t)n);
    L.ikey = take((size_t)2 * n);
    L.ival = take((size_t)2 * n);
    L.cntB = take((size_t)2 * steps);
    L.iflag = take(((size_t)2 * n + 3) / 4);
    L.ikeyB = take((size_t)2 * n);
    L.ivalB = take((size_t)2 * n);
    L.total = off;
    return L;
}

constexpr int RT_THREADS = 256;
constexpr int RT_ROWS = 8;
constexpr int RT_TILE = RT_THREADS * RT_ROWS;

__device__ __forceinline__ uint32_t route_id(const int64_t* a, const int64_t* b, int64_t s0, int Bs, int j) {
    return (uint32_t)((j < Bs) ? a[s0 + j] : b[s0 + j - Bs]);
}

// ---- stable per-step compaction --------------------------------------------------------------------------------
// The candidates [0, len) of a step are compacted in two launches over (tiles of RT_TILE, steps): compact_count_kernel
// counts per tile the ones a selector S keeps, compact_scatter_kernel hands each kept one its place -- the kept ones of
// the tiles before its own, then of the threads before it -- to S.emit.  S: len(step); count(step, j, len) (keep, plus
// any side output of the count launch); keep(step, j, len, v) (v: a value carried to emit); emit(step, p, j, v);
// total(step, t) (tile 0: the step's count).

// position of this thread's set flag among the flags of the NT threads of the block before it, and their total; s_w
// holds one word per warp and may be reused once the block has synchronised again
template <int NT>
__device__ __forceinline__ uint32_t block_rank(bool f, uint32_t* s_w, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t m = __ballot_sync(0xffffffffu, f);
    if (lane == 0) s_w[warp] = __popc(m);
    __syncthreads();
    uint32_t wbase = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) {
        const uint32_t c = s_w[w];
        if (w < warp) wbase += c;
        tot += c;
    }
    total = tot;
    return wbase + __popc(m & ((1u << lane) - 1u));
}

template <class S>
__global__ void __launch_bounds__(RT_THREADS)
compact_count_kernel(const S sel, uint32_t* __restrict__ tile_cnt, int tiles) {
    __shared__ uint32_t s_w[RT_THREADS / 32];
    const int64_t step = blockIdx.y;
    const int tile = blockIdx.x;
    const int len = sel.len(step);
    uint32_t cnt = 0;
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int j = tile * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (j < len) cnt += sel.count(step, j, len) ? 1u : 0u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < RT_THREADS / 32; ++w) t += s_w[w];
        tile_cnt[step * tiles + tile] = t;
    }
}

template <class S>
__global__ void __launch_bounds__(RT_THREADS)
compact_scatter_kernel(const S sel, const uint32_t* __restrict__ tile_cnt, int tiles) {
    __shared__ uint32_t s_w[RT_THREADS / 32], s_b[RT_THREADS / 32], s_t[RT_THREADS / 32];
    __shared__ uint32_t s_base;
    const int64_t step = blockIdx.y;
    const int tile = blockIdx.x;
    const int len = sel.len(step);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    {   // kept ones of the tiles before mine (tile 0 also publishes the step's total)
        uint32_t before = 0, total = 0;
        for (int t = threadIdx.x; t < tiles; t += RT_THREADS) {
            const uint32_t c = tile_cnt[step * tiles + t];
            total += c;
            if (t < tile) before += c;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            before += __shfl_xor_sync(0xffffffffu, before, o);
            total += __shfl_xor_sync(0xffffffffu, total, o);
        }
        if (lane == 0) { s_b[warp] = before; s_t[warp] = total; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t bb = 0, tt = 0;
            for (int w = 0; w < RT_THREADS / 32; ++w) { bb += s_b[w]; tt += s_t[w]; }
            s_base = bb;
            if (tile == 0) sel.total(step, tt);
        }
        __syncthreads();
    }
    uint32_t run = s_base;
    for (int r = 0; r < RT_ROWS; ++r) {
        const int j = tile * RT_TILE + r * RT_THREADS + threadIdx.x;
        uint32_t v = 0;
        const bool m = j < len && sel.keep(step, j, len, v);
        uint32_t tot;
        const uint32_t p = run + block_rank<RT_THREADS>(m, s_w, tot);
        if (m) sel.emit(step, p, j, v);
        run += tot;
        __syncthreads();
    }
}

// Route step: the lookups of a step (a[s0 + j], then b[s0 + j - Bs] when mult = 2) that this rank owns, as (local row,
// slot) pairs in slot order.  User space (samp != NULL): the rank's samples ARE its owned user lookups in slot order,
// so the pair's value is the sample's index in the rank's list (its slot is samp[index]); item space: the value is the
// slot itself
struct RouteSel {
    const int64_t *a, *b;
    int mult;
    int64_t n_samples;
    int B;
    uint32_t world, rank;
    uint32_t *out_key, *out_val, *samp, *own_cnt, *samp_cnt;
    __device__ __forceinline__ int Bs(int64_t step) const { return (int)min((int64_t)B, n_samples - step * B); }
    __device__ __forceinline__ int len(int64_t step) const { return mult * Bs(step); }
    __device__ __forceinline__ bool keep(int64_t step, int j, int, uint32_t& id) const {
        id = route_id(a, b, step * (int64_t)B, Bs(step), j);
        return id % world == rank;
    }
    __device__ __forceinline__ bool count(int64_t step, int j, int len) const {
        uint32_t id;
        return keep(step, j, len, id);
    }
    __device__ __forceinline__ void emit(int64_t step, uint32_t p, int j, uint32_t id) const {
        const int64_t seg = (int64_t)mult * step * B;
        out_key[seg + p] = id / world;
        out_val[seg + p] = samp ? p : (uint32_t)j;
        if (samp) samp[step * (int64_t)B + p] = (uint32_t)j;
    }
    __device__ __forceinline__ void total(int64_t step, uint32_t t) const {
        own_cnt[step * 2] = t;
        if (samp_cnt) samp_cnt[step] = t;
    }
};


// ---- which of a rank's samples read an item row that the PREVIOUS step updates ("dirty") ----------------------
// The kernel fetches the item rows of step s+1 while step s's owners are still updating (phase B): legal for every
// row step s does not touch.  Per step a hashed bitmap of the item rows looked up anywhere in the GLOBAL batch;
// a sample's lookup whose bit is set in the previous step's bitmap is flagged in its samp entry (bit 30: positive,
// bit 31: negative) and read after the step barrier instead.  False positives only cost latency.
// A blocked Bloom filter: the hashed id picks ONE 32-bit word and two bits in it (one atomicOr to set, one load to
// test); at 16 bits per lookup that is ~2 % false positives against 6 % for a single bit.
struct DirtyProbe { uint32_t word, mask; };
__device__ __forceinline__ DirtyProbe dirty_probe(uint32_t id, int log2_bits, bool exact) {
    DirtyProbe p;
    if (exact) {
        p.word = id >> 5;
        p.mask = 1u << (id & 31u);
    } else {
        uint32_t h = id * 0x9E3779B1u;
        h ^= h >> 15;
        h *= 0x85EBCA77u;
        h ^= h >> 13;
        p.word = h >> (37 - log2_bits);
        p.mask = (1u << (h & 31u)) | (1u << ((h >> 5) & 31u));
    }
    return p;
}
__device__ __forceinline__ bool dirty_test(const uint32_t* bm, uint32_t id, int log2_bits, bool exact) {
    const DirtyProbe p = dirty_probe(id, log2_bits, exact);
    return (bm[p.word] & p.mask) == p.mask;
}
__global__ void __launch_bounds__(RT_THREADS)
dirty_bitmap_kernel(const int64_t* __restrict__ pos, const int64_t* __restrict__ neg, int64_t n_samples, int B,
                    uint32_t* __restrict__ bitmap, int log2_bits, bool exact) {
    const int64_t step = blockIdx.y;
    const int Bs = (int)min((int64_t)B, n_samples - step * B);
    const int64_t s0 = step * (int64_t)B;
    uint32_t* bm = bitmap + ((size_t)step << (log2_bits - 5));
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int j = blockIdx.x * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (j < 2 * Bs) {
            const DirtyProbe p = dirty_probe(route_id(pos, neg, s0, Bs, j), log2_bits, exact);
            atomicOr(bm + p.word, p.mask);
        }
    }
}
__global__ void __launch_bounds__(RT_THREADS)
dirty_mark_kernel(const int64_t* __restrict__ pos, const int64_t* __restrict__ neg, int64_t n_samples, int B,
                  const uint32_t* __restrict__ bitmap, int log2_bits, bool exact, const uint32_t* __restrict__ samp_cnt,
                  uint32_t* __restrict__ samp) {
    const int64_t step = blockIdx.y;
    const int64_t s0 = step * (int64_t)B;
    const int n = (int)samp_cnt[step];
    const uint32_t* bm = step > 0 ? bitmap + ((size_t)(step - 1) << (log2_bits - 5)) : nullptr;
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int k = blockIdx.x * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (k < n) {
            const uint32_t b = samp[s0 + k];
            uint32_t fl = 3u;  // the first step of a plan: nothing is known about the step before it
            if (bm) {
                fl = (dirty_test(bm, (uint32_t)pos[s0 + b], log2_bits, exact) ? 1u : 0u) |
                     (dirty_test(bm, (uint32_t)neg[s0 + b], log2_bits, exact) ? 2u : 0u);
            }
            samp[s0 + k] = b | (fl << 30);
        }
    }
}
// the row of sorted pair k (of n) has another lookup in the step
__device__ __forceinline__ bool pair_multi(const uint32_t* K, int n, int k) {
    const uint32_t key = K[k];
    return (k > 0 && K[k - 1] == key) || (k + 1 < n && K[k + 1] == key);
}
// A user row looked up exactly ONCE in a step has no other reader or writer in that step (every sample of a user runs
// on the user row's owner): its sample updates it in phase A.  Marks the sample (SAMP_USER_SINGLE) and the sorted
// pair (VAL_DONE_IN_A: phase B skips it).  Runs after dirty_mark_kernel (which rewrites the samp entries); every
// sample has one user lookup, so no two threads touch the same entry.
// The user rows that are NOT single in a step are updated by its phase B: their (local) rows go into a hashed bitmap
// per step, and user_dirty_mark_kernel flags the next step's samples that read one of them (SAMP_DIRTY_USER).
__global__ void __launch_bounds__(RT_THREADS)
single_mark_kernel(const uint32_t* __restrict__ ukey, uint32_t* __restrict__ uval, const uint32_t* __restrict__ own_cnt,
                   uint32_t* __restrict__ samp, int B, uint32_t* __restrict__ ubitmap, int log2_bits) {
    const int64_t step = blockIdx.y;
    const int64_t s0 = step * (int64_t)B;
    const int n = (int)own_cnt[2 * step];
    const uint32_t* K = ukey + s0;
    uint32_t* P = uval + s0;
    uint32_t* S = samp + s0;
    uint32_t* bm = ubitmap + ((size_t)step << (log2_bits - 5));
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int k = blockIdx.x * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (k >= n) continue;
        const uint32_t key = K[k];
        if (pair_multi(K, n, k)) {
            const DirtyProbe p = dirty_probe(key, log2_bits, false);
            atomicOr(bm + p.word, p.mask);
            continue;
        }
        const uint32_t idx = P[k];  // the sample's index in the rank's list
        S[idx] |= 1u << 27;
        P[k] = idx | (1u << 31);
    }
}

// Phase B then only needs the user pairs that phase A does NOT finish: drop the marked ones (stable, in place, one CTA
// per step; a chunk is read completely before any of it is overwritten, and pairs only move towards the front).
__global__ void __launch_bounds__(1024)
user_compact_kernel(uint32_t* __restrict__ ukey, uint32_t* __restrict__ uval, uint32_t* __restrict__ own_cnt, int B) {
    __shared__ uint32_t s_w[32];
    const int64_t step = blockIdx.x;
    const int n = (int)own_cnt[2 * step];
    uint32_t* K = ukey + step * (int64_t)B;
    uint32_t* P = uval + step * (int64_t)B;
    uint32_t run = 0;
    for (int base = 0; base < n; base += 1024) {
        const int k = base + (int)threadIdx.x;
        uint32_t key = 0, val = 0;
        bool keep = false;
        if (k < n) {
            key = K[k];
            val = P[k];
            keep = (val & (1u << 31)) == 0u;
        }
        uint32_t tot;
        const uint32_t p = run + block_rank<1024>(keep, s_w, tot);
        if (keep) {
            K[p] = key;
            P[p] = val;
        }
        run += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) own_cnt[2 * step] = run;
}


__global__ void __launch_bounds__(RT_THREADS)
user_dirty_mark_kernel(const int64_t* __restrict__ user, int B, uint32_t world, const uint32_t* __restrict__ ubitmap,
                       int log2_bits, const uint32_t* __restrict__ samp_cnt, uint32_t* __restrict__ samp) {
    const int64_t step = blockIdx.y;
    const int64_t s0 = step * (int64_t)B;
    const int n = (int)samp_cnt[step];
    const uint32_t* bm = step > 0 ? ubitmap + ((size_t)(step - 1) << (log2_bits - 5)) : nullptr;
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int k = blockIdx.x * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (k < n) {
            const uint32_t e = samp[s0 + k];
            bool d = true;  // the first step of a plan: nothing is known about the step before it
            if (bm) {
                d = dirty_test(bm, (uint32_t)user[s0 + (e & 0x07FFFFFFu)] / world, log2_bits, false);
            }
            if (d) samp[s0 + k] = e | (1u << 28);
        }
    }
}

// One rank: an item row looked up ONCE in a step has no other reader or writer in it either, so the one-pass kernel
// updates it in phase A like a single user row.  Per step the count launch marks every item lookup slot single or not
// (iflag); the scatter launch copies the other pairs, whole runs in order, to ikeyB / ivalB: what phase B still does.
struct ItemMultiSel {
    const uint32_t *ikey, *ival, *own_cnt;
    int B;
    uint8_t* iflag;
    uint32_t *ikeyB, *ivalB, *cntB;
    __device__ __forceinline__ int len(int64_t step) const { return (int)own_cnt[2 * step + 1]; }
    __device__ __forceinline__ bool keep(int64_t step, int k, int n, uint32_t&) const {
        return pair_multi(ikey + 2 * step * (int64_t)B, n, k);
    }
    __device__ __forceinline__ bool count(int64_t step, int k, int n) const {
        const int64_t seg = 2 * step * (int64_t)B;
        const bool m = pair_multi(ikey + seg, n, k);
        iflag[seg + ival[seg + k]] = m ? 0 : 1;
        return m;
    }
    __device__ __forceinline__ void emit(int64_t step, uint32_t p, int k, uint32_t) const {
        const int64_t seg = 2 * step * (int64_t)B;
        ikeyB[seg + p] = ikey[seg + k];
        ivalB[seg + p] = ival[seg + k];
    }
    __device__ __forceinline__ void total(int64_t step, uint32_t t) const {
        cntB[2 * step] = own_cnt[2 * step];
        cntB[2 * step + 1] = t;
    }
};

// bits of a step's bitmap: 16x the item lookups of a step (~2 % false positives, see dirty_probe), or one bit per item if that is less
static int dirty_log2_bits(const trs_epoch* ep, int64_t n_items, bool* exact) {
    int lb = 10;
    while (((int64_t)1 << lb) < 32ll * ep->batch && lb < 28) ++lb;
    int le = 5;
    while (((int64_t)1 << le) < n_items) ++le;
    *exact = le <= lb;
    return *exact ? le : lb;
}

// scratch of the plan build: the radix sort's other (key, value) buffers, sized for the item space (two lookups per
// sample), the per-tile counts of the route kernels, the sort's digit histograms and the dirty bitmaps of every step,
// one for the item rows and one for the user rows
struct ShardPlanTmp {
    size_t tkey, tval, tile_cnt, hist, bitmap, ubitmap, total;
};
static ShardPlanTmp shard_plan_tmp(const trs_epoch* ep) {
    ShardPlanTmp L;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    const size_t n = (size_t)ep->n_samples, steps = (size_t)n_steps_of(ep);
    const size_t tiles = (size_t)((2ll * ep->batch + RT_TILE - 1) / RT_TILE);
    bool exact;
    const int lb = dirty_log2_bits(ep, (int64_t)1 << 40, &exact);  // the hashed size: an exact bitmap is never larger
    L.tkey = take(2 * n * sizeof(uint32_t));
    L.tval = take(2 * n * sizeof(uint32_t));
    L.tile_cnt = take(steps * tiles * sizeof(uint32_t));
    L.hist = take(hist_bytes(ep));
    L.bitmap = take((steps << lb) / 8);
    L.ubitmap = take((steps << lb) / 8);
    L.total = off;
    return L;
}

// ------------------------------------------------------------------------------------------------------------
// the step kernels
// ------------------------------------------------------------------------------------------------------------
// samp entries of the plan: position of the sample in its step | flags
constexpr uint32_t SAMP_POS = 0x07FFFFFFu;          // position b in the global step (global batch < 2^27)
constexpr uint32_t SAMP_USER_SINGLE = 1u << 27;     // the user row is looked up once in the step: phase A updates it
constexpr uint32_t SAMP_DIRTY_USER = 1u << 28;      // the user row had several lookups in the previous step (phase B updates it)
constexpr uint32_t SAMP_DIRTY_POS = 1u << 30;       // the positive / negative item row is updated by the previous step
constexpr uint32_t SAMP_DIRTY_NEG = 1u << 31;
constexpr uint32_t SAMP_DIRTY_ANY = SAMP_DIRTY_USER | SAMP_DIRTY_POS | SAMP_DIRTY_NEG;
constexpr uint32_t VAL_DONE_IN_A = 1u << 31;        // sorted (row, slot) pair whose row phase A updates itself

// Thread-private 16-byte shared-memory slots per chunk a lane owns: phase A keeps SB samples x {user, positive,
// negative} row in flight per row group, phase B PB owned rows x {gradient, parameter, state 0, state 1}.
template <int IT>
constexpr int shard_slots() { return 12; }

struct ShardCtx {  // everything one (virtual) rank needs; copied to shared memory by each of its CTAs
    int rank, world, dim;
    int overlap;  // phase A starts on the samples the previous step does not touch before that step's end barrier
    trs_table user[TRS_MAX_RANKS];
    trs_table item[TRS_MAX_RANKS];
    float* stage_u[TRS_MAX_RANKS];  // [B, dim]   gradient rows of the user lookups, slot = sample position in the step
    float* stage_i[TRS_MAX_RANKS];  // [2B, dim]  positives then negatives
    float* stage_b[TRS_MAX_RANKS];  // [2B]       d item_bias
    size_t stage_par;               // floats between the two copies of the staging buffers (step parity)
    unsigned* sync[TRS_MAX_RANKS];
    const uint32_t *samp_cnt, *own_cnt, *samp, *ukey, *uval, *ikey, *ival;
    float* loss_part;  // [n_steps][cta_per_rank]
    float* loss_out;   // [n_steps]
    int* status;
    unsigned long long* trace;  // debug (trs_debug_shard_trace): [n_steps][cta_per_rank][8] globaltimer stamps, or NULL
};

template <int IT>
constexpr int shard_threads() { return IT <= 2 ? 512 : 256; }
template <int IT>
constexpr size_t shard_smem_bytes() { return (size_t)shard_threads<IT>() * shard_slots<IT>() * IT * 16; }

// ---- barriers -------------------------------------------------------------------------------------------------
// A monotonic arrival counter per rank (word 64 of its sync words).  A CTA arrives with ONE release fence (bar.sync before it:
// the stores of its whole CTA happen before the fence) followed by a relaxed add of 1 to the counter of every rank
// it must meet, polls its OWN rank's counter with relaxed loads until all arrivals of this barrier are in, and ends
// the wait with one acquire load (the counter is a chain of read-modify-writes: reading its final value
// synchronises with every arrival).
//   * the fence is SYSTEM scope only after a phase that stored into peer memory (the gradient rows: they must have
//     landed before the peer sees the arrival).  After the owners' update -- stores into the rank's OWN memory, which
//     peers read over NVLink through this GPU's L2 -- a gpu-scope fence puts them there.
//   * measured on 2 x B200 with no work between barriers: 8.7 us per barrier with a release-add per peer plus an
//     acq_rel.sys fence after the wait (each system-scope fence costs 2-3 us), and ~10 us with the
//     sequentially-consistent __threadfence_system() of a last-CTA-posts-flags scheme.
// Arrivals are never reset across launches: the target only depends on how many barriers the group has passed,
// e * CTAs-per-rank * world.
__device__ __forceinline__ void spin_until(const ShardCtx& C, const unsigned* cnt, unsigned target, bool sys,
                                           unsigned long long timeout_ns) {
    volatile int* status = C.status;
    const unsigned long long t0 = global_ns();
    unsigned spins = 0;
    while ((int)((sys ? ld_relaxed_sys(cnt) : ld_relaxed_gpu(cnt)) - target) < 0) {
        if ((++spins & 1023u) == 0) {
            if (*status != 0) break;
            if (global_ns() - t0 > timeout_ns) {
                atomicExch(C.status, 1);
                break;
            }
        }
    }
}

// every CTA of every rank.  Split in two so that work which does not depend on the peers can sit between: arrive (one
// release fence + a relaxed add to every rank's counter) ...
__device__ __forceinline__ void cross_arrive(const ShardCtx& C, bool remote_writes) {
    __syncthreads();
    if (threadIdx.x == 0) {
        if (C.world > 1) {
            if (remote_writes) fence_acq_rel_sys(); else fence_acq_rel_gpu();
            for (int q = 0; q < C.world; ++q) red_relaxed_sys(C.sync[q] + 64);
        } else {
            fence_acq_rel_gpu();
            red_relaxed_gpu(C.sync[C.rank] + 64);
        }
    }
}
// ... and wait until every CTA of every rank has arrived at barrier number e (1-based over the life of the group)
__device__ __forceinline__ void cross_wait(const ShardCtx& C, unsigned e, unsigned cpr, unsigned long long timeout_ns) {
    if (threadIdx.x == 0) {
        const unsigned* mine = C.sync[C.rank] + 64;
        const unsigned target = e * cpr * (unsigned)C.world;
        const bool sys = C.world > 1;
        spin_until(C, mine, target, sys, timeout_ns);
        if (sys) (void)ld_acquire_sys(mine); else (void)ld_acquire_gpu(mine);
    }
    __syncthreads();
}

// samples per row group whose item rows the two-phase kernel fetches a step ahead (IT == 1 only: shared memory)
template <int G, int IT>
constexpr int shard_pf_samples() { return IT == 1 ? (G >= 8 ? 7 : 6) : 0; }  // what fits beside the 12 row slots in 227 KB
template <int G, int IT>
constexpr size_t shard_smem_total() {
    constexpr size_t NT = shard_threads<IT>(), GPB = NT / G, PFS = shard_pf_samples<G, IT>();
    return shard_smem_bytes<IT>() + GPB * PFS * 2 * ((size_t)G * IT * 16 + 16) + GPB * 8;
}
// The one-pass kernel has no region: per row group ONE_S samples in flight, each with its three rows and their
// optimizer states in ONE_SLOTS thread-private slots.  Two in flight measured 41.30 us per step at the benchmark's
// shape against 41.54 us with three (one B200 at 1000 W, profiles/shard_r3.md)
constexpr int ONE_S = 2, ONE_SLOTS = 9;
constexpr size_t one_pass_smem_total() { return (size_t)shard_threads<1>() * ONE_S * ONE_SLOTS * 16; }

// A sample's record, read once per step from plan + epoch data (immutable, so it may be fetched a step ahead):
// b = position in the step | flags (SAMP_*; 0xFFFFFFFF: no sample), lu / lp / ln the local rows of its user, positive
// and negative item.  q packs the owners of the three rows (4 bits each); the one-pass kernel, whose one rank owns
// every row, keeps there instead whether the positive (bit 0) / negative (bit 1) item row is looked up once in the step.
struct Rec { uint32_t b, q, lu, lp, ln; };
// the record that lane src of my row group holds
template <int G>
__device__ __forceinline__ Rec bcast_rec(const Rec& cur, int src) {
    Rec r;
    r.b = __shfl_sync(0xffffffffu, cur.b, src, G);
    r.q = __shfl_sync(0xffffffffu, cur.q, src, G);
    r.lu = __shfl_sync(0xffffffffu, cur.lu, src, G);
    r.lp = __shfl_sync(0xffffffffu, cur.lp, src, G);
    r.ln = __shfl_sync(0xffffffffu, cur.ln, src, G);
    return r;
}

// every thread of the CTA copies my rank's context into shared memory; the caller synchronises
template <int NT>
__device__ __forceinline__ void load_ctx(ShardCtx& C, const ShardCtx& ctx0, const ShardCtx* ctxs, int cpr) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(ctxs ? ctxs + blockIdx.x / cpr : &ctx0);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&C);
    for (int i = threadIdx.x; i < (int)(sizeof(ShardCtx) / 4); i += NT) dst[i] = src[i];
}

__device__ __forceinline__ int low_bit(uint32_t w) { return __ffs((int)w) - 1; }

// One thread of a step kernel: where its row group sits in the grid, its thread-private shared-memory slots, the
// current step, and the step pieces both kernels are built from.  Constructed after the context is in shared memory.
template <int KIND, int G, int IT>
struct StepThread {
    static constexpr int NT = shard_threads<IT>(), GPB = NT / G, GPW = 32 / G;
    static constexpr int PB = shard_slots<IT>() / 4;  // owned rows in flight per row group (phase B): 4 slots each
    static constexpr int DPL = (PB + G - 1) / G;      // row descriptors a lane fetches per phase-B round

    const ShardCtx& C;
    const OptScalars& opt;
    float4* const rows;  // [slot][IT][NT]
    const int cpr, c;    // CTAs per rank, mine among them
    const int gl, gfirst, gstride;
    const int goff;      // my group's position inside its warp: loops run on the warp's first group
    const int me, dim, nch;
    const uint32_t W;
    const bool wpow2;
    const int wshift;
    const trs_table& tU;
    const trs_table& tI;
    const bool item_lin;
    // L2 policies: a staged gradient row is written in phase A and read once in phase B of the same step -- it should
    // stay in L2 in between (evict_last) and leave right after (evict_first), while the table rows stream through.
    const uint64_t pol_keep, pol_drop;
    const unsigned sync_epoch;
    const unsigned long long timeout_ns;
    unsigned bar_no = 0;        // cross-rank barriers arrived at in this launch
    bool wait_pending = false;  // arrived at the barrier that ends a step, not yet waited for it (see phase A)
    // the current step (begin_step).  The staging buffers exist twice (step parity): a rank may already store step
    // s+1's gradient rows into a peer that is still reading step s's
    int64_t lo;
    int Bs, nU, nI;
    float invB, scale;
    size_t po;
    unsigned long long* tr;

    __device__ __forceinline__ StepThread(const ShardCtx& C_, const OptScalars& opt_, unsigned char* smem, int cpr_,
                                          unsigned sync_epoch_, unsigned long long timeout_ns_)
        : C(C_), opt(opt_), rows(reinterpret_cast<float4*>(smem)), cpr(cpr_), c(blockIdx.x % cpr_), gl(threadIdx.x % G),
          gfirst(c * GPB + threadIdx.x / G), gstride(cpr_ * GPB), goff((threadIdx.x / G) % GPW), me(C_.rank),
          dim(C_.dim), nch(C_.dim / 4), W((uint32_t)C_.world), wpow2((W & (W - 1u)) == 0u), wshift(low_bit(W)),
          tU(C_.user[me]), tI(C_.item[me]), item_lin(tI.lin != nullptr), pol_keep(l2_policy_evict_last()),
          pol_drop(l2_policy_evict_first()), sync_epoch(sync_epoch_), timeout_ns(timeout_ns_) {}

    // a global row id -> (owner rank, local row)
    __device__ __forceinline__ void split(uint32_t id, uint32_t& owner, uint32_t& local) const {
        if (wpow2) { owner = id & (W - 1u); local = id >> wshift; }
        else { owner = id % W; local = id / W; }
    }
    __device__ __forceinline__ void stamp(int k) const {
        if (tr && threadIdx.x == 0) tr[k] = global_ns();
    }

    // ---- slots ----
    __device__ __forceinline__ float4* slot(int j, int a) const { return rows + ((j * IT + a) * NT + threadIdx.x); }
    // my chunks of slot j; zero past the row's end, and everywhere when !valid (no sample: the scores still take
    // every lane of the group)
    __device__ __forceinline__ Row<4, IT> slot_row(int j, bool valid = true) const {
        Row<4, IT> x;
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            x.c[a] = Vec<4>::zero();
            if (valid && gl + a * G < nch) x.c[a].v = *slot(j, a);
        }
        return x;
    }
    // cp.async of my chunks of the row at base into slot j, with L2 policy *pol if given
    __device__ __forceinline__ void copy_row(int j, const float* base, const uint64_t* pol = nullptr) const {
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int ch = gl + a * G;
            if (ch < nch) {
                if (pol) cp_async16_hint(slot(j, a), base + (size_t)ch * 4, *pol);
                else cp_async16(slot(j, a), base + (size_t)ch * 4);
            }
        }
    }

    // ---- one sample -------------------------------------------------------------------------------------------
    // linear.py:78: s = <u, v> + b_u + b_i; loss.py:7-9: h = s- - s+ + 1, d/ds = [h >= 0] / B.  Returns h; g = d/ds
    // and the gradient rows of the user and both items (theirs as single rounded products: exactly what phase B
    // reads back from a staging buffer)
    __device__ __forceinline__ float sample_grads(const Row<4, IT>& xu, const Row<4, IT>& xp, const Row<4, IT>& xn,
                                                  float bu, float bip, float bin, float& g, Row<4, IT>& gu,
                                                  Row<4, IT>& gp, Row<4, IT>& gn) const {
        const float sp = (group_sum<G>(row_dot_partial(xu, xp)) + bu) + bip;
        const float sn = (group_sum<G>(row_dot_partial(xu, xn)) + bu) + bin;
        const float h = __fadd_rn(__fsub_rn(sn, sp), 1.0f);
        g = (h >= 0.f) ? invB : 0.f;
#pragma unroll
        for (int a = 0; a < IT; ++a)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                gu.c[a][e] = g * (xn.c[a][e] - xp.c[a][e]);
                gp.c[a][e] = __fmul_rn(-g, xu.c[a][e]);
                gn.c[a][e] = __fmul_rn(g, xu.c[a][e]);
            }
        return h;
    }
    // the optimizer state of a row (what KIND keeps) from slots s_slot, s_slot + 1
    __device__ __forceinline__ void slot_state(int s_slot, Row<4, IT>& s0, Row<4, IT>& s1) const {
        row_zero(s0);
        row_zero(s1);
        if (KIND != TRS_OPT_SGD) s0 = slot_row(s_slot);
        if (KIND == TRS_OPT_SPARSE_ADAM) s1 = slot_row(s_slot + 1);
    }
    // update row `row` of t from its parameter p and state s0 / s1 in registers with gradient g, and store it; lin:
    // also its width-1 companion (gradient gb, value pl, state l0 / l1)
    __device__ __forceinline__ void update_row(const trs_table& t, uint32_t row, Row<4, IT> p, Row<4, IT> s0,
                                               Row<4, IT> s1, const Row<4, IT>& g, bool lin = false, float gb = 0.f,
                                               float pl = 0.f, float l0 = 0.f, float l1 = 0.f) const {
        OptScalars ok = opt;
        ok.kind = KIND;  // compile-time optimizer: opt_update's branches fold
        update_store_row<4, G, IT>(t, (size_t)row * dim, nch, gl, ok, scale, p, s0, s1, g);
        if (lin && gl == 0) update_store_lin(t, row, ok, scale, gb, pl, l0, l1);
    }
    // store my chunks of gradient row g into a staging buffer at dst, with the L2 policy evict_last if hint, and the
    // bias gradient gb at bdst if given: the row's owner reads them once in phase B of this step
    __device__ __forceinline__ void stage_row(float* dst, const Row<4, IT>& g, bool hint, float* bdst = nullptr,
                                              float gb = 0.f) const {
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int ch = gl + a * G;
            if (ch < nch) {
                if (hint) st_v4_hint(dst + (size_t)ch * 4, g.c[a].v, pol_keep);
                else g.c[a].st(dst + (size_t)ch * 4);
            }
        }
        if (bdst && gl == 0) *bdst = gb;
    }
    // a row phase A updates itself: parameter x in registers, state in slots s_slot, s_slot + 1
    __device__ __forceinline__ void update_row_at(const trs_table& t, uint32_t row, const Row<4, IT>& x, int s_slot,
                                                  const Row<4, IT>& g, bool lin = false, float gb = 0.f,
                                                  float pl = 0.f, float l0 = 0.f, float l1 = 0.f) const {
        Row<4, IT> s0, s1;
        slot_state(s_slot, s0, s1);
        update_row(t, row, x, s0, s1, g, lin, gb, pl, l0, l1);
    }
    // the user row of sample bf (owner qu, local row lu): a row this step looks up ONCE (plan flag: no other sample of
    // the global batch reads or writes it, and its owner is this rank) is updated right here from its state in slots
    // su_slot + 1 / + 2; every other one goes to its owner's staging buffer
    __device__ __forceinline__ void user_row(uint32_t bf, uint32_t qu, uint32_t lu, const Row<4, IT>& xu,
                                             const Row<4, IT>& gu, int su_slot) const {
        if (bf & SAMP_USER_SINGLE) update_row_at(C.user[qu], lu, xu, su_slot + 1, gu);
        else stage_row(C.stage_u[qu] + po + (size_t)(bf & SAMP_POS) * dim, gu, true);
    }

    // ---- the step frame ---------------------------------------------------------------------------------------
    __device__ __forceinline__ void begin_step(const trs_epoch& ep, int64_t s, int si) {
        lo = s * (int64_t)ep.batch;
        Bs = (int)min((int64_t)ep.batch, ep.n_samples - lo);
        invB = 1.0f / (float)Bs;
        scale = opt.step_scale[s];
        nU = (int)C.own_cnt[2 * s];
        nI = (int)C.own_cnt[2 * s + 1];
        po = (s & 1) ? C.stage_par : 0;
        tr = C.trace ? C.trace + ((size_t)si * cpr + c) * 8 : nullptr;
        stamp(0);
        // this step's phase-B lists (sorted keys and slots, streamed from HBM exactly once) -> L2 now: a round's
        // descriptor fetch then costs an L2 hit instead of a DRAM round trip in front of every round
        const int lu = (nU * 4 + 127) / 128, li = (nI * 4 + 127) / 128;
        for (int t = c * NT + (int)threadIdx.x; t < 2 * (lu + li); t += cpr * NT) {
            const char* base = t < lu ? (const char*)(C.ukey + lo)
                             : t < 2 * lu ? (const char*)(C.uval + lo)
                             : t < 2 * lu + li ? (const char*)(C.ikey + 2 * lo) : (const char*)(C.ival + 2 * lo);
            const int line = t < lu ? t : t < 2 * lu ? t - lu : t < 2 * lu + li ? t - 2 * lu : t - 2 * lu - li;
            prefetch_l2(base + (size_t)line * 128);
        }
    }
    // wait for the barrier that ends the previous step (arrived at by arrive())
    __device__ __forceinline__ void wait_step_end() {
        stamp(5);
        cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);
        wait_pending = false;
        stamp(6);
    }
    // the CTA's hinge sum of the step (h: my row group's, valid on lane 0 of the group)
    __device__ __forceinline__ void loss_partial(int si, float h) const {
        __shared__ float s_loss[NT / 32];
        const float hsum = warp_sum(gl == 0 ? h : 0.f);
        if ((threadIdx.x & 31) == 0) s_loss[threadIdx.x >> 5] = hsum;
        __syncthreads();
        if (threadIdx.x == 0) {
            float H = 0.f;
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) H += s_loss[w];
            C.loss_part[(size_t)si * cpr + c] = H;
            if (tr) tr[1] = global_ns();
        }
    }
    // the gradient rows have landed in their owners' staging buffers
    __device__ __forceinline__ void phase_a_barrier() {
        ++bar_no;
        cross_arrive(C, true);
        cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);
        stamp(2);
    }
    // the owners' updates are done: arrive, and wait inside the next step's phase A
    __device__ __forceinline__ void arrive() {
        if (tr) {
            __syncthreads();
            stamp(3);
        }
        ++bar_no;
        cross_arrive(C, false);
        wait_pending = true;
        stamp(4);
    }
    // after the last step: per-step hinge sums of this rank, CTAs added in a fixed order
    __device__ __forceinline__ void finish(int n_steps) {
        if (wait_pending) cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);
        if (c == 0) {
            for (int si = threadIdx.x; si < n_steps; si += NT) {
                float H = 0.f;
                for (int q = 0; q < cpr; ++q) H += __ldcg(C.loss_part + (size_t)si * cpr + q);
                C.loss_out[si] = H;
            }
        }
    }

    // ---- phase B ----------------------------------------------------------------------------------------------
    // The owned lookups of a step are one list of positions, user space [0, nU) then item space [nU, nU + nI); lane gl
    // fetches the descriptors of positions gl, gl + G, ... of a round.  sf = slot | flags << 29; flag bits: 1 head
    // (first position of a run of equal rows that phase A has not updated already), 2 the run continues, 4 item space
    struct Desc { uint32_t key[DPL], sf[DPL]; };
    __device__ __forceinline__ void fetch_descs(Desc& Dd, int pb) const {
#pragma unroll
        for (int z = 0; z < DPL; ++z) {
            const int i = gl + z * G;
            const int p = pb + i * gstride;
            Dd.key[z] = Dd.sf[z] = 0u;
            if (i < PB && p < nU + nI) {
                const bool it = p >= nU;
                const int k = it ? p - nU : p, n = it ? nI : nU;
                const uint32_t* K = it ? C.ikey + 2 * lo : C.ukey + lo;
                const uint32_t* P = it ? C.ival + 2 * lo : C.uval + lo;
                const uint32_t key = __ldg(K + k);
                const uint32_t prev = k > 0 ? __ldg(K + k - 1) : ~key;
                const uint32_t next = k + 1 < n ? __ldg(K + k + 1) : ~key;
                const uint32_t v = __ldg(P + k);
                const bool head = prev != key && !(v & VAL_DONE_IN_A);
                // item space: the value is the staging slot; user space: the sample's index in the rank's list
                const uint32_t sl = it ? v : (head ? (__ldg(C.samp + lo + (v & 0x1FFFFFFFu)) & SAMP_POS) : 0u);
                Dd.key[z] = key;
                Dd.sf[z] = (sl & 0x1FFFFFFFu) | ((head ? 1u : 0u) | (next == key ? 2u : 0u) | (it ? 4u : 0u)) << 29;
            }
        }
    }
    // Owned rows: a row group takes PB positions of the step's sorted list per round (dB: my first round's
    // descriptors); only the first position of a run of equal rows works (it sums the run's staged rows in slot
    // order); rows phase A updated are skipped.
    __device__ __forceinline__ void phase_b(Desc& dB) const {
        const int nP = nU + nI;
        const float* const my_stage_u = C.stage_u[me] + po;
        const float* const my_stage_i = C.stage_i[me] + po;
        const float* const my_stage_b = C.stage_b[me] + po;
        for (int p0 = gfirst - goff; p0 < nP; p0 += gstride * PB) {  // warp-uniform trip count
            const int pb = p0 + goff;
            float bsc[PB];  // lanes 0..3: staged bias gradient, bias, its state 0 / 1 of position i
#pragma unroll
            for (int i = 0; i < PB; ++i) {
                const uint32_t key = __shfl_sync(0xffffffffu, dB.key[i / G], i % G, G);
                const uint32_t sf = __shfl_sync(0xffffffffu, dB.sf[i / G], i % G, G);
                const uint32_t sl = sf & 0x1FFFFFFFu;
                bsc[i] = 0.f;
                if (sf & (1u << 29)) {
                    const bool it = (sf >> 31) != 0u;
                    const trs_table& t = it ? tI : tU;
                    const size_t roff = (size_t)key * dim;
                    copy_row(i * 4 + 0, (it ? my_stage_i : my_stage_u) + (size_t)sl * dim, &pol_drop);
                    copy_row(i * 4 + 1, t.emb + roff);
                    if (KIND != TRS_OPT_SGD) copy_row(i * 4 + 2, t.emb_s0 + roff);
                    if (KIND == TRS_OPT_SPARSE_ADAM) copy_row(i * 4 + 3, t.emb_s1 + roff);
                    if (it && item_lin && gl < 4) {
                        if (gl == 0) bsc[i] = __ldcg(my_stage_b + sl);
                        else if (gl == 1) bsc[i] = __ldcg(t.lin + key);
                        else if (gl == 2) { if (KIND != TRS_OPT_SGD) bsc[i] = __ldcg(t.lin_s0 + key); }
                        else { if (KIND == TRS_OPT_SPARSE_ADAM) bsc[i] = __ldcg(t.lin_s1 + key); }
                    }
                }
                cp_async_commit();
            }
            Desc cur = dB;
            if (p0 + gstride * PB < nP) fetch_descs(dB, pb + gstride * PB);
#pragma unroll
            for (int i = 0; i < PB; ++i) {
                cp_async_wait(PB - 1 - i);
                const uint32_t key = __shfl_sync(0xffffffffu, cur.key[i / G], i % G, G);
                const uint32_t sf = __shfl_sync(0xffffffffu, cur.sf[i / G], i % G, G);
                const bool it = (sf >> 31) != 0u;
                float gb = 0.f, pl = 0.f, l0 = 0.f, l1 = 0.f;
                if (G < 32 || it) {  // one row group per warp: the branch is warp-uniform
                    gb = __shfl_sync(0xffffffffu, bsc[i], 0, G);
                    pl = __shfl_sync(0xffffffffu, bsc[i], 1, G);
                    if (KIND != TRS_OPT_SGD) l0 = __shfl_sync(0xffffffffu, bsc[i], 2, G);
                    if (KIND == TRS_OPT_SPARSE_ADAM) l1 = __shfl_sync(0xffffffffu, bsc[i], 3, G);
                }
                if (!(sf & (1u << 29))) continue;
                Row<4, IT> g = slot_row(i * 4 + 0), p = slot_row(i * 4 + 1), s0, s1;
                slot_state(i * 4 + 2, s0, s1);
                if (sf & (1u << 30)) {  // duplicates (rare under uniform ids): the rest of the run, in slot order
                    const int pos = pb + i * gstride;
                    const int k = it ? pos - nU : pos, n = it ? nI : nU;
                    const uint32_t* K = it ? C.ikey + 2 * lo : C.ukey + lo;
                    const uint32_t* P = it ? C.ival + 2 * lo : C.uval + lo;
                    const float* stage = it ? my_stage_i : my_stage_u;
                    for (int q = k + 1; q < n && __ldg(K + q) == key; ++q) {
                        const uint32_t v = __ldg(P + q) & 0x1FFFFFFFu;
                        const uint32_t j = it ? v : (__ldg(C.samp + lo + v) & SAMP_POS);
                        row_acc(g, load_row_cg<4, G, IT>(stage + (size_t)j * dim, nch, gl));
                        if (it && item_lin && gl == 0) gb = __fadd_rn(gb, __ldcg(my_stage_b + j));
                    }
                }
                update_row(it ? tI : tU, key, p, s0, s1, g, it && item_lin, gb, pl, l0, l1);
            }
        }
    }
};

// ---- the two-phase kernel ---------------------------------------------------------------------------------------
// The item rows (and the 16-byte line holding each one's bias) of my row group's first PFS samples, in a region of
// contiguous row slots: row j = 2 * sample ordinal + {0 positive, 1 negative}.  Filled a step ahead by bulk copies
// (one mbarrier per row group), or in phase A by cp.async for the rows the previous step updated.
template <int G, int IT>
struct ItemRegion {
    static constexpr int ROWB = G * IT * 16;  // bytes of a row slot
    unsigned char* rows;
    unsigned char* bias;
    uint64_t* bar;
    __device__ __forceinline__ Row<4, IT> row(int j, int gl, int nch, bool valid) const {  // as StepThread::slot_row
        Row<4, IT> x;
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            x.c[a] = Vec<4>::zero();
            if (valid && gl + a * G < nch) x.c[a].v = *reinterpret_cast<const float4*>(rows + (size_t)j * ROWB + (gl + a * G) * 16);
        }
        return x;
    }
    __device__ __forceinline__ void copy(int j, const float* base, int gl, int nch) const {
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int ch = gl + a * G;
            if (ch < nch) cp_async16(rows + (size_t)j * ROWB + ch * 16, base + (size_t)ch * 4);
        }
    }
    __device__ __forceinline__ float bias_of(int j, uint32_t lrow) const {
        return reinterpret_cast<const float*>(bias + (size_t)j * 16)[lrow & 3u];
    }
};

// Records of a two-phase round: lane gl fetches samples gl, gl + G, ... of the round (cnt of them, from my group's
// list position kb on) and splits their ids into (owner, local row) once
template <int RPL, int KIND, int G, int IT>
__device__ __forceinline__ void fetch_records(const StepThread<KIND, G, IT>& L, const trs_epoch& ep, Rec (&R)[RPL],
                                              int64_t lo, int nS, int kb, int cnt) {
    const uint32_t* samp = L.C.samp + lo;
#pragma unroll
    for (int z = 0; z < RPL; ++z) {
        const int i = L.gl + z * G;
        const int k = kb + i * L.gstride;
        R[z].b = 0xFFFFFFFFu;
        R[z].q = R[z].lu = R[z].lp = R[z].ln = 0u;
        if (i < cnt && k < nS) {
            const uint32_t bf = __ldg(samp + k);
            const uint32_t b = bf & SAMP_POS;
            R[z].b = bf;
            uint32_t qu, qp, qn;
            L.split((uint32_t)__ldg(ep.user + lo + b), qu, R[z].lu);
            L.split((uint32_t)__ldg(ep.pos + lo + b), qp, R[z].lp);
            L.split((uint32_t)__ldg(ep.neg + lo + b), qn, R[z].ln);
            R[z].q = qu | (qp << 4) | (qn << 8);
        }
    }
}

// One phase-A round of the two-phase kernel: NS samples of my row group with records cur, issued, then run in order.
// REGION: a regular round -- item rows in the region (sample ordinals o_lo ..; rows already there when pf_live and
// the sample is clean), user row + state in slots 3i .. 3i + 2, only the samples of this pass (late: the flagged ones,
// when overlap is on), hinges into hreg.  Otherwise an overflow round -- all five rows in slots 5i .. 5i + 4, hinges
// into hover.  Every item gradient row goes to its owner's staging buffer.
template <bool REGION, int NS, int RPL, int KIND, int G, int IT>
__device__ __forceinline__ void two_phase_round(const StepThread<KIND, G, IT>& L, const ItemRegion<G, IT>& R,
                                                const Rec (&cur)[RPL], int rnd, int o_lo, int n_r, bool late,
                                                bool overlap, bool pf_live, bool hint_remote, float (&hreg)[8],
                                                float& hover) {
    constexpr int ST = REGION ? 3 : 5;  // slots per sample
    const ShardCtx& C = L.C;
    const int gl = L.gl, dim = L.dim, nch = L.nch;
    auto runs = [&](uint32_t bf, int i) {
        return i < n_r && bf != 0xFFFFFFFFu && (!REGION || (overlap ? ((bf & SAMP_DIRTY_ANY) != 0u) == late : !late));
    };
    float bias_r[NS];  // lane t < 3 holds the width-1 companion of lookup t (user, positive, negative)
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        const Rec r = bcast_rec<G>(cur[i / G], i % G);
        bias_r[i] = 0.f;
        if (runs(r.b, i)) {
            const trs_table& TU = C.user[r.q & 15u];
            const trs_table& TP = C.item[(r.q >> 4) & 15u];
            const trs_table& TN = C.item[(r.q >> 8) & 15u];
            L.copy_row(i * ST + 0, TU.emb + (size_t)r.lu * dim);
            if (r.b & SAMP_USER_SINGLE) {
                if (KIND != TRS_OPT_SGD) L.copy_row(i * ST + 1, TU.emb_s0 + (size_t)r.lu * dim);
                if (KIND == TRS_OPT_SPARSE_ADAM) L.copy_row(i * ST + 2, TU.emb_s1 + (size_t)r.lu * dim);
            }
            bool have_p = false, have_n = false;
            if (REGION) {
                have_p = pf_live && !(r.b & SAMP_DIRTY_POS);
                have_n = pf_live && !(r.b & SAMP_DIRTY_NEG);
                if (!have_p) R.copy((o_lo + i) * 2 + 0, TP.emb + (size_t)r.lp * dim, gl, nch);
                if (!have_n) R.copy((o_lo + i) * 2 + 1, TN.emb + (size_t)r.ln * dim, gl, nch);
            } else {
                L.copy_row(i * ST + 3, TP.emb + (size_t)r.lp * dim);
                L.copy_row(i * ST + 4, TN.emb + (size_t)r.ln * dim);
            }
            if (gl < 3) {
                const float* lin = gl == 0 ? TU.lin : (gl == 1 ? TP.lin : TN.lin);
                const uint32_t lrow = gl == 0 ? r.lu : (gl == 1 ? r.lp : r.ln);
                const bool have = gl == 1 ? have_p : (gl == 2 ? have_n : false);
                if (lin) bias_r[i] = have ? R.bias_of((o_lo + i) * 2 + (gl - 1), lrow) : __ldcg(lin + lrow);
            }
        }
        cp_async_commit();
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        cp_async_wait(NS - 1 - i);
        const Rec r = bcast_rec<G>(cur[i / G], i % G);
        const bool valid = runs(r.b, i);
        const Row<4, IT> xu = L.slot_row(i * ST + 0, valid);
        const Row<4, IT> xp = REGION ? R.row((o_lo + i) * 2 + 0, gl, nch, valid) : L.slot_row(i * ST + 3, valid);
        const Row<4, IT> xn = REGION ? R.row((o_lo + i) * 2 + 1, gl, nch, valid) : L.slot_row(i * ST + 4, valid);
        const float bu = __shfl_sync(0xffffffffu, bias_r[i], 0, G);
        const float bip = __shfl_sync(0xffffffffu, bias_r[i], 1, G);
        const float bin = __shfl_sync(0xffffffffu, bias_r[i], 2, G);
        float g;
        Row<4, IT> gu, gp, gn;
        const float h = L.sample_grads(xu, xp, xn, bu, bip, bin, g, gu, gp, gn);
        float hv = 0.f;
        if (valid) {
            hv = fmaxf(h, 0.f);
            const uint32_t b = r.b & SAMP_POS, qp = (r.q >> 4) & 15u, qn = (r.q >> 8) & 15u;
            L.stage_row(C.stage_i[qp] + L.po + (size_t)b * dim, gp, hint_remote || (int)qp == L.me);
            L.stage_row(C.stage_i[qn] + L.po + (size_t)(L.Bs + b) * dim, gn, hint_remote || (int)qn == L.me);
            if (gl == 0) {
                (C.stage_b[qp] + L.po)[b] = -g;
                (C.stage_b[qn] + L.po)[L.Bs + b] = g;
            }
            L.user_row(r.b, r.q & 15u, r.lu, xu, gu, i * ST);
        }
        if (!REGION) hover += hv;
        else if (valid) {
            if (rnd == 0) hreg[i] = hv; else hreg[NS + i] = hv;
        }
    }
}

// Any group size, any row shape.  Phase A: the item rows of a group's first PFS samples sit in its region; the 12
// thread-private slots hold the USER row with its optimizer state for SBA = 4 samples at a time: regular rounds
// [0, SBA) and [SBA, PFS).  Samples beyond PFS (and every sample when there is no region, IT > 1) go SBO = 2 per
// overflow round.  With overlap on, the regular rounds run in two passes: pass 0 takes the samples none of whose
// three rows the previous step's owners update (plan flags) BEFORE waiting for the barrier that ends the previous
// step -- their rows are final, and their gradient rows go to the other copy of the staging buffers -- then the wait,
// then pass 1 (the flagged samples) and the overflow rounds.  Phase B updates every owned row from the staged rows.
template <int KIND, int G, int IT>
__global__ void __launch_bounds__((shard_threads<IT>()), 1)
shard_train_kernel(const __grid_constant__ ShardCtx ctx0, const ShardCtx* __restrict__ ctxs, const int cpr,
                   const __grid_constant__ trs_epoch ep, const __grid_constant__ OptScalars opt, const int first_step,
                   const int n_steps, const unsigned sync_epoch, const unsigned long long timeout_ns) {
    using T = StepThread<KIND, G, IT>;
    constexpr int NT = T::NT, GPB = T::GPB;
    // The loss adds a group's hinges in this layout's order whichever kernel runs: ordinals [0, HREG) one by one
    // (then a + 0 per unused regular slot), the later ordinals in a sum of their own.
    constexpr int PFS = shard_pf_samples<G, IT>();
    constexpr int SBA = 4, SBO = 2;
    constexpr int NREG = PFS ? 2 : 0;          // regular rounds
    constexpr int NPR = NREG ? NREG : 1;       // rounds whose records are fetched a step ahead
    constexpr int RPL = (SBA + G - 1) / G;     // sample records a lane holds per round
    constexpr int ROWB = ItemRegion<G, IT>::ROWB;
    static_assert(shard_smem_total<G, IT>() + 2048 <= 227 * 1024, "shared memory budget");
    static_assert(!PFS || (PFS > SBA && PFS <= 2 * SBA), "round layout");
    __shared__ ShardCtx C;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char* pf_rows = smem_raw + shard_smem_bytes<IT>();             // [GPB][PFS][2][ROWB]
    unsigned char* pf_bias = pf_rows + (size_t)GPB * PFS * 2 * ROWB;       // [GPB][PFS][2][16]
    uint64_t* pf_bars = reinterpret_cast<uint64_t*>(pf_bias + (size_t)GPB * PFS * 2 * 16);  // [GPB]
    load_ctx<NT>(C, ctx0, ctxs, cpr);
    const int g_in_cta = threadIdx.x / G;
    const ItemRegion<G, IT> R{pf_rows + (size_t)g_in_cta * PFS * 2 * ROWB, pf_bias + (size_t)g_in_cta * PFS * 2 * 16,
                              pf_bars + g_in_cta};
    if (PFS && threadIdx.x % G == 0) mbar_init(R.bar, 1);
    if (PFS) fence_barrier_init();
    __syncthreads();
    T L(C, opt, smem_raw, cpr, sync_epoch, timeout_ns);
    const int gl = L.gl, dim = L.dim;
    const bool overlap = (C.overlap & 1) != 0;
    const bool hint_remote = (C.overlap & 2) != 0;   // L2 policy also on stores into peer memory
    auto round_lo = [](int r) { return r < NREG ? (r == 0 ? 0 : SBA) : PFS + SBO * (r - NREG); };
    auto round_n = [](int r) { return r < NREG ? (r == 0 ? SBA : PFS - SBA) : SBO; };

    Rec recN[NPR][RPL];  // records of the next phase A's first NPR rounds
    int nS_cur = (int)C.samp_cnt[first_step];
#pragma unroll
    for (int r = 0; r < NPR; ++r)
        fetch_records(L, ep, recN[r], (int64_t)first_step * ep.batch, nS_cur, L.gfirst + round_lo(r) * L.gstride,
                      round_n(r));
    bool pf_live = false;     // the current step's region holds prefetched item rows (all but the dirty ones)
    uint32_t pf_parity = 0;

    for (int si = 0; si < n_steps; ++si) {
        const int64_t s = first_step + si;
        L.begin_step(ep, s, si);
        const int nS = nS_cur;
        const bool more = si + 1 < n_steps;
        const int nS_next = more ? (int)C.samp_cnt[s + 1] : 0;

        // ------------------------------ phase A ------------------------------------------
        // hinge terms: one per regular-round sample, added up in sample order afterwards (the order in which the two
        // passes visit them depends on plan flags, the loss must not), then the overflow rounds' in visiting order
        float hreg[2 * SBA], hover = 0.f;
#pragma unroll
        for (int i = 0; i < 2 * SBA; ++i) hreg[i] = 0.f;
        if (PFS && pf_live) {  // rows fetched while the previous step's owners were updating: landed?
            mbar_wait(R.bar, pf_parity);
            pf_parity ^= 1u;
        }
        for (int rr = 0;; ++rr) {
            if (L.wait_pending && (rr == NREG || !overlap)) L.wait_step_end();  // every warp of the CTA, once per step
            const bool late = rr >= NREG;            // pass 1 / overflow
            const int rnd = late ? rr - NREG : rr;
            const int o_lo = round_lo(rnd), n_r = round_n(rnd);
            const int k0 = L.gfirst - L.goff + o_lo * L.gstride;
            if (k0 >= nS) {  // warp-uniform
                if (late) break;
                continue;
            }
            Rec cur[RPL];
            if (rnd < NPR) {
#pragma unroll
                for (int r = 0; r < NPR; ++r)
                    if (r == rnd)
#pragma unroll
                        for (int z = 0; z < RPL; ++z) cur[z] = recN[r][z];
            } else {
                fetch_records(L, ep, cur, L.lo, nS, k0 + L.goff, n_r);
            }
            if (rnd < NREG) {
                if (late) {  // nothing flagged in the warp's groups: pass 0 did the whole round
                    if (!overlap) continue;
                    bool d = false;
#pragma unroll
                    for (int z = 0; z < RPL; ++z) d = d || (cur[z].b != 0xFFFFFFFFu && (cur[z].b & SAMP_DIRTY_ANY) != 0u);
                    if (!__any_sync(0xffffffffu, d)) continue;
                }
                two_phase_round<true, SBA>(L, R, cur, rnd, o_lo, n_r, late, overlap, pf_live, hint_remote, hreg, hover);
            } else {
                two_phase_round<false, SBO>(L, R, cur, rnd, o_lo, SBO, late, overlap, pf_live, hint_remote, hreg, hover);
            }
        }
        // the next step's first rounds of records (plan + epoch data), then my first phase-B descriptors: all in
        // flight across the barrier
        if (more) {
#pragma unroll
            for (int r = 0; r < NPR; ++r)
                fetch_records(L, ep, recN[r], L.lo + ep.batch, nS_next, L.gfirst + round_lo(r) * L.gstride, round_n(r));
        }
        nS_cur = nS_next;
        typename T::Desc dB;
        L.fetch_descs(dB, L.gfirst);
        float hsum = 0.f;
#pragma unroll
        for (int i = 0; i < 2 * SBA; ++i) hsum += hreg[i];
        L.loss_partial(si, hsum + hover);
        L.phase_a_barrier();

        // ------------------------------ phase B ------------------------------------------
        // First the NEXT step's item rows: every clean one (not updated by this step, plan flag) of my group's first
        // PFS samples starts its trip -- from the owner's HBM, mostly over NVLink -- into the region and lands while
        // the owners update.  The lane that holds a sample's record issues its copies.
        pf_live = false;
        if (PFS && more) {
#pragma unroll
            for (int r = 0; r < NREG; ++r) {
#pragma unroll
                for (int z = 0; z < RPL; ++z) {
                    const int i = gl + z * G;
                    const Rec& n = recN[r][z];
                    if (i < round_n(r) && n.b != 0xFFFFFFFFu) {
                        const trs_table& TP = C.item[(n.q >> 4) & 15u];
                        const trs_table& TN = C.item[(n.q >> 8) & 15u];
                        const bool fp = !(n.b & SAMP_DIRTY_POS), fn = !(n.b & SAMP_DIRTY_NEG);
                        const uint32_t per = (uint32_t)dim * 4u + (TP.lin ? 16u : 0u);
                        const uint32_t bytes = (fp ? per : 0u) + (fn ? per : 0u);
                        if (bytes) mbar_expect_tx(R.bar, bytes);
                        const int j = (round_lo(r) + i) * 2;
                        if (fp) {
                            bulk_g2s(R.rows + (size_t)j * ROWB, TP.emb + (size_t)n.lp * dim, (uint32_t)dim * 4u, R.bar);
                            if (TP.lin) bulk_g2s(R.bias + (size_t)j * 16, TP.lin + (n.lp & ~3u), 16u, R.bar);
                        }
                        if (fn) {
                            bulk_g2s(R.rows + (size_t)(j + 1) * ROWB, TN.emb + (size_t)n.ln * dim, (uint32_t)dim * 4u, R.bar);
                            if (TN.lin) bulk_g2s(R.bias + (size_t)(j + 1) * 16, TN.lin + (n.ln & ~3u), 16u, R.bar);
                        }
                    }
                }
            }
            __syncwarp();  // every expect_tx of the group precedes its one arrival
            if (gl == 0) mbar_arrive(R.bar);
            pf_live = true;
        }
        L.phase_b(dB);
        L.arrive();  // waited for inside the next phase A (after its pass 0 when overlap is on)
    }
    L.finish(n_steps);
}

// ---- the one-pass kernel ----------------------------------------------------------------------------------------
// One rank in one launch, one chunk per lane.  Every item row's owner is the rank that reads it, so an item row the
// step looks up once (plan: iflag) is updated in phase A like a single user row; phase B only updates the rows with
// several lookups (plan: ikeyB / ivalB).
//
// Phase A is one pass over my group's samples in ordinal order (the loss order), after the wait for the previous
// step's end.  Sample o + ONE_S's rows start their trip (cp.async into slots ONE_SLOTS * j ..) before sample o runs:
// user, positive, negative row at + 0 / 3 / 6, each followed by its optimizer state when phase A updates that row.
template <int KIND, int G>
struct OnePassPipe {
    using T = StepThread<KIND, G, 1>;
    const T& L;
    const trs_epoch& ep;
    const uint8_t* iflag;
    Rec blk_rec;  // lane gl: the record of my group's ordinal blk * G + gl (q: iflag bits)
    int blk;
    Rec rec[ONE_S];             // the samples in flight
    float tv0[ONE_S], tv1[ONE_S];  // lane t & 3 holds scalar t of a sample in tv0 (t < 4) or tv1 (see scalar)

    __device__ __forceinline__ void fetch(int64_t lo, int nS, int b) {
        blk = b;
        const int k = L.gfirst + (b * G + L.gl) * L.gstride;
        blk_rec.b = 0xFFFFFFFFu;
        blk_rec.q = blk_rec.lu = blk_rec.lp = blk_rec.ln = 0u;
        if (k < nS) {
            const int Bs_ = (int)min((int64_t)ep.batch, ep.n_samples - lo);
            const uint32_t bf = __ldg(L.C.samp + lo + k);
            const uint32_t pos = bf & SAMP_POS;
            blk_rec.b = bf;
            blk_rec.lu = (uint32_t)__ldg(ep.user + lo + pos);
            blk_rec.lp = (uint32_t)__ldg(ep.pos + lo + pos);
            blk_rec.ln = (uint32_t)__ldg(ep.neg + lo + pos);
            blk_rec.q = (uint32_t)__ldg(iflag + 2 * lo + pos) | ((uint32_t)__ldg(iflag + 2 * lo + Bs_ + pos) << 1);
        }
    }
    // scalar t of sample r: 0 user bias, 1 / 2 positive / negative bias, 3 / 4 and 5 / 6 their states
    __device__ __forceinline__ float scalar(int t, const Rec& r) const {
        const bool p = t == 1 || t == 3 || t == 4;
        const float* src = t == 0 ? L.tU.lin : (t <= 2 ? L.tI.lin : nullptr);
        if (t >= 3 && L.item_lin && (r.q & (p ? 1u : 2u))) {
            if ((t == 3 || t == 5) && KIND != TRS_OPT_SGD) src = L.tI.lin_s0;
            if ((t == 4 || t == 6) && KIND == TRS_OPT_SPARSE_ADAM) src = L.tI.lin_s1;
        }
        return src ? __ldcg(src + (t == 0 ? r.lu : (p ? r.lp : r.ln))) : 0.f;
    }
    // start ordinal o's trip into pipeline entry j (nothing past nord)
    __device__ __forceinline__ void issue(int o, int j, int nord, int64_t lo, int nS) {
        Rec r;
        r.b = 0xFFFFFFFFu;
        r.q = r.lu = r.lp = r.ln = 0u;
        if (o < nord) {
            if (o / G != blk) fetch(lo, nS, o / G);
            r = bcast_rec<G>(blk_rec, o % G);
        }
        rec[j] = r;
        tv0[j] = tv1[j] = 0.f;
        if (r.b != 0xFFFFFFFFu) {
            const int sl = j * ONE_SLOTS;
            const trs_table& tU = L.tU;
            const trs_table& tI = L.tI;
            const int dim = L.dim;
            L.copy_row(sl + 0, tU.emb + (size_t)r.lu * dim);
            if (r.b & SAMP_USER_SINGLE) {
                if (KIND != TRS_OPT_SGD) L.copy_row(sl + 1, tU.emb_s0 + (size_t)r.lu * dim);
                if (KIND == TRS_OPT_SPARSE_ADAM) L.copy_row(sl + 2, tU.emb_s1 + (size_t)r.lu * dim);
            }
            L.copy_row(sl + 3, tI.emb + (size_t)r.lp * dim);
            if (r.q & 1u) {
                if (KIND != TRS_OPT_SGD) L.copy_row(sl + 4, tI.emb_s0 + (size_t)r.lp * dim);
                if (KIND == TRS_OPT_SPARSE_ADAM) L.copy_row(sl + 5, tI.emb_s1 + (size_t)r.lp * dim);
            }
            L.copy_row(sl + 6, tI.emb + (size_t)r.ln * dim);
            if (r.q & 2u) {
                if (KIND != TRS_OPT_SGD) L.copy_row(sl + 7, tI.emb_s0 + (size_t)r.ln * dim);
                if (KIND == TRS_OPT_SPARSE_ADAM) L.copy_row(sl + 8, tI.emb_s1 + (size_t)r.ln * dim);
            }
            if (L.gl < 4) {
                tv0[j] = scalar(L.gl, r);
                tv1[j] = scalar(L.gl + 4, r);
            }
        }
        cp_async_commit();
    }
    // run pipeline entry j: scores, hinge (returned, 0 for no sample), and the updates / staged rows of its three rows
    __device__ __forceinline__ float run(int j) const {
        const Rec& r = rec[j];
        const bool valid = r.b != 0xFFFFFFFFu;
        const int sl = j * ONE_SLOTS;
        const Row<4, 1> xu = L.slot_row(sl + 0, valid), xp = L.slot_row(sl + 3, valid), xn = L.slot_row(sl + 6, valid);
        const float bu = __shfl_sync(0xffffffffu, tv0[j], 0, G);
        const float bip = __shfl_sync(0xffffffffu, tv0[j], 1, G);
        const float bin = __shfl_sync(0xffffffffu, tv0[j], 2, G);
        const float pl0 = __shfl_sync(0xffffffffu, tv0[j], 3, G);
        const float pl1 = __shfl_sync(0xffffffffu, tv1[j], 0, G);
        const float nl0 = __shfl_sync(0xffffffffu, tv1[j], 1, G);
        const float nl1 = __shfl_sync(0xffffffffu, tv1[j], 2, G);
        float g;
        Row<4, 1> gu, gp, gn;
        const float h = L.sample_grads(xu, xp, xn, bu, bip, bin, g, gu, gp, gn);
        if (!valid) return 0.f;
        const ShardCtx& C = L.C;
        const uint32_t b = r.b & SAMP_POS;
        const size_t dim = (size_t)L.dim;
        if (r.q & 1u) L.update_row_at(L.tI, r.lp, xp, sl + 4, gp, L.item_lin, -g, bip, pl0, pl1);
        else L.stage_row(C.stage_i[L.me] + L.po + b * dim, gp, true, C.stage_b[L.me] + L.po + b, -g);
        if (r.q & 2u) L.update_row_at(L.tI, r.ln, xn, sl + 7, gn, L.item_lin, g, bin, nl0, nl1);
        else L.stage_row(C.stage_i[L.me] + L.po + (L.Bs + b) * dim, gn, true, C.stage_b[L.me] + L.po + L.Bs + b, g);
        L.user_row(r.b, L.me, r.lu, xu, gu, sl);
        return fmaxf(h, 0.f);
    }
};

template <int KIND, int G>
__global__ void __launch_bounds__((shard_threads<1>()), 1)
shard_train_one_pass_kernel(const __grid_constant__ ShardCtx ctx0, const ShardCtx* __restrict__ ctxs, const int cpr,
                            const __grid_constant__ trs_epoch ep, const __grid_constant__ OptScalars opt,
                            const int first_step, const int n_steps, const unsigned sync_epoch,
                            const unsigned long long timeout_ns, const uint8_t* __restrict__ iflag) {
    using T = StepThread<KIND, G, 1>;
    constexpr int HREG = shard_pf_samples<G, 1>();  // the two-phase kernel's regular-round ordinals (loss order)
    static_assert(one_pass_smem_total() + 2048 <= 227 * 1024, "shared memory budget");
    __shared__ ShardCtx C;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    load_ctx<T::NT>(C, ctx0, ctxs, cpr);
    __syncthreads();
    T L(C, opt, smem_raw, cpr, sync_epoch, timeout_ns);
    OnePassPipe<KIND, G> P{L, ep, iflag};
    int nS_cur = (int)C.samp_cnt[first_step];
    P.fetch((int64_t)first_step * ep.batch, nS_cur, 0);

    for (int si = 0; si < n_steps; ++si) {
        const int64_t s = first_step + si;
        L.begin_step(ep, s, si);
        const int nS = nS_cur;
        const bool more = si + 1 < n_steps;
        const int nS_next = more ? (int)C.samp_cnt[s + 1] : 0;

        // ------------------------------ phase A ------------------------------------------
        // hinges of ordinals [0, HREG) in one sum and the later ones in another: the two-phase kernel's association
        float hreg = 0.f, hover = 0.f;
        if (L.wait_pending) L.wait_step_end();
        const int kw = L.gfirst - L.goff;  // the warp's first group: the trip count is warp-uniform
        const int nord = kw < nS ? (nS - kw + L.gstride - 1) / L.gstride : 0;
#pragma unroll
        for (int j = 0; j < ONE_S; ++j) P.issue(j, j, nord, L.lo, nS);
        for (int o0 = 0; o0 < nord; o0 += ONE_S) {
#pragma unroll
            for (int j = 0; j < ONE_S; ++j) {
                cp_async_wait(ONE_S - 1);
                if (o0 + j < nord) {
                    const float hv = P.run(j);
                    if (o0 + j < HREG) hreg += hv; else hover += hv;
                }
                P.issue(o0 + j + ONE_S, j, nord, L.lo, nS);
            }
        }
        // block 0 of the next step's records, then my first phase-B descriptors: in flight across the barrier
        if (more) P.fetch(L.lo + ep.batch, nS_next, 0);
        nS_cur = nS_next;
        typename T::Desc dB;
        L.fetch_descs(dB, L.gfirst);
        L.loss_partial(si, hreg + hover);
        L.phase_a_barrier();

        // ------------------------------ phase B ------------------------------------------
        L.phase_b(dB);
        L.arrive();  // waited for at the top of the next phase A
    }
    L.finish(n_steps);
}

struct ShardStage {
    size_t gU, gI, gb, total;
};
static ShardStage shard_stage_layout(int dim, int64_t B) {
    ShardStage L;
    size_t off = 0;
    auto take = [&](size_t n_floats) {
        size_t o = off;
        off += (n_floats * sizeof(float) + 255) / 256 * 256;
        return o;
    };
    L.gU = take((size_t)B * dim);
    L.gI = take((size_t)2 * B * dim);
    L.gb = take((size_t)2 * B);
    L.total = off;
    return L;
}

// Row shape of the sharded kernel: lanes per row group x 16-byte chunks per lane.  One chunk per lane where the row
// allows it (dim <= 128): only that shape leaves the shared memory for the cross-step prefetch of item rows.  (Two
// chunks per lane halve the per-row bookkeeping instructions; measured equal at one rank, trs_debug_shard_chunks_per_lane.)
static int g_shard_prefer_it = 1;
static unsigned long long* g_shard_trace = nullptr;
static int g_shard_overlap = -1;
static int g_shard_remote_hint = 1;
static int g_shard_one_pass = 1;
static int g_shard_last_one_pass = -1;

static bool pick_shard_shape(int dim, int* G, int* IT) {
    if (dim <= 0 || dim % 4 || dim > 512) return false;
    const int nch = dim / 4;
    int it = nch >= 8 ? g_shard_prefer_it : 1;
    int g = 4;
    while (g * it < nch && g < 32) g <<= 1;
    while (g * it < nch) it <<= 1;
    if (it == 3) it = 4;
    *G = g;
    *IT = it;
    return it <= 4;
}

int check_shard(const trs_shard* sh, RowShape* shape) {
    TRS_REQUIRE(sh != nullptr, "shard is NULL");
    TRS_REQUIRE(sh->world >= 1 && sh->world <= TRS_MAX_RANKS, "world %d outside 1..%d", sh->world, TRS_MAX_RANKS);
    TRS_REQUIRE(sh->rank >= 0 && sh->rank < sh->world, "rank %d outside the group of %d", sh->rank, sh->world);
    TRS_REQUIRE(sh->dim > 0 && sh->dim % 4 == 0 && pick_row_shape(sh->dim, shape),
                "row-sharded training needs n_factors to be a multiple of 4 up to 512 (got %d)", sh->dim);
    TRS_REQUIRE(sh->n_users > 0 && sh->n_users <= 0xFFFFFFFFll && sh->n_items > 0 && sh->n_items <= 0xFFFFFFFFll,
                "n_users / n_items out of range");
    return TRS_OK;
}

}  // namespace trs

using namespace trs;

extern "C" size_t trs_shard_stage_bytes(int dim, int global_batch) {
    if (dim <= 0 || global_batch <= 0) return 0;
    return 2 * shard_stage_layout(dim, global_batch).total;   // two copies, used by even / odd steps
}

extern "C" size_t trs_shard_plan_bytes(const trs_epoch* ep) {
    if (!ep || ep->batch <= 0) return 0;
    return shard_plan_layout(ep->n_samples, ep->batch).total;
}

extern "C" size_t trs_shard_plan_tmp_bytes(const trs_epoch* ep) {
    if (!ep || ep->batch <= 0) return 0;
    return shard_plan_tmp(ep).total;
}

extern "C" int trs_shard_plan_build(const trs_shard* sh, const trs_epoch* ep, void* plan, size_t plan_bytes,
                                    void* tmp, size_t tmp_bytes, trs_stream_t stream) {
    RowShape shape;
    int rc = check_shard(sh, &shape);
    if (rc) return rc;
    TRS_REQUIRE(ep && ep->user && ep->pos && ep->neg, "epoch ids are NULL");
    TRS_REQUIRE(ep->batch > 0 && ep->batch < (1 << 27), "global batch out of range (< 2^27)");
    TRS_REQUIRE(ep->pos_meta == nullptr && ep->neg_meta == nullptr, "row-sharded training does not take metadata");
    TRS_REQUIRE(plan && tmp, "plan / tmp is NULL");
    if (ep->n_samples == 0) return TRS_OK;
    TRS_REQUIRE(n_steps_of(ep) <= 65535, "shard_plan_build: %lld steps in one call (limit 65535)", (long long)n_steps_of(ep));
    const ShardPlanLayout L = shard_plan_layout(ep->n_samples, ep->batch);
    const ShardPlanTmp T = shard_plan_tmp(ep);
    if (plan_bytes < L.total || tmp_bytes < T.total) {
        set_error("shard plan workspace too small: plan %zu < %zu or tmp %zu < %zu", plan_bytes, L.total, tmp_bytes,
                  T.total);
        return TRS_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* P = (char*)plan;
    char* Tm = (char*)tmp;
    const int64_t n = ep->n_samples, steps = n_steps_of(ep);
    uint32_t* tkey = (uint32_t*)(Tm + T.tkey);
    uint32_t* tval = (uint32_t*)(Tm + T.tval);
    uint32_t* tile_cnt = (uint32_t*)(Tm + T.tile_cnt);
    uint32_t* hist = (uint32_t*)(Tm + T.hist);
    uint32_t* samp_cnt = (uint32_t*)(P + L.samp_cnt);
    uint32_t* own_cnt = (uint32_t*)(P + L.own_cnt);
    uint32_t* samp = (uint32_t*)(P + L.samp);
    const uint32_t W = (uint32_t)sh->world, r = (uint32_t)sh->rank;
    auto rows_of = [&](int64_t n_rows) { return (n_rows + W - 1) / W; };

    auto space = [&](const int64_t* a, const int64_t* b, int mult, int64_t n_rows, uint32_t* key, uint32_t* val,
                     int sp) -> int {
        const int tiles = (int)(((int64_t)mult * ep->batch + RT_TILE - 1) / RT_TILE);
        dim3 grid((unsigned)tiles, (unsigned)steps);
        // an odd number of radix passes ends in the other buffer: start there so the result lands in the plan
        const int npass = sort_passes(rows_of(n_rows));
        uint32_t* k0 = (npass & 1) ? tkey : key;
        uint32_t* v0 = (npass & 1) ? tval : val;
        uint32_t* k1 = (npass & 1) ? key : tkey;
        uint32_t* v1 = (npass & 1) ? val : tval;
        const RouteSel sel{a, b, mult, n, ep->batch, W, r, k0, v0, sp == 0 ? samp : nullptr, own_cnt + sp,
                           sp == 0 ? samp_cnt : nullptr};
        compact_count_kernel<<<grid, RT_THREADS, 0, st>>>(sel, tile_cnt, tiles);
        compact_scatter_kernel<<<grid, RT_THREADS, 0, st>>>(sel, tile_cnt, tiles);
        sort_pairs(k0, v0, k1, v1, mult, rows_of(n_rows), ep, own_cnt + sp, 2, hist, st);
        return TRS_OK;
    };
    space(ep->user, ep->user, 1, sh->n_users, (uint32_t*)(P + L.ukey), (uint32_t*)(P + L.uval), 0);
    space(ep->pos, ep->neg, 2, sh->n_items, (uint32_t*)(P + L.ikey), (uint32_t*)(P + L.ival), 1);
    {   // dirty flags of the rank's samples (see dirty_bitmap_kernel)
        bool exact;
        const int lb = dirty_log2_bits(ep, sh->n_items, &exact);
        uint32_t* bitmap = (uint32_t*)(Tm + T.bitmap);
        TRS_CUDA(cudaMemsetAsync(bitmap, 0, ((size_t)steps << lb) / 8, st));
        dim3 g2((unsigned)((2ll * ep->batch + RT_TILE - 1) / RT_TILE), (unsigned)steps);
        dirty_bitmap_kernel<<<g2, RT_THREADS, 0, st>>>(ep->pos, ep->neg, n, ep->batch, bitmap, lb, exact);
        dim3 g1((unsigned)(((int64_t)ep->batch + RT_TILE - 1) / RT_TILE), (unsigned)steps);
        dirty_mark_kernel<<<g1, RT_THREADS, 0, st>>>(ep->pos, ep->neg, n, ep->batch, bitmap, lb, exact, samp_cnt, samp);
        bool ex_unused;
        const int lbu = dirty_log2_bits(ep, (int64_t)1 << 40, &ex_unused);  // always hashed
        uint32_t* ubitmap = (uint32_t*)(Tm + T.ubitmap);
        TRS_CUDA(cudaMemsetAsync(ubitmap, 0, ((size_t)steps << lbu) / 8, st));
        single_mark_kernel<<<g1, RT_THREADS, 0, st>>>((const uint32_t*)(P + L.ukey), (uint32_t*)(P + L.uval), own_cnt, samp,
                                                     ep->batch, ubitmap, lbu);
        user_dirty_mark_kernel<<<g1, RT_THREADS, 0, st>>>(ep->user, ep->batch, W, ubitmap, lbu, samp_cnt, samp);
        user_compact_kernel<<<(unsigned)steps, 1024, 0, st>>>((uint32_t*)(P + L.ukey), (uint32_t*)(P + L.uval), own_cnt,
                                                             ep->batch);
    }
    if (W == 1) {  // after user_compact_kernel: cntB copies the final user counts
        const int tiles = (int)((2ll * ep->batch + RT_TILE - 1) / RT_TILE);
        const dim3 grid((unsigned)tiles, (unsigned)steps);
        const ItemMultiSel sel{(const uint32_t*)(P + L.ikey), (const uint32_t*)(P + L.ival), own_cnt, ep->batch,
                               (uint8_t*)(P + L.iflag), (uint32_t*)(P + L.ikeyB), (uint32_t*)(P + L.ivalB),
                               (uint32_t*)(P + L.cntB)};
        compact_count_kernel<<<grid, RT_THREADS, 0, st>>>(sel, tile_cnt, tiles);
        compact_scatter_kernel<<<grid, RT_THREADS, 0, st>>>(sel, tile_cnt, tiles);
    }
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

static int shard_cpr(int n_local) { return device_props().sm_count / (n_local > 0 ? n_local : 1); }

extern "C" size_t trs_shard_workspace_bytes(const trs_epoch* ep, int n_local) {
    if (!ep || ep->batch <= 0 || n_local < 1 || n_local > TRS_MAX_RANKS) return 0;
    const size_t ctx = ((size_t)n_local * sizeof(ShardCtx) + 255) / 256 * 256;
    const size_t part = ((size_t)n_local * n_steps_of(ep) * shard_cpr(n_local) * sizeof(float) + 255) / 256 * 256;
    return ctx + part;
}

extern "C" int trs_shard_train_steps(const trs_shard* shards, int n_local, const trs_epoch* ep, const trs_optim* optim,
                                     const void* const* plans_host, void* workspace, size_t workspace_bytes,
                                     int first_step, int n_steps, uint64_t sync_epoch, float* const* loss_sum_host,
                                     int32_t* status, int timeout_ms, trs_stream_t stream) {
    TRS_REQUIRE(shards && n_local >= 1 && n_local <= TRS_MAX_RANKS, "shard_train_steps: n_local out of range");
    TRS_REQUIRE(n_local == 1 || n_local == shards[0].world,
                "shard_train_steps: one launch hosts either one rank or the whole group");
    TRS_REQUIRE(ep && ep->user && ep->pos && ep->neg && ep->batch > 0, "epoch ids are NULL");
    TRS_REQUIRE(optim && optim->step_scale, "optimizer / step_scale is NULL");
    TRS_REQUIRE(optim->kind >= TRS_OPT_SGD && optim->kind <= TRS_OPT_SPARSE_ADAM, "unknown optimizer kind %d", optim->kind);
    TRS_REQUIRE(plans_host && workspace && loss_sum_host && status, "plans / workspace / loss / status is NULL");
    const int64_t steps = n_steps_of(ep);
    TRS_REQUIRE(first_step >= 0 && n_steps >= 0 && first_step + (int64_t)n_steps <= steps,
                "steps [%d, %d) outside the epoch's %lld steps", first_step, first_step + n_steps, (long long)steps);
    if (n_steps == 0) return TRS_OK;
    if (workspace_bytes < trs_shard_workspace_bytes(ep, n_local)) {
        set_error("shard workspace too small: %zu < %zu", workspace_bytes, trs_shard_workspace_bytes(ep, n_local));
        return TRS_ERR_WORKSPACE;
    }
    RowShape shape;
    const int cpr = shard_cpr(n_local);
    TRS_REQUIRE(cpr >= 1, "more local ranks than SMs");
    const ShardPlanLayout PL = shard_plan_layout(ep->n_samples, ep->batch);
    int sg = 0, sit = 0;
    const bool shape_ok = pick_shard_shape(shards[0].dim, &sg, &sit);
    // one rank in one launch: every item row's owner is the rank that reads it, so phase A updates the single ones
    const bool one = shape_ok && g_shard_one_pass && n_local == 1 && shards[0].world == 1 && sit == 1;
    const uint8_t* iflag = one ? (const uint8_t*)plans_host[0] + PL.iflag : nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    ShardCtx ctx[TRS_MAX_RANKS];
    const size_t ctx_bytes = ((size_t)n_local * sizeof(ShardCtx) + 255) / 256 * 256;
    float* loss_part = (float*)((char*)workspace + ctx_bytes);
    for (int i = 0; i < n_local; ++i) {
        const trs_shard& sh = shards[i];
        int rc = check_shard(&sh, &shape);
        if (rc) return rc;
        TRS_REQUIRE(sh.world == shards[0].world && sh.dim == shards[0].dim, "local ranks disagree on world / dim");
        const ShardStage SL = shard_stage_layout(sh.dim, ep->batch);
        ShardCtx& c = ctx[i];
        memset(&c, 0, sizeof(c));
        c.rank = sh.rank;
        c.world = sh.world;
        c.dim = sh.dim;
        c.stage_par = SL.total / sizeof(float);
        // on one GPU the barrier that ends a step costs about what the second pass does; across GPUs it is worth hiding
        c.overlap = (g_shard_overlap < 0 ? (sh.world > 1 ? 1 : 0) : g_shard_overlap) | (g_shard_remote_hint ? 2 : 0);
        for (int q = 0; q < sh.world; ++q) {
            TRS_REQUIRE(sh.user[q].emb && sh.item[q].emb && sh.stage[q] && sh.sync[q], "rank %d: peer %d is not mapped",
                        sh.rank, q);
            c.user[q] = sh.user[q];
            c.item[q] = sh.item[q];
            c.stage_u[q] = (float*)((char*)sh.stage[q] + SL.gU);
            c.stage_i[q] = (float*)((char*)sh.stage[q] + SL.gI);
            c.stage_b[q] = (float*)((char*)sh.stage[q] + SL.gb);
            c.sync[q] = (unsigned*)sh.sync[q];
        }
        const trs_table& mu = sh.user[sh.rank];
        const trs_table& mi = sh.item[sh.rank];
        if (optim->kind != TRS_OPT_SGD)
            TRS_REQUIRE(mu.emb_s0 && mi.emb_s0 && (!mi.lin || mi.lin_s0), "rank %d: optimizer state s0 is NULL", sh.rank);
        if (optim->kind == TRS_OPT_SPARSE_ADAM)
            TRS_REQUIRE(mu.emb_s1 && mi.emb_s1 && (!mi.lin || mi.lin_s1), "rank %d: optimizer state s1 is NULL", sh.rank);
        TRS_REQUIRE(plans_host[i] && loss_sum_host[i], "rank %d: plan / loss is NULL", sh.rank);
        const char* P = (const char*)plans_host[i];
        c.samp_cnt = (const uint32_t*)(P + PL.samp_cnt);
        c.own_cnt = (const uint32_t*)(P + PL.own_cnt);
        c.samp = (const uint32_t*)(P + PL.samp);
        c.ukey = (const uint32_t*)(P + PL.ukey);
        c.uval = (const uint32_t*)(P + PL.uval);
        c.ikey = (const uint32_t*)(P + (one ? PL.ikeyB : PL.ikey));
        c.ival = (const uint32_t*)(P + (one ? PL.ivalB : PL.ival));
        if (one) c.own_cnt = (const uint32_t*)(P + PL.cntB);
        c.loss_part = loss_part + (size_t)i * steps * cpr;
        c.loss_out = loss_sum_host[i];
        c.status = status;
        c.trace = g_shard_trace ? g_shard_trace + (size_t)i * n_steps * cpr * 8 : nullptr;
    }
    const ShardCtx* ctxs_dev = nullptr;
    if (n_local > 1) {  // emulation of a whole group on one GPU (tests): contexts travel through the workspace
        TRS_CUDA(cudaMemcpyAsync(workspace, ctx, (size_t)n_local * sizeof(ShardCtx), cudaMemcpyHostToDevice, st));
        ctxs_dev = (const ShardCtx*)workspace;
    }
    const OptScalars os = make_opt_scalars(optim);
    const unsigned long long timeout_ns = (unsigned long long)(timeout_ms > 0 ? timeout_ms : 20000) * 1000000ull;
    const unsigned se = (unsigned)sync_epoch;
    TRS_REQUIRE(shape_ok, "unsupported n_factors %d", shards[0].dim);
    // the two-phase kernel takes the first nine arguments, the one-pass kernel all ten
    void* args[] = {(void*)&ctx[0], (void*)&ctxs_dev, (void*)&cpr, (void*)ep, (void*)&os, (void*)&first_step,
                    (void*)&n_steps, (void*)&se, (void*)&timeout_ns, (void*)&iflag};
    const void* fn = nullptr;
    size_t smem = 0;
    int threads = 0;
    // one instantiation per (optimizer, row shape, kernel)
#define TRS_TWO_PHASE(K_, G_, IT_)                                                                                  \
    case ((K_ * 2 + 0) * 64 + G_) * 8 + IT_:                                                                        \
        fn = (const void*)shard_train_kernel<K_, G_, IT_>;                                                         \
        smem = shard_smem_total<G_, IT_>();                                                                         \
        threads = shard_threads<IT_>();                                                                             \
        break;
#define TRS_ONE_PASS(K_, G_)                                                                                        \
    case ((K_ * 2 + 1) * 64 + G_) * 8 + 1:                                                                          \
        fn = (const void*)shard_train_one_pass_kernel<K_, G_>;                                                     \
        smem = one_pass_smem_total();                                                                               \
        threads = shard_threads<1>();                                                                               \
        break;
#define TRS_SHARD_KERNELS(K_)                                                                                       \
    TRS_TWO_PHASE(K_, 4, 1) TRS_TWO_PHASE(K_, 8, 1) TRS_TWO_PHASE(K_, 16, 1) TRS_TWO_PHASE(K_, 32, 1)               \
    TRS_TWO_PHASE(K_, 4, 2) TRS_TWO_PHASE(K_, 8, 2) TRS_TWO_PHASE(K_, 16, 2) TRS_TWO_PHASE(K_, 32, 2)               \
    TRS_TWO_PHASE(K_, 32, 4)                                                                                        \
    TRS_ONE_PASS(K_, 4) TRS_ONE_PASS(K_, 8) TRS_ONE_PASS(K_, 16) TRS_ONE_PASS(K_, 32)
    switch (((os.kind * 2 + (one ? 1 : 0)) * 64 + sg) * 8 + sit) {
        TRS_SHARD_KERNELS(TRS_OPT_SGD)
        TRS_SHARD_KERNELS(TRS_OPT_ADAGRAD)
        TRS_SHARD_KERNELS(TRS_OPT_SPARSE_ADAM)
        default: break;
    }
#undef TRS_SHARD_KERNELS
#undef TRS_ONE_PASS
#undef TRS_TWO_PHASE
    TRS_REQUIRE(fn, "no sharded kernel for n_factors %d", shards[0].dim);
    TRS_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TRS_CUDA(cudaLaunchCooperativeKernel(fn, dim3(cpr * n_local), dim3(threads), args, smem, st));
    g_shard_last_one_pass = one ? 1 : 0;
    return TRS_OK;
}

// tuning hook (not part of trs.h): chunks per lane the sharded kernel prefers (1 or 2).  Results agree to rounding, not
// bit for bit: row_dot_partial sums a lane's IT chunks before group_sum<G> adds the lanes, so the dot products'
// association follows the row shape
extern "C" void trs_debug_shard_chunks_per_lane(int it) { g_shard_prefer_it = it == 1 ? 1 : 2; }
// debug hook: device buffer of n_local * n_steps * CTAs-per-rank * 8 uint64 that the next launches fill with phase
// time stamps (tools/shard_phases.py); NULL switches it off
extern "C" void trs_debug_shard_trace(void* buf) { g_shard_trace = (unsigned long long*)buf; }
// tuning hook (results do not depend on it): 1 / 0 forces the early first pass of phase A on / off, -1 = automatic
extern "C" void trs_debug_shard_overlap(int mode) { g_shard_overlap = mode < 0 ? -1 : (mode ? 1 : 0); }
// tuning hook: the evict_last policy on gradient rows stored into PEER memory (1, default) or only on local ones (0)
extern "C" void trs_debug_shard_remote_hint(int on) { g_shard_remote_hint = on ? 1 : 0; }
// tuning hook (results do not depend on it): 1 (default) lets a one-rank launch with one chunk per lane run the one-pass
// kernel, whose phase A also updates the item rows a step looks up once; 0 forces the two-phase kernel there
extern "C" void trs_debug_shard_one_pass(int on) { g_shard_one_pass = on ? 1 : 0; }
// debug hook: 1 if the last trs_shard_train_steps launch ran the one-pass kernel, 0 if the two-phase one, -1 before any
extern "C" int trs_debug_shard_last_one_pass(void) { return g_shard_last_one_pass; }


// ---- CUDA IPC plumbing ---------------------------------------------------------------------------------------
extern "C" int trs_ipc_export(const void* ptr, void* handle64_host, uint64_t* offset_host) {
    TRS_REQUIRE(ptr && handle64_host && offset_host, "ipc_export: NULL pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    typedef CUresult (*range_fn)(CUdeviceptr*, size_t*, CUdeviceptr);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    TRS_CUDA(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qres));
    TRS_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, "ipc_export: cuMemGetAddressRange is not available");
    CUdeviceptr base = 0;
    size_t size = 0;
    const CUresult cr = ((range_fn)fn)(&base, &size, (CUdeviceptr)ptr);
    TRS_REQUIRE(cr == CUDA_SUCCESS, "ipc_export: cuMemGetAddressRange failed (%d)", (int)cr);
    cudaIpcMemHandle_t h;
    TRS_CUDA(cudaIpcGetMemHandle(&h, (void*)base));
    memcpy(handle64_host, &h, sizeof(h));
    *offset_host = (uint64_t)((CUdeviceptr)ptr - base);
    return TRS_OK;
}

extern "C" int trs_ipc_open(const void* handle64_host, void** base_host) {
    TRS_REQUIRE(handle64_host && base_host, "ipc_open: NULL pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64_host, sizeof(h));
    TRS_CUDA(cudaIpcOpenMemHandle(base_host, h, cudaIpcMemLazyEnablePeerAccess));
    return TRS_OK;
}

extern "C" int trs_ipc_close(void* base) {
    TRS_REQUIRE(base, "ipc_close: NULL pointer");
    TRS_CUDA(cudaIpcCloseMemHandle(base));
    return TRS_OK;
}
