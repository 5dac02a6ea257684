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

// lookups of every tile that this rank owns
__global__ void __launch_bounds__(RT_THREADS)
route_count_kernel(const int64_t* __restrict__ a, const int64_t* __restrict__ b, int mult, int64_t n_samples, int B,
                   uint32_t world, uint32_t rank, uint32_t* __restrict__ tile_cnt, int tiles) {
    __shared__ uint32_t s_w[RT_THREADS / 32];
    const int64_t step = blockIdx.y;
    const int tile = blockIdx.x;
    const int Bs = (int)min((int64_t)B, n_samples - step * B);
    const int len = mult * Bs;
    const int64_t s0 = step * (int64_t)B;
    uint32_t cnt = 0;
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int j = tile * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (j < len) cnt += (route_id(a, b, s0, Bs, j) % world == rank) ? 1u : 0u;
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

// stable compaction of the owned lookups of a step: (local row, slot) pairs in slot order
__global__ void __launch_bounds__(RT_THREADS)
route_scatter_kernel(const int64_t* __restrict__ a, const int64_t* __restrict__ b, int mult, int64_t n_samples, int B,
                     uint32_t world, uint32_t rank, const uint32_t* __restrict__ tile_cnt, int tiles,
                     uint32_t* __restrict__ out_key, uint32_t* __restrict__ out_val, uint32_t* __restrict__ samp,
                     uint32_t* __restrict__ own_cnt, uint32_t* __restrict__ samp_cnt) {
    // user space (samp != NULL): the rank's samples ARE its owned user lookups in slot order, so the pair's value is
    // the sample's index in the rank's list (its slot is samp[index]); item space: the value is the slot itself
    __shared__ uint32_t s_w[RT_THREADS / 32];
    __shared__ uint32_t s_base;
    const int64_t step = blockIdx.y;
    const int tile = blockIdx.x;
    const int Bs = (int)min((int64_t)B, n_samples - step * B);
    const int len = mult * Bs;
    const int64_t s0 = step * (int64_t)B;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // pairs of the tiles before mine (tile 0 also publishes the step's total)
    {
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
        __shared__ uint32_t s_b[RT_THREADS / 32], s_t[RT_THREADS / 32];
        if (lane == 0) { s_b[warp] = before; s_t[warp] = total; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t bb = 0, tt = 0;
            for (int w = 0; w < RT_THREADS / 32; ++w) { bb += s_b[w]; tt += s_t[w]; }
            s_base = bb;
            if (tile == 0) {
                own_cnt[step * 2] = tt;
                if (samp_cnt) samp_cnt[step] = tt;
            }
        }
        __syncthreads();
    }
    uint32_t run = s_base;
    const int64_t seg = (int64_t)mult * step * B;
    for (int r = 0; r < RT_ROWS; ++r) {
        const int j = tile * RT_TILE + r * RT_THREADS + threadIdx.x;
        uint32_t id = 0;
        bool own = false;
        if (j < len) {
            id = route_id(a, b, s0, Bs, j);
            own = (id % world) == rank;
        }
        const uint32_t m = __ballot_sync(0xffffffffu, own);
        if (lane == 0) s_w[warp] = __popc(m);
        __syncthreads();
        uint32_t wbase = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < RT_THREADS / 32; ++w) {
            const uint32_t c = s_w[w];
            if (w < warp) wbase += c;
            tot += c;
        }
        if (own) {
            const uint32_t p = run + wbase + __popc(m & ((1u << lane) - 1u));
            out_key[seg + p] = id / world;
            out_val[seg + p] = samp ? p : (uint32_t)j;
            if (samp) samp[s0 + p] = (uint32_t)j;
        }
        run += tot;
        __syncthreads();
    }
}

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
        if ((k > 0 && K[k - 1] == key) || (k + 1 < n && K[k + 1] == key)) {
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
    __shared__ uint32_t s_run;
    const int64_t step = blockIdx.x;
    const int n = (int)own_cnt[2 * step];
    uint32_t* K = ukey + step * (int64_t)B;
    uint32_t* P = uval + step * (int64_t)B;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int k = base + (int)threadIdx.x;
        uint32_t key = 0, val = 0;
        bool keep = false;
        if (k < n) {
            key = K[k];
            val = P[k];
            keep = (val & (1u << 31)) == 0u;
        }
        const uint32_t m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_w[warp] = __popc(m);
        __syncthreads();
        uint32_t wbase = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < 32; ++w) {
            const uint32_t c = s_w[w];
            if (w < warp) wbase += c;
            tot += c;
        }
        const uint32_t run = s_run;
        __syncthreads();
        if (keep) {
            const uint32_t p = run + wbase + __popc(m & ((1u << lane) - 1u));
            K[p] = key;
            P[p] = val;
        }
        if (threadIdx.x == 0) s_run = run + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) own_cnt[2 * step] = s_run;
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
// updates it in phase A like a single user row.  Per step, item_single_count_kernel marks every item lookup slot single
// or not (iflag) and counts the other pairs per tile; item_single_scatter_kernel copies those pairs, whole runs in order,
// to ikeyB / ivalB: what phase B still does.  Grid (tiles of 2 B lookups, steps), as the route kernels.
__device__ __forceinline__ bool item_pair_multi(const uint32_t* K, int n, int k) {
    const uint32_t key = K[k];
    return (k > 0 && K[k - 1] == key) || (k + 1 < n && K[k + 1] == key);
}
__global__ void __launch_bounds__(RT_THREADS)
item_single_count_kernel(const uint32_t* __restrict__ ikey, const uint32_t* __restrict__ ival,
                         const uint32_t* __restrict__ own_cnt, int B, uint8_t* __restrict__ iflag,
                         uint32_t* __restrict__ tile_cnt, int tiles) {
    __shared__ uint32_t s_w[RT_THREADS / 32];
    const int64_t step = blockIdx.y;
    const int tile = blockIdx.x;
    const int n = (int)own_cnt[2 * step + 1];
    const int64_t seg = 2 * step * (int64_t)B;
    uint32_t cnt = 0;
#pragma unroll
    for (int r = 0; r < RT_ROWS; ++r) {
        const int k = tile * RT_TILE + r * RT_THREADS + threadIdx.x;
        if (k < n) {
            const bool m = item_pair_multi(ikey + seg, n, k);
            iflag[seg + ival[seg + k]] = m ? 0 : 1;
            cnt += m ? 1u : 0u;
        }
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
__global__ void __launch_bounds__(RT_THREADS)
item_single_scatter_kernel(const uint32_t* __restrict__ ikey, const uint32_t* __restrict__ ival,
                           const uint32_t* __restrict__ own_cnt, int B, const uint32_t* __restrict__ tile_cnt, int tiles,
                           uint32_t* __restrict__ ikeyB, uint32_t* __restrict__ ivalB, uint32_t* __restrict__ cntB) {
    __shared__ uint32_t s_w[RT_THREADS / 32], s_b[RT_THREADS / 32], s_t[RT_THREADS / 32];
    __shared__ uint32_t s_base;
    const int64_t step = blockIdx.y;
    const int tile = blockIdx.x;
    const int n = (int)own_cnt[2 * step + 1];
    const int64_t seg = 2 * step * (int64_t)B;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    {   // pairs kept by the tiles before mine (tile 0 also publishes the step's counts)
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
            if (tile == 0) {
                cntB[2 * step] = own_cnt[2 * step];
                cntB[2 * step + 1] = tt;
            }
        }
        __syncthreads();
    }
    uint32_t run = s_base;
    for (int r = 0; r < RT_ROWS; ++r) {
        const int k = tile * RT_TILE + r * RT_THREADS + threadIdx.x;
        const bool m = k < n && item_pair_multi(ikey + seg, n, k);
        const uint32_t bal = __ballot_sync(0xffffffffu, m);
        if (lane == 0) s_w[warp] = __popc(bal);
        __syncthreads();
        uint32_t wbase = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < RT_THREADS / 32; ++w) {
            const uint32_t c = s_w[w];
            if (w < warp) wbase += c;
            tot += c;
        }
        if (m) {
            const uint32_t p = run + wbase + __popc(bal & ((1u << lane) - 1u));
            ikeyB[seg + p] = ikey[seg + k];
            ivalB[seg + p] = ival[seg + k];
        }
        run += tot;
        __syncthreads();
    }
}

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
// the kernel
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

// one-pass kernel, per sample: bit 0 / 1 of fl the positive / negative item row is looked up once in the step, its
// local row, its slot (optimizer state in the next two) and its bias' optimizer state
struct OneItems {
    uint32_t fl, lp, ln;
    int sp, sn;
    float pl0, pl1, nl0, nl1;
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

// samples per row group whose item rows are fetched a step ahead (IT == 1 only: shared memory)
template <int G, int IT>
constexpr int shard_pf_samples() { return IT == 1 ? (G >= 8 ? 7 : 6) : 0; }  // what fits beside the 12 row slots in 227 KB
// The one-pass kernel (one rank, IT == 1) has no region: per row group ONE_S samples in flight, each with its three
// rows and their optimizer states in ONE_SLOTS thread-private slots.  Two in flight measured 41.30 us per step at the
// benchmark's shape against 41.54 us with three (one B200 at 1000 W, profiles/shard_r3.md)
constexpr int ONE_S = 2, ONE_SLOTS = 9;
template <int G, int IT, bool ONE>
constexpr size_t shard_smem_total() {
    constexpr size_t NT = shard_threads<IT>(), GPB = NT / G, PFS = shard_pf_samples<G, IT>();
    if (ONE) return NT * ONE_S * ONE_SLOTS * IT * 16;
    return shard_smem_bytes<IT>() + GPB * PFS * 2 * ((size_t)G * IT * 16 + 16) + GPB * 8;
}

template <int KIND, int G, int IT, bool ONE>
__global__ void __launch_bounds__((shard_threads<IT>()), 1)
shard_train_kernel(const __grid_constant__ ShardCtx ctx0, const ShardCtx* __restrict__ ctxs, const int cpr,
                   const __grid_constant__ trs_epoch ep, const __grid_constant__ OptScalars opt, const int first_step,
                   const int n_steps, const unsigned sync_epoch, const unsigned long long timeout_ns,
                   const uint8_t* __restrict__ iflag) {
    static_assert(!ONE || IT == 1, "the one-pass kernel takes one chunk per lane");
    constexpr int NT = shard_threads<IT>();
    constexpr int GPB = NT / G, GPW = 32 / G;
    constexpr int PB = shard_slots<IT>() / 4;  // owned rows in flight per row group (phase B): 4 slots each
    constexpr int DPL = (PB + G - 1) / G;      // row descriptors a lane fetches per phase-B round
    // Phase A rounds.  The item rows of a group's first PFS samples live in a per-group region of contiguous row
    // slots (filled a step ahead by bulk copies, or at the start of phase A for rows the previous step updated);
    // the 12 thread-private slots then hold the USER row with its optimizer state for SBA = 4 samples at a time:
    // regular rounds [0, SBA) and [SBA, PFS).  Samples beyond PFS (and every sample when there is no region, IT > 1)
    // go SBO = 2 per round with all five rows in the thread-private slots.
    // The loss adds a group's hinges in this layout's order whichever kernel runs: ordinals [0, HREG) one by one
    // (then a + 0 per unused regular slot), the later ordinals in a sum of their own.
    constexpr int HREG = shard_pf_samples<G, IT>();
    constexpr int PFS = ONE ? 0 : HREG;
    constexpr int SBA = 4, SBO = 2;
    constexpr int NREG = PFS ? 2 : 0;          // regular rounds
    constexpr int NPR = NREG ? NREG : 1;       // rounds whose records are fetched a step ahead
    constexpr int RPL = (SBA + G - 1) / G;     // sample records a lane holds per round
    constexpr int ROWB = G * IT * 16;          // bytes of a region row slot
    static_assert(shard_smem_total<G, IT, ONE>() + 2048 <= 227 * 1024, "shared memory budget");
    static_assert(!PFS || (PFS > SBA && PFS <= 2 * SBA), "round layout");
    __shared__ ShardCtx C;
    __shared__ float s_loss[NT / 32];
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float4* rows = reinterpret_cast<float4*>(smem_raw);  // [slot][IT][NT]
    unsigned char* pf_rows = smem_raw + shard_smem_bytes<IT>();             // [GPB][PFS][2][ROWB]
    unsigned char* pf_bias = pf_rows + (size_t)GPB * PFS * 2 * ROWB;       // [GPB][PFS][2][16]
    uint64_t* pf_bars = reinterpret_cast<uint64_t*>(pf_bias + (size_t)GPB * PFS * 2 * 16);  // [GPB]

    const int vr = blockIdx.x / cpr, c = blockIdx.x % cpr;
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(ctxs ? ctxs + vr : &ctx0);
        uint32_t* dst = reinterpret_cast<uint32_t*>(&C);
        for (int i = threadIdx.x; i < (int)(sizeof(ShardCtx) / 4); i += NT) dst[i] = src[i];
    }
    const int gl = threadIdx.x % G, g_in_cta = threadIdx.x / G;
    uint64_t* const my_bar = pf_bars + g_in_cta;
    unsigned char* const my_pf_rows = pf_rows + (size_t)g_in_cta * PFS * 2 * ROWB;
    unsigned char* const my_pf_bias = pf_bias + (size_t)g_in_cta * PFS * 2 * 16;
    if (PFS && gl == 0) mbar_init(my_bar, 1);
    if (PFS) fence_barrier_init();
    __syncthreads();
    const uint32_t W = (uint32_t)C.world;
    const bool wpow2 = (W & (W - 1u)) == 0u;
    const int wshift = __ffs((int)W) - 1;
    const int me = C.rank, dim = C.dim, nch = dim / 4;
    const int gfirst = c * GPB + g_in_cta, gstride = cpr * GPB;
    const int goff = g_in_cta % GPW;  // my group's position inside its warp: loops run on the warp's first group
    auto slot = [&](int j, int a) { return rows + ((j * IT + a) * NT + threadIdx.x); };
    auto slot_row = [&](int j) {
        Row<4, IT> x;
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            x.c[a] = Vec<4>::zero();
            if (gl + a * G < nch) x.c[a].v = *slot(j, a);
        }
        return x;
    };
    auto region_row = [&](int j) {  // region row j = 2 * sample ordinal + {0 positive, 1 negative} of my group
        Row<4, IT> x;
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            x.c[a] = Vec<4>::zero();
            if (gl + a * G < nch) x.c[a].v = *reinterpret_cast<const float4*>(my_pf_rows + (size_t)j * ROWB + (gl + a * G) * 16);
        }
        return x;
    };
    auto copy_row = [&](int j, const float* base) {
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int ch = gl + a * G;
            if (ch < nch) cp_async16(slot(j, a), base + (size_t)ch * 4);
        }
    };
    auto copy_region = [&](int j, const float* base) {
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int ch = gl + a * G;
            if (ch < nch) cp_async16(my_pf_rows + (size_t)j * ROWB + ch * 16, base + (size_t)ch * 4);
        }
    };
    auto ld_row = [&](const float* base) { return load_row_cg<4, G, IT>(base, nch, gl); };
    // L2 policies: a staged gradient row is written in phase A and read once in phase B of the same step -- it should
    // stay in L2 in between (evict_last) and leave right after (evict_first), while the table rows stream through.
    const uint64_t pol_keep = l2_policy_evict_last(), pol_drop = l2_policy_evict_first();
    auto copy_row_drop = [&](int j, const float* base) {  // a row nobody reads again: out of L2 first
#pragma unroll
        for (int a = 0; a < IT; ++a) {
            const int ch = gl + a * G;
            if (ch < nch) cp_async16_hint(slot(j, a), base + (size_t)ch * 4, pol_drop);
        }
    };
    const trs_table& tU = C.user[me];
    const trs_table& tI = C.item[me];
    const bool item_lin = tI.lin != nullptr;
    // the staging buffers exist twice (step parity): a rank may already store step s+1's gradient rows into a peer
    // that is still reading step s's
    unsigned bar_no = 0;   // cross-rank barriers arrived at in this launch
    bool wait_pending = false;  // arrived at the barrier that ends a step, not yet waited for it (see phase A)
    const bool overlap = (C.overlap & 1) != 0;
    const bool hint_remote = (C.overlap & 2) != 0;   // L2 policy also on stores into peer memory

    // ---- records of a phase-A round: lane gl fetches samples gl, gl + G, ... of the round and splits their ids
    //      into (owner, local row) ONCE (plan + epoch data: immutable, so the NEXT step's first rounds are fetched
    //      a whole step ahead).  b = position in the step | flags (SAMP_*); q packs the three owners ----
    struct Rec { uint32_t b[RPL], q[RPL], lu[RPL], lp[RPL], ln[RPL]; };
    auto split = [&](uint32_t id, uint32_t& owner, uint32_t& local) {
        if (wpow2) { owner = id & (W - 1u); local = id >> wshift; }
        else { owner = id % W; local = id / W; }
    };
    auto fetch_records = [&](Rec& R, int64_t lo_, int nS_, int kb, int cnt) {
        const uint32_t* samp = C.samp + lo_;
#pragma unroll
        for (int z = 0; z < RPL; ++z) {
            const int i = gl + z * G;
            const int k = kb + i * gstride;
            R.b[z] = 0xFFFFFFFFu;
            R.q[z] = R.lu[z] = R.lp[z] = R.ln[z] = 0u;
            if (i < cnt && k < nS_) {
                const uint32_t bf = __ldg(samp + k);
                const uint32_t b = bf & SAMP_POS;
                R.b[z] = bf;
                uint32_t qu, qp, qn;
                split((uint32_t)__ldg(ep.user + lo_ + b), qu, R.lu[z]);
                split((uint32_t)__ldg(ep.pos + lo_ + b), qp, R.lp[z]);
                split((uint32_t)__ldg(ep.neg + lo_ + b), qn, R.ln[z]);
                R.q[z] = qu | (qp << 4) | (qn << 8);
            }
        }
    };
    // one-pass kernel: lane gl holds the record of my group's ordinal blk * G + gl; one rank, so a local row is the id.
    // fl: bit 0 / 1 the positive / negative row is looked up once in the step (iflag at its lookup slot)
    struct Rec1 { uint32_t b, lu, lp, ln, fl; };
    auto fetch_one = [&](Rec1& R, int64_t lo_, int nS_, int blk) {
        const int k = gfirst + (blk * G + gl) * gstride;
        R.b = 0xFFFFFFFFu;
        R.lu = R.lp = R.ln = R.fl = 0u;
        if (k < nS_) {
            const int Bs_ = (int)min((int64_t)ep.batch, ep.n_samples - lo_);
            const uint32_t bf = __ldg(C.samp + lo_ + k);
            const uint32_t b = bf & SAMP_POS;
            R.b = bf;
            R.lu = (uint32_t)__ldg(ep.user + lo_ + b);
            R.lp = (uint32_t)__ldg(ep.pos + lo_ + b);
            R.ln = (uint32_t)__ldg(ep.neg + lo_ + b);
            R.fl = (uint32_t)__ldg(iflag + 2 * lo_ + b) | ((uint32_t)__ldg(iflag + 2 * lo_ + Bs_ + b) << 1);
        }
    };
    auto round_lo = [&](int r) { return r < NREG ? (r == 0 ? 0 : SBA) : PFS + SBO * (r - NREG); };
    auto round_n = [&](int r) { return r < NREG ? (r == 0 ? SBA : PFS - SBA) : SBO; };
    // ---- descriptors of a phase-B round: the owned lookups of a step are one list of positions, user space
    //      [0, nU) then item space [nU, nU + nI); lane gl fetches positions gl, gl + G, ... of the round ----
    // sf = slot | flags << 29; flag bits: 1 head (first position of a run of equal rows that phase A has not
    // updated already), 2 the run continues, 4 item space
    struct Desc { uint32_t key[DPL], sf[DPL]; };
    auto fetch_descs = [&](Desc& Dd, int64_t lo_, int nU_, int nI_, int pb, int pend) {
#pragma unroll
        for (int z = 0; z < DPL; ++z) {
            const int i = gl + z * G;
            const int p = pb + i * gstride;
            Dd.key[z] = Dd.sf[z] = 0u;
            if (i < PB && p < pend) {
                const bool it = p >= nU_;
                const int k = it ? p - nU_ : p, n = it ? nI_ : nU_;
                const uint32_t* K = it ? C.ikey + 2 * lo_ : C.ukey + lo_;
                const uint32_t* P = it ? C.ival + 2 * lo_ : C.uval + lo_;
                const uint32_t key = __ldg(K + k);
                const uint32_t prev = k > 0 ? __ldg(K + k - 1) : ~key;
                const uint32_t next = k + 1 < n ? __ldg(K + k + 1) : ~key;
                const uint32_t v = __ldg(P + k);
                const bool head = prev != key && !(v & VAL_DONE_IN_A);
                // item space: the value is the staging slot; user space: the sample's index in the rank's list
                const uint32_t sl = it ? v : (head ? (__ldg(C.samp + lo_ + (v & 0x1FFFFFFFu)) & SAMP_POS) : 0u);
                Dd.key[z] = key;
                Dd.sf[z] = (sl & 0x1FFFFFFFu) | ((head ? 1u : 0u) | (next == key ? 2u : 0u) | (it ? 4u : 0u)) << 29;
            }
        }
    };

    Rec recN[NPR];      // records of the next phase A's first NPR rounds
    Rec1 recO;          // one-pass kernel: the current block of records (block 0 of the next phase A between steps)
    int nS_cur = 0;
    {
        const int64_t lo0 = (int64_t)first_step * ep.batch;
        nS_cur = (int)C.samp_cnt[first_step];
        if constexpr (ONE) {
            fetch_one(recO, lo0, nS_cur, 0);
        } else {
#pragma unroll
            for (int r = 0; r < NPR; ++r) fetch_records(recN[r], lo0, nS_cur, gfirst + round_lo(r) * gstride, round_n(r));
        }
    }
    bool pf_live = false;     // the current step's region holds prefetched item rows (all but the dirty ones)
    uint32_t pf_parity = 0;

    for (int si = 0; si < n_steps; ++si) {
        const int64_t s = first_step + si;
        const int64_t lo = s * (int64_t)ep.batch;
        const int Bs = (int)min((int64_t)ep.batch, ep.n_samples - lo);
        const float invB = 1.0f / (float)Bs;
        const float scale = opt.step_scale[s];
        const int nS = nS_cur;
        const int nU = (int)C.own_cnt[2 * s], nI = (int)C.own_cnt[2 * s + 1];
        const bool more = si + 1 < n_steps;
        const int nS_next = more ? (int)C.samp_cnt[s + 1] : 0;
        const size_t po = (s & 1) ? C.stage_par : 0;
        float* const my_stage_u = C.stage_u[me] + po;
        float* const my_stage_i = C.stage_i[me] + po;
        const float* const my_stage_b = C.stage_b[me] + po;
        unsigned long long* tr = C.trace ? C.trace + ((size_t)si * cpr + c) * 8 : nullptr;
        if (tr && threadIdx.x == 0) tr[0] = global_ns();

        // ------------------------------ phase A ------------------------------------------
        {   // this step's phase-B lists (sorted keys and slots, streamed from HBM exactly once) -> L2 now: a round's
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
        // hinge terms: one per regular-round sample, added up in sample order afterwards (the order in which the two
        // passes visit them depends on plan flags, the loss must not), then the overflow rounds' in visiting order
        float hreg[2 * SBA], hover = 0.f;
#pragma unroll
        for (int i = 0; i < 2 * SBA; ++i) hreg[i] = 0.f;
        if (PFS && pf_live) {  // rows fetched while the previous step's owners were updating: landed?
            mbar_wait(my_bar, pf_parity);
            pf_parity ^= 1u;
        }
        // One sample: scores, hinge, gradient rows.  linear.py:78: s = <u, v> + b_u + b_i; loss.py:7-9:
        // h = s- - s+ + 1, d/ds = [h >= 0] / B.  A user row that this step looks up ONCE (plan flag: no other sample of
        // the global batch reads or writes it, and its owner is this rank) is updated right here from its state rows
        // in slots su_slot + 1 / + 2; every other gradient row goes to its owner's staging buffer.  The one-pass kernel
        // treats an item row that the step looks up once (oi.fl) the same way, from slots oi.sp / oi.sn + 1 / + 2.
        auto process = [&](bool valid, uint32_t bf, uint32_t q, uint32_t lu, const Row<4, IT>& xu, const Row<4, IT>& xp,
                           const Row<4, IT>& xn, float bu, float bip, float bin, int su_slot, float& hinge,
                           const OneItems& oi) {
            const float sp = (group_sum<G>(row_dot_partial(xu, xp)) + bu) + bip;
            const float sn = (group_sum<G>(row_dot_partial(xu, xn)) + bu) + bin;
            const float h = __fadd_rn(__fsub_rn(sn, sp), 1.0f);
            const float g = (h >= 0.f) ? invB : 0.f;
            if (!valid) return;
            hinge = fmaxf(h, 0.f);
            const uint32_t b = bf & SAMP_POS;
            const uint32_t qu = q & 15u, qp = (q >> 4) & 15u, qn = (q >> 8) & 15u;
            float* dp = C.stage_i[qp] + po + (size_t)b * dim;
            float* dn = C.stage_i[qn] + po + (size_t)(Bs + b) * dim;
            Row<4, IT> gu;
            if constexpr (ONE) {
                // the gradient rows exactly as phase B would read them back from the staging buffer (no contraction)
                Row<4, IT> gp, gn;
#pragma unroll
                for (int a = 0; a < IT; ++a)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        gu.c[a][e] = g * (xn.c[a][e] - xp.c[a][e]);
                        gp.c[a][e] = __fmul_rn(-g, xu.c[a][e]);
                        gn.c[a][e] = __fmul_rn(g, xu.c[a][e]);
                    }
                auto item_out = [&](bool single, uint32_t row, int sl, const Row<4, IT>& x, Row<4, IT>& gr, float* dst,
                                    float gb, float pl, float l0, float l1, uint32_t bslot) {
                    if (single) {
                        Row<4, IT> p = x, s0, s1;
                        row_zero(s0);
                        row_zero(s1);
                        if (KIND != TRS_OPT_SGD) s0 = slot_row(sl + 1);
                        if (KIND == TRS_OPT_SPARSE_ADAM) s1 = slot_row(sl + 2);
                        OptScalars ok = opt;
                        ok.kind = KIND;
                        update_store_row<4, G, IT>(tI, (size_t)row * dim, nch, gl, ok, scale, p, s0, s1, gr);
                        if (item_lin && gl == 0) update_store_lin(tI, row, ok, scale, gb, pl, l0, l1);
                    } else {
#pragma unroll
                        for (int a = 0; a < IT; ++a) {
                            const int ch = gl + a * G;
                            if (ch < nch) st_v4_hint(dst + (size_t)ch * 4, gr.c[a].v, pol_keep);
                        }
                        if (gl == 0) (C.stage_b[me] + po)[bslot] = gb;
                    }
                };
                item_out(oi.fl & 1u, oi.lp, oi.sp, xp, gp, dp, -g, bip, oi.pl0, oi.pl1, b);
                item_out(oi.fl & 2u, oi.ln, oi.sn, xn, gn, dn, g, bin, oi.nl0, oi.nl1, Bs + b);
            } else {
#pragma unroll
                for (int a = 0; a < IT; ++a) {
                    const int ch = gl + a * G;
#pragma unroll
                    for (int e = 0; e < 4; ++e) gu.c[a][e] = g * (xn.c[a][e] - xp.c[a][e]);
                    if (ch < nch) {
                        Vec<4> gp, gn;
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            gp[e] = -g * xu.c[a][e];
                            gn[e] = g * xu.c[a][e];
                        }
                        if (hint_remote || (int)qp == me) st_v4_hint(dp + (size_t)ch * 4, gp.v, pol_keep);
                        else gp.st(dp + (size_t)ch * 4);
                        if (hint_remote || (int)qn == me) st_v4_hint(dn + (size_t)ch * 4, gn.v, pol_keep);
                        else gn.st(dn + (size_t)ch * 4);
                    }
                }
                if (gl == 0) {
                    (C.stage_b[qp] + po)[b] = -g;
                    (C.stage_b[qn] + po)[Bs + b] = g;
                }
            }
            if (bf & SAMP_USER_SINGLE) {
                Row<4, IT> p = xu, s0, s1;
                row_zero(s0);
                row_zero(s1);
                if (KIND != TRS_OPT_SGD) s0 = slot_row(su_slot + 1);
                if (KIND == TRS_OPT_SPARSE_ADAM) s1 = slot_row(su_slot + 2);
                OptScalars ok = opt;
                ok.kind = KIND;  // compile-time optimizer: opt_update's branches fold
                update_store_row<4, G, IT>(C.user[qu], (size_t)lu * dim, nch, gl, ok, scale, p, s0, s1, gu);
            } else {
                float* du = C.stage_u[qu] + po + (size_t)b * dim;
#pragma unroll
                for (int a = 0; a < IT; ++a) {
                    const int ch = gl + a * G;
                    if (ch < nch) st_v4_hint(du + (size_t)ch * 4, gu.c[a].v, pol_keep);
                }
            }
        };
        const OneItems no_items{};
        if constexpr (ONE) {
            // One pass over my group's samples in ordinal order (the loss order), after the wait for the previous
            // step's end.  Sample o + ONE_S's rows start their trip (cp.async into slots ONE_SLOTS * j ..) before
            // sample o runs: user, positive, negative row at + 0 / 3 / 6, each followed by its optimizer state when
            // phase A updates that row.  Records come G samples at a time (Rec1); lane t & 3 holds scalar t of a
            // sample in tv0 (t < 4) or tv1: 0 user bias, 1 / 2 positive / negative bias, 3 / 4 and 5 / 6 their states.
            if (wait_pending) {
                if (tr && threadIdx.x == 0) tr[5] = global_ns();
                cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);
                wait_pending = false;
                if (tr && threadIdx.x == 0) tr[6] = global_ns();
            }
            const int kw = gfirst - goff;  // the warp's first group: the trip count is warp-uniform
            const int nord = kw < nS ? (nS - kw + gstride - 1) / gstride : 0;
            int blk = 0;
            uint32_t rb[ONE_S], ru[ONE_S], rp[ONE_S], rn[ONE_S], rf[ONE_S];
            float tv0[ONE_S], tv1[ONE_S];
            auto scalar = [&](int t, uint32_t lu, uint32_t lp, uint32_t ln, uint32_t fl) {
                const bool p = t == 1 || t == 3 || t == 4;
                const float* src = t == 0 ? tU.lin : (t <= 2 ? tI.lin : nullptr);
                if (t >= 3 && item_lin && (fl & (p ? 1u : 2u))) {
                    if ((t == 3 || t == 5) && KIND != TRS_OPT_SGD) src = tI.lin_s0;
                    if ((t == 4 || t == 6) && KIND == TRS_OPT_SPARSE_ADAM) src = tI.lin_s1;
                }
                return src ? __ldcg(src + (t == 0 ? lu : (p ? lp : ln))) : 0.f;
            };
            auto issue = [&](int o, int j) {
                uint32_t bf = 0xFFFFFFFFu, lu = 0u, lp = 0u, ln = 0u, fl = 0u;
                if (o < nord) {
                    if (o / G != blk) {
                        blk = o / G;
                        fetch_one(recO, lo, nS, blk);
                    }
                    bf = __shfl_sync(0xffffffffu, recO.b, o % G, G);
                    lu = __shfl_sync(0xffffffffu, recO.lu, o % G, G);
                    lp = __shfl_sync(0xffffffffu, recO.lp, o % G, G);
                    ln = __shfl_sync(0xffffffffu, recO.ln, o % G, G);
                    fl = __shfl_sync(0xffffffffu, recO.fl, o % G, G);
                }
                rb[j] = bf;
                ru[j] = lu;
                rp[j] = lp;
                rn[j] = ln;
                rf[j] = fl;
                tv0[j] = tv1[j] = 0.f;
                if (bf != 0xFFFFFFFFu) {
                    const int sl = j * ONE_SLOTS;
                    copy_row(sl + 0, tU.emb + (size_t)lu * dim);
                    if (bf & SAMP_USER_SINGLE) {
                        if (KIND != TRS_OPT_SGD) copy_row(sl + 1, tU.emb_s0 + (size_t)lu * dim);
                        if (KIND == TRS_OPT_SPARSE_ADAM) copy_row(sl + 2, tU.emb_s1 + (size_t)lu * dim);
                    }
                    copy_row(sl + 3, tI.emb + (size_t)lp * dim);
                    if (fl & 1u) {
                        if (KIND != TRS_OPT_SGD) copy_row(sl + 4, tI.emb_s0 + (size_t)lp * dim);
                        if (KIND == TRS_OPT_SPARSE_ADAM) copy_row(sl + 5, tI.emb_s1 + (size_t)lp * dim);
                    }
                    copy_row(sl + 6, tI.emb + (size_t)ln * dim);
                    if (fl & 2u) {
                        if (KIND != TRS_OPT_SGD) copy_row(sl + 7, tI.emb_s0 + (size_t)ln * dim);
                        if (KIND == TRS_OPT_SPARSE_ADAM) copy_row(sl + 8, tI.emb_s1 + (size_t)ln * dim);
                    }
                    if (gl < 4) {
                        tv0[j] = scalar(gl, lu, lp, ln, fl);
                        tv1[j] = scalar(gl + 4, lu, lp, ln, fl);
                    }
                }
                cp_async_commit();
            };
            auto run = [&](int o, int j) {
                const uint32_t bf = rb[j];
                const bool valid = bf != 0xFFFFFFFFu;
                const int sl = j * ONE_SLOTS;
                Row<4, IT> xu, xp, xn;
                if (valid) {
                    xu = slot_row(sl + 0);
                    xp = slot_row(sl + 3);
                    xn = slot_row(sl + 6);
                } else {
#pragma unroll
                    for (int a = 0; a < IT; ++a) xu.c[a] = xp.c[a] = xn.c[a] = Vec<4>::zero();
                }
                const float bu = __shfl_sync(0xffffffffu, tv0[j], 0, G);
                const float bip = __shfl_sync(0xffffffffu, tv0[j], 1, G);
                const float bin = __shfl_sync(0xffffffffu, tv0[j], 2, G);
                OneItems oi;
                oi.fl = rf[j];
                oi.lp = rp[j];
                oi.ln = rn[j];
                oi.sp = sl + 3;
                oi.sn = sl + 6;
                oi.pl0 = __shfl_sync(0xffffffffu, tv0[j], 3, G);
                oi.pl1 = __shfl_sync(0xffffffffu, tv1[j], 0, G);
                oi.nl0 = __shfl_sync(0xffffffffu, tv1[j], 1, G);
                oi.nl1 = __shfl_sync(0xffffffffu, tv1[j], 2, G);
                float hv = 0.f;
                process(valid, bf, 0u, ru[j], xu, xp, xn, bu, bip, bin, sl, hv, oi);
                if (valid) {
                    if (o < HREG) hreg[0] += hv; else hover += hv;
                }
            };
#pragma unroll
            for (int j = 0; j < ONE_S; ++j) issue(j, j);
            for (int o0 = 0; o0 < nord; o0 += ONE_S) {
#pragma unroll
                for (int j = 0; j < ONE_S; ++j) {
                    cp_async_wait(ONE_S - 1);
                    if (o0 + j < nord) run(o0 + j, j);
                    issue(o0 + j + ONE_S, j);
                }
            }
        } else {
            // Two passes over the regular rounds.  Pass 0 takes the samples none of whose three rows the previous
            // step's owners update (plan flags) BEFORE waiting for the barrier that ends the previous step: their rows
            // are final, and their gradient rows go to the other copy of the staging buffers.  Then the wait, then
            // pass 1 (the flagged samples) and the overflow rounds.
            for (int rr = 0;; ++rr) {
                if (wait_pending && (rr == NREG || !overlap)) {  // every warp of the CTA comes through here once per step
                    if (tr && threadIdx.x == 0) tr[5] = global_ns();
                    cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);
                    wait_pending = false;
                    if (tr && threadIdx.x == 0) tr[6] = global_ns();
                }
                const bool late = rr >= NREG;            // pass 1 / overflow
                const int rnd = late ? rr - NREG : rr;
                const int o_lo = round_lo(rnd), n_r = round_n(rnd);
                const int k0 = gfirst - goff + o_lo * gstride;
                if (k0 >= nS) {  // warp-uniform
                    if (late) break;
                    continue;
                }
                const int kb = k0 + goff;
                Rec cur;
                if (rnd < NPR) {
#pragma unroll
                    for (int r = 0; r < NPR; ++r)
                        if (r == rnd) cur = recN[r];
                } else {
                    fetch_records(cur, lo, nS, kb, n_r);
                }
                if (rnd < NREG) {
                    // ---- regular round: item rows in the region, user row + state in slots 3i .. 3i + 2 ----
                    if (late) {  // nothing flagged in the warp's groups: pass 0 did the whole round
                        if (!overlap) continue;
                        bool d = false;
#pragma unroll
                        for (int z = 0; z < RPL; ++z) d = d || (cur.b[z] != 0xFFFFFFFFu && (cur.b[z] & SAMP_DIRTY_ANY) != 0u);
                        if (!__any_sync(0xffffffffu, d)) continue;
                    }
                    float bias_r[SBA];  // lane t < 3 holds the width-1 companion of lookup t (user, positive, negative)
#pragma unroll
                    for (int i = 0; i < SBA; ++i) {
                        const uint32_t bf = __shfl_sync(0xffffffffu, cur.b[i / G], i % G, G);
                        const uint32_t q = __shfl_sync(0xffffffffu, cur.q[i / G], i % G, G);
                        const uint32_t lu = __shfl_sync(0xffffffffu, cur.lu[i / G], i % G, G);
                        const uint32_t lp = __shfl_sync(0xffffffffu, cur.lp[i / G], i % G, G);
                        const uint32_t ln = __shfl_sync(0xffffffffu, cur.ln[i / G], i % G, G);
                        bias_r[i] = 0.f;
                        if (i < n_r && bf != 0xFFFFFFFFu && (overlap ? ((bf & SAMP_DIRTY_ANY) != 0u) == late : !late)) {
                            const int ord = o_lo + i;
                            const bool have_p = pf_live && !(bf & SAMP_DIRTY_POS), have_n = pf_live && !(bf & SAMP_DIRTY_NEG);
                            const trs_table& TU = C.user[q & 15u];
                            const trs_table& TP = C.item[(q >> 4) & 15u];
                            const trs_table& TN = C.item[(q >> 8) & 15u];
                            copy_row(i * 3 + 0, TU.emb + (size_t)lu * dim);
                            if (bf & SAMP_USER_SINGLE) {
                                if (KIND != TRS_OPT_SGD) copy_row(i * 3 + 1, TU.emb_s0 + (size_t)lu * dim);
                                if (KIND == TRS_OPT_SPARSE_ADAM) copy_row(i * 3 + 2, TU.emb_s1 + (size_t)lu * dim);
                            }
                            if (!have_p) copy_region(ord * 2 + 0, TP.emb + (size_t)lp * dim);
                            if (!have_n) copy_region(ord * 2 + 1, TN.emb + (size_t)ln * dim);
                            if (gl < 3) {
                                const float* lin = gl == 0 ? TU.lin : (gl == 1 ? TP.lin : TN.lin);
                                const uint32_t lrow = gl == 0 ? lu : (gl == 1 ? lp : ln);
                                const bool have = gl == 1 ? have_p : (gl == 2 ? have_n : false);
                                if (lin) {
                                    if (have) bias_r[i] = reinterpret_cast<const float*>(
                                                  my_pf_bias + (size_t)(ord * 2 + (gl - 1)) * 16)[lrow & 3u];
                                    else bias_r[i] = __ldcg(lin + lrow);
                                }
                            }
                        }
                        cp_async_commit();
                    }
#pragma unroll
                    for (int i = 0; i < SBA; ++i) {
                        cp_async_wait(SBA - 1 - i);
                        const uint32_t bf = __shfl_sync(0xffffffffu, cur.b[i / G], i % G, G);
                        const uint32_t q = __shfl_sync(0xffffffffu, cur.q[i / G], i % G, G);
                        const uint32_t lu = __shfl_sync(0xffffffffu, cur.lu[i / G], i % G, G);
                        const bool valid = i < n_r && bf != 0xFFFFFFFFu &&
                                           (overlap ? ((bf & SAMP_DIRTY_ANY) != 0u) == late : !late);
                        Row<4, IT> xu, xp, xn;
                        if (valid) {
                            xu = slot_row(i * 3 + 0);
                            xp = region_row((o_lo + i) * 2 + 0);
                            xn = region_row((o_lo + i) * 2 + 1);
                        } else {
#pragma unroll
                            for (int a = 0; a < IT; ++a) xu.c[a] = xp.c[a] = xn.c[a] = Vec<4>::zero();
                        }
                        const float bu = __shfl_sync(0xffffffffu, bias_r[i], 0, G);
                        const float bip = __shfl_sync(0xffffffffu, bias_r[i], 1, G);
                        const float bin = __shfl_sync(0xffffffffu, bias_r[i], 2, G);
                        float hv = 0.f;
                        process(valid, bf, q, lu, xu, xp, xn, bu, bip, bin, i * 3, hv, no_items);
                        if (valid) {
                            if (rnd == 0) hreg[i] = hv; else hreg[SBA + i] = hv;
                        }
                    }
                } else {
                    // ---- overflow round: two samples, all five rows in the thread-private slots 5i .. 5i + 4 ----
                    float bias_r[SBO];
#pragma unroll
                    for (int i = 0; i < SBO; ++i) {
                        const uint32_t bf = __shfl_sync(0xffffffffu, cur.b[i / G], i % G, G);
                        const uint32_t q = __shfl_sync(0xffffffffu, cur.q[i / G], i % G, G);
                        const uint32_t lu = __shfl_sync(0xffffffffu, cur.lu[i / G], i % G, G);
                        const uint32_t lp = __shfl_sync(0xffffffffu, cur.lp[i / G], i % G, G);
                        const uint32_t ln = __shfl_sync(0xffffffffu, cur.ln[i / G], i % G, G);
                        bias_r[i] = 0.f;
                        if (bf != 0xFFFFFFFFu) {
                            const trs_table& TU = C.user[q & 15u];
                            const trs_table& TP = C.item[(q >> 4) & 15u];
                            const trs_table& TN = C.item[(q >> 8) & 15u];
                            copy_row(i * 5 + 0, TU.emb + (size_t)lu * dim);
                            if (bf & SAMP_USER_SINGLE) {
                                if (KIND != TRS_OPT_SGD) copy_row(i * 5 + 1, TU.emb_s0 + (size_t)lu * dim);
                                if (KIND == TRS_OPT_SPARSE_ADAM) copy_row(i * 5 + 2, TU.emb_s1 + (size_t)lu * dim);
                            }
                            copy_row(i * 5 + 3, TP.emb + (size_t)lp * dim);
                            copy_row(i * 5 + 4, TN.emb + (size_t)ln * dim);
                            if (gl < 3) {
                                const float* lin = gl == 0 ? TU.lin : (gl == 1 ? TP.lin : TN.lin);
                                const uint32_t lrow = gl == 0 ? lu : (gl == 1 ? lp : ln);
                                if (lin) bias_r[i] = __ldcg(lin + lrow);
                            }
                        }
                        cp_async_commit();
                    }
#pragma unroll
                    for (int i = 0; i < SBO; ++i) {
                        cp_async_wait(SBO - 1 - i);
                        const uint32_t bf = __shfl_sync(0xffffffffu, cur.b[i / G], i % G, G);
                        const uint32_t q = __shfl_sync(0xffffffffu, cur.q[i / G], i % G, G);
                        const uint32_t lu = __shfl_sync(0xffffffffu, cur.lu[i / G], i % G, G);
                        const bool valid = bf != 0xFFFFFFFFu;
                        Row<4, IT> xu, xp, xn;
                        if (valid) {
                            xu = slot_row(i * 5 + 0);
                            xp = slot_row(i * 5 + 3);
                            xn = slot_row(i * 5 + 4);
                        } else {
#pragma unroll
                            for (int a = 0; a < IT; ++a) xu.c[a] = xp.c[a] = xn.c[a] = Vec<4>::zero();
                        }
                        const float bu = __shfl_sync(0xffffffffu, bias_r[i], 0, G);
                        const float bip = __shfl_sync(0xffffffffu, bias_r[i], 1, G);
                        const float bin = __shfl_sync(0xffffffffu, bias_r[i], 2, G);
                        float hv = 0.f;
                        process(valid, bf, q, lu, xu, xp, xn, bu, bip, bin, i * 5, hv, no_items);
                        hover += hv;
                    }
                }
            }
        }
        // the next step's first rounds of records (plan + epoch data), then my first phase-B descriptors: all in
        // flight across the barrier
        if (more) {
            if constexpr (ONE) {
                fetch_one(recO, lo + ep.batch, nS_next, 0);
            } else {
#pragma unroll
                for (int r = 0; r < NPR; ++r)
                    fetch_records(recN[r], lo + ep.batch, nS_next, gfirst + round_lo(r) * gstride, round_n(r));
            }
        }
        nS_cur = nS_next;
        const int nP = nU + nI;
        Desc dB;
        fetch_descs(dB, lo, nU, nI, gfirst, nP);

        float hsum = 0.f;
#pragma unroll
        for (int i = 0; i < 2 * SBA; ++i) hsum += hreg[i];
        hsum = warp_sum(gl == 0 ? hsum + hover : 0.f);
        if ((threadIdx.x & 31) == 0) s_loss[threadIdx.x >> 5] = hsum;
        __syncthreads();
        if (threadIdx.x == 0) {
            float H = 0.f;
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) H += s_loss[w];
            C.loss_part[(size_t)si * cpr + c] = H;
            if (tr) tr[1] = global_ns();
        }
        ++bar_no;
        cross_arrive(C, true);
        cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);
        if (tr && threadIdx.x == 0) tr[2] = global_ns();

        // ------------------------------ phase B ------------------------------------------
        // First the NEXT step's item rows: every clean one (not updated by this step, plan flag) of my group's first
        // PFS samples starts its trip -- from the owner's HBM, mostly over NVLink -- into the region and lands while
        // the owners update (bulk async copies, one mbarrier per row group).  The lane that holds a sample's record
        // issues its copies.
        pf_live = false;
        if (PFS && more) {
#pragma unroll
            for (int r = 0; r < NREG; ++r) {
#pragma unroll
                for (int z = 0; z < RPL; ++z) {
                    const int i = gl + z * G;
                    const uint32_t bf = recN[r].b[z];
                    if (i < round_n(r) && bf != 0xFFFFFFFFu) {
                        const uint32_t q = recN[r].q[z];
                        const trs_table& TP = C.item[(q >> 4) & 15u];
                        const trs_table& TN = C.item[(q >> 8) & 15u];
                        const bool fp = !(bf & SAMP_DIRTY_POS), fn = !(bf & SAMP_DIRTY_NEG);
                        const uint32_t per = (uint32_t)dim * 4u + (TP.lin ? 16u : 0u);
                        const uint32_t bytes = (fp ? per : 0u) + (fn ? per : 0u);
                        if (bytes) mbar_expect_tx(my_bar, bytes);
                        const int j = (round_lo(r) + i) * 2;
                        if (fp) {
                            bulk_g2s(my_pf_rows + (size_t)j * ROWB, TP.emb + (size_t)recN[r].lp[z] * dim, (uint32_t)dim * 4u, my_bar);
                            if (TP.lin) bulk_g2s(my_pf_bias + (size_t)j * 16, TP.lin + (recN[r].lp[z] & ~3u), 16u, my_bar);
                        }
                        if (fn) {
                            bulk_g2s(my_pf_rows + (size_t)(j + 1) * ROWB, TN.emb + (size_t)recN[r].ln[z] * dim, (uint32_t)dim * 4u, my_bar);
                            if (TN.lin) bulk_g2s(my_pf_bias + (size_t)(j + 1) * 16, TN.lin + (recN[r].ln[z] & ~3u), 16u, my_bar);
                        }
                    }
                }
            }
            __syncwarp();  // every expect_tx of the group precedes its one arrival
            if (gl == 0) mbar_arrive(my_bar);
            pf_live = true;
        }
        // Owned rows: a row group takes PB positions of the step's sorted list per round; only the first position of
        // a run of equal rows works (it sums the run's staged rows in slot order); rows phase A updated are skipped.
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
                    copy_row_drop(i * 4 + 0, (it ? my_stage_i : my_stage_u) + (size_t)sl * dim);
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
            if (p0 + gstride * PB < nP) fetch_descs(dB, lo, nU, nI, pb + gstride * PB, nP);
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
                const trs_table& t = it ? tI : tU;
                Row<4, IT> g = slot_row(i * 4 + 0), p = slot_row(i * 4 + 1), s0, s1;
                row_zero(s0);
                row_zero(s1);
                if (KIND != TRS_OPT_SGD) s0 = slot_row(i * 4 + 2);
                if (KIND == TRS_OPT_SPARSE_ADAM) s1 = slot_row(i * 4 + 3);
                if (sf & (1u << 30)) {  // duplicates (rare under uniform ids): the rest of the run, in slot order
                    const int pos = pb + i * gstride;
                    const int k = it ? pos - nU : pos, n = it ? nI : nU;
                    const uint32_t* K = it ? C.ikey + 2 * lo : C.ukey + lo;
                    const uint32_t* P = it ? C.ival + 2 * lo : C.uval + lo;
                    const float* stage = it ? my_stage_i : my_stage_u;
                    for (int q = k + 1; q < n && __ldg(K + q) == key; ++q) {
                        const uint32_t v = __ldg(P + q) & 0x1FFFFFFFu;
                        const uint32_t j = it ? v : (__ldg(C.samp + lo + v) & SAMP_POS);
                        row_acc(g, ld_row(stage + (size_t)j * dim));
                        if (it && item_lin && gl == 0) gb = __fadd_rn(gb, __ldcg(my_stage_b + j));
                    }
                }
                OptScalars ok = opt;
                ok.kind = KIND;
                update_store_row<4, G, IT>(t, (size_t)key * dim, nch, gl, ok, scale, p, s0, s1, g);
                if (it && item_lin && gl == 0) update_store_lin(t, key, ok, scale, gb, pl, l0, l1);
            }
        }
        if (tr) {
            __syncthreads();
            if (threadIdx.x == 0) tr[3] = global_ns();
        }
        // the owners' updates are done: arrive, and wait inside the next step's phase A (after its pass 0)
        ++bar_no;
        cross_arrive(C, false);
        wait_pending = true;
        if (tr && threadIdx.x == 0) tr[4] = global_ns();
    }
    if (wait_pending) cross_wait(C, sync_epoch + bar_no, (unsigned)cpr, timeout_ns);

    // per-step hinge sums of this rank, CTAs added in a fixed order
    if (c == 0) {
        for (int si = threadIdx.x; si < n_steps; si += NT) {
            float H = 0.f;
            for (int q = 0; q < cpr; ++q) H += __ldcg(C.loss_part + (size_t)si * cpr + q);
            C.loss_out[si] = H;
        }
    }
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

template <int KIND, int G, int IT, bool ONE>
static cudaError_t launch_shard_k(const ShardCtx* ctx0, const ShardCtx* ctxs, int cpr, int n_local, const trs_epoch* ep,
                                  const OptScalars* os, int first_step, int n_steps, unsigned sync_epoch,
                                  unsigned long long timeout_ns, const uint8_t* iflag, cudaStream_t stream) {
    const void* fn = (const void*)shard_train_kernel<KIND, G, IT, ONE>;
    const size_t smem = shard_smem_total<G, IT, ONE>();
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    void* args[] = {(void*)ctx0, (void*)&ctxs, (void*)&cpr, (void*)ep, (void*)os, (void*)&first_step,
                    (void*)&n_steps, (void*)&sync_epoch, (void*)&timeout_ns, (void*)&iflag};
    return cudaLaunchCooperativeKernel(fn, dim3(cpr * n_local), dim3(shard_threads<IT>()), args, smem, stream);
}
template <int KIND, int G, int IT>
static cudaError_t launch_shard_o(bool one, const ShardCtx* ctx0, const ShardCtx* ctxs, int cpr, int n_local,
                                  const trs_epoch* ep, const OptScalars* os, int first_step, int n_steps,
                                  unsigned sync_epoch, unsigned long long timeout_ns, const uint8_t* iflag,
                                  cudaStream_t stream) {
    if constexpr (IT == 1) {
        if (one)
            return launch_shard_k<KIND, G, IT, true>(ctx0, ctxs, cpr, n_local, ep, os, first_step, n_steps, sync_epoch,
                                                     timeout_ns, iflag, stream);
    }
    return launch_shard_k<KIND, G, IT, false>(ctx0, ctxs, cpr, n_local, ep, os, first_step, n_steps, sync_epoch,
                                              timeout_ns, iflag, stream);
}
template <int G, int IT>
static cudaError_t launch_shard(bool one, const ShardCtx* ctx0, const ShardCtx* ctxs, int cpr, int n_local,
                                const trs_epoch* ep, const OptScalars* os, int first_step, int n_steps,
                                unsigned sync_epoch, unsigned long long timeout_ns, const uint8_t* iflag,
                                cudaStream_t stream) {
    switch (os->kind) {
        case TRS_OPT_SGD:
            return launch_shard_o<TRS_OPT_SGD, G, IT>(one, ctx0, ctxs, cpr, n_local, ep, os, first_step, n_steps, sync_epoch, timeout_ns, iflag, stream);
        case TRS_OPT_ADAGRAD:
            return launch_shard_o<TRS_OPT_ADAGRAD, G, IT>(one, ctx0, ctxs, cpr, n_local, ep, os, first_step, n_steps, sync_epoch, timeout_ns, iflag, stream);
        default:
            return launch_shard_o<TRS_OPT_SPARSE_ADAM, G, IT>(one, ctx0, ctxs, cpr, n_local, ep, os, first_step, n_steps, sync_epoch, timeout_ns, iflag, stream);
    }
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
        route_count_kernel<<<grid, RT_THREADS, 0, st>>>(a, b, mult, n, ep->batch, W, r, tile_cnt, tiles);
        // an odd number of radix passes ends in the other buffer: start there so the result lands in the plan
        const int npass = sort_passes(rows_of(n_rows));
        uint32_t* k0 = (npass & 1) ? tkey : key;
        uint32_t* v0 = (npass & 1) ? tval : val;
        uint32_t* k1 = (npass & 1) ? key : tkey;
        uint32_t* v1 = (npass & 1) ? val : tval;
        route_scatter_kernel<<<grid, RT_THREADS, 0, st>>>(a, b, mult, n, ep->batch, W, r, tile_cnt, tiles, k0, v0,
                                                         sp == 0 ? samp : nullptr, own_cnt + sp,
                                                         sp == 0 ? samp_cnt : nullptr);
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
        const uint32_t* ikey = (const uint32_t*)(P + L.ikey);
        const uint32_t* ival = (const uint32_t*)(P + L.ival);
        item_single_count_kernel<<<grid, RT_THREADS, 0, st>>>(ikey, ival, own_cnt, ep->batch, (uint8_t*)(P + L.iflag),
                                                              tile_cnt, tiles);
        item_single_scatter_kernel<<<grid, RT_THREADS, 0, st>>>(ikey, ival, own_cnt, ep->batch, tile_cnt, tiles,
                                                                (uint32_t*)(P + L.ikeyB), (uint32_t*)(P + L.ivalB),
                                                                (uint32_t*)(P + L.cntB));
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
    cudaError_t err = cudaErrorInvalidValue;
    TRS_REQUIRE(shape_ok, "unsupported n_factors %d", shards[0].dim);
#define TRS_SHARD_CASE(G_, IT_)                                                                                     \
    case G_ * 100 + IT_:                                                                                            \
        err = launch_shard<G_, IT_>(one, &ctx[0], ctxs_dev, cpr, n_local, ep, &os, first_step, n_steps,              \
                                    (unsigned)sync_epoch, timeout_ns, iflag, st);                                   \
        break;
    switch (sg * 100 + sit) {
        TRS_SHARD_CASE(4, 1)
        TRS_SHARD_CASE(8, 1)
        TRS_SHARD_CASE(16, 1)
        TRS_SHARD_CASE(32, 1)
        TRS_SHARD_CASE(4, 2)
        TRS_SHARD_CASE(8, 2)
        TRS_SHARD_CASE(16, 2)
        TRS_SHARD_CASE(32, 2)
        TRS_SHARD_CASE(32, 4)
        default: break;
    }
#undef TRS_SHARD_CASE
    TRS_CUDA(err);
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
