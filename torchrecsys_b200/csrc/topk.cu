// topk.cu -- batched predict (reference model.py:341-452: score one user against every item, sort, keep
// top_k) as a user-tile x all-items score GEMM on the tcgen05 tensor cores with the top-k selection fused
// into the epilogue, followed by an exact fp32 re-scoring of the surviving candidates.
//
// Why two phases: the reference ranks fp32 scores; tensor cores multiply bf16.  Phase 1 therefore only
// has to produce, per user, a SUPERSET of the exact top-k:
//   |s_bf16(u,i) - s_exact(u,i)| <= eps_u := 2^-7 (1+2^-9) * |u| * max_i |w_i| + 2^-8 * max_i |c_i|
//   (bf16 unit roundoff 2^-8 on both factors of every product u_d w_id, Cauchy-Schwarz over d; the constant 1
//   that multiplies c_i is exact, so the extra column only contributes the rounding of c_i itself)
//   so every exact top-k item has s_bf16 >= tau_k - 2 eps_u, tau_k = the k-th best bf16 score seen.
// Phase 2 recomputes the candidates' scores with the same fp32 code path as trs_scores and ranks them by
// (score descending, item id ascending) == torch.sort(stable=True, descending=True) on the reference's
// scores, so the returned indices are those of the fp32 path, tie-break "lower item id first".
//
// Phase 1 operands (prepared once per call):  Ub[q,:] = bf16([u_q, 1, 0..]),  Vb[i,:] = bf16([w_i, c_i, 0..])
//   Linear: w_i = item_i + sum_f meta_f(i)   c_i = item_bias_i                      (linear.py:64-78)
//   FM    : w_i = item_i + sum_f meta_f(i)   c_i = lin_item_i + sum_f lin_meta_f(i)
//                                                  + 1/2 sum_d [w_id^2 - item_id^2 - sum_f meta_f(i)_d^2]
//           so that z(u,i) = lin_user_u + <[u,1],[w_i,c_i]> is the FM logit (fm.py:81-97) and the score is
//           sigmoid(z), monotone in z.
// Kernel: CTA = 128 users (A tile resident in shared memory) x a range of 128-item tiles streamed by TMA
// through a ring; accumulators double-buffered in TMEM (2 x 128 columns) so the tensor core computes tile
// t+1 while the four epilogue warps filter tile t: thread = user row, one compare per score against the
// row's running threshold, survivors appended to the row's candidate list in global memory.  When a list
// nears its capacity the warp compacts its 32 rows (warp-parallel k-th-largest by bisection on the float
// bit pattern) and raises the thresholds.
#include <stdio.h>
#include <stdlib.h>

#include "scorer.cuh"
#include "tc.cuh"

namespace trs {

typedef __nv_bfloat16 bf16;
// Item tile = 192 rows: one tcgen05.mma (128 x 192 x 16) runs 96 cycles, so the ~300 cycles the issuing warp
// needs per tile for barriers and descriptors cost a quarter less than at 128, and two accumulators (2 x 192
// columns) plus the user tile (<= 120 columns) still fit the 512 columns of tensor memory.
constexpr int TK_BM = 128, TK_BN = 192, TK_CAP = 512, TK_THREADS = 192, TK_BOX_BYTES = TK_BN * 128;
constexpr int TK_SYNC_EVERY = 64, TK_SYNC_WINDOW = 768;  // tiles; 768 tiles of 192 x 288 B = 42 MB of the 126 MB L2
constexpr int TK_HALF = 2;  // 32-column chunks the epilogue holds in registers at a time
constexpr int TK_BATCHES = TK_BN / (32 * TK_HALF);
constexpr int TK_TMEM_COLS = 512;  // 2 x 192 accumulator columns + the user tile (Kp / 2 <= 120 columns)
constexpr int TK_MAX_SPLITS = 8;
constexpr int TK_MAX_STAGE2 = 4096;  // candidates one user may bring to phase 2 (>= TK_MAX_SPLITS * TK_CAP)

struct TopkDev {
    int n_query, n_items, nbox, kslices, stages, Kp;
    const bf16* Ub;       // [user_tiles * TK_BM, Kp] bf16([u, 1, 0..])
    int n_item_tiles, tiles_per_split, splits;
    int k, fm;
    const float* unorm;   // [n_query] |u|
    const float* ulin;    // [n_query] lin_user (FM) or 0
    const float* vmax2;   // [2] max_i |w_i|^2, max_i |c_i|
    float* cand_s;        // [n_query, splits, TK_CAP]
    int* cand_i;
    int* cand_cnt;        // [n_query, splits]
    int* overflow;        // [n_query]
    int sync_window;      // tiles a producer may run ahead of the slowest active CTA of its range
    int* progress;        // [splits, user_tiles] producer position of every CTA (-1 not started, INT_MAX finished)
    int trace_t0;
    long long* trace;     // debug (TRS_TOPK_TRACE): [TK_TRACE_TILES][8] clock64 stamps of CTA (0, 0), else null
};
constexpr int TK_TRACE_TILES = 1024;  // traced tiles: [trace_t0, trace_t0 + TILES)

__device__ __forceinline__ float key_float(uint32_t k) {  // inverse of float_key (common.cuh)
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// warp-cooperative compaction of one row's candidate list; returns the new count, sets thr
constexpr int TK_PER = TK_CAP / 32;  // list entries per lane
struct RowList {
    float e[TK_PER];
    int id[TK_PER];
};
__device__ __forceinline__ void load_list(const float* __restrict__ cs, const int* __restrict__ ci, int n, int lane,
                                          RowList& L) {
#pragma unroll
    for (int i = 0; i < TK_PER; ++i) {
        const int slot = i * 32 + lane;
        L.e[i] = slot < n ? cs[slot] : -INFINITY;
        L.id[i] = slot < n ? ci[slot] : 0;
    }
}
__device__ __forceinline__ int compact_row(float* __restrict__ cs, int* __restrict__ ci, const RowList& L, int n, int k,
                                           float margin2, float ulin, int fm, int lane, float& thr_out) {
    constexpr int PER = TK_PER;
    const float (&e)[TK_PER] = L.e;
    const int (&id)[TK_PER] = L.id;
    float keep = -INFINITY;
    if (n >= k) {
        // A lower bound of the k-th largest key, by bisection between the row's smallest and largest key down to
        // 1/256 of their spread (every candidate already passed the previous threshold, so the spread is small):
        // invariant #{key >= lo} >= k.  Stopping early only keeps a candidate or two more than the exact
        // k-th-largest would -- ~9 rounds instead of 32.
        uint32_t key[PER];
        uint32_t kmin = 0xffffffffu, kmax = 0u;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const bool in = i * 32 + lane < n;
            key[i] = in ? float_key(e[i]) : 0u;
            if (in) {
                kmin = min(kmin, key[i]);
                kmax = max(kmax, key[i]);
            }
        }
        uint32_t lo = __reduce_min_sync(0xffffffffu, kmin), hi = __reduce_max_sync(0xffffffffu, kmax);
        const uint32_t stop = (hi - lo) >> 8;
        while (hi - lo > stop) {
            const uint32_t mid = lo + ((hi - lo) >> 1) + 1u;  // upper middle: lo < mid <= hi
            int c = 0;
#pragma unroll
            for (int i = 0; i < PER; ++i) c += (key[i] >= mid) ? 1 : 0;
            c = __reduce_add_sync(0xffffffffu, c);
            if (c >= k) lo = mid;
            else hi = mid - 1u;
        }
        const float tau = key_float(lo);
        float margin = margin2;
        if (fm) {
            // distinct logits whose fp32 sigmoids coincide are ties the final ranking breaks by item id:
            // widen by the logit interval one ulp of sigmoid(tau) spans (inf once the sigmoid saturates)
            const float s = 1.0f / (1.0f + expf(-(tau + ulin)));
            const float d = s * (1.0f - s);
            margin += (d > 1e-30f) ? 1.2e-7f * fmaxf(s, 1e-30f) / d : INFINITY;
        }
        keep = tau - margin;
    }
    __syncwarp();
    int base = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const bool p = (i * 32 + lane < n) && (e[i] >= keep);
        const unsigned bal = __ballot_sync(0xffffffffu, p);
        if (p) {
            const int pos = base + __popc(bal & ((1u << lane) - 1u));
            cs[pos] = e[i];
            ci[pos] = id[i];
        }
        base += __popc(bal);
    }
    __syncwarp();
    thr_out = keep;
    return base;
}

__global__ void __launch_bounds__(TK_THREADS, 1)
topk_score_kernel(const __grid_constant__ CUtensorMap tmap_v,
                  const __grid_constant__ TopkDev g) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* sB = base;
    uint64_t* bars = (uint64_t*)(sB + g.stages * g.nbox * TK_BOX_BYTES);
    uint64_t* full = bars + 1;
    uint64_t* empty = full + g.stages;
    uint64_t* acc_full = empty + g.stages;   // [2]
    uint64_t* acc_empty = acc_full + 2;       // [2]
    uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int u0 = blockIdx.x * TK_BM;
    const int split = blockIdx.y;
    const int tile0 = split * g.tiles_per_split;
    const int ntiles = min(g.tiles_per_split, g.n_item_tiles - tile0);
    const bool tracing = g.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0;
    __shared__ int s_compact_req;  // last tile (+1) at which an epilogue warp asked for a list compaction
    if (threadIdx.x == 0) s_compact_req = 0;

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmap_v);
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], 4);  // one arrival per epilogue warp
        }
        fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, TK_TMEM_COLS);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    // The user tile is the A operand of every MMA of this CTA: it goes into tensor memory once (row = lane, two
    // bf16 per column), so the tensor core streams only the item tiles from shared memory.
    const uint32_t tmem_a = tmem + 2 * TK_BN;
    if (warp >= 2) {
        const int q = warp & 3;
        const uint32_t* urow = reinterpret_cast<const uint32_t*>(g.Ub + (size_t)(u0 + q * 32 + lane) * g.Kp);
        for (int c = 0; c < g.Kp / 2; c += 8) {
            uint32_t r[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = __ldg(urow + c + j);
            tc::tmem_st_32x8(tmem_a + ((uint32_t)(q * 32) << 16) + (uint32_t)c, r);
        }
        tc::tmem_st_wait();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();

    if (warp == 0) {
        // Producer.  Every CTA of an item range streams the same tiles: as long as they stay within an L2's reach
        // of each other one DRAM read serves them all, but a CTA that falls behind (list compactions are
        // data-dependent) re-reads everything from DRAM at 1/148 of the bandwidth and falls further behind.  So
        // the ranges run in loose lock-step: each producer publishes its position every TK_SYNC_EVERY tiles and
        // waits while an active CTA of its range is between TK_SYNC_WINDOW and 4x that many tiles behind it.
        // (Further behind = a CTA of a later wave: not waited for.  Only CTAs AHEAD ever wait, the last active
        // one never does, so there is no cycle.)
        int* prog = g.progress + (size_t)split * gridDim.x;
        int s = 0;
        uint32_t ph = 0;  // ring slot and its phase parity, advanced without divisions
        for (int t = 0; t < ntiles; ++t, ++s) {
            if (s == g.stages) { s = 0; ph ^= 1u; }
            if ((t & (TK_SYNC_EVERY - 1)) == 0) {
                if (lane == 0) *(volatile int*)(prog + blockIdx.x) = t;
                for (;;) {
                    int behind = 0;
                    for (int p = lane; p < (int)gridDim.x; p += 32) {
                        const int v = *(volatile const int*)(prog + p);
                        behind |= (v >= 0 && v < t - g.sync_window && v > t - 4 * g.sync_window) ? 1 : 0;
                    }
                    if (!__any_sync(0xffffffffu, behind)) break;
                    __nanosleep(500);
                }
            }
            mbar_wait(&empty[s], ph ^ 1u);
            if (tracing && lane == 0 && t >= g.trace_t0 && t < g.trace_t0 + TK_TRACE_TILES) g.trace[(t - g.trace_t0) * 8 + 0] = clock64();
            if (tc::elect_one()) {
                mbar_arrive_expect_tx(&full[s], g.nbox * TK_BOX_BYTES);
                for (int b = 0; b < g.nbox; ++b)
                    tc::tma_load_2d(sB + (s * g.nbox + b) * TK_BOX_BYTES, &tmap_v, &full[s], b * 64, (tile0 + t) * TK_BN);
            }
            __syncwarp();
        }
        if (lane == 0) *(volatile int*)(prog + blockIdx.x) = 0x7fffffff;  // finished: nobody waits for me
    } else if (warp == 1) {
        // the whole warp walks the tiles (uniform control flow), one elected lane issues the MMAs
        constexpr uint32_t idesc = tc::idesc_bf16_f32(TK_BM, TK_BN);
        int s = 0;
        uint32_t ph = 0;
        for (int t = 0; t < ntiles; ++t, ++s) {
            if (s == g.stages) { s = 0; ph ^= 1u; }
            const int buf = t & 1;
            const uint32_t bph = (uint32_t)(t >> 1) & 1u;
            mbar_wait(&acc_empty[buf], bph ^ 1u);
            if (tracing && lane == 0 && t >= g.trace_t0 && t < g.trace_t0 + TK_TRACE_TILES) g.trace[(t - g.trace_t0) * 8 + 1] = clock64();
            mbar_wait(&full[s], ph);
            if (tracing && lane == 0 && t >= g.trace_t0 && t < g.trace_t0 + TK_TRACE_TILES) g.trace[(t - g.trace_t0) * 8 + 2] = clock64();
            tc::tc_fence_after();
            if (tc::elect_one()) {
                for (int ks = 0; ks < g.kslices; ++ks) {
                    const int box = ks >> 2, kin = (ks & 3) * 16;
                    const uint64_t db = tc::smem_desc_sw128(sB + (s * g.nbox + box) * TK_BOX_BYTES, kin);
                    tc::umma_bf16_ts(tmem + (uint32_t)(buf * TK_BN), tmem_a + (uint32_t)(ks * 8), db, idesc, ks ? 1u : 0u);
                }
                tc::umma_commit(&empty[s]);
                tc::umma_commit(&acc_full[buf]);
            }
            __syncwarp();
            if (tracing && lane == 0 && (t & 255) == 0 && (t >> 8) < 1024) g.trace[TK_TRACE_TILES * 8 + (t >> 8)] = clock64();
            if (tracing && lane == 0 && t >= g.trace_t0 && t < g.trace_t0 + TK_TRACE_TILES) g.trace[(t - g.trace_t0) * 8 + 3] = clock64();
        }
    } else {
        const int q = warp & 3;
        const int row = u0 + q * 32 + lane;
        const bool valid = row < g.n_query;
        const size_t lst = ((size_t)(valid ? row : 0) * g.splits + split) * TK_CAP;
        float* cs = g.cand_s + lst;
        int* ci = g.cand_i + lst;
        const float wmax = sqrtf(__ldg(g.vmax2)), cmax = __ldg(g.vmax2 + 1);
        // 2 eps_u, with 0.4 % of slack for the fp32 accumulation and the fp32 evaluation of c_i
        const float margin2 = valid ? 1.004f * (0.015625f * __ldg(g.unorm + row) * wmax + 0.0078125f * cmax) : 0.f;
        const float ulin = valid ? __ldg(g.ulin + row) : 0.f;
        int cnt = 0, joined = 0;
        float thr = -INFINITY;
        bool over = false;
        for (int t = 0; t < ntiles; ++t) {
            const int buf = t & 1;
            const uint32_t bph = (uint32_t)(t >> 1) & 1u;
            mbar_wait(&acc_full[buf], bph);
            const bool etr = tracing && warp == 2 && lane == 0 && t >= g.trace_t0 && t < g.trace_t0 + TK_TRACE_TILES;
            if (etr) g.trace[(t - g.trace_t0) * 8 + 4] = clock64();
            tc::tc_fence_after();
            const int item0 = (tile0 + t) * TK_BN;
            const int ncols = min(TK_BN, g.n_items - item0);
            // the row's 32-column chunks are fetched in batches (one TMEM round trip each; 64 registers), the buffer
            // is handed back to the MMA warp after the last, and the filtering runs from registers.  The batch
            // loop is NOT unrolled: the filter's rarely taken append path is ~250 instructions per chunk, and the
            // MMA-issuing warp shares the instruction cache with this code.
#pragma unroll 1
            for (int half = 0; half < TK_BATCHES; ++half) {
                uint32_t r[TK_HALF][32];
#pragma unroll
                for (int c = 0; c < TK_HALF; ++c)
                    tc::tmem_ld_32x32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * TK_BN + (half * TK_HALF + c) * 32), r[c]);
                tc::tmem_ld_wait();
                if (half == TK_BATCHES - 1) {
                    tc::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[buf]);
                    if (etr) g.trace[(t - g.trace_t0) * 8 + 5] = clock64();
                }
                if (valid && !over) {
#pragma unroll
                    for (int c = 0; c < TK_HALF; ++c) {
                        // steady state: about k/n of the scores pass, so first ask whether ANY of the 32 does
                        // (branch-free max tree, independent pairs), and only then walk the chunk
                        float m16[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) m16[j] = fmaxf(__uint_as_float(r[c][j]), __uint_as_float(r[c][j + 16]));
#pragma unroll
                        for (int w = 8; w >= 4; w >>= 1)
#pragma unroll
                            for (int j = 0; j < w; ++j) m16[j] = fmaxf(m16[j], m16[j + w]);
                        // m16[jj], jj < 4: the maximum of the 8 columns jj, jj + 4, ..., jj + 28
                        if (fmaxf(fmaxf(m16[0], m16[1]), fmaxf(m16[2], m16[3])) >= thr) {
                            const int col0 = (half * TK_HALF + c) * 32;
                            const int lim = ncols - col0;  // columns of this chunk that are real items
#pragma unroll
                            for (int jj = 0; jj < 4; ++jj) {
                                if (m16[jj] < thr) continue;  // while the threshold still rises most of a chunk fails
#pragma unroll
                                for (int i = 0; i < 8; ++i) {
                                    const int j = jj + 4 * i;
                                    const float v = __uint_as_float(r[c][j]);
                                    if (v >= thr && j < lim) {
                                        if (cnt < TK_CAP) {
                                            cs[cnt] = v;
                                            ci[cnt] = item0 + col0 + j;
                                        }
                                        ++cnt;
                                    }
                                }
                            }
                        }
                    }
                }
            }
            if (etr) g.trace[(t - g.trace_t0) * 8 + 6] = clock64() + (cnt & 0);
            // a list that could overflow on the next tile -> the warp compacts all of its rows; after the
            // last tile every list is compacted once more, so phase 2 only sees scores >= tau_k - margin
            // The four epilogue warps compact TOGETHER: a compaction stalls the whole pipeline (the MMA warp
            // needs all four to release an accumulator), so four events at different tiles cost four stalls.
            // The warp that must compact posts the tile number; the others join at their next tile.
            const bool trig = __any_sync(0xffffffffu, cnt > TK_CAP - TK_BN || (t == ntiles - 1 && cnt > g.k));
            if (etr) g.trace[(t - g.trace_t0) * 8 + 7] = clock64();
            if (trig && lane == 0) atomicMax(&s_compact_req, t + 1);
            __syncwarp();
            const int req = *(volatile int*)&s_compact_req;
            if (trig || req > joined) {
                joined = max(req, t + 1);
                __syncwarp();
                const long long c_t0 = tracing ? clock64() : 0;
                int c_rows = 0;
                // only the rows that are filling up (every row with more than k entries after the last tile): the
                // others keep their threshold.  The next row's list is fetched while the current one is compacted.
                const bool need = valid && !over && cnt > (t == ntiles - 1 ? g.k : TK_CAP / 2);
                unsigned todo = __ballot_sync(0xffffffffu, need);
                RowList cur, nxt;
                auto list_of = [&](int rr) { return ((size_t)(u0 + q * 32 + rr) * g.splits + split) * TK_CAP; };
                if (todo) {
                    const int rr = __ffs(todo) - 1;
                    load_list(g.cand_s + list_of(rr), g.cand_i + list_of(rr), min(__shfl_sync(0xffffffffu, cnt, rr), TK_CAP), lane, cur);
                }
                while (todo) {
                    const int rr = __ffs(todo) - 1;
                    todo &= todo - 1;
                    if (todo) {
                        const int r2 = __ffs(todo) - 1;
                        load_list(g.cand_s + list_of(r2), g.cand_i + list_of(r2), min(__shfl_sync(0xffffffffu, cnt, r2), TK_CAP), lane, nxt);
                    }
                    ++c_rows;
                    const int n_r = __shfl_sync(0xffffffffu, cnt, rr);
                    const float m_r = __shfl_sync(0xffffffffu, margin2, rr);
                    const float ul_r = __shfl_sync(0xffffffffu, ulin, rr);
                    float thr_r;
                    const int new_n = compact_row(g.cand_s + list_of(rr), g.cand_i + list_of(rr), cur, min(n_r, TK_CAP), g.k, m_r,
                                                  ul_r, g.fm, lane, thr_r);
                    if (lane == rr) {
                        if (n_r > TK_CAP || new_n > TK_CAP - TK_BN) {
                            // the margin admits more candidates than a list holds: this user takes the
                            // exact fp32 path on the host side (trs_scores + sort)
                            over = true;
                            g.overflow[row] = 1;
                        }
                        cnt = over ? 0 : new_n;
                        thr = thr_r;
                    }
                    cur = nxt;
                }
                if (tracing && lane == 0 && (t >> 8) < 1024) {
                    atomicAdd((unsigned long long*)&g.trace[TK_TRACE_TILES * 8 + 1024 + (t >> 8)], (unsigned long long)c_rows);
                    atomicAdd((unsigned long long*)&g.trace[TK_TRACE_TILES * 8 + 2048 + (t >> 8)], (unsigned long long)(clock64() - c_t0));
                }
            }
        }
        if (valid) g.cand_cnt[(size_t)row * g.splits + split] = over ? 0 : min(cnt, TK_CAP);
        if (valid && cnt > TK_CAP) g.overflow[row] = 1;
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, TK_TMEM_COLS);
    }
}

// ---- operand preparation ------------------------------------------------------------------------------
// one warp per item: Vb[i] = bf16([w_i, c_i, 0...]) and max |[w_i, c_i]|^2.  VEC: n_factors % 4 == 0 -- every lane
// moves four consecutive factors per access (16-byte loads, 8-byte bf16 stores).
template <bool VEC>
__global__ void __launch_bounds__(256)
topk_prep_items_kernel(const __grid_constant__ trs_model m, const int64_t* __restrict__ item_meta, int64_t n_items,
                       int Kp, bf16* __restrict__ Vb, unsigned* __restrict__ vmax2_bits) {
    const int lane = threadIdx.x & 31;
    const int D = m.dim, F = m.n_meta;
    constexpr int W = VEC ? 4 : 1;
    float wmax = 0.f, cmax = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); i < n_items; i += (int64_t)gridDim.x * 8) {
        float c = m.item.lin ? m.item.lin[i] : 0.f;
        float half = 0.f, n2 = 0.f;
        bf16* out = Vb + (size_t)i * Kp;
        for (int d = lane * W; d < D; d += 32 * W) {
            float w[W], q[W];
            if (VEC) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(m.item.emb + (size_t)i * D + d));
                w[0] = v.x; w[W > 1 ? 1 : 0] = v.y; w[W > 2 ? 2 : 0] = v.z; w[W > 3 ? 3 : 0] = v.w;
            } else {
                w[0] = m.item.emb[(size_t)i * D + d];
            }
#pragma unroll
            for (int x = 0; x < W; ++x) q[x] = w[x] * w[x];
            for (int f = 0; f < F; ++f) {
                const float* mrow = m.meta[f].emb + (size_t)item_meta[i * F + f] * D + d;
                float e[W];
                if (VEC) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(mrow));
                    e[0] = v.x; e[W > 1 ? 1 : 0] = v.y; e[W > 2 ? 2 : 0] = v.z; e[W > 3 ? 3 : 0] = v.w;
                } else {
                    e[0] = mrow[0];
                }
#pragma unroll
                for (int x = 0; x < W; ++x) {
                    w[x] += e[x];
                    q[x] = fmaf(e[x], e[x], q[x]);
                }
            }
#pragma unroll
            for (int x = 0; x < W; ++x) {
                half += w[x] * w[x] - q[x];
                n2 = fmaf(w[x], w[x], n2);
            }
            if (VEC) {
                const __nv_bfloat162 lo = __floats2bfloat162_rn(w[0], w[W > 1 ? 1 : 0]);
                const __nv_bfloat162 hi = __floats2bfloat162_rn(w[W > 2 ? 2 : 0], w[W > 3 ? 3 : 0]);
                uint2 pk;
                pk.x = *reinterpret_cast<const uint32_t*>(&lo);
                pk.y = *reinterpret_cast<const uint32_t*>(&hi);
                *reinterpret_cast<uint2*>(out + d) = pk;
            } else {
                out[d] = __float2bfloat16_rn(w[0]);
            }
        }
        half = warp_sum(half);
        n2 = warp_sum(n2);
        if (m.net == TRS_NET_FM) {
            for (int f = 0; f < F; ++f)
                if (m.meta[f].lin) c += m.meta[f].lin[item_meta[i * F + f]];
            c += 0.5f * half;
        }
        // the extra K column and the zero padding up to Kp
        for (int d = D + lane; d < Kp; d += 32) out[d] = __float2bfloat16_rn(d == D ? c : 0.f);
        wmax = fmaxf(wmax, n2);
        cmax = fmaxf(cmax, fabsf(c));
    }
    if (lane == 0) {  // non-negative floats order like their bits
        atomicMax(vmax2_bits, __float_as_uint(wmax));
        atomicMax(vmax2_bits + 1, __float_as_uint(cmax));
    }
}

// one warp per query user: Ub[q] = bf16([u, 1, 0...]), |[u,1]|, lin_user
__global__ void __launch_bounds__(256)
topk_prep_users_kernel(const __grid_constant__ trs_model m, const int64_t* __restrict__ users, int n_query, int Kp,
                       bf16* __restrict__ Ub, float* __restrict__ unorm, float* __restrict__ ulin) {
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (q >= n_query) return;
    const int D = m.dim;
    const int64_t u = users[q];
    float n2 = 0.f;
    for (int d = lane; d < Kp; d += 32) {
        float v = d < D ? m.user.emb[(size_t)u * D + d] : (d == D ? 1.0f : 0.f);
        if (d < D) n2 = fmaf(v, v, n2);
        Ub[(size_t)q * Kp + d] = __float2bfloat16_rn(v);
    }
    n2 = warp_sum(n2);
    if (lane == 0) {
        unorm[q] = sqrtf(n2);
        ulin[q] = (m.net == TRS_NET_FM && m.user.lin) ? m.user.lin[u] : 0.f;
    }
}

// ---- phase 2: exact fp32 scores of the candidates, rank, write the top k ------------------------------------
template <int NET, int V, int G, int IT>
__global__ void __launch_bounds__(128)
topk_rescore_kernel(const __grid_constant__ trs_model m, const int64_t* __restrict__ users,
                    const int64_t* __restrict__ item_meta, const __grid_constant__ TopkDev g, int64_t item_offset,
                    int64_t* __restrict__ out_idx, float* __restrict__ out_score) {
    __shared__ float s_score[TK_MAX_STAGE2];
    __shared__ int s_idx[TK_MAX_STAGE2];
    __shared__ int s_n;
    const int q = blockIdx.x;
    const int64_t u = users[q];
    // gather the split lists (thread 0 computes the offsets; lists are short)
    if (threadIdx.x == 0) {
        int n = 0;
        for (int sp = 0; sp < g.splits; ++sp) n += g.cand_cnt[(size_t)q * g.splits + sp];
        if (n > TK_MAX_STAGE2) {
            g.overflow[q] = 1;
            n = 0;
        }
        if (g.overflow[q]) n = 0;
        s_n = n;
    }
    __syncthreads();
    const int n = s_n;
    if (n > 0) {
        int off = 0;
        for (int sp = 0; sp < g.splits; ++sp) {
            const int c = g.cand_cnt[(size_t)q * g.splits + sp];
            const int* src = g.cand_i + ((size_t)q * g.splits + sp) * TK_CAP;
            for (int j = threadIdx.x; j < c; j += 128) s_idx[off + j] = src[j];
            off += c;
        }
    }
    __syncthreads();
    // exact scores: one row group per candidate, warp-uniform trip count
    const int nch = m.dim / V, gl = threadIdx.x % G;
    constexpr int GPB = 128 / G, GPW = 32 / G;
    const int sub = (threadIdx.x / G) % GPW;
    for (int j0 = threadIdx.x / G - sub; j0 < n; j0 += GPB) {
        const bool ok = j0 + sub < n;
        const int j = ok ? j0 + sub : n - 1;
        const int64_t it = s_idx[j];
        const float s = score_one<NET, V, G, IT>(m, nch, gl, u, it, item_meta ? item_meta + it * m.n_meta : nullptr);
        if (gl == 0 && ok) s_score[j] = s;
    }
    __syncthreads();
    // rank by (score desc, item id asc): a strict total order, so ranks are distinct
    for (int j = threadIdx.x; j < n; j += 128) {
        const float s = s_score[j];
        const int id = s_idx[j];
        int rank = 0;
        for (int o = 0; o < n; ++o) {
            const float so = s_score[o];
            rank += (so > s || (so == s && s_idx[o] < id)) ? 1 : 0;
        }
        if (rank < g.k) {
            out_idx[(size_t)q * g.k + rank] = (int64_t)id + item_offset;
            out_score[(size_t)q * g.k + rank] = s;
        }
    }
    for (int r = n + threadIdx.x; r < g.k; r += 128) {  // fewer candidates than k (n_items < k) or overflow
        out_idx[(size_t)q * g.k + r] = -1;
        out_score[(size_t)q * g.k + r] = -INFINITY;
    }
}

template <int V, int G, int IT>
static void launch_rescore(const trs_model* m, const int64_t* users, const int64_t* item_meta, const TopkDev* g,
                           int64_t item_offset, int64_t* out_idx, float* out_score, cudaStream_t st) {
    if (m->net == TRS_NET_LINEAR)
        topk_rescore_kernel<TRS_NET_LINEAR, V, G, IT><<<g->n_query, 128, 0, st>>>(*m, users, item_meta, *g, item_offset,
                                                                                 out_idx, out_score);
    else
        topk_rescore_kernel<TRS_NET_FM, V, G, IT><<<g->n_query, 128, 0, st>>>(*m, users, item_meta, *g, item_offset,
                                                                             out_idx, out_score);
}

struct TopkLayout {
    int Kp, nbox, kslices, stages, n_item_tiles, user_tiles, splits, tiles_per_split;
    size_t Ub, Vb, unorm, ulin, vmax2, cand_s, cand_i, cand_cnt, overflow, progress, total;
    size_t smem;
};
static TopkLayout topk_layout(const trs_model* m, int64_t n_query) {
    TopkLayout L = {};
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += (bytes + 255) / 256 * 256;
        return o;
    };
    L.Kp = (m->dim + 1 + 15) / 16 * 16;
    L.kslices = L.Kp / 16;
    L.nbox = (L.Kp + 63) / 64;
    L.stages = L.nbox <= 3 ? 3 : 2;
    L.n_item_tiles = (int)((m->item.n_rows + TK_BN - 1) / TK_BN);
    L.user_tiles = (int)((n_query + TK_BM - 1) / TK_BM);
    // few users: cut the catalogue into up to TK_MAX_SPLITS item ranges so more SMs work; each range keeps
    // its own candidate list (<= TK_CAP - TK_BN entries after the final compaction), and a range needs
    // enough tiles for the running threshold to bite
    // (one CTA per SM and no more: every item range pays its own threshold warm-up -- the first ~2000 tiles of a
    // range run at a third of the steady-state rate -- so a second wave of ranges costs more than it balances)
    int want = (device_props().sm_count + L.user_tiles - 1) / L.user_tiles;
    if (want > TK_MAX_SPLITS) want = TK_MAX_SPLITS;
    if (want > L.n_item_tiles / 16) want = L.n_item_tiles / 16;
    L.splits = want < 1 ? 1 : want;
    L.tiles_per_split = (L.n_item_tiles + L.splits - 1) / L.splits;
    L.splits = (L.n_item_tiles + L.tiles_per_split - 1) / L.tiles_per_split;
    L.Ub = take((size_t)L.user_tiles * TK_BM * L.Kp * 2);
    L.Vb = take((size_t)m->item.n_rows * L.Kp * 2);
    L.unorm = take((size_t)n_query * 4);
    L.ulin = take((size_t)n_query * 4);
    L.vmax2 = take(256);
    L.cand_s = take((size_t)n_query * L.splits * TK_CAP * 4);
    L.cand_i = take((size_t)n_query * L.splits * TK_CAP * 4);
    L.cand_cnt = take((size_t)n_query * L.splits * 4);
    L.overflow = take((size_t)n_query * 4);
    L.progress = take((size_t)L.splits * L.user_tiles * 4);
    L.total = off;
    L.smem = 1024 + (size_t)L.stages * L.nbox * TK_BOX_BYTES + 8 * (2 * L.stages + 5) + 16;
    return L;
}

static int check_topk(const trs_model* m, int64_t n_query, int k) {
    RowShape shape;
    int rc = check_model(m, &shape);
    if (rc) return rc;
    TRS_REQUIRE(m->net != TRS_NET_MLP, "predict_topk: the MLP tower has no user x item factorisation; score with trs_mlp_forward");
    TRS_REQUIRE(m->dim <= 239, "predict_topk: n_factors up to 239 (got %d)", m->dim);
    TRS_REQUIRE(k >= 1 && k <= TK_CAP / 4, "predict_topk: top_k must be in 1..%d (got %d)", TK_CAP / 4, k);
    TRS_REQUIRE(n_query >= 0 && n_query < (1ll << 31) - TK_BM && m->item.n_rows < (1ll << 31) - TK_BN,
                "predict_topk: too many users / items for one call");
    return TRS_OK;
}

}  // namespace trs

using namespace trs;

extern "C" size_t trs_predict_topk_workspace_bytes(const trs_model* model, int64_t n_query, int k) {
    if (check_topk(model, n_query, k) || n_query == 0) return 0;
    return topk_layout(model, n_query).total;
}

extern "C" int trs_predict_topk(const trs_model* model, const int64_t* users, int64_t n_query,
                                const int64_t* item_meta, int k, int64_t item_offset, int64_t* out_idx,
                                float* out_score, int32_t* overflow, void* workspace, size_t workspace_bytes,
                                trs_stream_t stream) {
    return trs_predict_topk_reuse(model, users, n_query, item_meta, k, item_offset, out_idx, out_score, overflow,
                                  workspace, workspace_bytes, 0, stream);
}

extern "C" int trs_predict_topk_reuse(const trs_model* model, const int64_t* users, int64_t n_query,
                                      const int64_t* item_meta, int k, int64_t item_offset, int64_t* out_idx,
                                      float* out_score, int32_t* overflow, void* workspace, size_t workspace_bytes,
                                      int items_prepared, trs_stream_t stream) {
    int rc = check_topk(model, n_query, k);
    if (rc) return rc;
    if (n_query == 0) return TRS_OK;
    TRS_REQUIRE(users && out_idx && out_score && overflow && workspace, "predict_topk: NULL pointer");
    TRS_REQUIRE(model->n_meta == 0 || item_meta, "predict_topk: model has metadata tables but item_meta is NULL");
    const TopkLayout L = topk_layout(model, n_query);
    if (workspace_bytes < L.total) {
        set_error("predict_topk workspace too small: %zu < %zu", workspace_bytes, L.total);
        return TRS_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* W = (char*)workspace;
    const int64_t n_items = model->item.n_rows;
    // items_prepared: the workspace still holds the bf16 item operand (and its max norm) of a previous call with the
    // same item tables and n_query -- the 1.4 GB re-cast of an unchanged 5M x 128 table is skipped
    if (!items_prepared) TRS_CUDA(cudaMemsetAsync(W + L.vmax2, 0, 256, st));
    TRS_CUDA(cudaMemsetAsync(overflow, 0, (size_t)n_query * 4, st));
    TRS_CUDA(cudaMemsetAsync(W + L.Ub, 0, (size_t)L.user_tiles * TK_BM * L.Kp * 2, st));
    {
        long long blocks = (n_items + 7) / 8;
        const long long cap = (long long)device_props().sm_count * 32;
        if (items_prepared) {
        } else if (model->dim % 4 == 0)
            topk_prep_items_kernel<true><<<(int)(blocks > cap ? cap : blocks), 256, 0, st>>>(
                *model, item_meta, n_items, L.Kp, (bf16*)(W + L.Vb), (unsigned*)(W + L.vmax2));
        else
            topk_prep_items_kernel<false><<<(int)(blocks > cap ? cap : blocks), 256, 0, st>>>(
                *model, item_meta, n_items, L.Kp, (bf16*)(W + L.Vb), (unsigned*)(W + L.vmax2));
        topk_prep_users_kernel<<<(int)((n_query + 7) / 8), 256, 0, st>>>(*model, users, (int)n_query, L.Kp, (bf16*)(W + L.Ub),
                                                                         (float*)(W + L.unorm), (float*)(W + L.ulin));
    }
    TopkDev g = {};
    g.n_query = (int)n_query;
    g.n_items = (int)n_items;
    g.nbox = L.nbox;
    g.kslices = L.kslices;
    g.Kp = L.Kp;
    g.Ub = (const bf16*)(W + L.Ub);
    g.stages = L.stages;
    g.n_item_tiles = L.n_item_tiles;
    g.tiles_per_split = L.tiles_per_split;
    g.splits = L.splits;
    g.k = k;
    g.fm = model->net == TRS_NET_FM;
    g.unorm = (const float*)(W + L.unorm);
    g.ulin = (const float*)(W + L.ulin);
    g.vmax2 = (const float*)(W + L.vmax2);
    g.cand_s = (float*)(W + L.cand_s);
    g.cand_i = (int*)(W + L.cand_i);
    g.cand_cnt = (int*)(W + L.cand_cnt);
    g.overflow = overflow;
    g.progress = (int*)(W + L.progress);
    {
        g.sync_window = TK_SYNC_WINDOW;
#ifdef TRS_DEBUG
        const char* w_env = getenv("TRS_TOPK_WINDOW");  // tuning hook of debug builds only
        if (w_env && atoi(w_env) > 0) g.sync_window = atoi(w_env);
#endif
    }
    TRS_CUDA(cudaMemsetAsync(g.progress, 0xff, (size_t)L.splits * L.user_tiles * 4, st));
    CUtensorMap tv;
    if ((rc = make_tmap_bf16(&tv, W + L.Vb, n_items, L.Kp, L.Kp, TK_BN))) return rc;
    TRS_CUDA(cudaFuncSetAttribute(topk_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
    const char* trace_env = getenv("TRS_TOPK_TRACE");  // debug: pipeline timeline of CTA (0, 0) -> stderr
    if (trace_env && atoi(trace_env)) {
        g.trace_t0 = atoi(trace_env) - 1;  // TRS_TOPK_TRACE = first traced tile + 1
        TRS_CUDA(cudaMalloc(&g.trace, (TK_TRACE_TILES * 8 + 3072) * sizeof(long long)));
        TRS_CUDA(cudaMemsetAsync(g.trace, 0, (TK_TRACE_TILES * 8 + 3072) * sizeof(long long), st));
    }
    topk_score_kernel<<<dim3(L.user_tiles, L.splits), TK_THREADS, L.smem, st>>>(tv, g);
    TRS_CUDA(cudaGetLastError());
    if (g.trace) {
        static long long h[TK_TRACE_TILES * 8 + 3072];
        TRS_CUDA(cudaStreamSynchronize(st));
        TRS_CUDA(cudaMemcpy(h, g.trace, sizeof(h), cudaMemcpyDeviceToHost));
        TRS_CUDA(cudaFree(g.trace));
        const int a = 200, b = 1000;
        const char* nm[8] = {"producer: slot free", "mma: accumulator free", "mma: operands landed", "mma: issued + committed",
                             "epilogue: accumulator full", "epilogue: tmem read, buffer released", "epilogue: filtered (lane 0)",
                             "epilogue: warp reconverged"};
        fprintf(stderr, "topk trace (CTA 0, tiles %d..%d): period %.0f cycles/tile\n", g.trace_t0 + a, g.trace_t0 + b, (double)(h[b * 8 + 3] - h[a * 8 + 3]) / (b - a));
        for (int e = 0; e < 8; ++e) {
            double off = 0;
            for (int t = a; t < b; ++t) off += (double)(h[t * 8 + e] - h[t * 8 + 1]);
            fprintf(stderr, "  %-40s %+8.0f cycles after 'mma: accumulator free' of the same tile\n", nm[e], off / (b - a));
        }
        {
            int last = 0;
            while (last + 1 < 1024 && h[TK_TRACE_TILES * 8 + last + 1]) ++last;
            fprintf(stderr, "  CTA 0 total: %.2f Mcycles over %d tiles\n",
                    (double)(h[TK_TRACE_TILES * 8 + last] - h[TK_TRACE_TILES * 8]) / 1e6, last * 256);
        }
        fprintf(stderr, "  cycles/tile per 256-tile window:");
        for (int w = 0; w + 1 < 1024 && h[TK_TRACE_TILES * 8 + w + 1]; ++w)
            fprintf(stderr, " %.0f", (double)(h[TK_TRACE_TILES * 8 + w + 1] - h[TK_TRACE_TILES * 8 + w]) / 256);
        fprintf(stderr, "\n  rows compacted / kcycles spent compacting per window (4 epilogue warps):");
        for (int w = 0; w + 1 < 1024 && h[TK_TRACE_TILES * 8 + w + 1]; ++w)
            fprintf(stderr, " %lld/%lld", h[TK_TRACE_TILES * 8 + 1024 + w], h[TK_TRACE_TILES * 8 + 2048 + w] / 1000);
        fprintf(stderr, "\n");
        g.trace = nullptr;
    }
    RowShape shape;
    pick_row_shape(model->dim, &shape);
    TRS_DISPATCH_ROW_SHAPE(shape, launch_rescore, model, users, item_meta, &g, item_offset, out_idx, out_score, st);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}
