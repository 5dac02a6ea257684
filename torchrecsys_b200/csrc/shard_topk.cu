// shard_topk.cu -- exact top-k over a rank's own item shard of the row-sharded tables (trs_shard, csrc/shard.cu).
//   * trs_shard_topk_exact: exact fp32 top-k of the shard for dense query rows, bit-identical to trs_scores + a stable
//     descending sort, optionally leaving out given items (ShardedLinearTrainer.recommend; predict_topk's overflow).
//   * trs_shard_topk_merge_sorted: merge of such sorted lists -- item ranges of one rank, or ranks -- and of the
//     item blocks' trs_predict_topk lists of the item-sharded predict (sharded_predict_topk), ordered the same way.
// Kept out of shard_serve.cu: a kernel with dynamic shared memory in that module changes the shared-memory reservation,
// and so the SASS, of its existing kernels.
#include "scorer.cuh"

namespace trs {

// ---- exact top-k over the rank's own item shard ---------------------------------------------------------------------
// A CTA scores a tile of TK_UT query users (rows in shared memory) against one contiguous range of the shard's items,
// TK_NT items per tile: thread t takes item t % TK_NT for users (t / TK_NT) * TK_RU .. + TK_RU, item chunks straight from
// global memory, user chunks as shared-memory broadcasts.  Each (user, range) keeps a candidate list in the workspace:
// a score is appended only when it beats the running k-th best (and is not excluded); a list about to overflow is
// sorted by the CTA and cut to k, which raises the threshold.  The range's sorted top-k ends the CTA.
// Rows are float4 chunks only (V = 4): the row-sharded tables require dim % 4 == 0 (check_shard).
constexpr int TK_THREADS = 256, TK_UT = 16, TK_RU = 8, TK_NT = TK_THREADS * TK_RU / TK_UT, TK_MAX_RANGES = 16;

// (score desc, id asc) as one descending uint64: the score's order-preserving key above ~id.  -0 keys as +0: torch.sort
// treats equal values as ties.
__device__ __forceinline__ uint64_t topk_key(float s, uint32_t id) {
    return ((uint64_t)float_key(s == 0.f ? 0.f : s) << 32) | (uint64_t)(0xFFFFFFFFu - id);
}
__device__ __forceinline__ float key_score(uint64_t c) {
    const uint32_t k = (uint32_t)(c >> 32);
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

__device__ __forceinline__ bool excluded(const int64_t* __restrict__ ptr, const int64_t* __restrict__ ids, int64_t q,
                                         int64_t id) {
    if (!ptr) return false;
    int64_t lo = ptr[q], hi = ptr[q + 1];
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int64_t v = ids[mid];
        if (v == id) return true;
        if (v < id) lo = mid + 1;
        else hi = mid;
    }
    return false;
}

__host__ __device__ constexpr int ilog2c(int g) { return g <= 1 ? 0 : 1 + ilog2c(g >> 1); }
__host__ __device__ constexpr int brevc(int m, int bits) { return bits == 0 ? 0 : ((m & 1) << (bits - 1)) | brevc(m >> 1, bits - 1); }

// s[0 .. S) sorted descending (S a power of two) by the whole CTA
__device__ void cta_sort_desc(uint64_t* s, int S) {
    for (int size = 2; size <= S; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < (S >> 1); i += blockDim.x) {
                const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
                const uint64_t a = s[lo], b = s[hi];
                if (((lo & size) == 0) ? (a < b) : (a > b)) {
                    s[lo] = b;
                    s[hi] = a;
                }
            }
            __syncthreads();
        }
}

// Sorts the first n candidates of buf (n <= C) and keeps the best `keep`; returns the count kept.  Uniform in the CTA.
__device__ int cta_cut(uint64_t* __restrict__ buf, int n, int keep, uint64_t* scratch) {
    int S = 2;
    while (S < n) S <<= 1;
    for (int i = threadIdx.x; i < S; i += blockDim.x) scratch[i] = i < n ? buf[i] : 0ull;
    __syncthreads();
    cta_sort_desc(scratch, S);
    const int m = n < keep ? n : keep;
    for (int i = threadIdx.x; i < m; i += blockDim.x) buf[i] = scratch[i];
    __syncthreads();
    return m;
}

// Scores of RU users x one item exactly as trs_scores computes them with the row shape (V, G, IT): lane j's partial
// is the fmaf chain over chunks i * G + j (components in order, zero-padded chunks included), the G partials are added
// by group_sum's xor butterfly -- visited here in bit-reversed lane order, where the butterfly is a left-to-right
// pairwise tree kept on a stack of log2(G) + 1 values -- then (dot + b_u) + b_i.
__host__ __device__ constexpr int trailing_ones(int m) { return (m & 1) ? 1 + trailing_ones(m >> 1) : 0; }

// lane j = brev(M)'s partial for RU users, pushed onto the per-user stacks (M + 1 leaves so far: the pairs the
// binary counter closes are added)
template <int V, int G, int IT, int RU, int M>
__device__ __forceinline__ void topk_lane(const float* __restrict__ su, int dp, const float* __restrict__ vrow,
                                          bool valid, int nch, float (&acc)[RU][ilog2c(G) + 1]) {
    constexpr int j = brevc(M, ilog2c(G)), T = trailing_ones(M);
    float p[RU];
#pragma unroll
    for (int r = 0; r < RU; ++r) p[r] = 0.f;
#pragma unroll
    for (int i = 0; i < IT; ++i) {
        const int c = i * G + j;
        const Vec<V> v = (valid && c < nch) ? Vec<V>::ld(vrow + (size_t)c * V) : Vec<V>::zero();
#pragma unroll
        for (int r = 0; r < RU; ++r) {
            const Vec<V> u = Vec<V>::ld(su + r * dp + c * V);
#pragma unroll
            for (int k = 0; k < V; ++k) p[r] = fmaf(u[k], v[k], p[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < RU; ++r) {
        float x = p[r];
#pragma unroll
        for (int b = 0; b < T; ++b) x = acc[r][b] + x;
        acc[r][T] = x;
    }
    if constexpr (M + 1 < G) topk_lane<V, G, IT, RU, M + 1>(su, dp, vrow, valid, nch, acc);
}

// Scores of RU users x one item exactly as trs_scores computes them with the row shape (V, G, IT): lane j's partial
// is the fmaf chain over chunks i * G + j (components in order, zero-padded chunks included), the G partials are added
// by group_sum's xor butterfly -- visited here in bit-reversed lane order, where the butterfly is a left-to-right
// pairwise tree kept on a stack of log2(G) + 1 values -- then (dot + b_u) + b_i (by the caller).
template <int V, int G, int IT, int RU>
__device__ __forceinline__ void topk_scores(const float* __restrict__ su, int dp, const float* __restrict__ vrow,
                                            bool valid, int nch, float (&dot)[RU]) {
    float acc[RU][ilog2c(G) + 1];
    topk_lane<V, G, IT, RU, 0>(su, dp, vrow, valid, nch, acc);
#pragma unroll
    for (int r = 0; r < RU; ++r) dot[r] = acc[r][ilog2c(G)];
}

struct TopkExactArgs {
    const float* item_emb;
    const float* item_lin;
    int64_t rows;         // items on the shard
    int64_t range_rows;   // items per range (a multiple of 128)
    const float* user_emb;
    const float* user_lin;
    int64_t n_query;
    int dim, k, cap, rank, world;
    const int64_t* excl_ptr;
    const int64_t* excl_ids;
    uint64_t* cand;       // [tiles][ranges][TK_UT][cap]
    int64_t* out_idx;     // [ranges][n_query][k] (or the output when there is one range)
    float* out_score;
};

template <int V, int G, int IT>
__global__ void __launch_bounds__(TK_THREADS, 2) shard_topk_exact_kernel(const __grid_constant__ TopkExactArgs a) {
    extern __shared__ __align__(16) unsigned char tk_smem[];
    constexpr int DP = G * IT * V;   // a user row padded to whole chunks of every lane
    uint64_t* scratch = reinterpret_cast<uint64_t*>(tk_smem);
    uint64_t* thresh = scratch + a.cap;
    float* su = reinterpret_cast<float*>(thresh + TK_UT);
    float* sbu = su + TK_UT * DP;
    int* cnt = reinterpret_cast<int*>(sbu + TK_UT);

    const int dim = a.dim, nch = dim / V;
    const int64_t q0 = (int64_t)blockIdx.x * TK_UT;
    const int range = blockIdx.y;
    const int64_t lo = (int64_t)range * a.range_rows;
    const int64_t hi = min(lo + a.range_rows, a.rows);
    uint64_t* cand = a.cand + ((size_t)blockIdx.x * gridDim.y + range) * TK_UT * a.cap;

    for (int e = threadIdx.x; e < TK_UT * DP; e += blockDim.x) {
        const int u = e / DP, d = e % DP;
        const int64_t q = q0 + u;
        su[e] = (q < a.n_query && d < dim) ? a.user_emb[q * dim + d] : 0.f;
    }
    if (threadIdx.x < TK_UT) {
        const int64_t q = q0 + threadIdx.x;
        sbu[threadIdx.x] = (q < a.n_query && a.user_lin) ? a.user_lin[q] : 0.f;
        thresh[threadIdx.x] = 0ull;
        cnt[threadIdx.x] = 0;
    }
    __syncthreads();

    static_assert(V == 4, "the row-sharded tables have float4 rows");
    constexpr int RU = TK_RU, NT = TK_NT;
    const int t_item = threadIdx.x % NT, u0 = (threadIdx.x / NT) * RU;
    for (int64_t base = lo; base < hi; base += NT) {
        const int64_t id = base + t_item;
        const bool valid = id < hi;
        float dot[RU];
        topk_scores<V, G, IT, RU>(su + u0 * DP, DP, a.item_emb + (size_t)(valid ? id : lo) * dim, valid, nch, dot);
        if (valid) {
            const float bi = a.item_lin ? a.item_lin[id] : 0.f;
#pragma unroll
            for (int r = 0; r < RU; ++r) {
                const int u = u0 + r;
                const int64_t q = q0 + u;
                if (q >= a.n_query) break;
                const uint64_t c = topk_key((dot[r] + sbu[u]) + bi, (uint32_t)id);
                if (c > thresh[u] && !excluded(a.excl_ptr, a.excl_ids, q, id)) {
                    const int pos = atomicAdd(&cnt[u], 1);
                    cand[(size_t)u * a.cap + pos] = c;
                }
            }
        }
        __syncthreads();
        for (int u = 0; u < TK_UT; ++u) {   // cut every list that the next tile could overflow
            const int n = cnt[u];
            if (n > a.cap - NT) {
                __syncthreads();
                const int m = cta_cut(cand + (size_t)u * a.cap, n, a.k, scratch);
                if (threadIdx.x == 0) {
                    cnt[u] = m;
                    thresh[u] = m == a.k ? scratch[a.k - 1] : 0ull;
                }
                __syncthreads();
            }
        }
        __syncthreads();   // every count is read before the next tile's appends raise it
    }

    for (int u = 0; u < TK_UT; ++u) {
        const int64_t q = q0 + u;
        if (q >= a.n_query) break;
        const int m = cta_cut(cand + (size_t)u * a.cap, cnt[u], a.k, scratch);
        const size_t o = ((size_t)range * a.n_query + q) * a.k;
        for (int i = threadIdx.x; i < a.k; i += blockDim.x) {
            if (i < m) {
                const uint64_t c = scratch[i];
                a.out_idx[o + i] = (int64_t)(0xFFFFFFFFu - (uint32_t)c) * a.world + a.rank;
                a.out_score[o + i] = key_score(c);
            } else {
                a.out_idx[o + i] = -1;
                a.out_score[o + i] = -INFINITY;
            }
        }
        __syncthreads();
    }
}

// ---- merge of sorted lists: an element's output position is its rank in its own list plus, in every other list, the
// number of elements that precede it (binary search).  Excluded or padding elements are dropped by counting only the
// kept ones: cnt[l][p] = kept elements among list l's first p.
__device__ __forceinline__ bool precedes(float sb, int64_t ib, uint32_t ke, int64_t ie) {
    if (ib < 0) return false;
    const uint32_t kb = float_key(sb == 0.f ? 0.f : sb);
    return kb > ke || (kb == ke && ib < ie);
}

__global__ void __launch_bounds__(256) topk_merge_sorted_kernel(const float* __restrict__ score,
                                                                const int64_t* __restrict__ idx, int n_lists,
                                                                int64_t n_query, int k_in, int k_out,
                                                                const int64_t* __restrict__ excl_ptr,
                                                                const int64_t* __restrict__ excl_ids,
                                                                int64_t* __restrict__ out_idx,
                                                                float* __restrict__ out_score) {
    extern __shared__ int mg_cnt[];   // [n_lists][k_in + 1]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const size_t ls = (size_t)n_query * k_in;   // list stride
    for (int64_t q = blockIdx.x; q < n_query; q += gridDim.x) {
        for (int l = warp; l < n_lists; l += nw) {
            const size_t row = l * ls + (size_t)q * k_in;
            int run = 0;
            for (int p0 = 0; p0 < k_in; p0 += 32) {
                const int p = p0 + lane;
                bool keep = false;
                if (p < k_in) {
                    const int64_t id = idx[row + p];
                    keep = id >= 0 && !excluded(excl_ptr, excl_ids, q, id);
                }
                const unsigned b = __ballot_sync(0xffffffffu, keep);
                if (p < k_in) mg_cnt[l * (k_in + 1) + p] = run + __popc(b & ((1u << lane) - 1u));
                run += __popc(b);
            }
            if (lane == 0) mg_cnt[l * (k_in + 1) + k_in] = run;
        }
        __syncthreads();
        int total = 0;
        for (int l = 0; l < n_lists; ++l) total += mg_cnt[l * (k_in + 1) + k_in];
        for (int i = total + threadIdx.x; i < k_out; i += blockDim.x) {
            out_idx[(size_t)q * k_out + i] = -1;
            out_score[(size_t)q * k_out + i] = -INFINITY;
        }
        for (int e = threadIdx.x; e < n_lists * k_in; e += blockDim.x) {
            const int l = e / k_in, p = e % k_in;
            const int* cl = mg_cnt + l * (k_in + 1);
            if (cl[p + 1] == cl[p]) continue;   // excluded or padding
            int rank = cl[p];
            if (rank >= k_out) continue;
            const size_t at = l * ls + (size_t)q * k_in + p;
            const float s = score[at];
            const int64_t id = idx[at];
            const uint32_t ke = float_key(s == 0.f ? 0.f : s);
            for (int b = 0; b < n_lists && rank < k_out; ++b) {
                if (b == l) continue;
                const size_t rb = b * ls + (size_t)q * k_in;
                int lo = 0, hi = k_in;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (precedes(score[rb + mid], idx[rb + mid], ke, id)) lo = mid + 1;
                    else hi = mid;
                }
                rank += mg_cnt[b * (k_in + 1) + lo];
            }
            if (rank < k_out) {
                out_idx[(size_t)q * k_out + rank] = id;
                out_score[(size_t)q * k_out + rank] = s;
            }
        }
        __syncthreads();
    }
}

struct TopkExactPlan {
    int64_t tiles, range_rows;
    int ranges, cap;
    size_t cand_bytes, list_bytes, smem;
};

static int topk_exact_plan(const trs_shard* sh, int64_t n_query, int k, TopkExactPlan* p, RowShape* shape) {
    int rc = check_shard(sh, shape);
    if (rc) return rc;
    TRS_REQUIRE(k >= 1 && k <= 1024, "k must be in 1..1024, got %d", k);
    TRS_REQUIRE(n_query >= 0, "negative query count");
    const int64_t rows = sh->item[sh->rank].n_rows;
    int kp = 128;
    while (kp < k) kp <<= 1;
    p->cap = 2 * kp;
    p->tiles = (n_query + TK_UT - 1) / TK_UT;
    // enough CTAs for two per SM; a range keeps at least 1024 items
    const int64_t want = p->tiles ? (2 * (int64_t)device_props().sm_count + p->tiles - 1) / p->tiles : 1;
    const int64_t by_rows = (rows + 1023) / 1024;
    int64_t R = want < by_rows ? want : by_rows;
    R = R < 1 ? 1 : (R > TK_MAX_RANGES ? TK_MAX_RANGES : R);
    p->range_rows = ((rows + R - 1) / R + 127) / 128 * 128;
    if (p->range_rows == 0) p->range_rows = 128;
    p->ranges = (int)((rows + p->range_rows - 1) / p->range_rows);
    if (p->ranges < 1) p->ranges = 1;
    p->cand_bytes = ((size_t)p->tiles * p->ranges * TK_UT * p->cap * 8 + 255) / 256 * 256;
    p->list_bytes = p->ranges > 1 ? ((size_t)p->ranges * n_query * k * 12 + 255) / 256 * 256 : 0;
    const int DP = shape->G * shape->IT * shape->V;
    p->smem = (size_t)p->cap * 8 + TK_UT * 8 + (size_t)TK_UT * DP * 4 + TK_UT * 4 + TK_UT * 4;
    return TRS_OK;
}

template <int V, int G, int IT>
static void launch_topk_exact(const TopkExactPlan& p, const TopkExactArgs& a, cudaStream_t st, cudaError_t* err) {
    *err = cudaFuncSetAttribute(shard_topk_exact_kernel<V, G, IT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)p.smem);
    if (*err == cudaSuccess)
        shard_topk_exact_kernel<V, G, IT><<<dim3((unsigned)p.tiles, p.ranges), TK_THREADS, p.smem, st>>>(a);
}

static int launch_merge_sorted(const float* score, const int64_t* idx, int n_lists, int64_t n_query, int k_in,
                               int k_out, const int64_t* excl_ptr, const int64_t* excl_ids, int64_t* out_idx,
                               float* out_score, cudaStream_t st) {
    const size_t smem = (size_t)n_lists * (k_in + 1) * sizeof(int);
    TRS_REQUIRE(smem <= 160 * 1024, "%d lists of %d do not fit the merge's shared memory", n_lists, k_in);
    TRS_CUDA(cudaFuncSetAttribute(topk_merge_sorted_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t cap = (int64_t)device_props().sm_count * 8;
    const int grid = (int)(n_query < cap ? n_query : cap);
    topk_merge_sorted_kernel<<<grid, 256, smem, st>>>(score, idx, n_lists, n_query, k_in, k_out, excl_ptr, excl_ids,
                                                      out_idx, out_score);
    return TRS_OK;
}

}  // namespace trs

using namespace trs;

extern "C" size_t trs_shard_topk_exact_workspace_bytes(const trs_shard* shard, int64_t n_query, int k) {
    TopkExactPlan p;
    RowShape shape;
    if (topk_exact_plan(shard, n_query, k, &p, &shape)) return 0;
    return p.cand_bytes + p.list_bytes + 256;
}

extern "C" int trs_shard_topk_exact(const trs_shard* shard, const float* user_emb, const float* user_lin,
                                    int64_t n_query, int k, const int64_t* excl_ptr, const int64_t* excl_ids,
                                    int64_t* out_idx, float* out_score, void* workspace, size_t workspace_bytes,
                                    trs_stream_t stream) {
    TopkExactPlan p;
    RowShape shape;
    int rc = topk_exact_plan(shard, n_query, k, &p, &shape);
    if (rc) return rc;
    if (n_query == 0) return TRS_OK;
    TRS_REQUIRE(user_emb && out_idx && out_score, "NULL pointer");
    TRS_REQUIRE(!excl_ptr == !excl_ids, "exclusion ids and row pointers go together");
    const trs_table& it = shard->item[shard->rank];
    TRS_REQUIRE(it.emb || it.n_rows == 0, "rank %d's item shard is NULL", shard->rank);
    TRS_REQUIRE(it.n_rows < 0xFFFFFFFFll, "item shard of %lld rows: local ids must fit 32 bits", (long long)it.n_rows);
    TRS_REQUIRE(workspace && workspace_bytes >= p.cand_bytes + p.list_bytes,
                "workspace of %zu bytes, trs_shard_topk_exact_workspace_bytes() asks %zu", workspace_bytes,
                p.cand_bytes + p.list_bytes + 256);
    const cudaStream_t st = (cudaStream_t)stream;
    unsigned char* ws = (unsigned char*)workspace;
    TopkExactArgs a;
    a.item_emb = it.emb;
    a.item_lin = it.lin;
    a.rows = it.n_rows;
    a.range_rows = p.range_rows;
    a.user_emb = user_emb;
    a.user_lin = user_lin;
    a.n_query = n_query;
    a.dim = shard->dim;
    a.k = k;
    a.cap = p.cap;
    a.rank = shard->rank;
    a.world = shard->world;
    a.excl_ptr = excl_ptr;
    a.excl_ids = excl_ids;
    a.cand = (uint64_t*)ws;
    int64_t* list_idx = (int64_t*)(ws + p.cand_bytes);
    float* list_score = (float*)(list_idx + (size_t)p.ranges * n_query * k);
    a.out_idx = p.ranges > 1 ? list_idx : out_idx;
    a.out_score = p.ranges > 1 ? list_score : out_score;
    cudaError_t err = cudaErrorInvalidValue;
    switch (shape.G * 10 + shape.IT) {   // pick_row_shape's float4 shapes (check_shard requires dim % 4 == 0)
        case 41: launch_topk_exact<4, 4, 1>(p, a, st, &err); break;
        case 81: launch_topk_exact<4, 8, 1>(p, a, st, &err); break;
        case 161: launch_topk_exact<4, 16, 1>(p, a, st, &err); break;
        case 321: launch_topk_exact<4, 32, 1>(p, a, st, &err); break;
        case 322: launch_topk_exact<4, 32, 2>(p, a, st, &err); break;
        case 324: launch_topk_exact<4, 32, 4>(p, a, st, &err); break;
        default: TRS_REQUIRE(false, "no exact top-k for the row shape of dim %d", shard->dim);
    }
    TRS_CUDA(err);
    TRS_CUDA(cudaGetLastError());
    if (p.ranges > 1)
        return trs_shard_topk_merge_sorted(list_score, list_idx, p.ranges, n_query, k, k, nullptr, nullptr, out_idx,
                                           out_score, stream);
    return TRS_OK;
}

extern "C" int trs_shard_topk_merge_sorted(const float* score, const int64_t* idx, int n_lists, int64_t n_query,
                                           int k_in, int k_out, const int64_t* excl_ptr, const int64_t* excl_ids,
                                           int64_t* out_idx, float* out_score, trs_stream_t stream) {
    TRS_REQUIRE(n_lists >= 1 && k_in >= 1 && k_out >= 1, "n_lists, k_in and k_out must be positive");
    TRS_REQUIRE(n_query >= 0, "negative query count");
    if (n_query == 0) return TRS_OK;
    TRS_REQUIRE(score && idx && out_idx && out_score, "NULL pointer");
    TRS_REQUIRE(!excl_ptr == !excl_ids, "exclusion ids and row pointers go together");
    int rc = launch_merge_sorted(score, idx, n_lists, n_query, k_in, k_out, excl_ptr, excl_ids, out_idx, out_score,
                                 (cudaStream_t)stream);
    if (rc) return rc;
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}
