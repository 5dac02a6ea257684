// extra.cu -- the pieces around the fused training path that keep the reference's OTHER entry points on the device:
//   * trs_scores_backward: backward of net.forward for Linear / FM (collaborative/linear.py:54-80, fm.py:60-101 under
//     autograd): one gradient row per lookup, which the host wraps as the sparse COO gradients an
//     nn.Embedding(sparse=True) backward would produce -- so TorchRecSys.forward -> hinge_loss ->
//     TorchRecSys.backward(loss, optimizer) (model.py:171-200) works with ANY torch optimizer.
//   * trs_sorted_auc: sort-based ROC-AUC over all positive / negative scores (north_star: "evaluate gains an
//     on-device sort-based AUC"; nearest reference code: helper/evaluate.py:8-18, which calls sklearn):
//     radix sort of the scores + tie-averaged rank sum (Mann-Whitney U), exact integer arithmetic on the ranks.
//   * trs_epoch_shuffle / trs_gather_rows_i64: the loader's per-epoch shuffle (dataset/dataset.py:369-373:
//     torch.randperm + index_select per key) as Philox keys + the plan's radix sort + one fused gather of all id
//     columns.
#include "plan.cuh"
#include "scorer.cuh"

namespace trs {

static int grid_cap(int64_t n, int per_block, int cap) {
    int64_t g = (n + per_block - 1) / per_block;
    if (g < 1) g = 1;
    return (int)(g < cap ? g : cap);
}

// ------------------------------------------------------------------------------------------------------------
// backward of the scorers
// ------------------------------------------------------------------------------------------------------------
struct ScoreGrads {
    float* g_user;               // [n, dim]
    float* g_item;               // [n, dim]
    float* g_meta[TRS_MAX_META]; // [n, dim] each
    float* g_lin_user;           // [n] (nullable)
    float* g_lin_item;           // [n] (nullable)
    float* g_lin_meta[TRS_MAX_META];
};

template <int NET, int V, int G, int IT>
__global__ void __launch_bounds__(256)
scores_backward_kernel(trs_model m, const int64_t* __restrict__ user, const int64_t* __restrict__ item,
                       const int64_t* __restrict__ meta, int64_t n, const float* __restrict__ grad_out, ScoreGrads sg) {
    const int nch = m.dim / V, dim = m.dim, F = m.n_meta;
    const int gl = threadIdx.x % G;
    constexpr int GPW = 32 / G;
    const int64_t gpb = blockDim.x / G;
    const int sub = (threadIdx.x / G) % GPW;
    for (int64_t b0 = blockIdx.x * gpb + threadIdx.x / G - sub; b0 < n; b0 += (int64_t)gridDim.x * gpb) {  // warp-uniform
        const bool valid = b0 + sub < n;
        const int64_t b = valid ? b0 + sub : n - 1;
        const int64_t u = user[b], it = item[b];
        const int64_t* mt = meta ? meta + b * F : nullptr;
        const float go = grad_out[b];
        const Row<V, IT> ru = load_row<V, G, IT>(m.user.emb + (size_t)u * dim, nch, gl);
        const float bu = m.user.lin ? m.user.lin[u] : 0.f;
        Row<V, IT> a, ri;
        float d;  // d loss / d (pre-activation)
        if (NET == TRS_NET_LINEAR) {
            (void)linear_score<V, G, IT>(m, nch, gl, ru, bu, it, mt, a);  // a = pooled item vector v
            d = go;
        } else {
            const float s = sigmoidf_acc(fm_logit<V, G, IT>(m, nch, gl, ru, bu, it, mt, a, ri));  // a = S = sum of fields
            d = go * s * (1.0f - s);
        }
        if (!valid) continue;
        Row<V, IT> gu, gi;
#pragma unroll
        for (int i = 0; i < IT; ++i)
#pragma unroll
            for (int k = 0; k < V; ++k) {
                if (NET == TRS_NET_LINEAR) {  // s = <u, v> + b_u + b_i: ds/du = v, ds/dv = u (item row and every metadata row)
                    gu.c[i][k] = d * a.c[i][k];
                    gi.c[i][k] = d * ru.c[i][k];
                } else {                      // dz/de_k = S - e_k
                    gu.c[i][k] = d * (a.c[i][k] - ru.c[i][k]);
                    gi.c[i][k] = d * (a.c[i][k] - ri.c[i][k]);
                }
            }
        store_row<V, G, IT>(sg.g_user + (size_t)b * dim, nch, gl, gu);
        store_row<V, G, IT>(sg.g_item + (size_t)b * dim, nch, gl, gi);
        for (int f = 0; f < F; ++f) {
            if (NET == TRS_NET_LINEAR) {
                store_row<V, G, IT>(sg.g_meta[f] + (size_t)b * dim, nch, gl, gi);
            } else {
                const Row<V, IT> rm = load_row<V, G, IT>(m.meta[f].emb + (size_t)mt[f] * dim, nch, gl);
                Row<V, IT> gm;
#pragma unroll
                for (int i = 0; i < IT; ++i)
#pragma unroll
                    for (int k = 0; k < V; ++k) gm.c[i][k] = d * (a.c[i][k] - rm.c[i][k]);
                store_row<V, G, IT>(sg.g_meta[f] + (size_t)b * dim, nch, gl, gm);
            }
        }
        if (gl == 0) {
            if (sg.g_lin_user) sg.g_lin_user[b] = d;
            if (sg.g_lin_item) sg.g_lin_item[b] = d;
            for (int f = 0; f < F; ++f)
                if (sg.g_lin_meta[f]) sg.g_lin_meta[f][b] = d;
        }
    }
}

template <int V, int G, int IT>
static void launch_scores_backward(const trs_model* m, const int64_t* user, const int64_t* item, const int64_t* meta,
                                   int64_t n, const float* go, const ScoreGrads* sg, cudaStream_t st) {
    const int grid = grid_cap(n, 256 / G, device_props().sm_count * 16);
    if (m->net == TRS_NET_LINEAR)
        scores_backward_kernel<TRS_NET_LINEAR, V, G, IT><<<grid, 256, 0, st>>>(*m, user, item, meta, n, go, *sg);
    else
        scores_backward_kernel<TRS_NET_FM, V, G, IT><<<grid, 256, 0, st>>>(*m, user, item, meta, n, go, *sg);
}

// ------------------------------------------------------------------------------------------------------------
// sort-based ROC-AUC
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
auc_keys_kernel(const float* __restrict__ pos, int64_t n_pos, const float* __restrict__ neg, int64_t n_neg,
                uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
    const int64_t n = n_pos + n_neg;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const bool p = k < n_pos;
        float x = p ? pos[k] : neg[k - n_pos];
        if (x == 0.f) x = 0.f;  // -0.0 and +0.0 are one score
        key[k] = float_key(x);
        val[k] = p ? 1u : 0u;
    }
}

// twice the sum of the tie-averaged 1-based ranks of the positives: a score whose run of equal scores occupies sorted
// positions [lo, hi) has average rank lo + (hi - lo + 1) / 2
__global__ void __launch_bounds__(256)
auc_rank_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ val, int64_t n,
                unsigned long long* __restrict__ sum2) {
    unsigned long long local = 0;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        if (!val[k]) continue;
        const uint32_t x = key[k];
        int64_t lo = k, hi = k + 1;
        if (k > 0 && key[k - 1] == x) {  // lower bound of x in [0, k)
            int64_t a = 0, b = k;
            while (a < b) {
                const int64_t mid = (a + b) >> 1;
                if (key[mid] < x) a = mid + 1; else b = mid;
            }
            lo = a;
        }
        if (k + 1 < n && key[k + 1] == x) {  // upper bound of x in (k, n)
            int64_t a = k + 1, b = n;
            while (a < b) {
                const int64_t mid = (a + b) >> 1;
                if (key[mid] <= x) a = mid + 1; else b = mid;
            }
            hi = a;
        }
        local += (unsigned long long)(2 * lo + (hi - lo) + 1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(sum2, local);  // integer: any order gives the same sum
}

__global__ void auc_final_kernel(const unsigned long long* __restrict__ sum2, int64_t n_pos, int64_t n_neg,
                                 double* __restrict__ out) {
    const double rank_sum = (double)sum2[0] * 0.5;
    const double u = rank_sum - (double)n_pos * ((double)n_pos + 1.0) * 0.5;
    out[0] = (n_pos > 0 && n_neg > 0) ? u / ((double)n_pos * (double)n_neg) : __longlong_as_double(0x7ff8000000000000ll);
}

// ------------------------------------------------------------------------------------------------------------
// epoch shuffle
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t philox_word(uint64_t seed, uint64_t idx) {
    uint32_t c[4] = {(uint32_t)idx, (uint32_t)(idx >> 32), 0x5EED5EEDu, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    return c[0];
}
__global__ void __launch_bounds__(256)
shuffle_keys_kernel(uint64_t seed, int64_t n, uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        key[k] = philox_word(seed, (uint64_t)k);
        val[k] = (uint32_t)k;
    }
}
__global__ void __launch_bounds__(256)
perm_out_kernel(const uint32_t* __restrict__ val, int64_t n, int64_t* __restrict__ perm) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
        perm[k] = (int64_t)val[k];
}

struct GatherCols {
    const int64_t* src[8];
    int64_t* dst[8];
    int width[8];
    int n_cols;
};
__global__ void __launch_bounds__(256)
gather_rows_kernel(GatherCols gc, const int64_t* __restrict__ perm, int64_t n) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = perm[k];
        for (int c = 0; c < gc.n_cols; ++c) {
            const int w = gc.width[c];
            for (int j = 0; j < w; ++j) gc.dst[c][k * w + j] = gc.src[c][p * w + j];
        }
    }
}

static size_t pairs_bytes(int64_t n) { return ((size_t)4 * n * sizeof(uint32_t) + 1023) / 256 * 256; }
static trs_epoch one_segment(int64_t n) {
    trs_epoch ep = {};
    ep.n_samples = n;
    ep.batch = (int32_t)n;
    return ep;
}

}  // namespace trs

using namespace trs;

extern "C" int trs_scores_backward(const trs_model* model, const int64_t* user, const int64_t* item, const int64_t* meta,
                                   int64_t n, const float* grad_out, float* g_user, float* g_item,
                                   float* const* g_meta_host, float* g_lin_user, float* g_lin_item,
                                   float* const* g_lin_meta_host, trs_stream_t stream) {
    RowShape shape;
    int rc = check_model(model, &shape);
    if (rc) return rc;
    TRS_REQUIRE(model->net != TRS_NET_MLP, "trs_scores_backward: Linear / FM only");
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(user && item && grad_out && g_user && g_item, "NULL pointer");
    TRS_REQUIRE(model->n_meta == 0 || (meta && g_meta_host), "model has metadata tables but meta ids / gradient buffers are NULL");
    ScoreGrads sg = {};
    sg.g_user = g_user;
    sg.g_item = g_item;
    sg.g_lin_user = model->user.lin ? g_lin_user : nullptr;
    sg.g_lin_item = model->item.lin ? g_lin_item : nullptr;
    for (int f = 0; f < model->n_meta; ++f) {
        TRS_REQUIRE(g_meta_host[f], "gradient buffer of metadata table %d is NULL", f);
        sg.g_meta[f] = g_meta_host[f];
        sg.g_lin_meta[f] = (model->meta[f].lin && g_lin_meta_host) ? g_lin_meta_host[f] : nullptr;
    }
    TRS_DISPATCH_ROW_SHAPE(shape, launch_scores_backward, model, user, item, meta, n, grad_out, &sg, (cudaStream_t)stream);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" size_t trs_sort_workspace_bytes(int64_t n) {
    if (n <= 0) return 256;
    const trs_epoch ep = one_segment(n);
    return pairs_bytes(n) + hist_bytes(&ep) + 256;
}

extern "C" int trs_sorted_auc(const float* pos, int64_t n_pos, const float* neg, int64_t n_neg, double* auc_out,
                              void* workspace, size_t workspace_bytes, trs_stream_t stream) {
    TRS_REQUIRE(auc_out && workspace, "sorted_auc: NULL pointer");
    TRS_REQUIRE(n_pos >= 0 && n_neg >= 0 && n_pos + n_neg <= (1ll << 23),
                "sorted_auc: at most 2^23 scores per call (got %lld)", (long long)(n_pos + n_neg));
    TRS_REQUIRE((n_pos == 0 || pos) && (n_neg == 0 || neg), "sorted_auc: NULL scores");
    const int64_t n = n_pos + n_neg;
    if (workspace_bytes < trs_sort_workspace_bytes(n)) {
        set_error("sorted_auc workspace too small");
        return TRS_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* k0 = (uint32_t*)workspace;
    uint32_t* v0 = k0 + n;
    uint32_t* k1 = v0 + n;
    uint32_t* v1 = k1 + n;
    unsigned long long* sum2 = (unsigned long long*)((char*)workspace + pairs_bytes(n > 0 ? n : 1));
    uint32_t* hist = (uint32_t*)(sum2 + 32);
    TRS_CUDA(cudaMemsetAsync(sum2, 0, sizeof(unsigned long long), st));
    if (n > 0) {
        const int grid = grid_cap(n, 256, device_props().sm_count * 8);
        auc_keys_kernel<<<grid, 256, 0, st>>>(pos, n_pos, neg, n_neg, k0, v0);
        const trs_epoch ep = one_segment(n);
        const int npass = sort_pairs(k0, v0, k1, v1, 1, (int64_t)1 << 32, &ep, nullptr, 0, hist, st);
        const uint32_t* sk = (npass & 1) ? k1 : k0;
        const uint32_t* sv = (npass & 1) ? v1 : v0;
        auc_rank_kernel<<<grid, 256, 0, st>>>(sk, sv, n, sum2);
    }
    auc_final_kernel<<<1, 1, 0, st>>>(sum2, n_pos, n_neg, auc_out);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_epoch_shuffle(uint64_t seed, int64_t n, int64_t* perm, void* workspace, size_t workspace_bytes,
                                 trs_stream_t stream) {
    TRS_REQUIRE(n >= 0 && n <= (1ll << 23), "epoch_shuffle: at most 2^23 samples per call (got %lld)", (long long)n);
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(perm && workspace, "epoch_shuffle: NULL pointer");
    if (workspace_bytes < trs_sort_workspace_bytes(n)) {
        set_error("epoch_shuffle workspace too small");
        return TRS_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* k0 = (uint32_t*)workspace;
    uint32_t* v0 = k0 + n;
    uint32_t* k1 = v0 + n;
    uint32_t* v1 = k1 + n;
    uint32_t* hist = (uint32_t*)((char*)workspace + pairs_bytes(n) + 256);
    const int grid = grid_cap(n, 256, device_props().sm_count * 8);
    shuffle_keys_kernel<<<grid, 256, 0, st>>>(seed, n, k0, v0);
    const trs_epoch ep = one_segment(n);
    const int npass = sort_pairs(k0, v0, k1, v1, 1, (int64_t)1 << 32, &ep, nullptr, 0, hist, st);
    perm_out_kernel<<<grid, 256, 0, st>>>((npass & 1) ? v1 : v0, n, perm);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_gather_rows_i64(const int64_t* const* src_host, int64_t* const* dst_host, const int32_t* width_host,
                                   int n_cols, const int64_t* perm, int64_t n, trs_stream_t stream) {
    TRS_REQUIRE(n_cols >= 0 && n_cols <= 8, "gather_rows: at most 8 columns");
    if (n == 0 || n_cols == 0) return TRS_OK;
    TRS_REQUIRE(src_host && dst_host && width_host && perm, "gather_rows: NULL pointer");
    GatherCols gc = {};
    gc.n_cols = n_cols;
    for (int c = 0; c < n_cols; ++c) {
        TRS_REQUIRE(src_host[c] && dst_host[c] && width_host[c] >= 1, "gather_rows: column %d", c);
        gc.src[c] = src_host[c];
        gc.dst[c] = dst_host[c];
        gc.width[c] = width_host[c];
    }
    const int grid = grid_cap(n, 256, device_props().sm_count * 8);
    gather_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(gc, perm, n);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}
