// sharded.cu -- the kernels the multi-GPU paths need on top of the single-GPU ones (SURVEY.md §8e):
//   * trs_sparse_row_update: coalesce() + row-wise optimizer step of ONE table on an explicit list of
//     (row id, gradient row) pairs -- what the OWNER of a table shard runs on the gradient rows the other
//     ranks sent it (torch: optim/_functional.py:44-84, optim/adagrad.py:363-373).  Stable radix sort by row
//     id (plan.cu), then one row group per segment sums its rows in list order (= rank order, then lookup
//     order: deterministic) and applies SGD / Adagrad / SparseAdam.
//   * trs_linear_rows_step: forward x2 + hinge + closed-form backward of the Linear scorer
//     (collaborative/linear.py:54-80, helper/loss.py:5-9; SURVEY a7) on rows that were GATHERED ELSEWHERE
//     (the owners' shards) and arrive as dense [B, dim] buffers; emits one gradient row per lookup.
//   * trs_topk_merge: k-way merge of per-shard top-k lists (score desc, item id asc) after the allgather of
//     the item-sharded predict.
#include "plan.cuh"
#include "scorer.cuh"
#include "train.cuh"

namespace trs {

// ---- segmented reduce + update over sorted (row, lookup) pairs ----------------------------------------------
template <int V, int G, int IT>
__global__ void __launch_bounds__(256)
segment_update_kernel(const __grid_constant__ trs_table t, int dim, const uint32_t* __restrict__ K,
                      const uint32_t* __restrict__ P, int n, const float* __restrict__ grad,
                      const float* __restrict__ grad_lin, const __grid_constant__ OptScalars opt, int step) {
    const int nch = dim / V, gl = threadIdx.x % G;
    constexpr int GPW = 32 / G;
    const int gpb = blockDim.x / G;
    const int sub = (threadIdx.x / G) % GPW;
    const float scale = opt.step_scale[step];
    for (int k0 = blockIdx.x * gpb + threadIdx.x / G - sub; k0 < n; k0 += gridDim.x * gpb) {
        const int k = k0 + sub;
        if (k >= n) continue;
        const uint32_t key = K[k];
        if (k > 0 && K[k - 1] == key) continue;  // not a segment head
        Row<V, IT> g = load_row<V, G, IT>(grad + (size_t)P[k] * dim, nch, gl);
        float gl_sum = grad_lin ? grad_lin[P[k]] : 0.f;
        for (int q = k + 1; q < n && K[q] == key; ++q) {  // duplicates, in list order
            row_acc(g, load_row<V, G, IT>(grad + (size_t)P[q] * dim, nch, gl));
            if (grad_lin) gl_sum = __fadd_rn(gl_sum, grad_lin[P[q]]);
        }
        const size_t roff = (size_t)key * dim;
        Row<V, IT> p = load_row<V, G, IT>(t.emb + roff, nch, gl), s0, s1;
        row_zero(s0);
        row_zero(s1);
        if (opt.kind != TRS_OPT_SGD) s0 = load_row<V, G, IT>(t.emb_s0 + roff, nch, gl);
        if (opt.kind == TRS_OPT_SPARSE_ADAM) s1 = load_row<V, G, IT>(t.emb_s1 + roff, nch, gl);
        update_store_row<V, G, IT>(t, roff, nch, gl, opt, scale, p, s0, s1, g);
        if (grad_lin && t.lin && gl == 0) {
            float pl = t.lin[key], l0 = 0.f, l1 = 0.f;
            if (opt.kind != TRS_OPT_SGD) l0 = t.lin_s0[key];
            if (opt.kind == TRS_OPT_SPARSE_ADAM) l1 = t.lin_s1[key];
            update_store_lin(t, key, opt, scale, gl_sum, pl, l0, l1);
        }
    }
}

template <int V, int G, int IT>
static void launch_segment_update(const trs_table* t, int dim, const uint32_t* K, const uint32_t* P, int n,
                                  const float* grad, const float* grad_lin, const OptScalars* opt, int step,
                                  cudaStream_t st) {
    const int gpb = 256 / G;
    int grid = (n + gpb - 1) / gpb;
    const int cap = device_props().sm_count * 16;
    segment_update_kernel<V, G, IT><<<grid > cap ? cap : grid, 256, 0, st>>>(*t, dim, K, P, n, grad, grad_lin, *opt, step);
}

// ---- Linear scorer on gathered rows ---------------------------------------------------------------------------
template <int V, int G, int IT>
__global__ void __launch_bounds__(256)
linear_rows_kernel(int dim, int B, float inv_batch, const float* __restrict__ u, const float* __restrict__ vp,
                   const float* __restrict__ vn, const float* __restrict__ bu, const float* __restrict__ bip,
                   const float* __restrict__ bin, float* __restrict__ gu, float* __restrict__ gvp,
                   float* __restrict__ gvn, float* __restrict__ gbp, float* __restrict__ gbn,
                   float* __restrict__ loss_part) {
    __shared__ float s_h[8];
    const int nch = dim / V, gl = threadIdx.x % G;
    constexpr int GPW = 32 / G;
    const int gpb = blockDim.x / G;
    const int sub = (threadIdx.x / G) % GPW;
    float hsum = 0.f;
    for (int b0 = blockIdx.x * gpb + threadIdx.x / G - sub; b0 < B; b0 += gridDim.x * gpb) {  // warp-uniform
        const bool valid = b0 + sub < B;
        const int b = valid ? b0 + sub : B - 1;
        const Row<V, IT> ru = load_row<V, G, IT>(u + (size_t)b * dim, nch, gl);
        const Row<V, IT> rp = load_row<V, G, IT>(vp + (size_t)b * dim, nch, gl);
        const Row<V, IT> rn = load_row<V, G, IT>(vn + (size_t)b * dim, nch, gl);
        const float sp = (group_sum<G>(row_dot_partial(ru, rp)) + bu[b]) + bip[b];
        const float sn = (group_sum<G>(row_dot_partial(ru, rn)) + bu[b]) + bin[b];
        const float h = __fadd_rn(__fsub_rn(sn, sp), 1.0f);
        const float g = (h >= 0.f) ? inv_batch : 0.f;
        if (!valid) continue;
        if (gl == 0) hsum += fmaxf(h, 0.f);
        Row<V, IT> du, dp, dn;
#pragma unroll
        for (int a = 0; a < IT; ++a)
#pragma unroll
            for (int k = 0; k < V; ++k) {
                du.c[a][k] = g * (rn.c[a][k] - rp.c[a][k]);
                dp.c[a][k] = -g * ru.c[a][k];
                dn.c[a][k] = g * ru.c[a][k];
            }
        store_row<V, G, IT>(gu + (size_t)b * dim, nch, gl, du);
        store_row<V, G, IT>(gvp + (size_t)b * dim, nch, gl, dp);
        store_row<V, G, IT>(gvn + (size_t)b * dim, nch, gl, dn);
        if (gl == 0) {
            gbp[b] = -g;
            gbn[b] = g;
        }
    }
    hsum = warp_sum(hsum);
    if ((threadIdx.x & 31) == 0) s_h[threadIdx.x >> 5] = hsum;
    __syncthreads();
    if (threadIdx.x == 0) {
        float H = 0.f;
        for (int w = 0; w < 8; ++w) H += s_h[w];
        loss_part[blockIdx.x] = H;
    }
}
__global__ void __launch_bounds__(32)
loss_sum_kernel(const float* __restrict__ part, int n, float scale, float* __restrict__ out) {
    float a = 0.f;
    for (int i = threadIdx.x; i < n; i += 32) a += part[i];
    a = warp_sum(a);
    if (threadIdx.x == 0) out[0] = a * scale;
}

template <int V, int G, int IT>
static void launch_linear_rows(int dim, int B, float inv_batch, const float* u, const float* vp, const float* vn,
                               const float* bu, const float* bip, const float* bin, float* gu, float* gvp, float* gvn,
                               float* gbp, float* gbn, float* loss_part, int grid, cudaStream_t st) {
    linear_rows_kernel<V, G, IT><<<grid, 256, 0, st>>>(dim, B, inv_batch, u, vp, vn, bu, bip, bin, gu, gvp, gvn, gbp,
                                                      gbn, loss_part);
}

// ---- merge of per-shard top-k lists ----------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
topk_merge_kernel(const float* __restrict__ score, const int64_t* __restrict__ idx, int n_lists, int k, int n_query,
                  int64_t* __restrict__ out_idx, float* __restrict__ out_score) {
    extern __shared__ unsigned char sm[];
    const int total = n_lists * k;
    float* s = (float*)sm;
    int64_t* id = (int64_t*)(sm + (((size_t)total * 4 + 7) & ~(size_t)7));
    const int q = blockIdx.x;
    for (int j = threadIdx.x; j < total; j += 128) {  // list l of user q lives at [l][q][k]
        const int l = j / k, r = j % k;
        s[j] = score[((size_t)l * n_query + q) * k + r];
        id[j] = idx[((size_t)l * n_query + q) * k + r];
    }
    __syncthreads();
    for (int j = threadIdx.x; j < total; j += 128) {
        const float sj = s[j];
        const int64_t ij = id[j];
        if (ij < 0) continue;  // padding of a shard with fewer than k items
        int rank = 0;
        for (int o = 0; o < total; ++o) {
            const int64_t io = id[o];
            rank += (io >= 0 && (s[o] > sj || (s[o] == sj && io < ij))) ? 1 : 0;
        }
        if (rank < k) {
            out_idx[(size_t)q * k + rank] = ij;
            out_score[(size_t)q * k + rank] = sj;
        }
    }
}

}  // namespace trs

using namespace trs;

extern "C" size_t trs_sparse_update_workspace_bytes(int64_t n) {
    if (n <= 0) return 256;
    trs_epoch ep = {};
    ep.n_samples = n;
    ep.batch = (int32_t)n;
    return ((size_t)4 * n * sizeof(uint32_t) + 1023) / 256 * 256 + hist_bytes(&ep);
}

extern "C" int trs_sparse_row_update(const trs_table* table, int dim, const int64_t* ids, int64_t n,
                                     const float* grad_rows, const float* grad_lin, const trs_optim* optim, int step,
                                     void* workspace, size_t workspace_bytes, trs_stream_t stream) {
    TRS_REQUIRE(table && table->emb && optim && optim->step_scale, "sparse_row_update: NULL table / optimizer");
    TRS_REQUIRE(n >= 0 && n < (1ll << 30), "sparse_row_update: n out of range");
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(ids && grad_rows && workspace, "sparse_row_update: NULL pointer");
    TRS_REQUIRE(table->n_rows > 0 && table->n_rows <= 0xFFFFFFFFll, "sparse_row_update: n_rows out of range");
    TRS_REQUIRE(optim->kind >= TRS_OPT_SGD && optim->kind <= TRS_OPT_SPARSE_ADAM, "unknown optimizer kind %d", optim->kind);
    if (optim->kind != TRS_OPT_SGD) TRS_REQUIRE(table->emb_s0 && (!grad_lin || !table->lin || table->lin_s0), "optimizer state s0 is NULL");
    if (optim->kind == TRS_OPT_SPARSE_ADAM) TRS_REQUIRE(table->emb_s1 && (!grad_lin || !table->lin || table->lin_s1), "optimizer state s1 is NULL");
    RowShape shape;
    TRS_REQUIRE(pick_row_shape(dim, &shape), "unsupported n_factors %d", dim);
    if (workspace_bytes < trs_sparse_update_workspace_bytes(n)) {
        set_error("sparse_row_update workspace too small");
        return TRS_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    trs_epoch ep = {};
    ep.n_samples = n;
    ep.batch = (int32_t)n;
    uint32_t* key = (uint32_t*)workspace;
    uint32_t* val = key + n;
    uint32_t* tkey = val + n;
    uint32_t* tval = tkey + n;
    uint32_t* hist = (uint32_t*)((char*)workspace + ((size_t)4 * n * sizeof(uint32_t) + 1023) / 256 * 256);
    int rc = sort_space(ids, ids, 1, 0, 1, table->n_rows, &ep, key, val, tkey, tval, hist, st);
    if (rc) return rc;
    const OptScalars os = make_opt_scalars(optim);
    TRS_DISPATCH_ROW_SHAPE(shape, launch_segment_update, table, dim, key, val, (int)n, grad_rows, grad_lin, &os, step, st);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_linear_rows_step(int dim, int64_t batch, float inv_batch, const float* u_rows, const float* pos_rows,
                                    const float* neg_rows, const float* u_bias, const float* pos_bias,
                                    const float* neg_bias, float* g_u, float* g_pos, float* g_neg, float* g_pos_bias,
                                    float* g_neg_bias, float* loss_sum, float* workspace, size_t workspace_floats,
                                    trs_stream_t stream) {
    RowShape shape;
    TRS_REQUIRE(pick_row_shape(dim, &shape), "unsupported n_factors %d", dim);
    TRS_REQUIRE(batch > 0 && batch < (1ll << 30), "linear_rows_step: batch out of range");
    TRS_REQUIRE(u_rows && pos_rows && neg_rows && u_bias && pos_bias && neg_bias && g_u && g_pos && g_neg &&
                g_pos_bias && g_neg_bias && loss_sum && workspace, "linear_rows_step: NULL pointer");
    const int gpb = 256 / shape.G;
    int grid = (int)((batch + gpb - 1) / gpb);
    const int cap = device_props().sm_count * 8;
    if (grid > cap) grid = cap;
    TRS_REQUIRE(workspace_floats >= (size_t)grid, "linear_rows_step: workspace needs %d floats", grid);
    cudaStream_t st = (cudaStream_t)stream;
    TRS_DISPATCH_ROW_SHAPE(shape, launch_linear_rows, dim, (int)batch, inv_batch, u_rows, pos_rows, neg_rows, u_bias,
                           pos_bias, neg_bias, g_u, g_pos, g_neg, g_pos_bias, g_neg_bias, workspace, grid, st);
    loss_sum_kernel<<<1, 32, 0, st>>>(workspace, grid, 1.0f, loss_sum);  // sum of hinges: the caller divides
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_topk_merge(const float* score, const int64_t* idx, int n_lists, int k, int64_t n_query,
                              int64_t* out_idx, float* out_score, trs_stream_t stream) {
    TRS_REQUIRE(score && idx && out_idx && out_score, "topk_merge: NULL pointer");
    TRS_REQUIRE(n_lists >= 1 && k >= 1 && (size_t)n_lists * k * 12 + 8 <= 48 * 1024, "topk_merge: n_lists * k too large");
    if (n_query == 0) return TRS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    TRS_CUDA(cudaMemsetAsync(out_idx, 0xff, (size_t)n_query * k * 8, st));  // -1 where fewer than k items exist
    const size_t smem = (((size_t)n_lists * k * 4 + 7) & ~(size_t)7) + (size_t)n_lists * k * 8;
    topk_merge_kernel<<<(unsigned)n_query, 128, smem, st>>>(score, idx, n_lists, k, (int)n_query, out_idx, out_score);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}
