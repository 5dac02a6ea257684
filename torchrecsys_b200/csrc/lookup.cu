// lookup.cu -- row gather, scorer forward, pairwise evaluation, Philox negatives, id validation.
#include "scorer.cuh"

namespace trs {

static inline int grid_for(int64_t work_items, int items_per_block, int max_blocks) {
    int64_t b = (work_items + items_per_block - 1) / items_per_block;
    if (b < 1) b = 1;
    if (b > max_blocks) b = max_blocks;
    return (int)b;
}

// ---------------------------------------------------------------------------------------
// a1: out[b] = table[idx[b]] + sum_f meta[f][meta_idx[b,f]]
// ---------------------------------------------------------------------------------------
struct MetaPtrs {
    const float* t[TRS_MAX_META];
};

template <int V, int G, int IT>
__global__ void __launch_bounds__(256)
gather_sum_kernel(const float* __restrict__ table, int dim, const int64_t* __restrict__ idx,
                  int64_t n, MetaPtrs metas, const int64_t* __restrict__ meta_idx, int n_meta,
                  float* __restrict__ out) {
    const int nch = dim / V;
    const int gl = threadIdx.x % G;
    const int64_t gpb = blockDim.x / G;
    for (int64_t b = blockIdx.x * gpb + threadIdx.x / G; b < n; b += (int64_t)gridDim.x * gpb) {
        Row<V, IT> r = load_row<V, G, IT>(table + (size_t)idx[b] * dim, nch, gl);
        for (int f = 0; f < n_meta; ++f) {
            int64_t mi = meta_idx[b * n_meta + f];
            Row<V, IT> mrow = load_row<V, G, IT>(metas.t[f] + (size_t)mi * dim, nch, gl);
#pragma unroll
            for (int i = 0; i < IT; ++i)
#pragma unroll
                for (int k = 0; k < V; ++k) r.c[i][k] = __fadd_rn(r.c[i][k], mrow.c[i][k]);
        }
        store_row<V, G, IT>(out + (size_t)b * dim, nch, gl, r);
    }
}

template <int V, int G, int IT>
static void launch_gather(const float* table, int dim, const int64_t* idx, int64_t n,
                          MetaPtrs metas, const int64_t* meta_idx, int n_meta, float* out,
                          cudaStream_t st) {
    int grid = grid_for(n, 256 / G, device_props().sm_count * 16);
    gather_sum_kernel<V, G, IT><<<grid, 256, 0, st>>>(table, dim, idx, n, metas, meta_idx, n_meta, out);
}

// ---------------------------------------------------------------------------------------
// a2/a3: scores
// ---------------------------------------------------------------------------------------

template <int NET, int V, int G, int IT>
__global__ void __launch_bounds__(256)
scores_kernel(trs_model m, const int64_t* __restrict__ user, const int64_t* __restrict__ item,
              const int64_t* __restrict__ meta, int64_t n, float* __restrict__ out) {
    const int nch = m.dim / V;
    const int gl = threadIdx.x % G;
    constexpr int GPW = 32 / G;
    const int64_t gpb = blockDim.x / G;
    const int sub = (threadIdx.x / G) % GPW;  // my group inside the warp
    // warp-uniform trip count: group_sum shuffles need every lane of the warp
    for (int64_t b0 = blockIdx.x * gpb + threadIdx.x / G - sub; b0 < n; b0 += (int64_t)gridDim.x * gpb) {
        const bool valid = b0 + sub < n;
        const int64_t b = valid ? b0 + sub : n - 1;
        float s = score_one<NET, V, G, IT>(m, nch, gl, user[b], item[b],
                                           meta ? meta + b * m.n_meta : nullptr);
        if (gl == 0 && valid) out[b] = s;
    }
}

template <int V, int G, int IT>
static void launch_scores(const trs_model* m, const int64_t* user, const int64_t* item,
                          const int64_t* meta, int64_t n, float* out, cudaStream_t st) {
    int grid = grid_for(n, 256 / G, device_props().sm_count * 16);
    if (m->net == TRS_NET_LINEAR)
        scores_kernel<TRS_NET_LINEAR, V, G, IT><<<grid, 256, 0, st>>>(*m, user, item, meta, n, out);
    else
        scores_kernel<TRS_NET_FM, V, G, IT><<<grid, 256, 0, st>>>(*m, user, item, meta, n, out);
}

// ---------------------------------------------------------------------------------------
// a10: per-batch hinge mean and pairwise "auc"; one CTA walks whole batches
// ---------------------------------------------------------------------------------------
template <int NET, int V, int G, int IT>
__global__ void __launch_bounds__(256)
eval_kernel(trs_model m, trs_epoch ep, float* __restrict__ loss, float* __restrict__ auc,
            float* __restrict__ pos_out, float* __restrict__ neg_out) {
    __shared__ float s_h[8];
    __shared__ int s_c[8];
    const int nch = m.dim / V;
    const int gl = threadIdx.x % G;
    const int gpb = blockDim.x / G;
    const int64_t nb = (ep.n_samples + ep.batch - 1) / ep.batch;
    for (int64_t bt = blockIdx.x; bt < nb; bt += gridDim.x) {
        const int64_t lo = bt * ep.batch;
        const int64_t hi = min(lo + (int64_t)ep.batch, ep.n_samples);
        float hs = 0.f;
        int cnt = 0;
        constexpr int GPW = 32 / G;
        const int sub = (threadIdx.x / G) % GPW;
        for (int64_t b0 = lo + threadIdx.x / G - sub; b0 < hi; b0 += gpb) {  // warp-uniform
            const bool valid = b0 + sub < hi;
            const int64_t b = valid ? b0 + sub : hi - 1;
            int64_t u = ep.user[b];
            float sp = score_one<NET, V, G, IT>(m, nch, gl, u, ep.pos[b],
                                                ep.pos_meta ? ep.pos_meta + b * m.n_meta : nullptr);
            float sn = score_one<NET, V, G, IT>(m, nch, gl, u, ep.neg[b],
                                                ep.neg_meta ? ep.neg_meta + b * m.n_meta : nullptr);
            if (gl == 0 && valid) {
                hs += fmaxf(__fadd_rn(__fsub_rn(sn, sp), 1.0f), 0.f);
                cnt += sp > sn;
                if (pos_out) pos_out[b] = sp;
                if (neg_out) neg_out[b] = sn;
            }
        }
        hs = warp_sum(hs);
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if ((threadIdx.x & 31) == 0) {
            s_h[threadIdx.x >> 5] = hs;
            s_c[threadIdx.x >> 5] = cnt;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float H = 0.f;
            int C = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
                H += s_h[w];
                C += s_c[w];
            }
            const float len = (float)(hi - lo);
            if (loss) loss[bt] = H / len;
            if (auc) auc[bt] = (float)C / len;
        }
        __syncthreads();
    }
}

template <int V, int G, int IT>
static void launch_eval(const trs_model* m, const trs_epoch* ep, float* loss, float* auc,
                        float* pos_out, float* neg_out, cudaStream_t st) {
    int64_t nb = n_steps_of(ep);
    int grid = (int)(nb < (int64_t)device_props().sm_count * 4 ? nb : device_props().sm_count * 4);
    if (grid < 1) grid = 1;
    if (m->net == TRS_NET_LINEAR)
        eval_kernel<TRS_NET_LINEAR, V, G, IT><<<grid, 256, 0, st>>>(*m, *ep, loss, auc, pos_out, neg_out);
    else
        eval_kernel<TRS_NET_FM, V, G, IT><<<grid, 256, 0, st>>>(*m, *ep, loss, auc, pos_out, neg_out);
}

// ---------------------------------------------------------------------------------------
// a9: Philox4x32-10 negatives
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
philox_neg_kernel(uint64_t seed, uint64_t first, const int64_t* __restrict__ pos, int64_t n,
                  int64_t n_items, const int64_t* __restrict__ item_meta, int n_meta,
                  int64_t* __restrict__ neg, int64_t* __restrict__ neg_meta) {
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n;
         j += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t idx = first + (uint64_t)j;
        const int64_t p = pos[j];
        int64_t pick = -1;
        for (uint32_t block = 0; pick < 0; ++block) {
            uint32_t c[4] = {(uint32_t)idx, (uint32_t)(idx >> 32), block, 0u};
            philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                int64_t cand = (int64_t)(((uint64_t)c[w] * (uint64_t)n_items) >> 32);
                if (pick < 0 && cand != p) pick = cand;
            }
        }
        neg[j] = pick;
        if (neg_meta)
            for (int f = 0; f < n_meta; ++f) neg_meta[j * n_meta + f] = item_meta[pick * n_meta + f];
    }
}

__global__ void __launch_bounds__(256)
validate_ids_kernel(const int64_t* __restrict__ ids, int64_t n, int64_t n_rows, int32_t* bad) {
    int local = 0;
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n;
         j += (int64_t)gridDim.x * blockDim.x) {
        int64_t v = ids[j];
        local += (v < 0 || v >= n_rows);
    }
    local = __reduce_add_sync(0xffffffffu, local);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(bad, local);
}

}  // namespace trs

using namespace trs;

extern "C" int trs_device_info(int* sm_count_host, int* train_grid_host, int* train_block_host);

extern "C" int trs_embed_gather_sum(const float* table, int dim, const int64_t* idx, int64_t n,
                                    const float* const* meta_tables_host, const int64_t* meta_idx,
                                    int n_meta, float* out, trs_stream_t stream) {
    RowShape shape;
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(table && idx && out, "NULL pointer");
    TRS_REQUIRE(n_meta >= 0 && n_meta <= TRS_MAX_META, "n_meta %d out of range", n_meta);
    TRS_REQUIRE(n_meta == 0 || (meta_tables_host && meta_idx), "metadata pointers missing");
    TRS_REQUIRE(pick_row_shape(dim, &shape), "unsupported dim %d", dim);
    MetaPtrs mp = {};
    for (int f = 0; f < n_meta; ++f) mp.t[f] = meta_tables_host[f];
    TRS_DISPATCH_ROW_SHAPE(shape, launch_gather, table, dim, idx, n, mp, meta_idx, n_meta, out, stream);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_scores(const trs_model* model, const int64_t* user, const int64_t* item,
                          const int64_t* meta, int64_t n, float* out, trs_stream_t stream) {
    RowShape shape;
    int rc = check_model(model, &shape);
    if (rc) return rc;
    TRS_REQUIRE(model->net != TRS_NET_MLP, "trs_scores: use trs_mlp_forward for net_type mlp");
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(user && item && out, "NULL pointer");
    TRS_REQUIRE(model->n_meta == 0 || meta, "model has metadata tables but meta ids are NULL");
    TRS_DISPATCH_ROW_SHAPE(shape, launch_scores, model, user, item, meta, n, out, stream);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_eval_pairwise(const trs_model* model, const trs_epoch* epoch, float* loss,
                                 float* auc, float* pos_out, float* neg_out, trs_stream_t stream) {
    RowShape shape;
    int rc = check_model(model, &shape);
    if (rc) return rc;
    TRS_REQUIRE(model->net != TRS_NET_MLP, "trs_eval_pairwise: score the tower with trs_mlp_forward");
    TRS_REQUIRE(epoch, "epoch is NULL");
    if (epoch->n_samples == 0) return TRS_OK;
    TRS_REQUIRE(epoch->user && epoch->pos && epoch->neg, "epoch ids are NULL");
    TRS_REQUIRE(epoch->batch > 0, "batch must be positive");
    TRS_REQUIRE(model->n_meta == 0 || (epoch->pos_meta && epoch->neg_meta), "metadata ids are NULL");
    TRS_DISPATCH_ROW_SHAPE(shape, launch_eval, model, epoch, loss, auc, pos_out, neg_out, stream);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_philox_negatives(uint64_t seed, uint64_t first_index, const int64_t* pos,
                                    int64_t n, int64_t n_items, const int64_t* item_meta,
                                    int n_meta, int64_t* neg, int64_t* neg_meta,
                                    trs_stream_t stream) {
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(pos && neg, "NULL pointer");
    TRS_REQUIRE(n_items >= 2 && n_items <= 0xFFFFFFFFll, "n_items must be in [2, 2^32)");
    TRS_REQUIRE(!neg_meta || (item_meta && n_meta > 0), "neg_meta needs item_meta");
    if (n == 0) return TRS_OK;
    int grid = grid_for(n, 256, device_props().sm_count * 8);
    philox_neg_kernel<<<grid, 256, 0, stream>>>(seed, first_index, pos, n, n_items, item_meta,
                                                n_meta, neg, neg_meta);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_validate_ids(const int64_t* ids, int64_t n, int64_t n_rows, int32_t* bad_count,
                                trs_stream_t stream) {
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(ids && bad_count, "NULL pointer");
    int grid = grid_for(n, 256, device_props().sm_count * 8);
    validate_ids_kernel<<<grid, 256, 0, stream>>>(ids, n, n_rows, bad_count);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}
