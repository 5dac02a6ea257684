// shard_serve.cu -- evaluation and row lookups on the row-sharded tables where they live (trs_shard, csrc/shard.cu).
// Row r of a table is read from its owner, rank r % world at local row r / world, through the pointers of the
// trs_shard -- peer mappings in a real group -- so nothing is gathered onto one GPU first.
//   * trs_shard_eval_pairwise: trs_eval_pairwise (csrc/lookup.cu: eval_kernel) for a range of batches of the global
//     epoch, bit-identical to it on the gathered model: the same row shape, CTA per batch, warp-uniform sample loop,
//     score association (linear_score's) and reduction order.
//   * trs_shard_gather_rows: bit copies of the rows (and biases) of global ids.
#include "scorer.cuh"

namespace trs {

// (owner, local row) of a global id.  Ids are below 2^32 on this path (check_shard), so the divide is a 32-bit one;
// a group of one needs none.
template <bool ONE>
__device__ __forceinline__ void shard_split(int64_t id, uint32_t world, uint32_t& q, uint32_t& local) {
    if (ONE) {
        q = 0u;
        local = (uint32_t)id;
    } else {
        q = (uint32_t)id % world;
        local = (uint32_t)id / world;
    }
}

// scorer.cuh: linear_score's arithmetic on rows read here: (<u, v> + b_u) + b_i, the dot product reduced over the
// group.  A local copy: factoring this out of linear_score changed the SASS of six existing eval / top-k kernels.
template <int V, int G, int IT>
__device__ __forceinline__ float linear_row_score(const Row<V, IT>& ru, float bu, const Row<V, IT>& v,
                                                  const float* item_lin, uint32_t item_row) {
    const float dot = group_sum<G>(row_dot_partial(ru, v));
    const float bi = item_lin ? item_lin[item_row] : 0.f;
    return (dot + bu) + bi;
}

// the row of global id `id` of the table whose shards are t[0 .. world); its bias is lin[local] (lin may be NULL)
template <bool ONE, int V, int G, int IT>
__device__ __forceinline__ Row<V, IT> shard_row(const trs_table* t, int64_t id, uint32_t world, int dim, int nch,
                                                int gl, const float*& lin, uint32_t& local) {
    uint32_t q;
    shard_split<ONE>(id, world, q, local);
    lin = t[q].lin;
    return load_row<V, G, IT>(t[q].emb + (size_t)local * dim, nch, gl);
}

// batches [first, first + nbr) of the global epoch; one CTA walks whole batches, outputs relative to the range
template <bool ONE, int V, int G, int IT>
__global__ void __launch_bounds__(256)
shard_eval_kernel(const __grid_constant__ trs_shard sh, const __grid_constant__ trs_epoch ep, int64_t first,
                  int64_t nbr, float* __restrict__ loss, float* __restrict__ auc, float* __restrict__ pos_out,
                  float* __restrict__ neg_out) {
    __shared__ float s_h[8];
    __shared__ int s_c[8];
    const int dim = sh.dim;
    const int nch = dim / V;
    const int gl = threadIdx.x % G;
    const int gpb = blockDim.x / G;
    const uint32_t W = (uint32_t)sh.world;
    const int64_t s0 = first * ep.batch;
    for (int64_t r = blockIdx.x; r < nbr; r += gridDim.x) {
        const int64_t lo = (first + r) * ep.batch;
        const int64_t hi = min(lo + (int64_t)ep.batch, ep.n_samples);
        float hs = 0.f;
        int cnt = 0;
        constexpr int GPW = 32 / G;
        const int sub = (threadIdx.x / G) % GPW;
        for (int64_t b0 = lo + threadIdx.x / G - sub; b0 < hi; b0 += gpb) {  // warp-uniform
            const bool valid = b0 + sub < hi;
            const int64_t b = valid ? b0 + sub : hi - 1;
            const float *lu, *lp, *ln;
            uint32_t ru_at, rp_at, rn_at;
            const Row<V, IT> ru = shard_row<ONE, V, G, IT>(sh.user, ep.user[b], W, dim, nch, gl, lu, ru_at);
            const float bu = lu ? lu[ru_at] : 0.f;
            const Row<V, IT> rp = shard_row<ONE, V, G, IT>(sh.item, ep.pos[b], W, dim, nch, gl, lp, rp_at);
            const float sp = linear_row_score<V, G, IT>(ru, bu, rp, lp, rp_at);
            const Row<V, IT> rn = shard_row<ONE, V, G, IT>(sh.item, ep.neg[b], W, dim, nch, gl, ln, rn_at);
            const float sn = linear_row_score<V, G, IT>(ru, bu, rn, ln, rn_at);
            if (gl == 0 && valid) {
                hs += fmaxf(__fadd_rn(__fsub_rn(sn, sp), 1.0f), 0.f);
                cnt += sp > sn;
                if (pos_out) pos_out[b - s0] = sp;
                if (neg_out) neg_out[b - s0] = sn;
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
            if (loss) loss[r] = H / len;
            if (auc) auc[r] = (float)C / len;
        }
        __syncthreads();
    }
}

template <bool ONE, int V, int G, int IT>
__global__ void __launch_bounds__(256)
shard_gather_kernel(const __grid_constant__ trs_shard sh, int table, const int64_t* __restrict__ ids, int64_t n,
                    float* __restrict__ emb_out, float* __restrict__ lin_out) {
    const trs_table* t = table ? sh.item : sh.user;
    const int dim = sh.dim;
    const int nch = dim / V;
    const int gl = threadIdx.x % G;
    const int64_t gpb = blockDim.x / G;
    for (int64_t j = blockIdx.x * gpb + threadIdx.x / G; j < n; j += (int64_t)gridDim.x * gpb) {
        const float* lin;
        uint32_t local;
        const Row<V, IT> r = shard_row<ONE, V, G, IT>(t, ids[j], (uint32_t)sh.world, dim, nch, gl, lin, local);
        store_row<V, G, IT>(emb_out + (size_t)j * dim, nch, gl, r);
        if (lin_out && gl == 0) lin_out[j] = lin ? lin[local] : 0.f;
    }
}

template <int V, int G, int IT>
static void launch_shard_eval(const trs_shard* sh, const trs_epoch* ep, int64_t first, int64_t nbr, float* loss,
                              float* auc, float* pos_out, float* neg_out, cudaStream_t st) {
    const int64_t cap = (int64_t)device_props().sm_count * 4;  // trs_eval_pairwise's grid
    const int grid = (int)(nbr < cap ? nbr : cap);
    if (sh->world == 1)
        shard_eval_kernel<true, V, G, IT><<<grid, 256, 0, st>>>(*sh, *ep, first, nbr, loss, auc, pos_out, neg_out);
    else
        shard_eval_kernel<false, V, G, IT><<<grid, 256, 0, st>>>(*sh, *ep, first, nbr, loss, auc, pos_out, neg_out);
}

template <int V, int G, int IT>
static void launch_shard_gather(const trs_shard* sh, int table, const int64_t* ids, int64_t n, float* emb_out,
                                float* lin_out, cudaStream_t st) {
    const int64_t gpb = 256 / G, cap = (int64_t)device_props().sm_count * 16;
    const int64_t want = (n + gpb - 1) / gpb;
    const int grid = (int)(want < cap ? want : cap);
    if (sh->world == 1)
        shard_gather_kernel<true, V, G, IT><<<grid, 256, 0, st>>>(*sh, table, ids, n, emb_out, lin_out);
    else
        shard_gather_kernel<false, V, G, IT><<<grid, 256, 0, st>>>(*sh, table, ids, n, emb_out, lin_out);
}

// every rank's row pointers are set (the bias tables are optional, as in trs_model)
static int check_shard_rows(const trs_shard* sh) {
    for (int q = 0; q < sh->world; ++q)
        TRS_REQUIRE(sh->user[q].emb && sh->item[q].emb, "rank %d's user / item shard is NULL", q);
    return TRS_OK;
}

}  // namespace trs

using namespace trs;

extern "C" int trs_shard_eval_pairwise(const trs_shard* shard, const trs_epoch* epoch, int64_t first_batch,
                                       int64_t n_batches, float* loss, float* auc, float* pos_out, float* neg_out,
                                       trs_stream_t stream) {
    RowShape shape;
    int rc = check_shard(shard, &shape);
    if (rc) return rc;
    TRS_REQUIRE(epoch, "epoch is NULL");
    TRS_REQUIRE(epoch->batch > 0, "batch must be positive");
    TRS_REQUIRE(epoch->pos_meta == nullptr && epoch->neg_meta == nullptr, "row-sharded evaluation does not take metadata");
    const int64_t nb = n_steps_of(epoch);
    TRS_REQUIRE(first_batch >= 0 && n_batches >= 0 && first_batch + n_batches <= nb,
                "batches [%lld, %lld) outside the epoch's %lld", (long long)first_batch,
                (long long)(first_batch + n_batches), (long long)nb);
    if (n_batches == 0) return TRS_OK;
    TRS_REQUIRE(epoch->user && epoch->pos && epoch->neg, "epoch ids are NULL");
    if ((rc = check_shard_rows(shard))) return rc;
    TRS_DISPATCH_ROW_SHAPE(shape, launch_shard_eval, shard, epoch, first_batch, n_batches, loss, auc, pos_out, neg_out,
                           (cudaStream_t)stream);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

extern "C" int trs_shard_gather_rows(const trs_shard* shard, int table, const int64_t* ids, int64_t n, float* emb_out,
                                     float* lin_out, trs_stream_t stream) {
    RowShape shape;
    int rc = check_shard(shard, &shape);
    if (rc) return rc;
    TRS_REQUIRE(table == 0 || table == 1, "table must be 0 (user) or 1 (item), got %d", table);
    TRS_REQUIRE(n >= 0, "negative id count");
    if (n == 0) return TRS_OK;
    TRS_REQUIRE(ids && emb_out, "NULL pointer");
    if ((rc = check_shard_rows(shard))) return rc;
    TRS_DISPATCH_ROW_SHAPE(shape, launch_shard_gather, shard, table, ids, n, emb_out, lin_out, (cudaStream_t)stream);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}
