// gemm.cu -- C[M,N] = A[M,K] * B[N,K]^T on the 5th-generation tensor cores (tcgen05.mma, bf16 in,
// fp32 accumulate in TMEM), operands staged by TMA through a 128B-swizzled shared-memory ring.
//
// This is the dense contraction of the MLP tower (reference collaborative/mlp.py:107-113: nn.Linear
// forward, and its dgrad / wgrad in backward; SURVEY.md K7).  Every GEMM of the tower is brought to
// this one "TN" form (both operands contiguous along the reduction dimension):
//   forward   Z[rows, out]   = A[rows, in]    * W[out, in]^T          (+ bias, + BatchNorm column partials)
//   dgrad     dA[rows, in]   = dZ[rows, out]  * Wt[in, out]^T
//   wgrad     dW[out, in]    = dZt[out, rows] * At[in, rows]^T        (split-K over rows)
//
// One CTA computes one 128 x BN output tile (x one K split).  Warp roles (192 threads):
//   warp 0      TMA producer   (one elected lane): fills the STAGES-deep ring, waits on empty[]
//   warp 1      MMA issuer     (one elected lane): tcgen05.mma per 16-wide K slice, commit -> empty[]
//               also allocates / frees the TMEM accumulator (BN columns x 128 lanes)
//   warps 2-5   epilogue: tcgen05.ld of their 32-lane quadrant, bias, column statistics, stores
#include "tc.cuh"

namespace trs {

constexpr int GEMM_BM = 128, GEMM_BK = 64;
constexpr int GEMM_THREADS = 192;

struct GemmDev {
    int M, N, K;
    int kb_per_split;       // 64-wide K blocks per split (gridDim.z splits)
    void* out;              // fp32 or bf16, row-major, leading dimension ldc
    long long ldc;
    long long split_stride; // elements between the partial outputs of consecutive splits
    const float* bias;      // [N] or null
    float* col_sum;         // [ceil(M/128), N] or null: per-row-tile column sums of the output ...
    float* col_sumsq;       // ... and of its squares, over valid rows only
    int rows_per_half;      // a row m is valid iff m < M and (m % rows_per_half) < rows_valid
    int rows_valid;
};

template <int BN, int STAGES>
struct GemmSmem {
    static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;
    static constexpr int B_BYTES = BN * GEMM_BK * 2;
    static constexpr int RING = STAGES * (A_BYTES + B_BYTES);
    static constexpr int STAT = 2 * 4 * BN * 4;  // [2 kinds][4 quadrants][BN] floats
    static constexpr int TOTAL = 1024 /* alignment slack */ + RING + STAT + 8 * (2 * STAGES + 1) + 16;
};

// butterfly transpose-reduce: in: a[j] = this lane's (row's) value of column j; out: a[0] of lane l =
// sum over the 32 lanes of column l.  31 shuffles, fixed association.
__device__ __forceinline__ void column_sums_32(float (&a)[32], int lane) {
#pragma unroll
    for (int W = 16; W >= 1; W >>= 1) {
        const bool hi = (lane & W) != 0;
#pragma unroll
        for (int i = 0; i < W; ++i) {
            const float send = hi ? a[i] : a[i + W];
            const float keep = hi ? a[i + W] : a[i];
            a[i] = keep + __shfl_xor_sync(0xffffffffu, send, W);
        }
    }
}

// A_MN / B_MN: the operand is stored [k, mn] (mn contiguous, "MN-major") instead of [mn, k].  Its tile
// is then loaded as 64-column boxes of BK rows (row = one k, 128 bytes = 64 mn); boxes of consecutive
// 64-mn blocks lie BK*128 bytes apart (the descriptor's leading byte offset), 8-k groups 1024 bytes
// apart (stride byte offset), and a 16-wide K slice starts 16 rows = 2048 bytes further.
template <int BN, int STAGES, bool OUT_BF16, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ GemmDev g) {
    using S = GemmSmem<BN, STAGES>;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* sA = base;
    unsigned char* sB = base + STAGES * S::A_BYTES;
    float* s_stat = (float*)(base + S::RING);
    uint64_t* full = (uint64_t*)(base + S::RING + S::STAT);
    uint64_t* empty = full + STAGES;
    uint64_t* acc_full = empty + STAGES;
    uint32_t* tmem_slot = (uint32_t*)(acc_full + 1);

    constexpr int ST_ELEM = OUT_BF16 ? 2 : 4;          // output element size
    constexpr int ST_PITCH = BN * ST_ELEM + 16;         // staged row pitch in bytes
    static_assert(GEMM_BM * ST_PITCH <= S::RING, "the output tile is staged in the operand ring");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * GEMM_BM, n0 = blockIdx.y * BN;
    const int nkb_total = (g.K + GEMM_BK - 1) / GEMM_BK;
    const int kb0 = blockIdx.z * g.kb_per_split;
    const int nkb = min(g.kb_per_split, nkb_total - kb0);

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmap_a);
        tc::tma_prefetch_desc(&tmap_b);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(acc_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_slot, BN);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_acc = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
                mbar_wait(&empty[s], ph ^ 1u);
                mbar_arrive_expect_tx(&full[s], S::A_BYTES + S::B_BYTES);
                const int k = (kb0 + kb) * GEMM_BK;
                if (A_MN) {
#pragma unroll
                    for (int b = 0; b < GEMM_BM / 64; ++b)
                        tc::tma_load_2d(sA + s * S::A_BYTES + b * (GEMM_BK * 128), &tmap_a, &full[s], m0 + 64 * b, k);
                } else {
                    tc::tma_load_2d(sA + s * S::A_BYTES, &tmap_a, &full[s], k, m0);
                }
                if (B_MN) {
#pragma unroll
                    for (int b = 0; b < BN / 64; ++b)
                        tc::tma_load_2d(sB + s * S::B_BYTES + b * (GEMM_BK * 128), &tmap_b, &full[s], n0 + 64 * b, k);
                } else {
                    tc::tma_load_2d(sB + s * S::B_BYTES, &tmap_b, &full[s], k, n0);
                }
            }
        }
    } else if (warp == 1) {
        // the whole warp walks the k blocks (uniform control flow), one elected lane issues the MMAs
        constexpr uint32_t idesc = tc::idesc_bf16_f32(GEMM_BM, BN) | (A_MN ? (1u << 15) : 0u) | (B_MN ? (1u << 16) : 0u);
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
            mbar_wait(&full[s], ph);
            tc::tc_fence_after();
            if (tc::elect_one()) {
#pragma unroll
                for (int k = 0; k < GEMM_BK / 16; ++k) {
                    const uint64_t da = A_MN ? tc::smem_desc_sw128_mn(sA + s * S::A_BYTES + k * 2048, GEMM_BK * 128)
                                             : tc::smem_desc_sw128(sA + s * S::A_BYTES, k * 16);
                    const uint64_t db = B_MN ? tc::smem_desc_sw128_mn(sB + s * S::B_BYTES + k * 2048, GEMM_BK * 128)
                                             : tc::smem_desc_sw128(sB + s * S::B_BYTES, k * 16);
                    tc::umma_bf16(tmem_acc, da, db, idesc, (kb | k) ? 1u : 0u);
                }
                tc::umma_commit(&empty[s]);  // frees the ring slot once these MMAs have read it
            }
            __syncwarp();
        }
        if (tc::elect_one()) tc::umma_commit(acc_full);  // accumulator complete
        __syncwarp();
    } else {
        // ---- epilogue: quadrant q of the accumulator = TMEM lanes [32q, 32q+32) = tile rows ----
        const int q = warp & 3;
        const int row = m0 + q * 32 + lane;
        const bool row_in = row < g.M;
        const bool row_valid = row_in && (row % g.rows_per_half) < g.rows_valid;
        const bool stats = g.col_sum != nullptr;
        if (nkb > 0) {
            mbar_wait(acc_full, 0);
            tc::tc_fence_after();
        }
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
            const int col0 = n0 + c * 32;
            if (col0 >= g.N) break;
            uint32_t r[32];
            if (nkb > 0) {
                tc::tmem_ld_32x32(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), r);
                tc::tmem_ld_wait();
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) r[j] = 0u;
            }
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {  // N % 8 == 0 and bias is a tensor base: 16-byte aligned
                float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g.bias && col0 + j < g.N) b = __ldg(reinterpret_cast<const float4*>(g.bias + col0 + j));
                v[j + 0] = __uint_as_float(r[j + 0]) + b.x;
                v[j + 1] = __uint_as_float(r[j + 1]) + b.y;
                v[j + 2] = __uint_as_float(r[j + 2]) + b.z;
                v[j + 3] = __uint_as_float(r[j + 3]) + b.w;
            }
            // The tile goes through shared memory so that global stores are whole rows (one 16-byte piece per
            // lane, 256-512 contiguous bytes per row) instead of 32 scattered 16-byte pieces per instruction.
            // The staging area is the operand ring: every MMA has read it by the time acc_full fired.  Each
            // warp stages and later writes only its own 32 rows; pitch = row bytes + 16 keeps the per-row
            // 16-byte shared-memory stores of a quarter-warp on distinct banks.
            {
                unsigned char* srow = base + (size_t)(q * 32 + lane) * ST_PITCH + (size_t)c * 32 * ST_ELEM;
                if (OUT_BF16) {
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        uint4 pk;
                        __nv_bfloat162 t;
                        t = __floats2bfloat162_rn(v[j + 0], v[j + 1]); pk.x = *reinterpret_cast<uint32_t*>(&t);
                        t = __floats2bfloat162_rn(v[j + 2], v[j + 3]); pk.y = *reinterpret_cast<uint32_t*>(&t);
                        t = __floats2bfloat162_rn(v[j + 4], v[j + 5]); pk.z = *reinterpret_cast<uint32_t*>(&t);
                        t = __floats2bfloat162_rn(v[j + 6], v[j + 7]); pk.w = *reinterpret_cast<uint32_t*>(&t);
                        *reinterpret_cast<uint4*>(srow + j * 2) = pk;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; j += 4)
                        *reinterpret_cast<float4*>(srow + j * 4) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                }
            }
            if (stats) {
                float a[32], b[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    // statistics of the value the next kernel will read back (bf16-rounded when OUT_BF16)
                    const float x = OUT_BF16 ? __bfloat162float(__float2bfloat16_rn(v[j])) : v[j];
                    a[j] = row_valid ? x : 0.f;
                    b[j] = a[j] * a[j];
                }
                column_sums_32(a, lane);
                column_sums_32(b, lane);
                s_stat[(0 * 4 + q) * BN + c * 32 + lane] = a[0];
                s_stat[(1 * 4 + q) * BN + c * 32 + lane] = b[0];
            }
        }
        {   // this warp's 32 staged rows -> global memory, whole rows at a time
            __syncwarp();
            constexpr int LANES_PER_ROW = (BN * ST_ELEM) / 16;      // 16-byte pieces per tile row (8 .. 32)
            constexpr int ROWS_PER_IT = 32 / LANES_PER_ROW;
            const int piece = lane % LANES_PER_ROW;
            const int col = n0 + piece * (16 / ST_ELEM);             // first output column of my piece
            unsigned char* gout = (unsigned char*)g.out + (size_t)blockIdx.z * g.split_stride * ST_ELEM;
#pragma unroll 4
            for (int r0 = 0; r0 < 32; r0 += ROWS_PER_IT) {
                const int rl = q * 32 + r0 + lane / LANES_PER_ROW;
                const int grow = m0 + rl;
                if (grow < g.M && col < g.N) {
                    const uint4 pk = *reinterpret_cast<const uint4*>(base + (size_t)rl * ST_PITCH + (size_t)piece * 16);
                    *reinterpret_cast<uint4*>(gout + ((size_t)grow * g.ldc + col) * ST_ELEM) = pk;
                }
            }
        }
        if (stats) {
            asm volatile("bar.sync 1, 128;" ::: "memory");  // the four epilogue warps only
            const int t = threadIdx.x - 64;                  // 0..127
            for (int col = t; col < BN; col += 128) {
                if (n0 + col < g.N) {
                    float s = 0.f, ss = 0.f;
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) {  // fixed order: deterministic
                        s += s_stat[(0 * 4 + qq) * BN + col];
                        ss += s_stat[(1 * 4 + qq) * BN + col];
                    }
                    g.col_sum[(size_t)blockIdx.x * g.N + n0 + col] = s;
                    g.col_sumsq[(size_t)blockIdx.x * g.N + n0 + col] = ss;
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_acc, BN);
    }
}

// ---- host -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int64_t ld_elems, int box_rows) {
    // box = [box_rows, 64 columns]: K-major operands use box_rows = tile extent, MN-major ones box_rows = BK
    EncodeTiledFn fn = encode_fn();
    TRS_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
    TRS_REQUIRE(((uintptr_t)base & 15) == 0 && (ld_elems * 2) % 16 == 0,
                "bf16 GEMM operand must be 16-byte aligned with a leading dimension that is a multiple of 8");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld_elems * 2};
    cuuint32_t box[2] = {(cuuint32_t)GEMM_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld cols %lld ld %lld)", (int)r,
                  (long long)rows, (long long)cols, (long long)ld_elems);
        return TRS_ERR_CUDA;
    }
    return TRS_OK;
}

template <int BN, int STAGES, bool OUT_BF16, bool A_MN, bool B_MN>
static int launch_gemm(const trs_gemm_args* a, const GemmDev& g, int splits, cudaStream_t stream) {
    CUtensorMap ta, tb;
    int rc;
    if (A_MN) rc = make_tmap_bf16(&ta, a->a, a->k, a->m, a->lda, GEMM_BK);
    else rc = make_tmap_bf16(&ta, a->a, a->m, a->k, a->lda, GEMM_BM);
    if (rc) return rc;
    if (B_MN) rc = make_tmap_bf16(&tb, a->b, a->k, a->n, a->ldb, GEMM_BK);
    else rc = make_tmap_bf16(&tb, a->b, a->n, a->k, a->ldb, BN);
    if (rc) return rc;
    auto kern = gemm_tn_kernel<BN, STAGES, OUT_BF16, A_MN, B_MN>;
    constexpr int smem = GemmSmem<BN, STAGES>::TOTAL;
    TRS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    dim3 grid((unsigned)((a->m + GEMM_BM - 1) / GEMM_BM), (unsigned)((a->n + BN - 1) / BN), (unsigned)splits);
    kern<<<grid, GEMM_THREADS, smem, stream>>>(ta, tb, g);
    TRS_CUDA(cudaGetLastError());
    return TRS_OK;
}

}  // namespace trs

using namespace trs;

extern "C" int trs_gemm_bf16_tn(const trs_gemm_args* a, trs_stream_t stream) {
    TRS_REQUIRE(a && a->a && a->b && a->out, "gemm: NULL operand");
    TRS_REQUIRE(a->m > 0 && a->n > 0 && a->k > 0, "gemm: empty problem %lld x %lld x %lld", (long long)a->m,
                (long long)a->n, (long long)a->k);
    TRS_REQUIRE(a->m < (1ll << 31) && a->n < (1ll << 31) && a->k < (1ll << 31), "gemm: dimension too large");
    TRS_REQUIRE(a->k % 8 == 0 && a->n % 8 == 0, "gemm: K and N must be multiples of 8 (got K %lld, N %lld)",
                (long long)a->k, (long long)a->n);
    TRS_REQUIRE(a->ldc % 8 == 0, "gemm: ldc must be a multiple of 8");
    const int splits = a->splits > 0 ? a->splits : 1;
    TRS_REQUIRE(splits == 1 || (!a->out_bf16 && !a->bias && !a->col_sum),
                "gemm: split-K writes raw fp32 partials only");
    TRS_REQUIRE((a->col_sum == nullptr) == (a->col_sumsq == nullptr), "gemm: col_sum and col_sumsq go together");
    const int nkb = (int)((a->k + GEMM_BK - 1) / GEMM_BK);
    GemmDev g;
    g.M = (int)a->m;
    g.N = (int)a->n;
    g.K = (int)a->k;
    g.kb_per_split = (nkb + splits - 1) / splits;
    g.out = a->out;
    g.ldc = a->ldc;
    g.split_stride = a->split_stride;
    g.bias = a->bias;
    g.col_sum = a->col_sum;
    g.col_sumsq = a->col_sumsq;
    g.rows_per_half = a->rows_per_half > 0 ? (int)a->rows_per_half : (int)a->m;
    g.rows_valid = a->rows_per_half > 0 ? (int)a->rows_valid : (int)a->m;
    cudaStream_t s = (cudaStream_t)stream;
    TRS_REQUIRE(!(a->a_mn && !a->b_mn), "gemm: operand layout (a MN-major, b K-major) is not instantiated");
    TRS_REQUIRE((!a->a_mn || a->m % 8 == 0), "gemm: MN-major a needs m %% 8 == 0");
    const int layout = (a->a_mn ? 2 : 0) | (a->b_mn ? 1 : 0);
#define TRS_GEMM_CASE(BN_, ST_, BF_, L_, AM_, BM_) \
    if ((a->n > 64) == (BN_ == 128) && (a->out_bf16 != 0) == BF_ && layout == L_) \
        return launch_gemm<BN_, ST_, BF_, AM_, BM_>(a, g, splits, s);
    TRS_GEMM_CASE(128, 3, true, 0, false, false)
    TRS_GEMM_CASE(128, 3, false, 0, false, false)
    TRS_GEMM_CASE(64, 4, true, 0, false, false)
    TRS_GEMM_CASE(64, 4, false, 0, false, false)
    TRS_GEMM_CASE(128, 3, true, 1, false, true)
    TRS_GEMM_CASE(128, 3, false, 1, false, true)
    TRS_GEMM_CASE(64, 4, true, 1, false, true)
    TRS_GEMM_CASE(64, 4, false, 1, false, true)
    TRS_GEMM_CASE(128, 3, false, 3, true, true)
    TRS_GEMM_CASE(64, 4, false, 3, true, true)
#undef TRS_GEMM_CASE
    set_error("gemm: no kernel for this combination (MN-major a writes fp32 only)");
    return TRS_ERR_ARG;
}
