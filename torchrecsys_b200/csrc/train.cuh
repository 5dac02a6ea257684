// train.cuh -- the row-wise optimizer step shared by the training kernels (train.cu, shard.cu): the
// update of one value, of a row held in registers and of a width-1 companion, each followed by the stores of the
// parameter and its optimizer state; and what mlp.cu needs from train.cu: the reduce + update phase of the fused
// training kernel, run on gradient rows the MLP backward staged itself.
#pragma once
#include "common.cuh"

namespace trs {

// where the per-lookup gradient rows of one step live inside the train workspace
// (gU [B, dim]: one row per sample; gI / gM[f] [2B, dim]: positives then negatives)
struct StagePtrs {
    float* gU;
    float* gI;
    float* gM[TRS_MAX_META];
};
StagePtrs stage_pointers(const trs_model* model, const trs_epoch* ep, void* workspace);

struct OptScalars {
    int kind;
    float omb1, omb2, eps;  // 1-beta1, 1-beta2, eps rounded to fp32 as torch's scalar ops do
    const float* step_scale;
};

// ---- row-wise optimizers (torch: optim/_functional.py:65-84, optim/adagrad.py:363-373, sgd) ----
// Explicit _rn intrinsics keep nvcc from contracting mul+add into FMA where torch runs two ops.  torch on CUDA rounds
// Adagrad's product before the sum too; torch on the CPU fuses it.  The op stream is the contract stated in
// tests/test_train_exact.py, which checks it bit for bit, and oracle/cf_oracle.py: apply_rows restates it.
__device__ __forceinline__ void opt_update(const OptScalars& o, float scale, float g, float& p,
                                           float& s0, float& s1) {
    if (o.kind == TRS_OPT_SPARSE_ADAM) {
        const float um = __fmul_rn(__fsub_rn(g, s0), o.omb1);
        const float uv = __fmul_rn(__fsub_rn(__fmul_rn(g, g), s1), o.omb2);
        s0 = __fadd_rn(s0, um);
        s1 = __fadd_rn(s1, uv);
        const float denom = __fadd_rn(__fsqrt_rn(s1), o.eps);
        p = __fadd_rn(p, __fmul_rn(-scale, __fdiv_rn(s0, denom)));
    } else if (o.kind == TRS_OPT_ADAGRAD) {
        s0 = __fadd_rn(s0, __fmul_rn(g, g));
        const float stdv = __fadd_rn(__fsqrt_rn(s0), o.eps);
        p = __fadd_rn(p, __fmul_rn(-scale, __fdiv_rn(g, stdv)));
    } else {
        p = __fadd_rn(p, __fmul_rn(-scale, g));
    }
}

// update one row held in registers and write it (param + the optimizer's state tensors)
template <int V, int G, int IT>
__device__ __forceinline__ void update_store_row(const trs_table& t, size_t roff, int nch, int gl, const OptScalars& o,
                                                 float scale, Row<V, IT>& p, Row<V, IT>& s0, Row<V, IT>& s1,
                                                 const Row<V, IT>& g) {
#pragma unroll
    for (int a = 0; a < IT; ++a)
#pragma unroll
        for (int b = 0; b < V; ++b) opt_update(o, scale, g.c[a][b], p.c[a][b], s0.c[a][b], s1.c[a][b]);
#pragma unroll
    for (int a = 0; a < IT; ++a) {
        const int c = gl + a * G;
        if (c < nch) {
            p.c[a].st(t.emb + roff + (size_t)c * V);
            if (o.kind != TRS_OPT_SGD) s0.c[a].st(t.emb_s0 + roff + (size_t)c * V);
            if (o.kind == TRS_OPT_SPARSE_ADAM) s1.c[a].st(t.emb_s1 + roff + (size_t)c * V);
        }
    }
}
// the same for the width-1 companion of a row (bias / first-order weight), one thread: value p and state s0 / s1
// already loaded
__device__ __forceinline__ void update_store_lin(const trs_table& t, uint32_t key, const OptScalars& o, float scale,
                                                 float g, float p, float s0, float s1) {
    opt_update(o, scale, g, p, s0, s1);
    t.lin[key] = p;
    if (o.kind != TRS_OPT_SGD) t.lin_s0[key] = s0;
    if (o.kind == TRS_OPT_SPARSE_ADAM) t.lin_s1[key] = s1;
}

// fills OptScalars from the C-ABI optimizer description (beta / eps rounded to fp32 as torch's scalar ops do)
inline OptScalars make_opt_scalars(const trs_optim* optim) {
    OptScalars os;
    os.kind = optim->kind;
    os.omb1 = (float)(1.0 - optim->beta1);
    os.omb2 = (float)(1.0 - optim->beta2);
    os.eps = (float)optim->eps;
    os.step_scale = optim->step_scale;
    return os;
}

int run_train_steps(const trs_model* model, const trs_epoch* ep, const trs_optim* optim, const void* plan,
                    void* workspace, size_t workspace_bytes, int first_step, int n_steps, float* loss,
                    cudaStream_t stream);

}  // namespace trs
