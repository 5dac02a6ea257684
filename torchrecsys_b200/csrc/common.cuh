// common.cuh -- shared device/host helpers for libtrs_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/trs.h"

#ifndef __CUDA_ARCH_LIST__
#define __CUDA_ARCH_LIST__ 1000
#endif

namespace trs {

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define TRS_REQUIRE(cond, ...)          \
    do {                                \
        if (!(cond)) {                  \
            trs::set_error(__VA_ARGS__); \
            return TRS_ERR_ARG;         \
        }                               \
    } while (0)
#define TRS_CUDA(call)                                                                    \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            trs::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                           __LINE__);                                                     \
            return TRS_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

struct DeviceProps {
    int sm_count;
    int max_smem_optin;
};
const DeviceProps& device_props();

// ---- row vectors ------------------------------------------------------------------------
// A table row of `dim` floats is split into chunks of V floats (V = 4 -> one 128-bit access;
// V = 1 only when dim % 4 != 0).  A *group* of G lanes owns one row; lane l handles chunks
// l, l+G, ... (IT of them at most).
template <int V>
struct Vec;
template <>
struct Vec<4> {
    float4 v;
    __device__ __forceinline__ static Vec ld(const float* p) {
        Vec r;
        r.v = *reinterpret_cast<const float4*>(p);
        return r;
    }
    __device__ __forceinline__ static Vec ld_cg(const float* p) {  // L2 only, bypass L1
        Vec r;
        r.v = __ldcg(reinterpret_cast<const float4*>(p));
        return r;
    }
    __device__ __forceinline__ static Vec zero() {
        Vec r;
        r.v = make_float4(0.f, 0.f, 0.f, 0.f);
        return r;
    }
    __device__ __forceinline__ void st(float* p) const { *reinterpret_cast<float4*>(p) = v; }
    __device__ __forceinline__ float& operator[](int i) { return (&v.x)[i]; }
    __device__ __forceinline__ const float& operator[](int i) const { return (&v.x)[i]; }
};
template <>
struct Vec<1> {
    float v;
    __device__ __forceinline__ static Vec ld(const float* p) {
        Vec r;
        r.v = *p;
        return r;
    }
    __device__ __forceinline__ static Vec ld_cg(const float* p) {
        Vec r;
        r.v = __ldcg(p);
        return r;
    }
    __device__ __forceinline__ static Vec zero() {
        Vec r;
        r.v = 0.f;
        return r;
    }
    __device__ __forceinline__ void st(float* p) const { *p = v; }
    __device__ __forceinline__ float& operator[](int) { return v; }
    __device__ __forceinline__ const float& operator[](int) const { return v; }
};

template <int V, int IT>
struct Row {
    Vec<V> c[IT];
};

// chunk index -> valid?  (nch = dim / V chunks per row)
template <int V, int G, int IT>
__device__ __forceinline__ Row<V, IT> load_row(const float* __restrict__ base, int nch, int gl) {
    Row<V, IT> r;
#pragma unroll
    for (int i = 0; i < IT; ++i) {
        int c = gl + i * G;
        r.c[i] = (c < nch) ? Vec<V>::ld(base + (size_t)c * V) : Vec<V>::zero();
    }
    return r;
}
// same, through L2 only: for rows another SM wrote earlier in the same launch
template <int V, int G, int IT>
__device__ __forceinline__ Row<V, IT> load_row_cg(const float* __restrict__ base, int nch, int gl) {
    Row<V, IT> r;
#pragma unroll
    for (int i = 0; i < IT; ++i) {
        int c = gl + i * G;
        r.c[i] = (c < nch) ? Vec<V>::ld_cg(base + (size_t)c * V) : Vec<V>::zero();
    }
    return r;
}
template <int V, int G, int IT>
__device__ __forceinline__ void store_row(float* __restrict__ base, int nch, int gl,
                                          const Row<V, IT>& r) {
#pragma unroll
    for (int i = 0; i < IT; ++i) {
        int c = gl + i * G;
        if (c < nch) r.c[i].st(base + (size_t)c * V);
    }
}
template <int V, int IT>
__device__ __forceinline__ void row_zero(Row<V, IT>& r) {
#pragma unroll
    for (int i = 0; i < IT; ++i) r.c[i] = Vec<V>::zero();
}
template <int V, int IT>
__device__ __forceinline__ void row_acc(Row<V, IT>& a, const Row<V, IT>& b) {  // a += b, unfused
#pragma unroll
    for (int i = 0; i < IT; ++i)
#pragma unroll
        for (int k = 0; k < V; ++k) a.c[i][k] = __fadd_rn(a.c[i][k], b.c[i][k]);
}

// sum over the G lanes of a group (G a power of two, groups aligned inside the warp)
template <int G>
__device__ __forceinline__ float group_sum(float x) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

__device__ __forceinline__ float warp_sum(float x) { return group_sum<32>(x); }

// order-preserving map float -> uint32: a < b  <=>  float_key(a) < float_key(b)
__device__ __forceinline__ uint32_t float_key(float x) {
    const uint32_t u = __float_as_uint(x);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Philox4x32-10: the ten rounds on counter c under key (k0, k1); c holds the four output words afterwards
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0;
        c[1] = lo1;
        c[2] = n2;
        c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

// ---- launch-shape dispatch -----------------------------------------------------------------
// (V, G, IT) chosen from dim: see DESIGN.md "row layout".
struct RowShape {
    int V, G, IT;
};
inline bool pick_row_shape(int dim, RowShape* s) {
    if (dim <= 0) return false;
    if (dim % 4 == 0) {
        int nch = dim / 4;
        int G = 4;
        while (G < nch && G < 32) G <<= 1;
        int IT = (nch + G - 1) / G;
        if (IT > 4) return false;
        if (IT == 3) IT = 4;
        *s = {4, G, IT};
        return true;
    }
    int IT = (dim + 31) / 32;
    if (IT > 8) return false;
    int it2 = 1;
    while (it2 < IT) it2 <<= 1;
    *s = {1, 32, it2};
    return true;
}

// Expands to a switch over the supported (V,G,IT) instantiations and calls
// FN<V,G,IT>(args...).  Keep the list in sync with pick_row_shape.
#define TRS_DISPATCH_ROW_SHAPE(shape, FN, ...)                                      \
    do {                                                                            \
        const int key__ = (shape).V * 10000 + (shape).G * 100 + (shape).IT;         \
        switch (key__) {                                                            \
            case 40401: FN<4, 4, 1>(__VA_ARGS__); break;                            \
            case 40801: FN<4, 8, 1>(__VA_ARGS__); break;                            \
            case 41601: FN<4, 16, 1>(__VA_ARGS__); break;                           \
            case 43201: FN<4, 32, 1>(__VA_ARGS__); break;                           \
            case 43202: FN<4, 32, 2>(__VA_ARGS__); break;                           \
            case 43204: FN<4, 32, 4>(__VA_ARGS__); break;                           \
            case 13201: FN<1, 32, 1>(__VA_ARGS__); break;                           \
            case 13202: FN<1, 32, 2>(__VA_ARGS__); break;                           \
            case 13204: FN<1, 32, 4>(__VA_ARGS__); break;                           \
            case 13208: FN<1, 32, 8>(__VA_ARGS__); break;                           \
            default: break;                                                         \
        }                                                                           \
    } while (0)

int check_model(const trs_model* m, RowShape* shape);
// rank / world / dim / row counts of a row-sharded group (csrc/shard.cu)
int check_shard(const trs_shard* sh, RowShape* shape);

static inline int64_t n_steps_of(const trs_epoch* e) {
    return (e->n_samples + e->batch - 1) / e->batch;
}

}  // namespace trs
