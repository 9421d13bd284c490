// Shared host/device helpers for libups_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "../../include/ups_b200.h"
#include "canon_math.cuh"
#include "pk_math.cuh"

namespace ups {

constexpr int NUM_SMS = 148;  // B200: 2 dies x 74 SMs

void set_error(const char* fmt, ...);
void count_launch();
int after_launch(const char* what);  // cudaGetLastError -> status, counts the launch

int fused_pix_per_cta(int B, int P);  // step_fused.cu
size_t pool_ws_bytes(int B, int P, int KF);  // parts_ops.cu
size_t decode_bwd_tma_ws_bytes(int B, int P, int K, int F);  // step_decode_bwd_tma.cu
size_t moments_ws_bytes(int B, int P, int K);  // stats_ops.cu
size_t mumford_shah_ws_bytes(int B, int P, int K);  // priors_ops.cu
size_t priors_scalar_ws_bytes();                    // priors_ops.cu
bool parts_conv_bwd_tc_ok(int B, int H, int W, int K, int Co);   // parts_conv_bwd_tc.cu
int parts_conv_bwd_tc_launch(const float* g_h, const float* img, const float* V, float* dm_planes, float* ws_db, int B,
                             int H, int W, int K, cudaStream_t st);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

#define UPS_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            ::ups::set_error(__VA_ARGS__);     \
            return UPS_E_INVALID;              \
        }                                      \
    } while (0)

#define UPS_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t e__ = (call);                                                   \
        if (e__ != cudaSuccess) {                                                   \
            ::ups::set_error("%s failed: %s", #call, cudaGetErrorString(e__));      \
            return UPS_E_CUDA;                                                      \
        }                                                                           \
    } while (0)

// Kernels that run BESIDE the persistent K4 grid (the all-reduce, the stand-in gradient kernels): K4 configures its SM
// for the largest shared-memory carve-out; a kernel that prefers another carve-out cannot become resident on that SM
// until K4's CTA has left.  Asking for the same carve-out (once per kernel and process) removes that obstacle.
template <typename Kern>
inline void prefer_max_shared_carveout(Kern kern) {
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// the mean-field logit noise of one side of the step (canon_math.cuh::normal4_philox)
struct NoiseArgs {
    unsigned long long seed;
    long long sample_offset;   // global index of the launch's first sample
    float level;
    int draw;                  // 0: l0, 1: l1
};

#if defined(__CUDACC__)
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
// streaming variants: read-once inputs / write-once outputs should not displace reusable lines
__device__ __forceinline__ float4 ld4_stream(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4_stream(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }

// Parts 4c .. 4c+3 of pixel `pix` from a row-major [., row] tensor, for the kernels that work on K = 4*LPP lanes: row == K
// is the ordinary 16-byte load; a shorter row (a part count that is not a power of two, read in place instead of through
// a padded copy) is read element-wise, parts >= row come back as `pad`.
template <int LPP>
__device__ __forceinline__ float4 ld_row4(const float* __restrict__ base, size_t pix, int c, int row, float pad) {
    if (row == 4 * LPP) return ld4_stream(base + (pix * LPP + c) * 4);
    const float* p = base + pix * (size_t)row + 4 * c;
    const int k0 = 4 * c;
    float4 v;
    v.x = k0 < row ? __ldcs(p) : pad;
    v.y = k0 + 1 < row ? __ldcs(p + 1) : pad;
    v.z = k0 + 2 < row ? __ldcs(p + 2) : pad;
    v.w = k0 + 3 < row ? __ldcs(p + 3) : pad;
    return v;
}

// parts 4c .. 4c+3 of pixel p of sample b (of P pixels) sampled in registers: v + noise_level * z
__device__ __forceinline__ float4 add_noise4(float4 v, const NoiseArgs& n, int b, int P, int p, int c) {
    const unsigned long long g = (unsigned long long)(n.sample_offset + b) * (unsigned long long)P + (unsigned)p;
    float z0, z1, z2, z3;
    normal4_philox(n.seed, (uint32_t)n.draw, g, (uint32_t)c, z0, z1, z2, z3);
    return make_float4(sampled_logit(v.x, n.level, z0), sampled_logit(v.y, n.level, z1), sampled_logit(v.z, n.level, z2),
                       sampled_logit(v.w, n.level, z3));
}

// DSEED (the `_dseed` entry points): NoiseArgs::seed carries the ADDRESS of the seed, one device word, and the kernel reads
// it once, in its prologue.  A launch captured in a CUDA graph then draws with whatever the word holds when the graph is
// replayed.  DSEED = false is the by-value seed, returned unchanged.
template <bool DSEED>
__device__ __forceinline__ NoiseArgs resolve_seed(NoiseArgs nz) {
    if (DSEED) nz.seed = *reinterpret_cast<const unsigned long long*>(nz.seed);
    return nz;
}

template <int W>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
    for (int o = 1; o < W; o <<= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <int W>
__device__ __forceinline__ int group_min_int(int v) {
#pragma unroll
    for (int o = 1; o < W; o <<= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <int W>
__device__ __forceinline__ int group_sum_int(int v) {
#pragma unroll
    for (int o = 1; o < W; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// canonical adjacent-pair tree across W lanes (oracle/canon.py::sum_tree): NOT contracted
template <int W>
__device__ __forceinline__ float group_sum_canon(float v) {
#pragma unroll
    for (int o = 1; o < W; o <<= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <int W>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = 1; o < W; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Softmax of one pixel spread over LPP lanes, 4 consecutive parts per lane (K = 4*LPP), in the
// canonical order.  Returns probabilities; pmax = max prob of the pixel; arg = first index of
// the max; nmax = number of tied maxima.  `c` = lane's chunk index within the pixel.
template <int LPP>
__device__ __forceinline__ float4 softmax4(float4 v, int c, float& pmax, int& arg, int& nmax) {
    float m = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
    m = group_max<LPP>(m);
    // packed fp32x2 evaluation (pk_math.cuh): lanes bit-identical to exp_canon(__fsub_rn(v, m)) etc.
    const pk::Ops o;
    const pk::f2 m2 = pk::splat(m);
    const pk::f2 d[2] = {o.sub(pk::pack(v.x, v.y), m2), o.sub(pk::pack(v.z, v.w), m2)};
    pk::f2 ee[2];
    pk::exp_canon2n<2>(o, d, ee);
    const pk::f2 e01 = ee[0], e23 = ee[1];
    float4 e;
    pk::unpack(e01, e.x, e.y);
    pk::unpack(e23, e.z, e.w);
    float s = __fadd_rn(__fadd_rn(e.x, e.y), __fadd_rn(e.z, e.w));
    s = group_sum_canon<LPP>(s);
    const float rs = __frcp_rn(s);
    const pk::f2 rs2 = pk::splat(rs);
    float4 p;
    pk::unpack(o.mul(e01, rs2), p.x, p.y);
    pk::unpack(o.mul(e23, rs2), p.z, p.w);
    pmax = group_max<LPP>(fmaxf(fmaxf(p.x, p.y), fmaxf(p.z, p.w)));
    int a = 1 << 30;
    a = (p.w == pmax) ? 4 * c + 3 : a;
    a = (p.z == pmax) ? 4 * c + 2 : a;
    a = (p.y == pmax) ? 4 * c + 1 : a;
    a = (p.x == pmax) ? 4 * c + 0 : a;
    arg = group_min_int<LPP>(a);
    const int n = (p.x == pmax) + (p.y == pmax) + (p.z == pmax) + (p.w == pmax);
    nmax = group_sum_int<LPP>(n);
    return p;
}

// straight_through_estimator(hard_max(p), p) for the lane's 4 parts
__device__ __forceinline__ float4 hard_st4(float4 p, float pmax) {
    // fl(fl(h - p) + p), two parts per FFMA2
    const pk::Ops o;
    const pk::f2 p01 = pk::pack(p.x, p.y), p23 = pk::pack(p.z, p.w);
    const pk::f2 h01 = pk::pack(p.x == pmax ? 1.0f : 0.0f, p.y == pmax ? 1.0f : 0.0f);
    const pk::f2 h23 = pk::pack(p.z == pmax ? 1.0f : 0.0f, p.w == pmax ? 1.0f : 0.0f);
    float4 h;
    pk::unpack(o.add(o.sub(h01, p01), p01), h.x, h.y);
    pk::unpack(o.add(o.sub(h23, p23), p23), h.z, h.w);
    return h;
}
#endif

}  // namespace ups
