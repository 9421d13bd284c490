// K3: softmax(l0) -> labels -> ST(hard_max) -> sum_k unpool(feat) ++ mask, as a device-side body so that it can run as
// its own kernel (step_fused.cu) and as one role of the fused forward kernel (step_fwd_fused.cu).
// Reference chain: cub/code/SB_model48i/model.py:426,434-436,447,470,225-249,482-484.
#pragma once
#include "common.cuh"

namespace ups {

constexpr int FW = 4;           // warps per CTA
constexpr int FTPB = FW * 32;
constexpr unsigned FULL = 0xffffffffu;

// ============================================================================ K3 decode fwd
// general rows (tied maxima somewhere in these PW pixels): sum over parts in ascending k
template <int LPP>
__device__ __noinline__ void inject_rows_general(float4 mh, const float4* fs4, float* rows, int NF4, int FK, int lane) {
    constexpr int K = 4 * LPP, PW = 32 / LPP;
    const int nf_it = (NF4 + 31) >> 5;
    for (int pix_l = 0; pix_l < PW; ++pix_l) {
        for (int it = 0; it < nf_it; ++it) {
            const int f4 = it * 32 + lane;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int src = pix_l * LPP + (k >> 2);
                const float comp = ((k & 3) == 0) ? mh.x : ((k & 3) == 1) ? mh.y : ((k & 3) == 2) ? mh.z : mh.w;
                const float mk = __shfl_sync(FULL, comp, src);
                if (mk != 0.f && f4 < NF4) {
                    const float4 fv = fs4[k * NF4 + f4];
                    acc.x = fmaf(mk, fv.x, acc.x); acc.y = fmaf(mk, fv.y, acc.y);
                    acc.z = fmaf(mk, fv.z, acc.z); acc.w = fmaf(mk, fv.w, acc.w);
                }
            }
            if (f4 < NF4) st4_stream(rows + (size_t)pix_l * FK + 4 * f4, acc);
        }
    }
}

// FT = compile-time F (0: run-time F) so that the row/column split of the inject store is shifts.
// (split, b): the CTA's pixel range of sample b; fs4: K*F floats of shared memory (feat[b] as [K][F/4] float4)
// NOISE: l0 holds the means and the logits are sampled in registers right after the load (canon_math.cuh, the mean-field
// logit noise); the noise-free instantiation is the plain kernel.
template <int LPP, int FT, bool NOISE = false>
__device__ __forceinline__ void step_decode_fwd_body(const float* __restrict__ l0, const float* __restrict__ feat,
                                                     float* __restrict__ m0, long long* __restrict__ labels0,
                                                     float* __restrict__ inj, int P, int Frt, int pix_per_cta, int split,
                                                     int b, float4* fs4, int l0_row, const NoiseArgs& nz = NoiseArgs{}) {
    // l0_row: row length of l0 in floats (K, or the real part count when the logits of a padded K are read in place)
    constexpr int K = 4 * LPP, PW = 32 / LPP;
    const int F = FT > 0 ? FT : Frt;
    const int NF4 = F >> 2, FK = F + K;
    for (int i = threadIdx.x; i < K * NF4; i += FTPB) fs4[i] = ld4(feat + (size_t)b * K * F + 4 * i);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = lane & (LPP - 1), plq = lane / LPP;
    const int p_begin = split * pix_per_cta, p_end = min(P, p_begin + pix_per_cta);
    const int n_items = PW * NF4, n_it = (n_items + 31) >> 5;
    for (int pg = p_begin + warp * 32; pg < p_end; pg += FW * 32) {
        float4 v[LPP];
#pragma unroll
        for (int s = 0; s < LPP; ++s)
            v[s] = ld_row4<LPP>(l0, (size_t)b * P + pg + s * PW + plq, c, l0_row, -INFINITY);
        if (NOISE) {
#pragma unroll
            for (int s = 0; s < LPP; ++s) v[s] = add_noise4(v[s], nz, b, P, pg + s * PW + plq, c);
        }
#pragma unroll
        for (int s = 0; s < LPP; ++s) {
            const size_t pix = (size_t)b * P + pg + s * PW + plq;
            float pmax; int arg, nmax;
            const float4 p4 = softmax4<LPP>(v[s], c, pmax, arg, nmax);
            st4(m0 + (pix * LPP + c) * 4, p4);
            if (c == 0) labels0[pix] = arg;
            const float4 mh = hard_st4(p4, pmax);
            st4_stream(inj + pix * FK + F + 4 * c, mh);
            const float mon = st_value(1.0f, pmax);
            float* rows = inj + ((size_t)b * P + pg + s * PW) * FK;
            if (!__any_sync(FULL, nmax > 1)) {
                // one-hot fast path: row = mon * feat[arg, :]
#pragma unroll 4
                for (int it = 0; it < n_it; ++it) {
                    const int idx = it * 32 + lane;
                    const bool valid = idx < n_items;
                    const int pix_l = valid ? idx / NF4 : 0;
                    const int f4 = idx - pix_l * NF4;
                    const int k = __shfl_sync(FULL, arg, pix_l * LPP);
                    const float mv = __shfl_sync(FULL, mon, pix_l * LPP);
                    if (valid) {
                        const float4 fv = fs4[k * NF4 + f4];
                        st4_stream(rows + (size_t)pix_l * FK + 4 * f4,
                                   make_float4(fv.x * mv, fv.y * mv, fv.z * mv, fv.w * mv));
                    }
                }
            } else {
                inject_rows_general<LPP>(mh, fs4, rows, NF4, FK, lane);
            }
        }
    }
}

}  // namespace ups
