// Fused kernels of the per-step part-disentanglement path (SURVEY.md 8d: K2..K5).
//   K2 step_encode_fwd : softmax(l1) -> ST(hard_max) -> mask_parts(view1') part-major + mean pool
//   K3 step_decode_fwd : softmax(l0) -> labels -> ST(hard_max) -> sum_k unpool(feat) ++ mask
//   K4 step_decode_bwd : inject-bwd (dmask, dfeat) fused with softmax-bwd(m0)
//   K5 step_encode_bwd : mask_parts/pool-bwd fused with softmax-bwd(m1) [+ dimg1]
// Reference chain: cub/code/SB_model48i/model.py:426-485 (+ :50-52 pooling tail, nn.py:58-168).
//
// Data layout (all fp32, NHWC): logits/probs [B,P,K]; images [B,P,3]; feat [B,K,F];
// inj [B,P,F+K]; parts part-major [K*B,P,3] (nn.apply_partwise's fold, nn.py:100-103).
// Work split: CTA (split, b) owns a contiguous pixel range of sample b; 4 warps stride it in
// blocks of 32 pixels.  All global traffic is 16-byte vectors, contiguous per warp.
// Reductions over pixels (pooled, dfeat) are accumulated privately (per lane / per warp) in
// shared memory, reduced in a fixed order per CTA and summed over splits by a second tiny
// kernel: bit-reproducible run to run, no atomics.
#include <stdlib.h>

#include "common.cuh"
#include "step_decode_fwd.cuh"

namespace ups {

constexpr int MS = 34;          // row stride of the per-warp [K][32] mask stash (conflict-free)

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ============================================================================ K3 decode fwd (body: step_decode_fwd.cuh)
template <int LPP, int FT, bool NOISE, bool DSEED>
__global__ void __launch_bounds__(FTPB) step_decode_fwd_kernel(const float* __restrict__ l0,
                                                               const float* __restrict__ feat,
                                                               float* __restrict__ m0,
                                                               long long* __restrict__ labels0,
                                                               float* __restrict__ inj, int P, int Frt,
                                                               int pix_per_cta, int l0_row, NoiseArgs nz) {
    extern __shared__ float4 fs4[];  // feat[b] as [K][F/4] float4
    step_decode_fwd_body<LPP, FT, NOISE>(l0, feat, m0, labels0, inj, P, Frt, pix_per_cta, blockIdx.x, blockIdx.y, fs4, l0_row,
                                         resolve_seed<DSEED>(nz));
}

// ============================================================================ K2 encode fwd
template <int LPP>
struct EncFwdSmem {
    static constexpr int K = 4 * LPP;
    static constexpr int MW = K * MS;        // mask stash [K][MS]
    static constexpr int IW = 96;            // 32 pixels x 3 channels
    static constexpr int MON = 32, LAB = 32;
    static constexpr int ACC = K * 3 * 32;   // lane-private pooled accumulators [(k,c)][lane]
    static constexpr int WREG = MW + IW + MON + LAB + ACC;
};

// MINB: resident CTAs per SM asked of ptxas (an explicit value also keeps the exp chains interleaved)
// NOISE: l1 holds the means, sampled in registers right after the load (canon_math.cuh, the mean-field logit noise)
// DSEED: the seed is read from device memory (resolve_seed)
template <int LPP, int MINB, bool PAD, bool NOISE, bool DSEED>
__global__ void __launch_bounds__(FTPB, MINB) step_encode_fwd_kernel(const float* __restrict__ l1,
                                                               const float* __restrict__ img1,
                                                               float* __restrict__ m1, float* __restrict__ parts,
                                                               float* __restrict__ partial, int B, int P,
                                                               int pix_per_cta, int Kpl, int l1_row, NoiseArgs nz_arg) {
    // Kpl <= K: number of part planes that exist in `parts` (planes Kpl..K-1 are padding of a K that is not a power
    // of two: their mask is identically zero and they are neither written nor allocated)
    const NoiseArgs nz = resolve_seed<DSEED>(nz_arg);
    using L = EncFwdSmem<LPP>;
    constexpr int K = L::K, PW = 32 / LPP;
    extern __shared__ float4 smem4[];
    float* sm = reinterpret_cast<float*>(smem4);
    const int b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = lane & (LPP - 1), plq = lane / LPP;
    float* Mw = sm + warp * L::WREG;
    float* Iw = Mw + L::MW;
    float* monw = Iw + L::IW;
    int* labw = reinterpret_cast<int*>(monw + L::MON);
    float* acc = monw + L::MON + L::LAB;
    for (int i = lane; i < L::ACC; i += 32) acc[i] = 0.f;
    __syncwarp();
    const int p_begin = blockIdx.x * pix_per_cta, p_end = min(P, p_begin + pix_per_cta);
    for (int pg = p_begin + warp * 32; pg < p_end; pg += FW * 32) {
        float4 v[LPP];
#pragma unroll
        for (int s = 0; s < LPP; ++s)
            v[s] = ld_row4<LPP>(l1, (size_t)b * P + pg + s * PW + plq, c, l1_row, -INFINITY);
        if (NOISE) {
#pragma unroll
            for (int s = 0; s < LPP; ++s) v[s] = add_noise4(v[s], nz, b, P, pg + s * PW + plq, c);
        }
        if (lane < 24) st4(Iw + 4 * lane, ld4(img1 + ((size_t)b * P + pg) * 3 + 4 * lane));
#pragma unroll
        for (int s = 0; s < LPP; ++s) {
            const int pl = s * PW + plq;
            const size_t gi = ((size_t)b * P + pg + pl) * LPP + c;
            float pmax; int arg, nmax;
            const float4 p4 = softmax4<LPP>(v[s], c, pmax, arg, nmax);
            st4(m1 + 4 * gi, p4);
            const float4 mh = hard_st4(p4, pmax);
            Mw[(4 * c + 0) * MS + pl] = mh.x;
            Mw[(4 * c + 1) * MS + pl] = mh.y;
            Mw[(4 * c + 2) * MS + pl] = mh.z;
            Mw[(4 * c + 3) * MS + pl] = mh.w;
            if (c == 0) { labw[pl] = nmax > 1 ? -1 : arg; monw[pl] = st_value(1.0f, pmax); }
        }
        __syncwarp();
        // mask_parts, written part-major: plane (k*B+b) gets 96 contiguous floats per 32 pixels
#pragma unroll 4
        for (int it = 0; it < (K * 24) / 32; ++it) {
            const int idx = it * 32 + lane;
            const int k = idx / 24, q = idx - 24 * k;
            const int r0 = 4 * q, pa = r0 / 3, sft = r0 - 3 * pa;
            const float4 i4 = *reinterpret_cast<const float4*>(Iw + r0);
            const float ma = Mw[k * MS + pa], mb = Mw[k * MS + min(pa + 1, 31)];
            float4 o;
            o.x = i4.x * ma;
            o.y = i4.y * (sft == 2 ? mb : ma);
            o.z = i4.z * (sft >= 1 ? mb : ma);
            o.w = i4.w * mb;
            if (!PAD || k < Kpl) st4_stream(parts + (((size_t)k * B + b) * P + pg) * 3 + r0, o);
        }
        // mean pooling (model.py:50-52 tail): lane = pixel, lane-private accumulators
        {
            const int lab = labw[lane];
            const float i0 = Iw[3 * lane], i1 = Iw[3 * lane + 1], i2 = Iw[3 * lane + 2];
            if (lab >= 0) {
                const float mo = monw[lane];
                float* a = acc + (lab * 3) * 32 + lane;
                a[0] = fmaf(mo, i0, a[0]); a[32] = fmaf(mo, i1, a[32]); a[64] = fmaf(mo, i2, a[64]);
            } else {
                for (int k = 0; k < K; ++k) {
                    const float m = Mw[k * MS + lane];
                    if (m != 0.f) {
                        float* a = acc + (k * 3) * 32 + lane;
                        a[0] = fmaf(m, i0, a[0]); a[32] = fmaf(m, i1, a[32]); a[64] = fmaf(m, i2, a[64]);
                    }
                }
            }
        }
        __syncwarp();
    }
    __syncthreads();
    for (int t = threadIdx.x; t < K * 3; t += FTPB) {
        float s = 0.f;
        for (int w = 0; w < FW; ++w) {
            const float* a = sm + w * L::WREG + L::MW + L::IW + L::MON + L::LAB + t * 32;
            for (int l = 0; l < 32; ++l) s += a[(l + t) & 31];
        }
        partial[((size_t)b * gridDim.x + blockIdx.x) * (K * 3) + t] = s;
    }
}

// ============================================================================ K4 decode bwd
// lane = (pixel-in-step, part): PPW = 32/K pixels per warp step, the lane's feat row in
// registers, g_inj rows streamed global->shared with a cp.async ring (no register staging).
template <int K, int F>
struct DecBwdSmem {
    static constexpr int PPW = 32 / K, FK = F + K, NF4 = F / 4, GROUPS = 32 / NF4;
    static constexpr int NST = 4;                       // cp.async stages
    static constexpr int STAGE = PPW * FK;              // floats per stage
    static constexpr int ACC = GROUPS * K * F;          // per-warp dfeat accumulators
    static constexpr int WREG = NST * STAGE + ACC;
};

template <int K, int F>
__global__ void __launch_bounds__(FTPB) step_decode_bwd_kernel(const float* __restrict__ g_inj,
                                                               const float* __restrict__ m0,
                                                               const float* __restrict__ g_m0,
                                                               const float* __restrict__ feat,
                                                               float* __restrict__ dl0, float* __restrict__ partial,
                                                               int P, int pix_per_cta, int gm_row) {
    using L = DecBwdSmem<K, F>;
    constexpr int PPW = L::PPW, FK = L::FK, NF4 = L::NF4, GROUPS = L::GROUPS, NST = L::NST;
    constexpr int ROW4 = FK / 4, STAGE4 = PPW * ROW4;
    extern __shared__ float4 smem4[];
    float* sm = reinterpret_cast<float*>(smem4);
    const int b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = lane % K, pl = lane / K;
    float* Gw = sm + warp * L::WREG;
    float* acc = Gw + NST * L::STAGE;
    for (int i = lane; i < L::ACC; i += 32) acc[i] = 0.f;
    float fr[F];
#pragma unroll
    for (int f4 = 0; f4 < NF4; ++f4) {
        const float4 t = ld4(feat + ((size_t)b * K + k) * F + 4 * f4);
        fr[4 * f4] = t.x; fr[4 * f4 + 1] = t.y; fr[4 * f4 + 2] = t.z; fr[4 * f4 + 3] = t.w;
    }
    const int p_begin = blockIdx.x * pix_per_cta, p_end = min(P, p_begin + pix_per_cta);
    // this warp's steps: pixel groups pg = p_begin + (warp + FW*j)*PPW
    const int first = p_begin + warp * PPW;
    const int n_steps = first < p_end ? (p_end - first + FW * PPW - 1) / (FW * PPW) : 0;
    auto issue = [&](int j) {
        if (j < n_steps) {
            const float* src = g_inj + ((size_t)b * P + first + (size_t)j * FW * PPW) * FK;
            float* dst = Gw + (j % NST) * L::STAGE;
            for (int i = lane; i < STAGE4; i += 32) cp_async16(dst + 4 * i, src + 4 * i);
        }
        cp_async_commit();
    };
#pragma unroll
    for (int j = 0; j < NST - 1; ++j) issue(j);
    const int grp = lane / NF4, f4l = lane % NF4;
    float pr_n = 0.f, gm_n = 0.f;
    if (n_steps > 0) {
        const size_t o = ((size_t)b * P + first) * K + lane;
        pr_n = __ldcs(m0 + o);
        gm_n = (g_m0 && k < gm_row) ? __ldcs(g_m0 + ((size_t)b * P + first + pl) * gm_row + k) : 0.f;
    }
    __syncwarp();
    for (int j = 0; j < n_steps; ++j) {
        issue(j + NST - 1);
        const float pr = pr_n, gm = gm_n;
        const size_t o = ((size_t)b * P + first + (size_t)j * FW * PPW) * K + lane;
        if (j + 1 < n_steps) {
            const size_t on = o + (size_t)FW * PPW * K;
            pr_n = __ldcs(m0 + on);
            gm_n = (g_m0 && k < gm_row)
                       ? __ldcs(g_m0 + ((size_t)b * P + first + (size_t)(j + 1) * FW * PPW + pl) * gm_row + k) : 0.f;
        }
        cp_async_wait<NST - 1>();
        __syncwarp();
        const float* G = Gw + (j % NST) * L::STAGE;
        const float* gr = G + pl * FK;
        // dmask[k] = sum_f g[f]*feat[k,f] + g[F+k]      ((P x F).(F x K) contraction)
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int f4 = 0; f4 < NF4; ++f4) {
            const float4 g4 = *reinterpret_cast<const float4*>(gr + 4 * f4);
            a0 = fmaf(g4.x, fr[4 * f4], a0);
            a1 = fmaf(g4.y, fr[4 * f4 + 1], a1);
            a2 = fmaf(g4.z, fr[4 * f4 + 2], a2);
            a3 = fmaf(g4.w, fr[4 * f4 + 3], a3);
        }
        const float gp = ((a0 + a1) + (a2 + a3)) + gr[F + k] + gm;
        const float dot = group_sum<K>(gp * pr);
        __stcs(dl0 + o, pr * (gp - dot));
        // dfeat[k,f] += mh[k]*g[f]: only the (tied) maxima have mh != 0
        const float pmax = group_max<K>(pr);
        const float mh = st_value(pr == pmax ? 1.0f : 0.0f, pr);
        const unsigned nz = __ballot_sync(FULL, mh != 0.f);
        const int cnt = __popc(nz);
        for (int r = 0; r * GROUPS < cnt; ++r) {
            const int n = r * GROUPS + grp;
            unsigned m = nz;
            for (int i = 0; i < n; ++i) m &= m - 1;
            const bool valid = (n < cnt) && (F == 4 * NF4) && (lane < GROUPS * NF4);
            const int Ls = valid ? (__ffs(m) - 1) : 0;
            const float mv = __shfl_sync(FULL, mh, Ls);
            if (valid) {
                const int kk = Ls % K, pp = Ls / K;
                const float4 g4 = *reinterpret_cast<const float4*>(G + pp * FK + 4 * f4l);
                float4* a = reinterpret_cast<float4*>(acc + (grp * K + kk) * F + 4 * f4l);
                float4 t = *a;
                t.x = fmaf(mv, g4.x, t.x); t.y = fmaf(mv, g4.y, t.y);
                t.z = fmaf(mv, g4.z, t.z); t.w = fmaf(mv, g4.w, t.w);
                *a = t;
            }
        }
        __syncwarp();
    }
    cp_async_wait<0>();
    __syncthreads();
    for (int t = threadIdx.x; t < K * F; t += FTPB) {
        float s = 0.f;
        for (int w = 0; w < FW; ++w)
            for (int g = 0; g < GROUPS; ++g) s += sm[w * L::WREG + NST * L::STAGE + g * K * F + t];
        partial[((size_t)b * gridDim.x + blockIdx.x) * (K * F) + t] = s;
    }
}

// ============================================================================ K5 encode bwd
template <int LPP>
struct EncBwdSmem {
    static constexpr int K = 4 * LPP;
    static constexpr int GS = K * 96;        // g_parts chunks [K][96]
    static constexpr int IW = 96;
    static constexpr int DW = 32 * (K + 1);  // dm [pixel][K+1]
    static constexpr int MW = K * MS;        // mask stash (dimg only)
    static constexpr int WREG = GS + IW + DW + MW;
};

template <int LPP, bool DIMG, bool PAD>
__global__ void __launch_bounds__(FTPB) step_encode_bwd_kernel(const float* __restrict__ g_parts,
                                                               const float* __restrict__ g_pooled,
                                                               const float* __restrict__ img1,
                                                               const float* __restrict__ m1,
                                                               const float* __restrict__ g_m1,
                                                               float* __restrict__ dl1, float* __restrict__ dimg1,
                                                               int B, int P, int pix_per_cta, int Kpl, int gm_row) {
    // Kpl <= K: planes of g_parts that exist (see step_encode_fwd_kernel); the cotangent of a padding plane is zero
    using L = EncBwdSmem<LPP>;
    constexpr int K = L::K, PW = 32 / LPP;
    extern __shared__ float4 smem4[];
    float* sm = reinterpret_cast<float*>(smem4);
    float* gpool = sm + FW * L::WREG;  // [K][3], already divided by P
    const int b = blockIdx.y;
    for (int i = threadIdx.x; i < K * 3; i += FTPB)
        gpool[i] = g_pooled ? g_pooled[(size_t)b * K * 3 + i] / (float)P : 0.f;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = lane & (LPP - 1), plq = lane / LPP;
    float* Gs = sm + warp * L::WREG;
    float* Iw = Gs + L::GS;
    float* Dw = Iw + L::IW;
    float* Mw = Dw + L::DW;
    const int p_begin = blockIdx.x * pix_per_cta, p_end = min(P, p_begin + pix_per_cta);
    for (int pg = p_begin + warp * 32; pg < p_end; pg += FW * 32) {
        // async: K planes x 96 floats of g_parts + 96 floats of the image
        for (int i = lane; i < K * 24; i += 32) {
            const int k = i / 24, q = i - 24 * k;
            if (!PAD || k < Kpl) cp_async16(Gs + k * 96 + 4 * q, g_parts + (((size_t)k * B + b) * P + pg) * 3 + 4 * q);
            else *reinterpret_cast<float4*>(Gs + k * 96 + 4 * q) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (lane < 24) cp_async16(Iw + 4 * lane, img1 + ((size_t)b * P + pg) * 3 + 4 * lane);
        cp_async_commit();
        float4 p4[LPP], gm4[LPP];
#pragma unroll
        for (int s = 0; s < LPP; ++s) {
            const size_t gi = ((size_t)b * P + pg + s * PW + plq) * LPP + c;
            p4[s] = ld4_stream(m1 + 4 * gi);
            gm4[s] = g_m1 ? ld_row4<LPP>(g_m1, (size_t)b * P + pg + s * PW + plq, c, gm_row, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (DIMG) {
#pragma unroll
            for (int s = 0; s < LPP; ++s) {
                const int pl = s * PW + plq;
                const float pmax = group_max<LPP>(fmaxf(fmaxf(p4[s].x, p4[s].y), fmaxf(p4[s].z, p4[s].w)));
                const float4 mh = hard_st4(p4[s], pmax);
                Mw[(4 * c + 0) * MS + pl] = mh.x;
                Mw[(4 * c + 1) * MS + pl] = mh.y;
                Mw[(4 * c + 2) * MS + pl] = mh.z;
                Mw[(4 * c + 3) * MS + pl] = mh.w;
            }
        }
        cp_async_wait<0>();
        __syncwarp();
        {   // lane = pixel: dm[k] = sum_c img[c]*(g_parts[k,c] + g_pooled[k,c]/P)
            const float i0 = Iw[3 * lane], i1 = Iw[3 * lane + 1], i2 = Iw[3 * lane + 2];
            float d0 = 0.f, d1 = 0.f, d2 = 0.f;
#pragma unroll 4
            for (int k = 0; k < K; ++k) {
                const float g0 = Gs[k * 96 + 3 * lane] + gpool[k * 3];
                const float g1 = Gs[k * 96 + 3 * lane + 1] + gpool[k * 3 + 1];
                const float g2 = Gs[k * 96 + 3 * lane + 2] + gpool[k * 3 + 2];
                Dw[lane * (K + 1) + k] = fmaf(i2, g2, fmaf(i1, g1, i0 * g0));
                if (DIMG) {
                    const float m = Mw[k * MS + lane];
                    if (m != 0.f) { d0 = fmaf(m, g0, d0); d1 = fmaf(m, g1, d1); d2 = fmaf(m, g2, d2); }
                }
            }
            if (DIMG) {
                __syncwarp();
                Iw[3 * lane] = d0; Iw[3 * lane + 1] = d1; Iw[3 * lane + 2] = d2;
            }
        }
        __syncwarp();
        if (DIMG && lane < 24)
            st4_stream(dimg1 + ((size_t)b * P + pg) * 3 + 4 * lane, *reinterpret_cast<const float4*>(Iw + 4 * lane));
#pragma unroll
        for (int s = 0; s < LPP; ++s) {
            const int pl = s * PW + plq;
            const size_t gi = ((size_t)b * P + pg + pl) * LPP + c;
            const float* d = Dw + pl * (K + 1) + 4 * c;
            const float4 gp = make_float4(d[0] + gm4[s].x, d[1] + gm4[s].y, d[2] + gm4[s].z, d[3] + gm4[s].w);
            const float4 p = p4[s];
            float dot = gp.x * p.x + gp.y * p.y + gp.z * p.z + gp.w * p.w;
            dot = group_sum<LPP>(dot);
            st4_stream(dl1 + 4 * gi, make_float4(p.x * (gp.x - dot), p.y * (gp.y - dot), p.z * (gp.z - dot), p.w * (gp.w - dot)));
        }
        __syncwarp();
    }
}

// sums the per-split partials in ascending split order (deterministic), optional /divide_by
__global__ void split_finalize_kernel(const float* __restrict__ partial, float* __restrict__ out, int n_per, int splits,
                                      int divide_by, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long b = i / n_per; const int j = (int)(i % n_per);
    float s = 0.f;
    for (int sp = 0; sp < splits; ++sp) s += partial[((size_t)b * splits + sp) * n_per + j];
    out[i] = divide_by > 0 ? s / (float)divide_by : s;
}

// pixels per CTA: aim at ~96 CTAs per SM in total (many short waves: measured 16 -> 96 gives 3-7 % on the
// HBM-bound kernels, profiles/r01_tuning.md); multiple of 128
int fused_pix_per_cta(int B, int P) {
    static const int target = []() { const char* e = getenv("UPS_FUSED_CTAS_PER_SM"); return e && atoi(e) > 0 ? atoi(e) : 96; }();
    long long want = cdiv((long long)target * NUM_SMS, B > 0 ? B : 1);
    long long maxs = cdiv(P, 128);
    if (want > maxs) want = maxs;
    if (want < 1) want = 1;
    long long per = cdiv(cdiv(P, want), 128) * 128;
    return (int)per;
}

template <typename Kern>
int set_smem(Kern kern, size_t bytes) {
    if (bytes > 48 * 1024) UPS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return UPS_OK;
}

}  // namespace ups

using namespace ups;

static int fused_common_checks(const char* what, int B, int P, int K) {
    UPS_REQUIRE(B >= 0 && B <= 65535, "%s: B=%d out of range", what, B);
    UPS_REQUIRE(K == 4 || K == 8 || K == 16 || K == 32, "%s: fused path needs K in {4,8,16,32}, got %d", what, K);
    UPS_REQUIRE(P >= 32 && P % 32 == 0, "%s: fused path needs P %% 32 == 0, got %d", what, P);
    return UPS_OK;
}

extern "C" int ups_step_decode_fwd(const float* l0, const float* feat, float* m0, long long* labels0, float* inj,
                                   int B, int P, int K, int F, void* stream) {
    return ups_step_decode_fwd_rows(l0, K, feat, m0, labels0, inj, B, P, K, F, stream);
}

template <bool NOISE, bool DSEED = false>
static int decode_fwd_launch(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0, float* inj, int B,
                             int P, int K, int F, NoiseArgs nz, void* stream) {
    UPS_REQUIRE(l0 && feat && m0 && labels0 && inj, "step_decode_fwd: null pointer");
    UPS_REQUIRE(l0_row >= 1 && l0_row <= K, "step_decode_fwd: l0 rows of %d floats for K=%d", l0_row, K);
    if (int rc = fused_common_checks("step_decode_fwd", B, P, K)) return rc;
    UPS_REQUIRE(F >= 4 && F % 4 == 0 && (size_t)K * F * 4 <= 96 * 1024, "step_decode_fwd: F=%d unsupported", F);
    UPS_REQUIRE((l0_row < K || aligned16(l0)) && aligned16(feat) && aligned16(m0) && aligned16(inj), "step_decode_fwd: 16-byte alignment");
    if (B == 0) return UPS_OK;
    const int per = fused_pix_per_cta(B, P);
    dim3 grid((unsigned)cdiv(P, per), B);
    size_t sm = (size_t)K * F * sizeof(float);
    // tuning knob: cap the resident CTAs per SM (by shared-memory footprint) so that a co-running kernel
    // on another stream (K1, see step.py) keeps a share of every SM's registers
    static const int cap = []() { const char* e = getenv("UPS_DECODE_FWD_CTAS_PER_SM"); return e ? atoi(e) : 0; }();
    if (cap > 0) { const size_t want = (size_t)(200 * 1024) / cap - 1024; if (want > sm) sm = want; }
    cudaStream_t s = as_stream(stream);
#define UPS_DEC_FWD2(LPP, FT)                                                                           \
    {                                                                                                   \
        if (int rc = set_smem(step_decode_fwd_kernel<LPP, FT, NOISE, DSEED>, sm)) return rc;            \
        step_decode_fwd_kernel<LPP, FT, NOISE, DSEED><<<grid, FTPB, sm, s>>>(l0, feat, m0, labels0, inj, P, F, per, l0_row, nz); \
    }
#define UPS_DEC_FWD(LPP) \
    { if (F == 64) UPS_DEC_FWD2(LPP, 64) else if (F == 32) UPS_DEC_FWD2(LPP, 32) else if (F == 16) UPS_DEC_FWD2(LPP, 16) else UPS_DEC_FWD2(LPP, 0) }
    if (K == 4) UPS_DEC_FWD(1) else if (K == 8) UPS_DEC_FWD(2) else if (K == 16) UPS_DEC_FWD(4) else UPS_DEC_FWD(8)
#undef UPS_DEC_FWD2
#undef UPS_DEC_FWD
    return after_launch("step_decode_fwd_kernel");
}

extern "C" int ups_step_decode_fwd_rows(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0,
                                        float* inj, int B, int P, int K, int F, void* stream) {
    return decode_fwd_launch<false>(l0, l0_row, feat, m0, labels0, inj, B, P, K, F, NoiseArgs{}, stream);
}

extern "C" int ups_step_decode_fwd_noise(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0,
                                         float* inj, int B, int P, int K, int F, unsigned long long seed, long long sample_offset,
                                         float noise_level, void* stream) {
    UPS_REQUIRE(sample_offset >= 0, "step_decode_fwd: sample_offset=%lld", sample_offset);
    return decode_fwd_launch<true>(l0, l0_row, feat, m0, labels0, inj, B, P, K, F, NoiseArgs{seed, sample_offset, noise_level, 0},
                                   stream);
}

extern "C" int ups_step_decode_fwd_noise_dseed(const float* l0, int l0_row, const float* feat, float* m0, long long* labels0,
                                               float* inj, int B, int P, int K, int F, const unsigned long long* seed,
                                               long long sample_offset, float noise_level, void* stream) {
    UPS_REQUIRE(seed, "step_decode_fwd: null seed pointer");
    UPS_REQUIRE(sample_offset >= 0, "step_decode_fwd: sample_offset=%lld", sample_offset);
    return decode_fwd_launch<true, true>(l0, l0_row, feat, m0, labels0, inj, B, P, K, F,
                                         NoiseArgs{(unsigned long long)(uintptr_t)seed, sample_offset, noise_level, 0}, stream);
}

extern "C" int ups_step_encode_fwd(const float* l1, const float* img1, float* m1, float* parts_pm, float* pooled,
                                   int B, int P, int K, void* ws, size_t ws_bytes, void* stream) {
    return ups_step_encode_fwd_planes(l1, img1, m1, parts_pm, pooled, B, P, K, K, ws, ws_bytes, stream);
}

extern "C" int ups_step_encode_fwd_planes(const float* l1, const float* img1, float* m1, float* parts_pm, float* pooled,
                                          int B, int P, int K, int Kpl, void* ws, size_t ws_bytes, void* stream) {
    return ups_step_encode_fwd_rows(l1, K, img1, m1, parts_pm, pooled, B, P, K, Kpl, ws, ws_bytes, stream);
}

template <bool NOISE, bool DSEED = false>
static int encode_fwd_launch(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm, float* pooled, int B,
                             int P, int K, int Kpl, void* ws, size_t ws_bytes, NoiseArgs nz, void* stream) {
    UPS_REQUIRE(l1 && img1 && m1 && parts_pm && pooled, "step_encode_fwd: null pointer");
    UPS_REQUIRE(l1_row >= 1 && l1_row <= K, "step_encode_fwd: l1 rows of %d floats for K=%d", l1_row, K);
    UPS_REQUIRE(Kpl >= 1 && Kpl <= K, "step_encode_fwd: %d part planes of K=%d", Kpl, K);
    if (int rc = fused_common_checks("step_encode_fwd", B, P, K)) return rc;
    UPS_REQUIRE((l1_row < K || aligned16(l1)) && aligned16(img1) && aligned16(m1) && aligned16(parts_pm), "step_encode_fwd: 16-byte alignment");
    if (B == 0) return UPS_OK;
    const int per = fused_pix_per_cta(B, P);
    const int splits = (int)cdiv(P, per);
    const size_t need = (size_t)B * splits * K * 3 * sizeof(float);
    if (!ws || ws_bytes < need) { set_error("step_encode_fwd: workspace %zu < %zu bytes", ws_bytes, need); return UPS_E_WORKSPACE; }
    dim3 grid(splits, B);
    cudaStream_t s = as_stream(stream);
    float* partial = static_cast<float*>(ws);
    static const int minb = []() { const char* e = getenv("UPS_ENC_FWD_MINB"); return e ? atoi(e) : 6; }();
#define UPS_ENC_FWD2(LPP, MB)                                                                                 \
    {                                                                                                         \
        const size_t sm = (size_t)FW * EncFwdSmem<LPP>::WREG * sizeof(float);                                 \
        if (Kpl < K) {                                                                                        \
            if (int rc = set_smem(step_encode_fwd_kernel<LPP, MB, true, NOISE, DSEED>, sm)) return rc;               \
            step_encode_fwd_kernel<LPP, MB, true, NOISE, DSEED><<<grid, FTPB, sm, s>>>(l1, img1, m1, parts_pm, partial, B, P, per, Kpl, l1_row, nz); \
        } else {                                                                                              \
            if (int rc = set_smem(step_encode_fwd_kernel<LPP, MB, false, NOISE, DSEED>, sm)) return rc;              \
            step_encode_fwd_kernel<LPP, MB, false, NOISE, DSEED><<<grid, FTPB, sm, s>>>(l1, img1, m1, parts_pm, partial, B, P, per, Kpl, l1_row, nz); \
        }                                                                                                     \
    }
#define UPS_ENC_FWD(LPP) \
    { if (minb == 4) UPS_ENC_FWD2(LPP, 4) else if (minb == 5) UPS_ENC_FWD2(LPP, 5) else UPS_ENC_FWD2(LPP, 6) }
    if (K == 4) UPS_ENC_FWD(1) else if (K == 8) UPS_ENC_FWD(2) else if (K == 16) UPS_ENC_FWD(4) else UPS_ENC_FWD(8)
#undef UPS_ENC_FWD2
#undef UPS_ENC_FWD
    if (int rc = after_launch("step_encode_fwd_kernel")) return rc;
    const long long n = (long long)B * K * 3;
    split_finalize_kernel<<<(unsigned)cdiv(n, 128), 128, 0, s>>>(partial, pooled, K * 3, splits, P, n);
    return after_launch("split_finalize_kernel");
}

extern "C" int ups_step_encode_fwd_rows(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm,
                                        float* pooled, int B, int P, int K, int Kpl, void* ws, size_t ws_bytes,
                                        void* stream) {
    return encode_fwd_launch<false>(l1, l1_row, img1, m1, parts_pm, pooled, B, P, K, Kpl, ws, ws_bytes, NoiseArgs{}, stream);
}

extern "C" int ups_step_encode_fwd_noise(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm,
                                         float* pooled, int B, int P, int K, int Kpl, void* ws, size_t ws_bytes,
                                         unsigned long long seed, long long sample_offset, float noise_level, void* stream) {
    UPS_REQUIRE(sample_offset >= 0, "step_encode_fwd: sample_offset=%lld", sample_offset);
    return encode_fwd_launch<true>(l1, l1_row, img1, m1, parts_pm, pooled, B, P, K, Kpl, ws, ws_bytes,
                                   NoiseArgs{seed, sample_offset, noise_level, 1}, stream);
}

extern "C" int ups_step_encode_fwd_noise_dseed(const float* l1, int l1_row, const float* img1, float* m1, float* parts_pm,
                                               float* pooled, int B, int P, int K, int Kpl, void* ws, size_t ws_bytes,
                                               const unsigned long long* seed, long long sample_offset, float noise_level,
                                               void* stream) {
    UPS_REQUIRE(seed, "step_encode_fwd: null seed pointer");
    UPS_REQUIRE(sample_offset >= 0, "step_encode_fwd: sample_offset=%lld", sample_offset);
    return encode_fwd_launch<true, true>(l1, l1_row, img1, m1, parts_pm, pooled, B, P, K, Kpl, ws, ws_bytes,
                                         NoiseArgs{(unsigned long long)(uintptr_t)seed, sample_offset, noise_level, 1}, stream);
}

extern "C" int ups_step_decode_bwd(const float* g_inj, const float* m0, const float* g_m0, const float* feat,
                                   float* dl0, float* dfeat, int B, int P, int K, int F, void* ws, size_t ws_bytes,
                                   void* stream) {
    return ups_step_decode_bwd_rows(g_inj, m0, g_m0, K, feat, dl0, dfeat, B, P, K, F, ws, ws_bytes, stream);
}

extern "C" int ups_step_decode_bwd_rows(const float* g_inj, const float* m0, const float* g_m0, int gm_row, const float* feat,
                                        float* dl0, float* dfeat, int B, int P, int K, int F, void* ws, size_t ws_bytes,
                                        void* stream) {
    UPS_REQUIRE(g_inj && m0 && feat && dl0 && dfeat, "step_decode_bwd: null pointer");
    UPS_REQUIRE(gm_row >= 1 && gm_row <= K, "step_decode_bwd: g_m0 rows of %d floats for K=%d", gm_row, K);
    if (int rc = fused_common_checks("step_decode_bwd", B, P, K)) return rc;
    UPS_REQUIRE(K >= 8, "step_decode_bwd: fused path needs K in {8,16,32}, got %d", K);
    UPS_REQUIRE(F == 16 || F == 32 || F == 64, "step_decode_bwd: fused path needs F in {16,32,64}, got %d", F);
    UPS_REQUIRE(aligned16(g_inj) && aligned16(feat), "step_decode_bwd: 16-byte alignment");
    if (B == 0) return UPS_OK;
    const int per = fused_pix_per_cta(B, P);
    const int splits = (int)cdiv(P, per);
    const size_t need = (size_t)B * splits * K * F * sizeof(float);
    if (!ws || ws_bytes < need) { set_error("step_decode_bwd: workspace %zu < %zu bytes", ws_bytes, need); return UPS_E_WORKSPACE; }
    dim3 grid(splits, B);
    cudaStream_t s = as_stream(stream);
    float* partial = static_cast<float*>(ws);
#define UPS_DEC_BWD(KK, FF)                                                                                  \
    {                                                                                                        \
        const size_t sm = (size_t)FW * DecBwdSmem<KK, FF>::WREG * sizeof(float);                             \
        if (int rc = set_smem(step_decode_bwd_kernel<KK, FF>, sm)) return rc;                                \
        step_decode_bwd_kernel<KK, FF><<<grid, FTPB, sm, s>>>(g_inj, m0, g_m0, feat, dl0, partial, P, per, gm_row); \
    }
#define UPS_DEC_BWD_F(KK) \
    { if (F == 16) UPS_DEC_BWD(KK, 16) else if (F == 32) UPS_DEC_BWD(KK, 32) else UPS_DEC_BWD(KK, 64) }
    if (K == 8) UPS_DEC_BWD_F(8) else if (K == 16) UPS_DEC_BWD_F(16) else UPS_DEC_BWD_F(32)
#undef UPS_DEC_BWD_F
#undef UPS_DEC_BWD
    if (int rc = after_launch("step_decode_bwd_kernel")) return rc;
    const long long n = (long long)B * K * F;
    split_finalize_kernel<<<(unsigned)cdiv(n, 128), 128, 0, s>>>(partial, dfeat, K * F, splits, 0, n);
    return after_launch("split_finalize_kernel");
}

extern "C" int ups_step_encode_bwd(const float* g_parts_pm, const float* g_pooled, const float* img1, const float* m1,
                                   const float* g_m1, float* dl1, float* dimg1, int B, int P, int K, void* stream) {
    return ups_step_encode_bwd_planes(g_parts_pm, g_pooled, img1, m1, g_m1, dl1, dimg1, B, P, K, K, stream);
}

extern "C" int ups_step_encode_bwd_planes(const float* g_parts_pm, const float* g_pooled, const float* img1, const float* m1,
                                          const float* g_m1, float* dl1, float* dimg1, int B, int P, int K, int Kpl,
                                          void* stream) {
    return ups_step_encode_bwd_rows(g_parts_pm, g_pooled, img1, m1, g_m1, K, dl1, dimg1, B, P, K, Kpl, stream);
}

extern "C" int ups_step_encode_bwd_rows(const float* g_parts_pm, const float* g_pooled, const float* img1, const float* m1,
                                        const float* g_m1, int gm_row, float* dl1, float* dimg1, int B, int P, int K,
                                        int Kpl, void* stream) {
    UPS_REQUIRE(g_parts_pm && img1 && m1 && dl1, "step_encode_bwd: null pointer");
    UPS_REQUIRE(gm_row >= 1 && gm_row <= K, "step_encode_bwd: g_m1 rows of %d floats for K=%d", gm_row, K);
    UPS_REQUIRE(Kpl >= 1 && Kpl <= K, "step_encode_bwd: %d part planes of K=%d", Kpl, K);
    if (int rc = fused_common_checks("step_encode_bwd", B, P, K)) return rc;
    UPS_REQUIRE(aligned16(g_parts_pm) && aligned16(img1) && aligned16(m1) && aligned16(dl1) && (!g_m1 || gm_row < K || aligned16(g_m1)) &&
                    (!dimg1 || aligned16(dimg1)), "step_encode_bwd: 16-byte alignment");
    if (B == 0) return UPS_OK;
    const int per = fused_pix_per_cta(B, P);
    dim3 grid((unsigned)cdiv(P, per), B);
    cudaStream_t s = as_stream(stream);
#define UPS_ENC_BWD3(LPP, DI, PD)                                                                                     \
    {                                                                                                                 \
        if (int rc = set_smem(step_encode_bwd_kernel<LPP, DI, PD>, sm)) return rc;                                    \
        step_encode_bwd_kernel<LPP, DI, PD><<<grid, FTPB, sm, s>>>(g_parts_pm, g_pooled, img1, m1, g_m1, dl1, dimg1, B, P, per, Kpl, gm_row); \
    }
#define UPS_ENC_BWD(LPP)                                                                                              \
    {                                                                                                                 \
        const size_t sm = ((size_t)FW * EncBwdSmem<LPP>::WREG + 4 * LPP * 3 + 4) * sizeof(float);                     \
        if (dimg1) { if (Kpl < K) UPS_ENC_BWD3(LPP, true, true) else UPS_ENC_BWD3(LPP, true, false) }                 \
        else { if (Kpl < K) UPS_ENC_BWD3(LPP, false, true) else UPS_ENC_BWD3(LPP, false, false) }                     \
    }
    if (K == 4) UPS_ENC_BWD(1) else if (K == 8) UPS_ENC_BWD(2) else if (K == 16) UPS_ENC_BWD(4) else UPS_ENC_BWD(8)
#undef UPS_ENC_BWD
#undef UPS_ENC_BWD3
    return after_launch("step_encode_bwd_kernel");
}
