// Stand-alone part-map operators behind the reference's helper signatures
// (cub/code/nn.py:58-168,2086-2089,2469-2487; cub/code/SB_model48i/model.py:176-249;
// deepfashion/code/foo.py:287-307,462-498).  The fused per-step kernels are in step_fused.cu.
#include "common.cuh"

namespace ups {

constexpr int TPB = 256;

// =================================================================== softmax over parts
// Fast path: K = 4*LPP, LPP lanes per pixel, one float4 per lane, fully coalesced.
// MODE: SM_PLAIN softmax(logits); SM_EPS logits = mean + noise*eps first (MeanFieldDistribution.sample,
// cub/code/nn.py:1421-1427), one rounding per step; SM_PHILOX the same with eps drawn in registers (canon_math.cuh, the
// mean-field logit noise; pixel i is global pixel nz.sample_offset + i); SM_PHILOX_DSEED that with the seed read from
// device memory (resolve_seed).
constexpr int SM_PLAIN = 0, SM_EPS = 1, SM_PHILOX = 2, SM_PHILOX_DSEED = 3;
template <int LPP, int UNROLL, int MODE>
__global__ void __launch_bounds__(TPB) part_softmax_fwd_kernel(const float* __restrict__ logits,
                                                               const float* __restrict__ eps, float noise,
                                                               float* __restrict__ logits_out,
                                                               float* __restrict__ probs,
                                                               long long* __restrict__ labels,
                                                               float* __restrict__ hard, long long n4, NoiseArgs nz_arg) {
    // n4 = n_pix * LPP float4s in total; every lane stays alive for the shuffles
    const NoiseArgs nz = resolve_seed<MODE == SM_PHILOX_DSEED>(nz_arg);
    const long long base = ((long long)blockIdx.x * UNROLL) * TPB + threadIdx.x;
    float4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const long long i = base + (long long)u * TPB;
        const long long ii = i < n4 ? i : n4 - 1;
        v[u] = ld4_stream(logits + 4 * ii);
        if (MODE == SM_EPS) {
            const float4 e = ld4_stream(eps + 4 * ii);
            v[u] = make_float4(__fadd_rn(v[u].x, __fmul_rn(noise, e.x)), __fadd_rn(v[u].y, __fmul_rn(noise, e.y)),
                               __fadd_rn(v[u].z, __fmul_rn(noise, e.z)), __fadd_rn(v[u].w, __fmul_rn(noise, e.w)));
        }
        if (MODE >= SM_PHILOX) {
            float z0, z1, z2, z3;
            normal4_philox(nz.seed, (uint32_t)nz.draw, (unsigned long long)(nz.sample_offset + ii / LPP),
                           (uint32_t)(ii & (LPP - 1)), z0, z1, z2, z3);
            v[u] = make_float4(sampled_logit(v[u].x, nz.level, z0), sampled_logit(v[u].y, nz.level, z1),
                               sampled_logit(v[u].z, nz.level, z2), sampled_logit(v[u].w, nz.level, z3));
        }
        if (MODE != SM_PLAIN && logits_out && i < n4) st4(logits_out + 4 * i, v[u]);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const long long i = base + (long long)u * TPB;
        const int c = (int)(i & (LPP - 1));
        float pmax; int arg, nmax;
        const float4 p = softmax4<LPP>(v[u], c, pmax, arg, nmax);
        if (i < n4) {
            st4(probs + 4 * i, p);
            if (hard) st4(hard + 4 * i, hard_st4(p, pmax));
            if (labels && c == 0) labels[i / LPP] = arg;
        }
    }
}

// Generic K (e.g. the reference's shipped n_parts = 25): one thread per pixel.  MODE as part_softmax_fwd_kernel's
// (SM_PLAIN and SM_EPS share one instantiation: the eps mode is the run-time `eps != nullptr`).
template <int MODE>
__global__ void __launch_bounds__(128) part_softmax_fwd_generic_kernel(const float* __restrict__ logits,
                                                                       const float* __restrict__ eps, float noise,
                                                                       float* __restrict__ logits_out,
                                                                       float* __restrict__ probs,
                                                                       long long* __restrict__ labels,
                                                                       float* __restrict__ hard, long long n_pix,
                                                                       int K, NoiseArgs nz_arg) {
    const NoiseArgs nz = resolve_seed<MODE == SM_PHILOX_DSEED>(nz_arg);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pix) return;
    float x[KMAX], p[KMAX], e[KMAX];
    for (int k = 0; k < K; ++k) x[k] = logits[i * K + k];
    if (MODE < SM_PHILOX && eps) {
        for (int k = 0; k < K; ++k) {
            x[k] = __fadd_rn(x[k], __fmul_rn(noise, eps[i * K + k]));
            if (logits_out) logits_out[i * K + k] = x[k];
        }
    }
    if (MODE >= SM_PHILOX) {
        for (int j = 0; 4 * j < K; ++j) {
            float z[4];
            normal4_philox(nz.seed, (uint32_t)nz.draw, (unsigned long long)(nz.sample_offset + i), (uint32_t)j, z[0], z[1],
                           z[2], z[3]);
            for (int l = 0; l < 4 && 4 * j + l < K; ++l) x[4 * j + l] = sampled_logit(x[4 * j + l], nz.level, z[l]);
        }
        if (logits_out)
            for (int k = 0; k < K; ++k) logits_out[i * K + k] = x[k];
    }
    const float pmax = softmax_row_canon(x, p, e, K);
    int arg = -1;
    for (int k = 0; k < K; ++k) {
        probs[i * K + k] = p[k];
        if (p[k] == pmax && arg < 0) arg = k;
        if (hard) hard[i * K + k] = st_value(p[k] == pmax ? 1.0f : 0.0f, p[k]);
    }
    if (labels) labels[i] = arg;
}

template <int LPP>
__global__ void __launch_bounds__(TPB) part_softmax_bwd_kernel(const float* __restrict__ probs,
                                                               const float* __restrict__ g,
                                                               const float* __restrict__ g2,
                                                               const float* __restrict__ g3,
                                                               float* __restrict__ dlogits, long long n4) {
    const long long i = (long long)blockIdx.x * TPB + threadIdx.x;
    const long long ii = i < n4 ? i : n4 - 1;
    const float4 p = ld4_stream(probs + 4 * ii);
    float4 gg = ld4_stream(g + 4 * ii);
    if (g2) { const float4 t = ld4_stream(g2 + 4 * ii); gg.x += t.x; gg.y += t.y; gg.z += t.z; gg.w += t.w; }
    if (g3) { const float4 t = ld4_stream(g3 + 4 * ii); gg.x += t.x; gg.y += t.y; gg.z += t.z; gg.w += t.w; }
    float dot = p.x * gg.x + p.y * gg.y + p.z * gg.z + p.w * gg.w;
    dot = group_sum<LPP>(dot);
    if (i < n4) st4(dlogits + 4 * i, make_float4(p.x * (gg.x - dot), p.y * (gg.y - dot), p.z * (gg.z - dot), p.w * (gg.w - dot)));
}

__global__ void part_softmax_bwd_generic_kernel(const float* __restrict__ probs, const float* __restrict__ g,
                                                const float* __restrict__ g2, const float* __restrict__ g3,
                                                float* __restrict__ dlogits, long long n_pix, int K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pix) return;
    auto gsum = [&](long long j) {
        float v = g[j];
        if (g2) v += g2[j];
        if (g3) v += g3[j];
        return v;
    };
    float dot = 0.f;
    for (int k = 0; k < K; ++k) dot += probs[i * K + k] * gsum(i * K + k);
    for (int k = 0; k < K; ++k) dlogits[i * K + k] = probs[i * K + k] * (gsum(i * K + k) - dot);
}

// eps [n_pix, K] of global pixels pix_offset + i: one thread per (pixel, group of 4 parts); DSEED: see resolve_seed
template <bool DSEED>
__global__ void __launch_bounds__(TPB) normal_philox_kernel(float* __restrict__ out, long long n, int J, int K,
                                                            NoiseArgs nz_arg) {
    const NoiseArgs nz = resolve_seed<DSEED>(nz_arg);
    const long long t = (long long)blockIdx.x * TPB + threadIdx.x;   // over n_pix * J
    if (t >= n) return;
    const long long i = t / J;
    const int j = (int)(t - i * J);
    float z[4];
    normal4_philox(nz.seed, (uint32_t)nz.draw, (unsigned long long)(nz.sample_offset + i), (uint32_t)j, z[0], z[1], z[2], z[3]);
    float* o = out + i * K + 4 * j;
    if (4 * j + 4 <= K && (K & 3) == 0) {
        st4_stream(o, make_float4(z[0], z[1], z[2], z[3]));
    } else {
        for (int l = 0; l < 4 && 4 * j + l < K; ++l) __stcs(o + l, z[l]);
    }
}

// y += a*x  and  out[v] = g[v] (or 0) + (v == idx ? extra : 0): the two elementwise sums of the unfused step
__global__ void axpy_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, float a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = fmaf(a, x[i], y[i]);
}
__global__ void views_cotangent_kernel(const float* __restrict__ g, const float* __restrict__ extra,
                                       float* __restrict__ out, int idx, long long n_per_view, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long v = i / n_per_view;
    float r = g ? g[i] : 0.f;
    if (v == idx && extra) r += extra[i - v * n_per_view];
    out[i] = r;
}

// =================================================================== spatial softmax (nn.py:65-71)
// x [N,P,C]: softmax over P for every (n,c).  One CTA per sample; thread (r,c) strides rows.
constexpr int SS_TPB = 512;
__global__ void __launch_bounds__(SS_TPB) spatial_softmax_fwd_kernel(const float* __restrict__ x,
                                                                     float* __restrict__ probs, int P, int C) {
    extern __shared__ float red[];  // SS_TPB floats
    const int n = blockIdx.x;
    const int R = SS_TPB / C;  // row groups
    const int c = threadIdx.x % C, r = threadIdx.x / C;
    const bool live = r < R;
    const float* xb = x + (size_t)n * P * C;
    float* pb = probs + (size_t)n * P * C;
    float m = -INFINITY;
    if (live) for (int p = r; p < P; p += R) m = fmaxf(m, xb[(size_t)p * C + c]);
    red[threadIdx.x] = m;
    __syncthreads();
    if (r == 0) { for (int q = 1; q < R; ++q) m = fmaxf(m, red[q * C + c]); red[c] = m; }
    __syncthreads();
    m = red[c];
    __syncthreads();
    float s = 0.f;
    if (live) for (int p = r; p < P; p += R) s += expf(xb[(size_t)p * C + c] - m);
    red[threadIdx.x] = s;
    __syncthreads();
    if (r == 0) { for (int q = 1; q < R; ++q) s += red[q * C + c]; red[c] = s; }
    __syncthreads();
    s = red[c];
    if (live) for (int p = r; p < P; p += R) pb[(size_t)p * C + c] = expf(xb[(size_t)p * C + c] - m) / s;
}

__global__ void __launch_bounds__(SS_TPB) spatial_softmax_bwd_kernel(const float* __restrict__ probs,
                                                                     const float* __restrict__ g,
                                                                     float* __restrict__ dx, int P, int C) {
    extern __shared__ float red[];
    const int n = blockIdx.x;
    const int R = SS_TPB / C;
    const int c = threadIdx.x % C, r = threadIdx.x / C;
    const bool live = r < R;
    const size_t o = (size_t)n * P * C;
    float s = 0.f;
    if (live) for (int p = r; p < P; p += R) s += probs[o + (size_t)p * C + c] * g[o + (size_t)p * C + c];
    red[threadIdx.x] = s;
    __syncthreads();
    if (r == 0) { for (int q = 1; q < R; ++q) s += red[q * C + c]; red[c] = s; }
    __syncthreads();
    s = red[c];
    if (live) for (int p = r; p < P; p += R) {
        const size_t i = o + (size_t)p * C + c;
        dx[i] = probs[i] * (g[i] - s);
    }
}

// =================================================================== hard_max / ST / argmax / one_hot
__global__ void hard_max_kernel(const float* __restrict__ y, float* __restrict__ out, long long n_pix, int K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pix) return;
    float m = y[i * K];
    for (int k = 1; k < K; ++k) m = fmaxf(m, y[i * K + k]);
    for (int k = 0; k < K; ++k) out[i * K + k] = (y[i * K + k] == m) ? 1.0f : 0.0f;
}

__global__ void straight_through_kernel(const float* __restrict__ h, const float* __restrict__ y,
                                        float* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = st_value(h[i], y[i]);
}

__global__ void argmax_kernel(const float* __restrict__ y, long long* __restrict__ labels, long long n_pix, int K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pix) return;
    float m = y[i * K]; int a = 0;
    for (int k = 1; k < K; ++k) { const float v = y[i * K + k]; if (v > m) { m = v; a = k; } }
    labels[i] = a;
}

__global__ void one_hot_kernel(const long long* __restrict__ labels, float* __restrict__ out, long long n, int K) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over n_pix*K
    if (i < n) out[i] = (labels[i / K] == (i % K)) ? 1.0f : 0.0f;
}

// =================================================================== mask_parts (model.py:176-187)
__global__ void mask_parts_fwd_kernel(const float* __restrict__ image, const float* __restrict__ mask,
                                      float* __restrict__ parts, int B, int P, int K, int C, int part_major,
                                      long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long bp; int k, c;
    if (!part_major) {  // [B,P,K,C]
        c = (int)(i % C); k = (int)((i / C) % K); bp = i / ((long long)C * K);
    } else {            // [K,B,P,C]
        c = (int)(i % C); bp = (i / C) % ((long long)B * P); k = (int)(i / ((long long)C * B * P));
    }
    parts[i] = image[bp * C + c] * mask[bp * K + k];
}

__device__ __forceinline__ long long parts_index(long long bp, int k, int c, int B, int P, int K, int C, int pm) {
    return pm ? (((long long)k * B * P + bp) * C + c) : ((bp * K + k) * C + c);
}

__global__ void mask_parts_bwd_dmask_kernel(const float* __restrict__ g, const float* __restrict__ image,
                                            float* __restrict__ dmask, int B, int P, int K, int C, int pm,
                                            long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*P*K
    if (i >= n) return;
    const long long bp = i / K; const int k = (int)(i % K);
    float s = 0.f;
    for (int c = 0; c < C; ++c) s += g[parts_index(bp, k, c, B, P, K, C, pm)] * image[bp * C + c];
    dmask[i] = s;
}

__global__ void mask_parts_bwd_dimage_kernel(const float* __restrict__ g, const float* __restrict__ mask,
                                             float* __restrict__ dimage, int B, int P, int K, int C, int pm,
                                             long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*P*C
    if (i >= n) return;
    const long long bp = i / C; const int c = (int)(i % C);
    float s = 0.f;
    for (int k = 0; k < K; ++k) s += g[parts_index(bp, k, c, B, P, K, C, pm)] * mask[bp * K + k];
    dimage[i] = s;
}

// nn.apply_partwise transposes (nn.py:100-103,108-112): [B,P,K,C] <-> [K,B,P,C]
__global__ void partwise_fold_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int P, int K, int C,
                                     long long n, int unfold) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // index into the [K,B,P,C] side
    if (i >= n) return;
    const int c = (int)(i % C);
    const long long bp = (i / C) % ((long long)B * P);
    const int k = (int)(i / ((long long)C * B * P));
    const long long j = (bp * K + k) * C + c;  // index into the [B,P,K,C] side
    if (unfold) y[j] = x[i]; else y[i] = x[j];
}

// =================================================================== mask-weighted pooling
// out[b,k,f] = scale * sum_p fmap[b,p, (grouped? k*Fg : 0) + f] * mask[b,p,k]
// Stage 1: CTA = (split, b); each warp strides the pixels of its split, lanes own the (k,f)
// pairs j = lane + 32*a in NACC register accumulators; fixed-order cross-warp reduction.
// Stage 2: pool_finalize_kernel sums the splits in ascending order (deterministic).
constexpr int POOL_WARPS = 8;
template <int NACC>
__global__ void __launch_bounds__(POOL_WARPS * 32) part_pool_partial_kernel(
    const float* __restrict__ fmap, const float* __restrict__ mask, float* __restrict__ partial, int P, int K, int Fg,
    int grouped, int fmap_stride, int splits, int k0, int kc) {
    // this launch covers parts [k0, k0+kc): KFc = kc*Fg <= 32*NACC (k,f) pairs
    extern __shared__ float sm[];  // POOL_WARPS * KFc
    const int KF = K * Fg, KFc = kc * Fg;
    const int b = blockIdx.y, sp = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per = (P + splits - 1) / splits;
    const int p0 = sp * per, p1 = min(P, p0 + per);
    float acc[NACC];
    int kk[NACC], ff[NACC];
#pragma unroll
    for (int a = 0; a < NACC; ++a) {
        acc[a] = 0.f;
        const int j = lane + 32 * a;
        kk[a] = j < KFc ? k0 + j / Fg : 0;
        ff[a] = j < KFc ? (grouped ? k0 * Fg + j : j % Fg) : 0;
    }
    for (int p = p0 + warp; p < p1; p += POOL_WARPS) {
        const float* fr = fmap + ((size_t)b * P + p) * fmap_stride;
        const float* mr = mask + ((size_t)b * P + p) * K;
#pragma unroll
        for (int a = 0; a < NACC; ++a)
            if (lane + 32 * a < KFc) acc[a] = fmaf(__ldg(fr + ff[a]), __ldg(mr + kk[a]), acc[a]);
    }
#pragma unroll
    for (int a = 0; a < NACC; ++a)
        if (lane + 32 * a < KFc) sm[warp * KFc + lane + 32 * a] = acc[a];
    __syncthreads();
    for (int j = threadIdx.x; j < KFc; j += POOL_WARPS * 32) {
        float s = sm[j];
        for (int w = 1; w < POOL_WARPS; ++w) s += sm[w * KFc + j];
        partial[((size_t)b * splits + sp) * KF + k0 * Fg + j] = s;
    }
}

__global__ void pool_finalize_kernel(const float* __restrict__ partial, float* __restrict__ out, int KF, int splits,
                                     float scale, int divide_by, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*KF
    if (i >= n) return;
    const long long b = i / KF; const int j = (int)(i % KF);
    float s = 0.f;
    for (int sp = 0; sp < splits; ++sp) s += partial[((size_t)b * splits + sp) * KF + j];
    out[i] = divide_by > 0 ? s / (float)divide_by : s * scale;
}

__global__ void part_pool_bwd_dfmap_kernel(const float* __restrict__ g, const float* __restrict__ mask,
                                           float* __restrict__ dfmap, int P, int K, int Fg, int grouped, float scale,
                                           long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*P*(grouped? K*Fg : Fg)
    if (i >= n) return;
    const int row = grouped ? K * Fg : Fg;
    const long long bp = i / row; const int j = (int)(i % row);
    const long long b = bp / P;
    if (grouped) {
        const int k = j / Fg;
        dfmap[i] = scale * g[b * K * Fg + j] * mask[bp * K + k];
    } else {
        float s = 0.f;
        for (int k = 0; k < K; ++k) s = fmaf(g[(b * K + k) * Fg + j], mask[bp * K + k], s);
        dfmap[i] = scale * s;
    }
}

__global__ void part_pool_bwd_dmask_kernel(const float* __restrict__ g, const float* __restrict__ fmap,
                                           float* __restrict__ dmask, int P, int K, int Fg, int grouped,
                                           int fmap_stride, float scale, const float* __restrict__ extra,
                                           int extra_stride, int extra_off, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*P*K
    if (i >= n) return;
    const long long bp = i / K; const int k = (int)(i % K);
    const long long b = bp / P;
    const float* fr = fmap + bp * fmap_stride + (grouped ? k * Fg : 0);
    const float* gr = g + (b * K + k) * Fg;
    float s = 0.f;
    for (int f = 0; f < Fg; ++f) s = fmaf(gr[f], fr[f], s);
    s *= scale;
    if (extra) s += extra[bp * extra_stride + extra_off + k];
    dmask[i] = s;
}

// =================================================================== unpool / inject / gather
__global__ void part_unpool_fwd_kernel(const float* __restrict__ feat, const float* __restrict__ mask,
                                       float* __restrict__ out, int P, int K, int F, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*P*K*F
    if (i >= n) return;
    const int f = (int)(i % F); const int k = (int)((i / F) % K);
    const long long bp = i / ((long long)F * K); const long long b = bp / P;
    out[i] = mask[bp * K + k] * feat[(b * K + k) * F + f];
}

// inj[b,p,f] = sum_k mask*feat (ascending k), inj[b,p,F+k] = mask.  One warp per pixel,
// feat[b] staged in shared memory; zero mask entries are skipped (warp-uniform branch).
constexpr int INJ_TPB = 256;
constexpr int INJ_PIX = 64;  // pixels per CTA
__global__ void __launch_bounds__(INJ_TPB) part_inject_fwd_kernel(const float* __restrict__ feat,
                                                                  const float* __restrict__ mask,
                                                                  float* __restrict__ inj, int P, int K, int F) {
    extern __shared__ float fs[];  // K*F
    const int b = blockIdx.y;
    for (int i = threadIdx.x; i < K * F; i += INJ_TPB) fs[i] = feat[(size_t)b * K * F + i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p0 = blockIdx.x * INJ_PIX;
    for (int pl = warp; pl < INJ_PIX; pl += INJ_TPB / 32) {
        const int p = p0 + pl;
        if (p >= P) break;
        const float* mr = mask + ((size_t)b * P + p) * K;
        float* orow = inj + ((size_t)b * P + p) * (F + K);
        for (int f0 = 0; f0 < F; f0 += 32) {
            const int f = f0 + lane;
            float acc = 0.f;
            for (int k = 0; k < K; ++k) {
                const float m = __ldg(mr + k);
                if (m != 0.f && f < F) acc = fmaf(m, fs[k * F + f], acc);
            }
            if (f < F) orow[f] = acc;
        }
        for (int k = lane; k < K; k += 32) orow[F + k] = __ldg(mr + k);
    }
}

__global__ void part_gather_fwd_kernel(const float* __restrict__ feat, const long long* __restrict__ labels,
                                       float* __restrict__ out, int P, int K, int F, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*P*F
    if (i >= n) return;
    const int f = (int)(i % F); const long long bp = i / F; const long long b = bp / P;
    long long k = labels[bp];
    k = k < 0 ? 0 : (k >= K ? K - 1 : k);
    out[i] = feat[(b * K + k) * F + f];
}

}  // namespace ups

using namespace ups;

static inline unsigned nblk(long long n, int tpb) { return (unsigned)cdiv(n, tpb); }
#define UPS_GRID_OK(n, tpb) UPS_REQUIRE(cdiv((n), (tpb)) < (1ll << 31), "problem too large for one launch")

// nz != nullptr: the philox mode (eps == nullptr; dseed: nz->seed is the seed's device address); eps != nullptr: the eps
// mode; neither: plain softmax
static int part_softmax_fwd_impl(const char* what, const float* logits, const float* eps, float noise,
                                 float* logits_out, float* probs, long long* labels, float* hard_st, long long n_pix,
                                 int K, void* stream, const NoiseArgs* nz = nullptr, bool dseed = false) {
    UPS_REQUIRE(logits && probs, "%s: null pointer", what);
    UPS_REQUIRE(n_pix >= 0 && K >= 1 && K <= KMAX, "%s: n_pix=%lld K=%d (1..%d)", what, n_pix, K, KMAX);
    if (n_pix == 0) return UPS_OK;
    cudaStream_t s = as_stream(stream);
    const bool vec = aligned16(logits) && aligned16(probs) && (!hard_st || aligned16(hard_st)) && aligned16(eps) &&
                     aligned16(logits_out);
    constexpr int U = 4;
#define UPS_SM_FWD(LPP)                                                                                              \
    {                                                                                                                \
        const long long n4 = n_pix * LPP;                                                                            \
        UPS_GRID_OK(n4, TPB * U);                                                                                    \
        if (nz && dseed)                                                                                             \
            part_softmax_fwd_kernel<LPP, U, SM_PHILOX_DSEED><<<nblk(n4, TPB * U), TPB, 0, s>>>(                      \
                logits, nullptr, 0.f, logits_out, probs, labels, hard_st, n4, *nz);                                  \
        else if (nz)                                                                                                 \
            part_softmax_fwd_kernel<LPP, U, SM_PHILOX><<<nblk(n4, TPB * U), TPB, 0, s>>>(                            \
                logits, nullptr, 0.f, logits_out, probs, labels, hard_st, n4, *nz);                                  \
        else if (eps)                                                                                                \
            part_softmax_fwd_kernel<LPP, U, SM_EPS><<<nblk(n4, TPB * U), TPB, 0, s>>>(logits, eps, noise, logits_out, \
                                                                                      probs, labels, hard_st, n4,    \
                                                                                      NoiseArgs{});                  \
        else                                                                                                         \
            part_softmax_fwd_kernel<LPP, U, SM_PLAIN><<<nblk(n4, TPB * U), TPB, 0, s>>>(                             \
                logits, nullptr, 0.f, nullptr, probs, labels, hard_st, n4, NoiseArgs{});                             \
        return after_launch("part_softmax_fwd_kernel");                                                              \
    }
    if (vec && K == 4) UPS_SM_FWD(1)
    if (vec && K == 8) UPS_SM_FWD(2)
    if (vec && K == 16) UPS_SM_FWD(4)
    if (vec && K == 32) UPS_SM_FWD(8)
#undef UPS_SM_FWD
    UPS_GRID_OK(n_pix, 128);
    if (nz && dseed)
        part_softmax_fwd_generic_kernel<SM_PHILOX_DSEED><<<nblk(n_pix, 128), 128, 0, s>>>(logits, nullptr, 0.f, logits_out,
                                                                                      probs, labels, hard_st, n_pix, K, *nz);
    else if (nz)
        part_softmax_fwd_generic_kernel<SM_PHILOX><<<nblk(n_pix, 128), 128, 0, s>>>(logits, nullptr, 0.f, logits_out, probs,
                                                                                labels, hard_st, n_pix, K, *nz);
    else
        part_softmax_fwd_generic_kernel<SM_PLAIN><<<nblk(n_pix, 128), 128, 0, s>>>(logits, eps, noise, logits_out, probs,
                                                                               labels, hard_st, n_pix, K, NoiseArgs{});
    return after_launch("part_softmax_fwd_generic_kernel");
}

extern "C" int ups_part_softmax_fwd(const float* logits, float* probs, long long* labels, float* hard_st,
                                    long long n_pix, int K, void* stream) {
    return part_softmax_fwd_impl("part_softmax_fwd", logits, nullptr, 0.f, nullptr, probs, labels, hard_st, n_pix, K,
                                 stream);
}

extern "C" int ups_part_softmax_sampled_fwd(const float* mean, const float* eps, float noise_level, float* logits_out,
                                            float* probs, int64_t* labels, float* hard_st, long long n_pix, int K,
                                            void* stream) {
    UPS_REQUIRE(eps, "part_softmax_sampled_fwd: null pointer");
    return part_softmax_fwd_impl("part_softmax_sampled_fwd", mean, eps, noise_level, logits_out, probs,
                                 reinterpret_cast<long long*>(labels), hard_st, n_pix, K, stream);
}

extern "C" int ups_part_softmax_sampled_philox_fwd(const float* mean, unsigned long long seed, int draw, long long pix_offset,
                                                   float noise_level, float* logits_out, float* probs, int64_t* labels,
                                                   float* hard_st, long long n_pix, int K, void* stream) {
    UPS_REQUIRE(draw >= 0 && pix_offset >= 0, "part_softmax_sampled_philox_fwd: draw=%d pix_offset=%lld", draw, pix_offset);
    const NoiseArgs nz{seed, pix_offset, noise_level, draw};
    return part_softmax_fwd_impl("part_softmax_sampled_philox_fwd", mean, nullptr, 0.f, logits_out, probs,
                                 reinterpret_cast<long long*>(labels), hard_st, n_pix, K, stream, &nz);
}

extern "C" int ups_part_softmax_sampled_philox_fwd_dseed(const float* mean, const unsigned long long* seed, int draw,
                                                         long long pix_offset, float noise_level, float* logits_out,
                                                         float* probs, int64_t* labels, float* hard_st, long long n_pix, int K,
                                                         void* stream) {
    UPS_REQUIRE(seed, "part_softmax_sampled_philox_fwd: null seed pointer");
    UPS_REQUIRE(draw >= 0 && pix_offset >= 0, "part_softmax_sampled_philox_fwd: draw=%d pix_offset=%lld", draw, pix_offset);
    const NoiseArgs nz{(unsigned long long)(uintptr_t)seed, pix_offset, noise_level, draw};
    return part_softmax_fwd_impl("part_softmax_sampled_philox_fwd", mean, nullptr, 0.f, logits_out, probs,
                                 reinterpret_cast<long long*>(labels), hard_st, n_pix, K, stream, &nz, true);
}

// seed: the value (DSEED = false) or its device address
template <bool DSEED>
static int normal_philox_launch(unsigned long long seed, int draw, long long pix_offset, long long n_pix, int K, float* out,
                                void* stream) {
    UPS_REQUIRE(out, "normal_philox_fwd: null pointer");
    UPS_REQUIRE(n_pix >= 0 && K >= 1 && draw >= 0 && pix_offset >= 0, "normal_philox_fwd: n_pix=%lld K=%d draw=%d pix_offset=%lld",
                n_pix, K, draw, pix_offset);
    UPS_REQUIRE((K & 3) != 0 || aligned16(out), "normal_philox_fwd: 16-byte alignment");
    if (n_pix == 0) return UPS_OK;
    const int J = (K + 3) / 4;
    const long long n = n_pix * J;
    UPS_GRID_OK(n, TPB);
    normal_philox_kernel<DSEED><<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(out, n, J, K, NoiseArgs{seed, pix_offset, 1.0f, draw});
    return after_launch("normal_philox_kernel");
}

extern "C" int ups_normal_philox_fwd(unsigned long long seed, int draw, long long pix_offset, long long n_pix, int K, float* out,
                                     void* stream) {
    return normal_philox_launch<false>(seed, draw, pix_offset, n_pix, K, out, stream);
}

extern "C" int ups_normal_philox_fwd_dseed(const unsigned long long* seed, int draw, long long pix_offset, long long n_pix, int K,
                                           float* out, void* stream) {
    UPS_REQUIRE(seed, "normal_philox_fwd: null seed pointer");
    return normal_philox_launch<true>((unsigned long long)(uintptr_t)seed, draw, pix_offset, n_pix, K, out, stream);
}

extern "C" int ups_part_softmax_bwd(const float* probs, const float* g, float* dlogits, long long n_pix, int K,
                                    void* stream) {
    return ups_part_softmax_bwd2(probs, g, nullptr, nullptr, dlogits, n_pix, K, stream);
}

// dst[r, 0:n_cols] = src[r, 0:n_cols]; dst[r, n_cols:n_cols+n_fill] = fill.  Row strides in floats.
__global__ void copy_rows_kernel(const float* __restrict__ src, long long src_stride, float* __restrict__ dst,
                                 long long dst_stride, long long n_rows, int n_cols, int n_fill, float fill) {
    const int wd = n_cols + n_fill;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows * wd) return;
    const long long r = i / wd;
    const int c = (int)(i - r * wd);
    dst[r * dst_stride + c] = c < n_cols ? __ldcs(src + r * src_stride + c) : fill;
}

// the same copy with 16-byte accesses on the side whose rows are 16-byte aligned (PAD: the destination, row width
// n_cols + n_fill; !PAD: the source, n_fill == 0): one thread per float4 of the aligned rows, 32-bit index arithmetic
template <bool PAD>
__global__ void copy_rows_vec_kernel(const float* __restrict__ src, unsigned src_stride, float* __restrict__ dst,
                                     unsigned dst_stride, unsigned n_chunks_total, unsigned chunks, int n_cols, float fill) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_chunks_total) return;
    const unsigned r = i / chunks, c0 = 4 * (i - r * chunks);
    if (PAD) {
        const float* sp = src + (size_t)r * src_stride + c0;
        float4 v;
        v.x = (int)c0 < n_cols ? __ldcs(sp) : fill;
        v.y = (int)c0 + 1 < n_cols ? __ldcs(sp + 1) : fill;
        v.z = (int)c0 + 2 < n_cols ? __ldcs(sp + 2) : fill;
        v.w = (int)c0 + 3 < n_cols ? __ldcs(sp + 3) : fill;
        st4_stream(dst + (size_t)r * dst_stride + c0, v);
    } else {
        const float4 v = ld4_stream(src + (size_t)r * src_stride + c0);
        float* dp = dst + (size_t)r * dst_stride + c0;
        if ((int)c0 < n_cols) __stcs(dp, v.x);
        if ((int)c0 + 1 < n_cols) __stcs(dp + 1, v.y);
        if ((int)c0 + 2 < n_cols) __stcs(dp + 2, v.z);
        if ((int)c0 + 3 < n_cols) __stcs(dp + 3, v.w);
    }
}

extern "C" int ups_copy_rows(const float* src, long long src_stride, float* dst, long long dst_stride, long long n_rows,
                             int n_cols, int n_fill, float fill, void* stream) {
    UPS_REQUIRE(n_rows >= 0 && n_cols >= 0 && n_fill >= 0, "copy_rows: bad sizes");
    const long long n = n_rows * (n_cols + n_fill);
    if (n == 0) return UPS_OK;
    UPS_REQUIRE(dst && (src || n_cols == 0), "copy_rows: null pointer");
    UPS_REQUIRE(src_stride >= n_cols && dst_stride >= n_cols + n_fill, "copy_rows: row strides smaller than the rows");
    {
        const int wd = n_cols + n_fill;
        const bool small = src_stride < (1ll << 31) && dst_stride < (1ll << 31);
        // pad: the destination rows are whole float4s
        if (small && wd % 4 == 0 && dst_stride % 4 == 0 && aligned16(dst) && n_rows * (wd / 4) < (1ll << 31)) {
            const unsigned chunks = (unsigned)(wd / 4), total = (unsigned)(n_rows * chunks);
            copy_rows_vec_kernel<true><<<(total + TPB - 1) / TPB, TPB, 0, as_stream(stream)>>>(
                src, (unsigned)src_stride, dst, (unsigned)dst_stride, total, chunks, n_cols, fill);
            return after_launch("copy_rows_vec_kernel");
        }
        // cut: the source rows are whole float4s and nothing is filled
        if (small && n_fill == 0 && src_stride % 4 == 0 && aligned16(src) && n_rows * ((n_cols + 3) / 4) < (1ll << 31)) {
            const unsigned chunks = (unsigned)((n_cols + 3) / 4), total = (unsigned)(n_rows * chunks);
            copy_rows_vec_kernel<false><<<(total + TPB - 1) / TPB, TPB, 0, as_stream(stream)>>>(
                src, (unsigned)src_stride, dst, (unsigned)dst_stride, total, chunks, n_cols, fill);
            return after_launch("copy_rows_vec_kernel");
        }
    }
    UPS_GRID_OK(n, TPB);
    copy_rows_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(src, src_stride, dst, dst_stride, n_rows, n_cols, n_fill, fill);
    return after_launch("copy_rows_kernel");
}

extern "C" int ups_axpy(const float* x, float* y, long long n, float a, void* stream) {
    UPS_REQUIRE(x && y && n >= 0, "axpy: null pointer");
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    axpy_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(x, y, n, a);
    return after_launch("axpy_kernel");
}

extern "C" int ups_views_cotangent(const float* g_views, const float* extra, float* out, int V, int idx,
                                   long long n_per_view, void* stream) {
    UPS_REQUIRE(out && V >= 1 && n_per_view >= 0 && idx >= 0 && idx < V, "views_cotangent: bad arguments");
    const long long n = (long long)V * n_per_view;
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    views_cotangent_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(g_views, extra, out, idx, n_per_view, n);
    return after_launch("views_cotangent_kernel");
}

extern "C" int ups_part_softmax_bwd2(const float* probs, const float* g, const float* g2, const float* g3,
                                     float* dlogits, long long n_pix, int K, void* stream) {
    UPS_REQUIRE(probs && g && dlogits, "part_softmax_bwd: null pointer");
    UPS_REQUIRE(n_pix >= 0 && K >= 1, "part_softmax_bwd: n_pix=%lld K=%d", n_pix, K);
    if (n_pix == 0) return UPS_OK;
    cudaStream_t s = as_stream(stream);
    const bool vec = aligned16(probs) && aligned16(g) && aligned16(dlogits) && (!g2 || aligned16(g2)) && (!g3 || aligned16(g3));
#define UPS_SM_BWD(LPP)                                                                              \
    {                                                                                                \
        const long long n4 = n_pix * LPP;                                                            \
        UPS_GRID_OK(n4, TPB);                                                                        \
        part_softmax_bwd_kernel<LPP><<<nblk(n4, TPB), TPB, 0, s>>>(probs, g, g2, g3, dlogits, n4);   \
        return after_launch("part_softmax_bwd_kernel");                                              \
    }
    if (vec && K == 4) UPS_SM_BWD(1)
    if (vec && K == 8) UPS_SM_BWD(2)
    if (vec && K == 16) UPS_SM_BWD(4)
    if (vec && K == 32) UPS_SM_BWD(8)
#undef UPS_SM_BWD
    UPS_GRID_OK(n_pix, TPB);
    part_softmax_bwd_generic_kernel<<<nblk(n_pix, TPB), TPB, 0, s>>>(probs, g, g2, g3, dlogits, n_pix, K);
    return after_launch("part_softmax_bwd_generic_kernel");
}

extern "C" int ups_spatial_softmax_fwd(const float* x, float* probs, int N, int P, int C, void* stream) {
    UPS_REQUIRE(x && probs, "spatial_softmax_fwd: null pointer");
    UPS_REQUIRE(N >= 0 && P >= 1 && C >= 1 && C <= SS_TPB, "spatial_softmax_fwd: N=%d P=%d C=%d", N, P, C);
    if (N == 0) return UPS_OK;
    spatial_softmax_fwd_kernel<<<N, SS_TPB, SS_TPB * sizeof(float), as_stream(stream)>>>(x, probs, P, C);
    return after_launch("spatial_softmax_fwd_kernel");
}

extern "C" int ups_spatial_softmax_bwd(const float* probs, const float* g, float* dx, int N, int P, int C,
                                       void* stream) {
    UPS_REQUIRE(probs && g && dx, "spatial_softmax_bwd: null pointer");
    UPS_REQUIRE(N >= 0 && P >= 1 && C >= 1 && C <= SS_TPB, "spatial_softmax_bwd: N=%d P=%d C=%d", N, P, C);
    if (N == 0) return UPS_OK;
    spatial_softmax_bwd_kernel<<<N, SS_TPB, SS_TPB * sizeof(float), as_stream(stream)>>>(probs, g, dx, P, C);
    return after_launch("spatial_softmax_bwd_kernel");
}

extern "C" int ups_hard_max_fwd(const float* y, float* out, long long n_pix, int K, void* stream) {
    UPS_REQUIRE(y && out, "hard_max_fwd: null pointer");
    UPS_REQUIRE(n_pix >= 0 && K >= 1, "hard_max_fwd: n_pix=%lld K=%d", n_pix, K);
    if (n_pix == 0) return UPS_OK;
    UPS_GRID_OK(n_pix, TPB);
    hard_max_kernel<<<nblk(n_pix, TPB), TPB, 0, as_stream(stream)>>>(y, out, n_pix, K);
    return after_launch("hard_max_kernel");
}

extern "C" int ups_straight_through_fwd(const float* y_hard, const float* y, float* out, long long n, void* stream) {
    UPS_REQUIRE(y_hard && y && out, "straight_through_fwd: null pointer");
    UPS_REQUIRE(n >= 0, "straight_through_fwd: n=%lld", n);
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    straight_through_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(y_hard, y, out, n);
    return after_launch("straight_through_kernel");
}

extern "C" int ups_argmax_fwd(const float* y, long long* labels, long long n_pix, int K, void* stream) {
    UPS_REQUIRE(y && labels, "argmax_fwd: null pointer");
    UPS_REQUIRE(n_pix >= 0 && K >= 1, "argmax_fwd: n_pix=%lld K=%d", n_pix, K);
    if (n_pix == 0) return UPS_OK;
    UPS_GRID_OK(n_pix, TPB);
    argmax_kernel<<<nblk(n_pix, TPB), TPB, 0, as_stream(stream)>>>(y, labels, n_pix, K);
    return after_launch("argmax_kernel");
}

extern "C" int ups_one_hot_fwd(const long long* labels, float* out, long long n_pix, int K, void* stream) {
    UPS_REQUIRE(labels && out, "one_hot_fwd: null pointer");
    UPS_REQUIRE(n_pix >= 0 && K >= 1, "one_hot_fwd: n_pix=%lld K=%d", n_pix, K);
    if (n_pix == 0) return UPS_OK;
    UPS_GRID_OK(n_pix * K, TPB);
    one_hot_kernel<<<nblk(n_pix * K, TPB), TPB, 0, as_stream(stream)>>>(labels, out, n_pix * K, K);
    return after_launch("one_hot_kernel");
}

static int check_bpkc(const char* what, int B, int P, int K, int C) {
    UPS_REQUIRE(B >= 0 && P >= 1 && K >= 1 && C >= 1, "%s: B=%d P=%d K=%d C=%d", what, B, P, K, C);
    return UPS_OK;
}

extern "C" int ups_mask_parts_fwd(const float* image, const float* mask, float* parts, int B, int P, int K, int C,
                                  int part_major, void* stream) {
    UPS_REQUIRE(image && mask && parts, "mask_parts_fwd: null pointer");
    if (int rc = check_bpkc("mask_parts_fwd", B, P, K, C)) return rc;
    const long long n = (long long)B * P * K * C;
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    mask_parts_fwd_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(image, mask, parts, B, P, K, C, part_major, n);
    return after_launch("mask_parts_fwd_kernel");
}

extern "C" int ups_mask_parts_bwd(const float* g_parts, const float* image, const float* mask, float* dimage,
                                  float* dmask, int B, int P, int K, int C, int part_major, void* stream) {
    UPS_REQUIRE(g_parts && image && mask, "mask_parts_bwd: null pointer");
    if (int rc = check_bpkc("mask_parts_bwd", B, P, K, C)) return rc;
    if (B == 0) return UPS_OK;
    cudaStream_t s = as_stream(stream);
    if (dmask) {
        const long long n = (long long)B * P * K;
        UPS_GRID_OK(n, TPB);
        mask_parts_bwd_dmask_kernel<<<nblk(n, TPB), TPB, 0, s>>>(g_parts, image, dmask, B, P, K, C, part_major, n);
        if (int rc = after_launch("mask_parts_bwd_dmask_kernel")) return rc;
    }
    if (dimage) {
        const long long n = (long long)B * P * C;
        mask_parts_bwd_dimage_kernel<<<nblk(n, TPB), TPB, 0, s>>>(g_parts, mask, dimage, B, P, K, C, part_major, n);
        if (int rc = after_launch("mask_parts_bwd_dimage_kernel")) return rc;
    }
    return UPS_OK;
}

extern "C" int ups_partwise_fold(const float* x, float* y, int B, int P, int K, int C, void* stream) {
    UPS_REQUIRE(x && y, "partwise_fold: null pointer");
    if (int rc = check_bpkc("partwise_fold", B, P, K, C)) return rc;
    const long long n = (long long)B * P * K * C;
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    partwise_fold_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(x, y, B, P, K, C, n, 0);
    return after_launch("partwise_fold_kernel");
}

extern "C" int ups_partwise_unfold(const float* y, float* x, int B, int P, int K, int C, void* stream) {
    UPS_REQUIRE(x && y, "partwise_unfold: null pointer");
    if (int rc = check_bpkc("partwise_unfold", B, P, K, C)) return rc;
    const long long n = (long long)B * P * K * C;
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    partwise_fold_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(y, x, B, P, K, C, n, 1);
    return after_launch("partwise_fold_kernel");
}

// ---- pooling driver shared by part_pool_fwd, unpool_bwd (dfeat) and inject_bwd (dfeat)
namespace ups {
int pool_splits(int B, int P) {
    // enough CTAs for >= 4 waves of 148 SMs, at least 256 pixels per split
    int s = (int)cdiv(4 * NUM_SMS, B > 0 ? B : 1);
    const int smax = (int)cdiv(P, 256);
    if (s > smax) s = smax;
    if (s < 1) s = 1;
    return s;
}
size_t pool_ws_bytes(int B, int P, int KF) { return (size_t)B * pool_splits(B, P) * KF * sizeof(float); }

int run_pool(const float* fmap, const float* mask, float* out, int B, int P, int K, int Fg, int grouped,
             int fmap_stride, float scale, int divide_by, void* ws, size_t ws_bytes, cudaStream_t s) {
    const int KF = K * Fg;
    UPS_REQUIRE(Fg <= 1024, "pooling: %d features per part > 1024 unsupported", Fg);
    UPS_REQUIRE(B <= 65535, "pooling: B=%d exceeds grid.y limit", B);
    const int splits = pool_splits(B, P);
    if (ws_bytes < pool_ws_bytes(B, P, KF) || !ws) {
        set_error("pooling: workspace %zu < %zu bytes", ws_bytes, pool_ws_bytes(B, P, KF));
        return UPS_E_WORKSPACE;
    }
    float* partial = static_cast<float*>(ws);
    dim3 grid(splits, B);
    const int kchunk = 1024 / Fg;  // parts per launch: at most 1024 (k,f) pairs in registers
    for (int k0 = 0; k0 < K; k0 += kchunk) {
        const int kc = (K - k0 < kchunk) ? (K - k0) : kchunk;
        const int KFc = kc * Fg;
        const size_t sm = (size_t)POOL_WARPS * KFc * sizeof(float);
        const int nacc = (int)cdiv(KFc, 32);
#define UPS_POOL(N)                                                                                                  \
    part_pool_partial_kernel<N><<<grid, POOL_WARPS * 32, sm, s>>>(fmap, mask, partial, P, K, Fg, grouped, fmap_stride, \
                                                                  splits, k0, kc)
        if (nacc <= 1) UPS_POOL(1);
        else if (nacc <= 2) UPS_POOL(2);
        else if (nacc <= 4) UPS_POOL(4);
        else if (nacc <= 8) UPS_POOL(8);
        else if (nacc <= 16) UPS_POOL(16);
        else UPS_POOL(32);
#undef UPS_POOL
        if (int rc = after_launch("part_pool_partial_kernel")) return rc;
    }
    const long long n = (long long)B * KF;
    pool_finalize_kernel<<<nblk(n, 128), 128, 0, s>>>(partial, out, KF, splits, scale, divide_by, n);
    return after_launch("pool_finalize_kernel");
}
}  // namespace ups

extern "C" size_t ups_workspace_bytes(int op, int B, int P, int K, int F) {
    switch (op) {
        case UPS_OP_POOL:
        case UPS_OP_INJECT_BWD:
            return pool_ws_bytes(B, P, K * F) + 256;
        case UPS_OP_STEP: {
            if (B <= 0 || P <= 0) return 256;
            const size_t splits = (size_t)cdiv(P, fused_pix_per_cta(B, P));
            const size_t fused = (size_t)B * splits * K * (F > 3 ? F : 3) * sizeof(float);
            const size_t unfused = pool_ws_bytes(B, P, K * (F > 3 ? F : 3));
            const size_t tc = (K == 16 || K == 32) && F == 64 ? decode_bwd_tma_ws_bytes(B, P, K, F) : 0;
            const size_t m = fused > unfused ? fused : unfused;
            return (m > tc ? m : tc) + 256;
        }
        case UPS_OP_MOMENTS:
            return (B <= 0 || P <= 0) ? 256 : moments_ws_bytes(B, P, K);
        case UPS_OP_KL:
            return (size_t)NUM_SMS * 8 * sizeof(float) + 256;
        case UPS_OP_MUMFORD_SHAH:
            return (B <= 0 || P <= 0) ? 256 : mumford_shah_ws_bytes(B, P, K);
        case UPS_OP_LOGIT_PRIORS:
            return priors_scalar_ws_bytes();
        case UPS_OP_WEAK_XENT: {
            const size_t generic = (B <= 0 || P <= 0) ? 0 : (size_t)cdiv((long long)B * P, 128) * sizeof(float);
            const size_t fast = priors_scalar_ws_bytes();
            return (generic > fast ? generic : fast) + 256;
        }
        default:
            return 0;
    }
}

extern "C" int ups_part_pool_fwd(const float* fmap, const float* mask, float* out, int B, int P, int K, int Fg,
                                 int grouped, float scale, void* ws, size_t ws_bytes, void* stream) {
    UPS_REQUIRE(fmap && mask && out, "part_pool_fwd: null pointer");
    if (int rc = check_bpkc("part_pool_fwd", B, P, K, Fg)) return rc;
    if (B == 0) return UPS_OK;
    return run_pool(fmap, mask, out, B, P, K, Fg, grouped, grouped ? K * Fg : Fg, scale, 0, ws, ws_bytes, as_stream(stream));
}

extern "C" int ups_part_pool_bwd(const float* g_out, const float* fmap, const float* mask, float* dfmap, float* dmask,
                                 int B, int P, int K, int Fg, int grouped, float scale, void* stream) {
    UPS_REQUIRE(g_out && fmap && mask, "part_pool_bwd: null pointer");
    if (int rc = check_bpkc("part_pool_bwd", B, P, K, Fg)) return rc;
    if (B == 0) return UPS_OK;
    cudaStream_t s = as_stream(stream);
    const int row = grouped ? K * Fg : Fg;
    if (dfmap) {
        const long long n = (long long)B * P * row;
        UPS_GRID_OK(n, TPB);
        part_pool_bwd_dfmap_kernel<<<nblk(n, TPB), TPB, 0, s>>>(g_out, mask, dfmap, P, K, Fg, grouped, scale, n);
        if (int rc = after_launch("part_pool_bwd_dfmap_kernel")) return rc;
    }
    if (dmask) {
        const long long n = (long long)B * P * K;
        UPS_GRID_OK(n, TPB);
        part_pool_bwd_dmask_kernel<<<nblk(n, TPB), TPB, 0, s>>>(g_out, fmap, dmask, P, K, Fg, grouped, row, scale, nullptr, 0, 0, n);
        if (int rc = after_launch("part_pool_bwd_dmask_kernel")) return rc;
    }
    return UPS_OK;
}

extern "C" int ups_part_unpool_fwd(const float* feat, const float* mask, float* out, int B, int P, int K, int F,
                                   void* stream) {
    UPS_REQUIRE(feat && mask && out, "part_unpool_fwd: null pointer");
    if (int rc = check_bpkc("part_unpool_fwd", B, P, K, F)) return rc;
    const long long n = (long long)B * P * K * F;
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    part_unpool_fwd_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(feat, mask, out, P, K, F, n);
    return after_launch("part_unpool_fwd_kernel");
}

extern "C" int ups_part_unpool_bwd(const float* g_out, const float* feat, const float* mask, float* dfeat,
                                   float* dmask, int B, int P, int K, int F, void* ws, size_t ws_bytes, void* stream) {
    UPS_REQUIRE(g_out && feat && mask, "part_unpool_bwd: null pointer");
    if (int rc = check_bpkc("part_unpool_bwd", B, P, K, F)) return rc;
    if (B == 0) return UPS_OK;
    cudaStream_t s = as_stream(stream);
    if (dfeat) {  // dfeat[b,k,f] = sum_p g[b,p,k,f]*mask[b,p,k]  == grouped pooling of g
        if (int rc = run_pool(g_out, mask, dfeat, B, P, K, F, 1, K * F, 1.0f, 0, ws, ws_bytes, s)) return rc;
    }
    if (dmask) {  // dmask[b,p,k] = sum_f g[b,p,k,f]*feat[b,k,f]
        const long long n = (long long)B * P * K;
        UPS_GRID_OK(n, TPB);
        part_pool_bwd_dmask_kernel<<<nblk(n, TPB), TPB, 0, s>>>(feat, g_out, dmask, P, K, F, 1, K * F, 1.0f, nullptr, 0, 0, n);
        if (int rc = after_launch("part_pool_bwd_dmask_kernel")) return rc;
    }
    return UPS_OK;
}

extern "C" int ups_part_inject_fwd(const float* feat, const float* mask, float* inj, int B, int P, int K, int F,
                                   void* stream) {
    UPS_REQUIRE(feat && mask && inj, "part_inject_fwd: null pointer");
    if (int rc = check_bpkc("part_inject_fwd", B, P, K, F)) return rc;
    UPS_REQUIRE((size_t)K * F * sizeof(float) <= 48 * 1024, "part_inject_fwd: K*F=%d too large", K * F);
    UPS_REQUIRE(B <= 65535, "part_inject_fwd: B=%d exceeds grid.y limit", B);
    if (B == 0) return UPS_OK;
    dim3 grid((unsigned)cdiv(P, INJ_PIX), B);
    part_inject_fwd_kernel<<<grid, INJ_TPB, (size_t)K * F * sizeof(float), as_stream(stream)>>>(feat, mask, inj, P, K, F);
    return after_launch("part_inject_fwd_kernel");
}

extern "C" int ups_part_inject_bwd(const float* g_inj, const float* feat, const float* mask, float* dfeat,
                                   float* dmask, int B, int P, int K, int F, void* ws, size_t ws_bytes, void* stream) {
    UPS_REQUIRE(g_inj && feat && mask, "part_inject_bwd: null pointer");
    if (int rc = check_bpkc("part_inject_bwd", B, P, K, F)) return rc;
    if (B == 0) return UPS_OK;
    cudaStream_t s = as_stream(stream);
    if (dfeat) {  // dfeat[b,k,f] = sum_p mask[b,p,k]*g[b,p,f]  == dense pooling of g[..., :F] (row stride F+K)
        if (int rc = run_pool(g_inj, mask, dfeat, B, P, K, F, 0, F + K, 1.0f, 0, ws, ws_bytes, s)) return rc;
    }
    if (dmask) {  // dmask[b,p,k] = sum_f g[b,p,f]*feat[b,k,f] + g[b,p,F+k]
        const long long n = (long long)B * P * K;
        UPS_GRID_OK(n, TPB);
        part_pool_bwd_dmask_kernel<<<nblk(n, TPB), TPB, 0, s>>>(feat, g_inj, dmask, P, K, F, 0, F + K, 1.0f, g_inj, F + K, F, n);
        if (int rc = after_launch("part_pool_bwd_dmask_kernel")) return rc;
    }
    return UPS_OK;
}

extern "C" int ups_part_gather_fwd(const float* feat, const long long* labels, float* out, int B, int P, int K, int F,
                                   void* stream) {
    UPS_REQUIRE(feat && labels && out, "part_gather_fwd: null pointer");
    if (int rc = check_bpkc("part_gather_fwd", B, P, K, F)) return rc;
    const long long n = (long long)B * P * F;
    if (n == 0) return UPS_OK;
    UPS_GRID_OK(n, TPB);
    part_gather_fwd_kernel<<<nblk(n, TPB), TPB, 0, as_stream(stream)>>>(feat, labels, out, P, K, F, n);
    return after_launch("part_gather_fwd_kernel");
}
