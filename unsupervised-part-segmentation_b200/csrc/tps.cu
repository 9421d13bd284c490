// Thin-plate-spline equivariance warp: parameter transform, 11x11 solve, fused
// grid-evaluation + bilinear gather (forward) and scatter-add (backward).
// Reference: baselines/unsupervised-disentangling/transformations.py:59-77,93-244
// (the vendored copy of eddata.utils.tps called from cub/code/SB_model48i/model.py:300-309).
#include <stdlib.h>

#include "common.cuh"
#include "pk_math.cuh"
#include "tps_warp_fwd.cuh"

namespace ups {

// ------------------------------------------------------------------ a2: make_input_tps_param
__global__ void tps_input_param_kernel(const float* __restrict__ coord, const float* __restrict__ vector,
                                       const float* __restrict__ offset, const float* __restrict__ offset_2,
                                       const float* __restrict__ t_scal, const float* __restrict__ rot,
                                       float* __restrict__ t_vector, int N) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= N) return;
    float c[16], v[16], o[2], o2[2], ts[2], r[4], tv[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { c[i] = coord[b * 16 + i]; v[i] = vector[b * 16 + i]; }
#pragma unroll
    for (int i = 0; i < 2; ++i) { o[i] = offset[b * 2 + i]; o2[i] = offset_2[b * 2 + i]; ts[i] = t_scal[b * 2 + i]; }
#pragma unroll
    for (int i = 0; i < 4; ++i) r[i] = rot[b * 4 + i];
    tps_input_param(c, v, o, o2, ts, r, tv);
#pragma unroll
    for (int i = 0; i < 16; ++i) t_vector[b * 16 + i] = tv[i];
}

// ------------------------------------------------------------------ a3(ii): _solve_system
// One WARP per sample: lane r < 11 holds row r of the augmented 11x13 system in registers.
// Every row operation is the canonical one of canon_math.cuh::tps_solve / oracle solve_canon
// (same operands, same single-rounded mul / sub / div), only executed by 11 lanes at once, so
// the result is bit-identical to the sequential form (tests/test_canon_host.py pins that form).
constexpr int SOLVE_WARPS = 4;

// The solve of sample b by its warp: qx / qy = the flipped control points (every lane holds all 8), vec_at(k) = element
// k of the sample's vector [8,2] (called by lanes 0..7 for k = 2 lane, 2 lane + 1).
template <typename VecAt>
__device__ __forceinline__ void tps_solve_warp(const float (&qx)[8], const float (&qy)[8], VecAt vec_at,
                                               float* __restrict__ T, int b, int lane) {
    constexpr unsigned FULLM = 0xffffffffu;
    double row[13];
#pragma unroll
    for (int j = 0; j < 13; ++j) row[j] = 0.0;
    if (lane < 8) {
        float mx = 0.f, my = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) if (i == lane) { mx = qx[i]; my = qy[i]; }
        row[0] = 1.0; row[1] = (double)mx; row[2] = (double)my;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float d0 = __fsub_rn(1.0f, 1.0f);
            const float d1 = __fsub_rn(mx, qx[j]);
            const float d2_ = __fsub_rn(my, qy[j]);
            const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2_, d2_));
            row[3 + j] = (double)tps_rbf(d2);
        }
        row[11] = (double)__fadd_rn(mx, vec_at(2 * lane + 1));
        row[12] = (double)__fadd_rn(my, vec_at(2 * lane));
    } else if (lane < 11) {
#pragma unroll
        for (int j = 0; j < 8; ++j) row[3 + j] = (lane == 8) ? 1.0 : (lane == 9 ? (double)qx[j] : (double)qy[j]);
    }
    int pos = lane;  // logical row index of the row this lane holds (rows swap by swapping pos)
#pragma unroll
    for (int c = 0; c < 11; ++c) {
        // first-max partial pivoting over logical rows >= c
        double bv = (lane < 11 && pos >= c) ? fabs(row[c]) : -1.0;
        int bp = pos;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const double ov = __shfl_xor_sync(FULLM, bv, o);
            const int op = __shfl_xor_sync(FULLM, bp, o);
            if (ov > bv || (ov == bv && op < bp)) { bv = ov; bp = op; }
        }
        if (pos == bp) pos = c; else if (pos == c) pos = bp;
        const int pl = __ffs(__ballot_sync(FULLM, lane < 11 && pos == c)) - 1;  // lane holding the pivot row
        const double piv = __shfl_sync(FULLM, row[c], pl);
        const double f = (lane != pl) ? __ddiv_rn(row[c], piv) : 0.0;
#pragma unroll
        for (int j = c + 1; j < 13; ++j) {
            const double pj = __shfl_sync(FULLM, row[j], pl);
            if (lane != pl) row[j] = __dsub_rn(row[j], __dmul_rn(f, pj));
        }
    }
    if (lane < 11) {
        double d = row[0];
#pragma unroll
        for (int j = 1; j < 11; ++j) if (j == pos) d = row[j];
        T[b * 22 + pos] = (float)__ddiv_rn(row[11], d);
        T[b * 22 + 11 + pos] = (float)__ddiv_rn(row[12], d);
    }
}

__global__ void __launch_bounds__(SOLVE_WARPS * 32) tps_solve_kernel(const float* __restrict__ coord,
                                                                     const float* __restrict__ vector,
                                                                     float* __restrict__ T, int N) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * SOLVE_WARPS + (threadIdx.x >> 5);
    if (b >= N) return;  // warp-uniform
    float qx[8], qy[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { qx[i] = __ldg(coord + b * 16 + 2 * i + 1); qy[i] = __ldg(coord + b * 16 + 2 * i); }
    tps_solve_warp(qx, qy, [&](int k) { return __ldg(vector + b * 16 + k); }, T, b, lane);
}

// ------------------------------------------------------------------ a1 + a2 + a3(ii): draw, make_input_tps_param, solve
// One warp per row r = v * n_per_view + s (view v, global sample sample_offset + s).  Lanes 0..9 make one Philox call
// each (words 4 lane .. 4 lane + 3, canon_math.cuh "the TPS parameters"); every lane then gathers the 39 words, forms the
// fields with tps_fields and t_vector with tps_input_param, and the warp runs tps_solve_warp, the body of
// tps_solve_kernel.  coord / t_vector / T are bit for bit what ups_tps_input_param + ups_tps_solve give on the fields.
// DSEED: `seed` is the address of the seed (resolve_seed).  Each raw output may be null.
// a[i] of a register array, without local memory
template <int N>
__device__ __forceinline__ float pick(const float (&a)[N], int i) {
    float r = a[0];
#pragma unroll
    for (int k = 1; k < N; ++k) if (k == i) r = a[k];
    return r;
}

template <bool DSEED>
__global__ void __launch_bounds__(SOLVE_WARPS * 32) tps_draw_solve_kernel(
    unsigned long long seed, long long sample_offset, int n_per_view, int N, TpsDrawScalars sc, float* __restrict__ coord,
    float* __restrict__ vector, float* __restrict__ offset, float* __restrict__ offset_2, float* __restrict__ t_scal,
    float* __restrict__ rot_mat, float* __restrict__ t_vector, float* __restrict__ T) {
    constexpr unsigned FULLM = 0xffffffffu;
    if (DSEED) seed = *reinterpret_cast<const unsigned long long*>(seed);
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * SOLVE_WARPS + (threadIdx.x >> 5);
    if (b >= N) return;  // warp-uniform
    const int v = b / n_per_view;
    const unsigned long long g = (unsigned long long)(sample_offset + (b - v * n_per_view));
    uint32_t own[4];
    tps_words4(seed, v, g, (uint32_t)(lane < TPS_DRAW_CALLS ? lane : 0), own);
    uint32_t x[TPS_DRAW_WORDS];
#pragma unroll
    for (int w = 0; w < TPS_DRAW_WORDS; ++w) x[w] = __shfl_sync(FULLM, own[w & 3], w >> 2);
    float c[16], vec[16], o[2], o2[2], ts[2], rot[4], tv[16];
    tps_fields(sc, x, c, vec, o, o2, ts, rot);
    tps_input_param(c, vec, o, o2, ts, rot, tv);
    if (lane < 16) {
        if (coord) coord[b * 16 + lane] = pick(c, lane);
        if (vector) vector[b * 16 + lane] = pick(vec, lane);
        t_vector[b * 16 + lane] = pick(tv, lane);
    }
    if (lane < 2) {
        if (offset) offset[b * 2 + lane] = pick(o, lane);
        if (offset_2) offset_2[b * 2 + lane] = pick(o2, lane);
        if (t_scal) t_scal[b * 2 + lane] = pick(ts, lane);
    }
    if (lane < 4 && rot_mat) rot_mat[b * 4 + lane] = pick(rot, lane);
    float qx[8], qy[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { qx[i] = c[2 * i + 1]; qy[i] = c[2 * i]; }
    tps_solve_warp(qx, qy, [&](int k) { return pick(tv, k); }, T, b, lane);
}

// K1 as its own kernel.  MINB = resident CTAs per SM asked of ptxas: besides capping registers, an explicit value
// makes ptxas keep the interleaving of the four log chains (without it, it re-serialises them to save registers).
template <int C, int MINB>
__global__ void __launch_bounds__(WARP_TPB, MINB) tps_warp_fwd_kernel(const float* __restrict__ U,
                                                                const float* __restrict__ U2,
                                                                const float* __restrict__ coord,
                                                                const float* __restrict__ T,
                                                                const float* __restrict__ move,
                                                                const float* __restrict__ scal,
                                                                float* __restrict__ out, float* __restrict__ out2,
                                                                float* __restrict__ mesh, int N2, int H, int W,
                                                                int Crt, int oh, int ow) {
    __shared__ float sm_const[42];
    extern __shared__ __align__(16) float sm_out[];  // 2 * WARP_TPB * C floats
    tps_warp_fwd_body<C>(U, U2, coord, T, move, scal, out, out2, mesh, N2, H, W, Crt, oh, ow, blockIdx.x, blockIdx.y,
                         sm_const, sm_out);
}

// three consecutive floats at a 4-byte aligned address p (p + even offset is 8-byte aligned when the base is):
// one 8-byte vector reduction + one scalar reduction
__device__ __forceinline__ void red_add3(float* p, const float (&v)[3]) {
    if ((reinterpret_cast<uintptr_t>(p) & 7u) == 0) {
        asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v[0]), "f"(v[1]) : "memory");
        asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p + 2), "f"(v[2]) : "memory");
    } else {
        asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v[0]) : "memory");
        asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p + 1), "f"(v[1]), "f"(v[2]) : "memory");
    }
}

template <int C>
__global__ void __launch_bounds__(WARP_TPB) tps_warp_bwd_kernel(const float* __restrict__ g_out,
                                                                const float* __restrict__ g_out2,
                                                                const float* __restrict__ coord,
                                                                const float* __restrict__ T,
                                                                const float* __restrict__ move,
                                                                const float* __restrict__ scal, float* __restrict__ dU,
                                                                float* __restrict__ dU2, int N2, int H, int W, int Crt,
                                                                int oh, int ow, const float* __restrict__ extra, int x0,
                                                                int xn) {
    // cotangent of output sample b = g_out[b] (zeros when g_out is null) + extra[b - x0] for b in [x0, x0 + xn): the
    // fused step adds dimg1 (the encode side's cotangent of warped view 1) to the caller's g_warped here instead of
    // materialising the sum (model.py:282-311 differentiated)
    __shared__ float sm_const[42];
    extern __shared__ float sm_g[];  // 2 * WARP_TPB * C floats
    const int Cc = (C > 0) ? C : Crt;
    const int b = blockIdx.y;
    SampleConst k;
    load_sample_const(k, sm_const, coord, T, move, scal, b);
    const bool has_move = (move != nullptr);
    const bool second = (g_out2 != nullptr) && (b < N2);
    const float step_w = lin_step(ow), step_h = lin_step(oh);
    const int OP = oh * ow;
    float* Ub = dU + (size_t)b * H * W * Cc;
    float* Ub2 = second ? dU2 + (size_t)b * H * W * Cc : nullptr;
    float* sm_g2 = sm_g + WARP_TPB * Cc;
    const bool vec_red = ((reinterpret_cast<uintptr_t>(dU) | reinterpret_cast<uintptr_t>(dU2)) & 7u) == 0;
    if (g_out == nullptr && !second && !(extra != nullptr && b >= x0 && b < x0 + xn)) return;   // zero cotangent: dU stays 0
    const int tile0 = blockIdx.x * (WARP_TPB * WARP_PPT);
#pragma unroll 1
    for (int it = 0; it < WARP_PPT; ++it) {
        const int base = tile0 + it * WARP_TPB;
        if (base >= OP) break;
        const int n_live = min(WARP_TPB, OP - base) * Cc;
        const bool has_x = extra != nullptr && b >= x0 && b < x0 + xn;
        const float* gb = g_out ? g_out + ((size_t)b * OP + base) * Cc : nullptr;
        const float* xb = has_x ? extra + ((size_t)(b - x0) * OP + base) * Cc : nullptr;
        for (int e = threadIdx.x; e < n_live; e += WARP_TPB)
            sm_g[e] = (gb ? __ldcs(gb + e) : 0.f) + (xb ? __ldcs(xb + e) : 0.f);
        if (second) {
            const float* gb2 = g_out2 + ((size_t)b * OP + base) * Cc;
            for (int e = threadIdx.x; e < n_live; e += WARP_TPB) sm_g2[e] = __ldcs(gb2 + e);
        }
        __syncthreads();
        const int pix = base + threadIdx.x;
        const bool live = pix < OP;
        Bilinear s;
        int oa = -1, ob = -1, oc = -1, od = -1;
        if (live) {
            const int i = pix / ow, j = pix - i * ow;
            float x_s, y_s;
            sample_position(k, has_move, i, j, step_h, step_w, x_s, y_s);
            s = bilinear_stencil(x_s, y_s, W, H);
            oa = (s.y0 * W + s.x0) * Cc; ob = (s.y1 * W + s.x0) * Cc;
            oc = (s.y0 * W + s.x1) * Cc; od = (s.y1 * W + s.x1) * Cc;
        }
        if (C == 3 && vec_red) {
            // Scatter with a quarter of the reduction traffic.  (1) Neighbouring output pixels of a row sample
            // neighbouring source pixels: lane L's right corners (x1) are lane L+1's left corners (x0) whenever the
            // addresses coincide (~80 % of the lanes at the shipped scales), so L adds its neighbour's left
            // contributions to its own right ones in registers and the neighbour drops them.  The test is address
            // equality, so the result is the same sum whatever the warp looks like.  (2) A corner's three channels
            // go out as one 8-byte vector reduction + one scalar instead of three scalars.
            // Out-of-range samples keep all four (cancelling) contributions, as autodiff of the forward does.
            const unsigned FULLM = 0xffffffffu;
            const int lane = threadIdx.x & 31;
            const int n_oa = __shfl_down_sync(FULLM, oa, 1), n_ob = __shfl_down_sync(FULLM, ob, 1);
            const int p_oc = __shfl_up_sync(FULLM, oc, 1), p_od = __shfl_up_sync(FULLM, od, 1);
            const bool take_a = live && lane < 31 && n_oa == oc && n_oa >= 0;   // I absorb my right neighbour's a
            const bool take_b = live && lane < 31 && n_ob == od && n_ob >= 0;
            const bool gave_a = live && lane > 0 && p_oc == oa && p_oc >= 0;    // my a was absorbed by my left neighbour
            const bool gave_b = live && lane > 0 && p_od == ob && p_od >= 0;
            const int n_img = second ? 2 : 1;
            for (int im = 0; im < n_img; ++im) {
                const float* sg = (im ? sm_g2 : sm_g) + threadIdx.x * 3;
                float* Ud = im ? Ub2 : Ub;
                float ca[3], cb[3], cc[3], cd[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float g = live ? sg[c] : 0.f;
                    ca[c] = live ? s.wa * g : 0.f; cb[c] = live ? s.wb * g : 0.f;
                    cc[c] = live ? s.wc * g : 0.f; cd[c] = live ? s.wd * g : 0.f;
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float na = __shfl_down_sync(FULLM, ca[c], 1), nb = __shfl_down_sync(FULLM, cb[c], 1);
                    if (take_a) cc[c] += na;
                    if (take_b) cd[c] += nb;
                }
                if (live) {
                    if (!gave_a) red_add3(Ud + oa, ca);
                    if (!gave_b) red_add3(Ud + ob, cb);
                    red_add3(Ud + oc, cc);
                    red_add3(Ud + od, cd);
                }
            }
        } else if (live) {
            for (int c = 0; c < Cc; ++c) {
                // out-of-range samples have coinciding clipped corners whose weights cancel:
                // keep all four adds so that the sum matches autodiff of the forward exactly.
                const float g = sm_g[threadIdx.x * Cc + c];
                atomicAdd(Ub + oa + c, s.wa * g);
                atomicAdd(Ub + ob + c, s.wb * g);
                atomicAdd(Ub + oc + c, s.wc * g);
                atomicAdd(Ub + od + c, s.wd * g);
                if (second) {
                    const float g2 = sm_g2[threadIdx.x * Cc + c];
                    atomicAdd(Ub2 + oa + c, s.wa * g2);
                    atomicAdd(Ub2 + ob + c, s.wb * g2);
                    atomicAdd(Ub2 + oc + c, s.wc * g2);
                    atomicAdd(Ub2 + od + c, s.wd * g2);
                }
            }
        }
        __syncthreads();
    }
}

}  // namespace ups

using namespace ups;

extern "C" int ups_tps_input_param(const float* coord, const float* vector, const float* offset,
                                   const float* offset_2, const float* t_scal, const float* rot_mat, float* t_vector,
                                   int N, void* stream) {
    UPS_REQUIRE(coord && vector && offset && offset_2 && t_scal && rot_mat && t_vector, "tps_input_param: null pointer");
    UPS_REQUIRE(N >= 0, "tps_input_param: N=%d", N);
    if (N == 0) return UPS_OK;
    tps_input_param_kernel<<<(unsigned)cdiv(N, 64), 64, 0, as_stream(stream)>>>(coord, vector, offset, offset_2, t_scal,
                                                                                rot_mat, t_vector, N);
    return after_launch("tps_input_param_kernel");
}

extern "C" int ups_tps_solve(const float* coord, const float* vector, float* T, int N, void* stream) {
    UPS_REQUIRE(coord && vector && T, "tps_solve: null pointer");
    UPS_REQUIRE(N >= 0, "tps_solve: N=%d", N);
    if (N == 0) return UPS_OK;
    tps_solve_kernel<<<(unsigned)cdiv(N, SOLVE_WARPS), SOLVE_WARPS * 32, 0, as_stream(stream)>>>(coord, vector, T, N);
    return after_launch("tps_solve_kernel");
}

template <bool DSEED>
static int tps_draw_solve_launch(unsigned long long seed, long long sample_offset, int n_per_view, int n_views,
                                 const TpsDrawScalars& sc, float* coord, float* vector, float* offset, float* offset_2,
                                 float* t_scal, float* rot_mat, float* t_vector, float* T, void* stream) {
    UPS_REQUIRE(t_vector && T, "tps_draw_solve: null pointer");
    UPS_REQUIRE(n_per_view >= 0 && (n_views == 1 || n_views == 2) && sample_offset >= 0,
                "tps_draw_solve: n_per_view=%d n_views=%d sample_offset=%lld", n_per_view, n_views, sample_offset);
    UPS_REQUIRE((long long)n_per_view * n_views * 16 < (1ll << 31), "tps_draw_solve: n_per_view=%d too large", n_per_view);
    UPS_REQUIRE(sc.rot_turn >= 0.0f && sc.rot_turn <= 0.5f, "tps_draw_solve: rot_turn=%g outside [0, 1/2]", (double)sc.rot_turn);
    const int N = n_per_view * n_views;
    if (N == 0) return UPS_OK;
    tps_draw_solve_kernel<DSEED><<<(unsigned)cdiv(N, SOLVE_WARPS), SOLVE_WARPS * 32, 0, as_stream(stream)>>>(
        seed, sample_offset, n_per_view, N, sc, coord, vector, offset, offset_2, t_scal, rot_mat, t_vector, T);
    return after_launch("tps_draw_solve_kernel");
}

extern "C" int ups_tps_draw_solve(unsigned long long seed, long long sample_offset, int n_per_view, int n_views,
                                  float coord_lo, float coord_w, float vec_lo, float vec_w, float off_lo, float off_w,
                                  float scal_lo, float scal_w, float rescal, float rot_turn, float* coord, float* vector,
                                  float* offset, float* offset_2, float* t_scal, float* rot_mat, float* t_vector, float* T,
                                  void* stream) {
    const TpsDrawScalars sc{coord_lo, coord_w, vec_lo, vec_w, off_lo, off_w, scal_lo, scal_w, rescal, rot_turn};
    return tps_draw_solve_launch<false>(seed, sample_offset, n_per_view, n_views, sc, coord, vector, offset, offset_2,
                                        t_scal, rot_mat, t_vector, T, stream);
}

extern "C" int ups_tps_draw_solve_dseed(const unsigned long long* seed, long long sample_offset, int n_per_view, int n_views,
                                        float coord_lo, float coord_w, float vec_lo, float vec_w, float off_lo, float off_w,
                                        float scal_lo, float scal_w, float rescal, float rot_turn, float* coord,
                                        float* vector, float* offset, float* offset_2, float* t_scal, float* rot_mat,
                                        float* t_vector, float* T, void* stream) {
    UPS_REQUIRE(seed, "tps_draw_solve: null seed pointer");
    const TpsDrawScalars sc{coord_lo, coord_w, vec_lo, vec_w, off_lo, off_w, scal_lo, scal_w, rescal, rot_turn};
    return tps_draw_solve_launch<true>((unsigned long long)(uintptr_t)seed, sample_offset, n_per_view, n_views, sc, coord,
                                       vector, offset, offset_2, t_scal, rot_mat, t_vector, T, stream);
}

static int check_warp_args(const void* U, const void* coord, const void* T, const void* move, const void* scal,
                           const void* out, int N, int H, int W, int C, int oh, int ow) {
    UPS_REQUIRE(U && coord && T && out, "tps_warp: null pointer");
    UPS_REQUIRE((move == nullptr) == (scal == nullptr), "tps_warp: move and scal must be given together");
    UPS_REQUIRE(N >= 0 && H > 0 && W > 0 && C > 0 && oh > 1 && ow > 1, "tps_warp: bad dims N=%d H=%d W=%d C=%d out=%dx%d",
                N, H, W, C, oh, ow);
    UPS_REQUIRE(N <= 65535, "tps_warp: N=%d exceeds grid.y limit; split the batch", N);
    UPS_REQUIRE((long long)H * W * C < (1ll << 31) && (long long)oh * ow * C < (1ll << 31), "tps_warp: image too large");
    UPS_REQUIRE(C <= 64, "tps_warp: C=%d > 64 unsupported", C);
    return UPS_OK;
}

static int launch_warp_fwd(const float* U, const float* U2, const float* coord, const float* T, const float* move,
                           const float* scal, float* out, float* out2, float* mesh, int N, int N2, int H, int W, int C,
                           int out_h, int out_w, void* stream) {
    int rc = check_warp_args(U, coord, T, move, scal, out, N, H, W, C, out_h, out_w);
    if (rc) return rc;
    UPS_REQUIRE((U2 == nullptr) == (out2 == nullptr), "tps_warp_fwd: U2 and out2 must be given together");
    UPS_REQUIRE(N2 >= 0 && N2 <= N, "tps_warp_fwd: N2=%d not in [0, N=%d]", N2, N);
    if (N == 0) return UPS_OK;
    UPS_REQUIRE(mesh == nullptr || (reinterpret_cast<uintptr_t>(mesh) & 7u) == 0, "tps_warp_fwd: mesh must be 8-byte aligned");
    dim3 grid((unsigned)cdiv((long long)out_h * out_w, WARP_TPB * WARP_PPT), (unsigned)N);
    const size_t sm = (size_t)2 * WARP_TPB * C * sizeof(float);
    static const int minb = []() { const char* e = getenv("UPS_TPS_MINB"); return e ? atoi(e) : 8; }();
#define UPS_WARP_FWD(CC, MB) \
    tps_warp_fwd_kernel<CC, MB><<<grid, WARP_TPB, sm, as_stream(stream)>>>(U, U2, coord, T, move, scal, out, out2, mesh, N2, H, W, C, out_h, out_w)
    if (C == 3) {
        if (minb == 4) UPS_WARP_FWD(3, 4); else if (minb == 5) UPS_WARP_FWD(3, 5); else if (minb == 6) UPS_WARP_FWD(3, 6); else UPS_WARP_FWD(3, 8);
    } else {
        UPS_WARP_FWD(0, 6);
    }
#undef UPS_WARP_FWD
    return after_launch("tps_warp_fwd_kernel");
}

static int launch_warp_bwd(const float* g_out, const float* g_out2, const float* coord, const float* T,
                           const float* move, const float* scal, float* dU, float* dU2, int N, int N2, int H, int W,
                           int C, int out_h, int out_w, void* stream, const float* extra = nullptr, int x0 = 0, int xn = 0) {
    int rc = check_warp_args(g_out ? (const void*)g_out : (const void*)dU, coord, T, move, scal, dU, N, H, W, C, out_h, out_w);
    UPS_REQUIRE(g_out || extra || g_out2, "tps_warp_bwd: no cotangent at all");
    UPS_REQUIRE(!extra || (x0 >= 0 && xn >= 0 && x0 + xn <= N), "tps_warp_bwd: extra range [%d, %d) outside [0, %d)", x0, x0 + xn, N);
    if (rc) return rc;
    UPS_REQUIRE((g_out2 == nullptr) == (dU2 == nullptr), "tps_warp_bwd: g_out2 and dU2 must be given together");
    UPS_REQUIRE(N2 >= 0 && N2 <= N, "tps_warp_bwd: N2=%d not in [0, N=%d]", N2, N);
    if (N == 0) return UPS_OK;
    UPS_CUDA(cudaMemsetAsync(dU, 0, (size_t)N * H * W * C * sizeof(float), as_stream(stream)));
    if (dU2 && N2 > 0) UPS_CUDA(cudaMemsetAsync(dU2, 0, (size_t)N2 * H * W * C * sizeof(float), as_stream(stream)));
    dim3 grid((unsigned)cdiv((long long)out_h * out_w, WARP_TPB * WARP_PPT), (unsigned)N);
    const size_t sm = (size_t)2 * WARP_TPB * C * sizeof(float);
    if (C == 3)
        tps_warp_bwd_kernel<3><<<grid, WARP_TPB, sm, as_stream(stream)>>>(g_out, g_out2, coord, T, move, scal, dU, dU2, N2, H, W, C, out_h, out_w, extra, x0, xn);
    else
        tps_warp_bwd_kernel<0><<<grid, WARP_TPB, sm, as_stream(stream)>>>(g_out, g_out2, coord, T, move, scal, dU, dU2, N2, H, W, C, out_h, out_w, extra, x0, xn);
    return after_launch("tps_warp_bwd_kernel");
}

extern "C" int ups_tps_warp_fwd(const float* U, const float* coord, const float* T, const float* move,
                                const float* scal, float* out, float* mesh, int N, int H, int W, int C, int out_h,
                                int out_w, void* stream) {
    return launch_warp_fwd(U, nullptr, coord, T, move, scal, out, nullptr, mesh, N, 0, H, W, C, out_h, out_w, stream);
}

extern "C" int ups_tps_warp_bwd(const float* g_out, const float* coord, const float* T, const float* move,
                                const float* scal, float* dU, int N, int H, int W, int C, int out_h, int out_w,
                                void* stream) {
    return launch_warp_bwd(g_out, nullptr, coord, T, move, scal, dU, nullptr, N, 0, H, W, C, out_h, out_w, stream);
}

extern "C" int ups_tps_warp_pair_fwd(const float* U, const float* U2, const float* coord, const float* T, float* out,
                                     float* out2, int N, int N2, int H, int W, int C, int out_h, int out_w,
                                     void* stream) {
    UPS_REQUIRE(U2 && out2, "tps_warp_pair_fwd: null pointer");
    return launch_warp_fwd(U, U2, coord, T, nullptr, nullptr, out, out2, nullptr, N, N2, H, W, C, out_h, out_w, stream);
}

extern "C" int ups_tps_warp_pair_bwd(const float* g_out, const float* g_out2, const float* coord, const float* T,
                                     float* dU, float* dU2, int N, int N2, int H, int W, int C, int out_h, int out_w,
                                     void* stream) {
    UPS_REQUIRE(g_out2 && dU2, "tps_warp_pair_bwd: null pointer");
    return launch_warp_bwd(g_out, g_out2, coord, T, nullptr, nullptr, dU, dU2, N, N2, H, W, C, out_h, out_w, stream);
}

extern "C" int ups_tps_warp_bwd_sum(const float* g_out, const float* g_out2, const float* extra, int x0, int xn,
                                    const float* coord, const float* T, float* dU, float* dU2, int N, int N2, int H, int W,
                                    int C, int out_h, int out_w, void* stream) {
    UPS_REQUIRE((g_out2 == nullptr) == (dU2 == nullptr), "tps_warp_bwd_sum: g_out2 and dU2 must be given together");
    return launch_warp_bwd(g_out, g_out2, coord, T, nullptr, nullptr, dU, dU2, N, g_out2 ? N2 : 0, H, W, C, out_h, out_w,
                           stream, extra, x0, xn);
}
