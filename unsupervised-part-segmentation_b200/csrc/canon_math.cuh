// Canonical fp32 evaluation order shared with oracle/canon.py (see that file for the spec).
//
// Everything here uses only IEEE-754 correctly rounded single operations: on the device
// through the __f*_rn / __d*_rn intrinsics (which ptxas never contracts into FMAs), on the
// host through plain operators compiled with -ffp-contract=off.  The same header is
// compiled by g++ into libups_canon_host.so so that tests can compare it bit for bit with
// the oracle on a machine without a GPU.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define UPS_HD __host__ __device__ __forceinline__
#else
#define UPS_HD inline
#endif

#if defined(__CUDA_ARCH__)
#define UPS_FMUL(a, b) __fmul_rn((a), (b))
#define UPS_FADD(a, b) __fadd_rn((a), (b))
#define UPS_FSUB(a, b) __fsub_rn((a), (b))
#define UPS_FDIV(a, b) __fdiv_rn((a), (b))
#define UPS_FRCP(a) __frcp_rn(a)
#define UPS_DMUL(a, b) __dmul_rn((a), (b))
#define UPS_DSUB(a, b) __dsub_rn((a), (b))
#define UPS_DDIV(a, b) __ddiv_rn((a), (b))
#define UPS_F2I(x) __float_as_int(x)
#define UPS_I2F(x) __int_as_float(x)
#define UPS_FSQRT(a) __fsqrt_rn(a)
#define UPS_UMULHI(a, b) __umulhi((a), (b))
#else
#define UPS_FMUL(a, b) ((a) * (b))
#define UPS_FADD(a, b) ((a) + (b))
#define UPS_FSUB(a, b) ((a) - (b))
#define UPS_FDIV(a, b) ((a) / (b))
#define UPS_FRCP(a) (1.0f / (a))
#define UPS_DMUL(a, b) ((a) * (b))
#define UPS_DSUB(a, b) ((a) - (b))
#define UPS_DDIV(a, b) ((a) / (b))
static inline int ups_f2i_host(float x) { int i; memcpy(&i, &x, 4); return i; }
static inline float ups_i2f_host(int i) { float x; memcpy(&x, &i, 4); return x; }
#define UPS_F2I(x) ups_f2i_host(x)
#define UPS_I2F(x) ups_i2f_host(x)
#define UPS_FSQRT(a) sqrtf(a)
#define UPS_UMULHI(a, b) ((uint32_t)(((uint64_t)(a) * (uint64_t)(b)) >> 32))
#include <math.h>
#endif

namespace ups {

// exp_canon: oracle/canon.py::exp_canon
UPS_HD float exp_canon(float x) {
    const bool zero = x < -80.0f;
    x = x > 88.0f ? 88.0f : x;
    x = x < -80.0f ? -80.0f : x;
    const float n = floorf(UPS_FADD(UPS_FMUL(x, 1.44269504088896341f), 0.5f));
    float r = UPS_FSUB(x, UPS_FMUL(n, 0.693359375f));
    r = UPS_FSUB(r, UPS_FMUL(n, -2.12194440e-4f));
    const float z = UPS_FMUL(r, r);
    float y = UPS_FADD(UPS_FMUL(1.9875691500e-4f, r), 1.3981999507e-3f);
    y = UPS_FADD(UPS_FMUL(y, r), 8.3334519073e-3f);
    y = UPS_FADD(UPS_FMUL(y, r), 4.1665795894e-2f);
    y = UPS_FADD(UPS_FMUL(y, r), 1.6666665459e-1f);
    y = UPS_FADD(UPS_FMUL(y, r), 5.0000001201e-1f);
    y = UPS_FADD(UPS_FMUL(y, z), r);
    y = UPS_FADD(y, 1.0f);
    const float two_n = UPS_I2F(((int)n + 127) << 23);
    const float out = UPS_FMUL(y, two_n);
    return zero ? 0.0f : out;
}

// log_canon: oracle/canon.py::log_canon (normal positive x only)
UPS_HD float log_canon(float x) {
    const int bits = UPS_F2I(x);
    int e = ((bits >> 23) & 0xFF) - 126;
    float m = UPS_I2F((bits & 0x007FFFFF) | 0x3F000000);
    if (m < 0.707106781186547524f) {
        e -= 1;
        m = UPS_FSUB(UPS_FADD(m, m), 1.0f);
    } else {
        m = UPS_FSUB(m, 1.0f);
    }
    const float ef = (float)e;
    const float z = UPS_FMUL(m, m);
    float y = 7.0376836292e-2f;
    y = UPS_FADD(UPS_FMUL(y, m), -1.1514610310e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), 1.1676998740e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), -1.2420140846e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), 1.4249322787e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), -1.6668057665e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), 2.0000714765e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), -2.4999993993e-1f);
    y = UPS_FADD(UPS_FMUL(y, m), 3.3333331174e-1f);
    y = UPS_FMUL(UPS_FMUL(y, m), z);
    y = UPS_FADD(y, UPS_FMUL(ef, -2.12194440e-4f));
    y = UPS_FSUB(y, UPS_FMUL(0.5f, z));
    return UPS_FADD(UPS_FADD(m, y), UPS_FMUL(ef, 0.693359375f));
}

// r = d2 * log(d2 + 1e-6): the TPS radial basis (transformations.py:183,223)
UPS_HD float tps_rbf(float d2) { return UPS_FMUL(d2, log_canon(UPS_FADD(d2, 1e-6f))); }

// straight-through value fl(fl(h - y) + y)  (cub/code/nn.py:168)
UPS_HD float st_value(float h, float y) { return UPS_FADD(UPS_FSUB(h, y), y); }

constexpr int TPS_NPTS = 8;              // control points (transformations.py:18-19)
constexpr int TPS_N = TPS_NPTS + 3;      // system size 11

// make_input_tps_param (transformations.py:59-77), one sample; canonical order of
// oracle/tps.py::make_input_tps_param.  All arrays are the reference's layouts:
// coord/vector [8,2], offset/offset_2 [2], t_scal [2], rot [2,2]; out t_vector [8,2].
UPS_HD void tps_input_param(const float* coord, const float* vector, const float* offset,
                            const float* offset_2, const float* t_scal, const float* rot,
                            float* t_vector) {
    for (int c = 0; c < TPS_NPTS; ++c) {
        float u[2];
        for (int k = 0; k < 2; ++k) {
            float s = UPS_FSUB(UPS_FADD(coord[c * 2 + k], vector[c * 2 + k]), offset[k]);
            s = UPS_FADD(UPS_FMUL(t_scal[k], s), offset[k]);
            u[k] = UPS_FSUB(s, offset_2[k]);
        }
        for (int l = 0; l < 2; ++l) {
            float tv = UPS_FADD(UPS_FMUL(rot[l * 2 + 0], u[0]), UPS_FMUL(rot[l * 2 + 1], u[1]));
            tv = UPS_FADD(tv, offset_2[l]);
            t_vector[c * 2 + l] = UPS_FSUB(tv, coord[c * 2 + l]);
        }
    }
}

// _solve_system (transformations.py:215-235) for one sample.
// coord/vector are the CALLER's (un-flipped) [8,2] arrays; the ::-1 flip of
// transformations.py:95-96 happens here.  A is scratch [11][13] doubles with element
// stride `st` (so that a CTA can interleave samples in shared memory); T out [2][11] fp32.
template <typename Acc>
UPS_HD void tps_solve(const float* coord, const float* vector, Acc A, float* T) {
    constexpr int n = TPS_N, m = TPS_N + 2;
    float q[TPS_NPTS][2];
    for (int i = 0; i < TPS_NPTS; ++i) { q[i][0] = coord[i * 2 + 1]; q[i][1] = coord[i * 2 + 0]; }
    // W = [[p, r], [0, p^T]]  (fp32 entries, promoted) ; rhs = pad(coord + vector)
    for (int i = 0; i < TPS_NPTS; ++i) {
        A(i, 0) = 1.0; A(i, 1) = (double)q[i][0]; A(i, 2) = (double)q[i][1];
        for (int j = 0; j < TPS_NPTS; ++j) {
            const float d0 = UPS_FSUB(1.0f, 1.0f);
            const float d1 = UPS_FSUB(q[i][0], q[j][0]);
            const float d2_ = UPS_FSUB(q[i][1], q[j][1]);
            const float d2 = UPS_FADD(UPS_FADD(UPS_FMUL(d0, d0), UPS_FMUL(d1, d1)), UPS_FMUL(d2_, d2_));
            A(i, 3 + j) = (double)tps_rbf(d2);
        }
        A(i, n + 0) = (double)UPS_FADD(q[i][0], vector[i * 2 + 1]);
        A(i, n + 1) = (double)UPS_FADD(q[i][1], vector[i * 2 + 0]);
    }
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) A(TPS_NPTS + i, j) = 0.0;
        for (int j = 0; j < TPS_NPTS; ++j) A(TPS_NPTS + i, 3 + j) = (i == 0) ? 1.0 : (double)q[j][i - 1];
        A(TPS_NPTS + i, n + 0) = 0.0; A(TPS_NPTS + i, n + 1) = 0.0;
    }
    // canonical Gauss-Jordan (oracle/canon.py::solve_canon)
    for (int c = 0; c < n; ++c) {
        int p = c; double best = fabs(A(c, c));
        for (int r = c + 1; r < n; ++r) { const double v = fabs(A(r, c)); if (v > best) { best = v; p = r; } }
        if (p != c) for (int j = 0; j < m; ++j) { const double t = A(c, j); A(c, j) = A(p, j); A(p, j) = t; }
        const double piv = A(c, c);
        for (int r = 0; r < n; ++r) {
            if (r == c) continue;
            const double f = UPS_DDIV(A(r, c), piv);
            for (int j = c + 1; j < m; ++j) A(r, j) = UPS_DSUB(A(r, j), UPS_DMUL(f, A(c, j)));
        }
    }
    for (int c = 0; c < n; ++c) {
        T[0 * n + c] = (float)UPS_DDIV(A(c, n + 0), A(c, c));
        T[1 * n + c] = (float)UPS_DDIV(A(c, n + 1), A(c, c));
    }
}

// _meshgrid + T.grid (transformations.py:171-198) for one output pixel.
// q = flipped control points [8][2] (px = q[.][0], py = q[.][1]); T [2][11].
UPS_HD void tps_coords(const float* T, const float* qx, const float* qy, float x_t, float y_t,
                       float& x_s, float& y_s) {
    float ax = UPS_FADD(T[0], UPS_FMUL(T[1], x_t));
    ax = UPS_FADD(ax, UPS_FMUL(T[2], y_t));
    float ay = UPS_FADD(T[TPS_N + 0], UPS_FMUL(T[TPS_N + 1], x_t));
    ay = UPS_FADD(ay, UPS_FMUL(T[TPS_N + 2], y_t));
#pragma unroll
    for (int k = 0; k < TPS_NPTS; ++k) {
        const float dx = UPS_FSUB(x_t, qx[k]);
        const float dy = UPS_FSUB(y_t, qy[k]);
        const float d2 = UPS_FADD(UPS_FMUL(dx, dx), UPS_FMUL(dy, dy));
        const float r = tps_rbf(d2);
        ax = UPS_FADD(ax, UPS_FMUL(T[3 + k], r));
        ay = UPS_FADD(ay, UPS_FMUL(T[TPS_N + 3 + k], r));
    }
    x_s = ax; y_s = ay;
}

// tf.linspace(-1, 1, n)[i] = -1 + i*step, step = 2/(n-1)
UPS_HD float lin_step(int n) { return UPS_FDIV(2.0f, (float)(n - 1)); }
UPS_HD float lin_at(int i, float step) { return UPS_FADD(-1.0f, UPS_FMUL((float)i, step)); }

// _interpolate (transformations.py:114-169): stencil for one sample position.
struct Bilinear {
    int x0, x1, y0, y1;      // clipped corner indices
    float wa, wb, wc, wd;    // weights from the CLIPPED indices
    float X, Y;              // pixel-space position
};

UPS_HD Bilinear bilinear_stencil(float x_s, float y_s, int W, int H) {
    Bilinear b;
    b.X = UPS_FDIV(UPS_FMUL(UPS_FADD(x_s, 1.0f), (float)W), 2.0f);
    b.Y = UPS_FDIV(UPS_FMUL(UPS_FADD(y_s, 1.0f), (float)H), 2.0f);
    // floor in float, clamp in float (same result as int clamp for any finite value, and
    // immune to int overflow for far-out-of-range samples), then convert.
    const float fx = floorf(b.X), fy = floorf(b.Y);
    const float wmax = (float)(W - 1), hmax = (float)(H - 1);
    const float x0f = fminf(fmaxf(fx, 0.0f), wmax);
    const float x1f = fminf(fmaxf(UPS_FADD(fx, 1.0f), 0.0f), wmax);
    const float y0f = fminf(fmaxf(fy, 0.0f), hmax);
    const float y1f = fminf(fmaxf(UPS_FADD(fy, 1.0f), 0.0f), hmax);
    b.x0 = (int)x0f; b.x1 = (int)x1f; b.y0 = (int)y0f; b.y1 = (int)y1f;
    const float dx1 = UPS_FSUB(x1f, b.X), dx0 = UPS_FSUB(b.X, x0f);
    const float dy1 = UPS_FSUB(y1f, b.Y), dy0 = UPS_FSUB(b.Y, y0f);
    b.wa = UPS_FMUL(dx1, dy1);
    b.wb = UPS_FMUL(dx1, dy0);
    b.wc = UPS_FMUL(dx0, dy1);
    b.wd = UPS_FMUL(dx0, dy0);
    return b;
}

UPS_HD float bilinear_mix(const Bilinear& b, float Ia, float Ib, float Ic, float Id) {
    float o = UPS_FADD(UPS_FMUL(b.wa, Ia), UPS_FMUL(b.wb, Ib));
    o = UPS_FADD(o, UPS_FMUL(b.wc, Ic));
    return UPS_FADD(o, UPS_FMUL(b.wd, Id));
}

// Generic-K softmax row in canonical order (oracle/parts.py::_SoftmaxCanon.forward):
// p = exp_canon(x - max) * fl(1 / sum_tree(e)).  `e` is scratch with capacity >= next pow2 of K.
constexpr int KMAX = 64;
UPS_HD int next_pow2(int k) { int p = 1; while (p < k) p <<= 1; return p; }

UPS_HD float softmax_row_canon(const float* x, float* p, float* e, int K) {
    float mx = x[0];
    for (int k = 1; k < K; ++k) mx = x[k] > mx ? x[k] : mx;
    const int P2 = next_pow2(K);
    for (int k = 0; k < K; ++k) { const float v = exp_canon(UPS_FSUB(x[k], mx)); p[k] = v; e[k] = v; }
    for (int k = K; k < P2; ++k) e[k] = 0.0f;
    for (int w = P2 >> 1; w >= 1; w >>= 1)
        for (int i = 0; i < w; ++i) e[i] = UPS_FADD(e[2 * i], e[2 * i + 1]);
    const float rs = UPS_FRCP(e[0]);
    float pmax = 0.0f;
    for (int k = 0; k < K; ++k) { p[k] = UPS_FMUL(p[k], rs); pmax = p[k] > pmax ? p[k] : pmax; }
    return pmax;
}

// ---------------------------------------------------------------- the mean-field logit noise (oracle/noise.py::normal_philox)
// MeanFieldDistribution.sample (cub/code/nn.py:1421-1427) draws l = mean + noise_level * N(0,1).  The draw here is a pure
// function of (seed, draw, global pixel, part), so a kernel can generate it in registers wherever it reads the mean:
//   x[0..3] = Philox4x32-10(counter = (gpix lo, gpix hi, k / 4, draw), key = (seed lo, seed hi))
//             gpix = (sample_offset + b) * P + p;  draw = 0 for l0, 1 for l1
//   u(x)    = ((x >> 8) + 1) * 2^-24                       in (0, 1], exact in fp32
//   parts 4j, 4j+1 from (x0, x1), parts 4j+2, 4j+3 from (x2, x3), Box-Muller on (u_a, u_b):
//   r = sqrt(-2 * log_canon(u_a));  z = r * cos_canon(2 pi u_b),  r * sin_canon(2 pi u_b)      |z| <= 5.77, finite
//   sampled logit = fl(mean + fl(noise_level * z))  (-inf + finite = -inf: padded parts stay -inf)
// The value does not depend on K, the launch geometry or the batch split.
constexpr uint32_t PHILOX_M0 = 0xD2511F53u, PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u, PHILOX_W1 = 0xBB67AE85u;

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants): c <- philox(c, key)
UPS_HD void philox4x32_10(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = UPS_UMULHI(PHILOX_M0, c0), lo0 = PHILOX_M0 * c0;
        const uint32_t hi1 = UPS_UMULHI(PHILOX_M1, c2), lo1 = PHILOX_M1 * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += PHILOX_W0; k1 += PHILOX_W1;
    }
}

// (0, 1]: the top 24 bits of x plus one, times 2^-24 (integer -> float is exact below 2^24 + 1)
UPS_HD float uniform24(uint32_t x) { return UPS_FMUL((float)((x >> 8) + 1u), 5.9604644775390625e-8f); }

// sin and cos of 2 pi u for u in [0, 1], canonical order.  t = 4u and its fraction f are exact; f > 1/2 is folded to
// 1 - f (exact) so that the polynomial argument x = fl(g * pi/2) lies in [0, pi/4]; Cephes sinf / cosf polynomials,
// every operation rounded separately; the quadrant floor(t) mod 4 picks signs and the sin/cos swap.
UPS_HD void sincos2pi_canon(float u, float& s_out, float& c_out) {
    const float t = UPS_FMUL(u, 4.0f);
    const float q = floorf(t);
    const float f = UPS_FSUB(t, q);
    const bool fold = f > 0.5f;
    const float g = fold ? UPS_FSUB(1.0f, f) : f;
    const float x = UPS_FMUL(g, 1.57079632679489662f);
    const float z = UPS_FMUL(x, x);
    float sn = UPS_FADD(UPS_FMUL(-1.9515295891e-4f, z), 8.3321608736e-3f);
    sn = UPS_FADD(UPS_FMUL(sn, z), -1.6666654611e-1f);
    sn = UPS_FMUL(UPS_FMUL(sn, z), x);
    sn = UPS_FADD(sn, x);
    float cs = UPS_FADD(UPS_FMUL(2.443315711809948e-5f, z), -1.388731625493765e-3f);
    cs = UPS_FADD(UPS_FMUL(cs, z), 4.166664568298827e-2f);
    cs = UPS_FMUL(UPS_FMUL(cs, z), z);
    cs = UPS_FSUB(cs, UPS_FMUL(0.5f, z));
    cs = UPS_FADD(cs, 1.0f);
    const float s = fold ? cs : sn, c = fold ? sn : cs;   // sin, cos of (pi/2) f
    const int quad = ((int)q) & 3;
    s_out = quad == 0 ? s : quad == 1 ? c : quad == 2 ? -s : -c;
    c_out = quad == 0 ? c : quad == 1 ? -s : quad == 2 ? -c : s;
}

// two N(0,1) values from one pair of Philox words: (r cos, r sin)
UPS_HD void box_muller_canon(uint32_t xa, uint32_t xb, float& za, float& zb) {
    const float r = UPS_FSQRT(UPS_FMUL(-2.0f, log_canon(uniform24(xa))));
    float s, c;
    sincos2pi_canon(uniform24(xb), s, c);
    za = UPS_FMUL(r, c);
    zb = UPS_FMUL(r, s);
}

// the normals of parts 4j .. 4j+3 of global pixel `gpix`
UPS_HD void normal4_philox(unsigned long long seed, uint32_t draw, unsigned long long gpix, uint32_t j, float& z0,
                           float& z1, float& z2, float& z3) {
    uint32_t c0 = (uint32_t)gpix, c1 = (uint32_t)(gpix >> 32), c2 = j, c3 = draw;
    philox4x32_10(c0, c1, c2, c3, (uint32_t)seed, (uint32_t)(seed >> 32));
    box_muller_canon(c0, c1, z0, z1);
    box_muller_canon(c2, c3, z2, z3);
}

UPS_HD float sampled_logit(float mean, float noise_level, float z) { return UPS_FADD(mean, UPS_FMUL(noise_level, z)); }

}  // namespace ups
