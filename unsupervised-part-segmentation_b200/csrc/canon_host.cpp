// Host build of canon_math.cuh for CPU-side bit-exactness tests against oracle/canon.py.
// TEST SUPPORT ONLY: not linked into libups_b200.so and never called by the product.
// g++ -O2 -ffp-contract=off -shared -fPIC canon_host.cpp -o libups_canon_host.so
#include "canon_math.cuh"
#include <vector>

extern "C" {

void ups_host_exp(const float* x, float* y, long long n) { for (long long i = 0; i < n; ++i) y[i] = ups::exp_canon(x[i]); }
void ups_host_log(const float* x, float* y, long long n) { for (long long i = 0; i < n; ++i) y[i] = ups::log_canon(x[i]); }

// the mean-field logit noise (canon_math.cuh::normal4_philox)
void ups_host_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out, long long n) {
    for (long long i = 0; i < n; ++i) {
        uint32_t c[4] = {ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3]};
        ups::philox4x32_10(c[0], c[1], c[2], c[3], key[2 * i], key[2 * i + 1]);
        for (int j = 0; j < 4; ++j) out[4 * i + j] = c[j];
    }
}
void ups_host_box_muller(const uint32_t* xa, const uint32_t* xb, float* za, float* zb, long long n) {
    for (long long i = 0; i < n; ++i) ups::box_muller_canon(xa[i], xb[i], za[i], zb[i]);
}
void ups_host_sincos2pi(const float* u, float* s, float* c, long long n) {
    for (long long i = 0; i < n; ++i) ups::sincos2pi_canon(u[i], s[i], c[i]);
}
// eps [n_pix, K] for global pixels pix_offset .. pix_offset + n_pix - 1 (ups_normal_philox_fwd on the host)
void ups_host_normal_philox(unsigned long long seed, int draw, long long pix_offset, long long n_pix, int K, float* out) {
    for (long long i = 0; i < n_pix; ++i)
        for (int j = 0; 4 * j < K; ++j) {
            float z[4];
            ups::normal4_philox(seed, (uint32_t)draw, (unsigned long long)(pix_offset + i), (uint32_t)j, z[0], z[1], z[2], z[3]);
            for (int l = 0; l < 4 && 4 * j + l < K; ++l) out[i * K + 4 * j + l] = z[l];
        }
}

void ups_host_softmax(const float* x, float* p, long long* labels, float* hard, long long n_pix, int K) {
    std::vector<float> e(ups::KMAX * 2);
    for (long long i = 0; i < n_pix; ++i) {
        const float pmax = ups::softmax_row_canon(x + i * K, p + i * K, e.data(), K);
        int arg = -1;
        for (int k = 0; k < K; ++k) {
            const float v = p[i * K + k];
            if (v == pmax && arg < 0) arg = k;
            if (hard) hard[i * K + k] = ups::st_value(v == pmax ? 1.0f : 0.0f, v);
        }
        if (labels) labels[i] = arg;
    }
}

void ups_host_tps_input_param(const float* coord, const float* vector, const float* offset, const float* offset_2,
                              const float* t_scal, const float* rot, float* t_vector, int N) {
    for (int b = 0; b < N; ++b)
        ups::tps_input_param(coord + b * 16, vector + b * 16, offset + b * 2, offset_2 + b * 2, t_scal + b * 2,
                             rot + b * 4, t_vector + b * 16);
}

struct HostAcc {
    double* a;
    double& operator()(int i, int j) const { return a[i * 13 + j]; }
};

void ups_host_tps_solve(const float* coord, const float* vector, float* T, int N) {
    double A[11 * 13];
    for (int b = 0; b < N; ++b) ups::tps_solve(coord + b * 16, vector + b * 16, HostAcc{A}, T + b * 22);
}

// full forward warp on the host with the device's arithmetic (mesh = (y_s, x_s) like t_arr)
void ups_host_tps_warp(const float* U, const float* coord, const float* T, float* out, float* mesh, int N, int H,
                       int W, int C, int oh, int ow) {
    const float sw = ups::lin_step(ow), sh = ups::lin_step(oh);
    for (int b = 0; b < N; ++b) {
        float qx[8], qy[8];
        for (int k = 0; k < 8; ++k) { qx[k] = coord[b * 16 + k * 2 + 1]; qy[k] = coord[b * 16 + k * 2 + 0]; }
        for (int i = 0; i < oh; ++i)
            for (int j = 0; j < ow; ++j) {
                float xs, ys;
                ups::tps_coords(T + b * 22, qx, qy, ups::lin_at(j, sw), ups::lin_at(i, sh), xs, ys);
                const ups::Bilinear s = ups::bilinear_stencil(xs, ys, W, H);
                const long long o = ((long long)b * oh + i) * ow + j;
                if (mesh) { mesh[o * 2 + 0] = ys; mesh[o * 2 + 1] = xs; }
                const float* Ub = U + (long long)b * H * W * C;
                for (int c = 0; c < C; ++c)
                    out[o * C + c] = ups::bilinear_mix(s, Ub[(s.y0 * W + s.x0) * C + c], Ub[(s.y1 * W + s.x0) * C + c],
                                                       Ub[(s.y0 * W + s.x1) * C + c], Ub[(s.y1 * W + s.x1) * C + c]);
            }
    }
}
}
