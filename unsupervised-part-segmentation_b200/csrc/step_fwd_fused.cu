// K1 + K3 in ONE launch: the TPS warp of the views (FMA-pipe bound: 8 canonical logs per pixel, 16 % of DRAM
// bandwidth) and the decode-side forward (softmax(l0) -> labels -> inject; HBM bound, 34 % issue) do not depend on each
// other (model.py:282-311 vs :426-447,482-484), so their CTAs are interleaved in one grid: every SM holds CTAs of both
// roles and the arithmetic of one hides under the memory stream of the other.  Horizontal fusion, no second stream:
// the call is timed as one kernel whose algorithmic bytes are the sum of both roles'.
//
// Role of block i (n1 warp CTAs, n3 decode CTAs, G = n1 + n3): with c3(i) = floor(i*n3/G) the number of decode blocks
// among the first i, block i is a decode block iff c3(i+1) > c3(i) (its decode index is c3(i)); otherwise it is warp
// block i - c3(i).  Both roles therefore start and finish together, evenly mixed over the whole launch.
#include "common.cuh"
#include "step_decode_fwd.cuh"
#include "tps_warp_fwd.cuh"

namespace ups {

struct WarpArgs {
    const float* U; const float* U2; const float* coord; const float* T;
    float* out; float* out2;
    int N2, H, W, oh, ow, tiles_per_sample;
};
struct DecodeArgs {
    const float* l0; const float* feat; float* m0; long long* labels0; float* inj;
    int P, F, pix_per_cta, splits, l0_row;
    NoiseArgs nz;      // NOISE instantiations only: l0 holds the means
};

static_assert(WARP_TPB == FTPB, "both roles use 128-thread CTAs");

template <int LPP, int FT, int MINB, bool NOISE>
__global__ void __launch_bounds__(FTPB, MINB) step_warp_decode_fwd_kernel(const WarpArgs wa, const DecodeArgs da, unsigned n3,
                                                                         unsigned total) {
    extern __shared__ float4 dyn4[];   // decode role: K*F floats; warp role: 2*128*3 staged pixels + 42 constants
    const unsigned i = blockIdx.x;
    const unsigned c3 = (unsigned)(((unsigned long long)i * n3) / total);
    const unsigned c3n = (unsigned)(((unsigned long long)(i + 1) * n3) / total);
    if (c3n > c3) {
        const int b = (int)(c3 / (unsigned)da.splits), split = (int)(c3 - (unsigned)b * da.splits);
        step_decode_fwd_body<LPP, FT, NOISE>(da.l0, da.feat, da.m0, da.labels0, da.inj, da.P, da.F, da.pix_per_cta, split, b, dyn4,
                                             da.l0_row, da.nz);
    } else {
        const unsigned j = i - c3;
        const int b = (int)(j / (unsigned)wa.tiles_per_sample), tile = (int)(j - (unsigned)b * wa.tiles_per_sample);
        float* sm = reinterpret_cast<float*>(dyn4);
        tps_warp_fwd_body<3>(wa.U, wa.U2, wa.coord, wa.T, nullptr, nullptr, wa.out, wa.out2, nullptr, wa.N2, wa.H, wa.W, 3,
                             wa.oh, wa.ow, tile, b, sm + 2 * WARP_TPB * 3, sm);
    }
}

int fused_pix_per_cta(int B, int P);

}  // namespace ups

using namespace ups;

extern "C" int ups_step_warp_decode_fwd(const float* U, const float* U2, const float* coord, const float* T, float* out,
                                        float* out2, int N, int N2, int S, const float* l0, const float* feat, float* m0,
                                        long long* labels0, float* inj, int B, int K, int F, void* stream) {
    return ups_step_warp_decode_fwd_rows(U, U2, coord, T, out, out2, N, N2, S, l0, K, feat, m0, labels0, inj, B, K, F, stream);
}

template <bool NOISE>
static int warp_decode_fwd_launch(const float* U, const float* U2, const float* coord, const float* T, float* out, float* out2,
                                  int N, int N2, int S, const float* l0, int l0_row, const float* feat, float* m0,
                                  long long* labels0, float* inj, int B, int K, int F, NoiseArgs nz, void* stream) {
    UPS_REQUIRE(l0_row >= 1 && l0_row <= K, "step_warp_decode_fwd: l0 rows of %d floats for K=%d", l0_row, K);
    UPS_REQUIRE(U && coord && T && out && l0 && feat && m0 && labels0 && inj, "step_warp_decode_fwd: null pointer");
    UPS_REQUIRE((U2 == nullptr) == (out2 == nullptr), "step_warp_decode_fwd: U2 and out2 must be given together");
    UPS_REQUIRE(N > 0 && N <= 65535 && N2 >= 0 && N2 <= N && S > 1, "step_warp_decode_fwd: N=%d N2=%d S=%d", N, N2, S);
    UPS_REQUIRE(B > 0 && B <= 65535, "step_warp_decode_fwd: B=%d out of range", B);
    UPS_REQUIRE(K == 8 || K == 16 || K == 32, "step_warp_decode_fwd: needs K in {8,16,32}, got %d", K);
    UPS_REQUIRE(F == 16 || F == 32 || F == 64, "step_warp_decode_fwd: needs F in {16,32,64}, got %d", F);
    const int P = S * S;
    UPS_REQUIRE(P % 32 == 0 && (long long)S * S * 3 < (1ll << 31), "step_warp_decode_fwd: S=%d unsupported", S);
    UPS_REQUIRE((l0_row < K || aligned16(l0)) && aligned16(feat) && aligned16(m0) && aligned16(inj), "step_warp_decode_fwd: 16-byte alignment");
    WarpArgs wa{U, U2, coord, T, out, out2, N2, S, S, S, S, (int)cdiv((long long)P, WARP_TPB * WARP_PPT)};
    const int per = fused_pix_per_cta(B, P);
    DecodeArgs da{l0, feat, m0, labels0, inj, P, F, per, (int)cdiv(P, per), l0_row, nz};
    const unsigned long long n1 = (unsigned long long)N * wa.tiles_per_sample, n3 = (unsigned long long)B * da.splits;
    UPS_REQUIRE(n1 + n3 < (1ull << 31), "step_warp_decode_fwd: grid too large");
    const unsigned total = (unsigned)(n1 + n3);
    size_t sm = (size_t)K * F * sizeof(float);
    const size_t sm1 = ((size_t)2 * WARP_TPB * 3 + 48) * sizeof(float);
    if (sm1 > sm) sm = sm1;
    cudaStream_t s = as_stream(stream);
    static const int minb = []() { const char* e = getenv("UPS_FWD_FUSED_MINB"); return e ? atoi(e) : 5; }();
#define UPS_WD3(LPP, FT, MB)                                                                                    \
    {                                                                                                           \
        if (sm > 48 * 1024)                                                                                     \
            UPS_CUDA(cudaFuncSetAttribute(step_warp_decode_fwd_kernel<LPP, FT, MB, NOISE>,                      \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));               \
        step_warp_decode_fwd_kernel<LPP, FT, MB, NOISE><<<total, FTPB, sm, s>>>(wa, da, (unsigned)n3, total);   \
    }
#define UPS_WD2(LPP, FT) { if (minb == 5) UPS_WD3(LPP, FT, 5) else if (minb == 6) UPS_WD3(LPP, FT, 6) else UPS_WD3(LPP, FT, 4) }
#define UPS_WD(LPP) { if (F == 64) UPS_WD2(LPP, 64) else if (F == 32) UPS_WD2(LPP, 32) else UPS_WD2(LPP, 16) }
    if (K == 8) UPS_WD(2) else if (K == 16) UPS_WD(4) else UPS_WD(8)
#undef UPS_WD
#undef UPS_WD2
#undef UPS_WD3
    return after_launch("step_warp_decode_fwd_kernel");
}

extern "C" int ups_step_warp_decode_fwd_rows(const float* U, const float* U2, const float* coord, const float* T, float* out,
                                             float* out2, int N, int N2, int S, const float* l0, int l0_row, const float* feat,
                                             float* m0, long long* labels0, float* inj, int B, int K, int F, void* stream) {
    return warp_decode_fwd_launch<false>(U, U2, coord, T, out, out2, N, N2, S, l0, l0_row, feat, m0, labels0, inj, B, K, F,
                                         NoiseArgs{}, stream);
}

extern "C" int ups_step_warp_decode_fwd_noise(const float* U, const float* U2, const float* coord, const float* T, float* out,
                                              float* out2, int N, int N2, int S, const float* l0, int l0_row, const float* feat,
                                              float* m0, long long* labels0, float* inj, int B, int K, int F,
                                              unsigned long long seed, long long sample_offset, float noise_level,
                                              void* stream) {
    UPS_REQUIRE(sample_offset >= 0, "step_warp_decode_fwd: sample_offset=%lld", sample_offset);
    return warp_decode_fwd_launch<true>(U, U2, coord, T, out, out2, N, N2, S, l0, l0_row, feat, m0, labels0, inj, B, K, F,
                                        NoiseArgs{seed, sample_offset, noise_level, 0}, stream);
}
