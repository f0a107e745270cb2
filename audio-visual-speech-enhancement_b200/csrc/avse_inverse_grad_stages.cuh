// Warp-stage functions of the inverse's backward kernel ("IG"): the vector-Jacobian product of the mixture-phase
// reconstruction (avse_inverse without an explicit phase) with respect to its dB input, at the specialised geometry
// (640 / 160 / 80 / 20).  For frame t < T_use, with g = dL/dy:
//
//   h_t[n] = w[n] e[t hop + n],   e = g placed at offset 320 of the untrimmed signal / window sum-square
//   d_t[k] = (c_k / 640) Re(conj(phi_t[k]) rfft(h_t)[k]),   c = 2 inside, 1 at DC / Nyquist (only Re phi Re H there)
//   dL/d dB_t = ln(10) / 20 * 10^(dB_t / 20) * (F F^T)^-1 F d_t
//
// Every frame is independent (an analysis transform, no overlap-add): one warp runs one frame at a time through
//   ig_load (gradient and mixture samples of the frame) -> ig_pack (z = s h + i m into the FFT rows) -> ig_pass1 (DFT-16
//   per column + twiddle) -> ig_pass2 (DFT-40 per row) -> ig_post (unpack, phase, d) -> ig_mel (F d into the frame's slot),
// and after up to 32 frames ig_solve runs the tridiagonal solve and the dB chain rule with one lane per frame.
//
// Numerics: the gradient frame and the mixture frame of the same t share ONE packed float32 FFT.  Rounding of either channel
// leaks into the other in proportion to its raw power, and a loss gradient can sit 1e-8 under the mixture, so the gradient
// channel is scaled by s = 2^e chosen per frame to match the raw powers (ig_scale_exp); the scale is undone exactly in d.
// A frame whose windowed gradient is all zero gives exact zeros; a frame whose windowed mixture is all zero has phase 1 + 0j
// (librosa.magphase where D == 0), not the leakage of the gradient channel.  grad(2^k g) == 2^k grad(g) bitwise.
//
// Every function is __host__ __device__ (tests/emul runs a warp as a loop over lanes).
#pragma once
#include <cstring>
#include "avse_common.h"
#include "avse_dft.cuh"
#include "avse_inv8_stages.cuh"

namespace avse {

constexpr int IG_ROW = N2 + 1;                      // complex per FFT row (41: the 16 rows of pass 2 hit distinct banks)
constexpr int IG_FR_F = 2 * N1 * IG_ROW;            // 1312 floats: rows of the packed FFT, then its spectrum Z[0, 640)
constexpr int IG_D_F = 352;                         // d[k] for k < 321, zeros up to the widest band's reach (320 + MEL_WMAX)
constexpr int IG_FPC = 32;                          // frames per chunk: one per lane in the solve
constexpr int IG_FD_ROW = NMEL + 1;                 // F d of one frame (81: the solve's column reads hit distinct banks)
constexpr int IG_WARP_F = IG_FR_F + IG_D_F + IG_FPC * IG_FD_ROW;     // 4256 floats per warp
constexpr int IG_SPL = NFFT / 32;                   // 20 samples per lane
static_assert(2 * NFFT <= IG_FR_F && NBINS - 1 + MEL_WMAX <= IG_D_F, "buffers");

struct GradFrame {
    const float* pcm;      // mixture samples of the utterance
    int L;                 // reflect domain of librosa.stft
    int valid;             // samples present (zeros beyond)
    const float* grad;     // dL/dy of the utterance
    int out_len;           // 160 (T_use - 1)
    int T_use;
};

AVSE_HD unsigned ig_abs_bits(float x) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(fabsf(x));
#else
    unsigned u;
    const float a = std::fabs(x);
    std::memcpy(&u, &a, 4);
    return u;
#endif
}

// 2^k as a float, k clamped to the normal range (exact)
AVSE_HD float ig_pow2(int k) {
    k = k < -126 ? -126 : (k > 127 ? 127 : k);
    const unsigned u = (unsigned)(127 + k) << 23;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f;
    std::memcpy(&f, &u, 4);
    return f;
#endif
}

// exponent of the largest |x| (the bit pattern of a non-negative float orders like the float), floor(log2)
AVSE_HD int ig_exp_of_bits(unsigned b) { return b >= 0x00800000u ? (int)(b >> 23) - 127 : -127; }

// Lane's 20 samples n = lane + 32 i of frame t: the windowed, normalised gradient and the windowed mixture (reflect padding,
// zeros at or past `valid`).  am / ag: lane maxima of |.| as bit patterns.
AVSE_HD void ig_load(const GradFrame& f, int t, int lane, const float* s_win, float (&hg)[IG_SPL], float (&hm)[IG_SPL], unsigned& ag,
                     unsigned& am) {
    ag = 0u; am = 0u;
#pragma unroll
    for (int i = 0; i < IG_SPL; ++i) {
        const int n = lane + 32 * i;
        const int P = t * HOP + n;                 // untrimmed position
        const int o = P - HALF;                    // sample of y
        const float w = s_win[n];
        float e = 0.0f;
        if (o >= 0 && o < f.out_len) e = f.grad[o] * inv_wss_recip_w(P, f.T_use, s_win);
        const int j = i8_reflect_index(o, f.L);
        const float x = j >= 0 && j < f.valid ? f.pcm[j] : 0.0f;
        hg[i] = w * e;
        hm[i] = w * x;
        const unsigned bg = ig_abs_bits(hg[i]), bm = ig_abs_bits(hm[i]);
        ag = bg > ag ? bg : ag;
        am = bm > am ? bm : am;
    }
}

// Lane partial raw powers after normalising each channel by 2^-exponent(max |.|) (so that no square under- or overflows).
AVSE_HD void ig_power(const float (&hg)[IG_SPL], const float (&hm)[IG_SPL], int eg, int em, float& pg, float& pm) {
    const float sg = ig_pow2(-eg), sm = ig_pow2(-em);
    pg = 0.0f; pm = 0.0f;
#pragma unroll
    for (int i = 0; i < IG_SPL; ++i) {
        const float a = hg[i] * sg, b = hm[i] * sm;
        pg = fmaf(a, a, pg);
        pm = fmaf(b, b, pm);
    }
}

// Exponent e of the gradient channel's scale 2^e: raw powers equal to within a factor 4.  eg / em: exponents of the channels'
// largest |.|; pg / pm: their powers after normalisation by 2^-eg / 2^-em (warp sums).  A silent mixture frame: the gradient
// alone, normalised to about 1.
AVSE_HD int ig_scale_exp(int eg, int em, float pg, float pm, bool mix_any) {
    int e = -eg;
    if (mix_any) {
        e = em - eg;
        if (pg > 0.0f && pm > 0.0f) e += ig_exp_of_bits(ig_abs_bits(pm / pg)) >> 1;
    }
    return e < -120 ? -120 : (e > 120 ? 120 : e);
}

// z[n] = s h_g[n] + i h_m[n] into the rows: n = 40 a + b at complex index 41 a + b.
AVSE_HD void ig_pack(int lane, const float (&hg)[IG_SPL], const float (&hm)[IG_SPL], float s, float* fr) {
#pragma unroll
    for (int i = 0; i < IG_SPL; ++i) {
        const int n = lane + 32 * i, a = n / N2, b = n - a * N2;
        cstore(fr + 2 * (IG_ROW * a + b), cmake(s * hg[i], hm[i]));
    }
}

// Pass 1: column b (lanes 0..31, then 0..7 for b = 32..39): DFT-16 over a, twiddle W_640^{b c}, in place (row c, column b).
AVSE_HD void ig_pass1(int b, const float* s_tw, float* fr) {
    cpx x[16];
#pragma unroll
    for (int a = 0; a < N1; ++a) x[a] = cload(fr + 2 * (IG_ROW * a + b));
    dft16(x);
#pragma unroll
    for (int c = 0; c < N1; ++c) {
        const float* w = s_tw + 2 * (c * N2 + b);
        cstore(fr + 2 * (IG_ROW * c + b), c == 0 ? x[0] : cmul(x[c], w[0], w[1]));
    }
}

// Pass 2: row c (lanes 0..15): DFT-40 over b -> X[c + 16 d].  Load, then (after a __syncwarp) ig_pass2_store in natural order.
AVSE_HD void ig_pass2_load(int c, const float* fr, cpx (&x)[40]) {
#pragma unroll
    for (int b = 0; b < N2; ++b) x[b] = cload(fr + 2 * (IG_ROW * c + b));
    dft40_inplace(x);
}
AVSE_HD void ig_pass2_store(int c, const cpx (&x)[40], float* fr) {
#pragma unroll
    for (int p = 0; p < 5; ++p)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int k = (16 * p + 25 * q) % 40;           // dft40_inplace's output order
            cstore(fr + 2 * (c + N1 * k), x[(8 * p + 5 * q) % 40]);
        }
}

// Post: bins k = lane + 32 j.  Z = FFT(s h_g + i h_m): 2 G = Z_k + conj(Z_-k) (gradient), 2 M = -i (Z_k - conj(Z_-k)) (mixture),
// phi = M / |M| (1 + 0j on a silent mixture frame or where M == 0), d_k = (c_k / 640) 2^-e Re(conj(phi) 2 G) -- the 1/2 of the
// unpack cancels the 2 of the mel tables' 0.5 F weights.
AVSE_HD void ig_post(int lane, const float* fr, float inv_s, bool mix_any, float* d) {
    constexpr float C_IN = 2.0f / NFFT, C_EDGE = 1.0f / NFFT;
    for (int k = lane; k < NBINS; k += 32) {
        const cpx za = cload(fr + 2 * k), zb = cload(fr + 2 * ((NFFT - k) % NFFT));
        const float gr = cre(za) + cre(zb), gi = cim(za) - cim(zb);
        float pr = 1.0f, pi = 0.0f;
        if (mix_any) {
            const float mr = cim(za) + cim(zb), mi = cre(zb) - cre(za);
            const float r = hypotf(mr, mi);
            if (r > 0.0f) { pr = mr / r; pi = mi / r; }
        }
        const bool edge = k == 0 || k == HALF;
        d[k] = edge ? (C_EDGE * inv_s) * (pr * gr) : (C_IN * inv_s) * fmaf(pr, gr, pi * gi);
    }
}

// F d (80 bands, lanes m = lane + 32 j): the forward's banded 0.5 F weights [80][MEL_WROW], zero past each band's width.
AVSE_HD void ig_mel(int lane, const float* s_melw, const int* s_mello, const float* d, float* fd) {
    for (int m = lane; m < NMEL; m += 32) {
        const float* w = s_melw + m * MEL_WROW;
        const float* x = d + s_mello[m];
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < MEL_WMAX; ++j) acc = fmaf(w[j], x[j], acc);
        fd[m] = acc;
    }
}

// Lane j of the solve: (F F^T)^-1 (F d) by Thomas (the factors avse_mel_to_coef_kernel uses), times ln(10)/20 10^(dB/20),
// stored in mel_db's layout.  Frames t >= T_use (up to the frames the layout holds) get exact zeros.
AVSE_HD void ig_solve(const float* fd, int t, int T_use, const float* mel, float* out, int layout, int ld_t, const float* s_tri) {
    size_t base, mstride;
    if (layout == 0) {              // AVSE_LAYOUT_SLICES
        const int s = t / SPSS, tt = t - s * SPSS;
        base = (size_t)s * NMEL * SPSS + tt;
        mstride = SPSS;
    } else {
        base = (size_t)t;
        mstride = (size_t)ld_t;
    }
    if (t >= T_use) {
        for (int m = 0; m < NMEL; ++m) out[base + m * mstride] = 0.0f;
        return;
    }
    const float* tw = s_tri;
    const float* ipiv = s_tri + NMEL;
    const float* sup = s_tri + 2 * NMEL;
    float x[NMEL];
#pragma unroll
    for (int m = 0; m < NMEL; ++m) x[m] = fd[m];
#pragma unroll
    for (int m = 1; m < NMEL; ++m) x[m] -= tw[m] * x[m - 1];
    x[NMEL - 1] *= ipiv[NMEL - 1];
#pragma unroll
    for (int m = NMEL - 2; m >= 0; --m) x[m] = (x[m] - sup[m] * x[m + 1]) * ipiv[m];
    constexpr float K = 0.16609640474436813f;      // log2(10) / 20: 10^(dB/20) = 2^(K dB), as the forward computes it
    constexpr float LN10_20 = 0.11512925464970229f;
#pragma unroll
    for (int m = 0; m < NMEL; ++m) out[base + m * mstride] = LN10_20 * exp2f(K * mel[base + m * mstride]) * x[m];
}

}  // namespace avse
