// Host-side (float64) construction of the constant tables the kernels read:
// periodic Hann window, pass-1 twiddles, the Slaney mel filterbank in banded form, and the
// structured pseudo-inverse (pinv(F) = F^T (F F^T)^-1 with F F^T tridiagonal).
// Restates librosa.filters.mel / get_window as used at /root/reference/data_processor.py:79-89,
// :104-112 (library semantics: SURVEY.md Appendix A.1).  Plain C++, no CUDA.
#pragma once
#include <vector>
#include <string>
#include "avse_common.h"

namespace avse {

constexpr int SPIKE_P = 4;            // partitions of the 80-band tridiagonal solve
constexpr int SPIKE_Q = NMEL / SPIKE_P;   // 20 bands each
constexpr int SPIKE_ROW = 5 * SPIKE_Q + 16;   // 116 floats per partition
static_assert(SPIKE_P * SPIKE_Q == NMEL, "partition of the mel bands");
// Largest 1-norm cond(F F^T) build_tables accepts.  The I8 inverse's float32 solve drifts from np.linalg.pinv (dp:112) by about
// 1.5e-11 * cond of the output's peak (emulated I8 kernel, 16 kHz sweep of fmin 0...1500 / fmax 2000...8000): at cond <= 1e5 the
// error stays <= 1e-5, 10x under the 1e-4 gate; the first bank over the gate is at cond 5.6e6, 56x above this threshold.
constexpr double GRAM_COND_MAX = 1e5;

struct HostTables {
    int sample_rate = 16000;
    double fmin = 0.0, fmax = 8000.0;

    std::vector<float> window;        // [640]   periodic Hann
    std::vector<float> tw1t;          // [16][40][2]  W_640^{n2*k1}, k1-major (re, im)
    std::vector<double> fb;           // [80][321]  dense filterbank (float64, for tests/inverse)
    std::vector<int> mel_lo;          // [80]  first non-zero bin of each band
    std::vector<int> mel_width;       // [80]  number of non-zero bins
    std::vector<float> mel_w;         // [80][MEL_WROW]  0.5 * weight (0.5 = packed-FFT unpack factor)
    std::vector<int> mel_roundw;      // [5]   max width over bands 16r..16r+15

    // fused post+mel "scan" (see avse_fwd_stages.cuh stage_post_scan): valid when scan_ok
    bool scan_ok = false;
    std::vector<float> scan_w;        // [SCAN_BINS][4]  (wA, wA, wB, wB), 0.5 * weights (pairs feed packed FFMA2)
    std::vector<int> scan_mask;       // [16]  bit i of chunk p: a band is finished before bin 21p + i (emit accumulator A)
    std::vector<float> window2;       // [640][2]  (w, w) pairs of the periodic Hann window
    std::vector<int> scan_loc;        // [80][4]  frame-relative float offsets (SN0, M0, SN1, M1) of each band's <= 2 partial sums

    // F4 kernel (avse_fwd4_stages.cuh stage4_scan / stage4_db): 8 chunks of 41 bins, dense emission; valid when scan4_ok
    bool scan4_ok = false;
    std::vector<float> scan4_w;       // [328][2]  (wa, wb) = 0.5 * (F[seg-1][k], F[seg][k])
    std::vector<unsigned> scan4_mask; // [8][2]    bit i of chunk p (lo, hi words): a band is finished before bin 41 p + i
    std::vector<int> scan4_loc;       // [80][4]   (main, extra1, extra2, -) packed partial-sum offsets (sn | m << 16), -1 = absent

    // inverse path
    std::vector<float> tri_w;         // [80] Thomas forward multipliers (w[0] unused)
    std::vector<float> tri_ipiv;      // [80] 1 / pivot
    std::vector<float> tri_sup;       // [80] super-diagonal (sup[79] unused)
    double gram_cond = 0.0;           // 1-norm condition number of F F^T (float64)
    // the same solve partitioned for a warp (I8 inverse kernel): 4 blocks of 20 bands, "SPIKE" form -- per block the local Thomas
    // factors (w, 1/pivot, super-diagonal), the left / right spikes A_p^-1 (T[r0][r0-1] e_0), A_p^-1 (T[r0+19][r0+20] e_19) and the
    // two rows of the inverse 8 x 8 interface system that give x[r0-1] and x[r0+20] from the blocks' local (top, bottom) values
    std::vector<float> spike;         // [4][SPIKE_ROW]: lw[20] lipiv[20] lsup[20] wv[20] vv[20] rb[8] rt[8]
    std::vector<int> col_band;        // [321][2] band index of the (<=2) non-zeros in column k (or 0)
    std::vector<float> col_w;         // [321][2] their weights (0 when absent)
    // the same columns as a walk (I8 post stage): bin k reads the coefficient pair (y[post_b[k]], y[post_b[k] + 1]) with weights
    // post_w[k]; post_b is non-decreasing in steps of <= 1 and stays in [0, 78], so a lane walking a chunk of bins keeps the pair
    // in registers and advances it on the bits of a mask.  post_ok == false: the filterbank does not allow it; build_tables then
    // refuses the bank (the I8 kernel is the specialised context's only inverse) and the generic kernels serve it.
    bool post_ok = false;
    std::vector<int> post_b;          // [328]
    std::vector<float> post_w;        // [328][2]
    std::vector<unsigned> post_mask;  // [8][4] per chunk of 41 bins: (mask lo, mask hi, first band, 0); bit i: the pair advances before bin 41 p + i

    std::string error;                // non-empty when the configuration is unsupported
};

// Fills all tables.  Returns false (and sets t.error) when the configuration cannot be
// represented in banded form (empty band, band wider than MEL_WMAX, column with > 2 non-zeros,
// F F^T not tridiagonal), or when the I8 inverse cannot serve it (post_ok == false, or
// gram_cond > GRAM_COND_MAX).  The flags and gram_cond are set before the last two checks.
bool build_tables(HostTables& t, int sample_rate, double fmin, double fmax);

}  // namespace avse
