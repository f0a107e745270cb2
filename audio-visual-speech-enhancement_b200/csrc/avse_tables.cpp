// See avse_tables.h.  Float64 throughout; rounded to float32 once at the end.
#include "avse_tables.h"

#include <cmath>
#include <algorithm>

namespace avse {

namespace {

const double kPi = 3.14159265358979323846;

// librosa.hz_to_mel / mel_to_hz, htk=False (Slaney): linear below 1 kHz, log above.
double hz_to_mel(double f) {
    const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0;
    const double min_log_mel = min_log_hz / f_sp, logstep = std::log(6.4) / 27.0;
    return f >= min_log_hz ? min_log_mel + std::log(f / min_log_hz) / logstep : f / f_sp;
}
double mel_to_hz(double m) {
    const double f_sp = 200.0 / 3.0, min_log_hz = 1000.0;
    const double min_log_mel = min_log_hz / f_sp, logstep = std::log(6.4) / 27.0;
    return m >= min_log_mel ? min_log_hz * std::exp(logstep * (m - min_log_mel)) : f_sp * m;
}

}  // namespace

bool build_tables(HostTables& t, int sample_rate, double fmin, double fmax) {
    t.sample_rate = sample_rate;
    t.fmin = fmin;
    t.fmax = fmax;
    t.error.clear();

    // periodic Hann: scipy.signal.get_window('hann', n_fft, fftbins=True)
    t.window.resize(NFFT);
    for (int n = 0; n < NFFT; ++n) t.window[n] = (float)(0.5 - 0.5 * std::cos(2.0 * kPi * n / NFFT));

    // pass-1 twiddles W_640^{n2*k1} = exp(-2 pi i n2 k1 / 640), layout [k1][n2]
    t.tw1t.resize(N1 * N2 * 2);
    for (int k1 = 0; k1 < N1; ++k1)
        for (int n2 = 0; n2 < N2; ++n2) {
            const int e = (n2 * k1) % NFFT;
            const double a = -2.0 * kPi * e / NFFT;
            t.tw1t[(k1 * N2 + n2) * 2 + 0] = (float)std::cos(a);
            t.tw1t[(k1 * N2 + n2) * 2 + 1] = (float)std::sin(a);
        }

    // librosa.filters.mel(sr, n_fft, n_mels=80, fmin, fmax), htk=False, norm=1 (Slaney)
    std::vector<double> mel_f(NMEL + 2);
    {
        const double m0 = hz_to_mel(fmin), m1 = hz_to_mel(fmax);
        for (int j = 0; j < NMEL + 2; ++j) mel_f[j] = mel_to_hz(m0 + (m1 - m0) * j / (NMEL + 1));
    }
    t.fb.assign((size_t)NMEL * NBINS, 0.0);
    for (int m = 0; m < NMEL; ++m) {
        const double fd0 = mel_f[m + 1] - mel_f[m], fd1 = mel_f[m + 2] - mel_f[m + 1];
        const double enorm = 2.0 / (mel_f[m + 2] - mel_f[m]);
        for (int k = 0; k < NBINS; ++k) {
            const double fk = (double)sample_rate / 2.0 * k / (NBINS - 1);  // np.linspace(0, sr/2, 321)
            const double lower = -(mel_f[m] - fk) / fd0;
            const double upper = (mel_f[m + 2] - fk) / fd1;
            t.fb[(size_t)m * NBINS + k] = std::max(0.0, std::min(lower, upper)) * enorm;
        }
        // A bin that sits exactly on a mel point (e.g. bin 320 = fmax) has weight 0 in exact
        // arithmetic; libm rounding can leave ~1e-16.  Snap those to 0 so the support is exact.
        double rmax = 0.0;
        for (int k = 0; k < NBINS; ++k) rmax = std::max(rmax, t.fb[(size_t)m * NBINS + k]);
        for (int k = 0; k < NBINS; ++k)
            if (t.fb[(size_t)m * NBINS + k] < 1e-10 * rmax) t.fb[(size_t)m * NBINS + k] = 0.0;
    }

    // banded form
    t.mel_lo.assign(NMEL, 0);
    t.mel_width.assign(NMEL, 0);
    t.mel_w.assign((size_t)NMEL * MEL_WROW, 0.0f);
    t.mel_roundw.assign(MEL_ROUNDS, 0);
    for (int m = 0; m < NMEL; ++m) {
        int lo = -1, hi = -1;
        for (int k = 0; k < NBINS; ++k)
            if (t.fb[(size_t)m * NBINS + k] != 0.0) { if (lo < 0) lo = k; hi = k; }
        if (lo < 0) { t.error = "empty mel band (unsupported sr/fmin/fmax for n_fft=640, n_mels=80)"; return false; }
        for (int k = lo; k <= hi; ++k)
            if (t.fb[(size_t)m * NBINS + k] == 0.0) { t.error = "mel band support not contiguous"; return false; }
        const int w = hi - lo + 1;
        if (w > MEL_WMAX) { t.error = "mel band wider than MEL_WMAX"; return false; }
        if (lo < 1 || hi > NBINS - 2) { t.error = "mel band touches DC/Nyquist bin (unsupported by the packed-FFT post stage)"; return false; }
        t.mel_lo[m] = lo;
        t.mel_width[m] = w;
        for (int j = 0; j < w; ++j) t.mel_w[(size_t)m * MEL_WROW + j] = (float)(0.5 * t.fb[(size_t)m * NBINS + lo + j]);
        t.mel_roundw[m / 16] = std::max(t.mel_roundw[m / 16], w);
    }

    // column form (<= 2 non-zeros per bin) for lin = F^T y
    t.col_band.assign((size_t)NBINS * 2, 0);
    t.col_w.assign((size_t)NBINS * 2, 0.0f);
    for (int k = 0; k < NBINS; ++k) {
        int c = 0;
        for (int m = 0; m < NMEL; ++m) {
            const double w = t.fb[(size_t)m * NBINS + k];
            if (w != 0.0) {
                if (c == 2) { t.error = "filterbank column with more than 2 non-zeros"; return false; }
                t.col_band[k * 2 + c] = m;
                t.col_w[k * 2 + c] = (float)w;
                ++c;
            }
        }
    }

    {   // walk form of the columns (see avse_tables.h)
        constexpr int PB = 328;
        t.post_b.assign(PB, 0);
        t.post_w.assign((size_t)PB * 2, 0.0f);
        t.post_ok = NMEL >= 2;
        int prev = -1;                                     // -1: the walk has not been pinned by a tap yet
        for (int k = 0; k < NBINS && t.post_ok; ++k) {
            const int b0 = t.col_band[2 * k], b1 = t.col_band[2 * k + 1];
            const float w0 = t.col_w[2 * k], w1 = t.col_w[2 * k + 1];
            int b = prev < 0 ? 0 : prev;
            float wa = 0.0f, wb = 0.0f;
            if (w0 != 0.0f && w1 != 0.0f) {
                if (b1 != b0 + 1) { t.post_ok = false; break; }
                b = b0; wa = w0; wb = w1;
            } else if (w0 != 0.0f) {                       // one tap (band b0): it can be the pair's first or second member
                const bool first_ok = b0 <= NMEL - 2, second_ok = b0 >= 1;
                if (first_ok && (prev < 0 || b0 == prev || b0 == prev + 1) && !(second_ok && b0 - 1 == prev)) { b = b0; wa = w0; }
                else if (second_ok) { b = b0 - 1; wb = w0; }
                else { b = b0; wa = w0; }
            }
            if (prev >= 0 && b != prev && b != prev + 1) { t.post_ok = false; break; }
            t.post_b[k] = b; t.post_w[2 * k] = wa; t.post_w[2 * k + 1] = wb;
            if (w0 != 0.0f || prev >= 0) prev = b;
        }
        if (prev < 0) prev = 0;
        for (int k = NBINS; k < PB; ++k) t.post_b[k] = prev;
        for (int k = NBINS - 1; k > 0; --k)                // bins before the first tap sit on the first tap's pair
            if (t.post_w[2 * (k - 1)] == 0.0f && t.post_w[2 * (k - 1) + 1] == 0.0f && t.post_b[k - 1] > t.post_b[k]) t.post_b[k - 1] = t.post_b[k];
        for (int k = 1; k < PB && t.post_ok; ++k)
            if (t.post_b[k] < t.post_b[k - 1] || t.post_b[k] > t.post_b[k - 1] + 1 || t.post_b[k] > NMEL - 2) t.post_ok = false;
        constexpr int CH = 41;
        t.post_mask.assign(8 * 4, 0u);
        for (int p = 0; p < 8; ++p) {
            for (int i = 1; i < CH; ++i)
                if (t.post_b[CH * p + i] != t.post_b[CH * p + i - 1]) t.post_mask[4 * p + (i >> 5)] |= 1u << (i & 31);
            t.post_mask[4 * p + 2] = (unsigned)t.post_b[CH * p];
        }
    }

    // G = F F^T must be tridiagonal; Thomas factors in float64
    std::vector<double> diag(NMEL), sub(NMEL, 0.0), sup(NMEL, 0.0);
    for (int a = 0; a < NMEL; ++a)
        for (int b = 0; b < NMEL; ++b) {
            double g = 0.0;
            for (int k = 0; k < NBINS; ++k) g += t.fb[(size_t)a * NBINS + k] * t.fb[(size_t)b * NBINS + k];
            if (a == b) diag[a] = g;
            else if (b == a + 1) sup[a] = g;
            else if (b == a - 1) sub[a] = g;
            else if (g != 0.0) { t.error = "F F^T is not tridiagonal"; return false; }
        }
    t.tri_w.assign(NMEL, 0.0f);
    t.tri_ipiv.assign(NMEL, 0.0f);
    t.tri_sup.assign(NMEL, 0.0f);
    std::vector<double> piv(NMEL);
    piv[0] = diag[0];
    for (int i = 1; i < NMEL; ++i) {
        const double w = sub[i] / piv[i - 1];
        piv[i] = diag[i] - w * sup[i - 1];
        t.tri_w[i] = (float)w;
    }
    for (int i = 0; i < NMEL; ++i) {
        if (!(piv[i] > 0.0)) { t.error = "F F^T not positive definite"; return false; }
        t.tri_ipiv[i] = (float)(1.0 / piv[i]);
        t.tri_sup[i] = (float)sup[i];
    }
    {   // 1-norm condition number ||G||_1 ||G^-1||_1, the columns of G^-1 by the float64 Thomas factors
        double g_norm = 0.0, ginv_norm = 0.0;
        std::vector<double> x(NMEL);
        for (int j = 0; j < NMEL; ++j) {
            g_norm = std::max(g_norm, std::fabs(sub[j]) + diag[j] + std::fabs(sup[j]));
            for (int i = 0; i < NMEL; ++i) x[i] = i == j ? 1.0 : 0.0;
            for (int i = 1; i < NMEL; ++i) x[i] -= sub[i] / piv[i - 1] * x[i - 1];
            x[NMEL - 1] /= piv[NMEL - 1];
            for (int i = NMEL - 2; i >= 0; --i) x[i] = (x[i] - sup[i] * x[i + 1]) / piv[i];
            double s = 0.0;
            for (int i = 0; i < NMEL; ++i) s += std::fabs(x[i]);
            ginv_norm = std::max(ginv_norm, s);
        }
        t.gram_cond = g_norm * ginv_norm;
    }

    // ---- SPIKE partition of the same system (see avse_tables.h): everything in float64, rounded once ----
    {
        const int P = SPIKE_P, Q = SPIKE_Q;
        t.spike.assign((size_t)P * SPIKE_ROW, 0.0f);
        std::vector<std::vector<double>> wv(P, std::vector<double>(Q, 0.0)), vv(P, std::vector<double>(Q, 0.0));
        for (int p = 0; p < P; ++p) {
            const int r0 = Q * p;
            float* row = t.spike.data() + (size_t)p * SPIKE_ROW;
            std::vector<double> lp(Q), lw(Q, 0.0);
            lp[0] = diag[r0];
            for (int i = 1; i < Q; ++i) { lw[i] = sub[r0 + i] / lp[i - 1]; lp[i] = diag[r0 + i] - lw[i] * sup[r0 + i - 1]; }
            auto solve = [&](std::vector<double> d) {          // local Thomas solve in float64
                for (int i = 1; i < Q; ++i) d[i] -= lw[i] * d[i - 1];
                d[Q - 1] /= lp[Q - 1];
                for (int i = Q - 2; i >= 0; --i) d[i] = (d[i] - sup[r0 + i] * d[i + 1]) / lp[i];
                return d;
            };
            if (p > 0) { std::vector<double> e(Q, 0.0); e[0] = sub[r0]; wv[p] = solve(e); }
            if (p < P - 1) { std::vector<double> e(Q, 0.0); e[Q - 1] = sup[r0 + Q - 1]; vv[p] = solve(e); }
            for (int i = 0; i < Q; ++i) {
                row[i] = (float)lw[i];
                row[Q + i] = (float)(1.0 / lp[i]);
                row[2 * Q + i] = (float)(i < Q - 1 ? sup[r0 + i] : 0.0);
                row[3 * Q + i] = (float)wv[p][i];
                row[4 * Q + i] = (float)vv[p][i];
            }
        }
        // interface system (I + S) z = y,  z = (t_0, b_0, ..., t_3, b_3)
        const int M = 2 * P;
        std::vector<double> A((size_t)M * M, 0.0), R((size_t)M * M, 0.0);
        for (int i = 0; i < M; ++i) { A[(size_t)i * M + i] = 1.0; R[(size_t)i * M + i] = 1.0; }
        for (int p = 0; p < P; ++p) {
            if (p > 0) { A[(size_t)(2 * p) * M + 2 * (p - 1) + 1] = wv[p][0]; A[(size_t)(2 * p + 1) * M + 2 * (p - 1) + 1] = wv[p][Q - 1]; }
            if (p < P - 1) { A[(size_t)(2 * p) * M + 2 * (p + 1)] = vv[p][0]; A[(size_t)(2 * p + 1) * M + 2 * (p + 1)] = vv[p][Q - 1]; }
        }
        for (int c = 0; c < M; ++c) {                           // Gauss-Jordan with partial pivoting (8 x 8, diagonally dominant)
            int piv_r = c;
            for (int r = c + 1; r < M; ++r) if (std::fabs(A[(size_t)r * M + c]) > std::fabs(A[(size_t)piv_r * M + c])) piv_r = r;
            if (A[(size_t)piv_r * M + c] == 0.0) { t.error = "SPIKE interface system singular"; return false; }
            for (int k = 0; k < M; ++k) { std::swap(A[(size_t)c * M + k], A[(size_t)piv_r * M + k]); std::swap(R[(size_t)c * M + k], R[(size_t)piv_r * M + k]); }
            const double inv = 1.0 / A[(size_t)c * M + c];
            for (int k = 0; k < M; ++k) { A[(size_t)c * M + k] *= inv; R[(size_t)c * M + k] *= inv; }
            for (int r = 0; r < M; ++r) {
                if (r == c) continue;
                const double f = A[(size_t)r * M + c];
                if (f == 0.0) continue;
                for (int k = 0; k < M; ++k) { A[(size_t)r * M + k] -= f * A[(size_t)c * M + k]; R[(size_t)r * M + k] -= f * R[(size_t)c * M + k]; }
            }
        }
        for (int p = 0; p < P; ++p) {
            float* row = t.spike.data() + (size_t)p * SPIKE_ROW + 5 * SPIKE_Q;
            for (int k = 0; k < M; ++k) {
                row[k] = p > 0 ? (float)R[(size_t)(2 * (p - 1) + 1) * M + k] : 0.0f;          // x[r0 - 1]  = b_{p-1}
                row[M + k] = p < P - 1 ? (float)R[(size_t)(2 * (p + 1)) * M + k] : 0.0f;      // x[r0 + 20] = t_{p+1}
            }
        }
    }

    // ---- fused post+mel scan tables ----
    // Segment j = [mel_f[j], mel_f[j+1]); a bin in segment j feeds band j-1 (falling edge, accumulator A)
    // and band j (rising edge, accumulator B).  Lane chunk p scans bins 21p..21p+20 (p = 15: 315..319) and
    // emits A whenever the segment index advances; the two accumulators left at the chunk end are flushed.
    // Every band must end up with at most two partial sums ("locations") or the scan is not usable.
    t.window2.resize(2 * NFFT);
    for (int n = 0; n < NFFT; ++n) { t.window2[2 * n] = t.window[n]; t.window2[2 * n + 1] = t.window[n]; }
    t.scan_ok = true;
    t.scan_w.assign((size_t)SCAN_BINS * 4, 0.0f);
    t.scan_mask.assign(16, 0);
    t.scan_loc.assign((size_t)NMEL * 4, 0);
    std::vector<int> seg(NBINS, 0);
    for (int k = 0; k < NBINS; ++k) {
        const double fk = (double)sample_rate / 2.0 * k / (NBINS - 1);
        int j = 0;
        while (j < NMEL + 1 && mel_f[j + 1] <= fk) ++j;   // largest j with mel_f[j] <= fk (clamped to 80.. for fk >= fmax)
        seg[k] = j;
    }
    for (int k = 0; k < NBINS - 1 && t.scan_ok; ++k) {
        const int j = seg[k];
        for (int m = 0; m < NMEL; ++m)
            if (t.fb[(size_t)m * NBINS + k] != 0.0 && m != j - 1 && m != j) t.scan_ok = false;   // not a 2-tap triangular bank
        const double wa = (j >= 1 && j - 1 < NMEL) ? t.fb[(size_t)(j - 1) * NBINS + k] : 0.0;
        const double wb = (j < NMEL) ? t.fb[(size_t)j * NBINS + k] : 0.0;
        t.scan_w[k * 4 + 0] = t.scan_w[k * 4 + 1] = (float)(0.5 * wa);
        t.scan_w[k * 4 + 2] = t.scan_w[k * 4 + 3] = (float)(0.5 * wb);
    }
    std::vector<int> nloc(NMEL, 0);
    auto add_loc = [&](int band, int off_sn, int off_m) {
        if (band < 0 || band >= NMEL) return;
        if (nloc[band] >= 2) { t.scan_ok = false; return; }
        t.scan_loc[band * 4 + 2 * nloc[band] + 0] = off_sn;
        t.scan_loc[band * 4 + 2 * nloc[band] + 1] = off_m;
        ++nloc[band];
    };
    for (int p = 0; p < 16 && t.scan_ok; ++p) {
        const int k0 = POST_CHUNK * p;
        const int k1 = std::min(k0 + POST_CHUNK - 1, NBINS - 2);   // last bin of the chunk (<= 319)
        for (int k = k0 + 1; k <= k1; ++k) {
            if (seg[k] == seg[k - 1]) continue;
            if (seg[k] != seg[k - 1] + 1) { t.scan_ok = false; break; }   // empty segment
            // emission before bin k: A (band seg[k-1]-1) is written over bin k's own (already read) slots
            t.scan_mask[p] |= 1 << (k - k0);
            add_loc(seg[k - 1] - 1, 2 * k, 2 * (NFFT - k));
        }
        // chunk-end flush: A -> band seg[k1]-1, B -> band seg[k1]
        const int fl = FRAME_FLUSH_F + 6 * p;
        add_loc(seg[k1] - 1, fl + 0, fl + 4);
        add_loc(seg[k1], fl + 2, fl + 5);
    }
    for (int m = 0; m < NMEL && t.scan_ok; ++m) {
        if (nloc[m] == 0) { t.scan_ok = false; break; }
        for (int c = nloc[m]; c < 2; ++c) { t.scan_loc[m * 4 + 2 * c] = FRAME_ZERO_F; t.scan_loc[m * 4 + 2 * c + 1] = FRAME_ZERO_F + 2; }
    }

    // ---- F4 kernel scan tables: 8 chunks of CHUNK4 = 41 bins, emissions written densely ----
    // (constants restated from avse_fwd4_stages.cuh, which this plain-C++ file does not include)
    {
        constexpr int CH = 41, NCH = 8, FLUSH = 1284, ZERO4 = 1344;
        t.scan4_ok = t.scan_ok;
        t.scan4_w.assign((size_t)NCH * CH * 2, 0.0f);
        t.scan4_mask.assign(NCH * 2, 0u);
        t.scan4_loc.assign((size_t)NMEL * 4, -1);
        std::vector<int> n4(NMEL, 0);
        auto add4 = [&](int band, int off_sn, int off_m) {
            if (band < 0 || band >= NMEL) return;
            if (n4[band] >= 3) { t.scan4_ok = false; return; }
            t.scan4_loc[band * 4 + n4[band]] = off_sn | (off_m << 16);
            ++n4[band];
        };
        for (int k = 0; k < NBINS - 1 && t.scan4_ok; ++k) {
            const int j = seg[k];
            const double wa = (j >= 1 && j - 1 < NMEL) ? t.fb[(size_t)(j - 1) * NBINS + k] : 0.0;
            const double wb = (j < NMEL) ? t.fb[(size_t)j * NBINS + k] : 0.0;
            t.scan4_w[k * 2 + 0] = (float)(0.5 * wa);
            t.scan4_w[k * 2 + 1] = (float)(0.5 * wb);
        }
        for (int p = 0; p < NCH && t.scan4_ok; ++p) {
            const int k0 = CH * p;
            const int kl = std::min(k0 + CH - 1, NBINS - 2);   // last weighted bin of the chunk (<= 319)
            int e = 0;
            for (int k = k0 + 1; k <= kl; ++k) {
                if (seg[k] == seg[k - 1]) continue;
                if (seg[k] != seg[k - 1] + 1) { t.scan4_ok = false; break; }   // empty segment
                const int i = k - k0;
                t.scan4_mask[2 * p + (i >> 5)] |= 1u << (i & 31);
                add4(seg[k - 1] - 1, 2 * (k0 + e), 2 * NFFT + 1 - 2 * k0 - e);
                ++e;
            }
            const int fl = FLUSH + 6 * p;
            add4(seg[kl] - 1, fl + 0, fl + 4);
            add4(seg[kl], fl + 2, fl + 5);
        }
        for (int m = 0; m < NMEL && t.scan4_ok; ++m) {
            if (n4[m] == 0) t.scan4_ok = false;
            // no second partial sum: point it at the frame buffer's always-zero pad (floats 1344..1346) so that the dB stage adds it
            // without a divergent branch (every warp holds bands with and without one); a third one stays -1 (rare, warp-uniform skip)
            if (n4[m] == 1) t.scan4_loc[m * 4 + 1] = ZERO4 | ((ZERO4 + 2) << 16);
        }
    }

    // The I8 inverse is the only inverse of a specialised context: it needs the walk tables, and its float32 solve of
    // F F^T x = y drifts from pinv (dp:112) in proportion to cond(F F^T) (GRAM_COND_MAX).  Refused banks go to the generic kernels.
    if (!t.post_ok) { t.error = "filterbank columns do not form a walk (unsupported by the I8 inverse post stage)"; return false; }
    if (!(t.gram_cond <= GRAM_COND_MAX)) { t.error = "F F^T too ill-conditioned for the float32 tridiagonal solve"; return false; }
    return true;
}

}  // namespace avse
