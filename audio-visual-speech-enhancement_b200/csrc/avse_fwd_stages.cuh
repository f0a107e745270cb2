// Warp-stage functions of the fused forward kernel (mix at SNR -> STFT -> mel -> dB).
//
// One warp owns a group of FPG = 2 consecutive STFT frames of one utterance and walks them
// through warp-synchronous stages that exchange data only through that warp's private
// shared-memory region (no block-level barrier anywhere in the frame loop):
//
//   pass 1  lane = (frame, n2):   coalesced strided loads of speech + noise, Hann, packed z = s + i*n
//                                  (one complex FFT carries both spectra), DFT-16 over n1, twiddle
//                                  W_640^{n2 k1}                          -> rows [k1][n2]
//   pass 2  lane = (frame, k1):   DFT-40 over n2 (5 x 8 PFA)              -> Z[k] natural order
//   scan    lane = (chunk, frame): unpack S' = Z_k + conj Z_{N-k}, N' = (Z_k - conj Z_{N-k})/i,
//                                  M' = S' + f N' (STFT linearity), three magnitudes in registers,
//                                  accumulated straight into running mel band sums
//   dB      lane = band:           20 log10(max(1e-5, .)), running max, stores in slice layout
//
// Complex data are (re, im) register pairs so the butterflies use Blackwell's packed FP32 instructions
// (avse_dft.cuh).  Reference semantics: /root/reference/data_processor.py:77-96 (signal_to_spectrogram),
// :130-133 (SNR mix), :35-57 (slice layout); librosa/mediaio semantics per SURVEY.md App. A.
//
// Every function is __host__ __device__: tests/emul builds the same code with g++ and runs a
// warp as a loop over 32 lanes per stage (the stage boundaries are the __syncwarp points).
#pragma once
#include "avse_common.h"
#include "avse_dft.cuh"

#if !defined(__CUDACC__)
#include <cmath>
#endif

// Tuning switch (measured on B200, profiles/README.md): unroll factor of the scan loop (21 bins).
#if !defined(AVSE_POST_UNROLL)
#define AVSE_POST_UNROLL 7
#endif
#define AVSE_STR_(x) #x
#define AVSE_UNROLL_N_(n) _Pragma(AVSE_STR_(unroll n))

namespace avse {

struct alignas(8) vec2 { float x, y; };
struct alignas(16) vec4 { float x, y, z, w; };
struct alignas(16) ivec4 { int x, y, z, w; };

AVSE_HD float fast_sqrt(float x) {
#if defined(__CUDA_ARCH__)
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#else
    return sqrtf(x);
#endif
}

AVSE_HD float fast_log2(float x) {
#if defined(__CUDA_ARCH__)
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));   // x >= 1e-5: never denormal
    return y;
#else
    return log2f(x);
#endif
}

AVSE_HD float amp_to_db(float a) {
    // librosa.amplitude_to_db with ref=1, amin=1e-5 before the top_db floor (dp:94)
    constexpr float K = 6.0205999132796239f;  // 20 / log2(10)
    return K * fast_log2(a > AMIN ? a : AMIN);
}

// Constant tables (device pointers; the kernel stages what it needs in shared memory).
struct FwdTables {
    const float* window;      // [640]
    const float* window2;     // [640][2]  (w, w) pairs
    const float* tw1t;        // [16][40][2]
    const float* mel_w;       // [80][MEL_WROW]      generic path
    const int* mel_lo;        // [80]                generic path
    const int* mel_roundw;    // [MEL_ROUNDS]        generic path
    const float* scan_w;      // [SCAN_BINS][4]      scan path: (wA, wA, wB, wB), 0.5 * weights
    const int* scan_mask;     // [16]                scan path: bit i of chunk p = "band finished before bin 21p+i"
    const int* scan_loc;      // [80][4]             scan path: partial-sum locations of each band
    const float* scan4_w;     // [328][2]            F4 kernel: (wa, wb)
    const unsigned* scan4_mask;   // [8][2]          F4 kernel: emission masks (lo, hi)
    const int* scan4_loc;     // [80][4]             F4 kernel: packed partial-sum offsets
};

// One group of FPG frames of one utterance.
// S: sample type in HBM (float, or short for raw int16 WAV samples, dp:122-123: the decode is fused into the loads)
template <typename S>
struct FwdTileT {
    const S* sp;         // speech samples of this utterance
    const S* nz;         // noise samples, may be nullptr; period_n > 0: only the first period_n are read (see below)
    int L;               // signal length after pad/truncate (dp:37-42); reflect domain
    int valid_s;         // samples present in sp (zeros beyond, dp:40)
    int valid_n;         // samples present in nz
    int vmin;            // min(valid_s, valid_n) (0 when nz == nullptr): interior test
    int T;               // STFT frames: 1 + L / hop
    int t0;              // first frame of the group (multiple of FPG)
    // The SNR factor f (dp:130) is applied in two parts, f = gain * factor: the noise is multiplied by `gain`
    // (= sqrt(sum s^2 / sum n^2), the level equaliser) as it is LOADED, so that the two channels of the packed FFT
    // z = s + i (gain n) carry equal raw power whatever the levels and DC offsets of the two files (float vs int16
    // scale ...): fp32 rounding of the louder channel would otherwise leak into the quieter one through the unpack
    // S' = Z_k + conj Z_{N-k}.  The residual `factor` = f / gain (10^(-snr/20) for zero-mean files) is applied
    // after the unpack by STFT linearity.
    float gain;          // applied to the noise samples at load; 0 when nz == nullptr
    float factor;        // residual applied to the (gain-scaled) noise spectrum / mel sums; 0 when nz == nullptr
    int period_n;        // dp:125-128: noise[i] = nz[(phase_n + i) mod period_n] (the reference doubles the noise until it covers
                         // the speech, then truncates: a periodic tiling; phase_n != 0 only for pooled pairs, avse_mix_pooled);
                         // 0: nz covers [0, valid_n) itself
    int phase_n;         // 0 <= phase_n < period_n; 0 when period_n == 0
    float* mixed_pcm;    // [L] or nullptr: s + f*n (dp:133), zero-padded / truncated to L
};
using FwdTile = FwdTileT<float>;

// The noise row of a pair, n[i] = nz[(phase + i) mod period] for i < valid_n: a window that does not wrap (phase + valid_n <=
// period, or no period at all) is the contiguous row nz + phase, read with no modulo anywhere (period = phase = 0 on return).
template <typename S>
AVSE_HD void fit_noise_row(const S*& nz, int& period, int& phase, int valid_n) {
    if (period <= 0 || phase + valid_n <= period) {
        if (nz != nullptr) nz += phase;
        period = 0;
        phase = 0;
    }
}

// Sample i of a periodically tiled noise (dp:125-128).  Out of line: the integer modulo is ~25 instructions and the edge
// loaders are unrolled 16 x, which would put 400 cold instructions into the middle of the kernel's instruction stream.
template <typename S>
AVSE_HD_COLD float load_sample_periodic(const S* p, int i, int period, int phase) { return (float)p[(i + phase) % period]; }

template <typename S>
AVSE_HD float load_sample_edge(const S* p, int i, int L, int valid, int period = 0, int phase = 0) {
    // np.pad(y, n_fft//2, mode='reflect') on the length-L (zero padded) signal
    i = i < 0 ? -i : i;
    i = i >= L ? 2 * (L - 1) - i : i;
    i = i < 0 ? 0 : i;
    if (p == nullptr || i >= valid) return 0.0f;
    return period > 0 ? load_sample_periodic(p, i, period, phase) : (float)p[i];
}

// A group is "interior" when both of its frames exist and all their samples are present in both
// signals without reflection or zero padding.
AVSE_HD bool group_interior(const FwdTile& tl) {
    return tl.nz != nullptr && tl.period_n == 0 && tl.t0 * HOP - HALF >= 0 && (tl.t0 + 1) * HOP + HALF <= tl.vmin && tl.t0 + 1 < tl.T;
}

// ---------------------------------------------------------------------------------------
// pass 1.  80 (frame, n2) columns per group over 32 lanes in three rounds:
//   round 0: (frame 0, n2 = lane)   round 1: (frame 1, n2 = lane)   round 2: lanes 0..15 take
//   (frame lane/8, n2 = 32 + lane%8).  One rolled copy of the column code (I-cache); every round
//   loads its own 16 strides per signal (the 12 shared with the previous round come from L1/L2).
// s_win2: [640] (w, w) pairs so the window multiply is one packed instruction per sample pair.
// ---------------------------------------------------------------------------------------
// DFT-16 over n1, twiddle W_640^{n2 k1}, store column n2 of frame f as rows [k1][n2].
AVSE_HD void pass1_column(cpx (&x)[16], int f, int n2, const vec2* s_tw, float* frames) {
    // issue the 15 twiddle loads before the DFT so their latency hides behind its arithmetic
    vec2 tw[16];
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) tw[k1] = s_tw[k1 * N2 + n2];
    dft16(x);
    float* row = frames + f * FRAME_F + 2 * n2;
    cstore(row, x[0]);
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) cstore(row + k1 * ROW_F, cmul(x[k1], tw[k1].x, tw[k1].y));
}

AVSE_HD void stage_pass1_interior(const FwdTile& tl, int lane, const float* s_win2, const vec2* s_tw, float* frames) {
#pragma unroll 1
    for (int round = 0; round < 3; ++round) {
        if (round == 2 && lane >= 16) break;
        const int f = round < 2 ? round : (lane >> 3) & 1;
        const int n2 = round < 2 ? lane : 32 + (lane & 7);
        const int o = (tl.t0 + f) * HOP - HALF + n2;
        const float* ps = tl.sp + o;
        const float* pn = tl.nz + o;
        cpx x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = cmake(ps[N2 * j], tl.gain * pn[N2 * j]);
        if (tl.mixed_pcm != nullptr) {
            // this frame's own hop: original samples [160 t, 160 t + 160) = strides n1 = 8..11
            float* pm = tl.mixed_pcm + o + HALF;
#pragma unroll
            for (int j = 0; j < 4; ++j) pm[N2 * j] = cre(x[8 + j]) + tl.factor * cim(x[8 + j]);
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = cmul_pp(x[j], cload(s_win2 + 2 * (N2 * j + n2)));
        pass1_column(x, f, n2, s_tw, frames);
    }
}

// Edge / generic path (first and last frames, short or zero-padded signals, single-signal mode):
// every sample goes through the reflect + zero-pad loader.  Cold code.
AVSE_HD void stage_pass1_edge(const FwdTile& tl, int lane, const float* s_win2, const vec2* s_tw, float* frames) {
#pragma unroll 1
    for (int round = 0; round < 3; ++round) {
        if (round == 2 && lane >= 16) break;
        const int f = round < 2 ? round : (lane >> 3) & 1;
        const int n2 = round < 2 ? lane : 32 + (lane & 7);
        const int t_raw = tl.t0 + f;
        const int t = t_raw < tl.T ? t_raw : tl.T - 1;   // frames past the end duplicate the last one (never stored)
        const int base = t * HOP - HALF + n2;
        cpx x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
            x[j] = cmake(load_sample_edge(tl.sp, base + N2 * j, tl.L, tl.valid_s),
                         tl.gain * load_sample_edge(tl.nz, base + N2 * j, tl.L, tl.valid_n, tl.period_n, tl.phase_n));
        if (tl.mixed_pcm != nullptr && t_raw < tl.T) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = t * HOP + N2 * j + n2;    // this frame's own hop: strides 8..11
                if (i < tl.L) tl.mixed_pcm[i] = cre(x[8 + j]) + tl.factor * cim(x[8 + j]);
            }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = cmul_pp(x[j], cload(s_win2 + 2 * (N2 * j + n2)));
        pass1_column(x, f, n2, s_tw, frames);
    }
}

AVSE_HD void stage_pass1(const FwdTile& tl, int lane, const float* s_win2, const vec2* s_tw, float* frames) {
    if (group_interior(tl)) stage_pass1_interior(tl, lane, s_win2, s_tw, frames);
    else stage_pass1_edge(tl, lane, s_win2, s_tw, frames);
}

// ---------------------------------------------------------------------------------------
// pass 2: lane = (f = lane/16, k1 = lane%16): load row, in-place DFT-40; after a warp sync the
// results are stored in natural order Z[k1 + 16 k2] over the same frame buffer.
// ---------------------------------------------------------------------------------------
AVSE_HD void pass2_load(int lane, const float* frames, cpx (&x)[40]) {
    const int f = lane >> 4, k1 = lane & 15;
    const float* row = frames + f * FRAME_F + k1 * ROW_F;
#pragma unroll
    for (int q = 0; q < 20; ++q) cload2(row + 4 * q, x[2 * q], x[2 * q + 1]);
}

AVSE_HD void pass2_compute(int lane, const float* frames, cpx (&x)[40]) {
    pass2_load(lane, frames, x);
    dft40_inplace(x);
}

AVSE_HD void pass2_store(int lane, float* frames, const cpx (&x)[40]) {
    const int f = lane >> 4, k1 = lane & 15;
    float* z = frames + f * FRAME_F + 2 * k1;
#pragma unroll
    for (int c = 0; c < 5; ++c)
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            const int idx = (8 * c + 5 * d) % 40;     // register holding output (c, d)
            const int k2 = (16 * c + 25 * d) % 40;    // its frequency index within the DFT-40
            cstore(z + 2 * N1 * k2, x[idx]);          // Z[k1 + 16 k2]
        }
}

// ---------------------------------------------------------------------------------------
// Fused post + mel "scan" (used when HostTables::scan_ok): lane = (chunk p = lane/2, frame f = lane%2)
// walks its 21 bins in order, unpacks the three magnitudes in registers and accumulates them straight
// into two running band sums: A = band seg-1 (falling edge), B = band seg (rising edge).  When the
// segment index advances (bit i of the chunk's mask), A is complete for this lane: it is written over
// the bin's own, already consumed, slots and the accumulators rotate.  The two sums left at the end of
// the chunk go to the frame's flush area.  The magnitudes never touch shared memory.  Bins whose weights
// are zero (0, >= 320) are walked like any other (finite garbage times exact zero).
// s_scan: [SCAN_BINS] (wA, wA, wB, wB); s_mask: [16].
// STFT: also emit X_speech[k] (dp:79 D) to stft_row[0..320]  (cold variant).
// ---------------------------------------------------------------------------------------
template <bool STFT>
AVSE_HD void stage_post_scan(int lane, float factor, const vec4* s_scan, const int* s_mask, float* frames, vec2* stft_row) {
    const int f = lane & 1, p = lane >> 1;
    float* fr = frames + f * FRAME_F;
    float* za = fr + 2 * POST_CHUNK * p;            // slot k      = za + 2 i
    float* zc = fr + 2 * (NFFT - POST_CHUNK * p);   // slot 640-k  = zc - 2 i
    const vec4* tab = s_scan + POST_CHUNK * p;
    const int mask = s_mask[p];
    if (STFT && stft_row != nullptr && p == 15) {
        vec2 d; d.x = za[2 * ((NBINS - 1) - 15 * POST_CHUNK)]; d.y = 0.0f;   // Nyquist bin 320 (real for real input)
        stft_row[NBINS - 1] = d;
    }
    cpx Asn = cmake(0.0f, 0.0f), Bsn = cmake(0.0f, 0.0f);   // (speech, noise) sums of bands seg-1 / seg
    float Am = 0.0f, Bm = 0.0f;                             // mixture sums
    const cpx zero = cmake(0.0f, 0.0f);
    AVSE_UNROLL_N_(AVSE_POST_UNROLL)
    for (int i = 0; i < POST_CHUNK; ++i) {
        const cpx a = cload(za + 2 * i);
        const cpx c = cload(zc - 2 * i);
        cpx wa, wb;
        cload2(reinterpret_cast<const float*>(tab + i), wa, wb);
        const bool emit = (mask >> i) & 1;
        if (emit) {
            cstore(za + 2 * i, Asn);
            cstore(zc - 2 * i, cmake(Am, 0.0f));
        }
        const cpx s = cfma_pp(c, cmake(1.0f, -1.0f), a);                 // 2 X_speech[k] = Z_k + conj Z_{N-k}
        const cpx n = cmake(cim(a) + cim(c), cre(c) - cre(a));           // 2 X_noise[k]  = (Z_k - conj Z_{N-k}) / i
        const cpx m = cfma_s(n, factor, s);                              // 2 X_mixed[k]
        const float ms = fast_sqrt(cre(s) * cre(s) + cim(s) * cim(s));
        const float mn = fast_sqrt(cre(n) * cre(n) + cim(n) * cim(n));
        const float mm = fast_sqrt(cre(m) * cre(m) + cim(m) * cim(m));
        const cpx msn = cmake(ms, mn);
        const cpx a_sel = emit ? Bsn : Asn, b_sel = emit ? zero : Bsn;
        const float am_sel = emit ? Bm : Am, bm_sel = emit ? 0.0f : Bm;
        Asn = cfma_pp(msn, wa, a_sel);
        Bsn = cfma_pp(msn, wb, b_sel);
        Am = am_sel + cre(wa) * mm;
        Bm = bm_sel + cre(wb) * mm;
        if (STFT && stft_row != nullptr) {
            const int k = POST_CHUNK * p + i;
            if (k < NBINS - 1) {
                vec2 d;
                if (k == 0) { d.x = cre(a); d.y = 0.0f; }    // DC bin (real for real input)
                else { d.x = 0.5f * cre(s); d.y = 0.5f * cim(s); }
                stft_row[k] = d;
            }
        }
    }
    float* fl = fr + FRAME_FLUSH_F + 6 * p;
    cstore(fl + 0, Asn);
    cstore(fl + 2, Bsn);
    cstore(fl + 4, cmake(Am, Bm));
}

// output description shared by the dB stages
struct FwdOut {
    float* dst[3];    // base of this utterance's output per signal (nullptr: skip stores)
    int layout;       // 0: slices [ns][80][20], 1: spectrogram [80][ld_t]
    int n_slices;     // slices kept (dp:164: min(video, audio))
    int ld_t;         // leading dimension for layout 1
};

AVSE_HD float neg_inf() {
#if defined(__CUDA_ARCH__)
    return __int_as_float(0xff800000);
#else
    return -INFINITY;
#endif
}

// dB, max and store of one band's three signals for the group's two frames (mel[sig][frame]).
// Slices [n_slices][80][20] (dp:49-57) or spectrogram [80][ld_t]; mx[sig]: 0 speech, 1 noise, 2 mixture.
AVSE_HD void db_emit(int m, const float (&mel)[3][2], bool have_noise, const FwdOut& out, int t0, int T, float (&mx)[3]) {
    const bool v1 = t0 + 1 < T;    // frame t0 itself is always < T
    int off;                       // element offset of (band m, frame t0) inside this utterance's output
    bool store = true;
    if (out.layout == 0) {
        const int sl = t0 / SPSS, tt = t0 - sl * SPSS;   // 2 | t0 and 2 | 20: a group never straddles slices
        off = (sl * NMEL + m) * SPSS + tt;
        store = sl < out.n_slices;
    } else {
        off = m * out.ld_t + t0;
    }
#pragma unroll
    for (int sig = 0; sig < 3; ++sig) {
        if (sig > 0 && !have_noise) break;
        const float d0 = amp_to_db(mel[sig][0]);
        const float d1 = amp_to_db(mel[sig][1]);
        const float lm = (v1 && d1 > d0) ? d1 : d0;
        mx[sig] = lm > mx[sig] ? lm : mx[sig];
        float* dst = out.dst[sig];
        if (dst != nullptr && store) {
            if (v1 && !(off & 1)) {
                vec2 o; o.x = d0; o.y = d1;
                *reinterpret_cast<vec2*>(dst + off) = o;    // 8-byte aligned
            } else {
                dst[off] = d0;
                if (v1) dst[off + 1] = d1;
            }
        }
    }
}

// dB stage of the scan path: lane = band m = 32 q + lane; each band's mel sum is the sum of its two
// partial-sum locations (s_loc[m] = frame-relative offsets SN0, M0, SN1, M1; absent parts point at zeros).
AVSE_HD void stage_db_scan(int lane, int q, float factor, bool have_noise, const ivec4* s_loc, const float* frames,
                           const FwdOut& out, int t0, int T, float (&mx)[3]) {
    const int m = 32 * q + lane;
    if (m >= NMEL) return;
    const ivec4 loc = s_loc[m];
    float mel[3][2];
#pragma unroll
    for (int f = 0; f < 2; ++f) {
        const float* fr = frames + f * FRAME_F;
        const vec2 sn0 = *reinterpret_cast<const vec2*>(fr + loc.x);
        const vec2 sn1 = *reinterpret_cast<const vec2*>(fr + loc.z);
        mel[0][f] = sn0.x + sn1.x;
        mel[1][f] = (sn0.y + sn1.y) * factor;
        mel[2][f] = fr[loc.y] + fr[loc.w];
    }
    db_emit(m, mel, have_noise, out, t0, T, mx);
}

// ---------------------------------------------------------------------------------------
// Generic path (any filterbank whose bands are contiguous and <= MEL_WMAX wide): magnitudes are
// written in place (slot k <- (|S'|, |N'|), slot 640-k <- (|M'|, 0)), then gathered band by band.
// ---------------------------------------------------------------------------------------
template <bool STFT>
AVSE_HD void stage_post(int lane, float factor, float* frames, vec2* stft_row) {
    const int f = lane >> 4, p = lane & 15;
    float* za = frames + f * FRAME_F + 2 * POST_CHUNK * p;
    float* zc = frames + f * FRAME_F + 2 * (NFFT - POST_CHUNK * p);
    const bool last = p == 15;
    constexpr int LAST_N = (NBINS - 1) - 15 * POST_CHUNK;              // 5 bins in the last chunk
    if (STFT && stft_row != nullptr && last) {
        vec2 d; d.x = za[2 * LAST_N]; d.y = 0.0f;
        stft_row[NBINS - 1] = d;
    }
#pragma unroll 3
    for (int i = 0; i < POST_CHUNK; ++i) {
        if (i >= LAST_N && last) continue;      // slots >= 320 hold other bins' |M'|: must not be overwritten
        const cpx a = cload(za + 2 * i);
        const cpx c = cload(zc - 2 * i);
        const cpx s = cfma_pp(c, cmake(1.0f, -1.0f), a);
        const cpx n = cmake(cim(a) + cim(c), cre(c) - cre(a));
        const cpx m = cfma_s(n, factor, s);
        const float ms = fast_sqrt(cre(s) * cre(s) + cim(s) * cim(s));
        const float mn = fast_sqrt(cre(n) * cre(n) + cim(n) * cim(n));
        const float mm = fast_sqrt(cre(m) * cre(m) + cim(m) * cim(m));
        cstore(za + 2 * i, cmake(ms, mn));
        cstore(zc - 2 * i, cmake(mm, 0.0f));
        if (STFT && stft_row != nullptr) {
            vec2 d;
            if (i == 0 && p == 0) { d.x = cre(a); d.y = 0.0f; }
            else { d.x = 0.5f * cre(s); d.y = 0.5f * cim(s); }
            stft_row[POST_CHUNK * p + i] = d;
        }
    }
}

// mel round r: lane = (f = lane/16, band m = 16r + lane%16), roundw = max band width of the round
AVSE_HD void mel_round_generic(int lane, int r, int roundw, const float* s_melw, const int* s_mello, const float* frames,
                               float& as, float& an, float& am) {
    const int f = lane >> 4, m = 16 * r + (lane & 15);
    const int lo = s_mello[m];
    const float* wrow = s_melw + m * MEL_WROW;
    const float* zs = frames + f * FRAME_F + 2 * lo;
    const float* zm = frames + f * FRAME_F + 2 * (NFFT - lo);
    as = 0.0f; an = 0.0f; am = 0.0f;
#pragma unroll 1
    for (int j = 0; j < roundw; ++j) {
        const float w = wrow[j];
        const vec2 sn = *reinterpret_cast<const vec2*>(zs + 2 * j);
        const float mm = zm[-2 * j];
        as += w * sn.x;
        an += w * sn.y;
        am += w * mm;
    }
}

// All rounds; results stay in registers until every lane has finished reading the frame buffers, then
// stage_mel_store writes them over frame buffer 0: melst[(sig * 80 + band) * 2 + frame].
AVSE_HD void stage_mel(int lane, const int* roundw, const float* s_melw, const int* s_mello, const float* frames,
                       float (&acc)[MEL_ROUNDS][3]) {
#pragma unroll
    for (int r = 0; r < MEL_ROUNDS; ++r)
        mel_round_generic(lane, r, roundw[r], s_melw, s_mello, frames, acc[r][0], acc[r][1], acc[r][2]);
}

AVSE_HD void stage_mel_store(int lane, const float (&acc)[MEL_ROUNDS][3], float* melst) {
    const int f = lane >> 4;
#pragma unroll
    for (int r = 0; r < MEL_ROUNDS; ++r) {
        const int m = 16 * r + (lane & 15);
        melst[(0 * NMEL + m) * FPG + f] = acc[r][0];   // speech
        melst[(1 * NMEL + m) * FPG + f] = acc[r][1];   // noise (unscaled)
        melst[(2 * NMEL + m) * FPG + f] = acc[r][2];   // mixture
    }
}

AVSE_HD void stage_db(int lane, int q, float factor, bool have_noise, const float* melst, const FwdOut& out, int t0, int T,
                      float (&mx)[3]) {
    const int m = 32 * q + lane;
    if (m >= NMEL) return;
    float mel[3][2];
#pragma unroll
    for (int sig = 0; sig < 3; ++sig) {
        const vec2 v = *reinterpret_cast<const vec2*>(melst + (sig * NMEL + m) * FPG);
        const float scale = sig == 1 ? factor : 1.0f;
        mel[sig][0] = v.x * scale;
        mel[sig][1] = v.y * scale;
    }
    db_emit(m, mel, have_noise, out, t0, T, mx);
}

// order-preserving float <-> int key for atomicMax on floats of either sign
AVSE_HD int float_to_key(float x) {
#if defined(__CUDA_ARCH__)
    const int b = __float_as_int(x);
#else
    int b; { union { float f; int i; } u; u.f = x; b = u.i; }
#endif
    return b >= 0 ? b : (b ^ 0x7fffffff);
}
AVSE_HD float key_to_float(int k) {
    const int b = k >= 0 ? k : (k ^ 0x7fffffff);
#if defined(__CUDA_ARCH__)
    return __int_as_float(b);
#else
    union { float f; int i; } u; u.i = b; return u.f;
#endif
}

}  // namespace avse
