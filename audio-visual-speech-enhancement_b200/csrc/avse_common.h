// Shared constants and host/device qualifiers for the B200 spectral front/back end.
//
// The path mirrors /root/reference/data_processor.py:35-139 at the reference's hard-coded
// geometry (dp:44-45, dp:83-89): 16 kHz / 25 fps -> n_fft = 640 (= 2^7 * 5), hop = 160,
// 321 bins, 80 Slaney mel bands, 200 ms slices = 20 spectrogram frames.
#pragma once

#include <cmath>

#if defined(__CUDACC__)
#define AVSE_HD __host__ __device__ __forceinline__
#define AVSE_HD_COLD __host__ __device__ __noinline__     // cold helpers: ONE copy, kept out of the hot instruction stream
#else
#define AVSE_HD inline
#define AVSE_HD_COLD inline
#endif

namespace avse {

constexpr int NFFT = 640;            // dp:44   int(16000 / 25)
constexpr int HOP = 160;             // dp:45   int(n_fft / 4)
constexpr int NBINS = NFFT / 2 + 1;  // 321
constexpr int NMEL = 80;             // dp:86
constexpr int SPSS = 20;             // dp:49   spectrogram frames per 200 ms slice
constexpr int HALF = NFFT / 2;       // reflect-pad width of librosa.stft(center=True)

// FFT-640 factorisation: n = 40*n1 + n2, k = k1 + 16*k2  (DFT-16, twiddle, DFT-40 = 5 x 8 PFA)
constexpr int N1 = 16;
constexpr int N2 = 40;

// One warp owns a group of 2 consecutive STFT frames (10.9 KB of shared memory per warp -> 16 warps / SM).
constexpr int FPG = 2;
// Shared-memory frame buffer: 16 rows (k1) x 84 floats (40 complex + 2 pad) + 16 floats skew.
constexpr int ROW_F = 84;
// Layout of one frame region (floats): [0, 1344) rows / natural-order Z (Z uses [0, 1282)),
// [1344, 1360) never written (kept zero: "null" partial sums), [1360, 1456) chunk-end partial sums
// of the fused post+mel scan (16 chunks x 6 floats).
constexpr int FRAME_ZERO_F = N1 * ROW_F;        // 1344
constexpr int FRAME_FLUSH_F = N1 * ROW_F + 16;  // 1360
constexpr int FRAME_F = FRAME_FLUSH_F + 96;     // 1456 floats, == 16 (mod 32), multiple of 4
constexpr int SCAN_BINS = 336;                  // 16 chunks x POST_CHUNK bins (bins >= 320 unused)
constexpr int MEL_STAGE_F = 3 * NMEL * FPG;  // raw mel sums [sig][band][frame], staged over frame buffer 0
constexpr int WARP_SMEM_F = FPG * FRAME_F;   // 2720 floats = 10880 B per warp
static_assert(MEL_STAGE_F <= FRAME_F, "mel staging must fit in one frame buffer");

// mel tables
constexpr int MEL_WMAX = 24;    // max bins per band supported (reference config: 23)
constexpr int MEL_WROW = 28;    // padded row stride of the weight table (16-byte rows, bank spread)
constexpr int MEL_ROUNDS = NMEL / 16;   // one round = 16 consecutive bands x 2 frames
constexpr int POST_CHUNK = 21;  // bins per lane in the pointwise post stage (16 lanes x 21 >= 321; odd: bank spread)

constexpr float AMIN = 1e-5f;   // librosa.amplitude_to_db amin (dp:94)
constexpr float TOP_DB = 80.0f; // librosa.amplitude_to_db top_db (dp:94)

// Work split of the persistent kernels: `total` work items (tiles / groups), in order, are cut into one contiguous range per warp
// of a grid of `blocks` x `warps`: total / (blocks * warps) items each, the remainder one apiece to the first warps in grid order.
// (Round 2 first used ceil(total / warps) per warp, which left the last SM of a 1 000 x 3 s forward launch without work: + 0.5 %.
// Spreading the remainder over the blocks first -- AVSE_SPLIT_BLOCKS_FIRST=1, at most one extra item per SM -- measured equal for
// the forward kernel and 0.6 % slower for the inverse: an SM whose eight warps all run one more item keeps them overlapped, a lone
// extra item at the end of 112 SMs runs alone.)
#if !defined(AVSE_SPLIT_BLOCKS_FIRST)
#define AVSE_SPLIT_BLOCKS_FIRST 0   // 1: the remainder is spread over the blocks first (A/B runs)
#endif
struct WarpSplit {
    long long base;    // items per warp
    int q, r;          // extras per block: q + (block < r)
    long long extras;  // total % (blocks * warps)
};
inline WarpSplit make_warp_split(long long total, long long blocks, int warps) {
    WarpSplit s;
    const long long nw = blocks * warps;
    s.base = total / nw;
    s.extras = total % nw;
    s.q = (int)(s.extras / blocks);
    s.r = (int)(s.extras % blocks);
    return s;
}
AVSE_HD void warp_split_range(const WarpSplit& s, int block, int warp, int warps, long long& first, long long& count) {
#if AVSE_SPLIT_BLOCKS_FIRST
    const int eb = s.q + (block < s.r ? 1 : 0);
    first = ((long long)block * warps + warp) * s.base + (long long)block * s.q + (block < s.r ? block : s.r) + (warp < eb ? warp : eb);
    count = s.base + (warp < eb ? 1 : 0);
#else
    const long long gw = (long long)block * warps + warp;
    first = gw * s.base + (gw < s.extras ? gw : s.extras);
    count = s.base + (gw < s.extras ? 1 : 0);
#endif
}

// ---------------------------------------------------------------------------------------------
// Pooled pairs (avse_mix_pooled): row b of a batch mixes speech clip speech_index[b] with noise clip noise_index[b] read from
// its sample noise_offset[b] on, n[i] = z[(off + i) mod Ln] for i < Ls -- dp:119-139 on (s, z rotated by off).  off = 0 is
// the reference's own "double until long enough, then truncate" rule (dp:125-128).
// ---------------------------------------------------------------------------------------------
struct PoolRows {
    const long long* speech_index;   // [B]; nullptr: identity rows (avse_forward / avse_snr_factor batches)
    const long long* noise_index;    // [B]
    const int* noise_offset;         // [B] or nullptr (0 for every row)
    const int* speech_len;           // [n_speech] clip lengths (clamped to [0, speech_stride])
    const int* noise_len;            // [n_noise]  clip lengths (clamped to [0, noise_stride])
    long long speech_stride, noise_stride, n_speech, n_noise;
    int* bad_row_flag;               // set to 1 by the statistics pass for every invalid row (caller zeroes it)
};

// One resolved row: element offsets of the two clips, their lengths and the noise phase.  An invalid row (an index out of
// range, or off outside [0, Ln) -- which includes every empty noise clip) comes back as the empty pair: both lengths 0,
// nothing is read, factor 0, every log-mel at the amin floor.
struct PoolRow {
    long long s_off, n_off;
    int ls, ln, off;
    bool ok;
};

AVSE_HD PoolRow pool_row(const PoolRows& p, int b) {
    PoolRow r;
    r.s_off = 0; r.n_off = 0; r.ls = 0; r.ln = 0; r.off = 0;
    const long long si = p.speech_index[b], ni = p.noise_index[b];
    r.ok = si >= 0 && si < p.n_speech && ni >= 0 && ni < p.n_noise;
    if (!r.ok) return r;
    long long ls = p.speech_len[si], ln = p.noise_len[ni];
    ls = ls < 0 ? 0 : (ls < p.speech_stride ? ls : p.speech_stride);
    ln = ln < 0 ? 0 : (ln < p.noise_stride ? ln : p.noise_stride);
    const int off = p.noise_offset ? p.noise_offset[b] : 0;
    r.ok = off >= 0 && off < ln;
    if (!r.ok) return r;
    r.s_off = si * p.speech_stride;
    r.n_off = ni * p.noise_stride;
    r.ls = (int)ls; r.ln = (int)ln; r.off = off;
    return r;
}

// Sums of the noise n[i] = z[(off + i) mod Ln], i < n, of one pair (the SNR statistics, dp:130), in one of two regimes:
//   Ln >= n: the window [off, off + n) of z, read directly as at most two contiguous ranges [off, off + len0) and [0, len1)
//            (a 60 s noise under a 3 s speech reads 3 s of it, not 60);
//   Ln <  n: one pass over the stored clip, sample j weighted q + (((j - off) mod Ln) < rem), n = q Ln + rem.
struct NoiseSpan {
    bool periodic;
    int len0, len1;   // window regime
    int q, rem;       // periodic regime
};

AVSE_HD NoiseSpan noise_span(int n, int Ln, int off) {
    NoiseSpan w;
    w.periodic = Ln < n;
    if (w.periodic) {
        w.q = n / Ln; w.rem = n - w.q * Ln; w.len0 = Ln; w.len1 = 0;
    } else {
        w.q = 0; w.rem = 0;
        w.len0 = Ln - off < n ? Ln - off : n;
        w.len1 = n - w.len0;
    }
    return w;
}

AVSE_HD int noise_weight(const NoiseSpan& w, int j, int Ln, int off) {    // periodic regime, 0 <= j, off < Ln
    int d = j - off;
    d += d < 0 ? Ln : 0;
    return w.q + (d < w.rem ? 1 : 0);
}

// The statistics pass's epilogue: from the float64 sums t = (sum s, sum s^2, sum n, sum n^2) over the n samples of a pair, the
// SNR factor f = sqrt(var_s / var_n) 10^(-snr/20) (dp:130, population variances) and the level equaliser g = sqrt(sum s^2 /
// sum n^2).  The forward kernels pack z = s + i g n into one complex FFT and apply f / g after it, so any g gives s + f n; g only
// conditions the float32 arithmetic.  Rounding of either channel leaks into the other in proportion to its RAW power, mean
// included (a DC offset goes through the window and the FFT like any other component), so g balances the raw powers, not the
// variances.  n == 0 (empty files) gives f = g = 0; a silent noise gives inf / nan for both, like numpy; a constant non-zero
// noise (var_n == 0) gives a finite g and a non-finite f.
struct SnrGains { float factor, equalizer; };
AVSE_HD SnrGains snr_gains(int n, const double (&t)[4], double snr_db) {
    SnrGains r;
    r.factor = 0.0f;
    r.equalizer = 0.0f;
    if (n > 0) {
        const double inv = 1.0 / (double)n;
        const double ms = t[0] * inv, mn = t[2] * inv;
        const double vs = t[1] * inv - ms * ms, vn = t[3] * inv - mn * mn;
        r.factor = (float)(sqrt(vs / vn) * pow(10.0, -snr_db / 20.0));
        r.equalizer = (float)sqrt(t[1] / t[3]);
    }
    return r;
}

#if defined(__CUDACC__)
// Cooperative copy of a constant table (N4 16-byte words, 16-byte aligned) from global memory into registers at kernel start.
// The persistent kernels fetch ALL their tables first and store them to shared memory afterwards: a rolled "load, store, next"
// loop pays one L2 / HBM round trip per iteration, and the four tables of the forward kernel took 13 of them (about 8 us of a
// 545 us launch; ncu attributed 1.5 % of the kernel's stall samples to those four source lines).
template <int N4, int THREADS>
struct TableRegs {
    static constexpr int K = (N4 + THREADS - 1) / THREADS;
    float4 v[K];
};
template <int N4, int THREADS>
__device__ __forceinline__ void table_fetch(const void* g, int tid, TableRegs<N4, THREADS>& r) {
#pragma unroll
    for (int k = 0; k < TableRegs<N4, THREADS>::K; ++k) {
        const int i = tid + k * THREADS;
        r.v[k] = i < N4 ? __ldg(reinterpret_cast<const float4*>(g) + i) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
}
template <int N4, int THREADS>
__device__ __forceinline__ void table_put(float* s, int tid, const TableRegs<N4, THREADS>& r) {     // bit copy (int tables too)
#pragma unroll
    for (int k = 0; k < TableRegs<N4, THREADS>::K; ++k) {
        const int i = tid + k * THREADS;
        if (i < N4) reinterpret_cast<float4*>(s)[i] = r.v[k];
    }
}
template <int N4, int THREADS>
__device__ __forceinline__ void table_put_scaled(float* s, int tid, const TableRegs<N4, THREADS>& r, float scale) {
#pragma unroll
    for (int k = 0; k < TableRegs<N4, THREADS>::K; ++k) {
        const int i = tid + k * THREADS;
        if (i < N4) reinterpret_cast<float4*>(s)[i] = make_float4(r.v[k].x * scale, r.v[k].y * scale, r.v[k].z * scale, r.v[k].w * scale);
    }
}
#endif

}  // namespace avse
