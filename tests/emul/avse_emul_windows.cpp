// Host emulation of windowed pooled rows (avse_mix_pooled with speech_start) for the CPU tests (TEST INFRASTRUCTURE, not a
// product path).  Same approach as avse_emul_pool.cpp: the kernels' __host__ __device__ code built with g++, one warp run as a
// loop over 32 lanes per stage.  What this file adds is the row resolution itself: every row goes through pool_row
// (avse_common.h) exactly as the statistics pass, the F4 kernel's TILED loader and the 2-frame kernel resolve it, so the
// window's first sample and length come from the one place the kernels take them from.
#include <vector>
#include <cstring>
#include <cmath>
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_common.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_tables.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_fwd_stages.cuh"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_fwd4_stages.cuh"

using namespace avse;

namespace {

struct EmulWarp {
    alignas(16) float frames[WARP_SMEM_F];
    cpx x[32][40];
    float acc[32][MEL_ROUNDS][3];
};

// The 2-frame kernel's tile loop over one utterance (float samples only, like the kernel).
static void emul2_run(const HostTables& h, FwdTile tl, int n_slices, float* out_sp, float* out_nz, float* out_mix, float* max3) {
    static EmulWarp w;
    memset(w.frames, 0, sizeof(w.frames));
    const int T = tl.T, G = (T + FPG - 1) / FPG;
    FwdOut out{};
    out.dst[0] = out_sp; out.dst[1] = out_nz; out.dst[2] = out_mix;
    out.layout = 0; out.n_slices = n_slices; out.ld_t = 0;
    float mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    std::vector<vec4> scanw(SCAN_BINS);
    for (int k = 0; k < SCAN_BINS; ++k) { scanw[k].x = h.scan_w[4 * k]; scanw[k].y = h.scan_w[4 * k + 1]; scanw[k].z = h.scan_w[4 * k + 2]; scanw[k].w = h.scan_w[4 * k + 3]; }
    std::vector<ivec4> loc(NMEL);
    for (int m = 0; m < NMEL; ++m) { loc[m].x = h.scan_loc[4 * m]; loc[m].y = h.scan_loc[4 * m + 1]; loc[m].z = h.scan_loc[4 * m + 2]; loc[m].w = h.scan_loc[4 * m + 3]; }
    const vec2* s_tw = reinterpret_cast<const vec2*>(h.tw1t.data());
    for (int g = 0; g < G; ++g) {
        tl.t0 = g * FPG;
        for (int lane = 0; lane < 32; ++lane) stage_pass1(tl, lane, h.window2.data(), s_tw, w.frames);
        for (int lane = 0; lane < 32; ++lane) pass2_compute(lane, w.frames, w.x[lane]);
        for (int lane = 0; lane < 32; ++lane) pass2_store(lane, w.frames, w.x[lane]);
        for (int lane = 0; lane < 32; ++lane) stage_post_scan<false>(lane, tl.factor, scanw.data(), h.scan_mask.data(), w.frames, nullptr);
        for (int q = 0; q < 3; ++q)
            for (int lane = 0; lane < 32; ++lane) {
                float lm[3] = {-INFINITY, -INFINITY, -INFINITY};
                stage_db_scan(lane, q, tl.factor, true, loc.data(), w.frames, out, tl.t0, T, lm);
                for (int s = 0; s < 3; ++s) if (lm[s] > mx[s]) mx[s] = lm[s];
            }
    }
    for (int s = 0; s < 3; ++s) max3[s] = key_to_float(float_to_key(mx[s]));
}

struct EmulWarp4 {
    alignas(16) float frames[WARP4_SMEM_F];
    cpx x[32][40];
    float rs[32][RAW4], rn[32][RAW4];
    Lane4Const lc[32];
};

// The F4 kernel's TILED instantiation (which serves pooled rows) over one utterance, for float or int16 samples.
template <typename S>
static void emul4_run(const HostTables& h, FwdTileT<S> tl, int n_slices, float* out_sp, float* out_nz, float* out_mix, float* max3) {
    static EmulWarp4 w;
    memset(w.frames, 0, sizeof(w.frames));
    const int T = tl.T, G = (T + F4 - 1) / F4;
    const vec2* s_tw = reinterpret_cast<const vec2*>(h.tw1t.data());
    const vec2* s_scanw = reinterpret_cast<const vec2*>(h.scan4_w.data());
    std::vector<ivec4> loc(NMEL);
    for (int m = 0; m < NMEL; ++m) { loc[m].x = h.scan4_loc[4 * m]; loc[m].y = h.scan4_loc[4 * m + 1]; loc[m].z = h.scan4_loc[4 * m + 2]; loc[m].w = h.scan4_loc[4 * m + 3]; }
    for (int lane = 0; lane < 32; ++lane) lane4_const_init(lane, h.window.data(), s_tw, w.lc[lane]);
    FwdOut out{};
    out.dst[0] = out_sp; out.dst[1] = out_nz; out.dst[2] = out_mix;
    out.layout = 0; out.n_slices = n_slices; out.ld_t = 0;
    float mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int g = 0; g < G; ++g) {
        tl.t0 = g * F4;
        int nz_shift = 0;
        if (group4_interior<S, true>(tl, nz_shift)) {
            for (int lane = 0; lane < 32; ++lane) {
                p4_load_raw(tl, nz_shift, lane, w.rs[lane], w.rn[lane]);
                stage4_pass1_main(tl, lane, w.rs[lane], w.rn[lane], w.lc[lane], w.frames);
            }
            for (int lane = 0; lane < 32; ++lane) stage4_pass1_tail(tl, nz_shift, lane, h.window.data(), s_tw, w.frames);
        } else {
            for (int lane = 0; lane < 32; ++lane) stage4_pass1_edge<S, true>(tl, lane, h.window.data(), s_tw, w.frames);
        }
        for (int r = 0; r < 2; ++r) {
            for (int lane = 0; lane < 32; ++lane) p4_pass2_compute(lane, r, w.frames, w.x[lane]);
            for (int lane = 0; lane < 32; ++lane) p4_pass2_store(lane, r, w.frames, w.x[lane]);
        }
        for (int lane = 0; lane < 32; ++lane)
            stage4_scan(lane, tl.factor, s_scanw, h.scan4_mask[2 * (lane & 7)], h.scan4_mask[2 * (lane & 7) + 1], w.frames);
        for (int q = 0; q < 3; ++q)
            for (int lane = 0; lane < 32; ++lane) {
                float lm[3] = {-INFINITY, -INFINITY, -INFINITY};
                float ln[96]; for (int i = 0; i < 96; ++i) ln[i] = INFINITY;
                if (q == 2) stage4_db_last(lane, tl.factor, loc.data(), w.frames, out, tl.t0, T, lm, ln);
                else stage4_db(lane, q, tl.factor, loc.data(), w.frames, out, tl.t0, T, lm, ln);
                for (int s = 0; s < 3; ++s) if (lm[s] > mx[s]) mx[s] = lm[s];
            }
    }
    for (int s = 0; s < 3; ++s) max3[s] = key_to_float(float_to_key(mx[s]));
}

// The statistics pass of one resolved row in one thread's order: the speech window s[0, ls) and the noise n[i] = z[(off + i)
// mod ln], i < ls, through noise_span / noise_weight.
template <typename S>
static void emul_row_sums(const S* s, int n, const S* z, int ln, int off, double (&t)[4]) {
    t[0] = t[1] = t[2] = t[3] = 0.0;
    for (int i = 0; i < n; ++i) { const double v = (double)s[i]; t[0] += v; t[1] += v * v; }
    if (n <= 0) return;
    const NoiseSpan w = noise_span(n, ln, off);
    if (!w.periodic) {
        for (int i = 0; i < w.len0; ++i) { const double v = (double)z[off + i]; t[2] += v; t[3] += v * v; }
        for (int i = 0; i < w.len1; ++i) { const double v = (double)z[i]; t[2] += v; t[3] += v * v; }
    } else {
        for (int j = 0; j < ln; ++j) { const double v = (double)z[j], c = (double)noise_weight(w, j, ln, off); t[2] += c * v; t[3] += c * v * v; }
    }
}

template <typename S>
static int emul_row(const S* speech_pool, const int* speech_len, long long n_speech, long long speech_stride, const S* noise_pool,
                    const int* noise_len, long long n_noise, long long noise_stride, long long si, long long ni, int off, const int* start,
                    int L, double snr_db, int n_slices, float* out_sp, float* out_nz, float* out_mix, float* mixed_pcm, float* max3,
                    double* sums4, float* gains2, int f2, const HostTables& h) {
    PoolRows p{};
    p.speech_index = &si; p.noise_index = &ni; p.noise_offset = &off;
    p.speech_len = speech_len; p.noise_len = noise_len;
    p.speech_stride = speech_stride; p.noise_stride = noise_stride; p.n_speech = n_speech; p.n_noise = n_noise;
    p.speech_start = start; p.L = L;
    const PoolRow r = pool_row(p, 0);
    // statistics pass (avse_snr_factor_kernel's pooled branch): the row's window, its noise from its phase
    const S* s = speech_pool + r.s_off;
    const S* z = noise_pool + r.n_off;
    double t[4];
    emul_row_sums(s, r.ls, z, r.ln, r.off, t);
    for (int i = 0; i < 4; ++i) sums4[i] = t[i];
    const SnrGains g = snr_gains(r.ls, t, snr_db);
    gains2[0] = g.factor; gains2[1] = g.equalizer;
    // forward pass (the F4 kernel's / 2-frame kernel's pooled branch)
    FwdTileT<S> tl{};
    tl.sp = s; tl.nz = z; tl.L = L;
    tl.valid_s = r.ls < L ? r.ls : L;
    tl.valid_n = tl.valid_s;
    tl.vmin = tl.valid_s;
    int period = r.ln, phase = r.off;
    fit_noise_row(tl.nz, period, phase, tl.valid_n);
    tl.period_n = period;
    tl.phase_n = phase;
    tl.T = 1 + L / HOP;
    tl.gain = g.equalizer;
    tl.factor = g.equalizer != 0.0f ? g.factor / g.equalizer : 0.0f;
    tl.mixed_pcm = mixed_pcm;
    if (f2) {
        if constexpr (sizeof(S) == sizeof(float)) emul2_run(h, tl, n_slices, out_sp, out_nz, out_mix, max3);
        else return -4;
    } else {
        emul4_run<S>(h, tl, n_slices, out_sp, out_nz, out_mix, max3);
    }
    return r.ok ? 1 : 0;
}

}  // namespace

// One pooled row b = 0 of avse_mix_pooled on the reference context (16 kHz, fmin 0, fmax 8000): speech clip si of the pool
// [n_speech][speech_stride] (fmt 0: float32, 1: int16), noise clip ni read from `off`, speech window from *start (start NULL:
// the whole clip).  Writes the un-floored slices, the PCM, the dB maxima, the statistics sums (sum s, sum s^2, sum n, sum n^2)
// and (factor, equalizer).  Returns 1 for a valid row, 0 for an invalid one (processed as the empty pair), < 0 on error.
extern "C" int emul_window_row(const void* speech_pool, int fmt, const int* speech_len, long long n_speech, long long speech_stride,
                               const void* noise_pool, const int* noise_len, long long n_noise, long long noise_stride, long long si,
                               long long ni, int off, const int* start, int L, double snr_db, int n_slices, float* out_sp, float* out_nz,
                               float* out_mix, float* mixed_pcm, float* max3, double* sums4, float* gains2, int f2) {
    static HostTables h;
    static bool built = false;
    if (!built) {
        if (!build_tables(h, 16000, 0.0, 8000.0) || !h.scan4_ok || !h.scan_ok) return -2;
        built = true;
    }
    if (fmt == 0)
        return emul_row<float>((const float*)speech_pool, speech_len, n_speech, speech_stride, (const float*)noise_pool, noise_len, n_noise,
                               noise_stride, si, ni, off, start, L, snr_db, n_slices, out_sp, out_nz, out_mix, mixed_pcm, max3, sums4, gains2, f2, h);
    return emul_row<short>((const short*)speech_pool, speech_len, n_speech, speech_stride, (const short*)noise_pool, noise_len, n_noise,
                           noise_stride, si, ni, off, start, L, snr_db, n_slices, out_sp, out_nz, out_mix, mixed_pcm, max3, sums4, gains2, f2, h);
}
