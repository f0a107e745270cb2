// Host emulation of pooled-pair mixing (avse_mix_pooled) for the CPU tests (TEST INFRASTRUCTURE, not a product path).
// Same approach as avse_emul.cpp: the kernels' __host__ __device__ warp-stage functions built with g++, one warp run as a loop
// over 32 lanes per stage.  Here a row is a speech clip plus a noise clip read from a phase (n[i] = z[(phase + i) mod Ln]),
// resolved exactly as the kernels resolve it, through the F4 kernel's TILED instantiation or the 2-frame kernel; and the
// statistics pass's noise sums through noise_span / noise_weight.
#include <vector>
#include <cstring>
#include <cmath>
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_common.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_tables.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_fwd_stages.cuh"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_fwd4_stages.cuh"

using namespace avse;

namespace {

// One emulated warp: its private shared-memory region plus the per-lane registers that live across
// a __syncwarp() in the kernel.
struct EmulWarp {
    alignas(16) float frames[WARP_SMEM_F];
    cpx x[32][40];
    float acc[32][MEL_ROUNDS][3];
};

static void emul_fft_stages(EmulWarp& w, const HostTables& h, const float* win2, const FwdTile& tl) {
    const vec2* s_tw = reinterpret_cast<const vec2*>(h.tw1t.data());
    for (int lane = 0; lane < 32; ++lane) stage_pass1(tl, lane, win2, s_tw, w.frames);
    for (int lane = 0; lane < 32; ++lane) pass2_compute(lane, w.frames, w.x[lane]);
    for (int lane = 0; lane < 32; ++lane) pass2_store(lane, w.frames, w.x[lane]);
}

// The 2-frame kernel's tile loop over one utterance whose tile fields (rows, lengths, gain, factor, period, phase) are set.
static int emul2_run(const HostTables& h, bool scan, FwdTile tl, int layout, int n_slices, int ld_t, float* out_sp, float* out_nz,
                     float* out_mix, float* max3) {
    static EmulWarp w;
    memset(w.frames, 0, sizeof(w.frames));
    const int T = tl.T, G = (T + FPG - 1) / FPG;
    const bool have_noise = tl.nz != nullptr;
    FwdOut out{};
    out.dst[0] = out_sp; out.dst[1] = out_nz; out.dst[2] = out_mix;
    out.layout = layout; out.n_slices = n_slices; out.ld_t = ld_t;
    float mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    std::vector<vec4> scanw(SCAN_BINS);
    for (int k = 0; k < SCAN_BINS; ++k) { scanw[k].x = h.scan_w[4 * k]; scanw[k].y = h.scan_w[4 * k + 1]; scanw[k].z = h.scan_w[4 * k + 2]; scanw[k].w = h.scan_w[4 * k + 3]; }
    std::vector<ivec4> loc(NMEL);
    for (int m = 0; m < NMEL; ++m) { loc[m].x = h.scan_loc[4 * m]; loc[m].y = h.scan_loc[4 * m + 1]; loc[m].z = h.scan_loc[4 * m + 2]; loc[m].w = h.scan_loc[4 * m + 3]; }
    for (int g = 0; g < G; ++g) {
        tl.t0 = g * FPG;
        emul_fft_stages(w, h, h.window2.data(), tl);
        if (scan) {
            for (int lane = 0; lane < 32; ++lane)
                stage_post_scan<false>(lane, tl.factor, scanw.data(), h.scan_mask.data(), w.frames, nullptr);
        } else {
            for (int lane = 0; lane < 32; ++lane) stage_post<false>(lane, tl.factor, w.frames, nullptr);
            for (int lane = 0; lane < 32; ++lane)
                stage_mel(lane, h.mel_roundw.data(), h.mel_w.data(), h.mel_lo.data(), w.frames, w.acc[lane]);
            for (int lane = 0; lane < 32; ++lane) stage_mel_store(lane, w.acc[lane], w.frames);
        }
        for (int q = 0; q < 3; ++q)
            for (int lane = 0; lane < 32; ++lane) {
                float lm[3] = {-INFINITY, -INFINITY, -INFINITY};
                if (scan) stage_db_scan(lane, q, tl.factor, have_noise, loc.data(), w.frames, out, tl.t0, T, lm);
                else stage_db(lane, q, tl.factor, have_noise, w.frames, out, tl.t0, T, lm);
                for (int s = 0; s < 3; ++s) if (lm[s] > mx[s]) mx[s] = lm[s];
            }
    }
    for (int s = 0; s < 3; ++s) max3[s] = key_to_float(float_to_key(mx[s]));
    return scan ? 1 : 0;
}


// ---- F4 kernel (avse_fwd4_stages.cuh): one emulated warp = four frames ----
struct EmulWarp4 {
    alignas(16) float frames[WARP4_SMEM_F];
    cpx x[32][40];
    float rs[32][RAW4], rn[32][RAW4], ts[32][16], tn[32][16];
    Lane4Const lc[32];
};

// The tile loop of the F4 kernel's TILED instantiation (which serves pooled rows) over one utterance whose tile fields are set:
// interior groups (a wrapped noise shifted into its period) or the per-sample edge loader, never the reflect-only edge groups.
static int emul4_run(const HostTables& h, FwdTile tl, int layout, int n_slices, int ld_t, float* out_sp, float* out_nz,
                     float* out_mix, float* max3) {
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
    out.layout = layout; out.n_slices = n_slices; out.ld_t = ld_t;
    float mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int g = 0; g < G; ++g) {
        tl.t0 = g * F4;
        int nz_shift = 0;
        if (group4_interior<float, true>(tl, nz_shift)) {
#if defined(AVSE_EMUL_P1_UNIFIED)
            for (int lane = 0; lane < 32; ++lane) {
                p4_load_raw(tl, nz_shift, lane, w.rs[lane], w.rn[lane]);
                p4_load_tail_raw(tl, nz_shift, lane, w.ts[lane], w.tn[lane]);
                stage4_pass1_unified(tl, lane, w.rs[lane], w.rn[lane], w.ts[lane], w.tn[lane], w.lc[lane], h.window.data(), s_tw, w.frames);
            }
#else
            for (int lane = 0; lane < 32; ++lane) {
                p4_load_raw(tl, nz_shift, lane, w.rs[lane], w.rn[lane]);
                stage4_pass1_main(tl, lane, w.rs[lane], w.rn[lane], w.lc[lane], w.frames);     // consumes (rescales / rotates) rs, rn
            }
            for (int lane = 0; lane < 32; ++lane) stage4_pass1_tail(tl, nz_shift, lane, h.window.data(), s_tw, w.frames);
#endif
        } else {
            for (int lane = 0; lane < 32; ++lane) stage4_pass1_edge<float, true>(tl, lane, h.window.data(), s_tw, w.frames);
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
#if AVSE_DB_SPLIT_LAST && AVSE_DB_BRANCHFREE_EXTRA
                if (q == 2) stage4_db_last(lane, tl.factor, loc.data(), w.frames, out, tl.t0, T, lm, ln);     // the kernel's form of the last 16 bands
                else
#endif
                stage4_db(lane, q, tl.factor, loc.data(), w.frames, out, tl.t0, T, lm, ln);
                for (int s = 0; s < 3; ++s) if (lm[s] > mx[s]) mx[s] = lm[s];
            }
    }
    for (int s = 0; s < 3; ++s) max3[s] = key_to_float(float_to_key(mx[s]));
    return 1;
}

}  // namespace

// ---- pooled pairs (avse_mix_pooled): one row = speech clip s [Ls] + noise clip z [Ln] read from its phase ----
// The row exactly as the kernels resolve it: the speech truncated / zero padded to L, the noise n[i] = z[(phase + i) mod Ln]
// for i < min(Ls, L) (a window that does not wrap is the contiguous row z + phase).  f2 = 1: the 2-frame kernel's stages,
// 0: the F4 kernel's TILED instantiation.  A phase outside [0, Ln) is an invalid row, processed as the empty pair like the kernels.
extern "C" int emul_forward_pool(const float* speech, int Ls, const float* noise, int Ln, int phase, int L, float factor, float gain,
                                 int n_slices, float* out_sp, float* out_nz, float* out_mix, float* mixed_pcm, float* max3,
                                 int sample_rate, double fmin, double fmax, int f2) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    if (!f2 && !h.scan4_ok) return -3;
    const bool ok = phase >= 0 && phase < Ln;
    FwdTile tl{};
    tl.sp = speech; tl.nz = noise; tl.L = L;
    tl.valid_s = ok ? (Ls < L ? Ls : L) : 0;
    tl.valid_n = tl.valid_s;
    tl.vmin = tl.valid_s;
    int period = ok ? Ln : 0, ph = ok ? phase : 0;
    fit_noise_row(tl.nz, period, ph, tl.valid_n);
    tl.period_n = period;
    tl.phase_n = ph;
    if (gain == 0.0f) gain = factor;
    tl.T = 1 + L / HOP; tl.gain = ok ? gain : 0.0f; tl.factor = (ok && gain != 0.0f) ? factor / gain : 0.0f;
    tl.mixed_pcm = mixed_pcm;
    if (f2) return emul2_run(h, h.scan_ok, tl, 0, n_slices, 0, out_sp, out_nz, out_mix, max3);
    return emul4_run(h, tl, 0, n_slices, 0, out_sp, out_nz, out_mix, max3);
}

// The statistics pass's noise sums (sum n, sum n^2 in float64) of n[i] = z[(off + i) mod Ln], i < n, through noise_span /
// noise_weight (avse_common.h) in the kernel's two regimes, in one thread's order.  Returns 1 for the periodic regime, 0 for
// the window regime.
extern "C" int emul_noise_sums(const float* z, int Ln, int n, int off, double* out2) {
    const NoiseSpan w = noise_span(n, Ln, off);
    double b0 = 0.0, b1 = 0.0;
    if (!w.periodic) {
        for (int i = 0; i < w.len0; ++i) { const double v = z[off + i]; b0 += v; b1 += v * v; }
        for (int i = 0; i < w.len1; ++i) { const double v = z[i]; b0 += v; b1 += v * v; }
    } else {
        for (int j = 0; j < Ln; ++j) { const double v = z[j], c = (double)noise_weight(w, j, Ln, off); b0 += c * v; b1 += c * v * v; }
    }
    out2[0] = b0;
    out2[1] = b1;
    return w.periodic ? 1 : 0;
}
