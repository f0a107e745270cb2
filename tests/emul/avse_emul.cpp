// Host emulation of the forward kernel's warp stages (TEST INFRASTRUCTURE, not a product path).
// Builds the SAME __host__ __device__ stage functions with g++ and runs one warp as a loop over
// 32 lanes per stage; the loop boundaries are exactly the kernel's __syncwarp() points.  This
// lets the CPU-only test suite check the index maps, twiddles, tables and float32 arithmetic of
// csrc/avse_fwd_stages.cuh against the float64 oracle without a GPU.
#include <vector>
#include <cstring>
#include <cmath>
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_common.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_tables.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_fwd_stages.cuh"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_fwd4_stages.cuh"

using namespace avse;

extern "C" int emul_filterbank(int sample_rate, double fmin, double fmax, double* fb_out) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    memcpy(fb_out, h.fb.data(), sizeof(double) * NMEL * NBINS);
    return 0;
}

extern "C" int emul_tables_info(int sample_rate, double fmin, double fmax, int* lo, int* width, float* tri /*3*80*/) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    memcpy(lo, h.mel_lo.data(), sizeof(int) * NMEL);
    memcpy(width, h.mel_width.data(), sizeof(int) * NMEL);
    memcpy(tri, h.tri_w.data(), sizeof(float) * NMEL);
    memcpy(tri + NMEL, h.tri_ipiv.data(), sizeof(float) * NMEL);
    memcpy(tri + 2 * NMEL, h.tri_sup.data(), sizeof(float) * NMEL);
    return 0;
}

// build_tables' verdict (0 accepted, -2 refused) and out = (scan4_ok, scan_ok, post_ok); cond (may be NULL) = gram_cond.
// The flags and cond are those computed before the verdict; they are meaningful for a bank refused for post_ok or conditioning.
extern "C" int emul_table_flags(int sample_rate, double fmin, double fmax, int* out, double* cond) {
    HostTables h;
    const bool ok = build_tables(h, sample_rate, fmin, fmax);
    out[0] = h.scan4_ok; out[1] = h.scan_ok; out[2] = h.post_ok;
    if (cond) *cond = h.gram_cond;
    return ok ? 0 : -2;
}

// The inverse tables of an accepted bank: post_w [328][2], post_mask [8][4], tri (w, 1/pivot, sup) [3][80], spike [4][SPIKE_ROW].
extern "C" int emul_inverse_tables(int sample_rate, double fmin, double fmax, float* post_w, unsigned* post_mask, float* tri, float* spike) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    memcpy(post_w, h.post_w.data(), sizeof(float) * h.post_w.size());
    memcpy(post_mask, h.post_mask.data(), sizeof(unsigned) * h.post_mask.size());
    memcpy(tri, h.tri_w.data(), sizeof(float) * NMEL);
    memcpy(tri + NMEL, h.tri_ipiv.data(), sizeof(float) * NMEL);
    memcpy(tri + 2 * NMEL, h.tri_sup.data(), sizeof(float) * NMEL);
    memcpy(spike, h.spike.data(), sizeof(float) * h.spike.size());
    return 0;
}

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

// 640-point FFT of one complex frame through pass 1 (with unit window) + pass 2: checks the
// DFT-16 / twiddle / DFT-40 codelets and the shared-memory index maps in isolation.
extern "C" int emul_fft640(const float* re, const float* im, float* out_re, float* out_im) {
    HostTables h;
    if (!build_tables(h, 16000, 0.0, 8000.0)) return -2;
    std::vector<float> ones(2 * NFFT, 1.0f);
    static EmulWarp w;
    memset(w.frames, 0, sizeof(w.frames));
    const int L = 8 * NFFT;
    std::vector<float> s(L, 0.0f), n(L, 0.0f);
    const int t = 8;  // frame 8 covers original samples [8*160-320, 8*160+320); group t0 = 8 is interior
    for (int i = 0; i < NFFT; ++i) { s[t * HOP - HALF + i] = re[i]; n[t * HOP - HALF + i] = im[i]; }
    FwdTile tl{};
    tl.sp = s.data(); tl.nz = n.data(); tl.L = L; tl.valid_s = L; tl.valid_n = L; tl.vmin = L; tl.T = 1 + L / HOP; tl.t0 = 8;
    tl.factor = 0.0f; tl.gain = 1.0f; tl.period_n = 0; tl.mixed_pcm = nullptr;
    emul_fft_stages(w, h, ones.data(), tl);
    for (int k = 0; k < NFFT; ++k) { out_re[k] = w.frames[2 * k]; out_im[k] = w.frames[2 * k + 1]; }
    return 0;
}

// mode: 0 = what the library would pick (scan when the tables allow it), 1 = force the generic path
// factor = the full SNR factor (dp:130); gain = its level-equaliser part applied to the noise at load (0: apply the whole
// factor at load, like a NULL avse_forward_args::equalizer); period: noise[i] = noise[i mod period] (0: none).
extern "C" int emul_forward_mode_ex(const float* speech, const float* noise, int L, int valid_s, int valid_n, float factor, float gain,
                                    int period, int layout, int n_slices, int ld_t, float* out_sp, float* out_nz, float* out_mix,
                                    float* mixed_pcm, float* max3, int sample_rate, double fmin, double fmax, int mode) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    const bool scan = h.scan_ok && mode == 0;
    static EmulWarp w;
    memset(w.frames, 0, sizeof(w.frames));
    const int T = 1 + L / HOP, G = (T + FPG - 1) / FPG;
    const bool have_noise = noise != nullptr;
    FwdTile tl{};
    tl.sp = speech; tl.nz = noise; tl.L = L;
    tl.valid_s = valid_s < L ? valid_s : L;
    tl.valid_n = valid_n < L ? valid_n : L;
    tl.vmin = have_noise ? (tl.valid_s < tl.valid_n ? tl.valid_s : tl.valid_n) : 0;
    if (gain == 0.0f) gain = factor;
    tl.T = T; tl.gain = have_noise ? gain : 0.0f; tl.factor = have_noise ? (gain != 0.0f ? factor / gain : 0.0f) : 0.0f;
    tl.period_n = (have_noise && period > 0 && period < tl.valid_n) ? period : 0;
    tl.mixed_pcm = mixed_pcm;
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

extern "C" int emul_forward_mode(const float* speech, const float* noise, int L, int valid_s, int valid_n, float factor,
                                 int layout, int n_slices, int ld_t, float* out_sp, float* out_nz, float* out_mix,
                                 float* mixed_pcm, float* max3, int sample_rate, double fmin, double fmax, int mode) {
    return emul_forward_mode_ex(speech, noise, L, valid_s, valid_n, factor, 0.0f, 0, layout, n_slices, ld_t, out_sp, out_nz, out_mix,
                                mixed_pcm, max3, sample_rate, fmin, fmax, mode);
}

extern "C" int emul_forward(const float* speech, const float* noise, int L, int valid_s, int valid_n, float factor,
                            int layout, int n_slices, int ld_t, float* out_sp, float* out_nz, float* out_mix,
                            float* mixed_pcm, float* max3, int sample_rate, double fmin, double fmax) {
    const int rc = emul_forward_mode(speech, noise, L, valid_s, valid_n, factor, layout, n_slices, ld_t, out_sp, out_nz, out_mix,
                                     mixed_pcm, max3, sample_rate, fmin, fmax, 0);
    return rc < 0 ? rc : 0;
}


// ---- F4 kernel (avse_fwd4_stages.cuh): one emulated warp = four frames ----
struct EmulWarp4 {
    alignas(16) float frames[WARP4_SMEM_F];
    cpx x[32][40];
    float rs[32][RAW4], rn[32][RAW4], ts[32][16], tn[32][16];
    Lane4Const lc[32];
};

// Returns 1 when the F4 tables are usable, -3 when they are not (the library then uses the 2-frame kernel).
extern "C" int emul_forward4_ex(const float* speech, const float* noise, int L, int valid_s, int valid_n, float factor, float gain,
                                int period, int layout, int n_slices, int ld_t, float* out_sp, float* out_nz, float* out_mix,
                                float* mixed_pcm, float* max3, int sample_rate, double fmin, double fmax) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    if (!h.scan4_ok || noise == nullptr) return -3;
    static EmulWarp4 w;
    memset(w.frames, 0, sizeof(w.frames));
    const int T = 1 + L / HOP, G = (T + F4 - 1) / F4;
    const vec2* s_tw = reinterpret_cast<const vec2*>(h.tw1t.data());
    const vec2* s_scanw = reinterpret_cast<const vec2*>(h.scan4_w.data());
    std::vector<ivec4> loc(NMEL);
    for (int m = 0; m < NMEL; ++m) { loc[m].x = h.scan4_loc[4 * m]; loc[m].y = h.scan4_loc[4 * m + 1]; loc[m].z = h.scan4_loc[4 * m + 2]; loc[m].w = h.scan4_loc[4 * m + 3]; }
    for (int lane = 0; lane < 32; ++lane) lane4_const_init(lane, h.window.data(), s_tw, w.lc[lane]);
    FwdTile tl{};
    tl.sp = speech; tl.nz = noise; tl.L = L;
    tl.valid_s = valid_s < L ? valid_s : L;
    tl.valid_n = valid_n < L ? valid_n : L;
    tl.vmin = tl.valid_s < tl.valid_n ? tl.valid_s : tl.valid_n;
    if (gain == 0.0f) gain = factor;
    tl.T = T; tl.gain = gain; tl.factor = gain != 0.0f ? factor / gain : 0.0f;
    tl.period_n = (period > 0 && period < tl.valid_n) ? period : 0;
    tl.mixed_pcm = mixed_pcm;
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
        } else if (AVSE_F4_REFLECT_FAST && tl.period_n == 0 && group4_reflect_only<float, true>(tl)) {
            // the kernel's reflect-only edge groups (non-tiled instantiation): mirrored loads, guarded PCM stores, interior pass 1
            FwdTileT<float> tr = tl;
            for (int lane = 0; lane < 32; ++lane) {
                p4_load_raw_reflect<float, true>(tl, lane, w.rs[lane], w.rn[lane]);
                p4_load_tail_raw_reflect<float, true>(tl, lane, w.ts[lane], w.tn[lane]);
                stage4_store_pcm_guarded(tl, lane, w.rs[lane], w.rn[lane], w.ts[lane], w.tn[lane]);
            }
            tr.mixed_pcm = nullptr;
            for (int lane = 0; lane < 32; ++lane) stage4_pass1_main(tr, lane, w.rs[lane], w.rn[lane], w.lc[lane], w.frames);
            for (int lane = 0; lane < 32; ++lane) stage4_pass1_tail_compute(tr, lane, w.ts[lane], w.tn[lane], h.window.data(), s_tw, w.frames);
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

extern "C" int emul_forward4(const float* speech, const float* noise, int L, int valid_s, int valid_n, float factor,
                             int layout, int n_slices, int ld_t, float* out_sp, float* out_nz, float* out_mix,
                             float* mixed_pcm, float* max3, int sample_rate, double fmin, double fmax) {
    return emul_forward4_ex(speech, noise, L, valid_s, valid_n, factor, 0.0f, 0, layout, n_slices, ld_t, out_sp, out_nz, out_mix,
                            mixed_pcm, max3, sample_rate, fmin, fmax);
}
