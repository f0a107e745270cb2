// Host emulation of the inverse kernel's warp stages (TEST INFRASTRUCTURE, not a product path).
// Same idea as avse_emul.cpp: csrc/avse_inv_stages.cuh is compiled with g++ and one warp is run as a
// loop over 32 lanes per stage; per-lane registers that live across a __syncwarp() are kept in arrays.
#include <vector>
#include <cstring>
#include <cmath>
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_common.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_tables.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_inv_stages.cuh"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_inv8_stages.cuh"

using namespace avse;

namespace {

struct InvWarp {
    alignas(16) float smem[INV_WARP_SMEM_F];
    cpx x[32][40];
    float acc[32][INV_SIDE_ROWS];
    float keep[32][4], carry[32][4];
};

// avse_mel_to_coef_kernel restated for the host (float32, same operation order)
void mel_to_coef(const HostTables& h, const float* mel_slices, int T_use, int T_pad, std::vector<float>& work) {
    work.assign((size_t)NMEL * T_pad, 0.0f);
    const float K = 0.16609640474436813f;
    for (int t = 0; t < T_use; ++t) {
        const int s = t / SPSS, tt = t - s * SPSS;
        float d[NMEL];
        for (int m = 0; m < NMEL; ++m) d[m] = exp2f(K * mel_slices[((size_t)s * NMEL + m) * SPSS + tt]);
        for (int m = 1; m < NMEL; ++m) d[m] -= h.tri_w[m] * d[m - 1];
        d[NMEL - 1] *= h.tri_ipiv[NMEL - 1];
        for (int m = NMEL - 2; m >= 0; --m) d[m] = (d[m] - h.tri_sup[m] * d[m + 1]) * h.tri_ipiv[m];
        for (int m = 0; m < NMEL; ++m) work[(size_t)m * T_pad + t] = d[m];
    }
}

}  // namespace

// chunks > 1 splits the utterance like the kernel does (warm-up group per chunk) to test the carry logic.
extern "C" int emul_inverse(const float* mel_slices, int n_slices, const float* pcm, int L, int valid, float* out, int out_cap,
                            int chunks, int sample_rate, double fmin, double fmax) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    const int T = 1 + L / HOP;
    const int T_use = n_slices * SPSS < T ? n_slices * SPSS : T;
    const int G = (T_use + INV_FPG - 1) / INV_FPG;
    const int T_pad = INV_FPG * (G + 1);
    const int out_len = HOP * (T_use - 1);
    if (out_cap < out_len) return -1;
    std::vector<float> work;
    mel_to_coef(h, mel_slices, T_use, T_pad, work);

    // tables as the kernel stages them
    std::vector<vec2> tw(N1 * N2), twT(N1 * N2);
    for (int k1 = 0; k1 < N1; ++k1)
        for (int n2 = 0; n2 < N2; ++n2) {
            vec2 v; v.x = h.tw1t[(k1 * N2 + n2) * 2]; v.y = h.tw1t[(k1 * N2 + n2) * 2 + 1];
            tw[k1 * N2 + n2] = v;
            twT[n2 * N1 + k1] = v;
        }
    std::vector<ivec4> col(SCAN_BINS);
    for (int k = 0; k < SCAN_BINS; ++k) {
        ivec4 e; e.x = e.y = e.z = e.w = 0;
        if (k < NBINS) {
            e.x = h.col_band[2 * k]; e.y = h.col_band[2 * k + 1];
            union { float f; int i; } u0, u1; u0.f = h.col_w[2 * k]; u1.f = h.col_w[2 * k + 1];
            e.z = u0.i; e.w = u1.i;
        }
        col[k] = e;
    }
    const float* s_win = h.window2.data();   // (w, w) pairs

    static InvWarp w;
    const int cg = (G + chunks - 1) / chunks;
    const int n_chunks = (G + cg - 1) / cg;
    for (int c = 0; c < n_chunks; ++c) {
        const int g0 = c * cg;
        int g1 = g0 + cg;
        const bool last_chunk = g1 >= G;
        if (last_chunk) g1 = G;
        const int g_first = g0 > 0 ? g0 - 1 : 0;
        const int g_last = last_chunk ? G : g1 - 1;
        memset(w.smem, 0, sizeof(w.smem));
        memset(w.acc, 0, sizeof(w.acc));
        float* frames = w.smem;
        float* ybuf = frames + 2 * FRAME_F;
        float* side = ybuf + INV_Y_F;
        InvTile tl{};
        tl.pcm = pcm; tl.L = L; tl.valid = valid < L ? valid : L; tl.T = T; tl.T_use = T_use;
        for (int g = g_first; g <= g_last; ++g) {
            tl.t0 = g * INV_FPG;
            if (tl.t0 < T_use) {
                for (int m = 0; m < NMEL; ++m)
                    for (int e = 0; e < 4; ++e) ybuf[4 * m + e] = work[(size_t)m * T_pad + tl.t0 + e];
                for (int lane = 0; lane < 32; ++lane) inv_stage_pass1(tl, lane, s_win, tw.data(), frames);
                for (int lane = 0; lane < 32; ++lane) pass2_compute(lane, frames, w.x[lane]);
                for (int lane = 0; lane < 32; ++lane) pass2_store(lane, frames, w.x[lane]);
                for (int lane = 0; lane < 32; ++lane) inv_stage_post<false>(lane, col.data(), ybuf, frames, nullptr, nullptr);
                for (int lane = 0; lane < 32; ++lane) inv_passA_compute(lane, twT.data(), frames, w.x[lane]);
                for (int lane = 0; lane < 32; ++lane) inv_passA_store(lane, frames, w.x[lane]);
                for (int lane = 0; lane < 32; ++lane) inv_stage_passB_main(lane, s_win, frames, w.acc[lane]);
                for (int lane = 0; lane < 32; ++lane) inv_stage_passB_side(lane, 0, s_win, frames, side);
                for (int lane = 0; lane < 32; ++lane) inv_stage_passB_side(lane, 1, s_win, frames, side);
            }
            const bool write = g >= g0;
            for (int lane = 0; lane < 32; ++lane) inv_stage_emit_main(lane, tl.t0, T_use, out_len, write, s_win, out, w.acc[lane]);
            for (int lane = 0; lane < 32; ++lane)
                inv_stage_emit_side(lane, tl.t0, T_use, out_len, write, s_win, out, side, w.keep[lane], w.carry[lane]);
            for (int lane = 0; lane < 32; ++lane) inv_stage_rotate_side(lane, side, w.carry[lane]);
        }
    }
    return out_len;
}


// ---- I8 kernel (avse_inv8_stages.cuh): one emulated warp = eight real frames per group; mirrors avse_inverse8_kernel's loop ----
namespace {
struct Inv8Warp {
    alignas(16) float smem[I8_WARP_SMEM_F];
    cpx x[32][40];
    float acc[32][I8_ACC];
    float raw[32][I8_RAW], rt[32][20];
    float cd[32][SPIKE_Q];
    Lane4Const lc[32];
};
}  // namespace

// All three call forms of the I8 kernel, as avse_inverse sets them up:
//   layout 0 (AVSE_LAYOUT_SLICES): mel [n_slices][80][20];  layout 1 (AVSE_LAYOUT_SPEC): mel [80][ld_t], n_frames of them used;
//   phase == nullptr: the phase of the mixture pcm[L] (zeros from `valid` on);  otherwise the explicit phase [phase_frames][321]
//   (complex64) of the EXT instantiation, and pcm / L / valid are unused.
// The warp's shared memory persists across groups and chunks like the kernel's: nothing is re-zeroed between groups.
extern "C" int emul_inverse8_ex(const float* mel, int layout, int n_slices, int n_frames, int ld_t, const float* pcm, int L, int valid,
                                const float* phase, int phase_frames, float* out, int out_cap, int chunks, int sample_rate, double fmin,
                                double fmax) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    if (layout != 0 && layout != 1) return -3;
    const bool ext = phase != nullptr;
    const int T = ext ? phase_frames : 1 + L / HOP;
    const int t_mel = layout == 0 ? n_slices * SPSS : n_frames;
    const int T_use = t_mel < T ? t_mel : T;
    if (T_use < 2 || (layout == 1 && ld_t < T_use)) return -3;
    const int G = (T_use + I8_FPG - 1) / I8_FPG;
    const int out_len = HOP * (T_use - 1);
    if (out_cap < out_len) return -1;
    const vec2* ph = reinterpret_cast<const vec2*>(phase);

    std::vector<vec2> tw(N1 * N2), twT(N1 * N2);
    for (int k1 = 0; k1 < N1; ++k1)
        for (int n2 = 0; n2 < N2; ++n2) {
            vec2 v; v.x = h.tw1t[(k1 * N2 + n2) * 2]; v.y = h.tw1t[(k1 * N2 + n2) * 2 + 1];
            tw[k1 * N2 + n2] = v;
            twT[n2 * N1 + k1] = v;
        }
    std::vector<ivec4> col(SCAN4_BINS);
#if AVSE_I8_POST_WALK
    {   // the kernel's shared-memory image: [SCAN4_BINS] (w0, w1) / 640, then [8] (mask lo, mask hi, first band, -)
        float* f = reinterpret_cast<float*>(col.data());
        for (int k = 0; k < SCAN4_BINS; ++k) { f[2 * k] = h.post_w[2 * k] * INV_SCALE; f[2 * k + 1] = h.post_w[2 * k + 1] * INV_SCALE; }
        unsigned* e = reinterpret_cast<unsigned*>(f + 2 * SCAN4_BINS);
        for (int i = 0; i < 32; ++i) e[i] = h.post_mask[i];
    }
#else
    for (int k = 0; k < SCAN4_BINS; ++k) {
        ivec4 e; e.x = e.y = e.z = e.w = 0;
        if (k < NBINS) {
            e.x = h.col_band[2 * k]; e.y = h.col_band[2 * k + 1];
            union { float f; int i; } u0, u1; u0.f = h.col_w[2 * k] * INV_SCALE; u1.f = h.col_w[2 * k + 1] * INV_SCALE;
            e.z = u0.i; e.w = u1.i;
        }
        col[k] = e;
    }
#endif
    const float* s_win = h.window.data();

    static Inv8Warp w;
    for (int lane = 0; lane < 32; ++lane) lane4_const_init(lane, s_win, tw.data(), w.lc[lane]);
    const int cg = (G + chunks - 1) / chunks;
    const int n_chunks = (G + cg - 1) / cg;
    memset(w.smem, 0, sizeof(w.smem));
    for (int c = 0; c < n_chunks; ++c) {
        const int g0 = c * cg;
        int g1 = g0 + cg;
        const bool last_chunk = g1 >= G;
        if (last_chunk) g1 = G;
        const int g_first = g0 > 0 ? g0 - 1 : 0;
        const int g_last = last_chunk ? G : g1 - 1;
        float* frames = w.smem;
        float* ybuf = frames + I8_NC * FRAME4_F;
        float* side = ybuf + I8_Y_F;
        float* xch = side + 2 * I8_SIDE_F;
        memset(w.acc, 0, sizeof(w.acc));
        memset(side, 0, sizeof(float) * 2 * I8_SIDE_F);
        InvTile tl{};
        tl.pcm = pcm; tl.L = L; tl.valid = valid < L ? valid : L; tl.T = T; tl.T_use = T_use;
        for (int g = g_first; g <= g_last; ++g) {
            tl.t0 = g * I8_FPG;
            const bool have = tl.t0 < T_use;
            const bool write = g >= g0;
            const float* side_in = side + I8_SIDE_F * (g & 1);
            float* side_out = side + I8_SIDE_F * ((g & 1) ^ 1);
            // the kernel's FFT range of the group (AVSE_I8_SKIP_FFTS): warm-up groups need FFTs 2, 3 only; frames beyond T_use none
            const bool skip_ffts = AVSE_I8_SKIP_FFTS != 0;
            const int c_lo = skip_ffts ? (write ? 0 : 2) : 0;
            const int c_left = (T_use - tl.t0 + 1) >> 1;
            const int c_hi = skip_ffts ? (c_left < I8_NC ? c_left : I8_NC) : I8_NC;
            if (have) {
                for (int lane = 0; lane < 32; ++lane) i8_coef_load(lane, mel, layout, ld_t, tl.t0, T_use, w.cd[lane]);
                if (!ext) {      // EXT: no pass 1 (and no pass 2 below), the explicit phase replaces the mixture's spectrum
                    const bool interior = i8_group_interior(tl);
                    const bool mirrored = AVSE_I8_REFLECT_FAST && !interior && i8_group_reflect_only(tl);
                    if (interior || mirrored) {
                        for (int lane = 0; lane < 32; ++lane) {
                            if (interior) { i8_load_raw(tl, lane, w.raw[lane]); i8_load_tail_raw(tl, lane, w.rt[lane]); }
                            else { i8_load_raw_reflect(tl, lane, w.raw[lane]); i8_load_tail_raw_reflect(tl, lane, w.rt[lane]); }
                        }
                        for (int lane = 0; lane < 32; ++lane) i8_pass1_main(lane, w.raw[lane], w.lc[lane], frames, c_lo, c_hi);
                        for (int lane = 0; lane < 32; ++lane) i8_pass1_tail(lane, w.rt[lane], s_win, tw.data(), frames);
                    } else {
                        for (int lane = 0; lane < 32; ++lane) i8_pass1_edge(tl, lane, s_win, tw.data(), frames, c_lo, c_hi);
                    }
                }
                for (int lane = 0; lane < 32; ++lane) i8_coef_local(lane, h.spike.data(), w.cd[lane], xch);
                for (int lane = 0; lane < 32; ++lane) i8_coef_finish(lane, h.spike.data(), w.cd[lane], xch, ybuf);
                if (ext)
                    for (int lane = 0; lane < 32; ++lane) {
                        const int tA = tl.t0 + 2 * (lane >> 3);
                        const vec2* phA = tA < T_use ? ph + (size_t)tA * NBINS : nullptr;
                        const vec2* phB = tA + 1 < T_use ? ph + (size_t)(tA + 1) * NBINS : nullptr;
                        i8_stage_post<true>(lane, col.data(), ybuf, frames, phA, phB);
                    }
                for (int it = ext ? 2 : 0; it < 4; ++it) {
                    const int r = it & 1;
                    if (it == 2 && !ext)
                        for (int lane = 0; lane < 32; ++lane) i8_stage_post<false>(lane, col.data(), ybuf, frames, nullptr, nullptr);
                    if (2 * r + 1 < c_lo || 2 * r >= c_hi) continue;
                    for (int lane = 0; lane < 32; ++lane) {
                        if (it < 2) p4_pass2_load(lane, r, frames, w.x[lane]);
                        else i8_passA_load(lane, r, frames, w.x[lane]);
                        dft40_inplace(w.x[lane]);
#if !AVSE_I8_TW_IN_B
                        if (it >= 2) inv_passA_twiddle(lane, twT.data(), w.x[lane]);
#endif
                    }
                    for (int lane = 0; lane < 32; ++lane) {
                        if (it < 2) p4_pass2_store(lane, r, frames, w.x[lane]);
                        else i8_passA_store(lane, r, frames, w.x[lane]);
                    }
                }
                if (c_lo > 0 || c_hi < I8_NC)
                    for (int lane = 0; lane < 32; ++lane) i8_rearm_flags(lane, frames);
            }
            for (int cc = 0; cc < I8_NC; ++cc)
                for (int lane = 0; lane < 32; ++lane) {
                    if (have && cc >= c_lo && cc < c_hi) i8_passB_add(lane, cc, w.lc[lane], frames, w.acc[lane]);
                    i8_emit_main(lane, tl.t0 + 2 * cc, T_use, out_len, write, s_win, out, w.acc[lane]);
                }
            if (have)
                for (int lane = 0; lane < 32; ++lane) i8_passB_tail(lane, s_win, tw.data(), frames, ybuf, c_lo, c_hi);
            for (int lane = 0; lane < 32; ++lane)
                i8_tail_reduce_emit(lane, tl.t0, T_use, out_len, write, have, s_win, out, ybuf, side_in, side_out);
        }
    }
    return out_len;
}

extern "C" int emul_inverse8(const float* mel_slices, int n_slices, const float* pcm, int L, int valid, float* out, int out_cap,
                             int chunks, int sample_rate, double fmin, double fmax) {
    return emul_inverse8_ex(mel_slices, 0, n_slices, 0, 0, pcm, L, valid, nullptr, 0, out, out_cap, chunks, sample_rate, fmin, fmax);
}

// The I8 kernel's partitioned ("SPIKE") coefficient solve alone: dB slices [n_slices][80][20] -> c[t][80] for the 8 frames of group g.
extern "C" int emul_coefficients8(const float* mel_slices, int n_slices, int g, float* out /* [8][80] */, int sample_rate, double fmin,
                                  double fmax) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    const int T_use = n_slices * SPSS;
    static float cd[32][SPIKE_Q];
    std::vector<float> ybuf(I8_Y_F, 0.0f), xch(I8_XCH_F, 0.0f);
    for (int lane = 0; lane < 32; ++lane) i8_coef_load(lane, mel_slices, 0, 0, g * I8_FPG, T_use, cd[lane]);
    for (int lane = 0; lane < 32; ++lane) i8_coef_local(lane, h.spike.data(), cd[lane], xch.data());
    for (int lane = 0; lane < 32; ++lane) i8_coef_finish(lane, h.spike.data(), cd[lane], xch.data(), ybuf.data());
    for (int f = 0; f < I8_FPG; ++f)
        for (int m = 0; m < NMEL; ++m) out[f * NMEL + m] = ybuf[I8_YS * m + f];
    return 0;
}
