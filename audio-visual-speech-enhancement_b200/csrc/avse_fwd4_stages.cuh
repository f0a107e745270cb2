// Warp-stage functions of the fast forward kernel ("F4": one warp owns FOUR consecutive STFT frames).
//
// Same arithmetic as avse_fwd_stages.cuh (packed z = s + i n, 640 = 16 x 40, STFT linearity for the
// mixture, fused unpack + mel scan, dB); what changes is the mapping onto the SM, chosen from the ncu
// profile of the 2-frame kernel, whose limiter was the shared-memory / LSU data pipe (77 % busy):
//
//   * pass 1: lane = n2 for ALL four frames, so the 16 window values and 15 twiddles of a lane are the
//     same for every frame and every group: they live in registers for the whole kernel (no table loads),
//     and the four frames of a group (hop = 4 strides of 40 samples) share one batch of 28 strided loads
//     per signal (each sample is loaded once per group instead of 2.3 times).  The 8 residues
//     n2 = 32..39 of the four frames form a fifth full round (lane = (frame, n2 - 32)).
//     4 x 40 columns = 5 rounds of 32 lanes: every lane busy (the 2-frame kernel wasted 1/6 of pass 1).
//   * pass 2: 64 rows = 2 rounds (lane = (frame pair, k1)).
//   * scan:  lane = (frame, chunk of 41 bins); finished band sums are written DENSELY over the chunk's
//     own already-consumed slots, so the dB stage (lane = band) reads them without bank conflicts.
//   * dB:    lane = band; the four frames of a group are 16 contiguous bytes of the slice layout.
//
// 8 warps per SM with up to 255 registers each (instead of 16 x 128).
// Reference semantics: /root/reference/data_processor.py:77-96, :130-133, :35-57 (SURVEY.md App. A).
#pragma once
#include "avse_common.h"
#include "avse_dft.cuh"
#include "avse_fwd_stages.cuh"

#if !defined(AVSE_DB_FAST_MINMAX)
#define AVSE_DB_FAST_MINMAX 0     // 1: min / max of a full group's four frames without the per-frame validity selects
#endif
#if !defined(AVSE_SCAN4_UNROLL)
#define AVSE_SCAN4_UNROLL 8
#endif

namespace avse {

constexpr int F4 = 4;                          // frames per group
constexpr int CHUNK4 = 41;                     // bins per scan lane (odd: bank spread); 8 x 41 = 328 >= 321
constexpr int SCAN4_BINS = 8 * CHUNK4;         // 328
constexpr int FRAME4_F = N1 * ROW_F + 16;      // 1360 floats per frame buffer, == 16 (mod 32)
constexpr int ZERO4_F = N1 * ROW_F;             // floats [1344, 1360) of a frame buffer are never written: always zero
#ifndef AVSE_SCAN4_BLK
#define AVSE_SCAN4_BLK 4          // bins per unrolled block of the scan: 1 / 2 / 4 / 5 / 8 / 10 / 20 -> 0.567 / 0.548 / 0.532 / 0.537 / 0.533 / 0.542 / 0.553 ms
#endif
#ifndef AVSE_DB_BRANCHFREE_EXTRA
#define AVSE_DB_BRANCHFREE_EXTRA 1
#endif
constexpr int FLUSH4_F = 1284;                 // chunk-end partial sums: 8 chunks x 6 floats in [1284, 1332)
constexpr int WARP4_SMEM_F = F4 * FRAME4_F;    // 5440 floats = 21760 B per warp
constexpr int RAW4 = 16 + 4 * (F4 - 1);        // 28 strides of 40 samples cover the four frames of a group
static_assert(FLUSH4_F + 48 <= FRAME4_F && (FLUSH4_F % 2) == 0, "flush area");

// Loop-invariant per-lane constants of pass 1 (n2 = lane): registers for the whole kernel.
struct Lane4Const {
    float win[16];   // Hann w[40 j + lane]
    vec2 tw[16];     // W_640^{lane * k1}  (tw[0] unused)
};

AVSE_HD void lane4_const_init(int lane, const float* s_win, const vec2* s_tw, Lane4Const& lc) {
#pragma unroll
    for (int j = 0; j < 16; ++j) { lc.win[j] = s_win[N2 * j + lane]; lc.tw[j] = s_tw[j * N2 + lane]; }
}

// A group is "interior" when its four frames exist and need neither reflection nor zero padding, and -- for a
// periodically tiled noise (dp:125-128, period_n > 0, read from phase_n on) -- when the group's 1 120 samples do not
// straddle a period boundary.  nz_shift is then the offset that maps the group's sample indices into the stored period:
// noise[i] = nz[(phase_n + i) mod period_n] = nz[i + nz_shift] for every i of the group.
// TILED = false compiles the period logic out (the common kernel instantiation: see avse_forward4_kernel).
template <typename S, bool TILED>
AVSE_HD bool group4_interior(const FwdTileT<S>& tl, int& nz_shift) {
    nz_shift = 0;
    const int a = tl.t0 * HOP - HALF;                       // first sample of the group
    if (!(tl.nz != nullptr && a >= 0 && (tl.t0 + 3) * HOP + HALF <= tl.vmin && tl.t0 + 3 < tl.T)) return false;
    if (TILED && tl.period_n > 0) {
        const int j = a + tl.phase_n;
        const int q = j / tl.period_n;
        if ((j + (F4 - 1) * HOP + NFFT - 1) / tl.period_n != q) return false;
        nz_shift = tl.phase_n - q * tl.period_n;
    }
    return true;
}

// DFT-16 over n1, twiddle, store column as rows [k1][n2] of one frame buffer (dst = frame + 2 n2).
AVSE_HD void p4_column(cpx (&x)[16], const vec2 (&tw)[16], float* dst) {
    dft16(x);
    cstore(dst, x[0]);
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) cstore(dst + k1 * ROW_F, cmul(x[k1], tw[k1].x, tw[k1].y));
}

// The 28 strided samples per signal that the lane's column needs for the four frames (interior groups).
template <typename S>
AVSE_HD void p4_load_raw(const FwdTileT<S>& tl, int nz_shift, int lane, float (&rs)[RAW4], float (&rn)[RAW4]) {
    const int o = tl.t0 * HOP - HALF + lane;
    const S* ps = tl.sp + o;
    const S* pn = tl.nz + (o + nz_shift);
#pragma unroll
    for (int j = 0; j < RAW4; ++j) { rs[j] = (float)ps[N2 * j]; rn[j] = (float)pn[N2 * j]; }
}

// ---------------------------------------------------------------------------------------
// Reflect-only edge groups (AVSE_F4_REFLECT_FAST): the first group of an utterance and the last ones differ from an interior
// group only in WHERE their samples come from when both signals are full length (no zero padding) and the noise is not tiled:
// librosa's centre padding mirrors the index (pad_mode='reflect', dp:79).  Such a group takes the interior pass 1 with mirrored
// load indices instead of the per-sample edge loader (3 of the 76 groups of a 3 s utterance, each 3.4 x the interior cost).
// Frames past the last one read mirrored samples too (finite, never stored: the edge stage duplicates the last frame instead).
// The mixture PCM of the group's own hops is stored by stage4_store_pcm_guarded (the interior stores are unguarded).
// ---------------------------------------------------------------------------------------
#if !defined(AVSE_F4_REFLECT_FAST)
#define AVSE_F4_REFLECT_FAST 1
#endif
AVSE_HD int reflect_index(int i, int L) {
    i = i < 0 ? -i : i;
    const int m = 2 * (L - 1) - i;
    return i < m ? i : m;
}

// PAD (template parameter of the kernel, set by the launcher when the batch carries per-utterance lengths): utterances shorter than
// the row (pad_with_zeros, dp:40) take the fast path too, through a guarded variant of the mirrored loader -- a mirrored index at or
// past the valid length reads 0 without touching memory.  A separate instantiation like TILED: compiled into the common kernel the
// extra loader cost the full-length benchmark 2.2 % (register allocation of the tile loop) for 7 % on a ragged batch.
template <typename S, bool PAD>
AVSE_HD bool group4_reflect_only(const FwdTileT<S>& tl) {
    // L >= 4 n_fft keeps every mirrored index inside [0, L), the phantom frames of the last group included
    return tl.nz != nullptr && (PAD || tl.vmin >= tl.L) && tl.period_n == 0 && tl.L >= 4 * NFFT;
}

template <typename S, bool PAD>
AVSE_HD void p4_load_raw_reflect(const FwdTileT<S>& tl, int lane, float (&rs)[RAW4], float (&rn)[RAW4]) {
    const int o = tl.t0 * HOP - HALF + lane;
    if (!PAD || tl.vmin >= tl.L) {          // full-length rows (warp-uniform): no guard
#pragma unroll
        for (int j = 0; j < RAW4; ++j) { const int i = reflect_index(o + N2 * j, tl.L); rs[j] = (float)tl.sp[i]; rn[j] = (float)tl.nz[i]; }
    } else {                                             // zero padding: a mirrored index at or past the valid length reads 0, untouched
#pragma unroll
        for (int j = 0; j < RAW4; ++j) {
            const int i = reflect_index(o + N2 * j, tl.L);
            rs[j] = i < tl.valid_s ? (float)tl.sp[i] : 0.0f;
            rn[j] = i < tl.valid_n ? (float)tl.nz[i] : 0.0f;
        }
    }
}

template <typename S, bool PAD>
AVSE_HD void p4_load_tail_raw_reflect(const FwdTileT<S>& tl, int lane, float (&rs)[16], float (&rn)[16]) {
    const int o = (tl.t0 + (lane >> 3)) * HOP - HALF + 32 + (lane & 7);
    if (!PAD || tl.vmin >= tl.L) {
#pragma unroll
        for (int j = 0; j < 16; ++j) { const int i = reflect_index(o + N2 * j, tl.L); rs[j] = (float)tl.sp[i]; rn[j] = (float)tl.nz[i]; }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int i = reflect_index(o + N2 * j, tl.L);
            rs[j] = i < tl.valid_s ? (float)tl.sp[i] : 0.0f;
            rn[j] = i < tl.valid_n ? (float)tl.nz[i] : 0.0f;
        }
    }
}

// s + factor * (gain * n) of the group's own hops, samples < L only: the same arithmetic as the interior stores of
// stage4_pass1_main / stage4_pass1_tail_compute (rn, tn still unscaled here).
template <typename S>
AVSE_HD void stage4_store_pcm_guarded(const FwdTileT<S>& tl, int lane, const float (&rs)[RAW4], const float (&rn)[RAW4], const float (&ts)[16],
                                      const float (&tn)[16]) {
    if (tl.mixed_pcm == nullptr) return;
    const int i0 = tl.t0 * HOP + lane;
#pragma unroll
    for (int j = 8; j < 24; ++j) {
        const int i = i0 + N2 * (j - 8);
        if (i < tl.L) tl.mixed_pcm[i] = rs[j] + tl.factor * (rn[j] * tl.gain);
    }
    const int i1 = (tl.t0 + (lane >> 3)) * HOP + 32 + (lane & 7);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int i = i1 + N2 * j;
        if (i < tl.L) tl.mixed_pcm[i] = ts[8 + j] + tl.factor * (tn[8 + j] * tl.gain);
    }
}

// Rounds 0..3 of an interior group: frame f, column n2 = lane.  Also stores the mixture PCM (dp:133) of the
// group's own four hops (strides 8..23 of the batch) for the residues n2 < 32.
// The raw noise samples are scaled by the level equaliser tl.gain here (see FwdTileT).
// AVSE_P1_ROLL (tuning switch, A/B-measured on B200 -- profiles/README.md round 2):
//   9 = all 28 strides scaled up front, mixture PCM stored first, four frames unrolled   (0.549 ms, the default)
//   0 = scaled / stored frame by frame in consumption order, four frames unrolled         (0.558 ms)
//   4 = ONE copy of the column code in a rolled loop whose 16-stride window slides through the raw registers by
//       rotation: 590 fewer instructions in a hot loop that exceeds the 32 KB L1.5 instruction cache   (0.553 ms)
//   2 = two frames per iteration
#if !defined(AVSE_P1_ROLL)
#define AVSE_P1_ROLL 9
#endif
template <typename S>
AVSE_HD void stage4_pass1_main(const FwdTileT<S>& tl, int lane, float (&rs)[RAW4], float (&rn)[RAW4],
                               const Lane4Const& lc, float* frames) {
    const float gain = tl.gain;
#if AVSE_P1_ROLL == 9      // round-1 order: everything scaled up front, the mixture PCM stored first
#pragma unroll
    for (int j = 0; j < RAW4; ++j) rn[j] *= gain;
    if (tl.mixed_pcm != nullptr) {
        float* pm = tl.mixed_pcm + tl.t0 * HOP + lane;
#pragma unroll
        for (int j = 8; j < 24; ++j) pm[N2 * (j - 8)] = rs[j] + tl.factor * rn[j];
    }
#pragma unroll
    for (int f = 0; f < F4; ++f) {
        cpx x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = cmake(rs[4 * f + j] * lc.win[j], rn[4 * f + j] * lc.win[j]);
        p4_column(x, lc.tw, frames + f * FRAME4_F + 2 * lane);
    }
#elif AVSE_P1_ROLL == 0
#pragma unroll
    for (int j = 0; j < 12; ++j) rn[j] *= gain;
#pragma unroll
    for (int f = 0; f < F4; ++f) {
#pragma unroll
        for (int j = 12; j < 16; ++j) rn[4 * f + j] *= gain;
        if (tl.mixed_pcm != nullptr) {         // this frame's own hop (dp:133): strides 8..11 of its window
            float* pm = tl.mixed_pcm + (tl.t0 + f) * HOP + lane;
#pragma unroll
            for (int j = 0; j < 4; ++j) pm[N2 * j] = rs[4 * f + 8 + j] + tl.factor * rn[4 * f + 8 + j];
        }
        cpx x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = cmake(rs[4 * f + j] * lc.win[j], rn[4 * f + j] * lc.win[j]);
        p4_column(x, lc.tw, frames + f * FRAME4_F + 2 * lane);
    }
#else
    constexpr int STEP = AVSE_P1_ROLL == 4 ? 1 : 2;      // frames per loop iteration
    constexpr int W = 16 + 4 * (STEP - 1);              // strides the iteration reads
#pragma unroll
    for (int j = 0; j < 12; ++j) rn[j] *= gain;
    float* pm = tl.mixed_pcm != nullptr ? tl.mixed_pcm + tl.t0 * HOP + lane : nullptr;
    float* dst = frames + 2 * lane;
#pragma unroll 1
    for (int it = 0; it < F4 / STEP; ++it) {
#pragma unroll
        for (int j = 12; j < W; ++j) rn[j] *= gain;
#pragma unroll
        for (int f = 0; f < STEP; ++f) {
            if (pm != nullptr) {
#pragma unroll
                for (int j = 0; j < 4; ++j) pm[N2 * j] = rs[4 * f + 8 + j] + tl.factor * rn[4 * f + 8 + j];
                pm += HOP;
            }
            cpx x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = cmake(rs[4 * f + j] * lc.win[j], rn[4 * f + j] * lc.win[j]);
            p4_column(x, lc.tw, dst);
            dst += FRAME4_F;
        }
#pragma unroll
        for (int j = 0; j + 4 * STEP < RAW4; ++j) { rs[j] = rs[j + 4 * STEP]; rn[j] = rn[j + 4 * STEP]; }
    }
#endif
}

// Round 4 of an interior group: lane = (f = lane / 8, r = lane % 8), column n2 = 32 + r of frame f.
// Window / twiddles come from the CTA's shared tables (8 distinct addresses per load: one wavefront).
template <typename S>
AVSE_HD void p4_load_tail_raw(const FwdTileT<S>& tl, int nz_shift, int lane, float (&rs)[16], float (&rn)[16]) {
    const int f = lane >> 3, n2 = 32 + (lane & 7);
    const int o = (tl.t0 + f) * HOP - HALF + n2;
    const S* ps = tl.sp + o;
    const S* pn = tl.nz + (o + nz_shift);
#pragma unroll
    for (int j = 0; j < 16; ++j) { rs[j] = (float)ps[N2 * j]; rn[j] = (float)pn[N2 * j]; }
}

template <typename S>
AVSE_HD void stage4_pass1_tail_compute(const FwdTileT<S>& tl, int lane, const float (&rs)[16], float (&rn)[16], const float* s_win,
                                       const vec2* s_tw, float* frames) {
    const int f = lane >> 3, n2 = 32 + (lane & 7);
#pragma unroll
    for (int j = 0; j < 16; ++j) rn[j] *= tl.gain;
    vec2 tw[16];
#pragma unroll
    for (int k1 = 1; k1 < 16; ++k1) tw[k1] = s_tw[k1 * N2 + n2];
    tw[0].x = 1.0f; tw[0].y = 0.0f;
    if (tl.mixed_pcm != nullptr) {
        float* pm = tl.mixed_pcm + (tl.t0 + f) * HOP + n2;    // this frame's own hop: strides 8..11
#pragma unroll
        for (int j = 0; j < 4; ++j) pm[N2 * j] = rs[8 + j] + tl.factor * rn[8 + j];
    }
    cpx x[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) { const float w = s_win[N2 * j + n2]; x[j] = cmake(rs[j] * w, rn[j] * w); }
    p4_column(x, tw, frames + f * FRAME4_F + 2 * n2);
}

template <typename S>
AVSE_HD void stage4_pass1_tail(const FwdTileT<S>& tl, int nz_shift, int lane, const float* s_win, const vec2* s_tw, float* frames) {
    float rs[16], rn[16];
    p4_load_tail_raw(tl, nz_shift, lane, rs, rn);
    stage4_pass1_tail_compute(tl, lane, rs, rn, s_win, s_tw, frames);
}

// Pass 1 of an interior group as ONE rolled loop over its five rounds (four main rounds + the tail round): the round-specific
// part is only the 32 window multiplies (a switch over the round picks the statically indexed raw registers), the DFT-16 +
// twiddle + store code exists once.  The twiddles of a lane are no longer kernel-lifetime registers: they are (re)loaded from
// the CTA's table at round 0 (n2 = lane) and round 4 (n2 = 32 + lane % 8), 15 + 15 8-byte loads per group, which also frees 32
// registers.  Motivation: the hot loop of this kernel is ~45 KB against a 32 KB L1.5 instruction cache, and pass 1 was 1 500
// of its 2 800 instructions (AVSE_P1_UNIFIED, A/B in profiles/README.md).
template <typename S>
AVSE_HD void stage4_pass1_unified(const FwdTileT<S>& tl, int lane, float (&rs)[RAW4], float (&rn)[RAW4], const float (&ts)[16], float (&tn)[16],
                                  const Lane4Const& lc, const float* s_win, const vec2* s_tw, float* frames) {
    const float gain = tl.gain;
    const int tf = lane >> 3, tn2 = 32 + (lane & 7);          // the lane's (frame, column) in the tail round
#pragma unroll
    for (int j = 0; j < RAW4; ++j) rn[j] *= gain;
#pragma unroll
    for (int j = 0; j < 16; ++j) tn[j] *= gain;
    if (tl.mixed_pcm != nullptr) {
        float* pm = tl.mixed_pcm + tl.t0 * HOP + lane;
#pragma unroll
        for (int j = 8; j < 24; ++j) pm[N2 * (j - 8)] = rs[j] + tl.factor * rn[j];
        float* pt = tl.mixed_pcm + (tl.t0 + tf) * HOP + tn2;
#pragma unroll
        for (int j = 0; j < 4; ++j) pt[N2 * j] = ts[8 + j] + tl.factor * tn[8 + j];
    }
    vec2 tw[16];
    tw[0].x = 1.0f; tw[0].y = 0.0f;
#pragma unroll 1
    for (int round = 0; round < 5; ++round) {
        if (round == 0 || round == 4) {
            const int n2 = round == 0 ? lane : tn2;
#pragma unroll
            for (int k1 = 1; k1 < 16; ++k1) tw[k1] = s_tw[k1 * N2 + n2];
        }
        cpx x[16];
        float* dst;
        switch (round) {
        case 0:
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = cmake(rs[j] * lc.win[j], rn[j] * lc.win[j]);
            dst = frames + 2 * lane;
            break;
        case 1:
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = cmake(rs[4 + j] * lc.win[j], rn[4 + j] * lc.win[j]);
            dst = frames + FRAME4_F + 2 * lane;
            break;
        case 2:
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = cmake(rs[8 + j] * lc.win[j], rn[8 + j] * lc.win[j]);
            dst = frames + 2 * FRAME4_F + 2 * lane;
            break;
        case 3:
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = cmake(rs[12 + j] * lc.win[j], rn[12 + j] * lc.win[j]);
            dst = frames + 3 * FRAME4_F + 2 * lane;
            break;
        default:
#pragma unroll
            for (int j = 0; j < 16; ++j) { const float w = s_win[N2 * j + tn2]; x[j] = cmake(ts[j] * w, tn[j] * w); }
            dst = frames + tf * FRAME4_F + 2 * tn2;
            break;
        }
        p4_column(x, tw, dst);
    }
}

// Edge / generic groups (first and last frames of an utterance, short or zero-padded signals): every sample
// goes through the reflect + zero-pad loader.  Cold code, rolled over the five rounds.
template <typename S, bool TILED>
AVSE_HD void stage4_pass1_edge(const FwdTileT<S>& tl, int lane, const float* s_win, const vec2* s_tw, float* frames) {
#pragma unroll 1
    for (int round = 0; round < 5; ++round) {
        const int f = round < 4 ? round : lane >> 3;
        const int n2 = round < 4 ? lane : 32 + (lane & 7);
        const int t_raw = tl.t0 + f;
        const int t = t_raw < tl.T ? t_raw : tl.T - 1;   // frames past the end duplicate the last one (never stored)
        const int base = t * HOP - HALF + n2;
        float rs[16], rn[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            rs[j] = load_sample_edge(tl.sp, base + N2 * j, tl.L, tl.valid_s);
            rn[j] = tl.gain * load_sample_edge(tl.nz, base + N2 * j, tl.L, tl.valid_n, TILED ? tl.period_n : 0, TILED ? tl.phase_n : 0);
        }
        if (tl.mixed_pcm != nullptr && t_raw < tl.T) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int i = t * HOP + N2 * j + n2;     // this frame's own hop: strides 8..11
                if (i < tl.L) tl.mixed_pcm[i] = rs[8 + j] + tl.factor * rn[8 + j];
            }
        }
        vec2 tw[16];
#pragma unroll
        for (int k1 = 1; k1 < 16; ++k1) tw[k1] = s_tw[k1 * N2 + n2];
        tw[0].x = 1.0f; tw[0].y = 0.0f;
        cpx x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) { const float w = s_win[N2 * j + n2]; x[j] = cmake(rs[j] * w, rn[j] * w); }
        p4_column(x, tw, frames + f * FRAME4_F + 2 * n2);
    }
}

// ---------------------------------------------------------------------------------------
// pass 2, round r: lane = (f = 2 r + lane / 16, k1 = lane % 16): row -> in-place DFT-40 -> (after a warp
// sync) natural order Z[k1 + 16 k2] over the same frame buffer.
// ---------------------------------------------------------------------------------------
AVSE_HD void p4_pass2_load(int lane, int r, const float* frames, cpx (&x)[40]) {
    const int f = 2 * r + (lane >> 4), k1 = lane & 15;
    const float* row = frames + f * FRAME4_F + k1 * ROW_F;
#pragma unroll
    for (int q = 0; q < 20; ++q) cload2(row + 4 * q, x[2 * q], x[2 * q + 1]);
}

AVSE_HD void p4_pass2_compute(int lane, int r, const float* frames, cpx (&x)[40]) {
    p4_pass2_load(lane, r, frames, x);
    dft40_inplace(x);
}

AVSE_HD void p4_pass2_store(int lane, int r, float* frames, const cpx (&x)[40]) {
    const int f = 2 * r + (lane >> 4), k1 = lane & 15;
    float* z = frames + f * FRAME4_F + 2 * k1;
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
// Fused unpack + mel scan: lane = (f = lane / 8, chunk p = lane % 8) walks bins k = 41 p + i, i = 0..40.
//   S' = Z_k + conj Z_{N-k}, N' = (Z_k - conj Z_{N-k}) / i, M' = S' + factor N'   (2 x the three spectra)
//   band sums: A = band seg-1 (falling edge), B = band seg (rising edge), weights (wa, wb) = 0.5 F[.][k].
// When the segment advances before bin i (bit i of the chunk's mask) A is complete for this lane: its
// (speech, noise) pair goes to complex slot 41 p + e and its mixture sum to float 1281 - 82 p - e, e = number
// of earlier emissions of the lane (both locations were consumed by this lane in an earlier iteration).
// The two sums left at the end go to the flush area.  s_w: [SCAN4_BINS] (wa, wb).
// ---------------------------------------------------------------------------------------
AVSE_HD float fma_rn(float a, float b, float c) { return fmaf(a, b, c); }

// One bin of the scan.  n' = Z_k - conj Z_{N-k} = i N' has the same magnitude as N', and the mixture follows from
// M' = S' + factor N' = S' + factor (n'_im, -n'_re): bit-identical to forming N' first, with one packed op less.
AVSE_HD void scan4_bin(const float* za, const float* zc, const vec2* tab, int j, bool emit, float factor, float nfactor,
                       float*& esn, float*& em, cpx& Asn, cpx& Bsn, float& Am, float& Bm) {
    const cpx a = cload(za + 2 * j);
    const cpx c = cload(zc - 2 * j);
    const vec2 w = tab[j];                                                // (wa, wb): one 8-byte load (2 wavefronts; 16 bytes cost 4)
    if (emit) {
        cstore(esn, Asn);
        *em = Am;
        esn += 2;
        em -= 1;
        Asn = Bsn; Am = Bm;
        Bsn = cmake(0.0f, 0.0f); Bm = 0.0f;
    }
    const cpx s = cfma_pp(c, cmake(1.0f, -1.0f), a);                      // 2 X_speech[k] = Z_k + conj Z_{N-k}
    const cpx n = cfma_pp(c, cmake(-1.0f, 1.0f), a);                      // 2 i X_noise[k] = Z_k - conj Z_{N-k}
    const float mr = fma_rn(factor, cim(n), cre(s));                      // 2 X_mixed[k]
    const float mi = fma_rn(nfactor, cre(n), cim(s));
    const float ms = fast_sqrt(fma_rn(cim(s), cim(s), cre(s) * cre(s)));
    const float mn = fast_sqrt(fma_rn(cim(n), cim(n), cre(n) * cre(n)));
    const float mm = fast_sqrt(fma_rn(mi, mi, mr * mr));
    const cpx msn = cmake(ms, mn);
    Asn = cfma_pp(msn, cmake(w.x, w.x), Asn);
    Bsn = cfma_pp(msn, cmake(w.y, w.y), Bsn);
    Am = fma_rn(w.x, mm, Am);
    Bm = fma_rn(w.y, mm, Bm);
}

// s_w: [SCAN4_BINS] (wa, wb).  Blocks of 8 bins with compile-time mask bit positions (the mask is shifted
// once per block), so the emission test is a single predicate-setting logic op per bin.
AVSE_HD void stage4_scan(int lane, float factor, const vec2* s_w, unsigned mask_lo, unsigned mask_hi, float* frames) {
    const int f = lane >> 3, p = lane & 7;
    float* fr = frames + f * FRAME4_F;
    const float* za = fr + 2 * CHUNK4 * p;            // slot k      = za + 2 i
    const float* zc = fr + 2 * (NFFT - CHUNK4 * p);   // slot 640-k  = zc - 2 i
    const vec2* tab = s_w + CHUNK4 * p;
    float* esn = fr + 2 * CHUNK4 * p;                 // next (speech, noise) emission slot
    float* em = fr + 2 * (NFFT - CHUNK4 * p) + 1;     // next mixture emission float
    cpx Asn = cmake(0.0f, 0.0f), Bsn = cmake(0.0f, 0.0f);
    float Am = 0.0f, Bm = 0.0f;
    const float nfactor = -factor;
    unsigned mlo = mask_lo, mhi = mask_hi;
    static_assert(CHUNK4 == 41 && (40 % AVSE_SCAN4_BLK) == 0 && AVSE_SCAN4_BLK < 32, "blocks of AVSE_SCAN4_BLK bins + 1");
#pragma unroll 1
    for (int ib = 0; ib < 40; ib += AVSE_SCAN4_BLK) {
#pragma unroll
        for (int j = 0; j < AVSE_SCAN4_BLK; ++j) scan4_bin(za, zc, tab, j, ((mlo >> j) & 1u) != 0u, factor, nfactor, esn, em, Asn, Bsn, Am, Bm);
        za += 2 * AVSE_SCAN4_BLK; zc -= 2 * AVSE_SCAN4_BLK; tab += AVSE_SCAN4_BLK;
        mlo = (mlo >> AVSE_SCAN4_BLK) | (mhi << (32 - AVSE_SCAN4_BLK));
        mhi >>= AVSE_SCAN4_BLK;
    }
    scan4_bin(za, zc, tab, 0, (mlo & 1u) != 0u, factor, nfactor, esn, em, Asn, Bsn, Am, Bm);
    float* fl = fr + FLUSH4_F + 6 * p;
    cstore(fl + 0, Asn);
    cstore(fl + 2, Bsn);
    cstore(fl + 4, cmake(Am, Bm));
}

// ---------------------------------------------------------------------------------------
// dB stage: lane = band m = 32 q + lane.  s_loc[m] = (main, extra1, extra2, -): each a packed pair of
// frame-relative float offsets (speech/noise pair | mixture << 16) of one partial sum; extras are -1
// when absent (a band cut by a chunk boundary has up to three partial sums).
// ---------------------------------------------------------------------------------------
// mx[sig]: running max over ALL frames < T (librosa's max is over the whole (80, T) array, dp:94);
// mn[32 sig + lane]: per-lane running min over the values actually STORED (lets the floor pass skip utterances that need
// no clipping); kept in shared memory because three more loop-carried registers cost 12 % of the kernel (255-register cliff).
AVSE_HD void stage4_db(int lane, int q, float factor, const ivec4* s_loc, const float* frames, const FwdOut& out, int t0, int T,
                       float (&mx)[3], float* mn) {
    const int m = 32 * q + lane;
    if (m >= NMEL) return;
    const ivec4 loc = s_loc[m];
    float mel[3][F4];
#pragma unroll
    for (int f = 0; f < F4; ++f) {
        const float* fr = frames + f * FRAME4_F;
        const vec2 sn = *reinterpret_cast<const vec2*>(fr + (loc.x & 0xffff));
        mel[0][f] = sn.x; mel[1][f] = sn.y; mel[2][f] = fr[loc.x >> 16];
    }
#if AVSE_DB_BRANCHFREE_EXTRA
    {   // second partial sum: bands without one read the buffer's zero pad (ZERO4_F, avse_tables.cpp) -- no divergent branch
#pragma unroll
        for (int f = 0; f < F4; ++f) {
            const float* fr = frames + f * FRAME4_F;
            const vec2 sn = *reinterpret_cast<const vec2*>(fr + (loc.y & 0xffff));
            mel[0][f] += sn.x; mel[1][f] += sn.y; mel[2][f] += fr[loc.y >> 16];
        }
    }
#else
    if ((loc.y & 0xffff) != ZERO4_F) {
#pragma unroll
        for (int f = 0; f < F4; ++f) {
            const float* fr = frames + f * FRAME4_F;
            const vec2 sn = *reinterpret_cast<const vec2*>(fr + (loc.y & 0xffff));
            mel[0][f] += sn.x; mel[1][f] += sn.y; mel[2][f] += fr[loc.y >> 16];
        }
    }
#endif
    if (loc.z >= 0) {
#pragma unroll
        for (int f = 0; f < F4; ++f) {
            const float* fr = frames + f * FRAME4_F;
            const vec2 sn = *reinterpret_cast<const vec2*>(fr + (loc.z & 0xffff));
            mel[0][f] += sn.x; mel[1][f] += sn.y; mel[2][f] += fr[loc.z >> 16];
        }
    }
    const int nvalid = T - t0 < F4 ? T - t0 : F4;   // >= 1
    int off;
    bool store = true;
    if (out.layout == 0) {
        const int sl = t0 / SPSS, tt = t0 - sl * SPSS;   // 4 | t0 and 4 | 20: a group never straddles slices
        off = (sl * NMEL + m) * SPSS + tt;
        store = sl < out.n_slices;                        // implies nvalid == 4 (n_slices <= T / 20)
    } else {
        off = m * out.ld_t + t0;
    }
#pragma unroll
    for (int sig = 0; sig < 3; ++sig) {
        const float scale = sig == 1 ? factor : 1.0f;
        float d[F4];
        float lm = neg_inf(), ln = -neg_inf();
#pragma unroll
        for (int f = 0; f < F4; ++f) d[f] = amp_to_db(mel[sig][f] * scale);
#if AVSE_DB_FAST_MINMAX
        if (nvalid == F4) {                    // warp-uniform: every group but the utterance's last one
            lm = fmaxf(fmaxf(d[0], d[1]), fmaxf(d[2], d[3]));
            ln = fminf(fminf(d[0], d[1]), fminf(d[2], d[3]));
        } else
#endif
        {
#pragma unroll
            for (int f = 0; f < F4; ++f) {
                const bool v = f < nvalid;
                lm = v ? fmaxf(lm, d[f]) : lm;     // branch-free: selects, no divergent code in the hot dB loop
                ln = v ? fminf(ln, d[f]) : ln;
            }
        }
        mx[sig] = fmaxf(lm, mx[sig]);
        float* dst = out.dst[sig];
        mn[32 * sig + lane] = fminf(mn[32 * sig + lane], (dst != nullptr && store) ? ln : -neg_inf());
        if (dst != nullptr && store) {
            if (out.layout == 0) {
                vec4 o; o.x = d[0]; o.y = d[1]; o.z = d[2]; o.w = d[3];
                *reinterpret_cast<vec4*>(dst + off) = o;     // 16-byte aligned: off % 4 == 0
            } else {
#pragma unroll
                for (int f = 0; f < F4; ++f)
                    if (f < nvalid) dst[off + f] = d[f];
            }
        }
    }
}

// The last 16 bands (64..79) with all 32 lanes: lane = (half = lane / 16, band 64 + lane % 16) converts frames 2 half, 2 half + 1.
// As round q = 2 of stage4_db these bands keep 16 lanes idle for a whole round (80 bands on 32 lanes), a sixth of the dB stage;
// this form costs a second, smaller copy of the stage's code (AVSE_DB_SPLIT_LAST).  Same arithmetic per value, 8-byte stores.
#if !defined(AVSE_DB_SPLIT_LAST)
#define AVSE_DB_SPLIT_LAST 1
#endif
AVSE_HD void stage4_db_last(int lane, float factor, const ivec4* s_loc, const float* frames, const FwdOut& out, int t0, int T,
                            float (&mx)[3], float* mn) {
    const int half = lane >> 4, m = 64 + (lane & 15), f0 = 2 * half;
    const ivec4 loc = s_loc[m];
    float mel[3][2];
#pragma unroll
    for (int f = 0; f < 2; ++f) {
        const float* fr = frames + (f0 + f) * FRAME4_F;
        const vec2 sn = *reinterpret_cast<const vec2*>(fr + (loc.x & 0xffff));
        mel[0][f] = sn.x; mel[1][f] = sn.y; mel[2][f] = fr[loc.x >> 16];
        const vec2 s2 = *reinterpret_cast<const vec2*>(fr + (loc.y & 0xffff));      // zero pad when absent (AVSE_DB_BRANCHFREE_EXTRA)
        mel[0][f] += s2.x; mel[1][f] += s2.y; mel[2][f] += fr[loc.y >> 16];
    }
    if (loc.z >= 0) {
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            const float* fr = frames + (f0 + f) * FRAME4_F;
            const vec2 sn = *reinterpret_cast<const vec2*>(fr + (loc.z & 0xffff));
            mel[0][f] += sn.x; mel[1][f] += sn.y; mel[2][f] += fr[loc.z >> 16];
        }
    }
    const int nvalid = T - t0 < F4 ? T - t0 : F4;   // >= 1
    int off;
    bool store = true;
    if (out.layout == 0) {
        const int sl = t0 / SPSS, tt = t0 - sl * SPSS;
        off = (sl * NMEL + m) * SPSS + tt + f0;
        store = sl < out.n_slices;
    } else {
        off = m * out.ld_t + t0 + f0;
    }
#pragma unroll
    for (int sig = 0; sig < 3; ++sig) {
        const float scale = sig == 1 ? factor : 1.0f;
        float d[2];
        float lm = neg_inf(), ln = -neg_inf();
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            d[f] = amp_to_db(mel[sig][f] * scale);
            const bool v = f0 + f < nvalid;
            lm = v ? fmaxf(lm, d[f]) : lm;
            ln = v ? fminf(ln, d[f]) : ln;
        }
        mx[sig] = fmaxf(lm, mx[sig]);
        float* dst = out.dst[sig];
        mn[32 * sig + lane] = fminf(mn[32 * sig + lane], (dst != nullptr && store) ? ln : -neg_inf());
        if (dst != nullptr && store) {
            if (out.layout == 0) {
                vec2 o; o.x = d[0]; o.y = d[1];
                *reinterpret_cast<vec2*>(dst + off) = o;     // 8-byte aligned: off % 2 == 0
            } else {
#pragma unroll
                for (int f = 0; f < 2; ++f)
                    if (f0 + f < nvalid) dst[off + f] = d[f];
            }
        }
    }
}

}  // namespace avse
