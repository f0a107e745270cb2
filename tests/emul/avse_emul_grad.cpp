// Host emulation of the inverse's backward kernel (avse_inverse_grad_kernel), TEST INFRASTRUCTURE, not a product path:
// csrc/avse_inverse_grad_stages.cuh compiled with g++, one warp run as a loop over 32 lanes per stage, the warp reductions
// restated in the kernel's order (xor butterfly), frames in chunks of IG_FPC like a warp's items.
#include <cstring>
#include <vector>
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_common.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_tables.h"
#include "../../audio-visual-speech-enhancement_b200/csrc/avse_inverse_grad_stages.cuh"

using namespace avse;

namespace {

float warp_sum(const float (&v)[32]) {
    float a[32];
    std::memcpy(a, v, sizeof(a));
    for (int o = 16; o > 0; o >>= 1) {
        float b[32];
        for (int l = 0; l < 32; ++l) b[l] = a[l] + a[l ^ o];
        std::memcpy(a, b, sizeof(a));
    }
    return a[0];
}

}  // namespace

// layout 0: SLICES [n_slices][80][20]; 1: SPEC [80][ld_t] with n_frames columns.  grad: [160 (T_use - 1)].  grad_mel: mel's
// layout; only the elements the kernel stores are written.  Returns T_use, or < 0 on a bad configuration.
extern "C" int emul_inverse_backward(const float* mel, int layout, int n_slices, int n_frames, int ld_t, const float* pcm, int L, int valid,
                                     const float* grad, float* grad_mel, int sample_rate, double fmin, double fmax) {
    HostTables h;
    if (!build_tables(h, sample_rate, fmin, fmax)) return -2;
    const int T = 1 + L / HOP;
    const int t_mel = layout == 0 ? n_slices * SPSS : n_frames;
    const int T_use = t_mel < T ? t_mel : T;
    if (T_use < 2) return -1;
    const int t_write = layout == 1 ? (t_mel < ld_t ? t_mel : ld_t) : t_mel;
    std::vector<float> tri(3 * NMEL);
    for (int m = 0; m < NMEL; ++m) { tri[m] = h.tri_w[m]; tri[NMEL + m] = h.tri_ipiv[m]; tri[2 * NMEL + m] = h.tri_sup[m]; }
    const float* s_win = h.window.data();
    const float* s_tw = h.tw1t.data();

    static float buf[IG_WARP_F];
    std::memset(buf, 0, sizeof(buf));
    float* fr = buf;
    float* d = fr + IG_FR_F;
    float* fd = d + IG_D_F;
    GradFrame f;
    f.pcm = pcm; f.L = L; f.valid = valid < L ? valid : L; f.grad = grad; f.out_len = HOP * (T_use - 1); f.T_use = T_use;
    static float hg[32][IG_SPL], hm[32][IG_SPL];
    static cpx x[32][40];
    for (int t0 = 0; t0 < t_write; t0 += IG_FPC) {
        const int nf = t_write - t0 < IG_FPC ? t_write - t0 : IG_FPC;
        const int n_use = T_use - t0 < nf ? T_use - t0 : nf;
        for (int j = 0; j < n_use; ++j) {
            float* fdj = fd + j * IG_FD_ROW;
            unsigned ag = 0, am = 0;
            for (int l = 0; l < 32; ++l) {
                unsigned a, b;
                ig_load(f, t0 + j, l, s_win, hg[l], hm[l], a, b);
                ag = a > ag ? a : ag;
                am = b > am ? b : am;
            }
            if (ag == 0u) {
                for (int m = 0; m < NMEL; ++m) fdj[m] = 0.0f;
                continue;
            }
            const bool mix_any = am != 0u;
            const int eg = ig_exp_of_bits(ag), em = ig_exp_of_bits(am);
            float pg[32], pm[32];
            for (int l = 0; l < 32; ++l) ig_power(hg[l], hm[l], eg, em, pg[l], pm[l]);
            const int e = ig_scale_exp(eg, em, warp_sum(pg), warp_sum(pm), mix_any);
            for (int l = 0; l < 32; ++l) ig_pack(l, hg[l], hm[l], ig_pow2(e), fr);
            for (int b = 0; b < N2; ++b) ig_pass1(b, s_tw, fr);
            for (int c = 0; c < N1; ++c) ig_pass2_load(c, fr, x[c]);
            for (int c = 0; c < N1; ++c) ig_pass2_store(c, x[c], fr);
            for (int l = 0; l < 32; ++l) ig_post(l, fr, ig_pow2(-e), mix_any, d);
            for (int l = 0; l < 32; ++l) ig_mel(l, h.mel_w.data(), h.mel_lo.data(), d, fdj);
        }
        for (int l = 0; l < nf; ++l) ig_solve(fd + l * IG_FD_ROW, t0 + l, T_use, mel, grad_mel, layout, ld_t, tri.data());
    }
    return T_use;
}
