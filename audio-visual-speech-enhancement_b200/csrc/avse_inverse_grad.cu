// Backward of the inverse path: dL/d dB of the mixture-phase reconstruction.  See include/avse_b200.h (avse_inverse_backward)
// and avse_inverse_grad_stages.cuh.
#include <cuda_runtime.h>
#include <string>

#include "../../include/avse_b200.h"
#include "avse_common.h"
#include "avse_ctx.h"
#include "avse_inverse_grad_stages.cuh"

using namespace avse;

constexpr int IG_WARPS = 8;
constexpr int IG_THREADS = IG_WARPS * 32;
constexpr int IG_SM_WIN = IG_WARPS * IG_WARP_F;        // [640] window
constexpr int IG_SM_TW = IG_SM_WIN + NFFT;             // [16][40] (re, im) W_640^{b c}
constexpr int IG_SM_MELW = IG_SM_TW + 2 * N1 * N2;     // [80][MEL_WROW] 0.5 F, banded
constexpr int IG_SM_MELLO = IG_SM_MELW + NMEL * MEL_WROW;   // [80] first bin of each band
constexpr int IG_SM_TRI = IG_SM_MELLO + NMEL;          // [3][80] Thomas factors of F F^T (w, 1 / pivot, super-diagonal)
constexpr int IG_SMEM_F = IG_SM_TRI + 3 * NMEL;
constexpr int IG_SMEM_BYTES = IG_SMEM_F * 4;
static_assert((IG_WARP_F % 4) == 0 && (IG_SM_TW % 2) == 0, "alignment");
static_assert(IG_SMEM_BYTES + 1024 <= 232448, "IG shared memory must fit in one SM");

struct GradParams {
    avse_inverse_args a;
    const float* grad;        // [B][grad_stride]
    long long grad_stride;
    float* grad_mel;          // mel_db's layout
    const float* window;
    const float* tw1t;
    const float* mel_w;
    const int* mel_lo;
    const float* tri_w;
    const float* tri_ipiv;
    const float* tri_sup;
    int T_use;
    int t_write;              // frames of grad_mel written: every frame the layout holds (zeros from T_use on)
    int chunks;               // chunks of IG_FPC frames per utterance
    int out_len;
};

__device__ __forceinline__ float ig_warp_sum(float v) {      // fixed butterfly order: deterministic
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(IG_THREADS, 1) avse_inverse_grad_kernel(const __grid_constant__ GradParams P) {
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < NFFT; i += IG_THREADS) smem[IG_SM_WIN + i] = P.window[i];
    for (int i = threadIdx.x; i < 2 * N1 * N2; i += IG_THREADS) smem[IG_SM_TW + i] = P.tw1t[i];
    for (int i = threadIdx.x; i < NMEL * MEL_WROW; i += IG_THREADS) smem[IG_SM_MELW + i] = P.mel_w[i];
    for (int i = threadIdx.x; i < NMEL; i += IG_THREADS) {
        reinterpret_cast<int*>(smem + IG_SM_MELLO)[i] = P.mel_lo[i];
        smem[IG_SM_TRI + i] = P.tri_w[i];
        smem[IG_SM_TRI + NMEL + i] = P.tri_ipiv[i];
        smem[IG_SM_TRI + 2 * NMEL + i] = P.tri_sup[i];
    }
    float* fr = smem + warp * IG_WARP_F;
    float* d = fr + IG_FR_F;
    float* fd = d + IG_D_F;
    for (int i = lane; i < IG_D_F; i += 32) d[i] = 0.0f;
    __syncthreads();
    const float* s_win = smem + IG_SM_WIN;
    const float* s_tw = smem + IG_SM_TW;
    const float* s_melw = smem + IG_SM_MELW;
    const int* s_mello = reinterpret_cast<const int*>(smem + IG_SM_MELLO);
    const float* s_tri = smem + IG_SM_TRI;
    const avse_inverse_args& A = P.a;

    const long long items = (long long)A.B * P.chunks;
#pragma unroll 1
    for (long long item = (long long)blockIdx.x * IG_WARPS + warp; item < items; item += (long long)gridDim.x * IG_WARPS) {
        const int u = (int)(item / P.chunks);
        const int t0 = (int)(item - (long long)u * P.chunks) * IG_FPC;
        const int nf = P.t_write - t0 < IG_FPC ? P.t_write - t0 : IG_FPC;
        const int n_use = P.T_use - t0 < nf ? P.T_use - t0 : nf;
        GradFrame f;
        f.pcm = A.mixed_pcm + (size_t)u * A.pcm_stride;
        f.L = A.L;
        const int valid = A.len_pcm ? A.len_pcm[u] : A.L;
        f.valid = valid < 0 ? 0 : (valid < A.L ? valid : A.L);
        f.grad = P.grad + (size_t)u * P.grad_stride;
        f.out_len = P.out_len;
        f.T_use = P.T_use;
#pragma unroll 1
        for (int j = 0; j < n_use; ++j) {
            float* fdj = fd + j * IG_FD_ROW;
            float hg[IG_SPL], hm[IG_SPL];
            unsigned ag, am;
            ig_load(f, t0 + j, lane, s_win, hg, hm, ag, am);
            ag = __reduce_max_sync(0xffffffffu, ag);
            am = __reduce_max_sync(0xffffffffu, am);
            if (ag == 0u) {                       // no gradient reaches this frame: exact zeros
                for (int m = lane; m < NMEL; m += 32) fdj[m] = 0.0f;
                continue;
            }
            const bool mix_any = am != 0u;
            const int eg = ig_exp_of_bits(ag), em = ig_exp_of_bits(am);
            float pg, pm;
            ig_power(hg, hm, eg, em, pg, pm);
            pg = ig_warp_sum(pg);
            pm = ig_warp_sum(pm);
            const int e = ig_scale_exp(eg, em, pg, pm, mix_any);
            ig_pack(lane, hg, hm, ig_pow2(e), fr);
            __syncwarp();
            ig_pass1(lane, s_tw, fr);
            if (lane < N2 - 32) ig_pass1(32 + lane, s_tw, fr);
            __syncwarp();
            {
                cpx x[40];
                if (lane < N1) ig_pass2_load(lane, fr, x);
                __syncwarp();
                if (lane < N1) ig_pass2_store(lane, x, fr);
            }
            __syncwarp();
            ig_post(lane, fr, ig_pow2(-e), mix_any, d);
            __syncwarp();
            ig_mel(lane, s_melw, s_mello, d, fdj);
            __syncwarp();
        }
        __syncwarp();
        if (lane < nf)
            ig_solve(fd + lane * IG_FD_ROW, t0 + lane, P.T_use, A.mel_db + (size_t)u * A.mel_stride,
                     P.grad_mel + (size_t)u * A.mel_stride, A.layout, A.ld_t, s_tri);
        __syncwarp();
    }
}

extern "C" int avse_inverse_backward(avse_ctx* ctx, const avse_inverse_args* args, const float* grad_pcm, long long grad_pcm_stride,
                                     float* grad_mel, void* stream) {
    if (!ctx || !args) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: NULL argument");
    const avse_inverse_args& a = *args;
    if (a.phase) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: only the mixture-phase form (phase == NULL) is differentiable");
    if (a.out_format != AVSE_SAMPLE_F32) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: out_format must be AVSE_SAMPLE_F32");
    if (!a.mel_db || !a.mixed_pcm || !grad_pcm || !grad_mel) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: NULL buffer");
    const int n_fft = ctx->generic ? ctx->gen.geo.n_fft : NFFT;
    if (a.B <= 0 || a.L <= n_fft / 2) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: need B > 0 and L > n_fft / 2");
    if (a.layout != AVSE_LAYOUT_SLICES && a.layout != AVSE_LAYOUT_SPEC) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: bad layout");
    const int T = ctx->generic ? avse_generic_frames(ctx->gen.geo, a.L) : 1 + a.L / HOP;
    const int spss = ctx->generic ? ctx->gen.geo.spss : SPSS;
    const int t_mel = a.layout == AVSE_LAYOUT_SLICES ? a.n_slices * spss : a.n_frames;
    if (t_mel <= 0) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: no mel frames");
    const int T_use = t_mel < T ? t_mel : T;
    if (T_use < 2) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: fewer than 2 frames gives an empty signal");
    if (a.layout == AVSE_LAYOUT_SPEC && a.ld_t < T_use) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: ld_t < frames used");
    const int hop = ctx->generic ? ctx->gen.geo.hop : HOP;
    const int out_len = hop * (T_use - 1);
    if (a.B > 1 && grad_pcm_stride < out_len) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: grad_pcm_stride < hop (T_use - 1)");
    if (!a.len_pcm && a.pcm_stride < a.L) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: pcm_stride < L needs len_pcm");
    // SPEC: columns [0, min(n_frames, ld_t)) are written, [n_frames, ld_t) left alone
    const int t_write = a.layout == AVSE_LAYOUT_SPEC ? (t_mel < a.ld_t ? t_mel : a.ld_t) : t_mel;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != ctx->device) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: current device differs from the context's device");
    if (ctx->generic) return avse_generic_inverse_backward(ctx, args, T_use, t_write, grad_pcm, grad_pcm_stride, grad_mel, stream);

    GradParams P;
    P.a = a;
    P.grad = grad_pcm;
    P.grad_stride = grad_pcm_stride;
    P.grad_mel = grad_mel;
    P.window = ctx->fwd.window;
    P.tw1t = ctx->fwd.tw1t;
    P.mel_w = ctx->fwd.mel_w;
    P.mel_lo = ctx->fwd.mel_lo;
    P.tri_w = ctx->d_tri_w;
    P.tri_ipiv = ctx->d_tri_ipiv;
    P.tri_sup = ctx->d_tri_sup;
    P.T_use = T_use;
    P.t_write = t_write;
    P.chunks = (t_write + IG_FPC - 1) / IG_FPC;
    P.out_len = out_len;
    static thread_local int configured_dev = -1;
    if (configured_dev != dev) {
        CUDA_TRY(cudaFuncSetAttribute(avse_inverse_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, IG_SMEM_BYTES));
        configured_dev = dev;
    }
    const long long items = (long long)a.B * P.chunks;
    long long blocks = (items + IG_WARPS - 1) / IG_WARPS;
    if (blocks > ctx->num_sms) blocks = ctx->num_sms;
    avse_inverse_grad_kernel<<<(unsigned)blocks, IG_THREADS, IG_SMEM_BYTES, (cudaStream_t)stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return 0;
}
