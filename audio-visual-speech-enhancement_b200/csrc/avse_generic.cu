// Generic-geometry kernels (any n_fft / hop / n_mels / frames per slice): the correct-but-slower fallback behind the same
// C ABI as the specialised 640 / 160 path.  See avse_generic.h and include/avse_b200.h (avse_create_ex).
//
// Reference semantics: /root/reference/data_processor.py:35-139 with n_fft = int(sr / fps), hop = int(n_fft / 4)
// (dp:44-45); library semantics as in SURVEY.md Appendix A (librosa.stft center/reflect, magphase, filters.mel,
// amplitude_to_db, db_to_amplitude, np.linalg.pinv, librosa.istft with n_fft inferred as 2 (rows - 1)).
#include <cuda_runtime.h>
#include <string>

#include "../../include/avse_b200.h"
#include "avse_common.h"
#include "avse_ctx.h"

using namespace avse;

namespace avse_gen {

constexpr int GEN_THREADS = 256;

struct GenFwdParams {
    avse_forward_args a;
    GenericGeo geo;
    GenericDev d;
    int T;          // frames: 1 + (L + 2 (n_fft / 2) - n_fft) / hop
    PoolRows pool;  // avse_mix_pooled: row indirection into a.speech / a.noise (speech_index == nullptr otherwise)
};

struct GenInvParams {
    avse_inverse_args a;
    GenericGeo geo;
    GenericDev d;
    int T;          // mixture STFT frames (or phase_frames)
    int T_use;      // frames reconstructed (dp:68)
    int out_len;    // hop (T_use - 1)
};

template <typename S>
__device__ __forceinline__ float gen_sample(const S* p, int i, int L, int valid, int period = 0, int phase = 0) {
    // np.pad(y, n_fft // 2, mode='reflect') on the length-L (zero padded, dp:40) signal; period > 0: the signal is the
    // periodic tiling p[(phase + i) mod period] of a shorter noise file (dp:125-128; phase != 0: pooled pairs)
    i = i < 0 ? -i : i;
    i = i >= L ? 2 * (L - 1) - i : i;
    i = i < 0 ? 0 : i;
    if (p == nullptr || i >= valid) return 0.0f;
    return (float)p[period > 0 ? (i + phase) % period : i];
}

// out[k1 + n1 k2] = sum_n in[n] W^{n k},  n = n2 a + c2.  `out` may alias `in`; tmp is scratch (shared memory).
// Float64 data, twiddles (global table, L1/L2 resident) and accumulation: this path is the accuracy-first fallback, and
// in float32 the packed transform z = s + i n lets noise-level rounding leak into quiet speech bins (2e-3 dB at
// n_fft = 666 against the 1e-3 dB gate).
__device__ void gen_dft(const double2* in, double2* tmp, double2* out, const double2* __restrict__ W, int N, int n1, int n2) {
    for (int idx = threadIdx.x; idx < N; idx += blockDim.x) {
        const int k1 = idx / n2, c2 = idx - k1 * n2;
        const int step = (int)(((long long)n2 * k1) % N);
        int e = 0;
        double ar = 0.0, ai = 0.0;
        for (int a = 0; a < n1; ++a) {
            const double2 x = in[n2 * a + c2];
            const double2 w = __ldg(W + e);
            ar = fma(x.x, w.x, fma(-x.y, w.y, ar));
            ai = fma(x.x, w.y, fma(x.y, w.x, ai));
            e += step;
            if (e >= N) e -= N;
        }
        const double2 w = __ldg(W + (int)(((long long)c2 * k1) % N));
        tmp[idx] = make_double2(ar * w.x - ai * w.y, ar * w.y + ai * w.x);
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < N; idx += blockDim.x) {
        const int k2 = idx / n1, k1 = idx - k2 * n1;
        const int step = (int)(((long long)n1 * k2) % N);
        int e = 0;
        double ar = 0.0, ai = 0.0;
        const double2* row = tmp + k1 * n2;
        for (int c2 = 0; c2 < n2; ++c2) {
            const double2 x = row[c2];
            const double2 w = __ldg(W + e);
            ar = fma(x.x, w.x, fma(-x.y, w.y, ar));
            ai = fma(x.x, w.y, fma(x.y, w.x, ai));
            e += step;
            if (e >= N) e -= N;
        }
        out[idx] = make_double2(ar, ai);
    }
    __syncthreads();
}

__device__ __forceinline__ int gen_key(float x) {
    const int b = __float_as_int(x);
    return b >= 0 ? b : (b ^ 0x7fffffff);
}

// ---------------------------------------------------------------------------------------------
// forward: one CTA per (frame, utterance)
// ---------------------------------------------------------------------------------------------
template <typename S>
__global__ void __launch_bounds__(GEN_THREADS) avse_generic_forward_kernel(const __grid_constant__ GenFwdParams P) {
    extern __shared__ __align__(16) unsigned char gsm[];
    const GenericGeo& q = P.geo;
    const avse_forward_args& A = P.a;
    const int N = q.n_fft, bins = q.bins, M = q.n_mels;
    double2* X = reinterpret_cast<double2*>(gsm);
    double2* Y = X + N;
    float* mags = reinterpret_cast<float*>(Y + N);        // [3][bins]
    int* keys = reinterpret_cast<int*>(mags + 3 * bins);  // [3] max, [3] min
    const double2* W = reinterpret_cast<const double2*>(P.d.tw);
    const int u = blockIdx.x / P.T, t = blockIdx.x - u * P.T;     // linear (utterance, frame) index: B is not capped at 65 535
    const int tid = threadIdx.x;
    const bool have_noise = A.noise != nullptr;

    int vs, vn, period, phase;
    const S* sp;
    const S* nz;
    if (P.pool.speech_index != nullptr) {     // pooled pair (avse_mix_pooled): rows of the two pools, noise from its phase
        const PoolRow r = pool_row(P.pool, u);
        vs = r.ls < A.L ? r.ls : A.L;
        vn = vs;
        sp = reinterpret_cast<const S*>(A.speech) + r.s_off;
        nz = reinterpret_cast<const S*>(A.noise) + r.n_off;
        period = r.ln;
        phase = r.off;
    } else {
        vs = A.len_speech ? A.len_speech[u] : A.L;
        vn = A.len_noise ? A.len_noise[u] : vs;
        vs = vs < 0 ? 0 : (vs < A.L ? vs : A.L);
        vn = vn < 0 ? 0 : (vn < A.L ? vn : A.L);
        period = (have_noise && A.noise_period) ? A.noise_period[u] : 0;
        phase = 0;
        sp = reinterpret_cast<const S*>(A.speech) + (size_t)u * A.in_stride;
        nz = have_noise ? reinterpret_cast<const S*>(A.noise) + (size_t)u * A.in_stride : nullptr;
    }
    fit_noise_row(nz, period, phase, vn);          // a window that does not wrap is a contiguous row, read with no modulo
    // the whole SNR factor is applied after the transform: this path computes in float64, where the level equaliser of the
    // float32 kernels (avse_forward_args::equalizer) is not needed
    const float factor = have_noise ? (A.factor ? A.factor[u] : 1.0f) : 0.0f;

    if (tid < 3) { keys[tid] = (int)0x80000000; keys[3 + tid] = 0x7fffffff; }
    const int base = t * q.hop - N / 2;
    for (int n = tid; n < N; n += GEN_THREADS) {
        const double w = P.d.window[n];
        X[n] = make_double2(gen_sample(sp, base + n, A.L, vs) * w, gen_sample(nz, base + n, A.L, vn, period, phase) * w);
    }
    if (A.mixed_pcm != nullptr && have_noise) {     // this frame's own hop of s + f n (dp:133), zero padded / truncated to L
        float* pm = A.mixed_pcm + (size_t)u * A.pcm_stride;
        const int hi = (t + 1) * q.hop < A.L ? (t + 1) * q.hop : A.L;
        for (int i = t * q.hop + tid; i < hi; i += GEN_THREADS)
            pm[i] = (i < vs ? (float)sp[i] : 0.0f) + factor * (i < vn ? (float)nz[period > 0 ? (i + phase) % period : i] : 0.0f);
    }
    __syncthreads();
    gen_dft(X, Y, X, W, N, q.n1, q.n2);

    // unpack the packed transform z = s + i n (S = Z itself for a single real signal), magnitudes of the three signals
    float2* stft_row = A.stft_speech ? reinterpret_cast<float2*>(A.stft_speech) + ((size_t)u * P.T + t) * bins : nullptr;
    for (int k = tid; k < bins; k += GEN_THREADS) {
        const double2 a = X[k];
        const double2 c = X[k == 0 ? 0 : N - k];
        const double2 s = make_double2(0.5 * (a.x + c.x), 0.5 * (a.y - c.y));     // speech spectrum (== a for a single real signal)
        float mn = 0.0f, mm = 0.0f;
        if (have_noise) {
            const double2 n = make_double2(0.5 * (a.y + c.y), 0.5 * (c.x - a.x));
            const double f = (double)factor;
            mn = (float)(fabs(f) * hypot(n.x, n.y));
            mm = (float)hypot(fma(f, n.x, s.x), fma(f, n.y, s.y));
        }
        mags[k] = (float)hypot(s.x, s.y);
        mags[bins + k] = mn;
        mags[2 * bins + k] = mm;
        if (stft_row != nullptr) stft_row[k] = make_float2((float)s.x, (float)s.y);
    }
    __syncthreads();

    // mel projection (dp:91), amplitude_to_db without its top_db clip (dp:94), running extrema, store
    const int sl = t / q.spss, tt = t - sl * q.spss;
    for (int idx = tid; idx < 3 * M; idx += GEN_THREADS) {
        const int sig = idx / M, m = idx - sig * M;
        if (sig > 0 && !have_noise) continue;
        float* dst = sig == 0 ? A.out_speech : (sig == 1 ? A.out_noise : A.out_mixed);
        const float* mg = mags + sig * bins + P.d.band_lo[m];
        const float* w = P.d.band_w + P.d.band_off[m];
        const int cnt = P.d.band_cnt[m];
        float acc = 0.0f;
        for (int j = 0; j < cnt; ++j) acc = fmaf(w[j], mg[j], acc);
        const float db = 20.0f * log10f(fmaxf(acc, AMIN));
        atomicMax(&keys[sig], gen_key(db));
        if (dst == nullptr) continue;
        if (A.layout == AVSE_LAYOUT_SLICES) {
            if (sl >= A.n_slices) continue;
            dst[(size_t)u * A.out_stride + ((size_t)sl * M + m) * q.spss + tt] = db;
        } else {
            dst[(size_t)u * A.out_stride + (size_t)m * A.ld_t + t] = db;
        }
        atomicMin(&keys[3 + sig], gen_key(db));
    }
    __syncthreads();
    if (tid < 3 && (tid == 0 || have_noise)) {
        atomicMax(A.max_key + 3 * u + tid, keys[tid]);
        if (A.min_key) atomicMin(A.min_key + 3 * u + tid, keys[3 + tid]);
    }
}

// ---------------------------------------------------------------------------------------------
// inverse, kernel 1: one CTA per (frame, utterance): lin = pinv(F) 10^(dB/20), phase of the mixture's STFT frame (or the
// caller's phase), irfft, window -> work[u][t][n_inv]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(GEN_THREADS) avse_generic_inverse_frame_kernel(const __grid_constant__ GenInvParams P) {
    extern __shared__ __align__(16) unsigned char gsm[];
    const GenericGeo& q = P.geo;
    const avse_inverse_args& A = P.a;
    const int N = q.n_fft, Ni = q.n_inv, bins = q.bins, M = q.n_mels;
    const int NX = N > Ni ? N : Ni;
    double2* X = reinterpret_cast<double2*>(gsm);
    double2* Y = X + NX;
    float* amp = reinterpret_cast<float*>(Y + NX);   // [n_mels]
    float* lin = amp + M;                            // [bins]
    const double2* W = reinterpret_cast<const double2*>(P.d.tw);
    const double2* Wi = reinterpret_cast<const double2*>(P.d.tw_inv);
    const int u = blockIdx.x / P.T_use, t = blockIdx.x - u * P.T_use;
    const int tid = threadIdx.x;

    // db_to_amplitude (dp:101)
    const float* mel = A.mel_db + (size_t)u * A.mel_stride;
    constexpr float K = 0.16609640474436813f;   // log2(10) / 20
    for (int m = tid; m < M; m += GEN_THREADS) {
        float db;
        if (A.layout == AVSE_LAYOUT_SLICES) {
            const int sl = t / q.spss, tt = t - sl * q.spss;
            db = mel[((size_t)sl * M + m) * q.spss + tt];
        } else {
            db = mel[(size_t)m * A.ld_t + t];
        }
        amp[m] = exp2f(K * db);
    }
    const bool ext = A.phase != nullptr;
    if (!ext) {
        int valid = A.len_pcm ? A.len_pcm[u] : A.L;
        valid = valid < A.L ? valid : A.L;
        const float* pcm = A.mixed_pcm + (size_t)u * A.pcm_stride;
        const int base = t * q.hop - N / 2;
        for (int n = tid; n < N; n += GEN_THREADS) X[n] = make_double2((double)gen_sample(pcm, base + n, A.L, valid) * (double)P.d.window[n], 0.0);
    }
    __syncthreads();
    // np.dot(pinv(fb), magnitude) (dp:112): no clamp, may be negative
    for (int k = tid; k < bins; k += GEN_THREADS) {
        const float* row = P.d.pinv + (size_t)k * M;
        float acc = 0.0f;
        for (int m = 0; m < M; ++m) acc = fmaf(row[m], amp[m], acc);
        lin[k] = acc;
    }
    if (!ext) gen_dft(X, Y, X, W, N, q.n1, q.n2);      // ends with a barrier
    else __syncthreads();

    // Y = lin * phase; Hermitian extension for irfft(n = n_inv): conj(V) goes through the forward transform
    const float2* ph = ext ? reinterpret_cast<const float2*>(A.phase) + (size_t)u * A.phase_stride + (size_t)t * bins : nullptr;
    double2* V = ext ? X : Y;       // !ext: X holds the mixture spectrum, build V in Y
    for (int k = tid; k < bins; k += GEN_THREADS) {
        double px, py;
        if (ext) {
            const float2 p = ph[k];
            px = p.x; py = p.y;
        } else {
            const double2 z = X[k];
            const double r = hypot(z.x, z.y);
            if (r > 0.0) { px = z.x / r; py = z.y / r; }        // magphase (dp:80): D / |D|
            else { px = 1.0; py = 0.0; }                        // 1 + 0j where D == 0
        }
        const double l = (double)lin[k];
        const double yx = l * px;
        const double yy = (k == 0 || 2 * k == Ni) ? 0.0 : l * py;   // C2R transforms ignore the imaginary part of DC / Nyquist
        V[k] = make_double2(yx, -yy);                               // conj(V[k])
        if (k > 0 && 2 * k != Ni) V[Ni - k] = make_double2(yx, yy); // conj(V[N - k]) = Y[k]
    }
    __syncthreads();
    double2* O = ext ? Y : X;
    gen_dft(V, O, V, Wi, Ni, q.i1, q.i2);     // y[n] = Re(.) / n_inv
    float* dst = A.work + (size_t)u * A.work_stride + (size_t)t * Ni;
    const double sc = 1.0 / (double)Ni;
    for (int n = tid; n < Ni; n += GEN_THREADS) dst[n] = (float)(V[n].x * sc * (double)P.d.window_inv[n]);
}

__device__ __forceinline__ void gen_store(float* p, float v) { *p = v; }
__device__ __forceinline__ void gen_store(short* p, float v) {
    v = v < -32768.0f ? -32768.0f : (v > 32767.0f ? 32767.0f : v);
    *p = (short)(int)v;
}

// inverse, kernel 2: overlap-add as a gather (each output sample sums the <= ceil(n_inv / hop) frames covering it),
// window sum-square normalisation where > tiny(float32), centre trim (librosa.istft, dp:114).
template <typename O>
__global__ void __launch_bounds__(256) avse_generic_inverse_ola_kernel(const __grid_constant__ GenInvParams P) {
    const GenericGeo& q = P.geo;
    const int u = blockIdx.x;
    const int Ni = q.n_inv, hop = q.hop;
    const float* w = P.a.work + (size_t)u * P.a.work_stride;
    O* out = static_cast<O*>(P.a.out_pcm) + (size_t)u * P.a.out_stride;
    for (int o = blockIdx.y * blockDim.x + threadIdx.x; o < P.out_len; o += gridDim.y * blockDim.x) {
        const int pp = o + Ni / 2;
        int t_hi = pp / hop;
        if (t_hi > P.T_use - 1) t_hi = P.T_use - 1;
        int t_lo = (pp - Ni + hop) / hop;       // ceil((pp - Ni + 1) / hop) for pp - Ni + 1 > 0
        if (pp - Ni + 1 <= 0) t_lo = 0;
        float acc = 0.0f, wss = 0.0f;
        for (int t = t_lo; t <= t_hi; ++t) {
            const int n = pp - t * hop;
            acc += w[(size_t)t * Ni + n];
            const float wn = P.d.window_inv[n];
            wss = fmaf(wn, wn, wss);
        }
        gen_store(out + o, wss > 1.17549435e-38f ? acc / wss : acc);
    }
}

// ---------------------------------------------------------------------------------------------
// inverse backward: one CTA per (frame, utterance) of grad_mel.  dL/d dB_t = ln(10)/20 a_t pinv(F)^T d_t with
// d_t[k] = (c_k / n_inv) Re(conj(phi_t[k]) rfft_{n_inv}(w_inv e_t)[k]) (avse_inverse_grad_stages.cuh); float64 transforms
// and accumulation.  Frames t >= T_use get exact zeros.
// ---------------------------------------------------------------------------------------------
struct GenGradParams {
    avse_inverse_args a;
    GenericGeo geo;
    GenericDev d;
    const float* grad;
    long long grad_stride;
    float* grad_mel;
    int T_use;
    int t_write;
    int out_len;
};

__global__ void __launch_bounds__(GEN_THREADS) avse_generic_inverse_grad_kernel(const __grid_constant__ GenGradParams P) {
    extern __shared__ __align__(16) unsigned char gsm[];
    const GenericGeo& q = P.geo;
    const avse_inverse_args& A = P.a;
    const int N = q.n_fft, Ni = q.n_inv, bins = q.bins, M = q.n_mels, hop = q.hop;
    const int NX = N > Ni ? N : Ni;
    double2* X = reinterpret_cast<double2*>(gsm);
    double2* Y = X + NX;
    double2* phi = Y + NX;                               // [bins]
    double* dk = reinterpret_cast<double*>(Y);           // [bins], once Y is free
    const int u = blockIdx.x / P.t_write, t = blockIdx.x - u * P.t_write;
    const int tid = threadIdx.x;
    size_t base, mstride;
    if (A.layout == AVSE_LAYOUT_SLICES) {
        const int sl = t / q.spss, tt = t - sl * q.spss;
        base = (size_t)sl * M * q.spss + tt;
        mstride = q.spss;
    } else {
        base = t;
        mstride = A.ld_t;
    }
    float* gout = P.grad_mel + (size_t)u * A.mel_stride + base;
    if (t >= P.T_use) {
        for (int m = tid; m < M; m += GEN_THREADS) gout[(size_t)m * mstride] = 0.0f;
        return;
    }
    // phase of the mixture's STFT frame (magphase, dp:80)
    int valid = A.len_pcm ? A.len_pcm[u] : A.L;
    valid = valid < A.L ? valid : A.L;
    const float* pcm = A.mixed_pcm + (size_t)u * A.pcm_stride;
    const int mbase = t * hop - N / 2;
    for (int n = tid; n < N; n += GEN_THREADS) X[n] = make_double2((double)gen_sample(pcm, mbase + n, A.L, valid) * (double)P.d.window[n], 0.0);
    __syncthreads();
    gen_dft(X, Y, X, reinterpret_cast<const double2*>(P.d.tw), N, q.n1, q.n2);
    for (int k = tid; k < bins; k += GEN_THREADS) {
        const double2 z = X[k];
        const double r = hypot(z.x, z.y);
        phi[k] = r > 0.0 ? make_double2(z.x / r, z.y / r) : make_double2(1.0, 0.0);
    }
    __syncthreads();
    // the gradient frame: e = g at offset n_inv / 2 of the untrimmed signal, / window sum-square where > tiny(float32)
    const float* g = P.grad + (size_t)u * P.grad_stride;
    for (int n = tid; n < Ni; n += GEN_THREADS) {
        const int pp = t * hop + n, o = pp - Ni / 2;
        double e = 0.0;
        if (o >= 0 && o < P.out_len) {
            int t_hi = pp / hop;
            if (t_hi > P.T_use - 1) t_hi = P.T_use - 1;
            const int t_lo = pp - Ni + 1 <= 0 ? 0 : (pp - Ni + hop) / hop;
            float wss = 0.0f;                               // as the forward's overlap-add computes it
            for (int s = t_lo; s <= t_hi; ++s) {
                const float wn = P.d.window_inv[pp - s * hop];
                wss = fmaf(wn, wn, wss);
            }
            e = wss > 1.17549435e-38f ? (double)g[o] / (double)wss : (double)g[o];
        }
        X[n] = make_double2(e * (double)P.d.window_inv[n], 0.0);
    }
    __syncthreads();
    gen_dft(X, Y, X, reinterpret_cast<const double2*>(P.d.tw_inv), Ni, q.i1, q.i2);
    for (int k = tid; k < bins; k += GEN_THREADS) {
        const double2 h = X[k], p = phi[k];
        const bool edge = k == 0 || 2 * k == Ni;            // C2R reads only the real part of DC / Nyquist
        dk[k] = edge ? p.x * h.x / (double)Ni : 2.0 * (p.x * h.x + p.y * h.y) / (double)Ni;
    }
    __syncthreads();
    // pinv(F)^T d, dB chain rule (db_to_amplitude, dp:101)
    const float* mel = A.mel_db + (size_t)u * A.mel_stride + base;
    for (int m = tid; m < M; m += GEN_THREADS) {
        double acc = 0.0;
        for (int k = 0; k < bins; ++k) acc = fma((double)P.d.pinv[(size_t)k * M + m], dk[k], acc);
        const double amp = (double)exp2f(0.16609640474436813f * mel[(size_t)m * mstride]);
        gout[(size_t)m * mstride] = (float)(0.11512925464970229 * amp * acc);
    }
}

constexpr size_t kGenMaxSmem = 227 * 1024;   // opt-in ceiling of sm_100 (n_fft <= 4096 needs <= 157 KB)

size_t gen_fwd_smem(const GenericGeo& q) { return (size_t)q.n_fft * 32 + (size_t)q.bins * 12 + 32; }
size_t gen_inv_smem(const GenericGeo& q) {
    const size_t nx = q.n_fft > q.n_inv ? q.n_fft : q.n_inv;
    return nx * 32 + (size_t)(q.n_mels + q.bins) * 4 + 16;
}
size_t gen_grad_smem(const GenericGeo& q) {
    const size_t nx = q.n_fft > q.n_inv ? q.n_fft : q.n_inv;
    return (2 * nx + (size_t)q.bins) * 16;
}

}  // namespace avse_gen

using namespace avse_gen;

int avse_generic_frames(const avse::GenericGeo& q, int L) { return 1 + (L + 2 * (q.n_fft / 2) - q.n_fft) / q.hop; }

int avse_generic_forward(avse_ctx* ctx, const avse_forward_args* args, const PoolRows* pool, void* stream) {
    const avse_forward_args& a = *args;
    const GenericGeo& q = ctx->gen.geo;
    if (!a.speech || !a.max_key) return avse_fail(AVSE_E_ARG, "avse_forward: speech and max_key are required");
    if (a.B <= 0 || a.L <= q.n_fft / 2) return avse_fail(AVSE_E_ARG, "avse_forward: need B > 0 and L > n_fft / 2 (reflect padding)");
    if (!pool && !a.len_speech && a.in_stride < a.L) return avse_fail(AVSE_E_ARG, "avse_forward: in_stride < L needs len_speech");
    if (a.layout != AVSE_LAYOUT_SLICES && a.layout != AVSE_LAYOUT_SPEC) return avse_fail(AVSE_E_ARG, "avse_forward: bad layout");
    if (a.sample_format != AVSE_SAMPLE_F32 && a.sample_format != AVSE_SAMPLE_I16) return avse_fail(AVSE_E_ARG, "avse_forward: bad sample_format");
    GenFwdParams P;
    P.a = a;
    P.geo = q;
    P.d = ctx->gd;
    P.T = avse_generic_frames(q, a.L);
    P.pool = pool ? *pool : PoolRows{};
    if (P.T < 1 || (long long)P.T * a.B > 0x7fffffffLL) return avse_fail(AVSE_E_ARG, "avse_forward: B * frames exceeds 2^31; split the batch");
    if (a.layout == AVSE_LAYOUT_SLICES) {
        if (a.n_slices < 0 || (long long)a.n_slices * q.spss > P.T) return avse_fail(AVSE_E_ARG, "avse_forward: n_slices exceeds int(T / spss) (dp:50)");
        if (a.out_stride < (long long)a.n_slices * q.n_mels * q.spss) return avse_fail(AVSE_E_ARG, "avse_forward: out_stride too small");
    } else {
        if (a.ld_t < P.T) return avse_fail(AVSE_E_ARG, "avse_forward: ld_t < T");
        if (a.out_stride < (long long)q.n_mels * a.ld_t) return avse_fail(AVSE_E_ARG, "avse_forward: out_stride too small");
    }
    if (a.mixed_pcm && a.pcm_stride < a.L) return avse_fail(AVSE_E_ARG, "avse_forward: pcm_stride < L");
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != ctx->device) return avse_fail(AVSE_E_ARG, "avse_forward: current device differs from the context's device");
    const size_t smem = gen_fwd_smem(q);
    if (smem > ctx->gen_fwd_smem_set) {   // the opt-in is per function: only ever raise it (contexts of different geometry coexist)
        CUDA_TRY(cudaFuncSetAttribute(avse_generic_forward_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGenMaxSmem));
        CUDA_TRY(cudaFuncSetAttribute(avse_generic_forward_kernel<short>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGenMaxSmem));
        ctx->gen_fwd_smem_set = kGenMaxSmem;
    }
    dim3 grid((unsigned)((long long)P.T * a.B));
    if (a.sample_format == AVSE_SAMPLE_I16) avse_generic_forward_kernel<short><<<grid, GEN_THREADS, smem, (cudaStream_t)stream>>>(P);
    else avse_generic_forward_kernel<float><<<grid, GEN_THREADS, smem, (cudaStream_t)stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int avse_generic_inverse(avse_ctx* ctx, const avse_inverse_args* args, void* stream) {
    const avse_inverse_args& a = *args;
    const GenericGeo& q = ctx->gen.geo;
    if (!a.mel_db || (!a.mixed_pcm && !a.phase) || !a.out_pcm || !a.work) return avse_fail(AVSE_E_ARG, "avse_inverse: NULL buffer");
    if (a.B <= 0 || (!a.phase && a.L <= q.n_fft / 2)) return avse_fail(AVSE_E_ARG, "avse_inverse: need B > 0 and L > n_fft / 2");
    if (a.layout != AVSE_LAYOUT_SLICES && a.layout != AVSE_LAYOUT_SPEC) return avse_fail(AVSE_E_ARG, "avse_inverse: bad layout");
    if (a.out_format != AVSE_SAMPLE_F32 && a.out_format != AVSE_SAMPLE_I16) return avse_fail(AVSE_E_ARG, "avse_inverse: bad out_format");
    GenInvParams P;
    P.a = a;
    P.geo = q;
    P.d = ctx->gd;
    P.T = a.phase ? a.phase_frames : avse_generic_frames(q, a.L);
    const int t_mel = a.layout == AVSE_LAYOUT_SLICES ? a.n_slices * q.spss : a.n_frames;
    if (t_mel <= 0) return avse_fail(AVSE_E_ARG, "avse_inverse: no mel frames");
    P.T_use = t_mel < P.T ? t_mel : P.T;                       // dp:68
    if (P.T_use < 2) return avse_fail(AVSE_E_ARG, "avse_inverse: fewer than 2 frames gives an empty signal");
    P.out_len = q.hop * (P.T_use - 1) + q.n_inv - 2 * (q.n_inv / 2);
    if (a.layout == AVSE_LAYOUT_SPEC && a.ld_t < P.T_use) return avse_fail(AVSE_E_ARG, "avse_inverse: ld_t < frames used");
    if (a.work_stride < (long long)P.T_use * q.n_inv) return avse_fail(AVSE_E_ARG, "avse_inverse: work_stride too small (see avse_inverse_work_elems_ctx)");
    if (a.out_stride < P.out_len) return avse_fail(AVSE_E_ARG, "avse_inverse: out_stride < hop (T_use - 1)");
    if (a.phase && a.phase_stride < (long long)P.T_use * q.bins) return avse_fail(AVSE_E_ARG, "avse_inverse: phase_stride too small");
    if (!a.phase && !a.len_pcm && a.pcm_stride < a.L) return avse_fail(AVSE_E_ARG, "avse_inverse: pcm_stride < L needs len_pcm");
    if ((long long)P.T_use * a.B > 0x7fffffffLL) return avse_fail(AVSE_E_ARG, "avse_inverse: B * frames exceeds 2^31; split the batch");
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != ctx->device) return avse_fail(AVSE_E_ARG, "avse_inverse: current device differs from the context's device");
    const size_t smem = gen_inv_smem(q);
    if (smem > ctx->gen_inv_smem_set) {
        CUDA_TRY(cudaFuncSetAttribute(avse_generic_inverse_frame_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGenMaxSmem));
        ctx->gen_inv_smem_set = kGenMaxSmem;
    }
    cudaStream_t st = (cudaStream_t)stream;
    avse_generic_inverse_frame_kernel<<<dim3((unsigned)((long long)P.T_use * a.B)), GEN_THREADS, smem, st>>>(P);
    CUDA_TRY(cudaGetLastError());
    long long bx = (P.out_len + 255) / 256;
    if (bx > 1024) bx = 1024;
    if (a.out_format == AVSE_SAMPLE_I16) avse_generic_inverse_ola_kernel<short><<<dim3((unsigned)a.B, (unsigned)bx), 256, 0, st>>>(P);
    else avse_generic_inverse_ola_kernel<float><<<dim3((unsigned)a.B, (unsigned)bx), 256, 0, st>>>(P);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int avse_generic_inverse_backward(avse_ctx* ctx, const avse_inverse_args* args, int T_use, int t_write, const float* grad_pcm,
                                  long long grad_pcm_stride, float* grad_mel, void* stream) {
    const GenericGeo& q = ctx->gen.geo;
    GenGradParams P;
    P.a = *args;
    P.geo = q;
    P.d = ctx->gd;
    P.grad = grad_pcm;
    P.grad_stride = grad_pcm_stride;
    P.grad_mel = grad_mel;
    P.T_use = T_use;
    P.t_write = t_write;
    P.out_len = q.hop * (T_use - 1);
    if ((long long)t_write * args->B > 0x7fffffffLL) return avse_fail(AVSE_E_ARG, "avse_inverse_backward: B * frames exceeds 2^31; split the batch");
    const size_t smem = gen_grad_smem(q);
    if (smem > ctx->gen_grad_smem_set) {
        CUDA_TRY(cudaFuncSetAttribute(avse_generic_inverse_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGenMaxSmem));
        ctx->gen_grad_smem_set = kGenMaxSmem;
    }
    avse_generic_inverse_grad_kernel<<<dim3((unsigned)((long long)t_write * args->B)), GEN_THREADS, smem, (cudaStream_t)stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    return 0;
}
