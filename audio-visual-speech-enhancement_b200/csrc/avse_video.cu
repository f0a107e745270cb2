// HBM-bound reductions next to the spectral path (SURVEY 8(f) row 4):
//   VideoNormalizer (/root/reference/data_processor.py:201-212): per-pixel mean / std over (slices, frames) of the
//   mouth-crop tensor [N][H][W][F] and the in-place normalisation; the MSE-on-log-mel that network.evaluate reports
//   (/root/reference/network.py:214-220, loss = mean squared error over every element).
#include <cuda_runtime.h>
#include <string>

#include "../../include/avse_b200.h"
#include "avse_ctx.h"

namespace {

// partial sums of one chunk of slices.  VEC: thread = one 16-byte group of the flattened (pixel, frame) row -- every slice is one
// fully coalesced float4 load per thread, the four elements keep their own float64 sums (each is a fixed (pixel, frame) pair)
// and meet in the per-pixel accumulators at the end.  Scalar variant (row length not a multiple of 4): thread = pixel.
template <bool VEC>
__global__ void __launch_bounds__(256) avse_video_stats_kernel(const float* __restrict__ video, long long n_slices, int hw, int frames,
                                                               int slices_per_block, double* __restrict__ acc /* [hw][2] */) {
    const long long s0 = (long long)blockIdx.y * slices_per_block;
    long long s1 = s0 + slices_per_block;
    if (s1 > n_slices) s1 = n_slices;
    const size_t stride = (size_t)hw * frames;
    if (VEC) {
        const int j = blockIdx.x * blockDim.x + threadIdx.x;          // float4 index inside a slice
        if (4LL * j >= (long long)stride) return;
        double sum[4] = {0.0, 0.0, 0.0, 0.0}, sq[4] = {0.0, 0.0, 0.0, 0.0};
        const float4* q = reinterpret_cast<const float4*>(video + (size_t)s0 * stride) + j;
        const size_t stride4 = stride / 4;
        long long s = s0;
        for (; s + 1 < s1; s += 2, q += 2 * stride4) {                // two independent 16-byte loads in flight
            const float4 a = __ldg(q), b = __ldg(q + stride4);
            const float va[4] = {a.x, a.y, a.z, a.w}, vb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                sum[e] += (double)va[e] + (double)vb[e];
                sq[e] = fma((double)va[e], (double)va[e], fma((double)vb[e], (double)vb[e], sq[e]));
            }
        }
        if (s < s1) {
            const float4 a = __ldg(q);
            const float va[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) { sum[e] += (double)va[e]; sq[e] = fma((double)va[e], (double)va[e], sq[e]); }
        }
        // elements 4j .. 4j+3 belong to at most two pixels: merge before the atomics
        int p = (4 * j) / frames, r = (4 * j) - p * frames;
        double ps = 0.0, pq = 0.0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            ps += sum[e]; pq += sq[e];
            if (++r == frames || e == 3) {
                atomicAdd(acc + 2 * (size_t)p, ps);
                atomicAdd(acc + 2 * (size_t)p + 1, pq);
                ps = 0.0; pq = 0.0; r = 0; ++p;
            }
        }
        return;
    }
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    double sum = 0.0, sq = 0.0;
    const float* q = video + (size_t)s0 * stride + (size_t)p * frames;
    for (long long s = s0; s < s1; ++s, q += stride)
        for (int f = 0; f < frames; ++f) {
            const double v = (double)q[f];
            sum += v;
            sq = fma(v, v, sq);
        }
    atomicAdd(acc + 2 * (size_t)p, sum);
    atomicAdd(acc + 2 * (size_t)p + 1, sq);
}

__global__ void __launch_bounds__(256) avse_video_finalize_kernel(const double* __restrict__ acc, int hw, double count,
                                                                  float* __restrict__ mean, float* __restrict__ stdv) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    const double m = acc[2 * (size_t)p] / count;
    double var = acc[2 * (size_t)p + 1] / count - m * m;      // np.std: population (ddof = 0)
    if (var < 0.0) var = 0.0;
    mean[p] = (float)m;
    stdv[p] = (float)sqrt(var);
}

// In place, 16 bytes per thread when the tensor allows it (VEC): the (pixel, frame) position of a float4's first element is
// found with one division and then walked; scalar variant otherwise.
template <bool VEC>
__global__ void __launch_bounds__(256) avse_video_normalize_kernel(float* __restrict__ video, long long total, int hw, int frames,
                                                                   const float* __restrict__ mean, const float* __restrict__ stdv) {
    const long long step = (long long)gridDim.x * blockDim.x;
    if (VEC) {
        const long long n4 = total >> 2;
        float4* v4 = reinterpret_cast<float4*>(video);
        // (pixel, frame) of the thread's first element from one 64-bit division; every further float4 lies 4 * step elements on, so
        // the position is advanced by that stride's (quotient mod hw, remainder) with conditional subtractions -- the per-iteration
        // 64-bit divisions made the kernel instruction-bound next to its 4.9 TB/s of traffic
        long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        const long long i0 = 4 * j;
        const long long pix0 = i0 / frames;
        int r0 = (int)(i0 - pix0 * frames);
        int p0 = (int)(pix0 % hw);
        const long long stride = 4 * step;
        const int dr = (int)(stride % frames);
        const int dp = (int)((stride / frames) % hw);
        for (; j < n4; j += step) {
            float4 x = v4[j];
            int r = r0, p = p0;
            float v[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                v[e] = (v[e] - __ldg(mean + p)) / __ldg(stdv + p);           // dp:211-212: no epsilon, like the reference
                if (++r == frames) { r = 0; if (++p == hw) p = 0; }
            }
            x.x = v[0]; x.y = v[1]; x.z = v[2]; x.w = v[3];
            v4[j] = x;
            r0 += dr; p0 += dp;
            if (r0 >= frames) { r0 -= frames; ++p0; }
            if (p0 >= hw) p0 -= hw;
        }
    } else {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
            const int p = (int)((i / frames) % hw);
            video[i] = (video[i] - mean[p]) / stdv[p];
        }
    }
}

// Video half of a training batch: dst[i] = decode(pool[index[i]]), optionally normalised like avse_video_normalize, for rows of
// hw * frames elements (row4 float4 groups).  One CTA per output row at a time (a 128 x 128 x 5 slice is 320 KB of output), the
// CTAs striding over the rows so any n_out fits one launch.  A thread decodes 4 consecutive elements (one uchar4 or float4 load,
// one 16-byte store), four groups in flight; its (pixel, frame) position is walked like avse_video_normalize_kernel's.
template <typename P> struct Pix4;
template <> struct Pix4<unsigned char> {
    static __device__ __forceinline__ float4 load(const unsigned char* p, long long i) {
        const uchar4 t = __ldg(reinterpret_cast<const uchar4*>(p) + i);
        return make_float4((float)t.x, (float)t.y, (float)t.z, (float)t.w);
    }
};
template <> struct Pix4<float> {
    static __device__ __forceinline__ float4 load(const float* p, long long i) { return __ldg(reinterpret_cast<const float4*>(p) + i); }
};

template <typename P, bool NORM>
__global__ void __launch_bounds__(256) avse_gather_video_kernel(const P* __restrict__ pool, long long pool_slices, int row4, int frames,
                                                                const long long* __restrict__ index, long long n_out,
                                                                const float* __restrict__ mean, const float* __restrict__ stdv,
                                                                float* __restrict__ dst, int* __restrict__ bad) {
    constexpr int U = 4;                                     // float4 groups in flight per thread
    const int step = U * blockDim.x;
    // (pixel, frame) of the thread's first element and the advance of its position per step of 4 * blockDim.x elements
    const int e0 = 4 * threadIdx.x;
    const int p0 = NORM ? e0 / frames : 0, r0 = NORM ? e0 - p0 * frames : 0;
    const int ds = NORM ? 4 * (int)blockDim.x : 0;
    const int dp = NORM ? ds / frames : 0, dr = NORM ? ds - dp * frames : 0;
    for (long long i = blockIdx.x; i < n_out; i += gridDim.x) {
        const long long r = index[i];
        if (r < 0 || r >= pool_slices) { if (threadIdx.x == 0) atomicExch(bad, 1); continue; }
        const P* src = pool + r * (4LL * row4);
        float4* out = reinterpret_cast<float4*>(dst) + i * row4;
        int p = p0, q = r0;
        for (int j0 = threadIdx.x; j0 < row4; j0 += step) {
            float4 v[U];
#pragma unroll
            for (int k = 0; k < U; ++k) {
                const int j = j0 + k * blockDim.x;
                if (j < row4) v[k] = Pix4<P>::load(src, j);
            }
#pragma unroll
            for (int k = 0; k < U; ++k) {
                const int j = j0 + k * blockDim.x;
                if (j >= row4) break;
                if (NORM) {
                    int pp = p, qq = q;
                    auto norm = [&](float x) {                  // avse_video_normalize's arithmetic, then the next element
                        x = (x - __ldg(mean + pp)) / __ldg(stdv + pp);
                        if (++qq == frames) { qq = 0; ++pp; }
                        return x;
                    };
                    v[k].x = norm(v[k].x);
                    v[k].y = norm(v[k].y);
                    v[k].z = norm(v[k].z);
                    v[k].w = norm(v[k].w);
                    p += dp; q += dr;
                    if (q >= frames) { q -= frames; ++p; }
                }
                out[j] = v[k];
            }
        }
    }
}

__global__ void __launch_bounds__(256) avse_mse_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n,
                                                       double* __restrict__ acc) {
    double s = 0.0;
    const long long step = (long long)gridDim.x * blockDim.x;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool vec = ((((size_t)a | (size_t)b) & 15) == 0);
    const long long n4 = vec ? (n >> 2) : 0;
    for (long long i = tid; i < n4; i += step) {                      // 16-byte loads of both operands
        const float4 x = __ldg(reinterpret_cast<const float4*>(a) + i), y = __ldg(reinterpret_cast<const float4*>(b) + i);
        const double d0 = (double)x.x - (double)y.x, d1 = (double)x.y - (double)y.y, d2 = (double)x.z - (double)y.z, d3 = (double)x.w - (double)y.w;
        s = fma(d0, d0, fma(d1, d1, fma(d2, d2, fma(d3, d3, s))));
    }
    for (long long i = 4 * n4 + tid; i < n; i += step) {
        const double d = (double)a[i] - (double)b[i];
        s = fma(d, d, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        atomicAdd(acc, t);
    }
}

__global__ void avse_mse_finalize_kernel(const double* __restrict__ acc, double n, float* __restrict__ out) { *out = (float)(*acc / n); }

// librosa.core.magphase (dp:80): mag = |D|, phase = D / |D| with 1 + 0j where D == 0.  Also transposes the kernel's frame-major
// STFT [T][bins] into the reference's [bins][T] (dp:96 returns (freq, time) arrays).  One thread per output element.
__global__ void __launch_bounds__(256) avse_magphase_kernel(const float2* __restrict__ stft, long long n_utt, int T, int bins,
                                                            float* __restrict__ mag, float2* __restrict__ phase) {
    const long long total = n_utt * T * bins;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const long long u = i / ((long long)T * bins);
        const int r = (int)(i - u * (long long)T * bins);
        const int k = r / T, t = r - k * T;                       // output index [u][k][t]
        const float2 d = stft[(u * T + t) * bins + k];
        const float m = hypotf(d.x, d.y);
        if (mag) mag[i] = m;
        if (phase) phase[i] = m > 0.0f ? make_float2(d.x / m, d.y / m) : make_float2(1.0f, 0.0f);
    }
}

}  // namespace

extern "C" int avse_video_stats(avse_ctx* ctx, const float* video, long long n_slices, int hw, int frames, double* scratch,
                                float* mean_out, float* std_out, void* stream) {
    if (!ctx || !video || !scratch || !mean_out || !std_out) return avse_fail(AVSE_E_ARG, "avse_video_stats: NULL argument");
    if (n_slices <= 0 || hw <= 0 || frames <= 0) return avse_fail(AVSE_E_ARG, "avse_video_stats: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(scratch, 0, sizeof(double) * 2 * (size_t)hw, st));
    const long long row = (long long)hw * frames;
    const bool vec = (row % 4) == 0 && (((size_t)video) & 15) == 0;
    const int bx = vec ? (int)((row / 4 + 255) / 256) : (hw + 255) / 256;
    long long by = (8LL * ctx->num_sms + bx - 1) / bx;        // ~8 CTAs per SM in flight
    if (by > n_slices) by = n_slices;
    if (by > 65535) by = 65535;
    const int per = (int)((n_slices + by - 1) / by);
    by = (n_slices + per - 1) / per;
    if (vec) avse_video_stats_kernel<true><<<dim3((unsigned)bx, (unsigned)by), 256, 0, st>>>(video, n_slices, hw, frames, per, scratch);
    else avse_video_stats_kernel<false><<<dim3((unsigned)bx, (unsigned)by), 256, 0, st>>>(video, n_slices, hw, frames, per, scratch);
    CUDA_TRY(cudaGetLastError());
    avse_video_finalize_kernel<<<(hw + 255) / 256, 256, 0, st>>>(scratch, hw, (double)n_slices * frames, mean_out, std_out);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int avse_video_normalize(avse_ctx* ctx, float* video, long long n_slices, int hw, int frames, const float* mean,
                                    const float* stdv, void* stream) {
    if (!ctx || !video || !mean || !stdv) return avse_fail(AVSE_E_ARG, "avse_video_normalize: NULL argument");
    if (n_slices <= 0 || hw <= 0 || frames <= 0) return avse_fail(AVSE_E_ARG, "avse_video_normalize: bad sizes");
    const long long total = n_slices * hw * frames;
    long long bx = (total + 256 * 8 - 1) / (256 * 8);
    const long long cap = 16LL * ctx->num_sms;
    if (bx > cap) bx = cap;
    const bool vec = (total % 4) == 0 && (((size_t)video) & 15) == 0;
    if (vec) avse_video_normalize_kernel<true><<<(unsigned)bx, 256, 0, (cudaStream_t)stream>>>(video, total, hw, frames, mean, stdv);
    else avse_video_normalize_kernel<false><<<(unsigned)bx, 256, 0, (cudaStream_t)stream>>>(video, total, hw, frames, mean, stdv);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int avse_gather_video(avse_ctx* ctx, const void* pool, int pixel_format, long long pool_slices, int hw, int frames,
                                 const long long* index, long long n_out, const float* mean, const float* stdv, float* dst,
                                 int* bad_index_flag, void* stream) {
    if (n_out == 0) return 0;
    if (!ctx || !pool || !index || !dst || !bad_index_flag) return avse_fail(AVSE_E_ARG, "avse_gather_video: NULL argument");
    if ((mean == nullptr) != (stdv == nullptr)) return avse_fail(AVSE_E_ARG, "avse_gather_video: give both mean and stdv, or neither");
    if (pixel_format != AVSE_PIXEL_U8 && pixel_format != AVSE_PIXEL_F32) return avse_fail(AVSE_E_ARG, "avse_gather_video: bad pixel_format");
    const long long row = (long long)hw * frames;
    if (n_out < 0 || pool_slices <= 0 || hw <= 0 || frames <= 0 || (row & 3) || row / 4 > 0x7fffffffLL)
        return avse_fail(AVSE_E_ARG, "avse_gather_video: bad sizes (hw * frames must be a positive multiple of 4)");
    const size_t align = pixel_format == AVSE_PIXEL_U8 ? 3 : 15;
    if (((size_t)pool & align) || ((size_t)dst & 15))
        return avse_fail(AVSE_E_ARG, "avse_gather_video: dst must be 16-byte aligned, the pool aligned to 4 pixels");
    long long bx = 8LL * ctx->num_sms;                     // 8 CTAs of 256 threads per SM, each striding over the rows
    if (bx > n_out) bx = n_out;
    const int row4 = (int)(row / 4);
    cudaStream_t st = (cudaStream_t)stream;
    if (pixel_format == AVSE_PIXEL_U8) {
        const unsigned char* p = static_cast<const unsigned char*>(pool);
        if (mean) avse_gather_video_kernel<unsigned char, true><<<(unsigned)bx, 256, 0, st>>>(p, pool_slices, row4, frames, index, n_out, mean, stdv, dst, bad_index_flag);
        else avse_gather_video_kernel<unsigned char, false><<<(unsigned)bx, 256, 0, st>>>(p, pool_slices, row4, frames, index, n_out, mean, stdv, dst, bad_index_flag);
    } else {
        const float* p = static_cast<const float*>(pool);
        if (mean) avse_gather_video_kernel<float, true><<<(unsigned)bx, 256, 0, st>>>(p, pool_slices, row4, frames, index, n_out, mean, stdv, dst, bad_index_flag);
        else avse_gather_video_kernel<float, false><<<(unsigned)bx, 256, 0, st>>>(p, pool_slices, row4, frames, index, n_out, mean, stdv, dst, bad_index_flag);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int avse_mse(avse_ctx* ctx, const float* a, const float* b, long long n, double* scratch, float* out, void* stream) {
    if (!ctx || !a || !b || !scratch || !out) return avse_fail(AVSE_E_ARG, "avse_mse: NULL argument");
    if (n <= 0) return avse_fail(AVSE_E_ARG, "avse_mse: n must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(scratch, 0, sizeof(double), st));
    long long bx = (n + 256 * 8 - 1) / (256 * 8);
    const long long cap = 16LL * ctx->num_sms;
    if (bx > cap) bx = cap;
    avse_mse_kernel<<<(unsigned)bx, 256, 0, st>>>(a, b, n, scratch);
    CUDA_TRY(cudaGetLastError());
    avse_mse_finalize_kernel<<<1, 1, 0, st>>>(scratch, (double)n, out);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int avse_magphase(avse_ctx* ctx, const float* stft, long long n_utt, int n_frames, int n_bins, float* mag_out, float* phase_out,
                             void* stream) {
    if (!ctx || !stft || (!mag_out && !phase_out)) return avse_fail(AVSE_E_ARG, "avse_magphase: NULL argument");
    if (n_utt <= 0 || n_frames <= 0 || n_bins <= 0) return avse_fail(AVSE_E_ARG, "avse_magphase: bad sizes");
    const long long total = n_utt * n_frames * n_bins;
    long long bx = (total + 255) / 256;
    const long long cap = 16LL * ctx->num_sms;
    if (bx > cap) bx = cap;
    avse_magphase_kernel<<<(unsigned)bx, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float2*>(stft), n_utt, n_frames, n_bins, mag_out,
                                                                        reinterpret_cast<float2*>(phase_out));
    CUDA_TRY(cudaGetLastError());
    return 0;
}
