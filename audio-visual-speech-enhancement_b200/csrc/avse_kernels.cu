// CUDA kernels (sm_100a) + C ABI of the forward spectral path.  See include/avse_b200.h.
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <vector>
#include <new>

#include "../../include/avse_b200.h"
#include "avse_common.h"
#include "avse_tables.h"
#include "avse_ctx.h"
#include "avse_fwd_stages.cuh"
#include "avse_fwd4_stages.cuh"

using namespace avse;

// ---------------------------------------------------------------------------------------------
// context / errors
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_err;
int avse_fail(int code, const std::string& msg) { g_err = msg; return code; }
int avse_cuda_fail(cudaError_t e, const char* where) {
    g_err = std::string(where) + ": " + cudaGetErrorString(e);
    return (int)e;
}

extern "C" const char* avse_last_error(void) { return g_err.c_str(); }
extern "C" const char* avse_version(void) { return "avse_b200 0.4 (sm_100a)"; }

extern "C" int avse_create(int sample_rate, double fmin, double fmax, int device, avse_ctx** out) {
    if (out == nullptr) return avse_fail(AVSE_E_ARG, "avse_create: out is NULL");
    *out = nullptr;
    avse_ctx* c = new (std::nothrow) avse_ctx();
    if (c == nullptr) return avse_fail(AVSE_E_ARG, "avse_create: out of host memory");
    if (!build_tables(c->host, sample_rate, fmin, fmax)) {
        std::string e = c->host.error;
        delete c;
        return avse_fail(AVSE_E_CONFIG, "avse_create: " + e);
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { delete c; return avse_fail(AVSE_E_NOCUDA, "avse_create: no CUDA device (this library has no CPU path)"); }
    if (device < 0 || device >= ndev) { delete c; return avse_fail(AVSE_E_ARG, "avse_create: bad device index"); }
    c->device = device;
    { const char* e2 = getenv("AVSE_FORCE_F2"); c->force_f2 = e2 != nullptr && e2[0] == '1'; }   // testing: 2-frame kernel only
    int prev = 0;
    cudaGetDevice(&prev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device);

    const HostTables& h = c->host;
    // pack everything into one buffer, 256-byte aligned sections
    struct Sec { const void* src; size_t bytes; size_t off; };
    std::vector<Sec> secs = {
        {h.window.data(), h.window.size() * 4, 0},     {h.tw1t.data(), h.tw1t.size() * 4, 0},
        {h.mel_w.data(), h.mel_w.size() * 4, 0},       {h.mel_lo.data(), h.mel_lo.size() * 4, 0},
        {h.mel_roundw.data(), h.mel_roundw.size() * 4, 0}, {h.tri_w.data(), h.tri_w.size() * 4, 0},
        {h.tri_ipiv.data(), h.tri_ipiv.size() * 4, 0}, {h.tri_sup.data(), h.tri_sup.size() * 4, 0},
        {h.col_band.data(), h.col_band.size() * 4, 0}, {h.col_w.data(), h.col_w.size() * 4, 0},
        {h.scan_w.data(), h.scan_w.size() * 4, 0},     {h.scan_loc.data(), h.scan_loc.size() * 4, 0},
        {h.scan_mask.data(), h.scan_mask.size() * 4, 0}, {h.window2.data(), h.window2.size() * 4, 0},
        {h.scan4_w.data(), h.scan4_w.size() * 4, 0},   {h.scan4_mask.data(), h.scan4_mask.size() * 4, 0},
        {h.scan4_loc.data(), h.scan4_loc.size() * 4, 0},
        {h.spike.data(), h.spike.size() * 4, 0},
        {h.post_mask.data(), h.post_mask.size() * 4, 0}, {h.post_w.data(), h.post_w.size() * 4, 0},
    };
    size_t total = 0;
    for (auto& s : secs) { s.off = total; total += (s.bytes + 255) / 256 * 256; }
    std::vector<char> stage(total, 0);
    for (auto& s : secs) memcpy(stage.data() + s.off, s.src, s.bytes);
    e = cudaMalloc(&c->dbase, total);
    if (e != cudaSuccess) { delete c; cudaSetDevice(prev); return avse_cuda_fail(e, "cudaMalloc(tables)"); }
    e = cudaMemcpy(c->dbase, stage.data(), total, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(c->dbase); delete c; cudaSetDevice(prev); return avse_cuda_fail(e, "cudaMemcpy(tables)"); }
    char* b = (char*)c->dbase;
    c->fwd.window = (const float*)(b + secs[0].off);
    c->fwd.tw1t = (const float*)(b + secs[1].off);
    c->fwd.mel_w = (const float*)(b + secs[2].off);
    c->fwd.mel_lo = (const int*)(b + secs[3].off);
    c->fwd.mel_roundw = (const int*)(b + secs[4].off);
    c->d_tri_w = (const float*)(b + secs[5].off);
    c->d_tri_ipiv = (const float*)(b + secs[6].off);
    c->d_tri_sup = (const float*)(b + secs[7].off);
    c->d_col_band = (const int*)(b + secs[8].off);
    c->d_col_w = (const float*)(b + secs[9].off);
    c->fwd.scan_w = (const float*)(b + secs[10].off);
    c->fwd.scan_loc = (const int*)(b + secs[11].off);
    c->fwd.scan_mask = (const int*)(b + secs[12].off);
    c->fwd.window2 = (const float*)(b + secs[13].off);
    c->fwd.scan4_w = (const float*)(b + secs[14].off);
    c->fwd.scan4_mask = (const unsigned*)(b + secs[15].off);
    c->fwd.scan4_loc = (const int*)(b + secs[16].off);
    c->d_spike = (const float*)(b + secs[17].off);
    c->d_post_mask = (const unsigned*)(b + secs[18].off);
    c->d_post_w = (const float*)(b + secs[19].off);
    c->f4_tables = h.scan4_ok;   // fast F4 kernel (4 frames per warp)
    c->std_tables = h.scan_ok;   // fused post+mel scan kernel; otherwise the generic band-gather kernel
    cudaSetDevice(prev);
    *out = c;
    return 0;
}

extern "C" void avse_destroy(avse_ctx* ctx) {
    if (ctx == nullptr) return;
    if (ctx->dbase || ctx->gbase) {
        int prev = 0;
        cudaGetDevice(&prev);
        cudaSetDevice(ctx->device);
        if (ctx->dbase) cudaFree(ctx->dbase);
        if (ctx->gbase) cudaFree(ctx->gbase);
        cudaSetDevice(prev);
    }
    delete ctx;
}

extern "C" int avse_get_filterbank(const avse_ctx* ctx, double* host_out) {
    if (ctx == nullptr || host_out == nullptr) return avse_fail(AVSE_E_ARG, "avse_get_filterbank: NULL argument");
    if (ctx->generic) memcpy(host_out, ctx->gen.fb.data(), sizeof(double) * ctx->gen.fb.size());
    else memcpy(host_out, ctx->host.fb.data(), sizeof(double) * NMEL * NBINS);
    return 0;
}

extern "C" int avse_get_geometry(const avse_ctx* ctx, int* out6) {
    if (ctx == nullptr || out6 == nullptr) return avse_fail(AVSE_E_ARG, "avse_get_geometry: NULL argument");
    out6[0] = ctx->n_fft; out6[1] = ctx->hop; out6[2] = ctx->n_bins; out6[3] = ctx->n_mels; out6[4] = ctx->spss;
    out6[5] = ctx->generic ? 1 : 0;
    return 0;
}

// Any geometry the reference can derive (dp:44-45, dp:49): the specialised kernels for 640 / 160 / 80 / 20, the generic
// fallback kernels (avse_generic.cu) otherwise.
extern "C" int avse_create_ex(int sample_rate, int n_fft, int hop, int n_mels, int spss, double fmin, double fmax, int device,
                              avse_ctx** out) {
    const char* fg = getenv("AVSE_FORCE_GENERIC");     // testing: run the generic kernels at the specialised geometry too
    if (n_fft == NFFT && hop == HOP && n_mels == NMEL && spss == SPSS && !(fg != nullptr && fg[0] == '1')) {
        const int rc = avse_create(sample_rate, fmin, fmax, device, out);
        if (rc != AVSE_E_CONFIG) return rc;     // a filterbank the banded kernels cannot hold falls through to the generic path
    }
    if (out == nullptr) return avse_fail(AVSE_E_ARG, "avse_create_ex: out is NULL");
    *out = nullptr;
    avse_ctx* c = new (std::nothrow) avse_ctx();
    if (c == nullptr) return avse_fail(AVSE_E_ARG, "avse_create_ex: out of host memory");
    if (!build_generic(c->gen, sample_rate, n_fft, hop, n_mels, spss, fmin, fmax)) {
        std::string e = c->gen.error;
        delete c;
        return avse_fail(AVSE_E_CONFIG, "avse_create_ex: " + e);
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { delete c; return avse_fail(AVSE_E_NOCUDA, "avse_create_ex: no CUDA device (this library has no CPU path)"); }
    if (device < 0 || device >= ndev) { delete c; return avse_fail(AVSE_E_ARG, "avse_create_ex: bad device index"); }
    c->device = device;
    c->generic = true;
    c->n_fft = n_fft; c->hop = hop; c->n_bins = c->gen.geo.bins; c->n_mels = n_mels; c->spss = spss;
    int prev = 0;
    cudaGetDevice(&prev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device);
    const GenericHost& h = c->gen;
    struct Sec { const void* src; size_t bytes; size_t off; };
    std::vector<Sec> secs = {
        {h.window.data(), h.window.size() * 4, 0},         {h.tw.data(), h.tw.size() * 8, 0},
        {h.window_inv.data(), h.window_inv.size() * 4, 0}, {h.tw_inv.data(), h.tw_inv.size() * 8, 0},
        {h.band_lo.data(), h.band_lo.size() * 4, 0},       {h.band_cnt.data(), h.band_cnt.size() * 4, 0},
        {h.band_off.data(), h.band_off.size() * 4, 0},     {h.band_w.data(), h.band_w.size() * 4, 0},
        {h.pinv.data(), h.pinv.size() * 4, 0},
    };
    size_t total = 0;
    for (auto& sc : secs) { sc.off = total; total += (sc.bytes + 255) / 256 * 256; }
    std::vector<char> stage(total, 0);
    for (auto& sc : secs) memcpy(stage.data() + sc.off, sc.src, sc.bytes);
    e = cudaMalloc(&c->gbase, total);
    if (e != cudaSuccess) { delete c; cudaSetDevice(prev); return avse_cuda_fail(e, "cudaMalloc(generic tables)"); }
    e = cudaMemcpy(c->gbase, stage.data(), total, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(c->gbase); delete c; cudaSetDevice(prev); return avse_cuda_fail(e, "cudaMemcpy(generic tables)"); }
    char* b = (char*)c->gbase;
    c->gd.window = (const float*)(b + secs[0].off);
    c->gd.tw = (const double*)(b + secs[1].off);
    c->gd.window_inv = (const float*)(b + secs[2].off);
    c->gd.tw_inv = (const double*)(b + secs[3].off);
    c->gd.band_lo = (const int*)(b + secs[4].off);
    c->gd.band_cnt = (const int*)(b + secs[5].off);
    c->gd.band_off = (const int*)(b + secs[6].off);
    c->gd.band_w = (const float*)(b + secs[7].off);
    c->gd.pinv = (const float*)(b + secs[8].off);
    cudaSetDevice(prev);
    *out = c;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// SNR factor (dp:130) -- one CTA per utterance, float64 accumulation
// ---------------------------------------------------------------------------------------------
template <typename S> struct Sample4;
template <> struct Sample4<float> {
    typedef float4 vec;
    static __device__ __forceinline__ void load(const float* p, int i, float (&v)[4]) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p) + i); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
};
template <> struct Sample4<short> {
    typedef short4 vec;
    static __device__ __forceinline__ void load(const short* p, int i, float (&v)[4]) {
        const short4 t = __ldg(reinterpret_cast<const short4*>(p) + i); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
};

// Float64 sums (sum x, sum x^2) of p[0, len) for the statistics pass: the vector part (vec: p is aligned) is split over the P
// CTAs of the cluster, the scalar tail (the whole range when unaligned) goes to the last one.
template <typename S>
static __device__ __forceinline__ void range_sums(const S* p, int len, bool vec, int P, int part, double& x0, double& x1) {
    const int n4 = vec ? (len >> 2) : 0;
    const int per4 = (n4 + P - 1) / P;                       // this CTA's share of the vector part
    const int lo4 = part * per4, hi4 = lo4 + per4 < n4 ? lo4 + per4 : n4;
    for (int i = lo4 + threadIdx.x; i < hi4; i += blockDim.x) {
        float v[4];
        Sample4<S>::load(p, i, v);
        x0 += (double)v[0] + (double)v[1] + (double)v[2] + (double)v[3];
        x1 += (double)v[0] * v[0] + (double)v[1] * v[1] + (double)v[2] * v[2] + (double)v[3] * v[3];
    }
    if (part == P - 1)
        for (int i = 4 * n4 + threadIdx.x; i < len; i += blockDim.x) { const double v = (double)p[i]; x0 += v; x1 += v * v; }
}

// One thread-block CLUSTER per utterance: the P CTAs of a cluster each reduce a contiguous part of the utterance and
// rank 0 gathers their partial sums through distributed shared memory -- no scratch buffer, no second launch.  P = 1 for
// the 3 s utterances of configs 1-3 (1 000 CTAs already fill the GPU); long-form audio (config 5: 64 x 60 s per GPU)
// gets P = 8 so that all 148 SMs pull on HBM instead of 64.
// pool.speech_index != nullptr (avse_mix_pooled): row u is the pooled pair pool_row(pool, u) (avse_common.h), its noise read
// from its phase; otherwise row u of speech / noise, with the phase 0.
template <typename S, bool CLUSTER>
__global__ void __launch_bounds__(256) avse_snr_factor_kernel(const S* __restrict__ speech, const S* __restrict__ noise,
                                                              long long stride, const int* __restrict__ lengths,
                                                              const int* __restrict__ noise_period, int L, const PoolRows pool,
                                                              const float* __restrict__ snr_db, float* __restrict__ factor_out,
                                                              float* __restrict__ equalizer_out, int* __restrict__ max_key,
                                                              int* __restrict__ min_key) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int P = CLUSTER ? (int)cluster.num_blocks() : 1;
    const int part = CLUSTER ? (int)cluster.block_rank() : 0;
    const int u = blockIdx.x / P;
    const S* s;
    const S* z;
    int n, Pn, off = 0;
    bool bad = false;
    if (pool.speech_index != nullptr) {
        const PoolRow r = pool_row(pool, u);
        s = speech + r.s_off;
        z = noise + r.n_off;
        n = r.ls;                                            // dp:130: the whole clip, before the pad / truncate to L
        Pn = r.ln;
        off = r.off;
        bad = !r.ok;
    } else {
        n = lengths ? lengths[u] : L;
        n = n < 0 ? 0 : (n > L ? L : n);                      // never read past the row (stride >= L is checked by the launcher)
        // dp:125-128: a noise file shorter than the speech is doubled until it covers it and then truncated, i.e. tiled
        // periodically: noise[i] = nz[i mod Pn]
        Pn = noise_period ? noise_period[u] : n;
        Pn = (Pn <= 0 || Pn > n) ? n : Pn;
        s = speech + (size_t)u * stride;
        z = noise + (size_t)u * stride;
    }
    const NoiseSpan span = noise_span(n, Pn, off);
    double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
    constexpr size_t AL = sizeof(typename Sample4<S>::vec) - 1;
    // identity rows keep the joint alignment test of the two rows (the summation order of the existing entry points)
    const bool vec_s = ((((size_t)s | (pool.speech_index ? 0 : (size_t)z)) & AL) == 0);
    range_sums(s, n, vec_s, P, part, a0, a1);
    if (!span.periodic) {
        const S* z0 = z + off;
        range_sums(z0, span.len0, pool.speech_index ? (((size_t)z0 & AL) == 0) : vec_s, P, part, b0, b1);
        if (span.len1 > 0) range_sums(z, span.len1, ((size_t)z & AL) == 0, P, part, b0, b1);     // the window wraps
    } else {
        // tiled noise (the noise file is shorter than the utterance): one weighted pass over its period
        const int perp = (Pn + P - 1) / P;
        const int lop = part * perp, hip = lop + perp < Pn ? lop + perp : Pn;
        for (int i = lop + threadIdx.x; i < hip; i += blockDim.x) {
            const double zv = (double)z[i], w = (double)noise_weight(span, i, Pn, off);
            b0 += w * zv; b1 += w * zv * zv;
        }
    }
    if (bad && part == 0 && threadIdx.x == 0) atomicExch(pool.bad_row_flag, 1);
    __shared__ double red[4][8];
    __shared__ double partial[4];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        b0 += __shfl_xor_sync(0xffffffffu, b0, o);
        b1 += __shfl_xor_sync(0xffffffffu, b1, o);
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { red[0][w] = a0; red[1][w] = a1; red[2][w] = b0; red[3][w] = b1; }
    __syncthreads();
    if (threadIdx.x < 4) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
        partial[threadIdx.x] = t;
    }
    if (CLUSTER) cluster.sync();                             // every CTA's partial sums are visible cluster-wide
    else __syncthreads();
    if (part == 0 && threadIdx.x == 0) {
        double t[4] = {0.0, 0.0, 0.0, 0.0};
        for (int r = 0; r < P; ++r) {
            const double* qq = CLUSTER ? cluster.map_shared_rank(partial, r) : partial;   // distributed shared memory
            t[0] += qq[0]; t[1] += qq[1]; t[2] += qq[2]; t[3] += qq[3];
        }
        // n == 0 (empty files): the reference mixes two empty arrays and pads with zeros (dp:39-40); nothing is scaled,
        // so any finite factor gives its result: 0.  var(noise) == 0 with n > 0 gives inf / nan exactly like numpy.
        const SnrGains r = snr_gains(n, t, snr_db ? (double)snr_db[u] : 0.0);
        factor_out[u] = r.factor;
        if (equalizer_out) equalizer_out[u] = r.equalizer;
        if (max_key) { max_key[3 * u] = (int)0x80000000; max_key[3 * u + 1] = (int)0x80000000; max_key[3 * u + 2] = (int)0x80000000; }
        if (min_key) { min_key[3 * u] = 0x7fffffff; min_key[3 * u + 1] = 0x7fffffff; min_key[3 * u + 2] = 0x7fffffff; }
    }
    if (CLUSTER) cluster.sync();                             // keep every CTA's shared memory alive until rank 0 has read it
}

template <typename S>
static cudaError_t launch_snr_factor(int B, int P, cudaStream_t st, const S* speech, const S* noise, long long stride, const int* lengths,
                                     const int* noise_period, int L, const PoolRows& pool, const float* snr_db, float* factor_out,
                                     float* equalizer_out, int* max_key, int* min_key) {
    if (P == 1) {       // plain launch: cluster launches carry extra scheduling constraints
        avse_snr_factor_kernel<S, false><<<B, 256, 0, st>>>(speech, noise, stride, lengths, noise_period, L, pool, snr_db, factor_out,
                                                            equalizer_out, max_key, min_key);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * P));
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)P;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, avse_snr_factor_kernel<S, true>, speech, noise, stride, lengths, noise_period, L, pool, snr_db, factor_out,
                              equalizer_out, max_key, min_key);
}

// Statistics launch shared by avse_snr_factor (identity rows: pool.speech_index == nullptr) and avse_mix_pooled.  `L` sizes the
// cluster: the longest row the pass may read.
static int snr_factor_launch(avse_ctx* ctx, const void* speech, const void* noise, int sample_format, long long stride, const int* lengths,
                             const int* noise_period, int B, int L, const PoolRows& pool, const float* snr_db, float* factor_out,
                             float* equalizer_out, int* max_key, int* min_key, void* stream) {
    // cluster size: enough CTAs to occupy every SM a few times over, each with >= 64 K samples, at most 8 (portable limit)
    int P = 1;
    while (P < 8 && (long long)B * P < 4LL * ctx->num_sms && L / (2 * P) >= 65536) P *= 2;
    cudaError_t e;
    if (sample_format == AVSE_SAMPLE_F32)
        e = launch_snr_factor<float>(B, P, (cudaStream_t)stream, (const float*)speech, (const float*)noise, stride, lengths, noise_period, L,
                                     pool, snr_db, factor_out, equalizer_out, max_key, min_key);
    else if (sample_format == AVSE_SAMPLE_I16)
        e = launch_snr_factor<short>(B, P, (cudaStream_t)stream, (const short*)speech, (const short*)noise, stride, lengths, noise_period, L,
                                     pool, snr_db, factor_out, equalizer_out, max_key, min_key);
    else return avse_fail(AVSE_E_ARG, "avse_snr_factor: bad sample_format");
    if (e != cudaSuccess) return avse_cuda_fail(e, "avse_snr_factor launch");
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int avse_snr_factor(avse_ctx* ctx, const void* speech, const void* noise, int sample_format, long long stride,
                               const int* lengths, const int* noise_period, int B, int L, const float* snr_db, float* factor_out,
                               float* equalizer_out, int* max_key, int* min_key, void* stream) {
    if (!ctx || !speech || !noise || !factor_out) return avse_fail(AVSE_E_ARG, "avse_snr_factor: NULL argument");
    if (B <= 0 || L <= 0 || stride < L) return avse_fail(AVSE_E_ARG, "avse_snr_factor: bad sizes");
    const PoolRows identity = {};
    return snr_factor_launch(ctx, speech, noise, sample_format, stride, lengths, noise_period, B, L, identity, snr_db, factor_out,
                             equalizer_out, max_key, min_key, stream);
}

// ---------------------------------------------------------------------------------------------
// fused forward kernel: persistent warps, each owning a contiguous range of (utterance, group) tiles
// ---------------------------------------------------------------------------------------------
#ifndef AVSE_FWD_WARPS
#define AVSE_FWD_WARPS 8       // warps per CTA
#endif
#ifndef AVSE_FWD_CTAS
#define AVSE_FWD_CTAS 2        // resident CTAs per SM (sets the register cap through __launch_bounds__)
#endif
constexpr int FWD_WARPS = AVSE_FWD_WARPS;
constexpr int FWD_CTAS = AVSE_FWD_CTAS;
constexpr int FWD_THREADS = FWD_WARPS * 32;
// shared memory: per-warp frame buffers, then CTA-shared tables: window, twiddles, then either the
// scan tables (SCAN kernel) or the banded weight tables (generic kernel)
constexpr int FWD_SM_WIN = FWD_WARPS * WARP_SMEM_F;               // [640] (w, w) pairs
constexpr int FWD_SM_TW = FWD_SM_WIN + 2 * NFFT;                  // [16][40] vec2
constexpr int FWD_SM_MODE = FWD_SM_TW + N1 * N2 * 2;
constexpr int FWD_SM_SCANW = FWD_SM_MODE;                         // SCAN: [SCAN_BINS] vec4
constexpr int FWD_SM_SCANMASK = FWD_SM_SCANW + SCAN_BINS * 4;     // SCAN: [16] int
constexpr int FWD_SM_SCANLOC = FWD_SM_SCANMASK + 16;              // SCAN: [80] ivec4
constexpr int FWD_SM_MELW = FWD_SM_MODE;                          // generic: [80][MEL_WROW]
constexpr int FWD_SM_MELLO = FWD_SM_MELW + NMEL * MEL_WROW;       // generic: [80] int
constexpr int FWD_SM_ROUNDW = FWD_SM_MELLO + NMEL;                // generic: [16] int
constexpr int FWD_SMEM_F_SCAN = FWD_SM_SCANLOC + NMEL * 4;
constexpr int FWD_SMEM_F_GEN = FWD_SM_ROUNDW + 16;
constexpr int FWD_SMEM_F = FWD_SMEM_F_GEN > FWD_SMEM_F_SCAN ? FWD_SMEM_F_GEN : FWD_SMEM_F_SCAN;
constexpr int FWD_SMEM_BYTES = FWD_SMEM_F * 4;
static_assert((FWD_SM_MODE % 4) == 0 && (FWD_SM_TW % 2) == 0 && (FWD_SM_SCANLOC % 4) == 0, "table alignment");
static_assert(FWD_CTAS * (FWD_SMEM_BYTES + 1024) <= 233472, "the resident CTAs must fit in shared memory");

// f = gain * resid (see FwdTileT): gain = the level equaliser applied to the noise at load, resid = what is left for
// the linear stages.  Without an equaliser array the whole factor is applied at load.
struct MixGain { float gain, resid; };
static __device__ __forceinline__ MixGain mix_gain(const avse_forward_args& A, int u) {
    const float f = A.factor ? A.factor[u] : 1.0f;
    MixGain m;
    if (A.equalizer) { m.gain = A.equalizer[u]; m.resid = m.gain != 0.0f ? __fdividef(f, m.gain) : 0.0f; }
    else { m.gain = f; m.resid = 1.0f; }
    return m;
}

struct FwdParams {
    avse_forward_args a;
    FwdTables tb;
    int T;            // frames per utterance
    int G;            // groups of FPG frames per utterance
    int total_tiles;  // B * G
    int per_warp;     // tiles per warp (contiguous range): the 2-frame kernel
    WarpSplit split;  // F4 kernel: balanced contiguous ranges (avse_common.h)
    PoolRows pool;    // avse_mix_pooled: row indirection into the speech / noise pools (a.speech / a.noise); speech_index == nullptr otherwise
};

// SCAN = true: fused post+mel scan (tables with scan_ok); false: generic banded gather.
template <bool SCAN>
__global__ void __launch_bounds__(FWD_THREADS, FWD_CTAS) avse_forward_kernel(const __grid_constant__ FwdParams P) {
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (SCAN) {
        for (int i = threadIdx.x; i < SCAN_BINS * 4; i += FWD_THREADS) smem[FWD_SM_SCANW + i] = P.tb.scan_w[i];
        if (threadIdx.x < 16) reinterpret_cast<int*>(smem + FWD_SM_SCANMASK)[threadIdx.x] = P.tb.scan_mask[threadIdx.x];
        for (int i = threadIdx.x; i < NMEL * 4; i += FWD_THREADS) reinterpret_cast<int*>(smem + FWD_SM_SCANLOC)[i] = P.tb.scan_loc[i];
    } else {
        for (int i = threadIdx.x; i < NMEL * MEL_WROW; i += FWD_THREADS) smem[FWD_SM_MELW + i] = P.tb.mel_w[i];
        for (int i = threadIdx.x; i < NMEL; i += FWD_THREADS) reinterpret_cast<int*>(smem + FWD_SM_MELLO)[i] = P.tb.mel_lo[i];
        if (threadIdx.x < MEL_ROUNDS) reinterpret_cast<int*>(smem + FWD_SM_ROUNDW)[threadIdx.x] = P.tb.mel_roundw[threadIdx.x];
    }
    for (int i = threadIdx.x; i < 2 * NFFT; i += FWD_THREADS) smem[FWD_SM_WIN + i] = P.tb.window2[i];
    for (int i = threadIdx.x; i < N1 * N2 * 2; i += FWD_THREADS) smem[FWD_SM_TW + i] = P.tb.tw1t[i];
    float* frames = smem + warp * WARP_SMEM_F;
    // keep never-written pad slots finite (they are multiplied by exact-zero weights)
    for (int i = lane; i < WARP_SMEM_F; i += 32) frames[i] = 0.0f;
    __syncthreads();

    const float* s_melw = smem + FWD_SM_MELW;
    const int* s_mello = reinterpret_cast<const int*>(smem + FWD_SM_MELLO);
    const int* s_roundw = reinterpret_cast<const int*>(smem + FWD_SM_ROUNDW);
    const float* s_win = smem + FWD_SM_WIN;
    const vec2* s_tw = reinterpret_cast<const vec2*>(smem + FWD_SM_TW);

    const avse_forward_args& A = P.a;
    const bool have_noise = A.noise != nullptr;
    const int gw = blockIdx.x * FWD_WARPS + warp;
    int tile = gw * P.per_warp;
    int n_tiles = P.total_tiles - tile;
    n_tiles = n_tiles < P.per_warp ? n_tiles : P.per_warp;
    if (n_tiles <= 0) return;
    int u = tile / P.G;
    int g = tile - u * P.G;

    float mx[3] = {neg_inf(), neg_inf(), neg_inf()};
    float factor = 0.0f, gain = 0.0f;
    int vs = 0, vn = 0, period = 0, phase = 0;
    const float* sp_row = nullptr;
    const float* nz_row = nullptr;
    bool fresh = true;

    auto flush_max = [&](int uu) {
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            float v = mx[s];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
            if (lane == 0) atomicMax(A.max_key + 3 * uu + s, float_to_key(v));
            mx[s] = neg_inf();
        }
    };

#pragma unroll 1
    for (int it = 0; it < n_tiles; ++it) {
        if (fresh) {
            fresh = false;
            if (P.pool.speech_index != nullptr) {           // pooled pair (avse_mix_pooled): always a pair batch
                const PoolRow r = pool_row(P.pool, u);
                vs = r.ls < A.L ? r.ls : A.L;
                vn = vs;
                sp_row = static_cast<const float*>(A.speech) + r.s_off;
                nz_row = static_cast<const float*>(A.noise) + r.n_off;
                period = r.ln;
                phase = r.off;
            } else {
                vs = A.len_speech ? A.len_speech[u] : A.L;
                vn = A.len_noise ? A.len_noise[u] : vs;
                vs = vs < 0 ? 0 : (vs < A.L ? vs : A.L);
                vn = vn < 0 ? 0 : (vn < A.L ? vn : A.L);
                sp_row = static_cast<const float*>(A.speech) + (size_t)u * A.in_stride;
                nz_row = have_noise ? static_cast<const float*>(A.noise) + (size_t)u * A.in_stride : nullptr;
                period = (have_noise && A.noise_period) ? A.noise_period[u] : 0;
                phase = 0;
            }
            fit_noise_row(nz_row, period, phase, vn);        // a window that does not wrap is a contiguous row
            const MixGain mg = mix_gain(A, u);
            factor = have_noise ? mg.resid : 0.0f;
            gain = have_noise ? mg.gain : 0.0f;
        }
        FwdTile tl;
        tl.sp = sp_row;
        tl.nz = nz_row;
        tl.L = A.L;
        tl.valid_s = vs;
        tl.valid_n = vn;
        tl.vmin = have_noise ? (vs < vn ? vs : vn) : 0;
        tl.T = P.T;
        tl.t0 = g * FPG;
        tl.factor = factor;
        tl.gain = gain;
        tl.period_n = period;
        tl.phase_n = phase;
        tl.mixed_pcm = A.mixed_pcm ? A.mixed_pcm + (size_t)u * A.pcm_stride : nullptr;

        // ---- pass 1 ----
        stage_pass1(tl, lane, s_win, s_tw, frames);
        __syncwarp();

        // ---- pass 2 ----
        {
            cpx x[40];
            pass2_compute(lane, frames, x);
            __syncwarp();
            pass2_store(lane, frames, x);
        }
        __syncwarp();

        // ---- post (+ mel) ----
        {
            vec2* srow = nullptr;
            const int tf = g * FPG + (SCAN ? (lane & 1) : (lane >> 4));
            if (A.stft_speech != nullptr && tf < P.T)
                srow = reinterpret_cast<vec2*>(A.stft_speech) + ((size_t)u * P.T + tf) * NBINS;
            if (SCAN) {
                const vec4* s_scan = reinterpret_cast<const vec4*>(smem + FWD_SM_SCANW);
                const int* s_mask = reinterpret_cast<const int*>(smem + FWD_SM_SCANMASK);
                if (A.stft_speech != nullptr) stage_post_scan<true>(lane, factor, s_scan, s_mask, frames, srow);
                else stage_post_scan<false>(lane, factor, s_scan, s_mask, frames, nullptr);
            } else {
                if (A.stft_speech != nullptr) stage_post<true>(lane, factor, frames, srow);
                else stage_post<false>(lane, factor, frames, nullptr);
            }
        }
        __syncwarp();

        if (!SCAN) {
            // ---- generic mel (results staged over the now-dead frame buffer 0) ----
            float acc[MEL_ROUNDS][3];
            stage_mel(lane, s_roundw, s_melw, s_mello, frames, acc);
            __syncwarp();
            stage_mel_store(lane, acc, frames);
            __syncwarp();
        }

        // ---- dB + stores ----
        {
            FwdOut out;
#if AVSE_F4_PTR_SLOT
            float* const* ps = reinterpret_cast<float* const*>(utt_sm + F4_UTT_F * (u & 1) + 2);
            out.dst[0] = ps[0]; out.dst[1] = ps[1]; out.dst[2] = ps[2];
#else
            out.dst[0] = A.out_speech ? A.out_speech + (size_t)u * A.out_stride : nullptr;
            out.dst[1] = A.out_noise ? A.out_noise + (size_t)u * A.out_stride : nullptr;
            out.dst[2] = A.out_mixed ? A.out_mixed + (size_t)u * A.out_stride : nullptr;
#endif
            out.layout = A.layout;
            out.n_slices = A.n_slices;
            out.ld_t = A.ld_t;
            if (SCAN) {
                const ivec4* s_loc = reinterpret_cast<const ivec4*>(smem + FWD_SM_SCANLOC);
#pragma unroll
                for (int q = 0; q < 3; ++q) stage_db_scan(lane, q, factor, have_noise, s_loc, frames, out, g * FPG, P.T, mx);
            } else {
#pragma unroll
                for (int q = 0; q < 3; ++q) stage_db(lane, q, factor, have_noise, frames, out, g * FPG, P.T, mx);
            }
        }
        __syncwarp();

        if (++g == P.G) {
            flush_max(u);
            g = 0;
            ++u;
            fresh = true;
        }
    }
    if (!fresh) flush_max(u);
}


// ---------------------------------------------------------------------------------------------
// F4 forward kernel (pair batches with the standard 2-tap filterbank): one warp = four frames, 8 warps per SM,
// up to 255 registers per thread so that the pass-1 window / twiddle values stay in registers for the whole
// kernel.  See avse_fwd4_stages.cuh for the stage functions and the reasoning.
// ---------------------------------------------------------------------------------------------
#ifndef AVSE_P1_UNIFIED
#define AVSE_P1_UNIFIED 0      // 1: pass 1 as one rolled five-round loop (stage4_pass1_unified)
#endif
#ifndef AVSE_F4_PREFETCH
#define AVSE_F4_PREFETCH 2
#endif
#ifndef AVSE_F4_WARPS
#define AVSE_F4_WARPS 8
#endif
constexpr int F4_WARPS = AVSE_F4_WARPS;
constexpr int F4_THREADS = F4_WARPS * 32;
constexpr int F4_SM_WIN = F4_WARPS * WARP4_SMEM_F;             // [640]
constexpr int F4_SM_TW = F4_SM_WIN + NFFT;                     // [16][40] vec2
constexpr int F4_SM_SCANW = F4_SM_TW + N1 * N2 * 2;            // [328] vec2 (wa, wb)
constexpr int F4_SM_LOC = F4_SM_SCANW + SCAN4_BINS * 2;        // [80] ivec4
constexpr int F4_SM_MIN = F4_SM_LOC + NMEL * 4;                // [warps][3][32] per-lane running minima
#ifndef AVSE_F4_PTR_SLOT
#define AVSE_F4_PTR_SLOT 1         // 1: the utterance's output row pointers live in the per-warp slot (written once per utterance)
#endif
constexpr int F4_UTT_F = AVSE_F4_PTR_SLOT ? 12 : 2;            // per parity: gain, noise period [, 4 output row pointers, 2 pad]
constexpr int F4_UTT_TILED_F = F4_UTT_F + 6;                   // TILED: + input row pointers (speech, noise), noise phase, 1 pad
constexpr int F4_SM_UTT = F4_SM_MIN + F4_WARPS * 96;           // [warps][2][F4_UTT_F or F4_UTT_TILED_F] per-utterance values, see the kernel
constexpr int F4_SMEM_F = F4_SM_UTT + F4_WARPS * 2 * F4_UTT_TILED_F;
static_assert((F4_UTT_F % 2) == 0 && (F4_UTT_TILED_F % 2) == 0, "8-byte aligned pointer slots");
constexpr int F4_SMEM_BYTES = F4_SMEM_F * 4;
static_assert((F4_SM_TW % 2) == 0 && (F4_SM_SCANW % 2) == 0 && (F4_SM_LOC % 4) == 0 && (F4_SM_UTT % 4) == 0, "table alignment");
static_assert(F4_SMEM_BYTES + 1024 <= 232448, "F4 shared memory must fit in one SM");

#ifndef AVSE_F4_BATCHED_PROLOGUE
#define AVSE_F4_BATCHED_PROLOGUE 1
#endif
// Kernel start: the CTA's tables, every global load in flight before the first store (table_fetch, avse_common.h), the warp's
// frame buffers zeroed meanwhile.  Out of line on purpose: inlined, the same code changed the register allocation of the main
// loop of this kernel (255 registers) and cost 1.3 % (profiles/README.md).
__device__ __noinline__ void f4_fill_tables(float* smem, float* frames, const float* window, const float* tw1t, const float* scan4_w,
                                            const int* scan4_loc) {
    static_assert((F4_SM_WIN % 4) == 0 && (F4_SM_TW % 4) == 0 && (F4_SM_SCANW % 4) == 0 && (F4_SM_LOC % 4) == 0 && (WARP4_SMEM_F % 4) == 0, "16-byte table copies");
    const int tid = threadIdx.x, lane = threadIdx.x & 31;
    TableRegs<NFFT / 4, F4_THREADS> r_win;
    TableRegs<N1 * N2 * 2 / 4, F4_THREADS> r_tw;
    TableRegs<SCAN4_BINS * 2 / 4, F4_THREADS> r_sw;
    TableRegs<NMEL, F4_THREADS> r_loc;
    table_fetch(window, tid, r_win);
    table_fetch(tw1t, tid, r_tw);
    table_fetch(scan4_w, tid, r_sw);
    table_fetch(scan4_loc, tid, r_loc);
    for (int i = lane; i < WARP4_SMEM_F / 4; i += 32) reinterpret_cast<float4*>(frames)[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);   // pad slots stay finite
    table_put(smem + F4_SM_WIN, tid, r_win);
    table_put(smem + F4_SM_TW, tid, r_tw);
    table_put(smem + F4_SM_SCANW, tid, r_sw);
    table_put(smem + F4_SM_LOC, tid, r_loc);
}

// TILED: the batch carries per-utterance noise periods (avse_forward_args::noise_period, dp:125-128), or it is a pooled batch
// (avse_mix_pooled: per-row speech / noise clips of two pools, the noise read from a phase).  load_utt resolves, once per
// utterance, the two input row pointers, the noise period and the phase into the warp's slot; identity rows with phase 0 are
// the noise_period case.  A separate instantiation, because this kernel sits on the 255-register / 32 KB instruction-cache
// cliff: with the period logic compiled into the common kernel, batches that do not use it ran 4.5 % slower
// (profiles/README.md, round 2).
template <typename S, bool TILED, bool PAD>
__global__ void __launch_bounds__(F4_THREADS, 1) avse_forward4_kernel(const __grid_constant__ FwdParams P) {
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* frames = smem + warp * WARP4_SMEM_F;
#if AVSE_F4_BATCHED_PROLOGUE
    f4_fill_tables(smem, frames, P.tb.window, P.tb.tw1t, P.tb.scan4_w, P.tb.scan4_loc);
#else
    for (int i = threadIdx.x; i < NFFT; i += F4_THREADS) smem[F4_SM_WIN + i] = P.tb.window[i];
    for (int i = threadIdx.x; i < N1 * N2 * 2; i += F4_THREADS) smem[F4_SM_TW + i] = P.tb.tw1t[i];
    for (int i = threadIdx.x; i < SCAN4_BINS * 2; i += F4_THREADS) smem[F4_SM_SCANW + i] = P.tb.scan4_w[i];
    for (int i = threadIdx.x; i < NMEL * 4; i += F4_THREADS) reinterpret_cast<int*>(smem + F4_SM_LOC)[i] = P.tb.scan4_loc[i];
    for (int i = lane; i < WARP4_SMEM_F; i += 32) frames[i] = 0.0f;   // pad slots stay finite (they meet exact-zero weights)
#endif
    __syncthreads();

    const float* s_win = smem + F4_SM_WIN;
    const vec2* s_tw = reinterpret_cast<const vec2*>(smem + F4_SM_TW);
    const vec2* s_scanw = reinterpret_cast<const vec2*>(smem + F4_SM_SCANW);
    const ivec4* s_loc = reinterpret_cast<const ivec4*>(smem + F4_SM_LOC);

    Lane4Const lc;
    lane4_const_init(lane, s_win, s_tw, lc);
    const unsigned mask_lo = P.tb.scan4_mask[2 * (lane & 7)], mask_hi = P.tb.scan4_mask[2 * (lane & 7) + 1];

    const avse_forward_args& A = P.a;
    long long first, count;
    warp_split_range(P.split, (int)blockIdx.x, warp, F4_WARPS, first, count);
    int tile = (int)first;
    const int n_tiles = (int)count;
    if (n_tiles <= 0) return;
    int u = tile / P.G;
    int g = tile - u * P.G;

    float mx[3] = {neg_inf(), neg_inf(), neg_inf()};
    float* mn = smem + F4_SM_MIN + warp * 96;
    mn[lane] = -neg_inf(); mn[32 + lane] = -neg_inf(); mn[64 + lane] = -neg_inf();
    float factor = 0.0f;          // residual factor (see FwdTileT): rides along the tile loop like vs / vn
    int vs = 0, vn = 0;
    // the level-equaliser gain (and the noise period) are needed once per tile, at the top of pass 1: they live in a
    // per-warp shared-memory slot, double-buffered by the utterance's parity, instead of in loop-carried registers
    constexpr int UF = TILED ? F4_UTT_TILED_F : F4_UTT_F;         // slot floats per parity
    float* utt_sm = smem + F4_SM_UTT + warp * (2 * UF);
    const S* in_speech = reinterpret_cast<const S*>(A.speech);
    const S* in_noise = reinterpret_cast<const S*>(A.noise);
    constexpr int LINE = 128 / (int)sizeof(S);        // samples per 128-byte line

    auto flush_max = [&](int uu) {
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            float v = mx[s], w = mn[32 * s + lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
                w = fminf(w, __shfl_xor_sync(0xffffffffu, w, o));
            }
            if (lane == 0) {
                atomicMax(A.max_key + 3 * uu + s, float_to_key(v));
                if (A.min_key) atomicMin(A.min_key + 3 * uu + s, float_to_key(w));
            }
            mx[s] = neg_inf();
            mn[32 * s + lane] = -neg_inf();
        }
    };

    auto prefetch_ahead = [&](int it, int u, int g, const FwdTileT<S>& tc) {
#if AVSE_F4_PREFETCH > 0
        // L2 prefetch of the samples this warp first touches AVSE_F4_PREFETCH groups from now (own tiles only)
        if (it + AVSE_F4_PREFETCH < n_tiles) {
            int g2 = g + AVSE_F4_PREFETCH, u2 = u;
            if (g2 >= P.G) { g2 -= P.G; ++u2; }
            const int lo = g2 == 0 ? 0 : g2 * (F4 * HOP) + HOP;      // first sample not covered by group g2 - 1
            const int hi = g2 * (F4 * HOP) + (NFFT + HOP);           // window end of group g2 (exclusive)
            const int i0 = (lo & ~(LINE - 1)) + LINE * lane;         // one 128-byte line per lane
            if (TILED) {      // rows resolved per utterance: this utterance's own rows only, a tiled noise is not prefetched
                if (u2 == u && i0 < hi && i0 < tc.valid_s && lane < 22) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(tc.sp + i0));
                    if (tc.period_n == 0 && i0 < tc.valid_n) asm volatile("prefetch.global.L2 [%0];" ::"l"(tc.nz + i0));
                }
            } else if (i0 < hi && i0 < A.L && i0 < A.in_stride && lane < 22) {
                const size_t o = (size_t)u2 * A.in_stride + i0;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(in_speech + o));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(in_noise + o));
            }
        }
#endif
    };
    // Software-pipelined tile loop: the raw samples of tile it+1 are loaded into registers before the dB stage of
    // tile it, so their HBM/L2 latency is covered by the dB arithmetic and stores instead of stalling pass 1.
    auto load_utt = [&](int uu, int& ovs, int& ovn, float& of) {
        ovs = A.len_speech ? A.len_speech[uu] : A.L;
        ovn = A.len_noise ? A.len_noise[uu] : ovs;
        ovs = ovs < 0 ? 0 : (ovs < A.L ? ovs : A.L);
        ovn = ovn < 0 ? 0 : (ovn < A.L ? ovn : A.L);
        const MixGain mg = mix_gain(A, uu);
        of = mg.resid;
        utt_sm[UF * (uu & 1)] = mg.gain;                      // every lane writes the same value
#if AVSE_F4_PTR_SLOT
        {   // this utterance's output rows (null stays null): read back once per tile instead of 64-bit multiplies + null checks
            float** ps = reinterpret_cast<float**>(utt_sm + UF * (uu & 1) + 2);
            ps[0] = A.out_speech ? A.out_speech + (size_t)uu * A.out_stride : nullptr;
            ps[1] = A.out_noise ? A.out_noise + (size_t)uu * A.out_stride : nullptr;
            ps[2] = A.out_mixed ? A.out_mixed + (size_t)uu * A.out_stride : nullptr;
            ps[3] = A.mixed_pcm ? A.mixed_pcm + (size_t)uu * A.pcm_stride : nullptr;
        }
#endif
        if (TILED) {
            const S* sp;
            const S* nz;
            int period, phase;
            if (P.pool.speech_index != nullptr) {             // pooled pair: rows of the two pools, noise from its phase
                const PoolRow r = pool_row(P.pool, uu);
                ovs = r.ls < A.L ? r.ls : A.L;
                ovn = ovs;
                sp = in_speech + r.s_off;
                nz = in_noise + r.n_off;
                period = r.ln;
                phase = r.off;
            } else {
                sp = in_speech + (size_t)uu * A.in_stride;
                nz = in_noise + (size_t)uu * A.in_stride;
                period = A.noise_period[uu];
                phase = 0;
            }
            fit_noise_row(nz, period, phase, ovn);            // the stored noise already covers the window: no modulo
            int* si = reinterpret_cast<int*>(utt_sm + UF * (uu & 1));
            si[1] = period;
            si[F4_UTT_F + 4] = phase;
            const S** pi = reinterpret_cast<const S**>(utt_sm + UF * (uu & 1) + F4_UTT_F);
            pi[0] = sp;
            pi[1] = nz;
        }
    };
    auto make_tile = [&](int uu, int gg, int tvs, int tvn, float tf) {
        FwdTileT<S> t;
        if (TILED) {
            const S* const* pi = reinterpret_cast<const S* const*>(utt_sm + UF * (uu & 1) + F4_UTT_F);
            t.sp = pi[0];
            t.nz = pi[1];
        } else {
            t.sp = in_speech + (size_t)uu * A.in_stride;  // (the INPUT row pointers through the slot too: 3 % slower -- they feed the
            t.nz = in_noise + (size_t)uu * A.in_stride;   //  address generation of the software-pipelined loads)
        }
        t.L = A.L;
        t.valid_s = tvs;
        t.valid_n = tvn;
        t.vmin = tvs < tvn ? tvs : tvn;
        t.T = P.T;
        t.t0 = gg * F4;
        t.factor = tf;
        t.gain = 0.0f;            // read from the slot at the top of pass 1
        t.period_n = TILED ? reinterpret_cast<const int*>(utt_sm)[UF * (uu & 1) + 1] : 0;
        t.phase_n = TILED ? reinterpret_cast<const int*>(utt_sm)[UF * (uu & 1) + F4_UTT_F + 4] : 0;
#if AVSE_F4_PTR_SLOT
        t.mixed_pcm = reinterpret_cast<float* const*>(utt_sm + UF * (uu & 1) + 2)[3];
#else
        t.mixed_pcm = A.mixed_pcm ? A.mixed_pcm + (size_t)uu * A.pcm_stride : nullptr;
#endif
        return t;
    };
    load_utt(u, vs, vn, factor);
    FwdTileT<S> tl = make_tile(u, g, vs, vn, factor);
    int nz_shift = 0;
    bool interior = group4_interior<S, TILED>(tl, nz_shift);
    bool reflect = AVSE_F4_REFLECT_FAST && !TILED && !interior && group4_reflect_only<S, PAD>(tl);   // see avse_fwd4_stages.cuh
    float rs[RAW4], rn[RAW4], ts[16], tn[16];
    if (interior) {
        p4_load_raw(tl, nz_shift, lane, rs, rn);
        p4_load_tail_raw(tl, nz_shift, lane, ts, tn);
    } else if (reflect) {
        p4_load_raw_reflect<S, PAD>(tl, lane, rs, rn);
        p4_load_tail_raw_reflect<S, PAD>(tl, lane, ts, tn);
    }
#pragma unroll 1
    for (int it = 0; it < n_tiles; ++it) {
        prefetch_ahead(it, u, g, tl);
        // ---- pass 1 ----
        tl.gain = utt_sm[UF * (u & 1)];
        if (reflect) {                       // mirrored loads, interior arithmetic; this group's PCM stores need their bounds check
            stage4_store_pcm_guarded(tl, lane, rs, rn, ts, tn);
            tl.mixed_pcm = nullptr;
        }
        if (interior || reflect) {
#if AVSE_P1_UNIFIED
            stage4_pass1_unified(tl, lane, rs, rn, ts, tn, lc, s_win, s_tw, frames);
#else
            stage4_pass1_main(tl, lane, rs, rn, lc, frames);
            stage4_pass1_tail_compute(tl, lane, ts, tn, s_win, s_tw, frames);
#endif
        } else {
            stage4_pass1_edge<S, TILED>(tl, lane, s_win, s_tw, frames);
        }
        __syncwarp();

        // ---- pass 2 ----
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
            cpx x[40];
            p4_pass2_compute(lane, r, frames, x);
            __syncwarp();
            p4_pass2_store(lane, r, frames, x);
        }
        __syncwarp();

        // ---- unpack + mel scan ----
        stage4_scan(lane, tl.factor, s_scanw, mask_lo, mask_hi, frames);
        __syncwarp();

        // ---- next tile: issue its loads now ----
        int u2 = u, g2 = g + 1;
        int vs2 = vs, vn2 = vn;
        float factor2 = tl.factor;
        const bool last_of_utt = g2 == P.G;
        const bool have_next = it + 1 < n_tiles;
        if (last_of_utt) { g2 = 0; ++u2; if (have_next) load_utt(u2, vs2, vn2, factor2); }
        FwdTileT<S> tnx = make_tile(have_next ? u2 : u, have_next ? g2 : g, vs2, vn2, factor2);
        int nz_shift2 = 0;
        const bool interior2 = have_next && group4_interior<S, TILED>(tnx, nz_shift2);
        const bool reflect2 = AVSE_F4_REFLECT_FAST && !TILED && have_next && !interior2 && group4_reflect_only<S, PAD>(tnx);
        if (interior2) {
            p4_load_raw(tnx, nz_shift2, lane, rs, rn);
            p4_load_tail_raw(tnx, nz_shift2, lane, ts, tn);
        } else if (reflect2) {
            p4_load_raw_reflect<S, PAD>(tnx, lane, rs, rn);
            p4_load_tail_raw_reflect<S, PAD>(tnx, lane, ts, tn);
        }

        // ---- dB + stores ----
        {
            FwdOut out;
#if AVSE_F4_PTR_SLOT
            float* const* ps = reinterpret_cast<float* const*>(utt_sm + UF * (u & 1) + 2);
            out.dst[0] = ps[0]; out.dst[1] = ps[1]; out.dst[2] = ps[2];
#else
            out.dst[0] = A.out_speech ? A.out_speech + (size_t)u * A.out_stride : nullptr;
            out.dst[1] = A.out_noise ? A.out_noise + (size_t)u * A.out_stride : nullptr;
            out.dst[2] = A.out_mixed ? A.out_mixed + (size_t)u * A.out_stride : nullptr;
#endif
            out.layout = A.layout;
            out.n_slices = A.n_slices;
            out.ld_t = A.ld_t;
#pragma unroll 1
#if AVSE_DB_SPLIT_LAST && AVSE_DB_BRANCHFREE_EXTRA
            for (int q = 0; q < 2; ++q) stage4_db(lane, q, tl.factor, s_loc, frames, out, g * F4, P.T, mx, mn);
            stage4_db_last(lane, tl.factor, s_loc, frames, out, g * F4, P.T, mx, mn);
#else
            for (int q = 0; q < 3; ++q) stage4_db(lane, q, tl.factor, s_loc, frames, out, g * F4, P.T, mx, mn);
#endif
        }
        __syncwarp();

        if (last_of_utt || !have_next) flush_max(u);
        u = u2; g = g2; vs = vs2; vn = vn2;
        tl = tnx;
        interior = interior2;
        reflect = reflect2;
    }
}

__global__ void avse_reset_max_kernel(int* __restrict__ max_key, int* __restrict__ min_key, int n, int min_value);

// The forward launch of avse_forward (pool.speech_index == nullptr) and avse_mix_pooled (specialised geometry).
static int forward_launch(avse_ctx* ctx, const avse_forward_args& a, const PoolRows& pool, void* stream) {
    if (a.B <= 0 || a.L <= HALF) return avse_fail(AVSE_E_ARG, "avse_forward: need B > 0 and L > 320 (reflect padding)");
    if (a.layout != AVSE_LAYOUT_SLICES && a.layout != AVSE_LAYOUT_SPEC) return avse_fail(AVSE_E_ARG, "avse_forward: bad layout");
    FwdParams P;
    P.a = a;
    P.pool = pool;
    P.tb = ctx->fwd;
    P.T = 1 + a.L / HOP;
    P.G = (P.T + FPG - 1) / FPG;
    if (a.layout == AVSE_LAYOUT_SLICES) {
        if (a.n_slices < 0 || (long long)a.n_slices * AVSE_SPSS > P.T) return avse_fail(AVSE_E_ARG, "avse_forward: n_slices exceeds int(T/20) (dp:50)");
        if (a.out_stride < (long long)a.n_slices * NMEL * AVSE_SPSS) return avse_fail(AVSE_E_ARG, "avse_forward: out_stride too small");
    } else {
        if (a.ld_t < P.T) return avse_fail(AVSE_E_ARG, "avse_forward: ld_t < T");
        if (a.out_stride < (long long)NMEL * a.ld_t) return avse_fail(AVSE_E_ARG, "avse_forward: out_stride too small");
    }
    if (a.mixed_pcm && a.pcm_stride < a.L) return avse_fail(AVSE_E_ARG, "avse_forward: pcm_stride < L");
    float* outs[3] = {a.out_speech, a.out_noise, a.out_mixed};
    for (int s = 0; s < 3; ++s)
        if (outs[s] && (((size_t)outs[s] & 15) || (a.out_stride & 3))) return avse_fail(AVSE_E_ARG, "avse_forward: outputs must be 16-byte aligned with out_stride % 4 == 0");
    const long long total = (long long)a.B * P.G;
    if (total > 0x7fffffffLL) return avse_fail(AVSE_E_ARG, "avse_forward: B * groups exceeds 2^31; split the batch");

    static thread_local int configured_dev = -1;
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != ctx->device) return avse_fail(AVSE_E_ARG, "avse_forward: current device differs from the context's device");
    // F4 kernel: pair batches (noise present), standard 2-tap filterbank, no complex STFT output
    if (a.sample_format != AVSE_SAMPLE_F32 && a.sample_format != AVSE_SAMPLE_I16) return avse_fail(AVSE_E_ARG, "avse_forward: bad sample_format");
    const bool i16 = a.sample_format == AVSE_SAMPLE_I16;
    const bool use_f4 = ctx->f4_tables && a.noise != nullptr && a.stft_speech == nullptr && (!ctx->force_f2 || i16);
    if (i16 && !use_f4) return avse_fail(AVSE_E_ARG, "avse_forward: int16 samples are supported for pair batches (noise != NULL, no stft_speech) with the standard 2-tap filterbank; convert to float32 first");
    if (use_f4) {
        static thread_local int configured4_dev = -1;
        if (configured4_dev != dev) {
            CUDA_TRY(cudaFuncSetAttribute(avse_forward4_kernel<float, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM_BYTES));
            CUDA_TRY(cudaFuncSetAttribute(avse_forward4_kernel<short, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM_BYTES));
            CUDA_TRY(cudaFuncSetAttribute(avse_forward4_kernel<float, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM_BYTES));
            CUDA_TRY(cudaFuncSetAttribute(avse_forward4_kernel<short, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM_BYTES));
            CUDA_TRY(cudaFuncSetAttribute(avse_forward4_kernel<float, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM_BYTES));
            CUDA_TRY(cudaFuncSetAttribute(avse_forward4_kernel<short, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, F4_SMEM_BYTES));
            configured4_dev = dev;
        }
        P.G = (P.T + F4 - 1) / F4;
        const long long total4 = (long long)a.B * P.G;
        long long blocks4 = ctx->num_sms;
        const long long need4 = (total4 + F4_WARPS - 1) / F4_WARPS;
        if (blocks4 > need4) blocks4 = need4;
        const long long nwarps4 = blocks4 * F4_WARPS;
        P.total_tiles = (int)total4;
        P.per_warp = (int)((total4 + nwarps4 - 1) / nwarps4);
        P.split = make_warp_split(total4, blocks4, F4_WARPS);
        const bool tiled = a.noise_period != nullptr || pool.speech_index != nullptr;
        // PAD: the batch carries per-utterance lengths, so rows may be zero-padded (see avse_fwd4_stages.cuh); never together with TILED
        const bool pad = !tiled && (a.len_speech != nullptr || a.len_noise != nullptr);
        const cudaStream_t st4 = (cudaStream_t)stream;
        if (i16 && tiled) avse_forward4_kernel<short, true, false><<<(unsigned)blocks4, F4_THREADS, F4_SMEM_BYTES, st4>>>(P);
        else if (tiled) avse_forward4_kernel<float, true, false><<<(unsigned)blocks4, F4_THREADS, F4_SMEM_BYTES, st4>>>(P);
        else if (i16 && pad) avse_forward4_kernel<short, false, true><<<(unsigned)blocks4, F4_THREADS, F4_SMEM_BYTES, st4>>>(P);
        else if (pad) avse_forward4_kernel<float, false, true><<<(unsigned)blocks4, F4_THREADS, F4_SMEM_BYTES, st4>>>(P);
        else if (i16) avse_forward4_kernel<short, false, false><<<(unsigned)blocks4, F4_THREADS, F4_SMEM_BYTES, st4>>>(P);
        else avse_forward4_kernel<float, false, false><<<(unsigned)blocks4, F4_THREADS, F4_SMEM_BYTES, st4>>>(P);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (configured_dev != dev) {
        CUDA_TRY(cudaFuncSetAttribute(avse_forward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_BYTES));
        CUDA_TRY(cudaFuncSetAttribute(avse_forward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_BYTES));
        configured_dev = dev;
    }
    long long blocks = (long long)FWD_CTAS * ctx->num_sms;
    const long long need = (total + FWD_WARPS - 1) / FWD_WARPS;
    if (blocks > need) blocks = need;
    const long long nwarps = blocks * FWD_WARPS;
    P.total_tiles = (int)total;
    P.per_warp = (int)((total + nwarps - 1) / nwarps);
    if (ctx->std_tables) avse_forward_kernel<true><<<(unsigned)blocks, FWD_THREADS, FWD_SMEM_BYTES, (cudaStream_t)stream>>>(P);
    else avse_forward_kernel<false><<<(unsigned)blocks, FWD_THREADS, FWD_SMEM_BYTES, (cudaStream_t)stream>>>(P);
    CUDA_TRY(cudaGetLastError());
    if (a.min_key) {   // these kernels do not track the stored minimum: "minus infinity" makes the floor pass always run
        avse_reset_max_kernel<<<(3 * a.B + 255) / 256, 256, 0, (cudaStream_t)stream>>>(nullptr, a.min_key, 3 * a.B, (int)0x80000000);
        CUDA_TRY(cudaGetLastError());
    }
    return 0;
}

extern "C" int avse_forward(avse_ctx* ctx, const avse_forward_args* args, void* stream) {
    if (!ctx || !args) return avse_fail(AVSE_E_ARG, "avse_forward: NULL argument");
    if (ctx->generic) return avse_generic_forward(ctx, args, nullptr, stream);
    const avse_forward_args& a = *args;
    if (!a.speech || !a.max_key) return avse_fail(AVSE_E_ARG, "avse_forward: speech and max_key are required");
    if (a.B <= 0 || a.L <= HALF) return avse_fail(AVSE_E_ARG, "avse_forward: need B > 0 and L > 320 (reflect padding)");
    if (!a.len_speech && a.in_stride < a.L) return avse_fail(AVSE_E_ARG, "avse_forward: in_stride < L needs len_speech");
    const PoolRows identity = {};
    return forward_launch(ctx, a, identity, stream);
}

// ---------------------------------------------------------------------------------------------
// top_db floor (dp:94) in place, and floor + segment gather (dp:49-57)
// ---------------------------------------------------------------------------------------------
// blockIdx.z selects the signal (data0/1/2 with key column which0 + z).  Only 16-byte groups that actually hold a value
// below the floor are written back, and an utterance whose stored minimum (min_key, tracked by avse_forward) is already
// >= max - 80 is skipped without being read: the pass then costs one key load per CTA.
#ifndef AVSE_FLOOR_ZLOOP
#define AVSE_FLOOR_ZLOOP 1
#endif
static __device__ __forceinline__ void floor_store(float4* q, float4 v, float thr) {
    if (fminf(fminf(v.x, v.y), fminf(v.z, v.w)) < thr) {
        v.x = fmaxf(v.x, thr); v.y = fmaxf(v.y, thr); v.z = fmaxf(v.z, thr); v.w = fmaxf(v.w, thr);
        *q = v;
    }
}

__global__ void __launch_bounds__(256) avse_floor_inplace_kernel(float* __restrict__ data0, float* __restrict__ data1,
                                                                 float* __restrict__ data2, long long stride, long long n_per_utt,
                                                                 const int* __restrict__ max_key, const int* __restrict__ min_key,
                                                                 int which0, int n_sig) {
    const int u = blockIdx.x;                 // utterance on grid.x: B is not capped at 65 535
#if AVSE_FLOOR_ZLOOP
    // gridDim.z == 1 with n_sig signals looped here: at 1 000 utterances two thirds of the (utterance, signal) pairs need no
    // clipping, and 6 000 CTAs that only read a key and exit still cost their launch slots
    for (int z = 0; z < n_sig; ++z) {
#else
    const int z = blockIdx.z;
    {
#endif
    float* data = z == 0 ? data0 : (z == 1 ? data1 : data2);
    const float thr = key_to_float(max_key[3 * u + which0 + z]) - TOP_DB;
#if AVSE_FLOOR_ZLOOP
    if (min_key != nullptr && key_to_float(min_key[3 * u + which0 + z]) >= thr) continue;
#else
    if (min_key != nullptr && key_to_float(min_key[3 * u + which0 + z]) >= thr) return;
#endif
    float* p = data + (size_t)u * stride;
    const long long n4 = n_per_utt >> 2;
    const long long step = (long long)gridDim.y * blockDim.x;
    long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x;
    for (; i + 3 * step < n4; i += 4 * step) {          // four independent 16-byte loads in flight per thread
        float4* q = reinterpret_cast<float4*>(p) + i;
        const float4 v0 = q[0], v1 = q[step], v2 = q[2 * step], v3 = q[3 * step];
        floor_store(q, v0, thr);
        floor_store(q + step, v1, thr);
        floor_store(q + 2 * step, v2, thr);
        floor_store(q + 3 * step, v3, thr);
    }
    for (; i < n4; i += step) {
        float4 v = reinterpret_cast<float4*>(p)[i];
        if (fminf(fminf(v.x, v.y), fminf(v.z, v.w)) < thr) {
            v.x = fmaxf(v.x, thr); v.y = fmaxf(v.y, thr); v.z = fmaxf(v.z, thr); v.w = fmaxf(v.w, thr);
            reinterpret_cast<float4*>(p)[i] = v;
        }
    }
    for (long long j = 4 * n4 + (long long)blockIdx.y * blockDim.x + threadIdx.x; j < n_per_utt; j += step)
        p[j] = fmaxf(p[j], thr);
    }
}

static unsigned floor_grid_x(long long n_per_utt) {
    long long bx = (n_per_utt / 4 + 256 * 8 - 1) / (256 * 8);    // >= 8 float4 per thread
    if (bx < 1) bx = 1;
    if (bx > 256) bx = 256;
    return (unsigned)bx;
}

extern "C" int avse_floor_inplace3(avse_ctx* ctx, float* speech, float* noise, float* mixed, long long stride, long long n_per_utt,
                                   int B, const int* max_key, const int* min_key, void* stream) {
    if (!ctx || !speech || !noise || !mixed || !max_key) return avse_fail(AVSE_E_ARG, "avse_floor_inplace3: NULL argument");
    if (B <= 0 || n_per_utt <= 0 || stride < n_per_utt) return avse_fail(AVSE_E_ARG, "avse_floor_inplace3: bad sizes");
    if ((((size_t)speech | (size_t)noise | (size_t)mixed) & 15) || (stride & 3))
        return avse_fail(AVSE_E_ARG, "avse_floor_inplace3: data must be 16-byte aligned with stride % 4 == 0");
    dim3 grid((unsigned)B, floor_grid_x(n_per_utt), AVSE_FLOOR_ZLOOP ? 1 : 3);
    avse_floor_inplace_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(speech, noise, mixed, stride, n_per_utt, max_key, min_key, 0, 3);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int avse_floor_inplace(avse_ctx* ctx, float* data, long long stride, long long n_per_utt, int B, const int* max_key,
                                  const int* min_key, int which, void* stream) {
    if (!ctx || !data || !max_key) return avse_fail(AVSE_E_ARG, "avse_floor_inplace: NULL argument");
    if (B <= 0 || n_per_utt <= 0 || stride < n_per_utt || which < 0 || which > 2) return avse_fail(AVSE_E_ARG, "avse_floor_inplace: bad sizes");
    if (((size_t)data & 15) || (stride & 3)) return avse_fail(AVSE_E_ARG, "avse_floor_inplace: data must be 16-byte aligned with stride % 4 == 0");
    dim3 grid((unsigned)B, floor_grid_x(n_per_utt));
    avse_floor_inplace_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(data, data, data, stride, n_per_utt, max_key, min_key, which, 1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

__global__ void __launch_bounds__(256) avse_floor_gather_kernel(const float* __restrict__ spec, long long spec_stride, int ld_t,
                                                                float* __restrict__ slices, long long slices_stride, int n_slices,
                                                                const int* __restrict__ max_key, int which, int n_mels, int spss) {
    const int u = blockIdx.x;
    const float thr = key_to_float(max_key[3 * u + which]) - TOP_DB;
    const float* src = spec + (size_t)u * spec_stride;
    float* dst = slices + (size_t)u * slices_stride;
    const int n = n_slices * n_mels * spss;
    for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < n; i += gridDim.y * blockDim.x) {
        const int j = i % spss;
        const int m = (i / spss) % n_mels;
        const int s = i / (spss * n_mels);
        dst[i] = fmaxf(src[(size_t)m * ld_t + s * spss + j], thr);
    }
}

extern "C" int avse_floor_gather(avse_ctx* ctx, const float* spec, long long spec_stride, int ld_t, float* slices,
                                 long long slices_stride, int n_slices, int B, const int* max_key, int which, void* stream) {
    if (!ctx || !spec || !slices || !max_key) return avse_fail(AVSE_E_ARG, "avse_floor_gather: NULL argument");
    if (B <= 0 || n_slices <= 0 || ld_t < n_slices * ctx->spss || which < 0 || which > 2) return avse_fail(AVSE_E_ARG, "avse_floor_gather: bad sizes");
    const int n = n_slices * ctx->n_mels * ctx->spss;
    int bx = (n + 255) / 256;
    if (bx > 64) bx = 64;
    dim3 grid((unsigned)B, (unsigned)bx);
    avse_floor_gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(spec, spec_stride, ld_t, slices, slices_stride, n_slices, max_key, which,
                                                                     ctx->n_mels, ctx->spss);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

__global__ void avse_reset_max_kernel(int* __restrict__ max_key, int* __restrict__ min_key, int n, int min_value) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        if (max_key) max_key[i] = (int)0x80000000;
        if (min_key) min_key[i] = min_value;
    }
}

extern "C" int avse_reset_max(avse_ctx* ctx, int* max_key, int* min_key, int n, void* stream) {
    if (!ctx || !max_key || n <= 0) return avse_fail(AVSE_E_ARG, "avse_reset_max: bad argument");
    avse_reset_max_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(max_key, min_key, n, 0x7fffffff);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

__global__ void avse_max_db_kernel(const int* __restrict__ max_key, int n, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = key_to_float(max_key[i]);
}

extern "C" int avse_max_db(avse_ctx* ctx, const int* max_key, int n, float* out_db, void* stream) {
    if (!ctx || !max_key || !out_db || n <= 0) return avse_fail(AVSE_E_ARG, "avse_max_db: bad argument");
    avse_max_db_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(max_key, n, out_db);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Pooled pairs: preprocess_audio_pair (dp:119-139) of (speech clip speech_index[b], noise clip noise_index[b] read from
// noise_offset[b] on) for every output row b, straight from two device-resident clip pools (see include/avse_b200.h).
// Three launches on `stream`: the statistics pass (which also flags invalid rows), the forward kernel, the top_db floor.
// ---------------------------------------------------------------------------------------------
extern "C" int avse_mix_pooled(avse_ctx* ctx, const avse_pool_mix_args* args, void* stream) {
    if (!ctx || !args) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: NULL argument");
    const avse_pool_mix_args& m = *args;
    if (!m.speech_pool || !m.noise_pool || !m.speech_len || !m.noise_len || !m.speech_index || !m.noise_index)
        return avse_fail(AVSE_E_ARG, "avse_mix_pooled: pools, clip lengths and row indices are required");
    if (!m.out_speech || !m.out_noise || !m.out_mixed || !m.factor_out || !m.max_key || !m.bad_row_flag)
        return avse_fail(AVSE_E_ARG, "avse_mix_pooled: the three slice outputs, factor_out, max_key and bad_row_flag are required");
    if (m.n_speech <= 0 || m.n_noise <= 0 || m.speech_stride <= 0 || m.noise_stride <= 0)
        return avse_fail(AVSE_E_ARG, "avse_mix_pooled: empty pool (n_speech, n_noise and both strides must be > 0)");
    if (m.B <= 0 || m.n_slices <= 0) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: need B > 0 and n_slices > 0");
    if (m.sample_format != AVSE_SAMPLE_F32 && m.sample_format != AVSE_SAMPLE_I16) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: bad sample_format");
    PoolRows pool;
    pool.speech_index = m.speech_index;
    pool.noise_index = m.noise_index;
    pool.noise_offset = m.noise_offset;
    pool.speech_len = m.speech_len;
    pool.noise_len = m.noise_len;
    pool.speech_stride = m.speech_stride;
    pool.noise_stride = m.noise_stride;
    pool.n_speech = m.n_speech;
    pool.n_noise = m.n_noise;
    pool.bad_row_flag = m.bad_row_flag;
    avse_forward_args a = {};
    a.speech = m.speech_pool;
    a.noise = m.noise_pool;
    a.factor = m.factor_out;
    a.B = m.B;
    a.L = m.L;
    a.layout = AVSE_LAYOUT_SLICES;
    a.n_slices = m.n_slices;
    a.out_speech = m.out_speech;
    a.out_noise = m.out_noise;
    a.out_mixed = m.out_mixed;
    a.out_stride = m.out_stride;
    a.mixed_pcm = m.mixed_pcm;
    a.pcm_stride = m.pcm_stride;
    a.max_key = m.max_key;
    a.min_key = m.min_key;
    a.sample_format = m.sample_format;
    a.equalizer = m.equalizer_out;
    // refuse what the forward pass would refuse before the statistics pass is enqueued
    const int half = ctx->generic ? ctx->n_fft / 2 : HALF;
    if (m.L <= half) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: need L > n_fft / 2 (reflect padding)");
    const int T = ctx->generic ? avse_generic_frames(ctx->gen.geo, m.L) : 1 + m.L / HOP;
    if ((long long)m.n_slices * ctx->spss > T) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: n_slices exceeds int(T / spss) (dp:50)");
    const long long n_per_utt = (long long)m.n_slices * ctx->n_mels * ctx->spss;
    if (m.out_stride < n_per_utt) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: out_stride too small");
    float* outs[3] = {m.out_speech, m.out_noise, m.out_mixed};
    for (int s = 0; s < 3; ++s)
        if (((size_t)outs[s] & 15) || (m.out_stride & 3)) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: outputs must be 16-byte aligned with out_stride % 4 == 0");
    if (m.mixed_pcm && m.pcm_stride < m.L) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: pcm_stride < L");
    if (m.sample_format == AVSE_SAMPLE_I16 && !ctx->generic && !ctx->f4_tables)
        return avse_fail(AVSE_E_ARG, "avse_mix_pooled: int16 samples need the standard 2-tap filterbank; convert the pools to float32 first");
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev != ctx->device) return avse_fail(AVSE_E_ARG, "avse_mix_pooled: current device differs from the context's device");

    const int longest = m.speech_stride < 0x7fffffffLL ? (int)m.speech_stride : 0x7fffffff;     // sizes the statistics clusters
    int rc = snr_factor_launch(ctx, m.speech_pool, m.noise_pool, m.sample_format, 0, nullptr, nullptr, m.B, longest, pool, m.snr_db,
                               m.factor_out, m.equalizer_out, m.max_key, m.min_key, stream);
    if (rc != 0) return rc;
    rc = ctx->generic ? avse_generic_forward(ctx, &a, &pool, stream) : forward_launch(ctx, a, pool, stream);
    if (rc != 0) return rc;
    return avse_floor_inplace3(ctx, m.out_speech, m.out_noise, m.out_mixed, m.out_stride, n_per_utt, m.B, m.max_key, m.min_key, stream);
}

// ---------------------------------------------------------------------------------------------
// make_sample_set (speech_enhancer.py:241-262): np.concatenate over samples + ONE shared permutation, as a
// row gather on the device: dst_a[i][:] = src_a[index[i]][:] for up to three arrays that share the index.
// A row is one (80, 20) slice (6 400 bytes) -- or any multiple of 4 floats.  HBM-bound: 2 x row bytes per row.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) avse_gather_rows_kernel(const float* __restrict__ s0, const float* __restrict__ s1,
                                                               const float* __restrict__ s2, long long src_rows,
                                                               const long long* __restrict__ index, long long n_out, int row4,
                                                               float* __restrict__ d0, float* __restrict__ d1, float* __restrict__ d2,
                                                               int* __restrict__ bad) {
    const int z = blockIdx.y;
    const float4* src = reinterpret_cast<const float4*>(z == 0 ? s0 : (z == 1 ? s1 : s2));
    float4* dst = reinterpret_cast<float4*>(z == 0 ? d0 : (z == 1 ? d1 : d2));
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp; i < n_out; i += nwarps) {       // one warp per output row: coalesced 512-byte bursts
        const long long r = index[i];
        if (r < 0 || r >= src_rows) { if (lane == 0) atomicExch(bad, 1); continue; }
        const float4* sp = src + r * row4;
        float4* dp = dst + i * row4;
        int j = lane;
        for (; j + 96 < row4; j += 128) {
            const float4 a = sp[j], b = sp[j + 32], c = sp[j + 64], d = sp[j + 96];
            dp[j] = a; dp[j + 32] = b; dp[j + 64] = c; dp[j + 96] = d;
        }
        for (; j < row4; j += 32) dp[j] = sp[j];
    }
}

extern "C" int avse_gather_rows(avse_ctx* ctx, const float* src0, const float* src1, const float* src2, long long src_rows,
                                long long row_elems, const long long* index, long long n_out, float* dst0, float* dst1, float* dst2,
                                int* bad_index_flag, void* stream) {
    if (!ctx || !src0 || !dst0 || !index) return avse_fail(AVSE_E_ARG, "avse_gather_rows: NULL argument");
    if ((src1 == nullptr) != (dst1 == nullptr) || (src2 == nullptr) != (dst2 == nullptr) || (src2 && !src1))
        return avse_fail(AVSE_E_ARG, "avse_gather_rows: src/dst arrays must be given in matching pairs, in order");
    if (src_rows <= 0 || n_out <= 0 || row_elems <= 0 || (row_elems & 3) || row_elems > 0x7fffffffLL * 4)
        return avse_fail(AVSE_E_ARG, "avse_gather_rows: row_elems must be a positive multiple of 4");
    const float* ps[6] = {src0, src1, src2, dst0, dst1, dst2};
    for (int i = 0; i < 6; ++i)
        if ((size_t)ps[i] & 15) return avse_fail(AVSE_E_ARG, "avse_gather_rows: arrays must be 16-byte aligned");
    if (!bad_index_flag) return avse_fail(AVSE_E_ARG, "avse_gather_rows: bad_index_flag (device int, zeroed by the caller) is required");
    const int narr = src2 ? 3 : (src1 ? 2 : 1);
    long long bx = (n_out + 7) / 8;                      // 8 warps per CTA
    const long long cap = (long long)ctx->num_sms * 16;
    if (bx > cap) bx = cap;
    dim3 grid((unsigned)bx, (unsigned)narr);
    avse_gather_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src0, src1, src2, src_rows, index, n_out, (int)(row_elems / 4),
                                                                    dst0, dst1, dst2, bad_index_flag);
    CUDA_TRY(cudaGetLastError());
    return 0;
}
