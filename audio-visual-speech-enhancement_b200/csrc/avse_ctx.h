// Internal: the opaque context behind include/avse_b200.h and shared error helpers.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include "../../include/avse_b200.h"
#include "avse_tables.h"
#include "avse_generic.h"
#include "avse_fwd_stages.cuh"

struct avse_ctx {
    int device = 0;
    int num_sms = 148;
    bool f4_tables = false;       // scan4 tables usable -> F4 kernel for pair batches
    bool force_f2 = false;        // AVSE_FORCE_F2=1: keep the 2-frame kernel (tests / A-B runs)
    bool std_tables = false;      // mel round widths equal AVSE_STD_ROUNDW -> unrolled kernels
    avse::HostTables host;
    void* dbase = nullptr;        // one device allocation holding every table
    avse::FwdTables fwd{};
    const float* d_tri_w = nullptr;
    const float* d_tri_ipiv = nullptr;
    const float* d_tri_sup = nullptr;
    const int* d_col_band = nullptr;
    const float* d_col_w = nullptr;
    const float* d_spike = nullptr;
    const unsigned* d_post_mask = nullptr;
    const float* d_post_w = nullptr;
    // geometry served by this context; generic == true: the fallback kernels of avse_generic.cu (any n_fft)
    bool generic = false;
    int n_fft = 640, hop = 160, n_bins = 321, n_mels = 80, spss = 20;
    avse::GenericHost gen;
    avse::GenericDev gd;
    void* gbase = nullptr;        // device allocation holding the generic tables
    size_t gen_fwd_smem_set = 0, gen_inv_smem_set = 0, gen_grad_smem_set = 0;   // dynamic shared-memory opt-in already requested through this context
};

// pool == nullptr: rows of args->speech / args->noise; otherwise avse_mix_pooled's row indirection into them (avse_common.h)
int avse_generic_forward(avse_ctx* ctx, const avse_forward_args* args, const avse::PoolRows* pool, void* stream);
int avse_generic_inverse(avse_ctx* ctx, const avse_inverse_args* args, void* stream);
int avse_generic_frames(const avse::GenericGeo& q, int L);
// avse_inverse_backward on a generic-geometry context, arguments already validated
int avse_generic_inverse_backward(avse_ctx* ctx, const avse_inverse_args* args, int T_use, int t_write, const float* grad_pcm,
                                  long long grad_pcm_stride, float* grad_mel, void* stream);

int avse_fail(int code, const std::string& msg);
int avse_cuda_fail(cudaError_t e, const char* where);
#define CUDA_TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return avse_cuda_fail(e_, #x); } while (0)
