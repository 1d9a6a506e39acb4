// Bandwidth-bound building blocks of the encoder (see rowops.cu).
#pragma once
#include <algorithm>
#include "../../include/spkemb.h"
#include "common.cuh"

namespace spk {

struct PackSeg {
  const float* src;
  int64_t dst_off;   // elements into the packed arena
  int64_t n;
};
struct PackTable {
  PackSeg seg[24];
  int count;
};

int pack_weights(const PackTable& tab, void* dst, int64_t plane_stride, int planes, cudaStream_t st);
// The four mel kernels below take C = Mel_Dim at run time: a multiple of 8 in [16, 256], which make_plan checks.
// mel view (include/spkemb.h spk_mel_view) -> token-major split tensor [B*T, C]
int mel_pack(const spk_mel_view& mel, void* out, int64_t plane_stride, int planes, int B, int C, int T, cudaStream_t st);
// ragged batch (include/spkemb.h spk_mel_ragged) -> token-major split tensor, crop / reflect-pad to T in the load
int mel_pack_ragged(const spk_mel_ragged& mel, void* out, int64_t plane_stride, int planes, int B, int C, int T,
                    cudaStream_t st);
// token-major fp32 [B*T, C] (the input gradient) -> fp32 [B, C, T], the layout of the mel input
int mel_grad_unpack(const float* src, float* d_mel, int B, int C, int T, cudaStream_t st);
// Adjoint of mel_pack_ragged: token-major fp32 [B*T, C] -> d_data fp32 [C, mel.total_frames] (=), every slice folded
// back onto the columns it was cut from; columns no slice reads receive 0.  Slices form groups: segments[g] ..
// segments[g+1] - 1 (device int32 [groups + 1]), or runs of rows_per_group slices when segments is null.
// Precondition: the column spans of different groups (smallest start .. largest start + length of their slices) do not
// overlap; slices of one group may.  Every column is written by one thread, which adds its group's contributions in
// slice order and, within a slice, in frame order: no atomics, bit-identical results from identical calls.
int mel_grad_fold(const float* src, const spk_mel_ragged& mel, const int32_t* segments, int rows_per_group, int groups,
                  float* d_data, int B, int C, int T, cudaStream_t st);
int pe_transpose(const float* pe, float* pe_t, int D, int max_pos, int T, cudaStream_t st);

// y[r] = LN(z[r * z_row_step]) over 256 columns; stats[r] = (mean, rstd) (may be null)
int ln_fwd(const void* z, int64_t z_ps, int z_planes, int64_t z_row_step, const float* gamma, const float* beta,
           void* y, int64_t y_ps, int y_planes, float* stats, int64_t rows, cudaStream_t st);
int ln_bwd(const void* dy, int64_t dy_ps, int dy_planes, const void* z, int64_t z_ps, int z_planes, const float* stats,
           const float* gamma, void* dz, int64_t dz_ps, int dz_planes, void* dz_drop, DropCfg drop, uint32_t site,
           float* dgamma, float* dbeta, float* dbias, int64_t rows, const float* gscale, cudaStream_t st);

// scores / dP come either as split planes (s / dp) or as plain fp32 (s_f32 / dp_f32 != nullptr)
int softmax_fwd(const void* s, const float* s_f32, int64_t ps, int planes, void* p, void* p_drop, DropCfg drop,
                uint32_t site, int64_t rows, int T, int Tp, cudaStream_t st);
int softmax_bwd(const void* p, const void* dp, const float* dp_f32, int64_t ps, int planes, void* ds, DropCfg drop,
                uint32_t site, float scale, int64_t rows, int T, int Tp, cudaStream_t st);

int dropout_keep(uint64_t seed, float p, uint32_t site, uint64_t idx8_begin, int64_t n8, float* out, cudaStream_t st);
int colsum(const void* x, int64_t ps, int planes, float* out, int64_t rows, int C, cudaStream_t st);
int prenet_bwd(const void* dh, int64_t ps, int planes, const uint32_t* bits, const float* pe_t, DropCfg drop, uint32_t site,
               void* du, int64_t du_ps, float* dalpha, float* dbias, int64_t rows, int T, const float* gscale,
               cudaStream_t st);
int pe_alpha_grad(const void* dh, int64_t ps, int planes, const float* pe_t, DropCfg drop, uint32_t site, float* dalpha,
                  int64_t rows, int T, const float* gscale, cudaStream_t st);

}  // namespace spk
