// Fused GE2E loss forward + backward (see ge2e.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace spk {
// Loss variants (the SPK_GE2E_* bits of include/spkemb.h): 0 is the reference's softmax loss with inclusive centroids.
constexpr int GE2E_CONTRAST = 1;          // contrast loss (GE2E paper eq. 7) instead of the softmax loss (eq. 6)
constexpr int GE2E_EXCLUSIVE = 1 << 8;    // own-speaker column uses the centroid without the row itself (eq. 8)
constexpr int GE2E_MODE_BITS = GE2E_CONTRAST | GE2E_EXCLUSIVE;

size_t ge2e_workspace_bytes(int N, int M, int mode = 0);
// dE == nullptr -> forward only (loss).  w, b are device pointers to the 0-dim loss parameters.  `mode` is checked by
// the caller (spk_ge2e_loss_ex).
int ge2e_fused(const float* E, int N, int M, int D, const float* w, const float* b, float* loss, float* dE, float* dw,
               float* db, void* ws, size_t ws_bytes, cudaStream_t st, int mode = 0);
void ge2e_set_pdl(int on);       // programmatic dependent launch of the small-N row and centroid-gradient stages (default on)

// The centroid stage both paths start with, one block of 256 threads per speaker (D = 256).  Null pointers are outputs
// the call does not want.
struct Ge2eCentroids {
  const float* E;
  int N, M;
  float* loss;                    // zeroed: the row stage's accumulator
  float *dw, *db, *dchat;         // zeroed (gradient calls)
  float *einv, *chat, *cinv;      // 1 / max(|e_i|, eps); c_k / max(|c_k|, eps) in fp32; 1 / max(|c_k|, eps)
  float *cos_own, *urinv;         // exclusive centroids: each row's own-speaker cosine and 1 / max(|u_i| / (M-1), eps)
  __half *ehat_planes, *chat_planes;  // tensor-core path: Ehat and Chat as two fp16 planes (common.cuh)
  int64_t ehat_ps, chat_ps;           // their plane strides (elements)
};
int ge2e_centroids(const Ge2eCentroids& c, cudaStream_t st);

// tensor-core composition for large N (ge2e_tc.cu); ge2e_fused dispatches to it for N >= GE2E_TC_MIN_SPEAKERS
constexpr int GE2E_TC_MIN_SPEAKERS = 256;
size_t ge2e_tc_workspace_bytes(int N, int M, int mode = 0);
int ge2e_tc(const float* E, int N, int M, const float* w, const float* b, float* loss, float* dE, float* dw, float* db,
            void* ws, size_t ws_bytes, cudaStream_t st, int mode = 0);
}  // namespace spk
