// Fused GE2E loss forward + backward (see ge2e.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

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
void ge2e_set_tile_v2(int on);   // 0: first (16-row) row-tile stage for mode 0, 1: re-tiled stage (default, every mode)
void ge2e_set_pdl(int on);       // programmatic dependent launch between the three small-N stages (default on)
// tensor-core composition for large N (ge2e_tc.cu); ge2e_fused dispatches to it for N >= GE2E_TC_MIN_SPEAKERS
constexpr int GE2E_TC_MIN_SPEAKERS = 256;
size_t ge2e_tc_workspace_bytes(int N, int M, int mode = 0);
int ge2e_tc(const float* E, int N, int M, const float* w, const float* b, float* loss, float* dE, float* dw, float* db,
            void* ws, size_t ws_bytes, cudaStream_t st, int mode = 0);
}  // namespace spk
