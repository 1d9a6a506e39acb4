// Pieces of the GE2E loss shared by the small-N path (ge2e.cu) and the tensor-core path (ge2e_tc.cu): the mode
// dispatch, the contrast rule (GE2E paper eq. 7) and the exclusive centroids' diagonal gradient (eq. 8; DESIGN.md §3.3).
#pragma once
#include <stdint.h>

#include <type_traits>

#include "ge2e.h"

namespace spk {

// The instantiation of a kernel family templated on MODE for a runtime `mode`:
//   ge2e_for_mode(mode, [](auto m) { return some_kernel<decltype(m)::value>; })
template <class Pick>
auto ge2e_for_mode(int mode, Pick pick) {
  switch (mode) {
    case GE2E_CONTRAST: return pick(std::integral_constant<int, GE2E_CONTRAST>());
    case GE2E_EXCLUSIVE: return pick(std::integral_constant<int, GE2E_EXCLUSIVE>());
    case GE2E_CONTRAST | GE2E_EXCLUSIVE: return pick(std::integral_constant<int, GE2E_CONTRAST | GE2E_EXCLUSIVE>());
    default: return pick(std::integral_constant<int, 0>());
  }
}

// Contrast loss L = 1 - sigmoid(z_own) + sigmoid(z_k*), k* = the largest off-diagonal logit, ties to the lowest column.
// Each lane scans its columns in increasing order with a strict `>`; in the warp merge a lane's candidate (oz, oj) takes
// over from (bz, bj) when this is true.
__device__ __forceinline__ bool ge2e_argmax_takes(float bz, int bj, float oz, int oj) {
  return oz > bz || (oz == bz && oj < bj);
}
// sigmoid(z) and sigmoid(-z) = 1 - sigmoid(z) each from its own exp: no cancellation when |z| is large
__device__ __forceinline__ void ge2e_sigmoid_pair(float z, float& s, float& sn) {
  s = 1.f / (1.f + expf(-z));
  sn = 1.f / (1.f + expf(z));
}

// Exclusive own-speaker centroids: the part of dE that comes from the diagonal cosines.
// Row i = k*M + m of speaker k, u_i = sum_k - e_i, chat_i = u_i / (M-1) * urinv_i (urinv_i = 1 / max(|u_i|/(M-1), eps)),
// cos_i = ehat_i . chat_i and g_i = dL/dcos_i.  The diagonal is absent from the G that fed dEhat / dChat, so its two
// terms are added here:
//   row i itself:       g_i (chat_i - cos_i ehat_i) * einv_i
//   every other row k:  v_i = g_i (ehat_i - cos_i chat_i) * urinv_i / (M-1), summed over i != k, which is V - v_k.
// u_i is formed as sum - e_i (never from |M c - e|^2, which cancels when the other rows nearly sum to zero).
// One block of 256 threads per speaker, thread <-> column; `extra` is the caller's own per-column term for the speaker.
__device__ __forceinline__ void ge2e_excl_diag_grad(const float* __restrict__ E, int k, int M,
                                                    const float* __restrict__ einv, const float* __restrict__ cos_own,
                                                    const float* __restrict__ urinv, const float* __restrict__ gdiag,
                                                    float* __restrict__ dE, float extra) {
  constexpr int D = 256;
  const int d = threadIdx.x;
  const int64_t r0 = static_cast<int64_t>(k) * M;
  const float inv_m1 = 1.f / static_cast<float>(M - 1);
  float sum = 0.f;
  for (int m = 0; m < M; ++m) sum += __ldg(E + (r0 + m) * D + d);
  float V = 0.f;
  for (int m = 0; m < M; ++m) {
    const int64_t r = r0 + m;
    const float e = __ldg(E + r * D + d);
    const float sc = urinv[r] * inv_m1;
    V += gdiag[r] * (e * einv[r] - cos_own[r] * (sum - e) * sc) * sc;
  }
  for (int m = 0; m < M; ++m) {
    const int64_t r = r0 + m;
    const float e = __ldg(E + r * D + d);
    const float ei = einv[r], sc = urinv[r] * inv_m1, cs = cos_own[r], g = gdiag[r];
    const float eh = e * ei, ch = (sum - e) * sc;
    const float v = g * (eh - cs * ch) * sc;
    dE[r * D + d] += extra + (g * (ch - cs * eh) * ei + (V - v));
  }
}

}  // namespace spk
