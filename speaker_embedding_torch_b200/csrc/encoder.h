// Encoder forward / backward orchestration (see encoder.cu).
#pragma once
#include <cuda_runtime.h>
#include "../../include/spkemb.h"
#include "common.cuh"

namespace spk {
size_t encoder_workspace_bytes(const spk_encoder_config& c, int B, int T, int S, int P, int keep);
// exactly one of mel / ragged is non-null.  segments (device int32 [utterances + 1], ragged input, S == 1): utterance
// u averages slices segments[u] .. segments[u+1] - 1 (head_fwd_seg); null: B / S slices per d-vector.
int encoder_forward(const spk_encoder_config& cfg, const spk_encoder_params& w, const spk_mel_view* mel,
                    const spk_mel_ragged* ragged, int B, int T, int S, int P, int training, uint64_t seed, float* dvec,
                    void* ws, size_t ws_bytes, int keep, cudaStream_t st, const int32_t* segments = nullptr,
                    int utterances = 0);
// Backward of a ragged forward: segments as in encoder_forward, or null (B / S slices per d-vector); d_data null or
// [mel_dim, mel->total_frames] fp32, which receives (=) the adjoint of the crop / reflect-pad (mel_grad_fold).
struct RaggedGrad {
  const spk_mel_ragged* mel;
  const int32_t* segments;
  int utterances;
  float* d_data;
};
// grads null: no parameter gradient; d_mel null: no input gradient; rg: the ragged forms (d_mel must be null)
int encoder_backward(const spk_encoder_config& cfg, const spk_encoder_params& w, const spk_encoder_params* grads,
                     float* d_mel, const float* d_dvec, int B, int T, int S, int P, int training, uint64_t seed,
                     void* ws, size_t ws_bytes, cudaStream_t st, const RaggedGrad* rg = nullptr);
int encoder_debug_layout(const spk_encoder_config& c, int B, int T, int S, int P, int keep, char* buf, size_t cap);
void encoder_set_prune(bool on);
void encoder_set_fused_attn(bool on);
void encoder_set_infer_attn_two(int on);
void encoder_set_fuse_ln(int on);
void encoder_set_fused_train_attn(bool on);
int encoder_plan_flags();
void encoder_set_grad_scale_log2(int k);
}  // namespace spk
