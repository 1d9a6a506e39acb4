// Mel front-end (see melspec.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace spk {
// returns the number of frames (>= 1) or a negative SPK_E* code
int mel_spectrogram(const float* audio, int batch, int64_t samples, int n_fft, int hop, int win, const float* basis,
                    const int32_t* ranges, int n_mels, void* out, int out_fp16, cudaStream_t st);
// Backward with respect to the audio (see melspec.cu): d_audio [batch, samples] = dL/d(audio) for d_mel = dL/d(log-mel).
// bin_ranges: int32 [n_fft / 2 + 1][2] = [first, last + 1) filter with a non-zero weight at each bin.  The workspace
// holds the windowed gradient of every frame.  Returns 0 or a negative SPK_E* code; argument errors come back before
// any CUDA call.
size_t mel_backward_workspace_bytes(int batch, int64_t samples, int n_fft, int hop);   // 0 for a rejected shape
int mel_spectrogram_backward(const float* audio, const float* d_mel, int batch, int64_t samples, int n_fft, int hop,
                             int win, const float* basis, const int32_t* ranges, const int32_t* bin_ranges, int n_mels,
                             float* d_audio, void* workspace, size_t workspace_bytes, cudaStream_t st);
}  // namespace spk
