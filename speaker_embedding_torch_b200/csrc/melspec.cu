// Mel front-end on the device (SURVEY.md 8f N3): the reference's `mel_spectrogram` (meldataset.py:73-96, called from
// Inference.py:59-85 and Pattern_Generator.py:93-106) -- reflect padding, STFT (periodic Hann window, center = False),
// magnitude sqrt(re^2 + im^2 + 1e-9), triangular mel filters, log(clamp(., 1e-5)) -- as ONE kernel: audio in, log-mel
// [B, n_mels, frames] out; the spectrogram never exists in global memory.
//
// Per frame (256 threads, frames are looped over by persistent CTAs):
//   load     n_fft windowed samples (reflect index at the edges) packed as N/2 complex numbers z[m] = x[2m] + i x[2m+1],
//            written to shared memory in bit-reversed order
//   FFT      N/2-point complex radix-2 DIT in shared memory, twiddles from a table built once per CTA (sincospi)
//   unpack   X[k] = (Z[k] + conj Z[N/2-k]) / 2 - i W_N^k (Z[k] - conj Z[N/2-k]) / 2,  k = 0 .. N/2   (real-input FFT)
//   mel      thread m < n_mels: sum over the filter's non-zero bin range [lo_m, hi_m)   (the filters are sparse)
// HBM traffic per frame: hop new samples in, n_mels values out -- bandwidth-trivial; the kernel is bound by its
// shared-memory butterflies (~5 N log2 N / 2 flops per frame).
//
// Backward with respect to the audio (DESIGN.md 3.6): melspec_bwd_kernel recomputes each frame with the same stage
// functions and writes the frame's windowed gradient to a workspace; melspec_gather_kernel overlap-adds the frames and
// folds the reflect padding back, one thread per sample, without atomics.
#include "common.cuh"
#include "melspec.h"

namespace spk {

// ---- per-frame stages, shared by the forward and the backward (inlined: the forward's SASS is what it was before)
template <int NFFT>
struct Fft {
  static constexpr int H = NFFT / 2;        // complex FFT size
  static constexpr int LOGH = NFFT == 512 ? 8 : (NFFT == 1024 ? 9 : 10);
};

// Twiddles W_H^k (k < H/2) and W_NFFT^k (k <= H/2), and the periodic Hann window: built once per CTA.
template <int NFFT>
__device__ __forceinline__ void fft_tables(float2* tw, float2* tw2, float* window, int win, int tid) {
  constexpr int H = Fft<NFFT>::H;
  for (int k = tid; k < H / 2; k += 256) {
    float s, c;
    sincospif(-2.f * k / H, &s, &c);
    tw[k] = make_float2(c, s);
  }
  for (int k = tid; k <= H / 2; k += 256) {
    float s, c;
    sincospif(-2.f * k / NFFT, &s, &c);
    tw2[k] = make_float2(c, s);
  }
  const int wl = (NFFT - win) / 2;          // torch.stft centres a short window inside n_fft
  for (int n = tid; n < NFFT; n += 256) {
    const int j = n - wl;
    window[n] = (j >= 0 && j < win) ? 0.5f - 0.5f * cospif(2.f * j / win) : 0.f;     // periodic Hann
  }
}

// The frame's windowed samples z[m] = x[2m] + i x[2m+1], stored at the bit-reversed index of m.
template <int NFFT>
__device__ __forceinline__ void load_frame(const float* __restrict__ src, int64_t samples, int64_t period,
                                           int64_t start, const float* window, float2* z, int tid) {
  constexpr int H = Fft<NFFT>::H, LOGH = Fft<NFFT>::LOGH;
  for (int m = tid; m < H; m += 256) {
    float v[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      int64_t i = start + 2 * m + e;
      if (i < 0 || i >= samples) {        // reflect (no edge repeat), as F.pad(mode='reflect')
        if (period == 0) {
          i = 0;
        } else {
          i %= period;
          if (i < 0) i += period;
          if (i >= samples) i = period - i;
        }
      }
      v[e] = __ldg(src + i) * window[2 * m + e];
    }
    z[__brev(static_cast<unsigned>(m)) >> (32 - LOGH)] = make_float2(v[0], v[1]);
  }
}

// H-point radix-2 DIT butterflies in place: bit-reversed input, natural-order output, W_H = e^{-2 pi i / H}.
template <int NFFT>
__device__ __forceinline__ void fft_stages(float2* z, const float2* tw, int tid) {
  constexpr int H = Fft<NFFT>::H, LOGH = Fft<NFFT>::LOGH;
#pragma unroll 1
  for (int s = 0; s < LOGH; ++s) {
    const int half = 1 << s;
    for (int t = tid; t < H / 2; t += 256) {
      const int grp = t >> s, pos = t & (half - 1);
      const int i0 = (grp << (s + 1)) + pos, i1 = i0 + half;
      const float2 w = tw[pos << (LOGH - 1 - s)];
      const float2 a = z[i0], bq = z[i1];
      const float2 wb = make_float2(w.x * bq.x - w.y * bq.y, w.x * bq.y + w.y * bq.x);
      z[i0] = make_float2(a.x + wb.x, a.y + wb.y);
      z[i1] = make_float2(a.x - wb.x, a.y - wb.y);
    }
    __syncthreads();
  }
}

// W_NFFT^k for k = 0 .. H from the half table: W^k = -conj W^(H-k).
template <int NFFT>
__device__ __forceinline__ float2 twiddle_n(const float2* tw2, int k) {
  constexpr int H = Fft<NFFT>::H;
  return k <= H / 2 ? tw2[k] : make_float2(-tw2[H - k].x, tw2[H - k].y);
}

// Real-FFT unpack of bin k = 0 .. H: X[k] = (Z[k] + conj Z[H-k]) / 2 - i W_N^k (Z[k] - conj Z[H-k]) / 2.
template <int NFFT>
__device__ __forceinline__ float2 unpack_bin(const float2* z, const float2* tw2, int k) {
  constexpr int H = Fft<NFFT>::H;
  const float2 a = z[k & (H - 1)], bq = z[(H - k) & (H - 1)];
  const float er = 0.5f * (a.x + bq.x), ei = 0.5f * (a.y - bq.y);     // even part:  (Z[k] + conj Z[H-k]) / 2
  const float orr = 0.5f * (a.y + bq.y), oi = -0.5f * (a.x - bq.x);   // odd part:   (Z[k] - conj Z[H-k]) / (2i)
  const float2 w = twiddle_n<NFFT>(tw2, k);
  return make_float2(er + w.x * orr - w.y * oi, ei + w.x * oi + w.y * orr);
}

// Filter m's sum over its non-zero bin range [lo_m, hi_m).
__device__ __forceinline__ float mel_band(const float* __restrict__ basis, const int2* __restrict__ ranges,
                                          const float* mag, int bins, int m) {
  const int2 r = ranges[m];
  const float* brow = basis + static_cast<int64_t>(m) * bins;
  float acc = 0.f;
  for (int k = r.x; k < r.y; ++k) acc = fmaf(__ldg(brow + k), mag[k], acc);
  return acc;
}

template <int NFFT>
__global__ void __launch_bounds__(256) melspec_kernel(const float* __restrict__ audio, int64_t samples, int pad, int hop,
                                                      int win, int frames, int64_t total_frames,
                                                      const float* __restrict__ basis, const int2* __restrict__ ranges,
                                                      int n_mels, float* __restrict__ out_f32, __half* __restrict__ out_f16) {
  constexpr int H = Fft<NFFT>::H;
  __shared__ float2 z[H];
  __shared__ float2 tw[H / 2];              // W_H^k,  k < H/2
  __shared__ float2 tw2[H / 2 + 1];         // W_NFFT^k, k <= H/2
  __shared__ float window[NFFT];
  __shared__ float mag[H + 1];
  const int tid = threadIdx.x;
  fft_tables<NFFT>(tw, tw2, window, win, tid);
  __syncthreads();
  const int64_t period = 2 * (samples - 1);
  for (int64_t f = blockIdx.x; f < total_frames; f += gridDim.x) {
    const int64_t b = f / frames;
    const int fr = static_cast<int>(f % frames);
    load_frame<NFFT>(audio + b * samples, samples, period, static_cast<int64_t>(fr) * hop - pad, window, z, tid);
    __syncthreads();
    fft_stages<NFFT>(z, tw, tid);
    for (int k = tid; k <= H; k += 256) {
      const float2 x = unpack_bin<NFFT>(z, tw2, k);
      mag[k] = sqrtf(x.x * x.x + x.y * x.y + 1e-9f);
    }
    __syncthreads();
    if (tid < n_mels) {
      const float v = logf(fmaxf(mel_band(basis, ranges, mag, H + 1, tid), 1e-5f));
      const int64_t o = (b * n_mels + tid) * frames + fr;
      if (out_f32 != nullptr) out_f32[o] = v;
      else out_f16[o] = __float2half_rn(v);
    }
    __syncthreads();
  }
}

// Backward, per frame (same CTA shape and frame loop as the forward; nothing is saved by the forward):
//   recompute   load, FFT, unpack: X[k] = re + i im, mag[k]; acc[m] = sum_k basis[m,k] mag[k]   (the forward's code)
//   clamp gate  dacc[m] = g[m] / acc[m] if acc[m] >= 1e-5 (torch's clamp(min=) passes the gradient at equality), else 0
//   filters     dmag[k] = sum over m in bin_ranges[k] of basis[m,k] dacc[m]                       (fixed order)
//   magnitude   G[k] = dmag[k] X[k] / mag[k]                     (dL/dre + i dL/dim)
//   adjoint DFT dseg[n] = Re sum_{k=0..H} G[k] e^{+2 pi i k n / N}: the adjoint of the unpack,
//                 dZ[j] = (G[j] + conj G[H-j] + i conj(W_N^j) (G[j] - conj G[H-j])) / 2      j = 1 .. H-1
//                 dZ[0] = (1 + i) Re G[0] + (1 - i) Re G[H]                    (Im G[0], Im G[H] drop out)
//               then dz[m] = sum_j dZ[j] e^{+2 pi i j m / H} as conj(FFT(conj dZ)) on the forward's butterflies,
//               dseg[2m] = Re dz[m], dseg[2m+1] = Im dz[m]
//   out         window[n] * dseg[n] -> seg [frame][NFFT]  (overlap-add and reflect fold: melspec_gather_kernel)
template <int NFFT>
__global__ void __launch_bounds__(256) melspec_bwd_kernel(const float* __restrict__ audio, const float* __restrict__ d_mel,
                                                          int64_t samples, int pad, int hop, int win, int frames,
                                                          int64_t total_frames, const float* __restrict__ basis,
                                                          const int2* __restrict__ ranges,
                                                          const int2* __restrict__ bin_ranges, int n_mels,
                                                          float* __restrict__ seg) {
  constexpr int H = Fft<NFFT>::H, LOGH = Fft<NFFT>::LOGH;
  __shared__ float2 z[H];
  __shared__ float2 tw[H / 2];
  __shared__ float2 tw2[H / 2 + 1];
  __shared__ float window[NFFT];
  __shared__ float2 spec[H + 1];            // X[k], then G[k]
  __shared__ float mag[H + 1];
  __shared__ float dacc[256];
  const int tid = threadIdx.x;
  fft_tables<NFFT>(tw, tw2, window, win, tid);
  __syncthreads();
  const int64_t period = 2 * (samples - 1);
  for (int64_t f = blockIdx.x; f < total_frames; f += gridDim.x) {
    const int64_t b = f / frames;
    const int fr = static_cast<int>(f % frames);
    load_frame<NFFT>(audio + b * samples, samples, period, static_cast<int64_t>(fr) * hop - pad, window, z, tid);
    __syncthreads();
    fft_stages<NFFT>(z, tw, tid);
    for (int k = tid; k <= H; k += 256) {
      const float2 x = unpack_bin<NFFT>(z, tw2, k);
      spec[k] = x;
      mag[k] = sqrtf(x.x * x.x + x.y * x.y + 1e-9f);
    }
    __syncthreads();
    if (tid < n_mels) {
      const float acc = mel_band(basis, ranges, mag, H + 1, tid);
      const float g = __ldg(d_mel + (b * n_mels + tid) * frames + fr);
      dacc[tid] = acc >= 1e-5f ? g / acc : 0.f;
    }
    __syncthreads();
    for (int k = tid; k <= H; k += 256) {
      const int2 r = bin_ranges[k];
      float d = 0.f;
      for (int m = r.x; m < r.y; ++m) d = fmaf(__ldg(basis + static_cast<int64_t>(m) * (H + 1) + k), dacc[m], d);
      const float s = d / mag[k];
      spec[k] = make_float2(s * spec[k].x, s * spec[k].y);
    }
    __syncthreads();
    for (int j = tid; j < H; j += 256) {
      float2 dz;
      if (j == 0) {
        const float g0 = spec[0].x, gh = spec[H].x;
        dz = make_float2(g0 + gh, g0 - gh);
      } else {
        const float2 a = spec[j], c = spec[H - j];                     // G[j], G[H-j]
        const float pr = a.x + c.x, pi = a.y - c.y;                    // P = G[j] + conj G[H-j]
        const float qr = a.x - c.x, qi = a.y + c.y;                    // Q = G[j] - conj G[H-j]
        const float2 w = twiddle_n<NFFT>(tw2, j);                      // i conj(W) Q = (w.y qr - w.x qi) + i (w.x qr + w.y qi)
        dz = make_float2(0.5f * (pr + w.y * qr - w.x * qi), 0.5f * (pi + w.x * qr + w.y * qi));
      }
      z[__brev(static_cast<unsigned>(j)) >> (32 - LOGH)] = make_float2(dz.x, -dz.y);
    }
    __syncthreads();
    fft_stages<NFFT>(z, tw, tid);
    float2* out = reinterpret_cast<float2*>(seg + f * NFFT);
    for (int m = tid; m < H; m += 256) {
      const float2 r = z[m];
      out[m] = make_float2(r.x * window[2 * m], -r.y * window[2 * m + 1]);
    }
    __syncthreads();
  }
}

// Sum of the windowed frame gradients at padded position p, over the frames f with f * hop <= p < f * hop + n_fft
// in increasing order.
__device__ __forceinline__ float covering_frames(const float* __restrict__ seg, int64_t p, int hop, int n_fft,
                                                 int frames) {
  const int64_t lo = p >= n_fft ? (p - n_fft) / hop + 1 : 0;
  const int64_t hi = min(p / hop, static_cast<int64_t>(frames) - 1);
  float acc = 0.f;
  for (int64_t f = lo; f <= hi; ++f) acc += __ldg(seg + f * n_fft + (p - f * hop));
  return acc;
}

// dL/d(audio): one thread per sample s of utterance b, adding in a fixed order (deterministic, no atomics) the frames
// that cover padded position pad + s, then its left mirror pad - s (1 <= s <= pad), then its right mirror
// pad + 2 (S - 1) - s (s <= S - 2, inside the padded signal).  Padded positions past the last frame get nothing.
__global__ void __launch_bounds__(256) melspec_gather_kernel(const float* __restrict__ seg, int64_t samples, int pad,
                                                             int hop, int n_fft, int frames, int64_t total,
                                                             float* __restrict__ d_audio) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int64_t b = i / samples, s = i % samples;
  const float* src = seg + b * frames * static_cast<int64_t>(n_fft);
  float acc = covering_frames(src, pad + s, hop, n_fft, frames);
  if (s >= 1 && s <= pad) acc += covering_frames(src, pad - s, hop, n_fft, frames);
  const int64_t right = pad + 2 * (samples - 1) - s;
  if (s <= samples - 2 && right < samples + 2 * static_cast<int64_t>(pad))
    acc += covering_frames(src, right, hop, n_fft, frames);
  d_audio[i] = acc;
}

int mel_spectrogram(const float* audio, int batch, int64_t samples, int n_fft, int hop, int win, const float* basis,
                    const int32_t* ranges, int n_mels, void* out, int out_fp16, cudaStream_t st) {
  SPK_CHECK(audio && basis && ranges && out, "mel_spectrogram: null argument");
  SPK_CHECK(n_fft == 512 || n_fft == 1024 || n_fft == 2048, "mel_spectrogram: n_fft %d not in {512, 1024, 2048}", n_fft);
  SPK_CHECK(hop >= 1 && win >= 1 && win <= n_fft && n_mels >= 1 && n_mels <= 256, "mel_spectrogram: bad hop / win / n_mels");
  const int pad = (n_fft - hop) / 2;
  SPK_CHECK(batch >= 1 && samples > pad, "mel_spectrogram: %lld samples cannot be reflect-padded by %d",
            static_cast<long long>(samples), pad);
  const int64_t padded = samples + 2 * pad;
  SPK_CHECK(padded >= n_fft, "mel_spectrogram: signal shorter than one frame");
  const int frames = static_cast<int>(1 + (padded - n_fft) / hop);
  const int64_t total = static_cast<int64_t>(batch) * frames;
  int sms = 148;
  {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int grid = static_cast<int>(std::min<int64_t>(total, static_cast<int64_t>(sms) * 8));
  // algorithmic work: 2.5 N log2 N (real FFT) + 2 * bins * ~2 filters per frame; bytes: hop samples in, n_mels out
  ProfScope prof("mel_spectrogram", total * (2.5 * n_fft * 10 + 4.0 * (n_fft / 2 + 1)),
                 total * (4.0 * hop + (out_fp16 ? 2.0 : 4.0) * n_mels), st);
  float* o32 = out_fp16 ? nullptr : reinterpret_cast<float*>(out);
  __half* o16 = out_fp16 ? reinterpret_cast<__half*>(out) : nullptr;
  const int2* rg = reinterpret_cast<const int2*>(ranges);
  if (n_fft == 512)
    melspec_kernel<512><<<grid, 256, 0, st>>>(audio, samples, pad, hop, win, frames, total, basis, rg, n_mels, o32, o16);
  else if (n_fft == 1024)
    melspec_kernel<1024><<<grid, 256, 0, st>>>(audio, samples, pad, hop, win, frames, total, basis, rg, n_mels, o32, o16);
  else
    melspec_kernel<2048><<<grid, 256, 0, st>>>(audio, samples, pad, hop, win, frames, total, basis, rg, n_mels, o32, o16);
  SPK_CUDA(cudaGetLastError());
  return frames;
}

// Shape checks of the backward; returns 0 or SPK_EINVAL with the message set.  The backward accepts what the forward
// accepts except hop > n_fft, where the forward's padding (n_fft - hop) / 2 is negative and frames skip samples.
static int mel_backward_shape(int batch, int64_t samples, int n_fft, int hop, int* pad, int* frames) {
  SPK_CHECK(n_fft == 512 || n_fft == 1024 || n_fft == 2048, "mel_spectrogram_backward: n_fft %d not in {512, 1024, 2048}",
            n_fft);
  SPK_CHECK(hop >= 1 && hop <= n_fft, "mel_spectrogram_backward: hop %d not in [1, n_fft = %d]", hop, n_fft);
  *pad = (n_fft - hop) / 2;
  SPK_CHECK(batch >= 1 && samples > *pad, "mel_spectrogram_backward: %lld samples cannot be reflect-padded by %d",
            static_cast<long long>(samples), *pad);
  const int64_t padded = samples + 2 * static_cast<int64_t>(*pad);
  SPK_CHECK(padded >= n_fft, "mel_spectrogram_backward: signal shorter than one frame");
  *frames = static_cast<int>(1 + (padded - n_fft) / hop);
  return 0;
}

size_t mel_backward_workspace_bytes(int batch, int64_t samples, int n_fft, int hop) {
  int pad = 0, frames = 0;
  if (mel_backward_shape(batch, samples, n_fft, hop, &pad, &frames) != 0) return 0;
  return static_cast<size_t>(batch) * frames * n_fft * sizeof(float);
}

int mel_spectrogram_backward(const float* audio, const float* d_mel, int batch, int64_t samples, int n_fft, int hop,
                             int win, const float* basis, const int32_t* ranges, const int32_t* bin_ranges, int n_mels,
                             float* d_audio, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  SPK_CHECK(audio && d_mel && basis && ranges && bin_ranges && d_audio && workspace,
            "mel_spectrogram_backward: null argument");
  int pad = 0, frames = 0;
  SPK_TRY(mel_backward_shape(batch, samples, n_fft, hop, &pad, &frames));
  SPK_CHECK(win >= 1 && win <= n_fft && n_mels >= 1 && n_mels <= 256, "mel_spectrogram_backward: bad win / n_mels");
  const size_t need = mel_backward_workspace_bytes(batch, samples, n_fft, hop);
  SPK_CHECK(workspace_bytes >= need, "mel_spectrogram_backward: workspace of %zu bytes, %zu needed", workspace_bytes,
            need);
  SPK_CHECK(reinterpret_cast<uintptr_t>(workspace) % 16 == 0, "mel_spectrogram_backward: workspace not 16-byte aligned");
  const int64_t total = static_cast<int64_t>(batch) * frames;
  int sms = 148;
  {
    int dev = 0;
    SPK_CUDA(cudaGetDevice(&dev));
    SPK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int grid = static_cast<int>(std::min<int64_t>(total, static_cast<int64_t>(sms) * 8));
  float* seg = reinterpret_cast<float*>(workspace);
  const int2* rg = reinterpret_cast<const int2*>(ranges);
  const int2* brg = reinterpret_cast<const int2*>(bin_ranges);
  {
    // the forward's work twice (the recompute and the adjoint FFT) plus the two filter projections; bytes: hop
    // samples and n_mels gradients in, one windowed frame gradient out
    ProfScope prof("mel_spectrogram.bwd", total * (2 * 2.5 * n_fft * 10 + 8.0 * (n_fft / 2 + 1)),
                   total * (4.0 * hop + 4.0 * n_mels + 4.0 * n_fft), st);
    if (n_fft == 512)
      melspec_bwd_kernel<512><<<grid, 256, 0, st>>>(audio, d_mel, samples, pad, hop, win, frames, total, basis, rg, brg,
                                                    n_mels, seg);
    else if (n_fft == 1024)
      melspec_bwd_kernel<1024><<<grid, 256, 0, st>>>(audio, d_mel, samples, pad, hop, win, frames, total, basis, rg, brg,
                                                     n_mels, seg);
    else
      melspec_bwd_kernel<2048><<<grid, 256, 0, st>>>(audio, d_mel, samples, pad, hop, win, frames, total, basis, rg, brg,
                                                     n_mels, seg);
    SPK_CUDA(cudaGetLastError());
  }
  const int64_t n = static_cast<int64_t>(batch) * samples;
  // one add per covering frame; bytes: every frame gradient read once, the audio gradient written
  ProfScope prof("mel_spectrogram.bwd_gather", static_cast<double>(total) * n_fft,
                 total * 4.0 * n_fft + n * 4.0, st);
  melspec_gather_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(seg, samples, pad, hop, n_fft, frames,
                                                                                n, d_audio);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace spk
