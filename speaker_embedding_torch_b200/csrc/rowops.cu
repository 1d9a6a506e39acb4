// Bandwidth-bound kernels of the encoder: layout packing, LayerNorm fwd/bwd, softmax fwd/bwd,
// column sums (bias gradients).  All are coalesced 16-byte-vector kernels with warp-shuffle
// reductions; rows of the 256-wide model dimension are handled one warp per row (8 elements / lane).
#include "rowops.h"
#include "ptx.cuh"

#include <cuda_fp16.h>

namespace spk {

// ------------------------------------------------------------------------------------------------
// fp32 weights -> split-fp16 planes, all matrices in one launch.
__global__ void pack_weights_kernel(const __grid_constant__ PackTable tab, elem_t* dst, int64_t plane_stride,
                                    int planes) {
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  for (int s = 0; s < tab.count; ++s) {
    const float* src = tab.seg[s].src;
    const int64_t n = tab.seg[s].n, off = tab.seg[s].dst_off;
    // eight weights per thread and round (two 16-byte loads, one 16-byte store per plane) when the segment allows it
    const bool vec = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && (off & 7) == 0;
    const int64_t n8 = vec ? n / 8 : 0;
    for (int64_t i = tid; i < n8; i += nth) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(src) + 2 * i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(src) + 2 * i + 1);
      const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      store8_split(dst, plane_stride, planes, off + 8 * i, v);
    }
    for (int64_t i = n8 * 8 + tid; i < n; i += nth) store1_split(dst, plane_stride, planes, off + i, __ldg(src + i));
  }
}
int pack_weights(const PackTable& tab, void* dst, int64_t plane_stride, int planes, cudaStream_t st) {
  ProfScope prof("pack_weights", 0, 0, st);
  pack_weights_kernel<<<296, 256, 0, st>>>(tab, reinterpret_cast<elem_t*>(dst), plane_stride, planes);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// mel view -> token-major split tensor [B*T, C]   (C % 8 == 0).  Slice b = window b / spw, frames
// [ (b % spw) * hop, + T ) of a [windows, C, L] tensor in fp32 or fp16 (frames contiguous): the overlapping-slice
// collation and the fp16 -> fp32 upcast of the reference's inference collater happen in this load.
// The shared tile is [C][33] floats (dynamic, 33.8 KB at C = 256).
template <typename TIn>
__global__ void mel_pack_kernel(const TIn* __restrict__ mel, elem_t* __restrict__ out, int64_t plane_stride,
                                int planes, int C, int T, int L, int hop, int spw) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  extern __shared__ float tile[];
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * 32;
  const TIn* src = mel + static_cast<int64_t>(b / spw) * C * L + static_cast<int64_t>(b % spw) * hop;
  for (int i = threadIdx.x; i < C * 32; i += blockDim.x) {
    const int c = i >> 5, tl = i & 31;
    tile[c * 33 + tl] = (t0 + tl < T) ? static_cast<float>(__ldg(src + static_cast<int64_t>(c) * L + t0 + tl)) : 0.f;
  }
  __syncthreads();
  const int G = C / 8;
  for (int i = threadIdx.x; i < G * 32; i += blockDim.x) {
    const int tl = i / G, g = i % G;
    if (t0 + tl >= T) continue;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = tile[(g * 8 + j) * 33 + tl];
    store8_split(out, plane_stride, planes, (static_cast<int64_t>(b) * T + t0 + tl) * C + g * 8, v);
  }
}
int mel_pack(const spk_mel_view& mel, void* out, int64_t plane_stride, int planes, int B, int C, int T, cudaStream_t st) {
  const double in_b = mel.dtype == 1 ? 2.0 : 4.0;
  ProfScope prof("mel_pack", 0, 1.0 * B * C * T * (in_b + 2.0 * planes), st);
  SPK_CHECK(mel.data != nullptr && (mel.dtype == 0 || mel.dtype == 1), "mel view: dtype must be 0 (fp32) or 1 (fp16)");
  SPK_CHECK(mel.slices_per_window >= 1 && B % mel.slices_per_window == 0 && mel.hop >= 0,
            "mel view: batch %d is not a multiple of slices_per_window %d", B, mel.slices_per_window);
  SPK_CHECK(static_cast<int64_t>(mel.slices_per_window - 1) * mel.hop + T <= mel.window_frames,
            "mel view: %d slices of %d frames at hop %d do not fit a %d-frame window", mel.slices_per_window, T, mel.hop,
            mel.window_frames);
  dim3 grid((T + 31) / 32, B);
  const size_t smem = static_cast<size_t>(C) * 33 * sizeof(float);
  auto* o = reinterpret_cast<elem_t*>(out);
  if (mel.dtype == 0)
    mel_pack_kernel<float><<<grid, 256, smem, st>>>(reinterpret_cast<const float*>(mel.data), o, plane_stride, planes, C,
                                                    T, mel.window_frames, mel.hop, mel.slices_per_window);
  else
    mel_pack_kernel<__half><<<grid, 256, smem, st>>>(reinterpret_cast<const __half*>(mel.data), o, plane_stride, planes,
                                                     C, T, mel.window_frames, mel.hop, mel.slices_per_window);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// The mirror of mel_pack_kernel for the input gradient: token-major fp32 [B*T, C] -> d_mel [B, C, T] fp32.  The block's
// 32 tokens are C * 32 consecutive floats on the read side and 32-frame runs of every channel on the write side; the
// shared tile turns one into the other so that both are coalesced.
__global__ void mel_grad_unpack_kernel(const float* __restrict__ src, float* __restrict__ d_mel, int C, int T) {
  extern __shared__ float tile[];   // [C][33]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * 32;
  const int nt = T - t0 < 32 ? T - t0 : 32;
  const float* s = src + (static_cast<int64_t>(b) * T + t0) * C;
  for (int i = threadIdx.x; i < nt * C; i += blockDim.x) tile[(i % C) * 33 + i / C] = __ldg(s + i);
  __syncthreads();
  float* dst = d_mel + static_cast<int64_t>(b) * C * T + t0;
  for (int i = threadIdx.x; i < C * 32; i += blockDim.x) {
    const int c = i >> 5, tl = i & 31;
    if (tl < nt) dst[static_cast<int64_t>(c) * T + tl] = tile[c * 33 + tl];
  }
}
int mel_grad_unpack(const float* src, float* d_mel, int B, int C, int T, cudaStream_t st) {
  ProfScope prof("mel_grad_unpack", 0, 8.0 * B * C * T, st);
  mel_grad_unpack_kernel<<<dim3((T + 31) / 32, B), 256, static_cast<size_t>(C) * 33 * sizeof(float), st>>>(src, d_mel,
                                                                                                            C, T);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// Training collation on the device (Datasets.py:9-19 `Correction`, :72-86 `Collater`): the batch arrives as ONE ragged
// array [C, total_frames] (the utterances' patterns concatenated along time, fp16 as stored or fp32) plus a table
// (start, length, offset) per utterance; every utterance is cut (length > T: frames [offset, offset + T)) or
// reflect-padded (numpy 'reflect', floor / ceil of the missing frames left / right) to the batch's common T inside the
// load that packs the token-major operand planes.  Host-side padded / cropped copies never exist.
template <typename TIn>
__global__ void mel_pack_ragged_kernel(const TIn* __restrict__ mel, const int32_t* __restrict__ table, int64_t total,
                                       elem_t* __restrict__ out, int64_t plane_stride, int planes, int C, int T) {
  extern __shared__ float tile[];   // [C][33]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * 32;
  const int start = __ldg(table + 3 * b), len = __ldg(table + 3 * b + 1), off = __ldg(table + 3 * b + 2);
  const int pad_left = len > T ? 0 : (T - len) / 2;
  const int period = 2 * (len - 1);
  for (int i = threadIdx.x; i < C * 32; i += blockDim.x) {
    const int c = i >> 5, tl = i & 31, t = t0 + tl;
    float v = 0.f;
    if (t < T) {
      int idx;
      if (len > T) {
        idx = off + t;
      } else if (period == 0) {
        idx = 0;
      } else {
        idx = (t - pad_left) % period;
        if (idx < 0) idx += period;
        if (idx >= len) idx = period - idx;
      }
      v = static_cast<float>(__ldg(mel + static_cast<int64_t>(c) * total + start + idx));
    }
    tile[c * 33 + tl] = v;
  }
  __syncthreads();
  const int G = C / 8;
  for (int i = threadIdx.x; i < G * 32; i += blockDim.x) {
    const int tl = i / G, g = i % G;
    if (t0 + tl >= T) continue;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = tile[(g * 8 + j) * 33 + tl];
    store8_split(out, plane_stride, planes, (static_cast<int64_t>(b) * T + t0 + tl) * C + g * 8, v);
  }
}
int mel_pack_ragged(const spk_mel_ragged& mel, void* out, int64_t plane_stride, int planes, int B, int C, int T,
                    cudaStream_t st) {
  ProfScope prof("mel_pack_ragged", 0, 1.0 * B * C * T * ((mel.dtype == 1 ? 2.0 : 4.0) + 2.0 * planes), st);
  SPK_CHECK(mel.data != nullptr && mel.table != nullptr && (mel.dtype == 0 || mel.dtype == 1) && mel.total_frames > 0,
            "ragged mel: data / table missing or dtype not 0 (fp32) / 1 (fp16)");
  dim3 grid((T + 31) / 32, B);
  const size_t smem = static_cast<size_t>(C) * 33 * sizeof(float);
  auto* o = reinterpret_cast<elem_t*>(out);
  if (mel.dtype == 0)
    mel_pack_ragged_kernel<float><<<grid, 256, smem, st>>>(reinterpret_cast<const float*>(mel.data), mel.table,
                                                           mel.total_frames, o, plane_stride, planes, C, T);
  else
    mel_pack_ragged_kernel<__half><<<grid, 256, smem, st>>>(reinterpret_cast<const __half*>(mel.data), mel.table,
                                                            mel.total_frames, o, plane_stride, planes, C, T);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// Adjoint of mel_pack_ragged_kernel (the input gradient of a ragged forward).  Block (group g, column tiles of g's span
// strided by gridDim.y): 32 columns x C channels per tile.  Item i of the tile is (column i / C, channel i % C), so a
// warp reads the C contiguous floats of one token of dX (coalesced) and the tile leaves through shared memory as
// 32-column runs of every channel (coalesced writes), as in mel_grad_unpack_kernel.
//   crop row (length > T)  column p = col - start receives frame t = p - offset when 0 <= t < T;
//   padded row             frames t with (t - pad_left) mod 2 (length - 1) in {p, 2 (length - 1) - p}: two arithmetic
//                          sequences, walked merged in t order (length 1: every frame).
// Table and segment entries are clamped: reads stay inside dX and writes inside d_data whatever the device holds.
__global__ void __launch_bounds__(256) mel_grad_fold_kernel(const float* __restrict__ dx, const int32_t* __restrict__ table,
                                                            const int32_t* __restrict__ segments, int rows_per_group,
                                                            int B, int C, int T, int64_t total, float* __restrict__ d_data) {
  extern __shared__ float tile[];   // [C][33]
  __shared__ int64_t span[2];
  const int g = blockIdx.x;
  int r0, r1;
  if (segments != nullptr) {
    r0 = __ldg(segments + g);
    r1 = __ldg(segments + g + 1);
    r0 = r0 < 0 ? 0 : (r0 > B ? B : r0);
    r1 = r1 < r0 ? r0 : (r1 > B ? B : r1);
  } else {
    r0 = g * rows_per_group;
    r1 = r0 + rows_per_group > B ? B : r0 + rows_per_group;
  }
  if (threadIdx.x == 0) {
    int64_t lo = total, hi = 0;
    for (int r = r0; r < r1; ++r) {
      const int64_t start = __ldg(table + 3 * r), len = __ldg(table + 3 * r + 1);
      if (len < 1) continue;
      lo = start < lo ? start : lo;
      hi = start + len > hi ? start + len : hi;
    }
    span[0] = lo < 0 ? 0 : lo;
    span[1] = hi > total ? total : hi;
  }
  __syncthreads();
  const int64_t lo = span[0], hi = span[1];
  for (int64_t c0 = lo + static_cast<int64_t>(blockIdx.y) * 32; c0 < hi; c0 += static_cast<int64_t>(gridDim.y) * 32) {
    for (int i = threadIdx.x; i < C * 32; i += blockDim.x) {
      const int j = i / C, c = i % C;
      const int64_t col = c0 + j;
      float acc = 0.f;
      if (col < hi) {
        for (int r = r0; r < r1; ++r) {
          const int start = __ldg(table + 3 * r), len = __ldg(table + 3 * r + 1), off = __ldg(table + 3 * r + 2);
          const int64_t p64 = col - start;
          if (len < 1 || p64 < 0 || p64 >= len) continue;
          const int p = static_cast<int>(p64);
          const float* s = dx + static_cast<int64_t>(r) * T * C + c;
          if (len > T) {
            const int t = p - off;
            if (t >= 0 && t < T) acc += __ldg(s + static_cast<int64_t>(t) * C);
          } else if (len == 1) {
            for (int t = 0; t < T; ++t) acc += __ldg(s + static_cast<int64_t>(t) * C);
          } else {
            const int period = 2 * (len - 1), pad_left = (T - len) / 2;
            int ta = (p + pad_left) % period;                                          // rising pieces
            int tb = (p == 0 || p == len - 1) ? T : (period - p + pad_left) % period;  // falling pieces (ends: none)
            while (ta < T || tb < T) {
              if (ta < tb) { acc += __ldg(s + static_cast<int64_t>(ta) * C); ta += period; }
              else { acc += __ldg(s + static_cast<int64_t>(tb) * C); tb += period; }
            }
          }
        }
      }
      tile[c * 33 + j] = acc;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C * 32; i += blockDim.x) {
      const int c = i >> 5, j = i & 31;
      if (c0 + j < hi) d_data[static_cast<int64_t>(c) * total + c0 + j] = tile[c * 33 + j];
    }
    __syncthreads();
  }
}
int mel_grad_fold(const float* src, const spk_mel_ragged& mel, const int32_t* segments, int rows_per_group, int groups,
                  float* d_data, int B, int C, int T, cudaStream_t st) {
  SPK_CHECK(mel.table != nullptr && mel.total_frames > 0 && d_data != nullptr && groups >= 1 &&
                (segments != nullptr || rows_per_group >= 1),
            "mel_grad_fold: bad argument");
  ProfScope prof("mel_grad_fold", 0, 4.0 * C * (static_cast<double>(B) * T + mel.total_frames), st);
  // columns outside every group's span are zero; the fold overwrites the spans (disjoint: one writer per column)
  SPK_CUDA(cudaMemsetAsync(d_data, 0, static_cast<size_t>(C) * mel.total_frames * sizeof(float), st));
  // enough column tiles per group for an average span; longer spans loop
  const int64_t tiles = (mel.total_frames / groups + 31) / 32 + 1;
  dim3 grid(groups, static_cast<unsigned>(tiles < 64 ? tiles : 64));
  mel_grad_fold_kernel<<<grid, 256, static_cast<size_t>(C) * 33 * sizeof(float), st>>>(
      src, mel.table, segments, rows_per_group, B, C, T, mel.total_frames, d_data);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// pe buffer [1, D, max_pos] -> pe_t [T, D]
__global__ void pe_transpose_kernel(const float* __restrict__ pe, float* __restrict__ pe_t, int D, int max_pos, int T) {
  __shared__ float tile[32][33];
  const int t0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 256 threads: 8 rows per pass
  for (int r = ty; r < 32; r += 8) {
    const int d = d0 + r, t = t0 + tx;
    tile[r][tx] = (d < D && t < T) ? __ldg(pe + static_cast<int64_t>(d) * max_pos + t) : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int t = t0 + r, d = d0 + tx;
    if (t < T && d < D) pe_t[static_cast<int64_t>(t) * D + d] = tile[tx][r];
  }
}
int pe_transpose(const float* pe, float* pe_t, int D, int max_pos, int T, cudaStream_t st) {
  ProfScope prof("pe_transpose", 0, 8.0 * D * T, st);
  dim3 grid((T + 31) / 32, (D + 31) / 32);
  pe_transpose_kernel<<<grid, 256, 0, st>>>(pe, pe_t, D, max_pos, T);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over D = 256, one warp per row, NR rows per round: all NR x PL plane loads of a round are issued before any
// row is reduced (one row per round left a single 512-byte row in flight per warp behind the two dependent shuffle
// reductions: 45 % of the DRAM peak, ncu r02).  One-plane (inference) tensors move half the bytes per row and take four
// rows per round.
template <int PL, int NR>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const elem_t* __restrict__ z, int64_t z_ps,
                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     elem_t* __restrict__ y, int64_t y_ps, int y_planes,
                                                     float2* __restrict__ stats, int64_t rows, int64_t row_stride_rows,
                                                     float eps) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float g[8], b[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { g[i] = __ldg(gamma + lane * 8 + i); b[i] = __ldg(beta + lane * 8 + i); }
  for (int64_t r0 = warp; r0 < rows; r0 += NR * nwarps) {
    uint4 raw[NR][PL];
#pragma unroll
    for (int u = 0; u < NR; ++u) {
      const int64_t r = r0 + u * nwarps;
      if (r < rows) {
#pragma unroll
        for (int p = 0; p < PL; ++p)
          raw[u][p] = __ldg(reinterpret_cast<const uint4*>(z + p * z_ps + r * row_stride_rows * 256 + lane * 8));
      }
    }
#pragma unroll
    for (int u = 0; u < NR; ++u) {
      const int64_t r = r0 + u * nwarps;
      if (r >= rows) break;
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = 0.f;
#pragma unroll
      for (int p = 0; p < PL; ++p) {
        const uint32_t w[4] = {raw[u][p].x, raw[u][p].y, raw[u][p].z, raw[u][p].w};
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] += lo_to_f(w[i]); v[2 * i + 1] += hi_to_f(w[i]); }
      }
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s += v[i];
      const float mean = warp_sum(s) * (1.f / 256.f);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { v[i] -= mean; q += v[i] * v[i]; }
      const float rstd = rsqrtf(warp_sum(q) * (1.f / 256.f) + eps);
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = v[i] * rstd * g[i] + b[i];
      store8_split(y, y_ps, y_planes, r * 256 + lane * 8, o);
      if (lane == 0 && stats) stats[r] = make_float2(mean, rstd);
    }
  }
}
int ln_fwd(const void* z, int64_t z_ps, int z_planes, int64_t z_row_step, const float* gamma, const float* beta,
           void* y, int64_t y_ps, int y_planes, float* stats, int64_t rows, cudaStream_t st) {
  ProfScope prof("ln_fwd", 0, 512.0 * rows * (z_planes + y_planes), st);
  SPK_CHECK(z_planes >= 1 && z_planes <= 3, "ln_fwd: planes");
  const int blocks = static_cast<int>(std::min<int64_t>((rows + 7) / 8, 148 * 8));
  const elem_t* zp = reinterpret_cast<const elem_t*>(z);
  elem_t* yp = reinterpret_cast<elem_t*>(y);
  float2* sp = reinterpret_cast<float2*>(stats);
  if (z_planes == 1) ln_fwd_kernel<1, 4><<<blocks, 256, 0, st>>>(zp, z_ps, gamma, beta, yp, y_ps, y_planes, sp, rows, z_row_step, 1e-5f);
  else if (z_planes == 2) ln_fwd_kernel<2, 2><<<blocks, 256, 0, st>>>(zp, z_ps, gamma, beta, yp, y_ps, y_planes, sp, rows, z_row_step, 1e-5f);
  else ln_fwd_kernel<3, 2><<<blocks, 256, 0, st>>>(zp, z_ps, gamma, beta, yp, y_ps, y_planes, sp, rows, z_row_step, 1e-5f);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// dz = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma ; dgamma += dy * xhat ; dbeta += dy
// Optionally also writes dz_drop = dz * keep(site) (the gradient that enters the sub-layer's GEMMs).
// dgamma == nullptr: no parameter gradient at all (dbeta and dbias are then null too); dz / dz_drop are unchanged.
template <int PL>
__global__ void __launch_bounds__(256, 3) ln_bwd_kernel(const elem_t* __restrict__ dy, int64_t dy_ps, int dy_planes_rt,
                                                        const elem_t* __restrict__ z, int64_t z_ps, int z_planes_rt,
                                                     const float2* __restrict__ stats, const float* __restrict__ gamma,
                                                     elem_t* __restrict__ dz, int64_t dz_ps, int dz_planes,
                                                     elem_t* __restrict__ dz_drop, DropCfg drop, uint32_t site,
                                                     float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                     float* __restrict__ dbias, int64_t rows,
                                                     const float* __restrict__ gscale) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  __shared__ float red[3][8][256];
  // PL > 0: both inputs have PL planes (compile-time: fewer registers, three blocks per SM); PL == 0: run-time counts
  const int dy_planes = PL > 0 ? PL : dy_planes_rt, z_planes = PL > 0 ? PL : z_planes_rt;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float g[8], ag[8], ab[8], az[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { g[i] = __ldg(gamma + lane * 8 + i); ag[i] = 0.f; ab[i] = 0.f; az[i] = 0.f; }
  // software pipeline: the raw loads of the next row are issued before the current row is reduced
  uint4 nd[3], nz[3];
  float2 nms = make_float2(0.f, 0.f);
  auto fetch = [&](int64_t r) {
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      if (p < dy_planes) nd[p] = *reinterpret_cast<const uint4*>(dy + p * dy_ps + r * 256 + lane * 8);
      if (p < z_planes) nz[p] = *reinterpret_cast<const uint4*>(z + p * z_ps + r * 256 + lane * 8);
    }
    nms = stats[r];
  };
  auto unpack = [&](const uint4 (&raw)[3], int planes, float (&v)[8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      if (p < planes) {
        const uint32_t w[4] = {raw[p].x, raw[p].y, raw[p].z, raw[p].w};
#pragma unroll
        for (int i = 0; i < 4; ++i) { v[2 * i] += lo_to_f(w[i]); v[2 * i + 1] += hi_to_f(w[i]); }
      }
    }
  };
  if (warp < rows) fetch(warp);
  for (int64_t r = warp; r < rows; r += nwarps) {
    float d[8], x[8];
    unpack(nd, dy_planes, d);
    unpack(nz, z_planes, x);
    const float2 ms = nms;
    if (r + nwarps < rows) fetch(r + nwarps);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      x[i] = (x[i] - ms.x) * ms.y;
      ag[i] += d[i] * x[i];
      ab[i] += d[i];
      d[i] *= g[i];
      s1 += d[i];
      s2 += d[i] * x[i];
    }
    s1 = warp_sum(s1) * (1.f / 256.f);
    s2 = warp_sum(s2) * (1.f / 256.f);
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = ms.y * (d[i] - s1 - x[i] * s2);
    store8_split(dz, dz_ps, dz_planes, r * 256 + lane * 8, o);
    if (dz_drop != nullptr) {
      float k8[8];
      const uint64_t idx = static_cast<uint64_t>(r) * 256 + lane * 8;
      dropout_scale8(drop.seed, site, idx >> 3, drop.thresh, drop.inv_keep, k8);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] *= k8[i];
      store8_split(dz_drop, dz_ps, dz_planes, r * 256 + lane * 8, o);
    }
    // o is now the gradient of the sub-layer output (dz, or dz * keep): its column sum is that layer's bias grad
#pragma unroll
    for (int i = 0; i < 8; ++i) az[i] += o[i];
  }
  if (dgamma == nullptr) return;     // no parameter gradients wanted (block-uniform)
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    red[0][wib][lane * 8 + i] = ag[i]; red[1][wib][lane * 8 + i] = ab[i]; red[2][wib][lane * 8 + i] = az[i];
  }
  __syncthreads();
  float sg = 0.f, sb = 0.f, sz = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) { sg += red[0][w][threadIdx.x]; sb += red[1][w][threadIdx.x]; sz += red[2][w][threadIdx.x]; }
  const float inv_s = gscale != nullptr ? __ldg(gscale + 1) : 1.f;     // the gradients arrive scaled by gscale[0]
  atomicAdd(dgamma + threadIdx.x, sg * inv_s);
  atomicAdd(dbeta + threadIdx.x, sb * inv_s);
  if (dbias != nullptr) atomicAdd(dbias + threadIdx.x, sz * inv_s);
}
int ln_bwd(const void* dy, int64_t dy_ps, int dy_planes, const void* z, int64_t z_ps, int z_planes, const float* stats,
           const float* gamma, void* dz, int64_t dz_ps, int dz_planes, void* dz_drop, DropCfg drop, uint32_t site,
           float* dgamma, float* dbeta, float* dbias, int64_t rows, const float* gscale, cudaStream_t st) {
  ProfScope prof("ln_bwd", 0, 512.0 * rows * (dy_planes + z_planes + dz_planes * (drop.thresh ? 2 : 1)), st);
  const int blocks = static_cast<int>(std::min<int64_t>((rows + 7) / 8, 148 * 6));
  auto kern = (dy_planes == 2 && z_planes == 2) ? ln_bwd_kernel<2> : ln_bwd_kernel<0>;
  kern<<<blocks, 256, 0, st>>>(reinterpret_cast<const elem_t*>(dy), dy_ps, dy_planes,
                                        reinterpret_cast<const elem_t*>(z), z_ps, z_planes,
                                        reinterpret_cast<const float2*>(stats), gamma,
                                        reinterpret_cast<elem_t*>(dz), dz_ps, dz_planes,
                                        (drop.thresh != 0) ? reinterpret_cast<elem_t*>(dz_drop) : nullptr, drop,
                                        site, dgamma, dbeta, dbias, rows, gscale);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Row softmax over the first T of Tp columns (Tp % 8 == 0, Tp <= 1024); one warp per row.
// Writes P (and P_drop = P * keep / (1-p) when dropout is on); pad columns are written as zeros.
template <int CH>
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const elem_t* __restrict__ s,
                                                          const float* __restrict__ s_f32, int64_t ps, int planes,
                                                          elem_t* __restrict__ p, elem_t* __restrict__ p_drop,
                                                          DropCfg drop, uint32_t site, int64_t rows, int T, int Tp) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  // software pipeline for the common case (fp32 scores, T <= 256): next row's loads are issued one row ahead
  const bool pipelined = (CH == 1) && (s_f32 != nullptr) && (lane * 8 < Tp);
  float4 n0 = make_float4(0.f, 0.f, 0.f, 0.f), n1 = n0;
  if (pipelined && warp < rows) {
    n0 = *reinterpret_cast<const float4*>(s_f32 + warp * Tp + lane * 8);
    n1 = *reinterpret_cast<const float4*>(s_f32 + warp * Tp + lane * 8 + 4);
  }
  for (int64_t r = warp; r < rows; r += nwarps) {
    float v[CH][8];
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      const int col = c * 256 + lane * 8;
      if (col < Tp) {
        if (s_f32 != nullptr) {
          float4 a0, a1;
          if (pipelined) {
            a0 = n0; a1 = n1;
            if (r + nwarps < rows) {
              n0 = *reinterpret_cast<const float4*>(s_f32 + (r + nwarps) * Tp + col);
              n1 = *reinterpret_cast<const float4*>(s_f32 + (r + nwarps) * Tp + col + 4);
            }
          } else {
            a0 = *reinterpret_cast<const float4*>(s_f32 + r * Tp + col);
            a1 = *reinterpret_cast<const float4*>(s_f32 + r * Tp + col + 4);
          }
          v[c][0] = a0.x; v[c][1] = a0.y; v[c][2] = a0.z; v[c][3] = a0.w;
          v[c][4] = a1.x; v[c][5] = a1.y; v[c][6] = a1.z; v[c][7] = a1.w;
        } else {
          load8_split(s, ps, planes, r * Tp + col, v[c]);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (col + i >= T) v[c][i] = -INFINITY;
          mx = fmaxf(mx, v[c][i]);
        }
      }
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      const int col = c * 256 + lane * 8;
      if (col < Tp) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { v[c][i] = __expf(v[c][i] - mx); sum += v[c][i]; }
      }
    }
    const float inv = 1.f / warp_sum(sum);
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      const int col = c * 256 + lane * 8;
      if (col < Tp) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[c][i] *= inv;
        // with dropout the un-dropped P is only read by the (two-plane) backward pass: skip its third plane
        store8_split(p, ps, (p_drop != nullptr && planes > 2) ? 2 : planes, r * Tp + col, v[c]);
        if (p_drop != nullptr) {
          float k8[8];
          const uint64_t idx = static_cast<uint64_t>(r) * Tp + col;
          dropout_scale8(drop.seed, site, idx >> 3, drop.thresh, drop.inv_keep, k8);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[c][i] *= k8[i];
          store8_split(p_drop, ps, planes, r * Tp + col, v[c]);
        }
      }
    }
  }
}
int softmax_fwd(const void* s, const float* s_f32, int64_t ps, int planes, void* p, void* p_drop, DropCfg drop,
                uint32_t site, int64_t rows, int T, int Tp, cudaStream_t st) {
  ProfScope prof("softmax_fwd", 0, 2.0 * rows * Tp * planes * (drop.thresh ? 2 : 1) + rows * Tp * (s_f32 ? 4.0 : 2.0 * planes), st);
  SPK_CHECK(Tp % 8 == 0 && Tp <= 1024 && T <= Tp, "softmax: bad row length T=%d Tp=%d", T, Tp);
  const int blocks = static_cast<int>(std::min<int64_t>((rows + 7) / 8, 148 * 8));
  const int ch = (Tp + 255) / 256;
  auto* sp = reinterpret_cast<const elem_t*>(s);
  auto* pp = reinterpret_cast<elem_t*>(p);
  auto* pdp = drop.thresh != 0 ? reinterpret_cast<elem_t*>(p_drop) : nullptr;
  switch (ch) {
    case 1: softmax_fwd_kernel<1><<<blocks, 256, 0, st>>>(sp, s_f32, ps, planes, pp, pdp, drop, site, rows, T, Tp); break;
    case 2: softmax_fwd_kernel<2><<<blocks, 256, 0, st>>>(sp, s_f32, ps, planes, pp, pdp, drop, site, rows, T, Tp); break;
    case 3: softmax_fwd_kernel<3><<<blocks, 256, 0, st>>>(sp, s_f32, ps, planes, pp, pdp, drop, site, rows, T, Tp); break;
    default: softmax_fwd_kernel<4><<<blocks, 256, 0, st>>>(sp, s_f32, ps, planes, pp, pdp, drop, site, rows, T, Tp); break;
  }
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// dS = scale * P * (dP' - sum_k dP'_k P_k),  dP' = dP_drop * keep/(1-p)
// dp and ds may alias (in-place): a warp reads its whole row before writing it, so no __restrict__ here.
template <int CH>
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const elem_t* __restrict__ p,
                                                          const elem_t* dp, const float* dp_f32, int64_t ps,
                                                          int planes, elem_t* ds, DropCfg drop, uint32_t site,
                                                          float scale, int64_t rows, int T, int Tp) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  // software pipeline for the common case (fp32 dP, T <= 256): raw loads of the next row one row ahead
  const bool pipelined = (CH == 1) && (dp_f32 != nullptr) && (lane * 8 < Tp) && planes <= 3;
  float4 n0 = make_float4(0.f, 0.f, 0.f, 0.f), n1 = n0;
  uint4 np[3];
  auto fetch = [&](int64_t r) {
    n0 = *reinterpret_cast<const float4*>(dp_f32 + r * Tp + lane * 8);
    n1 = *reinterpret_cast<const float4*>(dp_f32 + r * Tp + lane * 8 + 4);
#pragma unroll
    for (int q = 0; q < 3; ++q)
      if (q < planes) np[q] = *reinterpret_cast<const uint4*>(p + q * ps + r * Tp + lane * 8);
  };
  if (pipelined && warp < rows) fetch(warp);
  for (int64_t r = warp; r < rows; r += nwarps) {
    float pv[CH][8], dv[CH][8];
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      const int col = c * 256 + lane * 8;
      if (col < Tp) {
        if (pipelined) {
#pragma unroll
          for (int i = 0; i < 8; ++i) pv[c][i] = 0.f;
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            if (q < planes) {
              const uint32_t w[4] = {np[q].x, np[q].y, np[q].z, np[q].w};
#pragma unroll
              for (int i = 0; i < 4; ++i) { pv[c][2 * i] += lo_to_f(w[i]); pv[c][2 * i + 1] += hi_to_f(w[i]); }
            }
          }
          dv[c][0] = n0.x; dv[c][1] = n0.y; dv[c][2] = n0.z; dv[c][3] = n0.w;
          dv[c][4] = n1.x; dv[c][5] = n1.y; dv[c][6] = n1.z; dv[c][7] = n1.w;
          if (r + nwarps < rows) fetch(r + nwarps);
        } else {
        load8_split(p, ps, planes, r * Tp + col, pv[c]);
        if (dp_f32 != nullptr) {
          const float4 a0 = *reinterpret_cast<const float4*>(dp_f32 + r * Tp + col);
          const float4 a1 = *reinterpret_cast<const float4*>(dp_f32 + r * Tp + col + 4);
          dv[c][0] = a0.x; dv[c][1] = a0.y; dv[c][2] = a0.z; dv[c][3] = a0.w;
          dv[c][4] = a1.x; dv[c][5] = a1.y; dv[c][6] = a1.z; dv[c][7] = a1.w;
        } else {
          load8_split(dp, ps, planes, r * Tp + col, dv[c]);
        }
        }
        if (drop.thresh != 0) {
          float k8[8];
          const uint64_t idx = static_cast<uint64_t>(r) * Tp + col;
          dropout_scale8(drop.seed, site, idx >> 3, drop.thresh, drop.inv_keep, k8);
#pragma unroll
          for (int i = 0; i < 8; ++i) dv[c][i] *= k8[i];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (col + i >= T) { pv[c][i] = 0.f; dv[c][i] = 0.f; }
          dot += pv[c][i] * dv[c][i];
        }
      }
    }
    dot = warp_sum(dot);
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      const int col = c * 256 + lane * 8;
      if (col < Tp) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = scale * pv[c][i] * (dv[c][i] - dot);
        store8_split(ds, ps, planes, r * Tp + col, o);
      }
    }
  }
}
int softmax_bwd(const void* p, const void* dp, const float* dp_f32, int64_t ps, int planes, void* ds, DropCfg drop,
                uint32_t site, float scale, int64_t rows, int T, int Tp, cudaStream_t st) {
  ProfScope prof("softmax_bwd", 0, 2.0 * rows * Tp * planes * 3, st);
  SPK_CHECK(Tp % 8 == 0 && Tp <= 1024 && T <= Tp, "softmax: bad row length T=%d Tp=%d", T, Tp);
  const int blocks = static_cast<int>(std::min<int64_t>((rows + 7) / 8, 148 * 8));
  const int ch = (Tp + 255) / 256;
  auto* pp = reinterpret_cast<const elem_t*>(p);
  auto* dpp = reinterpret_cast<const elem_t*>(dp);
  auto* dsp = reinterpret_cast<elem_t*>(ds);
  switch (ch) {
    case 1: softmax_bwd_kernel<1><<<blocks, 256, 0, st>>>(pp, dpp, dp_f32, ps, planes, dsp, drop, site, scale, rows, T, Tp); break;
    case 2: softmax_bwd_kernel<2><<<blocks, 256, 0, st>>>(pp, dpp, dp_f32, ps, planes, dsp, drop, site, scale, rows, T, Tp); break;
    case 3: softmax_bwd_kernel<3><<<blocks, 256, 0, st>>>(pp, dpp, dp_f32, ps, planes, dsp, drop, site, scale, rows, T, Tp); break;
    default: softmax_bwd_kernel<4><<<blocks, 256, 0, st>>>(pp, dpp, dp_f32, ps, planes, dsp, drop, site, scale, rows, T, Tp); break;
  }
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Test aid: the keep-scale (0 or 1 / (1 - p_q)) every dropout site applies to elements [8 * idx8_begin, 8 * (idx8_begin
// + n8)) of its index space -- the same pure function of (seed, site, index) the forward and backward kernels evaluate.
__global__ void dropout_keep_kernel(DropCfg drop, uint32_t site, uint64_t idx8_begin, int64_t n8, float* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float k8[8];
    dropout_scale8(drop.seed, site, idx8_begin + static_cast<uint64_t>(i), drop.thresh, drop.inv_keep, k8);
#pragma unroll
    for (int j = 0; j < 8; ++j) out[i * 8 + j] = k8[j];
  }
}
int dropout_keep(uint64_t seed, float p, uint32_t site, uint64_t idx8_begin, int64_t n8, float* out, cudaStream_t st) {
  SPK_CHECK(out != nullptr && n8 >= 0, "dropout_keep: bad argument");
  if (n8 == 0) return 0;
  const DropCfg drop = make_drop(seed, p, true);
  SPK_CHECK(drop.thresh != 0, "dropout_keep: p must be > 0");
  const int blocks = static_cast<int>(std::min<int64_t>((n8 + 255) / 256, 148 * 8));
  dropout_keep_kernel<<<blocks, 256, 0, st>>>(drop, site, idx8_begin, n8, out);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// out[c] += sum_r x[r, c]   (bias gradients).  C % 8 == 0, C <= 1024.
__global__ void __launch_bounds__(256) colsum_kernel(const elem_t* __restrict__ x, int64_t ps, int planes,
                                                     float* __restrict__ out, int64_t rows, int C, int rows_per_block) {
  const int groups = C / 8;
  const int lanes_r = 256 / groups > 0 ? 256 / groups : 1;   // row lanes per block
  const int g = threadIdx.x % groups, rl = threadIdx.x / groups;
  if (rl >= lanes_r) return;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_block;
  const int64_t r1 = min(r0 + rows_per_block, rows);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int64_t r = r0 + rl; r < r1; r += lanes_r) {
    float v[8];
    load8_split(x, ps, planes, r * C + g * 8, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] += v[i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) atomicAdd(out + g * 8 + i, acc[i]);
}
int colsum(const void* x, int64_t ps, int planes, float* out, int64_t rows, int C, cudaStream_t st) {
  ProfScope prof("colsum", 0, 2.0 * rows * C * planes, st);
  SPK_CHECK(C % 8 == 0 && C / 8 <= 256, "colsum: C=%d unsupported", C);
  const int rpb = 512;
  const int blocks = static_cast<int>((rows + rpb - 1) / rpb);
  colsum_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const elem_t*>(x), ps, planes, out, rows, C, rpb);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// Embedding backward in one pass over dH0 (replaces pe_alpha_grad + a recomputing GEMM):
//   g = dH0 * keep(site 0);   d_alpha += sum g * pe_t[t];   dU = g * 1[u > 0] (mask bits written by the forward prenet
//   epilogue, layout [256 / 32][rows]);   d_bias[col] += sum_rows dU.        Modules.py:50-52,98-105
// dbias == nullptr: only dU is written (dalpha is then null too).
__global__ void __launch_bounds__(256) prenet_bwd_kernel(const elem_t* __restrict__ dh, int64_t ps, int planes,
                                                         const uint32_t* __restrict__ bits, const float* __restrict__ pe_t,
                                                         DropCfg drop, uint32_t site, elem_t* __restrict__ du, int64_t du_ps,
                                                         float* __restrict__ dalpha, float* __restrict__ dbias, int64_t rows,
                                                         int T, const float* __restrict__ gscale) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  __shared__ float red[8];
  __shared__ float cs[8][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float acc = 0.f, col[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) col[i] = 0.f;
  for (int64_t r = warp; r < rows; r += nwarps) {
    float d[8];
    load8_split(dh, ps, planes, r * 256 + lane * 8, d);
    const uint32_t word = __ldg(bits + static_cast<int64_t>(lane >> 2) * rows + r) >> ((lane & 3) * 8);
    if (drop.thresh != 0) {
      float k8[8];
      const uint64_t idx = static_cast<uint64_t>(r) * 256 + lane * 8;
      dropout_scale8(drop.seed, site, idx >> 3, drop.thresh, drop.inv_keep, k8);
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] *= k8[i];
    }
    const float4* pr = reinterpret_cast<const float4*>(pe_t + (r % T) * 256 + lane * 8);
    const float4 p0 = __ldg(pr), p1 = __ldg(pr + 1);
    acc += d[0] * p0.x + d[1] * p0.y + d[2] * p0.z + d[3] * p0.w + d[4] * p1.x + d[5] * p1.y + d[6] * p1.z + d[7] * p1.w;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      d[i] = ((word >> i) & 1u) ? d[i] : 0.f;
      col[i] += d[i];
    }
    store8_split(du, du_ps, planes, r * 256 + lane * 8, d);
  }
  if (dbias == nullptr) return;      // no parameter gradients wanted (block-uniform)
  acc = warp_sum(acc);
  if (lane == 0) red[wib] = acc;
#pragma unroll
  for (int i = 0; i < 8; ++i) cs[wib][lane * 8 + i] = col[i];
  __syncthreads();
  const float inv_s = gscale != nullptr ? __ldg(gscale + 1) : 1.f;
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += cs[w][threadIdx.x];
  atomicAdd(dbias + threadIdx.x, s * inv_s);
  if (threadIdx.x == 0) {
    float a = 0.f;
    for (int w = 0; w < 8; ++w) a += red[w];
    atomicAdd(dalpha, a * inv_s);
  }
}
int prenet_bwd(const void* dh, int64_t ps, int planes, const uint32_t* bits, const float* pe_t, DropCfg drop, uint32_t site,
               void* du, int64_t du_ps, float* dalpha, float* dbias, int64_t rows, int T, const float* gscale,
               cudaStream_t st) {
  ProfScope prof("prenet_bwd", 0, 1024.0 * rows * planes + 32.0 * rows, st);
  const int blocks = static_cast<int>(std::min<int64_t>((rows + 7) / 8, 148 * 4));
  prenet_bwd_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const elem_t*>(dh), ps, planes, bits, pe_t, drop, site,
                                            reinterpret_cast<elem_t*>(du), du_ps, dalpha, dbias, rows, T, gscale);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// d_alpha += sum over tokens/channels of dH0 * keep(site 0) * pe_t[t]
__global__ void __launch_bounds__(256) pe_alpha_grad_kernel(const elem_t* __restrict__ dh, int64_t ps, int planes,
                                                            const float* __restrict__ pe_t, DropCfg drop, uint32_t site,
                                                            float* __restrict__ dalpha, int64_t rows, int T,
                                                            const float* __restrict__ gscale) {
  __shared__ float red[8];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float acc = 0.f;
  for (int64_t r = warp; r < rows; r += nwarps) {
    float d[8];
    load8_split(dh, ps, planes, r * 256 + lane * 8, d);
    if (drop.thresh != 0) {
      float k8[8];
      const uint64_t idx = static_cast<uint64_t>(r) * 256 + lane * 8;
      dropout_scale8(drop.seed, site, idx >> 3, drop.thresh, drop.inv_keep, k8);
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] *= k8[i];
    }
    const float* pr = pe_t + (r % T) * 256 + lane * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += d[i] * __ldg(pr + i);
  }
  acc = warp_sum(acc);
  if (lane == 0) red[wib] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w];
    atomicAdd(dalpha, s * (gscale != nullptr ? __ldg(gscale + 1) : 1.f));
  }
}
int pe_alpha_grad(const void* dh, int64_t ps, int planes, const float* pe_t, DropCfg drop, uint32_t site, float* dalpha,
                  int64_t rows, int T, const float* gscale, cudaStream_t st) {
  if (dalpha == nullptr) return 0;   // the kernel computes nothing else
  ProfScope prof("pe_alpha_grad", 0, 512.0 * rows * planes, st);
  const int blocks = static_cast<int>(std::min<int64_t>((rows + 7) / 8, 148 * 4));
  pe_alpha_grad_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const elem_t*>(dh), ps, planes, pe_t, drop, site,
                                               dalpha, rows, T, gscale);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace spk
