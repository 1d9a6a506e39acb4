// Last-layer attention for the single query row t = 0.
//
// The d-vector head consumes only the first frame of the last encoder layer (Modules.py:54,
// `x.permute(1, 2, 0)[:, :, :1]`), so in that layer only the t = 0 query is ever needed: K and V are
// still projected for every frame, but Q, the attention output, out-proj, both LayerNorms and the FFN
// run on one row per slice (exact; SURVEY.md Appendix B, "Last layer").  With one query per (slice, head)
// the score / softmax / PV contraction is 2 x T x 64 MACs -- a bandwidth-bound sweep over K and V that
// is done here in fp32 by one warp per (slice, head), forward and backward.
//
// Layouts: q0 [B, 256] and kv [B*T, 512] (K | V, head h at columns h*64) are split-fp16 tensors;
// probabilities p / p*keep are kept in fp32 [B*H, Tp] for the backward pass.
#include "rowops.h"
#include "ptx.cuh"

namespace spk {

constexpr int R0_WARPS = 4;   // warps per block == heads of one slice

__device__ __forceinline__ float2 load2_split(const elem_t* base, int64_t ps, int planes, int64_t off) {
  float2 r = make_float2(0.f, 0.f);
  for (int p = 0; p < planes; ++p) {
    const uint32_t w = *reinterpret_cast<const uint32_t*>(base + p * ps + off);
    r.x += lo_to_f(w);
    r.y += hi_to_f(w);
  }
  return r;
}
__device__ __forceinline__ void store2_split(elem_t* base, int64_t ps, int planes, int64_t off, float a, float b) {
  for (int p = 0; p < planes; ++p) {
    const uint32_t q = pack2(a, b);
    *reinterpret_cast<uint32_t*>(base + p * ps + off) = q;
    a -= lo_to_f(q);
    b -= hi_to_f(q);
  }
}
__device__ __forceinline__ float keep_of(const DropCfg& d, uint32_t site, uint64_t idx) {
  if (d.thresh == 0) return 1.f;
  float k8[8];
  dropout_scale8(d.seed, site, idx >> 3, d.thresh, d.inv_keep, k8);
  return k8[idx & 7];
}

// One warp per (slice b, head h).  Lane (g = lane >> 3, d8 = lane & 7): key group g handles keys t = 4 i + g,
// d8 selects 8 consecutive head dims (one 16-byte load per plane), so a warp instruction moves 4 keys x 128 B
// and the per-key reduction is 3 shuffles inside an 8-lane group.
__device__ __forceinline__ void load8f(const elem_t* base, int64_t ps, int planes, int64_t off, float (&v)[8]) {
  load8_split(base, ps, planes, off, v);
}
// Four rows (one per unrolled key step) of a PL-plane tensor: all 4 x PL 16-byte loads are issued before any is decoded,
// so a warp keeps 4 x PL x 512 B in flight (the plane loop of load8_split has a run-time bound and serialised them:
// ncu r02 showed one key step in flight per warp and 30 % of the DRAM peak).
template <int PL>
__device__ __forceinline__ void load_rows4(const elem_t* __restrict__ base, int64_t ps, const int64_t (&off)[4],
                                           float (&v)[4][8]) {
  uint4 raw[4][PL];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
#pragma unroll
    for (int p = 0; p < PL; ++p) raw[u][p] = __ldg(reinterpret_cast<const uint4*>(base + p * ps + off[u]));
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[u][i] = 0.f;
#pragma unroll
    for (int p = 0; p < PL; ++p) {
      const uint32_t w[4] = {raw[u][p].x, raw[u][p].y, raw[u][p].z, raw[u][p].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        v[u][2 * i] += lo_to_f(w[i]);
        v[u][2 * i + 1] += hi_to_f(w[i]);
      }
    }
  }
}
__device__ __forceinline__ float group8_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

template <int PL>
__global__ void __launch_bounds__(32 * R0_WARPS) attn_row0_fwd_kernel(
    const elem_t* __restrict__ q0, int64_t q_ps, const elem_t* __restrict__ kv, int64_t kv_ps, int planes,
    elem_t* __restrict__ att0, int64_t a_ps, float* __restrict__ p0, float* __restrict__ pd0, DropCfg drop,
    uint32_t site, int B, int H, int T, int Tp) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t bh = static_cast<int64_t>(blockIdx.x) * R0_WARPS + warp;
  if (bh >= static_cast<int64_t>(B) * H) return;
  const int b = static_cast<int>(bh / H), h = static_cast<int>(bh % H);
  const int g = lane >> 3, d8 = lane & 7;
  float* sc = sm + warp * Tp;
  float q[8];
  load8f(q0, q_ps, planes, static_cast<int64_t>(b) * 256 + h * 64 + d8 * 8, q);
  const int64_t kv_row0 = static_cast<int64_t>(b) * T * 512 + h * 64 + d8 * 8;
  // scores: 16 keys per round (four key steps of four groups)
  for (int t0 = 0; t0 < T; t0 += 16) {
    int64_t off[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) off[u] = kv_row0 + static_cast<int64_t>(min(t0 + 4 * u + g, T - 1)) * 512;
    float k[4][8];
    load_rows4<PL>(kv, kv_ps, off, k);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s = fmaf(q[i], k[u][i], s);
      s = group8_sum(s);
      if (d8 == 0 && t0 + 4 * u + g < T) sc[t0 + 4 * u + g] = s * 0.125f;
    }
  }
  __syncwarp();
  float mx = -INFINITY;
  for (int t = lane; t < T; t += 32) mx = fmaxf(mx, sc[t]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int t = lane; t < T; t += 32) {
    const float e = __expf(sc[t] - mx);
    sc[t] = e;
    sum += e;
  }
  const float inv = 1.f / warp_sum(sum);
  for (int t = lane; t < Tp; t += 32) {
    float p = 0.f, pd = 0.f;
    if (t < T) {
      p = sc[t] * inv;
      pd = p * keep_of(drop, site, static_cast<uint64_t>(bh) * Tp + t);
      sc[t] = pd;
    }
    if (p0 != nullptr) {
      p0[bh * Tp + t] = p;
      pd0[bh * Tp + t] = pd;
    }
  }
  __syncwarp();
  // o = sum_t pd_t V_t : each key group accumulates its keys, then the four groups are combined
  float o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int t0 = 0; t0 < T; t0 += 16) {
    int64_t off[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) off[u] = kv_row0 + 256 + static_cast<int64_t>(min(t0 + 4 * u + g, T - 1)) * 512;
    float v[4][8];
    load_rows4<PL>(kv, kv_ps, off, v);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = t0 + 4 * u + g;
      const float pd = t < T ? sc[t] : 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = fmaf(pd, v[u][i], o[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    o[i] += __shfl_xor_sync(0xffffffffu, o[i], 8);
    o[i] += __shfl_xor_sync(0xffffffffu, o[i], 16);
  }
  if (g == 0) store8_split(att0, a_ps, planes, static_cast<int64_t>(b) * 256 + h * 64 + d8 * 8, o);
}

int attn_row0_fwd(const void* q0, int64_t q_ps, const void* kv, int64_t kv_ps, int planes, void* att0, int64_t a_ps,
                  float* p0, float* pd0, DropCfg drop, uint32_t site, int B, int H, int T, int Tp, cudaStream_t st) {
  SPK_CHECK(H == R0_WARPS, "attn_row0: %d heads unsupported", H);
  ProfScope prof("attn_row0_fwd", 4.0 * B * H * T * 64, 2.0 * B * T * 512 * planes, st);
  const int blocks = (B * H + R0_WARPS - 1) / R0_WARPS;
  if (planes == 1) {
    constexpr int PLV = 1;
    attn_row0_fwd_kernel<PLV><<<blocks, 32 * R0_WARPS, R0_WARPS * Tp * sizeof(float), st>>>(
      reinterpret_cast<const elem_t*>(q0), q_ps, reinterpret_cast<const elem_t*>(kv), kv_ps, planes,
      reinterpret_cast<elem_t*>(att0), a_ps, p0, pd0, drop, site, B, H, T, Tp);
  } else if (planes == 2) {
    constexpr int PLV = 2;
    attn_row0_fwd_kernel<PLV><<<blocks, 32 * R0_WARPS, R0_WARPS * Tp * sizeof(float), st>>>(
      reinterpret_cast<const elem_t*>(q0), q_ps, reinterpret_cast<const elem_t*>(kv), kv_ps, planes,
      reinterpret_cast<elem_t*>(att0), a_ps, p0, pd0, drop, site, B, H, T, Tp);
  } else {
    constexpr int PLV = 3;
    attn_row0_fwd_kernel<PLV><<<blocks, 32 * R0_WARPS, R0_WARPS * Tp * sizeof(float), st>>>(
      reinterpret_cast<const elem_t*>(q0), q_ps, reinterpret_cast<const elem_t*>(kv), kv_ps, planes,
      reinterpret_cast<elem_t*>(att0), a_ps, p0, pd0, drop, site, B, H, T, Tp);
  }
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// Backward: given d(att0), produces dq0 [B,256], dense dK | dV rows [B*T, 512] and the three in-proj bias
// gradient slices.  p*dp' = pd*dp (pd = p*keep), so the saved p / pd pair is all the dropout state needed.
template <int PL>
__global__ void __launch_bounds__(32 * R0_WARPS) attn_row0_bwd_kernel(
    const elem_t* __restrict__ datt0, int64_t da_ps, int g_planes, const elem_t* __restrict__ q0,
    int64_t q_ps, const elem_t* __restrict__ kv, int64_t kv_ps, int planes, const float* __restrict__ p0,
    const float* __restrict__ pd0, elem_t* __restrict__ dq0, int64_t dq_ps, elem_t* __restrict__ dkv,
    int64_t dkv_ps, float* __restrict__ dbias /* [768] q | k | v */, const float* __restrict__ gscale, int B, int H,
    int T, int Tp) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t bh = static_cast<int64_t>(blockIdx.x) * R0_WARPS + warp;
  if (bh >= static_cast<int64_t>(B) * H) return;
  const int b = static_cast<int>(bh / H), h = static_cast<int>(bh % H);
  const int g = lane >> 3, d8 = lane & 7;
  float* ds = sm + warp * Tp;
  const int64_t col = h * 64 + d8 * 8;
  float dout[8], q[8];
  load8f(datt0, da_ps, g_planes, static_cast<int64_t>(b) * 256 + col, dout);
  load8f(q0, q_ps, planes, static_cast<int64_t>(b) * 256 + col, q);
  const int64_t kv_row0 = static_cast<int64_t>(b) * T * 512 + col;
  const float* p = p0 + bh * Tp;
  const float* pd = pd0 + bh * Tp;
  // dV rows and dp_t = dO . V_t
  float pd_sum = 0.f;
  for (int t0 = 0; t0 < T; t0 += 16) {
    int64_t off[4];
    float pdt[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = t0 + 4 * u + g;
      off[u] = kv_row0 + 256 + static_cast<int64_t>(min(t, T - 1)) * 512;
      pdt[u] = t < T ? __ldg(pd + t) : 0.f;
    }
    float v[4][8];
    load_rows4<PL>(kv, kv_ps, off, v);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = t0 + 4 * u + g;
      float dp = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) dp = fmaf(dout[i], v[u][i], dp);
      dp = group8_sum(dp);
      if (t < T) {
        if (d8 == 0) ds[t] = dp;
        pd_sum += pdt[u];
        float w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = pdt[u] * dout[i];
        store8_split(dkv, dkv_ps, g_planes, kv_row0 + 256 + static_cast<int64_t>(t) * 512, w);
      }
    }
  }
  // pd_sum currently holds this key group's share: combine the four groups
  pd_sum += __shfl_xor_sync(0xffffffffu, pd_sum, 8);
  pd_sum += __shfl_xor_sync(0xffffffffu, pd_sum, 16);
  __syncwarp();
  float dot = 0.f;
  for (int t = lane; t < T; t += 32) dot += pd[t] * ds[t];
  dot = warp_sum(dot);
  float ds_sum = 0.f;
  for (int t = lane; t < T; t += 32) {
    const float d = 0.125f * (pd[t] * ds[t] - p[t] * dot);
    ds[t] = d;
    ds_sum += d;
  }
  ds_sum = warp_sum(ds_sum);
  __syncwarp();
  float dq[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int t0 = 0; t0 < T; t0 += 16) {
    int64_t off[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) off[u] = kv_row0 + static_cast<int64_t>(min(t0 + 4 * u + g, T - 1)) * 512;
    float k[4][8];
    load_rows4<PL>(kv, kv_ps, off, k);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = t0 + 4 * u + g;
      if (t < T) {
        float w[8];
        const float d = ds[t];
#pragma unroll
        for (int i = 0; i < 8; ++i) { dq[i] = fmaf(d, k[u][i], dq[i]); w[i] = d * q[i]; }
        store8_split(dkv, dkv_ps, g_planes, kv_row0 + static_cast<int64_t>(t) * 512, w);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    dq[i] += __shfl_xor_sync(0xffffffffu, dq[i], 8);
    dq[i] += __shfl_xor_sync(0xffffffffu, dq[i], 16);
  }
  if (g == 0) {
    store8_split(dq0, dq_ps, g_planes, static_cast<int64_t>(b) * 256 + col, dq);
    if (dbias == nullptr) return;     // no parameter gradients wanted
    const float inv_s = gscale != nullptr ? __ldg(gscale + 1) : 1.f;     // gradients arrive scaled by gscale[0]
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      atomicAdd(dbias + col + i, dq[i] * inv_s);
      atomicAdd(dbias + 256 + col + i, ds_sum * q[i] * inv_s);
      atomicAdd(dbias + 512 + col + i, pd_sum * dout[i] * inv_s);
    }
  }
}

int attn_row0_bwd(const void* datt0, int64_t da_ps, int g_planes, const void* q0, int64_t q_ps, const void* kv,
                  int64_t kv_ps, int planes, const float* p0, const float* pd0, void* dq0, int64_t dq_ps, void* dkv,
                  int64_t dkv_ps, float* dbias, const float* gscale, int B, int H, int T, int Tp, cudaStream_t st) {
  SPK_CHECK(H == R0_WARPS, "attn_row0: %d heads unsupported", H);
  ProfScope prof("attn_row0_bwd", 8.0 * B * H * T * 64, 2.0 * B * T * 512 * (planes + g_planes), st);
  const int blocks = (B * H + R0_WARPS - 1) / R0_WARPS;
  if (planes == 1) {
    constexpr int PLV = 1;
    attn_row0_bwd_kernel<PLV><<<blocks, 32 * R0_WARPS, R0_WARPS * Tp * sizeof(float), st>>>(
      reinterpret_cast<const elem_t*>(datt0), da_ps, g_planes, reinterpret_cast<const elem_t*>(q0), q_ps,
      reinterpret_cast<const elem_t*>(kv), kv_ps, planes, p0, pd0, reinterpret_cast<elem_t*>(dq0), dq_ps,
      reinterpret_cast<elem_t*>(dkv), dkv_ps, dbias, gscale, B, H, T, Tp);
  } else if (planes == 2) {
    constexpr int PLV = 2;
    attn_row0_bwd_kernel<PLV><<<blocks, 32 * R0_WARPS, R0_WARPS * Tp * sizeof(float), st>>>(
      reinterpret_cast<const elem_t*>(datt0), da_ps, g_planes, reinterpret_cast<const elem_t*>(q0), q_ps,
      reinterpret_cast<const elem_t*>(kv), kv_ps, planes, p0, pd0, reinterpret_cast<elem_t*>(dq0), dq_ps,
      reinterpret_cast<elem_t*>(dkv), dkv_ps, dbias, gscale, B, H, T, Tp);
  } else {
    constexpr int PLV = 3;
    attn_row0_bwd_kernel<PLV><<<blocks, 32 * R0_WARPS, R0_WARPS * Tp * sizeof(float), st>>>(
      reinterpret_cast<const elem_t*>(datt0), da_ps, g_planes, reinterpret_cast<const elem_t*>(q0), q_ps,
      reinterpret_cast<const elem_t*>(kv), kv_ps, planes, p0, pd0, reinterpret_cast<elem_t*>(dq0), dq_ps,
      reinterpret_cast<elem_t*>(dkv), dkv_ps, dbias, gscale, B, H, T, Tp);
  }
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// dst[b * dst_row_step, :] += src[b, :]   (256 columns; scatters the t = 0 rows back into a token-major tensor)
__global__ void __launch_bounds__(256) rows_add_kernel(elem_t* __restrict__ dst, int64_t d_ps, int64_t dst_row_step,
                                                       const elem_t* __restrict__ src, int64_t s_ps, int planes,
                                                       int rows) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (r >= rows) return;
  float a[8], c[8];
  load8_split(dst, d_ps, planes, r * dst_row_step * 256 + lane * 8, a);
  load8_split(src, s_ps, planes, r * 256 + lane * 8, c);
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] += c[i];
  store8_split(dst, d_ps, planes, r * dst_row_step * 256 + lane * 8, a);
}
int rows_add(void* dst, int64_t d_ps, int64_t dst_row_step, const void* src, int64_t s_ps, int planes, int rows,
             cudaStream_t st) {
  ProfScope prof("rows_add", 0, 3.0 * rows * 512 * planes, st);
  rows_add_kernel<<<(rows + 7) / 8, 256, 0, st>>>(reinterpret_cast<elem_t*>(dst), d_ps, dst_row_step,
                                                  reinterpret_cast<const elem_t*>(src), s_ps, planes, rows);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace spk
