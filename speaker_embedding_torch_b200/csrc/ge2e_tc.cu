// GE2E loss for large speaker counts (N >= 256): the three contractions S = Ehat Chat^T, dEhat = G Chat,
// dChat = G^T Ehat have intensity 0.75 N FLOP/B (SURVEY.md 8d) and belong on the tensor cores, so above
// the threshold the loss is composed from the tcgen05 GEMM of gemm_tc.cu and three row kernels instead of
// the single fp32 SIMT kernel of ge2e.cu:
//
//   prep    (block / speaker)  row norms, centroids; Ehat, Chat as split-fp16 planes (+ fp32 Chat): ge2e_centroids
//   GEMM    S = Ehat Chat^T    3 planes (fp32-equivalent), fp32 output [NM, Np]
//   rows    (warp / row)       z = w S - b, log-sum-exp, loss, dw, db, G = (w/NM)(softmax - onehot) -> 2 planes
//   GEMM    dEhat = G Chat     (Chat read MN-major), fp32 output
//   GEMM    dChat = G^T Ehat   (both MN-major, split-K, fp32 atomics)
//   finish  (warp / row)       normalisation Jacobians, centroid scatter: dE
//   excl    (block / speaker)  exclusive centroids only: the diagonal's two gradient terms (ge2e_common.cuh)
//
// The [NM, N] logits are materialised here (1 GB at N = 4096) -- what the small-N kernel avoids -- but the
// reference's two [NM, N, D] operands (2 x 257 GB at N = 4096) still never exist.
#include "ge2e.h"
#include "ge2e_common.cuh"
#include "gemm.h"
#include "rowops.h"

namespace spk {

constexpr int TD = 256;

static inline size_t up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct TcPlan {
  int64_t NM, Np;
  size_t ehat, chat, g;          // split tensors (byte offsets); plane strides below
  int64_t ehat_ps, chat_ps, g_ps;
  size_t chat32, einv, cinv, s, dehat, dchat, scal, total;
  size_t cos_own = 0, urinv = 0, gdiag = 0;     // exclusive centroids only
};

static TcPlan tc_plan(int N, int M, int mode) {
  TcPlan p;
  p.NM = static_cast<int64_t>(N) * M;
  p.Np = (N + 7) / 8 * 8;
  size_t cur = 0;
  auto split = [&](int64_t elems, int planes, int64_t& ps) {
    size_t o = cur;
    ps = static_cast<int64_t>(up(elems, 128));
    cur = up(cur + static_cast<size_t>(ps) * planes * 2, 1024);
    return o;
  };
  auto f32 = [&](int64_t elems) {
    size_t o = cur;
    cur = up(cur + static_cast<size_t>(elems) * 4, 1024);
    return o;
  };
  p.ehat = split(p.NM * TD, 3, p.ehat_ps);
  p.chat = split(static_cast<int64_t>(N) * TD, 3, p.chat_ps);
  p.g = split(p.NM * p.Np, 2, p.g_ps);
  p.chat32 = f32(static_cast<int64_t>(N) * TD);
  p.einv = f32(p.NM);
  p.cinv = f32(N);
  p.s = f32(p.NM * p.Np);
  p.dehat = f32(p.NM * TD);
  p.dchat = f32(static_cast<int64_t>(N) * TD);
  p.scal = f32(4);
  if (mode & GE2E_EXCLUSIVE) {
    p.cos_own = f32(p.NM);
    p.urinv = f32(p.NM);
    p.gdiag = f32(p.NM);
  }
  p.total = cur + 256;
  return p;
}

size_t ge2e_tc_workspace_bytes(int N, int M, int mode) { return tc_plan(N, M, mode).total; }

// ---- rows: one warp per embedding row; lane handles columns lane*8 + 256*c
// MODE (GE2E_CONTRAST | GE2E_EXCLUSIVE bits): GE2E_EXCLUSIVE replaces each row's own-speaker cosine by `cos_own` (prep)
// and writes that column's G to `gdiag` (dL/dcos_own) and a zero to the G planes, so that neither GEMM carries it;
// GE2E_CONTRAST replaces the log-sum-exp by the own / strongest-impostor rule.
template <int MODE>
__global__ void __launch_bounds__(256) ge2e_rows_kernel(const float* __restrict__ S, int64_t NM, int N, int Np, int M,
                                                        const float* __restrict__ w_ptr, const float* __restrict__ b_ptr,
                                                        elem_t* __restrict__ G, int64_t g_ps,
                                                        float* __restrict__ loss, float* __restrict__ dw,
                                                        float* __restrict__ db, int need_grad,
                                                        const float* __restrict__ cos_own, float* __restrict__ gdiag) {
  constexpr bool EXCL = (MODE & GE2E_EXCLUSIVE) != 0, CONTRAST = (MODE & GE2E_CONTRAST) != 0;
  __shared__ float red[3][8];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const float w = __ldg(w_ptr), b = __ldg(b_ptr);
  const float inv_nm = 1.f / static_cast<float>(NM);
  float loss_acc = 0.f, dw_acc = 0.f, db_acc = 0.f;
  for (int64_t r = warp; r < NM; r += nwarps) {
    const float* srow = S + r * Np;
    const int label = static_cast<int>(r / M);
    const float own = EXCL ? __ldg(cos_own + r) : 0.f;
    if constexpr (CONTRAST) {
      // L = 1 - sigmoid(z_own) + sigmoid(z_k*), k* = the largest off-diagonal logit, ties to the lowest column
      float bz = -INFINITY;
      int bj = N;
      for (int c0 = lane * 8; c0 < Np; c0 += 256) {
        const float4 a0 = *reinterpret_cast<const float4*>(srow + c0);
        const float4 a1 = *reinterpret_cast<const float4*>(srow + c0 + 4);
        const float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float z = w * v[i] - b;
          if (c0 + i < N && c0 + i != label && z > bz) { bz = z; bj = c0 + i; }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float oz = __shfl_xor_sync(0xffffffffu, bz, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (ge2e_argmax_takes(bz, bj, oz, oj)) { bz = oz; bj = oj; }
      }
      const float s_own = EXCL ? own : srow[label];
      float so, son, sk, skn;
      ge2e_sigmoid_pair(w * s_own - b, so, son);
      ge2e_sigmoid_pair(bz, sk, skn);
      if (lane == 0) loss_acc += son + sk;
      if (need_grad) {
        const float go = -so * son, gk = sk * skn;      // dL/dz (x NM)
        if (lane == 0) {
          dw_acc += (go * s_own + gk * srow[bj]) * inv_nm;
          db_acc -= (go + gk) * inv_nm;
          if (EXCL) gdiag[r] = w * go * inv_nm;
        }
        for (int c0 = lane * 8; c0 < Np; c0 += 256) {
          float g[8];
#pragma unroll
          for (int i = 0; i < 8; ++i)
            g[i] = (c0 + i == label && !EXCL) ? w * go : (c0 + i == bj ? w * gk : 0.f);
          store8_split(G, g_ps, 2, r * Np + c0, g);
        }
      }
      continue;
    }
    // one sweep for the maximum and the sum (per-lane running pair, rescaled when the maximum moves): the logits are
    // read twice per call (here and for G) instead of three times
    float mx = -INFINITY, sum = 0.f;
    for (int c0 = lane * 8; c0 < Np; c0 += 256) {
      const float4 a0 = *reinterpret_cast<const float4*>(srow + c0);
      const float4 a1 = *reinterpret_cast<const float4*>(srow + c0 + 4);
      float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      if constexpr (EXCL) {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = (c0 + i == label) ? own : v[i];
      }
      float z[8], cm = -INFINITY;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        z[i] = (c0 + i < N) ? w * v[i] - b : -INFINITY;
        cm = fmaxf(cm, z[i]);
      }
      if (cm > -INFINITY) {
        const float nm = fmaxf(mx, cm);
        float part = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) part += expf(z[i] - nm);      // exp(-inf) = 0 for the padding columns
        sum = sum * expf(mx - nm) + part;                          // exp(-inf - nm) = 0 on the first chunk
        mx = nm;
      }
    }
    {
      const float all = warp_max(mx);
      sum = warp_sum(mx > -INFINITY ? sum * expf(mx - all) : 0.f);
      mx = all;
    }
    const float lse = mx + logf(sum);
    if (lane == 0) loss_acc += lse - (w * (EXCL ? own : srow[label]) - b);
    if (need_grad) {
      // (keeping the row in shared memory for this sweep was measured: 8 warps x 16 KB leaves one block per SM at
      // N = 4096 and the kernel ran 1.8x slower than re-reading the row, most of which L2 still holds)
      for (int c0 = lane * 8; c0 < Np; c0 += 256) {
        const float4 a0 = *reinterpret_cast<const float4*>(srow + c0);
        const float4 a1 = *reinterpret_cast<const float4*>(srow + c0 + 4);
        float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        if constexpr (EXCL) {
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = (c0 + i == label) ? own : v[i];
        }
        float g[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          g[i] = 0.f;
          if (c0 + i < N) {
            const float p = expf(w * v[i] - b - lse);
            const float pm1 = p - (c0 + i == label ? 1.f : 0.f);
            const float pm = pm1 * inv_nm;
            dw_acc += pm * v[i];
            db_acc -= pm;
            g[i] = w * pm1;      // G * NM: O(w), well inside the fp16 planes' range; 1 / NM is the GEMMs' alpha
            if (EXCL && c0 + i == label) {
              gdiag[r] = w * pm;
              g[i] = 0.f;
            }
          }
        }
        store8_split(G, g_ps, 2, r * Np + c0, g);
      }
    }
  }
  loss_acc = warp_sum(loss_acc);
  dw_acc = warp_sum(dw_acc);
  db_acc = warp_sum(db_acc);
  if (lane == 0) { red[0][wib] = loss_acc; red[1][wib] = dw_acc; red[2][wib] = db_acc; }
  __syncthreads();
  if (threadIdx.x == 0 || (threadIdx.x < 3 && need_grad)) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += red[threadIdx.x][i];
    atomicAdd(threadIdx.x == 0 ? loss : (threadIdx.x == 1 ? dw : db), threadIdx.x == 0 ? s * inv_nm : s);
  }
}

// ---- finish: one warp per row
__global__ void __launch_bounds__(256) ge2e_finish_kernel(const float* __restrict__ E, const float* __restrict__ einv,
                                                          const float* __restrict__ chat32, const float* __restrict__ cinv,
                                                          const float* __restrict__ dehat, const float* __restrict__ dchat,
                                                          float* __restrict__ dE, int64_t NM, int M) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < NM; r += nwarps) {
    const int64_t k = r / M;
    const float ei = einv[r];
    float e[8], de[8], c[8], dc[8];
    const float4 e0 = __ldg(reinterpret_cast<const float4*>(E + r * TD + lane * 8));
    const float4 e1 = __ldg(reinterpret_cast<const float4*>(E + r * TD + lane * 8 + 4));
    const float4 d0 = __ldg(reinterpret_cast<const float4*>(dehat + r * TD + lane * 8));
    const float4 d1 = __ldg(reinterpret_cast<const float4*>(dehat + r * TD + lane * 8 + 4));
    const float4 c0 = __ldg(reinterpret_cast<const float4*>(chat32 + k * TD + lane * 8));
    const float4 c1 = __ldg(reinterpret_cast<const float4*>(chat32 + k * TD + lane * 8 + 4));
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(dchat + k * TD + lane * 8));
    const float4 g1 = __ldg(reinterpret_cast<const float4*>(dchat + k * TD + lane * 8 + 4));
    e[0] = e0.x * ei; e[1] = e0.y * ei; e[2] = e0.z * ei; e[3] = e0.w * ei;
    e[4] = e1.x * ei; e[5] = e1.y * ei; e[6] = e1.z * ei; e[7] = e1.w * ei;
    de[0] = d0.x; de[1] = d0.y; de[2] = d0.z; de[3] = d0.w; de[4] = d1.x; de[5] = d1.y; de[6] = d1.z; de[7] = d1.w;
    c[0] = c0.x; c[1] = c0.y; c[2] = c0.z; c[3] = c0.w; c[4] = c1.x; c[5] = c1.y; c[6] = c1.z; c[7] = c1.w;
    dc[0] = g0.x; dc[1] = g0.y; dc[2] = g0.z; dc[3] = g0.w; dc[4] = g1.x; dc[5] = g1.y; dc[6] = g1.z; dc[7] = g1.w;
    float dot_e = 0.f, dot_c = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { dot_e += de[i] * e[i]; dot_c += dc[i] * c[i]; }
    dot_e = warp_sum(dot_e);
    dot_c = warp_sum(dot_c);
    const float cs = cinv[k] / static_cast<float>(M);
    float o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = (de[i] - dot_e * e[i]) * ei + (dc[i] - dot_c * c[i]) * cs;
    float4* dst = reinterpret_cast<float4*>(dE + r * TD + lane * 8);
    dst[0] = make_float4(o[0], o[1], o[2], o[3]);
    dst[1] = make_float4(o[4], o[5], o[6], o[7]);
  }
}

// ---- exclusive centroids: the diagonal's gradient terms, one block per speaker (after finish)
__global__ void __launch_bounds__(256) ge2e_excl_kernel(const float* __restrict__ E, int M, const float* __restrict__ einv,
                                                        const float* __restrict__ cos_own, const float* __restrict__ urinv,
                                                        const float* __restrict__ gdiag, float* __restrict__ dE) {
  ge2e_excl_diag_grad(E, blockIdx.x, M, einv, cos_own, urinv, gdiag, dE, 0.f);
}

int ge2e_tc(const float* E, int N, int M, const float* w, const float* b, float* loss, float* dE, float* dw, float* db,
            void* ws_v, size_t ws_bytes, cudaStream_t st, int mode) {
  const TcPlan pl = tc_plan(N, M, mode);
  const bool excl = (mode & GE2E_EXCLUSIVE) != 0;
  if (ws_bytes < pl.total) {
    set_error("ge2e: workspace too small (%zu < %zu)", ws_bytes, pl.total);
    return SPK_ENOMEM;
  }
  char* ws = reinterpret_cast<char*>(ws_v);
  auto bf = [&](size_t off) { return reinterpret_cast<elem_t*>(ws + off); };
  auto fp = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
  const int need_grad = dE != nullptr;
  const int64_t NM = pl.NM;
  {
    ProfScope prof("ge2e_tc.prep", 0, 4.0 * NM * TD + 6.0 * NM * TD, st);
    Ge2eCentroids c = {};
    c.E = E; c.N = N; c.M = M;
    c.loss = loss;
    if (need_grad) { c.dw = dw; c.db = db; c.dchat = fp(pl.dchat); }   // dchat: split-K target of the dChat GEMM
    c.einv = fp(pl.einv); c.chat = fp(pl.chat32); c.cinv = fp(pl.cinv);
    if (excl) { c.cos_own = fp(pl.cos_own); c.urinv = fp(pl.urinv); }
    c.ehat_planes = bf(pl.ehat); c.ehat_ps = pl.ehat_ps;
    c.chat_planes = bf(pl.chat); c.chat_ps = pl.chat_ps;
    SPK_TRY(ge2e_centroids(c, st));
  }
  {  // S = Ehat Chat^T
    GemmProblem g;
    g.tag = "ge2e_tc.gemm_s";
    g.A.base = bf(pl.ehat); g.A.plane_stride = pl.ehat_ps; g.A.rows = NM; g.A.cols = TD; g.A.ld = TD;
    g.B.base = bf(pl.chat); g.B.plane_stride = pl.chat_ps; g.B.rows = N; g.B.cols = TD; g.B.ld = TD;
    g.planes = 2; g.M = static_cast<int>(NM); g.N = static_cast<int>(pl.Np); g.K = TD;
    g.epi.flags = EPI_OUT_F32;
    g.epi.out = fp(pl.s); g.epi.out_ld = pl.Np;
    SPK_TRY(gemm_run(g, st));
  }
  {
    ProfScope prof("ge2e_tc.rows", 0, (need_grad ? 2.0 : 1.0) * NM * pl.Np * 4.0 + (need_grad ? 4.0 * NM * pl.Np : 0.0), st);
    const int blocks = static_cast<int>(std::min<int64_t>((NM + 7) / 8, static_cast<int64_t>(device_sm_count()) * 8));
    auto* rows = ge2e_for_mode(mode, [](auto m) { return ge2e_rows_kernel<decltype(m)::value>; });
    rows<<<blocks, 256, 0, st>>>(fp(pl.s), NM, N, static_cast<int>(pl.Np), M, w, b, bf(pl.g), pl.g_ps, loss, dw, db,
                                 need_grad, excl ? fp(pl.cos_own) : nullptr, excl ? fp(pl.gdiag) : nullptr);
    SPK_CUDA(cudaGetLastError());
  }
  if (need_grad) {
    {  // dEhat = G Chat
      GemmProblem g;
      g.tag = "ge2e_tc.gemm_dehat";
      g.A.base = bf(pl.g); g.A.plane_stride = pl.g_ps; g.A.rows = NM; g.A.cols = N; g.A.ld = pl.Np;
      g.B.base = bf(pl.chat); g.B.plane_stride = pl.chat_ps; g.B.rows = N; g.B.cols = TD; g.B.ld = TD;
      g.b_mn = true;
      g.planes = 2; g.M = static_cast<int>(NM); g.N = TD; g.K = N;
      g.epi.flags = EPI_OUT_F32;
      g.epi.alpha = 1.f / static_cast<float>(NM);
      g.epi.out = fp(pl.dehat); g.epi.out_ld = TD;
      SPK_TRY(gemm_run(g, st));
    }
    {  // dChat = G^T Ehat
      GemmProblem g;
      g.tag = "ge2e_tc.gemm_dchat";
      g.A.base = bf(pl.g); g.A.plane_stride = pl.g_ps; g.A.rows = NM; g.A.cols = N; g.A.ld = pl.Np;
      g.B.base = bf(pl.ehat); g.B.plane_stride = pl.ehat_ps; g.B.rows = NM; g.B.cols = TD; g.B.ld = TD;
      g.a_mn = true; g.b_mn = true;
      g.planes = 2; g.M = N; g.N = TD; g.K = static_cast<int>(NM);
      const int tiles = (N + 127) / 128;
      const int kb = static_cast<int>((NM + 63) / 64);
      int ks = (2 * device_sm_count() + tiles - 1) / tiles;
      g.ksplit = ks > kb ? kb : (ks < 1 ? 1 : ks);
      g.epi.flags = EPI_OUT_ATOMIC;
      g.epi.alpha = 1.f / static_cast<float>(NM);
      g.epi.out = fp(pl.dchat); g.epi.out_ld = TD;
      SPK_TRY(gemm_run(g, st));
    }
    {
      ProfScope prof("ge2e_tc.finish", 0, 12.0 * NM * TD, st);
      const int blocks = static_cast<int>(std::min<int64_t>((NM + 7) / 8, 148 * 8));
      ge2e_finish_kernel<<<blocks, 256, 0, st>>>(E, fp(pl.einv), fp(pl.chat32), fp(pl.cinv), fp(pl.dehat), fp(pl.dchat),
                                                 dE, NM, M);
      SPK_CUDA(cudaGetLastError());
    }
    if (excl) {
      ProfScope prof("ge2e_tc.excl", 0, 12.0 * NM * TD, st);
      ge2e_excl_kernel<<<N, 256, 0, st>>>(E, M, fp(pl.einv), fp(pl.cos_own), fp(pl.urinv), fp(pl.gdiag), dE);
      SPK_CUDA(cudaGetLastError());
    }
  }
  return 0;
}

}  // namespace spk
