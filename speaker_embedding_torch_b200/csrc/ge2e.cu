// Fused GE2E loss for N < 256 speakers: three stream-ordered launches (stages) compute centroids, row/centroid
// normalisation, the N*M x N cosine-similarity matrix, w*S - b, log-softmax cross-entropy, and its gradient
// (dE, dw, db) without ever materialising the [N*M, N] logits or the reference's two
// [N*M, N, D] expanded operands (/root/reference/Modules.py:121-156; math: SURVEY.md App. B).
//
//   stage 1  ge2e_centroid_kernel       (block per speaker)  c_k = mean_m E ; ehat scale 1/max(|E_i|,eps) ; chat_k ;
//                                                            zero dchat (also the tensor-core path's first kernel)
//   stage 2  ge2e_rows_tile_kernel      (block per 8 rows)   S rows -> log-sum-exp, loss ; G = (w/NM)(softmax - onehot)
//                                                            dehat += G * Chat   (registers)
//                                                            dchat += G^T * Ehat (fp32 RED)
//                                                            dE_i  = (dehat - (dehat.ehat) ehat) / |E_i|
//   stage 3  ge2e_centroid_grad_kernel  (block per speaker)  dE_i += (1/M) (dchat_j - (dchat_j.chat_j) chat_j) / |c_j|
//
// fp32 SIMT math throughout (bit-for-bit deterministic except the fp32 atomics of dchat/loss).
// D is fixed at 256 (= Embedding_Size of the reference hyper-parameters): thread <-> column.
#include "common.cuh"
#include "ge2e.h"
#include "ge2e_common.cuh"
#include "ptx.cuh"

namespace spk {

constexpr int GD = 256;        // embedding size
constexpr int TC = 64;         // centroids per tile
constexpr int CPAD = GD + 4;   // padded centroid row (floats), keeps 16-B alignment, breaks bank aliasing

// Programmatic dependent launch (pdl_trigger / pdl_wait, ptx.cuh): the stages are launched back to back with the
// stream-serialisation attribute; a stage touches its predecessor's results only after pdl_wait().
__device__ __forceinline__ float block_sum_256(float v, float* red8) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red8[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) s += red8[w];
  return s;
}

// Stage 1 of both paths (ge2e_centroids), one block per speaker: warp per row for the row norms and the column partial
// sums (lane owns columns lane*8 .. +7), thread <-> column for the centroid.  EXCL: exclusive own-speaker centroids,
// each row's diagonal cosine `cos_own` and `urinv` = 1 / max(|u_i| / (M-1), eps), u_i = sum - e_i.  SPLIT: Ehat and
// Chat also as two fp16 planes for the tensor-core GEMMs.
template <bool EXCL, bool SPLIT>
__global__ void __launch_bounds__(256) ge2e_centroid_kernel(const Ge2eCentroids c) {
  __shared__ float part[8][GD];
  __shared__ float colsum[GD];
  __shared__ float red8[8];
  const int k = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float eps = 1e-8f;
  pdl_trigger();      // the next launch reads nothing of this one before its pdl_wait()
  if (k == 0 && tid == 0) {
    c.loss[0] = 0.f;
    if (c.dw != nullptr) { c.dw[0] = 0.f; c.db[0] = 0.f; }
  }
  if (c.dchat != nullptr) c.dchat[static_cast<int64_t>(k) * GD + tid] = 0.f;
  float cp[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int m = warp; m < c.M; m += 8) {
    const int64_t row = static_cast<int64_t>(k) * c.M + m;
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(c.E + row * GD + lane * 8));
    const float4 a1 = __ldg(reinterpret_cast<const float4*>(c.E + row * GD + lane * 8 + 4));
    float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { q += v[i] * v[i]; cp[i] += v[i]; }
    const float inv = 1.f / fmaxf(sqrtf(warp_sum(q)), eps);
    if (lane == 0) c.einv[row] = inv;
    if constexpr (SPLIT) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] *= inv;
      store8_split(c.ehat_planes, c.ehat_ps, 2, row * GD + lane * 8, v);   // two fp16 planes carry an fp32 mantissa
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) part[warp][lane * 8 + i] = cp[i];
  __syncthreads();
  float cv = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) cv += part[w][tid];
  if constexpr (EXCL) colsum[tid] = cv;        // the speaker's column sum (visible after block_sum_256's barriers)
  cv *= 1.f / static_cast<float>(c.M);
  const float nrm = fmaxf(sqrtf(block_sum_256(cv * cv, red8)), eps);
  const float ch = cv / nrm;
  c.chat[static_cast<int64_t>(k) * GD + tid] = ch;
  if constexpr (SPLIT) store1_split(c.chat_planes, c.chat_ps, 2, static_cast<int64_t>(k) * GD + tid, ch);
  if (tid == 0) c.cinv[k] = 1.f / nrm;
  if constexpr (EXCL) {
    // warp per row, as above (lane 0 wrote einv of these rows): u_i = sum - e_i, formed directly
    const float inv_m1 = 1.f / static_cast<float>(c.M - 1);
    for (int m = warp; m < c.M; m += 8) {
      const int64_t r = static_cast<int64_t>(k) * c.M + m;
      const float4 a0 = __ldg(reinterpret_cast<const float4*>(c.E + r * GD + lane * 8));
      const float4 a1 = __ldg(reinterpret_cast<const float4*>(c.E + r * GD + lane * 8 + 4));
      const float4 s0 = *reinterpret_cast<const float4*>(&colsum[lane * 8]);
      const float4 s1 = *reinterpret_cast<const float4*>(&colsum[lane * 8 + 4]);
      const float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float sv[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
      float qu = 0.f, qeu = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float u = sv[i] - v[i];
        qu += u * u;
        qeu += v[i] * u;
      }
      qu = warp_sum(qu);
      qeu = warp_sum(qeu);
      if (lane == 0) {
        const float ur = 1.f / fmaxf(sqrtf(qu) * inv_m1, eps);
        c.urinv[r] = ur;
        c.cos_own[r] = qeu * c.einv[r] * (ur * inv_m1);
      }
    }
  }
}

// The per-speaker stages of the small-N path (1 and 3) are launched with 80 KB of dynamic shared memory that they do not
// use, so that at most two of their blocks share an SM.  Measured on a B200 at 1000 W (CUDA-graph replay): without it on
// stage 1 the call at N = 64 took 21.3 us instead of 17.5 us in every mode; without it on stage 3 the exclusive modes
// took 1.4 us more at N = 64; a larger reservation (90 KB) cost the exclusive modes 0.6 - 0.9 us at N = 64 and 128.
// The tensor-core path launches stage 1 without one.
constexpr int CENTROID_SPREAD_SMEM = 80 * 1024;

int ge2e_centroids(const Ge2eCentroids& c, cudaStream_t st) {
  static PerDeviceOnce once;
  SPK_TRY(once.run([]() -> int {
    for (auto* k : {ge2e_centroid_kernel<false, false>, ge2e_centroid_kernel<true, false>})
      SPK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, CENTROID_SPREAD_SMEM));
    return 0;
  }));
  auto* kernel = c.cos_own ? (c.ehat_planes ? ge2e_centroid_kernel<true, true> : ge2e_centroid_kernel<true, false>)
                           : (c.ehat_planes ? ge2e_centroid_kernel<false, true> : ge2e_centroid_kernel<false, false>);
  kernel<<<c.N, 256, c.ehat_planes ? 0 : CENTROID_SPREAD_SMEM, st>>>(c);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// Stage 3, one block per speaker: the centroid part of dE; EXCL adds the diagonal's terms from `gdiag` (written by the
// row stage, ge2e_common.cuh)
template <bool EXCL>
__global__ void __launch_bounds__(256)
ge2e_centroid_grad_kernel(const float* __restrict__ E, int M, const float* __restrict__ chat,
                          const float* __restrict__ cinv, const float* __restrict__ dchat,
                          const float* __restrict__ einv, const float* __restrict__ cos_own,
                          const float* __restrict__ urinv, const float* __restrict__ gdiag, float* __restrict__ dE) {
  __shared__ float red8[8];
  const int k = blockIdx.x, tid = threadIdx.x;
  pdl_wait();
  const float dc = dchat[static_cast<int64_t>(k) * GD + tid];
  const float ch = chat[static_cast<int64_t>(k) * GD + tid];
  const float dot = block_sum_256(dc * ch, red8);
  const float u = (dc - dot * ch) * cinv[k] * (1.f / static_cast<float>(M));
  if constexpr (EXCL) {
    ge2e_excl_diag_grad(E, k, M, einv, cos_own, urinv, gdiag, dE, u);
  } else {
    for (int m = 0; m < M; ++m) dE[(static_cast<int64_t>(k) * M + m) * GD + tid] += u;
  }
}

// ------------------------------------------------------------------------------------------------ stage 2: row tiles
// Tiled for the shared-memory pipe (ncu of a first 16-row version, since retired: L1/shared 64 % busy on the 60 SMs it
// used, 20 us of the 32 us call at N = 64):
//   * 8 rows per block instead of 16 -> 120 blocks at the training size (148 SMs), two blocks per SM;
//   * the centroid tile arrives by bulk copy (cp.async.bulk -> mbarrier), one 1 KB row per copy, while the block
//     normalises its rows;
//   * S tile: 2 x 2 outputs per thread, the warp covers 8 rows x 16 centroids, K split over the two warp halves of the
//     block: 4 shared-memory wavefronts per 16 FMA instructions (was 9);
//   * whole logit rows stay in shared memory (N < 256), warp <-> row for the log-sum-exp and G;
//   * one sweep over the centroids feeds both dEhat (8 row accumulators, thread <-> column) and dChat (row values of the
//     column in registers, one RED per centroid): 3 wavefronts per 16 FMA instructions (was 5 + 5).
constexpr int RT = 8;            // rows per tile
constexpr int EPAD = GD + 4;     // padded row: the four rows a warp reads at one d land in different banks
constexpr int NCAP = 256;        // this path serves N < GE2E_TC_MIN_SPEAKERS
constexpr int TILE_THREADS = 512;
static_assert(NCAP >= GE2E_TC_MIN_SPEAKERS - 1 && NCAP % TC == 0, "the row cache must hold every N of the SIMT path");

struct Ge2eTileSmem {
  float c[TC][CPAD];             // normalised centroid tile (bulk-copy destination)
  float e[RT][EPAD];             // normalised rows
  float s[RT][NCAP];             // cosine similarities of the whole row
  float gt[NCAP][RT];            // G^T: the 8 row values of one centroid are two 16-byte broadcasts
  float part[3][RT][TC];         // K quarters 1..3 of the S tile
  float red[8][RT];
  float scal[3][8];
  float rowv[RT];
  float einv[RT];
  unsigned long long bar;
};

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// MODE (GE2E_CONTRAST | GE2E_EXCLUSIVE bits): with GE2E_EXCLUSIVE the own-speaker cosine of each row is replaced by
// `cos_own` (stage 1) after pass A, and its G goes to `gdiag` instead of G^T, so that the inclusive centroid does not
// receive it; with GE2E_CONTRAST the log-sum-exp gives way to the own / strongest-impostor rule.
template <int MODE>
__global__ void __launch_bounds__(TILE_THREADS, 2)
ge2e_rows_tile_kernel(const float* __restrict__ E, int N, int M, const float* __restrict__ w_ptr,
                      const float* __restrict__ b_ptr, float* __restrict__ loss, float* __restrict__ dE,
                      float* __restrict__ dw, float* __restrict__ db, const float* __restrict__ chat,
                      const float* __restrict__ einv, float* __restrict__ dchat, int need_grad,
                      const float* __restrict__ cos_own, float* __restrict__ gdiag) {
  constexpr bool EXCL = (MODE & GE2E_EXCLUSIVE) != 0, CONTRAST = (MODE & GE2E_CONTRAST) != 0;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Ge2eTileSmem& sm = *reinterpret_cast<Ge2eTileSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t NM = static_cast<int64_t>(N) * M;
  const int64_t row0 = static_cast<int64_t>(blockIdx.x) * RT;
  const int col_tiles = (N + TC - 1) / TC;
  const float w = __ldg(w_ptr), b = __ldg(b_ptr);
  const float inv_nm = 1.f / static_cast<float>(NM);
  const uint32_t bar = smem_u32(&sm.bar);
  uint32_t parity = 0;

  pdl_trigger();
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  pdl_wait();               // the centroid stage is complete: chat, einv, zeroed accumulators
  // warp 0 requests centroid tile `ct`; every thread of the block has finished reading the previous tile (caller syncs)
  auto request_tile = [&](int ct) {
    if (warp == 0) {
      const int c0 = ct * TC;
      const int rows = min(TC, N - c0);
      if (lane == 0) {
        fence_proxy_async();
        mbar_arrive_expect_tx(bar, static_cast<uint32_t>(rows) * GD * 4u);
      }
      __syncwarp();
      for (int r = lane; r < rows; r += 32)
        bulk_g2s(smem_u32(&sm.c[r][0]), chat + static_cast<int64_t>(c0 + r) * GD, GD * 4u, bar);
    }
  };
  request_tile(0);

  if (warp < RT) {  // this block's rows, normalised: warp <-> row (warps 0..7)
    const int64_t gi = row0 + warp;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
    float sc = 0.f;
    if (gi < NM) {
      sc = __ldg(einv + gi);
      a0 = __ldg(reinterpret_cast<const float4*>(E + gi * GD + lane * 8));
      a1 = __ldg(reinterpret_cast<const float4*>(E + gi * GD + lane * 8 + 4));
    }
    a0.x *= sc; a0.y *= sc; a0.z *= sc; a0.w *= sc;
    a1.x *= sc; a1.y *= sc; a1.z *= sc; a1.w *= sc;
    *reinterpret_cast<float4*>(&sm.e[warp][lane * 8]) = a0;
    *reinterpret_cast<float4*>(&sm.e[warp][lane * 8 + 4]) = a1;
    if (lane == 0) sm.einv[warp] = sc;
  }
  __syncthreads();

  // ---- pass A: S = Ehat Chat^T for the whole rows
  const int kq = warp >> 2, wq = warp & 3, lr = lane >> 3, lc = lane & 7;      // kq: K quarter of the 16 warps
  const int ra = lr, rb = lr + 4, ca = 16 * wq + lc, cb = ca + 8;
  for (int ct = 0; ct < col_tiles; ++ct) {
    mbar_wait(bar, parity, 0x6e01);
    parity ^= 1;
    float s00 = 0.f, s01 = 0.f, s10 = 0.f, s11 = 0.f;
    const int d0 = kq * (GD / 4);
#pragma unroll 8
    for (int d = d0; d < d0 + GD / 4; d += 4) {
      const float4 ea = *reinterpret_cast<const float4*>(&sm.e[ra][d]);
      const float4 eb = *reinterpret_cast<const float4*>(&sm.e[rb][d]);
      const float4 va = *reinterpret_cast<const float4*>(&sm.c[ca][d]);
      const float4 vb = *reinterpret_cast<const float4*>(&sm.c[cb][d]);
      s00 = fmaf(ea.x, va.x, s00); s00 = fmaf(ea.y, va.y, s00); s00 = fmaf(ea.z, va.z, s00); s00 = fmaf(ea.w, va.w, s00);
      s01 = fmaf(ea.x, vb.x, s01); s01 = fmaf(ea.y, vb.y, s01); s01 = fmaf(ea.z, vb.z, s01); s01 = fmaf(ea.w, vb.w, s01);
      s10 = fmaf(eb.x, va.x, s10); s10 = fmaf(eb.y, va.y, s10); s10 = fmaf(eb.z, va.z, s10); s10 = fmaf(eb.w, va.w, s10);
      s11 = fmaf(eb.x, vb.x, s11); s11 = fmaf(eb.y, vb.y, s11); s11 = fmaf(eb.z, vb.z, s11); s11 = fmaf(eb.w, vb.w, s11);
    }
    if (kq != 0) {
      float(*pt)[TC] = sm.part[kq - 1];
      pt[ra][ca] = s00; pt[ra][cb] = s01; pt[rb][ca] = s10; pt[rb][cb] = s11;
    }
    __syncthreads();          // every read of this centroid tile is done; partial sums visible
    if (ct + 1 < col_tiles) request_tile(ct + 1);
    if (kq == 0) {
      const int c0 = ct * TC;
      sm.s[ra][c0 + ca] = s00 + (sm.part[0][ra][ca] + sm.part[1][ra][ca] + sm.part[2][ra][ca]);
      sm.s[ra][c0 + cb] = s01 + (sm.part[0][ra][cb] + sm.part[1][ra][cb] + sm.part[2][ra][cb]);
      sm.s[rb][c0 + ca] = s10 + (sm.part[0][rb][ca] + sm.part[1][rb][ca] + sm.part[2][rb][ca]);
      sm.s[rb][c0 + cb] = s11 + (sm.part[0][rb][cb] + sm.part[1][rb][cb] + sm.part[2][rb][cb]);
    }
    __syncthreads();          // part may be rewritten by the next tile; s complete after the last one
  }
  // the centroid tile needed first by pass B: tile 0 (still resident when there is only one)
  if (need_grad && col_tiles > 1) request_tile(0);

  // ---- log-sum-exp, loss, dw, db, G: warp <-> row (warps 0..7)
  if (warp < RT) {
    const int64_t gi = row0 + warp;
    const bool live = gi < NM;
    const int label = live ? static_cast<int>(gi / M) : -1;
    if constexpr (EXCL) {
      if (live && lane == 0) sm.s[warp][label] = __ldg(cos_own + gi);
      __syncwarp();
    }
    float lrow = 0.f, dw_part = 0.f, db_part = 0.f;
    if constexpr (CONTRAST) {
      // L = 1 - sigmoid(z_own) + sigmoid(z_k*), k* = the largest off-diagonal logit, ties to the lowest column
      float bz = -INFINITY;
      int bj = N;
      for (int j = lane; j < N; j += 32) {
        const float z = w * sm.s[warp][j] - b;
        if (j != label && z > bz) { bz = z; bj = j; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float oz = __shfl_xor_sync(0xffffffffu, bz, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (ge2e_argmax_takes(bz, bj, oz, oj)) { bz = oz; bj = oj; }
      }
      float so, son, sk, skn;
      ge2e_sigmoid_pair(live ? w * sm.s[warp][label] - b : 0.f, so, son);
      ge2e_sigmoid_pair(bz, sk, skn);
      if (live && lane == 0) lrow = son + sk;
      if (need_grad) {
        const float go = -so * son * inv_nm, gk = sk * skn * inv_nm;
        for (int j = lane; j < N; j += 32) {
          float gval = 0.f;
          if (live && (j == label || j == bj)) {
            const float pm = j == label ? go : gk;
            dw_part += pm * sm.s[warp][j];
            db_part -= pm;
            gval = w * pm;
            if (EXCL && j == label) { gdiag[gi] = gval; gval = 0.f; }
          }
          sm.gt[j][warp] = gval;
        }
        dw_part = warp_sum(dw_part);
        db_part = warp_sum(db_part);
      }
    } else {
      float mx = -INFINITY;
      for (int j = lane; j < N; j += 32) mx = fmaxf(mx, w * sm.s[warp][j] - b);
      mx = warp_max(mx);
      float sum = 0.f;
      for (int j = lane; j < N; j += 32) sum += expf(w * sm.s[warp][j] - b - mx);
      sum = warp_sum(sum);
      const float lse = mx + logf(sum);
      if (live && lane == 0) lrow = lse - (w * sm.s[warp][label] - b);
      if (need_grad) {
        for (int j = lane; j < N; j += 32) {
          float gval = 0.f;
          if (live) {
            const float sv = sm.s[warp][j];
            const float p = expf(w * sv - b - lse);
            const float pm = (p - (j == label ? 1.f : 0.f)) * inv_nm;
            dw_part += pm * sv;
            db_part -= pm;
            gval = w * pm;
            if (EXCL && j == label) { gdiag[gi] = gval; gval = 0.f; }
          }
          sm.gt[j][warp] = gval;
        }
        dw_part = warp_sum(dw_part);
        db_part = warp_sum(db_part);
      }
    }
    if (lane == 0) { sm.scal[0][warp] = lrow; sm.scal[1][warp] = dw_part; sm.scal[2][warp] = db_part; }
  }
  __syncthreads();
  if (tid < 3 && (tid == 0 || need_grad)) {
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += sm.scal[tid][i];
    atomicAdd(tid == 0 ? loss : (tid == 1 ? dw : db), tid == 0 ? a * inv_nm : a);
  }
  if (!need_grad) return;

  // ---- pass B: dEhat = G Chat (registers, thread <-> column) and dChat += G^T Ehat (RED per centroid)
  // the two halves of the block take alternate centroids of the sweep; thread <-> column `col` in both
  const int half = tid >> 8, col = tid & (GD - 1);
  float er[RT], dacc[RT];
#pragma unroll
  for (int r = 0; r < RT; ++r) { er[r] = sm.e[r][col]; dacc[r] = 0.f; }
  for (int ct = 0; ct < col_tiles; ++ct) {
    const int c0 = ct * TC;
    const int cols = min(TC, N - c0);
    if (col_tiles > 1) {
      mbar_wait(bar, parity, 0x6e02);
      parity ^= 1;
    }
    // every block starts its sweep at another centroid: the REDs of the 120 blocks then land on different lines (and
    // L2 slices) at any one time instead of queueing on the same 1 KB row
    const int rot = static_cast<int>(blockIdx.x % static_cast<unsigned>(cols));
#pragma unroll 4
    for (int i = half; i < cols; i += 2) {
      const int c = (i + rot >= cols) ? i + rot - cols : i + rot;
      const float4 g0 = *reinterpret_cast<const float4*>(&sm.gt[c0 + c][0]);
      const float4 g1 = *reinterpret_cast<const float4*>(&sm.gt[c0 + c][4]);
      const float cv = sm.c[c][col];
      dacc[0] = fmaf(g0.x, cv, dacc[0]); dacc[1] = fmaf(g0.y, cv, dacc[1]);
      dacc[2] = fmaf(g0.z, cv, dacc[2]); dacc[3] = fmaf(g0.w, cv, dacc[3]);
      dacc[4] = fmaf(g1.x, cv, dacc[4]); dacc[5] = fmaf(g1.y, cv, dacc[5]);
      dacc[6] = fmaf(g1.z, cv, dacc[6]); dacc[7] = fmaf(g1.w, cv, dacc[7]);
      float a = g0.x * er[0];
      a = fmaf(g0.y, er[1], a); a = fmaf(g0.z, er[2], a); a = fmaf(g0.w, er[3], a);
      a = fmaf(g1.x, er[4], a); a = fmaf(g1.y, er[5], a); a = fmaf(g1.z, er[6], a); a = fmaf(g1.w, er[7], a);
      atomicAdd(dchat + static_cast<int64_t>(c0 + c) * GD + col, a);
    }
    if (ct + 1 < col_tiles) {
      __syncthreads();
      request_tile(ct + 1);
    }
  }
  // the upper half hands its accumulators over (S is dead: its buffer carries them)
  if (half == 1) {
#pragma unroll
    for (int r = 0; r < RT; ++r) sm.s[r][col] = dacc[r];
  }
  __syncthreads();
  // project out the radial component, write the row part of dE
  if (half == 0) {
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      dacc[r] += sm.s[r][col];
      const float dot = warp_sum(dacc[r] * er[r]);
      if (lane == 0) sm.red[warp][r] = dot;
    }
  }
  __syncthreads();
  if (tid < RT) {
    float a = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) a += sm.red[wv][tid];
    sm.rowv[tid] = a;
  }
  __syncthreads();
  if (half == 0) {
#pragma unroll
    for (int r = 0; r < RT; ++r) {
      const int64_t gi = row0 + r;
      if (gi < NM) dE[gi * GD + col] = (dacc[r] - sm.rowv[r] * er[r]) * sm.einv[r];
    }
  }
}

static int g_ge2e_pdl = 1;         // spk_set_option("ge2e_dependent_launch", 0/1): programmatic dependent launch of stages 2, 3
void ge2e_set_pdl(int on) { g_ge2e_pdl = on != 0; }

static size_t ge2e_simt_workspace_bytes(int N, int M, int mode) {
  const size_t NM = static_cast<size_t>(N) * M;
  const size_t excl = (mode & GE2E_EXCLUSIVE) ? 3 * NM : 0;      // cos_own, urinv, gdiag
  return (2 * static_cast<size_t>(N) * GD + N + NM + excl) * sizeof(float) + 256;
}
size_t ge2e_workspace_bytes(int N, int M, int mode) {
  return N >= GE2E_TC_MIN_SPEAKERS ? ge2e_tc_workspace_bytes(N, M, mode) : ge2e_simt_workspace_bytes(N, M, mode);
}

static auto rows_tile_kernel_for(int mode) {
  return ge2e_for_mode(mode, [](auto m) { return ge2e_rows_tile_kernel<decltype(m)::value>; });
}

int ge2e_fused(const float* E, int N, int M, int D, const float* w, const float* b, float* loss, float* dE, float* dw,
               float* db, void* ws, size_t ws_bytes, cudaStream_t st, int mode) {
  SPK_CHECK(D == GD, "ge2e: embedding size %d not supported by this build (256)", D);
  SPK_CHECK(N >= 1 && M >= 1, "ge2e: need at least one speaker and one utterance");
  SPK_CHECK((reinterpret_cast<uintptr_t>(E) & 15) == 0, "ge2e: embeddings must be 16-byte aligned");
  if (N >= GE2E_TC_MIN_SPEAKERS)   // intensity 0.75 N FLOP/B: tensor-core composition (ge2e_tc.cu)
    return ge2e_tc(E, N, M, w, b, loss, dE, dw, db, ws, ws_bytes, st, mode);
  if (ws_bytes < ge2e_simt_workspace_bytes(N, M, mode)) {
    set_error("ge2e: workspace too small (%zu < %zu)", ws_bytes, ge2e_simt_workspace_bytes(N, M, mode));
    return SPK_ENOMEM;
  }
  const int need_grad = (dE != nullptr);
  const bool excl = (mode & GE2E_EXCLUSIVE) != 0;
  float* chat = reinterpret_cast<float*>(ws);
  float* dchat = chat + static_cast<size_t>(N) * GD;
  float* cinv = dchat + static_cast<size_t>(N) * GD;
  float* einv = cinv + N;
  float* cos_own = excl ? einv + static_cast<size_t>(N) * M : nullptr;
  float* urinv = excl ? cos_own + static_cast<size_t>(N) * M : nullptr;
  float* gdiag = excl ? urinv + static_cast<size_t>(N) * M : nullptr;

  static PerDeviceOnce once;
  const int smem = static_cast<int>(sizeof(Ge2eTileSmem));
  SPK_TRY(once.run([&]() -> int {
    for (int m : {0, GE2E_CONTRAST, GE2E_EXCLUSIVE, GE2E_CONTRAST | GE2E_EXCLUSIVE})
      SPK_CUDA(cudaFuncSetAttribute(rows_tile_kernel_for(m), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    for (auto* k : {ge2e_centroid_grad_kernel<false>, ge2e_centroid_grad_kernel<true>})
      SPK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, CENTROID_SPREAD_SMEM));
    return 0;
  }));
  const long long NM = 1LL * N * M;
  ProfScope prof(need_grad ? "ge2e_fused_fwd_bwd" : "ge2e_fused_fwd", (need_grad ? 6.0 : 2.0) * NM * N * GD,
                 (need_grad ? 2.0 : 1.0) * NM * GD * 4.0, st);
  // three launches in stream order: centroids | row tiles (loss, dE row part, dC) | centroid part of dE (stream order is
  // the grid-wide barrier: a cooperative launch with two grid.sync() cost 32 us at the training size, mostly in the syncs)
  Ge2eCentroids c = {};
  c.E = E; c.N = N; c.M = M;
  c.loss = loss;
  if (need_grad) { c.dw = dw; c.db = db; c.dchat = dchat; }
  c.einv = einv; c.chat = chat; c.cinv = cinv;
  c.cos_own = cos_own; c.urinv = urinv;
  SPK_TRY(ge2e_centroids(c, st));
  cudaLaunchAttribute pdl_attr[1];
  pdl_attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  pdl_attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.stream = st;
  cfg.attrs = pdl_attr;
  cfg.numAttrs = g_ge2e_pdl ? 1 : 0;
  cfg.gridDim = dim3(static_cast<unsigned>((NM + RT - 1) / RT));
  cfg.blockDim = dim3(TILE_THREADS);
  cfg.dynamicSmemBytes = smem;
  SPK_CUDA(cudaLaunchKernelEx(&cfg, rows_tile_kernel_for(mode), E, N, M, w, b, loss, dE, dw, db, chat, einv, dchat,
                              need_grad, cos_own, gdiag));
  if (need_grad) {
    cfg.gridDim = dim3(N);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = CENTROID_SPREAD_SMEM;
    SPK_CUDA(cudaLaunchKernelEx(&cfg, excl ? ge2e_centroid_grad_kernel<true> : ge2e_centroid_grad_kernel<false>, E, M,
                                chat, cinv, dchat, einv, cos_own, urinv, gdiag, dE));
  }
  return 0;
}

}  // namespace spk
