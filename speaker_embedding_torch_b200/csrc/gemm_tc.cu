// Persistent, warp-specialised tcgen05 GEMM for sm_100a on split-fp16 operands.
//
//   D[M,N] = epilogue( alpha * A[M,K] * B[N,K]^T )          (per batch, optional split-K)
//
// * operands are fetched by TMA (cp.async.bulk.tensor.4d, 128-byte swizzle) into a multi-stage
//   shared-memory ring; each operand may be K-major or MN-major (transposed reads for dgrad /
//   wgrad / P*V come from the descriptor, never from a transposed copy);
// * one elected thread issues tcgen05.mma (UMMA 128 x BLOCK_N x 16, fp16 in, fp32 accumulate in
//   TMEM); with two planes it issues Ah*Bh + Ah*Bl + Al*Bh into the same accumulator, with three
//   planes the six products down to 2^-16 (fp32-equivalent operands);
// * the accumulator is double-buffered in TMEM so the 12 epilogue warps (tcgen05.ld -> registers
//   -> fused bias / ReLU / positional term / dropout / residual / gate -> global) drain tile i
//   while the MMA warp works on tile i+1;
// * grid = min(#tiles, #SMs); tiles are assigned round-robin (persistent CTAs);
// * multi-plane problems with a K-major A and M >= 256 run on CTA pairs instead (gemm_pair_kernel below:
//   tcgen05.mma.cta_group::2, 256 x 256 tiles, each CTA stages half of B).
//
// Warp roles (512 threads): 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 3 = idle,
// 4..15 = epilogue (warp w owns TMEM lanes 32*(w%4) .. +31 == accumulator rows; the three warps of a lane quarter
// take its 32-column chunks round-robin: warp w the chunks c with c % 3 == (w-4) / 4).
#include "gemm.h"
#include "ptx.cuh"

#include <mutex>

namespace spk {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;              // 64 fp16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int SMEM_LIMIT = 232448;       // 227 KB opt-in limit per CTA
constexpr int BAR_BYTES = 256;
constexpr int NUM_EPI_WARPS = 12;        // three warps per TMEM lane quarter, round-robin over the 32-column chunks
constexpr int EPI_CG = NUM_EPI_WARPS / 4;  // column groups
constexpr int EPI_STAGE_BYTES = 2176;    // per warp: fp16 tile 32 x 32 (2 KB) or fp32 tile 32 x 17
constexpr int EPI_BIAS_BYTES = 512;      // per warp: the bias of its (up to four) 32-column chunks of the current tile
constexpr int EPI_SMEM = NUM_EPI_WARPS * (EPI_STAGE_BYTES + EPI_BIAS_BYTES);
// setmaxnreg: the CTA's register pool is its launch allocation, 512 x 128 >= 128 x 40 + 384 x 152 (a larger request
// spins forever): warps 0-3 (TMA / MMA / TMEM / idle) keep 40 registers, the epilogue warps get 152.  (Round 1 ran 8
// epilogue warps at 224 registers: the epilogue is a latency-bound chain per 32 x 32 chunk -- ncu r02: 14 cycles per
// issued instruction with two warps per scheduler -- so a third warp per scheduler buys more than the registers did.)
constexpr int LAUNCH_REGS = 128, CTRL_REGS = 40, EPI_REGS = 152;

struct GemmKernelArgs {
  CUtensorMap a_map[3];
  CUtensorMap b_map[3];
  int M, N, K;
  int tiles_m, tiles_n, nb0, nb1, ksplit, kb_total, kb_per_split;
  int a_batched, b_batched;
  GemmEpilogue epi;
};

template <int PLANES, int BLOCK_N>
struct TileCfg {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_ROWS = BLOCK_N;
  static constexpr int B_BYTES = B_ROWS * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = PLANES * (A_BYTES + B_BYTES);
  static constexpr int RAW_STAGES = (SMEM_LIMIT - 1024 - BAR_BYTES - EPI_SMEM) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 8 ? 8 : RAW_STAGES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES + EPI_SMEM;
  static constexpr int TMEM_COLS = (2 * BLOCK_N <= 128) ? 128 : (2 * BLOCK_N <= 256 ? 256 : 512);
  static_assert(STAGES >= 1, "operand ring does not fit shared memory");
  static_assert(2 * BLOCK_N <= 512, "accumulator double buffer must fit TMEM");
};

// ------------------------------------------------------------------------------------------------
// Epilogue of one 32 x 32 accumulator chunk per warp (lane == row).  Global traffic never goes out
// row-strided from the lanes: every residual / gate read and every output store is transposed through
// a per-warp shared-memory tile (32 rows x 64 B, 16-B chunks XOR-swizzled so that both the "lane owns a
// row" and the "8 lanes cover 2 rows x 64 B" access patterns are bank-conflict free), so each warp
// memory instruction touches 8 rows x 64 contiguous bytes (full 32-B sectors).
__device__ __forceinline__ uint32_t stage_off(int row, int chunk) {
  return static_cast<uint32_t>(row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4));
}

// Per-tile, per-lane addressing of the cooperative "8 rows x 64 B per instruction" pattern: lane (lane>>2, lane&3)
// touches row row0 + it*8 + (lane>>2), 16-byte chunk (lane&3), it = 0..3.  Computed once per tile so the
// per-chunk code has no 64-bit multiplies (ncu r01: address arithmetic was > 50 % of the epilogue's instructions).
struct CoopIO {
  int64_t off0;      // element offset of (row0 + (lane>>2), chunk (lane&3)) including the batch offset
  int64_t ld8;       // 8 rows further down
  uint32_t rowmask;  // bit it: row0 + it*8 + (lane>>2) < M
};
__device__ __forceinline__ CoopIO make_coop(int lane, int64_t boff, int64_t row0, int64_t ld, int M, int elems_per_chunk) {
  CoopIO io;
  const int64_t r = row0 + (lane >> 2);
  io.off0 = boff + r * ld + (lane & 3) * elems_per_chunk;
  io.ld8 = 8 * ld;
  io.rowmask = (r < M ? 1u : 0u) | (r + 8 < M ? 2u : 0u) | (r + 16 < M ? 4u : 0u) | (r + 24 < M ? 8u : 0u);
  return io;
}

// r[32] = aux[row0 + lane][col0 .. col0+31]  (split tensor, rows >= M / cols >= N read as 0).
// All planes' global loads are issued before the first wait so up to 12 x 16 B per lane are in flight.
__device__ __forceinline__ void load_aux_tile(uint32_t stage, int lane, const void* base_v, int64_t ps, int planes,
                                              const CoopIO& io, int col0, int N, float (&r)[32]) {
  const elem_t* base = reinterpret_cast<const elem_t*>(base_v) + io.off0 + col0;
  const bool col_ok = col0 + (lane & 3) * 8 < N;
#pragma unroll
  for (int i = 0; i < 32; ++i) r[i] = 0.f;
#pragma unroll
  for (int p0 = 0; p0 < 3; p0 += 2) {      // two planes (8 x 16 B per lane) in flight at a time
    if (p0 < planes) {
      uint4 g[2][4];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (p0 + q < planes && p0 + q < 3) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            g[q][it] = make_uint4(0u, 0u, 0u, 0u);
            if (col_ok && ((io.rowmask >> it) & 1u))
              g[q][it] = __ldg(reinterpret_cast<const uint4*>(base + (p0 + q) * ps + it * io.ld8));
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (p0 + q < planes && p0 + q < 3) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stage + stage_off(it * 8 + (lane >> 2), lane & 3)),
                         "r"(g[q][it].x), "r"(g[q][it].y), "r"(g[q][it].z), "r"(g[q][it].w)
                         : "memory");
          }
          __syncwarp();
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            uint32_t w0, w1, w2, w3;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3)
                         : "r"(stage + stage_off(lane, cc))
                         : "memory");
            const uint32_t ww[4] = {w0, w1, w2, w3};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              r[cc * 8 + 2 * i] += lo_to_f(ww[i]);
              r[cc * 8 + 2 * i + 1] += hi_to_f(ww[i]);
            }
          }
          __syncwarp();
        }
      }
    }
  }
}

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 w;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "r"(addr) : "memory");
  return w;
}

// out[row0 + lane][col0 .. col0+31] = v (split planes), coalesced through the staging tile.
// All 16 packed words / all four 16-byte rows live in distinct registers, so the four shared stores, the four shared
// loads and the four global stores of a plane issue back to back (ncu r01: with re-used registers every STS / LDS
// waited for the previous one to release its operands).
__device__ __forceinline__ void store_split_tile(uint32_t stage, int lane, void* base_v, int64_t ps, int planes,
                                                 const CoopIO& io, int col0, int N, float (&v)[32]) {
  elem_t* base = reinterpret_cast<elem_t*>(base_v) + io.off0 + col0;
  const bool col_ok = col0 + (lane & 3) * 8 < N;
  const uint32_t own = stage + lane * 64, sw = ((lane >> 1) & 3) << 4;   // own + ((cc << 4) ^ sw) == stage_off(lane, cc)
  const uint32_t coop = stage + stage_off(lane >> 2, lane & 3);          // + it * 512: the swizzle term does not depend on it
  for (int p = 0; p < planes; ++p) {
    const bool more = p + 1 < planes;   // the residual is only needed if another plane follows
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      w[i] = pack2(v[2 * i], v[2 * i + 1]);
    }
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) sts128(own + ((cc << 4) ^ sw), w[4 * cc], w[4 * cc + 1], w[4 * cc + 2], w[4 * cc + 3]);
    __syncwarp();
    uint4 o[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) o[it] = lds128(coop + it * 512);
    if (more) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        v[2 * i] -= lo_to_f(w[i]);
        v[2 * i + 1] -= hi_to_f(w[i]);
      }
    }
#pragma unroll
    for (int it = 0; it < 4; ++it)
      if (col_ok && ((io.rowmask >> it) & 1u)) *reinterpret_cast<uint4*>(base + p * ps + it * io.ld8) = o[it];
    __syncwarp();
  }
}

// fp32 tile, plain store: a 16-column half of the 32 x 32 chunk is 32 rows x 64 B -- the same geometry as one bf16
// plane -- so it goes through the same swizzled staging tile with 16-byte shared / global accesses.
// `io` is built with 4 elements per chunk.
__device__ __forceinline__ void store_f32_tile_plain(uint32_t stage, int lane, float* base_f, const CoopIO& io, int col0,
                                                     int N, const float (&v)[32]) {
  float* base = base_f + io.off0 + col0;
  const uint32_t own = stage + lane * 64, sw = ((lane >> 1) & 3) << 4;
  const uint32_t coop = stage + stage_off(lane >> 2, lane & 3);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
      sts128(own + ((cc << 4) ^ sw), __float_as_uint(v[h * 16 + cc * 4]), __float_as_uint(v[h * 16 + cc * 4 + 1]),
             __float_as_uint(v[h * 16 + cc * 4 + 2]), __float_as_uint(v[h * 16 + cc * 4 + 3]));
    __syncwarp();
    const bool col_ok = col0 + h * 16 + (lane & 3) * 4 < N;
    uint4 o[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) o[it] = lds128(coop + it * 512);
#pragma unroll
    for (int it = 0; it < 4; ++it)
      if (col_ok && ((io.rowmask >> it) & 1u)) *reinterpret_cast<uint4*>(base + h * 16 + it * io.ld8) = o[it];
    __syncwarp();
  }
}

// fp32 tile, atomic add (split-K weight gradients), through a 32 x 17 fp32 staging tile, 16 columns at a time:
// each instruction covers 2 rows x 64 contiguous bytes.
template <bool ATOMIC>
__device__ __forceinline__ void store_f32_tile(uint32_t stage, int lane, float* base, int64_t ld, int64_t boff,
                                               int64_t row0, int col0, int M, int N, const float (&v)[32]) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(stage + (lane * 17 + i) * 4), "f"(v[h * 16 + i]) : "memory");
    __syncwarp();
    const int cl = lane & 15, rh = lane >> 4;
    const bool col_ok = col0 + h * 16 + cl < N;
#pragma unroll 4
    for (int rr = 0; rr < 32; rr += 2) {
      float x;
      asm volatile("ld.shared.f32 %0, [%1];" : "=f"(x) : "r"(stage + ((rr + rh) * 17 + cl) * 4) : "memory");
      const int64_t grow = row0 + rr + rh;
      if (col_ok && grow < M) {
        float* dst = base + boff + grow * ld + col0 + h * 16 + cl;
        if (ATOMIC) atomicAdd(dst, x);
        else *dst = x;
      }
    }
    __syncwarp();
  }
}

// colsum[col0 + c] += sum over the warp's 32 rows of v[.][c]   (bias gradients, fused)
__device__ __forceinline__ void colsum_tile(uint32_t stage, int lane, float* colsum, int col0, int N,
                                            const float (&v)[32], float scale) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(stage + (lane * 17 + i) * 4), "f"(v[h * 16 + i]) : "memory");
    __syncwarp();
    const int cl = lane & 15, rh = lane >> 4;
    float sacc = 0.f;
#pragma unroll 8
    for (int rr = 0; rr < 16; ++rr) {
      float x;
      asm volatile("ld.shared.f32 %0, [%1];" : "=f"(x) : "r"(stage + ((rh * 16 + rr) * 17 + cl) * 4) : "memory");
      sacc += x;
    }
    sacc += __shfl_xor_sync(0xffffffffu, sacc, 16);
    if (rh == 0 && col0 + h * 16 + cl < N) atomicAdd(colsum + col0 + h * 16 + cl, sacc * scale);
    __syncwarp();
  }
}

// CT: compile-time superset of the flags that can be set for this launch -- everything outside CT is dead code, which
// keeps the common forward epilogues (bias / ReLU only) short (the epilogue is instruction-issue bound).
template <uint32_t CT>
__device__ __forceinline__ void epilogue32(const GemmEpilogue& e, uint32_t stage, uint32_t bias_s, int lane, int M, int N,
                                           int64_t row0, int64_t batch, int64_t out_boff, const CoopIO& io_out,
                                           const CoopIO& io_res, const CoopIO& io_gate, int64_t cs_boff, int col0,
                                           const uint32_t (&acc)[32], float pe_alpha, uint32_t gate_word, float alpha,
                                           float cs_scale) {
  const uint32_t f = e.flags & CT;
  const int64_t row = row0 + lane;
  const bool row_ok = row < M;
  float v[32];
  if (alpha != 1.f) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = alpha * __uint_as_float(acc[i]);
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(acc[i]);
  }
  if (f & EPI_BIAS) {   // staged in shared memory before the accumulator wait (zeros past N); same address in all lanes
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4 b;
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(bias_s + i * 16));
      v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
    }
  }
  if (f & EPI_RELU) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
  }
  if ((f & EPI_EMIT_BITS) && (f & EPI_PE)) {   // prenet: the mask is the ReLU's own (before the positional term and dropout)
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) m |= (v[i] > 0.f) ? (1u << i) : 0u;
    if (row_ok) e.gate_bits[static_cast<int64_t>(col0 >> 5) * M + row] = m;
  }
  if ((f & EPI_PE) && row_ok) {
    const float* pr = e.pe_t + (row % e.pe_T) * N + col0;
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      if (col0 + i < N) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(pr + i));
        v[i] += pe_alpha * q.x; v[i + 1] += pe_alpha * q.y; v[i + 2] += pe_alpha * q.z; v[i + 3] += pe_alpha * q.w;
      }
    }
  }
  const bool use_keep = (f & (EPI_DROPOUT | EPI_ACC_GATES_AUX)) && e.drop.thresh != 0;
  if (f & EPI_DROPOUT) {
    if (use_keep) {
      const uint64_t idx = (static_cast<uint64_t>(batch) * M + row) * N + col0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float k8[8];
        dropout_scale8(e.drop.seed, e.drop_site, (idx >> 3) + q, e.drop.thresh, e.drop.inv_keep, k8);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[q * 8 + i] *= k8[i];
      }
    }
  }
  if ((f & EPI_EMIT_BITS) && !(f & EPI_PE)) {   // ReLU mask of the final (post-dropout) activation, 1 bit per element
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) m |= (v[i] > 0.f) ? (1u << i) : 0u;
    if (row_ok) e.gate_bits[static_cast<int64_t>(col0 >> 5) * M + row] = m;   // chunk-major: a warp writes 128 contiguous bytes
  }
  if (f & EPI_GATE_BITS) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = ((gate_word >> i) & 1u) ? v[i] * e.gate_scale : 0.f;
  }
  if (f & (EPI_RES | EPI_ACC_GATES_AUX)) {
    float r[32];
    load_aux_tile(stage, lane, e.res, e.res_plane_stride, e.res_planes, io_res, col0, N, r);
    if (f & EPI_RES) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += r[i];
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = v[i] > 0.f ? r[i] : 0.f;
      if (use_keep) {
        const uint64_t idx = (static_cast<uint64_t>(batch) * M + row) * N + col0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float k8[8];
          dropout_scale8(e.drop.seed, e.drop_site, (idx >> 3) + q, e.drop.thresh, e.drop.inv_keep, k8);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[q * 8 + i] *= k8[i];
        }
      }
    }
  }
  if (f & EPI_GATE_POS) {
    float g[32];
    load_aux_tile(stage, lane, e.gate, e.gate_plane_stride, e.gate_planes, io_gate, col0, N, g);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = g[i] > 0.f ? v[i] * e.gate_scale : 0.f;
  }
  if (f & EPI_COLSUM) {   // rows past M must not contribute to the column sums (the stores are guarded per row)
    if (!row_ok) {
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = 0.f;
    }
    colsum_tile(stage, lane, e.colsum + cs_boff, col0, N, v, cs_scale);
  }
  if (f & EPI_OUT_ATOMIC) {
    store_f32_tile<true>(stage, lane, reinterpret_cast<float*>(e.out), e.out_ld, out_boff, row0, col0, M, N, v);
  } else if (f & EPI_OUT_F32) {
    if (((e.out_ld | N) & 3) == 0) store_f32_tile_plain(stage, lane, reinterpret_cast<float*>(e.out), io_out, col0, N, v);
    else store_f32_tile<false>(stage, lane, reinterpret_cast<float*>(e.out), e.out_ld, out_boff, row0, col0, M, N, v);
  } else {
    store_split_tile(stage, lane, e.out, e.out_plane_stride, e.out_planes, io_out, col0, N, v);
  }
}

__device__ __forceinline__ void tmem_st_32x32_acc(uint32_t taddr, const float (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
      "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]), "f"(v[16]), "f"(v[17]), "f"(v[18]),
      "f"(v[19]), "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]), "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]),
      "f"(v[28]), "f"(v[29]), "f"(v[30]), "f"(v[31])
      : "memory");
}

// EPI_LN: the tile owns whole rows (N == BLOCK_N == 256).  Pass A: every warp turns its chunks of the accumulator into
// z = alpha * acc + bias (+ dropout) + residual, keeps the row's partial sum / sum of squares and writes z BACK into
// tensor memory; the EPI_CG warps of a lane quarter exchange their partial sums through their staging tiles (named
// barrier per quarter); pass B re-reads z, normalises, applies gamma / beta and stores the planes.  z never reaches
// global memory and the separate LayerNorm pass over the tensor disappears (inference: 12 % of the forward).
template <int BLOCK_N>
__device__ __forceinline__ void ln_epilogue_tile(const GemmEpilogue& e, uint32_t stage_buf, uint32_t bias_buf, int lane,
                                                 int cgroup, int quarter, uint32_t t_row, int M, int N, int64_t row0,
                                                 int64_t batch, int64_t out_boff, int64_t res_boff, float alpha) {
  const CoopIO io_out = make_coop(lane, out_boff, row0, e.out_ld, M, 8);
  const bool has_res = (e.flags & EPI_RES) != 0;
  const CoopIO io_res = has_res ? make_coop(lane, res_boff, row0, e.res_ld, M, 8) : io_out;
  const bool use_drop = (e.flags & EPI_DROPOUT) && e.drop.thresh != 0;
  const int64_t row = row0 + lane;
  // Shifted sums: each warp sums d = z - piv, piv being the first z of the row it sees.  A one-pass E[z^2] - mean^2
  // loses the variance when |mean| >> std (relative error ~ (mean / std)^2 * 2^-24); about a pivot taken from the row
  // itself the sums stay of the order of the row's spread, whatever its offset.
  float s1 = 0.f, s2 = 0.f, piv = 0.f;
#pragma unroll 1
  for (int c = cgroup; c < BLOCK_N / 32; c += EPI_CG) {
    const int col0 = c * 32;
    uint32_t r[32];
    tmem_ld_32x32(t_row + c * 32, r);
    tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = alpha * __uint_as_float(r[i]);
    if (e.flags & EPI_BIAS) {
      const uint32_t bias_s = bias_buf + (c / EPI_CG) * 128;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float4 b;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "r"(bias_s + i * 16));
        v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
      }
    }
    if (use_drop) {
      const uint64_t idx = (static_cast<uint64_t>(batch) * M + row) * N + col0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float k8[8];
        dropout_scale8(e.drop.seed, e.drop_site, (idx >> 3) + q, e.drop.thresh, e.drop.inv_keep, k8);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[q * 8 + i] *= k8[i];
      }
    }
    if (has_res) {
      float rr[32];
      load_aux_tile(stage_buf, lane, e.res, e.res_plane_stride, e.res_planes, io_res, col0, N, rr);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] += rr[i];
    }
    if (c == cgroup) piv = v[0];
#pragma unroll
    for (int i = 0; i < 32; ++i) { const float d = v[i] - piv; s1 += d; s2 = fmaf(d, d, s2); }
    tmem_st_32x32_acc(t_row + c * 32, v);
    if (e.ln_z != nullptr)      // training: the backward pass needs the pre-normalisation rows (v is consumed by the split)
      store_split_tile(stage_buf, lane, e.ln_z, e.ln_z_plane_stride, e.out_planes, io_out, col0, N, v);
  }
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  // the quarter's EPI_CG warps meet: partial sums through the (currently idle) staging tiles
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(stage_buf + lane * 16), "f"(s1), "f"(s2), "f"(piv),
               "f"(0.f) : "memory");
  asm volatile("bar.sync %0, %1;" ::"r"(quarter + 1), "r"(32 * EPI_CG) : "memory");
  // merge about the pivot p0 of warp 0: sum (z - p0) = s1 + n dp, sum (z - p0)^2 = s2 + dp (2 s1 + n dp), dp = piv - p0
  // (two values of the same row: their difference is exact or of the order of the spread)
  float t1 = 0.f, t2 = 0.f, p0 = 0.f;
#pragma unroll
  for (int g = 0; g < EPI_CG; ++g) {
    float a, b, p, unused;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a), "=f"(b), "=f"(p), "=f"(unused)
                 : "r"(stage_buf + (g - cgroup) * 4 * (EPI_STAGE_BYTES + EPI_BIAS_BYTES) + lane * 16) : "memory");
    if (g == 0) p0 = p;
    const float n = static_cast<float>((BLOCK_N / 32 - g + EPI_CG - 1) / EPI_CG * 32);   // columns warp g summed
    const float dp = p - p0;
    t1 += fmaf(n, dp, a);
    t2 += fmaf(dp, fmaf(n, dp, 2.f * a), b);
  }
  asm volatile("bar.sync %0, %1;" ::"r"(quarter + 1), "r"(32 * EPI_CG) : "memory");   // read before the tiles are reused
  const float mc = t1 * (1.f / BLOCK_N);                  // mean - p0
  const float mean = p0 + mc;
  const float var = fmaxf(t2 * (1.f / BLOCK_N) - mc * mc, 0.f);
  const float rstd = rsqrtf(var + e.ln_eps);
  if (e.ln_stats != nullptr && cgroup == 0 && row < M) reinterpret_cast<float2*>(e.ln_stats)[row] = make_float2(mean, rstd);
#pragma unroll 1
  for (int c = cgroup; c < BLOCK_N / 32; c += EPI_CG) {
    const int col0 = c * 32;
    uint32_t r[32];
    tmem_ld_32x32(t_row + c * 32, r);
    tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(e.ln_gamma + col0 + i));
      const float4 b4 = __ldg(reinterpret_cast<const float4*>(e.ln_beta + col0 + i));
      v[i] = (__uint_as_float(r[i]) - mean) * rstd * g4.x + b4.x;
      v[i + 1] = (__uint_as_float(r[i + 1]) - mean) * rstd * g4.y + b4.y;
      v[i + 2] = (__uint_as_float(r[i + 2]) - mean) * rstd * g4.z + b4.z;
      v[i + 3] = (__uint_as_float(r[i + 3]) - mean) * rstd * g4.w + b4.w;
    }
    store_split_tile(stage_buf, lane, e.out, e.out_plane_stride, e.out_planes, io_out, col0, N, v);
  }
}

// All 32-column chunks of one accumulator tile that belong to this warp.
template <uint32_t CT, int BLOCK_N>
__device__ __forceinline__ void epilogue_tile(const GemmEpilogue& e, uint32_t stage_buf, uint32_t bias_buf, int lane, int cgroup,
                                              uint32_t t_row, int M, int N, int64_t row0, int64_t batch, int64_t out_boff,
                                              int64_t res_boff, int64_t cs_boff, int tn, float pe_alpha, float alpha,
                                              float cs_scale) {
  const CoopIO io_out = make_coop(lane, out_boff, row0, e.out_ld, M, (e.flags & EPI_OUT_F32) ? 4 : 8);
  CoopIO io_res = io_out, io_gate = io_out;
  if constexpr ((CT & (EPI_RES | EPI_ACC_GATES_AUX)) != 0) {
    if (e.flags & (EPI_RES | EPI_ACC_GATES_AUX)) io_res = make_coop(lane, res_boff, row0, e.res_ld, M, 8);
  }
  if constexpr ((CT & EPI_GATE_POS) != 0) {
    if (e.flags & EPI_GATE_POS) io_gate = make_coop(lane, 0, row0, e.gate_ld, M, 8);
  }
  // ReLU-mask words (EPI_GATE_BITS), layout [N / 32][M] (chunk-major: the 32 lanes of a warp = consecutive rows read 128
  // contiguous bytes); the word of chunk c + 2 is loaded while chunk c is processed
  const bool use_bits = (CT & EPI_GATE_BITS) != 0 && (e.flags & EPI_GATE_BITS) != 0 && row0 + lane < M;
  const uint32_t* bits_row = use_bits ? e.gate_bits + static_cast<int64_t>(tn) * (BLOCK_N / 32) * M + row0 + lane : nullptr;
  uint32_t next_word = (use_bits && tn * BLOCK_N + cgroup * 32 < N) ? __ldg(bits_row + static_cast<int64_t>(cgroup) * M) : 0u;
#pragma unroll 1
  for (int c = cgroup; c < BLOCK_N / 32; c += NUM_EPI_WARPS / 4) {
    const int col0 = tn * BLOCK_N + c * 32;
    if (col0 >= N) break;             // warp-uniform
    uint32_t r[32];
    tmem_ld_32x32(t_row + c * 32, r);
    const uint32_t word = next_word;
    const int cn = c + NUM_EPI_WARPS / 4;
    if (use_bits && cn < BLOCK_N / 32 && tn * BLOCK_N + cn * 32 < N) next_word = __ldg(bits_row + static_cast<int64_t>(cn) * M);
    tmem_ld_wait();
    epilogue32<CT>(e, stage_buf, bias_buf + (c / EPI_CG) * 128, lane, M, N, row0, batch, out_boff, io_out, io_res, io_gate,
                   cs_boff, col0, r, pe_alpha, word, alpha, cs_scale);
  }
}

// ------------------------------------------------------------------------------------------------
// Pieces shared by the single-CTA and the CTA-pair kernel.

// Tiles are numbered N tile fastest, then M tile, K split, batch index i0, batch index i1.
struct TileIdx {
  int tn, tm;
  int batch, i0, i1;          // batch = i0 + nb0 * i1
  int kb_begin, kb_end;       // the tile's k-blocks (its K split)
};
__device__ __forceinline__ int num_tiles(const GemmKernelArgs& a) {
  return a.nb0 * a.nb1 * a.ksplit * a.tiles_m * a.tiles_n;
}
__device__ __forceinline__ TileIdx decode_tile(const GemmKernelArgs& a, int tile) {
  TileIdx t;
  const int mn_tiles = a.tiles_m * a.tiles_n;
  const int outer = tile / mn_tiles;                  // the k-block range needs only this division and the next
  const int ks = outer % a.ksplit;
  const int mn = tile - outer * mn_tiles;
  t.tn = mn % a.tiles_n; t.tm = mn / a.tiles_n;
  t.batch = outer / a.ksplit;
  t.i0 = t.batch % a.nb0; t.i1 = t.batch / a.nb0;
  t.kb_begin = ks * a.kb_per_split;
  t.kb_end = min(t.kb_begin + a.kb_per_split, a.kb_total);
  return t;
}

// An operand ring stage (Cfg = TileCfg or PairCfg) holds the PLANES planes of A (BLOCK_M rows each, Cfg::A_BYTES apart
// from sa on), then those of B (Cfg::B_ROWS rows each, Cfg::B_BYTES apart from sb on).

// TMA load of k-block kb of one operand plane, ROWS rows from `row` on.  K-major: one box of BLOCK_K x ROWS.  MN-major:
// BLOCK_K rows of the stored [K, rows] tensor, in 64-element-wide chunks (one 128-byte swizzle row each).
template <bool MN, int ROWS>
__device__ __forceinline__ void tma_load_operand(uint32_t dst, const CUtensorMap* map, uint32_t bar, int kb, int row,
                                                 int i0, int i1) {
  if (!MN) {
    tma_load_4d(dst, map, bar, kb * BLOCK_K, row, i0, i1);
  } else {
#pragma unroll
    for (int c = 0; c < ROWS / 64; ++c) tma_load_4d(dst + c * (BLOCK_K * 128), map, bar, row + c * 64, kb * BLOCK_K, i0, i1);
  }
}

// Every plane of k-block kb into one stage: A rows from a_row, B rows from b_row, batch (i0, i1) of a batched operand.
template <class Cfg, int PLANES, bool A_MN, bool B_MN>
__device__ __forceinline__ void load_stage(const GemmKernelArgs& args, uint32_t sa, uint32_t sb, uint32_t bar, int kb,
                                           int a_row, int b_row, int i0, int i1) {
  const int a0 = args.a_batched ? i0 : 0, a1 = args.a_batched ? i1 : 0;
  const int b0 = args.b_batched ? i0 : 0, b1 = args.b_batched ? i1 : 0;
#pragma unroll
  for (int p = 0; p < PLANES; ++p) {
    tma_load_operand<A_MN, BLOCK_M>(sa + p * Cfg::A_BYTES, &args.a_map[p], bar, kb, a_row, a0, a1);
    tma_load_operand<B_MN, Cfg::B_ROWS>(sb + p * Cfg::B_BYTES, &args.b_map[p], bar, kb, b_row, b0, b1);
  }
}

// Plane products of one k-step, smallest terms first (plane 0 = hi, 1 = mid/lo, 2 = lo):
//   2 planes: a1*b0, a0*b1, a0*b0           3 planes: a1*b1, a0*b2, a2*b0, a0*b1, a1*b0, a0*b0
// Both kernels add them in this order, so a CTA-pair tile and a single-CTA tile agree bit for bit.
__host__ __device__ constexpr int plane_products(int planes) { return planes == 1 ? 1 : (planes == 2 ? 3 : 6); }
__device__ __forceinline__ int2 plane_product(int planes, int i) {   // (plane of A, plane of B) of product i
  constexpr int PA2[3] = {1, 0, 0}, PB2[3] = {0, 1, 0};
  constexpr int PA3[6] = {1, 0, 2, 0, 1, 0}, PB3[6] = {1, 2, 0, 1, 0, 0};
  if (planes == 1) return make_int2(0, 0);
  return planes == 2 ? make_int2(PA2[i], PB2[i]) : make_int2(PA3[i], PB3[i]);
}

// The MMAs of one stage into the accumulator at d_tmem; the first MMA of a tile (accumulate == 0) overwrites it.
// PAIR: tcgen05.mma.cta_group::2, issued by the leader of a CTA pair for both CTAs.
template <class Cfg, int PLANES, bool A_MN, bool B_MN, bool PAIR>
__device__ __forceinline__ void mma_stage(uint32_t sa, uint32_t sb, uint32_t d_tmem, uint32_t idesc, uint32_t& accumulate) {
#pragma unroll
  for (int i = 0; i < plane_products(PLANES); ++i) {
    const int2 pp = plane_product(PLANES, i);
    const uint32_t a_base = sa + pp.x * Cfg::A_BYTES, b_base = sb + pp.y * Cfg::B_BYTES;
#pragma unroll
    for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
      const uint64_t da = A_MN ? umma_smem_desc(a_base + k * (UMMA_K * 128), BLOCK_K * 128, 1024)
                               : umma_smem_desc(a_base + k * (UMMA_K * 2), 16, 1024);
      const uint64_t db = B_MN ? umma_smem_desc(b_base + k * (UMMA_K * 128), BLOCK_K * 128, 1024)
                               : umma_smem_desc(b_base + k * (UMMA_K * 2), 16, 1024);
      if constexpr (PAIR) umma_f16_pair(d_tmem, da, db, idesc, accumulate);
      else umma_f16(d_tmem, da, db, idesc, accumulate);
      accumulate = 1;
    }
  }
}

// The epilogue warps (4 .. 15) of either kernel: tiles first_tile, first_tile + tile_stride, ...  A tile has tile_rows
// accumulator rows; this CTA holds BLOCK_M of them from row_off on.  full_bar / drained_bar: the CTA's barriers
// "accumulator a complete" and "accumulator a drained" (32 * NUM_EPI_WARPS arrivals), a = 0 at the address given,
// a = 1 eight bytes on.  The wait for accumulator a reports wait_code + a to the watchdog.
template <int PLANES, int BLOCK_N, bool LN>
__device__ __forceinline__ void epilogue_role(const GemmKernelArgs& args, int warp, int lane, uint32_t epi_stage_base,
                                              uint32_t tmem_base, int first_tile, int tile_stride, int tile_rows,
                                              int row_off, uint32_t full_bar, uint32_t drained_bar, uint32_t wait_code) {
  setmaxnreg_inc<EPI_REGS>();
  const int w = (warp - 4) & 3;          // TMEM lane quarter (warp % 4) -> accumulator rows 32w .. 32w+31
  const int cgroup = (warp - 4) >> 2;    // this warp handles the 32-column chunks with c % EPI_CG == cgroup
  const GemmEpilogue& e = args.epi;
  const float pe_alpha = (e.flags & EPI_PE) ? __ldg(e.pe_alpha) : 0.f;
  const float alpha = e.alpha * (e.alpha_ptr != nullptr ? __ldg(e.alpha_ptr) : 1.f);
  const float cs_scale = e.colsum_scale_ptr != nullptr ? __ldg(e.colsum_scale_ptr) : 1.f;
  const uint32_t stage_buf = epi_stage_base + (warp - 4) * (EPI_STAGE_BYTES + EPI_BIAS_BYTES);
  const uint32_t bias_buf = stage_buf + EPI_STAGE_BYTES;
  const int total_tiles = num_tiles(args);
  int it = 0;
  for (int tile = first_tile; tile < total_tiles; tile += tile_stride, ++it) {
    const TileIdx t = decode_tile(args, tile);
    const int acc = it & 1;
    const uint32_t acc_phase = (it >> 1) & 1;
    if (e.flags & EPI_BIAS) {   // bias of this warp's chunks (cgroup + EPI_CG j) -> shared memory, before the accumulator is due
      const int j = lane >> 3;
      const int cloc = (cgroup + j * EPI_CG) * 32;
      const int col = t.tn * BLOCK_N + cloc + (lane & 7) * 4;
      float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
      if (cloc < BLOCK_N && col < args.N) b = __ldg(reinterpret_cast<const float4*>(e.bias + col));
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(bias_buf + lane * 16), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
      __syncwarp();
    }
    mbar_wait(full_bar + 8u * acc, acc_phase, wait_code + acc);
    tc_fence_after();
    const int64_t row0 = static_cast<int64_t>(t.tm) * tile_rows + row_off + w * 32;
    const int64_t out_boff = t.i0 * e.out_sb0 + t.i1 * e.out_sb1;
    const int64_t res_boff = t.i0 * e.res_sb0 + t.i1 * e.res_sb1;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(w * 32) << 16) + acc * BLOCK_N;
    const int64_t cs_boff = t.i0 * e.colsum_sb0;
    if constexpr (LN) {
      if (row0 < args.M)
        ln_epilogue_tile<BLOCK_N>(e, stage_buf, bias_buf, lane, cgroup, w, t_row, args.M, args.N, row0, t.batch, out_boff,
                                  res_boff, alpha);
    } else
    if (row0 < args.M) {   // warp-uniform
      constexpr uint32_t CT_LEAN = EPI_BIAS | EPI_RELU | EPI_OUT_F32;
      // the bit-mask classes only exist in the multi-plane kernels: the one-plane (inference) kernels stay small
      constexpr uint32_t CT_FWD = CT_LEAN | EPI_PE | EPI_DROPOUT | EPI_RES | (PLANES >= 2 ? EPI_EMIT_BITS : 0u);
      constexpr uint32_t CT_BWD = EPI_GATE_BITS | EPI_COLSUM | EPI_RES | EPI_OUT_F32;   // data gradients
      if ((e.flags & ~CT_LEAN) == 0)
        epilogue_tile<CT_LEAN, BLOCK_N>(e, stage_buf, bias_buf, lane, cgroup, t_row, args.M, args.N, row0, t.batch, out_boff,
                                        res_boff, cs_boff, t.tn, pe_alpha, alpha, cs_scale);
      else if ((e.flags & ~CT_FWD) == 0)
        epilogue_tile<CT_FWD, BLOCK_N>(e, stage_buf, bias_buf, lane, cgroup, t_row, args.M, args.N, row0, t.batch, out_boff,
                                       res_boff, cs_boff, t.tn, pe_alpha, alpha, cs_scale);
      else if (PLANES >= 2 && (e.flags & ~CT_BWD) == 0)
        epilogue_tile<(PLANES >= 2 ? CT_BWD : 0xFFFFFFFFu), BLOCK_N>(e, stage_buf, bias_buf, lane, cgroup, t_row, args.M, args.N,
                                                                     row0, t.batch, out_boff, res_boff, cs_boff, t.tn, pe_alpha,
                                                                     alpha, cs_scale);
      else
        epilogue_tile<0xFFFFFFFFu, BLOCK_N>(e, stage_buf, bias_buf, lane, cgroup, t_row, args.M, args.N, row0, t.batch, out_boff,
                                            res_boff, cs_boff, t.tn, pe_alpha, alpha, cs_scale);
    }
    tc_fence_before();
    mbar_arrive(drained_bar + 8u * acc);
  }
}

// ------------------------------------------------------------------------------------------------
// LN = true: the instantiation whose ONLY epilogue is the fused LayerNorm (EPI_LN); it is a kernel of its own so that the
// extra code and registers do not touch the other epilogues (built into the common kernel it cost them 2 %).
template <bool A_MN, bool B_MN, int PLANES, int BLOCK_N, bool LN = false>
__global__ void __launch_bounds__(128 + 32 * NUM_EPI_WARPS, 1) gemm_tc_kernel(const __grid_constant__ GemmKernelArgs args) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  using Cfg = TileCfg<PLANES, BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr uint32_t IDESC = umma_idesc_f16(BLOCK_M, BLOCK_N, A_MN, B_MN);

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * Cfg::STAGE_BYTES;
  // barrier layout: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2], tmem_ptr
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  const uint32_t epi_stage_base = bar_base + BAR_BYTES;
  auto sA = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };   // stage s: planes of A, then planes of B
  auto sB = [&](int s) { return sA(s) + PLANES * Cfg::A_BYTES; };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int p = 0; p < PLANES; ++p) {
      tma_prefetch_desc(&args.a_map[p]);
      tma_prefetch_desc(&args.b_map[p]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 32 * NUM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                          // everything above overlapped the previous kernel's tail; operands are ready now
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int total_tiles = num_tiles(args);

  if (warp < 4) {
    setmaxnreg_dec<CTRL_REGS>();
    if (warp == 0) {
      // ===================================================================== TMA producer
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
          const TileIdx t = decode_tile(args, tile);
          for (int kb = t.kb_begin; kb < t.kb_end; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, 0x100u + stage);
            mbar_arrive_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
            load_stage<Cfg, PLANES, A_MN, B_MN>(args, sA(stage), sB(stage), full_bar(stage), kb, t.tm * BLOCK_M,
                                                t.tn * BLOCK_N, t.i0, t.i1);
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    } else if (warp == 1) {
      // ===================================================================== MMA issuer
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
          const TileIdx t = decode_tile(args, tile);
          const int acc = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u, 0x200u + acc);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
          uint32_t accumulate = 0;
          for (int kb = t.kb_begin; kb < t.kb_end; ++kb) {
            mbar_wait(full_bar(stage), phase, 0x300u + stage);
            tc_fence_after();
            mma_stage<Cfg, PLANES, A_MN, B_MN, false>(sA(stage), sB(stage), d_tmem, IDESC, accumulate);
            umma_commit(empty_bar(stage));        // frees the smem slot when these MMAs retire
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
          umma_commit(tfull_bar(acc));            // accumulator ready for the epilogue
        }
      }
    }
  } else {
    // ===================================================================== epilogue
    epilogue_role<PLANES, BLOCK_N, LN>(args, warp, lane, epi_stage_base, tmem_base, blockIdx.x, gridDim.x, BLOCK_M, 0,
                                       tfull_bar(0), tempty_bar(0), 0x400u);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05.mma.cta_group::2): two CTAs of a cluster work on one 256 x BLOCK_N tile.  Each CTA
// stages its own 128 rows of A and HALF of the B tile (BLOCK_N / 2 rows), the leader (cluster rank 0) issues the
// MMAs for both tensor cores, each CTA's accumulator half (its 128 rows x BLOCK_N columns) lands in its own TMEM and
// is drained by its own epilogue warps.  Per SM the UMMA operand reads drop from 128 / 96 B/clk (BLOCK_N = 128 / 256
// single-CTA tiles) to 64 B/clk, which leaves shared-memory bandwidth for the epilogue's staging round trips
// (profiles/r01_gemm_epilogue.md), and a three-plane ring fits BLOCK_N = 256.
//   full[s]      local TMA completion of stage s                     (each CTA, its own loads)
//   peer_full[s] leader only: the peer's stage s is loaded           (remote arrive by the peer's relay lane)
//   empty[s]     both CTAs, signalled by the leader's commit (multicast)
//   tfull[a]     both CTAs, leader's commit (multicast): accumulator a complete
//   tlocal[a]    each CTA: its 384 epilogue threads have drained accumulator a (CTA-scope arrives: a cluster-scope
//                release from every epilogue thread would wait for its outstanding global stores)
//   tempty[a]    leader only: one remote arrive per CTA, forwarded by the idle warp 3 once tlocal[a] completes
template <int PLANES, int BLOCK_N>
struct PairCfg {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_ROWS = BLOCK_N / 2;
  static constexpr int B_BYTES = B_ROWS * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = PLANES * (A_BYTES + B_BYTES);
  static constexpr int RAW_STAGES = (SMEM_LIMIT - 1024 - BAR_BYTES - EPI_SMEM) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 6 ? 6 : RAW_STAGES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES + EPI_SMEM;
  static constexpr int TMEM_COLS = 512;
  static_assert(STAGES >= 2, "operand ring does not fit shared memory");
  static_assert(2 * BLOCK_N <= 512 && BLOCK_N % 128 == 0, "pair tile N");
};

template <bool B_MN, int PLANES, int BLOCK_N, bool LN = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128 + 32 * NUM_EPI_WARPS, 1)
    gemm_pair_kernel(const __grid_constant__ GemmKernelArgs args) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  using Cfg = PairCfg<PLANES, BLOCK_N>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr uint32_t IDESC = umma_idesc_f16(2 * BLOCK_M, BLOCK_N, false, B_MN);

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * Cfg::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto pfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (3 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (3 * STAGES + 2 + a); };
  auto tlocal_bar = [&](int a) { return bar_base + 8u * (3 * STAGES + 4 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (3 * STAGES + 6);
  const uint32_t epi_stage_base = bar_base + BAR_BYTES;
  auto sA = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };   // stage s: planes of A, then planes of B
  auto sB = [&](int s) { return sA(s) + PLANES * Cfg::A_BYTES; };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  // This pair's tiles: pair_id(), + num_pairs(), ...  The two are read where used: kept in registers across all warp
  // roles they cost spill slots (ptxas: 92 / 88 spill bytes instead of 120 / 132 at two planes).
  auto pair_id = [] { return static_cast<int>(cluster_id_x()); };
  auto num_pairs = [] { return static_cast<int>(cluster_count_x()); };

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int p = 0; p < PLANES; ++p) {
      tma_prefetch_desc(&args.a_map[p]);
      tma_prefetch_desc(&args.b_map[p]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
      mbar_init(pfull_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2);                       // one arrive per CTA, from its relay lane
      mbar_init(tlocal_bar(a), 32 * NUM_EPI_WARPS);      // this CTA's epilogue threads
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc2(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish2();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync();                      // barriers of both CTAs exist before any remote arrive / multicast commit
  pdl_wait();                          // the prologue overlapped the previous kernel's tail; operands are ready now
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int total_tiles = num_tiles(args);       // tiles_m counts 256-row tiles here

  if (warp < 4) {
    setmaxnreg_dec<CTRL_REGS>();
    if (warp == 0) {
      // ===================================================================== TMA producer (both CTAs)
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = pair_id(); tile < total_tiles; tile += num_pairs()) {
          const TileIdx t = decode_tile(args, tile);
          const int arow = t.tm * 2 * BLOCK_M + static_cast<int>(rank) * BLOCK_M;
          const int brow = t.tn * BLOCK_N + static_cast<int>(rank) * Cfg::B_ROWS;
          for (int kb = t.kb_begin; kb < t.kb_end; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, 0x900u + stage);
            mbar_arrive_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
            load_stage<Cfg, PLANES, false, B_MN>(args, sA(stage), sB(stage), full_bar(stage), kb, arow, brow, t.i0, t.i1);
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        if (rank != 0) {
          // =================================================================== peer: relay "my stage is loaded"
          for (int tile = pair_id(); tile < total_tiles; tile += num_pairs()) {
            const TileIdx t = decode_tile(args, tile);
            for (int kb = t.kb_begin; kb < t.kb_end; ++kb) {
              mbar_wait(full_bar(stage), phase, 0xA00u + stage);
              mbar_arrive_cluster(mapa_shared(pfull_bar(stage), 0));
              if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
          }
        } else {
          // =================================================================== leader: MMA issuer for the pair
          int it = 0;
          for (int tile = pair_id(); tile < total_tiles; tile += num_pairs(), ++it) {
            const TileIdx t = decode_tile(args, tile);
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait_cluster(tempty_bar(acc), acc_phase ^ 1u, 0xB00u + acc);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
            uint32_t accumulate = 0;
            for (int kb = t.kb_begin; kb < t.kb_end; ++kb) {
              mbar_wait(full_bar(stage), phase, 0xC00u + stage);
              mbar_wait_cluster(pfull_bar(stage), phase, 0xD00u + stage);
              tc_fence_after();
              mma_stage<Cfg, PLANES, false, B_MN, true>(sA(stage), sB(stage), d_tmem, IDESC, accumulate);
              umma_commit_pair(empty_bar(stage));       // frees the slot in both CTAs when these MMAs retire
              if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
            umma_commit_pair(tfull_bar(acc));           // both halves of the accumulator are complete
          }
        }
      }
    } else if (warp == 3) {
      // =================================================================== both CTAs: forward "accumulator drained"
      if (lane == 0) {
        const uint32_t te0 = mapa_shared(tempty_bar(0), 0), te1 = mapa_shared(tempty_bar(1), 0);
        int it = 0;
        for (int tile = pair_id(); tile < total_tiles; tile += num_pairs(), ++it) {
          const int acc = it & 1;
          mbar_wait(tlocal_bar(acc), (it >> 1) & 1, 0xF00u + acc);
          mbar_arrive_cluster(acc ? te1 : te0);
        }
      }
    }
  } else {
    // ===================================================================== epilogue (both CTAs, own rows)
    epilogue_role<PLANES, BLOCK_N, LN>(args, warp, lane, epi_stage_base, tmem_base, pair_id(), num_pairs(), 2 * BLOCK_M,
                                       static_cast<int>(rank) * BLOCK_M, tfull_bar(0), tlocal_bar(0), 0xE00u);
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync();                      // the leader's MMAs read the peer's shared memory: nobody leaves early
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// Host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int device_sm_count() {
  static int sms[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (sms[dev] == 0) {      // benign race: every thread writes the same value
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    sms[dev] = n;
  }
  return sms[dev];
}

// 4-D map {cols, rows, nb0, nb1}; box = {64, box_rows, 1, 1}; fp16; 128-byte swizzle; OOB -> zeros.
static int make_map(CUtensorMap* map, const SplitMat& m, int plane, int nb0, int nb1, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  SPK_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available");
  const bool batched = (m.sb0 != 0 || m.sb1 != 0);
  char* base = reinterpret_cast<char*>(const_cast<void*>(m.base)) + static_cast<int64_t>(plane) * m.plane_stride * 2;
  SPK_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "GEMM operand base must be 16-byte aligned");
  SPK_CHECK((m.ld * 2) % 16 == 0, "GEMM operand row stride must be a multiple of 16 bytes (ld=%lld)", (long long)m.ld);
  const int64_t dflt = m.rows * m.ld;
  cuuint64_t dims[4] = {(cuuint64_t)m.cols, (cuuint64_t)m.rows, (cuuint64_t)(batched ? nb0 : 1),
                        (cuuint64_t)(batched ? nb1 : 1)};
  int64_t s0 = (batched && nb0 > 1) ? m.sb0 : dflt;
  int64_t s1 = (batched && nb1 > 1) ? m.sb1 : dflt * (batched ? nb0 : 1);
  if (s0 <= 0) s0 = dflt;
  if (s1 <= 0) s1 = dflt;
  SPK_CHECK((s0 * 2) % 16 == 0 && (s1 * 2) % 16 == 0, "GEMM batch strides must be multiples of 16 bytes");
  cuuint64_t strides[3] = {(cuuint64_t)(m.ld * 2), (cuuint64_t)(s0 * 2), (cuuint64_t)(s1 * 2)};
  cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SPK_CHECK(r == CUDA_SUCCESS,
            "cuTensorMapEncodeTiled failed (%d): dims %llu x %llu x %llu x %llu ld %lld box_rows %d", (int)r,
            (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2],
            (unsigned long long)dims[3], (long long)m.ld, box_rows);
  return 0;
}

int encode_map_4d(CUtensorMap* map, const void* base, const int64_t dims[4], const int64_t strides[3], int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  SPK_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available");
  SPK_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "tensor map base must be 16-byte aligned");
  cuuint64_t d[4] = {(cuuint64_t)dims[0], (cuuint64_t)dims[1], (cuuint64_t)dims[2], (cuuint64_t)dims[3]};
  cuuint64_t st[3] = {(cuuint64_t)(strides[0] * 2), (cuuint64_t)(strides[1] * 2), (cuuint64_t)(strides[2] * 2)};
  SPK_CHECK(st[0] % 16 == 0 && st[1] % 16 == 0 && st[2] % 16 == 0, "tensor map strides must be multiples of 16 bytes");
  cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), d, st, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SPK_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

// A kernel instantiation, its dynamic shared memory size and its one-time set-up (per device).
struct GemmKernel {
  void (*fn)(GemmKernelArgs) = nullptr;
  int smem = 0;
  PerDeviceOnce* configured = nullptr;
};

// Three planes of A and B only fit a double-buffered operand ring up to BLOCK_N = 128.
constexpr int max_block_n(int planes) { return planes == 3 ? 128 : 256; }
constexpr int PAIR_BN = 256;

template <bool A_MN, bool B_MN, int PLANES, int BLOCK_N, bool LN = false>
static GemmKernel tc_entry() {
  if constexpr (BLOCK_N > max_block_n(PLANES)) {
    return {};
  } else {
    static PerDeviceOnce once;
    return {gemm_tc_kernel<A_MN, B_MN, PLANES, BLOCK_N, LN>, TileCfg<PLANES, BLOCK_N>::SMEM_BYTES, &once};
  }
}
template <bool A_MN, bool B_MN, int PLANES>
static GemmKernel tc_entry_bn(int block_n) {
  switch (block_n) {
    case 64: return tc_entry<A_MN, B_MN, PLANES, 64>();
    case 128: return tc_entry<A_MN, B_MN, PLANES, 128>();
    case 192: return tc_entry<A_MN, B_MN, PLANES, 192>();
    case 256: return tc_entry<A_MN, B_MN, PLANES, 256>();
  }
  return {};
}
template <int PLANES>
static GemmKernel tc_entry_planes(bool a_mn, bool b_mn, int block_n, bool ln) {
  if (ln) {   // the fused LayerNorm: K-major operands, BLOCK_N = N = 256, one or two planes
    if constexpr (PLANES <= 2)
      if (!a_mn && !b_mn && block_n == 256) return tc_entry<false, false, PLANES, 256, true>();
    return {};
  }
  if (!a_mn) return b_mn ? tc_entry_bn<false, true, PLANES>(block_n) : tc_entry_bn<false, false, PLANES>(block_n);
  return b_mn ? tc_entry_bn<true, true, PLANES>(block_n) : GemmKernel{};   // A MN-major with B K-major is not built
}
// The single-CTA instantiations: (A, B) K/K-, K/MN- or MN/MN-major, BLOCK_N = 64 / 128 / 192 / 256 up to
// max_block_n(planes), one to three planes, and the fused-LayerNorm kernels; {} for a combination that is not built.
static GemmKernel tc_kernel(bool a_mn, bool b_mn, int planes, int block_n, bool ln) {
  switch (planes) {
    case 1: return tc_entry_planes<1>(a_mn, b_mn, block_n, ln);
    case 2: return tc_entry_planes<2>(a_mn, b_mn, block_n, ln);
    case 3: return tc_entry_planes<3>(a_mn, b_mn, block_n, ln);
  }
  return {};
}

template <bool B_MN, int PLANES, bool LN = false>
static GemmKernel pair_entry() {
  static PerDeviceOnce once;
  return {gemm_pair_kernel<B_MN, PLANES, PAIR_BN, LN>, PairCfg<PLANES, PAIR_BN>::SMEM_BYTES, &once};
}
// The CTA-pair instantiations (A K-major, BLOCK_N = PAIR_BN): two or three planes; the fused LayerNorm at two planes
// with B K-major.
static GemmKernel pair_kernel(bool b_mn, int planes, bool ln) {
  if (ln) return (planes == 2 && !b_mn) ? pair_entry<false, 2, true>() : GemmKernel{};
  if (planes == 2) return b_mn ? pair_entry<true, 2>() : pair_entry<false, 2>();
  if (planes == 3) return b_mn ? pair_entry<true, 3>() : pair_entry<false, 3>();
  return {};
}

// Opt in to the kernel's dynamic shared memory size and check its register count, once per device.
static int configure(const GemmKernel& k) {
  return k.configured->run([&]() -> int {
    SPK_CUDA(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, k.smem));
    cudaFuncAttributes fa;
    SPK_CUDA(cudaFuncGetAttributes(&fa, k.fn));
    // setmaxnreg re-partitions the launch allocation; another launch register count would dead-lock the epilogue warps
    SPK_CHECK(fa.numRegs == LAUNCH_REGS, "gemm kernel was built with %d registers/thread, expected %d", fa.numRegs,
              LAUNCH_REGS);
    return 0;
  });
}
// The single-CTA kernels without the fused LayerNorm are configured up front (CUDA loads kernels lazily: a first launch
// of a new instantiation inside a timed region -- a new frame length picks another BLOCK_N -- would pay for the load).
// The fused-LayerNorm and CTA-pair kernels are configured on first use.
static int configure_all() {
  static PerDeviceOnce once;
  return once.run([]() -> int {
    for (int planes = 1; planes <= 3; ++planes)
      for (const bool a_mn : {false, true})
        for (const bool b_mn : {false, true})
          for (int block_n = 64; block_n <= 256; block_n += 64) {
            const GemmKernel k = tc_kernel(a_mn, b_mn, planes, block_n, false);
            if (k.fn != nullptr) SPK_TRY(configure(k));
          }
    return 0;
  });
}

// spk_set_option("gemm_dependent_launch", 0 | 1 | 2): 0 off, 1 inside the inference forward only, 2 (default) every GEMM.
// Measured (same process, alternating): inference 960 x 200 frames 1.904 -> 1.842 ms, 7 x 33 frames 0.246 -> 0.237 ms,
// identical d-vectors; training step, drift-balanced order (tools/train_ab_balanced.py): 8.623 (1) -> 8.574 ms (2).
static int g_gemm_pdl = 2;
void gemm_set_dependent_launch(int on) { g_gemm_pdl = on; }
static thread_local int t_gemm_pdl_scope = 0;      // > 0 while an inference forward enqueues its kernels
GemmDependentLaunchScope::GemmDependentLaunchScope(bool on) : on_(on) { if (on_) ++t_gemm_pdl_scope; }
GemmDependentLaunchScope::~GemmDependentLaunchScope() { if (on_) --t_gemm_pdl_scope; }

// A GEMM launched with the programmatic-stream-serialisation attribute runs its prologue under the tail of the kernel
// before it (which calls pdl_trigger() at its start) and its main part after pdl_wait().
static int launch_gemm_kernel(const GemmKernel& k, int grid, cudaStream_t stream, const GemmKernelArgs& args) {
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(128 + 32 * NUM_EPI_WARPS);
  cfg.dynamicSmemBytes = k.smem;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = (g_gemm_pdl >= 2 || (g_gemm_pdl == 1 && t_gemm_pdl_scope > 0)) ? 1 : 0;
  SPK_CUDA(cudaLaunchKernelEx(&cfg, k.fn, args));
  return 0;
}

static int g_cta_pairs = 1;            // spk_set_option("gemm_cta_pairs", 0/1)
void gemm_set_cta_pairs(int on) { g_cta_pairs = on; }

int gemm_run(const GemmProblem& p, cudaStream_t stream) {
  SPK_CHECK(p.M > 0 && p.N > 0 && p.K > 0, "gemm: empty problem %d x %d x %d", p.M, p.N, p.K);
  SPK_CHECK(p.planes >= 1 && p.planes <= 3, "gemm: planes must be 1, 2 or 3");
  SPK_CHECK(p.N % 8 == 0, "gemm: N (%d) must be a multiple of 8", p.N);
  SPK_CHECK(p.epi.out != nullptr, "gemm: no output");
  SPK_CHECK(p.ksplit == 1 || (p.epi.flags & EPI_OUT_ATOMIC), "gemm: split-K needs the atomic epilogue");
  if (p.epi.flags & (EPI_EMIT_BITS | EPI_GATE_BITS))
    SPK_CHECK(p.epi.gate_bits != nullptr && p.N % 32 == 0 && p.nb0 * p.nb1 == 1,
              "gemm: the ReLU bit mask needs N %% 32 == 0 and an unbatched problem");
  // the non-contraction extent of an operand may be smaller than M / N: TMA zero-fills the rest
  if (!p.a_mn) SPK_CHECK(p.A.rows <= p.M && p.A.cols == p.K, "gemm: A is not [<=M, K]");
  else SPK_CHECK(p.A.rows == p.K && p.A.cols <= p.M, "gemm: A is not [K, <=M]");
  if (!p.b_mn) SPK_CHECK(p.B.rows <= p.N && p.B.cols == p.K, "gemm: B is not [<=N, K]");
  else SPK_CHECK(p.B.rows == p.K && p.B.cols <= p.N, "gemm: B is not [K, <=N]");

  SPK_TRY(configure_all());

  const bool ln = (p.epi.flags & EPI_LN) != 0;
  if (ln)
    SPK_CHECK(p.N == 256 && p.nb0 * p.nb1 == 1 && p.ksplit <= 1 && p.epi.ln_gamma != nullptr && p.epi.ln_beta != nullptr &&
                  !p.a_mn && !p.b_mn && p.planes <= 2 &&
                  !(p.epi.flags & (EPI_OUT_F32 | EPI_OUT_ATOMIC | EPI_RELU | EPI_PE | EPI_COLSUM | EPI_GATE_BITS |
                                   EPI_GATE_POS | EPI_EMIT_BITS | EPI_ACC_GATES_AUX)),
              "gemm: the fused LayerNorm needs N == 256, an unbatched problem and a bias / dropout / residual epilogue");
  // Problems with few rows (the pruned last layer: M = slices) are latency-bound: 256-wide tiles would put them on 8-32
  // CTAs that each walk the whole K loop; 64-wide single-CTA tiles spread the same work over 4x as many SMs.
  int req_bn = p.block_n;
  if (req_bn == 0 && !p.a_mn && p.ksplit <= 1 && p.nb0 * p.nb1 == 1 && p.M <= 2048 && p.N >= 128) req_bn = 64;
  const bool ln_pair = ln && p.planes == 2 && p.M > 2048 && g_cta_pairs;
  if (ln && !ln_pair) req_bn = 256;      // the fused LayerNorm runs in its own instantiations

  // CTA-pair path: K-major A, two or three planes, no split-K, 256-wide N tiles (128 columns of B per CTA)
  const bool pair =
      g_cta_pairs && !p.a_mn && p.planes >= 2 && p.ksplit <= 1 && req_bn == 0 && p.N % 128 == 0 && p.M >= 256;
  int bn = pair ? PAIR_BN : req_bn;
  if (bn == 0) bn = p.N <= 64 ? 64 : (p.N <= 128 ? 128 : (p.N <= 192 ? 192 : 256));
  if (!pair && bn > max_block_n(p.planes)) bn = max_block_n(p.planes);
  const int tile_m = pair ? 2 * BLOCK_M : BLOCK_M;
  const GemmKernel kern = pair ? pair_kernel(p.b_mn, p.planes, ln) : tc_kernel(p.a_mn, p.b_mn, p.planes, bn, ln);
  SPK_CHECK(kern.fn != nullptr, "gemm: no kernel for %d planes, A %s-major, B %s-major, BLOCK_N %d%s", p.planes,
            p.a_mn ? "MN" : "K", p.b_mn ? "MN" : "K", bn, ln ? ", fused LayerNorm" : "");
  SPK_TRY(configure(kern));

  GemmKernelArgs a;
  memset(&a, 0, sizeof(a));
  for (int pl = 0; pl < p.planes; ++pl) {
    SPK_TRY(make_map(&a.a_map[pl], p.A, pl, p.nb0, p.nb1, p.a_mn ? BLOCK_K : BLOCK_M));
    SPK_TRY(make_map(&a.b_map[pl], p.B, pl, p.nb0, p.nb1, p.b_mn ? BLOCK_K : (pair ? bn / 2 : bn)));
  }
  a.M = p.M; a.N = p.N; a.K = p.K;
  a.tiles_m = (p.M + tile_m - 1) / tile_m;
  a.tiles_n = (p.N + bn - 1) / bn;
  a.nb0 = p.nb0; a.nb1 = p.nb1;
  a.kb_total = (p.K + BLOCK_K - 1) / BLOCK_K;
  int ks = p.ksplit < 1 ? 1 : p.ksplit;
  if (ks > a.kb_total) ks = a.kb_total;
  a.kb_per_split = (a.kb_total + ks - 1) / ks;
  a.ksplit = (a.kb_total + a.kb_per_split - 1) / a.kb_per_split;
  a.a_batched = (p.A.sb0 != 0 || p.A.sb1 != 0);
  a.b_batched = (p.B.sb0 != 0 || p.B.sb1 != 0);
  a.epi = p.epi;
  const long long total = 1LL * a.nb0 * a.nb1 * a.ksplit * a.tiles_m * a.tiles_n;
  SPK_CHECK(total < (1LL << 30), "gemm: too many tiles");
  const double nb = 1.0 * p.nb0 * p.nb1;
  const double esz = 2.0 * p.planes;
  const double out_b = (p.epi.flags & (EPI_OUT_F32 | EPI_OUT_ATOMIC)) ? 4.0 : esz;
  double bytes = nb * (1.0 * p.M * p.K * esz + 1.0 * p.M * p.N * out_b) +
                 (a.b_batched ? nb : 1.0) * p.N * p.K * esz;
  if (p.epi.flags & (EPI_RES | EPI_ACC_GATES_AUX)) bytes += nb * p.M * p.N * 2.0 * p.epi.res_planes;
  if (p.epi.flags & EPI_GATE_POS) bytes += nb * p.M * p.N * 2.0 * p.epi.gate_planes;
  const int sms = device_sm_count();
  ProfScope prof(p.tag, 2.0 * nb * p.M * p.N * p.K, bytes, stream);

  if (pair) {
    const int max_pairs = sms / 2;
    const int pairs = static_cast<int>(total < max_pairs ? total : max_pairs);
    return launch_gemm_kernel(kern, 2 * pairs, stream, a);   // __cluster_dims__(2,1,1)
  }
  return launch_gemm_kernel(kern, static_cast<int>(total < sms ? total : sms), stream, a);
}

}  // namespace spk
