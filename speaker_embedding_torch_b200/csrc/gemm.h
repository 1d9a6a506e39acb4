// Host-side description of one (batched, optionally split-K) tensor-core GEMM on split-fp16 operands.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace spk {

// A row-major matrix (cols contiguous) stored as 1 or 2 fp16 planes, optionally batched over two
// outer indices.  As a GEMM operand it is "K-major" when cols is the contraction dim and
// "MN-major" when rows is the contraction dim (A^T / B^T reads, no transposed copy is ever made).
struct SplitMat {
  const void* base = nullptr;   // fp16
  int64_t plane_stride = 0;     // elements from the hi plane to the lo plane
  int64_t rows = 0, cols = 0;   // per-batch extents as stored
  int64_t ld = 0;               // elements between consecutive rows
  int64_t sb0 = 0, sb1 = 0;     // batch strides, elements (both 0: broadcast over batches)
};

enum : uint32_t {
  EPI_BIAS = 1u << 0,       // v += bias[col]
  EPI_RELU = 1u << 1,       // v = max(v, 0)
  EPI_PE = 1u << 2,         // v += *pe_alpha * pe_t[(row % pe_T) * N + col]
  EPI_DROPOUT = 1u << 3,    // v *= keep(seed, site, elem) / (1 - p)
  EPI_RES = 1u << 4,        // v += res[row, col]                      (after dropout)
  EPI_GATE_POS = 1u << 5,   // v = gate[row, col] > 0 ? v * gate_scale : 0   (ReLU backward from saved output)
  EPI_ACC_GATES_AUX = 1u << 6,  // v = (v > 0) ? res[row, col] * dropout_keep : 0  (prenet backward by recompute)
  EPI_COLSUM = 1u << 7,     // colsum[col] += sum_rows(v)  (bias gradient fused into the producing GEMM)
  EPI_OUT_F32 = 1u << 8,    // plain fp32 store instead of split planes
  EPI_OUT_ATOMIC = 1u << 9,  // fp32 atomicAdd (split-K weight gradients)
  EPI_EMIT_BITS = 1u << 10,  // gate_bits[col/32, row]: bit i set iff v[col0 + i] > 0   (forward: ReLU mask for the backward;
                             // with EPI_PE the mask is taken right after the ReLU, otherwise after dropout)
  EPI_GATE_BITS = 1u << 11,  // v = bit ? v * gate_scale : 0 from gate_bits (ReLU backward, 1 bit per element)
  EPI_LN = 1u << 12          // out = LayerNorm(v) * ln_gamma + ln_beta over the row (after bias / dropout / residual):
                             // needs N == 256 (one tile owns whole rows), an unbatched problem and split-plane output
};

struct GemmEpilogue {
  uint32_t flags = 0;
  float alpha = 1.f;             // v = alpha * acc first
  const float* alpha_ptr = nullptr;   // optional device scalar multiplied into alpha (the backward pass's 1 / gradient scale)
  const float* colsum_scale_ptr = nullptr;   // optional device scalar applied to the fused column sums
  const float* bias = nullptr;   // [N] fp32
  const float* pe_t = nullptr;   // [pe_T, N] fp32
  const float* pe_alpha = nullptr;
  int pe_T = 1;
  DropCfg drop = {0, 0, 1.f};
  uint32_t drop_site = 0;
  // residual / aux operand, indexed like the output
  const void* res = nullptr;
  int64_t res_plane_stride = 0, res_ld = 0, res_sb0 = 0, res_sb1 = 0;
  int res_planes = 1;
  // gate operand
  const void* gate = nullptr;
  int64_t gate_plane_stride = 0, gate_ld = 0;
  int gate_planes = 1;
  float gate_scale = 1.f;
  uint32_t* gate_bits = nullptr;   // [N / 32, M] words, chunk-major (N % 32 == 0, unbatched): EPI_EMIT_BITS writes, EPI_GATE_BITS reads
  // fused LayerNorm over the N = 256 columns of every output row (EPI_LN)
  const float* ln_gamma = nullptr;
  const float* ln_beta = nullptr;
  float ln_eps = 1e-5f;
  void* ln_z = nullptr;            // optional: the pre-normalisation rows (split planes, laid out like `out`) for a backward pass
  int64_t ln_z_plane_stride = 0;
  float* ln_stats = nullptr;       // optional: (mean, rstd) per row, [M] float2
  // fused column sums (fp32, atomically accumulated); colsum_sb0: elements per batch index i0
  float* colsum = nullptr;
  int64_t colsum_sb0 = 0;
  // output: split planes (default) or fp32
  void* out = nullptr;
  int64_t out_plane_stride = 0, out_ld = 0, out_sb0 = 0, out_sb1 = 0;   // batch strides, elements
  int out_planes = 1;
};

struct GemmProblem {
  SplitMat A, B;        // A: [M,K] (K-major) or [K,M] (MN-major); B: [N,K] (K-major) or [K,N] (MN-major)
  bool a_mn = false, b_mn = false;
  int planes = 1;       // 1: Ah*Bh ; 2: + Ah*Bl + Al*Bh ; 3: six products (fp32-equivalent)
  int M = 0, N = 0, K = 0;
  int nb0 = 1, nb1 = 1; // batch extents; batch index = i1 * nb0 + i0, offset = i0 * sb0 + i1 * sb1
  int ksplit = 1;       // >1 requires EPI_OUT_ATOMIC
  int block_n = 0;      // 0 = auto (64/128/192/256)
  const char* tag = "gemm";   // profiler label
  GemmEpilogue epi;
};

// Enqueue on `stream`; returns 0 or a negative SPK_E* code (text via spk_last_error()).
int gemm_run(const GemmProblem& p, cudaStream_t stream);

int device_sm_count();
void gemm_set_dependent_launch(int mode);   // programmatic dependent launch of the GEMM kernels: 0 off, 1 inference, 2 all
// While one lives (and the option is 1), the calling thread's GEMM launches carry the dependent-launch attribute.
struct GemmDependentLaunchScope {
  explicit GemmDependentLaunchScope(bool on);
  ~GemmDependentLaunchScope();
  GemmDependentLaunchScope(const GemmDependentLaunchScope&) = delete;
  GemmDependentLaunchScope& operator=(const GemmDependentLaunchScope&) = delete;
 private:
  bool on_;
};
void gemm_set_cta_pairs(int on);   // route eligible multi-plane GEMMs through the cta_group::2 kernel

// fp16 4-D tiled tensor map {dims[0] (contiguous), dims[1], dims[2], dims[3]} with element strides for dims 1..3,
// box {64, box_rows, 1, 1}, 128-byte swizzle, out-of-bounds elements read as zero.
int encode_map_4d(CUtensorMap* map, const void* base, const int64_t dims[4], const int64_t strides[3], int box_rows);

// Map of Q (which = 0), K (1) or V (2) of one plane of the packed attention input qkv [B*T, 3*64*H], in which head h of
// Q / K / V sits at column which*64*H + h*64: dims {64, T, H, B}, so rows >= T of a (slice, head) read as zeros.
inline int encode_qkv_map(CUtensorMap* map, const void* qkv_plane, int which, int B, int H, int T, int box_rows) {
  const int64_t ld = 3 * 64 * H;
  const int64_t dims[4] = {64, T, H, B};
  const int64_t strides[3] = {ld, 64, static_cast<int64_t>(T) * ld};
  return encode_map_4d(map, static_cast<const elem_t*>(qkv_plane) + which * 64 * H, dims, strides, box_rows);
}

}  // namespace spk
