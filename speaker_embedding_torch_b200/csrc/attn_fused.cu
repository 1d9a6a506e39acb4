// Fused attention forward for inference (one fp16 plane, no dropout, T <= 256 frames):
//
//     O = softmax(Q K^T / 8) V     per (slice, head, 128-query tile), scores never leave the SM.
//
//   TMA       Q tile [128 x 64], K [Tk x 64], V [Tk x 64] straight out of the packed qkv buffer [B*T, 768]
//             (4-D tensor maps: head offset in the base pointer, frames as their own dimension -> rows >= T
//             arrive as zeros)
//   tcgen05   S = Q K^T  -> TMEM columns [0, 256)    (UMMA 128 x Tk16 x 16, both operands K-major)
//   4 warps   thread <-> query row: row max / exp / sum straight from TMEM (tcgen05.ld), unnormalised
//             probabilities written as fp16 into shared memory in the 128-byte-swizzled K-major layout
//             the tensor core reads (the same layout TMA produces), keys >= T as zeros
//   tcgen05   O = P V    -> TMEM columns [256, 320)  (V read MN-major: no transpose)
//   4 warps   O * (1 / row sum) -> fp16 -> out[(b*T + q) * 256 + h*64 ...]
//
// Replaces the QK^T GEMM + softmax kernel + PV GEMM of the dense layers in the inference path (the
// training path keeps multi-plane operands and materialised probabilities for the backward pass).
#include "gemm.h"
#include "ptx.cuh"

namespace spk {

constexpr int AF_KV_ROWS = 256;               // max keys (T <= 256)
constexpr int AF_STAGE = 16384 + 32768 + 32768;   // Q 128 x 128 B | K 256 x 128 B | V 256 x 128 B, double-buffered
constexpr int AF_SK = 16384;
constexpr int AF_SV = AF_SK + 32768;
constexpr int AF_SP = 2 * AF_STAGE;               // 4 k-blocks x (128 rows x 128 B)
constexpr int AF_BAR = AF_SP + 65536;
constexpr int AF_SMEM = AF_BAR + 128 + 1024;      // + alignment slack (230 528 B <= 227 KB)

struct AttnFusedArgs {
  CUtensorMap q_map, k_map, v_map;
  int B, H, T, Tk16, Tk64, mtiles;
  elem_t* out;      // [B*T, out_ld] plane 0, head h at column h*64
  int64_t out_ld;
};

__global__ void __launch_bounds__(256, 1) attn_fused_fwd_kernel(const __grid_constant__ AttnFusedArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sP = sbase + AF_SP;
  const uint32_t bar_load = sbase + AF_BAR /* [2] */, bar_s = bar_load + 16, bar_p = bar_load + 24, bar_o = bar_load + 32;
  const uint32_t tmem_slot = bar_load + 40;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.q_map); tma_prefetch_desc(&a.k_map); tma_prefetch_desc(&a.v_map);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(bar_load, 1); mbar_init(bar_load + 8, 1); mbar_init(bar_s, 1); mbar_init(bar_p, 128); mbar_init(bar_o, 1);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const uint32_t tmem_S = tmem_base, tmem_O = tmem_base + 256;

  const int items = a.B * a.H * a.mtiles;
  const uint32_t load_bytes = 128 * 128 + 2 * a.Tk64 * 128;

  if (warp == 0) {
    if (lane == 0) {
      // operand stages are double-buffered: the loads of item i+1 go out as soon as PV of item i-1 has retired
      int it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int mt = item % a.mtiles, bh = item / a.mtiles, h = bh % a.H, b = bh / a.H;
        const int s = it & 1;
        const uint32_t sQ = sbase + s * AF_STAGE, sK = sQ + AF_SK, sV = sQ + AF_SV, bl = bar_load + 8 * s;
        if (it >= 2) mbar_wait(bar_o, (it - 2) & 1, 0x500u);    // PV of item it-2 (same stage) done
        mbar_arrive_expect_tx(bl, load_bytes);
        tma_load_4d(sQ, &a.q_map, bl, 0, mt * 128, h, b);
        tma_load_4d(sK, &a.k_map, bl, 0, 0, h, b);
        tma_load_4d(sV, &a.v_map, bl, 0, 0, h, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc_s = umma_idesc_f16(128, a.Tk16, false, false);
      const uint32_t idesc_o = umma_idesc_f16(128, 64, false, true);
      auto issue_s = [&](int it) {
        const int s = it & 1;
        const uint32_t sQ = sbase + s * AF_STAGE, sK = sQ + AF_SK;
        mbar_wait(bar_load + 8 * s, (it >> 1) & 1, 0x510u);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_f16(tmem_S, umma_smem_desc(sQ + k * 32, 16, 1024), umma_smem_desc(sK + k * 32, 16, 1024), idesc_s,
                    k > 0 ? 1u : 0u);
        umma_commit(bar_s);
      };
      int it = 0;
      if (blockIdx.x < items) issue_s(0);
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const uint32_t sV = sbase + (it & 1) * AF_STAGE + AF_SV;
        mbar_wait(bar_p, it & 1, 0x520u);           // P(it) in shared memory, S(it) fully read
        tc_fence_after();
        uint32_t acc = 0;
        for (int kb = 0; kb < a.Tk64 / 64; ++kb) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_f16(tmem_O, umma_smem_desc(sP + kb * 16384 + k * 32, 16, 1024),
                      umma_smem_desc(sV + kb * 8192 + k * 2048, 8192, 1024), idesc_o, acc);
            acc = 1;
          }
        }
        umma_commit(bar_o);
        if (item + static_cast<int>(gridDim.x) < items) issue_s(it + 1);   // scores of the next item during this epilogue
      }
    }
  } else if (warp >= 4) {
    const int w = warp - 4;
    const int r = w * 32 + lane;                                  // query row inside the tile == TMEM lane
    const uint32_t t_lane = static_cast<uint32_t>(w * 32) << 16;
    const float sc = 0.125f * 1.4426950408889634f;                // 1/sqrt(64) * log2(e)
    int it = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
      const uint32_t ph = it & 1;
      const int mt = item % a.mtiles, bh = item / a.mtiles, h = bh % a.H, b = bh / a.H;
      mbar_wait(bar_s, ph, 0x530u);        // also keeps idle warps in lock-step with the barrier phases
      if (mt * 128 + w * 32 >= a.T) {      // warp-uniform: all 32 query rows of this warp lie past T -> nothing to do
        mbar_arrive(bar_p);
        continue;
      }
      tc_fence_after();
      uint32_t sreg[32];
      // pass 1: row max over the valid keys
      float mx = -INFINITY;
      for (int c = 0; c * 32 < a.T; ++c) {
        tmem_ld_32x32(tmem_S + t_lane + c * 32, sreg);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c * 32 + i < a.T) mx = fmaxf(mx, __uint_as_float(sreg[i]));
      }
      // pass 2: unnormalised probabilities -> fp16 -> swizzled shared memory; row sum in fp32
      const float mxs = mx * sc;
      float sum = 0.f;
      for (int c = 0; c * 32 < a.Tk64; ++c) {
        tmem_ld_32x32(tmem_S + t_lane + c * 32, sreg);
        tmem_ld_wait();
        const int kb = c >> 1;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int key = c * 32 + g * 8 + 2 * j;
            const float e0 = key < a.T ? fast_exp2(__uint_as_float(sreg[g * 8 + 2 * j]) * sc - mxs) : 0.f;
            const float e1 = key + 1 < a.T ? fast_exp2(__uint_as_float(sreg[g * 8 + 2 * j + 1]) * sc - mxs) : 0.f;
            sum += e0 + e1;
            pk[j] = pack2(e0, e1);
          }
          const int chunk = (c & 1) * 4 + g;                      // 16-byte chunk inside the 128-byte row of k-block kb
          const uint32_t dst = sP + kb * 16384 + r * 128 + ((chunk ^ (r & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3])
                       : "memory");
        }
      }
      fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor core (async proxy)
      tc_fence_before();
      mbar_arrive(bar_p);
      // epilogue: O / sum
      mbar_wait(bar_o, ph, 0x540u);
      tc_fence_after();
      const float inv = 1.f / sum;
      const int q = mt * 128 + r;
      elem_t* dst = a.out + (static_cast<int64_t>(b) * a.T + q) * a.out_ld + h * 64;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        tmem_ld_32x32(tmem_O + t_lane + c * 32, sreg);
        tmem_ld_wait();
        if (q < a.T) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 v;
            v.x = pack2(__uint_as_float(sreg[g * 8 + 0]) * inv, __uint_as_float(sreg[g * 8 + 1]) * inv);
            v.y = pack2(__uint_as_float(sreg[g * 8 + 2]) * inv, __uint_as_float(sreg[g * 8 + 3]) * inv);
            v.z = pack2(__uint_as_float(sreg[g * 8 + 4]) * inv, __uint_as_float(sreg[g * 8 + 5]) * inv);
            v.w = pack2(__uint_as_float(sreg[g * 8 + 6]) * inv, __uint_as_float(sreg[g * 8 + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + c * 32 + g * 8) = v;
          }
        }
      }
      tc_fence_before();            // TMEM reads of this item ordered before the next item's MMAs (via bar_p)
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int attn_fused_fwd(const void* qkv, void* out, int64_t out_ld, int B, int H, int T, cudaStream_t st) {
  SPK_CHECK(T >= 1 && T <= AF_KV_ROWS && H >= 1, "attn_fused: T=%d outside [1, 256]", T);
  AttnFusedArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.T = T;
  a.Tk16 = (T + 15) / 16 * 16;
  a.Tk64 = (T + 63) / 64 * 64;
  a.mtiles = (T + 127) / 128;
  a.out = reinterpret_cast<elem_t*>(out);
  a.out_ld = out_ld;
  SPK_TRY(encode_qkv_map(&a.q_map, qkv, 0, B, H, T, 128));
  SPK_TRY(encode_qkv_map(&a.k_map, qkv, 1, B, H, T, a.Tk64));
  SPK_TRY(encode_qkv_map(&a.v_map, qkv, 2, B, H, T, a.Tk64));
  static PerDeviceOnce once;
  SPK_TRY(once.run([]() -> int {
    SPK_CUDA(cudaFuncSetAttribute(attn_fused_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AF_SMEM));
    return 0;
  }));
  const int items = B * H * a.mtiles;
  const int grid = items < device_sm_count() ? items : device_sm_count();
  ProfScope prof("attn_fused_fwd", 4.0 * B * H * T * T * 64, 4.0 * B * T * 64 * H * 2.0, st);
  attn_fused_fwd_kernel<<<grid, 256, AF_SMEM, st>>>(a);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace spk
