// Fused attention for the TRAINING path (multi-plane split-fp16 operands, dropout on the probabilities, a backward
// pass that recomputes instead of reading stored probabilities).  Replaces, per dense layer, the QK^T GEMM + softmax
// kernel + PV GEMM of the forward and the dV / dP GEMMs + softmax-backward kernel + dQ / dK GEMMs of the backward
// (8 launches over a materialised [B*H, T, T] score tensor in 2-3 planes) by two kernels whose scores never leave the
// SM.  Reference: torch scaled_dot_product_attention inside nn.TransformerEncoderLayer (Modules.py:25-36,53), scale
// 1/sqrt(64), dropout on the probabilities.
//
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 3 idle, 4.. = compute warps: warp 4 + 4p + w owns
// TMEM lane quarter w (tcgen05.ld/st restrict a warp to lanes 32 (warp % 4) ..) and takes every (CW / 4)-th 16-column
// chunk (p = 0 .. CW / 4 - 1).  The per-element work (exp2, Philox, plane splits) is what these kernels are bound by,
// so it is spread over as many warps as the register file allows: 16 compute warps at one CTA per SM (the backward and
// the one-CTA forward), 8 in the forwards that run two CTAs per SM.
//
// Forward (attn_fwd_kernel), per (slice, head) and 128-query tile:
//   TMA       Q tile, K, V (PL planes each) out of the packed qkv buffer [B*T, 768]
//   tcgen05   S = Q K^T into TMEM (6 plane products for PL = 3, 3 for PL = 2, 1 for PL = 1), fp32
//   CW warps  thread <-> query row (CW / 4 warps per TMEM lane quarter, alternating 16-key chunks): row max, exp2, row
//             sum, Philox keep mask, split into fp16 planes and written BACK INTO TMEM over the scores they came from
//             (tcgen05.st): the probabilities are the A operand of the next MMA straight from tensor memory
//   tcgen05   O = P_drop V  (A from TMEM, V read MN-major from shared memory)
//   CW warps  O * (1 / ((1 - p) * row sum)) -> PL fp16 planes -> att[(b*T + q) * 256 + h*64 ...]
//   kept for the backward: (row max * log2e / 8, row sum) per query and one keep BIT per probability.
// Inference (PL = 1) has no dropout and keeps nothing.
//
// TMEM plane layout of P for key step t (16 keys = one MMA K step = 8 columns of packed fp16 pairs, even key in the low
// half -- tools/probe/ts_probe.cu): plane 0 at S columns [16t, 16t+8), plane 1 at [16t+8, 16t+16), plane 2 (PL = 3)
// at P_LO + [8t, 8t+8); i.e. planes 0 and 1 overwrite exactly the 16 score columns they were computed from.
#include "gemm.h"
#include "ptx.cuh"

namespace spk {

__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]: A is [128 lanes x K] packed fp16 pairs in tensor memory (K-major by construction)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// One lane of a CONVERGED warp (the MMA warp runs its loops with all 32 lanes and elects the issuer here: tcgen05.mma
// takes its operands from uniform registers, and issued from divergent `if (lane == 0)` code every MMA costs an
// election loop and register moves -- ~60 cycles each, more than a 128 x 64 x 16 MMA takes to execute).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// descriptor of the same tile `bytes` further on (the start-address field holds address >> 4 in its low 14 bits)
__device__ __forceinline__ uint64_t desc_add(uint64_t d, uint32_t bytes) { return d + (bytes >> 4); }
template <int NW = 4>
__device__ __forceinline__ void quarter_sync(int quarter) {   // the NW warps that share a TMEM lane quarter
  asm volatile("bar.sync %0, %1;" ::"r"(quarter + 1), "n"(32 * NW) : "memory");
}
// keep bits (bit i <-> element idx8 * 8 + i) of one Philox call; same function of (seed, site, element) as dropout_scale8
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t seed, uint32_t site, uint64_t idx8, uint32_t thresh) {
  const Philox4 r = philox4x32_7(static_cast<uint32_t>(idx8), static_cast<uint32_t>(idx8 >> 32), site, 0x5eedu,
                                 static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  uint32_t bits = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    bits |= ((w[i] & 0xFFFFu) >= thresh ? 1u : 0u) << (2 * i);
    bits |= ((w[i] >> 16) >= thresh ? 1u : 0u) << (2 * i + 1);
  }
  return bits;
}

constexpr int ATF_MAX_T = 192;                           // frames of every fused training / two-CTA inference forward
constexpr float ATF_SC = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e)

// Footprint of one forward instantiation: PL fp16 planes, CW compute warps (16: one CTA per SM, 512 TMEM columns with
// plane 2 of P at P_LO; 8: two CTAs per SM, 256 columns) and the load schedule.  KV_SHARED: ONE operand buffer holds K
// for the score MMAs and is then reloaded with V for the PV MMAs (K and V are needed at different times); otherwise K
// and V are loaded once per item into buffers of their own.
template <int PL, int CW, bool KV_SHARED>
struct AttnFwdLayout {
  static constexpr int THREADS = 128 + 32 * CW;
  static constexpr int NP = CW / 4;                           // compute warps per TMEM lane quarter = column parts
  static constexpr int Q_BYTES = 128 * 128, KV_BYTES = ATF_MAX_T * 128;
  static constexpr int OFF_K = PL * Q_BYTES, OFF_V = KV_SHARED ? OFF_K : OFF_K + PL * KV_BYTES;
  static constexpr int OFF_X = OFF_V + PL * KV_BYTES;         // float max parts [NP][128], sum parts [NP][128]
  static constexpr int OFF_STG = OFF_X + 2 * NP * 128 * 4;    // output staging: one plane, 128 rows x 128 B
  static constexpr int OFF_BAR = OFF_STG + 16384;
  static constexpr int SMEM = OFF_BAR + 128;
  static constexpr int TMEM_COLS = CW == 16 ? 512 : 256, TMEM_O = CW == 16 ? 384 : 192, TMEM_PLO = 256;
  // watchdog codes: producer WD + 0 / 1, MMA issuer WD + 0x10 .. 0x13, compute warps WD + 0x20 / 0x21
  static constexpr uint32_t WD = PL == 1 ? 0x640u : KV_SHARED ? 0x670u : 0x600u;
  static_assert(CW == 16 || 2 * (SMEM + 1024) <= 228 * 1024, "two CTAs of an 8-warp instantiation must share an SM");
};

struct AttnFwdArgs {
  CUtensorMap q_map[3], k_map[3], v_map[3];
  int B, H, T, Tp, Tk16, Tk64, mtiles, nC;
  elem_t* out;      // [PL][B*T, out_ld], head h at column h*64
  int64_t out_ps, out_ld;
  float2* stats;           // [B*H*T] (row max * ATF_SC, row sum of exp2), may be null
  uint16_t* mbits;         // [B*H][nC][T] keep bits of 16-key chunk c of query q, null without dropout
  DropCfg drop;
  uint32_t site;
};

// Instantiations: <1, 8, false> inference; <2, 8, true> two-CTA training; <2, 16, false> and <3, 16, false> one-CTA
// training.  The dropout keep mask, `stats` and `mbits` exist only for PL >= 2.
template <int PL, int CW, bool KV_SHARED>
__global__ void __launch_bounds__(128 + 32 * CW, CW == 8 ? 2 : 1) attn_fwd_kernel(const __grid_constant__ AttnFwdArgs a) {
  using L = AttnFwdLayout<PL, CW, KV_SHARED>;
  constexpr int NP = L::NP;
  constexpr uint32_t WD = L::WD;
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sbase = smem_u32(smem_raw);
  const uint32_t sQ = sbase, sK = sbase + L::OFF_K, sV = sbase + L::OFF_V;
  float* xch = reinterpret_cast<float*>(smem_raw + L::OFF_X);   // [0, 128 NP) max parts, [128 NP, 256 NP) sum parts
  // The first two barriers complete with the operands.  Separate buffers: bar_kv with K and V of an item, bar_q with Q
  // of a query tile.  Shared buffer: bar_qk with Q and K of a query tile, bar_v with its V.
  const uint32_t bar_kv = sbase + L::OFF_BAR, bar_q = bar_kv + 8, bar_qk = bar_kv, bar_v = bar_q;
  const uint32_t bar_s = bar_kv + 16, bar_p = bar_kv + 24, bar_o = bar_kv + 32, bar_oe = bar_kv + 40,
                 bar_kvfree = bar_kv + 48, tmem_slot = bar_kv + 56;
  // Every waiter of an mbarrier observes EVERY phase of it, in order (a parity wait that skips a phase passes
  // spuriously): per-unit barriers are waited on once per unit, per-item barriers once per item.
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((sbase & 1023u) != 0) __trap();     // the swizzled operand tiles need a 1024-byte aligned base

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int p = 0; p < PL; ++p) { tma_prefetch_desc(&a.q_map[p]); tma_prefetch_desc(&a.k_map[p]); tma_prefetch_desc(&a.v_map[p]); }
  }
  if (warp == 1 && lane == 0) {
    mbar_init(bar_kv, 1); mbar_init(bar_q, 1); mbar_init(bar_s, 1); mbar_init(bar_p, 32 * CW); mbar_init(bar_o, 1);
    mbar_init(bar_oe, 32 * CW);
    if constexpr (!KV_SHARED) mbar_init(bar_kvfree, 1);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, L::TMEM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const uint32_t tS = tmem_base, tPlo = tmem_base + L::TMEM_PLO, tO = tmem_base + L::TMEM_O;
  const int items = a.B * a.H;
  const int kv_plane = a.Tk64 * 128;      // bytes actually loaded per K / V plane

  if (warp == 0) {
    if (lane == 0) {
      uint32_t u = 0, it = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
        const int h = item % a.H, b = item / a.H;
        if constexpr (!KV_SHARED) {
          if (it > 0) mbar_wait(bar_kvfree, (it - 1) & 1u, WD);   // last PV of the previous item: K / V are free
          mbar_arrive_expect_tx(bar_kv, 2u * PL * kv_plane);
#pragma unroll
          for (int p = 0; p < PL; ++p) {
            tma_load_4d(sK + p * L::KV_BYTES, &a.k_map[p], bar_kv, 0, 0, h, b);
            tma_load_4d(sV + p * L::KV_BYTES, &a.v_map[p], bar_kv, 0, 0, h, b);
          }
        }
        for (int mt = 0; mt < a.mtiles; ++mt, ++u) {
          if constexpr (KV_SHARED) {
            if (u > 0) mbar_wait(bar_o, (u - 1) & 1u, WD);        // previous PV retired: the operand buffer (V) and Q are free
            mbar_arrive_expect_tx(bar_qk, PL * (L::Q_BYTES + kv_plane));
#pragma unroll
            for (int p = 0; p < PL; ++p) {
              tma_load_4d(sQ + p * L::Q_BYTES, &a.q_map[p], bar_qk, 0, mt * 128, h, b);
              tma_load_4d(sK + p * L::KV_BYTES, &a.k_map[p], bar_qk, 0, 0, h, b);
            }
            mbar_wait(bar_s, u & 1u, WD + 1);                     // score MMAs retired: K is dead, V takes its place
            mbar_arrive_expect_tx(bar_v, PL * kv_plane);
#pragma unroll
            for (int p = 0; p < PL; ++p) tma_load_4d(sV + p * L::KV_BYTES, &a.v_map[p], bar_v, 0, 0, h, b);
          } else {
            if (u > 0) mbar_wait(bar_s, (u - 1) & 1u, WD + 1);    // previous scores issued and retired: Q is free
            mbar_arrive_expect_tx(bar_q, PL * L::Q_BYTES);
#pragma unroll
            for (int p = 0; p < PL; ++p) tma_load_4d(sQ + p * L::Q_BYTES, &a.q_map[p], bar_q, 0, mt * 128, h, b);
          }
        }
      }
    }
  } else if (warp == 1) {
    // whole warp, converged; one elected lane issues
    const uint32_t idesc_s = umma_idesc_f16(128, a.Tk16, false, false);
    const uint32_t idesc_o = umma_idesc_f16(128, 64, false, true);
    // plane products (A plane, B plane), smallest terms first (plane 0 = hi)
    constexpr int NCOMBO = PL == 3 ? 6 : PL == 2 ? 3 : 1;
    constexpr int PA[3][6] = {{0}, {1, 0, 0}, {1, 0, 2, 0, 1, 0}}, PB[3][6] = {{0}, {0, 1, 0}, {1, 2, 0, 1, 0, 0}};
    const uint64_t dQ0 = umma_smem_desc(sQ, 16, 1024), dK0 = umma_smem_desc(sK, 16, 1024);
    const uint64_t dV0 = umma_smem_desc(sV, 8192, 1024);
    const int ksteps = a.Tk16 / 16;
    uint32_t u = 0, it = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
      for (int mt = 0; mt < a.mtiles; ++mt, ++u) {
        if constexpr (KV_SHARED) {
          mbar_wait(bar_qk, u & 1u, WD + 0x10);
        } else {
          mbar_wait(bar_q, u & 1u, WD + 0x10);
          if (mt == 0) mbar_wait(bar_kv, it & 1u, WD + 0x11);
        }
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int cb = 0; cb < NCOMBO; ++cb) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16(tS, desc_add(dQ0, PA[PL - 1][cb] * L::Q_BYTES + k * 32), desc_add(dK0, PB[PL - 1][cb] * L::KV_BYTES + k * 32),
                       idesc_s, (cb | k) ? 1u : 0u);
          }
          umma_commit(bar_s);
        }
        __syncwarp();
        mbar_wait(bar_p, u & 1u, WD + 0x12);                      // probabilities are in TMEM
        if constexpr (KV_SHARED) mbar_wait(bar_v, u & 1u, WD + 0x11);   // V is in the operand buffer
        if (u > 0) mbar_wait(bar_oe, (u - 1) & 1u, WD + 0x13);    // previous output tile drained
        tc_fence_after();
        if (elect_one()) {
          for (int t = 0; t < ksteps; ++t) {
            const uint32_t voff = (t >> 2) * 8192 + (t & 3) * 2048;
#pragma unroll
            for (int cb = 0; cb < NCOMBO; ++cb) {
              const int pa = PA[PL - 1][cb];
              const uint32_t ta = pa == 0 ? tS + 16 * t : (pa == 1 ? tS + 16 * t + 8 : tPlo + 8 * t);
              umma_f16_ts(tO, ta, desc_add(dV0, PB[PL - 1][cb] * L::KV_BYTES + voff), idesc_o, (t | cb) ? 1u : 0u);
            }
          }
          umma_commit(bar_o);
          if constexpr (!KV_SHARED) {
            if (mt == a.mtiles - 1) umma_commit(bar_kvfree);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    const int w = (warp - 4) & 3, part = (warp - 4) >> 2;          // lane quarter, column part (0 .. NP - 1)
    const int r = w * 32 + lane;
    const uint32_t t_lane = static_cast<uint32_t>(w * 32) << 16;
    const bool use_drop = PL >= 2 && a.drop.thresh != 0;           // no dropout in inference
    const float inv_keep = use_drop ? a.drop.inv_keep : 1.f;
    const int nchunks = a.Tk16 / 16;                               // 16-key chunks == MMA key steps
    uint32_t u = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int h = item % a.H, b = item / a.H;
      for (int mt = 0; mt < a.mtiles; ++mt, ++u) {
        const uint32_t ph = u & 1u;
        const int q = mt * 128 + r;
        const bool active = mt * 128 + w * 32 < a.T;              // warp-uniform
        mbar_wait(bar_s, ph, WD + 0x20);
        tc_fence_after();
        uint32_t sreg[16];
        float mx = -INFINITY;
        if (active) {
          for (int c = part; c * 16 < a.T; c += NP) {
            tmem_ld_32x16(tS + t_lane + c * 16, sreg);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c * 16 + i < a.T) mx = fmaxf(mx, __uint_as_float(sreg[i]));
          }
        }
        xch[part * 128 + r] = mx;
        quarter_sync<NP>(w);
        // the parts are combined in a fixed tree, so every row's max and sum are the same whatever the warp count
        if constexpr (NP == 4) mx = fmaxf(fmaxf(xch[r], xch[128 + r]), fmaxf(xch[256 + r], xch[384 + r]));
        else mx = fmaxf(xch[r], xch[128 + r]);
        const float mxs = mx * ATF_SC;
        float sum = 0.f;
        if (active) {
          const uint64_t row_idx8 = ((static_cast<uint64_t>(item) * a.T + q) * a.Tp) >> 3;   // Tp % 8 == 0
          for (int c = part; c < nchunks; c += NP) {
            tmem_ld_32x16(tS + t_lane + c * 16, sreg);
            uint32_t keep = 0xFFFFu;
            if (use_drop)
              keep = dropout_keep8(a.drop.seed, a.site, row_idx8 + 2 * c, a.drop.thresh) |
                     (dropout_keep8(a.drop.seed, a.site, row_idx8 + 2 * c + 1, a.drop.thresh) << 8);
            tmem_ld_wait();
            uint32_t o01[PL == 1 ? 8 : 16];                               // planes 0 and 1 of P
            uint32_t o2[8];                                               // plane 2 (PL = 3)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int key = c * 16 + 2 * j;
              float e0 = key < a.T ? fast_exp2(__uint_as_float(sreg[2 * j]) * ATF_SC - mxs) : 0.f;
              float e1 = key + 1 < a.T ? fast_exp2(__uint_as_float(sreg[2 * j + 1]) * ATF_SC - mxs) : 0.f;
              sum += e0 + e1;
              e0 = ((keep >> (2 * j)) & 1u) ? e0 : 0.f;
              e1 = ((keep >> (2 * j + 1)) & 1u) ? e1 : 0.f;
              const uint32_t hi = pack2(e0, e1);
              o01[j] = hi;                                                // plane 0 at columns 16c + j
              if constexpr (PL >= 2) {
                e0 -= lo_to_f(hi);
                e1 -= hi_to_f(hi);
                const uint32_t mid = pack2(e0, e1);
                o01[8 + j] = mid;                                         // plane 1 at columns 16c + 8 + j
                if constexpr (PL == 3) {
                  e0 -= lo_to_f(mid);
                  e1 -= hi_to_f(mid);
                  o2[j] = pack2(e0, e1);                                  // plane 2 at P_LO + 8c + j
                }
              }
            }
            if constexpr (PL == 1) {
              tmem_st_32x8(tS + t_lane + c * 16, o01);
            } else {
              tmem_st_32x16(tS + t_lane + c * 16, o01);
              if constexpr (PL == 3) tmem_st_32x8(tPlo + t_lane + c * 8, o2);
              if (a.mbits != nullptr && q < a.T)
                a.mbits[(static_cast<int64_t>(item) * a.nC + c) * a.T + q] = static_cast<uint16_t>(keep);
            }
          }
          tmem_st_wait();
        }
        xch[NP * 128 + part * 128 + r] = sum;
        tc_fence_before();
        mbar_arrive(bar_p);
        quarter_sync<NP>(w);
        if constexpr (NP == 4) sum = (xch[512 + r] + xch[640 + r]) + (xch[768 + r] + xch[896 + r]);
        else sum = xch[256 + r] + xch[384 + r];
        // ---- epilogue: O * inv_keep / sum -> PL planes.  This warp takes COLS of the head's 64 columns out of TMEM; the
        //      planes go through a shared-memory tile so that global memory sees full 128-byte rows (8 lanes x 16 B)
        mbar_wait(bar_o, ph, WD + 0x21);
        tc_fence_after();
        constexpr int COLS = 64 / NP;
        float v[COLS];
        if (active) {
#pragma unroll
          for (int hlf = 0; hlf < COLS / 16; ++hlf) {
            tmem_ld_32x16(tO + t_lane + part * COLS + hlf * 16, sreg);
            tmem_ld_wait();
            const float sc = inv_keep / sum;                      // placed after a load, the division overlaps it
#pragma unroll
            for (int i = 0; i < 16; ++i) v[hlf * 16 + i] = __uint_as_float(sreg[i]) * sc;
          }
          if constexpr (PL >= 2) {
            if (part == 0 && q < a.T && a.stats != nullptr) a.stats[static_cast<int64_t>(item) * a.T + q] = make_float2(mxs, sum);
          }
        }
        tc_fence_before();
        mbar_arrive(bar_oe);                                      // the accumulator is free for the next tile's PV
        if (active) {                                             // uniform over the quarter's NP warps
          const uint32_t stg = sbase + L::OFF_STG;
#pragma unroll
          for (int p = 0; p < PL; ++p) {
#pragma unroll
            for (int g = 0; g < COLS / 8; ++g) {                  // this warp's 16-byte chunks (COLS / 8) part + g
              uint32_t wv[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                wv[i] = pack2(v[g * 8 + 2 * i], v[g * 8 + 2 * i + 1]);
                if (p + 1 < PL) {
                  v[g * 8 + 2 * i] -= lo_to_f(wv[i]);
                  v[g * 8 + 2 * i + 1] -= hi_to_f(wv[i]);
                }
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + r * 128 + ((((COLS / 8) * part + g) ^ (r & 7)) << 4)),
                           "r"(wv[0]), "r"(wv[1]), "r"(wv[2]), "r"(wv[3]) : "memory");
            }
            quarter_sync<NP>(w);
#pragma unroll
            for (int it = 0; it < 8 / NP; ++it) {                 // 32 / NP of the quarter's 32 rows per warp, 4 rows per instruction
              const int row = w * 32 + part * (32 / NP) + it * 4 + (lane >> 3);
              uint4 val;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(val.x), "=r"(val.y), "=r"(val.z), "=r"(val.w)
                           : "r"(stg + row * 128 + (((lane & 7) ^ (row & 7)) << 4)) : "memory");
              const int qq = mt * 128 + row;
              if (qq < a.T)
                *reinterpret_cast<uint4*>(a.out + p * a.out_ps + (static_cast<int64_t>(b) * a.T + qq) * a.out_ld + h * 64 +
                                          (lane & 7) * 8) = val;
            }
            quarter_sync<NP>(w);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, L::TMEM_COLS);
  }
}

static int g_attn_fwd_two = 1;     // spk_set_option("training_attention_two_ctas", 0/1)
void attn_train_set_fwd_two(int on) { g_attn_fwd_two = on; }

// Fills the map and tile fields of `a` (B, H, T, Tp and the outputs are set) and launches one instantiation.
template <int PL, int CW, bool KV_SHARED>
static int attn_fwd_launch(AttnFwdArgs& a, const void* qkv, int64_t qkv_ps, const char* tag, cudaStream_t st) {
  using L = AttnFwdLayout<PL, CW, KV_SHARED>;
  a.Tk16 = (a.T + 15) / 16 * 16;
  a.Tk64 = (a.T + 63) / 64 * 64;
  a.mtiles = (a.T + 127) / 128;
  a.nC = (a.Tp + 15) / 16;
  for (int p = 0; p < PL; ++p) {
    const elem_t* plane = reinterpret_cast<const elem_t*>(qkv) + p * qkv_ps;
    SPK_TRY(encode_qkv_map(&a.q_map[p], plane, 0, a.B, a.H, a.T, 128));
    SPK_TRY(encode_qkv_map(&a.k_map[p], plane, 1, a.B, a.H, a.T, a.Tk64));
    SPK_TRY(encode_qkv_map(&a.v_map[p], plane, 2, a.B, a.H, a.T, a.Tk64));
  }
  static PerDeviceOnce once;
  SPK_TRY(once.run([]() -> int {
    SPK_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<PL, CW, KV_SHARED>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::SMEM));
    return 0;
  }));
  const int items = a.B * a.H, ctas = (CW == 8 ? 2 : 1) * device_sm_count();
  const int grid = items < ctas ? items : ctas;
  // algorithmic work: QK^T and PV (16-bit dense count); bytes: Q, K, V in, O out
  ProfScope prof(tag, 4.0 * a.B * a.H * a.T * a.T * 64, 4.0 * a.B * a.T * 64 * a.H * 2.0 * PL, st);
  attn_fwd_kernel<PL, CW, KV_SHARED><<<grid, L::THREADS, L::SMEM, st>>>(a);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

// qkv: [planes][B*T, 768] split tensor; out: [planes][B*T, 256]; stats [B*H*T] float2; mbits [B*H][ceil(Tp/16)][T] u16
int attn_train_fwd(const void* qkv, int64_t qkv_ps, int planes, void* out, int64_t out_ps, int64_t out_ld, float* stats,
                   uint32_t* mbits, DropCfg drop, uint32_t site, int B, int H, int T, int Tp, cudaStream_t st) {
  SPK_CHECK(planes == 2 || planes == 3, "attn_train_fwd: planes must be 2 or 3");
  SPK_CHECK(T >= 1 && T <= ATF_MAX_T && H >= 1, "attn_train_fwd: T=%d outside [1, %d]", T, ATF_MAX_T);
  SPK_CHECK(drop.thresh == 0 || mbits != nullptr, "attn_train_fwd: dropout needs the keep-bit buffer");
  AttnFwdArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.T = T; a.Tp = Tp;
  a.out = reinterpret_cast<elem_t*>(out);
  a.out_ps = out_ps; a.out_ld = out_ld;
  a.stats = reinterpret_cast<float2*>(stats);
  a.mbits = drop.thresh != 0 ? reinterpret_cast<uint16_t*>(mbits) : nullptr;
  a.drop = drop; a.site = site;
  if (planes == 3) return attn_fwd_launch<3, 16, false>(a, qkv, qkv_ps, "attn_train_fwd", st);
  if (g_attn_fwd_two) return attn_fwd_launch<2, 8, true>(a, qkv, qkv_ps, "attn_train_fwd", st);
  return attn_fwd_launch<2, 16, false>(a, qkv, qkv_ps, "attn_train_fwd", st);
}

// qkv: [B*T, 768] one plane; out: [B*T, out_ld] one plane (head h at column h*64).  T <= 192.
int attn_infer_fwd(const void* qkv, void* out, int64_t out_ld, int B, int H, int T, cudaStream_t st) {
  SPK_CHECK(T >= 1 && T <= ATF_MAX_T && H >= 1, "attn_infer_fwd: T=%d outside [1, %d]", T, ATF_MAX_T);
  AttnFwdArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.T = T;
  a.out = reinterpret_cast<elem_t*>(out);
  a.out_ld = out_ld;
  return attn_fwd_launch<1, 8, false>(a, qkv, 0, "attn_fused_fwd", st);
}

// =====================================================================================================================
// Backward.  Two fp16 planes everywhere (gradients are smooth in their inputs, DESIGN.md "precision").  Per (slice,
// head) the keys are walked in tiles i, the queries in tiles j of `rpt` rows each (rpt = the frames split evenly over
// ceil(T / 128) tiles, rounded up to 16: 160 frames -> 2 x 80, so that every (i, j) unit is the same size and keeps
// three of the four lane quarters busy); everything is computed TRANSPOSED (keys on the TMEM lanes) so that the two
// products contracted over queries take their A operand straight from tensor memory:
//
//   tcgen05   S^T  = K_i Q_j^T ,  dP^T = V_i dO_j^T                    -> TMEM (fp32)
//   16 warps  thread <-> key row: P^T = exp2(S^T * c - m_q) / l_q (row statistics saved by the forward), keep bit from
//             the forward's bit mask (32 x 32 bit transpose by warp shuffles), dS^T = P^T (keep dP^T/(1-p) - delta_q) / 8;
//             P_drop^T and dS^T go back into TMEM over S^T / dP^T as fp16 planes; dS^T also into shared memory in the
//             MN-major operand layout (probe: tools/probe/ts_probe.cu)
//   tcgen05   dV_i += P_drop^T dO_j  and  dK_i += dS^T Q_j   (A from TMEM, B MN-major from shared memory)
//             dQ_j += dS K_i                                  (A = dS from shared memory, MN-major)
//   16 warps  drain dV_i, dK_i after the last j, dQ_j after the last i -> dqkv planes; their column sums (the in-proj
//             bias gradient) stay in registers for the whole kernel (a CTA only ever sees one head) and are added to
//             global memory once per warp at the end.
// delta_q = sum_d dO_qd O_qd comes from attn_delta_kernel.  T <= 192: Q and dO of the whole slice stay resident.
// Optional phase timeline of CTA 0 (diagnostics: spk_set_debug_buffer): slot [unit * 8 + event] = clock64 at
//   0 operands of the unit are in shared memory   1 S^T / dP^T MMAs issued   2 P^T / dS^T written (bar_p seen by the MMA thread)
//   3 accumulating MMAs issued                     4 scores visible to a compute warp   5 that warp finished its chunks
static unsigned long long* g_attn_timeline = nullptr;
static size_t g_attn_timeline_slots = 0;
void attn_train_set_timeline(void* buf, size_t bytes) {
  g_attn_timeline = reinterpret_cast<unsigned long long*>(buf);
  g_attn_timeline_slots = bytes / 8;
}
#define ATB_STAMP(unit, ev)                                                                   \
  do {                                                                                        \
    if (a.timeline != nullptr && blockIdx.x == 0 && (threadIdx.x & 31) == 0 &&                \
        static_cast<size_t>((unit) * 8 + (ev)) < a.timeline_slots)                            \
      a.timeline[(unit) * 8 + (ev)] = clock64();                                              \
  } while (0)

constexpr int ATB_THREADS = 640;
constexpr int ATB_CW = 16;
constexpr int ATB_MAXT = 192;
constexpr int ATB_QROWS = ATB_MAXT * 128;                 // bytes per plane of Q / dO
constexpr int ATB_OFF_DO = 2 * ATB_QROWS;                 // 49152
constexpr int ATB_OFF_K = 4 * ATB_QROWS;                  // 98304
constexpr int ATB_OFF_V = ATB_OFF_K + 32768;              // 131072
constexpr int ATB_OFF_DS = ATB_OFF_V + 32768;             // 163840
constexpr int ATB_STATS = 224;                            // >= rpt + 128 (the last query tile's 16-query chunks may run past T)
constexpr int ATB_OFF_STAT = ATB_OFF_DS + 65536;          // 229376: float2 (m + log2 l, delta) [224]
constexpr int ATB_OFF_BAR = ATB_OFF_STAT + ATB_STATS * 8; // 231168
constexpr int ATB_SMEM = ATB_OFF_BAR + 128;               // 231296 <= 232448
constexpr int ATB_T_ST = 0, ATB_T_DP = 128, ATB_T_DV = 256, ATB_T_DK = 320, ATB_T_DQ = 384;

struct AttnTrainBwdArgs {
  CUtensorMap q_map[2], k_map[2], v_map[2], do_map[2];
  int B, H, T, Tk64, tiles, rpt, nC;
  const float2* stats;      // [B*H*T] from the forward
  const float* delta;       // [B*H*T]
  const uint16_t* mbits;    // [B*H][nC][T] or null (no dropout)
  elem_t* dqkv;      // [2][B*T, 768]
  int64_t dqkv_ps;
  float* dbias;             // [768] += column sums of dQ | dK | dV, times *(gscale + 1); null: not wanted
  const float* gscale;      // device (S, 1 / S): the gradients arrive scaled by S (may be null)
  float inv_keep;
  unsigned long long* timeline;
  size_t timeline_slots;
};

// lane r holds row r of a 32 x 32 bit matrix (bit c = column c); afterwards lane c holds column c (bit r = row r)
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const uint32_t m = s == 16 ? 0x0000FFFFu : s == 8 ? 0x00FF00FFu : s == 4 ? 0x0F0F0F0Fu : s == 2 ? 0x33333333u : 0x55555555u;
    const uint32_t o = __shfl_xor_sync(0xffffffffu, x, s);
    x = (lane & s) ? (((o >> s) & m) | (x & ~m)) : ((x & m) | ((o & m) << s));
  }
  return x;
}
// v[x] of lane r = element (r, x), 16 columns; returns (in every lane c and c + 16) the sum over all 32 lanes of column c & 15
__device__ __forceinline__ float column_sums16(float (&v)[16], int lane) {
#pragma unroll
  for (int s = 8; s >= 1; s >>= 1) {
#pragma unroll
    for (int k = 0; k < s; ++k) {
      const float send = (lane & s) ? v[k] : v[k + s];
      const float recv = __shfl_xor_sync(0xffffffffu, send, s);
      v[k] = ((lane & s) ? v[k + s] : v[k]) + recv;
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}
// 16 fp32 values -> two fp16 planes at dst / dst + ps (16-byte stores)
__device__ __forceinline__ void store16_two_planes(elem_t* dst, int64_t ps, const float (&v)[16]) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x0 = v[g * 8 + 2 * e], x1 = v[g * 8 + 2 * e + 1];
      hi[e] = pack2(x0, x1);
      lo[e] = pack2(x0 - lo_to_f(hi[e]), x1 - hi_to_f(hi[e]));
    }
    *reinterpret_cast<uint4*>(dst + g * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(dst + ps + g * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// 16 fp32 values -> two fp16 planes, 2 x 16 bytes each, into shared-memory staging chunks
__device__ __forceinline__ void stage16_two_planes(uint32_t hi0, uint32_t hi1, uint32_t lo0, uint32_t lo1, const float (&v)[16]) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float x0 = v[g * 8 + 2 * e], x1 = v[g * 8 + 2 * e + 1];
      hi[e] = pack2(x0, x1);
      lo[e] = pack2(x0 - lo_to_f(hi[e]), x1 - hi_to_f(hi[e]));
    }
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(g ? hi1 : hi0), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]) : "memory");
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(g ? lo1 : lo0), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3]) : "memory");
  }
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 w;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w) : "r"(addr) : "memory");
  return w;
}

__global__ void __launch_bounds__(ATB_THREADS, 1) attn_train_bwd_kernel(const __grid_constant__ AttnTrainBwdArgs a) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t sbase = smem_u32(smem_raw);
  const uint32_t sQ = sbase, sdO = sbase + ATB_OFF_DO, sK = sbase + ATB_OFF_K, sV = sbase + ATB_OFF_V, sdS = sbase + ATB_OFF_DS;
  float2* sStat = reinterpret_cast<float2*>(smem_raw + ATB_OFF_STAT);
  const uint32_t bar_qdo = sbase + ATB_OFF_BAR, bar_kv = bar_qdo + 8, bar_m1 = bar_qdo + 16, bar_p = bar_qdo + 24,
                 bar_tile = bar_qdo + 32, bar_kvd = bar_qdo + 40, bar_dqd = bar_qdo + 48, tmem_slot = bar_qdo + 56;
  // Every waiter of an mbarrier observes EVERY phase of it, in order: bar_m1 / bar_p advance once per (i, j) unit,
  // bar_kv / bar_tile / bar_kvd once per key tile, bar_qdo / bar_dqd once per slice.
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((sbase & 1023u) != 0) __trap();

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      tma_prefetch_desc(&a.q_map[p]); tma_prefetch_desc(&a.k_map[p]); tma_prefetch_desc(&a.v_map[p]); tma_prefetch_desc(&a.do_map[p]);
    }
  }
  if (warp == 1 && lane == 0) {
    mbar_init(bar_qdo, 1); mbar_init(bar_kv, 1); mbar_init(bar_m1, 1); mbar_init(bar_p, 32 * ATB_CW); mbar_init(bar_tile, 1);
    mbar_init(bar_kvd, 32 * ATB_CW); mbar_init(bar_dqd, 32 * ATB_CW);
    fence_mbar_init();
  }
  if (warp == 2) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const int items = a.B * a.H;
  const int tiles = a.tiles, rpt = a.rpt;                 // key tiles == query tiles, rpt rows each (rpt % 16 == 0)
  // rows of tile t that hold frames, and the same rounded up to the MMA's 16-row steps
  auto rows_of = [&](int t) { const int n = a.T - rpt * t; return n < rpt ? n : rpt; };
  auto rows16_of = [&](int t) { return (rows_of(t) + 15) & ~15; };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t kt = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int h = item % a.H, b = item / a.H;
        for (int i = 0; i < tiles; ++i, ++kt) {
          if (kt > 0) mbar_wait(bar_tile, (kt - 1) & 1u, 0x700u);   // every MMA that read the buffers loaded next has retired
          if (i == 0) {
            mbar_arrive_expect_tx(bar_qdo, 4u * a.Tk64 * 128);
#pragma unroll
            for (int p = 0; p < 2; ++p) {
              tma_load_4d(sQ + p * ATB_QROWS, &a.q_map[p], bar_qdo, 0, 0, h, b);
              tma_load_4d(sdO + p * ATB_QROWS, &a.do_map[p], bar_qdo, 0, 0, h, b);
            }
          }
          mbar_arrive_expect_tx(bar_kv, 4u * 16384);
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            tma_load_4d(sK + p * 16384, &a.k_map[p], bar_kv, 0, i * rpt, h, b);
            tma_load_4d(sV + p * 16384, &a.v_map[p], bar_kv, 0, i * rpt, h, b);
          }
        }
      }
    }
  } else if (warp == 1) {
    // whole warp, converged; one elected lane issues (see elect_one)
    constexpr int PA[3] = {1, 0, 0}, PB[3] = {0, 1, 0};          // lo*hi, hi*lo, hi*hi
    const uint32_t tST = tmem_base + ATB_T_ST, tDP = tmem_base + ATB_T_DP, tdV = tmem_base + ATB_T_DV,
                   tdK = tmem_base + ATB_T_DK;
    const uint32_t idesc_acc = umma_idesc_f16(128, 64, false, true);      // A from TMEM, B MN-major
    const uint32_t idesc_dq = umma_idesc_f16(128, 64, true, true);        // A and B MN-major from shared memory
    const uint64_t dKk = umma_smem_desc(sK, 16, 1024), dVk = umma_smem_desc(sV, 16, 1024);          // K-major A
    const uint64_t dQk = umma_smem_desc(sQ, 16, 1024), dOk = umma_smem_desc(sdO, 16, 1024);         // K-major B
    const uint64_t dQm = umma_smem_desc(sQ, 8192, 1024), dOm = umma_smem_desc(sdO, 8192, 1024);     // MN-major B
    const uint64_t dKm = umma_smem_desc(sK, 8192, 1024), dSm = umma_smem_desc(sdS, 8192, 1024);     // MN-major B / A
    uint32_t u = 0, kt = 0, it = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x, ++it) {
      mbar_wait(bar_qdo, it & 1u, 0x710u);
      for (int i = 0; i < tiles; ++i, ++kt) {
        mbar_wait(bar_kv, kt & 1u, 0x711u);
        const int nk = rows16_of(i) / 16;                        // key steps of this tile that hold frames
        for (int j = 0; j < tiles; ++j, ++u) {
          const int nq = rows16_of(j);
          const uint32_t qoff = static_cast<uint32_t>(j * rpt) * 128u;      // byte offset of query tile j (1024-aligned)
          const uint32_t idesc_s = umma_idesc_f16(128, nq, false, false);
          tc_fence_after();
          ATB_STAMP(u, 0);
          // ---- S^T = K_i Q_j^T, dP^T = V_i dO_j^T
          if (elect_one()) {
#pragma unroll
            for (int which = 0; which < 2; ++which) {
              const uint64_t da = which ? dVk : dKk, db = desc_add(which ? dOk : dQk, qoff);
              const uint32_t td = which ? tDP : tST;
#pragma unroll
              for (int cb = 0; cb < 3; ++cb) {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_f16(td, desc_add(da, PA[cb] * 16384 + k * 32), desc_add(db, PB[cb] * ATB_QROWS + k * 32), idesc_s,
                            (cb | k) ? 1u : 0u);
              }
            }
            umma_commit(bar_m1);
          }
          __syncwarp();
          ATB_STAMP(u, 1);
          mbar_wait(bar_p, u & 1u, 0x712u);
          ATB_STAMP(u, 2);
          if (j == 0 && kt > 0) mbar_wait(bar_kvd, (kt - 1) & 1u, 0x713u);            // dV / dK of the previous key tile drained
          if (i == 0 && j == 0 && it > 0) mbar_wait(bar_dqd, (it - 1) & 1u, 0x714u);  // dQ of the previous item drained
          tc_fence_after();
          if (elect_one()) {
            // ---- dV_i += P_drop^T dO_j ; dK_i += dS^T Q_j     (contraction over the nq queries of tile j)
#pragma unroll
            for (int which = 0; which < 2; ++which) {
              const uint32_t ta = which ? tDP : tST, td = which ? tdK : tdV;
              const uint64_t db = desc_add(which ? dQm : dOm, qoff);
              for (int t = 0; t < nq / 16; ++t) {
#pragma unroll
                for (int cb = 0; cb < 3; ++cb)
                  umma_f16_ts(td, ta + 16 * t + 8 * PA[cb], desc_add(db, PB[cb] * ATB_QROWS + t * 2048), idesc_acc,
                               (j > 0 || t > 0 || cb > 0) ? 1u : 0u);
              }
            }
            // ---- dQ_j += dS_ij K_i     (contraction over the keys of tile i)
            const uint32_t tdQ = tmem_base + ATB_T_DQ + 64 * j;
            for (int t = 0; t < nk; ++t) {
#pragma unroll
              for (int cb = 0; cb < 3; ++cb)
                umma_f16(tdQ, desc_add(dSm, PA[cb] * 32768 + (t >> 2) * 16384 + (t & 3) * 2048),
                          desc_add(dKm, PB[cb] * 16384 + t * 2048), idesc_dq, (i > 0 || t > 0 || cb > 0) ? 1u : 0u);
            }
            if (j == tiles - 1) umma_commit(bar_tile);       // dV_i / dK_i (and, after the last tile, dQ) are complete
          }
          __syncwarp();
          ATB_STAMP(u, 3);
        }
      }
    }
  } else if (warp >= 4) {
    const int w = (warp - 4) & 3, part = (warp - 4) >> 2;          // lane quarter, column part (0..3)
    const int rr = w * 32 + lane;
    const int cw = threadIdx.x - 128;                              // 0..511 among the compute threads
    const uint32_t t_lane = static_cast<uint32_t>(w * 32) << 16;
    const uint32_t tST = tmem_base + ATB_T_ST + t_lane, tDP = tmem_base + ATB_T_DP + t_lane;
    const int h = static_cast<int>(blockIdx.x) % a.H;              // gridDim.x % H == 0: one head per CTA
    float acc_dq = 0.f, acc_dk = 0.f, acc_dv = 0.f;                // bias-gradient column (part * 16 + (lane & 15)) of this head
    // this thread's row in the dS^T operand tile (row = key): plane 0 at +0, plane 1 at +32768, query chunk c64 at + c64 * 8192
    const uint32_t ds_row = sdS + (rr >> 6) * 16384 + (rr & 63) * 128;
    const uint32_t ds_swz = static_cast<uint32_t>(rr & 7);
    // The same addresses double as the staging tiles of the coalesced drains (tile t = tensor * 2 + plane at
    // (t >> 1) * 32768 + (t & 1) * 8192): a lane quarter only ever touches its own rows of that region, so its four warps
    // synchronise among themselves (quarter_sync) and never with the other quarters.
    auto stage_addr = [&](int t, int row, int ch) {
      return sdS + (t >> 1) * 32768 + (t & 1) * 8192 + (row >> 6) * 16384 + (row & 63) * 128 + ((ch ^ (row & 7)) << 4);
    };
    uint32_t u = 0, kt = 0;
    // per-query statistics (row max and sum from the forward, delta) of the NEXT item are fetched into registers while
    // the current item is still being drained: their global-memory latency used to sit between two block barriers at
    // the start of every item (~1 500 of 38 800 cycles per item in the phase timeline)
    float2 ml_next = make_float2(0.f, 1.f);
    float dl_next = 0.f;
    auto fetch_stats = [&](int item) {
      if (cw < a.T && item < items) {
        ml_next = __ldg(a.stats + static_cast<int64_t>(item) * a.T + cw);
        dl_next = __ldg(a.delta + static_cast<int64_t>(item) * a.T + cw);
      }
    };
    fetch_stats(blockIdx.x);
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int b = item / a.H;
      // ---- per-query statistics of this slice and head: (m + log2 l, delta); queries past T get m = +inf -> P = 0
      asm volatile("bar.sync 5, 512;" ::: "memory");               // everybody is done with the previous item's statistics
      if (cw < ATB_STATS) {
        float2 st = make_float2(INFINITY, 0.f);
        if (cw < a.T) {
          st.x = ml_next.x + __log2f(ml_next.y);
          st.y = dl_next;
        }
        sStat[cw] = st;
      }
      asm volatile("bar.sync 5, 512;" ::: "memory");
      for (int i = 0; i < tiles; ++i, ++kt) {
        const int krows = rows_of(i);
        const bool kvalid = rr < krows;                            // rows >= krows belong to the next tile or lie past T
        const bool warp_keys = w * 32 < rows16_of(i);              // warp-uniform: some key step of this warp is contracted
        for (int j = 0; j < tiles; ++j, ++u) {
          const int nq = rows16_of(j);
          // keep bits of this warp's 32 keys for the queries it will visit: issued before the scores are waited for
          uint32_t mword[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};
          if (a.mbits != nullptr && warp_keys) {
            const int kc = (rpt * i + w * 32) >> 4;                // first of the two 16-key chunks of this warp's keys
#pragma unroll
            for (int n = 0; n < 2; ++n) {
              const int c = part + 4 * n;
              uint32_t mine = 0;
              const int q = rpt * j + 16 * c + lane;               // lanes 0..15 fetch one query each
              if (lane < 16 && 16 * c < nq && q < a.T) {
                const uint16_t* mb = a.mbits + (static_cast<int64_t>(item) * a.nC + kc) * a.T + q;
                mine = __ldg(mb);
                if (kc + 1 < a.nC) mine |= static_cast<uint32_t>(__ldg(mb + a.T)) << 16;
              }
              mword[n] = mine;
            }
          }
          mbar_wait(bar_m1, u & 1u, 0x720u);
          tc_fence_after();
          if (warp == 4 && lane == 0) ATB_STAMP(u, 4);
          if (warp_keys) {
#pragma unroll
            for (int n = 0; n < 2; ++n) {                          // nq <= 128: at most 8 chunks of 16, two per warp
              const int c = part + 4 * n;
              if (16 * c >= nq) break;
              const int qt = 16 * c;                               // query inside the tile
              uint32_t s_[16], d_[16];
              tmem_ld_32x16(tST + qt, s_);
              tmem_ld_32x16(tDP + qt, d_);
              // this key's keep bits over the chunk's 16 queries (bit x = query qt + x)
              uint32_t word = 0xFFFFFFFFu;
              if (a.mbits != nullptr) word = transpose32(mword[n], lane);
              const float2* strow = sStat + rpt * j + qt;          // < ATB_STATS entries are initialised for every index used
              tmem_ld_wait();
              uint32_t op[16], ods[16];
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
                float pd[2], ds[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const int x = 2 * jj + e;
                  const float2 st = strow[x];                      // (m + log2 l, delta); +inf past the slice -> p = 0
                  const float kf = (word & (1u << x)) ? a.inv_keep : 0.f;
                  const float p = fast_exp2(fmaf(__uint_as_float(s_[x]), ATF_SC, -st.x));
                  pd[e] = p * kf;
                  ds[e] = (p * 0.125f) * fmaf(__uint_as_float(d_[x]), kf, -st.y);
                }
                op[jj] = pack2(pd[0], pd[1]);
                op[jj + 8] = pack2(pd[0] - lo_to_f(op[jj]), pd[1] - hi_to_f(op[jj]));
                ods[jj] = pack2(ds[0], ds[1]);
                ods[jj + 8] = pack2(ds[0] - lo_to_f(ods[jj]), ds[1] - hi_to_f(ods[jj]));
              }
              // rows of keys that do not belong to this tile produce rows of dV / dK nobody reads, but their dS is
              // CONTRACTED by dQ = dS K: zero it there (the shared-memory copy), leave the TMEM copy alone
              tmem_st_32x16(tST + qt, op);
              tmem_st_32x16(tDP + qt, ods);
              if (!kvalid) {
#pragma unroll
                for (int x = 0; x < 16; ++x) ods[x] = 0u;
              }
              // dS^T -> shared memory, MN-major operand layout: row = key, 64 queries per 128-byte row
#pragma unroll
              for (int g = 0; g < 2; ++g) {
                const int qq = qt + 8 * g;
                const uint32_t dst = ds_row + (qq >> 6) * 8192 + ((((qq & 63) >> 3) ^ ds_swz) << 4);
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(ods[4 * g]), "r"(ods[4 * g + 1]),
                             "r"(ods[4 * g + 2]), "r"(ods[4 * g + 3]) : "memory");
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 32768), "r"(ods[8 + 4 * g]),
                             "r"(ods[9 + 4 * g]), "r"(ods[10 + 4 * g]), "r"(ods[11 + 4 * g]) : "memory");
              }
            }
            tmem_st_wait();
          }
          if (warp == 4 && lane == 0) ATB_STAMP(u, 5);
          fence_proxy_async();
          tc_fence_before();
          mbar_arrive(bar_p);
        }
        // ---- dV_i, dK_i complete (last query tile's MMAs retired; the dS tile in shared memory is free): every warp
        //      takes 16 of the 64 columns of each out of TMEM, stages them as fp16 planes, then the quarter's four warps
        //      write one (tensor, plane) each with full 128-byte rows
        mbar_wait(bar_tile, kt & 1u, 0x721u);
        tc_fence_after();
        if (warp == 4 && lane == 0) ATB_STAMP(u - 1, 6);
        if (warp_keys) {
#pragma unroll
          for (int which = 0; which < 2; ++which) {                // 0: dV, 1: dK
            uint32_t acc[16];
            tmem_ld_32x16(tmem_base + t_lane + (which ? ATB_T_DK : ATB_T_DV) + part * 16, acc);
            tmem_ld_wait();
            float v[16];
#pragma unroll
            for (int x = 0; x < 16; ++x) v[x] = kvalid ? __uint_as_float(acc[x]) : 0.f;
            stage16_two_planes(stage_addr(2 * which, rr, 2 * part), stage_addr(2 * which, rr, 2 * part + 1),
                               stage_addr(2 * which + 1, rr, 2 * part), stage_addr(2 * which + 1, rr, 2 * part + 1), v);
            const float cs = column_sums16(v, lane);
            if (which) acc_dk += cs; else acc_dv += cs;
          }
        }
        tc_fence_before();
        mbar_arrive(bar_kvd);                                     // TMEM accumulators are drained
        if (warp_keys) {
          quarter_sync(w);
          {   // tile `part`: tensor part >> 1 (0 dV, 1 dK), plane part & 1
            elem_t* gbase = a.dqkv + (part & 1) * a.dqkv_ps + ((part >> 1) ? 1 : 2) * 64 * a.H + h * 64 + (lane & 7) * 8;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const int row = w * 32 + it * 4 + (lane >> 3);
              const uint4 val = lds128(stage_addr(part, row, lane & 7));
              if (row < krows)
                *reinterpret_cast<uint4*>(gbase + (static_cast<int64_t>(b) * a.T + rpt * i + row) * (3 * 64 * a.H)) = val;
            }
          }
          quarter_sync(w);                                         // staging rows are free before the quarter writes dS again
        }
        if (warp == 4 && lane == 0) ATB_STAMP(u - 1, 7);
      }
      fetch_stats(item + gridDim.x);
      // ---- dQ of the whole slice (thread <-> query row): both query tiles are staged at once (tile 2 j + plane of the
      //      staging region), then each of the quarter's four warps writes one (query tile, plane) with 128-byte rows
      {
        bool act[2];
        act[0] = w * 32 < rows16_of(0);
        act[1] = tiles > 1 && w * 32 < rows16_of(1);               // warp-uniform and uniform over the quarter
        if (act[0] || act[1]) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            if (!act[j]) continue;
            const bool qvalid = rr < rows_of(j);
            uint32_t acc[16];
            tmem_ld_32x16(tmem_base + t_lane + ATB_T_DQ + 64 * j + part * 16, acc);
            tmem_ld_wait();
            float v[16];
#pragma unroll
            for (int x = 0; x < 16; ++x) v[x] = qvalid ? __uint_as_float(acc[x]) : 0.f;
            stage16_two_planes(stage_addr(2 * j, rr, 2 * part), stage_addr(2 * j, rr, 2 * part + 1),
                               stage_addr(2 * j + 1, rr, 2 * part), stage_addr(2 * j + 1, rr, 2 * part + 1), v);
            acc_dq += column_sums16(v, lane);
          }
          quarter_sync(w);
          {
            const int j = part >> 1, plane = part & 1;
            if (act[j]) {
              const int qrows = rows_of(j);
              elem_t* gbase = a.dqkv + plane * a.dqkv_ps + h * 64 + (lane & 7) * 8;
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                const int row = w * 32 + it * 4 + (lane >> 3);
                const uint4 val = lds128(stage_addr(part, row, lane & 7));
                if (row < qrows)
                  *reinterpret_cast<uint4*>(gbase + (static_cast<int64_t>(b) * a.T + rpt * j + row) * (3 * 64 * a.H)) = val;
              }
            }
          }
          quarter_sync(w);
        }
      }
      tc_fence_before();
      mbar_arrive(bar_dqd);
    }
    // ---- in-proj bias gradient: one atomic per warp, tensor and column for the whole kernel
    if (a.dbias != nullptr && blockIdx.x < items && lane < 16) {   // null: no parameter gradients wanted
      const int col = h * 64 + part * 16 + lane;
      const float inv_s = a.gscale != nullptr ? __ldg(a.gscale + 1) : 1.f;
      atomicAdd(a.dbias + col, acc_dq * inv_s);
      atomicAdd(a.dbias + 64 * a.H + col, acc_dk * inv_s);
      atomicAdd(a.dbias + 2 * 64 * a.H + col, acc_dv * inv_s);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// delta[(b*H + h)*T + t] = sum_d dO[b*T + t, h*64 + d] * O[b*T + t, h*64 + d]      (two planes of each; H = 4)
__global__ void __launch_bounds__(256) attn_delta_kernel(const elem_t* __restrict__ dout, int64_t do_ps,
                                                         const elem_t* __restrict__ out, int64_t o_ps,
                                                         float* __restrict__ delta, int64_t tokens, int T) {
  pdl_trigger();   // the next kernel of the stream may start its prologue (ptx.cuh)
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t tok = warp; tok < tokens; tok += nwarps) {
    float x[8], y[8];
    load8_split(dout, do_ps, 2, tok * 256 + lane * 8, x);
    load8_split(out, o_ps, 2, tok * 256 + lane * 8, y);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s = fmaf(x[i], y[i], s);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    if ((lane & 7) == 0) {
      const int64_t b = tok / T, t = tok % T;
      delta[(b * 4 + (lane >> 3)) * T + t] = s;
    }
  }
}

// qkv: forward stash [>=2 planes][B*T, 768]; out: forward attention output [>=2 planes][B*T, 256]; dout: its gradient
// [2 planes][B*T, 256]; dqkv: [2 planes][B*T, 768] (every element of the Q | K | V columns is written); dbias [768] +=.
int attn_train_bwd(const void* qkv, int64_t qkv_ps, const void* out, int64_t out_ps, const void* dout, int64_t dout_ps,
                   const float* stats, const uint32_t* mbits, float* delta, void* dqkv, int64_t dqkv_ps, float* dbias,
                   const float* gscale, DropCfg drop, int B, int H, int T, int Tp, cudaStream_t st) {
  SPK_CHECK(H == 4, "attn_train_bwd: 4 heads of 64");
  SPK_CHECK(T >= 1 && T <= ATB_MAXT, "attn_train_bwd: T=%d outside [1, %d]", T, ATB_MAXT);
  SPK_CHECK(drop.thresh == 0 || mbits != nullptr, "attn_train_bwd: dropout needs the forward's keep bits");
  const int64_t tokens = static_cast<int64_t>(B) * T;
  {
    ProfScope prof("attn_delta", 0, 2.0 * tokens * 256 * 2 * 2 + 4.0 * tokens * H, st);
    const int blocks = static_cast<int>(std::min<int64_t>((tokens + 7) / 8, 148 * 8));
    attn_delta_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const elem_t*>(dout), dout_ps,
                                              reinterpret_cast<const elem_t*>(out), out_ps, delta, tokens, T);
    SPK_CUDA(cudaGetLastError());
  }
  AttnTrainBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.H = H; a.T = T;
  a.Tk64 = (T + 63) / 64 * 64;
  a.tiles = (T + 127) / 128;
  a.rpt = ((T + a.tiles - 1) / a.tiles + 15) / 16 * 16;      // frames split evenly over the tiles, in 16-row steps
  a.nC = (Tp + 15) / 16;
  a.stats = reinterpret_cast<const float2*>(stats);
  a.delta = delta;
  a.mbits = drop.thresh != 0 ? reinterpret_cast<const uint16_t*>(mbits) : nullptr;
  a.dqkv = reinterpret_cast<elem_t*>(dqkv);
  a.dqkv_ps = dqkv_ps;
  a.dbias = dbias;
  a.gscale = gscale;
  a.inv_keep = drop.thresh != 0 ? drop.inv_keep : 1.f;
  a.timeline = g_attn_timeline;
  a.timeline_slots = g_attn_timeline_slots;
  const int64_t dims[4] = {64, T, H, B};
  const int64_t ostrides[3] = {64 * H, 64, static_cast<int64_t>(T) * 64 * H};
  for (int p = 0; p < 2; ++p) {
    const elem_t* plane = reinterpret_cast<const elem_t*>(qkv) + p * qkv_ps;
    SPK_TRY(encode_qkv_map(&a.q_map[p], plane, 0, B, H, T, a.Tk64));
    SPK_TRY(encode_qkv_map(&a.k_map[p], plane, 1, B, H, T, 128));
    SPK_TRY(encode_qkv_map(&a.v_map[p], plane, 2, B, H, T, 128));
    SPK_TRY(encode_map_4d(&a.do_map[p], reinterpret_cast<const elem_t*>(dout) + p * dout_ps, dims, ostrides, a.Tk64));
  }
  static PerDeviceOnce once;
  SPK_TRY(once.run([]() -> int {
    SPK_CUDA(cudaFuncSetAttribute(attn_train_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATB_SMEM));
    return 0;
  }));
  const int items = B * H;
  int grid = items < device_sm_count() ? items : device_sm_count();
  grid -= grid % H;                       // a CTA must only ever see one head (register-resident bias-gradient sums)
  SPK_CHECK(grid >= H, "attn_train_bwd: no CTAs");
  // algorithmic work: dV, dP, dQ, dK (the recomputed S is not credited); bytes: Q, K, V, O, dO in, dQ, dK, dV out
  ProfScope prof("attn_train_bwd", 8.0 * B * H * T * T * 64, (5.0 + 3.0) * B * T * 64 * H * 2.0 * 2, st);
  attn_train_bwd_kernel<<<grid, ATB_THREADS, ATB_SMEM, st>>>(a);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace spk
