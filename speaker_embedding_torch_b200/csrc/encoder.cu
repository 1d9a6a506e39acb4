// Encoder orchestration: GE2E.forward / its backward as a fixed sequence of kernel launches over a
// caller-owned workspace.  Mirrors /root/reference/Modules.py:46-59 (forward order) and the
// post-LN torch.nn.TransformerEncoderLayer built at Modules.py:25-36; math: SURVEY.md Appendix B.
//
// Data layout in HBM (all token-major, tokens = slices * frames):
//   split tensors  [planes][rows][cols] fp16   activations and gradients that feed tensor-core GEMMs
//   fp32           LayerNorm statistics, head vectors, parameters and parameter gradients
// Dense contractions run in gemm_tc.cu (tcgen05/TMEM/TMA); everything else is a coalesced row kernel.
#include "encoder.h"
#include "gemm.h"
#include "rowops.h"

namespace spk {

int attn_row0_fwd(const void* q0, int64_t q_ps, const void* kv, int64_t kv_ps, int planes, void* att0, int64_t a_ps,
                  float* p0, float* pd0, DropCfg drop, uint32_t site, int B, int H, int T, int Tp, cudaStream_t st);
int attn_row0_bwd(const void* datt0, int64_t da_ps, int g_planes, const void* q0, int64_t q_ps, const void* kv,
                  int64_t kv_ps, int planes, const float* p0, const float* pd0, void* dq0, int64_t dq_ps, void* dkv,
                  int64_t dkv_ps, float* dbias, const float* gscale, int B, int H, int T, int Tp, cudaStream_t st);
int attn_fused_fwd(const void* qkv, void* out, int64_t out_ld, int B, int H, int T, cudaStream_t st);
int attn_infer_fwd(const void* qkv, void* out, int64_t out_ld, int B, int H, int T, cudaStream_t st);
int attn_train_fwd(const void* qkv, int64_t qkv_ps, int planes, void* out, int64_t out_ps, int64_t out_ld, float* stats,
                   uint32_t* mbits, DropCfg drop, uint32_t site, int B, int H, int T, int Tp, cudaStream_t st);
int attn_train_bwd(const void* qkv, int64_t qkv_ps, const void* out, int64_t out_ps, const void* dout, int64_t dout_ps,
                   const float* stats, const uint32_t* mbits, float* delta, void* dqkv, int64_t dqkv_ps, float* dbias,
                   const float* gscale, DropCfg drop, int B, int H, int T, int Tp, cudaStream_t st);
int rows_add(void* dst, int64_t d_ps, int64_t dst_row_step, const void* src, int64_t s_ps, int planes, int rows,
             cudaStream_t st);

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Split {
  size_t off = 0;      // byte offset into the workspace
  int64_t ps = 0;      // plane stride, elements
};

// The sublayer after the attention: out-proj + residual -> LayerNorm1 -> FFN -> residual -> LayerNorm2.
struct SublayerBufs {
  Split att, z1, h1, f, z2, hout;
  size_t st1 = 0, st2 = 0;
  size_t fbits = 0;   // dense layers: ReLU mask of the FFN hidden activation, one bit per element ([F/32, Mt] words)
};

struct LayerBufs {
  Split qkv, p, pd;
  size_t astat = 0;   // fused training attention: (row max, row sum) per (slice, head, query)
  size_t abits = 0;   // fused training attention: dropout keep bits [B*H][ceil(Tp/32)][T]
  SublayerBufs sub;
};

// Last layer, t = 0 rows only (see attn_row0.cu): compact [B, .] buffers + K|V for every frame.
struct LastBufs {
  Split kv, q0;
  SublayerBufs sub;
  size_t p0 = 0, pd0 = 0;
};

struct Plan {
  int B, T, S, P, Tp, H, D, F, C, L;
  int64_t Mt, BH;
  bool keep, prune, fused_infer, fused_train;
  size_t h0bits = 0;  // [256 / 32][Mt] words: prenet ReLU mask
  size_t gscale;      // backward: (S, 1 / S), the power-of-two scale the gradient planes are carried at
  bool attn_tr;       // the dense layers of this training plan use the fused attention kernels (attn_train.cu)
  size_t adelta;      // fused training attention backward: delta = rowsum(dO * O), [B*H*T] fp32
  LastBufs last;
  Split wpack;
  int64_t w_pre, w_in[SPK_MAX_LAYERS], w_out[SPK_MAX_LAYERS], w_l1[SPK_MAX_LAYERS], w_l2[SPK_MAX_LAYERS];
  Split x0, h0, scr;
  size_t pe_t;
  LayerBufs Lb[SPK_MAX_LAYERS];
  size_t hn, hst, emean, epre, de;
  Split dh_a, dh_b, dz, dzd, df, datt, dqkv, ds, dq0;
  size_t total;
};

static Split take_split(size_t& cur, int64_t elems, int planes) {
  Split s;
  s.off = cur;
  s.ps = static_cast<int64_t>(align_up(static_cast<size_t>(elems), 128));
  cur = align_up(cur + static_cast<size_t>(s.ps) * planes * 2, 1024);
  return s;
}
static size_t take_f32(size_t& cur, int64_t elems) {
  size_t o = cur;
  cur = align_up(cur + static_cast<size_t>(elems) * 4, 1024);
  return o;
}
// `rows` rows of the sublayer.  fbits: allocate the FFN ReLU mask; hout: the buffer the output aliases, or nullptr for
// one of its own.
static SublayerBufs take_sublayer(size_t& cur, int64_t rows, int64_t D, int64_t F, int P, bool fbits,
                                  const Split* hout) {
  SublayerBufs s;
  s.att = take_split(cur, rows * D, P);
  s.z1 = take_split(cur, rows * D, P);
  s.st1 = take_f32(cur, rows * 2);
  s.h1 = take_split(cur, rows * D, P);
  s.f = take_split(cur, rows * F, P);
  if (fbits) s.fbits = take_f32(cur, rows * (F / 32));
  s.z2 = take_split(cur, rows * D, P);
  s.st2 = take_f32(cur, rows * 2);
  s.hout = hout ? *hout : take_split(cur, rows * D, P);
  return s;
}

static bool g_prune_last = true;   // spk_set_option("prune_last_layer", 0/1)
void encoder_set_prune(bool on) { g_prune_last = on; }
static bool g_fused_attn = true;   // spk_set_option("fused_inference_attention", 0/1)
static bool g_infer_attn_two = true;   // spk_set_option("inference_attention_two_ctas", 0/1)
static bool g_fuse_ln = true;          // spk_set_option("fused_layernorm", 0 | 1 | 2): 0 off, 1 inference only,
static bool g_fuse_ln_train = true;    // 2 (default) the two-plane training forward as well
void encoder_set_fuse_ln(int on) { g_fuse_ln = on != 0; g_fuse_ln_train = on >= 2; }
void encoder_set_infer_attn_two(int on) { g_infer_attn_two = on != 0; }
void encoder_set_fused_attn(bool on) { g_fused_attn = on; }
static bool g_fused_train_attn = true;   // spk_set_option("fused_training_attention", 0/1)
void encoder_set_fused_train_attn(bool on) { g_fused_train_attn = on; }

// The options that shape the workspace layout travel with the call: `precision` carries them in its upper bits
// (SPK_PLAN_*, include/spkemb.h) so that a backward pass always rebuilds the plan its forward pass used, whatever
// spk_set_option did in between.  Without SPK_PLAN_EXPLICIT the process-wide options apply.
int encoder_plan_flags() {
  return SPK_PLAN_EXPLICIT | (g_prune_last ? SPK_PLAN_PRUNE : 0) | (g_fused_attn ? SPK_PLAN_FUSED_INFER_ATTN : 0) |
         (g_fused_train_attn ? SPK_PLAN_FUSED_TRAIN_ATTN : 0);
}

static int make_plan(const spk_encoder_config& c, int B, int T, int S, int Pflags, bool keep, Plan& pl) {
  const int P = Pflags & 0xFF;
  const int opt = (Pflags & SPK_PLAN_EXPLICIT) ? Pflags : encoder_plan_flags();
  // Mel_Dim is the K of the prenet GEMM and the N of the input dgrad / prenet wgrad: the GEMMs need N % 8 == 0, the
  // TMA maps of the fp16 x0 [Mt, C] planes 16-byte row strides, and mel_pack stores groups of 8 channels.  With
  // C % 8 == 0 the packed weights that follow w_pre (256 * C elements) stay 16-byte aligned as well.
  SPK_CHECK(c.mel_dim % 8 == 0 && c.mel_dim >= 16 && c.mel_dim <= 256,
            "encoder: Mel_Dim %d must be a multiple of 8 in [16, 256]", c.mel_dim);
  SPK_CHECK(c.emb == 256 && c.heads == 4 && c.ffn == 1024,
            "encoder: this build supports Embedding_Size 256, Head 4 (got %d/%d/%d)", c.emb, c.heads, c.ffn);
  SPK_CHECK(c.layers >= 1 && c.layers <= SPK_MAX_LAYERS, "encoder: Num_Layers %d out of range", c.layers);
  SPK_CHECK(B >= 1 && T >= 1 && T <= c.max_pos && T <= 1024, "encoder: frames %d outside [1, %d]", T,
            c.max_pos < 1024 ? c.max_pos : 1024);
  SPK_CHECK(S >= 1 && B % S == 0, "encoder: batch %d is not a multiple of samples %d", B, S);
  SPK_CHECK(P >= 1 && P <= 3, "encoder: precision must be 1 (fp16), 2 (hi+lo) or 3 (hi+mid+lo)");
  pl.B = B; pl.T = T; pl.S = S; pl.P = P; pl.Tp = (T + 7) / 8 * 8;
  pl.H = c.heads; pl.D = c.emb; pl.F = c.ffn; pl.C = c.mel_dim; pl.L = c.layers;
  pl.Mt = static_cast<int64_t>(B) * T;
  pl.BH = static_cast<int64_t>(B) * pl.H;
  pl.keep = keep;
  pl.prune = (opt & SPK_PLAN_PRUNE) != 0;
  pl.fused_infer = (opt & SPK_PLAN_FUSED_INFER_ATTN) != 0;
  pl.fused_train = (opt & SPK_PLAN_FUSED_TRAIN_ATTN) != 0;
  const int64_t D = pl.D, F = pl.F, Mt = pl.Mt;
  size_t cur = 0;
  // packed weights
  int64_t w = 0;
  pl.w_pre = w; w += D * pl.C;
  for (int l = 0; l < pl.L; ++l) {
    pl.w_in[l] = w; w += 3 * D * D;
    pl.w_out[l] = w; w += D * D;
    pl.w_l1[l] = w; w += F * D;
    pl.w_l2[l] = w; w += D * F;
  }
  pl.wpack = take_split(cur, w, P);
  pl.x0 = take_split(cur, Mt * pl.C, P);
  pl.h0 = take_split(cur, Mt * D, P);
  pl.h0bits = keep ? take_f32(cur, Mt * (D / 32)) : 0;     // 1-bit ReLU mask of the prenet (backward)
  pl.pe_t = take_f32(cur, static_cast<int64_t>(T) * D);
  // fused training attention (scores never leave the SM): multi-plane training plans up to 192 frames
  pl.attn_tr = keep && pl.fused_train && P >= 2 && T <= 192 && pl.H == 4;
  const int64_t score_elems = pl.attn_tr ? 128 : pl.BH * T * pl.Tp;     // the materialised path's score tensors
  pl.scr = take_split(cur, score_elems, P < 2 ? 2 : P);   // also holds fp32 scores / dP (4 B per element)
  const bool drop = keep;   // P_drop is only distinct in training; allocate with the stash
  const int dense_layers = pl.prune ? pl.L - 1 : pl.L;
  for (int l = 0; l < dense_layers; ++l) {
    if (l > 0 && !keep) { pl.Lb[l] = pl.Lb[0]; continue; }
    LayerBufs& b = pl.Lb[l];
    b.qkv = take_split(cur, Mt * 3 * D, P);
    b.p = take_split(cur, score_elems, P);
    b.pd = drop ? take_split(cur, score_elems, P) : b.p;
    if (pl.attn_tr) {
      b.astat = take_f32(cur, pl.BH * T * 2);
      b.abits = take_f32(cur, pl.BH * ((pl.Tp + 31) / 32) * T);
    }
    b.sub = take_sublayer(cur, Mt, D, F, P, true, keep ? nullptr : &pl.h0);
  }
  if (pl.prune) {
    LastBufs& lb = pl.last;
    lb.kv = take_split(cur, Mt * 2 * D, P);
    lb.q0 = take_split(cur, B * D, P);
    lb.sub = take_sublayer(cur, B, D, F, P, false, nullptr);
    lb.p0 = take_f32(cur, pl.BH * pl.Tp);
    lb.pd0 = take_f32(cur, pl.BH * pl.Tp);
  }
  const int64_t Bo = B / S;
  pl.hn = take_f32(cur, static_cast<int64_t>(B) * D);
  pl.hst = take_f32(cur, static_cast<int64_t>(B) * 2);
  pl.emean = take_f32(cur, Bo * D);
  pl.epre = take_f32(cur, Bo * D);
  pl.de = take_f32(cur, Bo * D);
  if (keep) {   // gradients are smooth in their inputs: two planes (~2^-16) are enough in the backward pass
    const int Pb = P < 2 ? P : 2;
    pl.dh_a = take_split(cur, Mt * D, Pb);
    pl.dh_b = take_split(cur, Mt * D, Pb);
    pl.dz = take_split(cur, Mt * D, Pb);
    pl.dzd = take_split(cur, Mt * D, Pb);
    pl.df = take_split(cur, Mt * F, Pb);
    // the input gradient dX (fp32 [Mt, C]) is written into df, dead once the last sublayer backward has run:
    // 2 * F * Pb >= 2048 bytes per token at every plane count, against 4 * C <= 1024
    SPK_CHECK(static_cast<size_t>(pl.df.ps) * Pb * 2 >= static_cast<size_t>(Mt) * pl.C * 4,
              "encoder: the dX region (%lld bytes) is smaller than %lld tokens x %d fp32 channels",
              (long long)pl.df.ps * Pb * 2, (long long)Mt, pl.C);
    pl.datt = take_split(cur, Mt * D, Pb);
    pl.dqkv = take_split(cur, Mt * 3 * D, Pb);
    pl.ds = take_split(cur, score_elems, Pb);
    pl.adelta = take_f32(cur, pl.BH * T);
    pl.gscale = take_f32(cur, 64);
    // compact [B, 256] gradient of the last layer's single query row (its own buffer: scr is BH*T*Tp elements per
    // plane, smaller than B*256 for T < 8)
    if (pl.prune) pl.dq0 = take_split(cur, static_cast<int64_t>(B) * D, Pb);
  }
  pl.total = cur + 1024;
  return 0;
}

size_t encoder_workspace_bytes(const spk_encoder_config& c, int B, int T, int S, int P, int keep) {
  Plan pl;
  if (make_plan(c, B, T, S, P, keep != 0, pl) != 0) return 0;
  return pl.total;
}

// Debug aid for the parity tests: byte offset / plane stride of every workspace buffer, one text line
// per buffer: "name offset plane_stride_elems" (layer buffers as "L<l>.<name>").
int encoder_debug_layout(const spk_encoder_config& c, int B, int T, int S, int P, int keep, char* buf, size_t cap) {
  Plan pl;
  SPK_TRY(make_plan(c, B, T, S, P, keep != 0, pl));
  size_t off = 0;
  auto put = [&](const char* pre, const char* name, size_t o, int64_t ps) {
    int n = snprintf(buf + off, off < cap ? cap - off : 0, "%s%s %zu %lld\n", pre, name, o, (long long)ps);
    if (n > 0 && off + n < cap) off += n;
  };
  auto put_sub = [&](const char* pre, const SublayerBufs& s, const char* att) {
    put(pre, att, s.att.off, s.att.ps);
    put(pre, "z1", s.z1.off, s.z1.ps); put(pre, "h1", s.h1.off, s.h1.ps); put(pre, "f", s.f.off, s.f.ps);
    put(pre, "z2", s.z2.off, s.z2.ps); put(pre, "hout", s.hout.off, s.hout.ps);
    put(pre, "st1", s.st1, 0); put(pre, "st2", s.st2, 0);
  };
  put("", "x0", pl.x0.off, pl.x0.ps); put("", "h0", pl.h0.off, pl.h0.ps);
  put("", "scr", pl.scr.off, pl.scr.ps); put("", "pe_t", pl.pe_t, 0);
  if (keep) put("", "h0bits", pl.h0bits, 0);
  for (int l = 0; l < (pl.prune ? pl.L - 1 : pl.L); ++l) {
    const LayerBufs& b = pl.Lb[l];
    char pre[16];
    snprintf(pre, sizeof(pre), "L%d.", l);
    put(pre, "qkv", b.qkv.off, b.qkv.ps); put(pre, "p", b.p.off, b.p.ps); put(pre, "pd", b.pd.off, b.pd.ps);
    put_sub(pre, b.sub, "att");
    put(pre, "fbits", b.sub.fbits, 0);
    if (pl.attn_tr) { put(pre, "astat", b.astat, 0); put(pre, "abits", b.abits, 0); }
  }
  if (pl.prune) {
    const LastBufs& lb = pl.last;
    put("last.", "kv", lb.kv.off, lb.kv.ps); put("last.", "q0", lb.q0.off, lb.q0.ps);
    put_sub("last.", lb.sub, "att0");
    put("last.", "p0", lb.p0, 0); put("last.", "pd0", lb.pd0, 0);
  }
  put("", "hn", pl.hn, 0); put("", "hst", pl.hst, 0); put("", "emean", pl.emean, 0);
  put("", "epre", pl.epre, 0); put("", "de", pl.de, 0);
  if (keep) {
    put("", "gscale", pl.gscale, 0);
    put("", "dh_a", pl.dh_a.off, pl.dh_a.ps); put("", "dh_b", pl.dh_b.off, pl.dh_b.ps);
    put("", "dz", pl.dz.off, pl.dz.ps); put("", "dzd", pl.dzd.off, pl.dzd.ps);
    put("", "df", pl.df.off, pl.df.ps); put("", "datt", pl.datt.off, pl.datt.ps);
    put("", "dqkv", pl.dqkv.off, pl.dqkv.ps); put("", "ds", pl.ds.off, pl.ds.ps);
  }
  return static_cast<int>(off);
}

// ------------------------------------------------------------------------------------------------
// Gradient scale of one backward pass.  The gradient tensors live in fp16 planes (common.cuh): they are carried
// multiplied by S = 2^k, k chosen so that max |dL/d dvec| * S lands in [2^11, 2^12) -- four binades of headroom below
// the fp16 maximum for growth inside the encoder (conversions saturate, they never produce inf), and as much range as
// possible below: a pair of fp16 planes carries 22 bits only down to 0.125, smaller values keep an ABSOLUTE precision of
// 2^-25, so the measured gradient error falls with S (2 x 2 x 1024 frames: 1.5e-3 at 2^8, 1.5e-4 at 2^12, 7e-5 at 2^14;
// tools/grad_probe.py).  Everything downstream of the head is linear in the gradient, so S travels through untouched; the kernels
// that meet unscaled quantities (parameter gradients: weight-gradient GEMMs, bias column sums, LayerNorm affine
// gradients, alpha) multiply by 1 / S, read from this buffer.  S is a device scalar: no host synchronisation.
static int g_grad_scale_log2 = 12;    // spk_set_option("grad_scale_log2", k): max |dL/d dvec| * S lands in [2^(k-1), 2^k)
void encoder_set_grad_scale_log2(int k) { g_grad_scale_log2 = k < -8 ? -8 : (k > 15 ? 15 : k); }
__global__ void __launch_bounds__(1024) grad_scale_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ out,
                                                          int target_log2) {
  __shared__ float red[32];
  float mx = 0.f;
  // one block (the result is one scalar), 16-byte loads, four in flight per thread: 245 760 values in ~6 us
  const int64_t n4 = (reinterpret_cast<uintptr_t>(g) & 15) == 0 ? n / 4 : 0;
  const float4* g4 = reinterpret_cast<const float4*>(g);
#pragma unroll 4
  for (int64_t i = threadIdx.x; i < n4; i += 1024) {
    const float4 v = __ldg(g4 + i);
    mx = fmaxf(fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  for (int64_t i = n4 * 4 + threadIdx.x; i < n; i += 1024) mx = fmaxf(mx, fabsf(g[i]));
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int w = 0; w < 32; ++w) m = fmaxf(m, red[w]);
    float s = 1.f;
    if (m > 0.f && isfinite(m)) {
      int e;
      frexpf(m, &e);                       // m = f * 2^e, f in [0.5, 1)
      int k = target_log2 - e;             // m * 2^k in [2^(target-1), 2^target)
      k = k < -24 ? -24 : (k > 40 ? 40 : k);
      s = ldexpf(1.f, k);
    }
    out[0] = s;
    out[1] = 1.f / s;
  }
}

// ------------------------------------------------------------------------------------------------
// d-vector head (Modules.py:54-57): final LayerNorm of the t = 0 token of every slice, mean over the
// `samples` slices of an utterance, 256x256 projection (fp32), L2 normalisation.
// Eight utterances per block, one warp each: the 256 KB projection matrix is read once per block (the first version
// ran one utterance per block and moved 960 x 256 KB through L2 per call: 45 us for 2 MB of real work).
// SEG (variable-length utterances): utterance u owns slices segments[u] .. segments[u+1] - 1 of the `batch` slices
// and is averaged with 1 / count; S is unused.  The fixed-S instantiation never reads the two trailing arguments.
constexpr int HEAD_UPB = 8;
// First slice and slice count of utterance u: the device table is clamped to [0, batch), whatever it holds.
__device__ __forceinline__ int seg_bounds(const int32_t* __restrict__ segments, int64_t u, int64_t batch,
                                          int64_t& first) {
  int64_t b = __ldg(segments + u), e = __ldg(segments + u + 1);
  b = b < 0 ? 0 : (b > batch ? batch : b);
  e = e < b ? b : (e > batch ? batch : e);
  first = b;
  return static_cast<int>(e - b);
}
template <bool SEG>
__global__ void __launch_bounds__(256) head_fwd_kernel(const elem_t* __restrict__ h, int64_t ps, int planes,
                                                       int T, int S, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, const float* __restrict__ wp,
                                                       const float* __restrict__ bp, float* __restrict__ hn,
                                                       float2* __restrict__ hst, float* __restrict__ emean,
                                                       float* __restrict__ epre, float* __restrict__ dvec, int64_t U,
                                                       const int32_t* __restrict__ segments, int64_t batch) {
  __shared__ __align__(16) float em[HEAD_UPB][256];
  __shared__ float wt[256][33];                      // projection rows n0 .. n0+31, transposed: wt[k][n - n0]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t u = static_cast<int64_t>(blockIdx.x) * HEAD_UPB + warp;
  const bool valid = u < U;
  // ---- final LayerNorm of the t = 0 token of each slice, mean over the slices (lane owns columns lane*8 .. +7)
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (valid) {
    float g[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { g[i] = __ldg(gamma + lane * 8 + i); b[i] = __ldg(beta + lane * 8 + i); }
    // The fixed-S loop is spelled out apart from the SEG one: sharing the body (a lambda, a common slice range) changed
    // the register allocation of the fixed-S kernel that the training step and the benchmark run.
    if constexpr (SEG) {
      int64_t first;
      const int count = seg_bounds(segments, u, batch, first);
      for (int s = 0; s < count; ++s) {
        const int64_t slice = first + s;
        float v[8];
        load8_split(h, ps, planes, slice * T * 256 + lane * 8, v);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) sum += v[i];
        const float mean = warp_sum(sum) * (1.f / 256.f);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { v[i] -= mean; q += v[i] * v[i]; }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / 256.f) + 1e-5f);
        float y[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { y[i] = v[i] * rstd * g[i] + b[i]; acc[i] += y[i]; }
        float4* dst = reinterpret_cast<float4*>(hn + slice * 256 + lane * 8);
        dst[0] = make_float4(y[0], y[1], y[2], y[3]);
        dst[1] = make_float4(y[4], y[5], y[6], y[7]);
        if (lane == 0) hst[slice] = make_float2(mean, rstd);
      }
      const float inv_s = 1.f / static_cast<float>(count > 0 ? count : 1);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] *= inv_s;
    } else {
      for (int s = 0; s < S; ++s) {
        const int64_t slice = u * S + s;
        float v[8];
        load8_split(h, ps, planes, slice * T * 256 + lane * 8, v);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) sum += v[i];
        const float mean = warp_sum(sum) * (1.f / 256.f);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) { v[i] -= mean; q += v[i] * v[i]; }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / 256.f) + 1e-5f);
        float y[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { y[i] = v[i] * rstd * g[i] + b[i]; acc[i] += y[i]; }
        float4* dst = reinterpret_cast<float4*>(hn + slice * 256 + lane * 8);
        dst[0] = make_float4(y[0], y[1], y[2], y[3]);
        dst[1] = make_float4(y[4], y[5], y[6], y[7]);
        if (lane == 0) hst[slice] = make_float2(mean, rstd);
      }
      const float inv_s = 1.f / static_cast<float>(S);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] *= inv_s;
    }
    float4* dst = reinterpret_cast<float4*>(emean + u * 256 + lane * 8);
    dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) em[warp][lane * 8 + i] = acc[i];
  // ---- projection: 32 outputs per round; lane = output within the round, warp = utterance
  // The next round's 32 weight rows travel from L2 into registers while this round is multiplied (one L2 latency per
  // round instead of four serialised load batches); four accumulators break the 256-long FMA chain.
  float eo[8];
  float wv[32];
#pragma unroll
  for (int it = 0; it < 32; ++it) wv[it] = __ldg(wp + static_cast<int64_t>(it) * 256 + tid);
#pragma unroll 1
  for (int t = 0; t < 8; ++t) {
    __syncthreads();                                 // em is written / the previous round's tile has been consumed
#pragma unroll
    for (int it = 0; it < 32; ++it) wt[tid][it] = wv[it];
    if (t + 1 < 8) {
#pragma unroll
      for (int it = 0; it < 32; ++it) wv[it] = __ldg(wp + static_cast<int64_t>((t + 1) * 32 + it) * 256 + tid);
    }
    __syncthreads();
    float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll 8
    for (int k = 0; k < 256; k += 4) {
      const float4 e4 = *reinterpret_cast<const float4*>(&em[warp][k]);
      d0 = fmaf(wt[k][lane], e4.x, d0);
      d1 = fmaf(wt[k + 1][lane], e4.y, d1);
      d2 = fmaf(wt[k + 2][lane], e4.z, d2);
      d3 = fmaf(wt[k + 3][lane], e4.w, d3);
    }
    eo[t] = ((d0 + d1) + (d2 + d3)) + __ldg(bp + t * 32 + lane);
  }
  if (valid) {
    float ss = 0.f;
#pragma unroll
    for (int t = 0; t < 8; ++t) ss += eo[t] * eo[t];
    const float nrm = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      epre[u * 256 + t * 32 + lane] = eo[t];
      dvec[u * 256 + t * 32 + lane] = eo[t] / nrm;
    }
  }
}

// Backward of the head, eight utterances per block (one warp each): d_dvec -> de (pre-normalisation), d_emean,
// final-LN backward into the t = 0 rows of dH (pre-zeroed), dgamma / dbeta of the final LayerNorm (both null: skipped).
// SEG: slices as in head_fwd_kernel<true>; each of an utterance's slices receives d_emean / count.
template <bool SEG>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ g_dvec, const float* __restrict__ epre,
                                                       const float* __restrict__ wp, const elem_t* __restrict__ h,
                                                       int64_t h_ps, int planes, const float2* __restrict__ hst,
                                                       const float* __restrict__ gamma, int T, int S,
                                                       float* __restrict__ de_out, elem_t* __restrict__ dh,
                                                       int64_t dh_ps, float* __restrict__ dgamma,
                                                       float* __restrict__ dbeta, const float* __restrict__ gscale,
                                                       int64_t U, const int32_t* __restrict__ segments, int64_t batch) {
  __shared__ float des[HEAD_UPB][256];
  __shared__ float wt[32][256];                      // projection rows n0 .. n0+31 (also the dgamma / dbeta exchange)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t u = static_cast<int64_t>(blockIdx.x) * HEAD_UPB + warp;
  const bool valid = u < U;
  // ---- L2-normalisation backward (lane owns outputs lane*8 .. +7)
  {
    float e[8], go[8], de[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { e[i] = 0.f; go[i] = 0.f; }
    if (valid) {
      const float4* ep = reinterpret_cast<const float4*>(epre + u * 256 + lane * 8);
      const float4* gp = reinterpret_cast<const float4*>(g_dvec + u * 256 + lane * 8);
      const float4 e0 = ep[0], e1 = ep[1], g0 = gp[0], g1 = gp[1];
      e[0] = e0.x; e[1] = e0.y; e[2] = e0.z; e[3] = e0.w; e[4] = e1.x; e[5] = e1.y; e[6] = e1.z; e[7] = e1.w;
      go[0] = g0.x; go[1] = g0.y; go[2] = g0.z; go[3] = g0.w; go[4] = g1.x; go[5] = g1.y; go[6] = g1.z; go[7] = g1.w;
    }
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) ss += e[i] * e[i];
    const float nrm = sqrtf(warp_sum(ss));
    if (nrm > 1e-12f) {            // warp-uniform
      float dot = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { e[i] /= nrm; dot += go[i] * e[i]; }
      dot = warp_sum(dot);
#pragma unroll
      for (int i = 0; i < 8; ++i) de[i] = (go[i] - dot * e[i]) / nrm;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) de[i] = go[i] / 1e-12f;
    }
    if (valid) {
      float4* dst = reinterpret_cast<float4*>(de_out + u * 256 + lane * 8);
      dst[0] = make_float4(de[0], de[1], de[2], de[3]);
      dst[1] = make_float4(de[4], de[5], de[6], de[7]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) des[warp][lane * 8 + i] = valid ? de[i] : 0.f;
  }
  // ---- d_emean[k] = sum_n Wp[n][k] * de[n]   (lane owns k = lane + 32 j)
  float dm[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) dm[j] = 0.f;
  float wv[32];                                      // next round's weight rows in flight while this one is consumed
#pragma unroll
  for (int it = 0; it < 32; ++it) wv[it] = __ldg(wp + static_cast<int64_t>(it) * 256 + tid);
#pragma unroll 1
  for (int t = 0; t < 8; ++t) {
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 32; ++it) wt[it][tid] = wv[it];
    if (t + 1 < 8) {
#pragma unroll
      for (int it = 0; it < 32; ++it) wv[it] = __ldg(wp + static_cast<int64_t>((t + 1) * 32 + it) * 256 + tid);
    }
    __syncthreads();
#pragma unroll 4
    for (int nl = 0; nl < 32; ++nl) {
      const float dv = des[warp][t * 32 + nl];
#pragma unroll
      for (int j = 0; j < 8; ++j) dm[j] = fmaf(wt[nl][lane + 32 * j], dv, dm[j]);
    }
  }
  // as in head_fwd_kernel, the fixed-S code is spelled out apart from the SEG code
  float ag[8], ab[8];
  if constexpr (SEG) {
    int64_t first = 0;
    int count = 0;
    if (valid) count = seg_bounds(segments, u, batch, first);
    const float inv_s = 1.f / static_cast<float>(count > 0 ? count : 1);   // gradient of every slice's LN output
    float gam[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { dm[j] *= inv_s; ag[j] = 0.f; ab[j] = 0.f; gam[j] = __ldg(gamma + lane + 32 * j); }
    if (valid) {
      const float gsc = __ldg(gscale);                     // the gradient enters the encoder scaled by S
      for (int s = 0; s < count; ++s) {
        const int64_t slice = first + s;
        const int64_t off = slice * T * 256 + lane;
        const float2 ms = hst[slice];
        float xh[8], gd[8];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          xh[j] = (load1_split(h, h_ps, planes, off + 32 * j) - ms.x) * ms.y;
          ag[j] += dm[j] * xh[j];
          ab[j] += dm[j];
          gd[j] = dm[j] * gam[j];
          s1 += gd[j];
          s2 += gd[j] * xh[j];
        }
        const float m1 = warp_sum(s1) * (1.f / 256.f);
        const float m2 = warp_sum(s2) * (1.f / 256.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) store1_split(dh, dh_ps, planes, off + 32 * j, ms.y * (gd[j] - m1 - xh[j] * m2) * gsc);
      }
    }
  } else {
    const float inv_s = 1.f / static_cast<float>(S);       // gradient of every slice's LayerNorm output
    float gam[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { dm[j] *= inv_s; ag[j] = 0.f; ab[j] = 0.f; gam[j] = __ldg(gamma + lane + 32 * j); }
    if (valid) {
      const float gsc = __ldg(gscale);                     // the gradient enters the encoder scaled by S
      for (int s = 0; s < S; ++s) {
        const int64_t slice = u * S + s;
        const int64_t off = slice * T * 256 + lane;
        const float2 ms = hst[slice];
        float xh[8], gd[8];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          xh[j] = (load1_split(h, h_ps, planes, off + 32 * j) - ms.x) * ms.y;
          ag[j] += dm[j] * xh[j];
          ab[j] += dm[j];
          gd[j] = dm[j] * gam[j];
          s1 += gd[j];
          s2 += gd[j] * xh[j];
        }
        const float m1 = warp_sum(s1) * (1.f / 256.f);
        const float m2 = warp_sum(s2) * (1.f / 256.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) store1_split(dh, dh_ps, planes, off + 32 * j, ms.y * (gd[j] - m1 - xh[j] * m2) * gsc);
      }
    }
  }
  // ---- dgamma / dbeta: the block's eight utterances meet in shared memory, one atomic per column and block
  if (dgamma == nullptr) return;   // no parameter gradients wanted (block-uniform)
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 8; ++j) { wt[warp][lane + 32 * j] = ag[j]; wt[8 + warp][lane + 32 * j] = ab[j]; }
  __syncthreads();
  float sg = 0.f, sb = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) { sg += wt[w][tid]; sb += wt[8 + w][tid]; }
  atomicAdd(dgamma + tid, sg);
  atomicAdd(dbeta + tid, sb);
}

// dWp[n][k] += sum_u de[u][n] * emean[u][k] ; dbp[n] += sum_u de[u][n]
// Block (32 outputs n, chunk of utterances): thread k keeps 32 accumulators, the chunk's de columns sit in shared memory
// (broadcast reads); partial sums meet in fp32 atomics.
constexpr int HEAD_WG_UCH = 64;                      // utterances per block
__global__ void __launch_bounds__(256) head_wgrad_kernel(const float* __restrict__ de, const float* __restrict__ emean,
                                                         int64_t U, float* __restrict__ dwp, float* __restrict__ dbp) {
  __shared__ __align__(16) float ds[HEAD_WG_UCH][32];
  const int n0 = blockIdx.x * 32, k = threadIdx.x;
  const int64_t u0 = static_cast<int64_t>(blockIdx.y) * HEAD_WG_UCH;
  const int nu = static_cast<int>(U - u0 < HEAD_WG_UCH ? U - u0 : HEAD_WG_UCH);
  for (int i = threadIdx.x; i < HEAD_WG_UCH * 32; i += 256) {
    const int uu = i >> 5, nn = i & 31;
    ds[uu][nn] = uu < nu ? __ldg(de + (u0 + uu) * 256 + n0 + nn) : 0.f;
  }
  __syncthreads();
  float acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
#pragma unroll 4
  for (int uu = 0; uu < nu; ++uu) {
    const float e = __ldg(emean + (u0 + uu) * 256 + k);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 d4 = *reinterpret_cast<const float4*>(&ds[uu][4 * q]);
      acc[4 * q] = fmaf(d4.x, e, acc[4 * q]);
      acc[4 * q + 1] = fmaf(d4.y, e, acc[4 * q + 1]);
      acc[4 * q + 2] = fmaf(d4.z, e, acc[4 * q + 2]);
      acc[4 * q + 3] = fmaf(d4.w, e, acc[4 * q + 3]);
    }
  }
#pragma unroll
  for (int i = 0; i < 32; ++i) atomicAdd(dwp + static_cast<int64_t>(n0 + i) * 256 + k, acc[i]);
  if (k < 32) {
    float sb = 0.f;
    for (int uu = 0; uu < nu; ++uu) sb += ds[uu][k];
    atomicAdd(dbp + n0 + k, sb);
  }
}

// ------------------------------------------------------------------------------------------------
namespace {

struct Ctx {
  const Plan& pl;
  char* ws;
  cudaStream_t st;
  int P;
  const float* gs = nullptr;   // backward: the device scalars (S, 1 / S) of grad_scale_kernel
  bool pgrad = true;           // backward: parameter gradients are wanted (spk_encoder_backward_input, grads != NULL)
  uint32_t colsum() const { return pgrad ? EPI_COLSUM : 0u; }   // bias gradients fused into a data-gradient GEMM
  // backward: gemm_run, handing 1 / S to every epilogue that produces parameter gradients (fp32 atomics of the weight
  // gradients, fused bias column sums)
  int run(GemmProblem& g) const {
    if (g.epi.flags & EPI_OUT_ATOMIC) g.epi.alpha_ptr = gs + 1;
    if (g.epi.flags & EPI_COLSUM) g.epi.colsum_scale_ptr = gs + 1;
    return gemm_run(g, st);
  }
  elem_t* ptr(const Split& s, int64_t elem_off = 0) const {
    return reinterpret_cast<elem_t*>(ws + s.off) + elem_off;
  }
  float* f32(size_t off) const { return reinterpret_cast<float*>(ws + off); }
  SplitMat mat(const Split& s, int64_t elem_off, int64_t rows, int64_t cols, int64_t ld, int64_t sb0 = 0,
               int64_t sb1 = 0) const {
    SplitMat m;
    m.base = ptr(s, elem_off);
    m.plane_stride = s.ps;
    m.rows = rows; m.cols = cols; m.ld = ld; m.sb0 = sb0; m.sb1 = sb1;
    return m;
  }
  void out(GemmEpilogue& e, const Split& s, int64_t elem_off, int64_t ld, int64_t sb0 = 0, int64_t sb1 = 0) const {
    e.out = ptr(s, elem_off);
    e.out_plane_stride = s.ps; e.out_ld = ld; e.out_sb0 = sb0; e.out_sb1 = sb1; e.out_planes = P;
  }
  void res(GemmEpilogue& e, const Split& s, int64_t ld) const {
    e.res = ptr(s);
    e.res_plane_stride = s.ps; e.res_ld = ld; e.res_planes = P;
  }
};

// p + off, or null when no parameter gradient is wanted
float* at(float* p, int64_t off) { return p != nullptr ? p + off : nullptr; }

int wgrad_ksplit(int64_t K, int M, int N) {
  const int tiles = ((M + 127) / 128) * ((N + 255) / 256);
  const int kb = static_cast<int>((K + 63) / 64);
  // two full waves of tiles x slices: rounding UP put 6 tiles x 50 slices = 300 work items on 148 CTAs (a third,
  // nearly empty wave: the QKV weight gradient ran 19 % longer than with 49 slices)
  int ks = (2 * device_sm_count()) / tiles;
  if (ks > kb) ks = kb;
  return ks < 1 ? 1 : ks;
}

// Y[rows, N] = X[rows, K] W^T, W = the packed weight [N, K] at w_off   (both operands K-major)
GemmProblem linear(const Ctx& c, const char* tag, const Split& x, int64_t rows, int64_t K, int64_t x_ld, int64_t w_off,
                   int64_t N) {
  GemmProblem g;
  g.tag = tag;
  g.A = c.mat(x, 0, rows, K, x_ld);
  g.B = c.mat(c.pl.wpack, w_off, N, K, K);
  g.planes = c.P;
  g.M = static_cast<int>(rows); g.N = static_cast<int>(N); g.K = static_cast<int>(K);
  return g;
}

// dX[rows, K] = dY[rows, N] W, W = the packed weight [N, K] at w_off   (W read MN-major)
GemmProblem dgrad(const Ctx& c, const char* tag, const Split& dy, int64_t rows, int64_t N, int64_t w_off, int64_t K) {
  GemmProblem g;
  g.tag = tag;
  g.A = c.mat(dy, 0, rows, N, N);
  g.B = c.mat(c.pl.wpack, w_off, N, K, K);
  g.b_mn = true;
  g.planes = c.P;
  g.M = static_cast<int>(rows); g.N = static_cast<int>(K); g.K = static_cast<int>(N);
  return g;
}

// dW[M_out, N_in] += dY^T[M_out, rows] * X[rows, N_in]   (both operands read MN-major, split-K, fp32 atomics; dY arrives
// scaled by S, c.run multiplies by 1 / S)
int wgrad(const Ctx& c, const char* tag, int64_t rows, const Split& dy, int64_t dy_cols, const Split& x, int64_t x_cols,
          int64_t x_ld, float* dw) {
  if (dw == nullptr) return 0;   // no parameter gradients wanted
  GemmProblem g;
  g.tag = tag;
  g.A = c.mat(dy, 0, rows, dy_cols, dy_cols);
  g.B = c.mat(x, 0, rows, x_cols, x_ld);
  g.a_mn = true; g.b_mn = true; g.planes = c.P;
  g.M = static_cast<int>(dy_cols); g.N = static_cast<int>(x_cols); g.K = static_cast<int>(rows);
  g.ksplit = wgrad_ksplit(rows, g.M, g.N);
  g.epi.flags = EPI_OUT_ATOMIC;
  g.epi.out = dw; g.epi.out_ld = x_cols;
  return c.run(g);
}

// The sublayer of layer l after its attention, over `rows` rows of s.att: out-proj + dropout1 + residual ->
// LayerNorm1 -> FFN1 + ReLU + dropout -> FFN2 + dropout2 + residual -> LayerNorm2.  The residual rows are read from
// hin every hin_ld elements (D; the pruned last layer gathers the t = 0 rows of every slice with T*D).
//   fuse_ln    both LayerNorms run inside the out-proj / FFN2 epilogues (EPI_LN); a plan that keeps the stash also
//              stores the pre-normalisation rows and the row statistics the backward needs
//   emit_bits  FFN1 writes its ReLU mask to s.fbits for the backward's gate
//   last       the pruned last layer (its profiler tags)
int sublayer_fwd(const Ctx& c, const spk_layer_params& lw, int l, const SublayerBufs& s, int64_t rows, const Split& hin,
                 int64_t hin_ld, bool fuse_ln, bool emit_bits, DropCfg drop, bool last) {
  const Plan& pl = c.pl;
  const int64_t D = pl.D, F = pl.F;
  const uint32_t drop_flag = drop.thresh ? EPI_DROPOUT : 0;
  // Runs a GEMM whose output rows z are LayerNorm-ed into y: inside its epilogue (the tile owns whole rows; inference:
  // z never leaves the SM) or by ln_fwd after it.
  auto gemm_ln = [&](GemmProblem& g, const float* gamma, const float* beta, const Split& z, size_t stats,
                     const Split& y) -> int {
    if (!fuse_ln) {
      c.out(g.epi, z, 0, D);
      SPK_TRY(gemm_run(g, c.st));
      return ln_fwd(c.ptr(z), z.ps, c.P, 1, gamma, beta, c.ptr(y), y.ps, c.P, c.f32(stats), rows, c.st);
    }
    g.epi.flags |= EPI_LN; g.epi.ln_gamma = gamma; g.epi.ln_beta = beta;
    c.out(g.epi, y, 0, D);
    if (pl.keep) { g.epi.ln_z = c.ptr(z); g.epi.ln_z_plane_stride = z.ps; g.epi.ln_stats = c.f32(stats); }
    return gemm_run(g, c.st);
  };
  {  // out-proj + dropout1 + residual -> LayerNorm1
    GemmProblem g = linear(c, last ? "gemm.last.out_proj" : "gemm.out_proj", s.att, rows, D, D, pl.w_out[l], D);
    g.epi.flags = EPI_BIAS | EPI_RES | drop_flag;
    g.epi.bias = lw.out_proj_b; g.epi.drop = drop; g.epi.drop_site = 2 + 4 * l;
    c.res(g.epi, hin, hin_ld);
    SPK_TRY(gemm_ln(g, lw.norm1_w, lw.norm1_b, s.z1, s.st1, s.h1));
  }
  {  // linear1 + ReLU + dropout
    GemmProblem g = linear(c, last ? "gemm.last.ffn1" : "gemm.ffn1", s.h1, rows, D, D, pl.w_l1[l], F);
    g.epi.flags = EPI_BIAS | EPI_RELU | drop_flag;
    g.epi.bias = lw.linear1_b; g.epi.drop = drop; g.epi.drop_site = 3 + 4 * l;
    if (emit_bits) {   // the backward's ReLU gate reads one bit per element instead of a whole plane of f
      g.epi.flags |= EPI_EMIT_BITS;
      g.epi.gate_bits = reinterpret_cast<uint32_t*>(c.f32(s.fbits));
    }
    c.out(g.epi, s.f, 0, F);
    SPK_TRY(gemm_run(g, c.st));
  }
  // linear2 + dropout2 + residual -> LayerNorm2
  GemmProblem g = linear(c, last ? "gemm.last.ffn2" : "gemm.ffn2", s.f, rows, F, F, pl.w_l2[l], D);
  g.epi.flags = EPI_BIAS | EPI_RES | drop_flag;
  g.epi.bias = lw.linear2_b; g.epi.drop = drop; g.epi.drop_site = 4 + 4 * l;
  c.res(g.epi, s.h1, D);
  return gemm_ln(g, lw.norm2_w, lw.norm2_b, s.z2, s.st2, s.hout);
}

// Backward of sublayer_fwd from the gradient dh of its output: LayerNorm2 -> FFN2 -> FFN1 (dH1 into dh_b) ->
// LayerNorm1 -> out-proj (dATT into datt), the parameter gradients on the way.  The FFN2 dgrad's ReLU gate reads the
// forward's mask bits s.fbits (gate_bits) or the sign of plane 0 of s.f.
int sublayer_bwd(const Ctx& c, const spk_layer_params& lw, const spk_layer_params& lg, int l, const SublayerBufs& s,
                 int64_t rows, const Split& dh, bool gate_bits, DropCfg drop, bool last) {
  const Plan& pl = c.pl;
  const int64_t D = pl.D, F = pl.F;
  const int P = c.P;
  const Split& dy = drop.thresh ? pl.dzd : pl.dz;
  // ---- LayerNorm2 backward: dH(out) -> dZ2 (residual path) and dZ2 * mask (FFN path)
  SPK_TRY(ln_bwd(c.ptr(dh), dh.ps, P, c.ptr(s.z2), s.z2.ps, P, c.f32(s.st2), lw.norm2_w, c.ptr(pl.dz), pl.dz.ps, P,
                 c.ptr(pl.dzd), drop, 4 + 4 * l, lg.norm2_w, lg.norm2_b, lg.linear2_b, rows, c.gs, c.st));
  SPK_TRY(wgrad(c, last ? "gemm.last.bwd.ffn2_wgrad" : "gemm.bwd.ffn2_wgrad", rows, dy, D, s.f, F, F, lg.linear2_w));
  {  // dU = (dY2 W2) * 1[f > 0] / (1 - p)
    GemmProblem g = dgrad(c, last ? "gemm.last.bwd.ffn2_dgrad" : "gemm.bwd.ffn2_dgrad", dy, rows, D, pl.w_l2[l], F);
    g.epi.flags = c.colsum();
    g.epi.colsum = lg.linear1_b;
    if (gate_bits) {
      g.epi.flags |= EPI_GATE_BITS;
      g.epi.gate_bits = reinterpret_cast<uint32_t*>(c.f32(s.fbits));   // written by the forward FFN1 epilogue
    } else {
      g.epi.flags |= EPI_GATE_POS;
      g.epi.gate = c.ptr(s.f); g.epi.gate_plane_stride = s.f.ps; g.epi.gate_ld = F; g.epi.gate_planes = 1;
    }
    g.epi.gate_scale = drop.inv_keep;
    c.out(g.epi, pl.df, 0, F);
    SPK_TRY(c.run(g));
  }
  SPK_TRY(wgrad(c, last ? "gemm.last.bwd.ffn1_wgrad" : "gemm.bwd.ffn1_wgrad", rows, pl.df, F, s.h1, D, D,
                lg.linear1_w));
  {  // dH1 = dU W1 + dZ2
    GemmProblem g = dgrad(c, last ? "gemm.last.bwd.ffn1_dgrad" : "gemm.bwd.ffn1_dgrad", pl.df, rows, F, pl.w_l1[l], D);
    g.epi.flags = EPI_RES;
    c.res(g.epi, pl.dz, D);
    c.out(g.epi, pl.dh_b, 0, D);
    SPK_TRY(c.run(g));
  }
  // ---- LayerNorm1 backward
  SPK_TRY(ln_bwd(c.ptr(pl.dh_b), pl.dh_b.ps, P, c.ptr(s.z1), s.z1.ps, P, c.f32(s.st1), lw.norm1_w, c.ptr(pl.dz),
                 pl.dz.ps, P, c.ptr(pl.dzd), drop, 2 + 4 * l, lg.norm1_w, lg.norm1_b, lg.out_proj_b, rows, c.gs, c.st));
  SPK_TRY(wgrad(c, last ? "gemm.last.bwd.out_wgrad" : "gemm.bwd.out_wgrad", rows, dy, D, s.att, D, D, lg.out_proj_w));
  {  // dATT = dY1 Wo
    GemmProblem g = dgrad(c, last ? "gemm.last.bwd.out_dgrad" : "gemm.bwd.out_dgrad", dy, rows, D, pl.w_out[l], D);
    c.out(g.epi, pl.datt, 0, D);
    SPK_TRY(c.run(g));
  }
  return 0;
}

}  // namespace

static void fill_pack_table(const Plan& pl, const spk_encoder_params& w, PackTable& tab) {
  int n = 0;
  auto add = [&](const float* src, int64_t off, int64_t cnt) { tab.seg[n].src = src; tab.seg[n].dst_off = off; tab.seg[n].n = cnt; ++n; };
  const int64_t D = pl.D, F = pl.F;
  add(w.prenet_w, pl.w_pre, D * pl.C);
  for (int l = 0; l < pl.L; ++l) {
    add(w.layer[l].in_proj_w, pl.w_in[l], 3 * D * D);
    add(w.layer[l].out_proj_w, pl.w_out[l], D * D);
    add(w.layer[l].linear1_w, pl.w_l1[l], F * D);
    add(w.layer[l].linear2_w, pl.w_l2[l], D * F);
  }
  tab.count = n;
}

int encoder_forward(const spk_encoder_config& cfg, const spk_encoder_params& w, const spk_mel_view* mel,
                    const spk_mel_ragged* ragged, int B, int T, int S, int P, int training, uint64_t seed, float* dvec,
                    void* ws_v, size_t ws_bytes, int keep, cudaStream_t st, const int32_t* segments, int utterances) {
  SPK_CHECK(segments == nullptr || (S == 1 && utterances >= 1 && utterances <= B),
            "encoder: a segmented call runs at samples 1 with 1 <= utterances <= batch (got %d, %d)", S, utterances);
  Plan pl;
  SPK_TRY(make_plan(cfg, B, T, S, P, keep != 0, pl));
  P = pl.P;     // the upper bits carried the plan options
  if (ws_bytes < pl.total) { set_error("encoder: workspace too small (%zu < %zu)", ws_bytes, pl.total); return SPK_ENOMEM; }
  SPK_CHECK((reinterpret_cast<uintptr_t>(ws_v) & 255) == 0, "encoder: workspace must be 256-byte aligned");
  SPK_CHECK(!training || keep, "encoder: training forward needs keep_stash (dropout P buffers live in the stash)");
  Ctx c{pl, reinterpret_cast<char*>(ws_v), st, P};
  GemmDependentLaunchScope dependent_launch(!keep && !training);   // inference: GEMM prologues under the previous kernel's tail
  const int64_t Mt = pl.Mt, D = pl.D;
  const int Tp = pl.Tp, H = pl.H;
  const DropCfg drop_pe = make_drop(seed, cfg.pe_dropout, training != 0);
  const DropCfg drop = make_drop(seed, cfg.dropout, training != 0);

  PackTable tab;
  fill_pack_table(pl, w, tab);
  SPK_TRY(pack_weights(tab, c.ptr(pl.wpack), pl.wpack.ps, P, st));
  if (ragged != nullptr) SPK_TRY(mel_pack_ragged(*ragged, c.ptr(pl.x0), pl.x0.ps, P, B, pl.C, T, st));
  else SPK_TRY(mel_pack(*mel, c.ptr(pl.x0), pl.x0.ps, P, B, pl.C, T, st));
  SPK_TRY(pe_transpose(w.pe, c.f32(pl.pe_t), pl.D, cfg.max_pos, T, st));

  {  // prenet k=1 conv + ReLU + alpha * PE (+ dropout)        Modules.py:50-52,98-105
    GemmProblem g = linear(c, "gemm.prenet", pl.x0, Mt, pl.C, pl.C, pl.w_pre, D);
    g.epi.flags = EPI_BIAS | EPI_RELU | EPI_PE | (drop_pe.thresh ? EPI_DROPOUT : 0);
    if (pl.keep && P >= 2) {   // the backward gates dH0 with the forward's own ReLU decisions
      g.epi.flags |= EPI_EMIT_BITS;
      g.epi.gate_bits = reinterpret_cast<uint32_t*>(c.f32(pl.h0bits));
    }
    g.epi.bias = w.prenet_b; g.epi.pe_t = c.f32(pl.pe_t); g.epi.pe_alpha = w.pe_alpha; g.epi.pe_T = T;
    g.epi.drop = drop_pe; g.epi.drop_site = 0;
    c.out(g.epi, pl.h0, 0, D);
    SPK_TRY(gemm_run(g, st));
  }
  const int dense_layers = pl.prune ? pl.L - 1 : pl.L;
  // both LayerNorms of the dense layers run inside the GEMM epilogues (the pruned last layer keeps ln_fwd)
  const bool fuse_ln = g_fuse_ln && P <= 2 && (!keep || (g_fuse_ln_train && P == 2));   // EPI_LN kernels exist for 1 and 2 planes
  for (int l = 0; l < dense_layers; ++l) {
    const LayerBufs& b = pl.Lb[l];
    const Split& hin = (l == 0) ? pl.h0 : pl.Lb[l - 1].sub.hout;
    const spk_layer_params& lw = w.layer[l];
    {  // in-proj
      GemmProblem g = linear(c, "gemm.qkv", hin, Mt, D, D, pl.w_in[l], 3 * D);
      g.epi.flags = EPI_BIAS; g.epi.bias = lw.in_proj_b;
      c.out(g.epi, b.qkv, 0, 3 * D);
      SPK_TRY(gemm_run(g, st));
    }
    // inference (one plane, nothing kept for a backward pass): scores, softmax and PV in one tcgen05 kernel
    const bool fused_attn = (P == 1) && !keep && !training && T <= 256 && pl.fused_infer;
    if (fused_attn && T <= 192 && g_infer_attn_two) {      // two CTAs per SM (attn_train.cu, inference variant)
      SPK_TRY(attn_infer_fwd(c.ptr(b.qkv), c.ptr(b.sub.att), D, B, H, T, st));
    } else if (fused_attn) {
      SPK_TRY(attn_fused_fwd(c.ptr(b.qkv), c.ptr(b.sub.att), D, B, H, T, st));
    } else if (pl.attn_tr) {
      SPK_TRY(attn_train_fwd(c.ptr(b.qkv), b.qkv.ps, P, c.ptr(b.sub.att), b.sub.att.ps, D, c.f32(b.astat),
                             reinterpret_cast<uint32_t*>(c.f32(b.abits)), drop, 1 + 4 * l, B, H, T, Tp, st));
    } else {
    {  // S = Q K^T / sqrt(dh), per (slice, head)
      GemmProblem g;
      g.tag = "gemm.attn_qk";
      g.A = c.mat(b.qkv, 0, T, 64, 3 * D, 64, (int64_t)T * 3 * D);
      g.B = c.mat(b.qkv, D, T, 64, 3 * D, 64, (int64_t)T * 3 * D);
      g.planes = P; g.M = T; g.N = Tp; g.K = 64; g.nb0 = H; g.nb1 = B;
      g.epi.alpha = 0.125f;
      c.out(g.epi, pl.scr, 0, Tp, (int64_t)T * Tp, (int64_t)H * T * Tp);
      if (P >= 2) g.epi.flags |= EPI_OUT_F32;   // multi-plane modes keep the scores in fp32 (cheaper epilogue, 4 B instead of 2P B)
      if (P >= 2) g.block_n = 64;   // K = 64 is one k-block per tile: 64-wide tiles keep a two-stage ring and finer work items
      SPK_TRY(gemm_run(g, st));
    }
    SPK_TRY(softmax_fwd(c.ptr(pl.scr), P >= 2 ? reinterpret_cast<const float*>(c.ptr(pl.scr)) : nullptr, pl.scr.ps, P,
                        c.ptr(b.p), c.ptr(b.pd), drop, 1 + 4 * l, pl.BH * T, T, Tp, st));
    {  // O = P V, heads written back interleaved into [tokens, 256]
      GemmProblem g;
      g.tag = "gemm.attn_pv";
      g.A = c.mat(drop.thresh ? b.pd : b.p, 0, T, T, Tp, (int64_t)T * Tp, (int64_t)H * T * Tp);
      g.B = c.mat(b.qkv, 2 * D, T, 64, 3 * D, 64, (int64_t)T * 3 * D);
      g.b_mn = true;
      g.planes = P; g.M = T; g.N = 64; g.K = T; g.nb0 = H; g.nb1 = B;
      c.out(g.epi, b.sub.att, 0, D, 64, (int64_t)T * D);
      SPK_TRY(gemm_run(g, st));
    }
    }
    SPK_TRY(sublayer_fwd(c, lw, l, b.sub, Mt, hin, D, fuse_ln, pl.keep, drop, false));
  }
  if (pl.prune) {
    // ---- last layer: only the t = 0 query row of every slice is consumed (Modules.py:54)
    const int l = pl.L - 1;
    const LastBufs& lb = pl.last;
    const Split& hin = (l == 0) ? pl.h0 : pl.Lb[l - 1].sub.hout;
    const spk_layer_params& lw = w.layer[l];
    {  // K | V for every frame
      GemmProblem g = linear(c, "gemm.last.kv", hin, Mt, D, D, pl.w_in[l] + D * D, 2 * D);
      g.epi.flags = EPI_BIAS; g.epi.bias = lw.in_proj_b + D;
      c.out(g.epi, lb.kv, 0, 2 * D);
      SPK_TRY(gemm_run(g, st));
    }
    {  // Q for the first frame of every slice (rows gathered by the row stride T*D)
      GemmProblem g = linear(c, "gemm.last.q0", hin, B, D, (int64_t)T * D, pl.w_in[l], D);
      g.epi.flags = EPI_BIAS; g.epi.bias = lw.in_proj_b;
      c.out(g.epi, lb.q0, 0, D);
      SPK_TRY(gemm_run(g, st));
    }
    SPK_TRY(attn_row0_fwd(c.ptr(lb.q0), lb.q0.ps, c.ptr(lb.kv), lb.kv.ps, P, c.ptr(lb.sub.att), lb.sub.att.ps,
                          keep ? c.f32(lb.p0) : nullptr, keep ? c.f32(lb.pd0) : nullptr, drop, 1 + 4 * l, B, H, T, Tp, st));
    SPK_TRY(sublayer_fwd(c, lw, l, lb.sub, B, hin, (int64_t)T * D, false, false, drop, true));
  }
  const Split& hl = pl.prune ? pl.last.sub.hout : pl.Lb[pl.L - 1].sub.hout;
  const int head_T = pl.prune ? 1 : T;     // the compact buffer holds one row per slice
  if (segments != nullptr) {   // variable slice counts per utterance; the plan is the samples = 1 plan (B >= U)
    ProfScope prof_head("head_fwd_seg", 2.0 * utterances * 256 * 256, 4.0 * B * 256 * 2, st);
    head_fwd_kernel<true><<<(utterances + HEAD_UPB - 1) / HEAD_UPB, 256, 0, st>>>(
        c.ptr(hl), hl.ps, P, head_T, 1, w.norm_w, w.norm_b, w.proj_w, w.proj_b, c.f32(pl.hn),
        reinterpret_cast<float2*>(c.f32(pl.hst)), c.f32(pl.emean), c.f32(pl.epre), dvec,
        static_cast<int64_t>(utterances), segments, static_cast<int64_t>(B));
    SPK_CUDA(cudaGetLastError());
    return 0;
  }
  ProfScope prof_head("head_fwd", 2.0 * (B / S) * 256 * 256, 4.0 * B * 256 * 2, st);
  head_fwd_kernel<false><<<(B / S + HEAD_UPB - 1) / HEAD_UPB, 256, 0, st>>>(
      c.ptr(hl), hl.ps, P, head_T, S, w.norm_w, w.norm_b, w.proj_w, w.proj_b, c.f32(pl.hn),
      reinterpret_cast<float2*>(c.f32(pl.hst)), c.f32(pl.emean), c.f32(pl.epre), dvec, static_cast<int64_t>(B / S),
      nullptr, 0);
  SPK_CUDA(cudaGetLastError());
  return 0;
}

int encoder_backward(const spk_encoder_config& cfg, const spk_encoder_params& w, const spk_encoder_params* grads,
                     float* d_mel, const float* d_dvec, int B, int T, int S, int P_fwd, int training, uint64_t seed,
                     void* ws_v, size_t ws_bytes, cudaStream_t st, const RaggedGrad* rg) {
  const int32_t* segments = rg != nullptr ? rg->segments : nullptr;
  SPK_CHECK(rg == nullptr || (rg->mel != nullptr && rg->utterances >= 1 && rg->utterances <= B &&
                              (segments != nullptr ? S == 1 : B / rg->utterances == S)),
            "encoder: ragged backward: bad utterance count %d for batch %d, samples %d", rg ? rg->utterances : 0, B, S);
  SPK_CHECK(rg == nullptr || d_mel == nullptr, "encoder: d_mel and a ragged input gradient are exclusive");
  const int64_t U = segments != nullptr ? rg->utterances : B / S;   // d-vectors
  Plan pl;
  SPK_TRY(make_plan(cfg, B, T, S, P_fwd, true, pl));
  P_fwd = pl.P;
  if (ws_bytes < pl.total) { set_error("encoder: workspace too small (%zu < %zu)", ws_bytes, pl.total); return SPK_ENOMEM; }
  const int P = P_fwd < 2 ? P_fwd : 2;   // the stash may hold 3 planes; the backward pass reads / writes 2
  Ctx c{pl, reinterpret_cast<char*>(ws_v), st, P};
  // grads == nullptr: every gradient pointer below is null, so no weight-gradient GEMM, column sum or atomic runs;
  // the data path (dz, dh, dqkv, datt, d_mel) is the same either way
  static const spk_encoder_params no_grads = {};
  const spk_encoder_params& gr = grads != nullptr ? *grads : no_grads;
  c.pgrad = grads != nullptr;
  const int64_t Mt = pl.Mt, D = pl.D;
  const int Tp = pl.Tp, H = pl.H;
  const DropCfg drop_pe = make_drop(seed, cfg.pe_dropout, training != 0);
  const DropCfg drop = make_drop(seed, cfg.dropout, training != 0);
  float* gs = c.f32(pl.gscale);   // gradient scale of this pass (device scalars S, 1 / S)
  c.gs = gs;
  grad_scale_kernel<<<1, 1024, 0, st>>>(d_dvec, U * 256, gs, g_grad_scale_log2);
  SPK_CUDA(cudaGetLastError());

  // ---- head
  const Split& hl = pl.prune ? pl.last.sub.hout : pl.Lb[pl.L - 1].sub.hout;
  const int head_T = pl.prune ? 1 : T;
  // dense: the gradient of the last layer's output is zero except the t = 0 rows; pruned: compact [B, 256] in dh_b
  const Split& dhead = pl.prune ? pl.dh_b : pl.dh_a;
  if (!pl.prune) SPK_CUDA(cudaMemsetAsync(c.ptr(pl.dh_a), 0, static_cast<size_t>(pl.dh_a.ps) * P * 2, st));
  // segmented: a slice that no segment covers (segments[U] < B breaks the ABI's precondition) gets a zero gradient row
  // instead of whatever the compact buffer held
  else if (segments != nullptr)
    SPK_CUDA(cudaMemsetAsync(c.ptr(pl.dh_b), 0, static_cast<size_t>(pl.dh_b.ps) * P * 2, st));
  {
  ProfScope prof_hb(segments != nullptr ? "head_bwd_seg" : "head_bwd", 4.0 * U * 256 * 256, 4.0 * B * 256 * 2, st);
  if (segments != nullptr)   // variable slice counts per utterance (plan at samples = 1)
    head_bwd_kernel<true><<<(U + HEAD_UPB - 1) / HEAD_UPB, 256, 0, st>>>(
        d_dvec, c.f32(pl.epre), w.proj_w, c.ptr(hl), hl.ps, P, reinterpret_cast<const float2*>(c.f32(pl.hst)),
        w.norm_w, head_T, 1, c.f32(pl.de), c.ptr(dhead), dhead.ps, gr.norm_w, gr.norm_b, gs, U, segments,
        static_cast<int64_t>(B));
  else
    head_bwd_kernel<false><<<(B / S + HEAD_UPB - 1) / HEAD_UPB, 256, 0, st>>>(
        d_dvec, c.f32(pl.epre), w.proj_w, c.ptr(hl), hl.ps, P, reinterpret_cast<const float2*>(c.f32(pl.hst)),
        w.norm_w, head_T, S, c.f32(pl.de), c.ptr(dhead), dhead.ps, gr.norm_w, gr.norm_b, gs,
        static_cast<int64_t>(B / S), nullptr, 0);
  SPK_CUDA(cudaGetLastError());
  if (c.pgrad) {   // de / emean hold one row per d-vector, whatever the slicing
    head_wgrad_kernel<<<dim3(8, (U + HEAD_WG_UCH - 1) / HEAD_WG_UCH), 256, 0, st>>>(c.f32(pl.de), c.f32(pl.emean), U,
                                                                                   gr.proj_w, gr.proj_b);
    SPK_CUDA(cudaGetLastError());
  }
  }

  if (pl.prune) {
    // ---- last layer on the compact t = 0 rows (buffers dh_b / dz / dzd / df / datt hold B rows here)
    const int l = pl.L - 1;
    const LastBufs& lb = pl.last;
    const Split& hin = (l == 0) ? pl.h0 : pl.Lb[l - 1].sub.hout;
    const spk_layer_params& lg = gr.layer[l];
    // the FFN2 dgrad gates on the sign of f: the last layer keeps no ReLU mask bits
    SPK_TRY(sublayer_bwd(c, w.layer[l], lg, l, lb.sub, B, pl.dh_b, false, drop, true));
    // single-query attention backward: dq0 (compact [B, 256]), dK | dV -> dqkv viewed as [Mt, 512]
    SPK_TRY(attn_row0_bwd(c.ptr(pl.datt), pl.datt.ps, P, c.ptr(lb.q0), lb.q0.ps, c.ptr(lb.kv), lb.kv.ps, P_fwd,
                          c.f32(lb.p0), c.f32(lb.pd0), c.ptr(pl.dq0), pl.dq0.ps, c.ptr(pl.dqkv), pl.dqkv.ps,
                          lg.in_proj_b, gs, B, H, T, Tp, st));
    SPK_TRY(wgrad(c, "gemm.last.bwd.q_wgrad", B, pl.dq0, D, hin, D, (int64_t)T * D, lg.in_proj_w));
    // dW[K|V rows] = dKV^T hin
    SPK_TRY(wgrad(c, "gemm.last.bwd.kv_wgrad", Mt, pl.dqkv, 2 * D, hin, D, D, at(lg.in_proj_w, D * D)));
    {  // dH(in) = dKV W[K|V rows]  for every frame
      GemmProblem g = dgrad(c, "gemm.last.bwd.kv_dgrad", pl.dqkv, Mt, 2 * D, pl.w_in[l] + D * D, D);
      c.out(g.epi, pl.dh_a, 0, D);
      SPK_TRY(c.run(g));
    }
    {  // t = 0 rows additionally receive dq0 Wq and the residual path dZ1
      GemmProblem g = dgrad(c, "gemm.last.bwd.q_dgrad", pl.dq0, B, D, pl.w_in[l], D);
      g.epi.flags = EPI_RES;
      c.res(g.epi, pl.dz, D);
      c.out(g.epi, pl.dh_b, 0, D);
      SPK_TRY(c.run(g));
    }
    SPK_TRY(rows_add(c.ptr(pl.dh_a), pl.dh_a.ps, T, c.ptr(pl.dh_b), pl.dh_b.ps, P, B, st));
  }

  for (int l = (pl.prune ? pl.L - 2 : pl.L - 1); l >= 0; --l) {
    const LayerBufs& b = pl.Lb[l];
    const Split& hin = (l == 0) ? pl.h0 : pl.Lb[l - 1].sub.hout;
    const spk_layer_params& lg = gr.layer[l];
    SPK_TRY(sublayer_bwd(c, w.layer[l], lg, l, b.sub, Mt, pl.dh_a, true, drop, false));
    // ---- attention backward, per (slice, head)
    if (pl.attn_tr) {
      SPK_TRY(attn_train_bwd(c.ptr(b.qkv), b.qkv.ps, c.ptr(b.sub.att), b.sub.att.ps, c.ptr(pl.datt), pl.datt.ps,
                             c.f32(b.astat), reinterpret_cast<const uint32_t*>(c.f32(b.abits)), c.f32(pl.adelta),
                             c.ptr(pl.dqkv), pl.dqkv.ps, lg.in_proj_b, gs, drop, B, H, T, Tp, st));
    } else {
    const Split& pdrop = drop.thresh ? b.pd : b.p;
    const int64_t sP0 = (int64_t)T * Tp, sP1 = (int64_t)H * T * Tp;
    const int64_t sQ0 = 64, sQ1 = (int64_t)T * 3 * D, sA1 = (int64_t)T * D;
    {  // dV = P_drop^T dO
      GemmProblem g;
      g.tag = "gemm.bwd.attn_dv";
      g.A = c.mat(pdrop, 0, T, T, Tp, sP0, sP1);
      g.B = c.mat(pl.datt, 0, T, 64, D, 64, sA1);
      g.a_mn = true; g.b_mn = true;
      g.planes = P; g.M = T; g.N = 64; g.K = T; g.nb0 = H; g.nb1 = B;
      g.epi.flags = c.colsum(); g.epi.colsum = at(lg.in_proj_b, 2 * D); g.epi.colsum_sb0 = 64;
      c.out(g.epi, pl.dqkv, 2 * D, 3 * D, sQ0, sQ1);
      SPK_TRY(c.run(g));
    }
    {  // dP_drop = dO V^T
      GemmProblem g;
      g.tag = "gemm.bwd.attn_dp";
      g.A = c.mat(pl.datt, 0, T, 64, D, 64, sA1);
      g.B = c.mat(b.qkv, 2 * D, T, 64, 3 * D, sQ0, sQ1);
      g.planes = P; g.M = T; g.N = Tp; g.K = 64; g.nb0 = H; g.nb1 = B;
      c.out(g.epi, pl.scr, 0, Tp, sP0, sP1);
      if (P >= 2) g.epi.flags |= EPI_OUT_F32;
      if (P >= 2) g.block_n = 64;   // as for QK^T
      SPK_TRY(c.run(g));
    }
    SPK_TRY(softmax_bwd(c.ptr(b.p), c.ptr(pl.scr), P >= 2 ? reinterpret_cast<const float*>(c.ptr(pl.scr)) : nullptr,
                        b.p.ps, P, c.ptr(pl.ds), drop, 1 + 4 * l, 0.125f, pl.BH * T, T, Tp, st));
    {  // dQ = dS K
      GemmProblem g;
      g.tag = "gemm.bwd.attn_dq";
      g.A = c.mat(pl.ds, 0, T, T, Tp, sP0, sP1);
      g.B = c.mat(b.qkv, D, T, 64, 3 * D, sQ0, sQ1);
      g.b_mn = true;
      g.planes = P; g.M = T; g.N = 64; g.K = T; g.nb0 = H; g.nb1 = B;
      g.epi.flags = c.colsum(); g.epi.colsum = lg.in_proj_b; g.epi.colsum_sb0 = 64;
      c.out(g.epi, pl.dqkv, 0, 3 * D, sQ0, sQ1);
      SPK_TRY(c.run(g));
    }
    {  // dK = dS^T Q
      GemmProblem g;
      g.tag = "gemm.bwd.attn_dk";
      g.A = c.mat(pl.ds, 0, T, T, Tp, sP0, sP1);
      g.B = c.mat(b.qkv, 0, T, 64, 3 * D, sQ0, sQ1);
      g.a_mn = true; g.b_mn = true;
      g.planes = P; g.M = T; g.N = 64; g.K = T; g.nb0 = H; g.nb1 = B;
      g.epi.flags = c.colsum(); g.epi.colsum = at(lg.in_proj_b, D); g.epi.colsum_sb0 = 64;
      c.out(g.epi, pl.dqkv, D, 3 * D, sQ0, sQ1);
      SPK_TRY(c.run(g));
    }
    }
    // ---- in-proj
    SPK_TRY(wgrad(c, "gemm.bwd.qkv_wgrad", Mt, pl.dqkv, 3 * D, hin, D, D, lg.in_proj_w));
    {  // dH(in) = dQKV Win + dZ1
      GemmProblem g = dgrad(c, "gemm.bwd.qkv_dgrad", pl.dqkv, Mt, 3 * D, pl.w_in[l], D);
      g.epi.flags = EPI_RES;
      c.res(g.epi, pl.dz, D);
      c.out(g.epi, pl.dh_a, 0, D);
      SPK_TRY(c.run(g));
    }
  }
  // ---- embedding: positional alpha, prenet weight / bias
  if (P >= 2) {   // one pass over dH0: dropout mask, d_alpha, ReLU gate from the forward's mask bits, bias gradient
    SPK_TRY(prenet_bwd(c.ptr(pl.dh_a), pl.dh_a.ps, P, reinterpret_cast<const uint32_t*>(c.f32(pl.h0bits)), c.f32(pl.pe_t),
                       drop_pe, 0, c.ptr(pl.dh_b), pl.dh_b.ps, gr.pe_alpha, gr.prenet_b, Mt, T, gs, st));
  } else {        // one-plane plans keep no mask: the gate is recomputed from x0 W^T + b
    SPK_TRY(pe_alpha_grad(c.ptr(pl.dh_a), pl.dh_a.ps, P, c.f32(pl.pe_t), drop_pe, 0, gr.pe_alpha, Mt, T, gs, st));
    {
      GemmProblem g = linear(c, "gemm.bwd.prenet_gate", pl.x0, Mt, pl.C, pl.C, pl.w_pre, D);
      g.planes = P_fwd;   // same operand planes as the forward prenet GEMM, so the recomputed ReLU gate is the forward's gate
      g.epi.flags = EPI_BIAS | EPI_ACC_GATES_AUX | c.colsum();
      g.epi.colsum = gr.prenet_b;
      g.epi.bias = w.prenet_b; g.epi.drop = drop_pe; g.epi.drop_site = 0;
      c.res(g.epi, pl.dh_a, D);
      c.out(g.epi, pl.dh_b, 0, D);
      SPK_TRY(c.run(g));
    }
  }
  SPK_TRY(wgrad(c, "gemm.bwd.prenet_wgrad", Mt, pl.dh_b, D, pl.x0, pl.C, pl.C, gr.prenet_w));
  if (d_mel != nullptr || (rg != nullptr && rg->d_data != nullptr)) {
    // ---- input: dX = dU W_pre (fp32, token-major, into df: dead after the last sublayer backward, and large enough
    // at every plane count, make_plan), then transposed to the [B, mel, T] layout of the input.  dU carries the
    // gradient scale S: alpha = 1 / S.
    float* dx = reinterpret_cast<float*>(c.ptr(pl.df));
    GemmProblem g = dgrad(c, "gemm.bwd.mel_dgrad", pl.dh_b, Mt, D, pl.w_pre, pl.C);
    g.epi.flags = EPI_OUT_F32;
    g.epi.alpha_ptr = gs + 1;
    g.epi.out = dx; g.epi.out_ld = pl.C; g.epi.out_planes = 1;
    SPK_TRY(c.run(g));
    if (rg != nullptr)   // ragged forward: fold every slice back onto the columns of mel->data it was cut from
      SPK_TRY(mel_grad_fold(dx, *rg->mel, segments, S, static_cast<int>(U), rg->d_data, B, pl.C, T, st));
    else
      SPK_TRY(mel_grad_unpack(dx, d_mel, B, pl.C, T, st));
  }
  return 0;
}

}  // namespace spk
