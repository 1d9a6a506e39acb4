// extern "C" surface of libspkemb.so (declared in include/spkemb.h).  No C++ exception crosses it.
#include "../../include/spkemb.h"
#include "encoder.h"
#include "ge2e.h"
#include "gemm.h"
#include "melspec.h"
#include "optim.h"
#include "rowops.h"

using namespace spk;

namespace spk {
void attn_train_set_timeline(void* buf, size_t bytes);   // attn_train.cu
void attn_train_set_fwd_two(int on);                        // attn_train.cu
}

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

int spk_abi_version(void) { return SPK_ABI_VERSION; }
const char* spk_last_error(void) { return last_error_buf(); }

size_t spk_encoder_workspace_bytes(const spk_encoder_config* cfg, int batch, int frames, int samples, int precision,
                                   int keep_stash) {
  if (!cfg) { set_error("null config"); return 0; }
  return encoder_workspace_bytes(*cfg, batch, frames, samples, precision, keep_stash);
}

int spk_encoder_forward(const spk_encoder_config* cfg, const spk_encoder_params* weights, const float* mel, int batch,
                        int frames, int samples, int precision, int training, uint64_t seed, float* dvec,
                        void* workspace, size_t workspace_bytes, int keep_stash, void* stream) {
  SPK_CHECK(cfg && weights && mel && dvec && workspace, "spk_encoder_forward: null argument");
  spk_mel_view view;
  view.data = mel; view.dtype = 0; view.window_frames = frames; view.hop = 0; view.slices_per_window = 1;
  return encoder_forward(*cfg, *weights, &view, nullptr, batch, frames, samples, precision, training, seed, dvec,
                         workspace, workspace_bytes, keep_stash, as_stream(stream));
}

int spk_encoder_forward_view(const spk_encoder_config* cfg, const spk_encoder_params* weights, const spk_mel_view* mel,
                             int batch, int frames, int samples, int precision, int training, uint64_t seed,
                             float* dvec, void* workspace, size_t workspace_bytes, int keep_stash, void* stream) {
  SPK_CHECK(cfg && weights && mel && mel->data && dvec && workspace, "spk_encoder_forward_view: null argument");
  return encoder_forward(*cfg, *weights, mel, nullptr, batch, frames, samples, precision, training, seed, dvec,
                         workspace, workspace_bytes, keep_stash, as_stream(stream));
}

int spk_encoder_forward_ragged(const spk_encoder_config* cfg, const spk_encoder_params* weights, const spk_mel_ragged* mel,
                               int batch, int frames, int samples, int precision, int training, uint64_t seed,
                               float* dvec, void* workspace, size_t workspace_bytes, int keep_stash, void* stream) {
  SPK_CHECK(cfg && weights && mel && mel->data && mel->table && dvec && workspace,
            "spk_encoder_forward_ragged: null argument");
  return encoder_forward(*cfg, *weights, nullptr, mel, batch, frames, samples, precision, training, seed, dvec,
                         workspace, workspace_bytes, keep_stash, as_stream(stream));
}

// Shape checks shared by the two segmented entry points; host-only, before any CUDA call.
static int check_segments(const char* fn, const spk_mel_ragged* mel, const int32_t* segments, int utterances,
                          int batch) {
  SPK_CHECK(mel->data && mel->table && (mel->dtype == 0 || mel->dtype == 1) && mel->total_frames > 0,
            "%s: ragged mel needs data, table, total_frames > 0 and dtype 0 (fp32) / 1 (fp16)", fn);
  SPK_CHECK(utterances >= 1 && batch >= utterances, "%s: need 1 <= utterances <= batch (got %d, %d)", fn, utterances,
            batch);
  SPK_CHECK(segments || batch % utterances == 0, "%s: segments is NULL and batch %d is not a multiple of utterances %d",
            fn, batch, utterances);
  return 0;
}

int spk_encoder_forward_segments(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                                 const spk_mel_ragged* mel, const int32_t* segments, int utterances, int batch,
                                 int frames, int precision, int training, uint64_t seed, float* dvec, void* workspace,
                                 size_t workspace_bytes, int keep_stash, void* stream) {
  SPK_CHECK(cfg && weights && mel && dvec && workspace, "spk_encoder_forward_segments: null argument");
  SPK_TRY(check_segments("spk_encoder_forward_segments", mel, segments, utterances, batch));
  const int samples = segments ? 1 : batch / utterances;
  return encoder_forward(*cfg, *weights, nullptr, mel, batch, frames, samples, precision, training, seed, dvec,
                         workspace, workspace_bytes, keep_stash, as_stream(stream), segments, utterances);
}

int spk_encoder_backward_segments(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                                  const spk_encoder_params* grads, const spk_mel_ragged* mel, const int32_t* segments,
                                  int utterances, float* d_data, const float* d_dvec, int batch, int frames,
                                  int precision, int training, uint64_t seed, void* workspace, size_t workspace_bytes,
                                  void* stream) {
  SPK_CHECK(cfg && weights && mel && d_dvec && workspace, "spk_encoder_backward_segments: null argument");
  SPK_CHECK(grads || d_data, "spk_encoder_backward_segments: grads and d_data are both NULL (nothing to compute)");
  SPK_TRY(check_segments("spk_encoder_backward_segments", mel, segments, utterances, batch));
  const int samples = segments ? 1 : batch / utterances;
  RaggedGrad rg{mel, segments, utterances, d_data};
  return encoder_backward(*cfg, *weights, grads, nullptr, d_dvec, batch, frames, samples, precision, training, seed,
                          workspace, workspace_bytes, as_stream(stream), &rg);
}

int spk_encoder_backward(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                         const spk_encoder_params* grads, const float* d_dvec, int batch, int frames, int samples,
                         int precision, int training, uint64_t seed, void* workspace, size_t workspace_bytes,
                         void* stream) {
  SPK_CHECK(cfg && weights && grads && d_dvec && workspace, "spk_encoder_backward: null argument");
  return encoder_backward(*cfg, *weights, grads, nullptr, d_dvec, batch, frames, samples, precision, training, seed,
                          workspace, workspace_bytes, as_stream(stream));
}

int spk_encoder_backward_input(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                               const spk_encoder_params* grads, float* d_mel, const float* d_dvec, int batch,
                               int frames, int samples, int precision, int training, uint64_t seed,
                               void* workspace, size_t workspace_bytes, void* stream) {
  SPK_CHECK(cfg && weights && d_dvec && workspace, "spk_encoder_backward_input: null argument");
  SPK_CHECK(grads || d_mel, "spk_encoder_backward_input: grads and d_mel are both NULL (nothing to compute)");
  return encoder_backward(*cfg, *weights, grads, d_mel, d_dvec, batch, frames, samples, precision, training, seed,
                          workspace, workspace_bytes, as_stream(stream));
}

int spk_encoder_debug_layout(const spk_encoder_config* cfg, int batch, int frames, int samples, int precision,
                              int keep_stash, char* buf, size_t cap) {
  SPK_CHECK(cfg && buf, "spk_encoder_debug_layout: null argument");
  return encoder_debug_layout(*cfg, batch, frames, samples, precision, keep_stash, buf, cap);
}

int spk_mel_frames(int64_t samples, int n_fft, int hop) {
  if (hop < 1 || n_fft < 1) return SPK_EINVAL;
  const int64_t padded = samples + 2 * ((n_fft - hop) / 2);
  if (padded < n_fft) return 0;
  return static_cast<int>(1 + (padded - n_fft) / hop);
}

int spk_mel_spectrogram(const float* audio, int batch, int64_t samples, int n_fft, int hop, int win, const float* basis,
                        const int32_t* ranges, int n_mels, void* out, int out_fp16, void* stream) {
  const int r = mel_spectrogram(audio, batch, samples, n_fft, hop, win, basis, ranges, n_mels, out, out_fp16,
                                as_stream(stream));
  return r < 0 ? r : 0;
}

size_t spk_mel_backward_workspace_bytes(int batch, int64_t samples, int n_fft, int hop) {
  return mel_backward_workspace_bytes(batch, samples, n_fft, hop);
}

int spk_mel_spectrogram_backward(const float* audio, const float* d_mel, int batch, int64_t samples, int n_fft, int hop,
                                 int win, const float* basis, const int32_t* ranges, const int32_t* bin_ranges,
                                 int n_mels, float* d_audio, void* workspace, size_t workspace_bytes, void* stream) {
  return mel_spectrogram_backward(audio, d_mel, batch, samples, n_fft, hop, win, basis, ranges, bin_ranges, n_mels,
                                  d_audio, workspace, workspace_bytes, as_stream(stream));
}

int spk_dropout_keep(uint64_t seed, float p, uint32_t site, uint64_t idx8_begin, int64_t n8, float* out, void* stream) {
  return dropout_keep(seed, p, site, idx8_begin, n8, out, as_stream(stream));
}

size_t spk_ge2e_workspace_bytes(int speakers, int per_speaker) { return ge2e_workspace_bytes(speakers, per_speaker); }

int spk_ge2e_loss(const float* emb, int speakers, int per_speaker, int dim, const float* weight, const float* bias,
                  float* loss, float* d_emb, float* d_weight, float* d_bias, void* workspace, size_t workspace_bytes,
                  void* stream) {
  SPK_CHECK(emb && weight && bias && loss && workspace, "spk_ge2e_loss: null argument");
  SPK_CHECK(d_emb == nullptr || (d_weight && d_bias), "spk_ge2e_loss: d_weight/d_bias required with d_emb");
  return ge2e_fused(emb, speakers, per_speaker, dim, weight, bias, loss, d_emb, d_weight, d_bias, workspace,
                    workspace_bytes, as_stream(stream));
}

static_assert(SPK_GE2E_CONTRAST == GE2E_CONTRAST && SPK_GE2E_EXCLUSIVE == GE2E_EXCLUSIVE, "GE2E mode bits");

// Mode checks shared by the two variant entry points; host-only.
static int check_ge2e_mode(const char* fn, int speakers, int per_speaker, int mode) {
  SPK_CHECK((mode & ~GE2E_MODE_BITS) == 0, "%s: unknown mode bits 0x%x (SPK_GE2E_CONTRAST | SPK_GE2E_EXCLUSIVE)", fn,
            mode & ~GE2E_MODE_BITS);
  SPK_CHECK(!(mode & GE2E_EXCLUSIVE) || per_speaker >= 2,
            "%s: exclusive centroids need at least 2 utterances per speaker (got %d)", fn, per_speaker);
  SPK_CHECK(!(mode & GE2E_CONTRAST) || speakers >= 2, "%s: the contrast loss needs at least 2 speakers (got %d)", fn,
            speakers);
  return 0;
}

size_t spk_ge2e_workspace_bytes_ex(int speakers, int per_speaker, int mode) {
  if (check_ge2e_mode("spk_ge2e_workspace_bytes_ex", speakers, per_speaker, mode) != 0) return 0;
  return ge2e_workspace_bytes(speakers, per_speaker, mode);
}

int spk_ge2e_loss_ex(const float* emb, int speakers, int per_speaker, int dim, int mode, const float* weight,
                     const float* bias, float* loss, float* d_emb, float* d_weight, float* d_bias, void* workspace,
                     size_t workspace_bytes, void* stream) {
  SPK_CHECK(emb && weight && bias && loss && workspace, "spk_ge2e_loss_ex: null argument");
  SPK_CHECK(d_emb == nullptr || (d_weight && d_bias), "spk_ge2e_loss_ex: d_weight/d_bias required with d_emb");
  SPK_TRY(check_ge2e_mode("spk_ge2e_loss_ex", speakers, per_speaker, mode));
  return ge2e_fused(emb, speakers, per_speaker, dim, weight, bias, loss, d_emb, d_weight, d_bias, workspace,
                    workspace_bytes, as_stream(stream), mode);
}

int spk_optim_step(const spk_optim_tensors* tensors, int kind, int64_t step, float lr, float beta1, float beta2,
                   float eps, float weight_decay, float max_grad_norm, float grad_scale, float* norm_scratch,
                   int phase, int chunk, int nchunks, void* stream) {
  SPK_CHECK(tensors && norm_scratch, "spk_optim_step: null argument");
  return optim_step(*tensors, kind, step, lr, beta1, beta2, eps, weight_decay, max_grad_norm, grad_scale, norm_scratch,
                    phase, chunk, nchunks, as_stream(stream));
}

int spk_gemm(const spk_gemm_desc* d, void* stream) {
  SPK_CHECK(d != nullptr, "spk_gemm: null descriptor");
  GemmProblem g;
  g.A.base = d->a; g.A.plane_stride = d->a_plane_stride; g.A.rows = d->a_rows; g.A.cols = d->a_cols; g.A.ld = d->a_ld;
  g.A.sb0 = d->a_sb0; g.A.sb1 = d->a_sb1; g.a_mn = d->a_mn != 0;
  g.B.base = d->b; g.B.plane_stride = d->b_plane_stride; g.B.rows = d->b_rows; g.B.cols = d->b_cols; g.B.ld = d->b_ld;
  g.B.sb0 = d->b_sb0; g.B.sb1 = d->b_sb1; g.b_mn = d->b_mn != 0;
  g.planes = d->planes; g.M = d->m; g.N = d->n; g.K = d->k; g.nb0 = d->nb0 < 1 ? 1 : d->nb0; g.nb1 = d->nb1 < 1 ? 1 : d->nb1;
  g.ksplit = d->ksplit < 1 ? 1 : d->ksplit; g.block_n = d->block_n;
  g.epi.flags = d->flags & (EPI_BIAS | EPI_RELU | EPI_OUT_F32 | EPI_OUT_ATOMIC);
  g.epi.alpha = d->alpha; g.epi.bias = d->bias;
  g.epi.out = d->out; g.epi.out_plane_stride = d->out_plane_stride; g.epi.out_ld = d->out_ld;
  g.epi.out_sb0 = d->out_sb0; g.epi.out_sb1 = d->out_sb1; g.epi.out_planes = d->out_planes < 1 ? 1 : d->out_planes;
  return gemm_run(g, as_stream(stream));
}

int spk_split_pack(const float* src, void* dst, int64_t plane_stride, int planes, int64_t n, void* stream) {
  SPK_CHECK(src && dst && n >= 0 && planes >= 1 && planes <= 3, "spk_split_pack: bad argument");
  PackTable tab;
  tab.count = 1;
  tab.seg[0].src = src; tab.seg[0].dst_off = 0; tab.seg[0].n = n;
  return pack_weights(tab, dst, plane_stride, planes, as_stream(stream));
}

int spk_set_option(const char* name, int value) {
  SPK_CHECK(name != nullptr, "spk_set_option: null name");
  if (strcmp(name, "prune_last_layer") == 0) { encoder_set_prune(value != 0); return 0; }
  if (strcmp(name, "training_attention_two_ctas") == 0) { attn_train_set_fwd_two(value); return 0; }
  if (strcmp(name, "fused_inference_attention") == 0) { encoder_set_fused_attn(value != 0); return 0; }
  if (strcmp(name, "inference_attention_two_ctas") == 0) { encoder_set_infer_attn_two(value); return 0; }
  if (strcmp(name, "fused_layernorm") == 0) { encoder_set_fuse_ln(value); return 0; }
  if (strcmp(name, "fused_training_attention") == 0) { encoder_set_fused_train_attn(value != 0); return 0; }
  if (strcmp(name, "grad_scale_log2") == 0) { encoder_set_grad_scale_log2(value); return 0; }
  if (strcmp(name, "ge2e_dependent_launch") == 0) { ge2e_set_pdl(value); return 0; }
  if (strcmp(name, "gemm_dependent_launch") == 0) { gemm_set_dependent_launch(value); return 0; }
  if (strcmp(name, "gemm_cta_pairs") == 0) { gemm_set_cta_pairs(value != 0); return 0; }
  set_error("spk_set_option: unknown option '%s'", name);
  return SPK_EINVAL;
}

int spk_plan_flags(void) { return encoder_plan_flags(); }

int spk_set_debug_buffer(void* device_buffer, size_t bytes) {
  attn_train_set_timeline(device_buffer, device_buffer ? bytes : 0);
  return 0;
}

int spk_prof_enable(int on) { prof_set(on != 0); return 0; }
int spk_prof_report(char* buf, size_t cap) { return prof_report(buf, cap); }

int spk_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  SPK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  SPK_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return 0;
}

}  // extern "C"
