/*
 * spkemb.h -- C ABI of libspkemb.so: the B200 (sm_100a) speaker-embedding hot path.
 *
 * The reference (CODEJIN/Speaker_Embedding_Torch) has no FFI: its hot path is the Python
 * import `from Modules import GE2E, GE2E_Loss` (Train.py:9, Inference.py:14, Trace.py:4) and
 * `from distributed import ...` (Train.py:15).  The entry points below are what a binding for
 * that path calls; `speaker_embedding_torch_b200/_native.py` is the ctypes binding and
 * `speaker_embedding_torch_b200/Modules.py` the drop-in module layer (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every device buffer (inputs, outputs, workspaces, gradients)
 *     is owned by the caller; the library allocates no device memory and keeps no pointers;
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work (no host sync);
 *   - return 0 on success, a negative errno-style code otherwise (SPK_EINVAL bad shape/alignment,
 *     SPK_ENOMEM workspace too small, SPK_EIO CUDA error); text via spk_last_error() (thread-local);
 *   - there is no CPU fallback: without a CUDA device every compute call fails with SPK_EIO.
 */
#ifndef SPKEMB_H_
#define SPKEMB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPK_ABI_VERSION 2
#define SPK_EINVAL (-22)
#define SPK_ENOMEM (-12)
#define SPK_EIO (-5)
#define SPK_MAX_LAYERS 8
#define SPK_PLAN_EXPLICIT (1 << 8)          /* the bits below are valid */
#define SPK_PLAN_PRUNE (1 << 9)             /* "prune_last_layer" */
#define SPK_PLAN_FUSED_INFER_ATTN (1 << 10) /* "fused_inference_attention" */
#define SPK_PLAN_FUSED_TRAIN_ATTN (1 << 11) /* "fused_training_attention" */

int spk_abi_version(void);
const char* spk_last_error(void);

/* Encoder hyper-parameters: the `GE2E:` block + Sound.Mel_Dim of Hyper_Parameters.yaml:3,10-18
 * (read by GE2E.__init__, Modules.py:10-44).  This build supports mel_dim a multiple of 8 in [16, 256], emb 256,
 * heads 4, ffn 1024 (= 4 * emb, hard-wired at Modules.py:29), 1..8 layers, max_pos >= T.  Any other mel_dim is
 * refused (workspace size 0, SPK_EINVAL) with a message that states the rule. */
typedef struct spk_encoder_config {
  int32_t mel_dim, emb, heads, ffn, layers, max_pos;
  float pe_dropout;  /* GE2E.Positional_Encoding.Dropout_Rate */
  float dropout;     /* GE2E.Transformer.Dropout_Rate */
} spk_encoder_config;

/* fp32 device pointers in the reference's state_dict layout (SURVEY.md Appendix A).  The same
 * struct describes the gradients (pe is ignored there; it is a buffer). */
typedef struct spk_layer_params {
  float* in_proj_w;  /* [3*emb, emb]  rows Wq | Wk | Wv */
  float* in_proj_b;  /* [3*emb] */
  float* out_proj_w; /* [emb, emb] */
  float* out_proj_b; /* [emb] */
  float* linear1_w;  /* [ffn, emb] */
  float* linear1_b;  /* [ffn] */
  float* linear2_w;  /* [emb, ffn] */
  float* linear2_b;  /* [emb] */
  float* norm1_w;    /* [emb] */
  float* norm1_b;
  float* norm2_w;
  float* norm2_b;
} spk_layer_params;

typedef struct spk_encoder_params {
  float* prenet_w;   /* [emb, mel_dim(,1)] */
  float* prenet_b;   /* [emb] */
  float* pe_alpha;   /* [1] */
  float* pe;         /* [1, emb, max_pos] buffer */
  spk_layer_params layer[SPK_MAX_LAYERS];
  float* norm_w;     /* final LayerNorm [emb] */
  float* norm_b;
  float* proj_w;     /* [emb, emb(,1)] */
  float* proj_b;     /* [emb] */
} spk_encoder_params;

/* precision (low 8 bits): 1 = fp16 operands (inference), 2 = split-fp16 hi+lo (3 MMAs per product), 3 = hi+mid+lo
 * (6 MMAs, fp32-equivalent forward; the backward pass then reads two of the three planes).
 * Upper bits: the library options that shape the workspace (SPK_PLAN_*).  A caller that wants its backward call to
 * be immune to spk_set_option() between forward and backward passes `precision | spk_plan_flags()` to
 * workspace_bytes / forward / backward alike; without SPK_PLAN_EXPLICIT the process-wide options apply.
 * keep_stash: 1 when spk_encoder_backward will follow (activations of every layer are kept). */
size_t spk_encoder_workspace_bytes(const spk_encoder_config* cfg, int batch, int frames, int samples,
                                   int precision, int keep_stash);

/* GE2E.forward (Modules.py:46-59): mel [batch, mel_dim, frames] fp32 -> dvec [batch/samples, emb] fp32.
 * training != 0 applies the 13 dropout sites with masks that are a pure function of `seed`. */
int spk_encoder_forward(const spk_encoder_config* cfg, const spk_encoder_params* weights, const float* mel,
                        int batch, int frames, int samples, int precision, int training, uint64_t seed,
                        float* dvec, void* workspace, size_t workspace_bytes, int keep_stash, void* stream);

/* The same forward over a strided view of the input, so that the inference collater's work (Inference.py:95-115:
 * five overlapping 64-frame slices cut from a 192-frame window, fp16 patterns upcast to fp32) happens inside the
 * prenet's input load instead of on the host and on PCIe:
 *   slice b = (window u = b / slices_per_window, s = b % slices_per_window) is frames [s*hop, s*hop + frames) of
 *   window u; data is [batch / slices_per_window, mel_dim, window_frames] in `dtype` (0 = fp32, 1 = fp16).
 * slices_per_window == 1, hop == 0, window_frames == frames describes the plain [batch, mel_dim, frames] input. */
typedef struct spk_mel_view {
  const void* data;
  int32_t dtype;             /* 0 = fp32, 1 = fp16 */
  int32_t window_frames;     /* frames per window (row stride of a mel channel) */
  int32_t hop;               /* frames between consecutive slices of a window */
  int32_t slices_per_window; /* >= 1; batch must be a multiple of it */
} spk_mel_view;
int spk_encoder_forward_view(const spk_encoder_config* cfg, const spk_encoder_params* weights, const spk_mel_view* mel,
                             int batch, int frames, int samples, int precision, int training, uint64_t seed,
                             float* dvec, void* workspace, size_t workspace_bytes, int keep_stash, void* stream);

/* The same forward fed by a RAGGED training batch, so that the training collater's work (Datasets.py:9-19 `Correction`,
 * :72-86 `Collater`: one frame count T per batch, every utterance cropped at a random offset or reflect-padded to it)
 * happens inside the prenet's input load:
 *   data   [mel_dim, total_frames] in `dtype`: the utterances' patterns concatenated along time;
 *   table  device int32 [batch][3] = (start column, length, crop offset) per utterance.  length > frames: frames
 *          [offset, offset + frames) are used; otherwise the utterance is reflect-padded (numpy 'reflect') with
 *          floor((frames - length) / 2) frames on the left, the rest on the right, exactly as np.pad does it.
 * The random draws (T and the offsets) stay on the host, in the reference's order, so a seeded run collates the same
 * batch as the reference's numpy collater.  samples is 1 for training batches but any divisor of batch is accepted. */
typedef struct spk_mel_ragged {
  const void* data;
  int32_t dtype;             /* 0 = fp32, 1 = fp16 */
  int64_t total_frames;      /* row stride of a mel channel */
  const int32_t* table;      /* device pointer, [batch][3] */
} spk_mel_ragged;
int spk_encoder_forward_ragged(const spk_encoder_config* cfg, const spk_encoder_params* weights, const spk_mel_ragged* mel,
                               int batch, int frames, int samples, int precision, int training, uint64_t seed,
                               float* dvec, void* workspace, size_t workspace_bytes, int keep_stash, void* stream);

/* Backward of the call above (same cfg/shape/precision/training/seed/workspace).  Accumulates
 * (+=) into `grads`, which the caller zero-initialises; replaces autograd through Modules.py:46-59. */
int spk_encoder_backward(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                         const spk_encoder_params* grads, const float* d_dvec, int batch, int frames,
                         int samples, int precision, int training, uint64_t seed, void* workspace,
                         size_t workspace_bytes, void* stream);

/* Backward of a forward call with optional outputs (same cfg / shape / precision / training / seed / workspace as
 * spk_encoder_backward).
 *   grads  NULL: no parameter gradient is computed (no weight-gradient GEMM, no bias column sums, no LayerNorm /
 *          head / attention bias sums); otherwise accumulated (+=) exactly as spk_encoder_backward does.
 *   d_mel  NULL: none; otherwise fp32 [batch, mel_dim, frames] receives (=) dL/d(slices): the gradient of the
 *          [batch, mel_dim, frames] slice tensor the forward consumed, whichever of plain / view / ragged produced it.
 * At least one of grads / d_mel is non-NULL.  Needs no more workspace than spk_encoder_backward.
 * spk_encoder_backward is this call with d_mel = NULL. */
int spk_encoder_backward_input(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                               const spk_encoder_params* grads, float* d_mel, const float* d_dvec, int batch,
                               int frames, int samples, int precision, int training, uint64_t seed,
                               void* workspace, size_t workspace_bytes, void* stream);

/* Variable-length utterances: mel is a ragged SLICE batch (one table row per slice, see spk_mel_ragged); slices
 * segments[u] .. segments[u+1]-1 form utterance u and their embeddings are averaged with 1 / count; dvec
 * [utterances, emb].  segments: device int32 [utterances + 1], segments[0] = 0, non-decreasing, every utterance at
 * least one slice, segments[utterances] = batch.  The library does not read the device array on the host, so it cannot
 * check this: entries are clamped to [0, batch] (nothing is read or written past the batch), and a slice that no
 * segment covers contributes to no d-vector and receives a zero gradient.
 * segments NULL: batch / utterances slices per utterance, i.e. spk_encoder_forward_ragged at samples = batch /
 * utterances.  Workspace: spk_encoder_workspace_bytes(cfg, batch, frames, 1, precision, keep_stash) with segments,
 * samples = batch / utterances without.  Modules.utterance_slices builds the table and the segments from
 * utterance lengths. */
int spk_encoder_forward_segments(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                                 const spk_mel_ragged* mel, const int32_t* segments, int utterances, int batch,
                                 int frames, int precision, int training, uint64_t seed, float* dvec,
                                 void* workspace, size_t workspace_bytes, int keep_stash, void* stream);
/* Backward of spk_encoder_forward_segments, or of spk_encoder_forward_ragged (segments NULL: batch / utterances
 * slices each), with the same cfg / shape / precision / training / seed / workspace.  grads as in
 * spk_encoder_backward_input.  d_data NULL or fp32 [mel_dim, total_frames]: receives (=) dL/d(mel->data), the
 * adjoint of the crop / reflect-pad; columns no slice reads receive 0.  Slices group by utterance; PRECONDITION: the
 * column spans of different utterances (smallest start .. largest start + length of their slices) do not overlap.
 * Deterministic: no atomics on d_data, two identical calls give bit-identical results.  Argument errors (utterances
 * < 1, batch < utterances, segments NULL and batch % utterances != 0, grads and d_data both NULL, missing data /
 * table, bad dtype) return SPK_EINVAL before any CUDA call. */
int spk_encoder_backward_segments(const spk_encoder_config* cfg, const spk_encoder_params* weights,
                                  const spk_encoder_params* grads, const spk_mel_ragged* mel,
                                  const int32_t* segments, int utterances, float* d_data, const float* d_dvec,
                                  int batch, int frames, int precision, int training, uint64_t seed,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* Test aid: text table "name byte_offset plane_stride" of the workspace buffers (returns bytes written). */
int spk_encoder_debug_layout(const spk_encoder_config* cfg, int batch, int frames, int samples, int precision,
                             int keep_stash, char* buf, size_t cap);

/* Mel front-end on the device (meldataset.py:73-96 `mel_spectrogram`, center = False; the step in front of the encoder
 * in Inference.py:59-85): audio [batch, samples] fp32 in [-1, 1] -> log-mel [batch, n_mels, frames] (fp32, or fp16 --
 * the format the reference stores its patterns in -- when out_fp16 != 0), frames = spk_mel_frames(samples, n_fft, hop).
 * Reflect padding by (n_fft - hop) / 2, periodic Hann window of `win` samples centred in n_fft, magnitude
 * sqrt(re^2 + im^2 + 1e-9), log(max(., 1e-5)).  basis: device fp32 [n_mels, n_fft / 2 + 1] (librosa.filters.mel);
 * ranges: device int32 [n_mels][2] = [first, last + 1) non-zero bin of every filter.  n_fft in {512, 1024, 2048}. */
int spk_mel_frames(int64_t samples, int n_fft, int hop);
int spk_mel_spectrogram(const float* audio, int batch, int64_t samples, int n_fft, int hop, int win, const float* basis,
                        const int32_t* ranges, int n_mels, void* out, int out_fp16, void* stream);

/* Backward of spk_mel_spectrogram with respect to the audio (the mel basis and the window are constants): for
 * d_mel = dL/d(log-mel), fp32 [batch, n_mels, frames], d_audio fp32 [batch, samples] receives (=) dL/d(audio).
 * The forward is recomputed from `audio`, so it needs to keep nothing.  Same arguments as the forward, plus
 * bin_ranges: device int32 [n_fft / 2 + 1][2] = [first, last + 1) filter with a non-zero weight at every bin.
 * Deterministic: no atomics, two identical calls give bit-identical d_audio.  hop > n_fft (negative padding) is
 * rejected.  workspace: device memory of at least spk_mel_backward_workspace_bytes(batch, samples, n_fft, hop)
 * bytes (one windowed frame gradient per frame, batch * frames * n_fft fp32), 16-byte aligned; that function
 * returns 0 for a shape the backward rejects.  Argument errors return SPK_EINVAL before any CUDA call. */
size_t spk_mel_backward_workspace_bytes(int batch, int64_t samples, int n_fft, int hop);
int spk_mel_spectrogram_backward(const float* audio, const float* d_mel, int batch, int64_t samples, int n_fft, int hop,
                                 int win, const float* basis, const int32_t* ranges, const int32_t* bin_ranges,
                                 int n_mels, float* d_audio, void* workspace, size_t workspace_bytes, void* stream);

/* Test aid: the dropout keep-scale (0 or 1 / (1 - p_q), p_q = round(p * 2^16) / 2^16) of elements
 * [8 * idx8_begin, 8 * (idx8_begin + n8)) of dropout site `site` under `seed` -- the pure function of
 * (seed, site, element) that the forward and backward kernels evaluate.  Sites: 0 = positional encoding
 * (Modules.py:103; element = token * emb + channel); layer l: 1 + 4l attention probabilities (element = ((slice *
 * heads + head) * frames + query) * frames_padded_to_8 + key; pruned last layer: (slice * heads + head) *
 * frames_padded_to_8 + key), 2 + 4l dropout1, 3 + 4l FFN inner (element = token * ffn + unit), 4 + 4l dropout2
 * (torch TransformerEncoderLayer; element = token * emb + channel; in the pruned last layer `token` = slice). */
int spk_dropout_keep(uint64_t seed, float p, uint32_t site, uint64_t idx8_begin, int64_t n8, float* out, void* stream);

/* GE2E_Loss.forward + backward (Modules.py:121-156) as one fused kernel.
 * emb [speakers*per_speaker, dim] fp32, speaker-major rows; weight/bias: device pointers to the
 * 0-dim parameters (logits = weight * cos - bias).  d_emb == NULL -> loss only. */
size_t spk_ge2e_workspace_bytes(int speakers, int per_speaker);
int spk_ge2e_loss(const float* emb, int speakers, int per_speaker, int dim, const float* weight,
                  const float* bias, float* loss, float* d_emb, float* d_weight, float* d_bias,
                  void* workspace, size_t workspace_bytes, void* stream);

/* The GE2E paper's loss variants (Wan et al., 2018).  `mode` ORs one loss with one centroid rule:
 *   SPK_GE2E_SOFTMAX    mean over rows of logsumexp_k z_ik - z_i,own (eq. 6; spk_ge2e_loss)
 *   SPK_GE2E_CONTRAST   mean over rows of 1 - sigmoid(z_i,own) + sigmoid(max_{k != own} z_ik) (eq. 7); ties in the
 *                       maximum go to the lowest speaker index.  Needs speakers >= 2.
 *   SPK_GE2E_EXCLUSIVE  the own-speaker column of row i uses the centroid of the speaker's other rows (eq. 8); every
 *                       other column keeps the inclusive centroid (eq. 9).  Needs per_speaker >= 2.
 * Mode 0 runs the kernels of spk_ge2e_loss, and spk_ge2e_workspace_bytes_ex(n, m, 0) equals
 * spk_ge2e_workspace_bytes(n, m).  Unknown mode bits and the shape limits above return SPK_EINVAL (workspace query: 0)
 * before any CUDA call.  With SPK_GE2E_CONTRAST, d_bias is no longer zero. */
#define SPK_GE2E_SOFTMAX 0
#define SPK_GE2E_CONTRAST 1
#define SPK_GE2E_EXCLUSIVE (1 << 8)
size_t spk_ge2e_workspace_bytes_ex(int speakers, int per_speaker, int mode);
int spk_ge2e_loss_ex(const float* emb, int speakers, int per_speaker, int dim, int mode, const float* weight,
                     const float* bias, float* loss, float* d_emb, float* d_weight, float* d_bias,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Fused optimiser over a list of tensors (replaces Radam.py:25-90 / torch AdamW + the
 * clip_grad_norm_ site Train.py:154-159).  One launch computes the global grad norm, one applies
 * clip + update.  kind: 0 = RAdam (Radam.py), 1 = AdamW.  step is 1-based.
 * The norm is reduced deterministically (per-block partials added in a fixed order), so data-parallel ranks that hold
 * bit-identical gradients compute bit-identical clip coefficients and weights.
 * More than 64 tensors, or parameter groups / step counts that need separate launches but ONE global norm
 * (clip_grad_norm_ is global): call phase 1 for every chunk c of n (norm partials), then phase 2 for every chunk
 * (update with the norm of all n chunks).  phase 0 = both for a single chunk (chunk 0 of 1).
 * norm_scratch: device fp32 [SPK_OPTIM_SCRATCH_FLOATS(n)]; element 0 receives the squared global norm. */
#define SPK_OPTIM_MAX_CHUNKS 16
#define SPK_OPTIM_SCRATCH_FLOATS(nchunks) (1 + 296 * (nchunks))
typedef struct spk_optim_tensors {
  int32_t count;
  float* param[64];
  float* grad[64];
  float* exp_avg[64];
  float* exp_avg_sq[64];
  int64_t numel[64];
} spk_optim_tensors;
int spk_optim_step(const spk_optim_tensors* tensors, int kind, int64_t step, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float max_grad_norm, float grad_scale,
                   float* norm_scratch, int phase, int chunk, int nchunks, void* stream);

/* Diagnostic / benchmark entry: one tensor-core GEMM on split-fp16 operands,
 * D[M,N] = A * B^T (+ bias, ReLU), used by the GEMM parity tests and the roofline bench. */
typedef struct spk_gemm_desc {
  const void* a; int64_t a_plane_stride, a_rows, a_cols, a_ld, a_sb0, a_sb1; int32_t a_mn;
  const void* b; int64_t b_plane_stride, b_rows, b_cols, b_ld, b_sb0, b_sb1; int32_t b_mn;
  int32_t planes, m, n, k, nb0, nb1, ksplit, block_n;
  uint32_t flags;      /* bit0 bias, bit1 relu, bit8 fp32 out, bit9 fp32 atomic out */
  float alpha;
  const float* bias;
  void* out; int64_t out_plane_stride, out_ld, out_sb0, out_sb1; int32_t out_planes;
} spk_gemm_desc;
int spk_gemm(const spk_gemm_desc* desc, void* stream);

/* fp32 [n] -> split-fp16 planes (hi at dst, lo at dst + plane_stride elements). */
int spk_split_pack(const float* src, void* dst, int64_t plane_stride, int planes, int64_t n, void* stream);

int spk_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Library options (all default 1):
 *   "prune_last_layer"           run the last encoder layer only for the t = 0 query row the d-vector head consumes
 *                                (exact; K and V are still projected for every frame);
 *   "fused_inference_attention"  one tcgen05 kernel for QK^T / softmax / PV in the one-plane inference path (T <= 256);
 *   "gemm_cta_pairs"             multi-plane GEMMs on CTA pairs (tcgen05.mma.cta_group::2); 0 = single-CTA kernel
 *                                (bit-identical results, used by the tests as the cross-check). */
int spk_set_option(const char* name, int value);
/* Snapshot of the options above as SPK_PLAN_* bits (SPK_PLAN_EXPLICIT set), to be OR-ed into `precision`. */
int spk_plan_flags(void);

/* Diagnostics: while a device buffer is registered, CTA 0 of the fused attention backward kernel records the SM clock
 * at the phase boundaries of its first units into it (8 uint64 slots per (key tile, query tile) unit; see
 * csrc/attn_train.cu).  NULL unregisters.  The caller owns the buffer and keeps it alive while registered. */
int spk_set_debug_buffer(void* device_buffer, size_t bytes);

/* Launch profiler (used by bench.py for the per-kernel roofline): when enabled every launcher brackets
 * its kernel with CUDA events on the launching stream.  spk_prof_report synchronises those events,
 * writes one text line per kernel tag -- "tag launches total_ms algorithmic_flops algorithmic_bytes" --
 * into buf, clears the records and returns the number of bytes written. */
int spk_prof_enable(int on);
int spk_prof_report(char* buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* SPKEMB_H_ */
