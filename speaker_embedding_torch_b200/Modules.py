"""Drop-in replacement for the reference's ``Modules.py`` (GE2E encoder + GE2E loss) on B200.

Same public surface as /root/reference/Modules.py:
  * ``GE2E(hyper_parameters)``; ``forward(features[B*S, Mel_Dim, T], samples=1) -> [B, Embedding_Size]``
    (Modules.py:5-59), same sub-module / parameter names, ``state_dict`` keys and shapes
    (SURVEY.md Appendix A), so reference checkpoints load with ``strict=True`` and vice versa;
  * ``GE2E_Loss(init_weight=10.0, init_bias=-5.0, loss_method="softmax", centroids="inclusive")``;
    ``forward(embeddings[N*M, D], pattern_per_speaker)`` -> 0-dim loss (Modules.py:112-156), ``weight`` / ``bias`` 0-dim parameters;
  * ``Conv1d`` and ``Positional_Encoding`` helper modules (Modules.py:61-109).

The modules only OWN parameters; the arithmetic runs in libspkemb.so (hand-written sm_100a
kernels behind the C ABI of include/spkemb.h).  There is no CPU or eager-PyTorch fallback:
CPU inputs raise ``RuntimeError``.

Precision: every tensor that feeds the tensor cores is stored as fp16 "planes" (csrc/common.cuh).  Inference uses
one plane (``eval_precision = 1``: fp16 operands, fp32 accumulate); when gradients are required forward and backward
run on two planes (``train_precision = 2``: hi + lo = an fp32-class 22-bit mantissa, three MMAs per product).  Two
planes matter for the GRADIENTS: a forward error delta flips ~delta of the ReLU gates and each flip is an O(1)
gradient error (DESIGN.md, "Precision"); two bf16 planes (16 bits) were not enough, two fp16 planes are.
``train_precision = 3`` (a third plane, six MMAs) is kept as a cross-check.
"""
import ctypes
import math
from argparse import Namespace

import torch

from . import _native as N

__all__ = ["GE2E", "GE2E_Loss", "Conv1d", "Positional_Encoding", "utterance_slices"]


# ------------------------------------------------------------------------------------------------
# parameter containers (same constructor signatures and initialisation as the reference)

class Conv1d(torch.nn.Conv1d):
    """k=1 convolution == per-frame linear layer; weight init by gain name (Modules.py:61-72)."""

    def __init__(self, w_init_gain="relu", *args, **kwargs):
        self.w_init_gain = w_init_gain
        super().__init__(*args, **kwargs)

    def reset_parameters(self):
        gain_name = self.w_init_gain
        if gain_name in ("relu", "leaky_relu"):
            torch.nn.init.kaiming_uniform_(self.weight, nonlinearity=gain_name)
        else:
            torch.nn.init.xavier_uniform_(self.weight, gain=torch.nn.init.calculate_gain(gain_name))
        if self.bias is not None:
            torch.nn.init.zeros_(self.bias)


def _sinusoid_table(max_position, embedding_size):
    """[1, embedding_size, max_position] table of Modules.py:86-92 (sin on even, cos on odd channels)."""
    position = torch.arange(0, max_position, dtype=torch.float).unsqueeze(1)
    freq = torch.exp(torch.arange(0, embedding_size, 2).float() * (-math.log(10000.0) / embedding_size))
    table = torch.zeros(max_position, embedding_size)
    table[:, 0::2] = torch.sin(position * freq)
    table[:, 1::2] = torch.cos(position * freq)
    return table.t().unsqueeze(0).contiguous()


class Positional_Encoding(torch.nn.Module):
    """Holds ``pe`` (buffer) and ``alpha`` (parameter); x + alpha * pe[:, :, :T] then dropout
    (Modules.py:76-109).  Inside ``GE2E`` this is fused into the prenet GEMM epilogue; standalone
    calls are not part of the accelerated path and are rejected."""

    def __init__(self, max_position: int, embedding_size: int, dropout_rate: float):
        super().__init__()
        self.dropout = torch.nn.Dropout(p=dropout_rate)
        self.register_buffer("pe", _sinusoid_table(max_position, embedding_size))
        self.alpha = torch.nn.Parameter(torch.ones(1), requires_grad=True)

    def forward(self, x):
        raise RuntimeError("Positional_Encoding is fused into GE2E.forward on this backend; call the encoder")


# ------------------------------------------------------------------------------------------------
# encoder

_PARAM_ORDER_HEAD = ("prenet.weight", "prenet.bias", "positional_encoding.alpha")
_LAYER_KEYS = (("self_attn.in_proj_weight", "in_proj_w"), ("self_attn.in_proj_bias", "in_proj_b"),
               ("self_attn.out_proj.weight", "out_proj_w"), ("self_attn.out_proj.bias", "out_proj_b"),
               ("linear1.weight", "linear1_w"), ("linear1.bias", "linear1_b"),
               ("linear2.weight", "linear2_w"), ("linear2.bias", "linear2_b"),
               ("norm1.weight", "norm1_w"), ("norm1.bias", "norm1_b"),
               ("norm2.weight", "norm2_w"), ("norm2.bias", "norm2_b"))


def _fill_params(struct, tensors, pe, layers):
    """tensors: dict name -> CUDA fp32 contiguous tensor (parameters or gradient views)."""
    struct.prenet_w = tensors["prenet.weight"].data_ptr()
    struct.prenet_b = tensors["prenet.bias"].data_ptr()
    struct.pe_alpha = tensors["positional_encoding.alpha"].data_ptr()
    struct.pe = pe.data_ptr() if pe is not None else 0
    for l in range(layers):
        for key, field in _LAYER_KEYS:
            setattr(struct.layer[l], field, tensors["transformer.layers.%d.%s" % (l, key)].data_ptr())
    struct.norm_w = tensors["transformer.norm.weight"].data_ptr()
    struct.norm_b = tensors["transformer.norm.bias"].data_ptr()
    struct.proj_w = tensors["projection.weight"].data_ptr()
    struct.proj_b = tensors["projection.bias"].data_ptr()
    return struct


def _workspace(cfg, batch, frames, samples, precision, keep, device):
    nbytes = N.lib().spk_encoder_workspace_bytes(ctypes.byref(cfg), batch, frames, samples, precision, keep)
    if nbytes == 0:
        N.check(-22, "spk_encoder_workspace_bytes")
    return torch.empty(nbytes + 256, dtype=torch.uint8, device=device), nbytes


def _aligned_ptr(ws):
    base = ws.data_ptr()
    return ctypes.c_void_p((base + 255) // 256 * 256)


def _run_forward(cfg, names, params, pe, features, samples, precision, training, seed, keep, slicing=None,
                 return_ragged=False):
    """One spk_encoder_forward_view call.  ``features`` is ``[Batch*Samples, Mel_Dim, Time]`` (fp32 or fp16: the
    reference stores its patterns as fp16, the upcast happens in the prenet load), or -- with
    ``slicing = (frame_length, hop, slices_per_window)`` -- un-sliced windows ``[Utterances, Mel_Dim, L]`` whose
    overlapping slices are cut by the same load.  ``return_ragged``: also return the RaggedMel the call read
    (contiguous data, int32 table / segments), or None for a dense input."""
    from .Datasets import RaggedMel
    ragged = features if isinstance(features, RaggedMel) else None
    if ragged is not None:            # training batch collated on the device (Datasets.Collater)
        N.require_cuda(ragged.data, "features")
        N.require_cuda(ragged.table, "features.table")
        data = ragged.data if ragged.data.dtype in (torch.float32, torch.float16) else ragged.data.float()
        segments = ragged.segments
        if segments is not None:
            N.require_cuda(segments, "features.segments")
            segments = segments.to(torch.int32).contiguous()
            if samples != 1:
                raise RuntimeError("a RaggedMel with segments gives one d-vector per segment: samples must be 1")
        ragged = RaggedMel(data.contiguous(), ragged.table.to(torch.int32).contiguous(), ragged.frames, segments,
                           _checked=True)
        features = ragged.data            # device / dtype bookkeeping below
        if slicing is not None or ragged.data.dim() != 2 or ragged.data.size(0) != cfg.mel_dim:
            raise RuntimeError("ragged features must be [Mel_Dim=%d, total_frames]" % cfg.mel_dim)
        # (the table was validated on the host when the RaggedMel was built; no device -> host sync here)
    else:
        N.require_cuda(features, "features")
        if features.dtype not in (torch.float32, torch.float16):
            features = features.float()
        features = features.contiguous()
    if ragged is not None:
        pass
    elif features.dim() != 3 or features.size(1) != cfg.mel_dim:
        raise RuntimeError("features must be [Batch*Samples, Mel_Dim=%d, Time], got %s"
                           % (cfg.mel_dim, tuple(features.shape)))
    if ragged is not None:
        batch, frames = ragged.table.size(0), ragged.frames
        if ragged.segments is not None and not 1 <= ragged.utterances <= batch:
            raise RuntimeError("RaggedMel: %d segments for %d slices" % (ragged.utterances, batch))
    elif slicing is None:
        batch, _, frames = features.shape
        window, hop, spw = frames, 0, 1
    else:
        frames, hop, spw = (int(v) for v in slicing)
        window = features.size(2)
        batch = features.size(0) * spw
        if spw < 1 or hop < 0 or (spw - 1) * hop + frames > window:
            raise RuntimeError("invalid slicing: %d slices of %d frames at hop %d from a %d-frame window"
                               % (spw, frames, hop, window))
    if samples < 1 or batch % samples != 0:
        raise RuntimeError("shape '[-1, %d, ...]' is invalid for a batch of %d slices" % (samples, batch))
    tensors = {}
    for n, p in zip(names, params):
        N.require_cuda(p, n)
        if p.dtype != torch.float32 or not p.is_contiguous():
            raise RuntimeError("parameter %s must be contiguous fp32" % n)
        tensors[n] = p
    if precision < 256:
        precision |= N.plan_flags()          # the backward call receives the same bits through ctx.meta
    with torch.cuda.device(features.device):
        weights = _fill_params(N.EncoderParams(), tensors, pe, cfg.layers)
        ws, nbytes = _workspace(cfg, batch, frames, samples, precision, int(keep), features.device)
        dvecs = batch // samples if ragged is None or ragged.segments is None else ragged.utterances
        dvec = torch.empty((dvecs, cfg.emb), dtype=torch.float32, device=features.device)
        if ragged is not None and ragged.segments is not None:      # variable slice counts per utterance
            N.check(N.lib().spk_encoder_forward_segments(ctypes.byref(cfg), ctypes.byref(weights),
                                                         ctypes.byref(_mel_ragged(ragged)), N.ptr(ragged.segments),
                                                         ragged.utterances, batch, frames, precision, int(training),
                                                         ctypes.c_uint64(seed), N.ptr(dvec), _aligned_ptr(ws), nbytes,
                                                         int(keep), N.stream_ptr(features.device)),
                    "spk_encoder_forward_segments")
        elif ragged is not None:
            view = _mel_ragged(ragged)
            N.check(N.lib().spk_encoder_forward_ragged(ctypes.byref(cfg), ctypes.byref(weights), ctypes.byref(view),
                                                       batch, frames, samples, precision, int(training),
                                                       ctypes.c_uint64(seed), N.ptr(dvec), _aligned_ptr(ws), nbytes,
                                                       int(keep), N.stream_ptr(features.device)),
                    "spk_encoder_forward_ragged")
        else:
            view = N.MelView(features.data_ptr(), 1 if features.dtype == torch.float16 else 0, window, hop, spw)
            N.check(N.lib().spk_encoder_forward_view(ctypes.byref(cfg), ctypes.byref(weights), ctypes.byref(view),
                                                     batch, frames, samples, precision, int(training),
                                                     ctypes.c_uint64(seed), N.ptr(dvec), _aligned_ptr(ws), nbytes,
                                                     int(keep), N.stream_ptr(features.device)),
                    "spk_encoder_forward_view")
    if return_ragged:
        return dvec, ws, nbytes, (batch, frames, precision), ragged
    return dvec, ws, nbytes, (batch, frames, precision)


def _mel_ragged(ragged):
    return N.MelRagged(ragged.data.data_ptr(), 1 if ragged.data.dtype == torch.float16 else 0, ragged.data.size(1),
                       ragged.table.data_ptr())


def utterance_slices(lengths, frame_length, overlap_length, starts=None):
    """The slicing rule of variable-length utterances, for ``GE2E.embed_utterances`` and ``RaggedMel(segments=...)``.

    An utterance of ``L`` frames gives, with hop ``h = frame_length - overlap_length``:
      * ``L <= frame_length``: one slice, the utterance reflect-padded to ``frame_length`` (numpy 'reflect', floor of
        the missing frames on the left, ceil on the right, as ``Datasets.Correction`` does it);
      * ``L > frame_length``: ``S = ceil((L - frame_length) / h) + 1`` slices at offsets ``min(s * h, L - frame_length)``
        (the last one end-aligned, so every frame is covered).
    When ``(L - frame_length) % h == 0`` these are the slices of ``Overlapped_Slices`` / ``GE2E.embed_windows``.
    ``starts``: the first column of every utterance in the ragged array (default: the utterances back to back).
    Returns ``(table int32 [slices, 3] = (start, length, offset), segments int32 [utterances + 1])`` on the host."""
    T, hop = int(frame_length), int(frame_length) - int(overlap_length)
    if T < 1 or hop <= 0:
        raise RuntimeError("invalid slicing: frame_length %d, overlap_length %d" % (frame_length, overlap_length))
    L = torch.as_tensor(lengths, dtype=torch.int64).reshape(-1)
    if L.numel() == 0 or int(L.min()) < 1:
        raise RuntimeError("utterance lengths must be >= 1 frame")
    if starts is None:
        starts = torch.cumsum(L, 0) - L
    starts = torch.as_tensor(starts, dtype=torch.int64).reshape(-1)
    extra = (L - T).clamp(min=0)
    count = torch.where(L > T, (extra + hop - 1) // hop + 1, torch.ones_like(L))
    segments = torch.zeros(L.numel() + 1, dtype=torch.int64)
    segments[1:] = torch.cumsum(count, 0)
    utt = torch.repeat_interleave(torch.arange(L.numel()), count)
    s = torch.arange(int(segments[-1])) - segments[:-1][utt]
    offset = torch.minimum(s * hop, extra[utt])
    table = torch.stack([starts[utt], L[utt], offset], dim=1)
    return table.to(torch.int32), segments.to(torch.int32)


class _EncoderFunction(torch.autograd.Function):
    """Differentiable encoder call: forward keeps the activation stash, backward runs
    spk_encoder_backward into one flat fp32 gradient buffer (returned as per-parameter views).  When ``features`` needs
    a gradient the backward is spk_encoder_backward_input, which also writes dL/d(features); with every parameter
    frozen it computes no parameter gradient at all and allocates no gradient arena.  ``ragged``: a RaggedMel whose
    ``data`` is ``features``; its backward is spk_encoder_backward_segments, which folds the slices' gradient back
    onto ``data``."""

    @staticmethod
    def forward(ctx, features, module, samples, precision, training, seed, ragged, *params):
        names = module._param_names
        cfg = module._cfg
        pe = module.positional_encoding.pe
        dvec, ws, nbytes, (batch, frames, precision), used = _run_forward(
            cfg, names, [p.detach() for p in params], pe, ragged if ragged is not None else features, samples,
            precision, training, seed, keep=True, return_ragged=True)
        ctx.module, ctx.ws, ctx.nbytes = module, ws, nbytes
        ctx.meta = (batch, frames, samples, precision, training, seed)
        ctx.ragged = used                 # the contiguous int32 table / segments the forward read (kept alive)
        ctx.features_dtype = features.dtype
        ctx.save_for_backward(*params)
        ctx.pe = pe
        return dvec

    @staticmethod
    def backward(ctx, grad_dvec):
        module = ctx.module
        cfg, names = module._cfg, module._param_names
        params = ctx.saved_tensors
        batch, frames, samples, precision, training, seed = ctx.meta
        device = grad_dvec.device
        grad_dvec = grad_dvec.contiguous().float()
        want_mel = ctx.needs_input_grad[0]
        # partial freezing keeps the full arena: only a fully frozen encoder skips the parameter gradients
        want_params = not want_mel or any(ctx.needs_input_grad[7:])
        ragged = ctx.ragged
        views, d_mel = None, None
        if want_params:
            sizes = [p.numel() for p in params]
            offsets, total = [], 0
            for s in sizes:
                offsets.append(total)
                total += (s + 3) // 4 * 4          # keep every view 16-byte aligned
            arena = module._grad_arena(total, device, params)
            views = [arena[o:o + s].view_as(p) for o, s, p in zip(offsets, sizes, params)]
        with torch.cuda.device(device):
            weights = _fill_params(N.EncoderParams(), dict(zip(names, [p.detach() for p in params])), ctx.pe,
                                   cfg.layers)
            grads = _fill_params(N.EncoderParams(), dict(zip(names, views)), None, cfg.layers) if want_params else None
            if ragged is not None and (want_mel or ragged.segments is not None):
                utterances = ragged.utterances if ragged.segments is not None else batch // samples
                if want_mel:
                    d_mel = torch.empty((cfg.mel_dim, ragged.data.size(1)), dtype=torch.float32, device=device)
                N.check(N.lib().spk_encoder_backward_segments(ctypes.byref(cfg), ctypes.byref(weights),
                                                              ctypes.byref(grads) if want_params else None,
                                                              ctypes.byref(_mel_ragged(ragged)),
                                                              N.ptr(ragged.segments), utterances, N.ptr(d_mel),
                                                              N.ptr(grad_dvec), batch, frames, precision,
                                                              int(training), ctypes.c_uint64(seed),
                                                              _aligned_ptr(ctx.ws), ctx.nbytes, N.stream_ptr(device)),
                        "spk_encoder_backward_segments")
                if want_mel:
                    d_mel = d_mel.to(ctx.features_dtype)
            elif not want_mel:
                N.check(N.lib().spk_encoder_backward(ctypes.byref(cfg), ctypes.byref(weights), ctypes.byref(grads),
                                                     N.ptr(grad_dvec), batch, frames, samples, precision,
                                                     int(training), ctypes.c_uint64(seed), _aligned_ptr(ctx.ws),
                                                     ctx.nbytes, N.stream_ptr(device)),
                        "spk_encoder_backward")
            else:
                d_mel = torch.empty((batch, cfg.mel_dim, frames), dtype=torch.float32, device=device)
                N.check(N.lib().spk_encoder_backward_input(ctypes.byref(cfg), ctypes.byref(weights),
                                                           ctypes.byref(grads) if want_params else None, N.ptr(d_mel),
                                                           N.ptr(grad_dvec), batch, frames, samples, precision,
                                                           int(training), ctypes.c_uint64(seed),
                                                           _aligned_ptr(ctx.ws), ctx.nbytes, N.stream_ptr(device)),
                        "spk_encoder_backward_input")
                d_mel = d_mel.to(ctx.features_dtype)      # fp16 patterns get an fp16 gradient
        if getattr(module, "_debug_keep_ws", False):      # parity tests read the stage buffers back
            module._last_ws, module._last_meta = ctx.ws, ctx.meta
        ctx.ws = ctx.ragged = None
        return (d_mel, None, None, None, None, None, None) + (tuple(views) if want_params else (None,) * len(params))


class GE2E(torch.nn.Module):
    """Transformer speaker encoder -> L2-normalised d-vector (Modules.py:5-59)."""

    def __init__(self, hyper_parameters: Namespace):
        super().__init__()
        self.hp = hyper_parameters
        hp = self.hp
        emb = hp.GE2E.Embedding_Size
        self.prenet = Conv1d(in_channels=hp.Sound.Mel_Dim, out_channels=emb, kernel_size=1, bias=True,
                             w_init_gain="relu")
        self.relu = torch.nn.ReLU()
        self.positional_encoding = Positional_Encoding(
            max_position=hp.GE2E.Positional_Encoding.Max_Position, embedding_size=emb,
            dropout_rate=hp.GE2E.Positional_Encoding.Dropout_Rate)
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")     # nested-tensor notice of nn.TransformerEncoder
            # parameter containers only: their forward() is never called
            self.transformer = torch.nn.TransformerEncoder(
                encoder_layer=torch.nn.TransformerEncoderLayer(
                    d_model=emb, nhead=hp.GE2E.Transformer.Head, dim_feedforward=emb * 4,
                    dropout=hp.GE2E.Transformer.Dropout_Rate),
                num_layers=hp.GE2E.Transformer.Num_Layers,
                norm=torch.nn.LayerNorm(normalized_shape=emb))
        self.projection = Conv1d(in_channels=emb, out_channels=emb, kernel_size=1, bias=True,
                                 w_init_gain="linear")

        self.train_precision = 2      # two fp16 planes (hi + lo ~ fp32 mantissa), forward and backward
        self.eval_precision = 1       # one fp16 plane for inference
        self.max_slices_per_call = 8192   # inference batches are processed in chunks of this many slices
        self._cfg = N.EncoderConfig(hp.Sound.Mel_Dim, emb, hp.GE2E.Transformer.Head, emb * 4,
                                    hp.GE2E.Transformer.Num_Layers, hp.GE2E.Positional_Encoding.Max_Position,
                                    float(hp.GE2E.Positional_Encoding.Dropout_Rate),
                                    float(hp.GE2E.Transformer.Dropout_Rate))
        self._param_names = [n for n, _ in self.named_parameters()]
        self._arena = None

    # flat fp32 gradient arena: every parameter gradient is a view of it, so the data-parallel
    # allreduce (distributed.apply_gradient_allreduce) is one in-place collective with no copies.
    # The arena is persistent (re-zeroed, not re-allocated, every backward) and carries four spare floats behind the
    # gradients: element `numel` is where distributed.allreduce_gradients parks the step's loss so that the logging
    # mean of Train.py:166-168 rides on the gradient collective (SURVEY.md C3).  If a caller still holds .grad tensors
    # that alias the arena (zero_grad(set_to_none=False)), autograd would accumulate a view onto itself, so a fresh
    # buffer is used for that backward instead.
    def _grad_arena(self, numel, device, params=()):
        arena = self._arena
        reusable = (arena is not None and arena.device == device and arena.numel() == numel + 4)
        if reusable:
            lo, hi = arena.data_ptr(), arena.data_ptr() + arena.numel() * 4
            reusable = not any(p.grad is not None and lo <= p.grad.data_ptr() < hi for p in params)
        if reusable:
            arena.zero_()
        else:
            arena = torch.zeros(numel + 4, dtype=torch.float32, device=device)
            self._arena = arena
        self._arena_numel = numel
        return arena

    def forward(self, features, samples=1):
        """features: [Batch * Sample, Mel_dim, Time] -> [Batch, Emb_dim] unit-norm d-vectors.  A ``RaggedMel``
        (Datasets.py) is cropped / reflect-padded on the device; with ``segments`` it gives one d-vector per segment
        (``samples`` must be 1).  Its ``data`` gets a gradient like a dense input when it requires one."""
        from .Datasets import RaggedMel
        samples = int(samples)
        params = list(self.parameters())
        ragged = features if isinstance(features, RaggedMel) else None
        # a frozen encoder used as a critic still differentiates with respect to its input
        input_grad = (ragged.data if ragged is not None else features).requires_grad
        need_grad = torch.is_grad_enabled() and (input_grad or any(p.requires_grad for p in params))
        if need_grad:
            if ragged is not None and input_grad and not ragged.spans_disjoint(samples):
                raise RuntimeError("RaggedMel: the column spans of different utterances overlap, so their gradients "
                                   "cannot be folded back onto `data`; give every utterance its own columns")
            seed = int(torch.empty((), dtype=torch.int64).random_().item()) if self.training else 0
            return _EncoderFunction.apply(ragged.data if ragged is not None else features, self, samples,
                                          self.train_precision, self.training, seed, ragged, *params)
        if self.training:
            raise RuntimeError("GE2E.forward in train() mode without gradients is not supported; call eval()")
        if ragged is not None:       # evaluation batches of the device collater (Train.py:198-212)
            return _run_forward(self._cfg, self._param_names, [p.detach() for p in params],
                                self.positional_encoding.pe, features, samples, self.eval_precision, False, 0,
                                keep=False)[0]
        return torch.ops.spkemb.encoder_infer(features, self.positional_encoding.pe, [p.detach() for p in params],
                                              samples, self.eval_precision, self.max_slices_per_call,
                                              self._cfg.mel_dim, self._cfg.emb, self._cfg.heads, self._cfg.layers,
                                              self._cfg.max_pos)


    def embed_windows(self, windows, frame_length, overlap_length):
        """Multi-slice d-vectors straight from un-sliced windows (the device-side form of Inference.py:95-115 +
        157-159): ``windows`` is ``[Utterances, Mel_Dim, samples*(frame_length-overlap_length)+overlap_length]``,
        fp32 or fp16; the overlapping slices are cut inside the prenet's input load (no sliced copy exists) and
        their embeddings are averaged per utterance.  Returns ``[Utterances, Emb_dim]``.  eval() only."""
        if self.training:
            raise RuntimeError("GE2E.embed_windows is an inference entry point; call eval()")
        hop = int(frame_length) - int(overlap_length)
        if windows.dim() != 3 or hop <= 0 or windows.size(2) < frame_length:
            raise RuntimeError("invalid slicing: frame_length %d, overlap_length %d, windows %s"
                               % (frame_length, overlap_length, tuple(windows.shape)))
        spw = (windows.size(2) - int(overlap_length)) // hop
        params = [p.detach() for p in self.parameters()]
        pe = self.positional_encoding.pe
        per_call = max(1, self.max_slices_per_call // spw)
        outs = []
        with torch.no_grad():
            for u in range(0, windows.size(0), per_call):
                outs.append(_run_forward(self._cfg, self._param_names, params, pe, windows[u:u + per_call], spw,
                                         self.eval_precision, False, 0, keep=False,
                                         slicing=(int(frame_length), hop, spw))[0])
        return outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)


    def embed_utterances(self, mels, frame_length, overlap_length, lengths=None):
        """Whole-utterance d-vectors of utterances of different lengths in one pass: every utterance is cut into
        ``frame_length``-frame slices by the rule of ``utterance_slices`` (short ones reflect-padded, long ones
        covered to their last frame), and its d-vector is the head over its own slices.  Returns ``[U, Emb_dim]``.

        ``mels``: a list of ``[Mel_Dim, L_u]`` tensors, or a padded ``[U, Mel_Dim, L_max]`` tensor with ``lengths``
        (padding columns are never read and get a zero gradient).  fp32 or fp16.  Runs at ``eval_precision`` in
        chunks of at most ``max_slices_per_call`` slices that never split an utterance; differentiable (at
        ``train_precision``, like ``forward``) when gradients are enabled and the mels or any parameter require them."""
        from .Datasets import RaggedMel
        if isinstance(mels, (list, tuple)):
            if lengths is not None:
                raise RuntimeError("embed_utterances: lengths is only for a padded [U, Mel_Dim, L_max] tensor")
            if not mels or any(m.dim() != 2 or m.size(0) != self._cfg.mel_dim for m in mels):
                raise RuntimeError("embed_utterances: every utterance must be [Mel_Dim=%d, L]" % self._cfg.mel_dim)
            lens = torch.tensor([m.size(1) for m in mels], dtype=torch.int64)
            starts = torch.cumsum(lens, 0) - lens
            data = torch.cat(list(mels), dim=1)
        else:
            if mels.dim() != 3 or mels.size(1) != self._cfg.mel_dim or lengths is None:
                raise RuntimeError("embed_utterances: a padded batch is [U, Mel_Dim=%d, L_max] with lengths"
                                   % self._cfg.mel_dim)
            lens = torch.as_tensor(lengths, dtype=torch.int64).cpu().reshape(-1)
            U, _, L_max = mels.shape
            if lens.numel() != U or int(lens.min()) < 1 or int(lens.max()) > L_max:
                raise RuntimeError("embed_utterances: lengths must be %d values in [1, %d]" % (U, L_max))
            starts = torch.arange(U, dtype=torch.int64) * L_max
            data = mels.permute(1, 0, 2).reshape(mels.size(1), U * L_max)     # one transposing copy
        table, segments = utterance_slices(lens, frame_length, overlap_length, starts)
        end = starts + lens
        device = data.device
        outs, u0 = [], 0
        U = lens.numel()
        seg = segments.to(torch.int64)
        while u0 < U:
            # whole utterances, at most max_slices_per_call slices (one utterance always fits a call)
            u1 = int(torch.searchsorted(seg, seg[u0] + self.max_slices_per_call, right=True)) - 1
            u1 = min(max(u1, u0 + 1), U)
            s0, s1 = int(seg[u0]), int(seg[u1])
            c0, c1 = int(starts[u0:u1].min()), int(end[u0:u1].max())
            t = table[s0:s1].clone()
            t[:, 0] -= c0
            chunk = RaggedMel(data[:, c0:c1], t, frame_length, segments[u0:u1 + 1] - s0, _checked=True,
                              _host=(t, segments[u0:u1 + 1] - s0))
            outs.append(self.forward(chunk.to(device)))
            u0 = u1
        return outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)


@torch.library.custom_op("spkemb::encoder_infer", mutates_args=())
def _encoder_infer(features: torch.Tensor, pe: torch.Tensor, params: list[torch.Tensor], samples: int,
                   precision: int, max_slices: int, mel_dim: int, emb: int, heads: int, layers: int,
                   max_pos: int) -> torch.Tensor:
    """Inference encoder as ONE dispatcher op, so ``torch.jit.trace`` (Trace.py) records a single opaque
    node.  Utterances are independent: large batches are cut into chunks of whole utterances."""
    cfg = N.EncoderConfig(mel_dim, emb, heads, emb * 4, layers, max_pos, 0.0, 0.0)
    names = _names_for(layers)
    batch = features.size(0)
    chunk = max(samples, (max_slices // samples) * samples)
    if batch <= chunk:
        return _run_forward(cfg, names, params, pe, features, samples, precision, False, 0, keep=False)[0]
    outs = []
    for s in range(0, batch, chunk):
        outs.append(_run_forward(cfg, names, params, pe, features[s:s + chunk], samples, precision, False, 0,
                                 keep=False)[0])
    return torch.cat(outs, dim=0)


@_encoder_infer.register_fake
def _(features, pe, params, samples, precision, max_slices, mel_dim, emb, heads, layers, max_pos):
    return features.new_empty((features.size(0) // samples, emb), dtype=torch.float32)


def _names_for(layers):
    names = list(_PARAM_ORDER_HEAD)
    for l in range(layers):
        names += ["transformer.layers.%d.%s" % (l, k) for k, _ in _LAYER_KEYS]
    names += ["transformer.norm.weight", "transformer.norm.bias", "projection.weight", "projection.bias"]
    return names


# ------------------------------------------------------------------------------------------------
# loss

def Overlapped_Slices(windows: torch.Tensor, frame_length: int, overlap_length: int) -> torch.Tensor:
    """Device-side form of the inference collater's slicing (Inference.py:95-115): ``windows`` is
    ``[Utterances, Mel_Dim, samples * (frame_length - overlap_length) + overlap_length]`` (what ``Correction``
    produces), the result is ``[Utterances * samples, Mel_Dim, frame_length]`` in utterance-major order, ready for
    ``GE2E.forward(features, samples)``.  Sending the un-sliced windows over PCIe and slicing here moves
    ``required_length`` instead of ``samples * frame_length`` frames per utterance (192 instead of 320 for the
    reference's 5 x 64 / 32 configuration)."""
    if windows.dim() != 3:
        raise RuntimeError("windows must be [Utterances, Mel_Dim, Time], got %s" % (tuple(windows.shape),))
    hop = frame_length - overlap_length
    if hop <= 0 or windows.size(2) < frame_length:
        raise RuntimeError("invalid slicing: frame_length %d, overlap_length %d, window %d"
                           % (frame_length, overlap_length, windows.size(2)))
    samples = (windows.size(2) - overlap_length) // hop
    sl = windows.unfold(2, frame_length, hop)[:, :, :samples]            # [U, Mel, samples, frame_length] (view)
    return sl.permute(0, 2, 1, 3).reshape(windows.size(0) * samples, windows.size(1), frame_length)


class _GE2ELossFunction(torch.autograd.Function):
    """Loss and gradients from ONE fused kernel launch (spk_ge2e_loss_ex); backward only rescales."""

    @staticmethod
    def forward(ctx, embeddings, weight, bias, per_speaker, mode=0):
        N.require_cuda(embeddings, "embeddings")
        emb = embeddings.detach().contiguous().float()
        if emb.dim() != 2 or emb.size(0) % per_speaker != 0:
            raise RuntimeError("embeddings must be [Speakers * Pattern_per_Speaker, Emb_dim]; got %s with "
                               "pattern_per_speaker=%d" % (tuple(embeddings.shape), per_speaker))
        speakers = emb.size(0) // per_speaker
        device = emb.device
        need_grad = any(ctx.needs_input_grad[:3])
        with torch.cuda.device(device):
            wsb = N.lib().spk_ge2e_workspace_bytes_ex(speakers, per_speaker, mode)
            if wsb == 0:                                                   # refused mode / shape
                raise RuntimeError("spk_ge2e_workspace_bytes_ex failed: %s"
                                   % N.lib().spk_last_error().decode("utf-8", "replace"))
            ws = torch.empty(wsb, dtype=torch.uint8, device=device)
            scal = torch.empty(3, dtype=torch.float32, device=device)      # loss, dw, db
            d_emb = torch.empty_like(emb) if need_grad else None
            N.check(N.lib().spk_ge2e_loss_ex(N.ptr(emb), speakers, per_speaker, emb.size(1), mode,
                                             N.ptr(weight.detach().float().contiguous()),
                                             N.ptr(bias.detach().float().contiguous()),
                                             ctypes.c_void_p(scal.data_ptr()), N.ptr(d_emb),
                                             ctypes.c_void_p(scal.data_ptr() + 4) if need_grad else None,
                                             ctypes.c_void_p(scal.data_ptr() + 8) if need_grad else None,
                                             N.ptr(ws), wsb, N.stream_ptr(device)), "spk_ge2e_loss_ex")
        ctx.d_emb, ctx.scal = d_emb, scal
        return scal[0].clone()

    @staticmethod
    def backward(ctx, grad_loss):
        d_emb, scal = ctx.d_emb, ctx.scal
        g_e = d_emb * grad_loss if ctx.needs_input_grad[0] else None
        g_w = scal[1] * grad_loss if ctx.needs_input_grad[1] else None
        g_b = scal[2] * grad_loss if ctx.needs_input_grad[2] else None
        return g_e, g_w, g_b, None, None


_GE2E_METHODS = {"softmax": 0, "contrast": N.GE2E_CONTRAST}
_GE2E_CENTROIDS = {"inclusive": 0, "exclusive": N.GE2E_EXCLUSIVE}


class GE2E_Loss(torch.nn.Module):
    """GE2E loss, logits = weight * cos(e, centroid) - bias (Modules.py:112-156).

    The defaults are the reference's: the softmax loss with inclusive centroids.  Its "within" similarity uses the
    inclusive sum-centroid, which after cosine normalisation is the diagonal block of the "between" matrix, so the loss
    is plain cross-entropy of the [N*M, N] scaled cosine matrix against the row's speaker (SURVEY.md D2).

    The GE2E paper's variants (DESIGN.md §3.3): ``loss_method="contrast"`` is
    ``1 - sigmoid(z_own) + max_{k != own} sigmoid(z_k)`` (eq. 7; needs two speakers), and ``centroids="exclusive"``
    computes each row's own-speaker similarity against the mean of the speaker's other utterances (eq. 8; needs two
    utterances per speaker)."""

    def __init__(self, init_weight=10.0, init_bias=-5.0, loss_method="softmax", centroids="inclusive"):
        super().__init__()
        if loss_method not in _GE2E_METHODS:
            raise ValueError("loss_method must be one of %s, got %r" % (sorted(_GE2E_METHODS), loss_method))
        if centroids not in _GE2E_CENTROIDS:
            raise ValueError("centroids must be one of %s, got %r" % (sorted(_GE2E_CENTROIDS), centroids))
        self.weight = torch.nn.Parameter(torch.tensor(init_weight))
        self.bias = torch.nn.Parameter(torch.tensor(init_bias))
        self.loss_method, self.centroids = loss_method, centroids
        self._mode = _GE2E_METHODS[loss_method] | _GE2E_CENTROIDS[centroids]

    def extra_repr(self):
        return "loss_method=%r, centroids=%r" % (self.loss_method, self.centroids)

    def forward(self, embeddings, pattern_per_speaker):
        """embeddings: [Batch, Emb_dim], speaker-major rows; returns the mean loss over the rows (0-dim)."""
        if not torch.is_grad_enabled():
            return _GE2ELossFunction.apply(embeddings.detach(), self.weight.detach(), self.bias.detach(),
                                           int(pattern_per_speaker), self._mode)
        loss = _GE2ELossFunction.apply(embeddings, self.weight, self.bias, int(pattern_per_speaker), self._mode)
        LAST_TRAINING_LOSS[loss.device] = loss.detach()      # picked up by distributed.allreduce_gradients
        return loss


# device -> the most recent training loss (a 0-dim tensor); see distributed.allreduce_gradients / reduce_tensor
LAST_TRAINING_LOSS = {}
