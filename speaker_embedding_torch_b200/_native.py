"""ctypes binding of libspkemb.so (C ABI declared in include/spkemb.h).

PyTorch is used only for device memory and streams: every call passes raw device
pointers (``tensor.data_ptr()``) and the current CUDA stream.  There is no CPU
path: a missing library or a non-CUDA tensor raises ``RuntimeError``.
"""
import ctypes
import os
import subprocess
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libspkemb.so")
CSRC = os.path.join(_HERE, "csrc")

SPK_MAX_LAYERS = 8
OPTIM_MAX_CHUNKS = 16      # SPK_OPTIM_MAX_CHUNKS
ABI_VERSION = 2
GE2E_CONTRAST = 1          # SPK_GE2E_CONTRAST
GE2E_EXCLUSIVE = 1 << 8    # SPK_GE2E_EXCLUSIVE

EXPORTS = (
    "spk_abi_version", "spk_last_error", "spk_encoder_workspace_bytes", "spk_encoder_forward",
    "spk_encoder_backward", "spk_ge2e_workspace_bytes", "spk_ge2e_loss", "spk_optim_step",
    "spk_gemm", "spk_split_pack", "spk_device_info", "spk_prof_enable", "spk_prof_report",
    "spk_encoder_debug_layout", "spk_set_option", "spk_encoder_forward_view", "spk_plan_flags",
    "spk_dropout_keep", "spk_encoder_forward_ragged",
    "spk_mel_frames", "spk_mel_spectrogram", "spk_set_debug_buffer", "spk_encoder_backward_input",
    "spk_mel_backward_workspace_bytes", "spk_mel_spectrogram_backward",
    "spk_encoder_forward_segments", "spk_encoder_backward_segments",
    "spk_ge2e_workspace_bytes_ex", "spk_ge2e_loss_ex",
)

c_f32p = ctypes.c_void_p  # device pointers travel as integers


class MelView(ctypes.Structure):
    """spk_mel_view: strided / fp16 view of the mel input (overlapping inference slices cut inside the prenet load)."""
    _fields_ = [("data", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("window_frames", ctypes.c_int32),
                ("hop", ctypes.c_int32), ("slices_per_window", ctypes.c_int32)]


class MelRagged(ctypes.Structure):
    """spk_mel_ragged: a training batch as one [Mel_Dim, total_frames] array + (start, length, offset) per utterance."""
    _fields_ = [("data", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("total_frames", ctypes.c_int64),
                ("table", ctypes.c_void_p)]


class EncoderConfig(ctypes.Structure):
    _fields_ = [("mel_dim", ctypes.c_int32), ("emb", ctypes.c_int32), ("heads", ctypes.c_int32),
                ("ffn", ctypes.c_int32), ("layers", ctypes.c_int32), ("max_pos", ctypes.c_int32),
                ("pe_dropout", ctypes.c_float), ("dropout", ctypes.c_float)]


LAYER_FIELDS = ("in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "linear1_w", "linear1_b",
                "linear2_w", "linear2_b", "norm1_w", "norm1_b", "norm2_w", "norm2_b")


class LayerParams(ctypes.Structure):
    _fields_ = [(n, c_f32p) for n in LAYER_FIELDS]


class EncoderParams(ctypes.Structure):
    _fields_ = [("prenet_w", c_f32p), ("prenet_b", c_f32p), ("pe_alpha", c_f32p), ("pe", c_f32p),
                ("layer", LayerParams * SPK_MAX_LAYERS),
                ("norm_w", c_f32p), ("norm_b", c_f32p), ("proj_w", c_f32p), ("proj_b", c_f32p)]


class OptimTensors(ctypes.Structure):
    _fields_ = [("count", ctypes.c_int32),
                ("param", c_f32p * 64), ("grad", c_f32p * 64), ("exp_avg", c_f32p * 64),
                ("exp_avg_sq", c_f32p * 64), ("numel", ctypes.c_int64 * 64)]


class GemmDesc(ctypes.Structure):
    _fields_ = [
        ("a", ctypes.c_void_p), ("a_plane_stride", ctypes.c_int64), ("a_rows", ctypes.c_int64),
        ("a_cols", ctypes.c_int64), ("a_ld", ctypes.c_int64), ("a_sb0", ctypes.c_int64),
        ("a_sb1", ctypes.c_int64), ("a_mn", ctypes.c_int32),
        ("b", ctypes.c_void_p), ("b_plane_stride", ctypes.c_int64), ("b_rows", ctypes.c_int64),
        ("b_cols", ctypes.c_int64), ("b_ld", ctypes.c_int64), ("b_sb0", ctypes.c_int64),
        ("b_sb1", ctypes.c_int64), ("b_mn", ctypes.c_int32),
        ("planes", ctypes.c_int32), ("m", ctypes.c_int32), ("n", ctypes.c_int32), ("k", ctypes.c_int32),
        ("nb0", ctypes.c_int32), ("nb1", ctypes.c_int32), ("ksplit", ctypes.c_int32),
        ("block_n", ctypes.c_int32), ("flags", ctypes.c_uint32), ("alpha", ctypes.c_float),
        ("bias", ctypes.c_void_p),
        ("out", ctypes.c_void_p), ("out_plane_stride", ctypes.c_int64), ("out_ld", ctypes.c_int64),
        ("out_sb0", ctypes.c_int64), ("out_sb1", ctypes.c_int64), ("out_planes", ctypes.c_int32),
    ]


def build(verbose=False):
    """Compile libspkemb.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    proc = subprocess.run(["make", "-j8", "-C", CSRC], capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        print(proc.stdout[-4000:])
        print(proc.stderr[-4000:])
    if proc.returncode != 0:
        raise RuntimeError("building libspkemb.so failed (nvcc -gencode arch=compute_100a,code=sm_100a)")
    return LIB_PATH


_lib = None
_lock = threading.Lock()


def lib():
    """Load the shared library (once) and declare the prototypes of include/spkemb.h."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libspkemb.so is missing (%s). Build it with `python -c 'import __graft_entry__ as g; g.build()'`"
                " or `make -C speaker_embedding_torch_b200/csrc`; there is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        vp, i32, i64, u64, f32, sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64,
                                      ctypes.c_float, ctypes.c_size_t)
        L.spk_abi_version.restype = i32
        L.spk_abi_version.argtypes = []
        L.spk_last_error.restype = ctypes.c_char_p
        L.spk_last_error.argtypes = []
        L.spk_encoder_workspace_bytes.restype = sz
        L.spk_encoder_workspace_bytes.argtypes = [ctypes.POINTER(EncoderConfig), i32, i32, i32, i32, i32]
        L.spk_encoder_forward.restype = i32
        L.spk_encoder_forward.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams), vp,
                                          i32, i32, i32, i32, i32, u64, vp, vp, sz, i32, vp]
        L.spk_encoder_forward_view.restype = i32
        L.spk_encoder_forward_view.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams),
                                               ctypes.POINTER(MelView), i32, i32, i32, i32, i32, u64, vp, vp, sz,
                                               i32, vp]
        L.spk_encoder_forward_ragged.restype = i32
        L.spk_encoder_forward_ragged.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams),
                                                 ctypes.POINTER(MelRagged), i32, i32, i32, i32, i32, u64, vp, vp, sz,
                                                 i32, vp]
        L.spk_encoder_forward_segments.restype = i32
        L.spk_encoder_forward_segments.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams),
                                                   ctypes.POINTER(MelRagged), vp, i32, i32, i32, i32, i32, u64, vp,
                                                   vp, sz, i32, vp]
        L.spk_encoder_backward_segments.restype = i32
        L.spk_encoder_backward_segments.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams),
                                                    ctypes.POINTER(EncoderParams), ctypes.POINTER(MelRagged), vp, i32,
                                                    vp, vp, i32, i32, i32, i32, u64, vp, sz, vp]
        L.spk_encoder_backward.restype = i32
        L.spk_encoder_backward.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams),
                                           ctypes.POINTER(EncoderParams), vp, i32, i32, i32, i32, i32, u64,
                                           vp, sz, vp]
        L.spk_encoder_backward_input.restype = i32
        L.spk_encoder_backward_input.argtypes = [ctypes.POINTER(EncoderConfig), ctypes.POINTER(EncoderParams),
                                                 ctypes.POINTER(EncoderParams), vp, vp, i32, i32, i32, i32, i32, u64,
                                                 vp, sz, vp]
        L.spk_ge2e_workspace_bytes.restype = sz
        L.spk_ge2e_workspace_bytes.argtypes = [i32, i32]
        L.spk_ge2e_loss.restype = i32
        L.spk_ge2e_loss.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]
        L.spk_ge2e_workspace_bytes_ex.restype = sz
        L.spk_ge2e_workspace_bytes_ex.argtypes = [i32, i32, i32]
        L.spk_ge2e_loss_ex.restype = i32
        L.spk_ge2e_loss_ex.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]
        L.spk_optim_step.restype = i32
        L.spk_optim_step.argtypes = [ctypes.POINTER(OptimTensors), i32, i64, f32, f32, f32, f32, f32, f32, f32,
                                     vp, i32, i32, i32, vp]
        L.spk_gemm.restype = i32
        L.spk_gemm.argtypes = [ctypes.POINTER(GemmDesc), vp]
        L.spk_split_pack.restype = i32
        L.spk_split_pack.argtypes = [vp, vp, i64, i32, i64, vp]
        L.spk_device_info.restype = i32
        L.spk_device_info.argtypes = [ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32)]
        L.spk_set_option.restype = i32
        L.spk_set_option.argtypes = [ctypes.c_char_p, i32]
        L.spk_set_debug_buffer.restype = i32
        L.spk_set_debug_buffer.argtypes = [vp, sz]
        L.spk_mel_frames.restype = i32
        L.spk_mel_frames.argtypes = [i64, i32, i32]
        L.spk_mel_spectrogram.restype = i32
        L.spk_mel_spectrogram.argtypes = [vp, i32, i64, i32, i32, i32, vp, vp, i32, vp, i32, vp]
        L.spk_mel_backward_workspace_bytes.restype = sz
        L.spk_mel_backward_workspace_bytes.argtypes = [i32, i64, i32, i32]
        L.spk_mel_spectrogram_backward.restype = i32
        L.spk_mel_spectrogram_backward.argtypes = [vp, vp, i32, i64, i32, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp]
        L.spk_dropout_keep.restype = i32
        L.spk_dropout_keep.argtypes = [u64, f32, ctypes.c_uint32, u64, i64, vp, vp]
        L.spk_plan_flags.restype = i32
        L.spk_plan_flags.argtypes = []
        L.spk_prof_enable.restype = i32
        L.spk_prof_enable.argtypes = [i32]
        L.spk_prof_report.restype = i32
        L.spk_prof_report.argtypes = [ctypes.c_char_p, sz]
        L.spk_encoder_debug_layout.restype = i32
        L.spk_encoder_debug_layout.argtypes = [ctypes.POINTER(EncoderConfig), i32, i32, i32, i32, i32,
                                               ctypes.c_char_p, sz]
        if L.spk_abi_version() != ABI_VERSION:
            raise RuntimeError("libspkemb.so ABI %d != binding ABI %d" % (L.spk_abi_version(), ABI_VERSION))
        for name, env in (("gemm_cta_pairs", "SPKEMB_GEMM_CTA_PAIRS"),):      # A/B switches for the benchmarks
            if env in os.environ:
                L.spk_set_option(name.encode(), int(os.environ[env]))
        _lib = L
    return _lib


def check(code, what):
    if code != 0:
        msg = lib().spk_last_error()
        raise RuntimeError("%s failed (%d): %s" % (what, code, msg.decode("utf-8", "replace") if msg else ""))


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: this framework has no CPU path" % name)
    return t


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


# ---------------------------------------------------------------------------------------------
# helpers shared by tests and bench: split-fp16 planes <-> fp32

def split_pack(x, planes):
    """fp32 CUDA tensor -> fp16 tensor [planes, *x.shape] (hi, lo) via the library's kernel."""
    require_cuda(x, "x")
    x = x.contiguous().float()
    out = torch.empty((planes,) + tuple(x.shape), dtype=torch.float16, device=x.device)
    check(lib().spk_split_pack(ptr(x), ptr(out), x.numel(), planes, x.numel(), stream_ptr(x.device)),
          "spk_split_pack")
    return out


def split_unpack(s):
    """fp16 [planes, ...] -> fp32 (hi + lo)."""
    return s.float().sum(dim=0)


def gemm(a, b, planes, m, n, k, a_mn=False, b_mn=False, bias=None, relu=False, out_f32=False,
         atomic_out=None, ksplit=1, block_n=0, alpha=1.0):
    """D[M,N] = alpha * A B^T on split operands (test / roofline entry, 2-D unbatched).

    a: fp16 [planes, M, K] (K-major) or [planes, K, M] (a_mn); b likewise with N.
    Returns fp16 [planes, M, N], or fp32 [M, N] when out_f32 / atomic_out.
    """
    require_cuda(a, "a")
    require_cuda(b, "b")
    d = GemmDesc()
    d.a, d.a_plane_stride = a.data_ptr(), a.stride(0)
    d.a_rows, d.a_cols, d.a_ld = a.shape[1], a.shape[2], a.stride(1)
    d.a_mn = int(a_mn)
    d.b, d.b_plane_stride = b.data_ptr(), b.stride(0)
    d.b_rows, d.b_cols, d.b_ld = b.shape[1], b.shape[2], b.stride(1)
    d.b_mn = int(b_mn)
    d.planes, d.m, d.n, d.k = planes, m, n, k
    d.nb0 = d.nb1 = 1
    d.ksplit, d.block_n, d.alpha = ksplit, block_n, alpha
    flags = 0
    if bias is not None:
        flags |= 1
        d.bias = bias.data_ptr()
    if relu:
        flags |= 2
    if atomic_out is not None:
        out = atomic_out
        flags |= 1 << 9
        d.out_planes = 1
    elif out_f32:
        out = torch.empty((m, n), dtype=torch.float32, device=a.device)
        flags |= 1 << 8
        d.out_planes = 1
    else:
        out = torch.empty((planes, m, n), dtype=torch.float16, device=a.device)
        d.out_plane_stride = out.stride(0)
        d.out_planes = planes
    d.flags = flags
    d.out, d.out_ld = out.data_ptr(), n
    check(lib().spk_gemm(ctypes.byref(d), stream_ptr(a.device)), "spk_gemm")
    return out


def debug_layout(cfg, batch, frames, samples, precision, keep):
    """{buffer name: (byte offset, plane stride in elements)} of the encoder workspace (tests only)."""
    buf = ctypes.create_string_buffer(1 << 14)
    n = lib().spk_encoder_debug_layout(ctypes.byref(cfg), batch, frames, samples, precision, int(keep), buf, len(buf))
    out = {}
    for line in buf.raw[:n].decode().splitlines():
        name, off, ps = line.split()
        out[name] = (int(off), int(ps))
    return out


def read_split(ws, layout, name, rows, cols, planes):
    """Read a split tensor [rows, cols] out of a workspace uint8 tensor as fp32 (hi + lo)."""
    off, ps = layout[name]
    base = (ws.data_ptr() + 255) // 256 * 256 - ws.data_ptr() + off
    out = None
    for p in range(planes):
        start = base + p * ps * 2
        t = ws[start:start + rows * cols * 2].view(torch.float16).view(rows, cols).float()
        out = t if out is None else out + t
    return out


def _ws_bytes(ws, layout, name, nbytes):
    off, _ = layout[name]
    base = (ws.data_ptr() + 255) // 256 * 256 - ws.data_ptr() + off
    return ws[base:base + nbytes]


def read_f32(ws, layout, name, n):
    """Read ``n`` fp32 values of a workspace buffer (statistics, head vectors, gradient scale) as a 1-D tensor."""
    return _ws_bytes(ws, layout, name, n * 4).view(torch.float32).clone()


def read_bits(ws, layout, name, rows, cols):
    """Read a 1-bit mask of a [rows, cols] tensor as bool [rows, cols].  The words are chunk-major ``[cols/32][rows]``:
    bit i of word (c, r) is element (r, 32c + i)."""
    words = _ws_bytes(ws, layout, name, (cols // 32) * rows * 4).view(torch.int32).view(cols // 32, rows)
    shifts = torch.arange(32, dtype=torch.int32, device=ws.device)
    bits = (words.unsqueeze(-1) >> shifts) & 1                       # [cols/32, rows, 32]
    return bits.permute(1, 0, 2).reshape(rows, cols).bool()


def prof_enable(on=True):
    lib().spk_prof_enable(int(on))


def prof_report():
    """-> {tag: dict(launches, ms, flops, bytes)} for the launches since the last report (synchronises)."""
    buf = ctypes.create_string_buffer(1 << 16)
    n = lib().spk_prof_report(buf, len(buf))
    out = {}
    for line in buf.raw[:n].decode().splitlines():
        tag, cnt, ms, fl, by = line.split()
        out[tag] = dict(launches=int(cnt), ms=float(ms), flops=float(fl), bytes=float(by))
    return out


def dropout_keep(seed, p, site, numel, device):
    """Keep-scales (0 or 1/(1-p_q)) of elements [0, numel) of dropout site ``site`` (tests: masks fed to the oracle)."""
    n8 = (numel + 7) // 8
    out = torch.empty(n8 * 8, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        check(lib().spk_dropout_keep(ctypes.c_uint64(seed), float(p), int(site), ctypes.c_uint64(0), n8, ptr(out),
                                     stream_ptr(device)), "spk_dropout_keep")
    return out[:numel]


def plan_flags():
    """SPK_PLAN_* snapshot of the layout-shaping options, OR-ed into ``precision`` by the module layer so that a
    backward call rebuilds exactly the plan of its forward call."""
    return int(lib().spk_plan_flags())


def set_option(name, value):
    check(lib().spk_set_option(name.encode(), int(value)), "spk_set_option")
