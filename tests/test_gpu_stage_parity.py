"""Every encoder stage, and every parameter gradient, against fp64 on the inputs the kernels themselves saw.

The end-to-end tests (test_gpu_parity_full.py) compare with the reference at the 1e-3 budget, most of which is ReLU
gates that flip where a pre-activation lies within rounding of zero.  Here nothing accumulates:

* B1: each forward stage is recomputed in fp64 from the stage inputs read back out of the workspace and compared with
  the stage output the kernel stored.  Errors are normalised by the magnitude of the sum that produced each element
  (|A| |B|^T + |bias| + |residual|), so the bound is the stage's own rounding: about 2^-22 of storage plus 5e-8 of
  accumulator truncation with two fp16 planes, about 2^-11 with one.
* B2: the fp64 oracle is forced onto the ReLU gates (and in train mode the dropout masks) the library chose, so its
  gradients are those of the same piecewise-linear function; every tensor is compared on its own.
* C1: a constant added to a bias before a LayerNorm shifts every row and, in exact arithmetic, changes nothing after it.
* C2: the power-of-two gradient scale of the backward pass under scaled, zero and non-finite upstream gradients.

References are computed with torch in float64 on the device.  Every bound carries the worst value measured on a B200
(1000 W power limit) beside it; each test prints its figures as one JSON line.
"""
import json
import math

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth

pytestmark = pytest.mark.gpu

D, F, H = 256, 1024, 4
DEV = "cuda"
SEED = 20261020
DEFAULTS = {"prune_last_layer": 1, "fused_layernorm": 2, "fused_training_attention": 1,
            "training_attention_two_ctas": 1, "grad_scale_log2": 12}

# ---- bounds: {precision: {metric: bound}}; the measured worst on a B200 is in the comment after each bound
BOUNDS = {
    2: {
        "gemm": 8e-6,          # 1.75e-6  normalised |out - ref| / (|A||B|^T + |bias| + |res|); also a ReLU bit's band
        "attn": 2e-7,          # 3.3e-8   |att - ref| / the attention's rounding scale (_Stages.attention)
        "stat_max": 1e-6,      # 1.8e-7   |row max * log2e/8 - ref| / (max |q||k| / 8 * log2e)
        "stat_sum": 4e-5,      # 7.5e-6   relative
        "ln_mean": 4e-6,       # 8.4e-7   |mean - ref| / std
        "ln_rstd": 1.6e-5,     # 3.2e-6   relative (z itself carries the GEMM's rounding)
        "ln_out": 6e-5,        # 1.2e-5   |h - ref| / (|gamma| + |beta|)
        "head": 4e-6,          # 7.2e-7   hn / emean / d-vector absolute, epre normalised
    },
    1: {   # one fp16 plane; ln_mean / ln_rstd: the pruned last layer's ln_fwd on its own stored input
        "gemm": 2e-3,          # 4.1e-4
        "attn": 3e-5,          # 5.9e-6
        "ln_mean": 2e-7,       # 3.5e-8
        "ln_rstd": 5e-7,       # 9.8e-8
        "ln_out": 2e-2,        # 4.3e-3
        "head": 3e-6,          # 5.6e-7
    },
    3: {
        "gemm": 4e-6,          # 8.7e-7
        "attn": 1.2e-7,        # 2.3e-8
        "ln_mean": 2e-7,       # 3.6e-8
        "ln_rstd": 2.2e-7,     # 4.3e-8
        "ln_out": 4e-5,        # 8.0e-6
        "head": 3e-6,          # 5.0e-7
    },
}
GRAD_REL = 1e-4          # 2.2e-5   per tensor, relative L2, against the gate-forced oracle
GRAD_ZERO = 4e-4         # 8.4e-5   K slice of in_proj_bias: |g| / |Q slice| (an fp32 sum that cancels to zero)
LOSS_REL = 2.5e-6        # 5.0e-7
DVEC_ABS = 4e-6          # 8.4e-7
POW2_REL = 1e-6          # 2.0e-7    g * 2^k against 2^k * (g): the same planes, split-K atomics reordered


def _record(kind, **kw):
    print("stage parity:", json.dumps(dict(kind=kind, **kw)))


class _Options:
    def __init__(self, **opts):
        self.opts = opts

    def __enter__(self):
        from speaker_embedding_torch_b200 import _native as N
        for k, v in self.opts.items():
            N.set_option(k, v)

    def __exit__(self, *exc):
        from speaker_embedding_torch_b200 import _native as N
        for k in self.opts:
            N.set_option(k, DEFAULTS[k])


def _model(seed, layers=3, bias_offset=None):
    """GE2E with synth.make_state weights; ``bias_offset = (name, c)`` adds c to one bias."""
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    hp = default_hyper_parameters()
    hp.GE2E.Transformer.Num_Layers = layers
    full = synth.make_state(seed)
    state = {k: v for k, v in full.items()
             if not k.startswith("transformer.layers.") or int(k.split(".")[2]) < layers}
    if bias_offset is not None:
        name, c = bias_offset
        state[name] = (state[name].astype(np.float64) + c).astype(np.float32)
    m = GE2E(hp)
    m.load_state_dict({k: torch.as_tensor(v) for k, v in state.items()}, strict=True)
    return m.to(DEV), state


def _dstate(state):
    return {k: torch.as_tensor(v).to(DEV, torch.float64) for k, v in state.items()}


def _forward_ws(m, mel, samples, precision, training, keep):
    from speaker_embedding_torch_b200 import Modules, _native as N
    params = [p.detach() for p in m.parameters()]
    dvec, ws, _, (B, T, pflags) = Modules._run_forward(m._cfg, m._param_names, params, m.positional_encoding.pe,
                                                       mel, samples, precision, training, SEED, keep=keep)
    torch.cuda.synchronize()
    return dvec, ws, N.debug_layout(m._cfg, B, T, samples, pflags, keep)


def _keep(site, numel, p):
    from speaker_embedding_torch_b200 import _native as N
    return N.dropout_keep(SEED, p, site, numel, DEV).double()


def _nerr(got, ref, mag, floor=0.0):
    """max |got - ref| / mag beyond the absolute floors: a split tensor keeps values below 2^-14 to an absolute 2^-25
    (the low fp16 plane is subnormal there), whatever the number of planes; ``floor`` is a stage's own."""
    return float((((got.double() - ref).abs() - 2.0 ** -25 - floor).clamp_min(0.0) / (mag + 1e-30)).max())


def _ln_ref(z, w, b):
    mu = z.mean(-1, keepdim=True)
    var = ((z - mu) ** 2).mean(-1, keepdim=True)
    return (z - mu) / torch.sqrt(var + O.LN_EPS) * w + b, mu[:, 0], 1.0 / torch.sqrt(var[:, 0] + O.LN_EPS)


class _Stages:
    """Reads a stage's inputs / outputs from one forward workspace and collects the normalised errors."""

    def __init__(self, ws, lay, st, B, T, S, P, training, p_pe, p):
        self.ws, self.lay, self.st = ws, lay, st
        self.B, self.T, self.S, self.P, self.Mt = B, T, S, P, B * T
        self.training, self.p_pe, self.p = training, p_pe, p
        self.err = {}
        self.flips = {}

    def split(self, name, rows, cols):
        from speaker_embedding_torch_b200 import _native as N
        return N.read_split(self.ws, self.lay, name, rows, cols, self.P).double()

    def f32(self, name, n):
        from speaker_embedding_torch_b200 import _native as N
        return N.read_f32(self.ws, self.lay, name, n).double()

    def bits(self, name, rows, cols):
        from speaker_embedding_torch_b200 import _native as N
        return N.read_bits(self.ws, self.lay, name, rows, cols)

    def note(self, key, v):
        self.err[key] = max(self.err.get(key, 0.0), v)

    def gemm(self, a, w, b=None):
        """fp64 a @ w^T (+ b) and its magnitude |a| |w|^T (+ |b|)."""
        ref = a @ w.t()
        mag = a.abs() @ w.abs().t()
        if b is not None:
            ref, mag = ref + b, mag + b.abs()
        return ref, mag

    def gate_check(self, key, bits, ref, u, mag):
        """ReLU-gate bits against fp64 (``ref``): a disagreement is allowed only within the rounding band of zero."""
        diff = bits != ref
        n = int(diff.sum())
        if n:
            band = float((u[diff].abs() / mag[diff]).max())
            self.note(key + ".gate_band", band)
        self.flips[key] = self.flips.get(key, 0) + n

    def ln(self, key, z_ref, mag, w, b, h_got, st_got=None, z_got=None):
        h_ref, mu, rstd = _ln_ref(z_ref, w, b)
        if z_got is not None:
            self.note("gemm", _nerr(z_got, z_ref, mag))
        if st_got is not None:
            st_got = st_got.view(-1, 2)
            std = 1.0 / rstd
            self.note("ln_mean", float(((st_got[:, 0] - mu).abs() / std).max()))
            self.note("ln_rstd", float(((st_got[:, 1] - rstd).abs() / rstd).max()))
        self.note("ln_out", _nerr(h_got, h_ref, w.abs() + b.abs()))
        return h_ref

    def attention(self, q, k, v, keep):
        """q [BH, Tq, 64], k / v [BH, T, 64], keep [BH, Tq, T] or None -> (out [BH, Tq, 64], mag, floor, s).

        ``mag`` is the scale of the relative rounding: a score carries an error relative to sum |q||k| / 8, which moves
        its own term p v and, through the row sum, every term (by p o, dropped keys included); a probability carries one
        relative to itself.  ``floor`` is absolute: the fp16 planes of a probability keep it to 2^-25 (subnormal low
        plane).  Where dropout removed a row's dominant keys the output is small and the floor is what bounds it."""
        s = q @ k.transpose(1, 2) / 8.0
        sabs = q.abs() @ k.abs().transpose(1, 2) / 8.0
        p0 = torch.softmax(s, dim=-1)
        pr, ones = (p0 * keep, keep) if keep is not None else (p0, torch.ones_like(p0))
        o = pr @ v
        mag = (pr * (1.0 + sabs)) @ v.abs() + (p0 * (1.0 + sabs)).sum(-1, keepdim=True) * o.abs()
        return o, mag, 2.0 ** -25 * (ones @ v.abs()), s

    def run(self, layers, prune, h0_emulated=False):
        B, T, Mt, st = self.B, self.T, self.Mt, self.st
        p, training = self.p, self.training
        # ---- prenet + positional encoding
        x0 = self.split("x0", Mt, 80)
        u, mag = self.gemm(x0, st["prenet.weight"][:, :, 0], st["prenet.bias"])
        pe_t = self.f32("pe_t", T * D).view(T, D)
        alpha = st["positional_encoding.alpha"]
        h0_ref = torch.relu(u) + alpha * pe_t.repeat(B, 1)
        mag0 = mag + alpha.abs() * pe_t.abs().repeat(B, 1)
        if training:
            kp = _keep(0, Mt * D, self.p_pe).view(Mt, D)
            h0_ref, mag0 = h0_ref * kp, mag0 * kp
        if "h0bits" in self.lay:
            self.gate_check("prenet", self.bits("h0bits", Mt, D), u > 0, u, mag)
        if h0_emulated:      # inference without a stash: h0's slot is reused for the last output
            h = h0_ref.float().half().double() if self.P == 1 else h0_ref
        else:
            h = self.split("h0", Mt, D)
            self.note("gemm", _nerr(h, h0_ref, mag0))
        dense = layers - 1 if prune else layers
        for l in range(dense):
            pre = "transformer.layers.%d." % l
            L = "L%d." % l
            qkv_ref, mag = self.gemm(h, st[pre + "self_attn.in_proj_weight"], st[pre + "self_attn.in_proj_bias"])
            qkv = self.split(L + "qkv", Mt, 3 * D)
            self.note("gemm", _nerr(qkv, qkv_ref, mag))
            heads = qkv.view(B, T, 3, H, 64).permute(2, 0, 3, 1, 4).reshape(3, B * H, T, 64)
            keep = None
            if training:
                Tp = (T + 7) // 8 * 8
                keep = _keep(1 + 4 * l, B * H * T * Tp, p).view(B * H, T, Tp)[..., :T]
            o_ref, o_mag, o_floor, s = self.attention(heads[0], heads[1], heads[2], keep)
            att = self.split(L + "att", Mt, D)
            o_ref, o_mag, o_floor = (t.view(B, H, T, 64).permute(0, 2, 1, 3).reshape(Mt, D)
                                     for t in (o_ref, o_mag, o_floor))
            self.note("attn", _nerr(att, o_ref, o_mag, o_floor))
            if L + "astat" in self.lay:
                self.attention_stats(L, heads[0], heads[1], s, l)
            # out-proj + dropout1 + residual + LayerNorm1
            a_ref, mag = self.gemm(att, st[pre + "self_attn.out_proj.weight"], st[pre + "self_attn.out_proj.bias"])
            if training:
                k2 = _keep(2 + 4 * l, Mt * D, p).view(Mt, D)
                a_ref, mag = a_ref * k2, mag * k2
            z1_ref, mag = a_ref + h, mag + h.abs()
            stash = L + "st1" in self.lay and self.keep_stats
            h1 = self.split(L + "h1", Mt, D)
            self.ln("ln", z1_ref, mag, st[pre + "norm1.weight"], st[pre + "norm1.bias"], h1,
                    self.f32(L + "st1", Mt * 2) if stash else None,
                    self.split(L + "z1", Mt, D) if self.z_stored else None)
            # FFN1 + ReLU + dropout
            u, mag = self.gemm(h1, st[pre + "linear1.weight"], st[pre + "linear1.bias"])
            f_ref = torch.relu(u)
            if training:
                k3 = _keep(3 + 4 * l, Mt * F, p).view(Mt, F)
                f_ref, mag_f = f_ref * k3, mag * k3
            else:
                mag_f = mag
            f = self.split(L + "f", Mt, F)
            self.note("gemm", _nerr(f, f_ref, mag_f))
            if self.keep_stats:
                ref = (u > 0) & (k3 > 0) if training else u > 0      # the bits are those of the post-dropout f
                self.gate_check("ffn%d" % l, self.bits(L + "fbits", Mt, F), ref, u, mag)
            # FFN2 + dropout2 + residual + LayerNorm2
            g_ref, mag = self.gemm(f, st[pre + "linear2.weight"], st[pre + "linear2.bias"])
            if training:
                k4 = _keep(4 + 4 * l, Mt * D, p).view(Mt, D)
                g_ref, mag = g_ref * k4, mag * k4
            z2_ref, mag = g_ref + h1, mag + h1.abs()
            hout = self.split(L + "hout", Mt, D)
            self.ln("ln", z2_ref, mag, st[pre + "norm2.weight"], st[pre + "norm2.bias"], hout,
                    self.f32(L + "st2", Mt * 2) if self.keep_stats else None,
                    self.split(L + "z2", Mt, D) if self.z_stored else None)
            h = hout
        if prune:
            h_last = self.last_layer(layers - 1, h)
        else:
            h_last = h.view(B, T, D)[:, 0]
        self.head(h_last)
        return self.err

    def attention_stats(self, L, q, k, s, l):
        """Fused training attention: (row max * log2e/8, sum of exp) per query and the dropout keep bits."""
        B, T = self.B, self.T
        BH = B * H
        stat = self.f32(L + "astat", BH * T * 2).view(BH, T, 2)
        smax = s.max(-1).values                         # s = q.k / 8
        scale = (q.abs() @ k.abs().transpose(1, 2)).max(-1).values / 8.0
        l2e = 1.0 / math.log(2.0)
        self.note("stat_max", float(((stat[..., 0] - smax * l2e).abs() / (scale * l2e)).max()))
        sum_ref = torch.exp(s - smax.unsqueeze(-1)).sum(-1)
        self.note("stat_sum", float(((stat[..., 1] - sum_ref).abs() / sum_ref).max()))
        if self.training:
            Tp = (T + 7) // 8 * 8
            nC = (Tp + 15) // 16
            from speaker_embedding_torch_b200 import _native as N
            off, _ = self.lay[L + "abits"]
            base = (self.ws.data_ptr() + 255) // 256 * 256 - self.ws.data_ptr() + off
            words = self.ws[base:base + BH * nC * T * 2].view(torch.int16).view(BH, nC, T).int() & 0xFFFF
            bits = (words.unsqueeze(-1) >> torch.arange(16, device=DEV, dtype=torch.int32)) & 1   # [BH, nC, T, 16]
            bits = bits.permute(0, 2, 1, 3).reshape(BH, T, nC * 16)[..., :T].bool()
            keep = _keep(1 + 4 * l, BH * T * Tp, self.p).view(BH, T, Tp)[..., :T] > 0
            mism = int((bits != keep).sum())
            assert mism == 0, (L, "attention keep bits differ from spk_dropout_keep", mism)

    def last_layer(self, l, h):
        """Pruned last layer: K | V for every frame, everything else for the t = 0 row of each slice."""
        B, T, Mt, st, p = self.B, self.T, self.Mt, self.st, self.p
        pre = "transformer.layers.%d." % l
        w_in, b_in = st[pre + "self_attn.in_proj_weight"], st[pre + "self_attn.in_proj_bias"]
        kv_ref, mag = self.gemm(h, w_in[D:], b_in[D:])
        kv = self.split("last.kv", Mt, 2 * D)
        self.note("gemm", _nerr(kv, kv_ref, mag))
        h_t0 = h.view(B, T, D)[:, 0]
        q0_ref, mag = self.gemm(h_t0, w_in[:D], b_in[:D])
        q0 = self.split("last.q0", B, D)
        self.note("gemm", _nerr(q0, q0_ref, mag))
        kvh = kv.view(B, T, 2, H, 64).permute(2, 0, 3, 1, 4).reshape(2, B * H, T, 64)
        keep = None
        if self.training:
            Tp = (T + 7) // 8 * 8
            keep = _keep(1 + 4 * l, B * H * Tp, p).view(B * H, 1, Tp)[..., :T]
        o_ref, o_mag, o_floor, _ = self.attention(q0.view(B, H, 1, 64).reshape(B * H, 1, 64), kvh[0], kvh[1], keep)
        att0 = self.split("last.att0", B, D)
        self.note("attn", _nerr(att0, o_ref.reshape(B, D), o_mag.reshape(B, D), o_floor.reshape(B, D)))
        a_ref, mag = self.gemm(att0, st[pre + "self_attn.out_proj.weight"], st[pre + "self_attn.out_proj.bias"])
        if self.training:
            k2 = _keep(2 + 4 * l, B * D, p).view(B, D)
            a_ref, mag = a_ref * k2, mag * k2
        z1 = self.split("last.z1", B, D)
        z1_ref, mag = a_ref + h_t0, mag + h_t0.abs()
        self.note("gemm", _nerr(z1, z1_ref, mag))
        h1 = self.split("last.h1", B, D)
        # ln_fwd normalises the stored z1 (its own input)
        self.ln("ln", z1, None, st[pre + "norm1.weight"], st[pre + "norm1.bias"], h1, self.f32("last.st1", B * 2))
        u, mag = self.gemm(h1, st[pre + "linear1.weight"], st[pre + "linear1.bias"])
        f_ref = torch.relu(u)
        if self.training:
            k3 = _keep(3 + 4 * l, B * F, p).view(B, F)
            f_ref, mag = f_ref * k3, mag * k3
        f = self.split("last.f", B, F)
        self.note("gemm", _nerr(f, f_ref, mag))
        g_ref, mag = self.gemm(f, st[pre + "linear2.weight"], st[pre + "linear2.bias"])
        if self.training:
            k4 = _keep(4 + 4 * l, B * D, p).view(B, D)
            g_ref, mag = g_ref * k4, mag * k4
        z2 = self.split("last.z2", B, D)
        z2_ref, mag = g_ref + h1, mag + h1.abs()
        self.note("gemm", _nerr(z2, z2_ref, mag))
        hout = self.split("last.hout", B, D)
        self.ln("ln", z2, None, st[pre + "norm2.weight"], st[pre + "norm2.bias"], hout, self.f32("last.st2", B * 2))
        return hout

    def head(self, h_t0):
        """Final LayerNorm of the t = 0 rows, mean over the samples, projection, L2 normalisation."""
        B, S, st = self.B, self.S, self.st
        U = B // S
        w, b = st["transformer.norm.weight"], st["transformer.norm.bias"]
        hn_ref, mu, rstd = _ln_ref(h_t0, w, b)
        hn = self.f32("hn", B * D).view(B, D)
        hst = self.f32("hst", B * 2).view(B, 2)
        self.note("head", float((hn - hn_ref).abs().max()))
        self.note("head", float(((hst[:, 0] - mu).abs() * rstd).max()))
        self.note("head", float(((hst[:, 1] - rstd).abs() / rstd).max()))
        em = self.f32("emean", U * D).view(U, D)
        self.note("head", float((em - hn.view(U, S, D).mean(1)).abs().max()))
        wp, bp = st["projection.weight"][:, :, 0], st["projection.bias"]
        epre = self.f32("epre", U * D).view(U, D)
        self.note("head", _nerr(epre, em @ wp.t() + bp, em.abs() @ wp.abs().t() + bp.abs()))
        self.dvec_ref = epre / epre.norm(dim=1, keepdim=True)


def _stage_errors(m, state, B, T, precision, training, prune, samples=1, layers=3, keep=True, fln=2):
    mel = torch.as_tensor(synth.make_mel(900 + T, B, T)).to(DEV)
    dvec, ws, lay = _forward_ws(m, mel, samples, precision, training, keep)
    stg = _Stages(ws, lay, _dstate(state), B, T, samples, precision, training, m._cfg.pe_dropout, m._cfg.dropout)
    stg.keep_stats = keep           # LayerNorm statistics and ReLU bits are written for the backward only
    stg.z_stored = keep or fln == 0 or precision > 2      # the fused LayerNorm of inference keeps z in tensor memory
    err = stg.run(layers, prune, h0_emulated=not keep and not prune)
    err["dvec"] = float((dvec.double() - stg.dvec_ref).abs().max())
    return err, stg.flips


def _check(err, P, ctx, ln_floor=0.0):
    """``ln_floor``: what a row offset c adds through the representation of z (test C1) to the mean and the output.  The
    variance has no such allowance: computed about a pivot from the row it does not depend on the offset."""
    b = BOUNDS[P]
    for key, v in err.items():
        if key.endswith(".gate_band"):
            bound = b["gemm"]
        elif key == "dvec":
            bound = b["head"]
        else:
            bound = b[key] + (ln_floor if key in ("ln_mean", "ln_out") else 0.0)
        assert v <= bound, (ctx, key, v, bound)


# ---- B1: training plans (two planes, stash kept), eval and train mode
TRAIN_CASES = [
    # (B, T, training, prune, fused_layernorm, fused_training_attention, training_attention_two_ctas)
    (6, 1, False, 1, 2, 1, 1),
    (6, 7, True, 1, 2, 1, 1),
    (6, 129, True, 0, 2, 1, 1),
    (6, 129, False, 1, 0, 1, 0),
    (4, 192, True, 1, 2, 1, 0),
    (4, 192, True, 0, 0, 0, 1),
    (4, 193, True, 1, 2, 1, 1),
    (2, 300, True, 0, 2, 1, 1),
    (2, 300, False, 1, 0, 1, 1),
    (13, 177, True, 1, 2, 1, 1),
    (13, 177, False, 0, 2, 0, 1),
]


@pytest.mark.parametrize("B,T,training,prune,fln,fta,two", TRAIN_CASES)
def test_training_forward_stages_match_fp64(B, T, training, prune, fln, fta, two):
    """Two-plane forward with the stash: every stage of every layer from the workspace, including the ReLU gate bits,
    the fused attention's row statistics and its dropout keep bits.  13 x 177 = 2301 tokens runs the CTA-pair GEMMs
    with a ragged tail."""
    with _Options(prune_last_layer=prune, fused_layernorm=fln, fused_training_attention=fta,
                  training_attention_two_ctas=two):
        m, state = _model(61)
        err, flips = _stage_errors(m, state, B, T, 2, training, prune, fln=fln)
    _record("train_forward", B=B, T=T, training=training, prune=prune, fln=fln, fta=fta, two=two, err=err, flips=flips)
    _check(err, 2, (B, T))


def test_benchmark_size_training_forward_matches_fp64():
    """960 x 160, the benchmark's batch, train mode (dropout on), default options: forward stages only."""
    m, state = _model(62)
    err, flips = _stage_errors(m, state, 960, 160, 2, True, 1)
    _record("train_forward_960x160", err=err, flips=flips)
    _check(err, 2, (960, 160))


# ---- B1: inference plans (nothing kept: one-layer models, the layer buffers are shared)
@pytest.mark.parametrize("precision", [1, 3])
@pytest.mark.parametrize("prune,fln,B,T", [(1, 2, 6, 129), (0, 2, 6, 129), (0, 0, 4, 193), (0, 2, 13, 177),
                                           (1, 2, 2, 300), (0, 2, 6, 1)])
def test_inference_forward_stages_match_fp64(precision, prune, fln, B, T):
    with _Options(prune_last_layer=prune, fused_layernorm=fln):
        m, state = _model(63, layers=1)
        err, flips = _stage_errors(m, state, B, T, precision, False, prune, layers=1, keep=False, fln=fln)
    _record("infer_forward", P=precision, B=B, T=T, prune=prune, fln=fln, err=err)
    _check(err, precision, (precision, B, T))


# ---- B2: gradients per tensor against the gate-forced fp64 oracle
def _relu_masks(m, B, T, prune, layers=3):
    from speaker_embedding_torch_b200 import _native as N
    ws, meta = m._last_ws, m._last_meta
    lay = N.debug_layout(m._cfg, B, T, meta[2], meta[3], True)
    masks = {"prenet": N.read_bits(ws, lay, "h0bits", B * T, D).view(B, T, D)}
    for l in range(layers):
        if prune and l == layers - 1:
            last = torch.ones(B, T, F, dtype=torch.bool, device=DEV)     # rows t > 0 never reach the d-vector
            last[:, 0] = N.read_split(ws, lay, "last.f", B, F, 2) > 0
            masks["ffn%d" % l] = last
        else:
            masks["ffn%d" % l] = N.read_bits(ws, lay, "L%d.fbits" % l, B * T, F).view(B, T, F)
    return masks


def _oracle(state, mel, utt, samples=1, drop_scales=None, relu_masks=None, cotangent=None):
    st = {k: v.clone().requires_grad_(not k.endswith(".pe")) for k, v in _dstate(state).items()}
    w = torch.tensor(10.0, dtype=torch.float64, device=DEV, requires_grad=True)
    b = torch.tensor(-5.0, dtype=torch.float64, device=DEV, requires_grad=True)
    layers = sum(1 for k in st if k.endswith("norm1.weight"))
    d = O.encoder_forward(st, mel.double(), samples=samples, layers=layers, drop_scales=drop_scales,
                          relu_masks=relu_masks)
    if cotangent is None:
        loss = O.ge2e_loss(d, utt, w, b)
        loss.backward()
        loss = float(loss.detach())
    else:
        d.backward(cotangent.double())
        loss = None
    grads = {k: v.grad for k, v in st.items() if v.requires_grad}
    grads["loss.weight"], grads["loss.bias"] = w.grad, b.grad
    return loss, d.detach(), grads


def _grad_errors(m, g_ref):
    return _rel_errors({name: p.grad for name, p in m.named_parameters()}, g_ref)


def _rel_errors(got, g_ref):
    """{name: relative L2} per tensor; the K slice of every in_proj_bias (zero: softmax is shift-invariant) against
    the norm of its Q slice instead."""
    out = {}
    for name, g in got.items():
        g, r = g.double(), g_ref[name].double()
        if name.endswith("in_proj_bias"):
            out[name + "[k]"] = float((g[D:2 * D] - r[D:2 * D]).norm() / r[:D].norm())
            g = torch.cat([g[:D], g[2 * D:]])
            r = torch.cat([r[:D], r[2 * D:]])
        out[name] = float((g - r).norm() / r.norm())
    return out


def _check_grads(errs, ctx, extra=1.0):
    for name, v in errs.items():
        bound = GRAD_ZERO if name.endswith("[k]") else GRAD_REL
        assert v <= bound * extra, (ctx, name, v)


def _train_step(m, mel, utt, training, samples=1, cotangent=None):
    from speaker_embedding_torch_b200 import GE2E_Loss
    m.train(training)
    m._debug_keep_ws = True
    torch.manual_seed(4242)
    seed = int(torch.empty((), dtype=torch.int64).random_().item())     # what GE2E.forward draws
    torch.manual_seed(4242)
    crit = GE2E_Loss().to(DEV)
    d = m(mel, samples)
    if cotangent is None:
        loss = crit(d, utt)
        loss.backward()
    else:
        loss = None
        d.backward(cotangent)
    torch.cuda.synchronize()
    return seed, d.detach(), loss, crit


GRAD_CASES = [
    # (speakers, utterances, frames, training, prune)
    (4, 3, 24, False, 1),
    (4, 3, 160, False, 1),
    (3, 2, 177, False, 1),
    (2, 2, 300, False, 1),
    (16, 4, 160, False, 1),
    (4, 3, 44, True, 1),
    (4, 3, 44, True, 0),
]


@pytest.mark.parametrize("nspk,utt,T,training,prune", GRAD_CASES)
def test_gradients_per_tensor_match_gate_forced_fp64(nspk, utt, T, training, prune):
    from test_gpu_parity_full import _site_scales
    B = nspk * utt
    with _Options(prune_last_layer=prune):
        m, state = _model(71)
        mel = torch.as_tensor(synth.make_mel(1300 + T, B, T)).to(DEV)
        seed, d, loss, crit = _train_step(m, mel, utt, training)
        masks = _relu_masks(m, B, T, prune)
    ds = None
    if training:
        ds, _ = _site_scales(seed, m._cfg.pe_dropout, m._cfg.dropout, B, T, H, 3, bool(prune), DEV)
        ds = {k: v.to(DEV) for k, v in ds.items()}
    loss_ref, d_ref, g_ref = _oracle(state, mel, utt, drop_scales=ds, relu_masks=masks)
    errs = _grad_errors(m, g_ref)
    errs["loss.weight"] = float(abs(crit.weight.grad.double() - g_ref["loss.weight"]) / abs(g_ref["loss.weight"]))
    loss_rel = abs(loss.item() - loss_ref) / abs(loss_ref)
    dvec = float((d.double() - d_ref).abs().max())
    worst = max(errs.items(), key=lambda kv: kv[1])
    _record("grads", case=[nspk, utt, T, training, prune], loss_rel=loss_rel, dvec=dvec, worst=worst, errs=errs,
            ge2e_bias_grad=crit.bias.grad.item())
    assert loss_rel <= LOSS_REL, loss_rel
    assert dvec <= DVEC_ABS, dvec
    assert abs(crit.bias.grad.item()) <= 1.5e-6, crit.bias.grad     # 2.8e-7; zero: the softmax rows sum to one
    _check_grads(errs, (nspk, utt, T, training, prune))


def test_training_with_samples_and_a_random_cotangent():
    """samples = 5 in train mode (head_bwd with S > 1), d.backward(g) with a random g instead of GE2E's gradient."""
    from test_gpu_parity_full import _site_scales
    B, T, S = 20, 48, 5
    m, state = _model(72)
    mel = torch.as_tensor(synth.make_mel(1400, B, T)).to(DEV)
    g = torch.randn(B // S, D, generator=torch.Generator().manual_seed(5), dtype=torch.float64).float().to(DEV)
    seed, d, _, _ = _train_step(m, mel, None, True, samples=S, cotangent=g)
    masks = _relu_masks(m, B, T, 1)
    ds, _ = _site_scales(seed, m._cfg.pe_dropout, m._cfg.dropout, B, T, H, 3, True, DEV)
    ds = {k: v.to(DEV) for k, v in ds.items()}
    _, d_ref, g_ref = _oracle(state, mel, None, samples=S, drop_scales=ds, relu_masks=masks, cotangent=g)
    errs = _grad_errors(m, g_ref)
    _record("grads_samples5", dvec=float((d.double() - d_ref).abs().max()), errs=errs)
    assert float((d.double() - d_ref).abs().max()) <= DVEC_ABS
    _check_grads(errs, "samples=5")


# ---- C1: LayerNorm under row offsets
def _row_std(state, mel, layers=3, layer=0):
    """Mean spread of the rows of layer ``layer``'s output in fp64 (eval mode): the scale of the next layer's z."""
    _, inter = O.encoder_forward(_dstate(state), mel.double(), layers=layers, return_intermediates=True)
    return float(inter["layer%d" % layer].reshape(-1, D).std(dim=1, unbiased=False).mean())


@pytest.mark.parametrize("fln", [2, 0])
@pytest.mark.parametrize("mult", [0, 16, 64, 256])
def test_training_layernorm_is_exact_under_row_offsets(fln, mult):
    """c = mult x the row spread added to layer 1's out_proj.bias shifts every row of z1 by c; LayerNorm1's output, the
    d-vectors and every gradient are unchanged in exact arithmetic.  The bounds may grow by what the fp32 / two-plane
    representation of z costs (c * 2^-24 in the forward, c * 2^-22 in the stored z the backward reads), not more."""
    B, T, utt = 12, 44, 3
    mel = torch.as_tensor(synth.make_mel(900 + T, B, T)).to(DEV)
    _, base = _model(81)
    c = mult * _row_std(base, mel)
    with _Options(fused_layernorm=fln):
        m, state = _model(81, bias_offset=("transformer.layers.1.self_attn.out_proj.bias", c))
        err, _ = _stage_errors(m, state, B, T, 2, False, 1, fln=fln)
        _, d, loss, crit = _train_step(m, mel, utt, False)
        masks = _relu_masks(m, B, T, 1)
    _, d_ref, g_ref = _oracle(state, mel, utt, relu_masks=masks)
    errs = _grad_errors(m, g_ref)
    worst = max(errs.items(), key=lambda kv: kv[1])
    _record("ln_offset_train", fln=fln, mult=mult, err=err, worst=worst)
    _check(err, 2, ("offset", mult, fln), ln_floor=mult * 2.0 ** -20)
    _check_grads(errs, ("offset", mult, fln), extra=1.0 + mult * 2.0 ** -22 / GRAD_REL)


@pytest.mark.parametrize("fln", [2, 0])
@pytest.mark.parametrize("mult", [0, 16, 64, 256])
def test_inference_layernorm_is_exact_under_row_offsets(fln, mult):
    """One plane, one dense layer: c added to linear2.bias shifts z2 (LayerNorm2 runs in the FFN2 epilogue when
    fused)."""
    B, T = 6, 129
    mel = torch.as_tensor(synth.make_mel(900 + T, B, T)).to(DEV)
    _, base = _model(82, layers=1)
    c = mult * _row_std(base, mel, layers=1)
    with _Options(prune_last_layer=0, fused_layernorm=fln):
        m, state = _model(82, layers=1, bias_offset=("transformer.layers.0.linear2.bias", c))
        err, _ = _stage_errors(m, state, B, T, 1, False, 0, layers=1, keep=False, fln=fln)
    _record("ln_offset_infer", fln=fln, mult=mult, err=err)
    # unfused, z2 is stored in one fp16 plane for ln_fwd: c * 2^-11 of representation (measured 0.13 at 256 sigma)
    _check(err, 1, ("offset", mult, fln), ln_floor=mult * (2.0 ** -20 if fln else 1.5 * 2.0 ** -11))


# ---- C2: the gradient-scale contract
def _grads_for(m, mel, g):
    m.zero_grad(set_to_none=True)
    _train_step(m, mel, None, False, cotangent=g)
    return {n: p.grad.detach().clone() for n, p in m.named_parameters()}


def test_gradient_scale_contract():
    B, T = 12, 44
    m, state = _model(91)
    mel = torch.as_tensor(synth.make_mel(1600, B, T)).to(DEV)
    g = torch.randn(B, D, generator=torch.Generator().manual_seed(9)).to(DEV)
    g1 = _grads_for(m, mel, g)
    masks = _relu_masks(m, B, T, 1)
    _, _, g_ref = _oracle(state, mel, None, relu_masks=masks, cotangent=g)
    # power-of-two multiples of g: the same planes, only the split-K fp32 atomics reorder
    pow2 = {}
    for c in (2.0 ** -20, 2.0 ** 16, 2.0 ** 24):
        gc = _grads_for(m, mel, g * c)
        errs = _rel_errors({n: t / c for n, t in gc.items()}, g1)
        pow2[c] = max((v, n) for n, v in errs.items() if not n.endswith("[k]"))
        _check_grads(errs, ("2^%d" % round(math.log2(c))))
    # other multiples and other gradient-scale targets: against fp64
    fp64 = {}
    for c in (1.0, 1.0 / 3.0, 1000.0):
        m.zero_grad(set_to_none=True)
        _train_step(m, mel, None, False, cotangent=g * c)
        errs = _grad_errors(m, {k: v * c for k, v in g_ref.items() if v is not None})
        fp64["c=%g" % c] = max(errs.items(), key=lambda kv: kv[1])
        _check_grads(errs, ("c", c))
    for k in (8, 12, 15):
        with _Options(grad_scale_log2=k):
            m.zero_grad(set_to_none=True)
            _train_step(m, mel, None, False, cotangent=g)
            errs = _grad_errors(m, g_ref)
        fp64["log2=%d" % k] = max(errs.items(), key=lambda kv: kv[1])
        _check_grads(errs, ("grad_scale_log2", k))
    _record("grad_scale", pow2={str(k): v for k, v in pow2.items()}, fp64=fp64)
    for c, (v, n) in pow2.items():
        assert v <= POW2_REL, (c, n, v)
    # zero upstream gradient: exactly zero, finite
    g0 = _grads_for(m, mel, torch.zeros_like(g))
    for n, t in g0.items():
        assert torch.isfinite(t).all() and (t == 0).all(), n


@pytest.mark.parametrize("bad", [float("nan"), float("inf")])
def test_non_finite_upstream_gradient_reaches_the_parameters(bad):
    """One NaN / +inf in the cotangent: every parameter gradient autograd makes non-finite is non-finite here too, so
    a loss scaler sees the overflow and skips the step."""
    B, T = 12, 44
    m, state = _model(92)
    mel = torch.as_tensor(synth.make_mel(1700, B, T)).to(DEV)
    g = torch.randn(B, D, generator=torch.Generator().manual_seed(11)).to(DEV)
    g[3, 17] = bad
    ours = _grads_for(m, mel, g)
    _, _, ref = _oracle(state, mel, None, cotangent=g)
    for n, t in ours.items():
        assert bool(torch.isfinite(t).all()) == bool(torch.isfinite(ref[n]).all()), n
        assert not torch.isfinite(t).all(), n
