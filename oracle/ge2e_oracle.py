"""CPU restatement of the reference hot path (encoder -> d-vector head -> GE2E loss).

TEST INFRASTRUCTURE (see oracle/__init__.py) -- never imported by the product.

The reference's arithmetic lives in PyTorch library modules
(``nn.TransformerEncoder``, ``nn.Conv1d``, ``nn.LayerNorm``,
``nn.CosineSimilarity``, ``nn.CrossEntropyLoss``; torch 2.11.0 in this image).
This file restates that arithmetic as plain matmuls / reductions on CPU so the
CUDA kernels can be checked stage by stage and in fp64.  It is pinned against
the reference's own modules by ``oracle/make_golden.py`` ->
``tests/golden/*.npz`` -> ``tests/test_oracle_golden.py``.

Reference sites followed:
  * encoder forward order ........ /root/reference/Modules.py:46-59
  * k=1 Conv1d prenet/projection . /root/reference/Modules.py:10-17,38-44,61-72
  * positional encoding .......... /root/reference/Modules.py:76-109
  * post-LN encoder layer ........ torch.nn.TransformerEncoderLayer (norm_first=False,
                                   relu, batch_first=False) as built at Modules.py:25-36
  * GE2E loss .................... /root/reference/Modules.py:112-156
"""
import math

import numpy as np
import torch

LN_EPS = 1e-5          # torch.nn.LayerNorm default (Modules.py:33-35)
NORMALIZE_EPS = 1e-12  # F.normalize default (Modules.py:57)
COS_EPS = 1e-8         # nn.CosineSimilarity default (Modules.py:118)


def to_torch_state(state, dtype=torch.float32, requires_grad=False):
    out = {}
    for k, v in state.items():
        t = torch.as_tensor(np.asarray(v)).to(dtype).clone()
        if requires_grad and not k.endswith(".pe"):
            t.requires_grad_(True)
        out[k] = t
    return out


def _layer_norm(x, w, b):
    # biased variance over the last dim, eps inside the sqrt (torch native_layer_norm)
    mu = x.mean(dim=-1, keepdim=True)
    xc = x - mu
    var = (xc * xc).mean(dim=-1, keepdim=True)
    return xc / torch.sqrt(var + LN_EPS) * w + b


def _dropout(x, p, gen, scale=None):
    if scale is not None:           # explicit keep-scales (0 or 1/(1-p)), e.g. the masks the CUDA kernels used
        return x * scale.to(x.dtype)
    if p <= 0.0:
        return x
    keep = (torch.rand(x.shape, generator=gen, dtype=torch.float32) >= p).to(x.dtype)
    return x * keep / (1.0 - p)


def encoder_forward(state, mel, samples=1, heads=4, layers=3, dropout_p=0.0, gen=None,
                    return_intermediates=False, drop_scales=None, relu_masks=None):
    """d-vectors [B/samples, D] from mel [B, mel_dim, T]  (Modules.py:46-59).

    ``state`` is a dict of torch tensors with the reference's state_dict names.
    Token-major restatement: h is [B, T, D]; every k=1 conv / linear is h @ W^T + b.
    ``dropout_p`` > 0 reproduces the reference's 13 train-mode dropout sites
    statistically (the RNG stream differs; SURVEY.md D9).  ``drop_scales`` = {site: keep-scale tensor}
    replaces the random masks by given ones (sites numbered as in include/spkemb.h: 0 positional encoding,
    1 + 4l attention probabilities [B, H, T, T], 2 + 4l dropout1, 3 + 4l FFN inner [B, T, 4D], 4 + 4l dropout2),
    which is how the tests check that the CUDA forward and backward apply one and the same mask per site.
    ``relu_masks`` = {site: bool tensor} likewise replaces ``relu(u)`` by ``u * mask`` (sites ``"prenet"`` [B, T, D]
    and ``"ffn<l>"`` [B, T, 4D]): fed the gates a kernel chose, the fp64 gradients are those of the kernel's own
    piecewise-linear function, free of the gates that flip when a pre-activation lies within rounding of zero.
    """
    ds = drop_scales or {}
    rm = relu_masks or {}

    def relu(u, site):
        return u * rm[site].to(u.dtype) if site in rm else torch.relu(u)

    x = mel.transpose(1, 2)                                   # [B, T, mel]
    B, T, _ = x.shape
    w_pre = state["prenet.weight"][:, :, 0]                   # [D, mel]
    h = relu(x @ w_pre.t() + state["prenet.bias"], "prenet")  # Modules.py:50-51
    D = h.shape[-1]
    pe = state["positional_encoding.pe"][0, :, :T].t()        # [T, D]  (Modules.py:107-109)
    h = h + state["positional_encoding.alpha"] * pe           # Modules.py:102
    h = _dropout(h, dropout_p, gen, ds.get(0))                # Modules.py:103
    dh = D // heads
    inter = {"embed": h}
    for l in range(layers):
        p = "transformer.layers.%d." % l
        w_in, b_in = state[p + "self_attn.in_proj_weight"], state[p + "self_attn.in_proj_bias"]
        qkv = h @ w_in.t() + b_in                             # [B, T, 3D]  rows Wq | Wk | Wv
        q, k, v = qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:]
        q = q.reshape(B, T, heads, dh).transpose(1, 2)        # [B, H, T, dh]
        k = k.reshape(B, T, heads, dh).transpose(1, 2)
        v = v.reshape(B, T, heads, dh).transpose(1, 2)
        s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)         # SDPA scale 1/sqrt(64)
        pr = torch.softmax(s, dim=-1)
        pr = _dropout(pr, dropout_p, gen, ds.get(1 + 4 * l))  # attention-prob dropout
        a = (pr @ v).transpose(1, 2).reshape(B, T, D)
        a = a @ state[p + "self_attn.out_proj.weight"].t() + state[p + "self_attn.out_proj.bias"]
        h = _layer_norm(h + _dropout(a, dropout_p, gen, ds.get(2 + 4 * l)), state[p + "norm1.weight"],
                        state[p + "norm1.bias"])
        f = relu(h @ state[p + "linear1.weight"].t() + state[p + "linear1.bias"], "ffn%d" % l)
        f = _dropout(f, dropout_p, gen, ds.get(3 + 4 * l))
        f = f @ state[p + "linear2.weight"].t() + state[p + "linear2.bias"]
        h = _layer_norm(h + _dropout(f, dropout_p, gen, ds.get(4 + 4 * l)), state[p + "norm2.weight"],
                        state[p + "norm2.bias"])
        inter["layer%d" % l] = h
    h0 = _layer_norm(h[:, 0, :], state["transformer.norm.weight"], state["transformer.norm.bias"])  # Modules.py:33-35,54
    e = h0.reshape(-1, samples, D).mean(dim=1)                # Modules.py:55
    e = e @ state["projection.weight"][:, :, 0].t() + state["projection.bias"]   # Modules.py:56
    n = e.norm(p=2, dim=1, keepdim=True).clamp_min(NORMALIZE_EPS)
    d = e / n                                                 # Modules.py:57
    if return_intermediates:
        inter["pre_norm"] = e
        return d, inter
    return d


def ge2e_loss(emb, per_speaker, weight=10.0, bias=-5.0):
    """Mean CE of w*cos(e_i, c_k) - b against the row's own speaker (Modules.py:121-156).

    Restated (SURVEY.md D2): the reference's "within" column uses the *inclusive* sum
    centroid, which after cosine normalisation equals the diagonal of the "between"
    matrix, and moving the true class to column 0 does not change cross-entropy.
    Each norm is clamped separately at 1e-8 (torch cosine_similarity).
    """
    NM, D = emb.shape
    N = NM // per_speaker
    c = emb.reshape(N, per_speaker, D).mean(dim=1)
    en = emb / emb.norm(dim=1, keepdim=True).clamp_min(COS_EPS)
    cn = c / c.norm(dim=1, keepdim=True).clamp_min(COS_EPS)
    z = weight * (en @ cn.t()) - bias
    labels = torch.arange(N).repeat_interleave(per_speaker)
    lse = torch.logsumexp(z, dim=1)
    return (lse - z[torch.arange(NM), labels]).mean()


def ge2e_loss_and_grads_closed_form(emb, per_speaker, weight=10.0, bias=-5.0):
    """fp64 numpy closed form of loss, dE, dw, db (SURVEY.md Appendix B).

    Used to check the fused CUDA kernel where autograd through the reference's
    O(N^2 M D) expansion does not fit (N > 512).
    """
    E = np.asarray(emb, dtype=np.float64)
    NM, D = E.shape
    M = per_speaker
    N = NM // M
    c = E.reshape(N, M, D).mean(axis=1)
    ne = np.maximum(np.linalg.norm(E, axis=1, keepdims=True), COS_EPS)
    nc = np.maximum(np.linalg.norm(c, axis=1, keepdims=True), COS_EPS)
    eh, ch = E / ne, c / nc
    S = eh @ ch.T
    z = weight * S - bias
    zmax = z.max(axis=1, keepdims=True)
    ex = np.exp(z - zmax)
    p = ex / ex.sum(axis=1, keepdims=True)
    lab = np.repeat(np.arange(N), M)
    loss = float(np.mean(np.log(ex.sum(axis=1)) + zmax[:, 0] - z[np.arange(NM), lab]))
    y = np.zeros_like(p)
    y[np.arange(NM), lab] = 1.0
    pm = (p - y) / NM
    dw = float((pm * S).sum())
    db = float(-pm.sum())
    G = weight * pm
    de_h = G @ ch
    dc_h = G.T @ eh
    dE = (de_h - (de_h * eh).sum(1, keepdims=True) * eh) / ne
    dc = (dc_h - (dc_h * ch).sum(1, keepdims=True) * ch) / nc
    dE = dE + np.repeat(dc, M, axis=0) / M
    return loss, dE, dw, db


def ge2e_closed_form_chunked(emb, per_speaker, weight=10.0, bias=-5.0, rows_per_chunk=4096):
    """The closed form above evaluated in row chunks, so that N = 4096 (a 61 440 x 4 096 logit matrix, 2 GB in
    fp64) never exists at once.  Same results as ``ge2e_loss_and_grads_closed_form`` (checked in the CPU tests)."""
    E = np.asarray(emb, dtype=np.float64)
    NM, D = E.shape
    M = per_speaker
    N = NM // M
    c = E.reshape(N, M, D).mean(axis=1)
    ne = np.maximum(np.linalg.norm(E, axis=1, keepdims=True), COS_EPS)
    nc = np.maximum(np.linalg.norm(c, axis=1, keepdims=True), COS_EPS)
    eh, ch = E / ne, c / nc
    lab = np.repeat(np.arange(N), M)
    loss = 0.0
    dw = 0.0
    db = 0.0
    de_h = np.empty_like(E)
    dc_h = np.zeros_like(c)
    for r0 in range(0, NM, rows_per_chunk):
        r1 = min(NM, r0 + rows_per_chunk)
        S = eh[r0:r1] @ ch.T
        z = weight * S - bias
        zmax = z.max(axis=1, keepdims=True)
        ex = np.exp(z - zmax)
        den = ex.sum(axis=1, keepdims=True)
        rows = np.arange(r1 - r0)
        loss += float(np.sum(np.log(den[:, 0]) + zmax[:, 0] - z[rows, lab[r0:r1]]))
        pm = ex / den
        pm[rows, lab[r0:r1]] -= 1.0
        pm /= NM
        dw += float((pm * S).sum())
        db += float(-pm.sum())
        G = weight * pm
        de_h[r0:r1] = G @ ch
        dc_h += G.T @ eh[r0:r1]
    dE = (de_h - (de_h * eh).sum(1, keepdims=True) * eh) / ne
    dc = (dc_h - (dc_h * ch).sum(1, keepdims=True) * ch) / nc
    dE = dE + np.repeat(dc, M, axis=0) / M
    return loss / NM, dE, dw, db


def train_step_grads(state_np, mel_np, per_speaker, weight=10.0, bias=-5.0, dtype=torch.float64,
                     samples=1, drop_scales=None, relu_masks=None):
    """Loss, d-vectors and every parameter gradient via autograd through the restatement."""
    st = to_torch_state(state_np, dtype=dtype, requires_grad=True)
    w = torch.tensor(weight, dtype=dtype, requires_grad=True)
    b = torch.tensor(bias, dtype=dtype, requires_grad=True)
    d = encoder_forward(st, torch.as_tensor(mel_np).to(dtype), samples=samples, drop_scales=drop_scales,
                        relu_masks=relu_masks)
    loss = ge2e_loss(d, per_speaker, w, b)
    loss.backward()
    grads = {k: v.grad.detach().numpy() for k, v in st.items() if v.requires_grad}
    grads["loss.weight"] = w.grad.numpy()
    grads["loss.bias"] = b.grad.numpy() if b.grad is not None else np.zeros(())
    return float(loss.detach()), d.detach().numpy(), grads


# --- optimiser restatements (SURVEY.md 8f N2; /root/reference/Radam.py:25-90,
#     /root/reference/Noam_Scheduler.py:17-29, /root/reference/Train.py:154-159) -------------

def clip_coef(total_norm, max_norm):
    """torch.nn.utils.clip_grad_norm_ scale factor (Train.py:154-159)."""
    return min(1.0, max_norm / (total_norm + 1e-6))


def modified_noam_lr(base_lr, step, base):
    """Modified_Noam_Scheduler.get_lr (Noam_Scheduler.py:25-29); step = last_epoch."""
    last = max(1, step)
    return base_lr * base ** 0.5 * (last + base) ** (-0.5)


def radam_step(p, g, m, v, step, lr, beta1=0.9, beta2=0.999, eps=1e-6, weight_decay=0.0):
    """One RAdam update on fp64 numpy arrays, in place (Radam.py:47-88). ``step`` is 1-based."""
    v *= beta2
    v += (1 - beta2) * g * g
    m *= beta1
    m += (1 - beta1) * g
    beta2_t = beta2 ** step
    n_sma_max = 2 / (1 - beta2) - 1
    n_sma = n_sma_max - 2 * step * beta2_t / (1 - beta2_t)
    if n_sma >= 5:
        step_size = math.sqrt((1 - beta2_t) * (n_sma - 4) / (n_sma_max - 4) * (n_sma - 2) / n_sma
                              * n_sma_max / (n_sma_max - 2)) / (1 - beta1 ** step)
    else:
        step_size = 1.0 / (1 - beta1 ** step)
    if weight_decay != 0:
        p += -weight_decay * lr * p
    if n_sma >= 5:
        p += -step_size * lr * m / (np.sqrt(v) + eps)
    else:
        p += -step_size * lr * m
    return p
