"""fp64 references for the GE2E paper's loss variants (test infrastructure; never imported by the product).

Notation (DESIGN.md §3.3): rows are speaker-major, i = j*M + m; logits z = w * cos - b;
cos(a, b) = a.b / (max(|a|, eps) * max(|b|, eps)), eps = 1e-8.
  * inclusive centroids: c_j = mean_m e_jm, used by every column (the reference's loss, ``oracle.ge2e_loss``);
  * exclusive centroids: the own-speaker column of row i uses c_j^(-i) = sum_{k in j, k != i} e_k / (M - 1) (eq. 8);
    every other column keeps the inclusive c_k (eq. 9);
  * softmax loss: L_i = logsumexp_k z_ik - z_i,own (eq. 6);
  * contrast loss: L_i = 1 - sigmoid(z_i,own) + sigmoid(z_i,k*), k* = argmax_{k != own} z_ik, ties to the lowest k
    (eq. 7);
  * the loss is the mean over the N*M rows.

``ge2e_loss_variant`` is written literally from those equations, row by row, so that autograd gives the reference
gradients.  ``ge2e_variant_closed_form`` is the algorithm of the kernels (one G matrix, the diagonal's own gradient
terms) in numpy fp64; it shares no code with the literal form.  ``train_step_grads_variant`` is
``oracle.ge2e_oracle.train_step_grads`` with a variant loss in place of the reference's.
"""
import numpy as np
import torch

from oracle import ge2e_oracle as O

METHODS = ("softmax", "contrast")
CENTROIDS = ("inclusive", "exclusive")
MODES = [(m, c) for m in METHODS for c in CENTROIDS]


def mode_bits(method, centroids):
    """The SPK_GE2E_* mode of include/spkemb.h."""
    return (1 if method == "contrast" else 0) | ((1 << 8) if centroids == "exclusive" else 0)


def ge2e_loss_variant(emb, M, w, b, method, centroids):
    """Literal restatement of eqs. 6-9 on a torch tensor [N*M, D] (autograd-able in emb, w, b)."""
    NM = emb.shape[0]
    N = NM // M
    cos = torch.nn.functional.cosine_similarity
    inclusive = [emb[j * M:(j + 1) * M].mean(dim=0) for j in range(N)]
    losses = []
    for i in range(NM):
        j = i // M
        e = emb[i]
        z = []
        for k in range(N):
            if k == j and centroids == "exclusive":
                others = [emb[r] for r in range(j * M, (j + 1) * M) if r != i]
                c = torch.stack(others).sum(dim=0) / (M - 1)
            else:
                c = inclusive[k]
            z.append(w * cos(e, c, dim=0, eps=O.COS_EPS) - b)
        z = torch.stack(z)
        if method == "softmax":
            losses.append(torch.logsumexp(z, dim=0) - z[j])
        else:
            kstar = None
            for k in range(N):
                if k != j and (kstar is None or float(z[k].detach()) > float(z[kstar].detach())):
                    kstar = k
            losses.append(1.0 - torch.sigmoid(z[j]) + torch.sigmoid(z[kstar]))
    return torch.stack(losses).mean()


def literal_loss_and_grads(E, M, w, b, method, centroids):
    """(loss, dE, dw, db) of ``ge2e_loss_variant`` by autograd in fp64."""
    e = torch.tensor(np.asarray(E, dtype=np.float64), requires_grad=True)
    wt = torch.tensor(float(w), dtype=torch.float64, requires_grad=True)
    bt = torch.tensor(float(b), dtype=torch.float64, requires_grad=True)
    loss = ge2e_loss_variant(e, M, wt, bt, method, centroids)
    loss.backward()
    db = float(bt.grad) if bt.grad is not None else 0.0
    return float(loss.detach()), e.grad.numpy(), float(wt.grad), db


def ge2e_variant_closed_form_chunked(E, M, w=10.0, b=-5.0, method="softmax", centroids="inclusive",
                                     rows_per_chunk=4096):
    """fp64 closed form in row chunks (N = 4096 never holds the 61 440 x 4 096 logits at once).

    Returns loss, dE, dw, db and each row's gap between its two largest off-diagonal cosines (inf for N = 2)."""
    E = np.asarray(E, dtype=np.float64)
    NM, D = E.shape
    N = NM // M
    w, b = float(w), float(b)
    excl = centroids == "exclusive"
    sums = E.reshape(N, M, D).sum(axis=1)
    c = sums / M
    ne = np.maximum(np.linalg.norm(E, axis=1, keepdims=True), O.COS_EPS)
    nc = np.maximum(np.linalg.norm(c, axis=1, keepdims=True), O.COS_EPS)
    eh, ch = E / ne, c / nc
    lab = np.repeat(np.arange(N), M)
    if excl:
        u = sums[lab] - E                                                  # sum of the speaker's other rows
        nu = np.maximum(np.linalg.norm(u, axis=1, keepdims=True) / (M - 1), O.COS_EPS)
        cu = u / (M - 1) / nu                                              # unit exclusive centroid
        cos_own = (eh * cu).sum(axis=1)
        gdiag = np.zeros(NM)
    loss = dw = db = 0.0
    gap = np.empty(NM)
    de_h = np.empty_like(E)
    dc_h = np.zeros_like(c)
    for r0 in range(0, NM, rows_per_chunk):
        r1 = min(NM, r0 + rows_per_chunk)
        rows = np.arange(r1 - r0)
        own = lab[r0:r1]
        S = eh[r0:r1] @ ch.T
        if excl:
            S[rows, own] = cos_own[r0:r1]
        z = w * S - b
        off = S.copy()
        off[rows, own] = -np.inf
        if N > 2:
            top2 = -np.partition(-off, 1, axis=1)[:, :2]
            gap[r0:r1] = top2[:, 0] - top2[:, 1]
        else:
            gap[r0:r1] = np.inf
        if method == "softmax":
            zmax = z.max(axis=1, keepdims=True)
            ex = np.exp(z - zmax)
            den = ex.sum(axis=1, keepdims=True)
            loss += float(np.sum(np.log(den[:, 0]) + zmax[:, 0] - z[rows, own]))
            dz = ex / den
            dz[rows, own] -= 1.0
        else:
            zoff = z.copy()
            zoff[rows, own] = -np.inf
            kstar = np.argmax(zoff, axis=1)                                # first maximum: the lowest index
            zo, zk = z[rows, own], z[rows, kstar]
            so, son = 1.0 / (1.0 + np.exp(-zo)), 1.0 / (1.0 + np.exp(zo))     # sigmoid(z), 1 - sigmoid(z)
            sk, skn = 1.0 / (1.0 + np.exp(-zk)), 1.0 / (1.0 + np.exp(zk))
            loss += float(np.sum(son + sk))
            dz = np.zeros_like(z)
            dz[rows, own] = -so * son
            dz[rows, kstar] = sk * skn
        pm = dz / NM
        dw += float((pm * S).sum())
        db += float(-pm.sum())
        G = w * pm
        if excl:
            gdiag[r0:r1] = G[rows, own]
            G[rows, own] = 0.0
        de_h[r0:r1] = G @ ch
        dc_h += G.T @ eh[r0:r1]
    dE = (de_h - (de_h * eh).sum(1, keepdims=True) * eh) / ne
    dc = (dc_h - (dc_h * ch).sum(1, keepdims=True) * ch) / nc
    dE = dE + np.repeat(dc, M, axis=0) / M
    if excl:
        g = gdiag[:, None]
        co = cos_own[:, None]
        dE += g * (cu - co * eh) / ne                                      # row i through its own e_i
        v = g * (eh - co * cu) / (nu * (M - 1))                            # every other row of the speaker
        V = v.reshape(N, M, D).sum(axis=1)
        dE += V[lab] - v
    return loss / NM, dE, dw, db, gap


def ge2e_variant_closed_form(E, M, w=10.0, b=-5.0, method="softmax", centroids="inclusive"):
    """The closed form above in one chunk (the whole logit matrix at once)."""
    return ge2e_variant_closed_form_chunked(E, M, w, b, method, centroids, rows_per_chunk=np.asarray(E).shape[0])


def train_step_grads_variant(state_np, mel_np, per_speaker, method, centroids, weight=10.0, bias=-5.0,
                             dtype=torch.float64, samples=1):
    """Loss, d-vectors and every parameter gradient via autograd through the encoder restatement and the literal
    variant loss (``oracle.ge2e_oracle.train_step_grads`` with ``ge2e_loss_variant`` as the loss)."""
    st = O.to_torch_state(state_np, dtype=dtype, requires_grad=True)
    w = torch.tensor(weight, dtype=dtype, requires_grad=True)
    b = torch.tensor(bias, dtype=dtype, requires_grad=True)
    d = O.encoder_forward(st, torch.as_tensor(mel_np).to(dtype), samples=samples)
    loss = ge2e_loss_variant(d, per_speaker, w, b, method, centroids)
    loss.backward()
    grads = {k: v.grad.detach().numpy() for k, v in st.items() if v.requires_grad}
    grads["loss.weight"] = w.grad.numpy()
    grads["loss.bias"] = b.grad.numpy() if b.grad is not None else np.zeros(())
    return float(loss.detach()), d.detach().numpy(), grads


def planted_embeddings(seed, speakers, utterances, emb=256, unit_norm=True):
    """Embeddings [speakers*utterances, emb] fp32 whose off-diagonal cosines have a clear maximum in every row, so that
    the contrast loss's k* is the same in fp32 and fp64: row (j, m) = base_j + 0.8 base_(impostor) + 0.15 noise, with
    a random impostor per row and random unit base directions."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((speakers, emb))
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    lab = np.repeat(np.arange(speakers), utterances)
    imp = (lab + 1 + rng.integers(0, speakers - 1, size=lab.shape)) % speakers
    e = base[lab] + 0.8 * base[imp] + 0.15 * rng.standard_normal((lab.size, emb)) / np.sqrt(emb)
    if unit_norm:
        e /= np.linalg.norm(e, axis=1, keepdims=True)
    else:
        e *= 0.5 + rng.random((lab.size, 1))
    return e.astype(np.float32)
