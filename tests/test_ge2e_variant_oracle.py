"""The GE2E variants' fp64 closed form (the kernels' algorithm) against the literal restatement of the paper's equations,
and the host-side checks of the variant entry points.  No GPU needed."""
import ctypes

import numpy as np
import pytest

from ge2e_variant_oracle import (MODES, ge2e_variant_closed_form, ge2e_variant_closed_form_chunked,
                                 literal_loss_and_grads, mode_bits, planted_embeddings)
from oracle import ge2e_oracle as O
from oracle import synth


def _close(a, b, tol=1e-10):
    return abs(a - b) <= tol * max(1.0, abs(b))


@pytest.mark.parametrize("method,centroids", MODES)
@pytest.mark.parametrize("n,m", [(2, 2), (3, 5), (7, 3), (16, 4)])
@pytest.mark.parametrize("unit", [True, False])
def test_closed_form_matches_the_literal_equations(method, centroids, n, m, unit):
    E = synth.make_embeddings(40 + 7 * n + m, n, m, unit_norm=unit)
    w, b = 7.5, -3.0
    l_ref, dE_ref, dw_ref, db_ref = literal_loss_and_grads(E, m, w, b, method, centroids)
    loss, dE, dw, db, gap = ge2e_variant_closed_form_chunked(E, m, w, b, method, centroids, rows_per_chunk=5)
    if method == "contrast":
        assert gap.min() > 1e-9            # k* is well defined, so the literal form's choice is the closed form's
    assert _close(loss, l_ref)
    assert np.abs(dE - dE_ref).max() <= 1e-10 * max(1.0, np.abs(dE_ref).max())
    assert _close(dw, dw_ref)
    assert _close(db, db_ref)
    if method == "softmax":
        assert abs(db) <= 1e-12            # sum_k (p_k - onehot_k) = 0 per row
    # chunked and unchunked agree
    one = ge2e_variant_closed_form(E, m, w, b, method, centroids)
    assert _close(one[0], loss, 1e-12) and _close(one[2], dw, 1e-12) and _close(one[3], db, 1e-12)
    assert np.abs(one[1] - dE).max() <= 1e-12 * max(1.0, np.abs(dE).max())


@pytest.mark.parametrize("n,m", [(3, 5), (16, 4)])
def test_inclusive_softmax_is_the_reference_loss(n, m):
    E = synth.make_embeddings(90 + n, n, m, unit_norm=False)
    loss, dE, dw, db, _ = ge2e_variant_closed_form(E, m)
    l_ref, dE_ref, dw_ref, db_ref = O.ge2e_loss_and_grads_closed_form(E, m)
    assert _close(loss, l_ref, 1e-12) and _close(dw, dw_ref, 1e-12)
    assert np.abs(dE - dE_ref).max() <= 1e-12 * np.abs(dE_ref).max()


def test_ties_go_to_the_lowest_speaker():
    """Speakers 1 and 2 have identical rows, so their centroids tie in every other row; the literal form (an explicit
    first-maximum scan) and the closed form (numpy argmax) both give the gradient to speaker 1."""
    E = planted_embeddings(5, 4, 3)
    E[6:9] = E[3:6]
    for centroids in ("inclusive", "exclusive"):
        l_ref, dE_ref, dw_ref, db_ref = literal_loss_and_grads(E, 3, 10.0, -5.0, "contrast", centroids)
        loss, dE, dw, db, _ = ge2e_variant_closed_form(E, 3, 10.0, -5.0, "contrast", centroids)
        assert _close(loss, l_ref) and _close(dw, dw_ref) and _close(db, db_ref)
        assert np.abs(dE - dE_ref).max() <= 1e-10 * np.abs(dE_ref).max()
        assert np.abs(dE[3:6] - dE[6:9]).max() > 0.1 * np.abs(dE).max()      # the tie is broken, not shared


def test_variant_entry_points_refuse_bad_modes_on_the_host():
    """spk_ge2e_workspace_bytes_ex / spk_ge2e_loss_ex: mode 0 sizes like spk_ge2e_workspace_bytes; unknown bits,
    exclusive with one utterance and contrast with one speaker return SPK_EINVAL before any CUDA call."""
    from speaker_embedding_torch_b200 import _native
    L = _native.lib()
    assert L.spk_ge2e_workspace_bytes_ex(1, 1, 0) == L.spk_ge2e_workspace_bytes(1, 1)
    for n, m in ((64, 15), (255, 3), (256, 3), (4096, 15)):
        assert L.spk_ge2e_workspace_bytes_ex(n, m, 0) == L.spk_ge2e_workspace_bytes(n, m)
        assert L.spk_ge2e_workspace_bytes_ex(n, m, 1) == L.spk_ge2e_workspace_bytes(n, m)
    for n, m in ((64, 15), (256, 3)):
        assert L.spk_ge2e_workspace_bytes_ex(n, m, 256) >= L.spk_ge2e_workspace_bytes(n, m) + 3 * n * m * 4
    fake = ctypes.c_void_p(256)            # never dereferenced: every call below is refused on the host
    cases = [(4, 3, 2, "unknown mode bits"), (4, 3, 1 << 9, "unknown mode bits"),
             (4, 1, mode_bits("softmax", "exclusive"), "at least 2 utterances"),
             (1, 4, mode_bits("contrast", "inclusive"), "at least 2 speakers")]
    for n, m, mode, msg in cases:
        assert L.spk_ge2e_workspace_bytes_ex(n, m, mode) == 0
        assert msg in L.spk_last_error().decode()
        rc = L.spk_ge2e_loss_ex(fake, n, m, 256, mode, fake, fake, fake, None, None, None, fake, 1 << 20, None)
        assert rc == -22
        assert msg in L.spk_last_error().decode()


def test_bad_keywords_raise_value_error():
    from speaker_embedding_torch_b200 import GE2E_Loss
    with pytest.raises(ValueError, match="loss_method"):
        GE2E_Loss(loss_method="triplet")
    with pytest.raises(ValueError, match="centroids"):
        GE2E_Loss(centroids="Exclusive")
    crit = GE2E_Loss()
    assert set(crit.state_dict()) == {"weight", "bias"}          # the variant is configuration, not state
