"""Fused GE2E kernel vs the reference's own outputs (tests/golden/ge2e_loss.npz) and the fp64 closed form."""
import os

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth
from oracle.make_golden import stored_rows

pytestmark = pytest.mark.gpu


def _run(E, M, w=10.0, b=-5.0, grad=True):
    from speaker_embedding_torch_b200 import GE2E_Loss
    crit = GE2E_Loss(init_weight=w, init_bias=b).cuda()
    e = torch.as_tensor(E).cuda().requires_grad_(grad)
    if grad:
        loss = crit(e, M)
        loss.backward()
        torch.cuda.synchronize()
        return loss.item(), e.grad.cpu().numpy().astype(np.float64), crit.weight.grad.item(), crit.bias.grad.item()
    with torch.no_grad():
        return crit(e, M).item(), None, None, None


def test_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "ge2e_loss.npz"))
    for i in range(int(g["num_cases"])):
        sd, N, M, un, w, b = g["case%d_meta" % i]
        E = synth.make_embeddings(int(sd), int(N), int(M), unit_norm=bool(un))
        loss, dE, dw, db = _run(E, int(M), float(w), float(b))
        ref_loss, ref_dE = float(g["case%d_f64_loss" % i]), g["case%d_f64_dE" % i]
        assert abs(loss - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss)), (i, loss, ref_loss)
        rel = np.linalg.norm(dE[stored_rows(g, "case%d_rows" % i)] - ref_dE) / np.linalg.norm(ref_dE)
        assert rel <= 2e-4, (i, rel)                       # fp32 kernel vs fp64 reference
        # every row, against the fp64 closed form (which tests/test_oracle_golden.py pins to the reference)
        full_dE = O.ge2e_loss_and_grads_closed_form(E, int(M), float(w), float(b))[1]
        assert np.linalg.norm(dE - full_dE) / np.linalg.norm(full_dE) <= 2e-4, i
        assert abs(dw - float(g["case%d_f64_dw" % i])) <= 1e-4 * abs(float(g["case%d_f64_dw" % i])) + 1e-7
        assert abs(db) <= 1e-6                             # dL/db == 0 (SURVEY.md D3)
        # forward-only path (no_grad) gives the same loss
        l2, _, _, _ = _run(E, int(M), float(w), float(b), grad=False)
        assert abs(l2 - loss) <= 1e-6 * max(1.0, abs(loss))


@pytest.mark.parametrize("n,m", [(1, 4), (2, 1), (3, 7), (130, 2), (255, 3), (256, 3), (261, 5), (512, 15), (1024, 15)])
def test_closed_form_sizes(n, m):
    """Sizes the reference cannot hold in memory are checked against the fp64 closed form (App. B)."""
    E = synth.make_embeddings(900 + n, n, m, unit_norm=(n % 2 == 0))
    loss, dE, dw, db = _run(E, m)
    l_ref, dE_ref, dw_ref, db_ref = O.ge2e_loss_and_grads_closed_form(E, m)
    assert abs(loss - l_ref) <= 2e-5 * max(1.0, abs(l_ref))
    den = np.linalg.norm(dE_ref)
    if den > 1e-12:
        assert np.linalg.norm(dE - dE_ref) / den <= 3e-4
    else:
        assert np.abs(dE).max() <= 1e-6
    assert abs(dw - dw_ref) <= 2e-4 * abs(dw_ref) + 1e-6


@pytest.mark.parametrize("n", [2048, 4096])
def test_large_speaker_counts_match_the_closed_form(n):
    """BASELINE config 5's upper end (the reference itself cannot hold N > ~512 in memory): fused kernel vs the fp64
    closed form evaluated in row chunks."""
    m = 15
    E = synth.make_embeddings(1300 + n, n, m, unit_norm=True)
    loss, dE, dw, db = _run(E, m)
    l_ref, dE_ref, dw_ref, db_ref = O.ge2e_closed_form_chunked(E, m)
    assert abs(loss - l_ref) <= 2e-5 * max(1.0, abs(l_ref)), (loss, l_ref)
    assert np.linalg.norm(dE - dE_ref) / np.linalg.norm(dE_ref) <= 3e-4
    assert abs(dw - dw_ref) <= 2e-4 * abs(dw_ref) + 1e-6
    assert abs(db) <= 1e-5


def test_grad_scaling_and_errors():
    from speaker_embedding_torch_b200 import GE2E_Loss
    E = synth.make_embeddings(3, 6, 4)
    crit = GE2E_Loss().cuda()
    e = torch.as_tensor(E).cuda().requires_grad_(True)
    (crit(e, 4) * 3.0).backward()
    g3 = e.grad.clone()
    e.grad = None
    crit(e, 4).backward()
    torch.testing.assert_close(g3, 3.0 * e.grad, rtol=1e-5, atol=1e-9)
    with pytest.raises(RuntimeError):
        crit(e, 5)                                         # 24 rows are not a multiple of 5
    with pytest.raises(RuntimeError, match="not supported"):
        crit(torch.randn(8, 128, device="cuda"), 2)


@pytest.mark.parametrize("n,m", [(1, 1), (1, 4), (2, 1), (3, 7), (5, 13), (64, 15), (65, 3), (100, 9), (128, 15), (129, 2),
                                 (192, 5), (255, 3)])
def test_row_tile_stage_matches_the_closed_form(n, m):
    """ge2e_rows_tile_kernel (8-row tiles, bulk-copied centroid tiles, K split over warp halves) against the fp64 closed
    form; every tile shape of the N < 256 path: rows not a multiple of 8, 1 .. 4 centroid tiles, a ragged last tile."""
    E = synth.make_embeddings(1700 + n, n, m, unit_norm=(n % 2 == 1))
    l_ref, dE_ref, dw_ref, db_ref = O.ge2e_loss_and_grads_closed_form(E, m)
    loss, dE, dw, db = _run(E, m)
    l_ng, _, _, _ = _run(E, m, grad=False)
    assert abs(l_ng - loss) <= 1e-6 * max(1.0, abs(loss))
    assert abs(loss - l_ref) <= 2e-5 * max(1.0, abs(l_ref))
    den = np.linalg.norm(dE_ref)
    if den > 1e-12:
        assert np.linalg.norm(dE - dE_ref) / den <= 3e-4
    else:
        assert np.abs(dE).max() <= 1e-6
    assert abs(dw - dw_ref) <= 2e-4 * abs(dw_ref) + 1e-6
    assert abs(db) <= 1e-5
