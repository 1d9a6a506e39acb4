"""CPU-side checks: the C-ABI library loads and exports what include/spkemb.h declares, the drop-in
modules keep the reference's layout, and compute calls fail loudly without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    from speaker_embedding_torch_b200 import _native
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    return _native


def test_library_exports_every_declared_symbol(native):
    header = open(os.path.join(ROOT, "include", "spkemb.h")).read()
    declared = set(re.findall(r"\b(spk_[a-z0-9_]+)\s*\(", header))
    assert declared == set(native.EXPORTS)
    L = native.lib()
    for name in declared:
        assert hasattr(L, name), name
    assert L.spk_abi_version() == native.ABI_VERSION == 2


def test_workspace_query_is_host_only(native):
    cfg = native.EncoderConfig(80, 256, 4, 1024, 3, 1024, 0.1, 0.1)
    L = native.lib()
    small = L.spk_encoder_workspace_bytes(ctypes.byref(cfg), 10, 64, 5, 1, 0)
    train = L.spk_encoder_workspace_bytes(ctypes.byref(cfg), 10, 64, 5, 2, 1)
    assert 0 < small < train
    # unsupported shapes are rejected with a message, not a crash
    bad = native.EncoderConfig(80, 128, 4, 512, 3, 1024, 0.1, 0.1)
    assert L.spk_encoder_workspace_bytes(ctypes.byref(bad), 10, 64, 5, 1, 0) == 0
    assert b"Embedding_Size 256" in L.spk_last_error()
    assert L.spk_encoder_workspace_bytes(ctypes.byref(cfg), 10, 2000, 1, 1, 0) == 0
    assert L.spk_encoder_workspace_bytes(ctypes.byref(cfg), 10, 64, 3, 1, 0) == 0   # 10 % 3 != 0
    assert L.spk_ge2e_workspace_bytes(64, 15) > 64 * 256 * 8


def test_option_switches_are_host_only_documented_and_retired_ones_unknown(native):
    """spk_set_option touches no device: every switch INTEGRATION.md lists is accepted here (and put back to its
    default), an unknown name is rejected with a message, and so is the switch of the retired first GE2E row stage."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    defaults = {"prune_last_layer": 1, "fused_training_attention": 1, "fused_inference_attention": 1,
                "inference_attention_two_ctas": 1, "training_attention_two_ctas": 1, "fused_layernorm": 2,
                "gemm_cta_pairs": 1, "gemm_dependent_launch": 2, "ge2e_dependent_launch": 1, "grad_scale_log2": 12}
    flags = native.plan_flags()
    for name, default in defaults.items():
        assert "`%s`" % name in text, name
        native.set_option(name, 0 if name != "grad_scale_log2" else 10)
        native.set_option(name, default)
    assert native.plan_flags() == flags
    with pytest.raises(RuntimeError, match="unknown option"):
        native.set_option("no_such_option", 1)
    with pytest.raises(RuntimeError, match="unknown option"):
        native.set_option("ge2e_row_tile_v2", 0)


def _model():
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    return GE2E(default_hyper_parameters())


def test_state_dict_layout_matches_reference():
    m = _model()
    sd = m.state_dict()
    want = synth.state_shapes()
    assert [k for k in sd] == [n for n, _ in want]
    for n, shape in want:
        assert tuple(sd[n].shape) == shape, n
    assert [n for n, _ in m.named_parameters()] == [n for n, _ in want if not n.endswith(".pe")]
    np.testing.assert_array_equal(sd["positional_encoding.pe"].numpy(), synth.positional_table())
    # reference-format checkpoints load strictly, in both directions
    state = {k: torch.as_tensor(v) for k, v in synth.make_state(3).items()}
    m.load_state_dict(state, strict=True)
    for k, v in m.state_dict().items():
        assert torch.equal(v, state[k])


def test_reference_initialisation_rules():
    torch.manual_seed(0)
    m = _model()
    assert float(m.prenet.bias.abs().max()) == 0.0 and float(m.projection.bias.abs().max()) == 0.0
    assert float(m.positional_encoding.alpha) == 1.0
    bound = (6.0 / 80) ** 0.5            # kaiming_uniform(relu), fan_in = 80 (Modules.py:67-68)
    assert float(m.prenet.weight.abs().max()) <= bound + 1e-6
    xb = (6.0 / 512) ** 0.5              # xavier_uniform, gain 1 (Modules.py:69-70)
    assert float(m.projection.weight.abs().max()) <= xb + 1e-6
    from speaker_embedding_torch_b200 import GE2E_Loss
    crit = GE2E_Loss()
    assert crit.weight.dim() == 0 and float(crit.weight) == 10.0 and float(crit.bias) == -5.0
    assert sorted(crit.state_dict()) == ["bias", "weight"]


def test_no_cpu_fallback():
    from speaker_embedding_torch_b200 import GE2E_Loss
    m = _model().eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        with torch.no_grad():
            m(torch.zeros(2, 80, 16))
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(2, 80, 16))
    with pytest.raises(RuntimeError, match="CUDA"):
        GE2E_Loss()(torch.zeros(4, 256), 2)


def test_schedulers_match_oracle_formula():
    from speaker_embedding_torch_b200.Noam_Scheduler import Modified_Noam_Scheduler, Noam_Scheduler
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=2e-3)
    sch = Modified_Noam_Scheduler(opt, base=4000)
    for t in range(6):
        np.testing.assert_allclose(opt.param_groups[0]["lr"], O.modified_noam_lr(2e-3, t, 4000), rtol=1e-12)
        opt.step()
        sch.step()
    opt2 = torch.optim.SGD([p], lr=1.0)
    sch2 = Noam_Scheduler(opt2, warmup_steps=10)
    lrs = []
    for t in range(30):
        lrs.append(opt2.param_groups[0]["lr"])
        opt2.step()
        sch2.step()
    assert np.argmax(lrs) == 10 and abs(lrs[10] - 1.0) < 1e-12


def test_arg_parser_contract():
    from speaker_embedding_torch_b200.Arg_Parser import Recursive_Parse
    hp = Recursive_Parse({"A": {"B": {"C": 3}}, "D": [1, 2], "E": "x"})
    assert hp.A.B.C == 3 and hp.D == [1, 2] and hp.E == "x"


def test_overlapped_slices_match_the_collater():
    """Device-side slicing == the reference collater's np.stack of strided windows (Inference.py:103-110)."""
    import numpy as np
    import torch
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices
    rs = np.random.RandomState(0)
    frame, overlap, samples = 64, 32, 5
    required = samples * (frame - overlap) + overlap
    feats = [rs.randn(80, required).astype(np.float32) for _ in range(3)]
    ref = np.vstack([np.stack([f[:, i:i + frame] for i in range(0, required - overlap, frame - overlap)]) for f in feats])
    got = Overlapped_Slices(torch.from_numpy(np.stack(feats)), frame, overlap)
    assert got.shape == (3 * samples, 80, frame)
    assert np.array_equal(got.numpy(), ref)
    import pytest
    with pytest.raises(RuntimeError):
        Overlapped_Slices(torch.zeros(2, 80, 32), 64, 32)


def test_dropin_harness_is_what_the_reference_expects(tmp_path):
    """tests/dropin_train_worker.py (the GPU drop-in test of the reference's unmodified Train.py) run against the
    REFERENCE's own modules on CPU: the synthetic patterns, yaml and call sequence are valid reference usage."""
    import subprocess
    import sys
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref, "Train.py")):
        pytest.skip("needs a reference checkout, staged to baseline/_ref by build() from SPK_REFERENCE")
    env = dict(os.environ, SPK_DROPIN_REFERENCE_MODULES="1", CUDA_VISIBLE_DEVICES="")
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_train_worker.py"), ref, str(tmp_path)],
                          capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=env)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
    assert "DROPIN_TRAIN_OK" in proc.stdout


def test_debug_layout_lists_the_stage_buffers_and_the_readers_decode_them(native):
    """The workspace map names every stage buffer the stage-parity tests read (fused attention statistics and keep
    bits, ReLU bits, the pruned last layer's compact rows, the head statistics, the gradient scale), and read_bits /
    read_f32 decode the chunk-major bit layout ([cols/32][rows] words, bit i of word (c, r) = element (r, 32c + i))."""
    cfg = native.EncoderConfig(80, 256, 4, 1024, 3, 1024, 0.1, 0.1)
    flags = native.plan_flags()
    lay = native.debug_layout(cfg, 6, 129, 1, 2 | flags, True)
    for name in ("h0bits", "L0.fbits", "L1.astat", "L1.abits", "L1.pd", "last.kv", "last.q0", "last.att0",
                 "last.z1", "last.st1", "last.h1", "last.f", "last.z2", "last.st2", "last.hout", "last.p0",
                 "last.pd0", "hst", "gscale"):
        assert name in lay, name
    infer = native.debug_layout(cfg, 6, 129, 1, 1 | flags, False)
    assert "h0bits" not in infer and "gscale" not in infer and "L0.astat" not in infer
    rows, cols = 5, 64
    mask = torch.rand(rows, cols, generator=torch.Generator().manual_seed(3)) > 0.5
    words = torch.zeros(cols // 32, rows, dtype=torch.int64)
    for c in range(cols // 32):
        for i in range(32):
            words[c] |= mask[:, 32 * c + i].long() << i
    ws = torch.zeros(4096, dtype=torch.uint8)
    base = (ws.data_ptr() + 255) // 256 * 256 - ws.data_ptr()
    payload = words.numpy().astype(np.uint32)
    ws[base + 256:base + 256 + payload.nbytes] = torch.from_numpy(payload.view(np.uint8).reshape(-1).copy())
    vals = torch.arange(7, dtype=torch.float32)
    ws[base + 1024:base + 1024 + 28] = vals.view(torch.uint8)
    fake = {"bits": (256, 0), "vals": (1024, 0)}
    assert torch.equal(native.read_bits(ws, fake, "bits", rows, cols), mask)
    assert torch.equal(native.read_f32(ws, fake, "vals", 7), vals)
