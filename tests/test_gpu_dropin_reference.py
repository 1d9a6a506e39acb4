"""The reference's own drivers on top of the drop-in modules (SURVEY.md section 4, INTEGRATION.md section 1).
Runs tests/dropin_train_worker.py in a fresh interpreter (it stubs librosa / pysptk / matplotlib in sys.modules and
shadows `Modules` / `distributed` with the two shim files, which must not leak into the other tests)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "Train.py")),
                    reason="needs a reference checkout, staged to baseline/_ref by build() from SPK_REFERENCE")
@pytest.mark.parametrize("device_collater", ["0", "1"])
def test_reference_train_py_runs_unmodified_on_the_drop_in_modules(tmp_path, device_collater):
    """device_collater = 1 additionally shadows Datasets.Collater with the on-device collater (RaggedMel batches)."""
    env = dict(os.environ, SPK_DROPIN_DEVICE_COLLATER=device_collater)
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_train_worker.py"), REF, str(tmp_path)],
                          capture_output=True, text=True, timeout=900, cwd=str(tmp_path), env=env)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    assert "DROPIN_TRAIN_OK" in proc.stdout, proc.stdout[-2000:]
