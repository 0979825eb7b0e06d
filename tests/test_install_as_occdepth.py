"""The documented drop-in order (INTEGRATION.md section 2): `occdepth_b200.install_as_occdepth()` BEFORE the
reference's imports, after which the body of the reference scripts must import -- `occdepth.models*` from this
package, everything else (`occdepth.data.*`, `occdepth.loss.*`) still from the reference tree.  The reference tree is
stood in for by a tree of the same layout (namespace packages, no __init__.py) whose modules define only the names the
import block touches, and whose own `occdepth.models` modules fail on import.  Runs in a subprocess so that the test
session's own sys.modules stay untouched."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WITH_REFERENCE = r"""
import sys
sys.path[:0] = [%(root)r, %(ref)r]
import occdepth_b200
occdepth_b200.install_as_occdepth()
# the import block of occdepth/scripts/generate_output.py:1-5 and eval.py (minus the third-party trainer)
from occdepth.models.OccDepth import OccDepth
import occdepth.loss.sscMetrics as sscMetrics
import occdepth.data.utils.helpers as helpers
import occdepth.data.semantic_kitti.collate as collate
from occdepth.models.unet3d_kitti import UNet3D
from occdepth.models.SFA import SFA
import occdepth
assert OccDepth.__module__ == "occdepth_b200.models.OccDepth", OccDepth.__module__
assert UNet3D.__module__ == "occdepth_b200.models.unet3d_kitti" and SFA.__module__ == "occdepth_b200.models.SFA"
assert "reference" in sscMetrics.__file__ or %(ref)r in sscMetrics.__file__, sscMetrics.__file__
assert hasattr(helpers, "vox2pix") and hasattr(collate, "collate_fn")
assert hasattr(occdepth, "__path__")
print("OK")
"""

WITHOUT_REFERENCE = r"""
import sys
sys.path.insert(0, %(root)r)
import occdepth_b200
occdepth_b200.install_as_occdepth()
from occdepth.models.OccDepth import OccDepth
from occdepth.models.flosp_depth.flosp_depth import FlospDepth
assert OccDepth.__module__ == "occdepth_b200.models.OccDepth"
try:
    import occdepth.data.utils.helpers
except ModuleNotFoundError as e:
    assert "is not a package" not in str(e), e
else:
    raise SystemExit("occdepth.data must not resolve without the reference tree")
print("OK")
"""


# the reference tree's layout around the modules that the import block above touches
REFERENCE_STANDIN = {
    "occdepth/models/OccDepth.py": "raise ImportError('the reference OccDepth was imported')\n",
    "occdepth/models/unet3d_kitti.py": "raise ImportError('the reference UNet3D was imported')\n",
    "occdepth/models/SFA.py": "raise ImportError('the reference SFA was imported')\n",
    "occdepth/loss/sscMetrics.py": "class SSCMetrics:\n    pass\n",
    "occdepth/data/utils/helpers.py": "def vox2pix(*args):\n    raise NotImplementedError\n",
    "occdepth/data/semantic_kitti/collate.py": "def collate_fn(batch):\n    return batch\n",
}


def _run(code):
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    return subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env, cwd="/tmp")


def test_install_then_reference_imports(tmp_path):
    ref = tmp_path / "reference"
    for rel, body in REFERENCE_STANDIN.items():
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text(body)
    r = _run(WITH_REFERENCE % {"root": ROOT, "ref": str(ref)})
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


def test_install_without_reference_tree():
    r = _run(WITHOUT_REFERENCE % {"root": ROOT})
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


def test_frame_pipeline_refuses_without_cuda():
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    from occdepth_b200.serving import FramePipeline
    with pytest.raises(RuntimeError, match="CUDA"):
        FramePipeline(None, (1, 2, 3, 8, 8), (2, 8, 1, 2), (2, 8, 1))
