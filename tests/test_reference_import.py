"""Import hygiene (SURVEY.md 8f N4): the reference's unedited modules import in an image without matplotlib / pytorch3d /
trimesh / pyrender / pybullet / submitit, and INTEGRATION.md's snippets run as written -- each in a FRESH interpreter.
No GPU work: nothing here launches a kernel."""
import os
import re
import subprocess
import sys

import pytest

import ptk_b200

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = ptk_b200.find_reference()
needs_reference = pytest.mark.skipif(REF is None, reason="no pterotactyl checkout (tools/install_reference.py / PTK_REFERENCE)")


def run(code):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT] + ([REF] if REF else [])))
    p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


def test_placeholders_import_subclass_and_refuse_use():
    out = run("""
import ptk_b200
stubbed = ptk_b200.install_import_stubs()
import matplotlib.pyplot as plt
from submitit.helpers import Checkpointable
class Engine(Checkpointable):
    def __init__(self, a): self.a = a
assert Engine(3).a == 3
for use in (lambda: plt.figure(), lambda: Checkpointable()):
    try:
        use()
    except ImportError as e:
        assert "not installed" in str(e)
    else:
        raise SystemExit("a placeholder let itself be used")
import numpy, torch                                     # installed packages are never shadowed
assert not ptk_b200.import_stubs.is_stub(numpy) and ptk_b200.import_stubs.is_stub(plt)
print(",".join(stubbed))
""")
    assert "matplotlib" in out


@needs_reference
def test_every_reference_entry_module_imports_unedited():
    mods = ["utility.utils", "utility.pretty_render", "utility.data_loaders", "reconstruction.vision.model",
            "reconstruction.vision.train", "reconstruction.touch.model", "reconstruction.touch.train",
            "reconstruction.autoencoder.model", "reconstruction.autoencoder.train", "policies.environment",
            "policies.baselines.greedy", "policies.DDQN.model", "policies.DDQN.train"]
    out = run(f"""
import ptk_b200
for m in ptk_b200.import_reference(*{mods!r}):
    print(m.__name__, m.__file__)
from pterotactyl.utility import utils
assert utils.cuda_cd.__module__ == "pytorch3d.loss.chamfer" and "pytorch3d_shim" in __import__("pytorch3d").__file__
assert utils.batch_sample.__module__ == "pterotactyl.utility.utils"
""")
    assert out.count("pterotactyl.") == len(mods) and "ptk_b200" not in out.replace("pytorch3d_shim", "")


@needs_reference
def test_integration_md_snippets_run_verbatim():
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    sec1 = text[text.index("## 1. Seam S1"):text.index("## 2. Seam S2")]
    sec2 = text[text.index("## 2. Seam S2"):text.index("## 3. Seam S3")]
    for sec, check in ((sec1, "assert utils.cuda_cd.__module__ == 'pytorch3d.loss.chamfer'"),
                       (sec2, "from pterotactyl.utility import utils\n"
                              "assert utils.chamfer_distance is ptk_b200.utils.chamfer_distance\n"
                              "assert vision_model.GCN is ptk_b200.GCN and ddqn_model.Graph_Model is ptk_b200.model.Graph_Model\n"
                              "ptk_b200.uninstall()\n"
                              "assert utils.chamfer_distance.__module__ == 'pterotactyl.utility.utils'")):
        code = re.findall(r"```python\n(.*?)```", sec, flags=re.S)[0]
        run(code + "\n" + check + "\n")
