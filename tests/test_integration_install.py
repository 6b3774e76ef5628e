"""CPU: integration.use_b200.install() against a stand-in reference tree (modules with the names and the attributes
eval.py imports, no reference code), so the binding is checked without an upstream YOLACT checkout:
tests/test_eval_drop_in.py runs the reference's own eval.py where one is available.  Runs in a subprocess so the
stand-in top-level packages (data, utils, layers, yolact) do not leak into the test session."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STUBS = {
    "data/__init__.py": "cfg = None\n",
    "yolact.py": "class Yolact(object):\n    pass\n",
    "layers/__init__.py": "",
    "layers/output_utils.py": "def postprocess(*args, **kwargs):\n    raise AssertionError('not rebound')\n",
    "layers/box_utils.py": "def mask_iou(*args):\n    pass\n\n\ndef jaccard(*args):\n    pass\n",
    "utils/__init__.py": "",
    "utils/augmentations.py": "class FastBaseTransform(object):\n    pass\n",
}

SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
import integration.use_b200 as ub
names = ub.install(%(ref)r)
import data, yolact, layers.output_utils as ou, layers.box_utils as bu, utils.augmentations as aug
import yolact_b200
from yolact_b200 import eval_utils
from tests.helpers import load_reference_cfgs
assert yolact.__file__.startswith(%(ref)r), yolact.__file__
assert yolact.Yolact is names["Yolact"] and issubclass(yolact.Yolact, yolact_b200.Yolact)
assert yolact.ReferenceYolact.__module__ == "yolact"                     # the reference graph stays reachable
assert ou.postprocess is names["postprocess"]
assert aug.FastBaseTransform is names["FastBaseTransform"]
assert issubclass(aug.FastBaseTransform, yolact_b200.FastBaseTransform)
assert bu.mask_iou is eval_utils.mask_iou and bu.jaccard is eval_utils.jaccard
# the reference's no-argument constructor reads the reference's global cfg (eval.py calls set_cfg before Yolact())
data.cfg = load_reference_cfgs()["yolact_plus_resnet50_config"]
net = yolact.Yolact()
assert net.cfg.backbone_layers == [3, 4, 6, 3] and net.cfg.use_maskiou and yolact_b200.cfg.use_maskiou
# keys the reference's callers flip on the global cfg between calls (prep_display sets rescore_bbox around
# postprocess) are re-read on every postprocess call
seen = []
yolact_b200.postprocess = lambda *args, **kwargs: seen.append(bool(yolact_b200.cfg.rescore_bbox))
for flag in (True, False):
    data.cfg.rescore_bbox = flag
    ou.postprocess([], 8, 6)
assert seen == [True, False], seen
print("INSTALL OK")
'''


def test_install_rebinds_the_names_eval_py_imports(tmp_path):
    for rel, src in STUBS.items():
        path = tmp_path / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(src)
    ref = str(tmp_path)
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT, "ref": ref}], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert "INSTALL OK" in r.stdout
