"""CPU, needs the reference compiled into oracle/_ref/ by build() (oracle/build_ref.py; skipped where build() found no
reference tree): the reference's eval.py, imported UNCHANGED after integration.use_b200.install(), binds Yolact /
postprocess / FastBaseTransform / mask_iou / jaccard to this package.  Runs in a subprocess so the reference's top-level
packages (data, utils, layers) do not leak into the test session."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "yolact")

SCRIPT = r'''
import sys, types
sys.path.insert(0, %(root)r)
import torch
# the same import shims oracle/gen_golden.py uses on a GPU-less box with no pycocotools
for m in ["pycocotools", "pycocotools.mask", "pycocotools.coco", "pycocotools.cocoeval", "matplotlib", "matplotlib.pyplot"]:
    sys.modules.setdefault(m, types.ModuleType(m))
sys.modules["pycocotools.coco"].COCO = object
torch.cuda.current_device = lambda: 0
import integration.use_b200 as ub
names = ub.install(%(ref)r)
import eval as E                                   # the reference's eval.py, unmodified
import yolact_b200
from yolact_b200 import eval_utils
assert E.__file__.startswith(%(ref)r), E.__file__
assert E.Yolact is names["Yolact"] and issubclass(E.Yolact, yolact_b200.Yolact)
assert E.postprocess is names["postprocess"]
assert issubclass(E.FastBaseTransform, yolact_b200.FastBaseTransform)
assert E.mask_iou is eval_utils.mask_iou and E.jaccard is eval_utils.jaccard
# eval.py's own flow up to the network construction (eval.py:1085-1097)
E.parse_args(["--config=yolact_resnet50_config", "--trained_model=none"])
E.set_cfg("yolact_resnet50_config")
net = E.Yolact()
assert net.cfg.backbone_layers == [3, 4, 6, 3] and net.cfg.max_size == 550
net.detect.use_fast_nms = E.args.fast_nms          # eval.py:871-872
net.detect.use_cross_class_nms = E.args.cross_class_nms
# prep_display of a YOLACT++ config (eval.py:147-157) flips cfg.rescore_bbox on the REFERENCE's global cfg around
# postprocess and then argsorts t[1]: the bound postprocess must see the live value (a stale snapshot would return the
# [scores, scores*maskiou] 2-list and `t[1].argsort` would raise).  The CUDA call is stubbed (no GPU here); what is
# tested is the binding's cfg plumbing.
E.parse_args(["--config=yolact_plus_resnet50_config", "--trained_model=none", "--display_masks=False",
              "--display_text=False", "--display_bboxes=False", "--top_k=3"])
E.set_cfg("yolact_plus_resnet50_config")
plus = E.Yolact()
assert plus.cfg.use_maskiou and plus.cfg.rescore_mask and not plus.cfg.rescore_bbox
seen = []
def stub(dets, w, h, **kw):
    seen.append(bool(yolact_b200.cfg.rescore_bbox))
    s = torch.tensor([0.2, 0.9, 0.5, 0.7])
    scores = s * 0.5 if yolact_b200.cfg.rescore_bbox else [s, s * 0.5]      # output_utils.py:84-88
    return torch.arange(4), scores, torch.zeros(4, 4, dtype=torch.long), torch.zeros(4, h, w)
yolact_b200.postprocess = stub
img = torch.full((6, 8, 3), 128.0)
out = E.prep_display([{"detection": {}, "net": plus}], img, None, None, undo_transform=False)
assert seen == [True] and out.shape == (6, 8, 3)
assert E.cfg.rescore_bbox is False                                           # prep_display restored it (eval.py:151)
print("DROP-IN OK", len(net.state_dict()))
'''


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "eval.pyc")),
                    reason="build() found no reference tree to compile into oracle/_ref")
def test_reference_eval_py_binds_to_the_b200_path():
    # oracle/_ref holds bytecode only, and TorchScript needs source text: PYTORCH_JIT=0 runs the reference's
    # @torch.jit.script helpers as plain Python (what is tested here is the binding, not TorchScript)
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT, "ref": REF}], capture_output=True, text=True,
                       timeout=300, cwd=ROOT, env=dict(os.environ, PYTORCH_JIT="0"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert "DROP-IN OK" in r.stdout
