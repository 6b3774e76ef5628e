"""Generates tests/golden/* by running the REAL reference (an upstream YOLACT checkout) on the CPU.

    python oracle/gen_golden.py [keys|units|eval|cfgs|full|nets ...]   # reference located by oracle/build_ref.py
The committed .npz files are what pins oracle/yolact_oracle.py and the CUDA path to the reference.

Shims (never edits to the reference; SURVEY.md section 8c): stub pycocotools / matplotlib in
sys.modules, torch.cuda.current_device -> 0, and -- for YOLACT++ configs -- a `dcn_v2` module whose
DCN has the reference's parameter names and calls torchvision.ops.deform_conv2d (the vendored CUDA
extension cannot be built: THC headers).  The deterministic weights come from oracle/weights.py.
"""
import copy
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.build_ref import reference_root  # noqa: E402
REF = reference_root() or ""
OUT = os.path.join(ROOT, "tests", "golden")


def install_shims():
    for m in ["pycocotools", "pycocotools.mask", "pycocotools.coco", "pycocotools.cocoeval", "matplotlib",
              "matplotlib.pyplot"]:
        sys.modules.setdefault(m, types.ModuleType(m))
    sys.modules["pycocotools.coco"].COCO = object
    torch.cuda.current_device = lambda: 0
    # use_jit=False (yolact.py:25): FastMaskIoUNet.forward is not a script_method and cannot run as a
    # ScriptModule on torch 2.x; the reference takes this same path whenever >1 GPU is visible
    torch.cuda.device_count = lambda: 2
    import torchvision
    from torch import nn

    class DCN(nn.Module):
        """Parameter-name compatible stand-in for external/DCNv2/dcn_v2.py:97-128."""

        def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation=1, deformable_groups=1):
            super().__init__()
            self.stride, self.padding, self.dilation = stride, padding, dilation
            self.weight = nn.Parameter(torch.empty(out_channels, in_channels, kernel_size, kernel_size))
            self.bias = nn.Parameter(torch.zeros(out_channels))
            self.conv_offset_mask = nn.Conv2d(in_channels, 27, kernel_size, stride=stride, padding=padding, bias=True)
            nn.init.normal_(self.weight, std=0.01)

        def forward(self, x):
            out = self.conv_offset_mask(x)
            o1, o2, mask = torch.chunk(out, 3, dim=1)
            offset = torch.cat((o1, o2), dim=1)
            mask = torch.sigmoid(mask)
            return torchvision.ops.deform_conv2d(x, offset, self.weight, self.bias, stride=self.stride,
                                                 padding=self.padding, dilation=self.dilation, mask=mask)

    mod = types.ModuleType("dcn_v2")
    mod.DCN = DCN
    sys.modules["dcn_v2"] = mod
    if REF not in sys.path:
        sys.path.insert(0, REF)


def install_cython_nms():
    """utils/cython_nms.pyx does not compile with Cython 3 / numpy 2 (`np.int_t`, `np.int` are gone).  Build it
    from a temporary copy with exactly those two aliases renamed (np.int_t -> np.intp_t, np.int -> np.intp; the
    algorithm is untouched) and register it as utils.cython_nms so Detect.traditional_nms imports it."""
    import importlib.util
    import shutil
    import subprocess
    import sysconfig
    import tempfile
    if "utils.cython_nms" in sys.modules:
        return
    src = open(os.path.join(REF, "utils", "cython_nms.pyx")).read()
    src = src.replace("np.int_t", "np.intp_t").replace("dtype=np.int)", "dtype=np.intp)")
    d = tempfile.mkdtemp(prefix="yb_cnms_")
    try:
        pyx = os.path.join(d, "cython_nms.pyx")
        open(pyx, "w").write(src)
        subprocess.run([sys.executable, "-m", "cython", "-3", pyx], check=True, capture_output=True)
        so = os.path.join(d, "cython_nms" + sysconfig.get_config_var("EXT_SUFFIX"))
        subprocess.run(["gcc", "-O2", "-shared", "-fPIC", "-I", sysconfig.get_paths()["include"], "-I", np.get_include(),
                        os.path.join(d, "cython_nms.c"), "-o", so], check=True, capture_output=True)
        spec = importlib.util.spec_from_file_location("utils.cython_nms", so)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    import utils as ref_utils
    sys.modules["utils.cython_nms"] = mod
    ref_utils.cython_nms = mod
    import pyximport
    pyximport.install = lambda *a, **k: None     # traditional_nms calls it before the import above resolves


def npz_save(name, **arrs):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **arrs)
    print("wrote %s (%.2f MB)" % (path, os.path.getsize(path) / 1e6))


def to_np(t):
    return t.detach().cpu().numpy()


def gen_network_case(tag, config_name, B, H, W, post_hw, seed=0, row_stride=1):
    from data.config import cfg, set_cfg
    import yolact as ref_yolact
    from layers.output_utils import postprocess
    from oracle.weights import deterministic_state_dict, deterministic_input

    set_cfg(config_name)
    cfg.mask_proto_debug = False
    net = ref_yolact.Yolact()
    net.load_state_dict(deterministic_state_dict(net.state_dict(), seed))
    net.detect.use_fast_nms = True
    net.detect.use_cross_class_nms = False
    x = deterministic_input(B, H, W, 1234 + seed)
    out = {"x": to_np(x), "config": np.array(config_name), "seed": np.array(seed), "post_hw": np.array(post_hw)}
    with torch.no_grad():
        # train() makes forward return the raw head tensors (yolact.py:639-647); freeze_bn() keeps
        # BatchNorm in eval mode (running statistics), i.e. exactly the inference arithmetic
        net.train()
        net.freeze_bn()
        raw = net(x)
        out["row_stride"] = np.array(row_stride)
        for k in ("loc", "conf", "mask"):
            out["raw_" + k] = to_np(raw[k]).astype(np.float32)[:, ::row_stride]
        for k in ("priors", "proto"):
            out["raw_" + k] = to_np(raw[k]).astype(np.float32)
        # intermediate features (backbone stage outputs + FPN levels) for stage-level parity
        bb = net.backbone(x)
        for i, f in enumerate(bb):
            out["feat_c%d_absmean" % i] = np.array(float(f.abs().mean()))
            out["feat_c%d_sample" % i] = to_np(f[:, ::7, ::3, ::3]).astype(np.float32)
        net.eval()
        preds = net(x)
    counts = []
    for b in range(B):
        det = preds[b]["detection"]
        n = 0 if det is None else int(det["score"].shape[0])
        counts.append(n)
        if det is None:
            continue
        for k in ("box", "mask", "class", "score"):
            out["det%d_%s" % (b, k)] = to_np(det[k])
        ph, pw = post_hw
        p2 = copy.deepcopy([{"detection": {k: v.clone() for k, v in det.items()}, "net": net}])
        with torch.no_grad():
            classes, scores, boxes, masks = postprocess(p2, pw, ph, batch_idx=0, crop_masks=True, score_threshold=0)
        out["post%d_classes" % b] = to_np(classes)
        if isinstance(scores, list):
            out["post%d_scores" % b] = to_np(scores[0])
            out["post%d_scores_maskiou" % b] = to_np(scores[1])
        else:
            out["post%d_scores" % b] = to_np(scores)
        out["post%d_boxes" % b] = to_np(boxes)
        out["post%d_masks_packed" % b] = np.packbits(to_np(masks).astype(np.uint8), axis=-1)
    out["det_counts"] = np.array(counts)
    sm = torch.softmax(raw["conf"], -1)[..., 1:].max(-1)[0]
    qs = [float(torch.quantile(sm.flatten(), q)) for q in (0.5, 0.9, 0.99, 1.0)]
    top = to_np(preds[0]["detection"]["score"])[:5] if preds[0]["detection"] is not None else []
    print(tag, config_name, "P =", raw["loc"].shape[1], "detections per image:", counts,
          "max|conf logit| %.2f" % float(raw["conf"].abs().max()), "proto max %.2f" % float(raw["proto"].max()),
          "fg-score quantiles 50/90/99/100:", ["%.3f" % q for q in qs], "n>0.05:", int((sm > 0.05).sum()),
          "top scores", top, "coef absmax %.2f" % float(raw["mask"].abs().max()))
    npz_save(tag, **out)


def gen_fullsize_case(tag, config_name, size, post_hw, seed=0, seed_x=99, head_stride=97, proto_stride=5):
    """One FULL-SIZE image of a BASELINE.json config through the real reference: eval-mode `net(x)` (Detect with
    fast_nms) + `postprocess` at `post_hw` (eval.py:949,266).  Kept small: the input is rebuilt from its seed, the raw
    head tensors are row-subsampled, the prototypes spatially subsampled; the 100 detections and their bit-packed
    masks are complete."""
    from data.config import cfg, set_cfg
    import yolact as ref_yolact
    from layers.output_utils import postprocess
    from oracle.weights import deterministic_state_dict, deterministic_input

    set_cfg(config_name)
    cfg.mask_proto_debug = False
    net = ref_yolact.Yolact()
    net.load_state_dict(deterministic_state_dict(net.state_dict(), seed))
    net.detect.use_fast_nms = True
    net.detect.use_cross_class_nms = False
    x = deterministic_input(1, size, size, seed_x)
    out = {"config": np.array(config_name), "seed": np.array(seed), "seed_x": np.array(seed_x), "size": np.array(size),
           "post_hw": np.array(post_hw), "head_stride": np.array(head_stride), "proto_stride": np.array(proto_stride)}
    with torch.no_grad():
        net.train()
        net.freeze_bn()
        raw = net(x)
        for k in ("loc", "conf", "mask"):
            out["raw_" + k] = to_np(raw[k]).astype(np.float32)[:, ::head_stride]
            out["raw_%s_absmax" % k] = np.array(float(raw[k].abs().max()))
        out["raw_proto"] = to_np(raw["proto"]).astype(np.float32)[:, ::proto_stride, ::proto_stride]
        out["raw_proto_absmax"] = np.array(float(raw["proto"].abs().max()))
        out["raw_priors"] = to_np(raw["priors"]).astype(np.float32)
        net.eval()
        preds = net(x)
    det = preds[0]["detection"]
    assert det is not None
    for k in ("box", "mask", "class", "score"):
        out["det_" + k] = to_np(det[k])
    ph, pw = post_hw
    p2 = copy.deepcopy([{"detection": {k: v.clone() for k, v in det.items()}, "net": net}])
    with torch.no_grad():
        classes, scores, boxes, masks = postprocess(p2, pw, ph, batch_idx=0, crop_masks=True, score_threshold=0)
    out["post_classes"] = to_np(classes)
    if isinstance(scores, list):
        out["post_scores"] = to_np(scores[0])
        out["post_scores_maskiou"] = to_np(scores[1])
    else:
        out["post_scores"] = to_np(scores)
    out["post_boxes"] = to_np(boxes)
    out["post_masks_packed"] = np.packbits(to_np(masks).astype(np.uint8), axis=-1)
    s = out["det_score"]
    print(tag, config_name, "P =", raw["loc"].shape[1], "detections:", len(s), "scores %.4f .. %.4f" % (s[0], s[-1]),
          "min gap between consecutive scores %.2e" % float(np.min(-np.diff(s))) if len(s) > 1 else "")
    npz_save(tag, **out)


FULL_CASES = [  # BASELINE.json configs 2-5 (+ the 640x480 postprocess target of eval.py:266)
    ("full_base_550", "yolact_base_config", 550, (550, 550)),
    ("full_base_550_to_480x640", "yolact_base_config", 550, (480, 640)),
    ("full_plus_resnet50_550", "yolact_plus_resnet50_config", 550, (550, 550)),
    ("full_im700_700", "yolact_im700_config", 700, (700, 700)),
    ("full_plus_base_550", "yolact_plus_base_config", 550, (550, 550)),
]


def gen_detect_unit(seed=3):
    """Synthetic pred_outs straight into the reference Detect (fast_nms and cc_fast_nms)."""
    from data.config import cfg, set_cfg
    from layers import Detect
    set_cfg("yolact_base_config")
    r = np.random.RandomState(seed)
    B, P, C, K = 2, 3000, 81, 32
    # priors: random centre-size boxes; loc: N(0,1); scores: peaked, unique
    priors = np.concatenate([r.uniform(0.05, 0.95, (P, 2)), r.uniform(0.03, 0.4, (P, 2))], 1).astype(np.float32)
    loc = r.standard_normal((B, P, 4)).astype(np.float32)
    logits = (r.standard_normal((B, P, C)) * 2.0).astype(np.float32)
    logits[:, :, 0] += 3.0
    hot = r.rand(B, P) < 0.25
    cls = r.randint(1, C, size=(B, P))
    for b in range(B):
        idx = np.nonzero(hot[b])[0]
        logits[b, idx, cls[b, idx]] += r.uniform(2.0, 9.0, size=idx.size).astype(np.float32)
    conf = torch.softmax(torch.from_numpy(logits), -1)
    mask = np.tanh(r.standard_normal((B, P, K))).astype(np.float32)
    out = {"loc": loc, "conf": to_np(conf), "mask": mask, "priors": priors}
    for cc in (False, True):
        d = Detect(C, bkg_label=0, top_k=200, conf_thresh=0.05, nms_thresh=0.5)
        d.use_fast_nms = True
        d.use_cross_class_nms = cc
        res = d({"loc": torch.from_numpy(loc), "conf": conf, "mask": torch.from_numpy(mask),
                 "priors": torch.from_numpy(priors)}, None)
        tag = "cc" if cc else "fast"
        for b in range(B):
            det = res[b]["detection"]
            for k in ("box", "mask", "class", "score"):
                out["%s%d_%s" % (tag, b, k)] = to_np(det[k])
            print("detect_unit", tag, b, "n =", det["score"].shape[0])
    # --fast_nms=False: Detect.traditional_nms (detection.py:182-228) with the reference's cython_nms
    install_cython_nms()
    for ms in (550, 138):
        cfg.max_size = ms
        d = Detect(C, bkg_label=0, top_k=200, conf_thresh=0.05, nms_thresh=0.5)
        d.use_fast_nms = False
        d.use_cross_class_nms = False
        res = d({"loc": torch.from_numpy(loc), "conf": conf, "mask": torch.from_numpy(mask),
                 "priors": torch.from_numpy(priors)}, None)
        for b in range(B):
            det = res[b]["detection"]
            for k in ("box", "mask", "class", "score"):
                out["trad%d_%d_%s" % (ms, b, k)] = to_np(det[k])
            print("detect_unit traditional max_size", ms, b, "n =", det["score"].shape[0])
    cfg.max_size = 550
    npz_save("detect_unit", **out)


def gen_postprocess_unit(seed=5):
    from data.config import cfg, set_cfg
    from layers.output_utils import postprocess
    set_cfg("yolact_base_config")
    cfg.mask_proto_debug = False
    r = np.random.RandomState(seed)
    n, ph, pw, K = 23, 138, 138, 32
    proto = np.maximum(r.standard_normal((ph, pw, K)), 0).astype(np.float32)
    # smooth the prototypes so masks have structure
    proto = (proto + np.roll(proto, 1, 0) + np.roll(proto, 1, 1) + np.roll(proto, (2, 3), (0, 1))) / 4
    coef = np.tanh(r.standard_normal((n, K))).astype(np.float32)
    c = r.uniform(0.15, 0.85, (n, 2))
    wh = r.uniform(0.05, 0.6, (n, 2))
    box = np.concatenate([c - wh / 2, c + wh / 2], 1).astype(np.float32)
    box[3, [0, 2]] = box[3, [2, 0]]      # x1 > x2: sanitize must swap
    box[5] = [-0.1, 0.2, 0.5, 1.2]       # partially outside the image
    score = np.sort(r.uniform(0.1, 0.99, n).astype(np.float32))[::-1].copy()
    cls = r.randint(0, 80, n).astype(np.int64)
    out = {"proto": proto, "coef": coef, "box": box, "score": score, "cls": cls}
    for (h, w) in ((550, 550), (203, 277), (64, 96)):
        for crop in (True, False):
            det = {"box": torch.from_numpy(box.copy()), "mask": torch.from_numpy(coef), "class": torch.from_numpy(cls),
                   "score": torch.from_numpy(score), "proto": torch.from_numpy(proto)}
            with torch.no_grad():
                classes, scores, boxes, masks = postprocess([{"detection": det, "net": None}], w, h, crop_masks=crop)
            tag = "%dx%d_%s" % (h, w, "crop" if crop else "nocrop")
            out["boxes_" + tag] = to_np(boxes)
            out["masks_" + tag] = np.packbits(to_np(masks).astype(np.uint8), axis=-1)
            print("postprocess_unit", tag, "mask fill %.4f" % float(masks.mean()))
    npz_save("postprocess_unit", **out)


def gen_dcn_unit(seed=7):
    """DCNv2 op: torchvision.ops.deform_conv2d (the practical stand-in for the reference extension),
    cross-checked against the numpy restatement of the reference's CUDA kernel, plus the reference's own
    zero-offset identity (external/DCNv2/test.py:32-67)."""
    import torchvision
    from oracle.yolact_oracle import dcn_v2_forward
    r = np.random.RandomState(seed)
    out = {}
    for tag, (B, C, H, W, Co, stride) in {"s1": (2, 16, 13, 11, 24, 1), "s2": (1, 32, 14, 17, 16, 2)}.items():
        x = r.standard_normal((B, C, H, W)).astype(np.float32)
        w = (r.standard_normal((Co, C, 3, 3)) * 0.1).astype(np.float32)
        bias = r.standard_normal(Co).astype(np.float32)
        Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
        offset = (r.standard_normal((B, 18, Ho, Wo)) * 2.0).astype(np.float32)
        mask = (1 / (1 + np.exp(-r.standard_normal((B, 9, Ho, Wo))))).astype(np.float32)
        y = torchvision.ops.deform_conv2d(torch.from_numpy(x), torch.from_numpy(offset), torch.from_numpy(w),
                                          torch.from_numpy(bias), stride=stride, padding=1, dilation=1,
                                          mask=torch.from_numpy(mask)).numpy()
        y2 = dcn_v2_forward(x, offset, mask, w, bias, stride, 1, 1)
        print("dcn_unit", tag, "torchvision vs restatement max abs diff", float(np.abs(y - y2).max()))
        assert np.abs(y - y2).max() < 2e-5
        out.update({tag + "_x": x, tag + "_w": w, tag + "_bias": bias, tag + "_offset": offset, tag + "_mask": mask,
                    tag + "_y": y, tag + "_stride": np.array(stride)})
    # zero-offset identity: weight = identity at the centre tap, mask = 0.5 -> 2*out == input
    C = 8
    x = r.standard_normal((2, C, 9, 9)).astype(np.float32)
    w = np.zeros((C, C, 3, 3), np.float32)
    for i in range(C):
        w[i, i, 1, 1] = 1.0
    y = dcn_v2_forward(x, np.zeros((2, 18, 9, 9), np.float32), np.full((2, 9, 9, 9), 0.5, np.float32), w,
                       np.zeros(C, np.float32), 1, 1, 1)
    assert np.abs(2 * y - x).max() < 1e-10, "zero-offset identity failed"
    print("dcn_unit zero-offset identity ok")
    npz_save("dcn_unit", **out)


def gen_eval_unit(seed=11):
    """Rows either side of the path: FastBaseTransform, mask_iou / jaccard, prep_display -- all from the real
    reference.  Shims: Tensor.cuda() -> identity (FastBaseTransform.__init__ moves its constants to the GPU);
    for prep_display a Tensor subclass whose `.device.index` is 0 plus Tensor.to(int) -> identity, because the
    reference only takes its GPU colour path when the image reports a CUDA device (eval.py:171-183,193)."""
    from data.config import cfg, set_cfg
    from utils.augmentations import FastBaseTransform
    from layers.box_utils import mask_iou, jaccard
    r = np.random.RandomState(seed)
    out = {}
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        cases = {"up": ("yolact_base_config", (2, 37, 53), 96, False),
                 "down": ("yolact_base_config", (1, 300, 211), 96, False),
                 "same": ("yolact_base_config", (1, 64, 64), 64, False),
                 "ar": ("yolact_base_config", (1, 120, 200), 80, True),
                 "dark": ("yolact_darknet53_config", (1, 50, 70), 96, False)}
        for tag, (cname, (B, H, W), S, ar) in cases.items():
            set_cfg(cname)
            cfg.max_size = S
            cfg.preserve_aspect_ratio = ar
            img = r.randint(0, 256, size=(B, H, W, 3)).astype(np.uint8)
            y = FastBaseTransform()(torch.from_numpy(img).float())
            out["xf_%s_img" % tag] = img
            out["xf_%s_out" % tag] = to_np(y)
            out["xf_%s_cfg" % tag] = np.array([S, int(ar), int(cfg.backbone.transform.normalize),
                                              int(cfg.backbone.transform.subtract_means), int(cfg.backbone.transform.to_float)])
            print("eval_unit transform", tag, tuple(y.shape), "absmax %.3f" % float(y.abs().max()))
    finally:
        torch.Tensor.cuda = orig_cuda
    set_cfg("yolact_base_config")
    cfg.mask_proto_debug = False

    # ---- mask_iou / jaccard
    def blobs(n, h, w):
        m = np.zeros((n, h, w), np.float32)
        for i in range(n):
            for _ in range(r.randint(1, 4)):
                y0, x0 = r.randint(0, h - 4), r.randint(0, w - 4)
                m[i, y0:y0 + r.randint(2, h // 2), x0:x0 + r.randint(2, w // 2)] = 1
        return m
    ma, mb = blobs(7, 45, 70), blobs(5, 45, 70)
    mb[4] = 0                       # empty mask: 0/0 -> NaN for non-crowd (kept: parity includes it)
    ba = np.sort(r.uniform(0, 300, (7, 2, 2)), axis=1).reshape(7, 4)[:, [0, 1, 2, 3]].astype(np.float32)
    bb = np.sort(r.uniform(0, 300, (5, 2, 2)), axis=1).reshape(5, 4).astype(np.float32)
    ba = ba[:, [0, 1, 2, 3]]
    out.update({"iou_masks_a": ma.astype(np.uint8), "iou_masks_b": mb.astype(np.uint8), "iou_boxes_a": ba, "iou_boxes_b": bb})
    for crowd in (False, True):
        t = "crowd" if crowd else "plain"
        out["iou_mask_" + t] = to_np(mask_iou(torch.from_numpy(ma), torch.from_numpy(mb), crowd))
        out["iou_box_" + t] = to_np(jaccard(torch.from_numpy(ba), torch.from_numpy(bb), crowd))
    print("eval_unit iou mask", out["iou_mask_plain"][0], "box", out["iou_box_plain"][0])

    # ---- prep_display (eval.py:135-262), production call form: undo_transform=False, img = BGR frame 0..255
    import eval as ref_eval

    class _OnGpu0(torch.Tensor):
        @property
        def device(self):
            return types.SimpleNamespace(index=0)

    orig_to = torch.Tensor.to

    def to_shim(self, *a, **k):
        if a and isinstance(a[0], int):
            return self
        return orig_to(self, *a, **k)

    n, ph, pw, K = 12, 69, 69, 32
    proto = np.maximum(r.standard_normal((ph, pw, K)), 0).astype(np.float32)
    proto = (proto + np.roll(proto, 1, 0) + np.roll(proto, 1, 1) + np.roll(proto, (2, 3), (0, 1))) / 4
    coef = np.tanh(r.standard_normal((n, K))).astype(np.float32)
    c = r.uniform(0.2, 0.8, (n, 2))
    wh = r.uniform(0.1, 0.6, (n, 2))
    box = np.concatenate([c - wh / 2, c + wh / 2], 1).astype(np.float32)
    score = np.sort(r.uniform(0.05, 0.99, n).astype(np.float32))[::-1].copy()
    cls = r.randint(0, 80, n).astype(np.int64)
    H, W = 203, 277
    frame = r.randint(0, 256, size=(H, W, 3)).astype(np.float32)
    out.update({"disp_proto": proto, "disp_coef": coef, "disp_box": box, "disp_score": score, "disp_cls": cls,
                "disp_frame": frame.astype(np.uint8)})
    torch.Tensor.to = to_shim
    try:
        for tag, argv, kw in (("masks", ["--top_k=8", "--score_threshold=0.15", "--display_text=False", "--display_bboxes=False"], {}),
                              ("classcolor", ["--top_k=15", "--score_threshold=0.3", "--display_text=False", "--display_bboxes=False"],
                               {"class_color": True}),
                              ("full", ["--top_k=5", "--score_threshold=0.15"], {})):
            ref_eval.parse_args(argv)
            ref_eval.color_cache.clear()
            det = {"box": torch.from_numpy(box.copy()), "mask": torch.from_numpy(coef), "class": torch.from_numpy(cls),
                   "score": torch.from_numpy(score), "proto": torch.from_numpy(proto)}
            img = torch.from_numpy(frame).as_subclass(_OnGpu0)
            with torch.no_grad():
                res = ref_eval.prep_display([{"detection": det, "net": None}], img, None, None, undo_transform=False, **kw)
            out["disp_" + tag] = np.asarray(res)
            print("eval_unit prep_display", tag, res.shape, res.dtype, "mean %.2f" % res.mean())
    finally:
        torch.Tensor.to = orig_to
    out["coco_classes"] = np.array(list(cfg.dataset.class_names))
    npz_save("eval_unit", **out)


def gen_state_keys():
    """state_dict key -> shape for every published config (SURVEY.md Appendix B)."""
    import json
    from data.config import cfg, set_cfg
    import yolact as ref_yolact
    out = {}
    for name in ("yolact_base_config", "yolact_resnet50_config", "yolact_im700_config", "yolact_darknet53_config",
                 "yolact_plus_base_config", "yolact_plus_resnet50_config"):
        set_cfg(name)
        net = ref_yolact.Yolact()
        out[name] = {k: list(v.shape) for k, v in net.state_dict().items()}
        x = torch.zeros(1, 3, cfg.max_size, cfg.max_size)
        print(name, len(out[name]), "keys")
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "state_keys.json"), "w") as f:
        json.dump(out, f)


def gen_reference_cfgs():
    """Every published config as plain JSON: exactly the fields yolact_b200.config.from_reference_cfg reads, so that
    the tests (tests/helpers.py load_reference_cfgs) can rebuild duck-typed cfg objects without the reference tree."""
    import json
    from data import config as rc
    switches = ("use_prediction_module", "use_yolo_regressors", "use_mask_scoring", "use_instance_coeff", "use_focal_loss",
                "use_objectness_score", "mask_proto_use_grid", "mask_proto_coeff_gate", "mask_proto_prototypes_as_features",
                "mask_proto_split_prototypes_by_head", "mask_proto_bias", "share_prediction_module", "use_maskiou",
                "rescore_mask", "rescore_bbox", "eval_mask_branch", "mask_proto_debug", "preserve_aspect_ratio")
    scalars = ("name", "max_size", "num_classes", "mask_dim", "nms_top_k", "nms_conf_thresh", "nms_thresh",
               "max_num_detections")
    out = {}
    for name in ("yolact_base_config", "yolact_resnet50_config", "yolact_im700_config", "yolact_darknet53_config",
                 "yolact_plus_base_config", "yolact_plus_resnet50_config"):
        c = getattr(rc, name)
        b = c.backbone
        d = {k: getattr(c, k) for k in scalars + switches if hasattr(c, k)}
        d["fpn"] = {"num_features": c.fpn.num_features}
        d["backbone"] = {
            "type": b.type.__name__, "args": [list(a) if isinstance(a, (list, tuple)) else a for a in b.args],
            "selected_layers": list(b.selected_layers), "pred_scales": [[float(v) for v in s] for s in b.pred_scales],
            "pred_aspect_ratios": [[list(r) for r in a] for a in b.pred_aspect_ratios],
            "use_square_anchors": b.use_square_anchors,
            "transform": {k: getattr(b.transform, k) for k in ("channel_order", "normalize", "subtract_means", "to_float")
                          if hasattr(b.transform, k)}}
        out[name] = d
        print("reference cfg", name, d["backbone"]["type"], d["backbone"]["args"])
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "reference_cfgs.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    if not os.path.isfile(os.path.join(REF, "eval.py")):
        raise SystemExit("no reference tree: set YOLACT_REFERENCE to the root of an upstream YOLACT checkout")
    install_shims()
    torch.set_num_threads(8)
    which = sys.argv[1:] or ["units", "nets"]
    if "keys" in which or "units" in which:
        gen_state_keys()
    if "units" in which:
        gen_detect_unit()
        gen_postprocess_unit()
        gen_dcn_unit()
    if "units" in which or "eval" in which:
        gen_eval_unit()
    if "units" in which or "cfgs" in which:
        gen_reference_cfgs()
    if "full" in which:
        for tag, name, size, post in FULL_CASES:
            gen_fullsize_case(tag, name, size, post)
    if "nets" in which:
        gen_network_case("net_resnet50_160", "yolact_resnet50_config", 1, 160, 160, (120, 150))
        gen_network_case("net_base_192x160_b2", "yolact_base_config", 2, 192, 160, (100, 100))
        gen_network_case("net_plus_resnet50_256", "yolact_plus_resnet50_config", 1, 256, 256, (160, 160), row_stride=4)
        gen_network_case("net_darknet53_160", "yolact_darknet53_config", 1, 160, 160, (96, 128))
