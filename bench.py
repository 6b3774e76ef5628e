#!/usr/bin/env python
"""bench.py -- frames/sec of the YOLACT inference path (Yolact.forward -> Detect -> postprocess) on
synthetic 550x550 frames, yolact_base (ResNet101-FPN), batch 8 per GPU (BASELINE.json configs[1]).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/<name>.npy

One step = one batch through the whole path.  Prints ONE JSON line (rank 0).  See DESIGN.md
"Measurement" for what each key means; in short:
  value     frames/s, inputs resident in HBM, fp32 masks [n,550,550] written for every detection
  e2e       (headline) frames/s through the reference-facing API with pinned HOST frames, eval.py's --benchmark
            protocol: H2D, `preds = net(x)`, per image `postprocess(preds, w, h, b)`, D2H of classes / scores /
            boxes / fp32 masks [:top_k] (eval.py:264-281), host-synchronised every step
  e2e_bits  (secondary) the batched extension API shipping ALL 100 masks per image 1 bit/pixel
  roofline  tcgen05 conv stack: algorithmic FLOPs (BASELINE.md section 3) / CUDA-event time of the conv-stack
            graph, against the measured cuBLAS bf16 peak of MEASURED_PEAKS.json (burst when the sampled clocks
            are unthrottled, sustained otherwise)
  fast_mode_f16tc  (secondary) the single-pass fp16 mode, which does NOT meet the 1e-3 tolerance
  cpu_baseline / --impl reference  the oracle port (torch-CPU fp32 conv stack + torch-CPU Detect/postprocess) on
            the same config and batch, all host threads; the reference arm imports no yolact_b200 module
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic conv FLOPs per image, 2*MAC (BASELINE.md section 3, counted from the reference model)
GFLOP_PER_IMAGE = {
    "yolact_resnet50_config": 118.28, "yolact_base_config": 164.68, "yolact_plus_resnet50_config": 141.38,
    "yolact_plus_base_config": 187.33, "yolact_im700_config": 262.93, "yolact_darknet53_config": 154.71,
}


# FPS the reference publishes for each config (BASELINE.md section 1: Titan Xp, batch 1, fp32, `eval.py --benchmark`,
# README.md:70-80).  Other hardware and batch size, so it is reported as an informational ratio, not as `vs_baseline`.
PUBLISHED_TITAN_XP_FPS = {
    "yolact_resnet50_config": 42.5, "yolact_darknet53_config": 40.0, "yolact_base_config": 33.5,
    "yolact_im700_config": 23.6, "yolact_plus_resnet50_config": 33.5, "yolact_plus_base_config": 27.3,
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="yolact_base_config")
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step")
    ap.add_argument("--size", type=int, default=0, help="image size (default: the config's max_size)")
    ap.add_argument("--precision", default="f16x3", choices=["f16x3", "f16tc", "f32"],
                    help="f16x3: split-precision tcgen05 (meets the reference tolerance; the headline mode); "
                         "f16tc: single-pass fp16 tcgen05 (fast mode); f32: CUDA-core fp32")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the secondary single-pass fp16 measurement")
    ap.add_argument("--cpu-sample", type=int, default=16, help="images in the cpu_baseline sample")
    ap.add_argument("--top-k", dest="top_k", type=int, default=5,
                    help="detections per image copied to the host in the e2e loop (eval.py --top_k default: 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of `value` returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs --steps >= 1")
    return args


# ---------------------------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU arm may use: affinity mask capped by the cgroup CPU quota (a container that sees
    128 CPUs but owns 16 of them must not spin 128 OpenMP threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def oracle_pipeline(cfg, sd):
    """The reference algorithm on the CPU (oracle port): net(x) + Detect + postprocess for one batch.
    torch-CPU fp32 conv stack (oracle/yolact_oracle.py) + torch-CPU Detect/postprocess
    (oracle/torch_port.py): the same ATen kernels the reference graph runs with --cuda=False."""
    import torch
    from oracle import yolact_oracle as O
    from oracle import torch_port as T
    orc = O.ConvStackOracle(cfg, sd)

    def run(x, out_hw):
        with torch.no_grad():
            raw = orc.forward(x)
            conf = torch.softmax(raw["conf"], -1)
            n_det = 0
            for b in range(x.shape[0]):
                det = T.detect_one(raw["loc"][b], conf[b], raw["mask"][b], raw["priors"], cfg.nms_conf_thresh,
                                   cfg.nms_thresh, cfg.nms_top_k, cfg.max_num_detections)
                if det is None:
                    continue
                det["proto"] = raw["proto"][b]
                fn = orc.maskiou if cfg.use_maskiou else None
                classes, scores, boxes, masks = T.postprocess_one(det, out_hw[1], out_hw[0], maskiou_fn=fn)
                n_det += int(masks.shape[0])
        return n_det
    return run


def pick_threads(run, size):
    """Best-performing thread count for the CPU arm (more threads is not always faster on a big host)."""
    import torch
    from oracle.weights import deterministic_input
    limit = host_threads()
    cands = sorted(set(min(c, limit) for c in (8, 16, 32, 64, 128, limit)))
    x = deterministic_input(1, size, size, 31337)
    best, best_t = cands[0], 1e30
    for c in cands:
        torch.set_num_threads(c)
        run(x, (size, size))
        t0 = time.perf_counter()
        run(x, (size, size))
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        elif dt > 1.5 * best_t:
            break   # past the knee: more threads only add synchronisation cost
    torch.set_num_threads(best)
    return best


def load_config_module():
    """yolact_b200/config.py loaded BY PATH (it has no package-relative imports): the reference arm must not import
    the yolact_b200 package, whose sub-modules bind the CUDA library."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_yb_config_standalone", os.path.join(ROOT, "yolact_b200", "config.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _Shape(object):
    def __init__(self, shape):
        self.shape = tuple(shape)


def reference_state_dict(config_name, seed=0):
    """Deterministic weights under the REFERENCE's state_dict keys / shapes (tests/golden/state_keys.json, written by
    oracle/gen_golden.py from the real reference model) -- identical to deterministic_state_dict(net.state_dict())."""
    from oracle.weights import deterministic_state_dict
    shapes = json.load(open(os.path.join(ROOT, "tests", "golden", "state_keys.json")))[config_name]
    return deterministic_state_dict({k: _Shape(v) for k, v in shapes.items()}, seed)


def time_cpu(cfg, sd, size, batch, steps, warmup, seed=8000):
    """The reference algorithm on the host cores: `steps` batches of `batch` images.  Returns (frames/s, s/step, dets/img)."""
    import torch
    from oracle.weights import deterministic_input
    run = oracle_pipeline(cfg, sd)
    pick_threads(run, size)
    for i in range(max(1, warmup)):
        run(deterministic_input(1, size, size, seed - 1 - i), (size, size))
    t0 = time.perf_counter()
    nd = 0
    for i in range(steps):
        nd += run(deterministic_input(batch, size, size, seed + i), (size, size))
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, nd / float(max(1, batch * steps))


MASK_SAMPLES = 1 << 21   # fp32 mask values kept by dump_outputs: 8 MB, plus 16 MB of float64 indices


def dump_outputs(out_dir, outputs):
    """Writes one step's outputs of the `value` path as out_dir/<name>.npy, so that two builds run with the same
    arguments (hence the same seeded inputs and weights) can be compared array by array.  Integer arrays are stored
    as float64, which holds them exactly.  The fp32 masks [B, M, h, w] are about 1 GB at the default workload, so
    only a fixed, seeded sample of their elements is written, with its flat indices."""
    import numpy as np
    import torch
    box, coef, cls, score, count, (masks, boxes_px) = outputs
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, masks.numel(), (min(MASK_SAMPLES, masks.numel()),), generator=g).sort().values
    arrays = {"box": box, "coef": coef, "class": cls, "score": score, "count": count, "box_px": boxes_px,
              "masks_sample": masks.reshape(-1)[idx.to(masks.device)], "masks_sample_index": idx}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def workload_string(cfg, size, B):
    return "%s @%d, batch %d/GPU, synthetic frames, random-init deterministic weights (100 detections/image)" % (
        cfg.name, size, B)


def reference_arm(args, rank):
    """bench.py --impl reference: the reference's CPU algorithm (oracle port: the ATen CPU kernels the reference itself
    runs with --cuda=False) on the SAME config / batch / metric.  Imports neither yolact_b200 nor any CUDA library."""
    if rank != 0:
        return 0
    import torch
    cm = load_config_module()
    cfg = cm.CONFIGS[args.config].copy()
    size = args.size or cfg.max_size
    B = args.batch
    sd = reference_state_dict(args.config, 0)
    steps = args.steps
    # bounded: a step is one batch of the same workload; cap the whole run at a few minutes of CPU time
    fps, s_per_step, nd = time_cpu(cfg, sd, size, B, steps, min(args.warmup, 2))
    line = {
        "metric": "frames/sec @ %dx%d %s (Yolact.forward + Detect + postprocess)" % (size, size, cfg.name),
        "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
        "impl": "reference", "value": fps, "ms_per_step": 1e3 * s_per_step, "dtype": "f32",
        "config": {"workload": workload_string(cfg, size, B), "global_batch": B, "image_size": size,
                   "detections_per_image": nd},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": "%d steps x %d images (the workload's batch), oracle port = torch-CPU fp32 conv stack + "
                                   "torch-CPU Detect/postprocess (the reference is Python and /root/reference does not exist "
                                   "on the GPU box); threads chosen by timing (host limit %d)" % (steps, B, host_threads())},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    assert not any(m == "yolact_b200" or m.startswith("yolact_b200.") for m in sys.modules), \
        "the reference arm must not import the product package"
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return reference_arm(args, rank)

    import torch
    import torch.distributed as dist
    import yolact_b200
    from yolact_b200.config import CONFIGS
    from yolact_b200.output_utils import assemble_masks_batch, postprocess
    from yolact_b200 import output_utils
    from yolact_b200.parallel import gather_detections
    from oracle.weights import deterministic_state_dict, deterministic_input

    cfg = CONFIGS[args.config].copy()
    size = args.size or cfg.max_size
    B = args.batch
    base = {
        "metric": "frames/sec @ %dx%d %s (Yolact.forward + Detect + postprocess)" % (size, size, cfg.name),
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "data": "synthetic",
    }
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    yolact_b200.cfg.replace(cfg.copy())

    def make_net(precision):
        net = yolact_b200.Yolact(cfg, precision=precision)
        net.detect.use_fast_nms = True   # what eval.py does from --fast_nms (default True, eval.py:50,871)
        net.load_state_dict(deterministic_state_dict(net.state_dict(), 0))
        net.eval()
        return net

    net = make_net(args.precision)
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}

    n_rot = 6  # 6 distinct input batches (6 x 29 MB = 174 MB > 126 MB L2) rotate through the loop
    xs = [deterministic_input(B, size, size, 1234 + 100 * rank + i).to(dev) for i in range(n_rot)]
    M, k = cfg.max_num_detections, cfg.mask_dim
    # Two compute streams: the mask assembly of step i (HBM-write bound) runs on s_post while the conv stack of step
    # i+1 (tensor / L2 bound) already runs on the main stream; outputs are double-buffered.  BENCH_OVERLAP=0 serialises.
    overlap = os.environ.get("BENCH_OVERLAP", "1") != "0"
    masks_f32 = [torch.empty(B, M, size, size, dtype=torch.float32, device=dev) for _ in range(2 if overlap else 1)]
    s_post = torch.cuda.Stream() if overlap else None
    # The network outputs of step i are read by s_post; they are kept referenced until step i+2, whose first action
    # is to make the main stream wait for step i's mask assembly -- so the caching allocator (which only tracks the
    # allocating stream) can never hand their memory to main-stream work that runs before s_post has read it.
    hold = [None, None]
    ev_post_v = [torch.cuda.Event(), torch.cuda.Event()]

    def step_device(net_, i, fmt="f32", out=None):
        if overlap and hold[i % 2] is not None:
            torch.cuda.current_stream().wait_event(ev_post_v[i % 2])
        box, coef, cls, score, count, proto = net_.infer_padded(xs[i % n_rot])
        # all M padded rows are assembled (no host sync on the count); with these weights count == M
        if overlap:
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(s_post):
                s_post.wait_event(ev)
                res = assemble_masks_batch(proto, coef, box, size, size, True, fmt, masks_out=out[i % 2])
                ev_post_v[i % 2].record(s_post)
            hold[i % 2] = (box, coef, proto, res)
        else:
            res = assemble_masks_batch(proto, coef, box, size, size, True, fmt, masks_out=out[0])
        if world > 1:
            gather_detections(box, coef, cls, score, count, per_rank_batch=B)
        return box, coef, cls, score, count, res

    def barrier_sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier_sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        if s_post is not None:
            torch.cuda.current_stream().wait_stream(s_post)   # the last steps' mask assembly is inside the timed region
        e1.record()
        barrier_sync()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- value: inputs resident in HBM, fp32 masks for all 100 detections of every image
    l0 = net.launch_count() + output_utils.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = {}

    def step_value(i):
        last["out"] = step_device(net, i, "f32", masks_f32)
    ms = timed(step_value, args.steps, max(3, args.warmup))
    clocks = sampler.stop() if rank == 0 else None
    # kernels launched inside the TIMED region only (the counter also saw the warm-up steps of `timed`)
    launches = (net.launch_count() + output_utils.launch_count() - l0) * args.steps // (args.steps + max(3, args.warmup))
    fps = world * B * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["out"])   # timed() has synchronised: the last step is complete
    last.clear()
    hold[0] = hold[1] = None

    # ---- e2e (headline): the reference-facing API with HOST frames, eval.py's --benchmark protocol --------------------
    #   batch = img.cuda()              (H2D from pinned memory, every step)            eval.py:940-942
    #   preds = net(batch)              (Yolact.forward + Detect, list of dicts)        eval.py:945
    #   per image: postprocess(preds, w, h, batch_idx, crop_masks, score_threshold)     eval.py:266 (prep_benchmark)
    #              classes / scores / boxes / fp32 masks [:top_k] -> host               eval.py:269-277 (top_k = 5, eval.py:46)
    #   synchronize                                                                      eval.py:279-281
    # Two extra streams double-buffer the copies (H2D of step i+1 and D2H of step i-1 overlap step i); net() itself
    # blocks the host once per step (Detect's variable-size output), like the reference.
    top_k = args.top_k
    hx = [deterministic_input(B, size, size, 555 + 10 * rank + i).pin_memory() for i in range(2)]
    dx = [torch.empty(B, 3, size, size, device=dev) for _ in range(2)]
    h_out = [{"classes": torch.empty(B, top_k, dtype=torch.int64).pin_memory(),
              "scores": torch.empty(B, top_k, dtype=torch.float32).pin_memory(),
              "scores2": torch.empty(B, top_k, dtype=torch.float32).pin_memory(),
              "boxes": torch.empty(B, top_k, 4, dtype=torch.int64).pin_memory(),
              "masks": torch.empty(B, top_k, size, size, dtype=torch.float32).pin_memory()} for _ in range(2)]
    h2d_api = B * 3 * size * size * 4
    d2h_api = B * top_k * (8 + 4 + 32 + size * size * 4)
    s_main = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_comp = [torch.cuda.Event() for _ in range(2)]
    ev_d2h = [torch.cuda.Event() for _ in range(2)]
    st = {"n": 0, "dets": 0}

    def issue_h2d(i):
        kk = i % 2
        with torch.cuda.stream(s_in):
            if i >= 2:
                s_in.wait_event(ev_comp[kk])         # dx[kk] was last read by the network of step i-2
            dx[kk].copy_(hx[kk], non_blocking=True)
            ev_in[kk].record(s_in)

    def step_api(_i):
        i = st["n"]
        st["n"] += 1
        kk = i % 2
        if i == 0:
            issue_h2d(0)
        s_main.wait_event(ev_in[kk])
        issue_h2d(i + 1)                             # next step's frames travel while this step computes
        preds = net(dx[kk])                          # Yolact.forward + Detect; host-syncs on the detection counts
        ev_comp[kk].record(s_main)
        ho = h_out[kk]
        for b in range(B):
            t = postprocess(preds, size, size, batch_idx=b, crop_masks=True, score_threshold=0)
            classes, scores, boxes, masks = [v[:top_k] if not isinstance(v, list) else [u[:top_k] for u in v] for v in t]
            n = int(classes.shape[0])
            st["dets"] += n
            ev = torch.cuda.Event()
            ev.record(s_main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev)
                sc = scores if not isinstance(scores, list) else scores[0]
                for tt in (classes, sc, boxes, masks):
                    tt.record_stream(s_out)
                ho["classes"][b, :n].copy_(classes, non_blocking=True)
                ho["scores"][b, :n].copy_(sc, non_blocking=True)
                if isinstance(scores, list):
                    scores[1].record_stream(s_out)
                    ho["scores2"][b, :n].copy_(scores[1], non_blocking=True)
                ho["boxes"][b, :n].copy_(boxes, non_blocking=True)
                ho["masks"][b, :n].copy_(masks, non_blocking=True)
        if world > 1:
            # the shard's detections join the global batch: one pack kernel + ONE NCCL all_gather of fixed-size records
            # (the analogue of CustomDataParallel.gather, eval.py:630-634)
            gather_detections(*net.last_padded_detections, per_rank_batch=B)
        ev_d2h[kk].record(s_out)
        if i >= 1:
            ev_d2h[(i - 1) % 2].synchronize()        # step i-1's results are on the host

    def api_drain():
        ev_d2h[(st["n"] - 1) % 2].synchronize()

    def timed_api(step_fn, drain_fn, steps, warmup):
        for i in range(warmup):
            step_fn(i)
        drain_fn()
        barrier_sync()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step_fn(i)
        drain_fn()
        s_main.wait_stream(s_out)
        s_main.wait_stream(s_in)
        if s_post is not None:
            s_main.wait_stream(s_post)
        e1.record()
        barrier_sync()
        wall = (time.perf_counter() - t0) * 1e3
        return max_over_ranks(e0.elapsed_time(e1)), wall

    ms_api, wall_api = timed_api(step_api, api_drain, args.steps, 3)
    fps_api = world * B * args.steps / (ms_api / 1e3)

    # ---- e2e_bits (secondary, labelled): same host-to-host loop through the batched extension API --
    # infer_padded (no host sync) + ONE mask-assembly launch per batch, ALL 100 masks per image shipped 1 bit/pixel.
    wpr = (size + 31) // 32
    h_cls = [torch.empty(B, M, dtype=torch.int64).pin_memory() for _ in range(2)]
    h_score = [torch.empty(B, M, dtype=torch.float32).pin_memory() for _ in range(2)]
    h_count = [torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(2)]
    h_boxes = [torch.empty(B, M, 4, dtype=torch.int64).pin_memory() for _ in range(2)]
    h_masks = [torch.empty(B, M, size, wpr, dtype=torch.int32).pin_memory() for _ in range(2)]
    d_masks = [torch.empty(B, M, size, wpr, dtype=torch.int32, device=dev) for _ in range(2)]
    d_boxes = [torch.empty(B, M, 4, dtype=torch.int64, device=dev) for _ in range(2)]
    d2h_bits = sum(t[0].numel() * t[0].element_size() for t in (h_cls, h_score, h_count, h_boxes, h_masks))
    ev_post = [torch.cuda.Event() for _ in range(2)]
    hold_e = [None, None]
    sb = {"n": 0}

    def step_bits(_i):
        i = sb["n"]
        sb["n"] += 1
        kk = i % 2
        with torch.cuda.stream(s_in):
            if i >= 2:
                s_in.wait_event(ev_comp[kk])          # dx[kk] was last read by the compute of step i-2
            dx[kk].copy_(hx[kk], non_blocking=True)
            ev_in[kk].record(s_in)
        s_main.wait_event(ev_in[kk])
        if i >= 2 and overlap:
            s_main.wait_event(ev_post[kk])            # step i-2's mask assembly has read its inputs (see `hold`)
        if i >= 2:
            (s_post if overlap else s_main).wait_event(ev_d2h[kk])   # d_masks[kk] / d_boxes[kk] were read by step i-2's D2H
        box, coef, cls, score, count, proto = net.infer_padded(dx[kk])
        ev_comp[kk].record(s_main)
        if overlap:
            with torch.cuda.stream(s_post):
                s_post.wait_event(ev_comp[kk])
                assemble_masks_batch(proto, coef, box, size, size, True, "bits", masks_out=d_masks[kk], boxes_out=d_boxes[kk])
                ev_post[kk].record(s_post)
            hold_e[kk] = (box, coef, proto)
        else:
            assemble_masks_batch(proto, coef, box, size, size, True, "bits", masks_out=d_masks[kk], boxes_out=d_boxes[kk])
            ev_post[kk].record(s_main)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_post[kk])
            for t in (cls, score, count):
                t.record_stream(s_out)
            h_cls[kk].copy_(cls, non_blocking=True)
            h_score[kk].copy_(score, non_blocking=True)
            h_count[kk].copy_(count, non_blocking=True)
            h_boxes[kk].copy_(d_boxes[kk], non_blocking=True)
            h_masks[kk].copy_(d_masks[kk], non_blocking=True)
            ev_d2h[kk].record(s_out)
        if i >= 1:
            ev_d2h[(i - 1) % 2].synchronize()

    def bits_drain():
        ev_d2h[(sb["n"] - 1) % 2].synchronize()

    torch.cuda.synchronize()
    ms_bits, wall_bits = timed_api(step_bits, bits_drain, args.steps, 3)
    fps_bits = world * B * args.steps / (ms_bits / 1e3)

    # ---- roofline of the dominant kernel family (tcgen05 conv stack), timed live with CUDA events
    def conv_ms(net_):
        net_.train()
        r = timed(lambda i: net_.forward_conv_only(xs[i % n_rot]), args.steps, 3)
        net_.eval()
        return r
    ms_conv = conv_ms(net)
    gflop = GFLOP_PER_IMAGE.get(args.config, 0.0) * size * size / float(cfg.max_size * cfg.max_size)
    achieved = gflop * B * args.steps / (ms_conv / 1e3) / 1e3   # algorithmic TFLOP/s per GPU
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # burst peak when the timed region ran unthrottled at (close to) the maximum SM clock, the sustained figure otherwise
    unthrottled = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and
                       clocks["sm_mhz"] >= 0.95 * clocks["sm_max_mhz"] and
                       not set(clocks.get("reasons") or []) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"})
    if peaks:
        peak = peaks.get("bf16_tflops") if (unthrottled or rank != 0) else peaks.get("bf16_tflops_sustained")
        peak = peak or peaks.get("bf16_tflops_sustained") or 1400.0
        peak_src = "MEASURED_PEAKS.json %s cuBLAS bf16" % ("burst (clocks unthrottled during the timed region)" if unthrottled else "sustained")
    else:
        peak, peak_src = 1400.0, "fallback ~1.4 PF sustained (B200_PROFILING.md)"
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        if args.config == "yolact_base_config" and B == 8 and size == cfg.max_size and isinstance(tj.get(args.precision), dict):
            traffic = tj[args.precision].get("traffic_bytes_per_step")   # measured for this workload only
    except Exception:
        pass
    passes = 3 if args.precision == "f16x3" else 1
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "tc_chain_kernel + tc_conv_kernel (all conv launches of one step)",
                "ms_conv_stack_per_step": ms_conv / args.steps, "peak_source": peak_src,
                "algorithmic_gflop_per_step": gflop * B,
                "mma_passes": passes, "tensor_pipe_tflops_issued": achieved * passes,
                "note": "achieved counts the reference's algorithmic FLOPs once; the split-precision mode issues 3 fp16 MMA "
                        "passes per k-block (hi*hi + lo*hi + hi*lo), so the tensor pipe executes 3x that" if passes == 3 else None}

    line = dict(base)
    line.update({
        "value": fps, "ms_per_step": ms / args.steps,
        "dtype": {"f16x3": "f16x3 (fp16 hi+lo operand pairs, 3 tcgen05 passes, fp32 accumulate: fp32-equivalent, parity-tested at 1e-3)",
                  "f16tc": "f16", "f32": "f32"}[args.precision],
        "config": {"workload": workload_string(cfg, size, B), "global_batch": world * B, "image_size": size,
                   "parallelism": "dp%d" % world, "detections_per_image": M, "precision": args.precision,
                   "mask_format_value": "f32 [n,h,w], all %d detections" % M,
                   "l2": "6 rotating input batches (174 MB) and ~2 GB of activations+masks per step exceed the 126 MB L2",
                   "cuda_graph": True,
                   "streams": "mask assembly of step i overlaps the conv stack of step i+1 (2 compute streams)" if overlap
                              else "single compute stream"},
        "e2e": {"value": fps_api, "unit": "frames/s", "h2d_bytes_per_step": h2d_api, "d2h_bytes_per_step": d2h_api,
                "ms_per_step": ms_api / args.steps, "host_wall_ms_per_step": wall_api / args.steps,
                "api": "preds = net(x); per image postprocess(preds, w, h, batch_idx) -> classes/scores/boxes/fp32 masks[:top_k] "
                       "to the host (eval.py prep_benchmark, :264-281)", "top_k": top_k,
                "detections_copied_per_image": st["dets"] / float(max(1, st["n"] * B)),
                "pipelining": "double-buffered copies: H2D(i+1) | net+postprocess(i) | D2H(i-1); the host blocks inside net() "
                              "(Detect's counts) and on each step's D2H"},
        "e2e_bits": {"value": fps_bits, "unit": "frames/s", "h2d_bytes_per_step": h2d_api, "d2h_bytes_per_step": d2h_bits,
                     "ms_per_step": ms_bits / args.steps, "host_wall_ms_per_step": wall_bits / args.steps,
                     "api": "extension API: infer_padded (no host sync) + one batched mask-assembly launch, ALL %d masks per "
                            "image shipped 1 bit/pixel" % M},
        "gpu_launches": int(launches),
        "vs_published_titan_xp": {"ratio_per_gpu": fps / world / PUBLISHED_TITAN_XP_FPS[args.config],
                                  "published_fps": PUBLISHED_TITAN_XP_FPS[args.config],
                                  "note": "reference README (BASELINE.md section 1): 1 Titan Xp, batch 1, fp32"}
        if args.config in PUBLISHED_TITAN_XP_FPS and size == cfg.max_size else None,
        "clocks": clocks,
        "roofline": roofline,
    })

    # ---- fast mode (secondary, labelled): single-pass fp16 tcgen05, outside the 1e-3 tolerance
    if args.precision == "f16x3" and not args.no_fast_mode:
        del net
        hold[0] = hold[1] = None
        hold_e[0] = hold_e[1] = None
        torch.cuda.empty_cache()
        fast = make_net("f16tc")
        ms_f = timed(lambda i: step_device(fast, i, "f32", masks_f32), args.steps, 3)
        ms_fc = conv_ms(fast)
        ach_f = gflop * B * args.steps / (ms_fc / 1e3) / 1e3
        line["fast_mode_f16tc"] = {
            "value": world * B * args.steps / (ms_f / 1e3), "unit": "frames/s", "ms_per_step": ms_f / args.steps,
            "ms_conv_stack_per_step": ms_fc / args.steps, "conv_tflops": ach_f, "conv_frac_of_peak": ach_f / peak,
            "note": "single-pass fp16 operands: head tensors ~2e-3 of range from the fp32 reference, class ids not "
                    "bit-exact (profiles/parity_r02.md) -- NOT the headline"}

    # ---- cpu_baseline (rank 0, N == 1 only): bounded sample of the same workload on the host cores
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        nsteps = max(1, args.cpu_sample // B)
        cpu_fps, _, nd = time_cpu(cfg, sd, size, B, nsteps, 1)
        line["cpu_baseline"] = {"value": cpu_fps, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": "%d step(s) x %d images of the same workload, %.0f detections/image" % (nsteps, B, nd)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
