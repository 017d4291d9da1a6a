#!/usr/bin/env python
"""bench.py — images/sec of the SSD hot path on N x B200, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--config cfg2|cfg3|cfg4|cfg5|cfg5stress] [--scaling weak|strong] [--batch B]
                    [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

Workloads (BASELINE.json configs[1..4], SURVEY 8d; synthetic uint8 images seed 1234, synthetic weights with the
reference's init statistics seed 0, post-process defaults thr 0.01 / IoU 0.6 / 300 per level / 100 detections /
DIoU + centerness rescore):
  cfg2 (default; the config the metric is quoted on)  SSD-ResNet50 512x512, 64 images per GPU, conv + decode + NMS
  cfg3        SSD-MobileNetV2 300x300, 64 images per GPU (512 over 8), conv + decode + NMS + detection all-gather
  cfg4        SSDFPN-ResNet50 640x640 training step front half: conv stack (logits) + match + MultiBoxLoss
              hard-negative mining, 16 images per GPU (128 over 8)
  cfg5        SSDBiFPN-RegNetX032 1280x1280, 4 images per GPU (32 over 8), conv + decode + NMS
  cfg5stress  same with 20 000 candidates per level: N = 100 000 boxes per image into NMS
--scaling weak (default): the per-GPU batch above at every N.  --scaling strong: the config's GLOBAL batch
(64 / 512 / 128 / 32 / 32) split over the N ranks.

A "step" = one batch through pack -> conv stack -> decode -> NMS [-> NCCL all-gather of the [B,100,6] detections
when N > 1] (cfg4: -> match -> loss).  Decode/NMS/all-gather of step i run on a side stream and overlap the conv
stack of step i+1; every step's work is inside the timed region (the region ends after a join).
  value     images/s with the batch already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e       images/s through the public host API (SSDDetector.detect_host / pipeline.LossStep.loss_host): pinned
            host batch -> H2D -> the same step -> D2H of the result, every step, inside the timed region
  roofline  the dominant kernel group of the config; `rooflines` has every group (conv, decode, nms, match,
            loss), each timed alone with CUDA events over K replays: algorithmic work per step (SURVEY 8d
            formulas) / device time, against MEASURED_PEAKS.json
  self_check  before anything is timed, the outputs of the timed plan (multi-way / weight-resident / paired
            launches, CUDA-graph replay) are compared bit for bit with the SAME model planned under
            SSDSB_WAYS=1 SSDSB_NO_PAIR=1 and replayed eagerly, and the detector's overlapped host path with
            its synchronous path.  A mismatch aborts the bench.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, installed by oracle/build_ref.py) through its own
            create_model / Decoder / extract_targets / MultiBoxLoss on this host's cores, on a bounded sample of
            the same workload (kind "reference"); the oracle port (kind "port") only if oracle/_ref is absent.
--impl reference times that CPU path alone and never imports ssds_pytorch_b200.
--dump-outputs DIR  after the timed steps, rank 0 writes what the last device-resident step returned as DIR/<name>.npy
            (detect: scores [B,100], boxes [B,100,4], classes [B,100]; cfg4: loss [3] = cls_loss, loc_loss,
            fg_targets), float32, so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec (fwd+decode+NMS)"
_R6, _R5 = [[1, 2, 0.5]] * 6, [[1, 2, 0.5]] * 5

CONFIGS = {
    "cfg2": dict(
        workload="SSD-ResNet50 512x512 bf16 inference: conv stack + decode + NMS (BASELINE.json configs[1])",
        model=dict(SSDS="SSD", NETS="ResNet50", IMAGE_SIZE=[512, 512], NUM_CLASSES=80,
                   FEATURE_LAYER=[[3, 4, 5, "Conv:S", "Conv:S", "Conv:S"], [512, 1024, 2048, 512, 256, 256]],
                   SIZES=[[2.0, 2.828]] * 6, ASPECT_RATIOS=_R6),
        kind="detect", batch=64, global_batch=64, per_level=300, cpu_images=8, dominant="conv", bound="tensor"),
    "cfg3": dict(
        workload="SSD-MobileNetV2 300x300 bf16 inference, 512 images over 8 GPUs (64 per GPU): conv stack + decode "
                 "+ NMS + NCCL all-gather of the detections (BASELINE.json configs[2])",
        model=dict(SSDS="SSD", NETS="MobileNetV2", IMAGE_SIZE=[300, 300], NUM_CLASSES=80,
                   FEATURE_LAYER=[[5, 7, "Conv:S", "Conv:S", "Conv:S", "Conv:S"], [96, 320, 512, 256, 256, 128]],
                   SIZES=[[2.0, 2.828]] * 6, ASPECT_RATIOS=_R6),
        kind="detect", batch=64, global_batch=512, per_level=300, cpu_images=32, dominant="conv", bound="hbm"),
    "cfg4": dict(
        workload="SSDFPN-ResNet50 640x640 training-step front half: conv stack (logits) + anchor match + MultiBoxLoss "
                 "hard-negative mining, 128 images over 8 GPUs (16 per GPU) (BASELINE.json configs[3])",
        model=dict(SSDS="SSDFPN", NETS="ResNet50", IMAGE_SIZE=[640, 640], NUM_CLASSES=80,
                   FEATURE_LAYER=[[3, 4, 5, "Conv:S", "Conv:S"], [512, 1024, 2048, 2048, 256]],
                   SIZES=[[4.0, 5.04, 6.35]] * 5, ASPECT_RATIOS=_R5),
        kind="loss", batch=16, global_batch=128, per_level=300, cpu_images=4, dominant="conv", bound="tensor"),
    "cfg5": dict(
        workload="SSDBiFPN-RegNetX032 1280x1280 bf16 inference, 32 images over 8 GPUs (4 per GPU): conv stack + "
                 "decode + NMS (BASELINE.json configs[4], default 300 candidates/level)",
        model=dict(SSDS="SSDBiFPN", NETS="RegNetX032", IMAGE_SIZE=[1280, 1280], NUM_CLASSES=80,
                   FEATURE_LAYER=[[2, 3, 4, "Conv:S", "Conv:S"], [192, 432, 1008, 1008, 256]],
                   SIZES=[[4.0]] * 5, ASPECT_RATIOS=_R5),
        kind="detect", batch=4, global_batch=32, per_level=300, cpu_images=2, dominant="conv", bound="tensor"),
}
CONFIGS["cfg5stress"] = dict(CONFIGS["cfg5"], per_level=20000, cpu_images=1,
                             workload=CONFIGS["cfg5"]["workload"].replace(
                                 "default 300 candidates/level", "100k-anchor NMS stress: 20 000 candidates/level"))


def cfg_dict(name="cfg2"):
    c = CONFIGS[name]
    return {"MODEL": dict(c["model"]), "DATASET": {"PREPROC": {"MEAN": 0, "STD": 255}},
            "POST_PROCESS": {"MAX_DETECTIONS_PER_LEVEL": c["per_level"]}}


def measured_conv_traffic(name):
    """DRAM bytes of all conv-stack launches of one step from the committed ncu launch list of this config
    (profiles/r2_conv_traffic_<config>.json, written by tools/conv_traffic.py), or None."""
    for f in (f"r2_conv_traffic_{name}.json",) + (("r1_conv_traffic.json",) if name == "cfg2" else ()):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", f)))
            return d["conv_dram_bytes_per_step"], f
        except Exception:
            pass
    return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed regions (B200_PROFILING.md's clocks line).  NVML through
    pynvml (a sample every ~10 ms: the timed regions last tenths of a second); nvidia-smi as a fallback (one sample
    per ~0.5 s).  Only samples taken while the GPU was busy (utilisation > 0 or power above idle) count as "under load"."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.source = index, [], False, "nvidia-smi"
        self.active = False          # bench code sets this True only inside timed regions

    def _nvml_loop(self):
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        bits = [N.nvmlClocksEventReasonHwSlowdown, N.nvmlClocksEventReasonHwThermalSlowdown,
                N.nvmlClocksEventReasonSwThermalSlowdown, N.nvmlClocksEventReasonSwPowerCap]
        self.source = "nvml"
        while not self.stop_flag:
            if self.active:
                sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
                r = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
            time.sleep(0.01)

    def run(self):
        try:
            self._nvml_loop()
            return
        except Exception:
            self.source = "nvidia-smi"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out and self.active:
                    self.samples.append([v.strip() for v in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(s) > 2 + i and s[2 + i] == "Active"
                                                              for s in self.samples)]
        mx = max([int(s[1]) for s in self.samples if s[1].isdigit()], default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": mx,
                "reasons": reasons, "samples": len(self.samples), "source": self.source,
                "when": "sampled inside the two timed regions (device-resident and end-to-end)"}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_run(name, n_images, threads, steps=1, warm=True):
    """The reference's own CPU path on `n_images` synthetic images.  Returns (seconds list, kind, what)."""
    c = CONFIGS[name]
    from oracle import ref_runner
    if ref_runner.available():
        t, what = ref_runner.run(c["model"], n_images, threads, steps=steps, warm=warm, kind=c["kind"],
                                 per_level=c["per_level"])
        return t, "reference", what
    if name != "cfg2":
        raise RuntimeError("oracle/_ref is missing (python oracle/build_ref.py) and the oracle port times cfg2 only")
    return [_cpu_port_run(n_images, threads, warm) for _ in range(steps)], "port", \
        "CPU port of the reference path (oracle/): torch fp32 conv stack + numpy decode/NMS"


def _cpu_port_run(n_images, threads, warm=True):
    """Fallback when oracle/_ref is absent: the oracle restatement (fp32 torch conv stack + numpy decode/NMS)."""
    import torch
    from collections import OrderedDict
    from oracle import box_oracle as O
    from oracle import model_oracle as M
    from ssds_pytorch_b200 import synth
    m = CONFIGS["cfg2"]["model"]
    torch.set_num_threads(threads)
    sd = synth.synthetic_state_dict(m["NETS"], m["FEATURE_LAYER"], [6] * 6, 80, seed=0, style="init")
    g = torch.Generator().manual_seed(1234)
    x = torch.randint(0, 256, (n_images, 512, 512, 3), generator=g, dtype=torch.uint8)
    x = (x.float() / 255.0).permute(0, 3, 1, 2).contiguous()

    def once(xx):
        with torch.no_grad():
            loc, conf = M.ssd_resnet_forward(sd, xx, m["FEATURE_LAYER"], training=False, policy="fp32")
        strides = [512 // c.shape[-1] for c in conf]
        anchors = OrderedDict((s, O.generate_anchors(s, m["ASPECT_RATIOS"][i], m["SIZES"][i]))
                              for i, s in enumerate(strides))
        return O.decoder_call([l.numpy() for l in loc], [c.numpy() for c in conf], anchors,
                              0.01, 0.6, 100, 300, True, True)

    if warm:
        once(x[:1])
    t0 = time.perf_counter()
    once(x)
    return time.perf_counter() - t0


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def best_cpu_threads(name):
    """The CPU arm is given its best case: torch's intra-op pool is probed on one image at 8, 16, 32, 64, ... threads
    up to the host's count, stopping as soon as a larger pool is slower (many-core hosts oversubscribe badly on
    these small convs and on the python NMS loop; the 100k-candidate stress would take minutes per image at 200
    threads); the fastest setting is used and reported as `cores`."""
    allc = host_threads()
    cands = [c for c in (8, 16, 32, 64, 128, 256) if c < allc] + [allc]
    if allc <= 8:
        cands = [allc]
    cpu_reference_run(name, 1, cands[0], warm=False)                      # page in / warm up
    best_t, best_c = None, cands[0]
    for c in cands:
        t = cpu_reference_run(name, 1, c, warm=False)[0][0]
        if best_t is not None and t > best_t:
            break
        best_t, best_c = t, c
    return best_c


def cpu_baseline(name, n, steps):
    threads = best_cpu_threads(name)
    t, kind, what = cpu_reference_run(name, n, threads, steps=steps, warm=True)
    sec = sorted(t)[len(t) // 2]
    H, W = CONFIGS[name]["model"]["IMAGE_SIZE"]
    return sec, {"value": n / sec, "unit": "images/s", "cores": threads, "kind": kind,
                 "sample": f"{n} images of {H}x{W} per step ({what}), median of {len(t)} step(s) after a 1-image "
                           f"warm-up; thread count = fastest of a probe over the host's {host_threads()} threads"}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    c = CONFIGS[args.config]
    n = args.cpu_images or c["cpu_images"]
    steps = args.steps
    sec, base = cpu_baseline(args.config, n, steps)
    v = n / sec
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": c["workload"], "name": args.config, "images_per_step": n,
                       "arm": "the unmodified reference on the host CPU (oracle/_ref)" if base["kind"] == "reference"
                       else "CPU port of the reference path (oracle/)"},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "native_so_loaded": "ssds_pytorch_b200" in sys.modules}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ B200 arm
def _timed(fn, K, barrier):
    import torch
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K


def _self_check(name, sd, dev_in, plan_outputs, make_model):
    """Bit-exact comparison of the timed plan's outputs with the 1-way, unpaired, un-fused (three launches per
    inverted residual), eagerly replayed plan."""
    import torch
    os.environ["SSDSB_WAYS"], os.environ["SSDSB_NO_PAIR"], os.environ["SSDSB_NO_MBFUSE"] = "1", "1", "1"
    try:
        plain = make_model()
        loc, conf = plain(dev_in, use_graph=False)
        torch.cuda.synchronize()
        n_pair = sum(v["kind"].startswith(("pair1x1", "mbconv")) for v in plain.plan_for(dev_in)["info"].values())
        assert n_pair == 0
        for a, b in zip(plan_outputs, list(loc) + list(conf)):
            if not torch.equal(a, b):
                raise SystemExit(f"bench self-check FAILED ({name}): timed plan output differs from the 1-way "
                                 f"unpaired eager plan (max |diff| {(a - b).abs().max().item()})")
    finally:
        del os.environ["SSDSB_WAYS"], os.environ["SSDSB_NO_PAIR"], os.environ["SSDSB_NO_MBFUSE"]
    del plain
    torch.cuda.empty_cache()
    return ("timed plan (multi-way/resident/paired/fused-block launches, CUDA-graph replay) == 1-way unpaired "
            "un-fused eager plan, bit for bit")


DUMP_LIMIT = 64 << 20


def dump_outputs(outdir, arrays):
    """One float32 .npy per output; above DUMP_LIMIT bytes in all, a fixed seeded sample of the images."""
    arrays = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        B = next(iter(arrays.values())).shape[0]
        keep = np.sort(np.random.default_rng(0).choice(B, max(1, B * DUMP_LIMIT // total), replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
    os.makedirs(outdir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(outdir, k + ".npy"), v)


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from ssds_pytorch_b200 import synth
    from ssds_pytorch_b200.box import decode_levels, nms as nms_op
    from ssds_pytorch_b200.model import number_box_from_cfg
    from ssds_pytorch_b200.pipeline import LossStep
    from ssds_pytorch_b200.ssds import SSDDetector, gather_detections

    name = args.config
    c = CONFIGS[name]
    m = c["model"]
    K, W = args.steps, max(args.warmup, 3)
    if args.batch:
        B = args.batch
    elif args.scaling == "strong":
        if c["global_batch"] % world:
            raise SystemExit(f"strong scaling: global batch {c['global_batch']} is not divisible by {world} ranks")
        B = c["global_batch"] // world
    else:
        B = c["batch"]
    H, Wd = m["IMAGE_SIZE"]
    L = len(m["FEATURE_LAYER"][0])
    C = m["NUM_CLASSES"]
    nb = number_box_from_cfg(m)
    sd = synth.synthetic_state_dict(m["NETS"], m["FEATURE_LAYER"], nb, C, seed=0, style="init", ssds=m["SSDS"])
    device = torch.device("cuda", local)
    g = torch.Generator().manual_seed(1234 + rank)              # rank r holds images [rB, (r+1)B)
    host = [torch.randint(0, 256, (B, H, Wd, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    dev_in = host[0].cuda()
    detect = c["kind"] == "detect"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if detect:
        det = SSDDetector(cfg_dict(name), sd, device=device, use_graph=True)
        model, anchors = det.model, det.anchors

        def make_plain():
            return SSDDetector(cfg_dict(name), sd, device=device, use_graph=False).model

        packed = torch.empty((B, 100, 6), dtype=torch.float32, device=device)

        def step_device():
            # decode + NMS (+ all-gather) of this step run on the detector's side stream and overlap the
            # conv stack of the next step; det.join() below makes the timed region wait for them
            out = det.detect_device(dev_in, overlap=True, packed_out=packed)
            if world > 1:
                with torch.cuda.stream(det._post_stream):
                    gather_detections(packed)
                    det._post_done = torch.cuda.Event()
                    det._post_done.record(det._post_stream)
            return out

        def step_host(i):
            return det.detect_host(host[i % 2], slot=i % 2, gather=world > 1)

        join = det.join
        api = "SSDDetector.detect_host(uint8 NHWC pinned batch)"
        h2d = B * H * Wd * 3
    else:
        ls = LossStep(cfg_dict(name), sd, device=device, use_graph=True)
        model, anchors = ls.model, ls.anchors
        tg_host = synth.synthetic_targets(B, seed=4321 + rank).pin_memory()
        tg_dev = tg_host.cuda()

        def make_plain():
            return LossStep(cfg_dict(name), sd, device=device, use_graph=False).model

        def step_device():
            return ls.loss_device(dev_in, tg_dev)

        def step_host(i):
            return ls.loss_host(host[i % 2], tg_host)

        join = lambda: None
        api = "pipeline.LossStep.loss_host(uint8 NHWC pinned batch, [B,32,5] pinned targets)"
        h2d = B * H * Wd * 3 + tg_host.numel() * 4
    plan = model.plan_for(dev_in)
    flops_step = plan["flops"]
    conv_bytes = sum(v.get("bytes", 0) for v in plan["info"].values())
    # what the plan as launched has to move at least (fused inverted residuals: block input + output only)
    conv_bytes_as_launched = sum(v.get("bytes_fused", v.get("bytes", 0)) for v in plan["info"].values())
    n_fused = sum(v["kind"].startswith("mbconv") for v in plan["info"].values())

    # ---- self-check (before anything is timed) ----
    self_check = None
    if not args.no_selfcheck:
        loc, conf = model(dev_in, use_graph=True)
        torch.cuda.synchronize()
        outs = [t.clone() for t in list(loc) + list(conf)]
        self_check = [_self_check(name, sd, dev_in, outs, make_plain)]
        del outs
        if detect:
            ref = det.detect_device(dev_in, overlap=False)
            ref = torch.cat([ref[0][..., None], ref[1], ref[2][..., None]], -1).cpu()
            got = det.detect_host(host[0], slot=0, gather=False)
            det.join()
            torch.cuda.synchronize()
            if not torch.equal(got, ref):
                raise SystemExit("bench self-check FAILED: detect_host (overlapped) != detect_device (synchronous)")
            self_check.append("detect_host (side-stream overlap, pinned H2D/D2H) == synchronous detect_device, bit for bit; "
                              f"{int((ref[..., 0] > 0).sum())} detections in the batch")

    # ---- warm-up (also captures the CUDA graph) ----
    for i in range(W):
        step_device()
        step_host(i)
    join()
    barrier()

    # ---- value: device-resident inputs ----
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active = True
    e0.record()
    for _ in range(K):
        last = step_device()
    join()
    e1.record()
    barrier()
    sampler.active = False
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        names = ["scores", "boxes", "classes"] if detect else ["loss"]
        last = last if detect else (last,)
        dumped = {n: t.float().cpu().numpy() for n, t in zip(names, last)}
    del last

    # ---- e2e: pinned host batch -> H2D -> step -> D2H, every step ----
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.active = True
    f0.record()
    for i in range(K):
        out = step_host(i)
    join()
    f1.record()
    barrier()
    sampler.active = False
    e2e_ms = f0.elapsed_time(f1)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    d2h = out.numel() * 4

    # ---- per-group sections, each replayed alone K times (rooflines) ----
    sec = {}
    sec["conv"] = _timed(lambda: model.run_plan(plan, use_graph=True), K, barrier)
    loc, conf = plan["loc"], plan["conf"]
    scores_img = sum(cf.shape[1] * cf.shape[2] * cf.shape[3] for cf in conf)
    anchors_img = scores_img // C
    launches = plan["launches"]
    if not args.no_sections:
        if detect:
            pl = c["per_level"]
            items = list(anchors.items())
            sec["decode"] = _timed(lambda: decode_levels(conf, loc, items, 0.01, pl, True), K, barrier)
            dec = decode_levels(conf, loc, items, 0.01, pl, True)
            sec["nms"] = _timed(lambda: nms_op(*dec, 0.6, 100, True), K, barrier)
        else:
            from ssds_pytorch_b200.pipeline import fused_loss_step
            out3 = torch.empty(3, dtype=torch.float32, device=device)
            sec["loss"] = _timed(lambda: fused_loss_step(loc, conf, tg_dev, anchors, C, "MultiBoxLoss", None, out=out3),
                                 K, barrier)
    launches += 3 if detect else 1

    t = torch.tensor([dev_ms, e2e_ms] + [sec[k] for k in sorted(sec)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    vals = t.tolist()
    dev_ms, e2e_ms = vals[:2]
    sec = dict(zip(sorted(sec), vals[2:]))

    if rank == 0:
        tf_peak, hbm_peak, src = peaks()
        value = world * B * K / (dev_ms / 1e3)
        e2e = world * B * K / (e2e_ms / 1e3)

        def roof(group, bound, work, formula):
            ms = sec[group]
            if bound == "tensor":
                ach, peak, unit = work / (ms / 1e3) / 1e12, tf_peak, "TFLOP/s"
            else:
                ach, peak, unit = work / (ms / 1e3) / 1e9, hbm_peak, "GB/s"
            return {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                    "ms_per_step": ms, "work_per_step": work, "work": formula,
                    "peak_source": f"{src} " + ("bf16 sustained" if bound == "tensor" else "HBM copy")}

        rl = {"conv": roof("conv", c["bound"], flops_step if c["bound"] == "tensor" else conv_bytes,
                           "sum over convs of 2*Cin/g*k*k*Cout*Ho*Wo (un-padded FLOPs)" if c["bound"] == "tensor" else
                           "sum over conv launches of (input + output activation elems)*2 B + weights once "
                           "(un-fused algorithmic bytes, SURVEY 8d)")}
        if "decode" in sec:
            pl = c["per_level"]
            rl["decode"] = roof("decode", "hbm", B * (4 * scores_img + L * pl * 56), "B*(4*scores + L*K*56) bytes")
            rl["nms"] = roof("nms", "hbm", B * (24 * L * pl + 24 * 100), "B*(24*N + 24*D) bytes, N = L*K candidates "
                             "(latency/sort-bound at N <= 1800: the fraction is not a bandwidth claim there)")
        if "loss" in sec:
            rl["loss"] = roof("loss", "hbm", B * (4 * scores_img + 8 * anchors_img),
                              "B*(4*scores + 8*anchors) bytes: anchor match + MultiBoxLoss hard-negative mining + masks + "
                              "normalisation of ALL levels in ONE launch (loss_step_kernel); logits read once")
        traffic, tfile = measured_conv_traffic(name)
        main_rl = dict(rl[c["dominant"]])
        if n_fused:
            main_rl["fused_blocks"] = n_fused
            main_rl["floor_bytes_as_launched"] = conv_bytes_as_launched
            main_rl["floor_note"] = ("with the fused inverted residuals the expanded tensors never reach DRAM: the HBM floor "
                                     "of the plan as launched is floor_bytes_as_launched, not work_per_step")
        main_rl.update({"kernel": "conv_igemm_kernel + conv_pair_kernel + mbconv_kernel (+ dwconv3x3 etc.): all conv-stack launches of a step",
                        "traffic": traffic,
                        "traffic_unit": f"DRAM bytes per step over the conv launches (ncu, profiles/{tfile})" if tfile else None,
                        "flops_per_step": flops_step, "conv_ms_per_step": sec["conv"]})
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": c["workload"], "name": name, "global_batch": world * B, "per_gpu_batch": B,
                       "parallelism": f"dp{world} (batch sharded; " +
                                      ("NCCL all-gather of [B,100,6] detections)" if detect else
                                       "per-rank loss normalisation like the reference, no collective)"),
                       "l2_policy": "per-step working set of activations >> 126 MB L2; no flush needed"
                                    if B * H * Wd >= 4 << 20 else "inputs alternate between two host slots; activations "
                                    "of a step exceed the 126 MB L2",
                       "weights": "synthetic, reference init statistics, seed 0; BN folded"},
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K, "api": api},
            "gpu_launches": launches * K,
            "roofline": main_rl, "rooflines": rl, "self_check": self_check,
            "clocks": sampler.summary(),
        }
        if world == 1 and not args.no_cpu:
            _, line["cpu_baseline"] = cpu_baseline(name, args.cpu_images or c["cpu_images"], 1)
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (overrides the config)")
    ap.add_argument("--cpu-images", type=int, default=0, help="images in the CPU baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-selfcheck", action="store_true")
    ap.add_argument("--no-sections", action="store_true", help="skip the per-group roofline timings")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
