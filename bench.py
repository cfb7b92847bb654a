#!/usr/bin/env python
"""bench.py -- RGB-D 480x640 frames/s through the DGGM + E-DSAM hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs to DIR/*.npy

A "step" is one pass of the depth-guidance hot path (reference mask2former/utils/custom_model.py:324-355:
ratio predictor -> depth decomposition -> 3 DSAM stages -> DGGM injection + branch sum) over one batch of
synthetic NYUv2-shaped frames: workload = BASELINE.json configs[1] (batch 32 per GPU, 480x640, Swin-T
feature pyramid, bf16 tensor-core operands with fp32 accumulation).  The Swin backbone / pixel decoder stay
on stock PyTorch and are outside the step (SURVEY.md section 8).

Prints ONE JSON line (rank 0).  `value` = hot-path frames/s with inputs resident in HBM.  `e2e` = the WHOLE RGB-D
Mask2Former (reference predictor path, mask2former/predictor.py:19-36 + :697-703) fed from pinned HOST uint8 frames:
H2D -> device front-end -> stock Swin / pixel decoder / transformer under bf16 autocast with the CUDA hot path in
between (plus, by default, the two decoder_ops kernels inside the stock decoders; `e2e_stock_decoders` = the same loop
without them) -> device post-processing -> instance maps back in pinned host memory.  `e2e_hot_path_host_features` = the hot
path alone through the nn.Module API with host features (the PCIe-bound secondary of round 1).  `train` = BASELINE
configs[3] restricted to the hot path (fwd + bwd + NCCL gradient all-reduce, batch 8 per GPU).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import signal
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

H, W = 480, 640
CHANS = (96, 192, 384, 768)
STRIDES = (4, 8, 16, 32)
BATCH = 32
METRIC = "rgbd_480x640_frames_per_sec_depth_guidance_hot_path"
UNIT = "frames/s"

# algorithmic work per frame (SURVEY.md section 8d / DESIGN.md)
FLOP_CONV5 = 2.0 * H * W * 256 * 9 * 128                      # 181.19 GFLOP: 3x3 128->256 conv of the predictor
FLOP_DSAM = sum(5 * 2.0 * (H // (2 * s)) * (W // (2 * s)) * co * 9 * ci
                for s, ci, co in zip(STRIDES[:3], CHANS[:3], CHANS[1:]))      # 23.89 GFLOP
FEAT_ELEMS = sum(c * (H // s) * (W // s) for c, s in zip(CHANS, STRIDES))      # 3 456 000
BYTES_DGGM = 3 * 4 * FEAT_ELEMS + 4 * 4 * H * W               # read colour + branch-1, write fused, read grad+mask
POST_THRESHOLD = 0.0     # the reference's Evaluator(threshold=0.0) (finetuning.py:95): every candidate segment is painted
DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much in all


WORKLOAD = "configs[1]: batch-32/GPU inference, 480x640 RGB-D, Swin-T pyramid, depth-guidance hot path"
FORCED_RATIO = None
SWIN = "tiny"


def set_workload(name: str) -> None:
    """`configs1` (default, the metric's configuration) or `configs4` = BASELINE.json configs[4]: 960x1280 frames, Swin-B
    channels, window ratio forced to output_max (a builder-run record; the driver always runs the default)."""
    global H, W, CHANS, BATCH, FLOP_CONV5, FLOP_DSAM, FEAT_ELEMS, BYTES_DGGM, WORKLOAD, FORCED_RATIO, SWIN
    if name == "configs1":
        return
    assert name == "configs4", name
    H, W, CHANS, BATCH, SWIN = 960, 1280, (128, 256, 512, 1024), 8, "base"
    FORCED_RATIO = 0.5
    WORKLOAD = "configs[4]: 960x1280 RGB-D, Swin-B pyramid, E-DSAM window ratio forced to output_max (0.5), batch 8/GPU"
    FLOP_CONV5 = 2.0 * H * W * 256 * 9 * 128
    FLOP_DSAM = sum(5 * 2.0 * (H // (2 * s)) * (W // (2 * s)) * co * 9 * ci for s, ci, co in zip(STRIDES[:3], CHANS[:3], CHANS[1:]))
    FEAT_ELEMS = sum(c * (H // s) * (W // s) for c, s in zip(CHANS, STRIDES))
    BYTES_DGGM = 3 * 4 * FEAT_ELEMS + 4 * 4 * H * W


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


def make_frames(n: int, first: int = 0):
    """Synthetic frames (SURVEY section 8d): uint8 RGB + uint8 depth."""
    from rgbd_b200 import synthetic
    rgbs, depths = [], []
    for j in range(n):
        rgb, d = synthetic.synth_rgbd_u8(first + j, H, W, "nyu")
        rgbs.append(rgb)
        depths.append(d)
    return np.stack(rgbs), np.stack(depths)


def make_features(n: int, seed: int, device) -> list:
    g = torch.Generator(device="cpu").manual_seed(seed)
    return [torch.randn(n, c, H // s, W // s, generator=g).to(device) for c, s in zip(CHANS, STRIDES)]


def workload_config(batch: int) -> dict:
    """The ONE config both arms print (the reference arm runs bounded 1-frame samples of it; see cpu_baseline.sample)."""
    step_mb = batch * (10 * H * W + FEAT_ELEMS) * 4 / 1e6
    return {"workload": WORKLOAD, "batch_per_gpu": batch, "frame": [H, W], "channels": list(CHANS),
            "l2": f"per-step inputs ({step_mb:.0f} MB) exceed the 126 MB L2; no flush needed"}


def build_whole_model():
    """RGB-D Mask2Former (Swin-T, 100 queries, 80 labels) with random-init stock weights and the deterministic
    depth-guidance weights (rgbd_b200.synthetic_weights)."""
    from rgbd_b200 import synthetic_weights as SW
    return SW.build_synthetic_rgbd_mask2former(CHANS, guidance_seed=42, torch_seed=0, swin=SWIN)


# --------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU path on the host cores (oracle port; DESIGN.md section 2)
# --------------------------------------------------------------------------------------------------------
def _cpu_inputs():
    from oracle import hotpath as O
    from rgbd_b200 import synthetic
    rgb, depth = make_frames(1, first=0)
    pv = torch.from_numpy(synthetic.assemble_pixel_values(rgb[0], depth[0], O.gradient_features))[None]
    return pv, make_features(1, 7, "cpu")


def _time_cpu(fn, steps, warmup):
    with torch.no_grad():
        for _ in range(warmup):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        return (time.perf_counter() - t0) / steps


def cpu_hot_path(steps: int, warmup: int, threads=None):
    """BASELINE.md section 2 (ii)+(i): the whole hot path CM:324-355 on one 480x640 frame (oracle port, torch-CPU fp32)."""
    from oracle import hotpath as O
    from rgbd_b200 import synthetic_weights as SW
    cores = threads or (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    w = SW.guidance_weights(seed=42, channels=CHANS)
    pv, feats = _cpu_inputs()
    sec = _time_cpu(lambda: O.depth_guidance_forward(w, pv, feats), steps, warmup)
    return {"value": 1.0 / sec, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} steps x 1 frame 480x640 (oracle port of CM:324-355, torch-CPU fp32, {cores} threads)"}, sec


def cpu_modules(steps: int, threads=None):
    """BASELINE.md section 2 (i) DGGM alone and (ii) E-DSAM alone (ratio predictor + decomposition + 3 DSAM stages)."""
    from oracle import hotpath as O
    from rgbd_b200 import synthetic_weights as SW
    cores = threads or (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    w = SW.guidance_weights(seed=42, channels=CHANS)
    pv, feats = _cpu_inputs()
    dggm_w = O._sub(w, "depth_gradient_injection.")

    def edsam():
        ratios = O.ratio_predictor_forward(O._sub(w, "ratio_predictor."), pv[:, 3:6])
        gray = O.to_grayscale(pv[0, 3:6].numpy())
        x = feats[0]
        for k in range(3):
            x = feats[k + 1] + O.dsam_forward(O._sub(w, f"dsam{k}."), x, gray, ratios[0].item())
    t_dggm = _time_cpu(lambda: O.dggm_forward(dggm_w, feats, pv[:, 6:9], pv[:, 9:10]), max(steps, 3), 1)
    t_edsam = _time_cpu(edsam, steps, 1)
    return {"dggm_alone_frames_per_s": 1.0 / t_dggm, "edsam_alone_frames_per_s": 1.0 / t_edsam, "cores": cores}


def cpu_whole_model(steps: int, warmup: int, threads=None):
    """BASELINE.md section 2 (iii): whole v0.4.0 model forward + HF post_process_instance_segmentation on one frame."""
    from oracle import model as OM
    cores = threads or (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    model, w = build_whole_model()
    cpu_model = OM.cpu_oracle_model(model, w)
    pv, _ = _cpu_inputs()
    sec = _time_cpu(lambda: OM.predict(cpu_model, pv, threshold=POST_THRESHOLD, target_sizes=[(H, W)]), steps, warmup)
    return {"value": 1.0 / sec, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} steps x 1 frame 480x640: stock HF Swin-T/pixel decoder/transformer on CPU fp32 + oracle hot path "
                      f"+ HF post_process_instance_segmentation ({cores} threads)"}, sec


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(args.steps, 1), max(args.warmup, 1)
    base, sec_per_step = cpu_hot_path(steps, warmup)
    whole, whole_sec = cpu_whole_model(steps, min(warmup, 2))
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch),
        "cpu_baseline": base,
        # like with like: `value` is the hot path alone (compare with the own arm's `value`), `e2e` the whole model from
        # pixel_values to instance maps (compare with the own arm's `e2e`); nothing crosses a host<->device link here
        "e2e": {"value": whole["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "ms_per_step": whole_sec * 1e3, "sample": whole["sample"]},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------------------
# own arm
# --------------------------------------------------------------------------------------------------------
PR_SET_PDEATHSIG = 1     # prctl(2) option: signal this process when its parent ends


class ClockSampler:
    def __init__(self, index: int):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        prctl, parent = ctypes.CDLL(None, use_errno=True).prctl, os.getpid()

        def die_with_parent():                 # in the child, before exec: SIGKILL when bench.py ends, however it ends
            prctl(PR_SET_PDEATHSIG, signal.SIGKILL)
            if os.getppid() != parent:         # bench.py ended before the line above took effect
                os._exit(1)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                       "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL, preexec_fn=die_with_parent)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nme, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(local: int):
    """Pin this rank's host threads (and therefore its pinned staging buffers, first-touch) to the CPUs NVML reports as
    local to its GPU, so H2D/D2H copies do not cross the socket interconnect.  Best effort; returns the old mask."""
    try:
        import pynvml
        old = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * wi + b for wi, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= old
        if cpus:
            os.sched_setaffinity(0, cpus)
        return old
    except Exception:
        return None


def static_profile():
    """ncu-derived numbers that cannot be measured inside a plain run (tensor-pipe utilisation, DRAM traffic): loaded from
    the committed profiles/r02_ncu.json, which records the commit and batch size of its capture."""
    p = os.path.join(ROOT, "profiles", "r02_ncu.json")
    if os.path.exists(p):
        return json.load(open(p))
    return None


def run_own(args):
    import torch.distributed as dist
    import rgbd_b200  # noqa: F401
    from rgbd_b200 import functional as Fn, modules, parallel, serving, synthetic, synthetic_weights as SW

    rank, local, world = parallel.env_rank_world()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    old_affinity = bind_to_gpu_numa_node(local)
    if world > 1:
        parallel.init_process_group("nccl", dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    scaling = "weak"
    B = args.batch
    if args.frames_total:
        # BASELINE configs[2]: a fixed set of frames split over the ranks (256 frames -> 128/64/32 per GPU at 2/4/8 GPUs)
        b0, b1 = parallel.shard_range(args.frames_total, rank, world)
        B = b1 - b0
        scaling = "strong"
    frames_per_step = sum(parallel.gather_counts(B, dev))
    model = modules.DepthGuidance(CHANS)
    model.load_state_dict(SW.guidance_weights(seed=42, channels=CHANS))
    model.to(dev).eval()

    # ---- synthetic inputs: a few distinct frames tiled to the batch, built with the device front-end (K0)
    n_distinct = min(B, 8)
    rgb_u8, depth_u8 = make_frames(n_distinct, first=rank * 1000)
    idx = np.arange(B) % n_distinct
    rgb_host = torch.from_numpy(np.ascontiguousarray(rgb_u8[idx])).pin_memory()        # (B,H,W,3) uint8
    depth_host = torch.from_numpy(np.ascontiguousarray(depth_u8[idx])).pin_memory()    # (B,H,W)   uint8
    pv = Fn.pack_pixel_values(rgb_host.to(dev), depth_host.to(dev))
    feats = make_features(B, 7 + rank, dev)

    use_graph = args.graph        # measured: 6.89 vs 7.02 ms/step -- launch gaps are ~2 % of the step now
    if FORCED_RATIO is not None:
        # configs[4] "max window": the predictor still runs (its cost is part of the step), its output is replaced
        forced = torch.full((B, 1), FORCED_RATIO, device=dev)
        rp_forward = model.ratio_predictor.forward
        model.ratio_predictor.forward = lambda d, *a, **k: rp_forward(d, *a, **k) * 0 + forced
    if use_graph:
        try:
            graphed = modules.GraphedDepthGuidance(model, pv, feats)     # CUDA graph of the whole step (static shapes)
        except Exception as e:                                           # never lose the measurement to a capture problem
            print(f"[bench] CUDA graph capture failed ({e!r}); launching kernel by kernel", file=sys.stderr)
            use_graph = False
    if use_graph:
        def step():
            return graphed()
    else:
        def step():
            with torch.no_grad():
                return model(pv, feats)

    Fn.LAUNCHES = 0
    with torch.no_grad():
        model(pv, feats)                       # count this library's kernel launches of one step
    launches_per_step = Fn.LAUNCHES
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # ---- timed region: inputs resident in HBM; per-step inputs (835 MB) exceed the 126 MB L2
    sampler = ClockSampler(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        fused = step()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fused)
    launches = launches_per_step * args.steps          # kernels of this library executed inside the timed region
    elapsed = parallel.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
    value = frames_per_step * args.steps / elapsed

    # ---- single-frame latency of the hot path (BASELINE configs[0] shape on the GPU): batch 1, CUDA-graph replay
    latency = None
    try:
        pv1, feats1 = pv[:1].clone(), [f[:1].clone() for f in feats]
        g1 = modules.GraphedDepthGuidance(model, pv1, feats1)
        for _ in range(3):
            g1()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            g1()
        e1.record()
        torch.cuda.synchronize()
        latency = {"batch": 1, "ms_per_frame": e0.elapsed_time(e1) / args.steps, "steps": args.steps, "launch": "CUDA graph replay"}
        del g1
    except Exception as e:                                   # reported, never fatal
        latency = {"error": repr(e)}

    # ---- e2e (headline): the whole RGB-D Mask2Former from pinned host uint8 frames to instance maps in pinned host memory
    e2e = None
    e2e_stock = None

    def whole_model_e2e(fast_decoder_ops: bool):
        nonlocal launches
        whole, _ = build_whole_model()
        whole.to(dev)
        if FORCED_RATIO is not None:
            wrp = whole.model.pixel_level_module.ratio_predictor
            wrp_forward = wrp.forward
            wrp.forward = lambda d, *a, **k: wrp_forward(d, *a, **k) * 0 + forced
        seg = serving.RgbdInstanceSegmenter(whole, B, (H, W), threshold=POST_THRESHOLD, fast_decoder_ops=fast_decoder_ops)
        for b in range(2):
            seg.in_host[b][0].copy_(rgb_host)
            seg.in_host[b][1].copy_(depth_host)
        Fn.LAUNCHES = 0
        seg.submit()
        whole_launches_per_step = Fn.LAUNCHES
        for _ in range(max(args.warmup, 3) - 1):
            seg.submit()
        seg.warmup()                                          # graph capture (one per staging buffer) belongs to the warm-up
        seg.drain()
        barrier()
        e0.record()
        for _ in range(args.steps):
            seg.submit()
        seg.drain()
        e1.record()
        barrier()
        whole_elapsed = parallel.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
        last = seg.out_host[(args.steps - 1) & 1]
        counts = last["count"].clone()
        kept = {k: last[k].clone() for k in ("labels", "segmentation")}
        # stage breakdown of one un-pipelined step (CUDA events around the stock sub-modules; reported, not the metric)
        marks = {}

        def timed(mod, name):
            def pre(m, a, k=None):
                marks[name] = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
                marks[name][0].record()

            def post(m, a, o):
                marks[name][1].record()
            return [mod.register_forward_pre_hook(pre), mod.register_forward_hook(post)]
        plm = whole.model.pixel_level_module
        graph_was, seg.cuda_graph = seg.cuda_graph, False      # the breakdown needs the modules' Python forwards (hooks): eager step
        hooks = timed(plm.encoder, "swin_encoder") + timed(plm.decoder, "pixel_decoder") + \
            timed(whole.model.transformer_module, "transformer_decoder") + timed(plm, "pixel_level_module")
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        seg.submit()
        seg.drain()
        t1.record()
        torch.cuda.synchronize()
        for h_ in hooks:
            h_.remove()
        seg.cuda_graph = graph_was
        br = {k: v[0].elapsed_time(v[1]) for k, v in marks.items()}
        br["hot_path_incl_float_casts"] = br["pixel_level_module"] - br["swin_encoder"] - br["pixel_decoder"]
        br["step_unpipelined"] = t0.elapsed_time(t1)
        br["note"] = "one EAGER step (module hooks need the Python forwards); the timed loop replays CUDA graphs" if graph_was else "eager"
        # the pipelined loop produced the real thing: its last result equals a synchronous call on the same frames (reported,
        # not asserted; the stock model's kernels are not guaranteed to be bit-reproducible)
        sync_res = seg.out_host[(seg._step - 1) & 1]
        e2e_check = {"same_instance_counts_as_synchronous_call": bool(torch.equal(sync_res["count"], counts)),
                     "same_labels": bool(torch.equal(sync_res["labels"], kept["labels"])),
                     "segmentation_pixels_equal_frac": float((sync_res["segmentation"] == kept["segmentation"]).float().mean())}
        hot_ms = elapsed / args.steps * 1e3
        e2e = {"value": frames_per_step * args.steps / whole_elapsed, "unit": UNIT,
               "h2d_bytes_per_step": seg.h2d_bytes_per_step, "d2h_bytes_per_step": seg.d2h_bytes_per_step,
               "ms_per_step": whole_elapsed / args.steps * 1e3,
               "how": "rgbd_b200.serving.RgbdInstanceSegmenter: pinned-host uint8 colour + depth frames -> H2D -> "
                      "rgbd_pack_pixel_values -> Mask2FormerForUniversalSegmentation (stock HF Swin-T / pixel decoder / "
                      "transformer decoder modules and weights, bf16 autocast, random-init) with the CUDA depth-guidance hot "
                      "path" + (" and the decoder_ops kernels inside the stock modules (rgbd_window_attention + bf16 pre-norm rgbd_layer_norm "
                                "in Swin, rgbd_msda_fwd in the pixel decoder's 6 deformable-attention layers, rgbd_attention_mask in "
                                "the 10 mask-predictor calls, rgbd_masked_cross_attention in the 9 decoder layers, rgbd_layer_norm for "
                                "every other LayerNorm)" if fast_decoder_ops else "") +
                      ("; the device part of a step is replayed as one CUDA graph" if seg.cuda_graph else "") +
                      " -> device "
                      "post_process_instance_segmentation (threshold 0.0, target 480x640) -> segmentation map + labels + "
                      "scores + counts to pinned host; H2D / compute / D2H on 3 streams, 2 buffers",
               "own_kernel_launches_per_step": whole_launches_per_step,
               "launch": "one CUDA graph replay per batch (front-end + model + post-processing)" if seg.cuda_graph else "eager",
               "hot_path_ms_per_step": hot_ms, "hot_path_share_of_step": hot_ms / (whole_elapsed / args.steps * 1e3),
               "breakdown_ms": br, "segments_last_step": int(counts.sum()), "check": e2e_check}
        if fast_decoder_ops:
            launches += whole_launches_per_step * args.steps
        del seg, whole
        torch.cuda.empty_cache()
        return e2e

    if not args.no_whole_model:
        e2e = whole_model_e2e(True)
        # the same loop with the stock decoders untouched (HF grid_sample-based deformable attention, ATen attention masks)
        e2e_stock = whole_model_e2e(False)
        e2e_stock = {k: e2e_stock[k] for k in ("value", "unit", "ms_per_step", "own_kernel_launches_per_step", "breakdown_ms")}
        e2e_stock["how"] = "same pipeline with decoder_ops disabled: every kernel outside the depth-guidance hot path is stock PyTorch/cuDNN"

    # ---- secondary e2e: the hot path ALONE through the nn.Module API with host-resident encoder features (what round 1
    # reported as e2e).  Every step ships uint8 frames + fp32 features in and the fp32 fused features out, so it is bound by
    # the host link, not by the path; in the real model those features never leave the GPU.
    hp = hot_path_host_features(args, model, B, rgb_host, depth_host, feats, pv, dev, barrier, world, frames_per_step)
    clocks = sampler.stop()          # sampled over the device-resident and the e2e timed regions

    # ---- per-kernel timing for the roofline (separate, after the headline measurement; CUDA events on the
    # launching stream around each stage of the same step)
    pk = PerKernel(model, pv, feats, args.steps)
    kt = pk.measure()
    pkv = peaks()
    sp = static_profile()
    conv5_tf = FLOP_CONV5 * B / kt["ratio_conv3x3"] / 1e12
    dggm_gbs = BYTES_DGGM * B / kt["dggm"] / 1e9
    dsam_tf = FLOP_DSAM * B / kt["dsam_gemm"] / 1e12
    traffic = None
    if sp and sp.get("batch") == B:
        traffic = sp.get("dram_bytes_per_launch", {}).get("conv3x3_2cta_kernel")
    roof = {"kernel": "conv3x3_2cta_kernel (ratio predictor 3x3 128->256 conv + BN + ReLU + AdaptiveAvgPool2d(4), CTA pairs)", "bound": "tensor",
            "achieved": conv5_tf, "peak": pkv["tf_burst"], "unit": "TFLOP/s", "frac": conv5_tf / pkv["tf_burst"],
            "frac_of_sustained": conv5_tf / pkv["tf_sustained"],
            "frac_of_nominal_dense_bf16": conv5_tf / 2250.0,      # frac can pass 1.0: the peak is what cuBLAS reaches here
            "traffic": traffic,
            "traffic_source": (f"static: {sp['source']} @ {sp['commit']} (batch {sp['batch']})" if traffic is not None else None),
            "peak_source": pkv["source"] + " burst bf16 cuBLAS (the kernel is timed alone, back to back)"}
    extra = [
        {"kernel": "dggm_fwd_kernel (DGGM + branch sum)", "bound": "hbm", "achieved": dggm_gbs, "peak": pkv["hbm_gbs"],
         "unit": "GB/s", "frac": dggm_gbs / pkv["hbm_gbs"], "bytes_per_frame": BYTES_DGGM},
        {"kernel": "3 DSAM stages (useful FLOPs: K padding not counted)",
         "bound": "tensor", "achieved": dsam_tf, "peak": pkv["tf_burst"], "unit": "TFLOP/s", "frac": dsam_tf / pkv["tf_burst"]},
    ]
    if "ratio_front" in kt:
        compact = model.ratio_predictor._compact(H, W)
        # stem GEMM (K = 147 useful taps of 256) + 192->128 + 128->64 + 64->128 point-wise layers
        front_tf = 2.0 * (147 * 192 + 192 * 128 + 128 * 64 + 64 * 128) * H * W * B / kt["ratio_front"] / 1e12
        front_gbs = ((16 if compact else 128) + 256) * H * W * B / kt["ratio_front"] / 1e9
        extra.append({"kernel": "ratio_front_kernel (stem + feature fusion + attention, one kernel)", "bound": "tensor",
                      "achieved": front_tf, "peak": pkv["tf_burst"], "unit": "TFLOP/s", "frac": front_tf / pkv["tf_burst"],
                      "hbm_gbs": front_gbs})

    # ---- the decoder_ops kernels at this workload's shapes (live CUDA-event timings; reported, never part of `value`)
    if not args.no_whole_model:
        try:
            extra.extend(decoder_ops_rooflines(B, pkv, dev, args.steps))
        except Exception as e:                               # reported, never fatal for the headline line
            extra.append({"kernel": "decoder_ops kernels", "error": repr(e)})

    # ---- BASELINE configs[3] on the hot path: fwd + bwd + gradient all-reduce, batch 8 per GPU
    train = None
    if not args.no_train:
        del model
        if use_graph:
            del graphed
        torch.cuda.empty_cache()
        train = train_record(args, dev, rank, world, barrier)
        if not args.no_whole_model:
            try:
                train["whole_model"] = train_whole_model_record(args, dev, rank, world, barrier)
            except Exception as e:                           # reported, never fatal for the headline line
                train["whole_model"] = {"error": repr(e)}

    if rank == 0:
        if old_affinity:
            os.sched_setaffinity(0, old_affinity)          # the CPU baseline uses every host core
        cpu_base, _ = cpu_hot_path(args.cpu_steps, 1)
        if not args.no_cpu_detail:
            one, _ = cpu_hot_path(1, 0, threads=1)
            wm, _ = cpu_whole_model(max(1, min(args.cpu_steps, 3)), 1)
            cpu_base["detail"] = {"hot_path_1_thread_frames_per_s": one["value"], **cpu_modules(max(1, min(args.cpu_steps, 3))),
                                  "whole_model_plus_postprocess_frames_per_s": wm["value"], "whole_model_sample": wm["sample"]}
        cfg = workload_config(B)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": cfg,
            "launch": "CUDA graph replay of the hot-path step" if use_graph else "kernel-by-kernel launches",
            "e2e": e2e if e2e is not None else hp,
            "e2e_stock_decoders": e2e_stock,
            "e2e_hot_path_host_features": hp,
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
            "roofline_extra": extra,
            # E-DSAM tensor-core utilisation (BASELINE metric): sm__pipe_tensor_cycles_active from a committed `ncu --set full`
            # capture -- static, never measured under this run; the file records its commit and batch
            "tc_util_pct_ncu": ({"source": f"static: {sp['source']} @ {sp['commit']} (batch {sp['batch']})", **sp["tc_util_pct"]}
                                if sp else None),
            "kernel_ms_per_step": {k: v * 1e3 for k, v in kt.items()},
            "latency_batch1": latency,
            "train": train,
            "cpu_baseline": cpu_base,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, fused) -> None:
    """--dump-outputs: what the last timed step returned -- the four fused feature maps handed to the pixel decoder -- as
    float32 ``fused<i>.npy``.  A map larger than its share of DUMP_BYTES is stored as a fixed sample of its elements (flat
    indices drawn from a generator seeded with ``i``, in increasing order), so runs with the same arguments store the same
    elements."""
    os.makedirs(out_dir, exist_ok=True)
    per_map = (DUMP_BYTES // len(fused) - 128) // 4          # elements; 128 bytes of .npy header
    for i, t in enumerate(fused):
        t = t.detach()
        if t.numel() > per_map:
            idx = np.sort(np.random.default_rng(i).choice(t.numel(), per_map, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"fused{i}.npy"), t.float().cpu().numpy())


def hot_path_host_features(args, model, B, rgb_host, depth_host, feats, pv, dev, barrier, world, frames_per_step):
    """Round 1's e2e loop, kept as a labelled secondary: pinned-host uint8 frames + fp32 encoder features in, fp32 fused
    features out, one slab per direction, H2D / compute / D2H on 3 streams with 2 buffers."""
    from rgbd_b200 import functional as Fn, parallel
    feats_host = [f.cpu().pin_memory() for f in feats]
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    s_main = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def carve(slab, shapes_dtypes):
        views, off = [], 0
        for shape, dt in shapes_dtypes:
            n = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
            off = (off + 255) // 256 * 256
            views.append(slab[off:off + n].view(dt).view(shape))
            off += n
        return views

    def slab_bytes(shapes_dtypes):
        off = 0
        for shape, dt in shapes_dtypes:
            off = (off + 255) // 256 * 256 + int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        return off

    feat_specs = [(tuple(f.shape), torch.float32) for f in feats_host]
    specs = [((B, H, W, 3), torch.uint8), ((B, H, W), torch.uint8)] + feat_specs
    in_host = torch.empty(slab_bytes(specs), dtype=torch.uint8).pin_memory()
    for v, src in zip(carve(in_host, specs), [rgb_host, depth_host] + feats_host):
        v.copy_(src)
    in_dev = []
    for _ in range(2):
        ds = torch.empty(in_host.numel(), dtype=torch.uint8, device=dev)
        in_dev.append((ds, carve(ds, specs)))
    pv_buf = [torch.empty_like(pv), torch.empty_like(pv)]
    out_dev, out_host = [], []
    for _ in range(2):
        ds = torch.empty(slab_bytes(feat_specs), dtype=torch.uint8, device=dev)
        out_dev.append((ds, carve(ds, feat_specs)))
        out_host.append(torch.empty(ds.numel(), dtype=torch.uint8).pin_memory())

    def run(n_steps):
        ev_in, ev_free, ev_d2h = [None, None], [None, None], [None, None]
        for i in range(n_steps):
            b = i & 1
            slab, views = in_dev[b]
            with torch.cuda.stream(s_in):
                if ev_free[b] is not None:
                    s_in.wait_event(ev_free[b])
                slab.copy_(in_host, non_blocking=True)
                ev_in[b] = s_in.record_event()
            s_main.wait_event(ev_in[b])
            if ev_d2h[b] is not None:
                s_main.wait_event(ev_d2h[b])               # output buffer b is free again
            with torch.no_grad():
                Fn.pack_pixel_values(views[0], views[1], out=pv_buf[b])
                model(pv_buf[b], views[2:], out=out_dev[b][1])
            ev_free[b] = s_main.record_event()
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_free[b])
                out_host[b].copy_(out_dev[b][0], non_blocking=True)
                ev_d2h[b] = s_out.record_event()
        for e in ev_d2h:
            if e is not None:
                s_main.wait_event(e)

    run(4)
    times = []
    for _ in range(2):                  # PCIe on these shared hosts is noisy: best of two runs of K steps each
        barrier()
        e0.record()
        run(args.steps)
        e1.record()
        barrier()
        times.append(parallel.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev))
    torch.cuda.synchronize()
    with torch.no_grad():
        want = model(pv, feats)
    got = carve(out_host[(args.steps - 1) & 1], feat_specs)
    check = {"bit_identical_to_device_resident_step": all(torch.equal(g_, w_.cpu()) for g_, w_ in zip(got, want))}
    return {"value": frames_per_step * args.steps / min(times), "unit": UNIT, "h2d_bytes_per_step": in_host.numel(),
            "d2h_bytes_per_step": out_host[0].numel(), "runs_s": times, "check": check,
            "how": "hot path only: pinned-host uint8 frames + fp32 encoder features -> rgbd_pack_pixel_values -> "
                   "DepthGuidance.forward -> fp32 fused features to pinned host (host-link bound; secondary)"}


def train_record(args, dev, rank, world, barrier):
    """BASELINE configs[3] restricted to the hot path (reference: HF Trainer step under finetuning.py:98-113): one
    fine-tuning step of the depth-guidance modules in .train() mode -- ratio predictor with batch-statistics BatchNorm and
    Dropout (no gradient: CM:339), DSAM wgrad / dgrad / dbias, DGGM dW / db -- at batch 8 per GPU; gradients are
    all-reduced over NCCL bucket by bucket while the backward of the earlier stages is still running."""
    from rgbd_b200 import functional as Fn, modules, parallel, synthetic_weights as SW
    B = 8
    model = modules.DepthGuidance(CHANS)
    model.load_state_dict(SW.guidance_weights(seed=42, channels=CHANS))
    model.to(dev).train()
    rgb_u8, depth_u8 = make_frames(B, first=rank * 1000)
    pv = Fn.pack_pixel_values(torch.from_numpy(rgb_u8).to(dev), torch.from_numpy(depth_u8).to(dev))
    feats = make_features(B, 7 + rank, dev)
    douts = [torch.randn_like(f) for f in feats]
    for p in model.ratio_predictor.parameters():
        p.requires_grad_(False)                            # CM:339: consumed through .item(), never receives a gradient
    buckets = [list(model.dsam2.parameters()), list(model.dsam1.parameters()),
               list(model.dsam0.parameters()) + list(model.depth_gradient_injection.parameters())]
    reducer = parallel.GradBucketReducer(buckets)

    def step():
        for b in buckets:
            for p in b:
                p.grad = None
        out = model(pv, feats)
        torch.autograd.backward(out, douts)
        reducer.finish()

    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for _ in range(3):
            step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
    t = parallel.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
    reducer.remove()
    return {"metric": "rgbd_480x640_train_frames_per_sec_depth_guidance_hot_path", "value": world * B * args.steps / t,
            "unit": UNIT, "ms_per_step": t / args.steps * 1e3, "batch_per_gpu": B, "n_gpus": world,
            "grad_elements_allreduced_per_step": reducer.n_elements if world > 1 else 0,
            "buckets": [sum(p.numel() for p in b) for b in buckets],
            "ratio_predictor_mode": "train (batch-statistics BatchNorm, Dropout)" if getattr(
                model.ratio_predictor, "TRAIN_MODE_SUPPORTED", False) else "eval semantics",
            "workload": "configs[3] hot-path share: fwd+bwd of ratio predictor (fwd) + DSAM x3 + DGGM, NCCL bucketed "
                        "gradient all-reduce overlapped with the backward"}


def train_whole_model_record(args, dev, rank, world, barrier):
    """BASELINE configs[3] as finetuning.py runs it (mask2former/finetuning.py:98-113, HF Trainer step): the WHOLE RGB-D
    Mask2Former in .train() mode under bf16 autocast, batch 8 per GPU, synthetic rectangle labels (<= 20 per frame, 48 classes)
    -> transformers' Mask2FormerLoss (Hungarian matching on the host, as in the reference) -> backward (stock autograd + this
    library's DSAM / DGGM backward kernels; the encoder and the ratio predictor receive no gradient, CM:332-339) -> bucketed NCCL
    all-reduce overlapped with the backward -> AdamW.  The stock modules run their stock forward / backward here (decoder_ops
    are inference kernels)."""
    import numpy as np
    from rgbd_b200 import functional as Fn, parallel
    B = 8
    model, _ = build_whole_model()
    model.to(dev).train()
    plm = model.model.pixel_level_module
    for p in (*plm.encoder.parameters(), *plm.ratio_predictor.parameters()):
        p.requires_grad_(False)
    rgb_u8, depth_u8 = make_frames(B, first=rank * 1000)
    pv = Fn.pack_pixel_values(torch.from_numpy(rgb_u8).to(dev), torch.from_numpy(depth_u8).to(dev))
    rs = np.random.RandomState(100 + rank)
    mask_labels, class_labels = [], []
    for _ in range(B):
        k = rs.randint(3, 21)
        m = torch.zeros(k, H, W)
        for j in range(k):
            h, w = rs.randint(H // 16, H // 2), rs.randint(W // 16, W // 2)
            y, x = rs.randint(0, H - h), rs.randint(0, W - w)
            m[j, y:y + h, x:x + w] = 1
        mask_labels.append(m.to(dev))
        class_labels.append(torch.from_numpy(rs.randint(0, 48, size=k)).to(dev))
    hot = set(id(p) for m_ in (plm.dsam0, plm.dsam1, plm.dsam2, plm.depth_gradient_injection) for p in m_.parameters())
    dec = [p for p in plm.decoder.parameters() if p.requires_grad]
    rest = [p for p in model.parameters() if p.requires_grad and id(p) not in hot and id(p) not in set(id(q) for q in dec)]
    buckets = [rest, dec, list(plm.dsam2.parameters()), list(plm.dsam1.parameters()),
               list(plm.dsam0.parameters()) + list(plm.depth_gradient_injection.parameters())]       # backward order
    reducer = parallel.GradBucketReducer(buckets)
    opt = torch.optim.AdamW([p for b in buckets for p in b], lr=1e-5)
    phases = []

    def step(timed=False):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timed else None
        if timed:
            ev[0].record()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model(pixel_values=pv, mask_labels=mask_labels, class_labels=class_labels)
        if timed:
            ev[1].record()
        out.loss.backward()
        reducer.finish()
        if timed:
            ev[2].record()
        opt.step()
        opt.zero_grad(set_to_none=True)
        if timed:
            ev[3].record()
            phases.append(ev)
        return out.loss

    import warnings
    steps = args.steps
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for _ in range(2):
            step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = step(timed=True)
        e1.record()
        barrier()
    t = parallel.max_over_ranks(e0.elapsed_time(e1) / 1e3, dev)
    ph = [[e[i].elapsed_time(e[i + 1]) for i in range(3)] for e in phases]
    med = [sorted(c)[len(c) // 2] for c in zip(*ph)]
    reducer.remove()
    grads = {"encoder_params_trainable": 0, "ratio_predictor_params_trainable": 0,
             "trainable_elements": reducer.n_elements}
    del model, opt
    torch.cuda.empty_cache()
    return {"metric": "rgbd_480x640_train_frames_per_sec_whole_model", "value": world * B * steps / t, "unit": UNIT,
            "ms_per_step": t / steps * 1e3, "steps": steps, "batch_per_gpu": B, "n_gpus": world,
            "phase_ms_median": {"forward_and_loss": med[0], "backward_and_allreduce": med[1], "adamw": med[2]},
            "grad_elements_allreduced_per_step": reducer.n_elements if world > 1 else 0, "final_loss": float(loss.detach()),
            **grads,
            "workload": "configs[3]: whole RGB-D Mask2Former fine-tuning step, bf16 autocast, batch 8 per GPU, synthetic rectangle "
                        "labels, HF Mask2FormerLoss, bucketed NCCL gradient all-reduce overlapped with the backward, AdamW"}


def decoder_ops_rooflines(B, pkv, dev, steps):
    """Live timings of the decoder_ops kernels that carry most bytes, at the shapes the whole model gives them for this workload
    (deformable attention of the pixel decoder's three coarse levels; LayerNorm of the pixel decoder's token stream)."""
    from rgbd_b200 import functional as Fn
    g = torch.Generator(device=dev).manual_seed(3)
    sp = [(H // 32, W // 32), (H // 16, W // 16), (H // 8, W // 8)]
    S = sum(a * b for a, b in sp)
    value = torch.randn(B, S, 8, 32, device=dev, generator=g).bfloat16()
    offs = (torch.randn(B, S, 8, 3, 4, 2, device=dev, generator=g) * 2.0).bfloat16()
    logit = torch.randn(B, S, 8, 12, device=dev, generator=g).bfloat16()
    ref = torch.rand(B, S, 3, 2, device=dev, generator=g)
    x = torch.randn(B * S, 256, device=dev, generator=g)
    w, b = torch.ones(256, device=dev), torch.zeros(256, device=dev)

    def timed(fn, n=steps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n / 1e3
    t_msda = timed(lambda: Fn.msda_forward(value, sp, offs, logit, reference_points=ref, softmax=True, out_dtype=torch.bfloat16))
    t_ln = timed(lambda: Fn.layer_norm(x, w, b, 1e-5))
    gathered = B * S * 8 * 12 * 4 * 64                       # bytes: (query, head, level x point, corner) x 32 bf16 channels
    hbm_msda = (value.numel() + offs.numel() + logit.numel() + B * S * 256) * 2 + ref.numel() * 4
    l2_peak = 43.0 * 148 * 1.965                              # GB/s: ~43 B/clk/SM delivered from L2 (profiles/r02_mma_rate.txt)
    return [
        {"kernel": "msda_fwd_quad_kernel (pixel decoder deformable attention: softmax + locations + bilinear gather)",
         "bound": "l2-gather", "achieved": gathered / t_msda / 1e9, "peak": l2_peak, "unit": "GB/s",
         "frac": gathered / t_msda / 1e9 / l2_peak, "us": t_msda * 1e6, "algorithmic_hbm_gbs": hbm_msda / t_msda / 1e9,
         "peak_source": "L2 -> SM delivery measured with bulk copies (43 B/clk/SM x 148 SMs x 1.965 GHz)"},
        {"kernel": "layer_norm_kernel (float32 in / out, (batch x 6300, 256))", "bound": "hbm", "achieved": x.numel() * 8 / t_ln / 1e9,
         "peak": pkv["hbm_gbs"], "unit": "GB/s", "frac": x.numel() * 8 / t_ln / 1e9 / pkv["hbm_gbs"], "us": t_ln * 1e6},
    ]


class PerKernel:
    """Times the stages of one hot-path step separately with CUDA events (same inputs, same stream)."""

    def __init__(self, model, pv, feats, steps):
        self.m, self.pv, self.feats, self.steps = model, pv, feats, steps

    def _time(self, fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(self.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / self.steps

    def measure(self):
        from rgbd_b200 import functional as Fn
        from rgbd_b200.modules import _best_box
        m, pv, feats = self.m, self.pv, self.feats
        B = pv.shape[0]
        rp = m.ratio_predictor
        out = {}
        with torch.no_grad():
            out["ratio_predictor_total"] = self._time(lambda: rp(pv[:, 3:6]))
            pk, ws = rp._refresh(), rp._workspace(B, H, W, pv.device)
            box = _best_box(H, W)
            out["ratio_conv3x3"] = self._time(lambda: Fn.conv_gemm(
                ws["x4"], (B, H, W, 128), 1, pk["w5"], pk["sl5"], 64, B, (H, W), box, 256, pk["sh5"],
                act=1, epi_mode=2, pool=ws["pool"], cells=(4, 4), tile_order=1, conv3x3_reuse=(box == (128, 1))))
            compact = rp._compact(H, W)
            if rp.use_fused_front:
                out["ratio_front"] = self._time(lambda: Fn.ratio_front(
                    ws["stem"], pk["w1c"] if compact else pk["w1"], pk["w2"], pk["w3"], pk["w4"], pk["sh1"], pk["sh2"], pk["sh3"],
                    pk["sh4"], ws["x4"], box))
            out["ratio_stem_pack"] = self._time(lambda: (Fn.ratio_stem_pack_compact if compact else Fn.ratio_stem_pack)(
                pv[:, 3:6], ws["stem"]))
            fcw, fcb = [pk[f"fw{j}"] for j in range(4)], [pk[f"fb{j}"] for j in range(4)]
            if rp.use_tensor_core_tail:
                out["ratio_tail"] = self._time(lambda: Fn.ratio_tail_tc(
                    ws["pool"], (H // 4) * (W // 4), ws["a6"], ws["gap_fx"], pk["w6_bf"], pk["sl6"], pk["sh6"], fcw, fcb,
                    rp.output_min, rp.output_max))
            else:
                out["ratio_tail"] = self._time(lambda: Fn.ratio_tail(
                    ws["pool"], (H // 4) * (W // 4), pk["w6"], pk["sc6"], pk["sh6"], fcw, fcb, rp.output_min, rp.output_max))
            ratios = rp(pv[:, 3:6])
            levels = [tuple(f.shape[2:]) for f in feats[:3]]
            out["depth_decompose"] = self._time(lambda: Fn.depth_decompose(ratios.reshape(-1), levels, depth3=pv[:, 3:6],
                                                                           want_codes=False))
            dec = Fn.depth_decompose(ratios.reshape(-1), levels, depth3=pv[:, 3:6])

            from rgbd_b200.modules import dsam_cascade
            dsams = (m.dsam0, m.dsam1, m.dsam2)
            # the cascade exactly as the step runs it: one pack kernel (stage 0), stages 1-2 get their operand from the
            # previous stage's epilogue
            out["dsam_cascade_total"] = self._time(lambda: dsam_cascade(dsams, feats, dec, False))
            # GEMM-only time of the three stages (operands already packed by the cascade above)
            def gemms():
                x = feats[0]
                for k, d in enumerate((m.dsam0, m.dsam1, m.dsam2)):
                    d._gemm_only = True
                    x = d.stage_forward(x, dec.pooled[k], dec.bias_variant, residual=feats[k + 1])
                    d._gemm_only = False
            out["dsam_gemm"] = self._time(gemms)
            cp1 = [f.clone() for f in feats]
            out["dggm"] = self._time(lambda: m.depth_gradient_injection.forward_fused_sum(feats, cp1, pv[:, 6:9], pv[:, 9:10]))
        return out


_REAL_STDOUT = None


def _quiet_stdout():
    """Libraries (NCCL's version banner, HF warnings) write to fd 1; the driver wants ONE JSON line there.
    Point fd 1 at stderr for the run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU and step (default: 32, or 8 for --workload configs4)")
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--workload", default="configs1", choices=["configs1", "configs4"],
                    help="configs4 = BASELINE.json configs[4] (960x1280, Swin-B, ratio forced to 0.5, batch 8/GPU): builder-run record")
    ap.add_argument("--frames-total", type=int, default=0,
                    help="BASELINE configs[2]: split this many frames over the ranks (strong scaling) instead of --batch per GPU")
    ap.add_argument("--no-whole-model", action="store_true", help="skip the whole-model e2e leg (e2e falls back to the hot-path loop)")
    ap.add_argument("--no-train", action="store_true", help="skip the configs[3] train sub-record")
    ap.add_argument("--no-cpu-detail", action="store_true", help="cpu_baseline: only the all-core hot-path figure")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch the ~22 kernels of a step one by one instead of replaying the step as one CUDA graph")
    ap.set_defaults(graph=True)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the fused feature maps of the last one as DIR/fused<i>.npy (float32; "
                         "rank 0; a seeded sample of each map's elements where all of them would pass 64 MB in total)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs writes the outputs of this repo's CUDA path (--impl own)")
    set_workload(args.workload)
    args.batch = args.batch or BATCH
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
