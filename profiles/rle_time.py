"""Cost of the run-length (COCO) output of the instance post-processing.

    python profiles/rle_time.py --out DIR      # writes DIR/r03_rle.json and prints it

1. ``encoder``: the four kernels of ``functional.label_map_rle`` (count, scan, base, emit) captured in one CUDA graph and
   replayed back to back, timed with CUDA events, on 32 painted 480x640 maps from model-sized outputs
   (``synth_outputs(seed, 32, 100, 48, 120, 160)``, threshold 0) and on a worst-case checkerboard (one run per pixel).
   Algorithmic bytes: the map read twice (count and emit passes) plus 8 bytes per run written; the 39 MB batch of maps fits
   in the 126 MB L2, so after the first replay it is read from there, and the HBM figure is a bound, not what was reached.
2. ``post_process``: wall time of ``post_process_instance_segmentation(return_coco_annotation=True)`` per 32 frames, beside
   the same call with the flag off and beside HF's ``convert_segmentation_to_rle`` of the same 32 maps on this host's CPU.
3. ``serving``: ``RgbdInstanceSegmenter`` (bench.py's whole model, batch 32, 480x640, CUDA graphs) with the flag off and on,
   alternated round by round in one process; every step's ``result`` is read, as a user would.  Also the host time
   spent inside ``result`` once the step's download has finished and ``d2h_bytes_per_step`` after each ``result`` (the tables plus, with the flag on, the
   runs that ``result`` copied).
``kernel_us_torch_profiler``: each encoder kernel's device time from torch.profiler, in a run of its own.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import re
import subprocess
import sys
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HBM_GBS = 7700.0      # HGX B200 data sheet, one GPU, at up to 1000 W


def card():
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def time_graph(fn, reps):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def kernel_us(Fn, seg, L, reps):
    """Device time of each encoder kernel from torch.profiler (a run of its own, after the graph timing)."""
    from torch.profiler import ProfilerActivity, profile
    out = Fn.label_map_rle_buffers(*seg.shape, L, seg.device)
    Fn.label_map_rle(seg, L, *out)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            Fn.label_map_rle(seg, L, *out)
        torch.cuda.synchronize()
    names = ((re.search(r"rle_\w+_kernel", e.key), e) for e in prof.key_averages())
    return {m.group(0): e.device_time_total / e.count for m, e in names if m}


def encoder(Fn, seg, L, reps):
    ms, out = time_graph(lambda: Fn.label_map_rle(seg, L), reps)
    runs = int(out.base[-1])
    nbytes = 2 * seg.numel() * 4 + 8 * runs
    return {"shape": list(seg.shape), "labels": L, "runs": runs, "us_per_batch": ms * 1e3,
            "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / (ms * 1e-3) / 1e9,
            "frac_of_hbm_datasheet": nbytes / (ms * 1e-3) / 1e9 / HBM_GBS,
            "kernel_us_torch_profiler": kernel_us(Fn, seg, L, 50)}


def post_process(PP, outs, sizes, reps):
    res = {}
    for name, kw in (("off", {}), ("coco", {"return_coco_annotation": True})):
        PP.post_process_instance_segmentation(outs, threshold=0.0, target_sizes=sizes, **kw)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = PP.post_process_instance_segmentation(outs, threshold=0.0, target_sizes=sizes, **kw)
            if name == "off":
                [x["segmentation"].cpu() for x in r]       # the maps on the host, like the coco lists
        torch.cuda.synchronize()
        res[f"ms_per_32_frames_{name}"] = (time.perf_counter() - t0) / reps * 1e3 * 32 / len(sizes)
    return res


def hf_host(maps):
    from transformers.models.mask2former.image_processing_mask2former import convert_segmentation_to_rle
    t0 = time.perf_counter()
    for m in maps:
        convert_segmentation_to_rle(m)
    return {"ms_per_32_frames_hf_convert_on_host": (time.perf_counter() - t0) * 1e3 * 32 / len(maps),
            "host_threads": torch.get_num_threads()}


def serving(rounds, steps):
    import bench
    from rgbd_b200 import serving as S
    B, (H, W) = 32, (bench.H, bench.W)
    model, _ = bench.build_whole_model()
    model.cuda()
    rgb, depth = bench.make_frames(8)
    idx = np.arange(B) % 8
    rgb, depth = torch.from_numpy(np.ascontiguousarray(rgb[idx])), torch.from_numpy(np.ascontiguousarray(depth[idx]))
    segs = {}
    for flag in (False, True):
        s = S.RgbdInstanceSegmenter(model, B, (H, W), threshold=0.0, return_coco_annotation=flag)
        for b in range(2):
            s.in_host[b][0].copy_(rgb)
            s.in_host[b][1].copy_(depth)
        s.warmup()
        segs["coco" if flag else "off"] = s
    times = {"off": [], "coco": []}
    in_result = {"off": [], "coco": []}               # host milliseconds per step inside result(), after the wait
    d2h = {"off": [], "coco": []}                     # d2h_bytes_per_step after each result()

    def read(s, name, b):
        s._ev_d2h[b].synchronize()                    # the wait for the device; what follows is host work
        t1 = time.perf_counter()
        s.result(b)
        d2h[name].append(s.d2h_bytes_per_step)
        return time.perf_counter() - t1

    for _ in range(rounds):
        for name, s in segs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pending, t_res = None, 0.0
            for _ in range(steps):
                b = s.submit()
                if pending is not None:
                    t_res += read(s, name, pending)
                pending = b
            t_res += read(s, name, pending)
            times[name].append(B * steps / (time.perf_counter() - t0))
            in_result[name].append(t_res / steps * 1e3)
    out = {"batch": B, "frame": [H, W], "steps_per_round": steps, "rounds": rounds}
    for name in times:
        out[f"frames_per_s_{name}"] = times[name]
        out[f"ms_in_result_per_step_{name}"] = in_result[name]
        out[f"d2h_bytes_per_step_{name}_mean"] = float(np.mean(d2h[name]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    info = card()
    import rgbd_b200  # noqa: F401
    from rgbd_b200 import functional as Fn, postprocess as PP
    from oracle.make_golden_postproc import synth_outputs
    cls, masks = synth_outputs(5, 32, 100, 48, 120, 160)
    outs = SimpleNamespace(class_queries_logits=cls.cuda(), masks_queries_logits=masks.cuda())
    r = Fn.post_process_instances(outs.class_queries_logits, outs.masks_queries_logits, 0.0, (480, 640))
    seg = r.segmentation.clone()
    yy, xx = torch.meshgrid(torch.arange(480), torch.arange(640), indexing="ij")
    checker = ((yy + xx) % 2 - 1).int().expand(32, 480, 640).contiguous().cuda()
    res = {"card": info,
           "encoder_model_sized": {**encoder(Fn, seg, 100, args.reps), "segments_kept": int(r.count.sum())},
           "encoder_checkerboard": encoder(Fn, checker, 100, args.reps),
           "post_process": {**post_process(PP, outs, [(480, 640)] * 32, 5), **hf_host([m.float() for m in seg.cpu()])}}
    res["serving"] = serving(args.rounds, args.steps)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r03_rle.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
