"""Cost of the pycocotools RLE output of the instance post-processing, beside the HF-format run-length output.

    python profiles/pycocotools_rle_time.py --out DIR      # writes DIR/r03_pycocotools_rle.json and prints it

1. ``encoder``: the nine kernels of ``functional.instance_rle`` (transpose, the four ``rle_*`` kernels on the transposed
   maps, size, scan, base, emit) captured in one CUDA graph and replayed back to back, timed with CUDA events, on 32 painted
   480x640 maps from model-sized outputs (``synth_outputs(5, 32, 100, 48, 120, 160)``, threshold 0) and on a checkerboard
   of one segment (one run per two pixels), beside ``functional.label_map_rle`` on the same maps.  The 39 MB batch of maps
   fits in the 126 MB L2, so after the first replay the maps are read from there.  Per-kernel device times come from
   torch.profiler in a run of their own.
2. ``post_process``: wall time of ``post_process_instance_segmentation`` per 32 frames with ``return_pycocotools_rle=True``,
   with both flags off (maps copied to the host) and with ``return_coco_annotation=True``.
3. ``serving``: ``RgbdInstanceSegmenter`` (bench.py's whole model, batch 32, 480x640, CUDA graphs) with both flags off, with
   ``return_coco_annotation`` and with ``return_pycocotools_rle``, alternated round by round in one process; every step's
   ``result`` is read.  Also the host time inside ``result`` once the step's download has finished, and
   ``d2h_bytes_per_step`` after each ``result``.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import re
import sys
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from rle_time import card, time_graph  # noqa: E402


def kernel_us(call, reps):
    """Device time per call of each kernel of ``call`` from torch.profiler (a run of its own, after the graph timing)."""
    from torch.profiler import ProfilerActivity, profile
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    names = ((re.search(r"(rle|coco)_\w+_kernel", e.key), e) for e in prof.key_averages())
    out = {}
    for m, e in names:
        if m:       # rle_base_kernel runs twice per instance_rle call
            out[m.group(0)] = out.get(m.group(0), 0.0) + e.device_time_total / reps
    return out


def encoders(Fn, seg, count, L, reps):
    pyc_bufs = Fn.instance_rle_buffers(*seg.shape, L, seg.device)
    hf_bufs = Fn.label_map_rle_buffers(*seg.shape, L, seg.device)
    ms, out = time_graph(lambda: Fn.instance_rle(seg, count, L, *pyc_bufs), reps)
    ms_hf, out_hf = time_graph(lambda: Fn.label_map_rle(seg, L, *hf_bufs), reps)
    assert int(out.bad[0]) == 0
    return {"shape": list(seg.shape), "labels": L, "segments": int(count.sum()), "characters": int(out.base[-1]),
            "runs_row_major": int(out_hf.base[-1]),
            "us_per_batch_pycocotools_rle": ms * 1e3, "us_per_batch_label_map_rle": ms_hf * 1e3,
            "kernel_us_torch_profiler_pycocotools_rle": kernel_us(lambda: Fn.instance_rle(seg, count, L, *pyc_bufs), 50),
            "kernel_us_torch_profiler_label_map_rle": kernel_us(lambda: Fn.label_map_rle(seg, L, *hf_bufs), 50)}


FLAGS = (("off", {}), ("coco", {"return_coco_annotation": True}), ("pycocotools", {"return_pycocotools_rle": True}))


def post_process(PP, outs, sizes, reps):
    res = {}
    for name, kw in FLAGS:
        PP.post_process_instance_segmentation(outs, threshold=0.0, target_sizes=sizes, **kw)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = PP.post_process_instance_segmentation(outs, threshold=0.0, target_sizes=sizes, **kw)
            if name == "off":
                [x["segmentation"].cpu() for x in r]       # the maps on the host, like the run-length outputs
        torch.cuda.synchronize()
        res[f"ms_per_32_frames_{name}"] = (time.perf_counter() - t0) / reps * 1e3 * 32 / len(sizes)
    return res


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
    for name, kw in FLAGS:
        s = S.RgbdInstanceSegmenter(model, B, (H, W), threshold=0.0, **kw)
        for b in range(2):
            s.in_host[b][0].copy_(rgb)
            s.in_host[b][1].copy_(depth)
        s.warmup()
        segs[name] = s
    times = {n: [] for n in segs}
    in_result = {n: [] for n in segs}                  # host milliseconds per step inside result(), after the wait
    d2h = {n: [] for n in segs}                        # d2h_bytes_per_step after each result()

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
    seg, count = r.segmentation.clone(), r.count.clone()
    yy, xx = torch.meshgrid(torch.arange(480), torch.arange(640), indexing="ij")
    checker = ((yy + xx) % 2 - 1).int().expand(32, 480, 640).contiguous().cuda()
    res = {"card": info,
           "encoder_model_sized": encoders(Fn, seg, count, 100, args.reps),
           "encoder_checkerboard": encoders(Fn, checker, torch.ones(32, dtype=torch.int32, device="cuda"), 100, args.reps),
           "post_process": post_process(PP, outs, [(480, 640)] * 32, 5)}
    res["serving"] = serving(args.rounds, args.steps)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r03_pycocotools_rle.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
