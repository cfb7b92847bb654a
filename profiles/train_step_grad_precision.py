"""Cost of the split-precision DSAM backward (DSAModule.grad_precision = "fp32").

    python profiles/train_step_grad_precision.py steps --out DIR    # step times of the train record, three configurations
    python profiles/train_step_grad_precision.py kernels --out DIR  # torch.profiler times of dsam_wgrad_kernel per stage

``steps``: the hot-path training step of bench.py's ``train`` record (DepthGuidance forward + backward, batch 8, 480x640,
Swin-T channels, ratio predictor frozen) with (precision, grad_precision) = (bf16, bf16), (bf16, fp32) and (fp32, fp32).
CUDA events after warm-up; the configurations alternate round by round within the one process.  ``kernels``: each DSAM
stage's weight-gradient kernel on its staged operands, bf16 and split, timed by torch.profiler; achieved TFLOP/s from
shapes (2 * N_out * n_seg * taps * C_in * B * Ho * Wo, three times that in split mode).  Both modes print one JSON object
and write it to DIR/train_grad_precision_<mode>.json, together with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = [("bf16", "bf16"), ("bf16", "fp32"), ("fp32", "fp32")]


def card():
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def steps(args):
    import bench
    from rgbd_b200 import functional as Fn, modules, synthetic_weights as SW
    dev = torch.device("cuda")
    B = 8
    rgb_u8, depth_u8 = bench.make_frames(B)
    pv = Fn.pack_pixel_values(torch.from_numpy(rgb_u8).to(dev), torch.from_numpy(depth_u8).to(dev))
    feats = bench.make_features(B, 7, dev)
    g = torch.Generator(device="cpu").manual_seed(11)
    douts = [torch.randn(f.shape, generator=g).to(dev) for f in feats]
    models = {}
    for prec, gprec in CONFIGS:
        m = modules.DepthGuidance(bench.CHANS, precision=prec, grad_precision=gprec)
        m.load_state_dict(SW.guidance_weights(seed=42, channels=bench.CHANS))
        m.to(dev).train()
        for p in m.ratio_predictor.parameters():
            p.requires_grad_(False)
        models[(prec, gprec)] = m

    def step(m):
        for p in m.parameters():
            p.grad = None
        torch.autograd.backward(m(pv, feats), douts)

    for m in models.values():
        for _ in range(args.warmup):
            step(m)
    torch.cuda.synchronize()
    times = {c: [] for c in CONFIGS}
    for _ in range(args.rounds):
        for c in CONFIGS:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(models[c])
            e1.record()
            torch.cuda.synchronize()
            times[c].append(e0.elapsed_time(e1) / args.steps)
    base = float(np.median(times[CONFIGS[0]]))
    res = {"what": "DepthGuidance train step (forward + backward), batch 8, 480x640, Swin-T channels, ms per step",
           "steps_per_round": args.steps, "rounds": args.rounds, "configs": {}}
    for c in CONFIGS:
        med = float(np.median(times[c]))
        res["configs"][f"precision={c[0]},grad_precision={c[1]}"] = {
            "ms_median": med, "ms_min": float(min(times[c])), "ms_max": float(max(times[c])), "ratio_to_bf16_bf16": med / base}
    return res


def kernels(args):
    from torch.autograd import DeviceType
    from torch.profiler import profile, ProfilerActivity
    from rgbd_b200 import functional as Fn
    dev = torch.device("cuda")
    B, H, W, R = 8, 480, 640, 3
    stages = [("dsam0", 96, 192, (H // 4, W // 4)), ("dsam1", 192, 384, (H // 8, W // 8)), ("dsam2", 384, 768, (H // 16, W // 16))]
    g = torch.Generator(device="cpu").manual_seed(5)
    res = {"what": "dsam_wgrad_kernel per DSAM stage of the train record (batch 8, 480x640, Swin-T), torch.profiler",
           "repeats": args.repeats, "stages": {}}
    for name, ci, co, (h, w) in stages:
        ho, wo = (h + 1) // 2, (w + 1) // 2
        c_pad = -(-ci // 64) * 64
        n_seg = R + 2
        pitch = -(-wo // 8) * 8
        x = torch.randn(B, ci, h, w, generator=g).to(dev)
        gr = torch.randn(B, co, ho, wo, generator=g).to(dev)
        codes = torch.randint(0, 16, (B, h, w), generator=g, dtype=torch.uint8).to(dev)
        gp, gp_lo = Fn.cast_bf16_pitched(gr, pitch, lo=True)
        xt = torch.zeros(2, B, n_seg, 6, c_pad, ho, pitch, dtype=torch.bfloat16, device=dev)
        Fn.dsam_pack_t(x, codes, xt[0], c_pad, pitch, n_seg, R + 1, True, out_lo=xt[1])
        calls = {"bf16": lambda: Fn.dsam_wgrad(gp, xt[0], co, c_pad, (ho, wo), n_seg, True),
                 "split": lambda: Fn.dsam_wgrad(gp, xt[0], co, c_pad, (ho, wo), n_seg, True, g_lo=gp_lo, xt_lo=xt[1])}
        flop = 2.0 * co * n_seg * 9 * ci * B * ho * wo
        out = {}
        for mode, call in calls.items():
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.repeats):
                    call()
                torch.cuda.synchronize()
            us = [e.time_range.elapsed_us() for e in prof.events()
                  if e.device_type == DeviceType.CUDA and "dsam_wgrad_kernel" in e.name]
            assert len(us) == args.repeats, (name, mode, len(us))
            t = float(np.median(us))
            f = flop * (3 if mode == "split" else 1)
            out[mode] = {"us_median": t, "us_min": float(min(us)), "us_max": float(max(us)), "gflop": f / 1e9,
                         "tflops": f / (t * 1e-6) / 1e12}
        out["time_ratio_split_to_bf16"] = out["split"]["us_median"] / out["bf16"]["us_median"]
        res["stages"][name] = {"c_in": ci, "n_out": co, "stage_input_hw": [h, w], "c_pad": c_pad, **out}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["steps", "kernels"])
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=20)
    args = ap.parse_args()
    info = card()
    res = {"card": info, **(steps(args) if args.mode == "steps" else kernels(args))}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, f"train_grad_precision_{args.mode}.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
