"""Per-stage DSAM GEMM times (operands pre-packed), batch 32, 480x640 pyramid.  RGBD_DSAM_PREMASKED=1 selects the
pre-masked five-fold operand + conv_gemm_2cta_kernel; default is dsam_fwd_kernel (masking in shared memory)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rgbd_b200 as R
from rgbd_b200.modules import DSAModule

torch.manual_seed(0)
B = int(os.environ.get("B", 32))
dev = "cuda"
chans = [96, 192, 384, 768]
sizes = [(120, 160), (60, 80), (30, 40)]
for i in range(3):
    torch.manual_seed(i)
    m = DSAModule(chans[i], chans[i + 1]).to(dev)
    H, W = sizes[i]
    x = torch.randn(B, chans[i], H, W, device=dev)
    codes = torch.randint(0, 16, (B, H, W), device=dev, dtype=torch.uint8)
    var = torch.full((B,), 4, device=dev, dtype=torch.int32)
    m._stage_forward_impl(x, codes, var)
    for mode in ("pack+gemm", "gemm"):
        m._gemm_only = mode == "gemm"
        for _ in range(3):
            m._stage_forward_impl(x, codes, var)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        n = 20
        for _ in range(n):
            m._stage_forward_impl(x, codes, var)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        flops = 2.0 * B * ((H + 1) // 2) * ((W + 1) // 2) * chans[i + 1] * 45 * chans[i]
        print(f"stage {i} {mode:10s} {ms*1e3:8.1f} us  {flops/ms/1e9:7.1f} TFLOP/s (useful)")
    out = m._stage_forward_impl(x, codes, var)
    print(f"   checksum {float(out.double().abs().sum()):.6e}")
