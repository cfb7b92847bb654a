"""The split-precision DSAM backward (``DSAModule.grad_precision = "fp32"``) on the GPU.

The lo parts of the staged operands must be bit-exact; the weight gradient kernel in split mode, the whole stage backward
and the whole ``DepthGuidance`` training step are held to the exact fp32 operands (``_split_reference.dsam_reference(
operands="fp32")``) at the split bars: element-wise (accumulation bar + TAU_SPLIT) * ref_abs and relative L2 1e-4
(``_split_reference.check_split``).  The bf16 mode must miss the L2 bar (the test can tell the modes apart) and the forward
output must not depend on the gradient mode.  Measured errors are logged with ``_parity_report.report``."""
import numpy as np
import pytest
import torch

import rgbd_b200  # noqa: F401
from rgbd_b200 import synthetic
from oracle import hotpath as O
from oracle import weights as OW
import _grad_reference as GR
import _split_reference as SR
from _parity_report import report

pytestmark = pytest.mark.gpu

R = 3


@pytest.fixture(scope="module")
def fn():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from rgbd_b200 import functional
    return functional


@pytest.fixture(scope="module")
def mods(fn):
    from rgbd_b200 import modules
    return modules


def _round_up(a, b):
    return -(-a // b) * b


def _c_pad(c_in):
    return _round_up(c_in, 64) if c_in > 32 else 32           # DSAModule._geometry


def _random_codes(rs, B, H, W, variant):
    codes = np.zeros((B, H, W), dtype=np.uint8)
    for b in range(B):
        for t in range(int(variant[b])):
            codes[b] |= (rs.rand(H, W) < 0.45).astype(np.uint8) << t
    return torch.from_numpy(codes)


def _check_all(case, results):
    bad = []
    for name, res in results.items():
        report(f"backward-fp32/{case}/{name}", **{k: v for k, v in res.items() if k != "ok"})
        if not res["ok"]:
            bad.append((name, res))
    assert not bad, bad


def _bf16_lo(t):
    """bf16(v - float(bf16(v))) as a bf16 tensor (host reference of the lo part)."""
    f = t.float()
    return (f - f.bfloat16().float()).bfloat16()


def _hard_values(shape, seed):
    """Normal values with exact bf16 rounding ties (low 16 bits 0x8000, both parities of the kept bit), some at 1e30 and
    some at 1e-35 (their lo parts are subnormal)."""
    rs = np.random.RandomState(seed)
    g = torch.from_numpy(rs.randn(*shape).astype(np.float32))
    bits = g.view(torch.int32).clone()
    bits.view(-1)[::7] = (bits.view(-1)[::7] & ~0xFFFF) | 0x8000
    g = bits.view(torch.float32)
    g.view(-1)[1::11] *= 1e30
    g.view(-1)[2::13] *= 1e-35
    return g


# ---------------------------------------------------------------------------------------------------
# a. staging of the lo parts: bit-exact
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 72, 15, 21), (3, 192, 60, 80), (1, 8, 5, 1)])
def test_cast_bf16_pitched_lo_part_is_bit_exact(fn, shape):
    g = _hard_values(shape, 3)
    W = shape[-1]
    pitch = _round_up(W, 8)
    hi, lo = (t.cpu() for t in fn.cast_bf16_pitched(g.cuda(), pitch, lo=True))
    assert hi.shape == lo.shape == (*shape[:-1], pitch) and lo.dtype == torch.bfloat16
    assert torch.equal(hi[..., :W].view(torch.int16), g.bfloat16().view(torch.int16))
    assert torch.equal(lo[..., :W].view(torch.int16), _bf16_lo(g).view(torch.int16))
    assert not hi[..., W:].view(torch.int16).any() and not lo[..., W:].view(torch.int16).any()
    # the hi output is the bf16 mode's output, bit for bit
    assert torch.equal(hi.view(torch.int16), fn.cast_bf16_pitched(g.cuda(), pitch).cpu().view(torch.int16))


def _pack_t_reference(x, codes, c_pad, n_seg, masked, split, w2p, part):
    """Index-built layout of dsam_pack_t (see tests/test_gpu_backward.py) of ``part(x * bit(code, seg))``."""
    B, C, H, W = x.shape
    H2 = (H + 1) // 2 if split else H
    n_par = 6 if split else 1
    out = torch.zeros(B, n_seg, n_par, c_pad, H2, w2p, dtype=torch.bfloat16)
    bits = GR.region_bits(codes, n_seg).bool()
    for s in range(n_seg):
        xm = part(torch.where(bits[:, s:s + 1], x, 0.0) if s < masked else x)          # +0, never -0
        if not split:
            out[:, s, 0, :C, :, :W] = xm
            continue
        for py in (0, 1):
            for px in (0, 1):
                p = xm[:, :, py::2, px::2]
                out[:, s, 2 * py + px, :C, :p.shape[2], :p.shape[3]] = p
            out[:, s, 4 + py, :, :, 1:] = out[:, s, 2 * py + 1, :, :, :-1]
    return out


@pytest.mark.parametrize("ci,co,hw,B", [(40, 72, (33, 47), 2), (96, 192, (12, 16), 2), (64, 128, (15, 20), 1),
                                        (24, 24, (9, 11), 3)], ids=["odd-40", "even-96-no-pitch", "odd-rows", "identity"])
def test_dsam_pack_t_lo_part_is_bit_exact(fn, ci, co, hw, B):
    rs = np.random.RandomState(ci + co)
    split = ci != co
    n_seg = R + 2 if split else R + 1
    H, W = hw
    H2, W2 = ((H + 1) // 2, (W + 1) // 2) if split else (H, W)
    w2p, c_pad = _round_up(W2, 8), _c_pad(ci)
    x = _hard_values((B, ci, H, W), ci)
    codes = _random_codes(rs, B, H, W, [4] * B)
    hi = torch.zeros(B, n_seg, 6 if split else 1, c_pad, H2, w2p, dtype=torch.bfloat16, device="cuda")
    lo = torch.zeros_like(hi)
    fn.dsam_pack_t(x.cuda(), codes.cuda(), hi, c_pad, w2p, n_seg, R + 1, split, out_lo=lo)
    hi, lo = hi.cpu(), lo.cpu()
    for got, part in ((hi, lambda t: t.bfloat16()), (lo, _bf16_lo)):    # masked-out pixels: +0 in both parts
        ref = _pack_t_reference(x, codes, c_pad, n_seg, R + 1, split, w2p, part)
        assert torch.equal(got.view(torch.int16), ref.view(torch.int16))
        assert not got[:, :, :, ci:].view(torch.int16).any()                          # pad channels
        if split:
            assert not got[:, :, 4:, :, :, 0].view(torch.int16).any()                 # shifted planes: column 0
            assert not got[:, :, :4, :, :, W2:].view(torch.int16).any()               # pitch columns
        else:
            assert not got[..., W:].view(torch.int16).any()


# ---------------------------------------------------------------------------------------------------
# b. dsam_wgrad in split mode
# ---------------------------------------------------------------------------------------------------
def _split_block_n(c_pad, max_smem):
    """BLOCK_N of rgbd_dsam_wgrad in split mode: the widest multiple of 32 dividing C_pad that leaves 3 stages."""
    for bn in range(256, 32, -32):
        if c_pad % bn == 0 and (max_smem - 2048 - 160) // (2 * (128 * 128 + bn * 128)) >= 3:
            return bn
    return 32


@pytest.mark.parametrize("ci,co,hw,B", [
    (96, 192, (120, 160), 8),        # Swin-T stage 0 at 480x640
    (384, 768, (30, 40), 8),         # Swin-T stage 2
    (512, 1024, (60, 80), 2),        # Swin-B stage 2 at 960x1280
    (40, 72, (15, 21), 5),           # C_pad 64, N 72 (one partial M tile), 5 images over uneven splits
    (96, 192, (33, 47), 3),          # odd sizes
    (64, 64, (30, 40), 3),           # identity 1x1 (no parity split)
], ids=["swinT-s0-B8", "swinT-s2-B8", "swinB-s2-B2", "40to72-B5", "odd-B3", "identity-B3"])
def test_dsam_wgrad_split(fn, ci, co, hw, B):
    rs = np.random.RandomState(ci * 7 + co + 1)
    split = ci != co
    n_seg = R + 2 if split else R + 1
    H, W = hw
    Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if split else (H, W)
    c_pad = _c_pad(ci)
    pitch = _round_up(Wo, 8)
    x = torch.from_numpy(rs.randn(B, ci, H, W).astype(np.float32))
    codes = _random_codes(rs, B, H, W, [4] * B)
    g = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32))
    gp, gp_lo = fn.cast_bf16_pitched(g.cuda(), pitch, lo=True)
    xt = torch.zeros(2, B, n_seg, 6 if split else 1, c_pad, Ho, pitch, dtype=torch.bfloat16, device="cuda")
    fn.dsam_pack_t(x.cuda(), codes.cuda(), xt[0], c_pad, pitch, n_seg, R + 1, split, out_lo=xt[1])
    dw = fn.dsam_wgrad(gp, xt[0], co, c_pad, (Ho, Wo), n_seg, split, g_lo=gp_lo, xt_lo=xt[1]).cpu()
    k = 3 if split else 1
    w = OW.dsam_weights(ci, co, seed=1)
    ref = SR.dsam_reference(x, codes, None, g, w, operands="fp32")
    names = [f"conv_layers.{t}.weight" for t in range(R + 1)] + (["rgb_projection.weight"] if split else [])
    results = {}
    for s, name in enumerate(names):
        got = dw[:, s, :, :ci].reshape(co, k, k, ci).permute(0, 3, 1, 2)
        results[name] = SR.check_split(got, *ref[name], GR.TAU_DW)
    results["pad_channels"] = GR.check(dw[..., ci:], torch.zeros_like(dw[..., ci:], dtype=torch.float64),
                                       torch.zeros_like(dw[..., ci:], dtype=torch.float64), 0.0)
    props = torch.cuda.get_device_properties(0)
    max_smem = getattr(props, "shared_memory_per_block_optin", 232448)
    bn = _split_block_n(c_pad, max_smem)
    report(f"backward-fp32/wgrad/{ci}to{co}/{H}x{W}/B{B}/geometry", block_n=bn)
    _check_all(f"wgrad/{ci}to{co}/{H}x{W}/B{B}/bn{bn}", results)


# ---------------------------------------------------------------------------------------------------
# c. whole stage backward through autograd
# ---------------------------------------------------------------------------------------------------
_FRAMES = [(20, "nyu"), (21, "constant"), (22, "nyu"), (23, "two_valued"), (24, "uniform"), (25, "nyu"),
           (26, "nyu"), (27, "constant")]
_RATIOS = [0.1, 0.3, 0.2, 0.4, 0.3, 0.15, 0.25, 0.35]


def _decomposition(fn, hw, dhw, frames):
    grays = []
    for idx, kind in frames:
        _, d = synthetic.synth_rgbd_u8(idx, dhw[0], dhw[1], kind)
        grays.append(O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2))))
    ratios = torch.tensor(_RATIOS[:len(frames)], device="cuda")
    dec = fn.depth_decompose(ratios, [hw], gray=torch.from_numpy(np.stack(grays)).cuda())
    return dec.pooled[0], dec.bias_variant


def _stage_backward(mods, fn, ci, co, hw, dhw, frames, seed, grad_precision="fp32"):
    """Stage forward + backward with the given gradient mode; results of the split bars against the exact operands."""
    w = OW.dsam_weights(ci, co, seed=seed)
    m = mods.DSAModule(ci, co, R)
    m.load_state_dict(w)
    m.grad_precision = grad_precision
    m.cuda().train()
    B = len(frames)
    codes, variant = _decomposition(fn, hw, dhw, frames)
    rs = np.random.RandomState(seed)
    proj = ci != co
    Ho, Wo = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if proj else hw
    x = torch.from_numpy(rs.randn(B, ci, *hw).astype(np.float32)).cuda().requires_grad_(True)
    res = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32)).cuda().requires_grad_(True)
    out = m.stage_forward(x, codes, variant, residual=res)
    g = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32))
    out.backward(g.cuda())
    ref = SR.dsam_reference(x, codes, variant, g, w, operands="fp32")
    results = {}
    for name, p in m.named_parameters():
        if name.endswith(".bias"):
            results[name] = GR.check(p.grad, *ref[name], GR.TAU_DB)
        else:
            results[name] = SR.check_split(p.grad, *ref[name], GR.TAU_DW)
    results["x"] = SR.check_split(x.grad, *ref["x"], GR.TAU_DX)
    assert torch.equal(res.grad.cpu(), g), "the residual's gradient is G itself"
    return results, variant.cpu(), {name: p.grad for name, p in m.named_parameters()}


_STAGE_CASES = [
    # ci, co, stage input hw, depth hw, frames
    ("swinT-s0", 96, 192, (120, 160), (480, 640), _FRAMES),
    ("swinT-s1", 192, 384, (60, 80), (480, 640), _FRAMES),
    ("swinT-s2", 384, 768, (30, 40), (480, 640), _FRAMES),
    ("swinB-s0", 128, 256, (240, 320), (960, 1280), _FRAMES[:2]),
    ("swinB-s1", 256, 512, (120, 160), (960, 1280), _FRAMES[:2]),
    ("swinB-s2", 512, 1024, (60, 80), (960, 1280), _FRAMES[:2]),
    ("odd", 96, 192, (33, 47), (132, 188), _FRAMES[:3]),
    ("cin40", 40, 72, (15, 21), (60, 84), _FRAMES[:5]),
    ("identity", 64, 64, (30, 40), (120, 160), _FRAMES[:3]),
    ("tiny", 32, 64, (8, 8), (32, 32), _FRAMES[:1]),
]


@pytest.mark.parametrize("case,ci,co,hw,dhw,frames", _STAGE_CASES,
                         ids=[f"{c[0]}-{c[1]}to{c[2]}-{c[3][0]}x{c[3][1]}-B{len(c[5])}" for c in _STAGE_CASES])
def test_dsam_stage_backward_fp32_against_exact_operands(mods, fn, case, ci, co, hw, dhw, frames):
    results, variant, _ = _stage_backward(mods, fn, ci, co, hw, dhw, frames, seed=700 + ci + co)
    report(f"backward-fp32/stage/{case}/geometry", variants=variant.tolist())
    _check_all(f"stage/{case}", results)


def test_dsam_unused_region_gets_an_exactly_zero_gradient_in_fp32_mode(mods, fn):
    frames = [(21, "constant"), (27, "constant")]
    results, variant, grads = _stage_backward(mods, fn, 96, 192, (30, 40), (120, 160), frames, seed=712)
    assert variant.tolist() == [2, 2]
    for name in ("conv_layers.1.weight", "conv_layers.2.weight", "conv_layers.3.weight", "conv_layers.2.bias",
                 "conv_layers.3.bias"):
        assert float(grads[name].abs().max()) == 0.0, name
    _check_all("stage/region-unused", results)


def test_dsam_stage_backward_fp32_is_within_the_bars_run_to_run(mods, fn):
    for rep in range(2):
        results, _, _ = _stage_backward(mods, fn, 96, 192, (120, 160), (480, 640), _FRAMES, seed=713)
        _check_all(f"stage/swinT-s0-repeat{rep}", results)


def test_bf16_gradients_miss_the_fp32_bar(mods, fn):
    """Negative control: the bf16 mode against the same exact-operand reference is well above relative L2 1e-4."""
    results, _, _ = _stage_backward(mods, fn, 96, 192, (120, 160), (480, 640), _FRAMES, seed=714, grad_precision="bf16")
    for name in [f"conv_layers.{t}.weight" for t in range(R + 1)] + ["rgb_projection.weight", "x"]:
        report(f"backward-fp32/negative-control-bf16/{name}", rel_l2=results[name]["rel_l2"],
               max_norm_err=results[name]["max_norm_err"])
        assert results[name]["rel_l2"] > SR.SPLIT_REL_L2, (name, results[name])


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_forward_output_does_not_depend_on_grad_precision(mods, fn, precision):
    ci, co, hw, dhw = 96, 192, (120, 160), (480, 640)
    w = OW.dsam_weights(ci, co, seed=715)
    codes, variant = _decomposition(fn, hw, dhw, _FRAMES)
    x = torch.from_numpy(np.random.RandomState(715).randn(len(_FRAMES), ci, *hw).astype(np.float32)).cuda()
    outs = []
    for gp in ("bf16", "fp32"):
        m = mods.DSAModule(ci, co, R)
        m.load_state_dict(w)
        m.precision, m.grad_precision = precision, gp
        m.cuda().train()
        outs.append(m.stage_forward(x.clone().requires_grad_(True), codes, variant).detach())
    assert torch.equal(outs[0], outs[1])


# ---------------------------------------------------------------------------------------------------
# d. the whole training step at the train record's shape against oracle autograd
# ---------------------------------------------------------------------------------------------------
def _swin_sizes(H, W):
    return [(-(-H // s), -(-W // s)) for s in (4, 8, 16, 32)]


def test_depth_guidance_fp32_gradients_at_the_train_record_shape(mods):
    """DepthGuidance(precision="fp32", grad_precision="fp32") in .train() at 480x640, batch 8, Swin-T channels against
    float64 torch autograd through the CPU oracle: every DSAM and DGGM parameter within relative L2 1e-4."""
    chans, (H, W), B = (96, 192, 384, 768), (480, 640), 8
    w = OW.guidance_weights(seed=701, channels=chans)
    m = mods.DepthGuidance(chans, precision="fp32", grad_precision="fp32")
    m.load_state_dict(w)
    m.cuda().train()
    pvs = []
    for j in range(B):
        rgb, d = synthetic.synth_rgbd_u8(90 + j, H, W, "nyu" if j % 4 else ("constant", "two_valued")[j // 4 % 2])
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))
    rs = np.random.RandomState(9)
    feats = [torch.from_numpy(rs.randn(B, c, h, ww).astype(np.float32)) for c, (h, ww) in zip(chans, _swin_sizes(H, W))]
    ratios = torch.tensor(_RATIOS, dtype=torch.float32)[:, None]
    douts = [torch.from_numpy(rs.randn(*f.shape).astype(np.float32)) for f in feats]
    out = m(pv.cuda(), [f.cuda() for f in feats], ratios=ratios.cuda())
    torch.autograd.backward(out, [d.cuda() for d in douts])
    wr = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in w.items()}
    ref, _ = O.depth_guidance_forward(wr, pv, feats, ratios=ratios)
    torch.autograd.backward(ref, douts)
    bad = []
    for name, p in m.named_parameters():
        if name.startswith("ratio_predictor."):
            assert p.grad is None, name
            continue
        g_ref = wr[name].grad
        if g_ref is None:           # a region no image used: exactly zero here (DSAModule's documented deviation)
            assert float(p.grad.abs().max()) == 0.0, name
            continue
        a, b = p.grad.double().cpu(), g_ref.double()
        err = float((a - b).norm() / b.norm().clamp_min(1e-30))
        bar = 1e-4
        report(f"backward-fp32/guidance-train-480x640-B8/{name}", rel_l2=err, bar=bar)
        if not err < bar:
            bad.append((name, err, bar))
    assert not bad, bad
