"""The DSAM and DGGM backward kernels against the float64 references of tests/_grad_reference.py, at the shapes the
training step runs (the ``train`` record of bench.py: batch 8, 480x640, Swin-T channels) and at the edges where the kernels
could go wrong: odd sizes, channel counts that are not multiples of 32, the 1x1 identity variant, a single M tile, split-K
over an uneven number of images.

Every operand a backward kernel uses is rebuilt exactly on the host (bf16 round-to-nearest of G, of x * bit_t(code) and of
the weights; fp32 G for the bias gradient and the identity residual), so the reference differs from a kernel only by fp32
accumulation order and the bar is element-wise: |got - ref| <= tau * ref_abs (``_grad_reference.check``).  Measured errors
are logged with ``_parity_report.report``."""
import numpy as np
import pytest
import torch

import rgbd_b200  # noqa: F401
from rgbd_b200 import synthetic
from rgbd_b200.functional import best_box
from oracle import hotpath as O
from oracle import weights as OW
import _grad_reference as GR
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
    """Region codes with every bit pattern of the bits an image uses (t < variant[b])."""
    codes = np.zeros((B, H, W), dtype=np.uint8)
    for b in range(B):
        for t in range(int(variant[b])):
            codes[b] |= (rs.rand(H, W) < 0.45).astype(np.uint8) << t
    return torch.from_numpy(codes)


def _check_all(case, results):
    """Log every tensor's measured error, then fail with the list of tensors over their bar."""
    bad = []
    for name, res in results.items():
        report(f"backward/{case}/{name}", **{k: v for k, v in res.items() if k != "ok"})
        if not res["ok"]:
            bad.append((name, res))
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------
# a. operand staging: bit-exact
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 72, 15, 21), (3, 192, 60, 80), (1, 8, 5, 1)])
def test_cast_bf16_pitched_is_round_to_nearest_with_zero_pitch(fn, shape):
    rs = np.random.RandomState(3)
    g = torch.from_numpy(rs.randn(*shape).astype(np.float32))
    # exact ties of the bf16 rounding (low 16 bits 0x8000, both parities of the kept bit) and a few large / tiny values
    bits = g.view(torch.int32).clone()
    bits.view(-1)[::7] = (bits.view(-1)[::7] & ~0xFFFF) | 0x8000
    g = bits.view(torch.float32)
    g.view(-1)[1::11] *= 1e30
    g.view(-1)[2::13] *= 1e-35
    W = shape[-1]
    pitch = _round_up(W, 8)
    out = fn.cast_bf16_pitched(g.cuda(), pitch).cpu()
    assert out.shape == (*shape[:-1], pitch) and out.dtype == torch.bfloat16
    assert torch.equal(out[..., :W].view(torch.int16), g.bfloat16().view(torch.int16))
    assert not out[..., W:].view(torch.int16).any()


def _pack_t_reference(x, codes, c_pad, n_seg, masked, split, w2p):
    """Index-built layout of dsam_pack_t: out[b][seg][par][c][y2][x2] = bf16(x[b,c,y,x] * bit(code, seg)) with
    (par, y2, x2) = ((y&1)*2 + (x&1), y>>1, x>>1) in the parity split; planes 4 / 5 are planes 1 / 3 (px = 1) shifted
    right by one pixel within the pitched row (column 0 zero), so that the x-1 taps read a 16-byte aligned box."""
    B, C, H, W = x.shape
    H2 = (H + 1) // 2 if split else H
    n_par = 6 if split else 1
    out = torch.zeros(B, n_seg, n_par, c_pad, H2, w2p, dtype=torch.bfloat16)
    bits = GR.region_bits(codes, n_seg).bool()
    for s in range(n_seg):
        xm = (torch.where(bits[:, s:s + 1], x, 0.0) if s < masked else x).bfloat16()      # +0, never -0
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
def test_dsam_pack_t_layout_bit_exact(fn, ci, co, hw, B):
    rs = np.random.RandomState(ci + co)
    split = ci != co
    n_seg = R + 2 if split else R + 1
    H, W = hw
    H2, W2 = ((H + 1) // 2, (W + 1) // 2) if split else (H, W)
    w2p, c_pad = _round_up(W2, 8), _c_pad(ci)
    x = torch.from_numpy(rs.randn(B, ci, H, W).astype(np.float32))
    codes = _random_codes(rs, B, H, W, [4] * B)
    buf = torch.zeros(B, n_seg, 6 if split else 1, c_pad, H2, w2p, dtype=torch.bfloat16, device="cuda")
    fn.dsam_pack_t(x.cuda(), codes.cuda(), buf, c_pad, w2p, n_seg, R + 1, split)
    got = buf.cpu()
    ref = _pack_t_reference(x, codes, c_pad, n_seg, R + 1, split, w2p)
    assert torch.equal(got.view(torch.int16), ref.view(torch.int16))
    # the properties the wgrad kernel relies on, spelled out
    assert not got[:, :, :, ci:].view(torch.int16).any()                          # pad channels
    if split:
        assert not got[:, :, 4:, :, :, 0].view(torch.int16).any()                 # shifted planes: column 0
        assert not got[:, :, :4, :, :, W2:].view(torch.int16).any()               # pitch columns of the parity planes
        if W % 2:
            assert not got[:, :, [1, 3], :, :, W2 - 1].view(torch.int16).any()    # px = 1 has one column fewer
        if H % 2:
            assert not got[:, :, [2, 3, 5], :, H2 - 1].view(torch.int16).any()    # py = 1 has one row fewer
    else:
        assert not got[..., W:].view(torch.int16).any()


# ---------------------------------------------------------------------------------------------------
# b. bias gradients
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,ohw,variant", [(8, 192, (60, 80), None), (8, 192, (60, 80), [4, 2, 3, 1, 4, 2, 4, 3]),
                                             (3, 72, (17, 24), [1, 4, 2]), (2, 1024, (30, 40), None)],
                         ids=["swinT-s0-all", "swinT-s0-mixed", "ragged-mixed", "swinB-s2-all"])
def test_dsam_dbias(fn, B, N, ohw, variant):
    rs = np.random.RandomState(N + B)
    g = torch.from_numpy(rs.randn(B, N, *ohw).astype(np.float32))
    v = torch.tensor(variant, dtype=torch.int32) if variant is not None else None
    db = fn.dsam_dbias(g.cuda(), v.cuda() if v is not None else None, R + 1).cpu()
    ref = GR.dsam_bias_reference(g, v, R + 1)
    _check_all(f"dbias/{B}x{N}x{ohw[0]}x{ohw[1]}/{'mixed' if variant else 'all'}",
               {f"db{t}": GR.check(db[t], r, ra, GR.TAU_DB) for t, (r, ra) in enumerate(ref)})


# ---------------------------------------------------------------------------------------------------
# c. weight gradients: dsam_wgrad on operands staged by (a)
# ---------------------------------------------------------------------------------------------------
def _ksplit(B, ci, co, split, num_sms):
    """dsam_wgrad's split-K factor over images (rgbd_dsam_wgrad)."""
    c_pad = _c_pad(ci)
    block_n = c_pad if c_pad <= 256 else next(bn for bn in range(256, 31, -32) if c_pad % bn == 0)
    base = (R + 2 if split else R + 1) * (9 if split else 1) * -(-co // 128) * (c_pad // block_n)
    k = 1
    while k * 2 <= B and base * k < 2 * num_sms:
        k *= 2
    return k, block_n, base


@pytest.mark.parametrize("ci,co,hw,B", [
    (96, 192, (120, 160), 8),        # Swin-T stage 0 at 480x640: BLOCK_N 128, 2 M tiles (N 192), ksplit 4 on 148 SMs
    (384, 768, (30, 40), 8),         # Swin-T stage 2: BLOCK_N 192, ksplit 1
    (512, 1024, (60, 80), 2),        # Swin-B stage 2 at 960x1280: BLOCK_N 256
    (40, 72, (15, 21), 5),           # C_pad 64, N 72 (one partial M tile), 5 images over 4 splits
    (96, 192, (33, 47), 3),          # odd sizes, 3 images over 2 splits
    (64, 64, (30, 40), 3),           # identity 1x1 (no parity split)
], ids=["swinT-s0-B8", "swinT-s2-B8", "swinB-s2-B2", "40to72-B5", "odd-B3", "identity-B3"])
def test_dsam_wgrad(fn, ci, co, hw, B):
    rs = np.random.RandomState(ci * 7 + co)
    split = ci != co
    n_seg = R + 2 if split else R + 1
    H, W = hw
    Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if split else (H, W)
    H2 = Ho
    c_pad = _c_pad(ci)
    pitch = _round_up(Wo, 8)
    x = torch.from_numpy(rs.randn(B, ci, H, W).astype(np.float32))
    codes = _random_codes(rs, B, H, W, [4] * B)
    g = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32))
    gp = fn.cast_bf16_pitched(g.cuda(), pitch)
    xt = torch.zeros(B, n_seg, 6 if split else 1, c_pad, H2, pitch, dtype=torch.bfloat16, device="cuda")
    fn.dsam_pack_t(x.cuda(), codes.cuda(), xt, c_pad, pitch, n_seg, R + 1, split)
    dw = fn.dsam_wgrad(gp, xt, co, c_pad, (Ho, Wo), n_seg, split).cpu()            # (co, n_seg, taps, c_pad)
    k = 3 if split else 1
    w = OW.dsam_weights(ci, co, seed=1)                                              # shapes only: dW needs no weights
    ref = GR.dsam_reference(x, codes, None, g, w)
    names = [f"conv_layers.{t}.weight" for t in range(R + 1)] + (["rgb_projection.weight"] if split else [])
    results = {}
    for s, name in enumerate(names):
        got = dw[:, s, :, :ci].reshape(co, k, k, ci).permute(0, 3, 1, 2)
        results[name] = GR.check(got, *ref[name], GR.TAU_DW)
    results["pad_channels"] = GR.check(dw[..., ci:], torch.zeros_like(dw[..., ci:], dtype=torch.float64),
                                       torch.zeros_like(dw[..., ci:], dtype=torch.float64), 0.0)
    ks, block_n, base = _ksplit(B, ci, co, split, torch.cuda.get_device_properties(0).multi_processor_count)
    report(f"backward/wgrad/{ci}to{co}/{H}x{W}/B{B}/geometry", ksplit=ks, block_n=block_n, base_tiles=base)
    _check_all(f"wgrad/{ci}to{co}/{H}x{W}/B{B}/ksplit{ks}/bn{block_n}", results)


# ---------------------------------------------------------------------------------------------------
# d. whole stage backward through autograd
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


def _m_tiles(ci, co, hw, B):
    """M tiles of the input-gradient GEMM: one per best_box tile of the (parity-class) input plane per image."""
    H2, W2 = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if ci != co else hw
    bx, by = best_box(H2, W2)
    return B * -(-H2 // by) * -(-W2 // bx)


def _stage_backward(mods, fn, ci, co, hw, dhw, frames, seed, sum_loss=False):
    w = OW.dsam_weights(ci, co, seed=seed)
    m = mods.DSAModule(ci, co, R)
    m.load_state_dict(w)
    m.cuda().train()
    B = len(frames)
    codes, variant = _decomposition(fn, hw, dhw, frames)
    rs = np.random.RandomState(seed)
    proj = ci != co
    Ho, Wo = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if proj else hw
    x = torch.from_numpy(rs.randn(B, ci, *hw).astype(np.float32)).cuda().requires_grad_(True)
    res = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32)).cuda().requires_grad_(True)
    out = m.stage_forward(x, codes, variant, residual=res)
    if sum_loss:                    # G arrives as a stride-0 expanded tensor
        out.sum().backward()
        g = torch.ones(B, co, Ho, Wo)
    else:
        g = torch.from_numpy(rs.randn(B, co, Ho, Wo).astype(np.float32))
        out.backward(g.cuda())
    ref = GR.dsam_reference(x, codes, variant, g, w)
    results = {name: GR.check(p.grad, *ref[name], GR.tau_for(name)) for name, p in m.named_parameters()}
    results["x"] = GR.check(x.grad, *ref["x"], GR.TAU_DX)
    assert torch.equal(res.grad.cpu(), g), "the residual's gradient is G itself"
    return results, variant.cpu(), {name: p.grad for name, p in m.named_parameters()}


_STAGE_CASES = [
    # ci, co, stage input hw, depth hw, frames, what it covers
    ("swinT-s0", 96, 192, (120, 160), (480, 640), _FRAMES),           # the train record's shape; C_pad 128
    ("swinT-s1", 192, 384, (60, 80), (480, 640), _FRAMES),
    ("swinT-s2", 384, 768, (30, 40), (480, 640), _FRAMES),            # wgrad ksplit 1
    ("swinB-s0", 128, 256, (240, 320), (960, 1280), _FRAMES[:2]),     # BLOCK_N 256, 8 M tiles
    ("swinB-s1", 256, 512, (120, 160), (960, 1280), _FRAMES[:2]),
    ("swinB-s2", 512, 1024, (60, 80), (960, 1280), _FRAMES[:2]),
    ("odd", 96, 192, (33, 47), (132, 188), _FRAMES[:3]),               # last row / column of the odd parity planes
    ("cin40", 40, 72, (15, 21), (60, 84), _FRAMES[:5]),                # padded channels and N
    ("identity", 64, 64, (30, 40), (120, 160), _FRAMES[:3]),           # stride 1, residual G in the epilogue
    ("tiny", 32, 64, (8, 8), (32, 32), _FRAMES[:1]),                   # single M tile (single-CTA kernel)
]


@pytest.mark.parametrize("case,ci,co,hw,dhw,frames", _STAGE_CASES,
                         ids=[f"{c[0]}-{c[1]}to{c[2]}-{c[3][0]}x{c[3][1]}-B{len(c[5])}-mtiles{_m_tiles(c[1], c[2], c[3], len(c[5]))}"
                              for c in _STAGE_CASES])
def test_dsam_stage_backward_against_float64(mods, fn, case, ci, co, hw, dhw, frames):
    results, variant, _ = _stage_backward(mods, fn, ci, co, hw, dhw, frames, seed=600 + ci + co)
    report(f"backward/stage/{case}/geometry", variants=variant.tolist(), m_tiles=_m_tiles(ci, co, hw, len(frames)))
    _check_all(f"stage/{case}", results)


def test_dsam_stage_backward_of_a_sum_loss(mods, fn):
    """loss = out.sum(): G is a stride-0 expanded tensor that _DsamStageFunction.backward makes contiguous."""
    results, _, _ = _stage_backward(mods, fn, 96, 192, (33, 47), (132, 188), _FRAMES[:3], seed=611, sum_loss=True)
    _check_all("stage/odd-sum-loss", results)


def test_dsam_unused_region_gets_an_exactly_zero_gradient(mods, fn):
    """Two one-mode (constant) frames add biases 0 and 1 only and set region bit 0 only: the weights of segments 1..3 and
    the biases of segments 2..3 get exactly zero (the reference would leave .grad None; DSAModule's documented deviation)."""
    frames = [(21, "constant"), (27, "constant")]
    results, variant, grads = _stage_backward(mods, fn, 96, 192, (30, 40), (120, 160), frames, seed=612)
    assert variant.tolist() == [2, 2]
    for name in ("conv_layers.1.weight", "conv_layers.2.weight", "conv_layers.3.weight", "conv_layers.2.bias",
                 "conv_layers.3.bias"):
        assert float(grads[name].abs().max()) == 0.0, name
    assert float(grads["conv_layers.1.bias"].abs().max()) > 0.0
    _check_all("stage/region-unused", results)


def test_dsam_stage_backward_is_within_the_bar_run_to_run(mods, fn):
    """wgrad and dbias finish with fp32 atomics, so the gradients are not bit-reproducible; every run must meet the bar."""
    runs = []
    for rep in range(2):
        results, _, grads = _stage_backward(mods, fn, 96, 192, (120, 160), (480, 640), _FRAMES, seed=613)
        _check_all(f"stage/swinT-s0-repeat{rep}", results)
        runs.append(grads)
    report("backward/stage/swinT-s0-repeat/bit_equal",
           **{name: bool(torch.equal(runs[0][name], runs[1][name])) for name in runs[0]})


# ---------------------------------------------------------------------------------------------------
# e. DGGM parameter gradients
# ---------------------------------------------------------------------------------------------------
def _swin_sizes(H, W):
    return [(-(-H // s), -(-W // s)) for s in (4, 8, 16, 32)]


@pytest.mark.parametrize("case,chans,hw,sizes,B,sum_loss", [
    ("swinT-480x640-B8", [96, 192, 384, 768], (480, 640), _swin_sizes(480, 640), 8, False),
    ("swinB-960x1280-B1", [128, 256, 512, 1024], (960, 1280), _swin_sizes(960, 1280), 1, False),
    ("ragged-50x70-B2", [4, 8, 12, 16], (50, 70), [(13, 18), (7, 9), (4, 5), (2, 3)], 2, False),
    ("ragged-50x70-B2-sum-loss", [4, 8, 12, 16], (50, 70), [(13, 18), (7, 9), (4, 5), (2, 3)], 2, True),
], ids=["swinT-480x640-B8", "swinB-960x1280-B1", "ragged-50x70-B2", "ragged-50x70-B2-sum-loss"])
def test_dggm_param_gradients_against_float64(mods, case, chans, hw, sizes, B, sum_loss):
    rs = np.random.RandomState(B + chans[0])
    w = OW.dggm_weights(chans, 3, seed=303)
    m = mods.DepthGradientInjectionResidual(chans, 3)
    m.load_state_dict(w)
    m.cuda().train()
    feats = [torch.from_numpy(rs.randn(B, c, h, ww).astype(np.float32)).cuda() for c, (h, ww) in zip(chans, sizes)]
    grad = torch.from_numpy(rs.rand(B, 3, *hw).astype(np.float32))
    mask = torch.from_numpy((rs.rand(B, 1, *hw) < 0.6).astype(np.float32))
    out = m(feats, grad.cuda(), mask.cuda())
    if sum_loss:                    # every dout is a stride-0 expanded tensor
        sum(o.sum() for o in out).backward()
        douts = [torch.ones(o.shape) for o in out]
    else:
        douts = [torch.from_numpy(rs.randn(*o.shape).astype(np.float32)) for o in out]
        torch.autograd.backward(out, [d.cuda() for d in douts])
    ref = GR.dggm_reference(w, grad, mask, douts)
    results = {}
    for name, p in m.named_parameters():
        r, ra, slack = ref[name]
        results[name] = GR.check(p.grad, r, ra, GR.TAU_DGGM, slack)
        results[name]["gate_band_elements"] = int((slack > 0).sum())      # elements with a pixel in the gate band
    _check_all(f"dggm/{case}", results)


# ---------------------------------------------------------------------------------------------------
# f. the composition at the train record's shape against oracle autograd
# ---------------------------------------------------------------------------------------------------
def test_depth_guidance_training_gradients_at_the_train_record_shape(mods):
    """DepthGuidance in .train() at 480x640, batch 8, Swin-T channels (bench.py's ``train`` record) against torch autograd
    through the CPU oracle: the DSAM parameters within relative L2 3e-2 (bf16 operands), the DGGM parameters within 1e-4
    (their gradient depends only on the douts and the gated map, not on the bf16 DSAM branch)."""
    chans, (H, W), B = (96, 192, 384, 768), (480, 640), 8
    w = OW.guidance_weights(seed=701, channels=chans)
    m = mods.DepthGuidance(chans)
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
        bar = 1e-4 if name.startswith("depth_gradient_injection.") else 3e-2
        report(f"backward/guidance-train-480x640-B8/{name}", rel_l2=err, bar=bar)
        if not err < bar:
            bad.append((name, err, bar))
    assert not bad, bad
