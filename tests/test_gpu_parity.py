"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on the same seeded inputs.

Bars (BASELINE.json north_star): integer / boolean / index artefacts bit-exact; floating point within
1e-4 relative where the kernel computes in fp32 (DGGM, gradient features) and within 1e-2 relative where
the tensor-core path uses bf16 operands (DSAM convs, ratio predictor)."""
import os

import numpy as np
import pytest
import torch

import rgbd_b200  # noqa: F401
from rgbd_b200 import synthetic
from oracle import hotpath as O
from oracle import weights as OW
from oracle.make_golden import decompose_cases, load_wiring
from rgbd_b200 import _lib as _rgbd_lib

pytestmark = pytest.mark.gpu

BF16_TOL = 1e-2
FP32_TOL = 1e-4


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


def rel_err(a: torch.Tensor, b: torch.Tensor) -> float:
    a = a.double().cpu()
    b = b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    a = a.double().cpu()
    b = b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------
# K0 gradient features: bit-exact
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["nyu", "uniform", "constant", "two_valued", "all_invalid"])
@pytest.mark.parametrize("hw", [(60, 84), (480, 640), (33, 31)])
def test_gradient_features_bit_exact(fn, kind, hw):
    ds = [synthetic.synth_rgbd_u8(40 + j, hw[0], hw[1], kind)[1] for j in range(3)]
    d = torch.from_numpy(np.stack(ds)).cuda()
    for inp in (d, d.float()):
        norm, vm = fn.gradient_features(inp)
        for j in range(3):
            rn, _, _, rv = O.gradient_features(ds[j])
            np.testing.assert_array_equal(vm[j, 0].cpu().numpy(), rv)
            for r in range(3):
                np.testing.assert_array_equal(norm[j, r].cpu().numpy(), rn)


def test_gradient_features_into_pixel_values_view(fn):
    ds = [synthetic.synth_rgbd_u8(3 + j, 64, 96, "nyu")[1] for j in range(2)]
    pv = torch.zeros(2, 10, 64, 96, device="cuda")
    fn.gradient_features(torch.from_numpy(np.stack(ds)).cuda(), norm_out=pv[:, 6:9], vmask_out=pv[:, 9:10])
    for j in range(2):
        rn, _, _, rv = O.gradient_features(ds[j])
        np.testing.assert_array_equal(pv[j, 8].cpu().numpy(), rn)
        np.testing.assert_array_equal(pv[j, 9].cpu().numpy(), rv)
    assert float(pv[:, :6].abs().max()) == 0.0


def test_pack_pixel_values_matches_huggingface_processor_golden(fn, golden_dir):
    """Device front-end against the outputs of the real HF processor + reference mapper (tests/golden/frontend.npz)."""
    g = np.load(os.path.join(golden_dir, "frontend.npz"))
    for j in range(3):
        rgb = torch.from_numpy(g[f"f{j}.rgb"])[None].cuda().contiguous()
        depth = torch.from_numpy(g[f"f{j}.depth"])[None].cuda().contiguous()
        pv = fn.pack_pixel_values(rgb, depth)
        assert torch.equal(pv[0].cpu(), torch.from_numpy(g[f"f{j}.pixel_values"])), j


def test_pack_pixel_values_front_end_bit_exact(fn):
    """uint8 colour + uint8 depth -> the whole 10-channel model input (DL:386-425), bit-exact with the numpy/HF path."""
    rgbs, ds, refs = [], [], []
    for j, kind in enumerate(["nyu", "uniform", "all_invalid"]):
        rgb, d = synthetic.synth_rgbd_u8(200 + j, 60, 84, kind)
        rgbs.append(rgb)
        ds.append(d)
        refs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = fn.pack_pixel_values(torch.from_numpy(np.stack(rgbs)).cuda(), torch.from_numpy(np.stack(ds)).cuda())
    np.testing.assert_array_equal(pv.cpu().numpy(), np.stack(refs))


# ---------------------------------------------------------------------------------------------------
# K2 depth decomposition: bit-exact histogram / modes / windows / masks / pooled masks
# ---------------------------------------------------------------------------------------------------
def _check_decomposition(fn, grays, ratios, levels):
    """grays: list of (H,W) float32 arrays of one shape."""
    g = torch.from_numpy(np.stack(grays)).cuda()
    r = torch.tensor(ratios, dtype=torch.float32).cuda()
    dec = fn.depth_decompose(r, levels, gray=g, debug=True)
    H, W = grays[0].shape
    for b, (gray, ratio) in enumerate(zip(grays, ratios)):
        ref = O.depth_decompose(gray, ratio)
        np.testing.assert_array_equal(dec.hist[b].cpu().numpy(), ref["hist"], err_msg=f"hist img {b}")
        np.testing.assert_array_equal(dec.edges[b].cpu().numpy(), ref["edges"], err_msg=f"edges img {b}")
        m = len(ref["centres"])
        assert int(dec.n_modes[b]) == m
        np.testing.assert_array_equal(dec.peak_bins[b, :m].cpu().numpy(), np.array(ref["peak_bins"], dtype=np.int32))
        np.testing.assert_array_equal(dec.centres[b, :m].cpu().numpy(), np.array(ref["centres"], dtype=np.float32))
        wins = np.array(ref["windows"], dtype=np.float32).reshape(-1, 2)
        np.testing.assert_array_equal(dec.windows[b, :m].cpu().numpy(), wins)
        codes = dec.codes[b].cpu().numpy()
        ref_codes = np.zeros((H, W), dtype=np.uint8)
        if m > 0:
            for t, mk in enumerate(ref["masks"]):
                ref_codes |= (mk.astype(np.uint8) << t)
        np.testing.assert_array_equal(codes, ref_codes, err_msg=f"codes img {b}")
        for lvl, (h, w) in enumerate(levels):
            ref_p = np.zeros((h, w), dtype=np.uint8)
            if m > 0:
                for t, mk in enumerate(ref["masks"]):
                    ref_p |= (O.adaptive_max_pool_mask(mk, (h, w)).astype(np.uint8) << t)
            np.testing.assert_array_equal(dec.pooled[lvl][b].cpu().numpy(), ref_p, err_msg=f"pooled L{lvl} img {b}")


def test_decompose_edge_cases_bit_exact(fn):
    for name, gray, ratio in decompose_cases(synthetic):
        H, W = gray.shape
        levels = [(H // 4, W // 4), (H // 8, W // 8), (max(H // 16, 1), max(W // 16, 1)), (7, 5)]
        _check_decomposition(fn, [gray], [ratio], levels)


def test_to_grayscale_method_mirrors_the_reference(golden_dir):
    """CustomMask2FormerPixelLevelModule.to_grayscale (CM:392-502): tensor and ndarray layouts, dtypes, errors."""
    from rgbd_b200 import pixel_level
    plm = pixel_level.CustomMask2FormerPixelLevelModule(pixel_level.swin_tiny_mask2former_config(num_labels=4), version="0.0.0")
    g = np.load(os.path.join(golden_dir, "gray.npz"))
    rs = np.random.RandomState(0)
    x = rs.randn(3, 37, 53).astype(np.float32)
    ref = O.to_grayscale(x)
    t = torch.from_numpy(x).cuda()
    assert torch.equal(plm.to_grayscale(t).cpu(), torch.from_numpy(ref)[None])                       # (3,H,W) -> (1,H,W)
    assert torch.equal(plm.to_grayscale(t.permute(1, 2, 0)).cpu(), torch.from_numpy(ref)[None])      # (H,W,3)
    b = torch.stack([t, t.flip(1)])
    gb = plm.to_grayscale(b)
    assert gb.shape == (2, 1, 37, 53) and torch.equal(gb[0, 0].cpu(), torch.from_numpy(ref))
    pv = torch.randn(2, 10, 24, 32, device="cuda")                                                   # strided view of pixel_values
    assert torch.equal(plm.to_grayscale(pv[:, 3:6])[1, 0].cpu(), torch.from_numpy(O.to_grayscale(pv[1, 3:6].cpu().numpy())))
    one = torch.randn(1, 5, 7, device="cuda")
    assert plm.to_grayscale(one) is one and plm.to_grayscale(one.permute(1, 2, 0)).shape == (1, 5, 7)
    # ndarray branch keeps the input dtype (uint8 truncation included), like the reference
    u8 = rs.randint(0, 256, (9, 11, 3)).astype(np.uint8)
    want = (0.299 * u8[:, :, 0] + 0.587 * u8[:, :, 1] + 0.114 * u8[:, :, 2]).astype(np.uint8)
    assert np.array_equal(plm.to_grayscale(u8), want) and plm.to_grayscale(u8).dtype == np.uint8
    assert np.array_equal(plm.to_grayscale(np.ascontiguousarray(u8.transpose(2, 0, 1))), want)
    assert plm.to_grayscale(u8[:, :, :1]).shape == (9, 11) and plm.to_grayscale(u8[:, :, 0]).shape == (9, 11)
    if "ref0" in g.files and "in0" in g.files:
        assert np.array_equal(plm.to_grayscale(torch.from_numpy(g["in0"]).cuda()).cpu().numpy()[0], g["ref0"])
    # other tensor dtypes: float32 arithmetic, result cast back (CM:499); uint8 equals the reference's own arithmetic (torch
    # promotes python-float x uint8 to float32 and truncates on the cast), float64 agrees to float32 precision
    tu8 = torch.from_numpy(np.ascontiguousarray(u8.transpose(2, 0, 1)))
    ref_u8 = (0.299 * tu8[0] + 0.587 * tu8[1] + 0.114 * tu8[2]).unsqueeze(0).to(torch.uint8)
    got_u8 = plm.to_grayscale(tu8.cuda())
    assert got_u8.dtype == torch.uint8 and torch.equal(got_u8.cpu(), ref_u8)
    t64 = torch.randn(2, 3, 6, 8, dtype=torch.float64)
    ref64 = (0.299 * t64[:, 0] + 0.587 * t64[:, 1] + 0.114 * t64[:, 2]).unsqueeze(1)
    got64 = plm.to_grayscale(t64.cuda())
    assert got64.dtype == torch.float64 and got64.shape == (2, 1, 6, 8) and torch.allclose(got64.cpu(), ref64, rtol=1e-6, atol=1e-6)
    with pytest.raises(TypeError):
        plm.to_grayscale([[1.0]])
    with pytest.raises(ValueError):
        plm.to_grayscale(np.zeros((2, 5, 7)))
    with pytest.raises(ValueError):
        plm.to_grayscale(torch.zeros(2, 5, 7, device="cuda"))
    with pytest.raises(ValueError):
        plm.to_grayscale(torch.zeros(5, device="cuda"))


def test_dsam_helper_methods_match_reference_goldens(mods, golden_dir):
    """DSAModule._calculate_depth_histogram / _select_depth_distribution_modes / _define_depth_interval_windows /
    _generate_depth_region_masks (CM:701-798) as methods, on the reference's own outputs (tests/golden/decompose.npz)."""
    g = np.load(os.path.join(golden_dir, "decompose.npz"))
    m = mods.DSAModule(8, 16, 3).cuda()
    for name, gray, ratio in decompose_cases(synthetic):
        if not np.isfinite(gray).any():                  # numpy raises inside the reference for this case
            continue
        hist, edges = m._calculate_depth_histogram(gray)
        assert np.array_equal(hist, g[f"{name}.hist"]) and np.array_equal(edges, g[f"{name}.edges"])
        modes = m._select_depth_distribution_modes(hist, edges, num_modes=3)
        ref_modes = g[f"{name}.modes"]
        assert len(modes) == len(ref_modes) and all(np.float32(a) == np.float32(b) for a, b in zip(modes, ref_modes)), name
        wins = m._define_depth_interval_windows(modes, window_size_ratio=ratio)
        ref_w = g[f"{name}.windows"]
        assert len(wins) == len(ref_w)
        for (lo, hi), (rl, rh) in zip(wins, ref_w):
            assert np.float32(lo) == rl and np.float32(hi) == rh, name
        if modes:
            masks = m._generate_depth_region_masks(gray, wins)
            ref_masks = np.unpackbits(g[f"{name}.masks"])[:(len(wins) + 1) * gray.size].reshape(len(wins) + 1, *gray.shape).astype(bool)
            assert len(masks) == len(wins) + 1
            for a, b in zip(masks, ref_masks):
                assert a.dtype == bool and np.array_equal(a, b), name
    # fewer modes on request, a stricter prominence threshold, and no windows at all
    name, gray, ratio = decompose_cases(synthetic)[0]
    hist, edges = g[f"{name}.hist"], g[f"{name}.edges"]
    assert m._select_depth_distribution_modes(hist, edges, num_modes=1) == [m._select_depth_distribution_modes(hist, edges)[0]]
    strict = m._select_depth_distribution_modes(hist, edges, num_modes=3, prominence_threshold=0.9)
    want = O.select_depth_modes(hist, edges, 3, 0.9)[1]
    assert [np.float32(v) for v in strict] == [np.float32(v) for v in want]
    rest = m._generate_depth_region_masks(gray, [])
    assert len(rest) == 1 and rest[0].all()


def test_decompose_full_size_batch_bit_exact(fn):
    grays, ratios = [], []
    for j, kind in enumerate(["nyu", "nyu", "nyu", "uniform", "constant", "two_valued"]):
        _, d = synthetic.synth_rgbd_u8(100 + j, 480, 640, kind)
        grays.append(O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2))))
        ratios.append([0.013, 0.21, 0.5, 0.1, 0.3, 0.07][j])
    _check_decomposition(fn, grays, ratios, [(120, 160), (60, 80), (30, 40)])


def test_gray_from_depth3_bit_exact(fn):
    rs = np.random.RandomState(11)
    d3 = (rs.randn(2, 3, 40, 56) * 1.3).astype(np.float32)
    pv = torch.zeros(2, 10, 40, 56, device="cuda")
    pv[:, 3:6] = torch.from_numpy(d3).cuda()
    dec = fn.depth_decompose(torch.tensor([0.1, 0.2], device="cuda"), [(10, 14)], depth3=pv[:, 3:6])
    for b in range(2):
        np.testing.assert_array_equal(dec.gray[b].cpu().numpy(), O.to_grayscale(d3[b]))


# ---------------------------------------------------------------------------------------------------
# K1 DGGM forward / K1b parameter gradients
# ---------------------------------------------------------------------------------------------------
def _dggm_case(chans, hw, sizes, B, seed):
    rs = np.random.RandomState(seed)
    feats = [torch.from_numpy(rs.randn(B, c, h, w).astype(np.float32)) for c, (h, w) in zip(chans, sizes)]
    grad = torch.from_numpy(rs.rand(B, 3, *hw).astype(np.float32))
    mask = torch.from_numpy((rs.rand(B, 1, *hw) < 0.6).astype(np.float32))
    return feats, grad, mask


@pytest.mark.parametrize("chans,hw,sizes,B", [
    ([4, 8, 12, 16], (64, 96), [(16, 24), (8, 12), (4, 6), (2, 3)], 2),
    ([4, 8, 12, 16], (50, 70), [(13, 18), (7, 9), (4, 5), (2, 3)], 2),
    ([96, 192, 384, 768], (480, 640), [(120, 160), (60, 80), (30, 40), (15, 20)], 2),
    ([128, 256, 512, 1024], (96, 128), [(24, 32), (12, 16), (6, 8), (3, 4)], 1),
])
def test_dggm_forward(mods, chans, hw, sizes, B):
    feats, grad, mask = _dggm_case(chans, hw, sizes, B, 9)
    w = OW.dggm_weights(chans, 3, seed=300)
    m = mods.DepthGradientInjectionResidual(chans, 3)
    m.load_state_dict(w)
    m.cuda().eval()
    ref = O.dggm_forward(w, feats, grad, mask)
    pv = torch.zeros(B, 10, *hw, device="cuda")       # exercise the strided pixel_values views
    pv[:, 6:9] = grad.cuda()
    pv[:, 9:10] = mask.cuda()
    with torch.no_grad():
        out = m([f.cuda() for f in feats], pv[:, 6:9], pv[:, 9:10])
        fused = m.forward_fused_sum([f.cuda() for f in feats], [(2 * f).cuda() for f in feats], pv[:, 6:9], pv[:, 9:10])
    for i in range(4):
        assert rel_err(out[i], ref[i]) < FP32_TOL
        assert rel_err(fused[i], 2 * feats[i] + ref[i]) < FP32_TOL
    # None -> passthrough, wrong scale count -> AssertionError (CM:1218-1219, 1263-1265)
    same = m([f.cuda() for f in feats], None, pv[:, 9:10])
    assert all(torch.equal(a.cpu(), b) for a, b in zip(same, feats))
    with pytest.raises(AssertionError):
        m([feats[0].cuda()], pv[:, 6:9], pv[:, 9:10])


def test_dggm_param_gradients(mods):
    chans, hw, sizes = [8, 16, 24, 32], (64, 96), [(16, 24), (8, 12), (4, 6), (2, 3)]
    feats, grad, mask = _dggm_case(chans, hw, sizes, 2, 21)
    w = OW.dggm_weights(chans, 3, seed=301)
    m = mods.DepthGradientInjectionResidual(chans, 3)
    m.load_state_dict(w)
    m.cuda().train()
    rs = np.random.RandomState(5)
    douts = [torch.from_numpy(rs.randn(*f.shape).astype(np.float32)) for f in feats]
    out = m([f.cuda() for f in feats], grad.cuda(), mask.cuda())
    loss = sum((o * d.cuda()).sum() for o, d in zip(out, douts))
    loss.backward()
    # oracle gradients by torch autograd on the CPU restatement
    wr = {k: v.clone().requires_grad_(True) for k, v in w.items()}
    ref = O.dggm_forward(wr, feats, grad, mask)
    sum((o * d).sum() for o, d in zip(ref, douts)).backward()
    for i in range(4):
        gw = m.depth_enhancement_layers[i][0].weight.grad
        gb = m.depth_enhancement_layers[i][0].bias.grad
        assert rel_err(gw, wr[f"depth_enhancement_layers.{i}.0.weight"].grad) < 1e-3
        assert rel_err(gb, wr[f"depth_enhancement_layers.{i}.0.bias"].grad) < 1e-3


# ---------------------------------------------------------------------------------------------------
# tensor-core implicit GEMM (tcgen05) against a float64 reference of the same bf16 operands
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kb,c,n,hw", [(64, 128, 64, (4, 128)), (64, 64, 256, (8, 64)), (32, 96, 192, (16, 24)),
                                       (64, 192, 64, (5, 50))])
def test_conv_gemm_1x1(fn, kb, c, n, hw):
    rs = np.random.RandomState(1)
    B, (H, W) = 2, hw
    a = torch.from_numpy(rs.randn(B, H, W, c).astype(np.float32)).cuda().to(torch.bfloat16)
    w = torch.from_numpy((rs.randn(n, c) / np.sqrt(c)).astype(np.float32)).cuda().to(torch.bfloat16)
    shift = torch.from_numpy(rs.randn(n).astype(np.float32)).cuda()
    scale = torch.from_numpy(rs.uniform(0.5, 1.5, n).astype(np.float32)).cuda()
    slices = torch.tensor([(kb * i, 0, 0, 0) for i in range(c // kb)], dtype=torch.int32).cuda()
    from rgbd_b200.modules import _best_box
    out = torch.zeros(B, H, W, n, device="cuda", dtype=torch.bfloat16)
    fn.conv_gemm(a, (B, H, W, c), 1, w, slices, kb, B, (H, W), _best_box(H, W), n, shift, scale=scale, act=1, out=out)
    ref = torch.relu((a.double() @ w.double().T) * scale.double() + shift.double())
    assert rel_err(out.double(), ref) < 8e-3            # one bf16 rounding of the output
    out32 = torch.zeros(B, n, H, W, device="cuda")
    res = torch.from_numpy(rs.randn(B, n, H, W).astype(np.float32)).cuda()
    fn.conv_gemm(a, (B, H, W, c), 1, w, slices, kb, B, (H, W), _best_box(H, W), n, shift, epi_mode=1, out=out32,
                 residual=res)
    ref32 = (a.double() @ w.double().T + shift.double()).permute(0, 3, 1, 2) + res.double()
    assert rel_err(out32, ref32) < 1e-4


def test_conv_gemm_3x3_pool(fn):
    rs = np.random.RandomState(2)
    B, H, W, c, n = 2, 16, 64, 128, 256
    a = torch.from_numpy(rs.randn(B, H, W, c).astype(np.float32)).cuda().to(torch.bfloat16)
    wt = torch.from_numpy((rs.randn(n, c, 3, 3) / np.sqrt(9 * c)).astype(np.float32)).cuda().to(torch.bfloat16)
    w = wt.permute(0, 2, 3, 1).reshape(n, 9 * c).contiguous()
    shift = torch.from_numpy(rs.randn(n).astype(np.float32) * 0.1).cuda()
    slices = torch.tensor([(64 * cb, dx - 1, dy - 1, 0) for dy in range(3) for dx in range(3) for cb in range(c // 64)],
                          dtype=torch.int32).cuda()
    pool = torch.zeros(B, 16, n, device="cuda", dtype=torch.int64)        # fixed-point cell sums
    from rgbd_b200.modules import _best_box
    fn.conv_gemm(a, (B, H, W, c), 1, w, slices, 64, B, (H, W), _best_box(H, W), n, shift, act=1, epi_mode=2, pool=pool,
                 cells=(4, 4), tile_order=1)
    y = torch.relu(torch.nn.functional.conv2d(a.double().permute(0, 3, 1, 2), wt.double(), shift.double(), padding=1))
    ref = torch.nn.functional.adaptive_avg_pool2d(y, 4) * (H // 4) * (W // 4)       # sums per cell
    ref = ref.permute(0, 2, 3, 1).reshape(B, 16, n)
    assert rel_err(pool.double() / fn.POOL_FIXED_ONE, ref) < 1e-4


@pytest.mark.parametrize("c,n,hw", [(128, 256, (8, 256)), (64, 128, (12, 200)), (192, 64, (4, 128))])
def test_conv3x3_a_reuse_path(fn, c, n, hw):
    """3x3 conv whose 130-pixel smem tile serves the three dx taps (row-shifted UMMA descriptors)."""
    rs = np.random.RandomState(4)
    B, (H, W) = 2, hw
    a = torch.from_numpy(rs.randn(B, H, W, c).astype(np.float32)).cuda().to(torch.bfloat16)
    wt = torch.from_numpy((rs.randn(n, c, 3, 3) / np.sqrt(9 * c)).astype(np.float32)).cuda().to(torch.bfloat16)
    w = wt.permute(0, 2, 3, 1).reshape(n, 9 * c).contiguous()
    shift = torch.from_numpy(rs.randn(n).astype(np.float32) * 0.1).cuda()
    y = torch.relu(torch.nn.functional.conv2d(a.double().permute(0, 3, 1, 2), wt.double(), shift.double(), padding=1))
    pool = torch.zeros(B, 16, n, device="cuda", dtype=torch.int64)        # fixed-point cell sums
    fn.conv_gemm(a, (B, H, W, c), 1, w, None, 64, B, (H, W), (128, 1), n, shift, act=1, epi_mode=2, pool=pool,
                 cells=(4, 4), tile_order=1, conv3x3_reuse=True)
    ref = (torch.nn.functional.adaptive_avg_pool2d(y, 4) * (H // 4) * (W // 4)).permute(0, 2, 3, 1).reshape(B, 16, n)
    assert rel_err(pool.double() / fn.POOL_FIXED_ONE, ref) < 1e-4
    out = torch.zeros(B, H, W, n, device="cuda", dtype=torch.bfloat16)
    fn.conv_gemm(a, (B, H, W, c), 1, w, None, 64, B, (H, W), (128, 1), n, shift, act=1, out=out, conv3x3_reuse=True)
    assert rel_err(out.double(), y.permute(0, 2, 3, 1)) < 8e-3


@pytest.mark.parametrize("hw", [(4, 128), (9, 50), (16, 200)])
def test_ratio_chain_fused(fn, hw):
    """Three chained GEMMs with TMEM-resident intermediates vs float64 math on the same bf16 operands."""
    rs = np.random.RandomState(3)
    B, (H, W) = 2, hw
    bf = torch.bfloat16
    x1 = torch.from_numpy(np.abs(rs.randn(B, H, W, 192)).astype(np.float32)).cuda().to(bf)
    w2 = torch.from_numpy((rs.randn(128, 192) / np.sqrt(192)).astype(np.float32)).cuda().to(bf)
    w3 = torch.from_numpy((rs.randn(64, 128) / np.sqrt(128)).astype(np.float32)).cuda().to(bf)
    w4 = torch.from_numpy((rs.randn(128, 64) / np.sqrt(64)).astype(np.float32)).cuda().to(bf)
    sc2 = torch.from_numpy(rs.uniform(0.5, 1.5, 128).astype(np.float32)).cuda()
    sh2, sh4 = (torch.from_numpy((rs.randn(128) * 0.2).astype(np.float32)).cuda() for _ in range(2))
    sh3 = torch.from_numpy((rs.randn(64) * 0.2).astype(np.float32)).cuda()
    out = torch.zeros(B, H, W, 128, device="cuda", dtype=bf)
    from rgbd_b200.modules import _best_box
    w2 = (w2.float() * sc2[:, None]).to(bf)          # the BN scale is folded into the weights
    fn.ratio_chain(x1, w2, w3, w4, sh2, sh3, sh4, out, _best_box(H, W))
    f = torch.relu(x1.double() @ w2.double().T + sh2.double()).to(bf).double()   # kernel rounds f to bf16
    a = torch.relu(f @ w3.double().T + sh3.double()).to(bf).double()
    ref = f * torch.sigmoid(a @ w4.double().T + sh4.double())
    assert rel_err(out.double(), ref) < 8e-3


def test_ratio_predictor_fused_chain_matches_unfused(mods):
    w = OW.ratio_weights(seed=500)
    frames = []
    for j in range(2):
        _, d = synthetic.synth_rgbd_u8(60 + j, 48, 64, "nyu")
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    x = torch.from_numpy(np.stack(frames)).cuda()
    res = []
    for fused in (True, False):
        m = mods.EnhancedDepthImageRatioPredictor(3)
        m.use_fused_front = False
        m.use_fused_chain = fused
        m.load_state_dict(w)
        m.cuda().eval()
        with torch.no_grad():
            res.append(m(x).cpu())
    assert float(((res[0] - res[1]).abs() / res[1]).max()) < 2e-3


@pytest.mark.parametrize("B,hw", [(1, (4, 128)), (2, (48, 64)), (3, (20, 36)), (5, (8, 256)), (2, (12, 640)), (1, (8, 384))])
def test_ratio_front_fused_matches_stem_gemm_plus_chain(mods, fn, B, hw):
    """ratio_front_kernel (stem GEMM + chain, two tile chains per CTA pair, all intermediates in tensor memory) against
    the two-kernel path on the same packed operands: identical bf16 rounding points, so the gated 128-channel map must
    agree to bf16 resolution; odd tile counts leave the last pair half empty."""
    w = OW.ratio_weights(seed=501)
    H, W = hw
    rs = np.random.RandomState(B)
    x = torch.from_numpy(rs.uniform(-2, 2, (B, 3, H, W)).astype(np.float32)).cuda()
    outs, ratios = [], []
    for fused in (True, False):
        m = mods.EnhancedDepthImageRatioPredictor(3)
        m.use_fused_front = fused
        m.load_state_dict(w)
        m.cuda().eval()
        with torch.no_grad():
            ratios.append(m(x).cpu())
        outs.append(next(iter(m._ws.values()))["x4"].float().cpu())
    assert outs[0].shape == (B, H, W, 128)
    # widths tiled by 128x1 boxes read the depth image through sliding-window tensor maps (compact operand)
    assert mods.EnhancedDepthImageRatioPredictor(3)._compact(H, W) == (mods._best_box(H, W) == (128, 1) and W % 2 == 0)
    assert rel_err(outs[0], outs[1]) < 1e-2, rel_err(outs[0], outs[1])
    assert rel_l2(outs[0], outs[1]) < 2e-3
    assert float(((ratios[0] - ratios[1]).abs() / ratios[1]).max()) < 2e-3


# ---------------------------------------------------------------------------------------------------
# E-DSAM: DSAModule / ratio predictor / v0.4.0 wiring
# ---------------------------------------------------------------------------------------------------
def _gray_for(j, kind, dhw):
    _, d = synthetic.synth_rgbd_u8(20 + j, dhw[0], dhw[1], kind)
    return O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))


@pytest.mark.parametrize("ci,co,hw,dhw", [(8, 16, (24, 32), (96, 128)), (8, 8, (24, 32), (96, 128)),
                                          (8, 24, (15, 20), (60, 80)), (96, 192, (30, 40), (120, 160)),
                                          (64, 64, (12, 20), (48, 80))])
def test_dsam_module(mods, ci, co, hw, dhw):
    w = OW.dsam_weights(ci, co, seed=100 + ci + co)
    m = mods.DSAModule(ci, co, 3)
    m.load_state_dict(w)
    m.cuda().eval()
    feat = torch.from_numpy(np.random.RandomState(5).randn(2, ci, *hw).astype(np.float32))
    for j, kind in enumerate(["nyu", "constant", "two_valued"]):
        gray = _gray_for(j, kind, dhw)
        with torch.no_grad():
            y = m(feat.cuda(), torch.from_numpy(gray)[None].cuda(), 0.3)
            y_np = m(feat.cuda(), gray, 0.3)                      # ndarray depth input (exp6_dsam.py:57-60)
        ref = torch.cat([O.dsam_forward(w, feat[b:b + 1], gray, 0.3) for b in range(2)])
        assert y.shape == ref.shape
        assert rel_err(y, ref) < BF16_TOL, (kind, rel_err(y, ref))
        assert rel_l2(y, ref) < BF16_TOL
        assert torch.equal(y, y_np)
    with pytest.raises(TypeError):
        m(feat.cuda(), [[0.0]], 0.3)


@pytest.mark.parametrize("ci,co,hw,dhw", [(96, 192, (30, 40), (120, 160)), (64, 128, (15, 21), (60, 84)),
                                          (192, 384, (31, 17), (124, 68)), (128, 96, (9, 130), (36, 520))])
def test_dsam_shared_memory_masking_matches_premasked_layout(mods, monkeypatch, ci, co, hw, dhw):
    """dsam_fwd_kernel (region masks applied to the tile in shared memory) against the five-fold pre-masked operand
    + generic GEMM, and both against the oracle; odd sizes exercise the parity-plane edges and half-empty pairs."""
    w = OW.dsam_weights(ci, co, seed=300 + ci + co)
    m = mods.DSAModule(ci, co, 3)
    m.load_state_dict(w)
    m.cuda().eval()
    feat = torch.from_numpy(np.random.RandomState(6).randn(3, ci, *hw).astype(np.float32))
    for j, kind in enumerate(["nyu", "two_valued"]):
        gray = _gray_for(j, kind, dhw)
        outs = []
        for premasked in (False, True):
            monkeypatch.setattr(mods, "_PREMASKED", premasked)
            with torch.no_grad():
                outs.append(m(feat.cuda(), torch.from_numpy(gray)[None].cuda(), 0.25))
        ref = torch.cat([O.dsam_forward(w, feat[b:b + 1], gray, 0.25) for b in range(3)])
        assert rel_err(outs[0], ref) < BF16_TOL and rel_err(outs[1], ref) < BF16_TOL
        assert rel_err(outs[0], outs[1]) < 1e-5, rel_err(outs[0], outs[1])     # same bf16 operands, other K order


@pytest.mark.parametrize("ci,co,hw,dhw", [(8, 16, (24, 32), (96, 128)), (96, 192, (30, 40), (120, 160)),
                                          (64, 64, (12, 20), (48, 80)), (40, 72, (15, 21), (60, 84))])
def test_dsam_module_fp32_precision_mode(mods, ci, co, hw, dhw):
    """Split-precision tensor-core path (x_hi W_hi + x_lo W_hi + x_hi W_lo): inside the fp32 bar of 1e-4."""
    w = OW.dsam_weights(ci, co, seed=100 + ci + co)
    m = mods.DSAModule(ci, co, 3)
    m.precision = "fp32"
    m.load_state_dict(w)
    m.cuda().eval()
    feat = torch.from_numpy(np.random.RandomState(5).randn(2, ci, *hw).astype(np.float32))
    for j, kind in enumerate(["nyu", "constant", "two_valued"]):
        gray = _gray_for(j, kind, dhw)
        with torch.no_grad():
            y = m(feat.cuda(), torch.from_numpy(gray)[None].cuda(), 0.3)
        ref = torch.cat([O.dsam_forward(w, feat[b:b + 1], gray, 0.3) for b in range(2)])
        assert rel_err(y, ref) < FP32_TOL, (kind, rel_err(y, ref))


def test_depth_guidance_fp32_precision_mode(mods, golden_dir):
    """fp32 bar of the north star (1e-4 relative) on the fused features handed to the pixel decoder."""
    g = load_wiring(golden_dir, "wiring.npz")
    m = mods.DepthGuidance((96, 192, 384, 768), precision="fp32")
    m.load_state_dict(OW.guidance_weights(seed=700))
    m.cuda().eval()
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs)).cuda()
    feats = [torch.from_numpy(g[f"feat{i}"]).cuda() for i in range(4)]
    with torch.no_grad():
        fused = m(pv, feats, ratios=torch.from_numpy(g["ratios"]).cuda())
    for i in range(4):
        ref = torch.from_numpy(g[f"fused{i}"])
        assert rel_err(fused[i], ref) < FP32_TOL, (i, rel_err(fused[i], ref))


@pytest.mark.parametrize("hw", [(48, 64), (96, 160)])
def test_ratio_predictor(mods, hw):
    w = OW.ratio_weights(seed=500)
    m = mods.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(w)
    m.cuda().eval()
    frames = []
    for j in range(3):
        _, d = synthetic.synth_rgbd_u8(60 + j, hw[0], hw[1], "nyu")
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    x = torch.from_numpy(np.stack(frames))
    ref = O.ratio_predictor_forward(w, x)
    with torch.no_grad():
        r = m(x.cuda())
    assert r.shape == (3, 1)
    assert ((r >= 0.01) & (r <= 0.5)).all()
    assert float(((r.cpu() - ref).abs() / ref.abs()).max()) < BF16_TOL
    with pytest.raises(AssertionError):
        m(x.cuda()[:, :2])


def test_depth_guidance_wiring(mods, golden_dir):
    g = load_wiring(golden_dir, "wiring.npz")
    w = OW.guidance_weights(seed=700)
    m = mods.DepthGuidance((96, 192, 384, 768))
    missing = m.load_state_dict(w, strict=True)
    m.cuda().eval()
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs)).cuda()
    feats = [torch.from_numpy(g[f"feat{i}"]).cuda() for i in range(4)]
    ref_ratio = torch.from_numpy(g["ratios"])
    with torch.no_grad():
        ratio = m.ratio_predictor(pv[:, 3:6])
        fused_given = m(pv, feats, ratios=ref_ratio.cuda())      # stage (i)/(iii): oracle-supplied ratio
        fused_own = m(pv, feats)                                  # end to end with our bf16 ratio
    assert float(((ratio.cpu() - ref_ratio).abs() / ref_ratio).max()) < BF16_TOL
    for i in range(4):
        ref = torch.from_numpy(g[f"fused{i}"])
        assert rel_err(fused_given[i], ref) < BF16_TOL, (i, rel_err(fused_given[i], ref))
        assert rel_l2(fused_given[i], ref) < BF16_TOL
        # with our own ratio a few boundary pixels of the region masks may flip (SURVEY H5)
        assert rel_l2(fused_own[i], ref) < 3 * BF16_TOL


# ---------------------------------------------------------------------------------------------------
# whole model: HF Mask2Former (stock Swin / pixel decoder / transformer decoder) + CUDA depth guidance
# ---------------------------------------------------------------------------------------------------
def test_whole_model_logits_match_cpu_oracle_model(mods):
    """BASELINE configs[0] in miniature: the v0.4.0 model on one synthetic RGB-D frame, GPU (CUDA hot path)
    against the same weights on CPU with the oracle hot path (reference predictor path, SURVEY section 3.3)."""
    import copy
    from rgbd_b200 import pixel_level
    torch.manual_seed(0)
    cfg = pixel_level.swin_tiny_mask2former_config(num_labels=8)
    model = pixel_level.build_rgbd_mask2former(cfg).eval()
    w = OW.guidance_weights(seed=700)
    plm = model.model.pixel_level_module
    missing = plm.load_state_dict(w, strict=False)
    assert not missing.unexpected_keys
    # every parameter is initialised (the pixel decoder's raw ``level_embed`` used to stay uninitialised memory)
    assert float(plm.decoder.level_embed.abs().max()) < 10 and all(bool(torch.isfinite(p).all()) for p in model.parameters())
    # a random-init head produces near-uniform class logits -- differences of almost equal numbers, whose RELATIVE error says
    # little; the decisive synthetic model behaves like a trained one (tests/test_gpu_map_parity.py)
    from rgbd_b200 import synthetic_weights as SW
    SW.make_decisive(model)
    H, W = 128, 160
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(90 + j, H, W, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))

    cpu_model = copy.deepcopy(model)
    cpu_plm = cpu_model.model.pixel_level_module

    def oracle_forward(pixel_values, output_hidden_states=False):
        feats = cpu_plm.encoder(pixel_values[:, 0:3]).feature_maps
        fused, _ = O.depth_guidance_forward(w, pixel_values, list(feats))
        dec = cpu_plm.decoder(fused, output_hidden_states=output_hidden_states)
        from transformers.models.mask2former.modeling_mask2former import Mask2FormerPixelLevelModuleOutput
        return Mask2FormerPixelLevelModuleOutput(encoder_last_hidden_state=fused[-1], encoder_hidden_states=None,
                                                 decoder_last_hidden_state=dec.mask_features,
                                                 decoder_hidden_states=dec.multi_scale_features)
    cpu_plm.forward = oracle_forward
    with torch.no_grad():
        ref = cpu_model(pixel_values=pv)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        out = model.cuda()(pixel_values=pv.cuda())
    for name in ("class_queries_logits", "masks_queries_logits"):
        a, b = getattr(out, name), getattr(ref, name)
        assert a.shape == b.shape
        assert rel_l2(a, b) < 2e-2, (name, rel_l2(a, b))
    # instance masks after the reference's post-processing threshold agree (mask parity, PR:701-703)
    pa = (out.masks_queries_logits.cpu().sigmoid() > 0.5)
    pb = (ref.masks_queries_logits.sigmoid() > 0.5)
    agree = float((pa == pb).float().mean())
    assert agree > 0.995, agree


# ---------------------------------------------------------------------------------------------------
# K3b: DSAM backward (wgrad / dbias / dgrad) and the training-mode cascade against oracle autograd
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ci,co,hw,dhw", [(32, 64, (24, 32), (96, 128)), (96, 192, (30, 40), (120, 160)),
                                          (64, 64, (12, 16), (48, 64)), (40, 72, (15, 20), (60, 80))])
def test_dsam_stage_backward(mods, fn, ci, co, hw, dhw):
    w = OW.dsam_weights(ci, co, seed=200 + ci + co)
    m = mods.DSAModule(ci, co, 3)
    m.load_state_dict(w)
    m.cuda().train()
    rs = np.random.RandomState(6)
    B = 3
    feat = torch.from_numpy(rs.randn(B, ci, *hw).astype(np.float32))
    kinds = ["nyu", "constant", "two_valued"]
    grays = [_gray_for(j, kinds[j], dhw) for j in range(B)]
    ratios = [0.3, 0.2, 0.4]
    dec = fn.depth_decompose(torch.tensor(ratios, device="cuda"), [hw], gray=torch.from_numpy(np.stack(grays)).cuda())
    x = feat.cuda().requires_grad_(True)
    out = m.stage_forward(x, dec.pooled[0], dec.bias_variant)
    dout = torch.from_numpy(rs.randn(*out.shape).astype(np.float32))
    (out * dout.cuda()).sum().backward()
    # oracle: torch autograd through the CPU restatement
    wr = {k: v.clone().requires_grad_(True) for k, v in w.items()}
    xr = feat.clone().requires_grad_(True)
    ref = torch.cat([O.dsam_forward(wr, xr[b:b + 1], grays[b], ratios[b]) for b in range(B)])
    (ref * dout).sum().backward()
    assert rel_l2(out, ref) < BF16_TOL
    assert rel_l2(x.grad, xr.grad) < 2e-2, rel_l2(x.grad, xr.grad)
    for name, p in m.named_parameters():
        g_ref = wr[name].grad
        if g_ref is None:            # region never used by any image: the reference leaves it without gradient
            assert float(p.grad.abs().max()) == 0.0, name
            continue
        assert rel_l2(p.grad, g_ref) < 2e-2, (name, rel_l2(p.grad, g_ref))


def test_depth_guidance_training_gradients(mods, golden_dir):
    """Fine-tuning semantics of CM:324-355: gradients reach all DSAM and DGGM parameters, none reach the encoder
    features or the ratio predictor (SURVEY section 8a row 10)."""
    g = load_wiring(golden_dir, "wiring.npz")
    w = OW.guidance_weights(seed=700)
    m = mods.DepthGuidance((96, 192, 384, 768))
    m.load_state_dict(w)
    m.cuda().train()
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))
    feats = [torch.from_numpy(g[f"feat{i}"]) for i in range(4)]
    ratios = torch.from_numpy(g["ratios"])
    rs = np.random.RandomState(8)
    douts = [torch.from_numpy(rs.randn(*f.shape).astype(np.float32)) for f in feats]
    feats_gpu = [f.cuda().requires_grad_(True) for f in feats]
    out = m(pv.cuda(), feats_gpu, ratios=ratios.cuda())
    sum((o * d.cuda()).sum() for o, d in zip(out, douts)).backward()
    wr = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in w.items()}
    ref, _ = O.depth_guidance_forward(wr, pv, feats, ratios=ratios)
    sum((o * d).sum() for o, d in zip(ref, douts)).backward()
    assert all(f.grad is None for f in feats_gpu)                               # detached (CM:332-333)
    for name, p in m.named_parameters():
        if name.startswith("ratio_predictor."):
            assert p.grad is None, name                                          # consumed via .item() (CM:339)
            continue
        g_ref = wr[name].grad
        assert g_ref is not None and p.grad is not None, name
        assert rel_l2(p.grad, g_ref) < 3e-2, (name, rel_l2(p.grad, g_ref))


# ---------------------------------------------------------------------------------------------------
# other geometries: Swin-B channels (BASELINE configs[4]) and image sizes that do not tile evenly
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chans,hw", [((128, 256, 512, 1024), (96, 128)), ((96, 192, 384, 768), (100, 132)),
                                      ((32, 64, 96, 160), (72, 88))])
def test_depth_guidance_other_geometries(mods, chans, hw):
    H, W = hw
    w = OW.guidance_weights(seed=900, channels=chans)
    m = mods.DepthGuidance(chans)
    m.load_state_dict(w)
    m.cuda().eval()
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(120 + j, H, W, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs))
    rs = np.random.RandomState(1)
    sizes = [(-(-H // s), -(-W // s)) for s in (4, 8, 16, 32)]           # Swin pads: ceil division
    feats = [torch.from_numpy(rs.randn(2, c, h, ww).astype(np.float32)) for c, (h, ww) in zip(chans, sizes)]
    ref, ref_ratio = O.depth_guidance_forward(w, pv, feats)
    with torch.no_grad():
        ratio = m.ratio_predictor(pv.cuda()[:, 3:6])
        out = m(pv.cuda(), [f.cuda() for f in feats], ratios=ref_ratio.cuda())
    assert float(((ratio.cpu() - ref_ratio).abs() / ref_ratio).max()) < BF16_TOL
    for i in range(4):
        assert out[i].shape == ref[i].shape
        assert rel_err(out[i], ref[i]) < BF16_TOL, (i, rel_err(out[i], ref[i]))


def test_hot_path_is_reproducible_run_to_run(mods, fn):
    """The window ratio feeds integer decisions (region codes), so the whole path must be bit-reproducible: the pooled
    sums of the 3x3 conv use fixed-point integer atomics, everything else has a fixed summation order."""
    chans, (H, W), B = (96, 192, 384, 768), (192, 256), 4
    m = mods.DepthGuidance(chans)
    m.load_state_dict(OW.guidance_weights(seed=77, channels=chans))
    m.cuda().eval()
    rgbs, ds = zip(*[synthetic.synth_rgbd_u8(700 + j, H, W, "nyu") for j in range(B)])
    pv = fn.pack_pixel_values(torch.from_numpy(np.stack(rgbs)).cuda(), torch.from_numpy(np.stack(ds)).cuda())
    g = torch.Generator(device="cpu").manual_seed(3)
    feats = [torch.randn(B, c, H // s, W // s, generator=g).cuda() for c, s in zip(chans, (4, 8, 16, 32))]
    runs = []
    for _ in range(3):
        with torch.no_grad():
            r = m.ratio_predictor(pv[:, 3:6]).clone()
            runs.append((r, [o.clone() for o in m(pv, feats)]))
    for r, outs in runs[1:]:
        assert torch.equal(r, runs[0][0])
        assert all(torch.equal(a, b) for a, b in zip(outs, runs[0][1]))


@pytest.mark.parametrize("chans,hw", [((96, 192, 384, 768), (192, 256)), ((32, 72, 96, 160), (72, 88)),
                                      ((128, 256, 512, 1024), (100, 132))])
def test_stage_operands_emitted_by_the_previous_epilogue_are_bit_identical(mods, fn, monkeypatch, chans, hw):
    """Inference cascade: stage k's epilogue writes stage k+1's packed bf16 operand (unmasked single copy or the five-fold
    pre-masked layout).  It must be exactly what the pack kernel builds from the fp32 result, so every output is
    bit-identical with the fusion switched off; odd sizes exercise the parity-plane padding."""
    H, W = hw
    B = 3
    m = mods.DepthGuidance(chans)
    m.load_state_dict(OW.guidance_weights(seed=78, channels=chans))
    m.cuda().eval()
    rgbs, ds = zip(*[synthetic.synth_rgbd_u8(800 + j, H, W, "nyu") for j in range(B)])
    pv = fn.pack_pixel_values(torch.from_numpy(np.stack(rgbs)).cuda(), torch.from_numpy(np.stack(ds)).cuda())
    g = torch.Generator(device="cpu").manual_seed(4)
    sizes = [(-(-H // s), -(-W // s)) for s in (4, 8, 16, 32)]
    feats = [torch.randn(B, c, h, w, generator=g).cuda() for c, (h, w) in zip(chans, sizes)]
    ratios = torch.tensor([[0.1], [0.3], [0.5]], device="cuda")
    outs = []
    for fused in (True, False, True):
        monkeypatch.setattr(mods, "FUSE_STAGE_PACKS", fused)
        n0 = fn.LAUNCHES
        with torch.no_grad():
            outs.append([o.clone() for o in m(pv, feats, ratios=ratios)])
        outs[-1].append(fn.LAUNCHES - n0)
    assert outs[0][4] < outs[1][4]                      # fewer launches with the fusion
    for a, b, c in zip(outs[0][:4], outs[1][:4], outs[2][:4]):
        assert torch.equal(a, b) and torch.equal(a, c)


def test_large_frame_swin_b_cross_implementation(mods, fn, monkeypatch):
    """BASELINE configs[4]: 960x1280 frames, Swin-B channels, window ratio forced to output_max.  No oracle at this size;
    the independent kernel variants of each stage must agree: fused front end (sliding-window operand) vs stem GEMM +
    chain, and shared-memory masking vs the pre-masked operand through the whole cascade."""
    chans, (H, W), B = (128, 256, 512, 1024), (960, 1280), 2
    w = OW.guidance_weights(seed=901, channels=chans)
    rgbs, ds = zip(*[synthetic.synth_rgbd_u8(500 + j, H, W, "nyu") for j in range(B)])
    pv = fn.pack_pixel_values(torch.from_numpy(np.stack(rgbs)).cuda(), torch.from_numpy(np.stack(ds)).cuda())
    g = torch.Generator(device="cpu").manual_seed(9)
    feats = [torch.randn(B, c, H // s, W // s, generator=g).cuda() for c, s in zip(chans, (4, 8, 16, 32))]
    forced = torch.full((B, 1), 0.5, device="cuda")
    outs, ratios = [], []
    for variant in range(2):
        monkeypatch.setattr(mods, "_PREMASKED", bool(variant))
        m = mods.DepthGuidance(chans)
        m.load_state_dict(w)
        m.cuda().eval()
        m.ratio_predictor.use_fused_front = variant == 0
        assert m.ratio_predictor._compact(H, W) == (variant == 0)
        with torch.no_grad():
            ratios.append(m.ratio_predictor(pv[:, 3:6]))
            outs.append(m(pv, feats, ratios=forced))
        del m
    assert float(((ratios[0] - ratios[1]).abs() / ratios[1]).max()) < 2e-3
    assert bool(((ratios[0] >= 0.01) & (ratios[0] <= 0.5)).all())
    for a, b in zip(*outs):
        assert a.shape == b.shape and torch.isfinite(a).all()
        # other K order -> fp32 sums differ in the last bits -> a few bf16 roundings of the next stage's input flip
        assert rel_err(a, b) < 2e-3, rel_err(a, b)


# ---------------------------------------------------------------------------------------------------
# size-independent properties at the full BASELINE size (batch 32, 480x640, Swin-T pyramid)
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def full_size(fn):
    B, H, W = 32, 480, 640
    rgbs, ds = [], []
    for j in range(4):
        rgb, d = synthetic.synth_rgbd_u8(300 + j, H, W, ["nyu", "nyu", "uniform", "two_valued"][j])
        rgbs.append(rgb)
        ds.append(d)
    idx = torch.arange(B) % 4
    rgb = torch.from_numpy(np.stack(rgbs)).cuda()[idx].contiguous()
    depth = torch.from_numpy(np.stack(ds)).cuda()[idx].contiguous()
    pv = fn.pack_pixel_values(rgb, depth)
    g = torch.Generator(device="cpu").manual_seed(5)
    feats = [torch.randn(B, c, H // s, W // s, generator=g).cuda() for c, s in zip((96, 192, 384, 768), (4, 8, 16, 32))]
    return pv, feats, depth


def test_full_size_decomposition_invariants(fn, full_size):
    pv, feats, depth = full_size
    B, _, H, W = pv.shape
    ratio = torch.linspace(0.01, 0.5, B, device="cuda")
    dec = fn.depth_decompose(ratio, [(120, 160), (60, 80), (30, 40)], depth3=pv[:, 3:6], debug=True)
    gray = dec.gray
    # every finite pixel lands in exactly one histogram bin; edges are monotone and span [nanmin, nanmax]
    assert torch.equal(dec.hist.sum(1), torch.isfinite(gray).flatten(1).sum(1))
    assert bool((dec.edges[:, 1:] > dec.edges[:, :-1]).all())
    assert torch.equal(dec.edges[:, 0], gray.flatten(1).min(1).values) and torch.equal(dec.edges[:, -1], gray.flatten(1).max(1).values)
    # identical images give identical artefacts (the batch repeats 4 frames); the ratio only moves the windows
    assert torch.equal(dec.hist[0], dec.hist[4]) and torch.equal(dec.peak_bins[1], dec.peak_bins[5])
    # region codes: with m >= 1 modes every pixel carries a bit, and the "remaining" bit m excludes the window bits
    m = dec.n_modes.view(B, 1, 1).to(torch.int32)
    codes = dec.codes.to(torch.int32)
    has_modes = m > 0
    assert bool(((codes > 0) | ~has_modes).all()) and bool(((codes == 0) | has_modes).all())
    rem = (codes >> m) & 1
    assert bool((((rem == 1) & ((codes & ((1 << m) - 1)) != 0)) == 0).all())
    assert bool((codes < (1 << (m + 1))).all())
    # pooled codes are the bitwise OR over the pooling window == per-bit max pooling
    for lvl, s in enumerate((4, 8, 16)):
        ref = torch.zeros_like(dec.pooled[lvl], dtype=torch.int32)
        for t in range(4):
            bit = ((codes >> t) & 1).float()[:, None]
            ref |= (torch.nn.functional.max_pool2d(bit, s)[:, 0].to(torch.int32) << t)
        assert torch.equal(dec.pooled[lvl].to(torch.int32), ref)
    # windows: lo = max(0, c - hw), hi = c + hw with hw = c*ratio/2 -> hi - c is proportional to the ratio
    hw_ = dec.windows[:, :, 1] - dec.centres
    k = dec.n_modes.min().item()
    if k > 0:
        assert torch.allclose(hw_[:, :k], dec.centres[:, :k] * ratio[:, None] / 2, rtol=1e-5, atol=1e-6)


def test_full_size_dggm_and_dsam_linearity(mods, fn, full_size):
    pv, feats, depth = full_size
    B = pv.shape[0]
    chans = (96, 192, 384, 768)
    m = mods.DepthGuidance(chans)
    m.load_state_dict(OW.guidance_weights(seed=11, channels=chans))
    m.cuda().eval()
    with torch.no_grad():
        # DGGM: the enhancement depends on grad/mask/weights only -> out(f) - f is the same for any f; zero mask -> relu(bias)
        dg = m.depth_gradient_injection
        a = dg(feats, pv[:, 6:9], pv[:, 9:10])
        b = dg([2 * f for f in feats], pv[:, 6:9], pv[:, 9:10])
        for i in range(4):
            assert rel_err(b[i] - 2 * feats[i], a[i] - feats[i]) < 1e-5
        z = dg(feats, pv[:, 6:9], torch.zeros_like(pv[:, 9:10]))
        for i in range(4):
            bias = torch.relu(dg.depth_enhancement_layers[i][0].bias).view(1, -1, 1, 1)
            assert rel_err(z[i], feats[i] + bias) < 1e-6
        # DSAM stage: linear in the features once the bias is removed (masks are data): f(2x) - f(0) = 2 (f(x) - f(0))
        ratio = torch.full((B,), 0.3, device="cuda")
        dec = fn.depth_decompose(ratio, [(120, 160)], depth3=pv[:, 3:6])
        d0 = m.dsam0
        y0 = d0.stage_forward(torch.zeros_like(feats[0]), dec.pooled[0], dec.bias_variant)
        y1 = d0.stage_forward(feats[0], dec.pooled[0], dec.bias_variant)
        y2 = d0.stage_forward(2 * feats[0], dec.pooled[0], dec.bias_variant)
        assert rel_err(y2 - y0, 2 * (y1 - y0)) < 1e-5          # scaling by 2 is exact in bf16
        # whole path: finite, right shapes, ratios inside the constrained range (CM:1485)
        r = m.ratio_predictor(pv[:, 3:6])
        assert bool(((r >= 0.01) & (r <= 0.5)).all())
        out = m(pv, feats)
        for o, f in zip(out, feats):
            assert o.shape == f.shape and bool(torch.isfinite(o).all())
        # identical frames (batch repeats 4) with identical features give identical outputs: no cross-image leakage
        same = [f.clone() for f in feats]
        for f in same:
            f[4] = f[0]
        out2 = m(pv, same)
        assert torch.equal(out2[3][0], out2[3][4]) and torch.equal(out2[0][0], out2[0][4])


@pytest.mark.parametrize("version", ["0.0.3", "0.1.2"])
def test_other_version_branches(mods, golden_dir, version):
    """SURVEY section 8f-4: the version branches built from the same kernels (DGGM only / DSAM cascade only)."""
    from rgbd_b200 import pixel_level
    g = load_wiring(golden_dir, f"wiring_v{version.replace('.', '')}.npz")
    cfg = pixel_level.swin_tiny_mask2former_config(num_labels=8)
    plm = pixel_level.CustomMask2FormerPixelLevelModule(cfg, version=version)
    w = OW.guidance_weights(seed=700)
    own = dict(plm.named_children())
    missing = plm.load_state_dict({k: v for k, v in w.items() if k.split(".")[0] in own}, strict=False)
    assert not missing.unexpected_keys
    assert ("ratio_predictor" in own) == (version == "0.4.0")
    plm.cuda().eval()
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs)).cuda()
    pvv = torch.cat([pv[:, 0:3], pv[:, 6:9], pv[:, 9:10]], dim=1) if version == "0.0.3" else pv[:, 0:6].contiguous()
    feats = [torch.from_numpy(g[f"feat{i}"]).cuda() for i in range(4)]
    with torch.no_grad():
        if version == "0.0.3":
            fused = plm.depth_gradient_injection(feats, pvv[:, 3:6], pvv[:, 6:7])
        else:
            fused = plm._dsam_only(pvv, feats)
    tol = FP32_TOL if version == "0.0.3" else BF16_TOL
    for i in range(4):
        assert rel_err(fused[i], torch.from_numpy(g[f"fused{i}"])) < tol, (version, i)
    with pytest.raises(NotImplementedError):
        pixel_level.CustomMask2FormerPixelLevelModule(cfg, version="0.2.0")


@pytest.mark.parametrize("version", ["0.1.3", "0.3.0"])
def test_depth_encoder_version_branches(mods, golden_dir, version):
    """Versions with a second (depth) encoder and the feature-based RatioPredictor (CM:258-322)."""
    from rgbd_b200 import pixel_level
    g = load_wiring(golden_dir, f"wiring_v{version.replace('.', '')}.npz")
    cfg = pixel_level.swin_tiny_mask2former_config(num_labels=8)
    torch.manual_seed(0)         # the stock (random-init) HF pixel decoder yields NaN for some seeds at this tiny size
    plm = pixel_level.CustomMask2FormerPixelLevelModule(cfg, version=version)
    own = dict(plm.named_children())
    assert "depth_encoder" in own and isinstance(plm.ratio_predictor, mods.RatioPredictor)
    assert ("depth_gradient_injection" in own) == (version == "0.3.0")
    w = OW.guidance_weights_feature_ratio(seed=700)
    missing = plm.load_state_dict({k: v for k, v in w.items() if k.split(".")[0] in own}, strict=False)
    assert not missing.unexpected_keys
    plm.cuda().eval()
    pvs = []
    for j in range(2):
        rgb, d = synthetic.synth_rgbd_u8(80 + j, 64, 96, "nyu")
        pvs.append(synthetic.assemble_pixel_values(rgb, d, O.gradient_features))
    pv = torch.from_numpy(np.stack(pvs)).cuda()
    feats = [torch.from_numpy(g[f"feat{i}"]).cuda() for i in range(4)]
    dfeats = [torch.from_numpy(g[f"dfeat{i}"]).cuda() for i in range(4)]
    with torch.no_grad():
        ratios = plm.ratio_predictor(dfeats)
        assert ratios.shape == (2, 1)
        assert rel_err(ratios, torch.from_numpy(g["ratios"])) < 1e-5
        fused = plm._dsam_only(pv, feats, ratios)
        if version == "0.3.0":
            fused = plm.depth_gradient_injection(fused, pv[:, 6:9], pv[:, 9:10])
        for i in range(4):
            assert rel_err(fused[i], torch.from_numpy(g[f"fused{i}"])) < BF16_TOL, (version, i)
        # the whole module (stock encoders + decoder around the hot path) runs end to end
        out = plm(pv if version == "0.3.0" else pv[:, 0:6].contiguous())
        assert out.decoder_last_hidden_state.shape[0] == 2 and torch.isfinite(out.encoder_last_hidden_state).all()
    with pytest.raises(AssertionError):
        plm.ratio_predictor(dfeats[:3])
    with pytest.raises(AssertionError):                      # CM:876: channel count per scale
        plm.ratio_predictor([dfeats[1], dfeats[1], dfeats[2], dfeats[3]])
    # odd plane sizes take the scalar (unaligned) pooling path
    odd = [torch.randn(3, c, 5, 7, device="cuda") for c in plm.ratio_predictor.depth_channels_list]
    w_rp = {k[len("ratio_predictor."):]: v for k, v in w.items() if k.startswith("ratio_predictor.")}
    assert rel_err(plm.ratio_predictor(odd), O.ratio_from_features_forward(w_rp, [t.cpu() for t in odd])) < 1e-5


# ---------------------------------------------------------------------------------------------------
# robustness of the host plumbing (ADVICE r1): graph-owned buffers, shape validation, device mismatch
# ---------------------------------------------------------------------------------------------------
def test_graphed_guidance_survives_cache_eviction_and_rejects_stale_weights(mods, fn):
    chans, (H, W) = (32, 64, 96, 160), (64, 96)
    m = mods.DepthGuidance(chans)
    m.load_state_dict(OW.guidance_weights(seed=31, channels=chans))
    m.cuda().eval()

    def inputs(B, seed):
        rgbs, ds = zip(*[synthetic.synth_rgbd_u8(seed + j, H, W, "nyu") for j in range(B)])
        pv = fn.pack_pixel_values(torch.from_numpy(np.stack(rgbs)).cuda(), torch.from_numpy(np.stack(ds)).cuda())
        g = torch.Generator(device="cpu").manual_seed(seed)
        return pv, [torch.randn(B, c, H // s, W // s, generator=g).cuda() for c, s in zip(chans, (4, 8, 16, 32))]
    pv, feats = inputs(2, 700)
    with torch.no_grad():
        want = [t.clone() for t in m(pv, feats)]
    graphed = mods.GraphedDepthGuidance(m, pv, feats)
    # eager calls at more shapes than the caches hold: the modules drop the captured workspaces, the graph keeps them
    with torch.no_grad():
        for B in range(3, 3 + mods.MAX_CACHED_SHAPES + 1):
            m(*inputs(B, 710 + B))
    junk = [torch.randn(64 << 20, device="cuda") for _ in range(4)]     # would reuse freed blocks
    got = graphed()
    torch.cuda.synchronize()
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    del junk
    with torch.no_grad():
        m.dsam0.conv_layers[0].weight.mul_(1.5)
    with pytest.raises(_rgbd_lib.RgbdB200Error):
        graphed()


def test_stage_forward_validates_pyramid_shapes(mods, fn):
    m = mods.DSAModule(32, 64, 3)
    m.load_state_dict(OW.dsam_weights(32, 64, seed=5))
    m.cuda().eval()
    feat = torch.randn(2, 32, 15, 20, device="cuda")
    gray = torch.from_numpy(np.stack([_gray_for(j, "nyu", (60, 80)) for j in range(2)])).cuda()
    dec = fn.depth_decompose(torch.tensor([0.2, 0.3]).cuda(), [(15, 20)], gray=gray)
    good = torch.zeros(2, 64, 8, 10, device="cuda")
    m.stage_forward(feat, dec.pooled[0], dec.bias_variant, residual=good)
    with pytest.raises(_rgbd_lib.RgbdB200Error):        # a backbone that floors odd sizes: 15 -> 7 instead of 8
        m.stage_forward(feat, dec.pooled[0], dec.bias_variant, residual=torch.zeros(2, 64, 7, 10, device="cuda"))
    with pytest.raises(_rgbd_lib.RgbdB200Error):
        m.stage_forward(feat, dec.pooled[0][:, :14].contiguous(), dec.bias_variant, residual=good)


def test_tensor_on_another_device_raises(fn):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    x = torch.zeros(1, 3, 8, 8, device="cuda:1")
    with torch.cuda.device(0), pytest.raises(_rgbd_lib.RgbdB200Error):
        fn.to_grayscale(x)
    with torch.cuda.device(1):
        fn.to_grayscale(x)                                # per-device launch state: works on the second GPU too


# ---------------------------------------------------------------------------------------------------
# train-mode ratio predictor: batch-statistics BatchNorm, running-stat updates, Dropout (SURVEY H6, CM:1380-1437)
# ---------------------------------------------------------------------------------------------------
def test_ratio_predictor_train_mode_matches_reference_golden(mods, golden_dir):
    from oracle.make_golden_train import SEED_W, train_inputs
    g = np.load(os.path.join(golden_dir, "ratio_train.npz"))
    m = mods.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(OW.ratio_weights(seed=SEED_W))
    m.cuda().train()
    for step in range(2):
        x, keep = train_inputs(synthetic, step)
        r = m(x.cuda(), dropout_masks=keep)
        assert not r.requires_grad
        ref = torch.from_numpy(g[f"step{step}.ratio"])
        assert float(((r.cpu() - ref).abs() / ref).max()) < BF16_TOL, (step, r.cpu().flatten(), ref.flatten())
        sd = m.state_dict()
        for k, v in sd.items():
            if "running" in k:
                want = torch.from_numpy(g[f"step{step}.{k}"])
                assert rel_err(v, want) < BF16_TOL, (step, k, rel_err(v, want))
            elif "num_batches" in k:
                assert int(v) == step + 1, (k, int(v))
    # eval() afterwards uses the UPDATED running statistics, like the reference
    m.eval()
    x, _ = train_inputs(synthetic, 0)
    w_after = {k: v.cpu() for k, v in m.state_dict().items()}
    with torch.no_grad():
        r_eval = m(x.cuda())
    ref_eval = O.ratio_predictor_forward(w_after, x)
    assert float(((r_eval.cpu() - ref_eval).abs() / ref_eval).max()) < BF16_TOL


@pytest.mark.parametrize("B,hw", [(2, (96, 160)), (8, (480, 640))])
def test_ratio_predictor_train_mode_against_oracle(mods, B, hw):
    """Larger shapes incl. the fine-tuning batch of BASELINE configs[3] (8 frames of 480x640) against the oracle's train-mode
    restatement (itself pinned by the reference golden above)."""
    w = OW.ratio_weights(seed=510)
    m = mods.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(w)
    m.cuda().train()
    kinds = ("nyu", "nyu", "uniform", "nyu", "two_valued", "nyu", "nyu", "constant")
    frames = []
    for j in range(B):
        _, d = synthetic.synth_rgbd_u8(170 + j, hw[0], hw[1], kinds[j % len(kinds)])
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    x = torch.from_numpy(np.stack(frames))
    rs = np.random.RandomState(3)
    keep = (torch.from_numpy(rs.rand(B, 128) >= 0.3), torch.from_numpy(rs.rand(B, 64) >= 0.2))
    ref, w_ref = O.ratio_predictor_forward_train(w, x, keep)
    r = m(x.cuda(), dropout_masks=keep)
    err = float(((r.cpu() - ref).abs() / ref).max())
    assert err < BF16_TOL, (err, r.cpu().flatten(), ref.flatten())
    for k, v in m.state_dict().items():
        if "running" in k:
            assert rel_err(v, w_ref[k]) < BF16_TOL, (k, rel_err(v, w_ref[k]))
    # without injected masks the module draws its own: still a valid ratio, and it differs from the masked run
    r2 = m(x.cuda())
    assert bool(((r2 >= 0.01) & (r2 <= 0.5)).all())


# ---------------------------------------------------------------------------------------------------
# round-2 kernel variants: fused codes + pyramid pooling, tensor-core tail
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(64, 48), (96, 128), (480, 640), (16, 16)])
def test_decompose_fused_pyramid_path_bit_exact(fn, hw):
    """Levels (H/4, H/8, H/16): codes and the three OR-pooled copies come from ONE kernel (a warp per 32x16 block, W % 32 != 0
    included); bit-exact against the oracle, and identical with and without the optional full-resolution code image."""
    H, W = hw
    kinds = ["nyu", "uniform", "two_valued", "constant", "all_invalid"]
    grays = [_gray_for(j, kinds[j % 5], hw) for j in range(5)]
    ratios = [0.5, 0.1, 0.3, 0.2, 0.4]
    levels = [(H // 4, W // 4), (H // 8, W // 8), (H // 16, W // 16)]
    _check_decomposition(fn, grays, ratios, levels)
    g = torch.from_numpy(np.stack(grays)).cuda()
    r = torch.tensor(ratios, dtype=torch.float32).cuda()
    a = fn.depth_decompose(r, levels, gray=g)
    b = fn.depth_decompose(r, levels, gray=g, want_codes=False)
    assert b.codes is None and a.codes is not None
    for x, y in zip(a.pooled, b.pooled):
        assert torch.equal(x, y)
    assert torch.equal(a.bias_variant, b.bias_variant) and torch.equal(a.windows, b.windows)


def test_ratio_predictor_tensor_core_tail_matches_fp32_tail(mods):
    w = OW.ratio_weights(seed=520)
    frames = []
    for j in range(5):
        _, d = synthetic.synth_rgbd_u8(260 + j, 96, 160, ["nyu", "uniform", "nyu", "two_valued", "constant"][j])
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    x = torch.from_numpy(np.stack(frames))
    ref = O.ratio_predictor_forward(w, x)
    outs = []
    for tc_tail in (True, False):
        m = mods.EnhancedDepthImageRatioPredictor(3)
        m.load_state_dict(w)
        m.cuda().eval()
        m.use_tensor_core_tail = tc_tail
        with torch.no_grad():
            outs.append(m(x.cuda()).cpu())
        assert float(((outs[-1] - ref).abs() / ref).max()) < BF16_TOL
    assert float(((outs[0] - outs[1]).abs() / outs[1]).max()) < 2e-3


def test_torch_ops_dggm_autograd_matches_module(mods):
    """``torch.ops.rgbd_b200.dggm_forward`` (dispatcher op + registered autograd formula) == the nn.Module path."""
    from rgbd_b200 import ops  # noqa: F401
    chans, hw, sizes, B = [8, 16, 24, 40], (32, 48), [(8, 12), (4, 6), (2, 3), (1, 2)], 2
    w = OW.dggm_weights(chans, 3, seed=77)
    m = mods.DepthGradientInjectionResidual(chans, 3)
    m.load_state_dict(w)
    m.cuda()
    rs = np.random.RandomState(3)
    feats = [torch.from_numpy(rs.randn(B, c, h, ww).astype(np.float32)).cuda().requires_grad_() for c, (h, ww) in zip(chans, sizes)]
    grad = torch.from_numpy(rs.rand(B, 3, *hw).astype(np.float32)).cuda()
    mask = torch.from_numpy((rs.rand(B, 1, *hw) < 0.6).astype(np.float32)).cuda()
    ws, bs = m._params()
    outs = torch.ops.rgbd_b200.dggm_forward(feats, grad, mask, list(ws), list(bs))
    ref = m(feats, grad, mask)
    for a, b in zip(outs, ref):
        assert torch.equal(a, b)
    douts = [torch.randn_like(o) for o in outs]
    g_op = torch.autograd.grad(outs, [*feats, *ws, *bs], douts)
    g_ref = torch.autograd.grad(ref, [*feats, *ws, *bs], douts)
    for a, b in zip(g_op, g_ref):            # dW / db are reduced with float atomics: equal up to the summation order
        assert rel_l2(a, b) < 1e-4, rel_l2(a, b)
    dec = torch.ops.rgbd_b200.depth_decompose(torch.randn(2, 3, 32, 48, device="cuda"), torch.tensor([0.2, 0.3], device="cuda"),
                                              [8, 4, 2], [12, 6, 3])
    assert dec[0].shape == (2, 8, 12) and dec[0].dtype == torch.uint8


# ---------------------------------------------------------------------------------------------------
# SURVEY 8f-2: the pixel decoder's input projections (Conv1x1 + GroupNorm) on this library's kernels
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,hw,bias", [(192, (60, 80), True), (768, (15, 20), True), (96, (24, 36), False), (100, (7, 9), True)])
def test_project_group_norm_matches_torch_modules(fn, c, hw, bias):
    torch.manual_seed(c)
    seq = torch.nn.Sequential(torch.nn.Conv2d(c, 256, 1, bias=bias), torch.nn.GroupNorm(32, 256)).cuda()
    with torch.no_grad():
        seq[1].weight.uniform_(0.5, 1.5)
        seq[1].bias.normal_()
    x = torch.randn(3, c, *hw, device="cuda") * 2 + 0.3
    with torch.no_grad():
        ref = seq(x)
        got = fn.project_group_norm(x, seq[0].weight, seq[0].bias, seq[1].weight, seq[1].bias, 32, seq[1].eps)
    assert got.shape == ref.shape
    assert rel_l2(got, ref) < 5e-3 and rel_err(got, ref) < BF16_TOL, (rel_l2(got, ref), rel_err(got, ref))


def test_pixel_level_module_with_fused_input_projections(mods):
    """The stock HF pixel decoder fed with projections computed by this library == the stock decoder doing them itself."""
    from rgbd_b200 import synthetic_weights as SW
    model, _ = SW.build_synthetic_rgbd_mask2former()
    plm = model.model.pixel_level_module.cuda()
    rgbs, ds = zip(*[synthetic.synth_rgbd_u8(400 + j, 128, 160, "nyu") for j in range(2)])
    from rgbd_b200 import functional as Fn
    pv = Fn.pack_pixel_values(torch.from_numpy(np.stack(rgbs)).cuda(), torch.from_numpy(np.stack(ds)).cuda())
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        n0 = Fn.LAUNCHES
        ref = plm(pv)
        n1 = Fn.LAUNCHES
        plm.fuse_input_projections = True
        got = plm(pv)
        assert (Fn.LAUNCHES - n1) - (n1 - n0) == 12        # 4 projections x (pack + GEMM + GroupNorm) on top of the hot path
        plm.fuse_input_projections = False
    assert torch.equal(got.encoder_last_hidden_state, ref.encoder_last_hidden_state)
    assert rel_l2(got.decoder_last_hidden_state, ref.decoder_last_hidden_state) < BF16_TOL
    for a, b in zip(got.decoder_hidden_states, ref.decoder_hidden_states):
        assert a.shape == b.shape and rel_l2(a, b) < BF16_TOL, rel_l2(a, b)
    # the decoder's own modules are back in place
    assert isinstance(plm.decoder.input_projections[0], torch.nn.Sequential)


@pytest.mark.parametrize("hw", [(50, 70), (33, 47), (62, 128)])
def test_ratio_predictor_sizes_not_divisible_by_four(mods, hw):
    """AdaptiveAvgPool2d(4) with overlapping windows (H or W not a multiple of 4): the map is pooled by a separate kernel."""
    w = OW.ratio_weights(seed=530)
    m = mods.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(w)
    m.cuda().eval()
    frames = []
    for j in range(3):
        _, d = synthetic.synth_rgbd_u8(280 + j, hw[0], hw[1], ["nyu", "uniform", "nyu"][j])
        frames.append(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
    x = torch.from_numpy(np.stack(frames))
    ref = O.ratio_predictor_forward(w, x)
    with torch.no_grad():
        r = m(x.cuda())
    assert float(((r.cpu() - ref).abs() / ref).max()) < BF16_TOL
    m.train()
    rs = np.random.RandomState(4)
    keep = (torch.from_numpy(rs.rand(3, 128) >= 0.3), torch.from_numpy(rs.rand(3, 64) >= 0.2))
    ref_t, _ = O.ratio_predictor_forward_train(w, x, keep)
    r_t = m(x.cuda(), dropout_masks=keep)
    assert float(((r_t.cpu() - ref_t).abs() / ref_t).max()) < BF16_TOL


def test_depth_guidance_fine_tuning_step_with_train_mode_predictor(mods):
    """BASELINE configs[3] semantics end to end on the hot path: ``.train()`` -> the ratio comes from the batch-statistics
    predictor (Dropout masks injected), it steers the region masks, and DSAM / DGGM gradients follow -- all against the
    oracle run with ITS train-mode ratio (no ratio is handed over, unlike test_depth_guidance_training_gradients)."""
    chans, (H, W), B = (32, 64, 96, 160), (64, 96), 3
    w = OW.guidance_weights(seed=41, channels=chans)
    m = mods.DepthGuidance(chans)
    m.load_state_dict(w)
    m.cuda().train()
    pvs = [synthetic.assemble_pixel_values(*synthetic.synth_rgbd_u8(330 + j, H, W, ["nyu", "nyu", "uniform"][j]), O.gradient_features)
           for j in range(B)]
    pv = torch.from_numpy(np.stack(pvs))
    rs = np.random.RandomState(12)
    feats = [torch.from_numpy(rs.randn(B, c, H // s, W // s).astype(np.float32)) for c, s in zip(chans, (4, 8, 16, 32))]
    douts = [torch.from_numpy(rs.randn(*f.shape).astype(np.float32)) for f in feats]
    keep = (torch.from_numpy(rs.rand(B, 128) >= 0.3), torch.from_numpy(rs.rand(B, 64) >= 0.2))
    ref_ratio, w_after = O.ratio_predictor_forward_train(O._sub(w, "ratio_predictor."), pv[:, 3:6], keep)
    wr = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and not k.startswith("ratio_predictor.") else v)
          for k, v in w.items()}
    ref, _ = O.depth_guidance_forward(wr, pv, feats, ratios=ref_ratio)
    sum((o * d).sum() for o, d in zip(ref, douts)).backward()
    m.ratio_predictor.dropout_masks_override = keep
    out = m(pv.cuda(), [f.cuda() for f in feats])
    sum((o * d.cuda()).sum() for o, d in zip(out, douts)).backward()
    for i in range(4):
        assert rel_l2(out[i], ref[i]) < 3 * BF16_TOL, (i, rel_l2(out[i], ref[i]))
    for name, p in m.named_parameters():
        if name.startswith("ratio_predictor."):
            assert p.grad is None, name
        else:
            assert rel_l2(p.grad, wr[name].grad) < 5e-2, (name, rel_l2(p.grad, wr[name].grad))
    for k, v in m.ratio_predictor.state_dict().items():      # the step moved the running statistics like the reference would
        if "running" in k:
            assert rel_err(v, w_after[k]) < BF16_TOL, k


@pytest.mark.parametrize("c_in,hw", [(1, (48, 64)), (4, (24, 40)), (2, (33, 47))])
def test_ratio_predictor_other_input_channel_counts(mods, c_in, hw):
    """``EnhancedDepthImageRatioPredictor(input_channels=c)`` for c = 1..4 (the reference default is 3; the stem operand pads
    every pixel to four channels), compact and row-im2col operands."""
    w = OW.ratio_weights(seed=540 + c_in, c_in=c_in)
    m = mods.EnhancedDepthImageRatioPredictor(c_in)
    m.load_state_dict(w)
    m.cuda().eval()
    x = torch.from_numpy(np.random.RandomState(c_in).randn(2, c_in, *hw).astype(np.float32))
    ref = O.ratio_predictor_forward(w, x)
    with torch.no_grad():
        r = m(x.cuda())
        m.use_compact_operand = False
        r2 = m(x.cuda())
    assert float(((r.cpu() - ref).abs() / ref).max()) < BF16_TOL and float(((r2.cpu() - ref).abs() / ref).max()) < BF16_TOL
    with pytest.raises(ValueError):
        mods.EnhancedDepthImageRatioPredictor(5)


def test_invalidate_packed_after_writes_that_bypass_the_version_counter(mods, fn):
    """``weight.data.mul_()`` (EMA swaps, fused optimizers) does not bump ``_version``: the bf16-packed copies stay stale until
    ``invalidate_packed()`` -- or a ``train()`` / ``eval()`` switch -- drops them (ADVICE r1)."""
    m = mods.DSAModule(32, 64, 3)
    m.load_state_dict(OW.dsam_weights(32, 64, seed=9))
    m.cuda().eval()
    feat = torch.randn(2, 32, 16, 24, device="cuda")
    gray = torch.from_numpy(np.stack([_gray_for(j, "nyu", (64, 96)) for j in range(2)])).cuda()
    dec = fn.depth_decompose(torch.tensor([0.2, 0.3]).cuda(), [(16, 24)], gray=gray)
    with torch.no_grad():
        y0 = m.stage_forward(feat, dec.pooled[0], dec.bias_variant).clone()
        v = m.rgb_projection.weight._version
        m.rgb_projection.weight.data.mul_(3.0)
        assert m.rgb_projection.weight._version == v                      # the write was invisible to the cache key
        y_stale = m.stage_forward(feat, dec.pooled[0], dec.bias_variant).clone()
        m.invalidate_packed()
        y_new = m.stage_forward(feat, dec.pooled[0], dec.bias_variant).clone()
        m.rgb_projection.weight.mul_(1.0 / 3.0)                            # a versioned write is picked up by itself
        y_back = m.stage_forward(feat, dec.pooled[0], dec.bias_variant)
    assert torch.equal(y_stale, y0) and not torch.equal(y_new, y0)
    assert rel_err(y_back, y0) < 1e-2
