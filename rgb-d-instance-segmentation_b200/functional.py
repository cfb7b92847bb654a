"""Torch-facing wrappers over the C ABI (include/rgbd_b200.h).  PyTorch is plumbing here: device
memory, the current CUDA stream and shape checks.  Every function requires CUDA tensors and raises
otherwise -- there is no CPU or eager fallback."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ConvGemmDesc, RgbdB200Error, check, int_array, ptr_array

HIST_BINS = 512

# kernels launched through this module since it was last reset (bench.py's `gpu_launches`)
LAUNCHES = 0


def _count(n: int) -> None:
    global LAUNCHES
    LAUNCHES += n


_last_device = None      # device index of the tensor most recently validated by _req


def _stream() -> int:
    """Current stream handle.  Kernels launch on the CURRENT device: a tensor that lives on another GPU would be
    dereferenced from the wrong device, so the mismatch raises here (wrap the call in ``torch.cuda.device(t.device)``)."""
    cur = torch.cuda.current_device()
    if _last_device is not None and _last_device != cur:
        raise RgbdB200Error(f"tensors live on cuda:{_last_device} but the current device is cuda:{cur}; "
                            f"call inside `with torch.cuda.device({_last_device}):`")
    return torch.cuda.current_stream().cuda_stream


def _req(t: torch.Tensor, name: str, dtype=None, contiguous: bool = True) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RgbdB200Error(f"{name} must be a CUDA tensor (rgbd_b200 has no CPU fallback); got device {t.device}")
    if dtype is not None and t.dtype != dtype:
        raise RgbdB200Error(f"{name} must be {dtype}, got {t.dtype}")
    if contiguous and not t.is_contiguous():
        raise RgbdB200Error(f"{name} must be contiguous")
    global _last_device
    _last_device = t.device.index
    return t


def _plane_strided(t: torch.Tensor, name: str) -> Tuple[int, int]:
    """(batch stride, channel stride) of a (B,C,H,W) view whose (H,W) planes are dense (e.g. pixel_values[:,6:9])."""
    B, Cc, H, W = t.shape
    if t.stride(3) != 1 or t.stride(2) != W or (Cc > 1 and t.stride(1) != H * W):
        raise RgbdB200Error(f"{name}: channel planes must be dense (strides {t.stride()})")
    return t.stride(0), H * W


# ------------------------------------------------------------------------------------------------
# DGGM
# ------------------------------------------------------------------------------------------------
def dggm_forward(feats: Sequence[torch.Tensor], grad: torch.Tensor, mask: torch.Tensor,
                 weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor],
                 branch1: Optional[Sequence[torch.Tensor]] = None,
                 outs: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
    """K1.  out_i = feats_i + ReLU(conv1x1_i(bilinear(grad) * nearest(mask))) [+ branch1_i].  ``outs``: preallocated
    results (e.g. views of one staging slab)."""
    lib = _lib.load()
    n = len(feats)
    _req(grad, "processed_depth_gradient_map", torch.float32, contiguous=False)
    _req(mask, "gradient_mask", torch.float32, contiguous=False)
    B, D, H, W = grad.shape
    if mask.shape != (B, 1, H, W):
        raise RgbdB200Error(f"gradient_mask must be {(B, 1, H, W)}, got {tuple(mask.shape)}")
    gbs, _ = _plane_strided(grad, "processed_depth_gradient_map")
    mbs, _ = _plane_strided(mask, "gradient_mask")
    given = outs
    outs = []
    ws, bs = [], []
    for i, f in enumerate(feats):
        _req(f, f"color_feature_maps[{i}]", torch.float32)
        if f.shape[0] != B:
            raise RgbdB200Error("batch size mismatch between features and gradient map")
        w = _req(weights[i].reshape(weights[i].shape[0], -1), f"weight[{i}]", torch.float32)
        b = _req(biases[i], f"bias[{i}]", torch.float32)
        if w.shape != (f.shape[1], D) or b.shape != (f.shape[1],):
            raise RgbdB200Error(f"scale {i}: weight {tuple(w.shape)} / bias {tuple(b.shape)} do not match C={f.shape[1]}, D={D}")
        ws.append(w)
        bs.append(b)
        if given is not None:
            if given[i].shape != f.shape:
                raise RgbdB200Error(f"outs[{i}] must have the shape of color_feature_maps[{i}]")
            outs.append(_req(given[i], f"outs[{i}]", torch.float32))
        else:
            outs.append(torch.empty_like(f))
        if branch1 is not None:
            _req(branch1[i], f"branch1[{i}]", torch.float32)
            if branch1[i].shape != f.shape:
                raise RgbdB200Error("branch1 shape mismatch")
    rc = lib.rgbd_dggm_fwd(
        n, ptr_array([f.data_ptr() for f in feats]),
        ptr_array([t.data_ptr() for t in branch1]) if branch1 is not None else None,
        ptr_array([o.data_ptr() for o in outs]),
        int_array([f.shape[1] for f in feats]), int_array([f.shape[2] for f in feats]),
        int_array([f.shape[3] for f in feats]),
        ptr_array([w.data_ptr() for w in ws]), ptr_array([b.data_ptr() for b in bs]),
        grad.data_ptr(), gbs, mask.data_ptr(), mbs, B, D, H, W, _stream())
    check(rc, "rgbd_dggm_fwd")
    _count(1)
    return outs


def dggm_backward_params(douts: Sequence[torch.Tensor], grad: torch.Tensor, mask: torch.Tensor,
                         weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor]
                         ) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
    """K1b.  (dW_i, db_i) of the 1x1 enhancement convs."""
    lib = _lib.load()
    B, D, H, W = grad.shape
    gbs, _ = _plane_strided(_req(grad, "grad", torch.float32, False), "grad")
    mbs, _ = _plane_strided(_req(mask, "mask", torch.float32, False), "mask")
    douts = [_req(d.contiguous(), f"dout[{i}]", torch.float32) for i, d in enumerate(douts)]
    ws = [_req(w.reshape(w.shape[0], -1), "weight", torch.float32) for w in weights]
    bs = [_req(b, "bias", torch.float32) for b in biases]
    dws = [torch.empty_like(w) for w in ws]
    dbs = [torch.empty_like(b) for b in bs]
    rc = lib.rgbd_dggm_bwd_params(
        len(douts), ptr_array([d.data_ptr() for d in douts]), int_array([d.shape[1] for d in douts]),
        int_array([d.shape[2] for d in douts]), int_array([d.shape[3] for d in douts]),
        ptr_array([w.data_ptr() for w in ws]), ptr_array([b.data_ptr() for b in bs]),
        ptr_array([w.data_ptr() for w in dws]), ptr_array([b.data_ptr() for b in dbs]),
        grad.data_ptr(), gbs, mask.data_ptr(), mbs, B, D, H, W, _stream())
    check(rc, "rgbd_dggm_bwd_params")
    _count(1)
    return [dw.reshape(weights[i].shape) for i, dw in enumerate(dws)], dbs


def gradient_features(depth: torch.Tensor, n_rep: int = 3, invalid_value: float = 0.0,
                      norm_out: Optional[torch.Tensor] = None, vmask_out: Optional[torch.Tensor] = None
                      ) -> Tuple[torch.Tensor, torch.Tensor]:
    """K0.  depth (B,H,W) float32 or uint8 -> (norm (B,n_rep,H,W), vmask (B,1,H,W)); the outputs may be views
    into a (B,10,H,W) pixel_values tensor (channels 6:9 and 9:10)."""
    lib = _lib.load()
    _req(depth, "depth")
    if depth.dtype == torch.float32:
        dt = 0
    elif depth.dtype == torch.uint8:
        dt = 2
    else:
        raise RgbdB200Error(f"depth must be float32 or uint8, got {depth.dtype}")
    if depth.dim() != 3:
        raise RgbdB200Error("depth must be (B,H,W)")
    B, H, W = depth.shape
    if norm_out is None:
        norm_out = torch.empty(B, n_rep, H, W, device=depth.device, dtype=torch.float32)
    if vmask_out is None:
        vmask_out = torch.empty(B, 1, H, W, device=depth.device, dtype=torch.float32)
    _req(norm_out, "norm_out", torch.float32, False)
    _req(vmask_out, "vmask_out", torch.float32, False)
    if norm_out.shape != (B, n_rep, H, W) or vmask_out.shape != (B, 1, H, W):
        raise RgbdB200Error("gradient_features: bad output shapes")
    nbs, _ = _plane_strided(norm_out, "norm_out")
    vbs, _ = _plane_strided(vmask_out, "vmask_out")
    ws = torch.empty(max(int(lib.rgbd_gradient_features_workspace_bytes(B)), 16), device=depth.device, dtype=torch.uint8)
    rc = lib.rgbd_gradient_features(depth.data_ptr(), dt, H * W, norm_out.data_ptr(), nbs, n_rep, vmask_out.data_ptr(),
                                    vbs, B, H, W, float(invalid_value), ws.data_ptr(), _stream())
    check(rc, "rgbd_gradient_features")
    _count(3)
    return norm_out, vmask_out


def pack_pixel_values(rgb_u8: torch.Tensor, depth_u8: torch.Tensor, out: Optional[torch.Tensor] = None,
                      mean=(0.48500001430511475, 0.4560000002384186, 0.4059999883174896),
                      std=(0.2290000021457672, 0.2239999920129776, 0.22499999403953552),   # preprocessor_config.json
                      rescale_factor: float = 0.00392156862745098, invalid_value: float = 0.0) -> torch.Tensor:
    """Front-end of ``map_10channel_case2`` (DL:386-425) on device: uint8 colour (B,H,W,3) + uint8 depth (B,H,W), already
    at the model resolution -> ``pixel_values`` (B,10,H,W) float32."""
    lib = _lib.load()
    _req(rgb_u8, "rgb", torch.uint8)
    _req(depth_u8, "depth", torch.uint8)
    B, H, W = depth_u8.shape
    if rgb_u8.shape != (B, H, W, 3):
        raise RgbdB200Error(f"rgb must be {(B, H, W, 3)}, got {tuple(rgb_u8.shape)}")
    if out is None:
        out = torch.empty(B, 10, H, W, device=depth_u8.device, dtype=torch.float32)
    _req(out, "pixel_values", torch.float32)
    ws = torch.empty(max(int(lib.rgbd_gradient_features_workspace_bytes(B)), 16), device=depth_u8.device, dtype=torch.uint8)
    m = (C.c_float * 3)(*[float(v) for v in mean])
    s = (C.c_float * 3)(*[float(v) for v in std])
    check(lib.rgbd_pack_pixel_values(rgb_u8.data_ptr(), depth_u8.data_ptr(), out.data_ptr(), out.stride(0), B, H, W,
                                     float(rescale_factor), m, s, float(invalid_value), ws.data_ptr(), _stream()),
          "rgbd_pack_pixel_values")
    _count(4)
    return out


def to_grayscale(rgb3: torch.Tensor) -> torch.Tensor:
    """(B,3,H,W) float32 (any batch / channel strides, contiguous planes) -> (B,H,W): CM:466-480, bit-exact."""
    lib = _lib.load()
    _req(rgb3, "image", torch.float32, False)
    if rgb3.dim() != 4 or rgb3.shape[1] != 3:
        raise RgbdB200Error("to_grayscale: expected (B,3,H,W)")
    B, _, H, W = rgb3.shape
    bs, cs = _plane_strided(rgb3, "image")
    out = torch.empty(B, H, W, device=rgb3.device, dtype=torch.float32)
    ws = torch.empty(int(lib.rgbd_depth_helper_workspace_bytes(B)), device=rgb3.device, dtype=torch.uint8)
    check(lib.rgbd_to_grayscale(rgb3.data_ptr(), bs, cs, out.data_ptr(), B, H * W, ws.data_ptr(), _stream()), "rgbd_to_grayscale")
    _count(2)
    return out


def depth_select_modes(hist: torch.Tensor, edges: torch.Tensor, num_modes: int = 3,
                       prominence_threshold: float = 0.01) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """``DSAModule._select_depth_distribution_modes`` (CM:720-752) on caller-supplied histograms: hist (B,512) int64,
    edges (B,513) fp32 -> (n_modes (B,), peak_bins (B,3), centres (B,3)) ordered by (height, centre) descending."""
    lib = _lib.load()
    _req(hist, "hist", torch.int64)
    _req(edges, "bin_edges", torch.float32)
    B = hist.shape[0]
    if hist.shape != (B, 512) or edges.shape != (B, 513):
        raise RgbdB200Error("depth_select_modes: the device peak finder is built for 512 bins (hist (B,512), edges (B,513))")
    dev = hist.device
    n = torch.empty(B, device=dev, dtype=torch.int32)
    bins = torch.empty(B, 3, device=dev, dtype=torch.int32)
    centres = torch.empty(B, 3, device=dev, dtype=torch.float32)
    ws = torch.empty(int(lib.rgbd_depth_helper_workspace_bytes(B)), device=dev, dtype=torch.uint8)
    check(lib.rgbd_depth_select_modes(hist.data_ptr(), edges.data_ptr(), B, int(num_modes), float(prominence_threshold),
                                      n.data_ptr(), bins.data_ptr(), centres.data_ptr(), ws.data_ptr(), _stream()),
          "rgbd_depth_select_modes")
    _count(3)
    return n, bins, centres


def depth_region_codes(gray: torch.Tensor, windows: torch.Tensor, n_windows: torch.Tensor) -> torch.Tensor:
    """``DSAModule._generate_depth_region_masks`` (CM:774-798) as one code byte per pixel: gray (B,...) fp32, windows
    (B,3,2) fp32, n_windows (B,) int32 -> codes (same shape as gray) uint8, bit n_windows[b] = the remaining region."""
    lib = _lib.load()
    _req(gray, "depth_map", torch.float32)
    _req(windows, "interval_windows", torch.float32)
    _req(n_windows, "n_windows", torch.int32)
    B = gray.shape[0]
    if windows.shape != (B, 3, 2) or n_windows.shape != (B,):
        raise RgbdB200Error("depth_region_codes: windows must be (B,3,2) and n_windows (B,)")
    codes = torch.empty(gray.shape, device=gray.device, dtype=torch.uint8)
    ws = torch.empty(int(lib.rgbd_depth_helper_workspace_bytes(B)), device=gray.device, dtype=torch.uint8)
    check(lib.rgbd_depth_region_codes(gray.data_ptr(), windows.data_ptr(), n_windows.data_ptr(), B, gray[0].numel(),
                                      codes.data_ptr(), ws.data_ptr(), _stream()), "rgbd_depth_region_codes")
    _count(2)
    return codes


def resize_pil_bilinear(img_u8: torch.Tensor, size: Tuple[int, int]) -> torch.Tensor:
    """(B,H,W,C) or (B,H,W) uint8 -> (B,h,w[,C]) uint8, bit-exact with ``PIL.Image.resize((w,h), BILINEAR)`` -- the resize
    of the HF image processor (PIL backend) the reference's mapper runs on the colour image and on ``depth.convert('RGB')``."""
    lib = _lib.load()
    _req(img_u8, "image", torch.uint8)
    squeeze = img_u8.dim() == 3
    x = img_u8[..., None] if squeeze else img_u8
    B, H, W, Cc = x.shape
    h, w = int(size[0]), int(size[1])
    out = torch.empty(B, h, w, Cc, device=x.device, dtype=torch.uint8)
    ws = torch.empty(max(int(lib.rgbd_resize_workspace_bytes(B, H, W, Cc, h, w)), 16), device=x.device, dtype=torch.uint8)
    check(lib.rgbd_resize_pil_bilinear_u8(x.data_ptr(), out.data_ptr(), B, H, W, Cc, h, w, ws.data_ptr(), _stream()),
          "rgbd_resize_pil_bilinear_u8")
    _count(4)
    return out[..., 0] if squeeze else out


def resize_cv_linear(img_u8: torch.Tensor, size: Tuple[int, int]) -> torch.Tensor:
    """(B,H,W) uint8 -> (B,h,w) uint8, bit-exact with ``cv2.resize(img, (w,h), interpolation=cv2.INTER_LINEAR)`` (DL:413)."""
    lib = _lib.load()
    _req(img_u8, "image", torch.uint8)
    B, H, W = img_u8.shape
    h, w = int(size[0]), int(size[1])
    out = torch.empty(B, h, w, device=img_u8.device, dtype=torch.uint8)
    ws = torch.empty(max(int(lib.rgbd_resize_workspace_bytes(B, H, W, 1, h, w)), 16), device=img_u8.device, dtype=torch.uint8)
    check(lib.rgbd_resize_cv_linear_u8(img_u8.data_ptr(), out.data_ptr(), B, H, W, h, w, ws.data_ptr(), _stream()),
          "rgbd_resize_cv_linear_u8")
    _count(3)
    return out


def map_10channel(rgb_u8: torch.Tensor, depth_u8: torch.Tensor, size: Optional[Tuple[int, int]] = (384, 384),
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The whole ``map_10channel_case2`` front-end (DL:386-425) on device: camera-resolution uint8 colour (B,H,W,3) and
    depth (B,H,W) -> ``pixel_values`` (B,10,h,w): Pillow-bilinear resize of colour and of the 3x-replicated depth (HF
    processor, ``size`` of preprocessor_config.json), rescale + normalise, OpenCV-linear resize of the depth for the Sobel
    gradient features (DL:413-414) and the validity mask.  ``size=None`` keeps the input resolution."""
    B, H, W = depth_u8.shape
    h, w = (H, W) if size is None else (int(size[0]), int(size[1]))
    if (h, w) == (H, W):
        return pack_pixel_values(rgb_u8, depth_u8, out=out)
    rgb_r = resize_pil_bilinear(rgb_u8, (h, w))
    depth_pil = resize_pil_bilinear(depth_u8, (h, w))          # per-channel filter: resizing 'L' then replicating == 'RGB'
    depth_cv = resize_cv_linear(depth_u8, (h, w))
    pv = pack_pixel_values(rgb_r, depth_pil, out=out)
    gradient_features(depth_cv, norm_out=pv[:, 6:9], vmask_out=pv[:, 9:10])     # DL:413-414: features of the OpenCV resize
    return pv


# ------------------------------------------------------------------------------------------------
# E-DSAM depth decomposition
# ------------------------------------------------------------------------------------------------
@dataclass
class Decomposition:
    gray: torch.Tensor                 # (B,H,W) f32
    codes: Optional[torch.Tensor]      # (B,H,W) u8, bit t = region mask t (None when not requested)
    pooled: List[torch.Tensor]         # per level (B,h,w) u8
    n_modes: torch.Tensor              # (B) i32
    centres: torch.Tensor              # (B,3) f32
    windows: torch.Tensor              # (B,3,2) f32
    peak_bins: torch.Tensor            # (B,3) i32
    status: torch.Tensor               # (B) i32
    bias_variant: torch.Tensor         # (B) i32: number of DSAM conv biases the reference adds for the image
    hist: Optional[torch.Tensor] = None    # (B,512) i64
    edges: Optional[torch.Tensor] = None   # (B,513) f32


def depth_decompose(ratio: torch.Tensor, levels: Sequence[Tuple[int, int]], depth3: Optional[torch.Tensor] = None,
                    gray: Optional[torch.Tensor] = None, num_modes: int = 3, debug: bool = False,
                    want_codes: bool = True) -> Decomposition:
    """K2.  Exactly one of depth3 (B,3,H,W) / gray (B,H,W).  ratio (B) float32.  ``want_codes=False`` skips the
    full-resolution code image when the levels are the aligned (H/4, H/8, H/16) pyramid (the DSAM stages only read the
    pooled copies)."""
    lib = _lib.load()
    if (depth3 is None) == (gray is None):
        raise RgbdB200Error("pass exactly one of depth3 / gray")
    _req(ratio, "ratio", torch.float32)
    if depth3 is not None:
        _req(depth3, "depth", torch.float32, False)
        B, c3, H, W = depth3.shape
        if c3 != 3:
            raise RgbdB200Error("depth must have 3 channels")
        dbs, dcs = _plane_strided(depth3, "depth")
        dev = depth3.device
        gray_out = torch.empty(B, H, W, device=dev, dtype=torch.float32)
        d3p, gip = depth3.data_ptr(), None
    else:
        _req(gray, "gray", torch.float32)
        B, H, W = gray.shape
        dev = gray.device
        gray_out = gray
        dbs = dcs = 0
        d3p, gip = None, gray.data_ptr()
    if ratio.numel() != B:
        raise RgbdB200Error(f"ratio must have {B} elements")
    pyramid = (len(levels) == 3 and H % 16 == 0 and W % 16 == 0
               and all(tuple(lv) == (H >> (2 + k), W >> (2 + k)) for k, lv in enumerate(levels)))
    codes = torch.empty(B, H, W, device=dev, dtype=torch.uint8) if (want_codes or not pyramid) else None
    pooled = [torch.empty(B, h, w, device=dev, dtype=torch.uint8) for h, w in levels]
    # the per-image tables share one allocation (six tiny tensors cost more host time than the kernels they feed)
    small = torch.empty(15 * B, device=dev, dtype=torch.int32)
    n_modes, status, bias_variant = small[0:B], small[B:2 * B], small[2 * B:3 * B]
    peak_bins = small[3 * B:6 * B].view(B, 3)
    centres = small[6 * B:9 * B].view(torch.float32).view(B, 3)
    windows = small[9 * B:15 * B].view(torch.float32).view(B, 3, 2)
    hist = torch.empty(B, HIST_BINS, device=dev, dtype=torch.int64) if debug else None
    edges = torch.empty(B, HIST_BINS + 1, device=dev, dtype=torch.float32) if debug else None
    ws = torch.empty(int(lib.rgbd_depth_decompose_workspace_bytes(B)), device=dev, dtype=torch.uint8)
    rc = lib.rgbd_depth_decompose(
        d3p, dbs, dcs, gip, ratio.data_ptr(), B, H, W, num_modes,
        gray_out.data_ptr() if depth3 is not None else None,
        hist.data_ptr() if debug else None, edges.data_ptr() if debug else None,
        n_modes.data_ptr(), peak_bins.data_ptr(), centres.data_ptr(), windows.data_ptr(), status.data_ptr(),
        bias_variant.data_ptr(), codes.data_ptr() if codes is not None else None, len(levels), int_array([h for h, _ in levels]), int_array([w for _, w in levels]),
        ptr_array([p.data_ptr() for p in pooled]), ws.data_ptr(), _stream())
    check(rc, "rgbd_depth_decompose")
    _count((4 if pyramid else 5 if levels else 4) + (1 if debug else 0))
    return Decomposition(gray_out, codes, pooled, n_modes, centres, windows, peak_bins, status, bias_variant, hist, edges)


# ------------------------------------------------------------------------------------------------
# tensor-core building blocks
# ------------------------------------------------------------------------------------------------
POOL_FIXED_ONE = float(1 << 24)      # RGBD_POOL_FIXED_ONE: unit of the fixed-point cell sums of conv_gemm's epilogue mode 2


def best_box(out_h: int, out_w: int) -> Tuple[int, int]:
    """(bx, by) with bx*by == 128 covering an out_h x out_w image with the least padding (the GEMM's 128-pixel M tile)."""
    best, best_eff = (128, 1), -1.0
    for bx in (128, 64, 32, 16, 8, 4, 2, 1):
        by = 128 // bx
        cover = (-(-out_w // bx) * bx) * (-(-out_h // by) * by)
        eff = out_h * out_w / cover
        if eff > best_eff + 1e-9:
            best, best_eff = (bx, by), eff
    return best


def pick_block_n(n_pad: int) -> int:
    if n_pad <= 256:
        return n_pad
    for bn in range(256, 31, -32):
        if n_pad % bn == 0:
            return bn
    return 32


def conv_gemm(a: torch.Tensor, a_dims: Tuple[int, int, int, int], plane_per_img: int, w: torch.Tensor,
              slices: torch.Tensor, kb: int, n_img: int, out_hw: Tuple[int, int], box: Tuple[int, int], n: int,
              shift: torch.Tensor, *, scale: Optional[torch.Tensor] = None, variant: Optional[torch.Tensor] = None,
              act: int = 0, epi_mode: int = 0, gate: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
              residual: Optional[torch.Tensor] = None, pool: Optional[torch.Tensor] = None,
              cells: Tuple[int, int] = (0, 0), tile_order: int = 0, block_n: Optional[int] = None,
              conv3x3_reuse: bool = False, codes: Optional[torch.Tensor] = None, in_hw: Tuple[int, int] = (0, 0),
              parity: Tuple[int, int] = (0, 0), m3_stride: int = 1, m3_masked_segs: int = 0, m3_n_seg: int = 0,
              dsam_masked: bool = False, next_operand: Optional[torch.Tensor] = None,
              next_codes: Optional[torch.Tensor] = None, next_geom: Tuple[int, int, int] = (0, 0, 0),
              pool_sq: Optional[torch.Tensor] = None) -> None:
    """Launch the tcgen05 implicit-GEMM kernel.  a_dims = (planes, y, x, c) of the bf16 channels-last operand.
    ``conv3x3_reuse``: 3x3 stride-1 conv whose A tile is shared by the three dx taps (``slices`` may be None).
    ``dsam_masked``: stride-2 DSAM stage on the unmasked operand, region masking in shared memory (``slices`` None)."""
    lib = _lib.load()
    _req(a, "a", torch.bfloat16)
    _req(w, "w", torch.bfloat16)
    if slices is not None:
        _req(slices, "slices", torch.int32)
    if shift is not None:
        _req(shift, "shift", torch.float32)
    n_pad = w.shape[0]
    planes, ay, ax, ac = a_dims
    if a.numel() != planes * ay * ax * ac:
        raise RgbdB200Error("conv_gemm: operand size does not match a_dims")
    if dsam_masked:
        n_slices = 9 * (ac // 64) * m3_n_seg
    else:
        n_slices = slices.shape[0] if slices is not None else 9 * ac // kb
    if w.shape[1] != n_slices * kb:
        raise RgbdB200Error(f"conv_gemm: weight K {w.shape[1]} != n_slices*kb {n_slices * kb}")
    if (shift is not None and shift.shape[-1] != n_pad) or (scale is not None and scale.numel() != n_pad):
        raise RgbdB200Error("conv_gemm: scale/shift must have n_pad entries")
    d = ConvGemmDesc()
    d.a = a.data_ptr(); d.a_c = ac; d.a_x = ax; d.a_y = ay; d.a_planes = planes
    d.plane_per_img = plane_per_img
    d.w = w.data_ptr(); d.slices = slices.data_ptr() if slices is not None else None
    d.n_slices = n_slices; d.kb_elems = kb
    d.conv3x3_reuse = 1 if conv3x3_reuse else 0
    d.dsam_masked = 1 if dsam_masked else 0
    d.next_operand = _req(next_operand, "next_operand", torch.bfloat16).data_ptr() if next_operand is not None else None
    d.next_codes = _req(next_codes, "next_codes", torch.uint8).data_ptr() if next_codes is not None else None
    d.next_c_pad, d.next_n_seg, d.next_masked_segs = next_geom
    d.n_img = n_img; d.out_h, d.out_w = out_hw; d.bx, d.by = box
    d.n = n; d.n_pad = n_pad; d.block_n = block_n or pick_block_n(n_pad)
    d.tile_order = tile_order; d.epi_mode = epi_mode; d.act = act
    d.scale = _req(scale, "scale", torch.float32).data_ptr() if scale is not None else None
    d.shift = shift.data_ptr() if shift is not None else None
    d.codes = _req(codes, "codes", torch.uint8).data_ptr() if codes is not None else None
    d.in_h, d.in_w = in_hw
    d.m3_py, d.m3_px = parity
    d.m3_stride = m3_stride; d.m3_masked_segs = m3_masked_segs; d.m3_n_seg = m3_n_seg
    d.variant = _req(variant, "variant", torch.int32).data_ptr() if variant is not None else None
    d.gate = _req(gate, "gate", torch.bfloat16).data_ptr() if gate is not None else None
    d.out = out.data_ptr() if out is not None else None
    d.residual = _req(residual, "residual", torch.float32).data_ptr() if residual is not None else None
    d.pool = _req(pool, "pool", torch.int64).data_ptr() if pool is not None else None
    d.pool_sq = _req(pool_sq, "pool_sq", torch.int64).data_ptr() if pool_sq is not None else None
    d.cells_y, d.cells_x = cells
    check(lib.rgbd_conv_gemm(C.byref(d), _stream()), "rgbd_conv_gemm")
    _count(1)


def dsam_pack(feat: torch.Tensor, codes: torch.Tensor, out: torch.Tensor, c_pad: int, n_seg: int, masked_segs: int,
              parity_split: bool, hi_lo: bool = False) -> None:
    lib = _lib.load()
    _req(feat, "feat", torch.float32)
    _req(codes, "codes", torch.uint8)
    _req(out, "packed", torch.bfloat16)
    B, Cc, H, W = feat.shape
    if codes.shape != (B, H, W):
        raise RgbdB200Error(f"codes must be {(B, H, W)}, got {tuple(codes.shape)}")
    check(lib.rgbd_dsam_pack(feat.data_ptr(), codes.data_ptr(), out.data_ptr(), B, Cc, c_pad, H, W, n_seg, masked_segs,
                             1 if parity_split else 0, 1 if hi_lo else 0, _stream()), "rgbd_dsam_pack")
    _count(1)


def project_group_norm(x: torch.Tensor, conv_w: torch.Tensor, conv_b: Optional[torch.Tensor], gn_w: torch.Tensor,
                       gn_b: torch.Tensor, groups: int, eps: float, w_cache: Optional[dict] = None) -> torch.Tensor:
    """``Sequential(Conv2d(C, N, 1), GroupNorm(groups, N))`` -- an ``input_projections`` / lateral ``adapter`` entry of HF's
    ``Mask2FormerPixelDecoder`` (called at CM:383; SURVEY 8f-2) -- on this library's kernels: fp32 NCHW (B,C,h,w) -> bf16
    channels-last copy -> tcgen05 1x1-conv GEMM (fp32 accumulate, fp32 NCHW out) -> in-place GroupNorm.  Inference only."""
    lib = _lib.load()
    _req(x, "features", torch.float32)
    B, Cc, h, w = x.shape
    N = conv_w.shape[0]
    if conv_w.shape[1] != Cc or N % 32 or N > 256:
        raise RgbdB200Error("project_group_norm: conv must be (N, C, 1, 1) with N a multiple of 32, at most 256")
    c_pad = (Cc + 63) // 64 * 64
    key = (conv_w.data_ptr(), conv_w._version, c_pad)
    if w_cache is not None and w_cache.get("key") == key:
        wk, sl, bias = w_cache["w"], w_cache["sl"], w_cache["b"]
    else:
        wk = torch.zeros(N, c_pad, device=x.device, dtype=torch.float32)
        wk[:, :Cc] = conv_w.detach().reshape(N, Cc).float()
        wk = wk.to(torch.bfloat16).contiguous()
        sl = torch.tensor([(64 * cb, 0, 0, 0) for cb in range(c_pad // 64)], device=x.device, dtype=torch.int32)
        bias = (conv_b.detach().float() if conv_b is not None else torch.zeros(N, device=x.device)).contiguous()
        if w_cache is not None:
            w_cache.update(key=key, w=wk, sl=sl, b=bias)
    a = torch.empty(B, h, w, c_pad, device=x.device, dtype=torch.bfloat16)
    check(lib.rgbd_dsam_pack(x.data_ptr(), None, a.data_ptr(), B, Cc, c_pad, h, w, 1, 0, 0, 0, _stream()), "rgbd_dsam_pack")
    _count(1)
    out = torch.empty(B, N, h, w, device=x.device, dtype=torch.float32)
    conv_gemm(a, (B, h, w, c_pad), 1, wk, sl, 64, B, (h, w), best_box(h, w), N, bias, epi_mode=1, out=out)
    check(lib.rgbd_group_norm_inplace(out.data_ptr(), _req(gn_w.detach().float().contiguous(), "gamma", torch.float32).data_ptr(),
                                      _req(gn_b.detach().float().contiguous(), "beta", torch.float32).data_ptr(), B, N, h * w,
                                      int(groups), float(eps), _stream()), "rgbd_group_norm_inplace")
    _count(1)
    return out


def cast_bf16_pitched(src: torch.Tensor, w_pitch: int, lo: bool = False):
    """(..., W) fp32 -> (..., w_pitch) bf16, zero padded (TMA row strides must be multiples of 16 bytes).  With ``lo``
    returns (hi, lo): hi = bf16(v) and lo = bf16(v - hi) in the same layout (split-precision operands)."""
    lib = _lib.load()
    _req(src, "src", torch.float32)
    W = src.shape[-1]
    rows = src.numel() // W
    out = torch.empty(*src.shape[:-1], w_pitch, device=src.device, dtype=torch.bfloat16)
    out_lo = torch.empty_like(out) if lo else None
    check(lib.rgbd_cast_bf16_pitched(src.data_ptr(), out.data_ptr(), out_lo.data_ptr() if lo else None, rows, W, w_pitch,
                                     _stream()), "rgbd_cast_bf16_pitched")
    _count(1)
    return (out, out_lo) if lo else out


def dsam_pack_t(feat: torch.Tensor, codes: torch.Tensor, out: torch.Tensor, c_pad: int, w2_pitch: int, n_seg: int,
                masked_segs: int, parity_split: bool, out_lo: Optional[torch.Tensor] = None) -> None:
    """``out_lo`` (same shape as ``out``, zeroed like it): also write the lo parts bf16(v - bf16(v))."""
    lib = _lib.load()
    _req(feat, "feat", torch.float32)
    _req(codes, "codes", torch.uint8)
    _req(out, "packed", torch.bfloat16)
    if out_lo is not None:
        _req(out_lo, "packed_lo", torch.bfloat16)
        if out_lo.shape != out.shape:
            raise RgbdB200Error(f"dsam_pack_t: out_lo must be {tuple(out.shape)}, got {tuple(out_lo.shape)}")
    B, Cc, H, W = feat.shape
    check(lib.rgbd_dsam_pack_t(feat.data_ptr(), codes.data_ptr(), out.data_ptr(),
                               out_lo.data_ptr() if out_lo is not None else None, B, Cc, c_pad, H, W, w2_pitch, n_seg,
                               masked_segs, 1 if parity_split else 0, _stream()), "rgbd_dsam_pack_t")
    _count(1)


def dsam_dbias(g: torch.Tensor, variant: Optional[torch.Tensor], n_bias: int) -> torch.Tensor:
    lib = _lib.load()
    _req(g, "grad_output", torch.float32)
    B, N, Ho, Wo = g.shape
    db = torch.empty(n_bias, N, device=g.device, dtype=torch.float32)
    check(lib.rgbd_dsam_dbias(g.data_ptr(), _req(variant, "variant", torch.int32).data_ptr() if variant is not None else None,
                              db.data_ptr(), B, N, Ho * Wo, n_bias, _stream()), "rgbd_dsam_dbias")
    _count(1)
    return db


def dsam_wgrad(g_bf16: torch.Tensor, xt: torch.Tensor, n_out: int, c_pad: int, out_hw: Tuple[int, int], n_seg: int,
               parity_split: bool, g_lo: Optional[torch.Tensor] = None, xt_lo: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dW[n][seg][tap][c_pad] fp32.  g_bf16: (B, n_out, Ho, Wp); xt: (B, n_seg, n_par, c_pad, H2, W2p).  With both lo
    parts (``cast_bf16_pitched(lo=True)``, ``dsam_pack_t(out_lo=...)``): split precision, g_hi.x_hi + g_lo.x_hi + g_hi.x_lo."""
    lib = _lib.load()
    _req(g_bf16, "g", torch.bfloat16)
    _req(xt, "x_t", torch.bfloat16)
    if (g_lo is None) != (xt_lo is None):
        raise RgbdB200Error("dsam_wgrad: give both lo parts (split precision) or neither")
    if g_lo is not None:
        _req(g_lo, "g_lo", torch.bfloat16)
        _req(xt_lo, "x_t_lo", torch.bfloat16)
        if g_lo.shape != g_bf16.shape or xt_lo.shape != xt.shape:
            raise RgbdB200Error("dsam_wgrad: lo parts must have the shapes of the hi parts")
    B = g_bf16.shape[0]
    taps = 9 if parity_split else 1
    dw = torch.empty(n_out, n_seg, taps, c_pad, device=g_bf16.device, dtype=torch.float32)
    check(lib.rgbd_dsam_wgrad(g_bf16.data_ptr(), g_lo.data_ptr() if g_lo is not None else None, g_bf16.shape[-1],
                              xt.data_ptr(), xt_lo.data_ptr() if xt_lo is not None else None, xt.shape[-1], xt.shape[-2],
                              dw.data_ptr(), B, n_out, c_pad, out_hw[0], out_hw[1], n_seg, 1 if parity_split else 0,
                              _stream()),
          "rgbd_dsam_wgrad")
    _count(1)
    return dw


def ratio_stem_pack(depth3: torch.Tensor, out: torch.Tensor) -> None:
    lib = _lib.load()
    _req(depth3, "depth", torch.float32, False)
    _req(out, "stem operand", torch.bfloat16)
    B, c3, H, W = depth3.shape
    if not 1 <= c3 <= 4:
        raise RgbdB200Error("the stem operand holds 1..4 input channels")
    bs, cs = _plane_strided(depth3, "depth")
    check(lib.rgbd_ratio_stem_pack(depth3.data_ptr(), bs, cs, out.data_ptr(), B, c3, H, W, _stream()), "rgbd_ratio_stem_pack")
    _count(1)


def ratio_stem_compact_width(W: int) -> int:
    return int(_lib.load().rgbd_ratio_stem_compact_width(int(W)))


def ratio_stem_pack_compact(depth3: torch.Tensor, out: torch.Tensor) -> None:
    """depth (B,3,H,W) fp32 -> E (B,2,H+6,Wp,4) bf16: channels-last depth with zero borders, two copies shifted by one pixel."""
    lib = _lib.load()
    _req(depth3, "depth", torch.float32, False)
    _req(out, "compact stem operand", torch.bfloat16)
    B, c3, H, W = depth3.shape
    if out.shape != (B, 2, H + 6, ratio_stem_compact_width(W), 4):
        raise RgbdB200Error("ratio_stem_pack_compact: out must be (B,2,H+6,Wp,4)")
    if not 1 <= c3 <= 4:
        raise RgbdB200Error("the stem operand holds 1..4 input channels")
    bs, cs = _plane_strided(depth3, "depth")
    check(lib.rgbd_ratio_stem_pack_compact(depth3.data_ptr(), bs, cs, out.data_ptr(), B, c3, H, W, _stream()),
          "rgbd_ratio_stem_pack_compact")
    _count(1)


def ratio_front(r: torch.Tensor, w1: torch.Tensor, w2: torch.Tensor, w3: torch.Tensor, w4: torch.Tensor, sh1: torch.Tensor,
                sh2: torch.Tensor, sh3: torch.Tensor, sh4: torch.Tensor, out: torch.Tensor, box: Tuple[int, int]) -> None:
    """K4a+K4b in one kernel: stem GEMM + BN + ReLU, feature_fusion, attention and gating (CM:1458-1470) with every
    intermediate in tensor memory -> out (B,H,W,128) bf16.  ``r`` is either the row-im2col tensor (B,H+6,W,64) with
    w1 (192,256), or the compact operand (B,2,H+6,Wp,4) of ``ratio_stem_pack_compact`` with w1 (192,224)."""
    lib = _lib.load()
    _req(r, "r", torch.bfloat16)
    _req(out, "out", torch.bfloat16)
    compact = r.dim() == 5
    if compact:
        B, two, H6, Wp, c = r.shape
        W = out.shape[2]
        ok = two == 2 and c == 4 and Wp == ratio_stem_compact_width(W)
        k1 = 224
    else:
        B, H6, W, c = r.shape
        ok = c == 64
        k1 = 256
    H = H6 - 6
    if not ok or H < 1 or out.shape != (B, H, W, 128):
        raise RgbdB200Error("ratio_front: r must be (B,H+6,W,64) or (B,2,H+6,Wp,4) and out (B,H,W,128)")
    for t, shp in ((w1, (192, k1)), (w2, (128, 192)), (w3, (64, 128)), (w4, (128, 64))):
        _req(t, "front weight", torch.bfloat16)
        if tuple(t.shape) != shp:
            raise RgbdB200Error(f"ratio_front: weight shape {tuple(t.shape)} != {shp}")
    for t, n in ((sh1, 192), (sh2, 128), (sh3, 64), (sh4, 128)):
        _req(t, "front shift", torch.float32)
        if t.numel() != n:
            raise RgbdB200Error("ratio_front: bad shift length")
    check(lib.rgbd_ratio_front(r.data_ptr(), w1.data_ptr(), w2.data_ptr(), w3.data_ptr(), w4.data_ptr(), sh1.data_ptr(),
                               sh2.data_ptr(), sh3.data_ptr(), sh4.data_ptr(), out.data_ptr(), B, H, W, box[0], box[1],
                               1 if compact else 0, _stream()), "rgbd_ratio_front")
    _count(1)


def ratio_chain(x1: torch.Tensor, w2: torch.Tensor, w3: torch.Tensor, w4: torch.Tensor, sh2: torch.Tensor,
                sh3: torch.Tensor, sh4: torch.Tensor, out: torch.Tensor, box: Tuple[int, int]) -> None:
    """K4b.  x1 (B,H,W,192) bf16 -> out (B,H,W,128) bf16 = f * sigmoid(W4 relu(W3 f + b3) + b4), f = relu(W2' x1 + sh2)
    where W2' already carries the folded BatchNorm scale."""
    lib = _lib.load()
    _req(x1, "x1", torch.bfloat16)
    _req(out, "out", torch.bfloat16)
    B, H, W, c = x1.shape
    if c != 192 or out.shape != (B, H, W, 128):
        raise RgbdB200Error("ratio_chain: x1 must be (B,H,W,192) and out (B,H,W,128)")
    for t, shp in ((w2, (128, 192)), (w3, (64, 128)), (w4, (128, 64))):
        _req(t, "chain weight", torch.bfloat16)
        if tuple(t.shape) != shp:
            raise RgbdB200Error(f"ratio_chain: weight shape {tuple(t.shape)} != {shp}")
    for t, n in ((sh2, 128), (sh3, 64), (sh4, 128)):
        _req(t, "chain scale/shift", torch.float32)
        if t.numel() != n:
            raise RgbdB200Error("ratio_chain: bad scale/shift length")
    check(lib.rgbd_ratio_chain(x1.data_ptr(), w2.data_ptr(), w3.data_ptr(), w4.data_ptr(), sh2.data_ptr(),
                               sh3.data_ptr(), sh4.data_ptr(), out.data_ptr(), B, H, W, box[0], box[1], _stream()),
          "rgbd_ratio_chain")
    _count(1)


def ratio_tail(pool: torch.Tensor, cell_pixels: int, conv_w: torch.Tensor, conv_scale: torch.Tensor,
               conv_shift: torch.Tensor, fc_w: Sequence[torch.Tensor], fc_b: Sequence[torch.Tensor],
               out_min: float, out_max: float) -> torch.Tensor:
    lib = _lib.load()
    _req(pool, "pool", torch.int64)
    B = pool.shape[0]
    gap = torch.empty(B, 512, device=pool.device, dtype=torch.float32)
    ratio = torch.empty(B, 1, device=pool.device, dtype=torch.float32)
    for t in (conv_w, conv_scale, conv_shift, *fc_w, *fc_b):
        _req(t, "ratio tail parameter", torch.float32)
    check(lib.rgbd_ratio_tail(pool.data_ptr(), pool.shape[-1], cell_pixels, conv_w.data_ptr(), conv_scale.data_ptr(),
                              conv_shift.data_ptr(), ptr_array([t.data_ptr() for t in fc_w]),
                              ptr_array([t.data_ptr() for t in fc_b]), out_min, out_max, gap.data_ptr(),
                              ratio.data_ptr(), B, _stream()), "rgbd_ratio_tail")
    _count(2)
    return ratio


def adaptive_avg_pool4(x5: torch.Tensor, pool: torch.Tensor) -> None:
    """``AdaptiveAvgPool2d(4)`` (CM:1417) of the bf16 channels-last (B,H,W,256) map into ``pool`` (B,16,256) int64 as fixed-
    point window means (read them with ``cell_pixels = 1``); the path for H or W not divisible by 4."""
    lib = _lib.load()
    _req(x5, "x5", torch.bfloat16)
    _req(pool, "pool", torch.int64)
    B, H, W, c = x5.shape
    if c != 256 or pool.shape != (B, 16, 256):
        raise RgbdB200Error("adaptive_avg_pool4: x5 must be (B,H,W,256) and pool (B,16,256)")
    check(lib.rgbd_adaptive_avg_pool4(x5.data_ptr(), pool.data_ptr(), B, H, W, _stream()), "rgbd_adaptive_avg_pool4")
    _count(1)


def ratio_tail_tc(pool: torch.Tensor, cell_pixels: int, a6: torch.Tensor, gap_fx: torch.Tensor, w6_bf16: torch.Tensor,
                  slices: torch.Tensor, shift6: torch.Tensor, fc_w: Sequence[torch.Tensor], fc_b: Sequence[torch.Tensor],
                  out_min: float, out_max: float) -> torch.Tensor:
    """CM:1473-1485 with the 3x3 256->512 conv on the tensor cores: pooled sums -> bf16 4x4 map ``a6`` (B,4,4,256) ->
    implicit GEMM (M = 16 pixels per image, N = 512, K = 2304; BatchNorm scale folded into ``w6_bf16`` (512, 9*256), ReLU and
    the global average pool in the epilogue) -> MLP -> ratio (B,1).  ``gap_fx`` (B,1,512) int64 is scratch."""
    lib = _lib.load()
    _req(pool, "pool", torch.int64)
    _req(a6, "a6", torch.bfloat16)
    _req(gap_fx, "gap_fx", torch.int64)
    B = pool.shape[0]
    if a6.shape != (B, 4, 4, 256) or gap_fx.numel() != B * 512:
        raise RgbdB200Error("ratio_tail_tc: a6 must be (B,4,4,256) and gap_fx (B,1,512)")
    for t in (*fc_w, *fc_b):
        _req(t, "ratio tail parameter", torch.float32)
    check(lib.rgbd_ratio_tail_prepare(pool.data_ptr(), pool.shape[-1], cell_pixels, a6.data_ptr(), gap_fx.data_ptr(), B, _stream()),
          "rgbd_ratio_tail_prepare")
    _count(1)
    conv_gemm(a6, (B, 4, 4, 256), 1, w6_bf16, slices, 64, B, (4, 4), (4, 32), 512, shift6, act=1, epi_mode=2, pool=gap_fx,
              cells=(1, 1))
    ratio = torch.empty(B, 1, device=pool.device, dtype=torch.float32)
    check(lib.rgbd_ratio_tail_mlp_fx(gap_fx.data_ptr(), ptr_array([t.data_ptr() for t in fc_w]),
                                     ptr_array([t.data_ptr() for t in fc_b]), out_min, out_max, ratio.data_ptr(), B, _stream()),
          "rgbd_ratio_tail_mlp_fx")
    _count(1)
    return ratio


def ratio_tail_train(pool: torch.Tensor, cell_pixels: int, conv_w: torch.Tensor, conv_bias: torch.Tensor,
                     bn_gamma: torch.Tensor, bn_beta: torch.Tensor, eps: float, momentum: float,
                     running_mean: Optional[torch.Tensor], running_var: Optional[torch.Tensor],
                     fc_w: Sequence[torch.Tensor], fc_b: Sequence[torch.Tensor], drop0: Optional[torch.Tensor],
                     drop1: Optional[torch.Tensor], out_min: float, out_max: float) -> torch.Tensor:
    """The predictor's tail under ``.train()`` (CM:1418-1437): batch-statistics BatchNorm2d(512) (running statistics
    updated IN PLACE when given) and Dropout multipliers ``keep / (1 - p)`` of shape (B,128) / (B,64)."""
    lib = _lib.load()
    _req(pool, "pool", torch.int64)
    B = pool.shape[0]
    dev = pool.device
    for t in (conv_w, conv_bias, bn_gamma, bn_beta, *fc_w, *fc_b):
        _req(t, "ratio tail parameter", torch.float32)
    for t, n in ((drop0, 128), (drop1, 64)):
        if t is not None:
            _req(t, "dropout multiplier", torch.float32)
            if tuple(t.shape) != (B, n):
                raise RgbdB200Error(f"dropout multiplier must be {(B, n)}, got {tuple(t.shape)}")
    if (running_mean is None) != (running_var is None):
        raise RgbdB200Error("pass both running statistics or neither")
    if running_mean is not None:
        _req(running_mean, "running_mean", torch.float32)
        _req(running_var, "running_var", torch.float32)
    raw = torch.empty(B, 512, 16, device=dev, dtype=torch.float32)
    gap = torch.empty(B, 512, device=dev, dtype=torch.float32)
    ratio = torch.empty(B, 1, device=dev, dtype=torch.float32)
    check(lib.rgbd_ratio_tail_train(
        pool.data_ptr(), pool.shape[-1], cell_pixels, conv_w.data_ptr(), conv_bias.data_ptr(), bn_gamma.data_ptr(),
        bn_beta.data_ptr(), float(eps), float(momentum), running_mean.data_ptr() if running_mean is not None else None,
        running_var.data_ptr() if running_var is not None else None, ptr_array([t.data_ptr() for t in fc_w]),
        ptr_array([t.data_ptr() for t in fc_b]), drop0.data_ptr() if drop0 is not None else None,
        drop1.data_ptr() if drop1 is not None else None, out_min, out_max, raw.data_ptr(), gap.data_ptr(), ratio.data_ptr(),
        B, _stream()), "rgbd_ratio_tail_train")
    _count(3)
    return ratio


def ratio_from_features(feats: Sequence[torch.Tensor], fc_w: Sequence[torch.Tensor], fc_b: Sequence[torch.Tensor],
                        out_min: float, out_max: float) -> torch.Tensor:
    """K6: ``RatioPredictor.forward`` (CM:860-898) -- GAP of every depth feature map, concat, 3-layer MLP -> (B,1)."""
    lib = _lib.load()
    feats = [_req(f.contiguous(), "depth feature map", torch.float32) for f in feats]
    B = feats[0].shape[0]
    for t in (*fc_w, *fc_b):
        _req(t, "ratio predictor parameter", torch.float32)
    c_total = sum(f.shape[1] for f in feats)
    if fc_w[0].shape != (64, c_total) or fc_w[1].shape != (32, 64) or fc_w[2].shape != (1, 32):
        raise RgbdB200Error("ratio_from_features: fc layers must be (64, sum C), (32, 64), (1, 32)")
    pooled = torch.empty(B, c_total, device=feats[0].device, dtype=torch.float32)
    ratio = torch.empty(B, 1, device=feats[0].device, dtype=torch.float32)
    cs = (C.c_int * len(feats))(*[f.shape[1] for f in feats])
    hws = (C.c_int * len(feats))(*[f.shape[2] * f.shape[3] for f in feats])
    check(lib.rgbd_ratio_from_features(len(feats), ptr_array([f.data_ptr() for f in feats]), cs, hws, B,
                                       ptr_array([t.data_ptr() for t in fc_w]), ptr_array([t.data_ptr() for t in fc_b]),
                                       float(out_min), float(out_max), pooled.data_ptr(), ratio.data_ptr(), _stream()),
          "rgbd_ratio_from_features")
    _count(2)
    return ratio


# ------------------------------------------------------------------------------------------------
# instance post-processing (SURVEY 8f-3)
# ------------------------------------------------------------------------------------------------
@dataclass
class InstanceBatch:
    """Device-side result of ``post_process_instances``; entries ``[b, :count[b]]`` are valid, in candidate order."""
    masks: torch.Tensor                # (B,Q,Ht,Wt) u8 0/1
    labels: torch.Tensor               # (B,Q) i32
    scores: torch.Tensor               # (B,Q) f32 (unrounded)
    query: torch.Tensor                # (B,Q) i32  query index of the segment
    count: torch.Tensor                # (B,) i32
    segmentation: Optional[torch.Tensor]   # (B,Ht,Wt) i32, -1 background


def post_process_instances(class_logits: torch.Tensor, mask_logits: torch.Tensor, threshold: float = 0.5,
                           target_size: Optional[Tuple[int, int]] = None, want_segmentation: bool = True) -> InstanceBatch:
    """HF ``post_process_instance_segmentation`` (model_essential_part.py:86-91) for a batch sharing one target size,
    without host synchronisation.  ``target_size=None`` keeps HF's 384x384 maps."""
    lib = _lib.load()
    _req(class_logits, "class_queries_logits", torch.float32)
    _req(mask_logits, "masks_queries_logits", torch.float32)
    if class_logits.dim() != 3 or mask_logits.dim() != 4 or class_logits.shape[:2] != mask_logits.shape[:2]:
        raise RgbdB200Error("post_process_instances: expected (B,Q,C+1) class logits and (B,Q,h,w) mask logits")
    B, Q, C1 = class_logits.shape
    h, w = mask_logits.shape[2:]
    Ht, Wt = (384, 384) if target_size is None else (int(target_size[0]), int(target_size[1]))
    dev = class_logits.device
    ws = torch.empty(max(int(lib.rgbd_postprocess_workspace_bytes(B, Q)), 16), device=dev, dtype=torch.uint8)
    masks = torch.empty(B, Q, Ht, Wt, device=dev, dtype=torch.uint8)
    labels = torch.empty(B, Q, device=dev, dtype=torch.int32)
    scores = torch.empty(B, Q, device=dev, dtype=torch.float32)
    query = torch.empty(B, Q, device=dev, dtype=torch.int32)
    count = torch.empty(B, device=dev, dtype=torch.int32)
    seg = torch.empty(B, Ht, Wt, device=dev, dtype=torch.int32) if want_segmentation else None
    check(lib.rgbd_postprocess_instances(class_logits.data_ptr(), mask_logits.data_ptr(), B, Q, C1, h, w, Ht, Wt,
                                         float(threshold), ws.data_ptr(), masks.data_ptr(), labels.data_ptr(),
                                         scores.data_ptr(), query.data_ptr(), count.data_ptr(),
                                         seg.data_ptr() if seg is not None else None, _stream()),
          "rgbd_postprocess_instances")
    _count(4 if (Ht >= 384 and Wt >= 384) else 5)      # select, grid, [target any], finalize, paint
    return InstanceBatch(masks, labels, scores, query, count, seg)


@dataclass
class RunLengths:
    """Device-side result of ``label_map_rle`` (CSR).  The runs of label ``k = id + 1`` in image ``b`` are
    ``runs[base[b] + offsets[b, k] : base[b] + offsets[b, k + 1]]``; the batch uses ``runs[:base[B]]``."""
    offsets: torch.Tensor              # (B, L+2) i32, relative to the image's base
    base: torch.Tensor                 # (B+1,) i32
    runs: torch.Tensor                 # (B*H*W, 2) i32: (start, end), 1-based, end inclusive
    bad: torch.Tensor                  # (1,) i32: pixels whose label lies outside [-1, L)


def _rle_workspace_bytes(B: int, H: int, W: int, L: int) -> int:
    ws_bytes = int(_lib.load().rgbd_label_map_rle_workspace_bytes(B, H, W, L))
    if ws_bytes == 0:
        raise RgbdB200Error(f"label_map_rle: unsupported shape (B,H,W)={(B, H, W)} or label count {L} "
                            "(at most 4096 labels, 65535 images, B*H*W < 2^31)")
    return ws_bytes


def _rle_outputs(B: int, H: int, W: int, L: int, device) -> RunLengths:
    i32 = dict(device=device, dtype=torch.int32)
    return RunLengths(torch.empty(B, L + 2, **i32), torch.empty(B + 1, **i32), torch.empty(B * H * W, 2, **i32),
                      torch.empty(1, **i32))


def label_map_rle_buffers(B: int, H: int, W: int, n_labels: int, device) -> Tuple[RunLengths, torch.Tensor]:
    """Output tensors and workspace of ``label_map_rle`` for (B,H,W) maps, to pass as ``out`` / ``workspace``."""
    ws_bytes = _rle_workspace_bytes(B, H, W, int(n_labels))          # checks the arguments before anything is allocated
    return _rle_outputs(B, H, W, int(n_labels), device), torch.empty(ws_bytes, device=device, dtype=torch.uint8)


def label_map_rle(seg: torch.Tensor, n_labels: int, out: Optional[RunLengths] = None,
                  workspace: Optional[torch.Tensor] = None) -> RunLengths:
    """Run-length encoding of (B,H,W) int32 label maps with labels in [-1, n_labels) (HF ``convert_segmentation_to_rle``
    per image), without host synchronisation.  Out-of-range pixels are counted in ``bad``, never encoded: check it.
    ``out`` / ``workspace`` (from ``label_map_rle_buffers``) are used in place when given; either one may be given alone."""
    lib = _lib.load()
    _req(seg, "seg", torch.int32)
    if seg.dim() != 3:
        raise RgbdB200Error("label_map_rle: expected a (B,H,W) int32 label map")
    B, H, W = seg.shape
    L = int(n_labels)
    ws_bytes = _rle_workspace_bytes(B, H, W, L)
    if out is None:
        out = _rle_outputs(B, H, W, L, seg.device)
    if workspace is None:
        workspace = torch.empty(ws_bytes, device=seg.device, dtype=torch.uint8)
    want = [(out.offsets, (B, L + 2)), (out.base, (B + 1,)), (out.runs, (B * H * W, 2)), (out.bad, (1,))]
    for t, shape in want:
        _req(t, "label_map_rle output", torch.int32)
        if tuple(t.shape) != shape:
            raise RgbdB200Error(f"label_map_rle: output of shape {tuple(t.shape)}, expected {shape}")
    _req(workspace, "label_map_rle workspace", torch.uint8)
    if workspace.numel() < ws_bytes:
        raise RgbdB200Error("label_map_rle: workspace too small")
    check(lib.rgbd_label_map_rle(seg.data_ptr(), B, H, W, L, workspace.data_ptr(), out.offsets.data_ptr(),
                                 out.base.data_ptr(), out.runs.data_ptr(), out.bad.data_ptr(), _stream()),
          "rgbd_label_map_rle")
    _count(4)                                           # count, scan, base, emit
    return out


@dataclass
class InstanceRle:
    """Device-side result of ``instance_rle`` (CSR).  The pycocotools "counts" string of segment ``s`` of image ``b`` is
    ``chars[base[b] + offsets[b, s] : base[b] + offsets[b, s + 1]]``; the batch uses ``chars[:base[B]]``."""
    offsets: torch.Tensor              # (B, L+1) i32, relative to the image's base
    base: torch.Tensor                 # (B+1,) i32
    chars: torch.Tensor                # (capacity,) u8, ASCII 48..111
    bad: torch.Tensor                  # (1,) i32: pixels outside [-1, L) or in [count[b], L), +1 per count outside [0, L]


def _instance_rle_sizes(B: int, H: int, W: int, L: int) -> Tuple[int, int]:
    lib = _lib.load()
    ws_bytes = int(lib.rgbd_instance_rle_workspace_bytes(B, H, W, L))
    capacity = int(lib.rgbd_instance_rle_capacity(B, H, W, L))
    if ws_bytes == 0 or capacity == 0:
        raise RgbdB200Error(f"instance_rle: unsupported shape (B,H,W)={(B, H, W)} or label count {L} "
                            "(at most 4096 labels, 65535 images, 7*B*(2*H*W + L) < 2^31)")
    return ws_bytes, capacity


def _instance_rle_outputs(B: int, L: int, capacity: int, device) -> InstanceRle:
    i32 = dict(device=device, dtype=torch.int32)
    return InstanceRle(torch.empty(B, L + 1, **i32), torch.empty(B + 1, **i32),
                       torch.empty(capacity, device=device, dtype=torch.uint8), torch.empty(1, **i32))


def instance_rle_buffers(B: int, H: int, W: int, n_labels: int, device) -> Tuple[InstanceRle, torch.Tensor]:
    """Output tensors and workspace of ``instance_rle`` for (B,H,W) maps, to pass as ``out`` / ``workspace``."""
    ws_bytes, capacity = _instance_rle_sizes(B, H, W, int(n_labels))   # checks the arguments before anything is allocated
    return (_instance_rle_outputs(B, int(n_labels), capacity, device),
            torch.empty(ws_bytes, device=device, dtype=torch.uint8))


def instance_rle(seg: torch.Tensor, count: torch.Tensor, n_labels: int, out: Optional[InstanceRle] = None,
                 workspace: Optional[torch.Tensor] = None) -> InstanceRle:
    """pycocotools RLE of the kept segments of (B,H,W) int32 painted maps, without host synchronisation: segment
    ``s < count[b]`` gets the "counts" string of ``pycocotools.mask.encode(np.asfortranarray(seg[b] == s))``.  Pixels
    outside [-1, n_labels) or in [count[b], n_labels) are counted in ``bad``, never encoded: check it.
    ``out`` / ``workspace`` (from ``instance_rle_buffers``) are used in place when given; either one may be given alone."""
    lib = _lib.load()
    _req(seg, "seg", torch.int32)
    _req(count, "count", torch.int32)
    if seg.dim() != 3:
        raise RgbdB200Error("instance_rle: expected a (B,H,W) int32 label map")
    B, H, W = seg.shape
    if tuple(count.shape) != (B,):
        raise RgbdB200Error(f"instance_rle: count of shape {tuple(count.shape)}, expected {(B,)}")
    L = int(n_labels)
    ws_bytes, capacity = _instance_rle_sizes(B, H, W, L)
    if out is None:
        out = _instance_rle_outputs(B, L, capacity, seg.device)
    if workspace is None:
        workspace = torch.empty(ws_bytes, device=seg.device, dtype=torch.uint8)
    want = [(out.offsets, (B, L + 1), torch.int32), (out.base, (B + 1,), torch.int32),
            (out.chars, (capacity,), torch.uint8), (out.bad, (1,), torch.int32)]
    for t, shape, dtype in want:
        _req(t, "instance_rle output", dtype)
        if tuple(t.shape) != shape:
            raise RgbdB200Error(f"instance_rle: output of shape {tuple(t.shape)}, expected {shape}")
    _req(workspace, "instance_rle workspace", torch.uint8)
    if workspace.numel() < ws_bytes:
        raise RgbdB200Error("instance_rle: workspace too small")
    check(lib.rgbd_instance_rle(seg.data_ptr(), count.data_ptr(), B, H, W, L, workspace.data_ptr(),
                                out.offsets.data_ptr(), out.base.data_ptr(), out.chars.data_ptr(), out.bad.data_ptr(),
                                _stream()), "rgbd_instance_rle")
    _count(9)                                           # transpose, 4 x rle_*, size, scan, base, emit
    return out


def mask_iou(pred_masks: torch.Tensor, gt_masks: torch.Tensor) -> torch.Tensor:
    """(P,H,W) x (G,H,W) 0/1 masks (bool or uint8) -> (P,G) float32 IoU."""
    lib = _lib.load()
    if pred_masks.dtype == torch.bool:
        pred_masks = pred_masks.view(torch.uint8)
    if gt_masks.dtype == torch.bool:
        gt_masks = gt_masks.view(torch.uint8)
    _req(pred_masks, "pred_masks", torch.uint8)
    _req(gt_masks, "gt_masks", torch.uint8)
    if pred_masks.dim() != 3 or gt_masks.dim() != 3 or pred_masks.shape[1:] != gt_masks.shape[1:]:
        raise RgbdB200Error("mask_iou: expected (P,H,W) and (G,H,W) masks of one size")
    P, G = pred_masks.shape[0], gt_masks.shape[0]
    iou = torch.zeros(P, G, device=pred_masks.device, dtype=torch.float32)
    if P and G:
        check(lib.rgbd_mask_iou(pred_masks.data_ptr(), gt_masks.data_ptr(), P, G, pred_masks.shape[1] * pred_masks.shape[2],
                                iou.data_ptr(), _stream()), "rgbd_mask_iou")
        _count(1)
    return iou


# ------------------------------------------------------------------------------------------------
# consumers of the fused pyramid (stock HF pixel decoder / transformer decoder): two inference kernels
# ------------------------------------------------------------------------------------------------
def _dt(t: torch.Tensor, name: str) -> int:
    if t.dtype == torch.float32:
        return 0                                     # RGBD_DTYPE_F32
    if t.dtype == torch.bfloat16:
        return 1                                     # RGBD_DTYPE_BF16
    raise RgbdB200Error(f"{name} must be float32 or bfloat16, got {t.dtype}")


def msda_forward(value: torch.Tensor, spatial_shapes: Sequence[Tuple[int, int]], offsets_or_locations: torch.Tensor,
                 attention: torch.Tensor, reference_points: Optional[torch.Tensor] = None, softmax: bool = False,
                 out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """Multi-scale deformable attention sampling (``rgbd_msda_fwd``; HF ``multi_scale_deformable_attention``).
    value (B,S,H,D); offsets_or_locations (B,Q,H,L,P,2); attention (B,Q,H,L,P) or (B,Q,H,L*P); -> (B,Q,H*D).
    Without ``reference_points`` the second argument holds sampling locations in [0,1] and ``attention`` the weights;
    with ``reference_points`` (B,Q,L,2) it holds raw offsets (location = reference + offset / (w_l, h_l)) and
    ``softmax=True`` softmaxes ``attention`` over L*P inside the kernel."""
    lib = _lib.load()
    _req(value, "value")
    _req(offsets_or_locations, "sampling offsets / locations")
    _req(attention, "attention weights")
    if value.dim() != 4 or offsets_or_locations.dim() != 6 or offsets_or_locations.shape[-1] != 2:
        raise RgbdB200Error("msda_forward: value must be (B,S,H,D) and offsets / locations (B,Q,H,L,P,2)")
    B, S, H, D = value.shape
    _, Q, H2, L, P, _ = offsets_or_locations.shape
    if offsets_or_locations.shape[0] != B or H2 != H or L != len(spatial_shapes):
        raise RgbdB200Error("msda_forward: batch / heads / levels of value, offsets and spatial_shapes disagree")
    if attention.numel() != B * Q * H * L * P:
        raise RgbdB200Error(f"msda_forward: attention must hold {B * Q * H * L * P} elements, got {attention.numel()}")
    ref = None
    if reference_points is not None:
        ref = _req(reference_points, "reference_points", torch.float32)
        if tuple(ref.shape) != (B, Q, L, 2):
            raise RgbdB200Error(f"reference_points must be {(B, Q, L, 2)}, got {tuple(ref.shape)}")
    elif softmax:
        raise RgbdB200Error("msda_forward: softmax=True belongs to the fused mode (reference_points given)")
    hw = int_array([v for s in spatial_shapes for v in (int(s[0]), int(s[1]))])
    out = torch.empty(B, Q, H * D, device=value.device, dtype=out_dtype)
    check(lib.rgbd_msda_fwd(value.data_ptr(), _dt(value, "value"), hw, L, offsets_or_locations.data_ptr(),
                            _dt(offsets_or_locations, "offsets"), ref.data_ptr() if ref is not None else None,
                            attention.data_ptr(), _dt(attention, "attention"), int(bool(softmax)), out.data_ptr(),
                            _dt(out, "out"), B, S, Q, H, D, P, _stream()), "rgbd_msda_fwd")
    _count(1)
    return out


def attention_mask(mask_logits: torch.Tensor, target_size: Tuple[int, int], num_heads: int) -> torch.Tensor:
    """``rgbd_attention_mask``: (B,Q,h,w) mask logits -> (B*heads, Q, th*tw) bool, True where
    sigmoid(bilinear(mask_logits -> target_size, align_corners=False)) < 0.5 (HF ``Mask2FormerMaskPredictor``)."""
    lib = _lib.load()
    _req(mask_logits, "mask_logits")
    if mask_logits.dim() != 4:
        raise RgbdB200Error("attention_mask: mask_logits must be (B,Q,h,w)")
    B, Q, h, w = mask_logits.shape
    th, tw = int(target_size[0]), int(target_size[1])
    out = torch.empty(B * num_heads, Q, th * tw, device=mask_logits.device, dtype=torch.bool)
    check(lib.rgbd_attention_mask(mask_logits.data_ptr(), _dt(mask_logits, "mask_logits"), B, Q, h, w, th, tw, int(num_heads),
                                  out.data_ptr(), _stream()), "rgbd_attention_mask")
    _count(1)
    return out


def window_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, bias: torch.Tensor, mask: Optional[torch.Tensor],
                     num_heads: int) -> torch.Tensor:
    """``rgbd_window_attention`` (transformers ``SwinSelfAttention``'s inner op): q / k / v (windows, N, heads*32) float32 or
    bfloat16, bias (heads, N, N) float32, mask (nW, N, N) float32 or None (window w uses mask[w % nW]) -> (windows, N, heads*32)
    of the inputs' dtype = softmax(q k^T / sqrt(32) + bias + mask) v."""
    lib = _lib.load()
    for t, name in ((q, "q"), (k, "k"), (v, "v")):
        _req(t, name, q.dtype)
    _req(bias, "bias", torch.float32)
    if q.dim() != 3 or k.shape != q.shape or v.shape != q.shape:
        raise RgbdB200Error("window_attention: q, k, v must share the shape (windows, N, C)")
    n_win, N, Cc = q.shape
    if Cc != num_heads * 32:
        raise RgbdB200Error(f"window_attention: C = {Cc} is not heads * 32 = {num_heads * 32}")
    if tuple(bias.shape) != (num_heads, N, N):
        raise RgbdB200Error(f"window_attention: bias must be {(num_heads, N, N)}, got {tuple(bias.shape)}")
    nw = 1
    if mask is not None:
        _req(mask, "mask", torch.float32)
        if mask.dim() != 3 or tuple(mask.shape[1:]) != (N, N):
            raise RgbdB200Error(f"window_attention: mask must be (nW, {N}, {N}), got {tuple(mask.shape)}")
        nw = mask.shape[0]
    out = torch.empty_like(q)
    ws = torch.empty(lib.rgbd_window_attention_workspace_bytes(N, int(num_heads), nw), device=q.device, dtype=torch.uint8)
    check(lib.rgbd_window_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), _dt(q, "q"), bias.data_ptr(),
                                    mask.data_ptr() if mask is not None else None, out.data_ptr(), n_win, N, int(num_heads), 32, nw,
                                    ws.data_ptr(), _stream()), "rgbd_window_attention")
    _count(2)
    return out


def layer_norm(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float,
               out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """``rgbd_layer_norm``: LayerNorm over the last dimension of a float32 or bfloat16 tensor, float32 arithmetic, float32 or
    bfloat16 output."""
    lib = _lib.load()
    _req(x, "x")
    _req(weight, "weight", torch.float32)
    _req(bias, "bias", torch.float32)
    Cc = x.shape[-1]
    if weight.numel() != Cc or bias.numel() != Cc:
        raise RgbdB200Error(f"layer_norm: weight / bias must have {Cc} elements")
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    check(lib.rgbd_layer_norm(x.data_ptr(), _dt(x, "x"), weight.data_ptr(), bias.data_ptr(), out.data_ptr(), _dt(out, "out"),
                              x.numel() // Cc, Cc, float(eps), _stream()), "rgbd_layer_norm")
    _count(1)
    return out


def masked_cross_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, attn_mask: torch.Tensor, num_heads: int) -> torch.Tensor:
    """``rgbd_masked_cross_attention``: q (L, B, heads*32), k / v (S, B, heads*32) bfloat16 (``batch_first=False`` projections of
    ``nn.MultiheadAttention``), attn_mask (B*heads, L, S) bool, True = may not attend -> (L, B, heads*32) bfloat16."""
    lib = _lib.load()
    for t_, name in ((q, "q"), (k, "k"), (v, "v")):
        _req(t_, name, torch.bfloat16)
    _req(attn_mask, "attn_mask", torch.bool)
    if q.dim() != 3 or k.dim() != 3 or v.shape != k.shape or k.shape[1:] != q.shape[1:]:
        raise RgbdB200Error("masked_cross_attention: q (L,B,E), k / v (S,B,E)")
    L, B, E = q.shape
    S = k.shape[0]
    if E != num_heads * 32:
        raise RgbdB200Error(f"masked_cross_attention: E = {E} is not heads * 32 = {num_heads * 32}")
    if tuple(attn_mask.shape) != (B * num_heads, L, S):
        raise RgbdB200Error(f"masked_cross_attention: attn_mask must be {(B * num_heads, L, S)}, got {tuple(attn_mask.shape)}")
    out = torch.empty_like(q)
    check(lib.rgbd_masked_cross_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), attn_mask.data_ptr(), out.data_ptr(), B,
                                          int(num_heads), L, S, 32, _stream()), "rgbd_masked_cross_attention")
    _count(1)
    return out
