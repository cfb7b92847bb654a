"""Drop-in ``nn.Module`` mirrors of the reference's depth-guidance modules
(mask2former/utils/custom_model.py, "CM").  Constructor / forward signatures, attribute names and
``state_dict`` keys are the reference's, so checkpoints move both ways; the arithmetic runs in the
sm_100a kernels behind include/rgbd_b200.h.  No CPU path exists: CPU tensors raise.

* ``DepthGradientInjectionResidual``      CM:1169-1269  (DGGM, kernel K1 / K1b)
* ``DSAModule``                           CM:622-799    (E-DSAM core, kernels K2 + K3)
* ``EnhancedDepthImageRatioPredictor``    CM:1363-1487  (E-DSAM window-ratio predictor, kernel K4)
* ``DepthGuidance``                       CM:324-355    (the v0.4.0 wiring as one batched, sync-free call)
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import nn

from . import functional as Fn
from ._lib import RgbdB200Error


#: False: every DSAM stage packs its own operand (A/B switch for the epilogue-emitted operands of the inference cascade)
FUSE_STAGE_PACKS = os.environ.get("RGBD_NO_STAGE_PACK_FUSION", "") in ("", "0")

#: RGBD_DSAM_PREMASKED=1 keeps the five-fold pre-masked DSAM operand in HBM (A/B measurements against the shared-memory masking kernel)
_PREMASKED = os.environ.get("RGBD_DSAM_PREMASKED", "") not in ("", "0")


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


_best_box = Fn.best_box


#: workspaces kept alive per module (distinct batch sizes / resolutions, e.g. a last partial batch); oldest evicted first
MAX_CACHED_SHAPES = 4


def _evict(cache: dict) -> None:
    while len(cache) >= MAX_CACHED_SHAPES:
        cache.pop(next(iter(cache)))


class _Versioned:
    """Re-pack derived tensors only when a source parameter changed (torch bumps ``_version`` on in-place
    updates such as optimizer steps / load_state_dict).  Writes through ``p.data`` (``weight.data.copy_()``, EMA swaps, fused
    optimizers of apex / DeepSpeed) bypass the version counter: call the module's ``invalidate_packed()`` after them
    (``module.train()`` / ``.eval()`` do it too)."""

    def __init__(self):
        self._key = None

    def invalidate(self) -> None:
        self._key = None

    def stale(self, tensors: Sequence[torch.Tensor]) -> bool:
        key = tuple((t.data_ptr(), t._version, t.device) for t in tensors)
        if key != self._key:
            self._key = key
            return True
        return False


class _PackedCacheMixin:
    """``invalidate_packed()``: drop the bf16-packed copies of the parameters (needed only after writes that bypass torch's
    version counter); switching between ``train()`` and ``eval()`` invalidates them as well."""

    def invalidate_packed(self) -> None:
        for name in ("_ver", "_ver_bwd", "_ver_train"):
            v = getattr(self, name, None)
            if v is not None:
                v.invalidate()

    def train(self, mode: bool = True):
        self.invalidate_packed()
        return super().train(mode)


# =====================================================================================================
# DGGM
# =====================================================================================================
class _DggmFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, grad_map, mask, n, *args):
        feats, weights, biases = args[:n], args[n:2 * n], args[2 * n:3 * n]
        outs = Fn.dggm_forward([f.contiguous() for f in feats], grad_map, mask, weights, biases)
        ctx.n = n
        ctx.save_for_backward(grad_map, mask, *weights, *biases)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *douts):
        n = ctx.n
        saved = ctx.saved_tensors
        grad_map, mask = saved[0], saved[1]
        weights, biases = saved[2:2 + n], saved[2 + n:2 + 2 * n]
        dws, dbs = Fn.dggm_backward_params(douts, grad_map, mask, weights, biases)
        # d(out)/d(color) is the identity; the gradient map and mask are data (SURVEY H11)
        return (None, None, None, *douts, *dws, *dbs)


class DepthGradientInjectionResidual(nn.Module):
    """CM:1169-1269.  Injects the gated depth-gradient map into every colour feature scale:
    ``fused_i = color_i + ReLU(Conv1x1_i(bilinear(grad) * nearest(mask)))``."""

    def __init__(self, color_channels: List[int], depth_gradient_channels: int):
        super().__init__()
        self.color_channels = color_channels
        self.depth_gradient_channels = depth_gradient_channels
        self.num_scales = len(color_channels)
        self.depth_enhancement_layers = nn.ModuleList()
        for channels in color_channels:
            self.depth_enhancement_layers.append(
                nn.Sequential(nn.Conv2d(depth_gradient_channels, channels, kernel_size=1), nn.ReLU(inplace=True)))

    def _params(self):
        ws = [l[0].weight for l in self.depth_enhancement_layers]
        bs = [l[0].bias for l in self.depth_enhancement_layers]
        return ws, bs

    def forward(self, color_feature_maps: List[torch.Tensor], processed_depth_gradient_map: Optional[torch.Tensor],
                gradient_mask: Optional[torch.Tensor]) -> List[torch.Tensor]:
        assert len(color_feature_maps) == self.num_scales, \
            f"Expected {self.num_scales} color feature maps, but got {len(color_feature_maps)}"
        if processed_depth_gradient_map is None or gradient_mask is None:
            return list(color_feature_maps)                                   # CM:1263-1265
        assert processed_depth_gradient_map.shape[1] == self.depth_gradient_channels
        assert gradient_mask.shape[1] == 1
        ws, bs = self._params()
        needs_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (*ws, *bs, *color_feature_maps))
        if needs_grad:
            return list(_DggmFunction.apply(processed_depth_gradient_map, gradient_mask, self.num_scales,
                                            *color_feature_maps, *ws, *bs))
        return Fn.dggm_forward([f.contiguous() for f in color_feature_maps], processed_depth_gradient_map,
                               gradient_mask, [w.detach() for w in ws], [b.detach() for b in bs])

    def forward_fused_sum(self, color_feature_maps, branch1, processed_depth_gradient_map, gradient_mask, outs=None):
        """``branch1_i + (color_i + enh_i)`` in one pass (the v0.4.0 branch sum, CM:354-355). Inference only."""
        ws, bs = self._params()
        return Fn.dggm_forward(color_feature_maps, processed_depth_gradient_map, gradient_mask,
                               [w.detach() for w in ws], [b.detach() for b in bs], branch1=branch1, outs=outs)


# =====================================================================================================
# E-DSAM core
# =====================================================================================================
class _DsamStageFunction(torch.autograd.Function):
    """Autograd of one DSAM stage (masks are constants; SURVEY H11): wgrad + dbias always, dgrad only when the
    stage input requires grad (stage 0's input is a detached clone, CM:332)."""

    @staticmethod
    def forward(ctx, module, x, codes, variant, residual, *params):
        out = module._stage_forward_impl(x, codes, variant, residual)
        ctx.module = module
        ctx.has_res = residual is not None
        ctx.save_for_backward(x, codes, variant)
        return out

    @staticmethod
    def backward(ctx, g):
        x, codes, variant = ctx.saved_tensors
        m = ctx.module
        dx, grads = m._stage_backward_impl(x, codes, variant, g.contiguous().float(), need_dx=ctx.needs_input_grad[1])
        return (None, dx, None, None, g if ctx.has_res else None, *grads)


class DSAModule(_PackedCacheMixin, nn.Module):
    """CM:622-799.  Depth-sensitive attention: depth histogram modes -> depth-interval region masks ->
    sum_t Conv_t(mask_t * F) + projection(F).  ``in != out``: 3x3 stride-2 convs + bias-free 3x3 stride-2
    ``rgb_projection``; ``in == out``: 1x1 convs + identity residual.

    One difference from the reference under autograd: a region conv that no image of the batch used (fewer than three depth
    modes, CM:683-691) receives a ZERO gradient here, where the reference leaves ``.grad`` as ``None``; optimizers with weight
    decay or momentum therefore still touch it.  (A fixed gradient layout is what lets the all-reduce buckets of
    ``parallel.GradBucketReducer`` be static.)"""

    #: "bf16": bf16 operands, fp32 accumulate (what torch.autocast gives the reference; ~1e-3 relative).
    #: "fp32": split precision -- activations and weights as bf16 hi + lo parts, three tensor-core products per term
    #: (~2^-16 relative, inside the 1e-4 fp32 bar) at three times the GEMM work.  Forward only: the backward follows
    #: ``grad_precision``.
    precision = "bf16"
    #: Operands of the weight and input gradient GEMMs (dW, dx), independent of ``precision``; the forward output does
    #: not depend on it.  "bf16": bf16 G, x and weights, fp32 accumulate (~2^-8 relative).  "fp32": the same split as the
    #: forward -- G, x * bit_t and the weights as bf16 hi + lo, products hi.hi + lo.hi + hi.lo (the three terms left out
    #: are each at most 2^-16 |g||x|) at three times the GEMM work.  dbias and the identity residual are fp32 sums in both.
    grad_precision = "bf16"

    def __init__(self, in_channels, out_channels, num_depth_regions=3):
        super().__init__()
        if not 1 <= num_depth_regions <= 3:
            raise ValueError("rgbd_b200 supports 1..3 depth regions (4-bit region codes)")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.num_depth_regions = num_depth_regions
        if in_channels != out_channels:
            self.conv_layers = nn.ModuleList([
                nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=2, padding=1)
                for _ in range(num_depth_regions + 1)])
            self.rgb_projection = nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=2, padding=1, bias=False)
        else:
            self.conv_layers = nn.ModuleList([
                nn.Conv2d(in_channels, out_channels, kernel_size=1) for _ in range(num_depth_regions + 1)])
        self._ver = _Versioned()
        self._packed: Dict[str, torch.Tensor] = {}
        self._ws: Dict[tuple, torch.Tensor] = {}
        self._ver_bwd = _Versioned()
        self._packed_bwd: Dict = {}
        self._ws_t: Dict[tuple, torch.Tensor] = {}

    # ---- operand packing -------------------------------------------------------------------------
    @property
    def _proj(self) -> bool:
        return self.in_channels != self.out_channels

    def _geometry(self):
        # 128-byte K rows (64 channels) keep TMA/L2 requests full-width; 96 channels are padded to 128 rather than
        # split into 64-byte rows (measured: fewer, wider K blocks win although 1/4 of the stage-0 MMAs multiply zeros)
        c_pad = _round_up(self.in_channels, 64) if self.in_channels > 32 else 32
        kb = 64 if c_pad % 64 == 0 else 32
        n_pad = _round_up(self.out_channels, 32)
        n_seg = self.num_depth_regions + 1 + (1 if self._proj else 0)
        return c_pad, kb, n_pad, n_seg

    def _refresh(self):
        srcs = [p for p in self.parameters()]
        split = self.precision == "fp32"
        if not self._ver.stale(srcs) and self._packed and self._packed.get("split") == split:
            return self._packed
        dev = srcs[0].device
        c_in, c_out, R = self.in_channels, self.out_channels, self.num_depth_regions
        c_pad, kb, n_pad, n_seg = self._geometry()
        taps = 9 if self._proj else 1
        k = 3 if self._proj else 1
        with torch.no_grad():
            w = torch.zeros(n_pad, n_seg, taps, c_pad, device=dev, dtype=torch.float32)
            for t in range(R + 1):
                w[:c_out, t, :, :c_in] = self.conv_layers[t].weight.reshape(c_out, c_in, k * k).permute(0, 2, 1)
            if self._proj:
                w[:c_out, R + 1, :, :c_in] = self.rgb_projection.weight.reshape(c_out, c_in, 9).permute(0, 2, 1)
            if split:
                # K blocks per (segment, tap): [x_hi . W_hi | x_lo . W_hi | x_hi . W_lo]
                w_hi = w.to(torch.bfloat16)
                w_lo = (w - w_hi.float()).to(torch.bfloat16)
                w_cat = torch.stack([w_hi, w_hi, w_lo], dim=3).reshape(n_pad, n_seg * taps * 3 * c_pad).contiguous()
            else:
                w_cat = w.reshape(n_pad, n_seg * taps * c_pad).to(torch.bfloat16).contiguous()
            w_masked = None
            if self._proj and c_pad % 64 == 0:
                # K order of the mask-in-shared-memory kernel: (tap, 64-channel block, segment, channel)
                w_masked = (w.reshape(n_pad, n_seg, taps, c_pad // 64, 64).permute(0, 2, 3, 1, 4)
                            .reshape(n_pad, taps * c_pad * n_seg).to(torch.bfloat16).contiguous())
            # bias table: variant v = sum of the first v conv biases (CM:683-691: only used regions add a bias)
            bias = torch.zeros(R + 2, n_pad, device=dev, dtype=torch.float32)
            run = torch.zeros(c_out, device=dev, dtype=torch.float32)
            for v in range(1, R + 2):
                run = run + self.conv_layers[v - 1].bias.float()
                bias[v, :c_out] = run
        n_par = 4 if self._proj else 1
        sl = []
        for seg in range(n_seg):
            for tap in range(taps):
                dy, dx = (tap // 3, tap % 3) if self._proj else (1, 1)
                if self._proj:
                    # input row 2*oy + dy - 1: dy=0 -> odd plane, row oy-1; dy=1 -> even plane, row oy; dy=2 -> odd, oy
                    py, yo = (1, -1) if dy == 0 else ((0, 0) if dy == 1 else (1, 0))
                    px, xo = (1, -1) if dx == 0 else ((0, 0) if dx == 1 else (1, 0))
                    par = py * 2 + px
                else:
                    par, yo, xo = 0, 0, 0
                if split:       # operand segments are stored (hi, lo) interleaved: segment index 2*seg + {0, 1}
                    for a_seg in (2 * seg, 2 * seg + 1, 2 * seg):
                        for cb in range(c_pad // kb):
                            sl.append((cb * kb, xo, yo, a_seg * n_par + par))
                else:
                    for cb in range(c_pad // kb):
                        sl.append((cb * kb, xo, yo, seg * n_par + par))
        slices = torch.tensor(sl, device=dev, dtype=torch.int32).contiguous()
        self._packed = {"w": w_cat, "w_masked": w_masked, "bias": bias, "slices": slices, "split": split}
        return self._packed

    def _workspace(self, B, H, W, dev, n_op=None):
        c_pad, kb, n_pad, n_seg = self._geometry()
        if n_op is None:
            n_op = n_seg * (2 if self.precision == "fp32" else 1)
        key = (B, H, W, str(dev), n_op)
        if key not in self._ws:
            if self._proj:
                shape = (B, n_op, 4, (H + 1) // 2, (W + 1) // 2, c_pad)
            else:
                shape = (B, n_op, 1, H, W, c_pad)
            _evict(self._ws)
            self._ws[key] = torch.zeros(shape, device=dev, dtype=torch.bfloat16)
        return self._ws[key]

    def _param_list(self):
        ps = []
        for conv in self.conv_layers:
            ps += [conv.weight, conv.bias]
        if self._proj:
            ps.append(self.rgb_projection.weight)
        return ps

    def stage_forward(self, rgb_features: torch.Tensor, codes: torch.Tensor, bias_variant: torch.Tensor,
                      residual: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Batched tensor-core path (see ``_stage_forward_impl``); differentiable w.r.t. the stage's parameters,
        its input features and the residual when autograd is recording."""
        ps = self._param_list()
        if torch.is_grad_enabled() and (rgb_features.requires_grad or any(p.requires_grad for p in ps)
                                        or (residual is not None and residual.requires_grad)):
            return _DsamStageFunction.apply(self, rgb_features, codes, bias_variant, residual, *ps)
        return self._stage_forward_impl(rgb_features, codes, bias_variant, residual)

    # ---- backward (K3b) ----------------------------------------------------------------------------
    def _split_grad(self) -> bool:
        if self.grad_precision not in ("bf16", "fp32"):
            raise ValueError(f"DSAModule.grad_precision must be 'bf16' or 'fp32', got {self.grad_precision!r}")
        return self.grad_precision == "fp32"

    def _refresh_bwd(self):
        """Per input-parity class: transposed weights [(channel block, segment, 32 ch)][(tap, n)] and tap offsets.  Split
        precision (``grad_precision == "fp32"``): every 64-row K block becomes three, [W_hi | W_hi | W_lo], read against
        the G planes (hi, lo, hi)."""
        srcs = [p for p in self.parameters()]
        split = self._split_grad()
        if not self._ver_bwd.stale(srcs) and self._packed_bwd and self._packed_bwd.get("split") == split:
            return self._packed_bwd
        dev = srcs[0].device
        c_in, c_out, R = self.in_channels, self.out_channels, self.num_depth_regions
        n_seg = R + 1 + (1 if self._proj else 0)
        c32 = _round_up(c_in, 32)
        np64 = _round_up(c_out, 64)
        ws = [c.weight.detach().float() for c in self.conv_layers] + ([self.rgb_projection.weight.detach().float()] if self._proj else [])
        classes = []
        par_list = [(py, px) for py in (0, 1) for px in (0, 1)] if self._proj else [(0, 0)]
        for py, px in par_list:
            if self._proj:
                dys = [(1, 0)] if py == 0 else [(0, 1), (2, 0)]       # (dy, oy offset): input row 2*y2+py = 2*oy+dy-1
                dxs = [(1, 0)] if px == 0 else [(0, 1), (2, 0)]
            else:
                dys, dxs = [(0, 0)], [(0, 0)]
            taps = [(dy, yo, dx, xo) for dy, yo in dys for dx, xo in dxs]
            wd = torch.zeros(c32 // 32, n_seg, 32, len(taps), np64, device=dev, dtype=torch.float32)
            for sg, w in enumerate(ws):
                for ti, (dy, yo, dx, xo) in enumerate(taps):
                    wt = torch.zeros(c32, np64, device=dev)
                    wt[:c_in, :c_out] = w[:, :, dy, dx].t()                 # (c, n)
                    wd[:, sg, :, ti, :] = wt.reshape(c32 // 32, 32, np64)
            wd = wd.reshape(c32 // 32 * n_seg * 32, len(taps) * np64)
            if split:
                w_hi = wd.reshape(wd.shape[0], len(taps) * np64 // 64, 64).to(torch.bfloat16)
                w_lo = (wd.reshape(w_hi.shape) - w_hi.float()).to(torch.bfloat16)
                wd = torch.stack([w_hi, w_hi, w_lo], dim=2).reshape(wd.shape[0], 3 * len(taps) * np64).contiguous()
                planes = (0, 1, 0)
            else:
                wd = wd.to(torch.bfloat16).contiguous()
                planes = (0,)
            sl = torch.tensor([(nb * 64, xo, yo, pl) for (dy, yo, dx, xo) in taps for nb in range(np64 // 64) for pl in planes],
                              device=dev, dtype=torch.int32).contiguous()
            classes.append({"py": py, "px": px, "w": wd, "slices": sl})
        self._packed_bwd = {"classes": classes, "n_seg": n_seg, "c32": c32, "np64": np64, "split": split}
        return self._packed_bwd

    def _stage_backward_impl(self, x: torch.Tensor, codes: torch.Tensor, variant: torch.Tensor, g: torch.Tensor, need_dx: bool):
        R, c_in, c_out = self.num_depth_regions, self.in_channels, self.out_channels
        c_pad, kb, n_pad, n_seg = self._geometry()
        B, _, H, W = x.shape
        _, _, Ho, Wo = g.shape
        split = self._split_grad()
        x = x.detach().contiguous().float()
        # ---- bias gradients: images use the first variant[b] biases
        db = Fn.dsam_dbias(g, variant, R + 1)
        # ---- weight gradients: GEMM over the output pixels (split precision: hi and lo parts of both operands)
        if split:
            gp, gp_lo = Fn.cast_bf16_pitched(g, _round_up(Wo, 8), lo=True)
        else:
            gp, gp_lo = Fn.cast_bf16_pitched(g, _round_up(Wo, 8)), None
        H2, W2 = ((H + 1) // 2, (W + 1) // 2) if self._proj else (H, W)
        key = (B, H, W, str(x.device), split)
        if key not in self._ws_t:
            _evict(self._ws_t)
            self._ws_t[key] = torch.zeros(2 if split else 1, B, n_seg, 6 if self._proj else 1, c_pad, H2, _round_up(W2, 8),
                                          device=x.device, dtype=torch.bfloat16)
        xt, xt_lo = self._ws_t[key][0], (self._ws_t[key][1] if split else None)
        Fn.dsam_pack_t(x, codes, xt, c_pad, xt.shape[-1], n_seg, R + 1, self._proj, out_lo=xt_lo)
        dw = Fn.dsam_wgrad(gp, xt, c_out, c_pad, (Ho, Wo), n_seg, self._proj, g_lo=gp_lo, xt_lo=xt_lo)   # (c_out, n_seg, taps, c_pad)
        k = 3 if self._proj else 1
        grads = []
        for t in range(R + 1):
            grads.append(dw[:, t, :, :c_in].reshape(c_out, k, k, c_in).permute(0, 3, 1, 2).contiguous())
            grads.append(db[t])
        if self._proj:
            grads.append(dw[:, R + 1, :, :c_in].reshape(c_out, 3, 3, c_in).permute(0, 3, 1, 2).contiguous())
        # ---- input gradient: one transposed-conv GEMM per input-parity class, masked segment sum in the epilogue
        dx = None
        if need_dx:
            pk = self._refresh_bwd()
            np64 = pk["np64"]
            n_pl = 2 if split else 1                          # split precision: planes (G_hi, G_lo) per image
            gcl = torch.empty(B, n_pl, Ho, Wo, np64, device=x.device, dtype=torch.bfloat16)
            Fn.dsam_pack(g, codes.reshape(-1)[:B * Ho * Wo].reshape(B, Ho, Wo), gcl, np64, 1, 0, False,   # plain NCHW -> channels-last
                         hi_lo=split)
            dx = torch.empty_like(x)
            direct = g if not self._proj else None            # identity residual (out = enh + F)
            for cl in pk["classes"]:
                Fn.conv_gemm(gcl, (B * n_pl, Ho, Wo, np64), n_pl, cl["w"], cl["slices"], 64, B, (H2, W2), _best_box(H2, W2), c_in, None,
                             epi_mode=3, out=dx, residual=direct, codes=codes, in_hw=(H, W), parity=(cl["py"], cl["px"]),
                             m3_stride=2 if self._proj else 1, m3_masked_segs=R + 1, m3_n_seg=n_seg,
                             block_n=32 * n_seg)
        return dx, grads

    def _uses_masked_kernel(self, B: int, H: int, W: int) -> bool:
        """Stride-2 stage handled by dsam_fwd_kernel (one unmasked operand copy, masking in shared memory)."""
        pk = self._refresh()
        c_pad, kb, n_pad, n_seg = self._geometry()
        Ho, Wo = (H + 1) // 2, (W + 1) // 2
        box = _best_box(Ho, Wo)
        return bool(self._proj and pk["w_masked"] is not None and not pk["split"] and not _PREMASKED
                    and n_pad // Fn.pick_block_n(n_pad) <= 2 and B * (-(-Ho // box[1])) * (-(-Wo // box[0])) >= 2)

    def _emit_target(self, B: int, H: int, W: int, dev):
        """(workspace, (c_pad, n_seg, masked_segs)) the PREVIOUS stage's epilogue can fill instead of this stage's pack
        kernel, or None (1x1 stages and the split-precision mode pack for themselves)."""
        pk = self._refresh()
        if not self._proj or pk["split"]:
            return None
        c_pad, kb, n_pad, n_seg = self._geometry()
        if self._uses_masked_kernel(B, H, W):
            return self._workspace(B, H, W, dev, n_op=1), (c_pad, 1, 0)
        return self._workspace(B, H, W, dev), (c_pad, n_seg, self.num_depth_regions + 1)

    def _stage_forward_impl(self, rgb_features: torch.Tensor, codes: torch.Tensor, bias_variant: torch.Tensor,
                            residual: Optional[torch.Tensor] = None, emit_next=None, prepacked: bool = False) -> torch.Tensor:
        """Batched tensor-core path: features (B,C_in,H,W) fp32, pooled region codes (B,H,W) uint8 and the
        per-image bias count (Decomposition.bias_variant) -> sum_t conv_t(F*p_t) + projection(F) [+ residual]
        (fp32 result, bf16 operands).  ``emit_next = (workspace, geometry, codes)`` of the next stage: the epilogue also
        writes that stage's packed operand; ``prepacked``: this stage's operand was written that way."""
        pk = self._refresh()
        x = Fn._req(rgb_features.detach().contiguous(), "rgb_features", torch.float32)
        if residual is not None:
            residual = residual.detach()
        B, Cc, H, W = x.shape
        assert Cc == self.in_channels, f"Expected {self.in_channels} channels, got {Cc}"
        c_pad, kb, n_pad, n_seg = self._geometry()
        R = self.num_depth_regions
        Ho, Wo = ((H + 1) // 2, (W + 1) // 2) if self._proj else (H, W)
        if tuple(codes.shape) != (B, H, W) or codes.dtype != torch.uint8:
            raise RgbdB200Error(f"region codes must be uint8 {(B, H, W)}, got {codes.dtype} {tuple(codes.shape)}")
        if bias_variant.numel() != B:
            raise RgbdB200Error(f"bias_variant must have {B} entries, got {bias_variant.numel()}")
        if residual is not None and tuple(residual.shape) != (B, self.out_channels, Ho, Wo):
            # the reference fails at `cp[k+1] += dsam_out` (CM:342) on a pyramid whose levels do not halve (ceil) exactly
            raise RgbdB200Error(f"residual must be {(B, self.out_channels, Ho, Wo)} (the stage's output shape), "
                                f"got {tuple(residual.shape)}")
        if emit_next is not None:
            nws, ngeom, ncodes = emit_next
            if tuple(ncodes.shape) != (B, Ho, Wo) or ncodes.dtype != torch.uint8:
                raise RgbdB200Error(f"next stage's region codes must be uint8 {(B, Ho, Wo)}, got {tuple(ncodes.shape)}")
        Ho, Wo = (H + 1) // 2, (W + 1) // 2
        box = _best_box(Ho, Wo)
        skip_pack = prepacked or getattr(self, "_gemm_only", False)     # bench.py times the GEMM alone on packed operands
        nxt = {}
        if emit_next is not None:
            nxt = dict(next_operand=emit_next[0], next_geom=emit_next[1], next_codes=emit_next[2])
        if self._uses_masked_kernel(B, H, W):
            # one unmasked operand copy; the kernel masks the tile per region in shared memory.  The masking is
            # redone for every N tile, so wide stages (768 outputs = 3 N tiles) keep the pre-masked operand
            # (measured, B=32: 406 us vs 302 us for stage 2; 492 vs 583 and 362 vs 399 us for stages 0 and 1)
            packed = self._workspace(B, H, W, x.device, n_op=1)
            if not skip_pack:
                Fn.dsam_pack(x, codes, packed, c_pad, 1, 0, True)
            out = torch.empty(B, self.out_channels, Ho, Wo, device=x.device, dtype=torch.float32)
            Fn.conv_gemm(packed, (B * 4, Ho, Wo, c_pad), 4, pk["w_masked"], None, 64, B, (Ho, Wo), box, self.out_channels,
                         pk["bias"], variant=bias_variant, epi_mode=1, out=out,
                         residual=residual.contiguous() if residual is not None else None, codes=codes, in_hw=(H, W),
                         m3_masked_segs=R + 1, m3_n_seg=n_seg, dsam_masked=True, **nxt)
            return out
        packed = self._workspace(B, H, W, x.device)
        if not skip_pack:
            Fn.dsam_pack(x, codes, packed, c_pad, n_seg, R + 1, self._proj, hi_lo=pk["split"])
        n_op = n_seg * (2 if pk["split"] else 1)
        if self._proj:
            Ho, Wo = (H + 1) // 2, (W + 1) // 2
            a_dims = (B * n_op * 4, Ho, Wo, c_pad)
            ppi = n_op * 4
        else:
            Ho, Wo = H, W
            a_dims = (B * n_op, H, W, c_pad)
            ppi = n_op
            residual = x if residual is None else residual + x
        out = torch.empty(B, self.out_channels, Ho, Wo, device=x.device, dtype=torch.float32)
        variant = bias_variant
        Fn.conv_gemm(packed, a_dims, ppi, pk["w"], pk["slices"], kb, B, (Ho, Wo), _best_box(Ho, Wo), self.out_channels,
                     pk["bias"], variant=variant, epi_mode=1, out=out,
                     residual=residual.contiguous() if residual is not None else None, **nxt)
        return out

    def forward(self, rgb_features, depth_map, window_size_ratio=0.1):
        """Reference signature (CM:647): one single-channel depth map shared by the batch of features."""
        if isinstance(depth_map, np.ndarray):
            depth_map = torch.from_numpy(np.ascontiguousarray(depth_map.squeeze(), dtype=np.float32))
        elif not isinstance(depth_map, torch.Tensor):
            raise TypeError("Depth map must be torch.Tensor or numpy.ndarray")
        gray = depth_map.detach().squeeze().to(device=rgb_features.device, dtype=torch.float32)
        if gray.dim() != 2:
            raise RgbdB200Error(f"depth_map must squeeze to (H,W), got {tuple(depth_map.shape)}")
        gray = gray.contiguous()[None]
        B, _, H, W = rgb_features.shape
        ratio = torch.tensor([float(window_size_ratio)], device=rgb_features.device, dtype=torch.float32)
        dec = Fn.depth_decompose(ratio, [(H, W)], gray=gray, num_modes=self.num_depth_regions)
        codes = dec.pooled[0].expand(B, H, W).contiguous()
        return self.stage_forward(rgb_features, codes, dec.bias_variant.expand(B).contiguous())

    # ---- reference helper API (CM:701-798), computed by the device kernel --------------------------
    def _calculate_depth_histogram(self, depth_map, bins=512, value_range=None):
        if bins != 512 or value_range is not None:
            raise RgbdB200Error("the device histogram is fixed to bins=512 over (nanmin, nanmax) (CM:701-718)")
        g = torch.as_tensor(np.ascontiguousarray(depth_map, dtype=np.float32)).reshape(1, 1, -1).cuda()
        dec = Fn.depth_decompose(torch.tensor([0.1], device=g.device), [], gray=g, debug=True)
        return dec.hist[0].cpu().numpy(), dec.edges[0].cpu().numpy()

    def _select_depth_distribution_modes(self, hist, bin_edges, num_modes=3, prominence_threshold=0.01):
        """CM:720-752: centres of the ``num_modes`` highest prominent histogram peaks (scipy ``find_peaks`` semantics),
        highest first; ``[]`` when no peak survives."""
        if not 1 <= num_modes <= 3:
            raise RgbdB200Error("the device peak finder selects 1..3 modes")
        h = torch.as_tensor(np.ascontiguousarray(hist, dtype=np.int64)).reshape(1, -1).cuda()
        e = torch.as_tensor(np.ascontiguousarray(bin_edges, dtype=np.float32)).reshape(1, -1).cuda()
        n, _, centres = Fn.depth_select_modes(h, e, num_modes, prominence_threshold)
        c = centres[0].cpu().numpy()
        return [c[k] for k in range(int(n[0]))]

    def _define_depth_interval_windows(self, depth_modes, window_size_ratio=0.1):
        """CM:754-772.  Six scalar operations on at most three numbers: the batched path does them inside the device
        kernel (decompose.cu); this mirror of the helper keeps the reference's float32 arithmetic and return types."""
        interval_windows = []
        for mode_center in depth_modes:
            window_half_width = mode_center * window_size_ratio / 2.0
            interval_windows.append((max(0, mode_center - window_half_width), mode_center + window_half_width))
        return interval_windows

    def _generate_depth_region_masks(self, depth_map, interval_windows):
        """CM:774-798: one boolean mask per window plus the remaining region (numpy arrays, like the reference)."""
        if len(interval_windows) > 3:
            raise RgbdB200Error("region codes hold at most 3 windows + the remaining region")
        d = np.ascontiguousarray(depth_map, dtype=np.float32)
        g = torch.from_numpy(d)[None].cuda()
        win = torch.zeros(1, 3, 2, dtype=torch.float32)
        for k, (lo, hi) in enumerate(interval_windows):
            win[0, k, 0], win[0, k, 1] = float(lo), float(hi)
        nw = torch.tensor([len(interval_windows)], dtype=torch.int32)
        codes = Fn.depth_region_codes(g, win.cuda(), nw.cuda())[0].cpu().numpy()
        if not interval_windows:                      # no windows: everything is "remaining"
            return [np.ones(d.shape, dtype=bool)]
        return [((codes >> t) & 1).astype(bool) for t in range(len(interval_windows) + 1)]


# =====================================================================================================
# E-DSAM ratio predictor
# =====================================================================================================
def _fold_bn(conv_bias: torch.Tensor, bn: nn.BatchNorm2d) -> Tuple[torch.Tensor, torch.Tensor]:
    scale = bn.weight.float() / torch.sqrt(bn.running_var.float() + bn.eps)
    shift = bn.bias.float() + (conv_bias.float() - bn.running_mean.float()) * scale
    return scale.contiguous(), shift.contiguous()


class EnhancedDepthImageRatioPredictor(_PackedCacheMixin, nn.Module):
    """CM:1363-1487: (B,3,H,W) depth -> (B,1) window_size_ratio in [0.01, 0.5].  ``eval()``: BatchNorm folded into the
    weights (running statistics), everything up to the 4x4 pooled map in two fused tensor-core kernels.  ``train()``:
    batch-statistics BatchNorm (a statistics pass + a normalising pass per BatchNorm layer, running statistics updated
    with momentum like torch) and Dropout with injectable keep-masks.  The module receives no gradient in the v0.4.0 model
    (its output is consumed through ``.item()``, CM:339), so only the forward exists."""

    def __init__(self, input_channels: int = 3):
        super().__init__()
        if not 1 <= input_channels <= 4:
            raise ValueError("rgbd_b200's stem operand holds 1..4 input channels per pixel (the reference default is 3)")
        self.input_channels = input_channels
        self.scale1_conv = nn.Sequential(nn.Conv2d(input_channels, 64, kernel_size=3, padding=1), nn.BatchNorm2d(64), nn.ReLU(inplace=True))
        self.scale2_conv = nn.Sequential(nn.Conv2d(input_channels, 64, kernel_size=5, padding=2), nn.BatchNorm2d(64), nn.ReLU(inplace=True))
        self.scale3_conv = nn.Sequential(nn.Conv2d(input_channels, 64, kernel_size=7, padding=3), nn.BatchNorm2d(64), nn.ReLU(inplace=True))
        self.feature_fusion = nn.Sequential(nn.Conv2d(192, 128, kernel_size=1), nn.BatchNorm2d(128), nn.ReLU(inplace=True))
        self.attention = nn.Sequential(nn.Conv2d(128, 64, kernel_size=1), nn.ReLU(inplace=True),
                                       nn.Conv2d(64, 128, kernel_size=1), nn.Sigmoid())
        self.feature_extractor = nn.Sequential(
            nn.Conv2d(128, 256, kernel_size=3, padding=1), nn.BatchNorm2d(256), nn.ReLU(inplace=True),
            nn.AdaptiveAvgPool2d(4),
            nn.Conv2d(256, 512, kernel_size=3, padding=1), nn.BatchNorm2d(512), nn.ReLU(inplace=True))
        self.global_avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc_layers = nn.Sequential(
            nn.Linear(512, 128), nn.ReLU(inplace=True), nn.Dropout(0.3),
            nn.Linear(128, 64), nn.ReLU(inplace=True), nn.Dropout(0.2),
            nn.Linear(64, 32), nn.ReLU(inplace=True), nn.Linear(32, 1))
        self.output_min = 0.01
        self.output_max = 0.5
        self.sigmoid = nn.Sigmoid()
        self.use_compact_operand = True    # fused front end reads the depth image itself (sliding-window TMA) when it can
        self.use_fused_front = True        # stem GEMM + chain in one kernel; False: stem GEMM, then ...
        self.use_fused_chain = True        # ... the fused chain, or (False) three separate GEMM launches (cross-checks)
        self.use_tensor_core_tail = True   # 3x3 256->512 conv of the tail as a tcgen05 GEMM; False: the fp32 CUDA-core kernel
        #: train mode: ((B,128), (B,64)) boolean keep-masks used by the NEXT forward calls instead of fresh draws (tests;
        #: callers that reach the module through a parent's forward and cannot pass ``dropout_masks=``)
        self.dropout_masks_override = None
        self._ver = _Versioned()
        self._packed: Dict[str, torch.Tensor] = {}
        self._ws: Dict[tuple, Dict[str, torch.Tensor]] = {}
        self._ver_train = _Versioned()
        self._packed_train: Dict[str, torch.Tensor] = {}

    def _refresh(self):
        srcs = list(self.parameters()) + list(self.buffers())
        if not self._ver.stale(srcs) and self._packed:
            return self._packed
        dev = srcs[0].device
        bf = torch.bfloat16
        with torch.no_grad():
            # stem: three convs embedded in one 7x7 frame; K = 4 slices x [(j, dx8, c4)], tap dy = 2t + j
            w1 = torch.zeros(192, 4, 2, 8, 4, device=dev, dtype=torch.float32)
            sc1, sh1 = [], []
            for idx, (seq, k) in enumerate(((self.scale1_conv, 3), (self.scale2_conv, 5), (self.scale3_conv, 7))):
                o = (7 - k) // 2
                wk = seq[0].weight.float()                       # (64, 3, k, k)
                full = torch.zeros(64, self.input_channels, 8, 8, device=dev)
                full[:, :, o:o + k, o:o + k] = wk
                # (n, c, dy, dx) -> (n, t, j, dx, c)
                w1[idx * 64:(idx + 1) * 64, :, :, :, :self.input_channels] = full.reshape(64, self.input_channels, 4, 2, 8).permute(0, 2, 3, 4, 1)
                s, h = _fold_bn(seq[0].bias, seq[1])
                sc1.append(s)
                sh1.append(h)
            # folded BatchNorm scales are multiplied into the weights before the bf16 rounding, so the
            # epilogues only add the shift
            sc1 = torch.cat(sc1)
            pk = {"w1": (w1.reshape(192, 256) * sc1[:, None]).to(bf).contiguous(), "sh1": torch.cat(sh1)}
            # compact-operand layout: K = (dy 7, dx 8, c 4); w1 above is (t, j, dx, c) with dy = 2t + j, row dy = 7 all zero
            pk["w1c"] = pk["w1"].reshape(192, 8, 32)[:, :7].reshape(192, 224).contiguous()
            sc2, pk["sh2"] = _fold_bn(self.feature_fusion[0].bias, self.feature_fusion[1])
            pk["w2"] = (self.feature_fusion[0].weight.float().reshape(128, 192) * sc2[:, None]).to(bf).contiguous()
            pk["w3"] = self.attention[0].weight.float().reshape(64, 128).to(bf).contiguous()
            pk["sh3"] = self.attention[0].bias.detach().float().contiguous()
            pk["w4"] = self.attention[2].weight.float().reshape(128, 64).to(bf).contiguous()
            pk["sh4"] = self.attention[2].bias.detach().float().contiguous()
            c5 = self.feature_extractor[0]
            sc5, pk["sh5"] = _fold_bn(c5.bias, self.feature_extractor[1])
            pk["w5"] = (c5.weight.float().permute(0, 2, 3, 1).reshape(256, 9 * 128) * sc5[:, None]).to(bf).contiguous()  # K = (tap, c)
            c6 = self.feature_extractor[4]
            pk["w6"] = c6.weight.detach().float().contiguous()
            pk["sc6"], pk["sh6"] = _fold_bn(c6.bias, self.feature_extractor[5])
            # tensor-core tail: K = (tap, c), BatchNorm scale folded before the bf16 rounding
            pk["w6_bf"] = (c6.weight.float().permute(0, 2, 3, 1).reshape(512, 9 * 256) * pk["sc6"][:, None]).to(bf).contiguous()
            for j, li in enumerate((0, 3, 6, 8)):
                pk[f"fw{j}"] = self.fc_layers[li].weight.detach().float().contiguous()
                pk[f"fb{j}"] = self.fc_layers[li].bias.detach().float().contiguous()

            def sl(entries):
                return torch.tensor(entries, device=dev, dtype=torch.int32).contiguous()
            pk["sl1"] = sl([(0, 0, 2 * t, 0) for t in range(4)])
            pk["sl2"] = sl([(64 * cb, 0, 0, 0) for cb in range(3)])
            pk["sl3"] = sl([(64 * cb, 0, 0, 0) for cb in range(2)])
            pk["sl4"] = sl([(0, 0, 0, 0)])
            pk["sl5"] = sl([(64 * cb, dx - 1, dy - 1, 0) for dy in range(3) for dx in range(3) for cb in range(2)])
            pk["sl6"] = sl([(64 * cb, dx - 1, dy - 1, 0) for dy in range(3) for dx in range(3) for cb in range(4)])
        self._packed = pk
        return pk

    def _workspace(self, B, H, W, dev):
        compact = self._compact(H, W)
        key = (B, H, W, str(dev), self.use_fused_chain, self.use_fused_front, compact)
        if key not in self._ws:
            bf = dict(device=dev, dtype=torch.bfloat16)
            _evict(self._ws)
            self._ws[key] = {
                "stem": (torch.empty(B, 2, H + 6, Fn.ratio_stem_compact_width(W), 4, **bf) if compact
                         else torch.empty(B, H + 6, W, 64, **bf)),
                "x1": torch.empty(B, H, W, 192, **bf) if not self.use_fused_front else None,
                "x2": torch.empty(B, H, W, 128, **bf) if not (self.use_fused_chain or self.use_fused_front) else None,
                "x3": torch.empty(B, H, W, 64, **bf) if not (self.use_fused_chain or self.use_fused_front) else None,
                "x4": torch.empty(B, H, W, 128, **bf),
                "pool": torch.empty(B, 16, 256, device=dev, dtype=torch.int64),     # fixed-point cell sums
                "a6": torch.empty(B, 4, 4, 256, **bf), "gap_fx": torch.empty(B, 1, 512, device=dev, dtype=torch.int64),
            }
        return self._ws[key]

    def _conv5_pool(self, ws, w5, sl5, sh5, B, H, W, box) -> int:
        """Conv3x3 128->256 + (folded) BN + ReLU + AdaptiveAvgPool2d(4) (CM:1412-1417) into ``ws["pool"]``; returns the divisor
        the tail applies to the pooled sums.  H, W divisible by 4: pooled inside the GEMM epilogue, the 256-channel map is
        never written.  Otherwise torch's windows overlap: the map goes to HBM as bf16 and a pooling kernel takes the means."""
        reuse = dict(tile_order=1, conv3x3_reuse=(box == (128, 1)))     # one 130-pixel smem tile serves the three dx taps
        if H % 4 == 0 and W % 4 == 0:
            ws["pool"].zero_()
            Fn.conv_gemm(ws["x4"], (B, H, W, 128), 1, w5, sl5, 64, B, (H, W), box, 256, sh5, act=1, epi_mode=2,
                         pool=ws["pool"], cells=(4, 4), **reuse)
            return (H // 4) * (W // 4)
        x5 = torch.empty(B, H, W, 256, device=ws["x4"].device, dtype=torch.bfloat16)
        Fn.conv_gemm(ws["x4"], (B, H, W, 128), 1, w5, sl5, 64, B, (H, W), box, 256, sh5, act=1, out=x5, **reuse)
        Fn.adaptive_avg_pool4(x5, ws["pool"])
        return 1

    def _compact(self, H: int, W: int) -> bool:
        """The fused front end can read the depth image through sliding-window tensor maps (no row-im2col tensor in HBM)
        when its tile is 128 consecutive pixels of a row and the width is even."""
        return self.use_fused_front and self.use_compact_operand and _best_box(H, W) == (128, 1) and W % 2 == 0

    # ---- .train(): batch-statistics BatchNorm + Dropout (CM:1380-1437 with the modules in training mode; SURVEY H6) -------
    TRAIN_MODE_SUPPORTED = True

    def _refresh_train(self):
        """Un-folded weights for the train-mode passes: the BatchNorm scale depends on the batch, so it is folded into the
        bf16 weights per step (after the statistics pass that ran on the plain bf16 weights)."""
        srcs = [p for p in self.parameters()]
        if not self._ver_train.stale(srcs) and self._packed_train:
            return self._packed_train
        dev = srcs[0].device
        bf = torch.bfloat16
        with torch.no_grad():
            w1 = torch.zeros(192, 4, 2, 8, 4, device=dev, dtype=torch.float32)
            for idx, (seq, k) in enumerate(((self.scale1_conv, 3), (self.scale2_conv, 5), (self.scale3_conv, 7))):
                o = (7 - k) // 2
                full = torch.zeros(64, self.input_channels, 8, 8, device=dev)
                full[:, :, o:o + k, o:o + k] = seq[0].weight.float()
                w1[idx * 64:(idx + 1) * 64, :, :, :, :self.input_channels] = full.reshape(64, self.input_channels, 4, 2, 8).permute(0, 2, 3, 4, 1)
            pk = {"w1": w1.reshape(192, 256).contiguous(),
                  "w2": self.feature_fusion[0].weight.float().reshape(128, 192).contiguous(),
                  "w5": self.feature_extractor[0].weight.float().permute(0, 2, 3, 1).reshape(256, 9 * 128).contiguous()}
            for k in ("w1", "w2", "w5"):
                pk[k + "_bf"] = pk[k].to(bf).contiguous()
            pk["zeros"] = torch.zeros(256, device=dev, dtype=torch.float32)
            # layers without BatchNorm + slice tables: the same operands as the eval path (kept here so that the running
            # statistics, which change every training step, do not invalidate them)
            pk["w3"] = self.attention[0].weight.float().reshape(64, 128).to(bf).contiguous()
            pk["sh3"] = self.attention[0].bias.detach().float().contiguous()
            pk["w4"] = self.attention[2].weight.float().reshape(128, 64).to(bf).contiguous()
            pk["sh4"] = self.attention[2].bias.detach().float().contiguous()
            pk["w6"] = self.feature_extractor[4].weight.detach().float().contiguous()
            for j, li in enumerate((0, 3, 6, 8)):
                pk[f"fw{j}"] = self.fc_layers[li].weight.detach().float().contiguous()
                pk[f"fb{j}"] = self.fc_layers[li].bias.detach().float().contiguous()

            def sl(entries):
                return torch.tensor(entries, device=dev, dtype=torch.int32).contiguous()
            pk["sl1"] = sl([(0, 0, 2 * t, 0) for t in range(4)])
            pk["sl2"] = sl([(64 * cb, 0, 0, 0) for cb in range(3)])
            pk["sl3"] = sl([(64 * cb, 0, 0, 0) for cb in range(2)])
            pk["sl4"] = sl([(0, 0, 0, 0)])
            pk["sl5"] = sl([(64 * cb, dx - 1, dy - 1, 0) for dy in range(3) for dx in range(3) for cb in range(2)])
        self._packed_train = pk
        return pk

    @staticmethod
    def _batch_norm_train(sum_fx: torch.Tensor, sq_fx: torch.Tensor, count: int, bn: nn.BatchNorm2d,
                          conv_bias: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Fixed-point per-image sums of the raw conv outputs (and of their squares) -> this batch's BatchNorm as a
        per-channel (scale, shift); ``bn``'s running statistics are updated like torch does (CM:1382 et al. in training
        mode: momentum * batch mean / UNBIASED batch variance).  The conv bias cancels in the normalised value."""
        c = bn.num_features
        mean = sum_fx[:c].double() / (Fn.POOL_FIXED_ONE * count)
        var = (sq_fx[:c].double() / (Fn.POOL_FIXED_ONE * count) - mean * mean).clamp_min(0.0)
        scale = bn.weight.double() / torch.sqrt(var + bn.eps)
        shift = bn.bias.double() - mean * scale
        if bn.track_running_stats and bn.running_mean is not None:
            bn.num_batches_tracked += 1
            m = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
            bn.running_mean.mul_(1 - m).add_((m * (mean + conv_bias.double())).float())
            bn.running_var.mul_(1 - m).add_((m * var * (count / max(count - 1, 1))).float())
        return scale.float(), shift.float()

    def _forward_train(self, depth_image: torch.Tensor, dropout_masks=None) -> torch.Tensor:
        B, _, H, W = depth_image.shape
        dev = depth_image.device
        pt = self._refresh_train()
        pk = pt
        key = (B, H, W, str(dev), "train")
        if key not in self._ws:
            _evict(self._ws)
            bf = dict(device=dev, dtype=torch.bfloat16)
            self._ws[key] = {"stem": torch.empty(B, H + 6, W, 64, **bf), "x1": torch.empty(B, H, W, 192, **bf),
                             "x2": torch.empty(B, H, W, 128, **bf), "x3": torch.empty(B, H, W, 64, **bf),
                             "x4": torch.empty(B, H, W, 128, **bf),
                             "pool": torch.empty(B, 16, 256, device=dev, dtype=torch.int64),
                             "stat": torch.empty(2, B, 1, 256, device=dev, dtype=torch.int64)}
        ws = self._ws[key]
        d = depth_image.detach()
        d = d if d.dtype == torch.float32 else d.float()
        box = _best_box(H, W)
        n = B * H * W
        bf = torch.bfloat16

        def stats(operand, a_dims, w_bf, slices, n_out, **kw):
            st = ws["stat"][:, :, :, :n_out].contiguous() if n_out != 256 else ws["stat"]
            st.zero_()
            Fn.conv_gemm(operand, a_dims, 1, w_bf, slices, 64, B, (H, W), box, n_out, pt["zeros"][:n_out], act=3, epi_mode=2,
                         pool=st[0], pool_sq=st[1], cells=(1, 1), **kw)
            return st[0].sum(dim=(0, 1)), st[1].sum(dim=(0, 1))

        with torch.no_grad():
            Fn.ratio_stem_pack(d, ws["stem"])
            # multi-scale stem (CM:1458-1463): statistics pass, then conv + BN(batch) + ReLU
            s1, q1 = stats(ws["stem"], (B, H + 6, W, 64), pt["w1_bf"], pk["sl1"], 192, tile_order=1)
            sc, sh = zip(*[self._batch_norm_train(s1[i * 64:(i + 1) * 64], q1[i * 64:(i + 1) * 64], n, seq[1], seq[0].bias)
                           for i, seq in enumerate((self.scale1_conv, self.scale2_conv, self.scale3_conv))])
            sc1, sh1 = torch.cat(sc), torch.cat(sh).contiguous()
            Fn.conv_gemm(ws["stem"], (B, H + 6, W, 64), 1, (pt["w1"] * sc1[:, None]).to(bf).contiguous(), pk["sl1"], 64, B, (H, W),
                         box, 192, sh1, act=1, out=ws["x1"], tile_order=1)
            # feature_fusion (CM:1466)
            s2, q2 = stats(ws["x1"], (B, H, W, 192), pt["w2_bf"], pk["sl2"], 128)
            sc2, sh2 = self._batch_norm_train(s2, q2, n, self.feature_fusion[1], self.feature_fusion[0].bias)
            Fn.conv_gemm(ws["x1"], (B, H, W, 192), 1, (pt["w2"] * sc2[:, None]).to(bf).contiguous(), pk["sl2"], 64, B, (H, W), box,
                         128, sh2.contiguous(), act=1, out=ws["x2"])
            # attention (CM:1469-1470; no BatchNorm)
            Fn.conv_gemm(ws["x2"], (B, H, W, 128), 1, pk["w3"], pk["sl3"], 64, B, (H, W), box, 64, pk["sh3"], act=1, out=ws["x3"])
            Fn.conv_gemm(ws["x3"], (B, H, W, 64), 1, pk["w4"], pk["sl4"], 64, B, (H, W), box, 128, pk["sh4"], act=2,
                         gate=ws["x2"], out=ws["x4"])
            # feature_extractor[0:4] (CM:1412-1416)
            reuse = dict(tile_order=1, conv3x3_reuse=(box == (128, 1)))
            s5, q5 = stats(ws["x4"], (B, H, W, 128), pt["w5_bf"], pk["sl5"], 256, **reuse)
            sc5, sh5 = self._batch_norm_train(s5, q5, n, self.feature_extractor[1], self.feature_extractor[0].bias)
            cell_pixels = self._conv5_pool(ws, (pt["w5"] * sc5[:, None]).to(bf).contiguous(), pk["sl5"], sh5.contiguous(), B, H, W, box)
            # feature_extractor[4:7] + GAP + fc_layers with Dropout (CM:1418-1437)
            mult = []
            for j, (p_drop, width) in enumerate(((self.fc_layers[2].p, 128), (self.fc_layers[5].p, 64))):
                keep = dropout_masks[j] if dropout_masks is not None else torch.rand(B, width, device=dev) >= p_drop
                keep = keep.to(device=dev)
                if tuple(keep.shape) != (B, width):
                    raise RgbdB200Error(f"dropout_masks[{j}] must be {(B, width)} keep-masks")
                mult.append((keep.float() / (1.0 - p_drop)).contiguous())
            bn6, c6 = self.feature_extractor[5], self.feature_extractor[4]
            track = bn6.track_running_stats and bn6.running_mean is not None
            if track:
                bn6.num_batches_tracked += 1
            m6 = bn6.momentum if bn6.momentum is not None else 1.0 / float(bn6.num_batches_tracked)
            return Fn.ratio_tail_train(ws["pool"], cell_pixels, pk["w6"], c6.bias.detach().float().contiguous(),
                                       bn6.weight.detach().float().contiguous(), bn6.bias.detach().float().contiguous(), bn6.eps,
                                       m6, bn6.running_mean if track else None, bn6.running_var if track else None,
                                       [pk[f"fw{j}"] for j in range(4)], [pk[f"fb{j}"] for j in range(4)], mult[0], mult[1],
                                       self.output_min, self.output_max)

    def forward(self, depth_image: torch.Tensor, dropout_masks=None) -> torch.Tensor:
        """``dropout_masks`` (train mode only): optional ((B,128), (B,64)) boolean KEEP masks of the two Dropout layers
        (CM:1430, 1433); drawn from torch's generator when omitted."""
        assert depth_image.dim() == 4, f"Expected 4D tensor, got {depth_image.dim()}D"
        assert depth_image.shape[1] == self.input_channels, \
            f"Expected {self.input_channels} channels, got {depth_image.shape[1]}"
        B, _, H, W = depth_image.shape
        if self.training:
            return self._forward_train(depth_image, dropout_masks if dropout_masks is not None else self.dropout_masks_override)
        pk = self._refresh()
        ws = self._workspace(B, H, W, depth_image.device)
        d = depth_image.detach()
        if d.dtype != torch.float32:
            d = d.float()
        box = _best_box(H, W)
        compact = self._compact(H, W)
        if compact:
            Fn.ratio_stem_pack_compact(d, ws["stem"])
        else:
            Fn.ratio_stem_pack(d, ws["stem"])
        if self.use_fused_front:
            # stem + feature_fusion + attention + gating (CM:1458-1470) in one kernel; intermediates in tensor memory
            Fn.ratio_front(ws["stem"], pk["w1c"] if compact else pk["w1"], pk["w2"], pk["w3"], pk["w4"], pk["sh1"], pk["sh2"],
                           pk["sh3"], pk["sh4"], ws["x4"], box)
        else:
            # multi-scale stem (CM:1458-1463) + BN + ReLU -> 192 channels
            Fn.conv_gemm(ws["stem"], (B, H + 6, W, 64), 1, pk["w1"], pk["sl1"], 64, B, (H, W), box, 192, pk["sh1"],
                         act=1, out=ws["x1"], tile_order=1)   # walk down columns: the 4 row taps re-hit L2
        if self.use_fused_front:
            pass
        elif self.use_fused_chain:
            # feature_fusion + attention + gating (CM:1466-1470) as one kernel, intermediates in tensor memory
            Fn.ratio_chain(ws["x1"], pk["w2"], pk["w3"], pk["w4"], pk["sh2"], pk["sh3"], pk["sh4"], ws["x4"], box)
        else:
            # feature_fusion (CM:1466)
            Fn.conv_gemm(ws["x1"], (B, H, W, 192), 1, pk["w2"], pk["sl2"], 64, B, (H, W), box, 128, pk["sh2"],
                         act=1, out=ws["x2"])
            # attention (CM:1469-1470): sigmoid(conv(relu(conv(f)))) * f
            Fn.conv_gemm(ws["x2"], (B, H, W, 128), 1, pk["w3"], pk["sl3"], 64, B, (H, W), box, 64, pk["sh3"], act=1,
                         out=ws["x3"])
            Fn.conv_gemm(ws["x3"], (B, H, W, 64), 1, pk["w4"], pk["sl4"], 64, B, (H, W), box, 128, pk["sh4"], act=2,
                         gate=ws["x2"], out=ws["x4"])
        # feature_extractor[0:4] (CM:1412-1416): conv3x3 + BN + ReLU + AdaptiveAvgPool2d(4), pooled in the epilogue
        cell_pixels = self._conv5_pool(ws, pk["w5"], pk["sl5"], pk["sh5"], B, H, W, box)
        fcw, fcb = [pk[f"fw{j}"] for j in range(4)], [pk[f"fb{j}"] for j in range(4)]
        if self.use_tensor_core_tail:
            return Fn.ratio_tail_tc(ws["pool"], cell_pixels, ws["a6"], ws["gap_fx"], pk["w6_bf"], pk["sl6"], pk["sh6"],
                                    fcw, fcb, self.output_min, self.output_max)
        return Fn.ratio_tail(ws["pool"], cell_pixels, pk["w6"], pk["sc6"], pk["sh6"], fcw, fcb,
                             self.output_min, self.output_max)


class RatioPredictor(nn.Module):
    """CM:823-898: window_size_ratio from the depth ENCODER's feature maps (versions 0.1.3 / 0.3.0): global average
    pool per scale, concat, Linear sum(C)->64->32->1 with ReLU, ``output_min + span * sigmoid`` -> (B,1).  Forward only
    (the reference consumes the result through ``.item()``, CM:275)."""

    def __init__(self, depth_channels_list: List[int]):
        super().__init__()
        self.depth_channels_list = list(depth_channels_list)
        self.num_scales = len(self.depth_channels_list)
        self.fc_layers = nn.Sequential(nn.Linear(sum(self.depth_channels_list), 64), nn.ReLU(inplace=True),
                                       nn.Linear(64, 32), nn.ReLU(inplace=True), nn.Linear(32, 1))
        self.global_avg_pool = nn.AdaptiveAvgPool2d(1)
        self.output_min = 0.01
        self.output_max = 0.5
        self.sigmoid = nn.Sigmoid()

    def forward(self, depth_feature_maps: List[torch.Tensor]) -> torch.Tensor:
        assert len(depth_feature_maps) == self.num_scales, \
            f"Expected {self.num_scales} depth feature maps, but got {len(depth_feature_maps)}"
        for i, f in enumerate(depth_feature_maps):
            assert f.shape[1] == self.depth_channels_list[i], \
                f"Expected {self.depth_channels_list[i]} channels for scale {i}, but got {f.shape[1]}"
        fcs = [self.fc_layers[i] for i in (0, 2, 4)]
        return Fn.ratio_from_features([f.detach().float() for f in depth_feature_maps],
                                      [l.weight.detach().float().contiguous() for l in fcs],
                                      [l.bias.detach().float().contiguous() for l in fcs], self.output_min, self.output_max)


# =====================================================================================================
# v0.4.0 wiring
# =====================================================================================================
class DepthGuidance(nn.Module):
    """The hot path between the encoder and the pixel decoder of the v0.4.0 model (CM:324-355), batched and
    free of host synchronisation: ratio predictor -> device-side depth decomposition -> 3 cascaded DSAM
    stages -> DGGM injection fused with the branch sum.  Child names match the reference's pixel-level
    module (``ratio_predictor, dsam0, dsam1, dsam2, depth_gradient_injection``)."""

    def __init__(self, color_channels: Sequence[int] = (96, 192, 384, 768), precision: str = "bf16",
                 grad_precision: str = "bf16"):
        super().__init__()
        c = list(color_channels)
        assert len(c) == 4
        assert precision in ("bf16", "fp32")
        if grad_precision not in ("bf16", "fp32"):
            raise ValueError(f"grad_precision must be 'bf16' or 'fp32', got {grad_precision!r}")
        self.ratio_predictor = EnhancedDepthImageRatioPredictor(3)
        self.dsam0 = DSAModule(in_channels=c[0], out_channels=c[1], num_depth_regions=3)
        self.dsam1 = DSAModule(in_channels=c[1], out_channels=c[2], num_depth_regions=3)
        self.dsam2 = DSAModule(in_channels=c[2], out_channels=c[3], num_depth_regions=3)
        self.depth_gradient_injection = DepthGradientInjectionResidual(c, 3)
        for d in (self.dsam0, self.dsam1, self.dsam2):
            d.precision = precision            # DSAM convolutions; DGGM is fp32 arithmetic in either mode
            d.grad_precision = grad_precision  # DSAM dW and dx; independent of the forward's precision

    def forward(self, pixel_values: torch.Tensor, color_feature_map: Sequence[torch.Tensor],
                ratios: Optional[torch.Tensor] = None, out: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
        """``out``: optional preallocated fused feature maps (inference path), e.g. views of one device slab that a
        serving loop copies to the host in a single transfer."""
        return depth_guidance_forward(self.ratio_predictor, (self.dsam0, self.dsam1, self.dsam2),
                                      self.depth_gradient_injection, pixel_values, color_feature_map, ratios, out)


def dsam_cascade(dsams: Sequence[DSAModule], feats: Sequence[torch.Tensor], dec, training: bool) -> List[torch.Tensor]:
    """CM:339-352: ``cp1[k+1] += dsam_k(cp1[k])`` with the UPDATED cp1[k]; returns cp1.  Inference: stage k's epilogue also
    writes stage k+1's packed bf16 operand (no pack kernel in between)."""
    cp1 = [feats[0]]
    x = feats[0]
    prepacked = False
    for k, dsam in enumerate(dsams):
        if training or not FUSE_STAGE_PACKS:
            x = dsam.stage_forward(x, dec.pooled[k], dec.bias_variant, residual=feats[k + 1])
        else:
            emit = None
            if k + 1 < len(dsams):
                tgt = dsams[k + 1]._emit_target(x.shape[0], feats[k + 1].shape[2], feats[k + 1].shape[3], x.device)
                if tgt is not None:
                    emit = (tgt[0], tgt[1], dec.pooled[k + 1])
            x = dsam._stage_forward_impl(x, dec.pooled[k], dec.bias_variant, residual=feats[k + 1], emit_next=emit,
                                         prepacked=prepacked)
            prepacked = emit is not None
        cp1.append(x)
    return cp1


def depth_guidance_forward(ratio_predictor: EnhancedDepthImageRatioPredictor, dsams: Sequence[DSAModule],
                           dggm: DepthGradientInjectionResidual, pixel_values: torch.Tensor,
                           color_feature_map: Sequence[torch.Tensor], ratios: Optional[torch.Tensor] = None,
                           out: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
    """CM:324-355 from the encoder's feature maps to the list handed to the pixel decoder (inference path)."""
    depth = pixel_values[:, 3:6]
    gradient_depth = pixel_values[:, 6:9]
    gradient_mask = pixel_values[:, 9:10]
    feats = [f.detach().contiguous().float() for f in color_feature_map]   # CM:332-333 (detach; no clone needed)
    if ratios is None:
        ratios = ratio_predictor(depth)                                     # CM:336
    ratios = ratios.detach()                                                # consumed through .item() in CM:339
    levels = [tuple(f.shape[2:]) for f in feats[:3]]
    dec = Fn.depth_decompose(ratios.reshape(-1).contiguous(), levels, depth3=depth, want_codes=False)
    training = torch.is_grad_enabled() and any(p.requires_grad for m in (*dsams, dggm) for p in m.parameters())
    cp1 = dsam_cascade(dsams, feats, dec, training)                         # CM:339-352
    if training:
        if out is not None:
            raise RgbdB200Error("preallocated outputs are an inference-path option")
        cp2 = dggm(feats, gradient_depth, gradient_mask)                    # CM:354 (autograd: K1b)
        return [a + b for a, b in zip(cp1, cp2)]                            # CM:355
    # CM:354-355: cp2 = DGGM(feats); out = cp1 + cp2, fused into the DGGM kernel
    return dggm.forward_fused_sum(feats, cp1, gradient_depth, gradient_mask, outs=out)


class GraphedDepthGuidance:
    """The inference hot path captured once into a CUDA graph (static shapes, static input tensors): one graph launch
    replaces ~40 kernel launches per step.  ``inputs`` are the tensors captured; copy new data into them (or pass them
    as views of a staging buffer) and call the object to replay.  Outputs are the same tensors on every replay.

    The graph bakes in raw pointers to the modules' workspaces and packed bf16 weights.  The wrapper therefore (i) keeps
    its own references to every such tensor (eager calls at other shapes may evict them from the modules' caches, but
    cannot free them), and (ii) refuses to replay once a parameter or buffer changed (optimizer step, load_state_dict):
    the packed weights inside the graph would be stale -- build a new ``GraphedDepthGuidance`` instead."""

    def __init__(self, module: DepthGuidance, pixel_values: torch.Tensor, color_feature_map: Sequence[torch.Tensor],
                 warmup: int = 2):
        if module.training:
            raise RgbdB200Error("GraphedDepthGuidance captures the INFERENCE path: call module.eval() first (in train mode the "
                                "ratio predictor would update its BatchNorm statistics on every replay)")
        self.module = module
        self.pixel_values = pixel_values
        self.features = list(color_feature_map)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):                       # allocates workspaces / packs weights outside the capture
                module(self.pixel_values, self.features)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self.outputs = module(self.pixel_values, self.features)
        self._keepalive = self._collect(module)
        self._param_key = self._versions(module)

    @staticmethod
    def _collect(module) -> list:
        """Every tensor reachable from the sub-modules' private caches (workspaces, packed weights, slice tables)."""
        kept = []

        def walk(o):
            if isinstance(o, torch.Tensor):
                kept.append(o)
            elif isinstance(o, dict):
                for v in o.values():
                    walk(v)
            elif isinstance(o, (list, tuple)):
                for v in o:
                    walk(v)
        for sub in module.modules():
            for name in ("_ws", "_ws_t", "_packed", "_packed_bwd"):
                walk(getattr(sub, name, None))
        return kept

    @staticmethod
    def _versions(module) -> tuple:
        return tuple((t.data_ptr(), t._version) for t in (*module.parameters(), *module.buffers()))

    def __call__(self) -> List[torch.Tensor]:
        if self._versions(self.module) != self._param_key:
            raise RgbdB200Error("GraphedDepthGuidance: a parameter or buffer changed after capture; the graph holds the "
                                "old packed weights -- capture a new graph")
        self.graph.replay()
        return self.outputs
