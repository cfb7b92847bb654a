"""``torch.ops.rgbd_b200.*``: the C-ABI entry points registered with the PyTorch dispatcher (SURVEY 8b).

The kernels live behind the C ABI (include/rgbd_b200.h, csrc/librgbd_b200.so); ``functional.py`` marshals tensors into it.
This module registers the same calls as dispatcher operators through ``torch.library`` (the Python face of
``TORCH_LIBRARY``): every op has a schema, a CUDA implementation that goes straight to the C ABI, a fake (meta) kernel so
``torch.compile`` / ``torch.export`` can trace through it as an opaque node, and -- where the reference's autograd reaches
the op -- an autograd formula (DGGM: CM:1251 has trainable 1x1 convs; the other ops are integer / data-side and carry none).
There is still no CPU implementation: calling an op with CPU tensors raises.

    import rgbd_b200.ops                      # registers the namespace
    outs = torch.ops.rgbd_b200.dggm_forward(feats, grad, mask, weights, biases)
"""


from typing import List, Tuple

import torch
from torch import Tensor

from . import functional as Fn

NAMESPACE = "rgbd_b200"


# ---------------------------------------------------------------------------------------------------------------------
# DGGM (K1 / K1b) -- differentiable w.r.t. the colour features (identity) and the 1x1 conv parameters
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NAMESPACE}::dggm_forward", mutates_args=())
def dggm_forward(feats: List[Tensor], grad: Tensor, mask: Tensor, weights: List[Tensor], biases: List[Tensor]) -> List[Tensor]:
    """``DepthGradientInjectionResidual.forward`` (CM:1204-1269): out_i = feats_i + ReLU(conv1x1_i(bilinear(grad) * nearest(mask)))."""
    return Fn.dggm_forward([f.contiguous() for f in feats], grad, mask, [w.detach() for w in weights], [b.detach() for b in biases])


@dggm_forward.register_fake
def _(feats, grad, mask, weights, biases):
    return [torch.empty_like(f) for f in feats]


@torch.library.custom_op(f"{NAMESPACE}::dggm_backward_params", mutates_args=())
def dggm_backward_params(douts: List[Tensor], grad: Tensor, mask: Tensor, weights: List[Tensor], biases: List[Tensor]) -> List[Tensor]:
    """Gradients of the DGGM 1x1 convs: [dW_0..dW_{n-1}, db_0..db_{n-1}]."""
    dws, dbs = Fn.dggm_backward_params(douts, grad, mask, weights, biases)
    return [*dws, *dbs]


@dggm_backward_params.register_fake
def _(douts, grad, mask, weights, biases):
    return [torch.empty_like(w) for w in weights] + [torch.empty_like(b) for b in biases]


def _dggm_setup(ctx, inputs, output):
    feats, grad, mask, weights, biases = inputs
    ctx.n = len(feats)
    ctx.save_for_backward(grad, mask, *weights, *biases)


def _dggm_backward(ctx, douts):
    n = ctx.n
    grad, mask = ctx.saved_tensors[:2]
    weights, biases = list(ctx.saved_tensors[2:2 + n]), list(ctx.saved_tensors[2 + n:2 + 2 * n])
    douts = [d.contiguous() for d in douts]
    g = torch.ops.rgbd_b200.dggm_backward_params(douts, grad, mask, weights, biases)
    # d(out)/d(feats) is the identity; the gradient map and the mask are data (SURVEY H11)
    return douts, None, None, g[:n], g[n:]


dggm_forward.register_autograd(_dggm_backward, setup_context=_dggm_setup)


# ---------------------------------------------------------------------------------------------------------------------
# front-end (K0), decomposition (K2), grayscale -- integer / data-side ops, no autograd
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NAMESPACE}::gradient_features", mutates_args=())
def gradient_features(depth: Tensor, n_rep: int = 3, invalid_value: float = 0.0) -> Tuple[Tensor, Tensor]:
    """``calculate_gradient_features`` (DP:1247-1305): depth (B,H,W) f32/u8 -> (normalised Sobel magnitude (B,n_rep,H,W), mask (B,1,H,W))."""
    return Fn.gradient_features(depth, n_rep, invalid_value)


@gradient_features.register_fake
def _(depth, n_rep=3, invalid_value=0.0):
    B, H, W = depth.shape
    return depth.new_empty((B, n_rep, H, W), dtype=torch.float32), depth.new_empty((B, 1, H, W), dtype=torch.float32)


@torch.library.custom_op(f"{NAMESPACE}::pack_pixel_values", mutates_args=())
def pack_pixel_values(rgb_u8: Tensor, depth_u8: Tensor) -> Tensor:
    """Front-end of ``map_10channel_case2`` (DL:386-425): uint8 colour (B,H,W,3) + depth (B,H,W) -> pixel_values (B,10,H,W)."""
    return Fn.pack_pixel_values(rgb_u8, depth_u8)


@pack_pixel_values.register_fake
def _(rgb_u8, depth_u8):
    B, H, W = depth_u8.shape
    return depth_u8.new_empty((B, 10, H, W), dtype=torch.float32)


@torch.library.custom_op(f"{NAMESPACE}::to_grayscale", mutates_args=())
def to_grayscale(image: Tensor) -> Tensor:
    """``to_grayscale`` (CM:466-480) for (B,3,H,W) float32: (0.299 r + 0.587 g) + 0.114 b, bit-exact."""
    return Fn.to_grayscale(image)


@to_grayscale.register_fake
def _(image):
    return image.new_empty((image.shape[0], image.shape[2], image.shape[3]))


@torch.library.custom_op(f"{NAMESPACE}::depth_decompose", mutates_args=())
def depth_decompose(depth3: Tensor, ratio: Tensor, level_h: List[int], level_w: List[int]) -> List[Tensor]:
    """CM:701-798 + CM:687 batched: [pooled region codes per level ..., bias_variant (B), n_modes (B), windows (B,3,2), centres (B,3)]."""
    dec = Fn.depth_decompose(ratio.reshape(-1).contiguous(), list(zip(level_h, level_w)), depth3=depth3, want_codes=False)
    # the per-image tables are views of one allocation inside functional.depth_decompose; dispatcher ops must not return
    # outputs that alias each other
    return [*dec.pooled, dec.bias_variant.clone(), dec.n_modes.clone(), dec.windows.clone(), dec.centres.clone()]


@depth_decompose.register_fake
def _(depth3, ratio, level_h, level_w):
    B = depth3.shape[0]
    u8 = dict(dtype=torch.uint8)
    return ([depth3.new_empty((B, h, w), **u8) for h, w in zip(level_h, level_w)] +
            [depth3.new_empty((B,), dtype=torch.int32), depth3.new_empty((B,), dtype=torch.int32),
             depth3.new_empty((B, 3, 2)), depth3.new_empty((B, 3))])


# ---------------------------------------------------------------------------------------------------------------------
# post-processing (K5)
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NAMESPACE}::post_process_instances", mutates_args=())
def post_process_instances(class_logits: Tensor, mask_logits: Tensor, threshold: float, target_h: int, target_w: int) -> List[Tensor]:
    """HF ``post_process_instance_segmentation`` (model_essential_part.py:86-91): [masks, labels, scores, query, count, segmentation]."""
    r = Fn.post_process_instances(class_logits, mask_logits, threshold, (target_h, target_w), want_segmentation=True)
    return [r.masks, r.labels, r.scores, r.query, r.count, r.segmentation]


@post_process_instances.register_fake
def _(class_logits, mask_logits, threshold, target_h, target_w):
    B, Q = class_logits.shape[:2]
    e = class_logits.new_empty
    return [e((B, Q, target_h, target_w), dtype=torch.uint8), e((B, Q), dtype=torch.int32), e((B, Q), dtype=torch.float32),
            e((B, Q), dtype=torch.int32), e((B,), dtype=torch.int32), e((B, target_h, target_w), dtype=torch.int32)]


@torch.library.custom_op(f"{NAMESPACE}::label_map_rle", mutates_args=())
def label_map_rle(seg: Tensor, n_labels: int) -> List[Tensor]:
    """HF ``convert_segmentation_to_rle`` per image of (B,H,W) int32 maps, as CSR: [offsets (B,L+2), base (B+1), runs
    (B*H*W,2) 1-based inclusive (start, end), out-of-range pixel count (1)]."""
    r = Fn.label_map_rle(seg, n_labels)
    return [r.offsets, r.base, r.runs, r.bad]


@label_map_rle.register_fake
def _(seg, n_labels):
    B, H, W = seg.shape
    e = seg.new_empty
    i32 = dict(dtype=torch.int32)
    return [e((B, n_labels + 2), **i32), e((B + 1,), **i32), e((B * H * W, 2), **i32), e((1,), **i32)]


@torch.library.custom_op(f"{NAMESPACE}::instance_rle", mutates_args=())
def instance_rle(seg: Tensor, count: Tensor, n_labels: int) -> List[Tensor]:
    """pycocotools RLE strings of the kept segments of (B,H,W) int32 painted maps, as CSR: [offsets (B,L+1), base (B+1),
    chars (7*B*(2*H*W+L),) uint8, bad pixel count (1)]."""
    r = Fn.instance_rle(seg, count, n_labels)
    return [r.offsets, r.base, r.chars, r.bad]


@instance_rle.register_fake
def _(seg, count, n_labels):
    B, H, W = seg.shape
    e = seg.new_empty
    i32 = dict(dtype=torch.int32)
    return [e((B, n_labels + 1), **i32), e((B + 1,), **i32), e((7 * B * (2 * H * W + n_labels),), dtype=torch.uint8),
            e((1,), **i32)]


@torch.library.custom_op(f"{NAMESPACE}::mask_iou", mutates_args=())
def mask_iou(pred_masks: Tensor, gt_masks: Tensor) -> Tensor:
    """(P,H,W) x (G,H,W) 0/1 masks -> (P,G) IoU (segm mAP of model_essential_part.py:111-170)."""
    return Fn.mask_iou(pred_masks, gt_masks)


@mask_iou.register_fake
def _(pred_masks, gt_masks):
    return pred_masks.new_empty((pred_masks.shape[0], gt_masks.shape[0]), dtype=torch.float32)


# ---------------------------------------------------------------------------------------------------------------------
# decoder_ops kernels: inference-only neighbours of the path inside the stock Hugging Face modules (no autograd)
# ---------------------------------------------------------------------------------------------------------------------
@torch.library.custom_op(f"{NAMESPACE}::msda_forward", mutates_args=())
def msda_forward(value: Tensor, level_h: List[int], level_w: List[int], sampling_locations: Tensor, attention_weights: Tensor) -> Tensor:
    """transformers ``multi_scale_deformable_attention(value, spatial_shapes, sampling_locations, attention_weights)``."""
    return Fn.msda_forward(value, list(zip(level_h, level_w)), sampling_locations, attention_weights)


@msda_forward.register_fake
def _(value, level_h, level_w, sampling_locations, attention_weights):
    B, _, H, D = value.shape
    return value.new_empty((B, sampling_locations.shape[1], H * D), dtype=torch.float32)


@torch.library.custom_op(f"{NAMESPACE}::attention_mask", mutates_args=())
def attention_mask(mask_logits: Tensor, target_h: int, target_w: int, num_heads: int) -> Tensor:
    """The attention-mask half of transformers ``Mask2FormerMaskPredictor.forward``: (B,Q,h,w) -> (B*heads, Q, th*tw) bool."""
    return Fn.attention_mask(mask_logits, (target_h, target_w), num_heads)


@attention_mask.register_fake
def _(mask_logits, target_h, target_w, num_heads):
    B, Q = mask_logits.shape[:2]
    return mask_logits.new_empty((B * num_heads, Q, target_h * target_w), dtype=torch.bool)


@torch.library.custom_op(f"{NAMESPACE}::window_attention", mutates_args=())
def window_attention(q: Tensor, k: Tensor, v: Tensor, bias: Tensor, mask: Tensor, num_heads: int) -> Tensor:
    """The inner op of transformers ``SwinSelfAttention.forward``; ``mask`` with zero windows (shape (0, N, N)) = no shift mask."""
    return Fn.window_attention(q, k, v, bias, mask if mask.shape[0] else None, num_heads)


@window_attention.register_fake
def _(q, k, v, bias, mask, num_heads):
    return torch.empty_like(q)


@torch.library.custom_op(f"{NAMESPACE}::masked_cross_attention", mutates_args=())
def masked_cross_attention(q: Tensor, k: Tensor, v: Tensor, attn_mask: Tensor, num_heads: int) -> Tensor:
    """The attention core of ``nn.MultiheadAttention`` with a boolean mask (Mask2Former decoder layers), bfloat16."""
    return Fn.masked_cross_attention(q, k, v, attn_mask, num_heads)


@masked_cross_attention.register_fake
def _(q, k, v, attn_mask, num_heads):
    return torch.empty_like(q)


@torch.library.custom_op(f"{NAMESPACE}::layer_norm", mutates_args=())
def layer_norm(x: Tensor, weight: Tensor, bias: Tensor, eps: float, bf16_out: bool = False) -> Tensor:
    """LayerNorm over the last dimension, float32 arithmetic, float32 or bfloat16 output."""
    return Fn.layer_norm(x, weight, bias, eps, out_dtype=torch.bfloat16 if bf16_out else torch.float32)


@layer_norm.register_fake
def _(x, weight, bias, eps, bf16_out=False):
    return x.new_empty(x.shape, dtype=torch.bfloat16 if bf16_out else torch.float32)


REGISTERED = ("dggm_forward", "dggm_backward_params", "gradient_features", "pack_pixel_values", "to_grayscale",
              "depth_decompose", "post_process_instances", "label_map_rle", "instance_rle", "mask_iou", "msda_forward", "attention_mask", "window_attention",
              "masked_cross_attention", "layer_norm")
