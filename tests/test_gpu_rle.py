"""Run-length (COCO) output on the device (csrc/postproc.cu rle_*_kernel): ``functional.label_map_rle``,
``post_process_instance_segmentation(return_coco_annotation=True)`` and ``RgbdInstanceSegmenter(return_coco_annotation=True)``
against HuggingFace's own ``convert_segmentation_to_rle``."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from transformers.models.mask2former.image_processing_mask2former import convert_segmentation_to_rle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

pytestmark = pytest.mark.gpu

from oracle.make_golden_postproc import CASES, synth_outputs           # noqa: E402
from test_rle_host import crafted_maps, csr_reference, hf_lists        # noqa: E402


@pytest.fixture(scope="module")
def fn():
    import rgbd_b200  # noqa: F401
    from rgbd_b200 import functional
    functional._lib.load()
    return functional


def encode(fn, seg: np.ndarray, L: int, preallocated: bool = False):
    buffers = fn.label_map_rle_buffers(*seg.shape, L, "cuda") if preallocated else ()
    r = fn.label_map_rle(torch.from_numpy(seg).cuda(), L, *buffers)
    base = r.base.cpu()
    return r.offsets.cpu(), base, r.runs[:int(base[-1])].cpu(), int(r.bad.cpu()[0])


def check_device_encoding(fn, seg: np.ndarray, L: int):
    from rgbd_b200.postprocess import rle_lists_from_csr
    offsets, base, runs, bad = encode(fn, seg, L)
    assert bad == 0
    ref = csr_reference(seg, L)
    assert np.array_equal(offsets.numpy(), ref[0]) and np.array_equal(base.numpy(), ref[1]) and np.array_equal(runs.numpy(), ref[2])
    assert rle_lists_from_csr(offsets, base, runs) == hf_lists(seg)
    again = encode(fn, seg, L, preallocated=True)     # deterministic: a second run gives identical tensors
    assert torch.equal(again[0], offsets) and torch.equal(again[1], base) and torch.equal(again[2], runs)


@pytest.mark.parametrize("name,seg,L", crafted_maps(), ids=[c[0] for c in crafted_maps()])
def test_device_encoder_on_crafted_maps(fn, name, seg, L):
    check_device_encoding(fn, seg[None], L)


def test_device_encoder_batches(fn):
    maps = [m for _, m, _ in crafted_maps() if m.shape == (8, 6)]
    check_device_encoding(fn, np.stack(maps + [np.full((8, 6), 2, np.int32), np.full((8, 6), -1, np.int32)] + maps), 4)
    rs = np.random.RandomState(9)
    blocks = np.kron(rs.randint(-1, 100, size=(5, 24, 32)), np.ones((1, 20, 20), int)).astype(np.int32)   # 480x640 maps
    check_device_encoding(fn, np.ascontiguousarray(blocks), 100)
    check_device_encoding(fn, np.ascontiguousarray(rs.randint(-1, 4096, size=(2, 33, 65)).astype(np.int32)), 4096)


def test_output_or_workspace_alone_is_used_in_place(fn):
    seg = crafted_maps()[-1][1][None]
    ref = encode(fn, seg, 8)
    t = torch.from_numpy(seg).cuda()
    out, ws = fn.label_map_rle_buffers(*seg.shape, 8, "cuda")
    assert fn.label_map_rle(t, 8, out=out) is out
    assert torch.equal(out.offsets.cpu(), ref[0]) and torch.equal(out.runs[:int(ref[1][-1])].cpu(), ref[2])
    r = fn.label_map_rle(t, 8, workspace=ws)
    assert torch.equal(r.offsets.cpu(), ref[0]) and torch.equal(r.runs[:int(ref[1][-1])].cpu(), ref[2])


def test_out_of_range_labels_are_counted_and_arguments_checked(fn):
    from rgbd_b200._lib import RgbdB200Error
    seg = np.array([[[0, 5, -2, 0], [1, 1, 3, 2]], [[-1, -1, 7, -1], [0, 0, 0, 0]]], np.int32)
    assert encode(fn, seg, 3)[3] == 4                 # 5, -2 and 3 in image 0, 7 in image 1
    with pytest.raises(RgbdB200Error):
        fn.label_map_rle(torch.zeros(1, 4, 4, dtype=torch.int32), 3)                       # CPU tensor
    with pytest.raises(RgbdB200Error):
        fn.label_map_rle(torch.zeros(1, 4, 4, dtype=torch.int64, device="cuda"), 3)        # wrong dtype
    with pytest.raises(RgbdB200Error):
        fn.label_map_rle(torch.zeros(1, 4, 4, dtype=torch.int32, device="cuda"), 4097)     # too many labels


MODEL_SIZED = [("default384", 31, 2, 100, 48, (96, 96), 0.05, None),
               ("b32_480x640", 32, 32, 100, 48, (120, 160), 0.0, (480, 640)),
               ("b2_960x1280", 33, 2, 100, 48, (240, 320), 0.05, (960, 1280))] + list(CASES)


@pytest.mark.parametrize("case", MODEL_SIZED, ids=[c[0] for c in MODEL_SIZED])
def test_post_process_rle_equals_hf_conversion_of_the_map(fn, case):
    from rgbd_b200 import postprocess as PP
    name, seed, B, Q, C, hw, thr, tgt = case
    cls, masks = synth_outputs(seed, B, Q, C, *hw)
    outs = SimpleNamespace(class_queries_logits=cls.cuda(), masks_queries_logits=masks.cuda())
    sizes = None if tgt is None else [tgt] * B
    maps = PP.post_process_instance_segmentation(outs, threshold=thr, target_sizes=sizes)
    rle = PP.post_process_instance_segmentation(outs, threshold=thr, target_sizes=sizes, return_coco_annotation=True)
    assert sum(len(r["segments_info"]) for r in maps) > 0
    for m, r in zip(maps, rle):
        assert r["segments_info"] == m["segments_info"]
        assert r["segmentation"] == convert_segmentation_to_rle(m["segmentation"].cpu())


def test_post_process_rle_mixed_target_sizes(fn):
    from rgbd_b200 import postprocess as PP
    cls, masks = synth_outputs(34, 3, 20, 8, 30, 40)
    outs = SimpleNamespace(class_queries_logits=cls.cuda(), masks_queries_logits=masks.cuda())
    sizes = [(480, 640), (120, 160), (480, 640)]
    maps = PP.post_process_instance_segmentation(outs, threshold=0.3, target_sizes=sizes)
    rle = PP.post_process_instance_segmentation(outs, threshold=0.3, target_sizes=sizes, return_coco_annotation=True)
    for m, r in zip(maps, rle):
        assert r["segments_info"] == m["segments_info"]
        assert r["segmentation"] == convert_segmentation_to_rle(m["segmentation"].cpu())


@pytest.mark.parametrize("cuda_graph", [False, True], ids=["eager", "cuda_graph"])
def test_serving_rle_equals_hf_conversion_of_maps(cuda_graph):
    """Pipelined batches through ``RgbdInstanceSegmenter(return_coco_annotation=True)``: each result equals HF's conversion of
    the map a segmenter with the flag off returns for the same frames."""
    from rgbd_b200 import serving, synthetic, synthetic_weights as SW
    model, _ = SW.build_synthetic_rgbd_mask2former(decisive=True, num_labels=8)
    model.cuda()
    B, H, W = 2, 128, 160
    kw = dict(threshold=0.5, cuda_graph=cuda_graph) if cuda_graph else dict(threshold=0.5, cuda_graph=False, autocast_dtype=None)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    on = serving.RgbdInstanceSegmenter(model, B, (H, W), return_coco_annotation=True, **kw)
    off = serving.RgbdInstanceSegmenter(model, B, (H, W), **kw)
    Q = model.config.num_queries
    tables = 4 * (2 * B * Q + B + B * (Q + 2) + B + 1 + 1)           # labels, scores, count, offsets, base, bad
    assert on.d2h_bytes_per_step == tables                         # no result read yet: the pinned tables only
    assert off.d2h_bytes_per_step > B * H * W * 4
    batches = []
    for k in range(6):
        rgbs, ds = zip(*[synthetic.synth_rgbd_u8(900 + 10 * k + j, H, W, "nyu") for j in range(B)])
        batches.append((torch.from_numpy(np.stack(rgbs)), torch.from_numpy(np.stack(ds))))
    got = []

    def take(b):
        got.append(on.result(b))
        n_runs = sum(len(lst) // 2 for img in got[-1] for lst in img["segmentation"])
        assert on.runs_d2h_bytes == 8 * n_runs and on.d2h_bytes_per_step == tables + 8 * n_runs
    pending = None
    for rgb, d in batches:                                         # two submits in flight
        b = on.submit(rgb, d)
        if pending is not None:
            take(pending)
        pending = b
    take(pending)
    n_segments = 0
    for (rgb, d), res in zip(batches, got):
        ref = off(rgb, d)
        for r, g in zip(ref, res):
            assert g["segments_info"] == r["segments_info"]
            assert g["segmentation"] == convert_segmentation_to_rle(r["segmentation"])
            n_segments += len(g["segments_info"])
    assert n_segments > 0
    if cuda_graph:
        assert on._graphs[0] is not None and on._graphs[1] is not None
