"""pycocotools RLE output on the device (csrc/postproc.cu coco_*_kernel): ``functional.instance_rle``,
``post_process_instance_segmentation(return_pycocotools_rle=True)`` and ``RgbdInstanceSegmenter(return_pycocotools_rle=True)``
against the numpy restatement of pycocotools' ``maskApi.c`` applied to the painted maps."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

pytestmark = pytest.mark.gpu

from oracle import pycocotools_rle as P                                         # noqa: E402
from oracle.make_golden_postproc import synth_outputs                            # noqa: E402
from test_gpu_rle import MODEL_SIZED                                             # noqa: E402
from test_pycocotools_rle_host import all_maps, instance_csr_reference          # noqa: E402


@pytest.fixture(scope="module")
def fn():
    import rgbd_b200  # noqa: F401
    from rgbd_b200 import functional
    functional._lib.load()
    return functional


def encode(fn, seg: np.ndarray, count, L: int, preallocated: bool = False):
    buffers = fn.instance_rle_buffers(*seg.shape, L, "cuda") if preallocated else ()
    r = fn.instance_rle(torch.from_numpy(seg).cuda(), torch.tensor(count, dtype=torch.int32, device="cuda"), L, *buffers)
    base = r.base.cpu()
    return r.offsets.cpu(), base, bytes(r.chars[:int(base[-1])].cpu().numpy()), int(r.bad.cpu()[0])


def check_device_encoding(fn, seg: np.ndarray, count, L: int):
    offsets, base, chars, bad = encode(fn, seg, count, L)
    ref = instance_csr_reference(seg, count, L)
    assert np.array_equal(offsets.numpy(), ref[0]) and np.array_equal(base.numpy(), ref[1])
    assert chars == ref[2] and bad == ref[3]
    again = encode(fn, seg, count, L, preallocated=True)     # deterministic: a second run gives identical outputs
    assert torch.equal(again[0], offsets) and torch.equal(again[1], base) and again[2] == chars and again[3] == bad


@pytest.mark.parametrize("name,seg,L", all_maps(), ids=[c[0] for c in all_maps()])
def test_device_encoder_on_crafted_maps(fn, name, seg, L):
    check_device_encoding(fn, seg[None], [L], L)


def test_device_encoder_batches_with_differing_counts(fn):
    maps = [m for _, m, _ in all_maps() if m.shape == (8, 6)]
    seg = np.stack(maps + [np.full((8, 6), 3, np.int32), np.full((8, 6), -1, np.int32)] + maps)
    check_device_encoding(fn, seg, [4, 2, 3, 0, 1, 4, 0][:seg.shape[0]], 4)
    rs = np.random.RandomState(9)
    blocks = np.kron(rs.randint(-1, 100, size=(5, 24, 32)), np.ones((1, 20, 20), int)).astype(np.int32)   # 480x640 maps
    check_device_encoding(fn, np.ascontiguousarray(blocks), [100, 100, 60, 1, 0], 100)
    yy, xx = np.mgrid[0:480, 0:640]
    checker = np.stack([np.where((yy + xx) % 2 == 0, 0, -1), np.where((yy + xx) % 2 == 0, 1, 0)]).astype(np.int32)
    check_device_encoding(fn, checker, [1, 2], 2)
    check_device_encoding(fn, np.ascontiguousarray(rs.randint(-1, 4096, size=(2, 33, 65)).astype(np.int32)),
                          [4096, 3000], 4096)


def test_out_of_range_ids_and_counts_go_to_bad(fn):
    seg = np.array([[[0, 5, -2, 0], [1, 1, 3, 2]], [[-1, -1, 7, -1], [0, 0, 2, 0]], [[0, 1, 0, 1], [2, 2, 2, 2]]],
                   np.int32)
    # image 0: 5, -2 and 3 lie outside [-1, 3); image 1: 7, and one pixel of id 2 >= count 2; image 2: count -1 adds 1
    # and leaves its 8 painted pixels without a segment
    offsets, base, chars, bad = encode(fn, seg, [3, 2, -1], 3)
    assert bad == 3 + 1 + 1 + (1 + 8)
    assert offsets[2].tolist() == [0, 0, 0, 0] and int(base[3]) == int(base[2])
    ref = instance_csr_reference(seg, [3, 2, -1], 3)
    assert np.array_equal(offsets.numpy(), ref[0]) and chars == ref[2] and bad == ref[3]
    assert encode(fn, seg[2:], [4], 3)[3] == 1 + 8                           # count above L


def test_output_or_workspace_alone_is_used_in_place(fn):
    _, seg, L = next(c for c in all_maps() if c[0] == "checker_big")
    seg = seg[None]
    ref = encode(fn, seg, [L], L)
    t, c = torch.from_numpy(seg).cuda(), torch.tensor([L], dtype=torch.int32, device="cuda")
    out, ws = fn.instance_rle_buffers(*seg.shape, L, "cuda")
    assert fn.instance_rle(t, c, L, out=out) is out
    assert torch.equal(out.offsets.cpu(), ref[0]) and bytes(out.chars[:int(ref[1][-1])].cpu().numpy()) == ref[2]
    r = fn.instance_rle(t, c, L, workspace=ws)
    assert torch.equal(r.offsets.cpu(), ref[0]) and bytes(r.chars[:int(ref[1][-1])].cpu().numpy()) == ref[2]


def test_arguments_checked(fn):
    from rgbd_b200._lib import RgbdB200Error
    seg = torch.zeros(1, 4, 4, dtype=torch.int32, device="cuda")
    cnt = torch.ones(1, dtype=torch.int32, device="cuda")
    for bad_args in [(seg.cpu(), cnt, 3), (seg.long(), cnt, 3), (seg, cnt.long(), 3), (seg, cnt[:0], 3), (seg, cnt, 4097)]:
        with pytest.raises(RgbdB200Error):
            fn.instance_rle(*bad_args)


def check_results(flag_off, flag_on):
    n_segments = 0
    for m, r in zip(flag_off, flag_on):
        assert r["segments_info"] == m["segments_info"]
        painted = m["segmentation"].cpu().numpy().astype(np.int64)
        assert len(r["segmentation"]) == len(m["segments_info"])
        for s, rle in enumerate(r["segmentation"]):
            assert rle == P.encode(painted == s)
            assert np.array_equal(P.decode(rle), (painted == s).astype(np.uint8))
        n_segments += len(r["segmentation"])
    return n_segments


@pytest.mark.parametrize("case", MODEL_SIZED, ids=[c[0] for c in MODEL_SIZED])
def test_post_process_pycocotools_rle_equals_encoding_of_the_map(fn, case):
    from rgbd_b200 import postprocess as PP
    name, seed, B, Q, C, hw, thr, tgt = case
    cls, masks = synth_outputs(seed, B, Q, C, *hw)
    outs = SimpleNamespace(class_queries_logits=cls.cuda(), masks_queries_logits=masks.cuda())
    sizes = None if tgt is None else [tgt] * B
    maps = PP.post_process_instance_segmentation(outs, threshold=thr, target_sizes=sizes)
    rle = PP.post_process_instance_segmentation(outs, threshold=thr, target_sizes=sizes, return_pycocotools_rle=True)
    assert check_results(maps, rle) > 0
    for r, size in zip(rle, sizes or [(384, 384)] * B):
        assert all(x["size"] == list(size) for x in r["segmentation"])


def test_post_process_pycocotools_rle_mixed_target_sizes_and_flags(fn):
    from rgbd_b200 import postprocess as PP
    cls, masks = synth_outputs(34, 3, 20, 8, 30, 40)
    outs = SimpleNamespace(class_queries_logits=cls.cuda(), masks_queries_logits=masks.cuda())
    sizes = [(480, 640), (120, 160), (480, 640)]
    maps = PP.post_process_instance_segmentation(outs, threshold=0.3, target_sizes=sizes)
    rle = PP.post_process_instance_segmentation(outs, threshold=0.3, target_sizes=sizes, return_pycocotools_rle=True)
    assert check_results(maps, rle) > 0
    assert [r["segmentation"][0]["size"] for r in rle if r["segmentation"]] == [list(s) for s, r in zip(sizes, rle)
                                                                               if r["segmentation"]]
    for other in ("return_coco_annotation", "return_binary_maps"):
        with pytest.raises(ValueError):
            PP.post_process_instance_segmentation(outs, target_sizes=sizes, return_pycocotools_rle=True, **{other: True})


@pytest.mark.parametrize("cuda_graph", [False, True], ids=["eager", "cuda_graph"])
def test_serving_pycocotools_rle_equals_encoding_of_maps(cuda_graph):
    """Pipelined batches through ``RgbdInstanceSegmenter(return_pycocotools_rle=True)``: each result equals the encoding of
    the map a segmenter with the flag off returns for the same frames, with the exact download size after each result."""
    from rgbd_b200 import serving, synthetic, synthetic_weights as SW
    model, _ = SW.build_synthetic_rgbd_mask2former(decisive=True, num_labels=8)
    model.cuda()
    B, H, W = 2, 128, 160
    kw = dict(threshold=0.5, cuda_graph=cuda_graph) if cuda_graph else dict(threshold=0.5, cuda_graph=False, autocast_dtype=None)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    with pytest.raises(ValueError):
        serving.RgbdInstanceSegmenter(model, B, (H, W), return_coco_annotation=True, return_pycocotools_rle=True, **kw)
    on = serving.RgbdInstanceSegmenter(model, B, (H, W), return_pycocotools_rle=True, **kw)
    off = serving.RgbdInstanceSegmenter(model, B, (H, W), **kw)
    Q = model.config.num_queries
    tables = 4 * (2 * B * Q + B + B * (Q + 1) + B + 1 + 1)           # labels, scores, count, offsets, base, bad
    assert on.d2h_bytes_per_step == tables                         # no result read yet: the pinned tables only
    batches = []
    for k in range(6):
        rgbs, ds = zip(*[synthetic.synth_rgbd_u8(900 + 10 * k + j, H, W, "nyu") for j in range(B)])
        batches.append((torch.from_numpy(np.stack(rgbs)), torch.from_numpy(np.stack(ds))))
    got = []

    def take(b):
        got.append(on.result(b))
        n_chars = sum(len(x["counts"]) for img in got[-1] for x in img["segmentation"])
        assert on.runs_d2h_bytes == n_chars and on.d2h_bytes_per_step == tables + n_chars
    pending = None
    for rgb, d in batches:                                         # two submits in flight
        b = on.submit(rgb, d)
        if pending is not None:
            take(pending)
        pending = b
    take(pending)
    n_segments = 0
    for (rgb, d), res in zip(batches, got):
        n_segments += check_results(off(rgb, d), res)
        assert all(x["size"] == [H, W] for img in res for x in img["segmentation"])
    assert n_segments > 0
    if cuda_graph:
        assert on._graphs[0] is not None and on._graphs[1] is not None
