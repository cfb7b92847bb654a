"""Run-length (COCO) output of the instance post-processing, host side: a numpy reference of the CSR layout that
``functional.label_map_rle`` returns equals HuggingFace's ``convert_segmentation_to_rle`` on crafted maps, the CPU assembly
``postprocess.rle_lists_from_csr`` turns that CSR into exactly HF's lists, and the dispatcher op traces with a fake kernel."""
import numpy as np
import pytest
import torch
from transformers.models.mask2former.image_processing_mask2former import convert_segmentation_to_rle

import rgbd_b200  # noqa: F401
from rgbd_b200.postprocess import rle_lists_from_csr


def crafted_maps():
    """(name, (H,W) int32 map with labels in [-1, L), L)."""
    rs = np.random.RandomState(5)
    yy, xx = np.mgrid[0:8, 0:6]
    maps = [
        ("hf_example", np.array([[-1, 0, 0, 1], [1, 1, -1, -1], [2, 2, 2, 2]]), 3),
        ("all_background", np.full((4, 5), -1), 3),
        ("one_id_everywhere", np.full((6, 7), 0), 1),
        ("painted_over", np.where(rs.rand(9, 11) > 0.5, 2, 0), 3),          # id 1 painted over completely: no list
        ("row_wrap", np.array([[0, 0, 0, 1, 1], [1, 1, 1, 1, 2], [2, 2, -1, -1, -1]]), 3),
        ("first_last_pixel", np.array([[3] + [0] * 6] + [[0] * 7] * 3 + [[0] * 6 + [4]]), 5),
        ("checker_even_w", np.where((yy + xx) % 2 == 0, 0, -1), 1),
        ("checker_odd_w", np.where((np.mgrid[0:7, 0:5].sum(0)) % 2 == 0, 1, 0), 2),
        ("one_by_one", np.array([[0]]), 1),
        ("one_by_one_bg", np.array([[-1]]), 0),
        ("one_row", rs.randint(-1, 3, size=(1, 37)), 3),
        ("one_col", rs.randint(-1, 3, size=(41, 1)), 3),
        ("odd_blobs", np.kron(rs.randint(-1, 5, size=(8, 10)), np.ones((5, 6), int))[:37, :53], 5),
        ("labels_150", rs.randint(-1, 150, size=(40, 60)), 150),
        # runs longer than a warp's 1024-pixel span and maps over several spans
        ("stripes", np.repeat(np.arange(-1, 4), 20)[:, None].repeat(64, 1)[:97], 4),
        ("checker_big", np.where((np.mgrid[0:97, 0:132].sum(0)) % 2 == 0, 7, -1), 8),
    ]
    return [(n, np.ascontiguousarray(m, dtype=np.int32), L) for n, m, L in maps]


def csr_reference(seg: np.ndarray, L: int):
    """numpy CSR of a (B,H,W) batch: offsets (B, L+2) relative to base (B+1), runs (base[B], 2) of 1-based inclusive
    (start, end), ordered by label, then position, image by image."""
    B = seg.shape[0]
    offsets = np.zeros((B, L + 2), np.int64)
    base = np.zeros(B + 1, np.int64)
    runs = []
    for b in range(B):
        f = seg[b].reshape(-1).astype(np.int64)
        N = f.size
        is_start = np.ones(N, bool)
        is_start[1:] = f[1:] != f[:-1]
        is_end = np.ones(N, bool)
        is_end[:-1] = f[:-1] != f[1:]
        s, e = np.flatnonzero(is_start), np.flatnonzero(is_end)
        order = np.lexsort((s, f[s]))                      # label-major, then position; the i-th end closes the i-th start
        s, e = s[order], e[np.lexsort((e, f[e]))]
        assert np.array_equal(f[s], f[e])
        offsets[b, 1:] = np.cumsum(np.bincount(f[s] + 1, minlength=L + 1))
        base[b + 1] = base[b] + len(s)
        runs.append(np.stack([s + 1, e + 1], axis=1))
    return offsets, base, np.concatenate(runs).reshape(-1, 2)


def hf_lists(seg: np.ndarray):
    return [convert_segmentation_to_rle(torch.from_numpy(m).float()) for m in seg]


def assert_same_lists(got, want):
    assert got == want
    for g_img in got:
        for lst in g_img:
            assert all(type(v) is int for v in lst)


def test_hf_worked_example():
    seg = np.array([[[-1, 0, 0, 1], [1, 1, -1, -1], [2, 2, 2, 2]]], np.int32)
    assert hf_lists(seg) == [[[1, 1, 7, 2], [2, 2], [4, 3], [9, 4]]]
    assert rle_lists_from_csr(*csr_reference(seg, 3)) == [[[1, 1, 7, 2], [2, 2], [4, 3], [9, 4]]]


@pytest.mark.parametrize("name,seg,L", crafted_maps(), ids=[c[0] for c in crafted_maps()])
def test_csr_reference_and_assembly_equal_hf(name, seg, L):
    offsets, base, runs = csr_reference(seg[None], L)
    assert runs.shape[0] == base[-1] <= seg.size
    assert_same_lists(rle_lists_from_csr(offsets, base, runs), hf_lists(seg[None]))


def test_assembly_of_a_batch_and_skipped_ids():
    maps = [m for _, m, _ in crafted_maps() if m.shape == (8, 6)]
    seg = np.stack(maps + [np.full((8, 6), 2, np.int32), np.full((8, 6), -1, np.int32)])
    offsets, base, runs = csr_reference(seg, 4)
    lists = rle_lists_from_csr(offsets, base, runs)
    assert_same_lists(lists, hf_lists(seg))
    assert lists[-2] == [[1, 48]] and lists[-1] == [[1, 48]]         # a lone id 2 and all background: one list each
    # torch CPU tensors and a base with only the first B entries work the same
    assert rle_lists_from_csr(torch.from_numpy(offsets).int(), torch.from_numpy(base[:-1]).int(), torch.from_numpy(runs).int()) == lists


def test_label_map_rle_fake_kernel_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from rgbd_b200 import ops
    assert "label_map_rle" in ops.REGISTERED
    with FakeTensorMode():
        out = torch.ops.rgbd_b200.label_map_rle(torch.empty(3, 48, 64, dtype=torch.int32, device="cuda"), 100)
        assert [tuple(t.shape) for t in out] == [(3, 102), (4,), (3 * 48 * 64, 2), (1,)]
        assert all(t.dtype == torch.int32 for t in out)


def test_workspace_query_applies_the_encoder_argument_rules():
    from rgbd_b200 import _lib, functional as Fn
    from rgbd_b200._lib import RgbdB200Error
    q = _lib.load().rgbd_label_map_rle_workspace_bytes
    assert q(32, 480, 640, 100) >= 32 * 101 * 300 * 4
    assert q(1, 46341, 46341, 1) == 0                          # H*W >= 2^31: the int product would overflow
    assert q(8, 16384, 16384, 1) == 0 and q(65536, 1, 1, 1) == 0 and q(1, 4, 4, 4097) == 0 and q(1, 4, 4, -1) == 0
    assert q(0, 4, 4, 1) == 0 and q(1, 0, 4, 1) == 0
    with pytest.raises(RgbdB200Error, match="unsupported"):
        Fn.label_map_rle_buffers(8, 16384, 16384, 1, "cpu")    # refused before the (B*H*W, 2) runs are allocated
