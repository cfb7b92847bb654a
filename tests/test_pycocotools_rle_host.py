"""pycocotools RLE output of the instance post-processing, host side: the numpy restatement of pycocotools' ``maskApi.c``
(``oracle/pycocotools_rle.py``) against known answers derived by hand from its rules, a numpy reference of the CSR that
``functional.instance_rle`` returns, a numpy walk of the device's item layout that must rebuild that CSR, the CPU
assembly ``postprocess.pycocotools_rle_from_csr``, ``postprocess.coco_results``, and the dispatcher op's fake kernel."""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import rgbd_b200  # noqa: E402,F401
from oracle import pycocotools_rle as P                                 # noqa: E402
from rgbd_b200.postprocess import coco_results, pycocotools_rle_from_csr  # noqa: E402
from test_rle_host import crafted_maps, csr_reference                   # noqa: E402


def _mask(h, w, pixels=(), rows=(), cols=()):
    m = np.zeros((h, w), np.uint8)
    for y, x in pixels:
        m[y, x] = 1
    for y in rows:
        m[y, :] = 1
    for x in cols:
        m[:, x] = 1
    return m


block = _mask(4, 4)
block[1:3, 1:3] = 1
KNOWN = [
    ("ones_2x2", np.ones((2, 2), np.uint8), [0, 4], b"04"),
    ("zeros_2x2", np.zeros((2, 2), np.uint8), [4], b"4"),
    ("zeros_10x10", np.zeros((10, 10), np.uint8), [100], b"T3"),
    ("first_pixel_3x4", _mask(3, 4, pixels=[(0, 0)]), [0, 1, 11], b"01;"),
    ("last_pixel_3x4", _mask(3, 4, pixels=[(2, 3)]), [11, 1], b";1"),
    ("row0_3x4", _mask(3, 4, rows=[0]), [0, 1, 2, 1, 2, 1, 2, 1, 2], b"012000000"),
    ("col1_3x4", _mask(3, 4, cols=[1]), [3, 3, 6], b"336"),
    ("block_4x4", block, [5, 2, 2, 2, 5], b"52203"),
    ("col_5x1", np.array([[1], [1], [1], [0], [1]], np.uint8), [0, 3, 1, 1], b"031N"),
]


@pytest.mark.parametrize("name,mask,counts,string", KNOWN, ids=[k[0] for k in KNOWN])
def test_known_answers(name, mask, counts, string):
    assert P.rle_counts(mask) == counts
    assert P.counts_to_string(counts) == string
    assert P.encode(mask) == {"size": list(mask.shape), "counts": string}
    assert P.string_to_counts(string) == counts
    assert np.array_equal(P.decode(P.encode(mask)), mask)


@pytest.mark.parametrize("value,string", [(15, b"?"), (16, b"`0"), (31, b"o0"), (32, b"P1"), (511, b"o?"), (512, b"P`0")])
def test_known_single_values(value, string):
    assert P.counts_to_string([value]) == string
    assert P.string_to_counts(string) == [value]


@pytest.mark.parametrize("delta,string", [(-1, b"O"), (-3, b"M"), (-16, b"@"), (-17, b"_O"), (16, b"`0"), (17, b"a0")])
def test_known_deltas(delta, string):
    # count 3 is written as count 3 - count 1; counts 0..2 are written as they are (i > 2, not i >= 2)
    counts = [0, 20, 1, 20 + delta]
    s = P.counts_to_string(counts)
    assert s == b"0" + P.counts_to_string([20]) + b"1" + string
    assert P.string_to_counts(s) == counts
    mask = P.decode_counts(counts + [1], sum(counts) + 1, 1)          # an N x 1 column holding those runs
    assert P.rle_counts(mask) == counts + [1]


def test_decode_inverts_encode_on_random_and_crafted_masks():
    rs = np.random.RandomState(3)
    masks = [rs.rand(h, w) < p for h, w, p in [(1, 1, 0.5), (1, 37, 0.5), (41, 1, 0.3), (17, 23, 0.5), (64, 48, 0.95),
                                              (64, 48, 0.02), (5, 300, 0.5)]]
    masks += [m == s for _, m, L in crafted_maps() for s in range(-1, L)]
    yy, xx = np.mgrid[0:31, 0:29]
    masks += [(yy + xx) % 2 == 0, (yy + xx) % 2 == 1, np.ones((31, 29), bool), np.zeros((31, 29), bool)]
    for m in masks:
        rle = P.encode(m)
        assert all(48 <= c <= 111 for c in rle["counts"])
        assert np.array_equal(P.decode(rle), m.astype(np.uint8))
        assert sum(P.rle_counts(m)) == m.size


# ---- the device CSR ------------------------------------------------------------------------------------------------
def instance_csr_reference(seg: np.ndarray, count, L: int):
    """What ``functional.instance_rle`` returns for (B,H,W) maps: offsets (B, L+1) relative to base (B+1), the used
    characters, and bad (pixels outside [-1, L) or in [count[b], L), plus 1 per count outside [0, L])."""
    B = seg.shape[0]
    offsets = np.zeros((B, L + 1), np.int64)
    base = np.zeros(B + 1, np.int64)
    chars = b""
    bad = int(((seg < -1) | (seg >= L)).sum())
    for b in range(B):
        n = int(count[b]) if 0 <= count[b] <= L else 0
        bad += (n != count[b]) + int(((seg[b] >= n) & (seg[b] < L)).sum())
        strings = [P.encode(seg[b] == s)["counts"] for s in range(n)]
        offsets[b, 1:] = np.cumsum([len(x) for x in strings] + [0] * (L - n))
        chars += b"".join(strings)
        base[b + 1] = len(chars)
    return offsets, base, chars, bad


def _put(x: int):
    return list(P.counts_to_string([x]))


def item_layout_csr(seg: np.ndarray, count, L: int):
    """The device's algorithm in numpy: label-major runs of the TRANSPOSED map, one item per run and one tail per segment
    placed at (run index - first non-background run + segment), character lengths from each run and the two before it,
    an exclusive scan per image, then the characters.  In-range ids only."""
    B, H, W = seg.shape
    N = H * W
    seg_t = np.ascontiguousarray(seg.transpose(0, 2, 1))
    off_r, base_r, runs = csr_reference(seg_t, L)
    offsets = np.zeros((B, L + 1), np.int64)
    images = []
    for b in range(B):
        o, rr, img = off_r[b], runs[base_r[b]:], seg_t[b].reshape(-1)
        n_runs = o[L + 1] - o[1]
        n = int(count[b]) if 0 <= count[b] <= L else 0
        length = np.zeros(n_runs + L, np.int64)
        items = []
        for t in range(n_runs + L):
            if t < n_runs:
                cur = rr[o[1] + t]
                s = img[cur[0] - 1]
                m = o[1] + t - o[s + 1]
                item = t + s
            else:
                s = t - n_runs
                m = o[s + 2] - o[s + 1]
                item = o[s + 2] - o[1] + s
            p1 = rr[o[s + 1] + m - 1] if m >= 1 else (0, 0)
            p2 = rr[o[s + 1] + m - 2] if m >= 2 else (0, 0)
            gap1 = p1[0] - 1 - p2[1]
            if t < n_runs:
                gap, ln = cur[0] - 1 - p1[1], cur[1] - cur[0] + 1
                values = [gap - gap1 if m >= 2 else gap, ln - (p1[1] - p1[0] + 1) if m >= 1 else ln]
            else:
                tail = N - p1[1]
                values = [tail - gap1 if m >= 2 else tail] if tail > 0 else []
            ch = [c for v in values for c in _put(int(v))] if s < n else []
            length[item] = len(ch)
            items.append((item, s, m == 0, ch))
        pos = np.concatenate([[0], np.cumsum(length)])
        offsets[b, L] = pos[-1]
        images.append((items, pos))
    base = np.concatenate([[0], np.cumsum(offsets[:, L])])
    chars = bytearray(int(base[-1]))
    for b, (items, pos) in enumerate(images):
        for item, s, first, ch in items:
            if first:
                offsets[b, s] = pos[item]
            chars[base[b] + pos[item]:base[b] + pos[item] + len(ch)] = bytes(ch)
    return offsets, base, bytes(chars)


def extra_maps():
    """(name, (H,W) map, L) for the cases the encoder must get right besides ``crafted_maps``."""
    yy, xx = np.mgrid[0:6, 0:5]
    one_run_tail = np.full((6, 5), -1)
    one_run_tail[:, 1] = 0                          # id 0: exactly one run and a trailing count (count 2, not a delta)
    deltas = np.full((69, 1), -1)                   # id 0's counts: [1, 20, 20, 4, 3, 1, 20], deltas -16, -17, -3, +17
    for a, b_ in [(1, 21), (41, 45), (48, 49)]:
        deltas[a:b_, 0] = 0
    return [("one_run_and_tail", one_run_tail, 2),  # id 1 empty: [h*w]
            ("covers_everything", np.zeros((7, 3)), 1),
            ("deltas_16_17", deltas, 1),
            ("deltas_row", deltas.T.copy(), 1),
            ("checker_ids", (yy + xx) % 3, 3)]


def all_maps():
    return crafted_maps() + [(n, np.ascontiguousarray(m, dtype=np.int32), L) for n, m, L in extra_maps()]


@pytest.mark.parametrize("name,seg,L", all_maps(), ids=[c[0] for c in all_maps()])
def test_csr_reference_and_item_layout(name, seg, L):
    for n in sorted({L, max(L - 1, 0), L // 2}):
        offsets, base, chars, bad = instance_csr_reference(seg[None], [n], L)
        assert bad == int(((seg >= n) & (seg < L)).sum())
        got = item_layout_csr(seg[None], [n], L)
        assert np.array_equal(got[0], offsets) and np.array_equal(got[1], base) and got[2] == chars
        (rles,) = pycocotools_rle_from_csr(offsets, base, np.frombuffer(chars, np.uint8), [n], seg.shape)
        assert len(rles) == n
        for s, rle in enumerate(rles):
            assert rle == P.encode(seg == s) and type(rle["counts"]) is bytes
            assert np.array_equal(P.decode(rle), (seg == s).astype(np.uint8))


def test_reference_cases():
    """The cases the CSR tests must contain are there: an empty segment, a segment covering every pixel, first and last
    pixel, one run with a trailing count, deltas of -16 and -17, 1 x N and N x 1 maps."""
    strings = [P.encode(m == s)["counts"] for _, m, L in all_maps() for s in range(L)]
    counts = [P.string_to_counts(x) for x in strings]
    assert any(len(c) == 1 for c in counts)                               # empty segment: [h*w]
    assert any(c[0] == 0 and len(c) == 2 for c in counts)                 # every pixel
    assert any(c[0] == 0 and len(c) > 2 for c in counts)                  # first pixel
    assert any(len(c) % 2 == 0 and len(c) > 2 for c in counts)            # last pixel (ends on a 1-run)
    assert any(len(c) == 3 and c[0] > 0 for c in counts)                  # one run and a trailing count
    deltas = [c[i] - c[i - 2] for c in counts for i in range(3, len(c))]
    assert -16 in deltas and -17 in deltas and 17 in deltas
    shapes = {m.shape for _, m, _ in all_maps()}
    assert any(h == 1 and w > 1 for h, w in shapes) and any(w == 1 and h > 1 for h, w in shapes)


def test_batch_with_differing_counts():
    maps = [m for _, m, _ in crafted_maps() if m.shape == (8, 6)]
    seg = np.stack(maps + [np.full((8, 6), 3, np.int32), np.full((8, 6), -1, np.int32)] + maps)
    count = [4, 2, 3, 0, 1, 4][:seg.shape[0]]
    offsets, base, chars, bad = instance_csr_reference(seg, count, 4)
    got = item_layout_csr(seg, count, 4)
    assert np.array_equal(got[0], offsets) and np.array_equal(got[1], base) and got[2] == chars
    assert bad == sum(int(((seg[b] >= count[b]) & (seg[b] < 4)).sum()) for b in range(seg.shape[0]))
    rles = pycocotools_rle_from_csr(torch.from_numpy(offsets).int(), torch.from_numpy(base[:-1]).int(),
                                    chars, count, (8, 6))                  # torch tensors, bytes, B base entries
    assert [len(r) for r in rles] == count
    for b, img in enumerate(rles):
        for s, rle in enumerate(img):
            assert rle == P.encode(seg[b] == s)
    # a count outside [0, L] adds 1 and leaves the image without segments
    offsets, base, chars, bad = instance_csr_reference(seg[:2], [5, -1], 4)
    assert base[-1] == 0 and bad == 2 + int(((seg[:2] >= 0) & (seg[:2] < 4)).sum())


def test_coco_results_survive_a_json_round_trip():
    seg = crafted_maps()[0][1]
    offsets, base, chars, _ = instance_csr_reference(seg[None], [3], 3)
    (rles,) = pycocotools_rle_from_csr(offsets, base, np.frombuffer(chars, np.uint8), [3], seg.shape)
    info = [{"id": j, "label_id": 7 + j, "was_fused": False, "score": 0.5 + 0.125 * j} for j in range(3)]
    results = [{"segmentation": rles, "segments_info": info}, {"segmentation": [], "segments_info": []}]
    coco = coco_results(results, [42, 43])
    assert [c["category_id"] for c in coco] == [7, 8, 9] and all(c["image_id"] == 42 for c in coco)
    back = json.loads(json.dumps(coco))
    assert back == coco
    for j, c in enumerate(back):
        assert c["score"] == info[j]["score"] and c["segmentation"]["size"] == [3, 4]
        assert np.array_equal(P.decode(c["segmentation"]), (seg == j).astype(np.uint8))
    with pytest.raises(ValueError):
        coco_results(results, [1])


def test_instance_rle_fake_kernel_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from rgbd_b200 import ops
    assert "instance_rle" in ops.REGISTERED
    with FakeTensorMode():
        out = torch.ops.rgbd_b200.instance_rle(torch.empty(3, 48, 64, dtype=torch.int32, device="cuda"),
                                               torch.empty(3, dtype=torch.int32, device="cuda"), 100)
        assert [tuple(t.shape) for t in out] == [(3, 101), (4,), (7 * 3 * (2 * 48 * 64 + 100),), (1,)]
        assert [t.dtype for t in out] == [torch.int32, torch.int32, torch.uint8, torch.int32]


def test_queries_apply_the_encoder_argument_rules():
    from rgbd_b200 import _lib, functional as Fn
    from rgbd_b200._lib import RgbdB200Error
    lib = _lib.load()
    ws, cap = lib.rgbd_instance_rle_workspace_bytes, lib.rgbd_instance_rle_capacity
    assert cap(32, 480, 640, 100) == 7 * 32 * (2 * 480 * 640 + 100)
    assert ws(32, 480, 640, 100) >= 32 * 480 * 640 * (4 + 8 + 4)   # transposed map, runs, item positions
    assert cap(1, 1, 1, 0) == 14 and ws(1, 1, 1, 0) > 0
    # 7*B*(2*H*W + L) < 2^31: at the bound and one past it
    hw = (2 ** 31 - 1) // 14                                        # 7 * 1 * 2 * hw <= 2^31 - 1
    assert cap(1, hw, 1, 0) == 14 * hw and ws(1, hw, 1, 0) > 0
    assert cap(1, hw + 1, 1, 0) == 0 and ws(1, hw + 1, 1, 0) == 0
    assert cap(1, hw, 1, 1) == 0                                     # the L term counts too
    for q in (ws, cap):
        assert q(0, 4, 4, 1) == 0 and q(1, 0, 4, 1) == 0 and q(1, 4, 0, 1) == 0
        assert q(1, 4, 4, 4097) == 0 and q(1, 4, 4, -1) == 0 and q(65536, 1, 1, 1) == 0
        assert q(1, 46341, 46341, 1) == 0 and q(1, 4, 4, 4096) > 0
    with pytest.raises(RgbdB200Error, match="unsupported"):
        Fn.instance_rle_buffers(8, 8192, 8192, 1, "cpu")           # B*H*W < 2^31, but not the characters
