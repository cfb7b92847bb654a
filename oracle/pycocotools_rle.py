"""numpy restatement of pycocotools' run-length format (``maskApi.c``): ``rleEncode`` / ``rleToString`` and their inverses
``rleFrString`` / ``rleDecode``, for one 2-D mask.  ``encode(mask)`` gives what
``pycocotools.mask.encode(np.asfortranarray(mask.astype(np.uint8)))`` gives: ``{"size": [h, w], "counts": bytes}``."""
from typing import Dict, List

import numpy as np


def rle_counts(mask: np.ndarray) -> List[int]:
    """``rleEncode``: the column-major scan of ``mask != 0`` as alternating run lengths of 0s and 1s, starting with 0s (the
    first count may be 0; the last run is always emitted)."""
    flat = (np.asarray(mask) != 0).reshape(-1, order="F").astype(np.int8)
    change = np.flatnonzero(np.diff(flat)) + 1                       # positions where the value changes
    edges = np.concatenate([[0], change, [flat.size]])
    counts = [int(c) for c in np.diff(edges)]
    return [0] + counts if flat[0] == 1 else counts


def counts_to_string(counts: List[int]) -> bytes:
    """``rleToString``: count i minus count i-2 when i > 2, then 5-bit groups, low bits first, 0x20 = more follow, +48."""
    out = bytearray()
    for i, x in enumerate(counts):
        x = int(x)
        if i > 2:
            x -= int(counts[i - 2])
        more = True
        while more:
            c = x & 0x1F
            x >>= 5                                                  # Python's >> is arithmetic, like the C on a long
            more = (x != -1) if (c & 0x10) else (x != 0)
            if more:
                c |= 0x20
            out.append(c + 48)
    return bytes(out)


def string_to_counts(s: bytes) -> List[int]:
    """``rleFrString``: the inverse of ``counts_to_string``."""
    counts: List[int] = []
    p = 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            c = s[p] - 48
            x |= (c & 0x1F) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)                                   # sign extension
        if len(counts) > 2:
            x += counts[-2]
        counts.append(x)
    return counts


def decode_counts(counts: List[int], h: int, w: int) -> np.ndarray:
    """``rleDecode``: the (h, w) uint8 mask of alternating 0/1 runs in column-major order."""
    vals = np.arange(len(counts)) % 2
    flat = np.repeat(vals.astype(np.uint8), np.asarray(counts, dtype=np.int64))
    if flat.size != h * w:
        raise ValueError(f"counts cover {flat.size} pixels, expected {h * w}")
    return flat.reshape((h, w), order="F")


def encode(mask: np.ndarray) -> Dict:
    h, w = np.asarray(mask).shape
    return {"size": [int(h), int(w)], "counts": counts_to_string(rle_counts(mask))}


def decode(rle: Dict) -> np.ndarray:
    h, w = rle["size"]
    counts = rle["counts"]
    return decode_counts(string_to_counts(counts.encode("ascii") if isinstance(counts, str) else counts), h, w)
