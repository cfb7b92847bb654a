"""Batched inference front door: uint8 RGB-D frames in host memory -> instance maps in host memory.

What ``predictor.predictor`` / ``process_prediction`` do per image in the reference (mask2former/predictor.py:19-36 and
:697-703: image processor -> model forward -> ``post_process_instance_segmentation``) as one pipelined, batched loop:

    pinned uint8 colour + depth  --H2D-->  rgbd_pack_pixel_values (K0: normalise + Sobel features, DL:386-425)
        -> RGB-D Mask2Former (stock Swin / pixel decoder / transformer decoder under bf16 autocast; the depth-guidance
           hot path CM:324-355 on this library's kernels; by default also the two decoder_ops kernels inside the stock
           decoders: deformable-attention sampling and the masked-attention mask)
        -> device post-processing (K5)  --D2H-->  pinned segmentation map + per-segment labels / scores / counts
           (``return_coco_annotation=True``: the map is run-length encoded on the device, and only the small CSR tables,
           then the used runs, are copied; ``return_pycocotools_rle=True``: the same with pycocotools' compressed strings, one
           per segment, instead of runs)

The device part of a step is replayed as one CUDA graph per staging buffer (``cuda_graph``), so the host only issues two copies
and a graph launch per batch.  Only ~1.2 MB per 480x640 frame crosses the host link on the way in and the painted instance map on the way out; encoder
features never leave the GPU.  H2D, compute and D2H run on three streams over two buffers, so step i's upload overlaps
step i-1's compute and step i-2's download.
"""
from __future__ import annotations

import contextlib
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import functional as Fn
from ._lib import RgbdB200Error


@contextlib.contextmanager
def _cached_host_tensors():
    """Stock Hugging Face code builds a few tiny device tensors from Python lists inside ``forward`` (``torch.as_tensor(
    spatial_shapes_list, device=...)`` in the pixel decoder): pageable host-to-device copies, which a stream capture rejects.
    Inside this context such calls are served from a cache keyed by the list's contents (filled by an eager run first)."""
    cache: Dict = {}
    orig = torch.as_tensor

    def as_tensor(data, dtype=None, device=None):
        if isinstance(data, (list, tuple)) and device is not None and torch.device(device).type == "cuda":
            key = (repr(data), dtype, str(device))
            if key not in cache:
                cache[key] = orig(data, dtype=dtype, device=device)
            return cache[key]
        return orig(data, dtype=dtype, device=device)
    torch.as_tensor = as_tensor
    try:
        yield cache
    finally:
        torch.as_tensor = orig


class RgbdInstanceSegmenter:
    """``model``: a ``Mask2FormerForUniversalSegmentation`` whose pixel-level module is the RGB-D one
    (``pixel_level.build_rgbd_mask2former``), already on ``device`` and in eval mode.  ``fast_decoder_ops`` (default) rebinds
    forwards of the MODEL's stock submodules (``decoder_ops.install_fast_decoder_ops``: a side effect on the caller's model that
    stays until ``decoder_ops.uninstall_fast_decoder_ops(model)``; training and autograd keep using the stock forwards)."""

    def __init__(self, model, batch: int, frame_hw: Tuple[int, int], threshold: float = 0.5,
                 target_size: Optional[Tuple[int, int]] = None, autocast_dtype: Optional[torch.dtype] = torch.bfloat16,
                 fast_decoder_ops: bool = True, cuda_graph: Optional[bool] = None, return_coco_annotation: bool = False,
                 return_pycocotools_rle: bool = False):
        if return_coco_annotation and return_pycocotools_rle:
            raise ValueError("return_coco_annotation and return_pycocotools_rle can not be both set to True.")
        p = next(model.parameters())
        if not p.is_cuda:
            raise RgbdB200Error("RgbdInstanceSegmenter: the model must live on a CUDA device (no CPU path)")
        from . import decoder_ops
        if fast_decoder_ops:     # rgbd_msda_fwd / rgbd_attention_mask inside the stock pixel decoder / transformer decoder
            decoder_ops.install_fast_decoder_ops(model)
        else:
            decoder_ops.uninstall_fast_decoder_ops(model)
        self.fast_decoder_ops = bool(fast_decoder_ops)
        #: replay the whole device step (front-end, model, post-processing) as ONE CUDA graph per staging buffer: the step is
        #: ~1 800 kernel launches and, with decoder_ops on, its kernels (55 ms per 32 frames) finish before the host has launched
        #: them (60+ ms).  Needs the decoder_ops forwards (the stock deformable attention builds a device tensor from a Python
        #: list in every layer) and static shapes; the first call on each buffer runs eagerly, the second captures.  Parameters
        #: must not change afterwards (the hot path's packed weights are baked in): call ``invalidate_graphs()`` if they do.
        self.cuda_graph = bool(fast_decoder_ops) if cuda_graph is None else bool(cuda_graph)
        if self.cuda_graph and not fast_decoder_ops:
            raise RgbdB200Error("RgbdInstanceSegmenter: cuda_graph=True needs fast_decoder_ops=True")
        self._graphs = [None, None]
        self._calls = [0, 0]
        self._pool = None
        self._keep = []
        self.model = model
        self.device = p.device
        self.B = int(batch)
        self.H, self.W = int(frame_hw[0]), int(frame_hw[1])
        self.threshold = float(threshold)
        self.target = (self.H, self.W) if target_size is None else (int(target_size[0]), int(target_size[1]))
        self.autocast_dtype = autocast_dtype
        self.Q = int(model.config.num_queries)
        B, H, W, Q = self.B, self.H, self.W, self.Q
        Ht, Wt = self.target
        dev = self.device
        # two buffers per direction; host side pinned
        self.in_host = [(torch.empty(B, H, W, 3, dtype=torch.uint8).pin_memory(),
                         torch.empty(B, H, W, dtype=torch.uint8).pin_memory()) for _ in range(2)]
        self.in_dev = [(torch.empty(B, H, W, 3, dtype=torch.uint8, device=dev),
                        torch.empty(B, H, W, dtype=torch.uint8, device=dev)) for _ in range(2)]
        self.pv = [torch.empty(B, 10, H, W, dtype=torch.float32, device=dev) for _ in range(2)]
        self.out_dev: List[Optional[Fn.InstanceBatch]] = [None, None]
        #: HF's run-length lists instead of painted maps: the maps are encoded inside the step (and its graph), the
        #: download carries only the small CSR tables, and ``result`` copies the used runs.  The encoder's outputs and
        #: workspace are allocated here, outside the graphs' shared memory pool: ``result`` reads a buffer's runs after the
        #: other buffer's graph has started, and that graph may reuse whatever memory the first one freed during capture.
        self.return_coco_annotation = bool(return_coco_annotation)
        #: ``return_pycocotools_rle``: the same scheme with one pycocotools RLE string per segment, and ``result`` copies the
        #: used characters.
        self.return_pycocotools_rle = bool(return_pycocotools_rle)
        self.rle_dev = None
        if return_coco_annotation:
            self.rle_dev = [Fn.label_map_rle_buffers(B, Ht, Wt, Q, dev) for _ in range(2)]
        elif return_pycocotools_rle:
            self.rle_dev = [Fn.instance_rle_buffers(B, Ht, Wt, Q, dev) for _ in range(2)]
        if self.rle_dev is not None:
            n_off = Q + 2 if return_coco_annotation else Q + 1
            tables = {"offsets": torch.empty(B, n_off, dtype=torch.int32), "base": torch.empty(B + 1, dtype=torch.int32),
                      "bad": torch.empty(1, dtype=torch.int32)}
        else:
            tables = {"segmentation": torch.empty(B, Ht, Wt, dtype=torch.int32)}
        self.out_host = [{**{k: v.pin_memory() for k, v in tables.items()},
                          "labels": torch.empty(B, Q, dtype=torch.int32).pin_memory(),
                          "scores": torch.empty(B, Q, dtype=torch.float32).pin_memory(),
                          "count": torch.empty(B, dtype=torch.int32).pin_memory()} for _ in range(2)]
        self.s_in, self.s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        self.s_runs = torch.cuda.Stream(device=dev) if self.rle_dev is not None else None
        self._runs_host: Optional[torch.Tensor] = None      # pinned, grown on demand, reused by every ``result``
        self._chars_host: Optional[torch.Tensor] = None     # the same for ``return_pycocotools_rle``
        self.h2d_bytes_per_step = B * H * W * 4
        self._table_d2h_bytes = sum(t.numel() * t.element_size() for t in self.out_host[0].values())
        #: bytes the last ``result`` copied after the tables: 8 per run with ``return_coco_annotation``, 1 per character
        #: with ``return_pycocotools_rle``, 0 with both off
        self.runs_d2h_bytes = 0
        self._ev_in = [None, None]
        self._ev_free = [None, None]
        self._ev_d2h = [None, None]
        self._step = 0

    @property
    def d2h_bytes_per_step(self) -> int:
        """Bytes copied device -> host per step: the pinned download of the step, plus, with ``return_coco_annotation``
        or ``return_pycocotools_rle``, the runs or characters of the step whose ``result`` was read last (their number
        depends on the frames)."""
        return self._table_d2h_bytes + self.runs_d2h_bytes

    # ---- one device step ---------------------------------------------------------------------------
    @property
    def ready(self) -> bool:
        """True once nothing one-off is left for the next ``submit`` (workspaces allocated, graphs captured)."""
        return all(g is not None for g in self._graphs) if self.cuda_graph else self._step >= 2

    def warmup(self) -> None:
        """Re-submit what the staging buffers hold until ``ready`` (the first two steps run eagerly, the next two capture)."""
        while not self.ready:
            self.submit()
        self.drain()

    def invalidate_graphs(self) -> None:
        """Drop the captured graphs (after ``load_state_dict`` / any parameter change); the next calls capture again."""
        self._graphs, self._calls, self._keep = [None, None], [0, 0], []

    def _compute(self, b: int) -> None:
        if not self.cuda_graph:
            return self._step_eager(b)
        if self._graphs[b] is None:
            self._calls[b] += 1
            if self._calls[b] < 2:        # first call on this buffer: eager (allocates workspaces, packs weights, warms cuBLAS)
                return self._step_eager(b)
            with _cached_host_tensors() as cache:
                self._step_eager(b)       # fills the host-tensor cache
                g = torch.cuda.CUDAGraph()
                # thread_local: CUDA calls of other threads (NCCL watchdog, samplers) must not invalidate this capture
                with torch.cuda.graph(g, pool=self._pool, capture_error_mode="thread_local"):
                    self._step_eager(b)
                if self._pool is None:
                    self._pool = g.pool()
                self._keep.append(cache)
            self._graphs[b] = g
        self._graphs[b].replay()

    def _step_eager(self, b: int) -> None:
        rgb, depth = self.in_dev[b]
        with torch.no_grad():
            Fn.pack_pixel_values(rgb, depth, out=self.pv[b])
            if self.autocast_dtype is not None:
                with torch.autocast("cuda", dtype=self.autocast_dtype):
                    out = self.model(pixel_values=self.pv[b])
            else:
                out = self.model(pixel_values=self.pv[b])
            self.out_dev[b] = Fn.post_process_instances(out.class_queries_logits.float().contiguous(),
                                                        out.masks_queries_logits.float().contiguous(),
                                                        self.threshold, self.target, want_segmentation=True)
            if self.return_coco_annotation:
                Fn.label_map_rle(self.out_dev[b].segmentation, self.Q, *self.rle_dev[b])
            elif self.return_pycocotools_rle:
                Fn.instance_rle(self.out_dev[b].segmentation, self.out_dev[b].count, self.Q, *self.rle_dev[b])

    def submit(self, rgb_u8: Optional[torch.Tensor] = None, depth_u8: Optional[torch.Tensor] = None) -> int:
        """Enqueue one batch (host uint8 tensors (B,H,W,3) / (B,H,W); ``None`` re-sends what the staging buffer holds).
        Returns the buffer index whose results ``result(b)`` reads once the download has finished."""
        b = self._step & 1
        self._step += 1
        main = torch.cuda.current_stream(self.device)
        if rgb_u8 is not None:
            # the staging buffer may still be read by the H2D of two steps ago
            if self._ev_in[b] is not None:
                self._ev_in[b].synchronize()
            self.in_host[b][0].copy_(rgb_u8)
            self.in_host[b][1].copy_(depth_u8)
        with torch.cuda.stream(self.s_in):
            if self._ev_free[b] is not None:
                self.s_in.wait_event(self._ev_free[b])
            self.in_dev[b][0].copy_(self.in_host[b][0], non_blocking=True)
            self.in_dev[b][1].copy_(self.in_host[b][1], non_blocking=True)
            self._ev_in[b] = self.s_in.record_event()
        main.wait_event(self._ev_in[b])
        if self._ev_d2h[b] is not None:
            main.wait_event(self._ev_d2h[b])
        self._compute(b)
        self._ev_free[b] = main.record_event()
        r = self.out_dev[b]
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self._ev_free[b])
            oh = self.out_host[b]
            if self.rle_dev is not None:
                e = self.rle_dev[b][0]
                oh["offsets"].copy_(e.offsets, non_blocking=True)
                oh["base"].copy_(e.base, non_blocking=True)
                oh["bad"].copy_(e.bad, non_blocking=True)
            else:
                oh["segmentation"].copy_(r.segmentation, non_blocking=True)
            oh["labels"].copy_(r.labels, non_blocking=True)
            oh["scores"].copy_(r.scores, non_blocking=True)
            oh["count"].copy_(r.count, non_blocking=True)
            self._ev_d2h[b] = self.s_out.record_event()
        return b

    def drain(self) -> None:
        """Make the current stream wait for every outstanding download (call before timing stops / reading results)."""
        main = torch.cuda.current_stream(self.device)
        for e in self._ev_d2h:
            if e is not None:
                main.wait_event(e)

    def result(self, b: int, copy: bool = True) -> List[Dict]:
        """HF-shaped results of buffer ``b`` (``post_process_instance_segmentation`` return structure, PR:701-703).  The pinned
        staging buffer is reused by the second-next ``submit``: the maps are copied out unless ``copy=False`` (then they are
        views that stay valid only until that submit).

        With ``return_coco_annotation`` "segmentation" is HF's run-length list of lists, and this call copies the used runs
        of buffer ``b`` from the device (8 bytes per run) after the table download.  That is valid only because ``result(b)``
        is called before the second-next ``submit``, which would overwrite them: the same rule as for the staging buffers.
        With ``return_pycocotools_rle`` "segmentation" is one ``{"size": [h, w], "counts": bytes}`` per segment, and this
        call copies the used characters of buffer ``b`` under the same rule (1 byte per character)."""
        self._ev_d2h[b].synchronize()
        oh = self.out_host[b]
        if self.return_coco_annotation:
            if int(oh["bad"][0]):
                raise RgbdB200Error(f"RgbdInstanceSegmenter: {int(oh['bad'][0])} painted pixels outside [-1, {self.Q})")
            n_runs = int(oh["base"][self.B])
            if self._runs_host is None or self._runs_host.shape[0] < n_runs:
                cap = max(n_runs, 2 * (0 if self._runs_host is None else self._runs_host.shape[0]), 1)
                self._runs_host = torch.empty(cap, 2, dtype=torch.int32).pin_memory()
            runs = self._runs_host[:n_runs]
            with torch.cuda.stream(self.s_runs):       # not behind the next step's work on the main / download streams
                runs.copy_(self.rle_dev[b][0].runs[:n_runs], non_blocking=True)
            self.s_runs.synchronize()
            self.runs_d2h_bytes = n_runs * 8
            from .postprocess import rle_lists_from_csr
            seg = rle_lists_from_csr(oh["offsets"].numpy(), oh["base"].numpy(), runs.numpy())
        elif self.return_pycocotools_rle:
            if int(oh["bad"][0]):
                raise RgbdB200Error(f"RgbdInstanceSegmenter: {int(oh['bad'][0])} painted pixels outside the kept segments")
            n_chars = int(oh["base"][self.B])
            if self._chars_host is None or self._chars_host.shape[0] < n_chars:
                cap = max(n_chars, 2 * (0 if self._chars_host is None else self._chars_host.shape[0]), 1)
                self._chars_host = torch.empty(cap, dtype=torch.uint8).pin_memory()
            chars = self._chars_host[:n_chars]
            with torch.cuda.stream(self.s_runs):       # not behind the next step's work on the main / download streams
                chars.copy_(self.rle_dev[b][0].chars[:n_chars], non_blocking=True)
            self.s_runs.synchronize()
            self.runs_d2h_bytes = n_chars
            from .postprocess import pycocotools_rle_from_csr
            seg = pycocotools_rle_from_csr(oh["offsets"].numpy(), oh["base"].numpy(), chars.numpy(), oh["count"].tolist(),
                                           self.target)
        else:
            seg = oh["segmentation"].clone() if copy else oh["segmentation"]
        res = []
        for i in range(self.B):
            n = int(oh["count"][i])
            info = [{"id": j, "label_id": int(oh["labels"][i, j]), "was_fused": False,
                     "score": round(float(oh["scores"][i, j]), 6)} for j in range(n)]
            res.append({"segmentation": seg[i], "segments_info": info})
        return res

    def __call__(self, rgb_u8: torch.Tensor, depth_u8: torch.Tensor) -> List[Dict]:
        """Synchronous convenience: one batch in, its results out."""
        b = self.submit(rgb_u8, depth_u8)
        return self.result(b)
