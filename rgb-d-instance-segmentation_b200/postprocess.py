"""Host-side mirror of the post-processing / evaluation interfaces the reference uses (SURVEY 8f-3).

* ``post_process_instance_segmentation`` has the signature and return structure of the HuggingFace
  ``Mask2FormerImageProcessor`` method the reference calls (mask2former/utils/model_essential_part.py:86-91,
  mask2former/predictor.py:34-36 and 701-703); the work runs in csrc/postproc.cu with ONE device->host read of the small
  per-segment tables at the end (HF syncs once per query through ``.item()``).  Segments come in a defined order (class
  score descending, flattened (query, label) index on ties); HF's ``topk(sorted=False)`` order is unspecified.
* ``postprocess_prediction_batch`` / ``MaskAP`` mirror ``Evaluator.postprocess_prediction_batch`` and the segm mAP the
  reference gets from torchmetrics (model_essential_part.py:83-170): IoU on the device, the COCO-style accumulation
  (101-point interpolated AP over IoU 0.50:0.05:0.95, per class, <= 100 detections per image) on the host.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import functional as Fn
from ._lib import RgbdB200Error


def _group_by_size(target_sizes: Sequence[Tuple[int, int]]) -> Dict[Tuple[int, int], List[int]]:
    groups: Dict[Tuple[int, int], List[int]] = {}
    for i, s in enumerate(target_sizes):
        groups.setdefault((int(s[0]), int(s[1])), []).append(i)
    return groups


def rle_lists_from_csr(offsets, base, runs) -> List[List[List[int]]]:
    """HF's ``convert_segmentation_to_rle`` lists from the CSR tables of ``functional.label_map_rle`` on the host:
    ``offsets`` (n, L+2) relative to ``base`` (>= n entries), ``runs`` the used prefix (R, 2) of 1-based inclusive
    (start, end) pairs.  Per image one ``[start_1, len_1, start_2, len_2, ...]`` list of Python ints for every label that
    has runs, in ascending label order."""
    offsets = np.asarray(offsets, dtype=np.int64)
    base = np.asarray(base, dtype=np.int64)
    runs = np.asarray(runs, dtype=np.int64).reshape(-1, 2)
    flat = np.stack([runs[:, 0], runs[:, 1] - runs[:, 0] + 1], axis=1).reshape(-1)
    out = []
    for b in range(offsets.shape[0]):
        bounds = 2 * (base[b] + offsets[b])
        present = np.flatnonzero(bounds[1:] > bounds[:-1])
        # slicing the array, then one tolist per list, makes each Python int once (measured faster than slicing a list)
        out.append([flat[lo:hi].tolist() for lo, hi in zip(bounds[present].tolist(), bounds[present + 1].tolist())])
    return out


def _download_with_rle(r: "Fn.InstanceBatch", n_labels: int):
    """Encode the painted maps of ``r`` on the device, then read the small tables in one copy and the used runs in one more.
    Returns (count list, labels (n,Q), scores (n,Q), per-image RLE lists)."""
    n, Q = r.labels.shape
    enc = Fn.label_map_rle(r.segmentation, n_labels)
    tables = torch.cat([r.count, r.labels.reshape(-1), r.scores.reshape(-1).view(torch.int32), enc.offsets.reshape(-1),
                        enc.base, enc.bad]).cpu()   # the one synchronisation of the batch
    sizes = [n, n * Q, n * Q, enc.offsets.numel(), n + 1, 1]
    count, labels, scores, offsets, base, bad = torch.split(tables, sizes)
    if int(bad[0]):
        raise RgbdB200Error(f"post_process_instance_segmentation: {int(bad[0])} painted pixels outside [-1, {n_labels})")
    runs = enc.runs[:int(base[n])].cpu()
    rle = rle_lists_from_csr(offsets.view(n, -1).numpy(), base.numpy(), runs.numpy())
    return count.tolist(), labels.view(n, Q), scores.view(torch.float32).view(n, Q), rle


def pycocotools_rle_from_csr(offsets, base, chars, count, size) -> List[List[Dict]]:
    """pycocotools RLEs from the CSR tables of ``functional.instance_rle`` on the host: ``offsets`` (n, L+1) relative to
    ``base`` (>= n entries), ``chars`` the used prefix of the characters (uint8 array or bytes), ``count`` the kept segments
    per image and ``size`` the maps' (h, w).  Per image one ``{"size": [h, w], "counts": bytes}`` per segment, in id order:
    what ``pycocotools.mask.encode`` returns for ``np.asfortranarray(map == s)``."""
    offsets = np.asarray(offsets, dtype=np.int64)
    base = np.asarray(base, dtype=np.int64)
    buf = chars if isinstance(chars, bytes) else np.ascontiguousarray(chars, dtype=np.uint8).tobytes()
    hw = [int(size[0]), int(size[1])]
    out = []
    for b in range(offsets.shape[0]):
        bounds = (base[b] + offsets[b, :int(count[b]) + 1]).tolist()
        out.append([{"size": list(hw), "counts": buf[lo:hi]} for lo, hi in zip(bounds[:-1], bounds[1:])])
    return out


def _download_with_pycocotools_rle(r: "Fn.InstanceBatch", n_labels: int, size):
    """Encode the kept segments of ``r`` on the device, then read the small tables in one copy and the used characters in
    one more.  Returns (count list, labels (n,Q), scores (n,Q), per-image pycocotools RLE lists)."""
    n, Q = r.labels.shape
    enc = Fn.instance_rle(r.segmentation, r.count, n_labels)
    tables = torch.cat([r.count, r.labels.reshape(-1), r.scores.reshape(-1).view(torch.int32), enc.offsets.reshape(-1),
                        enc.base, enc.bad]).cpu()   # the one synchronisation of the batch
    sizes = [n, n * Q, n * Q, enc.offsets.numel(), n + 1, 1]
    count, labels, scores, offsets, base, bad = torch.split(tables, sizes)
    if int(bad[0]):
        raise RgbdB200Error(f"post_process_instance_segmentation: {int(bad[0])} painted pixels outside the kept segments")
    chars = enc.chars[:int(base[n])].cpu()
    count = count.tolist()
    rle = pycocotools_rle_from_csr(offsets.view(n, -1).numpy(), base.numpy(), chars.numpy(), count, size)
    return count, labels.view(n, Q), scores.view(torch.float32).view(n, Q), rle


def coco_results(results: Sequence[Dict], image_ids: Sequence[int]) -> List[Dict]:
    """The COCO results list of ``results`` (from ``post_process_instance_segmentation(return_pycocotools_rle=True)`` or
    ``RgbdInstanceSegmenter(return_pycocotools_rle=True).result``), one entry per segment, ready for ``json.dump`` and
    ``COCO.loadRes``: ``{"image_id", "category_id", "segmentation": {"size", "counts": str}, "score"}``.  "category_id" is
    the model's ``label_id``; mapping it to a dataset's category ids is the caller's."""
    if len(results) != len(image_ids):
        raise ValueError(f"coco_results: {len(results)} results for {len(image_ids)} image ids")
    out = []
    for res, image_id in zip(results, image_ids):
        if len(res["segmentation"]) != len(res["segments_info"]):
            raise ValueError("coco_results: expected one pycocotools RLE per segment (return_pycocotools_rle=True)")
        for rle, info in zip(res["segmentation"], res["segments_info"]):
            out.append({"image_id": image_id, "category_id": info["label_id"],
                        "segmentation": {"size": list(rle["size"]), "counts": rle["counts"].decode("ascii")},
                        "score": info["score"]})
    return out


def post_process_instance_segmentation(outputs, threshold: float = 0.5, mask_threshold: float = 0.5,
                                       overlap_mask_area_threshold: float = 0.8,
                                       target_sizes: Optional[Sequence[Tuple[int, int]]] = None,
                                       return_coco_annotation: bool = False,
                                       return_binary_maps: bool = False,
                                       return_pycocotools_rle: bool = False) -> List[Dict]:
    """Drop-in for ``image_processor.post_process_instance_segmentation``.  ``mask_threshold`` and
    ``overlap_mask_area_threshold`` are accepted and unused, exactly as in HF's instance routine.
    ``return_coco_annotation=True`` returns HF's ``convert_segmentation_to_rle`` of the painted map as "segmentation": one
    run-length list per value present (ascending, so -1 first when there is background), encoded on the device.
    ``return_pycocotools_rle=True`` (not an HF option) returns, as "segmentation", one pycocotools RLE
    ``{"size": [h, w], "counts": bytes}`` per segment of ``segments_info``, equal to ``pycocotools.mask.encode`` of
    (painted map == id) and encoded on the device; ``coco_results`` turns such results into a COCO results list."""
    if return_coco_annotation and return_binary_maps:
        raise ValueError("return_coco_annotation and return_binary_maps can not be both set to True.")
    if return_pycocotools_rle and (return_coco_annotation or return_binary_maps):
        raise ValueError("return_pycocotools_rle can not be combined with return_coco_annotation or return_binary_maps.")
    cls = outputs.class_queries_logits
    msk = outputs.masks_queries_logits
    if not (cls.is_cuda and msk.is_cuda):
        raise RgbdB200Error("post_process_instance_segmentation: model outputs must be CUDA tensors (no CPU path)")
    cls = cls.detach().float().contiguous()
    msk = msk.detach().float().contiguous()
    B = cls.shape[0]
    sizes = [(384, 384)] * B if target_sizes is None else [tuple(int(v) for v in s) for s in target_sizes]
    if len(sizes) != B:
        raise ValueError("Make sure that you pass in as many target sizes as the batch dimension of the logits")
    results: List[Optional[Dict]] = [None] * B
    for size, idxs in _group_by_size(sizes).items():
        sel = torch.as_tensor(idxs, device=cls.device)
        whole = len(idxs) == B
        r = Fn.post_process_instances(cls if whole else cls[sel].contiguous(), msk if whole else msk[sel].contiguous(),
                                      threshold, size, want_segmentation=not return_binary_maps)
        if return_coco_annotation:
            count, labels, scores, rle = _download_with_rle(r, msk.shape[1])
        elif return_pycocotools_rle:
            count, labels, scores, rle = _download_with_pycocotools_rle(r, msk.shape[1], size)
        else:
            count = r.count.cpu().tolist()             # the one synchronisation of the batch
            labels, scores = r.labels.cpu(), r.scores.cpu()
        for k, i in enumerate(idxs):
            n = count[k]
            info = [{"id": j, "label_id": int(labels[k, j]), "was_fused": False, "score": round(float(scores[k, j]), 6)}
                    for j in range(n)]
            if return_coco_annotation or return_pycocotools_rle:
                seg = rle[k]
            elif return_binary_maps and n:
                seg = r.masks[k, :n].float()
            elif return_binary_maps:
                seg = torch.zeros(size, device=cls.device) - 1
            else:
                seg = r.segmentation[k].float()
            results[i] = {"segmentation": seg, "segments_info": info}
    return results


def postprocess_prediction_batch(prediction_batch, target_sizes, threshold: float = 0.0) -> List[Dict[str, torch.Tensor]]:
    """``Evaluator.postprocess_prediction_batch`` (model_essential_part.py:83-109): dictionaries with "masks" (bool),
    "labels", "scores" per image."""
    from types import SimpleNamespace
    out = post_process_instance_segmentation(
        SimpleNamespace(class_queries_logits=prediction_batch[0], masks_queries_logits=prediction_batch[1]),
        threshold=threshold, target_sizes=target_sizes, return_binary_maps=True)
    res = []
    for image_predictions, target_size in zip(out, target_sizes):
        if image_predictions["segments_info"]:
            res.append({"masks": image_predictions["segmentation"].to(dtype=torch.bool),
                        "labels": torch.tensor([x["label_id"] for x in image_predictions["segments_info"]]),
                        "scores": torch.tensor([x["score"] for x in image_predictions["segments_info"]])})
        else:
            res.append({"masks": torch.zeros([0, *target_size], dtype=torch.bool), "labels": torch.tensor([]),
                        "scores": torch.tensor([])})
    return res


class MaskAP:
    """Accumulates (prediction, target) pairs and computes segm mAP / mAP@50 / mAP@75 like the reference's
    ``MeanAveragePrecision(iou_type="segm")`` use (model_essential_part.py:111-170).  IoU matrices come from the device
    kernel; the matching and precision/recall integration are small host loops."""

    def __init__(self, thresholds: Sequence[float] = tuple(0.5 + 0.05 * i for i in range(10)), max_det: int = 100):
        self.thresholds = [float(t) for t in thresholds]
        self.max_det = max_det
        self.records: List[Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]] = []

    def update(self, preds: Sequence[Dict[str, torch.Tensor]], targets: Sequence[Dict[str, torch.Tensor]]) -> None:
        for p, t in zip(preds, targets):
            pm, gm = p["masks"], t["masks"]
            if pm.shape[0] and gm.shape[0]:
                iou = Fn.mask_iou(pm.cuda().contiguous(), gm.cuda().contiguous()).cpu().numpy().astype(np.float64)
            else:
                iou = np.zeros((pm.shape[0], gm.shape[0]))
            self.records.append((np.asarray(p["labels"].cpu(), dtype=np.int64), np.asarray(p["scores"].cpu(), dtype=np.float64),
                                 np.asarray(t["labels"].cpu(), dtype=np.int64), iou))

    def compute(self) -> Dict[str, float]:
        classes = sorted({int(c) for r in self.records for c in r[0]} | {int(c) for r in self.records for c in r[2]})
        rec_pts = np.linspace(0.0, 1.0, 101)
        ap = np.full((len(self.thresholds), len(classes)), -1.0)
        for ci, c in enumerate(classes):
            n_gt = sum(int((gl == c).sum()) for _, _, gl, _ in self.records)
            if n_gt == 0:
                continue
            for ti, thr in enumerate(self.thresholds):
                score_list, tp_list = [], []
                for pl, ps, gl, iou in self.records:
                    det = np.nonzero(pl == c)[0]
                    det = det[np.argsort(-ps[det], kind="mergesort")][:self.max_det]
                    gts = np.nonzero(gl == c)[0]
                    free = np.ones(len(gts), dtype=bool)
                    for d in det:
                        hit = -1
                        best = min(thr, 1 - 1e-10)
                        for gi, g in enumerate(gts):
                            if free[gi] and iou[d, g] >= best:
                                best, hit = iou[d, g], gi
                        if hit >= 0:
                            free[hit] = False
                        score_list.append(ps[d])
                        tp_list.append(hit >= 0)
                if not score_list:
                    ap[ti, ci] = 0.0
                    continue
                order = np.argsort(-np.asarray(score_list), kind="mergesort")
                tp = np.asarray(tp_list, dtype=np.float64)[order]
                ctp, cfp = np.cumsum(tp), np.cumsum(1.0 - tp)
                recall = ctp / n_gt
                precision = ctp / np.maximum(ctp + cfp, np.finfo(np.float64).eps)
                precision = np.maximum.accumulate(precision[::-1])[::-1]
                at = np.searchsorted(recall, rec_pts, side="left")
                ap[ti, ci] = float(np.where(at < len(precision), precision[np.minimum(at, len(precision) - 1)], 0.0).mean())

        def mean_valid(a: np.ndarray) -> float:
            v = a[a > -1]
            return float(v.mean()) if v.size else -1.0
        thr = [round(t, 2) for t in self.thresholds]
        return {"map": mean_valid(ap), "map_50": mean_valid(ap[thr.index(0.5)]) if 0.5 in thr else -1.0,
                "map_75": mean_valid(ap[thr.index(0.75)]) if 0.75 in thr else -1.0}
