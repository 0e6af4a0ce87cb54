"""numpy restatement of automatic mask generation (pc_sam.model.PointCloudAutomaticMaskGenerator): per-candidate stats,
the filter, the stable score order, exact integer IoU and greedy NMS, given per-candidate logits and IoU predictions.

Every ratio is an fp32 division of exact integer counts, every comparison is against the fp32 threshold, as in the
kernels, so the kernels are compared against this exactly."""
from __future__ import annotations

import numpy as np

F32 = np.float32


def pack_bits(masks: np.ndarray) -> np.ndarray:
    """bool [R, N] -> uint32 [R, ceil(N / 32)], bit j of word w = point 32 w + j, tail bits 0."""
    masks = np.asarray(masks, dtype=bool)
    R, N = masks.shape
    W = (N + 31) // 32
    b = np.packbits(masks, axis=1, bitorder="little")
    out = np.zeros((R, 4 * W), dtype=np.uint8)
    out[:, : b.shape[1]] = b
    return out.view("<u4").reshape(R, W)


def _ratio(num, den) -> np.ndarray:
    num, den = np.asarray(num), np.asarray(den)
    return np.where(den > 0, num.astype(F32) / np.maximum(den, 1).astype(F32), F32(0)).astype(F32)


def mask_stats(logits, iou_preds, mask_threshold=0.0, stability_score_offset=1.0, pred_iou_thresh=0.88,
               stability_score_thresh=0.95):
    """logits fp32 [R, N], iou_preds fp32 [R] -> (masks bool [R, N], area int64 [R], stability fp32 [R], keep bool [R])."""
    x = np.asarray(logits, dtype=F32)
    iou = np.asarray(iou_preds, dtype=F32)
    t, off = F32(mask_threshold), F32(stability_score_offset)
    masks = x > t
    area = masks.sum(axis=1)
    stability = _ratio((x > F32(t + off)).sum(axis=1), (x > F32(t - off)).sum(axis=1))
    keep = (iou > F32(pred_iou_thresh)) & (stability >= F32(stability_score_thresh)) & (area > 0)
    return masks, area, stability, keep


def pairwise_iou(masks_a, masks_b):
    """(inter int64 [Ka, Kb], iou fp32 [Ka, Kb]).  The fp32 product of 0/1 matrices is exact while N < 2^24."""
    a = np.asarray(masks_a, dtype=F32)
    b = np.asarray(masks_b, dtype=F32)
    inter = (a @ b.T).astype(np.int64)
    union = a.sum(axis=1).astype(np.int64)[:, None] + b.sum(axis=1).astype(np.int64)[None, :] - inter
    return inter, _ratio(inter, union)


def score_order(iou_preds, keep) -> np.ndarray:
    """Indices of the kept candidates by score descending, ties to the lower index (torch.sort(stable=True, descending=True))."""
    cand = np.nonzero(np.asarray(keep))[0]
    return cand[np.argsort(-np.asarray(iou_preds, dtype=F32)[cand], kind="stable")]


def greedy_nms(iou: np.ndarray, nms_thresh: float) -> np.ndarray:
    """iou [M, M] between candidates already in score order -> positions kept: a candidate is kept unless an earlier KEPT
    candidate has IoU > nms_thresh with it."""
    M = iou.shape[0]
    suppressed = np.zeros(M, dtype=bool)
    kept = []
    for i in range(M):
        if suppressed[i]:
            continue
        kept.append(i)
        suppressed |= iou[i] > F32(nms_thresh)
    return np.asarray(kept, dtype=np.int64)


def generate(logits, iou_preds, points_per_batch=None, pred_iou_thresh=0.88, stability_score_thresh=0.95,
             stability_score_offset=1.0, mask_threshold=0.0, nms_thresh=0.7) -> dict:
    """logits [K, N] and iou_preds [K] of candidates c = 3 prompt + mask_index -> the generator's output, in kept order
    (numpy); `candidates` = kept candidate indices, `passed` = how many passed the filter.  points_per_batch is accepted
    (and ignored) so that the generator's parameter dict can be passed as is."""
    masks, area, stability, keep = mask_stats(logits, iou_preds, mask_threshold, stability_score_offset, pred_iou_thresh,
                                              stability_score_thresh)
    order = score_order(iou_preds, keep)
    _, iou = pairwise_iou(masks[order], masks[order])
    cand = order[greedy_nms(iou, nms_thresh)]
    return dict(candidates=cand, passed=len(order), masks=masks[cand], iou_preds=np.asarray(iou_preds, dtype=F32)[cand],
                stability_scores=stability[cand], areas=area[cand], prompt_index=cand // 3, mask_index=cand % 3)
