"""Automatic mask generation ("segment everything") for Point-SAM, after SAM's SamAutomaticMaskGenerator.

The reference ships no automatic mask generator; the semantics here are this project's (DESIGN.md, "Automatic mask
generation"): an FPS sample of the cloud as single positive point prompts, three masks per prompt, filtering by predicted
IoU and stability score, then greedy mask NMS.  All of it runs in the sm_100a kernels behind ``psam_b200``."""
from __future__ import annotations

import math
from typing import Dict

import torch

from psam_b200 import engine


class PointCloudAutomaticMaskGenerator:
    """Masks for the whole cloud without clicks.  Defaults are SAM's: a candidate is kept if iou_pred > pred_iou_thresh,
    stability >= stability_score_thresh and its area is not 0; kept candidates are suppressed by an earlier (higher
    iou_pred) kept candidate with mask IoU > nms_thresh."""

    def __init__(self, model, points_per_cloud: int = 512, points_per_batch: int = 64, pred_iou_thresh: float = 0.88,
                 stability_score_thresh: float = 0.95, stability_score_offset: float = 1.0, mask_threshold: float = 0.0,
                 nms_thresh: float = 0.7):
        for name, v in (("points_per_cloud", points_per_cloud), ("points_per_batch", points_per_batch)):
            if isinstance(v, bool) or not isinstance(v, int) or v <= 0:
                raise ValueError(f"{name} must be a positive integer, got {v!r}")
        if 3 * points_per_cloud > engine.AMG_MAX_CANDIDATES:
            raise ValueError(f"points_per_cloud must be <= {engine.AMG_MAX_CANDIDATES // 3} (3 candidate masks per prompt)")
        floats = dict(pred_iou_thresh=pred_iou_thresh, stability_score_thresh=stability_score_thresh,
                      stability_score_offset=stability_score_offset, mask_threshold=mask_threshold, nms_thresh=nms_thresh)
        for name, v in floats.items():
            if isinstance(v, bool) or not isinstance(v, (int, float)) or not math.isfinite(v):
                raise ValueError(f"{name} must be a finite number, got {v!r}")
        if stability_score_offset < 0:
            raise ValueError("stability_score_offset must be >= 0")
        self.model = model
        self.points_per_cloud = points_per_cloud
        self.params = dict(points_per_batch=points_per_batch, **{k: float(v) for k, v in floats.items()})

    def generate(self, coords: torch.Tensor, features: torch.Tensor) -> Dict[str, torch.Tensor]:
        """coords [1, N, 3], features [1, N, 3] (the set_pointcloud conventions) -> device tensors in kept order:
        masks bool [k, N], iou_preds [k], stability_scores [k], areas int64 [k], prompt_coords [k, 3],
        prompt_index [k] (into the FPS prompt sample), mask_index [k] (multimask output 0..2).  k = 0 is a valid result."""
        if not (coords.is_cuda and features.is_cuda):
            raise RuntimeError("psam_b200: coords and features must be CUDA tensors (this path has no CPU implementation)")
        if self.model.training:
            raise ValueError("automatic mask generation needs the model in eval mode (call model.eval())")
        if coords.dim() != 3 or coords.shape[0] != 1 or coords.shape[2] != 3 or features.shape[:2] != coords.shape[:2]:
            raise ValueError(f"one cloud expected: coords [1, N, 3] and features [1, N, C], got {tuple(coords.shape)} and "
                             f"{tuple(features.shape)}")
        if self.points_per_cloud > coords.shape[1]:
            raise ValueError(f"points_per_cloud = {self.points_per_cloud} exceeds the cloud's {coords.shape[1]} points")
        with torch.no_grad():
            self.model.set_pointcloud(coords, features)
            cloud = self.model._cloud
            prompts = engine.run_amg_prompts(cloud, self.points_per_cloud)
            return engine.run_automatic_masks(self.model, cloud, prompts, self.params)
