from .automatic_mask_generator import PointCloudAutomaticMaskGenerator  # noqa: F401
from .pc_sam import PointCloudSAM, PointSAM, build_point_sam  # noqa: F401
