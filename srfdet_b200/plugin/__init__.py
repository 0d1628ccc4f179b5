"""Drop-in modules registered under the reference's `mmdet3d_plugin` names."""
from .registry import (DETECTORS, HEADS, MIDDLE_ENCODERS, NORM_LAYERS, ROI_EXTRACTORS, VOXEL_ENCODERS,  # noqa: F401
                       BACKBONES, NECKS, build_backbone, build_neck, build_head, build_middle_encoder, build_norm_layer, build_roi_extractor,
                       build_voxel_encoder, get_precision, load_config, set_precision)
from .ops import DynamicScatter, Voxelization  # noqa: F401
from .voxel_encoder import DynamicVFECustom, DynamicVFELayer, HardSimpleVFE, NaiveSyncBatchNorm1dCustom  # noqa: F401
from .sparse_encoder import SparseBasicBlock, SparseEncoderCustom, make_sparse_convmodule  # noqa: F401
from .roi import (SingleRoIExtractor, bbox2roi, boxes3d_to_corners3d, img_feats_sampling_bboxes_roi,  # noqa: F401
                  points_feats_sampling_bboxes_roi)
from .head import DynamicConv, SingleSRFDetHead, SingleSRFDetHeadLiDAR  # noqa: F401
from .pillar import PFNLayer, PillarFeatureNetCustom, PointPillarsScatter  # noqa: F401
from .bev_backbone import FPN, SECONDCustom  # noqa: F401
from .srfdet_head import SRFDetHead  # noqa: F401
from .nms import box3d_multiclass_nms, boxes_iou_bev, nms_bev, nms_normal_bev, xywhr2xyxyr  # noqa: F401
from .detector import SRFDetPointPath  # noqa: F401
