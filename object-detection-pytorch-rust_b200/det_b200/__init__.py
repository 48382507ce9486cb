"""det_b200 -- B200-native (sm_100a) post-backbone detection hot path.

Drop-in for the reference's Python callables on that path (SURVEY.md section 8b); every op forwards to
hand-written CUDA kernels in ``libdet_b200.so`` through the C ABI of ``include/det_b200.h``.
There is no CPU path and no PyTorch fallback.
"""
from . import _native
from .structures import (Boxes, Instances, pairwise_iou, pairwise_ioa, pairwise_intersection,
                         matched_boxlist_iou)
from .box_regression import Box2BoxTransform
from .anchors import AnchorGenerator, generate_cell_anchors
from .nms import batched_nms, nms, nms_images, DenseDetectWorkspace
from .yolo import YoloGridHead, DenseAnchorHead, YoloGridTrainer, YoloHostPipeline
from .matcher import Matcher, subsample_labels_
from .proposals import find_top_rpn_proposals, rpn_proposals_batched, add_ground_truth_to_proposals
from .rpn import RegionProposalNetwork, Assignment, _dense_box_regression_loss
from .roi import ROIHeads, subsample_labels
from .roi_pool import ROIAlign, ROIPooler, assign_boxes_to_levels, convert_boxes_to_pooler_format
from .fast_rcnn import FastRCNNOutputs, fast_rcnn_inference
from . import dist

__all__ = [
    "Boxes", "Instances", "pairwise_iou", "pairwise_ioa", "pairwise_intersection", "matched_boxlist_iou",
    "Box2BoxTransform", "AnchorGenerator", "generate_cell_anchors", "batched_nms", "nms", "nms_images",
    "YoloGridHead", "DenseAnchorHead", "YoloGridTrainer", "YoloHostPipeline", "DenseDetectWorkspace", "Matcher", "subsample_labels_", "find_top_rpn_proposals",
    "rpn_proposals_batched", "add_ground_truth_to_proposals", "RegionProposalNetwork", "Assignment",
    "_dense_box_regression_loss", "ROIHeads", "subsample_labels", "ROIAlign", "ROIPooler", "assign_boxes_to_levels",
    "convert_boxes_to_pooler_format", "FastRCNNOutputs", "fast_rcnn_inference", "dist",
]
