"""B200-native drop-in for the conv-stack hot path of tejasd-24/fpga-cnn-object-detection-accelerator.

128x128 u8 image -> Conv3x3 1->16->32->64 (+ >>shift, ReLU/saturate, 2x2 max-pool each) -> 64x16x16 u8
features, plus the classifier / CAM tail, behind the reference's own call surface.  Python here is only
the host-side mirror of the reference's engine objects; the work happens in libcnnacc.so (csrc/).
"""
from . import _lib
from ._lib import build, load
from .accelerator import (ARMEngine, B200Engine, CNNAccelerator, Classifier, MultiAccelerator, NAMES, alloc_host, bbox_vec,
                          classify_vec, dump_features, grid_rects, grid_regions, load_arm_cnn_lib, load_features, load_image_any,
                          pyramid_levels, pyramid_windows, region_boxes_to_frame, register_host, train_linear_classifier)

__all__ = ["ARMEngine", "B200Engine", "CNNAccelerator", "Classifier", "MultiAccelerator", "dump_features", "load_features", "NAMES", "alloc_host", "register_host", "load_image_any", "train_linear_classifier", "bbox_vec", "classify_vec",
           "grid_regions", "grid_rects", "pyramid_levels", "pyramid_windows", "region_boxes_to_frame",
           "load_arm_cnn_lib", "build", "load", "_lib"]
