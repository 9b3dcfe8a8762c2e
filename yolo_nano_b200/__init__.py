"""yolo_nano_b200 — B200-native YOLO-Nano-1.0x detection forward path.

Drop-in for `models/yolo_nano.py` of yjh0410/YOLO-Nano: `YOLONano` keeps the
reference constructor, `forward(x) -> (bboxes, scores, cls_inds)`, `set_grid`,
`fuse_conv_bn` behaviour and `state_dict` layout; the computation runs in
hand-written sm_100a CUDA behind the C ABI of `include/yolonano_b200.h`.
"""
from .topology import conv_table, num_anchor_boxes  # noqa: F401
from .fuse_conv_bn import fuse_conv_bn  # noqa: F401
from .yolo_nano import YOLONano, Conv, ShuffleNetV2, ShuffleV2Block  # noqa: F401
from .engine import Engine, EngineError  # noqa: F401
from .tta import TestTimeAugmentation, resize_bilinear  # noqa: F401
from .ema import ModelEMA  # noqa: F401
from . import evalfmt  # noqa: F401
from .voc_eval import VOCDetections  # noqa: F401
from .coco_eval import COCODetections  # noqa: F401

# anchors of the reference (data/config.py:11-17): constructor inputs, data not code
MULTI_ANCHOR_SIZE = [[30.65, 39.12], [50.3, 102.62], [94.98, 64.55],
                     [93.5, 177.51], [165.25, 113.85], [161.83, 240.95],
                     [304.64, 150.34], [251.28, 306.53], [369.38, 261.55]]
MULTI_ANCHOR_SIZE_COCO = [[11.89, 14.24], [30.14, 35.62], [45.99, 87.04],
                          [92.23, 44.43], [130.78, 99.73], [78.99, 170.81],
                          [290.39, 123.89], [165.27, 233.33], [332.57, 279.8]]
