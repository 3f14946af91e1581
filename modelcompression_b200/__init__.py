"""modelcompression_b200 — B200 (sm_100a) hot path of AnishDelft/ModelCompression behind the reference's own
Python API: the pruned YOLOv2-VOC forward, the pruning-mask computation, and region decode + NMS.

    reference                                      here
    src/nets.py            Darknet, parse_cfg ...  modelcompression_b200.nets
    src/nets2_utils.py     get_region_boxes, nms   modelcompression_b200.nets2_utils
    src/pruning/weightPruning/{layers,methods,utils}.py   modelcompression_b200.pruning.weightPruning.*

All arithmetic on the path runs in hand-written CUDA kernels (libmcb200.so, C-ABI in include/mcb200.h) loaded with
ctypes; PyTorch provides device memory, streams and torch.distributed.  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from .cfg import write_yolov2_voc_cfg, yolov2_voc_cfg_text  # noqa: F401
from .nets import Darknet, EmptyModule, Reorg, RegionLoss, getYOLOv2, parse_cfg  # noqa: F401
from .nets2_utils import bbox_iou, bbox_ious, detect_batch, do_detect, get_region_boxes, nms  # noqa: F401
from .optim import MaskedSGD  # noqa: F401
from .pruning.weightPruning.layers import MaskedConv2d, MaskedLinear  # noqa: F401
from .pruning.weightPruning.methods import filter_prune, prune_one_filter, quick_filter_prune, weight_prune  # noqa: F401
from .pruning.weightPruning.utils import are_masks_consistent, prune_rate, to_var  # noqa: F401

__version__ = "0.1.0"
