"""manuscript_b200 -- B200-native (sm_100a) detector->recognizer hot path of manuscript-ocr.

Host side of include/manuscript_b200.h: Python mirrors of the reference's function-level seam
(`decode_quads_from_maps`, `locality_aware_nms`, `expand_boxes`, the EAST box filters, the
Pipeline crop loop and the TRBA `ResizeAndPadA` batch assembly) that call the hand-written CUDA
kernels through the C ABI.  There is no CPU fallback: importing works anywhere, every compute call
needs libmanuscript_b200.so and a B200.
"""
from ._cabi import (  # noqa: F401
    CABIError,
    Context,
    EastParams,
    batch_dtype_code,
    library_path,
    load_library,
)
from .ops import (  # noqa: F401
    crop_resize_pad,
    decode_quads_from_maps,
    decode_rbox_from_maps,
    east_postprocess,
    expand_boxes,
    locality_aware_nms,
    polygon_iou,
    quad_crop_resize_pad,
    should_merge,
    standard_nms,
    warp_quad,
    word_reading_order,
    word_rects,
)
from .batch import PageBatch, PageBatchResult, shard_pages  # noqa: F401
from .east import EAST  # noqa: F401
from .imaging import read_image, visualize_page  # noqa: F401
from .pipeline import Pipeline  # noqa: F401
from .reading_order import (  # noqa: F401
    resolve_intersections,
    sort_boxes_reading_order,
    sort_boxes_reading_order_with_resolutions,
)
from .tps import TPSGrid, build_tps_constants  # noqa: F401
from .trba import TRBA  # noqa: F401
from .types import Block, Page, Word  # noqa: F401

__version__ = "0.1.0"
