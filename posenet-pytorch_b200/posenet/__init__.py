"""posenet -- drop-in for the reference package of the same name, running on B200 CUDA kernels.

Exports what the reference's ``posenet/__init__.py`` exports (constants, ``decode``, ``load_model``,
``MobileNetV1``, ``MOBILENET_V1_CHECKPOINTS``, the ``utils`` helpers) plus ``decode_multiple_poses``
at package level: the reference comments that import out (``__init__.py:2``) although its own
``benchmark.py:37`` calls ``posenet.decode_multiple_poses``; exporting both spellings lets
``benchmark.py`` and ``image_demo.py`` run unchanged (SURVEY.md F2).
"""
from posenet.constants import *  # noqa: F401,F403
from posenet import decode  # noqa: F401
from posenet import decode_multi  # noqa: F401
from posenet import sharding  # noqa: F401  (multi-GPU: shard images, gather pose records)
from posenet.decode_multi import decode_multiple_poses, decode_multiple_poses_batch  # noqa: F401
from posenet.models.model_factory import load_model, write_random_checkpoint  # noqa: F401
from posenet.models import MobileNetV1, MOBILENET_V1_CHECKPOINTS  # noqa: F401
from posenet.pipeline import BatchPipeline  # noqa: F401  (streaming batches: copies overlap the kernels)
from posenet.ingest import ImageStream  # noqa: F401  (threaded image-file decode into pinned batches)
from posenet.jpeg import imdecode_batch, imencode_batch  # noqa: F401  (baseline JPEG decode / encode on the GPU, bit-exact with cv2)
from posenet.png import imencode_png_batch  # noqa: F401  (PNG encode on the GPU, bit-exact with cv2)
from posenet.yuv import yuv_to_bgr_batch  # noqa: F401  (YUV video frames to BGR on the GPU, bit-exact with cv2.cvtColor)
from posenet.yuv import bgr_to_yuv_batch  # noqa: F401  (BGR frames to YUV on the GPU, bit-exact with cv2.cvtColor)
from posenet.track import OneEuro, PoseTracker  # noqa: F401  (pose track ids and keypoint smoothing across video frames, on the GPU)
from posenet.utils import *  # noqa: F401,F403
from posenet.utils import _process_input, process_input_gpu, resize_u8_gpu  # noqa: F401
from posenet.utils import draw_skel_and_kp_batch, draw_skeleton_batch  # noqa: F401  (overlays drawn on the GPU)
