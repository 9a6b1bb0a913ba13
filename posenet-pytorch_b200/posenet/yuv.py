"""Video frames in YUV 4:2:0 / 4:2:2 converted to BGR on the GPU, bit-exact with ``cv2.cvtColor(frame, code)``
(``pn_yuv_to_bgr``).  Video sources deliver YUV: software decoders I420, hardware decoders and capture devices NV12, UVC webcams
YUY2.  Shipping those to the device and converting there moves 1.5 or 2 bytes a pixel over PCIe instead of BGR's 3.

    frames = posenet.yuv_to_bgr_batch(yuv, cv2.COLOR_YUV2BGR_NV12)    # uint8 [N, h*3/2, w] -> CUDA uint8 [N, h, w, 3]

``BatchPipeline(..., yuv=code)`` takes such batches too (``posenet.pipeline``).

The other way, for video sinks (ffmpeg ``rawvideo``, GStreamer ``appsrc``, v4l2loopback, hardware encoders): BGR frames converted
to YUV on the GPU, bit-exact with ``cv2.cvtColor(frame, code)`` for ``COLOR_BGR2YUV_*`` codes (``pn_bgr_to_yuv``), so that 1.5 or 2
bytes a pixel come back to the host instead of 3:

    yuv = posenet.bgr_to_yuv_batch(frames, cv2.COLOR_BGR2YUV_I420)     # uint8 [N, h, w, 3] -> CUDA uint8 [N, h*3/2, w]

``BatchPipeline(..., overlay=..., yuv_out=code)`` returns its drawn frames that way.  ``frame_shape`` and ``frame_size`` give
cv2's frame shape of a layout in both directions.
"""
import ctypes as C

import cv2
import numpy as np
import torch

from posenet import _native as nat

# cv2's codes (its aliases share the values) -> pn_yuv_layout.  The BGRA / RGB variants and COLOR_YUV2BGR (packed 4:4:4) are not
# converted.
_LAYOUTS = {
    cv2.COLOR_YUV2BGR_I420: nat.YUV_I420,        # = COLOR_YUV2BGR_IYUV
    cv2.COLOR_YUV2BGR_YV12: nat.YUV_YV12,
    cv2.COLOR_YUV2BGR_NV12: nat.YUV_NV12,
    cv2.COLOR_YUV2BGR_NV21: nat.YUV_NV21,
    cv2.COLOR_YUV2BGR_YUY2: nat.YUV_YUY2,        # = COLOR_YUV2BGR_YUYV, COLOR_YUV2BGR_YUNV
    cv2.COLOR_YUV2BGR_UYVY: nat.YUV_UYVY,        # = COLOR_YUV2BGR_Y422, COLOR_YUV2BGR_UYNV
    cv2.COLOR_YUV2BGR_YVYU: nat.YUV_YVYU,
}


# cv2's BGR -> YUV codes -> pn_yuv_layout: the five layouts cv2 writes (it has no BGR -> NV12 / NV21).  The RGB / BGRA sources
# and COLOR_BGR2YUV (packed 4:4:4) are not converted.
_OUT_LAYOUTS = {
    cv2.COLOR_BGR2YUV_I420: nat.YUV_I420,        # = COLOR_BGR2YUV_IYUV
    cv2.COLOR_BGR2YUV_YV12: nat.YUV_YV12,
    cv2.COLOR_BGR2YUV_YUY2: nat.YUV_YUY2,        # = COLOR_BGR2YUV_YUYV, COLOR_BGR2YUV_YUNV
    cv2.COLOR_BGR2YUV_UYVY: nat.YUV_UYVY,        # = COLOR_BGR2YUV_Y422, COLOR_BGR2YUV_UYNV
    cv2.COLOR_BGR2YUV_YVYU: nat.YUV_YVYU,
}


def _is_code(code):
    return isinstance(code, (int, np.integer)) and not isinstance(code, bool)


def layout_of(code):
    """The pn_yuv_layout of a ``cv2.COLOR_YUV2BGR_*`` code; ValueError for any other code."""
    if _is_code(code) and int(code) in _LAYOUTS:
        return _LAYOUTS[int(code)]
    raise ValueError("cv2 code %r: the device converts COLOR_YUV2BGR_ I420 / IYUV / YV12 / NV12 / NV21 / YUY2 / YUYV / YUNV / "
                     "UYVY / Y422 / UYNV / YVYU" % (code,))


def layout_of_output(code):
    """The pn_yuv_layout of a ``cv2.COLOR_BGR2YUV_*`` code of a 4:2:0 or 4:2:2 layout; ValueError for any other code."""
    if _is_code(code) and int(code) in _OUT_LAYOUTS:
        return _OUT_LAYOUTS[int(code)]
    raise ValueError("cv2 code %r: the device converts to COLOR_BGR2YUV_ I420 / IYUV / YV12 / YUY2 / YUYV / YUNV / UYVY / Y422 / "
                     "UYNV / YVYU" % (code,))


def frame_shape(layout, h, w):
    """cv2's shape of one h x w frame in ``layout`` (the input of COLOR_YUV2BGR_*, the output of COLOR_BGR2YUV_*) of one h x w frame: [h*3/2, w] for 4:2:0, [h, w, 2] for 4:2:2.  ValueError for the sizes cv2 rejects:
    odd widths, and odd heights of 4:2:0."""
    if h <= 0 or w <= 0 or w % 2 or (h % 2 and layout <= nat.YUV_NV21):
        raise ValueError("YUV frames of %d x %d: cv2 converts only even widths, and even heights of 4:2:0" % (h, w))
    return (h * 3 // 2, w) if layout <= nat.YUV_NV21 else (h, w, 2)


def frame_size(layout, shape):
    """(h, w) of a frame of cv2's input ``shape``; ValueError when the shape is not one."""
    shape = tuple(int(d) for d in shape)
    if layout <= nat.YUV_NV21:
        ok = len(shape) == 2 and shape[0] % 3 == 0
        h, w = (shape[0] * 2 // 3, shape[1]) if ok else (0, 0)
    else:
        ok = len(shape) == 3 and shape[2] == 2
        h, w = shape[:2] if ok else (0, 0)
    if not ok:
        raise ValueError("frame shape %s is not cv2's %s layout" % (shape, "[h*3/2, w]" if layout <= nat.YUV_NV21 else "[h, w, 2]"))
    frame_shape(layout, h, w)
    return h, w


def convert(src, n, h, w, layout, dst):
    """pn_yuv_to_bgr of n dense frames of the CUDA buffer ``src`` into the CUDA uint8 [>= n, h, w, 3] ``dst`` on the current
    stream."""
    nbytes = int(np.prod(frame_shape(layout, h, w)))
    nat.check(nat.load().pn_yuv_to_bgr(C.c_void_p(src.data_ptr()), n, h, w, nbytes, layout, C.c_void_p(dst.data_ptr()),
                                       h * w * 3, nat.stream_ptr()), "pn_yuv_to_bgr")


def yuv_to_bgr_batch(yuv, code):
    """uint8 ``[N, h*3/2, w]`` (4:2:0) or ``[N, h, w, 2]`` (4:2:2), host (numpy or torch) or CUDA -- cv2's per-frame input of
    ``code`` stacked -- to CUDA uint8 ``[N, h, w, 3]`` BGR, equal to ``np.stack([cv2.cvtColor(f, code) for f in yuv])``."""
    layout = layout_of(code)
    if not isinstance(yuv, torch.Tensor):
        yuv = torch.from_numpy(np.ascontiguousarray(yuv))
    if yuv.dtype != torch.uint8 or yuv.dim() < 1:
        raise ValueError("yuv_to_bgr_batch takes a uint8 batch, got %s %s" % (yuv.dtype, tuple(yuv.shape)))
    h, w = frame_size(layout, yuv.shape[1:])
    nat.require_device()
    src = yuv.to("cuda").contiguous()
    out = torch.empty((yuv.shape[0], h, w, 3), dtype=torch.uint8, device=src.device)
    if yuv.shape[0]:
        with torch.cuda.device(src.device):
            convert(src, yuv.shape[0], h, w, layout, out)
    return out


def convert_out(src, n, h, w, layout, dst, src_stride=None):
    """pn_bgr_to_yuv of n BGR frames of the CUDA buffer ``src`` (``src_stride`` bytes apart, default h*w*3) into n dense frames
    of the CUDA uint8 buffer ``dst`` on the current stream."""
    nbytes = int(np.prod(frame_shape(layout, h, w)))
    nat.check(nat.load().pn_bgr_to_yuv(C.c_void_p(src.data_ptr()), n, h, w, src_stride or h * w * 3, layout,
                                       C.c_void_p(dst.data_ptr()), nbytes, nat.stream_ptr()), "pn_bgr_to_yuv")


def bgr_to_yuv_batch(frames, code):
    """uint8 ``[N, h, w, 3]`` BGR, host (numpy or torch) or CUDA, to CUDA uint8 ``[N, h*3/2, w]`` (4:2:0) or ``[N, h, w, 2]``
    (4:2:2), equal to ``np.stack([cv2.cvtColor(f, code) for f in frames])`` for a ``cv2.COLOR_BGR2YUV_*`` code."""
    layout = layout_of_output(code)
    if not isinstance(frames, torch.Tensor):
        frames = torch.from_numpy(np.ascontiguousarray(frames))
    if frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
        raise ValueError("bgr_to_yuv_batch takes uint8 [N, h, w, 3], got %s %s" % (frames.dtype, tuple(frames.shape)))
    h, w = int(frames.shape[1]), int(frames.shape[2])
    shape = frame_shape(layout, h, w)
    nat.require_device()
    src = frames.to("cuda").contiguous()
    out = torch.empty((frames.shape[0],) + shape, dtype=torch.uint8, device=src.device)
    if frames.shape[0]:
        with torch.cuda.device(src.device):
            convert_out(src, frames.shape[0], h, w, layout, out)
    return out
