"""Image ingest + overlay helpers with the reference's names (posenet/utils.py).

``_process_input`` keeps the reference's contract (utils.py:13-26): BGR uint8 HWC in, ``(float32
[1,3,H,W] numpy, source image, scale)`` out -- but the resize / colour swap / normalisation run in
the fused CUDA kernel ``pn_preprocess_u8`` (bit-exact with cv2's INTER_LINEAR).  For device-resident
pipelines use ``process_input_gpu``, which returns the CUDA tensor without the copy back.
The drawing helpers with the reference's names are host-side (cv2); ``draw_skel_and_kp_batch`` / ``draw_skeleton_batch`` draw
the same pixels on device-resident frames with the CUDA kernel ``pn_draw_poses``.
"""
import ctypes as C

import cv2
import numpy as np
import torch

import posenet.constants
from posenet import _native as nat


def valid_resolution(width, height, output_stride=16):
    snap = lambda v: (int(v) // output_stride) * output_stride + 1
    return snap(width), snap(height)


def process_input_gpu(source_img, scale_factor=1.0, output_stride=16, out=None):
    """uint8 BGR image(s) -> normalised RGB fp32 NCHW CUDA tensor.

    ``source_img``: numpy or torch uint8, [h,w,3] or [N,h,w,3] (host or device).  Returns
    ``(input [N,3,th,tw] float32 cuda, scale float64[2])``."""
    nat.require_device()
    img = source_img if torch.is_tensor(source_img) else torch.from_numpy(np.ascontiguousarray(source_img))
    if img.dim() == 3:
        img = img.unsqueeze(0)
    assert img.dim() == 4 and img.shape[3] == 3 and img.dtype == torch.uint8, "expected uint8 [h,w,3] / [N,h,w,3]"
    n, h, w = img.shape[0], img.shape[1], img.shape[2]
    tw, th = valid_resolution(w * scale_factor, h * scale_factor, output_stride=output_stride)
    scale = np.array([h / th, w / tw])
    dev = img.device if img.is_cuda else torch.device("cuda", torch.cuda.current_device())
    img = img.to(dev).contiguous()
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((n, 3, th, tw), dtype=torch.float32, device=dev)
        nat.check(nat.load().pn_preprocess_u8(C.c_void_p(img.data_ptr()), n, h, w, th, tw, C.c_void_p(out.data_ptr()),
                                              nat.stream_ptr()), "pn_preprocess_u8")
    return out, scale


def resize_u8_gpu(source_img, scale_factor=1.0, output_stride=16, out=None):
    """The resize stage of ``_process_input`` alone (utils.py:21 of the reference, cv2.resize INTER_LINEAR, bit-exact):
    uint8 BGR [h,w,3] / [N,h,w,3] -> uint8 BGR [N,th,tw,3] on the GPU, the input of ``MobileNetV1.forward_u8`` (which
    normalises inside the stem).  Returns ``(frames uint8 cuda, scale float64[2])``."""
    nat.require_device()
    img = source_img if torch.is_tensor(source_img) else torch.from_numpy(np.ascontiguousarray(source_img))
    if img.dim() == 3:
        img = img.unsqueeze(0)
    assert img.dim() == 4 and img.shape[3] == 3 and img.dtype == torch.uint8, "expected uint8 [h,w,3] / [N,h,w,3]"
    n, h, w = img.shape[0], img.shape[1], img.shape[2]
    tw, th = valid_resolution(w * scale_factor, h * scale_factor, output_stride=output_stride)
    scale = np.array([h / th, w / tw])
    dev = img.device if img.is_cuda else torch.device("cuda", torch.cuda.current_device())
    img = img.to(dev).contiguous()
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((n, th, tw, 3), dtype=torch.uint8, device=dev)
        assert tuple(out.shape) == (n, th, tw, 3) and out.dtype == torch.uint8 and out.is_contiguous()
        nat.check(nat.load().pn_resize_u8(C.c_void_p(img.data_ptr()), n, h, w, th, tw, C.c_void_p(out.data_ptr()), nat.stream_ptr()),
                  "pn_resize_u8")
    return out, scale


def _process_input(source_img, scale_factor=1.0, output_stride=16):
    x, scale = process_input_gpu(source_img, scale_factor, output_stride)
    return x.cpu().numpy(), source_img, scale


def read_cap(cap, scale_factor=1.0, output_stride=16):
    ok, frame = cap.read()
    if not ok:
        raise IOError("webcam failure")
    return _process_input(frame, scale_factor, output_stride)


def read_imgfile(path, scale_factor=1.0, output_stride=16):
    return _process_input(cv2.imread(path), scale_factor, output_stride)


# ---------------------------------------------------------------------------- overlays (host)
def _keypoints_above(keypoint_scores, keypoint_coords, threshold):
    return [cv2.KeyPoint(float(c[1]), float(c[0]), 10. * float(s))
            for s, c in zip(keypoint_scores, keypoint_coords) if s >= threshold]


def get_adjacent_keypoints(keypoint_scores, keypoint_coords, min_confidence=0.1):
    segments = []
    for a, b in posenet.constants.CONNECTED_PART_INDICES:
        if keypoint_scores[a] >= min_confidence and keypoint_scores[b] >= min_confidence:
            segments.append(np.array([keypoint_coords[a][::-1], keypoint_coords[b][::-1]]).astype(np.int32))
    return segments


def draw_keypoints(img, instance_scores, keypoint_scores, keypoint_coords,
                   min_pose_confidence=0.5, min_part_confidence=0.5):
    pts = []
    for i, score in enumerate(instance_scores):
        if score >= min_pose_confidence:
            pts += _keypoints_above(keypoint_scores[i], keypoint_coords[i], min_part_confidence)
    return cv2.drawKeypoints(img, pts, outImage=np.array([]))


def draw_skeleton(img, instance_scores, keypoint_scores, keypoint_coords,
                  min_pose_confidence=0.5, min_part_confidence=0.5):
    segments = []
    for i, score in enumerate(instance_scores):
        if score >= min_pose_confidence:
            segments += get_adjacent_keypoints(keypoint_scores[i], keypoint_coords[i], min_part_confidence)
    return cv2.polylines(img, segments, isClosed=False, color=(255, 255, 0))


def draw_skel_and_kp(img, instance_scores, keypoint_scores, keypoint_coords,
                     min_pose_score=0.5, min_part_score=0.5):
    out_img, segments, pts = img, [], []
    for i, score in enumerate(instance_scores):
        if score < min_pose_score:
            continue
        segments += get_adjacent_keypoints(keypoint_scores[i], keypoint_coords[i], min_part_score)
        pts += _keypoints_above(keypoint_scores[i], keypoint_coords[i], min_part_score)
    if pts:
        out_img = cv2.drawKeypoints(out_img, pts, outImage=np.array([]), color=(255, 255, 0),
                                    flags=cv2.DRAW_MATCHES_FLAGS_DRAW_RICH_KEYPOINTS)
    return cv2.polylines(out_img, segments, isClosed=False, color=(255, 255, 0))


# ---------------------------------------------------------------------------- overlays (device)
def _draw_batch(frames, pose_scores, keypoint_scores, keypoint_coords, min_pose, min_part, what):
    nat.require_device()
    assert torch.is_tensor(frames) and frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3, \
        "expected uint8 CUDA frames [N,h,w,3]"
    n, h, w = frames.shape[:3]
    st = frames.stride()
    assert st[3] == 1 and st[2] == 3 and st[1] == 3 * w and st[0] >= 3 * h * w, \
        "each frame must be stored densely (rows of w*3 bytes); frames may be further apart"
    dev = frames.device
    ps, ks, kc = (torch.as_tensor(t, dtype=torch.float64, device=dev).contiguous()
                  for t in (pose_scores, keypoint_scores, keypoint_coords))
    P = ps.shape[-1]
    assert tuple(ps.shape) == (n, P) and tuple(ks.shape) == (n, P, 17) and tuple(kc.shape) == (n, P, 17, 2), \
        "expected records [N,P], [N,P,17], [N,P,17,2] for %d frames" % n
    with torch.cuda.device(dev):
        nat.check(nat.load().pn_draw_poses(C.c_void_p(frames.data_ptr()), n, h, w, st[0], None, C.c_void_p(ps.data_ptr()),
                                           C.c_void_p(ks.data_ptr()), C.c_void_p(kc.data_ptr()), P, float(min_pose),
                                           float(min_part), what, nat.stream_ptr()), "pn_draw_poses")
    return frames


def draw_skel_and_kp_batch(frames, pose_scores, keypoint_scores, keypoint_coords, min_pose_score=0.5, min_part_score=0.5):
    """``draw_skel_and_kp`` of every frame of a batch, on the GPU and bit-exact with it.  ``frames``: uint8 CUDA [N,h,w,3]
    (BGR), drawn IN PLACE and returned; the records are ``decode_multiple_poses_batch``'s (float64 CUDA [N,P], [N,P,17],
    [N,P,17,2], coordinates in the frames' pixels)."""
    return _draw_batch(frames, pose_scores, keypoint_scores, keypoint_coords, min_pose_score, min_part_score,
                       nat.DRAW_KEYPOINTS | nat.DRAW_SKELETON)


def draw_skeleton_batch(frames, pose_scores, keypoint_scores, keypoint_coords, min_pose_confidence=0.5, min_part_confidence=0.5):
    """``draw_skeleton`` of every frame of a batch on the GPU (in place, bit-exact); arguments as ``draw_skel_and_kp_batch``."""
    return _draw_batch(frames, pose_scores, keypoint_scores, keypoint_coords, min_pose_confidence, min_part_confidence,
                       nat.DRAW_SKELETON)
