"""ctypes binding of libposenet_b200.so (declared in include/posenet_b200.h).

There is deliberately no fallback: if the library is missing or a call fails, the caller gets
an exception.  The library is looked up in-tree (``posenet-pytorch_b200/lib``); set
``POSENET_B200_LIB`` to override, or ``POSENET_B200_AUTOBUILD=1`` to compile it on first use.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_PKG_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("POSENET_B200_LIB", os.path.join(_PKG_ROOT, "lib", "libposenet_b200.so"))

PN_OK = 0
PN_F32, PN_BF16 = 0, 1
NUM_PARTS, NUM_EDGES, HEAD_CHANNELS, HEAD_ROWS = 17, 16, 115, 128
ABI_VERSION = 5
PLAN_UNFUSED = 1
DRAW_KEYPOINTS, DRAW_SKELETON = 1, 2
JPEG_SUPPORTED, JPEG_HOST = 0, 1
JPEG_WHY = {name: i for i, name in enumerate((
    "none", "not_jpeg", "truncated", "progressive", "arithmetic", "lossless", "precision", "multi_scan", "components", "rgb",
    "no_dht", "exif_orientation", "sampling", "bad_table", "unknown"))}
JPEG_OK, JPEG_SKIPPED = 0, 1
YUV_I420, YUV_YV12, YUV_NV12, YUV_NV21, YUV_YUY2, YUV_UYVY, YUV_YVYU = range(7)


class NativeError(RuntimeError):
    pass


class Map(C.Structure):
    """pn_map: strided f32 [n_img, channels, h, w] view (strides in elements)."""
    _fields_ = [("ptr", C.c_void_p), ("s_img", C.c_int64), ("s_ch", C.c_int64), ("s_y", C.c_int64), ("s_x", C.c_int64)]


class DecodeParams(C.Structure):
    _fields_ = [("output_stride", C.c_int), ("max_pose_detections", C.c_int),
                ("squared_nms_radius", C.c_double), ("min_pose_score", C.c_double)]


class Layer(C.Structure):
    _fields_ = [("cin", C.c_int), ("cout", C.c_int), ("stride", C.c_int), ("dilation", C.c_int),
                ("dw_w", C.c_void_p), ("dw_b", C.c_void_p), ("pw_w", C.c_void_p), ("pw_b", C.c_void_p)]


class NetDesc(C.Structure):
    _fields_ = [("dtype", C.c_int), ("n", C.c_int), ("h", C.c_int), ("w", C.c_int), ("input_u8", C.c_int),
                ("num_layers", C.c_int), ("layers", Layer * 16), ("head_w", C.c_void_p), ("head_b", C.c_void_p),
                ("flags", C.c_int)]


class JpegHuff(C.Structure):
    _fields_ = [("lookup", C.c_uint16 * 256), ("maxcode", C.c_int32 * 18), ("valoffset", C.c_int32 * 18), ("huffval", C.c_uint8 * 256)]


class JpegComp(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("h", "v", "hr", "vr", "dc", "ac", "bw", "bh", "dw", "dh")]


class JpegDesc(C.Structure):
    """pn_jpeg_desc: one file's headers as pn_jpeg_parse leaves them (file_offset is the caller's; orientation: the EXIF
    orientation the decode applies, 0 for none, 2..8 from pn_jpeg_parse_oriented)."""
    _fields_ = [(n, C.c_int32) for n in ("kind", "why", "height", "width", "ncomp", "mcus_x", "mcus_y", "blocks_per_mcu",
                                         "restart_interval", "n_segments")] + \
               [("file_offset", C.c_int64), ("file_bytes", C.c_int64), ("scan_offset", C.c_int64), ("comp", JpegComp * 3),
                ("mcu_comp", C.c_uint8 * 10), ("mcu_bx", C.c_uint8 * 10), ("mcu_by", C.c_uint8 * 10), ("orientation", C.c_uint8),
                ("pad", C.c_uint8 * 1),
                ("quant", (C.c_int16 * 64) * 3), ("huff", JpegHuff * 4)]


_SIGNATURES = {
    "pn_abi_version": (C.c_int, []),
    "pn_last_error_string": (C.c_char_p, []),
    "pn_device_check": (C.c_int, []),
    "pn_preprocess_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pn_resize_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pn_stem_conv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_int, C.c_void_p]),
    "pn_stem_conv_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int, C.c_void_p]),
    "pn_dwconv3x3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "pn_pwconv_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p]),
    "pn_sepconv_block": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "pn_sepconv_describe": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]),
    "pn_heads_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "pn_candidates": (C.c_int, [C.POINTER(Map), C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_void_p,
                                C.c_void_p]),
    "pn_decode_greedy": (C.c_int, [C.POINTER(Map), C.POINTER(Map), C.POINTER(Map), C.POINTER(Map), C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(DecodeParams), C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pn_traverse_to_targ_keypoint": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.c_int, C.POINTER(Map), C.POINTER(Map),
                                               C.POINTER(Map), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pn_decode_pose": (C.c_int, [C.c_double, C.c_int, C.POINTER(C.c_double), C.POINTER(Map), C.POINTER(Map), C.POINTER(Map),
                                 C.POINTER(Map), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pn_scale_keypoint_coords": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_void_p]),
    "pn_draw_poses": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int, C.c_double, C.c_double, C.c_int, C.c_void_p]),
    "pn_jpeg_parse": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(JpegDesc)]),
    "pn_jpeg_parse_oriented": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(JpegDesc)]),
    "pn_jpeg_workspace": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "pn_jpeg_decode": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p,
                                 C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "pn_jpeg_workspace_scaled": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "pn_jpeg_decode_scaled": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "pn_jpeg_encode_bound": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64)]),
    "pn_jpeg_encode_workspace": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "pn_jpeg_encode": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pn_png_encode_bound": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int64)]),
    "pn_png_encode_workspace": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "pn_png_encode": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                C.c_void_p, C.c_size_t, C.c_void_p]),
    "pn_yuv_to_bgr": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "pn_plan_query": (C.c_int, [C.POINTER(NetDesc), C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "pn_plan_create": (C.c_int, [C.POINTER(NetDesc), C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "pn_plan_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pn_plan_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float),
                                  C.c_int, C.c_void_p]),
    "pn_plan_num_launches": (C.c_int, [C.c_void_p]),
    "pn_plan_launch_name": (C.c_char_p, [C.c_void_p, C.c_int]),
    "pn_plan_destroy": (C.c_int, [C.c_void_p]),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def load():
    """Return the loaded library (symbols typed).  Raises NativeError if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and os.environ.get("POSENET_B200_AUTOBUILD") == "1":
        import importlib.util
        spec = importlib.util.spec_from_file_location("_pn_build", os.path.join(_PKG_ROOT, "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    if not os.path.exists(LIB_PATH):
        raise NativeError("libposenet_b200.so not found at %s -- build it with `python posenet-pytorch_b200/build.py` "
                          "(there is no CPU or PyTorch fallback)" % LIB_PATH)
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise NativeError("cannot load %s: %s" % (LIB_PATH, e))
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise NativeError("%s does not export %s (stale build?)" % (LIB_PATH, name))
        fn.restype = res
        fn.argtypes = args
    if lib.pn_abi_version() != ABI_VERSION:
        raise NativeError("ABI mismatch: library %d, binding %d" % (lib.pn_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc, what):
    if rc != PN_OK:
        msg = load().pn_last_error_string()
        raise NativeError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))


_device_ok = set()


def require_device():
    """Raise unless a B200-class CUDA device is current -- the product path has no other backend."""
    import torch
    if torch.cuda.is_available() and torch.cuda.current_device() in _device_ok:
        return
    if not torch.cuda.is_available():
        raise NativeError("posenet_b200 needs a CUDA device (sm_100a); torch.cuda.is_available() is False and "
                          "there is no CPU fallback")
    check(load().pn_device_check(), "pn_device_check")
    _device_ok.add(torch.cuda.current_device())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def make_map(t):
    """pn_map of a 4-D f32 CUDA tensor [n_img, C, h, w] with arbitrary strides."""
    assert t.dim() == 4 and t.is_cuda
    s = t.stride()
    return Map(t.data_ptr(), s[0], s[1], s[2], s[3])
