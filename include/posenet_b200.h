/*
 * posenet_b200.h -- C ABI of libposenet_b200.so: the B200 (sm_100a) PoseNet inference hot path
 *
 *     preprocess -> MobileNetV1 backbone + 4 heads -> part candidates -> greedy multi-pose decode
 *
 * The reference (michellelychan/posenet-pytorch) is pure Python and has no FFI / plugin /
 * operator interface; its boundary for this path is the Python API.  Each entry point below
 * therefore names the reference *function* (file:line, relative to the reference checkout)
 * whose arithmetic it replaces; posenet-pytorch_b200/posenet/ binds them with ctypes behind the
 * reference's own names (see INTEGRATION.md).
 *
 * Conventions
 *   - Plain pointers and sizes only.  Every pointer is a DEVICE pointer unless its name ends
 *     in _host.  The library never allocates device memory: the caller owns all buffers.
 *   - All work is enqueued on `stream` (a cudaStream_t); nothing synchronises.
 *   - Return value: PN_OK (0) or a negative PN_ERR_*; pn_last_error_string() describes the
 *     last failure on the calling thread.
 *   - Activations are NHWC ("pixel-major": [M = n*h*w, C]); `dtype` selects fp32 or bf16
 *     storage.  Head tensors and everything downstream are fp32 NCHW like the reference's.
 */
#ifndef POSENET_B200_H
#define POSENET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PN_ABI_VERSION 5

typedef void *pn_stream_t; /* cudaStream_t */

enum { PN_OK = 0, PN_ERR_ARG = -1, PN_ERR_CUDA = -2, PN_ERR_UNSUPPORTED = -3, PN_ERR_NO_DEVICE = -4 };
enum { PN_F32 = 0, PN_BF16 = 1 };

#define PN_NUM_PARTS 17
#define PN_NUM_EDGES 16
#define PN_HEAD_CHANNELS 115 /* 17 heatmap + 34 offset + 32 fwd + 32 bwd */
#define PN_HEAD_ROWS 128     /* packed head weight rows (115 padded to a UMMA-friendly 128) */

int pn_abi_version(void);
const char *pn_last_error_string(void);
/* PN_OK when the current CUDA device is an sm_100 part the kernels were built for. */
int pn_device_check(void);

/* ---- P1: posenet/utils.py:13-26 (_process_input; cv2.resize INTER_LINEAR + BGR->RGB + x*(2/255)-1)
 * src: uint8 [n, src_h, src_w, 3] BGR HWC.  dst: f32 [n, 3, dst_h, dst_w] RGB NCHW.  Bit-exact with cv2. */
int pn_preprocess_u8(const uint8_t *src, int n, int src_h, int src_w, int dst_h, int dst_w,
                     float *dst, pn_stream_t stream);
/* The resize stage of P1 alone (utils.py:21, cv2.resize INTER_LINEAR on uint8, bit-exact): uint8 [n, src_h, src_w, 3]
 * -> uint8 [n, dst_h, dst_w, 3], still BGR HWC -- the input format of pn_stem_conv_u8 / a uint8 plan, so frames of any
 * size (utils.py:51-55 read_cap at 1280x720) reach the uint8 fast path without a float round trip. */
int pn_resize_u8(const uint8_t *src, int n, int src_h, int src_w, int dst_h, int dst_w, uint8_t *dst,
                 pn_stream_t stream);

/* ---- B2: posenet/models/mobilenet_v1.py:47-54 (InputConv: relu6(conv3x3(x, stride, pad 1) + b), 3 -> cout)
 * x: f32 NCHW [n,3,h,w].  w: f32 [27, cout], row = (ky*3+kx)*3+ci.  y: NHWC [n,ho,wo,cout] of out_dtype. */
int pn_stem_conv(const float *x, const float *w, const float *bias, void *y, int n, int h, int wd,
                 int cout, int stride, int out_dtype, pn_stream_t stream);

/* ---- B2': P1 fused into B2 for already-sized images (identity resize): uint8 BGR HWC [n,h,w,3] in. */
int pn_stem_conv_u8(const uint8_t *img, const float *w, const float *bias, void *y, int n, int h, int wd,
                    int cout, int stride, int out_dtype, pn_stream_t stream);

/* ---- B3: mobilenet_v1.py:60-62,66 (SeperableConv.depthwise + relu6; stride 1|2, dilation 1|2|4,
 * padding ((s-1)+2d)/2 per mobilenet_v1.py:42-44).  x,y: NHWC of dtype.  w: f32 [9, c] tap-major. */
int pn_dwconv3x3(const void *x, const float *w, const float *bias, void *y, int n, int h, int wd, int c,
                 int stride, int dilation, int dtype, pn_stream_t stream);

/* ---- B4: mobilenet_v1.py:63,67 (SeperableConv.pointwise + relu6) == GEMM + bias + clamp(0,6)
 * a: [m,k] dtype.  w: [n,k] dtype (the OIHW 1x1 weight as stored).  bias: f32 [n].  y: [m,n] dtype.
 * bf16 runs on tcgen05 tensor cores (TMA-fed, TMEM accumulators); fp32 is the FFMA parity path. */
int pn_pwconv_gemm(const void *a, const void *w, const float *bias, void *y, int m, int k, int n,
                   int dtype, pn_stream_t stream);

/* ---- B3+B4 fused: mobilenet_v1.py:57-68 (SeperableConv.forward: relu6(pointwise(relu6(depthwise(x))))) as ONE
 * kernel -- the depthwise result is produced straight into the shared-memory A tile of the tcgen05 GEMM and never
 * reaches HBM.  bf16 only.  x: NHWC [n,h,wd,cin]; dw_w f32 [9,cin]; dw_b f32 [cin]; pw_w bf16 [cout,cin];
 * pw_b f32 [cout]; y: NHWC [n,ho,wo,cout].  cin % 8 == 0, cout % 16 == 0, (stride,dilation) in (1,1|2|4), (2,1). */
int pn_sepconv_block(const void *x, const float *dw_w, const float *dw_b, const void *pw_w, const float *pw_b, void *y,
                     int n, int h, int wd, int cin, int cout, int stride, int dilation, pn_stream_t stream);
/* Tile shape / pipeline depths pn_sepconv_block would pick for a block (host arithmetic only; diagnostics). */
int pn_sepconv_describe(int n, int h, int wd, int cin, int cout, int stride, int dilation, char *out_host, int capacity);

/* ---- H1: mobilenet_v1.py:151-154,158-161 (4 head convs + sigmoid on the heatmap) as ONE GEMM.
 * a: [n_img*hw, k] dtype.  w: [PN_HEAD_ROWS, k] dtype, rows heat|offset|fwd|bwd then zero padding.
 * Outputs f32 NCHW: heat [n_img,17,hw], off [n_img,34,hw], fwd/bwd [n_img,32,hw]. */
int pn_heads_gemm(const void *a, const void *w, const float *bias, float *heat, float *off, float *fwd,
                  float *bwd, int n_img, int hw, int k, int dtype, pn_stream_t stream);

/* A strided f32 view [n_img, channels, h, w]; strides in elements (NCHW or channels-last alike). */
typedef struct pn_map {
    const float *ptr;
    int64_t s_img, s_ch, s_y, s_x;
} pn_map;

/* ---- C1: posenet/decode_multi.py:27-34 (build_part_with_score_torch: 3x3 local max, -inf padding,
 * score >= fp32(threshold)).  keys: [n_img, capacity] 64-bit sort keys (high word orders by score
 * descending, low word = flat (part,y,x) index), UNORDERED within an image; counts: int32 [n_img].
 * capacity >= 17*h*w guarantees no candidate is dropped (counts never exceed capacity). */
int pn_candidates(const pn_map *heat, int n_img, int h, int wd, float score_threshold, uint64_t *keys,
                  int capacity, int *counts, pn_stream_t stream);

typedef struct pn_decode_params {
    int output_stride;
    int max_pose_detections;
    double squared_nms_radius; /* nms_radius ** 2, as the reference computes it on the host */
    double min_pose_score;
} pn_decode_params;

/* ---- D1-D4: decode_multi.py:61-148 + decode.py:9-63,131-182 (greedy multi-pose decode, float64).
 * One thread block per image; candidates are consumed in (score desc, flat index asc) order.
 * keys / counts are pn_candidates' outputs: the keys of an image must be pairwise distinct (they are -- the
 * low word is the cell index) and non-zero; the in-kernel radix selection relies on it.
 * Outputs (float64): pose_scores [n_img,P], kp_scores [n_img,P,17], kp_coords [n_img,P,17,2] (y,x),
 * kp_offsets [n_img,P,17,2]; pose_counts int32 [n_img].  The buffers need not be initialised: the rows
 * past pose_counts[i] are zero-padded by the kernel (the reference's np.zeros, decode_multi.py:94-100). */
int pn_decode_greedy(const pn_map *heat, const pn_map *off, const pn_map *fwd, const pn_map *bwd,
                     int n_img, int h, int wd, const uint64_t *keys, int capacity, const int *counts,
                     const pn_decode_params *params, double *pose_scores, double *kp_scores,
                     double *kp_coords, double *kp_offsets, int *pose_counts, pn_stream_t stream);

/* ---- D3: posenet/decode.py:9-63 (traverse_to_targ_keypoint) as a stand-alone call: ONE displacement hop along edge
 * `edge_id` from `source_keypoint_host` (float64 (y, x) image coordinates, HOST pointer) to part `target_keypoint_id`.
 * heat [1,17,h,w], off [1,34,h,w], disp [1,32,h,w] (channels 0..15 dy, 16..31 dx), any strides.
 * out7 (device, float64): score, image_coord y, x, displacement_vector y, x, offset y, x -- the fp32 values widened exactly. */
int pn_traverse_to_targ_keypoint(int edge_id, const double *source_keypoint_host, int target_keypoint_id,
                                 const pn_map *heat, const pn_map *off, const pn_map *disp, int h, int wd,
                                 int output_stride, double *out7, pn_stream_t stream);

/* ---- D2: posenet/decode.py:131-182 (decode_pose) as a stand-alone call for ONE root: backward edges 15..0 through `bwd`, then
 * forward edges 0..15 through `fwd`; a hop needs score[source] > 0.0 and an undecoded (== 0.0) target.
 * root_image_coord_host: float64 (y, x), HOST pointer.  out85 (device, float64): instance_keypoint_scores [17],
 * instance_keypoint_coords [17,2], instance_offsets [17,2] (the root's offset row stays 0, decode.py:150). */
int pn_decode_pose(double root_score, int root_id, const double *root_image_coord_host, const pn_map *heat,
                   const pn_map *off, const pn_map *fwd, const pn_map *bwd, int h, int wd, int output_stride,
                   double *out85, pn_stream_t stream);

/* ---- N4: image_demo.py:50 (`keypoint_coords *= output_scale`, output_scale = (src_h / target_h, src_w / target_w) of
 * utils.py:19) for a batch of pose records ON THE DEVICE: kp_coords float64 [n_img, points_per_img, 2] (y, x), multiplied in
 * place (IEEE float64 multiply, what numpy does).  scales: device float64 [n_img, 2] with one (y, x) factor per image (frames
 * of different sizes), or NULL for the uniform (scale_y, scale_x). */
int pn_scale_keypoint_coords(double *kp_coords, int n_img, int points_per_img, const double *scales, double scale_y,
                             double scale_x, pn_stream_t stream);

/* ---- N4: posenet/utils.py draw_skel_and_kp (image_demo.py:53) / draw_skeleton for a batch of frames ON THE DEVICE, drawn in
 * place and bit-exact with cv2 (drawKeypoints DRAW_RICH_KEYPOINTS circles, then polylines; colour (255, 255, 0) BGR).
 * frames: uint8 BGR HWC, image i at frames + i * frame_stride (bytes, >= h*w*3), rows w_i*3 bytes apart.  frame_hw: device
 * int32 [n_img, 2] with each frame's (h_i, w_i) (<= h, w; other rows, e.g. (0, 0), are skipped), or NULL for h x w everywhere.  The records
 * are pn_decode_greedy's (float64, coordinates (y, x) in frame pixels): pose_scores [n_img, max_poses], kp_scores
 * [n_img, max_poses, 17], kp_coords [n_img, max_poses, 17, 2]; max_poses <= 512.  `what`: PN_DRAW_KEYPOINTS | PN_DRAW_SKELETON
 * (both: draw_skel_and_kp; PN_DRAW_SKELETON alone: draw_skeleton).  Nothing outside a frame is written, whatever the
 * coordinates; within +-2^26 px they match cv2 bit for bit. */
#define PN_DRAW_KEYPOINTS 1
#define PN_DRAW_SKELETON 2
int pn_draw_poses(uint8_t *frames, int n_img, int h, int w, int64_t frame_stride, const int *frame_hw, const double *pose_scores,
                  const double *kp_scores, const double *kp_coords, int max_poses, double min_pose_score, double min_part_score,
                  int what, pn_stream_t stream);

/* ---- N2'': baseline JPEG files decoded ON THE DEVICE, bit-exact with cv2.imread / cv2.imdecode(IMREAD_COLOR) (libjpeg-turbo 3.1
 * with its defaults: jdhuff.c, the accurate integer IDCT of jidctint.c, fancy upsampling of jdsample.c, jdcolor.c YCbCr -> BGR).
 *
 * pn_jpeg_parse (host only, no device needed) reads a file's headers into a descriptor and classifies it: PN_JPEG_SUPPORTED
 * (1- or 3-component YCbCr / grayscale, 8-bit, baseline / extended Huffman, one interleaved scan, sampling factors 1..4 x 1..2 with
 * integral ratios, EXIF orientation 1 or absent -- or certain, with pn_jpeg_parse_oriented --, ending in an EOI) or PN_JPEG_HOST
 * with a PN_JPEG_WHY_* reason; host files are for cv2 to decode.  The descriptor carries everything the device needs: geometry, quantisation tables (natural order) and the derived
 * Huffman tables (validated like jpeg_make_d_derived_tbl). */
enum { PN_JPEG_SUPPORTED = 0, PN_JPEG_HOST = 1 };
enum {
    PN_JPEG_WHY_NONE = 0, PN_JPEG_WHY_NOT_JPEG, PN_JPEG_WHY_TRUNCATED, PN_JPEG_WHY_PROGRESSIVE, PN_JPEG_WHY_ARITHMETIC,
    PN_JPEG_WHY_LOSSLESS, PN_JPEG_WHY_PRECISION, PN_JPEG_WHY_MULTI_SCAN, PN_JPEG_WHY_COMPONENTS, PN_JPEG_WHY_RGB,
    PN_JPEG_WHY_NO_DHT, PN_JPEG_WHY_EXIF_ORIENTATION, PN_JPEG_WHY_SAMPLING, PN_JPEG_WHY_BAD_TABLE, PN_JPEG_WHY_UNKNOWN
};
/* pn_jpeg_decode's per-image status: 0 decoded, 1 skipped (a PN_JPEG_HOST descriptor: its frame is left untouched), < 0 the
 * descriptor or the entropy-coded data is malformed (its frame is written as zeros; cv2's recovery is not reproduced). */
enum { PN_JPEG_OK = 0, PN_JPEG_SKIPPED = 1, PN_JPEG_ERR_DESC = -1, PN_JPEG_ERR_NO_END = -2, PN_JPEG_ERR_RESTART = -3,
       PN_JPEG_ERR_CODE = -4, PN_JPEG_ERR_LENGTH = -5 };
#define PN_JPEG_MAX_BLOCKS 10 /* blocks per MCU (libjpeg's D_MAX_BLOCKS_IN_MCU) */

typedef struct pn_jpeg_huff {
    uint16_t lookup[256];  /* next 8 bits -> (code length << 8) | symbol; 0: the code is longer than 8 bits */
    int32_t maxcode[18];   /* largest code of length l, -1 if none; maxcode[17] is a sentinel */
    int32_t valoffset[18]; /* huffval index of a code of length l: code + valoffset[l] */
    uint8_t huffval[256];
} pn_jpeg_huff;

typedef struct pn_jpeg_comp {
    int32_t h, v;            /* sampling factors as coded in the MCU (1 x 1 for a single-component scan) */
    int32_t hr, vr;          /* upsampling ratios max_h / h, max_v / v */
    int32_t dc, ac;          /* pn_jpeg_desc.huff slots */
    int32_t bw, bh;          /* coefficient plane size in blocks (MCU-padded) */
    int32_t dw, dh;          /* downsampled_width / downsampled_height */
} pn_jpeg_comp;

typedef struct pn_jpeg_desc {
    int32_t kind, why;       /* PN_JPEG_SUPPORTED | PN_JPEG_HOST, PN_JPEG_WHY_* */
    int32_t height, width, ncomp;
    int32_t mcus_x, mcus_y, blocks_per_mcu;
    int32_t restart_interval; /* MCUs per restart interval (the whole scan when the file has no DRI) */
    int32_t n_segments;       /* restart intervals in the scan */
    int64_t file_offset;      /* set by the caller: byte offset of the file in pn_jpeg_decode's byte arena */
    int64_t file_bytes;
    int64_t scan_offset;      /* first entropy-coded byte, from the start of the file */
    pn_jpeg_comp comp[3];     /* in frame (SOF) order: Y, Cb, Cr */
    uint8_t mcu_comp[PN_JPEG_MAX_BLOCKS], mcu_bx[PN_JPEG_MAX_BLOCKS], mcu_by[PN_JPEG_MAX_BLOCKS];
    uint8_t orientation;      /* EXIF orientation the decode applies (cv2's): 0 or 1 none, 2..8 (pn_jpeg_parse_oriented) */
    uint8_t pad[1];
    int16_t quant[3][64];     /* per component, natural order (libjpeg's ISLOW_MULT_TYPE) */
    pn_jpeg_huff huff[4];
} pn_jpeg_desc;

/* Parse the headers of one file (HOST pointers).  PN_OK whatever the classification; PN_ERR_ARG for null pointers.  A file with an
 * Exif APP1 segment that cannot be read or gives an orientation other than 1 is PN_JPEG_HOST (PN_JPEG_WHY_EXIF_ORIENTATION);
 * desc->orientation is 0. */
int pn_jpeg_parse(const uint8_t *file_host, int64_t nbytes, pn_jpeg_desc *desc_host);
/* The same, except that a file whose EXIF orientation o in 2..8 is certain is PN_JPEG_SUPPORTED with desc->orientation = o, and
 * is decoded rotated / flipped as cv2.imread does (out(y, x) of the H x W frame r: 2 r(y, W-1-x), 3 r(H-1-y, W-1-x), 4 r(H-1-y, x),
 * 5 r(x, y), 6 r(H-1-x, y), 7 r(H-1-x, W-1-y), 8 r(x, W-1-y); 5..8 are W x H).  Certain: every Exif segment is readable (II / MM,
 * 42, IFD0 and all its entries inside the segment), each has at most one 0x0112 entry, a SHORT with count 1 whose preceding
 * entries are in TIFF order, of known types, with their data inside the segment, and all such entries agree.  Other files with an
 * orientation other than 1 stay PN_JPEG_HOST as with pn_jpeg_parse. */
int pn_jpeg_parse_oriented(const uint8_t *file_host, int64_t nbytes, pn_jpeg_desc *desc_host);

/* Progressive files (SOF2, Huffman-coded, jdphuff.c), decoded ON THE DEVICE when the caller opts in with
 * pn_jpeg_parse_progressive.  Such a descriptor is kind PN_JPEG_SUPPORTED_PROGRESSIVE: its geometry is that of one interleaved scan
 * of all components (one component: the plane's own block grid), restart_interval covers the whole image, n_segments is 1 and
 * huff[] is unused.  Its scans are described by a scan table the caller stores in the byte arena at file_offset +
 * align8(file_bytes), 8-byte aligned: a pn_jpeg_scans header, then n_scans pn_jpeg_scan, then n_huff pn_jpeg_huff.
 * A scan's wave is the length of the longest chain of earlier scans it depends on (same component, overlapping coefficients):
 * the scans of one wave touch disjoint coefficients and are decoded in parallel, waves in order. */
enum { PN_JPEG_SUPPORTED_PROGRESSIVE = 2 };
#define PN_JPEG_MAX_SCANS 64      /* scans of a progressive file; more: PN_JPEG_HOST */
#define PN_JPEG_MAX_SCAN_HUFF 32  /* derived Huffman tables its scans use (a DHT redefining a slot counts again); more: PN_JPEG_HOST */
typedef struct pn_jpeg_scan {
    int64_t start, end;        /* entropy-coded bytes [start, end) from the start of the file, RST markers included */
    int32_t restart_interval;  /* MCUs per restart interval in this scan (blocks in a one-component scan), 0 for none */
    int32_t wave;
    uint8_t ncomp, ss, se, ah, al;
    uint8_t comp[3];           /* frame component indices, in scan order */
    uint8_t dc[3], ac[3];      /* indices into the table's pn_jpeg_huff[]: DC tables of a first DC scan, the AC table of an AC scan */
    uint8_t pad[2];
} pn_jpeg_scan;
typedef struct pn_jpeg_scans {
    int32_t n_scans, n_huff, n_waves, pad;
} pn_jpeg_scans;
/* Baseline files come back exactly as pn_jpeg_parse (oriented = 0) or pn_jpeg_parse_oriented (oriented != 0) return them, with
 * *scans_bytes = 0.  A progressive file is PN_JPEG_SUPPORTED_PROGRESSIVE with its scan table in scans_host (*scans_bytes bytes)
 * when libjpeg-turbo decodes it without a warning and without block smoothing: a complete scan script (every coefficient of every
 * component refined to Al = 0), a legal progression (Ah equal to the coefficient's previous Al, Al <= 13, DC scans with Se = 0,
 * AC scans with one component and 1 <= Ss <= Se <= 63, no AC scan before the component's DC), at most PN_JPEG_MAX_SCANS scans and
 * PN_JPEG_MAX_SCAN_HUFF tables, and everything the baseline parser asks of a file's other headers.  Other progressive files are
 * PN_JPEG_HOST (PN_JPEG_WHY_PROGRESSIVE), as are files whose table needs more than scans_cap bytes (*scans_bytes is then what it
 * needs).  Host only. */
int pn_jpeg_parse_progressive(const uint8_t *file_host, int64_t nbytes, int oriented, pn_jpeg_desc *desc_host, void *scans_host,
                              int64_t scans_cap, int64_t *scans_bytes);
/* Device workspace (bytes, 256-byte aligned base) pn_jpeg_decode needs for up to n_img files of together at most arena_bytes
 * bytes, none larger than max_h x max_w. */
int pn_jpeg_workspace(int n_img, int64_t arena_bytes, int max_h, int max_w, size_t *bytes_host);
/* Decode n_img files at once.  files: device byte arena (file i at descs[i].file_offset, arena_bytes in all); descs: DEVICE array
 * of pn_jpeg_parse's descriptors with file_offset filled in.  Frame i is written as uint8 BGR HWC at its own size, contiguous
 * from frames + i * frame_stride (frame_stride >= 3 * max_h * max_w); nothing else in a row and nothing outside the frames is
 * written, and no byte outside a file's range is read, whatever the file contains.  frame_hw (optional, device int32 [n_img, 2])
 * receives each decoded frame's (h, w) -- after the descriptor's orientation, which max_h x max_w also bound --, (0, 0) for the others; status: device int32 [n_img], PN_JPEG_OK / _SKIPPED / < 0.  The
 * launch geometry depends only on the arguments, not on the descriptors' contents, so the call can be captured in a CUDA graph. */
int pn_jpeg_decode(const uint8_t *files, int64_t arena_bytes, const pn_jpeg_desc *descs, int n_img, int max_h, int max_w,
                   uint8_t *frames, int64_t frame_stride, int *frame_hw, void *workspace, size_t ws_bytes, int *status,
                   pn_stream_t stream);
/* The same at 1 / scale_denom (1, 2, 4 or 8; anything else is PN_ERR_ARG), bit-exact with cv2.imdecode(buf,
 * IMREAD_REDUCED_COLOR_<scale_denom>): libjpeg's DCT-domain scaling (jidctred.c), no full-size intermediate.  Frame i is
 * ceil(height / scale_denom) x ceil(width / scale_denom), and that is what frame_hw reports; max_h x max_w bound those reduced
 * sizes (a file up to scale_denom * max_h x scale_denom * max_w).  With scale_denom 1 these are pn_jpeg_workspace /
 * pn_jpeg_decode. */
int pn_jpeg_workspace_scaled(int n_img, int64_t arena_bytes, int max_h, int max_w, int scale_denom, size_t *bytes_host);
int pn_jpeg_decode_scaled(const uint8_t *files, int64_t arena_bytes, const pn_jpeg_desc *descs, int n_img, int max_h, int max_w,
                          int scale_denom, uint8_t *frames, int64_t frame_stride, int *frame_hw, void *workspace, size_t ws_bytes,
                          int *status, pn_stream_t stream);

/* ---- N5: image_demo.py:57 cv2.imwrite of the drawn frames: baseline JPEG files encoded ON THE DEVICE, bit-exact with
 * cv2.imencode(".jpg", frame, params) (libjpeg-turbo 3.1 as cv2 4.13 calls it: jccolor.c, jcsample.c, the accurate integer FDCT
 * of jfdctint.c, the Annex K Huffman tables, JFIF headers; no optimised tables, not progressive).
 *
 * sampling: cv2's IMWRITE_JPEG_SAMPLING_FACTOR_* value (0x411111, 0x221111, 0x211111, 0x121111, 0x111111); restart_interval:
 * MCUs per interval, 0 for none (cv2's IMWRITE_JPEG_RST_INTERVAL).
 *
 * pn_jpeg_encode_bound (host only): a true worst case of one file of h x w (every block at its largest Huffman code length,
 * every byte stuffed, markers and headers); 0 for 0 x 0. */
int pn_jpeg_encode_bound(int h, int w, int sampling, int restart_interval, int64_t *bytes_host);
/* Device workspace (bytes, 256-byte aligned base) pn_jpeg_encode needs for up to n_img frames of at most max_h x max_w. */
int pn_jpeg_encode_workspace(int n_img, int max_h, int max_w, int sampling, int restart_interval, size_t *bytes_host);
/* Encode n_img frames at once.  frames: device uint8 BGR HWC, frame i from frames + i * frame_stride (>= 3 * max_h * max_w), rows
 * of w_i * 3 bytes; frame_hw: device int32 [n_img, 2] with each frame's (h_i, w_i), a size outside 1..max_h x 1..max_w giving an
 * empty file, or NULL for max_h x max_w everywhere.  quality: 0..100 (0 behaves like 1, as in cv2).  out: device bytes, packed:
 * file i is out[out_offsets[i] .. out_offsets[i + 1]) with out_offsets device int64 [n_img + 1]; out_capacity must be at least
 * n_img * pn_jpeg_encode_bound(max_h, max_w, ..) and nothing at or past out_offsets[n_img] is written.  The frames are only read.
 * The launch geometry depends only on the capacity, so the call can be captured in a CUDA graph (quality is fixed then). */
int pn_jpeg_encode(const uint8_t *frames, int n_img, int max_h, int max_w, int64_t frame_stride, const int *frame_hw, int quality,
                   int sampling, int restart_interval, uint8_t *out, int64_t out_capacity, int64_t *out_offsets, void *workspace,
                   size_t ws_bytes, pn_stream_t stream);

/* ---- N6: image_demo.py:57 cv2.imwrite of the drawn frames to .png names: PNG files encoded ON THE DEVICE, bit-exact with
 * cv2.imencode(".png", frame) without params (libpng 1.6 with cv2's SUB filter, zlib 1.3 deflate at level 1 with Z_RLE, IDAT
 * chunks of 8192 bytes).
 *
 * pn_png_encode_bound (host only): a true worst case of one file of h x w (every block at its static coding, 9 bits a byte, or
 * stored, with block, zlib and chunk overhead); 0 for 0 x 0. */
int pn_png_encode_bound(int h, int w, int64_t *bytes_host);
/* Device workspace (bytes, 256-byte aligned base) pn_png_encode needs for up to n_img frames of at most max_h x max_w. */
int pn_png_encode_workspace(int n_img, int max_h, int max_w, size_t *bytes_host);
/* Encode n_img frames at once.  frames: device uint8 BGR HWC, frame i from frames + i * frame_stride (>= 3 * max_h * max_w), rows
 * of w_i * 3 bytes; frame_hw: device int32 [n_img, 2] with each frame's (h_i, w_i), a size outside 1..max_h x 1..max_w giving an
 * empty file, or NULL for max_h x max_w everywhere.  out: device bytes, packed: file i is out[out_offsets[i] .. out_offsets[i + 1])
 * with out_offsets device int64 [n_img + 1]; out_capacity must be at least n_img * pn_png_encode_bound(max_h, max_w) and nothing
 * at or past out_offsets[n_img] is written.  The frames are only read.  The launch geometry depends only on the capacity, so the
 * call can be captured in a CUDA graph. */
int pn_png_encode(const uint8_t *frames, int n_img, int max_h, int max_w, int64_t frame_stride, const int *frame_hw, uint8_t *out,
                  int64_t out_capacity, int64_t *out_offsets, void *workspace, size_t ws_bytes, pn_stream_t stream);

/* ---- N7: webcam_demo.py read_cap of video frames that arrive as YUV (software decoders give I420, hardware decoders and capture
 * devices NV12, UVC webcams YUY2): a batch converted to BGR ON THE DEVICE, bit-exact with cv2.cvtColor(frame,
 * cv2.COLOR_YUV2BGR_<layout>) (BT.601 limited range in 20-bit fixed point, nearest chroma).
 *
 * Frame i is read from src + i * src_stride in cv2's own layout (4:2:0: [h * 3 / 2, w], the Y plane then the chroma; 4:2:2:
 * [h, w, 2]) and written as uint8 BGR HWC [h, w, 3] at dst + i * dst_stride.  w must be even, and h too for 4:2:0 (what cv2
 * accepts).  src_stride is at least the frame's bytes (h * w * 3 / 2 or h * w * 2), dst_stride at least h * w * 3.  No byte
 * outside the frames is read or written.
 * The launch geometry depends only on the arguments, so the call can be captured in a CUDA graph. */
typedef enum pn_yuv_layout {
    PN_YUV_I420 = 0, /* Y, U (h/2 x w/2), V; COLOR_YUV2BGR_I420 / _IYUV */
    PN_YUV_YV12 = 1, /* Y, V, U; COLOR_YUV2BGR_YV12 */
    PN_YUV_NV12 = 2, /* Y, interleaved UV (h/2 x w); COLOR_YUV2BGR_NV12 */
    PN_YUV_NV21 = 3, /* Y, interleaved VU; COLOR_YUV2BGR_NV21 */
    PN_YUV_YUY2 = 4, /* Y0 U Y1 V; COLOR_YUV2BGR_YUY2 / _YUYV / _YUNV */
    PN_YUV_UYVY = 5, /* U Y0 V Y1; COLOR_YUV2BGR_UYVY / _Y422 / _UYNV */
    PN_YUV_YVYU = 6  /* Y0 V Y1 U; COLOR_YUV2BGR_YVYU */
} pn_yuv_layout;
int pn_yuv_to_bgr(const uint8_t *src, int n_img, int h, int w, int64_t src_stride, int layout, uint8_t *dst, int64_t dst_stride,
                  pn_stream_t stream);

/* ---- N8: the inverse, for video sinks (ffmpeg rawvideo, GStreamer appsrc, v4l2loopback, hardware encoders take YUV): a batch
 * of BGR frames converted to YUV ON THE DEVICE, bit-exact with cv2.cvtColor(frame, cv2.COLOR_BGR2YUV_<layout>), for the five
 * layouts cv2 writes: PN_YUV_I420 (COLOR_BGR2YUV_I420 / _IYUV), PN_YUV_YV12, PN_YUV_YUY2 (_YUY2 / _YUYV / _YUNV), PN_YUV_UYVY
 * (_UYVY / _Y422 / _UYNV) and PN_YUV_YVYU.  NV12 / NV21 (cv2 writes neither) give PN_ERR_ARG.  4:2:0 takes its chroma from the
 * top-left pixel of each 2x2 block, 4:2:2 from the average of each horizontal pair, as cv2 does.
 *
 * Frame i is read from src + i * src_stride (dense [h, w, 3] BGR, src_stride >= h * w * 3) and written at dst + i * dst_stride
 * in cv2's output layout (dst_stride >= h * w * 3 / 2 or h * w * 2).  Sizes follow cv2: w even, h even for 4:2:0.  Any strides;
 * nothing outside the frames is read or written.  The launch geometry depends only on the arguments (graph-capturable). */
int pn_bgr_to_yuv(const uint8_t *src, int n_img, int h, int w, int64_t src_stride, int layout, uint8_t *dst, int64_t dst_stride,
                  pn_stream_t stream);

/* ---- N9: pose tracking across video frames: the bounding-box tracker of TF.js pose-detection (BoundingBoxTracker), run ON
 * THE DEVICE on the records pn_decode_greedy writes, so that pose k of frame t keeps its id in frame t + 1.
 *
 * A stream is a video source with an id in 0 .. n_streams-1; stream_ids (device int32 [n_img]) names the stream of each row, and
 * a row whose id is outside 0 .. n_streams-1 is not tracked.  Each stream holds up to max_tracks tracks (id, box, the stream
 * frame at which it was last matched), a frame counter and the count of ids it issued.  Rows are frames, taken in row order per
 * stream.  A detection is a record with pose_score > 0; its box is the min / max of y and x over its keypoints with score >=
 * min_part_score (none: an empty box).  Per frame: the stream's counter becomes t; tracks with t - last > max_age are dropped
 * (stably); each detection in record order takes the unmatched track of largest IoU among those with IoU >= min_similarity (the
 * first such track on a tie), which takes its box and last = t, or else gets a new track with the next id (1, 2, ... per
 * stream); the tracks are then stably sorted by last, descending, and the first max_tracks kept.  IoU in float64 without FMA:
 * inter = (min(ymax) - max(ymin)) * (min(xmax) - max(xmin)) when both factors are > 0 and neither box is empty, else 0;
 * IoU = inter / (area_a + area_b - inter), 0 when that union is <= 0.
 *
 * pose_scores [n_img, P], keypoint_scores [n_img, P, 17], keypoint_coords [n_img, P, 17, 2] (y, x): float64, 8-byte aligned;
 * P <= 256.  ids: device int64 [n_img, P]: the track id of each detection, -1 for records that are not detections and for
 * untracked rows.  state: device, pn_track_state_bytes(n_streams, max_tracks) bytes, 8-byte aligned; ALL ZERO BYTES IS THE
 * START of every stream (zero a stream's pn_track_state_bytes(1, max_tracks) bytes at state + s * that to reset it).  The
 * state must be used with one (n_streams, max_tracks) only.  max_tracks <= 256, max_age >= 0.  One warp per stream: the
 * launch geometry depends only on n_streams, so the call can be captured in a CUDA graph. */
int pn_track_state_bytes(int n_streams, int max_tracks, size_t *bytes_host);
int pn_track_poses(const double *pose_scores, const double *keypoint_scores, const double *keypoint_coords, int n_img, int P,
                   const int *stream_ids, void *state, int n_streams, int max_tracks, int max_age, double min_similarity,
                   double min_part_score, int64_t *ids, pn_stream_t stream);

/* ---- N10: One Euro smoothing of tracked keypoints (Casiez et al., CHI 2012, the filter TF.js pose-detection runs per tracked
 * pose), ON THE DEVICE, on the ids pn_track_poses writes, so that a still person's keypoints stop jittering.
 *
 * Streams and rows as for pn_track_poses (stream_ids: device int32 [n_img]; a row whose id is outside 0 .. n_streams-1 is left
 * as it is).  Each stream holds a frame counter, which advances on every row of the stream, and a table of up to max_tracks
 * entries: a track id, the stream frame of its last update (last), and per coordinate the previous raw value, previous
 * filtered value and previous filtered derivative (float64).  Per frame: the counter becomes t; entries with t - last > max_age
 * are dropped (stably); each detection (record with id >= 1) in record order updates the entry of its id, or else appends a
 * fresh entry, or else (table full) replaces the entry of smallest last < t (the first on a tie); when every entry was updated
 * in this frame, or its id was already met in this frame, the record keeps its coordinates.  A fresh entry keeps x and stores
 * x_prev = x_hat = x, dx_hat = 0.  An update, per coordinate, in float64 without FMA and in this order:
 *   rate = fps / (t - last); dx = (x - x_prev) * rate; a_d = 1 / (1 + rate / (2 pi d_cutoff));
 *   dx_hat = a_d dx + (1 - a_d) dx_hat; cutoff = min_cutoff + beta |dx_hat|; a = 1 / (1 + rate / (2 pi cutoff));
 *   x_hat = a x + (1 - a) x_hat; x_prev = x; the output is x_hat.
 * All 17 keypoints are filtered whatever their score; scores are never read.
 *
 * ids: device int64 [n_img, P] (pn_track_poses's output); keypoint_coords: device float64 [n_img, P, 17, 2] (y, x), smoothed
 * IN PLACE; 8-byte aligned; P <= 256.  state: device, pn_smooth_state_bytes(n_streams, max_tracks) bytes, 8-byte aligned,
 * contiguous per stream; ALL ZERO BYTES IS THE START of every stream (zero a stream's pn_smooth_state_bytes(1, max_tracks)
 * bytes at state + s * that to reset it, together with its tracks).  The state must be used with one (n_streams, max_tracks)
 * only.  max_tracks <= 256, max_age >= 0; fps, min_cutoff, d_cutoff finite and > 0, beta finite and >= 0.  One CTA per
 * stream: the launch geometry depends only on n_streams, so the call can be captured in a CUDA graph. */
int pn_smooth_state_bytes(int n_streams, int max_tracks, size_t *bytes_host);
int pn_smooth_keypoints(const int64_t *ids, double *keypoint_coords, int n_img, int P, const int *stream_ids, void *state,
                        int n_streams, int max_tracks, int max_age, double fps, double min_cutoff, double beta, double d_cutoff,
                        pn_stream_t stream);

/* ---- Whole-network plan: mobilenet_v1.py:130-162 (MobileNetV1.__init__/forward) --------------------
 * The layer table is computed by the caller (posenet/models/mobilenet_v1.py mirrors
 * _to_output_strided_layers, mobilenet_v1.py:8-39) and passed in explicitly. */
typedef struct pn_layer {
    int cin, cout, stride, dilation;
    const float *dw_w, *dw_b; /* [9,cin], [cin]   (NULL for the stem) */
    const void *pw_w;         /* stem: f32 [27,cout]; blocks: [cout,cin] of plan dtype */
    const float *pw_b;        /* [cout] */
} pn_layer;

typedef struct pn_net_desc {
    int dtype;       /* PN_F32 | PN_BF16: activation + pointwise weight storage */
    int n, h, w;     /* batch and input size */
    int input_u8;    /* 0: f32 NCHW input (reference forward()); 1: uint8 BGR HWC of size h x w */
    int num_layers;  /* 14 */
    pn_layer layers[16];
    const void *head_w;    /* [PN_HEAD_ROWS, c_last] plan dtype */
    const float *head_b;   /* [PN_HEAD_ROWS] */
    int flags;             /* PN_PLAN_* */
} pn_net_desc;

/* bf16 plans run every SeperableConv block as one fused kernel (pn_sepconv_block) by default;
 * PN_PLAN_UNFUSED keeps depthwise and pointwise as two kernels (pn_dwconv3x3 + pn_pwconv_gemm). */
#define PN_PLAN_UNFUSED 1

typedef struct pn_plan pn_plan;

/* Bytes of activation arena pn_plan_create needs for `desc` (two ping-pong buffers), and the
 * head map size (out_h, out_w). */
int pn_plan_query(const pn_net_desc *desc, size_t *arena_bytes, int *out_h, int *out_w);
int pn_plan_create(const pn_net_desc *desc, void *arena, size_t arena_bytes, pn_plan **plan);
/* input: f32 NCHW or uint8 HWC as desc->input_u8 says.  Enqueues the kernels of one forward (15 fused, 28 unfused). */
int pn_plan_forward(pn_plan *plan, const void *input, float *heat, float *off, float *fwd, float *bwd,
                    pn_stream_t stream);
/* Same launches as pn_plan_forward with a CUDA event between consecutive kernels; synchronises `stream`
 * and writes the device time of each launch (ms, launch order; see pn_plan_launch_name)
 * into ms_host[0 .. pn_plan_num_launches).  Measurement aid for bench.py's roofline; host pointer. */
int pn_plan_profile(pn_plan *plan, const void *input, float *heat, float *off, float *fwd, float *bwd,
                    float *ms_host, int capacity, pn_stream_t stream);
/* number of kernel launches one pn_plan_forward enqueues */
int pn_plan_num_launches(const pn_plan *plan);
/* name of launch i in launch order: "stem", "dw3" / "pw3" (unfused), "sep3" (fused block 3), "heads" */
const char *pn_plan_launch_name(const pn_plan *plan, int i);
int pn_plan_destroy(pn_plan *plan);

#ifdef __cplusplus
}
#endif
#endif /* POSENET_B200_H */
