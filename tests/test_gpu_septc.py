"""Depthwise on the tensor pipe (csrc/septc.cu; the 256 -> 256 blocks at stride 1, dilation 1 or 2) through the C ABI on the B200.

(1) pn_dwtc_probe: the hardware behaviours the kernel relies on -- a SWIZZLE_128B UMMA descriptor advanced by whole 128-byte
    rows reads a shifted view of the TMA-written patch (depthwise taps; equal to numpy fp32 up to rare one-ulp flips of the bf16 rounding), and tcgen05.mma takes
    its A operand from TMEM (pointwise on the depthwise result).
(2) pn_sepconv_block on those blocks against a torch fp32 reference of mobilenet_v1.py:57-68 (SeperableConv) with the
    kernel's rounding points: bf16 input, bf16 depthwise weights, bf16 depthwise output, bf16 output."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import abi  # noqa: E402
from posenet import _native as nat  # noqa: E402

DEV = "cuda"
P = lambda t: C.c_void_p(t.data_ptr())


def _bf16(a):
    return torch.from_numpy(a).to(torch.bfloat16).to(torch.float32).numpy()


PROBE_CASES = [  # h, w, dilation, pitch, box x origin, band x0, band width, chunk
    (20, 33, 1, 34, -1, 0, 33, 0), (20, 33, 1, 34, -1, 0, 33, 3),     # full-width band, pitch W + D (shared zero gap)
    (24, 40, 1, 16, 7, 8, 14, 1),                                      # interior band with real neighbours either side
    (20, 29, 2, 31, -2, 0, 29, 2),                                     # dilation 2
]


@pytest.mark.parametrize("case", PROBE_CASES)
def test_shifted_descriptor_depthwise_and_tmem_operand(case):
    h, w, dil, wp, x_org, band_x0, tw, chunk = case
    rng = np.random.default_rng(chunk + h)
    x = _bf16(rng.uniform(0, 6, (h, w, 64)).astype(np.float32))
    wdw = _bf16(rng.normal(0, 0.4, (9, 64)).astype(np.float32))
    bias = rng.normal(0, 0.3, 64).astype(np.float32)
    pww = _bf16(rng.normal(0, 0.2, (64, 64)).astype(np.float32))
    diag = np.zeros((9, 16, 64), np.float32)
    for g in range(4):
        for n in range(16):
            diag[:, n, 16 * g + n] = wdw[:, 16 * g + n]
    q0 = chunk * 128
    row0 = q0 // wp
    rows_box = (q0 + 127) // wp - row0 + 1 + 2 * dil
    xd = torch.from_numpy(x).to(torch.bfloat16).to(DEV)
    dd = torch.from_numpy(diag.reshape(144, 64)).to(torch.bfloat16).to(DEV)
    wd_ = torch.from_numpy(pww).to(torch.bfloat16).to(DEV)
    bd = torch.from_numpy(bias).to(DEV)
    out_dw = torch.zeros((128, 64), dtype=torch.float32, device=DEV)
    out_pw = torch.zeros((128, 64), dtype=torch.float32, device=DEV)
    abi.check_diag(abi.load_diag().pn_dwtc_probe(P(xd), h, w, P(dd), P(wd_), P(bd), P(out_dw), P(out_pw), wp, dil, q0 - row0 * wp, rows_box,
                                       x_org, row0 - dil, 0, nat.stream_ptr()), "pn_dwtc_probe")
    torch.cuda.synchronize()
    got_dw, got_pw = out_dw.cpu().numpy(), out_pw.cpu().numpy()
    o = 2 * dil + 4
    xp = np.zeros((h + 2 * o, w + 2 * o, 64), np.float32)
    xp[o:o + h, o:o + w] = x
    valid = flips = 0
    for r in range(128):
        ty, tx = (q0 + r) // wp, (q0 + r) % wp
        gx = band_x0 + tx
        if tx >= tw or gx >= w or ty >= h:
            continue
        acc = np.zeros(64, np.float32)
        for t in range(9):                                   # the kernel's tap order: fp32 accumulation of exact products
            acc += xp[o + ty + (t // 3 - 1) * dil, o + gx + (t % 3 - 1) * dil] * wdw[t]
        ref = _bf16(np.clip(acc + bias, 0, 6).astype(np.float32))
        diff = np.abs(got_dw[r] - ref)                       # equal up to the fp32 summation order: at most one bf16 ulp, rarely
        assert (diff <= np.abs(ref) * 2.0 ** -7).all(), (r, diff.max())
        flips += int((diff > 0).sum())
        ref_pw = got_dw[r].astype(np.float64) @ pww.T.astype(np.float64)
        assert np.abs(got_pw[r] - ref_pw).max() < 1e-4
        valid += 1
    assert valid >= 100 and flips <= valid * 64 // 500


SHAPES = [  # n, h, w, cin, cout, dilation -- the blocks of models 101 / 50, one and two bands (ragged), tiny maps
    (2, 65, 65, 256, 256, 1), (3, 33, 33, 256, 256, 1), (5, 17, 17, 256, 256, 1), (1, 45, 81, 256, 256, 1), (1, 12, 33, 256, 256, 1),
    (2, 5, 3, 256, 256, 1), (1, 1, 1, 256, 256, 1),
    (1, 91, 161, 256, 256, 2), (1, 46, 81, 256, 256, 2), (2, 33, 33, 256, 256, 2), (1, 12, 33, 256, 256, 2), (2, 5, 3, 256, 256, 2),
    (1, 1, 1, 256, 256, 2), (4, 9, 9, 256, 256, 2),
]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "n%d-%dx%d-%dto%d-d%d" % s)
def test_sepconv_block_on_the_tensor_pipe(shape):
    n, h, w, cin, cout, dil = shape
    buf = C.create_string_buffer(512)
    assert nat.load().pn_sepconv_describe(n, h, w, cin, cout, 1, dil, buf, 512) == 0
    assert b"tensor-pipe depthwise" in buf.value, buf.value
    g = torch.Generator().manual_seed(h * 7 + cin + dil)
    x = (torch.rand((n, h, w, cin), generator=g) * 6).to(torch.bfloat16)
    wd = torch.randn((cin, 1, 3, 3), generator=g) * 0.35
    bd = torch.randn(cin, generator=g) * 0.3
    wp = (torch.randn((cout, cin), generator=g) * (1.5 / cin ** 0.5)).to(torch.bfloat16)
    bp = torch.randn(cout, generator=g) * 0.5
    t = F.relu6(F.conv2d(x.float().permute(0, 3, 1, 2), wd.to(torch.bfloat16).float(), bd, padding=dil, dilation=dil, groups=cin))
    t = t.to(torch.bfloat16).float()
    ref = F.relu6(F.conv2d(t, wp.float().reshape(cout, cin, 1, 1), bp)).permute(0, 2, 3, 1)
    w9 = wd.reshape(cin, 9).t().contiguous().to(DEV)
    y = torch.full((n, h, w, cout), float("nan"), dtype=torch.bfloat16, device=DEV)
    xd, bdd, wpd, bpd = x.to(DEV), bd.to(DEV), wp.to(DEV), bp.to(DEV)
    nat.check(nat.load().pn_sepconv_block(P(xd), P(w9), P(bdd), P(wpd), P(bpd), P(y), n, h, w, cin, cout, 1, dil, nat.stream_ptr()),
              "pn_sepconv_block")
    torch.cuda.synchronize()
    yf = y.float().cpu()
    assert not torch.isnan(yf).any(), "%d output cells never written" % int(torch.isnan(yf).sum())
    err = float((yf - ref).abs().max() / ref.abs().max())
    assert err < 6e-3, err                                   # one bf16 output rounding + rare 1-ulp flips of the intermediate
    y2 = abi.sepconv(xd, w9, bdd, wpd, bpd, 1, dil)
    assert torch.equal(y, y2)                                # deterministic


def test_tensor_pipe_takes_the_256_blocks_only():
    """Only the 256 -> 256 blocks (where it measured faster) take the tensor-pipe depthwise."""
    buf = C.create_string_buffer(512)
    assert nat.load().pn_sepconv_describe(2, 33, 33, 512, 512, 1, 1, buf, 512) == 0 and b"tensor-pipe" not in buf.value
    assert nat.load().pn_sepconv_describe(2, 91, 161, 256, 256, 1, 2, buf, 512) == 0 and b"tensor-pipe" in buf.value
