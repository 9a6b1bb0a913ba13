"""Fused SeperableConv block (pn_sepconv_block: depthwise 3x3 -> pointwise 1x1 in one kernel, the
depthwise result staying in shared memory) on the B200, through the C ABI.

Three checks per shape: (1) against a plain torch fp32 reference of the two convolutions with the
bf16 rounding points the kernel has (input, depthwise output, output); (2) against the two-kernel
path of this library (pn_dwconv3x3 + pn_pwconv_gemm), which does the same arithmetic in the same
order -> equal up to one bf16 ulp on a vanishing fraction of cells; (3) determinism."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import abi  # noqa: E402
import posenet  # noqa: E402
from oracle import net as onet  # noqa: E402
from posenet import _native as nat  # noqa: E402

DEV = "cuda"

SHAPES = [  # n, h, w, cin, cout, stride, dilation
    # the blocks of model 101 @ 513x513 OS16 (config 2), small batch
    (2, 257, 257, 32, 64, 1, 1), (2, 257, 257, 64, 128, 2, 1), (2, 129, 129, 128, 128, 1, 1), (2, 129, 129, 128, 256, 2, 1),
    (2, 65, 65, 256, 256, 1, 1), (2, 65, 65, 256, 512, 2, 1), (3, 33, 33, 512, 512, 1, 1), (2, 33, 33, 512, 1024, 1, 1),
    (2, 33, 33, 1024, 1024, 1, 2),
    # model 50 @ OS8 (config 3 geometry, reduced) incl. cin 16 / 32 with stride 2, and dilation 2
    (1, 91, 161, 16, 32, 1, 1), (1, 361, 641, 16, 32, 1, 1), (2, 37, 53, 16, 48, 1, 1), (1, 91, 161, 32, 64, 2, 1), (1, 46, 81, 64, 64, 1, 1), (1, 46, 81, 128, 256, 1, 1),
    (1, 46, 81, 256, 256, 1, 2),
    # stride 2 on the warp-autonomous path (cin 17..32): the real frame size, even / odd / degenerate maps, ragged cout
    (1, 361, 641, 32, 64, 2, 1), (2, 38, 54, 24, 48, 2, 1), (3, 9, 9, 32, 32, 2, 1), (1, 2, 2, 32, 64, 2, 1), (1, 1, 1, 32, 64, 2, 1),
    # model 75 (config 4): channel counts that are not multiples of 64 (ragged K and N tiles)
    (3, 129, 129, 24, 48, 1, 1), (3, 129, 129, 48, 96, 2, 1), (3, 65, 65, 96, 96, 1, 1), (3, 65, 65, 96, 192, 2, 1),
    (3, 33, 33, 192, 384, 2, 1), (5, 17, 17, 384, 384, 1, 1),
    # full-warp layout of the warp-autonomous kernel (48 -> 96 stride 2): ragged strips / rows, degenerate maps
    (1, 181, 321, 64, 64, 1, 1), (2, 7, 5, 48, 96, 2, 1), (2, 6, 10, 64, 64, 1, 1), (1, 1, 1, 48, 96, 2, 1), (1, 2, 3, 48, 96, 2, 1),
    # model 101 @ OS8: dilation 4; tiny and degenerate maps
    (1, 33, 33, 1024, 1024, 1, 4), (2, 5, 3, 64, 64, 1, 1), (1, 1, 1, 32, 64, 1, 1), (1, 2, 2, 64, 128, 2, 1), (4, 9, 9, 8, 16, 1, 1),
    # cin <= 32 at stride 1 wider than the warp-autonomous kernel takes: the CTA pipeline's half-warp layout
    (1, 33, 33, 32, 128, 1, 1),
]


def make(n, h, w, cin, cout, seed):
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand((n, h, w, cin), generator=g) * 6).to(torch.bfloat16)            # post-ReLU6-like input
    wd = torch.randn((cin, 1, 3, 3), generator=g) * 0.35
    bd = torch.randn(cin, generator=g) * 0.3
    wp = (torch.randn((cout, cin), generator=g) * (1.5 / cin ** 0.5)).to(torch.bfloat16)
    bp = torch.randn(cout, generator=g) * 0.5
    return x, wd, bd, wp, bp


@pytest.mark.parametrize("shape", SHAPES)
def test_sepconv_block(shape):
    n, h, w, cin, cout, stride, dil = shape
    x, wd, bd, wp, bp = make(n, h, w, cin, cout, seed=h * 7 + cin + stride + dil)
    pad = ((stride - 1) + 2 * dil) // 2
    # 256 -> 256 blocks run the depthwise on the tensor pipe by default (csrc/septc.cu): its depthwise weights are bf16
    import ctypes as C
    buf = C.create_string_buffer(512)
    assert nat.load().pn_sepconv_describe(n, h, w, cin, cout, stride, dil, buf, 512) == 0
    tensor_pipe = b"tensor-pipe" in buf.value
    assert tensor_pipe == (cin == 256 and cout == 256 and stride == 1 and dil <= 2)
    wd_k = wd.to(torch.bfloat16).float() if tensor_pipe else wd
    # torch fp32 reference with the kernel's rounding points
    t = F.relu6(F.conv2d(x.float().permute(0, 3, 1, 2), wd_k, bd, stride=stride, padding=pad, dilation=dil, groups=cin))
    t = t.to(torch.bfloat16).float()
    ref = F.relu6(F.conv2d(t, wp.float().reshape(cout, cin, 1, 1), bp)).permute(0, 2, 3, 1)

    w9 = wd.reshape(cin, 9).t().contiguous().to(DEV)
    xd, bdd, wpd, bpd = x.to(DEV), bd.to(DEV), wp.to(DEV), bp.to(DEV)
    y = abi.sepconv(xd, w9, bdd, wpd, bpd, stride, dil)
    torch.cuda.synchronize()
    yf = y.float().cpu()
    assert yf.shape == ref.shape, (yf.shape, ref.shape)
    assert not torch.isnan(yf).any(), "%d output cells never written" % int(torch.isnan(yf).sum())
    err = float((yf - ref).abs().max() / ref.abs().max().clamp_min(1e-6))
    assert err < 1.2e-2, err                      # one bf16 output rounding + rare 1-ulp flips of the intermediate

    # the two-kernel path: same math, same order
    t2 = abi.dwconv(xd, w9, bdd, stride, dil, nat.PN_BF16)
    y2 = abi.pwconv(t2.reshape(-1, cin), wpd, bpd, nat.PN_BF16).reshape(y.shape)
    diff = (y.float() - y2.float()).abs()
    if tensor_pipe:                                                             # fp32 vs bf16 depthwise weights: a few ulps
        assert float(diff.max() / y2.float().abs().max()) < 1.5e-2
    else:
        assert float(diff.max()) <= 0.0625, float(diff.max())                   # <= 1 bf16 ulp at magnitude <= 6
        assert float((diff > 0).float().mean()) < 1e-3

    y3 = abi.sepconv(xd, w9, bdd, wpd, bpd, stride, dil)
    assert torch.equal(y, y3)


def test_sepconv_rejects_unsupported():
    x, wd, bd, wp, bp = make(1, 8, 8, 64, 64, 0)
    w9 = wd.reshape(64, 9).t().contiguous().to(DEV)
    with pytest.raises(nat.NativeError):
        abi.sepconv(x.to(DEV), w9, bd.to(DEV), wp.to(DEV), bp.to(DEV), 2, 2)        # stride 2 with dilation: never produced
    with pytest.raises(nat.NativeError):
        abi.sepconv(x.to(DEV), w9, bd.to(DEV), wp[:24].contiguous().to(DEV), bp[:24].contiguous().to(DEV), 1, 3)


@pytest.mark.parametrize("mid,os_,H,W,N", [(101, 16, 513, 513, 2), (50, 8, 193, 257, 1), (75, 32, 257, 257, 3), (101, 8, 129, 129, 1)])
def test_fused_plan_matches_unfused_plan(mid, os_, H, W, N):
    """Whole network: the fused plan (15 launches + 1 per block wider than 512) against the two-kernel-per-block plan (28)."""
    sd = onet.init_params(mid, seed=3)
    m = posenet.MobileNetV1(mid, output_stride=os_)
    m.load_state_dict(sd)
    m = m.cuda().set_compute_dtype("bf16")
    x = torch.rand((N, 3, H, W), generator=torch.Generator().manual_seed(1)) * 2 - 1
    fused = [t.clone() for t in m.set_fused(True)(x.to(DEV))]
    n_fused = m.num_launches(N, H, W)
    unfused = m.set_fused(False)(x.to(DEV))
    n_unfused = m.num_launches(N, H, W)
    wide = sum(1 for L in m._layers[1:] if L["outp"] > 512)      # blocks wider than one 512-column tile stay two kernels
    assert (n_fused, n_unfused) == (15 + wide, 28)
    # blocks with 256 -> 256 channels take the tensor-pipe depthwise, whose depthwise weights are rounded to bf16
    tc_blocks = sum(1 for L in m._layers[1:] if L["inp"] == 256 and L["outp"] == 256 and L["stride"] == 1 and L["rate"] <= 2)
    for a, b in zip(fused, unfused):
        err = float((a - b).abs().max() / b.abs().max())
        print("fused vs unfused: model %d, %d tensor-pipe blocks, err %.3g" % (mid, tc_blocks, err))
        assert err < (6e-3 if tc_blocks else 2e-3), err

