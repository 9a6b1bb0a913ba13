"""Per-kernel parity on the B200, through the C ABI: preprocess (bit-exact vs the oracle / cv2
golden), stem, depthwise, fp32 GEMM and fp32 heads vs plain torch fp32 references."""
import hashlib
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import abi  # noqa: E402
import sepref  # noqa: E402
from golden.make_golden_cases import PRE_CASES  # noqa: E402
from oracle import preprocess as opre  # noqa: E402
from oracle import synth  # noqa: E402
from posenet import _native as nat  # noqa: E402

DEV = "cuda"


def rel_err(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


# ------------------------------------------------------------------------------------- P1
@pytest.mark.parametrize("i", range(len(PRE_CASES)))
def test_preprocess_bit_exact(golden_dir, i):
    h, w, sf, os_, seed, _ = PRE_CASES[i]
    g = np.load(os.path.join(golden_dir, "preprocess.npz"))
    img = synth.noise_image(h, w, seed)
    ref, _, _ = opre.process_input(img, sf, os_)
    tw, th = opre.valid_resolution(w * sf, h * sf, os_)
    out = abi.preprocess(torch.from_numpy(img).unsqueeze(0).to(DEV), th, tw).cpu().numpy()
    assert out.shape == ref.shape
    assert np.array_equal(out, ref), "max diff %g, %d cells" % (np.abs(out - ref).max(), (out != ref).sum())
    # and against the reference's own output (cv2) recorded in the golden file
    assert hashlib.sha256(out.tobytes()).hexdigest() == str(g["sha_%d" % i])


@pytest.mark.parametrize("i", range(len(PRE_CASES)))
def test_resize_u8_bit_exact(i):
    """pn_resize_u8 = the resize stage of P1 alone (cv2.resize INTER_LINEAR on uint8, utils.py:21), uint8 in / uint8 out."""
    h, w, sf, os_, seed, _ = PRE_CASES[i]
    img = synth.noise_image(h, w, seed)
    tw, th = opre.valid_resolution(w * sf, h * sf, os_)
    ref = opre.resize_linear_u8(img, tw, th)
    out = abi.resize_u8(torch.from_numpy(np.stack([img, img[::-1].copy()])).to(DEV), th, tw).cpu().numpy()
    assert np.array_equal(out[0], ref)
    assert np.array_equal(out[1], opre.resize_linear_u8(img[::-1].copy(), tw, th))


def test_preprocess_batch():
    imgs = np.stack([synth.noise_image(120, 200, s) for s in range(3)])
    tw, th = opre.valid_resolution(200 * 0.8, 120 * 0.8, 8)
    out = abi.preprocess(torch.from_numpy(imgs).to(DEV), th, tw).cpu().numpy()
    for b in range(3):
        assert np.array_equal(out[b], opre.process_input(imgs[b], 0.8, 8)[0][0])


# ------------------------------------------------------------------------------------- B2
@pytest.mark.parametrize("cout", [16, 24, 32])
@pytest.mark.parametrize("dtype", [nat.PN_F32, nat.PN_BF16])
def test_stem(cout, dtype):
    torch.manual_seed(cout)
    n, h, w = 2, 65, 97
    x = torch.rand(n, 3, h, w) * 2 - 1
    wt = torch.randn(cout, 3, 3, 3) * 0.5
    b = torch.randn(cout) * 0.5
    ref = F.relu6(F.conv2d(x, wt, b, stride=2, padding=1)).permute(0, 2, 3, 1)
    w27 = wt.permute(2, 3, 1, 0).reshape(27, cout).contiguous()
    y = abi.stem(x.to(DEV), w27.to(DEV), b.to(DEV), 2, dtype).float().cpu()
    assert y.shape == ref.shape
    assert (ref == 6).any() and (ref == 0).any()
    assert rel_err(y, ref) < (1e-5 if dtype == nat.PN_F32 else 5e-3)


def test_stem_u8_equals_preprocess_then_stem():
    img = np.stack([synth.noise_image(49, 81, s) for s in range(2)])
    torch.manual_seed(0)
    wt, b = torch.randn(32, 3, 3, 3) * 0.3, torch.randn(32) * 0.1
    w27 = wt.permute(2, 3, 1, 0).reshape(27, 32).contiguous().to(DEV)
    d = torch.from_numpy(img).to(DEV)
    x = abi.preprocess(d, 49, 81)
    y1 = abi.stem(x, w27, b.to(DEV), 2, nat.PN_F32)
    y2 = abi.stem(d, w27, b.to(DEV), 2, nat.PN_F32, u8=True)
    assert torch.equal(y1, y2)


@pytest.mark.parametrize("cout,n,h,w", [(32, 2, 513, 513), (16, 1, 721, 1281), (24, 3, 257, 257), (32, 5, 33, 47), (16, 2, 7, 5),
                                        (32, 1, 1, 1), (24, 4, 2, 300), (32, 3, 129, 64), (16, 1, 64, 2049),
                                        # segmented spans (wide images) with a ragged batch tail / tiles that straddle rows and images
                                        (24, 3, 9, 515), (16, 2, 3, 1283), (32, 5, 4, 259), (16, 1, 3, 6401)])
def test_stem_u8_tensor_core(cout, n, h, w):
    """Production stem: uint8 BGR image -> bf16 NHWC through the tcgen05 im2col GEMM (normalisation folded into
    the operands) against normalise-then-conv in fp32 (utils.py:23 + mobilenet_v1.py:47-54)."""
    rng = np.random.default_rng(cout + h)
    img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    img[0, :, :1] = 255                                           # saturated borders: padding must contribute exactly 0
    img[-1, -1:, :] = 0
    torch.manual_seed(cout)
    wt, b = torch.randn(cout, 3, 3, 3) * 0.25, torch.randn(cout) * 0.3
    x = torch.from_numpy(img[..., ::-1].copy()).permute(0, 3, 1, 2).float() * (2.0 / 255.0) - 1.0
    ref = F.relu6(F.conv2d(x, wt, b, stride=2, padding=1)).permute(0, 2, 3, 1)
    w27 = wt.permute(2, 3, 1, 0).reshape(27, cout).contiguous().to(DEV)
    y = abi.stem(torch.from_numpy(img).to(DEV), w27, b.to(DEV), 2, nat.PN_BF16, u8=True)
    torch.cuda.synchronize()
    y = y.float().cpu()
    assert y.shape == ref.shape, (y.shape, ref.shape)
    assert rel_err(y, ref) < 8e-3
    assert float((y - ref).abs().mean()) < 3e-3 * float(ref.abs().mean() + 1e-3)
    y2 = abi.stem(torch.from_numpy(img).to(DEV), w27, b.to(DEV), 2, nat.PN_BF16, u8=True).float().cpu()
    assert torch.equal(y, y2)
    # the two ways of staging the input (whole rows / per-row column segments, the latter for images too wide for whole rows) feed
    # the same im2col: same bits
    if (w + 2 - 3) // 2 + 1 >= 128:
        os.environ["PN_STEM_SEGMENTS"] = "1"
        try:
            y3 = abi.stem(torch.from_numpy(img).to(DEV), w27, b.to(DEV), 2, nat.PN_BF16, u8=True).float().cpu()
        finally:
            del os.environ["PN_STEM_SEGMENTS"]
        assert torch.equal(y, y3)
    # ring depth and CTAs per SM do not change the result either
    rows_only = {"PN_STEM_SEGMENTS": "0"} if w < 2000 else {}     # (wider images do not fit whole rows: forbidding segments = SIMT kernel)
    for env in (dict(rows_only, PN_STEM_NBUF="2"), {"PN_STEM_NBUF": "3"}, {"PN_STEM_NBUF": "4", "PN_STEM_CTAS": "1"}):
        os.environ.update(env)
        try:
            y4 = abi.stem(torch.from_numpy(img).to(DEV), w27, b.to(DEV), 2, nat.PN_BF16, u8=True).float().cpu()
        finally:
            for k in env:
                del os.environ[k]
        assert torch.equal(y, y4), env


# ------------------------------------------------------------------------------------- B3
@pytest.mark.parametrize("c,stride,dil,h,w", [(32, 1, 1, 33, 47), (64, 2, 1, 33, 47), (128, 2, 1, 32, 32), (256, 1, 2, 17, 23),
                                              (256, 1, 4, 19, 19), (24, 1, 1, 9, 9), (48, 2, 1, 65, 65), (512, 1, 1, 33, 33),
                                              (1024, 1, 2, 33, 33), (16, 1, 1, 5, 3), (8, 1, 1, 1, 1),
                                              # real layer shapes (tile search on odd maps) + a dilation without a TMA instantiation
                                              (32, 1, 1, 257, 257), (64, 2, 1, 257, 257), (128, 1, 1, 129, 129), (96, 1, 1, 65, 65),
                                              (192, 2, 1, 33, 33), (384, 1, 1, 17, 17), (16, 2, 1, 361, 641), (40, 1, 3, 20, 20)])
@pytest.mark.parametrize("dtype", [nat.PN_F32, nat.PN_BF16])
def test_dwconv(c, stride, dil, h, w, dtype):
    torch.manual_seed(c + stride + dil)
    n = 2
    tdt = abi.TORCH_DT[dtype]
    x = (torch.rand(n, c, h, w) * 8 - 2).to(tdt).float()          # values exactly representable in the storage dtype
    wt = torch.randn(c, 1, 3, 3) * 0.4
    b = torch.randn(c) * 0.5
    pad = ((stride - 1) + 2 * dil) // 2
    ref = F.relu6(F.conv2d(x, wt, b, stride=stride, padding=pad, dilation=dil, groups=c)).permute(0, 2, 3, 1)
    w9 = wt.reshape(c, 9).t().contiguous()
    xin = x.permute(0, 2, 3, 1).contiguous().to(tdt).to(DEV)
    y = abi.dwconv(xin, w9.to(DEV), b.to(DEV), stride, dil, dtype).float().cpu()
    assert y.shape == ref.shape, (y.shape, ref.shape)
    if dtype == nat.PN_F32:
        assert rel_err(y, ref) < 2e-6
    else:
        # every cell equal to the fp64 result rounded to bf16, or one ulp off where the fp32 sum may round the other way
        t, u = sepref.depthwise(x.permute(0, 2, 3, 1).to(tdt), w9, b, stride, dil)
        assert not torch.isnan(y).any()
        bad = (y.double() - t).abs() > u
        assert not bad.any(), "%d cells outside the bound, first %s" % (int(bad.sum()), tuple(bad.nonzero()[0].tolist()))


# ------------------------------------------------------------------------------------- B4 / H1 (fp32)
@pytest.mark.parametrize("m,k,n", [(1089, 512, 512), (300, 24, 48), (129, 32, 64), (1, 1024, 1024), (4225, 128, 256), (77, 384, 384)])
def test_gemm_fp32(m, k, n):
    torch.manual_seed(m)
    a = torch.rand(m, k) * 6
    w = torch.randn(n, k) / k ** 0.5
    b = torch.randn(n)
    ref = (a.double() @ w.double().t() + b.double()).clamp(0, 6).float()
    y = abi.pwconv(a.to(DEV), w.to(DEV), b.to(DEV), nat.PN_F32).cpu()
    assert rel_err(y, ref) < 2e-6


@pytest.mark.parametrize("n_img,hw,k", [(2, 33 * 33, 1024), (3, 17 * 17, 384), (1, 5, 256)])
def test_heads_fp32(n_img, hw, k):
    torch.manual_seed(hw)
    a = torch.rand(n_img * hw, k) * 3
    w = torch.zeros(128, k)
    w[:115] = torch.randn(115, k) / k ** 0.5 * 3
    b = torch.zeros(128)
    b[:115] = torch.randn(115)
    outs = abi.heads(a.to(DEV), w.to(DEV), b.to(DEV), n_img, hw, nat.PN_F32)
    z = (a.double() @ w.double().t() + b.double()).float().reshape(n_img, hw, 128).permute(0, 2, 1)
    refs = [torch.sigmoid(z[:, :17]), z[:, 17:51], z[:, 51:83], z[:, 83:115]]
    for o, r in zip(outs, refs):
        o = o.cpu()
        assert not torch.isnan(o).any()
        assert rel_err(o, r) < 5e-6
