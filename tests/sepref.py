"""fp64 reference of the fused separable block and a per-cell error bound for it (no GPU needed).

The block is  y = bf16(relu6(pw(t) + b_pw)),  t = bf16(relu6(dw3x3(x) + b_dw))  with the kernel's operands: bf16 input, fp32
depthwise weights and bias (bf16-rounded weights on the tensor-pipe depthwise), bf16 pointwise weights, fp32 pointwise bias.

The bound follows the rounding points instead of max|ref|, so one wrong cell anywhere in the map fails it:
  * depthwise: an fp32 sum of 10 terms is within delta = 10 eps (sum|x w| + |b|) of the exact sum (eps = 2^-24 for the FMA chain of
    the CUDA cores).  Rounding is monotone, so the kernel's intermediate lies in [r(d - delta), r(d + delta)], r = bf16 o relu6:
    equal to the reference's bf16 value unless a rounding midpoint is that close, then one ulp off (several only where ulps are
    smaller than delta, next to 0).  u = that distance, at least delta.
  * pointwise: E = sum_c |wp| u + K eps_pw (sum_c |wp t| + |b_pw|), eps_pw = 2^-22 (4x the textbook unit roundoff, for the tensor
    core's accumulation; test_gpu_sepconv_configs.py measures it: 1.93 x 2^-24 sum|a w| at K = 64 on a B200 at 1000 W, far inside).
  * output: |y - ref| <= E + ulp_bf16(|ref| + E) / 2  (ReLU6 is 1-Lipschitz; then one bf16 rounding).
"""
import os
import re

import torch
import torch.nn.functional as F

EPS_FMA = 2.0 ** -24          # fp32 unit roundoff: the depthwise FMA chain of the CUDA cores
EPS_TC = 2.0 ** -22           # tensor-core fp32 accumulation (pointwise MMAs; the tensor-pipe depthwise)


def conv_out(n, stride, dil):
    pad = ((stride - 1) + 2 * dil) // 2
    return (n + 2 * pad - 2 * dil - 1) // stride + 1


def make_case(n, h, w, cin, cout, seed):
    """Seeded operands in the kernel's layouts: x NHWC bf16 (post-ReLU6-like, with exact 0.0 and 6.0), w9 [9, cin] fp32 (tap
    ky * 3 + kx), b_dw [cin] fp32, w_pw [cout, cin] bf16, b_pw [cout] fp32."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((n, h, w, cin), generator=g) * 6
    m = torch.rand((n, h, w, cin), generator=g)
    x[m < 0.06] = 0.0
    x[m > 0.94] = 6.0
    w9 = torch.randn((9, cin), generator=g) * 0.35
    bd = torch.randn(cin, generator=g) * 0.3
    wp = (torch.randn((cout, cin), generator=g) * (1.5 / cin ** 0.5)).to(torch.bfloat16)
    bp = torch.randn(cout, generator=g) * 0.5
    bp[0] += 8.0                           # channel 0 sits at the upper clamp almost everywhere, even on 1 x 1 maps
    return x.to(torch.bfloat16), w9, bd, wp, bp


def _bf16(v):
    """fp64 -> the nearest bf16 value (as fp64); monotone, which is all the interval argument needs."""
    return v.float().to(torch.bfloat16).double()


def ulp_bf16(v):
    """bf16 ulp at |v| (fp64 tensor): 2^(e - 7) for 2^e <= |v| < 2^(e + 1); the subnormal spacing below 2^-126."""
    _, e = torch.frexp(v.abs())
    return torch.ldexp(torch.ones_like(v), (e - 8).clamp_min(-133))


def depthwise(x, w9, bd, stride, dil, dw_bf16=False, eps=EPS_FMA):
    """Reference intermediate t (bf16 values, fp64, NHWC) and its per-cell deviation bound u."""
    cin = x.shape[-1]
    pad = ((stride - 1) + 2 * dil) // 2
    xd = x.double().permute(0, 3, 1, 2)
    wk = (w9.to(torch.bfloat16) if dw_bf16 else w9).double().t().reshape(cin, 1, 3, 3)
    b = bd.double()
    conv = lambda a, wt, bb: F.conv2d(a, wt, bb, stride=stride, padding=pad, dilation=dil, groups=cin)
    d = conv(xd, wk, b)
    delta = 10 * eps * conv(xd.abs(), wk.abs(), b.abs())
    r = lambda v: _bf16(v.clamp(0, 6))
    t, lo, hi = r(d), r(d - delta), r(d + delta)
    u = torch.maximum(torch.maximum(hi - t, t - lo), delta)
    return t.permute(0, 2, 3, 1).contiguous(), u.permute(0, 2, 3, 1).contiguous()


def reference(x, w9, bd, wp, bp, stride, dil, dw_bf16=False, dw_eps=EPS_FMA, pw_eps=EPS_TC):
    """fp64 output (NHWC, before the final bf16 rounding) and the per-cell bound."""
    t, u = depthwise(x, w9, bd, stride, dil, dw_bf16, dw_eps)
    n, ho, wo, cin = t.shape
    W, b = wp.double(), bp.double()
    tt, uu = t.reshape(-1, cin), u.reshape(-1, cin)
    s = tt @ W.t() + b
    e = uu @ W.abs().t() + cin * pw_eps * (tt.abs() @ W.abs().t() + b.abs())
    ref = s.clamp(0, 6)
    bound = e + 0.5 * ulp_bf16(ref + e)
    return ref.reshape(n, ho, wo, -1), bound.reshape(n, ho, wo, -1)


def check(y, ref, bound, what="", saturates=True):
    """Every cell within its bound, none NaN; returns max |y - ref| / bound.  With `saturates` the output must also reach the
    clamps (exact 0 and exact 6), as ReLU6 blocks do."""
    yd = y.detach().double().cpu()
    assert yd.shape == ref.shape, (what, tuple(yd.shape), tuple(ref.shape))
    nan = torch.isnan(yd)
    assert not nan.any(), "%s: %d output cells never written, first at %s" % (what, int(nan.sum()), tuple(nan.nonzero()[0].tolist()))
    err = (yd - ref).abs()
    bad = err > bound
    if bad.any():
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError("%s: %d of %d cells outside the bound; first (n, y, x, c) = %s: got %.8g ref %.8g bound %.3g"
                             % (what, int(bad.sum()), bad.numel(), i, float(yd[i]), float(ref[i]), float(bound[i])))
    if saturates:
        assert (yd == 0).any() and (yd == 6).any(), "%s: the output never reaches 0 and 6" % what
    return float((err / bound).max())


# ---- the kernel's arithmetic, restated in torch fp32 (for the CPU test of the checker) --------------------------------------
def emulate_depthwise(x, w9, bd, stride, dil, dw_bf16=False, drop=None):
    """Bias first, then the nine taps in order ky * 3 + kx, each one fp32 FMA (exact product + add, rounded once), + ReLU6 ->
    bf16; `drop` = (image, row, col, tap) skips that tap at that pixel (all channels)."""
    n, h, w, cin = x.shape
    pad = ((stride - 1) + 2 * dil) // 2
    ho, wo = conv_out(h, stride, dil), conv_out(w, stride, dil)
    xp = F.pad(x.float().permute(0, 3, 1, 2), (pad, pad, pad, pad))
    wk = (w9.to(torch.bfloat16).float() if dw_bf16 else w9.float())
    acc = bd.float().reshape(1, cin, 1, 1).expand(n, cin, ho, wo).contiguous()
    for tap in range(9):
        ky, kx = divmod(tap, 3)
        sl = xp[:, :, ky * dil: ky * dil + (ho - 1) * stride + 1: stride, kx * dil: kx * dil + (wo - 1) * stride + 1: stride]
        new = (acc.double() + sl.double() * wk[tap].double().reshape(1, cin, 1, 1)).float()
        if drop is not None and drop[3] == tap:
            new[drop[0], :, drop[1], drop[2]] = acc[drop[0], :, drop[1], drop[2]]
        acc = new
    return acc.clamp(0, 6).to(torch.bfloat16).permute(0, 2, 3, 1).contiguous()


def emulate_pointwise(t, wp, bp):
    """fp32 accumulation of the exact bf16 products, + bias in fp32, ReLU6 -> bf16."""
    n, ho, wo, cin = t.shape
    s = t.float().reshape(-1, cin) @ wp.float().t() + bp.float()
    return s.clamp(0, 6).to(torch.bfloat16).reshape(n, ho, wo, -1)


def emulate(x, w9, bd, wp, bp, stride, dil, dw_bf16=False):
    return emulate_pointwise(emulate_depthwise(x, w9, bd, stride, dil, dw_bf16), wp, bp)


# ---- configurations of the CTA-pipeline kernel (csrc/sepconv.cu) ------------------------------------------------------------
DESCRIBE = re.compile(r"(half )?tile (\d+)x(\d+) subs (\d+) .* n_tile (\d+)\((\d+)x(\d+)\) x(\d+) kblocks (\d+) teams (\d+) "
                      r"stages p(\d+) w(\d+)(r?) a(\d+) stg(\d+) smem \d+ tiles (\d+)")
ENV = ("PN_SEP_TILE", "PN_SEP_STAGES", "PN_SEP_TEAMS")


def parse_describe(s):
    m = DESCRIBE.search(s)
    assert m, s
    v = m.groups()
    i = [int(a) for a in v[1:12]]
    return dict(half=bool(v[0]), th=i[0], tw=i[1], subs=i[2], n_tile=i[3], n_halves=i[4], n_half=i[5], n_tiles=i[6], kblocks=i[7],
                teams=i[8], p=i[9], w=i[10], w_res=bool(v[12]), a=int(v[13]), stg=int(v[14]), tiles=int(v[15]))


def config_env(cfg):
    """'th,tw,subs;p,w,a,stg;teams' (empty parts: not forced) -> {env var: value or None}."""
    return dict(zip(ENV, [p or None for p in cfg.split(";")]))


def config_honoured(cfg, d):
    """The described geometry `d` (parse_describe) equals every forced value of `cfg`."""
    tile, stages, teams = cfg.split(";")
    ok = True
    if tile:
        ok &= [int(v) for v in tile.split(",")] == [d["th"], d["tw"], d["subs"]]
    if stages:
        ok &= [int(v) for v in stages.split(",")] == [d["p"], d["w"], d["a"], d["stg"]]
    if teams:
        ok &= int(teams) == d["teams"]
    return ok


def tuned_rows():
    """csrc/sep_tuned.inc as tuples (cin, cout, stride, dilation, ho, wo, th, tw, subs, p, w, a, stg, teams)."""
    inc = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "posenet-pytorch_b200", "csrc", "sep_tuned.inc")
    return [tuple(int(v) for v in m.group(1).split(",")) for m in re.finditer(r"^\s*\{([\d, ]+)\}", open(inc).read(), re.M)]


# Representative blocks at small maps (n, h, w, cin, cout, stride, dilation), all on the CTA pipeline: the half-warp layout with
# ragged K and N (24 -> 96), stride 2 (64 -> 128, 96 -> 192 ragged K, 16 -> 32), double-buffered accumulators (128 / 256 wide),
# two column halves on one accumulator (192 -> 384 s2, 384 -> 384 with ringed depthwise weights), two n-tiles (512 -> 1024),
# dilation 4 and 2.
BLOCKS = [(2, 9, 11, 24, 96, 1, 1), (3, 23, 29, 64, 128, 2, 1), (2, 17, 19, 128, 128, 1, 1), (2, 13, 15, 128, 256, 1, 1),
          (2, 21, 23, 96, 192, 2, 1), (2, 13, 11, 192, 384, 2, 1), (3, 9, 9, 384, 384, 1, 1), (2, 9, 9, 512, 1024, 1, 1),
          (1, 11, 11, 256, 256, 1, 4), (1, 12, 13, 512, 512, 1, 2), (2, 15, 17, 16, 32, 2, 1)]

# Forced configurations per block, 'th,tw,subs;p,w,a,stg;teams'.  Drawn once with random.Random(2026) from what the host geometry
# accepted: a one-row, a one-column, a taller-than-the-map and a wider-than-the-map tile, one tile of each of 2-4 sub-tiles, four
# more tiles (default rings), then at the default tile and at the tile with the most sub-tiles one ring / team combination for each
# of stg 0-2 x teams 1-2, one with resident and one with ringed pointwise weights.  Written out so that a failure names one
# configuration and a change of the host geometry shows up in the CPU test, not as a different sweep.
SWEEP = {
    (2, 9, 11, 24, 96, 1, 1): [
        "1,4,1;;", "8,1,2;;", "16,6,2;;", "7,18,3;;", "12,6,2;;", "5,9,3;;",
        "16,3,4;;", "6,5,3;;", "14,2,3;;", "14,8,1;;", "12,10,1;;", "9,11,1;5,4,4,0;1",
        "9,11,1;6,3,5,0;2", "9,11,1;6,5,3,1;1", "9,11,1;6,1,4,1;2", "9,11,1;5,6,3,2;1", "9,11,1;4,5,2,2;2", "9,11,1;2,1,2,0;1",
        "9,11,1;2,6,4,1;1", "16,3,4;5,2,4,0;1", "16,3,4;5,4,5,1;1", "16,3,4;6,5,4,2;1", "16,3,4;5,1,3,0;1", "16,3,4;6,4,6,0;1",
    ],
    (3, 23, 29, 64, 128, 2, 1): [
        "1,1,1;;", "19,1,2;;", "18,3,2;;", "3,22,2;;", "4,11,2;;", "9,3,3;;",
        "10,9,4;;", "7,9,2;;", "7,11,4;;", "19,2,2;;", "7,17,1;;", "6,15,1;3,1,3,0;1",
        "6,15,1;2,2,2,0;2", "6,15,1;2,2,3,1;1", "6,15,1;2,1,2,1;2", "6,15,1;2,2,3,2;1", "6,15,1;2,3,2,2;2", "6,15,1;2,1,4,1;1",
        "6,15,1;2,3,2,0;1", "10,9,4;6,3,2,0;1", "10,9,4;5,1,6,1;1", "10,9,4;5,4,2,2;1", "10,9,4;5,1,2,0;1", "10,9,4;6,4,2,1;1",
    ],
    (2, 17, 19, 128, 128, 1, 1): [
        "1,12,1;;", "15,1,1;;", "22,5,3;;", "4,24,1;;", "3,21,2;;", "8,13,3;;",
        "20,3,4;;", "10,6,3;;", "9,3,2;;", "19,6,3;;", "3,15,1;;", "6,19,1;4,1,3,0;1",
        "6,19,1;4,6,2,0;2", "6,19,1;5,1,2,1;1", "6,19,1;4,3,4,1;2", "6,19,1;3,3,2,2;1", "6,19,1;3,2,2,2;2", "6,19,1;4,2,4,2;1",
        "6,19,1;5,4,3,0;1", "20,3,4;6,1,4,0;1", "20,3,4;6,1,6,1;1", "20,3,4;6,6,2,2;1", "20,3,4;5,2,2,0;1", "20,3,4;5,5,6,0;1",
    ],
    (2, 13, 15, 128, 256, 1, 1): [
        "1,5,1;;", "4,1,1;;", "20,1,1;;", "5,17,1;;", "17,4,2;;", "15,8,3;;",
        "7,5,4;;", "15,8,4;;", "13,2,1;;", "8,12,1;;", "9,8,3;;", "13,8,1;2,2,6,0;1",
        "13,8,1;4,2,3,0;2", "13,8,1;3,1,2,1;1", "13,8,1;2,4,2,1;2", "13,8,1;4,1,2,2;1", "13,8,1;5,1,3,2;2", "13,8,1;4,2,3,2;1",
        "13,8,1;3,3,3,0;1", "15,8,4;6,2,3,0;1", "15,8,4;6,1,5,1;1", "15,8,4;5,2,5,2;1", "15,8,4;6,2,3,2;1", "15,8,4;5,4,2,1;1",
    ],
    (2, 21, 23, 96, 192, 2, 1): [
        "1,10,1;;", "12,1,2;;", "18,3,2;;", "8,14,4;;", "13,5,2;;", "11,8,3;;",
        "14,9,4;;", "9,12,3;;", "5,13,2;;", "7,6,1;;", "6,17,3;;", "6,12,1;2,1,2,0;1",
        "6,12,1;2,1,2,0;2", "6,12,1;2,1,4,1;1", "6,12,1;3,2,2,1;2", "6,12,1;3,1,2,2;1", "6,12,1;3,1,2,2;2", "6,12,1;2,2,5,0;1",
        "6,12,1;2,1,6,0;1", "14,9,4;5,2,2,0;1", "14,9,4;6,1,2,1;1", "14,9,4;6,1,2,2;1", "14,9,4;5,2,3,1;1", "14,9,4;5,1,5,0;1",
    ],
    (2, 13, 11, 192, 384, 2, 1): [
        "1,13,1;;", "11,1,2;;", "13,6,2;;", "7,8,4;;", "2,9,2;;", "13,5,3;;",
        "8,13,4;;", "6,3,3;;", "7,12,1;;", "14,6,2;;", "12,7,4;;", "7,6,1;2,2,3,0;1",
        "7,6,1;4,1,4,0;2", "7,6,1;3,1,3,1;1", "7,6,1;4,2,3,1;2", "7,6,1;2,2,2,2;1", "7,6,1;3,2,2,2;2", "7,6,1;4,2,2,2;1",
        "12,7,4;5,1,4,0;1", "12,7,4;6,3,2,1;1", "12,7,4;5,2,2,2;1", "12,7,4;6,3,2,2;1",
    ],
    (3, 9, 9, 384, 384, 1, 1): [
        "1,16,1;;", "9,1,1;;", "11,1,2;;", "4,12,4;;", "16,8,2;;", "10,12,3;;",
        "7,4,4;;", "11,3,2;;", "1,15,1;;", "4,1,1;;", "1,1,1;;", "9,9,1;4,4,2,0;1",
        "9,9,1;5,3,3,0;2", "9,9,1;3,4,2,1;1", "9,9,1;3,1,2,1;2", "9,9,1;4,3,3,2;1", "9,9,1;6,1,2,2;2", "9,9,1;3,2,2,2;2",
        "7,4,4;5,4,2,0;1", "7,4,4;5,2,4,1;1", "7,4,4;5,1,4,2;1", "7,4,4;6,3,3,1;1",
    ],
    (2, 9, 9, 512, 1024, 1, 1): [
        "1,9,1;;", "14,1,1;;", "14,4,4;;", "3,16,1;;", "2,2,2;;", "9,1,3;;",
        "13,5,4;;", "14,7,4;;", "14,5,3;;", "12,2,3;;", "4,16,1;;", "9,9,1;4,1,6,0;1",
        "9,9,1;4,2,2,0;2", "9,9,1;4,2,2,1;1", "9,9,1;5,1,3,1;2", "9,9,1;2,2,5,2;1", "9,9,1;5,2,2,2;2", "9,9,1;3,2,2,1;1",
        "14,7,4;5,1,4,0;1", "14,7,4;6,1,4,1;1", "14,7,4;5,2,2,2;1", "14,7,4;5,2,3,1;1",
    ],
    (1, 11, 11, 256, 256, 1, 4): [
        "1,10,1;;", "11,1,3;;", "15,3,4;;", "4,17,2;;", "4,3,2;;", "8,5,3;;",
        "14,3,4;;", "1,16,1;;", "4,3,1;;", "10,10,2;;", "3,8,3;;", "11,11,1;2,1,2,0;1",
        "11,11,1;2,2,2,0;2", "11,11,1;2,1,4,1;1", "11,11,1;2,1,2,1;2", "11,11,1;2,1,2,2;1", "11,11,1;2,1,2,2;2", "11,11,1;2,1,4,0;1",
        "15,3,4;6,1,3,0;1", "15,3,4;5,2,2,1;1", "15,3,4;5,2,2,2;1", "15,3,4;5,1,5,1;1",
    ],
    (1, 12, 13, 512, 512, 1, 2): [
        "1,4,1;;", "19,1,2;;", "16,5,2;;", "5,18,3;;", "10,11,2;;", "6,7,3;;",
        "7,4,4;;", "13,7,1;;", "11,9,3;;", "5,13,1;;", "9,12,2;;", "6,13,1;6,1,3,0;1",
        "6,13,1;4,1,2,0;2", "6,13,1;3,1,5,1;1", "6,13,1;3,3,2,1;2", "6,13,1;2,1,4,2;1", "6,13,1;4,1,3,2;2", "6,13,1;4,2,2,0;2",
        "7,4,4;5,1,3,0;1", "7,4,4;5,2,3,1;1", "7,4,4;5,2,2,2;1", "7,4,4;5,1,4,0;1",
    ],
    (2, 15, 17, 16, 32, 2, 1): [
        "1,2,1;;", "10,1,3;;", "11,2,4;;", "7,14,3;;", "15,6,2;;", "3,6,3;;",
        "7,1,4;;", "13,2,4;;", "6,12,1;;", "12,9,4;;", "4,16,4;;", "8,9,1;2,3,2,0;1",
        "8,9,1;4,2,3,0;2", "8,9,1;2,3,3,1;1", "8,9,1;3,4,2,1;2", "8,9,1;2,4,4,2;1", "8,9,1;3,4,3,2;2", "8,9,1;3,1,5,1;1",
        "8,9,1;3,3,3,0;2", "13,2,4;6,6,2,0;1", "13,2,4;5,2,2,1;1", "13,2,4;5,5,6,2;1", "13,2,4;5,1,5,0;1", "13,2,4;5,5,3,0;1",
    ],
}
