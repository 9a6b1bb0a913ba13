"""The per-cell checker of the fused separable block (tests/sepref.py) and the forced-configuration sweep, on the CPU.

(1) The kernel's arithmetic restated in torch fp32 -- taps in order as FMAs, the block's bf16 rounding points, fp32 pointwise --
    passes the checker on every shape the GPU tests run.
(2) Subtly wrong outputs of that emulation fail it: one tap dropped at one pixel, one channel's depthwise bias missing, two
    intermediate channels swapped at one pixel, a dilated block reading undilated taps in its border rows, one output cell two
    ulps off, one cell never written.
(3) The sweep of tests/test_gpu_sepconv_configs.py is what the host geometry builds (a forced ring depth or team count that does
    not fit is ignored silently, so the sweep would test something else) and covers the kernel's switches."""
import ctypes as C

import pytest
import torch

import sepref
import test_gpu_sepconv
import test_gpu_septc
from posenet import _native as nat

TC = dict(dw_bf16=True, dw_eps=sepref.EPS_TC)          # tensor-pipe depthwise: bf16 weights, tensor-core accumulation


def _crop(n, h, w, seed, cells=40000):
    """The largest maps only: one image of a seeded smaller map of the same block (at most ~`cells` input pixels)."""
    if h * w <= cells:
        return n, h, w
    g = torch.Generator().manual_seed(seed)
    s = (cells / (h * w)) ** 0.5
    return min(n, 1), max(8, int(h * s) + int(torch.randint(0, 3, (1,), generator=g))), max(8, int(w * s))


CASES = [("sepconv", s) for s in test_gpu_sepconv.SHAPES] + [("septc", (n, h, w, ci, co, 1, d)) for (n, h, w, ci, co, d) in test_gpu_septc.SHAPES]


@pytest.mark.parametrize("kind,shape", CASES, ids=["%s-n%d-%dx%d-%dto%d-s%d-d%d" % ((k,) + s) for k, s in CASES])
def test_checker_accepts_the_kernel_arithmetic(kind, shape):
    n, h, w, cin, cout, s, d = shape
    n, h, w = _crop(n, h, w, seed=h + w)
    tc = kind == "septc" or (cin == 256 and cout == 256 and s == 1 and d <= 2)
    x, w9, bd, wp, bp = sepref.make_case(n, h, w, cin, cout, seed=h * 7 + cin + s + d)
    opt = TC if tc else {}
    y = sepref.emulate(x, w9, bd, wp, bp, s, d, dw_bf16=tc)
    ref, bound = sepref.reference(x, w9, bd, wp, bp, s, d, **opt)
    ratio = sepref.check(y, ref, bound, str(shape))
    assert ratio <= 1.0


MUT_SHAPE = (2, 17, 19, 64, 128, 1, 1)
MUT_SHAPE_D2 = (2, 12, 13, 64, 128, 1, 2)


def _old_check_passes(y, ref):
    """The max-relative assertion these blocks were checked with before (test_gpu_sepconv.py): no NaN and
    max|y - ref| / max|ref| < 1.2e-2."""
    yd = y.double()
    return not torch.isnan(yd).any() and float((yd - ref).abs().max() / ref.abs().max()) < 1.2e-2


def _mutant(name):
    shape = MUT_SHAPE_D2 if name == "dilation-1-border-rows" else MUT_SHAPE
    n, h, w, cin, cout, s, d = shape
    x, w9, bd, wp, bp = sepref.make_case(n, h, w, cin, cout, seed=11)
    ref, bound = sepref.reference(x, w9, bd, wp, bp, s, d)
    t = sepref.emulate_depthwise(x, w9, bd, s, d)
    y0 = sepref.emulate_pointwise(t, wp, bp)
    ho, wo = t.shape[1], t.shape[2]
    if name == "tap-dropped":                                    # centre tap of the last pixel of the last image
        y = sepref.emulate_pointwise(sepref.emulate_depthwise(x, w9, bd, s, d, drop=(n - 1, ho - 1, wo - 1, 4)), wp, bp)
    elif name == "dw-bias-missing-last-channel":
        b2 = bd.clone()
        b2[-1] = 0
        y = sepref.emulate_pointwise(sepref.emulate_depthwise(x, w9, b2, s, d), wp, bp)
    elif name == "channels-swapped":                             # the two adjacent channels that differ most at one pixel
        t2 = t.clone()
        px = t2[n - 1, ho // 2, wo // 2]
        c = int((px[1:].float() - px[:-1].float()).abs().argmax())
        px[[c, c + 1]] = px[[c + 1, c]]
        y = sepref.emulate_pointwise(t2, wp, bp)
    elif name == "dilation-1-border-rows":                      # rows within `d` of the top / bottom edge read distance-1 taps
        t1 = sepref.emulate_depthwise(x, w9, bd, s, 1)
        t2 = t.clone()
        rows = list(range(d)) + list(range(ho - d, ho))
        t2[:, rows] = t1[:, rows]
        y = sepref.emulate_pointwise(t2, wp, bp)
    elif name == "two-ulps-off":                                 # one unclamped cell of the last image
        y = y0.clone()
        yl = y[n - 1].double()
        i = ((yl >= 1) & (yl < 4)).nonzero()[-1]
        v = y[(n - 1,) + tuple(i.tolist())].double()
        y[(n - 1,) + tuple(i.tolist())] = (v + 2 * sepref.ulp_bf16(v)).to(torch.bfloat16)
    elif name == "cell-unwritten":
        y = y0.clone()
        y[n - 1, ho - 1, wo - 1, cout - 1] = float("nan")
    return y, y0, ref, bound


MUTATIONS = ["tap-dropped", "dw-bias-missing-last-channel", "channels-swapped", "dilation-1-border-rows", "two-ulps-off", "cell-unwritten"]


@pytest.mark.parametrize("name", MUTATIONS)
def test_checker_rejects_subtly_wrong_output(name):
    y, y0, ref, bound = _mutant(name)
    assert sepref.check(y0, ref, bound, "unmutated") <= 1.0
    assert not torch.equal(y, y0)
    with pytest.raises(AssertionError):
        sepref.check(y, ref, bound, name)
    print("%s: the max-relative check %s" % (name, "lets it through" if _old_check_passes(y, ref) else "rejects it"))


def test_every_table_row_is_parsed():
    import os
    inc = os.path.join(os.path.dirname(nat.__file__), "..", "csrc", "sep_tuned.inc")
    lines = [ln for ln in open(inc).read().splitlines() if ln.strip().startswith("{")]
    rows = sepref.tuned_rows()
    assert len(rows) == len(lines) >= 7 and len(set(rows)) == len(rows)


def test_sweep_is_what_the_host_geometry_builds(monkeypatch):
    """Every forced configuration of the sweep is honoured by pn_sepconv_describe (tile, sub-tiles, p / w / a / stg, teams), and the
    sweep covers the kernel's switches."""
    lib, buf = nat.load(), C.create_string_buffer(512)
    seen = []
    for blk in sepref.BLOCKS:
        n, h, w, k, nc, s, d = blk
        ho, wo = sepref.conv_out(h, s, d), sepref.conv_out(w, s, d)
        for cfg in [";;"] + sepref.SWEEP[blk]:
            for var, val in sepref.config_env(cfg).items():
                if val is None:
                    monkeypatch.delenv(var, raising=False)
                else:
                    monkeypatch.setenv(var, val)
            assert lib.pn_sepconv_describe(*blk, buf, 512) == 0, (blk, cfg, lib.pn_last_error_string())
            g = sepref.parse_describe(buf.value.decode())
            assert buf.value.startswith((b"tile", b"half tile")) and sepref.config_honoured(cfg, g), (blk, cfg, buf.value)
            seen.append(dict(g, k=k, nc=nc, stride=s, dil=d, ho=ho, wo=wo))
    have = lambda f: any(f(g) for g in seen)
    cover = {
        "teams 1": lambda g: g["teams"] == 1, "teams 2": lambda g: g["teams"] == 2,
        **{"stg%d on a double-buffered accumulator" % i: (lambda i: lambda g: g["stg"] == i and g["n_tile"] <= 256)(i) for i in range(3)},
        **{"stg%d on a single accumulator" % i: (lambda i: lambda g: g["stg"] == i and g["n_tile"] > 256)(i) for i in range(3)},
        **{"subs %d" % i: (lambda i: lambda g: g["subs"] == i)(i) for i in range(1, 5)},
        "resident W": lambda g: g["w_res"], "W ring": lambda g: not g["w_res"],
        "K <= 256 (resident depthwise weights)": lambda g: g["k"] <= 256, "K > 256": lambda g: g["k"] > 256,
        "two column halves": lambda g: g["n_halves"] == 2, "two n-tiles": lambda g: g["n_tiles"] == 2,
        "half-warp layout": lambda g: g["half"], "stride 2": lambda g: g["stride"] == 2,
        "dilation 2": lambda g: g["dil"] == 2, "dilation 4": lambda g: g["dil"] == 4,
        "ragged K": lambda g: g["k"] % 64 != 0, "ragged N": lambda g: g["nc"] % 64 != 0,
        "K in 24/48/96/192/384": lambda g: g["k"] in (24, 48, 96, 192, 384), "N in 24/48/96/192/384": lambda g: g["nc"] in (24, 48, 96, 192, 384),
        "tile taller than the map": lambda g: g["th"] > g["ho"], "tile wider than the map": lambda g: g["tw"] > g["wo"],
        "one-row tile": lambda g: g["th"] == 1, "one-column tile": lambda g: g["tw"] == 1,
        "more tiles than SMs": lambda g: g["tiles"] > 148,
    }
    missing = [name for name, f in cover.items() if not have(f)]
    assert not missing, missing
    assert 200 <= len(seen) <= 400, len(seen)
