"""The CTA-pipeline kernel of the fused separable block (csrc/sepconv.cu) in the configurations it can be given, cell by cell.

(1) Every row of the measured table (csrc/sep_tuned.inc) at its own output size, with enough images that the persistent grid wraps,
    against the fp64 reference and per-cell bound of tests/sepref.py.
(2) Representative blocks at small maps: the default configuration against the same bound, then every configuration of the
    seeded sweep (sepref.SWEEP: tiles, sub-tiles, ring depths, epilogues, teams), forced through PN_SEP_TILE / PN_SEP_STAGES /
    PN_SEP_TEAMS (read on every call), bit-equal to the default: each output pixel's depthwise sum runs in a fixed tap order and
    its pointwise sum in a fixed k-block order whatever the tile, ring or team.
(3) How far the tensor core's fp32 accumulation is from the exact sum (the slack sepref allows the pointwise sum)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import abi  # noqa: E402
import sepref  # noqa: E402
from posenet import _native as nat  # noqa: E402

DEV = "cuda"


def _describe(shape):
    buf = C.create_string_buffer(512)
    assert nat.load().pn_sepconv_describe(*shape, buf, 512) == 0, nat.load().pn_last_error_string()
    return sepref.parse_describe(buf.value.decode())


def _run(case, stride, dil):
    x, w9, bd, wp, bp = (t.to(DEV) for t in case)
    y = abi.sepconv(x, w9, bd, wp, bp, stride, dil)
    torch.cuda.synchronize()
    return y


def test_every_measured_row_at_its_production_size(monkeypatch):
    for var in sepref.ENV:
        monkeypatch.delenv(var, raising=False)
    rows = sepref.tuned_rows()
    tested, failures = set(), []
    for row in rows:
        k, nc, s, d, ho, wo, th, tw, subs, p, w, a, stg, teams = row
        h, wd = (ho - 1) * s + 1, (wo - 1) * s + 1                      # an input size that gives this output size
        n = 148 // (-(-ho // th) * -(-wo // tw)) + 1                    # more tiles than SMs: the persistent grid wraps
        shape = (n, h, wd, k, nc, s, d)
        g = _describe(shape)
        assert (g["th"], g["tw"], g["subs"], g["p"], g["w"], g["a"], g["stg"], g["teams"]) == (th, tw, subs, p, w, a, stg, teams), row
        assert g["tiles"] > 148, (row, g["tiles"])
        case = sepref.make_case(*shape[:5], seed=ho + wo + k)
        y = _run(case, s, d)
        ref, bound = sepref.reference(*case, s, d)
        try:
            ratio = sepref.check(y, ref, bound, "row %s" % (row,))
            print("row %s: n %d, tiles %d, max |err| / bound %.3f" % (row[:6], n, g["tiles"], ratio))
        except AssertionError as e:
            failures.append(str(e))
        tested.add(row)
    assert not failures, failures
    assert tested == set(rows) and len(rows) >= 7


@pytest.mark.parametrize("blk", sepref.BLOCKS, ids=lambda b: "n%d-%dx%d-%dto%d-s%d-d%d" % b)
def test_forced_configurations_are_bit_equal_to_the_default(blk, monkeypatch):
    n, h, w, k, nc, s, d = blk
    for var in sepref.ENV:
        monkeypatch.delenv(var, raising=False)
    case = sepref.make_case(n, h, w, k, nc, seed=h * w + k + nc)
    ref, bound = sepref.reference(*case, s, d)
    y0 = _run(case, s, d)
    ratio = sepref.check(y0, ref, bound, "default %s" % (_describe(blk),))
    failures = []
    for cfg in sepref.SWEEP[blk]:
        for var, val in sepref.config_env(cfg).items():
            if val is None:
                monkeypatch.delenv(var, raising=False)
            else:
                monkeypatch.setenv(var, val)
        g = _describe(blk)
        assert sepref.config_honoured(cfg, g), (cfg, g)
        y = _run(case, s, d)
        if not torch.equal(y, y0):
            ndiff = int(((y != y0) | torch.isnan(y)).sum())
            try:
                sepref.check(y, ref, bound, cfg)
                within = "within the bound"
            except AssertionError as e:
                within = str(e)
            failures.append("%s: %d cells differ from the default (%s)" % (cfg, ndiff, within))
    assert not failures, failures
    print("%s: %d configurations, default max |err| / bound %.3f" % (blk, len(sepref.SWEEP[blk]) + 1, ratio))


def test_tensor_core_accumulation_is_within_the_pointwise_slack():
    """tcgen05.mma kind::f16 with an fp32 accumulator (the pointwise GEMM of every fused block) through the tensor-pipe probe
    (K = 64, four k16 MMAs): its error against the exact sum, in units of 2^-24 sum|a w|, is below the 4 K that sepref allows."""
    P = abi.P
    h, w, dil, wp, x_org = 20, 33, 1, 34, -1
    rng = np.random.default_rng(7)
    bf = lambda a: torch.from_numpy(a.astype(np.float32)).to(torch.bfloat16)
    x = bf(rng.uniform(0, 6, (h, w, 64)))
    wdw = bf(rng.normal(0, 0.4, (9, 64)))
    pww = bf(rng.normal(0, 0.2, (64, 64)))
    bias = torch.from_numpy(rng.normal(0, 0.3, 64).astype(np.float32))
    diag = torch.zeros((9, 16, 64), dtype=torch.bfloat16)
    for g_ in range(4):
        for j in range(16):
            diag[:, j, 16 * g_ + j] = wdw[:, 16 * g_ + j]
    xd, dd, wd_, bd = x.to(DEV), diag.reshape(144, 64).to(DEV), pww.to(DEV), bias.to(DEV)
    out_dw = torch.zeros((128, 64), dtype=torch.float32, device=DEV)
    out_pw = torch.zeros((128, 64), dtype=torch.float32, device=DEV)
    rows_box = 127 // wp + 1 + 2 * dil
    abi.check_diag(abi.load_diag().pn_dwtc_probe(P(xd), h, w, P(dd), P(wd_), P(bd), P(out_dw), P(out_pw), wp, dil, 0, rows_box, x_org,
                                                 -dil, 0, nat.stream_ptr()), "pn_dwtc_probe")
    torch.cuda.synchronize()
    a = out_dw.cpu().double()                                   # bf16 values (the probe's A operand)
    assert torch.equal(a, a.to(torch.bfloat16).double())
    exact = a @ pww.double().t()
    scale = a.abs() @ pww.double().abs().t()
    units = float(((out_pw.cpu().double() - exact).abs() / (2.0 ** -24 * scale).clamp_min(1e-300)).max())
    print("tensor-core accumulation, K = 64: max error %.2f x 2^-24 sum|a w| (sepref allows %d)" % (units, 4 * 64))
    assert units <= 4 * 64
