"""CPU-only checks of the host side: the C-ABI library loads and exports every declared symbol,
the drop-in package mirrors the reference's API surface, and nothing silently falls back."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import posenet
from oracle import decode as odec
from oracle import net as onet
from posenet import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "posenet_b200.h")).read()
    declared = set(re.findall(r"\b(pn_[a-z0-9_]+)\s*\(", header))
    assert declared == set(nat.EXPORTS), declared ^ set(nat.EXPORTS)
    lib = nat.load()                                       # raises if missing / symbol absent / ABI mismatch
    for name in declared:
        assert hasattr(lib, name)
    assert lib.pn_abi_version() == nat.ABI_VERSION == 5
    # the product ABI is the hot path only: probes and traces live in a second library / a diagnostics build
    assert not [n for n in declared if n.startswith(("pn_debug", "pn_dwtc"))]
    for name in ("pn_dwtc_probe", "pn_debug_umma_cost", "pn_debug_tcs_trace", "pn_debug_sep_trace"):
        assert not hasattr(lib, name), name


def test_diagnostics_library_exports_its_header():
    import ctypes as C
    header = open(os.path.join(ROOT, "include", "posenet_b200_diag.h")).read()
    declared = set(re.findall(r"\b(pn_[a-z0-9_]+)\s*\(", header))
    assert declared == {"pn_diag_last_error_string", "pn_dwtc_probe", "pn_debug_umma_cost"}, declared
    lib = C.CDLL(os.path.join(os.path.dirname(nat.LIB_PATH), "libposenet_b200_diag.so"))
    for name in declared:
        assert hasattr(lib, name), name


def test_struct_layouts_match_header():
    import ctypes as C
    assert C.sizeof(nat.Map) == 40 and C.sizeof(nat.DecodeParams) == 24 and C.sizeof(nat.Layer) == 48
    assert C.sizeof(nat.NetDesc) == 24 + 16 * 48 + 16 + 8          # + flags, padded to pointer alignment


def test_sepconv_tile_geometry_is_host_computable():
    """pn_sepconv_describe is pure host arithmetic: every block of every model/stride has a tile shape."""
    import ctypes as C
    lib, buf = nat.load(), C.create_string_buffer(256)
    for mid, os_, hw in ((101, 16, 513), (101, 8, 257), (50, 8, 721), (75, 32, 257), (100, 32, 129)):
        m = posenet.MobileNetV1(mid, output_stride=os_)
        h = w = hw
        for L in m._layers:
            s, d = L["stride"], L["rate"]
            if L["block_id"]:
                assert lib.pn_sepconv_describe(2, h, w, L["inp"], L["outp"], s, d, buf, 256) == 0, lib.pn_last_error_string()
                assert b"tile" in buf.value or b"warp-autonomous strips" in buf.value or b"tensor-pipe" in buf.value
            pad = ((s - 1) + 2 * d) // 2
            h = w = (h + 2 * pad - 2 * d - 1) // s + 1
    assert lib.pn_sepconv_describe(2, 9, 9, 64, 64, 2, 2, buf, 256) != 0            # never produced by the tables


def test_tensor_pipe_depthwise_routing_and_geometry():
    """The 256 -> 256 blocks at stride 1, dilation 1 or 2 run on csrc/septc.cu (measured faster there); band layout is host
    arithmetic."""
    import ctypes as C
    lib, buf = nat.load(), C.create_string_buffer(512)
    for shp, want in (((64, 33, 33, 256, 256, 1, 1), b"bands 1 x 33 cols pitch 34"), ((32, 91, 161, 256, 256, 1, 2), b"kblocks 4"),
                      ((2, 5, 3, 256, 256, 1, 2), b"tensor-pipe")):
        assert lib.pn_sepconv_describe(*shp, buf, 512) == 0, lib.pn_last_error_string()
        assert b"tensor-pipe depthwise" in buf.value and want in buf.value, buf.value
    for shp in ((64, 33, 33, 512, 512, 1, 1), (64, 129, 129, 128, 128, 1, 1), (512, 17, 17, 384, 384, 1, 1), (64, 65, 65, 256, 512, 2, 1),
                (64, 65, 65, 256, 256, 2, 1), (2, 33, 33, 256, 256, 1, 4), (64, 257, 257, 32, 64, 1, 1), (2, 33, 33, 1024, 1024, 1, 2),
                (3, 65, 65, 96, 96, 1, 1)):
        assert lib.pn_sepconv_describe(*shp, buf, 512) == 0 and b"tensor-pipe" not in buf.value, shp    # other widths, stride 2, dilation 4


def test_measured_tile_table_and_forced_teams(monkeypatch):
    """csrc/sep_tuned.inc: every row is a configuration the geometry code accepts as written (tile, ring depths, teams), it is
    what the described block gets, and forced teams need rings deep enough."""
    import ctypes as C
    import re
    lib, buf = nat.load(), C.create_string_buffer(512)
    for k in ("PN_SEP_TILE", "PN_SEP_STAGES", "PN_SEP_TEAMS"):
        monkeypatch.delenv(k, raising=False)
    inc = os.path.join(os.path.dirname(nat.__file__), "..", "csrc", "sep_tuned.inc")
    rows = [tuple(int(v) for v in m.group(1).split(",")) for m in re.finditer(r"^\s*\{([\d, ]+)\}", open(inc).read(), re.M)]
    assert len(rows) >= 5
    pat = re.compile(r"tile (\d+)x(\d+) subs (\d+) .* teams (\d+) stages p(\d+) w(\d+)r? a(\d+) stg(\d+)")
    for (k, nc, s, d, ho, wo, th, tw, subs, p, w, a, stg, teams) in rows:
        h, wd = (ho - 1) * s + 1, (wo - 1) * s + 1                   # an input size that gives this output size (pad = dilation for stride 1)
        assert lib.pn_sepconv_describe(4, h, wd, k, nc, s, d, buf, 512) == 0, lib.pn_last_error_string()
        got = tuple(int(v) for v in pat.search(buf.value.decode()).groups())
        assert got == (th, tw, subs, teams, p, w, a, stg), (buf.value, (k, nc, s, d, ho, wo))
    # forced teams: one team of ten warps always; two teams of five only where two items fit the rings (p >= 2 subs, a >= 2, p >= a),
    # otherwise the request is ignored
    assert lib.pn_sepconv_describe(64, 129, 129, 128, 128, 1, 1, buf, 512) == 0 and b"teams 2" in buf.value
    assert lib.pn_sepconv_describe(64, 257, 257, 64, 128, 2, 1, buf, 512) == 0 and b"teams 1" in buf.value
    monkeypatch.setenv("PN_SEP_TEAMS", "1")
    assert lib.pn_sepconv_describe(64, 129, 129, 128, 128, 1, 1, buf, 512) == 0 and b"teams 1" in buf.value
    monkeypatch.setenv("PN_SEP_TEAMS", "2")
    assert lib.pn_sepconv_describe(64, 257, 257, 64, 128, 2, 1, buf, 512) == 0 and b"teams 2" in buf.value      # p2 a2
    assert lib.pn_sepconv_describe(64, 65, 65, 128, 256, 2, 1, buf, 512) == 0 and b"teams 1" in buf.value        # p4 with 3 subs
    # resident pointwise weights: one stage per (k-block, column block), marked "r"
    monkeypatch.delenv("PN_SEP_TEAMS")
    assert lib.pn_sepconv_describe(64, 129, 129, 128, 128, 1, 1, buf, 512) == 0 and b" w2r " in buf.value
    assert lib.pn_sepconv_describe(64, 33, 33, 512, 512, 1, 1, buf, 512) == 0 and b"r a" not in buf.value      # 512 KB of W: ring


def test_warp_autonomous_block_routing():
    """csrc/sepwarp.cu: which fused blocks run warp-autonomous -- cin <= 32 / cout <= 64 at stride 1 (quarter-warp layout up to cin
    16), stride 2 for cin 17..32, the full-warp layout for 48 -> 96 stride 2 -- and the output geometry of the stride-2 strips."""
    import ctypes as C
    lib, buf = nat.load(), C.create_string_buffer(512)

    def desc(*shape):
        assert lib.pn_sepconv_describe(*shape, buf, 512) == 0, lib.pn_last_error_string()
        return buf.value.decode()
    assert desc(32, 721, 1281, 16, 32, 1, 1).startswith("warp-autonomous strips 161 x")            # 1281 / 8
    # row blocks: the count that minimises the largest per-warp sum of input rows under the round-robin item assignment (148 SMs x 16
    # warps)
    assert "strips 33 x 10 row blocks of 26 rows" in desc(64, 257, 257, 32, 64, 1, 1)
    assert "strips 17 x 4 row blocks of 33 rows" in desc(512, 129, 129, 24, 48, 1, 1)
    assert "strips 41 x 7 row blocks of 26 rows" in desc(32, 361, 641, 32, 64, 2, 1)
    d = desc(32, 721, 1281, 32, 64, 2, 1)
    assert d.startswith("warp-autonomous stride 2 strips 81 x") and "k16 slices 2, n8 tiles 8" in d   # output 361 x 641: 641 / 8
    d = desc(512, 129, 129, 48, 96, 2, 1)
    assert d.startswith("warp-autonomous full-warp stride 2 strips 17 x") and "k16 slices 3, n8 tiles 12" in d   # output 65 wide: 65 / 4
    assert desc(32, 181, 321, 64, 64, 1, 1).startswith("tile ")                                       # measured slower there: CTA pipeline
    assert desc(32, 721, 1281, 16, 32, 2, 1).startswith("tile ")                                      # stride 2 needs cin > 16
    assert desc(64, 257, 257, 64, 128, 2, 1).startswith("tile ")


def test_warp_autonomous_row_blocks_minimise_the_busiest_warp():
    """sepwarp_geometry picks the row-block count whose round-robin item assignment leaves the busiest warp the least input rows:
    a Python model of the same simulation (items strips-fastest over 148 x 16 warps, cost = input rows of the block) agrees with the
    library on random shapes of the three layouts, and the rows cover the map exactly."""
    import ctypes as C
    import re
    lib, buf = nat.load(), C.create_string_buffer(512)
    warps = 148 * 16

    def model(n, ho, strips, s):
        best = None
        for cand in range(1, -(-ho // 8) + 1):
            rb = -(-ho // cand)
            if -(-ho // rb) != cand:
                continue
            load = [0] * warps
            for it in range(n * strips * cand):
                q = (it // strips) % cand
                load[it % warps] += min(rb, ho - q * rb) * s + (3 - s)
            if best is None or max(load) < best[0]:
                best = (max(load), cand, rb)
        return best[1], best[2]

    rng = np.random.default_rng(5)
    shapes = [(64, 257, 257, 32, 64, 1), (512, 129, 129, 24, 48, 1), (32, 361, 641, 16, 32, 1), (32, 361, 641, 32, 64, 2), (512, 129, 129, 48, 96, 2)]
    for _ in range(12):
        k, nc, s = [(32, 64, 1), (16, 32, 1), (24, 48, 1), (32, 64, 2), (48, 96, 2)][int(rng.integers(0, 5))]
        shapes.append((int(rng.integers(1, 40)), int(rng.integers(1, 300)), int(rng.integers(1, 300)), k, nc, s))
    for n, h, w, k, nc, s in shapes:
        assert lib.pn_sepconv_describe(n, h, w, k, nc, s, 1, buf, 512) == 0, lib.pn_last_error_string()
        m = re.search(r"strips (\d+) x (\d+) row blocks of (\d+) rows", buf.value.decode())
        assert m, buf.value
        strips, nq, rb = (int(v) for v in m.groups())
        ho, wo = (h - 1) // s + 1, (w - 1) // s + 1
        assert strips == -(-wo // (4 if (k, nc, s) == (48, 96, 2) else 8))
        assert (nq - 1) * rb < ho <= nq * rb
        assert (nq, rb) == model(n, ho, strips, s), (n, h, w, k, nc, s)


@pytest.mark.parametrize("mid", [50, 75, 100, 101])
@pytest.mark.parametrize("os_", [8, 16, 32])
def test_layer_table_and_state_dict_mirror_reference(mid, os_):
    m = posenet.MobileNetV1(mid, output_stride=os_)
    assert [(L["inp"], L["outp"], L["stride"], L["rate"]) for L in m._layers] == \
           [(L["cin"], L["cout"], L["stride"], L["dilation"]) for L in onet.layer_table(mid, os_)]
    sd = m.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == onet.param_shapes(mid)
    assert list(sd) == list(onet.param_shapes(mid))
    m.load_state_dict(onet.init_params(mid, 0), strict=True)
    assert m.output_stride == os_


def test_api_surface():
    for name in ("load_model", "MobileNetV1", "MOBILENET_V1_CHECKPOINTS", "decode_multiple_poses", "read_imgfile", "read_cap",
                 "valid_resolution", "draw_skel_and_kp", "draw_skeleton", "draw_keypoints", "get_adjacent_keypoints",
                 "PART_NAMES", "NUM_KEYPOINTS", "PARENT_CHILD_TUPLES", "CONNECTED_PART_INDICES", "LOCAL_MAXIMUM_RADIUS",
                 "POSE_CHAIN", "PART_IDS", "decode", "decode_multi"):
        assert hasattr(posenet, name), name
    assert posenet.decode_multi.decode_multiple_poses is posenet.decode_multiple_poses
    assert tuple(posenet.PARENT_CHILD_TUPLES) == tuple(odec.EDGES)
    assert posenet.NUM_KEYPOINTS == 17 and len(posenet.CONNECTED_PART_INDICES) == 12
    assert posenet.valid_resolution(1280 * 0.7125, 720 * 0.7125, 16) == (913, 513)
    import inspect
    assert list(inspect.signature(posenet.decode.decode_pose).parameters) == [
        "root_score", "root_id", "root_image_coord", "scores", "offsets", "output_stride", "displacements_fwd", "displacements_bwd"]
    assert list(inspect.signature(posenet.decode.traverse_to_targ_keypoint).parameters) == [
        "edge_id", "source_keypoint", "target_keypoint_id", "scores", "offsets", "output_stride", "displacements"]   # decode.py:9-11,131-138
    sig = inspect.signature(posenet.decode_multiple_poses)
    assert [(p.name, p.default) for p in sig.parameters.values()][4:] == [
        ("output_stride", inspect.Parameter.empty), ("max_pose_detections", 10), ("score_threshold", 0.5),
        ("nms_radius", 20), ("min_pose_score", 0.5)]


def test_load_model_needs_checkpoint_and_writes_random(tmp_path):
    with pytest.raises(FileNotFoundError):
        posenet.load_model(75, model_dir=str(tmp_path))
    posenet.write_random_checkpoint(75, str(tmp_path), seed=3)
    m = posenet.load_model(75, model_dir=str(tmp_path))
    assert sum(p.numel() for p in m.parameters()) == 1258195


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_silent_cpu_fallback():
    m = posenet.MobileNetV1(50)
    with pytest.raises(nat.NativeError):
        m(torch.zeros(1, 3, 33, 33))
    with pytest.raises(nat.NativeError):
        posenet.decode_multiple_poses(torch.zeros(17, 3, 3), torch.zeros(34, 3, 3), torch.zeros(32, 3, 3),
                                      torch.zeros(32, 3, 3), 16)
    with pytest.raises(nat.NativeError):
        posenet._process_input(np.zeros((17, 17, 3), np.uint8))
    with pytest.raises(nat.NativeError):
        posenet.decode.decode_pose(0.9, 0, np.zeros(2), np.zeros((17, 3, 3), np.float32), np.zeros((17, 3, 3, 2), np.float32), 16,
                                   np.zeros((16, 3, 3, 2), np.float32), np.zeros((16, 3, 3, 2), np.float32))
    with pytest.raises(nat.NativeError):
        posenet.decode.traverse_to_targ_keypoint(0, np.zeros(2), 1, np.zeros((17, 3, 3), np.float32),
                                                 np.zeros((17, 3, 3, 2), np.float32), 16, np.zeros((16, 3, 3, 2), np.float32))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "posenet-pytorch_b200")
    pat = re.compile(r"^\s*(import\s+oracle|from\s+oracle\b)|oracle/|oracle\.(net|decode|preprocess|synth)", re.M)
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                assert not pat.search(open(os.path.join(d, f)).read()), os.path.join(d, f)


def _path_walk_decode_pose(root_score, root_id, root_xy, scores, offsets, stride, fwd, bwd):
    """The scheme of csrc/decode.cu's speculative phase, restated on the host: the thread of part k walks the unique tree
    path root -> k (child -> parent hops with ``bwd`` first, then parent -> child hops with ``fwd``) and stops where the
    reference's ``score[source] > 0.0`` gate would; parts that are not reached keep zeros."""
    up, up_edge = [0] * odec.PARTS, [-1] * odec.PARTS
    for e, (parent, child) in enumerate(odec.EDGES):
        up[child], up_edge[child] = parent, e
    anc = []
    for k in range(odec.PARTS):
        chain, c = {k}, k
        while c != 0:
            c = up[c]
            chain.add(c)
        anc.append(chain)
    ks, kc, ko = np.zeros(odec.PARTS), np.zeros((odec.PARTS, 2)), np.zeros((odec.PARTS, 2))
    hops = 0
    for k in range(odec.PARTS):
        cur, sc, xy, off, reached, n = root_id, root_score, np.asarray(root_xy, dtype=np.float64), np.zeros(2), True, 0
        while cur != k:
            if not (sc > 0.0):
                reached = False
                break
            if cur not in anc[k]:                                   # climb: child -> parent
                nxt, e, disp = up[cur], up_edge[cur], bwd
            else:                                                   # descend towards k: parent -> child
                nxt = k
                while up[nxt] != cur:
                    nxt = up[nxt]
                e, disp = up_edge[nxt], fwd
            sc, xy, off = odec._hop(e, xy, nxt, scores, offsets, stride, disp)
            cur = nxt
            n += 1
        hops = max(hops, n)
        if reached:
            ks[k], kc[k], ko[k] = sc, xy, off
    return ks, kc, ko, hops


@pytest.mark.parametrize("seed", range(6))
def test_per_part_path_walk_equals_the_two_pass_decode_pose(seed):
    # decode.py:131-182 reaches every part along its tree path from the root, and a hop only depends on its source coordinates:
    # the equivalence the CUDA decoder's 17-threads-per-pose phase rests on, checked for every root part, with zero, negative
    # and NaN scores on the paths (the `> 0.0` / `== 0.0` gates), bit for bit
    from oracle import synth
    rng = np.random.default_rng(seed)
    h, w, stride = int(rng.integers(5, 30)), int(rng.integers(5, 30)), int(rng.choice([8, 16, 32]))
    heat, off, fwd, bwd = synth.random_heads(h, w, seed=seed, disp_scale=float(rng.uniform(5, 90)), off_scale=float(rng.uniform(1, 20)),
                                             zero_frac=float(rng.choice([0.0, 0.2, 0.5])))[:4]
    heat = heat.copy()
    if seed % 2:
        mask = rng.random(heat.shape)
        heat[mask < 0.05] = -0.25
        heat[mask > 0.97] = np.nan
    split = lambda a: np.asarray(a, dtype=np.float32).reshape(2, -1, h, w).transpose(1, 2, 3, 0)
    offs, f, b = split(off), split(fwd), split(bwd)
    longest = 0
    for root_id in range(odec.PARTS):
        for _ in range(4):
            y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
            root_score = float(rng.choice([heat[root_id, y, x], 0.7]))
            root = np.array([y, x]) * stride + offs[root_id, y, x]
            ref = odec.decode_pose(root_score, root_id, root, heat, offs, stride, f, b)
            got = _path_walk_decode_pose(root_score, root_id, root, heat, offs, stride, f, b)
            for a_, b_ in zip(got[:3], ref):
                assert np.array_equal(a_, b_, equal_nan=True)
            longest = max(longest, got[3])
    assert longest <= 8                                              # ankle -> nose -> other ankle


@pytest.mark.parametrize("mid,H,W,os_,fmap,total,gemm,dw,stem", [
    (101, 513, 513, 16, (33, 33), 9.066, 8.742, 0.210, 0.114),       # C1 / C2
    (50, 721, 1281, 8, (91, 161), 17.860, 16.936, None, None),      # C3
    (75, 257, 257, 32, (17, 17), 1.001, 0.940, None, None),         # C4 ("OS32" is really 16, SURVEY F4)
])
def test_bench_algorithmic_work_matches_the_survey(mid, H, W, os_, fmap, total, gemm, dw, stem):
    # SURVEY 8(d): the per-image flops bench.py's roofline entries are built from (2 * MACs), per config
    import bench
    rows, hw = bench.layer_costs(posenet.MobileNetV1(mid, output_stride=os_), 1, H, W)
    assert hw == fmap
    f = {name: flops for name, _, flops in rows}
    s_stem = f["stem"]
    s_dw = sum(v for k, v in f.items() if k.startswith("dw"))
    s_gemm = sum(v for k, v in f.items() if k.startswith("pw")) + f["heads"]
    assert round((s_stem + s_dw + s_gemm) / 1e9, 3) == total
    assert round(s_gemm / 1e9, 3) == gemm
    if dw is not None:
        assert round(s_dw / 1e9, 3) == dw and round(s_stem / 1e9, 3) == stem
    # a fused block moves its input and its output once: strictly less than depthwise + pointwise apart
    b = {name: nbytes for name, nbytes, _ in rows}
    for k in [k for k in b if k.startswith("sep")]:
        i = k[3:]
        assert b[k] < b["dw" + i] + b["pw" + i]


def _radix_chunks(keys, chunk=1024):
    """Host model of the candidate selection in csrc/decode.cu (decode_kernel, step 1): the best <= `chunk` keys greater than
    `lo` are cut off by an MSB-first radix descent (8 bits per level) that starts below the bits all remaining keys share."""
    keys = [int(k) for k in keys]
    lo, remaining, out = 0, len(keys), []
    while remaining > 0:
        pivot = (1 << 64) - 1
        if remaining > chunk:
            live = [k for k in keys if k > lo]
            mn, mx = min(live), max(live)
            bits = 64 - (mn ^ mx).bit_length()                      # __clzll(min ^ max)
            prefix = mn >> (64 - bits) if bits else 0
            while True:
                width = min(8, 64 - bits)
                shift = 64 - bits - width
                hist = [0] * 256
                for k in live:
                    if bits == 0 or (k >> (64 - bits)) == prefix:
                        hist[(k >> shift) & ((1 << width) - 1)] += 1
                cum, sel, first = 0, -1, -1
                for d in range(256):
                    c = hist[d]
                    if c and first < 0:
                        first = d
                    if cum + c > chunk:
                        break
                    cum += c
                    if c:
                        sel = d
                if sel >= 0:
                    pivot = (((prefix << width) | sel) << shift) | ((1 << shift) - 1)
                    break
                prefix, bits = (prefix << width) | first, bits + width
                assert bits <= 64
        got = sorted(k for k in keys if lo < k <= pivot)
        assert 1 <= len(got) <= max(chunk, 1) or remaining <= chunk
        out.append(got)
        lo, remaining = pivot, remaining - len(got)
    return out


@pytest.mark.parametrize("kind", ["random", "near_half", "plateaus", "two_levels"])
def test_radix_selection_model_partitions_the_sorted_candidates(kind):
    # keys as pn_candidates builds them: high word = inverted orderable score bits, low word = flat cell index (unique)
    rng = np.random.default_rng(5)
    n = 6000
    if kind == "random":
        score = rng.random(n, dtype=np.float32)
    elif kind == "near_half":                                        # random-init heatmaps: everything within 1e-3 of 0.5
        score = (0.5 + 1e-3 * rng.random(n)).astype(np.float32)
    elif kind == "plateaus":                                         # six distinct values only: the index word must separate
        score = rng.choice(np.linspace(0.3, 0.9, 6), n).astype(np.float32)
    else:
        score = np.where(rng.random(n) < 0.5, np.float32(0.75), rng.random(n, dtype=np.float32)).astype(np.float32)
    u = score.view(np.uint32).astype(np.uint64) ^ np.uint64(0x80000000)                  # positive floats: set the sign bit
    keys = ((~u & np.uint64(0xFFFFFFFF)) << np.uint64(32)) | rng.permutation(n).astype(np.uint64)
    chunks = _radix_chunks(keys)
    assert all(1 <= len(c) <= 1024 for c in chunks)
    flat = [k for c in chunks for k in c]
    assert flat == sorted(int(k) for k in keys)                      # ascending key == descending score, index ascending


def test_reference_scripts_are_pinned():
    """oracle/make_ref.py compiles benchmark.py / image_demo.py from the reference checkout only when their sha256 is the pinned
    one; the manifest of an existing oracle/_ref build records the same digests ("run unchanged" is checked, not assumed)."""
    from oracle import make_ref
    ref = "/root/reference"
    if os.path.isdir(ref):
        for name, digest in make_ref.SCRIPT_SHA256.items():
            assert make_ref.sha256_file(os.path.join(ref, name)) == digest, name
    m = make_ref.manifest()
    if m is not None:
        assert m["scripts_sha256"] == make_ref.SCRIPT_SHA256
        if os.path.isdir(ref):
            assert m["package_sha256"] == make_ref.tree_digest(os.path.join(ref, "posenet"))
    tracked = subprocess.run(["git", "ls-files", "oracle/_ref"], cwd=ROOT, capture_output=True, text=True).stdout.strip()
    assert tracked == "", "oracle/_ref must stay out of the history"
