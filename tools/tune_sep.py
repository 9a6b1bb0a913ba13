"""Measured tile shapes / ring depths for fused-block shapes (sepconv.cu): times the candidates the geometry code accepts
(PN_SEP_TILE / PN_SEP_STAGES / PN_SEP_TEAMS are read on every pn_sepconv_block call) and prints one `sep_tuned.inc` row per shape.

    python tools/tune_sep.py n,h,w,cin,cout,stride,dil [...]        # one child process per shape (a failing candidate costs one shape)

Level 1: tile shapes (th, tw, subs) with the default ring depths, the most pixel-efficient ones first.  Level 2: ring depths
(p, a, stg) and teams for the two best tiles.  Every timing = min of 3 replays of a CUDA graph of 10 launches."""
import os, re, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "posenet-pytorch_b200"), os.path.join(ROOT, "tests"), ROOT]

N_TILES, N_TOP = int(os.environ.get("TUNE_TILES", "36")), 2
ENV_KEYS = ("PN_SEP_TILE", "PN_SEP_STAGES", "PN_SEP_TEAMS")


def make_timer(shape):
    """(describe(env) -> geometry tuple or None, timeit(env, reps) -> us) for one block shape; tensors allocated once."""
    import ctypes as C
    import torch
    import abi
    from posenet import _native as nat
    n, h, w, cin, cout, stride, dil = shape
    lib = nat.load()
    g = torch.Generator().manual_seed(0)
    xs = [(torch.rand((n, h, w, cin), generator=g) * 6).to(torch.bfloat16).cuda() for _ in range(2)]
    w9 = (torch.randn((9, cin), generator=g) * 0.3).cuda()
    bd = torch.zeros(cin).cuda()
    wp = (torch.randn((cout, cin), generator=g) / cin ** 0.5).to(torch.bfloat16).cuda()
    bp = torch.zeros(cout).cuda()
    ho, wo = abi.conv_out(h, stride, dil), abi.conv_out(w, stride, dil)
    ys = [torch.empty((n, ho, wo, cout), dtype=torch.bfloat16, device="cuda") for _ in range(2)]
    P = abi.P
    side = torch.cuda.Stream()

    def setenv(env):
        for k in ENV_KEYS:
            if k in env: os.environ[k] = env[k]
            else: os.environ.pop(k, None)

    def describe(env):
        setenv(env)
        d = C.create_string_buffer(512)
        if lib.pn_sepconv_describe(n, h, w, cin, cout, stride, dil, d, 512) != 0: return None
        m = re.search(r"tile (\d+)x(\d+) subs (\d+) .* teams (\d+) stages p(\d+) w(\d+)(r?) a(\d+) stg(\d+)", d.value.decode())
        return tuple(int(v) if v not in ("", "r") else v for v in m.groups()) if m else None

    def launch(i):
        nat.check(lib.pn_sepconv_block(P(xs[i % 2]), P(w9), P(bd), P(wp), P(bp), P(ys[i % 2]), n, h, w, cin, cout, stride, dil,
                                       nat.stream_ptr()), "pn_sepconv_block")

    def timeit(env, reps=10):
        setenv(env)
        launch(0); launch(1)
        torch.cuda.synchronize()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for i in range(reps): launch(i)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); graph.replay(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / reps)
        return min(ts)

    return describe, timeit


def ab(shape, envs):
    """Times explicit configurations: envs = "PN_SEP_TEAMS=2,PN_SEP_STAGES=4.2.4.1;..." ('.' stands for ',' inside a value)."""
    describe, timeit = make_timer(shape)
    for spec in [""] + envs.split(";"):
        env = dict(kv.split("=") for kv in spec.split(",") if kv)
        env = {k: v.replace(".", ",") for k, v in env.items()}
        d = describe(env)
        if d is None:
            print("  %-60s rejected" % spec, flush=True)
            continue
        print("  %-60s %s  %.1f us" % (spec or "(default)", d, timeit(env, reps=20)), flush=True)


def one(shape):
    n, h, w, cin, cout, stride, dil = shape
    describe, timeit = make_timer(shape)
    ho, wo = (h + 2 * ((stride - 1 + 2 * dil) // 2) - 2 * dil - 1) // stride + 1, (w + 2 * ((stride - 1 + 2 * dil) // 2) - 2 * dil - 1) // stride + 1
    base_desc = describe({})
    if base_desc is None:
        print("shape %s: not a tile-kind block" % (shape,), flush=True)
        return
    t_base = timeit({})
    print("shape %s: default %s -> %.1f us" % (shape, base_desc, t_base), flush=True)
    sw = 8 if (cin <= 32 and stride == 1 and dil == 1) else 4
    cands = []
    for th in range(1, 65):
        for tw in range(1, 65):
            if th * tw > 128 or th > ho + 7 or tw > wo + 7: continue
            tiles = -(-ho // th) * -(-wo // tw)
            halo = ((th - 1) * stride + 2 * dil + 1) * ((tw - 1) * stride + 2 * dil + 1) / float(th * tw * stride * stride)
            eff = ho * wo / (tiles * 128.0) * (tw / float(sw * -(-tw // sw))) / halo ** 0.5      # MMA rows used x strip lanes used / halo re-reads
            cands.append((eff, th, tw))
    cands.sort(reverse=True)
    results = []
    seen = set()
    for eff, th, tw in cands[:N_TILES]:
        for subs in (1, 2, 3):
            env = {"PN_SEP_TILE": "%d,%d,%d" % (th, tw, subs)}
            d = describe(env)
            if d is None or d[:3] != (th, tw, subs) or d in seen: continue
            seen.add(d)
            try:
                t = timeit(env)
            except Exception as ex:                                  # a failed launch poisons the context: give up on this shape
                print("  FAILED %s: %s" % (env, ex), flush=True)
                return
            results.append((t, env, d))
    results.sort(key=lambda r: r[0])
    for t, env, d in results[:6]: print("  tile %-10s %s  %.1f us" % (env["PN_SEP_TILE"], d[3:], t), flush=True)
    best = results[0]
    for t0, env0, d0 in results[:N_TOP]:
        seen2 = {d0}
        for p in (2, 3, 4, 5, 6):
            for a in (2, 3, 4):
                for stg in (0, 1, 2):
                    env = dict(env0, PN_SEP_STAGES="%d,%d,%d,%d" % (p, d0[5], a, stg))
                    d = describe(env)
                    if d is None or d in seen2 or (d[4], d[7], d[8]) != (p, a, stg): continue
                    seen2.add(d)
                    try:
                        t = timeit(env)
                    except Exception as ex:
                        print("  FAILED %s: %s" % (env, ex), flush=True)
                        return
                    if t < best[0]: best = (t, env, d)
    # teams: the other setting for the best configuration so far
    t, env, d = best
    other = dict(env, PN_SEP_TEAMS=str(3 - d[3]))
    if "PN_SEP_STAGES" not in other: other["PN_SEP_STAGES"] = "%d,%d,%d,%d" % (d[4], d[5], d[7], d[8])
    d2 = describe(other)
    if d2 is not None and d2[3] == 3 - d[3]:
        try:
            t2 = timeit(other)
            if t2 < t: best = (t2, other, d2)
        except Exception as ex:
            print("  FAILED %s: %s" % (other, ex), flush=True)
            return
    t, env, d = best
    t_chk = timeit(env, reps=20)
    print("  best %s %s -> %.1f us (re-timed %.1f; default %.1f)" % (env, d, t, t_chk, t_base), flush=True)
    if t_chk < 0.985 * t_base:
        print("TUNED    {%d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d, %d},   // %.1f -> %.1f us (n %d)" % (
            cin, cout, stride, dil, ho, wo, d[0], d[1], d[2], d[4], d[5], d[7], d[8], d[3], t_base, t_chk, n), flush=True)


if __name__ == "__main__":
    if sys.argv[1] == "--one":
        one([int(v) for v in sys.argv[2].split(",")])
    elif sys.argv[1] == "--ab":
        print("shape %s" % sys.argv[2], flush=True)
        ab([int(v) for v in sys.argv[2].split(",")], sys.argv[3])
    else:
        for a in sys.argv[1:]:
            t0 = time.time()
            try:
                subprocess.run([sys.executable, __file__, "--one", a], timeout=int(os.environ.get("TUNE_TIMEOUT", "150")))
            except subprocess.TimeoutExpired:
                print("shape %s: timed out" % a, flush=True)
            print("  (%.0f s)" % (time.time() - t0), flush=True)
