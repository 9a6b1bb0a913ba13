"""Where a depthwise warp of the fused block spends its cycles (debug build: -DPN_SEP_TRACE -DPN_SEP_PHASES, see sepconv.cu).
usage: python tools/phases_sep.py n,h,w,cin,cout,stride,dil [...]"""
import ctypes as C, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "posenet-pytorch_b200"), os.path.join(ROOT, "tests"), ROOT]
import torch
import abi
from posenet import _native as nat

NAMES = ["wait A", "wait patch", "weights+table", "preload", "rows", "patch arrive", "fence + A arrive", "between items"]

def run(n, h, w, cin, cout, stride, dil):
    lib = nat.load()
    lib.pn_debug_sep_trace.argtypes = [C.c_void_p, C.c_int]
    g = torch.Generator().manual_seed(0)
    x = (torch.rand((n, h, w, cin), generator=g) * 6).to(torch.bfloat16).cuda()
    w9 = (torch.randn((9, cin), generator=g) * 0.3).cuda()
    bd = torch.zeros(cin).cuda()
    wp = (torch.randn((cout, cin), generator=g) / cin ** 0.5).to(torch.bfloat16).cuda()
    bp = torch.zeros(cout).cuda()
    for _ in range(2):
        abi.sepconv(x, w9, bd, wp, bp, stride, dil)
    torch.cuda.synchronize()
    cap = 4096
    buf = torch.zeros((4 * cap * 4,), dtype=torch.int64, device="cuda")
    assert lib.pn_debug_sep_trace(C.c_void_p(buf.data_ptr()), cap) == 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); abi.sepconv(x, w9, bd, wp, bp, stride, dil); e1.record()
    torch.cuda.synchronize()
    lib.pn_debug_sep_trace(None, 0)
    t = buf.cpu().numpy()[:16 * 8].reshape(16, 8)
    desc = C.create_string_buffer(512)
    lib.pn_sepconv_describe(n, h, w, cin, cout, stride, dil, desc, 512)
    print("== %s: %s" % ((n, h, w, cin, cout, stride, dil), desc.value.decode()))
    rows = [r for r in t if r.sum() > 0]
    tot = sum(float(r.sum()) for r in rows) / len(rows)
    print("   %d depthwise warps of block 0, %.0f cycles each (kernel %.1f us incl. launch)" % (len(rows), tot, e0.elapsed_time(e1) * 1e3))
    for i, nm in enumerate(NAMES):
        v = sum(float(r[i]) for r in rows) / len(rows)
        print("   %-18s %9.0f cycles  %5.1f %%" % (nm, v, 100 * v / tot))

if __name__ == "__main__":
    for a in sys.argv[1:]:
        run(*[int(v) for v in a.split(",")])
