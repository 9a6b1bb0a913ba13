"""Device time of one fused SeperableConv block shape (pn_sepconv_block), median of `reps` launches with CUDA events;
inputs rotate over two buffers.  usage: python tools/time_sep.py n,h,w,cin,cout,stride,dil [...]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "posenet-pytorch_b200"), os.path.join(ROOT, "tests"), ROOT]
import ctypes as C
import torch
import abi
from posenet import _native as nat


def run(n, h, w, cin, cout, stride, dil, reps=20):
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

    def launch(i):
        nat.check(lib.pn_sepconv_block(P(xs[i % 2]), P(w9), P(bd), P(wp), P(bp), P(ys[i % 2]), n, h, w, cin, cout, stride, dil,
                                       nat.stream_ptr()), "pn_sepconv_block")
    for i in range(3):
        launch(i)
    torch.cuda.synchronize()
    # `reps` launches back to back inside ONE CUDA graph: the host cost of a launch (five tensor-map encodes) would otherwise
    # sit between the two events of an eager measurement
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for i in range(reps):
                launch(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); graph.replay(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / reps)
    ts.sort()
    desc = C.create_string_buffer(512)
    lib.pn_sepconv_describe(n, h, w, cin, cout, stride, dil, desc, 512)
    print("%s: median %.1f us  min %.1f us | %s" % ((n, h, w, cin, cout, stride, dil), ts[len(ts) // 2], ts[0], desc.value.decode()), flush=True)


if __name__ == "__main__":
    for a in sys.argv[1:]:
        run(*[int(v) for v in a.split(",")])
