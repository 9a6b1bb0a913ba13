"""Device time of one pointwise GEMM shape (pn_pwconv_gemm, bf16), median over launches inside one CUDA graph.
usage: python tools/time_gemm.py m,k,n [...]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "posenet-pytorch_b200"), os.path.join(ROOT, "tests"), ROOT]
import torch
import abi
from posenet import _native as nat


def run(m, k, n, reps=20):
    lib = nat.load()
    g = torch.Generator().manual_seed(0)
    a = [(torch.randn((m, k), generator=g)).to(torch.bfloat16).cuda() for _ in range(2)]
    w = (torch.randn((n, k), generator=g) / k ** 0.5).to(torch.bfloat16).cuda()
    b = torch.randn(n, generator=g).cuda()
    y = [torch.empty((m, n), dtype=torch.bfloat16, device="cuda") for _ in range(2)]
    P = abi.P

    def launch(i):
        nat.check(lib.pn_pwconv_gemm(P(a[i % 2]), P(w), P(b), P(y[i % 2]), m, k, n, nat.PN_BF16, nat.stream_ptr()), "pn_pwconv_gemm")
    for i in range(3):
        launch(i)
    torch.cuda.synchronize()
    ref = torch.clamp(a[0][:512].float() @ w.float().t() + b, 0, 6)
    err = float((y[0][:512].float() - ref).abs().max() / ref.abs().max())
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
    t = ts[len(ts) // 2]
    print("%s: median %.1f us  %.0f TFLOP/s  rel err (first 512 rows) %.2e" % ((m, k, n), t, 2.0 * m * k * n / t / 1e6, err), flush=True)


if __name__ == "__main__":
    for s in sys.argv[1:]:
        run(*[int(v) for v in s.split(",")])
