"""Timeline of CTA 0 of septc_kernel (clock64 stamps at the hand-offs, see TCS_TR in csrc/septc.cu).
Needs a diagnostics build: PN_EXTRA_NVCC_FLAGS=-DPN_TCS_TRACE python posenet-pytorch_b200/build.py --force."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "posenet-pytorch_b200"), os.path.join(ROOT, "tests"), ROOT]
import torch

import abi
from posenet import _native as nat

shape = tuple(int(v) for v in (sys.argv[1].split(",") if len(sys.argv) > 1 else "64,33,33,256,256,1,1".split(",")))
n, h, w, cin, cout, stride, dil = shape
lo, hi = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (16, 28)
g = torch.Generator().manual_seed(1)
x = (torch.rand((n, h, w, cin), generator=g) * 6).to(torch.bfloat16).cuda()
w9 = (torch.randn((9, cin), generator=g) * 0.35).cuda()
bd = (torch.randn(cin, generator=g) * 0.3).cuda()
wp = (torch.randn((cout, cin), generator=g) * (1.5 / cin ** 0.5)).to(torch.bfloat16).cuda()
bp = (torch.randn(cout, generator=g) * 0.5).cuda()
lib = C.CDLL(nat.LIB_PATH)
cap = 64
buf = torch.zeros((6, cap, 4), dtype=torch.int64, device="cuda")
abi.sepconv(x, w9, bd, wp, bp, stride, dil)
torch.cuda.synchronize()
lib.pn_debug_tcs_trace.argtypes = [C.c_void_p, C.c_int]
assert lib.pn_debug_tcs_trace(C.c_void_p(buf.data_ptr()), cap) == 0
abi.sepconv(x, w9, bd, wp, bp, stride, dil)
torch.cuda.synchronize()
lib.pn_debug_tcs_trace(None, 0)
t = buf.cpu().numpy()
t0 = t[t > 0].min()
names = ["producers: patch_empty ok (d) | w_empty ok (s)", "pw issuer (s): start | tempty+w_full | a_full | issued", "dw issuer0 (d): dw_free | patch_full | diag_full | issued",
         "converter (d): dw_full | math done | a_empty | arrived", "diag writer (d): diag_empty | done", "epilogue (item): tfull | released | done"]
for s in range(lo, hi):
    print("step %d" % s)
    for r in range(6):
        vals = [int(v - t0) if v > 0 else -1 for v in t[r, s]]
        print("   %-62s %s" % (names[r], "  ".join("%7d" % v for v in vals)))
