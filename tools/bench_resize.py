"""pn_resize_u8 / pn_preprocess_u8 device time at C3's frame size (32 x 1280x720 -> 721x1281)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "posenet-pytorch_b200"), os.path.join(ROOT, "tests")]
import torch
import abi
torch.cuda.set_device(0)
x = torch.randint(0, 256, (32, 720, 1280, 3), dtype=torch.uint8, device="cuda")
for name, fn in (("resize_u8", lambda: abi.resize_u8(x, 721, 1281)), ("preprocess_u8 (f32 NCHW out)", lambda: abi.preprocess(x, 721, 1281))):
    for _ in range(3): fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(10): fn()
    e1.record(); torch.cuda.synchronize()
    print("%s: %.1f us per 32 frames" % (name, e0.elapsed_time(e1) * 100))
