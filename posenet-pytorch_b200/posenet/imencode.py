"""Device encoders' shared batch handling: frames given dense or as rows with per-frame sizes, encoded by ``jpeg.Encoder`` or
``png.Encoder`` and copied back as one ``bytes`` object per frame."""
import torch

from posenet import _native as nat


def encode_files(encoder, frames, params, shapes):
    """Encode a batch with ``encoder`` (``jpeg.Encoder`` or ``png.Encoder``): frames [N, h, w, 3], or rows and ``shapes`` as
    ``imencode_batch`` takes them; a list of ``bytes``."""
    nat.require_device()
    assert frames.is_cuda and frames.dtype == torch.uint8, "frames: a CUDA uint8 tensor"
    n = frames.shape[0]
    hw = None
    if shapes is None:
        assert frames.dim() == 4 and frames.shape[3] == 3, "frames: [N, h, w, 3] (or rows with shapes)"
        frames = frames.contiguous()
        H, W = int(frames.shape[1]), int(frames.shape[2])
        stride = H * W * 3
    else:
        shapes = [(int(h), int(w)) for h, w in shapes]
        assert len(shapes) == n, "one (h, w) per row"
        H, W = max(max(h for h, _ in shapes), 1), max(max(w for _, w in shapes), 1)
        frames = frames.reshape(n, -1)
        assert frames.stride(1) == 1 and all(h * w * 3 <= frames.shape[1] for h, w in shapes)
        stride = frames.stride(0)
        assert stride >= H * W * 3, "rows shorter than the largest frame's H * W * 3"
        hw = torch.tensor(shapes, dtype=torch.int32).to(frames.device)
    with torch.cuda.device(frames.device):
        enc = encoder(n, H, W, params, frames.device)
        enc.encode(frames, stride, hw)
        return enc.files()
