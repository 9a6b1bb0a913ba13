"""Pose overlays drawn on the GPU (pn_draw_poses) against the host helpers, byte for byte: draw_skel_and_kp_batch /
draw_skeleton_batch vs draw_skel_and_kp / draw_skeleton per image (on a copy), and BatchPipeline(overlay=...) vs the host loop
of image_demo.py (decode, scale to the frame, draw_skel_and_kp)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import posenet  # noqa: E402
from oracle import net as onet  # noqa: E402
from oracle import synth  # noqa: E402

DEV = "cuda"
THRESHOLDS = [(0.0, 0.0), (0.25, 0.25), (0.5, 0.5)]


def model(os_=16):
    sd = onet.init_params(50, seed=5, scheme="scaled", gain=0.8)
    m = posenet.MobileNetV1(50, output_stride=os_)
    m.load_state_dict(sd)
    return m.cuda().set_compute_dtype("bf16")


def host_draw(frames, ps, ks, kc, mp, mk, skeleton_only=False):
    fn = posenet.draw_skeleton if skeleton_only else posenet.draw_skel_and_kp
    return np.stack([fn(f.copy(), ps[i], ks[i], kc[i], mp, mk) for i, f in enumerate(frames)])


def check_batch(frames_np, ps, ks, kc):
    """Both batch helpers at every threshold pair equal the host helpers applied per image."""
    t = lambda a: torch.as_tensor(a, device=DEV)
    for mp, mk in THRESHOLDS:
        for skeleton_only in (False, True):
            fr = torch.from_numpy(frames_np).to(DEV)
            fn = posenet.draw_skeleton_batch if skeleton_only else posenet.draw_skel_and_kp_batch
            out = fn(fr, t(ps), t(ks), t(kc), mp, mk)
            assert out is fr
            ref = host_draw(frames_np, ps, ks, kc, mp, mk, skeleton_only)
            got = fr.cpu().numpy()
            assert np.array_equal(got, ref), (frames_np.shape, mp, mk, skeleton_only, int((got != ref).sum()))


@pytest.mark.parametrize("hw", [(513, 513), (257, 257), (720, 1280)])
def test_batch_draw_on_decoded_records(hw):
    """Records decoded by the model from seeded frames, mapped back to the frames' pixels (source coordinates)."""
    H, W = hw
    m = model()
    frames = np.stack([synth.smooth_image(H, W, 100 + i) for i in range(2)])
    x, scale = posenet.resize_u8_gpu(frames, 1.0, 16)
    ps, ks, kc, _, _ = posenet.decode_multiple_poses_batch(*m.forward_u8(x), output_stride=16, max_pose_detections=10,
                                                           min_pose_score=0.1)
    kc = kc * torch.as_tensor(scale, device=DEV)                 # image_demo.py:50
    ps, ks, kc = ps.cpu().numpy(), ks.cpu().numpy(), kc.cpu().numpy()
    assert ps.max() > 0
    check_batch(frames, ps, ks, kc)


def crowd(rng, n, P, H, W):
    ps = np.where(rng.uniform(size=(n, P)) < 0.8, np.sort(rng.uniform(0, 1, (n, P)))[:, ::-1], 0.)
    ps[:, ::7] = 0.25                                               # exactly at a threshold
    ks = rng.uniform(0, 1, (n, P, 17))
    ks[rng.uniform(size=(n, P, 17)) < 0.1] = 0.25
    ks[rng.uniform(size=(n, P, 17)) < 0.05] = 0.5
    kc = np.stack([rng.uniform(-20, H + 20, (n, P, 17)), rng.uniform(-20, W + 20, (n, P, 17))], -1)
    kc[:, :, :5] = np.round(kc[:, :, :5] * 32) / 32
    return ps, ks, kc


@pytest.mark.parametrize("n,H,W", [(1, 513, 513), (64, 257, 257), (64, 33, 47), (1, 720, 1280), (3, 129, 383)])
def test_batch_draw_synthetic_crowds(n, H, W):
    rng = np.random.default_rng(n * 1000 + W)
    P = 50
    frames = rng.integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    check_batch(frames, *crowd(rng, n, P, H, W))


def test_strided_frames_and_guard_bytes():
    """Frames further apart than their size (a view of taller frames) and guard bytes around the buffer stay untouched."""
    rng = np.random.default_rng(7)
    n, H, W, Hb, G = 5, 61, 77, 70, 4096
    ps, ks, kc = crowd(rng, n, 50, H, W)
    kc[:, :3] *= 1e6                                                # far outside the frames
    buf = torch.from_numpy(rng.integers(0, 256, G + n * Hb * W * 3 + G, dtype=np.uint8)).to(DEV)
    before = buf.cpu().numpy()
    frames = buf[G:G + n * Hb * W * 3].view(n, Hb, W, 3)[:, :H]
    assert frames.stride(0) == Hb * W * 3
    t = lambda a: torch.as_tensor(a, device=DEV)
    mp, mk = 0.25, 0.25
    posenet.draw_skel_and_kp_batch(frames, t(ps), t(ks), t(kc), mp, mk)
    after = buf.cpu().numpy()
    ref = host_draw(before[G:G + n * Hb * W * 3].reshape(n, Hb, W, 3)[:, :H], ps, ks, kc, mp, mk)
    assert np.array_equal(frames.cpu().numpy(), ref)
    assert np.array_equal(after[:G], before[:G]) and np.array_equal(after[-G:], before[-G:])
    gaps_a = after[G:G + n * Hb * W * 3].reshape(n, Hb, W, 3)[:, H:]
    gaps_b = before[G:G + n * Hb * W * 3].reshape(n, Hb, W, 3)[:, H:]
    assert np.array_equal(gaps_a, gaps_b)


def _host_loop(batches, recs, mp, mk, shapes=None):
    """image_demo.py per frame: the records of the frame (already in its pixels), draw_skel_and_kp on the frame itself."""
    out = []
    for b, rec in zip(batches, recs):
        ps, ks, kc = rec[:3]
        if shapes is None:
            out.append(host_draw(b.numpy(), ps, ks, kc, mp, mk))
        else:
            rows = b.numpy().reshape(b.shape[0], -1)
            out.append([posenet.draw_skel_and_kp(rows[i, :h * w * 3].reshape(h, w, 3).copy(), ps[i], ks[i], kc[i], mp, mk)
                        for i, (h, w) in enumerate(shapes)])
    return out


@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("mode", ["uniform", "resize", "mixed"])
def test_pipeline_overlay(mode, use_graph):
    mp, mk = 0.1, 0.1
    kw = dict(max_pose_detections=8, min_pose_score=0.05)
    if mode == "uniform":
        N, H, W, os_ = 3, 129, 161, 16
    elif mode == "resize":
        N, H, W, os_ = 2, 180, 320, 8
    else:
        N, H, W, os_ = 3, 161, 200, 16
    m = model(os_)
    if mode == "mixed":
        sizes = [[(129, 161), (100, 141), (161, 129)], [(64, 65), (150, 200)]]
        batches, items = [], []
        for b, shp in enumerate(sizes):
            hb = torch.zeros((N, H * W * 3), dtype=torch.uint8)
            for i, (h, w) in enumerate(shp):
                hb[i, :h * w * 3] = torch.from_numpy(synth.smooth_image(h, w, 50 + 10 * b + i).reshape(-1))
            hb = hb.pin_memory()
            batches.append(hb)
            items.append((hb, shp))
        common = dict(mixed=True, source_coords=True)
    else:
        batches = [torch.from_numpy(np.stack([synth.smooth_image(H, W, 20 * b + i) for i in range(N)])).pin_memory() for b in range(3)]
        items = batches
        common = dict(source_coords=(mode == "resize"))
    plain = list(posenet.BatchPipeline(m, N, H, W, depth=2, output_stride=os_, use_graph=use_graph, **common, **kw).run(items))
    pipe = posenet.BatchPipeline(m, N, H, W, depth=2, output_stride=os_, use_graph=use_graph, overlay=(mp, mk), **common, **kw)
    got = list(pipe.run(items))
    assert len(got) == len(plain) and any(r[0].max() > 0 for r in plain)
    for g, p in zip(got, plain):
        assert len(g) == 5
        for a, b in zip(g[:4], p):
            assert np.array_equal(a, b)
    if mode == "mixed":
        for k, (g, shp) in enumerate(zip(got, sizes)):
            ref = _host_loop([batches[k]], [plain[k]], mp, mk, shp)[0]
            assert len(g[4]) == len(shp)
            for a, b in zip(g[4], ref):
                assert np.array_equal(a, b)
    else:
        ref = _host_loop(batches, plain, mp, mk)
        for g, r in zip(got, ref):
            assert g[4].shape == (N, H, W, 3) and np.array_equal(g[4], r)
    if mode == "resize":
        with pytest.raises(AssertionError):
            posenet.BatchPipeline(m, N, H, W, output_stride=os_, overlay=(mp, mk), **kw)   # needs source_coords
