"""Motion-JPEG on the device: dgp_encode_jpeg and the fused estimate_pose / render / encode pass, byte for byte against
Pillow's encoder (whose bytes tests/test_jpeg.py pins to the numpy restatement of the contract)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from deepgraphpose_b200 import synthetic
from deepgraphpose_b200._lib import DgpError

from test_jpeg import QUALITIES, SIZES, frames_of, pillow_jpeg

pytestmark = pytest.mark.gpu
H, W = 96, 128


def live_resources():
    from deepgraphpose_b200 import _lib
    objs, nbytes = C.c_int64(), C.c_int64()
    _lib.load().dgp_debug_live_resources(C.byref(objs), C.byref(nbytes))
    return objs.value, nbytes.value


@pytest.fixture(scope="module")
def trained():
    return synthetic.make_weights(4, seed=3, location_refinement=False, trained_like=True)


@pytest.fixture(scope="module")
def engine():
    from deepgraphpose_b200.engine import Engine
    eng = Engine(4)
    yield eng
    eng.close()


@pytest.mark.parametrize("H,W", SIZES)
def test_encode_jpeg_equals_pillow(engine, H, W):
    imgs = frames_of(H, W)
    batch = torch.from_numpy(np.stack(list(imgs.values()))).cuda()
    for q in QUALITIES:
        got = engine.encode_jpeg(batch, q)
        for (name, img), g in zip(imgs.items(), got):
            assert g == pillow_jpeg(img, q), (name, q, len(g))


def test_bytes_independent_of_batch_and_position(engine):
    rng = np.random.default_rng(1)
    frames = synthetic.make_video(7, 75, 99, 4, seed=2)[0]
    frames[3] = rng.integers(0, 256, frames[3].shape, dtype=np.uint8)
    ref = [pillow_jpeg(np.ascontiguousarray(f), 85) for f in frames]
    dev = torch.from_numpy(frames).cuda()
    assert engine.encode_jpeg(dev, 85) == ref
    for k in range(7):
        assert engine.encode_jpeg(dev[k:k + 1], 85) == [ref[k]]
    perm = [5, 3, 0, 6, 1, 4, 2]
    assert engine.encode_jpeg(dev[perm], 85) == [ref[k] for k in perm]
    assert engine.encode_jpeg(dev[:0], 85) == []


def test_noise_q100_within_capacity(engine):
    from deepgraphpose_b200.engine import jpeg_capacity
    for h, w in ((747, 832), (1080, 1920), (16, 16383)):
        img = np.random.default_rng(h).integers(0, 256, (2, h, w, 3), dtype=np.uint8)
        got = engine.encode_jpeg(torch.from_numpy(img).cuda(), 100)
        for g, f in zip(got, img):
            assert len(g) <= jpeg_capacity(h, w)
            assert g == pillow_jpeg(f, 100)


def test_encode_jpeg_rejects_bad_arguments(engine):
    from deepgraphpose_b200 import _lib
    dev = torch.zeros((2, 8, 8, 3), dtype=torch.uint8, device="cuda")
    for q in (0, 101, 50.5):
        with pytest.raises(ValueError):
            engine.encode_jpeg(dev, q)
    out = torch.empty(10, dtype=torch.uint8, device="cuda")
    meta = torch.empty(4, dtype=torch.int64, device="cuda")
    rc = engine.lib.dgp_encode_jpeg(engine.h, C.c_void_p(dev.data_ptr()), 2, 8, 8, 90, C.c_void_p(out.data_ptr()), 10,
                                    C.c_void_p(meta.data_ptr()), C.c_void_p(meta.data_ptr() + 16), None)
    assert rc == -1 and b"capacity" in _lib.load().dgp_last_error(engine.h)


@pytest.mark.parametrize("new_size", [None, (72, 100)])
def test_fused_jpeg_stream(trained, new_size):
    from deepgraphpose_b200.engine import Engine
    nj, B, T = 4, 4, 10   # 2.5 batches: the tail batch is short
    frames, _ = synthetic.make_video(T, H, W, nj, seed=11)
    eng = Engine(nj, location_refinement=False)
    try:
        eng.load_weights(trained)
        mu0, peak0, lik0 = eng.estimate_pose_stream(iter(frames), H, W, T, batch=B, new_size=new_size)
        thr = float(np.sort(lik0.numpy().ravel())[T * nj // 2])
        raw = []
        eng.estimate_pose_render_stream(iter(frames), H, W, T, lambda fr: raw.append(fr.copy()), dotsize=3,
                                        mask_threshold=thr, new_size=new_size, batch=B)
        packets, per_call = [], []

        def writer(data, sizes):
            per_call.append(len(sizes))
            o = 0
            for s in sizes:
                packets.append(bytes(data[o:o + s]))
                o += int(s)

        mu, peak, lik = eng.estimate_pose_render_stream(iter(frames), H, W, T, writer, dotsize=3, mask_threshold=thr,
                                                        new_size=new_size, batch=B, encoder="jpeg", quality=75)
        assert torch.equal(mu, mu0) and torch.equal(peak, peak0) and torch.equal(lik, lik0)
        assert per_call == [4, 4, 2]
        drawn = np.concatenate(raw)
        assert (drawn != frames).any()
        assert packets == [pillow_jpeg(f, 75) for f in drawn]
    finally:
        eng.close()


def test_failing_packet_writer_raises_and_releases(trained):
    from deepgraphpose_b200.engine import Engine
    before = live_resources()
    frames, _ = synthetic.make_video(12, H, W, 4, seed=12)
    eng = Engine(4, location_refinement=False)
    eng.load_weights(trained)
    calls = []

    def writer(data, sizes):
        calls.append(len(sizes))
        return -7 if len(calls) == 2 else 0

    with pytest.raises(DgpError, match="writer failed"):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, writer, batch=4, encoder="jpeg")
    assert len(calls) == 2

    def raises(data, sizes):
        raise IOError("disk full")

    with pytest.raises(IOError):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, raises, batch=4, encoder="jpeg")
    with pytest.raises(ValueError):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, lambda d, s: None, batch=4, encoder="jpeg", quality=0)
    mu, _, _ = eng.estimate_pose_render_stream(iter(frames), H, W, 12, lambda d, s: None, batch=4, encoder="jpeg")
    assert mu.shape[0] == 12
    eng.encode_jpeg(torch.from_numpy(frames).cuda())
    eng.close()
    assert live_resources() == before


def test_plot_dgp_jpeg_end_to_end(tmp_path, trained):
    import cv2
    from deepgraphpose_b200 import eval as E
    from test_gpu_render import read_video, write_ffv1
    from test_render import draw_reference
    nj, T = 4, 10
    frames, _ = synthetic.make_video(T, H, W, nj, seed=13)
    video = tmp_path / "reach.avi"
    write_ffv1(video, frames, fps=29.97)
    cfg = {"num_joints": nj, "stride": 8.0}
    est = E.estimate_pose(cfg, trained, str(video), str(tmp_path / "est"), batch=4)
    thr = float(np.sort(est["likelihoods"].ravel())[T * nj // 2])
    cv_dir, jpg_dir = tmp_path / "cv2", tmp_path / "jpeg"
    E.plot_dgp(str(video), output_dir=str(cv_dir), proj_cfg_file=cfg, dgp_model_file=trained, mask_threshold=thr, batch=4,
               fourcc="FFV1")
    movie = E.plot_dgp(str(video), output_dir=str(jpg_dir), proj_cfg_file=cfg, dgp_model_file=trained, mask_threshold=thr,
                       batch=4, encoder="jpeg", quality=90)
    assert movie == str(jpg_dir / "reach_labeled.mp4")
    assert (jpg_dir / "reach_labeled.csv").read_bytes() == (cv_dir / "reach_labeled.csv").read_bytes()
    cap = cv2.VideoCapture(movie)
    assert abs(cap.get(cv2.CAP_PROP_FPS) - 29.97) < 1e-3
    cap.release()
    fused = read_video(movie)
    assert fused.shape == (T, H, W, 3)
    labels = E.load_pose_from_dlc_to_dict(str(jpg_dir / "reach_labeled.csv"))
    ref = draw_reference(frames, labels["x"], labels["y"], labels["likelihoods"], 3, thr, E.marker_colors(nj))
    assert np.abs(fused.astype(int) - ref.astype(int)).mean() < 4.0
    # the csv branch (draw_markers + encode_jpeg) writes the same bytes as the fused pass
    first = open(movie, "rb").read()
    os.remove(movie)
    E.plot_dgp(str(video), output_dir=str(jpg_dir), mask_threshold=thr, batch=3, encoder="jpeg", quality=90)
    assert open(movie, "rb").read() == first
