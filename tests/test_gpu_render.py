"""plot_dgp's labelled video on the device: dgp_draw_markers and the fused render pass of estimate_pose, byte for byte against
the numpy restatement of the drawing contract (tests/test_render.py)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from deepgraphpose_b200 import synthetic
from deepgraphpose_b200._lib import DgpError

from test_render import draw_reference

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


def hard_centres(rng, N, nj, h, w, d):
    """Coordinates that visit the interior, every border, negative centres, the far side of the right / bottom edges, NaN and
    infinities, with neighbouring joints close enough to overlap."""
    specials_x = [0.0, w - 1.0, w - 0.5, -0.7, -3.2, -d - 0.5, -d + 0.5, w + 5.3, 1e12, -1e12, np.inf, -np.inf, np.nan]
    specials_y = [0.0, h - 1.0, h - 0.3, -0.7, -2.9, -d + 0.5, h + 100.0, np.inf, np.nan]
    x = rng.uniform(-2 * d, w + 2 * d, (N, nj))
    y = rng.uniform(-2 * d, h + 2 * d, (N, nj))
    for t in range(N):
        for j in range(nj):
            k = (t * nj + j)
            if k % 3 == 0:
                x[t, j] = specials_x[(k // 3) % len(specials_x)]
            if k % 4 == 1:
                y[t, j] = specials_y[(k // 4) % len(specials_y)]
            if j and k % 5 == 2:   # overlap with the previous joint
                x[t, j], y[t, j] = x[t, j - 1] + 1.5, y[t, j - 1] - 1.0
    return x, y


@pytest.mark.parametrize("nj", [1, 4, 20])
@pytest.mark.parametrize("dotsize", [0, 1, 3, 7])
def test_draw_markers_equals_reference(nj, dotsize):
    from deepgraphpose_b200.engine import Engine, marker_colors
    rng = np.random.default_rng(nj * 100 + dotsize)
    N, h, w = 9, 61, 77
    frames = rng.integers(0, 256, (N, h, w, 3), dtype=np.uint8)
    x, y = hard_centres(rng, N, nj, h, w, max(dotsize, 1))
    thr = 0.25
    lik = rng.uniform(0, 1, (N, nj))
    lik.flat[::7] = thr                 # equal to the threshold: not drawn
    lik.flat[3::11] = np.nan
    eng = Engine(nj)
    try:
        for colors in (None, rng.integers(0, 256, (nj, 3)).astype(np.uint8)):
            tab = marker_colors(nj) if colors is None else colors
            dev = torch.from_numpy(frames).cuda()
            eng.draw_markers(dev, x, y, lik, dotsize, thr, colors)
            got = dev.cpu().numpy()
            ref = draw_reference(frames, x, y, lik, dotsize, thr, tab)
            assert np.array_equal(got, ref)
            if dotsize:
                assert (ref != frames).any()
    finally:
        eng.close()


def numpy_xy(mu, stride, sx, sy):
    """eval.estimate_pose's coordinates: float64 markers * stride + stride / 2, then the resize scale."""
    m = mu.numpy().astype(np.float64)
    return (m[:, :, 1] * stride + 0.5 * stride) * sx, (m[:, :, 0] * stride + 0.5 * stride) * sy


@pytest.mark.parametrize("new_size", [None, (72, 100)])
def test_fused_render_stream(trained, new_size):
    from deepgraphpose_b200.engine import Engine, marker_colors
    nj, B = 4, 4
    T = 10   # 2.5 batches: the tail batch is short
    frames, _ = synthetic.make_video(T, H, W, nj, seed=11)
    eng = Engine(nj, location_refinement=False)
    try:
        eng.load_weights(trained)
        mu0, peak0, lik0 = eng.estimate_pose_stream(iter(frames), H, W, T, batch=B, new_size=new_size)
        thr = float(np.sort(lik0.numpy().ravel())[T * nj // 2])    # joints above, below and one equal to it
        got = []
        mu, peak, lik = eng.estimate_pose_render_stream(iter(frames), H, W, T, lambda fr: got.append(fr.copy()), dotsize=3,
                                                        mask_threshold=thr, new_size=new_size, batch=B)
        assert torch.equal(mu, mu0) and torch.equal(peak, peak0) and torch.equal(lik, lik0)
        written = np.concatenate(got)
        assert written.shape == (T, H, W, 3)
        sx, sy = (1.0, 1.0) if new_size is None else (W / new_size[1], H / new_size[0])
        x, y = numpy_xy(mu, eng.stride, sx, sy)
        ref = draw_reference(frames, x, y, lik.numpy().astype(np.float64), 3, thr, marker_colors(nj))
        assert (ref != frames).any()
        assert np.array_equal(written, ref)
    finally:
        eng.close()


def test_failing_writer_raises_and_releases(trained):
    from deepgraphpose_b200.engine import Engine
    before = live_resources()
    frames, _ = synthetic.make_video(12, H, W, 4, seed=12)
    eng = Engine(4, location_refinement=False)
    eng.load_weights(trained)
    calls = []

    def writer(fr):
        calls.append(fr.shape[0])
        return -7 if len(calls) == 2 else 0

    with pytest.raises(DgpError, match="writer failed"):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, writer, batch=4)
    assert len(calls) == 2

    def raises(fr):
        raise IOError("disk full")

    with pytest.raises(IOError):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, raises, batch=4)
    # the engine still works afterwards
    mu, _, _ = eng.estimate_pose_render_stream(iter(frames), H, W, 12, lambda fr: None, batch=4)
    assert mu.shape[0] == 12
    eng.close()
    assert live_resources() == before


def write_ffv1(path, frames, fps=25.0):
    import cv2
    vw = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"FFV1"), fps, (frames.shape[2], frames.shape[1]))
    assert vw.isOpened()
    for fr in frames:
        vw.write(np.ascontiguousarray(fr[:, :, ::-1]))
    vw.release()


def read_video(path):
    import cv2
    cap = cv2.VideoCapture(str(path))
    out = []
    while True:
        ok, fr = cap.read()
        if not ok:
            break
        out.append(fr[:, :, ::-1])
    cap.release()
    return np.stack(out)


def test_plot_dgp_end_to_end(tmp_path, trained):
    from deepgraphpose_b200 import eval as E
    nj, T = 4, 10
    frames, _ = synthetic.make_video(T, H, W, nj, seed=13)
    video = tmp_path / "reach.avi"
    write_ffv1(video, frames)
    src = read_video(video)
    assert np.array_equal(src, frames)
    cfg = {"num_joints": nj, "stride": 8.0}
    est = E.estimate_pose(cfg, trained, str(video), str(tmp_path / "est"), batch=4)
    thr = float(np.sort(est["likelihoods"].ravel())[T * nj // 2])
    out_dir = tmp_path / "out"
    movie = E.plot_dgp(str(video), output_dir=str(out_dir), proj_cfg_file=cfg, dgp_model_file=trained, mask_threshold=thr,
                       batch=4, fourcc="FFV1")
    assert movie == str(out_dir / "reach_labeled.mp4")
    csv = out_dir / "reach_labeled.csv"
    assert csv.read_bytes() == (tmp_path / "est" / "reach_labeled.csv").read_bytes()
    labels = E.load_pose_from_dlc_to_dict(str(csv))
    ref = draw_reference(src, labels["x"], labels["y"], labels["likelihoods"], 3, thr, E.marker_colors(nj))
    assert (ref != src).any()
    fused = read_video(movie)
    assert np.array_equal(fused, ref)
    # an existing movie is kept; without it, the csv drives a render-only pass that writes the same frames
    assert E.plot_dgp(str(video), output_dir=str(out_dir), fourcc="FFV1") == movie
    os.remove(movie)
    E.plot_dgp(str(video), output_dir=str(out_dir), mask_threshold=thr, batch=3, fourcc="FFV1")
    assert np.array_equal(read_video(movie), fused)
