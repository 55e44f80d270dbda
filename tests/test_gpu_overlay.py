"""Skeleton lines and joint trails of plot_dgp's labelled video on the device: dgp_draw_markers and the fused render passes
(raw and Motion-JPEG) byte for byte against the numpy restatement of the overlay contract (tests/test_overlay.py)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from deepgraphpose_b200 import synthetic
from deepgraphpose_b200._lib import DgpError

from test_overlay import draw_overlay_reference
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


def hard_labels(rng, N, nj, h, w, d, thr):
    """Random labels with off-frame and far endpoints (both sides of the -2^20 bound), NaN / infinities, masked joints,
    likelihoods equal to the threshold, and neighbours close enough for trails, lines and discs to overlap."""
    specials = [0.0, w - 1.0, -0.7, -d - 0.5, w + 5.3, 3 * w, -3 * w, 1e7, -1e7, -1048576.9, -1048577.0, 1e12, np.inf,
                -np.inf, np.nan]
    x = rng.uniform(-2 * d, w + 2 * d, (N, nj))
    y = rng.uniform(-2 * d, h + 2 * d, (N, nj))
    for t in range(1, N):   # slow drift for half the joints: trail discs overlap the current ones
        x[t, ::2] = x[t - 1, ::2] + rng.uniform(-2, 2, x[t, ::2].shape)
        y[t, ::2] = y[t - 1, ::2] + rng.uniform(-2, 2, y[t, ::2].shape)
    flat = rng.choice(N * nj, size=max(1, N * nj // 4), replace=False)
    for n, i in enumerate(flat):
        (x if n % 2 else y).flat[i] = specials[n % len(specials)]
    lik = rng.uniform(0, 1, (N, nj))
    lik.flat[::7] = thr
    lik.flat[5::13] = np.nan
    return x, y, lik


def edge_table(rng, nj):
    if nj == 1:
        return [(0, 0)]
    chain = [(j, j + 1) for j in range(nj - 1)]
    return chain + [tuple(int(v) for v in rng.integers(0, nj, 2)) for _ in range(nj)]


@pytest.mark.parametrize("nj", [1, 4, 20])
@pytest.mark.parametrize("K", [0, 1, 2, 10, 64])
def test_draw_overlay_equals_reference(nj, K):
    from deepgraphpose_b200.engine import Engine, marker_colors
    rng = np.random.default_rng(nj * 1000 + K)
    N, h, w, d, thr = 12, 61, 77, 3, 0.25
    frames = rng.integers(0, 256, (N, h, w, 3), dtype=np.uint8)
    x, y, lik = hard_labels(rng, N, nj, h, w, d, thr)
    edges = edge_table(rng, nj)
    sk = tuple(int(v) for v in rng.integers(0, 256, 3))
    colors = marker_colors(nj)
    ref = draw_overlay_reference(frames, x, y, lik, d, thr, colors, edges, sk, K)
    if nj > 1 or K > 1:   # (nj 1's only edge is one pixel under its disc)
        assert (ref != draw_overlay_reference(frames, x, y, lik, d, thr, colors)).any()   # the overlay shows
    eng = Engine(nj)
    try:
        # all frames in one call, then in two calls whose second one gets the trail rows as history
        dev = torch.from_numpy(frames).cuda()
        eng.draw_markers(dev, x, y, lik, d, thr, None, edges, sk, K)
        assert np.array_equal(dev.cpu().numpy(), ref)
        n1 = 5
        hist = min(max(K - 1, 0), n1)
        a, b = torch.from_numpy(frames[:n1]).cuda(), torch.from_numpy(frames[n1:]).cuda()
        eng.draw_markers(a, x[:n1], y[:n1], lik[:n1], d, thr, None, edges, sk, K)
        eng.draw_markers(b, x[n1 - hist:], y[n1 - hist:], lik[n1 - hist:], d, thr, None, edges, sk, K, hist)
        assert np.array_equal(np.concatenate([a.cpu().numpy(), b.cpu().numpy()]), ref)
        # lines alone (dotsize 0)
        dev = torch.from_numpy(frames).cuda()
        eng.draw_markers(dev, x, y, lik, 0, thr, None, edges, sk, K)
        assert np.array_equal(dev.cpu().numpy(), draw_overlay_reference(frames, x, y, lik, 0, thr, colors, edges, sk, K))
    finally:
        eng.close()


def test_long_lines_and_overlay_off():
    """Lines across a 1080x1920 frame from far off it, and the markers-only bytes with the overlay off."""
    from deepgraphpose_b200.engine import Engine, marker_colors
    rng = np.random.default_rng(5)
    N, h, w, nj = 3, 1080, 1920, 4
    frames = rng.integers(0, 256, (N, h, w, 3), dtype=np.uint8)
    x = np.array([[-900000.5, 2500.0, 10.0, 1919.9], [5.0, 1e9, -40000.0, 960.0], [100.0, 101.0, 100.0, 1e7]])
    y = np.array([[-700000.0, 1079.5, 3000.0, 0.0], [1070.0, 20.0, 540.0, -1048576.0], [5.0, 1079.0, 1000.0, 300.0]])
    lik = np.ones((N, nj))
    edges = [(0, 1), (1, 2), (2, 3), (3, 0), (0, 2)]
    eng = Engine(nj)
    try:
        dev = torch.from_numpy(frames).cuda()
        eng.draw_markers(dev, x, y, lik, 4, 0.5, None, edges, (255, 0, 0), 2)
        ref = draw_overlay_reference(frames, x, y, lik, 4, 0.5, marker_colors(nj), edges, (255, 0, 0), 2)
        assert np.array_equal(dev.cpu().numpy(), ref)
        for K in (0, 1):
            dev = torch.from_numpy(frames).cuda()
            eng.draw_markers(dev, x, y, lik, 4, 0.5, None, None, (255, 0, 0), K)
            assert np.array_equal(dev.cpu().numpy(), draw_reference(frames, x, y, lik, 4, 0.5, marker_colors(nj)))
    finally:
        eng.close()


def numpy_xy(mu, stride):
    m = mu.numpy().astype(np.float64)
    return m[:, :, 1] * stride + 0.5 * stride, m[:, :, 0] * stride + 0.5 * stride


def test_fused_overlay_is_batch_independent(trained, tmp_path):
    from deepgraphpose_b200 import eval as E
    from deepgraphpose_b200.engine import Engine, marker_colors
    nj, T, K = 4, 75, 10
    frames, _ = synthetic.make_video(T, H, W, nj, seed=21)
    edges = [(0, 1), (1, 2), (2, 3), (3, 0)]
    sk = (250, 10, 20)
    eng = Engine(nj, location_refinement=False)
    try:
        eng.load_weights(trained)
        mu0, peak0, lik0 = eng.estimate_pose_stream(iter(frames), H, W, T, batch=7)
        thr = float(np.sort(lik0.numpy().ravel())[T * nj // 3])
        style = dict(dotsize=3, mask_threshold=thr, edges=edges, skeleton_color=sk, trailpoints=K)
        raw, jpeg = {}, {}
        for B in (7, 31):
            got = []
            out = eng.estimate_pose_render_stream(iter(frames), H, W, T, lambda fr: got.append(fr.copy()), batch=B, **style)
            assert all(torch.equal(p, q) for p, q in zip(out, (mu0, peak0, lik0)))
            raw[B] = np.concatenate(got)
            pk = []
            out = eng.estimate_pose_render_stream(iter(frames), H, W, T, lambda d, s: pk.append((d.copy(), s.copy())),
                                                  batch=B, encoder="jpeg", quality=85, **style)
            assert all(torch.equal(p, q) for p, q in zip(out, (mu0, peak0, lik0)))
            jpeg[B] = [bytes(d[o - s_:o]) for d, s in pk for o, s_ in zip(np.cumsum(s), s)]
        assert np.array_equal(raw[7], raw[31]) and jpeg[7] == jpeg[31]
        x, y = numpy_xy(mu0, eng.stride)
        lk = lik0.numpy().astype(np.float64)
        ref = draw_overlay_reference(frames, x, y, lk, 3, thr, marker_colors(nj), edges, sk, K)
        assert np.array_equal(raw[7], ref)
        assert jpeg[7] == eng.encode_jpeg(torch.from_numpy(raw[7]).cuda(), 85)
        # the render-only path on the same coordinates, batch by batch with history rows
        movie = tmp_path / "csv_branch.avi"
        E.create_annotated_movie(frames, x, y, lk > thr, dotsize=3, filename=str(movie), fps=25.0, fourcc="FFV1",
                                 batch=6, engine=eng, skeleton=edges, skeleton_color=sk, trailpoints=K)
        from test_gpu_render import read_video
        assert np.array_equal(read_video(movie), raw[7])
    finally:
        eng.close()


def test_failing_writer_with_overlay_releases(trained):
    from deepgraphpose_b200.engine import Engine
    before = live_resources()
    frames, _ = synthetic.make_video(12, H, W, 4, seed=12)
    eng = Engine(4, location_refinement=False)
    eng.load_weights(trained)
    style = dict(edges=[(0, 1), (2, 3)], skeleton_color=(9, 9, 9), trailpoints=5)
    calls = []

    def writer(fr):
        calls.append(fr.shape[0])
        return -7 if len(calls) == 2 else 0

    with pytest.raises(DgpError, match="writer failed"):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, writer, batch=3, **style)
    assert len(calls) == 2
    with pytest.raises(DgpError, match="writer failed"):
        eng.estimate_pose_render_stream(iter(frames), H, W, 12, lambda d, s: -3, batch=3, encoder="jpeg", **style)
    mu, _, _ = eng.estimate_pose_render_stream(iter(frames), H, W, 12, lambda fr: None, batch=4, **style)
    assert mu.shape[0] == 12
    eng.close()
    assert live_resources() == before


def test_plot_dgp_overlay_branches_agree(tmp_path, trained):
    from deepgraphpose_b200 import eval as E
    from test_gpu_render import read_video, write_ffv1
    nj, T = 4, 23
    frames, _ = synthetic.make_video(T, H, W, nj, seed=31)
    video = tmp_path / "walk.avi"
    write_ffv1(video, frames)
    cfg = {"num_joints": nj, "stride": 8.0, "all_joints_names": ["a", "b", "c", "d"],
           "skeleton": [["a", "b"], ["b", "c"], ["d", "a"]]}
    kw = dict(draw_skeleton=True, skeleton_color=(0, 255, 0), trailpoints=5, fourcc="FFV1", mask_threshold=0.05)
    out_dir = tmp_path / "out"
    movie = E.plot_dgp(str(video), output_dir=str(out_dir), proj_cfg_file=cfg, dgp_model_file=trained, batch=4, **kw)
    fused = read_video(movie)
    plain = E.plot_dgp(str(video), output_dir=str(tmp_path / "plain"), proj_cfg_file=cfg, dgp_model_file=trained, batch=4,
                       fourcc="FFV1", mask_threshold=0.05)
    assert not np.array_equal(fused, read_video(plain))
    os.remove(movie)
    E.plot_dgp(str(video), output_dir=str(out_dir), proj_cfg_file=cfg, batch=3, **kw)   # the csv branch
    assert np.array_equal(read_video(movie), fused)
