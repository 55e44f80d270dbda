"""Skeleton lines and joint trails of plot_dgp's labelled video without a GPU: the numpy restatement of the overlay contract
(include/dgp_b200.h, DESIGN.md §4.5) that the device kernel is compared against, its own checks (line shape, clipping, the
skip rules, the painting order) and the argument validation of every entry."""
import os

import numpy as np
import pytest

MIN_CENTRE = -2 ** 20


def _centre(x, y, lik, thr, H, W):
    """The disc rule's mask and centre: (xc, yc) as Python floats, or None when the joint is not drawn."""
    x, y, lik = float(x), float(y), float(lik)
    if not lik > thr or np.isnan(x) or np.isnan(y):
        return None
    return min(np.trunc(x), W - 1.0), min(np.trunc(y), H - 1.0)


def paint_disc(frame, x, y, lik, dotsize, thr, colour):
    H, W, _ = frame.shape
    c = _centre(x, y, lik, thr, H, W)
    if c is None or dotsize == 0:
        return
    xc, yc = c
    if xc <= -dotsize or yc <= -dotsize:
        return
    xc, yc = int(xc), int(yc)
    r0, r1, c0, c1 = max(yc - dotsize + 1, 0), min(yc + dotsize, H), max(xc - dotsize + 1, 0), min(xc + dotsize, W)
    if r0 >= r1 or c0 >= c1:
        return
    rr, cc = np.ogrid[r0:r1, c0:c1]
    frame[r0:r1, c0:c1][(rr - yc) ** 2 + (cc - xc) ** 2 < dotsize * dotsize] = colour


def line_offsets(k, d, n):
    """floor((2 k d + n) / 2n) for the int64 array k (0 when n == 0)."""
    if n == 0:
        return np.zeros_like(k)
    return np.floor_divide(2 * k * d + n, 2 * n)


def full_line(ra, ca, rb, cb):
    """Every pixel k = 0..n of the line, on an unbounded canvas."""
    dr, dc = rb - ra, cb - ca
    n = max(abs(dr), abs(dc))
    k = np.arange(n + 1, dtype=np.int64)
    return ra + line_offsets(k, dr, n), ca + line_offsets(k, dc, n)


def _clip_axis(p0, d, n, hi, k0, k1):
    """The k whose coordinate p0 + floor((2kd + n) / 2n) lies in [0, hi], intersected with [k0, k1] (exact integers)."""
    if d == 0:
        return (k0, k1) if 0 <= p0 <= hi else (k0, -1)
    if d > 0:
        lo_k = -((2 * n * p0 + n) // (2 * d))
        hi_k = (2 * n * (hi + 1 - p0) - n - 1) // (2 * d)
    else:
        e = -d
        lo_k = -((2 * n * (hi + 1 - p0) - n - 1) // (2 * e))
        hi_k = (n + 2 * n * p0) // (2 * e)
    return max(k0, lo_k), min(k1, hi_k)


def visible_line(ra, ca, rb, cb, H, W):
    """The pixels of the line inside an H x W frame, from the visible k range only (never the off-frame part)."""
    dr, dc = rb - ra, cb - ca
    n = max(abs(dr), abs(dc))
    k0, k1 = _clip_axis(ra, dr, n, H - 1, 0, n)
    k0, k1 = _clip_axis(ca, dc, n, W - 1, k0, k1)
    k = np.arange(k0, k1 + 1, dtype=np.int64) if k0 <= k1 else np.zeros(0, np.int64)
    return ra + line_offsets(k, dr, n), ca + line_offsets(k, dc, n)


def line_endpoints(xa, ya, la, xb, yb, lb, thr, H, W):
    """(ra, ca, rb, cb) of a skeleton edge, or None when it is skipped: either joint masked, a non-finite coordinate or a
    centre below -2^20."""
    a, b = _centre(xa, ya, la, thr, H, W), _centre(xb, yb, lb, thr, H, W)
    if a is None or b is None or not np.isfinite([xa, ya, xb, yb]).all():
        return None
    if min(a + b) < MIN_CENTRE:
        return None
    return int(a[1]), int(a[0]), int(b[1]), int(b[0])


def draw_overlay_reference(frames, x, y, lik, dotsize, thr, colors, edges=(), skeleton_color=(0, 0, 0), trailpoints=0,
                           history=0):
    """The overlay contract in numpy: frames uint8 (N,H,W,3); x / y / lik float64 (history + N, nj), row history + t being
    frame t -> annotated copy.  Per frame: trail discs (k = K-1 .. 1, joints in order), skeleton lines, then the discs."""
    out = np.array(frames, dtype=np.uint8, copy=True)
    N, H, W, _ = out.shape
    nj = x.shape[1]
    edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    for t in range(N):
        i = history + t
        for k in range(trailpoints - 1, 0, -1):
            if i - k < 0:
                continue
            for j in range(nj):
                paint_disc(out[t], x[i - k, j], y[i - k, j], lik[i - k, j], dotsize, thr, colors[j])
        for a, b in edges:
            e = line_endpoints(x[i, a], y[i, a], lik[i, a], x[i, b], y[i, b], lik[i, b], thr, H, W)
            if e is not None:
                rr, cc = visible_line(*e, H, W)
                out[t][rr, cc] = skeleton_color
        for j in range(nj):
            paint_disc(out[t], x[i, j], y[i, j], lik[i, j], dotsize, thr, colors[j])
    return out


def test_line_shape():
    rng = np.random.default_rng(0)
    pts = [(0, 0, 0, 0), (3, 4, 3, 4), (0, 0, 0, 9), (0, 0, 9, 0), (5, 5, -3, -3), (0, 0, 7, 3), (2, 9, -4, 1)]
    pts += [tuple(int(v) for v in rng.integers(-50, 50, 4)) for _ in range(300)]
    for ra, ca, rb, cb in pts:
        r, c = full_line(ra, ca, rb, cb)
        n = max(abs(rb - ra), abs(cb - ca))
        assert len(r) == n + 1
        assert (r[0], c[0]) == (ra, ca) and (r[-1], c[-1]) == (rb, cb)
        assert len(set(zip(r.tolist(), c.tolist()))) == n + 1
        if n:
            # 8-connected, and the long axis advances by one pixel per step
            assert np.abs(np.diff(r)).max() <= 1 and np.abs(np.diff(c)).max() <= 1
            assert (np.maximum(np.abs(np.diff(r)), np.abs(np.diff(c))) == 1).all()
        # monotone on both axes (what the clipping relies on)
        assert (np.diff(r) * np.sign(rb - ra) >= 0).all() and (np.diff(c) * np.sign(cb - ca) >= 0).all()
    # a shallow line steps down where 2k dr + n crosses a multiple of 2n
    r, c = full_line(0, 0, 2, 5)
    assert list(zip(r.tolist(), c.tolist())) == [(0, 0), (0, 1), (1, 2), (1, 3), (2, 4), (2, 5)]


def test_clipping_equals_padded_canvas():
    rng = np.random.default_rng(1)
    for H, W in ((1, 1), (5, 9), (37, 23), (120, 200)):
        for _ in range(250):
            span = int(rng.choice([3, 40, 4000]))
            ra, rb = (int(v) for v in rng.integers(-span, H + span, 2))
            ca, cb = (int(v) for v in rng.integers(-span, W + span, 2))
            r, c = full_line(ra, ca, rb, cb)
            keep = (r >= 0) & (r < H) & (c >= 0) & (c < W)
            vr, vc = visible_line(ra, ca, rb, cb, H, W)
            assert np.array_equal(vr, r[keep]) and np.array_equal(vc, c[keep]), (H, W, ra, ca, rb, cb)
    # a line far off the frame that crosses it: the visible range is found without walking the far part
    vr, vc = visible_line(-1_000_000, -999_990, 1_000_000, 1_000_010, 40, 60)
    assert len(vr) > 0 and vr.min() >= 0 and vr.max() < 40 and vc.min() >= 0 and vc.max() < 60


def test_skip_rules():
    H, W, thr = 30, 40, 0.5
    assert line_endpoints(1.5, 2.5, 1, 30.9, 20.1, 1, thr, H, W) == (2, 1, 20, 30)
    assert line_endpoints(1.5, 2.5, 1, 30.9, 20.1, thr, thr, H, W) is None           # equal to the threshold: masked
    assert line_endpoints(1.5, 2.5, np.nan, 3, 4, 1, thr, H, W) is None
    for bad in (np.nan, np.inf, -np.inf):
        assert line_endpoints(bad, 2.5, 1, 3, 4, 1, thr, H, W) is None
        assert line_endpoints(1, 2.5, 1, 3, bad, 1, thr, H, W) is None
    # the -2^20 bound, after truncation toward zero
    assert line_endpoints(-1048576.9, 2, 1, 3, 4, 1, thr, H, W) == (2, -1048576, 4, 3)
    assert line_endpoints(-1048577.0, 2, 1, 3, 4, 1, thr, H, W) is None
    assert line_endpoints(3, 4, 1, 3, -1048577.5, 1, thr, H, W) is None
    # the far side clamps to the last row / column as the disc centre does
    assert line_endpoints(1e12, 5, 1, 3, 1e9, 1, thr, H, W) == (5, W - 1, H - 1, 3)
    f = np.zeros((1, H, W, 3), np.uint8)
    x = np.array([[-1048577.0, 10.0]])
    y = np.array([[5.0, 5.0]])
    out = draw_overlay_reference(f, x, y, np.ones((1, 2)), 0, thr, [(1, 1, 1), (2, 2, 2)], [(0, 1)], (9, 9, 9))
    assert not out.any()
    x[0, 0] = -1048576.0
    out = draw_overlay_reference(f, x, y, np.ones((1, 2)), 0, thr, [(1, 1, 1), (2, 2, 2)], [(0, 1)], (9, 9, 9))
    assert (out[0, 5, :11] == 9).all() and out[0].any(axis=2).sum() == 11


def test_painting_order():
    H, W, thr = 12, 16, 0.1
    cols = [(10, 0, 0), (20, 0, 0)]
    sk = (0, 99, 0)
    # frame 1: joint 0 at (4, 4), joint 1 at (4, 10); frame 0: joint 1 at (4, 5) (its trail disc sits under joint 0's disc
    # and on the line), joint 0 off the mask
    x = np.array([[0.0, 5.0], [4.0, 10.0]])
    y = np.array([[0.0, 4.0], [4.0, 4.0]])
    lik = np.array([[0.0, 1.0], [1.0, 1.0]])
    f = np.zeros((2, H, W, 3), np.uint8)
    out = draw_overlay_reference(f, x, y, lik, 2, thr, cols, [(0, 1)], sk, trailpoints=2)[1]
    assert tuple(out[4, 4]) == cols[0]       # the disc of frame t over the trail disc and the line
    assert tuple(out[4, 6]) == sk            # the line over the trail disc of frame t-1 (joint 1 at column 5, radius 2)
    assert tuple(out[3, 6]) == cols[1]       # the trail disc where neither the line nor a current disc reaches
    assert tuple(out[4, 10]) == cols[1] and tuple(out[4, 8]) == sk
    # frame 0 has no earlier frame: no trail; K = 0 / 1 and no edges give the markers alone
    first = draw_overlay_reference(f, x, y, lik, 2, thr, cols, [(0, 1)], sk, trailpoints=2)[0]
    assert first.any(axis=2).sum() == 9
    from test_render import draw_reference
    for K in (0, 1):
        assert np.array_equal(draw_overlay_reference(f, x, y, lik, 2, thr, cols, (), sk, K), draw_reference(f, x, y, lik, 2, thr, cols))
    # history rows: the same frames drawn from a table that starts K - 1 rows earlier
    rng = np.random.default_rng(2)
    N, nj, K = 6, 3, 4
    xs, ys = rng.uniform(-3, W + 3, (N, nj)), rng.uniform(-3, H + 3, (N, nj))
    lk = rng.uniform(0, 1, (N, nj))
    fr = rng.integers(0, 256, (N, H, W, 3), dtype=np.uint8)
    c3 = [(1, 2, 3), (4, 5, 6), (7, 8, 9)]
    whole = draw_overlay_reference(fr, xs, ys, lk, 2, 0.3, c3, [(0, 1), (1, 2)], sk, K)
    tail = draw_overlay_reference(fr[3:], xs, ys, lk, 2, 0.3, c3, [(0, 1), (1, 2)], sk, K, history=3)
    assert np.array_equal(whole[3:], tail)


def test_style_validation():
    from deepgraphpose_b200.engine import marker_style
    st, _ = marker_style(4)
    assert (st.n_edges, st.trailpoints, st.history, bytes(st.skeleton_color)) == (0, 0, 0, b"\0\0\0") and not st.edges
    st, keep = marker_style(4, edges=[(0, 1), (1, 3)], skeleton_color=(1, 2, 3), trailpoints=5, history=4)
    assert st.n_edges == 2 and list(st.skeleton_color) == [1, 2, 3] and (st.trailpoints, st.history) == (5, 4)
    assert keep[1].tolist() == [[0, 1], [1, 3]] and st.edges == keep[1].ctypes.data
    for kw in ({"edges": [(0, 4)]}, {"edges": [(-1, 0)]}, {"edges": [(0, 1, 2)]}, {"edges": [[0.0, 1.0]]},
               {"edges": [(0, 1)] * 257}, {"trailpoints": 65}, {"trailpoints": -1}, {"trailpoints": 2.0},
               {"trailpoints": 5, "history": 5}, {"history": 1}, {"trailpoints": 1, "history": 1},
               {"skeleton_color": (0, 0, 256)}, {"skeleton_color": (0, 0)}, {"skeleton_color": "black"}):
        with pytest.raises(ValueError):
            marker_style(4, **kw)


def test_entries_validate_before_any_work(tmp_path):
    from deepgraphpose_b200 import eval as E
    x = np.zeros((3, 4))
    clip = np.zeros((3, 8, 8, 3), np.uint8)
    for kw in ({"skeleton": [(0, 9)]}, {"trailpoints": 99}, {"skeleton_color": (300, 0, 0)}):
        with pytest.raises(ValueError):
            E.create_annotated_movie(clip, x, x, fps=30, filename=str(tmp_path / "m.mp4"), **kw)
    video = str(tmp_path / "missing.avi")
    cfg = {"num_joints": 4, "stride": 8.0, "all_joints_names": ["nose", "ear", "paw", "tail"]}
    for c, kw in ((cfg, {"draw_skeleton": True}),                                   # no skeleton in the config
                  (dict(cfg, skeleton=[["nose", "whisker"]]), {"draw_skeleton": True}),
                  (dict(cfg, skeleton=[[0, 7]]), {"draw_skeleton": True}),
                  (dict(cfg, skeleton=[["nose", "ear"]]), {"draw_skeleton": True, "trailpoints": 65}),
                  (cfg, {"trailpoints": -2})):
        with pytest.raises(ValueError):
            E.plot_dgp(video, output_dir=str(tmp_path), proj_cfg_file=c, dgp_model_file="synthetic", **kw)
    assert not os.listdir(tmp_path)


def test_skeleton_names_from_project_config(tmp_path):
    from deepgraphpose_b200 import eval as E
    yaml = pytest.importorskip("yaml")
    proj = tmp_path / "config.yaml"
    proj.write_text(yaml.safe_dump({"bodyparts": ["snout", "l_ear", "r_ear", "tail"],
                                    "skeleton": [["snout", "l_ear"], ["snout", "r_ear"], ["tail", "snout"]]}))
    cfg = E._load_dlc_cfg(str(proj))
    assert cfg["skeleton"] == [["snout", "l_ear"], ["snout", "r_ear"], ["tail", "snout"]]
    assert E.skeleton_from_cfg(cfg).tolist() == [[0, 1], [0, 2], [3, 0]]
    assert E.skeleton_from_cfg({"num_joints": 4, "skeleton": [(2, 3), (0, 1)]}).tolist() == [[2, 3], [0, 1]]
    bad = tmp_path / "bad.yaml"
    bad.write_text(yaml.safe_dump({"bodyparts": ["snout", "tail"], "skeleton": [["snout", "ear"]]}))
    with pytest.raises(ValueError, match="ear"):
        E.skeleton_from_cfg(E._load_dlc_cfg(str(bad)))
    none = tmp_path / "none.yaml"
    none.write_text(yaml.safe_dump({"bodyparts": ["snout", "tail"]}))
    with pytest.raises(ValueError):
        E.plot_dgp(str(tmp_path / "missing.avi"), output_dir=str(tmp_path / "out"), proj_cfg_file=str(none),
                   dgp_model_file="synthetic", draw_skeleton=True)
    assert not (tmp_path / "out").exists()
