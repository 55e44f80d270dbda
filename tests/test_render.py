"""plot_dgp's marker drawing without a GPU: the numpy restatement of the drawing contract (include/dgp_b200.h, DESIGN.md) that
the device kernel is compared against, the 'cool' colour table, disc shapes, argument validation and the ctypes mirror of
dgp_marker_style."""
import ctypes as C
import os

import numpy as np
import pytest


def draw_reference(frames, x, y, lik, dotsize, mask_threshold, colors):
    """The drawing contract in numpy: frames uint8 (N,H,W,3), x / y / lik float64 (N,nj) -> annotated copy.  Every disc is
    the whole-frame mask (r - yc)^2 + (c - xc)^2 < dotsize^2, independent of how the kernel bounds its loops."""
    out = np.array(frames, dtype=np.uint8, copy=True)
    N, H, W, _ = out.shape
    rr, cc = np.mgrid[0:H, 0:W].astype(np.float64)
    d2 = float(dotsize) * float(dotsize)
    for t in range(N):
        for j in range(x.shape[1]):
            xv, yv, lv = float(x[t, j]), float(y[t, j]), float(lik[t, j])
            if not lv > mask_threshold or np.isnan(xv) or np.isnan(yv):
                continue
            xc = min(np.trunc(xv), W - 1.0)   # truncation toward zero, as Python's int(); +inf clamps to the edge
            yc = min(np.trunc(yv), H - 1.0)
            m = (rr - yc) ** 2 + (cc - xc) ** 2 < d2
            out[t][m] = colors[j]
    return out


def disc(dotsize, size=21):
    f = np.zeros((1, size, size, 3), np.uint8)
    c = size // 2
    return draw_reference(f, np.array([[c + 0.4]]), np.array([[c]]), np.array([[1.0]]), dotsize, 0.1, [(255, 0, 0)])[0, :, :, 0] > 0


def test_cool_table():
    from deepgraphpose_b200.eval import marker_colors
    expect = {1: [0], 2: [0, 255], 4: [0, 85, 170, 255], 5: [0, 64, 128, 192, 255]}
    for nj, idx in expect.items():
        tab = marker_colors(nj)
        assert tab.dtype == np.uint8 and tab.shape == (nj, 3)
        assert tab.tolist() == [[i, 255 - i, 255] for i in idx], nj
    tab = marker_colors(20)
    idx = [min(255, (256 * j) // 19) for j in range(20)]
    assert tab[:, 0].tolist() == idx and idx[1] == 13 and idx[-1] == 255
    assert (tab[:, 1].astype(int) == 255 - tab[:, 0]).all() and (tab[:, 2] == 255).all()


def test_disc_shapes():
    c = 10
    assert disc(0).sum() == 0
    d1 = disc(1)
    assert d1.sum() == 1 and d1[c, c]
    d2 = disc(2)
    assert d2.sum() == 9 and d2[c - 1:c + 2, c - 1:c + 2].all()
    d3 = disc(3)
    assert d3.sum() == 25 and d3[c - 2:c + 3, c - 2:c + 3].all()
    d4 = disc(4)
    box = d4[c - 3:c + 4, c - 3:c + 4]
    assert d4.sum() == 45 and box.sum() == 45
    assert not box[0, 0] and not box[0, 6] and not box[6, 0] and not box[6, 6]


def test_centres_mask_and_order():
    f = np.full((1, 8, 10, 3), 7, np.uint8)
    cols = [(1, 2, 3), (4, 5, 6), (9, 9, 9)]
    # x = -0.7 truncates to 0 (drawn at column 0), -3.2 to -3 (a dotsize-3 disc then misses the frame), past the right edge
    # clamps to the last column; lik equal to the threshold is not drawn; NaN is never drawn
    out = draw_reference(f, np.array([[-0.7, -3.2, 55.0]]), np.array([[2.0, 2.0, 6.9]]), np.array([[0.5, 0.9, 0.9]]), 1, 0.4,
                         cols)[0]
    assert tuple(out[2, 0]) == (1, 2, 3) and tuple(out[6, 9]) == (9, 9, 9)
    assert (out != 7).any(axis=2).sum() == 2
    same = draw_reference(f, np.array([[3.0, np.nan, 3.0]]), np.array([[3.0, 3.0, 3.0]]), np.array([[0.4, 1.0, np.nan]]), 2,
                          0.4, cols)
    assert (same == f).all()
    # overlapping discs: the higher joint index wins
    ov = draw_reference(f, np.array([[4.0, 5.0, 0.0]]), np.array([[4.0, 4.0, 0.0]]), np.array([[1.0, 1.0, 0.0]]), 2, 0.4, cols)
    assert tuple(ov[0, 4, 4]) == (4, 5, 6) and tuple(ov[0, 4, 3]) == (1, 2, 3)


def test_arguments_are_validated_before_any_engine(tmp_path):
    from deepgraphpose_b200 import eval as E
    with pytest.raises(ValueError):
        E.marker_colors(4, "viridis")
    cfg = {"num_joints": 4, "stride": 8.0}
    video = str(tmp_path / "missing.avi")
    for kw in ({"colormap": "jet"}, {"dotsize": 65}, {"dotsize": -1}, {"dotsize": 2.5},
               {"colormap": np.zeros((3, 3), np.uint8)}, {"colormap": np.zeros((4, 4), np.uint8)}):
        with pytest.raises(ValueError):
            E.plot_dgp(video, output_dir=str(tmp_path), proj_cfg_file=cfg, dgp_model_file="synthetic", **kw)
    x = np.zeros((2, 4))
    with pytest.raises(ValueError):
        E.create_annotated_movie(np.zeros((2, 8, 8, 3), np.uint8), x, x, colormap="hot", fps=30)
    with pytest.raises(ValueError):
        E.create_annotated_movie(np.zeros((2, 8, 8, 3), np.uint8), x, x, dotsize=100, fps=30)
    with pytest.raises(ValueError):
        E.create_annotated_movie(np.zeros((2, 8, 8, 3), np.uint8), x, x, colormap=np.zeros((4, 2), np.uint8), fps=30)
    assert not os.listdir(tmp_path)


def test_marker_style_struct_matches_header(tmp_path):
    """sizeof / offsetof of dgp_marker_style (include/dgp_b200.h compiled with gcc) against the ctypes mirror."""
    import shutil
    import subprocess
    from deepgraphpose_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ct = L.DgpMarkerStyle
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dgp_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(dgp_marker_style));']
    for fname, _ in ct._fields_:
        lines.append('  printf("%s %%zu\\n", offsetof(dgp_marker_style, %s));' % (fname, fname))
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct)
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname
