"""estimate_pose's frame resize + crop (dgp_resize_crop): the numpy restatement of Pillow's 8-bit BICUBIC resample below
equals PIL bit for bit, and the library's host-side table (dgp_resize_coefficients), dims and struct layout follow it.
The device passes are checked against PIL in test_gpu_resize.py."""
import ctypes as C
import os

import numpy as np
import pytest
from PIL import Image

PRECISION_BITS = 22

# (H0, W0, new_size (h, w) or None, crop box (x0, y0, x1, y1) or None)
GRID = [
    (40, 100, (40, 50), None),            # downscale 2, width only
    (60, 30, (40, 30), None),             # downscale 1.5, height only
    (37, 74, (10, 74), None),             # downscale 3.7, height only
    (32, 160, (32, 10), None),            # downscale 16, width only
    (5, 400, (5, 2), None),               # downscale 200, width only
    (400, 6, (2, 6), None),               # downscale 200, height only
    (30, 40, (39, 52), None),             # upscale 1.3
    (7, 9, (28, 36), None),               # upscale 4
    (47, 61, (23, 30), None),             # both axes down
    (33, 35, (33, 20), None),             # one axis unchanged
    (20, 30, (20, 30), None),             # identity
    (1, 17, (3, 5), None),                # 1-pixel source
    (13, 1, (1, 1), None),                # 1-pixel source and output
    (5, 7, (1, 1), None),
    (2, 2, (600, 9), None),
    (300, 1000, (7, 5), None),
    (48, 64, (30, 41), (3, 4, 25, 20)),   # crop inside the resized frame
    (48, 64, (30, 41), (-5, -3, 36, 22)), # crop partly outside (left / top)
    (48, 64, (30, 41), (20, 10, 50, 40)), # crop partly outside (right / bottom)
    (48, 64, (30, 41), (-9, -7, 50, 40)), # crop around the whole frame
    (48, 64, (30, 41), (45, 2, 60, 9)),   # crop fully outside
    (48, 64, None, (5, 7, 38, 30)),       # crop without resize
    (48, 64, None, (-4, 40, 70, 55)),     # crop without resize, partly outside
    (31, 45, (31, 17), (2, 3, 13, 29)),   # width-only resize + crop
    (31, 45, (52, 45), (-1, 9, 44, 40)),  # height-only resize + crop
]


def bicubic(x):
    a = -0.5
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def taps(in_size, out_size):
    return int(np.ceil(2.0 * max(in_size / out_size, 1.0))) * 2 + 1


def coefficients(in_size, out_size):
    """Pillow's precompute_coeffs + normalize_coeffs_8bpc: (first, count, int weights (out, taps))."""
    scale = in_size / out_size
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ss = 1.0 / fs
    ksize = taps(in_size, out_size)
    first = np.zeros(out_size, np.int64)
    count = np.zeros(out_size, np.int64)
    K = np.zeros((out_size, ksize), np.int64)
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), in_size) - xmin
        w = [bicubic((x + xmin - center + 0.5) * ss) for x in range(n)]
        ww = 0.0
        for v in w:
            ww += v
        w = [v / ww if ww != 0 else v for v in w]
        for x, v in enumerate(w):
            K[xx, x] = int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
        first[xx], count[xx] = xmin, n
    return first, count, K


def resample_axis(a, out_size, axis):
    first, count, K = coefficients(a.shape[axis], out_size)
    a = np.moveaxis(a, axis, 0).astype(np.int64)
    out = np.empty((out_size,) + a.shape[1:], np.int64)
    for xx in range(out_size):
        s = np.full(a.shape[1:], 1 << (PRECISION_BITS - 1), np.int64)
        for x in range(count[xx]):
            s += a[first[xx] + x] * K[xx, x]
        out[xx] = np.clip(s >> PRECISION_BITS, 0, 255)
    return np.moveaxis(out, 0, axis).astype(np.uint8)


def restated(img, new_size, crop):
    """Image.resize((w, h)) (horizontal pass first, a pass skipped when its size is unchanged) then Image.crop(box)."""
    out = img
    if new_size is not None:
        if new_size[1] != out.shape[1]:
            out = resample_axis(out, new_size[1], 1)
        if new_size[0] != out.shape[0]:
            out = resample_axis(out, new_size[0], 0)
    if crop is not None:
        x0, y0, x1, y1 = crop
        box = np.zeros((y1 - y0, x1 - x0, 3), np.uint8)
        h, w = out.shape[:2]
        sx0, sy0, sx1, sy1 = max(x0, 0), max(y0, 0), min(x1, w), min(y1, h)
        if sx1 > sx0 and sy1 > sy0:
            box[sy0 - y0:sy1 - y0, sx0 - x0:sx1 - x0] = out[sy0:sy1, sx0:sx1]
        out = box
    return out


def pil(img, new_size, crop):
    """What the reference's estimate_pose does to a frame (eval.py:316-322)."""
    im = Image.fromarray(img)
    if new_size is not None:
        im = im.resize(size=(new_size[1], new_size[0]))
    if crop is not None:
        im = im.crop(crop)
    return np.asarray(im)


def frame(H0, W0, seed):
    return np.random.default_rng(seed).integers(0, 256, (H0, W0, 3), dtype=np.uint8)


@pytest.mark.parametrize("case", range(len(GRID)))
def test_restatement_equals_pillow(case):
    H0, W0, new_size, crop = GRID[case]
    img = frame(H0, W0, case)
    assert np.array_equal(restated(img, new_size, crop), pil(img, new_size, crop))


def test_pillow_default_rgb_filter_is_bicubic():
    img = Image.fromarray(frame(37, 53, 1))
    for size in ((20, 11), (90, 70)):
        assert np.array_equal(np.asarray(img.resize(size)), np.asarray(img.resize(size, Image.BICUBIC)))


def _lib():
    from deepgraphpose_b200 import _lib as L
    return L, L.load()


@pytest.mark.parametrize("case", range(len(GRID)))
def test_library_coefficients_equal_restatement(lib_built, case):
    H0, W0, new_size, _ = GRID[case]
    if new_size is None:
        pytest.skip("no resize")
    _, lib = _lib()
    for n_in, n_out in ((W0, new_size[1]), (H0, new_size[0])):
        first, count, K = coefficients(n_in, n_out)
        for max_taps in (K.shape[1], K.shape[1] + 3):
            f = np.zeros(n_out, np.int32)
            c = np.zeros(n_out, np.int32)
            w = np.full((n_out, max_taps), -7, np.int32)
            assert lib.dgp_resize_coefficients(n_in, n_out, max_taps, f.ctypes.data, c.ctypes.data, w.ctypes.data) == 0
            assert np.array_equal(f, first) and np.array_equal(c, count)
            assert np.array_equal(w[:, :K.shape[1]], K) and (w[:, K.shape[1]:] == 0).all()
        if count.max() > 1:  # a table narrower than the widest window is refused
            f, c = np.zeros(n_out, np.int32), np.zeros(n_out, np.int32)
            w = np.zeros((n_out, count.max() - 1), np.int32)
            assert lib.dgp_resize_coefficients(n_in, n_out, int(count.max()) - 1, f.ctypes.data, c.ctypes.data,
                                               w.ctypes.data) == -1


def test_transform_dims_closed_form(lib_built):
    from deepgraphpose_b200.engine import transform_dims
    L, lib = _lib()
    for H0, W0, new_size, crop in GRID:
        h, w = new_size if new_size is not None else (H0, W0)
        if crop is not None:
            h, w = crop[3] - crop[1], crop[2] - crop[0]
        assert transform_dims(H0, W0, new_size, crop) == (h, w)
        assert transform_dims(H0, W0, new_size, crop) == pil(frame(H0, W0, 0), new_size, crop).shape[:2]
    H, W = C.c_int(), C.c_int()
    assert lib.dgp_transform_dims(1494, 1664, None, C.byref(H), C.byref(W)) == 0 and (H.value, W.value) == (1494, 1664)
    t = L.DgpFrameTransform(747, 832, 0, 0, 0, 0)
    assert lib.dgp_transform_dims(1494, 1664, C.byref(t), C.byref(H), C.byref(W)) == 0 and (H.value, W.value) == (747, 832)
    bad = [(0, 10, 0, 0, 0, 0), (10, -1, 0, 0, 0, 0), (-3, -3, 0, 0, 0, 0), (0, 0, 5, 5, 5, 9), (0, 0, 5, 9, 8, 9),
           (0, 0, 3, 0, 0, 0), (0, 0, 0, 0, 0, 4), (10, 10, 9, 2, 1, 5)]
    for fields in bad:
        t = L.DgpFrameTransform(*fields)
        assert lib.dgp_transform_dims(100, 120, C.byref(t), C.byref(H), C.byref(W)) == -1, fields
    assert lib.dgp_transform_dims(0, 120, None, C.byref(H), C.byref(W)) == -1
    for new_size, crop in (((0, 5), None), (None, (4, 4, 4, 9)), (None, (4, 9, 8, 2))):
        with pytest.raises(ValueError):
            transform_dims(100, 120, new_size, crop)


def test_frame_transform_struct_matches_header(tmp_path):
    """sizeof / offsetof of dgp_frame_transform (include/dgp_b200.h compiled with gcc) against the ctypes mirror."""
    import shutil
    import subprocess
    from deepgraphpose_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ct = L.DgpFrameTransform
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dgp_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(dgp_frame_transform));']
    for fname, _ in ct._fields_:
        lines.append('  printf("%s %%zu\\n", offsetof(dgp_frame_transform, %s));' % (fname, fname))
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct)
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname
