"""Augmentation of fit_dgp's labelled frames (dgp_augment): the numpy restatements below of OpenCV's fixed-point bilinear
warpAffine / remap, the integer motion blur, the dropout mask's nearest upsample and the counter hash are checked against
cv2 (bit for bit, or within 1 LSB where stated), and the library's host-side blur table, the struct layout and
fitdgp_util.build_aug against them.  The device passes are checked against the same oracles in test_gpu_augment.py."""
import ctypes as C
import math
import os

import cv2
import numpy as np
import pytest

M64 = np.uint64


# ---------------------------------------------------------------------------------------------------- counter hash
def aug_hash(seed, plane, row, col):
    """splitmix64 of (seed, plane, row, col) (include/dgp_b200.h), element-wise over the row / col arrays."""
    with np.errstate(over="ignore"):
        row, col = np.broadcast_arrays(np.asarray(row, dtype=np.uint64), np.asarray(col, dtype=np.uint64))
        c = (M64(plane) << M64(48)) | (row << M64(24)) | col
        z = M64(int(seed) % 2 ** 64) + (c + M64(1)) * M64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> M64(30))) * M64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> M64(27))) * M64(0x94D049BB133111EB)
        return z ^ (z >> M64(31))


def noise(seed, plane, H, W):
    """(b + 0.5) / 2^23 - 1 of the top 24 bits, float32 (H, W)."""
    b = (aug_hash(seed, plane, np.arange(H)[:, None], np.arange(W)[None, :]) >> M64(40)).astype(np.int64)
    return (2 * b + 1 - (1 << 24)).astype(np.float32) * np.float32(2.0 ** -24)


def u01(seed, plane, H, W):
    b = (aug_hash(seed, plane, np.arange(H)[:, None], np.arange(W)[None, :]) >> M64(40)).astype(np.float64)
    return (b + 0.5) * 2.0 ** -24


def reflect101(p, n):
    """cv::borderInterpolate(BORDER_REFLECT_101) of an index array."""
    p = np.array(p, dtype=np.int64)
    if n == 1:
        return np.zeros_like(p)
    while True:
        bad = (p < 0) | (p >= n)
        if not bad.any():
            return p
        p = np.where(p < 0, -p, np.where(p >= n, 2 * n - 2 - p, p))


# ---------------------------------------------------------------------------------------------------- bilinear sampler
def bilinear_table():
    """OpenCV's INTER_LINEAR int16 weights (initInterTab2D): (1024, 4) for (fy * 32 + fx, dy * 2 + dx)."""
    T = np.zeros((1024, 4), np.int64)
    for i in range(32):
        for j in range(32):
            fy, fx = np.float32(i) * np.float32(1 / 32), np.float32(j) * np.float32(1 / 32)
            vy, vx = [np.float32(1) - fy, fy], [np.float32(1) - fx, fx]
            it = [int(np.rint(np.float32(vy[a] * vx[b]) * np.float32(32768))) for a in range(2) for b in range(2)]
            d = sum(it) - 32768
            if d:
                mk = Mk = 0
                for k in range(4):
                    if it[k] < it[mk]:
                        mk = k
                    elif it[k] > it[Mk]:
                        Mk = k
                if d < 0:
                    it[Mk] -= d
                else:
                    it[mk] -= d
            T[i * 32 + j] = it
    return T


TAB = bilinear_table()


def _sample(img, X, Y):
    """Fixed-point bilinear sample at X, Y (5 fraction bits) with 0 outside the frame."""
    H, W = img.shape[:2]
    sx, sy = np.clip(X >> 5, -32768, 32767), np.clip(Y >> 5, -32768, 32767)
    w = TAB[(Y & 31) * 32 + (X & 31)]
    acc = np.full(X.shape + (3,), 1 << 14, np.int64)
    for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        py, px = sy + dy, sx + dx
        ok = (py >= 0) & (py < H) & (px >= 0) & (px < W)
        v = img[np.clip(py, 0, H - 1), np.clip(px, 0, W - 1)].astype(np.int64) * ok[..., None]
        acc += w[..., k:k + 1] * v
    return np.clip(acc >> 15, 0, 255).astype(np.uint8)


def rotation_matrix(deg, H, W):
    t = deg * (math.pi / 180.0)
    c, s = math.cos(t), math.sin(t)
    cx, cy = W / 2 - 0.5, H / 2 - 0.5
    return np.array([[c, -s, cx - c * cx + s * cy], [s, c, cy - s * cx - c * cy]])


def invert_affine(M):
    """cv::warpAffine's inversion of the forward matrix."""
    m = [float(v) for v in np.asarray(M, dtype=np.float64).ravel()]
    D = m[0] * m[4] - m[1] * m[3]
    D = 1.0 / D if D != 0 else 0.0
    A11, A22 = m[4] * D, m[0] * D
    m[0] = A11
    m[1] *= -D
    m[3] *= -D
    m[4] = A22
    b1 = -m[0] * m[2] - m[1] * m[5]
    b2 = -m[3] * m[2] - m[4] * m[5]
    m[2], m[5] = b1, b2
    return m


def warp_affine(img, M):
    """cv2.warpAffine(img, M, (W, H), INTER_LINEAR, BORDER_CONSTANT, 0) through OpenCV's fixed-point path."""
    H, W = img.shape[:2]
    m = invert_affine(M)
    y = np.arange(H, dtype=np.float64)
    x = np.arange(W, dtype=np.float64)
    X0 = np.rint((m[1] * y + m[2]) * 1024).astype(np.int64) + 16
    Y0 = np.rint((m[4] * y + m[5]) * 1024).astype(np.int64) + 16
    adx = np.rint(m[0] * x * 1024).astype(np.int64)
    ady = np.rint(m[3] * x * 1024).astype(np.int64)
    X = (X0[:, None] + adx[None, :]) >> 5
    Y = (Y0[:, None] + ady[None, :]) >> 5
    return _sample(img, X, Y)


def remap(img, mx, my):
    """cv2.remap(img, mx, my, INTER_LINEAR, BORDER_CONSTANT, 0) with float32 maps through OpenCV's fixed-point path."""
    X = np.rint(mx.astype(np.float32) * np.float32(32)).astype(np.int64)
    Y = np.rint(my.astype(np.float32) * np.float32(32)).astype(np.int64)
    return _sample(img, X, Y)


def elastic_maps(dx, dy):
    H, W = dx.shape
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    return (xx + dx.astype(np.float32)).astype(np.float32), (yy + dy.astype(np.float32)).astype(np.float32)


# ---------------------------------------------------------------------------------------------------- motion blur
def motion_blur_table(k, angle_deg, direction):
    """The int32 k x k table of dgp_motion_blur_kernel (include/dgp_b200.h), in the library's double operations."""
    d = (direction + 1.0) / 2.0
    img = np.zeros((k, k))
    img[:, k // 2] = np.linspace(d, 1.0 - d, k)
    t = angle_deg * (math.pi / 180.0)
    ca, sa, c = math.cos(t), math.sin(t), (k - 1) / 2.0

    def at(yy, xx):
        return float(img[yy, xx]) if 0 <= yy < k and 0 <= xx < k else 0.0

    rot = np.zeros((k, k))
    total = 0.0
    for i in range(k):
        for j in range(k):
            u, v = j - c, i - c
            sx, sy = ca * u + sa * v + c, -sa * u + ca * v + c
            fx0, fy0 = math.floor(sx), math.floor(sy)
            x0, y0 = int(fx0), int(fy0)
            fx, fy = sx - fx0, sy - fy0
            val = (1.0 - fy) * ((1.0 - fx) * at(y0, x0) + fx * at(y0, x0 + 1)) + \
                fy * ((1.0 - fx) * at(y0 + 1, x0) + fx * at(y0 + 1, x0 + 1))
            rot[i, j] = val
            total += val
    w = np.rint(rot / total * 16384.0).astype(np.int64).ravel()
    w[np.argmax(w)] += 16384 - w.sum()
    return w.reshape(k, k)


def blur_int(img, w):
    """(sum w p + 2^13) >> 14 per channel, correlation with a reflect-101 border, saturated."""
    H, W = img.shape[:2]
    k = w.shape[0]
    r = k // 2
    iy = reflect101(np.arange(-r, H + r), H)
    ix = reflect101(np.arange(-r, W + r), W)
    pad = img[iy][:, ix].astype(np.int64)
    acc = np.full(img.shape, 1 << 13, np.int64)
    for i in range(k):
        for j in range(k):
            acc += int(w[i, j]) * pad[i:i + H, j:j + W]
    return np.clip(acc >> 14, 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------------- dropout
def dropout_grid(H, W, sp):
    return max(1, int(np.rint(H * sp))), max(1, int(np.rint(W * sp)))


def nearest_index(n_out, n_in):
    """cv2.resize(INTER_NEAREST)'s source index of each output index: floor(i * (1 / (n_out / n_in))), in double."""
    return np.minimum(np.floor(np.arange(n_out, dtype=np.float64) * (1.0 / (n_out / n_in))).astype(np.int64), n_in - 1)


def dropout_mask(H, W, p, sp, seed):
    """(H, W) bool: True where the pixel is dropped."""
    gh, gw = dropout_grid(H, W, sp)
    cells = u01(seed, 2, gh, gw) < p
    return cells[nearest_index(H, gh)][:, nearest_index(W, gw)]


# ---------------------------------------------------------------------------------------------------- elastic field
def elastic_field64(H, W, alpha, sigma, seed):
    """The elastic fields (dx, dy) in float64: hash noise, separable Gaussian (reflect-101), times alpha."""
    R = int(math.ceil(4.0 * sigma))
    k = np.arange(-R, R + 1)
    g = np.exp(-(k * k).astype(np.float64) / (2.0 * sigma * sigma))
    g /= g.sum()
    out = []
    for plane in (0, 1):
        n = noise(seed, plane, H, W).astype(np.float64)
        ix = reflect101(np.arange(W)[:, None] + k[None, :], W)
        t = (n[:, ix] * g).sum(-1)
        iy = reflect101(np.arange(H)[:, None] + k[None, :], H)
        out.append(alpha * np.einsum("ykx,k->yx", t[iy], g))
    return out


def elastic_labels(q, dx, dy, iters=20):
    """The inverse of the backward map at pixel points q (m, 2) = (x, y): p <- q - d(p) from p = q, d bilinear in the
    float32 fields with coordinates clamped to the frame."""
    H, W = dx.shape
    dx, dy = dx.astype(np.float64), dy.astype(np.float64)

    def bil(f, px, py):
        cx, cy = np.clip(px, 0, W - 1), np.clip(py, 0, H - 1)
        x0 = np.minimum(np.floor(cx).astype(np.int64), max(W - 2, 0))
        y0 = np.minimum(np.floor(cy).astype(np.int64), max(H - 2, 0))
        x1, y1 = np.minimum(x0 + 1, W - 1), np.minimum(y0 + 1, H - 1)
        fx, fy = cx - x0, cy - y0
        return (1 - fy) * ((1 - fx) * f[y0, x0] + fx * f[y0, x1]) + fy * ((1 - fx) * f[y1, x0] + fx * f[y1, x1])

    px, py = q[:, 0].copy(), q[:, 1].copy()
    for _ in range(iters):
        px, py = q[:, 0] - bil(dx, px, py), q[:, 1] - bil(dy, px, py)
    return np.stack([px, py], 1)


def frame(H, W, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


# ================================================================================================================ tests
SIZES = [(1, 1), (3, 5), (5, 3), (61, 83), (747, 832)]
ANGLES = [-25.0, -17.3, -3.1, 0.7, 12.5, 25.0, 47.0, 90.0, -135.5, 180.0]


@pytest.mark.parametrize("H,W", SIZES)
def test_warp_affine_restatement_equals_cv2(H, W):
    img = frame(H, W, H * 7 + W)
    for deg in ANGLES if H * W < 1000 or H < 100 else ANGLES[::3]:
        M = rotation_matrix(deg, H, W)
        ref = cv2.warpAffine(img, M, (W, H), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        assert np.array_equal(warp_affine(img, M), ref.reshape(img.shape)), deg


@pytest.mark.parametrize("H,W,amp", [(1, 1, 3.0), (3, 5, 4.0), (61, 83, 2.5), (61, 83, 200.0), (120, 97, 25.0),
                                     (747, 832, 8.0)])
def test_remap_restatement_equals_cv2(H, W, amp):
    """Maps up to `amp` pixels off the identity; 200 reaches far outside the frame."""
    rng = np.random.default_rng(int(amp * 10) + H)
    img = frame(H, W, H + W)
    dx = rng.uniform(-amp, amp, (H, W)).astype(np.float32)
    dy = rng.uniform(-amp, amp, (H, W)).astype(np.float32)
    mx, my = elastic_maps(dx, dy)
    ref = cv2.remap(img, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    assert np.array_equal(remap(img, mx, my), ref.reshape(img.shape))


@pytest.mark.parametrize("k,angle,direction", [(7, 0.0, 0.0), (7, 33.3, -0.4), (7, -90.0, 1.0), (3, 45.0, -1.0),
                                               (5, 71.2, 0.25), (15, -12.0, 0.9)])
def test_integer_motion_blur_within_one_lsb_of_filter2d(k, angle, direction):
    w = motion_blur_table(k, angle, direction)
    assert w.sum() == 16384 and (w >= 0).all()
    for H, W in ((61, 83), (4, 3), (1, 1), (747, 832)):
        img = frame(H, W, k + H)
        ref = cv2.filter2D(img, -1, w.astype(np.float32) / 16384.0, borderType=cv2.BORDER_REFLECT_101)
        got = blur_int(img, w)
        assert np.abs(got.astype(int) - ref.reshape(img.shape).astype(int)).max() <= 1


def test_library_motion_blur_table_equals_restatement(lib_built):
    from deepgraphpose_b200 import _lib as L
    lib = L.load()
    rng = np.random.default_rng(5)
    for k in (3, 5, 7, 9, 15):
        for _ in range(12):
            angle, direction = rng.uniform(-180, 180), rng.uniform(-1, 1)
            w = np.zeros((k, k), np.int32)
            assert lib.dgp_motion_blur_kernel(k, angle, direction, w.ctypes.data) == 0
            assert np.array_equal(w, motion_blur_table(k, angle, direction)), (k, angle, direction)
            assert int(w.sum()) == 16384
    w = np.zeros(400, np.int32)
    for k, d in ((4, 0.0), (1, 0.0), (17, 0.0), (7, 1.5), (7, float("nan"))):
        assert lib.dgp_motion_blur_kernel(k, 10.0, d, w.ctypes.data) == -1


def test_nearest_upsample_equals_cv2_resize():
    rng = np.random.default_rng(2)
    for H, W in ((1, 1), (3, 5), (61, 83), (747, 832), (1000, 1001)):
        for sp in (0.01, 0.013, 0.02, 0.037, 0.05, 0.5):
            gh, gw = dropout_grid(H, W, sp)
            m = rng.integers(0, 256, (gh, gw), dtype=np.uint8)
            ref = cv2.resize(m, (W, H), interpolation=cv2.INTER_NEAREST)
            assert np.array_equal(m[nearest_index(H, gh)][:, nearest_index(W, gw)], ref.reshape(H, W)), (H, W, sp)


def test_hash_restatement_is_deterministic_and_uniform():
    a = noise(123, 0, 64, 80)
    assert np.array_equal(a, noise(123, 0, 64, 80))
    assert not np.array_equal(a, noise(124, 0, 64, 80)) and not np.array_equal(a, noise(123, 1, 64, 80))
    assert a.dtype == np.float32 and a.min() >= -1 and a.max() < 1 and abs(float(a.mean())) < 0.02
    z = aug_hash(0, 0, np.array([0]), np.array([0]))
    assert int(z[0]) == int(aug_hash(0, 0, np.array([0]), np.array([0]))[0])
    u = u01(9, 2, 100, 100)
    assert u.min() > 0 and u.max() < 1 and abs(float(u.mean()) - 0.5) < 0.02


def test_build_aug_ranges_switches_and_seeds():
    from deepgraphpose_b200.fitdgp_util import build_aug
    draws = build_aug(seed=7).sample(2000)
    assert draws == build_aug(seed=7).sample(2000)
    assert draws != build_aug(seed=8).sample(2000)
    rot = np.array([d["rotate_deg"] for d in draws])
    assert (np.abs(rot) <= 25).all() and 0.4 < (rot != 0).mean() < 0.6
    on = [d for d in draws if d["blur_k"]]
    assert all(d["blur_k"] == 7 for d in on) and 0.4 < len(on) / len(draws) < 0.6
    assert all(-90 <= d["blur_angle_deg"] <= 90 and -1 <= d["blur_direction"] <= 1 for d in draws)
    drop = [d for d in draws if d["drop_size_percent"]]
    assert all(0 <= d["drop_p"] <= 0.02 and 0.01 <= d["drop_size_percent"] <= 0.05 for d in drop)
    assert 0.4 < len(drop) / len(draws) < 0.6
    alpha = np.array([d["elastic_alpha"] for d in draws])
    assert (alpha >= 0).all() and (alpha <= 40).all() and 0.4 < (alpha != 0).mean() < 0.6
    assert all(d["elastic_sigma"] == 5 and 0 <= d["seed"] < 2 ** 63 for d in draws)
    off = build_aug(apply_prob=0, seed=1).sample(300)
    assert all(d["rotate_deg"] == 0 and d["blur_k"] == 0 and d["drop_p"] == 0 and d["drop_size_percent"] == 0
               and d["elastic_alpha"] == 0 for d in off)
    every = build_aug(apply_prob=1, seed=1).sample(300)
    assert all(d["blur_k"] == 7 and d["drop_size_percent"] > 0 for d in every)
    with pytest.raises(ValueError):
        build_aug(motion_blur_k=4)


def test_augment_params_struct_matches_header(tmp_path):
    """sizeof / offsetof of dgp_augment_params (include/dgp_b200.h compiled with gcc) against the ctypes mirror."""
    import shutil
    import subprocess
    from deepgraphpose_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ct = L.DgpAugmentParams
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dgp_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(dgp_augment_params));']
    for fname, _ in ct._fields_:
        lines.append('  printf("%s %%zu\\n", offsetof(dgp_augment_params, %s));' % (fname, fname))
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct)
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname
