"""Augmentation of labelled training frames on the device (dgp_augment, Engine.augment, fitdgp_util.data_aug and fit_dgp's
aug_pipeline): every op alone and the whole pipeline equal the sequential cv2 / numpy oracle of test_augment.py bit for bit
(cv2.remap fed the device's own elastic fields), labels move with the pixels, untouched frames stay untouched, and the
training loops are reproducible with a seeded pipeline and unchanged without one."""
import ctypes as C

import cv2
import numpy as np
import pytest
import torch

from test_augment import (blur_int, dropout_mask, elastic_field64, elastic_labels, elastic_maps, frame, motion_blur_table,
                          rotation_matrix)

pytestmark = pytest.mark.gpu
NJ = 4
STRIDE = 8.0


@pytest.fixture(scope="module")
def eng():
    from deepgraphpose_b200.engine import Engine
    e = Engine(NJ, location_refinement=False, stride=STRIDE)
    yield e
    e.close()


def P(**kw):
    base = dict(rotate_deg=0.0, blur_k=0, blur_angle_deg=0.0, blur_direction=0.0, drop_p=0.0, drop_size_percent=0.0,
                elastic_alpha=0.0, elastic_sigma=5.0, seed=0)
    base.update(kw)
    return base


def oracle(eng, img, p):
    """The pipeline frame by frame with cv2 and the numpy restatements."""
    H, W = img.shape[:2]
    out = img
    if p["rotate_deg"] != 0:
        out = cv2.warpAffine(out, rotation_matrix(p["rotate_deg"], H, W), (W, H), flags=cv2.INTER_LINEAR,
                             borderMode=cv2.BORDER_CONSTANT, borderValue=0).reshape(H, W, 3)
    if p["blur_k"]:
        out = blur_int(out, motion_blur_table(p["blur_k"], p["blur_angle_deg"], p["blur_direction"]))
    if p["drop_p"] > 0 and p["drop_size_percent"] > 0:
        out = out * ~dropout_mask(H, W, p["drop_p"], p["drop_size_percent"], p["seed"])[..., None]
    if p["elastic_alpha"] != 0:
        dx, dy = eng.elastic_field(H, W, p["elastic_alpha"], p["elastic_sigma"], p["seed"])
        mx, my = elastic_maps(dx.cpu().numpy(), dy.cpu().numpy())
        out = cv2.remap(np.ascontiguousarray(out), mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT,
                        borderValue=0).reshape(H, W, 3)
    return out.astype(np.uint8)


def run(eng, frames, positions, params, joint_loc=None):
    dev = torch.from_numpy(frames).cuda()
    jl = eng.augment(dev, positions, joint_loc, params)
    torch.cuda.synchronize()
    return dev.cpu().numpy(), (jl.cpu().numpy() if jl is not None else None)


def assert_same(got, ref):
    bad = np.argwhere(got != ref)
    assert bad.size == 0, "%d bytes differ, first at %s" % (len(bad), bad[:3].tolist())


OPS = {
    "rotate": [P(rotate_deg=17.3), P(rotate_deg=-25.0), P(rotate_deg=133.0)],
    "blur": [P(blur_k=7, blur_angle_deg=-61.0, blur_direction=0.3), P(blur_k=3, blur_angle_deg=12.0, blur_direction=-1.0),
             P(blur_k=15, blur_angle_deg=90.0, blur_direction=0.9)],
    "dropout": [P(drop_p=0.02, drop_size_percent=0.05, seed=3), P(drop_p=0.5, drop_size_percent=0.013, seed=4),
                P(drop_p=1.0, drop_size_percent=0.3, seed=5)],
    "elastic": [P(elastic_alpha=40.0, seed=11), P(elastic_alpha=7.5, elastic_sigma=2.0, seed=12),
                P(elastic_alpha=-300.0, elastic_sigma=3.0, seed=13)],
    "blur+dropout": [P(blur_k=7, blur_angle_deg=45.0, blur_direction=-0.2, drop_p=0.3, drop_size_percent=0.04, seed=8)],
    "all": [P(rotate_deg=-21.0, blur_k=7, blur_angle_deg=80.0, blur_direction=0.5, drop_p=0.2, drop_size_percent=0.03,
              elastic_alpha=33.0, seed=21),
            P(rotate_deg=9.0, elastic_alpha=12.0, elastic_sigma=4.0, seed=22),
            P(rotate_deg=3.0, blur_k=5, blur_angle_deg=-10.0, blur_direction=0.0, seed=23)],
}
SIZES = [(747, 832), (61, 83), (37, 53), (3, 5), (1, 1)]


@pytest.mark.parametrize("H,W", SIZES)
@pytest.mark.parametrize("op", sorted(OPS))
def test_each_op_and_pipeline_equal_the_oracle(eng, op, H, W):
    params = OPS[op]
    nt = len(params) + 2
    frames = np.stack([frame(H, W, 10 * H + i) for i in range(nt)])
    positions = list(range(nt - 1, 0, -1))[:len(params)]       # frame 0 is not listed
    got, _ = run(eng, frames, positions, params)
    assert_same(got[0], frames[0])
    for pos, p in zip(positions, params):
        assert_same(got[pos], oracle(eng, frames[pos], p))


def test_many_frames_per_call_equal_one_frame_per_call(eng):
    """More frames than one launch carries; a frame's result does not depend on the other frames of the call."""
    from deepgraphpose_b200.fitdgp_util import build_aug
    H, W = 45, 67
    frames = np.stack([frame(H, W, 300 + i) for i in range(40)])
    params = build_aug(apply_prob=0.7, seed=5).sample(37)
    positions = list(range(3, 40))
    whole, _ = run(eng, frames, positions, params)
    for pos, p in zip(positions, params):
        one, _ = run(eng, frames[pos:pos + 1].copy(), [0], [p])
        assert_same(whole[pos], one[0])
        assert_same(whole[pos], oracle(eng, frames[pos], p))
    assert_same(whole[:3], frames[:3])


@pytest.mark.parametrize("H,W", [(747, 832), (61, 83), (1, 1)])
def test_elastic_field_matches_float64(eng, H, W):
    for alpha, sigma, seed in ((40.0, 5.0, 1), (17.0, 2.5, 2), (3.0, 16.0, 3)):
        dx, dy = eng.elastic_field(H, W, alpha, sigma, seed)
        rx, ry = elastic_field64(H, W, alpha, sigma, seed)
        assert np.abs(dx.cpu().numpy() - rx).max() <= 1e-5 and np.abs(dy.cpu().numpy() - ry).max() <= 1e-5


def _labels(n, seed, H, W):
    rng = np.random.default_rng(seed)
    jl = np.stack([rng.uniform(-1, H / STRIDE, (n, NJ)), rng.uniform(-1, W / STRIDE, (n, NJ))], axis=2)
    jl[0, 1] = np.nan
    jl[-1, 2, 0] = np.nan
    return jl


def _to_px(jl):
    return np.stack([jl[..., 1] * STRIDE + STRIDE / 2, jl[..., 0] * STRIDE + STRIDE / 2], -1)   # (x, y)


def _from_px(p):
    return np.stack([(p[..., 1] - STRIDE / 2) / STRIDE, (p[..., 0] - STRIDE / 2) / STRIDE], -1)


def test_labels_follow_rotation_and_elastic(eng):
    H, W = 120, 160
    params = [P(rotate_deg=23.0), P(elastic_alpha=35.0, seed=4), P(rotate_deg=-14.0, elastic_alpha=25.0, seed=5),
              P(blur_k=7, blur_angle_deg=30.0, drop_p=0.5, drop_size_percent=0.05, seed=6)]
    jl = _labels(len(params), 0, H, W)
    frames = np.stack([frame(H, W, i) for i in range(len(params))])
    _, got = run(eng, frames, list(range(len(params))), params, torch.from_numpy(jl.copy()).cuda())
    assert np.array_equal(np.isnan(got), np.isnan(jl))
    for k, p in enumerate(params):
        q = _to_px(jl[k])
        if p["rotate_deg"]:
            M = rotation_matrix(p["rotate_deg"], H, W)
            q = q @ M[:, :2].T + M[:, 2]
        if p["elastic_alpha"]:
            dx, dy = eng.elastic_field(H, W, p["elastic_alpha"], p["elastic_sigma"], p["seed"])
            ok = ~np.isnan(q).any(1)
            q[ok] = elastic_labels(q[ok], dx.cpu().numpy(), dy.cpu().numpy())
        ref = _from_px(q)
        tol = 1e-6 if p["elastic_alpha"] else 1e-9 / STRIDE
        ok = ~np.isnan(ref)
        assert np.abs(got[k][ok] - ref[ok]).max() <= tol, k
    assert np.array_equal(got[3], jl[3], equal_nan=True)       # blur and dropout leave labels alone


def test_blob_peaks_follow_their_labels(eng):
    """Isolated Gaussian blobs drawn at the labels: after rotation + elastic the brightest pixel near each moved label lies
    within 1 px of it."""
    H, W = 240, 320
    rng = np.random.default_rng(3)
    jl = np.zeros((3, NJ, 2))
    frames = np.zeros((3, H, W, 3), np.uint8)
    yy, xx = np.mgrid[0:H, 0:W]
    for k in range(3):
        for j in range(NJ):
            jl[k, j] = ((40 + 50 * j + rng.uniform(-5, 5)) / STRIDE, (70 + 60 * j + rng.uniform(-5, 5)) / STRIDE)
            x, y = jl[k, j, 1] * STRIDE + STRIDE / 2, jl[k, j, 0] * STRIDE + STRIDE / 2
            blob = 250 * np.exp(-((xx - x) ** 2 + (yy - y) ** 2) / (2 * 2.5 ** 2))
            frames[k] = np.maximum(frames[k], blob[..., None].astype(np.uint8))
    params = [P(rotate_deg=19.0), P(elastic_alpha=40.0, seed=9), P(rotate_deg=-24.0, elastic_alpha=40.0, seed=10)]
    got, moved = run(eng, frames, [0, 1, 2], params, torch.from_numpy(jl.copy()).cuda())
    for k in range(3):
        lum = got[k].astype(np.int64).sum(-1)
        for j in range(NJ):
            x, y = moved[k, j, 1] * STRIDE + STRIDE / 2, moved[k, j, 0] * STRIDE + STRIDE / 2
            x0, y0 = int(round(x)), int(round(y))
            win = lum[y0 - 8:y0 + 9, x0 - 8:x0 + 9]
            py, px = np.unravel_index(np.argmax(win), win.shape)
            assert np.hypot(px + x0 - 8 - x, py + y0 - 8 - y) <= 1.0, (k, j)


def test_all_ops_off_leaves_frames_and_launches_alone(eng):
    frames = np.stack([frame(61, 83, i) for i in range(4)])
    jl = _labels(3, 1, 61, 83)
    before = eng.launch_count()
    got, moved = run(eng, frames, [0, 2, 3], [P(seed=1), P(elastic_sigma=-1.0), P()], torch.from_numpy(jl.copy()).cuda())
    assert eng.launch_count() == before
    assert_same(got, frames)
    assert np.array_equal(moved, jl, equal_nan=True)


def test_invalid_arguments_launch_nothing(eng):
    from deepgraphpose_b200 import _lib as L
    lib = eng.lib
    H, W, nt = 20, 30, 3
    fr = torch.zeros((nt, H, W, 3), dtype=torch.uint8, device="cuda")
    jl = torch.zeros((2, NJ, 2), dtype=torch.float64, device="cuda")
    dx = torch.zeros((H, W), dtype=torch.float32, device="cuda")
    good = [P(rotate_deg=5.0), P(elastic_alpha=3.0)]

    def call(idx, params, H=H, W=W, nt=nt, frames=fr.data_ptr(), jl_ptr=jl.data_ptr(), stride=STRIDE):
        idx = np.asarray(idx, np.int32)
        par = (L.DgpAugmentParams * max(len(params), 1))(*[L.DgpAugmentParams(**p) for p in params])
        return lib.dgp_augment(eng.h, frames, nt, H, W, idx.ctypes.data, len(idx), par, jl_ptr, stride, None)

    before = eng.launch_count()
    cases = [
        ([0, 3], good), ([-1, 0], good), ([1, 1], good),                               # index outside [0, nt), duplicate
        ([0, 1], [P(blur_k=4), good[1]]), ([0, 1], [P(blur_k=1), good[1]]), ([0, 1], [P(blur_k=17), good[1]]),
        ([0, 1], [good[0], P(elastic_alpha=3.0, elastic_sigma=0.0)]),
        ([0, 1], [good[0], P(elastic_alpha=3.0, elastic_sigma=-2.0)]),
        ([0, 1], [good[0], P(elastic_alpha=3.0, elastic_sigma=17.0)]),
        ([0, 1], [P(drop_p=1.5, drop_size_percent=0.1), good[1]]), ([0, 1], [P(rotate_deg=float("nan")), good[1]]),
        ([0, 1], [P(blur_k=7, blur_direction=2.0), good[1]]),
    ]
    for idx, params in cases:
        assert call(idx, params) == -1, (idx, params)
    assert call([0, 1], good, H=40000) == -1 and call([0, 1], good, W=0) == -1
    assert call([0, 1], good, H=30000, W=30000) == -1                                  # frame bytes overflow int
    assert call([0, 1], good, frames=0) == -1 and call([0, 1], good, stride=0.0) == -1
    assert lib.dgp_elastic_field(eng.h, H, W, 1.0, 0.0, 1, dx.data_ptr(), dx.data_ptr(), None) == -1
    assert lib.dgp_elastic_field(eng.h, H, W, 1.0, 2.0, 1, None, dx.data_ptr(), None) == -1
    assert eng.launch_count() == before
    assert call([0, 1], good) == 0 and eng.launch_count() > before


# ---------------------------------------------------------------------------------------------------- training loops
def _fit(labeled_only, pipeline, seed=3):
    from deepgraphpose_b200 import fitdgp
    from test_gpu_drivers import NT, _Batcher, _cfg
    b = _Batcher(seed=seed)
    frame_lists = ([b.visible], [np.array([], dtype=np.int64)], [np.arange(NT)])
    if labeled_only:
        hist = fitdgp.fit_dgp_labeledonly("synthetic:0", "/nonexistent", saveiters=100, data_batcher=b, dgp_cfg=_cfg(),
                                          frame_lists=frame_lists, batch_ind_all=[np.array([5, 0]), np.array([1, 0])] * 2,
                                          snapshot_fn=lambda *a: None, verbose=False, aug_pipeline=pipeline)
    else:
        windows = [np.array([0, 1, 2, 3, 0], dtype=np.int32), np.array([4, 5, 6, 7, 0], dtype=np.int32),
                   np.array([7, 8, 9, 10, 0], dtype=np.int32)]
        hist = fitdgp.fit_dgp("synthetic:0", "/nonexistent", batch_size=4, gm2=1, gm3=3, wt=0, saveiters=100, displayiters=100,
                              data_batcher=b, dgp_cfg=_cfg(), frame_lists=frame_lists, batch_ind_all=windows,
                              snapshot_fn=lambda *a: None, verbose=False, aug_pipeline=pipeline)
    return [{k: float(v) for k, v in h.items()} for h in hist]


@pytest.mark.parametrize("labeled_only", [False, True])
def test_fit_loops_with_a_seeded_pipeline(labeled_only):
    from deepgraphpose_b200.fitdgp_util import build_aug
    plain = _fit(labeled_only, None)
    assert _fit(labeled_only, build_aug(apply_prob=0, seed=1)) == plain
    a = _fit(labeled_only, build_aug(apply_prob=1, seed=7))
    b = _fit(labeled_only, build_aug(apply_prob=1, seed=7))
    assert a == b
    assert a != plain and all(np.isfinite(list(h.values())).all() for h in a)


def test_data_aug_leaves_its_inputs_and_feeds_device_tensors():
    from deepgraphpose_b200.fitdgp_util import build_aug, data_aug
    frames = np.stack([frame(64, 96, i) for i in range(5)]).astype(np.float64)
    jl = _labels(2, 2, 64, 96)
    fr, moved = data_aug(frames, [1, 3], jl.copy(), build_aug(apply_prob=1, seed=3), {"stride": STRIDE})
    assert fr.is_cuda and fr.dtype == torch.uint8 and moved.is_cuda and moved.dtype == torch.float64
    got = fr.cpu().numpy()
    assert_same(got[[0, 2, 4]], frames[[0, 2, 4]].astype(np.uint8))
    assert not np.array_equal(got[1], frames[1].astype(np.uint8))
    assert np.array_equal(np.isnan(moved.cpu().numpy()), np.isnan(jl))
    dev = torch.from_numpy(frames.astype(np.uint8)).cuda()
    fr2, _ = data_aug(dev, [1, 3], torch.from_numpy(jl).cuda(), build_aug(apply_prob=1, seed=3), {"stride": STRIDE})
    assert_same(fr2.cpu().numpy(), got)
    assert_same(dev.cpu().numpy(), frames.astype(np.uint8))
