"""Frame resize + crop on the device (dgp_resize_crop and the estimate_pose entries' new_size / crop_size): bit-identical
to the reference's per-frame PIL.Image.resize (Pillow's default filter, BICUBIC) + crop, and estimate_pose's read-outs
on device-transformed frames bit-identical to the untransformed entries on frames PIL transformed on the host."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from deepgraphpose_b200 import synthetic
from test_resize import GRID, frame, pil

pytestmark = pytest.mark.gpu
NJ = 4


@pytest.fixture(scope="module")
def eng():
    from deepgraphpose_b200.engine import Engine
    e = Engine(NJ, location_refinement=False)
    e.load_weights(synthetic.make_weights(NJ, seed=0, location_refinement=False))
    yield e
    e.close()


def _device_vs_pil(eng, frames, new_size, crop):
    got = eng.resize_crop(torch.from_numpy(frames).cuda(), new_size, crop).cpu().numpy()
    ref = np.stack([pil(f, new_size, crop) for f in frames])
    assert got.shape == ref.shape
    bad = np.argwhere(got != ref)
    assert bad.size == 0, "%d bytes differ, first at %s" % (len(bad), bad[:3].tolist())


@pytest.mark.parametrize("case", range(len(GRID)))
def test_resize_crop_equals_pillow_on_grid(eng, case):
    H0, W0, new_size, crop = GRID[case]
    frames = np.stack([frame(H0, W0, 100 * case + i) for i in range(3)])
    _device_vs_pil(eng, frames, new_size, crop)


@pytest.mark.parametrize("H0,W0,new_size,crop", [
    (1494, 1664, (747, 832), None),
    (1080, 1920, (540, 960), None),
    (480, 640, (747, 832), None),
    (1494, 1664, (747, 832), (40, 17, 700, 707)),
])
def test_resize_crop_equals_pillow_at_video_sizes(eng, H0, W0, new_size, crop):
    _device_vs_pil(eng, np.stack([frame(H0, W0, i) for i in range(2)]), new_size, crop)


def test_resize_crop_odd_widths_batches_and_unaligned_sources(eng):
    """Odd frame sizes put rows and frames at every byte alignment; a batch gives each frame the result it gets alone."""
    frames = np.stack([frame(37, 53, 40 + i) for i in range(7)])
    for new_size, crop in (((29, 41), None), ((61, 77), (-3, 5, 70, 50)), (None, (3, 1, 50, 36)), ((37, 21), None)):
        _device_vs_pil(eng, frames, new_size, crop)
        dev = torch.from_numpy(frames).cuda()
        whole = eng.resize_crop(dev, new_size, crop)
        for i in range(frames.shape[0]):
            # dev[i:i + 1] starts at an odd byte offset for odd i: the passes must not assume an aligned source
            assert torch.equal(eng.resize_crop(dev[i:i + 1], new_size, crop), whole[i:i + 1])


def _transformed(frames, new_size, crop):
    return np.stack([pil(f, new_size, crop) for f in frames])


def _same(a, b):
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_estimate_pose_host_with_transform_equals_host_pil_path(eng):
    frames, _ = synthetic.make_video(23, 150, 190, NJ, seed=3)
    for new_size, crop in (((96, 128), None), ((120, 150), (6, 9, 134, 105)), (None, (-8, 20, 120, 116))):
        ref = eng.estimate_pose_host(torch.from_numpy(_transformed(frames, new_size, crop)), batch=5)
        got = eng.estimate_pose_host(torch.from_numpy(frames), batch=5, new_size=new_size, crop_size=crop)
        _same(got, ref)


def test_estimate_pose_stream_with_transform_equals_host_pil_path(eng):
    frames, _ = synthetic.make_video(9, 150, 190, NJ, seed=4)
    new_size, crop = (120, 150), (6, 9, 134, 105)
    video = np.stack([frames[t % 9] for t in range(23)])
    ref = eng.estimate_pose_host(torch.from_numpy(_transformed(video, new_size, crop)), batch=5)
    got = eng.estimate_pose_stream(iter(video), 150, 190, 23, batch=5, new_size=new_size, crop_size=crop)
    _same(got, ref)
    pool = torch.from_numpy(frames).pin_memory()
    got = eng.estimate_pose_stream(pool, 150, 190, 23, batch=5, new_size=new_size, crop_size=crop)
    _same(got, ref)
    got = eng.estimate_pose_stream(pool, 150, 190, 11, batch=5, start=6, new_size=new_size, crop_size=crop)
    _same(got, tuple(r[6:17] for r in ref))


def test_sharded_one_rank_with_transform_equals_unsharded(eng):
    from deepgraphpose_b200 import eval as dgp_eval
    frames, _ = synthetic.make_video(11, 150, 190, NJ, seed=6)
    new_size, crop = (96, 128), (0, 4, 120, 90)
    edges = synthetic.chain_skeleton(NJ)
    ws, ws_max = np.full(3, 12.0, np.float32), np.full(3, 90.0, np.float32)
    res = dgp_eval.estimate_pose_sharded(eng, torch.from_numpy(frames).pin_memory(), 11, 150, 190, edges, ws, ws_max, 0.0,
                                         batch=4, new_size=new_size, crop_size=crop)
    ref = dgp_eval.estimate_pose_stream(eng, iter(frames), 150, 190, 11, batch=4, new_size=new_size, crop_size=crop)
    for k in ("x", "y", "likelihoods", "mu_likelihoods", "markers"):
        assert np.array_equal(res[k], ref[k]), k
    host = dgp_eval.estimate_pose_frames(eng, _transformed(frames, new_size, crop), batch=4)
    assert np.array_equal(res["markers"], host["markers"])


def _write_avi(path, frames):
    import cv2
    vw = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"MJPG"), 30, (frames.shape[2], frames.shape[1]))
    assert vw.isOpened()
    for f in frames:
        vw.write(np.ascontiguousarray(f[:, :, ::-1]))
    vw.release()


def test_eval_estimate_pose_video_and_array_with_transform(eng, tmp_path):
    """estimate_pose on an MJPG .avi / an array: the labels of the previous host path (decode, PIL resize + crop per frame,
    estimate_pose_frames, coordinates scaled back to the video)."""
    from deepgraphpose_b200 import eval as dgp_eval
    from deepgraphpose_b200.engine import Engine
    frames, _ = synthetic.make_video(13, 150, 190, NJ, seed=7)
    video = tmp_path / "clip.avi"
    _write_avi(video, frames)
    decoded = np.stack(list(dgp_eval._iter_video(video)))
    cfg = {"num_joints": NJ, "stride": 8.0}
    ref_eng = Engine(NJ, location_refinement=False)
    ref_eng.load_weights(dgp_eval.load_variables("synthetic:0", NJ, False))
    for new_size, crop in (((96, 128), (5, 3, 120, 90)), (None, (10, 20, 170, 140))):
        res = dgp_eval.estimate_pose_frames(ref_eng, _transformed(decoded, new_size, crop), batch=4)
        sx, sy = (190 / new_size[1], 150 / new_size[0]) if new_size is not None else (1.0, 1.0)
        for src in (str(video), decoded):
            out = tmp_path / ("out_%s_%d" % (new_size is None, isinstance(src, str)))
            got = dgp_eval.estimate_pose(cfg, "synthetic:0", src, str(out), save_pose=False, new_size=new_size, crop_size=crop,
                                         batch=4)
            assert np.array_equal(got["x"], res["x"] * sx) and np.array_equal(got["y"], res["y"] * sy)
            assert np.array_equal(got["likelihoods"], res["likelihoods"])
    ref_eng.close()


def test_stream_with_transform_keeps_host_memory_bounded(eng):
    """The ring holds source-size frames: resident memory does not grow with the video."""
    import psutil
    from deepgraphpose_b200 import eval as dgp_eval
    base, _ = synthetic.make_video(8, 192, 256, NJ, seed=8)
    n = 3000

    def gen():
        for t in range(n):
            yield base[t % 8]

    kw = dict(new_size=(96, 128), crop_size=(0, 0, 128, 96))
    dgp_eval.estimate_pose_stream(eng, gen(), 192, 256, n_frames=64, batch=32, **kw)   # warm-up: ring, tables, plans
    proc = psutil.Process(os.getpid())
    rss0 = proc.memory_info().rss
    res = dgp_eval.estimate_pose_stream(eng, gen(), 192, 256, n_frames=None, batch=32, **kw)
    grown = proc.memory_info().rss - rss0
    assert res["x"].shape == (n, NJ) and np.array_equal(res["x"][:8], res["x"][8:16])
    assert grown < 64 * 2 ** 20, "resident memory grew by %.1f MB" % (grown / 2 ** 20)


def test_invalid_geometry_is_refused_and_launches_nothing(eng):
    from deepgraphpose_b200 import _lib
    frames = np.stack([frame(40, 50, i) for i in range(2)])
    dev = torch.from_numpy(frames).cuda()
    for new_size, crop in (((0, 10), None), ((-2, 5), None), (None, (5, 5, 5, 9)), (None, (9, 2, 3, 8))):
        with pytest.raises(ValueError):
            eng.resize_crop(dev, new_size, crop)
        with pytest.raises(ValueError):
            eng.estimate_pose_host(torch.from_numpy(frames), batch=2, new_size=new_size, crop_size=crop)
        with pytest.raises(ValueError):
            eng.estimate_pose_stream(iter(frames), 40, 50, 2, batch=2, new_size=new_size, crop_size=crop)
    out = torch.empty((2, 40, 50, 3), dtype=torch.uint8, device="cuda")
    before = eng.launch_count()
    for fields in ((0, 10, 0, 0, 0, 0), (0, 0, 3, 0, 0, 0), (0, 0, 0, 0, 0, 4), (20, 20, 9, 2, 1, 5)):
        t = _lib.DgpFrameTransform(*fields)
        assert eng.lib.dgp_resize_crop(eng.h, C.c_void_p(dev.data_ptr()), 2, 40, 50, C.byref(t), C.c_void_p(out.data_ptr()),
                                       None) == -1
        mu = torch.empty((2, NJ, 2))
        assert eng.lib.dgp_estimate_pose_host_transform(eng.h, C.c_void_p(frames.ctypes.data), 2, 40, 50, C.byref(t), 2, 1.0,
                                                        1.0, C.c_void_p(mu.data_ptr()), None, None) == -1
    torch.cuda.synchronize()
    assert eng.launch_count() == before
    # later calls are unaffected
    _device_vs_pil(eng, frames, (30, 20), (1, 2, 19, 29))
    got = eng.estimate_pose_host(torch.from_numpy(frames), batch=2, new_size=(64, 80))
    _same(got, eng.estimate_pose_host(torch.from_numpy(_transformed(frames, (64, 80), None)), batch=2))
