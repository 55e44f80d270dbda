"""Each kernel of the training backward and of the parameter arena on its own, against an explicit float64 (or exactly
rounded torch) reference.

The whole-network tests (test_gpu_train.py and friends) compare every variable's gradient with fp32 autograd under a bound
loose enough for ReLU masks and pool winners taken from rounded activations; an error confined to one channel group, one tap
or one tail unit of a kernel passes them.  These tests call the launchers of libdgp_b200.so directly through a small C shim
(tests/backward_kernels_shim.cu, built here into tests/build/) on synthetic inputs.  Wherever a comparison is bitwise, the
inputs lie on a grid of multiples of 2^-8 in a small range, so that the fp32 sums inside the kernels are exact and the only
rounding is the one the kernel's contract names."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SHIM_SRC = os.path.join(HERE, "backward_kernels_shim.cu")
SHIM_LIB = os.path.join(HERE, "build", "libbackward_kernels_shim.so")
CSRC = os.path.join(ROOT, "deepgraphpose_b200", "csrc")

ERR_INVALID = 1  # cudaErrorInvalidValue

_vp, _i, _f, _ll = C.c_void_p, C.c_int, C.c_float, C.c_longlong
SIGNATURES = {
    "shim_sizeof_wgrad_params": (_i, []),
    "shim_sizeof_bn_group": (_i, []),
    "shim_sizeof_dgrad_w_job": (_i, []),
    "shim_max_dgrad_w_jobs": (_i, []),
    "shim_masked_dgrad": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "shim_make_wgrad_params": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "shim_make_conv1_wgrad_params": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "shim_wgrad_info": (_ll, [_vp, _vp]),
    "shim_wgrad_gemm": (_i, [_vp, _vp, _vp, _vp]),
    "shim_wgrad_reduce": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "shim_prep_s2d": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp]),
    "shim_relu_bn_bwd_blocks": (_i, [_i, _i]),
    "shim_relu_bn_bwd": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    "shim_maxpool_relu_bwd_rows": (_i, [_i, _i, _i]),
    "shim_maxpool_relu_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "shim_bn_finalize_all": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp]),
    "shim_upsample2": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "shim_col2im_bwd": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "shim_head_bias_blocks": (_i, []),
    "shim_head_bias_grad": (_i, [_vp, _ll, _i, _vp, _vp, _vp, _vp]),
    "shim_scale_inplace": (_i, [_vp, _ll, _f, _vp]),
    "shim_build_dgrad_w": (_i, [_vp, _i, _i, _vp, _vp, _i, _vp]),
    "shim_build_head_dgrad_w": (_i, [_vp, _i, _i, _vp, _i, _i, _vp]),
    "shim_refresh_w16": (_i, [_vp, _vp, _ll, _i, _vp]),
    "shim_refresh_bn": (_i, [_vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _vp]),
    "shim_sqnorm_partials": (_i, []),
    "shim_global_norm": (_i, [_vp, _ll, _f, _f, _vp, _vp, _vp]),
}

BN_GROUP = np.dtype([("part_off", "<u8"), ("rd_off", "<u8"), ("rows", "<i4"), ("C", "<i4"), ("col", "<i4"), ("K4", "<i4")])
DGRAD_W_JOB = np.dtype([("w_off", "<u8"), ("wd", "<u8"), ("ch_off", "<i4"), ("Cout", "<i4"), ("taps", "<i4"), ("Cin", "<i4"),
                        ("tile_start", "<i4"), ("pad", "<i4")])
GRAD_MODE = np.dtype([("accumulate", "<i4"), ("out_scale", "<f4")])


def build_shim():
    """Compiles the shim against the library (same nvcc and flags), only when the shim, a csrc header, the C header or the
    library is newer than the last build.  The run-path is relative, so a built tree can be moved."""
    from deepgraphpose_b200 import build
    lib = build.build()
    deps = [SHIM_SRC, lib, os.path.join(ROOT, "include", "dgp_b200.h")]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    if os.path.exists(SHIM_LIB) and all(os.path.getmtime(d) <= os.path.getmtime(SHIM_LIB) for d in deps):
        return SHIM_LIB
    os.makedirs(os.path.dirname(SHIM_LIB), exist_ok=True)
    tmp = SHIM_LIB + ".%d.tmp" % os.getpid()
    cmd = [build._nvcc()] + build.NVCC_FLAGS + ["-shared", "-o", tmp, SHIM_SRC, "-L" + os.path.dirname(lib), "-ldgp_b200",
                                                "-Xlinker=-rpath,$ORIGIN/../../deepgraphpose_b200"]
    subprocess.check_call(cmd)
    os.replace(tmp, SHIM_LIB)
    return SHIM_LIB


def load_shim():
    lib = C.CDLL(build_shim())
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


@pytest.fixture(scope="module")
def shim():
    return load_shim()


@pytest.fixture(scope="module", params=["fp16", "bf16"])
def eng(request):
    from deepgraphpose_b200.engine import Engine
    e = Engine(4, precision=request.param)
    yield e
    e.close()


@pytest.fixture(params=[torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def dt(request):
    return request.param


# ---------------------------------------------------------------------------------------------------------------- helpers
_in_flight = []   # tensors whose pointers were handed to a launch: kept alive (and their blocks unshared) until ok()


def P(t):
    if t is None:
        return None
    _in_flight.append(t)
    return C.c_void_p(t.data_ptr())


def S():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ok(rc):
    assert rc == 0, rc
    torch.cuda.synchronize()
    _in_flight.clear()


def is_fp16(dtype):
    return 1 if dtype == torch.float16 else 0


def bits(t):
    return t.contiguous().view(torch.int16)


def grid(rng, shape, lim=64):
    """Multiples of 2^-8 in [-lim/256, lim/256]: exact in bf16 and fp16 for lim <= 255."""
    return rng.integers(-lim, lim + 1, size=shape).astype(np.float64) / 256.0


def to16(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(dtype)


def grad_mode(accumulate, out_scale):
    m = np.zeros(1, GRAD_MODE)
    m["accumulate"], m["out_scale"] = accumulate, out_scale
    return torch.from_numpy(m.view(np.uint8).copy()).cuda()


def im2col(x, R, dil):
    """x (N,H,W,C) float64 -> (N*H*W, R*R*C), stride 1, symmetric SAME padding; column = (r*R + s)*C + c."""
    N, H, W, Cc = x.shape
    p = dil * (R - 1) // 2
    xp = np.pad(x, ((0, 0), (p, p), (p, p), (0, 0)))
    cols = [xp[:, r * dil:r * dil + H, s * dil:s * dil + W, :] for r in range(R) for s in range(R)]
    return np.concatenate(cols, axis=3).reshape(N * H * W, R * R * Cc)


def s2d_reference(frames, mean):
    """prep_s2d's layout in float64 before rounding: pad 3 (conv2d_same), 2x2 space-to-depth, channel (u*2+v)*3+c, 4 zeros."""
    N, H, W, _ = frames.shape
    H1, W1 = -(-H // 2), -(-W // 2)
    Hs, Ws = H1 + 3, W1 + 3
    x = frames.astype(np.float64) - np.asarray(mean, np.float32).astype(np.float64)
    xp = np.zeros((N, 2 * Hs, 2 * Ws, 3))
    xp[:, 3:3 + H, 3:3 + W] = x
    out = np.zeros((N, Hs, Ws, 16))
    for u in range(2):
        for v in range(2):
            out[..., (u * 2 + v) * 3:(u * 2 + v) * 3 + 3] = xp[:, u::2, v::2][:, :Hs, :Ws]
    return out


def conv1_s2d_weights(w77):
    """The [64][256] space-to-depth matrix of a 7x7x3x64 conv1 (build_conv1_layer), and its mask of real taps."""
    wm = np.zeros((64, 256))
    mask = np.zeros((64, 256))
    for a in range(4):
        for b in range(4):
            for u in range(2):
                for v in range(2):
                    kh, kw = 2 * a + u, 2 * b + v
                    if kh >= 7 or kw >= 7:
                        continue
                    for c in range(3):
                        d = a * 64 + b * 16 + (u * 2 + v) * 3 + c
                        wm[:, d] = w77[kh, kw, c, :]
                        mask[:, d] = 1.0
    return wm, mask


def conv2d_same_7x7s2(x, w77):
    """slim conv2d_same(7, stride 2) in float64: x (N,H,W,3), w (7,7,3,64) -> (N,ceil(H/2),ceil(W/2),64)."""
    xt = torch.from_numpy(x).permute(0, 3, 1, 2)
    xt = F.pad(xt, (3, 3, 3, 3))
    y = F.conv2d(xt, torch.from_numpy(w77).permute(3, 2, 0, 1), stride=2)
    return y.permute(0, 2, 3, 1).numpy()


def maxpool_bwd_reference(x, gout, pad_t, pad_l):
    """Gradient of the 3x3 / 2 max-pool routed to the FIRST maximum of each window (row-major over the window's in-image
    positions, strict >), float64 sum per pixel.  x (N,H,W,C), gout (N,Ho,Wo,C)."""
    N, H, W, Cc = x.shape
    Ho, Wo = gout.shape[1], gout.shape[2]
    gx = np.zeros(x.shape)
    n_idx = np.arange(N)[:, None]
    c_idx = np.arange(Cc)[None, :]
    for p in range(Ho):
        for q in range(Wo):
            pos = [(y, xx) for y in range(2 * p - pad_t, 2 * p - pad_t + 3) for xx in range(2 * q - pad_l, 2 * q - pad_l + 3)
                   if 0 <= y < H and 0 <= xx < W]
            vals = np.stack([x[:, y, xx, :] for y, xx in pos], axis=1)       # (N, npos, C)
            win = np.argmax(vals, axis=1)                                     # first maximum
            ys = np.array([y for y, _ in pos])[win]
            xs = np.array([xx for _, xx in pos])[win]
            np.add.at(gx, (n_idx, ys, xs, c_idx), gout[:, p, q, :])
    return gx


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_shim_builds_links_and_loads():
    """The shim compiles for sm_100a against this commit's internal headers, links the library and loads; the structs the
    tests lay out in numpy have the library's sizes; the host-side sizing helpers answer without a device."""
    lib = load_shim()
    assert lib.shim_sizeof_bn_group() == BN_GROUP.itemsize
    assert lib.shim_sizeof_dgrad_w_job() == DGRAD_W_JOB.itemsize
    assert lib.shim_max_dgrad_w_jobs() == 256
    assert lib.shim_sizeof_wgrad_params() > 2 * 128
    assert lib.shim_relu_bn_bwd_blocks(1000, 64) == -(-1000 // 32)
    assert lib.shim_relu_bn_bwd_blocks(10 ** 6, 2048) == 148 * 4
    assert lib.shim_maxpool_relu_bwd_rows(3, 17, 33) == 3 * 3 * 2


def test_launchers_reject_invalid_arguments():
    """Argument checks that return before any launch (so they hold without a device)."""
    lib = load_shim()
    dummy = C.c_void_p(16)
    for Cc in (60, 24, 4096):           # C % 8, 256 % (C / 8), C / 8 > 256
        assert lib.shim_relu_bn_bwd(dummy, dummy, 64, Cc, dummy, 1, None, 0, 0, 0, 0, None) == ERR_INVALID
    # scatter source with M not a whole number of (H, W) images, or an empty image
    assert lib.shim_relu_bn_bwd(dummy, dummy, 100, 64, dummy, 1, dummy, 7, 7, 4, 4, None) == ERR_INVALID
    assert lib.shim_relu_bn_bwd(dummy, dummy, 98, 64, dummy, 1, dummy, 0, 7, 4, 4, None) == ERR_INVALID
    for pt, pl in ((2, 0), (0, -1)):
        assert lib.shim_maxpool_relu_bwd(dummy, dummy, 1, 8, 8, 4, 4, pt, pl, dummy, dummy, 1, None) == ERR_INVALID
    assert lib.shim_head_bias_grad(dummy, 10, 257, dummy, dummy, None, None) == ERR_INVALID
    assert lib.shim_build_dgrad_w(dummy, 257, 1000, dummy, dummy, 1, None) == ERR_INVALID
    assert lib.shim_global_norm(dummy, 1022, 1.0, 10.0, dummy, dummy, None) == ERR_INVALID
    assert lib.shim_refresh_w16(dummy, dummy, 12, 1, None) == ERR_INVALID


@pytest.mark.parametrize("H,W,pad_t,pad_l", [(6, 9, 0, 1), (7, 8, 1, 0), (5, 5, 1, 1), (8, 6, 0, 0)])
def test_maxpool_reference_routes_like_autograd(H, W, pad_t, pad_l):
    """On tie-free input the reference's routing is torch max_pool2d's (and TF's MaxPoolGrad's), with -inf padding."""
    rng = np.random.default_rng(H * 100 + W * 10 + pad_t * 2 + pad_l)
    N, Cc = 2, 3
    Ho, Wo = -(-H // 2), -(-W // 2)
    x = rng.permutation(N * H * W * Cc).reshape(N, H, W, Cc).astype(np.float64) + 1.0
    gout = rng.standard_normal((N, Ho, Wo, Cc))
    pad_b, pad_r = 2 * (Ho - 1) + 3 - H - pad_t, 2 * (Wo - 1) + 3 - W - pad_l
    xt = torch.from_numpy(x).permute(0, 3, 1, 2).requires_grad_(True)
    y = F.max_pool2d(F.pad(xt, (pad_l, pad_r, pad_t, pad_b), value=-np.inf), 3, 2)
    assert y.shape[2:] == (Ho, Wo)
    (y * torch.from_numpy(gout).permute(0, 3, 1, 2)).sum().backward()
    ref = xt.grad.permute(0, 2, 3, 1).numpy()
    np.testing.assert_allclose(maxpool_bwd_reference(x, gout, pad_t, pad_l), ref, rtol=0, atol=1e-12)


@pytest.mark.parametrize("H,W", [(13, 18), (16, 11)])
def test_conv1_space_to_depth_map_is_conv2d_same(H, W):
    """A 4x4 stride-1 conv of the space-to-depth input with the mapped [64][256] matrix is slim's 7x7 / 2 conv2d_same; the
    mask marks exactly the 7x7x3 real taps."""
    rng = np.random.default_rng(H * W)
    frames = rng.integers(0, 256, (2, H, W, 3)).astype(np.uint8)
    mean = (123.68, 116.779, 103.939)
    w77 = rng.standard_normal((7, 7, 3, 64))
    wm, mask = conv1_s2d_weights(w77)
    assert mask.sum() == 64 * 7 * 7 * 3
    s2d = s2d_reference(frames, mean)
    H1, W1 = -(-H // 2), -(-W // 2)
    cols = np.concatenate([s2d[:, a:a + H1, b:b + W1, :] for a in range(4) for b in range(4)], axis=3)
    got = cols.reshape(-1, 256) @ wm.T
    ref = conv2d_same_7x7s2(frames.astype(np.float64) - np.asarray(mean, np.float32).astype(np.float64), w77)
    np.testing.assert_allclose(got.reshape(ref.shape), ref, rtol=0, atol=1e-9 * np.abs(ref).max())


# ---------------------------------------------------------------------------------------------------------------- GPU
DGRAD_CASES = [
    # images, H, W, K (dy channels), N (out channels), R, dilation, residual
    (1, 16, 16, 64, 64, 1, 1, False),       # M = 256: whole 256-row tiles (msub 2)
    (2, 10, 8, 128, 128, 1, 1, True),       # M = 160: 32-row units but a partial 128-row tile
    (2, 13, 17, 64, 256, 1, 1, False),      # M = 442: tail unit of 26 rows
    (3, 13, 17, 128, 512, 1, 1, True),      # M = 663, CTA pair, shortcut dgrad (+ Gy)
    (1, 16, 32, 64, 1024, 1, 1, False),     # M = 512, CTA pair
    (1, 12, 12, 256, 2048, 1, 1, True),     # M = 144: tail of 16 rows, 8 column blocks
    (2, 13, 17, 128, 64, 3, 1, True),       # 3x3, msub 2, tail
    (1, 15, 19, 256, 128, 3, 2, False),     # dilation 2, M = 285
    (1, 24, 20, 128, 256, 3, 4, True),      # dilation 4, M = 480
    (2, 16, 16, 128, 512, 3, 2, False),     # dilation 2, CTA pair, M = 512
    (1, 20, 26, 256, 1024, 3, 4, True),     # dilation 4, CTA pair, M = 520
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", DGRAD_CASES, ids=[str(i) for i in range(len(DGRAD_CASES))])
def test_masked_dgrad_epilogue(shim, eng, case):
    """conv_gemm_kernel<kMask>: out = (GEMM + residual) * [act > 0] rounded once, and colsum_part[r][n] = the sum of the
    stored out over rows 32r .. min(32r + 31, M - 1); rows past M are neither stored nor summed."""
    nimg, H, W, K, N, R, dil, res = case
    dtype = eng.act_dtype
    rng = np.random.default_rng(sum(case[:7]) * 31 + res)
    M = nimg * H * W
    dy = to16(grid(rng, (nimg, H, W, K)), dtype).cuda()
    w = to16(grid(rng, (N, R * R * K)), dtype).cuda()
    act = to16(rng.choice([-1.0, 0.0, 0.0, 0.5, 1.0, 2.0], (M + 64, N)), dtype).cuda()
    residual = to16(grid(rng, (M, N), 255), dtype).cuda() if res else None
    sentinel = torch.full((M + 64, N), 0x3C01, dtype=torch.int16)
    out = sentinel.clone().view(dtype).cuda()
    nunits = -(-M // 32)
    colsum = torch.full((nunits + 2, N), float("nan"), device="cuda")
    info = (C.c_int * 3)()
    ok(shim.shim_masked_dgrad(eng.h, P(dy), nimg, H, W, K, P(w), N, R, dil, P(out), P(act), P(colsum), P(residual), S(), info))
    assert info[0] == 1, "the mask rides only in the staged epilogue"
    if N <= 128:
        assert info[1] == 2
    if N >= 256 and M >= 512:
        assert info[2] == 1

    ref = im2col(dy.double().cpu().numpy(), R, dil) @ w.double().cpu().numpy().T
    if res:
        ref = ref + residual.double().cpu().numpy()
    got = out.cpu()
    a = act.cpu()[:M].float().numpy()
    o = got[:M].double().numpy()
    masked = a <= 0
    assert (bits(got[:M]).numpy()[masked] == 0).all(), "masked entries must be +0"
    tol = 8e-4 if dtype == torch.float16 else 6e-3
    err = np.abs(o - ref)[~masked].max() / np.abs(ref).max()
    assert err < tol, err
    assert torch.equal(bits(got[M:]), sentinel[M:]), "rows past M were written"

    cs = colsum.cpu().double().numpy()
    assert np.isnan(cs[nunits:]).all()
    rows = np.arange(nunits)
    unit_sum = np.add.reduceat(o, rows * 32, axis=0)
    unit_abs = np.add.reduceat(np.abs(o), rows * 32, axis=0)
    assert np.isfinite(cs[:nunits]).all(), "a 32-row unit left no dbeta partial"
    assert (np.abs(cs[:nunits] - unit_sum) <= 1e-6 * unit_abs).all()


WGRAD_CASES = [
    # images, H, W, Cin, Cout, R, reduce variant (threads per float4 of the gradient) on 148 SMs
    (4, 47, 52, 64, 64, 1, 16),
    (2, 30, 40, 64, 256, 3, 4),
    (1, 9, 11, 2048, 512, 1, 1),
]


def reduce_variant(splits, Cout, Kw):
    total = Cout * Kw // 4
    if splits >= 32 and total <= 32768:
        return 16
    if splits >= 8 and total <= 262144:
        return 4
    return 1


@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD_CASES, ids=["sg16", "sg4", "sg1"])
def test_wgrad_reduce_modes(shim, eng, case):
    """wgrad_reduce_kernel: the plain result is the fixed-order sum of the GEMM's split partials; every other mode is that
    result put through ((raw * rowscale) * mask) * out_scale (+ old), bitwise, and rowdot_part is <W, raw> per float4."""
    nimg, H, W, Cin, Cout, R, sg = case
    if torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the split counts of these shapes are chosen for 148 SMs")
    dtype = eng.act_dtype
    rng = np.random.default_rng(Cin + Cout + R)
    x = to16(grid(rng, (nimg, H, W, Cin)), dtype).cuda()
    dy = to16(grid(rng, (nimg, H, W, Cout)), dtype).cuda()
    wp = C.create_string_buffer(shim.shim_sizeof_wgrad_params())
    ok(shim.shim_make_wgrad_params(eng.h, R, Cin, Cout, 1, 1, P(x), nimg, H, W, 1 if R > 1 else 0, P(dy), wp))
    info = (C.c_int * 5)()
    ws_bytes = shim.shim_wgrad_info(wp, info)
    _, Kw, nmb, nnb, splits = list(info)
    assert Kw == R * R * Cin
    assert reduce_variant(splits, Cout, Kw) == sg
    part = torch.empty(ws_bytes // 4, device="cuda")
    ok(shim.shim_wgrad_gemm(eng.h, wp, P(part), S()))

    def run(rowscale=None, mask=None, mode=None, wmaster=None, rowdot=None, init=None):
        g = (torch.full((Cout, Kw), float("nan")) if init is None else init.clone()).cuda()
        ok(shim.shim_wgrad_reduce(wp, P(part), P(rowscale), P(mask), P(g), P(mode), P(wmaster), P(rowdot), S()))
        return g.cpu()

    raw = run()
    # against the float64 weight gradient and the float64 sum of the partials
    ref = im2col(x.double().cpu().numpy(), R, 1).T @ dy.double().cpu().numpy().reshape(-1, Cout)
    assert np.abs(raw.double().numpy() - ref.T).max() <= 2e-5 * np.abs(ref).max()
    pt = part.cpu().double().view(nmb, nnb, splits, 128, 256)
    psum = pt.sum(2).permute(0, 2, 1, 3).reshape(nmb * 128, nnb * 256)[:Cout, :Kw]
    pabs = pt.abs().sum(2).permute(0, 2, 1, 3).reshape(nmb * 128, nnb * 256)[:Cout, :Kw]
    assert ((raw.double() - psum).abs() <= 1e-6 * pabs).all()

    rs = torch.from_numpy(rng.uniform(0.5, 1.5, Cout).astype(np.float32))
    mask = torch.from_numpy((rng.random((Cout, Kw)) < 0.7).astype(np.float32))
    old = torch.from_numpy(rng.standard_normal((Cout, Kw)).astype(np.float32))
    wm = torch.from_numpy(rng.standard_normal((Cout, Kw)).astype(np.float32))
    assert torch.equal(run(rowscale=rs.cuda()), raw * rs[:, None])
    assert torch.equal(run(mask=mask.cuda()), raw * mask)
    assert torch.equal(run(mode=grad_mode(0, 1.0)), raw)
    assert torch.equal(run(mode=grad_mode(0, 1.0 / 1024)), raw * (1.0 / 1024))
    assert torch.equal(run(mode=grad_mode(1, 1.0), init=old), old + raw)
    rowdot = torch.full((Cout * Kw // 4,), float("nan"), device="cuda")
    got = run(rowscale=rs.cuda(), mask=mask.cuda(), mode=grad_mode(1, 1.0 / 1024), init=old, wmaster=wm.cuda(), rowdot=rowdot)
    assert torch.equal(got, old + ((raw * rs[:, None]) * mask) * (1.0 / 1024))
    terms = (raw.double() * wm.double()).view(-1, 4)
    rd = rowdot.cpu().double()
    assert ((rd - terms.sum(1)).abs() <= 1e-6 * terms.abs().sum(1)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,W", [(2, 37, 50), (2, 44, 29)])
def test_conv1_wgrad(shim, eng, N, H, W):
    """conv1's weight gradient through prep_s2d and make_conv1_wgrad_params, reduced with the BN scale and the mask of
    real taps, against float64 autograd of slim's 7x7 / 2 conv2d_same on the 16-bit mean-subtracted image."""
    dtype = eng.act_dtype
    rng = np.random.default_rng(N * H * W)
    mean = (123.68, 116.779, 103.939)
    frames = rng.integers(0, 256, (N, H, W, 3)).astype(np.uint8)
    H1, W1 = -(-H // 2), -(-W // 2)
    Hs, Ws = H1 + 3, W1 + 3
    s2d = torch.empty((N, Hs, Ws, 16), dtype=dtype, device="cuda")
    fr = torch.from_numpy(frames).cuda()
    ok(shim.shim_prep_s2d(P(fr), N, H, W, (C.c_float * 3)(*mean), P(s2d), Hs, Ws, is_fp16(dtype), S()))
    s2d_ref = to16(s2d_reference(frames, mean), dtype)
    assert torch.equal(bits(s2d.cpu()), bits(s2d_ref))

    dy = to16(grid(rng, (N * H1 * W1, 64)), dtype).cuda()
    wp = C.create_string_buffer(shim.shim_sizeof_wgrad_params())
    ok(shim.shim_make_conv1_wgrad_params(eng.h, P(dy), P(s2d), N, H1, W1, Hs, Ws, wp))
    info = (C.c_int * 5)()
    part = torch.empty(shim.shim_wgrad_info(wp, info) // 4, device="cuda")
    assert tuple(info)[:2] == (64, 256)
    ok(shim.shim_wgrad_gemm(eng.h, wp, P(part), S()))
    scale = torch.from_numpy(rng.uniform(0.5, 1.5, 64).astype(np.float32))
    _, mask = conv1_s2d_weights(np.zeros((7, 7, 3, 64)))
    grad = torch.full((64, 256), float("nan"), device="cuda")
    ok(shim.shim_wgrad_reduce(wp, P(part), P(scale.cuda()), P(torch.from_numpy(mask.astype(np.float32)).cuda()), P(grad),
                              None, None, None, S()))

    x = torch.from_numpy((frames.astype(np.float32) - np.asarray(mean, np.float32))).to(dtype).double()
    w77 = torch.zeros((7, 7, 3, 64), dtype=torch.float64, requires_grad=True)
    y = F.conv2d(F.pad(x.permute(0, 3, 1, 2), (3, 3, 3, 3)), w77.permute(3, 2, 0, 1), stride=2)
    (y * dy.cpu().double().view(N, H1, W1, 64).permute(0, 3, 1, 2)).sum().backward()
    ref, _ = conv1_s2d_weights(w77.grad.numpy())
    ref = ref * scale.double().numpy()[:, None]
    got = grad.cpu().double().numpy()
    assert (got[mask == 0] == 0).all(), "padded taps must be exactly 0"
    assert np.abs(got - ref).max() <= 2e-5 * np.abs(ref).max()


RELU_BN_CASES = [
    # M, C, scatter (N, H, W, P, Q) or None
    (1000, 64, None),
    (20000, 64, None),            # more rows than 592 blocks cover at once: grid-stride loop
    (777, 128, None),
    (4099, 256, None),
    (333, 512, None),
    (129, 1024, None),
    (45, 2048, None),
    (180, 256, (2, 10, 9, 5, 5)),      # H = 2P, W = 2Q - 1
    (216, 64, (2, 9, 12, 5, 6)),       # H = 2P - 1, W = 2Q
    (49, 2048, (1, 7, 7, 4, 4)),       # both odd
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", RELU_BN_CASES, ids=[str(i) for i in range(len(RELU_BN_CASES))])
def test_relu_bn_bwd(shim, dt, case):
    """dy = round16(g (+ zero-inserted d)) * [act > 0] in place, bitwise, and the per-block channel sums of the stored dy."""
    M, Cc, sc = case
    rng = np.random.default_rng(M * 7 + Cc)
    g = to16(grid(rng, (M, Cc), 255), dt)
    act = to16(rng.choice([-1.0, 0.0, 0.5, 1.0], (M, Cc)), dt)
    gsum = g.float().clone()
    d = None
    if sc is not None:
        N, H, W, Pp, Q = sc
        assert N * H * W == M
        d = to16(grid(rng, (N, Pp, Q, Cc), 255), dt)
        gsum.view(N, H, W, Cc)[:, ::2, ::2] += d.float()
    ref = torch.where(act.float() > 0, gsum, torch.zeros(())).to(dt)
    blocks = shim.shim_relu_bn_bwd_blocks(M, Cc)
    part = torch.full((blocks, Cc), float("nan"), device="cuda")
    gd = g.cuda()
    Hh, Ww, Pp, Q = (sc[1], sc[2], sc[3], sc[4]) if sc else (0, 0, 0, 0)
    ok(shim.shim_relu_bn_bwd(P(gd), P(act.cuda()), M, Cc, P(part), is_fp16(dt), P(d.cuda() if d is not None else None),
                             Hh, Ww, Pp, Q, S()))
    assert torch.equal(bits(gd.cpu()), bits(ref))
    stored = gd.cpu().double()
    total = part.cpu().double().sum(0)
    assert (torch.abs(total - stored.sum(0)) <= 1e-6 * stored.abs().sum(0)).all()


MAXPOOL_CASES = [
    # N, H, W, pad_t, pad_l
    (2, 5, 7, 0, 0),       # smaller than one 8 x 32 tile
    (2, 5, 7, 1, 1),
    (1, 3, 3, 1, 0),
    (3, 19, 45, 0, 1),
    (2, 26, 70, 1, 0),
    (2, 16, 64, 1, 1),     # whole tiles
    (1, 33, 31, 0, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", MAXPOOL_CASES, ids=[str(i) for i in range(len(MAXPOOL_CASES))])
def test_maxpool_relu_bwd(shim, dt, case):
    """Pooled gradient routed to each window's first maximum, conv1's ReLU mask, one rounding: bitwise, with ties among
    positive maxima common; the partial sums add up to the sum of the stored gx."""
    N, H, W, pad_t, pad_l = case
    rng = np.random.default_rng(N * H * W + pad_t * 2 + pad_l)
    Ho, Wo = -(-H // 2), -(-W // 2)
    x = to16(rng.choice([0.0, 0.5, 1.0, 1.5], (N, H, W, 64)), dt)
    gout = to16(grid(rng, (N, Ho, Wo, 64), 255), dt)
    ref = maxpool_bwd_reference(x.double().numpy(), gout.double().numpy(), pad_t, pad_l)
    ref = torch.from_numpy(np.where(x.double().numpy() > 0, ref, 0.0)).to(dt)
    rows = shim.shim_maxpool_relu_bwd_rows(N, H, W)
    part = torch.full((rows, 64), float("nan"), device="cuda")
    gx = torch.empty((N, H, W, 64), dtype=dt, device="cuda")
    ok(shim.shim_maxpool_relu_bwd(P(x.cuda()), P(gout.cuda()), N, H, W, Ho, Wo, pad_t, pad_l, P(gx), P(part), is_fp16(dt), S()))
    assert torch.equal(bits(gx.cpu()), bits(ref))
    assert torch.equal(part.cpu().double().sum(0), gx.cpu().double().sum((0, 1, 2)))


BN_LAYERS = [
    # channels, part columns (row stride), column of the layer's first channel, K4, partial rows
    (64, 64, 0, 16, 1),
    (128, 256, 128, 144, 127),
    (256, 256, 0, 576, 128),
    (64, 128, 64, 4608, 129),
    (512, 512, 0, 64, 600),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [None, (0, 1.0), (0, 1.0 / 1024), (1, 0.5)], ids=["none", "overwrite", "scaled", "accumulate"])
def test_bn_finalize_all(shim, mode):
    """dbeta = the float64 sum of each channel's dy partials; dgamma = (sum of rowdot - mean * dbeta) / sqrt(var + eps),
    through every GradMode."""
    rng = np.random.default_rng(3)
    groups, parts, rowdots = [], [], []
    part_off = rd_off = 0
    for Cc, Cp, col, K4, rows in BN_LAYERS:
        parts.append(rng.standard_normal(rows * Cp))
        rowdots.append(rng.standard_normal(Cc * K4))
        for c in range(0, Cc, 8):
            groups.append((part_off, rd_off + c * K4, rows, Cp, col + c, K4))
        part_off += rows * Cp
        rd_off += Cc * K4
    table = np.array(groups, BN_GROUP)
    n_ch = 8 * len(groups)
    part = np.concatenate(parts).astype(np.float32)
    rowdot = np.concatenate(rowdots).astype(np.float32)
    mean = rng.uniform(-2, 2, n_ch).astype(np.float32)
    var = rng.uniform(0.1, 3, n_ch).astype(np.float32)
    eps = 1e-3
    old_g = rng.standard_normal(n_ch).astype(np.float32)
    old_b = rng.standard_normal(n_ch).astype(np.float32)
    dgamma, dbeta = torch.from_numpy(old_g).cuda(), torch.from_numpy(old_b).cuda()
    tab = torch.from_numpy(table.view(np.uint8).copy()).cuda()
    md = grad_mode(*mode) if mode else None
    cuda = lambda a: torch.from_numpy(a).cuda()  # noqa: E731
    ok(shim.shim_bn_finalize_all(P(tab), len(groups), P(cuda(part)), P(cuda(rowdot)), P(cuda(mean)), P(cuda(var)), eps,
                                 P(dgamma), P(dbeta), P(md), S()))
    db, db_abs, s1, s1_abs = (np.zeros(n_ch) for _ in range(4))
    for gi, (po, ro, rows, Cp, col, K4) in enumerate(groups):
        for cl in range(8):
            c = gi * 8 + cl
            v = part[po + col + cl + Cp * np.arange(rows)].astype(np.float64)
            r = rowdot[ro + cl * K4:ro + (cl + 1) * K4].astype(np.float64)
            db[c], db_abs[c], s1[c], s1_abs[c] = v.sum(), np.abs(v).sum(), r.sum(), np.abs(r).sum()
    inv = 1.0 / np.sqrt(var.astype(np.float64) + np.float64(np.float32(eps)))
    dg = (s1 - mean * db) * inv
    tol_b = 1e-6 * db_abs
    tol_g = (2e-6 * (s1_abs + np.abs(mean) * db_abs) * inv + 1e-6 * np.abs(dg))
    scale = mode[1] if mode else 1.0
    if mode and mode[0]:
        db, dg = old_b + scale * db, old_g + scale * dg
    else:
        db, dg = scale * db, scale * dg
    tol_b = scale * tol_b + 1e-7 * np.abs(db)
    tol_g = scale * tol_g + 1e-7 * np.abs(dg)
    assert (np.abs(dbeta.cpu().double().numpy() - db) <= tol_b).all()
    assert (np.abs(dgamma.cpu().double().numpy() - dg) <= tol_g).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N,h,w,nj,locref,Kd", [(2, 5, 7, 4, True, 128), (1, 6, 9, 5, False, 64), (3, 3, 4, 17, True, 512)])
def test_col2im_bwd(shim, dt, N, h, w, nj, locref, Kd):
    """dG[m][(kh*3+kw)*ctot + co] = round16(head gradient at (2i+kh, 2j+kw)), zero outside the cropped map and in the padding
    columns past 9 * ctot."""
    rng = np.random.default_rng(N * h * w + nj)
    ctot = 3 * nj if locref else nj
    assert Kd > 9 * ctot
    gl = rng.standard_normal((N, 2 * h, 2 * w, nj)).astype(np.float32)
    gr = rng.standard_normal((N, 2 * h, 2 * w, 2 * nj)).astype(np.float32) if locref else None
    gall = np.concatenate([gl, gr], axis=3) if locref else gl
    gpad = np.zeros((N, 2 * h + 1, 2 * w + 1, ctot), np.float32)
    gpad[:, :2 * h, :2 * w] = gall
    ref = np.zeros((N, h, w, Kd), np.float32)
    for kh in range(3):
        for kw in range(3):
            t = kh * 3 + kw
            ref[..., t * ctot:(t + 1) * ctot] = gpad[:, kh:kh + 2 * h:2, kw:kw + 2 * w:2]
    dG = torch.empty((N * h * w, Kd), dtype=dt, device="cuda")
    ok(shim.shim_col2im_bwd(P(torch.from_numpy(gl).cuda()), P(torch.from_numpy(gr).cuda() if locref else None), N, h, w, ctot,
                            nj, P(dG), Kd, is_fp16(dt), S()))
    assert torch.equal(bits(dG.cpu()), bits(torch.from_numpy(ref.reshape(-1, Kd)).to(dt)))


@pytest.mark.gpu
@pytest.mark.parametrize("npix", [1, 4099, 100003])
@pytest.mark.parametrize("Cc", [1, 3, 5, 10, 17, 34, 85, 170, 256])
def test_head_bias_grad(shim, Cc, npix):
    rng = np.random.default_rng(Cc * 1000 + npix)
    g = rng.standard_normal((npix, Cc)).astype(np.float32)
    partial = torch.empty(shim.shim_head_bias_blocks() * 256, device="cuda")
    dbias = torch.full((Cc,), float("nan"), device="cuda")
    ok(shim.shim_head_bias_grad(P(torch.from_numpy(g).cuda()), npix, Cc, P(partial), P(dbias), None, S()))
    ref = g.astype(np.float64).sum(0)
    assert (np.abs(dbias.cpu().double().numpy() - ref) <= 1e-6 * np.abs(g).astype(np.float64).sum(0) + 1e-30).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N,P_,Q,H,W,Cc", [(2, 5, 6, 10, 11, 64), (1, 7, 4, 13, 8, 256), (3, 1, 1, 1, 2, 8)])
def test_upsample2(shim, dt, N, P_, Q, H, W, Cc):
    rng = np.random.default_rng(N + P_ * Q)
    x = to16(rng.standard_normal((N, P_, Q, Cc)), dt)
    ref = torch.zeros((N, H, W, Cc), dtype=dt)
    ref[:, ::2, ::2] = x[:, :-(-H // 2), :-(-W // 2)]
    out = torch.full((N, H, W, Cc), float("nan"), dtype=dt, device="cuda")
    ok(shim.shim_upsample2(P(x.cuda()), N, P_, Q, Cc, P(out), H, W, S()))
    assert torch.equal(bits(out.cpu()), bits(ref))


@pytest.mark.gpu
def test_scale_inplace(shim):
    rng = np.random.default_rng(11)
    x = torch.from_numpy(rng.standard_normal(1000003).astype(np.float32))
    xd = x.cuda()
    ok(shim.shim_scale_inplace(P(xd), x.numel(), 0.37, S()))
    assert torch.equal(xd.cpu(), x * np.float32(0.37))
    ok(shim.shim_scale_inplace(P(xd), 0, 2.0, S()))


@pytest.mark.gpu
def test_build_dgrad_w(shim, dt):
    """All 154 layers of a ResNet-152-sized table in one launch: wd[ci][T-1-tap][co] = round16(w[co][tap][ci] * scale[co])."""
    rng = np.random.default_rng(152)
    jobs, layers = [], []
    w_off = ch_off = wd_off = tiles = 0
    for j in range(154):
        Cin, Cout = int(rng.choice([32, 64, 96, 128])), int(rng.choice([32, 64, 128]))
        T = 9 if j % 3 == 1 else 1
        layers.append((w_off, ch_off, wd_off, Cout, T, Cin))
        jobs.append([w_off, wd_off, ch_off, Cout, T, Cin, tiles, 0])
        w_off += Cout * T * Cin
        ch_off += Cout
        wd_off += Cin * T * Cout
        tiles += (Cin // 32) * (Cout // 32) * T
    master = torch.from_numpy(rng.standard_normal(w_off).astype(np.float32))
    scale = torch.from_numpy(rng.uniform(0.2, 2.0, ch_off).astype(np.float32))
    wd = torch.zeros(wd_off, dtype=dt, device="cuda")
    table = np.zeros(len(jobs), DGRAD_W_JOB)
    for k, name in enumerate(DGRAD_W_JOB.names):
        table[name] = [jb[k] for jb in jobs]
    table["wd"] = wd.data_ptr() + 2 * table["wd"]   # element offsets -> device addresses
    tab = torch.from_numpy(table.view(np.uint8).copy()).cuda()
    ok(shim.shim_build_dgrad_w(P(tab), len(jobs), tiles, P(master.cuda()), P(scale.cuda()), is_fp16(dt), S()))
    got = wd.cpu()
    for wo, co, do, Cout, T, Cin in layers:
        w = master[wo:wo + Cout * T * Cin].view(Cout, T, Cin) * scale[co:co + Cout][:, None, None]
        ref = w.to(dt).flip(1).permute(2, 1, 0).reshape(-1)
        assert torch.equal(bits(got[do:do + Cin * T * Cout]), bits(ref)), (Cout, T, Cin)


@pytest.mark.gpu
def test_build_head_dgrad_w(shim, dt):
    rng = np.random.default_rng(9)
    rows, Cc, Kd = 9 * 12, 256, 128
    wh = torch.from_numpy(rng.standard_normal((rows, Cc)).astype(np.float32))
    whT = torch.full((Cc, Kd), float("nan"), dtype=dt, device="cuda")
    ok(shim.shim_build_head_dgrad_w(P(wh.cuda()), rows, Cc, P(whT), Kd, is_fp16(dt), S()))
    ref = torch.zeros((Cc, Kd), dtype=dt)
    ref[:, :rows] = wh.t().to(dt)
    assert torch.equal(bits(whT.cpu()), bits(ref))


@pytest.mark.gpu
def test_refresh_w16(shim, dt):
    """Round to nearest even, including halfway ties and subnormals; fp16 storage saturates at +-65504 (half_utils.cuh) where
    an RNE cast would give inf."""
    rng = np.random.default_rng(16)
    if dt == torch.float16:
        special = [1 + 2 ** -11, 1 + 3 * 2 ** -11, -(1 + 2 ** -11), 2 ** -24, 2 ** -25, 3 * 2 ** -25, 2 ** -26, 5 * 2 ** -16,
                   6e-5, -6e-8, 65504.0, 65519.0, 65520.0, 1e6, -7e4, 0.0, -0.0, 2.0 ** -14 * (1 + 2 ** -11)]
    else:
        special = [1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 2 ** -133, 3 * 2 ** -134, 2 ** -126 * (1 + 2 ** -8), 1e-40,
                   3.3895e38, 3.4028e38, -3.4028e38, 0.0, -0.0, 65520.0]
    vals = np.concatenate([np.array(special), rng.standard_normal(4000) * 10.0 ** rng.integers(-6, 6, 4000)])
    vals = np.concatenate([vals, np.zeros(-len(vals) % 8)]).astype(np.float32)
    master = torch.from_numpy(vals)
    out = torch.empty(len(vals), dtype=dt, device="cuda")
    ok(shim.shim_refresh_w16(P(master.cuda()), P(out), len(vals), is_fp16(dt), S()))
    ref = (master.clamp(-65504.0, 65504.0) if dt == torch.float16 else master).to(dt)
    assert torch.equal(bits(out.cpu()), bits(ref))


@pytest.mark.gpu
def test_refresh_bn(shim):
    rng = np.random.default_rng(17)
    n = 5000
    gamma, beta, mean = (rng.standard_normal(n).astype(np.float32) for _ in range(3))
    var = rng.uniform(0.0, 4.0, n).astype(np.float32)
    eps = np.float32(1e-5)
    scale, shift = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    cuda = lambda a: torch.from_numpy(a).cuda()  # noqa: E731
    ok(shim.shim_refresh_bn(P(cuda(gamma)), P(cuda(beta)), P(cuda(mean)), P(cuda(var)), float(eps), n, P(scale), P(shift), S()))
    s = scale.cpu().numpy()
    ref_s = gamma.astype(np.float64) / np.sqrt(var.astype(np.float64) + np.float64(eps))
    assert (np.abs(s - ref_s) <= 2 * np.spacing(np.abs(ref_s).astype(np.float32))).all()
    ref_t = beta.astype(np.float64) - mean.astype(np.float64) * s.astype(np.float64)
    prod = np.abs(mean.astype(np.float64) * s).astype(np.float32)
    tol = 2 * np.spacing(np.abs(ref_t).astype(np.float32)) + np.spacing(prod)
    assert (np.abs(shift.cpu().numpy() - ref_t) <= tol).all()


@pytest.mark.gpu
def test_global_norm(shim):
    """norm_clip = (|grad_scale| * ||g||, clip / max(norm, clip), or 1 when clip <= 0), against float64."""
    partial = torch.empty(shim.shim_sqnorm_partials(), device="cuda")
    norm_clip = torch.empty(2, device="cuda")

    def run(g, gs, clip):
        ok(shim.shim_global_norm(P(g), g.numel(), gs, clip, P(partial), P(norm_clip), S()))
        return norm_clip.cpu().double().numpy()

    gen = torch.Generator(device="cuda").manual_seed(5)
    big = torch.randn(60_000_004, device="cuda", generator=gen) * 1e-3
    ref = float(big.double().pow(2).sum().sqrt())
    for gs, clip in ((1.0, 10.0), (-0.5, 0.0), (2.0, -1.0), (1.0, 0.5 * ref), (-3.0, 1e6)):
        norm, f = run(big, gs, clip)
        want = abs(gs) * ref
        assert abs(norm - want) <= 1e-5 * want
        want_f = clip / max(want, clip) if clip > 0 else 1.0
        assert abs(f - want_f) <= 1e-5 * want_f, (gs, clip)
    assert run(big, 1.0, 0.5 * ref)[1] < 1.0
    zeros = torch.zeros(1024, device="cuda")
    assert tuple(run(zeros, 1.0, 10.0)) == (0.0, 1.0)
    assert tuple(run(zeros, 1.0, 0.0)) == (0.0, 1.0)
