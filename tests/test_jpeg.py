"""Motion-JPEG of the labelled video without a GPU: the numpy restatement of the encoding contract (include/dgp_b200.h,
DESIGN.md §4.5) byte-equal to Pillow's encoder, which the device encoder is compared against in test_gpu_jpeg.py; the mp4
muxer read back by OpenCV; argument checks that run before any engine exists."""
import io

import numpy as np
import pytest
from PIL import Image

ZZ = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
               21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60,
               61, 54, 47, 55, 62, 63])
LQ = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51,
               87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101,
               72, 92, 95, 98, 112, 100, 103, 99])
CQ = np.array([17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99,
               99, 99, 99] + [99] * 32)
DC_L_BITS = [0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]
DC_C_BITS = [0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0]
DC_VAL = list(range(12))
AC_L_BITS = [0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d]
AC_L_VAL = bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738393a434445"
    "464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3b4b5"
    "b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa")
AC_C_BITS = [0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77]
AC_C_VAL = bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a35363738393a4344"
    "45464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6a7a8a9aab2b3"
    "b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa")

SIZES = [(1, 1), (7, 9), (16, 16), (17, 33), (37, 53), (480, 640), (747, 832)]
QUALITIES = [1, 50, 75, 90, 95, 100]


def huff_codes(bits, vals):
    code, k, out = 0, 0, {}
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            out[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return out


def qtable(base, q):
    scale = 5000 // q if q < 50 else 200 - 2 * q
    return np.clip((base * scale + 50) // 100, 1, 255)


def fdct_islow(blocks):
    """libjpeg's jfdctint.c on (n, 8, 8) int64 centred samples: coefficients scaled by 8."""
    CB, P1 = 13, 2
    F = dict(a=2446, b=3196, c=4433, d=6270, e=7373, f=9633, g=12299, h=15137, i=16069, j=16819, k=20995, l=25172)

    def desc(x, n):
        return (x + (1 << (n - 1))) >> n

    def pass_(d, first):
        d0, d1, d2, d3, d4, d5, d6, d7 = [d[..., i] for i in range(8)]
        t0, t7, t1, t6, t2, t5, t3, t4 = d0 + d7, d0 - d7, d1 + d6, d1 - d6, d2 + d5, d2 - d5, d3 + d4, d3 - d4
        t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
        o = [None] * 8
        sh = CB - P1 if first else CB + P1
        if first:
            o[0], o[4] = (t10 + t11) << P1, (t10 - t11) << P1
        else:
            o[0], o[4] = desc(t10 + t11, P1), desc(t10 - t11, P1)
        z1 = (t12 + t13) * F["c"]
        o[2] = desc(z1 + t13 * F["d"], sh)
        o[6] = desc(z1 - t12 * F["h"], sh)
        z1, z2, z3, z4 = t4 + t7, t5 + t6, t4 + t6, t5 + t7
        z5 = (z3 + z4) * F["f"]
        t4, t5, t6, t7 = t4 * F["a"], t5 * F["j"], t6 * F["l"], t7 * F["g"]
        z1, z2, z3, z4 = -z1 * F["e"], -z2 * F["k"], -z3 * F["i"], -z4 * F["b"]
        z3 += z5
        z4 += z5
        o[7], o[5], o[3], o[1] = desc(t4 + z1 + z3, sh), desc(t5 + z2 + z4, sh), desc(t6 + z2 + z3, sh), desc(t7 + z1 + z4, sh)
        return np.stack(o, axis=-1)

    r = pass_(blocks, True)
    c = pass_(np.swapaxes(r, -1, -2), False)
    return np.swapaxes(c, -1, -2)


def quantize(coef, qt):
    d = (qt.reshape(8, 8) * 8).astype(np.int64)
    return np.sign(coef) * ((np.abs(coef) + (d >> 1)) // d)


def rgb_ycc(img):
    F = lambda x: int(x * 65536 + 0.5)  # noqa: E731
    r, g, b = [img[..., i].astype(np.int64) for i in range(3)]
    half, off = 1 << 15, 128 << 16
    y = (F(0.299) * r + F(0.587) * g + F(0.114) * b + half) >> 16
    cb = (-F(0.16874) * r - F(0.33126) * g + F(0.5) * b + off + half - 1) >> 16
    cr = (F(0.5) * r - F(0.41869) * g - F(0.08131) * b + off + half - 1) >> 16
    return y, cb, cr


class BitWriter:
    def __init__(self):
        self.acc, self.n, self.buf = 0, 0, bytearray()

    def put(self, code, length):
        self.acc = (self.acc << length) | (code & ((1 << length) - 1))
        self.n += length
        while self.n >= 8:
            byte = (self.acc >> (self.n - 8)) & 0xFF
            self.buf.append(byte)
            if byte == 0xFF:
                self.buf.append(0)
            self.n -= 8
        self.acc &= (1 << self.n) - 1 if self.n else 0

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def encode_reference(img, q):
    """The encoding contract in numpy: uint8 (H, W, 3) RGB -> the JPEG file's bytes."""
    H, W, _ = img.shape
    y, cb, cr = rgb_ycc(img)
    mcux, mcuy = -(-W // 16), -(-H // 16)
    ywib, yhib = -(-W // 8), -(-H // 8)
    Yp = np.pad(y, ((0, mcuy * 16 - H), (0, ywib * 8 - W)), mode="edge")
    cW, cH = -(-W // 2), -(-H // 2)
    cwib = -(-cW // 8)

    def down(p):
        pp = np.pad(p, ((0, 2 * cH - H), (0, cwib * 16 - W)), mode="edge")
        s = pp[0::2, 0::2] + pp[0::2, 1::2] + pp[1::2, 0::2] + pp[1::2, 1::2]
        bias = np.tile(np.array([1, 2]), cwib * 8 // 2 + 1)[: cwib * 8]
        return np.pad((s + bias[None, :]) >> 2, ((0, mcuy * 8 - cH), (0, 0)), mode="edge")

    qtl, qtc = qtable(LQ, q), qtable(CQ, q)

    def qblocks(p, wib, qt):
        R = p.shape[0] // 8
        bl = (p - 128).reshape(R, 8, wib, 8).transpose(0, 2, 1, 3)
        return quantize(fdct_islow(bl.reshape(-1, 8, 8)), qt).reshape(R, wib, 8, 8)

    QY, QCb, QCr = qblocks(Yp, ywib, qtl), qblocks(down(cb), cwib, qtc), qblocks(down(cr), cwib, qtc)
    dcl, acl = huff_codes(DC_L_BITS, DC_VAL), huff_codes(AC_L_BITS, AC_L_VAL)
    dcc, acc = huff_codes(DC_C_BITS, DC_VAL), huff_codes(AC_C_BITS, AC_C_VAL)
    out = bytearray(b"\xff\xd8" + b"\xff\xe0\x00\x10JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for t, qt in ((0, qtl), (1, qtc)):
        out += b"\xff\xdb\x00\x43" + bytes([t]) + bytes(qt[ZZ].astype(np.uint8))
    out += b"\xff\xc0\x00\x11\x08" + H.to_bytes(2, "big") + W.to_bytes(2, "big") + b"\x03\x01\x22\x00\x02\x11\x01\x03\x11\x01"
    for cls_id, bits, vals in ((0x00, DC_L_BITS, DC_VAL), (0x10, AC_L_BITS, AC_L_VAL), (0x01, DC_C_BITS, DC_VAL),
                               (0x11, AC_C_BITS, AC_C_VAL)):
        body = bytes([cls_id]) + bytes(bits) + bytes(vals)
        out += b"\xff\xc4" + (len(body) + 2).to_bytes(2, "big") + body
    out += b"\xff\xdd\x00\x04" + mcux.to_bytes(2, "big")
    out += b"\xff\xda\x00\x0c\x03\x01\x00\x02\x11\x03\x11\x00\x3f\x00"

    def enc_block(bw, blk, pred, dct, act):
        z = blk.reshape(64)[ZZ]
        diff = int(z[0]) - pred
        s = abs(diff).bit_length()
        bw.put(*dct[s])
        if s:
            bw.put(diff if diff > 0 else diff - 1, s)
        run = 0
        for k in range(1, 64):
            v = int(z[k])
            if v == 0:
                run += 1
                continue
            while run > 15:
                bw.put(*act[0xF0])
                run -= 16
            s = abs(v).bit_length()
            bw.put(*act[(run << 4) | s])
            bw.put(v if v > 0 else v - 1, s)
            run = 0
        if run:
            bw.put(*act[0x00])
        return int(z[0])

    for my in range(mcuy):
        bw = BitWriter()
        py = pcb = pcr = 0
        for mx in range(mcux):
            # a luma block outside the component is zero with the DC of the block before it in MCU order
            mb = []
            for yi in range(2):
                for xi in range(2):
                    if 2 * my + yi < yhib and 2 * mx + xi < ywib:
                        mb.append(QY[2 * my + yi, 2 * mx + xi])
                    else:
                        d = np.zeros((8, 8), np.int64)
                        d[0, 0] = mb[-1][0, 0]
                        mb.append(d)
            for b in mb:
                py = enc_block(bw, b, py, dcl, acl)
            pcb = enc_block(bw, QCb[my, mx], pcb, dcc, acc)
            pcr = enc_block(bw, QCr[my, mx], pcr, dcc, acc)
        bw.flush()
        out += bw.buf
        if my < mcuy - 1:
            out += bytes([0xFF, 0xD0 + (my % 8)])
    out += b"\xff\xd9"
    return bytes(out)


def pillow_jpeg(img, q):
    b = io.BytesIO()
    Image.fromarray(img).save(b, format="JPEG", quality=q, subsampling=2, restart_marker_rows=1)
    return b.getvalue()


def frames_of(H, W, seed=0):
    """Noise, gradients and a synthetic.make_video frame of one size."""
    from deepgraphpose_b200 import synthetic
    rng = np.random.default_rng(seed + H * 7 + W)
    yy, xx = np.mgrid[0:H, 0:W]
    video = synthetic.make_video(1, H, W, 4, seed=seed)[0][0]
    return {"noise": rng.integers(0, 256, (H, W, 3), dtype=np.uint8),
            "gradient": np.stack([(xx * 3 + yy) % 256, (yy * 2) % 256, (xx * yy) % 256], -1).astype(np.uint8),
            "video": np.ascontiguousarray(video)}


@pytest.mark.parametrize("q", QUALITIES)
@pytest.mark.parametrize("H,W", SIZES)
def test_reference_equals_pillow(H, W, q):
    for name, img in frames_of(H, W).items():
        ref, pil = encode_reference(img, q), pillow_jpeg(img, q)
        assert ref == pil, (name, len(ref), len(pil))


def test_capacity_bounds_pillow(lib_built):
    """dgp_jpeg_capacity: header + per MCU row 2 x (6 x 216 x MCUs + 1) + RSTn, + EOI, and it holds noise at q 100."""
    from deepgraphpose_b200.engine import jpeg_capacity
    for H, W in SIZES + [(16383, 16383), (1080, 1920)]:
        mcux, mcuy = -(-W // 16), -(-H // 16)
        assert jpeg_capacity(H, W) == 629 + mcuy * (2 * (6 * 216 * mcux + 1) + 2) + 2
    for H, W in SIZES:
        img = frames_of(H, W)["noise"]
        assert len(pillow_jpeg(img, 100)) <= jpeg_capacity(H, W)
    for bad in ((0, 5), (5, 0), (16384, 5), (5, 16384)):
        with pytest.raises(ValueError):
            jpeg_capacity(*bad)


def ffmpeg_still(packet, path):
    """FFmpeg's decode of one JPEG file, through the same OpenCV backend that reads the movie."""
    import cv2
    path.write_bytes(packet)
    cap = cv2.VideoCapture(str(path), cv2.CAP_FFMPEG)
    ok, fr = cap.read()
    cap.release()
    assert ok
    return fr


@pytest.mark.parametrize("fps", [30.0, 29.97])
def test_mp4_muxer_round_trip(tmp_path, fps):
    """N Pillow packets -> the muxer -> cv2.VideoCapture: N frames at fps, MJPG, each frame FFmpeg's decode of its packet.
    (FFmpeg's MJPEG decoder upsamples chroma unlike libjpeg, so frames differ from cv2.imdecode by a few levels; the
    comparison with imdecode is a bound, the one with the still decode is exact.)"""
    import cv2
    from deepgraphpose_b200 import synthetic
    from deepgraphpose_b200.mp4 import MJPEGWriter
    N, H, W = 9, 61, 83
    frames = synthetic.make_video(N, H, W, 4, seed=5)[0]
    packets = [pillow_jpeg(np.ascontiguousarray(f), 90) for f in frames]
    path = tmp_path / "m.mp4"
    with MJPEGWriter(str(path), fps, W, H) as w:
        for p in packets[:4]:
            w.write(p)
        w.write_packed(np.frombuffer(b"".join(packets[4:]) + b"tail", np.uint8), np.array([len(p) for p in packets[4:]]))
    cap = cv2.VideoCapture(str(path))
    assert cap.isOpened()
    assert abs(cap.get(cv2.CAP_PROP_FPS) - fps) < 1e-6
    assert int(cap.get(cv2.CAP_PROP_FRAME_COUNT)) == N
    fourcc = int(cap.get(cv2.CAP_PROP_FOURCC))
    assert "".join(chr((fourcc >> (8 * i)) & 0xFF) for i in range(4)).upper() == "MJPG"
    got = []
    while True:
        ok, fr = cap.read()
        if not ok:
            break
        got.append(fr)
    cap.release()
    assert len(got) == N
    for k, (fr, p) in enumerate(zip(got, packets)):
        assert np.array_equal(fr, ffmpeg_still(p, tmp_path / ("%d.jpg" % k)))
        ref = cv2.imdecode(np.frombuffer(p, np.uint8), cv2.IMREAD_COLOR)
        assert np.abs(fr.astype(int) - ref.astype(int)).mean() < 3.0


def test_arguments_checked_before_any_engine(tmp_path, monkeypatch):
    from deepgraphpose_b200 import eval as E

    def no_engine(*a, **k):
        raise AssertionError("an engine was created before the arguments were checked")

    monkeypatch.setattr(E, "Engine", no_engine)
    monkeypatch.setattr(E, "_setup_eval_graph", no_engine)
    video = str(tmp_path / "v.avi")
    cfg = {"num_joints": 2, "stride": 8.0}
    for kw in ({"encoder": "h264"}, {"encoder": "jpeg", "quality": 0}, {"encoder": "jpeg", "quality": 101},
               {"encoder": "jpeg", "quality": 90.0}, {"encoder": "jpeg", "quality": True}):
        with pytest.raises(ValueError):
            E.plot_dgp(video, output_dir=str(tmp_path), proj_cfg_file=cfg, dgp_model_file={}, **kw)
        with pytest.raises(ValueError):
            E.create_annotated_movie(np.zeros((2, 8, 8, 3), np.uint8), np.zeros((2, 2)), np.zeros((2, 2)), fps=30.0,
                                     filename=str(tmp_path / "m.mp4"), **kw)
    assert not any(p.suffix == ".mp4" for p in tmp_path.iterdir())
