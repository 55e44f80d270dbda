"""A minimal ISO-BMFF (.mp4) muxer for Motion-JPEG: one video track whose samples are complete JPEG files.

The layout is the one FFmpeg writes when OpenCV is asked for MJPG in an ``.mp4``: an ``mp4v`` sample entry whose ``esds``
names object type 0x6C (JPEG), one ``stts`` run at a constant rate, ``stsz`` with every packet's size and a ``co64`` chunk
offset into an ``mdat`` with a 64-bit size.  Packets are appended as they come (only their sizes stay in memory); the
``moov`` box is written by ``close()``.  FFmpeg / OpenCV read such a file back as MJPG at the given rate."""
import struct
from fractions import Fraction


def _box(kind, *parts):
    body = b"".join(parts)
    return struct.pack(">I4s", 8 + len(body), kind) + body


def _full_box(kind, version, flags, *parts):
    return _box(kind, struct.pack(">I", (version << 24) | flags), *parts)


_MATRIX = struct.pack(">9I", 0x10000, 0, 0, 0, 0x10000, 0, 0, 0, 0x40000000)


def _timebase(fps):
    """(timescale, ticks per frame) of a frame rate: the rate as a fraction (denominator at most 1001, so 29.97 and
    30000/1001 stay exact), doubled up to a timescale of at least 10000 as FFmpeg's muxer does."""
    fr = Fraction(fps).limit_denominator(1001)
    if fr <= 0:
        raise ValueError("fps must be positive, got %r" % (fps,))
    scale, delta = fr.numerator, fr.denominator
    while scale < 10000:
        scale, delta = 2 * scale, 2 * delta
    return scale, delta


def _esds():
    dec_config = bytes([0x6C, 0x11]) + b"\x00\x00\x00" + struct.pack(">II", 0, 0)  # JPEG, visual stream
    dec_specific_sl = bytes([0x06, 0x80, 0x80, 0x80, 0x01, 0x02])
    dcd = bytes([0x04, 0x80, 0x80, 0x80, len(dec_config)]) + dec_config
    es = struct.pack(">HB", 1, 0) + dcd + dec_specific_sl
    return _full_box(b"esds", 0, 0, bytes([0x03, 0x80, 0x80, 0x80, len(es)]) + es)


class MJPEGWriter:
    """``MJPEGWriter(path, fps, width, height)``; ``write(packet)`` appends one JPEG file (bytes-like), ``close()`` writes
    the index.  Also a context manager."""

    def __init__(self, path, fps, width, height):
        self.timescale, self.delta = _timebase(fps)
        self.width, self.height = int(width), int(height)
        if not (0 < self.width < 65536 and 0 < self.height < 65536):
            raise ValueError("frame size %dx%d outside 1..65535" % (self.width, self.height))
        self.sizes = []
        self.f = open(path, "wb")
        self.f.write(_box(b"ftyp", b"isom", struct.pack(">I", 0x200), b"isom", b"iso2", b"mp41"))
        self.mdat_at = self.f.tell()
        self.f.write(struct.pack(">I4sQ", 1, b"mdat", 0))  # 64-bit size, set by close()
        self.data_at = self.f.tell()

    def write(self, packet):
        mv = memoryview(packet).cast("B")
        if mv.nbytes >= 1 << 32:
            raise ValueError("a packet of %d bytes does not fit an stsz entry" % mv.nbytes)
        self.f.write(mv)
        self.sizes.append(mv.nbytes)

    def write_packed(self, data, sizes):
        """Appends len(sizes) packets stored back to back in ``data``."""
        mv = memoryview(data).cast("B")
        total = int(sum(int(s) for s in sizes))
        if total > mv.nbytes:
            raise ValueError("sizes add up to %d bytes, the buffer holds %d" % (total, mv.nbytes))
        self.f.write(mv[:total])
        self.sizes.extend(int(s) for s in sizes)

    def close(self):
        if self.f is None:
            return
        try:
            end = self.f.tell()
            self.f.seek(self.mdat_at + 8)
            self.f.write(struct.pack(">Q", end - self.mdat_at))
            self.f.seek(end)
            self.f.write(self._moov())
        finally:
            self.f.close()
            self.f = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _moov(self):
        n = len(self.sizes)
        media_duration = n * self.delta
        movie_duration = media_duration * 1000 // self.timescale  # mvhd / tkhd / elst in milliseconds
        mvhd = _full_box(b"mvhd", 0, 0, struct.pack(">IIII", 0, 0, 1000, movie_duration), struct.pack(">IH", 0x10000, 0x100),
                         b"\x00" * 10, _MATRIX, b"\x00" * 24, struct.pack(">I", 2))
        tkhd = _full_box(b"tkhd", 0, 3, struct.pack(">IIIII", 0, 0, 1, 0, movie_duration), b"\x00" * 8,
                         struct.pack(">HHHH", 0, 0, 0, 0), _MATRIX, struct.pack(">II", self.width << 16, self.height << 16))
        edts = _box(b"edts", _full_box(b"elst", 0, 0, struct.pack(">IIIHH", 1, movie_duration, 0, 1, 0)))
        mdhd = _full_box(b"mdhd", 0, 0, struct.pack(">IIII", 0, 0, self.timescale, media_duration), struct.pack(">HH", 0x55C4, 0))
        hdlr = _full_box(b"hdlr", 0, 0, b"\x00" * 4, b"vide", b"\x00" * 12, b"VideoHandler\x00")
        vmhd = _full_box(b"vmhd", 0, 1, b"\x00" * 8)
        dinf = _box(b"dinf", _full_box(b"dref", 0, 0, struct.pack(">I", 1), _full_box(b"url ", 0, 1)))
        entry = _box(b"mp4v", b"\x00" * 6, struct.pack(">H", 1), b"\x00" * 16, struct.pack(">HH", self.width, self.height),
                     struct.pack(">II", 0x480000, 0x480000), b"\x00" * 4, struct.pack(">H", 1), b"\x00" * 32,
                     struct.pack(">Hh", 0x18, -1), _esds())
        stsd = _full_box(b"stsd", 0, 0, struct.pack(">I", 1), entry)
        stts = _full_box(b"stts", 0, 0, struct.pack(">III", 1, n, self.delta) if n else struct.pack(">I", 0))
        stsc = _full_box(b"stsc", 0, 0, struct.pack(">IIII", 1, 1, n, 1) if n else struct.pack(">I", 0))
        stsz = _full_box(b"stsz", 0, 0, struct.pack(">II", 0, n), struct.pack(">%dI" % n, *self.sizes))
        co64 = _full_box(b"co64", 0, 0, struct.pack(">IQ", 1, self.data_at) if n else struct.pack(">I", 0))
        stbl = _box(b"stbl", stsd, stts, stsc, stsz, co64)
        minf = _box(b"minf", vmhd, dinf, stbl)
        mdia = _box(b"mdia", mdhd, hdlr, minf)
        trak = _box(b"trak", tkhd, edts, mdia)
        return _box(b"moov", mvhd, trak)
