"""Image file helpers of the public API (SURVEY section 8f rank 4: "image file I/O helpers"): PGM / PPM / PNM / PAM and Y4M.
CPU tests: the product's gj_common.c + gj_imageio.c run over host stand-ins for CUDA (tests/_shims.py io_shim) and are held
against the reference's own pam.c / y4m.c compiled in place (oracle/_ref/libgpujpeg_refcpu.so; its answers recorded in
tests/golden/ref_image_io.json) and against the rules of its delegates (src/utils/image_delegate.c:149-340)."""
import ctypes as C
import os

import numpy as np
import pytest

import _oracle as o
from _refstore import digest, want
from _shims import io

U8, P012, P0P1P2_444, P1020, P0P1P2_422, P0P1P2_420, P0123 = range(7)
RGB, BT601, BT601_256, BT709 = 1, 2, 3, 4
PIXFMT_AUTODETECT, PIXFMT_NO_ALPHA, PIXFMT_STD, CS_DEFAULT = -2, -3, -4, -1


class ImageParameters(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("color_space", C.c_int), ("pixel_format", C.c_int),
                ("width_padding", C.c_int)]


io.gpujpeg_image_save_to_file.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(ImageParameters)]
io.gpujpeg_image_load_from_file.argtypes = [C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
io.gpujpeg_image_get_properties.argtypes = [C.c_char_p, C.POINTER(ImageParameters), C.c_int]
io.gpujpeg_image_destroy.argtypes = [C.c_void_p]
io.gpujpeg_image_calculate_size.argtypes = [C.POINTER(ImageParameters)]
io.gpujpeg_image_calculate_size.restype = C.c_size_t


class PamMeta(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("ch_count", C.c_int), ("maxval", C.c_int), ("bitmap_pbm", C.c_bool)]


class Y4mMeta(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("bitdepth", C.c_int), ("subsampling", C.c_int), ("limited", C.c_bool)]


_libc = C.CDLL(None)
_ALLOC = C.CFUNCTYPE(C.c_void_p, C.c_size_t)
_malloc = _ALLOC(lambda n: _libc_malloc(n))
_libc.malloc.restype = C.c_void_p
_libc.malloc.argtypes = [C.c_size_t]
_libc.free.argtypes = [C.c_void_p]


def _libc_malloc(n):
    return _libc.malloc(n)


def _ref():
    """the reference's pam.c / y4m.c (only called while recording their answers)"""
    o.ref.pam_read.argtypes = [C.c_char_p, C.POINTER(PamMeta), C.POINTER(C.c_void_p), _ALLOC]
    o.ref.pam_read.restype = C.c_bool
    o.ref.pam_write.argtypes = [C.c_char_p, C.c_uint, C.c_uint, C.c_uint, C.c_int, C.c_int, C.c_void_p, C.c_bool]
    o.ref.pam_write.restype = C.c_bool
    o.ref.y4m_read.argtypes = [C.c_char_p, C.POINTER(Y4mMeta), C.POINTER(C.c_void_p), _ALLOC]
    o.ref.y4m_read.restype = C.c_size_t
    o.ref.y4m_write.argtypes = [C.c_char_p, C.POINTER(Y4mMeta), C.c_void_p]
    o.ref.y4m_write.restype = C.c_bool
    return o.ref


def _recorded(request, live):
    return want("image_io", request.node.name, live)


def _size(w, h, fmt):
    p = ImageParameters(w, h, RGB, fmt, 0)
    return io.gpujpeg_image_calculate_size(C.byref(p))


def _save(path, data, w, h, fmt, cs):
    p = ImageParameters(w, h, cs, fmt, 0)
    name = C.create_string_buffer(str(path).encode())   # mutable: ".XXX" is rewritten in place
    rc = io.gpujpeg_image_save_to_file(name, data.ctypes.data, data.size, C.byref(p))
    return rc, name.value.decode()


def _load(path):
    ptr, size = C.c_void_p(), C.c_size_t(0)
    rc = io.gpujpeg_image_load_from_file(str(path).encode(), C.byref(ptr), C.byref(size))
    if rc != 0:
        return rc, None
    out = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), (size.value,)).copy()
    io.gpujpeg_image_destroy(ptr)
    return 0, out


def _props(path, exists=1):
    p = ImageParameters(0, 0, 0, -1, 0)
    rc = io.gpujpeg_image_get_properties(str(path).encode(), C.byref(p), exists)
    return rc, p


def _rand(n, seed=1):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)


# ---- Netpbm ----
@pytest.mark.parametrize("ext,fmt,cs,depth,head", [
    ("pgm", U8, BT601_256, 1, b"P5\n37 21\n255\n"),
    ("pnm", U8, BT601_256, 1, b"P5\n37 21\n255\n"),
    ("ppm", P012, RGB, 3, b"P6\n37 21\n255\n"),
    ("pnm", P012, RGB, 3, b"P6\n37 21\n255\n"),
    ("pam", U8, BT601_256, 1, b"P7\nWIDTH 37\nHEIGHT 21\nDEPTH 1\nMAXVAL 255\nTUPLTYPE GRAYSCALE\nENDHDR\n"),
    ("pam", P012, RGB, 3, b"P7\nWIDTH 37\nHEIGHT 21\nDEPTH 3\nMAXVAL 255\nTUPLTYPE RGB\nENDHDR\n"),
    ("pam", P0123, RGB, 4, b"P7\nWIDTH 37\nHEIGHT 21\nDEPTH 4\nMAXVAL 255\nTUPLTYPE RGB_ALPHA\nENDHDR\n"),
])
def test_netpbm_save_load(request, tmp_path, ext, fmt, cs, depth, head):
    w, h = 37, 21
    data = _rand(w * h * depth)
    path = tmp_path / ("img." + ext)
    rc, _ = _save(path, data, w, h, fmt, cs)
    assert rc == 0
    raw = path.read_bytes()
    assert raw == head + data.tobytes()                      # the reference's header text, then the samples
    rc, back = _load(path)
    assert rc == 0 and np.array_equal(back, data)
    rc, p = _props(path)
    assert rc == 0 and (p.width, p.height, p.pixel_format) == (w, h, fmt)
    assert p.color_space == (BT601_256 if depth == 1 else RGB)

    def live():
        ref, ref_path = _ref(), tmp_path / ("ref." + ext)
        assert ref.pam_write(str(ref_path).encode(), w, w, h, depth, 255, data.ctypes.data, ext != "pam")
        m, ptr = PamMeta(), C.c_void_p()
        assert ref.pam_read(str(path).encode(), C.byref(m), C.byref(ptr), _malloc)
        got = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), (data.size,)).copy()
        _libc.free(ptr)
        return [digest(np.frombuffer(ref_path.read_bytes(), np.uint8)), [m.width, m.height, m.ch_count, m.maxval], digest(got)]
    ref_file, meta, got = _recorded(request, live)
    assert digest(np.frombuffer(raw, np.uint8)) == ref_file              # byte-identical files
    assert meta == [w, h, depth, 255] and got == digest(data)           # the reference reads the product's file


def test_netpbm_headers_with_comments(request, tmp_path):
    data = _rand(5 * 4 * 3)
    p = tmp_path / "c.ppm"
    p.write_bytes(b"P6\n# made by hand\n5 # width\n 4\n#\n255\n" + data.tobytes())
    rc, back = _load(p)
    assert rc == 0 and np.array_equal(back, data)
    rc, pr = _props(p)
    assert rc == 0 and (pr.width, pr.height, pr.pixel_format, pr.color_space) == (5, 4, P012, RGB)
    q = tmp_path / "c.pam"
    q.write_bytes(b"P7\n# comment\nHEIGHT 4\nWIDTH 5\nMAXVAL 255\nDEPTH 4\nTUPLTYPE RGB_ALPHA\nENDHDR\n" + _rand(80).tobytes())
    rc, pr = _props(q)
    assert rc == 0 and (pr.width, pr.height, pr.pixel_format) == (5, 4, P0123)
    rc, back = _load(q)
    assert rc == 0 and back.size == 80

    def live():
        metas = []
        for f in (p, q):
            m = PamMeta()
            metas.append([bool(_ref().pam_read(str(f).encode(), C.byref(m), None, _ALLOC(0))), m.width, m.height, m.ch_count, m.maxval])
        return metas
    assert _recorded(request, live) == [[True, 5, 4, 3, 255], [True, 5, 4, 4, 255]]


@pytest.mark.parametrize("content,why", [
    (b"P3\n2 2\n255\n1 2 3 4 5 6 7 8 9 10 11 12\n", "plain PNM"),
    (b"P4\n8 1\n\xff", "bitmap"),
    (b"P6\n2 2\n65535\n" + bytes(24), "16-bit samples"),
    (b"P6\n2 2\n255 " + bytes(12), "no newline after maxval"),
    (b"P6\n2 2\n", "header ends early"),
    (b"P7\nWIDTH 2\nHEIGHT 2\nMAXVAL 255\nENDHDR\n" + bytes(12), "PAM without DEPTH"),
    (b"P6\n2 2\n255\n" + bytes(5), "samples missing"),
    (b"GIF89a", "not Netpbm"),
    (b"P7\nWIDTH 2147483647\nHEIGHT 2147483647\nDEPTH 2147483647\nMAXVAL 255\nENDHDR\n" + bytes(64), "sizes whose product wraps"),
    (b"P6\n70000 2\n255\n" + bytes(64), "wider than a JPEG can be"),
])
def test_netpbm_refused(request, tmp_path, content, why):
    p = tmp_path / "bad.pnm"
    p.write_bytes(content)
    rc, _ = _load(p)
    assert rc != 0, why
    if why != "samples missing":
        rc, _ = _props(p)
        assert rc < 0, why
    if why not in ("16-bit samples", "bitmap", "sizes whose product wraps", "wider than a JPEG can be"):   # (pam.c reads those; the delegates then refuse everything but 255 levels)
        m, ptr = PamMeta(), C.c_void_p()
        assert not _recorded(request, lambda: bool(_ref().pam_read(str(p).encode(), C.byref(m), C.byref(ptr), _malloc))), why


def test_netpbm_save_rules(tmp_path):
    w, h = 8, 8
    # PNM cannot hold four channels; PAM / PNM want RGB unless grey; subsampled formats are refused
    assert _save(tmp_path / "a.pnm", _rand(w * h * 4), w, h, P0123, RGB)[0] != 0
    assert _save(tmp_path / "b.pam", _rand(w * h * 3), w, h, P012, BT601_256)[0] != 0
    assert _save(tmp_path / "c.pam", _rand(w * h * 2), w, h, P1020, RGB)[0] != 0
    assert _save(tmp_path / "d.pam", _rand(w * h), w, h, U8, BT709)[0] == 0      # grey: any colour space


# ---- Y4M ----
@pytest.mark.parametrize("fmt,cs,chroma,rng,ss", [
    (U8, BT601_256, "mono", "FULL", 400), (P0P1P2_420, BT601_256, "420", "FULL", 420), (P0P1P2_422, BT601, "422", "LIMITED", 422),
    (P0P1P2_444, BT709, "444", "LIMITED", 444), (P0P1P2_420, BT601, "420", "LIMITED", 420),
])
@pytest.mark.parametrize("w,h", [(32, 16), (37, 21)])
def test_y4m_save_load(request, tmp_path, fmt, cs, chroma, rng, ss, w, h):
    n = _size(w, h, fmt)
    data = _rand(n)
    path = tmp_path / "f.y4m"
    assert _save(path, data, w, h, fmt, cs)[0] == 0
    raw = path.read_bytes()
    head = ("YUV4MPEG2 W%d H%d F25:1 Ip A0:0 C%s XCOLORRANGE=%s\nFRAME\n" % (w, h, chroma, rng)).encode()
    assert raw == head + data.tobytes()
    rc, back = _load(path)
    assert rc == 0 and np.array_equal(back, data)
    rc, p = _props(path)
    assert rc == 0 and (p.width, p.height, p.pixel_format) == (w, h, fmt)
    assert p.color_space == (BT601 if rng == "LIMITED" else BT601_256)

    def live():
        ref, ref_path = _ref(), tmp_path / "ref.y4m"
        m = Y4mMeta(w, h, 8, ss, rng == "LIMITED")
        assert ref.y4m_write(str(ref_path).encode(), C.byref(m), data.ctypes.data)
        m2, ptr = Y4mMeta(), C.c_void_p()
        size = ref.y4m_read(str(path).encode(), C.byref(m2), C.byref(ptr), _malloc)
        _libc.free(ptr)
        return [digest(np.frombuffer(ref_path.read_bytes(), np.uint8)), size, [m2.width, m2.height, m2.bitdepth, m2.subsampling, m2.limited]]
    ref_file, size, meta = _recorded(request, live)
    assert digest(np.frombuffer(raw, np.uint8)) == ref_file
    assert size == n and meta == [w, h, 8, ss, rng == "LIMITED"]


def test_y4m_foreign_headers(request, tmp_path):
    w, h = 6, 4
    n420 = w * h + 2 * 3 * 2
    p = tmp_path / "ff.y4m"
    p.write_bytes(b"YUV4MPEG2 W6 H4 F30000:1001 Ip A1:1 C420jpeg XYSCSS=420JPEG\nFRAME\n" + _rand(n420).tobytes())
    rc, pr = _props(p)
    assert rc == 0 and (pr.width, pr.height, pr.pixel_format, pr.color_space) == (w, h, P0P1P2_420, BT601_256)
    rc, back = _load(p)
    assert rc == 0 and back.size == n420
    ref_reads = {}
    for head, why in ((b"YUV4MPEG2 W6 H4 C420p10\nFRAME\n", "10 bits"), (b"YUV4MPEG2 W6 H4 C444alpha\nFRAME\n", "alpha"),
                      (b"YUV4MPEG2 W6 H4\nFRAME\n", "no chroma tag: the reference does not assume 4:2:0"),
                      (b"YUV4MPEG2 W6 H4 C420\nFRAME \n", "FRAME with parameters"), (b"YUV4MPEG W6 H4 C420\nFRAME\n", "magic"),
                      (b"YUV4MPEG2 W2147483647 H2147483647 C444\nFRAME\n", "sizes whose product wraps"), (b"YUV4MPEG2 W0 H4 C444\nFRAME\n", "no width")):
        q = tmp_path / "bad.y4m"
        q.write_bytes(head + bytes(200))
        assert _props(q)[0] < 0, why
        if why in ("no chroma tag: the reference does not assume 4:2:0", "FRAME with parameters", "magic"):
            ref_reads[why] = q.read_bytes()

    def live():
        m, sizes = Y4mMeta(), {}
        for why, content in ref_reads.items():
            q.write_bytes(content)
            sizes[why] = _ref().y4m_read(str(q).encode(), C.byref(m), None, _ALLOC(0))
        return sizes
    sizes = _recorded(request, live)
    assert sorted(sizes) == sorted(ref_reads) and not any(sizes.values()), sizes
    assert _save(tmp_path / "x.y4m", _rand(w * h * 3), w, h, P012, BT601_256)[0] != 0     # packed format
    assert _save(tmp_path / "y.y4m", _rand(w * h * 3), w, h, P0P1P2_444, RGB)[0] != 0     # RGB


# ---- names ----
def test_properties_of_names():
    """what a file name alone says (file_exists = 0) [ref: src/utils/image_delegate.c:149-168, 257-262;
    src/gpujpeg_common.c:1321-1371]"""
    want = {"a.pgm": (1, U8, BT601_256), "a.ppm": (1, P012, CS_DEFAULT), "a.pnm": (1, PIXFMT_NO_ALPHA, CS_DEFAULT),
            "a.pam": (1, PIXFMT_AUTODETECT, CS_DEFAULT), "a.y4m": (0, PIXFMT_STD, BT601_256), "a.rgb": (1, P012, RGB),
            "a.rgba": (1, P0123, RGB), "a.yuv": (1, P012, BT601_256), "a.yuva": (1, P0123, BT601_256),
            "a.uyvy": (1, P1020, BT601_256), "a.i420": (1, P0P1P2_420, BT601_256), "a.r": (1, U8, BT601_256),
            "a.raw": (1, PIXFMT_STD, 0)}
    for name, (rc_want, fmt, cs) in want.items():
        rc, p = _props(name, 0)
        assert (rc, p.pixel_format, p.color_space) == (rc_want, fmt, cs), name
    assert _props("a.jpg", 0)[0] < 0 and _props("noext", 0)[0] < 0 and _props("a.png", 0)[0] < 0


def test_placeholder_extension(tmp_path):
    """"name.XXX" gets the extension that can hold the image [ref: src/gpujpeg_common.c:1258-1275]"""
    w, h = 8, 2
    for fmt, cs, ext in ((P012, RGB, "pnm"), (U8, BT601_256, "pnm"), (P0123, RGB, "pam"), (P0P1P2_444, BT601_256, "y4m")):
        rc, name = _save(tmp_path / "out.XXX", _rand(_size(w, h, fmt)), w, h, fmt, cs)
        assert rc == 0 and name.endswith("out." + ext) and os.path.exists(name)
        os.remove(name)


def test_raw_dump_and_tst(tmp_path):
    data = _rand(300)
    p = tmp_path / "x.rgb"
    assert _save(p, data, 10, 10, P012, RGB)[0] == 0 and p.read_bytes() == data.tobytes()
    rc, back = _load(p)
    assert rc == 0 and np.array_equal(back, data)
    rc, img = _load("16x8.p_u8.blank_7.tst")
    assert rc == 0 and img.size == 128 and (img == 7).all()
