"""Exif header, user Exif tags and orientation metadata (SURVEY section 8f rank 4: "Exif/SPIFF headers + orientation
metadata").  CPU tests of the host writer / reader (tests/_shims.py host_shim) against the reference's own writer and
Exif code compiled in place (oracle/_ref/libgpujpeg_refcpu.so: gpujpeg_writer.c + gpujpeg_exif.c), whose answers are recorded
in tests/golden/ref_exif_metadata.json."""
import ctypes as C
import itertools

import numpy as np
import pytest

import _oracle as o
from _refstore import digest, want
from _shims import hs

HDR_DEFAULT, HDR_JFIF, HDR_SPIFF, HDR_ADOBE, HDR_EXIF = 0, 1, 2, 4, 8
CS_RGB, CS_601, CS_601_256, CS_709 = 1, 2, 3, 4

hs.shim_add_exif_tag.argtypes = [C.c_char_p]
hs.shim_parse_meta.argtypes = [np.ctypeslib.ndpointer(np.uint8), C.c_size_t, np.ctypeslib.ndpointer(np.int32)]


def _recorded(request, live):
    return want("exif_metadata", request.node.name, live)


def _mine(w, h, header_type, orientation=None, tags=(), internal=CS_601_256, comps=3):
    hs.shim_set_header_type(header_type)
    hs.shim_set_orientation(*((1,) + orientation if orientation else (0, 0, 0)))
    hs.shim_clear_exif_tags()
    rc = [hs.shim_add_exif_tag(t.encode()) for t in tags]
    out = np.zeros(70000, np.uint8)
    n = hs.shim_header2(w, h, 75, 4, 0, comps, 1, 1, internal, out)
    hs.shim_set_header_type(0)
    hs.shim_set_orientation(0, 0, 0)
    hs.shim_clear_exif_tags()
    return out[:n].copy(), rc


def _ref(w, h, header_type, orientation=None, tags=(), internal=CS_601_256, comps=3):
    """the reference writer's file for an all-zero image; its first bytes are header + first SOS"""
    o.ref.ref_add_exif_tag.argtypes = [C.c_char_p]
    o.ref.ref_set_header_type(header_type)
    o.ref.ref_set_orientation(*((1,) + orientation if orientation else (0, 0, 0)))
    o.ref.ref_clear_exif_tags()
    rc = [o.ref.ref_add_exif_tag(t.encode()) for t in tags]
    bx, by = (w + 7) // 8, (h + 7) // 8
    coef = np.zeros(comps * bx * by * 64, np.int16)
    out = np.zeros(70000 + coef.size, np.uint8)
    if internal == CS_601_256:
        n = o.ref.ref_encode_from_coef_ss(coef, w, h, comps, 75, 4, 0, 1, 1, out, out.size)
    elif internal == CS_RGB:
        n = o.ref.ref_encode_from_coef_rgb(coef, w, h, 75, 4, 0, 1, 1, out, out.size)
    else:
        n = o.ref.ref_encode_from_coef_cs(coef, w, h, 75, 4, 0, 1, 1, internal, out, out.size)
    o.ref.ref_set_header_type(0)
    o.ref.ref_set_orientation(0, 0, 0)
    o.ref.ref_clear_exif_tags()
    assert n > 0
    return out[:n].copy(), rc


def _mask_datetime(a):
    """blank the 19 characters of a DateTime value ("YYYY:MM:DD HH:MM:SS"): the two writers run a moment apart"""
    b = a.copy()
    s = bytes(a)
    i = 0
    while True:
        i = s.find(b":", i)
        if i < 0 or i + 16 > len(s):
            return b
        if s[i + 3:i + 4] == b":" and s[i + 6:i + 7] == b" " and s[i + 9:i + 10] == b":" and s[i + 12:i + 13] == b":" and i >= 4:
            b[i - 4:i + 15] = 0
            return b
        i += 1


def _parse(buf):
    out = np.zeros(5, np.int32)
    full = np.concatenate([buf, np.array([0xFF, 0xD9], np.uint8)])
    assert hs.shim_parse_meta(full, full.size, out) == 0
    return tuple(int(v) for v in out)


ORIENTATIONS = [(r, f) for r in range(4) for f in range(2)]


@pytest.mark.parametrize("orientation", [None] + ORIENTATIONS)
def test_exif_header_bytes(request, orientation):
    """enc_hdr=Exif, with and without enc_metadata=orientation: bytes of the reference writer (DateTime blanked)"""
    w, h = 70, 50
    mine, _ = _mine(w, h, HDR_EXIF, orientation)
    app1 = bytes(mine).find(b"\xff\xe1")
    seg = np.frombuffer(bytes(mine[app1 + 2:]), np.uint8).copy()

    def live():
        theirs, _ = _ref(w, h, HDR_EXIF, orientation)
        o.ref.ref_exif_parse.argtypes = [np.ctypeslib.ndpointer(np.uint8), C.c_size_t]
        return [digest(_mask_datetime(theirs[:mine.size])), o.ref.ref_exif_parse(seg, seg.size)]
    theirs, got = _recorded(request, live)
    assert mine.size > 400 and digest(_mask_datetime(mine)) == theirs
    assert not np.array_equal(mine, _mask_datetime(mine))          # (there was a DateTime to blank)
    # and the reader finds the header type and the orientation again
    ht, oset, rot, flip, cs = _parse(mine)
    assert ht == HDR_EXIF and cs == CS_601_256
    assert (oset, rot, flip) == ((1,) + orientation if orientation else (1, 0, 0))   # Exif always carries an Orientation tag
    assert (got & 1, got >> 8, (got >> 4) & 1) == (oset, rot, flip)   # the reference's parser on the product's segment


TAG_SETS = [
    ("DateTime=2024:02:29 12:34:56",),
    ("DateTime=2024:02:29 12:34:56", "Orientation=6"),
    ("DateTime=2024:02:29 12:34:56", "Sofware=a codec with a long name", "XResolution=300/1", "YResolution=300/2"),
    ("DateTime=2024:02:29 12:34:56", "0x10F:ASCII=maker", "0x110:ascii=x", "0x9286:UNDEFINED=user comment bytes"),
    ("DateTime=2024:02:29 12:34:56", "WhitePoint=3127/10000,3290/10000", "0x829A:RATIONAL=1/250", "0x8827:SHORT=100,200,300"),
    ("DateTime=2024:02:29 12:34:56", "PixelXDimension=1234"),                                    # replaces a default of the Exif IFD
    ("DateTime=2024:02:29 12:34:56", "PixelYDimension=7", "ColorSpace=65535", "ExifVersion=0232"),
    ("DateTime=2024:02:29 12:34:56", "ColorSpace=2", "PixelYDimension=7"),
    ("DateTime=2024:02:29 12:34:56", "0x9204:SRATIONAL=-1/3", "0x9201:SLONG=-5", "0xA401:SHORT=1", "0x100:LONG=1,2", "0x101:BYTE=1,2,3,4,5"),
    ("DateTime=2024:02:29 12:34:56", "0x8769:LONG=8"),                                            # even the IFD pointer
    ("DateTime=2024:02:29 12:34:56", "0x131:ASCII=" + "x" * 3000, "0x9286:UNDEFINED=" + "y" * 5000),
    ("DateTime=2024:02:29 12:34:56", "Orientation="),                                            # (an empty UNDEFINED value aborts the reference)
    ("DateTime=2024:02:29 12:34:56", "0x112:SHORT=3", "0x112:SHORT=8"),
]


@pytest.mark.parametrize("tags", TAG_SETS)
def test_exif_user_tags_bytes(request, tags):
    """enc_exif_tag: every way of writing a tag (by name, by number and type, lists, rationals, strings), tags that replace
    defaults, long values -- byte-identical to the reference writer (a user DateTime fixes the clock)"""
    w, h = 1920, 1080
    mine, rc_mine = _mine(w, h, HDR_EXIF, (1, 0), tags)

    def live():
        theirs, rc = _ref(w, h, HDR_EXIF, (1, 0), tags)
        return [rc, digest(theirs[:mine.size])]
    rc_want, theirs = _recorded(request, live)
    assert rc_mine == rc_want == [0] * len(tags)
    assert digest(mine) == theirs


@pytest.mark.parametrize("bad", ["Nonsense=1", "0x112=3", "0x112:FLOAT=3", "0x112:SHORT", "Orientation=1x", "XResolution=1/2,", "help",
                                 "Orientation"])
def test_exif_tag_syntax_errors(request, bad):
    hs.shim_clear_exif_tags()
    mine = hs.shim_add_exif_tag(bad.encode())
    hs.shim_clear_exif_tags()

    def live():   # (after a trailing comma the reference reads one byte past the terminator: a second NUL there)
        o.ref.ref_clear_exif_tags()
        rc = o.ref.ref_add_exif_tag(C.create_string_buffer(bad.encode(), len(bad) + 2))
        o.ref.ref_clear_exif_tags()
        return rc
    want = _recorded(request, live)
    if bad == "XResolution=1/2,":
        assert mine == want == 0          # a trailing comma reads one more (empty) rational in the reference; same here
    else:
        assert mine != 0 and want != 0


@pytest.mark.parametrize("internal,header_type", [(CS_601_256, HDR_DEFAULT), (CS_601_256, HDR_SPIFF), (CS_709, HDR_DEFAULT),
                                                  (CS_RGB, HDR_DEFAULT), (CS_601_256, HDR_JFIF)])
@pytest.mark.parametrize("orientation", [(0, 0), (1, 0), (2, 1), (3, 1)])
def test_orientation_in_spiff_directory(request, internal, header_type, orientation):
    """an orientation makes the default header SPIFF (whatever the colour space) and goes into its directory; JFIF has no
    place for it"""
    w, h = 70, 50
    mine, _ = _mine(w, h, header_type, orientation, internal=internal)
    assert digest(mine) == _recorded(request, lambda: digest(_ref(w, h, header_type, orientation, internal=internal)[0][:mine.size]))
    ht, oset, rot, flip, cs = _parse(mine)
    if header_type == HDR_JFIF:
        assert (ht, oset) == (HDR_JFIF, 0)
    else:
        assert (ht, oset, rot, flip, cs) == (HDR_SPIFF, 1) + orientation + (internal,)


def test_exif_reader_on_foreign_headers():
    """little-endian Exif (what cameras write), orientation as the only tag; broken headers leave the metadata alone"""
    base, _ = _mine(64, 48, HDR_JFIF)

    def with_app1(payload):
        n = len(payload) + 2
        return np.frombuffer(bytes(base[:20]) + b"\xff\xe1" + bytes([n >> 8, n & 255]) + payload + bytes(base[20:]), np.uint8)   # behind APP0

    def tiff(le, entries, offset=8):
        e16 = (lambda v: bytes([v & 255, v >> 8])) if le else (lambda v: bytes([v >> 8, v & 255]))
        e32 = (lambda v: e16(v & 0xFFFF) + e16(v >> 16)) if le else (lambda v: e16(v >> 16) + e16(v & 0xFFFF))
        body = (b"II" if le else b"MM") + e16(42) + e32(offset) + bytes(offset - 8) + e16(len(entries))
        for tag, typ, count, val in entries:
            v = e16(val) + bytes(2) if typ == 3 else e32(val)
            body += e16(tag) + e16(typ) + e32(count) + v
        return b"Exif\0\0" + body + e32(0)

    for le, val in itertools.product((0, 1), range(1, 9)):
        ht, oset, rot, flip, _ = _parse(with_app1(tiff(le, [(0x10F, 2, 4, 26), (0x112, 3, 1, val), (0x128, 3, 1, 2)], offset=8 + 4 * le)))
        want = [(0, 0), (0, 1), (2, 0), (2, 1), (1, 1), (1, 0), (3, 1), (3, 0)][val - 1]
        assert (ht, oset, rot, flip) == (HDR_EXIF, 1) + want, (le, val)
    for payload in (tiff(0, [(0x112, 3, 1, 9)]), tiff(1, [(0x112, 3, 1, 0)]), b"Exif\0\0XX" + bytes(20), b"Exif\0\0MM\0\x2b" + bytes(20),
                    b"Exif\0\0MM\0\x2a\0\x01\0\0" + bytes(8), tiff(0, [])[:-4] + b"\xff\xff" + bytes(2)):
        ht, oset, _, _, _ = _parse(with_app1(payload))
        assert (ht, oset) == (HDR_EXIF, 0)
    ht, oset, _, _, _ = _parse(with_app1(b"http://ns.adobe.com/xap/1.0/\0<x/>"))     # XMP: skipped
    assert (ht, oset) == (HDR_JFIF, 0)
    assert bytes(base[2:4]) == b"\xff\xe0" and bytes(base[20:22]) == b"\xff\xdb"
