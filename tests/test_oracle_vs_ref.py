"""Differential tests: oracle restatement vs the reference's own CPU sources compiled in place
(oracle/_ref/libgpujpeg_refcpu.so).  The reference's answers for these inputs are recorded in
tests/golden/ref_oracle_vs_ref.json (tests/_refstore.py), so the tests need no reference at run time.  CPU only."""
import numpy as np
import pytest

import _oracle as o
from _refcpu import ref_decode_coef, ref_encode_coef, ref_idct_planes
from _refstore import digest, want


def ref(request, live):
    return want("oracle_vs_ref", request.node.name, live)


@pytest.mark.parametrize("q", [1, 10, 25, 50, 75, 90, 95, 100])
def test_quant_tables(request, q):
    raw, fwd, inv = o.quant_tables(q)

    def live():
        r2, f2, i2 = np.zeros_like(raw), np.zeros_like(fwd), np.zeros_like(inv)
        assert o.ref.ref_quant_tables(q, r2, f2, i2) == 0
        return [digest(r2), digest(i2), digest(f2.view(np.uint32))]
    r2, i2, f2 = ref(request, live)
    assert digest(raw) == r2 and digest(inv) == i2
    assert digest(fwd.view(np.uint32)) == f2, "forward float table must be bit-identical"


@pytest.mark.parametrize("cls,kind", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_huffman_tables(request, cls, kind):
    code, size = np.zeros(256, np.uint16), np.zeros(256, np.uint8)
    o.lib.orc_huff_encoder_table(cls, kind, code, size)

    def live():
        c2, s2 = np.zeros(256, np.uint32), np.zeros(256, np.uint8)
        o.ref.ref_huff_encoder_table(cls, kind, c2, s2)
        return [digest(c2), digest(s2)]
    assert [digest(code.astype(np.uint32)), digest(size)] == ref(request, live)


CASES = [("random", 1920, 1080, 75, 24, 0), ("photo", 1920, 1080, 75, 24, 0), ("random", 1119, 561, 75, 8, 0),
         ("gradient", 640, 480, 75, 12, 0), ("zero", 256, 256, 75, 36, 0), ("random", 200, 120, 100, 36, 0),
         ("photo", 640, 360, 30, 7, 1), ("random", 64, 64, 75, 0, 0), ("photo", 16, 8, 75, 1, 0),
         ("random", 8, 8, 95, 24, 1)]


@pytest.mark.parametrize("kind,w,h,q,rst,il", CASES)
def test_encode_bytes_and_decode_coefficients(request, kind, w, h, q, rst, il):
    img = o.gen_image(kind, w, h)
    jpeg, coef = o.encode(img, q, rst, il, want_coef=True)
    ref_jpeg, ref_coef = ref(request, lambda: [digest(ref_encode_coef(coef, w, h, q, rst, il)),
                                               digest(ref_decode_coef(jpeg, w, h, rst, il))])
    assert digest(jpeg) == ref_jpeg, "oracle bytes != reference header writer + CPU Huffman encoder"
    assert digest(coef) == ref_coef, "reference CPU Huffman decoder must recover the encoder's coefficients"
    _, coef_dec = o.decode(jpeg, want_coef=True)
    assert np.array_equal(coef_dec, coef)


SS_CASES = [("photo", 640, 360, 75, 6), ("random", 1119, 561, 75, 8), ("random", 33, 17, 90, 2), ("photo", 16, 16, 75, 1),
            ("random", 100, 50, 60, 0), ("random", 8, 8, 95, 3)]


@pytest.mark.parametrize("il", [0, 1])
@pytest.mark.parametrize("sampling", [(2, 2), (2, 1), (1, 2)], ids=["420", "422", "440"])
@pytest.mark.parametrize("kind,w,h,q,rst", SS_CASES)
def test_subsampled_encode_bytes_and_decode_coefficients(request, kind, w, h, q, rst, sampling, il):
    """chroma subsampling: component geometry, MCU block order, per-component scans and SOF0 sampling factors of the
    oracle against the reference's header writer + CPU Huffman coder [ref: src/gpujpeg_huffman_cpu_encoder.c:234-290]"""
    img = o.gen_image(kind, w, h)
    jpeg, coef = o.encode(img, q, rst, il, want_coef=True, sampling=sampling)
    ref_jpeg, ref_coef = ref(request, lambda: [digest(ref_encode_coef(coef, w, h, q, rst, il, sampling=sampling)),
                                               digest(ref_decode_coef(jpeg, w, h, rst, il, sampling=sampling))])
    assert digest(jpeg) == ref_jpeg, "oracle bytes != reference header writer + CPU Huffman encoder"
    assert digest(coef) == ref_coef, "reference CPU Huffman decoder must recover the encoder's coefficients"
    out, coef_dec = o.decode(jpeg, want_coef=True)
    assert np.array_equal(coef_dec, coef) and out.shape == (h, w, 3)


@pytest.mark.parametrize("il,sampling", [(0, (1, 1)), (1, (1, 1)), (1, (2, 2))])
def test_rgb_internal_stream_bytes(request, il, sampling):
    """RGB-internal JPEG (no colour transform of RGB input): Adobe APP14 header, component ids 'R','G','B', one DQT and
    one DHT pair, luminance tables for all three components -- oracle bytes against the reference's header writer +
    CPU Huffman encoder fed with the same coefficients [ref: src/gpujpeg_writer.c:255-276, 462-470, 487-505]"""
    w, h, q, rst = 100, 60, 85, 5
    img = o.gen_image("photo", w, h)
    jpeg = o.encode_any(img, w, h, o.FMT_444_P012, o.CS_RGB, q, rst, il, sampling, internal=o.CS_RGB)
    assert jpeg[2:4].tobytes() == b"\xff\xee" and b"Adobe" in jpeg[:20].tobytes()
    _, coef = o.decode(jpeg, want_coef=True)          # pixels are meaningless here (RGB samples), coefficients are not

    def live():
        out = np.empty(4096 + coef.size * 8, np.uint8)
        n = o.ref.ref_encode_from_coef_rgb(np.ascontiguousarray(coef).reshape(-1), w, h, q, rst, il, sampling[0], sampling[1],
                                           out, out.size)
        assert n > 0
        return digest(out[:n])
    assert digest(jpeg) == ref(request, live)
    back = o.decode_any(jpeg, o.FMT_444_P012, o.CS_RGB).reshape(h, w, 3).astype(int)
    assert np.abs(back - img).mean() < 12


@pytest.mark.parametrize("internal,il,sampling", [(o.CS_709, 1, (2, 1)), (o.CS_601, 0, (1, 1)), (o.CS_709, 1, (2, 2))])
def test_spiff_stream_bytes(request, internal, il, sampling):
    """BT.601 / BT.709 internal colour space: SPIFF APP8 header + end-of-directory + second SOI (and the CS=ITU601
    comment) -- oracle bytes against the reference's header writer + CPU Huffman encoder on the same coefficients
    [ref: src/gpujpeg_writer.c:171-245, 462-466, 513-515]"""
    w, h, q, rst = 100, 60, 85, 5
    img = o.gen_image("photo", w, h)
    jpeg = o.encode_any(img, w, h, o.FMT_444_P012, o.CS_RGB, q, rst, il, sampling, internal=internal)
    assert jpeg[2:4].tobytes() == b"\xff\xe8" and jpeg[6:12].tobytes() == b"SPIFF\x00"
    _, coef = o.decode(jpeg, want_coef=True)          # coefficients only; the pixels of o.decode assume YCbCr JPEG

    def live():
        out = np.empty(4096 + coef.size * 8, np.uint8)
        n = o.ref.ref_encode_from_coef_cs(np.ascontiguousarray(coef).reshape(-1), w, h, q, rst, il, sampling[0], sampling[1],
                                          internal, out, out.size)
        assert n > 0
        return digest(out[:n])
    assert digest(jpeg) == ref(request, live)
    back = o.decode_any(jpeg, o.FMT_444_P012, o.CS_RGB).reshape(h, w, 3).astype(int)
    assert np.abs(back - img).mean() < 12


def test_subsampled_chroma_is_point_sampled():
    """the preprocessor keeps every second chroma sample unfiltered and the postprocessor replicates it
    [ref: src/gpujpeg_preprocessor.cu:50-64, src/gpujpeg_postprocessor.cu:55-76]: an image whose colour only changes
    at even pixel positions decodes to the same pixels with 4:2:0 as with 4:4:4 at quality 100 (up to DCT rounding)"""
    rng = np.random.default_rng(5)
    base = rng.integers(0, 256, (24, 32, 3), dtype=np.uint8)
    img = np.repeat(np.repeat(base, 2, axis=0), 2, axis=1)
    a = o.decode(o.encode(img, 100, 4, 1, sampling=(2, 2))).astype(int)
    b = o.decode(o.encode(img, 100, 4, 1)).astype(int)
    assert np.abs(a - img).max() <= 6 and np.abs(b - img).max() <= 6


@pytest.mark.parametrize("kind,q", [("random", 75), ("photo", 75), ("random", 100), ("gradient", 20)])
def test_integer_idct_matches_gpujpeg_idct_cpu(request, kind, q):
    w, h = 256, 128
    img = o.gen_image(kind, w, h)
    _, coef = o.encode(img, q, 8, want_coef=True)
    planes = ref(request, lambda: [digest(p) for p in ref_idct_planes(coef, w, h, q)])
    _, _, inv = o.quant_tables(q)
    for c in range(3):
        plane = np.zeros(w * h, np.uint8)
        o.lib.orc_idct_plane(np.ascontiguousarray(coef[c]), w, h, inv[0 if c == 0 else 1], o.IDCT_INT, plane)
        assert digest(plane.reshape(h, w)) == planes[c]


def test_idct_saturating_blocks(request):
    """sparse blocks whose reconstruction overshoots [-256,255] but stays inside the reference's
    1024-entry clip table (outside it the reference reads out of bounds, src/gpujpeg_dct_cpu.c:42-43)."""
    rng = np.random.default_rng(7)
    _, _, inv = o.quant_tables(50)
    blocks = []
    for _ in range(3000):
        blk = np.zeros(64, np.int16)
        idx = rng.choice(64, 6, replace=False)
        blk[idx] = rng.integers(-10, 11, 6)
        blk[0] = rng.integers(-24, 25)
        if np.abs(blk.astype(np.int64) * inv[0]).sum() > 1900:
            continue
        blocks.append(blk)
    blocks = np.array(blocks)
    mine = blocks.copy()
    for a in mine:
        o.lib.orc_idct_int_block(a, inv[0])

    def live():
        theirs = blocks.copy()
        for b in theirs:
            o.ref.ref_idct_block(b, inv[0])
        return digest(theirs)
    assert digest(mine) == ref(request, live)


@pytest.mark.parametrize("hdr", [1, 2, 4])           # GPUJPEG_HEADER_JFIF, _SPIFF, _ADOBE
@pytest.mark.parametrize("internal", [0, 1, 2, 4])   # YCbCr JPEG, RGB, BT.601, BT.709
def test_forced_header_flavours_equal_the_reference_writer(request, hdr, internal):
    """enc_hdr=JFIF|SPIFF|Adobe [ref: src/gpujpeg_encoder.c:759-766, src/gpujpeg_writer.c:451-518]: the product's host writer
    (gj_write_header through the host shim) against the reference's own gpujpeg_writer.c compiled in place, for every
    internal colour space -- including the combinations that make little sense (Adobe transform 0 on a YCbCr stream),
    which the reference writes just the same"""
    from _shims import hs
    w, h, q, rst = 64, 48, 75, 4
    coef = np.zeros((3, 64 * 48), np.int16)

    def live():
        o.ref.ref_set_header_type.argtypes = [__import__("ctypes").c_int]
        o.ref.ref_set_header_type(hdr)
        try:
            if internal == 1:
                out = np.empty(1 << 16, np.uint8)
                n = o.ref.ref_encode_from_coef_rgb(coef.reshape(-1), w, h, q, rst, 0, 1, 1, out, out.size)
            elif internal in (2, 4):
                out = np.empty(1 << 16, np.uint8)
                n = o.ref.ref_encode_from_coef_cs(coef.reshape(-1), w, h, q, rst, 0, 1, 1, internal, out, out.size)
            else:
                out = np.empty(1 << 16, np.uint8)
                n = o.ref.ref_encode_from_coef_ss(coef.reshape(-1), w, h, 3, q, rst, 0, 1, 1, out, out.size)
        finally:
            o.ref.ref_set_header_type(0)
        sos = bytes(out[:n]).index(b"\xff\xda")
        return [sos, digest(out[:sos])]
    sos, ref_head = ref(request, live)
    got = np.zeros(4096, np.uint8)
    hs.shim_set_header_type(hdr)
    try:
        m = hs.shim_header2(w, h, q, rst, 0, 3, 1, 1, internal if internal else 3, got)
    finally:
        hs.shim_set_header_type(0)
    assert digest(got[:sos]) == ref_head, "header bytes differ from the reference writer"
    assert m >= sos
