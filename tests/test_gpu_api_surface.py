"""GPU tests of the last pieces of SURVEY section 8f rank 4: 4-component (alpha) JPEGs, the Exif header and orientation
metadata through the encoder / decoder options, image-file helpers through the public API -- product against the CPU
oracle and against the reference GPU library itself (its outputs for these inputs recorded in
tests/golden/ref_gpu_api_surface.json, tests/_refstore.py)."""
import ctypes as C

import numpy as np
import pytest

import _oracle as o
from _refstore import digest, want as _want
from test_alpha_component import rgba
from test_ref_gpu import ref_file, run_ref

pytestmark = pytest.mark.gpu
RGB, YCC = 1, 3
FMT_RGB, FMT_RGBA = 1, 6


def recorded(request, live):
    return _want("gpu_api_surface", request.node.name, live)


@pytest.mark.parametrize("w,h,q,rst,il,ss", [(640, 360, 80, 6, 0, "4:4:4"), (640, 360, 80, 6, 1, "4:4:4"), (333, 77, 90, 3, 1, "4:2:0"),
                                             (322, 201, 75, 0, 0, "4:2:2"), (1118, 561, 85, 8, 0, "4:2:0"), (64, 64, 95, 1, 1, "4:4:0")])
def test_four_component_jpeg_against_oracle(w, h, q, rst, il, ss):
    """comp_count = 4: bytes of the oracle; decoded to RGBA (alpha from the fourth component), to RGB (alpha dropped) and to
    planar YCbCr -- pixels of the oracle"""
    import gpujpeg_b200 as g
    img = rgba(w, h)
    sampling = g.api.SUBSAMPLING[ss]
    want = o.encode_any(img, w, h, o.FMT_4444_P0123, o.CS_RGB, q, rst, il, sampling, threads=4, alpha=True)
    e = g.Encoder()
    got = e.encode_samples(img.reshape(-1), w, h, FMT_RGBA, q, rst, il, color_space=RGB, subsampling=ss, alpha=True)
    assert got.size == want.size and np.array_equal(got, want), "4-component JPEG bytes differ from the oracle"
    e.close()
    d = g.Decoder()
    out, pi = d.decode_samples(want)                      # default request: autodetect -> 4444-u8-p0123, RGB
    assert (pi.pixel_format, pi.color_space) == (FMT_RGBA, RGB)
    assert np.array_equal(out, o.decode_any(want, o.FMT_4444_P0123, o.CS_RGB, threads=4))
    d.set_output_format(RGB, g.api.GPUJPEG_PIXFMT_NO_ALPHA)
    out, pi = d.decode_samples(want)
    assert pi.pixel_format == FMT_RGB and np.array_equal(out, o.decode_any(want, o.FMT_444_P012, o.CS_RGB, threads=4))
    if w % 2 == 0:
        d.set_output_format(YCC, g.api.GPUJPEG_420_U8_P0P1P2)
        out, _ = d.decode_samples(want)
        assert np.array_equal(out, o.decode_any(want, o.FMT_420_P0P1P2, o.CS_JPEG, threads=4))
    d.close()


@pytest.mark.parametrize("il,packed,ss", [(0, 0x11111111, (1, 1)), (1, 0x11111111, (1, 1)), (1, 0x22111122, (2, 2))])
def test_four_component_jpeg_against_reference_gpu(request, tmp_path, il, packed, ss):
    """the reference GPU library with comp_count = 4: its bytes == oracle == product; its decoder (RGBA out) == float
    flavour of oracle and product"""
    import gpujpeg_b200 as g
    w, h, q, rst = 640, 360, 85, 6
    img = rgba(w, h)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"

    def live():
        img.tofile(src)
        run_ref("encode_raw", src, FMT_RGBA, RGB, w, h, q, rst, il, path, "sub:%#x" % packed)
        reply = run_ref("decode_fmt", path, RGB, g.api.GPUJPEG_PIXFMT_AUTODETECT, dst)
        return [ref_file(path), reply["pixel_format"], ref_file(dst)]
    ref, pixel_format, pix = recorded(request, live)
    want = o.encode_any(img, w, h, o.FMT_4444_P0123, o.CS_RGB, q, rst, il, ss, threads=4, alpha=True)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    e = g.Encoder()
    name = {(1, 1): "4:4:4", (2, 2): "4:2:0"}[ss]
    got = e.encode_samples(img.reshape(-1), w, h, FMT_RGBA, q, rst, il, color_space=RGB, subsampling=name, alpha=True)
    assert digest(got) == ref, "product != reference GPU library output"
    e.close()
    assert pixel_format == FMT_RGBA
    assert digest(o.decode_any(want, o.FMT_4444_P0123, o.CS_RGB, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle != reference GPU decoder"
    d = g.Decoder(idct="float_gpuref")
    out, _ = d.decode_samples(want)
    assert digest(out) == pix, "product decode != reference GPU decoder"
    d.close()


def _info(jpeg):
    """gpujpeg_decoder_get_image_info2 -> (header type, orientation (set, rotation, flip))"""
    import gpujpeg_b200.api as api

    class Info(C.Structure):
        _fields_ = [("param_image", api.ImageParameters), ("param", api.Parameters), ("segment_count", C.c_int),
                    ("header_type", C.c_int), ("comment", C.c_char_p), ("metadata", C.c_uint32 * 2), ("pad", C.c_char * 512)]
    fn = api.lib.gpujpeg_decoder_get_image_info2
    fn.restype, fn.argtypes = C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(Info), C.c_int, C.c_uint]
    info = Info()
    assert fn(jpeg.ctypes.data, jpeg.size, C.byref(info), 0, 0) == 0
    m = info.metadata
    return info.header_type, (int(m[1] & 1), int(m[0] & 3), int((m[0] >> 2) & 1))


def _body(jpeg):
    """everything from the first DQT on (what the header flavour does not touch)"""
    return bytes(jpeg)[bytes(jpeg).find(b"\xff\xdb"):]


def test_exif_and_orientation_through_the_coders():
    """enc_hdr=Exif / enc_exif_tag / enc_metadata on the encoder; the decoder hands the orientation out with the picture and
    gpujpeg_decoder_get_image_info2 reports it; the coded picture is untouched by any of it"""
    import gpujpeg_b200 as g
    w, h = 320, 200
    img = o.gen_image("photo", w, h)
    plain = o.encode(img, 80, 6)
    d = g.Decoder()
    for opts, hdr, want in (([("enc_hdr", "Exif")], 8, (1, 0, 0)),
                            ([("enc_exif_tag", "0x10F:ASCII=maker"), ("enc_metadata", "orientation=270-")], 8, (1, 3, 1)),
                            ([("enc_metadata", "orientation=90")], 2, (1, 1, 0)),
                            ([("enc_metadata", "orientation=180-"), ("enc_hdr", "JFIF")], 1, (0, 0, 0))):
        e = g.Encoder()
        for k, v in opts:
            e.set_option(k, v)
        jpeg = e.encode(img, 80, 6)
        e.close()
        assert _body(jpeg) == _body(plain)
        assert _info(jpeg) == (hdr, want)
        out = d.decode_raw(jpeg.ctypes.data, jpeg.size)
        m = (C.c_uint32 * 2).from_address(out.metadata)
        assert (int(m[1] & 1), int(m[0] & 3), int((m[0] >> 2) & 1)) == want
        pix = np.ctypeslib.as_array((C.c_uint8 * out.data_size).from_address(out.data)).reshape(h, w, 3)
        assert np.array_equal(pix, o.decode(plain))
    d.close()
    e = g.Encoder()
    with pytest.raises(g.api.GpuJpegError):
        e.set_option("enc_metadata", "orientation=45")
    with pytest.raises(g.api.GpuJpegError):
        e.set_option("enc_exif_tag", "NoSuchTag=1")
    e.close()


@pytest.mark.parametrize("opts", [["enc_hdr=Exif", "enc_exif_tag=DateTime=2024:02:29 12:34:56"],
                                  ["enc_exif_tag=DateTime=2024:02:29 12:34:56", "enc_metadata=orientation=90-", "enc_exif_tag=0x9286:UNDEFINED=hello"],
                                  ["enc_metadata=orientation=180"], ["enc_metadata=orientation=270-", "enc_hdr=SPIFF"]])
def test_exif_and_orientation_against_reference_gpu(request, tmp_path, opts):
    """whole files of the reference GPU library with the same options: identical bytes (a user DateTime fixes the clock);
    the reference decoder reads the product's orientation back"""
    import gpujpeg_b200 as g
    w, h = 320, 200
    img = o.gen_image("photo", w, h)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"
    e = g.Encoder()
    for x in opts:
        k, _, v = x.partition("=")
        e.set_option(k, v)
    got = e.encode(img, 80, 6)
    e.close()

    def live():
        img.tofile(src)
        run_ref("encode_raw", src, FMT_RGB, RGB, w, h, 80, 6, 0, path, *["opt:" + x for x in opts])
        ref = ref_file(path)
        got.tofile(path)
        return [ref, run_ref("decode_fmt", path, RGB, FMT_RGB, dst)["orientation"]]
    ref, orientation = recorded(request, live)
    assert digest(got) == ref, "product file != reference GPU library file"
    assert orientation == list(_info(got)[1])


FILES = [("a.ppm", FMT_RGB, RGB), ("a.pgm", 0, YCC), ("a.pam", FMT_RGBA, RGB), ("a.pnm", FMT_RGB, RGB), ("a.y4m", 5, YCC), ("a.y4m", 2, 2)]


@pytest.mark.parametrize("name,fmt,cs", FILES)
def test_image_files_through_the_public_api(request, tmp_path, name, fmt, cs):
    """gpujpeg_image_save_to_file / _get_properties / _load_from_file (pinned memory) of the product; against the reference GPU
    library: its files are byte-identical, it loads the product's files and answers get_properties the same"""
    import gpujpeg_b200.api as api
    lib = api.lib
    w, h = 70, 50
    pi = api.image_parameters(w, h, 0, fmt, cs)
    lib.gpujpeg_image_calculate_size.restype = C.c_size_t
    raw = o.gen_raw(fmt, w, h) if fmt != FMT_RGBA else rgba(w, h).reshape(-1)
    assert lib.gpujpeg_image_calculate_size(C.byref(pi)) == raw.size
    path = str(tmp_path / name).encode()
    lib.gpujpeg_image_save_to_file.argtypes = [C.c_char_p, C.c_void_p, C.c_size_t, C.POINTER(api.ImageParameters)]
    assert lib.gpujpeg_image_save_to_file(path, raw.ctypes.data, raw.size, C.byref(pi)) == 0
    got = api.ImageParameters()
    lib.gpujpeg_image_get_properties.argtypes = [C.c_char_p, C.POINTER(api.ImageParameters), C.c_int]
    assert lib.gpujpeg_image_get_properties(path, C.byref(got), 1) == 0
    assert (got.width, got.height, got.pixel_format) == (w, h, fmt)
    ptr, size = C.c_void_p(), C.c_size_t(0)
    lib.gpujpeg_image_load_from_file.argtypes = [C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    assert lib.gpujpeg_image_load_from_file(path, C.byref(ptr), C.byref(size)) == 0 and size.value == raw.size
    assert np.array_equal(np.ctypeslib.as_array((C.c_uint8 * size.value).from_address(ptr.value)), raw)
    lib.gpujpeg_image_destroy.argtypes = [C.c_void_p]
    lib.gpujpeg_image_destroy(ptr)
    src, ref_path, dump = tmp_path / "in.raw", tmp_path / ("ref_" + name), tmp_path / "dump.raw"
    probes = ("x.pnm", "x.pam", "x.pgm", "x.y4m", "x.rgb", "x.i420")   # names of files still to be written

    def live():
        raw.tofile(src)
        rc, _ = run_ref("file_save", src, ref_path, fmt, cs, w, h)
        return {"save": [rc, ref_file(ref_path)], "props": run_ref("file_props", path.decode(), 1),
                "load": run_ref("file_load", path.decode(), dump) + [ref_file(dump)],
                "probes": [run_ref("file_props", probe, 0) for probe in probes]}
    ref = recorded(request, live)
    assert ref["save"] == [0, digest(np.fromfile(path.decode(), np.uint8))], "file of the reference library differs"
    assert ref["props"] == [0, got.width, got.height, got.color_space, got.pixel_format]
    assert ref["load"] == [0, raw.size, digest(raw)]
    for probe, want in zip(probes, ref["probes"]):
        mine = api.ImageParameters(0, 0, 0, -1, 0)
        rc = lib.gpujpeg_image_get_properties(probe.encode(), C.byref(mine), 0)
        assert [rc, mine.color_space, mine.pixel_format] == [want[0], want[3], want[4]], probe


@pytest.mark.parametrize("w,h,stripes,ss,il", [(1920, 1080, 8, "4:4:4", 0), (1119, 561, 5, "4:4:4", 0), (640, 136, 8, "4:4:4", 0),
                                               (3840, 2160, 0, "4:4:4", 0), (1119, 561, 7, "4:4:4", 1), (1280, 720, 8, "4:4:4", 1), (1119, 561, 7, "4:2:0", 1), (1118, 562, 8, "4:2:0", 0),
                                               (642, 361, 6, "4:2:2", 1), (640, 300, 4, "4:4:0", 0), (3840, 2160, 0, "4:2:0", 1)])
def test_stripe_pipeline_of_host_buffers(monkeypatch, w, h, stripes, ss, il):
    """host images of 8 MB or more are copied and transformed stripe by stripe (K1 behind the upload, the download behind K4):
    the same bytes and pixels as ever -- pinned and pageable buffers, frame heights that do not divide into the stripes,
    chroma subsampling (stripes of whole MCU rows), and small frames with the threshold lowered"""
    import torch
    import gpujpeg_b200 as g
    if stripes:
        monkeypatch.setenv("GPUJPEG_B200_STRIPES", str(stripes))
        monkeypatch.setenv("GPUJPEG_B200_STRIPE_MIN_BYTES", "1")
    img = o.gen_image("photo", w, h)
    want = o.encode(img, 80, 12, il, threads=4, sampling=g.api.SUBSAMPLING[ss])
    pix = o.decode(want, threads=4)
    e, d = g.Encoder(), g.Decoder()
    pinned = torch.from_numpy(img).pin_memory()
    for src in (img, pinned, img):
        assert np.array_equal(e.encode(src, 80, 12, il, subsampling=ss), want)
    out = torch.empty((h, w, 3), dtype=torch.uint8).pin_memory()
    d.decode(want, out=out.numpy())
    assert np.array_equal(out.numpy(), pix)
    assert np.array_equal(d.decode(want), pix)
    assert np.array_equal(d.decode(want, out=np.zeros((h, w, 3), np.uint8)), pix)
    e.close()
    d.close()
