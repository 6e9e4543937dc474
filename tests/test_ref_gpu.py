"""Level-2 cross-check on the GPU: the REFERENCE GPU library itself (compiled in place by `make -C oracle refgpu` into
oracle/_ref/libgpujpeg_refgpu.so) against the oracle restatement and against the product.  This is what validates the
restated float FDCT (FMA placement) and colour transforms on real hardware.  The reference's outputs for these inputs are
recorded in tests/golden/ref_ref_gpu.json (tests/_refstore.py; recorded on a B200), so the tests need no reference at run
time."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _oracle as o
from _refstore import digest, want as _want

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


_server = None


def run_ref(*args):
    """one command for the reference GPU library; all commands of a session go to ONE child process (`_refgpu.py
    serve`: one interpreter start, one CUDA context -- 70 separate children cost 2-3 s each, most of the GPU suite)"""
    import atexit
    import json
    global _server
    if _server is None or _server.poll() is not None:
        _server = subprocess.Popen([sys.executable, os.path.join(HERE, "_refgpu.py"), "serve"], stdin=subprocess.PIPE,
                                   stdout=subprocess.PIPE, text=True)
        assert json.loads(_server.stdout.readline()).get("ready"), "reference GPU library did not start"
        atexit.register(lambda p=_server: (p.stdin.close(), p.wait(timeout=30)))
    _server.stdin.write(json.dumps([str(a) for a in args]) + "\n")
    _server.stdin.flush()
    line = _server.stdout.readline()
    assert line, "reference GPU library process died"
    reply = json.loads(line)
    assert reply["ok"], reply.get("error")
    return reply["reply"]


def recorded(request, live):
    return _want("ref_gpu", request.node.name, live)


def ref_file(path, shape=None):
    """digest of a file the reference library wrote"""
    a = np.fromfile(path, np.uint8)
    return digest(a if shape is None else a.reshape(shape))


@pytest.mark.parametrize("kind,w,h,q,rst,il", [("random", 1920, 1080, 75, 24, 0), ("photo", 1920, 1080, 75, 24, 0),
                                               ("random", 1119, 561, 75, 8, 0), ("photo", 640, 360, 90, 7, 1),
                                               ("random", 512, 512, 100, 12, 0), ("photo", 3840, 2160, 75, 24, 0)])
def test_reference_gpu_encoder_bytes_equal_oracle_and_product(request, tmp_path, kind, w, h, q, rst, il):
    path = tmp_path / "ref.jpg"

    def live():
        run_ref("encode", kind, w, h, q, rst, il, path)
        return ref_file(path)
    ref = recorded(request, live)
    img = o.gen_image(kind, w, h)
    want = o.encode(img, q, rst, il, threads=4)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    import gpujpeg_b200 as g
    e = g.Encoder()
    assert digest(e.encode(img, q, rst, il)) == ref, "product != reference GPU library output"
    e.close()


@pytest.mark.parametrize("kind,w,h,q", [("random", 1920, 1080, 75), ("photo", 1920, 1080, 75), ("random", 333, 77, 95)])
def test_reference_gpu_decoder_pixels_equal_float_flavour(request, tmp_path, kind, w, h, q):
    jpeg = o.encode(o.gen_image(kind, w, h), q, 24)
    src, dst = tmp_path / "in.jpg", tmp_path / "out.rgb"

    def live():
        jpeg.tofile(src)
        run_ref("decode", src, dst)
        return ref_file(dst, (h, w, 3))
    ref = recorded(request, live)
    want = o.decode(jpeg, o.IDCT_FLOAT_GPUREF)
    assert want.shape == (h, w, 3) and digest(want) == ref, "float-GPU-reference IDCT restatement != reference GPU library output"
    import gpujpeg_b200 as g
    d = g.Decoder(idct="float_gpuref")
    assert digest(d.decode(jpeg)) == ref
    d.close()


SS = [("4:2:0", (2, 2)), ("4:2:2", (2, 1)), ("4:4:0", (1, 2))]


@pytest.mark.parametrize("il", [0, 1])
@pytest.mark.parametrize("name,sampling", SS)
@pytest.mark.parametrize("kind,w,h,q,rst", [("photo", 1920, 1080, 75, 12), ("random", 1119, 561, 90, 8)])
def test_reference_gpu_subsampled_encode_and_decode(request, tmp_path, kind, w, h, q, rst, name, sampling, il):
    """chroma subsampling: reference GPU encoder bytes == oracle == product; reference GPU decoder pixels ==
    float flavour of oracle and product"""
    path, dst = tmp_path / "ref.jpg", tmp_path / "out.rgb"

    def live():
        run_ref("encode", kind, w, h, q, rst, il, path, sampling[0], sampling[1])
        run_ref("decode", path, dst)
        return [ref_file(path), ref_file(dst, (h, w, 3))]
    ref, pix = recorded(request, live)
    img = o.gen_image(kind, w, h)
    want = o.encode(img, q, rst, il, threads=4, sampling=sampling)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    import gpujpeg_b200 as g
    e = g.Encoder()
    assert digest(e.encode(img, q, rst, il, subsampling=name)) == ref, "product != reference GPU library output"
    e.close()
    assert digest(o.decode(want, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle decode != reference GPU decoder"
    d = g.Decoder(idct="float_gpuref")
    assert digest(d.decode(want)) == pix, "product decode != reference GPU decoder"
    d.close()


FMTS = {0: "u8", 1: "444-u8-p012", 2: "444-u8-p0p1p2", 3: "422-u8-p1020", 4: "422-u8-p0p1p2", 5: "420-u8-p0p1p2"}


@pytest.mark.parametrize("il", [0, 1])
@pytest.mark.parametrize("fmt", sorted(FMTS), ids=[FMTS[f] for f in sorted(FMTS)])
@pytest.mark.parametrize("w,h,q,rst", [(640, 360, 80, 6), (1118, 561, 90, 8)])
def test_reference_gpu_raw_formats(request, tmp_path, w, h, q, rst, fmt, il):
    """grey / planar / packed YCbCr input in the JPEG colour space (no colour transform): reference GPU encoder bytes
    == oracle == product; reference GPU decoder samples (same format requested) == float flavour of oracle and product"""
    raw = o.gen_raw(fmt, w, h)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"

    def live():
        raw.tofile(src)
        run_ref("encode_raw", src, fmt, 3, w, h, q, rst, il, path)     # 3 = GPUJPEG_YCBCR_BT601_256LVLS
        run_ref("decode_fmt", path, 3, fmt, dst)
        return [ref_file(path), ref_file(dst)]
    ref, pix = recorded(request, live)
    want = o.encode_ycc(raw, w, h, fmt, q, rst, il, threads=4)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    import gpujpeg_b200 as g
    e = g.Encoder()
    assert digest(e.encode_samples(raw, w, h, fmt, q, rst, il)) == ref, "product != reference GPU library output"
    e.close()
    assert digest(o.decode_ycc(want, fmt, w, h, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle != reference GPU decoder"
    d = g.Decoder(idct="float_gpuref")
    d.set_output_format(g.api.GPUJPEG_YCBCR_JPEG, fmt)
    out, _ = d.decode_samples(want)
    assert digest(out) == pix, "product decode != reference GPU decoder"
    d.close()


@pytest.mark.parametrize("il", [0, 1])
@pytest.mark.parametrize("fmt,cs,w,h", [(1, 4, 640, 360), (1, 2, 322, 201), (3, 4, 640, 360), (3, 1, 320, 200), (2, 1, 640, 360),
                                        (4, 2, 640, 360), (5, 4, 640, 360), (5, 1, 322, 200)])
def test_reference_gpu_colour_spaces(request, tmp_path, fmt, cs, w, h, il):
    """input in RGB / BT.601 / BT.709 in every pixel format (colour transform to the JPEG's YCbCr, the JPEG takes the
    format's sampling): reference GPU encoder bytes == oracle == product, and the reference GPU decoder asked for the
    same format and colour space == float flavour of oracle and product"""
    raw = o.gen_raw(fmt, w, h)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"

    def live():
        raw.tofile(src)
        run_ref("encode_raw", src, fmt, cs, w, h, 85, 6, il, path)
        run_ref("decode_fmt", path, cs, fmt, dst)
        return [ref_file(path), ref_file(dst)]
    ref, pix = recorded(request, live)
    want = o.encode_any(raw, w, h, fmt, cs, 85, 6, il, o.FMT_SAMPLING[fmt], threads=4)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    import gpujpeg_b200 as g
    e = g.Encoder()
    assert digest(e.encode_samples(raw, w, h, fmt, 85, 6, il, color_space=cs)) == ref, "product != reference GPU library"
    e.close()
    assert digest(o.decode_any(want, fmt, cs, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle != reference GPU decoder"
    d = g.Decoder(idct="float_gpuref")
    d.set_output_format(cs, fmt)
    out, _ = d.decode_samples(want)
    assert digest(out) == pix, "product decode != reference GPU decoder"
    d.close()


@pytest.mark.parametrize("fmt,cs,il,internal", [(1, 1, 0, 1), (1, 1, 1, 1), (2, 1, 0, 1), (1, 4, 1, 1), (3, 4, 1, 4), (1, 1, 0, 4),
                                                (5, 3, 1, 2), (1, 2, 0, 2)])
def test_reference_gpu_rgb_internal_jpeg(request, tmp_path, fmt, cs, il, internal):
    """color_space_internal = GPUJPEG_RGB (Adobe APP14 header, luminance tables for every component) or BT.601 / BT.709
    (SPIFF header): reference GPU encoder bytes == oracle == product; reference GPU decoder == oracle == product for
    the same output request"""
    w, h = 640, 360
    raw = o.gen_raw(fmt, w, h) if cs != 1 else np.ascontiguousarray(o.gen_image("photo", w, h)).reshape(-1)
    if fmt == 2:    # planar RGB
        raw = np.ascontiguousarray(raw.reshape(h, w, 3).transpose(2, 0, 1)).reshape(-1)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"

    def live():
        raw.tofile(src)
        run_ref("encode_raw", src, fmt, cs, w, h, 85, 6, il, path, internal)
        run_ref("decode_fmt", path, cs, fmt, dst)
        return [ref_file(path), ref_file(dst)]
    ref, pix = recorded(request, live)
    want = o.encode_any(raw, w, h, fmt, cs, 85, 6, il, o.FMT_SAMPLING[fmt], threads=4, internal=internal)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    import gpujpeg_b200 as g
    e = g.Encoder()
    p = g.api.default_parameters(85, 6, il)
    p.color_space_internal = internal
    addr, size = e.encode_raw(raw, p, g.api.image_parameters(w, h, 0, fmt, cs))
    got = np.ctypeslib.as_array((__import__("ctypes").c_uint8 * size).from_address(addr)).copy()
    assert digest(got) == ref, "product != reference GPU library output"
    e.close()
    assert digest(o.decode_any(want, fmt, cs, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle != reference GPU decoder"
    d = g.Decoder(idct="float_gpuref")
    d.set_output_format(cs, fmt)
    out, _ = d.decode_samples(want)
    assert digest(out) == pix, "product decode != reference GPU decoder"
    d.close()


def test_reference_gpu_rgba(request, tmp_path):
    """4444-u8-p0123 input / output with the default 3-component JPEG: reference GPU library == oracle == product"""
    w, h = 640, 360
    img = o.gen_image("photo", w, h)
    rgba = np.ascontiguousarray(np.concatenate([img, np.full((h, w, 1), 77, np.uint8)], axis=2)).reshape(-1)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"

    def live():
        rgba.tofile(src)
        run_ref("encode_raw", src, 6, 1, w, h, 85, 6, 1, path)
        run_ref("decode_fmt", path, 1, 6, dst)
        return [ref_file(path), ref_file(dst)]
    ref, pix = recorded(request, live)
    want = o.encode_any(rgba, w, h, 6, 1, 85, 6, 1, (1, 1), threads=4)
    assert digest(want) == ref, "oracle != reference GPU library"
    import gpujpeg_b200 as g
    e = g.Encoder()
    assert digest(e.encode_samples(rgba, w, h, 6, 85, 6, 1, color_space=1)) == ref, "product != reference GPU library"
    e.close()
    assert digest(o.decode_any(want, 6, 1, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle != reference GPU decoder"
    d = g.Decoder(idct="float_gpuref")
    d.set_output_format(1, 6)
    assert digest(d.decode_samples(want)[0]) == pix, "product decode != reference GPU decoder"
    d.close()


@pytest.mark.parametrize("fmt,cs,w,h,flipped,remap", [(1, 1, 322, 201, True, None), (1, 1, 320, 208, True, None), (1, 1, 160, 96, False, "210"), (1, 1, 322, 200, True, "2Z0"),
                                                      (6, 1, 128, 64, False, "1230"), (5, 3, 320, 200, True, None)])
def test_reference_gpu_flip_and_channel_remap(request, tmp_path, fmt, cs, w, h, flipped, remap):
    """enc/dec_opt_flipped and enc/dec_opt_channel_remap: reference GPU library == oracle == product"""
    raw = o.gen_raw(fmt, w, h) if fmt not in (1, 6) else np.ascontiguousarray(o.gen_image("photo", w, h)).reshape(-1)
    if fmt == 6:
        raw = np.random.default_rng(7).integers(0, 256, w * h * 4, dtype=np.uint8)
    src, path, dst = tmp_path / "in.raw", tmp_path / "ref.jpg", tmp_path / "out.raw"
    eopts = (["opt:enc_opt_flipped=1"] if flipped else []) + (["opt:enc_opt_channel_remap=" + remap] if remap else [])
    dopts = (["opt:dec_opt_flipped=1"] if flipped else []) + (["opt:dec_opt_channel_remap=" + remap] if remap else [])

    def live():
        raw.tofile(src)
        run_ref("encode_raw", src, fmt, cs, w, h, 85, 6, 1, path, *eopts)
        run_ref("decode_fmt", path, cs, fmt, dst, *dopts)
        return [ref_file(path), ref_file(dst)]
    ref, pix = recorded(request, live)
    with o.flip_remap(flipped, remap):
        want = o.encode_any(raw, w, h, fmt, cs, 85, 6, 1, o.FMT_SAMPLING[fmt] if fmt != 6 else (1, 1), threads=4)
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    with o.flip_remap(flipped, remap):
        assert digest(o.decode_any(want, fmt, cs, o.IDCT_FLOAT_GPUREF, threads=4)) == pix, "oracle != reference GPU decoder"
    import gpujpeg_b200 as g
    d = g.Decoder(idct="float_gpuref")
    try:
        if flipped:
            d.set_option("dec_opt_flipped", "1")
        if remap:
            d.set_option("dec_opt_channel_remap", remap)
        d.set_output_format(cs, fmt)
        assert digest(d.decode_samples(want)[0]) == pix, "product decode != reference GPU decoder"
    finally:
        d.close()


@pytest.mark.parametrize("kind,w,h,q,rst,il,name,sampling", [("photo", 640, 360, 75, 12, 0, "4:4:4", (1, 1)), ("random", 333, 177, 85, 3, 1, "4:4:4", (1, 1)),
                                                             ("photo", 640, 368, 75, 4, 0, "4:2:0", (2, 2)),
                                                             ("photo", 1024, 1032, 60, 1, 0, "4:4:4", (1, 1))])   # 16 512 segments per scan: two APP13 headers each
def test_reference_gpu_segment_info(request, tmp_path, kind, w, h, q, rst, il, name, sampling):
    """struct gpujpeg_parameters.segment_info: APP13 tables of the restart segments' positions in front of every scan
    [ref: src/gpujpeg_writer.c:522-599]: reference GPU encoder bytes == oracle == product, and the reference decoder -- which
    then splits the scans by the table instead of searching for markers, src/gpujpeg_reader.c:1168-1215 -- decodes the
    product's stream to the same picture"""
    path, mine, dst = tmp_path / "ref.jpg", tmp_path / "mine.jpg", tmp_path / "out.rgb"
    extra = (sampling[0], sampling[1]) if sampling != (1, 1) else ()
    img = o.gen_image(kind, w, h)
    with o.segment_info():
        want = o.encode(img, q, rst, il, threads=4, sampling=sampling)
    plain = o.encode(img, q, rst, il, threads=4, sampling=sampling)
    import gpujpeg_b200 as g
    e = g.Encoder()
    got = e.encode(img, q, rst, il, subsampling=name, segment_info=1)

    def live():
        run_ref("encode", kind, w, h, q, rst, il, path, *extra, "par:segment_info=1")
        got.tofile(mine)
        run_ref("decode", mine, dst)
        return [int(np.fromfile(path, np.uint8).size), ref_file(path), ref_file(dst, (h, w, 3))]
    ref_size, ref, pix = recorded(request, live)
    assert ref_size > plain.size
    assert digest(want) == ref, "oracle restatement != reference GPU library output"
    assert digest(got) == ref, "product != reference GPU library output"
    assert np.array_equal(e.encode(img, q, rst, il, subsampling=name), plain), "the same encoder without segment info afterwards"
    e.close()
    d = g.Decoder(idct="float_gpuref")
    assert digest(d.decode(got)) == pix, "product decode != reference GPU decoder on a stream with segment info"
    d.close()
