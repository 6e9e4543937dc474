"""4-component JPEGs (SURVEY section 8f rank 4: "4-component alpha"): an RGBA image encoded with comp_count = 4 keeps its
alpha samples as a fourth component.  CPU tests: the oracle restatement against the reference's own header writer + CPU
Huffman coder compiled in place (their answers recorded in tests/golden/ref_alpha_component.json), and the product's host
writer / reader against the oracle."""
import ctypes as C

import numpy as np
import pytest

import _oracle as o
from _refstore import digest, want
from _shims import hs


def rgba(w, h, seed=3):
    img = np.empty((h, w, 4), np.uint8)
    img[:, :, :3] = o.gen_image("photo", w, h, seed)
    yy, xx = np.mgrid[0:h, 0:w]
    img[:, :, 3] = ((xx * 3 + yy * 5) % 256).astype(np.uint8)     # a ramp: alpha that compresses, unlike noise
    return img


CASES = [(100, 60, 85, 5, 0, (1, 1)), (100, 60, 85, 5, 1, (1, 1)), (64, 48, 75, 0, 0, (1, 1)), (33, 17, 90, 2, 1, (1, 1)),
         (100, 60, 80, 3, 1, (2, 2)), (101, 61, 80, 4, 0, (2, 1)), (96, 64, 70, 6, 1, (1, 2))]


@pytest.mark.parametrize("w,h,q,rst,il,sampling", CASES)
@pytest.mark.parametrize("internal", [o.CS_JPEG, o.CS_RGB])
def test_four_component_stream_bytes(request, w, h, q, rst, il, sampling, internal):
    """SPIFF header (profile, colour space code 3 / 10), four SOF0 components with ids 1..4 / 'R','G','B','A', the fourth coded
    with the luminance tables and the first component's sampling, four scans or one interleaved scan: oracle bytes against
    the reference's header writer + CPU Huffman encoder on the same coefficients"""
    if internal == o.CS_RGB and sampling != (1, 1):
        pytest.skip("RGB-internal streams are not subsampled")
    img = rgba(w, h)
    jpeg = o.encode_any(img, w, h, o.FMT_4444_P0123, o.CS_RGB, q, rst, il, sampling, internal=internal, alpha=True)
    assert jpeg[2:4].tobytes() == b"\xff\xe8" and jpeg[6:12].tobytes() == b"SPIFF\x00"
    assert o.probe(jpeg).comp_count == 4
    coef = o.coefficients(jpeg)

    def live():
        out = np.empty(4096 + coef.size * 8, np.uint8)
        if internal == o.CS_RGB:
            n = ref_encode_rgb4(coef, w, h, q, rst, il, out)
        else:
            n = o.ref.ref_encode_from_coef_ss(coef, w, h, 4, q, rst, il, sampling[0], sampling[1], out, out.size)
        assert n > 0
        if internal == o.CS_RGB:
            return [digest(out[:n]), None]
        from _refcpu import ref_decode_coef
        return [digest(out[:n]), digest(ref_decode_coef(jpeg, w, h, rst, il, comps=4, sampling=sampling).reshape(-1))]
    ref_jpeg, ref_coef = want("alpha_component", request.node.name, live)
    assert digest(jpeg) == ref_jpeg, "oracle bytes != reference header writer + CPU Huffman encoder"
    if internal != o.CS_RGB:   # and back: the reference's CPU Huffman decoder recovers the coefficients of all four components
        assert digest(coef) == ref_coef, "reference CPU Huffman decoder != oracle coefficients"
    back = o.decode_any(jpeg, o.FMT_4444_P0123, o.CS_RGB).reshape(h, w, 4).astype(int)
    assert np.abs(back[:, :, :3] - img[:, :, :3]).mean() < 14 and np.abs(back[:, :, 3] - img[:, :, 3]).mean() < 8
    # without alpha on the way out: the colour samples are the same
    rgb = o.decode_any(jpeg, o.FMT_444_P012, o.CS_RGB).reshape(h, w, 3)
    assert np.array_equal(rgb, back[:, :, :3])


def ref_encode_rgb4(coef, w, h, q, rst, il, out):
    """the reference writer for an RGB-internal stream with four components (harness switch + component count)"""
    fn = o.ref.ref_encode_from_coef_rgb_n
    fn.restype = C.c_size_t
    fn.argtypes = [np.ctypeslib.ndpointer(np.int16), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                   np.ctypeslib.ndpointer(np.uint8), C.c_size_t]
    return fn(coef, w, h, 4, q, rst, il, out, out.size)


@pytest.mark.parametrize("il,sampling", [(0, (1, 1)), (1, (1, 1)), (1, (2, 2)), (0, (2, 1))])
@pytest.mark.parametrize("internal", [o.CS_JPEG, o.CS_RGB, o.CS_709])
def test_host_writer_and_reader_with_four_components(il, sampling, internal):
    """gj_write_header / gj_write_sos for comp_count = 4 against the first bytes of an oracle stream; the reader's view of it"""
    if internal == o.CS_RGB and sampling != (1, 1):
        pytest.skip("RGB-internal streams are not subsampled")
    w, h, q, rst = 70, 50, 80, 3
    jpeg = o.encode_any(rgba(w, h), w, h, o.FMT_4444_P0123, o.CS_RGB, q, rst, il, sampling, internal=internal, alpha=True)
    mine = np.zeros(4096, np.uint8)
    hs.shim_set_alpha_sampling(1)
    n = hs.shim_header2(w, h, q, rst, il, 4, sampling[0], sampling[1], internal, mine)
    hs.shim_set_alpha_sampling(0)
    assert n > 300 and np.array_equal(mine[:n], jpeg[:n])
    info = np.zeros(8, np.int32)
    off, ln = np.zeros(4096, np.uint32), np.zeros(4096, np.uint32)
    nseg = hs.shim_parse(jpeg, jpeg.size, info, off, ln, 4096)
    assert nseg > 0 and tuple(info[:3]) == (w, h, 4) and info[4] == (1 if il else 4) and info[7] == internal
