"""CPU tests of the product's host side through the C-ABI (no GPU): the library loads and exports every declared
symbol, its Huffman decoder/encoder agree with the oracle byte for byte, and the CUDA-only paths fail loudly."""
import hashlib
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ZZ = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
               35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])
INPUTS = ["in_420_base_355x237.jpg", "in_420_prog_355x237.jpg", "in_444_base_355x237.jpg", "in_422_base_355x237.jpg",
          "in_gray_base_355x237.jpg", "in_420_base_640x480.jpg", "in_420_tiny_17x9.jpg", "in_420_tiny_3x3.jpg"]


def _no_gpu():
    import torch
    return not torch.cuda.is_available()


def test_abi_exports_every_declared_symbol(L):
    hdr = open(os.path.join(ROOT, "include", "b200_caesium.h")).read()
    declared = sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L.lib(), name), f"{name} declared in include/b200_caesium.h but not exported"


def test_params_default_and_sniff(L):
    p = L.default_params()
    assert (p.jpeg_quality, p.jpeg_progressive, p.jpeg_preserve_icc, p.png_optimization_level, p.width, p.height) == (80, 1, 1, 3, 0, 0)
    assert L.sniff_format(b"\xff\xd8\xff\xe0....") == L.FMT_JPEG
    assert L.sniff_format(b"\x89PNG\r\n\x1a\n....") == L.FMT_PNG
    assert L.sniff_format(b"RIFF\x00\x00\x00\x00WEBPVP8 ") == L.FMT_WEBP
    assert L.sniff_format(b"GIF89a......") == L.FMT_GIF
    assert L.sniff_format(b"II*\x00......") == L.FMT_TIFF
    assert L.sniff_format(b"hello world!") == L.FMT_UNKNOWN
    assert L.sniff_format(b"") == L.FMT_UNKNOWN


def test_quant_table_matches_oracle(L, O):
    for q in (0, 1, 5, 25, 49, 50, 51, 80, 95, 100):
        assert np.array_equal(L.jpeg_quant_table(q), O.quant_table(q))


@pytest.mark.parametrize("name", INPUTS)
def test_host_huffman_decode_matches_oracle(L, O, golden, name):
    data = golden(name)
    lay, co = L.jpeg_decode_coefficients(data)
    j = O.Jpeg(data)
    assert (lay.width, lay.height, lay.ncomp) == (j.s.width, j.s.height, j.s.ncomp)
    for c in range(lay.ncomp):
        assert np.array_equal(L.component_view(lay, co, c), j.coef(c)[:, :, ZZ])
        assert np.array_equal(np.array(lay.qt[c][:], dtype=np.uint16), j.qtable(c)[ZZ])


@pytest.mark.parametrize("rel", ["j0.JPG", "level_1_0/j1.jpg"])   # paths in the reference's samples/; the copies are flat
def test_host_progressive_decode_on_reference_fixtures(L, O, rel):
    data = open(os.path.join(ROOT, "tests", "golden", "reference_samples", os.path.basename(rel)), "rb").read()
    lay, co = L.jpeg_decode_coefficients(data)
    j = O.Jpeg(data)
    for c in range(3):
        assert np.array_equal(L.component_view(lay, co, c), j.coef(c)[:, :, ZZ])


@pytest.mark.parametrize("name", INPUTS)
@pytest.mark.parametrize("prog", [0, 1])
def test_lossless_transcode_bytes_match_oracle(L, O, golden, name, prog):
    """libcaesium jpeg::lossless (compressor.rs:427 -> jpeg.optimize): host-only entropy transcode, byte-identical."""
    data = golden(name)
    p = L.default_params()
    p.jpeg_optimize, p.jpeg_progressive = 1, prog
    out = L.compress_in_memory(data, p)
    assert out == O.jpeg_lossless(data, O.params(80, 0, bool(prog)))
    exp = json.load(open(os.path.join(ROOT, "tests", "golden", "expected.json")))[name]["lossless"][f"p{prog}"]
    assert hashlib.sha256(out).hexdigest() == exp["sha256"]
    # coefficients are carried bit-exactly
    l0, c0 = L.jpeg_decode_coefficients(data)
    l1, c1 = L.jpeg_decode_coefficients(out)
    for c in range(l0.ncomp):
        assert np.array_equal(L.component_view(l0, c0, c)[:l0.rbh[c], :l0.rbw[c]], L.component_view(l1, c1, c)[:l0.rbh[c], :l0.rbw[c]])


def _pillow_jpeg(**kw):
    import io
    from PIL import Image
    yy, xx = np.mgrid[0:237, 0:355]
    rgb = np.stack([(xx * 3 + yy) % 256, (xx + yy * 2) % 256, (xx * yy // 64) % 256], -1).astype(np.uint8)
    b = io.BytesIO()
    Image.fromarray(rgb).save(b, format="JPEG", **kw)
    return b.getvalue()


@pytest.mark.parametrize("kw", [dict(quality=85, restart_marker_blocks=7), dict(quality=85, restart_marker_rows=1),
                                dict(quality=85, progressive=True, restart_marker_rows=2), dict(quality=85, optimize=True)])
def test_restart_intervals_and_custom_tables_decode_like_the_oracle(L, O, kw):
    """Inputs with DRI / RSTn markers (baseline and progressive) and optimised Huffman tables: the host decoder (the route
    such files take, they are not device-decodable) must carry the coefficients exactly; checked through the transcode."""
    data = _pillow_jpeg(**kw)
    assert (b"\xff\xdd" in data) == any(k.startswith("restart") for k in kw)
    p = L.default_params()
    p.jpeg_optimize = 1
    assert L.compress_in_memory(data, p) == O.jpeg_lossless(data, O.params(80, 0, True))


@pytest.mark.parametrize("prog", [0, 1])
def test_host_huffman_encode_matches_oracle_writer(L, O, golden, prog):
    """Entropy-code the ORACLE's forward coefficients with the product's encoder: files must be identical."""
    data = golden("in_420_base_355x237.jpg")
    planes = O.Jpeg(data).decode_native()
    for ss in (420, 444, 422, 411):
        fw = O.forward(planes, O.params(70, ss, bool(prog)))
        ref = O.write(fw, O.params(70, ss, bool(prog)))
        lay, co = L.jpeg_decode_coefficients(ref)        # same coefficients, product layout
        assert L.jpeg_encode_coefficients(lay, co, prog) == ref


def test_output_layout(L, golden):
    lay, _ = L.jpeg_decode_coefficients(golden("in_444_base_355x237.jpg"))
    p = L.default_params()
    for ss, (h, v) in {444: (1, 1), 422: (2, 1), 420: (2, 2), 411: (4, 1), 0: (2, 2)}.items():
        p.jpeg_chroma_subsampling = ss
        o = L.jpeg_output_layout(lay, p)
        assert (o.hs[0], o.vs[0], o.hs[1], o.vs[1]) == (h, v, 1, 1)
        assert o.bw[0] == -(-355 // (8 * h)) * h and o.rbw[1] == -(-(-(-355 // h)) // 8)
    p.jpeg_chroma_subsampling = 7
    with pytest.raises(L.B200Error):
        L.jpeg_output_layout(lay, p)


def test_corrupt_and_unknown_inputs_return_errors(L, golden):
    p = L.default_params()
    p.jpeg_optimize = 1
    for bad, code in [(b"", L.ERR_UNKNOWN_FORMAT), (b"plain text", L.ERR_UNKNOWN_FORMAT), (b"\xff\xd8\xff\xe0\x00\x10JFIF", L.ERR_CORRUPT_INPUT),
                      (golden("in_420_base_355x237.jpg")[:300], L.ERR_CORRUPT_INPUT)]:
        with pytest.raises(L.B200Error) as e:
            L.compress_in_memory(bad, p)
        assert e.value.code == code
        assert str(e.value).endswith(f"[{code}]")          # CaesiumError Display: "{message} [{code}]"
    with pytest.raises(L.B200Error) as e:
        L.convert_in_memory(golden("in_420_base_355x237.jpg"), p, L.FMT_JPEG)
    assert e.value.code == L.ERR_SAME_FORMAT


def test_cuda_paths_fail_loudly_without_a_gpu(L, golden):
    """No CPU fallback: on a box without a B200 the lossy path must return B200_ERR_NO_DEVICE, never pixels."""
    if not _no_gpu():
        pytest.skip("a GPU is visible")
    p = L.default_params()
    with pytest.raises(L.B200Error) as e:
        L.compress_in_memory(golden("in_420_base_355x237.jpg"), p)
    assert e.value.code == L.ERR_NO_DEVICE
    lay, co = L.jpeg_decode_coefficients(golden("in_420_base_355x237.jpg"))
    with pytest.raises(L.B200Error) as e:
        L.jpeg_requantize(lay, co, L.jpeg_output_layout(lay, p))
    assert e.value.code == L.ERR_NO_DEVICE
    res = L.compress_batch([golden("in_420_base_355x237.jpg")] * 3, p, 2)
    assert all(r[1] == L.ERR_NO_DEVICE for r in res)
