"""CPU tests that PIN THE ORACLE (oracle/jpeg_oracle.c) -- the reference itself cannot be built here.

Pins, in order of strength:
  * known-answer vectors taken from the reference's own fixtures (SURVEY.md §8c KAT-1..3): the DQT of samples/j0.JPG
    (mozjpeg Robidoux table @ q51), the Annex-K DQT of level_1_0/j1.jpg, both files' progressive scan scripts;
  * a sibling implementation: libjpeg-turbo (via Pillow), the code base mozjpeg is a fork of -- bit-exact decode in
    native YCbCr and bit-exact forward path (downsample + ISLOW FDCT + quantise) on odd-sized inputs;
  * the committed golden vectors in tests/golden/expected.json (oracle drift detector);
  * the four numeric facts the reference's tests assert (compressor.rs:1051-1068).
The reference's fixtures are read from their copies in tests/golden/reference_samples.
"""
import hashlib
import io
import json
import os

import numpy as np
import pytest
from PIL import Image

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_samples")

J0_DQT = [16, 16, 16, 18, 25, 36, 55, 83, 16, 17, 20, 26, 33, 39, 52, 74, 16, 20, 24, 30, 42, 61, 89, 132, 18, 26, 30, 39, 52, 73, 104, 153,
          25, 33, 42, 52, 68, 92, 128, 185, 36, 39, 61, 73, 92, 122, 166, 233, 55, 52, 89, 104, 128, 166, 221, 305, 83, 74, 132, 153, 185, 233, 305, 410]
J1_DQT_LUMA = [8, 6, 5, 8, 12, 20, 26, 31, 6, 6, 7, 10, 13, 29, 30, 28, 7, 7, 8, 12, 20, 29, 35, 28, 7, 9, 11, 15, 26, 44, 40, 31,
               9, 11, 19, 28, 34, 55, 52, 39, 12, 18, 28, 32, 41, 52, 57, 46, 25, 32, 39, 44, 52, 61, 60, 51, 36, 46, 48, 49, 56, 50, 52, 50]
J0_SCANS = [(3, 0, 0, 0, 0), (1, 1, 2, 0, 1), (1, 3, 63, 0, 1), (1, 1, 63, 0, 1), (1, 1, 63, 0, 1), (1, 1, 63, 1, 0), (1, 1, 63, 1, 0), (1, 1, 63, 1, 0)]
INPUTS = ["in_420_base_355x237.jpg", "in_420_prog_355x237.jpg", "in_444_base_355x237.jpg", "in_422_base_355x237.jpg",
          "in_gray_base_355x237.jpg", "in_420_base_640x480.jpg", "in_420_tiny_17x9.jpg", "in_420_tiny_3x3.jpg"]


def pillow_native(data):
    im = Image.open(io.BytesIO(data))
    if im.mode != "L":
        im.draft("YCbCr", im.size)
    a = np.asarray(im)
    return a[None] if a.ndim == 2 else a.transpose(2, 0, 1)


def test_kat1_quant_table_matches_j0_fixture(O):
    # mozjpeg table idx 3 scaled by jpeg_set_quality(51, FALSE) must reproduce samples/j0.JPG's 16-bit DQT exactly
    assert list(map(int, O.quant_table(51))) == J0_DQT
    assert list(map(int, O.quant_table(80)))[:8] == [6, 6, 6, 7, 10, 15, 22, 34]
    assert list(map(int, O.quant_table(80)))[-8:] == [34, 30, 54, 62, 76, 95, 124, 167]
    assert int(O.quant_table(100).max()) == 1 and int(O.quant_table(0)[-1]) == O.quant_table(1)[-1] == 20900


def test_kat_fixture_headers(O):
    j0 = O.Jpeg(open(os.path.join(REF, "j0.JPG"), "rb").read())
    assert (j0.s.width, j0.s.height, j0.s.progressive) == (2000, 3000, 1)
    assert list(map(int, j0.qtable(0))) == J0_DQT and list(map(int, j0.qtable(1))) == J0_DQT
    assert [s[:5] for s in j0.scans()] == J0_SCANS                       # KAT-3
    j1 = O.Jpeg(open(os.path.join(REF, "j1.jpg"), "rb").read())
    assert list(map(int, j1.qtable(0))) == J1_DQT_LUMA                   # KAT-2 (Annex K @ q75)
    assert len(j1.scans()) == 10 and j1.scans()[5][:5] == (1, 1, 63, 2, 1)


@pytest.mark.parametrize("rel", ["j0.JPG", "level_1_0/j1.jpg"])   # paths in the reference's samples/; the copies are flat
def test_progressive_decode_matches_libjpeg_turbo_on_reference_fixtures(O, rel):
    data = open(os.path.join(REF, os.path.basename(rel)), "rb").read()
    assert np.array_equal(O.Jpeg(data).decode_native(), pillow_native(data))


@pytest.mark.parametrize("name", INPUTS)
def test_decode_matches_libjpeg_turbo(O, golden, name):
    data = golden(name)
    assert np.array_equal(O.Jpeg(data).decode_native(), pillow_native(data))


@pytest.mark.parametrize("w,h,ss,ssn", [(355, 237, 2, 420), (129, 65, 1, 422), (77, 33, 0, 444), (16, 16, 2, 420), (9, 200, 2, 420)])
def test_forward_path_matches_libjpeg_turbo(O, w, h, ss, ssn):
    """downsample (edge rules) + ISLOW FDCT + quantise == libjpeg-turbo's, incl. the dummy blocks of partial MCUs."""
    from tools.synth import synth_rgb
    ycc = np.asarray(Image.fromarray(synth_rgb(w, h, 9), "RGB").convert("YCbCr")).transpose(2, 0, 1).copy()
    q = O.quant_table(80)
    b = io.BytesIO()
    Image.fromarray(ycc.transpose(1, 2, 0), "YCbCr").save(b, "JPEG", qtables=[list(map(int, q))] * 2, subsampling=ss)
    turbo = O.Jpeg(b.getvalue())
    mine = O.forward(ycc, O.params(80, ssn, False))
    for c in range(3):
        assert np.array_equal(turbo.coef(c), mine.coef(c))


def test_writer_roundtrip_and_independent_decoder(O, golden):
    data = golden("in_420_base_355x237.jpg")
    for prog in (False, True):
        for ss in (420, 444, 422, 411):
            out = O.jpeg_lossy(data, O.params(80, ss, prog))
            assert np.array_equal(O.Jpeg(out).decode_native(), pillow_native(out))   # libjpeg-turbo reads what we write
    # lossless: coefficients survive, pixels identical
    j = O.Jpeg(data)
    for prog in (False, True):
        out = O.jpeg_lossless(data, O.params(80, 0, prog))
        j2 = O.Jpeg(out)
        for c in range(3):
            assert np.array_equal(j.coef(c)[:j.s.rbh[c], :j.s.rbw[c]], j2.coef(c)[:j.s.rbh[c], :j.s.rbw[c]])
        assert np.array_equal(pillow_native(out), pillow_native(data))


def test_golden_vectors(O, golden):
    exp = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "expected.json")))
    for name, e in exp.items():
        data = golden(name)
        assert hashlib.sha256(data).hexdigest() == e["input_sha256"]
        for key, v in e["lossy"].items():
            q, ss, p = key.split("_")
            out = O.jpeg_lossy(data, O.params(int(q[1:]), int(ss[1:]), bool(int(p[1:]))))
            assert (len(out), hashlib.sha256(out).hexdigest()) == (v["size"], v["sha256"]), (name, key)
        for key, v in e["lossless"].items():
            out = O.jpeg_lossless(data, O.params(80, 0, bool(int(key[1:]))))
            assert hashlib.sha256(out).hexdigest() == v["sha256"]


def test_reference_test_suite_size_bounds(O):
    """The only numbers the reference's tests pin (compressor.rs:1051-1068): j0@q95 > 391,657 B, j0@q50 < 790,435 B."""
    data = open(os.path.join(REF, "j0.JPG"), "rb").read()
    assert len(O.jpeg_lossy(data, O.params(95, 0, True))) > 391657
    assert len(O.jpeg_lossy(data, O.params(50, 0, True))) < 790435
    assert len(O.jpeg_lossy(data, O.params(100, 0, True))) >= len(O.jpeg_lossy(data, O.params(80, 0, True)))


def test_block_primitives_against_float_dct(O):
    """ISLOW integer DCT pair vs an orthonormal float DCT: within the fixed-point error budget (<= 1 LSB after round trip)."""
    rng = np.random.default_rng(3)
    k = np.arange(8)
    C = np.sqrt(2 / 8) * np.cos((2 * k[None, :] + 1) * k[:, None] * np.pi / 16)
    C[0] /= np.sqrt(2)
    q1 = np.ones(64, dtype=np.uint16)
    for _ in range(50):
        px = rng.integers(0, 256, size=(8, 8)).astype(np.uint8)
        dct, qz = O.fdct_quant(px, q1)
        ref = C @ (px.astype(np.float64) - 128) @ C.T
        assert np.abs(dct / 8.0 - ref).max() < 1.0
        back = O.idct_islow(qz.reshape(64), q1)
        assert np.abs(back.astype(int) - px.astype(int)).max() <= 1
