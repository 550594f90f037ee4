"""CPU tests of the PNG lossless leg (SURVEY.md §8 row a8): the oracle restatement (oracle/png_oracle.c) pinned against
Pillow/libpng + zlib, and the product's HOST half (container parse, inflate, unfilter, DEFLATE writer) through the C-ABI.
No device work is called here."""
import io
import os
import zlib

import numpy as np
import pytest

from pngutil import frame_png, idat_stream, pil_pixels, pil_png, synth

P0_FILTER_HISTOGRAM = [3, 28, 211, 8, 150]      # per-row filter types 0..4 of the reference's samples/p0.png (known answer)

CT = {1: 0, 2: 4, 3: 2, 4: 6}     # channels -> PNG colour type


@pytest.mark.parametrize("channels", [1, 2, 3, 4])
@pytest.mark.parametrize("strategy", range(10))
def test_oracle_filter_is_lossless_and_libpng_agrees(O, channels, strategy):
    img = synth(37, 53, channels, seed=strategy * 7 + channels, kind="photo" if strategy % 2 else "flat")
    raw = img.reshape(37, 53 * channels)
    filt = O.png_filter(raw, channels, strategy)
    if strategy < 5:
        assert (filt[:, 0] == strategy).all()
    assert filt[:, 0].max() <= 4
    assert np.array_equal(O.png_unfilter(filt, channels), raw)
    # libpng (through Pillow) must reconstruct the same pixels from the oracle's filtered rows
    png = frame_png(53, 37, 8, CT[channels], zlib.compress(filt.tobytes(), 6))
    got = np.asarray(pil_pixels(png)).reshape(37, 53 * channels)
    assert np.array_equal(got, raw)


def test_oracle_heuristics_pick_the_expected_filter(O):
    # a horizontal ramp is constant under Sub; a vertical ramp under Up
    x = np.tile(np.arange(200, dtype=np.uint8) * 1, (20, 1))
    y = np.tile((np.arange(20, dtype=np.uint8) * 3)[:, None], (1, 200))
    for s in ("minsum", "entropy", "bigrams", "bigent", "brute"):
        f = O.png_filter(x, 1, O.PNG_STRATEGIES[s])
        assert (f[1:, 0] != 0).all(), s                # never None on a ramp (rows after the first may also pick Up/Paeth)
    # constant rows: byte statistics cannot tell the filters apart except MinSum, which must leave None behind
    assert (O.png_filter(y, 1, O.PNG_STRATEGIES["minsum"])[2:, 0] != 0).all()
    # all-zero rows: every filter ties, the first (None) wins
    z = np.zeros((5, 64), dtype=np.uint8)
    for s in range(5, 10):
        assert (O.png_filter(z, 1, s)[:, 0] == 0).all()


@pytest.mark.parametrize("kind,channels", [("photo", 3), ("flat", 3), ("flat", 1), ("noise", 4), ("photo", 2)])
def test_oracle_lz77_round_trips(O, kind, channels):
    img = synth(64, 97, channels, seed=3, kind=kind)
    filt = O.png_filter(img.reshape(64, -1), channels, O.PNG_STRATEGIES["paeth" if kind == "photo" else "none"])
    stream = filt.reshape(-1)
    tok, hist = O.png_lz77(stream, channels, filt.shape[1])
    assert np.array_equal(O.png_expand(tok, stream.size), stream)
    lits = tok[tok < 0x80000000]
    assert hist[:256].sum() == lits.size and hist[257:286].sum() == (tok >= 0x80000000).sum() == hist[286:].sum()
    if kind == "flat":
        assert tok.size < stream.size // 4              # flat art must compress
    if kind == "noise":
        assert tok.size > stream.size * 0.9


def test_host_deflate_writer_round_trips_through_zlib(L, O):
    for kind, channels in (("photo", 3), ("flat", 4), ("noise", 1)):
        img = synth(80, 120, channels, seed=11, kind=kind)
        filt = O.png_filter(img.reshape(80, -1), channels, 4)
        stream = filt.reshape(-1)
        tok, _ = O.png_lz77(stream, channels, filt.shape[1])
        z = L.png_deflate_tokens(tok, zlib.adler32(stream.tobytes()))
        assert zlib.decompress(z) == stream.tobytes()
        if kind != "noise":
            assert len(z) < stream.size
    # empty token stream is still a valid zlib stream
    assert zlib.decompress(L.png_deflate_tokens(np.zeros(0, np.uint32), 1)) == b""


def test_host_deflate_writer_many_blocks(L, O):
    rng = np.random.default_rng(5)
    stream = rng.integers(0, 7, 300000).astype(np.uint8)        # > 4 blocks of 65536 tokens
    tok, _ = O.png_lz77(stream, 1, 1000)
    z = L.png_deflate_tokens(tok, zlib.adler32(stream.tobytes()))
    assert zlib.decompress(z) == stream.tobytes()


def test_host_deflate_writer_every_distance_and_length(L):
    """every match distance 1..32768 and every length 3..258 through the writer (closed-form distance codes, merged code + extra-bit
    pieces, branch-free bit packing): the stream must inflate to what the tokens say"""
    rng = np.random.default_rng(17)
    head = rng.integers(0, 256, 32768).astype(np.uint8)
    tok = list(head.astype(np.uint32))
    out = bytearray(head.tobytes())
    for d in range(1, 32769):
        ln = 3 + (d * 7) % 256
        tok.append(0x80000000 | ((ln - 3) << 16) | (d - 1))
        for _ in range(ln):
            out.append(out[-d])
        if d % 5 == 0:
            tok.append(int(d & 255)); out.append(d & 255)
    for ln in range(3, 259):
        tok.append(0x80000000 | ((ln - 3) << 16) | (4 - 1))
        for _ in range(ln):
            out.append(out[-4])
    z = L.png_deflate_tokens(np.array(tok, dtype=np.uint32), zlib.adler32(bytes(out)))
    assert zlib.decompress(z) == bytes(out)


@pytest.mark.parametrize("mode", ["L", "LA", "RGB", "RGBA", "P", "1", "I;16", "L2", "L4"])
def test_host_png_decode_matches_pillow(L, mode):
    from PIL import Image
    rng = np.random.default_rng(9)
    h, w = 45, 67
    if mode in ("L", "LA", "RGB", "RGBA"):
        ch = {"L": 1, "LA": 2, "RGB": 3, "RGBA": 4}[mode]
        arr = synth(h, w, ch, seed=2)
        png = pil_png(arr)
        info, raw = L.png_decode(png)
        assert (info.width, info.height, info.bit_depth, info.color_type, info.bpp, info.row_bytes) == (w, h, 8, CT[ch], ch, w * ch)
        assert np.array_equal(raw, arr.reshape(h, w * ch))
    elif mode == "P":
        idx = rng.integers(0, 16, (h, w)).astype(np.uint8)
        im = Image.fromarray(idx, mode="P"); im.putpalette([int(v) for v in rng.integers(0, 256, 48)])
        info, raw = L.png_decode(pil_png(im))
        assert info.color_type == 3
        bits = info.bit_depth
        # unpack and compare the indices
        un = np.unpackbits(raw, axis=1).reshape(h, -1, bits)
        vals = (un * (1 << np.arange(bits - 1, -1, -1))).sum(-1)[:, :w]
        assert np.array_equal(vals, idx)
    elif mode == "1":
        b = rng.integers(0, 2, (h, w)).astype(bool)
        info, raw = L.png_decode(pil_png(Image.fromarray(b)))
        assert (info.bit_depth, info.color_type, info.row_bytes) == (1, 0, (w + 7) // 8)
        assert np.array_equal(np.unpackbits(raw, axis=1)[:, :w].astype(bool), b)
    elif mode == "I;16":
        a = rng.integers(0, 65536, (h, w)).astype(np.uint16)
        info, raw = L.png_decode(pil_png(Image.fromarray(a)))
        assert (info.bit_depth, info.color_type, info.bpp, info.row_bytes) == (16, 0, 2, 2 * w)
        assert np.array_equal(raw.reshape(h, w, 2)[:, :, 0].astype(np.uint16) * 256 + raw.reshape(h, w, 2)[:, :, 1], a)
    else:
        bits = int(mode[1])
        vals = rng.integers(0, 1 << bits, (h, w)).astype(np.uint8)
        packed = np.packbits(np.unpackbits(vals[:, :, None], axis=2)[:, :, 8 - bits:].reshape(h, -1), axis=1)
        rows = np.concatenate([np.zeros((h, 1), np.uint8), packed], axis=1)
        png = frame_png(w, h, bits, 0, zlib.compress(rows.tobytes()))
        info, raw = L.png_decode(png)
        assert (info.bit_depth, info.bpp, info.row_bytes) == (bits, 1, packed.shape[1])
        assert np.array_equal(raw, packed)


def test_host_png_decode_every_filter_type_and_split_idat(L, O):
    import struct
    from pngutil import chunk
    img = synth(33, 41, 3, seed=4)
    raw = img.reshape(33, -1)
    # rows cycle through the five filter types; IDAT split into many small chunks; stored + fixed + dynamic blocks
    rows = np.stack([O.png_filter(raw, 3, y % 5)[y] for y in range(33)])
    for level in (0, 1, 9):
        z = zlib.compress(rows.tobytes(), level)
        parts = b"".join(chunk(b"IDAT", z[i:i + 100]) for i in range(0, len(z), 100))
        png = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 41, 33, 8, 2, 0, 0, 0)) + parts + chunk(b"IEND", b"")
        _, got = L.png_decode(png)
        assert np.array_equal(got, raw)


def test_host_png_decode_rejects_bad_input(L):
    good = pil_png(synth(16, 16, 3))
    flipped = good[:60] + bytes([good[60] ^ 0x55]) + good[61:]
    for bad, code in ((good[:40], 4), (flipped, 4), (b"\x89PNG\r\n\x1a\n" + b"\0" * 40, 4)):
        with pytest.raises(L.B200Error) as e:
            L.png_decode(bad)
        assert e.value.code == code, e.value
    # Adam7: hand-made header with the interlace byte set must be refused as unsupported (code 3), not mis-decoded
    import struct
    from pngutil import chunk
    png = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", 4, 4, 8, 0, 0, 0, 1)) + chunk(b"IDAT", zlib.compress(b"\0" * 64)) + chunk(b"IEND", b"")
    with pytest.raises(L.B200Error) as e:
        L.png_decode(png)
    assert e.value.code == 3


def test_png_level_strategy_sets(L):
    assert L.png_level_strategies(0) == [0]
    for lvl in range(1, 7):
        s = L.png_level_strategies(lvl)
        assert s[0] == 0 and len(set(s)) == len(s) and all(0 <= v <= 9 for v in s)
    assert len(L.png_level_strategies(6)) > len(L.png_level_strategies(3)) > len(L.png_level_strategies(1))


def test_idat_helper_on_pillow_file():
    ihdr, idat, order = idat_stream(pil_png(synth(8, 8, 3)))
    assert ihdr[:2] == (8, 8) and order[0] == b"IHDR" and order[-1] == b"IEND" and len(zlib.decompress(idat)) == 8 * 25


def _unpack(raw, depth, width):
    """packed PNG index rows (MSB first) -> [h, width] indices"""
    if depth == 8:
        return raw[:, :width]
    per = 8 // depth
    shifts = (8 - depth - depth * np.arange(per)).astype(np.uint8)
    return ((raw[:, :, None] >> shifts) & ((1 << depth) - 1)).reshape(raw.shape[0], -1)[:, :width]


def test_palette_reduction_is_lossless_and_declines_when_it_should(L):
    """oxipng reduction::palette on the host: <= 256 distinct RGB / RGBA pixels -> 8-bit indices + PLTE (+ tRNS, non-opaque
    entries first); photographs, grey images, inputs with tRNS / 16-bit / palette stay as decoded."""
    from PIL import Image
    rng = np.random.default_rng(21)
    # flat art, RGB and RGBA (with partly transparent colours)
    for ch in (3, 4):
        img = synth(90, 140, ch, seed=5 + ch, kind="flat")
        if ch == 4:
            img[10:30, 20:60, 3] = 0; img[40:50, :, 3] = 128
        info, raw, pal = L.png_decode_reduced(pil_png(img))
        n = len(np.unique(img.reshape(-1, ch), axis=0))
        depth = 1 if n <= 2 else 2 if n <= 4 else 4 if n <= 16 else 8
        assert pal is not None and info.color_type == 3 and info.bit_depth == depth and info.bpp == 1 and info.row_bytes == (140 * depth + 7) // 8
        assert len(pal) == n <= 256
        rgba = pal[_unpack(raw, info.bit_depth, 140)]               # [h, w, 4]
        want = img if ch == 4 else np.concatenate([img, np.full((90, 140, 1), 255, np.uint8)], axis=2)
        assert np.array_equal(rgba, want)
        a = pal[:, 3]
        assert np.all(a[:np.count_nonzero(a != 255)] != 255)       # the non-opaque entries lead
    # 2, 4, 16, 17 colours -> 1, 2, 4, 8 bits per index; odd widths pad the last byte of a row
    for n, depth in ((2, 1), (3, 2), (4, 2), (5, 4), (16, 4), (17, 8)):
        cols = rng.integers(0, 256, (n, 3)).astype(np.uint8); cols[:, 0] = np.arange(n)       # distinct, not grey
        cols[:, 1] = 255 - cols[:, 0]
        img = cols[rng.integers(0, n, (23, 37))]
        img.reshape(-1, 3)[:n] = cols
        info, raw, pal = L.png_decode_reduced(pil_png(img))
        assert pal is not None and info.bit_depth == depth and info.row_bytes == (37 * depth + 7) // 8 and len(pal) == n
        assert np.array_equal(pal[_unpack(raw, depth, 37)][:, :, :3], img)
    # exactly 256 colours still fits, 257 does not
    cols = rng.permutation(256 * 256)[:257]
    base = np.stack([cols % 256, cols // 256, (cols * 7) % 256], axis=1).astype(np.uint8)
    for n, expect in ((256, True), (257, False)):
        img = base[rng.integers(0, n, (64, 64))]
        img.reshape(-1, 3)[:n] = base[:n]
        info, raw, pal = L.png_decode_reduced(pil_png(img))
        assert (pal is not None) == expect
        if expect:
            assert np.array_equal(pal[raw][:, :, :3], img)
        else:
            assert info.color_type == 2 and np.array_equal(raw.reshape(64, 64, 3), img)
    # declined: photograph, grey RGB (left to the grey reduction), grey+alpha, 16-bit, palette input, RGB with a tRNS colour
    assert L.png_decode_reduced(pil_png(synth(50, 60, 3, seed=1)))[2] is None
    g = synth(50, 60, 1, seed=2, kind="flat")
    assert L.png_decode_reduced(pil_png(np.repeat(g, 3, axis=2)))[2] is None
    assert L.png_decode_reduced(pil_png(np.concatenate([g, g], axis=2)))[2] is None
    assert L.png_decode_reduced(pil_png(Image.fromarray((g[:, :, 0].astype(np.uint16) * 257))))[2] is None
    im = Image.fromarray((g[:, :, 0] % 4).astype(np.uint8), mode="P"); im.putpalette([0, 0, 0, 255, 0, 0, 0, 255, 0, 0, 0, 255])
    assert L.png_decode_reduced(pil_png(im))[2] is None
    b = io.BytesIO(); Image.fromarray(synth(30, 30, 3, seed=3, kind="flat")).save(b, format="PNG", transparency=(255, 255, 255))
    assert L.png_decode_reduced(b.getvalue())[2] is None
    # a single pixel, and a single colour
    info, raw, pal = L.png_decode_reduced(pil_png(np.array([[[9, 200, 30]]], dtype=np.uint8)))
    assert pal is not None and np.array_equal(pal, [[9, 200, 30, 255]]) and raw.tolist() == [[0]] and info.bit_depth == 1


def test_reference_fixture_p0_png_known_answers(L, O):
    """SURVEY.md §8c KAT-4 on the reference's own fixture (its copy in tests/golden/reference_samples): one IDAT
    that inflates to 480,400 bytes (400 rows of 400 RGB pixels + filter bytes); the product's host decoder and the oracle's
    unfilter must both reproduce libpng's pixels; the file's row-filter histogram is the known answer recorded here."""
    data = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_samples", "p0.png"), "rb").read()
    ihdr, idat, order = idat_stream(data)
    assert ihdr[:5] == (400, 400, 8, 2, 0) and order.count(b"IDAT") == 1
    filt = np.frombuffer(zlib.decompress(idat), dtype=np.uint8)
    assert filt.size == 480400
    rows = filt.reshape(400, 1201)
    assert np.bincount(rows[:, 0], minlength=5).tolist() == P0_FILTER_HISTOGRAM
    want = np.asarray(pil_pixels(data).convert("RGB"))
    info, raw = L.png_decode(data)
    assert (info.width, info.height, info.bit_depth, info.color_type, info.bpp, info.row_bytes) == (400, 400, 8, 2, 3, 1200)
    assert np.array_equal(raw.reshape(400, 400, 3), want)
    assert np.array_equal(O.png_unfilter(rows, 3).reshape(400, 400, 3), want)
