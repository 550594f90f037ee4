"""CPU tests of the C++ host mirror of compressor.rs (caesium-clt_b200/csrc/compressor.cpp), modelled on the
reference's own inline unit tests (/root/reference/src/compressor.rs:607-1109, options.rs:259-452).  The codec call
used here is --lossless JPEG, the one path that is host-only by design (coefficient-domain transcode), so these run
without a GPU; the lossy variants of the same flows are in test_cli_gpu.py."""
import ctypes as C
import io
import json
import os
import subprocess

import pytest
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "caesium-clt_b200")


class Opt(C.Structure):
    _fields_ = [("quality", C.c_int), ("max_size", C.c_longlong), ("lossless", C.c_int), ("exif", C.c_int), ("png_opt_level", C.c_int), ("zopfli", C.c_int),
                ("width", C.c_int), ("height", C.c_int), ("long_edge", C.c_int), ("short_edge", C.c_int),
                ("output_folder", C.c_char_p), ("same_folder_as_input", C.c_int), ("base_path", C.c_char_p), ("suffix", C.c_char_p),
                ("overwrite_policy", C.c_int), ("format", C.c_int), ("keep_dates", C.c_int), ("keep_structure", C.c_int),
                ("jpeg_chroma_subsampling", C.c_uint), ("jpeg_baseline", C.c_int), ("no_upscale", C.c_int), ("strip_icc", C.c_int), ("min_savings", C.c_char_p)]


def setup_options(**kw):
    o = Opt(quality=80, max_size=-1, lossless=0, exif=0, png_opt_level=3, zopfli=0, width=-1, height=-1, long_edge=-1, short_edge=-1,
            output_folder=None, same_folder_as_input=0, base_path=b"", suffix=None, overwrite_policy=0, format=5, keep_dates=0, keep_structure=0,
            jpeg_chroma_subsampling=0, jpeg_baseline=0, no_upscale=0, strip_icc=0, min_savings=None)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


@pytest.fixture(scope="module")
def H(L):
    return C.CDLL(os.path.join(PKG, "libb200clt.so"))


def jpeg_bytes(w, h, exif_orientation=None):
    b = io.BytesIO()
    im = Image.new("RGB", (w, h), (120, 60, 200))
    kw = {}
    if exif_orientation:
        ex = Image.Exif()
        ex[0x0112] = exif_orientation
        kw["exif"] = ex
    im.save(b, "JPEG", quality=90, **kw)
    return b.getvalue()


def build_params(H, L, opt, buf):
    p = L.Params()
    err = C.create_string_buffer(256)
    rc = H.b200clt_build_compression_parameters(C.byref(opt), buf, C.c_size_t(len(buf)), C.byref(p), err, C.c_size_t(256))
    return rc, p, err.value.decode()


def test_build_compression_parameters_mapping(H, L):
    """compressor.rs:411-446 and main.rs tests :403-430."""
    buf = jpeg_bytes(64, 48)
    rc, p, _ = build_params(H, L, setup_options(quality=55, exif=1, strip_icc=1, jpeg_baseline=1, jpeg_chroma_subsampling=422, png_opt_level=5, zopfli=1), buf)
    assert rc == 0
    assert (p.jpeg_quality, p.png_quality, p.webp_quality, p.gif_quality) == (55, 55, 55, 55)
    assert (p.keep_metadata, p.jpeg_preserve_icc, p.jpeg_progressive, p.jpeg_chroma_subsampling) == (1, 0, 0, 422)
    assert (p.png_optimization_level, p.png_force_zopfli, p.jpeg_optimize, p.png_optimize, p.webp_lossless) == (5, 1, 0, 0, 0)
    rc, p, _ = build_params(H, L, setup_options(quality=-1, lossless=1), buf)
    assert (p.jpeg_quality, p.gif_quality, p.jpeg_optimize, p.png_optimize, p.webp_lossless) == (80, 100, 1, 1, 1)
    rc, p, _ = build_params(H, L, setup_options(quality=0), buf)      # gif quality 0 -> 1 (compressor.rs:986-1010)
    assert (p.jpeg_quality, p.gif_quality) == (0, 1)


def test_build_resize_parameters(H, L):
    """compressor.rs:933-983 on a portrait JPEG like samples/j0.JPG (2000x3000)."""
    buf = jpeg_bytes(200, 300)
    for kw, exp in [(dict(width=100, height=100), (100, 100)), (dict(width=100), (100, 0)), (dict(height=100), (0, 100)),
                    (dict(long_edge=100), (0, 100)), (dict(short_edge=50), (50, 0)), (dict(no_upscale=1, width=20000), (0, 0))]:
        rc, p, _ = build_params(H, L, setup_options(**kw), buf)
        assert rc == 0 and (p.width, p.height) == exp, kw
    land = jpeg_bytes(300, 200)
    rc, p, _ = build_params(H, L, setup_options(long_edge=100), land)
    assert (p.width, p.height) == (100, 0)
    rc, p, _ = build_params(H, L, setup_options(short_edge=50), land)
    assert (p.width, p.height) == (0, 50)


def test_no_upscale_prevents_resize(H, L):
    """compressor.rs:898-931."""
    w, h = 120, 80
    buf = jpeg_bytes(w, h)
    for kw in (dict(width=w + 100), dict(height=h + 100), dict(long_edge=max(w, h) + 100), dict(short_edge=min(w, h) + 100)):
        rc, p, _ = build_params(H, L, setup_options(no_upscale=1, **kw), buf)
        assert rc == 0 and (p.width, p.height) == (0, 0)


def test_exif_orientation_swaps_resolution(H, L):
    """get_real_resolution (compressor.rs:538-561): orientation 5..8 swaps w/h only when metadata is kept."""
    buf = jpeg_bytes(300, 200, exif_orientation=6)
    rc, p, _ = build_params(H, L, setup_options(long_edge=100, exif=1), buf)
    assert (p.width, p.height) == (0, 100)          # treated as portrait
    rc, p, _ = build_params(H, L, setup_options(long_edge=100, exif=0), buf)
    assert (p.width, p.height) == (100, 0)
    rc, _, err = build_params(H, L, setup_options(width=10), b"not an image")
    assert rc == 1 and err


def test_compute_output_full_path(H, tmp_path):
    """compressor.rs:615-766, all ten cases."""
    out = tmp_path / "output"
    base = tmp_path / "base"
    folder = base / "folder"
    out.mkdir()
    folder.mkdir(parents=True)

    def run(inp, keep, fmt, same=0, basedir=base):
        d, n = C.create_string_buffer(1024), C.create_string_buffer(1024)
        rc = H.b200clt_compute_output_full_path(str(out).encode(), str(inp).encode(), str(basedir).encode(), keep, b"_suffix", fmt, same, d, n, C.c_size_t(1024))
        assert rc == 0
        return d.value.decode(), n.value.decode()

    assert run(folder / "test.jpg", 1, 5) == (str(out / "folder"), "test_suffix.jpg")
    assert run(folder / "test.jpg", 0, 5) == (str(out), "test_suffix.jpg")
    assert run(folder / "test", 0, 5) == (str(out), "test_suffix")
    other = tmp_path / "different_base" / "folder"
    other.mkdir(parents=True)
    assert run(other / "test.jpg", 0, 5) == (str(out), "test_suffix.jpg")
    for fmt, ext in [(0, "jpg"), (1, "png"), (3, "webp"), (4, "tiff"), (2, "gif")]:
        assert run(other / "test.jpg", 0, fmt) == (str(out), f"test_suffix.{ext}")
    sub = folder / "subfolder"
    sub.mkdir()
    assert run(sub / "test.jpg", 1, 5, same=1) == (str(sub), "test_suffix.jpg")


def test_min_savings_parser(H):
    """options.rs:388-451."""
    def parse(s):
        ip, pc, by = C.c_int(), C.c_double(), C.c_ulonglong()
        rc = H.b200clt_parse_min_savings(s.encode(), C.byref(ip), C.byref(pc), C.byref(by))
        return None if rc else (("pct", pc.value) if ip.value else ("bytes", by.value))
    assert parse("10%") == ("pct", 10.0) and parse("0%") == ("pct", 0.0) and parse("100%") == ("pct", 100.0) and parse("1.5%") == ("pct", 1.5)
    assert parse("100KB") == ("bytes", 100_000) and parse("1MB") == ("bytes", 1_000_000) and parse("1MiB") == ("bytes", 1_048_576)
    assert parse("1B") == ("bytes", 1) and parse("100") == ("bytes", 100) and parse("1KiB") == ("bytes", 1024)
    assert parse("101%") is None and parse("-5%") is None and parse("") is None and parse("abc") is None


def _cli(*args):
    r = subprocess.run([os.path.join(PKG, "b200clt"), *args], capture_output=True, text=True)
    return r.returncode, r.stdout, r.stderr


def _tree(tmp_path, golden):
    src = tmp_path / "in"
    (src / "level_1" / "level_2").mkdir(parents=True)
    (src / "a.jpg").write_bytes(golden("in_420_base_355x237.jpg"))
    (src / "level_1" / "b.JPG").write_bytes(golden("in_444_base_355x237.jpg"))
    (src / "level_1" / "level_2" / "c.jpeg").write_bytes(golden("in_420_prog_355x237.jpg"))
    (src / "notes.txt").write_text("not an image")
    (src / "fake.jpg").write_text("extension lies")
    return src


def test_cli_lossless_tree_structure_policies_and_json(L, golden, tmp_path):
    """test_perform_compression (compressor.rs:769-896) shape: all Success, exact output paths with / without
    keep_structure, Never/Bigger overwrite policies, dry-run, keep-dates, and the JSON schema of main.rs:643-727."""
    src = _tree(tmp_path, golden)
    out = tmp_path / "out"
    rc, so, _ = _cli("--lossless", "-o", str(out), "-R", "-S", "--json", "--keep-dates", str(src))
    assert rc == 0
    d = json.loads(so)
    assert d["version"] == "1.0.0" and d["dry_run"] is False and d["error"] is None
    assert d["summary"]["total_files"] == 3 and d["summary"]["success"] == 3 and d["summary"]["errors"] == 0
    outs = sorted(f["output_path"] for f in d["files"])
    assert outs == sorted([str(out / "a.jpg"), str(out / "level_1" / "b.JPG"), str(out / "level_1" / "level_2" / "c.jpeg")])
    for f in d["files"]:
        assert os.path.getsize(f["output_path"]) == f["compressed_size"]
        assert abs(os.path.getmtime(f["output_path"]) - os.path.getmtime(f["original_path"])) < 1e-3      # keep_dates
        assert set(f) == {"original_path", "output_path", "original_size", "compressed_size", "status", "message"}
    assert d["summary"]["savings_bytes"] == d["summary"]["original_size"] - d["summary"]["compressed_size"]
    # flat (no keep_structure), with suffix
    flat = tmp_path / "flat"
    rc, so, _ = _cli("--lossless", "-o", str(flat), "-R", "--suffix", "_x", "--json", str(src))
    assert sorted(os.listdir(flat)) == ["a_x.jpg", "b_x.JPG", "c_x.jpeg"]
    # overwrite never -> all skipped; bigger -> skipped because the existing files are not larger
    for pol in ("never", "bigger"):
        rc, so, _ = _cli("--lossless", "-o", str(out), "-R", "-S", "--json", "-O", pol, str(src))
        d2 = json.loads(so)
        assert d2["summary"]["skipped"] == 3
        assert all(f["message"] == "File already exists, skipped due overwrite policy" and f["compressed_size"] == f["original_size"] for f in d2["files"])
    # dry run writes nothing
    dry = tmp_path / "dry"
    rc, so, _ = _cli("--lossless", "-o", str(dry), "-R", "--dry-run", "--json", str(src))
    d3 = json.loads(so)
    assert d3["dry_run"] is True and d3["summary"]["success"] == 3 and not dry.exists()
    # non-recursive scan sees only the top level; the fake .jpg is rejected by the magic sniff (scan_files.rs:30-40)
    rc, so, _ = _cli("--lossless", "-o", str(tmp_path / "top"), "--json", str(src))
    assert json.loads(so)["summary"]["total_files"] == 1


def test_cli_min_savings_and_same_folder(L, golden, tmp_path):
    """test_min_savings_skips_files (compressor.rs:1013-1080) on the host-only path."""
    src = _tree(tmp_path, golden)
    rc, so, _ = _cli("--lossless", "--same-folder-as-input", "--suffix", "_c", "-R", "--json", "--min-savings", "99%", str(src))
    d = json.loads(so)
    assert d["summary"]["skipped"] == 3 and all(f["message"].startswith("Insufficient savings: ") and f["message"].endswith("%, skipped") for f in d["files"])
    rc, so, _ = _cli("--lossless", "--same-folder-as-input", "--suffix", "_c", "-R", "--json", "--min-savings", "1B", str(src))
    d = json.loads(so)
    assert d["summary"]["success"] == 3 and (src / "a_c.jpg").exists() and (src / "level_1" / "b_c.JPG").exists()


def test_cli_many_files_cross_the_batch_chunks_in_order(L, golden, tmp_path):
    """start_compression hands the codec calls to b200_compress_batch in chunks of 256 files: 300 files (two chunks, several
    sizes, one unreadable entry in the middle) must come back complete and in input order, each output equal to the single call.
    The scan sniffs every file's first bytes and leaves out one it cannot read (scan_files.rs:18-40); root reads it anyway."""
    src = tmp_path / "in"; src.mkdir()
    names = ["in_420_base_355x237.jpg", "in_444_base_355x237.jpg", "in_420_prog_355x237.jpg", "in_gray_base_355x237.jpg"]
    for i in range(300):
        (src / f"f{i:03d}.jpg").write_bytes(golden(names[i % 4]))
    os.chmod(src / "f130.jpg", 0)
    listed = [f"f{i:03d}.jpg" for i in range(300) if i != 130 or os.access(src / "f130.jpg", os.R_OK)]
    out = tmp_path / "out"
    rc, so, _ = _cli("--lossless", "-o", str(out), "--json", str(src))
    d = json.loads(so)
    assert d["summary"]["total_files"] == len(listed)
    assert [os.path.basename(f["original_path"]) for f in d["files"]] == listed
    p = L.default_params(); p.jpeg_optimize = 1
    want = {n: L.compress_in_memory(golden(n), p) for n in names}
    bad = [f for f in d["files"] if f["status"] != "success"]
    assert len(bad) <= 1 and all(os.path.basename(f["original_path"]) == "f130.jpg" and f["message"] == "Error reading input file" for f in bad)
    for i in (0, 1, 2, 3, 255, 256, 257, 299):
        assert (out / f"f{i:03d}.jpg").read_bytes() == want[names[i % 4]]


def test_cli_flag_groups(L):
    """options.rs:141,181: exactly one compression mode and one destination."""
    assert _cli("-o", "/tmp/x", "f.jpg")[0] == 2
    assert _cli("-q", "80", "--lossless", "-o", "/tmp/x", "f.jpg")[0] == 2
    assert _cli("-q", "80", "f.jpg")[0] == 2
    assert _cli("-q", "101", "-o", "/tmp/x", "f.jpg")[0] == 2
    assert _cli("--lossless", "--png-opt-level", "7", "-o", "/tmp/x", "f.jpg")[0] == 2


def test_lossy_cli_fails_loudly_without_gpu(L, golden, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible")
    src = _tree(tmp_path, golden)
    rc, so, _ = _cli("-q", "80", "-o", str(tmp_path / "o"), "-R", "--json", str(src))
    d = json.loads(so)
    assert d["summary"]["errors"] == 3 and all("no CUDA device" in f["message"].lower() or "[5]" in f["message"] for f in d["files"])
