#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: megapixels/s, JPEG q=80 4:2:0 re-encode of 3840x2160 inputs (configs[1]), plus one
sub-record per other GPU workload of BASELINE.json (configs[2..4]) under "configs" in the same JSON line.

One "step" = one pass of the hot path over one batch of synthetic inputs.
  value : the FULL device path with the inputs resident in HBM -- entropy-coded scan bytes in HBM -> Huffman decode ->
          dequant/IDCT/chroma resample/FDCT/quantise -> Huffman encode (optimal tables, progressive script, byte stuffing) ->
          entropy-coded scan bytes in HBM (b200_jpeg_pipe_*), timed with CUDA events on the launching stream, max over ranks.
  e2e   : the same metric through the reference-facing C-ABI (b200_compress_batch: JPEG file bytes in host memory -> JPEG file
          bytes in host memory; marker parsing, pinned H2D, the same kernels, D2H, file assembly inside the timed region).
  roofline : per-kernel table from one megabatch run alone with an event after every launch; the headline entry is the kernel
          with the longest launch; `path` is the whole device path on SURVEY 8d's fused 6 B/pixel figure.
  cpu_baseline / --impl reference : the CPU restatement of the reference path (oracle/, "port": the Rust reference cannot be
          built in this image) on the box's usable host cores.
Launch: python bench.py [--gpus N --steps K --warmup W] or torchrun --nproc-per-node N bench.py --gpus N ...
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the library drives one CUDA stream per in-flight megabatch; give them separate hardware queues (must precede CUDA init,
# and torch may create the context before the library does)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line

W4K, H4K = 3840, 2160
MP_PER_IMAGE = W4K * H4K / 1e6
QUALITY, SUBSAMPLING = 80, 420
METRIC = "megapixels/sec JPEG q=80 4K re-encode"


def usable_cores():
    n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, -(-int(q) // int(p))))
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


# ---- synthetic inputs (seeded; SURVEY.md 8d) -----------------------------------------------------------------------------------
def _gen_one(job):
    kind, idx = job
    from tools import synth
    if kind == "jpeg4k":
        return synth.synth_jpeg(W4K, H4K, idx)
    if kind == "jpeg24mp":
        return synth.synth_jpeg(6000, 4000, idx)
    if kind == "png4096":
        return synth.synth_png_rgba(4096, 4096, idx)
    raise ValueError(kind)


def make_inputs(n_unique, first_index, kind="jpeg4k", procs=None, indices=None):
    """n_unique seeded sources: 4K JPEGs (q=90, 4:2:0, baseline, Annex-K tables via Pillow/libjpeg-turbo), 6000x4000 JPEGs of
    the same kind, or 4096x4096 RGBA PNGs (Paeth rows, zlib level 6).  indices: explicit seed indices (a rank's shard)."""
    import multiprocessing as mp
    if indices is not None:
        n_unique = len(indices)
    procs = min(n_unique, procs or usable_cores())
    jobs = [(kind, i) for i in indices] if indices is not None else [(kind, first_index + i) for i in range(n_unique)]
    if procs <= 1:
        return [_gen_one(j) for j in jobs]
    with mp.get_context("fork").Pool(procs) as pool:
        return pool.map(_gen_one, jobs)


def load_pkg_shallow():
    """register the package (its directory name is not an identifier) without loading the shared library"""
    pkg_dir = os.path.join(ROOT, "caesium-clt_b200")
    if "caesium_clt_b200" not in sys.modules:
        spec = importlib.util.spec_from_file_location("caesium_clt_b200", os.path.join(pkg_dir, "__init__.py"), submodule_search_locations=[pkg_dir])
        mod = importlib.util.module_from_spec(spec)
        sys.modules["caesium_clt_b200"] = mod
        spec.loader.exec_module(mod)


def load_pkg():
    load_pkg_shallow()
    import caesium_clt_b200._lib as lib
    lib.lib()
    return lib


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed regions run."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


# ---- CPU legs (the oracle: test infrastructure, used here only as the timed CPU baseline) -----------------------------------------
def cpu_rate(fn, work, cores, mp_each, min_seconds=0.0):
    """Run fn over `work` on `cores` threads (the oracle releases the GIL inside its C calls), repeating the list until at least
    min_seconds have passed -> (MP/s, seconds, items)."""
    done, t0 = 0, time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        while True:
            list(ex.map(fn, work))
            done += len(work)
            dt = time.perf_counter() - t0
            if dt >= min_seconds:
                break
    return done * mp_each / dt, dt, done


def cpu_jpeg_lossy(datas, cores, n_images, min_seconds=0.0):
    from oracle import oracle as O
    O.lib()
    p = O.params(QUALITY, SUBSAMPLING, True)
    work = [datas[i % len(datas)] for i in range(n_images)]
    return cpu_rate(lambda d: len(O.jpeg_lossy(d, p)), work, cores, MP_PER_IMAGE, min_seconds)


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = usable_cores()
    datas = make_inputs(min(16, 2 * cores), 0)
    n = 2 * cores
    for _ in range(args.warmup):
        cpu_jpeg_lossy(datas, cores, min(n, cores))
    t_total, imgs = 0.0, 0
    for _ in range(args.steps):
        _, dt, k = cpu_jpeg_lossy(datas, cores, n)
        t_total += dt; imgs += k
    v = imgs * MP_PER_IMAGE / t_total
    sample = f"{n} images/step of the 3840x2160 q90 4:2:0 synthetic set ({len(datas)} unique), {cores} threads, oracle jpeg_lossy (progressive, optimised Huffman; no trellis / scan search), {t_total:.1f} s in all"
    _emit(({
        "impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": "MP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * t_total / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
        "config": {"workload": "configs[1]: 3840x2160 RGB JPEG q90 4:2:0 -> -q 80 --jpeg-chroma-subsampling 4:2:0", "images_per_step": n, "l2": "n/a (CPU)"},
        "images_per_sec": round(v / MP_PER_IMAGE, 2),
        "cpu_baseline": {"value": round(v, 2), "unit": "MP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 2), "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


_RESULT_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too at the C level (NCCL's version banner under
    torchrun), so file descriptor 1 is pointed at stderr for the whole run and the result line goes to a private duplicate
    of the original stdout."""
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def _emit(obj):
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def _peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


# Algorithmic bytes per launch of each kernel of the JPEG path, per image of the megabatch (DESIGN.md 4; px = pixels of the image,
# S_in / S_out = entropy-coded bytes of the input / output file).  Coefficients are int16: 3 B/px at 4:2:0; u8 planes 1.5 B/px.
def jpeg_kernel_bytes(px, s_in, s_out, lossless):
    coef = 3.0 * px
    blocks = 1.5 * px / 64
    b = {
        "k_gd_unstuff_count": s_in, "k_gd_unstuff_scatter": 2 * s_in,
        "k_gd_round0": s_in, "k_gd_round": s_in,                       # every round re-reads (part of) the stream; nothing else
        "k_gd_write": s_in + coef,                                     # stream in, coefficients out (the memset before it is its own launch)
        "k_gd_dc_gather": blocks * 2 + blocks * 4, "k_gd_dc_scatter": blocks * 4 + blocks * 2,
        "k_fused_same": px * 4.0, "k_idct_plane": px * 1.5, "k_chroma420_refdct": px * 1.5,
        "k_geb_classify": coef + blocks * 24,                          # coefficients in, threshold masks out
        "k_geb_hist": coef + blocks * 24, "k_geb_len": coef + blocks * 24,
        "k_geb_emit": coef + blocks * 24 + s_out,
        "k_ge_ffcount": s_out, "k_ge_scatter": 2 * s_out, "k_ge_zero": s_out,
    }
    if lossless:
        for k in ("k_fused_same", "k_idct_plane", "k_chroma420_refdct"):
            b.pop(k)
    return b


def time_pipe(torch, dist, world, pipe, stream, steps, warmup, which=0):
    """K steps of the resident pipe timed with CUDA events on the launching stream; max over ranks; -> (ms total, launches/step)"""
    sh = stream.cuda_stream
    launches = 0
    for _ in range(warmup):
        launches = pipe.run(sh, which)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        pipe.run(sh, which)
    e1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), launches


def dump_pipe_outputs(pipe, out_dir, budget_bytes=60_000_000):
    """The JPEG files of the pipe's last run, as a caller fetches them: jpeg_sizes.npy (float64, bytes per image) and
    jpeg_bytes.npy (float32, images x K): each file's bytes at K fixed relative offsets, drawn once from a seeded generator so
    that files of equal length are sampled at equal positions; K is capped so that both arrays stay under budget_bytes."""
    n = pipe.n
    k = min(1 << 16, budget_bytes // (4 * n))
    frac = np.sort(np.random.default_rng(0).random(k))
    sizes = np.zeros(n, dtype=np.float64)
    sample = np.zeros((n, k), dtype=np.float32)
    for i in range(n):
        f = np.frombuffer(pipe.fetch(i), dtype=np.uint8)
        sizes[i] = f.size
        sample[i] = f[(frac * f.size).astype(np.int64)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "jpeg_sizes.npy"), sizes)
    np.save(os.path.join(out_dir, "jpeg_bytes.npy"), sample)


def jpeg_e2e(args, L, torch, dist, world, datas, params, threads, e2e_threads):
    # ---- end to end through the C-ABI with host buffers
    Be = args.e2e_batch
    ework = [datas[i % len(datas)] for i in range(Be)]
    bi = L.BatchInputs(ework)                                  # pointer/length arrays built once: the timed call is the C-ABI call
    L.compress_batch(ework[:max(threads, 8)], params, e2e_threads, copy=False)      # warm slot pools / pinned buffers
    for _ in range(max(2, args.warmup)):
        L.compress_batch(bi, params, e2e_threads, copy=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    out_bytes = 0
    for _ in range(args.steps):
        # copy=False: outputs are read where the library malloc'ed them (length + SOI marker) and freed; duplicating
        # every file into a Python bytes object is ctypes overhead, not part of the C-ABI a host program calls
        res = L.compress_batch(bi, params, e2e_threads, copy=False)
        assert all(r[1] == 0 and r[3] == b"\xff\xd8" for r in res), [r[2] for r in res if r[1]][:1]
        out_bytes = sum(r[0] for r in res)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    e2e_val = world * Be * MP_PER_IMAGE * args.steps / dt
    in_bytes = sum(len(w) for w in ework)
    e2e = {"value": round(e2e_val, 2), "unit": "MP/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
           "images_per_sec": round(e2e_val / MP_PER_IMAGE, 2), "images_per_step_per_gpu": Be, "host_threads": e2e_threads, "host_cores": threads,
           "in_bytes_per_step": in_bytes, "out_bytes_per_step": out_bytes,
           "megabatch": int(os.environ.get("B200_MEGABATCH", "8")), "group_workers": min(e2e_threads, int(os.environ.get("B200_GROUP_WORKERS", "16"))),
           "note": "JPEG files in host memory -> JPEG files in host memory via b200_compress_batch (the batch form of start_compression's par_iter), all inside the timed region: marker parsing, pinned H2D of the entropy-coded scans, device Huffman decode, transform kernels, device Huffman encode (statistics, optimal tables, bit packing, stuffing), D2H of the scans, file assembly."}
    return e2e


def jpeg_e2e_only(args, L, torch, dist, world, datas, params, threads, e2e_threads):
    e2e = jpeg_e2e(args, L, torch, dist, world, datas, params, threads, e2e_threads)
    return {"value": e2e["value"], "ms_total": 0.0, "launches": 0, "roofline": None, "e2e": e2e, "not_settled": 0, "encoder_retries": 0, "out_bytes_per_image": 0, "in_bytes_per_image": 0}


def jpeg_workload(args, L, torch, dist, world, rank, datas, params, lossless, threads, e2e_threads, with_kernels=True, dump_dir=None):
    """Resident full-path rate (`value`), per-kernel table, and the C-ABI rate (`e2e`) of one JPEG re-encode configuration;
    dump_dir: where rank 0 writes the outputs of the last timed step (dump_pipe_outputs)."""
    px = W4K * H4K
    B = args.batch
    work = [datas[i % len(datas)] for i in range(B)]
    if args.only_e2e:
        return jpeg_e2e_only(args, L, torch, dist, world, datas, params, threads, e2e_threads)
    stream = torch.cuda.Stream()            # a real (non-NULL) stream: the pipe forks from / joins into it and the events are recorded on it
    pipe = L.JpegPipe(work, params, group=args.group)
    ms_total, launches = time_pipe(torch, dist, world, pipe, stream, args.steps, args.warmup)
    sizes, not_settled, retries = pipe.finish()
    if dump_dir and rank == 0:
        dump_pipe_outputs(pipe, dump_dir)
    value = world * B * MP_PER_IMAGE * args.steps / (ms_total / 1e3)
    if args.only_value:
        if rank == 0:
            _emit({"only_value": True, "value": round(value, 1), "images_per_sec": round(value / MP_PER_IMAGE, 1), "group": args.group, "batch": B, "not_settled": not_settled,
                   "rounds": os.environ.get("B200_DEC_ROUNDS"), "launches_per_step": launches})
        pipe.close()
        raise SystemExit(0)
    stage = {}
    for which, name in ((1, "entropy_decode"), (2, "transform"), (3, "entropy_encode")):
        if lossless and which == 2:
            continue
        ms, _ = time_pipe(torch, dist, 1, pipe, stream, max(3, args.steps // 2), 1, which)
        stage[name] = round(ms / max(3, args.steps // 2), 4)
    pipe.finish()
    kern = pipe.kernel_times(3) if with_kernels else {}
    pipe.close()
    peak, peak_src = _peaks()
    s_in = sum(len(w) for w in work[:args.group]) / args.group
    s_out = sum(sizes[:args.group]) / args.group
    alg = jpeg_kernel_bytes(px, s_in, s_out, lossless)
    table = {}
    for name, (ms, cnt) in sorted(kern.items()):
        e = {"ms": round(ms, 4), "launches": cnt}
        if name in alg:
            gbs = alg[name] * args.group / (ms / 1e3) / 1e9
            e["GBps"] = round(gbs, 1); e["frac"] = round(gbs / peak, 4)
        table[name] = e
    named = {k: v for k, v in table.items() if "frac" in v}
    dom = max(named, key=lambda k: named[k]["ms"]) if named else None
    path_bytes = (3.0 + 3.0) * px                                    # SURVEY 8d: fused K1->K5 = coefficients in + coefficients out
    path_gbs = path_bytes * world * B * args.steps / (ms_total / 1e3) / 1e9 / world
    roofline = {"bound": "hbm", "kernel": dom, "achieved": named[dom]["GBps"] if dom else None, "peak": peak, "unit": "GB/s",
                "frac": named[dom]["frac"] if dom else None, "traffic": None, "peak_source": peak_src,
                "ms_per_launch": named[dom]["ms"] if dom else None, "images_per_launch": args.group,
                "path": {"what": "whole device path per GPU on SURVEY 8d's fused figure (6 B/pixel: int16 coefficients in + out)", "GBps": round(path_gbs, 1), "frac": round(path_gbs / peak, 4)},
                "stages_ms_per_step": stage, "all_kernels": table,
                "note": "entropy kernels are latency / issue bound (dependent symbol decodes, bit packing), not HBM bound: their fractions say how far the byte streams are from the memory roofline, see DESIGN.md 4"}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file) and dom:
        try:
            tr = json.load(open(traffic_file))
            roofline["traffic"] = tr.get(dom + "_bytes_per_launch")
        except Exception:
            pass

    e2e = jpeg_e2e(args, L, torch, dist, world, datas, params, threads, e2e_threads)
    return {"value": value, "ms_total": ms_total, "launches": launches, "roofline": roofline, "e2e": e2e,
            "not_settled": not_settled, "encoder_retries": retries, "out_bytes_per_image": s_out, "in_bytes_per_image": s_in}


# ---- configs[3]: 4096x4096 RGBA PNG, --lossless --png-opt-level 3 -----------------------------------------------------------------
def png_stage_times(L, png):
    """Device side of the PNG path on one 4096x4096 image with an event after every launch (b200_png_device_times): the
    device-busy rate (sum of the kernels' own durations; PCIe copies and host decision waits listed but not counted) and the
    per-kernel roofline table on SURVEY 8d's algorithmic bytes (K6: 8 B/px-byte per strategy; K7 >= 4)."""
    try:
        t = L.png_device_times(png, 3, 2)
    except Exception as e:
        return {"error": str(e)[:200]}
    peak, peak_src = _peaks()
    n = 4096 * (4096 * 4 + 1)                      # bytes of the filtered stream (the unit every PNG kernel works on)
    alg = {"k_png_unfilter": 2 * n, "k_png_filter": 2 * n, "k_png_match": n + 4 * n, "k_png_hashmatch": n + 8 * n, "k_png_parse": 4 * n + 4 * n, "k_png_adler": n,
           "k_png_compact": 8 * n, "k_png_probe": n, "k_png_colours": n, "k_dfl_hist": 4 * n, "k_dfl_len": 4 * n, "k_dfl_emit": 4 * n + n}
    table, busy = {}, 0.0
    for name, (ms, cnt) in sorted(t.items()):
        e = {"ms": round(ms, 4), "launches": cnt}
        if name.startswith("k_") or name in ("cub_scan", "memset"):
            busy += ms * cnt
        if name in alg:
            gbs = alg[name] / (ms / 1e3) / 1e9
            e["GBps"] = round(gbs, 1); e["frac"] = round(gbs / peak, 4)
        table[name] = e
    named = {k: v for k, v in table.items() if "frac" in v}
    dom = max(named, key=lambda k: named[k]["ms"] * named[k]["launches"]) if named else None
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(f"{dom}_bytes_per_launch")
    except Exception:
        pass
    return {"value": round(16.777216 / (busy / 1e3), 1) if busy else None, "device_busy_ms_per_image": round(busy, 3),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": named[dom]["GBps"] if dom else None, "peak": peak, "unit": "GB/s", "frac": named[dom]["frac"] if dom else None,
                         "traffic": traffic, "peak_source": peak_src, "ms_per_launch": named[dom]["ms"] if dom else None, "all_kernels": table},
            "value_scope": "device-busy rate of one image's whole launch sequence (un-filter, checksum, probes, 4 filter trials + winner with K6 / K7 fixed + hash candidates / parse, DEFLATE coding): sum of kernel durations from events after every launch; inflate (host) and PCIe copies are in e2e only"}


def cpu_png(datas, L, cores, seconds):
    """Oracle (restated oxipng level-3 filter trials + LZ77) on a bounded sample: one 4096 x 256 strip per thread."""
    from oracle import oracle as O
    O.lib()
    info, raw = L.png_decode(datas[0])
    strips = [np.ascontiguousarray(raw[i * 256:(i + 1) * 256]) for i in range(min(cores, raw.shape[0] // 256))]

    def one(strip):
        best = None
        for s in L.png_level_strategies(3):
            f = O.png_filter(strip, info.bpp, s)
            tok, _ = O.png_lz77(f.reshape(-1), info.bpp, f.shape[1])
            best = tok.size if best is None else min(best, tok.size)
        return best
    v, dt, k = cpu_rate(one, strips, cores, 4096 * 256 / 1e6, seconds)
    return {"value": round(v, 3), "unit": "MP/s", "cores": cores, "kind": "port",
            "sample": f"{k} strips of 4096x256 RGBA from the same source image on {cores} threads: oracle row-filter trials (level-3 strategy set) + LZ77 parse per strip, {dt:.1f} s (inflate / entropy coding of the real reference not included: conservative)"}


# ---- configs[4]: 6000x4000 JPEG -> -q 85 --width 1920 --format webp ---------------------------------------------------------------
def cpu_webp(datas, cores, seconds):
    from oracle import oracle as O
    O.lib()

    def one(d):
        ycc = O.Jpeg(d).decode_native()
        rgb = O.ycc_to_rgb(ycc)
        nw, nh = O.compute_dimensions(6000, 4000, 1920, 0)
        rgb = np.stack([O.resize_plane(rgb[c], nw, nh) for c in range(3)])
        return len(O.webp_encode(rgb, 85)[0])
    work = [datas[i % len(datas)] for i in range(cores)]
    v, dt, k = cpu_rate(one, work, cores, 24.0, seconds)
    return {"value": round(v, 2), "unit": "MP/s", "cores": cores, "kind": "port",
            "sample": f"{k} of the same 6000x4000 inputs on {cores} threads: oracle decode + Lanczos3 + VP8 encode, {dt:.1f} s"}


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=128, help="images per step per GPU, device-resident leg (128 x ~1.5 MB of scan bytes > L2)")
    ap.add_argument("--group", type=int, default=8, help="images per launch sequence (megabatch) in the device-resident leg")
    ap.add_argument("--e2e-batch", type=int, default=1024, help="images per step per GPU (C-ABI leg); one blocking b200_compress_batch call per step, so every step pays one pipeline fill and drain (~8 ms): 256 images per step under-reports the steady-state rate by ~10 %")
    ap.add_argument("--unique", type=int, default=64, help="unique synthetic sources per rank, cycled to fill a batch")
    ap.add_argument("--configs", default=None, help="comma list of BASELINE configs to run (1 = the headline; 2,3,4 = sub-records); default 1,2,3,4 on one GPU, 1 under torchrun")
    ap.add_argument("--png-unique", type=int, default=4); ap.add_argument("--png-batch", type=int, default=64)
    ap.add_argument("--png-threads", type=int, default=0, help="callers in flight for the PNG leg (default: twice the usable cores, 16..48: a caller spends 0.2 s inflating on its core and then waits for its share of the device, which is the bound -- measured 16 / 24 / 32 / 48 callers: 429 / 466 / 479 / 493 MP/s)")
    ap.add_argument("--webp-unique", type=int, default=8); ap.add_argument("--webp-batch", type=int, default=64)
    ap.add_argument("--cpu-seconds", type=float, default=6.0, help="minimum CPU work per cpu_baseline sample")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-threads", type=int, default=0, help="host threads per rank for the C-ABI leg (default: the rank's share of the usable cores, at least 8)")
    ap.add_argument("--only-e2e", action="store_true", help="diagnostics: skip the device-resident leg and the per-kernel table")
    ap.add_argument("--only-value", action="store_true", help="diagnostics: the device-resident leg only (prints a short JSON line)")
    ap.add_argument("--only-configs", action="store_true", help="diagnostics: skip configs[1]; prints {\"configs\": {...}} for the sub-records named by --configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the JPEG files of configs[1]'s last timed step under DIR as .npy (rank 0's shard), to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.only_e2e or args.only_configs):
        ap.error("--dump-outputs needs the device-resident leg of configs[1]")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    which = set(int(x) for x in (args.configs.split(",") if args.configs else (["1", "2", "3", "4"] if world == 1 else ["1"])))

    # ---- inputs first (fork pool must run before CUDA is initialised in this process)
    cores = usable_cores()
    threads = max(1, cores // max(1, world))
    # the data set is world x unique seeded sources; each rank owns a shard of it (caesium-clt_b200/sharding.py: the same code the
    # world_size-2 gloo test runs on CPU); no image ever crosses ranks
    from importlib import import_module
    load_pkg_shallow()
    S = import_module("caesium_clt_b200.sharding")
    shard = S.shard_indices([1] * (world * args.unique), world, rank, policy="rr")
    datas = make_inputs(len(shard), 0, "jpeg4k", procs=threads, indices=shard if not args.only_configs else shard[:2])
    png_datas = make_inputs(args.png_unique, 0, "png4096") if 3 in which else None
    webp_datas = make_inputs(args.webp_unique, 0, "jpeg24mp") if 4 in which else None
    # batch workers mostly wait for their stream: on a box with few cores per GPU a rank still keeps eight megabatches in flight
    e2e_threads = args.e2e_threads if args.e2e_threads > 0 else max(threads, 8)

    import torch
    import torch.distributed as dist
    L = load_pkg()
    torch.cuda.set_device(local_rank)
    if L.lib().b200_init_device(local_rank) != 0:
        raise SystemExit("bench.py: no B200 visible -- the product has no CPU fallback")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # quant tables: computed on rank 0, broadcast over NCCL (the only collective of this path), checked locally
    got = S.broadcast_quant_table(L.jpeg_quant_table(QUALITY, 0), dist if world > 1 else None, 0, device="cuda")
    assert np.array_equal(got, L.jpeg_quant_table(QUALITY, 0)), "quant-table handshake failed"

    p = L.default_params()
    p.jpeg_quality, p.jpeg_chroma_subsampling, p.jpeg_progressive = QUALITY, SUBSAMPLING, 1

    clocks = ClockSampler(local_rank)
    clocks.start()
    r1 = None if args.only_configs else jpeg_workload(args, L, torch, dist, world, rank, datas, p, False, threads, e2e_threads, dump_dir=args.dump_outputs)
    clk = clocks.stop()

    sub = {}
    cpu = None
    if rank == 0 and world == 1:
        if 2 in which:
            p2 = L.default_params(); p2.jpeg_optimize = 1; p2.jpeg_progressive = 1
            r2 = jpeg_workload(args, L, torch, dist, 1, 0, datas, p2, True, threads, e2e_threads)
            rec = {"workload": "configs[2]: the same 3840x2160 JPEGs, --lossless (coefficient-domain transcode: device Huffman decode -> device Huffman encode, optimal tables, progressive script)",
                   "metric": "megapixels/sec lossless JPEG transcode", "unit": "MP/s", "value": round(r2["value"], 1), "ms_per_step": round(r2["ms_total"] / args.steps, 4),
                   "images_per_sec": round(r2["value"] / MP_PER_IMAGE, 1), "e2e": r2["e2e"], "roofline": r2["roofline"], "gpu_launches": r2["launches"] * args.steps}
            if not args.skip_cpu_baseline:
                from oracle import oracle as O
                O.lib()
                po = O.params(80, 0, True)
                v, cdt, k = cpu_rate(lambda d: len(O.jpeg_lossless(d, po)), [datas[i % len(datas)] for i in range(2 * cores)], cores, MP_PER_IMAGE, args.cpu_seconds)
                rec["cpu_baseline"] = {"value": round(v, 2), "unit": "MP/s", "cores": cores, "kind": "port", "sample": f"{k} of the same 4K inputs, {cores} threads, oracle jpeg_lossless, {cdt:.1f} s"}
            sub["2"] = rec
        if 3 in which:
            rec, _ = config_png_run(args, L, cores, png_datas)
            if not args.skip_cpu_baseline:
                rec["cpu_baseline"] = cpu_png(png_datas, L, cores, args.cpu_seconds)
            sub["3"] = rec
        if 4 in which:
            rec, _ = config_webp_run(args, L, cores, webp_datas)
            if not args.skip_cpu_baseline:
                rec["cpu_baseline"] = cpu_webp(webp_datas, cores, args.cpu_seconds)
            sub["4"] = rec
        if not args.skip_cpu_baseline:
            n = 2 * cores
            cpu_jpeg_lossy(datas, cores, cores)
            v, cdt, k = cpu_jpeg_lossy(datas, cores, n, args.cpu_seconds)
            cpu = {"value": round(v, 2), "unit": "MP/s", "cores": cores, "kind": "port",
                   "sample": f"{k} of the same 4K inputs ({len(datas)} unique), {cores} threads, oracle jpeg_lossy (restated reference: progressive + optimised Huffman, no trellis/scan search), {cdt:.1f} s"}

    if rank == 0 and args.only_configs:
        _emit({"configs": sub})
    elif rank == 0:
        B = args.batch
        _emit(({
            "metric": METRIC, "value": round(r1["value"], 1), "unit": "MP/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(r1["ms_total"] / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
            "config": {"workload": "configs[1]: 3840x2160 RGB JPEG q90 4:2:0 -> -q 80 --jpeg-chroma-subsampling 4:2:0 (progressive, optimised Huffman)",
                       "value_scope": "FULL device path, inputs resident: entropy-coded scans in HBM -> Huffman decode -> K1-K5 transform -> Huffman encode -> entropy-coded scans in HBM (b200_jpeg_pipe_*); no host wait inside the timed region",
                       "images_per_step_per_gpu": B, "megabatch": args.group, "unique_sources_per_gpu": len(datas), "parallelism": f"dp{world} (images sharded, no collective on the path)",
                       "l2": f"per step and GPU {B * r1['in_bytes_per_image'] / 1e6:.0f} MB of scan bytes are read and {B * 2 * W4K * H4K * 3 / 1e9:.1f} GB of coefficients pass through HBM (L2 = 126 MB): nothing of a step survives in L2 to the next"},
            "images_per_sec": round(r1["value"] / MP_PER_IMAGE, 1),
            "e2e": r1["e2e"], "gpu_launches": r1["launches"] * args.steps, "roofline": r1["roofline"], "cpu_baseline": cpu, "clocks": clk,
            "decoder_not_settled": r1["not_settled"], "encoder_retries": r1["encoder_retries"],
            "configs": sub,
        }))
    if os.environ.get("B200_TRACE"):
        L.lib().b200_shutdown()             # prints the per-stage wall-clock table
    if world > 1:
        dist.destroy_process_group()


def config_png_run(args, L, cores, datas):
    w = h = 4096
    mp = w * h / 1e6
    p = L.default_params(); p.png_optimize = 1; p.png_optimization_level = 3
    n = args.png_batch
    work = [datas[i % len(datas)] for i in range(n)]
    nt = args.png_threads if args.png_threads > 0 else min(48, max(2 * cores, 16))
    L.compress_batch(work[:min(n, nt)], p, nt, copy=False)
    bi = L.BatchInputs(work)
    steps = max(1, args.steps // 5)
    t0 = time.perf_counter()
    out_bytes = 0
    for _ in range(steps):
        res = L.compress_batch(bi, p, nt, copy=False)
        assert all(r[1] == 0 for r in res), [r[2] for r in res if r[1]][:1]
        out_bytes = sum(r[0] for r in res)
    dt = time.perf_counter() - t0
    rate = n * steps * mp / dt
    in_bytes = sum(len(x) for x in work)
    stage = png_stage_times(L, datas[0])
    rec = {"workload": "configs[3]: 4096x4096 RGBA8 PNG (Paeth rows, zlib 6) -> --lossless --png-opt-level 3", "metric": "megapixels/sec lossless PNG re-encode", "unit": "MP/s",
           "value": stage.get("value") if isinstance(stage, dict) else None, "device": stage, "roofline": stage.get("roofline") if isinstance(stage, dict) else None,
           "e2e": {"value": round(rate, 2), "unit": "MP/s", "images_per_sec": round(rate / mp, 3), "h2d_bytes_per_step": n * w * h * 4, "d2h_bytes_per_step": out_bytes,
                   "in_bytes_per_step": in_bytes, "out_bytes_per_step": out_bytes, "images_per_step": n, "steps": steps, "host_threads": nt,
                   "note": "PNG files in host memory -> PNG files in host memory via b200_compress_batch: container parse + inflate + unfilter, device row-filter selection (K6) and LZ77 (K7), entropy coding, container"},
           "out_over_in_bytes": round(out_bytes / in_bytes, 4)}
    return rec, datas


def config_webp_run(args, L, cores, datas):
    mp = 24.0
    p = L.default_params(); p.webp_quality = 85; p.width = 1920
    n = args.webp_batch
    work = [datas[i % len(datas)] for i in range(n)]

    def conv(d):
        return len(L.convert_in_memory(d, p, 3))
    nt = max(cores, 16)
    with ThreadPoolExecutor(nt) as ex:
        list(ex.map(conv, work[:nt]))
        steps = max(1, args.steps // 3)
        d2h0 = L.lib().b200_webp_d2h_bytes()
        t0 = time.perf_counter()
        out_bytes = 0
        for _ in range(steps):
            out_bytes = sum(ex.map(conv, work))
        dt = time.perf_counter() - t0
        d2h = (L.lib().b200_webp_d2h_bytes() - d2h0) // steps
    rate = n * steps * mp / dt
    rec = {"workload": "configs[4]: 6000x4000 JPEG q90 4:2:0 -> -q 85 --width 1920 --format webp (1920x1280 lossy VP8)", "metric": "input megapixels/sec JPEG -> resized WebP", "unit": "MP/s",
           "value": None,
           "e2e": {"value": round(rate, 2), "unit": "MP/s", "images_per_sec": round(rate / mp, 2), "h2d_bytes_per_step": sum(len(x) for x in work), "d2h_bytes_per_step": int(d2h),
                   "out_bytes_per_step": out_bytes, "images_per_step": n, "steps": steps, "host_threads": nt,
                   "note": "JPEG file in host memory -> WebP file in host memory via b200_convert_in_memory on a thread pool: device Huffman decode, IDCT, upsample, YCbCr->RGB, Lanczos3 (K3), VP8 wavefront (K8), residual token pass; D2H of the frame's decision records + tallies + modes; host boolean coder"}}
    return rec, datas


if __name__ == "__main__":
    main()
