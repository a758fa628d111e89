#!/usr/bin/env python
"""bench.py -- megapixels/s of HEIC-grid decode -> RGB on B200 (BASELINE.json metric), one JSON line on stdout.

Workload (BASELINE configs[2]): a synthetic 16384x16384 HEIC grid = 256 independent 1024x1024 HEVC-intra tiles
(8-bit 4:2:0, fixed QP 27, CTB 32, WPP, SAO + deblocking on; seed 0xB200 + tile index; SURVEY.md 8d) decoded to
interleaved RGB24.  One "step" = the whole grid once.
  value : device-timed (CUDA events) MP/s with the compressed tiles resident in HBM: entropy decoding (K0) + reconstruction
          (K1) + deblocking + SAO/paste + colour conversion (+ the NCCL gather of the RGB bands when N > 1).
  e2e   : host bitstreams -> host RGB through ONE call of the C ABI per rank (b200_decode_grid_to_rgb_host): header parse on
          the host cores, H2D of the compressed tiles, all kernels, D2H of the RGB into page-locked host memory (N > 1: every
          rank writes its row band into one shared host buffer over its own PCIe link), all inside the timed region.
  parity_checked : the RGB of the top-left sub-grid of the e2e result is compared, byte for byte, with what the UNMODIFIED
          reference libheif (heif_decode_image + CPU decoder plugin) produces for the same tiles in the same run.
  --impl reference : heif_decode_image() of the unmodified reference (oracle/_ref/libheif_ref.so) with the oracle's CPU
          decoder plugin (FFmpeg in the libde265 role), heif_context_set_max_decoding_threads(cores), on a HEIC grid file
          holding the very same tiles (oracle/ref_arm.py, oracle/heic_writer.py) -- the whole 256-tile grid per step.
Multi-GPU (torchrun, one rank per GPU): tile rows are sharded across ranks (strong scaling: the grid is fixed); the only
collective is the final gather of RGB row bands to rank 0 (NCCL over NVLink) in the device-timed leg.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TILE = 1024
QP = 27
DUMP_SAMPLES = 1 << 22      # bytes of RGB per dumped array: 16 MB as float32


def dump_sample_index(nbytes):
    """The byte offsets --dump-outputs samples: fixed by the seed and the picture size alone."""
    return np.sort(np.random.default_rng(0xB200).integers(0, nbytes, min(DUMP_SAMPLES, nbytes)))


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def make_tile(idx, tile=TILE, log2_ctb=5):
    from libheif_b200 import hevc_enc
    y, cb, cr = hevc_enc.synthetic_image(0xB200 + idx, tile, tile, 8, True)
    return hevc_enc.encode_intra(y, cb, cr, bit_depth=8, log2_ctb_size=log2_ctb, qp=QP, wpp=1, seed=0xB200 + idx, vui_present=1,
                                 colour_description_present=1, colour_primaries=1, transfer_characteristics=13,
                                 matrix_coefficients=6, full_range=0)


def make_tiles(indices, tile=TILE, workers=None, log2_ctb=5):
    """Encoded tiles (deterministic in idx).  B200_BENCH_TILE_CACHE names a directory this process and its reference-arm
    children share, so that the 256 tiles are encoded once per bench run (input generation is untimed either way)."""
    workers = workers or min(64, effective_cores())
    cache = os.environ.get("B200_BENCH_TILE_CACHE")

    def one(i):
        f = os.path.join(cache, f"t{tile}_c{log2_ctb}_q{QP}_{i}.au") if cache else None
        if f and os.path.exists(f):
            return open(f, "rb").read()
        au = make_tile(i, tile, log2_ctb)
        if f:
            tmp = f + f".{os.getpid()}.tmp"
            with open(tmp, "wb") as fh:
                fh.write(au)
            os.replace(tmp, f)
        return au
    with ThreadPoolExecutor(workers) as ex:
        return list(ex.map(one, indices))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.samples = []
        self.stop = False
        self.idx = gpu_index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                r = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5)
                f = [x.strip() for x in r.stdout.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        reasons = set()
        for s in self.samples:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": sorted(reasons), "samples": len(sm)}


def effective_cores():
    """Host cores this process may actually use: min(visible CPUs, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ------------------------------------------------------------------------------------------ reference CPU arm
def reference_arm(side, sub, steps, warmup, cores, dump=None, log2_ctb=5, extra=()):
    """heif_decode_image() of the unmodified reference on the same tiles, in a child process (oracle/ref_arm.py; the
    reference library must not share a process with torch).  Returns (dict, None) or (None, reason)."""
    cmd = [sys.executable, "-m", "oracle.ref_arm", "--side", str(side), "--sub", str(sub), "--steps", str(steps), "--warmup", str(warmup),
           "--threads", str(cores), "--ctb", str(log2_ctb)]
    if dump:
        cmd += ["--dump", dump]
    cmd += list(extra)
    try:
        r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=3000)
    except Exception as e:  # noqa: BLE001
        return None, f"reference child failed: {e}"
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        return None, "reference child failed: " + (r.stderr or "")[-300:].replace("\n", " | ")
    res = json.loads(lines[-1])
    if "unavailable" in res:
        return None, res["unavailable"]
    res["sample"] = (f"whole grid: {side}x{side} tiles" if sub == side else f"top-left {sub}x{sub} tiles of the same grid") + \
        f" ({res['width']}x{res['height']}, {res['pixels'] / 1e6:.1f} MP) per step, {res['api']}"
    return res, None


def load_traffic():
    """dram__bytes_read + dram__bytes_write per launch of each kernel, from the ncu captures of THIS code committed under
    profiles/ (profiles/r02_traffic.json names the capture each figure comes from); None when no capture exists."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return json.load(open(p))
    except Exception:  # noqa: BLE001
        return {}


def main():
    if "B200_BENCH_TILE_CACHE" not in os.environ:
        import atexit
        import shutil
        import tempfile
        d = tempfile.mkdtemp(prefix="b200_bench_tiles_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        os.environ["B200_BENCH_TILE_CACHE"] = d
        atexit.register(shutil.rmtree, d, True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tiles-side", type=int, default=16, help="grid is tiles-side x tiles-side tiles of 1024x1024 (16 = BASELINE config)")
    ap.add_argument("--ref-sample-side", type=int, default=16, help="sub-grid the in-run parity check / cpu_baseline decodes with the reference (default: the whole 16 x 16 grid, ~2.4 s per decode on 16 cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-plugin-leg", action="store_true", help="skip the heif_decode_image + plugin legs (e2e_plugin, e2e_plugin_n2)")
    ap.add_argument("--no-ctb64", action="store_true", help="skip the additional CTB 64 measurement (x265's default CTB size)")
    ap.add_argument("--ctb", type=int, default=5, choices=[4, 5, 6], help="log2 CTB size of the synthetic tiles (5 = the benchmark workload)")
    ap.add_argument("--front-end", default="device", choices=["device", "host"], help="where CABAC runs: GPU (one warp per WPP sub-stream) or host cores")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the RGB of the last timed step of the device leg (rgb.npy) and of the e2e legs "
                    f"(rgb_e2e.npy) as float32, each a fixed seeded sample of {DUMP_SAMPLES} bytes of the picture, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    warmup = max(3, args.warmup)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    side = args.tiles_side
    cores = effective_cores()
    workload = f"{side * TILE}x{side * TILE} HEIC grid, {side * side} x {TILE}x{TILE} HEVC-intra tiles, 8-bit 4:2:0 -> RGB24, QP {QP}, CTB {1 << args.ctb}, WPP, SAO+deblock"

    if args.impl == "reference":
        if rank != 0:
            return
        res, why = reference_arm(side, side, args.steps, warmup, cores, log2_ctb=args.ctb)
        if res is None:
            print(json.dumps({"impl": "reference", "unavailable": why}))
            return
        line = {"impl": "reference", "metric": "megapixels/sec HEIC-grid decode->RGB", "value": res["mp_s"], "unit": "MP/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": {"workload": workload, "sample": res["sample"], "decoding_threads": res["threads"]},
                "rgb_md5": res["rgb_md5"],
                "cpu_baseline": {"value": res["mp_s"], "unit": "MP/s", "cores": cores, "kind": "reference", "sample": res["sample"]},
                "e2e": {"value": res["mp_s"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import hashlib
    import mmap
    import torch
    import torch.distributed as dist
    import libheif_b200 as lb
    from libheif_b200 import _lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # ---- shard: contiguous tile-row bands per rank (libheif_b200/sharding.py, gloo-tested in tests/test_sharding.py)
    from libheif_b200 import sharding
    r0, nrows, my_idx = sharding.my_band(side, side, world, rank)
    t_gen = time.perf_counter()
    tiles = make_tiles(my_idx, workers=max(4, cores // world), log2_ctb=args.ctb)
    t_gen = time.perf_counter() - t_gen
    W, H = side * TILE, side * TILE
    band_h = nrows * TILE
    dec = lb.Decoder(host_threads=max(1, cores // world))
    dec.set_front_end(args.front_end == "device")
    band = torch.empty((max(band_h, 1), W * 3), dtype=torch.uint8, device=dev)
    full = torch.empty((H, W * 3), dtype=torch.uint8, device=dev) if (rank == 0 and world > 1) else None
    stream = torch.cuda.current_stream()
    # ---- host destination of the e2e leg: one page-locked buffer for the whole picture.  N > 1: a shared-memory mapping
    # every rank registers with CUDA and writes its own row band into (per-rank PCIe links instead of gather + one D2H).
    l = _lib.lib()
    shm_path = f"/dev/shm/b200_bench_{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if world > 1 else os.getpid()}.rgb"
    if world > 1:
        if rank == 0:
            with open(shm_path, "wb") as f:
                f.truncate(H * W * 3)
        dist.barrier()
        fd = os.open(shm_path, os.O_RDWR)
        mm = mmap.mmap(fd, H * W * 3)
        host_out = np.frombuffer(mm, dtype=np.uint8).reshape(H, W * 3)
        l.b200_host_register.argtypes = [ctypes.c_void_p, ctypes.c_size_t]
        _lib.check(l.b200_host_register(host_out.ctypes.data, host_out.nbytes))
    else:
        host_t = torch.empty((H, W * 3), dtype=torch.uint8, pin_memory=True)
        host_out = host_t.numpy()
    my_out = host_out[r0 * TILE:r0 * TILE + band_h] if nrows else None

    def gather():
        return sharding.gather_bands(band, side, TILE, world, rank, full) if world > 1 else band

    def device_step():
        if nrows:
            dec.rerun_device(stream)
            dec.to_rgb_device(lb.CHROMA_INTERLEAVED_RGB, out=band, stream=stream)
        return gather()

    def e2e_step():
        if nrows:                       # ONE C-ABI call: host bitstreams in, host RGB out (b200_decode_grid_to_rgb_host)
            dec.decode_grid_to_rgb_host(tiles, side, nrows, lb.CHROMA_INTERLEAVED_RGB, out=my_out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up (also uploads the compressed tiles for the device leg)
    for _ in range(warmup):
        e2e_step()
    st0 = dec.stats() if nrows else None
    with ClockSampler(local_rank) as clk:
        # ---- leg A: kernels with the compressed tiles resident in HBM (CUDA events, max over ranks)
        for _ in range(warmup):
            device_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            rgb_dev = device_step()
        e1.record(stream)
        barrier()
        dev_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
        dump_dev = None
        if args.dump_outputs and rank == 0:
            flat = rgb_dev.reshape(-1)
            dump_dev = flat[torch.from_numpy(dump_sample_index(flat.numel())).to(dev)].float().cpu().numpy()
        # ---- leg B: end to end through the C ABI, host buffers in, page-locked host RGB out (wall clock around a synchronised region)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        barrier()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
        stats_e2e = dec.stats() if nrows else None
        # ---- leg C: the same through the throughput form of the call (b200_decode_grid_to_rgb_host_async + b200_decoder_wait):
        # the D2H of step i overlaps the kernels of step i + 1; every step still parses, uploads, decodes and delivers its RGB
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            if nrows:
                dec.decode_grid_to_rgb_host_async(tiles, side, nrows, lb.CHROMA_INTERLEAVED_RGB, out=my_out)
        if nrows:
            dec.wait()
        barrier()
        pipe_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    # ---- per-kernel device times (outside the timed regions): average over a few launches, CUDA events
    kern = {"entropy": 0.0, "recon": 0.0, "deblock": 0.0, "sao_paste": 0.0, "k6_colour": 0.0}
    nk = 5
    overlapped = False
    chunked = bool(nrows) and stats_e2e.front_end == 3
    if nrows:
        # the e2e legs above ran K1 .. K6 in row bands (D2H of a band overlaps the kernels of the next); the per-kernel times are
        # taken with one launch per kernel for the whole grid (B200_CHUNKS=0)
        os.environ["B200_CHUNKS"] = "0"
        os.environ["B200_TAIL_OVERLAP"] = "0"          # per-kernel times: K1 after K0, not inside K0's draining tail
        dec.decode_grid(tiles, cols=side, rows=nrows)
        for _ in range(nk):
            dec.rerun_device(stream)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record(stream); dec.to_rgb_device(lb.CHROMA_INTERLEAVED_RGB, out=band, stream=stream); k1.record(stream)
            torch.cuda.synchronize()
            s = dec.stats()
            overlapped = s.front_end == 2
            kern["entropy"] += s.entropy_ms / nk; kern["recon"] += s.recon_ms / nk; kern["deblock"] += s.deblock_ms / nk; kern["sao_paste"] += s.sao_ms / nk; kern["k6_colour"] += k0.elapsed_time(k1) / nk
    os.environ.pop("B200_CHUNKS", None)
    os.environ.pop("B200_TAIL_OVERLAP", None)
    barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- rank 0: report
    pixels = W * H
    my_px = band_h * W
    peak, peak_src = measured_peak()
    C = st0.command_bytes / my_px                                     # measured command-stream bytes per pixel
    bpp = st0.bitstream_bytes / my_px
    # algorithmic B/px (SURVEY.md 8(d), 8-bit): entropy reads the bitstream and writes the command stream once
    alg = {"entropy": bpp + C, "recon": 1.5 + C, "deblock": 3.0, "sao_paste": 3.0, "k6_colour": 4.5}
    if args.front_end == "host":
        kern.pop("entropy")
    if overlapped:                                   # K0 and K1 ran concurrently: one time for both, one algorithmic figure
        kern["entropy+recon"] = kern.pop("entropy") + kern.pop("recon")
        alg["entropy+recon"] = bpp + 1.5 + C         # bitstream read, planes written; the command stream stays in L2 / HBM in between
    dom = max(kern, key=kern.get)
    ach = alg[dom] * my_px / (kern[dom] * 1e-3) / 1e9
    tr = load_traffic().get(dom) if (world == 1 and side == 16 and args.ctb == 5) else None      # the captures are of this exact workload
    bins = 2.0 * my_px                               # ~2.0 CABAC bins per pixel on this workload (1.57 context-coded + 0.43 bypass, counted by the host front-end)
    line = {
        "metric": "megapixels/sec HEIC-grid decode->RGB", "value": pixels / 1e6 / (dev_ms / 1e3), "unit": "MP/s", "n_gpus": world,
        "steps": args.steps, "warmup": warmup, "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload, "sharding": f"{world} x contiguous tile-row bands, NCCL gather of RGB bands to rank 0 (device leg); per-rank D2H into one shared page-locked host buffer (e2e leg)" if world > 1 else "single GPU",
                   "l2": "inputs larger than L2 (command stream + planes > 126 MB per GPU)" if st0.command_bytes + my_px * 1.5 > 126e6 else "flush not needed: see note",
                   "bits_per_pixel": 8.0 * st0.bitstream_bytes / my_px, "command_bytes_per_pixel": C, "host_parser_threads": max(1, cores // world), "front_end": args.front_end + (" (CABAC on the GPU, one warp per WPP sub-stream)" if args.front_end == "device" else " (CABAC on the host cores)")},
        "e2e": {"value": pixels / 1e6 / (e2e_ms / 1e3), "unit": "MP/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(stats_e2e.h2d_bytes * (pixels / my_px)),
                "d2h_bytes_per_step": pixels * 3, "host_parse_ms": stats_e2e.parse_ms, "host_pack_ms": stats_e2e.pack_ms,
                "api": "b200_decode_grid_to_rgb_host (one C-ABI call per rank: host access units -> page-locked host RGB)"},
        "e2e_pipelined": {"value": pixels / 1e6 / (pipe_ms / 1e3), "unit": "MP/s", "ms_per_step": pipe_ms,
                          "api": "b200_decode_grid_to_rgb_host_async x steps + b200_decoder_wait: D2H of step i overlaps the kernels of step i + 1 (throughput of a batch job; e2e above is the latency of one call)"},
        "pipeline": {"bands": stats_e2e.bands, "entropy_ms_in_e2e_leg": stats_e2e.entropy_ms, "band_pipeline_ms_in_e2e_leg": stats_e2e.recon_ms + stats_e2e.deblock_ms + stats_e2e.sao_ms,
                     "tail_overlap": os.environ.get("B200_TAIL_OVERLAP", "1") != "0",
                     "note": "e2e legs of large grids: the tile rows go through K1 -> K3 -> K4 -> K6 in row bands and the D2H of band c overlaps the kernels of band c + 1; K1 is queued behind the full-occupancy entropy kernel and follows it CTB by CTB in the SM slots its draining wavefronts free (tail overlap), so band_pipeline_ms is what remains after the entropy kernel has ended (kernels_ms below: one launch per kernel for the whole grid, one after the other: B200_CHUNKS=0 B200_TAIL_OVERLAP=0)"},
        "gpu_launches": (stats_e2e.kernel_launches + (stats_e2e.bands if chunked else 1)) * args.steps,   # K0 (+ gate), (K1, K3 x2, K4 luma + chroma) per band as counted by the library, + K6 per band -- of the e2e leg
        "clocks": clk.summary(),
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": tr["bytes_per_launch"] if tr else None, "traffic_source": tr["source"] if tr else None,
                     "peak_source": peak_src, "algorithmic_bytes_per_pixel": alg[dom],
                     "kernels_ms": kern, "kernels_gb_s": {k: alg[k] * my_px / (v * 1e-3) / 1e9 if v > 0 else None for k, v in kern.items()},
                     "entropy_gbins_per_s": bins / (kern["entropy"] * 1e-3) / 1e9 if kern.get("entropy") else None,
                     "pipeline_A_bytes_per_pixel": 12.0 + C,
                     "pipeline_gb_s": (12.0 + C) * my_px / (sum(kern.values()) * 1e-3) / 1e9 if sum(kern.values()) > 0 else None},
        "setup": {"tile_generation_s": t_gen},
    }
    # ---- parity inside the bench + CPU baseline: the unmodified reference decodes the top-left sub-grid of the SAME tiles
    line["rgb_md5"] = hashlib.md5(host_out.tobytes()).hexdigest()    # full 16384x16384 RGB; the reference arm prints the md5 of its own result
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "rgb.npy"), dump_dev)
        np.save(os.path.join(args.dump_outputs, "rgb_e2e.npy"), host_out.reshape(-1)[dump_sample_index(host_out.size)].astype(np.float32))
    if not args.no_cpu_baseline:
        sub = min(side, args.ref_sample_side)
        dump = f"/dev/shm/b200_bench_ref_{os.getpid()}.rgb"
        res, why = reference_arm(side, sub, args.steps, 1, cores, dump=dump, log2_ctb=args.ctb)
        if res:
            ref = np.fromfile(dump, dtype=np.uint8).reshape(sub * TILE, sub * TILE * 3)
            os.unlink(dump)
            ours = host_out[:sub * TILE, :sub * TILE * 3]
            line["parity_checked"] = bool(np.array_equal(ours, ref))
            line["parity"] = {"compared": f"top-left {sub}x{sub} tiles ({sub * sub * TILE * TILE / 1e6:.1f} MP) of the e2e result vs heif_decode_image of the unmodified reference, byte for byte",
                              "mismatching_bytes": int(np.count_nonzero(ours != ref))}
            line["cpu_baseline"] = {"value": res["mp_s"], "unit": "MP/s", "cores": cores, "kind": "reference", "sample": res["sample"]}
        else:
            line["parity_checked"] = False
            line["parity"] = {"compared": f"unavailable: {why}"}
            line["cpu_baseline"] = {"value": None, "unit": "MP/s", "cores": cores, "kind": "reference", "sample": f"unavailable: {why}"}
    # ---- the drop-in path: heif_decode_image() of the unmodified reference library with THIS plugin selected, one libheif
    # decoding thread per tile so that the plugin's submission queue sees the whole grid (INTEGRATION.md 1); then the same
    # through the second reference build that carries the GPU colour operation (SURVEY 8f N2)
    if world == 1 and not args.no_plugin_leg and args.front_end == "device":
        for key, extra in (("e2e_plugin", []), ("e2e_plugin_n2", ["--lib", "libheif_ref_b200.so"])):
            dump = f"/dev/shm/b200_bench_plug_{os.getpid()}.rgb"
            res, why = reference_arm(side, side, args.steps, 2, side * side, dump=dump, log2_ctb=args.ctb, extra=["--decoder", "b200"] + extra)
            if res:
                got = np.fromfile(dump, dtype=np.uint8)
                os.unlink(dump)
                line[key] = {"value": res["mp_s"], "unit": "MP/s", "ms_per_step": res["ms_per_step"], "libheif_threads": res["threads"], "plugin_queue": res["plugin_queue"],
                             "identical_to_e2e_result": bool(got.size == host_out.size and np.array_equal(got, host_out.reshape(-1))), "api": res["api"]}
            else:
                line[key] = {"value": None, "unavailable": why}
    # ---- the same grid coded with CTB 64 (x265's default): longer wavefront per tile; device leg only, few steps
    if world == 1 and not args.no_ctb64 and args.ctb == 5 and args.front_end == "device":
        try:
            t64 = make_tiles(my_idx, workers=max(4, cores), log2_ctb=6)
            dec.decode_grid_to_rgb_host(t64, side, nrows, lb.CHROMA_INTERLEAVED_RGB, out=my_out)
            ts = []
            for _ in range(args.steps):
                t0 = time.perf_counter(); dec.decode_grid_to_rgb_host(t64, side, nrows, lb.CHROMA_INTERLEAVED_RGB, out=my_out); ts.append(time.perf_counter() - t0)
            s64 = dec.stats()
            line["ctb64"] = {"e2e_mp_s": pixels / 1e6 / (sum(ts) / len(ts)), "e2e_ms_per_step": 1e3 * sum(ts) / len(ts), "entropy_ms": s64.entropy_ms, "recon_ms": s64.recon_ms,
                             "deblock_ms": s64.deblock_ms, "sao_paste_ms": s64.sao_ms, "bits_per_pixel": 8.0 * s64.bitstream_bytes / my_px,
                             "note": f"same pictures, same QP, coded with CTB 64 (x265 default); {args.steps} e2e steps after 1 warm-up"}
        except Exception as e:  # noqa: BLE001
            line["ctb64"] = {"error": str(e)[:200]}
    print(json.dumps(line))
    if world > 1:
        try:
            os.unlink(shm_path)
        except OSError:
            pass
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
