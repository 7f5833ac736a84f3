#!/usr/bin/env python
"""bench.py -- disparity Mpix/s of the dense block-matching hot path (BASELINE.json metric).

Headline workload (`value`, `e2e`): vw::stereo::calc_disparity / best_of_search_convolution over a synthetic 8192x8192
stereo pair, 128x128 search window, 21x21 kernel, AbsoluteCost, integer-valued 12-bit imagery (SURVEY.md section 8d "NS").
A step = one full-image pass.  At N = 1 the same JSON line also carries, under "configs", one device-resident measurement
of every other BASELINE.json configuration (NS with SquaredCost / NCC, config 2, config 3, config 4) and, at N = 8,
config 5 (16384^2, 256x256 window, sharded by tile row with NCCL halo rows).

  python bench.py --gpus N --steps K --warmup W          our arm (torchrun for N > 1)
  python bench.py --impl reference ...                   the reference algorithm on the host cores (rank 0 only)
  python bench.py --gpus 1 ... --dump-outputs DIR        also write the headline disparity of the last timed step to DIR

N > 1: the image is sharded into contiguous output-row bands, one per rank (strong scaling).  Inputs are row-sharded too:
every step each rank receives the halo rows it needs (kernel-1 rows of the left raster, kernel-1 + search-1 rows of the
right raster) from the next rank with NCCL send/recv over NVLink, inside the timed region.  No other collective exists.
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (which may be read-only)

COSTS = {"abs": 0, "sq": 1, "ncc": 2}
# measured on this pool's B200 (tools/microbench.cu, profiles/microbench_r01.txt): 3.9 warp-instructions / clk / SM
ISSUE_PEAK_TOPS = 148 * 3.9 * 32 * 1.965e9 / 1e12          # 36.3 T lane-ops/s
OPS_PER_EVAL = 10                                            # SURVEY 8(d): ops per pixel*disparity evaluation


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cost", default="abs", choices=list(COSTS))
    ap.add_argument("--size", type=int, default=8192)
    ap.add_argument("--search", type=int, default=128)
    ap.add_argument("--kernel", type=int, default=21)
    ap.add_argument("--seed", type=int, default=106)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only (skip the other BASELINE configurations)")
    ap.add_argument("--cfg5-size", type=int, default=0, help="run config 5 at this raster size on any N > 1 (default: 16384 at N = 8 only)")
    ap.add_argument("--cpu-tile", type=int, default=0, help="output tile per CPU thread of the reference arm (0 = the largest of "
                    "1024 / 512 / 256 / 128 whose step stays near 12 s; BASELINE.md asks for 1024^2 tiles)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline disparity of the last timed step as float32 .npy "
                    "files under DIR (a fixed sample of rows when the whole raster is larger than DUMP_BYTES); --gpus 1 only")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.gpus != 1 or a.impl != "ours"):
        ap.error("--dump-outputs needs --gpus 1 and --impl ours")
    return a


DUMP_BYTES = 48 << 20          # float32 disparity rows written by --dump-outputs (the row index adds a few KB)


def dump_outputs(d, disp):
    """disparity.npy: float32 (n, W, 3) {dx, dy, valid} rows of the (H, W, 3) int32 result; disparity_rows.npy: float64 (n,)
    the row of each.  All rows when they fit in DUMP_BYTES, else a sorted sample drawn with a fixed seed, so that two
    builds run with the same arguments write the same rows."""
    H, W = disp.shape[:2]
    n = min(H, max(1, DUMP_BYTES // (W * 3 * 4)))
    rows = np.arange(H) if n == H else np.sort(np.random.default_rng(0).choice(H, n, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "disparity.npy"), disp[rows].astype(np.float32))
    np.save(os.path.join(d, "disparity_rows.npy"), rows.astype(np.float64))


def workload_name(a):
    return (f"calc_disparity single level {a.size}x{a.size}, search {a.search}x{a.search}, kernel {a.kernel}x{a.kernel}, "
            f"cost {a.cost.upper()}, synthetic 12-bit integer-valued pair (seed {a.seed})")


def gen_rasters(a):
    from visionworkbench_b200.synth import make_rasters
    return make_rasters(a.size, a.size, (a.search, a.search), (a.kernel, a.kernel), seed=a.seed)


def _cgroup_cpu_limit():
    """CPU quota of this container in cores (cgroup v2 cpu.max / v1 cfs quota), or None"""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return float(q) / float(p)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / p
    except Exception:
        pass
    return None


_CORES = None
_T64 = None          # seconds one thread needs for a 64 x 64 output tile with the full window (from the calibration)


def host_cores():
    """Threads the CPU arm uses = the cores this process can really run on: the affinity mask (torchrun's
    OMP_NUM_THREADS=1 says nothing about the machine), capped by the container's CPU quota, and checked by a short
    calibration (n threads x one 64^2 tile each against one thread x one tile): a box whose lease owns fewer cores than its
    mask shows (round 1: 128 in the mask, ~2 usable) would otherwise time 128 threads fighting over 2 cores."""
    global _CORES, _T64
    if _CORES is not None:
        return _CORES
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    lim = _cgroup_cpu_limit()
    if lim:
        n = max(1, min(n, int(lim + 0.5)))
    try:
        import oracle
        oracle.build()
        from visionworkbench_b200.synth import make_rasters
        t, s, k = 64, 128, 21
        best, best_n, cand = 0.0, 1, n
        while cand >= 1:                      # n, n/2, n/4, ...: keep the thread count with the highest tile throughput
            per_row = min(cand, 16)
            rows = (cand + per_row - 1) // per_row
            l, r = make_rasters(per_row * t, rows * t, (s, s), (k, k), seed=1)
            t0 = time.perf_counter()
            oracle.calc_disparity_tiled(0, l, r, (s, s), (k, k), tile=t, nthreads=cand)
            thr = per_row * rows / (time.perf_counter() - t0)
            if thr > best * 1.05:
                best, best_n = thr, cand
                _T64 = cand / thr
            if cand == 1:
                break
            cand //= 2
        n = best_n
    except Exception:
        pass
    _CORES = n
    return n


# ------------------------------------------------------------------------------------------------
# CPU side: the reference algorithm (oracle restatement) on the host cores, bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_tile_size(a):
    if a.cpu_tile:
        return a.cpu_tile
    host_cores()
    t64 = (_T64 or 0.2) * (a.search * a.search) / (128.0 * 128.0)
    for t in (1024, 512, 256):
        if t64 * (t / 64.0) ** 2 <= 12.0 and t <= a.size:
            return t
    return 128


def cpu_sample(a, left, right, nthreads, tile):
    """`nthreads` output tiles of tile x tile pixels from the CENTRE of the raster, each with the full search window,
    one tile per thread -- the reference's parallelisation (independent tiles on a FIFO pool, Image/ImageIO.h:289-311;
    BASELINE.md section 2).  Returns (pixels, seconds)."""
    import oracle
    k, s = a.kernel, a.search
    per_row = max(1, min(nthreads, a.size // tile))
    rows = (nthreads + per_row - 1) // per_row
    Wc, Hc = per_row * tile, min(rows * tile, a.size)
    x0, y0 = max(0, (a.size - Wc) // 2), max(0, (a.size - Hc) // 2)
    l = np.ascontiguousarray(left[y0:y0 + Hc + k - 1, x0:x0 + Wc + k - 1])
    r = np.ascontiguousarray(right[y0:y0 + Hc + k - 1 + s - 1, x0:x0 + Wc + k - 1 + s - 1])
    t0 = time.perf_counter()
    oracle.calc_disparity_tiled(COSTS[a.cost], l, r, (s, s), (k, k), tile=tile, nthreads=nthreads)
    return Wc * Hc, time.perf_counter() - t0


def cpu_measure(a, left, right, budget_s=25.0):
    """best-of-3 (time permitting) at all host cores + one run at the reference's default of 4 threads"""
    import oracle
    oracle.build()
    n = host_cores()
    tile = cpu_tile_size(a)
    runs, t_used = [], 0.0
    while len(runs) < 3 and (not runs or t_used + runs[-1][1] < budget_s):
        p, dt = cpu_sample(a, left, right, n, tile)
        runs.append((p, dt))
        t_used += dt
    best = max(p / dt for p, dt in runs) / 1e6
    p4, dt4 = cpu_sample(a, left, right, min(4, n), tile)
    return {"value": best, "unit": "Mpix/s", "cores": n, "kind": "port",
            "sample": f"{n} centre tiles of {tile}x{tile} output pixels (one per thread), full {a.search}x{a.search} window, best of {len(runs)}",
            "runs_mpix_s": [round(p / dt / 1e6, 4) for p, dt in runs],
            "value_4_threads": p4 / dt4 / 1e6, "note_4_threads": "VW_NUM_THREADS default of the reference build (src/vw/CMakeLists.txt:27)"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    n = host_cores()
    tile = cpu_tile_size(a)
    left, right = gen_rasters(a)
    for _ in range(min(a.warmup, 1)):
        cpu_sample(a, left, right, n, tile)
    pix, t, per = 0, 0.0, []
    for _ in range(a.steps):
        p, dt = cpu_sample(a, left, right, n, tile)
        pix += p
        t += dt
        per.append(p / dt / 1e6)
    v = pix / t / 1e6
    p4, dt4 = cpu_sample(a, left, right, min(4, n), tile)
    line = {
        "impl": "reference", "metric": "disparity Mpix/s", "value": v, "unit": "Mpix/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * t / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 cost / f64 sums", "data": "synthetic",
        "config": {"workload": workload_name(a), "note": "reference algorithm (CPU restatement of best_of_search_convolution; the "
                   "reference itself cannot be compiled here: no Boost/GDAL headers), tile-parallel like block_write_image"},
        "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": n, "kind": "port",
                         "sample": f"per step: {n} centre tiles of {tile}x{tile} output pixels (one per thread), full {a.search}x{a.search} window; "
                                   f"threads = usable cores (affinity mask capped by the CPU quota, calibrated)",
                         "steps_mpix_s": [round(x, 4) for x in per], "best_step": max(per),
                         "value_4_threads": p4 / dt4 / 1e6},
        "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.idx = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [ln.split(",") for ln in open(self.f.name).read().strip().splitlines() if ln.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows)
        out["sm_mhz"] = sm[len(sm) // 2]
        out["sm_max_mhz"] = float(rows[0][2])
        out["power_w_max"] = max(float(r[3]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, n in enumerate(names):
            if any(r[5 + i].strip().lower().startswith("active") for r in rows):
                out["reasons"].append(n)
        out["samples"] = len(rows)
        return out


def hbm_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if p.get("hbm_gbs"):
            return float(p["hbm_gbs"]), "measured"
    except Exception:
        pass
    return 6650.0, "fallback"


def alu_roofline(evals, kernel_ms, alg_bytes, kernel):
    peak, which = hbm_peak()
    tops = evals * OPS_PER_EVAL / (kernel_ms * 1e-3) / 1e12
    return {"bound": "alu", "achieved": tops, "peak": ISSUE_PEAK_TOPS, "unit": "Tlane-op/s", "frac": tops / ISSUE_PEAK_TOPS,
            "peak_is": "measured issue rate: 148 SM x 3.9 warp-instr/clk x 32 lanes x 1.965 GHz (profiles/microbench_r01.txt)",
            "ops_per_eval": OPS_PER_EVAL, "evals_per_launch": evals, "achieved_Teval_s": evals / (kernel_ms * 1e-3) / 1e12,
            "kernel": kernel, "kernel_ms": kernel_ms,
            "hbm": {"achieved": alg_bytes / (kernel_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / peak,
                    "peak_is": which, "algorithmic_bytes_per_launch": alg_bytes}}


def oracle_tile_check(cost, left, right, out_np, search, kernel, tiles, t):
    """compare sampled output tiles with the oracle (calc_disparity is local: crops suffice)"""
    import oracle
    oracle.build()
    sx, sy = search
    kx, ky = kernel

    def one(o):
        x, y = o
        l = np.ascontiguousarray(left[y:y + t + ky - 1, x:x + t + kx - 1])
        r = np.ascontiguousarray(right[y:y + t + ky - 1 + sy - 1, x:x + t + kx - 1 + sx - 1])
        ref = oracle.calc_disparity(cost, l, r, search, kernel)
        return int((ref != out_np[y:y + t, x:x + t]).any(-1).sum())
    with cf.ThreadPoolExecutor(max_workers=min(len(tiles), host_cores())) as ex:
        return sum(ex.map(one, tiles))


# ------------------------------------------------------------------------------------------------
# the other BASELINE configurations (N = 1, rank 0, device resident)
# ------------------------------------------------------------------------------------------------
def time_calc(v, cost, dl, dr, s, k, steps=2, warmup=1):
    import torch
    for _ in range(warmup):
        out = v.calc_disparity(cost, dl, dr, (s, s), (k, k))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kms = []
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        out = v.calc_disparity(cost, dl, dr, (s, s), (k, k))
        kms.append(v.last_k1_stats()["kernel_ms"])
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1) / steps, float(np.mean(kms)), v.last_k1_stats()["path"]


def cfg_calc(v, name, cost_name, size, s, k, seed, left=None, right=None, tiles=2):
    import torch
    from visionworkbench_b200.synth import make_rasters
    if left is None:
        left, right = make_rasters(size, size, (s, s), (k, k), seed=seed)
    dl, dr = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
    out, ms, kms, path = time_calc(v, COSTS[cost_name], dl, dr, s, k)
    evals = size * size * s * s
    kern = "k1_fast_abs_kernel" if (cost_name == "abs" and path == "exact-int") else ("k1_screen_kernel" if path == "exact-int" else "k1_generic_kernel")
    rng = np.random.default_rng(seed)
    tl = [(int(rng.integers(0, size - 127)), int(rng.integers(0, size - 127))) for _ in range(tiles)]
    bad = oracle_tile_check(COSTS[cost_name], left, right, out.cpu().numpy(), (s, s), (k, k), tl, 128) if tiles else None
    del dl, dr, out
    torch.cuda.empty_cache()
    return {"workload": f"calc_disparity {size}x{size}, search {s}x{s}, kernel {k}x{k}, cost {cost_name.upper()} (seed {seed})",
            "ms": ms, "Mpix_s": size * size / ms / 1e3, "kernel_path": path, "kernel_share_of_step": kms / ms,
            "roofline": alu_roofline(evals, kms, size * size * 20, kern),
            "parity_sample": {"tiles": tiles, "tile": 128, "mismatches": bad}}


def cfg3_view(v, size=8192, tile=1024, threads=16):
    """config 3: PyramidCorrelationView, 5 levels, SquaredCost 15x15, 128x128 window, L/R check 2, filter radius 5, 1024^2
    tiles rasterised from `threads` host threads (the reference's block_write_image pattern), device-resident inputs"""
    import torch
    from visionworkbench_b200.synth import make_pair
    search, kernel = (-64, -64, 64, 64), (15, 15)
    left, right, lm, rm, _ = make_pair(size, size, search, seed=103)
    dl, dr = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
    dlm, drm = torch.from_numpy(lm).cuda(), torch.from_numpy(rm).cuda()
    view = v.pyramid_correlate(dl, dr, dlm, drm, v.PREFILTER_NONE, 0.0, search, kernel, v.SQUARED_DIFFERENCE, 0, 0.0, 2.0, 0, 5, 5)
    out = torch.empty((size, size, 3), dtype=torch.float32, device="cuda")
    boxes = [(x, y, min(x + tile, size), min(y + tile, size)) for y in range(0, size, tile) for x in range(0, size, tile)]
    streams = [torch.cuda.Stream() for _ in range(threads)]

    def work(i):
        with torch.cuda.stream(streams[i % threads]):
            for b in boxes[i::threads]:
                view.rasterize(out[b[1]:b[3], b[0]:b[2]], b)

    def run():
        n0 = v.kernel_launches()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(work, range(threads)))
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, v.kernel_launches() - n0
    run()
    ms, launches = min((run() for _ in range(2)), key=lambda r: r[0])
    peak, which = hbm_peak()
    alg = size * size * 110                      # SURVEY 8(d): ~110 B per output pixel
    valid = float((out[..., 2] == 1).float().mean())
    # parity of one tile against the oracle on a crop (the pyramid reads bbox +- 224 + search 64)
    import oracle
    oracle.build()
    m, b = 512, boxes[len(boxes) // 2 + 1]
    x0, y0, x1, y1 = max(b[0] - m, 0), max(b[1] - m, 0), min(b[2] + m, size), min(b[3] + m, size)
    sub = 256                                    # a 256^2 window of the tile keeps the CPU check short
    bb = (b[0] + 300, b[1] + 300, b[0] + 300 + sub, b[1] + 300 + sub)
    view2 = v.pyramid_correlate(dl, dr, dlm, drm, v.PREFILTER_NONE, 0.0, search, kernel, v.SQUARED_DIFFERENCE, 0, 0.0, 2.0, 0, 5, 5)
    got = view2.rasterize(None, bb).cpu().numpy()
    p = oracle.make_params(search, kernel, cost=1, consistency_threshold=2.0, filter_half_kernel=5, max_pyramid_levels=5)
    ref = oracle.pyramid_correlate(p, left[y0:y1, x0:x1], right[y0:y1, x0:x1], lm[y0:y1, x0:x1], rm[y0:y1, x0:x1],
                                   bbox=(bb[0] - x0, bb[1] - y0, bb[2] - x0, bb[3] - y0))
    bad = int((got != ref).any(-1).sum())
    del view, view2, dl, dr, dlm, drm, out
    torch.cuda.empty_cache()
    return {"workload": f"PyramidCorrelationView 5 levels, {size}x{size}, SquaredCost 15x15, window 128x128, L/R check 2, filter r=5, "
                        f"{tile}x{tile} tiles from {threads} host threads (seed 103)",
            "ms": ms, "Mpix_s": size * size / ms / 1e3, "gpu_launches": launches, "valid_fraction": valid,
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak,
                         "peak_is": which, "algorithmic_bytes_per_launch": alg, "note": "110 B per output pixel (SURVEY 8d); wall time of the whole tile loop"},
            "parity_sample": {"tiles": 1, "tile": sub, "mismatches": bad}}


def cfg4_sgm(v, size=4096, search=128):
    """config 4: SemiGlobalMatcher, census 5, 8 paths, per-pixel boxes from a half-resolution prior, search_buffer (2, 2)"""
    import torch
    from visionworkbench_b200 import api
    from visionworkbench_b200.synth import make_sgm_case
    left, right, prev, true = make_sgm_case(size, search, 5, seed=104)
    dl, dr, dp = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda(), torch.from_numpy(prev).cuda()
    sp = api._sgm_params((search, search), 5, api.CENSUS_TRANSFORM, False, api.SUBPIXEL_LC_BLEND, (2, 2), 1e9)
    ow, oh = C.c_int(0), C.c_int(0)
    L = v.lib()
    head = (C.byref(sp), dl.data_ptr(), dl.shape[1], dl.shape[0], dl.stride(0), dr.data_ptr(), dr.shape[1], dr.shape[0], dr.stride(0))
    api._check(L.vwb200_sgm_calc_disparity_ex(*head, None, 0, None, 0, 0, 0, None, 0, 0, 0, None, None, 0, None, 0, None, C.byref(ow), C.byref(oh), 1, None))
    out = torch.empty((oh.value, ow.value, 3), dtype=torch.int32, device="cuda")
    sub = torch.empty((oh.value, ow.value, 3), dtype=torch.float32, device="cuda")

    def run():
        n0 = v.kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        api._check(L.vwb200_sgm_calc_disparity_ex(*head, None, 0, None, 0, 0, 0, dp.data_ptr(), dp.shape[1], dp.shape[0], dp.stride(0) // 3, None,
                                                  out.data_ptr(), ow.value, sub.data_ptr(), ow.value, None, C.byref(ow), C.byref(oh), 1,
                                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), v.kernel_launches() - n0
    run()
    ms, launches = min((run() for _ in range(3)), key=lambda r: r[0])
    o = out.cpu().numpy()
    t = true[2:2 + oh.value, 2:2 + ow.value]
    ok = float(((o[..., 0] == t[..., 0]) & (o[..., 1] == t[..., 1]) & (o[..., 2] == 1)).mean())
    npx = oh.value * ow.value
    # parity: the oracle on a crop of the problem (a 192^2 window with its own prior) -- the whole pipeline through the C ABI
    import oracle
    oracle.build()
    cs = 192
    l2 = np.ascontiguousarray(left[:cs, :cs])
    r2 = np.ascontiguousarray(right[:cs + search, :cs + search])
    oh2, ow2 = oracle.sgm_output_shape(l2, r2, (search, search), 5)
    pv2 = np.ascontiguousarray(prev[:(oh2 + 1) // 2, :(ow2 + 1) // 2])
    gi, gf = v.calc_disparity_sgm_ex(v.CENSUS_TRANSFORM, l2, r2, (search, search), 5, subpixel_mode=5, prev_disparity=pv2, memory_limit_mb=1e9)
    ri, rf, _ = oracle.calc_disparity_sgm(l2, r2, (search, search), 5, subpixel_mode=5, prev=pv2, memory_limit_mb=1e9)
    bad = int((gi != ri).any(-1).sum()) + int((np.abs(gf - rf) > 1e-5).any(-1).sum())
    peak, which = hbm_peak()
    alg = npx * 25 * 41
    del dl, dr, dp, out, sub
    torch.cuda.empty_cache()
    return {"workload": f"SemiGlobalMatcher census 5x5, 8 paths, {size}x{size}, window [0,{search}]^2, 5x5 boxes from a half-resolution prior "
                        "(search_buffer (2,2)), LC_BLEND sub-pixel (seed 104)",
            "ms": ms, "Mpix_s": npx / ms / 1e3, "gpu_launches": launches, "correct_fraction": ok,
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak,
                         "peak_is": which, "algorithmic_bytes_per_launch": alg,
                         "note": "reference-equivalent traffic 41 B per (pixel, disparity) x 25 (SURVEY 8d); whole pipeline (u8, census, boxes, costs, 8 paths, WTA)",
                         "fused_minimum_frac": npx * 275 / (ms * 1e-3) / 1e9 / peak},
            "parity_sample": {"tiles": 1, "tile": cs, "mismatches": bad}}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def sharded_calc(v, comm, left_band, right_band, p, world, cost, s, k, steps, warmup, dist, torch):
    """the sharded calc_disparity loop: halo exchange + kernel per step; returns (ms total max over ranks, kernel_ms list, out)"""
    def step():
        comm.exchange_halos(p, left_band, right_band)          # ncclSend / ncclRecv behind the C ABI, on the current stream
        return v.calc_disparity(cost, left_band, right_band, (s, s), (k, k))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        out = step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kms = []
    e0.record()
    for _ in range(steps):
        out = step()
        kms.append(v.last_k1_stats()["kernel_ms"])
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), kms, out


def cfg5_sharded(v, comm, world, rank, dist, torch, size=16384, s=256, k=15):
    """config 5: 16384^2 ortho pair, Abs 15x15, 256x256 window, tile-row bands over the ranks, NCCL halo rows.  Each rank
    synthesises the rows it owns (seed 105 + rank); the halo rows arrive from the neighbour over NVLink every step."""
    from visionworkbench_b200 import sharding
    from visionworkbench_b200.synth import make_rasters
    p = sharding.plan(rank, world, size, k, s)
    H = p.y1 - p.y0
    own_l, own_r = make_rasters(size, H, (s, s), (k, k), seed=105 + rank)      # (H + k - 1) and (H + k - 1 + s - 1) rows: covers the owned rows
    dl = torch.zeros((p.left_rows, own_l.shape[1]), dtype=torch.float32, device="cuda")
    dr = torch.zeros((p.right_rows, own_r.shape[1]), dtype=torch.float32, device="cuda")
    dl[:p.own_left].copy_(torch.from_numpy(own_l[:p.own_left]))
    dr[:p.own_right].copy_(torch.from_numpy(own_r[:p.own_right]))
    ms, kms, out = sharded_calc(v, comm, dl, dr, p, world, 0, s, k, 2, 1, dist, torch)
    ms /= 2
    bad = None
    if rank == 0:      # parity of sampled tiles on rank 0 (rows assembled from its own band + the received halo)
        L, R = dl.cpu().numpy(), dr.cpu().numpy()
        tiles = [(0, 0), (size - 128, H - 128), (min(236 * 11 - 64, size - 128), H - 128), (min(5000, size - 128), 32 * 7 - 64)]
        bad = oracle_tile_check(0, L, R, out.cpu().numpy(), (s, s), (k, k), tiles, 128)
    evals = size * size * s * s
    kmean = float(np.mean(kms))
    return {"workload": f"calc_disparity {size}x{size}, search {s}x{s}, kernel {k}x{k}, cost ABS, {world} tile-row bands with NCCL halo rows (seed 105+rank)",
            "ms": ms, "Mpix_s": size * size / ms / 1e3, "kernel_ms_rank0": kmean, "halo_bytes_per_boundary": int((k - 1) * dl.shape[1] * 4 + (k - 1 + s - 1) * dr.shape[1] * 4),
            "roofline": alu_roofline(evals // world, kmean, size * H * 20, "k1_fast_abs_kernel"),
            "parity_sample": {"tiles": 4, "tile": 128, "mismatches": bad}}


def cfg3_sharded(v, world, rank, dist, torch, size=8192, tile=1024, threads=8):
    """config 3 over N GPUs: the 1024^2 tiles of the view are the units, tile rows are split over the ranks, no data-path
    collective -- every rank holds the rows of its tiles plus the margin the pyramid padding and the search window reach
    (a real ortho pair would be read from the file that way).  Each rank synthesises its band (seed 103 + rank)."""
    import concurrent.futures as cf2
    from visionworkbench_b200.synth import make_pair
    search, kernel = (-64, -64, 64, 64), (15, 15)
    rows = size // world
    m = 512                                                   # >= 15/2 * 2^5 (pyramid padding) + 64 (search) rows of margin
    y0, y1 = rank * rows, (rank + 1) * rows
    top, bot = min(m, y0), min(m, size - y1)
    ok, err = 1, None
    try:
        left, right, lm, rm, _ = make_pair(size, rows + top + bot, search, seed=103 + rank)
        dl, dr = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
        dlm, drm = torch.from_numpy(lm).cuda(), torch.from_numpy(rm).cuda()
        view = v.pyramid_correlate(dl, dr, dlm, drm, v.PREFILTER_NONE, 0.0, search, kernel, v.SQUARED_DIFFERENCE, 0, 0.0, 2.0, 0, 5, 5)
        out = torch.empty((rows, size, 3), dtype=torch.float32, device="cuda")
        view.rasterize(out[:64, :64], (0, top, 64, top + 64))      # one small tile before anybody waits in a collective
    except Exception as e:
        ok, err = 0, e
    flag = torch.tensor([ok], device="cuda", dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)                   # every rank is ready, or nobody enters the timed loop
    if int(flag.item()) == 0:
        raise RuntimeError(f"config 3 set-up failed on a rank: {err!r}")
    boxes = [(x, top + y, min(x + tile, size), top + min(y + tile, rows)) for y in range(0, rows, tile) for x in range(0, size, tile)]
    streams = [torch.cuda.Stream() for _ in range(threads)]

    def work(i):
        with torch.cuda.stream(streams[i % threads]):
            for b in boxes[i::threads]:
                view.rasterize(out[b[1] - top:b[3] - top, b[0]:b[2]], b)

    def run():
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        with cf2.ThreadPoolExecutor(max_workers=threads) as ex:
            list(ex.map(work, range(threads)))
        torch.cuda.synchronize()
        t = torch.tensor([(time.perf_counter() - t0) * 1e3], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    run()
    ms = min(run() for _ in range(2))
    bad = None
    if rank == 0:
        import oracle
        oracle.build()
        b = boxes[min(1, len(boxes) - 1)]
        bb = (b[0] + 300, b[1] + 300, b[0] + 556, b[1] + 556)
        x0, yy0, x1, yy1 = max(bb[0] - 512, 0), max(bb[1] - 512, 0), min(bb[2] + 512, size), min(bb[3] + 512, left.shape[0])
        got = view.rasterize(None, bb).cpu().numpy()
        pp = oracle.make_params(search, kernel, cost=1, consistency_threshold=2.0, filter_half_kernel=5, max_pyramid_levels=5)
        ref = oracle.pyramid_correlate(pp, left[yy0:yy1, x0:x1], right[yy0:yy1, x0:x1], lm[yy0:yy1, x0:x1], rm[yy0:yy1, x0:x1],
                                       bbox=(bb[0] - x0, bb[1] - yy0, bb[2] - x0, bb[3] - yy0))
        bad = int((got != ref).any(-1).sum())
    del view, dl, dr, dlm, drm, out
    torch.cuda.empty_cache()
    return {"workload": f"PyramidCorrelationView 5 levels, {size}x{size}, SquaredCost 15x15, window 128x128, L/R check 2, filter r=5: "
                        f"{len(boxes)} tiles of {tile}^2 per rank ({world} tile-row bands, rows + {m}-row margins resident per rank, no collective), "
                        f"{threads} host threads per rank (seed 103+rank)",
            "ms": ms, "Mpix_s": size * size / ms / 1e3, "parity_sample": {"tiles": 1, "tile": 256, "mismatches": bad}}


def run_ours(a):
    import torch
    import torch.distributed as dist
    import visionworkbench_b200 as v

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's version / INFO lines) is sent to stderr by
    # pointing fd 1 at fd 2 for the run; the JSON line is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ["NCCL_DEBUG"] = "INFO"              # communicator size, rings, NVLS: on stderr for the driver's rank check
        os.environ.pop("NCCL_DEBUG_FILE", None)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert v.device_count() > 0
    cost = COSTS[a.cost]
    k, s, S = a.kernel, a.search, a.size
    left, right = gen_rasters(a)                        # same seed on every rank
    # ---- shard output rows into bands; each rank OWNS the input rows of its band (visionworkbench_b200/sharding.py) ----
    from visionworkbench_b200 import sharding
    p = sharding.plan(rank, world, S, k, s, left.shape[0], right.shape[0])
    y0, y1, H = p.y0, p.y1, p.y1 - p.y0
    lh_need, rh_need = p.left_rows, p.right_rows          # rows this rank's kernel launch reads
    dl = torch.empty((lh_need, left.shape[1]), dtype=torch.float32, device="cuda")
    dr = torch.empty((rh_need, right.shape[1]), dtype=torch.float32, device="cuda")
    dl.zero_(); dr.zero_()
    dl[:p.own_left].copy_(torch.from_numpy(left[y0:y0 + p.own_left]))
    dr[:p.own_right].copy_(torch.from_numpy(right[y0:y0 + p.own_right]))

    # the halo rows travel through the C ABI (vwb200_shard_exchange_halos: ncclSend / ncclRecv in one group); torch.distributed
    # only hands rank 0's NCCL id to the other ranks and carries the timing reductions
    comm = sharding.ShardComm(rank, world, sharding.torch_broadcast if world > 1 else None)

    def step_device():
        comm.exchange_halos(p, dl, dr)
        return v.calc_disparity(cost, dl, dr, (s, s), (k, k))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- host-resident copies for the e2e leg (pinned) ----
    hl = torch.empty((lh_need, left.shape[1]), dtype=torch.float32, pin_memory=True)
    hr = torch.empty((rh_need, right.shape[1]), dtype=torch.float32, pin_memory=True)
    hl.copy_(torch.from_numpy(left[y0:y0 + lh_need]))
    hr.copy_(torch.from_numpy(right[y0:y0 + rh_need]))
    hout = torch.empty((H, S, 3), dtype=torch.int32, pin_memory=True)
    hl_np, hr_np, hout_np = hl.numpy(), hr.numpy(), hout.numpy()
    L = v.lib()

    def step_e2e():
        rc = L.vwb200_calc_disparity(cost, hl_np.ctypes.data, hl_np.shape[1], hl_np.shape[0], hl_np.shape[1],
                                     hr_np.ctypes.data, hr_np.shape[1], hr_np.shape[0], hr_np.shape[1],
                                     s, s, k, k, hout_np.ctypes.data, S, 0, None)
        if rc:
            raise RuntimeError(L.vwb200_last_error().decode())

    # ---- warm-up ----
    for _ in range(a.warmup):
        out = step_device()
    path = v.last_k1_stats()["path"]
    # ---- timed: device-resident ----
    clocks = Clocks(local)
    barrier()
    if rank == 0:
        clocks.start()
    n0 = v.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    e0.record()
    for _ in range(a.steps):
        out = step_device()
        kernel_ms.append(v.last_k1_stats()["kernel_ms"])
    e1.record()
    barrier()
    launches = v.kernel_launches() - n0
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    nl = torch.tensor([float(launches)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(nl, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    value = S * S * a.steps / (ms * 1e-3) / 1e6
    # ---- timed: end to end through the C ABI with host buffers ----
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step_e2e()
    torch.cuda.synchronize()
    te = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([te], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    te = float(t.item())
    e2e = S * S * a.steps / (te * 1e-3) / 1e6
    out_np = out.cpu().numpy()
    same = bool(np.array_equal(hout_np, out_np))         # the e2e result must equal the device-resident result
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, out_np)
    # ---- sampled-tile parity of this run against the oracle (rank 0's band) ----
    parity = None
    if rank == 0:
        rng = np.random.default_rng(a.seed)
        tl = [(0, 0), (S - 128, H - 128)] + [(int(rng.integers(0, S - 127)), int(rng.integers(0, H - 127))) for _ in range(2)]
        Lb, Rb = dl.cpu().numpy(), dr.cpu().numpy()
        parity = {"tiles": len(tl), "tile": 128, "mismatches": oracle_tile_check(cost, Lb, Rb, out_np, (s, s), (k, k), tl, 128)}
    configs = {}
    del out
    if world > 1 and (world == 8 or a.cfg5_size) and not a.no_configs:
        try:
            configs["cfg5"] = cfg5_sharded(v, comm, world, rank, dist, torch, size=a.cfg5_size or 16384)
        except Exception as e:          # never lose the headline line to a side measurement
            configs["cfg5"] = {"error": repr(e)[:300]}
    if world > 1 and not a.no_configs:
        try:
            configs["cfg3"] = cfg3_sharded(v, world, rank, dist, torch)
        except Exception as e:
            configs["cfg3"] = {"error": repr(e)[:300]}
    if rank == 0:
        kms = float(np.mean(kernel_ms))
        alg_bytes = H * S * (4 + 4 + 12)                 # SURVEY 8(d): left + right + 12-byte disparity pixel
        evals = H * S * s * s
        kname = "k1_generic_kernel" if path != "exact-int" else ("k1_fast_abs_kernel" if a.cost == "abs" else "k1_screen_kernel")
        traffic = None
        try:          # measured once under ncu for the default workload; null for any other
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic_r01.json"))).get(f"{kname}|{S}|{s}|{a.kernel}|{a.cost}")
            if tr and world == 1:
                traffic = tr["dram_read_bytes"] + tr["dram_write_bytes"]
        except Exception:
            pass
        roof = alu_roofline(evals, kms, alg_bytes, kname)
        roof["traffic"] = traffic
        roof["traffic_unit"] = "DRAM bytes per launch (ncu, profiles/traffic_r01.json)"
        roof["kernel_share_of_step"] = kms * a.steps / ms if world == 1 else None
        roof["note"] = ("ALU/issue-bound by construction (SURVEY 8d): ~10 issue slots per pixel*disparity vs 20 B per pixel; "
                        "frac = evaluations x 10 / measured issue peak, the HBM figures sit under 'hbm'")
        line = {
            "metric": "disparity Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32 on u16 (exact)" if path == "exact-int" else "f32 cost / f64 sums", "data": "synthetic",
            "config": {"workload": workload_name(a), "kernel_path": path, "l2": "inputs larger than L2 (2 x 270 MB rasters, 805 MB output)",
                       "parallelism": f"{world} output-row band(s), halo rows by ncclSend/ncclRecv behind the C ABI" if world > 1 else "1 GPU, persistent CTAs",
                       "e2e_equals_device_result": same},
            "e2e": {"value": e2e, "unit": "Mpix/s", "h2d_bytes_per_step": int(hl_np.nbytes + hr_np.nbytes),
                    "d2h_bytes_per_step": int(hout_np.nbytes), "ms_per_step": te / a.steps, "bytes_are": "per rank"},
            "gpu_launches": int(nl.item()),
            "clocks": clk,
            "roofline": roof,
            "parity_sample": parity,
        }
        if world == 1 and not a.no_configs and a.cost == "abs" and S == 8192:
            del dl, dr
            torch.cuda.empty_cache()
            t0 = time.perf_counter()
            for name, fn in [("ns_sq", lambda: cfg_calc(v, "ns_sq", "sq", 8192, 128, 21, 106, left, right)),
                             ("ns_ncc", lambda: cfg_calc(v, "ns_ncc", "ncc", 8192, 128, 21, 106, left, right)),
                             ("cfg2", lambda: cfg_calc(v, "cfg2", "ncc", 4096, 128, 21, 102)),
                             ("cfg3", lambda: cfg3_view(v)), ("cfg4", lambda: cfg4_sgm(v))]:
                try:
                    configs[name] = fn()
                except Exception as e:      # never lose the headline line to a side measurement
                    configs[name] = {"error": repr(e)[:300]}
            configs["wall_s"] = time.perf_counter() - t0
        if configs:
            line["configs"] = configs
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_measure(a, left, right)
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    comm.close()
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.close(real_stdout)        # fd 1 keeps pointing at stderr: NCCL still prints INFO lines while the process exits


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
