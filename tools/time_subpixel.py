"""Throughput of PyramidSubpixelView (LK / affine / Bayes-EM) on one GPU; prints one JSON line.

Input: a 4096^2 smooth random pair scaled to [0,1] with a sub-pixel shift, a seeded integer starting disparity with about
5 % invalid pixels.  For each algorithm and kernel (7x7 as in the reference's tests, 35x35 as in its SlipTest) the full
image is rasterised in 1024^2 tiles (device-resident inputs, default 2 pyramid levels) after one warm-up tile; the best of
--reps runs is reported, synchronised on the device.  The counters of vwb200_last_subpixel_stats give window evaluations
per second, SIMT efficiency (window evaluations / lane slots) and validity-fixpoint rounds.  parity_sample: one tile
recomputed by the CPU oracle (256^2 for 7x7, 64^2 for 35x35), compared bit for bit; the oracle's single-thread Mpix/s on
that tile is reported beside it.

    python tools/time_subpixel.py [--size 4096] [--tile 1024] [--reps 2] [--out profiles/subpixel_r03.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def make_pair(n, seed=1):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.rand((n // 8 + 4, n // 8 + 4), generator=g, device="cuda")
    img = torch.nn.functional.interpolate(base[None, None], scale_factor=8, mode="bicubic", align_corners=False)[0, 0, :n, :n]
    img = (img - img.min()) / (img.max() - img.min())
    # the right image is the left shifted by (1.4, -0.3) pixels (bilinear resampling)
    ys, xs = torch.meshgrid(torch.arange(n, device="cuda", dtype=torch.float32), torch.arange(n, device="cuda", dtype=torch.float32),
                            indexing="ij")
    grid = torch.stack(((xs - 1.4) / (n - 1) * 2 - 1, (ys + 0.3) / (n - 1) * 2 - 1), -1)[None]
    right = torch.nn.functional.grid_sample(img[None, None], grid, mode="bilinear", align_corners=True)[0, 0]
    disp = torch.zeros((n, n, 3), device="cuda")
    disp[..., 0] = 1.0
    disp[..., 2] = (torch.rand((n, n), generator=g, device="cuda") > 0.05).float()
    return img.contiguous(), right.contiguous(), disp.contiguous()


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits"], capture_output=True, text=True,
                           timeout=20)
        return float(r.stdout.strip().splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--tile", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--kernels", default="7,35")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import visionworkbench_b200 as v
    from oracle import subpixel
    L = v.lib()
    n, t = a.size, a.tile
    left, right, disp = make_pair(n)
    names = {0: "lk", 1: "affine", 2: "bayes_em"}
    res = {"metric": "PyramidSubpixelView Mpix/s", "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(),
           "size": n, "tile": t, "levels": 2, "prefilter": "LOG 1.4", "configs": []}
    st = torch.cuda.current_stream()

    def run_tile(alg, k, x0, y0, x1, y1, out):
        rc = L.vwb200_pyramid_subpixel(disp.data_ptr(), n, n, left.data_ptr(), n, right.data_ptr(), n, n, n, k, k, 1, 1.4,
                                       x0, y0, x1, y1, out.data_ptr(), x1 - x0, 1, C.c_void_p(st.cuda_stream), 2, alg)
        if rc:
            raise RuntimeError(L.vwb200_last_error().decode())
        return v.last_subpixel_stats()

    for k in [int(s) for s in a.kernels.split(",")]:
        for alg in (0, 1, 2):
            out = torch.empty((t, t, 3), device="cuda")
            run_tile(alg, k, 0, 0, t, t, out)                       # warm-up
            best, tot = None, None
            for _ in range(a.reps):
                agg = {"window_evaluations": 0, "lane_slots": 0, "fixpoint_rounds": 0, "levels": 0, "pixels_reevaluated": 0}
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for y in range(0, n, t):
                    for x in range(0, n, t):
                        s = run_tile(alg, k, x, y, min(x + t, n), min(y + t, n), out)
                        for key in agg:
                            agg[key] += s[key]
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                if best is None or dt < best:
                    best, tot = dt, agg
            ps = 256 if k <= 9 else 64
            x0 = y0 = n // 2
            sub = torch.empty((ps, ps, 3), device="cuda")
            run_tile(alg, k, x0, y0, x0 + ps, y0 + ps, sub)
            hd, hl, hr = disp.cpu().numpy(), left.cpu().numpy(), right.cpu().numpy()
            c0 = time.perf_counter()
            ref = subpixel.pyramid_subpixel(hd, hl, hr, (k, k), 1, 1.4, 2, alg, bbox=(x0, y0, x0 + ps, y0 + ps))
            cdt = time.perf_counter() - c0
            mism = int((sub.cpu().numpy().view(np.uint32) != ref.view(np.uint32)).any(-1).sum())
            res["configs"].append({
                "algorithm": names[alg], "kernel": k, "seconds": best, "mpix_per_s": n * n / best / 1e6,
                "window_evals_per_s": tot["window_evaluations"] / best,
                "simt_efficiency": tot["window_evaluations"] / tot["lane_slots"] if tot["lane_slots"] else 0.0,
                "fixpoint_rounds_per_level": tot["fixpoint_rounds"] / max(tot["levels"], 1),
                "pixels_reevaluated": tot["pixels_reevaluated"],
                "parity_sample": {"tile": ps, "mismatches": mism},
                "oracle_mpix_per_s_1thread": ps * ps / cdt / 1e6, "oracle_cores": os.cpu_count(),
            })
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
