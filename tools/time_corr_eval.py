"""Throughput of CorrEval on one GPU; prints one JSON line.

Input: a 4096^2 smooth random texture and its copy resampled at a (2.3, -0.7) pixel shift, as PixelMask<float> rasters
(all valid), and a smooth fractional disparity around that shift with about 5 % invalid pixels; everything device-resident.
For each metric, kernel (5x5 and 21x21) and round_to_int the full image is rasterised in 1024^2 tiles (sample_rate 1,
prefilter_kernel_width 1.4) into one device buffer after one warm-up tile; the best of --reps runs is reported,
synchronised on the device.  window_samples_per_s counts right-image samples: kx * ky per pixel for ncc, twice that for
stddev (two passes), five times for the curvature metrics.  parity_sample: one 256^2 bbox recomputed by the CPU oracle and
compared bit for bit.  The card's name and power limit are read in the same run.

    python tools/time_corr_eval.py [--size 4096] [--tile 1024] [--reps 3] [--out profiles/corr_eval_r04.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

METRICS = ("ncc", "stddev", "parabola_curvature", "cramer_rao")
PASSES = {"ncc": 1, "stddev": 2, "parabola_curvature": 5, "cramer_rao": 5}
SHIFT = (2.3, -0.7)


def make_scene(n, seed=1):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.rand((n // 8 + 4, n // 8 + 4), generator=g, device="cuda")
    img = torch.nn.functional.interpolate(base[None, None], scale_factor=8, mode="bicubic", align_corners=False)[0, 0, :n, :n]
    ys, xs = torch.meshgrid(torch.arange(n, device="cuda", dtype=torch.float32), torch.arange(n, device="cuda", dtype=torch.float32),
                            indexing="ij")
    grid = torch.stack(((xs - SHIFT[0]) / (n - 1) * 2 - 1, (ys - SHIFT[1]) / (n - 1) * 2 - 1), -1)[None]
    right = torch.nn.functional.grid_sample(img[None, None], grid, mode="bilinear", align_corners=True)[0, 0]
    disp = torch.zeros((n, n, 3), device="cuda")
    disp[..., 0] = SHIFT[0] + 0.4 * torch.sin(xs / 170.0) * torch.cos(ys / 230.0)
    disp[..., 1] = SHIFT[1] + 0.3 * torch.cos(xs / 190.0) * torch.sin(ys / 130.0)
    disp[..., 2] = (torch.rand((n, n), generator=g, device="cuda") > 0.05).float()
    ones = torch.ones_like(img)
    return torch.stack((img, ones), -1).contiguous(), torch.stack((right, ones), -1).contiguous(), disp.contiguous()


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"], capture_output=True,
                           text=True, timeout=20)
        name, pl = r.stdout.strip().splitlines()[0].split(", ")
        return name, float(pl)
    except Exception:
        return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--tile", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernels", default="5,21")
    ap.add_argument("--parity", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import visionworkbench_b200 as v
    from oracle import corr_eval
    n, t, ps = a.size, a.tile, a.parity
    left, right, disp = make_scene(n)
    name, pl = card()
    res = {"metric": "CorrEval Mpix/s", "device": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit_w": pl,
           "size": n, "tile": t, "sample_rate": 1, "prefilter_kernel_width": 1.4, "invalid_fraction": 0.05, "configs": []}
    hl, hr, hd = left.cpu().numpy(), right.cpu().numpy(), disp.cpu().numpy()
    out = torch.empty((n, n, 2), device="cuda")
    for k in [int(s) for s in a.kernels.split(",")]:
        for metric in METRICS:
            for rnd in (False, True):
                view = v.CorrEval(left, right, disp, (k, k), metric, 1, rnd, 0, 1.4)
                view.rasterize(out[:t, :t], (0, 0, t, t))                          # warm-up
                best = None
                for _ in range(a.reps):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for y in range(0, n, t):
                        for x in range(0, n, t):
                            x1, y1 = min(x + t, n), min(y + t, n)
                            view.rasterize(out[y:y1, x:x1], (x, y, x1, y1))
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                x0 = y0 = n // 2
                sub = view.rasterize(None, (x0, y0, x0 + ps, y0 + ps)).cpu().numpy()
                c0 = time.perf_counter()
                ref = corr_eval.corr_eval(hl, hr, hd, (k, k), metric, 1, rnd, 1.4, bbox=(x0, y0, x0 + ps, y0 + ps))
                cdt = time.perf_counter() - c0
                mism = int((sub.view(np.uint32) != ref.view(np.uint32)).any(-1).sum())
                res["configs"].append({
                    "metric": metric, "kernel": k, "round_to_int": rnd, "seconds": best, "mpix_per_s": n * n / best / 1e6,
                    "window_samples_per_s": n * n * k * k * PASSES[metric] / best,
                    "valid_fraction": float(out[..., 1].mean().item()),
                    "parity_sample": {"bbox": ps, "mismatches": mism, "valid": int(ref[..., 1].sum())},
                    "oracle_mpix_per_s": ps * ps / cdt / 1e6, "oracle_cores": os.cpu_count(),
                })
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
