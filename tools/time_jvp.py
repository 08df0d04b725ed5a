"""Tangent-linear advection (paradis::sl_advect_jvp with field, u and v tangents) against the forward
(paradis::sl_advect), alternating the two in one process.

    python tools/time_jvp.py [--repeats 7] [--steps 20] [--out profiles/jvp.json]

Cases: C3 (721 x 1440, B = 1, V = 64, bilinear, FAST) and C2 (128 x 256, B = 8, V = 64, bicubic, FAST), pole_fix on.
Per op: CUDA-event ms per call (median, min, max over the repeats), the algorithmic bytes per arrival point (forward:
read field, u, v, write out = 16 B; tangent: read field, dfield, u, v, du, dv, write dout = 28 B) and their rate as a
share of the device-to-device copy rate measured in the same run.  C3 works on 266 MB per tensor, more than the
126 MB of L2; C2 (67 MB per tensor) partly fits.  The card's name and power limit are part of the result."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from oracle import sl_oracle as O
from paradis_model_b200 import ops

DT = 21600 * 7.29212e-5 / 8
CASES = {"C3": (721, 1440, 1, 64, "bilinear"), "C2": (128, 256, 8, 64, "bicubic")}
BYTES = {"forward": 16, "jvp": 28}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def copy_rate(nbytes=1 << 31, reps=20):
    """Device-to-device copy rate (read + write bytes per second) of a buffer larger than L2."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes / (e0.elapsed_time(e1) / reps * 1e-3)


def timed(arms, repeats, steps):
    times = {a: [] for a in arms}
    for step in arms.values():
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        for a, step in arms.items():
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            times[a].append(e0.elapsed_time(e1) / steps)
    return {a: sorted(t) for a, t in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="JSON file for the results (default: print only)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_jvp measures on the GPU"
    peak = copy_rate()
    res = {"card": card(), "copy_TB_per_s": round(peak / 1e12, 3), "steps": args.steps, "repeats": args.repeats,
           "cases": {}}
    for name, (H, W, B, V, interp) in CASES.items():
        lat, lon, field, u, v, _ = O.bench_inputs(H, W, B, V, True, DT, seed=0)
        field, u, v = field.cuda(), u.cuda(), v.cuda()
        g = torch.Generator().manual_seed(1)
        df, du, dv = [(torch.randn(t.shape, generator=g) * float(t.abs().mean())).cuda() for t in (field, u, v)]
        geo = ops.SLGeometry.from_grids(lat.cuda(), lon.cuda())
        a = (geo.tables, geo.scalars, DT, ops._lib.INTERP[interp], True, ops._lib.MATH["fast"], geo.windows)
        arms = {"forward": lambda: torch.ops.paradis.sl_advect(field, u, v, *a, ops.DEFAULT_CFL_CELLS),
                "jvp": lambda: torch.ops.paradis.sl_advect_jvp(field, u, v, df, du, dv, *a)}
        t = timed(arms, args.repeats, args.steps)
        ops.check_status()
        pts = B * V * H * W
        r = {"shape": [B, V, H, W], "interp": interp, "math": "fast"}
        for arm, ts in t.items():
            ms = statistics.median(ts)
            rate = BYTES[arm] * pts / (ms * 1e-3)
            r[arm] = {"ms_median": round(ms, 4), "ms_min": round(ts[0], 4), "ms_max": round(ts[-1], 4),
                      "bytes_per_point": BYTES[arm], "TB_per_s": round(rate / 1e12, 3),
                      "share_of_copy": round(rate / peak, 3)}
        r["jvp_over_forward"] = round(r["jvp"]["ms_median"] / r["forward"]["ms_median"], 3)
        res["cases"][name] = r
        print(name, json.dumps(r), flush=True)
        del field, u, v, df, du, dv
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
