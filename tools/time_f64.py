"""float64 advection against fp32: forward (paradis::sl_advect), backward (paradis::sl_advect_backward / _f64, all
three gradients) and tangent-linear model (paradis::sl_advect_jvp with field, u and v tangents), alternating the six
arms in one process.

    python tools/time_f64.py [--repeats 5] [--steps 10] [--out profiles/f64.json]

Cases: C3 (721 x 1440, B = 1, V = 64, bilinear) and C2 (128 x 256, B = 8, V = 64, bicubic), pole_fix on, FAST math
for fp32 (fp64 has one arithmetic).  The fp32 backward is the library's default plan (fused sweep, cfl hint 8); the
fp64 backward is the per-point kernel plus the deterministic gather.  Per arm: CUDA-event ms per call (median, min,
max over the repeats), the algorithmic bytes per arrival point and their rate as a share of the device-to-device copy
rate measured in the same run.  The card's name, power limit and SM clocks are read in the same run."""
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
# values read + written per arrival point: forward field, u, v, out; backward grad_out, field, u, v (twice: per-point
# kernel and gather) and three gradients; jvp field, dfield, u, v, du, dv, dout
VALUES = {"forward": 4, "backward": 11, "jvp": 7}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
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
        for _ in range(2):
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
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None, help="JSON file for the results (default: print only)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_f64 measures on the GPU"
    peak = copy_rate()
    res = {"card": card(), "card_fields": "name, power.limit, clocks.sm, clocks.max.sm",
           "copy_TB_per_s": round(peak / 1e12, 3), "steps": args.steps, "repeats": args.repeats, "cases": {}}
    for name, (H, W, B, V, interp) in CASES.items():
        lat, lon, field, u, v, go = O.bench_inputs(H, W, B, V, True, DT, seed=0)
        g = torch.Generator().manual_seed(1)
        df, du, dv = [torch.randn(t.shape, generator=g) * float(t.abs().mean()) for t in (field, u, v)]
        geo = ops.SLGeometry.from_grids(lat.double().cuda(), lon.double().cuda())
        it, pf, wnd = ops._lib.INTERP[interp], True, geo.windows
        arms = {}
        for dt_name, dtype in (("fp32", torch.float32), ("fp64", torch.float64)):
            f, uu, vv, gg, dff, duu, dvv = [t.to(dtype).cuda() for t in (field, u, v, go, df, du, dv)]
            if dtype == torch.float64:
                tab, sc, math = geo.tables64, geo.scalars64, ops._lib.MATH["exact"]
                bwd = lambda f=f, uu=uu, vv=vv, gg=gg, tab=tab, sc=sc, math=math: \
                    torch.ops.paradis.sl_advect_backward_f64(gg, f, uu, vv, tab, sc, DT, it, pf, math, wnd, True, True)
            else:
                tab, sc, math = geo.tables, geo.scalars, ops._lib.MATH["fast"]
                bwd = lambda f=f, uu=uu, vv=vv, gg=gg, tab=tab, sc=sc, math=math: \
                    torch.ops.paradis.sl_advect_backward(gg, f, uu, vv, tab, sc, DT, it, pf, math, wnd,
                                                         ops.DEFAULT_CFL_CELLS, True, True)
            arms[f"forward_{dt_name}"] = lambda f=f, uu=uu, vv=vv, tab=tab, sc=sc, math=math: \
                torch.ops.paradis.sl_advect(f, uu, vv, tab, sc, DT, it, pf, math, wnd, ops.DEFAULT_CFL_CELLS)
            arms[f"backward_{dt_name}"] = bwd
            arms[f"jvp_{dt_name}"] = lambda f=f, uu=uu, vv=vv, dff=dff, duu=duu, dvv=dvv, tab=tab, sc=sc, math=math: \
                torch.ops.paradis.sl_advect_jvp(f, uu, vv, dff, duu, dvv, tab, sc, DT, it, pf, math, wnd)
        t = timed(arms, args.repeats, args.steps)
        ops.check_status()
        pts = B * V * H * W
        r = {"shape": [B, V, H, W], "interp": interp}
        for arm, ts in t.items():
            op, dt_name = arm.split("_")
            ms = statistics.median(ts)
            nbytes = VALUES[op] * (8 if dt_name == "fp64" else 4)
            rate = nbytes * pts / (ms * 1e-3)
            r[arm] = {"ms_median": round(ms, 4), "ms_min": round(ts[0], 4), "ms_max": round(ts[-1], 4),
                      "bytes_per_point": nbytes, "TB_per_s": round(rate / 1e12, 3), "share_of_copy": round(rate / peak, 3)}
        for op in VALUES:
            r[f"{op}_fp64_over_fp32"] = round(r[f"{op}_fp64"]["ms_median"] / r[f"{op}_fp32"]["ms_median"], 2)
        res["cases"][name] = r
        print(name, json.dumps(r), flush=True)
        arms.clear()
        torch.cuda.empty_cache()
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
