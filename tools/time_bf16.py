"""Native bf16 storage against the upcast path: one autograd fwd + bwd of sl_advect with bf16 field / u / v (what bf16
autocast hands the op), ops.NATIVE_BF16 True against False, alternating in one process.

    python tools/time_bf16.py [--repeats 7] [--steps 20] [--out profiles/bf16_native.json]

Per workload and arm: CUDA-event ms per step (median and spread over the repeats), peak memory of one step above the
inputs, and the bytes the traffic model charges per grid point * channel: native 34 B (fwd: 3 x 2 B in, 4 B out; bwd:
3 x 2 B in + 4 B grad_out, grad_u / grad_v 2 x 2 B, grad_field 4 B accumulated + 4 B re-read + 2 B rounded) against
98 B for the upcast path (the 44 B of the fp32 kernels + 54 B of casts: 3 fp32 copies in forward and again in backward
at 6 B each, 3 gradient casts at 6 B each).  Inputs are white noise (synthetic.white_noise_inputs) at more than the 126 MB
of L2 at C3; C2 partly fits it."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import paradis_model_b200 as P
from paradis_model_b200 import ops
from paradis_model_b200 import synthetic as S

WORKLOADS = {  # name: H, W, B, V, poles, interpolation
    "C3": (721, 1440, 1, 64, True, "bilinear"),
    "C2": (128, 256, 8, 64, False, "bicubic"),
}
BYTES = {"native": 34, "upcast": 98}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="JSON file for the results (default: print only)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_bf16 measures on the GPU"
    res = {"card": card(), "steps": args.steps, "repeats": args.repeats, "workloads": {}}
    for name, (H, W, B, V, poles, interp) in WORKLOADS.items():
        lat, lon = S.make_grids(H, W, poles)
        geo = P.SLGeometry.from_grids(lat.cuda(), lon.cuda())
        field, u, v, go = [t.cuda() for t in S.white_noise_inputs(H, W, B, V)]
        f, uu, vv = [t.to(torch.bfloat16).requires_grad_(True) for t in (field, u, v)]
        del field, u, v

        def step():
            f.grad = uu.grad = vv.grad = None
            P.sl_advect(f, uu, vv, geo, S.DT_DEFAULT, interp).backward(go)

        arms = {"native": True, "upcast": False}
        times = {a: [] for a in arms}
        peaks = {}
        for a, flag in arms.items():           # warm-up and peak memory of one step per arm
            ops.NATIVE_BF16 = flag
            for _ in range(3):
                step()
            f.grad = uu.grad = vv.grad = None
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            step()
            torch.cuda.synchronize()
            peaks[a] = torch.cuda.max_memory_allocated() - base
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.repeats):           # alternating arms
            for a, flag in arms.items():
                ops.NATIVE_BF16 = flag
                step()
                torch.cuda.synchronize()
                e0.record()
                for _ in range(args.steps):
                    step()
                e1.record()
                torch.cuda.synchronize()
                times[a].append(e0.elapsed_time(e1) / args.steps)
        ops.NATIVE_BF16 = True
        P.check_status()
        units = B * V * H * W
        out = {"shape": [B, V, H, W], "interpolation": interp}
        for a in arms:
            t = sorted(times[a])
            med = statistics.median(t)
            out[a] = {"ms_median": round(med, 4), "ms_min": round(t[0], 4), "ms_max": round(t[-1], 4),
                      "model_bytes_per_unit": BYTES[a], "model_GB_per_step": round(BYTES[a] * units / 1e9, 3),
                      "model_TB_per_s": round(BYTES[a] * units / med / 1e9, 2),
                      "peak_MB_above_inputs": round(peaks[a] / 2**20, 1)}
        out["speedup_median"] = round(out["upcast"]["ms_median"] / out["native"]["ms_median"], 3)
        res["workloads"][name] = out
        print(name, json.dumps(out), flush=True)
    print(json.dumps({"card": res["card"]}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
