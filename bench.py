#!/usr/bin/env python
"""bench.py -- SL advection fwd+bwd throughput (grid-pts*ch/s) on B200, per the driver contract.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # reference algorithm on the host CPUs
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

A "step" is one forward + one backward of the operator core (model/advection.py:129-169) over
one batch of synthetic fields.  Workload at N=1: the configuration BASELINE.json's metric is
quoted on, 0.25 deg (721x1440), 64 channels, batch 1 (SURVEY 8d "C3").  With N>1 the SAME global
problem is split into latitude bands (BASELINE.json configs[2]; strong scaling; halos read in place
from the neighbours over NVLink peer memory) and the line carries the communication-free
batch-sharded figure (one replica per GPU, weak scaling) as the extra key `batch_sharded`;
`--decomp batch` makes the batch-sharded run the headline instead.

Keys beyond the base contract: roofline (dominant kernel), roofline_step (whole step, 44 B per
grid-pt*ch), cpu_baseline (oracle port timed on the host cores, bounded sample), e2e (host
buffers through the C-ABI host entry, copies inside the timed region), clocks, gpu_launches.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (H, W, V, batch per GPU, pole-including grid)
    "c3": (721, 1440, 64, 1, True),    # BASELINE configs[2]: 0.25 deg, 64 ch
    "c2": (128, 256, 64, 8, False),    # BASELINE configs[1]: 1.40625 deg, 64 ch, batch 8
}
BYTES_FWD, BYTES_BWD = 16, 28                                   # algorithmic B per grid-pt*ch (DESIGN.md)
BYTES_STEP = 44
CFL_CELLS = 6.0        # the benchmark clips |u|, |v| at 4 cells: great-circle step <= 4*sqrt(2) < 6 cells
CPU_SAMPLE_V = 8                                                # channels of the bounded CPU sample
DUMP_SAMPLES = 1 << 21      # per output: four float32 outputs of 8 MB each stay under 64 MB
OUTPUT_NAMES = ("out", "grad_field", "grad_u", "grad_v")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=list(WORKLOADS))
    ap.add_argument("--interp", default="bilinear", choices=["bilinear", "bicubic"])
    ap.add_argument("--math", default="fast", choices=["fast", "exact"])
    ap.add_argument("--decomp", default="auto", choices=["auto", "batch", "latband"],
                    help="N>1: latitude bands of ONE global problem (strong scaling; default for c3) or one replica "
                         "per GPU (weak scaling)")
    ap.add_argument("--no-batch", action="store_true", help="latband: skip the batch-sharded comparison leg")
    ap.add_argument("--pull-all", action="store_true", help="lat bands: pull the halo rows of all four tensors into local buffers")
    ap.add_argument("--pull-field", action="store_true",
                    help="latband: pull the neighbours' field rows into a local buffer after the publish barrier instead of "
                         "reading them in place with the stencil taps (measured: no gain)")
    ap.add_argument("--no-p2p", action="store_true", help="latband: NCCL transport for the field halo too")
    ap.add_argument("--no-graph", action="store_true", help="latband: eager autograd step instead of a CUDA graph")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write out / grad_field / grad_u / grad_v of the last step as "
                         "DIR/<name>.npy (float32); outputs of more than DUMP_SAMPLES elements are reduced to the "
                         "flat-index sample of sample_index().  --impl reference writes its [1, CPU_SAMPLE_V, H, W] "
                         "CPU sample, so its files compare with those of other reference runs, not with the b200 arm's")
    return ap.parse_args()


def sample_index(numel):
    """The fixed, seeded sample of flat indices that --dump-outputs writes of a large output (sorted, unique)."""
    import numpy as np
    return np.unique(np.random.default_rng(0).integers(0, numel, DUMP_SAMPLES))


def dump_outputs(path, outputs):
    """Write each tensor of `outputs` (name -> tensor, all of one shape) as <path>/<name>.npy in float32: whole when
    it has at most DUMP_SAMPLES elements, else the elements at sample_index(numel) of its flattened form."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    idx = None
    numel = next(iter(outputs.values())).numel()
    if numel > DUMP_SAMPLES:
        idx = torch.from_numpy(sample_index(numel))
    for name, t in outputs.items():
        t = t.detach()
        if idx is not None:
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(phase, captured_config):
    """DRAM bytes (read + write) per step of ALL kernels of `phase` ("forward" / "backward"), summed from the committed
    `ncu --set full` capture of the final kernels (profiles/traffic_r2.json, written by tools/ncu_traffic.py); None for
    any configuration other than the one the capture was taken on (C3, bilinear, fast math)."""
    if not captured_config:
        return None
    path = os.path.join(ROOT, "profiles", "traffic_r2.json")
    try:
        return json.load(open(path))["phases"][phase]["dram_bytes"]
    except Exception:
        return None


def aux_kernel_rooflines(torch, P, H, W, dev, peak):
    C = 64
    x = torch.randn(1, C, H, W, device=dev)
    w5 = torch.randn(C, 1, 5, 5, device=dev) / 5
    pad2 = torch.empty(1, C, H + 4, W + 4, device=dev)

    def timed(fn, n=20):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    el, elp = x.numel(), pad2.numel()
    cases = {
        "geocyclic_pad_fwd p=2": (lambda: P.geocyclic_pad(x, 2), 4 * (el + elp)),
        "geocyclic_pad_bwd p=2": (lambda: torch.ops.paradis.geocyclic_pad_backward(pad2, 2), 4 * (el + elp)),
        "geocyclic_dwconv_fwd k=5": (lambda: P.geocyclic_dwconv(x, w5), 8 * el),
        "geocyclic_avgpool5 stride 4": (lambda: P.geocyclic_avgpool5(x, 4), 4 * el + 4 * el // 16),
    }
    out = {}
    for name, (fn, nbytes) in cases.items():
        ms = timed(fn)
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "achieved": gbs, "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes": nbytes}
    return out


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (NVML, 20 ms period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml as N
            N.nvmlInit()
            self.N, self.h = N, N.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = N.nvmlDeviceGetMaxClockInfo(self.h, N.NVML_CLOCK_SM)
        except Exception:
            self.N = None

    def run(self):
        if self.N is None:
            return
        N = self.N
        names = {"hw_slowdown": getattr(N, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(N, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(N, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(N, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM))
                try:
                    mask = N.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = N.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------
def cpu_port_time(H, W, poles, interp, V, repeats):
    """fwd+bwd of the oracle's op-order replay of model/advection.py:129-169 (torch CPU eager,
    all host threads) on [1, V, H, W]; returns best seconds."""
    import torch
    from oracle import sl_oracle as O
    from paradis_model_b200 import synthetic as S
    torch.set_num_threads(os.cpu_count() or 1)
    lat, lon = O.make_grids(H, W, poles)
    field, u, v, go = S.white_noise_inputs(H, W, 1, V)
    best = float("inf")
    for i in range(repeats + 1):                 # first pass is the warm-up
        t0 = time.perf_counter()
        O.sl_advect_fwd_bwd(field, u, v, lat, lon, S.DT_DEFAULT, go, interp)
        dt = time.perf_counter() - t0
        if i:
            best = min(best, dt)
    return best, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    H, W, V, Bg, poles = WORKLOADS[args.workload]
    steps = args.steps
    warm = max(1, min(args.warmup, 1))
    import torch
    from oracle import sl_oracle as O
    from paradis_model_b200 import synthetic as S
    torch.set_num_threads(os.cpu_count() or 1)
    lat, lon = O.make_grids(H, W, poles)
    field, u, v, go = S.white_noise_inputs(H, W, 1, CPU_SAMPLE_V)
    for _ in range(warm):
        O.sl_advect_fwd_bwd(field, u, v, lat, lon, S.DT_DEFAULT, go, args.interp)
    t0 = time.perf_counter()
    for _ in range(steps):
        res = O.sl_advect_fwd_bwd(field, u, v, lat, lon, S.DT_DEFAULT, go, args.interp)
    sec = (time.perf_counter() - t0) / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(OUTPUT_NAMES, res)))
    pts = CPU_SAMPLE_V * H * W
    val = pts / sec
    sample = f"[1,{CPU_SAMPLE_V},{H},{W}] slice of the workload per step ({steps} steps, {warm} warm-up)"
    line = {"impl": "reference", "metric": "SL advection fwd+bwd grid-pts*ch/s", "value": val, "unit": "grid-pt*ch/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {H}x{W}, V={V} (CPU sample V={CPU_SAMPLE_V}), {args.interp}",
                       "note": "oracle port of model/advection.py:129-169 (torch CPU eager); /root/reference is not on the GPU box"},
            "cpu_baseline": {"value": val, "unit": "grid-pt*ch/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": val, "unit": "grid-pt*ch/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import paradis_model_b200 as P
    from paradis_model_b200 import synthetic as S
    from paradis_model_b200.ops import RawAdvection

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    decomp = args.decomp
    if decomp == "auto":      # BASELINE.json configs[2]: "0.25 deg ... 1/2/4/8 B200 with latitude-band halo exchange"
        decomp = "latband" if (world > 1 and args.workload == "c3") else "batch"
    if decomp == "latband" and world > 1:
        if args.dump_outputs:
            raise SystemExit("--dump-outputs needs one whole output per process: use --decomp batch")
        from paradis_model_b200 import halo
        return halo.bench_latband(args, WORKLOADS[args.workload], rank, world, dev)

    H, W, V, Bg, poles = WORKLOADS[args.workload]
    dt = S.DT_DEFAULT
    lat, lon = S.make_grids(H, W, poles)
    geo = P.SLGeometry.from_grids(lat.to(dev), lon.to(dev))
    h_in = S.white_noise_inputs(H, W, Bg, V, dt, seed=rank, pin=not args.no_e2e)
    field, u, v, go = [t.to(dev) for t in h_in]
    R = RawAdvection(geo, Bg, V, args.interp, True, args.math, CFL_CELLS)
    pts_rank = Bg * V * H * W

    def step():
        R.forward(field, u, v, dt)
        R.backward(go, field, u, v, dt, 3)

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    torch.cuda.synchronize()
    t_wall = time.perf_counter()
    for k in range(args.steps):
        ev[k][0].record()
        R.forward(field, u, v, dt)
        ev[k][1].record()
        R.backward(go, field, u, v, dt, 3)
        ev[k][2].record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    clocks = sampler.stop()
    if world > 1:
        dist.barrier()
    P.check_status(dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(OUTPUT_NAMES, (R.out, R.gfield, R.gu, R.gv))))
    total_ms = ev[0][0].elapsed_time(ev[-1][2])
    phase = [sum(e[i].elapsed_time(e[i + 1]) for e in ev) / args.steps for i in range(2)]
    t = torch.tensor([total_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_step = total_ms / args.steps

    # ---- end to end: host buffers through the C-ABI host entry (H2D + kernels + D2H timed)
    e2e = None
    if not args.no_e2e:
        h_out = [torch.empty(Bg, V, H, W, pin_memory=True) for _ in range(4)]
        scratch = None
        n_e2e = max(2, min(args.steps, 5))
        scratch = P.host_fwd_bwd(geo, *h_in, *h_out, dt, args.interp, True, args.math, 4, scratch, CFL_CELLS)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            scratch = P.host_fwd_bwd(geo, *h_in, *h_out, dt, args.interp, True, args.math, 4, scratch, CFL_CELLS)
        te = torch.tensor([(time.perf_counter() - t0) / n_e2e], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        nbytes = 4 * pts_rank * 4
        e2e = {"value": world * pts_rank / float(te.item()), "unit": "grid-pt*ch/s", "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": nbytes, "ms_per_step": float(te.item()) * 1e3, "steps": n_e2e,
               "api": "paradis_sl_advect_fwd_bwd_host (pinned host tensors, 4-plane chunks, 4 streams)"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    # forward = pole_means + sl_fwd_kernel + pole_rows_fix; backward = 2 x pole_means + rows_prep + the row-sweep
    # kernel (all latitudes) + guard / pole fix-ups + the three (normally empty) launches of the fallback path.
    # Both phases are timed with CUDA events on the launching stream; `traffic` sums the DRAM bytes of every
    # kernel of the phase from the committed ncu capture.
    bilinear = args.interp == "bilinear"
    names = ["sl_fwd_kernel", "sl_bwd_rows_kernel" if bilinear else "sl_bwd_sweep_kernel"]
    phase_names = ["forward", "backward"]
    alg = [BYTES_FWD, BYTES_BWD]
    dom = max(range(2), key=lambda i: phase[i])
    achieved = alg[dom] * pts_rank / (phase[dom] * 1e-3) / 1e9
    captured = args.workload == "c3" and bilinear and args.math == "fast"
    roofline = {"bound": "hbm", "kernel": names[dom], "phase": phase_names[dom] + " (all kernels of the phase)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(phase_names[dom], captured), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg[dom] * pts_rank, "ms_per_launch": phase[dom],
                "phases_ms": dict(zip(phase_names, phase)),
                "phases_frac": {n: alg[i] * pts_rank / (phase[i] * 1e-3) / 1e9 / peak for i, n in enumerate(phase_names)},
                "phases_traffic": {n: ncu_traffic(n, captured) for n in phase_names}}
    step_gbs = BYTES_STEP * pts_rank / (ms_step * 1e-3) / 1e9
    line = {"metric": "SL advection fwd+bwd grid-pts*ch/s", "value": world * pts_rank / (ms_step * 1e-3),
            "unit": "grid-pt*ch/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: {H}x{W} mesh, V={V} channels, batch {Bg} per GPU, {args.interp}, "
                                   f"math={args.math}, pole_fix, cfl_cells={CFL_CELLS}",
                       "inputs": "field~N(0,1); u,v~N(0,(2 cells)^2) clipped at +-4 cells; grad_out~N(0,1); seed=rank",
                       "l2": "inputs (1.06 GB per GPU at c3) exceed the 126 MB L2; no flush needed",
                       "parallelism": f"batch-sharded x{world}, no data-path collective"},
            "roofline": roofline,
            "roofline_step": {"bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
                              "bytes_per_unit": BYTES_STEP, "frac_of_8TBs": step_gbs / 8000.0},
            "clocks": clocks, "gpu_launches": (12 if bilinear else 15) * args.steps, "wall_ms_timed_region": wall_ms}
    if e2e:
        line["e2e"] = e2e
    if world == 1:
        # the other kernels of the boundary (GeoCyclic padding op, padding fused into the depthwise convolution, strided
        # PhysicalDownsample), one [1, 64, H, W] tensor each: GB/s of algorithmic traffic against the same measured peak
        line["aux_kernels"] = aux_kernel_rooflines(torch, P, H, W, dev, peak)
    if world == 1 and not args.no_cpu:
        sec, cores = cpu_port_time(H, W, poles, args.interp, CPU_SAMPLE_V, 2)
        line["cpu_baseline"] = {"value": CPU_SAMPLE_V * H * W / sec, "unit": "grid-pt*ch/s", "cores": cores,
                                "kind": "port",
                                "sample": f"[1,{CPU_SAMPLE_V},{H},{W}] slice of the workload, best of 2 after 1 warm-up"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
