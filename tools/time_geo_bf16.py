"""Native bf16 storage of the GeoCyclic ops against the upcast path: one autograd fwd + bwd of geocyclic_pad,
geocyclic_dwconv and geocyclic_avgpool5 with a bf16 input (what bf16 autocast hands them), ops.NATIVE_BF16 True against
False, alternating in one process.

    python tools/time_geo_bf16.py [--repeats 7] [--steps 20] [--out profiles/geo_bf16.json]

Per op and arm: CUDA-event ms per step (median, min, max over the repeats), the bytes the traffic model charges for the
step (computed from the shapes below: each tensor read or written once per kernel or cast, stencil re-reads not counted)
and the implied TB/s.  Input [1, 64, 721, 1440] bf16 (133 MB, more than the 126 MB of L2), fp32 weight for dwconv.

Also timed: the fp32 avgpool5 backward, the strided adjoint kernel against the full-resolution composition it replaced
(kept inline below as the comparator), and one end-to-end training fwd + bwd of oracle.paradis_assembly.Assembly(dropin=
True) under bf16 autocast at 721 x 1440 with default_cfg(latent=64, vels=16) and a 30 min base step, switch on against
off."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from paradis_model_b200 import ops

B, C, H, W = 1, 64, 721, 1440
BF = torch.bfloat16
MODEL_BASE_DT = 1800


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def traffic(op, arg):
    """Bytes of one fwd + bwd per arm.  N input elements, M output elements; native: 2 B per element read or written;
    upcast: each bf16 -> fp32 cast 6 B, each fp32 -> bf16 cast 6 B, each fp32 kernel access 4 B."""
    N = B * C * H * W
    if op == "pad":
        M = B * C * (H + 2 * arg) * (W + 2 * arg)
        return {"native": 2 * (N + M) * 2, "upcast": (6 * N + 4 * (N + M) + 6 * M) * 2}
    if op == "dwconv":                      # fwd, grad input, grad weight (x and grad_y read again)
        return {"native": 4 * N + 4 * N + 4 * N, "upcast": 20 * N + 20 * N + 14 * N}
    M = B * C * ((H - 1) // arg + 1) * ((W - 1) // arg + 1)
    return {"native": 2 * (N + M) * 2, "upcast": (6 * N + 4 * (N + M) + 6 * M) * 2}


def timed(arms, repeats, steps):
    """arms: name -> (setup, step); setup() runs before the arm's steps (switches).  Alternating repeats."""
    times = {a: [] for a in arms}
    for a, (setup, step) in arms.items():      # warm-up
        setup()
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        for a, (setup, step) in arms.items():
            setup()
            step()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            times[a].append(e0.elapsed_time(e1) / steps)
    ops.NATIVE_BF16 = True
    out = {}
    for a, t in times.items():
        t = sorted(t)
        out[a] = {"ms_median": round(statistics.median(t), 4), "ms_min": round(t[0], 4), "ms_max": round(t[-1], 4)}
    return out


def switch(flag):
    def setup():
        ops.NATIVE_BF16 = flag
    return setup


def op_step(op, arg, x, w, gy):
    def step():
        x.grad = None
        if w is not None:
            w.grad = None
        if op == "pad":
            y = ops.geocyclic_pad(x, arg)
        elif op == "dwconv":
            y = ops.geocyclic_dwconv(x, w)
        else:
            y = ops.geocyclic_avgpool5(x, arg)
        y.backward(gy)
    return step


def composition_bwd(gy, s):
    """The avgpool5 adjoint before it had a kernel of its own (fp32)."""
    g_full = torch.zeros((B, C, H, W), dtype=torch.float32, device=gy.device)
    g_full[:, :, ::s, ::s] = gy
    box = torch.full((C, 1, 5, 5), 1.0 / 25.0, dtype=torch.float32, device=gy.device)
    return torch.ops.paradis.geocyclic_dwconv_backward(g_full, g_full, box, True, False, False)[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--model-steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON file for the results (default: print only)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_geo_bf16 measures on the GPU"
    res = {"card": card(), "shape": [B, C, H, W], "steps": args.steps, "repeats": args.repeats, "ops": {}}
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, C, H, W, generator=g).cuda().to(BF).requires_grad_(True)
    for op, vals in (("pad", (1, 2, 3)), ("dwconv", (3, 5, 7)), ("avgpool5", (1, 2, 4))):
        for arg in vals:
            w = (torch.randn(C, 1, arg, arg, generator=g) / arg).cuda().requires_grad_(True) if op == "dwconv" else None
            with torch.no_grad():
                y = (ops.geocyclic_pad(x, arg) if op == "pad" else ops.geocyclic_dwconv(x, w) if op == "dwconv"
                     else ops.geocyclic_avgpool5(x, arg))
            gy = torch.randn(y.shape, generator=g).cuda().to(BF)
            del y
            step = op_step(op, arg, x, w, gy)
            r = timed({"native": (switch(True), step), "upcast": (switch(False), step)}, args.repeats, args.steps)
            model = traffic(op, arg)
            for a in r:
                r[a]["model_bytes"] = model[a]
                r[a]["model_TB_per_s"] = round(model[a] / (r[a]["ms_median"] * 1e-3) / 1e12, 2)
            r["speedup_median"] = round(r["upcast"]["ms_median"] / r["native"]["ms_median"], 3)
            name = f"{op}_{'p' if op == 'pad' else 'k' if op == 'dwconv' else 's'}{arg}"
            res["ops"][name] = r
            print(name, json.dumps(r), flush=True)
            del gy, w

    # fp32 avgpool5 backward: the strided adjoint kernel against the composition it replaced
    res["avgpool5_fp32_backward"] = {}
    for s in (1, 2, 4):
        gy = torch.randn(B, C, (H - 1) // s + 1, (W - 1) // s + 1, generator=g).cuda()
        new = lambda: torch.ops.paradis.geocyclic_avgpool5_backward(gy, H, W, s)
        old = lambda: composition_bwd(gy, s)
        assert torch.equal(new(), old())
        nop = lambda: None
        r = timed({"kernel": (nop, new), "composition": (nop, old)}, args.repeats, args.steps)
        No = gy.numel()
        r["kernel"]["model_bytes"] = 4 * (No + B * C * H * W)
        r["composition"]["model_bytes"] = 4 * B * C * H * W + 8 * No + 8 * B * C * H * W   # zero fill, scatter, kernel
        r["speedup_median"] = round(r["composition"]["ms_median"] / r["kernel"]["ms_median"], 3)
        res["avgpool5_fp32_backward"][f"s{s}"] = r
        print("avgpool5 fp32 backward", s, json.dumps(r), flush=True)
        del gy
    del x

    # end to end: one training fwd + bwd of the drop-in assembly under bf16 autocast
    from oracle import paradis_assembly as A
    from oracle.sl_oracle import make_grids
    import paradis_model_b200 as P
    lat, lon = make_grids(H, W, True)
    torch.manual_seed(0)
    cfg = A.default_cfg(latent=64, vels=16)
    # 0.25 degree cells are 5.6x smaller than the 1.40625 degree ones the model tests use: with the default 6 h step the
    # untrained velocity nets move points by more than the 126 rows the advection kernels support, so 30 min here
    cfg["model"]["base_dt"] = MODEL_BASE_DT
    model = A.Assembly(A.FakeDataModule, cfg, lat, lon, dropin=True).cuda()
    xin = torch.randn(1, 22, H, W, generator=g).cuda()
    tgt = torch.randn(1, 7, H, W, generator=g).cuda()

    def train_step():
        model.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=BF):
            loss = torch.nn.functional.mse_loss(model(xin).float(), tgt)
        loss.backward()

    r = timed({"native": (switch(True), train_step), "upcast": (switch(False), train_step)}, args.repeats,
              args.model_steps)
    P.check_status()
    r["speedup_median"] = round(r["upcast"]["ms_median"] / r["native"]["ms_median"], 3)
    r["config"] = ("Assembly(dropin=True), default_cfg(latent=64, vels=16) (2 layers, bicubic) with base_dt "
                   f"{MODEL_BASE_DT} s, input [1, 22, 721, 1440], bf16 autocast, end to end (forward, loss, backward)")
    res["model_train_step_end_to_end"] = r
    print("model", json.dumps(r), flush=True)
    print(json.dumps({"card": res["card"]}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
