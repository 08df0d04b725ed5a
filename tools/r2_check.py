"""Round-2 development check (GPU box): row-sweep backward vs the general two-kernel path on several shapes,
then timings at C3.  usage: r2_check.py [check|time|both]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import paradis_model_b200 as P
from paradis_model_b200 import synthetic as S
from paradis_model_b200.ops import RawAdvection
from oracle import sl_oracle as O

DT = S.DT_DEFAULT
mode = sys.argv[1] if len(sys.argv) > 1 else "both"


import threading
_progress = {"what": "start", "t": time.time()}


def _watchdog(limit=45.0):
    while True:
        time.sleep(1.0)
        if time.time() - _progress["t"] > limit:
            print(f"WATCHDOG: '{_progress['what']}' has not finished after {limit:.0f} s -- hung kernel? exiting", flush=True)
            os._exit(3)


def mark(what):
    _progress["what"], _progress["t"] = what, time.time()


threading.Thread(target=_watchdog, daemon=True).start()


def relmax(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def check():
    cases = [(33, 64, 2, 2, True, 2.0, 3.0), (64, 128, 1, 4, True, 2.0, 6.0), (128, 256, 2, 3, False, 4.0, 6.0),
             (181, 360, 1, 3, True, 4.0, 6.0), (181, 360, 1, 3, True, 1.0, 8.0), (96, 192, 2, 3, True, 8.0, 8.0),
             (721, 1440, 1, 2, True, 4.0, 6.0), (240, 512, 1, 2, False, 1.5, 2.0),
             (181, 360, 2, 32, True, 4.0, 6.0), (721, 1440, 1, 8, True, 4.0, 6.0)]   # many planes: every CTA range cut
    ok = True
    for interp in ("bilinear", "bicubic"):
        for (H, W, B, V, poles, clip, cfl) in cases:
            mark(f"{interp} {H}x{W} B{B} V{V} cfl={cfl}")
            lat, lon, field, u, v, go = O.bench_inputs(H, W, B, V, poles, DT, cells_sigma=clip / 2, cells_clip=clip)
            geo = P.SLGeometry.from_grids(lat.cuda(), lon.cuda())
            f, uu, vv, g = [t.cuda() for t in (field, u, v, go)]
            R0 = RawAdvection(geo, B, V, interp, True, "fast", 0.0)
            R1 = RawAdvection(geo, B, V, interp, True, "fast", cfl)
            a = [t.clone() for t in R0.backward(g, f, uu, vv, DT, 3)]
            torch.cuda.synchronize()
            t0 = time.time()
            b = [t.clone() for t in R1.backward(g, f, uu, vv, DT, 3 | 8)]
            torch.cuda.synchronize()
            c = [t.clone() for t in R1.backward(g, f, uu, vv, DT, 3 | 8)]
            torch.cuda.synchronize()
            errs = [relmax(x, y) for x, y in zip(b, a)]
            det = all(torch.equal(x, y) for x, y in zip(b, c))
            # worst row of grad_field
            d = (b[0] - a[0]).abs().amax(dim=(0, 1, 3))
            wr = int(d.argmax())
            good = errs[0] < 5e-6 and errs[1] < 1e-5 and errs[2] < 1e-5 and det
            ok = ok and good
            print(f"{'OK ' if good else 'BAD'} {interp:8s} {H}x{W} B{B} V{V} poles={poles} clip={clip} cfl={cfl}: "
                  f"gf {errs[0]:.2e} gu {errs[1]:.2e} gv {errs[2]:.2e} det={det} worst gf row {wr} ({float(d[wr]):.2e})",
                  flush=True)
    P.check_status()
    print("CHECK", "PASSED" if ok else "FAILED", flush=True)


def timeit(fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def times():
    H, W, B, V = 721, 1440, 1, 64
    lat, lon = S.make_grids(H, W, True)
    geo = P.SLGeometry.from_grids(lat.cuda(), lon.cuda())
    f, u, v, g = [t.cuda() for t in S.white_noise_inputs(H, W, B, V)]
    pts = B * V * H * W
    for interp in (sys.argv[2:] or ["bilinear", "bicubic"]):
        mark(f"time {interp}")
        R = RawAdvection(geo, B, V, interp, True, "fast", 6.0)
        tf = timeit(lambda: R.forward(f, u, v, DT))
        tb = timeit(lambda: R.backward(g, f, u, v, DT, 3))
        print(f"TIME C3 {interp} lib={os.path.basename(os.environ.get('PARADIS_SL_LIB','default'))}: fwd {tf:.3f} ms "
              f"({16*pts/tf/1e6:.0f} GB/s) bwd {tb:.3f} ms ({28*pts/tb/1e6:.0f} GB/s) step {tf+tb:.3f} ms", flush=True)
    P.check_status()


if mode in ("check", "both"):
    check()
if mode in ("time", "both"):
    times()
