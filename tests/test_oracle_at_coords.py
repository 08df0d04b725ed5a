"""CPU tests of the fp64 reference at given departure coordinates (oracle.sl_oracle.sl_advect_at_coords): it
reproduces the closed form, its per-point bounds hold for an fp32 run of the same computation with the grad_field sum
in a shuffled order, and a wrong term anywhere is flagged at exactly the points it changes."""
import math

import numpy as np
import pytest
import torch

from conftest import relmax
from oracle import sl_oracle as O

DT = 21600 * 7.29212e-5 / 8


def _closed_form_coords(u, v, lat, lon, dt, interp):
    """[B, V, 11, H, W] departure coordinates from the op-order replay (departure_pixels + sampler_coords), not from
    sl_advect_explicit, with the intermediates of the rotated-pole map."""
    H, W = lat.shape
    p = O.INTERP_PAD[interp]
    geo = O.Geometry(lat, lon)
    pix_x, pix_y = O.departure_pixels(u, v, geo, dt)
    _, _, ix, iy = O.sampler_coords(pix_x, pix_y, H, W, p)
    lat_r, lon_r = -v * dt, -u * dt
    sa, ca, sb, cb = torch.sin(lat_r), torch.cos(lat_r), torch.sin(lon_r), torch.cos(lon_r)
    sp, cp = torch.sin(geo.lat), torch.cos(geo.lat)
    s = sa * cp + ca * cb * sp
    num, den = ca * sb, ca * cb * cp - sa * sp
    lat_d, lon_d = O.departure_latlon(u, v, geo, dt)
    return torch.stack(torch.broadcast_tensors(ix, iy, sa, ca, sb, cb, s, num, den, lat_d, lon_d), dim=2)


def _case(H, W, poles, interp, B=1, V=2, seed=0):
    """fp32 inputs, fp32 coordinates (what the parity instrument returns) and the fp32 sin / cos tables."""
    lat, lon, field, u, v, go = O.bench_inputs(H, W, B, V, poles, DT, seed=seed)
    lat64, lon64 = O.make_grids(H, W, poles, torch.float64)
    coords = _closed_form_coords(u.double(), v.double(), lat64, lon64, DT, interp).float()
    sl, cl = torch.sin(lat[:, 0].float()), torch.cos(lat[:, 0].float())
    geo = O.Geometry(lat64, lon64)
    return field, go, coords, sl, cl, geo


@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("poles", [True, False])
def test_at_coords_reproduces_closed_form_fp64(poles, interp, pole_fix):
    H, W, B, V, dt = 17, 24, 2, 2, 0.19688724
    lat, lon = O.make_grids(H, W, poles, torch.float64)
    g = torch.Generator().manual_seed(5)
    field = torch.randn(B, V, H, W, generator=g, dtype=torch.float64)
    sig = 3.0 * math.pi / H / dt
    u = torch.randn(B, V, H, W, generator=g, dtype=torch.float64) * sig
    v = torch.randn(B, V, H, W, generator=g, dtype=torch.float64) * sig
    go = torch.randn(B, V, H, W, generator=g, dtype=torch.float64)
    coords = _closed_form_coords(u, v, lat, lon, dt, interp)
    r = O.sl_advect_at_coords(field, go, coords, torch.sin(lat[:, 0]), torch.cos(lat[:, 0]), dt,
                              O.Geometry(lat, lon), interp, pole_fix)
    ref = O.sl_advect_explicit(field, u, v, lat, lon, dt, go, interp, pole_fix)
    for x, y in zip(r.values(), ref):
        assert relmax(x, y) < 1e-12


SHAPES = [(5, 6), (7, 18), (33, 50), (16, 1442)]          # test_gpu_parity.py::test_ragged_shapes_scalar_paths


@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("poles", [True, False])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("H,W", SHAPES)
def test_bounds_hold_for_fp32_in_any_summation_order(H, W, interp, poles, pole_fix):
    field, go, coords, sl, cl, geo = _case(H, W, poles, interp, seed=H + W)
    ref = O.sl_advect_at_coords(field, go, coords, sl, cl, DT, geo, interp, pole_fix)
    for seed in (0, 1):
        f32 = O.sl_advect_at_coords(field, go, coords, sl, cl, DT, geo, interp, pole_fix,
                                    compute_dtype=torch.float32, scatter_order=torch.Generator().manual_seed(seed))
        ratios = [O.worst_ratio(x, y, b) for x, y, b in zip(f32.values(), ref.values(), ref.bounds())]
        print(f"{H}x{W} {interp} poles={poles} pole_fix={pole_fix} order {seed}: max error/bound "
              + " ".join(f"{n}={q:.3f}" for n, q in zip(("out", "grad_field", "grad_u", "grad_v"), ratios)))
        for name, x, y, b in zip(("out", "grad_field", "grad_u", "grad_v"), f32.values(), ref.values(), ref.bounds()):
            assert not O.over_bound(x, y, b).any(), name


# ------------------------------------------------------------------ negative controls
def _flagged(got, ref, bound):
    return {tuple(int(i) for i in t) for t in O.over_bound(got, ref, bound).nonzero()}


@pytest.fixture(scope="module", params=["bilinear", "bicubic"])
def run33(request):
    interp = request.param
    field, go, coords, sl, cl, geo = _case(33, 64, False, interp, B=1, V=2, seed=3)   # cell-centred: cap taps
    ref = O.sl_advect_at_coords(field, go, coords, sl, cl, DT, geo, interp, True)
    f32 = O.sl_advect_at_coords(field, go, coords, sl, cl, DT, geo, interp, True, compute_dtype=torch.float32,
                                scatter_order=torch.Generator().manual_seed(0))
    for x, y, b in zip(f32.values(), ref.values(), ref.bounds()):
        assert not O.over_bound(x, y, b).any()
    return dict(interp=interp, field=field, go=go, coords=coords, sl=sl, cl=cl, geo=geo, ref=ref, f32=f32)


def _contributions(r, rows):
    """(|c|, plane, arrival (y, x), source cell (i, j), padded (R, C), c) of every in-plane grad_field contribution
    of arrival rows ``rows``; g' = grad_out after the pole-mean adjoint."""
    ref = r["ref"]
    g = O._pole_mean_adjoint(r["go"].double())
    B, V, H, W = g.shape
    res = []
    for idx, ok, w, (a, b, Rc, Cc) in ref.taps:
        c = (w * g)
        for pl in range(B * V):
            bb, vv = divmod(pl, V)
            for y in rows:
                for x in range(W):
                    if ok[bb, vv, y, x]:
                        k = int(idx[bb, vv, y, x])
                        res.append((abs(float(c[bb, vv, y, x])), (bb, vv), (y, x), divmod(k, W),
                                    (int(Rc[bb, vv, y, x]), int(Cc[bb, vv, y, x])), float(c[bb, vv, y, x])))
    return res


def test_moved_grad_field_contribution_is_flagged(run33):
    ref, f32 = run33["ref"], run33["f32"]
    H, W = 33, 64
    cand = [t for t in _contributions(run33, range(14, 19)) if 3 <= t[3][0] <= H - 4]
    mag, (b, v), _, (i, j), _, c = max(cand)
    gf = f32.grad_field.clone()
    gf[b, v, i, j] -= c
    gf[b, v, i, (j + 1) % W] += c
    assert _flagged(gf, ref.grad_field, ref.grad_field_bound) == {(b, v, i, j), (b, v, i, (j + 1) % W)}


@pytest.mark.parametrize("mutation", ["dropped", "unshifted"])
def test_cap_fold_mistake_is_flagged(run33, mutation):
    ref, f32 = run33["ref"], run33["f32"]
    H, W = 33, 64
    p = O.INTERP_PAD[run33["interp"]]
    cand = [t for t in _contributions(run33, list(range(0, 5)) + list(range(H - 5, H)))
            if t[4][0] < p or t[4][0] >= H + p]
    assert cand, "no cap contribution in the case"
    mag, (b, v), _, (i, j), (R, C), c = max(cand)
    gf = f32.grad_field.clone()
    gf[b, v, i, j] -= c
    want = {(b, v, i, j)}
    if mutation == "unshifted":
        j2 = (C - p) % W                   # the padded column without the 180-degree shift
        assert j2 != j
        gf[b, v, i, j2] += c
        want.add((b, v, i, j2))
    assert _flagged(gf, ref.grad_field, ref.grad_field_bound) == want


def test_dropped_small_weight_tap_is_flagged(run33):
    ref, f32 = run33["ref"], run33["f32"]
    H = 33
    src = O.pole_mean(run33["field"].double()).reshape(1, 2, -1)
    best = None
    for idx, ok, w, _ in ref.taps:
        val = torch.gather(src, 2, idx.reshape(1, 2, -1)).reshape(w.shape) * ok
        tw = torch.where((w.abs() < 1e-3) & ok, (w * val).abs(), torch.zeros_like(w))
        tw[:, :, 0] = 0
        tw[:, :, H - 1] = 0                # output pole rows are means: a point there is not isolated
        k = int(tw.argmax())
        if best is None or float(tw.flatten()[k]) > best[0]:
            best = (float(tw.flatten()[k]), np.unravel_index(k, w.shape), float((w * val).flatten()[k]))
    _, pt, term = best
    out = f32.out.clone()
    out[pt] -= term
    assert _flagged(out, ref.out, ref.out_bound) == {tuple(int(i) for i in pt)}


def test_one_ulp_of_ix_is_flagged(run33):
    """One ulp of ix at the interior point where it moves out the most relative to the bound is flagged, and only
    there.  Not every point's one-ulp change exceeds its bound: where out hardly depends on ix it stays inside."""
    ref = run33["ref"]
    H = 33
    c = run33["coords"]
    args = (run33["field"], run33["go"])
    rest = (run33["sl"], run33["cl"], DT, run33["geo"], run33["interp"], True)
    bumped = c.clone()
    bumped[:, :, 0] = torch.nextafter(c[:, :, 0], torch.tensor(math.inf))
    every = O.sl_advect_at_coords(*args, bumped, *rest).out
    score = (every - ref.out).abs() / ref.out_bound
    score[:, :, 0] = 0
    score[:, :, H - 1] = 0
    pt = np.unravel_index(int(score.argmax()), score.shape)
    one = c.clone()
    one[pt[0], pt[1], 0, pt[2], pt[3]] = bumped[pt[0], pt[1], 0, pt[2], pt[3]]
    out = O.sl_advect_at_coords(*args, one, *rest).out
    assert _flagged(out, ref.out, ref.out_bound) == {tuple(int(i) for i in pt)}
