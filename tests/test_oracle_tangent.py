"""CPU tests of the fp64 tangent-linear reference at given departure coordinates
(tangent_reference.sl_advect_tangent_at_coords): it is the derivative of the closed form (central differences), its
per-point bounds hold for an fp32 run of the kernel's chain, and a dropped velocity term or a dropped pole-mean tangent
is flagged where it changes the result."""
import math

import pytest
import torch

from oracle import sl_oracle as O
from tangent_reference import sl_advect_tangent_at_coords
from test_oracle_at_coords import DT, _case, _closed_form_coords


def _inputs(H, W, B, V, seed):
    g = torch.Generator().manual_seed(seed)
    sig = 3.0 * math.pi / H / 0.19688724
    r = lambda s=1.0: torch.randn(B, V, H, W, generator=g, dtype=torch.float64) * s
    return r(), r(sig), r(sig), r(), r(sig), r(sig)      # field, u, v, dfield, du, dv


@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("poles", [True, False])
@pytest.mark.parametrize("with_dfield", [True, False])
def test_tangent_matches_central_difference_fp64(poles, interp, pole_fix, with_dfield):
    H, W, B, V, dt, h = 17, 24, 1, 2, 0.19688724, 1e-6
    lat, lon = O.make_grids(H, W, poles, torch.float64)
    field, u, v, dfield, du, dv = _inputs(H, W, B, V, seed=7)
    if not with_dfield:
        dfield = None
    geo = O.Geometry(lat, lon)
    sl, cl = torch.sin(lat[:, 0]), torch.cos(lat[:, 0])
    coords = _closed_form_coords(u, v, lat, lon, dt, interp)
    r = sl_advect_tangent_at_coords(field, dfield, du, dv, coords, sl, cl, dt, geo, interp, pole_fix)

    def at(s):
        f = field if dfield is None else field + s * dfield
        return O.sl_advect_explicit(f, u + s * du, v + s * dv, lat, lon, dt, None, interp, pole_fix)
    fd = (at(h) - at(-h)) / (2 * h)
    # points whose stencil cell stays put across +-h (a floor() change is a kink of the interpolant)
    keep = torch.ones(B, V, H, W, dtype=torch.bool)
    for s in (h, -h):
        c = _closed_form_coords(u + s * du, v + s * dv, lat, lon, dt, interp)
        for k in (0, 1):
            keep &= torch.floor(c[:, :, k]) == torch.floor(coords[:, :, k])
    if pole_fix:                                 # a mean row depends on every point of the row
        for row in (0, H - 1):
            keep[:, :, row, :] &= keep[:, :, row, :].all(dim=-1, keepdim=True)
    assert keep.float().mean() > 0.8
    err = (r.out - fd).abs()[keep].max() / fd.abs().max()
    print(f"poles={poles} {interp} pole_fix={pole_fix} dfield={with_dfield}: rel err {err:.2e}")
    assert err < 1e-8


SHAPES = [(5, 6), (7, 18), (33, 50), (16, 1442)]


def _tl_case(H, W, poles, interp, seed):
    field, _, coords, sl, cl, geo = _case(H, W, poles, interp, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    sig = 3.0 * math.pi / H / DT
    dfield = torch.randn(field.shape, generator=g)
    du, dv = torch.randn(field.shape, generator=g) * sig, torch.randn(field.shape, generator=g) * sig
    return field, dfield, du, dv, coords, sl, cl, geo


@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("poles", [True, False])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("H,W", SHAPES)
def test_tangent_bound_holds_for_fp32_chain(H, W, interp, poles, pole_fix):
    field, dfield, du, dv, coords, sl, cl, geo = _tl_case(H, W, poles, interp, seed=H + W)
    for df in (dfield, None):
        ref = sl_advect_tangent_at_coords(field, df, du, dv, coords, sl, cl, DT, geo, interp, pole_fix)
        f32 = sl_advect_tangent_at_coords(field, df, du, dv, coords, sl, cl, DT, geo, interp, pole_fix,
                                            compute_dtype=torch.float32)
        ratio = O.worst_ratio(f32.out, ref.out, ref.out_bound)
        print(f"{H}x{W} {interp} poles={poles} pole_fix={pole_fix} dfield={df is not None}: max error/bound {ratio:.3f}")
        assert not O.over_bound(f32.out, ref.out, ref.out_bound).any()


def _flagged(got, ref, bound):
    return {tuple(int(i) for i in t) for t in O.over_bound(got, ref, bound).nonzero()}


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_dropped_velocity_term_is_flagged(interp):
    H, W = 33, 64
    field, dfield, du, dv, coords, sl, cl, geo = _tl_case(H, W, False, interp, seed=3)
    ref = sl_advect_tangent_at_coords(field, dfield, du, dv, coords, sl, cl, DT, geo, interp, True)
    f32 = sl_advect_tangent_at_coords(field, dfield, du, dv, coords, sl, cl, DT, geo, interp, True,
                                        compute_dtype=torch.float32)
    ones = torch.ones(field.shape, dtype=torch.float64)
    g1 = O.sl_advect_at_coords(field, ones, coords, sl, cl, DT, geo, interp, True)
    for term in (g1.grad_u * du.double(), g1.grad_v * dv.double()):
        t = term.clone()
        t[:, :, 0] = 0
        t[:, :, H - 1] = 0                 # a mean row is not a single point
        pt = tuple(int(i) for i in torch.unravel_index(t.abs().argmax(), t.shape))
        out = f32.out.clone()
        out[pt] -= float(term[pt])
        assert _flagged(out, ref.out, ref.out_bound) == {pt}


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_dropped_pole_mean_tangent_is_flagged(interp):
    """A kernel that reads dfield's pole rows raw instead of their zonal means (the tangent of the pole-mean taps) is
    flagged at the points whose stencil reaches a pole row, and nowhere else."""
    H, W = 17, 24
    field, dfield, du, dv, coords, sl, cl, geo = _tl_case(H, W, True, interp, seed=5)
    ref = sl_advect_tangent_at_coords(field, dfield, du, dv, coords, sl, cl, DT, geo, interp, True)
    good = sl_advect_tangent_at_coords(field, dfield, du, dv, coords, sl, cl, DT, geo, interp, True,
                                         compute_dtype=torch.float32).out
    ones = torch.ones(field.shape)
    g1 = O.sl_advect_at_coords(field, ones, coords, sl, cl, DT, geo, interp, True, compute_dtype=torch.float32)
    raw = O.sl_advect_at_coords(dfield, None, coords, sl, cl, DT, geo, interp, False, compute_dtype=torch.float32).out
    bad = O._pole_mean_sequential(O._F32(g1.grad_u).fma(du, O._F32(g1.grad_v).fma(dv, raw)).v)
    change = (bad.double() - good.double()).abs()
    flagged = _flagged(bad, ref.out, ref.out_bound)
    assert flagged, "the case has no stencil on a pole row"
    assert flagged <= {tuple(int(i) for i in t) for t in (change > 0).nonzero()}
    assert flagged >= {tuple(int(i) for i in t) for t in (change > 1e-3 * ref.out.abs().max()).nonzero()}
