"""Every advection kernel path against an fp64 evaluation at the kernels' OWN departure coordinates.

The parity instrument (ops.departure_coords) returns, per arrival point, the fp32 ix, iy and the intermediates of the
rotated-pole map.  out and grad_field are linear in field / grad_out with weights that are exact functions of (ix, iy),
so oracle.sl_advect_at_coords evaluates them in fp64 with no floor() ambiguity, and grad_u / grad_v by the kernels'
Jacobian formula, each with a rigorous per-point rounding bound.  A case passes when NO point of any of the four
outputs is over its bound; it also asserts (torch.profiler kernel names) that the path it targets ran.  The reference
takes the instrument's coordinates, so a kernel whose own trajectory (the packed fp32x2 one of the forward and the row
sweep included) disagrees with the instrument's fails wherever the change of out / grad_u / grad_v that the different
coordinate causes exceeds the point's rounding bound; one ulp of ix does at the most sensitive points
(test_mutated_kernel_output_fails_the_check), not at every point (DESIGN §4.1)."""
import math
import re

import numpy as np
import pytest
import torch

from oracle import sl_oracle as O

pytestmark = pytest.mark.gpu
DT = 21600 * 7.29212e-5 / 8
LABELS = ("out", "grad_field", "grad_u", "grad_v")
MODES = [("fast", True), ("fast", False), ("exact", True), ("exact", False)]

ROWS = r"sl_bwd_rows_kernel<"
GROW = r"rows_grow_fix_kernel"
SWEEP = r"sl_bwd_sweep_kernel<"
GATHER = r"sl_bwd_gather_kernel<"
FWD4 = r"sl_fwd_kernel<\w+, \d, 4,"
FWD1 = r"sl_fwd_kernel<\w+, \d, 1,"


@pytest.fixture(autouse=True)
def _switches():
    from paradis_model_b200 import ops
    saved = (ops.FORCE_ROW_SWEEP, ops.NATIVE_BF16)
    yield
    ops.FORCE_ROW_SWEEP, ops.NATIVE_BF16 = saved


def _pkg():
    import paradis_model_b200 as pkg
    return pkg


def _geo(H, W, poles):
    lat, lon = O.make_grids(H, W, poles)
    return _pkg().SLGeometry.from_grids(lat.cuda(), lon.cuda())


def _tables(geo):
    from paradis_model_b200 import ops
    H, Hp = geo.H, ops._hpad(geo.H)
    return geo.tables[:H], geo.tables[Hp:Hp + H]


def _noise(H, W, B, V, poles, seed=0, sigma=2.0, clip=4.0, dtype=torch.float32):
    lat, lon, field, u, v, go = O.bench_inputs(H, W, B, V, poles, DT, seed=seed, cells_sigma=sigma, cells_clip=clip)
    return [t.cuda().to(dtype) for t in (field, u, v)] + [go.cuda()]


def _kernels(fn):
    """Run fn under the profiler; returns (its result, names of the CUDA kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    return r, {e.name for e in prof.events()}


def _assert_ran(names, *patterns, absent=()):
    for pat in patterns:
        assert any(re.search(pat, n) for n in names), f"kernel {pat!r} did not run; ran: {sorted(names)}"
    for pat in absent:
        assert not any(re.search(pat, n) for n in names), f"kernel {pat!r} ran; ran: {sorted(names)}"


def _fwd_bwd(field, u, v, go, geo, interp, math_mode, pole_fix, cfl, strided=False):
    """One autograd forward + backward through the public op, under the profiler.  A field that is a leaf requiring
    grad is passed as it is (its layout is part of the case), any other is cloned."""
    pkg = _pkg()
    V = field.shape[1]

    def run():
        f = field if field.requires_grad else field.clone().requires_grad_(True)
        if strided:
            uv = torch.cat([u, v], 1).requires_grad_(True)
            uu, vv = uv[:, :V], uv[:, V:]
        else:
            uu, vv = u.clone().requires_grad_(True), v.clone().requires_grad_(True)
        out = pkg.sl_advect(f, uu, vv, geo, DT, interp, pole_fix, math_mode, cfl)
        out.backward(go)
        gu, gv = (uv.grad[:, :V], uv.grad[:, V:]) if strided else (uu.grad, vv.grad)
        return out.detach(), f.grad, gu, gv

    got, names = _kernels(run)
    pkg.check_status()
    return got, names


def _reference(field, u, v, go, geo, interp, math_mode, pole_fix):
    from paradis_model_b200 import ops
    coords = ops.departure_coords(u, v, geo, DT, interp, math_mode)
    sl, cl = _tables(geo)
    return O.sl_advect_at_coords(field.detach().float(), go, coords, sl, cl, DT, geo, interp, pole_fix), coords


def _check(tag, got, ref, bf16=False, rows=None):
    """Zero points over the bound in all four outputs; prints the largest error / bound ratio of each."""
    ratios, bad = [], []
    sel = (slice(None), slice(None), rows) if rows is not None else (slice(None),)
    for lab, x, y, b in zip(LABELS, got, ref.values(), ref.bounds()):
        y, b = y[sel], b[sel]
        if bf16 and lab != "out":
            b = O.bf16_bounds(y, b)
        over = O.over_bound(x, y, b)
        ratios.append(O.worst_ratio(x, y, b))
        if over.any():
            i = tuple(int(k) for k in over.nonzero()[0])
            bad.append(f"{lab}: {int(over.sum())} points over the bound, first {i}: got {float(x[i]):.9g}, "
                       f"ref {float(y[i]):.9g}, bound {float(b[i]):.3g}")
    print(f"[{tag}] max error/bound " + " ".join(f"{n}={q:.3g}" for n, q in zip(LABELS, ratios)))
    assert not bad, f"[{tag}] " + "; ".join(bad)


def _case(tag, field, u, v, go, geo, interp, math_mode, pole_fix, cfl, kernels, absent=(), strided=False):
    got, names = _fwd_bwd(field, u, v, go, geo, interp, math_mode, pole_fix, cfl, strided)
    _assert_ran(names, *kernels, absent=absent)
    ref, coords = _reference(field, u, v, go, geo, interp, math_mode, pole_fix)
    _check(tag, got, ref, bf16=field.dtype == torch.bfloat16)
    return got, ref, coords


# ------------------------------------------------------------------ full mesh, row sweep (warm-up scheme)
@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_full_mesh_row_sweep_v8(math_mode, pole_fix):
    field, u, v, go = _noise(721, 1440, 1, 8, True, seed=1)
    _case(f"C3 V=8 {math_mode} pole_fix={pole_fix}", field, u, v, go, _geo(721, 1440, True), "bilinear", math_mode,
          pole_fix, 6.0, [ROWS, FWD4])


def test_full_mesh_row_sweep_v16_and_smooth():
    geo = _geo(721, 1440, True)
    field, u, v, go = _noise(721, 1440, 1, 16, True, seed=2)
    _case("C3 V=16 fast", field, u, v, go, geo, "bilinear", "fast", True, 6.0, [ROWS, FWD4])
    lat, lon = O.make_grids(721, 1440, True)
    f = O.smooth_field(lat, lon, 1, 4).float().cuda()
    us, vs = [t.float().cuda() for t in O.smooth_velocity(lat, lon, 1, 4, 4.0, DT)]
    _case("C3 smooth fast", f, us, vs, go[:, :4].contiguous(), geo, "bilinear", "fast", True, 6.0, [ROWS, FWD4])


# ------------------------------------------------------------------ ragged strips of the row sweep
@pytest.mark.parametrize("W", [1000, 904])
@pytest.mark.parametrize("poles", [True, False])
def test_row_sweep_ragged_strips(W, poles):
    H = 361 if poles else 360
    field, u, v, go = _noise(H, W, 1, 3, poles, seed=W)
    _case(f"{H}x{W} poles={poles}", field, u, v, go, _geo(H, W, poles), "bilinear", "fast", True, 6.0, [ROWS, FWD4])


# ------------------------------------------------------------------ forced row sweep
@pytest.mark.parametrize("math_mode,pole_fix", [("fast", True), ("exact", False)])
@pytest.mark.parametrize("interp", ["bicubic", "bilinear"])
def test_row_sweep_forced(interp, math_mode, pole_fix):
    from paradis_model_b200 import ops
    ops.FORCE_ROW_SWEEP = True
    field, u, v, go = _noise(181, 360, 2, 3, True, seed=3)
    _case(f"forced rows 181x360 {interp} {math_mode} pole_fix={pole_fix}", field, u, v, go, _geo(181, 360, True),
          interp, math_mode, pole_fix, 6.0, [ROWS], strided=True)


@pytest.mark.parametrize("H,W,cfl", [(33, 64, 3.0), (33, 32, 3.0), (8, 64, 1.0)])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_row_sweep_forced_one_strip_and_short_mesh(H, W, cfl, interp):
    """W = 32: one strip, its guard columns wrap onto itself; H = 8: the shortest mesh the row sweep takes."""
    from paradis_model_b200 import ops
    ops.FORCE_ROW_SWEEP = True
    field, u, v, go = _noise(H, W, 1, 3, True, seed=H * W, sigma=0.5 * cfl, clip=cfl)
    _case(f"forced rows {H}x{W} {interp}", field, u, v, go, _geo(H, W, True), interp, "fast", True, cfl, [ROWS])


# ------------------------------------------------------------------ strip sweep + polar caps on side streams
@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_strip_sweep_bicubic_c3(math_mode, pole_fix):
    field, u, v, go = _noise(721, 1440, 1, 2, True, seed=4)
    _case(f"C3 bicubic V=2 {math_mode} pole_fix={pole_fix}", field, u, v, go, _geo(721, 1440, True), "bicubic",
          math_mode, pole_fix, 6.0, [SWEEP, GATHER, FWD1], absent=[ROWS])


@pytest.mark.parametrize("H,W", [(128, 256), (181, 360)])
@pytest.mark.parametrize("pole_fix", [True, False])
def test_strip_sweep_bilinear(H, W, pole_fix):
    field, u, v, go = _noise(H, W, 2, 3, H % 2 == 1, seed=H)
    _case(f"strip sweep {H}x{W} pole_fix={pole_fix}", field, u, v, go, _geo(H, W, H % 2 == 1), "bilinear", "fast",
          pole_fix, 6.0, [SWEEP, GATHER, FWD4], absent=[ROWS])


# ------------------------------------------------------------------ general path (arrival + gather)
@pytest.mark.parametrize("H,W,poles", [(5, 6, True), (6, 18, False), (7, 50, True), (33, 1442, False)])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_general_path_ragged(H, W, poles, interp):
    field, u, v, go = _noise(H, W, 2, 2, poles, seed=H + W)
    _case(f"general {H}x{W} {interp}", field, u, v, go, _geo(H, W, poles), interp, "fast", True, 0.0,
          [GATHER, FWD1], absent=[ROWS, SWEEP])


@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_general_path_misaligned_and_strided(math_mode, pole_fix):
    """cfl = 0; a field one element off 16-byte alignment (scalar forward) and batch-strided u / v views."""
    field, u, v, go = _noise(128, 256, 2, 3, True, seed=5)
    geo = _geo(128, 256, True)
    store = torch.empty(field.numel() + 1, device="cuda")
    mis = store[1:].view(field.shape)
    mis.copy_(field)
    mis.requires_grad_(True)
    _case(f"general misaligned {math_mode} pole_fix={pole_fix}", mis, u, v, go, geo, "bilinear", math_mode, pole_fix,
          0.0, [GATHER, FWD1], absent=[ROWS, SWEEP])
    _case(f"general strided {math_mode} pole_fix={pole_fix}", field, u, v, go, geo, "bicubic", math_mode, pole_fix,
          0.0, [GATHER], absent=[ROWS, SWEEP], strided=True)


# ------------------------------------------------------------------ contract fallback
@pytest.mark.parametrize("force_rows", [False, True])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_contract_fallback(force_rows, interp):
    """One plane moves up to 8 cells against a hint of 3: the sweep flags it, the filtered general path redoes it."""
    from paradis_model_b200 import ops
    ops.FORCE_ROW_SWEEP = force_rows
    field, u, v, go = _noise(181, 360, 1, 4, True, seed=6, sigma=1.0, clip=2.0)
    u[:, 1] *= 4.0
    v[:, 2] *= 4.0
    _case(f"fallback {interp} rows={force_rows}", field, u, v, go, _geo(181, 360, True), interp, "fast", True, 3.0,
          [ROWS if force_rows else SWEEP, GATHER])


# ------------------------------------------------------------------ cross-pole departures
@pytest.mark.parametrize("force_rows", [False, True])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_cross_pole_departures(force_rows, interp):
    """The 4 rows next to each pole move 3.5 cells poleward (lat' = -v dt: v > 0 is southward), so their departure
    points lie beyond the pole: same latitude band on the other side, longitude shifted by about pi."""
    from paradis_model_b200 import ops
    ops.FORCE_ROW_SWEEP = force_rows
    H, W = 181, 360
    field, u, v, go = _noise(H, W, 1, 3, True, seed=7, sigma=1.0, clip=2.0)
    cell = math.pi / H / DT
    v[:, :, :4] = 3.5 * cell           # southern rows move south across the south pole
    v[:, :, -4:] = -3.5 * cell         # northern rows north across the north pole
    geo = _geo(H, W, True)
    _, _, coords = _case(f"cross-pole {interp} rows={force_rows}", field, u, v, go, geo, interp, "fast", True, 6.0,
                         [ROWS if force_rows else SWEEP])
    lon_arr = geo.tables[2 * ops._hpad(H):]
    shift = (coords[:, :, 10] - lon_arr + math.pi).remainder(2 * math.pi) - math.pi
    crossed = shift.abs() > math.pi / 2
    p = 1 if interp == "bilinear" else 2
    row = torch.floor(coords[:, :, 1]) - p                 # row of the departure cell
    for rows in (slice(1, 4), slice(H - 4, H - 1)):
        assert float(crossed[:, :, rows].float().mean()) > 0.9, "departures of the pole rows did not cross the pole"
    if interp == "bicubic":                                # stencil rows beyond the pole: the cap fold
        assert bool((row[:, :, :4] - 1 < 0).any()) and bool((row[:, :, -4:] + 2 > H - 1).any())


# ------------------------------------------------------------------ latitude bands on one GPU
def _band_case(H, W, V, own, ext, cfl, field, u, v, go, geo, ref, tag):
    sl = slice(own[0], own[0] + own[1])
    e = slice(ext[0], ext[0] + ext[1])
    gb = geo.band(own, ext, ext)
    fo = geo.band(own, own, ext)

    def run():
        out = torch.ops.paradis.sl_advect(field[:, :, e].contiguous(), u[:, :, sl].contiguous(),
                                          v[:, :, sl].contiguous(), fo.tables, fo.scalars, DT, 1, True, 0,
                                          fo.windows, cfl)
        g = torch.ops.paradis.sl_advect_backward(go[:, :, e].contiguous(), field[:, :, e].contiguous(),
                                                 u[:, :, e].contiguous(), v[:, :, e].contiguous(), gb.tables,
                                                 gb.scalars, DT, 1, True, 0, gb.windows, cfl, True, True)
        return (out,) + tuple(g)

    got, names = _kernels(run)
    _pkg().check_status()
    _check(tag, got, ref, rows=sl)
    return names


@pytest.mark.parametrize("world", [2, 4, 8])
def test_latitude_bands_c3(world):
    """Every band of the 2 / 4 / 8-way split takes the cut mode (its own arrival rows only, the partial rows beyond
    the cuts added by rows_grow_fix_kernel)."""
    from paradis_model_b200 import halo
    H, W, V, cfl = 721, 1440, 4, 6.0
    field, u, v, go = _noise(H, W, 1, V, True, seed=8)
    geo = _geo(H, W, True)
    ref, _ = _reference(field, u, v, go, geo, "bilinear", "fast", True)
    for rank in range(world):
        own, ext = halo.make_plan(H, W, rank, world, cfl, "bilinear").windows()
        names = _band_case(H, W, V, own, ext, cfl, field, u, v, go, geo, ref, f"band {rank}/{world}")
        _assert_ran(names, ROWS, GROW)


@pytest.mark.parametrize("H,W,V,own,ext,cfl,cut", [
    (721, 1440, 4, (0, 47), (0, 56), 6.0, True),          # southern polar band of the balanced 8-way split
    (721, 1440, 4, (149, 105), (140, 123), 6.0, True),    # a mid-latitude band of it
    (64, 128, 2, (0, 12), (0, 21), 6.0, True),            # 12 own rows: ranges shorter than the guard depth
    (181, 360, 2, (61, 60), (45, 92), 13.0, False),       # hint 13: rr + NT = 15 guard rows exceed the side buffer
])
def test_band_shapes_cut_and_warm_up(H, W, V, own, ext, cfl, cut):
    """Band shapes of test_partition.py through the kernels (row sweep forced on the narrow meshes), with the scheme
    each one takes: cut mode (rows_grow_fix_kernel runs) or the warm-up scheme (it does not)."""
    from paradis_model_b200 import ops
    ops.FORCE_ROW_SWEEP = True
    field, u, v, go = _noise(H, W, 1, V, True, seed=H + own[0], sigma=1.5, clip=3.0)
    geo = _geo(H, W, True)
    ref, _ = _reference(field, u, v, go, geo, "bilinear", "fast", True)
    names = _band_case(H, W, V, own, ext, cfl, field, u, v, go, geo, ref, f"band {own} of {H}x{W} cfl {cfl}")
    _assert_ran(names, ROWS, *([GROW] if cut else []), absent=[] if cut else [GROW])


# ------------------------------------------------------------------ FAST wrap rule (DESIGN §7)
def _wrap_velocity(geo, y):
    """u at column 0 of row y whose FAST-mode ix rounds up to W + p (wrapped to p by the kernels), by bisection with
    the instrument over u > 0 (departures west of longitude 0, i.e. just below 2 pi)."""
    from paradis_model_b200 import ops
    H, W = geo.H, geo.W

    def probe(us):
        n = us.numel()
        uu = torch.zeros(1, n, H, W, device="cuda")
        uu[0, :, y, 0] = us
        c = ops.departure_coords(uu, torch.zeros_like(uu), geo, DT, "bilinear", "fast")[0, :, :, y, 0]
        return c[:, 0], c[:, 10]                    # ix, lon

    lo, hi = 0.0, 1e-3 / DT                          # lon(lo) = 0, lon(hi) just below 2 pi
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        _, lon = probe(torch.tensor([mid], device="cuda"))
        lo, hi = (mid, hi) if float(lon[0]) < math.pi else (lo, mid)
    cand = torch.tensor(hi, dtype=torch.float32, device="cuda")
    steps = [cand]
    for _ in range(7):
        steps.append(torch.nextafter(steps[-1], torch.tensor(math.inf, device="cuda")))
    us = torch.stack(steps)
    ix, lon = probe(us)
    hit = ((lon > math.pi) & (ix < 1.5)).nonzero()
    assert hit.numel(), "no fp32 u of the bisection bracket rounds ix up to W + p"
    return float(us[int(hit[0])])


def test_fast_wrap_rule():
    H, W, y = 721, 1440, 300
    geo = _geo(H, W, True)
    field, u, v, go = _noise(H, W, 1, 2, True, seed=9)
    uw = _wrap_velocity(geo, y)
    u[0, 0, y, 0] = uw
    v[0, 0, y, 0] = 0.0
    _, _, coords = _case("wrap", field, u, v, go, geo, "bilinear", "fast", True, 6.0, [ROWS, FWD4])
    assert float(coords[0, 0, 0, y, 0]) == 1.0 and float(coords[0, 0, 10, y, 0]) > math.pi


# ------------------------------------------------------------------ bf16 storage
def test_bf16_row_sweep_and_strip_sweep():
    field, u, v, go = _noise(721, 1440, 1, 4, True, seed=10, dtype=torch.bfloat16)
    _case("bf16 C3 rows", field, u, v, go, _geo(721, 1440, True), "bilinear", "fast", True, 6.0, [ROWS, FWD4])
    field, u, v, go = _noise(128, 256, 2, 3, True, seed=11, dtype=torch.bfloat16)
    _case("bf16 strip sweep bicubic", field, u, v, go, _geo(128, 256, True), "bicubic", "fast", True, 6.0,
          [SWEEP, GATHER])


# ------------------------------------------------------------------ the check catches a wrong kernel output
def test_mutated_kernel_output_fails_the_check():
    H, W = 181, 360
    field, u, v, go = _noise(H, W, 1, 2, True, seed=12)
    geo = _geo(H, W, True)
    got, ref, coords = _case("mutation base", field, u, v, go, geo, "bilinear", "fast", True, 6.0, [SWEEP])
    out, gf = got[0].clone(), got[1].clone()
    # one grad_field contribution of an arrival point at mid-latitude moved one column sideways
    idx, ok, w, _ = max(ref.taps, key=lambda t: float(t[2][0, 0, 90, 100].abs()))
    g = O._pole_mean_adjoint(go.double())
    c = float(w[0, 0, 90, 100] * g[0, 0, 90, 100])
    i, j = divmod(int(idx[0, 0, 90, 100]), W)
    gf[0, 0, i, j] -= c
    gf[0, 0, i, (j + 1) % W] += c
    over = O.over_bound(gf, ref.grad_field, ref.grad_field_bound)
    assert {tuple(int(k) for k in t) for t in over.nonzero()} == {(0, 0, i, j), (0, 0, i, (j + 1) % W)}
    # one ulp of one ix, applied to out
    sl, cl = _tables(geo)
    bumped = coords.clone()
    bumped[:, :, 0] = torch.nextafter(coords[:, :, 0], torch.tensor(math.inf, device="cuda"))
    every = O.sl_advect_at_coords(field, go, bumped, sl, cl, DT, geo, "bilinear", True).out
    score = (every - ref.out).abs() / ref.out_bound
    score[:, :, 0] = 0
    score[:, :, H - 1] = 0
    pt = tuple(int(k) for k in np.unravel_index(int(score.argmax()), score.shape))
    out[pt] += float(every[pt] - ref.out[pt])
    over = O.over_bound(out, ref.out, ref.out_bound)
    assert {tuple(int(k) for k in t) for t in over.nonzero()} == {pt}


# ------------------------------------------------------------------ displacement limit: 126 rows
def _class_velocity(geo, y, x, k):
    """v at (y, x) whose departure row class floor(iy) - (y + p) is k, by bisection with the instrument on iy
    crossing y + p + k + 1/2."""
    from paradis_model_b200 import ops
    H, W = geo.H, geo.W
    target = y + 1 + k + 0.5

    def iy(vv):
        t = torch.zeros(1, 1, H, W, device="cuda")
        t[0, 0, y, x] = vv
        return float(ops.departure_coords(torch.zeros_like(t), t, geo, DT, "bilinear", "fast")[0, 0, 1, y, x])

    lim = 1.5 / DT                                   # 1.5 rad of latitude either way
    lo, hi = (-lim, 0.0) if k > 0 else (0.0, lim)    # v < 0: lat' = -v dt > 0, northward
    for _ in range(60):                              # iy decreases from lo to hi either way
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if iy(mid) > target else (lo, mid)
    vv = 0.5 * (lo + hi)
    assert math.floor(iy(vv)) - (y + 1) == k
    return vv


@pytest.mark.parametrize("cfl", [0.0, 6.0], ids=["general", "sweep-fallback"])
def test_displacement_126_rows(cfl):
    H, W, y, x = 361, 720, 180, 100
    geo = _geo(H, W, True)
    field, u, v, go = _noise(H, W, 1, 2, True, seed=13, sigma=1.0, clip=2.0)
    u[:, :, y, x] = 0.0
    v[0, 0, y, x] = _class_velocity(geo, y, x, 126)
    v[0, 1, y, x] = _class_velocity(geo, y, x, -126)
    _, ref, coords = _case(f"126 rows cfl={cfl}", field, u, v, go, geo, "bilinear", "fast", True, cfl,
                           [GATHER] if cfl == 0 else [SWEEP, GATHER])
    assert [math.floor(float(coords[0, c, 1, y, x])) - (y + 1) for c in (0, 1)] == [126, -126]
    _pkg().check_status()


def test_displacement_127_rows_is_reported():
    pkg = _pkg()
    H, W, y, x = 361, 720, 180, 100
    geo = _geo(H, W, True)
    field, u, v, go = _noise(H, W, 1, 2, True, seed=14, sigma=1.0, clip=2.0)
    for c, k in ((0, 127), (1, -127)):
        vv = v.clone()
        vv[0, c, y, x] = _class_velocity(geo, y, x, k)
        f = field.clone().requires_grad_(True)
        uu, vq = u.clone().requires_grad_(True), vv.requires_grad_(True)
        pkg.sl_advect(f, uu, vq, geo, DT, "bilinear", True, "fast", 0.0).backward(go)
        with pytest.raises(RuntimeError, match="DISPLACEMENT"):
            pkg.check_status()
