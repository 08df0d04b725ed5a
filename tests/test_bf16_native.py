"""Native bf16 storage of the advection op (include/paradis_sl_bf16.h, ops.NATIVE_BF16): with bf16 field / u / v the
kernels read bf16 and write bf16 gradients.  Every comparison is torch.equal against the fp32 op run on .float() copies
of the same bf16 values, with the gradients rounded by .to(torch.bfloat16) -- the upcast path the native one replaces."""
import math

import pytest
import torch

from oracle import sl_oracle as O
from paradis_model_b200 import ops
from paradis_model_b200 import synthetic as S

pytestmark = pytest.mark.gpu
DT = S.DT_DEFAULT
BF = torch.bfloat16


@pytest.fixture(autouse=True)
def _restore_switches():
    yield
    ops.NATIVE_BF16 = True
    ops.FORCE_ROW_SWEEP = False


def _pkg():
    import paradis_model_b200 as pkg
    return pkg


def _inputs(H, W, B, V, poles, seed=0, clip=4.0):
    field, u, v, go = S.white_noise_inputs(H, W, B, V, seed=seed, cells_clip=clip)
    lat, lon = O.make_grids(H, W, poles)
    geo = _pkg().SLGeometry.from_grids(lat.cuda(), lon.cuda())
    return geo, field.cuda().to(BF), u.cuda().to(BF), v.cuda().to(BF), go.cuda()


def _fwd_bwd(field, u, v, go, geo, interp, math_mode, pole_fix, cfl, req=(True, True, True), strided=False):
    """One autograd fwd + bwd; strided: u, v are views of one [B, 2V, H, W] tensor (model/paradis.py:235-237)."""
    V = field.shape[1]
    f = field.clone().requires_grad_(req[0])
    if strided:
        uv = torch.cat([u, v], 1).requires_grad_(req[1])
        uu, vv = uv[:, :V], uv[:, V:]
    else:
        uu, vv = u.clone().requires_grad_(req[1]), v.clone().requires_grad_(req[2])
    out = _pkg().sl_advect(f, uu, vv, geo, DT, interp, pole_fix, math_mode, cfl)
    out.backward(go)
    _pkg().check_status()
    if strided:
        gu, gv = (uv.grad[:, :V], uv.grad[:, V:]) if req[1] else (None, None)
    else:
        gu, gv = uu.grad, vv.grad
    return out.detach(), f.grad, gu, gv


def _check_native(field, u, v, go, geo, interp, math_mode="fast", pole_fix=True, cfl=8.0, req=(True, True, True),
                  strided=False):
    got = _fwd_bwd(field, u, v, go, geo, interp, math_mode, pole_fix, cfl, req, strided)
    ref = _fwd_bwd(field.float(), u.float(), v.float(), go, geo, interp, math_mode, pole_fix, cfl, req, strided)
    assert got[0].dtype == torch.float32 and torch.equal(got[0], ref[0]), "out"
    for k, name in ((1, "grad_field"), (2, "grad_u"), (3, "grad_v")):
        if ref[k] is None:
            assert got[k] is None, name
            continue
        assert got[k].dtype == BF, name
        assert torch.equal(got[k], ref[k].to(BF)), name


MODES = [("fast", True), ("fast", False), ("exact", True), ("exact", False)]


@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_row_sweep_c3(math_mode, pole_fix):
    """721 x 1440 bilinear: the warp-specialised row sweep (TMA-staged bf16 rows of u, v)."""
    geo, field, u, v, go = _inputs(721, 1440, 1, 2, True)
    _check_native(field, u, v, go, geo, "bilinear", math_mode, pole_fix)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_row_sweep_forced_small_mesh(interp, math_mode, pole_fix):
    ops.FORCE_ROW_SWEEP = True
    geo, field, u, v, go = _inputs(181, 360, 2, 3, True, seed=1)
    _check_native(field, u, v, go, geo, interp, math_mode, pole_fix, strided=True)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_strip_sweep_and_caps(interp, math_mode, pole_fix):
    """128 x 256: the strip sweep over the mid-latitudes plus the general path on the polar caps."""
    geo, field, u, v, go = _inputs(128, 256, 2, 4, True, seed=2)
    _check_native(field, u, v, go, geo, interp, math_mode, pole_fix)
    _check_native(field, u, v, go, geo, interp, math_mode, pole_fix, strided=True)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_general_path(interp, math_mode, pole_fix):
    """cfl_cells = 0 on a sweepable mesh, and W = 64 (too narrow for either sweep)."""
    geo, field, u, v, go = _inputs(128, 256, 2, 3, True, seed=3)
    _check_native(field, u, v, go, geo, interp, math_mode, pole_fix, cfl=0.0)
    geo, field, u, v, go = _inputs(33, 64, 2, 3, True, seed=4)
    _check_native(field, u, v, go, geo, interp, math_mode, pole_fix, strided=True)


@pytest.mark.parametrize("force_rows", [False, True])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("math_mode,pole_fix", MODES)
def test_contract_violating_plane_recomputed(force_rows, interp, math_mode, pole_fix):
    """One plane moves up to 6 cells against a CFL hint of 3: the sweep flags it and the general path recomputes it."""
    ops.FORCE_ROW_SWEEP = force_rows
    geo, field, u, v, go = _inputs(128, 256, 2, 3, True, seed=5, clip=1.5)
    u, v = u.clone(), v.clone()
    u[0, 1] *= 4
    v[0, 1] *= 4
    _check_native(field, u, v, go, geo, interp, math_mode, pole_fix, cfl=3.0)


@pytest.mark.parametrize("req", [(True, False, False), (False, True, True)], ids=["field-only", "uv-only"])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_partial_requires_grad(req, interp):
    geo, field, u, v, go = _inputs(128, 256, 2, 3, True, seed=6)
    _check_native(field, u, v, go, geo, interp, req=req)
    _check_native(field, u, v, go, geo, interp, req=req, strided=True)


def _ops_in(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


def test_native_call_launches_no_cast():
    geo, field, u, v, go = _inputs(128, 256, 2, 4, True, seed=7)
    f, uu, vv = [t.clone().requires_grad_(True) for t in (field, u, v)]

    def step():
        _pkg().sl_advect(f, uu, vv, geo, DT, "bilinear").backward(go)

    step()                                                   # warm-up (library load, side streams)
    names = _ops_in(step)
    assert "aten::_to_copy" not in names, sorted(names)
    ops.NATIVE_BF16 = False
    assert "aten::_to_copy" in _ops_in(step)


def _peak_fwd_bwd(field, u, v, go, geo):
    f, uu, vv = [t.clone().requires_grad_(True) for t in (field, u, v)]
    _pkg().sl_advect(f, uu, vv, geo, DT, "bilinear").backward(go)        # warm-up: allocator pools, library
    f.grad = uu.grad = vv.grad = None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    _pkg().sl_advect(f, uu, vv, geo, DT, "bilinear").backward(go)
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_peak_memory_lower_than_upcast():
    geo, field, u, v, go = _inputs(181, 360, 1, 64, True, seed=8)
    native = _peak_fwd_bwd(field, u, v, go, geo)
    ops.NATIVE_BF16 = False
    upcast = _peak_fwd_bwd(field, u, v, go, geo)
    three_copies = 3 * field.numel() * 4
    assert upcast - native >= three_copies, (native, upcast, three_copies)


@pytest.mark.parametrize("case", ["fp16", "mixed", "w_not_8", "lat_band"])
def test_ineligible_calls_unchanged(case):
    """fp16, mixed bf16 / fp32, W % 8 != 0 and a latitude-band call take the upcast path: same values and dtypes with
    the native switch on and off."""
    H, W = (36, 68) if case == "w_not_8" else (64, 128)
    geo, field, u, v, go = _inputs(H, W, 2, 3, True, seed=9, clip=1.5)
    if case == "fp16":
        field, u, v = field.half(), u.half(), v.half()
    elif case == "mixed":
        u = u.float()
    if case == "lat_band":
        own = (20, 24)
        band = geo.band(own, own, (0, H))
        runs = []
        for native in (True, False):
            ops.NATIVE_BF16 = native
            runs.append(_pkg().sl_advect(field, u[:, :, 20:44], v[:, :, 20:44], band, DT, "bilinear"))
        _pkg().check_status()
        assert runs[0].dtype == torch.float32 and torch.equal(runs[0], runs[1])
        return
    runs = []
    for native in (True, False):
        ops.NATIVE_BF16 = native
        runs.append(_fwd_bwd(field, u, v, go, geo, "bicubic", "fast", True, 8.0))
    for a, b in zip(*runs):
        assert a.dtype == b.dtype and torch.equal(a, b)
    assert runs[0][1].dtype == field.dtype and runs[0][2].dtype == u.dtype


def test_compile_autocast_checkpoint_bit_equal_to_eager():
    from torch.utils.checkpoint import checkpoint
    geo, field, u, v, go = _inputs(128, 256, 2, 4, True, seed=10)
    fn = lambda a, b, c: _pkg().sl_advect(a, b, c, geo, DT, "bicubic")

    def grads(call, amp=False, ckpt=False):
        f, uu, vv = [t.clone().requires_grad_(True) for t in (field, u, v)]
        with torch.autocast("cuda", dtype=BF, enabled=amp):
            out = checkpoint(call, f, uu, vv, use_reentrant=False) if ckpt else call(f, uu, vv)
        out.backward(go)
        return out.detach(), f.grad, uu.grad, vv.grad

    eager = grads(fn)
    assert all(g.dtype == BF for g in eager[1:])
    compiled = torch.compile(fn, fullgraph=True)
    for other in (grads(compiled), grads(fn, amp=True), grads(fn, ckpt=True), grads(compiled, amp=True)):
        for a, b in zip(eager, other):
            assert a.dtype == b.dtype and torch.equal(a, b)
