"""Tangent-linear advection (paradis::sl_advect_jvp, sl_tl_kernel) and forward-mode AD through every public op.

The tangent is checked against tangent_reference.sl_advect_tangent_at_coords at the kernels' own fp32 departure
coordinates (ops.departure_coords), with zero points over the per-point fp64 bound; against the forward where it must reduce to it
exactly; and against the existing backward by the dot-product test <J t, g> = <t, J^T g>.  Every advection case
asserts by profiler kernel name whether the tangent-linear kernel ran."""
import math

import pytest
import torch
import torch.autograd.forward_ad as fwAD

from oracle import paradis_assembly as A
from oracle import sl_oracle as O
from tangent_reference import sl_advect_tangent_at_coords
from test_kernel_coords_fp64 import DT, _assert_ran, _geo, _noise, _tables, _wrap_velocity

pytestmark = pytest.mark.gpu
TL = r"sl_tl_kernel<"


@pytest.fixture(autouse=True)
def _fp32_convolutions():
    """True fp32 convolutions (cuDNN defaults to TF32) for the dot-product tests through the model."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _kernels(fn):
    """Run fn under the profiler; returns (its result, names of the events, CUDA kernels included).  In a long process
    (after the compiled-model tests) the profiler was seen to lose the last device record of a session, so a fill
    kernel follows fn inside the session, and a session without any device record is repeated (up to three times)."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r = fn()
            torch.zeros(1, device="cuda")
            torch.cuda.synchronize()
        events = prof.events()
        if any(e.device_type == torch.autograd.DeviceType.CUDA for e in events):
            break
    return r, {e.name for e in events}


def _ops():
    from paradis_model_b200 import ops
    return ops


def _advect(geo, interp, math_mode, pole_fix):
    return lambda f, u, v: _ops().sl_advect(f, u, v, geo, DT, interp, pole_fix, math_mode)


def _jvp(geo, interp, math_mode, pole_fix, primals, tangents):
    return torch.func.jvp(_advect(geo, interp, math_mode, pole_fix), primals, tangents)[1]


def _tangents(field, u, v, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda t, s: torch.randn(t.shape, generator=g, device="cuda") * s
    sig = float(u.abs().mean())
    return r(field, 1.0), r(u, sig), r(v, sig)


def _check_tl(tag, field, u, v, df, du, dv, geo, interp, math_mode, pole_fix):
    """Tangent through torch.func.jvp against the fp64 reference; asserts the tangent-linear kernel ran."""
    got, names = _kernels(lambda: _jvp(geo, interp, math_mode, pole_fix, (field, u, v), (df, du, dv)))
    _ops().check_status()
    _assert_ran(names, TL)
    coords = _ops().departure_coords(u, v, geo, DT, interp, math_mode)
    sl, cl = _tables(geo)
    ref = sl_advect_tangent_at_coords(field.float(), df.float(), du.float(), dv.float(), coords, sl, cl, DT, geo,
                                        interp, pole_fix)
    over = O.over_bound(got, ref.out, ref.out_bound)
    print(f"[{tag}] max error/bound {O.worst_ratio(got, ref.out, ref.out_bound):.3g}")
    assert not over.any(), f"[{tag}] {int(over.sum())} points over the bound"
    return got


# ------------------------------------------------------------------ fp64 bound
@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("math_mode", ["fast", "exact"])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_tangent_fp64_bound_128x256(interp, math_mode, pole_fix):
    H, W = 128, 256
    field, u, v, _ = _noise(H, W, 2, 3, False, seed=1)
    _check_tl(f"128x256 {interp} {math_mode} pole_fix={pole_fix}", field, u, v, *_tangents(field, u, v, 2),
              _geo(H, W, False), interp, math_mode, pole_fix)


@pytest.mark.parametrize("H,W,poles", [(181, 360, True), (64, 1000, True), (64, 904, False), (33, 50, True),
                                       (5, 6, True), (7, 50, False)])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_tangent_fp64_bound_shapes(H, W, poles, interp):
    """Ragged widths, a width without float4 rows (33 x 50: one point per thread) and tiny meshes."""
    field, u, v, _ = _noise(H, W, 1, 2, poles, seed=H + W)
    for math_mode, pole_fix in (("fast", True), ("exact", False)):
        _check_tl(f"{H}x{W} {interp} {math_mode} pole_fix={pole_fix}", field, u, v, *_tangents(field, u, v, 3),
                  _geo(H, W, poles), interp, math_mode, pole_fix)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_tangent_cross_pole_departures(interp):
    H, W = 181, 360
    field, u, v, _ = _noise(H, W, 1, 3, True, seed=7, sigma=1.0, clip=2.0)
    cell = math.pi / H / DT
    v[:, :, :4] = 3.5 * cell
    v[:, :, -4:] = -3.5 * cell
    geo = _geo(H, W, True)
    coords = _ops().departure_coords(u, v, geo, DT, interp, "fast")
    shift = (coords[:, :, 10] - geo.tables[2 * _ops()._hpad(H):] + math.pi).remainder(2 * math.pi) - math.pi
    assert float((shift[:, :, 1:4].abs() > math.pi / 2).float().mean()) > 0.9
    _check_tl(f"cross-pole {interp}", field, u, v, *_tangents(field, u, v, 4), geo, interp, "fast", True)


def test_tangent_fast_wrap_point():
    H, W, y = 721, 1440, 300
    geo = _geo(H, W, True)
    field, u, v, _ = _noise(H, W, 1, 2, True, seed=9)
    u[0, 0, y, 0] = _wrap_velocity(geo, y)
    v[0, 0, y, 0] = 0.0
    coords = _ops().departure_coords(u, v, geo, DT, "bilinear", "fast")
    assert float(coords[0, 0, 0, y, 0]) == 1.0
    _check_tl("wrap", field, u, v, *_tangents(field, u, v, 5), geo, "bilinear", "fast", True)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_tangent_batch_strided_views(interp):
    """u, v and du, dv as the two halves of one [B, 2V, H, W] tensor each (model/paradis.py:235-237)."""
    H, W, B, V = 128, 256, 2, 3
    field, u, v, _ = _noise(H, W, B, V, True, seed=11)
    df, du, dv = _tangents(field, u, v, 6)
    uv, duv = torch.cat([u, v], 1), torch.cat([du, dv], 1)
    got = _check_tl(f"strided {interp}", field, uv[:, :V], uv[:, V:], df, duv[:, :V], duv[:, V:], _geo(H, W, True),
                    interp, "fast", True)
    ref = _jvp(_geo(H, W, True), interp, "fast", True, (field, u, v), (df, du, dv))
    assert torch.equal(got, ref)


# ------------------------------------------------------------------ exact reductions
@pytest.mark.parametrize("H,W", [(128, 256), (33, 50)])
@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("math_mode", ["fast", "exact"])
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_zero_velocity_tangent_is_the_forward_on_dfield(interp, math_mode, pole_fix, H, W):
    field, u, v, _ = _noise(H, W, 2, 3, True, seed=12)
    geo = _geo(H, W, True)
    df, _, _ = _tangents(field, u, v, 7)
    fn = _advect(geo, interp, math_mode, pole_fix)
    zu, zv = torch.zeros_like(u), torch.zeros_like(v)
    got, names = _kernels(lambda: _jvp(geo, interp, math_mode, pole_fix, (field, u, v), (df, zu, zv)))
    _assert_ran(names, TL)
    assert torch.equal(got, fn(df, u, v))
    got, names = _kernels(lambda: torch.func.jvp(lambda f: fn(f, u, v), (field,), (df,))[1])
    _assert_ran(names, absent=[TL])
    assert torch.equal(got, fn(df, u, v))


# ------------------------------------------------------------------ TL / AD dot-product test
def _dot_ratio(jt, g, t, jtg):
    """|<J t, g> - <t, J^T g>| / sum of |terms|, the sums in fp64 from the fp32 results."""
    lhs = (jt.double() * g.double())
    rhs = [(a.double() * b.double()) for a, b in zip(t, jtg)]
    diff = lhs.sum() - sum(r.sum() for r in rhs)
    scale = lhs.abs().sum() + sum(r.abs().sum() for r in rhs)
    return float(diff.abs() / scale)


@pytest.mark.parametrize("H,W,B,V,interp", [(721, 1440, 1, 8, "bilinear"), (128, 256, 8, 64, "bicubic")])
def test_dot_product_against_backward(H, W, B, V, interp):
    field, u, v, go = _noise(H, W, B, V, True, seed=13)
    geo = _geo(H, W, True)
    t = _tangents(field, u, v, 8)
    jt = _jvp(geo, interp, "fast", True, (field, u, v), t)
    prim = [x.clone().requires_grad_(True) for x in (field, u, v)]
    out = _advect(geo, interp, "fast", True)(*prim)
    jtg = torch.autograd.grad(out, prim, go)
    r = _dot_ratio(jt, go, t, jtg)
    print(f"[dot {H}x{W} B={B} V={V} {interp}] ratio {r:.3g}")
    assert r <= 1e-5


# ------------------------------------------------------------------ interfaces and determinism
def test_func_jvp_and_forward_ad_agree_and_repeat_bit_equal():
    H, W = 128, 256
    field, u, v, _ = _noise(H, W, 2, 3, True, seed=14)
    geo = _geo(H, W, True)
    t = _tangents(field, u, v, 9)
    a = _jvp(geo, "bicubic", "fast", True, (field, u, v), t)
    b = _jvp(geo, "bicubic", "fast", True, (field, u, v), t)
    with fwAD.dual_level():
        duals = [fwAD.make_dual(p, d) for p, d in zip((field, u, v), t)]
        c = fwAD.unpack_dual(_advect(geo, "bicubic", "fast", True)(*duals)).tangent
    assert torch.equal(a, b) and torch.equal(a, c)
    assert a.abs().max() > 0


def test_bf16_primals_are_upcast():
    H, W = 128, 256
    field, u, v, _ = _noise(H, W, 2, 3, True, seed=15)
    t = _tangents(field, u, v, 10)
    geo = _geo(H, W, True)
    bf = tuple(x.to(torch.bfloat16) for x in (field, u, v))
    tb = tuple(x.to(torch.bfloat16) for x in t)
    got, names = _kernels(lambda: _jvp(geo, "bilinear", "fast", True, bf, tb))
    _assert_ran(names, TL)
    assert got.dtype == torch.float32
    assert torch.equal(got, _jvp(geo, "bilinear", "fast", True, tuple(x.float() for x in bf),
                                  tuple(x.float() for x in tb)))


# ------------------------------------------------------------------ GeoCyclic ops
def _geo_inputs(dtype=torch.float32):
    g = torch.Generator(device="cuda").manual_seed(16)
    r = lambda *s: torch.randn(*s, generator=g, device="cuda")
    return r(2, 3, 16, 32).to(dtype), r(2, 3, 16, 32).to(dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pad_and_avgpool5_tangents(dtype):
    ops = _ops()
    x, dx = _geo_inputs(dtype)
    for fn in (lambda a: ops.geocyclic_pad(a, 2), lambda a: ops.geocyclic_avgpool5(a, 2)):
        y, ty = torch.func.jvp(fn, (x,), (dx,))
        assert torch.equal(ty, fn(dx)) and ty.dtype == y.dtype
        if dtype == torch.float32:                 # dot-product test against the existing backward
            g = torch.randn_like(y)
            xr = x.clone().requires_grad_(True)
            (gx,) = torch.autograd.grad(fn(xr), xr, g)
            r = _dot_ratio(ty, g, [dx], [gx])
            print(f"[dot geocyclic] ratio {r:.3g}")
            assert r <= 1e-5


@pytest.mark.parametrize("k", [3, 5, 7])
def test_dwconv_tangent(k):
    ops = _ops()
    x, dx = _geo_inputs()
    gen = torch.Generator(device="cuda").manual_seed(k)
    w, dw = [torch.randn(3, 1, k, k, generator=gen, device="cuda") for _ in range(2)]
    b, db = [torch.randn(3, generator=gen, device="cuda") for _ in range(2)]
    y, ty = torch.func.jvp(ops.geocyclic_dwconv, (x, w, b), (dx, dw, db))
    want = ops.geocyclic_dwconv(dx, w) + ops.geocyclic_dwconv(x, dw) + db.view(1, -1, 1, 1)
    assert torch.equal(ty, want)
    _, t_x = torch.func.jvp(lambda a: ops.geocyclic_dwconv(a, w, b), (x,), (dx,))
    assert torch.equal(t_x, ops.geocyclic_dwconv(dx, w))
    g = torch.randn_like(y)
    prim = [t.clone().requires_grad_(True) for t in (x, w, b)]
    grads = torch.autograd.grad(ops.geocyclic_dwconv(*prim), prim, g)
    r = _dot_ratio(ty, g, [dx, dw, db], grads)
    print(f"[dot dwconv k={k}] ratio {r:.3g}")
    assert r <= 1e-5


# ------------------------------------------------------------------ whole model
def _model_dot(fn, primals, tangents, names=None):
    out, jt = torch.func.jvp(fn, primals, tangents)
    assert jt.abs().max() > 0
    g = torch.randn_like(out)
    prim = [p.detach().clone().requires_grad_(True) for p in primals]
    grads = torch.autograd.grad(fn(*prim), prim, g)
    return _dot_ratio(jt, g, tangents, grads)


def test_neural_semi_lagrangian_jvp():
    """Through NeuralSemiLagrangian the tangent of the advection was zero before forward-mode AD was supported: its
    down / up projections are linear, so the whole tangent was zero and this test failed."""
    import paradis_model_b200 as pkg
    H, W, hidden, nv = 32, 64, 16, 8
    lat, lon = O.make_grids(H, W, True)
    cfg = A.default_cfg(latent=hidden, vels=nv, interp="bicubic")
    torch.manual_seed(0)
    m = pkg.NeuralSemiLagrangian(cfg, hidden, (H, W), num_vels=nv, lat_grid=lat, lon_grid=lon,
                                 interpolation="bicubic").cuda()
    g = torch.Generator(device="cuda").manual_seed(17)
    r = lambda *s: torch.randn(*s, generator=g, device="cuda")
    h, u, v = r(2, hidden, H, W), r(2, nv, H, W) * 3, r(2, nv, H, W) * 3
    prim, tang = (h, u, v), (r(2, hidden, H, W), r(2, nv, H, W), r(2, nv, H, W))
    got, names = _kernels(lambda: torch.func.jvp(lambda a, b, c: m(a, b, c, 0.05), prim, tang))
    _assert_ran(names, TL)
    ratio = _model_dot(lambda a, b, c: m(a, b, c, 0.05), prim, tang)
    print(f"[dot NeuralSemiLagrangian] ratio {ratio:.3g}")
    assert ratio <= 1e-5


def test_assembly_jvp_inputs_and_parameters():
    H, W = 32, 64
    cfg = A.default_cfg(interp="bicubic", checkpointing=False)
    lat, lon = O.make_grids(H, W, False)
    torch.manual_seed(0)
    model = A.Assembly(A.FakeDataModule, cfg, lat, lon, dropin=True).cuda()
    g = torch.Generator(device="cuda").manual_seed(18)
    x = torch.randn(2, 22, H, W, generator=g, device="cuda")
    dx = torch.randn(2, 22, H, W, generator=g, device="cuda")
    (ratio_x) = _model_dot(model, (x,), (dx,))
    print(f"[dot Assembly inputs] ratio {ratio_x:.3g}")
    assert ratio_x <= 1e-4
    params = {k: p.detach() for k, p in model.named_parameters()}
    keys = list(params)
    tang = [torch.randn(params[k].shape, generator=g, device="cuda") for k in keys]
    fn = lambda *ps: torch.func.functional_call(model, dict(zip(keys, ps)), (x,))
    _, names = _kernels(lambda: torch.func.jvp(fn, tuple(params[k] for k in keys), tuple(tang)))
    _assert_ran(names, TL)
    ratio_p = _model_dot(fn, tuple(params[k] for k in keys), tuple(tang))
    print(f"[dot Assembly parameters] ratio {ratio_p:.3g}")
    assert ratio_p <= 1e-4


# ------------------------------------------------------------------ loud failures
def test_unsupported_forward_mode_uses_raise():
    ops = _ops()
    H, W = 32, 64
    field, u, v, go = _noise(H, W, 1, 2, True, seed=19)
    geo = _geo(H, W, True)
    df, _, _ = _tangents(field, u, v, 11)
    fn = lambda f: ops.sl_advect(f, u, v, geo, DT)
    with pytest.raises(NotImplementedError, match="forward-over-reverse"):
        torch.func.jvp(lambda f: torch.func.vjp(fn, f)[1](go)[0], (field,), (df,))
    with pytest.raises(NotImplementedError, match="forward-over-reverse"):
        with fwAD.dual_level():
            f = fwAD.make_dual(field.clone().requires_grad_(True), df)
            torch.autograd.grad(fn(f), f, go, create_graph=True)
    with pytest.raises(NotImplementedError, match="vmap"):
        torch.func.jacfwd(lambda f: ops.sl_advect(f, u[:, :1, :8], v[:, :1, :8], _geo(8, W, True), DT))(
            field[:, :1, :8].contiguous())
    x, dx = _geo_inputs()
    with pytest.raises(NotImplementedError, match="vmap"):
        torch.func.jacfwd(lambda a: ops.geocyclic_pad(a, 1))(x[:1, :1, :4, :8].contiguous())
    band = geo.band((8, 16), (8, 16), (0, H))
    with pytest.raises(NotImplementedError, match="latitude-band"):
        torch.func.jvp(lambda a: ops.sl_advect(field, a, v[:, :, 8:24], band, DT), (u[:, :, 8:24],),
                       (torch.ones_like(u[:, :, 8:24]),))


# ------------------------------------------------------------------ compile
def test_compiled_training_step_has_no_graph_break():
    """The compiled training step of test_model_configs (fullgraph, bf16 autocast, checkpointing) still compiles as
    one graph: the tangent check of the public wrappers traces without a break."""
    import test_model_configs
    test_model_configs.test_config4_training_step_compile_autocast_checkpoint()
    H, W = 128, 256
    lat, lon = O.make_grids(H, W, False)
    model = A.Assembly(A.FakeDataModule, A.default_cfg(interp="bicubic", checkpointing=True), lat, lon,
                       dropin=True).cuda()
    x = torch.randn(2, 22, H, W, device="cuda")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        ex = torch._dynamo.explain(model)(x)
    print(f"[explain] graphs {ex.graph_count}, graph breaks {ex.graph_break_count}")
    assert ex.graph_break_count == 0
