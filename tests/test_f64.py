"""float64 path of the advection and GeoCyclic ops (include/paradis_sl_f64.h), on the GPU.

Each case checks by torch.profiler kernel name that the fp64 kernels ran and that no fp32 / bf16 kernel of these ops
and no dtype copy (``aten::_to_copy``) did.  References:
  - the oracle's op replay of the reference (oracle/sl_oracle.py) run by torch-CUDA in float64 on the same GPU: the
    departure coordinates and every intermediate bit for bit, out and the gradients to 1e-12 of the maximum;
  - the same replay on the CPU (1e-10 on smooth fields), F.conv2d / AvgPool2d after the oracle's padding (1e-13);
  - torch.autograd.gradcheck with check_forward_ad, and dot-product tests of the jvp against the backward.
"""
import re

import pytest
import torch
import torch.nn.functional as F

import paradis_model_b200 as P
from paradis_model_b200 import ops
from paradis_model_b200.blocks import PhysicalDownsample, SepConv
from oracle import paradis_assembly as A
from oracle import sl_oracle as O

pytestmark = pytest.mark.gpu
DT = 21600 * 7.29212e-5 / 8
D = torch.float64
_OUR_KERNEL = re.compile(r"(sl_\w*|pole_\w*|geocyclic_\w*|geo_\w*|departure_coords\w*)_kernel")


def relmax(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _ran(fn):
    """Run fn under the profiler; assert that only fp64 kernels of the package ran and no dtype copy was made."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    ours = {n for n in names if _OUR_KERNEL.search(n) and "plane_reach_kernel" not in n}
    assert ours and all("f64" in n for n in ours), sorted(ours)
    assert "aten::_to_copy" not in names
    return res, ours


def _grids(H, W, poles=True):
    lat, lon = O.make_grids(H, W, poles, D)
    return lat.cuda(), lon.cuda()


def _case(H, W, B, V, poles=True, cells=3.0, noise=False, seed=0):
    lat, lon = _grids(H, W, poles)
    g = torch.Generator(device="cpu").manual_seed(seed)
    if noise:
        field = torch.randn(B, V, H, W, generator=g, dtype=D)
        u, v = [torch.randn(B, V, H, W, generator=g, dtype=D) * (cells * 0.5 * 3.14159 / H / DT) for _ in range(2)]
    else:
        field = O.smooth_field(lat.cpu(), lon.cpu(), B, V, seed=seed).to(D)
        u, v = [t.to(D) for t in O.smooth_velocity(lat.cpu(), lon.cpu(), B, V, cells, DT, seed=seed + 1)]
    go = torch.randn(B, V, H, W, generator=g, dtype=D)
    return lat, lon, field.cuda(), u.cuda(), v.cuda(), go.cuda()


# ---------------------------------------------------------------------------------------------------------------
# GeoCyclic ops
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", [1, 2, 3])
@pytest.mark.parametrize("H,W", [(6, 8), (33, 64), (721, 1440)])
def test_pad_exact(p, H, W):
    g = torch.Generator(device="cpu").manual_seed(p)
    x = torch.randn(2, 3, H, W, generator=g, dtype=D).cuda().requires_grad_(True)
    gy = torch.randint(-1000, 1000, (2, 3, H + 2 * p, W + 2 * p), generator=g).to(D).cuda()   # exact sums

    def run():
        y = P.GeoCyclicPadding(p)(x)
        y.backward(gy)
        return y

    y, _ = _ran(run)
    assert y.dtype == D and torch.equal(y, O.geocyclic_pad(x.detach(), p))
    assert torch.equal(x.grad, O.geocyclic_pad_adjoint(gy, p))


@pytest.mark.parametrize("k", [3, 5, 7])
def test_dwconv_against_conv2d(k):
    g = torch.Generator(device="cpu").manual_seed(k)
    x = torch.randn(2, 3, 33, 64, generator=g, dtype=D).cuda()
    w = torch.randn(3, 1, k, k, generator=g, dtype=D).cuda()
    b = torch.randn(3, generator=g, dtype=D).cuda()
    gy = torch.randn(2, 3, 33, 64, generator=g, dtype=D).cuda()
    ref = [t.clone().requires_grad_(True) for t in (x, w, b)]
    y_ref = O.geocyclic_depthwise(*ref)
    y_ref.backward(gy)
    got = [t.clone().requires_grad_(True) for t in (x, w, b)]

    def run():
        y = ops.geocyclic_dwconv(*got)
        y.backward(gy)
        return y

    y, _ = _ran(run)
    assert y.dtype == D and relmax(y, y_ref) <= 1e-13
    for a, r in zip(got, ref):
        assert a.grad.dtype == D and relmax(a.grad, r.grad) <= 1e-13


@pytest.mark.parametrize("stride", [1, 2, 3, 4])
@pytest.mark.parametrize("H,W", [(33, 64), (65, 128)])
def test_avgpool5_against_downsample(stride, H, W):
    g = torch.Generator(device="cpu").manual_seed(stride)
    x = torch.randn(2, 3, H, W, generator=g, dtype=D).cuda()
    ref_x, x = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    y_ref = A.Downsample(stride, A.OraclePadding)(ref_x)
    gy = torch.randn(y_ref.shape, generator=g, dtype=D).cuda()
    y_ref.backward(gy)

    def run():
        y = PhysicalDownsample(stride)(x)
        y.backward(gy)
        return y

    y, _ = _ran(run)
    assert y.dtype == D and relmax(y, y_ref) <= 1e-13 and relmax(x.grad, ref_x.grad) <= 1e-13


def test_sepconv_module_after_double():
    m = SepConv(3, 4, (33, 64), kernel_size=5).cuda().double()
    x = torch.randn(2, 3, 33, 64, dtype=D, device="cuda")
    ref = F.conv2d(O.geocyclic_depthwise(x, m.depthwise.weight), m.pointwise.weight, m.pointwise.bias)
    assert relmax(m(x), ref) <= 1e-13


# ---------------------------------------------------------------------------------------------------------------
# departure coordinates: bit for bit against the oracle's op replay in fp64 on the same GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("H,W", [(128, 256), (721, 1440)])
def test_departure_coords_bit_identical(interp, H, W):
    lat, lon, field, u, v, go = _case(H, W, 1, 2, cells=4.0, seed=3)
    geo = P.SLGeometry.from_grids(lat, lon)
    c, _ = _ran(lambda: ops.departure_coords(u, v, geo, DT, interp))
    c = c[0]                                    # [V, 11, H, W]
    # the oracle's op replay (departure_latlon, departure_pixels, sampler_coords), intermediates kept
    G = O.Geometry(lat, lon)
    lon_r, lat_r = -u[0] * DT, -v[0] * DT
    sa, ca, sb, cb = torch.sin(lat_r), torch.cos(lat_r), torch.sin(lon_r), torch.cos(lon_r)
    sp, cp = torch.sin(G.lat), torch.cos(G.lat)
    s = sa * cp + ca * cb * sp
    lat_d = torch.arcsin(torch.clamp(s, -1 + 1e-7, 1 - 1e-7))
    num = ca * sb
    den = ca * cb * cp - sa * sp
    lon_d = torch.remainder(G.lon + torch.atan2(num, den) + 2 * torch.pi, 2 * torch.pi)
    px = (lon_d - G.min_lon) / G.d_lon * (G.Wf - 1.0)
    py = (lat_d - G.min_lat) / G.d_lat * (G.Hf - 1.0)
    _, _, ix, iy = O.sampler_coords(px, py, H, W, O.INTERP_PAD[interp])
    want = [ix, iy, sa, ca, sb, cb, s, num, den, lat_d, lon_d]
    for k, w in enumerate(want):
        w = w.reshape(c[:, k].shape)
        assert torch.equal(c[:, k], w), (k, int((c[:, k] != w).sum()))


# ---------------------------------------------------------------------------------------------------------------
# out, grad_field, grad_u, grad_v against the oracle in fp64
# ---------------------------------------------------------------------------------------------------------------
CASES = [  # H, W, B, V, poles, cells, noise
    (33, 64, 2, 3, True, 3.0, False),
    (32, 64, 2, 3, False, 3.0, False),
    (33, 64, 1, 3, True, 14.0, False),        # cross-pole departures
    (24, 1000, 1, 2, True, 3.0, False),       # ragged widths
    (24, 904, 1, 2, False, 3.0, True),
    (5, 6, 2, 2, True, 1.0, False),
    (12, 16, 2, 3, True, 2.0, True),          # white noise
]


def _fwd_bwd(field, u, v, go, geo, interp, pole_fix, strided=False):
    f = field.clone().requires_grad_(True)
    if strided:          # u, v as batch-strided views of one [B, 2V, H, W] tensor (model/paradis.py:235-237)
        uv = torch.cat([u, v], 1).requires_grad_(True)
        V = u.shape[1]
        uu, vv = uv[:, :V], uv[:, V:]
    else:
        uu, vv = u.clone().requires_grad_(True), v.clone().requires_grad_(True)
    out = P.sl_advect(f, uu, vv, geo, DT, interp, pole_fix)
    out.backward(go)
    P.check_status()
    if strided:
        return out.detach(), f.grad, uv.grad[:, :V], uv.grad[:, V:]
    return out.detach(), f.grad, uu.grad, vv.grad


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("case", CASES)
def test_advect_against_oracle_on_gpu(case, interp, pole_fix):
    H, W, B, V, poles, cells, noise = case
    lat, lon, field, u, v, go = _case(H, W, B, V, poles, cells, noise, seed=H + W)
    geo = P.SLGeometry.from_grids(lat, lon)
    ref = O.sl_advect_fwd_bwd(field, u, v, lat, lon, DT, go, interp, pole_fix)
    got, _ = _ran(lambda: _fwd_bwd(field, u, v, go, geo, interp, pole_fix))
    for name, a, r in zip(("out", "grad_field", "grad_u", "grad_v"), got, ref):
        assert a.dtype == D and relmax(a, r) <= 1e-12, (name, relmax(a, r))
    strided = _fwd_bwd(field, u, v, go, geo, interp, pole_fix, strided=True)
    for a, b in zip(strided, got):
        assert torch.equal(a, b)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_advect_against_cpu_oracle_smooth(interp):
    lat, lon, field, u, v, go = _case(33, 64, 2, 2, True, 3.0, seed=5)
    ref = O.sl_advect_fwd_bwd(*[t.cpu() for t in (field, u, v, lat, lon)], DT, go.cpu(), interp)
    got = _fwd_bwd(field, u, v, go, P.SLGeometry.from_grids(lat, lon), interp, True)
    for a, r in zip(got, ref):
        assert relmax(a.cpu(), r) <= 1e-10


# ---------------------------------------------------------------------------------------------------------------
# gradcheck (reverse and forward mode), dot-product test, determinism, dtypes, contract errors
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
@pytest.mark.parametrize("pole_fix", [True, False])
@pytest.mark.parametrize("H,W", [(6, 8), (9, 16)])
def test_gradcheck_sl_advect(interp, pole_fix, H, W):
    lat, lon, field, u, v, go = _case(H, W, 1, 2, True, 0.7, seed=H)
    geo = P.SLGeometry.from_grids(lat, lon)
    fn = lambda f, uu, vv: P.sl_advect(f, uu, vv, geo, DT, interp, pole_fix)
    args = [t.clone().requires_grad_(True) for t in (field, u, v)]
    assert torch.autograd.gradcheck(fn, args, check_forward_ad=True, eps=1e-7, atol=1e-7, rtol=1e-6)


def test_gradcheck_geocyclic_ops():
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.randn(1, 2, 9, 16, generator=g, dtype=D).cuda().requires_grad_(True)
    w = torch.randn(2, 1, 3, 3, generator=g, dtype=D).cuda().requires_grad_(True)
    b = torch.randn(2, generator=g, dtype=D).cuda().requires_grad_(True)
    kw = dict(check_forward_ad=True)
    assert torch.autograd.gradcheck(lambda t: ops.geocyclic_pad(t, 2), [x], **kw)
    assert torch.autograd.gradcheck(ops.geocyclic_dwconv, [x, w, b], **kw)
    assert torch.autograd.gradcheck(lambda t: ops.geocyclic_avgpool5(t, 2), [x], **kw)


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_dot_product_jvp_vs_backward(interp):
    lat, lon, field, u, v, go = _case(33, 64, 2, 3, True, 3.0, seed=9)
    geo = P.SLGeometry.from_grids(lat, lon)
    g = torch.Generator(device="cpu").manual_seed(2)
    tan = [torch.randn(field.shape, generator=g, dtype=D).cuda() for _ in range(3)]
    fn = lambda f, uu, vv: P.sl_advect(f, uu, vv, geo, DT, interp)
    (out, jt), _ = _ran(lambda: torch.func.jvp(fn, (field, u, v), tuple(tan)))
    assert jt.dtype == D
    prim = [t.clone().requires_grad_(True) for t in (field, u, v)]
    jtg = torch.autograd.grad(fn(*prim), prim, go)
    lhs = (jt * go).sum()
    terms = [(a * b) for a, b in zip(tan, jtg)]
    rhs = sum(t.sum() for t in terms)
    scale = (jt * go).abs().sum() + sum(t.abs().sum() for t in terms)
    assert float((lhs - rhs).abs() / scale) <= 1e-13


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_backward_bit_equal_across_runs(interp):
    lat, lon, field, u, v, go = _case(128, 256, 1, 4, True, 8.0, True, seed=4)
    geo = P.SLGeometry.from_grids(lat, lon)
    a = _fwd_bwd(field, u, v, go, geo, interp, True)
    b = _fwd_bwd(field, u, v, go, geo, interp, True)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_mixed_dtypes_promote_to_float64():
    lat, lon, field, u, v, go = _case(33, 64, 1, 2, True, 3.0, seed=2)
    geo = P.SLGeometry.from_grids(lat, lon)
    uf, vf = u.float(), v.float()
    ref = _fwd_bwd(field, uf.double(), vf.double(), go, geo, "bicubic", True)
    f, uu, vv = field.clone().requires_grad_(True), uf.clone().requires_grad_(True), vf.clone().requires_grad_(True)
    out = P.sl_advect(f, uu, vv, geo, DT, "bicubic")
    out.backward(go)
    assert out.dtype == D and torch.equal(out, ref[0]) and torch.equal(f.grad, ref[1])
    assert uu.grad.dtype == torch.float32 and torch.equal(uu.grad, ref[2].float())
    c = ops.departure_coords(uf, v, geo, DT)
    assert c.dtype == D and torch.equal(c, ops.departure_coords(uf.double(), v, geo, DT))


def test_displacement_over_126_rows_raises():
    lat, lon, field, u, v, go = _case(400, 32, 1, 1, True, 0.0, seed=1)
    v = torch.full_like(v, -140 * 3.14159 / 399 / DT)            # 140 rows northward
    f, uu, vv = [t.clone().requires_grad_(True) for t in (field, torch.zeros_like(u), v)]
    P.sl_advect(f, uu, vv, P.SLGeometry.from_grids(lat, lon), DT, "bilinear", False).backward(go)
    with pytest.raises(RuntimeError, match="DISPLACEMENT"):
        P.check_status()


def test_latitude_band_raises():
    lat, lon, field, u, v, go = _case(32, 64, 1, 1, True, 1.0)
    geo = P.SLGeometry.from_grids(lat, lon).band((8, 8), (4, 16), (0, 32))
    with pytest.raises(RuntimeError, match="full mesh only"):
        P.sl_advect(field, u[:, :, 4:20], v[:, :, 4:20], geo, DT)


def _nsl(interp="bicubic"):
    lat, lon = _grids(32, 64)
    torch.manual_seed(0)
    return P.NeuralSemiLagrangian(A.default_cfg(interp=interp), 6, (32, 64), 4, lat, lon, interp).cuda().double()


def test_compiled_neural_semi_lagrangian_matches_eager():
    m = _nsl()
    g = torch.Generator(device="cpu").manual_seed(0)
    x = torch.randn(2, 6, 32, 64, generator=g, dtype=D).cuda()
    u, v = [torch.randn(2, 4, 32, 64, generator=g, dtype=D).cuda() * 0.01 for _ in range(2)]   # ~2 cells per step
    w = torch.randn(2, 6, 32, 64, generator=g, dtype=D).cuda()

    def step(fn):
        m.zero_grad()
        xx = x.clone().requires_grad_(True)
        y = fn(xx, u, v, DT)
        (y * w).sum().backward()
        return [y.detach(), xx.grad] + [p.grad.clone() for p in m.parameters()]

    eager = step(m)
    compiled = step(torch.compile(m, fullgraph=True))
    assert eager[0].dtype == D
    for a, b in zip(compiled, eager):
        assert relmax(a, b) <= 1e-13


@pytest.mark.parametrize("interp", ["bilinear", "bicubic"])
def test_double_assembly_against_reference_ops(interp):
    cfg = A.default_cfg(interp=interp)
    lat, lon = O.make_grids(32, 64, True)
    torch.manual_seed(0)
    ref = A.Assembly(A.FakeDataModule, cfg, lat, lon, dropin=False).cuda().double()
    new = A.Assembly(A.FakeDataModule, cfg, lat, lon, dropin=True).cuda().double()
    new.load_state_dict(ref.state_dict(), strict=True)
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(2, 22, 32, 64, generator=g, dtype=D).cuda()
    w = torch.randn(2, 7, 32, 64, generator=g, dtype=D).cuda()
    y_ref, y = ref(x), new(x)
    assert y.dtype == D and relmax(y, y_ref) <= 1e-11
    (y_ref * w).sum().backward()
    (y * w).sum().backward()
    for (n1, p1), (n2, p2) in zip(ref.named_parameters(), new.named_parameters()):
        assert n1 == n2 and relmax(p2.grad, p1.grad) <= 1e-9, (n1, relmax(p2.grad, p1.grad))
    # forward mode through the whole drop-in model: <J t, w> = <t, J^T w>
    t = torch.randn(x.shape, generator=g, dtype=D).cuda()
    _, jt = torch.func.jvp(lambda z: new(z), (x,), (t,))
    xx = x.clone().requires_grad_(True)
    (gx,) = torch.autograd.grad(new(xx), xx, w)
    lhs, rhs = (jt * w).sum(), (t * gx).sum()
    assert float((lhs - rhs).abs() / ((jt * w).abs().sum() + (t * gx).abs().sum())) <= 1e-13
