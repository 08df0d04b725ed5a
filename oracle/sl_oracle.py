"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the semi-Lagrangian advection path.

Two independent restatements of the reference algorithm live here:

* :func:`sl_advect` replays the reference's fp32 operation order
  (model/advection.py:129-169) with plain torch ops and hands the sampling to
  ``torch.nn.functional.grid_sample`` exactly like the reference call site
  (model/advection.py:161-167).  Gradients come from autograd.  On the same
  device it is bit-identical to the reference module (pinned by
  tests/test_oracle_vs_reference.py and by the fixtures in tests/golden/).
  This is also the "port" that bench.py times as the CPU baseline.

* :func:`sl_advect_explicit` is the closed form the CUDA kernels implement:
  explicit taps through the GeoCyclic index map, explicit Jacobian of the
  rotated-pole transform and an explicit adjoint scatter.  No autograd, no
  grid_sample.  It is checked against :func:`sl_advect` in fp64.

The arithmetic of ``grid_sample`` itself is a third-party dependency of the
reference (PyTorch, unpinned ``torch>=2.0.0`` in requirements.txt:2; de-facto
pin = torch 2.11.0 of this image).  Its published algorithm
(ATen/native/GridSampler.h:27-36, 205-297; ATen/native/UpSample.h:398-423) is
restated in :func:`_cubic_weights` / :func:`sl_advect_explicit`.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

INTERP_PAD = {"bilinear": 1, "bicubic": 2}


# --------------------------------------------------------------------------
# GeoCyclic padding (reference: model/padding.py:11-39)
# --------------------------------------------------------------------------
def geocyclic_source_index(H: int, W: int, p: int) -> tuple[np.ndarray, np.ndarray]:
    """Integer source map of the padded plane.

    Returns ``(src_row[Hp, Wp], src_col[Hp, Wp])`` such that
    ``padded[R, C] == x[src_row[R, C], src_col[R, C]]``.

    model/padding.py:26-31: the cap rows are rows ``1..p`` (resp.
    ``H-1-p..H-2``) rolled by ``W/2`` and flipped, i.e. a reflection about the
    first (last) row that *excludes* that row, shifted by 180 degrees.
    model/padding.py:35-37: longitude is periodic.
    """
    if W % 2:
        raise AssertionError("Number of longitude points must be even")
    Hp, Wp = H + 2 * p, W + 2 * p
    i = np.arange(Hp, dtype=np.int64)[:, None] - p
    j = np.arange(Wp, dtype=np.int64)[None, :] - p
    north = i < 0
    south = i >= H
    row = np.where(north, -i, np.where(south, 2 * (H - 1) - i, i))
    shift = np.where(north | south, W // 2, 0)
    col = np.mod(j - shift, W)
    return np.broadcast_to(row, (Hp, Wp)).copy(), col.astype(np.int64)


def geocyclic_pad(x: torch.Tensor, p: int) -> torch.Tensor:
    """Gather-based restatement of ``GeoCyclicPadding(p)(x)``."""
    if p == 0:
        return x
    assert x.dim() == 4, "Input must be 4-dimensional [batch, channels, lat, lon]"
    H, W = x.shape[-2:]
    row, col = geocyclic_source_index(H, W, p)
    row_t = torch.from_numpy(row).to(x.device)
    col_t = torch.from_numpy(col).to(x.device)
    return x[:, :, row_t, col_t]


def geocyclic_pad_adjoint(g: torch.Tensor, p: int) -> torch.Tensor:
    """Adjoint of :func:`geocyclic_pad`: fold the pads back onto their sources."""
    if p == 0:
        return g
    Hp, Wp = g.shape[-2:]
    H, W = Hp - 2 * p, Wp - 2 * p
    row, col = geocyclic_source_index(H, W, p)
    flat = torch.from_numpy(row * W + col).reshape(-1).to(g.device)
    out = torch.zeros(g.shape[:2] + (H * W,), dtype=g.dtype, device=g.device)
    out.index_add_(2, flat, g.reshape(g.shape[0], g.shape[1], -1))
    return out.reshape(g.shape[0], g.shape[1], H, W)


def geocyclic_depthwise(x: torch.Tensor, weight: torch.Tensor, bias=None) -> torch.Tensor:
    """First two lines of SepConv.forward (model/blocks.py:112-114): GeoCyclic pad by (k-1)//2, then the
    depthwise k x k convolution (groups = channels, no conv padding)."""
    k = weight.shape[-1]
    return F.conv2d(geocyclic_pad(x, (k - 1) // 2), weight, bias, groups=x.shape[1])


# --------------------------------------------------------------------------
# Pole continuity (reference: model/advection.py:100-114)
# --------------------------------------------------------------------------
def pole_mean(x: torch.Tensor) -> torch.Tensor:
    """Rows 0 and H-1 are replaced by their zonal mean (unconditionally)."""
    y = x.clone()
    y[:, :, 0, :] = x[:, :, 0:1, :].mean(dim=3, keepdim=True).squeeze(-1)
    y[:, :, -1, :] = x[:, :, -1:, :].mean(dim=3, keepdim=True).squeeze(-1)
    return y


# --------------------------------------------------------------------------
# Geometry (reference: model/advection.py:56-72)
# --------------------------------------------------------------------------
class Geometry:
    """0-dim tensors in the dtype of the grids, as the reference registers them."""

    def __init__(self, lat_grid: torch.Tensor, lon_grid: torch.Tensor):
        H, W = lat_grid.shape
        self.H, self.W = H, W
        self.lat = lat_grid.reshape(1, 1, H, W)
        self.lon = lon_grid.reshape(1, 1, H, W)
        self.Hf = torch.tensor(float(H), dtype=lat_grid.dtype, device=lat_grid.device)
        self.Wf = torch.tensor(float(W), dtype=lat_grid.dtype, device=lat_grid.device)
        self.min_lat = lat_grid.min()
        self.min_lon = lon_grid.min()
        self.d_lat = lat_grid.max() - self.min_lat
        self.d_lon = lon_grid.max() - self.min_lon


def make_grids(H: int, W: int, poles: bool, dtype=torch.float32):
    """Synthetic ERA5-style grids (data/era5_dataset.py:178-182: fp64 deg2rad, then cast).

    ``poles=True``  : lat = linspace(-90, 90, H)            (0.25 deg ERA5, H = 721)
    ``poles=False`` : lat = -90 + 180/H * (i + 1/2)         (WB2 pole-less grids)
    lon = 360/W * j in both cases.
    """
    if poles:
        lat = np.linspace(-90.0, 90.0, H)
    else:
        lat = -90.0 + 180.0 / H * (np.arange(H) + 0.5)
    lon = 360.0 / W * np.arange(W)
    lat_g, lon_g = np.meshgrid(np.deg2rad(lat), np.deg2rad(lon), indexing="ij")
    return (torch.from_numpy(lat_g).to(dtype), torch.from_numpy(lon_g).to(dtype))


# --------------------------------------------------------------------------
# Departure points, reference operation order
# --------------------------------------------------------------------------
def departure_latlon(u, v, geo: Geometry, dt: float):
    """model/advection.py:131-136 + 74-98 (rotated pole -> geographic)."""
    lon_r = -u * dt
    lat_r = -v * dt
    s_lat_r, c_lat_r = torch.sin(lat_r), torch.cos(lat_r)
    s_lon_r, c_lon_r = torch.sin(lon_r), torch.cos(lon_r)
    s_lat_p, c_lat_p = torch.sin(geo.lat), torch.cos(geo.lat)

    s = s_lat_r * c_lat_p + c_lat_r * c_lon_r * s_lat_p
    lat_dep = torch.arcsin(torch.clamp(s, -1 + 1e-7, 1 - 1e-7))
    num = c_lat_r * s_lon_r
    den = c_lat_r * c_lon_r * c_lat_p - s_lat_r * s_lat_p
    lon_dep = geo.lon + torch.atan2(num, den)
    lon_dep = torch.remainder(lon_dep + 2 * torch.pi, 2 * torch.pi)
    return lat_dep, lon_dep


def departure_pixels(u, v, geo: Geometry, dt: float):
    """model/advection.py:138-139: unpadded pixel coordinates of the departure point."""
    lat_dep, lon_dep = departure_latlon(u, v, geo, dt)
    pix_x = (lon_dep - geo.min_lon) / geo.d_lon * (geo.Wf - 1.0)
    pix_y = (lat_dep - geo.min_lat) / geo.d_lat * (geo.Hf - 1.0)
    return pix_x, pix_y


def sampler_coords(pix_x, pix_y, H: int, W: int, p: int):
    """model/advection.py:143-150 followed by ATen's un-normalisation
    (GridSampler.h:27-36, align_corners=True): the coordinates the sampler
    actually floors.  Same fp32 round trip as reference + ATen."""
    Hp, Wp = H + 2 * p, W + 2 * p
    gx = 2.0 * ((pix_x + p) / float(Wp - 1)) - 1.0
    gy = 2.0 * ((pix_y + p) / float(Hp - 1)) - 1.0
    ix = ((gx + 1) / 2) * (Wp - 1)
    iy = ((gy + 1) / 2) * (Hp - 1)
    return gx, gy, ix, iy


def sl_advect(field, u, v, lat_grid, lon_grid, dt: float, interpolation: str = "bilinear",
              pole_fix: bool = True):
    """Operator core: reference model/advection.py:129-169 (projections excluded).

    field, u, v: [B, V, H, W]; returns [B, V, H, W].  Differentiable (autograd).
    """
    B, V, H, W = field.shape
    p = INTERP_PAD[interpolation]
    geo = Geometry(lat_grid, lon_grid)
    src = pole_mean(field) if pole_fix else field
    pix_x, pix_y = departure_pixels(u, v, geo, dt)
    padded = geocyclic_pad(src, p)
    gx, gy, _, _ = sampler_coords(pix_x, pix_y, H, W, p)
    grid = torch.stack([gx.reshape(B * V, H, W), gy.reshape(B * V, H, W)], dim=-1)
    out = F.grid_sample(padded.reshape(B * V, 1, H + 2 * p, W + 2 * p), grid,
                        align_corners=True, mode=interpolation, padding_mode="zeros")
    out = out.reshape(B, V, H, W)
    return pole_mean(out) if pole_fix else out


def sl_advect_fwd_bwd(field, u, v, lat_grid, lon_grid, dt, grad_out, interpolation="bilinear",
                      pole_fix=True):
    """One forward + backward through autograd.  Returns (out, gfield, gu, gv)."""
    f = field.detach().clone().requires_grad_(True)
    uu = u.detach().clone().requires_grad_(True)
    vv = v.detach().clone().requires_grad_(True)
    out = sl_advect(f, uu, vv, lat_grid, lon_grid, dt, interpolation, pole_fix)
    out.backward(grad_out)
    return out.detach(), f.grad, uu.grad, vv.grad


# --------------------------------------------------------------------------
# Explicit closed form (what the CUDA kernels compute)
# --------------------------------------------------------------------------
_A = -0.75


def _cubic_weights(t):
    """ATen/native/UpSample.h:398-423 (A=-0.75), taps at floor-1 .. floor+2."""
    def cc1(x):
        return ((_A + 2) * x - (_A + 3)) * x * x + 1

    def cc2(x):
        return ((_A * x - 5 * _A) * x + 8 * _A) * x - 4 * _A

    return [cc2(t + 1.0), cc1(t), cc1(1.0 - t), cc2((1.0 - t) + 1.0)]


def _cubic_weights_grad(t):
    """d(weight)/dt.  ATen/native/GridSampler.h:280-297 tabulates the NEGATIVE of
    these (its caller subtracts: ``gix -= value * coeff_grad * ...``)."""
    x0, x1, x2, x3 = -1 - t, -t, 1 - t, 2 - t
    return [-((-3 * _A * x0 - 10 * _A) * x0 - 8 * _A),
            -((-3 * (_A + 2) * x1 - 2 * (_A + 3)) * x1),
            -((3 * (_A + 2) * x2 - 2 * (_A + 3)) * x2),
            -((3 * _A * x3 - 10 * _A) * x3 + 8 * _A)]


def _stencil(ix, iy, interpolation):
    """Per-axis tap offsets, weights and weight derivatives."""
    x0, y0 = torch.floor(ix), torch.floor(iy)
    tx, ty = ix - x0, iy - y0
    if interpolation == "bilinear":
        offs = [0, 1]
        wx, wy = [1 - tx, tx], [1 - ty, ty]
        one = torch.ones_like(tx)
        dwx, dwy = [-one, one], [-one, one]
    else:
        offs = [-1, 0, 1, 2]
        wx, wy = _cubic_weights(tx), _cubic_weights(ty)
        dwx, dwy = _cubic_weights_grad(tx), _cubic_weights_grad(ty)
    return x0.long(), y0.long(), offs, wx, wy, dwx, dwy


def sl_advect_explicit(field, u, v, lat_grid, lon_grid, dt, grad_out=None,
                       interpolation="bilinear", pole_fix=True):
    """Closed-form forward and (if ``grad_out`` is given) backward.

    Forward : out = sum_taps w * field[src(R, C)]                      (SURVEY 8a)
    Backward: grad_u, grad_v through the Jacobian of the rotated-pole map,
              grad_field by the adjoint scatter through the GeoCyclic map.
    The departure coordinates are computed in the dtype of the inputs (use fp64 for formula
    checks); the interpolation and its adjoint are :func:`sl_advect_at_coords` at them.
    """
    H, W = field.shape[-2:]
    p = INTERP_PAD[interpolation]
    geo = Geometry(lat_grid, lon_grid)

    lon_r, lat_r = -u * dt, -v * dt
    sa, ca = torch.sin(lat_r), torch.cos(lat_r)          # phi'
    sb, cb = torch.sin(lon_r), torch.cos(lon_r)          # lambda'
    sp, cp = torch.sin(geo.lat), torch.cos(geo.lat)      # arrival point
    s = sa * cp + ca * cb * sp
    lo, hi = -1 + 1e-7, 1 - 1e-7
    s_c = torch.clamp(s, lo, hi)
    num = ca * sb
    den = ca * cb * cp - sa * sp
    lat_dep = torch.arcsin(s_c)
    lon_dep = torch.remainder(geo.lon + torch.atan2(num, den) + 2 * math.pi, 2 * math.pi)
    Ax = (geo.Wf - 1.0) / geo.d_lon
    Ay = (geo.Hf - 1.0) / geo.d_lat
    ix = (lon_dep - geo.min_lon) * Ax + p
    iy = (lat_dep - geo.min_lat) * Ay + p
    coords = torch.stack(torch.broadcast_tensors(ix, iy, sa, ca, sb, cb, s, num, den, lat_dep, lon_dep), dim=2)

    r = sl_advect_at_coords(field, grad_out, coords, sp[0, 0, :, 0], cp[0, 0, :, 0], dt, geo, interpolation,
                            pole_fix)
    if grad_out is None:
        return r.out.to(field.dtype)
    return tuple(t.to(field.dtype) for t in (r.out, r.grad_field, r.grad_u, r.grad_v))


# --------------------------------------------------------------------------
# fp64 reference at given departure coordinates, with per-point rounding bounds
# --------------------------------------------------------------------------
U32 = 2.0 ** -24          # unit roundoff of fp32
U_BF16 = 2.0 ** -8        # unit roundoff of bf16 (8-bit significand): |bf16(x) - x| <= 2^-8 |x|
K_OUT = 8                 # roundings per forward term, see sl_advect_at_coords
K_GFIELD = 4              # roundings per grad_field contribution before the sum
K_GRAD_UV = 24            # roundings along the longest chain of grad_u / grad_v


class AtCoords:
    """Result of :func:`sl_advect_at_coords`: fp64 values and per-point bounds of |kernel - value|."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def values(self):
        return self.out, self.grad_field, self.grad_u, self.grad_v

    def bounds(self):
        return self.out_bound, self.grad_field_bound, self.grad_u_bound, self.grad_v_bound


def pixel_scales(geometry, dt):
    """(Ax, Ay, dt) as the kernels hold them.

    ``geometry`` is either an ``SLGeometry`` (anything with ``scalars`` = [min_lat, d_lat, min_lon, d_lon], ``H``,
    ``W``): fp32 ``(W - 1) / d_lon``, ``(H - 1) / d_lat`` and fp32 ``dt``, like ``fill_params`` in paradis_sl.cu; or
    this module's :class:`Geometry`, whose scales are taken in the dtype of its grids (the closed form)."""
    if hasattr(geometry, "scalars"):
        _, d_lat, _, d_lon = geometry.scalars
        f = np.float32
        return (float(f(f(geometry.W) - f(1)) / f(d_lon)), float(f(f(geometry.H) - f(1)) / f(d_lat)),
                float(f(dt)))
    return (float((geometry.Wf - 1.0) / geometry.d_lon), float((geometry.Hf - 1.0) / geometry.d_lat), float(dt))


class _RunErr:
    """First-order running error of an fp32 chain: value (fp64) and error bound in units of U32.
    Each rounded operation adds |its result|; inputs carry their own bounds (Higham, ASNA 2nd ed., 3.3)."""

    def __init__(self, v, r=0.0):
        self.v, self.r = v, r

    def neg(self):                  # exact
        return _RunErr(-self.v, self.r)

    def add(self, o):
        o = o if isinstance(o, _RunErr) else _RunErr(o)
        v = self.v + o.v
        return _RunErr(v, self.r + o.r + abs(v))

    def mul(self, o):
        o = o if isinstance(o, _RunErr) else _RunErr(o)
        v = self.v * o.v
        return _RunErr(v, abs(self.v) * o.r + abs(o.v) * self.r + abs(v))

    def fma(self, o, c):            # self * o + c, one rounding
        o = o if isinstance(o, _RunErr) else _RunErr(o)
        c = c if isinstance(c, _RunErr) else _RunErr(c)
        v = self.v * o.v + c.v
        return _RunErr(v, abs(self.v) * o.r + abs(o.v) * self.r + c.r + abs(v))


class _F32:
    """The same chains evaluated in fp32, one rounding per operation.  fma: the product of two fp32 values is exact in
    fp64, so ``a * b + c`` rounds to fp64 and then to fp32 (a double rounding, at most 2^-29 ulp from the fused
    result)."""

    def __init__(self, v):
        self.v = v

    @staticmethod
    def _val(o):
        return o.v if isinstance(o, _F32) else o

    def neg(self):
        return _F32(-self.v)

    def add(self, o):
        return _F32(self.v + self._val(o))

    def mul(self, o):
        return _F32(self.v * self._val(o))

    def fma(self, o, c):
        d = lambda x: x.double() if torch.is_tensor(x) else x
        return _F32((d(self.v) * d(self._val(o)) + d(self._val(c))).float())


def _axis_weights(t, interpolation, num):
    """The kernels' fp32 axis weights and their derivatives at fraction ``t`` (``axis_weights`` in sl_device.cuh, same
    operation order), with ``num`` = :class:`_RunErr` (running-error bounds) or :class:`_F32` (fp32 values).  The
    sampler coordinates are >= p - 1/2 > 0, so ``t = ix - floor(ix)`` is exact in fp32.  Bilinear: ``1 - t`` is one
    rounding, ``t`` is exact.  The cubic weights cancel (w -> 0 at the stencil's edge while the Horner terms stay
    O(1)), so their error is not relative to the weight: it is carried as an absolute bound instead of a count in K."""
    T = num(t)
    if interpolation == "bilinear":
        return [num(1.0).add(T.neg()), T], [num(-1.0), num(1.0)]
    A = -0.75
    t1 = T.add(1.0)
    u0 = num(1.0).add(T.neg())
    u1 = u0.add(1.0)

    def outer(x):           # fma(fma(fma(A, x, -5A), x, 8A), x, -4A)
        return num(A).fma(x, -5 * A).fma(x, 8 * A).fma(x, -4 * A)

    def inner(x):           # fma(fma(A + 2, x, -(A + 3)) * x, x, 1)
        return num(A + 2).fma(x, -(A + 3)).mul(x).fma(x, 1.0)

    def d_outer(x):         # fma(fma(3A, x, -10A), x, 8A)
        return num(3 * A).fma(x, -10 * A).fma(x, 8 * A)

    def d_inner(x):         # fma(3(A + 2), x, -2(A + 3)) * x
        return num(3 * (A + 2)).fma(x, -2 * (A + 3)).mul(x)

    return ([outer(t1), inner(T), inner(u0), outer(u1)],
            [d_outer(t1), d_inner(T), d_inner(u0).neg(), d_outer(u1).neg()])


def _weight_rounding(t, interpolation):
    """Running-error bounds (units of U32) of the kernels' fp32 axis weights and derivatives (:func:`_axis_weights`)."""
    w, dw = _axis_weights(t.double(), interpolation, _RunErr)
    z = torch.zeros_like(t, dtype=torch.float64)
    return [x.r + z for x in w], [x.r + z for x in dw]


def _pole_mean_adjoint(g):
    gg = g.clone()
    gg[:, :, 0, :] = g[:, :, 0, :].mean(dim=-1, keepdim=True)
    gg[:, :, -1, :] = g[:, :, -1, :].mean(dim=-1, keepdim=True)
    return gg


def _pole_mean_sequential(x):
    """Rows 0 and H-1 replaced by their zonal mean, summed one value after the other in the dtype of ``x`` (the
    order with the largest error bound) and divided by W."""
    y = x.clone()
    for r in (0, x.shape[2] - 1):
        acc = torch.zeros_like(x[:, :, r, 0])
        for j in range(x.shape[3]):
            acc = acc + x[:, :, r, j]
        y[:, :, r, :] = (acc / x.shape[3])[..., None]
    return y


def _row_mean_at_poles(x, extra):
    """Rows 0 and H-1 of a bound replaced by their zonal mean plus ``extra`` (same rows)."""
    y = x.clone()
    for r in (0, -1):
        y[:, :, r, :] = (x[:, :, r, :] + extra[:, :, r, :]).mean(dim=-1, keepdim=True)
    return y


def _ordered_scatter(n, idx, val, gen):
    """fp32 sum of ``val`` into ``n`` cells at ``idx`` (1-D), each cell's terms added one by one in an order drawn
    from ``gen``: what a kernel with any fixed summation order could do."""
    perm = torch.randperm(idx.numel(), generator=gen)
    idx, val = idx[perm], val[perm]
    order = torch.sort(idx, stable=True).indices
    idx, val = idx[order], val[order]
    _, counts = torch.unique_consecutive(idx, return_counts=True)
    starts = torch.cumsum(counts, 0) - counts
    rank = torch.arange(idx.numel()) - torch.repeat_interleave(starts, counts)
    acc = torch.zeros(n, dtype=val.dtype)
    for k in range(int(rank.max()) + 1 if rank.numel() else 0):
        sel = rank == k
        acc[idx[sel]] = acc[idx[sel]] + val[sel]
    return acc


def sl_advect_at_coords(field, grad_out, coords, sin_lat, cos_lat, dt, geometry, interpolation="bilinear",
                        pole_fix=True, compute_dtype=torch.float64, scatter_order=None):
    """The operator and its adjoint evaluated AT GIVEN departure coordinates, with a rounding bound per point.

    ``coords`` [B, V, 11, H, W] is what ``ops.departure_coords`` returns (ix, iy, sin lat', cos lat', sin lon',
    cos lon', s, num, den, lat, lon); ``sin_lat``, ``cos_lat`` [H] are the geometry's fp32 tables (``SLGeometry.tables``)
    for a kernel check.  ``out`` and ``grad_field`` are linear in ``field`` / ``grad_out`` with weights that are exact
    functions of (ix, iy), so evaluated in fp64 there is no ``floor()`` ambiguity left: any misrouted, missing or doubled
    term shows up at its point, whatever its weight.  ``grad_u`` / ``grad_v`` use the kernels' Jacobian formula
    (``velocity_grads`` in sl_device.cuh) on the fp32 intermediates, evaluated in fp64, except that ``1 - s^2`` is
    rounded like the kernels and torch's autograd round it, ``fl32(1 - fl32(sc * sc))`` (DESIGN §7), when the
    coordinates are fp32.  Everything runs on the device of the inputs.

    Bounds (first order in u = 2^-24; fp32 kernel minus the fp64 value, per point, no allowance for outliers):

    * out: ``u * sum_t (K_OUT + m_t) |w_t| |f_t| + u * sum_t |f_t| (|wy| rx + ry |wx|)``.  K_OUT = 8: one rounding
      forms the tap weight ``wx * wy`` (bilinear forward), or the taps are summed along x and then along y by FMA
      chains of NT = 4 (bicubic), and a term passes through at most 4 + 4 accumulations.  ``rx``, ``ry`` are the
      running-error bounds of the fp32 axis weights (:func:`_weight_rounding`): 0 or ``|1 - t|`` for bilinear, the
      Horner chain's bound for the cancelling cubic weights.  A pole-mean tap (``pole_fix``) stands for an fp32 sum of
      W values: ``|f_t|`` is the row's mean absolute value and m_t = W (W - 1 additions and one scaling); m_t = 0
      otherwise.  On the output pole rows the bound is the row mean of the bounds plus ``u W`` times the row mean of
      ``sum_t |w_t f_t|``.
    * grad_field: ``u * (K_GFIELD + n_c + m) * sum |w g'|`` over the contributions a cell receives, plus the weights'
      running errors as above.  K_GFIELD = 4 covers the products ``g * wx * wy`` in any association (2 roundings) with
      a margin of 2; n_c (a second scatter_add counts them) bounds the rounding of their sum in ANY order; g' is
      ``grad_out`` after the pole-mean adjoint, and a pole row's g' is a mean (m = W, ``|g'|`` = mean ``|grad_out|``).
      Pole rows of ``grad_field`` (``pole_fix``) are row means again, as for ``out``.
    * grad_u, grad_v: ``u * (K_GRAD_UV + m)`` times the same formula with every sum replaced by the sum of absolute
      values, plus the weights' running errors through it.  K_GRAD_UV = 24: the longest chain is the bicubic
      derivative sum (4 + 4 accumulations), ``g * dx``, ``* Ax``, ``dlam_da`` (``sa cb``, FMA, product, FMA,
      ``* inv_r2``, and 3 for ``inv_r2``: FMA, product, approximate reciprocal of <= 1 ulp), the final FMA and ``* -dt``
      = 19; ``ky`` adds the approximate rsqrt (<= 2 ulp).  m = W when a pole mean enters the point.
    * bf16 gradients (``|ref| + bound``) times U_BF16 = 2^-8 on top: one round-to-nearest of a value with an 8-bit
      significand (half an ulp is up to 2^-8 relative, at the bottom of a binade).

    ``compute_dtype`` / ``scatter_order`` (a torch.Generator) run the same computation in fp32 instead: the axis weights
    by the kernels' fp32 Horner chains, the pole means summed one value after the other, the grad_field sum taken in a
    random order.  That is the test that the bounds are not too tight.  Bounds are only formed in fp64.
    """
    B, V, H, W = field.shape
    p = INTERP_PAD[interpolation]
    Hp, Wp = H + 2 * p, W + 2 * p
    dev = field.device
    fp64 = compute_dtype == torch.float64
    cd = compute_dtype
    Ax, Ay, dt = pixel_scales(geometry, dt)
    c = coords.to(torch.float64)
    ix, iy = c[:, :, 0], c[:, :, 1]
    sa, ca, sb, cb, s, num, den = [c[:, :, k].to(cd) for k in range(2, 9)]
    sp = sin_lat.to(dev, cd).reshape(1, 1, H, 1)
    cp = cos_lat.to(dev, cd).reshape(1, 1, H, 1)

    f = field.to(cd)
    pmean = pole_mean if fp64 else _pole_mean_sequential
    src = pmean(f) if pole_fix else f
    fmag = f.abs()
    if pole_fix:           # a pole tap is an fp32 mean of W values: bound it by the mean absolute value
        fmag = fmag.clone()
        fmag[:, :, 0, :] = f[:, :, 0, :].abs().mean(dim=-1, keepdim=True)
        fmag[:, :, -1, :] = f[:, :, -1, :].abs().mean(dim=-1, keepdim=True)

    x0, y0, offs, wx, wy, dwx, dwy = _stencil(ix, iy, interpolation)
    if not fp64:           # fp32 run: the kernels' fp32 weight chains, fp32 arithmetic from there on
        (wx, dwx), (wy, dwy) = [[[w.v for w in ws] for ws in _axis_weights((t - torch.floor(t)).float(), interpolation,
                                                                           _F32)] for t in (ix, iy)]
    rwx, rdwx = _weight_rounding(ix - torch.floor(ix), interpolation)
    rwy, rdwy = _weight_rounding(iy - torch.floor(iy), interpolation)
    row_map, col_map = geocyclic_source_index(H, W, p)
    flat_map = torch.from_numpy(row_map * W + col_map).to(dev)      # [Hp, Wp]
    src_flat = src.reshape(B, V, H * W)
    mag_flat = fmag.reshape(B, V, H * W)

    def gather(t, idx):
        return torch.gather(t, 2, idx.reshape(B, V, -1)).reshape(B, V, H, W)

    zero = torch.zeros(B, V, H, W, dtype=cd, device=dev)
    out, dsum_x, dsum_y = zero.clone(), zero.clone(), zero.clone()
    m_out = zero.clone().double()         # sum |w f|
    b_out = zero.clone().double()         # sum (K + m_t) |w f| + weight rounding, units of u
    mx, my, ex, ey = [zero.clone().double() for _ in range(4)]   # |.|-sums of dsum_x / dsum_y and weight terms
    pole_pt = torch.zeros(B, V, H, W, dtype=torch.bool, device=dev)
    taps = []
    for a, oy in enumerate(offs):
        row, drow = zero.clone(), zero.clone()          # along x first, then along y (the kernels' order)
        for b, ox in enumerate(offs):
            R, C = y0 + oy, x0 + ox
            ok = (R >= 0) & (R < Hp) & (C >= 0) & (C < Wp)          # padding_mode="zeros"
            Rc, Cc = R.clamp(0, Hp - 1), C.clamp(0, Wp - 1)
            idx = flat_map[Rc, Cc]                                   # [B,V,H,W]
            val = torch.where(ok, gather(src_flat, idx), zero)
            row = row + wx[b] * val
            drow = drow + dwx[b] * val
            taps.append((idx, ok, wy[a] * wx[b], (a, b, Rc, Cc)))
            if not fp64:
                continue
            fm = torch.where(ok, gather(mag_flat, idx), zero)
            srow = idx // W
            pole_tap = ok & bool(pole_fix) & ((srow == 0) | (srow == H - 1))
            pole_pt |= pole_tap
            awx, awy, adx, ady = wx[b].abs(), wy[a].abs(), dwx[b].abs(), dwy[a].abs()
            m_out += awy * awx * fm
            b_out += fm * ((K_OUT + W * pole_tap) * awy * awx + awy * rwx[b] + rwy[a] * awx)
            mx += awy * adx * fm
            my += ady * awx * fm
            ex += fm * (awy * rdwx[b] + rwy[a] * adx)
            ey += fm * (ady * rwx[b] + rdwy[a] * awx)
        out = out + wy[a] * row
        dsum_x = dsum_x + wy[a] * drow
        dsum_y = dsum_y + dwy[a] * row
    res = pmean(out) if pole_fix else out
    if fp64:
        out_bound = b_out
        if pole_fix:
            out_bound = _row_mean_at_poles(b_out, W * m_out)
        out_bound = out_bound * U32
    if grad_out is None:
        if not fp64:
            return AtCoords(out=res)
        return AtCoords(out=res, out_bound=out_bound)

    g0 = grad_out.to(cd)
    g = (_pole_mean_adjoint if fp64 else _pole_mean_sequential)(g0) if pole_fix else g0
    gmag = g0.abs().double()
    if pole_fix:
        gmag = _pole_mean_adjoint(gmag)
        pole_pt[:, :, 0, :] = True
        pole_pt[:, :, -1, :] = True
    gix, giy = g * dsum_x, g * dsum_y

    r2 = num * num + den * den
    dlam_db = (den * ca * cb + num * ca * sb * cp) / r2
    dlam_da = (-den * sa * sb + num * (sa * cb * cp + ca * sp)) / r2
    lo = torch.tensor(-1 + 1e-7, dtype=coords.dtype).item()
    hi = torch.tensor(1 - 1e-7, dtype=coords.dtype).item()
    s_in = coords[:, :, 6]
    inside = ((s_in >= lo) & (s_in <= hi)).to(cd)
    sc = torch.clamp(s_in, lo, hi)
    om = (1 - sc * sc).to(cd)              # rounded in the dtype of the coordinates, like the kernels
    dphi_ds = inside / torch.sqrt(om)
    ds_db = -ca * sb * sp
    ds_da = ca * cp - sa * cb * sp
    grad_u = -dt * (gix * Ax * dlam_db + giy * Ay * dphi_ds * ds_db)
    grad_v = -dt * (gix * Ax * dlam_da + giy * Ay * dphi_ds * ds_da)

    gsrc = torch.zeros(B, V, H * W, dtype=cd, device=dev)
    if scatter_order is not None:
        all_idx = (torch.cat([idx.reshape(B * V, -1) for idx, *_ in taps], 1)
                   + (torch.arange(B * V, device=dev) * (H * W))[:, None]).reshape(-1)
        all_val = torch.cat([torch.where(ok, w * g, torch.zeros_like(g)).reshape(B * V, -1)
                             for idx, ok, w, _ in taps], 1).reshape(-1)
        gsrc = _ordered_scatter(B * V * H * W, all_idx.cpu(), all_val.cpu(), scatter_order).to(dev).reshape(
            B, V, H * W)
    else:
        for idx, ok, w, _ in taps:
            contrib = torch.where(ok, w * g, torch.zeros_like(g))
            gsrc.scatter_add_(2, idx.reshape(B, V, -1), contrib.reshape(B, V, -1))
    gsrc = gsrc.reshape(B, V, H, W)
    grad_field = (_pole_mean_adjoint if fp64 else _pole_mean_sequential)(gsrc) if pole_fix else gsrc
    if not fp64:
        return AtCoords(out=res, grad_field=grad_field, grad_u=grad_u, grad_v=grad_v)

    # grad_field: sum |w g'| with (K + m) per contribution, the weights' rounding, and the count n_c
    m_arr = torch.zeros(B, V, H, W, dtype=torch.float64, device=dev)
    if pole_fix:
        m_arr[:, :, 0, :] = W
        m_arr[:, :, -1, :] = W
    s_mag = torch.zeros(B, V, H * W, dtype=torch.float64, device=dev)
    s_bnd = torch.zeros_like(s_mag)
    n_c = torch.zeros_like(s_mag)
    for idx, ok, w, (a, b, _, _) in taps:
        okd = ok.double()
        mag = okd * gmag * wy[a].abs() * wx[b].abs()
        bnd = (K_GFIELD + m_arr) * mag + okd * gmag * (wy[a].abs() * rwx[b] + rwy[a] * wx[b].abs())
        for acc, t in ((s_mag, mag), (s_bnd, bnd), (n_c, okd)):
            acc.scatter_add_(2, idx.reshape(B, V, -1), t.reshape(B, V, -1))
    gf_bound = (s_bnd + n_c * s_mag).reshape(B, V, H, W)
    if pole_fix:
        gf_bound = _row_mean_at_poles(gf_bound, W * s_mag.reshape(B, V, H, W))
    gf_bound = gf_bound * U32

    # grad_u / grad_v: absolute-value version of the formula
    kx_m, ky_m = gmag * mx * Ax, gmag * my * Ay * dphi_ds
    kx_e, ky_e = gmag * ex * Ax, gmag * ey * Ay * dphi_ds
    adb = ((den * ca * cb).abs() + (num * ca * sb * cp).abs()) / r2
    ada = ((den * sa * sb).abs() + (num * sa * cb * cp).abs() + (num * ca * sp).abs()) / r2
    adsb, adsa = (ca * sb * sp).abs(), (ca * cp).abs() + (sa * cb * sp).abs()
    kk = K_GRAD_UV + W * pole_pt.double()
    gu_bound = U32 * abs(dt) * (kk * (kx_m * adb + ky_m * adsb) + kx_e * adb + ky_e * adsb)
    gv_bound = U32 * abs(dt) * (kk * (kx_m * ada + ky_m * adsa) + kx_e * ada + ky_e * adsa)
    return AtCoords(out=res, grad_field=grad_field, grad_u=grad_u, grad_v=grad_v, out_bound=out_bound,
                    grad_field_bound=gf_bound, grad_u_bound=gu_bound, grad_v_bound=gv_bound, n_c=n_c.reshape(
                        B, V, H, W), taps=taps)


def bf16_bounds(ref, bound):
    """Bound of a bf16 result: the fp32 bound plus one bf16 rounding of a value within it."""
    return bound + U_BF16 * (ref.abs() + bound)


def over_bound(got, ref, bound):
    """Boolean mask of the points where |got - ref| exceeds the bound (NaN counts as over)."""
    err = (got.double() - ref).abs()
    return ~(err <= bound)


def worst_ratio(got, ref, bound):
    """max |got - ref| / bound (0 where both are 0)."""
    err = (got.double() - ref).abs()
    r = torch.where(bound > 0, err / torch.where(bound > 0, bound, torch.ones_like(bound)),
                    torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    return float(r.max())


# --------------------------------------------------------------------------
# Synthetic inputs shared by tests and bench (SURVEY 8c / 8d)
# --------------------------------------------------------------------------
def smooth_field(lat_grid, lon_grid, B: int, V: int, seed: int = 0):
    """Band-limited analytic fields, different phase/amplitude per plane."""
    g = torch.Generator().manual_seed(seed)
    amp = 0.5 + torch.rand(B, V, 1, 1, generator=g, dtype=torch.float64)
    ph = 2 * math.pi * torch.rand(B, V, 1, 1, generator=g, dtype=torch.float64)
    la, lo = lat_grid.double()[None, None], lon_grid.double()[None, None]
    f = amp * (torch.sin(3 * lo + ph) * torch.cos(la) ** 3
               + torch.cos(5 * lo + 1 + ph) * torch.cos(la) ** 5 * torch.sin(2 * la))
    return f


def smooth_velocity(lat_grid, lon_grid, B: int, V: int, cells: float, dt: float, seed: int = 1):
    """Smooth (u, v) whose displacement is about ``cells`` latitude cells."""
    H = lat_grid.shape[0]
    g = torch.Generator().manual_seed(seed)
    ph = 2 * math.pi * torch.rand(2, B, V, 1, 1, generator=g, dtype=torch.float64)
    la, lo = lat_grid.double()[None, None], lon_grid.double()[None, None]
    scale = cells * (math.pi / H) / dt
    u = scale * (torch.cos(2 * lo + ph[0]) * torch.cos(la) + 0.3 * torch.sin(la + ph[1]))
    v = scale * (torch.sin(3 * lo + ph[1]) * torch.cos(2 * la) + 0.3 * torch.cos(lo + ph[0]))
    return u, v


def bench_inputs(H: int, W: int, B: int, V: int, poles: bool, dt: float, seed: int = 0,
                 cells_sigma: float = 2.0, cells_clip: float = 4.0):
    """SURVEY 8d synthetic inputs: field~N(0,1); u,v~N(0,sigma^2) with
    sigma = cells_sigma*dphi/dt clipped at +-cells_clip cells; grad_out~N(0,1)."""
    lat_grid, lon_grid = make_grids(H, W, poles)
    g = torch.Generator().manual_seed(seed)
    dphi = math.pi / H
    sigma, clip = cells_sigma * dphi / dt, cells_clip * dphi / dt
    field = torch.randn(B, V, H, W, generator=g)
    u = (torch.randn(B, V, H, W, generator=g) * sigma).clamp_(-clip, clip)
    v = (torch.randn(B, V, H, W, generator=g) * sigma).clamp_(-clip, clip)
    grad_out = torch.randn(B, V, H, W, generator=g)
    return lat_grid, lon_grid, field, u, v, grad_out
