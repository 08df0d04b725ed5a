"""fp64 reference of the tangent-linear advection (``paradis_sl_advect_jvp``) at given departure coordinates, with a
per-point rounding bound.  Test infrastructure beside oracle/sl_oracle.py, whose ``sl_advect_at_coords`` it is built
from."""
import torch

from oracle.sl_oracle import K_OUT, U32, AtCoords, _F32, _pole_mean_sequential, pole_mean, sl_advect_at_coords


def sl_advect_tangent_at_coords(field, dfield, du, dv, coords, sin_lat, cos_lat, dt, geometry,
                                interpolation="bilinear", pole_fix=True, compute_dtype=torch.float64):
    """The tangent-linear model ``dout = (d out / d field) dfield + (d out / d u) du + (d out / d v) dv`` AT GIVEN
    departure coordinates, with a rounding bound per point (``paradis_sl_advect_jvp``).  Arguments as
    :func:`sl_advect_at_coords`; ``dfield`` may be None (velocity tangents only).  Returns an :class:`AtCoords` with
    ``out`` (the tangent) and, in fp64, ``out_bound``.

    The identity is exact in fp64: ``dout = out_at(dfield) + P(gu1 du + gv1 dv)``, where ``gu1``, ``gv1`` are
    :func:`sl_advect_at_coords`'s ``grad_u``, ``grad_v`` with ``grad_out = 1`` and ``P`` replaces rows 0 / H-1 by their
    zonal means when ``pole_fix`` (the identity otherwise).  With ``grad_out = 1`` the pole-mean adjoint leaves 1, so a
    pole-row point's ``grad_u`` is its own pre-mean derivative; and the tangent of the field's pole-mean taps is the
    mean of the tangent's pole rows, which ``out_at(dfield)`` uses.

    The kernel forms, per point, ``o = fma(gu, du, fma(gv, dv, val))`` with ``val`` the stencil of ``dfield`` and
    ``gu``, ``gv`` the velocity derivatives of the stencil of ``field`` (no ``grad_out`` factor), then the row means.
    Bound (first order in u = 2^-24), with ``T = |gu1 du| + |gv1 dv|`` and ``M`` a bound of ``|val|``:

    * off the mean rows: ``out_bound(dfield) + |du| grad_u_bound + |dv| grad_v_bound + u (3 T + 2 M)``: the
      components' own bounds, one product per velocity term (T; an FMA rounds less) and two adds (each at most
      ``u (T + M)``).  ``M = out_bound / (K_OUT u)``: the forward bound counts at least K_OUT roundings of ``sum |w f|``.
    * the mean rows (``pole_fix``): ``out_bound(dfield)`` (which holds the row mean of ``val`` already), plus the row
      mean of the velocity part above, plus ``(W + 1) u`` times the row mean of T (W - 1 additions, one scaling, of the
      velocity terms within the row sum).  There the row mean of M is ``out_bound / ((K_OUT + W) u)``.

    ``compute_dtype=torch.float32`` runs the kernel's chain in fp32 instead (value only): the stencil of the fp32 pole
    means of ``dfield`` without the output mean, the two FMAs, and the row means summed one value after the other.
    """
    B, V, H, W = field.shape
    fp64 = compute_dtype == torch.float64
    cd = compute_dtype
    ones = torch.ones(B, V, H, W, dtype=cd, device=field.device)
    g1 = sl_advect_at_coords(field, ones, coords, sin_lat, cos_lat, dt, geometry, interpolation, pole_fix,
                             compute_dtype=cd)
    du, dv = du.to(cd), dv.to(cd)
    if not fp64:
        val = torch.zeros_like(ones)
        if dfield is not None:
            src = _pole_mean_sequential(dfield.to(cd)) if pole_fix else dfield.to(cd)
            val = sl_advect_at_coords(src, None, coords, sin_lat, cos_lat, dt, geometry, interpolation, False,
                                      compute_dtype=cd).out
        o = _F32(g1.grad_u).fma(du, _F32(g1.grad_v).fma(dv, val)).v
        return AtCoords(out=_pole_mean_sequential(o) if pole_fix else o)

    vel = g1.grad_u * du + g1.grad_v * dv
    T = (g1.grad_u * du).abs() + (g1.grad_v * dv).abs()
    e_vel = du.abs() * g1.grad_u_bound + dv.abs() * g1.grad_v_bound + U32 * 3 * T
    out = torch.zeros_like(vel)
    out_b = torch.zeros_like(vel)
    if dfield is not None:
        r = sl_advect_at_coords(dfield, None, coords, sin_lat, cos_lat, dt, geometry, interpolation, pole_fix)
        out, out_b = r.out, r.out_bound
    M = out_b / (K_OUT * U32)
    bound = out_b + e_vel + U32 * 2 * M
    if pole_fix:
        vel = pole_mean(vel)
        for row in (0, H - 1):
            m_pole = out_b[:, :, row, :] / ((K_OUT + W) * U32)
            bound[:, :, row, :] = (out_b[:, :, row, :] + e_vel[:, :, row, :].mean(dim=-1, keepdim=True)
                                   + U32 * 2 * m_pole + U32 * (W + 1) * T[:, :, row, :].mean(dim=-1, keepdim=True))
    return AtCoords(out=out + vel, out_bound=bound)
