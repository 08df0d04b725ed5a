// Tangent-linear model of the advection (include/paradis_sl_tl.h):
//
//   dout = (d out / d field) dfield + (d out / d u) du + (d out / d v) dv
//
// A pure gather, one output per arrival point: the departure point comes from the same trajectory<EXACT>() as the
// forward and the backward (so ix, iy, the FAST wrap at ix = W + p and the clamp of s agree bit for bit), the stencil
// of `field` gives d val / d ix and d val / d iy, velocity_grads() turns them into d val / d u and d val / d v, and
// the stencil of `dfield` at the same taps is the forward's own evaluation -- with du = dv = 0 the result is the
// forward applied to dfield, bit for bit.  No scatter, no atomics: deterministic.
//
// pole_fix: the tangent of a pole-row mean is the mean of the tangent, so the zonal means of dfield's pole rows
// replace its pole taps (as the field's means replace the field's), and dout's rows 0 / H-1 are replaced by their
// zonal means afterwards (pole_rows_fix_kernel), as the forward does with out.
//
// Full mesh only: the windows of P are (0, H) and no peer halos are set.

struct TLArgs {
  const float* __restrict__ dfield;   // may be NULL: velocity tangents only
  const float* __restrict__ du;       // du and dv both NULL (field tangent only) or both set
  const float* __restrict__ dv;
  const float* __restrict__ dmean;    // [planes][2] zonal means of dfield rows 0 / H-1 (pole_fix)
  long long dfield_sB, du_sB, dv_sB;
};

template <bool EXACT, int INTERP, int VEC>
__global__ void __launch_bounds__(256) sl_tl_kernel(const Params P, const TLArgs A) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const unsigned unit = blockIdx.x * blockDim.x + threadIdx.x;
  if (unit >= (unsigned)(P.ownN * P.upr)) return;
  const unsigned r = P.w4_mul ? fast_div(unit, P.w4_mul, P.w4_shift) : unit / (unsigned)P.upr;
  const int x = (unit - r * P.upr) * VEC;
  const int y = (int)r;                       // full mesh: arrival row = own row
  const float sp = __ldg(P.sin_lat + y), cp = __ldg(P.cos_lat + y);
  const long long aoff = (long long)y * P.W + x;
  const float* f = plane_ptr_bc(P.field, P.field_sB, b, c, P.H, P.W);
  const float* df = A.dfield ? plane_ptr_bc(A.dfield, A.dfield_sB, b, c, P.H, P.W) : nullptr;
  const bool vel = A.du != nullptr;
  const float* up = plane_ptr_bc(P.u, P.u_sB, b, c, P.H, P.W) + aoff;
  const float* vp = plane_ptr_bc(P.v, P.v_sB, b, c, P.H, P.W) + aoff;
  float mean0 = 0.0f, mean1 = 0.0f, dmean0 = 0.0f, dmean1 = 0.0f;
  if (P.pole_fix) {
    mean0 = __ldg(P.fmean + 2 * pl); mean1 = __ldg(P.fmean + 2 * pl + 1);
    if (df) { dmean0 = __ldg(A.dmean + 2 * pl); dmean1 = __ldg(A.dmean + 2 * pl + 1); }
  }
  float uu[VEC], vv[VEC], ll[VEC], du[VEC], dv[VEC], oo[VEC];
  if (VEC == 4) {
    *reinterpret_cast<float4*>(uu) = ldcs4_f(up);
    *reinterpret_cast<float4*>(vv) = ldcs4_f(vp);
    *reinterpret_cast<float4*>(ll) = __ldg(reinterpret_cast<const float4*>(P.lon + x));
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) { uu[k] = ldcs_f(up + k); vv[k] = ldcs_f(vp + k); ll[k] = __ldg(P.lon + x + k); }
  }
  if (vel) {
    const float* dup = plane_ptr_bc(A.du, A.du_sB, b, c, P.H, P.W) + aoff;
    const float* dvp = plane_ptr_bc(A.dv, A.dv_sB, b, c, P.H, P.W) + aoff;
    if (VEC == 4) {
      *reinterpret_cast<float4*>(du) = ldcs4_f(dup);
      *reinterpret_cast<float4*>(dv) = ldcs4_f(dvp);
    } else {
#pragma unroll
      for (int k = 0; k < VEC; ++k) { du[k] = ldcs_f(dup + k); dv[k] = ldcs_f(dvp + k); }
    }
  }
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    Traj t;
    trajectory<EXACT>(P, uu[k], vv[k], sp, cp, ll[k], t);
    float o = 0.0f, dx, dy;
    if (df) stencil_eval<INTERP, false, false>(P, df, pl, t, dmean0, dmean1, o, dx, dy);
    if (vel) {
      float val, gu, gv;
      stencil_eval<INTERP, true, false>(P, f, pl, t, mean0, mean1, val, dx, dy);
      velocity_grads<EXACT>(P, t, sp, cp, dx, dy, gu, gv);
      o = __fmaf_rn(gu, du[k], __fmaf_rn(gv, dv[k], o));
    }
    oo[k] = o;
  }
  float* op = P.out + (long long)pl * P.H * P.W + aoff;
  if (VEC == 4) __stcs(reinterpret_cast<float4*>(op), *reinterpret_cast<float4*>(oo));
  else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) __stcs(op + k, oo[k]);
  }
}

template <bool EXACT, int INTERP>
static void launch_tl(const Params& P, const TLArgs& A, int vec, dim3 grid, cudaStream_t st) {
  if (vec == 4) sl_tl_kernel<EXACT, INTERP, 4><<<grid, 256, 0, st>>>(P, A);
  else sl_tl_kernel<EXACT, INTERP, 1><<<grid, 256, 0, st>>>(P, A);
}
