// float64 advection (include/paradis_sl_f64.h): forward, adjoint, tangent-linear model and the departure-point
// instrument with double storage and double arithmetic in registers.
//
// The fp32 kernels are untouched: their arithmetic is fp32 in every helper (trajectory, stencils, Jacobian) and a
// compute-type template over them would change the machine code of every existing kernel.  These kernels are the
// same algorithms, one point per thread, on the full mesh only:
//   pole_means_f64_kernel / pole_rows_fix_f64_kernel   zonal pole means (deterministic block sums)
//   sl_fwd_f64_kernel          departure point + GeoCyclic stencil gather
//   sl_bwd_arrival_f64_kernel  grad_u, grad_v and the row class of the departure cell (as sl_bwd_arrival_kernel)
//   plane_reach_kernel         shared with the fp32 path (byte classes only)
//   sl_bwd_gather_f64_kernel   grad_field over inverse stencils, double accumulator rows, no atomics
//   sl_tl_f64_kernel           tangent-linear model
//   departure_coords_f64_kernel  the 11 planes of the parity instrument
#include "../../include/paradis_sl_f64.h"

namespace psl64 {

constexpr double kTwoPi = 6.283185307179586;          // 2 * math.pi (advection.py:96), a Python double
constexpr double kA = -0.75;                           // ATen/native/UpSample.h:415

struct Params {
  int H, W, p, Hp, Wp, halfW, B, V, pole_fix, nblk;
  const double* __restrict__ sin_lat;
  const double* __restrict__ cos_lat;
  const double* __restrict__ lon;
  double min_lat, d_lat, min_lon, d_lon, dt;
  double Wm1, Hm1, Wpm1, Hpm1, pf, inv_Wpm1, inv_Hpm1;   // W-1, H-1, Wp-1, Hp-1, p, 1/(Wp-1), 1/(Hp-1)
  double Ax, Ay;                                          // d ix / d lon, d iy / d lat
  double clamp_lo, clamp_hi;                              // -1+1e-7, 1-1e-7 (advection.py:90)
  const double* __restrict__ field;
  const double* __restrict__ u;
  const double* __restrict__ v;
  const double* __restrict__ gout;
  double* __restrict__ out;
  double* __restrict__ gfield;
  double* __restrict__ gu;
  double* __restrict__ gv;
  long long field_sB, u_sB, v_sB, gout_sB;
  const double* __restrict__ fmean;     // [planes][2] zonal means of field rows 0 / H-1
  const double* __restrict__ gmean;     // [planes][2] zonal means of grad_out rows 0 / H-1
  signed char* __restrict__ cls;        // [planes][H][W] row class floor(iy) - (y + p)
  unsigned char* __restrict__ blkmax;   // [planes][nblk] per-block max |class|
  int* __restrict__ plane_reach;        // [planes]
  int* __restrict__ status;
};

struct Traj { double ix, iy, sa, ca, sb, cb, s, num, den, lat, lon; };

__device__ __forceinline__ const double* plane(const double* base, long long sB, int b, int c, int H, int W) {
  return base + (long long)b * sB + (long long)c * H * W;
}

// The reference's chain in double, one rounding per torch op (sl_device.cuh::trajectory<EXACT> in fp32).
__device__ __forceinline__ void trajectory(const Params& P, double u, double v, double sp, double cp, double lonp,
                                           Traj& t) {
  const double lon_r = __dmul_rn(-u, P.dt);
  const double lat_r = __dmul_rn(-v, P.dt);
  t.sa = sin(lat_r); t.ca = cos(lat_r);
  t.sb = sin(lon_r); t.cb = cos(lon_r);
  const double cc = __dmul_rn(t.ca, t.cb);
  t.s = __dadd_rn(__dmul_rn(t.sa, cp), __dmul_rn(cc, sp));
  t.den = __dsub_rn(__dmul_rn(cc, cp), __dmul_rn(t.sa, sp));
  t.num = __dmul_rn(t.ca, t.sb);
  const double sc = fmin(fmax(t.s, P.clamp_lo), P.clamp_hi);
  t.lat = asin(sc);
  double lon = __dadd_rn(lonp, atan2(t.num, t.den));
  // remainder(lon + 2pi, 2pi): the argument is in [pi, 5pi), fmod is one exact subtraction of 4pi or 2pi (Sterbenz)
  lon = __dadd_rn(lon, kTwoPi);
  if (lon >= 2.0 * kTwoPi) lon = __dsub_rn(lon, 2.0 * kTwoPi);
  if (lon >= kTwoPi) lon = __dsub_rn(lon, kTwoPi);
  t.lon = lon;
  // advection.py:138-139: division by the 0-dim tensors d_lon / d_lat is an IEEE division
  const double px = __dmul_rn(__ddiv_rn(__dsub_rn(lon, P.min_lon), P.d_lon), P.Wm1);
  const double py = __dmul_rn(__ddiv_rn(__dsub_rn(t.lat, P.min_lat), P.d_lat), P.Hm1);
  // advection.py:149-150: ATen-CUDA divides by a Python scalar as x * (1 / s), the reciprocal in double
  const double gx = __dsub_rn(__dmul_rn(2.0, __dmul_rn(__dadd_rn(px, P.pf), P.inv_Wpm1)), 1.0);
  const double gy = __dsub_rn(__dmul_rn(2.0, __dmul_rn(__dadd_rn(py, P.pf), P.inv_Hpm1)), 1.0);
  // GridSampler.h: ((g + 1) / 2) * (size - 1)
  t.ix = __dmul_rn(__dmul_rn(__dadd_rn(gx, 1.0), 0.5), P.Wpm1);
  t.iy = __dmul_rn(__dmul_rn(__dadd_rn(gy, 1.0), 0.5), P.Hpm1);
}

// d ix / d u and d iy / d v folded with (gix, giy): the closed form of sl_device.cuh::velocity_grads, in double
__device__ __forceinline__ void velocity_grads(const Params& P, const Traj& t, double sp, double cp, double gix,
                                               double giy, double& gu, double& gv) {
  const double r2 = __dadd_rn(__dmul_rn(t.num, t.num), __dmul_rn(t.den, t.den));
  const double inv_r2 = r2 > 0.0 ? __ddiv_rn(1.0, r2) : 0.0;
  const double cacb = t.ca * t.cb, casb = t.ca * t.sb, sasb = t.sa * t.sb, sacb = t.sa * t.cb;
  const double dlam_db = fma(t.den, cacb, t.num * casb * cp) * inv_r2;
  const double dlam_da = fma(-t.den, sasb, t.num * fma(sacb, cp, t.ca * sp)) * inv_r2;
  const bool inside = (t.s >= P.clamp_lo) && (t.s <= P.clamp_hi);
  const double sc = fmin(fmax(t.s, P.clamp_lo), P.clamp_hi);
  const double om = __dsub_rn(1.0, __dmul_rn(sc, sc));
  const double dphi_ds = inside ? __ddiv_rn(1.0, __dsqrt_rn(om)) : 0.0;
  const double ds_db = -casb * sp;
  const double ds_da = fma(t.ca, cp, -sacb * sp);
  const double kx = gix * P.Ax, ky = giy * P.Ay * dphi_ds;
  gu = -P.dt * fma(kx, dlam_db, ky * ds_db);
  gv = -P.dt * fma(kx, dlam_da, ky * ds_da);
}

template <int INTERP> struct Stencil;
template <> struct Stencil<1> { static constexpr int NT = 2, OMIN = 0; };
template <> struct Stencil<2> { static constexpr int NT = 4, OMIN = -1; };

template <int INTERP>
__device__ __forceinline__ void axis_weights(double t, double (&w)[Stencil<INTERP>::NT],
                                             double (&dw)[Stencil<INTERP>::NT]) {
  if (INTERP == 1) {
    w[0] = 1.0 - t; w[1] = t;
    dw[0] = -1.0; dw[1] = 1.0;
  } else {
    const double t1 = t + 1.0, u0 = 1.0 - t, u1 = u0 + 1.0;
    w[0] = fma(fma(fma(kA, t1, -5.0 * kA), t1, 8.0 * kA), t1, -4.0 * kA);
    w[1] = fma(fma(kA + 2.0, t, -(kA + 3.0)) * t, t, 1.0);
    w[2] = fma(fma(kA + 2.0, u0, -(kA + 3.0)) * u0, u0, 1.0);
    w[3] = fma(fma(fma(kA, u1, -5.0 * kA), u1, 8.0 * kA), u1, -4.0 * kA);
    dw[0] = fma(fma(3.0 * kA, t1, -10.0 * kA), t1, 8.0 * kA);
    dw[1] = fma(3.0 * (kA + 2.0), t, -2.0 * (kA + 3.0)) * t;
    dw[2] = -(fma(3.0 * (kA + 2.0), u0, -2.0 * (kA + 3.0)) * u0);
    dw[3] = -fma(fma(3.0 * kA, u1, -10.0 * kA), u1, 8.0 * kA);
  }
}

// value of the (pole-fixed) field at padded (R, C); zero outside the padded plane (padding_mode="zeros")
__device__ __forceinline__ double tap_value(const Params& P, const double* __restrict__ f, int R, int C, double mean0,
                                            double mean1) {
  if ((unsigned)R >= (unsigned)P.Hp || (unsigned)C >= (unsigned)P.Wp) return 0.0;
  int i = R - P.p, j = C - P.p;
  if (i < 0) { i = -i; j -= P.halfW; }
  else if (i >= P.H) { i = 2 * (P.H - 1) - i; j -= P.halfW; }
  if (j < 0) j += P.W;
  else if (j >= P.W) j -= P.W;
  if (P.pole_fix) {
    if (i == 0) return mean0;
    if (i == P.H - 1) return mean1;
  }
  return __ldg(f + (long long)i * P.W + j);
}

// value (and with GRAD, d/d ix, d/d iy) of the stencil at a departure point; ATen bicubic order (rows along x, then y)
template <int INTERP, bool GRAD>
__device__ __forceinline__ void stencil_eval(const Params& P, const double* __restrict__ f, const Traj& t, double mean0,
                                             double mean1, double& val, double& dx, double& dy) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  const double fx = floor(t.ix), fy = floor(t.iy);
  const int x0 = (int)fx + OMIN, y0 = (int)fy + OMIN;
  double wx[NT], wy[NT], dwx[NT], dwy[NT];
  axis_weights<INTERP>(t.ix - fx, wx, dwx);
  axis_weights<INTERP>(t.iy - fy, wy, dwy);
  val = 0.0; dx = 0.0; dy = 0.0;
#pragma unroll
  for (int a = 0; a < NT; ++a) {
    double r = 0.0, rd = 0.0;
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      const double tap = tap_value(P, f, y0 + a, x0 + b, mean0, mean1);
      r = fma(tap, wx[b], r);
      if (GRAD) rd = fma(tap, dwx[b], rd);
    }
    val = fma(r, wy[a], val);
    if (GRAD) { dx = fma(rd, wy[a], dx); dy = fma(r, dwy[a], dy); }
  }
}

constexpr int kPoleThreads = 128;

__device__ __forceinline__ double block_row_sum(const double* row, int W) {
  __shared__ double part[kPoleThreads / 32];
  double s = 0.0;
  for (int x = threadIdx.x; x < W; x += kPoleThreads) s += row[x];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  double t = part[0];
#pragma unroll
  for (int w = 1; w < kPoleThreads / 32; ++w) t += part[w];
  __syncthreads();
  return t;
}

// means[pl][k] of rows 0 / H-1 of `t`; jobs past planes * 2 do the same for t2 -> means2.  One CTA per (plane, pole).
__global__ void __launch_bounds__(kPoleThreads) pole_means_f64_kernel(const double* __restrict__ t, long long sB,
                                                                      const double* __restrict__ t2, long long sB2,
                                                                      int V, int H, int W, int planes,
                                                                      double* __restrict__ means,
                                                                      double* __restrict__ means2) {
  int job = blockIdx.x;
  if (job >= planes * 2) { job -= planes * 2; t = t2; sB = sB2; means = means2; }
  const int pl = job >> 1, b = pl / V, c = pl - b * V;
  const double* row = plane(t, sB, b, c, H, W) + (long long)((job & 1) ? H - 1 : 0) * W;
  const double m = block_row_sum(row, W) / (double)W;
  if (threadIdx.x == 0) means[job] = m;
}

// rows 0 / H-1 of a contiguous [planes, H, W] tensor <- their zonal mean
__global__ void __launch_bounds__(kPoleThreads) pole_rows_fix_f64_kernel(double* __restrict__ t, int H, int W) {
  const int job = blockIdx.x, pl = job >> 1;
  double* row = t + ((long long)pl * H + ((job & 1) ? H - 1 : 0)) * W;
  const double m = block_row_sum(row, W) / (double)W;
  for (int x = threadIdx.x; x < W; x += kPoleThreads) row[x] = m;
}

template <int INTERP>
__global__ void __launch_bounds__(256) sl_fwd_f64_kernel(const Params P) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P.H * P.W) return;
  const int y = idx / P.W, x = idx - y * P.W;
  double mean0 = 0.0, mean1 = 0.0;
  if (P.pole_fix) { mean0 = P.fmean[2 * pl]; mean1 = P.fmean[2 * pl + 1]; }
  Traj t;
  trajectory(P, __ldg(plane(P.u, P.u_sB, b, c, P.H, P.W) + idx), __ldg(plane(P.v, P.v_sB, b, c, P.H, P.W) + idx),
             __ldg(P.sin_lat + y), __ldg(P.cos_lat + y), __ldg(P.lon + x), t);
  double val, dx, dy;
  stencil_eval<INTERP, false>(P, plane(P.field, P.field_sB, b, c, P.H, P.W), t, mean0, mean1, val, dx, dy);
  P.out[(long long)pl * P.H * P.W + idx] = val;
}

template <int INTERP>
__global__ void __launch_bounds__(256) sl_bwd_arrival_f64_kernel(const Params P) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int reach = 0;
  if (idx < P.H * P.W) {
    const int y = idx / P.W, x = idx - y * P.W;
    const double sp = __ldg(P.sin_lat + y), cp = __ldg(P.cos_lat + y);
    Traj t;
    trajectory(P, __ldg(plane(P.u, P.u_sB, b, c, P.H, P.W) + idx), __ldg(plane(P.v, P.v_sB, b, c, P.H, P.W) + idx),
               sp, cp, __ldg(P.lon + x), t);
    int rc = (int)floor(t.iy) - (y + P.p);
    const int ac = abs(rc);
    if (ac > PARADIS_SL_MAX_DISP_ROWS) {
      if (P.status) *P.status = PARADIS_ERR_DISPLACEMENT;
      rc = rc > 0 ? 127 : -127;
    }
    reach = min(ac, 127);
    if (P.cls) P.cls[(long long)pl * P.H * P.W + idx] = (signed char)rc;
    if (P.gu) {
      double g = __ldg(plane(P.gout, P.gout_sB, b, c, P.H, P.W) + idx);
      double mean0 = 0.0, mean1 = 0.0;
      if (P.pole_fix) {
        mean0 = P.fmean[2 * pl]; mean1 = P.fmean[2 * pl + 1];
        if (y == 0) g = P.gmean[2 * pl];                  // adjoint of the output pole mean
        else if (y == P.H - 1) g = P.gmean[2 * pl + 1];
      }
      double val, dx, dy, gu, gv;
      stencil_eval<INTERP, true>(P, plane(P.field, P.field_sB, b, c, P.H, P.W), t, mean0, mean1, val, dx, dy);
      velocity_grads(P, t, sp, cp, g * dx, g * dy, gu, gv);
      P.gu[(long long)pl * P.H * P.W + idx] = gu;
      P.gv[(long long)pl * P.H * P.W + idx] = gv;
    }
  }
  if (P.blkmax) {   // per-block maximum, no atomics
    __shared__ int smax[8];
    reach = __reduce_max_sync(0xffffffffu, reach);
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = reach;
    __syncthreads();
    if (threadIdx.x == 0) {
      int m = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) m = max(m, smax[w]);
      P.blkmax[(long long)pl * P.nblk + blockIdx.x] = (unsigned char)m;
    }
  }
}

// grad_field: sl_bwd_gather_kernel (paradis_sl.cu) with a double accumulator row per warp.  One warp owns one output
// row; it visits the destination rows folding onto it, compacts the arrival points whose stencil reaches them (raster
// order) and adds their weights 32 at a time, lanes with the same base column combined in lane order by the lowest
// one.  Every add into acc has a single writer and a data-independent order.
constexpr int kGatherWarps = 8;
constexpr int kQueue = 288;     // >= 31 left over + 32 lanes * 8 candidates

template <int INTERP>
__device__ __forceinline__ void gather_chunk(const Params& P, const double* u, const double* v, const double* g,
                                             double gm0, double gm1, int Rd, int shift, double* acc,
                                             const unsigned* queue, int n, int lane) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  double c[NT];
#pragma unroll
  for (int b = 0; b < NT; ++b) c[b] = 0.0;
  int key = -1 - lane;
  if (lane < n) {
    const unsigned e = queue[lane];
    const int y = (int)(e >> 16), x = (int)(e & 0xffffu);
    const long long off = (long long)y * P.W + x;
    double gg = __ldg(g + off);
    if (P.pole_fix) {
      if (y == 0) gg = gm0;
      else if (y == P.H - 1) gg = gm1;
    }
    Traj t;
    trajectory(P, __ldg(u + off), __ldg(v + off), __ldg(P.sin_lat + y), __ldg(P.cos_lat + y), __ldg(P.lon + x), t);
    const double fx = floor(t.ix), fy = floor(t.iy);
    const int a = Rd - ((int)fy + OMIN);
    if (a >= 0 && a < NT) {
      double wx[NT], wy[NT], d0[NT], d1[NT];
      axis_weights<INTERP>(t.ix - fx, wx, d0);
      axis_weights<INTERP>(t.iy - fy, wy, d1);
      double wya = wy[0];
#pragma unroll
      for (int k = 1; k < NT; ++k) wya = (a == k) ? wy[k] : wya;
      const double val = gg * wya;
      const int xb = (int)fx + OMIN;
#pragma unroll
      for (int b = 0; b < NT; ++b) c[b] = ((unsigned)(xb + b) < (unsigned)P.Wp) ? val * wx[b] : 0.0;
      int j = xb - P.p - shift;
      if (j < 0) j += P.W;
      else if (j >= P.W) j -= P.W;
      if ((unsigned)j < (unsigned)P.W) key = j;
      else {
#pragma unroll
        for (int b = 0; b < NT; ++b) c[b] = 0.0;
      }
    }
  }
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  const int leader = __ffs(peers) - 1;
  const int nmax = __reduce_max_sync(0xffffffffu, __popc(peers));
  unsigned rest = peers & (peers - 1);
  for (int rr = 1; rr < nmax; ++rr) {
    const int src = rest ? __ffs(rest) - 1 : lane;
    const bool take = (lane == leader) && rest;
    rest &= rest - 1;
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      const double o = __shfl_sync(0xffffffffu, c[b], src);
      if (take) c[b] += o;
    }
  }
  const bool writer = (lane == leader) && (key >= 0);
#pragma unroll
  for (int b = 0; b < NT; ++b) {
    if (writer) {
      int j = key + b;
      if (j >= P.W) j -= P.W;
      acc[j] += c[b];
    }
    __syncwarp();
  }
}

template <int INTERP>
__global__ void __launch_bounds__(kGatherWarps * 32) sl_bwd_gather_f64_kernel(const Params P) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  extern __shared__ double smem64[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pl = blockIdx.y, b = pl / P.V, c = pl - b * P.V;
  const int r = blockIdx.x * kGatherWarps + warp;
  if (r >= P.H) return;
  double* acc = reinterpret_cast<double*>(reinterpret_cast<char*>(smem64) +
                                          (size_t)warp * (P.W * sizeof(double) + kQueue * sizeof(unsigned)));
  unsigned* queue = reinterpret_cast<unsigned*>(acc + P.W);
  for (int x = lane; x < P.W; x += 32) acc[x] = 0.0;
  __syncwarp();
  const int reach = P.plane_reach[pl];
  const signed char* cls = P.cls + (long long)pl * P.H * P.W;
  const double* u = plane(P.u, P.u_sB, b, c, P.H, P.W);
  const double* v = plane(P.v, P.v_sB, b, c, P.H, P.W);
  const double* g = plane(P.gout, P.gout_sB, b, c, P.H, P.W);
  double gm0 = 0.0, gm1 = 0.0;
  if (P.pole_fix) { gm0 = P.gmean[2 * pl]; gm1 = P.gmean[2 * pl + 1]; }
  for (int src = 0; src < 3; ++src) {          // destination rows folding onto r: itself, north cap, south cap
    int Rd, shift;
    if (src == 0) { Rd = r + P.p; shift = 0; }
    else if (src == 1) { if (r < 1 || r > P.p) continue; Rd = P.p - r; shift = P.halfW; }
    else { const int i = 2 * (P.H - 1) - r; if (i < P.H || i >= P.H + P.p) continue; Rd = i + P.p; shift = P.halfW; }
    const int ylo = max(Rd - P.p - (OMIN + NT - 1) - reach, 0), yhi = min(Rd - P.p - OMIN + reach, P.H - 1);
    int qn = 0;
    for (int y = ylo; y <= yhi; ++y) {
      const signed char* crow = cls + (long long)y * P.W;
      const int cbase = Rd - (y + P.p) - OMIN;  // tap index a = cbase - class must be in [0, NT)
      for (int x0 = 0; x0 < P.W; x0 += 8 * 32) {
        const int x = x0 + lane * 8;
        unsigned m = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (x + k < P.W && (unsigned)(cbase - crow[x + k]) < (unsigned)NT) m |= 1u << k;
        const int cnt = __popc(m);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += t;
        }
        int pos = qn + incl - cnt;
        while (m) {
          const int k = __ffs(m) - 1;
          m &= m - 1;
          queue[pos++] = ((unsigned)y << 16) | (unsigned)(x + k);
        }
        qn += __shfl_sync(0xffffffffu, incl, 31);
        __syncwarp();
        int head = 0;
        while (qn - head >= 32) {
          gather_chunk<INTERP>(P, u, v, g, gm0, gm1, Rd, shift, acc, queue + head, 32, lane);
          head += 32;
        }
        if (head) {
          const int rem = qn - head;
          unsigned e = 0;
          if (lane < rem) e = queue[head + lane];
          __syncwarp();
          if (lane < rem) queue[lane] = e;
          __syncwarp();
          qn = rem;
        }
      }
    }
    if (qn) gather_chunk<INTERP>(P, u, v, g, gm0, gm1, Rd, shift, acc, queue, qn, lane);
  }
  // adjoint of the first enforce_pole_continuity (advection.py:129): pole rows get their mean
  double* orow = P.gfield + ((long long)pl * P.H + r) * P.W;
  if (P.pole_fix && (r == 0 || r == P.H - 1)) {
    double s = 0.0;
    for (int x = lane; x < P.W; x += 32) s += acc[x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double m = s / (double)P.W;
    for (int x = lane; x < P.W; x += 32) orow[x] = m;
  } else {
    for (int x = lane; x < P.W; x += 32) orow[x] = acc[x];
  }
}

struct TLArgs {
  const double* __restrict__ dfield;
  const double* __restrict__ du;
  const double* __restrict__ dv;
  const double* __restrict__ dmean;
  long long dfield_sB, du_sB, dv_sB;
};

// tangent-linear model (sl_tangent.cuh in double): one gather per arrival point, no atomics
template <int INTERP>
__global__ void __launch_bounds__(256) sl_tl_f64_kernel(const Params P, const TLArgs A) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P.H * P.W) return;
  const int y = idx / P.W, x = idx - y * P.W;
  const double sp = __ldg(P.sin_lat + y), cp = __ldg(P.cos_lat + y);
  double mean0 = 0.0, mean1 = 0.0, dmean0 = 0.0, dmean1 = 0.0;
  if (P.pole_fix) {
    mean0 = P.fmean[2 * pl]; mean1 = P.fmean[2 * pl + 1];
    if (A.dfield) { dmean0 = A.dmean[2 * pl]; dmean1 = A.dmean[2 * pl + 1]; }
  }
  Traj t;
  trajectory(P, __ldg(plane(P.u, P.u_sB, b, c, P.H, P.W) + idx), __ldg(plane(P.v, P.v_sB, b, c, P.H, P.W) + idx),
             sp, cp, __ldg(P.lon + x), t);
  double o = 0.0, dx, dy;
  if (A.dfield) stencil_eval<INTERP, false>(P, plane(A.dfield, A.dfield_sB, b, c, P.H, P.W), t, dmean0, dmean1, o, dx, dy);
  if (A.du) {
    double val, gu, gv;
    stencil_eval<INTERP, true>(P, plane(P.field, P.field_sB, b, c, P.H, P.W), t, mean0, mean1, val, dx, dy);
    velocity_grads(P, t, sp, cp, dx, dy, gu, gv);
    o = fma(gu, __ldg(plane(A.du, A.du_sB, b, c, P.H, P.W) + idx), fma(gv, __ldg(plane(A.dv, A.dv_sB, b, c, P.H, P.W) + idx), o));
  }
  P.out[(long long)pl * P.H * P.W + idx] = o;
}

__global__ void __launch_bounds__(256) departure_coords_f64_kernel(const Params P, double* __restrict__ coords) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P.H * P.W) return;
  const int y = idx / P.W, x = idx - y * P.W;
  Traj t;
  trajectory(P, __ldg(plane(P.u, P.u_sB, b, c, P.H, P.W) + idx), __ldg(plane(P.v, P.v_sB, b, c, P.H, P.W) + idx),
             __ldg(P.sin_lat + y), __ldg(P.cos_lat + y), __ldg(P.lon + x), t);
  const long long n = (long long)P.H * P.W;
  double* o = coords + (long long)pl * 11 * n + idx;
  o[0] = t.ix; o[n] = t.iy; o[2 * n] = t.sa; o[3 * n] = t.ca; o[4 * n] = t.sb; o[5 * n] = t.cb;
  o[6 * n] = t.s; o[7 * n] = t.num; o[8 * n] = t.den; o[9 * n] = t.lat; o[10 * n] = t.lon;
}

// ---- host side --------------------------------------------------------------------------------
static int fill(Params& P, const paradis_sl_geom_f64* g, int B, int V, double dt, int interp, int pole_fix, int math) {
  if (!g) return fail(PARADIS_ERR_NULL_POINTER, "geom is NULL");
  if (!g->sin_lat || !g->cos_lat || !g->lon) return fail(PARADIS_ERR_NULL_POINTER, "geom tables are NULL");
  if (interp != PARADIS_INTERP_BILINEAR && interp != PARADIS_INTERP_BICUBIC)
    return fail(PARADIS_ERR_BAD_INTERP, "interp must be 1 (bilinear) or 2 (bicubic), got %d", interp);
  (void)math;                                  // one arithmetic in fp64: the reference's op order
  const int p = interp;
  if (B <= 0 || V <= 0 || g->H <= 0 || g->W <= 0) return fail(PARADIS_ERR_BAD_SHAPE, "non-positive dimension");
  if (g->W % 2) return fail(PARADIS_ERR_ODD_WIDTH, "Number of longitude points must be even (W=%d)", g->W);
  if (g->H < p + 2) return fail(PARADIS_ERR_BAD_SHAPE, "H=%d too small for padding %d", g->H, p);
  if (g->H > 65535 || g->W > 65535) return fail(PARADIS_ERR_BAD_SHAPE, "mesh larger than 65535 not supported");
  if ((long long)g->H * g->W > (1ll << 30)) return fail(PARADIS_ERR_BAD_SHAPE, "mesh larger than 2^30 points");
  if ((long long)B * V > 65535) return fail(PARADIS_ERR_BAD_SHAPE, "B*V=%lld exceeds 65535 planes per call", (long long)B * V);
  memset(&P, 0, sizeof(P));
  P.H = g->H; P.W = g->W; P.p = p; P.Hp = g->H + 2 * p; P.Wp = g->W + 2 * p; P.halfW = g->W / 2;
  P.B = B; P.V = V; P.pole_fix = pole_fix ? 1 : 0;
  P.sin_lat = g->sin_lat; P.cos_lat = g->cos_lat; P.lon = g->lon;
  P.min_lat = g->min_lat; P.d_lat = g->d_lat; P.min_lon = g->min_lon; P.d_lon = g->d_lon;
  P.dt = dt;
  P.Wm1 = (double)g->W - 1.0; P.Hm1 = (double)g->H - 1.0;
  P.Wpm1 = (double)(P.Wp - 1); P.Hpm1 = (double)(P.Hp - 1); P.pf = (double)p;
  P.inv_Wpm1 = 1.0 / P.Wpm1; P.inv_Hpm1 = 1.0 / P.Hpm1;
  P.Ax = P.Wm1 / g->d_lon; P.Ay = P.Hm1 / g->d_lat;
  P.clamp_lo = -1 + 1e-7; P.clamp_hi = 1 - 1e-7;
  return PARADIS_OK;
}

static dim3 point_grid(const Params& P) { return dim3((unsigned)(((long long)P.H * P.W + 255) / 256), P.V, P.B); }

static size_t means_bytes(int B, int V) { return align_up((size_t)B * V * 2 * sizeof(double), 256); }

struct BwdWs { size_t fmean, gmean, reach, blkmax, cls, total; int nblk; };
static BwdWs bwd_layout(int B, int V, int H, int W) {
  BwdWs w;
  const size_t planes = (size_t)B * V;
  w.nblk = (int)(((size_t)H * W + 255) / 256);
  size_t off = 0;
  w.fmean = off; off += means_bytes(B, V);
  w.gmean = off; off += means_bytes(B, V);
  w.reach = off; off += align_up(planes * sizeof(int), 256);
  w.blkmax = off; off += align_up(planes * (size_t)w.nblk, 256);
  w.cls = off; off += align_up(planes * (size_t)H * W, 256);
  w.total = off;
  return w;
}

static size_t gather_smem(int W) { return (size_t)kGatherWarps * (W * sizeof(double) + kQueue * sizeof(unsigned)); }

}  // namespace psl64

extern "C" size_t paradis_sl_advect_fwd_f64_workspace(int B, int V) { return psl64::means_bytes(B, V); }

extern "C" int paradis_sl_advect_fwd_f64(const paradis_sl_geom_f64* geom, const double* field, const double* u,
                                         const double* v, double* out, int B, int V, int64_t field_sB, int64_t u_sB,
                                         int64_t v_sB, double dt, int interp, int pole_fix, int math, void* workspace,
                                         size_t workspace_bytes, int32_t* status, void* stream) {
  using namespace psl64;
  using psl64::Params; using psl64::TLArgs; using psl64::BwdWs; using psl64::kPoleThreads; using psl64::kGatherWarps;
  Params P;
  if (int rc = fill(P, geom, B, V, dt, interp, pole_fix, math)) return rc;
  if (!field || !u || !v || !out) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if (pole_fix && (!workspace || workspace_bytes < paradis_sl_advect_fwd_f64_workspace(B, V)))
    return fail(PARADIS_ERR_WORKSPACE, "forward workspace too small (%zu bytes)", workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  P.field = field; P.u = u; P.v = v; P.out = out;
  P.field_sB = field_sB; P.u_sB = u_sB; P.v_sB = v_sB;
  P.status = status;
  const int planes = B * V;
  if (pole_fix) {
    P.fmean = (const double*)workspace;
    pole_means_f64_kernel<<<planes * 2, kPoleThreads, 0, st>>>(field, field_sB, nullptr, 0, V, P.H, P.W, planes,
                                                              (double*)P.fmean, nullptr);
  }
  if (interp == 1) sl_fwd_f64_kernel<1><<<point_grid(P), 256, 0, st>>>(P);
  else sl_fwd_f64_kernel<2><<<point_grid(P), 256, 0, st>>>(P);
  if (pole_fix) pole_rows_fix_f64_kernel<<<planes * 2, kPoleThreads, 0, st>>>(out, P.H, P.W);
  return check_launch("paradis_sl_advect_fwd_f64");
}

extern "C" size_t paradis_sl_advect_bwd_f64_workspace(int B, int V, int H, int W) {
  return psl64::bwd_layout(B, V, H, W).total;
}

extern "C" int paradis_sl_advect_bwd_f64(const paradis_sl_geom_f64* geom, const double* grad_out, const double* field,
                                         const double* u, const double* v, double* grad_field, double* grad_u,
                                         double* grad_v, int B, int V, int64_t gout_sB, int64_t field_sB, int64_t u_sB,
                                         int64_t v_sB, double dt, int interp, int pole_fix, int math, void* workspace,
                                         size_t workspace_bytes, int32_t* status, void* stream) {
  using namespace psl64;
  using psl64::Params; using psl64::TLArgs; using psl64::BwdWs; using psl64::kPoleThreads; using psl64::kGatherWarps;
  Params P;
  if (int rc = fill(P, geom, B, V, dt, interp, pole_fix, math)) return rc;
  if (!grad_out || !field || !u || !v) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if ((grad_u == nullptr) != (grad_v == nullptr))
    return fail(PARADIS_ERR_NULL_POINTER, "grad_u and grad_v must both be given or both be NULL");
  const size_t smem = gather_smem(P.W);
  if (grad_field && smem > 227 * 1024)
    return fail(PARADIS_ERR_BAD_SHAPE, "W=%d too wide for the fp64 gather kernel's shared memory", P.W);
  const BwdWs L = psl64::bwd_layout(B, V, P.H, P.W);
  if (!workspace || workspace_bytes < L.total)
    return fail(PARADIS_ERR_WORKSPACE, "backward workspace too small (%zu < %zu bytes)", workspace_bytes, L.total);
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  const int planes = B * V;
  P.field = field; P.u = u; P.v = v; P.gout = grad_out; P.gfield = grad_field; P.gu = grad_u; P.gv = grad_v;
  P.field_sB = field_sB; P.u_sB = u_sB; P.v_sB = v_sB; P.gout_sB = gout_sB;
  P.status = status;
  P.fmean = (const double*)(ws + L.fmean); P.gmean = (const double*)(ws + L.gmean);
  P.plane_reach = (int*)(ws + L.reach);
  P.blkmax = grad_field ? (unsigned char*)(ws + L.blkmax) : nullptr;
  P.cls = grad_field ? (signed char*)(ws + L.cls) : nullptr;
  P.nblk = L.nblk;
  if (pole_fix)     // zonal pole means of field and grad_out in one launch
    pole_means_f64_kernel<<<planes * 4, kPoleThreads, 0, st>>>(field, field_sB, grad_out, gout_sB, V, P.H, P.W, planes,
                                                              (double*)P.fmean, (double*)P.gmean);
  if (interp == 1) sl_bwd_arrival_f64_kernel<1><<<point_grid(P), 256, 0, st>>>(P);
  else sl_bwd_arrival_f64_kernel<2><<<point_grid(P), 256, 0, st>>>(P);
  if (grad_field) {
    plane_reach_kernel<<<(planes * 32 + 255) / 256, 256, 0, st>>>(P.blkmax, P.nblk, planes, P.plane_reach, nullptr,
                                                                   nullptr, 0);
    auto kern = interp == 1 ? sl_bwd_gather_f64_kernel<1> : sl_bwd_gather_f64_kernel<2>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(PARADIS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    kern<<<dim3((P.H + kGatherWarps - 1) / kGatherWarps, planes), kGatherWarps * 32, smem, st>>>(P);
  }
  return check_launch("paradis_sl_advect_bwd_f64");
}

extern "C" size_t paradis_sl_advect_jvp_f64_workspace(int B, int V) { return 2 * psl64::means_bytes(B, V); }

extern "C" int paradis_sl_advect_jvp_f64(const paradis_sl_geom_f64* geom, const double* field, const double* dfield,
                                         const double* u, const double* v, const double* du, const double* dv,
                                         double* dout, int B, int V, int64_t field_sB, int64_t dfield_sB, int64_t u_sB,
                                         int64_t v_sB, int64_t du_sB, int64_t dv_sB, double dt, int interp,
                                         int pole_fix, int math, void* workspace, size_t workspace_bytes,
                                         int32_t* status, void* stream) {
  using namespace psl64;
  using psl64::Params; using psl64::TLArgs; using psl64::BwdWs; using psl64::kPoleThreads; using psl64::kGatherWarps;
  Params P;
  if (int rc = fill(P, geom, B, V, dt, interp, pole_fix, math)) return rc;
  if (!field || !u || !v || !dout) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if ((du == nullptr) != (dv == nullptr)) return fail(PARADIS_ERR_NULL_POINTER, "du and dv must both be given or both be NULL");
  if (pole_fix && (!workspace || workspace_bytes < paradis_sl_advect_jvp_f64_workspace(B, V)))
    return fail(PARADIS_ERR_WORKSPACE, "jvp workspace too small (%zu bytes)", workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  const int planes = B * V;
  P.field = field; P.u = u; P.v = v; P.out = dout;
  P.field_sB = field_sB; P.u_sB = u_sB; P.v_sB = v_sB;
  P.status = status;
  TLArgs A;
  A.dfield = dfield; A.du = du; A.dv = dv; A.dmean = nullptr;
  A.dfield_sB = dfield_sB; A.du_sB = du_sB; A.dv_sB = dv_sB;
  if (pole_fix) {
    P.fmean = (const double*)workspace;
    A.dmean = (const double*)((char*)workspace + means_bytes(B, V));
    pole_means_f64_kernel<<<planes * (dfield ? 4 : 2), kPoleThreads, 0, st>>>(
        field, field_sB, dfield, dfield_sB, V, P.H, P.W, planes, (double*)P.fmean, (double*)A.dmean);
  }
  if (interp == 1) sl_tl_f64_kernel<1><<<point_grid(P), 256, 0, st>>>(P, A);
  else sl_tl_f64_kernel<2><<<point_grid(P), 256, 0, st>>>(P, A);
  if (pole_fix) pole_rows_fix_f64_kernel<<<planes * 2, kPoleThreads, 0, st>>>(dout, P.H, P.W);
  return check_launch("paradis_sl_advect_jvp_f64");
}

extern "C" int paradis_sl_departure_coords_f64(const paradis_sl_geom_f64* geom, const double* u, const double* v,
                                               double* coords, int B, int V, int64_t u_sB, int64_t v_sB, double dt,
                                               int interp, int math, void* stream) {
  using namespace psl64;
  using psl64::Params; using psl64::TLArgs; using psl64::BwdWs; using psl64::kPoleThreads; using psl64::kGatherWarps;
  Params P;
  if (int rc = fill(P, geom, B, V, dt, interp, 0, math)) return rc;
  if (!u || !v || !coords) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  P.u = u; P.v = v; P.u_sB = u_sB; P.v_sB = v_sB;
  departure_coords_f64_kernel<<<point_grid(P), 256, 0, (cudaStream_t)stream>>>(P, coords);
  return check_launch("paradis_sl_departure_coords_f64");
}
