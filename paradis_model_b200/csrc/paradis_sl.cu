// libparadis_sl.so -- fused semi-Lagrangian advection + GeoCyclic padding for B200 (sm_100a).
//
// Replaces the reference's Python hot path model/advection.py:129-169 and
// model/padding.py:11-39 (see include/paradis_sl.h for the boundary).
//
// Kernels
//   pole_means_kernel      zonal means of rows 0 / H-1 (advection.py:100-114), deterministic
//   sl_fwd_kernel          backtrack + GeoCyclic index map + bilinear/bicubic gather, fused
//   pole_rows_fix_kernel   post pole-mean of the output rows 0 / H-1
//   sl_bwd_arrival_kernel  per arrival point: grad_u, grad_v (+ row class of the departure cell)
//   plane_reach_kernel     per-plane max |row class| (bounds the inverse-stencil window)
//   sl_bwd_gather_kernel   grad_field: each output row gathers the arrival points whose stencil
//                          covers it (inverse stencils), fixed order, no atomics
//   geocyclic_pad_{fwd,bwd}_kernel  standalone padding op and its adjoint
//   sl_tl_kernel           tangent-linear model: d out along (dfield, du, dv), one gather per point (sl_tangent.cuh)
//   *_f64_kernel           float64 storage and arithmetic, full mesh (sl_f64.cuh)
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <vector>

#include "../../include/paradis_sl.h"
#include "../../include/paradis_sl_bf16.h"
#include "../../include/paradis_geocyclic.h"
#include "../../include/paradis_sl_tl.h"
#include "sl_device.cuh"

using namespace psl;

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

void psl_set_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg); }   // for geo_dwconv.cu

static int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(PARADIS_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return PARADIS_OK;
}

extern "C" int paradis_sl_abi_version(void) { return PARADIS_SL_ABI_VERSION; }
extern "C" const char* paradis_last_error(void) { return g_err; }

// ---------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ const T* plane_ptr(const T* base, long long sB, int V, int rows, int W, int pl) {
  const int b = pl / V, c = pl - b * V;
  return base + (long long)b * sB + (long long)c * rows * W;
}
// same, for kernels launched on a (blocks, V, B) grid: no integer division
template <typename T>
__device__ __forceinline__ const T* plane_ptr_bc(const T* base, long long sB, int b, int c, int rows, int W) {
  return base + (long long)b * sB + (long long)c * rows * W;
}

// deterministic zonal sum of one row by one warp (fixed lane/iteration order)
__device__ __forceinline__ float warp_row_sum(const float* row, int W, int lane) {
  float s = 0.0f;
  for (int x = lane; x < W; x += 32) s += row[x];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}

// deterministic zonal sum of one row by one 128-thread CTA: fixed per-thread order, shuffle tree, the four warp
// partials added in warp order (one warp walking a 1440-element row took 8.5 us per launch, five launches per step)
constexpr int kPoleThreads = 128;
template <typename T>
__device__ __forceinline__ float block_row_sum(const T* row, int W) {
  __shared__ float part[kPoleThreads / 32];
  float s = 0.0f;
  for (int x = threadIdx.x; x < W; x += kPoleThreads) s += ld_f(row + x);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  float t = part[0];
#pragma unroll
  for (int w = 1; w < kPoleThreads / 32; ++w) t += part[w];
  __syncthreads();
  return t;
}

// means[pl][k], k = 0: global row 0, k = 1: global row H-1 of tensor `t` whose window is (row0, rows); one CTA per
// (plane, pole).  A second tensor (t2 -> means2, its own window) rides in the same launch (backward: field, grad_out).
// T = storage type of `t` (field); t2 (grad_out) is fp32.
template <typename T>
__device__ __forceinline__ float pole_row_mean(const T* t, long long sB, int V, int rows, int row0, int H, int W, int job) {
  const int pl = job >> 1, k = job & 1;
  const int gr = k ? H - 1 : 0, lr = gr - row0;
  float m = 0.0f;
  if (lr >= 0 && lr < rows) {
    const T* row = plane_ptr(t, sB, V, rows, W, pl) + (long long)lr * W;
    m = block_row_sum(row, W) / (float)W;
  }
  return m;
}
template <typename T>
__global__ void __launch_bounds__(kPoleThreads) pole_means_kernel(const T* __restrict__ t, long long sB, int V, int rows, int row0,
                                                                  int H, int W, int planes, float* __restrict__ means,
                                                                  const float* __restrict__ t2, long long sB2, int rows2,
                                                                  int row02, float* __restrict__ means2) {
  int job = blockIdx.x;
  if (job >= planes * 2) {
    if (!t2) return;
    job -= planes * 2;
    if constexpr (kIsF32<T>) {
      t = t2; sB = sB2; rows = rows2; row0 = row02; means = means2;
    } else {                                   // fp32 grad_out beside a bf16 field
      const float m = pole_row_mean(t2, sB2, V, rows2, row02, H, W, job);
      if (threadIdx.x == 0) means2[job] = m;
      return;
    }
  }
  const float m = pole_row_mean(t, sB, V, rows, row0, H, W, job);
  if (threadIdx.x == 0) means[job] = m;
}

// out rows 0 / H-1 <- their zonal mean (second enforce_pole_continuity, advection.py:169); one CTA per (plane, pole)
__global__ void __launch_bounds__(kPoleThreads) pole_rows_fix_kernel(float* __restrict__ t, int rows, int row0, int H, int W, int planes) {
  const int job = blockIdx.x;
  const int pl = job >> 1, k = job & 1;
  const int gr = k ? H - 1 : 0, lr = gr - row0;
  if (lr < 0 || lr >= rows) return;
  float* row = t + ((long long)pl * rows + lr) * W;
  const float m = block_row_sum(row, W) / (float)W;
  for (int x = threadIdx.x; x < W; x += kPoleThreads) row[x] = m;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
template <bool EXACT, int INTERP, int VEC, bool PEER, typename T>
__global__ void __launch_bounds__(256) sl_fwd_kernel(const Params P) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const unsigned unit = blockIdx.x * blockDim.x + threadIdx.x;
  if (unit >= (unsigned)(P.ownN * P.upr)) return;
  const unsigned r = P.w4_mul ? fast_div(unit, P.w4_mul, P.w4_shift) : unit / (unsigned)P.upr;
  const int x = (unit - r * P.upr) * VEC;
  const int y = P.own0 + (int)r;  // global arrival row
  const float sp = __ldg(P.sin_lat + y), cp = __ldg(P.cos_lat + y);
  const T* f = plane_ptr_bc(as<T>(P.field), P.field_sB, b, c, P.fldN, P.W);
  const int aoff = (y - P.uvg0) * P.W + x;
  const T* up = plane_ptr_bc(as<T>(P.u), P.u_sB, b, c, P.uvgN, P.W) + aoff;
  const T* vp = plane_ptr_bc(as<T>(P.v), P.v_sB, b, c, P.uvgN, P.W) + aoff;
  float mean0 = 0.0f, mean1 = 0.0f;
  if (P.pole_fix) { mean0 = __ldg(P.fmean + 2 * pl); mean1 = __ldg(P.fmean + 2 * pl + 1); }
  float uu[VEC], vv[VEC], ll[VEC], oo[VEC];
  if (VEC == 4) {
    *reinterpret_cast<float4*>(uu) = ldcs4_f(up);
    *reinterpret_cast<float4*>(vv) = ldcs4_f(vp);
    *reinterpret_cast<float4*>(ll) = __ldg(reinterpret_cast<const float4*>(P.lon + x));
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) { uu[k] = ldcs_f(up + k); vv[k] = ldcs_f(vp + k); ll[k] = __ldg(P.lon + x + k); }
  }
  if (!EXACT && VEC == 4) {
    // FAST math: the 4 departure points of the thread as two packed pairs (FFMA2 / FMUL2 / FADD2), bit-identical to
    // the scalar chain
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      Traj2 t2;
      trajectory_2(P, make_float2(uu[2 * h], uu[2 * h + 1]), make_float2(vv[2 * h], vv[2 * h + 1]), f2s(sp), f2s(cp),
                   make_float2(ll[2 * h], ll[2 * h + 1]), t2);
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const Traj t = traj_half(t2, e);
        float dx, dy;
        stencil_eval<INTERP, false, PEER>(P, f, pl, t, mean0, mean1, oo[2 * h + e], dx, dy);
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      Traj t;
      trajectory<EXACT>(P, uu[k], vv[k], sp, cp, ll[k], t);
      float dx, dy;
      stencil_eval<INTERP, false, PEER>(P, f, pl, t, mean0, mean1, oo[k], dx, dy);
    }
  }
  float* op = P.out + ((long long)pl * P.ownN + r) * P.W + x;
  if (VEC == 4) __stcs(reinterpret_cast<float4*>(op), *reinterpret_cast<float4*>(oo));
  else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) __stcs(op + k, oo[k]);
  }
}

// ---------------------------------------------------------------------------------------------
// backward, per arrival point: grad_u, grad_v and the row class of the departure cell
// ---------------------------------------------------------------------------------------------
#include "sl_sweep.cuh"
#include "sl_rows.cuh"
#include "sl_partition.cuh"

template <bool EXACT, int INTERP, int VEC, bool PEER, typename T>
__global__ void __launch_bounds__(256) sl_bwd_arrival_kernel(const Params P) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  if (P.plane_filter && !P.plane_filter[pl]) return;   // uniform per block
  int reach = 0;
  // grid-stride over the units of the plane: the fallback launch behind the row sweep (plane_filter set, almost
  // always nothing to do) runs a handful of blocks per plane instead of one per 256 units
  for (unsigned unit = blockIdx.x * blockDim.x + threadIdx.x; unit < (unsigned)(P.it_arrN * P.upr);
       unit += gridDim.x * blockDim.x) {
    const unsigned r = P.w4_mul ? fast_div(unit, P.w4_mul, P.w4_shift) : unit / (unsigned)P.upr;
    const int x = (unit - r * P.upr) * VEC;
    const int y = P.it_arr0 + (int)r;  // global arrival row
    const bool own = (y >= P.it_own0) && (y < P.it_own0 + P.it_ownN) && (P.gu != nullptr);
    const float sp = __ldg(P.sin_lat + y), cp = __ldg(P.cos_lat + y);
    const T* up = arr_row<PEER>(P, plane_ptr_bc(as<T>(P.u), P.u_sB, b, c, P.uvgN, P.W), 0, pl, y) + x;
    const T* vp = arr_row<PEER>(P, plane_ptr_bc(as<T>(P.v), P.v_sB, b, c, P.uvgN, P.W), 1, pl, y) + x;
    float uu[VEC], vv[VEC], ll[VEC], gg[VEC], ou[VEC], ov[VEC];
    signed char cc[VEC];
    if (VEC == 4) {
      *reinterpret_cast<float4*>(uu) = ldg4_f(up);
      *reinterpret_cast<float4*>(vv) = ldg4_f(vp);
      *reinterpret_cast<float4*>(ll) = __ldg(reinterpret_cast<const float4*>(P.lon + x));
    } else {
#pragma unroll
      for (int k = 0; k < VEC; ++k) { uu[k] = ldg_f(up + k); vv[k] = ldg_f(vp + k); ll[k] = __ldg(P.lon + x + k); }
    }
    const T* f = nullptr;
    float mean0 = 0.0f, mean1 = 0.0f;
    if (own) {
      f = plane_ptr_bc(as<T>(P.field), P.field_sB, b, c, P.fldN, P.W);
      const float* gp = arr_row<PEER>(P, plane_ptr_bc(P.gout, P.gout_sB, b, c, P.uvgN, P.W), 2, pl, y) + x;
      if (VEC == 4) *reinterpret_cast<float4*>(gg) = __ldg(reinterpret_cast<const float4*>(gp));
      else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) gg[k] = __ldg(gp + k);
      }
      if (P.pole_fix) {
        mean0 = __ldg(P.fmean + 2 * pl); mean1 = __ldg(P.fmean + 2 * pl + 1);
        if (y == 0 || y == P.H - 1) {  // adjoint of the output pole mean
          const float gm = __ldg(P.gmean + 2 * pl + (y == 0 ? 0 : 1));
#pragma unroll
          for (int k = 0; k < VEC; ++k) gg[k] = gm;
        }
      }
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      Traj t;
      trajectory<EXACT>(P, uu[k], vv[k], sp, cp, ll[k], t);
      int rc = (int)floorf(t.iy) - (y + P.p);
      const int ac = abs(rc);
      if (ac > PARADIS_SL_MAX_DISP_ROWS) {
        if (P.status) *P.status = PARADIS_ERR_DISPLACEMENT;
        rc = rc > 0 ? 127 : -127;
      }
      reach = max(reach, min(ac, 127));
      cc[k] = (signed char)rc;
      if (own) {
        float val, dx, dy;
        stencil_eval<INTERP, true, PEER>(P, f, pl, t, mean0, mean1, val, dx, dy);
        velocity_grads<EXACT>(P, t, sp, cp, gg[k] * dx, gg[k] * dy, ou[k], ov[k]);
      }
    }
    if (P.cls) {
      signed char* cp8 = P.cls + ((long long)pl * P.arrN + (y - P.arr0)) * P.W + x;
      if (VEC == 4) *reinterpret_cast<char4*>(cp8) = make_char4(cc[0], cc[1], cc[2], cc[3]);
      else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) cp8[k] = cc[k];
      }
    }
    if (own) {
      const long long ooff = ((long long)pl * P.ownN + (y - P.own0)) * P.W + x;
      if (VEC == 4) {
        stcs4_f(as<T>(P.gu) + ooff, *reinterpret_cast<float4*>(ou));
        stcs4_f(as<T>(P.gv) + ooff, *reinterpret_cast<float4*>(ov));
      } else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) { stcs_f(as<T>(P.gu) + ooff + k, ou[k]); stcs_f(as<T>(P.gv) + ooff + k, ov[k]); }
      }
    }
  }
  if (P.blkmax) {  // per-block maximum, no atomics: warp max -> smem -> thread 0
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

__global__ void plane_reach_kernel(const unsigned char* __restrict__ blkmax, int nblk, int planes,
                                   int* __restrict__ plane_reach, const unsigned char* __restrict__ filter,
                                   unsigned char* __restrict__ flag, int limit) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= planes) return;
  if (filter && !filter[warp]) return;
  int m = 0;
  for (int i = lane; i < nblk; i += 32) m = max(m, (int)blkmax[(long long)warp * nblk + i]);
  m = __reduce_max_sync(0xffffffffu, m);
  if (lane == 0) {
    plane_reach[warp] = m;
    if (flag && m > limit) flag[warp] = 1;   // contract of the fused sweep violated by this plane
  }
}

// ---------------------------------------------------------------------------------------------
// backward, grad_field: gather over inverse stencils.
//
// One warp owns one output row (plane, r) and a private accumulator acc[W] in shared memory.
// It visits, in a fixed order, every padded destination row Rd that folds onto r through the
// GeoCyclic map (r itself, plus a reflected cap row when r is within p rows of a pole).  For each
// Rd it scans the row classes of the arrival rows that can reach Rd, compacts the matching arrival
// points (ballot/popc, raster order) into a small queue and, 32 at a time, recomputes their
// trajectory and adds their weights into acc.  Lanes that hit the same column are combined in lane
// order by the lowest lane (match_any + shuffles), so every add into acc has a single writer and a
// data-independent order: deterministic, no atomics.
// ---------------------------------------------------------------------------------------------
constexpr int kGatherWarps = 8;
constexpr int kScan = 8;     // class bytes examined per lane and scan step
constexpr int kQueue = 32 * kScan + 32;  // >= 31 left over + 32 * kScan new entries

template <typename T>
struct GatherPlane { const T* __restrict__ u; const T* __restrict__ v; const float* __restrict__ g; float gm0, gm1; int pl; };

template <bool EXACT, int INTERP, bool PEER, typename T>
__device__ __forceinline__ void gather_chunk(const Params& P, const GatherPlane<T>& G, int Rd, int shift, float* acc,
                                             const unsigned* queue, int n, int lane) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  float c[NT];
#pragma unroll
  for (int b = 0; b < NT; ++b) c[b] = 0.0f;
  int key = -1 - lane;  // idle lanes: unique keys, zero contributions
  int xb = 0;
  if (lane < n) {
    const unsigned e = queue[lane];
    const int y = (int)(e >> 16), x = (int)(e & 0xffffu);  // global arrival row, column
    const float uu = ldg_f(arr_row<PEER>(P, G.u, 0, G.pl, y) + x), vv = ldg_f(arr_row<PEER>(P, G.v, 1, G.pl, y) + x);
    float g = __ldg(arr_row<PEER>(P, G.g, 2, G.pl, y) + x);
    if (P.pole_fix) {                         // adjoint of the output pole mean
      if (y == 0) g = G.gm0;
      else if (y == P.H - 1) g = G.gm1;
    }
    Traj t;
    trajectory<EXACT>(P, uu, vv, __ldg(P.sin_lat + y), __ldg(P.cos_lat + y), __ldg(P.lon + x), t);
    const float fx = floorf(t.ix), fy = floorf(t.iy);
    const float tx = __fsub_rn(t.ix, fx), ty = __fsub_rn(t.iy, fy);
    const int a = Rd - ((int)fy + OMIN);  // which y-tap of this point lands on Rd
    if (a >= 0 && a < NT) {
      float wx[NT], wy[NT], d0[NT], d1[NT];
      axis_weights<INTERP, false>(tx, wx, d0);
      axis_weights<INTERP, false>(ty, wy, d1);
      float wya = wy[0];
#pragma unroll
      for (int k = 1; k < NT; ++k) wya = (a == k) ? wy[k] : wya;
      const float val = g * wya;
      xb = (int)fx + OMIN;  // padded column of tap 0
#pragma unroll
      for (int b = 0; b < NT; ++b) c[b] = ((unsigned)(xb + b) < (unsigned)P.Wp) ? val * wx[b] : 0.0f;
      // fold the column through the GeoCyclic map once, at the key level
      int j = xb - P.p - shift;  // in [-p - 1 - W/2, W + p) for any finite trajectory
      if (j < 0) j += P.W;
      else if (j >= P.W) j -= P.W;
      if ((unsigned)j < (unsigned)P.W) key = j;
      else {
#pragma unroll
        for (int b = 0; b < NT; ++b) c[b] = 0.0f;  // non-finite coordinates: every tap is out of bounds
      }
    }
  }
  // combine lanes with the same base column, ascending lane order, lowest lane writes
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  const int leader = __ffs(peers) - 1;
  const int npeer = __popc(peers);
  const int nmax = __reduce_max_sync(0xffffffffu, npeer);
  unsigned rest = peers & (peers - 1);  // peers without the leader
  for (int rr = 1; rr < nmax; ++rr) {
    const int src = rest ? __ffs(rest) - 1 : lane;
    const bool take = (lane == leader) && rest;
    rest &= rest - 1;
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      const float o = __shfl_sync(0xffffffffu, c[b], src);
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

template <bool EXACT, int INTERP, bool PEER, typename T>
__global__ void __launch_bounds__(kGatherWarps * 32) sl_bwd_gather_kernel(const Params P) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pl = blockIdx.y;
  if (P.plane_filter && !P.plane_filter[pl]) return;
  const int lr = blockIdx.x * kGatherWarps + warp;  // row within the iteration window
  if (lr >= P.it_ownN) return;
  const int r = P.it_own0 + lr;                      // global output row
  float* acc = smem + (size_t)warp * (P.W + kQueue);
  unsigned* queue = reinterpret_cast<unsigned*>(acc + P.W);
  for (int x = lane; x < P.W; x += 32) acc[x] = 0.0f;
  __syncwarp();
  const int reach = P.plane_reach[pl];
  const signed char* cls = P.cls + (long long)pl * P.arrN * P.W;
  GatherPlane<T> G;
  G.pl = pl;
  G.u = plane_ptr(as<T>(P.u), P.u_sB, P.V, P.uvgN, P.W, pl);
  G.v = plane_ptr(as<T>(P.v), P.v_sB, P.V, P.uvgN, P.W, pl);
  G.g = plane_ptr(P.gout, P.gout_sB, P.V, P.uvgN, P.W, pl);
  G.gm0 = G.gm1 = 0.0f;
  if (P.pole_fix) { G.gm0 = __ldg(P.gmean + 2 * pl); G.gm1 = __ldg(P.gmean + 2 * pl + 1); }

  // destination rows (padded coordinates) folding onto r: itself, north cap, south cap
  for (int src = 0; src < 3; ++src) {
    int Rd, shift;
    if (src == 0) { Rd = r + P.p; shift = 0; }
    else if (src == 1) { if (r < 1 || r > P.p) continue; Rd = P.p - r; shift = P.halfW; }
    else { const int i = 2 * (P.H - 1) - r; if (i < P.H || i >= P.H + P.p) continue; Rd = i + P.p; shift = P.halfW; }
    // arrival rows y with floor(iy) + OMIN <= Rd <= floor(iy) + OMIN + NT - 1, floor(iy) = y + p + class
    int ylo = Rd - P.p - (OMIN + NT - 1) - reach, yhi = Rd - P.p - OMIN + reach;
    ylo = max(ylo, P.it_arr0); yhi = min(yhi, P.it_arr0 + P.it_arrN - 1);
    int qn = 0;
    for (int y = ylo; y <= yhi; ++y) {
      const signed char* crow = cls + (long long)(y - P.arr0) * P.W;
      const int cbase = Rd - (y + P.p) - OMIN;  // tap index a = cbase - class must be in [0, NT)
      // byte patterns of the NT matching classes (0x80 = -128 is never stored: no match)
      unsigned pat[NT];
#pragma unroll
      for (int a = 0; a < NT; ++a) {
        const int cv = cbase - a;
        pat[a] = ((cv >= -127 && cv <= 127) ? (unsigned)(cv & 0xff) : 0x80u) * 0x01010101u;
      }
      for (int x0 = 0; x0 < P.W; x0 += kScan * 32) {
        const int x = x0 + lane * kScan;
        unsigned m = 0;                      // bit k: candidate x + k matches
        if (x + kScan - 1 < P.W && (P.W & (kScan - 1)) == 0) {
          const uint2 q = *reinterpret_cast<const uint2*>(crow + x);
          unsigned e0 = 0, e1 = 0;
#pragma unroll
          for (int a = 0; a < NT; ++a) { e0 |= __vcmpeq4(q.x, pat[a]); e1 |= __vcmpeq4(q.y, pat[a]); }
          // one bit per byte: 0xFF bytes -> bits 0..3
          m = (((e0 & 0x01010101u) * 0x01020408u) >> 24) | ((((e1 & 0x01010101u) * 0x01020408u) >> 24) << 4);
        } else {
#pragma unroll
          for (int k = 0; k < kScan; ++k)
            if (x + k < P.W && (unsigned)(cbase - crow[x + k]) < (unsigned)NT) m |= 1u << k;
        }
        // raster-order compaction: exclusive prefix of the per-lane counts, then the lane's own bits in order
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
          gather_chunk<EXACT, INTERP, PEER>(P, G, Rd, shift, acc, queue + head, 32, lane);
          head += 32;
        }
        if (head) {  // move the tail (< 32 entries) to the front
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
    if (qn) gather_chunk<EXACT, INTERP, PEER>(P, G, Rd, shift, acc, queue, qn, lane);
  }
  // adjoint of the first enforce_pole_continuity (advection.py:129): pole rows get their mean
  float* orow = P.gfield + ((long long)pl * P.ownN + (r - P.own0)) * P.W;
  if (P.pole_fix && (r == 0 || r == P.H - 1)) {
    const float m = warp_row_sum(acc, P.W, lane) / (float)P.W;
    for (int x = lane; x < P.W; x += 32) orow[x] = m;
  } else {
    for (int x = lane; x < P.W; x += 32) orow[x] = acc[x];
  }
}

// ---------------------------------------------------------------------------------------------
// standalone GeoCyclic padding (model/padding.py:11-39) and its adjoint
// ---------------------------------------------------------------------------------------------
// T = storage type of x / y (fp32 or bf16).  The bf16 forward copies the 2-byte words as they are, two padded columns
// per thread and one 4-byte store (Wp and every row start are even).
template <typename T>
__global__ void geocyclic_pad_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int H, int W, int p) {
  const int Hp = H + 2 * p, Wp = W + 2 * p;
  const long long pl = blockIdx.z;
  const int R = blockIdx.y;
  int i = R - p, shift = 0;
  if (i < 0) { i = -i; shift = W / 2; }
  else if (i >= H) { i = 2 * (H - 1) - i; shift = W / 2; }
  const T* src = x + (pl * H + i) * W;
  T* dst = y + (pl * Hp + R) * Wp;
  if constexpr (kIsF32<T>) {
    for (int C = blockIdx.x * blockDim.x + threadIdx.x; C < Wp; C += gridDim.x * blockDim.x) {
      int j = C - p - shift;
      if (j < 0) j += W; else if (j >= W) j -= W;
      dst[C] = __ldg(src + j);
    }
  } else {
    const unsigned short* s16 = reinterpret_cast<const unsigned short*>(src);
    for (int C = 2 * (blockIdx.x * blockDim.x + threadIdx.x); C < Wp; C += 2 * gridDim.x * blockDim.x) {
      int j = C - p - shift;
      if (j < 0) j += W; else if (j >= W) j -= W;
      const int j1 = j + 1 == W ? 0 : j + 1;
      *reinterpret_cast<unsigned*>(dst + C) = (unsigned)__ldg(s16 + j) | ((unsigned)__ldg(s16 + j1) << 16);
    }
  }
}

// gx[i, j] = sum of every padded cell whose source is (i, j); fixed order: interior row first,
// then north cap, then south cap; within a row: centre, left wrap, right wrap.  fp32 sums for either storage type,
// one rounding per bf16 output.
template <typename T>
__global__ void geocyclic_pad_bwd_kernel(const T* __restrict__ gy, T* __restrict__ gx, int H, int W, int p) {
  const int Hp = H + 2 * p, Wp = W + 2 * p;
  const long long pl = blockIdx.z;
  const int i = blockIdx.y;
  const T* g = gy + pl * (long long)Hp * Wp;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < W; j += gridDim.x * blockDim.x) {
    float s = 0.0f;
    for (int src = 0; src < 3; ++src) {
      int R, shift;
      if (src == 0) { R = i + p; shift = 0; }
      else if (src == 1) { if (i < 1 || i > p) continue; R = p - i; shift = W / 2; }
      else { const int ii = 2 * (H - 1) - i; if (ii < H || ii >= H + p) continue; R = ii + p; shift = W / 2; }
      // padded columns C with (C - p - shift) mod W == j
      int c = j + shift; if (c >= W) c -= W;   // C - p in [0, W)
      const T* row = g + (long long)R * Wp + p;
      s += ld_f(row + c);
      if (c >= W - p) s += ld_f(row + (c - W));  // left wrap columns  C - p in [-p, 0)
      if (c < p) s += ld_f(row + (c + W));     // right wrap columns C - p in [W, W + p)
    }
    st_f(gx + (pl * H + i) * W + j, s);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
// Points per thread of the forward / arrival kernels.  4 consecutive columns (float4 rows, 4 independent
// trajectories in flight) win for the 4-tap bilinear stencil (0.43 vs 0.59 ms at C3); the 16-tap bicubic
// stencil is bound by its gathers and wants one point per lane -- consecutive lanes hit consecutive
// addresses (few sectors per request) and 32 registers give full occupancy (0.97 vs 1.89 ms at C3).
static int points_per_thread(int interp, bool vec_ok) {
  if (!vec_ok) return 1;
  return interp == PARADIS_INTERP_BICUBIC ? 1 : 4;
}

static int fill_params(Params& P, const paradis_sl_geom* g, int B, int V, float dt, int interp, int pole_fix) {
  if (!g) return fail(PARADIS_ERR_NULL_POINTER, "geom is NULL");
  if (!g->sin_lat || !g->cos_lat || !g->lon) return fail(PARADIS_ERR_NULL_POINTER, "geom tables are NULL");
  if (interp != PARADIS_INTERP_BILINEAR && interp != PARADIS_INTERP_BICUBIC)
    return fail(PARADIS_ERR_BAD_INTERP, "interp must be 1 (bilinear) or 2 (bicubic), got %d", interp);
  const int p = interp;
  if (B <= 0 || V <= 0 || g->H <= 0 || g->W <= 0) return fail(PARADIS_ERR_BAD_SHAPE, "non-positive dimension");
  if (g->W % 2) return fail(PARADIS_ERR_ODD_WIDTH, "Number of longitude points must be even (W=%d)", g->W);
  if (g->H < p + 2) return fail(PARADIS_ERR_BAD_SHAPE, "H=%d too small for padding %d", g->H, p);
  if (g->H > 65535 || g->W > 65535) return fail(PARADIS_ERR_BAD_SHAPE, "mesh larger than 65535 not supported");
  if ((long long)B * V > 65535) return fail(PARADIS_ERR_BAD_SHAPE, "B*V=%lld exceeds 65535 planes per call", (long long)B * V);
  auto inside = [&](int r0, int n) { return n > 0 && r0 >= 0 && r0 + n <= g->H; };
  if (!inside(g->own_row0, g->own_rows) || !inside(g->arr_row0, g->arr_rows) || !inside(g->fld_row0, g->fld_rows))
    return fail(PARADIS_ERR_BAD_SHAPE, "row window outside the mesh");
  if (g->arr_row0 > g->own_row0 || g->arr_row0 + g->arr_rows < g->own_row0 + g->own_rows)
    return fail(PARADIS_ERR_BAD_SHAPE, "arr window must contain own window");
  memset(&P, 0, sizeof(P));
  P.H = g->H; P.W = g->W; P.p = p; P.Hp = g->H + 2 * p; P.Wp = g->W + 2 * p; P.halfW = g->W / 2;
  P.own0 = g->own_row0; P.ownN = g->own_rows; P.arr0 = g->arr_row0; P.arrN = g->arr_rows;
  P.fld0 = g->fld_row0; P.fldN = g->fld_rows;
  if (g->fld_peer_rows > 0 && (g->fld_peer_lo || g->fld_peer_hi)) {
    P.f_lo = g->fld_peer_lo; P.f_hi = g->fld_peer_hi; P.f_halo = g->fld_peer_rows;
  }
  P.it_own0 = P.own0; P.it_ownN = P.ownN; P.it_arr0 = P.arr0; P.it_arrN = P.arrN;
  P.uvg0 = P.arr0; P.uvgN = P.arrN;
  if (g->arr_peer_rows > 0) {
    const int h = g->arr_peer_rows;
    const bool lo = g->arr_peer_lo[0] != nullptr, hi = g->arr_peer_hi[0] != nullptr;
    for (int k = 0; k < 3; ++k) {
      if ((g->arr_peer_lo[k] != nullptr) != lo || (g->arr_peer_hi[k] != nullptr) != hi)
        return fail(PARADIS_ERR_NULL_POINTER, "arr_peer_lo / arr_peer_hi must be given for u, v and grad_out alike");
      P.a_lo[k] = g->arr_peer_lo[k]; P.a_hi[k] = g->arr_peer_hi[k];
    }
    if (lo || hi) {
      P.a_halo = h;
      P.uvg0 = P.arr0 + (lo ? h : 0);
      P.uvgN = P.arrN - (lo ? h : 0) - (hi ? h : 0);
      if (P.uvgN <= 0) return fail(PARADIS_ERR_BAD_SHAPE, "arr window smaller than its peer halos");
    }
  }
  P.sin_lat = g->sin_lat; P.cos_lat = g->cos_lat; P.lon = g->lon;
  P.min_lat = g->min_lat; P.d_lat = g->d_lat; P.min_lon = g->min_lon; P.d_lon = g->d_lon;
  P.dt = dt;
  P.Wm1 = (float)g->W - 1.0f; P.Hm1 = (float)g->H - 1.0f;
  P.Wpm1 = (float)(P.Wp - 1); P.Hpm1 = (float)(P.Hp - 1); P.pf = (float)p;
  P.inv_Wpm1 = 1.0f / P.Wpm1; P.inv_Hpm1 = 1.0f / P.Hpm1;
  P.Ax = P.Wm1 / g->d_lon; P.Ay = P.Hm1 / g->d_lat;
  P.Cx = (float)((double)p - (double)g->min_lon * (double)P.Ax);
  P.Cy = (float)((double)p - (double)g->min_lat * (double)P.Ay);
  P.clamp_lo = (float)(-1 + 1e-7); P.clamp_hi = (float)(1 - 1e-7);
  P.Wf = (float)g->W; P.ix_wrap = (float)(g->W + p);
  P.B = B; P.V = V; P.pole_fix = pole_fix ? 1 : 0;
  {  // rows (global, of tap row 0) whose whole stencil is plain field data inside the window
    const int nt = interp == 1 ? 2 : 4;
    const int lo = P.fld0 > (pole_fix ? 1 : 0) ? P.fld0 : (pole_fix ? 1 : 0);
    const int top = (P.fld0 + P.fldN - 1) < (pole_fix ? P.H - 2 : P.H - 1) ? (P.fld0 + P.fldN - 1) : (pole_fix ? P.H - 2 : P.H - 1);
    const int hi = top - (nt - 1);
    if (hi >= lo && P.W >= nt) { P.fast_y0 = lo; P.fast_yspan = hi - lo; }
    else { P.fast_y0 = 1 << 30; P.fast_yspan = 0; }
  }
  return PARADIS_OK;
}

static void set_units(Params& P, int vec, int rows) {
  P.upr = P.W / vec;
  P.w4_mul = 0; P.w4_shift = 0;
  // n / upr == umulhi(n, ceil(2^32 / upr)) for n * upr < 2^32
  const unsigned long long n_max = (unsigned long long)rows * P.upr;
  if (P.upr > 1 && n_max * P.upr < (1ull << 32)) P.w4_mul = (unsigned)(((1ull << 32) + P.upr - 1) / P.upr);
}

static bool aligned16(const void* ptr) { return ((uintptr_t)ptr & 15u) == 0; }

extern "C" size_t paradis_sl_advect_fwd_workspace(int B, int V) {
  return align_up((size_t)B * V * 2 * sizeof(float), 256);
}

// Peer halos are fp32 (latitude bands): the bf16 instantiations take the PEER = false kernel for both branches.
template <bool EXACT, int INTERP, typename T>
static void launch_fwd(const Params& P, int vec, dim3 grid, cudaStream_t st) {
  constexpr bool kPeer = kIsF32<T>;
  const bool peer = P.f_halo > 0;
  if (vec == 4) {
    if (peer) sl_fwd_kernel<EXACT, INTERP, 4, kPeer, T><<<grid, 256, 0, st>>>(P);
    else sl_fwd_kernel<EXACT, INTERP, 4, false, T><<<grid, 256, 0, st>>>(P);
  } else {
    if (peer) sl_fwd_kernel<EXACT, INTERP, 1, kPeer, T><<<grid, 256, 0, st>>>(P);
    else sl_fwd_kernel<EXACT, INTERP, 1, false, T><<<grid, 256, 0, st>>>(P);
  }
}

// Forward of either storage type once the arguments are checked; `field`, `u`, `v` hold T.
template <typename T>
static int advect_fwd(Params& P, const void* field, const void* u, const void* v, float* out, int B, int V,
                      int64_t field_sB, int64_t u_sB, int64_t v_sB, int interp, int pole_fix, int math, void* workspace,
                      size_t workspace_bytes, int32_t* status, cudaStream_t st) {
  const int planes = B * V;
  P.field = (const float*)field; P.u = (const float*)u; P.v = (const float*)v; P.out = out;
  P.field_sB = field_sB; P.u_sB = u_sB; P.v_sB = v_sB;
  P.status = status;
  if (pole_fix) {
    if (!workspace || workspace_bytes < paradis_sl_advect_fwd_workspace(B, V))
      return fail(PARADIS_ERR_WORKSPACE, "forward workspace too small (%zu bytes)", workspace_bytes);
    float* fmean = (float*)workspace;
    P.fmean = fmean;
    pole_means_kernel<T><<<planes * 2, kPoleThreads, 0, st>>>((const T*)field, field_sB, V, P.fldN, P.fld0, P.H, P.W, planes,
                                                               fmean, nullptr, 0, 0, 0, nullptr);
  }
  const bool vec_ok = (P.W % 4 == 0) && aligned16(field) && aligned16(u) && aligned16(v) && aligned16(out) &&
                      aligned16(P.lon) && (u_sB % 4 == 0) && (v_sB % 4 == 0);
  const int vec = points_per_thread(interp, vec_ok);
  set_units(P, vec, P.ownN);
  const unsigned units = (unsigned)P.ownN * P.upr;
  dim3 grid((units + 255) / 256, V, B);
  const bool exact = math == PARADIS_MATH_EXACT;
  if (interp == 1) { if (exact) launch_fwd<true, 1, T>(P, vec, grid, st); else launch_fwd<false, 1, T>(P, vec, grid, st); }
  else             { if (exact) launch_fwd<true, 2, T>(P, vec, grid, st); else launch_fwd<false, 2, T>(P, vec, grid, st); }
  if (pole_fix) pole_rows_fix_kernel<<<planes * 2, kPoleThreads, 0, st>>>(out, P.ownN, P.own0, P.H, P.W, planes);
  return PARADIS_OK;
}

extern "C" int paradis_sl_advect_fwd(const paradis_sl_geom* geom, const float* field, const float* u,
                                     const float* v, float* out, int B, int V, int64_t field_sB, int64_t u_sB,
                                     int64_t v_sB, float dt, int interp, int pole_fix, int math, void* workspace,
                                     size_t workspace_bytes, int32_t* status, void* stream) {
  Params P;
  if (int rc = fill_params(P, geom, B, V, dt, interp, pole_fix)) return rc;
  if (!field || !u || !v || !out) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if (int rc = advect_fwd<float>(P, field, u, v, out, B, V, field_sB, u_sB, v_sB, interp, pole_fix, math, workspace,
                                 workspace_bytes, status, (cudaStream_t)stream))
    return rc;
  return check_launch("paradis_sl_advect_fwd");
}

// workspace layout (backward): fmean | gmean | plane_reach[3] | plane_flag | hx | guard | blkmax[3] | cls
// (three reach / blkmax sets: the two polar caps run concurrently with the sweep, then the fallback)
struct BwdWs { size_t fmean, gmean, reach, reach_stride, flag, hx, guard, grow, grow_bytes, blkmax, blkmax_stride, cls, total; int nblk; };
constexpr int kRowsMaxGuardRows = 14;   // cut mode of the rows kernel up to rr + NT = 14 (cfl hint <= 10 cells)
static BwdWs bwd_layout(int B, int V, int arr_rows, int W) {
  BwdWs w;
  const size_t planes = (size_t)B * V;
  // blocks per plane of the arrival kernel in the worst case (VEC = 1)
  w.nblk = (int)(((size_t)arr_rows * W + 255) / 256);
  size_t off = 0;
  w.fmean = off; off += align_up(planes * 2 * sizeof(float), 256);
  w.gmean = off; off += align_up(planes * 2 * sizeof(float), 256);
  w.reach_stride = align_up(planes * sizeof(int), 256);
  w.reach = off; off += 3 * w.reach_stride;
  w.flag = off; off += align_up(planes, 256);
  w.hx = off; off += 65536 * sizeof(int);          // longitudinal reach per arrival row (rows kernel)
  // guard columns of the rows kernel: [planes][rows][strips][NT - 1], sized for kRowsWarps strips and NT = 4
  w.guard = off; off += align_up(planes * (size_t)arr_rows * kRowsWarps * 3 * sizeof(float), 256);
  // partial destination rows either side of the cuts of the rows kernel: [CTAs][2][GR][strips * pitch]
  w.grow_bytes = align_up((size_t)kRowsMaxCtas * 2 * kRowsMaxGuardRows * ((size_t)W + 256) * sizeof(float), 256);
  w.grow = off; off += w.grow_bytes;
  w.blkmax_stride = align_up(planes * (size_t)w.nblk, 256);
  w.blkmax = off; off += 3 * w.blkmax_stride;
  w.cls = off; off += align_up(planes * (size_t)arr_rows * W, 256);
  w.total = off;
  return w;
}

extern "C" size_t paradis_sl_advect_bwd_workspace(int B, int V, int arr_rows, int W) {
  return bwd_layout(B, V, arr_rows, W).total;
}

// General (two-kernel) backward over the iteration windows set in P.
template <bool EXACT, int INTERP, typename T>
static int launch_general(Params P, int vec, cudaStream_t st, bool want_field, int phases, int max_nblk) {
  constexpr bool kPeer = kIsF32<T>;   // see launch_fwd
  const int planes = P.B * P.V;
  // the filtered (fallback) launch mostly consists of blocks that exit at once: keep their number small
  vec = (P.plane_filter && vec == 4) ? 4 : points_per_thread(INTERP, vec == 4);
  set_units(P, vec, P.it_arrN);
  const unsigned units = (unsigned)P.it_arrN * P.upr;
  dim3 grid((units + 255) / 256, P.V, P.B);
  if (P.plane_filter && grid.x > 8) grid.x = 8;       // see the grid-stride loop of the arrival kernel
  if ((int)grid.x > max_nblk) return fail(PARADIS_ERR_WORKSPACE, "internal: blkmax layout");
  P.nblk = grid.x;
  if (phases & PARADIS_BWD_ARRIVAL) {
    const bool peer = P.f_halo > 0 || P.a_halo > 0;
    if (vec == 4) {
      if (peer) sl_bwd_arrival_kernel<EXACT, INTERP, 4, kPeer, T><<<grid, 256, 0, st>>>(P);
      else sl_bwd_arrival_kernel<EXACT, INTERP, 4, false, T><<<grid, 256, 0, st>>>(P);
    } else {
      if (peer) sl_bwd_arrival_kernel<EXACT, INTERP, 1, kPeer, T><<<grid, 256, 0, st>>>(P);
      else sl_bwd_arrival_kernel<EXACT, INTERP, 1, false, T><<<grid, 256, 0, st>>>(P);
    }
    if (want_field)
      plane_reach_kernel<<<(planes * 32 + 255) / 256, 256, 0, st>>>(P.blkmax, P.nblk, planes, P.plane_reach,
                                                                   P.plane_filter, P.plane_flag, P.reach_limit);
  }
  if (!want_field || !(phases & PARADIS_BWD_GATHER)) return PARADIS_OK;
  const size_t smem = (size_t)kGatherWarps * (P.W + kQueue) * sizeof(float);
  if (smem > 227 * 1024) return fail(PARADIS_ERR_BAD_SHAPE, "W=%d too wide for the gather kernel's shared memory", P.W);
  auto kern = P.a_halo > 0 ? sl_bwd_gather_kernel<EXACT, INTERP, kPeer, T> : sl_bwd_gather_kernel<EXACT, INTERP, false, T>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return fail(PARADIS_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  dim3 ggrid((P.it_ownN + kGatherWarps - 1) / kGatherWarps, planes);
  kern<<<ggrid, kGatherWarps * 32, smem, st>>>(P);
  return PARADIS_OK;
}

// ---- plan of the fused sweep -------------------------------------------------------------------
// cfl_cells bounds the great-circle displacement |(u, v)| * dt in units of the latitude spacing.
// From it: the row reach rr, and per arrival row the longitudinal reach in cells (it grows as
// 1 / cos(lat), see halo_cells()).  Destination rows all of whose arrival rows have a reach of at
// most kSweepMaxHalo{2,4} are swept; they are cut into bands of equal cost, enough of them to fill the
// GPU about once.
// Longest halo (cells either side of a strip) a swept row may need; rows poleward of it go to the general path.
// Recomputing a wide halo costs the 2x2 stencil as much as the general path does (measured: 32 best), while the
// general path visits every arrival point four times for the 4x4 stencil (96: 3.98 -> 3.83 ms backward).
constexpr int kSweepMaxHalo2 = 32, kSweepMaxHalo4 = 96;
constexpr int kSweepStrip = 128;

template <int INTERP>
static bool plan_sweep(const Params& P, float cfl_cells, int planes, int capacity_warps, SweepPlan& S, int& lo,
                       int& hi) {
  constexpr int NT = Stencil<INTERP>::NT;
  const int H = P.H, W = P.W, wc = kSweepStrip;
  if (!(cfl_cells > 0.0f) || H < 8) return false;
  const double dphi = (double)P.d_lat / (H - 1), dlam = (double)P.d_lon / (W - 1);
  const double delta = (double)cfl_cells * dphi;
  const int rr = (int)ceil((double)cfl_cells);
  if (rr > 40 || delta > 0.7) return false;
  const int yh = rr + NT;                      // arrival rows either side that can reach a destination row
  S.reach.sin_delta = (float)sin(delta); S.reach.cos_delta = (float)cos(delta);
  S.reach.inv_dlam = (float)(1.0 / dlam); S.reach.extra = NT + 2;
  S.reach.max_halo = NT == 2 ? kSweepMaxHalo2 : kSweepMaxHalo4;
  while (wc + 2 * (S.reach.max_halo + 16) > W && S.reach.max_halo > 16) S.reach.max_halo -= 16;
  if (wc + 2 * (S.reach.max_halo + 16) > W) return false;
  std::vector<int> need(H);
  for (int y = 0; y < H; ++y) {
    const double lat = (double)P.min_lat + y * dphi;
    need[y] = halo_cells(S.reach, (float)sin(lat), (float)cos(lat));
  }
  // a destination row is sweepable if every arrival row that can reach it fits the halo limit with a
  // margin of one 16-column step (the device re-evaluates halo_cells from its own fp32 tables)
  std::vector<char> okrow(H, 0);
  for (int i = yh + 1; i < H - yh - 1; ++i) {
    int n = 0;
    for (int y = i - yh; y <= i + yh; ++y) n = n > need[y] ? n : need[y];
    okrow[i] = n <= S.reach.max_halo;
  }
  const int own_lo = P.own0, own_hi = P.own0 + P.ownN;
  lo = hi = -1;
  {
    int best = 0, start = -1;
    for (int i = own_lo; i <= own_hi; ++i) {
      const bool ok = i < own_hi && okrow[i];
      if (ok && start < 0) start = i;
      if (!ok && start >= 0) {
        if (i - start > best) { best = i - start; lo = start; hi = i; }
        start = -1;
      }
    }
    if (best < 4 * yh) return false;           // not worth a sweep
  }
  const int nstrips = (W + wc - 1) / wc;
  const int ncore = wc / 32;
  auto row_cost = [&](int y) { return (double)(ncore + (2 * (need[y] < 1024 ? need[y] : 1024) + 31) / 32); };
  double total = 0.0;
  for (int i = lo; i < hi; ++i) total += row_cost(i);
  int nb = capacity_warps / (planes * nstrips);  // bands so that all tasks are resident at once
  if (nb < 1) nb = 1;
  while (nb > 1 && (hi - lo) / nb < 4 * yh) --nb;  // keep the row halo a minor cost
  if (nb > kMaxBands) nb = kMaxBands;
  S.nbands = nb;
  {
    int i = lo; double accum = 0.0;
    for (int k = 0; k < nb; ++k) {
      S.ra[k] = i;
      const double goal = total * (k + 1) / nb;
      while (i < hi && (accum + row_cost(i) <= goal || i == S.ra[k])) { accum += row_cost(i); ++i; }
      if (k == nb - 1) i = hi;
      S.rb[k] = i;
    }
  }
  S.nstrips = nstrips; S.wc = wc; S.rr = rr; S.ring = 2 * rr + NT; S.pitch = sweep_pitch(wc);
  S.planes = planes;
  return true;
}


// ---- plan + launch of the warp-specialised row sweep (sl_rows.cuh) -------------------------------
// hx_tab[y] = longitudinal reach of arrival row y in cells (1 << 20: unbounded, scan the whole circle); also clears
// the per-plane contract flags.  One tiny launch in front of the sweep.
__global__ void rows_prep_kernel(const float* __restrict__ sin_lat, const float* __restrict__ cos_lat, int H,
                                 ReachModel reach, int* __restrict__ hx_tab, unsigned char* __restrict__ flag, int planes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < H) hx_tab[i] = halo_cells(reach, sin_lat[i], cos_lat[i]);
  if (i < planes) flag[i] = 0;
}

template <bool EXACT, int INTERP, typename T>
static bool launch_rows(const Params& P, cudaStream_t st, float cfl_cells, const BwdWs& L, char* ws, bool forced) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  const int H = P.H, W = P.W, planes = P.B * P.V;
  if (!(cfl_cells > 0.0f) || H < 8 || W < 32 || W > 32767) return false;
  const int rr = (int)ceil((double)cfl_cells);
  const double dphi = (double)P.d_lat / (H - 1), dlam = (double)P.d_lon / (W - 1);
  const double delta = (double)cfl_cells * dphi;
  if (rr > 40 || delta > 0.7) return false;
  RowsPlan S;
  memset(&S, 0, sizeof(S));
  S.planes = planes; S.rr = rr; S.ring = 2 * rr + NT;
  // one strip per consumer warp, at least 32 columns wide: 6 consumer warps for the 2x2 stencil (1.58 ms at C3 against
  // 1.69 / 1.63 / 1.71 for 5 / 7 / 8, DESIGN.md section 8), 8 for the 4x4 stencil
  int nS = INTERP == 1 ? 6 : 8;
  int wc = ((W + nS - 1) / nS + 3) & ~3;
  if (wc < 32) wc = 32;
  nS = (W + wc - 1) / wc;
  S.nC = nS; S.nS = nS; S.wc = wc; S.nP = kRowsWarps - 1 - nS;
  if (S.nP < 1) return false;
  S.nsteps = (W + 32 * kStepSub - 1) / (32 * kStepSub);
  // a row is cut into nsteps producer steps and at most kRowRecs rows are in flight: narrow meshes leave most of the
  // producer warps without work (C2, 128x256: 1.27 ms/step against 0.75 for the strip sweep), so they keep the strip sweep
  if (!forced && S.nsteps < 8) return false;
  S.total_rows = planes * P.ownN;
  S.pitch = (wc + NT - 1 + 3) & ~3;
  S.ring_stride = (S.ring + NT - 1) * S.pitch;
  size_t off = (size_t)nS * S.ring_stride * sizeof(float);
  S.off_stage = (unsigned)off; off += (size_t)kRowStages * 3 * W * sizeof(float);   // (bf16 u, v use 2 W bytes each of it)
  S.off_rec = (unsigned)off; off += (size_t)kRowRecs * W * sizeof(float4);
  S.off_tag = (unsigned)off; off += (size_t)nS * kTagBytes;
  S.off_bar = (unsigned)off; off += (2 * kRowStages + 2 * kRowRecs) * sizeof(uint64_t);
  const size_t smem = off;
  if (smem > 227 * 1024) return false;
  auto kern = (P.f_halo > 0 || P.a_halo > 0) ? sl_bwd_rows_kernel<EXACT, INTERP, kIsF32<T>, T> : sl_bwd_rows_kernel<EXACT, INTERP, false, T>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  int dev = 0, nsm = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  ReachModel reach;
  reach.sin_delta = (float)sin(delta); reach.cos_delta = (float)cos(delta);
  reach.inv_dlam = (float)(1.0 / dlam); reach.extra = NT + 2; reach.max_halo = 0;
  int* hx_tab = (int*)(ws + L.hx);
  unsigned char* flag = (unsigned char*)(ws + L.flag);
  const int nprep = H > planes ? H : planes;
  rows_prep_kernel<<<(nprep + 255) / 256, 256, 0, st>>>(P.sin_lat, P.cos_lat, H, reach, hx_tab, flag, planes);
  S.hx_tab = hx_tab; S.plane_flag = flag; S.out0 = P.own0; S.outN = P.ownN;
  S.guard = (float*)(ws + L.guard);
  // one CTA per SM unless that leaves a CTA fewer than ~12 own rows (a ring warm-up is ring - 1 rows).  The floor was 24
  // at first: the 47-row polar band of the 8-way split then ran on 125 of the 148 SMs (backward 0.38 instead of 0.32 ms)
  int grid = S.total_rows / 12;
  if (grid < 1) grid = 1;
  if (grid > nsm) grid = nsm;
  if (grid > kRowsMaxCtas) grid = kRowsMaxCtas;
  // Cut mode (see RowsPlan::cut): on for latitude bands, where a CTA owns few rows and the ring - 1 warm-up rows of
  // every segment weigh most (8-way split of C3: band backward 0.32 / 0.30 -> 0.275 ms); a full mesh gains nothing
  // (1.58 ms either way).
  S.GR = rr + NT;
  S.grow = (float*)(ws + L.grow);
  S.cut = (P.ownN < H && S.GR <= kRowsMaxGuardRows &&
           (size_t)grid * 2 * S.GR * nS * S.pitch * sizeof(float) <= L.grow_bytes) ? 1 : 0;
  rows_partition<INTERP>(P, S, reach, wc, planes, grid);
  kern<<<grid, kRowsWarps * 32, smem, st>>>(P, S);
  {
    const long long nfix = (long long)S.total_rows * nS * (NT - 1);
    rows_guard_fix_kernel<<<(unsigned)((nfix + 255) / 256), 256, 0, st>>>(P.gfield, S.guard, S.total_rows, W, nS, wc, NT - 1);
  }
  if (S.cut) {
    const dim3 fgrid((W / 4 + 127) / 128, S.GR, grid);
    for (int side = 1; side >= 0; --side)
      rows_grow_fix_kernel<<<fgrid, 128, 0, st>>>(P.gfield, S, side, W, P.own0, P.ownN, NT, OMIN);
  }
  if (P.pole_fix) {
    // adjoint of the first enforce_pole_continuity (advection.py:129): pole rows of grad_field get their zonal mean
    pole_rows_fix_kernel<<<planes * 2, kPoleThreads, 0, st>>>(P.gfield, P.ownN, P.own0, H, W, planes);
  }
  return true;
}

// Side streams for the two polar caps (they run beside the sweep, which leaves issue slots idle).
// Created once per host thread and device; fork/join with events, so the call stays asynchronous
// and capturable.  This is the only resource the library keeps between calls.
struct SideStreams { bool ok = false; cudaStream_t s[2]; cudaEvent_t fork, join[2]; };
static SideStreams* side_streams() {
  static thread_local SideStreams ctx[16];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
  SideStreams& c = ctx[dev];
  if (!c.ok) {
    bool good = true;
    for (int i = 0; i < 2; ++i) {
      good = good && cudaStreamCreateWithFlags(&c.s[i], cudaStreamNonBlocking) == cudaSuccess;
      good = good && cudaEventCreateWithFlags(&c.join[i], cudaEventDisableTiming) == cudaSuccess;
    }
    good = good && cudaEventCreateWithFlags(&c.fork, cudaEventDisableTiming) == cudaSuccess;
    if (!good) { cudaGetLastError(); return nullptr; }
    c.ok = true;
  }
  return &c;
}

static int device_capacity(const void* kern, int threads, size_t smem, int& nsm) {
  int dev = 0, blocks = 0;
  nsm = 148;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, kern, threads, smem) != cudaSuccess) return 0;
  return blocks;
}

template <bool EXACT, int INTERP, typename T>
static int launch_bwd(Params P, int vec, cudaStream_t st, int phases, float cfl_cells, const BwdWs& L, char* ws) {
  const bool force_rows = (phases & PARADIS_BWD_ROWSWEEP) != 0;
  phases &= PARADIS_BWD_ALL;
  const bool want_field = P.gfield != nullptr;
  const int planes = P.B * P.V;
  P.plane_filter = nullptr; P.plane_flag = nullptr; P.reach_limit = 1 << 20;
  if (!want_field || phases != PARADIS_BWD_ALL || !(cfl_cells > 0.0f) || vec != 4)   // the sweep needs float4 rows
    return launch_general<EXACT, INTERP, T>(P, vec, st, want_field, phases, L.nblk);

  // ---- warp-specialised row sweep (all latitudes); planes that break its contract fall back below
  // (4x4 stencil: the round-1 strip sweep is still the faster kernel, 3.65 against 4.6 ms at C3; PARADIS_BWD_ROWSWEEP
  // forces the row sweep for it)
  if ((force_rows || INTERP == 1) && launch_rows<EXACT, INTERP, T>(P, st, cfl_cells, L, ws, force_rows)) {
    Params Q = P;
    Q.plane_filter = (unsigned char*)(ws + L.flag);
    Q.gu = nullptr; Q.gv = nullptr;                   // grad_u / grad_v are already complete
    return launch_general<EXACT, INTERP, T>(Q, vec, st, true, PARADIS_BWD_ALL, L.nblk);
  }
  // ---- fused sweep over the mid-latitudes
  constexpr int NT = Stencil<INTERP>::NT;
  SweepPlan S;
  memset(&S, 0, sizeof(S));
  auto kern = (P.f_halo > 0 || P.a_halo > 0) ? sl_bwd_sweep_kernel<EXACT, INTERP, kIsF32<T>, T> : sl_bwd_sweep_kernel<EXACT, INTERP, false, T>;
  const int rr = (int)ceil((double)cfl_cells);
  const size_t smem = (size_t)kSweepWarps * sweep_warp_floats(2 * rr + NT, sweep_pitch(kSweepStrip)) * sizeof(float);
  int lo = -1, hi = -1, nsm = 148;
  bool ok = smem <= 200 * 1024;
  if (ok) ok = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
  int blocks_per_sm = ok ? device_capacity((const void*)kern, kSweepWarps * 32, smem, nsm) : 0;
  ok = ok && blocks_per_sm > 0 && plan_sweep<INTERP>(P, cfl_cells, planes, blocks_per_sm * nsm * kSweepWarps, S, lo, hi);
  if (!ok) {
    cudaGetLastError();
    return launch_general<EXACT, INTERP, T>(P, vec, st, want_field, phases, L.nblk);
  }
  unsigned char* flag = (unsigned char*)(ws + L.flag);
  cudaMemsetAsync(flag, 0, planes, st);
  S.plane_flag = flag; S.out0 = P.own0; S.outN = P.ownN;

  // ---- the caps (rows the sweep does not own): general path on row sub-windows, on side streams
  SideStreams* side = side_streams();
  if (side) cudaEventRecord(side->fork, st);
  // the sweep goes first so that the (smaller) cap kernels fill the issue slots it leaves idle
  const unsigned nblocks = (unsigned)((S.nbands * planes * S.nstrips + kSweepWarps - 1) / kSweepWarps);
  kern<<<nblocks, kSweepWarps * 32, smem, st>>>(P, S);
  const int yh = rr + NT + 1;
  const int own_hi = P.own0 + P.ownN, arr_hi = P.arr0 + P.arrN;
  const int sub[2][2] = {{P.own0, lo}, {hi, own_hi}};
  bool forked[2] = {false, false};
  for (int k = 0; k < 2; ++k) {
    if (sub[k][1] <= sub[k][0]) continue;
    Params Q = P;
    Q.it_own0 = sub[k][0]; Q.it_ownN = sub[k][1] - sub[k][0];
    int a0 = sub[k][0] - yh, a1 = sub[k][1] + yh;
    if (a0 < P.arr0) a0 = P.arr0;
    if (a1 > arr_hi) a1 = arr_hi;
    Q.it_arr0 = a0; Q.it_arrN = a1 - a0;
    Q.plane_flag = flag; Q.reach_limit = rr;       // a cap row reaching further than the contract: redo the plane
    Q.plane_reach = (int*)(ws + L.reach + (k + 1) * L.reach_stride);
    Q.blkmax = (unsigned char*)(ws + L.blkmax + (k + 1) * L.blkmax_stride);
    cudaStream_t cs = st;
    if (side) { cs = side->s[k]; cudaStreamWaitEvent(cs, side->fork, 0); forked[k] = true; }
    if (int rc = launch_general<EXACT, INTERP, T>(Q, vec, cs, true, PARADIS_BWD_ALL, L.nblk)) return rc;
    if (side) cudaEventRecord(side->join[k], cs);
  }
  for (int k = 0; k < 2; ++k)
    if (forked[k]) cudaStreamWaitEvent(st, side->join[k], 0);
  // ---- planes that broke the contract are recomputed entirely by the general path
  Params Q = P;
  Q.plane_filter = flag;
  Q.gu = nullptr; Q.gv = nullptr;                   // grad_u / grad_v are already complete
  return launch_general<EXACT, INTERP, T>(Q, vec, st, true, PARADIS_BWD_ALL, L.nblk);
}

// Backward of either storage type once the arguments are checked; `field`, `u`, `v`, `grad_u`, `grad_v` hold T,
// grad_field is fp32 (the bf16 entry passes its fp32 accumulation buffer).
template <typename T>
static int advect_bwd(Params& P, const BwdWs& L, const float* grad_out, const void* field, const void* u, const void* v,
                      float* grad_field, void* grad_u, void* grad_v, int B, int V, int64_t gout_sB, int64_t field_sB,
                      int64_t u_sB, int64_t v_sB, int interp, int pole_fix, int math, int phases, float cfl_cells,
                      char* ws, int32_t* status, cudaStream_t st) {
  const int planes = B * V;
  float* fmean = (float*)(ws + L.fmean);
  float* gmean = (float*)(ws + L.gmean);
  P.field = (const float*)field; P.u = (const float*)u; P.v = (const float*)v; P.gout = grad_out;
  P.gfield = grad_field; P.gu = (float*)grad_u; P.gv = (float*)grad_v;
  P.field_sB = field_sB; P.u_sB = u_sB; P.v_sB = v_sB; P.gout_sB = gout_sB;
  P.status = status;
  P.fmean = fmean; P.gmean = gmean;
  P.plane_reach = (int*)(ws + L.reach);
  P.blkmax = grad_field ? (unsigned char*)(ws + L.blkmax) : nullptr;
  P.cls = grad_field ? (signed char*)(ws + L.cls) : nullptr;
  P.nblk = L.nblk;
  if (pole_fix && (phases & PARADIS_BWD_ARRIVAL))      // zonal pole means of field and grad_out in one launch
    pole_means_kernel<T><<<planes * 4, kPoleThreads, 0, st>>>((const T*)field, field_sB, V, P.fldN, P.fld0, P.H, P.W, planes,
                                                               fmean, grad_out, gout_sB, P.uvgN, P.uvg0, gmean);
  const bool vec_ok = (P.W % 4 == 0) && aligned16(field) && aligned16(u) && aligned16(v) && aligned16(grad_out) &&
                      aligned16(P.lon) && (!grad_u || (aligned16(grad_u) && aligned16(grad_v))) &&
                      (!grad_field || aligned16(grad_field)) &&   // the sweep retires rows with float4 stores
                      (u_sB % 4 == 0) && (v_sB % 4 == 0) && (gout_sB % 4 == 0);
  const int vec = vec_ok ? 4 : 1;   // float4 rows available (the sweep needs them); the arrival kernel picks its own
  const bool exact = math == PARADIS_MATH_EXACT;
  if (interp == 1)
    return exact ? launch_bwd<true, 1, T>(P, vec, st, phases, cfl_cells, L, ws) : launch_bwd<false, 1, T>(P, vec, st, phases, cfl_cells, L, ws);
  return exact ? launch_bwd<true, 2, T>(P, vec, st, phases, cfl_cells, L, ws) : launch_bwd<false, 2, T>(P, vec, st, phases, cfl_cells, L, ws);
}

extern "C" int paradis_sl_advect_bwd(const paradis_sl_geom* geom, const float* grad_out, const float* field,
                                     const float* u, const float* v, float* grad_field, float* grad_u,
                                     float* grad_v, int B, int V, int64_t gout_sB, int64_t field_sB, int64_t u_sB,
                                     int64_t v_sB, float dt, int interp, int pole_fix, int math, int phases,
                                     float cfl_cells, void* workspace, size_t workspace_bytes, int32_t* status,
                                     void* stream) {
  Params P;
  if (int rc = fill_params(P, geom, B, V, dt, interp, pole_fix)) return rc;
  if (!grad_out || !field || !u || !v) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if ((phases & ~(PARADIS_BWD_ALL | PARADIS_BWD_ROWSWEEP)) || !(phases & PARADIS_BWD_ALL))
    return fail(PARADIS_ERR_BAD_SHAPE, "phases must be 1, 2 or 3 (optionally | PARADIS_BWD_ROWSWEEP)");
  if ((grad_u == nullptr) != (grad_v == nullptr)) return fail(PARADIS_ERR_NULL_POINTER, "grad_u and grad_v must both be given or both be NULL");
  const BwdWs L = bwd_layout(B, V, P.arrN, P.W);
  if (!workspace || workspace_bytes < L.total)
    return fail(PARADIS_ERR_WORKSPACE, "backward workspace too small (%zu < %zu bytes)", workspace_bytes, L.total);
  if (int rc = advect_bwd<float>(P, L, grad_out, field, u, v, grad_field, grad_u, grad_v, B, V, gout_sB, field_sB, u_sB,
                                 v_sB, interp, pole_fix, math, phases, cfl_cells, (char*)workspace, status,
                                 (cudaStream_t)stream))
    return rc;
  return check_launch("paradis_sl_advect_bwd");
}

// ---------------------------------------------------------------------------------------------
// bf16 storage (include/paradis_sl_bf16.h): the same kernels instantiated with T = bf16, same plan
// ---------------------------------------------------------------------------------------------
// grad_field: fp32 accumulation buffer -> bf16, 8 values per thread, rounded once after the last pass that adds to it
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n8) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(src) + 2 * i);
    const float4 b = __ldcs(reinterpret_cast<const float4*>(src) + 2 * i + 1);
    __stcs(reinterpret_cast<uint4*>(dst) + i, make_uint4(f2_to_bf2(a.x, a.y), f2_to_bf2(a.z, a.w), f2_to_bf2(b.x, b.y),
                                                          f2_to_bf2(b.z, b.w)));
  }
}

// Entry points that serve the full mesh only (default windows, no peer halos): PARADIS_ERR_BAD_SHAPE otherwise.
static int full_mesh_check(const paradis_sl_geom* g, const char* who, const char* bands) {
  const int H = g->H;
  if (g->own_row0 != 0 || g->own_rows != H || g->arr_row0 != 0 || g->arr_rows != H || g->fld_row0 != 0 ||
      g->fld_rows != H)
    return fail(PARADIS_ERR_BAD_SHAPE, "%s work on the full mesh (latitude bands: %s)", who, bands);
  bool peers = g->fld_peer_lo || g->fld_peer_hi;
  for (int k = 0; k < 3; ++k) peers = peers || g->arr_peer_lo[k] || g->arr_peer_hi[k];
  if (peers) return fail(PARADIS_ERR_BAD_SHAPE, "%s take no peer halo pointers", who);
  return PARADIS_OK;
}

// Native bf16 path: full mesh only, W % 8 == 0, 16-byte aligned tensors, batch strides in multiples of 8 elements
// (bf16) resp. 4 elements (fp32): every row then starts on 16 bytes.
static int bf16_check(const paradis_sl_geom* g, const void* const* ptrs, int nptrs, const int64_t* sB8, int nsB8,
                      const int64_t* sB4, int nsB4) {
  if (int rc = full_mesh_check(g, "bf16 entry points", "use the fp32 entry points")) return rc;
  if (g->W % 8) return fail(PARADIS_ERR_BAD_SHAPE, "bf16 entry points need W %% 8 == 0 (W=%d)", g->W);
  if (!aligned16(g->lon)) return fail(PARADIS_ERR_BAD_SHAPE, "bf16 entry points need a 16-byte aligned lon table");
  for (int k = 0; k < nptrs; ++k)
    if (ptrs[k] && !aligned16(ptrs[k])) return fail(PARADIS_ERR_BAD_SHAPE, "bf16 entry points need 16-byte aligned tensors");
  for (int k = 0; k < nsB8; ++k)
    if (sB8[k] % 8) return fail(PARADIS_ERR_BAD_SHAPE, "bf16 tensors need batch strides in multiples of 8 elements");
  for (int k = 0; k < nsB4; ++k)
    if (sB4[k] % 4) return fail(PARADIS_ERR_BAD_SHAPE, "grad_out needs a batch stride in multiples of 4 elements");
  return PARADIS_OK;
}

extern "C" int paradis_sl_advect_fwd_bf16(const paradis_sl_geom* geom, const void* field, const void* u, const void* v,
                                          float* out, int B, int V, int64_t field_sB, int64_t u_sB, int64_t v_sB,
                                          float dt, int interp, int pole_fix, int math, void* workspace,
                                          size_t workspace_bytes, int32_t* status, void* stream) {
  Params P;
  if (int rc = fill_params(P, geom, B, V, dt, interp, pole_fix)) return rc;
  if (!field || !u || !v || !out) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  const void* ptrs[4] = {field, u, v, out};
  const int64_t sB8[3] = {field_sB, u_sB, v_sB};
  if (int rc = bf16_check(geom, ptrs, 4, sB8, 3, nullptr, 0)) return rc;
  if (int rc = advect_fwd<bf16>(P, field, u, v, out, B, V, field_sB, u_sB, v_sB, interp, pole_fix, math, workspace,
                                workspace_bytes, status, (cudaStream_t)stream))
    return rc;
  return check_launch("paradis_sl_advect_fwd_bf16");
}

// fp32 workspace of the backward, then the fp32 grad_field accumulation buffer
extern "C" size_t paradis_sl_advect_bwd_bf16_workspace(int B, int V, int arr_rows, int W) {
  return bwd_layout(B, V, arr_rows, W).total + align_up((size_t)B * V * arr_rows * W * sizeof(float), 256);
}

extern "C" int paradis_sl_advect_bwd_bf16(const paradis_sl_geom* geom, const float* grad_out, const void* field,
                                          const void* u, const void* v, void* grad_field, void* grad_u, void* grad_v,
                                          int B, int V, int64_t gout_sB, int64_t field_sB, int64_t u_sB, int64_t v_sB,
                                          float dt, int interp, int pole_fix, int math, int phases, float cfl_cells,
                                          void* workspace, size_t workspace_bytes, int32_t* status, void* stream) {
  Params P;
  if (int rc = fill_params(P, geom, B, V, dt, interp, pole_fix)) return rc;
  if (!grad_out || !field || !u || !v) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if ((phases & ~(PARADIS_BWD_ALL | PARADIS_BWD_ROWSWEEP)) || !(phases & PARADIS_BWD_ALL))
    return fail(PARADIS_ERR_BAD_SHAPE, "phases must be 1, 2 or 3 (optionally | PARADIS_BWD_ROWSWEEP)");
  if ((grad_u == nullptr) != (grad_v == nullptr)) return fail(PARADIS_ERR_NULL_POINTER, "grad_u and grad_v must both be given or both be NULL");
  const void* ptrs[7] = {grad_out, field, u, v, grad_field, grad_u, grad_v};
  const int64_t sB8[3] = {field_sB, u_sB, v_sB}, sB4[1] = {gout_sB};
  if (int rc = bf16_check(geom, ptrs, 7, sB8, 3, sB4, 1)) return rc;
  const BwdWs L = bwd_layout(B, V, P.arrN, P.W);
  if (!workspace || workspace_bytes < paradis_sl_advect_bwd_bf16_workspace(B, V, P.arrN, P.W))
    return fail(PARADIS_ERR_WORKSPACE, "backward workspace too small (%zu < %zu bytes)", workspace_bytes,
                paradis_sl_advect_bwd_bf16_workspace(B, V, P.arrN, P.W));
  cudaStream_t st = (cudaStream_t)stream;
  // grad_field is accumulated in fp32 (ring retire, guard / cut / pole fix-ups and the recompute of flagged planes all
  // add to or overwrite fp32 values after the first store) and rounded to bf16 once at the end
  float* gf32 = grad_field ? (float*)((char*)workspace + L.total) : nullptr;
  if (int rc = advect_bwd<bf16>(P, L, grad_out, field, u, v, gf32, grad_u, grad_v, B, V, gout_sB, field_sB, u_sB, v_sB,
                                interp, pole_fix, math, phases, cfl_cells, (char*)workspace, status, st))
    return rc;
  if (grad_field && (phases & PARADIS_BWD_GATHER)) {
    const long long n8 = (long long)B * V * P.ownN * P.W / 8;
    long long blocks = (n8 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    f32_to_bf16_kernel<<<(unsigned)blocks, 256, 0, st>>>(gf32, (bf16*)grad_field, n8);
  }
  return check_launch("paradis_sl_advect_bwd_bf16");
}

// ---------------------------------------------------------------------------------------------
// parity instrument: the departure-point chain alone
// ---------------------------------------------------------------------------------------------
template <bool EXACT>
__global__ void departure_coords_kernel(const Params P, float* __restrict__ coords) {
  const int c = blockIdx.y, b = blockIdx.z, pl = b * P.V + c;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P.ownN * P.W) return;
  const int r = idx / P.W, x = idx - r * P.W, y = P.own0 + r;
  const int aoff = (y - P.uvg0) * P.W + x;
  const float uu = plane_ptr_bc(P.u, P.u_sB, b, c, P.uvgN, P.W)[aoff];
  const float vv = plane_ptr_bc(P.v, P.v_sB, b, c, P.uvgN, P.W)[aoff];
  Traj t;
  trajectory<EXACT>(P, uu, vv, __ldg(P.sin_lat + y), __ldg(P.cos_lat + y), __ldg(P.lon + x), t);
  const long long plane = (long long)P.ownN * P.W;
  float* o = coords + (long long)pl * 11 * plane + idx;
  o[0] = t.ix; o[plane] = t.iy; o[2 * plane] = t.sa; o[3 * plane] = t.ca; o[4 * plane] = t.sb;
  o[5 * plane] = t.cb; o[6 * plane] = t.s; o[7 * plane] = t.num; o[8 * plane] = t.den;
  o[9 * plane] = t.lat; o[10 * plane] = t.lon;
}

extern "C" int paradis_sl_departure_coords(const paradis_sl_geom* geom, const float* u, const float* v, float* coords,
                                           int B, int V, int64_t u_sB, int64_t v_sB, float dt, int interp, int math,
                                           void* stream) {
  Params P;
  if (int rc = fill_params(P, geom, B, V, dt, interp, 0)) return rc;
  if (!u || !v || !coords) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  P.u = u; P.v = v; P.u_sB = u_sB; P.v_sB = v_sB;
  dim3 grid((P.ownN * P.W + 255) / 256, V, B);
  if (math == PARADIS_MATH_EXACT) departure_coords_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(P, coords);
  else departure_coords_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(P, coords);
  return check_launch("paradis_sl_departure_coords");
}

// ---------------------------------------------------------------------------------------------
// padding op
// ---------------------------------------------------------------------------------------------
static int pad_check(const void* a, const void* b, int64_t planes, int H, int W, int p) {
  if (!a || !b) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if (planes <= 0 || H <= 0 || W <= 0 || p < 0) return fail(PARADIS_ERR_BAD_SHAPE, "non-positive dimension");
  if (W % 2) return fail(PARADIS_ERR_ODD_WIDTH, "Number of longitude points must be even (W=%d)", W);
  if (H < p + 1 || W < 2 * p) return fail(PARADIS_ERR_BAD_SHAPE, "pad width %d too large for %dx%d", p, H, W);
  if (planes > 65535 || H + 2 * p > 65535) return fail(PARADIS_ERR_BAD_SHAPE, "too many planes/rows for one launch");
  return PARADIS_OK;
}

// Halo outbox of the latitude-band decomposition: first / last h rows of up to four tensors in one launch.
struct HaloPackArgs { const float* src[4]; long long sB[4]; };

template <int VEC>
__global__ void halo_pack_kernel(HaloPackArgs a, int n, int V, int rows, int Wv, int h, float* __restrict__ box, long long total) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long planes_hw = (long long)h * Wv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    // i = (((k * 2 + side) * planes + pl) * h + r) * Wv + x
    long long q = i / planes_hw;
    const long long rx = i - q * planes_hw;
    const int r = (int)(rx / Wv), x = (int)(rx - (long long)r * Wv);
    const long long planes = total / ((long long)n * 2 * planes_hw);
    const int pl = (int)(q % planes); q /= planes;
    const int side = (int)(q & 1), k = (int)(q >> 1);
    const int b = pl / V, c = pl - b * V;
    const int row = side ? rows - h + r : r;
    const float* sp = a.src[k] + b * a.sB[k] + ((long long)c * rows + row) * (Wv * VEC);
    if (VEC == 4) reinterpret_cast<float4*>(box)[i] = __ldg(reinterpret_cast<const float4*>(sp) + x);
    else box[i] = __ldg(sp + x);
  }
}

extern "C" int paradis_halo_pack(const float* const* src, const int64_t* src_sB, int n, int B, int V, int rows, int W,
                                 int h, float* box, void* stream) {
  if (!src || !src_sB || !box) return fail(PARADIS_ERR_NULL_POINTER, "halo_pack: NULL pointer");
  if (n < 1 || n > 4 || B < 1 || V < 1 || W < 1 || h < 1 || rows < h)
    return fail(PARADIS_ERR_BAD_SHAPE, "halo_pack: need 1 <= n <= 4 tensors and 1 <= h <= rows (n=%d h=%d rows=%d)", n, h, rows);
  HaloPackArgs a;
  bool vec = (W % 4 == 0) && ((uintptr_t)box % 16 == 0);
  for (int k = 0; k < 4; ++k) {
    a.src[k] = k < n ? src[k] : nullptr;
    a.sB[k] = k < n ? (long long)src_sB[k] : 0;
    if (k < n && !src[k]) return fail(PARADIS_ERR_NULL_POINTER, "halo_pack: NULL tensor pointer");
    if (k < n && ((uintptr_t)src[k] % 16 != 0 || src_sB[k] % 4 != 0)) vec = false;
  }
  const int VEC = vec ? 4 : 1, Wv = W / VEC;
  const long long total = (long long)n * 2 * B * V * h * Wv;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (vec) halo_pack_kernel<4><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, n, V, rows, Wv, h, box, total);
  else halo_pack_kernel<1><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, n, V, rows, Wv, h, box, total);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : fail(PARADIS_ERR_CUDA, "halo_pack: %s", cudaGetErrorString(e));
}

template <typename T>
static int pad_fwd(const T* x, T* y, int64_t planes, int H, int W, int p, void* stream, const char* what) {
  if (int rc = pad_check(x, y, planes, H, W, p)) return rc;
  const int Wp = W + 2 * p, per_thread = kIsF32<T> ? 1 : 2;
  dim3 grid((Wp / per_thread + 255) / 256, H + 2 * p, (unsigned)planes);
  geocyclic_pad_fwd_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, H, W, p);
  return check_launch(what);
}

template <typename T>
static int pad_bwd(const T* gy, T* gx, int64_t planes, int H, int W, int p, void* stream, const char* what) {
  if (int rc = pad_check(gy, gx, planes, H, W, p)) return rc;
  dim3 grid((W + 255) / 256, H, (unsigned)planes);
  geocyclic_pad_bwd_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(gy, gx, H, W, p);
  return check_launch(what);
}

extern "C" int paradis_geocyclic_pad_fwd(const float* x, float* y, int64_t planes, int H, int W, int p, void* stream) {
  return pad_fwd(x, y, planes, H, W, p, stream, "paradis_geocyclic_pad_fwd");
}

extern "C" int paradis_geocyclic_pad_bwd(const float* gy, float* gx, int64_t planes, int H, int W, int p, void* stream) {
  return pad_bwd(gy, gx, planes, H, W, p, stream, "paradis_geocyclic_pad_bwd");
}

// bf16 storage (include/paradis_geocyclic.h); the forward writes its output in 4-byte words
extern "C" int paradis_geocyclic_pad_fwd_bf16(const void* x, void* y, int64_t planes, int H, int W, int p, void* stream) {
  if (x && y && (uintptr_t)y % 4) return fail(PARADIS_ERR_BAD_SHAPE, "geocyclic_pad bf16: output must be 4-byte aligned");
  return pad_fwd((const bf16*)x, (bf16*)y, planes, H, W, p, stream, "paradis_geocyclic_pad_fwd_bf16");
}

extern "C" int paradis_geocyclic_pad_bwd_bf16(const void* gy, void* gx, int64_t planes, int H, int W, int p, void* stream) {
  return pad_bwd((const bf16*)gy, (bf16*)gx, planes, H, W, p, stream, "paradis_geocyclic_pad_bwd_bf16");
}

// ---------------------------------------------------------------------------------------------
// host-buffer entry: chunks of planes pipelined over three streams (H2D | kernels | D2H overlap
// across chunks because consecutive chunks live on different streams and slots)
// ---------------------------------------------------------------------------------------------
// chunks in flight (each on its own stream): H2D of one, kernels of another, D2H of a third overlap; more slots keep
// both copy engines busy across the slot-reuse dependency (25.4-26.5 ms at C3 for 3-6 slots: PCIe bound)
static constexpr int kSlots = 4;

struct HostSlot { size_t field, u, v, gout, out, gfield, gu, gv, wsf, wsb, status, total; };
static HostSlot host_slot_layout(int H, int W, int c) {
  HostSlot s;
  const size_t t = align_up((size_t)c * H * W * sizeof(float), 256);
  size_t off = 0;
  s.field = off; off += t; s.u = off; off += t; s.v = off; off += t; s.gout = off; off += t;
  s.out = off; off += t; s.gfield = off; off += t; s.gu = off; off += t; s.gv = off; off += t;
  s.wsf = off; off += paradis_sl_advect_fwd_workspace(1, c);
  s.wsb = off; off += paradis_sl_advect_bwd_workspace(1, c, H, W);
  s.status = off; off += 256;
  s.total = off;
  return s;
}

extern "C" size_t paradis_sl_host_scratch_bytes(int H, int W, int chunk_planes) {
  if (H <= 0 || W <= 0 || chunk_planes <= 0) return 0;
  return host_slot_layout(H, W, chunk_planes).total * kSlots;
}

extern "C" int paradis_sl_advect_fwd_bwd_host(const paradis_sl_geom* geom, const float* h_field, const float* h_u,
                                              const float* h_v, const float* h_grad_out, float* h_out,
                                              float* h_grad_field, float* h_grad_u, float* h_grad_v, int64_t planes,
                                              float dt, int interp, int pole_fix, int math, float cfl_cells,
                                              int chunk_planes,
                                              void* d_scratch, size_t scratch_bytes) {
  if (!geom) return fail(PARADIS_ERR_NULL_POINTER, "geom is NULL");
  if (!h_field || !h_u || !h_v || !h_grad_out || !h_out || !h_grad_field || !h_grad_u || !h_grad_v)
    return fail(PARADIS_ERR_NULL_POINTER, "NULL host pointer");
  if (planes <= 0 || chunk_planes <= 0) return fail(PARADIS_ERR_BAD_SHAPE, "non-positive plane count");
  const int H = geom->H, W = geom->W;
  if (geom->own_row0 != 0 || geom->own_rows != H || geom->arr_rows != H || geom->fld_rows != H)
    return fail(PARADIS_ERR_BAD_SHAPE, "host entry works on the full mesh");
  const HostSlot L = host_slot_layout(H, W, chunk_planes);
  if (!d_scratch || scratch_bytes < L.total * kSlots)
    return fail(PARADIS_ERR_WORKSPACE, "host-entry scratch too small (%zu < %zu bytes)", scratch_bytes, L.total * kSlots);
  cudaStream_t st[kSlots];
  for (int i = 0; i < kSlots; ++i)
    if (cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking) != cudaSuccess)
      return fail(PARADIS_ERR_CUDA, "cudaStreamCreate failed");
  int rc = PARADIS_OK;
  const size_t plane_elems = (size_t)H * W;
  int64_t done = 0;
  for (int it = 0; done < planes && rc == PARADIS_OK; ++it) {
    const int c = (int)((planes - done < chunk_planes) ? planes - done : chunk_planes);
    const int slot = it % kSlots;
    char* base = (char*)d_scratch + (size_t)slot * L.total;
    cudaStream_t s = st[slot];
    const size_t bytes = (size_t)c * plane_elems * sizeof(float), off = (size_t)done * plane_elems;
    float *df = (float*)(base + L.field), *du = (float*)(base + L.u), *dv = (float*)(base + L.v),
          *dg = (float*)(base + L.gout), *dout = (float*)(base + L.out), *dgf = (float*)(base + L.gfield),
          *dgu = (float*)(base + L.gu), *dgv = (float*)(base + L.gv);
    cudaMemcpyAsync(df, h_field + off, bytes, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(du, h_u + off, bytes, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(dv, h_v + off, bytes, cudaMemcpyHostToDevice, s);
    cudaMemcpyAsync(dg, h_grad_out + off, bytes, cudaMemcpyHostToDevice, s);
    const int64_t sB = (int64_t)c * plane_elems;
    rc = paradis_sl_advect_fwd(geom, df, du, dv, dout, 1, c, sB, sB, sB, dt, interp, pole_fix, math, base + L.wsf,
                               paradis_sl_advect_fwd_workspace(1, c), nullptr, s);
    if (rc) break;
    cudaMemcpyAsync(h_out + off, dout, bytes, cudaMemcpyDeviceToHost, s);
    rc = paradis_sl_advect_bwd(geom, dg, df, du, dv, dgf, dgu, dgv, 1, c, sB, sB, sB, sB, dt, interp, pole_fix, math,
                               PARADIS_BWD_ALL, cfl_cells, base + L.wsb, paradis_sl_advect_bwd_workspace(1, c, H, W), nullptr, s);
    if (rc) break;
    cudaMemcpyAsync(h_grad_field + off, dgf, bytes, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(h_grad_u + off, dgu, bytes, cudaMemcpyDeviceToHost, s);
    cudaMemcpyAsync(h_grad_v + off, dgv, bytes, cudaMemcpyDeviceToHost, s);
    done += c;
  }
  for (int i = 0; i < kSlots; ++i) {
    cudaError_t e = cudaStreamSynchronize(st[i]);
    if (e != cudaSuccess && rc == PARADIS_OK) rc = fail(PARADIS_ERR_CUDA, "host entry: %s", cudaGetErrorString(e));
    cudaStreamDestroy(st[i]);
  }
  return rc;
}

// ---------------------------------------------------------------------------------------------
// tangent-linear model (include/paradis_sl_tl.h)
// ---------------------------------------------------------------------------------------------
#include "sl_tangent.cuh"

extern "C" size_t paradis_sl_advect_jvp_workspace(int B, int V) {
  return 2 * paradis_sl_advect_fwd_workspace(B, V);      // zonal pole means of field | of dfield
}

extern "C" int paradis_sl_advect_jvp(const paradis_sl_geom* geom, const float* field, const float* dfield,
                                     const float* u, const float* v, const float* du, const float* dv, float* dout,
                                     int B, int V, int64_t field_sB, int64_t dfield_sB, int64_t u_sB, int64_t v_sB,
                                     int64_t du_sB, int64_t dv_sB, float dt, int interp, int pole_fix, int math,
                                     void* workspace, size_t workspace_bytes, int32_t* status, void* stream) {
  Params P;
  if (int rc = fill_params(P, geom, B, V, dt, interp, pole_fix)) return rc;
  if (!field || !u || !v || !dout) return fail(PARADIS_ERR_NULL_POINTER, "NULL tensor pointer");
  if ((du == nullptr) != (dv == nullptr)) return fail(PARADIS_ERR_NULL_POINTER, "du and dv must both be given or both be NULL");
  if (int rc = full_mesh_check(geom, "tangent-linear entry points", "not supported")) return rc;
  if (pole_fix && (!workspace || workspace_bytes < paradis_sl_advect_jvp_workspace(B, V)))
    return fail(PARADIS_ERR_WORKSPACE, "jvp workspace too small (%zu bytes)", workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  const int planes = B * V;
  P.field = field; P.u = u; P.v = v; P.out = dout;
  P.field_sB = field_sB; P.u_sB = u_sB; P.v_sB = v_sB;
  P.status = status;
  TLArgs A;
  A.dfield = dfield; A.du = du; A.dv = dv; A.dmean = nullptr;
  A.dfield_sB = dfield_sB; A.du_sB = du_sB; A.dv_sB = dv_sB;
  if (pole_fix) {      // zonal pole means of field and dfield in one launch
    P.fmean = (const float*)workspace;
    A.dmean = (const float*)((char*)workspace + paradis_sl_advect_fwd_workspace(B, V));
    pole_means_kernel<float><<<planes * (dfield ? 4 : 2), kPoleThreads, 0, st>>>(
        field, field_sB, V, P.fldN, P.fld0, P.H, P.W, planes, (float*)P.fmean, dfield, dfield_sB, P.fldN, P.fld0,
        (float*)A.dmean);
  }
  const bool vec_ok = (P.W % 4 == 0) && aligned16(field) && aligned16(u) && aligned16(v) && aligned16(dout) &&
                      aligned16(P.lon) && (!dfield || aligned16(dfield)) && (!du || (aligned16(du) && aligned16(dv))) &&
                      (field_sB % 4 == 0) && (dfield_sB % 4 == 0) && (u_sB % 4 == 0) && (v_sB % 4 == 0) &&
                      (du_sB % 4 == 0) && (dv_sB % 4 == 0);
  const int vec = points_per_thread(interp, vec_ok);
  set_units(P, vec, P.ownN);
  dim3 grid(((unsigned)P.ownN * P.upr + 255) / 256, V, B);
  const bool exact = math == PARADIS_MATH_EXACT;
  if (interp == 1) { if (exact) launch_tl<true, 1>(P, A, vec, grid, st); else launch_tl<false, 1>(P, A, vec, grid, st); }
  else             { if (exact) launch_tl<true, 2>(P, A, vec, grid, st); else launch_tl<false, 2>(P, A, vec, grid, st); }
  if (pole_fix) pole_rows_fix_kernel<<<planes * 2, kPoleThreads, 0, st>>>(dout, P.ownN, P.own0, P.H, P.W, planes);
  return check_launch("paradis_sl_advect_jvp");
}

// ---------------------------------------------------------------------------------------------
// float64 (include/paradis_sl_f64.h)
// ---------------------------------------------------------------------------------------------
#include "sl_f64.cuh"
