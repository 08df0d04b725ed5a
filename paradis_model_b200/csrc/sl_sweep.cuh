// Fused backward kernel: one pass over the arrival points produces grad_u, grad_v AND grad_field.
//
// Work unit ("task") = one warp = (plane, band of destination rows [ra, rb), strip of destination
// columns [ja, jb)).  The warp sweeps the arrival rows that can reach its tile in ascending order;
// per row it visits its own columns ("core" chunks: full work incl. grad_u / grad_v) and `hx` halo
// columns either side (trajectory + adjoint only).  Adjoint contributions go into a warp-private
// ring of `ring` destination rows in shared memory; a destination row is written to grad_field
// (coalesced) as soon as no later arrival row can reach it.
//
// Determinism without atomics: only this warp ever touches its ring, rows/chunks/tap phases are
// visited in a fixed order, and within one 32-lane step two lanes can only clash when their
// departure cells coincide.  Clashes are detected with one-byte tags (plain stores: who wins only
// signals that a clash exists), then every clashing cell is resolved by a ballot on the exact key
// and summed into its lowest lane in ascending lane order, so each add into the ring has a single
// writer and a data-defined order.
//
// Contract: |floor(iy) - row| <= rr and the longitudinal reach of a band <= its hx.  Every core
// point checks it; a violation marks the plane in `plane_flag`, and the host always enqueues the
// general (two-kernel) path behind the sweep, which recomputes exactly the flagged planes.
//
// What the kernel does about latency (it runs at 16 warps / SM, DESIGN.md section 8 has the measurements):
// 4 points per lane in the core step (2x2 stencil); "touches" that pull the lines of the next row step into L1
// one row ahead; no branch in `asin`, one range check for the 8 backtrack angles of a lane; the per-row halo
// width computed once per 32 rows and shuffled; finished ring rows retired and cleared with float4 accesses.
#pragma once
#include "sl_device.cuh"

namespace psl {

constexpr int kSweepWarps = 4;
constexpr int kMaxBands = 48;

constexpr int kTagRows = 4;                   // clash tags cover (slot mod kTagRows, column)
// Ring row layout: kRingLead margin columns, the strip's own wc columns (16-byte aligned, so that a finished row is
// retired and cleared with float4 accesses), margin up to kRingPad columns in total.
constexpr int kRingLead = 4, kRingPad = 8;
__host__ __device__ constexpr int sweep_pitch(int wc) { return wc + kRingPad; }
// floats per warp: ring + clash tags, rounded to 16 bytes
__host__ __device__ constexpr int sweep_warp_floats(int ring, int pitch) {
  return ring * pitch + (((kTagRows * pitch + 3) / 4 + 3) & ~3);
}

// Longitudinal reach (in cells, rounded up to 16) of an arrival row: the halo a strip needs on
// either side.  |dlon| <= asin(sin(delta) / cos(|lat| + delta)) for a great-circle step delta.
// Evaluated identically by every task (and by the host plan, which only uses it for balancing).
struct ReachModel { float sin_delta, cos_delta, inv_dlam; int extra, max_halo; };
__host__ __device__ __forceinline__ int halo_cells(const ReachModel& m, float sin_lat, float cos_lat) {
  const float c = cos_lat * m.cos_delta - fabsf(sin_lat) * m.sin_delta;   // cos(|lat| + delta)
  if (!(c > m.sin_delta)) return 1 << 20;
  const int n = (int)ceilf(asinf(m.sin_delta / c) * m.inv_dlam) + m.extra;
  return (n + 15) & ~15;
}

struct SweepPlan {
  int nbands, nstrips, wc, rr, ring, pitch;   // pitch = sweep_pitch(wc)
  int planes;
  ReachModel reach;
  int ra[kMaxBands], rb[kMaxBands];           // band k owns destination rows [ra[k], rb[k]); bands are
                                              // sorted by decreasing cost
  unsigned char* plane_flag;                  // [planes] set to 1 on a contract violation
  int out0, outN;                             // rows held by the output tensors (global first row, count)
};

template <int NT>
__device__ __forceinline__ void resolve_clashes(int key, int tkey, unsigned char* tag, int lane,
                                                float (&c)[NT * NT], bool& writer) {
  // tkey: tag slot (hashed rows; a false alias only costs one pass of the loop below)
  if (key >= 0) tag[tkey] = (unsigned char)lane;
  __syncwarp();
  const bool lost = (key >= 0) && (tag[tkey] != (unsigned char)lane);
  unsigned pending = __ballot_sync(0xffffffffu, lost);
  writer = key >= 0;
  while (pending) {  // uniform loop: one iteration per clashing cell
    const int j = __ffs(pending) - 1;
    const int kj = __shfl_sync(0xffffffffu, key, j);
    const unsigned group = __ballot_sync(0xffffffffu, key == kj);
    pending &= ~group;
    const int leader = __ffs(group) - 1;
    unsigned rest = group & (group - 1);
    while (rest) {
      const int src = __ffs(rest) - 1;
      rest &= rest - 1;
#pragma unroll
      for (int t = 0; t < NT * NT; ++t) {
        const float o = __shfl_sync(0xffffffffu, c[t], src);
        if (lane == leader) c[t] += o;
      }
    }
    if (lane != leader && ((group >> lane) & 1u)) writer = false;
  }
}

// Warp-uniform state of the row being swept (T: storage type of u, v, grad_u, grad_v).
template <typename T>
struct SweepRow {
  const T* __restrict__ urow;
  const T* __restrict__ vrow;
  const float* __restrict__ grow;
  T* __restrict__ gu_row;          // nullptr when this row's grad_u / grad_v are not produced here
  T* __restrict__ gv_row;
  float sp, cp;
  int y, head, hx;
};

// What one lane contributes to the ring in one 32-lane step.
template <int NT> struct StepOut {
  int key;                         // ring cell of tap (0, 0), < 0: nothing to add
  int slot0, cidx;
  int off1;                        // ring cell of tap (1, 0) (2x2 stencil: the scatter needs no slot arithmetic)
  float cc[NT * NT];
};

// Trajectory, contract check, (for own points) grad_u / grad_v, and the stencil weights of one
// arrival point.  x: column (unwrapped, for the ring index), xw: wrapped column.
template <bool EXACT, int INTERP, bool CORE, bool PEER, bool SMALL = false, typename T>
__device__ __forceinline__ void sweep_compute(const Params& P, const SweepRow<T>& R, const T* __restrict__ f,
                                              int pl, float mean0, float mean1, int ja, int wc, int ring, int pitch,
                                              int rr, int x, int xw, float uu, float vv, float g, float lonp, bool& violated,
                                              StepOut<Stencil<INTERP>::NT>& o, float& ou, float& ov) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  o.key = -1; o.slot0 = 0; o.cidx = 0; o.off1 = 0;
  Traj t;
  trajectory<EXACT, SMALL>(P, uu, vv, R.sp, R.cp, lonp, t);
  const float fx = floorf(t.ix), fy = floorf(t.iy);
  const float tx = __fsub_rn(t.ix, fx), ty = __fsub_rn(t.iy, fy);
  const int x0 = (int)fx + OMIN;                 // padded column of tap 0
  const int cls = (int)fy - (R.y + P.p);         // row class
  int dx = x0 - P.p - xw;                        // longitudinal cell displacement of tap 0
  if (dx < -P.halfW) dx += P.W; else if (dx >= P.halfW) dx -= P.W;
  const bool in_ring = (unsigned)(cls + rr) <= (unsigned)(2 * rr);
  if (CORE) {
    // every arrival point a task sees in its own columns is checked against the contract
    if (!in_ring || dx < -R.hx || dx > R.hx - NT + 1) violated = true;
    if (R.gu_row) {
      float val, ddx, ddy;
      stencil_eval<INTERP, true, PEER>(P, f, pl, t, mean0, mean1, val, ddx, ddy);
      velocity_grads<EXACT>(P, t, R.sp, R.cp, g * ddx, g * ddy, ou, ov);
    }
  }
  const int cidx = (x - ja) + dx + kRingLead;    // ring column of tap 0
  const bool hit = in_ring && (unsigned)(cidx - (kRingLead - NT + 1)) <= (unsigned)(wc + NT - 2);
  float wx[NT], wy[NT], d0[NT], d1[NT];
  axis_weights<INTERP, false>(tx, wx, d0);
  axis_weights<INTERP, false>(ty, wy, d1);
  int slot0 = R.head + cls + rr;
  if (slot0 >= ring) slot0 -= ring;
  o.slot0 = hit ? slot0 : 0; o.cidx = hit ? cidx : 0;
  o.key = hit ? slot0 * pitch + cidx : -1;
  if (NT == 2) {
    const int slot1 = slot0 + 1 == ring ? 0 : slot0 + 1;
    o.off1 = hit ? slot1 * pitch + cidx : 0;
  } else {
    o.off1 = 0;
  }
  const float gh = hit ? g : 0.0f;
#pragma unroll
  for (int a = 0; a < NT; ++a) {
    const float gw = __fmul_rn(gh, wy[a]);
#pragma unroll
    for (int bb = 0; bb < NT; ++bb)   // padding_mode="zeros": only the last tap columns can leave the padded plane
      o.cc[a * NT + bb] = (bb == 0 || x0 + bb < P.Wp) ? __fmul_rn(gw, wx[bb]) : 0.0f;
  }
}

// Add one step's contributions to the ring: clash resolution, then NT*NT single-writer phases.
template <int NT>
__device__ __forceinline__ void sweep_scatter(StepOut<NT>& o, float* acc, unsigned char* tag, int ring, int pitch,
                                              int lane) {
  bool writer;
  resolve_clashes<NT>(o.key, (o.slot0 & (kTagRows - 1)) * pitch + o.cidx, tag, lane, o.cc, writer);
  if (NT == 2) {
    float* r0 = acc + (writer ? o.key : 0);
    float* r1 = acc + o.off1;
    if (writer) r0[0] += o.cc[0];
    __syncwarp();
    if (writer) r0[1] += o.cc[1];
    __syncwarp();
    if (writer) r1[0] += o.cc[2];
    __syncwarp();
    if (writer) r1[1] += o.cc[3];
    __syncwarp();
    return;
  }
  float* base = acc + o.cidx;
#pragma unroll
  for (int a = 0; a < NT; ++a) {
    int sl = o.slot0 + a;
    if (sl >= ring) sl -= ring;
    float* row = base + sl * pitch;
#pragma unroll
    for (int bb = 0; bb < NT; ++bb) {
      if (writer) row[bb] += o.cc[a * NT + bb];
      __syncwarp();
    }
  }
}

// 4 CTAs / SM for the 2x2 stencil (more resident warps measured slower: 2.19 -> 2.23 ms backward at 0.25 deg);
// 6 CTAs / SM = 80 registers for 4x4, where a fourth row band of resident tasks pays for the few spills
// (4.54 -> 3.98 ms)
template <bool EXACT, int INTERP, bool PEER, typename T>
__global__ void __launch_bounds__(kSweepWarps * 32, INTERP == 2 ? 6 : 4) sl_bwd_sweep_kernel(const Params P, const SweepPlan S) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1-D grid, most expensive bands first: task -> (band, plane, strip)
  const int task = blockIdx.x * kSweepWarps + warp;
  const int per_band = S.planes * S.nstrips;
  if (task >= S.nbands * per_band) return;
  const int band = task / per_band, rem = task - band * per_band;
  const int pl = rem / S.nstrips, strip = rem - pl * S.nstrips;
  const int b = pl / P.V, c = pl - b * P.V;
  const int ra = S.ra[band], rb = S.rb[band];
  const int ja = strip * S.wc, jb = min(ja + S.wc, P.W), wc = jb - ja;
  const int ring = S.ring, pitch = S.pitch, rr = S.rr;
  const int cells = ring * pitch;
  float* acc = smem + (size_t)warp * sweep_warp_floats(ring, pitch);
  unsigned char* tag = reinterpret_cast<unsigned char*>(acc + cells);
  for (int i = lane; i < cells; i += 32) acc[i] = 0.0f;
  __syncwarp();

  const T* up = plane_ptr_bc(as<T>(P.u), P.u_sB, b, c, P.uvgN, P.W);
  const T* vp = plane_ptr_bc(as<T>(P.v), P.v_sB, b, c, P.uvgN, P.W);
  const float* gp = plane_ptr_bc(P.gout, P.gout_sB, b, c, P.uvgN, P.W);
  const T* f = plane_ptr_bc(as<T>(P.field), P.field_sB, b, c, P.fldN, P.W);
  T* gu_pl = P.gu ? as<T>(P.gu) + (long long)pl * S.outN * P.W : nullptr;
  T* gv_pl = P.gu ? as<T>(P.gv) + (long long)pl * S.outN * P.W : nullptr;
  float* gf_pl = P.gfield + (long long)pl * S.outN * P.W + ja;
  float mean0 = 0.0f, mean1 = 0.0f;
  if (P.pole_fix) { mean0 = __ldg(P.fmean + 2 * pl); mean1 = __ldg(P.fmean + 2 * pl + 1); }
  const int arr_lo = P.arr0, arr_hi = P.arr0 + P.arrN, W = P.W;
  bool violated = false;

  // destination row i_done(y) = y - rr + OMIN is complete after arrival row y; it sits in slot `head`
  const int y_first = ra - (ring - 1) + rr - OMIN, y_last = rb - 1 + rr - OMIN;
  SweepRow<T> R;
  R.head = 0;
  // Warm-up loads ("touches"): while a row is processed, each lane loads one word of a 128-byte line the NEXT
  // row step will need -- u, v, grad_out of the next arrival row and the field row that enters the stencil
  // window with it -- over the columns [ja - 64, ja + 192).  The value is only consumed at the end of the row
  // step, so the load never stalls; it replaces ~3.4k stall cycles per row on first-touch L2 / DRAM latency
  // (`prefetch.global.L1` did not have that effect).  Measured 2.19 -> 2.07 ms backward at 0.25 deg.  The 4x4 kernel
  // is register-bound at 80: touches cost it more than they save.
  constexpr bool kTouch = NT == 2;
  const int pf_arr = lane >> 3;
  int pf_col = ja - 64 + ((lane & 7) << 5);
  if (pf_col < 0) pf_col += W; else if (pf_col >= W) pf_col -= W;
  float pf_sink = 0.0f;
  int hx_lane = 0;
  for (int y = y_first; y <= y_last; ++y) {
    // the halo width is a function of the row only: lane l evaluates it for row y + l once every 32 rows
    // (halo_cells costs ~40 instructions; evaluated per row by every lane it was 2 % of the kernel)
    if (((y - y_first) & 31) == 0) {
      const int yy = min(max(y + lane, arr_lo), arr_hi - 1);
      hx_lane = halo_cells(S.reach, __ldg(P.sin_lat + yy), __ldg(P.cos_lat + yy));
    }
    float pf_val = 0.0f;
    if (kTouch) {
      const int yn = y + 1;
      if (yn >= arr_lo && yn < arr_hi && yn <= y_last) {
        if constexpr (kIsF32<T>) {
          const float* q = nullptr;
          if (pf_arr == 0) q = arr_row<PEER>(P, up, 0, pl, yn);
          else if (pf_arr == 1) q = arr_row<PEER>(P, vp, 1, pl, yn);
          else if (pf_arr == 2) q = arr_row<PEER>(P, gp, 2, pl, yn);
          else {
            const int yf = yn + rr + NT - 1 + OMIN;   // last stencil row the next arrival row can reach
            if (!PEER && yf >= P.fld0 && yf < P.fld0 + P.fldN) q = f + (long long)(yf - P.fld0) * W;
          }
          if (q) pf_val = __ldg(q + pf_col);
        } else {                                      // bf16 rows: same words, half the bytes (over-touches u, v, field)
          const T* q = nullptr;
          if (pf_arr == 0) q = arr_row<PEER>(P, up, 0, pl, yn);
          else if (pf_arr == 1) q = arr_row<PEER>(P, vp, 1, pl, yn);
          else if (pf_arr == 3) {
            const int yf = yn + rr + NT - 1 + OMIN;
            if (yf >= P.fld0 && yf < P.fld0 + P.fldN) q = f + (long long)(yf - P.fld0) * W;
          }
          if (q) pf_val = ldg_f(q + pf_col);
          else if (pf_arr == 2) pf_val = __ldg(arr_row<PEER>(P, gp, 2, pl, yn) + pf_col);
        }
      }
    }
    if (y >= arr_lo && y < arr_hi) {
      R.y = y;
      R.sp = __ldg(P.sin_lat + y); R.cp = __ldg(P.cos_lat + y);
      R.urow = arr_row<PEER>(P, up, 0, pl, y);   // a neighbour's row when y lies in the peer halo
      R.vrow = arr_row<PEER>(P, vp, 1, pl, y);
      R.grow = arr_row<PEER>(P, gp, 2, pl, y);
      const bool core_row = (y >= ra) && (y < rb) && gu_pl;
      R.gu_row = core_row ? gu_pl + (y - S.out0) * W : nullptr;
      R.gv_row = core_row ? gv_pl + (y - S.out0) * W : nullptr;
      int hx = __shfl_sync(0xffffffffu, hx_lane, (y - y_first) & 31);   // <= max_halo for every row a band may visit
      R.hx = min(hx, S.reach.max_halo + 16);          // (host/device rounding may differ by one step)
      const int nhalo = (2 * R.hx + 31) >> 5;
      if (NT == 2) {
      // own columns: one step of 4 consecutive points per lane (float4 loads / stores, 4 independent
        // trajectories in flight), scattered as 4 sub-steps of points 4 columns apart
        {
          const int x = ja + 4 * lane;
          StepOut<NT> o[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            o[k].key = -1; o[k].slot0 = 0; o[k].cidx = 0; o[k].off1 = 0;
#pragma unroll
            for (int t = 0; t < NT * NT; ++t) o[k].cc[t] = 0.0f;
          }
          if (x < jb) {
            float uu[4], vv[4], gg[4], ll[4], ou[4], ov[4];
            *reinterpret_cast<float4*>(uu) = ldg4_f(R.urow + x);
            *reinterpret_cast<float4*>(vv) = ldg4_f(R.vrow + x);
            *reinterpret_cast<float4*>(gg) = __ldg(reinterpret_cast<const float4*>(R.grow + x));
            *reinterpret_cast<float4*>(ll) = __ldg(reinterpret_cast<const float4*>(P.lon + x));
            // one range check for the lane's 8 backtrack angles instead of one per point (-1 % here; the same
            // hoist costs the forward kernel registers and occupancy, so it is not used there)
            if (!EXACT && small_angles<4>(P.dt, uu, vv)) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                sweep_compute<EXACT, INTERP, true, PEER, true>(P, R, f, pl, mean0, mean1, ja, wc, ring, pitch, rr, x + k, x + k,
                                                               uu[k], vv[k], gg[k], ll[k], violated, o[k], ou[k], ov[k]);
            } else {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                sweep_compute<EXACT, INTERP, true, PEER>(P, R, f, pl, mean0, mean1, ja, wc, ring, pitch, rr, x + k, x + k, uu[k],
                                                         vv[k], gg[k], ll[k], violated, o[k], ou[k], ov[k]);
            }
            if (R.gu_row) {
              stcs4_f(R.gu_row + x, *reinterpret_cast<float4*>(ou));
              stcs4_f(R.gv_row + x, *reinterpret_cast<float4*>(ov));
            }
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) sweep_scatter<NT>(o[k], acc, tag, ring, pitch, lane);
        }
      } else {
        // wide stencils: one point per lane and step (16 weights per point do not fit 4-fold in registers)
        for (int ch = 0; ch < ((wc + 31) >> 5); ++ch) {
          StepOut<NT> oa;
          oa.key = -1; oa.slot0 = 0; oa.cidx = 0; oa.off1 = 0;
#pragma unroll
          for (int t = 0; t < NT * NT; ++t) oa.cc[t] = 0.0f;
          const int xa = ja + (ch << 5) + lane;
          if (xa < jb) {
            float ou = 0.0f, ov = 0.0f;
            sweep_compute<EXACT, INTERP, true, PEER>(P, R, f, pl, mean0, mean1, ja, wc, ring, pitch, rr, xa, xa, ldg_f(R.urow + xa),
                                               ldg_f(R.vrow + xa), __ldg(R.grow + xa), __ldg(P.lon + xa), violated, oa, ou,
                                               ov);
            if (R.gu_row) { stcs_f(R.gu_row + xa, ou); stcs_f(R.gv_row + xa, ov); }
          }
          sweep_scatter<NT>(oa, acc, tag, ring, pitch, lane);
        }
      }
      // halo columns: [ja - hx, ja) then [jb, jb + hx), one point per lane
      for (int ch = 0; ch < nhalo; ++ch) {
        StepOut<NT> oa;
        oa.key = -1; oa.slot0 = 0; oa.cidx = 0; oa.off1 = 0;
#pragma unroll
        for (int t = 0; t < NT * NT; ++t) oa.cc[t] = 0.0f;
        const int h = (ch << 5) + lane;
        const int xa = h < R.hx ? ja - R.hx + h : jb + (h - R.hx);
        int xw = xa;
        if (xw < 0) xw += W; else if (xw >= W) xw -= W;
        if (h < 2 * R.hx) {
          float ou, ov;
          sweep_compute<EXACT, INTERP, false, PEER>(P, R, f, pl, mean0, mean1, ja, wc, ring, pitch, rr, xa, xw, ldg_f(R.urow + xw),
                                              ldg_f(R.vrow + xw), __ldg(R.grow + xw), __ldg(P.lon + xw), violated, oa, ou,
                                              ov);
        }
        sweep_scatter<NT>(oa, acc, tag, ring, pitch, lane);
      }
    }
    // retire destination row i = y - rr + OMIN
    const int i = y - rr + OMIN;
    float* row = acc + R.head * pitch;
    if (i >= ra && i < rb) {
      float* orow = gf_pl + (i - S.out0) * W;
      for (int k = 4 * lane; k < wc; k += 128)
        *reinterpret_cast<float4*>(orow + k) = *reinterpret_cast<const float4*>(row + kRingLead + k);
    }
    __syncwarp();
    for (int k = 4 * lane; k < pitch; k += 128) *reinterpret_cast<float4*>(row + k) = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    R.head = R.head + 1 == ring ? 0 : R.head + 1;
    if (kTouch) pf_sink += pf_val;
  }
  if (kTouch && pf_sink == 1.2345e-30f) violated = true;     // keeps the touches alive
  if (__any_sync(0xffffffffu, violated) && lane == 0) S.plane_flag[pl] = 1;
}

}  // namespace psl
