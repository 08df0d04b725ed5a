// Host-side work partition of the warp-specialised row sweep (sl_rows.cuh): which (plane, row) range every persistent CTA
// owns.  Pure host code (no CUDA calls): paradis_sl.cu includes it, and tests/partition_harness.cu compiles it alone so
// that the CPU test-suite can check its invariants (tests/test_partition.py).
#pragma once
#include <string.h>
#include <math.h>
#include <vector>
#include "sl_device.cuh"
#include "sl_sweep.cuh"
#include "sl_rows.cuh"

namespace psl {

// Min-max partition of the concatenated (plane, own row) space into `grid` contiguous CTA ranges.
// Cost of a range = sum over its segments (one per plane it touches) of the cost of the ARRIVAL rows the segment sweeps:
// its own rows plus the ring - 1 warm-up rows, clipped to the arrival window.  A row costs kRowW0 + k(y), k = 32-record
// steps a consumer scans for it (the whole circle near the poles).  The smallest per-CTA budget T for which a greedy
// left-to-right fill needs at most `grid` ranges is found by bisection; tiny segments are avoided by construction
// (they pay a full warm-up).  An earlier version split proportionally to the own rows' cost and snapped boundaries
// onto plane boundaries: 5 % slower at C3, 11-22 % on thin latitude bands.  Only balance depends on the model.
// The result is cached per shape (it costs ~1 ms of host time).
constexpr int kRowW0 = 4;   // shallow optimum at 3-6 (DESIGN.md section 8)
struct RowsPartKey { long long v[13]; };
struct RowsPartEntry { RowsPartKey key; int bound[kRowsMaxCtas + 1]; int cut; bool valid; };

template <int INTERP>
static void rows_partition(const Params& P, RowsPlan& S, const ReachModel& reach, int wc, int planes, int grid) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  static thread_local RowsPartEntry cache[8];
  static thread_local int cache_next = 0;
  RowsPartKey key;
  memset(&key, 0, sizeof(key));
  const int H = P.H, W = P.W, ownN = P.ownN;
  int fbits[2];
  memcpy(&fbits[0], &P.min_lat, 4); memcpy(&fbits[1], &P.d_lat, 4);
  const long long kv[13] = {H, W, planes, P.own0, ownN, P.arr0, P.arrN, S.rr + 1000 * S.cut, NT, wc, grid, fbits[0], fbits[1]};
  memcpy(key.v, kv, sizeof(kv));
  for (auto& e : cache)
    if (e.valid && memcmp(&e.key, &key, sizeof(key)) == 0) { memcpy(S.bound, e.bound, sizeof(S.bound)); S.cut = e.cut; return; }

  const double dphi = (double)P.d_lat / (H - 1);
  std::vector<double> A(H + 1, 0.0);                       // prefix of the arrival-row costs over global rows
  for (int y = 0; y < H; ++y) {
    const double lat = (double)P.min_lat + y * dphi;
    const int hx = halo_cells(reach, (float)sin(lat), (float)cos(lat));
    int len = wc + 2 * (hx < W ? hx : W);
    if (len > W) len = W;
    int k = (len + 31) >> 5;
    if ((k & 3) == 0) ++k;
    A[y + 1] = A[y] + kRowW0 + k;
  }
  const int arr_lo = P.arr0, arr_hi = P.arr0 + P.arrN;
  auto seg_cost = [&](int ra, int rb) {                     // destination rows [ra, rb) (global) of one plane
    // cut mode: a segment that starts / ends inside the plane processes its own arrival rows only and stores the
    // partial rows beyond the cut (about the cost of retiring as many own rows)
    const bool cut_lo = S.cut && ra > P.own0, cut_hi = S.cut && rb < P.own0 + ownN;
    int y0 = cut_lo ? ra : ra - (S.ring - 1) + S.rr - OMIN, y1 = cut_hi ? rb - 1 : rb - 1 + S.rr - OMIN;
    if (y0 < arr_lo) y0 = arr_lo;
    if (y1 > arr_hi - 1) y1 = arr_hi - 1;
    return (y1 >= y0 ? A[y1 + 1] - A[y0] : 0.0) + (double)kRowW0 * S.GR * ((cut_lo ? 1 : 0) + (cut_hi ? 1 : 0));
  };
  const long long total = (long long)planes * ownN;
  const double plane_cost = seg_cost(P.own0, P.own0 + ownN);
  // greedy fill with budget T starting at position b: returns the end of the range (> b unless one row exceeds T)
  auto fill = [&](long long b, double T) {
    double used = 0.0;
    long long e = b;
    while (e < total) {
      const int r = (int)(e % ownN);
      if (r == 0 && used + plane_cost <= T) { used += plane_cost; e += ownN; continue; }   // a whole plane fits
      // largest rb in (r, ownN] with used + seg_cost(own0 + r, own0 + rb) <= T (seg_cost is monotone in rb)
      int lo = r, hi = ownN;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (used + seg_cost(P.own0 + r, P.own0 + mid) <= T) lo = mid; else hi = mid - 1;
      }
      // cut mode: two cuts inside one plane stay at least GR rows apart (rows_grow_fix_kernel: one source per element)
      if (S.cut && r > 0 && used == 0.0 && lo < ownN && lo - r < S.GR) lo = r + S.GR < ownN ? r + S.GR : ownN;
      if (lo == r) break;
      used += seg_cost(P.own0 + r, P.own0 + lo);
      e += lo - r;
      if (lo < ownN) break;
    }
    return e;
  };
  auto ranges_needed = [&](double T) {
    long long b = 0;
    int n = 0;
    while (b < total) {
      const long long e = fill(b, T);
      if (e == b) return 1 << 30;
      b = e; ++n;
      if (n > grid) break;
    }
    return n;
  };
  double lo = 0.0, hi = plane_cost * planes + 1.0;
  for (int it = 0; it < 40; ++it) {
    const double mid = 0.5 * (lo + hi);
    if (ranges_needed(mid) <= grid) hi = mid; else lo = mid;
  }
  long long b = 0;
  S.bound[0] = 0;
  for (int c = 1; c <= grid; ++c) {
    if (b < total) b = fill(b, hi);
    S.bound[c] = (int)b;
  }
  S.bound[grid] = (int)total;
  if (S.cut) {
    // safety net of the cut mode: two cuts of one plane closer than GR rows -> partition again without cuts
    bool ok = true;
    int prev = -1;
    for (int c = 1; c < grid && ok; ++c) {
      const int gcut = S.bound[c];
      if (gcut % ownN == 0 || gcut == prev) continue;
      if (prev >= 0 && prev / ownN == gcut / ownN && gcut - prev < S.GR) ok = false;
      prev = gcut;
    }
    if (!ok) {
      S.cut = 0;
      rows_partition<INTERP>(P, S, reach, wc, planes, grid);        // (cached under its own key)
    }
  }
  RowsPartEntry& e = cache[cache_next];
  cache_next = (cache_next + 1) % 8;
  e.key = key; memcpy(e.bound, S.bound, sizeof(S.bound)); e.cut = S.cut; e.valid = true;
}

}  // namespace psl
