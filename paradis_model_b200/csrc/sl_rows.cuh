// Fused backward, round-2 design: one persistent, warp-specialised CTA per SM sweeps whole latitude
// circles.  One pass over the arrival points produces grad_u, grad_v AND grad_field, at every latitude
// (mid-latitudes and polar caps alike), deterministic and without atomics.
//
// Roles inside a CTA (one CTA per SM, launched once, walks a contiguous range of (plane, row) work):
//
//   loader     1 warp, one elected lane: streams the u, v, grad_out rows of the next arrival rows into
//              shared memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx), kRowStages
//              rows ahead of the producers.
//   producers  nP warps: per arrival point the departure trajectory, the stencil gather of `field`
//              with its derivative (grad_u, grad_v -> global, coalesced) and a 16-byte RECORD
//              {frac x, frac y, grad_out, (row class | departure column)} into a shared-memory row of
//              records.  Embarrassingly parallel: 4 x 32 consecutive columns per warp step, no scatter.
//   consumers  nC warps: each OWNS a strip of destination columns of the CTA-wide ring of `ring`
//              destination rows (full longitude circle, shared memory).  It scans the records of the
//              arrival columns that can reach its strip ([ja - hx, jb + hx), hx = longitudinal reach of
//              the row, the whole circle near the poles), and adds the stencil weights of the taps that
//              fall into ITS columns.  A destination row leaves the ring (coalesced float4 store to
//              grad_field) once no later arrival row can reach it.
//
// No trajectory is ever recomputed for a halo: a point is computed once per CTA and its record is read by
// the (one or two) consumers whose strips it touches.  The GeoCyclic cap rows fold back onto rows 1..p /
// H-1-p..H-2 (180 degrees shifted) when they are scattered, so the same kernel serves the polar caps.
//
// Determinism without atomics: a ring cell is only ever written by the consumer that owns its column;
// that consumer visits arrival rows, scan steps and tap phases in a fixed order; lanes of one step that
// hit the same departure cell are detected with one-byte tags and summed into the lowest lane in lane
// order (resolve_clashes), so every add has a single writer and a data-defined order.
//
// Cut mode (RowsPlan::cut, latitude bands): a segment that starts / ends inside a plane processes only its own
// arrival rows instead of replaying ring - 1 rows of its neighbour; the destination rows its arrival rows reach
// beyond the cut are parked (rows_park_row / rows_flush_row) and added to the rows their owner stored by
// rows_grow_fix_kernel -- one source per element and launch, so the result stays bit-reproducible.
//
// Pipelines (all mbarrier based, no __syncthreads after start-up):
//   stage_full / stage_free [kRowStages]   loader -> producers   (TMA transaction count / nP arrivals)
//   rec_full   / rec_free   [kRowRecs]     producers -> consumers (nP arrivals / nC arrivals)
//
// Contract: |floor(iy) - row| <= rr and |departure column - arrival column| <= hx(row).  Every point is
// checked by its producer; a violation marks the plane in `plane_flag` and the host always enqueues the
// general (two-kernel) path behind this kernel, which recomputes exactly the flagged planes.
#pragma once
#include "sl_device.cuh"

namespace psl {

#ifndef PSL_ROWS_STAGES
#define PSL_ROWS_STAGES 2
#endif
#ifndef PSL_ROWS_RECS
#define PSL_ROWS_RECS 3
#endif
constexpr int kRowStages = PSL_ROWS_STAGES;   // u, v, grad_out rows in flight (TMA)
constexpr int kRowRecs = PSL_ROWS_RECS;       // record rows in flight between producers and consumers
#ifndef PSL_ROWS_SUB
#define PSL_ROWS_SUB 4
#endif
constexpr int kStepSub = PSL_ROWS_SUB;   // 32-column sub-blocks per producer step
constexpr int kTagBytes = 512;     // clash tags per strip (hashed, power of two)
#ifndef PSL_ROWS_STREAMS
#define PSL_ROWS_STREAMS 1
#endif
constexpr int kStreams = PSL_ROWS_STREAMS;   // strips a consumer warp works on in an interleaved manner
constexpr int kRowsMaxCtas = 192;
// Warp budget: loader + producers + consumers.  20 warps = 640 threads -> 96 registers, no spills.  (Re-partitioning
// the register file between the roles with setmaxnreg -- 16 producers at 96-104 registers, loader + 7 consumers at
// 40-64 -- was tried: slower, 2.2-2.9 ms against 1.82, and two of the four splits hung; removed.)
#ifndef PSL_ROWS_WARPS
#define PSL_ROWS_WARPS 20
#endif
constexpr int kRowsWarps = PSL_ROWS_WARPS;
constexpr int kRowsMaxConsumers = kRowsWarps - 2;

struct RowsPlan {
  int planes, rr, ring;            // ring = 2 rr + NT destination rows
  int nP, nC;                      // producer / consumer warps (warp 0 is the loader)
  int nS;                          // strips = private rings (kStreams per consumer warp)
  int wc;                          // strip width (multiple of 4)
  int pitch, ring_stride;          // private ring of a consumer: (ring + NT - 1) rows of `pitch` floats = ring_stride
  float* guard;                    // [planes][outN][nS][NT - 1] guard columns of the retired rows (added by a post-kernel)
  int cut;                         // 1: a CTA range that starts / ends inside a plane does not replay the ring warm-up rows
                                   // of its neighbour; the partial destination rows either side of the cut go to `grow`
  int GR;                          // guard rows kept per side of a cut (rr + NT)
  float* grow;                     // [CTAs][2][GR][nS][pitch] partial destination rows beyond a cut (0: below the
                                   // start of the CTA's first segment, 1: above the end of its last one)
  int nsteps;                      // producer steps per arrival row = ceil(W / 128)
  int total_rows;                  // planes * ownN
  int bound[kRowsMaxCtas + 1];     // CTA k owns rows [bound[k], bound[k + 1]) of the concatenated (plane, own row)
                                   // space: equal COST (rows near the poles keep the consumers busy several times
                                   // longer), boundaries close to a plane boundary snapped onto it (host plan)
  const int* __restrict__ hx_tab;  // [H] longitudinal reach (cells) of an arrival row; >= W: whole circle
  unsigned char* plane_flag;       // [planes] set to 1 on a contract violation
  int out0, outN;                  // rows held by the output tensors
  unsigned off_stage, off_rec, off_tag, off_bar;   // byte offsets in dynamic shared memory (ring at 0)
};

// ---- mbarrier / bulk-copy wrappers (PTX; SASS: SYNCS.*, UBLKCP) ---------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  // (a suspend-time hint on try_wait was measured: fewer polls, but 3 % slower overall)
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(b)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// destination rows [ra, rb) of plane pl (global rows); arrival rows y_first .. y_last are processed (cut mode: a
// segment that starts / ends inside its plane processes its own arrival rows only, and its consumers flush the
// ring - 1 rows still in the ring after the last one)
struct RowsSeg { int pl, ra, rb, y_first, y_last; };

template <int INTERP>
__device__ __forceinline__ bool rows_next_seg(const Params& P, const RowsPlan& S, int& g, int g1, RowsSeg& s) {
  constexpr int OMIN = Stencil<INTERP>::OMIN;
  if (g >= g1) return false;
  s.pl = g / P.ownN;
  const int r = g - s.pl * P.ownN;
  const int n = min(P.ownN - r, g1 - g);
  s.ra = P.own0 + r; s.rb = s.ra + n;
  // destination row i = y - rr + OMIN is complete after arrival row y
  s.y_first = (S.cut && r > 0) ? s.ra : s.ra - (S.ring - 1) + S.rr - OMIN;       // starts / ends at a cut inside the plane
  s.y_last = (S.cut && r + n < P.ownN) ? s.rb - 1 : s.rb - 1 + S.rr - OMIN;
  g += n;
  return true;
}

// Lanes of one step that hit the same departure cell: every clashing cell is resolved by a ballot on the exact key
// and summed into its lowest lane in ascending lane order (single writer, data-defined order).  `lost`: this lane
// found another lane's id in the tag of its cell (a hashed tag may alias: that only costs a pass of the loop).
template <int NN>
__device__ __forceinline__ void rows_resolve_pending(int key, bool lost, int lane, float (&c)[NN], bool& writer) {
  unsigned pending = __ballot_sync(0xffffffffu, lost);
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
      for (int t = 0; t < NN; ++t) {
        const float o = __shfl_sync(0xffffffffu, c[t], src);
        if (lane == leader) c[t] += o;
      }
    }
    if (lane != leader && ((group >> lane) & 1u)) writer = false;
  }
}

// Record (16 bytes per arrival point, written once by its producer, read by the consumer(s) it concerns):
//   2x2 stencil: { g * (1 - tx), g * tx, ty, key }      4x4 stencil: { tx, ty, g, key }
// key: bits [31:16] ring slot of tap row 0 (the producer knows the row sequence of the segment), bit 15: the last
// tap column lies outside the padded plane (padding_mode="zeros"), bits [14:0] unpadded column of tap 0 wrapped
// into [0, W).  key < 0: no contribution (contract violated or non-finite coordinates).
__device__ __forceinline__ int rows_key(int slot0, int col0, bool last_out) {
  return (slot0 << 16) | (last_out ? 0x8000 : 0) | col0;
}

// The NT x NT contributions g * wy[a] * wx[b] of a record.
template <int INTERP>
__device__ __forceinline__ void rows_weights(const float4 rec, bool act, bool last_out,
                                             float (&cc)[Stencil<INTERP>::NT * Stencil<INTERP>::NT]) {
  constexpr int NT = Stencil<INTERP>::NT;
  if (INTERP == 1) {
    const float gx0 = act ? rec.x : 0.0f, gx1 = (act && !last_out) ? rec.y : 0.0f;
    const float wy1 = rec.z, wy0 = __fsub_rn(1.0f, wy1);
    cc[0] = __fmul_rn(gx0, wy0); cc[1] = __fmul_rn(gx1, wy0);
    cc[2] = __fmul_rn(gx0, wy1); cc[3] = __fmul_rn(gx1, wy1);
  } else {
    float wx[NT], wy[NT], d0[NT], d1[NT];
    axis_weights<INTERP, false>(rec.x, wx, d0);
    axis_weights<INTERP, false>(rec.y, wy, d1);
    const float g = act ? rec.z : 0.0f;
    if (last_out) wx[NT - 1] = 0.0f;
#pragma unroll
    for (int a = 0; a < NT; ++a) {
      const float gw = __fmul_rn(g, wy[a]);
#pragma unroll
      for (int b = 0; b < NT; ++b) cc[a * NT + b] = __fmul_rn(gw, wx[b]);
    }
  }
}

// ---- consumer: one step (32 records of each of the warp's kStreams strips), rows whose stencils stay inside
// rows 0 .. H-1 (no cap fold).
// A strip's ring is private: `pitch` columns = its wc own columns + NT-1 guard columns (taps that spill into the
// next strip; a post-kernel adds them to that strip's first columns), ring + NT-1 rows (the last NT-1 alias the
// first ones, folded together when a row retires).  A record belongs to the strip that owns the column of its
// tap 0, and all its taps sit at base + a * pitch + b: no wrap, no per-tap ownership test.
// The strips of a warp are advanced together: their rings are disjoint, so between two warp barriers there are
// kStreams independent load-add-store chains instead of one (the consumers are latency bound).
struct RowsStrip { float* ring; unsigned char* tag; int ja, wc; };

template <int INTERP>
__device__ __forceinline__ void rows_scatter_plain(const float4 (&rec)[kStreams], const bool (&inr)[kStreams],
                                                   const RowsStrip (&T)[kStreams], int pitch, int lane) {
  constexpr int NT = Stencil<INTERP>::NT;
  int key[kStreams], base[kStreams];
  bool act[kStreams], any_act = false;
#pragma unroll
  for (int s = 0; s < kStreams; ++s) {
    key[s] = inr[s] ? __float_as_int(rec[s].w) : -1;
    const int rel = (key[s] & 0x7fff) - T[s].ja;
    act[s] = key[s] >= 0 && (unsigned)rel < (unsigned)T[s].wc;
    base[s] = (key[s] >> 16) * pitch + rel;
    any_act = any_act || act[s];
  }
  if (!__any_sync(0xffffffffu, any_act)) return;
  float cc[kStreams][NT * NT];
  bool lost = false;
#pragma unroll
  for (int s = 0; s < kStreams; ++s) {
    rows_weights<INTERP>(rec[s], act[s], (key[s] & 0x8000) != 0, cc[s]);
    if (act[s]) T[s].tag[base[s] & (kTagBytes - 1)] = (unsigned char)lane;
  }
  __syncwarp();
  bool writer[kStreams], lst[kStreams];
#pragma unroll
  for (int s = 0; s < kStreams; ++s) {
    lst[s] = act[s] && T[s].tag[base[s] & (kTagBytes - 1)] != (unsigned char)lane;
    lost = lost || lst[s];
    writer[s] = act[s];
  }
  if (__any_sync(0xffffffffu, lost)) {
#pragma unroll
    for (int s = 0; s < kStreams; ++s) rows_resolve_pending<NT * NT>(act[s] ? base[s] : -1, lst[s], lane, cc[s], writer[s]);
  }
  float* q[kStreams];
#pragma unroll
  for (int s = 0; s < kStreams; ++s) q[s] = T[s].ring + (writer[s] ? base[s] : 0);
#pragma unroll
  for (int a = 0; a < NT; ++a) {
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      float v[kStreams];
#pragma unroll
      for (int s = 0; s < kStreams; ++s) v[s] = writer[s] ? q[s][a * pitch + b] : 0.0f;
#pragma unroll
      for (int s = 0; s < kStreams; ++s)
        if (writer[s]) q[s][a * pitch + b] = v[s] + cc[s][a * NT + b];
      __syncwarp();
    }
  }
}

// ---- consumer: one 32-record step of a row near a pole: tap rows outside 0 .. H-1 fold back through the
// GeoCyclic map (model/padding.py:26-37: reflect about the first / last row excluding it, 180 degrees
// shifted), so the owner of a tap row is decided per row (the folded rows belong to the strip half a circle
// away).  Two points with different departure cells can meet in one tap phase only when one of the taps is
// folded and the other is not, so every tap phase is split in two (plain taps, then folded taps); within each
// half distinct departure cells still mean distinct ring cells.
template <int INTERP>
__device__ __noinline__ void rows_scatter_fold(int W, int H, const float4 rec, bool inr, float* myring,
                                               unsigned char* tag, int pitch, int ring, int head, int y, int rr, int ja,
                                               int wc, int lane) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  constexpr int pad = INTERP;                    // padding width = interpolation id (advection.py:22-24)
  const int halfW = W >> 1;
  const int key = inr ? __float_as_int(rec.w) : -1;
  const int s0 = key >> 16, cx = key & 0x7fff;
  int t = s0 - head;                              // row class + rr
  if (t < 0) t += ring;
  const int i0 = y + (t - rr) + OMIN;             // unpadded row of tap row 0
  const int i_ret = y - rr + OMIN;                // row in slot `head`
  float cc[NT * NT];
  rows_weights<INTERP>(rec, key >= 0, (key & 0x8000) != 0, cc);
  const int k = key >= 0 ? (t * W + cx) : -1;     // same arrival row: (class, column) identifies the departure cell
  if (key >= 0) tag[k & (kTagBytes - 1)] = (unsigned char)lane;
  __syncwarp();
  const bool lost = key >= 0 && tag[k & (kTagBytes - 1)] != (unsigned char)lane;
  bool writer = key >= 0;
  rows_resolve_pending<NT * NT>(k, lost, lane, cc, writer);
  int cf = cx - halfW;                            // column of a folded tap row
  if (cf < 0) cf += W;
#pragma unroll
  for (int a = 0; a < NT; ++a) {
    int i = i0 + a;
    bool ok = writer && i >= -pad && i <= H - 1 + pad;      // outside the padded plane: zeros
    bool fold = false;
    if (i < 0) { i = -i; fold = true; }
    else if (i >= H) { i = 2 * (H - 1) - i; fold = true; }
    int sl = head + (i - i_ret);
    ok = ok && (unsigned)(i - i_ret) < (unsigned)ring;
    if (sl >= ring) sl -= ring;
    const int rel = (fold ? cf : cx) - ja;
    const bool mine = ok && (unsigned)rel < (unsigned)wc;
    float* q = myring + (mine ? sl * pitch + rel : 0);
    const bool any_fold = __any_sync(0xffffffffu, mine && fold);
#pragma unroll
    for (int b = 0; b < NT; ++b) {
      if (mine && !fold) q[b] += cc[a * NT + b];
      __syncwarp();
      if (any_fold) {
        if (mine && fold) q[b] += cc[a * NT + b];
        __syncwarp();
      }
    }
  }
}

// ---- producer: one arrival point -> record (+ grad_u, grad_v for the rows this segment owns) -----
template <bool EXACT, int INTERP, bool PEER, bool SMALL, typename T>
__device__ __forceinline__ float4 rows_point(const Params& P, const T* __restrict__ f, int pl, float mean0,
                                             float mean1, float sp, float cp, int y, int x, int rr, int hx, int hbase,
                                             int ring, bool core, float uu, float vv, float g, float lonp,
                                             bool& violated, float& ou, float& ov) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  Traj t;
  trajectory<EXACT, SMALL>(P, uu, vv, sp, cp, lonp, t);
  const float fx = floorf(t.ix), fy = floorf(t.iy);
  const float tx = __fsub_rn(t.ix, fx), ty = __fsub_rn(t.iy, fy);
  const int x0 = (int)fx + OMIN;                 // padded column of tap 0
  const int cls = (int)fy - (y + P.p);           // row class
  int dx = x0 - P.p - x;                         // longitudinal cell displacement of tap 0
  if (dx < -P.halfW) dx += P.W; else if (dx >= P.halfW) dx -= P.W;
  const bool in_ring = (unsigned)(cls + rr) <= (unsigned)(2 * rr);
  if (!in_ring || dx < -hx || dx > hx - NT + 1) violated = true;
  if (core) {
    float val, ddx, ddy;
    stencil_eval<INTERP, true, PEER>(P, f, pl, t, mean0, mean1, val, ddx, ddy);
    velocity_grads<EXACT>(P, t, sp, cp, g * ddx, g * ddy, ou, ov);
  }
  int col0 = x + dx;
  if (col0 < 0) col0 += P.W; else if (col0 >= P.W) col0 -= P.W;
  const bool valid = in_ring && (unsigned)col0 < (unsigned)P.W;   // false for non-finite coordinates
  int s0 = hbase + cls + rr;                     // ring slot of tap row 0 (hbase: slot of the row retiring after y)
  if (s0 >= ring) s0 -= ring;
  const int key = valid ? rows_key(s0, col0, x0 + NT - 1 >= P.Wp) : -1;
  if (INTERP == 1) return make_float4(__fmul_rn(g, __fsub_rn(1.0f, tx)), __fmul_rn(g, tx), ty, __int_as_float(key));
  return make_float4(tx, ty, g, __int_as_float(key));
}

// FAST math: two arrival points of one row at a time, trajectory and Jacobian on the packed fp32x2 pipe
// (bit-identical to rows_point<false, ...> for each of them)
template <int INTERP, bool PEER, typename T>
__device__ __forceinline__ void rows_pair(const Params& P, const T* __restrict__ f, int pl, float mean0, float mean1,
                                          float sp, float cp, int y, const int (&x)[2], int rr, int hx, int hbase, int ring,
                                          bool core, f2 uu, f2 vv, f2 g, f2 lonp, bool& violated, float4 (&rec)[2], f2& ou,
                                          f2& ov) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  Traj2 t2;
  trajectory_2(P, uu, vv, f2s(sp), f2s(cp), lonp, t2);
  float ddx[2] = {0.0f, 0.0f}, ddy[2] = {0.0f, 0.0f};
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const Traj t = traj_half(t2, e);
    const float ge = e ? g.y : g.x;
    const float fx = floorf(t.ix), fy = floorf(t.iy);
    const float tx = __fsub_rn(t.ix, fx), ty = __fsub_rn(t.iy, fy);
    const int x0 = (int)fx + OMIN;                 // padded column of tap 0
    const int cls = (int)fy - (y + P.p);           // row class
    int dx = x0 - P.p - x[e];                      // longitudinal cell displacement of tap 0
    if (dx < -P.halfW) dx += P.W; else if (dx >= P.halfW) dx -= P.W;
    const bool in_ring = (unsigned)(cls + rr) <= (unsigned)(2 * rr);
    if (!in_ring || dx < -hx || dx > hx - NT + 1) violated = true;
    if (core) {
      float val;
      stencil_eval<INTERP, true, PEER>(P, f, pl, t, mean0, mean1, val, ddx[e], ddy[e]);
    }
    int col0 = x[e] + dx;
    if (col0 < 0) col0 += P.W; else if (col0 >= P.W) col0 -= P.W;
    const bool valid = in_ring && (unsigned)col0 < (unsigned)P.W;   // false for non-finite coordinates
    int s0 = hbase + cls + rr;                     // ring slot of tap row 0
    if (s0 >= ring) s0 -= ring;
    const int key = valid ? rows_key(s0, col0, x0 + NT - 1 >= P.Wp) : -1;
    if (INTERP == 1) rec[e] = make_float4(__fmul_rn(ge, __fsub_rn(1.0f, tx)), __fmul_rn(ge, tx), ty, __int_as_float(key));
    else rec[e] = make_float4(tx, ty, ge, __int_as_float(key));
  }
  if (core) velocity_grads_2(P, t2, f2s(sp), f2s(cp), mul2(g, make_float2(ddx[0], ddx[1])), mul2(g, make_float2(ddy[0], ddy[1])), ou, ov);
}

// ---- cold paths of the cut mode (not inlined: the hot loops of the kernel keep their register allocation) ----
__device__ __noinline__ void rows_park_row(const float* row, float* dst, int pitch, int lane) {
  for (int k = 4 * lane; k < pitch; k += 128)
    __stcs(reinterpret_cast<float4*>(dst + k), *reinterpret_cast<const float4*>(row + k));
}

// retire ring slot `head` without a new arrival row: alias rows in, row out (own row -> orow + guard columns gcol;
// partial row beyond the cut -> park; neither -> dropped), slot cleared
__device__ __noinline__ void rows_flush_row(float* ringp, int head, int ring, int pitch, int wc, int ng, float* orow,
                                            float* gcol, float* park, int lane) {
  float* row = ringp + head * pitch;
  if (head < ng) {
    float* alias = ringp + (ring + head) * pitch;
    for (int k = 4 * lane; k < pitch; k += 128) {
      float4 a = *reinterpret_cast<const float4*>(row + k);
      const float4 b = *reinterpret_cast<const float4*>(alias + k);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      *reinterpret_cast<float4*>(row + k) = a;
      *reinterpret_cast<float4*>(alias + k) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();
  }
  if (orow) {
    for (int k = 4 * lane; k < wc; k += 128)
      __stcs(reinterpret_cast<float4*>(orow + k), *reinterpret_cast<const float4*>(row + k));
    if (lane < ng) gcol[lane] = row[wc + lane];
  } else if (park) {
    for (int k = 4 * lane; k < pitch; k += 128)
      __stcs(reinterpret_cast<float4*>(park + k), *reinterpret_cast<const float4*>(row + k));
  }
  __syncwarp();
  for (int k = 4 * lane; k < pitch; k += 128) *reinterpret_cast<float4*>(row + k) = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
}

// T: storage type of field, u, v, grad_u, grad_v.  A stage holds the u, v rows (W * sizeof(T) bytes each) and the fp32
// grad_out row, back to back; its size is 3 W floats whatever T is, so the plan does not depend on it.
template <bool EXACT, int INTERP, bool PEER, typename T>
__global__ void __launch_bounds__(kRowsWarps * 32, 1) sl_bwd_rows_kernel(const Params P, const RowsPlan S) {
  constexpr int NT = Stencil<INTERP>::NT, OMIN = Stencil<INTERP>::OMIN;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int W = P.W, ring = S.ring, rr = S.rr;
  float* ring_base = reinterpret_cast<float*>(smem_raw);
  float* stage_base = reinterpret_cast<float*>(smem_raw + S.off_stage);      // [kRowStages][3][W]
  float4* rec_base = reinterpret_cast<float4*>(smem_raw + S.off_rec);        // [kRowRecs][W]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + S.off_bar);
  uint64_t* stage_full = bars;
  uint64_t* stage_free = bars + kRowStages;
  uint64_t* rec_full = bars + 2 * kRowStages;
  uint64_t* rec_free = bars + 2 * kRowStages + kRowRecs;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kRowStages; ++i) { mbar_init(&stage_full[i], 1); mbar_init(&stage_free[i], S.nP); }
    for (int i = 0; i < kRowRecs; ++i) { mbar_init(&rec_full[i], S.nP); mbar_init(&rec_free[i], S.nC); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  int g = S.bound[blockIdx.x];
  const int g1 = S.bound[blockIdx.x + 1];
  const int arr_lo = P.arr0, arr_hi = P.arr0 + P.arrN;
  RowsSeg sg;

  // role of this warp: 0 = loader, then nP producers, then nC consumers
  const bool is_loader = warp == 0;
  const int prod0 = 1;
  const bool is_producer = warp >= prod0 && warp < prod0 + S.nP;
  const int cons0 = 1 + S.nP;

  if (is_loader) {
    // ===================================== loader =====================================
    // (an L2 prefetch of the `field` row entering the stencil window, issued from this warp's idle lanes, was
    // measured: no effect, 1.837 against 1.835 ms)
    if (lane != 0) return;
    int n = 0;
    const uint32_t row_bytes = (uint32_t)W * 4u, uv_bytes = (uint32_t)(W * sizeof(T));   // bf16: W % 8 == 0 (16-byte copies)
    while (rows_next_seg<INTERP>(P, S, g, g1, sg)) {
      const T* up = plane_ptr(as<T>(P.u), P.u_sB, P.V, P.uvgN, W, sg.pl);
      const T* vp = plane_ptr(as<T>(P.v), P.v_sB, P.V, P.uvgN, W, sg.pl);
      const float* gp = plane_ptr(P.gout, P.gout_sB, P.V, P.uvgN, W, sg.pl);
      for (int y = max(sg.y_first, arr_lo); y <= min(sg.y_last, arr_hi - 1); ++y, ++n) {
        const int st = n % kRowStages;
        mbar_wait(&stage_free[st], ((n / kRowStages) & 1) ^ 1);
        T* dst = reinterpret_cast<T*>(stage_base + (size_t)st * 3 * W);
        mbar_arrive_expect_tx(&stage_full[st], kIsF32<T> ? 3 * row_bytes : 2 * uv_bytes + row_bytes);
        bulk_g2s(dst, arr_row<PEER>(P, up, 0, sg.pl, y), uv_bytes, &stage_full[st]);
        bulk_g2s(dst + W, arr_row<PEER>(P, vp, 1, sg.pl, y), uv_bytes, &stage_full[st]);
        bulk_g2s(dst + 2 * W, arr_row<PEER>(P, gp, 2, sg.pl, y), row_bytes, &stage_full[st]);
      }
    }
    return;
  }

  if (is_producer) {
    // ==================================== producers ====================================
    const int p = warp - prod0;
    int n = 0;
    int next = p;                     // global step index (row sequence number * nsteps + step) this warp does next
    bool violated = false;
    int flagged_pl = -1;
    while (rows_next_seg<INTERP>(P, S, g, g1, sg)) {
      const int pl = sg.pl;
      const int b = pl / P.V, c = pl - b * P.V;
      const T* f = plane_ptr_bc(as<T>(P.field), P.field_sB, b, c, P.fldN, W);
      T* gu_pl = P.gu ? as<T>(P.gu) + (long long)pl * S.outN * W : nullptr;
      T* gv_pl = P.gu ? as<T>(P.gv) + (long long)pl * S.outN * W : nullptr;
      float mean0 = 0.0f, mean1 = 0.0f, gm0 = 0.0f, gm1 = 0.0f;
      if (P.pole_fix) {
        mean0 = __ldg(P.fmean + 2 * pl); mean1 = __ldg(P.fmean + 2 * pl + 1);
        gm0 = __ldg(P.gmean + 2 * pl); gm1 = __ldg(P.gmean + 2 * pl + 1);
      }
      const int y_begin = max(sg.y_first, arr_lo);
      int hbase = (y_begin - sg.y_first) % ring;      // ring slot of the row that retires after the arrival row
      for (int y = y_begin; y <= min(sg.y_last, arr_hi - 1); ++y, ++n, hbase = hbase + 1 == ring ? 0 : hbase + 1) {
        const int row_end = (n + 1) * S.nsteps;
        const int st = n % kRowStages, rs = n % kRowRecs;
        // Every producer warp takes part in every row of both pipelines (it arrives on stage_free and rec_full
        // whether or not one of the row's steps is its own): a parity wait can only tell the current phase of an
        // mbarrier from the previous one, so no waiter may fall -- or run -- more than one phase away from it.
        mbar_wait(&stage_full[st], (n / kRowStages) & 1);
        mbar_wait(&rec_free[rs], ((n / kRowRecs) & 1) ^ 1);
        if (next >= row_end) {
          if (lane == 0) { mbar_arrive(&stage_free[st]); mbar_arrive(&rec_full[rs]); }
          continue;
        }
        const T* su = reinterpret_cast<const T*>(stage_base + (size_t)st * 3 * W);     // u | v | grad_out (fp32)
        const float* sg_row = reinterpret_cast<const float*>(su + 2 * W);
        float4* recs = rec_base + (size_t)rs * W;
        const float sp = __ldg(P.sin_lat + y), cp = __ldg(P.cos_lat + y);
        const int hx = __ldg(S.hx_tab + y);
        const bool core = (y >= sg.ra) && (y < sg.rb) && gu_pl != nullptr;
        const bool pole_row = P.pole_fix && (y == 0 || y == P.H - 1);
        const float gpole = y == 0 ? gm0 : gm1;
        for (; next < row_end; next += S.nP) {
          const int xb = (next - n * S.nsteps) * (32 * kStepSub);
          float uu[kStepSub], vv[kStepSub], gg[kStepSub], ll[kStepSub];
#pragma unroll
          for (int j = 0; j < kStepSub; ++j) {
            const int x = min(xb + 32 * j + lane, W - 1);   // lanes past the row end redo its last point (not stored)
            uu[j] = ld_f(su + x);
            vv[j] = ld_f(su + W + x);
            gg[j] = pole_row ? gpole : sg_row[x];           // adjoint of the output pole mean (advection.py:169)
            ll[j] = __ldg(P.lon + x);
          }
          const bool last_step = next + S.nP >= row_end;     // this warp's last step in this row
          __syncwarp();
          if (last_step && lane == 0) mbar_arrive(&stage_free[st]);
          // one sub-block after the other, results stored at once: the compiler interleaves as far as the register
          // budget allows (the kernel runs 1024 threads per SM at 64 registers)
          T* gu_row = core ? gu_pl + (long long)(y - S.out0) * W : nullptr;
          T* gv_row = core ? gv_pl + (long long)(y - S.out0) * W : nullptr;
#if !defined(PSL_DBG_NOPRODUCE) && !defined(PSL_ROWS_NO_PAIRS)
          if (!EXACT && (kStepSub % 2) == 0) {
#pragma unroll
            for (int j = 0; j < kStepSub; j += 2) {
              if (xb + 32 * j < W) {                   // uniform: the last step of a row may be short
                const int x0 = xb + 32 * j + lane, x1 = x0 + 32;
                const int xs[2] = {min(x0, W - 1), min(x1, W - 1)};
                float4 rec[2];
                f2 ou = f2s(0.0f), ov = f2s(0.0f);
                rows_pair<INTERP, PEER>(P, f, pl, mean0, mean1, sp, cp, y, xs, rr, hx, hbase, ring, core,
                                        make_float2(uu[j], uu[j + 1]), make_float2(vv[j], vv[j + 1]),
                                        make_float2(gg[j], gg[j + 1]), make_float2(ll[j], ll[j + 1]), violated, rec, ou, ov);
                if (x0 < W) {
                  recs[x0] = rec[0];
                  if (core) { stcs_f(gu_row + x0, ou.x); stcs_f(gv_row + x0, ov.x); }
                }
                if (x1 < W) {
                  recs[x1] = rec[1];
                  if (core) { stcs_f(gu_row + x1, ou.y); stcs_f(gv_row + x1, ov.y); }
                }
              }
            }
          } else
#endif
          {
#pragma unroll
          for (int j = 0; j < kStepSub; ++j) {
            if (xb + 32 * j < W) {                     // uniform: the last step of a row may be short
              const int x = xb + 32 * j + lane;
              float ou = 0.0f, ov = 0.0f;
#ifdef PSL_DBG_NOPRODUCE
              const float4 rec = make_float4(uu[j], vv[j], gg[j], __int_as_float(rows_key(hbase + rr, min(x, W - 1), false)));
              ou = uu[j]; ov = vv[j];
#else
              const float4 rec = rows_point<EXACT, INTERP, PEER, false>(P, f, pl, mean0, mean1, sp, cp, y, min(x, W - 1), rr, hx,
                                                                        hbase, ring, core, uu[j], vv[j], gg[j], ll[j], violated, ou, ov);
#endif
              if (x < W) {
                recs[x] = rec;
                if (core) { stcs_f(gu_row + x, ou); stcs_f(gv_row + x, ov); }
              }
            }
          }
          }
          if (last_step) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&rec_full[rs]);
          }
        }
      }
      if (__any_sync(0xffffffffu, violated) && flagged_pl != pl) {
        if (lane == 0) S.plane_flag[pl] = 1;
        flagged_pl = pl;
      }
      violated = false;
    }
    return;
  }

  if (warp >= cons0 && warp < cons0 + S.nC) {
    // ==================================== consumers ====================================
    const int cidx = warp - cons0;
    const int pitch = S.pitch;
    RowsStrip T[kStreams];
    int sidx[kStreams];
#pragma unroll
    for (int q = 0; q < kStreams; ++q) {
      sidx[q] = cidx * kStreams + q;                       // strips past the last one are empty (wc = 0)
      const int ja = min(sidx[q] * S.wc, W);
      T[q].ja = ja; T[q].wc = min(ja + S.wc, W) - ja;
      const int slot = min(sidx[q], S.nS - 1);
      T[q].ring = ring_base + (size_t)slot * S.ring_stride;
      T[q].tag = smem_raw + S.off_tag + slot * kTagBytes;
    }
    int n = 0;
    while (rows_next_seg<INTERP>(P, S, g, g1, sg)) {
      float* gf_pl = P.gfield + (long long)sg.pl * S.outN * W;
      float* guard_pl = S.guard + (long long)sg.pl * S.outN * S.nS * (NT - 1);
#pragma unroll
      for (int q = 0; q < kStreams; ++q)
        if (T[q].wc > 0)
          for (int k = 4 * lane; k < S.ring_stride; k += 128)
            *reinterpret_cast<float4*>(T[q].ring + k) = make_float4(0.f, 0.f, 0.f, 0.f);
      __syncwarp();
      int head = 0;
      for (int y = sg.y_first; y <= sg.y_last; ++y) {
        if (y >= arr_lo && y < arr_hi) {
          const int rs = n % kRowRecs;
          mbar_wait(&rec_full[rs], (n / kRowRecs) & 1);
          const float4* recs = rec_base + (size_t)rs * W;
          const int hx = __ldg(S.hx_tab + y);
          const bool fold_row = (y + OMIN - rr < 0) || (y + OMIN + rr + NT - 1 >= P.H);
          // Lane l of stream q visits the records start_q + l * k + s, s = 0 .. k-1: the lanes of one step are
          // k >= len / 32 columns apart, so two of them rarely share a departure cell (consecutive columns clash
          // about twice per step with white-noise velocities; the records sit in shared memory, any order costs
          // the same).  k not a multiple of 4: the ring accesses of a step then spread over the banks.
          int len = S.wc + 2 * hx;
          const bool whole = hx >= W || len >= W;
          if (whole) len = W;
          int k = (len + 31) >> 5;
          if ((k & 3) == 0) ++k;
          int idx[kStreams];
          bool inr[kStreams];
          float4 rec[kStreams];
#pragma unroll
          for (int q = 0; q < kStreams; ++q) {
            int start = whole ? 0 : T[q].ja - hx;
            if (start < 0) start += W;
            idx[q] = start + lane * k;                   // < 2 W + 32
            if (idx[q] >= W) idx[q] -= W;
            if (idx[q] >= W) idx[q] -= W;
            inr[q] = lane * k < len && T[q].wc > 0;
            rec[q] = inr[q] ? recs[idx[q]] : make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
          }
          for (int s = 0; s < k; ++s) {
            // fetch the next records before the ring updates of these (the compiler cannot move a shared-memory
            // load across them)
            float4 nxt[kStreams];
            bool inn[kStreams];
#pragma unroll
            for (int q = 0; q < kStreams; ++q) {
              idx[q] = idx[q] + 1 == W ? 0 : idx[q] + 1;
              inn[q] = (s + 1 < k) && (lane * k + s + 1 < len) && T[q].wc > 0;
              nxt[q] = recs[idx[q]];                       // always a valid address; `inn` masks the key when it is used
            }
#ifndef PSL_DBG_NOCONSUME
            if (fold_row) {
#pragma unroll
              for (int q = 0; q < kStreams; ++q)
                rows_scatter_fold<INTERP>(W, P.H, rec[q], inr[q], T[q].ring, T[q].tag, pitch, ring, head, y, rr, T[q].ja,
                                          T[q].wc, lane);
            } else {
              rows_scatter_plain<INTERP>(rec, inr, T, pitch, lane);
            }
#endif
#pragma unroll
            for (int q = 0; q < kStreams; ++q) { rec[q] = nxt[q]; inr[q] = inn[q]; }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&rec_free[rs]);
          ++n;
        }
        // retire destination row i = y - rr + OMIN (slot `head`); slots 0 .. NT-2 first take in their alias rows
        const int i = y - rr + OMIN;
#pragma unroll
        for (int q = 0; q < kStreams; ++q) {
          if (T[q].wc <= 0) continue;
          float* row = T[q].ring + head * pitch;
          if (head < NT - 1) {
            float* alias = T[q].ring + (ring + head) * pitch;
            for (int k = 4 * lane; k < pitch; k += 128) {
              float4 a = *reinterpret_cast<const float4*>(row + k);
              const float4 b = *reinterpret_cast<const float4*>(alias + k);
              a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
              *reinterpret_cast<float4*>(row + k) = a;
              *reinterpret_cast<float4*>(alias + k) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            __syncwarp();
          }
          if (i >= sg.ra && i < sg.rb) {
            float* orow = gf_pl + (long long)(i - S.out0) * W + T[q].ja;
            for (int k = 4 * lane; k < T[q].wc; k += 128)
              __stcs(reinterpret_cast<float4*>(orow + k), *reinterpret_cast<const float4*>(row + k));
            if (lane < NT - 1)
              guard_pl[((long long)(i - S.out0) * S.nS + sidx[q]) * (NT - 1) + lane] = row[T[q].wc + lane];
          } else if (S.cut && i < sg.ra && i >= P.own0 && sg.ra > P.own0) {
            // cut mode, rows below the start cut: partial rows of the neighbouring segment (this segment's arrival rows
            // reach across the cut); the whole ring row, guard columns included, is parked for rows_grow_fix_kernel
            rows_park_row(row, S.grow + ((((size_t)blockIdx.x * 2) * S.GR + (i - (sg.ra - S.GR))) * S.nS + sidx[q]) * pitch,
                          pitch, lane);
          }
          __syncwarp();
          for (int k = 4 * lane; k < pitch; k += 128) *reinterpret_cast<float4*>(row + k) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncwarp();
        head = head + 1 == ring ? 0 : head + 1;
      }
      if (S.cut && sg.rb < P.own0 + P.ownN) {
        // cut mode, end cut: retire the ring - 1 rows still in the ring -- the last own rows, then the partial rows
        // above the cut (parked; rows outside the own window belong to a latitude neighbour or do not exist)
        for (int t = 0; t < ring - 1; ++t) {
          const int i = sg.y_last + 1 + t - rr + OMIN;
#pragma unroll
          for (int q = 0; q < kStreams; ++q) {
            if (T[q].wc <= 0) continue;
            // (a segment shorter than the ring still holds rows BELOW its start cut here)
            const bool own = i >= sg.ra && i < sg.rb;
            float* orow = own ? gf_pl + (long long)(i - S.out0) * W + T[q].ja : nullptr;
            float* gcol = own ? guard_pl + ((long long)(i - S.out0) * S.nS + sidx[q]) * (NT - 1) : nullptr;
            float* park = nullptr;
            if (i >= sg.rb && i < P.own0 + P.ownN)
              park = S.grow + ((((size_t)blockIdx.x * 2 + 1) * S.GR + (i - sg.rb)) * S.nS + sidx[q]) * pitch;
            else if (i < sg.ra && i >= P.own0 && sg.ra > P.own0)
              park = S.grow + ((((size_t)blockIdx.x * 2) * S.GR + (i - (sg.ra - S.GR))) * S.nS + sidx[q]) * pitch;
            rows_flush_row(T[q].ring, head, ring, pitch, T[q].wc, NT - 1, orow, gcol, park, lane);
          }
          head = head + 1 == ring ? 0 : head + 1;
        }
      }
    }
  }
}

// Guard columns (taps that spilled over the end of a consumer's strip) are added to the first columns of the
// next strip: one thread per (plane, row, strip, guard column); every target cell has one source.
__global__ void rows_guard_fix_kernel(float* __restrict__ gfield, const float* __restrict__ guard, long long rows_total,
                                      int W, int nC, int wc, int ng) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows_total * nC * ng) return;
  const int gcol = (int)(idx % ng);
  const int c = (int)((idx / ng) % nC);
  const long long row = idx / ((long long)ng * nC);
  int col = min((c + 1) * wc, W) + gcol;
  if (col >= W) col -= W;
  gfield[row * W + col] += guard[idx];
}

// Cut mode: the partial destination rows a CTA accumulated beyond the cuts of its range are added to the rows their
// owner stored.  One launch per side (first the rows above the ends, then the rows below the starts); cuts of one plane
// are at least GR rows apart (host partition), so within a launch every gfield element has at most one source.  A guard
// row is a whole ring row per strip: `wc` main columns plus NT - 1 guard columns that belong to the next strip's first
// columns (the last strip's wrap to column 0), as in rows_guard_fix_kernel.
__global__ void rows_grow_fix_kernel(float* __restrict__ gfield, const RowsPlan S, int side, int W, int own0, int ownN,
                                     int NT, int OMIN) {
  // grid: x = float4 groups of a row, y = guard row j, z = CTA of the sweep
  const int c = blockIdx.z, j = blockIdx.y;
  const int col = 4 * (blockIdx.x * blockDim.x + threadIdx.x);
  if (col >= W || S.bound[c + 1] <= S.bound[c]) return;
  const int g = side ? S.bound[c + 1] : S.bound[c];
  const int pl = g / ownN, r = g - pl * ownN;
  if (r == 0) return;                                        // a plane boundary (or the end of the work) is not a cut
  const int il = side ? r + j : r - S.GR + j;                // own-row index of the destination row
  if (side) { if (j >= S.rr + OMIN + NT - 1 || il >= ownN) return; }
  else      { if (j < S.GR - (S.rr - OMIN) || il < 0) return; }
  const int s = col / S.wc, k = col - s * S.wc;              // strips start at multiples of 4: one strip per float4
  const float* blk = S.grow + (((size_t)c * 2 + side) * S.GR + j) * S.nS * S.pitch;
  float4 v = *reinterpret_cast<const float4*>(blk + s * S.pitch + k);
  if (k == 0) {
    const int sp = s == 0 ? S.nS - 1 : s - 1;
    const float* gc = blk + sp * S.pitch + (min((sp + 1) * S.wc, W) - sp * S.wc);
    v.x += gc[0];
    if (NT - 1 > 1) { v.y += gc[1]; v.z += gc[2]; }
  }
  float4* dst = reinterpret_cast<float4*>(gfield + ((long long)pl * S.outN + (own0 + il - S.out0)) * W + col);
  float4 a = *dst;
  a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
  *dst = a;
}

}  // namespace psl
