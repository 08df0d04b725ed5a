/*
 * paradis_sl.h -- C ABI of libparadis_sl.so (sm_100a only).
 *
 * B200-native semi-Lagrangian advection operator + GeoCyclic padding for PARADIS.
 * Every entry point replaces a piece of the reference's Python hot path; the
 * reference interface it stands in for is cited as (file:line) relative to the
 * reference repository root.
 *
 * Conventions
 *   - All tensors are fp32, NCHW, W innermost, device pointers unless the
 *     function name ends in _host.  bf16 storage of the advection core's field, u, v
 *     and their gradients: include/paradis_sl_bf16.h (same struct and status codes).
 *   - The caller owns every buffer (inputs, outputs, workspace).  The library
 *     never allocates or frees device memory and keeps no pointer after return.
 *   - Calls are asynchronous on `stream` (a cudaStream_t passed as void*), never
 *     synchronise the host and keep no global mutable state other than the
 *     thread-local last-error string.
 *   - Return value: 0 = OK, otherwise a paradis_status code;
 *     paradis_last_error() gives the message for the calling thread.
 *   - There is no CPU fallback.
 */
#ifndef PARADIS_SL_H_
#define PARADIS_SL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PARADIS_SL_ABI_VERSION 2

typedef enum paradis_status {
  PARADIS_OK = 0,
  PARADIS_ERR_BAD_SHAPE = 1,      /* non-positive dims, H < pad+2, windows outside the mesh ... */
  PARADIS_ERR_ODD_WIDTH = 2,      /* model/padding.py:21 "Number of longitude points must be even" */
  PARADIS_ERR_BAD_INTERP = 3,
  PARADIS_ERR_NULL_POINTER = 4,
  PARADIS_ERR_WORKSPACE = 5,      /* workspace too small */
  PARADIS_ERR_CUDA = 6,           /* launch / runtime error, see paradis_last_error() */
  PARADIS_ERR_DISPLACEMENT = 7,   /* device-side: displacement above PARADIS_SL_MAX_DISP_ROWS, or a
                                     departure stencil outside the rows held by `field` (halo too small) */
  PARADIS_ERR_NO_DEVICE = 8
} paradis_status;

/* interpolation = padding width of the reference (model/advection.py:22-24) */
#define PARADIS_INTERP_BILINEAR 1
#define PARADIS_INTERP_BICUBIC 2

/* arithmetic of the departure-point chain */
#define PARADIS_MATH_FAST 0  /* fused multiply-adds, reciprocal scaling of pixel coordinates */
#define PARADIS_MATH_EXACT 1 /* replays the reference's fp32 op order (advection.py:131-150 +
                                ATen GridSampler.h:27-36): no FMA contraction, IEEE divides */

/* Largest |floor(iy) - arrival row| the deterministic adjoint tracks (int8 classes). */
#define PARADIS_SL_MAX_DISP_ROWS 126

/*
 * Geometry of the (separable) lat-lon mesh.  Replaces the non-persistent buffers
 * registered in model/advection.py:58-72.  The tables are device arrays over the
 * GLOBAL mesh; the trigonometric tables are computed by the caller with the same
 * fp32 torch ops the reference applies to lat_grid (advection.py:86-87) so that
 * EXACT mode sees identical values.
 *
 * Row windows (latitude-band decomposition, SURVEY 8e).  Every tensor of a call
 * holds full longitude circles of a contiguous range of global rows:
 *   own : rows this call produces  (out, grad_field, grad_u, grad_v)
 *   arr : rows held by u, v (and grad_out in backward); must contain `own`
 *   fld : rows held by field; must contain every departure stencil of `own`
 * Single GPU: all three are (0, H).
 */
typedef struct paradis_sl_geom {
  int32_t H, W;
  const float* sin_lat; /* [H] sin(lat_grid[:,0]) */
  const float* cos_lat; /* [H] cos(lat_grid[:,0]) */
  const float* lon;     /* [W] lon_grid[0,:] (radians) */
  float min_lat, d_lat; /* advection.py:66,71 */
  float min_lon, d_lon; /* advection.py:68,70 */
  int32_t own_row0, own_rows;
  int32_t arr_row0, arr_rows;
  int32_t fld_row0, fld_rows;
  /* Optional peer halos of `field` (fused halo exchange over NVLink peer memory): instead of
   * assembling the neighbours' boundary rows into `field`, pass pointers to them where they live
   * (e.g. the neighbour GPUs' symmetric-memory outboxes, mapped into this process).  Each is
   * [B*V, fld_peer_rows, W] and holds global rows [fld_row0 - fld_peer_rows, fld_row0) resp.
   * [fld_row0 + fld_rows, fld_row0 + fld_rows + fld_peer_rows).  The kernels load stencil taps that
   * fall there straight from the peer.  NULL / 0 when unused. */
  const float* fld_peer_lo;
  const float* fld_peer_hi;
  int32_t fld_peer_rows;
  /* Same for the arrival-window tensors of the backward, index 0 = u, 1 = v, 2 = grad_out.  When
   * arr_peer_rows > 0 the three tensors hold only the rows of the arr window that are NOT covered by a
   * non-NULL peer pointer: the first arr_peer_rows rows of the window are read from arr_peer_lo[k]
   * (if non-NULL) and the last arr_peer_rows rows from arr_peer_hi[k], each [B*V, arr_peer_rows, W].
   * With both sides present the tensors are [B, V, arr_rows - 2 * arr_peer_rows, W]. */
  const float* arr_peer_lo[3];
  const float* arr_peer_hi[3];
  int32_t arr_peer_rows;
} paradis_sl_geom;

int paradis_sl_abi_version(void);
const char* paradis_last_error(void);

/* ---- GeoCyclic padding: model/padding.py:11-39 ------------------------------------
 * y[planes, H+2p, W+2p] = pad(x[planes, H, W]);   planes = B*C.
 * bwd is the adjoint (fold-add of the pads back onto their sources), deterministic. */
int paradis_geocyclic_pad_fwd(const float* x, float* y, int64_t planes, int H, int W, int p,
                              void* stream);
int paradis_geocyclic_pad_bwd(const float* gy, float* gx, int64_t planes, int H, int W, int p,
                              void* stream);

/* ---- Depthwise convolution with the GeoCyclic padding applied on the fly ------------------------
 * Replaces `GeoCyclicPadding((k-1)/2)` + depthwise `nn.Conv2d(C, C, k, groups=C)` of SepConv
 * (model/blocks.py:92-116) and of the static encoder (model/paradis.py:186-190) without materialising
 * the padded tensor.  x, y, gy, gx: [B, C, H, W]; weight: [C, 1, k, k] (k = 3, 5 or 7); bias: [C] or NULL.
 * All three are deterministic (no atomics).  bwd_weight needs caller scratch of
 * paradis_geocyclic_dwconv_wgrad_workspace() bytes; gbias may be NULL. */
int paradis_geocyclic_dwconv_fwd(const float* x, const float* weight, const float* bias, float* y, int B,
                                 int C, int H, int W, int k, void* stream);
int paradis_geocyclic_dwconv_bwd_input(const float* gy, const float* weight, float* gx, int B, int C,
                                       int H, int W, int k, void* stream);
size_t paradis_geocyclic_dwconv_wgrad_workspace(int B, int C, int H, int W, int k);
int paradis_geocyclic_dwconv_bwd_weight(const float* x, const float* gy, float* gweight, float* gbias,
                                        int B, int C, int H, int W, int k, void* workspace,
                                        size_t workspace_bytes, void* stream);

/* PhysicalDownsample (model/blocks.py:57-71): GeoCyclic pad 2 + AvgPool2d(kernel 5, stride) in one kernel that only
 * computes the strided outputs.  x [B, C, H, W] -> y [B, C, (H - 1) / stride + 1, (W - 1) / stride + 1]. */
int paradis_geocyclic_avgpool5_fwd(const float* x, float* y, int B, int C, int H, int W, int stride, void* stream);

/* ---- Latitude-band halo outbox (no counterpart in the reference, whose only parallelism is DDP, train.py:49) ----
 * Copies the first and the last `h` rows of `n` (1..4) band tensors [B, V, rows, W] (batch stride src_sB[k] elements,
 * inner three dims contiguous) into box[n][2][B*V][h][W] -- side 0 = first rows, side 1 = last rows -- in ONE launch.
 * `box` is the symmetric-memory buffer the latitude neighbours read their halo rows from over NVLink
 * (paradis_sl_geom.fld_peer_* / arr_peer_*).  src and src_sB are HOST arrays, read before the call returns. */
int paradis_halo_pack(const float* const* src, const int64_t* src_sB, int n, int B, int V, int rows, int W, int h,
                      float* box, void* stream);

/* ---- Semi-Lagrangian advection core: model/advection.py:129-169 --------------------
 * (pole mean -> rotated-pole backtrack -> pixel coords -> GeoCyclic pad -> grid_sample
 *  -> pole mean), fused.
 *   field [B, V, fld_rows, W], u, v [B, V, arr_rows, W], out [B, V, own_rows, W].
 * *_sB = batch stride in elements (u and v may be views of one [B, 2V, H, W] tensor,
 * model/paradis.py:235-237); the inner three dims are contiguous.  out is contiguous.
 * `status` (optional) points to one device int32 that kernels set to a paradis_status
 * on a device-side contract violation.
 * Alignment: any float pointer is accepted.  The vectorised kernels (4 points per thread, and the
 * fused backward sweep) are used when W % 4 == 0, every tensor pointer and the geometry tables are
 * 16-byte aligned and the batch strides are multiples of 4 elements -- true for PyTorch allocations;
 * otherwise the scalar forward (bit-identical output) and the general two-kernel backward (same sums in a
 * different, equally deterministic order) run. */
size_t paradis_sl_advect_fwd_workspace(int B, int V);
int paradis_sl_advect_fwd(const paradis_sl_geom* geom, const float* field, const float* u,
                          const float* v, float* out, int B, int V, int64_t field_sB,
                          int64_t u_sB, int64_t v_sB, float dt, int interp, int pole_fix,
                          int math, void* workspace, size_t workspace_bytes, int32_t* status,
                          void* stream);

/* Backward of the above: recomputes the trajectory from (u, v); nothing is saved by
 * forward.  grad_field is produced by a deterministic gather over inverse stencils
 * (no atomics).
 *   grad_out, u, v [B, V, arr_rows, W]; field [B, V, fld_rows, W];
 *   grad_field, grad_u, grad_v [B, V, own_rows, W] contiguous.
 * grad_field may be NULL (skips the adjoint gather); grad_u and grad_v may both be NULL.
 * `phases` selects the kernels to enqueue: PARADIS_BWD_ARRIVAL (grad_u, grad_v and the row
 * classes of every arrival point, kept in the workspace), PARADIS_BWD_GATHER (grad_field
 * from the classes left in the SAME workspace by an earlier ARRIVAL call), or both.
 *
 * `cfl_cells` > 0 (with phases == PARADIS_BWD_ALL) enables the fused single-pass backward for
 * the mid-latitudes: it is the caller's bound on the great-circle displacement |(u, v)| * dt in
 * units of the latitude spacing (the semi-Lagrangian CFL number).  The bound is checked on the
 * device for every arrival point; planes that exceed it are transparently recomputed by the
 * general two-kernel path, so results never depend on it -- only speed does.  <= 0 disables it. */
#define PARADIS_BWD_ARRIVAL 1
#define PARADIS_BWD_GATHER 2
#define PARADIS_BWD_ALL 3
/* OR-ed into PARADIS_BWD_ALL: use the warp-specialised row sweep (sl_rows.cuh) whenever its plan fits, also on meshes
 * narrower than ~900 columns and for the 4x4 stencil, where the round-1 strip sweep is the default (tests). */
#define PARADIS_BWD_ROWSWEEP 8
size_t paradis_sl_advect_bwd_workspace(int B, int V, int arr_rows, int W);
int paradis_sl_advect_bwd(const paradis_sl_geom* geom, const float* grad_out,
                          const float* field, const float* u, const float* v, float* grad_field,
                          float* grad_u, float* grad_v, int B, int V, int64_t gout_sB,
                          int64_t field_sB, int64_t u_sB, int64_t v_sB, float dt, int interp,
                          int pole_fix, int math, int phases, float cfl_cells, void* workspace,
                          size_t workspace_bytes, int32_t* status, void* stream);

/* Departure coordinates only (parity instrument): for every arrival point of the own window writes
 * the 11 intermediates of model/advection.py:82-94,138-150 as planes
 *   coords[B, V, 11, own_rows, W] = { ix, iy, sin(lat'), cos(lat'), sin(lon'), cos(lon'), sin_lat, num, den,
 *                                    lat_dep, lon_dep }
 * with ix, iy the sampler coordinates in the padded plane (what ATen floors, GridSampler.h:27-36). */
int paradis_sl_departure_coords(const paradis_sl_geom* geom, const float* u, const float* v,
                                float* coords, int B, int V, int64_t u_sB, int64_t v_sB, float dt,
                                int interp, int math, void* stream);

/* ---- Host-buffer entry (end-to-end path) --------------------------------------------
 * Same operator (single GPU, full mesh) with HOST pointers (pinned memory recommended):
 * the library stages `chunk_planes` (b, v) planes at a time through caller-provided
 * device scratch on its own streams (H2D / compute / D2H overlapped) and returns when
 * all results are on the host.  Tables inside `geom` are still device pointers. */
size_t paradis_sl_host_scratch_bytes(int H, int W, int chunk_planes);
int paradis_sl_advect_fwd_bwd_host(const paradis_sl_geom* geom, const float* h_field,
                                   const float* h_u, const float* h_v, const float* h_grad_out,
                                   float* h_out, float* h_grad_field, float* h_grad_u,
                                   float* h_grad_v, int64_t planes, float dt, int interp,
                                   int pole_fix, int math, float cfl_cells, int chunk_planes,
                                   void* d_scratch, size_t scratch_bytes);

#ifdef __cplusplus
}
#endif
#endif /* PARADIS_SL_H_ */
