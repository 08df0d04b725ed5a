/*
 * paradis_sl_f64.h -- float64 entry points of libparadis_sl.so (sm_100a): the advection, its adjoint, its
 * tangent-linear model, the departure-point instrument and the GeoCyclic padding / depthwise-convolution /
 * downsampling ops with double storage and double arithmetic.
 *
 * Arithmetic.  fp64 has one arithmetic: the reference's op order (model/advection.py:131-150, then ATen's
 * un-normalisation of the sampler coordinates) in IEEE double, one rounding per torch op, with libdevice's double
 * sin / cos / asin / atan2.  As in ATen-CUDA: a division by a Python scalar multiplies by the double reciprocal, the
 * clamp bounds are the doubles -1+1e-7 and 1-1e-7, 2 pi is a double and remainder() is the exact (Sterbenz)
 * subtraction.  `math` is accepted and checked like everywhere else but does not change the result (FAST is an fp32
 * speed device).  Stencil taps, bicubic A = -0.75, the GeoCyclic map, the pole means and the 126-row displacement
 * contract of the adjoint (status word PARADIS_ERR_DISPLACEMENT) are those of the fp32 kernels.
 *
 * Conventions are those of paradis_sl.h (status codes, ABI version, caller-owned buffers, asynchronous on `stream`,
 * contiguous [B, V, H, W] outputs, batch strides *_sB in elements), plus:
 *   - the geometry is paradis_sl_geom_f64: full mesh only, no latitude bands and no peer halos;
 *   - every tensor, every table, `dt`, the weights and the bias are double;
 *   - the adjoint is deterministic (fixed summation order, no atomics).
 */
#ifndef PARADIS_SL_F64_H_
#define PARADIS_SL_F64_H_

#include "paradis_sl.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct paradis_sl_geom_f64 {
  int32_t H, W;            /* mesh; W even, H >= interp + 2 */
  const double* sin_lat;   /* [H] sin of the arrival latitudes (torch fp64 on the device) */
  const double* cos_lat;   /* [H] */
  const double* lon;       /* [W] arrival longitudes */
  double min_lat, d_lat, min_lon, d_lon;   /* the module's buffers, as they are */
} paradis_sl_geom_f64;

/* advection: out [B, V, H, W] */
size_t paradis_sl_advect_fwd_f64_workspace(int B, int V);
int paradis_sl_advect_fwd_f64(const paradis_sl_geom_f64* geom, const double* field, const double* u, const double* v,
                              double* out, int B, int V, int64_t field_sB, int64_t u_sB, int64_t v_sB, double dt,
                              int interp, int pole_fix, int math, void* workspace, size_t workspace_bytes,
                              int32_t* status, void* stream);

/* adjoint: grad_field may be NULL; grad_u and grad_v both or neither.  Per-point gradients of u and v, then one gather
 * per output row of grad_field over the arrival points whose stencil covers it (W <= 3400). */
size_t paradis_sl_advect_bwd_f64_workspace(int B, int V, int H, int W);
int paradis_sl_advect_bwd_f64(const paradis_sl_geom_f64* geom, const double* grad_out, const double* field,
                              const double* u, const double* v, double* grad_field, double* grad_u, double* grad_v,
                              int B, int V, int64_t gout_sB, int64_t field_sB, int64_t u_sB, int64_t v_sB, double dt,
                              int interp, int pole_fix, int math, void* workspace, size_t workspace_bytes,
                              int32_t* status, void* stream);

/* tangent-linear model: dfield may be NULL, du and dv both or neither (see paradis_sl_tl.h) */
size_t paradis_sl_advect_jvp_f64_workspace(int B, int V);
int paradis_sl_advect_jvp_f64(const paradis_sl_geom_f64* geom, const double* field, const double* dfield,
                              const double* u, const double* v, const double* du, const double* dv, double* dout,
                              int B, int V, int64_t field_sB, int64_t dfield_sB, int64_t u_sB, int64_t v_sB,
                              int64_t du_sB, int64_t dv_sB, double dt, int interp, int pole_fix, int math,
                              void* workspace, size_t workspace_bytes, int32_t* status, void* stream);

/* parity instrument: coords [B, V, 11, H, W] = (ix, iy, sin lat', cos lat', sin lon', cos lon', s, num, den, lat, lon) */
int paradis_sl_departure_coords_f64(const paradis_sl_geom_f64* geom, const double* u, const double* v, double* coords,
                                    int B, int V, int64_t u_sB, int64_t v_sB, double dt, int interp, int math,
                                    void* stream);

/* GeoCyclic ops: same shapes and checks as their fp32 entry points in paradis_sl.h / paradis_geocyclic.h */
int paradis_geocyclic_pad_fwd_f64(const double* x, double* y, int64_t planes, int H, int W, int p, void* stream);
int paradis_geocyclic_pad_bwd_f64(const double* gy, double* gx, int64_t planes, int H, int W, int p, void* stream);
int paradis_geocyclic_dwconv_fwd_f64(const double* x, const double* weight, const double* bias /* nullable */,
                                     double* y, int B, int C, int H, int W, int k, void* stream);
int paradis_geocyclic_dwconv_bwd_input_f64(const double* gy, const double* weight, double* gx, int B, int C, int H,
                                           int W, int k, void* stream);
size_t paradis_geocyclic_dwconv_wgrad_f64_workspace(int B, int C, int H, int W, int k);
int paradis_geocyclic_dwconv_bwd_weight_f64(const double* x, const double* gy, double* gweight,
                                            double* gbias /* nullable */, int B, int C, int H, int W, int k,
                                            void* workspace, size_t workspace_bytes, void* stream);
int paradis_geocyclic_avgpool5_fwd_f64(const double* x, double* y, int B, int C, int H, int W, int stride,
                                       void* stream);
int paradis_geocyclic_avgpool5_bwd_f64(const double* gy, double* gx, int B, int C, int H, int W, int stride,
                                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PARADIS_SL_F64_H_ */
