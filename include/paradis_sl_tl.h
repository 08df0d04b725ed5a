/*
 * paradis_sl_tl.h -- tangent-linear model of the semi-Lagrangian advection core of libparadis_sl.so (sm_100a).
 *
 * The forward paradis_sl_advect_fwd computes out(field, u, v).  This entry point computes its directional derivative
 *
 *   dout = (d out / d field) dfield + (d out / d u) du + (d out / d v) dv
 *
 * at the same departure points (the forward's own fp32 trajectory, in both math modes), with the same pole
 * treatment: with pole_fix, dfield's pole rows are replaced by their zonal means and so are dout's rows 0 / H-1.
 * One gather per arrival point, no atomics: the result is deterministic.  With du = dv = 0 it equals the forward
 * applied to dfield bit for bit.  It is the transpose of paradis_sl_advect_bwd: <J t, g> = <t, J^T g>.
 *
 * Conventions are those of paradis_sl.h (shared geometry struct, status codes, caller-owned buffers, asynchronous
 * on `stream`), plus:
 *   - fp32 storage only; dout [B, V, H, W] contiguous, the six inputs with batch strides *_sB (elements).
 *   - dfield may be NULL (velocity tangents only); du and dv are both NULL (field tangent only) or both set,
 *     otherwise PARADIS_ERR_NULL_POINTER.
 *   - Full mesh only: own, arr and fld windows all (0, H) and no peer halo pointers; otherwise
 *     PARADIS_ERR_BAD_SHAPE.
 *   - Any displacement is accepted, as by the forward.
 *   - NULL field / u / v / dout, a bad interpolation or a small workspace return the codes of the forward.
 */
#ifndef PARADIS_SL_TL_H_
#define PARADIS_SL_TL_H_

#include "paradis_sl.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Workspace bytes (needed when pole_fix): zonal pole means of field and dfield. */
size_t paradis_sl_advect_jvp_workspace(int B, int V);

int paradis_sl_advect_jvp(const paradis_sl_geom* geom, const float* field, const float* dfield /* nullable */,
                          const float* u, const float* v, const float* du, const float* dv /* both or neither */,
                          float* dout, int B, int V, int64_t field_sB, int64_t dfield_sB, int64_t u_sB,
                          int64_t v_sB, int64_t du_sB, int64_t dv_sB, float dt, int interp, int pole_fix, int math,
                          void* workspace, size_t workspace_bytes, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PARADIS_SL_TL_H_ */
