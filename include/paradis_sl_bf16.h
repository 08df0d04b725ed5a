/*
 * paradis_sl_bf16.h -- bf16 storage for the semi-Lagrangian advection core of libparadis_sl.so (sm_100a).
 *
 * Under bf16 autocast (the reference's default "bf16-mixed" training, train.py:56) `field` comes out of
 * down_projection and u, v out of velocity_net in bf16 (model/paradis.py:235-237).  These entry points read
 * field, u, v as bf16 and write grad_field, grad_u, grad_v as bf16, computing in fp32 in registers, so no fp32
 * copy of any of them is made.  Results are bit-identical to the fp32 entry points of paradis_sl.h run on fp32
 * copies of the inputs (bf16 -> fp32 is exact), with the gradients then rounded to bf16 (round to nearest even,
 * as torch's `.to(torch.bfloat16)`), in both math modes and on every backward path.
 *
 * Conventions are those of paradis_sl.h (shared geometry struct, status codes, caller-owned buffers,
 * asynchronous on `stream`), plus:
 *   - bf16 tensors are passed as `void*` holding IEEE bfloat16 (torch.bfloat16) values; `out` and `grad_out` are
 *     fp32 (the op's output is fp32, as the reference's grid_sample under autocast).
 *   - Full mesh only: own, arr and fld windows all (0, H) and no peer halo pointers; otherwise
 *     PARADIS_ERR_BAD_SHAPE.  Latitude bands, the host-buffer entry and paradis_sl_departure_coords stay fp32.
 *   - W % 8 == 0, every tensor pointer and the lon table 16-byte aligned, batch strides (in elements) multiples
 *     of 8 for the bf16 tensors and of 4 for grad_out -- true for PyTorch allocations and for u, v as views of one
 *     [B, 2V, H, W] tensor; otherwise PARADIS_ERR_BAD_SHAPE (use the fp32 entry points on fp32 copies).
 *   - NULL pointers, a bad interpolation or a small workspace return the codes of the fp32 entry points.
 */
#ifndef PARADIS_SL_BF16_H_
#define PARADIS_SL_BF16_H_

#include "paradis_sl.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Forward: field [B, V, H, W] bf16, u, v [B, V, H, W] bf16 (batch strides *_sB), out [B, V, H, W] fp32
 * contiguous.  Workspace: paradis_sl_advect_fwd_workspace(B, V) bytes (needed when pole_fix). */
int paradis_sl_advect_fwd_bf16(const paradis_sl_geom* geom, const void* field, const void* u, const void* v,
                               float* out, int B, int V, int64_t field_sB, int64_t u_sB, int64_t v_sB, float dt,
                               int interp, int pole_fix, int math, void* workspace, size_t workspace_bytes,
                               int32_t* status, void* stream);

/* Backward: grad_out fp32, field, u, v bf16; grad_field, grad_u, grad_v bf16 [B, V, H, W] contiguous (grad_field
 * may be NULL, grad_u and grad_v both NULL).  Arguments as paradis_sl_advect_bwd.  The workspace holds the fp32
 * one plus an fp32 grad_field accumulation buffer, which is rounded to bf16 once, after the last pass. */
size_t paradis_sl_advect_bwd_bf16_workspace(int B, int V, int arr_rows, int W);
int paradis_sl_advect_bwd_bf16(const paradis_sl_geom* geom, const float* grad_out, const void* field,
                               const void* u, const void* v, void* grad_field, void* grad_u, void* grad_v, int B,
                               int V, int64_t gout_sB, int64_t field_sB, int64_t u_sB, int64_t v_sB, float dt,
                               int interp, int pole_fix, int math, int phases, float cfl_cells, void* workspace,
                               size_t workspace_bytes, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PARADIS_SL_BF16_H_ */
