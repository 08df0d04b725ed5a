/*
 * paradis_geocyclic.h -- bf16 storage for the GeoCyclic padding, depthwise-convolution and downsampling ops of
 * libparadis_sl.so (sm_100a), and the strided adjoint of the 5x5 average pooling.
 *
 * Under bf16 autocast (the reference's "bf16-mixed" training, train.py:56) the activations that reach
 * GeoCyclicPadding, SepConv's depthwise convolution and PhysicalDownsample are bf16.  The *_bf16 entry points read
 * and write those tensors as bf16 and compute in fp32 in registers, so no fp32 copy of them is made.
 *
 * Bit-identity: every bf16 result is bit-identical to the fp32 entry point (paradis_sl.h, or
 * paradis_geocyclic_avgpool5_bwd below) run on fp32 copies of the inputs (bf16 -> fp32 is exact), with the result
 * then rounded to bf16 once (round to nearest even, as torch's `.to(torch.bfloat16)`).  Sums run in the same fixed
 * order as the fp32 kernels.  In particular the bf16 grad input of the depthwise convolution adds the polar-cap fold
 * to the direct part in fp32 before its single rounding.  NaN inputs give NaN outputs; the NaN payload is not
 * specified.
 *
 * Arguments and status codes are those of the fp32 entry points in paradis_sl.h (caller-owned buffers,
 * asynchronous on `stream`), plus:
 *   - bf16 tensors are passed as `void*` holding IEEE bfloat16 (torch.bfloat16) values, contiguous [B, C, H, W];
 *     weight, bias, grad weight and grad bias stay fp32 ([C, k, k] and [C]).
 *   - NULL tensor: PARADIS_ERR_NULL_POINTER.  Odd W: PARADIS_ERR_ODD_WIDTH.  k not in {3, 5, 7}:
 *     PARADIS_ERR_BAD_INTERP.  Mesh too small (dwconv / avgpool5: H < k + 1 or W < k - 1; pad: H < p + 1 or
 *     W < 2p), B * C > 65535, stride < 1: PARADIS_ERR_BAD_SHAPE.  Short weight-gradient workspace:
 *     PARADIS_ERR_WORKSPACE.
 *   - The output y of paradis_geocyclic_pad_fwd_bf16 must be 4-byte aligned, as every PyTorch allocation is (two
 *     values are stored per 4-byte word); otherwise PARADIS_ERR_BAD_SHAPE.
 */
#ifndef PARADIS_GEOCYCLIC_H_
#define PARADIS_GEOCYCLIC_H_

#include "paradis_sl.h"

#ifdef __cplusplus
extern "C" {
#endif

/* GeoCyclic padding (as paradis_geocyclic_pad_fwd / _bwd): x [planes, H, W] -> y [planes, H + 2p, W + 2p] and the
 * adjoint gy -> gx.  The forward copies the bf16 values unchanged. */
int paradis_geocyclic_pad_fwd_bf16(const void* x, void* y, int64_t planes, int H, int W, int p, void* stream);
int paradis_geocyclic_pad_bwd_bf16(const void* gy, void* gx, int64_t planes, int H, int W, int p, void* stream);

/* Depthwise k x k convolution with the GeoCyclic padding applied on the fly (as paradis_geocyclic_dwconv_*).
 * bwd_weight takes paradis_geocyclic_dwconv_wgrad_workspace(B, C, H, W, k) bytes of scratch; gbias may be NULL. */
int paradis_geocyclic_dwconv_fwd_bf16(const void* x, const float* weight, const float* bias, void* y, int B, int C,
                                      int H, int W, int k, void* stream);
int paradis_geocyclic_dwconv_bwd_input_bf16(const void* gy, const float* weight, void* gx, int B, int C, int H, int W,
                                            int k, void* stream);
int paradis_geocyclic_dwconv_bwd_weight_bf16(const void* x, const void* gy, float* gweight, float* gbias, int B,
                                             int C, int H, int W, int k, void* workspace, size_t workspace_bytes,
                                             void* stream);

/* GeoCyclic pad 2 + AvgPool2d(5, stride): x [B, C, H, W] -> y [B, C, (H - 1) / stride + 1, (W - 1) / stride + 1]
 * (as paradis_geocyclic_avgpool5_fwd), and its adjoint gy -> gx [B, C, H, W] (H, W are the input's).  The adjoint
 * gathers, for every input point, only the strided outputs whose 5x5 window covers it; the fp32 variant is
 * bit-identical to paradis_geocyclic_dwconv_bwd_input with the 1/25 box filter applied to gy scattered into a
 * zero-filled [B, C, H, W] grid at every stride-th point. */
int paradis_geocyclic_avgpool5_fwd_bf16(const void* x, void* y, int B, int C, int H, int W, int stride, void* stream);
int paradis_geocyclic_avgpool5_bwd(const float* gy, float* gx, int B, int C, int H, int W, int stride, void* stream);
int paradis_geocyclic_avgpool5_bwd_bf16(const void* gy, void* gx, int B, int C, int H, int W, int stride,
                                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PARADIS_GEOCYCLIC_H_ */
