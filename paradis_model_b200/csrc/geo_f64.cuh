// float64 GeoCyclic ops (include/paradis_sl_f64.h): padding and its adjoint, the padded depthwise convolution with
// its two gradients, and the padded 5x5 average pooling with its adjoint.  Double storage, double weights / bias and
// double sums; the fp32 / bf16 kernels above keep their machine code.  Every sum has a fixed order (no atomics).
//
// The adjoints are gathers over the padded cells whose GeoCyclic source is the input point (pad_cells): the interior
// cell, the wrapped columns and, next to a pole, the reflected cap cells -- the order of geocyclic_pad_bwd_kernel.
#include "../../include/paradis_sl_f64.h"

namespace {

// source of padded cell (i, j) (unpadded coordinates) of a pad-P plane; 0 outside it (model/padding.py:26-37)
__device__ __forceinline__ double geo_load64(const double* __restrict__ x, int i, int j, int H, int W, int P) {
  if (i < -P || i >= H + P || j < -P || j >= W + P) return 0.0;
  int shift = 0;
  if (i < 0) { i = -i; shift = W / 2; }
  else if (i >= H) { i = 2 * (H - 1) - i; shift = W / 2; }
  j -= shift;
  if (j < 0) j += W; else if (j >= W) j -= W;
  return __ldg(x + (long long)i * W + j);
}

// f(R, C) for every padded cell (R, C) of a pad-P plane whose source is (i, j), in a fixed order: interior row, north
// cap, south cap; within a row: centre, left wrap, right wrap.  Needs W >= 2P.
template <typename F>
__device__ __forceinline__ void pad_cells(int i, int j, int H, int W, int P, F&& f) {
  for (int src = 0; src < 3; ++src) {
    int R, shift;
    if (src == 0) { R = i + P; shift = 0; }
    else if (src == 1) { if (i < 1 || i > P) continue; R = P - i; shift = W / 2; }
    else { const int ii = 2 * (H - 1) - i; if (ii < H || ii >= H + P) continue; R = ii + P; shift = W / 2; }
    int c = j + shift; if (c >= W) c -= W;    // C - P in [0, W)
    f(R, c + P);
    if (c >= W - P) f(R, c - W + P);          // left wrap columns  C - P in [-P, 0)
    if (c < P) f(R, c + W + P);               // right wrap columns C - P in [W, W + P)
  }
}

__global__ void geocyclic_pad_fwd_f64_kernel(const double* __restrict__ x, double* __restrict__ y, int H, int W, int p) {
  const int Hp = H + 2 * p, Wp = W + 2 * p;
  const long long pl = blockIdx.z;
  const int R = blockIdx.y;
  for (int C = blockIdx.x * blockDim.x + threadIdx.x; C < Wp; C += gridDim.x * blockDim.x)
    y[(pl * Hp + R) * Wp + C] = geo_load64(x + pl * H * W, R - p, C - p, H, W, p);
}

__global__ void geocyclic_pad_bwd_f64_kernel(const double* __restrict__ gy, double* __restrict__ gx, int H, int W, int p) {
  const int Wp = W + 2 * p;
  const long long pl = blockIdx.z;
  const int i = blockIdx.y;
  const double* g = gy + pl * (long long)(H + 2 * p) * Wp;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < W; j += gridDim.x * blockDim.x) {
    double s = 0.0;
    pad_cells(i, j, H, W, p, [&](int R, int C) { s += g[(long long)R * Wp + C]; });
    gx[(pl * H + i) * W + j] = s;
  }
}

// y[i, j] = bias + sum_{a, b} w[a, b] xpad[i + a, j + b]
template <int K>
__global__ void __launch_bounds__(256) geo_dwconv_fwd_f64_kernel(const double* __restrict__ x, const double* __restrict__ w,
                                                                 const double* __restrict__ bias, double* __restrict__ y,
                                                                 int C, int H, int W) {
  constexpr int P = (K - 1) / 2;
  const int plane = blockIdx.z, c = plane % C, i = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= W) return;
  const double* s = x + (long long)plane * H * W;
  const double* wc = w + c * K * K;
  double acc = bias ? __ldg(bias + c) : 0.0;
#pragma unroll
  for (int a = 0; a < K; ++a)
#pragma unroll
    for (int b = 0; b < K; ++b) acc = fma(__ldg(wc + a * K + b), geo_load64(s, i + a - P, j + b - P, H, W, P), acc);
  y[((long long)plane * H + i) * W + j] = acc;
}

// gx[i, j] = sum over the padded cells (R, C) of (i, j) of sum_{a, b} w[a, b] gy[R - a, C - b] (outputs in the mesh)
template <int K>
__global__ void __launch_bounds__(256) geo_dwconv_bwd_input_f64_kernel(const double* __restrict__ gy,
                                                                       const double* __restrict__ w,
                                                                       double* __restrict__ gx, int C, int H, int W) {
  constexpr int P = (K - 1) / 2;
  const int plane = blockIdx.z, c = plane % C, i = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= W) return;
  const double* g = gy + (long long)plane * H * W;
  const double* wc = w + c * K * K;
  double acc = 0.0;
  pad_cells(i, j, H, W, P, [&](int R, int Cc) {
    for (int a = 0; a < K; ++a) {
      const int oi = R - a;
      if (oi < 0 || oi >= H) continue;
      for (int b = 0; b < K; ++b) {
        const int oj = Cc - b;
        if (oj >= 0 && oj < W) acc = fma(__ldg(wc + a * K + b), __ldg(g + (long long)oi * W + oj), acc);
      }
    }
  });
  gx[((long long)plane * H + i) * W + j] = acc;
}

// grad weight / grad bias: per (plane, band of kWgradRows rows) partial sums [plane][band][K*K+1]; lanes reduced by
// an xor tree, then the warps in order
constexpr int kWgradRows = 16;
template <int K>
__global__ void __launch_bounds__(256) geo_dwconv_wgrad_f64_kernel(const double* __restrict__ x,
                                                                   const double* __restrict__ gy,
                                                                   double* __restrict__ partial, int H, int W) {
  constexpr int P = (K - 1) / 2, NV = K * K + 1;
  __shared__ double red[8][NV];
  const int plane = blockIdx.y, band = blockIdx.x;
  const double* s = x + (long long)plane * H * W;
  const double* g = gy + (long long)plane * H * W;
  double acc[NV];
#pragma unroll
  for (int t = 0; t < NV; ++t) acc[t] = 0.0;
  const int i0 = band * kWgradRows, i1 = min(i0 + kWgradRows, H);
  for (int q = threadIdx.x; q < (i1 - i0) * W; q += 256) {
    const int i = i0 + q / W, j = q - (q / W) * W;
    const double gv = __ldg(g + (long long)i * W + j);
#pragma unroll
    for (int a = 0; a < K; ++a)
#pragma unroll
      for (int b = 0; b < K; ++b) acc[a * K + b] = fma(gv, geo_load64(s, i + a - P, j + b - P, H, W, P), acc[a * K + b]);
    acc[K * K] += gv;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    double v = acc[t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][t] = v;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double v = 0.0;
    for (int wq = 0; wq < 8; ++wq) v += red[wq][threadIdx.x];
    partial[((long long)plane * gridDim.x + band) * NV + threadIdx.x] = v;
  }
}

// gw[c][t] = sum over batch n and bands (ascending) of partial[n*C+c][band][t]
__global__ void geo_dwconv_wgrad_reduce_f64_kernel(const double* __restrict__ partial, double* __restrict__ gw,
                                                   double* __restrict__ gbias, int B, int C, int nbands, int NV) {
  const int c = blockIdx.x, t = threadIdx.x;
  if (t >= NV) return;
  double s = 0.0;
  for (int n = 0; n < B; ++n) {
    const double* p = partial + ((long long)(n * C + c) * nbands) * NV + t;
    for (int k = 0; k < nbands; ++k) s += p[(long long)k * NV];
  }
  if (t < NV - 1) gw[c * (NV - 1) + t] = s;
  else if (gbias) gbias[c] = s;
}

template <int K>
int dwconv_f64(int what, const double* a, const double* gy, const double* w, const double* bias, double* out,
               double* gw, double* gb, double* ws, int B, int C, int H, int W, cudaStream_t st) {
  const dim3 grid((W + 255) / 256, H, B * C);
  if (what == 0) geo_dwconv_fwd_f64_kernel<K><<<grid, 256, 0, st>>>(a, w, bias, out, C, H, W);
  else if (what == 1) geo_dwconv_bwd_input_f64_kernel<K><<<grid, 256, 0, st>>>(a, w, out, C, H, W);
  else {
    const int nbands = (H + kWgradRows - 1) / kWgradRows;
    geo_dwconv_wgrad_f64_kernel<K><<<dim3(nbands, B * C), 256, 0, st>>>(a, gy, ws, H, W);
    geo_dwconv_wgrad_reduce_f64_kernel<<<C, 64, 0, st>>>(ws, gw, gb, B, C, nbands, K * K + 1);
  }
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : err(PARADIS_ERR_CUDA, cudaGetErrorString(e));
}

int dispatch_f64(int what, const double* a, const double* gy, const double* w, const double* bias, double* out,
                 double* gw, double* gb, double* ws, int B, int C, int H, int W, int k, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (k == 3) return dwconv_f64<3>(what, a, gy, w, bias, out, gw, gb, ws, B, C, H, W, st);
  if (k == 5) return dwconv_f64<5>(what, a, gy, w, bias, out, gw, gb, ws, B, C, H, W, st);
  return dwconv_f64<7>(what, a, gy, w, bias, out, gw, gb, ws, B, C, H, W, st);
}

// AvgPool2d(5, stride) of the pad-2 plane: y[io, jo] = (sum of the 5 x 5 window at (io * stride, jo * stride)) / 25
__global__ void geo_avgpool5_fwd_f64_kernel(const double* __restrict__ x, double* __restrict__ y, int H, int W, int Ho,
                                            int Wo, int stride) {
  const long long pl = blockIdx.z;
  const int io = blockIdx.y, jo = blockIdx.x * blockDim.x + threadIdx.x;
  if (jo >= Wo) return;
  const double* xp = x + pl * (long long)H * W;
  double s = 0.0;
#pragma unroll
  for (int a = 0; a < 5; ++a)
#pragma unroll
    for (int b = 0; b < 5; ++b) s += geo_load64(xp, io * stride + a - 2, jo * stride + b - 2, H, W, 2);
  y[(pl * Ho + io) * Wo + jo] = s / 25.0;
}

// adjoint: gx[i, j] = sum over the padded cells (R, C) of (i, j) and the outputs whose window covers them of gy / 25
__global__ void geo_avgpool5_bwd_f64_kernel(const double* __restrict__ gy, double* __restrict__ gx, int H, int W, int Ho,
                                            int Wo, int stride) {
  const long long pl = blockIdx.z;
  const int i = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= W) return;
  const double* g = gy + pl * (long long)Ho * Wo;
  double acc = 0.0;
  pad_cells(i, j, H, W, 2, [&](int R, int Cc) {
    for (int a = 0; a < 5; ++a) {
      const int r = R - a;                         // window origin row io * stride
      if (r < 0 || r % stride || r / stride >= Ho) continue;
      for (int b = 0; b < 5; ++b) {
        const int q = Cc - b;
        if (q >= 0 && q % stride == 0 && q / stride < Wo) acc += __ldg(g + (long long)(r / stride) * Wo + q / stride);
      }
    }
  });
  gx[(pl * H + i) * W + j] = acc / 25.0;
}

int avgpool5_f64(bool backward, const double* src, double* dst, int B, int C, int H, int W, int stride, void* stream) {
  if (int rc = check(src, dst, B, C, H, W, 5)) return rc;
  if (stride < 1) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_avgpool5: stride must be >= 1");
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  if (backward)
    geo_avgpool5_bwd_f64_kernel<<<dim3((W + 127) / 128, H, B * C), 128, 0, (cudaStream_t)stream>>>(src, dst, H, W, Ho,
                                                                                                   Wo, stride);
  else
    geo_avgpool5_fwd_f64_kernel<<<dim3((Wo + 127) / 128, Ho, B * C), 128, 0, (cudaStream_t)stream>>>(src, dst, H, W, Ho,
                                                                                                    Wo, stride);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : err(PARADIS_ERR_CUDA, cudaGetErrorString(e));
}

int pad_check64(const void* a, const void* b, int64_t planes, int H, int W, int p) {
  if (!a || !b) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_pad: NULL tensor pointer");
  if (planes <= 0 || H <= 0 || W <= 0 || p < 0) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_pad: non-positive dimension");
  if (W % 2) return err(PARADIS_ERR_ODD_WIDTH, "Number of longitude points must be even");
  if (H < p + 1 || W < 2 * p) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_pad: pad width too large for the mesh");
  if (planes > 65535 || H + 2 * p > 65535) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_pad: too many planes/rows for one launch");
  return PARADIS_OK;
}

}  // namespace

extern "C" int paradis_geocyclic_pad_fwd_f64(const double* x, double* y, int64_t planes, int H, int W, int p, void* stream) {
  if (int rc = pad_check64(x, y, planes, H, W, p)) return rc;
  const dim3 grid((W + 2 * p + 255) / 256, H + 2 * p, (unsigned)planes);
  geocyclic_pad_fwd_f64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, H, W, p);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : err(PARADIS_ERR_CUDA, cudaGetErrorString(e));
}

extern "C" int paradis_geocyclic_pad_bwd_f64(const double* gy, double* gx, int64_t planes, int H, int W, int p, void* stream) {
  if (int rc = pad_check64(gy, gx, planes, H, W, p)) return rc;
  const dim3 grid((W + 255) / 256, H, (unsigned)planes);
  geocyclic_pad_bwd_f64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(gy, gx, H, W, p);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : err(PARADIS_ERR_CUDA, cudaGetErrorString(e));
}

extern "C" int paradis_geocyclic_dwconv_fwd_f64(const double* x, const double* weight, const double* bias, double* y,
                                                int B, int C, int H, int W, int k, void* stream) {
  if (int rc = check(x, y, B, C, H, W, k)) return rc;
  if (!weight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: weight is NULL");
  return dispatch_f64(0, x, nullptr, weight, bias, y, nullptr, nullptr, nullptr, B, C, H, W, k, stream);
}

extern "C" int paradis_geocyclic_dwconv_bwd_input_f64(const double* gy, const double* weight, double* gx, int B, int C,
                                                      int H, int W, int k, void* stream) {
  if (int rc = check(gy, gx, B, C, H, W, k)) return rc;
  if (!weight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: weight is NULL");
  return dispatch_f64(1, gy, nullptr, weight, nullptr, gx, nullptr, nullptr, nullptr, B, C, H, W, k, stream);
}

extern "C" size_t paradis_geocyclic_dwconv_wgrad_f64_workspace(int B, int C, int H, int W, int k) {
  (void)W;
  return (size_t)B * C * ((H + kWgradRows - 1) / kWgradRows) * (k * k + 1) * sizeof(double);
}

extern "C" int paradis_geocyclic_dwconv_bwd_weight_f64(const double* x, const double* gy, double* gweight, double* gbias,
                                                       int B, int C, int H, int W, int k, void* workspace,
                                                       size_t workspace_bytes, void* stream) {
  if (int rc = check(x, gy, B, C, H, W, k)) return rc;
  if (!gweight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: grad weight is NULL");
  if (!workspace || workspace_bytes < paradis_geocyclic_dwconv_wgrad_f64_workspace(B, C, H, W, k))
    return err(PARADIS_ERR_WORKSPACE, "geocyclic_dwconv: weight-gradient workspace too small");
  return dispatch_f64(2, x, gy, nullptr, nullptr, nullptr, gweight, gbias, (double*)workspace, B, C, H, W, k, stream);
}

extern "C" int paradis_geocyclic_avgpool5_fwd_f64(const double* x, double* y, int B, int C, int H, int W, int stride,
                                                  void* stream) {
  return avgpool5_f64(false, x, y, B, C, H, W, stride, stream);
}

extern "C" int paradis_geocyclic_avgpool5_bwd_f64(const double* gy, double* gx, int B, int C, int H, int W, int stride,
                                                  void* stream) {
  return avgpool5_f64(true, gy, gx, B, C, H, W, stride, stream);
}
