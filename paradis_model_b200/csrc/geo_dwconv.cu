// Depthwise k x k convolution with the GeoCyclic padding applied on the fly (sm_100a).
//
// Replaces, in one kernel, `GeoCyclicPadding((k-1)/2)` followed by the depthwise `nn.Conv2d(C, C, k,
// groups=C)` of the reference's SepConv (model/blocks.py:92-116) and of the static encoder
// (model/paradis.py:186-190): the padded tensor [B, C, H+k-1, W+k-1] is never written or read.
// SURVEY section 8(f) rank 3.  Algorithmic traffic: read x (4 B) + write y (4 B) per element instead of
// 16 B for pad-then-convolve.
//
//   forward      y[i,j]  = bias + sum_{a,b} w[a,b] * xpad[i+a, j+b]
//   grad input   gx      = P^T ( full correlation of gy with w ): longitude is periodic, so the direct part
//                          is the same tiled kernel with the flipped filter, zero rows outside the mesh and
//                          circular columns; the two polar caps fold a few rows back (fixed order, no atomics)
//   grad weight  gw[a,b] = sum_{n,i,j} gy[i,j] * xpad[i+a, j+b]: per-tile partial sums, then a fixed-order
//                          reduction over tiles and batch (deterministic)
//
// Storage type T of the large tensors (x, y, gy, gx): fp32 (include/paradis_sl.h) or bf16
// (include/paradis_geocyclic.h).  Weights, bias, partial sums and grad weight / grad bias are fp32, and the arithmetic
// is fp32 in registers either way: a bf16 result is the fp32 kernel's value rounded once (cvt.rn), i.e. bit-identical
// to running the fp32 entry points on .float() copies and casting back with .to(torch.bfloat16).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/paradis_sl.h"
#include "../../include/paradis_geocyclic.h"
#include "sl_device.cuh"

using psl::bf16;
using psl::kIsF32;
using psl::ldg_f;
using psl::st_f;

void psl_set_error(const char* msg);   // paradis_sl.cu: the calling thread's paradis_last_error() string

namespace {

constexpr int TW = 32, TH = 32, RPT = 4;   // tile 32 x 32 outputs, 256 threads, 4 vertically adjacent outputs each

// source of padded cell (i, j) (unpadded coordinates, may be outside [0,H) x [0,W)); model/padding.py:26-37
template <typename T>
__device__ __forceinline__ float geo_load(const T* __restrict__ x, int i, int j, int H, int W, int P) {
  if (i < -P || i >= H + P || j < -P || j >= W + P) return 0.0f;
  int shift = 0;
  if (i < 0) { i = -i; shift = W / 2; }
  else if (i >= H) { i = 2 * (H - 1) - i; shift = W / 2; }
  j -= shift;
  if (j < 0) j += W; else if (j >= W) j -= W;
  return ldg_f(x + (long long)i * W + j);
}

// zero rows outside the mesh, circular columns (the adjoint's view of grad_y)
template <typename T>
__device__ __forceinline__ float zc_load(const T* __restrict__ g, int i, int j, int H, int W) {
  if (i < 0 || i >= H) return 0.0f;
  if (j < 0) j += W; else if (j >= W) j -= W;
  if (j < 0 || j >= W) return 0.0f;
  return ldg_f(g + (long long)i * W + j);
}

// Polar-cap fold of grad input at (i, j): the padded row R folding onto row i (R = P-i north, 2(H-1)-i+P south),
// shifted by W/2.  Fixed order: taps a, then b.
template <int K, typename T>
__device__ __forceinline__ float cap_fold(const T* __restrict__ g, const float* __restrict__ wc, int R, int j, int H,
                                          int W) {
  constexpr int P = (K - 1) / 2;
  float s = 0.0f;
  for (int a = 0; a < K; ++a) {
    const int gi = R - a;                                        // output row that used padded row R with tap a
    if (gi < 0 || gi >= H) continue;
    for (int b = 0; b < K; ++b) {
      int gj = j + W / 2 + P - b;                                // padded column C = j + W/2 + P (mod W), output col C - b
      gj %= W;
      if (gj < 0) gj += W;
      s = fmaf(__ldg(wc + a * K + b), ldg_f(g + (long long)gi * W + gj), s);
    }
  }
  return s;
}

// MODE 0: forward (GeoCyclic source, filter as is, + bias).  MODE 1: direct part of grad input
// (zero-row / circular-column source, flipped filter).  T = storage type of src and dst.  With bf16 storage, MODE 1
// also folds the polar caps into rows 1..P and H-1-P..H-2 in registers, fl(direct + fold) in the caps kernel's order,
// so that each bf16 value is rounded once; the fp32 variant leaves that to geo_dwconv_bwd_caps_kernel.
template <int K, int MODE, typename T>
__global__ void __launch_bounds__(256) geo_dwconv_tile_kernel(const T* __restrict__ src, const float* __restrict__ w,
                                                              const float* __restrict__ bias, T* __restrict__ dst,
                                                              int C, int H, int W) {
  constexpr int P = (K - 1) / 2, SW = TW + K - 1, SH = TH + K - 1;
  __shared__ float tile[SH][SW + 1];
  const int plane = blockIdx.z, c = plane % C;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
  const T* s = src + (long long)plane * H * W;
  for (int idx = threadIdx.x; idx < SH * SW; idx += 256) {
    const int r = idx / SW, q = idx - r * SW;
    tile[r][q] = MODE == 0 ? geo_load(s, y0 + r - P, x0 + q - P, H, W, P) : zc_load(s, y0 + r - P, x0 + q - P, H, W);
  }
  float wk[K * K];
#pragma unroll
  for (int t = 0; t < K * K; ++t) wk[t] = __ldg(w + c * K * K + (MODE == 0 ? t : K * K - 1 - t));
  __syncthreads();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float acc[RPT];
  const float b0 = (MODE == 0 && bias) ? __ldg(bias + c) : 0.0f;
#pragma unroll
  for (int r = 0; r < RPT; ++r) acc[r] = b0;
#pragma unroll
  for (int b = 0; b < K; ++b) {
    float v[RPT + K - 1];
#pragma unroll
    for (int m = 0; m < RPT + K - 1; ++m) v[m] = tile[ty * RPT + m][tx + b];
#pragma unroll
    for (int a = 0; a < K; ++a)
#pragma unroll
      for (int r = 0; r < RPT; ++r) acc[r] = fmaf(wk[a * K + b], v[r + a], acc[r]);
  }
  const int j = x0 + tx;
  if (j < W) {
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      const int i = y0 + ty * RPT + r;
      if constexpr (MODE == 1 && !kIsF32<T>) {       // H >= 2P + 2: the two caps never fold onto the same row
        if (i >= 1 && i <= P) acc[r] += cap_fold<K>(s, w + c * K * K, P - i, j, H, W);
        else if (i >= H - 1 - P && i <= H - 2) acc[r] += cap_fold<K>(s, w + c * K * K, 2 * (H - 1) - i + P, j, H, W);
      }
      if (i < H) st_f(dst + ((long long)plane * H + i) * W + j, acc[r]);
    }
  }
}

// Polar-cap part of grad input (fp32 storage): rows 1..P receive the fold of padded rows P-i (north), rows
// H-1-P..H-2 the fold of padded rows 2(H-1)-i+P (south), both shifted by W/2.  Runs after the direct kernel (single
// writer per cell).
template <int K>
__global__ void geo_dwconv_bwd_caps_kernel(const float* __restrict__ gy, const float* __restrict__ w,
                                           float* __restrict__ gx, int C, int H, int W) {
  constexpr int P = (K - 1) / 2;
  const int plane = blockIdx.z, c = plane % C;
  const int which = blockIdx.y / P, k = blockIdx.y % P;            // which: 0 north, 1 south
  const int i = which == 0 ? 1 + k : H - 2 - k;                    // source row
  if (i < 1 || i > H - 2) return;
  if (which == 1 && i <= P && H - 2 - k <= P) { /* tiny meshes: both folds hit the row, handled below alike */ }
  const float* g = gy + (long long)plane * H * W;
  const float* wc = w + c * K * K;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < W; j += gridDim.x * blockDim.x) {
    const int R = which == 0 ? P - i : 2 * (H - 1) - i + P;       // padded row folding onto row i
    gx[((long long)plane * H + i) * W + j] += cap_fold<K>(g, wc, R, j, H, W);
  }
}

// grad weight / grad bias: per-tile partial sums, [plane][tile][K*K+1]
template <int K, typename T>
__global__ void __launch_bounds__(256) geo_dwconv_wgrad_kernel(const T* __restrict__ x, const T* __restrict__ gy,
                                                               float* __restrict__ partial, int C, int H, int W) {
  constexpr int P = (K - 1) / 2, SW = TW + K - 1, SH = TH + K - 1, NV = K * K + 1;
  __shared__ float tile[SH][SW + 1];
  __shared__ float red[8][NV];
  const int plane = blockIdx.z;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
  const T* s = x + (long long)plane * H * W;
  for (int idx = threadIdx.x; idx < SH * SW; idx += 256) {
    const int r = idx / SW, q = idx - r * SW;
    tile[r][q] = geo_load(s, y0 + r - P, x0 + q - P, H, W, P);
  }
  __syncthreads();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, lane = tx;
  float g[RPT];
#pragma unroll
  for (int r = 0; r < RPT; ++r) {
    const int i = y0 + ty * RPT + r, j = x0 + tx;
    g[r] = (i < H && j < W) ? ldg_f(gy + ((long long)plane * H + i) * W + j) : 0.0f;
  }
  float acc[NV];
#pragma unroll
  for (int t = 0; t < NV; ++t) acc[t] = 0.0f;
#pragma unroll
  for (int b = 0; b < K; ++b) {
    float v[RPT + K - 1];
#pragma unroll
    for (int m = 0; m < RPT + K - 1; ++m) v[m] = tile[ty * RPT + m][tx + b];
#pragma unroll
    for (int a = 0; a < K; ++a)
#pragma unroll
      for (int r = 0; r < RPT; ++r) acc[a * K + b] = fmaf(g[r], v[r + a], acc[a * K + b]);
  }
#pragma unroll
  for (int r = 0; r < RPT; ++r) acc[K * K] += g[r];
  // fixed-order reduction: lanes (xor tree), then the 8 warps in order
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    float vsum = acc[t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vsum += __shfl_xor_sync(0xffffffffu, vsum, o);
    if (lane == 0) red[ty][t] = vsum;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    float vsum = 0.0f;
    for (int wq = 0; wq < 8; ++wq) vsum += red[wq][threadIdx.x];
    const int tile_id = blockIdx.y * gridDim.x + blockIdx.x, ntiles = gridDim.x * gridDim.y;
    partial[((long long)plane * ntiles + tile_id) * NV + threadIdx.x] = vsum;
  }
}

// gw[c][t] = sum over batch n and tiles (ascending) of partial[n*C+c][tile][t]
__global__ void geo_dwconv_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ gw,
                                               float* __restrict__ gbias, int B, int C, int ntiles, int NV) {
  const int c = blockIdx.x, t = threadIdx.x;
  if (t >= NV) return;
  float s = 0.0f;
  for (int n = 0; n < B; ++n) {
    const float* p = partial + ((long long)(n * C + c) * ntiles) * NV + t;
    for (int k = 0; k < ntiles; ++k) s += p[(long long)k * NV];
  }
  if (t < NV - 1) gw[c * (NV - 1) + t] = s;
  else if (gbias) gbias[c] = s;
}

int err(int code, const char* msg) {
  psl_set_error(msg);
  return code;
}

int check(const void* a, const void* b, int B, int C, int H, int W, int k) {
  if (!a || !b) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: NULL tensor pointer");
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_dwconv: non-positive dimension");
  if (W % 2) return err(PARADIS_ERR_ODD_WIDTH, "Number of longitude points must be even");
  if (k != 3 && k != 5 && k != 7) return err(PARADIS_ERR_BAD_INTERP, "geocyclic_dwconv: kernel size must be 3, 5 or 7");
  // H >= 2P + 2: the north and the south cap never fold onto the same row (the cap kernel of the backward adds one
  // fold per block, see geo_dwconv_bwd_caps_kernel)
  if (H < k + 1 || W < k - 1) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_dwconv: mesh too small for the kernel size (H >= k + 1, W >= k - 1)");
  if ((long long)B * C > 65535) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_dwconv: B*C exceeds 65535 planes per call");
  return PARADIS_OK;
}

template <int K, typename T>
int run(int what, const T* a, const T* gy, const float* w, const float* bias, T* out, float* gw, float* gb, float* ws,
        int B, int C, int H, int W, cudaStream_t st) {
  dim3 grid((W + TW - 1) / TW, (H + TH - 1) / TH, B * C);
  if (what == 0) geo_dwconv_tile_kernel<K, 0, T><<<grid, 256, 0, st>>>(a, w, bias, out, C, H, W);
  else if (what == 1) {
    geo_dwconv_tile_kernel<K, 1, T><<<grid, 256, 0, st>>>(a, w, nullptr, out, C, H, W);
    if constexpr (kIsF32<T>) {                       // bf16: the caps are folded by the tile kernel
      dim3 cg((W + 255) / 256, 2 * ((K - 1) / 2), B * C);
      geo_dwconv_bwd_caps_kernel<K><<<cg, 256, 0, st>>>(a, w, out, C, H, W);
    }
  } else {
    geo_dwconv_wgrad_kernel<K, T><<<grid, 256, 0, st>>>(a, gy, ws, C, H, W);
    geo_dwconv_wgrad_reduce_kernel<<<C, 64, 0, st>>>(ws, gw, gb, B, C, grid.x * grid.y, K * K + 1);
  }
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : err(PARADIS_ERR_CUDA, cudaGetErrorString(e));
}

template <typename T>
int dispatch(int what, const T* a, const T* gy, const float* w, const float* bias, T* out, float* gw, float* gb,
             float* ws, int B, int C, int H, int W, int k, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (k == 3) return run<3>(what, a, gy, w, bias, out, gw, gb, ws, B, C, H, W, st);
  if (k == 5) return run<5>(what, a, gy, w, bias, out, gw, gb, ws, B, C, H, W, st);
  return run<7>(what, a, gy, w, bias, out, gw, gb, ws, B, C, H, W, st);
}


// PhysicalDownsample (model/blocks.py:57-71): GeoCyclic pad 2 + AvgPool2d(5, stride) = the 5x5 box mean of the padded
// field at every stride-th point.  One thread per OUTPUT point: only Ho x Wo values are computed and written (the
// round-1 version ran the full-resolution depthwise kernel and discarded all but 1 / stride^2 of it).
template <typename T>
__global__ void geo_avgpool5_kernel(const T* __restrict__ x, T* __restrict__ y, int H, int W, int Ho, int Wo,
                                    int stride) {
  const long long pl = blockIdx.z;
  const int io = blockIdx.y, jo = blockIdx.x * blockDim.x + threadIdx.x;
  if (jo >= Wo) return;
  const T* xp = x + pl * (long long)H * W;
  const int halfW = W >> 1;
  float s = 0.0f;
#pragma unroll
  for (int a = 0; a < 5; ++a) {
    int i = io * stride + a - 2, shift = 0;         // unpadded row of the tap
    if (i < 0) { i = -i; shift = halfW; }
    else if (i >= H) { i = 2 * (H - 1) - i; shift = halfW; }
    const T* row = xp + (long long)i * W;
    float r = 0.0f;
#pragma unroll
    for (int b = 0; b < 5; ++b) {
      int j = jo * stride + b - 2 - shift;
      if (j < 0) j += W;
      if (j < 0) j += W;
      if (j >= W) j -= W;
      r += ldg_f(row + j);
    }
    s += r;
  }
  st_f(y + (pl * Ho + io) * Wo + jo, s * (1.0f / 25.0f));
}

// Adjoint of geo_avgpool5_kernel, one thread per INPUT point (i, j): it gathers only the strided outputs whose 5x5
// GeoCyclic window covers it (about 25 / stride^2 of them; one integer division per coordinate outside the rare
// wrapped columns and cap rows).  It is the full-resolution grad-input composition -- grad_y scattered into a zero-filled
// [H, W] plane at every stride-th point, then the MODE-1 tile kernel with the flipped 1/25 box and the caps kernel --
// with the zero terms left out and the others visited in the same order: the direct part in the tile loop order
// (columns b outer, rows a inner), the polar-cap fold in the caps kernel's order, then fl(direct + fold).  Both sums
// start at +0 and can never reach -0, so adding an exact zero changes none of their bits: the result is bit-identical
// to the composition.
template <typename T>
__global__ void geo_avgpool5_bwd_kernel(const T* __restrict__ gy, T* __restrict__ gx, int H, int W, int Ho, int Wo,
                                        int stride) {
  const long long pl = blockIdx.z;
  const int i = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= W) return;
  const T* g = gy + pl * (long long)Ho * Wo;
  const float wbox = 1.0f / 25.0f;
  // covering output rows io = io0, io0 + 1, ...: mesh rows i + a - 2 = io * stride for a = a0, a0 + stride, ... <= a1
  const int io0 = ((i < 2 ? 0 : i - 2) + stride - 1) / stride;
  const int a0 = io0 * stride - i + 2, a1 = min(4, H + 1 - i);
  float acc = 0.0f;
  if (j >= 2 && j < W - 2) {                        // no column wraps: every stride-th column from jo0
    const int jo0 = (j - 2 + stride - 1) / stride;
    for (int b = jo0 * stride - j + 2, jo = jo0; b < 5; b += stride, ++jo)
      for (int a = a0, io = io0; a <= a1; a += stride, ++io)
        acc = fmaf(wbox, ldg_f(g + (long long)io * Wo + jo), acc);
  } else {
    for (int b = 0; b < 5; ++b) {
      int jj = j + b - 2;                           // circular columns
      if (jj < 0) jj += W; else if (jj >= W) jj -= W;
      if (jj % stride) continue;
      const int jo = jj / stride;
      for (int a = a0, io = io0; a <= a1; a += stride, ++io)
        acc = fmaf(wbox, ldg_f(g + (long long)io * Wo + jo), acc);
    }
  }
  if ((i >= 1 && i <= 2) || (i >= H - 3 && i <= H - 2)) {   // H >= 6: the two caps never fold onto the same row
    const int R = i <= 2 ? 2 - i : 2 * (H - 1) - i + 2;    // padded row folding onto row i
    float s = 0.0f;
    for (int a = 0; a < 5; ++a) {
      const int gi = R - a;
      if (gi < 0 || gi >= H || gi % stride) continue;
      const T* row = g + (long long)(gi / stride) * Wo;
      for (int b = 0; b < 5; ++b) {
        int gj = j + W / 2 + 2 - b;
        gj %= W;
        if (gj < 0) gj += W;
        if (gj % stride == 0) s = fmaf(wbox, ldg_f(row + gj / stride), s);
      }
    }
    acc += s;
  }
  st_f(gx + (pl * H + i) * W + j, acc);
}

template <typename T>
int avgpool5(bool backward, const T* src, T* dst, int B, int C, int H, int W, int stride, void* stream) {
  if (int rc = check(src, dst, B, C, H, W, 5)) return rc;
  if (stride < 1) return err(PARADIS_ERR_BAD_SHAPE, "geocyclic_avgpool5: stride must be >= 1");
  const int Ho = (H + 4 - 5) / stride + 1, Wo = (W + 4 - 5) / stride + 1;     // AvgPool2d(5, stride) of the padded plane
  if (backward) {
    dim3 grid((W + 127) / 128, H, B * C);
    geo_avgpool5_bwd_kernel<T><<<grid, 128, 0, (cudaStream_t)stream>>>(src, dst, H, W, Ho, Wo, stride);
  } else {
    dim3 grid((Wo + 127) / 128, Ho, B * C);
    geo_avgpool5_kernel<T><<<grid, 128, 0, (cudaStream_t)stream>>>(src, dst, H, W, Ho, Wo, stride);
  }
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? PARADIS_OK : err(PARADIS_ERR_CUDA, cudaGetErrorString(e));
}

}  // namespace

extern "C" int paradis_geocyclic_dwconv_fwd(const float* x, const float* weight, const float* bias, float* y, int B,
                                            int C, int H, int W, int k, void* stream) {
  if (int rc = check(x, y, B, C, H, W, k)) return rc;
  if (!weight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: weight is NULL");
  return dispatch<float>(0, x, nullptr, weight, bias, y, nullptr, nullptr, nullptr, B, C, H, W, k, stream);
}

extern "C" int paradis_geocyclic_dwconv_bwd_input(const float* gy, const float* weight, float* gx, int B, int C, int H,
                                                  int W, int k, void* stream) {
  if (int rc = check(gy, gx, B, C, H, W, k)) return rc;
  if (!weight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: weight is NULL");
  return dispatch<float>(1, gy, nullptr, weight, nullptr, gx, nullptr, nullptr, nullptr, B, C, H, W, k, stream);
}

extern "C" size_t paradis_geocyclic_dwconv_wgrad_workspace(int B, int C, int H, int W, int k) {
  const size_t tiles = (size_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH);
  return (size_t)B * C * tiles * (k * k + 1) * sizeof(float);
}

extern "C" int paradis_geocyclic_dwconv_bwd_weight(const float* x, const float* gy, float* gweight, float* gbias,
                                                   int B, int C, int H, int W, int k, void* workspace,
                                                   size_t workspace_bytes, void* stream) {
  if (int rc = check(x, gy, B, C, H, W, k)) return rc;
  if (!gweight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: grad weight is NULL");
  if (!workspace || workspace_bytes < paradis_geocyclic_dwconv_wgrad_workspace(B, C, H, W, k))
    return err(PARADIS_ERR_WORKSPACE, "geocyclic_dwconv: weight-gradient workspace too small");
  return dispatch<float>(2, x, gy, nullptr, nullptr, nullptr, gweight, gbias, (float*)workspace, B, C, H, W, k, stream);
}

extern "C" int paradis_geocyclic_avgpool5_fwd(const float* x, float* y, int B, int C, int H, int W, int stride, void* stream) {
  return avgpool5<float>(false, x, y, B, C, H, W, stride, stream);
}

extern "C" int paradis_geocyclic_avgpool5_bwd(const float* gy, float* gx, int B, int C, int H, int W, int stride,
                                              void* stream) {
  return avgpool5<float>(true, gy, gx, B, C, H, W, stride, stream);
}

// bf16 storage (include/paradis_geocyclic.h)
extern "C" int paradis_geocyclic_dwconv_fwd_bf16(const void* x, const float* weight, const float* bias, void* y, int B,
                                                 int C, int H, int W, int k, void* stream) {
  if (int rc = check(x, y, B, C, H, W, k)) return rc;
  if (!weight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: weight is NULL");
  return dispatch<bf16>(0, (const bf16*)x, nullptr, weight, bias, (bf16*)y, nullptr, nullptr, nullptr, B, C, H, W, k,
                        stream);
}

extern "C" int paradis_geocyclic_dwconv_bwd_input_bf16(const void* gy, const float* weight, void* gx, int B, int C,
                                                       int H, int W, int k, void* stream) {
  if (int rc = check(gy, gx, B, C, H, W, k)) return rc;
  if (!weight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: weight is NULL");
  return dispatch<bf16>(1, (const bf16*)gy, nullptr, weight, nullptr, (bf16*)gx, nullptr, nullptr, nullptr, B, C, H, W,
                        k, stream);
}

extern "C" int paradis_geocyclic_dwconv_bwd_weight_bf16(const void* x, const void* gy, float* gweight, float* gbias,
                                                        int B, int C, int H, int W, int k, void* workspace,
                                                        size_t workspace_bytes, void* stream) {
  if (int rc = check(x, gy, B, C, H, W, k)) return rc;
  if (!gweight) return err(PARADIS_ERR_NULL_POINTER, "geocyclic_dwconv: grad weight is NULL");
  if (!workspace || workspace_bytes < paradis_geocyclic_dwconv_wgrad_workspace(B, C, H, W, k))
    return err(PARADIS_ERR_WORKSPACE, "geocyclic_dwconv: weight-gradient workspace too small");
  return dispatch<bf16>(2, (const bf16*)x, (const bf16*)gy, nullptr, nullptr, nullptr, gweight, gbias,
                        (float*)workspace, B, C, H, W, k, stream);
}

extern "C" int paradis_geocyclic_avgpool5_fwd_bf16(const void* x, void* y, int B, int C, int H, int W, int stride,
                                                   void* stream) {
  return avgpool5<bf16>(false, (const bf16*)x, (bf16*)y, B, C, H, W, stride, stream);
}

extern "C" int paradis_geocyclic_avgpool5_bwd_bf16(const void* gy, void* gx, int B, int C, int H, int W, int stride,
                                                   void* stream) {
  return avgpool5<bf16>(true, (const bf16*)gy, (bf16*)gx, B, C, H, W, stride, stream);
}
