// Train-mode conv4_2 of the VGGish body (reference vggish.py:108-118, features.13 = Conv2d(512, 512, 3, padding=1) +
// ReLU + MaxPool2d(2, 2)) with conv1 .. conv4_1 frozen: the gradient stops at conv4_2's weights, so no transposed
// convolution is needed.
//
//   forward   conv4_1's 16-bit output -> im2col planes [pixels][3 * 4608] -> z = im2col W^T + b  [n * 96][512] fp32
//             -> relu, 2x2 max-pool, (h, w, c) flatten -> fc1's input planes (fc_train.cu takes it from there)
//   backward  dX1 (fc1's input gradient) -> dz: each pooled element's gradient to the first maximum of its window in
//             scan order (as PyTorch), masked by z > 0 -> db = colsum dz, dW = sum over pixels dz^T im2col
//
// Every GEMM is the head trainer's three-plane split-bf16 GEMM (planes_gemm_sm100.cu, fp32-equivalent operands,
// DESIGN §5.5).  conv4_1's outputs are bf16, fp16 or hi + lo bf16 values, all exact in fp32, and their three-plane split
// is exact.  The 4 608-column contraction of the forward GEMM runs in kFwdSlice slices added into a zeroed z; the
// weight gradient contracts over the pixels in slices of at most kDwSlice rows.  The im2col planes (2.65 MB per
// example) are built kConv42Chunk examples at a time into one buffer, in the forward pass and again in the backward
// pass, from conv4_1's output that the workspace keeps.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "fc_train.cuh"
#include "igemm_sm100.cuh"
#include "kernels.cuh"

namespace vmb {

namespace {

constexpr int kPl = 3;
constexpr int kC = kConv42C, kPix = kConv42Pix, kK = kConv42K;
constexpr int kH = 12, kW = 8;

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

unsigned grid_for(long long total) {
  return static_cast<unsigned>(std::max<long long>(1, std::min<long long>((total + 255) / 256, 148LL * 16)));
}

__device__ __forceinline__ void store3(float v, __nv_bfloat16* dst, long long plane_stride) {
  __nv_bfloat16 h, m, l;
  split_bf16(v, h, m, l);
  dst[0] = h;
  dst[plane_stride] = m;
  dst[2 * plane_stride] = l;
}

// one activation of conv4_1's output (NHWC [n][12][8][512]; precision 1: [n][2][12][8][512] hi | lo) as fp32 (exact)
__device__ __forceinline__ float act_at(const void* act, int precision, long long e) {
  if (precision == 1) {
    const long long img = e / (kPix * kC), r = e - img * (kPix * kC);
    const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(act) + img * (2 * kPix * kC) + r;
    return __bfloat162float(p[0]) + __bfloat162float(p[kPix * kC]);
  }
  if (precision == 2) return __half2float(static_cast<const __half*>(act)[e]);
  return __bfloat162float(static_cast<const __nv_bfloat16*>(act)[e]);
}

// w fp32 OIHW [512][512][3][3] -> planes [512][3 * 4608], column k = (kh * 3 + kw) * 512 + c (the im2col order)
__global__ void __launch_bounds__(256)
conv42_weight_planes_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ planes) {
  const long long total = static_cast<long long>(kC) * kK;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long o = i / kK;
    const int k = static_cast<int>(i - o * kK);
    const int tap = k / kC, c = k - tap * kC;
    store3(__ldg(w + (o * kC + c) * 9 + tap), planes + o * (kPl * kK) + k, kK);
  }
}

// im2col planes of examples [e0, e0 + e): row r = (example - e0) * 96 + h * 8 + w, column (kh * 3 + kw) * 512 + c holds
// act[example][h + kh - 1][w + kw - 1][c], zero outside the 12 x 8 image (Conv2d padding 1).  One thread per 8 channels.
__global__ void __launch_bounds__(256)
im2col_planes_kernel(const void* __restrict__ act, int precision, long long e0, long long e,
                     __nv_bfloat16* __restrict__ cols) {
  constexpr int kGroups = kK / 8;   // 576 groups of 8 columns per row
  const long long total = e * kPix * kGroups;
  for (long long u = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; u < total;
       u += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = u / kGroups;
    const int gi = static_cast<int>(u - r * kGroups);
    const int tap = gi / (kC / 8), c0 = (gi - tap * (kC / 8)) * 8;
    const long long ex = e0 + r / kPix;
    const int pix = static_cast<int>(r % kPix);
    const int hh = pix / kW + tap / 3 - 1, ww = pix % kW + tap % 3 - 1;
    alignas(16) __nv_bfloat16 pl[3][8];
    const bool in = hh >= 0 && hh < kH && ww >= 0 && ww < kW;
    const long long src = ((ex * kH + hh) * kW + ww) * kC + c0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = in ? act_at(act, precision, src + j) : 0.f;
      split_bf16(v, pl[0][j], pl[1][j], pl[2][j]);
    }
    __nv_bfloat16* dst = cols + r * (kPl * kK) + tap * kC + c0;
#pragma unroll
    for (int p = 0; p < 3; ++p) *reinterpret_cast<uint4*>(dst + p * kK) = *reinterpret_cast<const uint4*>(pl[p]);
  }
}

// z [n * 96][512] -> relu(max over each 2x2 window) -> fc1's input planes [n_pad][3 * 12288], column (ph * 4 + pw) * 512
// + c (the (h, w, c) flatten, vggish.py:26-29); rows >= n zero
__global__ void __launch_bounds__(256)
pool_fwd_kernel(const float* __restrict__ z, long long n, long long n_pad, __nv_bfloat16* __restrict__ planes) {
  constexpr int F = kFcTrainIn;
  const long long total = n_pad * F;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / F;
    const int j = static_cast<int>(i - row * F);
    float v = 0.f;
    if (row < n) {
      const int win = j / kC, c = j - win * kC;
      const float* p = z + (row * kPix + (win / 4) * 2 * kW + (win % 4) * 2) * kC + c;
      v = fmaxf(fmaxf(fmaxf(__ldg(p), __ldg(p + kC)), fmaxf(__ldg(p + kW * kC), __ldg(p + (kW + 1) * kC))), 0.f);
    }
    store3(v, planes + row * (kPl * F) + j, F);
  }
}

// dX1 [n][12288] -> dz planes [n * 96][3 * 512] and colsum[c] += sum of dz (double).  Each window's gradient goes to the
// first maximum in scan order ((0,0), (0,1), (1,0), (1,1)), masked by z > 0; the other three elements get zero.
// grid (512 / 128, ceil(n * 24 / kWin)), block 128 = one channel per thread, kWin windows per block.
constexpr int kWin = 64;
__global__ void __launch_bounds__(128)
pool_bwd_kernel(const float* __restrict__ dx1, const float* __restrict__ z, long long n,
                __nv_bfloat16* __restrict__ dz, double* __restrict__ colsum) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  const long long w0 = static_cast<long long>(blockIdx.y) * kWin, windows = n * 24;
  double s = 0.0;
  for (int i = 0; i < kWin; ++i) {
    const long long wi = w0 + i;
    if (wi >= windows) break;
    const long long ex = wi / 24;
    const int win = static_cast<int>(wi - ex * 24);
    const long long pix0 = ex * kPix + (win / 4) * 2 * kW + (win % 4) * 2;
    const long long off[4] = {pix0, pix0 + 1, pix0 + kW, pix0 + kW + 1};
    float zv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) zv[q] = __ldg(z + off[q] * kC + c);
    int arg = 0;
#pragma unroll
    for (int q = 1; q < 4; ++q)
      if (zv[q] > zv[arg]) arg = q;
    const float g = zv[arg] > 0.f ? __ldg(dx1 + ex * kFcTrainIn + win * kC + c) : 0.f;
    s += g;
#pragma unroll
    for (int q = 0; q < 4; ++q) store3(q == arg ? g : 0.f, dz + off[q] * (kPl * kC) + c, kC);
  }
  atomicAdd(colsum + c, s);
}

// dw [512][4608] in (kh, kw, c) order -> grads OIHW [512][512][3][3], then the bias [512] from colsum
__global__ void __launch_bounds__(256)
conv42_grad_store_kernel(const float* __restrict__ dw, const double* __restrict__ colsum, float* __restrict__ grads) {
  const long long total = kConv42GradCount;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (i >= static_cast<long long>(kC) * kK) {
      grads[i] = static_cast<float>(colsum[i - static_cast<long long>(kC) * kK]);
      continue;
    }
    const long long o = i / kK;
    const int r = static_cast<int>(i - o * kK);
    const int c = r / 9, tap = r - c * 9;
    grads[i] = __ldg(dw + o * kK + tap * kC + c);
  }
}

int fail(const char* what) {
  set_kernel_error("conv4_2 train: %s", what);
  return 1;
}

int im2col(const void* act, int precision, long long e0, long long e, void* cols, cudaStream_t st) {
  im2col_planes_kernel<<<grid_for(e * kPix * (kK / 8)), 256, 0, st>>>(act, precision, e0, e,
                                                                      static_cast<__nv_bfloat16*>(cols));
  count_launch();
  return check_launch("im2col_planes_kernel");
}

}  // namespace

Conv42Layout conv4_2_layout(long long n, size_t conv_bytes) {
  Conv42Layout L{};
  L.fc = fc_train_layout(n, conv_bytes);
  const size_t rows = size_t(n) * kPix;
  size_t o = L.fc.total;
  auto take = [&](size_t bytes) {
    const size_t at = o;
    o = align_up(o + bytes, 1024);
    return at;
  };
  L.z = take(rows * kC * 4);
  L.dz = take(rows * kPl * kC * 2);
  L.dx1 = take(size_t(n) * kFcTrainIn * 4);
  L.dw = take(size_t(kC) * kK * 4);
  L.colsum = take(size_t(kC) * 8);
  L.cols = take(size_t(std::min<long long>(n, kConv42Chunk)) * kPix * kPl * kK * 2);
  L.total = o;
  return L;
}

int conv4_2_weight_planes(const float* w_oihw, void* planes, cudaStream_t st) {
  conv42_weight_planes_kernel<<<grid_for(static_cast<long long>(kC) * kK), 256, 0, st>>>(
      w_oihw, static_cast<__nv_bfloat16*>(planes));
  count_launch();
  return check_launch("conv42_weight_planes_kernel");
}

int conv4_2_train_forward(const void* w_planes, const float* bias, const void* act, int precision, long long n, char* ws,
                          const Conv42Layout& L, cudaStream_t st) {
  float* z = reinterpret_cast<float*>(ws + L.z);
  if (cudaMemsetAsync(z, 0, size_t(n) * kPix * kC * 4, st) != cudaSuccess) return fail("z clear failed");
  const int ks = (kK + kFwdSlice - 1) / kFwdSlice;
  for (long long e0 = 0; e0 < n; e0 += kConv42Chunk) {
    const long long e = std::min<long long>(kConv42Chunk, n - e0);
    if (im2col(act, precision, e0, e, ws + L.cols, st)) return 1;
    if (planes_gemm(ws + L.cols, w_planes, bias, z + e0 * kPix * kC, kC, 0, int(e * kPix), kC, kK, kPl, ks, st))
      return fail(planes_gemm_last_error());
  }
  pool_fwd_kernel<<<grid_for(L.fc.n_pad * kFcTrainIn), 256, 0, st>>>(z, n, L.fc.n_pad,
                                                                     reinterpret_cast<__nv_bfloat16*>(ws + L.fc.x));
  count_launch();
  return check_launch("pool_fwd_kernel");
}

int conv4_2_train_backward(const void* act, int precision, long long n, char* ws, const Conv42Layout& L, float* grads,
                           cudaStream_t st) {
  const float* z = reinterpret_cast<const float*>(ws + L.z);
  __nv_bfloat16* dz = reinterpret_cast<__nv_bfloat16*>(ws + L.dz);
  float* dw = reinterpret_cast<float*>(ws + L.dw);
  double* colsum = reinterpret_cast<double*>(ws + L.colsum);
  if (cudaMemsetAsync(colsum, 0, size_t(kC) * 8, st) != cudaSuccess ||
      cudaMemsetAsync(dw, 0, size_t(kC) * kK * 4, st) != cudaSuccess)
    return fail("gradient clear failed");
  {
    const dim3 grid(kC / 128, static_cast<unsigned>((n * 24 + kWin - 1) / kWin));
    pool_bwd_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const float*>(ws + L.dx1), z, n, dz, colsum);
    count_launch();
    if (check_launch("pool_bwd_kernel")) return 1;
  }
  for (long long e0 = 0; e0 < n; e0 += kConv42Chunk) {
    const long long e = std::min<long long>(kConv42Chunk, n - e0);
    const int rows = int(e * kPix);
    const int ks = (rows + kDwSlice - 1) / kDwSlice;
    if (im2col(act, precision, e0, e, ws + L.cols, st)) return 1;
    if (planes_gemm_mn(dz + e0 * kPix * kPl * kC, kC, ws + L.cols, kK, dw, kK, kC, kK, rows, kPl, ks > 1 ? ks : -1, st))
      return fail(planes_gemm_last_error());
  }
  conv42_grad_store_kernel<<<grid_for(kConv42GradCount), 256, 0, st>>>(dw, colsum, grads);
  count_launch();
  return check_launch("conv42_grad_store_kernel");
}

}  // namespace vmb
