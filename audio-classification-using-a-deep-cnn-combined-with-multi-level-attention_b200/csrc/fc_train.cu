// Train-mode FC stack of the VGGish body (reference vggish.py:13-19, :31 — embeddings.{0,2,4} = Linear + ReLU three
// times — trained by train.py:133-138 with the second Adam of train.py:370), with the conv stack frozen.
//
// Every Linear runs on the head trainer's GEMM engine (planes_gemm_sm100.cu) with three-plane split-bf16 operands
// (hi | mid | lo: fp32-equivalent, DESIGN §5.5): the handle's 16-bit FC weights would move pre-activations by ~1e-3 and
// flip ReLU masks, and one flipped mask moves a whole weight-gradient row.
//
//   forward   X planes (conv features) -> Z1 = X W1^T + b1 -> A1 = relu(Z1) -> Z2 -> A2 -> Z3 -> E = relu(Z3)
//   backward  G3 = dE [Z3 > 0]   -> dW3 = G3^T A2, db3 = colsum G3, dA2 = G3 W3
//             G2 = dA2 [Z2 > 0]  -> dW2 = G2^T A1, db2,             dA1 = G2 W2
//             G1 = dA1 [Z1 > 0]  -> dW1 = G1^T X,  db1              (no dX: the convs are frozen)
//
// Contractions longer than kFwdSlice columns (fc1: 12 288, fc2 / fc3 and the dgrad of fc2: 4 096) are cut into K slices
// that run on different SMs and add into a zeroed fp32 output: one tcgen05 accumulator over 768 K-steps truncates
// enough to miss the oracle (the wide head layer, DESIGN §5.5), slices of 768 columns do not.  The weight gradients
// contract over the B*T rows in slices of at most kDwSlice rows (planes_gemm_dw, shared with the head trainer).
// Between GEMMs one element-wise pass per layer applies the ReLU (forward) or the ReLU mask (backward), writes the next
// operand planes and, in the backward pass, the column sums that are the bias gradient.
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

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__device__ __forceinline__ void store3(float v, __nv_bfloat16* dst, long long plane_stride) {
  __nv_bfloat16 h, m, l;
  split_bf16(v, h, m, l);
  dst[0] = h;
  dst[plane_stride] = m;
  dst[2 * plane_stride] = l;
}

// W fp32 [rows][cols] -> planes [rows][3 * cols] and (optionally) the transposed planes [cols][3 * rows].
// rows, cols multiples of 32; block (32, 8), one 32 x 32 tile per CTA.
__global__ void __launch_bounds__(256)
fc_weight_planes_kernel(const float* __restrict__ w, int rows, int cols, __nv_bfloat16* __restrict__ planes,
                        __nv_bfloat16* __restrict__ planes_t) {
  __shared__ float tile[32][33];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + ty + 8 * i, c = c0 + tx;
    const float v = __ldg(w + static_cast<long long>(r) * cols + c);
    tile[ty + 8 * i][tx] = v;
    if (planes) store3(v, planes + static_cast<long long>(r) * (kPl * cols) + c, cols);
  }
  if (!planes_t) return;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + ty + 8 * i, r = r0 + tx;
    store3(tile[tx][ty + 8 * i], planes_t + static_cast<long long>(c) * (kPl * rows) + r, rows);
  }
}

// conv features [n][12288] in the handle's format -> fp32 value -> planes [n_pad][3 * 12288] (rows >= n: zero).
// precision 0: bf16; 1: hi | lo bf16 pair per row ([n][2 * 12288]); 2: fp16.  Every 16-bit value (and hi + lo) is
// exact in fp32 and its three-plane split is exact: the planes carry the features the inference path computed.
__global__ void __launch_bounds__(256)
fc_feature_planes_kernel(const void* __restrict__ feat, int precision, long long n, long long n_pad,
                         __nv_bfloat16* __restrict__ planes) {
  constexpr int F = kFcTrainIn;
  const long long total = n_pad * F;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / F;
    const int c = static_cast<int>(i - r * F);
    float v = 0.f;
    if (r < n) {
      if (precision == 1) {
        const __nv_bfloat16* row = static_cast<const __nv_bfloat16*>(feat) + r * (2 * F);
        v = __bfloat162float(row[c]) + __bfloat162float(row[F + c]);
      } else if (precision == 2) {
        v = __half2float(static_cast<const __half*>(feat)[r * F + c]);
      } else {
        v = __bfloat162float(static_cast<const __nv_bfloat16*>(feat)[r * F + c]);
      }
    }
    store3(v, planes + r * (kPl * F) + c, F);
  }
}

// One element-wise pass between GEMMs over z fp32 [rows][cols] (cols % 128 == 0):
//   forward  (mask == null): v = relu(z)
//   backward (mask != null): v = z * [mask > 0]   (mask: the layer's saved pre-activation)
// v -> planes [rows_pad][3 * cols] (rows >= rows: zero), out fp32 [rows][cols] (optional), colsum[c] += sum_r v
// (optional, double).  grid (cols / 128, ceil(rows_pad / 64)), block 256 = 128 columns x 2 row lanes.
__global__ void __launch_bounds__(256)
fc_act_kernel(const float* __restrict__ z, const float* __restrict__ mask, long long rows, long long rows_pad, int cols,
              __nv_bfloat16* __restrict__ planes, float* __restrict__ out, double* __restrict__ colsum) {
  const int c = blockIdx.x * 128 + (threadIdx.x & 127);
  const int ty = threadIdx.x >> 7;
  const long long r0 = static_cast<long long>(blockIdx.y) * 64;
  double s = 0.0;
  for (int i = ty; i < 64; i += 2) {
    const long long r = r0 + i;
    if (r >= rows_pad) break;
    float v = 0.f;
    if (r < rows) {
      const long long e = r * cols + c;
      const float a = __ldg(z + e);
      v = mask ? (__ldg(mask + e) > 0.f ? a : 0.f) : fmaxf(a, 0.f);
      if (out) out[e] = v;
      s += v;
    }
    store3(v, planes + r * (kPl * cols) + c, cols);
  }
  if (!colsum) return;
  __shared__ double part[128];
  if (ty == 1) part[threadIdx.x & 127] = s;
  __syncthreads();
  if (ty == 0) atomicAdd(colsum + c, s + part[threadIdx.x]);
}

__global__ void fc_colsum_store_kernel(const double* __restrict__ acc, float* __restrict__ dst, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = static_cast<float>(acc[i]);
}

int launch_check(const char* what) { return check_launch(what); }

int act(const float* z, const float* mask, long long rows, long long rows_pad, int cols, void* planes, float* out,
        double* colsum, cudaStream_t st) {
  const dim3 grid(static_cast<unsigned>(cols / 128), static_cast<unsigned>((rows_pad + 63) / 64));
  fc_act_kernel<<<grid, 256, 0, st>>>(z, mask, rows, rows_pad, cols, static_cast<__nv_bfloat16*>(planes), out, colsum);
  count_launch();
  return launch_check(mask ? "fc_act_kernel (ReLU mask)" : "fc_act_kernel (ReLU)");
}

// out fp32 [M][N] = A[M][K] W[N][K]^T (+ bias), K sliced by kFwdSlice columns into a zeroed out when K is longer
int gemm(const void* a, const void* w, const float* bias, float* out, long long M, int N, int K, cudaStream_t st) {
  const int ks = K > kFwdSlice ? (K + kFwdSlice - 1) / kFwdSlice : 0;
  if (ks && cudaMemsetAsync(out, 0, size_t(M) * N * sizeof(float), st) != cudaSuccess) {
    set_kernel_error("fc_train: GEMM output clear failed");
    return 1;
  }
  if (planes_gemm(a, w, bias, out, N, 0, int(M), N, K, kPl, ks, st)) {
    set_kernel_error("fc_train: %s", planes_gemm_last_error());
    return 1;
  }
  return 0;
}

// dW fp32 [M][N] = sum over the K rows of a[r][m] b[r][n]
int gemm_dw(const void* a, int a_cols, const void* b, int b_cols, float* out, int M, int N, long long K,
            cudaStream_t st) {
  if (planes_gemm_dw(a, a_cols, b, b_cols, out, N, M, N, int(K), kPl, st)) {
    set_kernel_error("fc_train: %s", planes_gemm_last_error());
    return 1;
  }
  return 0;
}

}  // namespace

FcTrainLayout fc_train_layout(long long n, size_t conv_bytes) {
  FcTrainLayout L{};
  L.n_pad = (n + 63) / 64 * 64;
  const size_t np = size_t(L.n_pad);
  size_t o = 0;
  auto take = [&](size_t bytes) {
    const size_t at = o;
    o = align_up(o + bytes, 1024);
    return at;
  };
  L.x = take(np * kPl * kFcTrainIn * 2);
  L.a1 = take(np * kPl * 4096 * 2);
  L.a2 = take(np * kPl * 4096 * 2);
  L.z1 = take(np * 4096 * 4);
  L.z2 = take(np * 4096 * 4);
  L.z3 = take(np * 128 * 4);
  L.g = take(np * kPl * 4096 * 2);
  L.da = take(np * 4096 * 4);
  L.colsum = take(size_t(4096 + 4096 + 128) * 8);
  L.conv = take(conv_bytes);
  L.total = o;
  return L;
}

int fc_weight_planes(const float* w, int rows, int cols, void* planes, void* planes_t, cudaStream_t st) {
  fc_weight_planes_kernel<<<dim3(cols / 32, rows / 32), dim3(32, 8), 0, st>>>(
      w, rows, cols, static_cast<__nv_bfloat16*>(planes), static_cast<__nv_bfloat16*>(planes_t));
  count_launch();
  return launch_check("fc_weight_planes_kernel");
}

int fc_train_forward(const void* const w_planes[3], const float* const bias[3], const void* features, int precision,
                     long long n, char* ws, const FcTrainLayout& L, float* emb, cudaStream_t st) {
  const long long np = L.n_pad;
  void* x = ws + L.x;
  if (features) {
    const long long total = np * kFcTrainIn;
    const unsigned grid = static_cast<unsigned>(std::min<long long>((total + 255) / 256, 148LL * 16));
    fc_feature_planes_kernel<<<grid, 256, 0, st>>>(features, precision, n, np, static_cast<__nv_bfloat16*>(x));
    count_launch();
    if (launch_check("fc_feature_planes_kernel")) return 1;
  }
  float* z1 = reinterpret_cast<float*>(ws + L.z1);
  float* z2 = reinterpret_cast<float*>(ws + L.z2);
  float* z3 = reinterpret_cast<float*>(ws + L.z3);
  if (gemm(x, w_planes[0], bias[0], z1, n, 4096, kFcTrainIn, st)) return 1;
  if (act(z1, nullptr, n, np, 4096, ws + L.a1, nullptr, nullptr, st)) return 1;
  if (gemm(ws + L.a1, w_planes[1], bias[1], z2, n, 4096, 4096, st)) return 1;
  if (act(z2, nullptr, n, np, 4096, ws + L.a2, nullptr, nullptr, st)) return 1;
  if (gemm(ws + L.a2, w_planes[2], bias[2], z3, n, 128, 4096, st)) return 1;
  // E = relu(Z3): the embeddings; the planes written on the way are overwritten by the backward pass's G3
  return act(z3, nullptr, n, np, 128, ws + L.g, emb, nullptr, st);
}

int fc_train_backward(const void* const wt_planes[3], long long n, char* ws, const FcTrainLayout& L,
                      const float* d_emb, float* grads, float* dx, cudaStream_t st) {
  const long long np = L.n_pad;
  const float* z1 = reinterpret_cast<const float*>(ws + L.z1);
  const float* z2 = reinterpret_cast<const float*>(ws + L.z2);
  const float* z3 = reinterpret_cast<const float*>(ws + L.z3);
  float* da = reinterpret_cast<float*>(ws + L.da);
  void* g = ws + L.g;
  double* colsum = reinterpret_cast<double*>(ws + L.colsum);
  const bool wgrad = grads != nullptr;
  float* dw[3] = {grads + kFcGradW1, grads + kFcGradW2, grads + kFcGradW3};
  float* db[3] = {grads + kFcGradB1, grads + kFcGradB2, grads + kFcGradB3};
  double* cs[3] = {nullptr, nullptr, nullptr};
  if (wgrad) {
    cs[0] = colsum, cs[1] = colsum + 4096, cs[2] = colsum + 8192;
    if (cudaMemsetAsync(colsum, 0, size_t(4096 + 4096 + 128) * 8, st) != cudaSuccess) {
      set_kernel_error("fc_train: column-sum clear failed");
      return 1;
    }
  }
  // fc3
  if (act(d_emb, z3, n, np, 128, g, nullptr, cs[2], st)) return 1;
  if (wgrad && gemm_dw(g, 128, ws + L.a2, 4096, dw[2], 128, 4096, np, st)) return 1;
  if (gemm(g, wt_planes[2], nullptr, da, n, 4096, 128, st)) return 1;
  // fc2
  if (act(da, z2, n, np, 4096, g, nullptr, cs[1], st)) return 1;
  if (wgrad && gemm_dw(g, 4096, ws + L.a1, 4096, dw[1], 4096, 4096, np, st)) return 1;
  if (gemm(g, wt_planes[1], nullptr, da, n, 4096, 4096, st)) return 1;
  // fc1: weight and bias gradients, and with dx the input gradient (K = 4096, sliced like fc2's dgrad)
  if (act(da, z1, n, np, 4096, g, nullptr, cs[0], st)) return 1;
  if (wgrad && gemm_dw(g, 4096, ws + L.x, kFcTrainIn, dw[0], 4096, kFcTrainIn, np, st)) return 1;
  if (dx && gemm(g, wt_planes[0], nullptr, dx, n, kFcTrainIn, 4096, st)) return 1;
  for (int i = 0; i < 3 && wgrad; ++i) {
    const int nb = i == 2 ? 128 : 4096;
    fc_colsum_store_kernel<<<(nb + 255) / 256, 256, 0, st>>>(cs[i], db[i], nb);
    count_launch();
    if (launch_check("fc_colsum_store_kernel")) return 1;
  }
  return 0;
}

}  // namespace vmb
