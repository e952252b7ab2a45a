// Multi-level attention head: one training step (forward in train mode + backward) on the B200.
// Reference semantics: model.py:200-269 run under train.py:119-138 — BatchNorm1d(T) with batch statistics per time
// step over (batch, features) (SURVEY F5), Dropout(p) after each ReLU, fcv feeding both attention branches and fcf
// never used (F3: no gradient), softmax over the class axis (F4), BatchNorm1d(K) + sigmoid on the output Linear,
// nn.CrossEntropyLoss applied to the sigmoid outputs (train.py:131,372).  Running statistics are updated like
// nn.BatchNorm1d does (momentum 0.1, unbiased variance).
//
// Every Linear (forward, dX and dW) is a 3-plane split-bf16 tcgen05 GEMM (planes_gemm_sm100.cu with hi | mid | lo
// operands = fp32-equivalent: with 2 planes the 4e-5 error on pre-activations flipped a few ReLU masks per step against
// the fp32 reference, which moves whole gradient elements).  The dW GEMMs read the same row-major planes as the forward
// and dX GEMMs, as MN-major operands (planes_gemm_dw).  Everything between GEMMs is fp32 CUDA-core work in a handful of
// kernels:
//   bn_time_stats / bn_col_stats   sum and sum-of-squares per time step (or per class), finalised by the last block
//   tile_split<Functor>            64x64 tiles: evaluate an element-wise functor (BN + ReLU + dropout, BN backward),
//                                  write hi|mid|lo bf16 planes row-major (the weights also transposed: the dX GEMMs'
//                                  B operand), optionally the fp32 values and the column sums (bias gradients)
//   att_forward / att_backward     attention pooling over the T time steps of one clip per CTA
//   out_loss_rows / out_bn_backward  sigmoid + cross-entropy + BatchNorm1d(K) backward
// Gradients land in one flat fp32 buffer with the layout of the parameters (vmb_mla_train_layout), ready for a single
// NCCL all-reduce; vmb_adam_step applies torch.optim.Adam's update to the flat buffers.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/vggish_mla_b200.h"
#include "igemm_sm100.cuh"
#include "sm100_ptx.cuh"
#include "kernels.cuh"

namespace vmb {
void set_api_error(const char* msg);
}

namespace {

constexpr int kMaxLevels = 4, kMaxFc = 4, kMaxBn = kMaxLevels * (1 + kMaxFc) + 2 * kMaxLevels + 1;
constexpr float kBnEps = 1e-5f;
constexpr float kBnMomentum = 0.1f;
constexpr int kPl = 3;   // bf16 planes per GEMM operand: hi | mid | lo (fp32-equivalent, see vmb::split_bf16)

int fail(const char* fmt, const char* detail = "") {
  char buf[640];
  snprintf(buf, sizeof buf, fmt, detail);
  vmb::set_api_error(buf);
  return 1;
}
int pad128(int v) { return (v + 127) / 128 * 128; }
long long pad64(long long v) { return (v + 63) / 64 * 64; }
size_t up(size_t v) { return (v + 1023) / 1024 * 1024; }

// ------------------------------------------------------------------ statistics
// acc[ch] = {sum, sum of squares}; stat[ch] = {mean, rstd}.  The last block to finish turns acc into stat and
// updates the running statistics.
struct StatJob {
  double* acc;          // [channels][2], zeroed at step start
  float* stat;          // [channels][2]
  unsigned* counter;    // zeroed at step start
  float* run_mean;      // may be null
  float* run_var;
  double count;         // elements per channel
  int channels;
};

__device__ void finalize_stats(const StatJob& j) {
  for (int c = threadIdx.x; c < j.channels; c += blockDim.x) {
    const double mean = j.acc[2 * c] / j.count;
    double var = j.acc[2 * c + 1] / j.count - mean * mean;
    if (var < 0) var = 0;
    j.stat[2 * c] = static_cast<float>(mean);
    j.stat[2 * c + 1] = static_cast<float>(1.0 / sqrt(var + double(kBnEps)));
    if (j.run_mean) {
      const double unbiased = j.count > 1 ? var * j.count / (j.count - 1) : var;
      j.run_mean[c] = (1.f - kBnMomentum) * j.run_mean[c] + kBnMomentum * static_cast<float>(mean);
      j.run_var[c] = (1.f - kBnMomentum) * j.run_var[c] + kBnMomentum * static_cast<float>(unbiased);
    }
  }
}

__device__ bool last_block_done(unsigned* counter, unsigned total) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(counter, 1u) == total - 1);
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// BatchNorm1d(T) on [rows = (b, t)][F]: channel = r % T.  grid = (chunks, T); block 256.  Rows of a multiple of four
// floats at 16-byte aligned addresses are read as float4 with 32-bit index arithmetic.
__global__ void __launch_bounds__(256)
bn_time_stats_kernel(const float* __restrict__ x, long long ld, long long batch, int F, int T, StatJob job) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  const int t = blockIdx.y;
  const long long per_t = batch * F;
  double s1 = 0, s2 = 0;
  if (F % 4 == 0 && ld % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && per_t < 0x7fffffffLL) {
    const unsigned f4 = static_cast<unsigned>(F) / 4, n4 = static_cast<unsigned>(per_t / 4);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
      const unsigned b = i / f4, c = (i - b * f4) * 4;
      const float4 v = __ldg(reinterpret_cast<const float4*>(x + (static_cast<long long>(b) * T + t) * ld + c));
      const float a1 = (v.x + v.y) + (v.z + v.w);
      const float a2 = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
      s1 += a1;
      s2 += a2;
    }
  } else {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < per_t;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
      const long long b = i / F;
      const int c = static_cast<int>(i - b * F);
      const float v = __ldg(x + (b * T + t) * ld + c);
      s1 += v;
      s2 += double(v) * v;
    }
  }
  __shared__ double r1[8], r2[8];
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int w = 0; w < 8; ++w) { a += r1[w]; b += r2[w]; }
    atomicAdd(job.acc + 2 * t, a);
    atomicAdd(job.acc + 2 * t + 1, b);
  }
  if (last_block_done(job.counter, gridDim.x * gridDim.y)) finalize_stats(job);
}

// normf normalises the same tensor as normv: re-derive the statistics and update ITS running buffers
__global__ void bn_running_only_kernel(StatJob job) { finalize_stats(job); }

// BatchNorm1d(K) on [batch][K]: channel = column.  grid = ceil(K / 8); block = 8 columns x 32 row groups (a warp reads
// four rows of 32 bytes: whole sectors), so that K = 527 spreads over 66 CTAs rather than 17.
constexpr int kColsPerCta = 8, kRowGroups = 32;
__global__ void __launch_bounds__(256)
bn_col_stats_kernel(const float* __restrict__ x, long long ld, long long batch, int K, StatJob job) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  const int tx = threadIdx.x % kColsPerCta, ty = threadIdx.x / kColsPerCta;
  const int c = blockIdx.x * kColsPerCta + tx;
  double s1 = 0, s2 = 0;
  if (c < K)
    for (long long b = ty; b < batch; b += kRowGroups) {
      const float v = __ldg(x + b * ld + c);
      s1 += v;
      s2 += double(v) * v;
    }
  __shared__ double r1[kRowGroups][kColsPerCta], r2[kRowGroups][kColsPerCta];
  r1[ty][tx] = s1;
  r2[ty][tx] = s2;
  __syncthreads();
  if (ty == 0 && c < K) {
    double a = 0, b = 0;
    for (int w = 0; w < kRowGroups; ++w) { a += r1[w][tx]; b += r2[w][tx]; }
    job.acc[2 * c] = a;
    job.acc[2 * c + 1] = b;
  }
  if (last_block_done(job.counter, gridDim.x)) finalize_stats(job);
}

// ------------------------------------------------------------------ dropout (counter-based, recomputed in backward)
using vmb::dropout_scale;   // igemm_sm100.cuh: shared with the gradient-statistics epilogue of the GEMM

// ------------------------------------------------------------------ 32x32 tile kernel with element functor
struct TileOut {
  __nv_bfloat16* planes;    // [rows_pad][3 * cols_pad] hi | mid | lo   (may be null)
  float* f32;               // [rows][ld_f32]                     (may be null)
  long long ld_f32;
  float* col_sum;           // [cols] += sum over rows (atomic)   (may be null)
  long long rows, rows_pad;
  int cols, cols_pad;
  // BatchNorm1d(T) batch statistics of the values this pass produces (channel = row % stats_T), accumulated from the
  // tile in shared memory and finalised by the last block like bn_time_stats_kernel does: stats_T > 0 switches it on
  StatJob stats = {};
  int stats_T = 0;
  __nv_bfloat16* planes_t = nullptr;   // [cols_pad][3 * rows_pad] hi | mid | lo: the weights' transposed planes
};

using vmb::split_bf16;

__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return __bfloat16_as_ushort(a) | (uint32_t(__bfloat16_as_ushort(b)) << 16);
}
// two adjacent elements of one row -> one 4-byte store per plane
__device__ __forceinline__ void store_split_pair(float v0, float v1, __nv_bfloat16* row, long long plane_stride) {
  __nv_bfloat16 h0, m0, l0, h1, m1, l1;
  split_bf16(v0, h0, m0, l0);
  split_bf16(v1, h1, m1, l1);
  *reinterpret_cast<uint32_t*>(row) = pack2(h0, h1);
  *reinterpret_cast<uint32_t*>(row + plane_stride) = pack2(m0, m1);
  *reinterpret_cast<uint32_t*>(row + 2 * plane_stride) = pack2(l0, l1);
}

// 64 x 64 tile per CTA.  A thread evaluates the functor on column PAIRS (row-major outputs: a warp writes 128 contiguous
// bytes per plane row) and, after the transpose through shared memory, writes row PAIRS of the transposed planes (again
// 128 bytes per warp and plane row).  The functor gets the row's time step t = r % T from the kernel: one 32-bit modulo
// per row instead of a 64-bit one per element.
constexpr int kTile = 64;
template <class F>
__device__ __forceinline__ void tile_body(F& f, const TileOut& o, int bx, int by) {
  __shared__ float tile[kTile][kTile + 1];
  f.prologue(bx == 0 && by == 0);
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int r0 = by * kTile;
  const int c0 = bx * kTile;
  const int tmod = f.time_steps();
  const bool need_tile = o.planes_t || o.col_sum || o.stats_T > 0;   // nothing else reads the shared-memory copy
  {
    const int c = c0 + 2 * tx;
#pragma unroll
    for (int i = 0; i < kTile / 8; ++i) {
      const int r = r0 + ty + 8 * i;
      float v0 = 0.f, v1 = 0.f;
      if (r < o.rows) {
        const int t = tmod > 1 ? r % tmod : 0;
        if (c < o.cols) v0 = f(r, t, c);
        if (c + 1 < o.cols) v1 = f(r, t, c + 1);
      }
      if (need_tile) {
        tile[ty + 8 * i][2 * tx] = v0;
        tile[ty + 8 * i][2 * tx + 1] = v1;
      }
      if (r < o.rows_pad && c < o.cols_pad) {
        if (o.planes)
          store_split_pair(v0, v1, o.planes + static_cast<long long>(r) * (static_cast<long long>(kPl) * o.cols_pad) + c,
                           o.cols_pad);
        if (o.f32 && r < o.rows) *reinterpret_cast<float2*>(o.f32 + static_cast<long long>(r) * o.ld_f32 + c) = make_float2(v0, v1);
      }
    }
  }
  if (!need_tile) return;
  __syncthreads();
  if (o.stats_T > 0) {
    // per-row sums in fp32 (64 terms; columns past `cols` hold zeros), per-time-step sums of the tile in double
    __shared__ double st_s[32];
    if (threadIdx.x < 32) st_s[threadIdx.x] = 0.0;
    __syncthreads();
    if (threadIdx.x < kTile && r0 + static_cast<int>(threadIdx.x) < o.rows) {
      float s1 = 0.f, s2 = 0.f;
#pragma unroll 8
      for (int j = 0; j < kTile; ++j) {
        const float v = tile[threadIdx.x][j];
        s1 += v;
        s2 = fmaf(v, v, s2);
      }
      const int t = (r0 + static_cast<int>(threadIdx.x)) % o.stats_T;
      atomicAdd(&st_s[2 * t], static_cast<double>(s1));
      atomicAdd(&st_s[2 * t + 1], static_cast<double>(s2));
    }
    __syncthreads();
    if (threadIdx.x < 2 * o.stats_T) atomicAdd(o.stats.acc + threadIdx.x, st_s[threadIdx.x]);
    if (last_block_done(o.stats.counter, gridDim.x * gridDim.y)) finalize_stats(o.stats);
  }
  if (o.planes_t) {
    const int r = r0 + 2 * tx;
#pragma unroll
    for (int i = 0; i < kTile / 8; ++i) {
      const int c = c0 + ty + 8 * i;
      if (c < o.cols_pad && r < o.rows_pad)
        store_split_pair(tile[2 * tx][ty + 8 * i], tile[2 * tx + 1][ty + 8 * i],
                         o.planes_t + static_cast<long long>(c) * (static_cast<long long>(kPl) * o.rows_pad) + r, o.rows_pad);
    }
  }
  if (o.col_sum && threadIdx.x < kTile && c0 + threadIdx.x < o.cols) {
    float s = 0.f;
#pragma unroll 8
    for (int j = 0; j < kTile; ++j) s += tile[j][threadIdx.x];
    atomicAdd(o.col_sum + c0 + threadIdx.x, s);
  }
}

template <class F>
__global__ void __launch_bounds__(256) tile_split_kernel(F f, TileOut o) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  tile_body(f, o, blockIdx.x, blockIdx.y);
}

// identity (weights, plain copies)
struct FIdentity {
  const float* x; long long ld;
  const float* bias_src = nullptr; float* bias_dst = nullptr; int n_bias = 0;   // block (0,0) copies the bias
  __device__ void prologue(bool first_block) {
    if (bias_dst && first_block)
      for (int i = threadIdx.x; i < n_bias; i += blockDim.x) bias_dst[i] = bias_src[i];
  }
  __device__ int time_steps() const { return 1; }
  __device__ float operator()(int r, int, int c) const { return __ldg(x + static_cast<long long>(r) * ld + c); }
};

// Every weight matrix of the head -> operand planes (row-major and transposed) + padded bias, in ONE launch: the jobs'
// tiles are laid end to end over blockIdx.x (nine launches of 20-100 CTAs each left most of the GPU idle).
constexpr int kMaxWeightJobs = 4 * (4 + 1) + 1;
struct WeightJobs {
  int n;
  int first_tile[kMaxWeightJobs + 1];
  int tiles_x[kMaxWeightJobs];
  FIdentity f[kMaxWeightJobs];
  TileOut o[kMaxWeightJobs];
};
__global__ void __launch_bounds__(256) weights_split_kernel(const __grid_constant__ WeightJobs jobs) {
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  int j = 0;
  while (j + 1 < jobs.n && static_cast<int>(blockIdx.x) >= jobs.first_tile[j + 1]) ++j;
  const int local = blockIdx.x - jobs.first_tile[j];
  FIdentity f = jobs.f[j];
  tile_body(f, jobs.o[j], local % jobs.tiles_x[j], local / jobs.tiles_x[j]);
}

// forward: a = dropout(relu?(gamma_t * (u - mu_t) * rstd_t + beta_t))
struct FBnAct {
  const float* u; long long ld; int T, F;
  const float* stat; const float* gamma; const float* beta;
  int relu; float p; const unsigned long long* seed; unsigned layer;   // *seed: the step's dropout seed (device memory)
  __device__ void prologue(bool) {}
  __device__ int time_steps() const { return T; }
  __device__ float operator()(int r, int t, int c) const {
    float v = fmaf(__ldg(gamma + t) * __ldg(stat + 2 * t + 1), __ldg(u + static_cast<long long>(r) * ld + c) - __ldg(stat + 2 * t),
                   __ldg(beta + t));
    if (relu) v = fmaxf(v, 0.f);
    return v * dropout_scale(p > 0.f ? __ldg(seed) : 0ull, layer, static_cast<unsigned long long>(r) * F + c, p);
  }
};

// upstream gradient of a BN(+ReLU+dropout) block: g = (da1 + da2) * dropout * [v > 0]
struct GradIn {
  const float* da1; long long ld1; const float* da2; long long ld2;   // da2 may be null
  const float* u; long long ldu; int T, F;
  const float* stat; const float* gamma; const float* beta;
  int relu; float p; const unsigned long long* seed; unsigned layer;
  __device__ __forceinline__ float xhat(long long r, int t, int c) const {
    return (__ldg(u + r * ldu + c) - __ldg(stat + 2 * t)) * __ldg(stat + 2 * t + 1);
  }
  __device__ __forceinline__ float g(long long r, int t, int c, float xh) const {
    float d = __ldg(da1 + r * ld1 + c);
    if (da2) d += __ldg(da2 + r * ld2 + c);
    if (relu && fmaf(__ldg(gamma + t), xh, __ldg(beta + t)) <= 0.f) return 0.f;
    return d * dropout_scale(p > 0.f ? __ldg(seed) : 0ull, layer, static_cast<unsigned long long>(r) * F + c, p);
  }
};

// phase A of BN backward: S1_t = sum g, S2_t = sum g * xhat  (double atomics), grid = (chunks, T)
__global__ void __launch_bounds__(256)
bn_time_backward_reduce_kernel(GradIn in, long long batch, double* __restrict__ acc) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  const int t = blockIdx.y;
  const long long per_t = batch * in.F;
  double s1 = 0, s2 = 0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < per_t;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / in.F;
    const int c = static_cast<int>(i - b * in.F);
    const long long r = b * in.T + t;
    const float xh = in.xhat(r, t, c);
    const float g = in.g(r, t, c, xh);
    s1 += g;
    s2 += double(g) * xh;
  }
  __shared__ double r1[8], r2[8];
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int w = 0; w < 8; ++w) { a += r1[w]; b += r2[w]; }
    atomicAdd(acc + 2 * t, a);
    atomicAdd(acc + 2 * t + 1, b);
  }
}

// phase B: du = gamma_t * rstd_t * (g - S1_t / n - xhat * S2_t / n); block (0,0) also writes dgamma = S2, dbeta = S1
struct FBnBackward {
  GradIn in; const double* acc; double n; float* dgamma; float* dbeta;
  float* coef;   // shared memory [T][3]: gamma * rstd, S1 / n, S2 / n   (set by prologue)
  __device__ void prologue(bool first_block) {
    __shared__ float coef_s[16 * 3];
    coef = coef_s;
    if (threadIdx.x < in.T) {
      const int t = threadIdx.x;
      coef_s[3 * t] = in.gamma[t] * in.stat[2 * t + 1];
      coef_s[3 * t + 1] = static_cast<float>(acc[2 * t] / n);
      coef_s[3 * t + 2] = static_cast<float>(acc[2 * t + 1] / n);
      if (first_block) {
        dbeta[t] = static_cast<float>(acc[2 * t]);
        dgamma[t] = static_cast<float>(acc[2 * t + 1]);
      }
    }
    __syncthreads();
  }
  __device__ int time_steps() const { return in.T; }
  __device__ float operator()(int r, int t, int c) const {
    const float xh = in.xhat(r, t, c);
    const float g = in.g(r, t, c, xh);
    return coef[3 * t] * (g - coef[3 * t + 1] - xh * coef[3 * t + 2]);
  }
};

// ------------------------------------------------------------------ wide first layer (emb_in wider than the hidden width)
// The level-0 norm0 output y = gamma_t xhat + beta_t never exists: the first Linear reads the planes of xhat, and a tile
// pass applies the affine to its output (FAffine: U = gamma_t P + beta_t s + b with P = xhat W^T and
// s[o] = sum_f W[o][f]).  In the backward pass, with G = dL/dU of block (0, 0):
//   dbeta_t  = sum_{r in t} G[r,:] . s          dgamma_t = sum_{r in t} G[r,:] . P[r,:]
//   dW[o][f] = sum_r (gamma_t G[r][o]) xhat[r][f] + c[o],   c[o] = sum_t beta_t sum_{r in t} G[r][o]
// so no GEMM over the input width runs but the forward one and dW, and nothing divides by gamma.  Both contract in
// slices of at most vmb::kFwdSlice (forward: input columns) / vmb::kDwSlice (dW: rows) per tcgen05 accumulator.

// xhat = (x - mean_t) rstd_t (the same expression GradIn::xhat evaluates)
struct FNormalize {
  const float* u; long long ld; int T;
  const float* stat;
  __device__ void prologue(bool) {}
  __device__ int time_steps() const { return T; }
  __device__ float operator()(int r, int t, int c) const {
    return (__ldg(u + static_cast<long long>(r) * ld + c) - __ldg(stat + 2 * t)) * __ldg(stat + 2 * t + 1);
  }
};

// U = gamma_t P + (beta_t s[c] + b[c]) from P = xhat W^T
struct FAffine {
  const float* p; long long ld; int T;
  const float *gamma, *beta, *s, *bias;
  __device__ void prologue(bool) {}
  __device__ int time_steps() const { return T; }
  __device__ float operator()(int r, int t, int c) const {
    return fmaf(__ldg(gamma + t), __ldg(p + static_cast<long long>(r) * ld + c), fmaf(__ldg(beta + t), __ldg(s + c), __ldg(bias + c)));
  }
};

// s[o] = sum_f W[o][f] in double, one CTA per row
__global__ void __launch_bounds__(256) row_sum_kernel(const float* __restrict__ w, int n_in, float* __restrict__ s) {
  const float* row = w + static_cast<long long>(blockIdx.x) * n_in;
  double acc = 0;
  for (int f = threadIdx.x; f < n_in; f += blockDim.x) acc += __ldg(row + f);
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ double red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0;
    for (int i = 0; i < 8; ++i) a += red[i];
    s[blockIdx.x] = static_cast<float>(a);
  }
}

struct WideGradOut {
  __nv_bfloat16* planes;      // [rows_pad][3 * cols_pad]: gamma_t G (the dW GEMM's A operand)
  long long rows, rows_pad;
  int cols, cols_pad;
  const float* gamma0;        // norm0 weight [T]
  const float* P; long long ldp;   // xhat W^T [rows][ldp] from the forward GEMM
  const float* wsum;          // s [cols_pad]
  float* col_sum;             // d(bias) [cols] += sum over rows of G
  float* col_sum_t;           // [T][cols_pad] += sum over the rows of time step t of G (zeroed by the caller)
  double* acc0;               // norm0's backward slot [T][2] += {G . s, G . P}
};

// Block (0, 0)'s BatchNorm backward (FBnBackward, G = dL/dU) on 64 x 64 tiles, as tile_body runs it, writing what the
// wide first layer needs instead of G's planes: see the identities above.
__global__ void __launch_bounds__(256) wide_grad_tile_kernel(FBnBackward f, WideGradOut o) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  __shared__ float tile[kTile][kTile + 1];
  __shared__ double dots[16][2];
  f.prologue(blockIdx.x == 0 && blockIdx.y == 0);
  if (threadIdx.x < 32) dots[threadIdx.x >> 1][threadIdx.x & 1] = 0.0;
  __syncthreads();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int r0 = blockIdx.y * kTile, c0 = blockIdx.x * kTile;
  const int T = f.time_steps();
  const int c = c0 + 2 * tx;
  const float s0 = c < o.cols_pad ? __ldg(o.wsum + c) : 0.f, s1 = c + 1 < o.cols_pad ? __ldg(o.wsum + c + 1) : 0.f;
#pragma unroll
  for (int i = 0; i < kTile / 8; ++i) {
    const int r = r0 + ty + 8 * i;   // one row per warp: the row's dot products are warp sums
    float v0 = 0.f, v1 = 0.f, gs = 0.f, gp = 0.f, gam = 0.f;
    int t = 0;
    if (r < o.rows) {
      t = T > 1 ? r % T : 0;
      gam = __ldg(o.gamma0 + t);
      const float* prow = o.P + static_cast<long long>(r) * o.ldp;
      if (c < o.cols) { v0 = f(r, t, c); gs = v0 * s0; gp = v0 * __ldg(prow + c); }
      if (c + 1 < o.cols) { v1 = f(r, t, c + 1); gs = fmaf(v1, s1, gs); gp = fmaf(v1, __ldg(prow + c + 1), gp); }
    }
    tile[ty + 8 * i][2 * tx] = v0;
    tile[ty + 8 * i][2 * tx + 1] = v1;
    if (r < o.rows_pad && c < o.cols_pad)
      store_split_pair(gam * v0, gam * v1, o.planes + static_cast<long long>(r) * (static_cast<long long>(kPl) * o.cols_pad) + c,
                       o.cols_pad);
#pragma unroll
    for (int off = 16; off; off >>= 1) {
      gs += __shfl_xor_sync(0xffffffffu, gs, off);
      gp += __shfl_xor_sync(0xffffffffu, gp, off);
    }
    if (tx == 0 && r < o.rows) {
      atomicAdd(&dots[t][0], static_cast<double>(gs));
      atomicAdd(&dots[t][1], static_cast<double>(gp));
    }
  }
  __syncthreads();
  if (threadIdx.x < kTile && c0 + static_cast<int>(threadIdx.x) < o.cols) {
    const int cc = c0 + threadIdx.x;
    float s = 0.f;
#pragma unroll 8
    for (int j = 0; j < kTile; ++j) s += tile[j][threadIdx.x];
    atomicAdd(o.col_sum + cc, s);
    for (int t = 0; t < T; ++t) {   // rows past `rows` hold zeros
      float st = 0.f;
      for (int j = (t - r0 % T + T) % T; j < kTile; j += T) st += tile[j][threadIdx.x];
      atomicAdd(o.col_sum_t + static_cast<long long>(t) * o.cols_pad + cc, st);
    }
  }
  if (threadIdx.x < 2 * T) atomicAdd(o.acc0 + threadIdx.x, dots[threadIdx.x >> 1][threadIdx.x & 1]);
}

// grads dW [n_out][n_in] = the GEMM's sum_r (gamma_t G) xhat [n_out][ldw] + c[o]; grid = (column chunks, n_out)
__global__ void __launch_bounds__(256)
wide_dw_finish_kernel(const float* __restrict__ dw, long long ldw, float* __restrict__ dst, int n_in,
                      const float* __restrict__ col_sum_t, int ldc, const float* __restrict__ beta0, int T) {
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  const int o = blockIdx.y;
  __shared__ float c_o;
  if (threadIdx.x == 0) {
    double c = 0;
    for (int t = 0; t < T; ++t) c += double(__ldg(beta0 + t)) * __ldg(col_sum_t + static_cast<long long>(t) * ldc + o);
    c_o = static_cast<float>(c);
  }
  __syncthreads();
  const float* src = dw + static_cast<long long>(o) * ldw;
  float* out = dst + static_cast<long long>(o) * n_in;
  for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < n_in; f += gridDim.x * blockDim.x) out[f] = src[f] + c_o;
}

// ------------------------------------------------------------------ attention (one CTA per clip)
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct AttParams {
  const float* z; long long ldz; int K, T;
  const float* stat;                       // [T][2] batch statistics of z (shared by both branches)
  const float *gv, *bv, *gf, *bf;          // normv / normf affine parameters [T]
};

// y[clip][col0 + k] = sum_t cla * att / sum_t att; row_stats[r] = {max, sum} of the class softmax of row r.
// The same values also go out as the operand planes of the output Linear, yp [rows_pad][3 * yp_cols]; the grid covers
// the padded rows, which are written as zeros.
__global__ void __launch_bounds__(256)
att_forward_kernel(AttParams a, float* __restrict__ y, long long ystride, int col0, float* __restrict__ row_stats,
                   __nv_bfloat16* __restrict__ yp, int yp_cols, long long batch) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  __shared__ float rmax[16], rsum[16], sa_v[16], sb_v[16], sa_f[16], sb_f[16];
  const long long clip = blockIdx.x;
  if (clip >= batch) {   // padding row of the planes
    __nv_bfloat16* row = yp + clip * (static_cast<long long>(kPl) * yp_cols) + col0;
    for (int k = threadIdx.x; k < a.K; k += blockDim.x)
      for (int pl = 0; pl < kPl; ++pl) row[pl * yp_cols + k] = __float2bfloat16_rn(0.f);
    return;
  }
  const float* zc = a.z + clip * a.T * a.ldz;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < a.T) {
    const int t = threadIdx.x;
    const float mu = a.stat[2 * t], rs = a.stat[2 * t + 1];
    sa_v[t] = a.gv[t] * rs; sb_v[t] = a.bv[t] - a.gv[t] * rs * mu;
    sa_f[t] = a.gf[t] * rs; sb_f[t] = a.bf[t] - a.gf[t] * rs * mu;
  }
  __syncthreads();
  for (int t = warp; t < a.T; t += 8) {
    float m = -INFINITY;
    for (int c = lane; c < a.K; c += 32) m = fmaxf(m, fmaf(sa_v[t], __ldg(zc + t * a.ldz + c), sb_v[t]));
    m = warp_max(m);
    float s = 0.f;
    for (int c = lane; c < a.K; c += 32) s += expf(fmaf(sa_v[t], __ldg(zc + t * a.ldz + c), sb_v[t]) - m);
    s = warp_sum(s);
    if (lane == 0) {
      rmax[t] = m; rsum[t] = s;
      row_stats[2 * (clip * a.T + t)] = m;
      row_stats[2 * (clip * a.T + t) + 1] = s;
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < a.K; k += blockDim.x) {
    float num = 0.f, den = 0.f;
    for (int t = 0; t < a.T; ++t) {
      const float zz = __ldg(zc + t * a.ldz + k);
      const float att = expf(fmaf(sa_v[t], zz, sb_v[t]) - rmax[t]) / rsum[t];
      const float cla = 1.f / (1.f + expf(-fmaf(sa_f[t], zz, sb_f[t])));
      num = fmaf(cla, att, num);
      den += att;
    }
    const float val = num / den;
    y[clip * ystride + col0 + k] = val;
    __nv_bfloat16 hi, mid, lo;
    split_bf16(val, hi, mid, lo);
    __nv_bfloat16* row = yp + clip * (static_cast<long long>(kPl) * yp_cols) + col0 + k;
    row[0] = hi;
    row[yp_cols] = mid;
    row[2 * yp_cols] = lo;
  }
}

// Backward of the pooling for one clip: writes gv = d(BN^v output), gf = d(BN^f output) as fp32 [rows][ldg] and adds
// the four BatchNorm reductions (sum g, sum g * zhat for both branches) to acc_v / acc_f.  att and cla of the clip
// (T x K each) are computed once into shared memory.
__global__ void __launch_bounds__(256)
att_backward_kernel(AttParams a, const float* __restrict__ y, const float* __restrict__ dy, long long ystride, int col0,
                    const float* __restrict__ row_stats, float* __restrict__ gv, float* __restrict__ gf, long long ldg,
                    double* __restrict__ acc_v, double* __restrict__ acc_f) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  extern __shared__ float att_sm[];
  float* att = att_sm;                 // [T][K]
  float* cla = att + a.T * a.K;        // [T][K]
  __shared__ float sa_v[16], sb_v[16], sa_f[16], sb_f[16], dot[16];
  __shared__ double red[8][16][4];
  const long long clip = blockIdx.x;
  const float* zc = a.z + clip * a.T * a.ldz;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < a.T) {
    const int t = threadIdx.x;
    const float mu = a.stat[2 * t], rs = a.stat[2 * t + 1];
    sa_v[t] = a.gv[t] * rs; sb_v[t] = a.bv[t] - a.gv[t] * rs * mu;
    sa_f[t] = a.gf[t] * rs; sb_f[t] = a.bf[t] - a.gf[t] * rs * mu;
    dot[t] = 0.f;
  }
  __syncthreads();
  // att / cla of the clip into shared memory, one time step at a time (no index division, the row's softmax statistics
  // read once per row)
  for (int t = 0; t < a.T; ++t) {
    const float* rs2 = row_stats + 2 * (clip * a.T + t);
    const float m = __ldg(rs2), inv = 1.f / __ldg(rs2 + 1);
    const float av = sa_v[t], bv = sb_v[t], af = sa_f[t], bf = sb_f[t];
    const float* zt = zc + t * a.ldz;
    for (int k = threadIdx.x; k < a.K; k += blockDim.x) {
      const float zz = __ldg(zt + k);
      att[t * a.K + k] = expf(fmaf(av, zz, bv) - m) * inv;
      cla[t * a.K + k] = 1.f / (1.f + expf(-fmaf(af, zz, bf)));
    }
  }
  __syncthreads();
  // A thread owns the classes k = threadIdx.x + 256 i, i < kIter (K <= 1024): what depends on k alone — 1 / sum_t att,
  // y and dy — stays in registers for both passes.
  // s[k] = sum_t att; datt = dy (cla - y) / s; dot[t] = sum_k datt * att  (the softmax backward needs it per row)
  constexpr int kIter = 4;
  float si_r[kIter], yy_r[kIter], d_r[kIter];
  float pdot[16];
#pragma unroll
  for (int t = 0; t < 16; ++t) pdot[t] = 0.f;
#pragma unroll
  for (int i = 0; i < kIter; ++i) {
    const int k = threadIdx.x + 256 * i;
    si_r[i] = yy_r[i] = d_r[i] = 0.f;
    if (k < a.K) {
      float s = 0.f;
      for (int t = 0; t < a.T; ++t) s += att[t * a.K + k];
      si_r[i] = 1.f / s;
      yy_r[i] = __ldg(y + clip * ystride + col0 + k);
      d_r[i] = __ldg(dy + clip * ystride + col0 + k);
      const float dsi = d_r[i] * si_r[i];
#pragma unroll
      for (int t = 0; t < 16; ++t)
        if (t < a.T) pdot[t] = fmaf(dsi * (cla[t * a.K + k] - yy_r[i]), att[t * a.K + k], pdot[t]);
    }
  }
#pragma unroll
  for (int t = 0; t < 16; ++t) {
    float v = pdot[t];
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && t < a.T) atomicAdd(&dot[t], v);
  }
  __syncthreads();
  // second pass, one time step per iteration so the BatchNorm reductions stay per t (no barrier inside the loop); a
  // thread adds its <= 4 terms in fp32, everything above that in double
  for (int t = 0; t < a.T; ++t) {
    const float mu = a.stat[2 * t], rstd = a.stat[2 * t + 1], dt = dot[t];
    float* gvr = gv + (clip * a.T + t) * ldg;
    float* gfr = gf + (clip * a.T + t) * ldg;
    const float* zt = zc + t * a.ldz;
    float q1v = 0.f, q2v = 0.f, q1f = 0.f, q2f = 0.f;
#pragma unroll
    for (int i = 0; i < kIter; ++i) {
      const int k = threadIdx.x + 256 * i;
      if (k < a.K) {
        const float at = att[t * a.K + k], cl = cla[t * a.K + k];
        const float dsi = d_r[i] * si_r[i];
        const float g_f = dsi * at * cl * (1.f - cl);
        const float g_v = at * (dsi * (cl - yy_r[i]) - dt);
        gvr[k] = g_v;
        gfr[k] = g_f;
        const float zh = (__ldg(zt + k) - mu) * rstd;
        q1v += g_v; q2v = fmaf(g_v, zh, q2v);
        q1f += g_f; q2f = fmaf(g_f, zh, q2f);
      }
    }
    double p1v = q1v, p2v = q2v, p1f = q1f, p2f = q2f;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      p1v += __shfl_xor_sync(0xffffffffu, p1v, o);
      p2v += __shfl_xor_sync(0xffffffffu, p2v, o);
      p1f += __shfl_xor_sync(0xffffffffu, p1f, o);
      p2f += __shfl_xor_sync(0xffffffffu, p2f, o);
    }
    if (lane == 0) { red[warp][t][0] = p1v; red[warp][t][1] = p2v; red[warp][t][2] = p1f; red[warp][t][3] = p2f; }
  }
  // one cross-warp reduction for all time steps: thread (t, j) adds the eight warps' partial sums of quantity j
  __syncthreads();
  if (threadIdx.x < 4 * a.T) {
    const int t = threadIdx.x >> 2, j = threadIdx.x & 3;
    double sum = 0;
    for (int w = 0; w < 8; ++w) sum += red[w][t][j];
    atomicAdd((j < 2 ? acc_v : acc_f) + 2 * t + (j & 1), sum);
  }
}

// dz = gamma^v rstd (gv - S1v/n - zhat S2v/n) + gamma^f rstd (gf - S1f/n - zhat S2f/n); block (0,0) writes the four
// affine-parameter gradients
struct FAttCombine {
  AttParams a; const float* gv; const float* gf; long long ldg;
  const double* acc_v; const double* acc_f; double n;
  float *dgv, *dbv, *dgf, *dbf;
  float* coef;   // shared memory [T][8]: mu, rstd, gamma^v rstd, S1v / n, S2v / n, gamma^f rstd, S1f / n, S2f / n
  __device__ void prologue(bool first_block) {
    __shared__ float coef_s[16 * 8];
    coef = coef_s;
    if (threadIdx.x < a.T) {
      const int t = threadIdx.x;
      const float rstd = a.stat[2 * t + 1];
      coef_s[8 * t] = a.stat[2 * t];
      coef_s[8 * t + 1] = rstd;
      coef_s[8 * t + 2] = a.gv[t] * rstd;
      coef_s[8 * t + 3] = float(acc_v[2 * t] / n);
      coef_s[8 * t + 4] = float(acc_v[2 * t + 1] / n);
      coef_s[8 * t + 5] = a.gf[t] * rstd;
      coef_s[8 * t + 6] = float(acc_f[2 * t] / n);
      coef_s[8 * t + 7] = float(acc_f[2 * t + 1] / n);
      if (first_block) {
        dbv[t] = static_cast<float>(acc_v[2 * t]); dgv[t] = static_cast<float>(acc_v[2 * t + 1]);
        dbf[t] = static_cast<float>(acc_f[2 * t]); dgf[t] = static_cast<float>(acc_f[2 * t + 1]);
      }
    }
    __syncthreads();
  }
  __device__ int time_steps() const { return a.T; }
  __device__ float operator()(int r, int t, int c) const {
    const float* k = coef + 8 * t;
    const float zh = (__ldg(a.z + static_cast<long long>(r) * a.ldz + c) - k[0]) * k[1];
    const float v = k[2] * (__ldg(gv + static_cast<long long>(r) * ldg + c) - k[3] - zh * k[4]);
    const float f = k[5] * (__ldg(gf + static_cast<long long>(r) * ldg + c) - k[6] - zh * k[7]);
    return v + f;
  }
};

// ------------------------------------------------------------------ output layer: BN_K + sigmoid + cross-entropy
// one block per batch row: out = sigmoid(BN_K(o)); lse[b] = log sum_k exp(out); loss += (lse - out[label]) / B
__global__ void __launch_bounds__(256)
out_loss_rows_kernel(const float* __restrict__ o, long long ldo, int K, const float* __restrict__ stat,
                     const float* __restrict__ gamma, const float* __restrict__ beta, const long long* __restrict__ labels,
                     long long batch, float* __restrict__ scores, float* __restrict__ lse, float* __restrict__ loss) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  const long long b = blockIdx.x;
  __shared__ float red[8];
  __shared__ float s_lab;
  if (threadIdx.x == 0) s_lab = 0.f;
  __syncthreads();
  const long long lab = labels ? labels[b] : -1;
  float m = 0.f, picked = 0.f;  // outputs are in (0, 1): exp() cannot overflow, no max shift needed
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const float p = fmaf(gamma[k] * stat[2 * k + 1], o[b * ldo + k] - stat[2 * k], beta[k]);
    const float s = 1.f / (1.f + expf(-p));
    if (scores) scores[b * K + k] = s;
    m += expf(s);
    if (k == lab) picked = s;
  }
  m = warp_sum(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  if (lab >= 0 && lab < K && threadIdx.x == lab % blockDim.x) s_lab = picked;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < 8; ++w) tot += red[w];
    const float l = logf(tot);
    lse[b] = l;
    if (labels) atomicAdd(loss, (l - s_lab) / static_cast<float>(batch));
  }
}

// dp[b][k] = dout * out (1 - out) with dout = (exp(out - lse_b) - [k == label_b]) / B (cross-entropy on the sigmoid
// outputs) or an externally supplied d(loss)/d(scores); BN_K backward over the batch per class:
// do = gamma rstd (dp - mean_b dp - xhat mean_b(dp xhat)).  grid = ceil(K/8), block = 8 columns x 32 row groups (see
// bn_col_stats_kernel); a thread keeps dp and xhat of its first kKeep rows in registers between the two passes.
__global__ void __launch_bounds__(256)
out_bn_backward_kernel(const float* __restrict__ o, long long ldo, int K, const float* __restrict__ stat,
                       const float* __restrict__ gamma, const float* __restrict__ beta,
                       const long long* __restrict__ labels, const float* __restrict__ lse,
                       const float* __restrict__ dscores, long long batch, float* __restrict__ d_o, long long ldd, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  vmb::pdl_launch_dependents();   // programmatic dependent launch: see sm100_ptx.cuh
  vmb::pdl_wait();
  constexpr int kKeep = 16;       // batch <= 512 rows: everything stays in registers
  const int tx = threadIdx.x % kColsPerCta, ty = threadIdx.x / kColsPerCta;
  const int k = blockIdx.x * kColsPerCta + tx;
  __shared__ double r1[kRowGroups][kColsPerCta], r2[kRowGroups][kColsPerCta];
  __shared__ float m1[kColsPerCta], m2[kColsPerCta];
  const bool ok = k < K;
  const float mu = ok ? stat[2 * k] : 0.f, rstd = ok ? stat[2 * k + 1] : 0.f, g = ok ? gamma[k] : 0.f,
              be = ok ? beta[k] : 0.f;
  auto dp_of = [&](long long b, float& xh) {
    xh = (o[b * ldo + k] - mu) * rstd;
    const float s = 1.f / (1.f + expf(-fmaf(g, xh, be)));
    const float dout = dscores ? dscores[b * K + k]
                               : (expf(s - lse[b]) - (labels[b] == k ? 1.f : 0.f)) / static_cast<float>(batch);
    return dout * s * (1.f - s);
  };
  float keep_dp[kKeep], keep_xh[kKeep];
  double s1 = 0, s2 = 0;
  if (ok) {
#pragma unroll
    for (int i = 0; i < kKeep; ++i) {
      const long long b = ty + static_cast<long long>(i) * kRowGroups;
      keep_dp[i] = 0.f;
      keep_xh[i] = 0.f;
      if (b < batch) {
        keep_dp[i] = dp_of(b, keep_xh[i]);
        s1 += keep_dp[i];
        s2 += double(keep_dp[i]) * keep_xh[i];
      }
    }
    for (long long b = ty + static_cast<long long>(kKeep) * kRowGroups; b < batch; b += kRowGroups) {
      float xh;
      const float dp = dp_of(b, xh);
      s1 += dp;
      s2 += double(dp) * xh;
    }
  }
  r1[ty][tx] = s1;
  r2[ty][tx] = s2;
  __syncthreads();
  if (ty == 0) {
    double a = 0, b = 0;
    for (int w = 0; w < kRowGroups; ++w) { a += r1[w][tx]; b += r2[w][tx]; }
    m1[tx] = static_cast<float>(a / double(batch));
    m2[tx] = static_cast<float>(b / double(batch));
    if (ok) { dbeta[k] = static_cast<float>(a); dgamma[k] = static_cast<float>(b); }
  }
  __syncthreads();
  if (ok) {
#pragma unroll
    for (int i = 0; i < kKeep; ++i) {
      const long long b = ty + static_cast<long long>(i) * kRowGroups;
      if (b < batch) d_o[b * ldd + k] = g * rstd * (keep_dp[i] - m1[tx] - keep_xh[i] * m2[tx]);
    }
    for (long long b = ty + static_cast<long long>(kKeep) * kRowGroups; b < batch; b += kRowGroups) {
      float xh;
      const float dp = dp_of(b, xh);
      d_o[b * ldd + k] = g * rstd * (dp - m1[tx] - xh * m2[tx]);
    }
  }
}

__global__ void set_seed_kernel(unsigned long long* dst, unsigned long long seed) { *dst = seed; }

// ------------------------------------------------------------------ Adam (torch.optim.Adam, amsgrad = False)
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
            float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt, float gscale) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float gr = g[i] * gscale;
    if (wd != 0.f) gr = fmaf(wd, p[i], gr);
    const float mi = fmaf(b1, m[i], (1.f - b1) * gr);       // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = fmaf(b2, v[i], (1.f - b2) * gr * gr);  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ trainer handle
// offsets into params (gamma, beta) / running (mean; var = mean + n); statistic slots for the forward batch statistics
// and for the backward reductions
struct BnRef { long long g, b, rm; int n; int slot, bslot; };
struct FcRef {
  long long w, b; int n_out, n_in, n_out_pad, n_in_pad;
  float* bias_pad;      // [n_out_pad] zero-padded copy of the bias (the GEMM epilogue reads whole tiles)
  __nv_bfloat16* wp;    // [n_out_pad][2 n_in_pad]
  __nv_bfloat16* wtp;   // [n_in_pad][2 n_out_pad]
};
struct LevelRef { BnRef norm0; int n_fc; FcRef fc[kMaxFc]; BnRef norms[kMaxFc]; FcRef fcv; BnRef normv, normf; };

struct vmb_mla_trainer {
  int n_levels, emb_in, H, K, T;
  long long max_batch;
  LevelRef lvl[kMaxLevels];
  FcRef fc_out;
  BnRef norm_out;
  long long n_params = 0, n_running = 0;
  int n_slots = 0;          // statistic slots; slot s: acc at s*kSlot doubles, stat at s*kSlot floats
  char* ws = nullptr;       // single workspace allocation
  size_t ws_bytes = 0;
  // the weight-gradient GEMMs (dW = dU^T A) feed nothing but `grads`: they run on a side stream, next to the dX chain
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_dw = nullptr, ev_att = nullptr, ev_w = nullptr;
  // recorded in the backward pass where every gradient from `tail_offset` on is final (all but level 0's embedding chain):
  // a data-parallel caller starts the all-reduce of that part of the bucket while the rest of the backward pass runs
  cudaEvent_t ev_tail = nullptr;
  long long tail_offset = 0;
  // backward: the attention branches of every level but the last need only dY and forward state, so they run on a second
  // side stream (with their own scratch: G_p2 .. dWtmp2, one dAtt per level) while the last level's chain runs
  cudaStream_t side2 = nullptr;
  cudaEvent_t ev_attb[kMaxLevels] = {};
  __nv_bfloat16* G_p2 = nullptr;
  float *GV2 = nullptr, *GF2 = nullptr, *dWtmp2 = nullptr;
  float* dAtt[kMaxLevels] = {};
  // carved pointers
  double* acc = nullptr; size_t acc_bytes = 0;      // zeroed every step (together with the counters)
  unsigned* counters = nullptr;
  float* stat = nullptr;
  __nv_bfloat16* xin_p = nullptr;                  // level-0 norm0 output planes [Rp][3 inpad]
  float* U[kMaxLevels][kMaxFc] = {};               // pre-BN Linear outputs [R][Hp]
  __nv_bfloat16* A_p[kMaxLevels][kMaxFc] = {};     // post-activation planes (input of the next Linear / fcv)
  float* E[kMaxLevels] = {};                       // fp32 embeddings of each level (input of the next level's norm0)
  __nv_bfloat16* N_p[kMaxLevels] = {};             // norm0 output planes of levels >= 1
  float* Z[kMaxLevels] = {};                       // fcv outputs
  float* row_stats[kMaxLevels] = {};
  float *Y = nullptr, *dY = nullptr;               // [B][ycols]
  __nv_bfloat16* Y_p = nullptr;
  float *O = nullptr, *dO = nullptr, *lse = nullptr;
  __nv_bfloat16* G_p = nullptr;                    // gradient planes (reused)
  float *GV = nullptr, *GF = nullptr;              // attention branch gradients / general fp32 scratch [R][Hp]
  float *dA = nullptr, *dB = nullptr, *dEnext = nullptr;  // fp32 gradient buffers [R][Hp]
  float* dWtmp = nullptr;                          // padded dW GEMM output
  int Hp, inpad, ycols, ycols_pad;
  // wide first layer (inpad > Hp): xin_p holds the planes of xhat, not of the norm0 output (see FNormalize)
  bool wide = false;
  float* P0 = nullptr;                             // xhat W^T of the first Linear [R][Hp]
  float* wsum = nullptr;                           // s[o] = sum_f W[o][f] [Hp]
  float* gsum_t = nullptr;                         // per-time-step column sums of block (0, 0)'s G [T][Hp]
  // The dropout seed of the step lives in device memory, so that a captured step can be replayed with a new seed.
  unsigned long long* seed_dev = nullptr;
  // CUDA graph of the whole step (vmb_mla_train_step): ~110 kernel launches, memsets and stream fork / join events cost
  // the host about as long as the GPU needs to run them; a replayed graph is one launch.  The inputs are copied into
  // staging buffers first, so the graph does not depend on the caller's x / labels addresses; one graph per distinct
  // (params, running, grads, loss, scores, batch, dropout_p) — the peer-memory step alternates two gradient buffers.
  float* x_stage = nullptr;
  long long* labels_stage = nullptr;
  cudaStream_t gstream = nullptr;     // the graph runs here (stream capture is not allowed on the legacy default stream)
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  struct GraphSlot {
    const void *params, *running, *grads, *loss, *scores;
    long long batch;
    float dropout_p;
    cudaGraphExec_t exec;
    int launches;                     // kernels in the graph (for vmb_launch_count)
  } graphs[4] = {};
  int n_graphs = 0, next_graph = 0;
  int eager_steps = 0;                // the first step of a handle runs eagerly: one-time set-up must not be captured
  bool graph_broken = false;          // capture or instantiation failed once: stay on the eager path
  bool capturing = false;
};

namespace {
constexpr int kSlot = 1024;  // channels per statistic slot (>= max(T, K padded))

struct Carver {
  char* base; size_t off = 0;
  template <class T> T* take(size_t n) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += up(n * sizeof(T));
    return p;
  }
};

void carve(vmb_mla_trainer* h, char* base) {
  Carver c{base};
  const long long B = h->max_batch, R = B * h->T, Rp = pad64(R), Bp = pad64(B);
  const int Hp = h->Hp, inpad = h->inpad;
  h->acc = c.take<double>(size_t(h->n_slots) * kSlot * 2);
  h->counters = c.take<unsigned>(size_t(h->n_slots));
  h->acc_bytes = c.off;
  h->stat = c.take<float>(size_t(h->n_slots) * kSlot * 2);
  h->xin_p = c.take<__nv_bfloat16>(size_t(Rp) * kPl * inpad);
  if (h->wide) {
    h->P0 = c.take<float>(size_t(R) * Hp);
    h->wsum = c.take<float>(size_t(Hp));
    h->gsum_t = c.take<float>(size_t(h->T) * Hp);
  }
  for (int l = 0; l < h->n_levels; ++l) {
    for (int j = 0; j < h->lvl[l].n_fc; ++j) {
      h->U[l][j] = c.take<float>(size_t(R) * Hp);
      h->A_p[l][j] = c.take<__nv_bfloat16>(size_t(Rp) * kPl * Hp);
    }
    h->E[l] = c.take<float>(size_t(R) * Hp);
    if (l > 0) h->N_p[l] = c.take<__nv_bfloat16>(size_t(Rp) * kPl * Hp);
    h->Z[l] = c.take<float>(size_t(R) * Hp);
    h->row_stats[l] = c.take<float>(size_t(R) * 2);
  }
  h->Y = c.take<float>(size_t(B) * h->ycols_pad);
  h->dY = c.take<float>(size_t(B) * h->ycols_pad);
  h->Y_p = c.take<__nv_bfloat16>(size_t(Bp) * kPl * h->ycols_pad);
  h->O = c.take<float>(size_t(B) * Hp);
  h->dO = c.take<float>(size_t(B) * Hp);
  h->lse = c.take<float>(size_t(B));
  h->G_p = c.take<__nv_bfloat16>(size_t(Rp) * kPl * Hp);
  h->GV = c.take<float>(size_t(R) * Hp);
  h->GF = c.take<float>(size_t(R) * Hp);
  h->dA = c.take<float>(size_t(R) * Hp);
  h->dB = c.take<float>(size_t(R) * Hp);
  h->dEnext = c.take<float>(size_t(R) * Hp);
  h->seed_dev = c.take<unsigned long long>(2);
  h->x_stage = c.take<float>(size_t(R) * h->emb_in);
  h->labels_stage = c.take<long long>(size_t(B));
  const int widest = std::max(h->ycols_pad, std::max(Hp, inpad));
  h->dWtmp = c.take<float>(size_t(Hp) * widest);
  if (h->n_levels > 1) {
    h->G_p2 = c.take<__nv_bfloat16>(size_t(Rp) * kPl * Hp);
    h->GV2 = c.take<float>(size_t(R) * Hp);
    h->GF2 = c.take<float>(size_t(R) * Hp);
    h->dWtmp2 = c.take<float>(size_t(Hp) * Hp);
    for (int l = 0; l + 1 < h->n_levels; ++l) h->dAtt[l] = c.take<float>(size_t(R) * Hp);
  }
  auto planes_for = [&](FcRef& f) {
    f.bias_pad = c.take<float>(size_t(f.n_out_pad));
    f.wp = c.take<__nv_bfloat16>(size_t(f.n_out_pad) * kPl * f.n_in_pad);
    // the transposed weights feed only the dX GEMM, which the wide first layer does not run
    f.wtp = (h->wide && &f == &h->lvl[0].fc[0]) ? nullptr
                                                 : c.take<__nv_bfloat16>(size_t(f.n_in_pad) * kPl * f.n_out_pad);
  };
  for (int l = 0; l < h->n_levels; ++l) {
    for (int j = 0; j < h->lvl[l].n_fc; ++j) planes_for(h->lvl[l].fc[j]);
    planes_for(h->lvl[l].fcv);
  }
  planes_for(h->fc_out);
  h->ws_bytes = c.off;
}

// the flat layout: named_parameters() order of the reference module with fcf left out (model.py:200-256)
void build_layout(vmb_mla_trainer* h, const int* n_fc) {
  long long p = 0, r = 0;
  int slot = 0;
  auto bn = [&](int n) {
    BnRef b{p, p + n, r, n, slot, slot + 1};
    slot += 2;
    p += 2 * n;
    r += 2 * n;
    return b;
  };
  // every hidden / class dimension is padded to the common width Hp, the embedding input to inpad and the
  // concatenated attention outputs to ycols_pad, so that a plane written for one GEMM can feed the next
  auto fc = [&](int n_out, int n_in, int n_in_pad) {
    FcRef f{};
    f.w = p; f.b = p + 1LL * n_out * n_in;
    f.n_out = n_out; f.n_in = n_in; f.n_out_pad = h->Hp; f.n_in_pad = n_in_pad;
    p += 1LL * n_out * n_in + n_out;
    return f;
  };
  for (int l = 0; l < h->n_levels; ++l) {
    LevelRef& L = h->lvl[l];
    L.n_fc = n_fc[l];
    L.norm0 = bn(h->T);
    for (int j = 0; j < L.n_fc; ++j) {
      const bool first = l == 0 && j == 0;
      L.fc[j] = fc(h->H, first ? h->emb_in : h->H, first ? h->inpad : h->Hp);
    }
    for (int j = 0; j < L.n_fc; ++j) L.norms[j] = bn(h->T);
  }
  for (int l = 0; l < h->n_levels; ++l) {
    LevelRef& L = h->lvl[l];
    L.fcv = fc(h->K, h->H, h->Hp);
    L.normv = bn(h->T);
    L.normf = bn(h->T);
  }
  h->fc_out = fc(h->K, h->n_levels * h->K, h->ycols_pad);
  h->norm_out = bn(h->K);
  h->n_params = p;
  h->n_running = r;
  h->n_slots = slot;
  // level 0's embedding chain is the last thing the backward pass computes; everything after it in the flat order is final earlier
  h->tail_offset = h->n_levels > 1 ? h->lvl[1].norm0.g : h->lvl[0].fcv.w;
}

dim3 tile_grid(long long rows_pad, int cols_pad) {
  return dim3(static_cast<unsigned>((cols_pad + kTile - 1) / kTile), static_cast<unsigned>((rows_pad + kTile - 1) / kTile));
}

template <class F>
int run_tile(F f, TileOut o, cudaStream_t st, const char* what) {
  vmb::launch_pdl(tile_split_kernel<F>, tile_grid(o.rows_pad, o.cols_pad), dim3(256), 0, st, f, o);
  vmb::count_launch();
  return vmb::check_launch(what);
}

// dW [M][N] = sum over the rows r of g[r][m] b[r][n]: the gradient planes g [rows][kPl * M] against the layer input's
// planes b [rows][kPl * N], both row-major as the forward / dX GEMMs consume them
int gemm_dw(const void* g_planes, int M, const void* b_planes, int N, float* out, long long rows, cudaStream_t st) {
  if (vmb::planes_gemm_dw(g_planes, M, b_planes, N, out, N, M, N, int(rows), kPl, st)) {
    vmb::set_kernel_error("%s", vmb::planes_gemm_last_error());
    return 1;
  }
  return 0;
}

int gemm(const void* a_planes, const void* w_planes, const float* bias, float* out, long long ldo, long long M, int N,
         int K, cudaStream_t st) {
  if (vmb::planes_gemm(a_planes, w_planes, bias, out, ldo, 0, int(M), N, K, kPl, 0, st)) {
    vmb::set_kernel_error("%s", vmb::planes_gemm_last_error());
    return 1;
  }
  return 0;
}

// Linear + the BatchNorm statistics of its output in one kernel (planes_gemm_stats)
int gemm_stats(const void* a_planes, const void* w_planes, const float* bias, float* out, long long ldo, long long M, int N,
               int K, const StatJob& j, int cols, cudaStream_t st) {
  vmb::PlanesStats ps{j.acc, j.stat, j.counter, j.run_mean, j.run_var, j.count, j.channels, cols, kBnEps, kBnMomentum};
  if (vmb::planes_gemm_stats(a_planes, w_planes, bias, out, ldo, int(M), N, K, kPl, ps, st)) {
    vmb::set_kernel_error("%s", vmb::planes_gemm_last_error());
    return 1;
  }
  return 0;
}

// dX GEMM + the BatchNorm-backward reductions of the block that consumes its output (planes_gemm_gradstats): replaces
// gemm() followed by bn_time_backward_reduce_kernel when the block's only upstream gradient is this GEMM's output.
bool gradstats_in_gemm(const GradIn& gi) {
  return !gi.da2 && gi.ldu % 4 == 0 && (gi.F + 3) / 4 * 4 <= gi.ldu && (reinterpret_cast<uintptr_t>(gi.u) & 15) == 0;
}

int gemm_gradstats(const void* a_planes, const void* w_planes, float* out, long long ldo, long long M, int N, int K,
                   const GradIn& gi, double* acc, cudaStream_t st) {
  vmb::PlanesGradStats gs{gi.u, gi.ldu, gi.stat, gi.gamma, gi.beta, acc, gi.seed, gi.layer, gi.p, gi.relu, gi.T, gi.F, gi.F};
  if (vmb::planes_gemm_gradstats(a_planes, w_planes, out, ldo, int(M), N, K, kPl, gs, st)) {
    vmb::set_kernel_error("%s", vmb::planes_gemm_last_error());
    return 1;
  }
  return 0;
}

}  // namespace

extern "C" {

long long vmb_mla_train_param_count(int n_levels, const int* n_fc, int emb_in, int hidden, int n_classes, int t_steps,
                                    long long* n_running_out) {
  if (n_levels < 1 || n_levels > kMaxLevels || !n_fc) return -1;
  vmb_mla_trainer tmp{};
  tmp.n_levels = n_levels; tmp.emb_in = emb_in; tmp.H = hidden; tmp.K = n_classes; tmp.T = t_steps;
  tmp.Hp = std::max(pad128(hidden), pad128(n_classes));
  tmp.inpad = pad128(emb_in);
  tmp.ycols_pad = pad128(n_levels * n_classes);
  build_layout(&tmp, n_fc);
  if (n_running_out) *n_running_out = tmp.n_running;
  return tmp.n_params;
}

int vmb_mla_trainer_create(vmb_mla_trainer_t** handle, int n_levels, const int* n_fc, int emb_in, int hidden,
                           int n_classes, int t_steps, long long max_batch, void* stream) {
  if (!handle || !n_fc) return fail("vmb_mla_trainer_create: null argument");
  if (n_levels < 1 || n_levels > kMaxLevels) return fail("vmb_mla_trainer_create: 1..4 levels supported");
  for (int l = 0; l < n_levels; ++l)
    if (n_fc[l] < 1 || n_fc[l] > kMaxFc) return fail("vmb_mla_trainer_create: 1..4 fully connected layers per level");
  if (t_steps < 1 || t_steps > 16) return fail("vmb_mla_trainer_create: 1 <= T <= 16");
  if (emb_in < 1 || emb_in > 16384 || hidden < 1 || hidden > 1024 || n_classes < 1 || n_classes > 1024)
    return fail("vmb_mla_trainer_create: hidden and n_classes must be in 1..1024, emb_in in 1..16384");
  if (max_batch < 2 || max_batch * t_steps > 0x7fffffffLL / 2048) return fail("vmb_mla_trainer_create: bad max_batch");
  const bool wide = pad128(emb_in) > std::max(pad128(hidden), pad128(n_classes));
  if (wide) {
    // The wide first layer's largest per-step buffer is the operand planes of xhat, [pad64(batch * T)][3 * inpad]
    // bf16: its element count stays within a signed 32-bit index (at emb_in 12288, T = 10: 5824 clips)
    const long long per_row = static_cast<long long>(kPl) * pad128(emb_in);
    const long long max_rows = 0x7fffffffLL / per_row / 64 * 64;
    if (pad64(max_batch * t_steps) > max_rows) {
      char msg[256];
      snprintf(msg, sizeof msg, "vmb_mla_trainer_create: max_batch %lld too large for emb_in %d, T %d: at most %lld clips",
               max_batch, emb_in, t_steps, max_rows / t_steps);
      return fail("%s", msg);
    }
  }
  vmb_mla_trainer* h = new vmb_mla_trainer();
  h->n_levels = n_levels; h->emb_in = emb_in; h->H = hidden; h->K = n_classes; h->T = t_steps;
  h->max_batch = max_batch;
  h->wide = wide;
  h->Hp = std::max(pad128(hidden), pad128(n_classes));
  h->inpad = pad128(emb_in);
  h->ycols = n_levels * n_classes;
  h->ycols_pad = pad128(h->ycols);
  build_layout(h, n_fc);
  carve(h, nullptr);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (cudaMalloc(reinterpret_cast<void**>(&h->ws), h->ws_bytes) != cudaSuccess) {
    delete h;
    return fail("vmb_mla_trainer_create: workspace allocation failed (%s)", cudaGetErrorString(cudaGetLastError()));
  }
  carve(h, h->ws);
  // padding of every plane / fp32 buffer stays zero for the life of the handle
  if (cudaMemsetAsync(h->ws, 0, h->ws_bytes, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
    cudaFree(h->ws);
    delete h;
    return fail("vmb_mla_trainer_create: workspace clear failed");
  }
  *handle = h;
  return 0;
}

void vmb_mla_trainer_destroy(vmb_mla_trainer_t* h) {
  if (h && h->side) {
    cudaStreamSynchronize(h->side);
    cudaStreamDestroy(h->side);
  }
  if (h && h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h && h->ev_dw) cudaEventDestroy(h->ev_dw);
  if (h && h->ev_att) cudaEventDestroy(h->ev_att);
  if (h && h->ev_w) cudaEventDestroy(h->ev_w);
  if (h && h->ev_tail) cudaEventDestroy(h->ev_tail);
  if (h && h->side2) {
    cudaStreamSynchronize(h->side2);
    cudaStreamDestroy(h->side2);
  }
  for (int i = 0; h && i < kMaxLevels; ++i)
    if (h->ev_attb[i]) cudaEventDestroy(h->ev_attb[i]);
  if (!h) return;
  for (int i = 0; i < h->n_graphs; ++i)
    if (h->graphs[i].exec) cudaGraphExecDestroy(h->graphs[i].exec);
  if (h->gstream) {
    cudaStreamSynchronize(h->gstream);
    cudaStreamDestroy(h->gstream);
  }
  if (h->ev_in) cudaEventDestroy(h->ev_in);
  if (h->ev_out) cudaEventDestroy(h->ev_out);
  cudaFree(h->ws);
  delete h;
}

}  // extern "C"

namespace {
enum { kPhaseForward = 1, kPhaseBackward = 2 };

// One implementation for forward, backward and the fused step: the phases share the layout arithmetic.
int train_phases(int phases, vmb_mla_trainer* h, const float* params, float* running, const float* x,
                 const long long* labels, const float* dscores, long long batch, float dropout_p,
                 unsigned long long seed, float* grads, float* loss, float* scores, void* stream, float* dx = nullptr) {
  if (!h) return fail("vmb_mla_train: null handle");
  if (!params || !x) return fail("vmb_mla_train: null pointer");
  if ((phases & kPhaseForward) && !running) return fail("vmb_mla_train: forward needs the running-statistics buffer");
  if ((phases & kPhaseBackward) && (!grads || (!labels && !dscores)))
    return fail("vmb_mla_train: backward needs grads and either labels or d(scores)");
  if (labels && !loss) return fail("vmb_mla_train: labels given but no loss output");
  if (batch < 2 || batch > h->max_batch) return fail("vmb_mla_train: batch must be in 2..max_batch");
  if (dropout_p < 0.f || dropout_p >= 1.f) return fail("vmb_mla_train: dropout_p must be in [0, 1)");
  const bool do_fwd = phases & kPhaseForward, do_bwd = phases & kPhaseBackward;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!h->capturing) {   // a captured step reads the seed its replay was given (vmb_mla_train_step)
    set_seed_kernel<<<1, 1, 0, st>>>(h->seed_dev, seed);
    vmb::count_launch();
  }
  const int T = h->T, H = h->H, K = h->K, Hp = h->Hp, inpad = h->inpad;
  const long long B = batch, R = B * T, Rp = pad64(R), Bp = pad64(B);
  int rc = 0;
#define TRY(expr) do { if (!rc && (expr)) rc = 1; } while (0)

  // forward statistics live in even slots, backward reductions in odd slots: the forward clears everything, a
  // separate backward call must not (it still needs the forward statistics) — backward slots are re-zeroed below
  if (do_fwd && (cudaMemsetAsync(h->acc, 0, h->acc_bytes, st) != cudaSuccess ||
                 (loss && cudaMemsetAsync(loss, 0, 4, st) != cudaSuccess)))
    return fail("vmb_mla_train: memset failed");
  if (do_bwd && cudaMemsetAsync(grads, 0, size_t(h->n_params) * 4, st) != cudaSuccess)
    return fail("vmb_mla_train: memset failed");
  if (do_bwd && !do_fwd)
    for (int s = 1; s < h->n_slots; s += 2)
      if (cudaMemsetAsync(h->acc + size_t(s) * kSlot * 2, 0, size_t(kSlot) * 2 * sizeof(double), st) != cudaSuccess)
        return fail("vmb_mla_train: memset failed");
  auto slotacc = [&](int s) { return h->acc + size_t(s) * kSlot * 2; };
  auto slotstat = [&](int s) { return h->stat + size_t(s) * kSlot * 2; };
  auto statjob = [&](const BnRef& bn, double count) {
    return StatJob{slotacc(bn.slot), slotstat(bn.slot), h->counters + bn.slot, running + bn.rm, running + bn.rm + bn.n,
                   count, bn.n};
  };
  // Side stream (created on first use): work that feeds nothing on the critical chain runs there — in the forward pass
  // the attention branch of every level but the last (fcv GEMM, statistics, pooling: only the concatenation at the end
  // needs it), in the backward pass the weight-gradient GEMMs.
  if (!h->side) {
    if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_dw, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_att, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_w, cudaEventDisableTiming) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->side2, cudaStreamNonBlocking) != cudaSuccess)
      return fail("vmb_mla_train: cannot create the side stream");
    for (int i = 0; i < kMaxLevels; ++i)
      if (cudaEventCreateWithFlags(&h->ev_attb[i], cudaEventDisableTiming) != cudaSuccess)
        return fail("vmb_mla_train: cannot create the side stream");
  }
  WeightJobs wj{};
  auto weights = [&](const FcRef& f) {
    const int j = wj.n++;
    wj.o[j] = TileOut{f.wp, nullptr, 0, nullptr, f.n_out, f.n_out_pad, f.n_in, f.n_in_pad};
    wj.o[j].planes_t = f.wtp;
    wj.f[j] = FIdentity{params + f.w, f.n_in, params + f.b, f.bias_pad, f.n_out};
    const dim3 g = tile_grid(f.n_out_pad, f.n_in_pad);
    wj.tiles_x[j] = int(g.x);
    wj.first_tile[j + 1] = wj.first_tile[j] + int(g.x * g.y);
    return 0;
  };
  const LevelRef& L0 = h->lvl[0];
  // Linear (+ bias) into `out` and the BatchNorm statistics of its first `cols` columns
  auto gemm_bn = [&](const void* a, const FcRef& fc, float* out, int k_pad, int cols, const BnRef& bn, cudaStream_t ss) {
    if (h->wide && &fc == &L0.fc[0]) {
      // P = xhat W^T with the K loop cut into slices of kFwdSlice columns (fp32 reductions into a zeroed P): one
      // tcgen05 accumulator summed over all 12288 columns loses ~1e-4 relative to its per-step truncation, which moved
      // gradients past the fp32 reference's tolerance.  Then U = gamma_t P + beta_t s + b and U's statistics.
      if (cudaMemsetAsync(h->P0, 0, size_t(R) * Hp * sizeof(float), ss) != cudaSuccess) {
        vmb::set_kernel_error("wide-layer output clear failed");
        return 1;
      }
      if (vmb::planes_gemm(a, fc.wp, nullptr, h->P0, Hp, 0, int(R), Hp, k_pad, kPl,
                           (k_pad + vmb::kFwdSlice - 1) / vmb::kFwdSlice, ss)) {
        vmb::set_kernel_error("%s", vmb::planes_gemm_last_error());
        return 1;
      }
      FAffine f{h->P0, Hp, T, params + L0.norm0.g, params + L0.norm0.b, h->wsum, fc.bias_pad};
      TileOut o{nullptr, out, Hp, nullptr, R, R, cols, Hp};
      o.stats = statjob(bn, double(B) * cols);
      o.stats_T = T;
      return run_tile(f, o, ss, "wide-layer affine + statistics");
    }
    return gemm_stats(a, fc.wp, fc.bias_pad, out, Hp, R, Hp, k_pad, statjob(bn, double(B) * cols), cols, ss);
  };

  if (do_fwd) {
  // ---- weights -> hi|mid|lo planes, row-major and transposed (they changed in the last optimiser step), on the side
  // stream: the first Linear needs them only after the level-0 norm0 statistics and its activation pass, which do not
  // depend on the weights
  cudaEventRecord(h->ev_fork, st);   // after the optimiser step (and everything else) on the caller's stream
  cudaStreamWaitEvent(h->side, h->ev_fork, 0);
  for (int l = 0; l < h->n_levels; ++l) {
    for (int j = 0; j < h->lvl[l].n_fc; ++j) TRY(weights(h->lvl[l].fc[j]));
    TRY(weights(h->lvl[l].fcv));
  }
  TRY(weights(h->fc_out));
  if (!rc) {
    vmb::launch_pdl(weights_split_kernel, dim3(unsigned(wj.first_tile[wj.n])), dim3(256), 0, h->side, wj);
    vmb::count_launch();
    TRY(vmb::check_launch("weights_split_kernel"));
  }
  if (!rc && h->wide) {   // s[o] = sum_f W[o][f] of the wide first Linear (its GEMM epilogue and the backward pass)
    row_sum_kernel<<<static_cast<unsigned>(L0.fc[0].n_out), 256, 0, h->side>>>(params + L0.fc[0].w, L0.fc[0].n_in,
                                                                              h->wsum);
    vmb::count_launch();
    TRY(vmb::check_launch("row_sum_kernel"));
  }
  cudaEventRecord(h->ev_w, h->side);
  bool weights_pending = true;

  // =============================================================================== forward
  bool att_pending = false;
  for (int l = 0; l < h->n_levels && !rc; ++l) {
    const LevelRef& L = h->lvl[l];
    const float* in = l == 0 ? x : h->E[l - 1];
    const long long ld_in = l == 0 ? h->emb_in : Hp;
    const int F_in = l == 0 ? h->emb_in : H;
    const int in_pad = l == 0 ? inpad : Hp;
    __nv_bfloat16* np = l == 0 ? h->xin_p : h->N_p[l];
    if (l == 0) {   // the statistics of a later level's input come with the pass that writes it (below)
      const StatJob j = statjob(L.norm0, double(B) * F_in);
      const unsigned chunks = static_cast<unsigned>(std::min<long long>((B * F_in + 256 * 8 - 1) / (256 * 8), 64));
      vmb::launch_pdl(bn_time_stats_kernel, dim3(chunks, T), dim3(256), 0, st, in, ld_in, B, F_in, T, j);
      vmb::count_launch();
      TRY(vmb::check_launch("bn_time_stats_kernel"));
    }
    if (l == 0 && h->wide) {
      TileOut o{np, nullptr, 0, nullptr, R, Rp, F_in, in_pad};
      TRY(run_tile(FNormalize{in, ld_in, T, slotstat(L.norm0.slot)}, o, st, "norm0 forward (xhat)"));
    } else {
      FBnAct f{in, ld_in, T, F_in, slotstat(L.norm0.slot), params + L.norm0.g, params + L.norm0.b, 0, 0.f, h->seed_dev, 0};
      TileOut o{np, nullptr, 0, nullptr, R, Rp, F_in, in_pad};
      TRY(run_tile(f, o, st, "norm0 forward"));
    }
    const __nv_bfloat16* a = np;
    if (weights_pending) {
      cudaStreamWaitEvent(st, h->ev_w, 0);           // join: every weight plane is written
      weights_pending = false;
    }
    for (int j = 0; j < L.n_fc && !rc; ++j) {
      const FcRef& fc = L.fc[j];
      TRY(gemm_bn(a, fc, h->U[l][j], fc.n_in_pad, H, L.norms[j], st));
      const bool last = j == L.n_fc - 1;
      FBnAct f{h->U[l][j], Hp, T, H, slotstat(L.norms[j].slot), params + L.norms[j].g, params + L.norms[j].b, 1,
               dropout_p, h->seed_dev, unsigned(1 + l * kMaxFc + j)};
      TileOut o{h->A_p[l][j], last ? h->E[l] : nullptr, Hp, nullptr, R, Rp, H, Hp};
      if (last && l + 1 < h->n_levels) {
        // the embedding this pass writes is the input of the next level's norm0: its batch statistics ride along
        o.stats = statjob(h->lvl[l + 1].norm0, double(B) * H);
        o.stats_T = T;
      }
      TRY(run_tile(f, o, st, "fc forward activation"));
      a = h->A_p[l][j];
    }
    // attention branch of this level: every buffer it writes is per level (Z[l], its statistic slots, columns l*K.. of Y),
    // so with another level still to come it runs on the side stream next to that level's chain
    const bool side = l + 1 < h->n_levels;
    cudaStream_t as = side ? h->side : st;
    if (side && !rc) {
      cudaEventRecord(h->ev_fork, st);               // the level's last activation planes (a) are complete
      cudaStreamWaitEvent(h->side, h->ev_fork, 0);
    }
    TRY(gemm_bn(a, L.fcv, h->Z[l], Hp, K, L.normv, as));
    if (!rc) {
      // normf shares the batch statistics but keeps its own running buffers
      StatJob j = statjob(L.normf, double(B) * K);
      j.acc = slotacc(L.normv.slot);
      j.stat = slotstat(L.normf.slot);
      bn_running_only_kernel<<<1, 32, 0, as>>>(j);
      vmb::count_launch();
      TRY(vmb::check_launch("bn_running_only_kernel"));
      AttParams ap{h->Z[l], Hp, K, T, slotstat(L.normv.slot), params + L.normv.g, params + L.normv.b,
                   params + L.normf.g, params + L.normf.b};
      // the pooling kernel also writes the output Linear's operand planes
      vmb::launch_pdl(att_forward_kernel, dim3(static_cast<unsigned>(Bp)), dim3(256), 0, as, ap, h->Y,
                      static_cast<long long>(h->ycols_pad), l * K, h->row_stats[l], h->Y_p, h->ycols_pad, B);
      vmb::count_launch();
      TRY(vmb::check_launch("att_forward_kernel"));
    }
    if (side) {
      cudaEventRecord(h->ev_att, h->side);
      att_pending = true;
    }
  }
  if (att_pending) cudaStreamWaitEvent(st, h->ev_att, 0);   // join: the concatenation below reads every level's pooling
  // output layer
  TRY(gemm(h->Y_p, h->fc_out.wp, h->fc_out.bias_pad, h->O, Hp, B, Hp, h->ycols_pad, st));
  if (!rc) {
    StatJob j = statjob(h->norm_out, double(B));
    vmb::launch_pdl(bn_col_stats_kernel, dim3((K + kColsPerCta - 1) / kColsPerCta), dim3(256), 0, st, h->O, Hp, B, K, j);
    vmb::count_launch();
    TRY(vmb::check_launch("bn_col_stats_kernel"));
    const float* stat = slotstat(h->norm_out.slot);
    out_loss_rows_kernel<<<static_cast<unsigned>(B), 256, 0, st>>>(h->O, Hp, K, stat, params + h->norm_out.g,
                                                                   params + h->norm_out.b, labels, B, scores, h->lse, loss);
    vmb::count_launch();
    TRY(vmb::check_launch("out_loss_rows_kernel"));
  }
  }  // do_fwd
  if (do_bwd) {
  // =============================================================================== backward
  // Weight-gradient GEMMs on the side stream: each reads the gradient planes G_p the tile kernel just wrote and an
  // activation's planes, and writes only its slice of `grads` — nothing on the dX chain waits for it.  The chain only
  // has to wait (ev_dw) before the NEXT tile kernel overwrites G_p, one dX GEMM and one reduction later.
  bool dw_pending = false;
  // dW [n_out][n_in] of a Linear (G_p against its input's planes b [rows][kPl * b_cols]) -> dst, its block of `grads`
  auto dw_job = [&](const void* b, int b_cols, long long rows, float* dst, int n_out, int n_in) {
    cudaEventRecord(h->ev_fork, st);
    cudaStreamWaitEvent(h->side, h->ev_fork, 0);
    int r = gemm_dw(h->G_p, Hp, b, b_cols, h->dWtmp, rows, h->side);
    if (!r && dst == grads + L0.fc[0].w && h->wide) {
      // the wide first Linear: dW = the GEMM's sum_r (gamma_t G) xhat + c[o] (see wide_grad_tile_kernel)
      vmb::launch_pdl(wide_dw_finish_kernel, dim3(unsigned((n_in + 1023) / 1024), unsigned(n_out)), dim3(256), 0,
                      h->side, static_cast<const float*>(h->dWtmp), static_cast<long long>(b_cols), dst, n_in,
                      static_cast<const float*>(h->gsum_t), Hp, params + L0.norm0.b, T);
      vmb::count_launch();
      r = vmb::check_launch("wide_dw_finish_kernel");
    } else if (!r && cudaMemcpy2DAsync(dst, size_t(n_in) * 4, h->dWtmp, size_t(b_cols) * 4, size_t(n_in) * 4, n_out,
                                       cudaMemcpyDeviceToDevice, h->side) != cudaSuccess) {
      vmb::set_kernel_error("dW copy failed");
      r = 1;
    }
    cudaEventRecord(h->ev_dw, h->side);
    dw_pending = true;
    return r;
  };
  auto before_g_overwrite = [&]() {   // G_p (and dWtmp's reader) are about to be rewritten by the chain
    if (dw_pending) {
      cudaStreamWaitEvent(st, h->ev_dw, 0);
      dw_pending = false;
    }
  };
  if (!rc) {
    const float* stat = slotstat(h->norm_out.slot);
    out_bn_backward_kernel<<<(K + kColsPerCta - 1) / kColsPerCta, 256, 0, st>>>(h->O, Hp, K, stat, params + h->norm_out.g, params + h->norm_out.b,
                                                          labels, h->lse, dscores, B, h->dO, Hp, grads + h->norm_out.g,
                                                          grads + h->norm_out.b);
    vmb::count_launch();
    TRY(vmb::check_launch("out_bn_backward_kernel"));
  }
  {
    // dO planes and d(bias) = column sums
    TileOut o{h->G_p, nullptr, 0, grads + h->fc_out.b, B, Bp, K, Hp};
    TRY(run_tile(FIdentity{h->dO, Hp}, o, st, "dO split"));
    // dW_fc [K][L*K] = dO^T [K x B] * Y [B x L*K]
    TRY(dw_job(h->Y_p, h->ycols_pad, Bp, grads + h->fc_out.w, K, h->ycols));
    // dY [B][L*K] = dO [B x K] * W_fc [K x L*K]
    TRY(gemm(h->G_p, h->fc_out.wtp, nullptr, h->dY, h->ycols_pad, B, h->ycols_pad, Hp, st));
  }
  // attention branch of level l: d(loss)/dZ_l from dY, its BatchNorm / fcv parameter gradients, dWv, and the gradient it
  // sends into the level's embedding (dE_att -> out_dA).  With own_side == false it runs on the caller's stream with the
  // chain's scratch (and its dW GEMM goes through dw_job); with own_side == true everything runs on `s` with the second
  // set of scratch buffers.
  // The BatchNorm (+ ReLU + dropout) block (l, j) — j == -1: the level's norm0 — as the backward pass sees it, with its
  // upstream gradient(s); and the slot of its two backward reductions.
  auto block_gi = [&](int l, int j, const float* da1, const float* da2) {
    const LevelRef& L = h->lvl[l];
    if (j >= 0)
      return GradIn{da1, Hp, da2, Hp, h->U[l][j], Hp, T, H, slotstat(L.norms[j].slot), params + L.norms[j].g,
                    params + L.norms[j].b, 1, dropout_p, h->seed_dev, unsigned(1 + l * kMaxFc + j)};
    const float* in = l == 0 ? x : h->E[l - 1];
    const long long ld_in = l == 0 ? h->emb_in : Hp;
    const int F_in = l == 0 ? h->emb_in : H;
    return GradIn{da1, Hp, nullptr, 0, in, ld_in, T, F_in, slotstat(L.norm0.slot), params + L.norm0.g,
                  params + L.norm0.b, 0, 0.f, h->seed_dev, 0};
  };
  auto block_acc = [&](int l, int j) { return slotacc(j >= 0 ? h->lvl[l].norms[j].bslot : h->lvl[l].norm0.bslot); };
  // dX GEMM into `out`, the upstream gradient of block (l, j): when that is the block's only upstream gradient, the
  // block's reductions ride in the GEMM's epilogue and `pre_reduced` tells the consumer not to launch its own pass
  bool pre_reduced = false;
  auto gemm_into_block = [&](const void* a, const void* wt, float* out, int n_pad, int l, int j, const float* da2,
                             cudaStream_t s) {
    const GradIn gi = block_gi(l, j, out, da2);
    if (gradstats_in_gemm(gi)) {
      pre_reduced = true;
      return gemm_gradstats(a, wt, out, Hp, R, n_pad, Hp, gi, block_acc(l, j), s);
    }
    pre_reduced = false;
    return gemm(a, wt, nullptr, out, Hp, R, n_pad, Hp, s);
  };
  // att / cla of one clip, [T][K] fp32 each: 128 KB at the largest accepted shape (T = 16, K = 1024)
  const size_t att_smem = size_t(2) * T * K * sizeof(float);
  static std::atomic<unsigned long long> att_attr{0};   // one bit per device: the attribute is per device
  if (vmb::device_needs_setup(att_attr))
    cudaFuncSetAttribute(att_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         int(2 * 16 * 1024 * sizeof(float)));
  auto att_branch = [&](int l, cudaStream_t s, bool own_side, float* out_dA) {
    const LevelRef& L = h->lvl[l];
    const __nv_bfloat16* e_p = h->A_p[l][L.n_fc - 1];
    __nv_bfloat16* gp = own_side ? h->G_p2 : h->G_p;
    float* gv = own_side ? h->GV2 : h->GV;
    float* gf = own_side ? h->GF2 : h->GF;
    AttParams ap{h->Z[l], Hp, K, T, slotstat(L.normv.slot), params + L.normv.g, params + L.normv.b,
                 params + L.normf.g, params + L.normf.b};
    double* acc_v = slotacc(L.normv.bslot);
    double* acc_f = slotacc(L.normf.bslot);
    att_backward_kernel<<<static_cast<unsigned>(B), 256, att_smem, s>>>(ap, h->Y, h->dY, h->ycols_pad, l * K,
                                                                        h->row_stats[l], gv, gf, Hp, acc_v, acc_f);
    vmb::count_launch();
    TRY(vmb::check_launch("att_backward_kernel"));
    {
      FAttCombine f{ap, gv, gf, Hp, acc_v, acc_f, double(B) * K, grads + L.normv.g, grads + L.normv.b,
                    grads + L.normf.g, grads + L.normf.b};
      TileOut o{gp, nullptr, 0, grads + L.fcv.b, R, Rp, K, Hp};
      if (!own_side) before_g_overwrite();
      TRY(run_tile(f, o, s, "attention BN backward"));
    }
    // dWv [K][H] = dZ^T * E ; dE_att [R][H] = dZ * Wv
    if (own_side) {
      TRY(gemm_dw(gp, Hp, e_p, Hp, h->dWtmp2, Rp, s));
      if (!rc && cudaMemcpy2DAsync(grads + L.fcv.w, size_t(H) * 4, h->dWtmp2, size_t(Hp) * 4, size_t(H) * 4, K,
                                   cudaMemcpyDeviceToDevice, s) != cudaSuccess)
        rc = 1;
    } else {
      TRY(dw_job(e_p, Hp, Rp, grads + L.fcv.w, K, H));
    }
    if (own_side) {
      TRY(gemm(gp, L.fcv.wtp, nullptr, out_dA, Hp, R, Hp, Hp, s));     // joins the chain as one of two upstream gradients
    } else {
      TRY(gemm_into_block(gp, L.fcv.wtp, out_dA, Hp, l, L.n_fc - 1, (l + 1 < h->n_levels) ? h->dEnext : nullptr, s));
    }
  };
  // fork: every level below the last starts its attention branch now (dY is complete), on the second side stream
  const bool att_fork = h->n_levels > 1;
  if (att_fork && !rc) {
    cudaEventRecord(h->ev_fork, st);
    cudaStreamWaitEvent(h->side2, h->ev_fork, 0);
    for (int l = h->n_levels - 2; l >= 0; --l) {
      att_branch(l, h->side2, true, h->dAtt[l]);
      cudaEventRecord(h->ev_attb[l], h->side2);
    }
  }
  // levels in reverse
  for (int l = h->n_levels - 1; l >= 0 && !rc; --l) {
    const LevelRef& L = h->lvl[l];
    const float* da1 = h->dA;
    if (att_fork && l + 1 < h->n_levels) {
      cudaStreamWaitEvent(st, h->ev_attb[l], 0);    // this level's attention gradient comes from the side branch
      da1 = h->dAtt[l];
    } else {
      att_branch(l, st, false, h->dA);
    }
    if (l == 0) {
      // everything but level 0's embedding chain has its gradient: the weight-gradient GEMMs still on the side stream
      // are joined, then the tail event marks grads[tail_offset ..] final (vmb_mla_train_wait_tail)
      before_g_overwrite();
      if (!h->ev_tail && cudaEventCreateWithFlags(&h->ev_tail, cudaEventDisableTiming) != cudaSuccess) {
        vmb::set_kernel_error("cannot create the tail event");
        rc = 1;
      }
      if (h->ev_tail) cudaEventRecordWithFlags(h->ev_tail, st, h->capturing ? cudaEventRecordExternal : cudaEventRecordDefault);
    }
    // embedding chain of this level, last Linear first; gradient wrt E_l = attention part (+ next level's input grad)
    const float* da2 = (l + 1 < h->n_levels) ? h->dEnext : nullptr;
    for (int j = L.n_fc - 1; j >= 0 && !rc; --j) {
      const FcRef& fc = L.fc[j];
      const GradIn gi = block_gi(l, j, da1, da2);
      double* acc = block_acc(l, j);
      if (!pre_reduced) {
        const unsigned chunks = static_cast<unsigned>(std::min<long long>((B * H + 256 * 8 - 1) / (256 * 8), 64));
        vmb::launch_pdl(bn_time_backward_reduce_kernel, dim3(chunks, T), dim3(256), 0, st, gi, B, acc);
        vmb::count_launch();
        TRY(vmb::check_launch("bn_time_backward_reduce_kernel"));
      }
      FBnBackward f{gi, acc, double(B) * H, grads + L.norms[j].g, grads + L.norms[j].b};
      const bool wide0 = h->wide && l == 0 && j == 0;
      before_g_overwrite();
      if (wide0) {
        // G of the wide first Linear: gamma_t-scaled planes for dW, the sums for c[o] and for norm0's two gradients
        if (cudaMemsetAsync(h->gsum_t, 0, size_t(T) * Hp * sizeof(float), st) != cudaSuccess) {
          vmb::set_kernel_error("wide-layer column sums clear failed");
          rc = 1;
        }
        WideGradOut o{h->G_p, R, Rp, H, Hp, params + L.norm0.g, h->P0, Hp, h->wsum, grads + fc.b, h->gsum_t,
                      block_acc(0, -1)};
        if (!rc) {
          vmb::launch_pdl(wide_grad_tile_kernel, tile_grid(Rp, Hp), dim3(256), 0, st, f, o);
          vmb::count_launch();
          TRY(vmb::check_launch("wide_grad_tile_kernel"));
        }
      } else {
        TileOut o{h->G_p, nullptr, Hp, grads + fc.b, R, Rp, H, Hp};
        TRY(run_tile(f, o, st, "fc BN backward"));
      }
      // dW [H][n_in] = dU^T * A_prev ; dA_prev [R][n_in] = dU * W
      const __nv_bfloat16* prev_p = j > 0 ? h->A_p[l][j - 1] : (l == 0 ? h->xin_p : h->N_p[l]);
      TRY(dw_job(prev_p, fc.n_in_pad, Rp, grads + fc.w, H, fc.n_in));
      float* dprev = (da1 == h->dA) ? h->dB : h->dA;
      if (wide0)
        pre_reduced = true;   // no dX GEMM: norm0's two reductions came from wide_grad_tile_kernel
      else
        TRY(gemm_into_block(h->G_p, fc.wtp, dprev, fc.n_in_pad, l, j - 1, nullptr, st));   // j - 1 == -1: the level's norm0
      da1 = dprev;
      da2 = nullptr;
    }
    // norm0 of this level: gradient wrt its input (= E_{l-1} for l > 0) and its affine parameters
    {
      const int F_in = l == 0 ? h->emb_in : H;
      const GradIn gi = block_gi(l, -1, da1, nullptr);
      double* acc = block_acc(l, -1);
      if (!pre_reduced) {
        const unsigned chunks = static_cast<unsigned>(std::min<long long>((B * F_in + 256 * 8 - 1) / (256 * 8), 64));
        vmb::launch_pdl(bn_time_backward_reduce_kernel, dim3(chunks, T), dim3(256), 0, st, gi, B, acc);
        vmb::count_launch();
        TRY(vmb::check_launch("bn_time_backward_reduce_kernel"));
      }
      pre_reduced = false;
      FBnBackward f{gi, acc, double(B) * F_in, grads + L.norm0.g, grads + L.norm0.b};
      // level 0: only the parameter gradients are needed (written by the prologue); still run one tile row so
      // the prologue executes (with the wide first layer no element is evaluated: there is no dY).  level > 0: fp32
      // gradient wrt E_{l-1}
      TileOut o{nullptr, l > 0 ? h->dEnext : nullptr, Hp, nullptr, l > 0 ? R : 1, l > 0 ? R : 1,
                (l == 0 && h->wide) ? 0 : F_in, l > 0 ? Hp : 32};
      float* dx_pad = (da1 == h->dA) ? h->dB : h->dA;   // level 0 with dx: the chain buffer norm0's input does not use
      if (l == 0 && dx) o = TileOut{nullptr, dx_pad, Hp, nullptr, R, R, F_in, inpad};
      TRY(run_tile(f, o, st, "norm0 backward"));
      if (l == 0 && dx && !rc &&
          cudaMemcpy2DAsync(dx, size_t(F_in) * 4, dx_pad, size_t(Hp) * 4, size_t(F_in) * 4, size_t(R),
                            cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        vmb::set_kernel_error("dx copy failed");
        rc = 1;
      }
    }
  }
  before_g_overwrite();   // join: every weight gradient is in `grads` before anything the caller enqueues next
  }  // do_bwd
#undef TRY
  if (rc) return fail("vmb_mla_train: %s", vmb::kernels_last_error());
  return 0;
}
}  // namespace

namespace {
bool train_graph_enabled() {
  static const bool on = [] {
    const char* e = getenv("VMB_TRAIN_GRAPH");
    return !(e && e[0] == '0');
  }();
  return on;
}

// Replays (capturing it first if needed) the graph of one whole step on the trainer's own stream, between two events
// that order it after / before the caller's stream.  Returns 0 on success, 1 on a real error, -1 when the graph path
// cannot be used (the caller falls back to eager launches).
int train_step_graph(vmb_mla_trainer* h, const float* params, float* running, const float* x, const long long* labels,
                     long long batch, float dropout_p, unsigned long long seed, float* grads, float* loss, float* scores,
                     cudaStream_t st) {
  if (!h->gstream) {
    if (cudaStreamCreateWithFlags(&h->gstream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      return -1;
    }
  }
  vmb_mla_trainer::GraphSlot* slot = nullptr;
  for (int i = 0; i < h->n_graphs; ++i) {
    auto& g = h->graphs[i];
    if (g.params == params && g.running == running && g.grads == grads && g.loss == loss && g.scores == scores &&
        g.batch == batch && g.dropout_p == dropout_p)
      slot = &g;
  }
  cudaStream_t gs = h->gstream;
  if (cudaEventRecord(h->ev_in, st) != cudaSuccess || cudaStreamWaitEvent(gs, h->ev_in, 0) != cudaSuccess) return -1;
  if (!slot) {
    const long long l0 = vmb_launch_count();
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError();
      return -1;
    }
    h->capturing = true;
    const int rc = train_phases(kPhaseForward | kPhaseBackward, h, params, running, h->x_stage, h->labels_stage, nullptr,
                                batch, dropout_p, 0, grads, loss, scores, gs);
    h->capturing = false;
    const cudaError_t ce = cudaStreamEndCapture(gs, &graph);
    const int launches = static_cast<int>(vmb_launch_count() - l0);
    vmb::count_launch(-launches);          // nothing has run yet
    if (rc || ce != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      return -1;
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess || !exec) {
      cudaGetLastError();
      return -1;
    }
    const int n_slots = static_cast<int>(sizeof h->graphs / sizeof h->graphs[0]);
    int idx;
    if (h->n_graphs < n_slots) {
      idx = h->n_graphs++;
    } else {
      idx = h->next_graph;
      h->next_graph = (h->next_graph + 1) % n_slots;
      cudaGraphExecDestroy(h->graphs[idx].exec);
    }
    h->graphs[idx] = {params, running, grads, loss, scores, batch, dropout_p, exec, launches};
    slot = &h->graphs[idx];
  }
  const size_t x_bytes = size_t(batch) * h->T * h->emb_in * sizeof(float);
  if (cudaMemcpyAsync(h->x_stage, x, x_bytes, cudaMemcpyDeviceToDevice, gs) != cudaSuccess ||
      cudaMemcpyAsync(h->labels_stage, labels, size_t(batch) * sizeof(long long), cudaMemcpyDeviceToDevice, gs) != cudaSuccess)
    return fail("vmb_mla_train_step: staging copy failed: %s", cudaGetErrorString(cudaGetLastError()));
  set_seed_kernel<<<1, 1, 0, gs>>>(h->seed_dev, seed);
  if (cudaGraphLaunch(slot->exec, gs) != cudaSuccess)
    return fail("vmb_mla_train_step: cudaGraphLaunch failed: %s", cudaGetErrorString(cudaGetLastError()));
  vmb::count_launch(1 + slot->launches);
  if (cudaEventRecord(h->ev_out, gs) != cudaSuccess || cudaStreamWaitEvent(st, h->ev_out, 0) != cudaSuccess)
    return fail("vmb_mla_train_step: cannot join the graph stream: %s", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
}  // namespace

extern "C" {

int vmb_mla_train_step(vmb_mla_trainer_t* h, const float* params, float* running, const float* x,
                       const long long* labels, long long batch, float dropout_p, unsigned long long seed,
                       float* grads, float* loss, float* scores, void* stream) {
  if (!labels) return fail("vmb_mla_train_step: labels are required");
  // The first step of a handle runs eagerly (streams, events and kernel attributes are created on the way); from the
  // second one on the step is a CUDA graph replay.  VMB_TRAIN_GRAPH=0 keeps the eager path.
  if (h && h->eager_steps > 0 && !h->graph_broken && train_graph_enabled() && params && running && x && grads && loss &&
      batch >= 2 && batch <= h->max_batch && dropout_p >= 0.f && dropout_p < 1.f) {
    const int rc = train_step_graph(h, params, running, x, labels, batch, dropout_p, seed, grads, loss, scores,
                                    static_cast<cudaStream_t>(stream));
    if (rc >= 0) return rc;
    h->graph_broken = true;     // fall through to the eager path, now and for the rest of the handle's life
  }
  const int rc = train_phases(kPhaseForward | kPhaseBackward, h, params, running, x, labels, nullptr, batch, dropout_p, seed,
                              grads, loss, scores, stream);
  if (!rc && h) ++h->eager_steps;
  return rc;
}

long long vmb_mla_train_tail_offset(const vmb_mla_trainer_t* h) {
  if (!h) return -1;
  return h->tail_offset;
}

int vmb_mla_train_wait_tail(vmb_mla_trainer_t* h, void* stream) {
  if (!h) return fail("vmb_mla_train_wait_tail: null handle");
  if (!h->ev_tail) return fail("vmb_mla_train_wait_tail: no backward pass has been enqueued on this trainer");
  if (cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), h->ev_tail, 0) != cudaSuccess)
    return fail("vmb_mla_train_wait_tail: cudaStreamWaitEvent failed: %s", cudaGetErrorString(cudaGetLastError()));
  return 0;
}

int vmb_mla_train_forward(vmb_mla_trainer_t* h, const float* params, float* running, const float* x, long long batch,
                          float dropout_p, unsigned long long seed, float* scores, void* stream) {
  if (!scores) return fail("vmb_mla_train_forward: null scores");
  return train_phases(kPhaseForward, h, params, running, x, nullptr, nullptr, batch, dropout_p, seed, nullptr, nullptr,
                      scores, stream);
}

int vmb_mla_train_backward(vmb_mla_trainer_t* h, const float* params, const float* x, const float* dscores,
                           long long batch, float dropout_p, unsigned long long seed, float* grads, void* stream) {
  if (!dscores) return fail("vmb_mla_train_backward: null d(scores)");
  return train_phases(kPhaseBackward, h, params, nullptr, x, nullptr, dscores, batch, dropout_p, seed, grads, nullptr,
                      nullptr, stream);
}

int vmb_mla_train_backward_dx(vmb_mla_trainer_t* h, const float* params, const float* x, const float* dscores,
                              long long batch, float dropout_p, unsigned long long seed, float* grads, float* dx,
                              void* stream) {
  if (!dscores) return fail("vmb_mla_train_backward_dx: null d(scores)");
  if (!dx) return fail("vmb_mla_train_backward_dx: null dx");
  if (h && h->wide)
    return fail("vmb_mla_train_backward_dx: the input gradient is formed only when the padded input width does not "
                "exceed the padded hidden width (the wide first layer runs no dX GEMM)");
  return train_phases(kPhaseBackward, h, params, nullptr, x, nullptr, dscores, batch, dropout_p, seed, grads, nullptr,
                      nullptr, stream, dx);
}

int vmb_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, long long step, float grad_scale,
                  void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq) return fail("vmb_adam_step: null pointer");
  if (n <= 0) return 0;
  if (step < 1) return fail("vmb_adam_step: step counts from 1");
  const float bc1 = 1.f - std::pow(beta1, static_cast<float>(step));
  const float bc2 = 1.f - std::pow(beta2, static_cast<float>(step));
  const unsigned grid = static_cast<unsigned>(std::min<long long>((n + 255) / 256, 148LL * 8));
  adam_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                   eps, weight_decay, bc1, std::sqrt(bc2), grad_scale);
  vmb::count_launch();
  if (vmb::check_launch("adam_kernel")) return fail("vmb_adam_step: %s", vmb::kernels_last_error());
  return 0;
}

}  // extern "C"
