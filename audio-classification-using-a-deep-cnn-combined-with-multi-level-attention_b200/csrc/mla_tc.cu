// Multi-level attention head, eval mode, on the tensor cores (reference model.py:199-269).
//
// Every Linear of the head is a split-bf16 tcgen05 GEMM (planes_gemm with two planes: operands carried as hi + lo bf16
// planes, three products, fp32 accumulation — ~16 mantissa bits, so the head adds nothing visible to the ranking
// metric); the glue between GEMMs is three small kernels:
//   rows_affine_split   v = [a2_t * ] relu?(a1_t * u + b1_t) [+ b2_t]  -> hi | lo planes   (BatchNorm1d(T) in eval mode
//                       is a per-time-step affine, SURVEY F5; ReLU; the next level's norm0 folded in)
//   attention_pool      att = softmax_K(BN^v(z)), cla = sigmoid(BN^f(z)), y = sum_t cla att / sum_t att   (model.py:236-240;
//                       fcv feeds both branches, fcf is never used — SURVEY F3; softmax over classes — F4)
//   sigmoid_affine      out = sigmoid(BN_K(fc(concat_l y_l))) after one more split GEMM for fc              (model.py:267-268)
// Row r of every matrix is (clip r / T, time step r % T).
#include <cuda_bf16.h>

#include <algorithm>
#include <atomic>

#include "igemm_sm100.cuh"
#include "kernels.cuh"
#include "mla_internal.cuh"
#include "sm100_ptx.cuh"

namespace vmb_head {

namespace {

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

// src fp32 [rows][lds] (first `cols` columns meaningful) -> dst bf16 [rows][2 * cpad] = hi | lo, zero padded.
// One thread converts 4 consecutive columns.  With dst2 != nullptr the un-normalised h = relu(a1 u + b1) goes to dst
// and a2 h + b2 (the next level's norm0 applied to the same embedding) to dst2: one pass over u for both consumers.
__device__ __forceinline__ void store_split4(const float (&v)[4], __nv_bfloat16* d, int cpad) {
  __nv_bfloat16 hi[4], lo[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    hi[j] = __float2bfloat16_rn(v[j]);
    lo[j] = __float2bfloat16_rn(v[j] - __bfloat162float(hi[j]));
  }
  *reinterpret_cast<uint2*>(d) = make_uint2(
      __bfloat16_as_ushort(hi[0]) | (uint32_t(__bfloat16_as_ushort(hi[1])) << 16),
      __bfloat16_as_ushort(hi[2]) | (uint32_t(__bfloat16_as_ushort(hi[3])) << 16));
  *reinterpret_cast<uint2*>(d + cpad) = make_uint2(
      __bfloat16_as_ushort(lo[0]) | (uint32_t(__bfloat16_as_ushort(lo[1])) << 16),
      __bfloat16_as_ushort(lo[2]) | (uint32_t(__bfloat16_as_ushort(lo[3])) << 16));
}

__global__ void __launch_bounds__(256)
rows_affine_split_kernel(const float* __restrict__ src, long long lds, long long rows, int cols, int cpad, int T,
                         const float* __restrict__ a1, const float* __restrict__ b1, int relu,
                         const float* __restrict__ a2, const float* __restrict__ b2,
                         __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst2) {
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  const int quads = cpad / 4;
  const long long total = rows * quads;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / quads;
    const int c0 = static_cast<int>(i - r * quads) * 4;
    const int t = static_cast<int>(r % T);
    const float s1 = a1 ? __ldg(a1 + t) : 1.f, o1 = a1 ? __ldg(b1 + t) : 0.f;
    const float s2 = a2 ? __ldg(a2 + t) : 1.f, o2 = a2 ? __ldg(b2 + t) : 0.f;
    float h[4], v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float x = 0.f, y = 0.f;
      if (c0 + j < cols) {
        x = fmaf(s1, __ldg(src + r * lds + c0 + j), o1);
        if (relu) x = fmaxf(x, 0.f);
        y = fmaf(s2, x, o2);
      }
      h[j] = x;
      v[j] = y;
    }
    if (dst2) {
      store_split4(h, dst + r * (2LL * cpad) + c0, cpad);
      store_split4(v, dst2 + r * (2LL * cpad) + c0, cpad);
    } else {
      store_split4(v, dst + r * (2LL * cpad) + c0, cpad);
    }
  }
}

// One CTA per clip: z fp32 [T rows][ldz] -> y[clip][col0 + k].  T <= 16.
__global__ void __launch_bounds__(256)
attention_pool_kernel(const float* __restrict__ z, long long ldz, int K, int T, const float* __restrict__ av,
                      const float* __restrict__ bv, const float* __restrict__ af, const float* __restrict__ bf,
                      float* __restrict__ y, long long ystride, int col0) {
  __shared__ float rmax[16], rsum[16];
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  const long long clip = blockIdx.x;
  const float* zc = z + clip * T * ldz;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = warp; t < T; t += 8) {
    const float a = __ldg(av + t), b = __ldg(bv + t);
    float m = -INFINITY;
    for (int c = lane; c < K; c += 32) m = fmaxf(m, fmaf(a, __ldg(zc + t * ldz + c), b));
    m = warp_max(m);
    float s = 0.f;
    for (int c = lane; c < K; c += 32) s += expf(fmaf(a, __ldg(zc + t * ldz + c), b) - m);
    s = warp_sum(s);
    if (lane == 0) { rmax[t] = m; rsum[t] = s; }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float num = 0.f, den = 0.f;
    for (int t = 0; t < T; ++t) {
      const float zz = __ldg(zc + t * ldz + k);
      const float att = expf(fmaf(__ldg(av + t), zz, __ldg(bv + t)) - rmax[t]) / rsum[t];
      const float cla = 1.f / (1.f + expf(-fmaf(__ldg(af + t), zz, __ldg(bf + t))));
      num = fmaf(cla, att, num);
      den += att;
    }
    y[clip * ystride + col0 + k] = num / den;
  }
}

// The same with the clip's z tile staged in shared memory: one coalesced pass over global memory instead of three
// dependent ones, and each exponential evaluated once.  Same expressions in the same order as attention_pool_kernel
// (the att numerators are kept instead of recomputed), so the results are bit-identical to it.
// Dynamic shared memory: 2 * T * kp floats (z and exp(v - max)), kp = K rounded up to 32.
__global__ void __launch_bounds__(256)
attention_pool_smem_kernel(const float* __restrict__ z, long long ldz, int K, int T, const float* __restrict__ av,
                           const float* __restrict__ bv, const float* __restrict__ af, const float* __restrict__ bf,
                           float* __restrict__ y, long long ystride, int col0, __nv_bfloat16* __restrict__ yp, int yp_kpad,
                           int yp_zero_to) {
  extern __shared__ float sm_att[];
  __shared__ float rsum[16];
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  const int kp = (K + 31) & ~31;
  float* sz = sm_att;              // [T][kp] z
  float* se = sm_att + T * kp;     // [T][kp] exp(a z + b - max)
  const long long clip = blockIdx.x;
  const float* zc = z + clip * T * ldz;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = warp; t < T; t += 8) {
    const float a = __ldg(av + t), b = __ldg(bv + t);
    float m = -INFINITY;
    for (int c = lane; c < K; c += 32) {
      const float zz = __ldg(zc + t * ldz + c);
      sz[t * kp + c] = zz;
      m = fmaxf(m, fmaf(a, zz, b));
    }
    m = warp_max(m);
    float s = 0.f;
    for (int c = lane; c < K; c += 32) {
      const float e = expf(fmaf(a, sz[t * kp + c], b) - m);
      se[t * kp + c] = e;
      s += e;
    }
    s = warp_sum(s);
    if (lane == 0) rsum[t] = s;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float num = 0.f, den = 0.f;
    for (int t = 0; t < T; ++t) {
      const float att = se[t * kp + k] / rsum[t];
      const float cla = 1.f / (1.f + expf(-fmaf(__ldg(af + t), sz[t * kp + k], __ldg(bf + t))));
      num = fmaf(cla, att, num);
      den += att;
    }
    const float r = num / den;
    if (y) y[clip * ystride + col0 + k] = r;
    if (yp) {   // the operand planes of the output Linear, written here instead of by a split pass over y
      const __nv_bfloat16 hi = __float2bfloat16_rn(r);
      yp[clip * (2LL * yp_kpad) + col0 + k] = hi;
      yp[clip * (2LL * yp_kpad) + yp_kpad + col0 + k] = __float2bfloat16_rn(r - __bfloat162float(hi));
    }
  }
  // the last level also clears the K padding of the planes (columns col0 + K .. yp_zero_to - 1)
  if (yp)
    for (int k = col0 + K + threadIdx.x; k < yp_zero_to; k += blockDim.x) {
      yp[clip * (2LL * yp_kpad) + k] = __float2bfloat16_rn(0.f);
      yp[clip * (2LL * yp_kpad) + yp_kpad + k] = __float2bfloat16_rn(0.f);
    }
}

// scores[clip][c] = sigmoid(a_c * u[clip][c] + b_c): eval-mode BatchNorm1d(K) + sigmoid on the output Linear (model.py:268)
__global__ void __launch_bounds__(256)
sigmoid_affine_kernel(const float* __restrict__ u, long long ldu, long long batch, int K, const float* __restrict__ oa,
                      const float* __restrict__ ob, float* __restrict__ out) {
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  const long long total = batch * K;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / K;
    const int c = static_cast<int>(i - r * K);
    out[i] = 1.f / (1.f + expf(-fmaf(__ldg(oa + c), __ldg(u + r * ldu + c), __ldg(ob + c))));
  }
}

// out[r][c] = relu?(a_t * u[r][c] + b_t), t = r % T: the fp32 result of an EmbeddedMapping (model.py:217-222) when it is
// asked for on its own rather than consumed by the next GEMM as planes
__global__ void __launch_bounds__(256)
rows_affine_f32_kernel(const float* __restrict__ src, long long lds, long long rows, int cols, int T,
                       const float* __restrict__ a1, const float* __restrict__ b1, int relu, float* __restrict__ dst) {
  vmb::pdl_launch_dependents();
  vmb::pdl_wait();
  const long long total = rows * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i - r * cols);
    const int t = static_cast<int>(r % T);
    float x = fmaf(__ldg(a1 + t), __ldg(src + r * lds + c), __ldg(b1 + t));
    if (relu) x = fmaxf(x, 0.f);
    dst[i] = x;
  }
}

unsigned grid_for(long long items, int per_block) {
  return static_cast<unsigned>(std::min<long long>((items + per_block - 1) / per_block, 148LL * 8));
}

int split_rows(const float* src, long long lds, long long rows, int cols, int cpad, int T, const float* a1,
               const float* b1, int relu, const float* a2, const float* b2, void* dst, cudaStream_t st,
               void* dst2 = nullptr) {
  if (vmb::launch_pdl(rows_affine_split_kernel, dim3(grid_for(rows * (cpad / 4), 256)), dim3(256), 0, st, src, lds, rows,
                      cols, cpad, T, a1, b1, relu, a2, b2, static_cast<__nv_bfloat16*>(dst),
                      static_cast<__nv_bfloat16*>(dst2)) != cudaSuccess) {
    vmb::set_kernel_error("rows_affine_split_kernel: launch failed");
    return 1;
  }
  vmb::count_launch();
  return vmb::check_launch("rows_affine_split_kernel");
}

size_t up(size_t v) { return (v + 1023) / 1024 * 1024; }

}  // namespace

// Fused GEMM epilogues (planes_gemm_fused), on by default; mla_fuse_set(0) keeps the stand-alone affine / split / sigmoid
// passes, the reference of the bit-identity tests.
static std::atomic<int> g_fuse{1};
int mla_fuse_set(int on) { return g_fuse.exchange(on != 0, std::memory_order_relaxed); }

// With more than one level, each level's attention branch but the last runs on the handle's side stream: created on
// first use together with the events that fork and join it.
static int ensure_side_stream(Handle& h) {
  if (h.side) return 0;
  bool ok = cudaStreamCreateWithFlags(&h.side, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < kMaxLevels && ok; ++i)
    ok = cudaEventCreateWithFlags(&h.fork_ev[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&h.gemm_ev[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&h.join_ev[i], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    vmb::set_kernel_error("mla: cannot create the side stream: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  return 0;
}

static int tc_forward_fused(Handle& h, const float* emb, long long batch, float* scores, cudaStream_t st);

int tc_forward(Handle& h, const float* emb, long long batch, float* scores, cudaStream_t st) {
  const HeadDev& d = h.dev;
  const size_t pool_smem = size_t(2) * d.T * ((d.K + 31) & ~31) * sizeof(float);
  if (g_fuse.load(std::memory_order_relaxed) && pool_smem <= 48 * 1024) return tc_forward_fused(h, emb, batch, scores, st);
  const long long rows = batch * d.T;
  if (rows > 0x7fffffffLL) {
    vmb::set_kernel_error("mla: too many rows for one call");
    return 1;
  }
  const int in_pad = d.lvl[0].fc[0].kpad;            // emb_in padded to 64
  const int hpad = kPad;                             // hidden / class width padded to 640
  const int ystride = (d.n_levels * d.K + 3) & ~3;
  // workspace: x planes | two activation plane buffers | normed-input planes | fp32 GEMM output | y
  const size_t sz_x = up(size_t(rows) * 2 * in_pad * 2), sz_p = up(size_t(rows) * 2 * hpad * 2);
  const size_t sz_u = up(size_t(rows) * hpad * 4), sz_y = up(size_t(batch) * ystride * 4);
  const size_t sz_yp = up(size_t(batch) * 2 * d.fc_kpad * 2);
  // The attention branch of a level (z = fcv(emb_l), pooling) does not feed the next level: with more than one level it
  // runs on the handle's side stream, concurrently with the next level's Linear chain (these kernels are 4-22 us each
  // on a fraction of the SMs, so two of them share the GPU).  Needs its own fp32 GEMM output per forked level.
  if (d.n_levels > 1 && ensure_side_stream(h)) return 1;
  const int n_fork = d.n_levels - 1;
  const size_t total = sz_x + 3 * sz_p + (1 + n_fork) * sz_u + sz_y + sz_yp;
  char* ws = nullptr;
  if (cudaMallocAsync(reinterpret_cast<void**>(&ws), total, st) != cudaSuccess) {
    vmb::set_kernel_error("mla: workspace allocation of %zu bytes failed: %s", total,
                          cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  void* X = ws;
  void* P[2] = {ws + sz_x, ws + sz_x + sz_p};
  void* Pn = ws + sz_x + 2 * sz_p;
  float* U = reinterpret_cast<float*>(ws + sz_x + 3 * sz_p);
  float* Y = reinterpret_cast<float*>(ws + sz_x + 3 * sz_p + (1 + n_fork) * sz_u);
  void* Yp = ws + sz_x + 3 * sz_p + (1 + n_fork) * sz_u + sz_y;
  int rc = 0;
  auto gemm_to = [&](const void* a, const FcDev& fc, float* out, cudaStream_t s) {
    if (!rc && vmb::planes_gemm(a, fc.wp, fc.bias, out, hpad, 0, int(rows), hpad, fc.kpad, 2, 0, s)) {
      vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
      rc = 1;
    }
  };
  auto gemm = [&](const void* a, const FcDev& fc) { gemm_to(a, fc, U, st); };
  // level 0 input: norm0 applied to the embeddings
  rc = split_rows(emb, d.emb_in, rows, d.emb_in, in_pad, d.T, d.lvl[0].n0a, d.lvl[0].n0b, 0, nullptr, nullptr, X, st);
  const void* cur = X;
  int pp = 0;
  const void* side_buf[kMaxLevels] = {};   // planes buffer the forked fcv GEMM of level l may still be reading
  for (int l = 0; l < d.n_levels && !rc; ++l) {
    const LevelDev& L = d.lvl[l];
    for (int j = 0; j < L.n_fc && !rc; ++j) {
      gemm(cur, L.fc[j]);
      for (int s = 0; s < l; ++s)
        if (side_buf[s] == P[pp]) {   // the ping-pong comes back to a buffer a forked fcv GEMM reads: wait for that GEMM
          cudaStreamWaitEvent(st, h.gemm_ev[s], 0);
          side_buf[s] = nullptr;
        }
      // h = relu(BN(u)) as planes for the next Linear of this level (or for fcv); after the level's last Linear the
      // same pass also writes the embedding with the next level's norm0 applied
      if (!rc) {
        if (j == L.n_fc - 1 && l + 1 < d.n_levels)
          rc = split_rows(U, hpad, rows, d.hidden, hpad, d.T, L.fc[j].a, L.fc[j].b, 1, d.lvl[l + 1].n0a,
                          d.lvl[l + 1].n0b, P[pp], st, Pn);
        else
          rc = split_rows(U, hpad, rows, d.hidden, hpad, d.T, L.fc[j].a, L.fc[j].b, 1, nullptr, nullptr, P[pp], st);
      }
      cur = P[pp];
      pp ^= 1;
    }
    // attention branch of this level: on the side stream unless it is the last level (nothing left to overlap with)
    const bool side = l + 1 < d.n_levels;
    cudaStream_t as = side ? h.side : st;
    float* Uz = side ? U + (1 + l) * (sz_u / sizeof(float)) : U;
    if (side && !rc) {
      cudaEventRecord(h.fork_ev[l], st);            // emb_l planes (cur) are complete here
      cudaStreamWaitEvent(h.side, h.fork_ev[l], 0);
    }
    gemm_to(cur, L.fcv, Uz, as);   // z = fcv(emb_l)
    if (side) {
      cudaEventRecord(h.gemm_ev[l], h.side);
      side_buf[l] = cur;
    }
    if (!rc) {
      const size_t att_smem = size_t(2) * d.T * ((d.K + 31) & ~31) * sizeof(float);
      if (att_smem <= 48 * 1024)     // K = 527, T = 10: 42 KB
        vmb::launch_pdl(attention_pool_smem_kernel, dim3(static_cast<unsigned>(batch)), dim3(256), att_smem, as, Uz, hpad,
                        d.K, d.T, L.av, L.bv, L.af, L.bf, Y, ystride, l * d.K, static_cast<__nv_bfloat16*>(nullptr), 0, 0);
      else
        vmb::launch_pdl(attention_pool_kernel, dim3(static_cast<unsigned>(batch)), dim3(256), 0, as, Uz, hpad, d.K, d.T,
                        L.av, L.bv, L.af, L.bf, Y, ystride, l * d.K);
      vmb::count_launch();
      rc = vmb::check_launch("attention_pool_kernel");
    }
    if (side) cudaEventRecord(h.join_ev[l], h.side);
    cur = Pn;
  }
  // the concatenated y needs every level's pooling: join the side branches (also on the error path, so that the
  // workspace is not freed under them)
  for (int l = 0; l + 1 < d.n_levels; ++l) cudaStreamWaitEvent(st, h.join_ev[l], 0);
  // out = sigmoid(BN_K(fc(concat y))): y -> planes, one more split GEMM into U ([batch][640]), then the sigmoid
  if (!rc) rc = split_rows(Y, ystride, batch, d.n_levels * d.K, d.fc_kpad, 1, nullptr, nullptr, 0, nullptr, nullptr, Yp, st);
  if (!rc && vmb::planes_gemm(Yp, d.fc_wp, d.fc_bias, U, hpad, 0, int(batch), hpad, d.fc_kpad, 2, 0, st)) {
    vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
    rc = 1;
  }
  if (!rc) {
    vmb::launch_pdl(sigmoid_affine_kernel, dim3(grid_for(batch * d.K, 256)), dim3(256), 0, st, U, hpad, batch, d.K, d.out_a,
                    d.out_b, scores);
    vmb::count_launch();
    rc = vmb::check_launch("sigmoid_affine_kernel");
  }
  cudaFreeAsync(ws, st);
  return rc;
}

// The same forward with the glue folded into the GEMMs: every Linear of an embedding chain writes the next Linear's
// operand planes from its epilogue (BatchNorm1d(T) affine + ReLU + split, and the next level's norm0 for the level's
// last Linear), the pooling kernel writes the output Linear's operand planes; the output Linear's
// BatchNorm1d(K) + sigmoid stays a pass of its own.  10 launches for model_conf [2, 1] instead of 14, no fp32 round trip
// of the hidden activations; each value is computed by the same expressions as in tc_forward above, so the scores are
// bit-identical to it (tested).
static int tc_forward_fused(Handle& h, const float* emb, long long batch, float* scores, cudaStream_t st) {
  const HeadDev& d = h.dev;
  const long long rows = batch * d.T;
  if (rows > 0x7fffffffLL) {
    vmb::set_kernel_error("mla: too many rows for one call");
    return 1;
  }
  const int in_pad = d.lvl[0].fc[0].kpad, hpad = kPad;
  const size_t sz_x = up(size_t(rows) * 2 * in_pad * 2), sz_p = up(size_t(rows) * 2 * hpad * 2);
  const size_t sz_u = up(size_t(rows) * hpad * 4), sz_yp = up(size_t(batch) * 2 * d.fc_kpad * 2);
  if (d.n_levels > 1 && ensure_side_stream(h)) return 1;
  // workspace: x planes | three rotating activation plane buffers | normed-input planes | one fp32 z buffer per level |
  // y planes.  Three buffers, not two: a forked fcv GEMM still reads the level's embedding planes while the next level's
  // chain runs, and with two buffers the second GEMM of that chain would have to wait for it before it may start.
  // Two normed-input buffers alternating by level when there are more than two levels: the only Linear of a middle
  // level reads its input from one while its epilogue writes the next level's input, and the GEMM's tiles are not
  // ordered, so a tile writing in place could overwrite columns that a sibling tile has still to read.
  const int n_pn = d.n_levels > 2 ? 2 : 1;
  const size_t total = sz_x + (3 + n_pn) * sz_p + d.n_levels * sz_u + sz_yp;
  char* ws = nullptr;
  if (cudaMallocAsync(reinterpret_cast<void**>(&ws), total, st) != cudaSuccess) {
    vmb::set_kernel_error("mla: workspace allocation of %zu bytes failed: %s", total,
                          cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  void* X = ws;
  void* P[3] = {ws + sz_x, ws + sz_x + sz_p, ws + sz_x + 2 * sz_p};
  void* Pn[2] = {ws + sz_x + 3 * sz_p, ws + sz_x + (2 + n_pn) * sz_p};   // level l writes level l + 1's input to Pn[l & 1]
  float* U = reinterpret_cast<float*>(ws + sz_x + (3 + n_pn) * sz_p);
  void* Yp = ws + sz_x + (3 + n_pn) * sz_p + d.n_levels * sz_u;
  int rc = split_rows(emb, d.emb_in, rows, d.emb_in, in_pad, d.T, d.lvl[0].n0a, d.lvl[0].n0b, 0, nullptr, nullptr, X, st);
  const void* cur = X;
  int pp = 0;
  const void* side_buf[kMaxLevels] = {};   // planes buffer the forked fcv GEMM of level l may still be reading
  for (int l = 0; l < d.n_levels && !rc; ++l) {
    const LevelDev& L = d.lvl[l];
    for (int j = 0; j < L.n_fc && !rc; ++j) {
      for (int s = 0; s < l; ++s)
        if (side_buf[s] == P[pp]) {   // this GEMM overwrites a buffer a forked fcv GEMM reads: wait for that GEMM
          cudaStreamWaitEvent(st, h.gemm_ev[s], 0);
          side_buf[s] = nullptr;
        }
      vmb::PlanesEpi e{};
      e.mode = 1;
      e.T = d.T;
      e.relu = 1;
      e.cols = d.hidden;
      e.cpad = hpad;
      e.a1 = L.fc[j].a;
      e.b1 = L.fc[j].b;
      e.dst = P[pp];
      if (j == L.n_fc - 1 && l + 1 < d.n_levels) {   // the embedding with the next level's norm0 applied, same pass
        e.a2 = d.lvl[l + 1].n0a;
        e.b2 = d.lvl[l + 1].n0b;
        e.dst2 = Pn[l & 1];
      }
      if (vmb::planes_gemm_fused(cur, L.fc[j].wp, L.fc[j].bias, e, int(rows), hpad, L.fc[j].kpad, st)) {
        vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
        rc = 1;
      }
      cur = P[pp];
      pp = (pp + 1) % 3;
    }
    if (rc) break;
    const bool side = l + 1 < d.n_levels;
    cudaStream_t as = side ? h.side : st;
    float* Uz = U + l * (sz_u / sizeof(float));
    if (side) {
      cudaEventRecord(h.fork_ev[l], st);            // emb_l planes (cur) are complete here
      cudaStreamWaitEvent(h.side, h.fork_ev[l], 0);
    }
    if (vmb::planes_gemm(cur, L.fcv.wp, L.fcv.bias, Uz, hpad, 0, int(rows), hpad, L.fcv.kpad, 2, 0, as)) {   // z = fcv(emb_l)
      vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
      rc = 1;
    }
    if (side) {
      cudaEventRecord(h.gemm_ev[l], h.side);
      side_buf[l] = cur;
    }
    if (!rc) {
      const size_t att_smem = size_t(2) * d.T * ((d.K + 31) & ~31) * sizeof(float);
      const bool last = l + 1 == d.n_levels;
      vmb::launch_pdl(attention_pool_smem_kernel, dim3(static_cast<unsigned>(batch)), dim3(256), att_smem, as, Uz,
                      static_cast<long long>(hpad), d.K, d.T, L.av, L.bv, L.af, L.bf, static_cast<float*>(nullptr), 0LL,
                      l * d.K, static_cast<__nv_bfloat16*>(Yp), d.fc_kpad, last ? d.fc_kpad : 0);
      vmb::count_launch();
      rc = vmb::check_launch("attention_pool_smem_kernel");
    }
    if (side) cudaEventRecord(h.join_ev[l], h.side);
    cur = Pn[l & 1];
  }
  // join the side branches (also on the error path, so that the workspace is not freed under them)
  for (int l = 0; l + 1 < d.n_levels; ++l) cudaStreamWaitEvent(st, h.join_ev[l], 0);
  // The output Linear keeps its separate sigmoid pass: a fused epilogue (planes_gemm mode 2) was measured at 30 us against
  // 12.5 + 3.8 us — ten CTAs each writing 527-float rows with scalar stores lose more than the launch saves.
  if (!rc) {
    float* Uo = U;   // level 0's z buffer is free again: its pooling has been joined
    if (vmb::planes_gemm(Yp, d.fc_wp, d.fc_bias, Uo, hpad, 0, int(batch), hpad, d.fc_kpad, 2, 0, st)) {
      vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
      rc = 1;
    }
    if (!rc) {
      vmb::launch_pdl(sigmoid_affine_kernel, dim3(grid_for(batch * d.K, 256)), dim3(256), 0, st, Uo,
                      static_cast<long long>(hpad), batch, d.K, d.out_a, d.out_b, scores);
      vmb::count_launch();
      rc = vmb::check_launch("sigmoid_affine_kernel");
    }
  }
  cudaFreeAsync(ws, st);
  return rc;
}

// EmbeddedMapping.forward of level `level` on its own (eval mode, model.py:217-222): x fp32 [batch * T][in] ->
// out fp32 [batch * T][hidden] = the level's chain norm0 -> (Linear -> BN_T -> ReLU) x n_fc.  Same kernels and the same
// arithmetic as inside tc_forward.
int tc_embedded_mapping(const Handle& h, int level, const float* x, long long batch, float* out, cudaStream_t st) {
  const HeadDev& d = h.dev;
  const LevelDev& L = d.lvl[level];
  const long long rows = batch * d.T;
  if (rows > 0x7fffffffLL) {
    vmb::set_kernel_error("mla: too many rows for one call");
    return 1;
  }
  const int in_dim = level == 0 ? d.emb_in : d.hidden;
  const int in_pad = L.fc[0].kpad, hpad = kPad;
  const size_t sz_x = up(size_t(rows) * 2 * in_pad * 2), sz_p = up(size_t(rows) * 2 * hpad * 2);
  const size_t sz_u = up(size_t(rows) * hpad * 4);
  char* ws = nullptr;
  if (cudaMallocAsync(reinterpret_cast<void**>(&ws), sz_x + sz_p + sz_u, st) != cudaSuccess) {
    vmb::set_kernel_error("mla: workspace allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  void* X = ws;
  void* P = ws + sz_x;
  float* U = reinterpret_cast<float*>(ws + sz_x + sz_p);
  int rc = split_rows(x, in_dim, rows, in_dim, in_pad, d.T, L.n0a, L.n0b, 0, nullptr, nullptr, X, st);
  const void* cur = X;
  for (int j = 0; j < L.n_fc && !rc; ++j) {
    if (vmb::planes_gemm(cur, L.fc[j].wp, L.fc[j].bias, U, hpad, 0, int(rows), hpad, L.fc[j].kpad, 2, 0, st)) {
      vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
      rc = 1;
      break;
    }
    if (j + 1 < L.n_fc) {
      // the planes buffer is free again: the GEMM that read it (as `cur`) precedes this kernel in the stream
      rc = split_rows(U, hpad, rows, d.hidden, hpad, d.T, L.fc[j].a, L.fc[j].b, 1, nullptr, nullptr, P, st);
      cur = P;
    } else {
      vmb::launch_pdl(rows_affine_f32_kernel, dim3(grid_for(rows * d.hidden, 256)), dim3(256), 0, st, U,
                      static_cast<long long>(hpad), rows, d.hidden, d.T, L.fc[j].a, L.fc[j].b, 1, out);
      vmb::count_launch();
      rc = vmb::check_launch("rows_affine_f32_kernel");
    }
  }
  cudaFreeAsync(ws, st);
  return rc;
}

// AttentionModule.forward of level `level` on its own (eval mode, model.py:235-242): hemb fp32 [batch * T][hidden] ->
// y fp32 [batch][K].
int tc_attention(const Handle& h, int level, const float* hemb, long long batch, float* y, cudaStream_t st) {
  const HeadDev& d = h.dev;
  const LevelDev& L = d.lvl[level];
  const long long rows = batch * d.T;
  if (rows > 0x7fffffffLL) {
    vmb::set_kernel_error("mla: too many rows for one call");
    return 1;
  }
  const int hpad = kPad;
  const size_t sz_p = up(size_t(rows) * 2 * hpad * 2), sz_u = up(size_t(rows) * hpad * 4);
  char* ws = nullptr;
  if (cudaMallocAsync(reinterpret_cast<void**>(&ws), sz_p + sz_u, st) != cudaSuccess) {
    vmb::set_kernel_error("mla: workspace allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  float* U = reinterpret_cast<float*>(ws + sz_p);
  int rc = split_rows(hemb, d.hidden, rows, d.hidden, hpad, d.T, nullptr, nullptr, 0, nullptr, nullptr, ws, st);
  if (!rc && vmb::planes_gemm(ws, L.fcv.wp, L.fcv.bias, U, hpad, 0, int(rows), hpad, L.fcv.kpad, 2, 0, st)) {
    vmb::set_kernel_error("mla: %s", vmb::planes_gemm_last_error());
    rc = 1;
  }
  if (!rc) {
    const size_t att_smem = size_t(2) * d.T * ((d.K + 31) & ~31) * sizeof(float);
    if (att_smem <= 48 * 1024)
      vmb::launch_pdl(attention_pool_smem_kernel, dim3(static_cast<unsigned>(batch)), dim3(256), att_smem, st, U,
                      static_cast<long long>(hpad), d.K, d.T, L.av, L.bv, L.af, L.bf, y, static_cast<long long>(d.K), 0,
                      static_cast<__nv_bfloat16*>(nullptr), 0, 0);
    else
      vmb::launch_pdl(attention_pool_kernel, dim3(static_cast<unsigned>(batch)), dim3(256), 0, st, U,
                      static_cast<long long>(hpad), d.K, d.T, L.av, L.bv, L.af, L.bf, y, static_cast<long long>(d.K), 0);
    vmb::count_launch();
    rc = vmb::check_launch("attention_pool_kernel");
  }
  cudaFreeAsync(ws, st);
  return rc;
}

}  // namespace vmb_head
