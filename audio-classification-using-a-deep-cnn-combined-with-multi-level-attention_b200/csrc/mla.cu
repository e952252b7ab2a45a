// Multi-level attention head, eval mode, one fused kernel (reference model.py:199-269).
//
//   level l:  h = norm0_l(h_prev);  h = ReLU(BN_T(fc_j(h))) for each fc j          (EmbeddedMapping, :217-222)
//             z = fcv_l(h);  att = softmax_K(BN_T^v(z));  cla = sigmoid(BN_T^f(z))   (AttentionModule,  :236-238;
//             y_l[k] = sum_t cla * att / sum_t att                                    fcv is used twice, fcf never)
//   out = sigmoid(BN_K(fc(concat_l y_l)))                                            (:267-268)
//
// BatchNorm1d(T) on a (B,T,F) tensor normalises per time step (SURVEY F5): in eval mode it is the per-t affine
// a[t]*x + b[t], folded on the host at create time.  The head is 0.17 % of the path's FLOPs and feeds a ranking
// metric, so it runs in fp32 on the CUDA cores: one CTA owns G clips (G*T rows) and keeps every activation in
// shared memory; weights stream from L2 (pre-transposed, zero-padded to 640 columns so the inner loop has no
// guards).  Row reductions (softmax max / sum) are warp-shuffle reductions.
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/vggish_mla_b200.h"
#include <cuda_bf16.h>

#include "kernels.cuh"
#include "mla_internal.cuh"

namespace vmb {
void set_api_error(const char* msg);
}

struct vmb_mla : vmb_head::Handle {};

namespace {
using namespace vmb_head;

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

// dst[r][c] = epi( sum_k src[r][k] * wt[k][c] + bias[c] ),  r < 4*RPT, c < n_out.
// epi: v = a[t]*v + b[t] (if bn) ; ReLU (if relu).  Thread tile: RPT rows x 10 strided columns.
template <int RPT>
__device__ __forceinline__ void dense_layer(const float* __restrict__ src, float* __restrict__ dst, const FcDev& L,
                                            int n_out, int T, bool bn, bool relu) {
  const int tid = threadIdx.x;
  const int ct = tid & (kColThreads - 1);
  const int rg = tid >> 6;
  float acc[RPT][kColsPerThread];
#pragma unroll
  for (int r = 0; r < RPT; ++r)
#pragma unroll
    for (int j = 0; j < kColsPerThread; ++j) acc[r][j] = 0.f;
  const float* xrow = src + rg * RPT * kMaxDim;
  const float* wp = L.wt + ct;
  for (int k = 0; k < L.in; k += 4) {  // `in` is padded to a multiple of 4 with zero rows
    float4 x[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) x[r] = *reinterpret_cast<const float4*>(xrow + r * kMaxDim + k);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      float w[kColsPerThread];
#pragma unroll
      for (int j = 0; j < kColsPerThread; ++j) w[j] = __ldg(wp + size_t(k + kk) * kPad + j * kColThreads);
#pragma unroll
      for (int r = 0; r < RPT; ++r) {
        const float xv = kk == 0 ? x[r].x : kk == 1 ? x[r].y : kk == 2 ? x[r].z : x[r].w;
#pragma unroll
        for (int j = 0; j < kColsPerThread; ++j) acc[r][j] = fmaf(xv, w[j], acc[r][j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < kColsPerThread; ++j) {
    const int c = ct + j * kColThreads;
    if (c < n_out) {
      const float bias = __ldg(L.bias + c);
#pragma unroll
      for (int r = 0; r < RPT; ++r) {
        const int row = rg * RPT + r;
        float v = acc[r][j] + bias;
        if (bn) {
          const int t = row % T;
          v = fmaf(__ldg(L.a + t), v, __ldg(L.b + t));
        }
        if (relu) v = fmaxf(v, 0.f);
        dst[row * kMaxDim + c] = v;
      }
    }
  }
}

// G clips per CTA, T == 10 => rows = 10*G, RPT = rows/4 must be integral: G in {2, 4}.
template <int G>
__global__ void __launch_bounds__(kThreads, 1)
mla_forward_kernel(const HeadDev hd, const float* __restrict__ emb, long long batch, float* __restrict__ out,
                   int ystride) {
  constexpr int kRows = G * 10;
  constexpr int RPT = kRows / 4;
  extern __shared__ float sm[];
  float* P = sm;                          // [kRows][kMaxDim]
  float* Q = P + kRows * kMaxDim;         // [kRows][kMaxDim]
  float* Y = Q + kRows * kMaxDim;         // [G][ystride]  (ystride >= n_levels * K)
  float* rmax = Y + G * ystride;          // [kRows]
  float* rsum = rmax + kRows;             // [kRows]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = hd.T;  // == 10
  const long long clip0 = static_cast<long long>(blockIdx.x) * G;

  // zero both activation buffers: padded columns are multiplied by zero weights and must not hold NaN bits
  for (int i = tid; i < 2 * kRows * kMaxDim; i += kThreads) P[i] = 0.f;
  __syncthreads();

  // ---- load the G x T x emb_in input rows into Q with level-0 norm0 applied; zero-fill missing clips / padding
  {
    const LevelDev& L0 = hd.lvl[0];
    const int in_pad = (hd.emb_in + 3) & ~3;
    for (int i = tid; i < kRows * in_pad; i += kThreads) {
      const int r = i / in_pad, c = i - r * in_pad;
      const long long clip = clip0 + r / T;
      float v = 0.f;
      if (clip < batch && c < hd.emb_in) {
        const int t = r % T;
        v = fmaf(__ldg(L0.n0a + t), __ldg(emb + (clip * T + t) * hd.emb_in + c), __ldg(L0.n0b + t));
      }
      Q[r * kMaxDim + c] = v;
    }
  }
  __syncthreads();

  float* cur = Q;   // holds the current level's input / running activation
  float* oth = P;
  for (int l = 0; l < hd.n_levels; ++l) {
    const LevelDev& L = hd.lvl[l];
    if (l > 0) {
      // norm0 of this level applied in place to the previous level's embedding (no longer needed elsewhere)
      for (int i = tid; i < kRows * hd.hidden; i += kThreads) {
        const int r = i / hd.hidden, c = i - r * hd.hidden;
        const int t = r % T;
        cur[r * kMaxDim + c] = fmaf(__ldg(L.n0a + t), cur[r * kMaxDim + c], __ldg(L.n0b + t));
      }
      __syncthreads();
    }
    for (int j = 0; j < L.n_fc; ++j) {
      dense_layer<RPT>(cur, oth, L.fc[j], hd.hidden, T, true, true);
      __syncthreads();
      float* tmp = cur; cur = oth; oth = tmp;
    }
    // cur = emb_l.  z = fcv(emb_l) -> oth
    dense_layer<RPT>(cur, oth, L.fcv, hd.K, T, false, false);
    __syncthreads();
    // row statistics of softmax over the class axis of BN^v(z)
    for (int r = warp; r < kRows; r += kThreads / 32) {
      const int t = r % T;
      const float a = __ldg(L.av + t), b = __ldg(L.bv + t);
      float m = -INFINITY;
      for (int c = lane; c < hd.K; c += 32) m = fmaxf(m, fmaf(a, oth[r * kMaxDim + c], b));
      m = warp_max(m);
      float s = 0.f;
      for (int c = lane; c < hd.K; c += 32) s += expf(fmaf(a, oth[r * kMaxDim + c], b) - m);
      s = warp_sum(s);
      if (lane == 0) { rmax[r] = m; rsum[r] = s; }
    }
    __syncthreads();
    // y_l[g][k] = sum_t cla*att / sum_t att
    for (int i = tid; i < G * hd.K; i += kThreads) {
      const int g = i / hd.K, k = i - g * hd.K;
      float num = 0.f, den = 0.f;
      for (int t = 0; t < T; ++t) {
        const int r = g * T + t;
        const float z = oth[r * kMaxDim + k];
        const float att = expf(fmaf(__ldg(L.av + t), z, __ldg(L.bv + t)) - rmax[r]) / rsum[r];
        const float cla = 1.f / (1.f + expf(-fmaf(__ldg(L.af + t), z, __ldg(L.bf + t))));
        num = fmaf(cla, att, num);
        den += att;
      }
      Y[g * ystride + l * hd.K + k] = num / den;
    }
    __syncthreads();
  }

  // ---- out = sigmoid(BN_K(fc(concat y)))
  const int kin = hd.n_levels * hd.K;
  for (int c = tid; c < hd.K; c += kThreads) {
    float acc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) acc[g] = 0.f;
    for (int k = 0; k < kin; ++k) {
      const float w = __ldg(hd.fc_wt + size_t(k) * kPad + c);
#pragma unroll
      for (int g = 0; g < G; ++g) acc[g] = fmaf(Y[g * ystride + k], w, acc[g]);
    }
    const float bias = __ldg(hd.fc_bias + c), a = __ldg(hd.out_a + c), b = __ldg(hd.out_b + c);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const long long clip = clip0 + g;
      if (clip < batch) out[clip * hd.K + c] = 1.f / (1.f + expf(-fmaf(a, acc[g] + bias, b)));
    }
  }
}

constexpr size_t head_smem_bytes(int G, int ystride) {
  return (size_t(2) * G * 10 * kMaxDim + size_t(G) * ystride + 2 * G * 10) * sizeof(float);
}
constexpr size_t kMaxDynSmem = 227 * 1024;

}  // namespace

namespace {

int fail(const char* msg) {
  vmb::set_api_error(msg);
  return 1;
}

long long param_count(int n_levels, const int* n_fc, int emb_in, int H, int K, int T) {
  long long n = 0;
  for (int l = 0; l < n_levels; ++l) {
    n += 4LL * T;
    for (int j = 0; j < n_fc[l]; ++j) {
      const int in = (l == 0 && j == 0) ? emb_in : H;
      n += 1LL * H * in + H + 4LL * T;
    }
  }
  for (int l = 0; l < n_levels; ++l) n += 1LL * K * H + K + 8LL * T;
  n += 1LL * K * n_levels * K + K + 4LL * K;
  return n;
}

}  // namespace

extern "C" {

long long vmb_mla_param_count(int n_levels, const int* n_fc, int emb_in, int hidden, int n_classes, int t_steps) {
  if (n_levels < 1 || n_levels > kMaxLevels || !n_fc) return -1;
  return param_count(n_levels, n_fc, emb_in, hidden, n_classes, t_steps);
}

int vmb_mla_create(vmb_mla_t** handle, int n_levels, const int* n_fc, int emb_in, int H, int K, int T,
                   const float* params_dev, long long n_params, void* stream) {
  if (!handle || !n_fc || !params_dev) return fail("vmb_mla_create: null argument");
  if (n_levels < 1 || n_levels > kMaxLevels) return fail("vmb_mla_create: 1..4 levels supported");
  for (int l = 0; l < n_levels; ++l)
    if (n_fc[l] < 1 || n_fc[l] > kMaxFc) return fail("vmb_mla_create: 1..4 fully connected layers per level supported");
  if (T != 10) return fail("vmb_mla_create: T must be 10 (params.py:26; BatchNorm1d(T) hard-wires it, model.py:205)");
  if (emb_in < 1 || emb_in > 16384 || H < 1 || H > kMaxDim || K < 1 || K > kMaxDim)
    return fail("vmb_mla_create: hidden and n_classes must be in 1..608, emb_in in 1..16384");
  if (n_params != param_count(n_levels, n_fc, emb_in, H, K, T))
    return fail("vmb_mla_create: n_params does not match the documented flat layout");
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  std::vector<float> p(static_cast<size_t>(n_params));
  if (cudaMemcpyAsync(p.data(), params_dev, p.size() * 4, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail("vmb_mla_create: reading the parameters failed");

  // ---- fold + transpose on the host (float64 arithmetic, one time)
  std::vector<float> blob;
  auto reserve = [&](size_t n) { size_t o = blob.size(); blob.resize(o + ((n + 3) & ~size_t(3)), 0.f); return o; };
  const double eps = 1e-5;  // nn.BatchNorm1d default
  size_t cur = 0;
  auto take = [&](size_t n) { size_t o = cur; cur += n; return p.data() + o; };
  auto fold_bn = [&](int n, size_t& oa, size_t& ob) {
    const float *w = take(n), *b = take(n), *m = take(n), *v = take(n);
    oa = reserve(n);
    ob = reserve(n);
    for (int i = 0; i < n; ++i) {
      const double a = double(w[i]) / std::sqrt(double(v[i]) + eps);
      blob[oa + i] = float(a);
      blob[ob + i] = float(double(b[i]) - double(m[i]) * a);
    }
  };
  std::vector<uint16_t> planes;  // bf16 bits
  auto bf16_split = [](float v, uint16_t* hi, uint16_t* lo) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    *hi = __bfloat16_as_ushort(h);
    *lo = __bfloat16_as_ushort(l);
  };
  size_t cur_planes = 0;
  int cur_kpad = 0;
  // kpad: the contraction length of the weight planes, which is also the row pitch (per plane) of the operand planes
  // the GEMM reads.  The head lays out every activation of hidden width with a pitch of kPad columns (mla_tc.cu), so a
  // Linear fed by one takes kpad = kPad; the head's input and the pooled scores come padded to a multiple of 64.
  auto transpose_w = [&](int n_out, int n_in, int kpad, size_t& owt, size_t& obias) {
    const float* w = take(size_t(n_out) * n_in);
    const float* b = take(n_out);
    const int in_pad = (n_in + 3) & ~3;
    const bool small = n_in <= 4096;   // the transposed fp32 copy feeds the fused fp32 kernel and the output FC
    owt = reserve(small ? size_t(in_pad) * kPad : 4);
    obias = reserve(kPad);
    cur_planes = planes.size();
    cur_kpad = kpad;
    planes.resize(planes.size() + size_t(kPad) * 2 * kpad, 0);
    for (int o = 0; o < n_out; ++o) {
      uint16_t* row = planes.data() + cur_planes + size_t(o) * 2 * kpad;
      for (int i = 0; i < n_in; ++i) {
        const float v = w[size_t(o) * n_in + i];
        if (small) blob[owt + size_t(i) * kPad + o] = v;
        bf16_split(v, row + i, row + kpad + i);
      }
      blob[obias + o] = b[o];
    }
  };
  struct FcOff { size_t wt, bias, a, b; int in; size_t wp; int kpad; };
  struct LvlOff { size_t n0a, n0b; int n_fc; FcOff fc[kMaxFc]; FcOff fcv; size_t av, bv, af, bf; };
  LvlOff lo[kMaxLevels];
  for (int l = 0; l < n_levels; ++l) {
    fold_bn(T, lo[l].n0a, lo[l].n0b);
    lo[l].n_fc = n_fc[l];
    // reference state_dict order inside EmbeddedMapping: norm0, fc.{j}, norms.{j}; the flat layout interleaves
    // (fc j, norm j) as documented in the header
    for (int j = 0; j < n_fc[l]; ++j) {
      const bool first = l == 0 && j == 0;
      const int in = first ? emb_in : H;
      transpose_w(H, in, first ? (in + 63) / 64 * 64 : kPad, lo[l].fc[j].wt, lo[l].fc[j].bias);
      lo[l].fc[j].wp = cur_planes;
      lo[l].fc[j].kpad = cur_kpad;
      fold_bn(T, lo[l].fc[j].a, lo[l].fc[j].b);
      lo[l].fc[j].in = (in + 3) & ~3;
    }
  }
  for (int l = 0; l < n_levels; ++l) {
    transpose_w(K, H, kPad, lo[l].fcv.wt, lo[l].fcv.bias);
    lo[l].fcv.wp = cur_planes;
    lo[l].fcv.kpad = cur_kpad;
    lo[l].fcv.in = (H + 3) & ~3;
    lo[l].fcv.a = lo[l].fcv.b = 0;
    fold_bn(T, lo[l].av, lo[l].bv);
    fold_bn(T, lo[l].af, lo[l].bf);
  }
  size_t fc_wt, fc_bias, out_a, out_b;
  transpose_w(K, n_levels * K, (n_levels * K + 63) / 64 * 64, fc_wt, fc_bias);
  const size_t fc_wp = cur_planes;
  const int fc_kpad = cur_kpad;
  fold_bn(K, out_a, out_b);
  if (cur != p.size()) return fail("vmb_mla_create: internal layout mismatch");

  vmb_mla* h = new vmb_mla();
  cudaGetDevice(&h->device);
  if (cudaMalloc(&h->blob, blob.size() * 4) != cudaSuccess ||
      cudaMalloc(&h->planes, planes.size() * 2) != cudaSuccess ||
      cudaMemcpyAsync(h->blob, blob.data(), blob.size() * 4, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemcpyAsync(h->planes, planes.data(), planes.size() * 2, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess) {
    if (h->blob) cudaFree(h->blob);
    if (h->planes) cudaFree(h->planes);
    delete h;
    return fail("vmb_mla_create: device allocation / upload failed");
  }
  const float* B = h->blob;
  const uint16_t* WP = static_cast<const uint16_t*>(h->planes);
  HeadDev& d = h->dev;
  std::memset(&d, 0, sizeof d);
  d.n_levels = n_levels; d.emb_in = emb_in; d.hidden = H; d.K = K; d.T = T;
  for (int l = 0; l < n_levels; ++l) {
    LevelDev& L = d.lvl[l];
    L.n0a = B + lo[l].n0a; L.n0b = B + lo[l].n0b; L.n_fc = lo[l].n_fc;
    for (int j = 0; j < L.n_fc; ++j)
      L.fc[j] = FcDev{WP + lo[l].fc[j].wp, lo[l].fc[j].kpad, B + lo[l].fc[j].wt, B + lo[l].fc[j].bias,
                      B + lo[l].fc[j].a,   B + lo[l].fc[j].b, lo[l].fc[j].in};
    L.fcv = FcDev{WP + lo[l].fcv.wp, lo[l].fcv.kpad, B + lo[l].fcv.wt, B + lo[l].fcv.bias, nullptr, nullptr, lo[l].fcv.in};
    L.av = B + lo[l].av; L.bv = B + lo[l].bv; L.af = B + lo[l].af; L.bf = B + lo[l].bf;
  }
  d.fc_wp = WP + fc_wp; d.fc_kpad = fc_kpad;
  d.fc_wt = B + fc_wt; d.fc_bias = B + fc_bias; d.out_a = B + out_a; d.out_b = B + out_b;
  *handle = h;
  return 0;
}

int vmb_mla_num_classes(const vmb_mla_t* h) { return h ? h->dev.K : -1; }

void vmb_mla_destroy(vmb_mla_t* h) {
  if (!h) return;
  if (h->side) {
    cudaStreamSynchronize(h->side);
    cudaStreamDestroy(h->side);
  }
  for (int i = 0; i < kMaxLevels; ++i) {
    if (h->fork_ev[i]) cudaEventDestroy(h->fork_ev[i]);
    if (h->gemm_ev[i]) cudaEventDestroy(h->gemm_ev[i]);
    if (h->join_ev[i]) cudaEventDestroy(h->join_ev[i]);
  }
  if (h->blob) cudaFree(h->blob);
  if (h->planes) cudaFree(h->planes);
  delete h;
}

int vmb_mla_forward(vmb_mla_t* h, const float* emb, long long batch, float* scores, void* stream) {
  if (!h) return fail("vmb_mla_forward: null handle");
  if (batch < 0) return fail("vmb_mla_forward: negative batch");
  if (batch == 0) return 0;
  if (!emb || !scores) return fail("vmb_mla_forward: null pointer");
  if (batch > 200000000LL) return fail("vmb_mla_forward: batch too large for one call");
  if (vmb_head::tc_forward(*h, emb, batch, scores, static_cast<cudaStream_t>(stream)))
    return fail(vmb::kernels_last_error());
  return 0;
}

int vmb_mla_fuse_enable(int on) { return vmb_head::mla_fuse_set(on); }

int vmb_mla_embedded_mapping(vmb_mla_t* h, int level, const float* x, long long batch, float* out, void* stream) {
  if (!h) return fail("vmb_mla_embedded_mapping: null handle");
  if (level < 0 || level >= h->dev.n_levels) return fail("vmb_mla_embedded_mapping: no such level");
  if (batch < 0) return fail("vmb_mla_embedded_mapping: negative batch");
  if (batch == 0) return 0;
  if (!x || !out) return fail("vmb_mla_embedded_mapping: null pointer");
  if (vmb_head::tc_embedded_mapping(*h, level, x, batch, out, static_cast<cudaStream_t>(stream)))
    return fail(vmb::kernels_last_error());
  return 0;
}

int vmb_mla_attention(vmb_mla_t* h, int level, const float* hemb, long long batch, float* y, void* stream) {
  if (!h) return fail("vmb_mla_attention: null handle");
  if (level < 0 || level >= h->dev.n_levels) return fail("vmb_mla_attention: no such level");
  if (batch < 0) return fail("vmb_mla_attention: negative batch");
  if (batch == 0) return 0;
  if (!hemb || !y) return fail("vmb_mla_attention: null pointer");
  if (vmb_head::tc_attention(*h, level, hemb, batch, y, static_cast<cudaStream_t>(stream)))
    return fail(vmb::kernels_last_error());
  return 0;
}

int vmb_mla_forward_fp32(vmb_mla_t* h, const float* emb, long long batch, float* scores, void* stream) {
  if (!h) return fail("vmb_mla_forward_fp32: null handle");
  if (batch < 0) return fail("vmb_mla_forward_fp32: negative batch");
  if (batch == 0) return 0;
  if (!emb || !scores) return fail("vmb_mla_forward_fp32: null pointer");
  if (h->dev.emb_in > kMaxDim) return fail("vmb_mla_forward_fp32: emb_in > 608 is only supported by vmb_mla_forward");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ystride = (h->dev.n_levels * h->dev.K + 3) & ~3;
  static std::atomic<unsigned long long> attr_done{0};   // one bit per device: the attribute is per device
  if (vmb::device_needs_setup(attr_done)) {
    if (cudaFuncSetAttribute(mla_forward_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             int(kMaxDynSmem)) != cudaSuccess ||
        cudaFuncSetAttribute(mla_forward_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             int(kMaxDynSmem)) != cudaSuccess)
    {
      vmb::device_setup_failed(attr_done);
      return fail("vmb_mla_forward_fp32: cannot raise the dynamic shared memory limit");
    }
  }
  // small batches: 2 clips per CTA so more SMs take part; large batches: 4 clips per CTA (half the weight traffic)
  if (batch <= 2 * 148 || head_smem_bytes(4, ystride) > kMaxDynSmem) {
    const unsigned grid = static_cast<unsigned>((batch + 1) / 2);
    mla_forward_kernel<2><<<grid, kThreads, head_smem_bytes(2, ystride), st>>>(h->dev, emb, batch, scores, ystride);
  } else {
    const unsigned grid = static_cast<unsigned>((batch + 3) / 4);
    mla_forward_kernel<4><<<grid, kThreads, head_smem_bytes(4, ystride), st>>>(h->dev, emb, batch, scores, ystride);
  }
  vmb::count_launch();
  if (vmb::check_launch("mla_forward_kernel")) return fail(vmb::kernels_last_error());
  return 0;
}

}  // extern "C"
