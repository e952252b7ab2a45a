// fp32-equivalent GEMM from bf16 operand planes on tcgen05 (the Linear layers of the attention head and of its
// training step: reference model.py:217-222, :235-242, :258-269 and their autograd transposes, train.py:130-138).
//
//   out[M][N] (+)= sum over plane pairs (pa, pb), pa + pb <= PLANES - 1, of  A_pa[M][K] * B_pb[N][K]^T   (+ bias)
//
// A is stored as bf16 [M][PLANES * K] (the planes hi | (mid |) lo of every row side by side), B likewise [N][PLANES * K].
// igemm_bf16_kernel runs the same contraction as ONE long K loop over the plane pairs, which loads every plane K-block
// once per product it takes part in: 6 x 32 KB per 64 columns of K for PLANES = 3, twice the 96 KB that are distinct,
// and the kernel is bound by exactly that L2 -> shared memory traffic (ncu: 41 us for a 5120 x 640 x 640 GEMM whose
// MMAs take 8 us per tile).  Here a pipeline stage holds ALL planes of one 32-column K-block of A and of B (SWIZZLE_64B
// rows of 64 bytes: 48 KB per stage for three planes, four stages; 32 KB and six stages for two) and the MMA warp issues
// every plane product from it, so each operand byte crosses L2 -> shared memory once per tile.
//
// Two TMEM accumulators per tile: the hi * hi product goes to one, the small cross products to the other, and the
// epilogue adds them in fp32.  tcgen05.mma truncates when it aligns an addend to the accumulator, so small products
// added into a large running sum would lose their low bits on every K step; kept apart they are accumulated among
// themselves (the order the long-K-loop kernel had: small products first) whatever the K-block interleaving.
//
// Warp roles as in igemm_bf16_kernel: warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2-9 epilogue (two
// per TMEM lane quarter, alternating 32-column chunks).  Persistent over tiles; both accumulators double-buffered
// (2 x 2 x 128 = 512 TMEM columns).  Split-K (the weight-gradient GEMMs: a few output tiles, K = batch * T rows): tile
// index = (K slice, m tile, n tile), partial sums added with 16-byte vector reductions into a zeroed output.
//
// Fused epilogue of the eval-mode head (PlanesEpi, EPI = 1): what used to be a separate pass over the fp32 GEMM output
// — BatchNorm1d(T) as a per-time-step affine + ReLU + the hi | lo split that feeds the next Linear (model.py:219-221) —
// is applied to the accumulator row each epilogue thread already holds, with the same expressions in the same order as
// rows_affine_split_kernel (mla_tc.cu), so the results are bit-identical to the unfused chain.  (A second mode that
// applied BatchNorm1d(K) + sigmoid in the output Linear's epilogue was measured slower than the separate 4 us pass —
// ten CTAs writing unaligned 527-float rows with scalar stores — and removed.)
#include <atomic>
#include <cstdio>
#include <cstdlib>

#include "igemm_sm100.cuh"
#include "kernels.cuh"
#include "sm100_ptx.cuh"

namespace vmb {

namespace {

constexpr int kBM = 128, kBK = 32;
constexpr int kPlaneBytes = 128 * kBK * 2;   // one plane of one K-block of A: 128 rows x 64 bytes = 8 KB
constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreads = 64 + kEpiThreads;
constexpr int kMaxStatChannels = 16;         // BatchNorm1d(T) channels the statistics epilogue can carry (T = 10)

// BN = 128, or 64 when 128-wide tiles would leave most of the last wave idle (head training: 5120 x 640 outputs are 200
// tiles of 128 x 128 on 148 SMs — two waves, the second a third full — but 400 tiles of 128 x 64 — 2.7 waves of half the
// work each; the narrower MMA re-reads A from shared memory twice as often per flop, which costs less than the idle SMs).
template <int PLANES, int BN>
struct PCfg {
  static constexpr int kBPlaneBytes = BN * kBK * 2;                      // one plane of one K-block of B
  static constexpr int kStageBytes = PLANES * (kPlaneBytes + kBPlaneBytes);   // A planes, then B planes
  static constexpr int kStages = 192 * 1024 / kStageBytes;               // 4 / 5 (three planes), 6 / 8 (two)
  static constexpr int kBiasBytes = 2 * BN * 4;
  static constexpr int kBarBytes = (2 * kStages + 4) * 8 + 16;
  // statistics epilogue: {sum, sum of squares} per channel + a flag, and two buffers of per-thread partial sums
  static constexpr int kStatBytes = kMaxStatChannels * 2 * 8 + 16 + 2 * kEpiThreads * 2 * 8;
  static constexpr int kSmemBytes = 1024 + kStages * kStageBytes + kBiasBytes + kBarBytes + kStatBytes;
  static constexpr int kTmemCols = 4 * BN;                               // 2 buffers x (hi*hi | cross products) x BN
};

struct PlanesParams {
  int M, N;
  int num_kb;        // K / 32 (of one plane)
  int a_plane_cols, b_plane_cols;   // MN-major operands: padded width of one plane of A / B
  int num_m_tiles, num_n_tiles;
  int ksplit;        // <= 1: none
  int relu;
  long long ldo;
  const float* bias;
  float* out;
  PlanesEpi epi;     // EPI == 1 only
  PlanesStats stats; // EPI == 3 only
  PlanesGradStats gs; // EPI == 4 only
};

// hi | lo bf16 split of 32 consecutive values of one row -> two 64-byte runs (full 32-byte sectors)
__device__ __forceinline__ void store_split32(const float (&v)[32], __nv_bfloat16* hi_dst, __nv_bfloat16* lo_dst) {
  uint32_t h[16], l[16];
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v[j]), h1 = __float2bfloat16_rn(v[j + 1]);
    const __nv_bfloat16 l0 = __float2bfloat16_rn(v[j] - __bfloat162float(h0));
    const __nv_bfloat16 l1 = __float2bfloat16_rn(v[j + 1] - __bfloat162float(h1));
    h[j / 2] = __bfloat16_as_ushort(h0) | (uint32_t(__bfloat16_as_ushort(h1)) << 16);
    l[j / 2] = __bfloat16_as_ushort(l0) | (uint32_t(__bfloat16_as_ushort(l1)) << 16);
  }
  st_global_256(hi_dst, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7]);
  st_global_256(hi_dst + 16, h[8], h[9], h[10], h[11], h[12], h[13], h[14], h[15]);
  st_global_256(lo_dst, l[0], l[1], l[2], l[3], l[4], l[5], l[6], l[7]);
  st_global_256(lo_dst + 16, l[8], l[9], l[10], l[11], l[12], l[13], l[14], l[15]);
}

template <int PLANES, bool ATOMIC, int EPI, int BN, bool MNMAJOR>
__global__ void __launch_bounds__(kThreads, 1)
planes_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const PlanesParams p) {
  using C = PCfg<PLANES, BN>;
  constexpr int kBN = BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* bias_s = reinterpret_cast<float*>(smem + C::kStages * C::kStageBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes + C::kBiasBytes);
  uint64_t* empty_bar = full_bar + C::kStages;
  uint64_t* tmem_full = empty_bar + C::kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  double* stat_s = reinterpret_cast<double*>(smem + C::kStages * C::kStageBytes + C::kBiasBytes + C::kBarBytes);
  int* last_flag = reinterpret_cast<int*>(stat_s + 2 * kMaxStatChannels);
  double* part_s = stat_s + 2 * kMaxStatChannels + 2;   // [2][kEpiThreads][2]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int mn_tiles = p.num_m_tiles * p.num_n_tiles;
  const int ksplit = p.ksplit > 1 ? p.ksplit : 1;
  const int num_tiles = mn_tiles * ksplit;

  pdl_launch_dependents();
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], kEpiWarps);
    }
    mbar_fence_init();
  }
  if (EPI >= 3 && threadIdx.x < 2 * kMaxStatChannels) stat_s[threadIdx.x] = 0.0;
  if (warp == 1) tmem_alloc(tmem_slot, C::kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      const int plane_cols = p.num_kb * kBK;   // K of one plane
      uint32_t stage = 0, phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int ks = tile / mn_tiles;
        const int mn = tile - ks * mn_tiles;
        const int kb0 = p.num_kb * ks / ksplit, kb1 = p.num_kb * (ks + 1) / ksplit;
        const int m_tile = mn / p.num_n_tiles;
        const int n_tile = mn - m_tile * p.num_n_tiles;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* dst = smem + stage * C::kStageBytes;
          mbar_expect_tx(&full_bar[stage], C::kStageBytes);
          if (MNMAJOR) {
            // operands stored [K rows][planes * width]: a plane tile is two boxes of {64 elements along M / N, 32 rows}
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl)
#pragma unroll
              for (int hh = 0; hh < kBM / 64; ++hh)
                tma_load_2d(dst + pl * kPlaneBytes + hh * (64 * kBK * 2), &tmap_a, &full_bar[stage],
                            pl * p.a_plane_cols + m_tile * kBM + hh * 64, kb * kBK);
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl)
#pragma unroll
              for (int hh = 0; hh < kBN / 64; ++hh)
                tma_load_2d(dst + PLANES * kPlaneBytes + pl * C::kBPlaneBytes + hh * (64 * kBK * 2), &tmap_b, &full_bar[stage],
                            pl * p.b_plane_cols + n_tile * kBN + hh * 64, kb * kBK);
          } else {
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl)
              tma_load_2d(dst + pl * kPlaneBytes, &tmap_a, &full_bar[stage], pl * plane_cols + kb * kBK, m_tile * kBM);
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl)
              tma_load_2d(dst + PLANES * kPlaneBytes + pl * C::kBPlaneBytes, &tmap_b, &full_bar[stage],
                          pl * plane_cols + kb * kBK, n_tile * kBN);
          }
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc =
        umma_idesc_bf16_f32(kBM, kBN) | (MNMAJOR ? (kUmmaIdescAMnMajor | kUmmaIdescBMnMajor) : 0u);
    constexpr uint32_t kBoxBytes = 64 * kBK * 2;       // MN-major: one box of 64 elements x 32 rows
    constexpr uint32_t kStep = MNMAJOR ? (16 * 128) >> 4 : 2;   // descriptor advance per 16-element K step
    // cross products (a plane, b plane), smallest magnitude first; hi * hi has its own accumulator
    constexpr int kCross = PLANES == 3 ? 5 : 2;
    constexpr int cross_a3[5] = {2, 1, 0, 1, 0}, cross_b3[5] = {0, 1, 2, 0, 1};
    constexpr int cross_a2[2] = {1, 0}, cross_b2[2] = {0, 1};
    uint32_t stage = 0, phase = 0, it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      const int ks = tile / mn_tiles;
      const int kb0 = p.num_kb * ks / ksplit, kb1 = p.num_kb * (ks + 1) / ksplit;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after_sync();
      const uint32_t d_big = tmem_base + acc * (2 * kBN);
      const uint32_t d_small = d_big + kBN;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t a0 = smem_u32(smem + stage * C::kStageBytes);
          const uint32_t b0 = a0 + PLANES * kPlaneBytes;
          const uint32_t first = static_cast<uint32_t>(kb - kb0);
#pragma unroll
          for (int q = 0; q < kCross; ++q) {
            const int pa = PLANES == 3 ? cross_a3[q] : cross_a2[q];
            const int pb = PLANES == 3 ? cross_b3[q] : cross_b2[q];
            const uint64_t a_desc = MNMAJOR ? umma_desc_mnmajor_sw128(a0 + pa * kPlaneBytes, kBoxBytes)
                                            : umma_desc_kmajor_sw64(a0 + pa * kPlaneBytes);
            const uint64_t b_desc = MNMAJOR ? umma_desc_mnmajor_sw128(b0 + pb * C::kBPlaneBytes, kBoxBytes)
                                            : umma_desc_kmajor_sw64(b0 + pb * C::kBPlaneBytes);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)   // K-major: +32 bytes per 16-element K step; MN-major: +16 rows of 128 bytes
              umma_bf16_ss(d_small, a_desc + kStep * k, b_desc + kStep * k, idesc, (first | q | k) != 0);
          }
          {
            const uint64_t a_desc = MNMAJOR ? umma_desc_mnmajor_sw128(a0, kBoxBytes) : umma_desc_kmajor_sw64(a0);
            const uint64_t b_desc = MNMAJOR ? umma_desc_mnmajor_sw128(b0, kBoxBytes) : umma_desc_kmajor_sw64(b0);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)
              umma_bf16_ss(d_big, a_desc + kStep * k, b_desc + kStep * k, idesc, (first | k) != 0);
          }
          umma_commit(&empty_bar[stage]);
          if (kb == kb1 - 1) umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
        if (++stage == C::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..9)
    const int q = warp & 3;              // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;    // the two warps of a quarter alternate over the 32-column chunks
    const int ep_tid = threadIdx.x - 64;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int ks = tile / mn_tiles;
      const int mn = tile - ks * mn_tiles;
      const int m_tile = mn / p.num_n_tiles;
      const int n_tile = mn - m_tile * p.num_n_tiles;
      const int n0 = n_tile * kBN;
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      float* bias_t = bias_s + acc * kBN;
      for (int i = ep_tid; i < kBN; i += kEpiThreads) bias_t[i] = (p.bias && ks == 0) ? __ldg(p.bias + n0 + i) : 0.f;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after_sync();
      const int row = m_tile * kBM + q * 32 + lane;
      const bool valid = row < p.M;
      float* out_row = p.out + static_cast<size_t>(row) * p.ldo + n0;
      float s1 = 1.f, o1 = 0.f, s2 = 1.f, o2 = 0.f;
      if (EPI == 4 && valid) {   // s1 = mean_t, o1 = rstd_t, s2 = gamma_t, o2 = beta_t of the block being differentiated
        const int t = row % p.gs.T;
        s1 = __ldg(p.gs.stat + 2 * t);
        o1 = __ldg(p.gs.stat + 2 * t + 1);
        s2 = __ldg(p.gs.gamma + t);
        o2 = __ldg(p.gs.beta + t);
      }
      if (EPI == 1 && valid) {
        const int t = row % p.epi.T;
        if (p.epi.a1) { s1 = __ldg(p.epi.a1 + t); o1 = __ldg(p.epi.b1 + t); }
        if (p.epi.a2) { s2 = __ldg(p.epi.a2 + t); o2 = __ldg(p.epi.b2 + t); }
      }
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * (2 * kBN);
      // EPI == 3: this row's sum / sum of squares over the 64 columns this thread sees of the tile (fp32: 64 terms of
      // similar size; everything above that level is added in double)
      float st1 = 0.f, st2 = 0.f;
#pragma unroll 1
      for (int ch = half; ch < kBN / 32; ch += 2) {
        uint32_t big[32], small[32];
        tmem_ld_32x32(t_addr + ch * 32, big);
        tmem_ld_32x32(t_addr + kBN + ch * 32, small);
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(bias_t + ch * 32 + j);
          f[j + 0] = (__uint_as_float(big[j + 0]) + __uint_as_float(small[j + 0])) + b4.x;
          f[j + 1] = (__uint_as_float(big[j + 1]) + __uint_as_float(small[j + 1])) + b4.y;
          f[j + 2] = (__uint_as_float(big[j + 2]) + __uint_as_float(small[j + 2])) + b4.z;
          f[j + 3] = (__uint_as_float(big[j + 3]) + __uint_as_float(small[j + 3])) + b4.w;
        }
        if (!ATOMIC && p.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        if (EPI == 3 && valid) {
          const int c0 = n0 + ch * 32;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (c0 + j < p.stats.cols) {
              st1 += f[j];
              st2 = fmaf(f[j], f[j], st2);
            }
        }
        if (EPI == 4 && valid) {
          const int c0 = n0 + ch * 32;
          const float* urow = p.gs.u + static_cast<size_t>(row) * p.gs.ldu + c0;
          const unsigned long long seed = p.gs.p > 0.f ? __ldg(p.gs.seed) : 0ull;
          const unsigned long long e0 = static_cast<unsigned long long>(row) * p.gs.F + c0;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (c0 + j < p.gs.cols) {   // cols is a multiple of 4 or the row is padded: u rows are 16-byte aligned
              const float4 u4 = __ldg(reinterpret_cast<const float4*>(urow + j));
              const float uu[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4) {
                if (c0 + j + q4 < p.gs.cols) {
                  const float xh = (uu[q4] - s1) * o1;
                  float g = f[j + q4] * dropout_scale(seed, p.gs.layer, e0 + j + q4, p.gs.p);
                  if (p.gs.relu && fmaf(s2, xh, o2) <= 0.f) g = 0.f;
                  st1 += g;
                  st2 = fmaf(g, xh, st2);
                }
              }
            }
          }
        }
        if (EPI == 1) {
          // h = relu?(a1_t u + b1_t) as hi | lo planes; with dst2 also a2_t h + b2_t (the next level's norm0).  Columns
          // past `cols` are the zero padding of the next GEMM's K.
          if (valid) {
            const int c0 = n0 + ch * 32;
            float x[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float t = fmaf(s1, f[j], o1);
              if (p.epi.relu) t = fmaxf(t, 0.f);
              x[j] = c0 + j < p.epi.cols ? t : 0.f;
            }
            __nv_bfloat16* d = static_cast<__nv_bfloat16*>(p.epi.dst) + static_cast<size_t>(row) * (2 * p.epi.cpad) + c0;
            if (p.epi.dst2) {
              float y[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) y[j] = c0 + j < p.epi.cols ? fmaf(s2, x[j], o2) : 0.f;
              __nv_bfloat16* d2 =
                  static_cast<__nv_bfloat16*>(p.epi.dst2) + static_cast<size_t>(row) * (2 * p.epi.cpad) + c0;
              store_split32(x, d, d + p.epi.cpad);
              store_split32(y, d2, d2 + p.epi.cpad);
            } else {
              store_split32(x, d, d + p.epi.cpad);
            }
          }
        } else if (valid) {
          float* dst = out_row + ch * 32;
          if (ATOMIC) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              asm volatile("red.global.v4.f32.add [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(f[j]), "f"(f[j + 1]),
                           "f"(f[j + 2]), "f"(f[j + 3])
                           : "memory");
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              st_global_256(dst + j, __float_as_uint(f[j]), __float_as_uint(f[j + 1]), __float_as_uint(f[j + 2]),
                            __float_as_uint(f[j + 3]), __float_as_uint(f[j + 4]), __float_as_uint(f[j + 5]),
                            __float_as_uint(f[j + 6]), __float_as_uint(f[j + 7]));
          }
        }
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (EPI >= 3) {
        // Per-channel sums without atomics: every thread leaves its row's partial sums in shared memory (the two warps
        // of a lane quarter hold the two halves of a row's columns), then thread (t, j) adds the rows of the tile whose
        // time step is t.  Two buffers, so one named barrier per tile is enough: a buffer is rewritten two tiles later,
        // after the barrier of the tile in between, which the reading thread only reaches when it is done reading.
        double* part = part_s + (it & 1) * (kEpiThreads * 2);
        const int slot = half * kBM + q * 32 + lane;
        part[2 * slot] = valid ? double(st1) : 0.0;
        part[2 * slot + 1] = valid ? double(st2) : 0.0;
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        const int T = EPI == 3 ? p.stats.channels : p.gs.T;
        if (ep_tid < 2 * T) {
          const int t = ep_tid >> 1, j = ep_tid & 1;
          const int first = (t - (m_tile * kBM) % T + T) % T;   // first row of the tile with time step t
          double sum = 0.0;
          for (int i = first; i < kBM; i += T) sum += part[2 * i + j] + part[2 * (kBM + i) + j];
          stat_s[ep_tid] += sum;
        }
      }
    }
    if (EPI == 4) {
      if (ep_tid < 2 * p.gs.T) atomicAdd(p.gs.acc + ep_tid, stat_s[ep_tid]);   // stat_s[i] belongs to thread i
    }
    if (EPI == 3) {
      // BatchNorm statistics of the output (model.py:221 in train mode): this CTA's partial sums go to the global
      // accumulators; the CTA that arrives last turns them into {mean, rstd} and updates the running statistics, exactly
      // as bn_time_stats_kernel does after its own pass over the matrix
      const PlanesStats& j = p.stats;
      if (ep_tid < 2 * j.channels) atomicAdd(j.acc + ep_tid, stat_s[ep_tid]);   // stat_s[i] belongs to thread i
      __threadfence();
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
      if (ep_tid == 0) *last_flag = atomicAdd(j.counter, 1u) == gridDim.x - 1;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
      if (*last_flag) {
        __threadfence();
        for (int c = ep_tid; c < j.channels; c += kEpiThreads) {
          const double mean = __ldcg(j.acc + 2 * c) / j.count;
          double var = __ldcg(j.acc + 2 * c + 1) / j.count - mean * mean;
          if (var < 0) var = 0;
          j.stat[2 * c] = static_cast<float>(mean);
          j.stat[2 * c + 1] = static_cast<float>(1.0 / sqrt(var + double(j.eps)));
          if (j.run_mean) {
            const double unbiased = j.count > 1 ? var * j.count / (j.count - 1) : var;
            j.run_mean[c] = (1.f - j.momentum) * j.run_mean[c] + j.momentum * static_cast<float>(mean);
            j.run_var[c] = (1.f - j.momentum) * j.run_var[c] + j.momentum * static_cast<float>(unbiased);
          }
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

thread_local char g_perr[384] = "";

template <int PLANES, bool ATOMIC, int EPI = 0, int BN = 128, bool MNMAJOR = false>
int launch_planes(const CUtensorMap& ta, const CUtensorMap& tb, const PlanesParams& p, cudaStream_t stream) {
  auto kern = planes_gemm_kernel<PLANES, ATOMIC, EPI, BN, MNMAJOR>;
  static std::atomic<unsigned long long> attr_set{0};   // one bit per device: the attribute is per device
  constexpr int smem = PCfg<PLANES, BN>::kSmemBytes;
  if (device_needs_setup(attr_set)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) {
      device_setup_failed(attr_set);
      snprintf(g_perr, sizeof g_perr, "planes_gemm: cudaFuncSetAttribute(smem=%d): %s", smem, cudaGetErrorString(e));
      return 1;
    }
  }
  const int tiles = p.num_m_tiles * p.num_n_tiles * (p.ksplit > 1 ? p.ksplit : 1);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  cudaError_t e = launch_pdl(kern, dim3(grid), dim3(kThreads), smem, stream, ta, tb, p);
  count_launch();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_perr, sizeof g_perr, "planes_gemm launch failed: %s", cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

}  // namespace

const char* planes_gemm_last_error() { return g_perr; }

// out fp32 [M][ldo] = act(sum of plane products + bias), or with ksplit > 1 / == -1: out += the K slices' partial sums.
// K % 32 == 0, N % 128 == 0, planes 2 or 3; the operands' rows are planes * K bf16 long.  With epi != nullptr (planes
// == 2, no K split) the epilogue of PlanesEpi::mode replaces the fp32 store.
static int planes_gemm_any(const void* a_planes, const void* b_planes, const float* bias, float* out, long long ldo,
                           int relu, int M, int N, int K, int planes, int ksplit, const PlanesEpi* epi,
                           cudaStream_t stream, const PlanesStats* stats = nullptr, const PlanesGradStats* gs = nullptr) {
  if (M <= 0) return 0;
  if (K % kBK != 0 || N % 128 != 0 || (planes != 2 && planes != 3)) {
    snprintf(g_perr, sizeof g_perr, "planes_gemm: need K %% 32 == 0, N %% 128 == 0, planes 2|3 (K=%d N=%d planes=%d)", K, N,
             planes);
    return 1;
  }
  // fp32 out without a K split: plain stores of one full 32-byte sector per lane and store
  const bool reduce = ksplit > 1 || ksplit == -1;
  if (!epi && !reduce && (ldo % 8 != 0 || (reinterpret_cast<uintptr_t>(out) & 31))) {
    snprintf(g_perr, sizeof g_perr, "planes_gemm: out must be 32-byte aligned and ldo a multiple of 8 floats (ldo=%lld)",
             ldo);
    return 1;
  }
  if (epi) {
    if (planes != 2 || ksplit != 0 || epi->mode != 1 || epi->cols <= 0 || epi->cols > N || !epi->dst || epi->T <= 0 ||
        epi->cpad < N || epi->cpad % 16 != 0 || (epi->a1 && !epi->b1) || (epi->dst2 && (!epi->a2 || !epi->b2)) ||
        (reinterpret_cast<uintptr_t>(epi->dst) & 31) || (reinterpret_cast<uintptr_t>(epi->dst2) & 31)) {
      snprintf(g_perr, sizeof g_perr, "planes_gemm: bad fused-epilogue arguments (mode %d)", epi->mode);
      return 1;
    }
  }
  // Tile width: 128, or 64 (three planes, plain stores or the gradient-statistics epilogue) when that shortens the
  // schedule — whole waves of 148 tiles at one unit of time each against waves of half-width tiles at ~0.6 units (the
  // narrower MMA re-reads A twice as often).  The statistics epilogue keeps 128-wide tiles: its per-tile barrier and
  // partial-sum pass cost more per tile than the fuller last wave gives back.  Measured on the training step: 0.884 ms
  // with 128-wide tiles everywhere, 0.875 ms with 64-wide tiles allowed for plain stores and gradient statistics (this
  // policy), 0.895 ms with the statistics epilogue allowed them as well.
  const int m_tiles = (M + kBM - 1) / kBM;
  int bn = 128;
  if (planes == 3 && !epi && !stats && ksplit == 0) {
    const int sms = num_sms();
    const int t128 = m_tiles * (N / 128);
    const double cost128 = double((t128 + sms - 1) / sms), cost64 = 0.6 * double((2 * t128 + sms - 1) / sms);
    if (cost64 < cost128) bn = 64;
  }
  const int kBN = bn;
  CUtensorMap ta, tb;
  {
    uint64_t dims[2] = {uint64_t(planes) * K, uint64_t(M)};
    uint64_t str[1] = {uint64_t(planes) * K * 2};
    uint32_t box[2] = {kBK, kBM};
    if (make_tmap_bf16(&ta, a_planes, 2, dims, str, box, 64)) {
      snprintf(g_perr, sizeof g_perr, "planes_gemm: %s", igemm_last_error());
      return 1;
    }
  }
  {
    uint64_t dims[2] = {uint64_t(planes) * K, uint64_t(N)};
    uint64_t str[1] = {uint64_t(planes) * K * 2};
    uint32_t box[2] = {kBK, uint32_t(kBN)};
    if (make_tmap_bf16(&tb, b_planes, 2, dims, str, box, 64)) {
      snprintf(g_perr, sizeof g_perr, "planes_gemm: %s", igemm_last_error());
      return 1;
    }
  }
  PlanesParams p{};
  p.M = M;
  p.N = N;
  p.num_kb = K / kBK;
  p.num_m_tiles = m_tiles;
  p.num_n_tiles = N / kBN;
  p.ksplit = ksplit;
  p.relu = relu;
  p.ldo = ldo;
  p.bias = bias;
  p.out = out;
  if (epi) {
    p.epi = *epi;
    return launch_planes<2, false, 1>(ta, tb, p, stream);
  }
  if (gs) {
    p.gs = *gs;
    if (bn == 64) return launch_planes<3, false, 4, 64>(ta, tb, p, stream);
    return planes == 3 ? launch_planes<3, false, 4>(ta, tb, p, stream) : launch_planes<2, false, 4>(ta, tb, p, stream);
  }
  if (stats) {
    if (ksplit != 0 || stats->channels <= 0 || stats->channels > kMaxStatChannels || stats->cols <= 0 || stats->cols > N ||
        !stats->acc || !stats->stat || !stats->counter || (stats->run_mean && !stats->run_var)) {
      snprintf(g_perr, sizeof g_perr, "planes_gemm: bad statistics arguments");
      return 1;
    }
    p.stats = *stats;
    return planes == 3 ? launch_planes<3, false, 3>(ta, tb, p, stream) : launch_planes<2, false, 3>(ta, tb, p, stream);
  }
  if (reduce)
    return planes == 3 ? launch_planes<3, true>(ta, tb, p, stream) : launch_planes<2, true>(ta, tb, p, stream);
  if (bn == 64) return launch_planes<3, false, 0, 64>(ta, tb, p, stream);
  return planes == 3 ? launch_planes<3, false>(ta, tb, p, stream) : launch_planes<2, false>(ta, tb, p, stream);
}

// out [M][ldo] += sum_r A[r][m] B[r][n] over plane products: both operands stored ROW-major over the contraction index,
// a_planes bf16 [K][planes * a_cols], b_planes bf16 [K][planes * b_cols] (the layout the forward / dX GEMMs consume), read
// as MN-major UMMA operands — the weight-gradient GEMMs need no transposed copies of the activations and gradients.
// M <= a_cols, N <= b_cols, both multiples of 128; K % 32 == 0; ksplit > 1 or -1: out is added to; ksplit 0: out is
// overwritten with plain stores (outputs of many tiles and a short contraction, e.g. the 600 x 12288 weight gradient of
// a wide first Linear at up to 1024 rows: 480 tiles of 128 x 128 fill the SMs without a K split).
int planes_gemm_mn(const void* a_planes, int a_cols, const void* b_planes, int b_cols, float* out, long long ldo, int M,
                   int N, int K, int planes, int ksplit, cudaStream_t stream) {
  if (M <= 0) return 0;
  if (K % kBK != 0 || M % 128 != 0 || N % 128 != 0 || M > a_cols || N > b_cols || (planes != 2 && planes != 3) ||
      (ksplit < 0 && ksplit != -1) || ksplit == 1 || ldo < N || !out ||
      (ksplit == 0 && (ldo % 8 || (reinterpret_cast<uintptr_t>(out) & 31)))) {
    snprintf(g_perr, sizeof g_perr, "planes_gemm_mn: bad shape (M=%d N=%d K=%d planes=%d ksplit=%d)", M, N, K, planes, ksplit);
    return 1;
  }
  CUtensorMap ta, tb;
  for (int which = 0; which < 2; ++which) {
    const int cols = which ? b_cols : a_cols;
    uint64_t dims[2] = {uint64_t(planes) * cols, uint64_t(K)};
    uint64_t str[1] = {uint64_t(planes) * cols * 2};
    uint32_t box[2] = {64, kBK};
    if (make_tmap_bf16(which ? &tb : &ta, which ? b_planes : a_planes, 2, dims, str, box, 128)) {
      snprintf(g_perr, sizeof g_perr, "planes_gemm_mn: %s", igemm_last_error());
      return 1;
    }
  }
  PlanesParams p{};
  p.M = M;
  p.N = N;
  p.num_kb = K / kBK;
  p.a_plane_cols = a_cols;
  p.b_plane_cols = b_cols;
  p.num_m_tiles = M / kBM;
  p.num_n_tiles = N / 128;
  p.ksplit = ksplit;
  p.ldo = ldo;
  p.out = out;
  if (ksplit == 0)
    return planes == 3 ? launch_planes<3, false, 0, 128, true>(ta, tb, p, stream)
                       : launch_planes<2, false, 0, 128, true>(ta, tb, p, stream);
  return planes == 3 ? launch_planes<3, true, 0, 128, true>(ta, tb, p, stream)
                     : launch_planes<2, true, 0, 128, true>(ta, tb, p, stream);
}

int planes_gemm_dw(const void* a_planes, int a_cols, const void* b_planes, int b_cols, float* out, long long ldo, int M,
                   int N, int K, int planes, cudaStream_t stream) {
  const int mn = (M / 128) * (N / 128);
  int ks = num_sms() / mn;
  if (ks == 0) ks = (K + kDwSlice - 1) / kDwSlice;
  const bool plain = ks == 1 && mn > num_sms();
  if (ks > K / 32 / 4) ks = K / 32 / 4;
  if (ks < 1) ks = 1;
  if (!plain && cudaMemsetAsync(out, 0, size_t(M) * ldo * sizeof(float), stream) != cudaSuccess) {
    snprintf(g_perr, sizeof g_perr, "planes_gemm_dw: output clear failed");
    return 1;
  }
  return planes_gemm_mn(a_planes, a_cols, b_planes, b_cols, out, ldo, M, N, K, planes, plain ? 0 : ks > 1 ? ks : -1,
                        stream);
}

int planes_gemm(const void* a_planes, const void* b_planes, const float* bias, float* out, long long ldo, int relu, int M,
                int N, int K, int planes, int ksplit, cudaStream_t stream) {
  return planes_gemm_any(a_planes, b_planes, bias, out, ldo, relu, M, N, K, planes, ksplit, nullptr, stream);
}

int planes_gemm_gradstats(const void* a_planes, const void* b_planes, float* out, long long ldo, int M, int N, int K,
                          int planes, const PlanesGradStats& gs, cudaStream_t stream) {
  if (gs.T <= 0 || gs.T > kMaxStatChannels || gs.cols <= 0 || gs.cols > N || !gs.u || !gs.stat || !gs.gamma || !gs.beta ||
      !gs.acc || !gs.seed || gs.ldu % 4 != 0 || (gs.cols + 3) / 4 * 4 > gs.ldu || (reinterpret_cast<uintptr_t>(gs.u) & 15)) {
    snprintf(g_perr, sizeof g_perr, "planes_gemm: bad gradient-statistics arguments");
    return 1;
  }
  return planes_gemm_any(a_planes, b_planes, nullptr, out, ldo, 0, M, N, K, planes, 0, nullptr, stream, nullptr, &gs);
}

int planes_gemm_stats(const void* a_planes, const void* b_planes, const float* bias, float* out, long long ldo, int M,
                      int N, int K, int planes, const PlanesStats& stats, cudaStream_t stream) {
  return planes_gemm_any(a_planes, b_planes, bias, out, ldo, 0, M, N, K, planes, 0, nullptr, stream, &stats);
}

int planes_gemm_fused(const void* a_planes, const void* b_planes, const float* bias, const PlanesEpi& epi, int M, int N,
                      int K, cudaStream_t stream) {
  return planes_gemm_any(a_planes, b_planes, bias, nullptr, 0, 0, M, N, K, 2, 0, &epi, stream);
}

}  // namespace vmb
