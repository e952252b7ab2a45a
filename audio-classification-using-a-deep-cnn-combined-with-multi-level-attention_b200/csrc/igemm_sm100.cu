// tcgen05 implicit-GEMM kernel + host launchers.  See igemm_sm100.cuh for the design notes.
#include "igemm_sm100.cuh"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "kernels.cuh"
#include "sm100_ptx.cuh"

namespace vmb {

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                          // 64 bf16 = one 128-byte swizzle row
constexpr int kABytes = kBlockM * kBlockK * 2;       // 16 KiB
constexpr int kQuarterBytes = 32 * kBlockK * 2;      // one 32-row quarter of A (one TMA box in CONV mode)
constexpr int kEpiWarps = 8;                          // two per TMEM lane quarter (the short-K layers are epilogue-paced)
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kNumThreads = 64 + kEpiThreads;

// MT = number of 128-row sub-tiles per CTA tile that share one B stage (MT = 2 doubles the smem reuse of the
// weights when BLOCK_N is only 128: a 256 x 128 tile moves as many bytes per FLOP as a 128 x 256 one).
// HALO (CONV + BIG, Wb = 16, Hb = 2): a stage holds, per sub-tile, ONE activation box with a one-row halo above and below
// (10 rows x 16 pixels x 64 channels = 20 KB, loaded at column offset dx) plus the three weight tiles of the taps
// (dy = -1, 0, 1; dx).  The three MMAs groups of a stage read the same box at row offsets 0 / 16 / 32 (2 KB apart,
// which keeps the 128-byte swizzle phase), so the activations cross L2 -> shared memory 3 times per tile instead of 9:
// 59 instead of 96 B/clk/SM for conv2, i.e. the same bytes in flight now cover 3 000 cycles of load latency, not 2 000.
constexpr int kHaloRows = 10, kHaloWb = 16;
constexpr int kHaloBytes = kHaloRows * kHaloWb * kBlockK * 2;   // 20480
template <int BLOCK_N, int MT, bool HALO = false>
struct Cfg {
  static constexpr int kBBytes = BLOCK_N * kBlockK * 2;
  static constexpr int kStageBytes = HALO ? MT * kHaloBytes + 3 * kBBytes : MT * kABytes + kBBytes;
  static constexpr int kStages = HALO ? (200 * 1024 / kStageBytes) : ((kStageBytes >= 48 * 1024) ? 4 : 6);
  static_assert(kStages >= 2, "need a double-buffered stage ring");
  static constexpr int kTmemCols = 2 * MT * BLOCK_N;  // two accumulator buffers; 256 or 512 (power of two)
  static_assert(kTmemCols <= 512, "TMEM holds 512 columns");
  static constexpr int kBiasBytes = 2 * BLOCK_N * 4;
  static constexpr int kBarBytes = (2 * kStages + 4) * 8 + 16;
  static constexpr int kSmemBytes = 1024 /*align slack*/ + kStages * kStageBytes + kBiasBytes + kBarBytes;
};

constexpr int kOutBf16 = 0, kOutF32 = 1, kOutSplit = 2, kOutF32Atomic = 3;   // epilogue output: bf16, fp32, hi | lo bf16
                                                                              // planes, or fp32 atomicAdd (split-K)

template <int BLOCK_N, int MT, bool CONV, bool POOL, int OUT, bool BIG = false, bool HALO = false>
__global__ void __launch_bounds__(kNumThreads, 1)
igemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                  const IgemmParams p) {
  static_assert(!HALO || (CONV && BIG && OUT == kOutBf16), "HALO is a variant of the bf16 big-box conv");
  using C = Cfg<BLOCK_N, MT, HALO>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  uint8_t* stage_base = smem;
  float* bias_s = reinterpret_cast<float*>(smem + C::kStages * C::kStageBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes + C::kBiasBytes);
  uint64_t* empty_bar = full_bar + C::kStages;
  uint64_t* tmem_full = empty_bar + C::kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // split-K (PLAIN, kOutF32Atomic): tile index = (k slice, m tile, n tile); every slice adds into the zeroed output
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
      mbar_init(&tmem_empty[s], kEpiWarps);  // one arrival per epilogue warp
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform by construction
  pdl_wait();   // everything above overlapped the previous kernel's tail; global memory is touched only below

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        // split-K is the rare case: keep the divisions out of the ordinary tile loop
        int mn = tile, kb0 = 0, kb1 = p.num_kb;
        if (ksplit > 1) {
          const int ks = tile / mn_tiles;
          mn = tile - ks * mn_tiles;
          kb0 = p.num_kb * ks / ksplit;
          kb1 = p.num_kb * (ks + 1) / ksplit;
        }
        const int m_tile = mn / p.num_n_tiles;
        const int n_tile = mn - m_tile * p.num_n_tiles;
        int bx[4 * MT], by[4 * MT], bn[4 * MT];
        if (CONV && BIG) {
          // one TMA box per 128-pixel sub-tile: Wb columns x 4*Hb rows (its four 32-pixel quarters stacked vertically)
#pragma unroll
          for (int sub = 0; sub < MT; ++sub) {
            const int g = m_tile * MT + sub;
            const int n_img = g / p.boxes_per_img;
            const int r = g - n_img * p.boxes_per_img;
            const int yy = r / p.boxes_per_row;
            bn[sub] = n_img;
            by[sub] = yy * 4 * p.Hb;
            bx[sub] = (r - yy * p.boxes_per_row) * p.Wb;
          }
        } else if (CONV) {
#pragma unroll
          for (int q = 0; q < 4 * MT; ++q) {
            const int g = m_tile * 4 * MT + q;
            const int n_img = g / p.boxes_per_img;
            const int r = g - n_img * p.boxes_per_img;
            const int yy = r / p.boxes_per_row;
            bn[q] = n_img;
            by[q] = yy * p.Hb;
            bx[q] = (r - yy * p.boxes_per_row) * p.Wb;
          }
        }
        if (HALO) {
          for (int s = 0; s < 3 * p.cblks; ++s) {
            const int cbh = s / 3, dxi = s - cbh * 3;
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* a_dst = stage_base + stage * C::kStageBytes;
            uint8_t* b_dst = a_dst + MT * kHaloBytes;
            mbar_expect_tx(&full_bar[stage], C::kStageBytes);
#pragma unroll
            for (int sub = 0; sub < MT; ++sub)
              tma_load_4d(a_dst + sub * kHaloBytes, &tmap_a, &full_bar[stage], cbh * kBlockK, bx[sub] + dxi - 1,
                          by[sub] - 1, bn[sub]);
#pragma unroll
            for (int dyi = 0; dyi < 3; ++dyi)
              tma_load_2d(b_dst + dyi * C::kBBytes, &tmap_b, &full_bar[stage], ((dyi * 3 + dxi) * p.cblks + cbh) * kBlockK,
                          n_tile * BLOCK_N);
            if (++stage == C::kStages) { stage = 0; phase ^= 1; }
          }
          continue;
        }
        // CONV K order: channel block outermost, then dx, then dy — the order the HALO variant needs (its stage is one
        // (channel block, dx) and feeds the three dy taps), used by every bf16 conv kernel so that all of them add the
        // same partial products in the same order (results are bit-identical whichever kernel a batch size selects)
        int tap = 0, cb = 0;   // tap = dxi * 3 + dyi
        int b_conv_kb = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = stage_base + stage * C::kStageBytes;
          uint8_t* b_dst = a_dst + MT * kABytes;
          mbar_expect_tx(&full_bar[stage], C::kStageBytes);
          if (CONV && p.conv_split) {
            // activations [n][2][H][W][C] (hi | lo planes per image), weights [C_out][hi(9 C_in) | lo(9 C_in)]:
            // the K loop runs over the products hi*hi, lo*hi, hi*lo, each over (tap, c_in block)
            const int per = 9 * p.cblks;
            const int prod = kb / per, kk = kb - prod * per;
            const int tp = kk / p.cblks, cbb = kk - tp * p.cblks;
            const int dh = tp / 3 - 1, dw = tp % 3 - 1;
#pragma unroll
            for (int q = 0; q < 4 * MT; ++q)
              tma_load_5d(a_dst + q * kQuarterBytes, &tmap_a, &full_bar[stage], cbb * kBlockK, bx[q] + dw, by[q] + dh,
                          prod == 1 ? 1 : 0, bn[q]);
            tma_load_2d(b_dst, &tmap_b, &full_bar[stage], ((prod == 2 ? per : 0) + kk) * kBlockK, n_tile * BLOCK_N);
            if (++stage == C::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
          if (CONV) {
            const int dxi = tap / 3, dyi = tap - dxi * 3;
            const int dh = dyi - 1, dw = dxi - 1;
            b_conv_kb = (dyi * 3 + dxi) * p.cblks + cb;   // weights are stored [C_out][(kh, kw, c)]
            if (BIG) {
#pragma unroll
              for (int sub = 0; sub < MT; ++sub)
                tma_load_4d(a_dst + sub * kABytes, &tmap_a, &full_bar[stage], cb * kBlockK, bx[sub] + dw,
                            by[sub] + dh, bn[sub]);
            } else {
#pragma unroll
              for (int q = 0; q < 4 * MT; ++q)
                tma_load_4d(a_dst + q * kQuarterBytes, &tmap_a, &full_bar[stage], cb * kBlockK, bx[q] + dw,
                            by[q] + dh, bn[q]);
            }
            if (++tap == 9) { tap = 0; ++cb; }
          } else {
            // split mode (p.split_nkb > 0): A and B are stored as column blocks of 2 (hi | lo) or 3 (hi | mid | lo)
            // bf16 planes and the K loop runs over the products with plane index sum <= planes - 1, smallest first
            // (see igemm_linear_split)
            int a_kb = kb;
            if (p.split_nkb) {
              const int q = kb / p.split_nkb;
              const int pa = p.split_planes == 3 ? ((0x210100 >> (4 * (5 - q))) & 0xF) : (q == 1 ? 1 : 0);
              a_kb = pa * p.split_nkb + (kb - q * p.split_nkb);
            }
#pragma unroll
            for (int sub = 0; sub < MT; ++sub)
              tma_load_2d(a_dst + sub * kABytes, &tmap_a, &full_bar[stage], a_kb * kBlockK,
                          (m_tile * MT + sub) * kBlockM);
          }
          int b_kb = CONV ? b_conv_kb : kb;
          if (p.split_nkb) {
            const int q = kb / p.split_nkb;
            const int pb = p.split_planes == 3 ? ((0x012010 >> (4 * (5 - q))) & 0xF) : (q == 2 ? 1 : 0);
            b_kb = pb * p.split_nkb + (kb - q * p.split_nkb);
          }
          tma_load_2d(b_dst, &tmap_b, &full_bar[stage], b_kb * kBlockK, n_tile * BLOCK_N);
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc = p.f16 ? umma_idesc_f16_f32(kBlockM, BLOCK_N) : umma_idesc_bf16_f32(kBlockM, BLOCK_N);
    uint32_t stage = 0, phase = 0, it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      int kb0 = 0, kb1 = p.num_kb;
      if (ksplit > 1) {
        const int ks = tile / mn_tiles;
        kb0 = p.num_kb * ks / ksplit;
        kb1 = p.num_kb * (ks + 1) / ksplit;
      }
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + acc * (MT * BLOCK_N);
      if (HALO) {
        const int n_st = 3 * p.cblks;
        for (int s = 0; s < n_st; ++s) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          if (elect_one()) {
            const uint32_t a_addr = smem_u32(stage_base + stage * C::kStageBytes);
            const uint32_t b_addr = a_addr + MT * kHaloBytes;
#pragma unroll
            for (int dyi = 0; dyi < 3; ++dyi) {
              const uint64_t b_desc = umma_desc_kmajor_sw128(b_addr + dyi * C::kBBytes);
#pragma unroll
              for (int sub = 0; sub < MT; ++sub) {
                // rows dyi*16 .. dyi*16+127 of the halo box = the 8 x 16 output pixels shifted by dy = dyi - 1
                const uint64_t a_desc = umma_desc_kmajor_sw128(a_addr + sub * kHaloBytes + dyi * (kHaloWb * kBlockK * 2));
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k)
                  umma_bf16_ss(d_tmem + sub * BLOCK_N, a_desc + 2 * k, b_desc + 2 * k, idesc, (s | dyi | k) != 0);
              }
            }
            umma_commit(&empty_bar[stage]);
            if (s == n_st - 1) umma_commit(&tmem_full[acc]);
          }
          __syncwarp();
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        continue;
      }
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after_sync();
        if (elect_one()) {
          const uint32_t a_addr = smem_u32(stage_base + stage * C::kStageBytes);
          const uint64_t b_desc = umma_desc_kmajor_sw128(a_addr + MT * kABytes);
#pragma unroll
          for (int sub = 0; sub < MT; ++sub) {
            const uint64_t a_desc = umma_desc_kmajor_sw128(a_addr + sub * kABytes);
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k)  // +32 bytes (>>4 = 2) per 16-element K step inside the swizzle row
              umma_bf16_ss(d_tmem + sub * BLOCK_N, a_desc + 2 * k, b_desc + 2 * k, idesc, ((kb - kb0) | k) != 0);
          }
          umma_commit(&empty_bar[stage]);
          if (kb == kb1 - 1) umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
        if (++stage == C::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..5)
    // warp w may read TMEM lanes 32*(w%4)..+31; the two warps of a quarter split the tile's sub-tiles (MT = 2) or
    // alternate over its 32-column chunks (MT = 1)
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int ep_tid = threadIdx.x - 64;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      int mn = tile, ks = 0;
      if (ksplit > 1) {
        ks = tile / mn_tiles;
        mn = tile - ks * mn_tiles;
      }
      const int m_tile = mn / p.num_n_tiles;
      const int n_tile = mn - m_tile * p.num_n_tiles;
      const int n0 = n_tile * BLOCK_N;
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      float* bias_t = bias_s + acc * BLOCK_N;
      for (int i = ep_tid; i < BLOCK_N; i += kEpiThreads)
        bias_t[i] = (p.bias && ks == 0) ? __ldg(p.bias + n0 + i) : 0.f;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after_sync();
#pragma unroll 1
      for (int mt = (MT == 2 ? half : 0); mt < (MT == 2 ? half + 1 : 1); ++mt) {
      // Where does this thread's accumulator row go?
      bool valid;
      size_t out_off;  // element offset of column n0 for this thread's output row / pooled pixel
      int sub = 0;
      if (CONV) {
        // quarter q of this sub-tile: its own 32-pixel box, or rows [q*Hb, (q+1)*Hb) of one 128-pixel box
        const int g = BIG ? (m_tile * MT + mt) : (m_tile * MT + mt) * 4 + q;
        const int n_img = g / p.boxes_per_img;
        const int r = g - n_img * p.boxes_per_img;
        const int yy = r / p.boxes_per_row;
        const int hh = lane / p.Wb, ww = lane - hh * p.Wb;
        const int h = BIG ? yy * 4 * p.Hb + q * p.Hb + hh : yy * p.Hb + hh;
        const int w = (r - yy * p.boxes_per_row) * p.Wb + ww;
        valid = n_img < p.M;
        if (POOL) {
          sub = (ww & 1) | ((hh & 1) << 1);
          out_off = static_cast<size_t>(n_img) * p.out_img_stride +
                    (static_cast<size_t>(h >> 1) * (p.W >> 1) + (w >> 1)) * p.N + n0;
        } else {
          out_off = static_cast<size_t>(n_img) * p.out_img_stride + (static_cast<size_t>(h) * p.W + w) * p.N + n0;
        }
      } else {
        const int row = (m_tile * MT + mt) * kBlockM + q * 32 + lane;
        valid = row < p.M;
        out_off = static_cast<size_t>(row) * p.ldo + n0;
      }

      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * (MT * BLOCK_N) + mt * BLOCK_N;
      uint32_t sat_max = 0;   // fp16 mode: running maximum of the packed outputs

#pragma unroll 1
      for (int ch = (MT == 2 ? 0 : half); ch < BLOCK_N / 32; ch += (MT == 2 ? 1 : 2)) {
        uint32_t v[32];
        tmem_ld_32x32(t_addr + ch * 32, v);
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(bias_t + ch * 32 + j);
          f[j + 0] = __uint_as_float(v[j + 0]) + b4.x;
          f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
          f[j + 2] = __uint_as_float(v[j + 2]) + b4.z;
          f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
        }
        if (p.relu && !(OUT == kOutBf16 && POOL)) {   // the pooled bf16 path applies ReLU after the pooling (fewer values)
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        if (OUT == kOutSplit) {
          if (POOL) {
            // pool on the fp32 values (the hi/lo split does not commute with max)
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              f[j] = fmaxf(f[j], __shfl_xor_sync(0xffffffffu, f[j], 1));
              f[j] = fmaxf(f[j], __shfl_xor_sync(0xffffffffu, f[j], p.Wb));
            }
          }
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(f[2 * j], f[2 * j + 1]);
            hi[j] = *reinterpret_cast<const uint32_t*>(&h2);
            lo[j] = pack_bf16x2(f[2 * j] - __low2float(h2), f[2 * j + 1] - __high2float(h2));
          }
          __nv_bfloat16* outp = static_cast<__nv_bfloat16*>(p.out) + out_off + ch * 32;
          if (POOL) {
            // the four lanes of a window share the 32 results: each stores one full 32-byte sector (hi: sub 0/1, lo: sub 2/3)
            const bool up = sub & 1;
            if (valid) {
              if (!(sub & 2))
                st_global_256(outp + (up ? 16 : 0), up ? hi[8] : hi[0], up ? hi[9] : hi[1], up ? hi[10] : hi[2],
                              up ? hi[11] : hi[3], up ? hi[12] : hi[4], up ? hi[13] : hi[5], up ? hi[14] : hi[6],
                              up ? hi[15] : hi[7]);
              else
                st_global_256(outp + p.lo_off + (up ? 16 : 0), up ? lo[8] : lo[0], up ? lo[9] : lo[1],
                              up ? lo[10] : lo[2], up ? lo[11] : lo[3], up ? lo[12] : lo[4], up ? lo[13] : lo[5],
                              up ? lo[14] : lo[6], up ? lo[15] : lo[7]);
            }
          } else if (valid) {
            st_global_256(outp, hi[0], hi[1], hi[2], hi[3], hi[4], hi[5], hi[6], hi[7]);
            st_global_256(outp + 16, hi[8], hi[9], hi[10], hi[11], hi[12], hi[13], hi[14], hi[15]);
            st_global_256(outp + p.lo_off, lo[0], lo[1], lo[2], lo[3], lo[4], lo[5], lo[6], lo[7]);
            st_global_256(outp + p.lo_off + 16, lo[8], lo[9], lo[10], lo[11], lo[12], lo[13], lo[14], lo[15]);
          }
        } else if (OUT == kOutF32Atomic) {
          if (valid) {   // split-K partial sums: 16-byte vector reductions (one L2 request per four columns)
            float* dst = static_cast<float*>(p.out) + out_off + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              asm volatile("red.global.v4.f32.add [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(f[j]), "f"(f[j + 1]),
                           "f"(f[j + 2]), "f"(f[j + 3])
                           : "memory");
          }
        } else if (OUT == kOutF32) {
          if (valid) {
            float* dst = static_cast<float*>(p.out) + out_off + ch * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              st_global_256(dst + j, __float_as_uint(f[j]), __float_as_uint(f[j + 1]), __float_as_uint(f[j + 2]),
                            __float_as_uint(f[j + 3]), __float_as_uint(f[j + 4]), __float_as_uint(f[j + 5]),
                            __float_as_uint(f[j + 6]), __float_as_uint(f[j + 7]));
          }
        } else {
          void* outp = static_cast<uint16_t*>(p.out) + out_off + ch * 32;
          if (p.f16)
            sat_max = max_f16x2(sat_max, store_row32_16bit<true, POOL>(f, sub, p.Wb, p.relu != 0, valid, outp));
          else
            store_row32_16bit<false, POOL>(f, sub, p.Wb, p.relu != 0, valid, outp);
        }
      }
      if (OUT == kOutBf16 && p.f16 && p.sat_flag && saturated_f16x2(sat_max)) *reinterpret_cast<volatile int*>(p.sat_flag) = 1;
      }  // mt
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------- host side
thread_local char g_err[512] = "";

// the epilogues write one full 32-byte sector per lane (STG.256)
bool misaligned32(const void* out, const char* who) {
  if (reinterpret_cast<uintptr_t>(out) % 32 == 0) return false;
  snprintf(g_err, sizeof g_err, "%s: the output buffer must be 32-byte aligned", who);
  return true;
}

using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

}  // namespace

// rank-`rank` bf16 tensor map, zero OOB fill.  strides_bytes has rank-1 entries.  swizzle_bytes: 128 or 64.
int make_tmap_bf16(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
    return 1;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUtensorMapSwizzle swz = swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), dims, strides_bytes, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled failed: CUresult %d (rank %d)", int(r), rank);
    return 1;
  }
  return 0;
}

int make_tmap_plain(CUtensorMap* m, const void* base, int elem_bytes, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
    return 1;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUtensorMapDataType ty = elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16;
  CUresult r = fn(m, ty, rank, const_cast<void*>(base), dims, strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_err, sizeof g_err, "cuTensorMapEncodeTiled (plain, %d-byte elements) failed: CUresult %d (rank %d)",
             elem_bytes, int(r), rank);
    return 1;
  }
  return 0;
}

int num_sms() {
  static std::atomic<int> cache[64];   // per device
  int dev = 0;
  cudaGetDevice(&dev);
  std::atomic<int>& slot = cache[dev & 63];
  int n = slot.load(std::memory_order_relaxed);
  if (!n) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    slot.store(n, std::memory_order_relaxed);
  }
  return n;
}

namespace {

template <int BLOCK_N, int MT, bool CONV, bool POOL, int OUT, bool BIG = false, bool HALO = false>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const IgemmParams& p, cudaStream_t stream) {
  auto kern = igemm_bf16_kernel<BLOCK_N, MT, CONV, POOL, OUT, BIG, HALO>;
  static std::atomic<unsigned long long> attr_set{0};   // one bit per device: the attribute is per device
  constexpr int smem = Cfg<BLOCK_N, MT, HALO>::kSmemBytes;
  if (device_needs_setup(attr_set)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) {
      device_setup_failed(attr_set);
      snprintf(g_err, sizeof g_err, "cudaFuncSetAttribute(smem=%d): %s", smem, cudaGetErrorString(e));
      return 1;
    }
  }
  const int tiles = p.num_m_tiles * p.num_n_tiles * (p.ksplit > 1 ? p.ksplit : 1);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  cudaError_t e = launch_pdl(kern, dim3(grid), dim3(kNumThreads), smem, stream, ta, tb, p);
  count_launch();
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof g_err, "igemm launch failed: %s", cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

}  // namespace

const char* igemm_last_error() { return g_err; }

#ifndef VMB_PAIR_DEFAULT
#define VMB_PAIR_DEFAULT 1
#endif
namespace {
std::atomic<int> g_pair_override{-1};   // -1: follow the environment / build default
}
bool igemm_use_pair() {
  const int o = g_pair_override.load(std::memory_order_relaxed);
  if (o >= 0) return o != 0;
  static const bool on = [] {
    const char* e = getenv("VMB_IGEMM_PAIR");
    return e ? (e[0] != '0') : (VMB_PAIR_DEFAULT != 0);
  }();
  return on;
}
namespace {
std::atomic<int> g_halo_override{-1};
}
bool igemm_use_halo() {
  const int o = g_halo_override.load(std::memory_order_relaxed);
  if (o >= 0) return o != 0;
  static const bool on = [] {
    const char* e = getenv("VMB_IGEMM_HALO");
    return !(e && e[0] == '0');
  }();
  return on;
}
int igemm_set_halo(int on) {
  const int prev = igemm_use_halo() ? 1 : 0;
  g_halo_override.store(on < 0 ? -1 : (on ? 1 : 0), std::memory_order_relaxed);
  return prev;
}
int igemm_set_pair(int on) {
  const int prev = igemm_use_pair() ? 1 : 0;
  g_pair_override.store(on < 0 ? -1 : (on ? 1 : 0), std::memory_order_relaxed);
  return prev;
}

namespace {
int pair_result(int rc) {
  if (rc) snprintf(g_err, sizeof g_err, "%s", igemm_pair_last_error());
  return rc ? 1 : 0;
}
}  // namespace

int igemm_linear(const void* a, const void* w, const float* bias, void* out, int out_f32, int relu, int M, int N,
                 int K, cudaStream_t stream, int fmt, int* sat_flag) {
  if (M <= 0) return 0;
  if (misaligned32(out, "igemm_linear")) return 1;
  if (K % kBlockK != 0 || N % 128 != 0) {
    snprintf(g_err, sizeof g_err, "igemm_linear: need K %% 64 == 0 and N %% 128 == 0 (got K=%d N=%d)", K, N);
    return 1;
  }
  if (!out_f32 && N % 256 == 0 && M >= 256 && igemm_use_pair())
    return pair_result(igemm_pair_linear(a, w, bias, out, relu, M, N, K, stream, fmt, sat_flag));
  const int block_n = (N % 256 == 0) ? 256 : 128;
  CUtensorMap ta, tb;
  {
    uint64_t dims[2] = {uint64_t(K), uint64_t(M)};
    uint64_t str[1] = {uint64_t(K) * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    if (make_tmap_bf16(&ta, a, 2, dims, str, box)) return 1;
  }
  {
    uint64_t dims[2] = {uint64_t(K), uint64_t(N)};
    uint64_t str[1] = {uint64_t(K) * 2};
    uint32_t box[2] = {kBlockK, uint32_t(block_n)};
    if (make_tmap_bf16(&tb, w, 2, dims, str, box)) return 1;
  }
  IgemmParams p{};
  p.M = M;
  p.N = N;
  p.num_kb = K / kBlockK;
  p.num_m_tiles = (M + kBlockM - 1) / kBlockM;
  p.num_n_tiles = N / block_n;
  p.relu = relu;
  p.ldo = N;
  p.bias = bias;
  p.out = out;
  p.f16 = fmt == kFmtF16;
  p.sat_flag = sat_flag;
  if (block_n == 256)
    return out_f32 ? launch<256, 1, false, false, kOutF32>(ta, tb, p, stream)
                   : launch<256, 1, false, false, kOutBf16>(ta, tb, p, stream);
  return out_f32 ? launch<128, 1, false, false, kOutF32>(ta, tb, p, stream)
                 : launch<128, 1, false, false, kOutBf16>(ta, tb, p, stream);
}

int igemm_linear_rect(const void* a, const void* w, const float* bias, void* out, long long ldo, int relu, int M, int N,
                         int K, cudaStream_t stream, int fmt, int* sat_flag) {
  if (M <= 0 || N <= 0) return 0;
  if (misaligned32(out, "igemm_linear_rect")) return 1;
  if (K % kBlockK != 0 || N % 128 != 0 || ldo % 16 != 0) {
    snprintf(g_err, sizeof g_err, "igemm_linear_rect: need K %% 64 == 0, N %% 128 == 0, ldo %% 16 == 0");
    return 1;
  }
  CUtensorMap ta, tb;
  {
    uint64_t dims[2] = {uint64_t(K), uint64_t(M)};
    uint64_t str[1] = {uint64_t(K) * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    if (make_tmap_bf16(&ta, a, 2, dims, str, box)) return 1;
  }
  // 64-wide tiles when 128-wide ones would leave more than half of the SMs without a tile
  const int m_tiles = (M + kBlockM - 1) / kBlockM;
  const int block_n = (2 * m_tiles * (N / 128) <= num_sms()) ? 64 : 128;
  {
    uint64_t dims[2] = {uint64_t(K), uint64_t(N)};
    uint64_t str[1] = {uint64_t(K) * 2};
    uint32_t box[2] = {kBlockK, uint32_t(block_n)};
    if (make_tmap_bf16(&tb, w, 2, dims, str, box)) return 1;
  }
  IgemmParams p{};
  p.M = M;
  p.N = N;
  p.num_kb = K / kBlockK;
  p.num_m_tiles = m_tiles;
  p.num_n_tiles = N / block_n;
  p.relu = relu;
  p.ldo = ldo;
  p.bias = bias;
  p.out = out;
  p.f16 = fmt == kFmtF16;
  p.sat_flag = sat_flag;
  return block_n == 64 ? launch<64, 1, false, false, kOutBf16>(ta, tb, p, stream)
                       : launch<128, 1, false, false, kOutBf16>(ta, tb, p, stream);
}

int igemm_linear_split(const void* a_planes, const void* w_planes, const float* bias, float* out, long long ldo,
                       int relu, int M, int N, int K, cudaStream_t stream, int planes) {
  if (M <= 0) return 0;
  if (misaligned32(out, "igemm_linear_split")) return 1;
  if (ldo % 8 != 0) {
    snprintf(g_err, sizeof g_err, "igemm_linear_split: ldo must be a multiple of 8 floats (32-byte rows), got %lld", ldo);
    return 1;
  }
  if (planes != 2 && planes != 3) {
    snprintf(g_err, sizeof g_err, "igemm_linear_split: planes must be 2 or 3");
    return 1;
  }
  if (K % kBlockK != 0 || N % 128 != 0) {
    snprintf(g_err, sizeof g_err, "igemm_linear_split: need K %% 64 == 0 and N %% 128 == 0 (got K=%d N=%d)", K, N);
    return 1;
  }
  if (planes_gemm_enabled()) {
    // every plane of a K-block loaded once per tile (planes_gemm_sm100.cu); the kernel below is kept for A/B timing
    if (planes_gemm(a_planes, w_planes, bias, out, ldo, relu, M, N, K, planes, 0, stream)) {
      snprintf(g_err, sizeof g_err, "%s", planes_gemm_last_error());
      return 1;
    }
    return 0;
  }
  const int block_n = (N % 256 == 0) ? 256 : 128;
  CUtensorMap ta, tb;
  {
    uint64_t dims[2] = {uint64_t(planes) * K, uint64_t(M)};
    uint64_t str[1] = {uint64_t(planes) * K * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    if (make_tmap_bf16(&ta, a_planes, 2, dims, str, box)) return 1;
  }
  {
    uint64_t dims[2] = {uint64_t(planes) * K, uint64_t(N)};
    uint64_t str[1] = {uint64_t(planes) * K * 2};
    uint32_t box[2] = {kBlockK, uint32_t(block_n)};
    if (make_tmap_bf16(&tb, w_planes, 2, dims, str, box)) return 1;
  }
  IgemmParams p{};
  p.M = M;
  p.N = N;
  p.split_nkb = K / kBlockK;
  p.split_planes = planes;
  p.num_kb = (planes == 3 ? 6 : 3) * p.split_nkb;
  p.num_m_tiles = (M + kBlockM - 1) / kBlockM;
  p.num_n_tiles = N / block_n;
  p.relu = relu;
  p.ldo = ldo;
  p.bias = bias;
  p.out = out;
  return block_n == 256 ? launch<256, 1, false, false, kOutF32>(ta, tb, p, stream)
                        : launch<128, 1, false, false, kOutF32>(ta, tb, p, stream);
}

int igemm_linear_split_out(const void* a_planes, const void* w_planes, const float* bias, void* out_planes, int relu,
                           int M, int N, int K, cudaStream_t stream) {
  if (M <= 0) return 0;
  if (misaligned32(out_planes, "igemm_linear_split_out")) return 1;
  if (K % kBlockK != 0 || N % 256 != 0) {
    snprintf(g_err, sizeof g_err, "igemm_linear_split_out: need K %% 64 == 0 and N %% 256 == 0 (got K=%d N=%d)", K, N);
    return 1;
  }
  CUtensorMap ta, tb;
  {
    uint64_t dims[2] = {uint64_t(2) * K, uint64_t(M)};
    uint64_t str[1] = {uint64_t(2) * K * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    if (make_tmap_bf16(&ta, a_planes, 2, dims, str, box)) return 1;
  }
  {
    uint64_t dims[2] = {uint64_t(2) * K, uint64_t(N)};
    uint64_t str[1] = {uint64_t(2) * K * 2};
    uint32_t box[2] = {kBlockK, 256};
    if (make_tmap_bf16(&tb, w_planes, 2, dims, str, box)) return 1;
  }
  IgemmParams p{};
  p.M = M;
  p.N = N;
  p.split_nkb = K / kBlockK;
  p.split_planes = 2;
  p.num_kb = 3 * p.split_nkb;
  p.num_m_tiles = (M + kBlockM - 1) / kBlockM;
  p.num_n_tiles = N / 256;
  p.relu = relu;
  p.ldo = 2LL * N;     // [M][hi(N) | lo(N)]
  p.lo_off = N;
  p.bias = bias;
  p.out = out_planes;
  return launch<256, 1, false, false, kOutSplit>(ta, tb, p, stream);
}

int igemm_conv3x3_split(const void* act_planes, const void* w_planes, const float* bias, void* out_planes, int n_img,
                        int H, int W, int C_in, int C_out, int pool, cudaStream_t stream) {
  if (n_img <= 0) return 0;
  if (misaligned32(out_planes, "igemm_conv3x3_split")) return 1;
  const int Wb = (W % 16 == 0) ? 16 : 8;
  const int Hb = 32 / Wb;
  if (C_in % kBlockK != 0 || C_out % 128 != 0 || W % Wb != 0 || H % Hb != 0) {
    snprintf(g_err, sizeof g_err, "igemm_conv3x3_split: unsupported geometry H=%d W=%d C_in=%d C_out=%d", H, W, C_in, C_out);
    return 1;
  }
  const int block_n = (C_out % 256 == 0) ? 256 : 128;
  const int K = 9 * C_in;
  CUtensorMap ta, tb;
  {
    uint64_t dims[5] = {uint64_t(C_in), uint64_t(W), uint64_t(H), 2, uint64_t(n_img)};
    uint64_t str[4] = {uint64_t(C_in) * 2, uint64_t(W) * C_in * 2, uint64_t(H) * W * C_in * 2, uint64_t(2) * H * W * C_in * 2};
    uint32_t box[5] = {kBlockK, uint32_t(Wb), uint32_t(Hb), 1, 1};
    if (make_tmap_bf16(&ta, act_planes, 5, dims, str, box)) return 1;
  }
  {
    uint64_t dims[2] = {uint64_t(2) * K, uint64_t(C_out)};
    uint64_t str[1] = {uint64_t(2) * K * 2};
    uint32_t box[2] = {kBlockK, uint32_t(block_n)};
    if (make_tmap_bf16(&tb, w_planes, 2, dims, str, box)) return 1;
  }
  IgemmParams p{};
  p.M = n_img;
  p.N = C_out;
  p.cblks = C_in / kBlockK;
  p.num_kb = 3 * 9 * p.cblks;
  p.conv_split = 1;
  p.H = H;
  p.W = W;
  p.Hb = Hb;
  p.Wb = Wb;
  p.boxes_per_row = W / Wb;
  p.boxes_per_img = (H / Hb) * (W / Wb);
  p.total_boxes = n_img * p.boxes_per_img;
  p.num_m_tiles = (p.total_boxes + 3) / 4;
  p.num_n_tiles = C_out / block_n;
  p.relu = 1;
  p.ldo = C_out;
  p.bias = bias;
  p.out = out_planes;
  const long long plane = static_cast<long long>(pool ? (H / 2) * (W / 2) : H * W) * C_out;
  p.out_img_stride = 2 * plane;
  p.lo_off = plane;
  if (block_n == 256)
    return pool ? launch<256, 1, true, true, kOutSplit>(ta, tb, p, stream)
                : launch<256, 1, true, false, kOutSplit>(ta, tb, p, stream);
  if (p.num_m_tiles >= 4 * num_sms()) {   // C_out = 128: 256-row CTA tiles, as in igemm_conv3x3
    p.num_m_tiles = (p.total_boxes + 7) / 8;
    return pool ? launch<128, 2, true, true, kOutSplit>(ta, tb, p, stream)
                : launch<128, 2, true, false, kOutSplit>(ta, tb, p, stream);
  }
  return pool ? launch<128, 1, true, true, kOutSplit>(ta, tb, p, stream)
              : launch<128, 1, true, false, kOutSplit>(ta, tb, p, stream);
}

int igemm_conv3x3(const void* act, const void* w, const float* bias, void* out, int n_img, int H, int W, int C_in,
                  int C_out, int pool, cudaStream_t stream, int fmt, int* sat_flag) {
  if (n_img <= 0) return 0;
  if (misaligned32(out, "igemm_conv3x3")) return 1;
  const int Wb = (W % 16 == 0) ? 16 : 8;
  const int Hb = 32 / Wb;
  if (C_in % kBlockK != 0 || C_out % 128 != 0 || W % Wb != 0 || H % Hb != 0) {
    snprintf(g_err, sizeof g_err, "igemm_conv3x3: unsupported geometry H=%d W=%d C_in=%d C_out=%d", H, W, C_in, C_out);
    return 1;
  }
  // C_out = 128 (conv2) stays on the single-CTA 256 x 128 tiles: at N = 128 the MMA's operand fetch saturates shared
  // memory either way and the pair kernel measured no faster
  if (igemm_use_pair() && C_out % 256 == 0)
    return pair_result(igemm_pair_conv3x3(act, w, bias, out, n_img, H, W, C_in, C_out, pool, stream, fmt, sat_flag));
  const int block_n = (C_out % 256 == 0) ? 256 : 128;
  const int K = 9 * C_in;
  // when the image height allows it, one TMA box brings a whole 128-pixel sub-tile (Wb x 4*Hb pixels) instead of four
  // 32-pixel quarters: the single producer thread issues 2-3 copies per K block instead of 5-9
  const bool big = H % (4 * Hb) == 0;
  CUtensorMap ta, tb;
  {
    uint64_t dims[4] = {uint64_t(C_in), uint64_t(W), uint64_t(H), uint64_t(n_img)};
    uint64_t str[3] = {uint64_t(C_in) * 2, uint64_t(W) * C_in * 2, uint64_t(H) * W * C_in * 2};
    uint32_t box[4] = {kBlockK, uint32_t(Wb), uint32_t(big ? 4 * Hb : Hb), 1};
    if (make_tmap_bf16(&ta, act, 4, dims, str, box)) return 1;
  }
  {
    uint64_t dims[2] = {uint64_t(K), uint64_t(C_out)};
    uint64_t str[1] = {uint64_t(K) * 2};
    uint32_t box[2] = {kBlockK, uint32_t(block_n)};
    if (make_tmap_bf16(&tb, w, 2, dims, str, box)) return 1;
  }
  IgemmParams p{};
  p.M = n_img;
  p.N = C_out;
  p.num_kb = K / kBlockK;
  p.cblks = C_in / kBlockK;
  p.H = H;
  p.W = W;
  p.Hb = Hb;
  p.Wb = Wb;
  p.boxes_per_row = W / Wb;
  p.big_box = big ? 1 : 0;
  // "box" = the unit the tile index counts: a 32-pixel quarter, or a whole 128-pixel sub-tile in big-box mode
  p.boxes_per_img = big ? (H / (4 * Hb)) * (W / Wb) : (H / Hb) * (W / Wb);
  p.total_boxes = n_img * p.boxes_per_img;
  const int sub_tiles = big ? p.total_boxes : (p.total_boxes + 3) / 4;   // 128-pixel sub-tiles
  p.num_m_tiles = sub_tiles;
  p.num_n_tiles = C_out / block_n;
  p.relu = 1;
  p.ldo = C_out;
  p.bias = bias;
  p.out = out;
  p.f16 = fmt == kFmtF16;
  p.sat_flag = sat_flag;
  p.out_img_stride = static_cast<long long>(pool ? (H / 2) * (W / 2) : H * W) * C_out;
  if (block_n == 256) {
    if (big)
      return pool ? launch<256, 1, true, true, kOutBf16, true>(ta, tb, p, stream)
                  : launch<256, 1, true, false, kOutBf16, true>(ta, tb, p, stream);
    return pool ? launch<256, 1, true, true, kOutBf16>(ta, tb, p, stream)
                : launch<256, 1, true, false, kOutBf16>(ta, tb, p, stream);
  }
  // C_out = 128: pair two 128-pixel sub-tiles per CTA tile when there are enough tiles to keep every SM busy
  if (p.num_m_tiles >= 4 * num_sms()) {
    p.num_m_tiles = (sub_tiles + 1) / 2;
    if (big && Wb == kHaloWb && 4 * Hb + 2 == kHaloRows && igemm_use_halo()) {
      // one haloed activation box per (channel block, dx) instead of one box per tap (see Cfg)
      CUtensorMap th;
      uint64_t dims[4] = {uint64_t(C_in), uint64_t(W), uint64_t(H), uint64_t(n_img)};
      uint64_t str[3] = {uint64_t(C_in) * 2, uint64_t(W) * C_in * 2, uint64_t(H) * W * C_in * 2};
      uint32_t box[4] = {kBlockK, uint32_t(kHaloWb), uint32_t(kHaloRows), 1};
      if (make_tmap_bf16(&th, act, 4, dims, str, box)) return 1;
      return pool ? launch<128, 2, true, true, kOutBf16, true, true>(th, tb, p, stream)
                  : launch<128, 2, true, false, kOutBf16, true, true>(th, tb, p, stream);
    }
    if (big)
      return pool ? launch<128, 2, true, true, kOutBf16, true>(ta, tb, p, stream)
                  : launch<128, 2, true, false, kOutBf16, true>(ta, tb, p, stream);
    return pool ? launch<128, 2, true, true, kOutBf16>(ta, tb, p, stream)
                : launch<128, 2, true, false, kOutBf16>(ta, tb, p, stream);
  }
  if (big)
    return pool ? launch<128, 1, true, true, kOutBf16, true>(ta, tb, p, stream)
                : launch<128, 1, true, false, kOutBf16, true>(ta, tb, p, stream);
  return pool ? launch<128, 1, true, true, kOutBf16>(ta, tb, p, stream)
              : launch<128, 1, true, false, kOutBf16>(ta, tb, p, stream);
}

}  // namespace vmb
