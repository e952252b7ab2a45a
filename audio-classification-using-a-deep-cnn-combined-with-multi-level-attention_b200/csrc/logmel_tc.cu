// Tensor-core log-mel front end (sm_100a): framing + periodic Hann + 512-point real DFT as split-precision tcgen05
// GEMMs, magnitude + HTK mel projection + log fused into the epilogue.
// Replaces torchvggish/mel_features.py:21-45 (frame), :48-68 (periodic_hann), :71-92 (stft_magnitude),
// :114-189 (spectrogram_to_mel_matrix), :192-223 (log_mel_spectrogram).
//
// Two kernels live here:
//  * logmel_eo_kernel (second half of the file, the default): centred even / odd form of the DFT (K = 200), raw samples
//    framed by TMA straight from the caller's waveform, fp16 hi + lo operand planes built in shared memory, three
//    products.  Its header comment has the algebra and the data flow.
//  * split_wave_kernel + logmel_tc_kernel (first half, the first tensor-core version): the waveform is split into three
//    bf16 planes in HBM, A tiles are TMA boxes of an overlapping-rows view of those planes, straight K = 400 DFT, six
//    products.  Serves inputs that are not 16-byte aligned.
//
//   S[f][c] = sum_n x[160 f + n] * W[n][c],   W[n][2j] = hann[n] cos(2 pi k_j n / 512), W[n][2j+1] = hann[n] sin(..)
//   |X_j| = sqrt(S[f][2j]^2 + S[f][2j+1]^2);  mel[f][m] = sum_j |X_j| M[k_j][m];  out = log(mel + 0.01)
//
// Shared by both:
// * Only DFT bins 4..243 are evaluated (2 N-tiles of 120 bins): the HTK mel matrix is exactly zero outside bins
//   5..239 (checked when the tables are built).
// * Epilogue: one thread owns one frame (TMEM lane); it walks the bins in order and, because every bin feeds at
//   most the two adjacent mel bands, keeps just two running band sums, emitting log(band + 0.01) as bands complete.
//
// The plane kernel in detail:
// * Precision.  log(mel + 0.01) has slope up to 100, so the DFT needs fp32-class accuracy (SURVEY §7 H1): plain
//   bf16/tf32 operands miss the 1e-4 bound by orders of magnitude.  Both operands are split exactly into
//   three bf16 terms (x = x0 + x1 + x2, 24 mantissa bits) and the six products with i + j <= 2 are accumulated
//   in the same fp32 TMEM accumulator, smallest first: A2B0, A1B1, A0B2, A1B0, A0B1, A0B0.
// * Framing is never materialised: the A operand is a 3-D TMA tensor map over the split waveform planes with
//   dims {416 (sample in frame), frames (stride 160 samples), plane*clip}; rows overlap in memory.  The Hann window
//   is folded into W; columns 400..415 of W are zero (K padded to 13 blocks of 32).
// * Warp roles (320 threads): warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 / 6-9 epilogue of N-tile 0 / 1.
//   Persistent over 128-frame tiles; the two N-tiles of a frame tile use the two halves of TMEM so the epilogue of one
//   overlaps the MMAs of the next.  Smem: 3 stages x {A0,A1,A2 (128x32), B0,B1,B2 (240x32)} bf16, 64-byte swizzle = 207 KB.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <mutex>
#include <vector>

#include "igemm_sm100.cuh"
#include "kernels.cuh"
#include "sm100_ptx.cuh"

namespace vmb {

namespace {

constexpr int kWin = 400, kHop = 160, kFft = 512, kBins = 257, kMel = 64;
constexpr int kBinLo = 4;               // first evaluated DFT bin
constexpr int kTileBins = 120;          // bins per N-tile
constexpr int kNTiles = 2;              // bins 4..243
constexpr int kEvalBins = kTileBins * kNTiles;
constexpr int kTM = 128;                // frames per tile (UMMA M)
constexpr int kTN = 2 * kTileBins;      // 240 (UMMA N)
constexpr int kBK = 32;                 // K block: 32 bf16 = one 64-byte swizzle row
constexpr int kKB = 13;                 // 13 * 32 = 416 >= 400
constexpr int kKPad = kKB * kBK;
constexpr int kATile = kTM * kBK * 2;   // 8192
constexpr int kBTile = kTN * kBK * 2;   // 15360
constexpr int kStageBytes = 3 * (kATile + kBTile);  // 70656
constexpr int kStages = 3;
constexpr int kThreads = 320;          // producer, MMA issuer, 2 x 4 epilogue warps
constexpr int kHandFloats = 8;          // per-row walk state handed from the N-tile-0 epilogue to the N-tile-1 one
constexpr int kSmemBytes = 1024 + kStages * kStageBytes + 512 + 2 * kTM * kHandFloats * 4;
constexpr int kTmemCols = 512;          // accumulator t lives at column 256 t
constexpr double kPi = 3.14159265358979323846;
constexpr float kLogOffset = 0.01f;
// Ill-conditioned frames.  log(mel + 0.01) amplifies an absolute error of the band sum by 1 / (mel + 0.01), and what the
// split-precision tensor-core DFT leaves in an (almost) empty band scales with the frame's total spectral energy:
// operand planes carry 22-24 bits and the fp32 accumulation inside tcgen05.mma truncates.  With
//     R = sqrt(sum_k |X_k|^2) / (min_band mel + 0.01)
// the emulation of the kernels' arithmetic (tools/logmel_precision_emulation.py; 22 signal types) gives
// |log-mel error| <= 3e-6 + 2.3e-8 R.  Frames with R > kExactRatio (a loud tone or band-limited signal over a digitally
// silent band: > 70 dB between the spectrum's energy and its quietest mel band) are flagged by the epilogue and redone
// in float64 by logmel_exact_kernel, so that the 1e-4 bound against the float64 reference holds for every input
// (<= 8.4e-5 from the tensor-core path, ~1e-7 from the exact one).  ~0.35 % of the frames of the synthetic bench batch
// (the late part of the chirp family) are flagged; noise-like audio never is.
constexpr float kExactRatio = 3500.f;
// The plane kernel (straight K = 400 DFT, six bf16 products: 150 truncating accumulation steps per bin) follows
// |error| <= 3e-6 + 7.3e-8 R in the same emulation, hence its lower threshold.
constexpr float kExactRatioPlanes = 1200.f;

// mel walk tables: bin kBinLo + i feeds band e-1 with weight wf and band e with weight wr (e in 0..64)
__constant__ int c_band[kEvalBins];
__constant__ float c_wfall[kEvalBins];
__constant__ float c_wrise[kEvalBins];
__constant__ int c_mel_lo[kMel], c_mel_hi[kMel];   // evaluated bins [lo, hi) carrying weight for each band (exact path)

// ------------------------------------------------------------------ waveform -> three bf16 planes
// planes[p][clip][pitch]; samples >= n_samples are written as zero so that K padding never meets garbage.
// IN = float (waveform in [-1, 1]) or int16_t (PCM, scaled by 1/32768 like vggish_input.py:98 — exact in fp32).
template <class IN>
__device__ __forceinline__ float load_sample(const IN* p);
template <>
__device__ __forceinline__ float load_sample<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_sample<int16_t>(const int16_t* p) { return static_cast<float>(__ldg(p)) * (1.0f / 32768.0f); }

template <class IN>
__global__ void __launch_bounds__(256)
split_wave_kernel(const IN* __restrict__ wave, long long n_samples, long long clip_stride, long long pitch,
                  long long n_clips, __nv_bfloat16* __restrict__ planes) {
  pdl_launch_dependents();   // logmel_tc_kernel's prologue may start while the last blocks here still run
  const long long groups_per_clip = pitch / 8;
  const long long total = groups_per_clip * n_clips;
  const long long plane_elems = n_clips * pitch;
  for (long long g = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; g < total;
       g += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long clip = g / groups_per_clip;
    const long long s0 = (g - clip * groups_per_clip) * 8;
    const IN* src = wave + clip * clip_stride + s0;
    uint32_t h0[4], h1[4], h2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float x[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) x[u] = (s0 + 2 * i + u < n_samples) ? load_sample<IN>(src + 2 * i + u) : 0.f;
      __nv_bfloat16 a[2], b[2], c[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        a[u] = __float2bfloat16_rn(x[u]);
        const float r1 = x[u] - __bfloat162float(a[u]);      // exact
        b[u] = __float2bfloat16_rn(r1);
        const float r2 = r1 - __bfloat162float(b[u]);        // exact
        c[u] = __float2bfloat16_rn(r2);
      }
      h0[i] = static_cast<uint32_t>(__bfloat16_as_ushort(a[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(a[1])) << 16);
      h1[i] = static_cast<uint32_t>(__bfloat16_as_ushort(b[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(b[1])) << 16);
      h2[i] = static_cast<uint32_t>(__bfloat16_as_ushort(c[0])) | (static_cast<uint32_t>(__bfloat16_as_ushort(c[1])) << 16);
    }
    __nv_bfloat16* dst = planes + clip * pitch + s0;
    *reinterpret_cast<uint4*>(dst) = make_uint4(h0[0], h0[1], h0[2], h0[3]);
    *reinterpret_cast<uint4*>(dst + plane_elems) = make_uint4(h1[0], h1[1], h1[2], h1[3]);
    *reinterpret_cast<uint4*>(dst + 2 * plane_elems) = make_uint4(h2[0], h2[1], h2[2], h2[3]);
  }
}

// ------------------------------------------------------------------ the GEMM + mel/log epilogue
struct LogmelParams {
  int a_planes;             // 3 for fp32 input; 2 for 16-bit PCM (x = m / 32768 splits exactly into two bf16 terms,
                            // the third plane is identically zero and its product A2*B0 is skipped)
  long long frames_out;     // frames written per clip
  int tiles_per_clip;       // ceil(frames_out / 128)
  int n_clips;
  long long total_tiles;    // n_clips * tiles_per_clip
  float* out;               // [n_clips][frames_out][64]
  uint32_t* exact_list;     // flagged frames (tile * 128 + row in the tile) to be redone in float64, see kExactRatio
  unsigned* exact_count;    // entries in exact_list (zeroed by the host before the launch)
};


struct BandWalk {
  int e = 0;          // lo accumulates band e-1, hi band e
  float lo = 0.f, hi = 0.f;
  float4 pend;        // four finished bands waiting for one 16-byte store
  float e2 = 0.f;     // sum of |X_k|^2 over the bins walked so far
  float mn = 3.0e38f; // smallest finished band sum
};

__device__ __forceinline__ void emit_band(BandWalk& w, float* __restrict__ row_out, bool valid) {
  const int band = w.e - 1;
  if (band >= 0 && band < kMel) {
    const float v = __logf(w.lo + kLogOffset);
    w.mn = fminf(w.mn, w.lo);
    const int slot = band & 3;
    if (slot == 0) w.pend.x = v;
    else if (slot == 1) w.pend.y = v;
    else if (slot == 2) w.pend.z = v;
    else {
      w.pend.w = v;
      if (valid) *reinterpret_cast<float4*>(row_out + band - 3) = w.pend;
    }
  }
  w.lo = w.hi;
  w.hi = 0.f;
  ++w.e;
}

template <int NB>  // NB bins = 2*NB accumulator columns in v
__device__ __forceinline__ void walk_bins(BandWalk& w, const uint32_t* v, int bin0, float* __restrict__ row_out,
                                          bool valid) {
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    const float re = __uint_as_float(v[2 * j]), im = __uint_as_float(v[2 * j + 1]);
    float mag;   // sqrt.approx: 2 ulp, far below what the band sums resolve; exact zero stays zero
    const float ss = fmaf(re, re, im * im);
    w.e2 += ss;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(mag) : "f"(ss));
    const int e = c_band[bin0 + j];
    while (w.e < e) emit_band(w, row_out, valid);      // warp-uniform: depends on the bin index only
    w.lo = fmaf(c_wfall[bin0 + j], mag, w.lo);
    w.hi = fmaf(c_wrise[bin0 + j], mag, w.hi);
  }
}

__global__ void __launch_bounds__(kThreads, 1)
logmel_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const LogmelParams p) {
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full = empty_bar + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* hand_full = tmem_empty + 2;       // [2 buffers][4 lane quarters]
  uint64_t* hand_empty = hand_full + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(hand_empty + 8);
  float* hand = reinterpret_cast<float*>(smem + kStages * kStageBytes + 512);   // [2][kTM][kHandFloats]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 4);
    }
    for (int s = 0; s < 8; ++s) {
      mbar_init(&hand_full[s], 1);
      mbar_init(&hand_empty[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform by construction
  pdl_wait();   // the sample planes (split_wave_kernel's output) are read below

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int clip = static_cast<int>(tile / p.tiles_per_clip);
        const int row0 = static_cast<int>(tile - static_cast<long long>(clip) * p.tiles_per_clip) * kTM;
        for (int nt = 0; nt < kNTiles; ++nt) {
          for (int kb = 0; kb < kKB; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* base = smem + stage * kStageBytes;
            mbar_expect_tx(&full_bar[stage], p.a_planes * kATile + 3 * kBTile);
#pragma unroll
            for (int pl = 0; pl < 3; ++pl) {
              if (pl < p.a_planes)
                tma_load_3d(base + pl * kATile, &tmap_a, &full_bar[stage], kb * kBK, row0, pl * p.n_clips + clip);
              tma_load_2d(base + 3 * kATile + pl * kBTile, &tmap_b, &full_bar[stage], kb * kBK,
                          pl * kEvalBins * 2 + nt * kTN);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_bf16_f32(kTM, kTN);
    uint32_t stage = 0, phase = 0, it = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      for (int nt = 0; nt < kNTiles; ++nt, ++it) {
        const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = 0; kb < kKB; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          if (elect_one()) {
            const uint32_t a0 = smem_u32(smem + stage * kStageBytes);
            const uint32_t b0 = a0 + 3 * kATile;
            // products (a plane, b plane), smallest magnitude first
            constexpr int prod_a[6] = {2, 1, 0, 1, 0, 0};
            constexpr int prod_b[6] = {0, 1, 2, 0, 1, 0};
            const int q0 = p.a_planes == 3 ? 0 : 1;   // two A planes: skip the A2*B0 product
#pragma unroll
            for (int q = 0; q < 6; ++q) {
              if (q < q0) continue;
              const uint64_t a_desc = umma_desc_kmajor_sw64(a0 + prod_a[q] * kATile);
              const uint64_t b_desc = umma_desc_kmajor_sw64(b0 + prod_b[q] * kBTile);
#pragma unroll
              for (int k = 0; k < kBK / 16; ++k)   // +32 bytes (>>4 = 2) per 16-element K step
                umma_bf16_ss(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | (q - q0) | k) != 0);
            }
            umma_commit(&empty_bar[stage]);
            if (kb == kKB - 1) umma_commit(&tmem_full[acc]);
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    // Two sets of four warps: set 0 (warps 2-5) walks the bins of N-tile 0, set 1 (warps 6-9) those of N-tile 1, so
    // the two halves of a frame tile are post-processed concurrently.  The band walk is sequential over the bins, so
    // warp q of set 0 hands its per-row state (two running band sums + the partly filled group of four outputs) to
    // warp q of set 1 through shared memory; the arithmetic and its order are exactly those of a single walk.
    const int set = (warp - 2) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    uint32_t mi = 0;   // frame-tile iteration of this CTA
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++mi) {
      const long long clip = tile / p.tiles_per_clip;
      const long long frame = (tile - clip * p.tiles_per_clip) * kTM + row;
      const bool valid = frame < p.frames_out;
      float* row_out = p.out + (clip * p.frames_out + (valid ? frame : 0)) * kMel;
      const uint32_t hb = mi & 1, hphase = (mi >> 1) & 1;
      float* hrow = hand + (hb * kTM + row) * kHandFloats;
      BandWalk w;
      w.pend = make_float4(0.f, 0.f, 0.f, 0.f);
      if (set == 1) {
        mbar_wait(&hand_full[hb * 4 + q], hphase);
        w.e = c_band[kTileBins - 1];            // where the walk over bins 0..119 stops (uniform)
        w.lo = hrow[0]; w.hi = hrow[1];
        w.pend = make_float4(hrow[2], hrow[3], hrow[4], 0.f);
        w.e2 = hrow[6]; w.mn = hrow[7];
        __syncwarp();
        if (lane == 0) mbar_arrive(&hand_empty[hb * 4 + q]);
      }
      const uint32_t acc = set, acc_phase = mi & 1;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after_sync();
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * 256;
#pragma unroll 1
      for (int ch = 0; ch < kTN / 32; ++ch) {     // 7 chunks of 32 columns = 16 bins
        uint32_t v[32];
        tmem_ld_32x32(t_addr + ch * 32, v);
        tmem_ld_wait();
        walk_bins<16>(w, v, set * kTileBins + ch * 16, row_out, valid);
      }
      {                                            // last 16 columns = 8 bins
        uint32_t v[16];
        tmem_ld_32x16(t_addr + (kTN / 32) * 32, v);
        tmem_ld_wait();
        walk_bins<8>(w, v, set * kTileBins + (kTN / 32) * 16, row_out, valid);
      }
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (set == 0) {
        mbar_wait(&hand_empty[hb * 4 + q], hphase ^ 1);
        hrow[0] = w.lo; hrow[1] = w.hi;
        hrow[2] = w.pend.x; hrow[3] = w.pend.y; hrow[4] = w.pend.z;
        hrow[6] = w.e2; hrow[7] = w.mn;
        __syncwarp();
        if (lane == 0) mbar_arrive(&hand_full[hb * 4 + q]);
      } else {
        while (w.e <= kMel) emit_band(w, row_out, valid);   // flush the remaining bands (up to band 63)
        const float lim = kExactRatioPlanes * (w.mn + kLogOffset);
        const bool mine = valid && w.e2 > lim * lim;
        const uint32_t bad = __ballot_sync(0xffffffffu, mine);
        if (bad) {   // one atomic per warp reserves the slots, every flagged frame writes its own entry
          uint32_t base = 0;
          if (lane == 0) base = atomicAdd(p.exact_count, static_cast<unsigned>(__popc(bad)));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (mine) p.exact_list[base + __popc(bad & ((1u << lane) - 1u))] = static_cast<uint32_t>(tile * kTM + row);
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ================================================================== centred even / odd variant (the default path)
// |X_k| does not change when the time origin of a frame moves to its centre sample (a phase factor of modulus 1).  About
// that centre the periodic Hann window is even (g[m] = hann[200 + m] = g[-m], hann[0] = 0), so with
//     E[m] = x[200 + m] + x[200 - m],   O[m] = x[200 + m] - x[200 - m],   m = 0 .. 199
//     Re Y_k = sum_m E[m] g[m] cos(2 pi k m / 512) (the m = 0 weight halved),   Im Y_k = -sum_m O[m] g[m] sin(2 pi k m / 512)
// the DFT is two GEMMs with K = 200 (13 steps of 16) and N = 120 bins each instead of one with K = 400 and N = 240: half
// the tensor-core work.  The price: E and O are not strided views of the waveform, so the A tiles are built by hand.
// The raw samples of a stage arrive by TMA (two boxes of the overlapping-rows view of the caller's waveform, no split
// pass over HBM) in the region the operand planes will occupy; eight producer warps read them, form E and O in fp32,
// split them and write the planes in the no-swizzle core-matrix layout (8 rows x 16 bytes per core matrix, K chunks
// 160 bytes apart).  The basis tiles arrive by TMA as well (64-byte swizzle).
// Operand precision: both operands are split into TWO fp16 terms (v = hi + lo, 22 mantissa bits; fp16 rather than bf16
// because 2 x 11 bits need three products where 3 x 8 bits need six) and the three products lo*hi, hi*lo, hi*hi are
// accumulated in one fp32 TMEM accumulator, smallest first.  ncu on the six-product bf16 version of this kernel showed
// the shared-memory pipe at 92 % with the tensor pipe at 41 %: every tcgen05.mma re-reads its A and B tiles from shared
// memory (8 KB per 64 tensor cycles at N = 128), so the number of MMA instructions, not the flops, is what is paid for.
// Per frame tile (128 frames) and N-tile (120 bins): TMEM columns [0, 128) = Re, [128, 256) = Im (columns 120..127 of
// each are zero padding); 7 K-blocks of 32 (the last one issues a single K step), each 2 parts x 3 products.
// 576 threads: warps 0-7 A producers, warp 8 TMA (raw sample tiles and basis), warp 9 MMA issuer, warps 10-13 / 14-17
// epilogue of N-tile 0 / 1.
constexpr int eoHalf = kWin / 2;                 // 200 centred lags
constexpr int eoBK = 32;                         // K block (lags per stage)
constexpr int eoKB = 7;                          // blocks 0..6 cover lags 0..223; block 6 issues one K step (192..207)
constexpr int eoKPad = eoKB * eoBK;              // 224 columns in the basis table (zero from lag 200 on)
constexpr int eoTN = 128;                        // accumulator columns per part: 120 bins + 8 zero columns
constexpr int eoPlanes = 2;                      // fp16 hi, lo
constexpr int eoLbo = 160;                       // bytes between the 16-byte K chunks of one 8-row group: 128 + 32, so that
                                                 // the four chunks a half-warp writes at once fall into different banks
constexpr int eoSbo = (eoBK / 8) * eoLbo;        // 640 bytes between 8-row groups
constexpr int eoATile = (kTM / 8) * eoSbo;       // 10240 B: one fp16 plane of the 128 x 32 A tile (core-matrix layout)
constexpr int eoBTile = kTM * eoBK * 2;          // 8192 B: one fp16 plane of the 128 x 32 basis tile (64-byte swizzle)
constexpr int eoABytes = 2 * eoPlanes * eoATile; // E_hi E_lo O_hi O_lo
constexpr int eoBBytes = 2 * eoPlanes * eoBTile; // C_hi C_lo S_hi S_lo
constexpr int eoStageBytes = eoABytes + eoBBytes;      // 72 KB
constexpr int eoStages = 3;
constexpr int eoRawTile = kTM * eoBK * 4;        // 16 KB: the forward raw fp32 sample tile; it and the backward one (18 KB) land
                                                 // in the A region of a stage (4 x 10 KB) before the producers turn them
                                                 // into the four planes
constexpr float eoScaleA = 4096.f;               // E, O and the basis are scaled by powers of two so that the lo planes
constexpr double eoScaleB = 1024.0;              // stay clear of the fp16 subnormal range; undone exactly in the epilogue
constexpr float eoUnscale = 1.0f / (4096.f * 1024.f);
constexpr int eoProdWarps = 8;
constexpr int eoTmaWarp = eoProdWarps, eoMmaWarp = eoProdWarps + 1, eoEpiWarp0 = eoProdWarps + 2;
constexpr int eoThreads = (eoEpiWarp0 + 8) * 32; // 576
constexpr int eoSmemBytes = 1024 + eoStages * eoStageBytes + 512 + 2 * kTM * kHandFloats * 4;

// K-major, no swizzle: element (row r, 16-byte chunk j) at (r / 8) * SBO + j * LBO + (r % 8) * 16
__device__ __forceinline__ uint64_t umma_desc_kmajor_cores(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(eoLbo >> 4) << 16;
  d |= static_cast<uint64_t>(eoSbo >> 4) << 32;
  d |= 1ull << 46;
  return d;
}

// Raw sample tiles of one stage, landed in shared memory by TMA (two boxes of the overlapping-rows view of the waveform:
// row = frame, 160 samples apart): fwd[r][l] = x[lag 32 kb + l] to the right of the centre sample, bwd[r][l] = the
// sample at lag 32 kb + 32 - l to its left (the box runs forwards in memory, so the lags run backwards in it).  Elements
// outside the frame (lags >= 200 at either end) and frames past the end of the clip are zero-filled by TMA.
// Each lane converts four consecutive lags of one frame: one 16-byte (fp32) or 8-byte (PCM) read from either tile.
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
constexpr float eoPcmScale = eoScaleA / 32768.0f;
__device__ __forceinline__ float pcm_lo(uint32_t w) { return static_cast<float>(static_cast<int16_t>(w & 0xffffu)) * eoPcmScale; }
__device__ __forceinline__ float pcm_hi(uint32_t w) { return static_cast<float>(static_cast<int32_t>(w) >> 16) * eoPcmScale; }
// TMA box starts must be 16-byte aligned in global memory, and a mirrored group of four lags starts one element off
// a four-element boundary, so the backward box is 4 (fp32) / 8 (PCM) elements wider than it needs to be: column l of
// it holds lag 32 kb + 32 - l, a lane reads columns 28 - 4 c4 .. 31 - 4 c4 (aligned) plus column 32 - 4 c4.
template <class IN> struct RawLags;
template <> struct RawLags<float> {
  uint4 f, b;
  uint32_t s;
  static constexpr int kRowBytes = eoBK * 4, kBwdCols = eoBK + 4, kBwdRowBytes = kBwdCols * 4;
  __device__ __forceinline__ void read(uint32_t fwd, uint32_t bwd, int row, int c4) {
    f = lds128(fwd + row * kRowBytes + c4 * 16);
    b = lds128(bwd + row * kBwdRowBytes + (7 - c4) * 16);       // lags m+4, m+3, m+2, m+1
    s = lds32(bwd + row * kBwdRowBytes + (8 - c4) * 16);        // lag m
  }
  // xp keeps its scale factor for the fused multiply-add that forms E and O; xm is scaled here
  __device__ __forceinline__ void unpack(float (&xp)[4], float (&xm)[4]) const {
    xp[0] = __uint_as_float(f.x); xp[1] = __uint_as_float(f.y); xp[2] = __uint_as_float(f.z); xp[3] = __uint_as_float(f.w);
    xm[0] = __uint_as_float(s) * eoScaleA; xm[1] = __uint_as_float(b.w) * eoScaleA;
    xm[2] = __uint_as_float(b.z) * eoScaleA; xm[3] = __uint_as_float(b.y) * eoScaleA;
  }
  static constexpr float xp_scale = eoScaleA;
};
template <> struct RawLags<int16_t> {
  uint2 f, b;
  uint32_t s;
  static constexpr int kRowBytes = eoBK * 2, kBwdCols = eoBK + 8, kBwdRowBytes = kBwdCols * 2;
  __device__ __forceinline__ void read(uint32_t fwd, uint32_t bwd, int row, int c4) {
    f = lds64(fwd + row * kRowBytes + c4 * 8);
    b = lds64(bwd + row * kBwdRowBytes + (7 - c4) * 8);         // lags m+4, m+3, m+2, m+1
    s = lds32(bwd + row * kBwdRowBytes + (8 - c4) * 8);         // lag m in the low half
  }
  __device__ __forceinline__ void unpack(float (&xp)[4], float (&xm)[4]) const {
    xp[0] = pcm_lo(f.x); xp[1] = pcm_hi(f.x); xp[2] = pcm_lo(f.y); xp[3] = pcm_hi(f.y);
    xm[0] = pcm_lo(s); xm[1] = pcm_hi(b.y); xm[2] = pcm_lo(b.y); xm[3] = pcm_hi(b.x);
  }
  static constexpr float xp_scale = 1.0f;
};

// v ~ hi + lo (two fp16 terms, 22 mantissa bits; the residual v - hi is exact in fp32), two values per register
__device__ __forceinline__ void split2_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(v0, v1);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const __half2 l = __floats2half2_rn(v0 - __low2float(h), v1 - __high2float(h));
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ void st_shared_v2(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

struct LogmelEoParams {
  long long frames_out;     // frames written per clip
  int tiles_per_clip;       // ceil(frames_out / 128)
  long long total_tiles;    // n_clips * tiles_per_clip
  float* out;               // [n_clips][frames_out][64]
  uint32_t* exact_list;     // flagged frames (tile * 128 + row in the tile) for logmel_exact_kernel, see kExactRatio
  unsigned* exact_count;    // entry count, zeroed by the host before the launch
};

// The band walk of the epilogue with everything about the mel layout resolved at compile time.  kBandOfBin is the
// interval index of every evaluated bin (bin kBinLo + i feeds band e - 1 on its falling side and band e on its rising
// side) for the reference's fixed parameters (16 kHz, 512-point DFT, 64 HTK bands 125..7500 Hz); build_tables() compares
// it with the layout derived from the float64 mel matrix and refuses to run on a mismatch.  With static bin indices the
// weights are constant-bank operands of the FFMAs, the places where a band completes are known, and so is the slot of
// the 16-byte output group it lands in: no loads, no branches, ~7 instructions per bin.  (The first version walked with
// run-time tables: ~30 instructions and four branches per bin made the epilogue, not the tensor pipe, the limiter.)
constexpr unsigned char kBandOfBin[kEvalBins] = {
    0, 1, 2, 3, 3, 4, 5, 6, 7, 8, 9, 9, 10, 11, 12, 12, 13, 14, 14, 15, 15, 16, 17, 17, 18, 18, 19, 19, 20, 20,
    21, 21, 22, 22, 23, 23, 24, 24, 25, 25, 26, 26, 26, 27, 27, 28, 28, 28, 29, 29, 30, 30, 30, 31, 31, 31, 32,
    32, 32, 33, 33, 33, 34, 34, 34, 35, 35, 35, 36, 36, 36, 36, 37, 37, 37, 38, 38, 38, 38, 39, 39, 39, 39, 40,
    40, 40, 41, 41, 41, 41, 41, 42, 42, 42, 42, 43, 43, 43, 43, 44, 44, 44, 44, 44, 45, 45, 45, 45, 46, 46, 46,
    46, 46, 47, 47, 47, 47, 47, 48, 48, 48, 48, 48, 49, 49, 49, 49, 49, 49, 50, 50, 50, 50, 50, 51, 51, 51, 51,
    51, 51, 52, 52, 52, 52, 52, 52, 53, 53, 53, 53, 53, 53, 54, 54, 54, 54, 54, 54, 55, 55, 55, 55, 55, 55, 55,
    56, 56, 56, 56, 56, 56, 56, 57, 57, 57, 57, 57, 57, 57, 58, 58, 58, 58, 58, 58, 58, 59, 59, 59, 59, 59, 59,
    59, 59, 60, 60, 60, 60, 60, 60, 60, 60, 61, 61, 61, 61, 61, 61, 61, 61, 62, 62, 62, 62, 62, 62, 62, 62, 62,
    63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

struct WalkState {
  float lo, hi;       // running sums of band e - 1 (complete after its falling side) and band e
  float pend[4];      // finished bands of the current group of four, waiting for one 16-byte store
  float e2;           // sum of |X_k|^2 over the bins walked so far
  float mn;           // smallest finished band sum
};

template <int E>   // close interval E: band E - 1 is complete
__device__ __forceinline__ void emit_static(WalkState& w, float* __restrict__ row_out, bool valid) {
  constexpr int band = E - 1;
  if constexpr (band >= 0 && band < kMel) {
    w.pend[band & 3] = __logf(w.lo + kLogOffset);
    w.mn = fminf(w.mn, w.lo);
    if constexpr ((band & 3) == 3) {
      if (valid) *reinterpret_cast<float4*>(row_out + band - 3) = make_float4(w.pend[0], w.pend[1], w.pend[2], w.pend[3]);
    }
  }
  w.lo = w.hi;
  w.hi = 0.f;
}

template <int G0, int J, int NB, int E>   // bin J of the NB-bin chunk that starts at table index G0; current interval E
__device__ __forceinline__ void walk_static(WalkState& w, const float (&mag)[NB], float* __restrict__ row_out, bool valid) {
  if constexpr (J < NB) {
    constexpr int g = G0 + J;
    constexpr int e = kBandOfBin[g];
    static_assert(e == E || e == E + 1, "a bin closes at most one band");
    if constexpr (e > E) emit_static<E>(w, row_out, valid);
    w.lo = fmaf(c_wfall[g], mag[J], w.lo);
    w.hi = fmaf(c_wrise[g], mag[J], w.hi);
    w.e2 = fmaf(mag[J], mag[J], w.e2);
    walk_static<G0, J + 1, NB, e>(w, mag, row_out, valid);
  }
}

template <int E>
__device__ __forceinline__ void flush_static(WalkState& w, float* __restrict__ row_out, bool valid) {
  if constexpr (E <= kMel) {
    emit_static<E>(w, row_out, valid);
    flush_static<E + 1>(w, row_out, valid);
  }
}

constexpr int eoChunkBins = 8;
constexpr int eoChunks = kTileBins / eoChunkBins;   // 15

// Chunk CH of N-tile SET: on entry the TMEM loads of its 8 Re and 8 Im columns are in flight in re / im; the next
// chunk's loads are issued as soon as the magnitudes have been formed, so they overlap the walk.
template <int SET, int CH>
__device__ __forceinline__ void epilogue_chunks(uint32_t t_addr, uint32_t (&re)[8], uint32_t (&im)[8], WalkState& w,
                                                float* __restrict__ row_out, bool valid) {
  tmem_ld_wait();
  float mag[eoChunkBins];
#pragma unroll
  for (int j = 0; j < eoChunkBins; ++j) {
    const float r = __uint_as_float(re[j]), i = __uint_as_float(im[j]);
    float m;     // sqrt.approx: 2 ulp, far below what the band sums resolve; exact zero stays zero
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(m) : "f"(fmaf(r, r, i * i)));
    mag[j] = m * eoUnscale;                              // exact: the operands carried 2^12 and 2^10
  }
  if constexpr (CH + 1 < eoChunks) {
    tmem_ld_32x8(t_addr + (CH + 1) * eoChunkBins, re);
    tmem_ld_32x8(t_addr + eoTN + (CH + 1) * eoChunkBins, im);
  }
  constexpr int g0 = SET * kTileBins + CH * eoChunkBins;
  constexpr int e0 = g0 == 0 ? 0 : kBandOfBin[g0 - 1];
  walk_static<g0, 0, eoChunkBins, e0>(w, mag, row_out, valid);
  if constexpr (CH + 1 < eoChunks) epilogue_chunks<SET, CH + 1>(t_addr, re, im, w, row_out, valid);
}

template <class IN>
__global__ void __launch_bounds__(eoThreads, 1)
logmel_eo_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_xb,
                 const __grid_constant__ CUtensorMap tmap_b, const LogmelEoParams p) {
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + eoStages * eoStageBytes);
  uint64_t* empty_bar = full_bar + eoStages;
  uint64_t* tmem_full = empty_bar + eoStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* hand_full = tmem_empty + 2;       // [2 buffers][4 lane quarters]
  uint64_t* hand_empty = hand_full + 8;
  uint64_t* raw_full = hand_empty + 8;        // [eoStages]: the raw sample tiles of the stage have landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_full + eoStages);
  float* hand = reinterpret_cast<float*>(smem + eoStages * eoStageBytes + 512);   // [2][kTM][kHandFloats]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == eoTmaWarp && lane == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_xb);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < eoStages; ++s) {
      mbar_init(&full_bar[s], eoProdWarps * 32 + 1);   // every producer thread + the TMA thread's expect_tx
      mbar_init(&empty_bar[s], 1);
      mbar_init(&raw_full[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 4);
    }
    for (int s = 0; s < 8; ++s) {
      mbar_init(&hand_full[s], 1);
      mbar_init(&hand_empty[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == eoMmaWarp) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform by construction
  pdl_wait();   // the waveform may have been written by the previous kernel in the stream

  if (warp < eoProdWarps) {
    // ------------------------------------------------------------------ A producers: E / O planes of 16 frames per warp
    // lane = (row within a 4-row group, 4 lags).  The raw sample tiles of the stage arrive by TMA in the very region
    // the operand planes go to, so the conversion is: read (all producers) -> named barrier -> write.  A half-warp's
    // 8-byte plane stores cover all 32 banks (LBO = 160), a quarter-warp's raw read is one contiguous row.
    const int rs = lane >> 3, c4 = lane & 7;
    const uint32_t lane_off = warp * 2 * eoSbo + rs * 16 + (c4 >> 1) * eoLbo + (c4 & 1) * 8;
    uint32_t stage = 0, phase = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      for (int nt = 0; nt < kNTiles; ++nt) {
        for (int kb = 0; kb < eoKB; ++kb) {
          const uint32_t a_base = smem_u32(smem + stage * eoStageBytes);
          mbar_wait(&raw_full[stage], phase);
          RawLags<IN> raw[4];
#pragma unroll
          for (int it = 0; it < 4; ++it) raw[it].read(a_base, a_base + eoRawTile, warp * 16 + it * 4 + rs, c4);
          asm volatile("bar.sync 1, %0;" ::"n"(eoProdWarps * 32) : "memory");   // every raw row has been read
          if (kb < eoKB - 1 || c4 < 4) {                   // chunks from lag 208 on are never read by an MMA
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              float xp[4], xm[4];
              raw[it].unpack(xp, xm);
              uint32_t eh[2], el[2], oh[2], ol[2];
#pragma unroll
              for (int t = 0; t < 2; ++t) {
                constexpr float sc = RawLags<IN>::xp_scale;
                split2_pair(fmaf(xp[2 * t], sc, xm[2 * t]), fmaf(xp[2 * t + 1], sc, xm[2 * t + 1]), eh[t], el[t]);
                split2_pair(fmaf(xp[2 * t], sc, -xm[2 * t]), fmaf(xp[2 * t + 1], sc, -xm[2 * t + 1]), oh[t], ol[t]);
              }
              // rows 16 * warp + 4 * it + rs: 8-row group 2 * warp + (it >> 1), row (it & 1) * 4 + rs within it
              const uint32_t dst = a_base + lane_off + (it >> 1) * eoSbo + (it & 1) * 64;
              st_shared_v2(dst + 0 * eoATile, eh[0], eh[1]);
              st_shared_v2(dst + 1 * eoATile, el[0], el[1]);
              st_shared_v2(dst + 2 * eoATile, oh[0], oh[1]);
              st_shared_v2(dst + 3 * eoATile, ol[0], ol[1]);
            }
          }
          fence_proxy_async_smem();        // generic-proxy smem writes -> visible to the tensor core (async proxy)
          mbar_arrive(&full_bar[stage]);
          if (++stage == eoStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == eoTmaWarp) {
    // ------------------------------------------------------------------ raw sample tiles and basis tiles by TMA
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int clip = static_cast<int>(tile / p.tiles_per_clip);
        const int row0 = static_cast<int>(tile - static_cast<long long>(clip) * p.tiles_per_clip) * kTM;
        for (int nt = 0; nt < kNTiles; ++nt) {
          for (int kb = 0; kb < eoKB; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* a_base = smem + stage * eoStageBytes;
            uint8_t* b_base = a_base + eoABytes;
            // samples eoHalf + 32 kb .. + 31 of every frame, and eoHalf - 32 kb - 32 .. eoHalf - 32 kb (+ padding)
            mbar_expect_tx(&raw_full[stage], kTM * (RawLags<IN>::kRowBytes + RawLags<IN>::kBwdRowBytes));
            tma_load_3d(a_base, &tmap_x, &raw_full[stage], eoHalf + kb * eoBK, row0, clip);
            tma_load_3d(a_base + eoRawTile, &tmap_xb, &raw_full[stage], eoHalf - kb * eoBK - eoBK, row0, clip);
            mbar_expect_tx(&full_bar[stage], eoBBytes);
#pragma unroll
            for (int t = 0; t < 2 * eoPlanes; ++t)   // tile t = part * 2 + plane; table rows ((plane * 2 + part) * 2 + nt) * 128
              tma_load_2d(b_base + t * eoBTile, &tmap_b, &full_bar[stage], kb * eoBK,
                          (((t % eoPlanes) * 2 + t / eoPlanes) * kNTiles + nt) * eoTN);
            if (++stage == eoStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == eoMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = umma_idesc_f16_f32(kTM, eoTN);
    uint32_t stage = 0, phase = 0, it = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      for (int nt = 0; nt < kNTiles; ++nt, ++it) {
        const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = 0; kb < eoKB; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after_sync();
          if (elect_one()) {
            const uint32_t a0 = smem_u32(smem + stage * eoStageBytes);
            const uint32_t b0 = a0 + eoABytes;
            const int nks = (kb == eoKB - 1) ? 1 : 2;
            // products (a plane, b plane), smallest magnitude first
            constexpr int prod_a[3] = {1, 0, 0};
            constexpr int prod_b[3] = {0, 1, 0};
#pragma unroll
            for (int part = 0; part < 2; ++part) {       // E x C -> Re columns, O x S -> Im columns
#pragma unroll
              for (int q = 0; q < 3; ++q) {
                const uint64_t a_desc = umma_desc_kmajor_cores(a0 + (part * eoPlanes + prod_a[q]) * eoATile);
                const uint64_t b_desc = umma_desc_kmajor_sw64(b0 + (part * eoPlanes + prod_b[q]) * eoBTile);
#pragma unroll
                for (int k = 0; k < 2; ++k)   // K step 16 lags: two chunks = 2 * LBO in A, 32 bytes in the swizzled B row
                  if (k < nks)
                    umma_bf16_ss(d_tmem + part * eoTN, a_desc + k * (2 * eoLbo >> 4), b_desc + 2 * k, idesc,
                                 (kb | q | k) != 0);
              }
            }
            umma_commit(&empty_bar[stage]);
            if (kb == eoKB - 1) umma_commit(&tmem_full[acc]);
          }
          __syncwarp();
          if (++stage == eoStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    // Two sets of four warps: set 0 (warps 10-13) walks the bins of N-tile 0, set 1 (warps 14-17) those of N-tile 1.
    // The band walk is sequential over the bins, so warp q of set 0 hands its per-row state to warp q of set 1 through
    // shared memory; the arithmetic and its order are exactly those of a single walk.
    const int set = (warp - eoEpiWarp0) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    uint32_t mi = 0;   // frame-tile iteration of this CTA
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++mi) {
      const long long clip = tile / p.tiles_per_clip;
      const long long frame = (tile - clip * p.tiles_per_clip) * kTM + row;
      const bool valid = frame < p.frames_out;
      float* row_out = p.out + (clip * p.frames_out + (valid ? frame : 0)) * kMel;
      const uint32_t hb = mi & 1, hphase = (mi >> 1) & 1;
      float* hrow = hand + (hb * kTM + row) * kHandFloats;
      const uint32_t acc = set, acc_phase = mi & 1;
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * 256;
      WalkState w;
      uint32_t re[8], im[8];
      if (set == 0) {
        w.lo = w.hi = 0.f;
        w.pend[0] = w.pend[1] = w.pend[2] = w.pend[3] = 0.f;
        w.e2 = 0.f;
        w.mn = 3.0e38f;
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after_sync();
        tmem_ld_32x8(t_addr, re);
        tmem_ld_32x8(t_addr + eoTN, im);
        epilogue_chunks<0, 0>(t_addr, re, im, w, row_out, valid);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        mbar_wait(&hand_empty[hb * 4 + q], hphase ^ 1);
        hrow[0] = w.lo; hrow[1] = w.hi;
        hrow[2] = w.pend[0]; hrow[3] = w.pend[1]; hrow[4] = w.pend[2]; hrow[5] = w.pend[3];
        hrow[6] = w.e2; hrow[7] = w.mn;
        __syncwarp();
        if (lane == 0) mbar_arrive(&hand_full[hb * 4 + q]);
      } else {
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after_sync();
        tmem_ld_32x8(t_addr, re);
        tmem_ld_32x8(t_addr + eoTN, im);
        mbar_wait(&hand_full[hb * 4 + q], hphase);
        w.lo = hrow[0]; w.hi = hrow[1];
        w.pend[0] = hrow[2]; w.pend[1] = hrow[3]; w.pend[2] = hrow[4]; w.pend[3] = hrow[5];
        w.e2 = hrow[6]; w.mn = hrow[7];
        __syncwarp();
        if (lane == 0) mbar_arrive(&hand_empty[hb * 4 + q]);
        epilogue_chunks<1, 0>(t_addr, re, im, w, row_out, valid);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        flush_static<kBandOfBin[kEvalBins - 1]>(w, row_out, valid);   // the remaining bands (up to band 63)
        const float lim = kExactRatio * (w.mn + kLogOffset);
        const bool mine = valid && w.e2 > lim * lim;
        const uint32_t bad = __ballot_sync(0xffffffffu, mine);
        if (bad) {   // one atomic per warp reserves the slots, every flagged frame writes its own entry
          uint32_t base = 0;
          if (lane == 0) base = atomicAdd(p.exact_count, static_cast<unsigned>(__popc(bad)));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (mine) p.exact_list[base + __popc(bad & ((1u << lane) - 1u))] = static_cast<uint32_t>(tile * kTM + row);
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == eoMmaWarp) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ================================================================== float64 path for the flagged frames
// The same centred even / odd DFT in float64 on the CUDA cores.  The epilogues of the tensor-core kernels append every
// flagged frame to a list (one atomicAdd per warp; the order of the list varies from run to run, the results do not:
// every frame is computed on its own).  One CTA per SM takes the list 8 frames at a time: E, O of the 8 frames in shared
// memory ([lag][frame]: the frames of a lag are broadcast reads), thread = (DFT bin, 2 of the 8 frames).  The float64
// basis (768 KB, L2-resident) is streamed through a four-stage shared-memory ring by 1-D bulk copies, 10 lags per
// stage — register-staged loads left the loop bound by one L2 round trip per pair of lags (33 us per pass; the copies
// take it to the L2 -> SM bandwidth).  Follows mel_features.py:86-92, :215-223 to ~1e-13, so the fp32 output is the
// float64 reference rounded once.  An empty list costs one 4-byte read per CTA.
constexpr int kExactFrames = 8;      // frames per pass.  Measured: a pass costs ~26 us + 2 us per frame (float64 FMAs), so
                                     // with ~800 flagged frames in a batch small passes on all SMs beat big ones (8 per
                                     // pass: 42 us, 16 per pass: 58 us for the bench batch)
constexpr int kExactThreads = 1024;  // thread = (bin [256, 240 used], two of the 8 frames)
constexpr int kExactLags = 10;       // lags per basis stage
constexpr int kExactStages = 4;      // three chunks in flight while one is being consumed
constexpr int kExactStageBytes = 2 * kExactLags * kEvalBins * 8;   // cos rows | sin rows: 38 400 B
constexpr int kExactSmem = kExactStages * kExactStageBytes + 2 * eoHalf * kExactFrames * 8 + kExactFrames * kEvalBins * 8 + kExactFrames * 8;

struct ExactParams {
  long long frames_out;
  int tiles_per_clip;
  long long clip_stride;        // samples
  const uint32_t* list;         // flagged frames: tile * 128 + row
  const unsigned* count;
  const double* basis;          // [2: cos, sin][200 lags][240 bins]
  const double* mel;            // [240 bins][64 bands]
  float* out;                   // [n_clips][frames_out][64]
};

template <class IN>
__device__ __forceinline__ double load_sample_f64(const IN* p);
template <>
__device__ __forceinline__ double load_sample_f64<float>(const float* p) { return static_cast<double>(__ldg(p)); }
template <>
__device__ __forceinline__ double load_sample_f64<int16_t>(const int16_t* p) { return static_cast<double>(__ldg(p)) / 32768.0; }

template <class IN>
__global__ void __launch_bounds__(kExactThreads)
logmel_exact_kernel(const IN* __restrict__ wave, const ExactParams p) {
  extern __shared__ __align__(128) uint8_t exact_smem[];
  double* ring = reinterpret_cast<double*>(exact_smem);                               // [4][cos 10 x 240 | sin 10 x 240]
  double* E = reinterpret_cast<double*>(exact_smem + kExactStages * kExactStageBytes);  // [200][8]
  double* O = E + eoHalf * kExactFrames;                                                // [200][8]
  double* mag = O + eoHalf * kExactFrames;                                              // [8][240]
  long long* frame_of = reinterpret_cast<long long*>(mag + kExactFrames * kEvalBins);   // [8] clip * frames_out + frame
  __shared__ uint64_t full_bar[kExactStages];
  const int tid = threadIdx.x;
  pdl_launch_dependents();
  if (tid == 0) {
    for (int s = 0; s < kExactStages; ++s) mbar_init(&full_bar[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  pdl_wait();   // the list (and the rows this kernel overwrites) come from the tensor-core kernel before it
  const unsigned n_frames = *reinterpret_cast<const volatile unsigned*>(p.count);
  constexpr int kChunks = eoHalf / kExactLags;   // 20
  uint32_t fills = 0;                            // bulk copies issued so far (thread 0), chunks consumed so far (all)
  uint32_t used = 0;
  auto issue = [&](int chunk) {                  // thread 0 only
    const uint32_t s = fills % kExactStages;
    double* dst = ring + s * (kExactStageBytes / 8);
    mbar_expect_tx(&full_bar[s], kExactStageBytes);
    bulk_load_1d(dst, p.basis + chunk * kExactLags * kEvalBins, kExactStageBytes / 2, &full_bar[s]);
    bulk_load_1d(dst + kExactLags * kEvalBins, p.basis + (eoHalf + chunk * kExactLags) * kEvalBins, kExactStageBytes / 2,
                 &full_bar[s]);
    ++fills;
  };
  for (unsigned g0 = blockIdx.x * kExactFrames; g0 < n_frames; g0 += gridDim.x * kExactFrames) {
    const int ng = n_frames - g0 < kExactFrames ? static_cast<int>(n_frames - g0) : kExactFrames;
    if (tid == 0) {
      for (int c = 0; c < kExactStages - 1; ++c) issue(c);
    }
    if (tid < kExactFrames) {
      long long fo = -1;
      if (tid < ng) {
        const uint32_t id = __ldg(p.list + g0 + tid);
        const long long tile = id / kTM;
        const long long clip = tile / p.tiles_per_clip;
        fo = clip * p.frames_out + (tile - clip * p.tiles_per_clip) * kTM + (id % kTM);
      }
      frame_of[tid] = fo;
    }
    __syncthreads();
    // E[m][f] = x[200 + m] + x[200 - m], O[m][f] = x[200 + m] - x[200 - m] (lag 0: E = 2 x[200], its weight is halved)
    for (int i = tid; i < eoHalf * kExactFrames; i += kExactThreads) {
      const int f = i / eoHalf, m = i - f * eoHalf;
      double e = 0.0, o = 0.0;
      const long long fo = frame_of[f];
      if (fo >= 0) {
        const long long clip = fo / p.frames_out;
        const IN* x = wave + clip * p.clip_stride + (fo - clip * p.frames_out) * kHop + eoHalf;
        const double xp = load_sample_f64<IN>(x + m), xm = load_sample_f64<IN>(x - m);
        e = xp + xm;
        o = xp - xm;
      }
      E[m * kExactFrames + f] = e;
      O[m * kExactFrames + f] = o;
    }
    __syncthreads();
    const int bin = tid & 255, f0 = (tid >> 8) * 2;
    const int bsafe = bin < kEvalBins ? bin : 0;
    double re0 = 0.0, re1 = 0.0, im0 = 0.0, im1 = 0.0;
    for (int ch = 0; ch < kChunks; ++ch, ++used) {
      // the stage of chunk ch - 1 was released by the barrier at the end of the previous iteration: refill it
      if (tid == 0 && ch + kExactStages - 1 < kChunks) issue(ch + kExactStages - 1);
      const uint32_t s = used % kExactStages;
      mbar_wait(&full_bar[s], (used / kExactStages) & 1);
      const double* cs = ring + s * (kExactStageBytes / 8) + bsafe;
      const double* sn = cs + kExactLags * kEvalBins;
      const double* e = E + ch * kExactLags * kExactFrames + f0;
      const double* o = O + ch * kExactLags * kExactFrames + f0;
#pragma unroll
      for (int u = 0; u < kExactLags; ++u) {
        const double c = cs[u * kEvalBins], sv = sn[u * kEvalBins];
        const double2 ev = *reinterpret_cast<const double2*>(e + u * kExactFrames);
        const double2 ov = *reinterpret_cast<const double2*>(o + u * kExactFrames);
        re0 = fma(ev.x, c, re0);
        re1 = fma(ev.y, c, re1);
        im0 = fma(ov.x, sv, im0);
        im1 = fma(ov.y, sv, im1);
      }
      __syncthreads();                                   // every thread is done with stage s
    }
    if (bin < kEvalBins) {
      mag[f0 * kEvalBins + bin] = sqrt(re0 * re0 + im0 * im0);
      mag[(f0 + 1) * kEvalBins + bin] = sqrt(re1 * re1 + im1 * im1);
    }
    __syncthreads();
    {
      // (frame, band) = a pair of lanes: even bins of the band's run on one, odd bins on the other, summed by shuffle
      // (band `band` has weight on a short run of bins only — HTK triangles: [c_mel_lo, c_mel_hi))
      const int i = tid >> 1, par = tid & 1;
      const int f = i / kMel, band = i - f * kMel;
      const long long fo = frame_of[f];
      double acc = 0.0;
      if (fo >= 0) {
        const double* mg = mag + f * kEvalBins;
        const int b_lo = c_mel_lo[band], b_hi = c_mel_hi[band];
#pragma unroll 4
        for (int b = b_lo + par; b < b_hi; b += 2) acc = fma(mg[b], __ldg(p.mel + b * kMel + band), acc);
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      if (fo >= 0 && par == 0) p.out[fo * kMel + band] = static_cast<float>(log(acc + 0.01));
    }
    __syncthreads();
  }
}

template <class IN>
int launch_exact(const IN* wave, long long clip_stride, long long frames_out, int tiles_per_clip, const uint32_t* list,
                 const unsigned* count, const double* basis, const double* mel, float* out, cudaStream_t stream) {
  ExactParams e{};
  e.frames_out = frames_out;
  e.tiles_per_clip = tiles_per_clip;
  e.clip_stride = clip_stride;
  e.list = list;
  e.count = count;
  e.basis = basis;
  e.mel = mel;
  e.out = out;
  const cudaError_t le = launch_pdl(logmel_exact_kernel<IN>, dim3(static_cast<unsigned>(num_sms())), dim3(kExactThreads),
                                    kExactSmem, stream, wave, e);
  count_launch();
  if (le != cudaSuccess) {
    set_kernel_error("logmel_exact_kernel: %s", cudaGetErrorString(le));
    return 1;
  }
  return check_launch("logmel_exact_kernel");
}

// The flag list of one launch: [count (16 bytes)][one entry per frame]; the count is zeroed on the stream.
int alloc_exact_list(long long total_tiles, cudaStream_t stream, void** buf) {
  if (cudaMallocAsync(buf, 16 + size_t(total_tiles) * kTM * sizeof(uint32_t), stream) != cudaSuccess ||
      cudaMemsetAsync(*buf, 0, 16, stream) != cudaSuccess) {
    set_kernel_error("logmel: flag list allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  return 0;
}

// ================================================================== stft_magnitude (mel_features.py:71-92) on its own
// |rfft(frame * hann, 512)| for all 257 bins in float64: the reference's standalone function returns float64, and the
// fused log-mel kernel never materialises the magnitudes (it evaluates bins 4..243 only), so the drop-in gets the same
// centred even / odd DFT as logmel_exact_kernel over the whole bin range.  16 frames per CTA, thread = bin.
constexpr int kStftThreads = 288;   // 9 warps: bins 0..256
constexpr int kStftFrames = 8;      // frames per CTA (E, O in static shared memory: 25.6 KB)

__global__ void __launch_bounds__(kStftThreads)
stft_magnitude_kernel(const double* __restrict__ signal, long long n_frames, const double* __restrict__ basis,
                      double* __restrict__ out) {
  __shared__ __align__(16) double E[eoHalf * kStftFrames];
  __shared__ __align__(16) double O[eoHalf * kStftFrames];
  const int tid = threadIdx.x;
  const long long f0 = static_cast<long long>(blockIdx.x) * kStftFrames;
  const int ng = n_frames - f0 < kStftFrames ? static_cast<int>(n_frames - f0) : kStftFrames;
  for (int i = tid; i < eoHalf * kStftFrames; i += kStftThreads) {
    const int f = i / eoHalf, m = i - f * eoHalf;
    double e = 0.0, o = 0.0;
    if (f < ng) {
      const double* x = signal + (f0 + f) * kHop + eoHalf;
      const double xp = __ldg(x + m), xm = __ldg(x - m);
      e = xp + xm;
      o = xp - xm;
    }
    E[m * kStftFrames + f] = e;
    O[m * kStftFrames + f] = o;
  }
  __syncthreads();
  if (tid >= kBins) return;
  double re[kStftFrames], im[kStftFrames];
#pragma unroll
  for (int f = 0; f < kStftFrames; ++f) re[f] = im[f] = 0.0;
  const double* bc = basis + tid;
  const double* bs = basis + eoHalf * kBins + tid;
#pragma unroll 2
  for (int m = 0; m < eoHalf; ++m) {
    const double c = __ldg(bc + m * kBins), sn = __ldg(bs + m * kBins);
    const double2* e2 = reinterpret_cast<const double2*>(E + m * kStftFrames);
    const double2* o2 = reinterpret_cast<const double2*>(O + m * kStftFrames);
#pragma unroll
    for (int f = 0; f < kStftFrames / 2; ++f) {
      const double2 ev = e2[f], ov = o2[f];
      re[2 * f] = fma(ev.x, c, re[2 * f]);
      re[2 * f + 1] = fma(ev.y, c, re[2 * f + 1]);
      im[2 * f] = fma(ov.x, sn, im[2 * f]);
      im[2 * f + 1] = fma(ov.y, sn, im[2 * f + 1]);
    }
  }
#pragma unroll
  for (int f = 0; f < kStftFrames; ++f)
    if (f < ng) out[(f0 + f) * kBins + tid] = sqrt(re[f] * re[f] + im[f] * im[f]);
}

// ------------------------------------------------------------------ per-device constant tables
struct TcTables {
  __nv_bfloat16* basis = nullptr;  // [3][480][416] bf16: row = 2*bin_index + {cos, sin}, col = sample in frame
  __half* basis_eo = nullptr;      // [2 planes: hi, lo][2 parts: cos, sin][2 N-tiles][128 bins (120 used)][224 lags (200 used)]
  double* basis_f64 = nullptr;     // [2: cos, sin][200 lags][240 bins], centred, Hann folded in (logmel_exact_kernel)
  double* mel_f64 = nullptr;       // [240 bins][64 bands]
  double* basis257 = nullptr;      // [2: cos, sin][200 lags][257 bins] (stft_magnitude_kernel; built on first use)
  bool ready = false;
};
std::mutex g_mu;
TcTables g_tabs[64];

uint16_t bf16_bits(double v, double* back) {
  const __nv_bfloat16 h = __float2bfloat16_rn(static_cast<float>(v));
  *back = static_cast<double>(__bfloat162float(h));
  return __bfloat16_as_ushort(h);
}

int build_tables(TcTables& t) {
  std::vector<double> hann(kWin), mel(size_t(kBins) * kMel);
  front_end_tables_host(hann.data(), mel.data());
  // every bin feeds at most two adjacent bands; anything else (or weight outside the evaluated bins) is an error
  std::vector<int> band(kEvalBins, kMel + 1);
  std::vector<float> wf(kEvalBins, 0.f), wr(kEvalBins, 0.f);
  int prev = 0;
  for (int k = 0; k < kBins; ++k) {
    int first = -1, last = -1, nnz = 0;
    for (int m = 0; m < kMel; ++m)
      if (mel[size_t(k) * kMel + m] != 0.0) {
        if (first < 0) first = m;
        last = m;
        ++nnz;
      }
    const int i = k - kBinLo;
    if (i < 0 || i >= kEvalBins) {
      if (nnz) {
        set_kernel_error("logmel: mel matrix has weight outside the evaluated bins (bin %d)", k);
        return 1;
      }
      continue;
    }
    if (nnz > 2 || (nnz == 2 && last != first + 1)) {
      set_kernel_error("logmel: bin %d feeds non-adjacent mel bands", k);
      return 1;
    }
    // interval index e: the bin feeds band e-1 (falling side) and band e (rising side).  Two weights -> e is the
    // upper band; a lone weight at band c can sit on either side, whichever keeps the walk monotone.
    int e = prev;
    if (nnz == 2) e = last;
    else if (nnz == 1) e = (first >= prev) ? first : first + 1;
    if (e < prev) {
      set_kernel_error("logmel: mel band walk is not monotone at bin %d", k);
      return 1;
    }
    band[i] = e;
    wf[i] = (e - 1 >= 0 && e - 1 < kMel) ? static_cast<float>(mel[size_t(k) * kMel + e - 1]) : 0.f;
    wr[i] = (e < kMel) ? static_cast<float>(mel[size_t(k) * kMel + e]) : 0.f;
    // whatever the interval choice, both non-zero weights of the row must be covered
    for (int m = 0; m < kMel; ++m)
      if (mel[size_t(k) * kMel + m] != 0.0 && m != e - 1 && m != e) {
        set_kernel_error("logmel: bin %d weight for band %d not representable in the two-band walk", k, m);
        return 1;
      }
    prev = e;
  }
  for (int i = 0; i < kEvalBins; ++i)
    if (band[i] != kBandOfBin[i]) {
      set_kernel_error("logmel: compiled mel band layout differs from the float64 tables at bin %d (%d vs %d)", kBinLo + i,
                       int(kBandOfBin[i]), band[i]);
      return 1;
    }
  if (cudaMemcpyToSymbol(c_band, band.data(), sizeof(int) * kEvalBins) != cudaSuccess ||
      cudaMemcpyToSymbol(c_wfall, wf.data(), sizeof(float) * kEvalBins) != cudaSuccess ||
      cudaMemcpyToSymbol(c_wrise, wr.data(), sizeof(float) * kEvalBins) != cudaSuccess) {
    set_kernel_error("logmel: constant table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  const size_t plane = size_t(kEvalBins) * 2 * kKPad;
  std::vector<uint16_t> basis(3 * plane, 0);
  for (int i = 0; i < kEvalBins; ++i)
    for (int n = 0; n < kWin; ++n) {
      const int kn = ((kBinLo + i) * n) % kFft;            // exact argument reduction
      const double ang = 2 * kPi * kn / kFft;
      const double val[2] = {hann[n] * std::cos(ang), hann[n] * std::sin(ang)};
      for (int c = 0; c < 2; ++c) {
        double r = val[c], back;
        for (int pl = 0; pl < 3; ++pl) {
          basis[pl * plane + (size_t(2 * i + c)) * kKPad + n] = bf16_bits(r, &back);
          r -= back;
        }
      }
    }
  void* d = nullptr;
  if (cudaMalloc(&d, basis.size() * 2) != cudaSuccess ||
      cudaMemcpy(d, basis.data(), basis.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) {
    set_kernel_error("logmel: basis upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  t.basis = static_cast<__nv_bfloat16*>(d);
  // centred basis of the even / odd kernel: g[m] cos / sin(2 pi k m / 512), g[m] = hann[200 + m]; the lag-0 cosine
  // weight is halved because E[0] = 2 x[200]
  const size_t rows_eo = size_t(eoPlanes) * 2 * kNTiles * eoTN;
  std::vector<uint16_t> beo(rows_eo * eoKPad, 0);
  for (int nt = 0; nt < kNTiles; ++nt)
    for (int r = 0; r < kTileBins; ++r)
      for (int m = 0; m < eoHalf; ++m) {
        const int km = ((kBinLo + nt * kTileBins + r) * m) % kFft;       // exact argument reduction
        const double ang = 2 * kPi * km / kFft, g = eoScaleB * hann[eoHalf + m] * (m == 0 ? 0.5 : 1.0);
        const double val[2] = {g * std::cos(ang), g * std::sin(ang)};
        for (int c = 0; c < 2; ++c) {
          double rem = val[c];
          for (int pl = 0; pl < eoPlanes; ++pl) {
            const __half h = __float2half_rn(static_cast<float>(rem));
            beo[(size_t((pl * 2 + c) * kNTiles + nt) * eoTN + r) * eoKPad + m] = __half_as_ushort(h);
            rem -= static_cast<double>(__half2float(h));
          }
        }
      }
  void* de = nullptr;
  if (cudaMalloc(&de, beo.size() * 2) != cudaSuccess ||
      cudaMemcpy(de, beo.data(), beo.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) {
    set_kernel_error("logmel: centred basis upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  t.basis_eo = static_cast<__half*>(de);
  // float64 tables of the exact path: the same centred basis unsplit and unscaled, and rows 4..243 of the mel matrix
  std::vector<double> bd(size_t(2) * eoHalf * kEvalBins), md(size_t(kEvalBins) * kMel);
  for (int m = 0; m < eoHalf; ++m)
    for (int i = 0; i < kEvalBins; ++i) {
      const int km = ((kBinLo + i) * m) % kFft;
      const double ang = 2 * kPi * km / kFft, g = hann[eoHalf + m] * (m == 0 ? 0.5 : 1.0);
      bd[size_t(m) * kEvalBins + i] = g * std::cos(ang);
      bd[size_t(eoHalf + m) * kEvalBins + i] = g * std::sin(ang);
    }
  for (int i = 0; i < kEvalBins; ++i)
    for (int b = 0; b < kMel; ++b) md[size_t(i) * kMel + b] = mel[size_t(kBinLo + i) * kMel + b];
  std::vector<int> mlo(kMel, kEvalBins), mhi(kMel, 0);
  for (int i = 0; i < kEvalBins; ++i)
    for (int b = 0; b < kMel; ++b)
      if (md[size_t(i) * kMel + b] != 0.0) {
        mlo[b] = std::min(mlo[b], i);
        mhi[b] = std::max(mhi[b], i + 1);
      }
  if (cudaMemcpyToSymbol(c_mel_lo, mlo.data(), sizeof(int) * kMel) != cudaSuccess ||
      cudaMemcpyToSymbol(c_mel_hi, mhi.data(), sizeof(int) * kMel) != cudaSuccess) {
    set_kernel_error("logmel: band range upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  void *dbd = nullptr, *dmd = nullptr;
  if (cudaMalloc(&dbd, bd.size() * 8) != cudaSuccess || cudaMalloc(&dmd, md.size() * 8) != cudaSuccess ||
      cudaMemcpy(dbd, bd.data(), bd.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(dmd, md.data(), md.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
    set_kernel_error("logmel: float64 table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  t.basis_f64 = static_cast<double*>(dbd);
  t.mel_f64 = static_cast<double*>(dmd);
  t.ready = true;
  return 0;
}

int get_tables(TcTables** out) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
    set_kernel_error("logmel: cudaGetDevice failed");
    return 1;
  }
  std::lock_guard<std::mutex> lk(g_mu);
  TcTables& t = g_tabs[dev];
  if (!t.ready) {
    if (build_tables(t)) return 1;
    if (cudaFuncSetAttribute(logmel_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) != cudaSuccess ||
        cudaFuncSetAttribute(logmel_eo_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, eoSmemBytes) != cudaSuccess ||
        cudaFuncSetAttribute(logmel_eo_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, eoSmemBytes) != cudaSuccess ||
        cudaFuncSetAttribute(logmel_exact_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, kExactSmem) != cudaSuccess ||
        cudaFuncSetAttribute(logmel_exact_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, kExactSmem) != cudaSuccess) {
      set_kernel_error("logmel: cannot raise dynamic shared memory to %d / %d bytes", kSmemBytes, eoSmemBytes);
      return 1;
    }
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      uint64_t keep = ~0ull;   // keep freed workspace in the pool: the next call reuses it without a driver call
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  *out = &t;
  return 0;
}

// last frame reads up to sample 160 (frames - 1) + 415 <= samples + 15; rows of the A tensor map must stay inside the
// plane; a multiple of 160 keeps every stride a multiple of the 320-byte frame stride
long long logmel_tc_pitch(long long samples_per_clip) { return (samples_per_clip + 16 + kHop - 1) / kHop * kHop; }

// The raw sample tiles are TMA boxes, so the clip base and the clip stride must be 16-byte aligned; other inputs
// take the plane kernel, which accepts any alignment.
template <class IN>
bool logmel_eo_accepts(const IN* wave, long long n_clips, long long clip_stride) {
  return reinterpret_cast<uintptr_t>(wave) % 16 == 0 &&
         (n_clips == 1 || (clip_stride * static_cast<long long>(sizeof(IN))) % 16 == 0);
}

template <class IN>
int logmel_eo_forward(TcTables* t, const IN* wave, long long n_clips, long long clip_stride, long long frames_out,
                      float* logmel, cudaStream_t stream) {
  if (n_clips <= 0 || frames_out <= 0) return 0;
  CUtensorMap tx, txb, tb;
  {
    // frames as overlapping rows of the waveform: element (sample in frame, frame, clip)
    uint64_t dims[3] = {uint64_t(kWin), uint64_t(frames_out), uint64_t(n_clips)};
    // (a single clip never uses its stride: any legal value will do)
    const uint64_t cs = n_clips == 1 ? uint64_t(frames_out + 3) * kHop : uint64_t(clip_stride);
    uint64_t str[2] = {uint64_t(kHop) * sizeof(IN), cs * sizeof(IN)};
    uint32_t box[3] = {eoBK, kTM, 1};
    uint32_t boxb[3] = {uint32_t(RawLags<IN>::kBwdCols), kTM, 1};
    if (make_tmap_plain(&tx, wave, sizeof(IN), 3, dims, str, box) ||
        make_tmap_plain(&txb, wave, sizeof(IN), 3, dims, str, boxb)) {
      set_kernel_error("logmel: %s", igemm_last_error());
      return 1;
    }
  }
  {
    uint64_t dims[2] = {uint64_t(eoKPad), uint64_t(eoPlanes * 2 * kNTiles * eoTN)};
    uint64_t str[1] = {uint64_t(eoKPad) * 2};
    uint32_t box[2] = {eoBK, eoTN};
    if (make_tmap_bf16(&tb, t->basis_eo, 2, dims, str, box, 64)) {   // 16-bit elements: the map only moves bytes
      set_kernel_error("logmel: %s", igemm_last_error());
      return 1;
    }
  }
  LogmelEoParams p{};
  p.frames_out = frames_out;
  p.tiles_per_clip = static_cast<int>((frames_out + kTM - 1) / kTM);
  p.total_tiles = static_cast<long long>(p.tiles_per_clip) * n_clips;
  p.out = logmel;
  if (p.total_tiles <= 0) return 0;
  void* flags = nullptr;
  if (alloc_exact_list(p.total_tiles, stream, &flags)) return 1;
  p.exact_count = static_cast<unsigned*>(flags);
  p.exact_list = reinterpret_cast<uint32_t*>(static_cast<char*>(flags) + 16);
  const long long grid = std::min<long long>(p.total_tiles, num_sms());
  const cudaError_t le = launch_pdl(logmel_eo_kernel<IN>, dim3(static_cast<unsigned>(grid)), dim3(eoThreads), eoSmemBytes,
                                    stream, tx, txb, tb, p);
  count_launch();
  if (le != cudaSuccess) {
    set_kernel_error("logmel_eo_kernel: %s", cudaGetErrorString(le));
    return 1;
  }
  if (check_launch("logmel_eo_kernel")) return 1;
  if (launch_exact<IN>(wave, n_clips == 1 ? 0 : clip_stride, frames_out, p.tiles_per_clip, p.exact_list, p.exact_count,
                       t->basis_f64, t->mel_f64, logmel, stream))
    return 1;
  if (cudaFreeAsync(flags, stream) != cudaSuccess) {
    set_kernel_error("logmel: cudaFreeAsync failed");
    return 1;
  }
  return 0;
}

template <class IN>
int logmel_tc_forward_impl(const IN* wave, long long n_clips, long long samples_per_clip, long long clip_stride,
                           long long frames_out, float* logmel, cudaStream_t stream) {
  TcTables* t = nullptr;
  if (get_tables(&t)) return 1;
  if (3 * n_clips > 0x7fffffffLL || frames_out > 0x7fffffffLL) {
    set_kernel_error("logmel: too many clips / frames for one launch");
    return 1;
  }
  if (logmel_eo_accepts(wave, n_clips, clip_stride))
    return logmel_eo_forward<IN>(t, wave, n_clips, clip_stride, frames_out, logmel, stream);
  constexpr int a_planes = sizeof(IN) == 2 ? 2 : 3;
  const long long pitch = logmel_tc_pitch(samples_per_clip);
  const size_t plane_bytes = size_t(n_clips) * pitch * 2;
  void* planes = nullptr;
  if (cudaMallocAsync(&planes, 3 * plane_bytes, stream) != cudaSuccess) {
    set_kernel_error("logmel: workspace allocation of %zu bytes failed: %s", 3 * plane_bytes,
                     cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  {
    const long long groups = pitch / 8 * n_clips;
    const unsigned grid = static_cast<unsigned>(std::min<long long>((groups + 255) / 256, 148LL * 16));
    split_wave_kernel<IN><<<grid, 256, 0, stream>>>(wave, samples_per_clip, clip_stride, pitch, n_clips,
                                                    static_cast<__nv_bfloat16*>(planes));
    count_launch();
    if (check_launch("split_wave_kernel")) return 1;
  }
  CUtensorMap ta, tb;
  {
    uint64_t dims[3] = {uint64_t(kKPad), uint64_t(frames_out), uint64_t(3 * n_clips)};
    uint64_t str[2] = {uint64_t(kHop) * 2, uint64_t(pitch) * 2};
    uint32_t box[3] = {kBK, kTM, 1};
    if (make_tmap_bf16(&ta, planes, 3, dims, str, box, 64)) {
      set_kernel_error("logmel: %s", igemm_last_error());
      return 1;
    }
  }
  {
    uint64_t dims[2] = {uint64_t(kKPad), uint64_t(3 * kEvalBins * 2)};
    uint64_t str[1] = {uint64_t(kKPad) * 2};
    uint32_t box[2] = {kBK, kTN};
    if (make_tmap_bf16(&tb, t->basis, 2, dims, str, box, 64)) {
      set_kernel_error("logmel: %s", igemm_last_error());
      return 1;
    }
  }
  LogmelParams p{};
  p.a_planes = a_planes;
  p.frames_out = frames_out;
  p.tiles_per_clip = static_cast<int>((frames_out + kTM - 1) / kTM);
  p.n_clips = static_cast<int>(n_clips);
  p.total_tiles = static_cast<long long>(p.tiles_per_clip) * n_clips;
  p.out = logmel;
  void* flags = nullptr;
  if (alloc_exact_list(p.total_tiles, stream, &flags)) return 1;
  p.exact_count = static_cast<unsigned*>(flags);
  p.exact_list = reinterpret_cast<uint32_t*>(static_cast<char*>(flags) + 16);
  const long long grid = std::min<long long>(p.total_tiles, num_sms());
  const cudaError_t le = launch_pdl(logmel_tc_kernel, dim3(static_cast<unsigned>(grid)), dim3(kThreads), kSmemBytes,
                                    stream, ta, tb, p);
  count_launch();
  if (le != cudaSuccess) {
    set_kernel_error("logmel_tc_kernel: %s", cudaGetErrorString(le));
    return 1;
  }
  if (check_launch("logmel_tc_kernel")) return 1;
  if (launch_exact<IN>(wave, n_clips == 1 ? 0 : clip_stride, frames_out, p.tiles_per_clip, p.exact_list, p.exact_count,
                       t->basis_f64, t->mel_f64, logmel, stream))
    return 1;
  if (cudaFreeAsync(flags, stream) != cudaSuccess || cudaFreeAsync(planes, stream) != cudaSuccess) {
    set_kernel_error("logmel: cudaFreeAsync failed");
    return 1;
  }
  return 0;
}

}  // namespace

int stft_magnitude_f64(const double* signal, long long n_samples, double* mag, cudaStream_t stream) {
  const long long n_frames = n_samples < kWin ? 0 : 1 + (n_samples - kWin) / kHop;
  if (n_frames <= 0) return 0;
  TcTables* t = nullptr;
  if (get_tables(&t)) return 1;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!t->basis257) {
      std::vector<double> hann(kWin), mel(size_t(kBins) * kMel), b(size_t(2) * eoHalf * kBins);
      front_end_tables_host(hann.data(), mel.data());
      for (int m = 0; m < eoHalf; ++m)
        for (int k = 0; k < kBins; ++k) {
          const double ang = 2 * kPi * ((k * m) % kFft) / kFft, g = hann[eoHalf + m] * (m == 0 ? 0.5 : 1.0);
          b[size_t(m) * kBins + k] = g * std::cos(ang);
          b[size_t(eoHalf + m) * kBins + k] = g * std::sin(ang);
        }
      void* d = nullptr;
      if (cudaMalloc(&d, b.size() * 8) != cudaSuccess ||
          cudaMemcpy(d, b.data(), b.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_kernel_error("stft_magnitude: table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        return 1;
      }
      t->basis257 = static_cast<double*>(d);
    }
  }
  const long long blocks = (n_frames + kStftFrames - 1) / kStftFrames;
  if (blocks > 0x7fffffffLL) {
    set_kernel_error("stft_magnitude: signal too long for one call");
    return 1;
  }
  stft_magnitude_kernel<<<static_cast<unsigned>(blocks), kStftThreads, 0, stream>>>(signal, n_frames, t->basis257, mag);
  count_launch();
  return check_launch("stft_magnitude_kernel");
}

int logmel_tc_forward(const float* wave, long long n_clips, long long samples_per_clip, long long clip_stride,
                      long long frames_out, float* logmel, cudaStream_t stream) {
  return logmel_tc_forward_impl<float>(wave, n_clips, samples_per_clip, clip_stride, frames_out, logmel, stream);
}

int logmel_tc_forward_pcm16(const int16_t* pcm, long long n_clips, long long samples_per_clip, long long clip_stride,
                            long long frames_out, float* logmel, cudaStream_t stream) {
  return logmel_tc_forward_impl<int16_t>(pcm, n_clips, samples_per_clip, clip_stride, frames_out, logmel, stream);
}

}  // namespace vmb
