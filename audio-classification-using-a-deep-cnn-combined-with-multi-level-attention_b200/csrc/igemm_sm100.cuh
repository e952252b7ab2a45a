// Implicit-GEMM engine for the VGGish conv3x3 / FC layers on sm_100a (tcgen05 + TMEM + TMA).
//
//   D[M x N] = act( A[M x K] * B[N x K]^T + bias[N] ),  A, B bf16 (K-major), accumulation fp32 in TMEM.
//
// Two A-operand modes share one kernel:
//   * PLAIN : A is a row-major [M][K] bf16 matrix (the FC layers, reference vggish.py:13-19).
//   * CONV  : A is never materialised.  The activation tensor is NHWC bf16 and the K axis runs over
//             (tap, c_in) = (kh*3+kw)*C_in + c.  For K-block kb the producer issues four 4-D TMA box loads
//             (64 channels x Wb x Hb pixels, Wb*Hb = 32) at the tap-shifted coordinates; TMA zero-fills the
//             out-of-range halo, which is exactly Conv2d(padding=1) (reference vggish.py:113).  Each box is
//             one 32-row quarter of the 128-row UMMA tile, so one epilogue warp owns whole 2x2 pooling
//             windows and MaxPool2d(2,2) (vggish.py:111) is a pair of warp shuffles.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (one lane),
// warps 2-9 = epilogue, two per TMEM lane quarter (TMEM -> regs -> bias/ReLU/pool -> global, one full 32-byte sector per
// lane and store).  Persistent over tiles, accumulators double-buffered in TMEM so the epilogue of tile i overlaps the
// MMAs of tile i+1.
//
// Variants: BIG (one 128-pixel TMA box per sub-tile when the image height allows), HALO (one haloed box per (channel
// block, dx) feeding the three dy taps — conv2), MT = 2 (256 x 128 tiles for C_out = 128), and the CTA-pair kernel of
// igemm_pair_sm100.cu (tcgen05 cta_group::2, 256 x 256 tiles) for C_out / N multiples of 256.  Every bf16 conv variant
// walks K in the same (channel block, dx, dy) order, so their results are bit-identical.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace vmb {

struct IgemmParams {
  int M;             // PLAIN: rows of A / D.  CONV: number of images.
  int N;             // output columns (C_out)
  int num_kb;        // K / 64
  int cblks;         // CONV: C_in / 64
  int H, W;          // CONV: input (= conv output) spatial size
  int Hb, Wb;        // CONV: quarter = Hb x Wb pixels, Hb*Wb == 32, both even
  int big_box;       // CONV: one TMA box per 128-pixel sub-tile (Wb x 4*Hb) instead of four quarter boxes
  int boxes_per_row; // W / Wb
  int boxes_per_img; // (H / Hb) * (W / Wb)
  int total_boxes;   // M * boxes_per_img
  int num_m_tiles;
  int num_n_tiles;
  int relu;
  int split_nkb;     // PLAIN split mode: K / 64 of one plane (0 = ordinary GEMM)
  int split_planes;  // 2 (hi | lo: 3 products) or 3 (hi | mid | lo: 6 products)
  int ksplit;        // PLAIN + atomic fp32 output: number of K slices (<= 1: none)
  int tile_count;    // pair kernel: process only the first tile_count tiles (0 = all); see igemm_pair_linear
  int conv_split;    // CONV: activations are [n][2][H][W][C] hi | lo planes, weights [C_out][2 * 9 C_in]
  int f16;           // operands (and 16-bit outputs) are fp16 instead of bf16: the fp16 mode of the VGGish body
  int* sat_flag;     // fp16 mode: set to 1 when an output saturated the fp16 range (may be null; mapped host memory)
  long long out_img_stride;  // CONV: output elements per image (2 planes when the output is split)
  long long lo_off;          // split output: element offset of the lo plane relative to the hi element
  long long ldo;     // PLAIN: output row stride (elements)
  const float* bias; // [N]
  void* out;         // bf16 (or fp32 when OUT_F32)
};

// Launchers (defined in igemm_sm100.cu).  All return cudaError_t-compatible ints; 0 = ok.
// PLAIN: out[M][N] (+ldo) = act(A[M][K] B[N][K]^T + bias).  K % 64 == 0, N % block_n == 0.
// fmt: kFmtBf16 (0) or kFmtF16 (1) — the element format of a, w and of a 16-bit out; sat_flag: see IgemmParams.
int igemm_linear(const void* a_bf16, const void* w_bf16, const float* bias, void* out, int out_f32, int relu,
                 int M, int N, int K, cudaStream_t stream, int fmt = 0, int* sat_flag = nullptr);
// PLAIN, split-bf16.  planes = 2: A = [A_hi | A_lo] as bf16 [M][2K], W likewise [N][2K];
// out fp32 [M][ldo] = act(A_hi W_hi^T + A_lo W_hi^T + A_hi W_lo^T + bias): ~16 mantissa bits per operand (the
// eval-mode attention head, where plain bf16 would move the ranking metric).  planes = 3: [hi | mid | lo] as
// [M][3K], the six products with plane-index sum <= 2: fp32-equivalent operands (head training, where ReLU masks
// must not flip against the fp32 reference).  bias may be null.  K % 64 == 0, N % 128 == 0.
int igemm_linear_split(const void* a_planes, const void* w_planes, const float* bias, float* out, long long ldo,
                       int relu, int M, int N, int K, cudaStream_t stream, int planes = 2);
// Split in, split out (the accuracy mode of the VGGish body): out planes bf16 [M][hi(N) | lo(N)] =
// split(act(A_hi W_hi^T + A_lo W_hi^T + A_hi W_lo^T + bias)).  K % 64 == 0, N % 256 == 0.
int igemm_linear_split_out(const void* a_planes, const void* w_planes, const float* bias, void* out_planes, int relu,
                           int M, int N, int K, cudaStream_t stream);
// CONV 3x3 with hi | lo activations [n][2][H][W][C_in], hi | lo weights [C_out][2 * 9 C_in] and hi | lo output
// [n][2][H(/2)][W(/2)][C_out] (pooling, when asked, on the fp32 accumulators).
int igemm_conv3x3_split(const void* act_planes, const void* w_planes, const float* bias, void* out_planes, int n_img,
                        int H, int W, int C_in, int C_out, int pool, cudaStream_t stream);
// CONV 3x3 pad 1 (+bias, ReLU, optional 2x2 maxpool): act NHWC bf16 [n][H][W][C_in], weights [C_out][9*C_in]
// ((kh,kw,c) order), out NHWC bf16 [n][H or H/2][W or W/2][C_out].  C_in % 64 == 0, C_out % 128 == 0.
int igemm_conv3x3(const void* act_bf16, const void* w_bf16, const float* bias, void* out_bf16, int n_img, int H,
                  int W, int C_in, int C_out, int pool, cudaStream_t stream, int fmt = 0, int* sat_flag = nullptr);

// CTA-pair (cta_group::2) kernels for the bf16 layers with C_out / N a multiple of 256 (igemm_pair_sm100.cu);
// igemm_conv3x3 / igemm_linear route to them when igemm_use_pair() (env VMB_IGEMM_PAIR=0/1 overrides the default).
int igemm_pair_linear(const void* a_bf16, const void* w_bf16, const float* bias, void* out_bf16, int relu, int M, int N,
                      int K, cudaStream_t stream, int fmt = 0, int* sat_flag = nullptr);
int igemm_pair_conv3x3(const void* act_bf16, const void* w_bf16, const float* bias, void* out_bf16, int n_img, int H,
                       int W, int C_in, int C_out, int pool, cudaStream_t stream, int fmt = 0, int* sat_flag = nullptr);
const char* igemm_pair_last_error();
// A rectangle of a PLAIN bf16 GEMM on the single-CTA kernel with 128- or 64-wide tiles: out[M][N] (row stride ldo) =
// act(A[M][K] W[N][K]^T + bias); used by igemm_pair_linear for the tiles of an incomplete last round.
int igemm_linear_rect(const void* a_bf16, const void* w_bf16, const float* bias, void* out_bf16, long long ldo, int relu,
                         int M, int N, int K, cudaStream_t stream, int fmt = 0, int* sat_flag = nullptr);
bool igemm_use_pair();
int igemm_set_pair(int on);
// Haloed activation boxes for the C_out = 128 conv (conv2): same contract as igemm_set_pair.
bool igemm_use_halo();
int igemm_set_halo(int on);   // 1 / 0 force the choice, -1 returns to the default; returns the previous setting

const char* igemm_last_error();

// Keep / drop decision of dropout element idx of layer `layer` in the step seeded `seed` (head training; counter based,
// recomputed in the backward pass): a 32-bit finaliser (murmur3's fmix32) over the element index keyed by (seed, layer)
// — 8 integer instructions per element; the first version ran a 64-bit splitmix (two 64-bit multiplies = a dozen 32-bit
// IMADs) for every element of every element-wise kernel.  Returns the inverted-dropout scale: 1 / (1 - p) or 0.
__device__ __forceinline__ float dropout_scale(unsigned long long seed, unsigned layer, unsigned long long idx, float p) {
  if (p <= 0.f) return 1.f;
  const unsigned key = static_cast<unsigned>(seed) ^ (static_cast<unsigned>(seed >> 32) * 0x9E3779B1u) ^
                       (layer * 0x85EBCA77u + 0xC2B2AE3Du);
  unsigned h = (static_cast<unsigned>(idx) ^ key) * 0x9E3779B1u + static_cast<unsigned>(idx >> 32) * 0x27D4EB2Fu;
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  const float u = static_cast<float>(h >> 8) * (1.0f / 16777216.0f);
  return u >= p ? 1.f / (1.f - p) : 0.f;
}

// The three-plane split of the training GEMMs' operands (hi | mid | lo, planes = 3 above): fp32-equivalent operands.
__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& mid, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(hi);      // exact
  mid = __float2bfloat16_rn(r1);
  lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
}

// planes_gemm_sm100.cu: the split GEMMs with every operand plane of a K-block loaded once per tile and the hi * hi
// product in its own TMEM accumulator.  The training paths call it directly; igemm_linear_split (the eval-mode head)
// routes to it when planes_gemm_enabled() (default; env VMB_PLANES_GEMM=0 selects the long-K-loop kernel above).
// ksplit > 1: that many K slices, vector reductions into a zeroed out; ksplit == -1: one slice but still adding into
// out; ksplit == 0: plain stores (+ bias, optional ReLU).
int planes_gemm(const void* a_planes, const void* b_planes, const float* bias, float* out, long long ldo, int relu, int M,
                int N, int K, int planes, int ksplit, cudaStream_t stream);
// Fused epilogue of the eval-mode head (two planes, no K split): the accumulator row u of (clip, time step
// t = row % T) becomes h = relu?(a1_t u + b1_t) [columns >= cols: 0], written as bf16 hi | lo planes dst[M][2 * cpad]
// (and, with dst2, a2_t h + b2_t likewise) — BatchNorm1d(T) in eval mode + ReLU + the operand split of the next Linear
// (model.py:219-221).  Same expressions, same order as rows_affine_split_kernel (mla_tc.cu).
struct PlanesEpi {
  int mode;                        // 1
  int T, relu, cols, cpad;
  const float *a1, *b1, *a2, *b2;  // [T]; a1 may be null (identity), a2 / b2 only with dst2
  void *dst, *dst2;                // bf16 planes, 32-byte aligned
};
int planes_gemm_fused(const void* a_planes, const void* b_planes, const float* bias, const PlanesEpi& epi, int M, int N,
                      int K, cudaStream_t stream);
// Statistics epilogue (head training): besides storing out fp32 [M][ldo] = products + bias, the kernel accumulates
// {sum, sum of squares} of the first `cols` columns per channel = row % channels (BatchNorm1d(T) over a (clip, time step)
// row index, model.py:221 in train mode) into acc (double [channels][2], zeroed by the caller), and the CTA that finishes
// last writes stat[channels][2] = {mean, 1 / sqrt(var + eps)} and, when run_mean != null, updates the running statistics
// with torch's momentum rule (unbiased variance).  counter must be zero on entry.  channels <= 16.
struct PlanesStats {
  double* acc;
  float* stat;
  unsigned* counter;
  float *run_mean, *run_var;
  double count;       // elements per channel
  int channels, cols;
  float eps, momentum;
};
// Gradient-statistics epilogue (head training, backward): the GEMM computes d(loss)/d(activation) of a
// BatchNorm1d(T) (+ ReLU + dropout) block, out fp32 [M][ldo]; the block's backward pass first needs, per time step
// t = row % T, S1_t = sum g and S2_t = sum g * xhat with g = out * [BN output > 0] * dropout keep scale and
// xhat = (u - mean_t) * rstd_t (u: the block's pre-BatchNorm input saved by the forward pass).  The epilogue adds both
// sums into acc (double [T][2], zeroed by the caller) from the accumulator rows it holds — the separate reduction pass
// over out and u (bn_time_backward_reduce_kernel, mla_train.cu) is not launched.
struct PlanesGradStats {
  const float* u;
  long long ldu;
  const float *stat, *gamma, *beta;     // [T][2] {mean, rstd}; [T]; [T]
  double* acc;
  const unsigned long long* seed;       // device memory: the step's dropout seed
  unsigned layer;
  float p;
  int relu, T, F, cols;                 // F: elements per row in the dropout element index; cols: valid columns
};
int planes_gemm_gradstats(const void* a_planes, const void* b_planes, float* out, long long ldo, int M, int N, int K,
                          int planes, const PlanesGradStats& gs, cudaStream_t stream);
int planes_gemm_stats(const void* a_planes, const void* b_planes, const float* bias, float* out, long long ldo, int M,
                      int N, int K, int planes, const PlanesStats& stats, cudaStream_t stream);
// GEMM over ROW-major operands read as MN-major UMMA operands (head training, weight gradients dW = G^T A):
// out fp32 [M][ldo] (+)= sum_r a[r][m] b[r][n]; a_planes bf16 [K][planes * a_cols], b_planes bf16 [K][planes * b_cols].
// ksplit > 1 or -1: K slices added into out with vector reductions (out zeroed by the caller); ksplit 0: plain stores.
int planes_gemm_mn(const void* a_planes, int a_cols, const void* b_planes, int b_cols, float* out, long long ldo, int M,
                   int N, int K, int planes, int ksplit, cudaStream_t stream);
// Contraction lengths per tcgen05 accumulator of the three-plane training GEMMs: one accumulator summed over thousands
// of K steps truncates enough to miss the fp32 reference, so a longer contraction is cut into slices whose fp32 partial
// sums are added in the output.  Forward GEMMs slice their input columns by kFwdSlice (the caller zeroes the output and
// passes the slice count as ksplit); planes_gemm_dw slices the rows of a weight gradient by at most kDwSlice.
constexpr int kFwdSlice = 768, kDwSlice = 1024;
// Weight gradient of a training Linear, dW = G^T A over the rows: planes_gemm_mn with one wave of (K slice, tile)
// work items, each slice at least four 32-row K-blocks long.  An output of more tiles than SMs (the 12288-wide first
// layer of the head) is split only into slices of at most kDwSlice rows, and with one slice stored plainly.  Clears
// out (M rows of ldo floats) on the stream first whenever the slices add into it.
int planes_gemm_dw(const void* a_planes, int a_cols, const void* b_planes, int b_cols, float* out, long long ldo, int M,
                   int N, int K, int planes, cudaStream_t stream);
bool planes_gemm_enabled();
const char* planes_gemm_last_error();

// Shared host helpers (igemm_sm100.cu): bf16 tensor map with 128- or 64-byte swizzle (error text goes to
// igemm_last_error()), and the SM count of the current device.
int make_tmap_bf16(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, int swizzle_bytes = 128);
// Unswizzled tensor map over 4-byte (fp32) or 2-byte (16-bit integer) elements; out-of-range box elements read as zero.
int make_tmap_plain(CUtensorMap* m, const void* base, int elem_bytes, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box);
int num_sms();

}  // namespace vmb
