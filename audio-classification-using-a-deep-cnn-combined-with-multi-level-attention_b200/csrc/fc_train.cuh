// Train-mode FC stack of the VGGish body (fc_train.cu), driven by the vmb_vggish_* entry points of vggish.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace vmb {

constexpr int kFcTrainIn = 12288;   // fc1's input: the (h, w, c)-flattened conv features
// Flat FC gradient layout (state_dict order of embeddings.{0,2,4}), in floats
constexpr long long kFcGradW1 = 0;
constexpr long long kFcGradB1 = kFcGradW1 + 4096LL * 12288;
constexpr long long kFcGradW2 = kFcGradB1 + 4096;
constexpr long long kFcGradB2 = kFcGradW2 + 4096LL * 4096;
constexpr long long kFcGradW3 = kFcGradB2 + 4096;
constexpr long long kFcGradB3 = kFcGradW3 + 128LL * 4096;
constexpr long long kFcGradCount = kFcGradB3 + 128;

// Byte offsets of the train-mode workspace regions (each 1024-byte aligned).  n_pad = n rounded up to 64 rows; the
// operand planes are bf16 [n_pad][3 * width] (hi | mid | lo), z1 / z2 / z3 the fp32 pre-activations [n][width].
struct FcTrainLayout {
  size_t x, a1, a2, z1, z2, z3, g, da, colsum, conv, total;
  long long n_pad;
};
FcTrainLayout fc_train_layout(long long n, size_t conv_bytes);

// fp32 W [rows][cols] -> three bf16 planes [rows][3 * cols] (skipped when planes is null), and with planes_t != null the
// transposed planes [cols][3 * rows] (the B operand of the dgrad GEMM).  rows, cols multiples of 32.
int fc_weight_planes(const float* w, int rows, int cols, void* planes, void* planes_t, cudaStream_t st);

// features: the conv stack's output in the handle's precision (0 bf16, 1 hi | lo pairs, 2 fp16), or null when the
// operand planes of X are already in ws (conv4_2 trained, conv_train.cu).  Writes the operand planes of X, A1, A2 and
// the pre-activations Z1..Z3 into ws, and the embeddings relu(Z3) fp32 [n][128] to emb.
int fc_train_forward(const void* const w_planes[3], const float* const bias[3], const void* features, int precision,
                     long long n, char* ws, const FcTrainLayout& L, float* emb, cudaStream_t st);
// wt_planes[1], wt_planes[2]: transposed planes of W2, W3.  d_emb fp32 [n][128] -> grads (kFcGradCount floats, every
// one written; 32-byte aligned), or with grads null no weight or bias gradient (fc1-fc3 frozen).  With dx != null
// (conv4_2 trained) also fc1's input gradient dx fp32 [n][12288] = G1 W1 from wt_planes[0], W1's transposed planes.
int fc_train_backward(const void* const wt_planes[3], long long n, char* ws, const FcTrainLayout& L,
                      const float* d_emb, float* grads, float* dx, cudaStream_t st);

// ------------------------------------------------------------------------- conv4_2 trainable (conv_train.cu)
// features.13 (the last conv, 512 -> 512, 12 x 8, vggish.py:108-118) trained with conv1 .. conv4_1 frozen.
constexpr int kConv42C = 512, kConv42Pix = 96, kConv42K = 9 * 512;   // channels, pixels per example, (kh, kw, c)
constexpr long long kConv42GradCount = 512LL * 4608 + 512;           // features.13.weight (OIHW), then .bias
constexpr long long kConv42Chunk = 256;                              // examples per im2col chunk
// The conv4_2 train workspace: the FC train layout (same offsets) followed by these regions (each 1024-byte aligned).
// conv4_1's output stays where the conv stack left it, at fc.conv (the start of the conv scratch).
struct Conv42Layout {
  FcTrainLayout fc;
  size_t z;       // fp32 [n * 96][512]        conv4_2 pre-activation, row = (example, h, w)
  size_t dz;      // bf16 [n * 96][3 * 512]    d(loss)/dz operand planes
  size_t dx1;     // fp32 [n][12288]           fc1's input gradient
  size_t dw;      // fp32 [512][4608]          weight gradient in (kh, kw, c) order
  size_t colsum;  // double [512]              bias gradient accumulator
  size_t cols;    // bf16 [min(n, 256) * 96][3 * 4608]   im2col planes of one chunk
  size_t total;
};
Conv42Layout conv4_2_layout(long long n, size_t conv_bytes);
// fp32 OIHW [512][512][3][3] -> three bf16 planes [512][3 * 4608] in (kh, kw, c) column order
int conv4_2_weight_planes(const float* w_oihw, void* planes, cudaStream_t st);
// conv4_1's output act (NHWC [n][12][8][512] in the handle's precision, see fc_train_forward) -> z, then ReLU, the 2x2
// max-pool and the (h, w, c) flatten into the operand planes of fc1's input (ws + L.fc.x)
int conv4_2_train_forward(const void* w_planes, const float* bias, const void* act, int precision, long long n, char* ws,
                          const Conv42Layout& L, cudaStream_t st);
// fc1's input gradient (ws + L.dx1) -> grads (kConv42GradCount floats: weight OIHW, then bias)
int conv4_2_train_backward(const void* act, int precision, long long n, char* ws, const Conv42Layout& L, float* grads,
                           cudaStream_t st);

}  // namespace vmb
