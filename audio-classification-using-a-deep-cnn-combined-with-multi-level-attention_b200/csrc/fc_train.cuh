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

// fp32 W [rows][cols] -> three bf16 planes [rows][3 * cols], and with planes_t != null the transposed planes
// [cols][3 * rows] (the B operand of the dgrad GEMM).  rows, cols multiples of 32.
int fc_weight_planes(const float* w, int rows, int cols, void* planes, void* planes_t, cudaStream_t st);

// features: the conv stack's output in the handle's precision (0 bf16, 1 hi | lo pairs, 2 fp16).  Writes the operand
// planes of X, A1, A2 and the pre-activations Z1..Z3 into ws, and the embeddings relu(Z3) fp32 [n][128] to emb.
int fc_train_forward(const void* const w_planes[3], const float* const bias[3], const void* features, int precision,
                     long long n, char* ws, const FcTrainLayout& L, float* emb, cudaStream_t st);
// wt_planes[1], wt_planes[2]: transposed planes of W2, W3.  d_emb fp32 [n][128] -> grads (kFcGradCount floats, every
// one written; 32-byte aligned).
int fc_train_backward(const void* const wt_planes[3], long long n, char* ws, const FcTrainLayout& L,
                      const float* d_emb, float* grads, cudaStream_t st);

}  // namespace vmb
