// Shared definitions of the multi-level attention head (mla.cu: handle + fused fp32 kernel, mla_tc.cu: tensor-core
// path).  Reference: model.py:199-269.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace vmb_head {

constexpr int kMaxLevels = 4;
constexpr int kMaxFc = 4;
constexpr int kPad = 640;      // padded column count of every transposed weight
constexpr int kMaxDim = 608;   // activation row pitch in shared memory (floats); multiple of 4
constexpr int kThreads = 256;
constexpr int kColThreads = 64;
constexpr int kColsPerThread = kPad / kColThreads;  // 10

struct FcDev {
  const void* wp;     // bf16 [kPad][2 * kpad]: hi | lo planes of W (rows = outputs, zero padded)   (tensor-core path)
  int kpad;           // contraction length: kPad for inputs of hidden width, else the inputs padded to 64
  const float* wt;    // [in][kPad]
  const float* bias;  // [kPad]
  const float* a;     // [T] folded BN scale
  const float* b;     // [T] folded BN shift
  int in;
};
struct LevelDev {
  const float* n0a;  // [T]
  const float* n0b;
  int n_fc;
  FcDev fc[kMaxFc];
  FcDev fcv;         // a/b unused
  const float *av, *bv, *af, *bf;  // [T] each
};
struct HeadDev {
  int n_levels, emb_in, hidden, K, T;
  LevelDev lvl[kMaxLevels];
  const void* fc_wp;     // bf16 [kPad][2 * fc_kpad]: hi | lo planes of the output Linear
  int fc_kpad;           // L*K padded to a multiple of 64
  const float* fc_wt;    // [L*K][kPad]
  const float* fc_bias;  // [kPad]
  const float* out_a;    // [K] folded BN_K
  const float* out_b;
};


struct Handle {
  HeadDev dev;
  float* blob = nullptr;      // every folded fp32 table
  void* planes = nullptr;     // every bf16 weight plane
  int device = 0;
  // tc_forward runs each level's attention branch (fcv GEMM + pooling) on a side stream while the next level's embedding
  // chain continues on the caller's stream: created on first use, owned by the handle
  cudaStream_t side = nullptr;
  cudaEvent_t fork_ev[kMaxLevels] = {}, gemm_ev[kMaxLevels] = {}, join_ev[kMaxLevels] = {};
};

// Tensor-core forward (mla_tc.cu).  Returns 0 / 1 (message via vmb::kernels_last_error()).
int tc_forward(Handle& h, const float* emb, long long batch, float* scores, cudaStream_t st);
// 0 selects the unfused forward, 1 or -1 the fused-epilogue forward (the default); returns the previous setting (0 / 1)
int mla_fuse_set(int on);
// One level's EmbeddedMapping / AttentionModule on its own (model.py:217-222, :235-242), from the same kernels.
int tc_embedded_mapping(const Handle& h, int level, const float* x, long long batch, float* out, cudaStream_t st);
int tc_attention(const Handle& h, int level, const float* hemb, long long batch, float* y, cudaStream_t st);

}  // namespace vmb_head
