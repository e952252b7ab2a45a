// VGGish model handle (reference torchvggish/vggish.py:9-31, 108-118) and the whole waveform -> scores pipeline
// (model.py:58-62 fed by vggish_input.py:30-82).  The handle owns bf16 weights re-laid-out for the implicit-GEMM
// kernels; activations ping-pong between two caller-provided workspace regions in NHWC bf16.
#include <cuda_bf16.h>

#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/vggish_mla_b200.h"
#include "fc_train.cuh"
#include "igemm_sm100.cuh"
#include "kernels.cuh"

namespace vmb {
void set_api_error(const char* msg);
}

// Cached staging of the host-buffer entry points (grown on demand, freed with the handle).  Two device wave buffers
// alternate between micro-batches — across calls too — so the H2D copy of the next micro-batch (or of the next
// submitted call) overlaps the compute of the current one; two result slots let one call be in flight while the
// previous one is being collected.
struct HostStage {
  cudaStream_t copy_st = nullptr;
  cudaEvent_t wave_ready[2] = {}, wave_free[2] = {};
  void* d_wave[2] = {};           // fp32 or int16 samples, whichever the call brings
  size_t wave_cap[2] = {};
  unsigned long long batches = 0;   // micro-batches issued so far (selects the wave buffer)
  void* d_ws = nullptr;
  size_t ws_cap = 0;
  float* d_scores[2] = {};
  size_t scores_cap[2] = {};
  cudaEvent_t done[2] = {};
  bool busy[2] = {false, false};
  unsigned long long calls = 0;
};

struct vmb_vggish {
  int precision = 0;         // 0: bf16 activations and weights; 1: hi | lo split bf16 activations and weights (accuracy
                             // mode); 2: fp16 activations and weights (same tensor rate as bf16, 11 mantissa bits)
  bool has_fc = true;        // false: built without the FC stack (conv features only, model.py:161-166)
  int* sat = nullptr;        // precision 2: [8] saturation flags (conv1, conv2..conv4_2, fc1, fc2) in mapped pinned host
                             // memory — the kernels store 1 when an output reached the fp16 maximum
  float* conv1_w = nullptr;  // fp32 [64][9]
  float* conv_b[6] = {};     // fp32 biases (index 0 = conv1)
  void* conv_w[6] = {};      // bf16 [C_out][9*C_in] (precision 1: [C_out][2*9*C_in] hi | lo), index 1..5
  void* fc_w[3] = {};        // bf16 [out][in]       (precision 1: [out][2*in] hi | lo)
  float* fc_b[3] = {};
  // train-mode FC stack (fc_train.cu): three-plane copies of the FC weights, allocated and derived by the first
  // vmb_vggish_refresh_fc — row-major [out][3 * in] for the forward GEMMs, transposed [in][3 * out] for the dgrad of
  // fc2 and fc3, and of fc1 once vmb_vggish_refresh_conv4_2 has allocated train_wt[0] (conv4_2 trained)
  void* train_w[3] = {};
  void* train_wt[3] = {};
  // train-mode conv4_2 (conv_train.cu): three-plane copy of its weights [512][3 * 4608] in (kh, kw, c) order, allocated
  // and derived by the first vmb_vggish_refresh_conv4_2, which also allocates fc1's transposed planes train_wt[0]
  void* conv_train_w = nullptr;
  HostStage stage;
};

namespace {

struct ConvGeom { int H, W, C_in, C_out, pool; };
// features.{3,6,8,11,13}: input geometry of each tensor-core conv (after the preceding pools)
constexpr ConvGeom kConv[5] = {{48, 32, 64, 128, 1}, {24, 16, 128, 256, 0}, {24, 16, 256, 256, 1},
                               {12, 8, 256, 512, 0}, {12, 8, 512, 512, 1}};
constexpr int kFcIn[3] = {12288, 4096, 4096};
constexpr int kFcOut[3] = {4096, 4096, 128};
constexpr size_t kBufA = 196608;  // bytes per example: largest activation (48x32x64 or 24x16x256 bf16)
constexpr size_t kBufB = 98304;   // 24x16x128 / 12x8x512 bf16

int fail(const char* fmt, const char* detail = "") {
  char buf[640];
  snprintf(buf, sizeof buf, fmt, detail);
  vmb::set_api_error(buf);
  return 1;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// fp32 masters -> the inference copy of FC layer i in the handle's precision (create and refresh share it, so a
// refreshed handle holds bit for bit what a fresh build would)
bool fc_inference_copy(vmb_vggish* h, int i, const float* w, const float* b, cudaStream_t st) {
  if (cudaMemcpyAsync(h->fc_b[i], b, size_t(kFcOut[i]) * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess) return false;
  const int fmt = h->precision == 2 ? 1 : 0;
  return (h->precision == 1 ? vmb::split_f32_to_planes(w, h->fc_w[i], kFcOut[i], kFcIn[i], st)
                            : vmb::cast_f32_to_bf16(w, h->fc_w[i], static_cast<long long>(kFcOut[i]) * kFcIn[i], st,
                                                    fmt)) == 0;
}

// conv1 + the five tensor-core convs into the ping-pong workspace; returns the buffer holding the (h, w, c)-flattened
// features [n][12288] ([n][hi | lo] in split mode), or null after recording the error.  convs = 4 stops after conv4_1:
// the returned buffer (the workspace's first region) then holds conv4_1's output NHWC [n][12][8][512] ([n][2][...] split)
char* conv_stack(vmb_vggish* h, const float* examples, long long n, void* workspace, cudaStream_t st, const char* who,
                 int convs = 5) {
  const bool split = h->precision == 1;
  const int fmt = h->precision == 2 ? 1 : 0;
  int* sat = h->sat;   // null unless fp16
  const size_t mul = split ? 2 : 1;
  char* A = static_cast<char*>(workspace);
  char* B = A + align_up(size_t(n) * kBufA * mul, 1024);
  {
    vmb::StageTimer t(VMB_STAGE_CONV1, st);
    if (vmb::conv1_tc_relu_pool(examples, h->conv1_w, h->conv_b[0], A, n, st, split, fmt, sat)) {
      fail("%s", (std::string(who) + ": " + vmb::kernels_last_error()).c_str());
      return nullptr;
    }
  }
  char* src = A;
  char* dst = B;
  for (int i = 0; i < convs; ++i) {
    const ConvGeom& g = kConv[i];
    vmb::StageTimer t(VMB_STAGE_CONV2 + i, st);
    const int rc = split ? vmb::igemm_conv3x3_split(src, h->conv_w[i + 1], h->conv_b[i + 1], dst, int(n), g.H, g.W, g.C_in,
                                                    g.C_out, g.pool, st)
                         : vmb::igemm_conv3x3(src, h->conv_w[i + 1], h->conv_b[i + 1], dst, int(n), g.H, g.W, g.C_in,
                                              g.C_out, g.pool, st, fmt, sat ? sat + 1 + i : nullptr);
    if (rc) {
      fail("%s", (std::string(who) + ": " + vmb::igemm_last_error()).c_str());
      return nullptr;
    }
    char* sw = src; src = dst; dst = sw;
  }
  return src;
}

}  // namespace

extern "C" {

int vmb_vggish_create(vmb_vggish_t** handle, const float* const conv_w[6], const float* const conv_b[6],
                      const float* const fc_w[3], const float* const fc_b[3], void* stream) {
  return vmb_vggish_create_ex(handle, conv_w, conv_b, fc_w, fc_b, 0, stream);
}

int vmb_vggish_create_ex(vmb_vggish_t** handle, const float* const conv_w[6], const float* const conv_b[6],
                         const float* const fc_w[3], const float* const fc_b[3], int precision, void* stream) {
  if (!handle || !conv_w || !conv_b) return fail("vmb_vggish_create: null argument");
  if ((fc_w == nullptr) != (fc_b == nullptr)) return fail("vmb_vggish_create: fc weights and biases go together");
  const bool has_fc = fc_w != nullptr;   // without them the handle serves the conv features only (just_bottlenecks)
  if (precision < 0 || precision > 2) return fail("vmb_vggish_create: precision must be 0 (bf16), 1 (split) or 2 (fp16)");
  for (int i = 0; i < 6; ++i)
    if (!conv_w[i] || !conv_b[i]) return fail("vmb_vggish_create: null conv tensor");
  for (int i = 0; i < 3 && has_fc; ++i)
    if (!fc_w[i] || !fc_b[i]) return fail("vmb_vggish_create: null fc tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  vmb_vggish* h = new vmb_vggish();
  h->precision = precision;
  h->has_fc = has_fc;
  const size_t wmul = precision == 1 ? 2 : 1;
  const int fmt = precision == 2 ? 1 : 0;
  bool ok = true;
  if (precision == 2) {
    ok = cudaHostAlloc(reinterpret_cast<void**>(&h->sat), 8 * sizeof(int), cudaHostAllocMapped) == cudaSuccess;
    if (ok) memset(h->sat, 0, 8 * sizeof(int));
  }
  auto dmalloc = [&](void** p, size_t bytes) { ok = ok && cudaMalloc(p, bytes) == cudaSuccess; };
  auto dcopy = [&](void* d, const void* s, size_t bytes) {
    ok = ok && cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
  };
  dmalloc(reinterpret_cast<void**>(&h->conv1_w), 64 * 9 * 4);
  dmalloc(reinterpret_cast<void**>(&h->conv_b[0]), 64 * 4);
  if (ok) {
    dcopy(h->conv1_w, conv_w[0], 64 * 9 * 4);
    dcopy(h->conv_b[0], conv_b[0], 64 * 4);
  }
  for (int i = 0; i < 5 && ok; ++i) {
    const ConvGeom& g = kConv[i];
    dmalloc(&h->conv_w[i + 1], size_t(g.C_out) * 9 * g.C_in * 2 * wmul);
    dmalloc(reinterpret_cast<void**>(&h->conv_b[i + 1]), size_t(g.C_out) * 4);
    if (!ok) break;
    dcopy(h->conv_b[i + 1], conv_b[i + 1], size_t(g.C_out) * 4);
    ok = ok && (precision == 1 ? vmb::relayout_conv_weight_split(conv_w[i + 1], h->conv_w[i + 1], g.C_out, g.C_in, st)
                               : vmb::relayout_conv_weight(conv_w[i + 1], h->conv_w[i + 1], g.C_out, g.C_in, st, fmt)) == 0;
  }
  for (int i = 0; i < 3 && ok && has_fc; ++i) {
    dmalloc(&h->fc_w[i], size_t(kFcOut[i]) * kFcIn[i] * 2 * wmul);
    dmalloc(reinterpret_cast<void**>(&h->fc_b[i]), size_t(kFcOut[i]) * 4);
    if (!ok) break;
    ok = ok && fc_inference_copy(h, i, fc_w[i], fc_b[i], st);
  }
  ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
  if (!ok) {
    const char* why = cudaGetErrorString(cudaGetLastError());
    vmb_vggish_destroy(h);
    return fail("vmb_vggish_create: allocation / re-layout failed (%s)", why);
  }
  *handle = h;
  return 0;
}

void vmb_vggish_destroy(vmb_vggish_t* h) {
  if (!h) return;
  cudaFree(h->conv1_w);
  for (int i = 0; i < 6; ++i) {
    cudaFree(h->conv_b[i]);
    cudaFree(h->conv_w[i]);
  }
  for (int i = 0; i < 3; ++i) {
    cudaFree(h->fc_w[i]);
    cudaFree(h->fc_b[i]);
    cudaFree(h->train_w[i]);
    cudaFree(h->train_wt[i]);
  }
  cudaFree(h->conv_train_w);
  if (h->sat) cudaFreeHost(h->sat);
  HostStage& hs = h->stage;
  for (int i = 0; i < 2; ++i) {
    cudaFree(hs.d_wave[i]);
    cudaFree(hs.d_scores[i]);
    if (hs.wave_ready[i]) cudaEventDestroy(hs.wave_ready[i]);
    if (hs.wave_free[i]) cudaEventDestroy(hs.wave_free[i]);
    if (hs.done[i]) cudaEventDestroy(hs.done[i]);
  }
  cudaFree(hs.d_ws);
  if (hs.copy_st) cudaStreamDestroy(hs.copy_st);
  delete h;
}

size_t vmb_vggish_workspace_bytes(long long n) {
  if (n <= 0) return 0;
  return align_up(size_t(n) * kBufA, 1024) + align_up(size_t(n) * kBufB, 1024);
}

size_t vmb_vggish_handle_workspace_bytes(const vmb_vggish_t* h, long long n) {
  if (n <= 0 || !h) return 0;
  const size_t mul = h->precision == 1 ? 2 : 1;   // split mode: every activation is a hi | lo pair
  return align_up(size_t(n) * kBufA * mul, 1024) + align_up(size_t(n) * kBufB * mul, 1024);
}

int vmb_vggish_precision(const vmb_vggish_t* h) { return h ? h->precision : -1; }

int vmb_vggish_saturation(vmb_vggish_t* h, int clear) {
  if (!h || !h->sat) return 0;
  int mask = 0;
  for (int i = 0; i < 8; ++i) {
    if (*reinterpret_cast<volatile int*>(h->sat + i)) mask |= 1 << i;
    if (clear) h->sat[i] = 0;
  }
  return mask;
}

int vmb_vggish_forward(vmb_vggish_t* h, const float* examples, long long n, float* emb, void* bottleneck,
                       void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return fail("vmb_vggish_forward: null handle");
  if (n < 0) return fail("vmb_vggish_forward: negative n");
  if (n == 0) return 0;
  if (n > 1000000) return fail("vmb_vggish_forward: at most 1 000 000 examples per call (chunk on the host)");
  if (!examples || !workspace || (!emb && !bottleneck)) return fail("vmb_vggish_forward: null pointer");
  if (emb && !h->has_fc) return fail("vmb_vggish_forward: this handle was built without the FC stack (bottleneck features only)");
  if (workspace_bytes < vmb_vggish_handle_workspace_bytes(h, n)) return fail("vmb_vggish_forward: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace) % 1024) return fail("vmb_vggish_forward: workspace must be 1024-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool split = h->precision == 1;
  const int fmt = h->precision == 2 ? 1 : 0;
  int* sat = h->sat;   // null unless fp16
  const size_t mul = split ? 2 : 1;
  char* A = static_cast<char*>(workspace);
  char* B = A + align_up(size_t(n) * kBufA * mul, 1024);
  char* src = conv_stack(h, examples, n, workspace, st, "vmb_vggish_forward");
  if (!src) return 1;
  char* dst = src == A ? B : A;
  // src == B now holds the NHWC [n][6][4][512] features == the (h,w,c)-flattened [n][12288] matrix (vggish.py:26-29);
  // in split mode [n][hi(12288) | lo(12288)]
  if (bottleneck) {
    const cudaError_t e = split
        ? cudaMemcpy2DAsync(bottleneck, size_t(12288) * 2, src, size_t(2) * 12288 * 2, size_t(12288) * 2, size_t(n),
                            cudaMemcpyDeviceToDevice, st)      // the hi plane
        : cudaMemcpyAsync(bottleneck, src, size_t(n) * 12288 * 2, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return fail("vmb_vggish_forward: bottleneck copy failed");
  }
  if (!emb) return 0;   // conv features only
  // fc1: B -> A, fc2: A -> B, fc3: B -> emb (fp32)
  const void* fc_in[3] = {src, dst, src};
  void* fc_out[3] = {dst, src, emb};
  for (int i = 0; i < 3; ++i) {
    vmb::StageTimer t(VMB_STAGE_FC1 + i, st);
    int rc;
    if (!split)
      rc = vmb::igemm_linear(fc_in[i], h->fc_w[i], h->fc_b[i], fc_out[i], i == 2, 1, int(n), kFcOut[i], kFcIn[i], st, fmt,
                             (sat && i < 2) ? sat + 6 + i : nullptr);
    else if (i < 2)
      rc = vmb::igemm_linear_split_out(fc_in[i], h->fc_w[i], h->fc_b[i], fc_out[i], 1, int(n), kFcOut[i], kFcIn[i], st);
    else if (vmb::planes_gemm(fc_in[i], h->fc_w[i], h->fc_b[i], emb, kFcOut[i], 1, int(n), kFcOut[i], kFcIn[i], 2, 0, st))
      return fail("vmb_vggish_forward: %s", vmb::planes_gemm_last_error());
    else
      rc = 0;
    if (rc) return fail("vmb_vggish_forward: %s", vmb::igemm_last_error());
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ train-mode FC stack
namespace {
// the conv scratch of the train-mode workspace is sized for the split precision (the largest)
vmb::FcTrainLayout train_layout(long long n) { return vmb::fc_train_layout(n, vmb_vggish_workspace_bytes(n) * 2); }
vmb::Conv42Layout conv4_2_layout(long long n) { return vmb::conv4_2_layout(n, vmb_vggish_workspace_bytes(n) * 2); }

int check_train_args(const vmb_vggish_t* h, long long n, const void* ws, size_t ws_bytes, const char* who,
                     bool conv4_2 = false) {
  char msg[256];
  auto bad = [&](const char* why) {
    snprintf(msg, sizeof msg, "%s: %s", who, why);
    return fail("%s", msg);
  };
  if (!h) return bad("null handle");
  if (!h->has_fc) return bad("this handle was built without the FC stack (bottleneck features only)");
  if (!h->train_w[0]) return bad("no training copy of the FC weights: call vmb_vggish_refresh_fc first");
  if (n < 1) return bad("n must be at least 1");
  if (n > 1000000) return bad("at most 1 000 000 examples per call");
  if (!ws) return bad("null workspace");
  if (reinterpret_cast<uintptr_t>(ws) % 1024) return bad("workspace must be 1024-byte aligned");
  if (conv4_2 && !h->conv_train_w)
    return bad("no training copy of conv4_2's weights: call vmb_vggish_refresh_conv4_2 first");
  if (ws_bytes < (conv4_2 ? conv4_2_layout(n).total : train_layout(n).total))
    return bad("workspace too small for n examples");
  return 0;
}
}  // namespace

extern "C" {

size_t vmb_vggish_fc_train_workspace_bytes(long long n) {
  if (n <= 0) return 0;
  return train_layout(n).total;
}

long long vmb_vggish_fc_grad_count(void) { return vmb::kFcGradCount; }

int vmb_vggish_refresh_fc(vmb_vggish_t* h, const float* const fc_w[3], const float* const fc_b[3], void* stream) {
  if (!h) return fail("vmb_vggish_refresh_fc: null handle");
  if (!h->has_fc) return fail("vmb_vggish_refresh_fc: this handle was built without the FC stack");
  if (!fc_w || !fc_b) return fail("vmb_vggish_refresh_fc: null argument");
  for (int i = 0; i < 3; ++i)
    if (!fc_w[i] || !fc_b[i]) return fail("vmb_vggish_refresh_fc: null fc tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bool ok = true;
  for (int i = 0; i < 3 && ok; ++i) {   // first call: the training copies (the only allocation; later calls reuse them)
    if (!h->train_w[i])
      ok = cudaMalloc(&h->train_w[i], size_t(kFcOut[i]) * kFcIn[i] * 2 * 3) == cudaSuccess;
    if (ok && i > 0 && !h->train_wt[i])
      ok = cudaMalloc(&h->train_wt[i], size_t(kFcOut[i]) * kFcIn[i] * 2 * 3) == cudaSuccess;
  }
  if (!ok) {
    for (int i = 0; i < 3; ++i) {
      cudaFree(h->train_w[i]);
      cudaFree(h->train_wt[i]);
      h->train_w[i] = h->train_wt[i] = nullptr;
    }
    return fail("vmb_vggish_refresh_fc: allocation failed (%s)", cudaGetErrorString(cudaGetLastError()));
  }
  for (int i = 0; i < 3; ++i) {
    if (!fc_inference_copy(h, i, fc_w[i], fc_b[i], st))
      return fail("vmb_vggish_refresh_fc: %s", vmb::kernels_last_error());
    if (vmb::fc_weight_planes(fc_w[i], kFcOut[i], kFcIn[i], h->train_w[i], h->train_wt[i], st))
      return fail("vmb_vggish_refresh_fc: %s", vmb::kernels_last_error());
  }
  return 0;
}

int vmb_vggish_forward_train(vmb_vggish_t* h, const float* examples, long long n, float* emb, void* workspace,
                             size_t workspace_bytes, void* stream) {
  if (check_train_args(h, n, workspace, workspace_bytes, "vmb_vggish_forward_train")) return 1;
  if (!examples || !emb) return fail("vmb_vggish_forward_train: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const vmb::FcTrainLayout L = train_layout(n);
  char* ws = static_cast<char*>(workspace);
  const char* feat = conv_stack(h, examples, n, ws + L.conv, st, "vmb_vggish_forward_train");
  if (!feat) return 1;
  const void* w[3] = {h->train_w[0], h->train_w[1], h->train_w[2]};
  const float* b[3] = {h->fc_b[0], h->fc_b[1], h->fc_b[2]};
  if (vmb::fc_train_forward(w, b, feat, h->precision, n, ws, L, emb, st))
    return fail("vmb_vggish_forward_train: %s", vmb::kernels_last_error());
  return 0;
}

int vmb_vggish_fc_backward(vmb_vggish_t* h, void* workspace, size_t workspace_bytes, const float* d_emb, long long n,
                           float* grads, void* stream) {
  if (check_train_args(h, n, workspace, workspace_bytes, "vmb_vggish_fc_backward")) return 1;
  if (!d_emb || !grads) return fail("vmb_vggish_fc_backward: null pointer");
  if (reinterpret_cast<uintptr_t>(grads) % 32) return fail("vmb_vggish_fc_backward: grads must be 32-byte aligned");
  const void* wt[3] = {nullptr, h->train_wt[1], h->train_wt[2]};
  if (vmb::fc_train_backward(wt, n, static_cast<char*>(workspace), train_layout(n), d_emb, grads, nullptr,
                             static_cast<cudaStream_t>(stream)))
    return fail("vmb_vggish_fc_backward: %s", vmb::kernels_last_error());
  return 0;
}

// ------------------------------------------------------------------------------------------ train-mode conv4_2
size_t vmb_vggish_conv4_2_train_workspace_bytes(long long n) {
  if (n <= 0) return 0;
  return conv4_2_layout(n).total;
}

int vmb_vggish_refresh_conv4_2(vmb_vggish_t* h, const float* w, const float* b, const float* fc1_w, void* stream) {
  if (!h) return fail("vmb_vggish_refresh_conv4_2: null handle");
  if (!h->has_fc) return fail("vmb_vggish_refresh_conv4_2: this handle was built without the FC stack");
  if (!w || !b || !fc1_w) return fail("vmb_vggish_refresh_conv4_2: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool first = !h->conv_train_w;
  if (first) {   // the only allocations; later calls reuse them
    bool ok = cudaMalloc(&h->conv_train_w, size_t(512) * vmb::kConv42K * 2 * 3) == cudaSuccess;
    if (ok && !h->train_wt[0]) ok = cudaMalloc(&h->train_wt[0], size_t(kFcOut[0]) * kFcIn[0] * 2 * 3) == cudaSuccess;
    if (!ok) {
      cudaFree(h->conv_train_w);
      h->conv_train_w = nullptr;
      return fail("vmb_vggish_refresh_conv4_2: allocation failed (%s)", cudaGetErrorString(cudaGetLastError()));
    }
  }
  // the inference copy, with the create path's own kernels: bit for bit what vmb_vggish_create_ex would build
  const ConvGeom& g = kConv[4];
  if (cudaMemcpyAsync(h->conv_b[5], b, size_t(g.C_out) * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return fail("vmb_vggish_refresh_conv4_2: bias copy failed");
  if ((h->precision == 1 ? vmb::relayout_conv_weight_split(w, h->conv_w[5], g.C_out, g.C_in, st)
                         : vmb::relayout_conv_weight(w, h->conv_w[5], g.C_out, g.C_in, st, h->precision == 2 ? 1 : 0)))
    return fail("vmb_vggish_refresh_conv4_2: %s", vmb::kernels_last_error());
  if (vmb::conv4_2_weight_planes(w, h->conv_train_w, st))
    return fail("vmb_vggish_refresh_conv4_2: %s", vmb::kernels_last_error());
  // fc1's transposed planes (the dgrad of fc1); vmb_vggish_refresh_fc keeps them current from then on
  if (first && vmb::fc_weight_planes(fc1_w, kFcOut[0], kFcIn[0], nullptr, h->train_wt[0], st))
    return fail("vmb_vggish_refresh_conv4_2: %s", vmb::kernels_last_error());
  return 0;
}

int vmb_vggish_forward_train_conv4_2(vmb_vggish_t* h, const float* examples, long long n, float* emb, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  const char* who = "vmb_vggish_forward_train_conv4_2";
  if (check_train_args(h, n, workspace, workspace_bytes, who, true)) return 1;
  if (!examples || !emb) return fail("vmb_vggish_forward_train_conv4_2: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const vmb::Conv42Layout L = conv4_2_layout(n);
  char* ws = static_cast<char*>(workspace);
  const char* act = conv_stack(h, examples, n, ws + L.fc.conv, st, who, 4);
  if (!act) return 1;
  if (vmb::conv4_2_train_forward(h->conv_train_w, h->conv_b[5], act, h->precision, n, ws, L, st))
    return fail("vmb_vggish_forward_train_conv4_2: %s", vmb::kernels_last_error());
  const void* w[3] = {h->train_w[0], h->train_w[1], h->train_w[2]};
  const float* b[3] = {h->fc_b[0], h->fc_b[1], h->fc_b[2]};
  if (vmb::fc_train_forward(w, b, nullptr, h->precision, n, ws, L.fc, emb, st))
    return fail("vmb_vggish_forward_train_conv4_2: %s", vmb::kernels_last_error());
  return 0;
}

int vmb_vggish_conv4_2_backward(vmb_vggish_t* h, void* workspace, size_t workspace_bytes, const float* d_emb,
                                long long n, float* conv_grads, float* fc_grads, void* stream) {
  if (check_train_args(h, n, workspace, workspace_bytes, "vmb_vggish_conv4_2_backward", true)) return 1;
  if (!d_emb || !conv_grads) return fail("vmb_vggish_conv4_2_backward: null pointer");
  if (reinterpret_cast<uintptr_t>(fc_grads) % 32) return fail("vmb_vggish_conv4_2_backward: fc_grads must be 32-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const vmb::Conv42Layout L = conv4_2_layout(n);
  char* ws = static_cast<char*>(workspace);
  const void* wt[3] = {h->train_wt[0], h->train_wt[1], h->train_wt[2]};
  if (vmb::fc_train_backward(wt, n, ws, L.fc, d_emb, fc_grads, reinterpret_cast<float*>(ws + L.dx1), st) ||
      vmb::conv4_2_train_backward(ws + L.fc.conv, h->precision, n, ws, L, conv_grads, st))
    return fail("vmb_vggish_conv4_2_backward: %s", vmb::kernels_last_error());
  return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------ whole path
namespace {
struct PipeLayout { size_t examples, emb, vgg, total; long long n_ex; };
PipeLayout pipe_layout(long long n_clips, long long samples_per_clip, int precision = 1) {
  PipeLayout L{};
  const long long per = vmb_num_examples(samples_per_clip);
  L.n_ex = per > 0 ? per * n_clips : 0;
  L.examples = 0;
  L.emb = align_up(size_t(L.n_ex) * 96 * 64 * 4, 1024);
  L.vgg = L.emb + align_up(size_t(L.n_ex) * 128 * 4, 1024);
  L.total = L.vgg + vmb_vggish_workspace_bytes(L.n_ex) * (precision == 1 ? 2 : 1);
  return L;
}
}  // namespace

size_t vmb_pipeline_workspace_bytes(long long n_clips, long long samples_per_clip) {
  if (n_clips <= 0) return 0;
  return pipe_layout(n_clips, samples_per_clip).total;
}

}  // extern "C"

namespace {
// wave: fp32 samples in [-1, 1] (pcm16 == false) or int16 PCM (scaled by 1/32768 on the device)
int pipeline_forward_any(vmb_vggish_t* vggish, vmb_mla_t* mla, const void* wave, bool pcm16, long long n_clips,
                         long long samples_per_clip, float* scores, float* emb_out, void* workspace,
                         size_t workspace_bytes, void* stream) {
  if (!vggish || !mla) return fail("vmb_pipeline_forward: null handle");
  if (n_clips < 0) return fail("vmb_pipeline_forward: negative n_clips");
  if (n_clips == 0) return 0;
  if (!wave || !scores || !workspace) return fail("vmb_pipeline_forward: null pointer");
  const long long per = vmb_num_examples(samples_per_clip);
  if (per != 10)
    return fail("vmb_pipeline_forward: samples_per_clip must yield exactly T = 10 examples (params.py:26)");
  const PipeLayout L = pipe_layout(n_clips, samples_per_clip, vggish->precision);
  if (workspace_bytes < L.total) return fail("vmb_pipeline_forward: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace) % 1024) return fail("vmb_pipeline_forward: workspace must be 1024-byte aligned");
  char* ws = static_cast<char*>(workspace);
  float* examples = reinterpret_cast<float*>(ws + L.examples);
  float* emb = reinterpret_cast<float*>(ws + L.emb);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // log-mel of the first 96*10 frames of every clip == the (n_clips*10, 96, 64) example tensor
  for (long long c0 = 0; c0 < n_clips; c0 += 32768) {
    const long long nc = n_clips - c0 < 32768 ? n_clips - c0 : 32768;
    vmb::StageTimer t(VMB_STAGE_LOGMEL, st);
    const int rc = pcm16 ? vmb_logmel_pcm16(static_cast<const int16_t*>(wave) + c0 * samples_per_clip, nc,
                                            samples_per_clip, samples_per_clip, per * 96,
                                            examples + c0 * per * 96 * 64, stream)
                         : vmb_logmel(static_cast<const float*>(wave) + c0 * samples_per_clip, nc, samples_per_clip,
                                      samples_per_clip, per * 96, examples + c0 * per * 96 * 64, stream);
    if (rc) return 1;
  }
  if (vmb_vggish_forward(vggish, examples, L.n_ex, emb, nullptr, ws + L.vgg, workspace_bytes - L.vgg, stream)) return 1;
  if (emb_out && cudaMemcpyAsync(emb_out, emb, size_t(L.n_ex) * 128 * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    return fail("vmb_pipeline_forward: embedding copy failed");
  vmb::StageTimer t(VMB_STAGE_MLA, st);
  return vmb_mla_forward(mla, emb, n_clips, scores, stream);
}
}  // namespace

extern "C" {

int vmb_pipeline_forward(vmb_vggish_t* vggish, vmb_mla_t* mla, const float* wave, long long n_clips,
                         long long samples_per_clip, float* scores, float* emb_out, void* workspace,
                         size_t workspace_bytes, void* stream) {
  return pipeline_forward_any(vggish, mla, wave, false, n_clips, samples_per_clip, scores, emb_out, workspace,
                              workspace_bytes, stream);
}

int vmb_pipeline_forward_pcm16(vmb_vggish_t* vggish, vmb_mla_t* mla, const int16_t* pcm, long long n_clips,
                               long long samples_per_clip, float* scores, float* emb_out, void* workspace,
                               size_t workspace_bytes, void* stream) {
  return pipeline_forward_any(vggish, mla, pcm, true, n_clips, samples_per_clip, scores, emb_out, workspace,
                              workspace_bytes, stream);
}

}  // extern "C"

namespace {
int submit_host_any(vmb_vggish_t* vggish, vmb_mla_t* mla, const void* wave_host, bool pcm16, long long n_clips,
                    long long samples_per_clip, float* scores_host, long long clips_per_batch, void* stream) {
  const size_t esz = pcm16 ? 2 : 4;
  if (!vggish || !mla) return -fail("vmb_pipeline_submit_host: null handle");
  if (n_clips <= 0 || clips_per_batch <= 0) return -fail("vmb_pipeline_submit_host: bad sizes");
  if (!wave_host || !scores_host) return -fail("vmb_pipeline_submit_host: null pointer");
  if (vmb_num_examples(samples_per_clip) != 10)
    return -fail("vmb_pipeline_submit_host: samples_per_clip must yield exactly T = 10 examples (params.py:26)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (clips_per_batch > n_clips) clips_per_batch = n_clips;
  const int n_classes = vmb_mla_num_classes(mla);
  HostStage& hs = vggish->stage;
  const int slot = static_cast<int>(hs.calls & 1);
  if (hs.busy[slot]) return -fail("vmb_pipeline_submit_host: two calls are already in flight; wait for the oldest first");
  const size_t wave_bytes = size_t(clips_per_batch) * samples_per_clip * 4;   // sized for fp32 either way
  const size_t ws_bytes = vmb_pipeline_workspace_bytes(clips_per_batch, samples_per_clip);
  const size_t score_bytes = size_t(n_clips) * n_classes * 4;
  bool ok = true;
  if (!hs.copy_st) {
    ok = cudaStreamCreateWithFlags(&hs.copy_st, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i)
      ok = cudaEventCreateWithFlags(&hs.wave_ready[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&hs.wave_free[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&hs.done[i], cudaEventDisableTiming) == cudaSuccess;
  }
  auto grow = [&](void** p, size_t* cap, size_t need) {
    if (!ok || *cap >= need) return;
    cudaStreamSynchronize(hs.copy_st);   // growing is rare: drain both streams before replacing a buffer
    cudaStreamSynchronize(st);
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    ok = cudaMalloc(p, need) == cudaSuccess;
    if (ok) *cap = need;
  };
  grow(&hs.d_wave[0], &hs.wave_cap[0], wave_bytes);
  grow(&hs.d_wave[1], &hs.wave_cap[1], wave_bytes);
  grow(&hs.d_ws, &hs.ws_cap, ws_bytes);
  grow(reinterpret_cast<void**>(&hs.d_scores[slot]), &hs.scores_cap[slot], score_bytes);
  if (!ok) return -fail("vmb_pipeline_submit_host: staging allocation failed (%s)", cudaGetErrorString(cudaGetLastError()));

  int rc = 0;
  for (long long c0 = 0; c0 < n_clips && rc == 0; c0 += clips_per_batch, ++hs.batches) {
    const int s = static_cast<int>(hs.batches & 1);
    const long long nc = n_clips - c0 < clips_per_batch ? n_clips - c0 : clips_per_batch;
    // the buffer is free once the compute that read it two micro-batches ago has finished
    if (hs.batches >= 2) cudaStreamWaitEvent(hs.copy_st, hs.wave_free[s], 0);
    if (cudaMemcpyAsync(hs.d_wave[s], static_cast<const char*>(wave_host) + size_t(c0) * samples_per_clip * esz,
                        size_t(nc) * samples_per_clip * esz, cudaMemcpyHostToDevice, hs.copy_st) != cudaSuccess) {
      rc = fail("vmb_pipeline_submit_host: H2D copy failed (%s)", cudaGetErrorString(cudaGetLastError()));
      break;
    }
    cudaEventRecord(hs.wave_ready[s], hs.copy_st);
    cudaStreamWaitEvent(st, hs.wave_ready[s], 0);
    rc = pipeline_forward_any(vggish, mla, hs.d_wave[s], pcm16, nc, samples_per_clip, hs.d_scores[slot] + c0 * n_classes,
                              nullptr, hs.d_ws, hs.ws_cap, stream);
    cudaEventRecord(hs.wave_free[s], st);
  }
  if (rc == 0 && cudaMemcpyAsync(scores_host, hs.d_scores[slot], score_bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess)
    rc = fail("vmb_pipeline_submit_host: D2H copy failed (%s)", cudaGetErrorString(cudaGetLastError()));
  cudaEventRecord(hs.done[slot], st);
  if (rc) {
    cudaStreamSynchronize(hs.copy_st);
    cudaStreamSynchronize(st);
    return -1;
  }
  hs.busy[slot] = true;
  ++hs.calls;
  return slot;
}
}  // namespace

extern "C" {

int vmb_pipeline_submit_host(vmb_vggish_t* vggish, vmb_mla_t* mla, const float* wave_host, long long n_clips,
                             long long samples_per_clip, float* scores_host, long long clips_per_batch, void* stream) {
  return submit_host_any(vggish, mla, wave_host, false, n_clips, samples_per_clip, scores_host, clips_per_batch, stream);
}

int vmb_pipeline_submit_host_pcm16(vmb_vggish_t* vggish, vmb_mla_t* mla, const int16_t* pcm_host, long long n_clips,
                                   long long samples_per_clip, float* scores_host, long long clips_per_batch,
                                   void* stream) {
  return submit_host_any(vggish, mla, pcm_host, true, n_clips, samples_per_clip, scores_host, clips_per_batch, stream);
}

int vmb_pipeline_wait_host(vmb_vggish_t* vggish, int ticket) {
  if (!vggish) return fail("vmb_pipeline_wait_host: null handle");
  if (ticket < 0 || ticket > 1 || !vggish->stage.busy[ticket]) return fail("vmb_pipeline_wait_host: unknown ticket");
  vggish->stage.busy[ticket] = false;
  if (cudaEventSynchronize(vggish->stage.done[ticket]) != cudaSuccess)
    return fail("vmb_pipeline_wait_host: %s", cudaGetErrorString(cudaGetLastError()));
  if (const int mask = vmb_vggish_saturation(vggish, 1)) {
    char m[16];
    snprintf(m, sizeof m, "0x%x", mask);
    return fail("vmb_pipeline_wait_host: fp16 activations saturated (layer mask %s: bit 0 conv1 .. bit 7 fc2); "
                "create the handle with precision 0 (bf16) or 1 (split)", m);
  }
  return 0;
}

int vmb_pipeline_forward_host(vmb_vggish_t* vggish, vmb_mla_t* mla, const float* wave_host, long long n_clips,
                              long long samples_per_clip, float* scores_host, long long clips_per_batch,
                              void* stream) {
  if (n_clips == 0) return 0;
  const int ticket = vmb_pipeline_submit_host(vggish, mla, wave_host, n_clips, samples_per_clip, scores_host,
                                              clips_per_batch, stream);
  if (ticket < 0) return 1;
  return vmb_pipeline_wait_host(vggish, ticket);
}

}  // extern "C"
