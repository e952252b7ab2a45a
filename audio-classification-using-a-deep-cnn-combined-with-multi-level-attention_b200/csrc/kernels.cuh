// Internal (C++) launch interfaces of the non-GEMM kernels.  Every function returns 0 on success; on failure
// kernels_last_error() holds the reason.  Device pointers throughout.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <utility>

namespace vmb {

const char* kernels_last_error();
void set_kernel_error(const char* fmt, ...);
// cudaGetLastError() -> 0 / 1 with the message recorded.
int check_launch(const char* what);

// Launch `kern` so that it may overlap the tail of the previous kernel in the stream (programmatic dependent launch).
// Only for kernels that call pdl_wait() (sm100_ptx.cuh) before their first access to global memory.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// One-time, PER DEVICE set-up of a kernel (cudaFuncSetAttribute is a per-device property: a process that runs on
// cuda:0 and then on cuda:1 must opt in on both).  `mask` is the call site's static flag word, one bit per device id.
// Returns true when the current device has not been set up through this flag yet; call device_setup_failed() when the
// set-up then fails so that the next call retries.
inline bool device_needs_setup(std::atomic<unsigned long long>& mask) {
  int dev = 0;
  cudaGetDevice(&dev);
  const unsigned long long bit = 1ull << (dev & 63);
  return !(mask.fetch_or(bit, std::memory_order_acq_rel) & bit);
}
inline void device_setup_failed(std::atomic<unsigned long long>& mask) {
  int dev = 0;
  cudaGetDevice(&dev);
  mask.fetch_and(~(1ull << (dev & 63)), std::memory_order_acq_rel);
}

// ---- accounting (profile.cu)
// Every kernel launcher calls count_launch(); StageTimer brackets one stage with CUDA events when profiling is on.
void count_launch(int n = 1);
class StageTimer {
 public:
  StageTimer(int stage, cudaStream_t st);
  ~StageTimer();
  StageTimer(const StageTimer&) = delete;
  StageTimer& operator=(const StageTimer&) = delete;

 private:
  int stage_;
  cudaStream_t st_;
  bool on_;
  cudaEvent_t a_ = nullptr, b_ = nullptr;
};

// ---- front end (frontend.cu)
// Constant tables exactly as mel_features.py builds them (float64): periodic_hann(400) and
// spectrogram_to_mel_matrix(64, 257, 16000, 125, 7500).
void front_end_tables_host(double* hann400, double* mel257x64);
// Tensor-core front end (logmel_tc.cu): centred even / odd DFT as fp16-split tcgen05 GEMMs over TMA-framed raw samples
// with the magnitude / mel / log epilogue; inputs that are not 16-byte aligned take the first version of the kernel
// (bf16 planes of the waveform + straight K = 400 DFT).
int logmel_tc_forward(const float* wave, long long n_clips, long long samples_per_clip, long long clip_stride,
                      long long frames_out, float* logmel, cudaStream_t stream);
// Same for 16-bit PCM input scaled by 1/32768 (vggish_input.py:96-98): the same kernel with 16-bit TMA boxes.
int logmel_tc_forward_pcm16(const int16_t* pcm, long long n_clips, long long samples_per_clip, long long clip_stride,
                            long long frames_out, float* logmel, cudaStream_t stream);
// stft_magnitude (mel_features.py:71-92) on its own, float64 in and out: mag [n_frames][257]
int stft_magnitude_f64(const double* signal, long long n_samples, double* mag, cudaStream_t stream);
// CUDA-core fp32 version of the same computation (frontend.cu); kept as an on-device cross-check, not on the path.
int logmel_forward(const float* wave, long long n_clips, long long samples_per_clip, long long clip_stride,
                   long long frames_out, float* logmel, cudaStream_t stream);

// ---- VGGish odd layers (layers.cu)
// conv1 on the tensor cores (conv1_tc.cu): hand-built im2col tiles, pooling as a max over four TMEM column blocks.
// fmt 1 (kFmtF16): fp16 output (not with split_out); sat_flag: set to 1 when an output saturates the fp16 range.
int conv1_tc_relu_pool(const float* examples, const float* w, const float* b, void* out_bf16, long long n,
                       cudaStream_t stream, bool split_out = false, int fmt = 0, int* sat_flag = nullptr);
// conv1 on the CUDA cores in fp32 (layers.cu): the first implementation, kept as the on-device cross-check.
int conv1_relu_pool(const float* examples, const float* w, const float* b, void* out_bf16, long long n,
                    cudaStream_t stream);
int postprocess(const float* emb, const float* eigen, const float* means, float* out_f32, uint8_t* out_u8,
                long long n, cudaStream_t stream);
// dataset.create_spec + split tiling of <= 4 examples per clip into T windows of (64, 96)
int spec_tiles(const float* examples, long long n_clips, int n_ex, int T, int step, float* out, cudaStream_t stream);
// OIHW fp32 [C_out][C_in][3][3] -> bf16 [C_out][(kh*3+kw)*C_in + c]
int relayout_conv_weight(const float* w_oihw, void* w_bf16, int C_out, int C_in, cudaStream_t stream, int fmt = 0);
// OIHW fp32 -> bf16 [C_out][hi(9 C_in) | lo(9 C_in)], (kh, kw, c) order inside each plane
int relayout_conv_weight_split(const float* w_oihw, void* planes, int C_out, int C_in, cudaStream_t stream);
// fp32 [rows][cols] -> bf16 [rows][hi(cols) | lo(cols)]
int split_f32_to_planes(const float* src, void* planes, long long rows, long long cols, cudaStream_t stream);
// fp32 -> bf16 (fmt 0) or fp16 (fmt 1, saturating) elementwise
int cast_f32_to_bf16(const float* src, void* dst, long long n, cudaStream_t stream, int fmt = 0);

}  // namespace vmb
