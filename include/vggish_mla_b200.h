/* vggish_mla_b200.h — C-ABI of the B200-native waveform -> log-mel -> VGGish -> multi-level-attention path.
 *
 * This is the drop-in boundary behind the reference's Python import surface (the reference has no FFI of
 * its own; SURVEY.md §8b).  Every entry point below names the reference code it replaces
 * (paths relative to the reference root).  All pointers named *_dev are CUDA device pointers owned by the
 * caller (the Python shims pass torch tensors' data_ptr()); `stream` is a cudaStream_t passed as void*.
 * Functions return 0 on success and non-zero on failure; vmb_last_error() then returns a message
 * (thread-local).  Nothing here falls back to the CPU: without a CUDA device every compute entry point fails.
 *
 * Build: libvggish_mla_b200.so, compiled for sm_100a only (see __graft_entry__.build()).
 */
#ifndef VGGISH_MLA_B200_H_
#define VGGISH_MLA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vmb_vggish vmb_vggish_t;
typedef struct vmb_mla vmb_mla_t;
typedef struct vmb_mla_trainer vmb_mla_trainer_t;

/* ------------------------------------------------------------------------------------------ misc */
const char* vmb_last_error(void);
int vmb_abi_version(void);
/* Compute capability of `device` as major*10+minor (100 on B200), or a negative value on error. */
int vmb_device_arch(int device);

/* ------------------------------------------------------------------------------------------ accounting
 * (no reference counterpart: the reference only wall-clocks whole epochs, train.py:71,164-165)
 * Number of CUDA kernels this library has launched in this process.                                   */
long long vmb_launch_count(void);
/* Kernel selection for the bf16 conv3x3 / FC layers with C_out (N) a multiple of 256: 1 = the CTA-pair kernel
 * (tcgen05 cta_group::2, the default), 0 = the single-CTA kernel (kept as the A/B baseline; results are bit-identical),
 * -1 = back to the default (environment VMB_IGEMM_PAIR, else 1).  Returns the previous setting (0/1).  Diagnostics only:
 * the reference has no counterpart (vggish.py:13-19, :108-118 are the layers both kernels implement). */
int vmb_igemm_pair_enable(int on);
/* Same switch for the haloed-box variant of the C_out = 128 conv (conv2, vggish.py:113 with 64 -> 128 channels): one
 * activation box with a one-row halo per (channel block, dx) feeds the three dy taps, instead of one box per tap.
 * 1 (default) / 0 / -1 as above; every bf16 conv kernel adds its partial products in the same order, so the results are
 * bit-identical either way. */
int vmb_igemm_halo_enable(int on);
/* Eval-mode head (model.py:258-269): 1 (default) = the glue between the Linear layers of an embedding chain —
 * BatchNorm1d(T) affine + ReLU + operand split (model.py:219-221) — runs in the GEMM epilogues; 0 = as separate
 * kernels (the A/B baseline: every value is computed by the same expressions, so the scores are bit-identical);
 * -1 = back to the default (environment VMB_MLA_FUSE, else 1).  Returns the previous override (-1 / 0 / 1). */
int vmb_mla_fuse_enable(int on);
/* Per-stage device timing with CUDA events recorded on the caller's stream around each stage of
 * vmb_vggish_forward / vmb_pipeline_forward.  Stage ids: */
enum {
  VMB_STAGE_LOGMEL = 0, VMB_STAGE_CONV1 = 1, VMB_STAGE_CONV2 = 2, VMB_STAGE_CONV3_1 = 3, VMB_STAGE_CONV3_2 = 4,
  VMB_STAGE_CONV4_1 = 5, VMB_STAGE_CONV4_2 = 6, VMB_STAGE_FC1 = 7, VMB_STAGE_FC2 = 8, VMB_STAGE_FC3 = 9,
  VMB_STAGE_MLA = 10, VMB_STAGE_POSTPROCESS = 11, VMB_NUM_STAGES = 12
};
int vmb_profile_enable(int on);
/* Synchronises the recorded events, adds them to the running totals and copies the totals out
 * (milliseconds and call counts per stage, VMB_NUM_STAGES entries each; either may be NULL).           */
int vmb_profile_collect(double* ms_per_stage, long long* calls_per_stage, int reset);

/* ------------------------------------------------------------------------------------------ front end
 * torchvggish/mel_features.py:21-45 (frame), :48-68 (periodic_hann), :71-92 (stft_magnitude),
 * :114-189 (spectrogram_to_mel_matrix), :192-223 (log_mel_spectrogram) and the example framing of
 * torchvggish/vggish_input.py:66-76, with the constants of torchvggish/vggish_params.py:22-36.       */

/* frame(): 1 + floor((n - 400) / 160); negative when n < 400 (the reference raises ValueError there). */
long long vmb_num_frames(long long n_samples);
/* Number of 96-frame examples waveform_to_examples() yields for n_samples at 16 kHz (0 if < 15 600). */
long long vmb_num_examples(long long n_samples);

/* log_mel_spectrogram() for n_clips equally long mono 16 kHz fp32 clips.
 *   wave_dev   [n_clips][clip_stride] fp32 (first samples_per_clip samples of each row are used)
 *   logmel_dev [n_clips][frames_out][64] fp32 where frames_out <= vmb_num_frames(samples_per_clip)
 * Only the first frames_out frames of each clip are produced (pass 96*vmb_num_examples(..) to get the
 * (n_examples, 96, 64) example tensor of waveform_to_examples, vggish_input.py:73-80).
 * The waveform is read in place through TMA; with wave_dev (and, for n_clips > 1, the clip stride in bytes) 16-byte
 * aligned the centred even/odd kernel runs, any other alignment takes the plane kernel (same tolerance, different
 * rounding, so results are bit-identical only between calls that take the same kernel).                   */
int vmb_logmel(const float* wave_dev, long long n_clips, long long samples_per_clip, long long clip_stride,
               long long frames_out, float* logmel_dev, void* stream);

/* The same for 16-bit PCM (what wavfile_to_examples reads, vggish_input.py:96-98): samples are scaled by 1/32768
 * on the device, which is exact in fp32, so the result is bit-identical to vmb_logmel on pcm / 32768.0f (same
 * alignment class); half the input bytes.                                                                        */
int vmb_logmel_pcm16(const int16_t* pcm_dev, long long n_clips, long long samples_per_clip, long long clip_stride,
                     long long frames_out, float* logmel_dev, void* stream);

/* stft_magnitude() on its own (mel_features.py:71-92 with fft_length 512, hop 160, window 400): float64 samples in,
 * float64 magnitudes out like the reference, mag_dev [vmb_num_frames(n_samples)][257].  The fused log-mel kernel never
 * materialises the magnitudes; this is the same centred even / odd DFT in float64 on the CUDA cores, all 257 bins. */
int vmb_stft_magnitude(const double* signal_dev, long long n_samples, double* mag_dev, void* stream);

/* The same computation on the CUDA cores in plain fp32 (the first implementation).  Diagnostic only: an on-device
 * cross-check for the tensor-core kernel at sizes the CPU oracle cannot reach; vmb_pipeline_forward never uses it. */
int vmb_logmel_cudacore(const float* wave_dev, long long n_clips, long long samples_per_clip, long long clip_stride,
                        long long frames_out, float* logmel_dev, void* stream);

/* dataset.create_spec (torchvggish branch, dataset.py:318-326) + dataset.split (dataset.py:329-363) for 4 s clips:
 * the <= 4 examples of each clip [n_clips][n_examples_per_clip][96][64] are laid side by side as a (64 mel, 384 time)
 * spectrogram (missing examples are zero) and cut into n_frames windows of (64, 96): overlapping with step
 * 288 / (n_frames - 1), or contiguous.  out_dev fp32 [n_clips][n_frames][64][96].                         */
int vmb_spec_tiles(const float* examples_dev, long long n_clips, int n_examples_per_clip, int n_frames, int overlap,
                   float* out_dev, void* stream);

/* The constant tables the kernel uses (host copies, for the parity tests against mel_features.py):
 * periodic Hann (400 doubles) and the 257x64 HTK mel matrix (row-major doubles).                      */
int vmb_front_end_tables(double* hann400, double* mel257x64);

/* ------------------------------------------------------------------------------------------ VGGish layers
 * Layer-level entry points (used by the per-layer parity tests and by vmb_vggish_forward).            */

/* features.0 + ReLU + MaxPool (vggish.py:108-118, first conv, C_in = 1): examples fp32 [n][96][64] ->
 * NHWC bf16 [n][48][32][64].  w_dev fp32 [64][9] (OIHW with I = 1), b_dev fp32 [64].                 */
int vmb_conv1_relu_pool(const float* examples_dev, const float* w_dev, const float* b_dev, void* out_bf16_dev,
                        long long n, void* stream);
/* The same with the element type of the output chosen: dtype 0 = bf16, 1 = fp16 (the two 16-bit formats tcgen05
 * kind::f16 multiplies at the same rate; fp16 carries 11 mantissa bits instead of 8).                       */
int vmb_conv1_relu_pool_ex(const float* examples_dev, const float* w_dev, const float* b_dev, void* out_16bit_dev,
                           long long n, int dtype, void* stream);
/* The same layer on the CUDA cores in plain fp32 (the first implementation).  Diagnostic cross-check only. */
int vmb_conv1_relu_pool_cudacore(const float* examples_dev, const float* w_dev, const float* b_dev,
                                 void* out_bf16_dev, long long n, void* stream);

/* Conv2d(3x3, padding=1) + ReLU (+ MaxPool2d(2,2) when pool != 0) as a tcgen05 implicit GEMM.
 *   act_bf16_dev NHWC bf16 [n][H][W][C_in]; w_bf16_dev bf16 [C_out][9*C_in] in (kh, kw, c_in) order;
 *   out NHWC bf16 [n][H(/2)][W(/2)][C_out].  C_in % 64 == 0, C_out % 128 == 0.                       */
int vmb_conv3x3_relu(const void* act_bf16_dev, const void* w_bf16_dev, const float* bias_dev, void* out_bf16_dev,
                     long long n, int H, int W, int C_in, int C_out, int pool, void* stream);

/* dtype 0 = bf16, 1 = fp16: element type of act, w and out (fp16 outputs saturate at 65504 instead of overflowing). */
int vmb_conv3x3_relu_ex(const void* act_dev, const void* w_dev, const float* bias_dev, void* out_dev, long long n, int H,
                        int W, int C_in, int C_out, int pool, int dtype, void* stream);

/* Linear (+ReLU when relu != 0): out[M][N] = act(A[M][K] W[N][K]^T + b).  A, W bf16; out bf16, or fp32 when
 * out_f32 != 0.  K % 64 == 0, N % 128 == 0 (vggish.py:13-19).                                          */
int vmb_linear(const void* a_bf16_dev, const void* w_bf16_dev, const float* bias_dev, void* out_dev, int out_f32,
               int relu, long long M, int N, int K, void* stream);

/* dtype 0 = bf16, 1 = fp16: element type of a, w and of a 16-bit out. */
int vmb_linear_ex(const void* a_dev, const void* w_dev, const float* bias_dev, void* out_dev, int out_f32, int relu,
                  long long M, int N, int K, int dtype, void* stream);

/* Postprocessor.postprocess (vggish.py:62-102): out = round((clamp(E (x - mu), -2, 2) + 2) * 63.75), values
 * 0..255 stored as fp32 like the reference (F6) and optionally also as uint8.  emb_dev fp32 [n][128],
 * eigen_dev fp32 [128][128], means_dev fp32 [128].  Either output may be NULL.                          */
int vmb_postprocess(const float* emb_dev, const float* eigen_dev, const float* means_dev, float* out_f32_dev,
                    uint8_t* out_u8_dev, long long n, void* stream);

/* ------------------------------------------------------------------------------------------ VGGish model
 * VGG.forward (vggish.py:21-31) with weights taken from a reference state_dict (SURVEY.md §8b keys).
 * conv_w_dev[i]: fp32 OIHW, i = features.{0,3,6,8,11,13}; fc_w_dev[i]: fp32 [out][in], i = embeddings.{0,2,4}.
 * The handle owns bf16 re-laid-out copies; the caller's tensors are not referenced after create returns.   */
int vmb_vggish_create(vmb_vggish_t** handle, const float* const conv_w_dev[6], const float* const conv_b_dev[6],
                      const float* const fc_w_dev[3], const float* const fc_b_dev[3], void* stream);
/* precision 0 = vmb_vggish_create (bf16 activations and weights, fp32 accumulation: the throughput mode);
 * precision 1 = accuracy mode: every activation and weight is carried as a hi + lo bf16 pair (16 mantissa bits) and
 * every conv / FC runs the three products hi*hi, lo*hi, hi*lo on the same tcgen05 kernels — 3x the tensor work, for
 * the long-form embedding extraction where the 8-bit quantised output must match the fp32 reference (SURVEY §7 H2). */
/* fc_w_dev and fc_b_dev may both be NULL: the handle then holds the conv stack only and vmb_vggish_forward serves the
 * bottleneck features (emb_dev = NULL) — the reference's just_bottlenecks re-wrap drops the FC layers (model.py:161-166).
 * precision 2 = fp16 activations and weights, fp32 accumulation: the same kernels and the same tensor rate as
 * precision 0 with 11 mantissa bits instead of 8 (operand rounding 8x smaller: the ranking metric of the scores agrees
 * with the fp32 reference to 3 decimals, DESIGN 3).  fp16 ends at 65504: every 16-bit epilogue converts with
 * saturation and raises a per-layer flag when an output reached that maximum; vmb_vggish_saturation() reads the flags
 * and vmb_pipeline_wait_host() fails when one is set (activations of VGGish are O(10), vggish.py:21-31).          */
int vmb_vggish_create_ex(vmb_vggish_t** handle, const float* const conv_w_dev[6], const float* const conv_b_dev[6],
                         const float* const fc_w_dev[3], const float* const fc_b_dev[3], int precision, void* stream);
int vmb_vggish_precision(const vmb_vggish_t* handle);
/* fp16 mode: bit mask of the layers whose 16-bit output saturated since the flags were last cleared (bit 0 conv1,
 * bits 1-5 conv2 .. conv4_2, bit 6 fc1, bit 7 fc2); 0 for the other precisions.  The flags live in mapped host memory
 * and are complete for all work the caller has synchronised with.  clear != 0 resets them.                       */
int vmb_vggish_saturation(vmb_vggish_t* handle, int clear);
void vmb_vggish_destroy(vmb_vggish_t* handle);
/* Scratch bytes vmb_vggish_forward needs for n examples (caller allocates, 1024-byte aligned). */
size_t vmb_vggish_workspace_bytes(long long n_examples);
/* Same for a given handle (the accuracy mode needs twice as much). */
size_t vmb_vggish_handle_workspace_bytes(const vmb_vggish_t* handle, long long n_examples);
/* examples_dev fp32 [n][96][64] -> emb_dev fp32 [n][128] (post-ReLU embeddings, vggish.py:31).
 * If bottleneck_bf16_dev != NULL the (h,w,c)-flattened conv features [n][12288] (vggish.py:26-29; bf16, or fp16
 * for a precision-2 handle) are copied there as well (the reference's just_bottlenecks variant, model.py:162-167).                      */
/* emb_dev may be NULL when only the bottleneck features are wanted (the FC stack is then skipped).            */
int vmb_vggish_forward(vmb_vggish_t* handle, const float* examples_dev, long long n, float* emb_dev,
                       void* bottleneck_bf16_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------ VGGish FC fine-tuning
 * Training embeddings.{0,2,4} (fc1-fc3, vggish.py:13-19,31) with the conv stack frozen: the reference's loop with the
 * CNN's FC parameters given to its Adam (train.py:133-138, the optimiser of train.py:370).  The conv stack runs exactly
 * as in vmb_vggish_forward (same kernels, the handle's precision); the FC stack runs on three-plane split-bf16 operands
 * (hi | mid | lo, fp32-equivalent, the head trainer's GEMMs) from a training copy of the weights that
 * vmb_vggish_refresh_fc derives.  The input gradient of fc1 is not formed.
 *
 * vmb_vggish_refresh_fc: fp32 masters fc_w_dev[i] [out][in], fc_b_dev[i] [out] -> every device copy of the FC weights
 *   (the inference copy in the handle's precision, bit for bit what vmb_vggish_create_ex would build, and the training
 *   planes).  Stream-ordered, no synchronisation; the first call allocates the training planes (~0.5 GB).
 * vmb_vggish_forward_train: examples fp32 [n][96][64] -> emb_dev fp32 [n][128] (post-ReLU embeddings).  The workspace
 *   (vmb_vggish_fc_train_workspace_bytes(n), 1024-byte aligned) keeps what the backward pass needs; it begins with the
 *   operand planes of the conv features, bf16 [pad64(n)][3][12288] (hi, mid, lo: their sum is the fp32 feature).
 * vmb_vggish_fc_backward: d(loss)/d(emb) fp32 [n][128] of the last vmb_vggish_forward_train on this workspace ->
 *   grads_dev, one flat fp32 buffer of vmb_vggish_fc_grad_count() floats (32-byte aligned) in state_dict order:
 *   embeddings.0.weight [4096][12288], .0.bias [4096], .2.weight [4096][4096], .2.bias [4096], .4.weight [128][4096],
 *   .4.bias [128].  Every element is written.                                                                  */
size_t vmb_vggish_fc_train_workspace_bytes(long long n_examples);
long long vmb_vggish_fc_grad_count(void);
int vmb_vggish_refresh_fc(vmb_vggish_t* handle, const float* const fc_w_dev[3], const float* const fc_b_dev[3],
                          void* stream);
int vmb_vggish_forward_train(vmb_vggish_t* handle, const float* examples_dev, long long n, float* emb_dev,
                             void* workspace_dev, size_t workspace_bytes, void* stream);
int vmb_vggish_fc_backward(vmb_vggish_t* handle, void* workspace_dev, size_t workspace_bytes, const float* d_emb_dev,
                           long long n, float* grads_dev, void* stream);

/* ------------------------------------------------------------------------------------------ MLA head
 * MultiLevelAttention.forward in eval mode (model.py:258-269; EmbeddedMapping :217-222, AttentionModule
 * :236-242).  `params_dev` is one flat fp32 device buffer holding, in this order (T = time steps):
 *   for each level l:  norm0 {weight[T], bias[T], running_mean[T], running_var[T]}
 *                      for each fc j of the level: W[H][in] bias[H] norm {weight, bias, mean, var}[T each]
 *   for each level l:  fcv W[K][H] bias[K]; normv {w,b,mean,var}[T]; normf {w,b,mean,var}[T]
 *   fc W[K][L*K] bias[K]; norm {weight, bias, running_mean, running_var}[K each]
 * (fcf is constructed by the reference but never used in forward, model.py:231,238 — it is not passed.) */
int vmb_mla_create(vmb_mla_t** handle, int n_levels, const int* n_fc, int emb_in, int hidden, int n_classes,
                   int t_steps, const float* params_dev, long long n_params, void* stream);
void vmb_mla_destroy(vmb_mla_t* handle);
int vmb_mla_num_classes(const vmb_mla_t* handle);
long long vmb_mla_param_count(int n_levels, const int* n_fc, int emb_in, int hidden, int n_classes, int t_steps);
/* emb_dev fp32 [B][T][emb_in] -> scores_dev fp32 [B][K] (sigmoid outputs, model.py:268).  Every Linear runs as a
 * split-bf16 tcgen05 GEMM (hi + lo operand planes, fp32 accumulation).                                   */
int vmb_mla_forward(vmb_mla_t* handle, const float* emb_dev, long long batch, float* scores_dev, void* stream);
/* One level on its own, for callers that use the reference's sub-modules directly (eval mode):
 *   EmbeddedMapping.forward (model.py:217-222): x_dev fp32 [B][T][in] (in = emb_in for level 0, hidden otherwise) ->
 *     out_dev fp32 [B][T][hidden] = norm0 -> (Linear -> BatchNorm1d(T) -> ReLU) x n_fc (dropout is the identity in eval);
 *   AttentionModule.forward (model.py:235-242): h_dev fp32 [B][T][hidden] -> y_dev fp32 [B][K]
 *     (softmax over the class axis, fcv feeding both branches: SURVEY F3, F4).
 * Same kernels and arithmetic as inside vmb_mla_forward.                                                       */
int vmb_mla_embedded_mapping(vmb_mla_t* handle, int level, const float* x_dev, long long batch, float* out_dev,
                             void* stream);
int vmb_mla_attention(vmb_mla_t* handle, int level, const float* h_dev, long long batch, float* y_dev, void* stream);
/* The same head as ONE fused CUDA-core fp32 kernel (the first implementation; emb_in <= 608).  Diagnostic: the
 * on-device cross-check for vmb_mla_forward; vmb_pipeline_forward never uses it.                         */
int vmb_mla_forward_fp32(vmb_mla_t* handle, const float* emb_dev, long long batch, float* scores_dev, void* stream);

/* ------------------------------------------------------------------------------------------ MLA head training
 * One optimisation step of the head as the reference's train loop runs it (train.py:119-138, :369-372) with the CNN
 * frozen (model.py:159-160): forward in train mode — BatchNorm with batch statistics per time step (SURVEY F5),
 * Dropout(p) after each ReLU (model.py:212,220), nn.CrossEntropyLoss on the sigmoid outputs — and backward.
 * Flat layouts (fp32):
 *   params / grads: named_parameters() order of MultiLevelAttention with fcf left out (it never gets a gradient, F3):
 *     for each level l: norm0.{weight,bias}[T]; fc.{j}.{weight[H][in],bias[H]} for all j; norms.{j}.{weight,bias}[T];
 *     for each level l: fcv.{weight[K][H],bias[K]}; normv.{weight,bias}[T]; normf.{weight,bias}[T];
 *     fc.{weight[K][L*K],bias[K]}; norm.{weight,bias}[K]
 *   running: for every BatchNorm in the same order {running_mean[n], running_var[n]} — updated in place like
 *     nn.BatchNorm1d does (momentum 0.1, unbiased variance).
 * vmb_mla_train_step zeroes `grads` and `loss`, then writes d(loss)/d(params) of THIS rank's batch into grads (ready
 * for one flat NCCL all-reduce across data-parallel ranks) and the mean loss into *loss_dev.  scores_dev (optional)
 * receives the train-mode outputs [batch][K].  Dropout uses a counter-based generator keyed by (seed, layer, element).
 * The first vmb_mla_train_step of a handle launches its kernels one by one; from the second call on the whole step —
 * ~47 kernels, memsets and the fork / join of the handle's side streams — is replayed as ONE CUDA graph on a stream
 * owned by the handle, ordered after / before `stream` by events.  x / labels are copied into staging buffers owned by
 * the handle first and the seed is written to device memory, so any input addresses and any seed may follow; a distinct
 * (params, running, grads, loss, scores, batch, dropout_p) captures its own graph (four are kept).  Environment
 * VMB_TRAIN_GRAPH=0 keeps the eager launches; the results are the same either way.
 * vmb_mla_trainer_create: 1..4 levels of 1..4 Linears, hidden and n_classes in 1..1024, T in 1..16, emb_in in
 * 1..16384.  An emb_in wider than the hidden width (padded to 128: the just_bottlenecks head, emb_in = 12288) takes a
 * wide-first-layer path: no gradient with respect to the input is formed (the CNN is frozen), only the forward and the
 * weight-gradient GEMM run over the input width.
 * max_batch: 2 <= max_batch and max_batch * T <= 2^31 / 2048; with the wide path also
 * pad64(max_batch * T) * 3 * pad128(emb_in) < 2^31 (the element count of the input's operand planes; 5824 clips at
 * emb_in = 12288, T = 10).  A larger max_batch is rejected before anything is allocated. */
long long vmb_mla_train_param_count(int n_levels, const int* n_fc, int emb_in, int hidden, int n_classes, int t_steps,
                                    long long* n_running_out);
int vmb_mla_trainer_create(vmb_mla_trainer_t** handle, int n_levels, const int* n_fc, int emb_in, int hidden,
                           int n_classes, int t_steps, long long max_batch, void* stream);
void vmb_mla_trainer_destroy(vmb_mla_trainer_t* handle);
int vmb_mla_train_step(vmb_mla_trainer_t* handle, const float* params_dev, float* running_dev, const float* emb_dev,
                       const long long* labels_dev, long long batch, float dropout_p, unsigned long long seed,
                       float* grads_dev, float* loss_dev, float* scores_dev, void* stream);
/* Overlapping the gradient all-reduce with the backward pass (train.py:133-138 under data parallelism): the backward
 * pass computes level 0's embedding chain last, and that chain's parameters come first in the flat order, so
 * grads[vmb_mla_train_tail_offset() .. n_params) are final before it starts.  vmb_mla_train_wait_tail makes `stream`
 * wait for that point of the most recently enqueued vmb_mla_train_step / vmb_mla_train_backward: a caller enqueues the
 * all-reduce of the tail there and only the head of the bucket after the whole step. */
long long vmb_mla_train_tail_offset(const vmb_mla_trainer_t* handle);
int vmb_mla_train_wait_tail(vmb_mla_trainer_t* handle, void* stream);
/* The same step in two calls, for callers that compute the loss themselves (the reference's `criterion(outputs,
 * labels); loss.backward()`, train.py:130-136): forward leaves its state in the handle, backward takes
 * d(loss)/d(scores) [batch][K].  One step in flight per handle.                                              */
int vmb_mla_train_forward(vmb_mla_trainer_t* handle, const float* params_dev, float* running_dev, const float* emb_dev,
                          long long batch, float dropout_p, unsigned long long seed, float* scores_dev, void* stream);
int vmb_mla_train_backward(vmb_mla_trainer_t* handle, const float* params_dev, const float* emb_dev,
                           const float* dscores_dev, long long batch, float dropout_p, unsigned long long seed,
                           float* grads_dev, void* stream);
/* vmb_mla_train_backward plus the gradient with respect to the embeddings, dx_dev fp32 [batch][T][emb_in] (the input of
 * a trainable CNN body in front of the head, train.py:133-138 with the optimiser of train.py:370): norm0's backward
 * pass to its input, dx = gamma_t rstd_t (g - mean_t g - xhat mean_t(g xhat)).  Only when the padded emb_in does not
 * exceed the padded hidden width (the wide first layer has no dX GEMM): otherwise it fails.                      */
int vmb_mla_train_backward_dx(vmb_mla_trainer_t* handle, const float* params_dev, const float* emb_dev,
                              const float* dscores_dev, long long batch, float dropout_p, unsigned long long seed,
                              float* grads_dev, float* dx_dev, void* stream);
/* torch.optim.Adam (amsgrad = False) on flat buffers (train.py:369): step counts from 1; grads are multiplied by
 * grad_scale first (1/world_size after a SUM all-reduce).                                                 */
int vmb_adam_step(float* params_dev, const float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev, long long n,
                  float lr, float beta1, float beta2, float eps, float weight_decay, long long step, float grad_scale,
                  void* stream);

/* ------------------------------------------------------------------------------------------ data-parallel optimiser step
 * (the reference trains on one device: train.py:133-138 `loss.backward(); optimizer.step()`; BASELINE configs[4] runs that
 * step data-parallel over the GPUs of one box, which adds "average the gradients over the ranks" between the two calls).
 * One process per GPU.  Every rank creates a vmb_dp: its arena (params | two gradient buffers | flags) is device memory
 * owned by the library and exported through CUDA IPC; the ranks exchange the VMB_DP_IPC_HANDLE_BYTES-byte handles by any
 * host-side means (the Python layer uses torch.distributed.all_gather_object) and call vmb_dp_connect with all `world`
 * handles in rank order.  vmb_mla_train_step then takes vmb_dp_params() as params_dev and vmb_dp_grads(parity) as
 * grads_dev, parity alternating 0 / 1 from step to step, and vmb_dp_adam_step(parity) replaces all-reduce + vmb_adam_step:
 * a cross-GPU barrier, ONE kernel that sums this rank's slice (vmb_dp_slice) of all ranks' gradient buffers over NVLink
 * peer loads in rank order, scales by 1 / world, applies the Adam update of vmb_adam_step to the slice and stores the new
 * parameters into every rank's arena, and a second barrier.  exp_avg / exp_avg_sq: this rank's moments, (n_params + 3) / 4
 * * 4 floats each, only the rank's slice is used.  A barrier that a rank does not reach within 10 s gives up and
 * vmb_dp_status() reports it (non-zero) instead of hanging the GPU.  Shutdown: every rank calls vmb_dp_disconnect, the
 * ranks synchronise on the host, then vmb_dp_destroy frees the arena. */
#define VMB_DP_IPC_HANDLE_BYTES 64
typedef struct vmb_dp vmb_dp_t;
void vmb_dp_slice(long long n_params, int world, int rank, long long* begin, long long* end);
int vmb_dp_create(vmb_dp_t** handle, long long n_params, int rank, int world, void* ipc_handle_out);
int vmb_dp_connect(vmb_dp_t* handle, const void* all_handles);
float* vmb_dp_params(vmb_dp_t* handle);
float* vmb_dp_grads(vmb_dp_t* handle, int parity);
int vmb_dp_adam_step(vmb_dp_t* handle, int parity, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2,
                     float eps, float weight_decay, long long step, void* stream);
int vmb_dp_status(vmb_dp_t* handle);
void vmb_dp_disconnect(vmb_dp_t* handle);
void vmb_dp_destroy(vmb_dp_t* handle);

/* ------------------------------------------------------------------------------------------ whole path
 * Ensemble.forward for cnn_type == "vggish" (model.py:58-62) fed from raw audio:
 * wave [n_clips][samples_per_clip] fp32 16 kHz -> scores [n_clips][K].  samples_per_clip must yield exactly
 * T examples (10 s -> 10).  Device-resident variant: everything already in HBM.                         */
/* (sized for the accuracy mode, i.e. enough for either precision) */
size_t vmb_pipeline_workspace_bytes(long long n_clips, long long samples_per_clip);
int vmb_pipeline_forward(vmb_vggish_t* vggish, vmb_mla_t* mla, const float* wave_dev, long long n_clips,
                         long long samples_per_clip, float* scores_dev, float* emb_dev_or_null,
                         void* workspace_dev, size_t workspace_bytes, void* stream);
/* The same fed with 16-bit PCM (pcm / 32768 on the device, exact; see vmb_logmel_pcm16): half the input bytes. */
int vmb_pipeline_forward_pcm16(vmb_vggish_t* vggish, vmb_mla_t* mla, const int16_t* pcm_dev, long long n_clips,
                               long long samples_per_clip, float* scores_dev, float* emb_dev_or_null,
                               void* workspace_dev, size_t workspace_bytes, void* stream);
/* Host-buffer variant (the end-to-end number of bench.py): wave_host / scores_host are HOST pointers
 * (pinned for full speed); the call copies H2D, runs the path on `stream` in micro-batches of
 * `clips_per_batch` (the copy of micro-batch i+1 overlaps the compute of micro-batch i), copies the scores D2H
 * and synchronises before returning.                                                                    */
int vmb_pipeline_forward_host(vmb_vggish_t* vggish, vmb_mla_t* mla, const float* wave_host, long long n_clips,
                              long long samples_per_clip, float* scores_host, long long clips_per_batch,
                              void* stream);
/* The same call split in two so that a caller can keep the device busy across calls (a DataLoader-style loop):
 * submit enqueues the H2D copies, the compute and the D2H copy and returns a ticket (0 or 1) at once, or a
 * negative value on error; wait blocks until that call's scores are in scores_host.  At most two calls in flight;
 * wave_host must stay valid until wait returns.  Tickets must be waited in submission order.                 */
int vmb_pipeline_submit_host(vmb_vggish_t* vggish, vmb_mla_t* mla, const float* wave_host, long long n_clips,
                             long long samples_per_clip, float* scores_host, long long clips_per_batch, void* stream);
int vmb_pipeline_submit_host_pcm16(vmb_vggish_t* vggish, vmb_mla_t* mla, const int16_t* pcm_host, long long n_clips,
                                   long long samples_per_clip, float* scores_host, long long clips_per_batch,
                                   void* stream);
int vmb_pipeline_wait_host(vmb_vggish_t* vggish, int ticket);

#ifdef __cplusplus
}
#endif
#endif /* VGGISH_MLA_B200_H_ */
