/* vadx.h -- C ABI of libvadx.so, the B200 (sm_100a) batched VAD engine.
 *
 * This is the drop-in boundary for the hot path of DakeQQ/Voice-Activity-Detection-VAD-ONNX:
 * where the reference calls `onnxruntime.InferenceSession.run()` on one chunk of one stream
 * (FSMN/Inference_FSMN_VAD_ONNX.py:177-187, FireRedVAD/Inference_FireRed_ONNX.py:567-572,
 * NVIDIA_Frame_VAD_Multilingual_MarbleNet/Inference_NVIDIA_MarbleNet_VAD_ONNX.py:366-377,
 * DFSMN/near_and_far_end_audio/Inference_DFSMN_VAD_ONNX.py:229-230,
 * Silero/modeling_modified/utils_vad.py:114-123) a caller binds `vadx_forward` on S streams at
 * once, and where the reference runs its Python post-processing loops
 * (FireRedVAD/Inference_FireRed_ONNX.py:102-305, FSMN/Inference_FSMN_VAD_ONNX.py:188-234) it
 * binds `vadx_postprocess_*`.
 *
 * Conventions
 *   - plain C: pointers and sizes only; no torch / C++ types cross this boundary.
 *   - every pointer named `d_*` is a DEVICE pointer owned by the caller; the library borrows it
 *     for the duration of the (asynchronous) call and never allocates after vadx_create /
 *     vadx_set_tensor.  `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, a negative VADX_E* code otherwise;
 *     vadx_last_error() returns the message of the calling thread's last failure.
 *   - activations are TIME-MAJOR: [stream][frame][channel], channel contiguous, fp32.
 *   - there is no CPU implementation behind this ABI: without a CUDA device every compute entry
 *     point fails with VADX_ENODEVICE.
 */
#ifndef VADX_H_
#define VADX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VADX_ABI_VERSION 1

enum {
  VADX_OK = 0,
  VADX_EINVAL = -1,    /* bad argument / shape (ORT: InvalidArgument) */
  VADX_ENODEVICE = -2, /* no CUDA device / driver */
  VADX_ECUDA = -3,     /* a CUDA call or kernel launch failed */
  VADX_EMISSING = -4,  /* a tensor the model needs was never set */
  VADX_ENOMEM = -5     /* caller workspace too small */
};

enum { VADX_DT_I16 = 0, VADX_DT_F32 = 1, VADX_DT_I32 = 2 };
/* activation codes; OR VADX_ACT_RES_FIRST in to add the residual BEFORE the activation
 * (JasperBlock: relu(conv + residual)) instead of after it (DFSMN: act(conv) + residual).
 * VADX_ACT_SOFTMAX is only valid for narrow heads (n_out <= 8): softmax across the n_out outputs. */
enum { VADX_ACT_NONE = 0, VADX_ACT_RELU = 1, VADX_ACT_SIGMOID = 2, VADX_ACT_SOFTMAX = 3,
       /* tensor-core path only (the log-mel contraction as a dense layer): y = log(x.W + bias), and
        * y = log(max(x.W, bias)) with the bias vector holding the per-column floor */
       VADX_ACT_LOG = 4, VADX_ACT_LOG_CLAMP = 5, VADX_ACT_RES_FIRST = 16 };
enum { VADX_FLOOR_CLAMP = 0, VADX_FLOOR_ADD = 1 };
/* pre-emphasis flavours: NONE; ZERO_HISTORY: y[0]=x[0]-c*0 (pad(1,0)+conv[-c,1],
 * FireRedVAD/Export_FireRedVAD.py:440, NVIDIA_Frame_VAD_Multilingual_MarbleNet/Export_NVIDIA_MarbleNet_VAD.py:245-246);
 * KEEP_FIRST: y[0]=x[0] (FSMN/Export_FSMN_VAD.py:78-79, DFSMN Export_DFSMN_VAD.py:338-341) */
enum { VADX_PREEMPH_NONE = 0, VADX_PREEMPH_ZERO_HISTORY = 1, VADX_PREEMPH_KEEP_FIRST = 2 };

int vadx_abi_version(void);
const char* vadx_last_error(void);
/* number of CUDA devices visible (0 when there is none); never fails */
int vadx_device_count(void);
/* kernels launched by this library since load (all threads); used by bench.py for gpu_launches */
uint64_t vadx_launch_count(void);

/* Optional per-stage device timing (used by bench.py for the live roofline numbers): while enabled,
 * every per-kernel entry point brackets its launches with CUDA events on the caller's stream.
 * vadx_profile_collect synchronises those events, ADDS the elapsed milliseconds and the number of
 * calls of each stage into ms[] / calls[] (n_stages entries, indexed by VADX_STAGE_*) and clears
 * the recorded events. */
enum {
  VADX_STAGE_PREP = 0,
  VADX_STAGE_STFT = 1,
  VADX_STAGE_MEL = 2,
  VADX_STAGE_LINEAR = 3,
  VADX_STAGE_MEMORY = 4,
  VADX_STAGE_HEAD = 5,
  VADX_STAGE_POSTPROC = 6,
  VADX_STAGE_COUNT = 7
};
int vadx_profile_enable(int on);
int vadx_profile_collect(double* ms, uint64_t* calls, int n_stages);
/* The same records per KERNEL: every entry point also reports the name of the kernel it launches and the algorithmic
 * bytes (tensors read + written once) and flops (2 x MACs) of the call, so a caller gets achieved GB/s and FLOP/s per
 * kernel without re-deriving shapes.  Fills out[0 .. *n_out) and clears the totals; when capacity is too small only
 * *n_out is set (nothing is cleared).  Names are static strings owned by the library. */
typedef struct vadx_kernel_stat {
  const char* name;
  double ms;
  uint64_t calls;
  double bytes;
  double flops;
} vadx_kernel_stat;
int vadx_profile_collect_kernels(vadx_kernel_stat* out, int capacity, int* n_out);

/* ------------------------------------------------------------------------------------------
 * Per-kernel entry points (also what the unit parity tests and ncu captures call).
 * ------------------------------------------------------------------------------------------ */

/* a2 -- cast / scale / DC removal / pre-emphasis / zero centre-pad, one pass.
 * d_audio [S][in_stride] (int16 or fp32; in_stride < n_samples = overlapping windows of one recording) -> d_out
 * [S][out_stride] fp32 with
 * out[s][pad_left + n] = y[n], zeros in [0,pad_left) and [pad_left+L, out_stride).
 * remove_dc: subtract the mean over the L samples of the stream's chunk first
 * (FSMN/Export_FSMN_VAD.py:77). */
int vadx_prep_audio(const void* d_audio, int in_dtype, int64_t n_streams, int64_t n_samples,
                    int64_t in_stride, float scale, int remove_dc, int preemph_mode, float preemph,
                    int64_t pad_left, float* d_out, int64_t out_stride, void* stream);

/* a1 -- framed real DFT as a GEMM + power: for frame t of stream s
 *   re/im[f] = sum_k d_sig[s][t*hop + k] * basis[k][2f / 2f+1]   (k < n_taps)
 *   d_power[(s*T + t)*ld_power + f] = re^2 + im^2
 * d_basis is [n_taps][ld_basis] with re/im interleaved along the row (ld_basis >= 2*n_bins,
 * multiple of 4).  Replaces STFT_Process.stft_B_forward (FSMN/STFT_Process.py:144-157,
 * FireRedVAD/STFT_Process.py:264-278) followed by `real*real + imag*imag`. */
int vadx_stft_power_f32(const float* d_sig, int64_t sig_stride, int64_t n_streams, int n_frames, int hop,
                        int n_taps, const float* d_basis, int ld_basis, int n_bins, float* d_power,
                        int64_t ld_power, void* stream);

/* a1 + a2 on the tensor cores, straight from int16 audio (tcgen05.mma, TMEM accumulators): valid when every
 * frame lies inside the stream's n_samples and no DC removal is needed (FireRedVAD).  The int16 sample
 * splits exactly into two bf16 terms; pre-emphasis (y[i] = x[i] - c*x[i-1], x[-1] = 0) and the scale are
 * folded into the basis, which vadx_pack_stft_basis_tc splits into three bf16 terms and lays out as the
 * shared-memory operand image (h_basis = the fp32 table of vadx_stft_power_f32; h_img = NULL queries the
 * size).  Result: d_power[(s*T + t)*ld_power + f] = re^2 + im^2, fp32-grade. */
int vadx_stft_tc_supported(int n_taps, int n_bins);
int vadx_pack_stft_basis_tc(const float* h_basis, int ld_basis, int n_taps, int n_bins, double preemph, double scale,
                            void* h_img, size_t img_capacity, size_t* img_bytes);
int vadx_stft_power_tc_i16(const int16_t* d_audio, int64_t in_stride, int64_t n_samples, int64_t n_streams,
                           int n_frames, int hop, int n_taps, const void* d_img, int n_bins, float* d_power,
                           int64_t ld_power, void* stream);
/* Centre-padded and / or DC-removed frontends (FSMN, MarbleNet) on the same kernel: frame t starts pad_left
 * samples before t*hop (zeros outside [0, n_samples)); with the mean given (vadx_stream_mean_i16 splits it into
 * its nearest integer and the remainder) it is removed BEFORE the pre-emphasis, as FSMN/Export_FSMN_VAD.py:76-79
 * does: the integer part exactly, from the samples in the loaders, the remainder in the frequency domain,
 * X(x - m) = X(x) - m * D_t, D_t the folded basis applied to the mean's coefficient pattern
 * (vadx_pack_stft_dc_tc: one row for interior frames, one per frame touching the pad, then the tail rows that
 * undo the folded pre-emphasis' spill past the end of the stream). */
int vadx_pack_stft_dc_tc(const float* h_basis, int ld_basis, int n_taps, int n_bins, double preemph, double scale,
                         int64_t n_samples, int hop, int pad_left, int n_frames, float* h_tables, size_t capacity_floats,
                         size_t* n_floats, int* n_edge_lo, int* t_edge_hi);
int vadx_stream_mean_i16(const int16_t* d_audio, int64_t in_stride, int64_t n_samples, int64_t n_streams,
                         float* d_mean_frac, int32_t* d_mean_int, void* stream);
int vadx_stft_power_tc_i16_ex(const int16_t* d_audio, int64_t in_stride, int64_t n_samples, int64_t n_streams,
                              int n_frames, int hop, int n_taps, const void* d_img, int n_bins, float* d_power,
                              int64_t ld_power, int pad_left, const float* d_mean_frac, const int32_t* d_mean_int,
                              const float* d_dc_tables, int n_edge_lo, int t_edge_hi, float power_scale,
                              int operand_format, void* stream);
/* Operand format of a DFT basis image and of the samples the loaders build to match it: bf16 (the default of
 * vadx_pack_stft_basis_tc) or fp16 -- fp16 makes the exact int16 split three half2 operations per pair of
 * samples and gives the two-term basis 22 bits; it cannot carry the 17-bit mean-removed samples, and a scale
 * such as 1/32768 must stay out of the basis (pass scale = 1 and power_scale = scale^2 to the kernel). */
enum { VADX_TC_FMT_BF16 = 0, VADX_TC_FMT_F16 = 1 };
int vadx_pack_stft_basis_tc_fmt(const float* h_basis, int ld_basis, int n_taps, int n_bins, double preemph, double scale,
                                int operand_format, void* h_img, size_t img_capacity, size_t* img_bytes);

/* a3 -- triangular filterbank contraction + floor + ln.  The bank is passed in its sparse form:
 * filter m covers bins [start[m], start[m]+len[m]) with weights d_w[m*max_len + j].
 * out[row*ld_out + m] = ln(floor(sum_j w*power)). */
int vadx_mel_log_f32(const float* d_power, int64_t ld_power, int64_t n_rows, int n_bins, int n_mels,
                     const int32_t* d_start, const int32_t* d_len, const float* d_w, int max_len,
                     int floor_mode, float floor_value, float* d_out, int64_t ld_out, void* stream);

/* a8 -- dense layer on [rows][in]: Y = act(X * Wt + bias) (+ residual).
 * d_wt is the TRANSPOSED weight [in][ldw] (ldw >= out, multiple of 4, zero padded). */
int vadx_linear_f32(const float* d_x, int64_t ldx, const float* d_wt, int ldw, const float* d_bias,
                    const float* d_residual, int64_t ldr, float* d_y, int64_t ldy, int64_t n_rows, int n_in,
                    int n_out, int act, void* stream);

/* a8 on the tensor cores (tcgen05.mma, TMEM accumulators): same contract as vadx_linear_f32 but the
 * weight is passed as the packed operand image built ONCE on the host by vadx_pack_weight_tc
 * (bf16 hi/lo split, K-major, 128-byte swizzled 64-column tiles).  fp32-grade: both operands are
 * split into two bf16 terms and three products are accumulated in fp32.
 * vadx_tc_supported: 1 when (n_in, n_out) fits the weights-stationary kernel (n_out in 9..256 and
 * the image + two activation stages fit in shared memory).
 * vadx_pack_weight_tc: h_w is the reference-layout weight [n_out][n_in] on the HOST; call with
 * h_img = NULL to query *img_bytes.
 * Output rows without a residual input leave through 2-D tensor-map bulk stores (cp.async.bulk.tensor) when ldy % 4 == 0
 * and d_y is 16-byte aligned; the map is encoded per call (cuTensorMapEncodeTiled via cudaGetDriverEntryPoint; the library
 * does not link against libcuda) and the per-lane store path is taken when the driver does not export the encoder. */
int vadx_tc_supported(int n_in, int n_out);
int vadx_pack_weight_tc(const float* h_w, int n_out, int n_in, void* h_img, size_t img_capacity, size_t* img_bytes);
int vadx_linear_tc_f32(const float* d_x, int64_t ldx, const void* d_wimg, const float* d_bias,
                       const float* d_residual, int64_t ldr, float* d_y, int64_t ldy, int64_t n_rows, int n_in,
                       int n_out, int act, void* stream);

/* a12 -- depthwise conv1d over time on time-major activations [S][T_in][C] (MarbleNet / Jasper separable
 * blocks): y[s][t][c] = sum_j w[c][j] * x[s][t*stride - pad + j*dilation][c], zeros outside [0, T_in). */
int vadx_depthwise_conv1d_f32(const float* d_x, int64_t ldx, const float* d_w, int kernel, int stride, int dilation,
                              int pad, float* d_y, int64_t ldy, int64_t n_streams, int t_in, int t_out,
                              int n_channels, void* stream);

/* a8 with the 1-output sigmoid head fused into the epilogue (FireRed: dnn 128->256 + ReLU, out 256->1, sigmoid):
 * d_head_out[row] = sigmoid(sum_n act(x*W^T + b)[n] * d_head_w[n] + head_bias); the n_out-wide layer output
 * never leaves the SM. */
int vadx_linear_head_tc_f32(const float* d_x, int64_t ldx, const void* d_wimg, const float* d_bias, int64_t n_rows,
                            int n_in, int n_out, int act, const float* d_head_w, float head_bias, float* d_head_out,
                            void* stream);

/* a5/a6/a7 -- FSMN / DFSMN memory block on time-major activations [S][T][C]:
 *   out[t] = p[t] + sum_k wl[c][k] * p[t - (n_back-1-k)*stride_back]
 *                 + sum_k wr[c][k] * p[t + (k+1)*stride_ahead]        (only when T > 1)
 *                 (+ residual[t])
 * frames before 0 come from d_cache_in [S][C][(n_back-1)*stride_back] (channel-first, the
 * reference's cache layout: FSMN/Export_FSMN_VAD.py:116, FireRedVAD/Export_FireRedVAD.py:496-515)
 * or are zero when it is NULL; frames >= T are zero.  d_cache_out (optional) receives the last
 * (n_back-1)*stride_back frames of cat(cache, p).  d_wl is [C][n_back], d_wr is [C][n_ahead]. */
int vadx_fsmn_memory_f32(const float* d_p, int64_t ldp, const float* d_wl, int n_back, int stride_back,
                         const float* d_wr, int n_ahead, int stride_ahead, const float* d_residual,
                         int64_t ldr, float* d_out, int64_t ldo, int64_t n_streams, int n_frames,
                         int n_channels, const float* d_cache_in, float* d_cache_out, void* stream);

/* a8 + a6 fused -- one DFSMN block (FireRedVAD/Export_FireRedVAD.py:253-263 fc1/fc2, :213-236 memory block) as TWO
 * tensor-core kernels that hand the hidden rows over in the MMA operand format:
 *   vadx_linear_tc_stream_stages_f32:  h = act(x W1^T + b1), written as per-stream operand stages
 *       d_himg [S][n_out/64][hi | lo][round_up(T,16) rows x 128 B] (two-term bf16 split, 128-byte swizzled);
 *       d_x [S*T][n_in] fp32 rows, n_out % 64 == 0, rows_per_stream = T;
 *   vadx_fc2_memory_stages_f32:  p = act(h W2^T + b2) issued transposed (accumulator = p^T in tensor memory),
 *       out = p + FIR_back(p) + FIR_ahead(p) (+ residual); d_residual / d_out [S*T][128]; p never reaches HBM.
 * Supported: n_out(fc2) = 128, n_in(fc2) in {64,128,192,256}, n_frames = 98, 20 + 20 unit-stride taps (a chunk is
 * zero-padded in time by definition, so there is no halo); act NONE or RELU.  d_wimg from vadx_pack_weight_tc.
 * d_himg, d_wimg and d_residual must be 16-byte aligned (they are read with bulk copies); d_wl and d_wr are required.
 * The stages are written with bulk stores (shared -> global) when rows_per_stream >= 32, else with per-lane stores. */
size_t vadx_fc2_memory_stages_stream_bytes(int n_in, int n_frames);
int vadx_fc2_memory_stages_supported(int n_in, int n_out, int n_frames, int n_back, int stride_back, int n_ahead,
                                     int stride_ahead);
int vadx_linear_tc_stream_stages_f32(const float* d_x, const void* d_wimg, const float* d_bias, void* d_himg,
                                     int64_t n_rows, int rows_per_stream, int n_in, int n_out, int act, void* stream);
int vadx_fc2_memory_stages_f32(const void* d_himg, int n_in, const void* d_wimg, const float* d_bias, int act,
                               const float* d_wl, int n_back, const float* d_wr, int n_ahead, const float* d_residual,
                               float* d_out, int64_t n_streams, int n_frames, void* stream);

/* a4 -- FunASR low-frame-rate stacking + CMVN (FSMN/Export_FSMN_VAD.py:65-70,82-86):
 * out[s][t][j*n_mels + m] = (mel[s][clamp(t + j - (lfr_m-1)/2, 0, T-1)][m] + mean[..]) * var[..]; lfr_n = 1. */
int vadx_lfr_cmvn_f32(const float* d_mel, int64_t ld_mel, const float* d_mean, const float* d_var, float* d_out,
                      int64_t ld_out, int64_t n_streams, int n_frames, int n_mels, int lfr_m, int lfr_n, void* stream);

/* a8 head of the FunASR encoder: softmax over n_classes, keep class 0 (= P(silence),
 * FSMN/modeling_modified/encoder.py:217). */
int vadx_softmax_class0_f32(const float* d_logits, int64_t ld, int64_t n_rows, int n_classes, float* d_p0,
                            void* stream);

/* a9 -- frame energy of the prepared signal: out[s][t] = log10(sum_{n<win}(sig[s][offset+t*hop+n]*scale)^2 + eps)
 * for t < n_energy, the last value replicated up to n_frames (FSMN/Export_FSMN_VAD.py:93-97). */
int vadx_frame_energy_log10_f32(const float* d_sig, int64_t sig_stride, int64_t offset, int64_t n_streams, int win,
                                int hop, int n_energy, int n_frames, float scale, float eps, float* d_out,
                                void* stream);

/* a9 -- gate: score2 = p + (ratio>1 ? p^ratio : ratio<1 ? 1 : p); speech = score2 <= thr && power >= noise[s];
 * d_score u8 [S][T]; d_noisy_dB[s] = mean(power[~speech]) (NaN when empty) (FSMN/Export_FSMN_VAD.py:87-100). */
int vadx_fsmn_gate(const float* d_p_sil, const float* d_power_dB, const float* d_noise_avg,
                   float one_minus_speech_threshold, float speech_2_noise_ratio, int64_t n_streams, int n_frames,
                   uint8_t* d_score, float* d_noisy_dB, void* stream);

/* a13 -- look-ahead hysteresis of FSMN (mode 0: uint8 flags) and DFSMN (mode 1: fp32 probabilities), one
 * stream per lane, all stream state on the device: d_silence_state[s] (1 = silence), d_n_saved[s],
 * d_saved [S][ld_saved] (1 = silence, appended), and, when d_noise_avg/d_noisy_dB are given, the
 * running background level noise = 0.5*(noise + noisy + snr) if noisy > 0
 * (FSMN/Inference_FSMN_VAD_ONNX.py:188-234; DFSMN/near_and_far_end_audio/Inference_DFSMN_VAD_ONNX.py:231-273).
 * Every call appends n_frames - look_backward decisions; is_final also appends the tail frames. */
int vadx_lookahead_hysteresis(const void* d_in, int mode, int64_t ld_in, int64_t n_streams, int n_frames,
                              int look_backward, double speaking_score, double silence_score, int is_final,
                              uint8_t* d_silence_state, int32_t* d_n_saved, uint8_t* d_saved, int64_t ld_saved,
                              float* d_noise_avg, const float* d_noisy_dB, float snr_threshold, void* stream);

/* a9 + a13 for ALL windows of a recording in one launch (whole-file mode, see vadx_forward kind "fsmn" with the scalar
 * input.n_windows): d_p_sil / d_power_dB [S][W][T] from one forward over every window; per stream the windows are walked in
 * order -- gate of window w against the running background level, non-speech mean, look-ahead machine on the window's
 * flags (the last window flushes the tail), level update (FSMN/Inference_FSMN_VAD_ONNX.py:177-234).  Optional traces:
 * d_score u8 [S][W][T], d_noisy_dB / d_noise_in fp32 [S][W].  State arguments as vadx_lookahead_hysteresis. */
int vadx_fsmn_gate_hysteresis_windows(const float* d_p_sil, const float* d_power_dB, int64_t n_streams, int n_windows,
                                      int n_frames, float one_minus_speech_threshold, float speech_2_noise_ratio,
                                      int look_backward, double speaking_score, double silence_score, uint8_t* d_score,
                                      float* d_noisy_dB, float* d_noise_in, uint8_t* d_silence_state, int32_t* d_n_saved,
                                      uint8_t* d_saved, int64_t ld_saved, float* d_noise_avg, float snr_threshold,
                                      void* stream);

/* whole-file mode helper: d_out [S*W][n_samples] = the W windows of every recording, window w of stream s starting at
 * d_in + s*stream_stride + w*window_stride */
int vadx_gather_windows_i16(const int16_t* d_in, int64_t stream_stride, int64_t n_streams, int n_windows, int64_t window_stride,
                            int64_t n_samples, int16_t* d_out, void* stream);

/* a14 -- runs of non-silence flags -> (start, end-exclusive) frame pairs per stream
 * (vad_to_timestamps, FSMN/Inference_FSMN_VAD_ONNX.py:124-141). */
int vadx_runs_to_segments(const uint8_t* d_silence_flags, int64_t ld, const int32_t* d_n_flags, int64_t n_streams,
                          int32_t* d_seg_count, int32_t* d_segments, int max_segments, void* stream);

/* a11 helpers (Silero): right reflect padding of each row (out[s][n_in + j] = x[s][n_in - 2 - j]), in-place
 * square root (power -> magnitude) and the LSTM cell update (PyTorch gate order i,f,g,o;
 * c' = sig(f)*c + sig(i)*tanh(g), h' = sig(o)*tanh(c'); d_h_relu optional = relu(h')). */
/* (re, im)-interleaved DFT rows -> magnitudes [n_windows][n_frames][n_bins]; the input has rows_per_window rows per window
 * of which the first n_frames are frames (the framed DFT as a dense layer over hop-strided rows, csrc/model_silero.cu). */
int vadx_stft_mag_compact_f32(const float* d_y, int64_t ldy, int64_t n_windows, int rows_per_window, int n_frames,
                              int n_bins, float* d_mag, void* stream);
int vadx_reflect_window_f32(const float* d_x, int64_t in_stride, int64_t n_streams, int n_in, int pad, float* d_out,
                            void* stream);
/* all W windows of a multi-window call at once: d_out [W][S][n_in + pad], window w of stream s starts at
 * d_x + s*in_stride + w*window_step */
int vadx_reflect_windows_f32(const float* d_x, int64_t in_stride, int64_t n_streams, int n_windows, int64_t window_step,
                             int n_in, int pad, float* d_out, void* stream);
int vadx_sqrt_inplace_f32(float* d_p, int64_t n, void* stream);
/* y[i] = a * x[i] + b (MarbleNet's fused tail: P(silence) = 1 - P(active) of the two-class softmax head) */
int vadx_affine_f32(const float* d_x, float a, float b, float* d_y, int64_t n, void* stream);
int vadx_lstm_cell_f32(const float* d_gates, const float* d_c_in, float* d_h_out, float* d_c_out, float* d_h_relu,
                       int64_t n_streams, int hidden, void* stream);

/* a11 -- the LSTM recurrence of a multi-window call in ONE launch (persistent CTAs own 28 streams each and walk the
 * windows with h, c in shared memory): d_gates_in [W][S][4H] = the input half of the gates incl. both biases, d_wt_hh the
 * TRANSPOSED recurrent weight [H][ldw], state [2][S][H] (h ; c) in -> out (distinct), d_head_w [H] + head_bias the 1-output
 * head on relu(h) -> d_probs [W][S].  PyTorch gate order (i, f, g, o); hidden = 128; exact fp32. */
int vadx_silero_lstm_windows_f32(const float* d_gates_in, const float* d_wt_hh, int ldw, const float* d_state_in,
                                 float* d_state_out, const float* d_head_w, float head_bias, float* d_probs,
                                 int64_t n_streams, int n_windows, int hidden, void* stream);

/* a16 -- the trigger / release / max-speech machine of Silero's get_speech_timestamps
 * (Silero/modeling_modified/utils_vad.py:374-462), one stream per lane: d_probs [S][ld] (one value per
 * window), d_n_windows[s], d_n_samples[s] (audio length) -> raw (start, end) SAMPLE pairs in
 * d_segments [S][max_segments][2] (int64) and d_seg_count[s].  Thresholds are doubles because the reference
 * compares Python floats; speech padding and rounding (:464-482) are per-segment host work. */
int vadx_silero_timestamps(const float* d_probs, int64_t ld, const int32_t* d_n_windows, const int64_t* d_n_samples,
                           int64_t n_streams, double threshold, double neg_threshold, double min_speech_samples,
                           double max_speech_samples, double min_silence_samples,
                           double min_silence_samples_at_max_speech, int window, int use_max_poss_sil,
                           int32_t* d_seg_count, int64_t* d_segments, int max_segments, void* stream);

/* a10 -- building blocks of the SDAEC / ICCRN echo estimator (DFSMN/near_and_far_end_audio/
 * Export_DFSMN_VAD.py:65-354) on [stream][frame][bin][channel] fp32 activations.
 *  vadx_stft_complex_f32: like vadx_stft_power_f32 but keeps (re, im) interleaved: out[(s*T+t)*ld_out + 2f / 2f+1].
 *  vadx_permute4_f32: out dims = (n[p0], n[p1], n[p2], n[p3]); out[i0][i1][i2][i3] = in[j], j[p_k] = i_k.
 *  vadx_layernorm_f32: per row of row_len contiguous values: (x - mean) / (std_unbiased + eps) * w[d] + b[d]
 *      (LayerNorm over (C, F), :163-167).
 *  vadx_lstm_seq_f32: n_seq independent LSTM sequences (PyTorch gate order, zero initial state); sequence
 *      q = o*n_inner + i starts at d_x + o*x_outer + i*x_inner, steps are x_step floats apart (same for d_y,
 *      which receives the hidden state of every step); reverse = 1 walks the sequence backwards.
 *  vadx_ew2_f32: op 0 a+b, 1 a*b, 2 a - scalar*b, 3 copy a, 4 gate (out = a*b, out2 = b - a*b), row-strided.
 *  vadx_ceps_cmul_f32: complex product of [rows][re(C) | im(C)] tensors (CepsUnit, :145-146).
 *  vadx_im2col_f3_f32: out[(blk,f)][j*C + c] = x[(blk, f+j-1)][c] (zero padded) for the (3,1) frequency conv.
 *  vadx_alpha_x4_f32: AlphaPredictor (:326-336) + assembly of the 4-channel ICCRN input.
 *  vadx_istft_ola_f32: overlap-add + crop + window-sum normalisation of NET.istft (:226-230). */
int vadx_stft_complex_f32(const float* d_sig, int64_t sig_stride, int64_t n_streams, int n_frames, int hop, int n_taps,
                          const float* d_basis, int ld_basis, int n_bins, float* d_out, int64_t ld_out, void* stream);
int vadx_permute4_f32(const float* d_in, float* d_out, int64_t n0, int64_t n1, int64_t n2, int64_t n3, int p0, int p1,
                      int p2, int p3, void* stream);
int vadx_layernorm_f32(const float* d_x, int64_t n_rows, int row_len, const float* d_w, const float* d_b, float eps,
                       float* d_out, void* stream);
/* The same building blocks with the layout changes of the cepstral unit folded in (no permute4 launches):
 *  vadx_layernorm_perm_f32: LayerNorm of rows that are [n1][n2][n3] blocks, written in the axis order (q0, q1, q2); the affine
 *      tables are indexed in input order, or in output order with w_out_order = 1.  Output rows are out_stride floats apart
 *      (0 = dense) with `pad` zeros written before and after each row: the zero padding of a following 3-tap frequency conv
 *      that runs as a dense layer over OVERLAPPING rows (vadx_linear_tc_f32 with ldx < n_in) instead of an im2col copy.
 *  vadx_ceps_cmul_t_f32: q [B][cb][re(C) | im(C)] x spec [B][C][re(cb) | im(cb)] -> product in spec's layout.
 *  vadx_add_transposed_f32: out[b][f][c] = a[b][f][c] + t[b][c][f]; a's blocks are a_block_stride floats apart (0 = dense). */
int vadx_layernorm_perm_f32(const float* d_x, int64_t n_rows, int n1, int n2, int n3, int q0, int q1, int q2, const float* d_w,
                            const float* d_b, int w_out_order, float eps, float* d_out, int64_t out_stride, int pad, void* stream);
int vadx_ceps_cmul_t_f32(const float* d_q, const float* d_spec, float* d_out, int64_t n_blocks, int n_channels, int n_ceps,
                         void* stream);
int vadx_add_transposed_f32(const float* d_a, int64_t a_block_stride, const float* d_t, float* d_out, int64_t n_blocks, int n_bins,
                            int n_channels, void* stream);
/* The front of a gated conv block in one kernel (CFB, Export_DFSMN_VAD.py:87-93,133-154), one CTA per (stream, frame)
 * block of n_bins bins:  g = sigmoid(W_g LN0(x) + b_g), xi = W_i x + b_i, gx = g*xi, d = xi - gx;
 *   d_col = LN1(gx) as zero-padded rows [n_blocks][n_bins + 2][C]   (input of the frequency conv as a dense layer over
 *           overlapping rows),   d_z = LN2(d) transposed [n_blocks][C][n_bins]   (input of the cepstral DFT layer).
 * d_x [n_blocks][n_bins][n_in]; W_g, W_i [C][n_in] in the reference layout; LayerNorm tables [n_bins][.]; C = 20, n_in 20 | 40. */
int vadx_cfb_front_supported(int n_in, int n_channels, int n_bins);
int vadx_cfb_front_f32(const float* d_x, int64_t n_blocks, int n_bins, int n_in, int n_channels, const float* d_ln0_w,
                       const float* d_ln0_b, const float* d_wg, const float* d_bg, const float* d_wi, const float* d_bi,
                       const float* d_ln1_w, const float* d_ln1_b, const float* d_ln2_w, const float* d_ln2_b, float eps,
                       float* d_col, float* d_z, void* stream);
int vadx_lstm_seq_f32(const float* d_x, int64_t x_outer, int64_t x_inner, int64_t x_step, float* d_y, int64_t y_outer,
                      int64_t y_inner, int64_t y_step, const float* d_w_ih, const float* d_w_hh, const float* d_b_ih,
                      const float* d_b_hh, int64_t n_seq, int n_inner, int seq_len, int n_in, int hidden, int reverse,
                      void* stream);
/* LSTM with the input projection hoisted out of the recurrence: d_gates_in holds x W_ih^T + b_ih + b_hh for every step of
 * every sequence, computed beforehand as one dense layer, with the gate rows PERMUTED to row' = 4*unit + gate (i, f, g, o);
 * d_w_hh_perm is W_hh in the same order, [hidden][4][hidden].  Sequence / step addressing as vadx_lstm_seq_f32 (strides in
 * floats, multiples of 4); d_y receives h of every step.  One thread per sequence, no barrier inside the time loop. */
int vadx_lstm_recurrence_supported(int hidden);
int vadx_lstm_recurrence_f32(const float* d_gates_in, int64_t g_outer, int64_t g_inner, int64_t g_step, float* d_y,
                             int64_t y_outer, int64_t y_inner, int64_t y_step, const float* d_w_hh_perm, int64_t n_seq,
                             int n_inner, int seq_len, int hidden, int reverse, void* stream);
int vadx_ew2_f32(int op, const float* d_a, int64_t lda, const float* d_b, int64_t ldb, float* d_out, int64_t ldo,
                 float* d_out2, int64_t ldo2, int64_t n_rows, int n_cols, float scalar, void* stream);
int vadx_ceps_cmul_f32(const float* d_q, const float* d_p, float* d_out, int64_t n_rows, int n_channels, void* stream);
int vadx_im2col_f3_f32(const float* d_x, float* d_out, int64_t n_blocks, int n_bins, int n_channels, void* stream);
int vadx_alpha_x4_f32(const float* d_near_ri, const float* d_far_ri, int64_t n_streams, int n_frames, int n_bins, int k,
                      float w1_far, float w1_mix, float b1, const float* d_w2, float b2, float* d_x4, float* d_alpha,
                      void* stream);
/* near-end-only graph (DFSMN/only_near_end_audio/Export_DFSMN_VAD.py:319-335): as vadx_alpha_x4_f32 with the far
 * end's power window and spectrum given as the graph's constants d_pow_far [F][t_max][k], d_far_comp [2][F][t_max] */
int vadx_alpha_x4_const_f32(const float* d_near_ri, const float* d_pow_far, const float* d_far_comp, int t_max,
                            int64_t n_streams, int n_frames, int n_bins, int k, float w1_far, float w1_mix, float b1,
                            const float* d_w2, float b2, float* d_x4, float* d_alpha, void* stream);
int vadx_istft_ola_f32(const float* d_frames, int64_t ld, int64_t n_streams, int n_frames, int n_fft, int hop,
                       const float* d_wsum_inv, int n_out, float* d_y, int64_t ldy, void* stream);

/* next-3 -- real-audio ingest on device: interleaved int16 PCM (1 or 2 channels, any rate) -> mono int16 at
 * out_rate, bit-identical to the reference loader's pydub chain
 * `AudioSegment.from_file(p).set_channels(1).set_frame_rate(sr)` (FSMN/Inference_FSMN_VAD_ONNX.py:68), i.e.
 * audioop.tomono(0.5, 0.5) = floor((l + r) / 2) followed by audioop.ratecv with default weights, whose
 * sequential recurrence has the closed form  out[k] = floor((prev*d + cur*(b - d)) / b),
 * n = ceil(k*a/b) + 1, cur = x[n-1], prev = x[n-2] (0 before the start), d = (n-1)*b - k*a,
 * a/b = in_rate/out_rate in lowest terms.  d_pcm [S][in_stride] int16 (n_channels interleaved),
 * d_n_in [S] frames per stream (NULL = n_frames_in); d_out [S][out_stride], entries past a stream's
 * own output count are zero; d_n_out [S] (optional) receives the counts.
 * vadx_ingest_out_frames: output frames for n_in input frames (what ratecv returns). */
int64_t vadx_ingest_out_frames(int64_t n_frames_in, int in_rate, int out_rate);
int vadx_ingest_pcm16(const int16_t* d_pcm, int64_t in_stride, const int64_t* d_n_in, int64_t n_streams,
                      int64_t n_frames_in, int n_channels, int in_rate, int out_rate, int16_t* d_out,
                      int64_t out_stride, int64_t* d_n_out, void* stream);

/* next-3 -- the in-graph resampler of the FireRed / MarbleNet wrappers for IN_SAMPLE_RATE != 16000
 * (FireRedVAD/Export_FireRedVAD.py:431-449): F.interpolate(x, scale_factor, mode='linear', align_corners=False),
 * out[i] = (1-w)*x[i0] + w*x[min(i0+1, n_in-1)], src = max(0, (float)(1/scale)*(i+0.5) - 0.5), i0 = floor(src),
 * w = src - i0, n_out = floor(n_in * scale).  d_in [S][in_stride] -> d_out [S][out_stride], written at column
 * out_offset (room for the STFT's centre pad); vadx_resample_out_len returns n_out. */
int64_t vadx_resample_out_len(int64_t n_in, double scale);
int vadx_resample_linear_f32(const float* d_in, int64_t in_stride, int64_t n_in, int64_t n_streams, double scale,
                             float* d_out, int64_t out_stride, int64_t out_offset, void* stream);

/* a15 -- FireRed / MarbleNet VadPostprocessor on device, one stream per lane, sequential in time so
 * that the float32 running sum rounds exactly like np.cumsum
 * (FireRedVAD/Inference_FireRed_ONNX.py:181-304).  d_probs [S][ld_probs]; d_n_frames [S] valid
 * frames per stream (NULL = all n_frames).  Outputs: d_decisions [S][n_frames] int8 (optional),
 * d_seg_count [S], d_segments [S][max_segments][2] int32 frame indices (start, end-exclusive). */
typedef struct {
  int32_t smooth_window;
  float threshold;
  int32_t min_speech_frame;
  int32_t max_speech_frame;
  int32_t min_silence_frame;
  int32_t merge_silence_frame;
  int32_t extend_speech_frame;
} vadx_post_cfg;
int vadx_postprocess_frames(const float* d_probs, int64_t ld_probs, const int32_t* d_n_frames,
                            int64_t n_streams, int n_frames, const vadx_post_cfg* cfg, int8_t* d_decisions,
                            int32_t* d_seg_count, int32_t* d_segments, int max_segments, void* stream);

/* next-1 -- FireRed StreamVadPostprocessor on device, one stream per lane, state carried between calls
 * (FireRedVAD/Inference_FireRed_ONNX.py:307-490: ring-buffer mean in float32, 1-based frame counter,
 * pad_start, max-speech re-arm).  d_state is [S][vadx_stream_post_state_words(smooth_window)] int32;
 * all-zero bytes are the reset state (the reference's reset(), :335-346).  Each call consumes
 * d_n_frames[s] (NULL = n_frames) frames of d_probs [S][ld_probs] and APPENDS the segments closed in
 * this call to d_segments [S][max_segments][2] at index d_seg_count[s] (the caller zeroes the counts
 * when a stream starts); a count may exceed max_segments, the overflow is not stored.  Segments are
 * 0-based frame pairs (start, end), both as the reference emits them before the multiplication by
 * 1/frames-per-second.  d_open [S][2] receives the segment still open after the call, as
 * (start, last frame seen), or (-1, -1): the reference reports it at the end of every process_batch
 * call (:470-474). */
typedef struct {
  int32_t smooth_window;
  float threshold;
  int32_t pad_start_frame;
  int32_t min_speech_frame;
  int32_t max_speech_frame;
  int32_t min_silence_frame;
} vadx_stream_post_cfg;
int vadx_stream_post_state_words(int smooth_window);
int vadx_stream_postprocess(const float* d_probs, int64_t ld_probs, const int32_t* d_n_frames, int64_t n_streams,
                            int n_frames, const vadx_stream_post_cfg* cfg, int32_t* d_state, int32_t* d_seg_count,
                            int32_t* d_segments, int max_segments, int32_t* d_open, void* stream);

/* Stream-VAD slot server: n_slots independent streams, one tick per chunk of chunk_samples.  Per tick and slot s the
 * caller gives d_n_samples[s] in [0, chunk_samples] and d_last[s] (uint8, != 0 = the stream's last chunk):
 *   n > 0, last 0: feed a full chunk (n == chunk_samples; anything shorter is rejected);
 *   n > 0, last 1: feed the stream's last chunk, which may be short, then finalize the slot;
 *   n = 0, last 0: hold -- caches and segmenter state unchanged, no frames consumed;
 *   n = 0, last 1: finalize now without new audio.
 * Frames per chunk follow the reference loop (Inference_FireRed_ONNX.py:786-811): 1 + (n - frame_len) / frame_hop, one
 * frame for a chunk shorter than frame_len, and the stream's total cut at the frames of its samples so far (a 64-bit
 * sample counter in the state words 10..11).  Finalize emits a still-open segment's end at the last frame consumed and
 * zeroes the slot's state and caches_out rows, so the next stream in the slot starts fresh.
 *
 * vadx_stream_serve_zero_tail runs BEFORE the model forward on the tick's chunk [n_slots][ld_chunk] int16: it zeroes
 * samples [n, frame_len) of every chunk with 0 < n < frame_len (the reference zero-pads such a chunk to one frame);
 * every other sample past n only reaches frames the server discards.
 *
 * vadx_stream_serve_step runs AFTER the forward on its probabilities d_probs [n_slots][ld_probs] (n_frames columns):
 *   - runs the vadx_stream_postprocess segmenter (same state layout) over the tick's frames of every slot, writing the
 *     frames consumed to d_frames [n_slots];
 *   - applies the slot lifecycle to the caches (layout [n_cache_blocks][n_slots][cache_row] fp32, distinct buffers): a
 *     held slot's caches_out rows <- its caches_in rows, a finalized slot's caches_out rows <- 0.  Both may be NULL
 *     (segmenter and lifecycle without a model);
 *   - writes the tick's events to d_events [n][3] int32 (slot, kind, frame), ordered by slot, then emission order, and
 *     the header d_header[2] = {n, error bits}.  kind: VADX_SERVE_START (the segmenter confirmed a segment starting at
 *     `frame`), VADX_SERVE_END (closed by min-silence or max-speech), VADX_SERVE_END_OF_STREAM (open at finalize);
 *     frames are 0-based from the stream's first frame.  d_events must hold n_slots * (2 * n_frames + 1) triples.
 *     A slot whose control words break the rules above is left unchanged and sets VADX_SERVE_ERR_* in the header.
 *   - h_events / h_header (optional, together): page-locked host memory of the same sizes that receives the same
 *     events and header from the device, so the bytes sent to the host grow with the events, not with n_slots.
 * d_scratch = NULL: only writes the scratch size to *scratch_needed and returns. */
#define VADX_SERVE_START 0
#define VADX_SERVE_END 1
#define VADX_SERVE_END_OF_STREAM 2
#define VADX_SERVE_ERR_RANGE 1 /* n_samples outside [0, chunk_samples] */
#define VADX_SERVE_ERR_SHORT 2 /* a short chunk that is not the stream's last */
int vadx_stream_serve_zero_tail(int16_t* d_chunk, int64_t ld_chunk, const int32_t* d_n_samples, int64_t n_slots,
                                int chunk_samples, int frame_len, void* stream);
int vadx_stream_serve_step(const float* d_probs, int64_t ld_probs, int n_frames, const int32_t* d_n_samples,
                           const uint8_t* d_last, int64_t n_slots, int chunk_samples, int frame_len, int frame_hop,
                           const vadx_stream_post_cfg* cfg, int32_t* d_state, const float* d_caches_in,
                           float* d_caches_out, int n_cache_blocks, int64_t cache_row, int32_t* d_frames,
                           int32_t* d_events, int32_t* d_header, int32_t* h_events, int32_t* h_header, void* d_scratch,
                           size_t scratch_bytes, size_t* scratch_needed, void* stream);

/* Silero slot server: n_slots independent streams, one tick per W = windows_per_tick windows of 512 samples (16 kHz).
 * Per tick and slot s the caller gives d_n_samples[s] in [0, W*512] and d_last[s] with the four actions of the
 * Stream-VAD slot server above (feed a full chunk, feed a possibly short last chunk and finalize, hold, finalize
 * without audio) and the same VADX_SERVE_ERR_* rules.  A slot consumes ceil(n / 512) windows; a short last window is
 * zero-padded to 512 and counts as 512 samples, as the reference VADIterator counts a padded window.
 *
 * vadx_silero_serve_load runs BEFORE the model forward: it converts the int16 chunk d_chunk [n_slots][W*512]
 * (contiguous) into columns [64, 64 + W*512) of the model input d_x [n_slots][64 + W*512] fp32 (both 16-byte
 * aligned: the kernels move 16-byte vectors; a misaligned pointer is rejected), scaled by the
 * reference's 0.000030517578 (exactly 2^-15 in float32) and zero from n on.  Columns 0..63 hold the slot's carried
 * context and are not touched.  The forward reads d_x with input.row_stride = 64 + W*512 and input.n_windows = W.
 *
 * vadx_silero_serve_step runs AFTER the forward on its probabilities d_probs [W][ld_probs] (n_slots columns):
 *   - runs the reference VADIterator (Silero/modeling_modified/utils_vad.py:494-585) over the slot's windows, comparing
 *     each probability in double with `threshold` and `threshold - 0.15`, and a silence of (w - w_t) * 512 samples with
 *     min_silence_samples; its state is d_state [n_slots][3] int32 (all zero = a fresh stream).  Writes the windows
 *     consumed to d_windows [n_slots];
 *   - rolls the context in d_x (may be NULL; 16-byte aligned): a fed slot's last 64 samples become columns 0..63, a finalized slot's
 *     are zeroed, a held slot's are unchanged;
 *   - applies the slot lifecycle to the LSTM state [2][n_slots][128] fp32 (d_state_in / d_state_out: both or neither,
 *     distinct): a held slot's out rows <- its in rows, a finalized slot's out rows <- 0;
 *   - writes the events to d_events [n][3] int32 (slot, kind, window) and d_header {n, error bits}, ordered by slot,
 *     then emission order, and to the optional pinned host mirror h_events / h_header, as vadx_stream_serve_step does.
 *     Windows count from the stream's first window, so a stream may run 2^31 windows (about 2.2 years).
 *     VADX_SERVE_START: the iterator triggered on window w (its sample: max(0, w*512 - pad));
 *     VADX_SERVE_END: the silence that ended the segment began on window w_t, the iterator's temp_end (its sample:
 *     w_t*512 + pad); VADX_SERVE_END_OF_STREAM: the stream was finalized while triggered, the value is the windows
 *     consumed.  d_events must hold n_slots * (W + 1) triples.
 * d_scratch = NULL: only writes the scratch size to *scratch_needed and returns. */
int vadx_silero_serve_load(const int16_t* d_chunk, const int32_t* d_n_samples, int64_t n_slots, int windows_per_tick,
                           float* d_x, void* stream);
int vadx_silero_serve_step(const float* d_probs, int64_t ld_probs, const int32_t* d_n_samples, const uint8_t* d_last,
                           int64_t n_slots, int windows_per_tick, double threshold, double min_silence_samples,
                           int32_t* d_state, float* d_x, const float* d_state_in, float* d_state_out,
                           int32_t* d_windows, int32_t* d_events, int32_t* d_header, int32_t* h_events,
                           int32_t* h_header, void* d_scratch, size_t scratch_bytes, size_t* scratch_needed,
                           void* stream);

/* FSMN slot server: n_slots independent FSMN-VAD streams, one reference window of chunk_len samples per tick.  Windows
 * follow the reference (FSMN/Inference_FSMN_VAD_ONNX.py:79-99): window k of a stream covers samples
 * [k*stride, k*stride + chunk_len), stride = chunk_len - (look_backward + 1) * 160 (both multiples of 8).  Per tick and slot
 * s the caller gives d_n_samples[s] and d_last[s] with the four actions of the slot servers above (feed a full chunk, feed
 * a possibly short last chunk and finalize, hold, finalize without audio) and the same VADX_SERVE_ERR_* rules, where a
 * full chunk is min(stride, chunk_len - received) until the slot holds chunk_len samples and stride from then on
 * (VADX_SERVE_ERR_RANGE: n outside [0, full]).  The tick that completes a slot's first chunk_len samples runs its first
 * window, every later fed tick one more; a stream that ends earlier gets one window, zero-padded, as does a short last
 * chunk.  Finalize without audio flushes the look-ahead of the latest window (its last look_backward score flags are in
 * the state).  The state is d_state [n_slots][vadx_fsmn_serve_state_words(look_backward)] int32, all zero = a fresh slot.
 *
 * vadx_fsmn_serve_load runs BEFORE the forward: it writes the int16 chunk d_chunk [n_slots][stride] into the slot's row of
 * the window buffer d_window [n_slots][chunk_len] (the forward's input; both 16-byte aligned: the kernel moves 16-byte
 * vectors, a misaligned pointer is rejected): before the first window at the samples received so far, afterwards after
 * shifting the row left by stride; zeros from n on; a held slot's row is not touched.  It also writes each slot's
 * background level (the gate's noise_average_dB input) to d_noise_avg [n_slots].
 *
 * vadx_fsmn_serve_step runs AFTER the forward on its score flags d_score [n_slots][ld_score] (n_frames columns, 0 / 1) and
 * noisy_dB [n_slots]:
 *   - runs the look-ahead hysteresis (lookahead_hysteresis, mode 0) over each window's flags, writes the decisions of the
 *     tick to d_decisions [n_slots], and updates the level as the reference does (if noisy_dB > 0: level =
 *     0.5 * ((level + noisy_dB) + snr_threshold), fp32);
 *   - turns the decisions into the reference's final timestamps, process_timestamps(runs_to_timestamps(...), fusion,
 *     min_duration) (:102-141), in Python doubles, emitting each event as soon as it is certain: VADX_SERVE_START a (time
 *     a*d), VADX_SERVE_END b (the run closed by silence decision b, time b*d + d), VADX_SERVE_END_OF_STREAM n (the
 *     segment was open at finalize after n decisions, time n*d), d = frame_duration.  Decisions count from the stream's
 *     first window as int32, so a stream may run 2^31 decisions (about 248 days at 100 per second);
 *   - applies the slot lifecycle to the caches [n_cache_blocks][n_slots][cache_row] fp32 as vadx_stream_serve_step does
 *     (a slot that ran no window holds them) and writes d_events [n][3] (slot, kind, decision) / d_header and the optional
 *     pinned host mirror.  d_events must hold n_slots * (2 * n_frames + 2) triples.
 * d_scratch = NULL: only writes the scratch size to *scratch_needed and returns. */
typedef struct {
  double speaking_score;
  double silence_score;
  double frame_duration;        /* seconds per decision: 160 / 16000 */
  double fusion_threshold;      /* seconds */
  double min_speech_duration;   /* seconds */
  float snr_threshold;          /* snr_threshold_dB * 0.1 */
  float noise_init;             /* the initial background level */
} vadx_fsmn_serve_cfg;
int vadx_fsmn_serve_state_words(int look_backward);
int vadx_fsmn_serve_load(const int16_t* d_chunk, const int32_t* d_n_samples, const uint8_t* d_last,
                         const int32_t* d_state, int64_t n_slots, int chunk_len, int stride, int look_backward,
                         float noise_init, int16_t* d_window, float* d_noise_avg, void* stream);
int vadx_fsmn_serve_step(const uint8_t* d_score, int64_t ld_score, const float* d_noisy_dB, int n_frames,
                         const int32_t* d_n_samples, const uint8_t* d_last, int64_t n_slots, int chunk_len, int stride,
                         int look_backward, const vadx_fsmn_serve_cfg* cfg, int32_t* d_state, const float* d_caches_in,
                         float* d_caches_out, int n_cache_blocks, int64_t cache_row, int32_t* d_decisions,
                         int32_t* d_events, int32_t* d_header, int32_t* h_events, int32_t* h_header, void* d_scratch,
                         size_t scratch_bytes, size_t* scratch_needed, void* stream);

/* MarbleNet slot server: n_slots independent MarbleNet Frame-VAD streams, one static-axis window of window_samples = L
 * samples per tick (the reference's non-overlapping windows, audio_io.align_non_overlapping), of which the model's first
 * n_frames = F = T' - 1 frames count (signal_len).  Per tick and slot s the caller gives d_n_samples[s] in [0, L] and
 * d_last[s] with the four actions of the slot servers above and the same VADX_SERVE_ERR_* rules (a full chunk is L).
 * A fed tick consumes F frames; a short last chunk is zero-padded to L by vadx_stream_serve_zero_tail (frame_len = L)
 * before the forward.  The model keeps no state across windows, so there are no caches.
 *
 * vadx_marblenet_serve_step runs AFTER the forward on its active-class probabilities d_probs [n_slots][ld_probs]:
 *   - runs the reference's VadPostprocessor (the passes of vadx_postprocess_frames: smoothing, the four-state machine,
 *     the rising-edge extension by the smoothing window, the gap merge, the dilation, the max-speech split at the first
 *     arg-min of the raw probabilities) online, one thread per slot.  A frame's decision before the split is final
 *     D = D2 + D3 + D4 + D5 frames after it, D2 = max(min_speech, 1) (0 when min_speech <= 0 and min_silence <= 0),
 *     D3 = ws (when ws > 1), D4 = max(merge - 1, 0), D5 = max(extend, 0): at most max(min_speech, 1) + ws + merge +
 *     extend, 15 frames at MarbleNet's defaults.  Finalize flushes what is still in flight as the whole-track passes
 *     treat a track's end.  The state is d_state [n_slots][vadx_marblenet_serve_state_words(cfg)] int32, all zero = a
 *     fresh slot; D is at most 65536.  Writes the frames consumed to d_frames [n_slots];
 *   - writes the events to d_events [n][3] int32 (slot, kind, value) / d_header {n, error bits} and the optional pinned
 *     host mirror, as vadx_stream_serve_step does: VADX_SERVE_START a (a final segment starts at frame a, time
 *     float32(a) * frame_shift), VADX_SERVE_END b (it ends before frame b, max-speech cuts included),
 *     VADX_SERVE_END_OF_STREAM (the last segment was open at finalize): the value is the bit pattern of the reference's
 *     float32 end, n * frame_shift after n frames, replaced by samples / 16000 when that is smaller (compared in double,
 *     then rounded to float32; samples is a 64-bit count in the state).  Frames count from the stream's first window as
 *     int32, so a stream may run 2^31 frames.  A tick stages at most 2 (F + D) + 2 events per slot; d_events must hold
 *     n_slots * (2 * (n_frames + D) + 2) triples.
 * d_scratch = NULL: only writes the scratch size to *scratch_needed and returns. */
int vadx_marblenet_serve_state_words(const vadx_post_cfg* cfg);
int vadx_marblenet_serve_step(const float* d_probs, int64_t ld_probs, int n_frames, const int32_t* d_n_samples,
                              const uint8_t* d_last, int64_t n_slots, int window_samples, const vadx_post_cfg* cfg,
                              float frame_shift, int32_t* d_state, int32_t* d_frames, int32_t* d_events,
                              int32_t* d_header, int32_t* h_events, int32_t* h_header, void* d_scratch,
                              size_t scratch_bytes, size_t* scratch_needed, void* stream);

/* ------------------------------------------------------------------------------------------
 * Model-level API: the replacement for InferenceSession(...).run(...)
 * ------------------------------------------------------------------------------------------ */
typedef struct vadx_model vadx_model;

/* kind: "firered" | "fsmn" | "marblenet" | "silero".  `hparams` is a flat int32 array, meaning per kind:
 *   firered: {idim, R, M, H, P, N1, S1, N2, S2, odim, n_fft, win_length, hop, n_mels}
 *            (DetectModel args, FireRedVAD/Export_FireRedVAD.py:310-316, frontend :38-49)
 *   fsmn:    {input_dim, input_affine_dim, fsmn_layers, linear_dim, proj_dim, lorder, rorder, lstride, rstride,
 *             output_affine_dim, output_dim, n_fft, win_length, hop, n_mels, lfr_m, lfr_n}
 *            (FunASR FSMN encoder, FSMN/modeling_modified/encoder.py:159-206; frontend FSMN/Export_FSMN_VAD.py:24-34)
 *   marblenet: {feat_in, n_blocks, [filters, repeat, kernel, stride, dilation, residual] x n_blocks,
 *             num_classes, n_fft, win_length, hop, n_mels}; tensors are the BN-FOLDED layers
 *             "b{i}.r{j}.dw" [C][k], "b{i}.r{j}.pw" [out][in], "b{i}.r{j}.pw_bias", "b{i}.res", "b{i}.res_bias",
 *             "decoder.weight", "decoder.bias" (folding: NVIDIA_Frame_VAD_Multilingual_MarbleNet/
 *             Export_NVIDIA_MarbleNet_VAD.py:58-151)
 *   silero:  {window, context, reflect_pad, n_fft, hop, hidden, n_enc_layers, [out, in] x n_enc_layers}; tensors
 *             "frontend.basis", "enc.{i}.weight/bias" (dense form of the k=3 conv stack), "rnn.weight_ih",
 *             "rnn.weight_hh", "rnn.bias" (= bias_ih + bias_hh), "head.weight", "head.bias" */
int vadx_create(const char* kind, const int32_t* hparams, int n_hparams, vadx_model** out);
void vadx_destroy(vadx_model* m);

/* Upload a named constant (weights keep the reference state_dict names, e.g.
 * "dfsmn.fc1.0.weight"; frontend tables are "frontend.basis", "frontend.mel_start",
 * "frontend.mel_len", "frontend.mel_w").  h_data is a HOST pointer; the library copies it into
 * device memory it owns (this is the only place it allocates). dims[] are the logical sizes. */
int vadx_set_tensor(vadx_model* m, const char* name, const void* h_data, int dtype, const int64_t* dims,
                    int n_dims);
int vadx_set_scalar(vadx_model* m, const char* name, double value);

/* bytes of caller-provided device workspace vadx_forward needs for (n_streams, n_samples) */
int vadx_workspace_bytes(const vadx_model* m, int64_t n_streams, int64_t n_samples, size_t* out_bytes);
/* frames per stream the model emits for n_samples */
int vadx_output_frames(const vadx_model* m, int64_t n_samples, int32_t* out_frames);

/* One pass of the model over S independent chunks.
 *   firered: inputs[0] = d_audio int16 [S][n_samples]; outputs[0] = d_probs fp32 [S][odim][T]
 *            (the reference's (1, odim, 98) with the leading 1 generalised to S,
 *            FireRedVAD/Export_FireRedVAD.py:794-807). state = NULL for the static graphs;
 *            Stream-VAD twin (N2 = 0): state = {caches_in, caches_out}, each fp32
 *            [R][S][P][(N1-1)*S1], distinct buffers (the reference's (R,1,P,Lb),
 *            FireRedVAD/Export_FireRedVAD.py:863-876, Inference_FireRed_ONNX.py:758-803).
 *            Scalar "frontend.in_sample_rate" (default 16000) selects the wrapper's in-graph linear
 *            resampler (Export_FireRedVAD.py:389-393,431-449); T then follows the resampled length.
 *   fsmn:    inputs  = {audio int16 [S][L], noise_average_dB fp32 [S]}
 *            outputs = {score uint8 [S][T], noisy_dB fp32 [S], P(silence) fp32 [S][T] or NULL,
 *                       power_dB fp32 [S][T] or NULL}
 *            state   = {cache_0..3 in, cache_0..3 out}, each fp32 [S][128][19], distinct buffers
 *            (FSMN/Export_FSMN_VAD.py:122-134); thresholds are scalars set with vadx_set_scalar.
 *   marblenet: inputs = {audio int16 [S][L]}; outputs = {score_silence fp32 [S][T'], score_active fp32 [S][T']}
 *            with T' = vadx_output_frames(L); the reference's signal_len output is T' - 1
 *            (NVIDIA_Frame_VAD_Multilingual_MarbleNet/Export_NVIDIA_MarbleNet_VAD.py:444-457).
 *   silero:  inputs = {x fp32 [S][576] = 64-sample context + 512-sample window}; outputs = {out fp32 [S][1]};
 *            state = {state in fp32 [2][S][128], state out}; n_samples = 576
 *            (the 'input'/'state' -> 'output'/'stateN' contract of Silero/modeling_modified/utils_vad.py:114-123).
 *            Scalars: "input.row_stride" (default 576: rows may be strided views of one long signal) and
 *            "input.n_windows" = W (default 1): one call covers W consecutive 512-sample windows of every stream,
 *            outputs[0] is then fp32 [W][S][1] and the state spans all W windows; everything that does not
 *            depend on the LSTM state runs once over S*W rows, the recurrence runs per window. */
int vadx_forward(vadx_model* m, const void* const* d_inputs, void* const* d_outputs, void* const* d_state,
                 int64_t n_streams, int64_t n_samples, void* d_workspace, size_t workspace_bytes,
                 void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VADX_H_ */
