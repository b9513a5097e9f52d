// fsmn_extra.cu -- the FunASR-FSMN specific stages: LFR + CMVN (a4), softmax class-0 head (a8),
// frame-energy gate (a9), look-ahead hysteresis with on-device stream state (a13) and run-length
// extraction (a14).
#include "hysteresis.cuh"

namespace vadx {

// a4: out[s][t][j*n_mels + m] = (mel[s][clamp(t*lfr_n + j - half, 0, T-1)][m] + mean) * var
__global__ void __launch_bounds__(256) lfr_cmvn_kernel(const float* __restrict__ mel, int64_t ld_mel,
                                                       const float* __restrict__ mean, const float* __restrict__ var,
                                                       float* __restrict__ out, int64_t ld_out, int64_t n_streams,
                                                       int T, int n_mels, int lfr_m, int lfr_n) {
  const int D = n_mels * lfr_m, half = (lfr_m - 1) / 2;
  const int64_t total = n_streams * T * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int d = (int)(i % D);
    int64_t st = i / D;
    int t = (int)(st % T);
    int64_t s = st / T;
    int j = d / n_mels, m = d - j * n_mels;
    int src = t * lfr_n + j - half;
    src = src < 0 ? 0 : (src > T - 1 ? T - 1 : src);
    out[st * ld_out + d] = (mel[(s * T + src) * ld_mel + m] + mean[d]) * var[d];
  }
}

// the same with float4 rows and 32-bit index arithmetic (the scalar kernel above does three 64-bit divisions per element and
// ran at 0.17 of the HBM copy rate): one CTA per output row, thread = one float4 of the lfr_m * n_mels wide row
__global__ void __launch_bounds__(128) lfr_cmvn_v4_kernel(const float* __restrict__ mel, int64_t ld_mel,
                                                          const float* __restrict__ mean, const float* __restrict__ var,
                                                          float* __restrict__ out, int64_t ld_out, int64_t n_rows, int T,
                                                          int n_mels4, int lfr_m, int lfr_n) {
  const int half = (lfr_m - 1) / 2;
  const int Q = n_mels4 * lfr_m;
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    const int t = (int)(row % T);
    const int64_t s_base = row - t;
    float4* o = reinterpret_cast<float4*>(out + row * ld_out);
    for (int q = threadIdx.x; q < Q; q += blockDim.x) {
      const int j = q / n_mels4, m4 = q - j * n_mels4;
      int src = t * lfr_n + j - half;
      src = src < 0 ? 0 : (src > T - 1 ? T - 1 : src);
      const float4 v = __ldg(reinterpret_cast<const float4*>(mel + (s_base + src) * ld_mel) + m4);
      const float4 mu = __ldg(reinterpret_cast<const float4*>(mean) + q), sc = __ldg(reinterpret_cast<const float4*>(var) + q);
      o[q] = make_float4((v.x + mu.x) * sc.x, (v.y + mu.y) * sc.y, (v.z + mu.z) * sc.z, (v.w + mu.w) * sc.w);
    }
  }
}

// softmax over n classes, keep class 0: one warp per row
__global__ void __launch_bounds__(256) softmax_class0_kernel(const float* __restrict__ logits, int64_t ld,
                                                             int64_t n_rows, int n, float* __restrict__ p0) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp; row < n_rows; row += n_warps) {
    const float* x = logits + row * ld;
    float mx = -INFINITY;
    for (int k = lane; k < n; k += 32) mx = fmaxf(mx, x[k]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    float sum = 0.f;
    for (int k = lane; k < n; k += 32) sum += expf(x[k] - mx);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
    if (lane == 0) p0[row] = expf(x[0] - mx) / sum;
  }
}

// a9: power_dB[s][t] = log10(sum_{n<win} (y[s][t*hop+n]*scale)^2 + eps) for t < n_energy, then the
// last value replicated up to T.  One warp per (stream, frame).
__global__ void __launch_bounds__(256) frame_energy_kernel(const float* __restrict__ sig, int64_t sig_stride,
                                                           int64_t offset, int64_t n_streams, int win, int hop,
                                                           int n_energy, int T, float scale, float eps,
                                                           float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < n_streams * T; i += n_warps) {
    const int64_t s = i / T;
    int t = (int)(i - s * T);
    if (t >= n_energy) t = n_energy - 1;
    const float* y = sig + s * sig_stride + offset + (int64_t)t * hop;
    float acc = 0.f;
    for (int n = lane; n < win; n += 32) {
      float v = y[n] * scale;
      acc = fmaf(v, v, acc);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) out[i] = log10f(acc + eps);
  }
}

// a9: gate.  One block per stream.
__global__ void __launch_bounds__(128) fsmn_gate_kernel(const float* __restrict__ p_sil, const float* __restrict__ power,
                                                        const float* __restrict__ noise_avg, float one_minus_thr,
                                                        float ratio, int T, uint8_t* __restrict__ score,
                                                        float* __restrict__ noisy_dB) {
  const int64_t s = blockIdx.x;
  __shared__ float s_sum[128];
  __shared__ int s_cnt[128];
  float sum = 0.f;
  int cnt = 0;
  const float noise = noise_avg[s];
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    float p = p_sil[s * T + t];
    float sc = p + (ratio > 1.0f ? powf(p, ratio) : (ratio < 1.0f ? 1.0f : p));
    float pw = power[s * T + t];
    bool cond = (sc <= one_minus_thr) && (pw >= noise);
    score[s * T + t] = cond ? 1 : 0;
    if (!cond) { sum += pw; ++cnt; }
  }
  s_sum[threadIdx.x] = sum;
  s_cnt[threadIdx.x] = cnt;
  __syncthreads();
  for (int off = 64; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) {
      s_sum[threadIdx.x] += s_sum[threadIdx.x + off];
      s_cnt[threadIdx.x] += s_cnt[threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) noisy_dB[s] = s_sum[0] / (float)s_cnt[0];  // 0/0 = NaN like torch.mean of nothing
}

// a13: look-ahead hysteresis (hysteresis.cuh), one stream per lane, state carried on the device between chunks; the
// decisions are appended to saved[n...].
__global__ void __launch_bounds__(128) lookahead_hysteresis_kernel(const void* __restrict__ in, int mode, int64_t ld_in,
                                                                   int64_t n_streams, int T, int look_backward,
                                                                   double speaking_score, double silence_score,
                                                                   int is_final, uint8_t* __restrict__ silence_state,
                                                                   int32_t* __restrict__ n_saved,
                                                                   uint8_t* __restrict__ saved, int64_t ld_saved,
                                                                   float* __restrict__ noise_avg,
                                                                   const float* __restrict__ noisy_dB, float snr) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_streams) return;
  bool silence = silence_state[s] != 0;
  int n = n_saved[s];
  uint8_t* out = saved + s * ld_saved;
  hysteresis_chunk(static_cast<const uint8_t*>(in) + s * ld_in, static_cast<const float*>(in) + s * ld_in, mode, T, look_backward,
                   speaking_score, silence_score, is_final, silence, [&](bool sil) {
                     if (n < ld_saved) out[n] = sil ? 1 : 0;
                     ++n;
                   });
  silence_state[s] = silence ? 1 : 0;
  n_saved[s] = n;
  if (noise_avg && noisy_dB) {
    float nd = noisy_dB[s];
    if (nd > 0.0f) noise_avg[s] = 0.5f * ((noise_avg[s] + nd) + snr);
  }
}

// a9 + a13 over ALL windows of a recording in one launch (whole-file mode of the FSMN path): the only sequential
// dependence between windows is the running background level -- window w's gate compares against the level windows
// 0..w-1 produced (FSMN/Inference_FSMN_VAD_ONNX.py:177-187,224-225) -- so one block per stream walks the windows: the 128
// threads evaluate the gate of window w and reduce its non-speech mean exactly like fsmn_gate_kernel (same striding, same
// tree: bit-identical noisy_dB), thread 0 then runs the look-ahead machine on that window's flags and updates the level.
__global__ void __launch_bounds__(128) fsmn_gate_hysteresis_windows_kernel(
    const float* __restrict__ p_sil, const float* __restrict__ power, int W, int T, float one_minus_thr, float ratio,
    int look_backward, double speaking_score, double silence_score, uint8_t* __restrict__ score_out, float* __restrict__ noisy_out,
    float* __restrict__ noise_in_out, uint8_t* __restrict__ silence_state, int32_t* __restrict__ n_saved,
    uint8_t* __restrict__ saved, int64_t ld_saved, float* __restrict__ noise_avg, float snr) {
  extern __shared__ uint8_t s_flags[];       // [T]
  __shared__ float s_sum[128];
  __shared__ int s_cnt[128];
  __shared__ float s_noise;
  const int64_t s = blockIdx.x;
  bool silence = silence_state[s] != 0;
  int n = n_saved[s];
  if (threadIdx.x == 0) s_noise = noise_avg[s];
  __syncthreads();
  for (int w = 0; w < W; ++w) {
    const float noise = s_noise;
    const int64_t base = (s * W + w) * (int64_t)T;
    float sum = 0.f;
    int cnt = 0;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      const float p = p_sil[base + t];
      const float sc = p + (ratio > 1.0f ? powf(p, ratio) : (ratio < 1.0f ? 1.0f : p));
      const float pw = power[base + t];
      const bool cond = (sc <= one_minus_thr) && (pw >= noise);
      s_flags[t] = cond ? 1 : 0;
      if (score_out) score_out[base + t] = cond ? 1 : 0;
      if (!cond) { sum += pw; ++cnt; }
    }
    s_sum[threadIdx.x] = sum;
    s_cnt[threadIdx.x] = cnt;
    __syncthreads();
    for (int off = 64; off > 0; off >>= 1) {
      if ((int)threadIdx.x < off) {
        s_sum[threadIdx.x] += s_sum[threadIdx.x + off];
        s_cnt[threadIdx.x] += s_cnt[threadIdx.x + off];
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      const float nd = s_sum[0] / (float)s_cnt[0];      // 0/0 = NaN like torch.mean of nothing
      if (noisy_out) noisy_out[s * W + w] = nd;
      if (noise_in_out) noise_in_out[s * W + w] = noise;
      uint8_t* out = saved + s * ld_saved;
      hysteresis_chunk(s_flags, nullptr, 0, T, look_backward, speaking_score, silence_score, w == W - 1, silence, [&](bool sil) {
        if (n < ld_saved) out[n] = sil ? 1 : 0;
        ++n;
      });
      if (nd > 0.0f) s_noise = 0.5f * ((noise + nd) + snr);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    silence_state[s] = silence ? 1 : 0;
    n_saved[s] = n;
    noise_avg[s] = s_noise;
  }
}

// whole-file mode: the W overlapping windows of every recording as dense rows [S*W][L] (int16), so that the batched
// frontend kernels see ordinary streams
__global__ void __launch_bounds__(256) gather_windows_i16_kernel(const int16_t* __restrict__ in, int64_t stream_stride,
                                                                 int64_t n_streams, int W, int64_t window_stride, int64_t L,
                                                                 int16_t* __restrict__ out) {
  const int64_t total = n_streams * W * L;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / L, k = i - row * L;
    const int64_t s = row / W, w = row - s * W;
    out[i] = in[s * stream_stride + w * window_stride + k];
  }
}

// a14: runs of "not silence" -> (start, end-exclusive) frame pairs
__global__ void __launch_bounds__(128) runs_to_segments_kernel(const uint8_t* __restrict__ silence_flags, int64_t ld,
                                                               const int32_t* __restrict__ n_flags, int64_t n_streams,
                                                               int32_t* __restrict__ seg_count,
                                                               int32_t* __restrict__ segments, int max_segments) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_streams) return;
  const uint8_t* f = silence_flags + s * ld;
  int n = n_flags[s];
  if (n > ld) n = (int)ld;
  int32_t* seg = segments + s * (int64_t)max_segments * 2;
  int count = 0, start = -1;
  for (int i = 0; i <= n; ++i) {
    bool sil = i < n ? f[i] != 0 : true;
    if (sil) {
      if (start >= 0) {
        if (count < max_segments) { seg[2 * count] = start; seg[2 * count + 1] = i; }
        ++count;
        start = -1;
      }
    } else if (start < 0) {
      start = i;
    }
  }
  seg_count[s] = count;
}

}  // namespace vadx

using namespace vadx;

static inline unsigned grid_for(int64_t items, int per_block, int cap = 148 * 16) {
  int64_t b = ceil_div(items, per_block);
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(b, cap));
}

extern "C" int vadx_lfr_cmvn_f32(const float* d_mel, int64_t ld_mel, const float* d_mean, const float* d_var,
                                 float* d_out, int64_t ld_out, int64_t n_streams, int n_frames, int n_mels, int lfr_m,
                                 int lfr_n, void* stream) {
  StageTimer _timer(VADX_STAGE_MEL, (cudaStream_t)stream, "lfr_cmvn_kernel", 4.0 * n_streams * n_frames * n_mels * (1.0 + lfr_m));
  VADX_REQUIRE(d_mel && d_mean && d_var && d_out, "vadx_lfr_cmvn_f32: null pointer");
  VADX_REQUIRE(n_streams >= 0 && n_frames >= 1 && n_mels >= 1 && lfr_m >= 1 && lfr_n == 1 && ld_mel >= n_mels &&
                   ld_out >= n_mels * lfr_m,
               "vadx_lfr_cmvn_f32: bad shape (lfr_n must be 1)");
  if (n_streams == 0) return VADX_OK;
  if ((n_mels & 3) == 0 && (ld_mel & 3) == 0 && (ld_out & 3) == 0 && aligned16(d_mel) && aligned16(d_out) && aligned16(d_mean) &&
      aligned16(d_var)) {
    const int64_t n_rows = n_streams * n_frames;
    lfr_cmvn_v4_kernel<<<(unsigned)std::min<int64_t>(n_rows, 148 * 64), 128, 0, (cudaStream_t)stream>>>(
        d_mel, ld_mel, d_mean, d_var, d_out, ld_out, n_rows, n_frames, n_mels / 4, lfr_m, lfr_n);
    return after_launch("vadx_lfr_cmvn_f32");
  }
  lfr_cmvn_kernel<<<grid_for(n_streams * n_frames * n_mels * lfr_m, 256), 256, 0, (cudaStream_t)stream>>>(
      d_mel, ld_mel, d_mean, d_var, d_out, ld_out, n_streams, n_frames, n_mels, lfr_m, lfr_n);
  return after_launch("vadx_lfr_cmvn_f32");
}

extern "C" int vadx_softmax_class0_f32(const float* d_logits, int64_t ld, int64_t n_rows, int n_classes, float* d_p0,
                                       void* stream) {
  StageTimer _timer(VADX_STAGE_HEAD, (cudaStream_t)stream, "softmax_class0_kernel", 4.0 * n_rows * (n_classes + 1.0));
  VADX_REQUIRE(d_logits && d_p0 && n_rows >= 0 && n_classes >= 1 && ld >= n_classes, "vadx_softmax_class0_f32: bad argument");
  if (n_rows == 0) return VADX_OK;
  softmax_class0_kernel<<<grid_for(n_rows, 8), 256, 0, (cudaStream_t)stream>>>(d_logits, ld, n_rows, n_classes, d_p0);
  return after_launch("vadx_softmax_class0_f32");
}

extern "C" int vadx_frame_energy_log10_f32(const float* d_sig, int64_t sig_stride, int64_t offset, int64_t n_streams,
                                           int win, int hop, int n_energy, int n_frames, float scale, float eps,
                                           float* d_out, void* stream) {
  StageTimer _timer(VADX_STAGE_HEAD, (cudaStream_t)stream, "frame_energy_log10_kernel");
  VADX_REQUIRE(d_sig && d_out, "vadx_frame_energy_log10_f32: null pointer");
  VADX_REQUIRE(n_streams >= 0 && win >= 1 && hop >= 1 && n_energy >= 1 && n_frames >= n_energy && offset >= 0 &&
                   sig_stride >= offset + (int64_t)(n_energy - 1) * hop + win,
               "vadx_frame_energy_log10_f32: bad shape");
  if (n_streams == 0) return VADX_OK;
  frame_energy_kernel<<<grid_for(n_streams * n_frames, 8), 256, 0, (cudaStream_t)stream>>>(
      d_sig, sig_stride, offset, n_streams, win, hop, n_energy, n_frames, scale, eps, d_out);
  return after_launch("vadx_frame_energy_log10_f32");
}

extern "C" int vadx_fsmn_gate(const float* d_p_sil, const float* d_power_dB, const float* d_noise_avg,
                              float one_minus_speech_threshold, float speech_2_noise_ratio, int64_t n_streams,
                              int n_frames, uint8_t* d_score, float* d_noisy_dB, void* stream) {
  StageTimer _timer(VADX_STAGE_HEAD, (cudaStream_t)stream, "fsmn_gate_kernel", 9.0 * n_streams * n_frames);
  VADX_REQUIRE(d_p_sil && d_power_dB && d_noise_avg && d_score && d_noisy_dB, "vadx_fsmn_gate: null pointer");
  VADX_REQUIRE(n_streams >= 0 && n_frames >= 1, "vadx_fsmn_gate: bad shape");
  if (n_streams == 0) return VADX_OK;
  fsmn_gate_kernel<<<(unsigned)n_streams, 128, 0, (cudaStream_t)stream>>>(d_p_sil, d_power_dB, d_noise_avg,
                                                                          one_minus_speech_threshold,
                                                                          speech_2_noise_ratio, n_frames, d_score,
                                                                          d_noisy_dB);
  return after_launch("vadx_fsmn_gate");
}

extern "C" int vadx_lookahead_hysteresis(const void* d_in, int mode, int64_t ld_in, int64_t n_streams, int n_frames,
                                         int look_backward, double speaking_score, double silence_score, int is_final,
                                         uint8_t* d_silence_state, int32_t* d_n_saved, uint8_t* d_saved,
                                         int64_t ld_saved, float* d_noise_avg, const float* d_noisy_dB,
                                         float snr_threshold, void* stream) {
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "lookahead_hysteresis_kernel");
  VADX_REQUIRE(d_in && d_silence_state && d_n_saved && d_saved, "vadx_lookahead_hysteresis: null pointer");
  VADX_REQUIRE((mode == 0 || mode == 1) && n_streams >= 0 && n_frames >= 1 && look_backward >= 0 &&
                   look_backward <= n_frames && ld_in >= n_frames && ld_saved >= 0,
               "vadx_lookahead_hysteresis: bad argument");
  if (n_streams == 0) return VADX_OK;
  lookahead_hysteresis_kernel<<<(unsigned)ceil_div(n_streams, 128), 128, 0, (cudaStream_t)stream>>>(
      d_in, mode, ld_in, n_streams, n_frames, look_backward, speaking_score, silence_score, is_final, d_silence_state,
      d_n_saved, d_saved, ld_saved, d_noise_avg, d_noisy_dB, snr_threshold);
  return after_launch("vadx_lookahead_hysteresis");
}

extern "C" int vadx_fsmn_gate_hysteresis_windows(const float* d_p_sil, const float* d_power_dB, int64_t n_streams, int n_windows,
                                                 int n_frames, float one_minus_speech_threshold, float speech_2_noise_ratio,
                                                 int look_backward, double speaking_score, double silence_score,
                                                 uint8_t* d_score, float* d_noisy_dB, float* d_noise_in,
                                                 uint8_t* d_silence_state, int32_t* d_n_saved, uint8_t* d_saved,
                                                 int64_t ld_saved, float* d_noise_avg, float snr_threshold, void* stream) {
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "fsmn_gate_hysteresis_windows_kernel",
                    9.0 * n_streams * n_windows * n_frames);
  VADX_REQUIRE(d_p_sil && d_power_dB && d_silence_state && d_n_saved && d_saved && d_noise_avg,
               "vadx_fsmn_gate_hysteresis_windows: null pointer");
  VADX_REQUIRE(n_streams >= 0 && n_windows >= 1 && n_frames >= 1 && look_backward >= 0 && look_backward <= n_frames &&
                   ld_saved >= 0 && n_frames <= 48 * 1024,
               "vadx_fsmn_gate_hysteresis_windows: bad argument");
  if (n_streams == 0) return VADX_OK;
  fsmn_gate_hysteresis_windows_kernel<<<(unsigned)n_streams, 128, (size_t)n_frames, (cudaStream_t)stream>>>(
      d_p_sil, d_power_dB, n_windows, n_frames, one_minus_speech_threshold, speech_2_noise_ratio, look_backward, speaking_score,
      silence_score, d_score, d_noisy_dB, d_noise_in, d_silence_state, d_n_saved, d_saved, ld_saved, d_noise_avg, snr_threshold);
  return after_launch("vadx_fsmn_gate_hysteresis_windows");
}

namespace vadx {
// 16-byte copies, one CTA per window row (every offset a multiple of 8 samples)
__global__ void __launch_bounds__(256) gather_windows_v8_kernel(const int16_t* __restrict__ in, int64_t stream_stride, int64_t n_rows,
                                                                int W, int64_t window_stride, int64_t L, int16_t* __restrict__ out) {
  const int n_vec = (int)(L >> 3);
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    const int64_t s = row / W, w = row - s * W;
    const int4* src = reinterpret_cast<const int4*>(in + s * stream_stride + w * window_stride);
    int4* dst = reinterpret_cast<int4*>(out + row * L);
    for (int i = threadIdx.x; i < n_vec; i += blockDim.x) dst[i] = __ldg(src + i);
  }
}
}  // namespace vadx

extern "C" int vadx_gather_windows_i16(const int16_t* d_in, int64_t stream_stride, int64_t n_streams, int n_windows,
                                       int64_t window_stride, int64_t n_samples, int16_t* d_out, void* stream) {
  StageTimer _timer(VADX_STAGE_PREP, (cudaStream_t)stream, "gather_windows_i16_kernel", 4.0 * n_streams * n_windows * n_samples);
  VADX_REQUIRE(d_in && d_out && n_streams >= 0 && n_windows >= 1 && window_stride >= 1 && n_samples >= 1 &&
                   stream_stride >= n_samples + (int64_t)(n_windows - 1) * window_stride,
               "vadx_gather_windows_i16: bad argument");
  if (n_streams == 0) return VADX_OK;
  if (((stream_stride | window_stride | n_samples) & 7) == 0 && aligned16(d_in) && aligned16(d_out)) {
    const int64_t n_rows = n_streams * n_windows;
    gather_windows_v8_kernel<<<(unsigned)std::min<int64_t>(n_rows, 148 * 32), 256, 0, (cudaStream_t)stream>>>(
        d_in, stream_stride, n_rows, n_windows, window_stride, n_samples, d_out);
    return after_launch("vadx_gather_windows_i16");
  }
  gather_windows_i16_kernel<<<grid_for(n_streams * n_windows * n_samples, 256), 256, 0, (cudaStream_t)stream>>>(
      d_in, stream_stride, n_streams, n_windows, window_stride, n_samples, d_out);
  return after_launch("vadx_gather_windows_i16");
}

extern "C" int vadx_runs_to_segments(const uint8_t* d_silence_flags, int64_t ld, const int32_t* d_n_flags,
                                     int64_t n_streams, int32_t* d_seg_count, int32_t* d_segments, int max_segments,
                                     void* stream) {
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "runs_to_segments_kernel");
  VADX_REQUIRE(d_silence_flags && d_n_flags && d_seg_count && d_segments && max_segments >= 1 && ld >= 0,
               "vadx_runs_to_segments: bad argument");
  if (n_streams == 0) return VADX_OK;
  runs_to_segments_kernel<<<(unsigned)ceil_div(n_streams, 128), 128, 0, (cudaStream_t)stream>>>(
      d_silence_flags, ld, d_n_flags, n_streams, d_seg_count, d_segments, max_segments);
  return after_launch("vadx_runs_to_segments");
}
