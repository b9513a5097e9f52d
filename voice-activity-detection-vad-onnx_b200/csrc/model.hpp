// model.hpp -- shared state of the native model runtime (model.cu, model_fsmn.cu, ...).
#pragma once
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"

namespace vadx {
int linear_narrow(const float* d_x, int64_t ldx, const float* d_wt, int ldw, const float* d_bias, float* d_y,
                  int64_t n_rows, int n_in, int n_out, int act, int rows_per_group, int64_t group_stride,
                  int64_t out_stride, cudaStream_t st);

struct HostTensor {
  std::vector<char> bytes;
  std::vector<int64_t> dims;
  int dtype = VADX_DT_F32;
  int64_t numel() const {
    int64_t n = 1;
    for (auto d : dims) n *= d;
    return n;
  }
  const float* f32() const { return reinterpret_cast<const float*>(bytes.data()); }
};

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

struct Workspace {  // bump allocator over the caller's buffer
  char* base;
  size_t cap, off = 0;
  bool dry;  // only measure
  Workspace(void* b, size_t c, bool d) : base((char*)b), cap(c), dry(d) {}
  template <typename T>
  T* take(int64_t n) {
    size_t bytes = (size_t)round_up((int64_t)(n * sizeof(T)), 256);
    char* p = dry ? nullptr : base + off;
    off += bytes;
    return reinterpret_cast<T*>(p);
  }
};

}  // namespace vadx

// gemm_tc.cu: dense layer whose input and/or output is in the tensor-core operand-stage format ([row tile][K chunk][hi | lo]
// 16 KB swizzled bf16 images, rows padded to whole 128-row tiles) instead of fp32 rows
int linear_tc_stages_f32(const float* d_x, const void* d_wimg, const float* d_bias, float* d_y, int64_t n_rows, int n_in,
                         int n_out, int act, int x_split, int y_split, void* stream);

// gemm_tc.cu / block_stages.cu: fc1 writing per-stream operand stages, and the fused fc2 + memory block that consumes them
int linear_tc_stream_stages_f32(const float* d_x, const void* d_wimg, const float* d_bias, float* d_y, int64_t n_rows,
                                int rows_per_stream, int n_in, int n_out, int act, void* stream);
size_t fc2_memory_stages_stream_bytes(int n_in, int n_frames);
bool fc2_memory_stages_supported(int n_in, int n_out, int n_frames, int n_back, int stride_back, int n_ahead, int stride_ahead);
int fc2_memory_stages_f32(const void* d_himg, int n_in, const void* d_wimg, const float* d_bias, int act, const float* d_wl,
                          int n_back, const float* d_wr, int n_ahead, const float* d_res, float* d_out, int64_t n_streams,
                          int n_frames, void* stream);

using namespace vadx;

struct vadx_model {
  std::string kind;
  std::vector<int32_t> hp;
  std::map<std::string, HostTensor> host;
  std::map<std::string, double> scalars;
  std::map<std::string, DevBuf> dev;  // derived, device-resident constants
  bool finalized = false;

  ~vadx_model() { release(); }
  void release() {
    for (auto& kv : dev)
      if (kv.second.p) cudaFree(kv.second.p);
    dev.clear();
    finalized = false;
  }
  double scalar(const char* name, double dflt) const {
    auto it = scalars.find(name);
    return it == scalars.end() ? dflt : it->second;
  }
  const HostTensor* find(const std::string& n) const {
    auto it = host.find(n);
    return it == host.end() ? nullptr : &it->second;
  }
    int upload(const std::string& key, const void* src, size_t bytes) {
    DevBuf b;
    b.bytes = bytes;
    cudaError_t e = cudaMalloc(&b.p, std::max<size_t>(bytes, 16));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(constant)");
    e = cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cudaFree(b.p);
      return cuda_fail(e, "cudaMemcpy(constant)");
    }
    auto it = dev.find(key);
    if (it != dev.end() && it->second.p) cudaFree(it->second.p);
    dev[key] = b;
    return VADX_OK;
  }
  // [out][in](,1) host weight -> device [in][ldw] (ldw = out rounded up to 4, zero padded)
  int upload_linear(const std::string& name, int n_out, int n_in) {
    const HostTensor* t = find(name);
    if (!t) {
      set_error("model '%s': tensor '%s' was never set", kind.c_str(), name.c_str());
      return VADX_EMISSING;
    }
    if (t->dtype != VADX_DT_F32 || t->numel() != (int64_t)n_out * n_in) {
      set_error("tensor '%s': expected %d x %d fp32, got %lld elements", name.c_str(), n_out, n_in,
                (long long)t->numel());
      return VADX_EINVAL;
    }
    int ldw = (int)round_up(n_out, 4);
    std::vector<float> wt((size_t)n_in * ldw, 0.f);
    const float* w = t->f32();
    for (int o = 0; o < n_out; ++o)
      for (int i = 0; i < n_in; ++i) wt[(size_t)i * ldw + o] = w[(size_t)o * n_in + i];
    VADX_TRY(upload(name + "#T", wt.data(), wt.size() * sizeof(float)));
    bool placed = false;
    if (vadx_tc_supported(n_in, n_out)) {
      size_t bytes = 0;
      VADX_TRY(vadx_pack_weight_tc(w, n_out, n_in, nullptr, 0, &bytes));
      std::vector<uint8_t> img(bytes);
      VADX_TRY(vadx_pack_weight_tc(w, n_out, n_in, img.data(), img.size(), &bytes));
      VADX_TRY(upload(name + "#TC", img.data(), img.size()));
      placed = true;
    } else if (n_in > 256 && n_out > 8 && n_out <= 256) {
      // K too long for one stationary operand image (FSMN 400 -> 140, Silero 516 -> 128): equal 64-aligned K parts
      // "#TCK<j>", each launch accumulating onto the previous one through the residual input (bias in the first part,
      // activation in the last)
      const int n_parts = (n_in + 255) / 256;
      const int pk = (int)round_up((n_in + n_parts - 1) / n_parts, 64);
      if (vadx_tc_supported(pk, n_out) && n_in - (n_parts - 1) * pk > 0) {
        for (int part = 0; part < n_parts; ++part) {
          const int k0 = part * pk, kn = std::min(pk, n_in - k0);
          std::vector<float> sub((size_t)n_out * kn);
          for (int o = 0; o < n_out; ++o)
            for (int i = 0; i < kn; ++i) sub[(size_t)o * kn + i] = w[(size_t)o * n_in + k0 + i];
          size_t bytes = 0;
          VADX_TRY(vadx_pack_weight_tc(sub.data(), n_out, kn, nullptr, 0, &bytes));
          std::vector<uint8_t> img(bytes);
          VADX_TRY(vadx_pack_weight_tc(sub.data(), n_out, kn, img.data(), img.size(), &bytes));
          VADX_TRY(upload(name + "#TCK" + std::to_string(part), img.data(), img.size()));
        }
        scalars["derived.ksplit." + name] = pk;
        placed = true;
      }
    }
    if (!placed && n_out > 16) {
      // N too wide for one stationary image (more than 256 columns, or the image leaves no room for the activation
      // stages: Silero 128 -> 512, FSMN 140 -> 250): column blocks "#TCN<j>" of equal 16-aligned width, one launch per
      // block writing its slice of the output rows (the input rows are read once per block)
      for (int wmax : {256, 128, 64}) {
        const int n_blocks = (n_out + wmax - 1) / wmax;
        const int bw = (int)round_up((n_out + n_blocks - 1) / n_blocks, 16);
        if (n_blocks < 2 || !vadx_tc_supported(n_in, bw) || n_out - (n_blocks - 1) * bw <= 8) continue;
        for (int j = 0; j < n_blocks; ++j) {
          const int c0 = j * bw, cn = std::min(bw, n_out - c0);
          size_t bytes = 0;
          VADX_TRY(vadx_pack_weight_tc(w + (size_t)c0 * n_in, cn, n_in, nullptr, 0, &bytes));
          std::vector<uint8_t> img(bytes);
          VADX_TRY(vadx_pack_weight_tc(w + (size_t)c0 * n_in, cn, n_in, img.data(), img.size(), &bytes));
          VADX_TRY(upload(name + "#TCN" + std::to_string(j), img.data(), img.size()));
        }
        scalars["derived.nsplit." + name] = bw;
        break;
      }
    }
    return VADX_OK;
  }
  // Y = act(X W^T + b) (+ res) for the layer uploaded by upload_linear(name, ...): one stationary tensor-core image when it
  // fits, two K halves (activation-free layers only), N column blocks, or the exact-fp32 FFMA kernel (use_tc = false, rows
  // <= kSkinnyMaxRows, shapes none of the above covers)
  int linear(const std::string& name, const float* x, int64_t ldx, const float* bias, const float* res, int64_t ldr, float* y,
             int64_t ldy, int64_t n_rows, int n_in, int n_out, int act, bool use_tc, void* st) const {
    if (use_tc && n_rows > kSkinnyMaxRows) {
      if (const uint8_t* img = d<uint8_t>(name + "#TC"))
        return vadx_linear_tc_f32(x, ldx, img, bias, res, ldr, y, ldy, n_rows, n_in, n_out, act, st);
      const int pk = (int)scalar(("derived.ksplit." + name).c_str(), 0.0);
      if (pk > 0 && !res && (act & VADX_ACT_RES_FIRST) == 0) {
        // long K in parts: y = x[:, :pk] W0^T + b, then y += x[:, pk:2pk] W1^T ..., the activation applied by the last part
        // on (partial sum + its own product)
        for (int part = 0, k0 = 0; k0 < n_in; ++part, k0 += pk) {
          const bool first = part == 0, last = k0 + pk >= n_in;
          VADX_TRY(vadx_linear_tc_f32(x + k0, ldx, d<uint8_t>(name + "#TCK" + std::to_string(part)), first ? bias : nullptr,
                                      first ? nullptr : y, ldy, y, ldy, n_rows, std::min(pk, n_in - k0), n_out,
                                      last ? (act | (first ? 0 : VADX_ACT_RES_FIRST)) : VADX_ACT_NONE, st));
        }
        return VADX_OK;
      }
      const int bw = (int)scalar(("derived.nsplit." + name).c_str(), 0.0);
      if (bw > 0 && ((ldy & 3) == 0 || (bw & 3) == 0)) {
        for (int j = 0, c0 = 0; c0 < n_out; ++j, c0 += bw)
          VADX_TRY(vadx_linear_tc_f32(x, ldx, d<uint8_t>(name + "#TCN" + std::to_string(j)), bias ? bias + c0 : nullptr,
                                      res ? res + c0 : nullptr, ldr, y + c0, ldy, n_rows, n_in, std::min(bw, n_out - c0), act, st));
        return VADX_OK;
      }
    }
    return vadx_linear_f32(x, ldx, d<float>(name + "#T"), (int)round_up(n_out, 4), bias, res, ldr, y, ldy, n_rows, n_in, n_out,
                           act, st);
  }
  // the sparse filterbank (frontend.mel_start / mel_len / mel_w) as a dense [n_mels][n_bins] tensor-core layer image
  // ("frontend.mel#TC") plus its per-column floor / epsilon vector ("frontend.mel_floor"); no-op when it does not fit
  int upload_mel_dense_tc(int n_mels, int n_bins, float floor_value) {
    const HostTensor* ms = find("frontend.mel_start");
    const HostTensor* ml = find("frontend.mel_len");
    const HostTensor* mw = find("frontend.mel_w");
    if (!ms || !ml || !mw || ms->numel() != n_mels || ml->numel() != n_mels || !vadx_tc_supported(n_bins, n_mels)) return VADX_OK;
    const int max_len = (int)(mw->numel() / n_mels);
    const int32_t* a = reinterpret_cast<const int32_t*>(ms->bytes.data());
    const int32_t* b = reinterpret_cast<const int32_t*>(ml->bytes.data());
    std::vector<float> dense((size_t)n_mels * n_bins, 0.f);
    for (int i = 0; i < n_mels; ++i)
      for (int j = 0; j < b[i] && a[i] + j < n_bins; ++j) dense[(size_t)i * n_bins + a[i] + j] = mw->f32()[(size_t)i * max_len + j];
    size_t bytes = 0;
    VADX_TRY(vadx_pack_weight_tc(dense.data(), n_mels, n_bins, nullptr, 0, &bytes));
    std::vector<uint8_t> img(bytes);
    VADX_TRY(vadx_pack_weight_tc(dense.data(), n_mels, n_bins, img.data(), img.size(), &bytes));
    VADX_TRY(upload("frontend.mel#TC", img.data(), img.size()));
    std::vector<float> fl((size_t)n_mels, floor_value);
    return upload("frontend.mel_floor", fl.data(), fl.size() * sizeof(float));
  }
  int upload_raw(const std::string& name, int64_t expect_numel, int dtype) {
    const HostTensor* t = find(name);
    if (!t) {
      set_error("model '%s': tensor '%s' was never set", kind.c_str(), name.c_str());
      return VADX_EMISSING;
    }
    if (t->dtype != dtype || (expect_numel >= 0 && t->numel() != expect_numel)) {
      set_error("tensor '%s': expected %lld elements of dtype %d, got %lld of dtype %d", name.c_str(),
                (long long)expect_numel, dtype, (long long)t->numel(), t->dtype);
      return VADX_EINVAL;
    }
    return upload(name, t->bytes.data(), t->bytes.size());
  }
  template <typename T>
  const T* d(const std::string& key) const {
    auto it = dev.find(key);
    return it == dev.end() ? nullptr : reinterpret_cast<const T*>(it->second.p);
  }
  bool has(const std::string& n) const { return host.count(n) != 0; }
};

// ------------------------------------------------------------------------------------------ log-mel frontend
// int16 audio -> power spectrum -> log-mel rows, shared by FireRed, FSMN and MarbleNet: the in-graph resampler path, the
// int16 tensor-core STFT or the fp32 FFMA STFT, then log-mel on the tensor cores or the sparse filterbank kernel.  Its
// tensors are "frontend.basis" (fp32 [n_taps][ld_basis], re/im interleaved) and the sparse filterbank "frontend.mel_start" /
// "mel_len" / "mel_w".

// framing: the window's n_taps non-zero taps start first_tap samples into the n_fft-point frame
struct FrontendGeom {
  int n_fft, win, hop, n_mels;
  int n_taps() const { return win < n_fft ? win : n_fft; }
  int first_tap() const { return win < n_fft ? (n_fft - win) / 2 : 0; }
  int n_bins() const { return n_fft / 2 + 1; }
  int ld_basis() const { return (int)round_up(2 * n_bins(), 4); }
  int ld_power() const { return (int)round_up(n_bins(), 4); }
  int pad_left() const { return n_fft / 2 - first_tap(); }  // centre pad ahead of the first tap
};

struct FrontendBufs {  // the caller's workspace
  float* sig;          // [S][Lp] prepped fp32 signal
  float* sig2;         // [S][Lp] second signal (resampler only)
  int64_t Lp;
  float* power;        // [S*T][ld_power]
  float* mean;         // [S] row means (remove_dc only)
  int32_t* mean_int;   // [S]
  float* mel;          // [S*T][n_mels] log-mel output
};

// What differs between the models' frontends.  The tensor-core paths run when engine.use_tc is set and S*T exceeds
// kSkinnyMaxRows; the int16 tensor-core STFT also needs L and pad_left to be multiples of 8, hop a multiple of 16 and
// 16-byte aligned audio.
struct Frontend {
  FrontendGeom g;
  int n_bins;          // DFT bins computed (<= g.n_bins())
  int pad_left;        // frame t starts at sample t*hop - pad_left, zeros outside the clip
  float in_scale;      // int16 -> fp32 sample scale; the tensor-core STFT scales the power by its square instead
  bool remove_dc;      // each row's mean removed before the pre-emphasis
  int preemph_mode;    // VADX_PREEMPH_* of the fp32 paths
  int tc_format;       // VADX_TC_FMT_* of the tensor-core DFT image
  int floor_mode;      // VADX_FLOOR_*: ln(max(mel, floor)) or ln(mel + floor)
  float floor_value;
  double rate_scale;   // in-graph resampler, 1 = none
  bool keep_signal;    // the prepped fp32 signal is produced on every path (read after the frontend)

  // uploads the basis, its tensor-core image, the mel tables and the dense tensor-core mel image
  int finalize(vadx_model* m) const;
  // audio [S][L] int16 (L at the input rate) -> b.mel [S*T][n_mels] on stream st
  int run(vadx_model* m, const int16_t* audio, int64_t S, int64_t L, int T, const FrontendBufs& b, cudaStream_t st) const;
};

// IN_SAMPLE_RATE != 16000 (Export_FireRedVAD.py:389-393, Export_NVIDIA_MarbleNet_VAD.py:180-183): scale = 1 / (in_rate /
// 16000), the in-graph linear resampler leaves floor(L * scale) samples at the model's 16 kHz
inline double frontend_rate_scale(const vadx_model* m) {
  const double in_rate = m->scalar("frontend.in_sample_rate", 16000.0);
  return in_rate == 16000.0 ? 1.0 : 1.0 / (in_rate / 16000.0);
}

inline int Frontend::finalize(vadx_model* m) const {
  VADX_TRY(m->upload_raw("frontend.basis", (int64_t)g.n_taps() * g.ld_basis(), VADX_DT_F32));
  if (vadx_stft_tc_supported(g.n_taps(), n_bins)) {
    // tensor-core DFT image: the pre-emphasis folded into the 2-term basis; a scale such as 1/32768 stays out of it (fp16
    // range) and multiplies the power instead
    const double preemph = m->scalar("frontend.preemph", 0.97);
    const float* hb = m->find("frontend.basis")->f32();
    size_t bytes = 0;
    VADX_TRY(vadx_pack_stft_basis_tc_fmt(hb, g.ld_basis(), g.n_taps(), n_bins, preemph, 1.0, tc_format, nullptr, 0, &bytes));
    std::vector<uint8_t> img(bytes);
    VADX_TRY(vadx_pack_stft_basis_tc_fmt(hb, g.ld_basis(), g.n_taps(), n_bins, preemph, 1.0, tc_format, img.data(), img.size(),
                                         &bytes));
    VADX_TRY(m->upload("frontend.basis#TC", img.data(), img.size()));
  }
  VADX_TRY(m->upload_raw("frontend.mel_start", g.n_mels, VADX_DT_I32));
  VADX_TRY(m->upload_raw("frontend.mel_len", g.n_mels, VADX_DT_I32));
  VADX_TRY(m->upload_raw("frontend.mel_w", -1, VADX_DT_F32));
  return m->upload_mel_dense_tc(g.n_mels, n_bins, floor_value);
}

inline int Frontend::run(vadx_model* m, const int16_t* audio, int64_t S, int64_t L, int T, const FrontendBufs& b,
                         cudaStream_t st) const {
  const int64_t rows = S * T;
  const bool use_tc = m->scalar("engine.use_tc", 1.0) != 0.0 && rows > kSkinnyMaxRows;
  const float preemph = (float)m->scalar("frontend.preemph", 0.97);
  const int pre = preemph > 0.f ? preemph_mode : 0;
  const int64_t Lp = b.Lp;
  const uint8_t* stft_img = use_tc ? m->d<uint8_t>("frontend.basis#TC") : nullptr;
  if (rate_scale != 1.0) {
    // in-graph resampler (Export_FireRedVAD.py:431-449, Export_NVIDIA_MarbleNet_VAD.py:236-254): downsample before the
    // scale + pre-emphasis, upsample after it
    if (rate_scale < 1.0) {
      VADX_TRY(vadx_prep_audio(audio, VADX_DT_I16, S, L, L, 1.0f, 0, 0, 0.f, 0, b.sig2, Lp, st));
      VADX_TRY(vadx_resample_linear_f32(b.sig2, Lp, L, S, rate_scale, b.sig, Lp, 0, st));
      VADX_TRY(vadx_prep_audio(b.sig, VADX_DT_F32, S, vadx_resample_out_len(L, rate_scale), Lp, in_scale, remove_dc, pre,
                               preemph, pad_left, b.sig2, Lp, st));
    } else {
      VADX_TRY(vadx_prep_audio(audio, VADX_DT_I16, S, L, L, in_scale, remove_dc, pre, preemph, 0, b.sig, Lp, st));
      if (pad_left > 0) {  // centre pad around the resampled signal
        cudaError_t e = cudaMemsetAsync(b.sig2, 0, (size_t)S * Lp * sizeof(float), st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(frontend centre pad)");
      }
      VADX_TRY(vadx_resample_linear_f32(b.sig, Lp, L, S, rate_scale, b.sig2, Lp, pad_left, st));
    }
    VADX_TRY(vadx_stft_power_f32(b.sig2, Lp, S, T, g.hop, g.n_taps(), m->d<float>("frontend.basis"), g.ld_basis(), n_bins,
                                 b.power, g.ld_power(), st));
  } else {
    const bool tc = stft_img && (L % 8) == 0 && (g.hop % 16) == 0 && (pad_left % 8) == 0 && aligned16(audio);
    if (keep_signal || !tc)
      VADX_TRY(vadx_prep_audio(audio, VADX_DT_I16, S, L, L, in_scale, remove_dc, pre, preemph, pad_left, b.sig, Lp, st));
    if (tc) {
      // framed DFT on the tensor cores straight from the int16 samples.  Frames reaching outside the clip and the mean
      // removal take per-frame correction tables (vadx_pack_stft_dc_tc), built per chunk length at first use
      const float* dc = nullptr;
      int lo = 0, hi = T;
      if (remove_dc || pad_left > 0) {
        const std::string key = "frontend.dc#" + std::to_string((long long)L);
        const std::string k_lo = key + ".lo", k_hi = key + ".hi";
        if (!m->d<float>(key)) {
          size_t n = 0;
          const float* hb = m->find("frontend.basis")->f32();
          VADX_TRY(vadx_pack_stft_dc_tc(hb, g.ld_basis(), g.n_taps(), n_bins, preemph, 1.0, L, g.hop, pad_left, T, nullptr, 0,
                                        &n, &lo, &hi));
          std::vector<float> tab(n);
          VADX_TRY(vadx_pack_stft_dc_tc(hb, g.ld_basis(), g.n_taps(), n_bins, preemph, 1.0, L, g.hop, pad_left, T, tab.data(),
                                        tab.size(), &n, &lo, &hi));
          VADX_TRY(m->upload(key, tab.data(), tab.size() * sizeof(float)));
          m->scalars[k_lo] = lo;
          m->scalars[k_hi] = hi;
        }
        dc = m->d<float>(key);
        lo = (int)m->scalar(k_lo.c_str(), 0.0);
        hi = (int)m->scalar(k_hi.c_str(), (double)T);
      }
      if (remove_dc) VADX_TRY(vadx_stream_mean_i16(audio, L, L, S, b.mean, b.mean_int, st));
      VADX_TRY(vadx_stft_power_tc_i16_ex(audio, L, L, S, T, g.hop, g.n_taps(), stft_img, n_bins, b.power, g.ld_power(), pad_left,
                                         remove_dc ? b.mean : nullptr, remove_dc ? b.mean_int : nullptr, dc, lo, hi,
                                         in_scale * in_scale, tc_format, st));
    } else {
      VADX_TRY(vadx_stft_power_f32(b.sig, Lp, S, T, g.hop, g.n_taps(), m->d<float>("frontend.basis"), g.ld_basis(), n_bins,
                                   b.power, g.ld_power(), st));
    }
  }
  if (use_tc && m->d<uint8_t>("frontend.mel#TC")) {
    // log-mel as a dense tensor-core layer: [rows][bins] x [bins][n_mels], the floor / epsilon in the bias slot
    return vadx_linear_tc_f32(b.power, g.ld_power(), m->d<uint8_t>("frontend.mel#TC"), m->d<float>("frontend.mel_floor"),
                              nullptr, 0, b.mel, g.n_mels, rows, n_bins, g.n_mels,
                              floor_mode == VADX_FLOOR_CLAMP ? VADX_ACT_LOG_CLAMP : VADX_ACT_LOG, st);
  }
  const int mel_max = (int)(m->find("frontend.mel_w")->numel() / g.n_mels);
  return vadx_mel_log_f32(b.power, g.ld_power(), rows, n_bins, g.n_mels, m->d<int32_t>("frontend.mel_start"),
                          m->d<int32_t>("frontend.mel_len"), m->d<float>("frontend.mel_w"), mel_max, floor_mode, floor_value,
                          b.mel, g.n_mels, st);
}


// per-kind entry points
int firered_check(const vadx_model* m);
int firered_finalize(vadx_model* m);
int firered_frames(const vadx_model* m, int64_t n_samples, int32_t* out);
int firered_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S,
                int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st);
int marblenet_check(const vadx_model* m);
int marblenet_finalize(vadx_model* m);
int marblenet_frames(const vadx_model* m, int64_t n_samples, int32_t* out);
int marblenet_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S,
                  int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st);
int silero_check(const vadx_model* m);
int silero_finalize(vadx_model* m);
int silero_frames(const vadx_model* m, int64_t n_samples, int32_t* out);
int silero_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S,
               int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st);
int fsmn_check(const vadx_model* m);
int fsmn_finalize(vadx_model* m);
int fsmn_frames(const vadx_model* m, int64_t n_samples, int32_t* out);
int fsmn_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S,
             int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st);
int dfsmn_check(const vadx_model* m);
int dfsmn_finalize(vadx_model* m);
int dfsmn_frames(const vadx_model* m, int64_t n_samples, int32_t* out);
int dfsmn_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S, int64_t L,
              void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st);
