// model_fsmn.cu -- FunASR FSMN-VAD graph (FSMN/Export_FSMN_VAD.py:75-101 around
// FSMN/modeling_modified/encoder.py:208-217) as a kernel sequence on the caller's stream.
//
// vadx_forward contract for kind "fsmn":
//   hparams  {input_dim, input_affine_dim, fsmn_layers, linear_dim, proj_dim, lorder, rorder, lstride,
//             rstride, output_affine_dim, output_dim, n_fft, win_length, hop, n_mels, lfr_m, lfr_n}
//   inputs   [0] audio int16 [S][L]        [1] noise_average_dB fp32 [S]
//   outputs  [0] score uint8 [S][T]        [1] noisy_dB fp32 [S]
//            [2] P(silence) fp32 [S][T] (optional)   [3] power_dB fp32 [S][T] (optional)
//   state    [0..n-1] caches in fp32 [S][proj][lorder-1], [n..2n-1] caches out (distinct buffers)
//   scalars  one_minus_speech_threshold (1.0), speech_2_noise_ratio (1.0), frontend.preemph (0.97),
//            frontend.log_floor (1e-5)
#include <cmath>

#include "model.hpp"

extern "C" {
int vadx_lfr_cmvn_f32(const float*, int64_t, const float*, const float*, float*, int64_t, int64_t, int, int, int, int,
                      void*);
int vadx_softmax_class0_f32(const float*, int64_t, int64_t, int, float*, void*);
int vadx_frame_energy_log10_f32(const float*, int64_t, int64_t, int64_t, int, int, int, int, float, float, float*,
                                void*);
int vadx_fsmn_gate(const float*, const float*, const float*, float, float, int64_t, int, uint8_t*, float*, void*);
int vadx_gather_windows_i16(const int16_t*, int64_t, int64_t, int, int64_t, int64_t, int16_t*, void*);
}

namespace {
struct FsmnHP : FrontendGeom {
  int input_dim, affine, layers, linear, proj, lorder, rorder, lstride, rstride, out_affine, out_dim, lfr_m, lfr_n;
  int frames(int64_t L) const { return (int)(L / hop + 1); }
};

int fsmn_hp(const vadx_model* m, FsmnHP* h) {
  VADX_REQUIRE(m->hp.size() == 17, "fsmn: expected 17 hyper-parameters, got %zu", m->hp.size());
  const int32_t* v = m->hp.data();
  *h = FsmnHP{{v[11], v[12], v[13], v[14]}, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], v[9], v[10], v[15], v[16]};
  VADX_REQUIRE(h->input_dim == h->n_mels * h->lfr_m, "fsmn: input_dim %d != n_mels*lfr_m", h->input_dim);
  VADX_REQUIRE(h->layers >= 1 && h->layers <= 8 && h->proj >= 1 && h->lorder >= 1 && h->lstride >= 1 && h->hop >= 1 &&
                   h->lfr_n == 1 && h->out_dim >= 2,
               "fsmn: hyper-parameter out of range");
  VADX_REQUIRE(h->rorder == 0, "fsmn: the reference never applies conv_right (encoder.py:78-83); rorder must be 0");
  return VADX_OK;
}

// the mean removed before the pre-emphasis (the tensor-core STFT corrects for it in the frequency domain); the fp32 signal
// is prepped on every path because the frame energy reads it
Frontend fsmn_frontend(const vadx_model* m, const FsmnHP& h) {
  return Frontend{h, h.n_bins(), h.pad_left(), 1.0f, true, VADX_PREEMPH_KEEP_FIRST, VADX_TC_FMT_BF16, VADX_FLOOR_CLAMP,
                  (float)m->scalar("frontend.log_floor", 1e-5), 1.0, true};
}
}  // namespace

int fsmn_check(const vadx_model* m) {
  FsmnHP h;
  return fsmn_hp(m, &h);
}
int fsmn_frames(const vadx_model* m, int64_t n_samples, int32_t* out) {
  FsmnHP h;
  VADX_TRY(fsmn_hp(m, &h));
  *out = h.frames(n_samples);
  return VADX_OK;
}

int fsmn_finalize(vadx_model* m) {
  FsmnHP h;
  VADX_TRY(fsmn_hp(m, &h));
  VADX_TRY(fsmn_frontend(m, h).finalize(m));
  VADX_TRY(m->upload_raw("cmvn_means", h.input_dim, VADX_DT_F32));
  VADX_TRY(m->upload_raw("cmvn_vars", h.input_dim, VADX_DT_F32));
  VADX_TRY(m->upload_linear("in_linear1.linear.weight", h.affine, h.input_dim));
  VADX_TRY(m->upload_raw("in_linear1.linear.bias", h.affine, VADX_DT_F32));
  VADX_TRY(m->upload_linear("in_linear2.linear.weight", h.linear, h.affine));
  VADX_TRY(m->upload_raw("in_linear2.linear.bias", h.linear, VADX_DT_F32));
  for (int i = 0; i < h.layers; ++i) {
    std::string p = "fsmn." + std::to_string(i) + ".";
    VADX_TRY(m->upload_linear(p + "linear.linear.weight", h.proj, h.linear));
    VADX_TRY(m->upload_raw(p + "fsmn_block.conv_left.weight", (int64_t)h.proj * h.lorder, VADX_DT_F32));
    VADX_TRY(m->upload_linear(p + "affine.linear.weight", h.linear, h.proj));
    VADX_TRY(m->upload_raw(p + "affine.linear.bias", h.linear, VADX_DT_F32));
  }
  VADX_TRY(m->upload_linear("out_linear1.linear.weight", h.out_affine, h.linear));
  VADX_TRY(m->upload_raw("out_linear1.linear.bias", h.out_affine, VADX_DT_F32));
  VADX_TRY(m->upload_linear("out_linear2.linear.weight", h.out_dim, h.out_affine));
  VADX_TRY(m->upload_raw("out_linear2.linear.bias", h.out_dim, VADX_DT_F32));
  return VADX_OK;
}

int fsmn_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S,
             int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st) {
  FsmnHP h;
  VADX_TRY(fsmn_hp(m, &h));
  const int T = h.frames(L);
  // Whole-file mode ("input.n_windows" = W > 1): in[0] is the chunk-aligned recording [S][input.stream_stride], the call
  // covers its W overlapping windows of L samples, "input.window_stride" apart.  Everything window-local (DC removal,
  // framing, mel, LFR, the dense layers, frame energy) runs ONCE over S*W window rows; the FSMN caches across windows are
  // nothing but a causal FIR over the concatenation of all windows' frames (encoder.py:78-83: cache_out = the last 19 frames
  // of cat(cache_in, p)), so every memory block runs as S streams of W*T frames.  Only the running background level is
  // sequential: the gate + look-ahead machine run afterwards (vadx_fsmn_gate_hysteresis_windows); this call returns
  // P(silence) and power_dB [S][W][T] (outputs 2, 3) and leaves outputs 0, 1 untouched.
  const int W = std::max(1, (int)m->scalar("input.n_windows", 1.0));
  const int64_t wstride = (int64_t)m->scalar("input.window_stride", (double)L);
  const int64_t sstride = (int64_t)m->scalar("input.stream_stride", (double)(L + (W - 1) * wstride));
  const int64_t S_streams = S;
  S = S * W;                                                     // window rows from here on
  const int64_t rows = S * T;
  const int64_t Lp = round_up(h.pad_left() + L + h.n_taps(), 4);
  const int wide = std::max(std::max(h.affine, h.linear), std::max(h.out_affine, h.out_dim));
  const int ldw = (int)round_up(wide, 4);
  Workspace ws(ws_ptr, ws_bytes, dry);
  float* sig = ws.take<float>(S * Lp);
  float* power = ws.take<float>(rows * h.ld_power());
  float* mel = ws.take<float>(rows * h.n_mels);
  float* feat = ws.take<float>(rows * h.input_dim);
  float* bufA = ws.take<float>(rows * ldw);
  float* bufB = ws.take<float>(rows * ldw);
  float* bufP = ws.take<float>(rows * h.proj);
  float* bufM = ws.take<float>(rows * h.proj);
  float* p_sil_ws = ws.take<float>(rows);
  float* power_db_ws = ws.take<float>(rows);
  float* mean_ws = ws.take<float>(S);
  int32_t* mean_int_ws = ws.take<int32_t>(S);
  int16_t* win16 = W > 1 ? ws.take<int16_t>(S * L) : nullptr;       // whole-file mode: the windows as dense int16 rows
  if (need) *need = ws.off;
  if (dry) return VADX_OK;
  if (ws.off > ws_bytes) {
    set_error("fsmn: workspace of %zu bytes is smaller than the %zu needed", ws_bytes, ws.off);
    return VADX_ENOMEM;
  }
  VADX_REQUIRE(L >= h.n_fft, "fsmn: chunk of %lld samples is shorter than the %d-sample energy frame", (long long)L,
               h.n_fft);
  VADX_REQUIRE(state && (W > 1 ? (out[2] && out[3]) : (in[1] && out[1])),
               W > 1 ? "fsmn: whole-file mode needs the P(silence) and power_dB outputs and the cache state"
                     : "fsmn: noise_average_dB input, noisy_dB output and cache state are required");
  VADX_REQUIRE(W == 1 || (wstride >= 1 && sstride >= L + (int64_t)(W - 1) * wstride),
               "fsmn: input.stream_stride %lld does not hold %d windows of %lld samples, %lld apart", (long long)sstride, W,
               (long long)L, (long long)wstride);
  for (int i = 0; i < 2 * h.layers; ++i) VADX_REQUIRE(state[i], "fsmn: cache state %d is null", i);
  const float* noise_avg = static_cast<const float*>(in[1]);
  uint8_t* score = static_cast<uint8_t*>(out[0]);
  float* noisy = static_cast<float*>(out[1]);
  float* p_sil = out[2] ? static_cast<float*>(out[2]) : p_sil_ws;
  float* power_db = out[3] ? static_cast<float*>(out[3]) : power_db_ws;
  const float thr = (float)m->scalar("one_minus_speech_threshold", 1.0);
  const float ratio = (float)m->scalar("speech_2_noise_ratio", 1.0);

  const int16_t* audio = static_cast<const int16_t*>(in[0]);
  if (W > 1) {
    // the W windows of every stream become ordinary rows; everything below is the batched single-window path over S*W rows
    VADX_TRY(vadx_gather_windows_i16(audio, sstride, S_streams, W, wstride, L, win16, st));
    audio = win16;
  }
  VADX_TRY(fsmn_frontend(m, h).run(m, audio, S, L, T, FrontendBufs{sig, nullptr, Lp, power, mean_ws, mean_int_ws, mel}, st));
  VADX_TRY(vadx_lfr_cmvn_f32(mel, h.n_mels, m->d<float>("cmvn_means"), m->d<float>("cmvn_vars"), feat, h.input_dim, S,
                             T, h.n_mels, h.lfr_m, h.lfr_n, st));
  const bool tc_rows = m->scalar("engine.use_tc", 1.0) != 0.0;
  auto lin = [&](const float* x, int64_t ldx, int n_in, const std::string& w, const char* b, float* y, int64_t ldy,
                 int n_out, int act) -> int {
    return m->linear(w, x, ldx, b ? m->d<float>(b) : nullptr, nullptr, 0, y, ldy, rows, n_in, n_out, act, tc_rows, st);
  };
  VADX_TRY(lin(feat, h.input_dim, h.input_dim, "in_linear1.linear.weight", "in_linear1.linear.bias", bufA, ldw,
               h.affine, VADX_ACT_NONE));
  VADX_TRY(lin(bufA, ldw, h.affine, "in_linear2.linear.weight", "in_linear2.linear.bias", bufB, ldw, h.linear,
               VADX_ACT_RELU));
  float* hcur = bufB;
  float* hnext = bufA;
  const int halo = (h.lorder - 1) * h.lstride;
  for (int i = 0; i < h.layers; ++i) {
    std::string p = "fsmn." + std::to_string(i) + ".";
    std::string ab = p + "affine.linear.bias";
    VADX_TRY(lin(hcur, ldw, h.linear, p + "linear.linear.weight", nullptr, bufP, h.proj, h.proj, VADX_ACT_NONE));
    VADX_TRY(vadx_fsmn_memory_f32(bufP, h.proj, m->d<float>(p + "fsmn_block.conv_left.weight"), h.lorder, h.lstride,
                                  nullptr, 0, 1, nullptr, 0, bufM, h.proj, S_streams, W * T, h.proj,
                                  halo > 0 ? static_cast<const float*>(state[i]) : nullptr,
                                  halo > 0 ? static_cast<float*>(state[h.layers + i]) : nullptr, st));
    VADX_TRY(lin(bufM, h.proj, h.proj, p + "affine.linear.weight", ab.c_str(), hnext, ldw, h.linear, VADX_ACT_RELU));
    std::swap(hcur, hnext);
  }
  VADX_TRY(lin(hcur, ldw, h.linear, "out_linear1.linear.weight", "out_linear1.linear.bias", hnext, ldw, h.out_affine,
               VADX_ACT_NONE));
  VADX_TRY(lin(hnext, ldw, h.out_affine, "out_linear2.linear.weight", "out_linear2.linear.bias", hcur, ldw, h.out_dim,
               VADX_ACT_NONE));
  VADX_TRY(vadx_softmax_class0_f32(hcur, ldw, rows, h.out_dim, p_sil, st));
  const int n_energy = (int)((L - h.n_fft) / h.hop + 1);
  const float inv_ref = (float)(1.0 / (std::sqrt((double)L) * 2e-5));
  VADX_TRY(vadx_frame_energy_log10_f32(sig, Lp, h.pad_left(), S, h.n_fft, h.hop, n_energy, T, inv_ref, 0.00002f,
                                       power_db, st));
  if (W > 1) return VADX_OK;      // the gate needs the running background level: vadx_fsmn_gate_hysteresis_windows
  VADX_TRY(vadx_fsmn_gate(p_sil, power_db, noise_avg, thr, ratio, S, T, score, noisy, st));
  return VADX_OK;
}
