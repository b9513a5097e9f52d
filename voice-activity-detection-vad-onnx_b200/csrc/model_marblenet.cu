// model_marblenet.cu -- NVIDIA Frame-VAD MarbleNet graph (wrapper:
// NVIDIA_Frame_VAD_Multilingual_MarbleNet/Export_NVIDIA_MarbleNet_VAD.py:222-275; the Jasper encoder
// itself is NeMo code that the reference does not vendor -- see oracle/marblenet.py) as a kernel
// sequence: prep -> framed DFT + power -> slaney mel + log -> [depthwise conv -> pointwise GEMM
// (+folded BN bias, +residual, ReLU)]* -> 2-class softmax head.
#include "model.hpp"

extern "C" int vadx_affine_f32(const float*, float, float, float*, int64_t, void*);
extern "C" int vadx_depthwise_conv1d_f32(const float*, int64_t, const float*, int, int, int, int, float*, int64_t,
                                         int64_t, int, int, int, void*);

namespace {
struct Block {
  int filters, repeat, kernel, stride, dilation, residual;
};
struct MarbleHP : FrontendGeom {
  int feat_in;
  std::vector<Block> blocks;
  int n_classes;
  int stft_frames(int64_t L) const { return (int)(L / hop + 1); }
  static int conv_len(int t, int k, int stride, int dil) {
    int pad = (dil * (k - 1)) / 2;
    return (t + 2 * pad - dil * (k - 1) - 1) / stride + 1;
  }
  int out_frames(int64_t L) const {
    int t = stft_frames(L);
    for (const auto& b : blocks)
      for (int r = 0; r < b.repeat; ++r) t = conv_len(t, b.kernel, b.stride, b.dilation);
    return t;
  }
  int max_channels() const {
    int c = feat_in;
    for (const auto& b : blocks) c = std::max(c, b.filters);
    return c;
  }
};

int marble_hp(const vadx_model* m, MarbleHP* h) {
  const auto& v = m->hp;
  VADX_REQUIRE(v.size() >= 2 && (int)v.size() == 2 + 6 * v[1] + 5, "marblenet: malformed hyper-parameter list (%zu)",
               v.size());
  h->feat_in = v[0];
  h->blocks.clear();
  for (int b = 0; b < v[1]; ++b) {
    const int32_t* p = &v[2 + 6 * b];
    h->blocks.push_back(Block{p[0], p[1], p[2], p[3], p[4], p[5]});
    VADX_REQUIRE(p[0] >= 1 && p[1] >= 1 && p[2] >= 1 && p[3] >= 1 && p[4] >= 1, "marblenet: block %d out of range", b);
    VADX_REQUIRE(p[3] == 1 || p[1] == 1, "marblenet: a strided block must have repeat == 1");
  }
  const int32_t* t = &v[2 + 6 * v[1]];
  h->n_classes = t[0]; h->n_fft = t[1]; h->win = t[2]; h->hop = t[3]; h->n_mels = t[4];
  VADX_REQUIRE(h->n_classes >= 2 && h->n_classes <= 8 && h->feat_in == h->n_mels, "marblenet: head/frontend mismatch");
  return VADX_OK;
}

// samples scaled by 1/32768, log(mel + eps); the resampler zeroes the centre pad before writing the upsampled signal
Frontend marble_frontend(const vadx_model* m, const MarbleHP& h) {
  return Frontend{h, h.n_bins(), h.pad_left(), 1.0f / 32768.0f, false, VADX_PREEMPH_ZERO_HISTORY, VADX_TC_FMT_F16,
                  VADX_FLOOR_ADD, (float)m->scalar("frontend.log_eps", 1e-7), frontend_rate_scale(m), false};
}
}  // namespace

int marblenet_check(const vadx_model* m) {
  MarbleHP h;
  return marble_hp(m, &h);
}
int marblenet_frames(const vadx_model* m, int64_t n_samples, int32_t* out) {
  MarbleHP h;
  VADX_TRY(marble_hp(m, &h));
  const double sc = frontend_rate_scale(m);
  *out = h.out_frames(sc == 1.0 ? n_samples : vadx_resample_out_len(n_samples, sc));
  return VADX_OK;
}

int marblenet_finalize(vadx_model* m) {
  MarbleHP h;
  VADX_TRY(marble_hp(m, &h));
  VADX_TRY(marble_frontend(m, h).finalize(m));
  int c_in = h.feat_in;
  for (size_t b = 0; b < h.blocks.size(); ++b) {
    const Block& k = h.blocks[b];
    int c = c_in;
    for (int r = 0; r < k.repeat; ++r) {
      std::string p = "b" + std::to_string(b) + ".r" + std::to_string(r) + ".";
      VADX_TRY(m->upload_raw(p + "dw", (int64_t)c * k.kernel, VADX_DT_F32));
      VADX_TRY(m->upload_linear(p + "pw", k.filters, c));
      VADX_TRY(m->upload_raw(p + "pw_bias", k.filters, VADX_DT_F32));
      c = k.filters;
    }
    if (k.residual) {
      std::string p = "b" + std::to_string(b) + ".";
      VADX_TRY(m->upload_linear(p + "res", k.filters, c_in));
      VADX_TRY(m->upload_raw(p + "res_bias", k.filters, VADX_DT_F32));
    }
    c_in = k.filters;
  }
  VADX_TRY(m->upload_linear("decoder.weight", h.n_classes, c_in));
  VADX_TRY(m->upload_raw("decoder.bias", h.n_classes, VADX_DT_F32));
  // Fused tail: when the last block is a single k = 1 separable block (marblenet_3x2x64: 128 x k1) its depthwise conv is a
  // per-channel scale that folds into the pointwise weight, and a 2-class softmax head is sigmoid((w1 - w0).y + b1 - b0): the
  // last pointwise layer and the head then run as ONE tensor-core kernel (vadx_linear_head_tc_f32), its 128-wide output
  // never leaves the SM.
  const Block& lb = h.blocks.back();
  if (h.n_classes == 2 && lb.repeat == 1 && lb.kernel == 1 && lb.stride == 1 && !lb.residual && h.blocks.size() >= 2) {
    const int cl = h.blocks[h.blocks.size() - 2].filters;                 // input channels of the last block
    const std::string p = "b" + std::to_string(h.blocks.size() - 1) + ".r0.";
    const HostTensor* dw = m->find(p + "dw");
    const HostTensor* pw = m->find(p + "pw");
    const HostTensor* dec = m->find("decoder.weight");
    const HostTensor* db = m->find("decoder.bias");
    if (dw && pw && dec && db && vadx_tc_supported(cl, lb.filters)) {
      HostTensor f;
      f.dtype = VADX_DT_F32;
      f.dims = {lb.filters, cl};
      f.bytes.resize((size_t)lb.filters * cl * sizeof(float));
      float* w = reinterpret_cast<float*>(f.bytes.data());
      for (int o = 0; o < lb.filters; ++o)
        for (int c = 0; c < cl; ++c) w[(size_t)o * cl + c] = pw->f32()[(size_t)o * cl + c] * dw->f32()[c];
      m->host["tail.pw_folded"] = std::move(f);
      VADX_TRY(m->upload_linear("tail.pw_folded", lb.filters, cl));
      std::vector<float> diff((size_t)lb.filters);
      for (int o = 0; o < lb.filters; ++o) diff[o] = dec->f32()[(size_t)lb.filters + o] - dec->f32()[o];
      VADX_TRY(m->upload("tail.head_w", diff.data(), diff.size() * sizeof(float)));
      m->scalars["derived.tail_head_b"] = (double)(db->f32()[1] - db->f32()[0]);
      m->scalars["derived.tail_fused"] = 1.0;
    }
  }
  return VADX_OK;
}

int marblenet_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S,
                  int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st) {
  (void)state;
  MarbleHP h;
  VADX_TRY(marble_hp(m, &h));
  const Frontend fe = marble_frontend(m, h);
  const double rate_scale = fe.rate_scale;
  const int64_t L_in = L;
  if (rate_scale != 1.0) L = vadx_resample_out_len(L_in, rate_scale);   // from here on L counts 16 kHz samples
  const int T0 = h.stft_frames(L);
  const int Tout = h.out_frames(L);
  const int64_t rows0 = S * T0;
  const int64_t Lp = round_up(h.pad_left() + std::max(L, L_in) + h.n_taps(), 4);
  const int maxc = h.max_channels();
  Workspace ws(ws_ptr, ws_bytes, dry);
  float* sig = ws.take<float>(S * Lp);
  float* sig2 = rate_scale == 1.0 ? nullptr : ws.take<float>(S * Lp);
  float* power = ws.take<float>(rows0 * h.ld_power());
  float* B[5];  // roles: 0 block input, 1 depthwise out, 2/3 pointwise ping-pong, 4 residual branch
  for (auto& b : B) b = ws.take<float>(rows0 * maxc);
  if (need) *need = ws.off;
  if (dry) return VADX_OK;
  if (ws.off > ws_bytes) {
    set_error("marblenet: workspace of %zu bytes is smaller than the %zu needed", ws_bytes, ws.off);
    return VADX_ENOMEM;
  }
  VADX_REQUIRE(out[1], "marblenet: outputs are {score_silence, score_active}");
  VADX_REQUIRE((char*)out[1] == (char*)out[0] + (size_t)S * Tout * sizeof(float),
               "marblenet: score_active must directly follow score_silence ([2][S][T'] planes)");
  const bool use_tc = m->scalar("engine.use_tc", 1.0) != 0.0;
  VADX_TRY(fe.run(m, static_cast<const int16_t*>(in[0]), S, L_in, T0, FrontendBufs{sig, sig2, Lp, power, nullptr, nullptr, B[0]},
                  st));
  auto lin = [&](const float* a, int n_in, const std::string& w, const std::string& b, const float* res, float* y,
                 int n_out, int64_t rows, int act) -> int {
    const uint8_t* img = use_tc && rows > kSkinnyMaxRows ? m->d<uint8_t>(w + "#TC") : nullptr;
    if (img) return vadx_linear_tc_f32(a, n_in, img, m->d<float>(b), res, n_out, y, n_out, rows, n_in, n_out, act, st);
    return vadx_linear_f32(a, n_in, m->d<float>(w + "#T"), (int)round_up(n_out, 4), m->d<float>(b), res, n_out, y, n_out,
                           rows, n_in, n_out, act, st);
  };
  int c_in = h.feat_in, t = T0;
  const bool fused_tail = use_tc && S * (int64_t)Tout > kSkinnyMaxRows && m->scalar("derived.tail_fused", 0.0) != 0.0 &&
                          m->scalar("engine.fuse_tail", 1.0) != 0.0 && m->d<uint8_t>("tail.pw_folded#TC");
  for (size_t bi = 0; bi < h.blocks.size(); ++bi) {
    const Block& k = h.blocks[bi];
    if (fused_tail && bi + 1 == h.blocks.size()) {
      // last block + decoder: p_active = sigmoid(head . relu(W' x + b)), p_silence = 1 - p_active
      const int64_t rows = S * (int64_t)t;
      float* planes = static_cast<float*>(out[0]);
      const std::string p = "b" + std::to_string(bi) + ".r0.";
      VADX_TRY(vadx_linear_head_tc_f32(B[0], c_in, m->d<uint8_t>("tail.pw_folded#TC"), m->d<float>(p + "pw_bias"), rows, c_in,
                                       k.filters, VADX_ACT_RELU, m->d<float>("tail.head_w"),
                                       (float)m->scalar("derived.tail_head_b", 0.0), planes + rows, st));
      VADX_REQUIRE(t == Tout, "marblenet: internal frame-count mismatch (%d vs %d)", t, Tout);
      return vadx_affine_f32(planes + rows, -1.0f, 1.0f, planes, rows, st);
    }
    const std::string bp = "b" + std::to_string(bi) + ".";
    if (k.residual)
      VADX_TRY(lin(B[0], c_in, bp + "res", bp + "res_bias", nullptr, B[4], k.filters, S * (int64_t)t, VADX_ACT_NONE));
    const float* cur = B[0];
    int c = c_in, out_slot = 2;
    for (int rep = 0; rep < k.repeat; ++rep) {
      const std::string p = bp + "r" + std::to_string(rep) + ".";
      const int pad = (k.dilation * (k.kernel - 1)) / 2;
      const int t_next = MarbleHP::conv_len(t, k.kernel, k.stride, k.dilation);
      VADX_TRY(vadx_depthwise_conv1d_f32(cur, c, m->d<float>(p + "dw"), k.kernel, k.stride, k.dilation, pad, B[1], c, S,
                                         t, t_next, c, st));
      t = t_next;
      out_slot = 2 + (rep & 1);
      const bool last = rep == k.repeat - 1;
      const bool add_res = last && k.residual;
      VADX_TRY(lin(B[1], c, p + "pw", p + "pw_bias", add_res ? B[4] : nullptr, B[out_slot], k.filters, S * (int64_t)t,
                   VADX_ACT_RELU | (add_res ? VADX_ACT_RES_FIRST : 0)));
      cur = B[out_slot];
      c = k.filters;
    }
    std::swap(B[0], B[out_slot]);  // the block output becomes the next block's input
    c_in = k.filters;
  }
  VADX_REQUIRE(t == Tout, "marblenet: internal frame-count mismatch (%d vs %d)", t, Tout);
  // head: [S*T'][C] -> softmax -> planes [2][S*T']
  return linear_narrow(B[0], c_in, m->d<float>("decoder.weight#T"), (int)round_up(h.n_classes, 4),
                       m->d<float>("decoder.bias"), static_cast<float*>(out[0]), S * (int64_t)t, c_in, h.n_classes,
                       VADX_ACT_SOFTMAX, (int)std::min<int64_t>(S * (int64_t)t, 0x7fffffff), 0, S * (int64_t)t, st);
}
