// model.cu -- the native runtime behind vadx_create / vadx_set_tensor / vadx_forward: owns the
// constants of one model, lays the caller's workspace out, and enqueues the kernel sequence of a
// whole forward pass on the caller's stream (no host synchronisation, no allocation).
#include "model.hpp"

// ------------------------------------------------------------------------------------------ FireRed
struct FireRedHP : FrontendGeom {
  int idim, R, M, H, P, N1, S1, N2, S2, odim;
  int frames(int64_t L) const { return L < n_taps() ? 0 : (int)(1 + (L - n_taps()) / hop); }
};

static int firered_hp(const vadx_model* m, FireRedHP* h) {
  VADX_REQUIRE(m->hp.size() == 14, "firered: expected 14 hyper-parameters, got %zu", m->hp.size());
  const int32_t* v = m->hp.data();
  *h = FireRedHP{{v[10], v[11], v[12], v[13]}, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], v[9]};
  VADX_REQUIRE(h->idim == h->n_mels, "firered: idim (%d) must equal n_mels (%d)", h->idim, h->n_mels);
  VADX_REQUIRE(h->R >= 1 && h->M >= 1 && h->H >= 1 && h->P >= 1 && h->N1 >= 1 && h->S1 >= 1 && h->N2 >= 0 &&
                   h->odim >= 1 && h->odim <= 8 && h->hop >= 1 && h->n_fft >= 2,
               "firered: hyper-parameter out of range");
  return VADX_OK;
}

// DFT over derived.bins_used only; no centre pad: frames start at sample 0
static Frontend firered_frontend(const vadx_model* m, const FireRedHP& h) {
  return Frontend{h, (int)m->scalar("derived.bins_used", (double)h.n_bins()), 0, 1.0f, false, VADX_PREEMPH_ZERO_HISTORY,
                  VADX_TC_FMT_F16, VADX_FLOOR_CLAMP, (float)m->scalar("frontend.log_floor", 1e-7), frontend_rate_scale(m),
                  false};
}

int firered_finalize(vadx_model* m) {
  FireRedHP h;
  VADX_TRY(firered_hp(m, &h));
  // bins the filterbank actually reads: the Kaldi-style bank gives zero weight to DC and Nyquist, so the
  // DFT only has to produce bins [0, bins_used) (FireRed: 200 of 201 -> 400 columns = exactly five 80-wide tiles)
  int bins_used = 1;
  {
    const HostTensor* ms = m->find("frontend.mel_start");
    const HostTensor* ml = m->find("frontend.mel_len");
    if (ms && ml && ms->dtype == VADX_DT_I32 && ml->dtype == VADX_DT_I32 && ms->numel() == h.n_mels && ml->numel() == h.n_mels) {
      const int32_t* a = reinterpret_cast<const int32_t*>(ms->bytes.data());
      const int32_t* b = reinterpret_cast<const int32_t*>(ml->bytes.data());
      for (int i = 0; i < h.n_mels; ++i) bins_used = std::max(bins_used, a[i] + b[i]);
    } else {
      bins_used = h.n_bins();
    }
    bins_used = std::min(bins_used, h.n_bins());
    m->scalars["derived.bins_used"] = bins_used;
  }
  VADX_TRY(firered_frontend(m, h).finalize(m));
  VADX_TRY(m->upload_linear("dfsmn.fc1.0.weight", h.H, h.idim));
  VADX_TRY(m->upload_raw("dfsmn.fc1.0.bias", h.H, VADX_DT_F32));
  VADX_TRY(m->upload_linear("dfsmn.fc2.0.weight", h.P, h.H));
  VADX_TRY(m->upload_raw("dfsmn.fc2.0.bias", h.P, VADX_DT_F32));
  auto memory = [&](const std::string& pre) -> int {
    VADX_TRY(m->upload_raw(pre + "lookback_filter.weight", (int64_t)h.P * h.N1, VADX_DT_F32));
    if (h.N2 > 0) VADX_TRY(m->upload_raw(pre + "lookahead_filter.weight", (int64_t)h.P * h.N2, VADX_DT_F32));
    return VADX_OK;
  };
  VADX_TRY(memory("dfsmn.fsmn1."));
  for (int i = 0; i < h.R - 1; ++i) {
    std::string pre = "dfsmn.fsmns." + std::to_string(i) + ".";
    VADX_TRY(m->upload_linear(pre + "fc1.0.weight", h.H, h.P));
    VADX_TRY(m->upload_raw(pre + "fc1.0.bias", h.H, VADX_DT_F32));
    VADX_TRY(m->upload_linear(pre + "fc2.weight", h.P, h.H));
    VADX_TRY(memory(pre + "fsmn."));
  }
  VADX_TRY(m->upload_linear("dfsmn.dnns.0.weight", h.H, h.P));
  VADX_TRY(m->upload_raw("dfsmn.dnns.0.bias", h.H, VADX_DT_F32));
  for (int j = 1; j < h.M; ++j) {
    std::string n = "dfsmn.dnns." + std::to_string(2 * j);
    VADX_TRY(m->upload_linear(n + ".weight", h.H, h.H));
    VADX_TRY(m->upload_raw(n + ".bias", h.H, VADX_DT_F32));
  }
  VADX_TRY(m->upload_linear("out.weight", h.odim, h.H));
  VADX_TRY(m->upload_raw("out.weight", (int64_t)h.odim * h.H, VADX_DT_F32));
  VADX_TRY(m->upload_raw("out.bias", h.odim, VADX_DT_F32));
  return VADX_OK;
}

int firered_check(const vadx_model* m) {
  FireRedHP h;
  return firered_hp(m, &h);
}
int firered_frames(const vadx_model* m, int64_t n_samples, int32_t* out) {
  FireRedHP h;
  VADX_TRY(firered_hp(m, &h));
  const double sc = frontend_rate_scale(m);
  *out = h.frames(sc == 1.0 ? n_samples : vadx_resample_out_len(n_samples, sc));
  return VADX_OK;
}

// Optional slab execution: with engine.slab_streams = n > 0 the network runs n streams at a time over
// slab-sized activation buffers (bounds the workspace; a slab's intermediates stay L2-resident).  Off by
// default: measured on B200 the layer kernels are bound by their own load pipelines, not by HBM traffic,
// so slabs only add launches (8192 chunks: 11.9 ms whole, 13.8 ms at 1536, 18.1 ms at 384 per slab).
static int64_t firered_slab(const vadx_model* m, int64_t S) {
  int64_t slab = (int64_t)m->scalar("engine.slab_streams", 0.0);
  if (slab <= 0 || slab > S) slab = S;
  return slab;
}

// lays out (dry = true) or runs the forward pass
int firered_run(vadx_model* m, bool dry, const void* const* in, void* const* out, void* const* state, int64_t S_all,
                int64_t L, void* ws_ptr, size_t ws_bytes, size_t* need, cudaStream_t st) {
  FireRedHP h;
  VADX_TRY(firered_hp(m, &h));
  const int16_t* d_audio_all = dry ? nullptr : static_cast<const int16_t*>(in[0]);
  float* d_probs_all = dry ? nullptr : static_cast<float*>(out[0]);
  // Stream-VAD twin (Export_FireRedVAD.py:496-622): state[0] = caches_in, state[1] = caches_out, both
  // [R][S][P][(N1-1)*S1] -- the reference's (R,1,P,Lb) with the unit axis generalised to S streams
  const float* cin_all = (!dry && state && state[0]) ? static_cast<const float*>(state[0]) : nullptr;
  float* cout_all = (!dry && state && state[0]) ? static_cast<float*>(state[1]) : nullptr;
  if (cin_all) {
    VADX_REQUIRE(h.N2 == 0, "firered: the streaming graph has no look-ahead taps (N2 must be 0, got %d)", h.N2);
    VADX_REQUIRE(cout_all && cout_all != cin_all, "firered: streaming needs a caches_out buffer distinct from caches_in");
  }
  const int64_t cache_stream = (int64_t)h.P * (h.N1 - 1) * h.S1;
  const int64_t cache_layer = S_all * cache_stream;
  const Frontend fe = firered_frontend(m, h);
  const double rate_scale = fe.rate_scale;
  const int64_t L16 = rate_scale == 1.0 ? L : vadx_resample_out_len(L, rate_scale);   // samples at the model's 16 kHz
  const int T = h.frames(L16);
  VADX_REQUIRE(T >= 1, "firered: %lld samples are shorter than one %d-sample frame", (long long)L16, h.n_taps());
  const int64_t slab = firered_slab(m, S_all);
  const int64_t slab_rows = slab * T;
  const int64_t Lp = round_up(std::max(L, L16), 4);
  Workspace ws(ws_ptr, ws_bytes, dry);
  float* sig = ws.take<float>(slab * Lp);
  float* sig2 = rate_scale == 1.0 ? nullptr : ws.take<float>(slab * Lp);
  float* power = ws.take<float>(slab_rows * h.ld_power());
  float* feat = ws.take<float>(slab_rows * h.n_mels);
  // whole row tiles / per-stream image sets: bufH may hold operand stages instead of fp32 rows (split_hidden, fuse_stages)
  const int64_t bufH_floats = std::max<int64_t>(round_up(slab_rows, 128) * h.H,
                                                (h.H % 64) == 0 ? slab * (int64_t)(fc2_memory_stages_stream_bytes(h.H, T) / 4) : 0);
  float* bufH = ws.take<float>(bufH_floats);
  float* bufH2 = h.M > 1 ? ws.take<float>(slab_rows * h.H) : nullptr;
  float* bufP = ws.take<float>(slab_rows * h.P);
  float* memA0 = ws.take<float>(slab_rows * h.P);
  float* memB0 = ws.take<float>(slab_rows * h.P);
  if (need) *need = ws.off;
  if (dry) return VADX_OK;
  if (ws.off > ws_bytes) {
    set_error("firered: workspace of %zu bytes is smaller than the %zu needed", ws_bytes, ws.off);
    return VADX_ENOMEM;
  }

  for (int64_t s0 = 0; s0 < S_all; s0 += slab) {
    const int64_t S = std::min(slab, S_all - s0);
    const int64_t rows = S * T;
    const int16_t* d_audio = d_audio_all + s0 * L;
    float* d_probs = d_probs_all + s0 * (int64_t)h.odim * T;
    const float* cin = cin_all ? cin_all + s0 * cache_stream : nullptr;
    float* cout = cin_all ? cout_all + s0 * cache_stream : nullptr;
    float* memA = memA0;
    float* memB = memB0;
    const bool use_tc = m->scalar("engine.use_tc", 1.0) != 0.0 && rows > kSkinnyMaxRows;
    VADX_TRY(fe.run(m, d_audio, S, L, T, FrontendBufs{sig, sig2, Lp, power, nullptr, nullptr, feat}, st));
    auto lin = [&](const float* x, int n_in, const std::string& w, const char* b, const float* res, float* y, int n_out,
                   int act) -> int {
      const uint8_t* img = use_tc ? m->d<uint8_t>(w + "#TC") : nullptr;
      if (img)
        return vadx_linear_tc_f32(x, n_in, img, b ? m->d<float>(b) : nullptr, res, n_out, y, n_out, rows, n_in, n_out,
                                  act, st);
      return vadx_linear_f32(x, n_in, m->d<float>(w + "#T"), (int)round_up(n_out, 4), b ? m->d<float>(b) : nullptr, res,
                             n_out, y, n_out, rows, n_in, n_out, act, st);
    };
    auto memory = [&](int layer, const std::string& pre, const float* p, const float* res, float* o) -> int {
      return vadx_fsmn_memory_f32(p, h.P, m->d<float>(pre + "lookback_filter.weight"), h.N1, h.S1,
                                  h.N2 > 0 ? m->d<float>(pre + "lookahead_filter.weight") : nullptr, h.N2,
                                  h.N2 > 0 ? h.S2 : 1, res, h.P, o, h.P, S, T, h.P,
                                  cin ? cin + layer * cache_layer : nullptr, cin ? cout + layer * cache_layer : nullptr,
                                  st);
    };
    // fc1 -> fc2 hand-over in the tensor-core operand format: fc1's epilogue writes relu(h) already split into the two bf16
    // terms and swizzled into the 16 KB stage images fc2's MMA reads, fc2 streams them in with bulk copies (same bytes in
    // HBM as fp32 rows; fc2 loses its load/convert/store loader, the stage the L1 data pipe was saturated by)
    const bool split_hidden = use_tc && (h.H % 64) == 0 && m->scalar("engine.split_hidden", 1.0) != 0.0;
    // fc2 + memory block + residual in one kernel fed by per-stream stages (block_stages.cu): p never reaches HBM
    const bool fuse_stages = split_hidden && !cin && fc2_memory_stages_supported(h.H, h.P, T, h.N1, h.S1, h.N2, h.N2 > 0 ? h.S2 : 1) &&
                             m->scalar("engine.fuse_stages", 1.0) != 0.0 &&
                             // fc1's epilogue addresses a stream's image set with 32-bit byte offsets
                             S * (int64_t)fc2_memory_stages_stream_bytes(h.H, T) < (1LL << 32);
    auto fc1 = [&](const float* x, int n_in, const std::string& w, const char* b) -> int {
      if (fuse_stages)
        return linear_tc_stream_stages_f32(x, m->d<uint8_t>(w + "#TC"), b ? m->d<float>(b) : nullptr, bufH, rows, T, n_in, h.H,
                                           VADX_ACT_RELU, st);
      const uint8_t* img = split_hidden ? m->d<uint8_t>(w + "#TC") : nullptr;
      if (img) return linear_tc_stages_f32(x, img, b ? m->d<float>(b) : nullptr, bufH, rows, n_in, h.H, VADX_ACT_RELU, 0, 1, st);
      return lin(x, n_in, w, b, nullptr, bufH, h.H, VADX_ACT_RELU);
    };
    auto block_tail = [&](const std::string& w, const char* b, int act, const std::string& mem_pre, int layer, const float* res,
                          float* o) -> int {
      if (fuse_stages)
        return fc2_memory_stages_f32(bufH, h.H, m->d<uint8_t>(w + "#TC"), b ? m->d<float>(b) : nullptr, act,
                                     m->d<float>(mem_pre + "lookback_filter.weight"), h.N1,
                                     m->d<float>(mem_pre + "lookahead_filter.weight"), h.N2, res, o, S, T, st);
      const uint8_t* simg = split_hidden ? m->d<uint8_t>(w + "#TC") : nullptr;
      if (simg) VADX_TRY(linear_tc_stages_f32(bufH, simg, b ? m->d<float>(b) : nullptr, bufP, rows, h.H, h.P, act, 1, 0, st));
      else VADX_TRY(lin(bufH, h.H, w, b, nullptr, bufP, h.P, act));
      return memory(layer, mem_pre, bufP, res, o);
    };
    VADX_TRY(fc1(feat, h.idim, "dfsmn.fc1.0.weight", "dfsmn.fc1.0.bias"));
    VADX_TRY(block_tail("dfsmn.fc2.0.weight", "dfsmn.fc2.0.bias", VADX_ACT_RELU, "dfsmn.fsmn1.", 0, nullptr, memA));
    for (int i = 0; i < h.R - 1; ++i) {
      std::string pre = "dfsmn.fsmns." + std::to_string(i) + ".";
      std::string b1 = pre + "fc1.0.bias";
      VADX_TRY(fc1(memA, h.P, pre + "fc1.0.weight", b1.c_str()));
      VADX_TRY(block_tail(pre + "fc2.weight", nullptr, VADX_ACT_NONE, pre + "fsmn.", i + 1, memA, memB));
      std::swap(memA, memB);
    }
    if (use_tc && h.M == 1 && h.odim == 1 && m->d<uint8_t>("dfsmn.dnns.0.weight#TC")) {
      // last dense layer + 1-output sigmoid head in one tensor-core kernel: [S*T][1] == [S][1][T]
      const HostTensor* ob = m->find("out.bias");
      VADX_TRY(vadx_linear_head_tc_f32(memA, h.P, m->d<uint8_t>("dfsmn.dnns.0.weight#TC"),
                                       m->d<float>("dfsmn.dnns.0.bias"), rows, h.P, h.H, VADX_ACT_RELU,
                                       m->d<float>("out.weight"), ob->f32()[0], d_probs, st));
      continue;
    }
    VADX_TRY(lin(memA, h.P, "dfsmn.dnns.0.weight", "dfsmn.dnns.0.bias", nullptr, bufH, h.H, VADX_ACT_RELU));
    float* hcur = bufH;
    float* hnext = bufH2;
    for (int j = 1; j < h.M; ++j) {
      std::string n = "dfsmn.dnns." + std::to_string(2 * j);
      std::string b = n + ".bias";
      VADX_TRY(lin(hcur, h.H, n + ".weight", b.c_str(), nullptr, hnext, h.H, VADX_ACT_RELU));
      std::swap(hcur, hnext);
    }
    // head: [S*T][H] -> probs [S][odim][T]
    VADX_TRY(linear_narrow(hcur, h.H, m->d<float>("out.weight#T"), (int)round_up(h.odim, 4), m->d<float>("out.bias"),
                           d_probs, rows, h.H, h.odim, VADX_ACT_SIGMOID, T, (int64_t)h.odim * T, T, st));
  }
  return VADX_OK;
}

// ------------------------------------------------------------------------------------------ C ABI
namespace {
struct KindOps {
  const char* name;
  int (*check)(const vadx_model*);
  int (*finalize)(vadx_model*);
  int (*frames)(const vadx_model*, int64_t, int32_t*);
  int (*run)(vadx_model*, bool, const void* const*, void* const*, void* const*, int64_t, int64_t, void*, size_t,
             size_t*, cudaStream_t);
};
const KindOps kKinds[] = {
    {"firered", firered_check, firered_finalize, firered_frames, firered_run},
    {"fsmn", fsmn_check, fsmn_finalize, fsmn_frames, fsmn_run},
    {"silero", silero_check, silero_finalize, silero_frames, silero_run},
    {"marblenet", marblenet_check, marblenet_finalize, marblenet_frames, marblenet_run},
    {"dfsmn_aec", dfsmn_check, dfsmn_finalize, dfsmn_frames, dfsmn_run},
};
const KindOps* ops_of(const std::string& kind) {
  for (const auto& k : kKinds)
    if (kind == k.name) return &k;
  return nullptr;
}
}  // namespace

extern "C" int vadx_create(const char* kind, const int32_t* hparams, int n_hparams, vadx_model** out) {
  VADX_REQUIRE(kind && out && (n_hparams == 0 || hparams), "vadx_create: null pointer");
  const KindOps* ops = ops_of(kind);
  VADX_REQUIRE(ops, "vadx_create: unknown model kind '%s'", kind);
  if (vadx_device_count() < 1) {
    set_error("vadx_create: no CUDA device is visible; libvadx has no CPU path");
    return VADX_ENODEVICE;
  }
  vadx_model* m = new vadx_model();
  m->kind = kind;
  m->hp.assign(hparams, hparams + n_hparams);
  int rc = ops->check(m);
  if (rc != VADX_OK) {
    delete m;
    return rc;
  }
  *out = m;
  return VADX_OK;
}

extern "C" void vadx_destroy(vadx_model* m) { delete m; }

extern "C" int vadx_set_tensor(vadx_model* m, const char* name, const void* h_data, int dtype, const int64_t* dims,
                               int n_dims) {
  VADX_REQUIRE(m && name && h_data && dims && n_dims >= 1 && n_dims <= 8, "vadx_set_tensor: bad argument");
  VADX_REQUIRE(dtype == VADX_DT_I16 || dtype == VADX_DT_F32 || dtype == VADX_DT_I32, "vadx_set_tensor: dtype %d", dtype);
  HostTensor t;
  t.dtype = dtype;
  t.dims.assign(dims, dims + n_dims);
  for (int i = 0; i < n_dims; ++i) VADX_REQUIRE(dims[i] >= 0, "vadx_set_tensor: negative dim");
  size_t esz = dtype == VADX_DT_I16 ? 2 : 4;
  t.bytes.resize((size_t)t.numel() * esz);
  memcpy(t.bytes.data(), h_data, t.bytes.size());
  m->host[name] = std::move(t);
  m->finalized = false;
  return VADX_OK;
}

extern "C" int vadx_set_scalar(vadx_model* m, const char* name, double value) {
  VADX_REQUIRE(m && name, "vadx_set_scalar: null pointer");
  if (!strncmp(name, "frontend.", 9)) m->finalized = false;  // folded into device-side constants
  m->scalars[name] = value;
  return VADX_OK;
}

extern "C" int vadx_output_frames(const vadx_model* m, int64_t n_samples, int32_t* out_frames) {
  VADX_REQUIRE(m && out_frames, "vadx_output_frames: null pointer");
  return ops_of(m->kind)->frames(m, n_samples, out_frames);
}

extern "C" int vadx_workspace_bytes(const vadx_model* m, int64_t n_streams, int64_t n_samples, size_t* out_bytes) {
  VADX_REQUIRE(m && out_bytes && n_streams >= 0 && n_samples >= 0, "vadx_workspace_bytes: bad argument");
  return ops_of(m->kind)->run(const_cast<vadx_model*>(m), true, nullptr, nullptr, nullptr, n_streams, n_samples,
                              nullptr, 0, out_bytes, nullptr);
}

extern "C" int vadx_forward(vadx_model* m, const void* const* d_inputs, void* const* d_outputs, void* const* d_state,
                            int64_t n_streams, int64_t n_samples, void* d_workspace, size_t workspace_bytes,
                            void* stream) {
  VADX_REQUIRE(m && d_inputs && d_outputs && d_inputs[0] && d_outputs[0], "vadx_forward: null pointer");
  VADX_REQUIRE(n_streams >= 0 && n_samples > 0, "vadx_forward: bad shape S=%lld L=%lld", (long long)n_streams,
               (long long)n_samples);
  VADX_REQUIRE(d_workspace || workspace_bytes == 0, "vadx_forward: null workspace");
  const KindOps* ops = ops_of(m->kind);
  if (!m->finalized) {
    m->release();
    VADX_TRY(ops->finalize(m));
    m->finalized = true;
  }
  if (n_streams == 0) return VADX_OK;
  return ops->run(m, false, d_inputs, d_outputs, d_state, n_streams, n_samples, d_workspace, workspace_bytes, nullptr,
                  (cudaStream_t)stream);
}
