// postproc.cu -- on-device post-processing state machines (a15).
//
// One stream per lane, strictly sequential in time: the reference smooths with a float32
// np.cumsum (a sequential running sum) and thresholds the result, so a tree scan would flip
// decisions at ties.  Every arithmetic step below reproduces one numpy float32 operation of
// FireRedVAD/Inference_FireRed_ONNX.py:181-304 (MarbleNet copy:
// NVIDIA_*/Inference_NVIDIA_MarbleNet_VAD_ONNX.py:160-353).
#include "hysteresis.cuh"

namespace vadx {

constexpr int kMaxSmooth = 64;

// One warp = 32 streams.  The decision arrays of the warp's streams live in shared memory
// (byte-interleaved by lane: dec(t) of lane l at sdec[t*32 + l], conflict-free), so the back-fill,
// merge, dilation and split passes never touch global memory; probabilities are pulled through the
// read-only path, decisions are written back once at the end.
__global__ void __launch_bounds__(32) postprocess_frames_kernel(const float* __restrict__ probs, int64_t ld_probs,
                                                                const int32_t* __restrict__ n_frames_per_stream,
                                                                int64_t n_streams, int n_frames_max,
                                                                const vadx_post_cfg cfg, int8_t* __restrict__ dec_all,
                                                                int32_t* __restrict__ seg_count,
                                                                int32_t* __restrict__ segments, int max_segments,
                                                                int use_smem) {
  extern __shared__ int8_t sdec[];
  const int lane = threadIdx.x;
  const int64_t s = (int64_t)blockIdx.x * 32 + lane;
  if (s >= n_streams) return;
  int n = n_frames_per_stream ? n_frames_per_stream[s] : n_frames_max;
  if (n > n_frames_max) n = n_frames_max;
  if (n < 0) n = 0;
  const float* p = probs + s * ld_probs;
  int8_t* gdec = dec_all + s * (int64_t)n_frames_max;
  // dec(t): shared (stride 32, offset lane) or global (stride 1)
  int8_t* dec = use_smem ? sdec + lane : gdec;
  const int ds = use_smem ? 32 : 1;
  const int ws = cfg.smooth_window < 1 ? 1 : cfg.smooth_window;
  const float thr = cfg.threshold;
  const int min_sp = cfg.min_speech_frame, min_si = cfg.min_silence_frame;
  const float inv_ws = (float)(1.0 / (double)ws);

  // ---- smoothing + threshold + 4-state machine (:181-233) ----
  float ring[kMaxSmooth + 1];  // running sums cumsum[i+1-ws .. i+1]
  float run = 0.f;
  ring[0] = 0.f;
  const bool plain = (min_sp <= 0 && min_si <= 0);
  int state = 0, speech_start = 0, silence_start = 0;  // 0 SIL, 1 POSSIBLE_SPEECH, 2 SPEECH, 3 POSSIBLE_SILENCE
  for (int t = 0; t < n; ++t) {
    float sm;
    const float pt = __ldg(p + t);
    if (ws > 1) {
      run = __fadd_rn(run, pt);             // cumsum[t+1]
      ring[(t + 1) % (ws + 1)] = run;
      if (t < ws - 1) sm = __fdiv_rn(run, (float)(t + 1));
      else sm = __fmul_rn(__fsub_rn(run, ring[(t + 1 - ws) % (ws + 1)]), inv_ws);
    } else {
      sm = pt;
    }
    const bool hot = sm >= thr;
    if (plain) {
      dec[t * ds] = hot ? 1 : 0;
      continue;
    }
    if (state == 0) {
      if (hot) { state = 1; speech_start = t; }
    } else if (state == 1) {
      if (hot) {
        if (t - speech_start >= min_sp) {
          state = 2;
          for (int j = speech_start; j < t; ++j) dec[j * ds] = 1;
        }
      } else {
        state = 0;
      }
    } else if (state == 2) {
      if (!hot) { state = 3; silence_start = t; }
    } else {
      if (!hot) {
        if (t - silence_start >= min_si) state = 0;
      } else {
        state = 2;
      }
    }
    dec[t * ds] = state >= 2 ? 1 : 0;
  }

  // ---- rising edges move left by ws (:235-243) ----
  if (ws > 1) {
    for (int t = 1; t < n; ++t) {
      if (dec[t * ds] == 1 && dec[(t - 1) * ds] == 0) {
        int start = t >= ws ? t - ws : 0;
        for (int j = start; j < t; ++j) dec[j * ds] = 1;
      }
    }
  }
  // ---- short gaps are filled (:245-257) ----
  if (cfg.merge_silence_frame > 0) {
    int gap = -1;
    for (int t = 1; t < n; ++t) {
      int a = dec[(t - 1) * ds], b = dec[t * ds];
      if (a == 1 && b == 0 && gap < 0) {
        gap = t;
      } else if (a == 0 && b == 1 && gap >= 0) {
        if (t - gap < cfg.merge_silence_frame)
          for (int j = gap; j < t; ++j) dec[j * ds] = 1;
        gap = -1;
      }
    }
  }
  // ---- dilation (:259-277) ----
  if (cfg.extend_speech_frame > 0) {
    const int ext = cfg.extend_speech_frame;
    int dist = ext + 1;
    for (int t = 0; t < n; ++t) {
      if (dec[t * ds]) dist = 0;
      else if (++dist <= ext) dec[t * ds] = 1;
    }
    dist = ext + 1;
    for (int t = n - 1; t >= 0; --t) {
      if (dec[t * ds]) dist = 0;
      else if (++dist <= ext) dec[t * ds] = 1;
    }
  }
  // ---- split over-long runs at the least likely frame of the back half (:279-304) ----
  {
    const int max_sf = cfg.max_speech_frame, half = cfg.max_speech_frame >> 1;
    int t = 0;
    while (t < n) {
      if (!dec[t * ds]) { ++t; continue; }
      int seg_start = t;
      while (t < n && dec[t * ds]) ++t;
      if (t - seg_start > max_sf) {
        int pos = seg_start;
        const int seg_end = t;
        while (pos + max_sf < seg_end) {
          int a = pos + half, b = pos + max_sf;
          if (b > seg_end) b = seg_end;
          if (a >= b) break;
          int arg = a;
          float best = __ldg(p + a);
          for (int j = a + 1; j < b; ++j) {
            float v = __ldg(p + j);
            if (v < best) { best = v; arg = j; }
          }
          dec[arg * ds] = 0;
          pos = arg + 1;
        }
      }
    }
  }
  // ---- edges -> (start, end) frame pairs (decision_to_segment :146-166) + decisions out ----
  int count = 0;
  int32_t* seg = segments ? segments + s * (int64_t)max_segments * 2 : nullptr;
  int prev = 0, start = 0;
  for (int t = 0; t <= n; ++t) {
    int cur = t < n ? dec[t * ds] : 0;
    if (use_smem && t < n) gdec[t] = (int8_t)cur;
    if (cur && !prev) start = t;
    if (!cur && prev) {
      if (seg && count < max_segments) { seg[2 * count] = start; seg[2 * count + 1] = t; }
      ++count;
    }
    prev = cur;
  }
  if (seg_count) seg_count[s] = count;
}


// Warp-per-stream variant (the default whenever a stream's frames fit in shared memory): lanes load
// the probabilities coalesced, lane 0 forms the float32 running sum in order (the only truly
// sequential float arithmetic), ALL lanes evaluate the smoothed value and the threshold test for
// their frames in parallel from that running sum (each is one subtraction + one multiply of
// already-rounded operands, so the result is bit-identical to numpy's), lane 0 then walks the
// integer state machines over shared memory, and all lanes write the decisions back coalesced.
// One stream per warp means no lane divergence in the sequential part.
constexpr int kPpWarps = 4;
__global__ void __launch_bounds__(kPpWarps * 32) postprocess_frames_warp_kernel(
    const float* __restrict__ probs, int64_t ld_probs, const int32_t* __restrict__ n_frames_per_stream,
    int64_t n_streams, int n_frames_max, const vadx_post_cfg cfg, int8_t* __restrict__ dec_all,
    int32_t* __restrict__ seg_count, int32_t* __restrict__ segments, int max_segments, int per_warp_floats) {
  extern __shared__ float smem_f[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t s = (int64_t)blockIdx.x * kPpWarps + warp;
  if (s >= n_streams) return;
  int n = n_frames_per_stream ? n_frames_per_stream[s] : n_frames_max;
  if (n > n_frames_max) n = n_frames_max;
  if (n < 0) n = 0;
  float* sp = smem_f + (size_t)warp * per_warp_floats;   // probs [n_frames_max]
  float* cs = sp + n_frames_max;                          // running sums [n_frames_max + 1]
  int8_t* dec = reinterpret_cast<int8_t*>(cs + n_frames_max + 1);
  const float* p = probs + s * ld_probs;
  int8_t* gdec = dec_all + s * (int64_t)n_frames_max;
  const int ws = cfg.smooth_window < 1 ? 1 : cfg.smooth_window;
  const float thr = cfg.threshold;
  const int min_sp = cfg.min_speech_frame, min_si = cfg.min_silence_frame;
  const float inv_ws = (float)(1.0 / (double)ws);

  for (int t = lane; t < n; t += 32) sp[t] = __ldg(p + t);
  __syncwarp();
  if (ws > 1) {
    if (lane == 0) {
      float run = 0.f;
      cs[0] = 0.f;
      for (int t = 0; t < n; ++t) {
        run = __fadd_rn(run, sp[t]);
        cs[t + 1] = run;
      }
    }
    __syncwarp();
  }
  for (int t = lane; t < n; t += 32) {
    float sm;
    if (ws > 1) {
      if (t < ws - 1) sm = __fdiv_rn(cs[t + 1], (float)(t + 1));
      else sm = __fmul_rn(__fsub_rn(cs[t + 1], cs[t + 1 - ws]), inv_ws);
    } else {
      sm = sp[t];
    }
    dec[t] = sm >= thr ? 1 : 0;   // "hot" flags; turned into decisions in place below
  }
  __syncwarp();
  int count = 0;
  if (lane == 0) {
    if (!(min_sp <= 0 && min_si <= 0)) {
      int state = 0, speech_start = 0, silence_start = 0;
      for (int t = 0; t < n; ++t) {
        const bool hot = dec[t] != 0;
        if (state == 0) {
          if (hot) { state = 1; speech_start = t; }
        } else if (state == 1) {
          if (hot) {
            if (t - speech_start >= min_sp) {
              state = 2;
              for (int j = speech_start; j < t; ++j) dec[j] = 1;
            }
          } else {
            state = 0;
          }
        } else if (state == 2) {
          if (!hot) { state = 3; silence_start = t; }
        } else {
          if (!hot) {
            if (t - silence_start >= min_si) state = 0;
          } else {
            state = 2;
          }
        }
        dec[t] = state >= 2 ? 1 : 0;
      }
    }
    if (ws > 1) {
      for (int t = 1; t < n; ++t) {
        if (dec[t] == 1 && dec[t - 1] == 0) {
          int start = t >= ws ? t - ws : 0;
          for (int j = start; j < t; ++j) dec[j] = 1;
        }
      }
    }
    if (cfg.merge_silence_frame > 0) {
      int gap = -1;
      for (int t = 1; t < n; ++t) {
        int a = dec[t - 1], b = dec[t];
        if (a == 1 && b == 0 && gap < 0) {
          gap = t;
        } else if (a == 0 && b == 1 && gap >= 0) {
          if (t - gap < cfg.merge_silence_frame)
            for (int j = gap; j < t; ++j) dec[j] = 1;
          gap = -1;
        }
      }
    }
    if (cfg.extend_speech_frame > 0) {
      const int ext = cfg.extend_speech_frame;
      int dist = ext + 1;
      for (int t = 0; t < n; ++t) {
        if (dec[t]) dist = 0;
        else if (++dist <= ext) dec[t] = 1;
      }
      dist = ext + 1;
      for (int t = n - 1; t >= 0; --t) {
        if (dec[t]) dist = 0;
        else if (++dist <= ext) dec[t] = 1;
      }
    }
    {
      const int max_sf = cfg.max_speech_frame, half = cfg.max_speech_frame >> 1;
      int t = 0;
      while (t < n) {
        if (!dec[t]) { ++t; continue; }
        int seg_start = t;
        while (t < n && dec[t]) ++t;
        if (t - seg_start > max_sf) {
          int pos = seg_start;
          const int seg_end = t;
          while (pos + max_sf < seg_end) {
            int a = pos + half, b = pos + max_sf;
            if (b > seg_end) b = seg_end;
            if (a >= b) break;
            int arg = a;
            float best = sp[a];
            for (int j = a + 1; j < b; ++j)
              if (sp[j] < best) { best = sp[j]; arg = j; }
            dec[arg] = 0;
            pos = arg + 1;
          }
        }
      }
    }
    int32_t* seg = segments ? segments + s * (int64_t)max_segments * 2 : nullptr;
    int prev = 0, start = 0;
    for (int t = 0; t <= n; ++t) {
      int cur = t < n ? dec[t] : 0;
      if (cur && !prev) start = t;
      if (!cur && prev) {
        if (seg && count < max_segments) { seg[2 * count] = start; seg[2 * count + 1] = t; }
        ++count;
      }
      prev = cur;
    }
    if (seg_count) seg_count[s] = count;
  }
  __syncwarp();
  for (int t = lane; t < n; t += 32) gdec[t] = dec[t];
}

// ---- run-based variant of the warp-per-stream kernel ----
// Same results, different cost model: after the (inherently sequential) float32 running sum, the frame
// flags become a bit mask (__ballot_sync) and the state machines advance from run to run with
// find-first-set instead of frame by frame.  The 4-state machine, the window extension of rising edges,
// the gap merge and the dilation are closed-form on (start, end) pairs:
//   * a speech segment opens at the first frame a of a run of flags that stays set through frame
//     a + max(min_speech, 1) (the reference back-fills to a, :196-204);
//   * it closes at e = b + max(min_silence, 1), b the first cleared frame after which the flags stay
//     clear through e (possible-silence frames count as speech, :209-221), or at the end of the stream;
//   * every segment that does not start at frame 0 grows left by the smoothing window (:235-243),
//     gaps shorter than merge_silence close (:245-257), extend_speech dilates both ways (:259-277);
//   * max_speech splitting at the first minimum of the raw probabilities in the second half of the
//     window (:279-304) is done while the final pairs are emitted, the arg-min by all lanes.
// Every lane executes the same control flow on the same shared data (no divergence), lane 0 writes.
__device__ __forceinline__ int pp_next_set(const uint32_t* w, int t, int n) {
  if (t >= n) return n;
  const int nw = (n + 31) >> 5;
  int wi = t >> 5;
  uint32_t cur = w[wi] & (0xffffffffu << (t & 31));
  while (!cur) {
    if (++wi >= nw) return n;
    cur = w[wi];
  }
  const int r = (wi << 5) + __ffs(cur) - 1;
  return r < n ? r : n;
}
__device__ __forceinline__ int pp_next_clear(const uint32_t* w, int t, int n) {
  if (t >= n) return n;
  const int nw = (n + 31) >> 5;
  int wi = t >> 5;
  uint32_t cur = ~w[wi] & (0xffffffffu << (t & 31));
  while (!cur) {
    if (++wi >= nw) return n;
    cur = ~w[wi];
  }
  const int r = (wi << 5) + __ffs(cur) - 1;
  return r < n ? r : n;
}

__global__ void __launch_bounds__(kPpWarps * 32) postprocess_frames_runs_kernel(
    const float* __restrict__ probs, int64_t ld_probs, const int32_t* __restrict__ n_frames_per_stream,
    int64_t n_streams, int n_frames_max, const vadx_post_cfg cfg, int8_t* __restrict__ dec_all,
    int32_t* __restrict__ seg_count, int32_t* __restrict__ segments, int max_segments, int per_warp_floats) {
  extern __shared__ float smem_f[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t s = (int64_t)blockIdx.x * kPpWarps + warp;
  if (s >= n_streams) return;
  int n = n_frames_per_stream ? n_frames_per_stream[s] : n_frames_max;
  if (n > n_frames_max) n = n_frames_max;
  if (n < 0) n = 0;
  float* sp = smem_f + (size_t)warp * per_warp_floats;     // probs [n_frames_max]
  float* cs = sp + n_frames_max;                            // running sums [n_frames_max + 1], then the pairs
  int* pairs = reinterpret_cast<int*>(cs);                  // (start, end) x up to (n + 1) / 2
  int8_t* dec = reinterpret_cast<int8_t*>(cs + n_frames_max + 1);
  uint32_t* hot = reinterpret_cast<uint32_t*>(dec + ((n_frames_max + 3) & ~3));
  const float* p = probs + s * ld_probs;
  int8_t* gdec = dec_all + s * (int64_t)n_frames_max;
  const int ws = cfg.smooth_window < 1 ? 1 : cfg.smooth_window;
  const float thr = cfg.threshold;
  const int min_sp = cfg.min_speech_frame, min_si = cfg.min_silence_frame;
  const float inv_ws = (float)(1.0 / (double)ws);

  for (int t = lane; t < n; t += 32) sp[t] = __ldg(p + t);
  __syncwarp();
  if (ws > 1) {
    if (lane == 0) {
      float run = 0.f;
      cs[0] = 0.f;
      int t = 0;
      for (; t + 4 <= n; t += 4) {   // four independent loads per trip; the additions stay in order
        const float a = sp[t], b = sp[t + 1], c = sp[t + 2], d = sp[t + 3];
        run = __fadd_rn(run, a); cs[t + 1] = run;
        run = __fadd_rn(run, b); cs[t + 2] = run;
        run = __fadd_rn(run, c); cs[t + 3] = run;
        run = __fadd_rn(run, d); cs[t + 4] = run;
      }
      for (; t < n; ++t) { run = __fadd_rn(run, sp[t]); cs[t + 1] = run; }
    }
    __syncwarp();
  }
  for (int t0 = 0; t0 < n; t0 += 32) {
    const int t = t0 + lane;
    bool h = false;
    if (t < n) {
      float sm;
      if (ws > 1) {
        if (t < ws - 1) sm = __fdiv_rn(cs[t + 1], (float)(t + 1));
        else sm = __fmul_rn(__fsub_rn(cs[t + 1], cs[t + 1 - ws]), inv_ws);
      } else {
        sm = sp[t];
      }
      h = sm >= thr;
    }
    const uint32_t word = __ballot_sync(0xffffffffu, h);
    if (lane == 0) hot[t0 >> 5] = word;
    if (t < n) dec[t] = 0;
  }
  __syncwarp();   // cs is dead from here: its storage becomes the pair list

  // ---- pass A: flags -> speech segments (all lanes, same control flow) ----
  int ns = 0;
  auto push = [&](int a, int e) {
    if (lane == 0) { pairs[2 * ns] = a; pairs[2 * ns + 1] = e; }
    ++ns;
  };
  if (min_sp <= 0 && min_si <= 0) {
    int t = 0;
    while (t < n) {
      const int a = pp_next_set(hot, t, n);
      if (a >= n) break;
      const int e = pp_next_clear(hot, a + 1, n);
      push(a, e);
      t = e;
    }
  } else {
    const int need_sp = min_sp > 1 ? min_sp : 1, need_si = min_si > 1 ? min_si : 1;
    int t = 0;
    while (t < n) {
      const int a = pp_next_set(hot, t, n);
      if (a >= n) break;
      const int b = pp_next_clear(hot, a + 1, n);
      if (a + need_sp >= b) { t = b; continue; }          // the run ends before speech is confirmed
      int cur = b, e;
      while (true) {
        if (cur >= n) { e = n; break; }
        const int c = pp_next_set(hot, cur + 1, n);
        const int lim = cur + need_si;
        if (lim < c && lim < n) { e = lim; break; }        // silence confirmed at frame lim
        if (c >= n) { e = n; break; }                      // the stream ends inside possible silence
        cur = pp_next_clear(hot, c + 1, n);
      }
      push(a, e);
      t = e;
    }
  }
  __syncwarp();
  // ---- passes B-D on the pair list, in place (each pass only ever shrinks the list) ----
  auto sweep = [&](int grow_left, int grow_left_skip0, int grow_right, int merge_below) {
    // grow every pair, then fuse pairs that touch/overlap or whose gap is < merge_below
    int m = 0, pa = 0, pe = 0;
    for (int k = 0; k < ns; ++k) {
      int a = pairs[2 * k], e = pairs[2 * k + 1];
      if (!(grow_left_skip0 && a == 0)) a = a - grow_left < 0 ? 0 : a - grow_left;
      e = e + grow_right > n ? n : e + grow_right;
      if (m > 0 && (a <= pe || a - pe < merge_below)) {
        if (e > pe) pe = e;
      } else {
        if (m > 0) {
          __syncwarp();
          if (lane == 0) { pairs[2 * (m - 1)] = pa; pairs[2 * (m - 1) + 1] = pe; }
        }
        pa = a; pe = e; ++m;
      }
    }
    __syncwarp();
    if (m > 0 && lane == 0) { pairs[2 * (m - 1)] = pa; pairs[2 * (m - 1) + 1] = pe; }
    __syncwarp();
    ns = m;
  };
  if (ws > 1) sweep(ws, 1, 0, 0);
  if (cfg.merge_silence_frame > 0) sweep(0, 0, 0, cfg.merge_silence_frame);
  if (cfg.extend_speech_frame > 0) sweep(cfg.extend_speech_frame, 0, cfg.extend_speech_frame, 0);

  // ---- pass E + emission: split long segments, write pairs, rasterise the decisions ----
  int count = 0;
  int32_t* seg = segments ? segments + s * (int64_t)max_segments * 2 : nullptr;
  auto emit = [&](int a, int e) {
    if (e <= a) return;
    if (lane == 0 && seg && count < max_segments) { seg[2 * count] = a; seg[2 * count + 1] = e; }
    ++count;
    for (int t = a + lane; t < e; t += 32) dec[t] = 1;
  };
  const int max_sf = cfg.max_speech_frame, half = cfg.max_speech_frame >> 1;
  for (int k = 0; k < ns; ++k) {
    const int a0 = pairs[2 * k], e0 = pairs[2 * k + 1];
    int pos = a0;
    if (e0 - a0 > max_sf) {
      while (pos + max_sf < e0) {
        const int lo = pos + half, hi = pos + max_sf;     // hi < e0
        if (lo >= hi) break;
        float best = INFINITY;
        int arg = 0x7fffffff;
        for (int j = lo + lane; j < hi; j += 32) {
          const float v = sp[j];
          if (v < best) { best = v; arg = j; }            // strided scan keeps the lowest index per lane
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, best, off);
          const int oa = __shfl_xor_sync(0xffffffffu, arg, off);
          if (ov < best || (ov == best && oa < arg)) { best = ov; arg = oa; }
        }
        emit(pos, arg);
        pos = arg + 1;
      }
    }
    emit(pos, e0);
  }
  if (lane == 0 && seg_count) seg_count[s] = count;
  __syncwarp();
  for (int t = lane; t < n; t += 32) gdec[t] = dec[t];
}

// ---- Stream-VAD segmenter (FireRedVAD/Inference_FireRed_ONNX.py:307-490) ----
// state words per stream: 0 head, 1 fill, 2 frame (1-based, last consumed), 3 mode, 4 speech run, 5 silence run,
// 6 re-arm flag, 7 first frame of the open segment (0 = none), 8 last frame of the latest closed segment
// (0 = none), 9 ring sum (float bits), 10..11 samples consumed (int64, low word first; the slot server's
// counter, stream_serve_seg_kernel), 12..15 spare, 16.. ring of smooth_window floats.
constexpr int kSpHeader = 16;

// One stream's segmenter state in registers (the ring in local memory); load / store move it from / to its state words.
struct SpState {
  float ring[kMaxSmooth];
  int head, fill, frame, mode, n_sp, n_si, open_from, closed_at;
  bool rearm;
  float acc;

  __device__ __forceinline__ void load(const int32_t* st, int ws) {
    for (int i = 0; i < ws; ++i) ring[i] = __int_as_float(st[kSpHeader + i]);
    head = st[0]; fill = st[1]; frame = st[2]; mode = st[3]; n_sp = st[4]; n_si = st[5];
    rearm = st[6] != 0;
    open_from = st[7]; closed_at = st[8];
    acc = __int_as_float(st[9]);
  }
  __device__ __forceinline__ void store(int32_t* st, int ws) const {
    st[0] = head; st[1] = fill; st[2] = frame; st[3] = mode; st[4] = n_sp; st[5] = n_si; st[6] = rearm ? 1 : 0;
    st[7] = open_from; st[8] = closed_at; st[9] = __float_as_int(acc);
    for (int i = 0; i < ws; ++i) st[kSpHeader + i] = __float_as_int(ring[i]);
  }
};

// One frame of the segmenter.  On return (all 1-based, 0 = not set): `opened` is the first frame of a segment
// the segmenter confirmed on this frame; a segment closed on this frame iff begin > 0 && end > 0, and is
// [begin, end].  At most one segment opens and at most one closes per frame; when both happen the open comes first.
__device__ __forceinline__ void sp_frame(SpState& g, float pt, const vadx_stream_post_cfg& cfg, int ws, int pad,
                                         int& opened, int& begin, int& end) {
  ++g.frame;
  float sm = pt;
  if (ws > 1) {
    const float gone = g.ring[g.head];
    g.ring[g.head] = pt;
    g.acc = __fadd_rn(g.acc, __fsub_rn(pt, gone));
    g.head = g.head + 1 == ws ? 0 : g.head + 1;
    if (g.fill < ws) ++g.fill;
    sm = __fdiv_rn(g.acc, (float)g.fill);
  }
  const bool speech = sm >= cfg.threshold;
  opened = begin = end = 0;
  bool force_close = false;
  if (g.rearm) { opened = begin = g.open_from = g.frame; g.rearm = false; }
  if (g.mode == 0) {
    if (speech) { g.mode = 1; g.n_sp = 1; }
    else { ++g.n_si; g.n_sp = 0; }
  } else if (g.mode == 1) {
    if (speech) {
      if (++g.n_sp >= cfg.min_speech_frame) {
        g.mode = 2;
        int b = g.frame - g.n_sp + 1 - pad;
        if (b < 1) b = 1;
        if (b < g.closed_at + 1) b = g.closed_at + 1;
        opened = begin = g.open_from = b;
        g.n_si = 0;
      }
    } else { g.mode = 0; g.n_si = 1; g.n_sp = 0; }
  } else if (g.mode == 2) {
    ++g.n_sp;
    if (speech) { g.n_si = 0; force_close = g.n_sp >= cfg.max_speech_frame; }
    else { g.mode = 3; g.n_si = 1; }
  } else {
    ++g.n_sp;
    if (speech) { g.mode = 2; g.n_si = 0; force_close = g.n_sp >= cfg.max_speech_frame; }
    else if (++g.n_si >= cfg.min_silence_frame) {
      g.mode = 0;
      begin = g.open_from; end = g.frame;
      g.open_from = 0; g.closed_at = g.frame; g.n_sp = 0;
    }
  }
  if (force_close) {
    g.rearm = true;
    g.n_sp = 0;
    begin = g.open_from; end = g.frame;
    g.open_from = 0; g.closed_at = g.frame;
  }
}

__global__ void __launch_bounds__(128) stream_post_kernel(const float* __restrict__ probs, int64_t ld_probs,
                                                          const int32_t* __restrict__ n_frames_per_stream,
                                                          int64_t n_streams, int n_frames_max,
                                                          const vadx_stream_post_cfg cfg, int32_t* __restrict__ state,
                                                          int32_t* __restrict__ seg_count,
                                                          int32_t* __restrict__ segments, int max_segments,
                                                          int32_t* __restrict__ open_seg) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_streams) return;
  int n = n_frames_per_stream ? n_frames_per_stream[s] : n_frames_max;
  n = n < 0 ? 0 : (n > n_frames_max ? n_frames_max : n);
  const int ws = cfg.smooth_window < 1 ? 1 : cfg.smooth_window;
  const int pad = cfg.pad_start_frame > ws ? cfg.pad_start_frame : ws;
  int32_t* st = state + s * (int64_t)(kSpHeader + ws);
  SpState g;
  g.load(st, ws);
  int count = seg_count ? seg_count[s] : 0;
  int32_t* seg = segments ? segments + s * (int64_t)max_segments * 2 : nullptr;
  const float* p = probs + s * ld_probs;
  for (int t = 0; t < n; ++t) {
    int opened, begin, end;
    sp_frame(g, __ldg(p + t), cfg, ws, pad, opened, begin, end);
    if (begin > 0 && end > 0) {
      if (seg && count < max_segments) { seg[2 * count] = begin - 1; seg[2 * count + 1] = end - 1; }
      ++count;
    }
  }
  g.store(st, ws);
  if (seg_count) seg_count[s] = count;
  if (open_seg) {
    open_seg[2 * s] = g.open_from > 0 ? g.open_from - 1 : -1;
    open_seg[2 * s + 1] = g.open_from > 0 ? g.frame - 1 : -1;
  }
}

// ---- Stream-VAD slot server (vadx_stream_serve_step) ----
// Per slot and tick: an action (what happens to the slot's caches) and up to 2*T + 1 staged events.
constexpr int kServeThreads = 128;
enum : int8_t { kServeAdvance = 0, kServeHold = 1, kServeFinalize = 2 };

// The control-word rule of every slot server: n outside [0, full] is out of range, and a chunk shorter than full must
// be the stream's last.  Returns the slot's VADX_SERVE_ERR_* bits (0: the words are valid).
__device__ __forceinline__ int serve_control_error(int n, bool fin, int full) {
  return (n < 0 || n > full) ? VADX_SERVE_ERR_RANGE : (n > 0 && n < full && !fin) ? VADX_SERVE_ERR_SHORT : 0;
}

// Zero samples [n, frame_len) of every slot fed a short chunk: a chunk shorter than one frame is zero-padded to
// one frame (the reference's np.pad, Inference_FireRed_ONNX.py:790-792); later frames of a short chunk lie wholly
// inside its n samples, and whatever lies past them only reaches frames the server discards.
__global__ void __launch_bounds__(256) stream_serve_tail_kernel(int16_t* __restrict__ chunk, int64_t ld_chunk,
                                                                const int32_t* __restrict__ n_samples,
                                                                int64_t n_slots, int chunk_samples, int frame_len) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t s = i / frame_len;
  const int k = (int)(i - s * frame_len);
  if (s >= n_slots) return;
  const int n = n_samples[s];
  if (n > 0 && n < frame_len && k >= n && k < chunk_samples) chunk[s * ld_chunk + k] = 0;
}

// Block totals of a serve segmenter kernel: warp sums, then the first warp adds the four.  Every thread of the block
// calls this (threads past n_slots with count = err = 0).
__device__ __forceinline__ void serve_block_totals(int count, int err, int32_t* __restrict__ block_info) {
  __shared__ int wsum[kServeThreads / 32], werr[kServeThreads / 32];
  int c = count, e = err;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    c += __shfl_xor_sync(0xffffffffu, c, off);
    e |= __shfl_xor_sync(0xffffffffu, e, off);
  }
  if ((threadIdx.x & 31) == 0) { wsum[threadIdx.x >> 5] = c; werr[threadIdx.x >> 5] = e; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int tc = 0, te = 0;
    for (int w = 0; w < kServeThreads / 32; ++w) { tc += wsum[w]; te |= werr[w]; }
    block_info[2 * blockIdx.x] = tc;
    block_info[2 * blockIdx.x + 1] = te;
  }
}

// Thread per slot: validate the slot's control words, run the segmenter over this tick's frames, stage the events
// slot-major in `staged` [S][2T+1] (kind, frame) and count them.  Each block writes its event total and its error
// bits to block_info[2b], [2b+1]; stream_serve_emit_kernel turns those into offsets.  No atomics anywhere.
__global__ void __launch_bounds__(kServeThreads) stream_serve_seg_kernel(
    const float* __restrict__ probs, int64_t ld_probs, int n_frames_max, const int32_t* __restrict__ n_samples,
    const uint8_t* __restrict__ last, int64_t n_slots, int chunk_samples, int frame_len, int frame_hop,
    const vadx_stream_post_cfg cfg, int32_t* __restrict__ state, int32_t* __restrict__ frames_out,
    int32_t* __restrict__ staged, int32_t* __restrict__ counts, int8_t* __restrict__ action,
    int32_t* __restrict__ block_info) {
  const int64_t s = (int64_t)blockIdx.x * kServeThreads + threadIdx.x;
  int count = 0, err = 0;
  if (s < n_slots) {
    const int n = n_samples[s];
    const bool fin = last[s] != 0;
    err = serve_control_error(n, fin, chunk_samples);
    int f = 0;
    if (err || (n == 0 && !fin)) {
      action[s] = kServeHold;                       // hold, or a rejected tick: the slot stays exactly as it was
    } else {
      const int ws = cfg.smooth_window < 1 ? 1 : cfg.smooth_window;
      const int pad = cfg.pad_start_frame > ws ? cfg.pad_start_frame : ws;
      int32_t* st = state + s * (int64_t)(kSpHeader + ws);
      SpState g;
      g.load(st, ws);
      // frames of this chunk, cut at valid_frame_count(samples so far + n) (firered_vad.stream_frame_plan)
      const int64_t total = ((int64_t)(uint32_t)st[10] | ((int64_t)st[11] << 32)) + n;
      const int64_t valid = total < frame_len ? 0 : 1 + (total - frame_len) / frame_hop;
      f = n == 0 ? 0 : (n < frame_len ? 1 : 1 + (n - frame_len) / frame_hop);
      if (f > n_frames_max) f = n_frames_max;
      if ((int64_t)f > valid - g.frame) f = (int)max((int64_t)0, valid - g.frame);
      const int cap = 2 * n_frames_max + 1;
      int2* ev = reinterpret_cast<int2*>(staged) + s * cap;
      const float* p = probs + s * ld_probs;
      for (int t = 0; t < f; ++t) {
        int opened, begin, end;
        sp_frame(g, __ldg(p + t), cfg, ws, pad, opened, begin, end);
        if (opened > 0) ev[count++] = make_int2(VADX_SERVE_START, opened - 1);
        if (begin > 0 && end > 0) ev[count++] = make_int2(VADX_SERVE_END, end - 1);
      }
      if (fin) {
        if (g.open_from > 0) ev[count++] = make_int2(VADX_SERVE_END_OF_STREAM, g.frame - 1);
        for (int i = 0; i < kSpHeader + ws; ++i) st[i] = 0;     // the next stream in this slot starts fresh
        action[s] = kServeFinalize;
      } else {
        g.store(st, ws);
        st[10] = (int32_t)(uint32_t)total;
        st[11] = (int32_t)(total >> 32);
        action[s] = kServeAdvance;
      }
    }
    frames_out[s] = f;
    counts[s] = count;
  }
  serve_block_totals(count, err, block_info);
}

// Blocks [0, n_seg_blocks): compact the staged events of their 128 slots to events [n][3] (slot, kind, frame) at
// offset = events of all earlier blocks + events of earlier slots in the block; the last of them writes the header
// {n_events, error bits}.  Every event and the header also go to the host mirror when one is given (pinned host memory,
// written through unified addressing).  Blocks [n_seg_blocks, n_seg_blocks + S): slot blockIdx - n_seg_blocks applies
// its action to the caches: hold copies its caches_in rows to caches_out, finalize zeroes its caches_out rows.
__global__ void __launch_bounds__(kServeThreads) stream_serve_emit_kernel(
    int64_t n_slots, int n_seg_blocks, int cap, const int32_t* __restrict__ staged, const int32_t* __restrict__ counts,
    const int8_t* __restrict__ action, const int32_t* __restrict__ block_info, int32_t* __restrict__ events,
    int32_t* __restrict__ header, int32_t* __restrict__ h_events, int32_t* __restrict__ h_header,
    const float* __restrict__ caches_in, float* __restrict__ caches_out, int n_cache_blocks, int64_t cache_row) {
  __shared__ int red[kServeThreads / 32][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if ((int)blockIdx.x >= n_seg_blocks) {
    const int64_t s = blockIdx.x - n_seg_blocks;
    const int8_t a = action[s];
    if (a == kServeAdvance || !caches_out) return;
    for (int r = 0; r < n_cache_blocks; ++r) {
      const int64_t base = ((int64_t)r * n_slots + s) * cache_row;
      if (a == kServeHold)
        for (int64_t i = threadIdx.x; i < cache_row; i += kServeThreads) caches_out[base + i] = caches_in[base + i];
      else
        for (int64_t i = threadIdx.x; i < cache_row; i += kServeThreads) caches_out[base + i] = 0.0f;
    }
    return;
  }
  const int b = blockIdx.x;
  // events and error bits of every earlier block (the last block also adds its own for the header)
  int before = 0, err = 0;
  const int upto = b == n_seg_blocks - 1 ? n_seg_blocks : b;
  for (int i = threadIdx.x; i < upto; i += kServeThreads) {
    if (i < b) before += block_info[2 * i];
    err |= block_info[2 * i + 1];
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    before += __shfl_xor_sync(0xffffffffu, before, off);
    err |= __shfl_xor_sync(0xffffffffu, err, off);
  }
  if (lane == 0) { red[warp][0] = before; red[warp][1] = err; }
  __syncthreads();
  before = 0; err = 0;
  for (int w = 0; w < kServeThreads / 32; ++w) { before += red[w][0]; err |= red[w][1]; }
  __syncthreads();
  // exclusive scan of the slot counts within the block
  const int64_t s = (int64_t)b * kServeThreads + threadIdx.x;
  const int c = s < n_slots ? counts[s] : 0;
  int incl = c;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += v;
  }
  if (lane == 31) red[warp][0] = incl;
  __syncthreads();
  int at = before + incl - c;
  for (int w = 0; w < warp; ++w) at += red[w][0];
  if (c > 0) {
    const int2* ev = reinterpret_cast<const int2*>(staged) + s * cap;
    for (int j = 0; j < c; ++j) {
      const int2 e = ev[j];
      int32_t* o = events + 3 * (int64_t)(at + j);
      o[0] = (int32_t)s; o[1] = e.x; o[2] = e.y;
      if (h_events) {
        int32_t* h = h_events + 3 * (int64_t)(at + j);
        h[0] = (int32_t)s; h[1] = e.x; h[2] = e.y;
      }
    }
  }
  if (b == n_seg_blocks - 1 && threadIdx.x == kServeThreads - 1) {
    int total = before;
    for (int w = 0; w < kServeThreads / 32; ++w) total += red[w][0];
    header[0] = total; header[1] = err;
    if (h_header) { h_header[0] = total; h_header[1] = err; }
  }
}

// ---- Silero slot server (vadx_silero_serve_load, vadx_silero_serve_step) ----
// A slot's model input row is [64 context | W*512 samples]; window w of the tick is columns [w*512, w*512 + 576).
constexpr int kSileroWindow = 512, kSileroContext = 64, kSileroHidden = 128;
constexpr int kSileroServeStateWords = 3;   // {windows so far, triggered, temp_end window + 1 (0 = none)}
constexpr int kSileroMaxWindowsPerTick = 1 << 20;   // keeps W * 512 + 64 an int
// the reference's int16 scale (Inference_Silero_VAD_ONNX.py:83); as float32 it is exactly 2^-15, so the product is exact
constexpr float kSileroInt16Scale = 0.000030517578f;

// Thread per 8 samples: int16 chunk [S][W*512] -> scaled fp32 in columns [64, 64 + W*512) of x, zero from n on.
// The context columns 0..63 hold the slot's carried samples and are not touched.
__global__ void __launch_bounds__(256) silero_serve_load_kernel(const int16_t* __restrict__ chunk,
                                                                const int32_t* __restrict__ n_samples, int64_t n_slots,
                                                                int chunk_samples, float* __restrict__ x) {
  const int per_row = chunk_samples / 8;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t s = i / per_row;
  if (s >= n_slots) return;
  const int k0 = (int)(i - s * per_row) * 8;
  const int n = n_samples[s];
  const int4 raw = __ldg(reinterpret_cast<const int4*>(chunk + s * chunk_samples + k0));
  const int16_t* v = reinterpret_cast<const int16_t*>(&raw);
  float f[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = k0 + j < n ? (float)v[j] * kSileroInt16Scale : 0.0f;
  float4* o = reinterpret_cast<float4*>(x + s * (int64_t)(kSileroContext + chunk_samples) + kSileroContext + k0);
  o[0] = make_float4(f[0], f[1], f[2], f[3]);
  o[1] = make_float4(f[4], f[5], f[6], f[7]);
}

// Thread per slot: validate the control words (same rules and error bits as stream_serve_seg_kernel), run the
// reference VADIterator (utils_vad.py:494-585) over the slot's ceil(n/512) windows of probs [W][ld_probs], comparing
// in double as the reference compares Python floats, and stage at most W + 1 events (kind, window) in `staged`
// [S][W+1].  Then the block rolls its slots' context in x: a fed slot's last 64 samples become columns 0..63, a
// finalized slot's are zeroed, a held one's are left alone.
__global__ void __launch_bounds__(kServeThreads) silero_serve_seg_kernel(
    const float* __restrict__ probs, int64_t ld_probs, const int32_t* __restrict__ n_samples,
    const uint8_t* __restrict__ last, int64_t n_slots, int W, double threshold, double min_silence_samples,
    int32_t* __restrict__ state, float* __restrict__ x, int32_t* __restrict__ windows_out, int32_t* __restrict__ staged,
    int32_t* __restrict__ counts, int8_t* __restrict__ action, int32_t* __restrict__ block_info) {
  __shared__ int8_t s_act[kServeThreads];
  const int64_t s = (int64_t)blockIdx.x * kServeThreads + threadIdx.x;
  const int chunk_samples = W * kSileroWindow;
  int count = 0, err = 0;
  int8_t act = kServeHold;
  if (s < n_slots) {
    const int n = n_samples[s];
    const bool fin = last[s] != 0;
    err = serve_control_error(n, fin, chunk_samples);
    int nw = 0;
    if (!err && (n > 0 || fin)) {
      int32_t* st = state + s * kSileroServeStateWords;
      int cur = st[0], tend = st[2];
      bool trig = st[1] != 0;
      nw = (n + kSileroWindow - 1) / kSileroWindow;
      int2* ev = reinterpret_cast<int2*>(staged) + s * (W + 1);
      const double neg = threshold - 0.15;
      for (int w = 0; w < nw; ++w) {
        const double p = (double)__ldg(probs + w * ld_probs + s);
        const int gw = cur + w;
        if (p >= threshold) {
          tend = 0;
          if (!trig) { trig = true; ev[count++] = make_int2(VADX_SERVE_START, gw); }
        } else if (trig && p < neg) {
          if (tend == 0) tend = gw + 1;
          // current_sample - temp_end = (gw - w_t) * 512 samples
          if ((double)(gw - (tend - 1)) * kSileroWindow >= min_silence_samples) {
            ev[count++] = make_int2(VADX_SERVE_END, tend - 1);
            tend = 0;
            trig = false;
          }
        }
      }
      cur += nw;
      if (fin) {
        if (trig) ev[count++] = make_int2(VADX_SERVE_END_OF_STREAM, cur);
        st[0] = st[1] = st[2] = 0;                  // the next stream in this slot starts fresh
        act = kServeFinalize;
      } else {
        st[0] = cur; st[1] = trig ? 1 : 0; st[2] = tend;
        act = kServeAdvance;
      }
    }
    action[s] = act;
    windows_out[s] = nw;
    counts[s] = count;
  }
  s_act[threadIdx.x] = act;
  serve_block_totals(count, err, block_info);      // its barrier also publishes s_act
  if (!x) return;
  // 16 threads per row: columns 0..63 <- columns [W*512, W*512 + 64) (fed) or 0 (finalized), as float4s
  const int64_t ld_x = kSileroContext + chunk_samples;
  for (int i = threadIdx.x; i < kServeThreads * (kSileroContext / 4); i += kServeThreads) {
    const int r = i / (kSileroContext / 4), q = i % (kSileroContext / 4);
    const int64_t ss = (int64_t)blockIdx.x * kServeThreads + r;
    const int8_t a = s_act[r];
    if (ss >= n_slots || a == kServeHold) continue;
    float4* row = reinterpret_cast<float4*>(x + ss * ld_x);
    row[q] = a == kServeFinalize ? make_float4(0.0f, 0.0f, 0.0f, 0.0f) : row[chunk_samples / 4 + q];
  }
}


// ---- FSMN slot server (vadx_fsmn_serve_load, vadx_fsmn_serve_step) ----
// State words per slot: 0 samples received before the first window (chunk_len from the first window on), 1 the machine
// is out of silence (0 = silence, the reference's initial state), 2 decisions so far, 3 background level bits XOR the
// initial level's bits (0 = the initial level), 4 first decision of the open run + 1 (0 = none), 5 segment state
// (kFsmnSeg*), 6 closing decision of the pending segment's last run, 7 spare (0), 8.. the last look_backward score
// flags of the latest window, one bit each.  All zero is a fresh slot.
constexpr int kFsmnServeHeader = 8;
constexpr int kFsmnMaxChunk = 1 << 24;
enum : int { kFsmnSegNone = 0, kFsmnSegOpen = 1, kFsmnSegPending = 2 };
enum : int { kFsmnHold = 0, kFsmnFill = 1, kFsmnWindow = 2, kFsmnFlush = 3 };

__host__ __device__ __forceinline__ int fsmn_serve_words(int look_backward) { return kFsmnServeHeader + (look_backward + 31) / 32; }

// What a slot does this tick, from its control words and the samples it holds.  Until a slot has `chunk_len` samples a
// full chunk is min(stride, chunk_len - received), so no stream is carried past its first window; from then on it is
// `stride`.  kFsmnFill: samples only; kFsmnWindow: one window (the first one once chunk_len samples are in, or a
// zero-padded one at a short stream's end); kFsmnFlush: finalize without new audio after the last window (or a stream
// that never got a sample).  Load and step decide alike.
__device__ __forceinline__ int fsmn_serve_plan(int n, bool fin, int received, int chunk_len, int stride, int& err) {
  const int full = received < chunk_len ? min(stride, chunk_len - received) : stride;
  err = serve_control_error(n, fin, full);
  if (err || (n == 0 && !fin)) return kFsmnHold;
  if (received < chunk_len) {
    if (received + n < chunk_len && !fin) return kFsmnFill;
    return received + n > 0 ? kFsmnWindow : kFsmnFlush;   // a stream that ends before its first window gets a padded one
  }
  return n > 0 ? kFsmnWindow : kFsmnFlush;
}

__device__ __forceinline__ int4 fsmn_chunk_vec(const int16_t* src, int k, int n) {
  if (k + 8 <= n) return __ldg(reinterpret_cast<const int4*>(src + k));
  int4 v = make_int4(0, 0, 0, 0);
  int16_t* e = reinterpret_cast<int16_t*>(&v);
#pragma unroll
  for (int j = 0; j < 8; ++j) e[j] = k + j < n ? src[k + j] : (int16_t)0;
  return v;
}

// CTA per slot: the tick's samples into the slot's window row [chunk_len] (the forward's input), 8 samples per thread
// and vector, zeros from n on.  Before the first window the chunk lands at `received` and zeros fill the rest of the row.
// From then on the row moves left by `stride` and the chunk fills its last `stride` samples: the shift overlaps itself
// whenever chunk_len - stride > stride, so it runs in strips of 8 * blockDim samples, all reads of a strip before a
// barrier and all its writes after it (a strip's writes lie below every later strip's reads).  A held slot's row is not
// touched.  Thread 0 also writes the slot's background level, the forward's gate input.
__global__ void __launch_bounds__(256) fsmn_serve_load_kernel(const int16_t* __restrict__ chunk,
                                                             const int32_t* __restrict__ n_samples,
                                                             const uint8_t* __restrict__ last,
                                                             const int32_t* __restrict__ state, int words, int chunk_len,
                                                             int stride, float noise_init, int16_t* __restrict__ window,
                                                             float* __restrict__ noise_avg) {
  const int64_t s = blockIdx.x;
  const int32_t* st = state + s * words;
  const int received = st[0], n = n_samples[s];
  if (threadIdx.x == 0) noise_avg[s] = __int_as_float(st[3] ^ __float_as_int(noise_init));
  int err;
  const int plan = fsmn_serve_plan(n, last[s] != 0, received, chunk_len, stride, err);
  if (plan == kFsmnHold || plan == kFsmnFlush) return;
  int16_t* row = window + s * chunk_len;
  const int16_t* src = chunk + s * stride;
  if (received < chunk_len) {
    for (int k = received + 8 * threadIdx.x; k < chunk_len; k += 8 * blockDim.x)
      *reinterpret_cast<int4*>(row + k) = fsmn_chunk_vec(src, k - received, n);
    return;
  }
  const int keep = chunk_len - stride;
  for (int base = 0; base < chunk_len; base += 8 * blockDim.x) {
    const int k = base + 8 * threadIdx.x;
    int4 v = make_int4(0, 0, 0, 0);
    if (k < keep) v = *reinterpret_cast<const int4*>(row + k + stride);
    else if (k < chunk_len) v = fsmn_chunk_vec(src, k - keep, n);
    __syncthreads();
    if (k < chunk_len) *reinterpret_cast<int4*>(row + k) = v;
  }
}

// The reference's final timestamps, online.  Offline they are process_timestamps(runs_to_timestamps(saved, d), fusion,
// min_dur) (FSMN/Inference_FSMN_VAD_ONNX.py:102-141): a run of non-silence decisions a..b-1 is (a*d, b*d + d), one still
// open at the end (a*d, n*d); runs shorter than min_dur go, then neighbours with start - previous end <= fusion fuse (the
// second fusion pass never fuses again).  Here every double is formed as Python forms it (no contraction into FMAs), and
// an event leaves as soon as it is certain:
//   - an open run is kept once m*d - a*d >= min_dur (m decisions so far): every end it can still get is >= m*d;
//   - a pending segment's end is final once the earliest start a later kept run can have (the open run's, else m) lies
//     more than `fusion` after it.
struct FsmnTimestamps {
  int m, run_a, seg, seg_b;      // run_a < 0: no open run; seg_b: the closing decision of the pending segment's last run
  double d, fusion, min_dur;
  int2* ev;
  int count;

  __device__ __forceinline__ double at(int i) const { return __dmul_rn((double)i, d); }
  __device__ __forceinline__ double end_at(int b) const { return __dadd_rn(at(b), d); }
  __device__ __forceinline__ void push(int kind, int v) { ev[count++] = make_int2(kind, v); }
  // the run starting at a is kept: it fuses into the pending segment or ends it and opens the next
  __device__ __forceinline__ void kept(int a) {
    if (seg == kFsmnSegPending) {
      if (__dsub_rn(at(a), end_at(seg_b)) <= fusion) { seg = kFsmnSegOpen; return; }
      push(VADX_SERVE_END, seg_b);
    }
    push(VADX_SERVE_START, a);
    seg = kFsmnSegOpen;
  }
  __device__ __forceinline__ void decide(bool silence) {
    const int i = m++;
    if (!silence) {
      if (run_a < 0) run_a = i;
      if (seg != kFsmnSegOpen && __dsub_rn(at(m), at(run_a)) >= min_dur) kept(run_a);
    } else if (run_a >= 0) {
      if (seg == kFsmnSegOpen || __dsub_rn(end_at(i), at(run_a)) >= min_dur) {
        if (seg != kFsmnSegOpen) kept(run_a);
        seg = kFsmnSegPending;
        seg_b = i;
      }
      run_a = -1;
    }
    if (seg == kFsmnSegPending && __dsub_rn(at(run_a >= 0 ? run_a : m), end_at(seg_b)) > fusion) {
      push(VADX_SERVE_END, seg_b);
      seg = kFsmnSegNone;
    }
  }
  __device__ __forceinline__ void finish() {
    if (run_a >= 0 && (seg == kFsmnSegOpen || __dsub_rn(at(m), at(run_a)) >= min_dur)) {
      if (seg != kFsmnSegOpen) kept(run_a);
      push(VADX_SERVE_END_OF_STREAM, m);
    } else if (seg == kFsmnSegPending) {
      push(VADX_SERVE_END, seg_b);
    }
  }
};

// Thread per slot, after the forward: validate the control words (fsmn_serve_plan), run the look-ahead hysteresis over
// the slot's score row [T] feeding every decision to the timestamp machine, update the background level, and stage at
// most 2T + 2 events (kind, decision) in `staged` [S][2T+2]: a tick hands D <= T decisions to the machine, at most one
// START per decision (a run that is only kept at finalize has its last decision in this tick, which started nothing,
// unless D = 0), and every END / END_OF_STREAM closes a segment started in this tick or the one open before it; so
// events <= 2D + 1 <= 2T + 1 for D >= 1, and 3 <= 2T + 2 for D = 0.
__global__ void __launch_bounds__(kServeThreads) fsmn_serve_seg_kernel(
    const uint8_t* __restrict__ score, int64_t ld_score, const float* __restrict__ noisy_dB, int T,
    const int32_t* __restrict__ n_samples, const uint8_t* __restrict__ last, int64_t n_slots, int chunk_len, int stride,
    int look_backward, const vadx_fsmn_serve_cfg cfg, int32_t* __restrict__ state, int32_t* __restrict__ decisions_out,
    int32_t* __restrict__ staged, int32_t* __restrict__ counts, int8_t* __restrict__ action, int32_t* __restrict__ block_info) {
  const int64_t s = (int64_t)blockIdx.x * kServeThreads + threadIdx.x;
  int count = 0, err = 0;
  if (s < n_slots) {
    const int words = fsmn_serve_words(look_backward);
    int32_t* st = state + s * words;
    const int n = n_samples[s];
    const bool fin = last[s] != 0;
    const int plan = fsmn_serve_plan(n, fin, st[0], chunk_len, stride, err);
    int8_t act = kServeHold;                         // no window ran: the caches stay as they were
    int D = 0;
    if (plan == kFsmnFill) {
      st[0] += n;
    } else if (plan != kFsmnHold) {
      const int32_t init_bits = __float_as_int(cfg.noise_init);
      bool silence = st[1] == 0;
      FsmnTimestamps ts{st[2], st[4] - 1, st[5], st[6], cfg.frame_duration, cfg.fusion_threshold, cfg.min_speech_duration,
                        reinterpret_cast<int2*>(staged) + s * (2 * (int64_t)T + 2), 0};
      const int m0 = ts.m;
      if (plan == kFsmnWindow) {
        const uint8_t* fl = score + s * ld_score;
        hysteresis_chunk(fl, nullptr, 0, T, look_backward, cfg.speaking_score, cfg.silence_score, fin, silence,
                         [&](bool sil) { ts.decide(sil); });
        const float nd = noisy_dB[s];
        if (nd > 0.0f) {
          const float level = __int_as_float(st[3] ^ init_bits);
          st[3] = __float_as_int(0.5f * ((level + nd) + cfg.snr_threshold)) ^ init_bits;
        }
        for (int w = 0; w < (look_backward + 31) / 32; ++w) {
          uint32_t bits = 0;
          for (int j = 0; j < 32 && 32 * w + j < look_backward; ++j)
            bits |= (fl[T - look_backward + 32 * w + j] != 0 ? 1u : 0u) << j;
          st[kFsmnServeHeader + w] = (int32_t)bits;
        }
        st[0] = chunk_len;
      } else if (st[0] == chunk_len) {               // finalize without audio: the flush of the latest window
        for (int j = 0; j < look_backward; ++j) {
          const bool speech = ((uint32_t)st[kFsmnServeHeader + j / 32] >> (j & 31)) & 1u;
          silence = hysteresis_tail(silence, speech, !speech);
          ts.decide(silence);
        }
      }
      D = ts.m - m0;
      if (fin) {
        ts.finish();
        for (int i = 0; i < words; ++i) st[i] = 0;   // the next stream in this slot starts fresh
        act = kServeFinalize;
      } else {
        st[1] = silence ? 0 : 1;
        st[2] = ts.m; st[4] = ts.run_a + 1; st[5] = ts.seg; st[6] = ts.seg_b;
        act = kServeAdvance;
      }
      count = ts.count;
    }
    action[s] = act;
    decisions_out[s] = D;
    counts[s] = count;
  }
  serve_block_totals(count, err, block_info);
}

// ---- MarbleNet slot server (vadx_marblenet_serve_step) ----
// The reference's VadPostprocessor (oracle/postproc.frame_decisions + segments_from_decisions, the passes of
// postprocess_frames_runs_kernel) online: each whole-track pass only reaches a bounded number of frames back, so it
// becomes a stage with a fixed delay that hands final decisions, in frame order, to the next one:
//   2. the four-state machine back-fills at most D2 = max(min_speech, 1) frames (0 in the plain-threshold case);
//   3. a rising edge at t sets [t - ws, t) (D3 = ws when ws > 1);
//   4. a gap [g, t) is filled when t - g < merge, so t <= g + merge - 1 (D4 = max(merge - 1, 0));
//   5. dilation by extend is "a 1 in [f - extend, f + extend]" (D5 = max(extend, 0), no ring: the latest 1 suffices);
//   6. the max-speech split runs on the final decisions with a running first-minimum of the raw probabilities.
// A frame's pre-split decision is final D = D2 + D3 + D4 + D5 frames after it (16 at MarbleNet's defaults; D <= K =
// max(min_speech, 1) + ws + merge + extend).  Stages 2-4 keep their provisional decisions in bit rings of D_i + 1 bits
// (a back-fill never reaches past the ring), the split reads the raw probabilities from a ring of D + 1 floats.
// State words per slot: 0 frames consumed, 1..2 samples consumed (int64, low word first), 3 running sum (float bits),
// 4 machine state, 5 t_sp, 6 t_si, 7 previous stage-3 input, 8 previous stage-4 input, 9 gap start + 1 (0 = none),
// 10 latest stage-5 speech frame + 1 (0 = none), 11 in a run, 12 piece start, 13 piece START emitted, 14 running
// minimum (float bits), 15 its frame, then the running-sum ring [ws] (ws > 1), the probability ring [D + 1] and the
// bit rings of stages 2, 3, 4.  All zero = a fresh slot.
constexpr int kMnHeader = 16;
constexpr int kMnMaxDelay = 1 << 16;       // keeps a slot's state words and staged events well inside int

struct MnLayout {
  int ws, D2, D3, D4, D5, D, o_cs, o_p, o_r2, o_r3, o_r4, words;
  __host__ __device__ explicit MnLayout(const vadx_post_cfg& c) {
    ws = c.smooth_window < 1 ? 1 : c.smooth_window;
    D2 = (c.min_speech_frame <= 0 && c.min_silence_frame <= 0) ? 0 : (c.min_speech_frame > 1 ? c.min_speech_frame : 1);
    D3 = ws > 1 ? ws : 0;
    D4 = c.merge_silence_frame > 1 ? c.merge_silence_frame - 1 : 0;
    D5 = c.extend_speech_frame > 0 ? c.extend_speech_frame : 0;
    D = D2 + D3 + D4 + D5;
    o_cs = kMnHeader;
    o_p = o_cs + (ws > 1 ? ws : 0);
    o_r2 = o_p + D + 1;
    o_r3 = o_r2 + (D2 + 32) / 32;
    o_r4 = o_r3 + (D3 + 32) / 32;
    words = o_r4 + (D4 + 32) / 32;
  }
};

struct MnSeg {
  const MnLayout lay;
  int32_t* st;
  int max_sf, half, min_sp, min_si, merge, extend;
  int t, mode, t_sp, t_si, prev3, prev4, gap, l1, in_run, pos, started, best_i;
  float run, best;
  int2* ev;
  int count;

  __device__ __forceinline__ bool bit(int off, int size, int f) const {
    const int i = f % size;
    return ((uint32_t)st[off + (i >> 5)] >> (i & 31)) & 1u;
  }
  __device__ __forceinline__ void set_bit(int off, int size, int f, bool v) {
    const int i = f % size;
    const uint32_t m = 1u << (i & 31), w = (uint32_t)st[off + (i >> 5)];
    st[off + (i >> 5)] = (int32_t)(v ? (w | m) : (w & ~m));
  }
  __device__ __forceinline__ void push(int kind, int v) { ev[count++] = make_int2(kind, v); }
  __device__ __forceinline__ void reset_min() { best = INFINITY; best_i = 0; }

  // 6: the max-speech split on final decisions, in frame order.  A START leaves once its frame can no longer be cut:
  // at once for max_speech >= 2 (a cut lies at least half >= 1 past the piece start), with the piece's END for 1.
  __device__ __forceinline__ void in6(int f, bool d) {
    const bool defer = max_sf == 1;
    if (d) {
      if (!in_run) {
        in_run = 1; pos = f; started = 0; reset_min();
        if (!defer) { push(VADX_SERVE_START, f); started = 1; }
      } else if (max_sf >= 1 && f == pos + max_sf) {   // frame pos + max is speech: cut at the first arg-min
        const int cut = best_i;
        if (cut > pos) {
          if (!started) push(VADX_SERVE_START, pos);
          push(VADX_SERVE_END, cut);
        }
        pos = cut + 1; started = 0; reset_min();           // the next window starts at cut + 1 + half >= f
        if (!defer) { push(VADX_SERVE_START, pos); started = 1; }
      }
      if (max_sf >= 1 && f >= pos + half) {
        const float p = __int_as_float(st[lay.o_p + f % (lay.D + 1)]);
        if (p < best) { best = p; best_i = f; }
      }
    } else if (in_run) {
      if (!started) push(VADX_SERVE_START, pos);
      push(VADX_SERVE_END, f);
      in_run = 0;
    }
  }
  // 5: dilation by extend
  __device__ __forceinline__ bool dilated(int f) const { return l1 > 0 && l1 - 1 >= f - extend; }
  __device__ __forceinline__ void in5(int i, bool b) {
    if (lay.D5 == 0) { in6(i, b); return; }
    if (b) l1 = i + 1;
    if (i - lay.D5 >= 0) in6(i - lay.D5, dilated(i - lay.D5));
  }
  // 4: gaps shorter than merge are filled
  __device__ __forceinline__ void in4(int i, bool b) {
    if (lay.D4 == 0) { in5(i, b); return; }
    const int R = lay.D4 + 1;
    set_bit(lay.o_r4, R, i, b);
    if (i >= 1) {
      if (prev4 && !b && gap == 0) {
        gap = i + 1;
      } else if (!prev4 && b && gap > 0) {
        if (i - (gap - 1) < merge)
          for (int g = gap - 1; g < i; ++g) set_bit(lay.o_r4, R, g, true);
        gap = 0;
      }
    }
    prev4 = b;
    if (i - lay.D4 >= 0) in5(i - lay.D4, bit(lay.o_r4, R, i - lay.D4));
  }
  // 3: rising edges move left by ws
  __device__ __forceinline__ void in3(int i, bool b) {
    if (lay.D3 == 0) { in4(i, b); return; }
    const int R = lay.D3 + 1;
    set_bit(lay.o_r3, R, i, b);
    if (i >= 1 && b && !prev3)
      for (int g = i - lay.ws < 0 ? 0 : i - lay.ws; g < i; ++g) set_bit(lay.o_r3, R, g, true);
    prev3 = b;
    if (i - lay.D3 >= 0) in4(i - lay.D3, bit(lay.o_r3, R, i - lay.D3));
  }
  // 1 + 2: smoothing with postprocess_frames_runs_kernel's rounding, then the four-state machine.  The mean of the
  // stream's first ws - 1 frames divides by u + 1; its flag comes in as early_hot (see early_flags).
  __device__ __forceinline__ void frame(float p, bool early_hot) {
    const int u = t++;
    st[lay.o_p + u % (lay.D + 1)] = __float_as_int(p);
    bool hot = p >= __int_as_float(thr_bits);
    if (lay.ws > 1) {
      const int k = lay.o_cs + u % lay.ws;
      const float old = __int_as_float(st[k]);           // the running sum ws frames back (0 before the stream)
      run = __fadd_rn(run, p);
      hot = u < lay.ws - 1 ? early_hot
                           : __fmul_rn(__fsub_rn(run, old), (float)(1.0 / (double)lay.ws)) >= __int_as_float(thr_bits);
      st[k] = __float_as_int(run);
    }
    if (lay.D2 == 0) { in3(u, hot); return; }
    const int R = lay.D2 + 1;
    if (mode == 0) {
      if (hot) { mode = 1; t_sp = u; }
    } else if (mode == 1) {
      if (!hot) {
        mode = 0;
      } else if (u - t_sp >= min_sp) {
        mode = 2;
        for (int g = t_sp; g < u; ++g) set_bit(lay.o_r2, R, g, true);   // u - t_sp == D2
      }
    } else if (mode == 2) {
      if (!hot) { mode = 3; t_si = u; }
    } else {
      if (hot) mode = 2;
      else if (u - t_si >= min_si) mode = 0;
    }
    set_bit(lay.o_r2, R, u, mode >= 2);
    if (u - lay.D2 >= 0) in3(u - lay.D2, bit(lay.o_r2, R, u - lay.D2));
  }
  // finalize: every stage flushes its delay line in order (a MAYBE_SP stretch stays silence, an open gap is not
  // merged, dilation runs to n), then a run reaching n ends the stream
  __device__ __forceinline__ void finish(float frame_shift, int64_t samples) {
    const int n = t;
    if (lay.D2) for (int o = n - lay.D2 < 0 ? 0 : n - lay.D2; o < n; ++o) in3(o, bit(lay.o_r2, lay.D2 + 1, o));
    if (lay.D3) for (int o = n - lay.D3 < 0 ? 0 : n - lay.D3; o < n; ++o) in4(o, bit(lay.o_r3, lay.D3 + 1, o));
    if (lay.D4) for (int o = n - lay.D4 < 0 ? 0 : n - lay.D4; o < n; ++o) in5(o, bit(lay.o_r4, lay.D4 + 1, o));
    if (lay.D5) for (int o = n - lay.D5 < 0 ? 0 : n - lay.D5; o < n; ++o) in6(o, dilated(o));
    if (in_run) {
      if (!started) push(VADX_SERVE_START, pos);
      // PP.segments_to_seconds: n * fs in float32, replaced by the recording's duration when that is smaller
      const float e = __fmul_rn(__int2float_rn(n), frame_shift);
      const double dur = __ddiv_rn((double)samples, 16000.0);
      push(VADX_SERVE_END_OF_STREAM, __float_as_int(dur < (double)e ? __double2float_rn(dur) : e));
    }
  }
  int32_t thr_bits;
};

// Thread per slot, after the forward: validate the slot's control words, run the online post-processor over the F
// frames of a fed tick (none on a hold or a finalize without audio), and stage the events (kind, value) in `staged`
// [S][2 (F + D) + 2].  The split stage receives at most F + D frames in a tick (F new ones, and D more when finalize
// flushes the delay lines); each of them emits at most one START (a run opens, a piece starts after a cut, or a deferred
// START leaves with its END) and one END (a cut or a run's end), and finalize adds at most a deferred START and the
// END_OF_STREAM.
__global__ void __launch_bounds__(kServeThreads) marblenet_serve_seg_kernel(
    const float* __restrict__ probs, int64_t ld_probs, int F, const int32_t* __restrict__ n_samples,
    const uint8_t* __restrict__ last, int64_t n_slots, int window_samples, const vadx_post_cfg cfg, float frame_shift,
    int32_t* __restrict__ state, int32_t* __restrict__ frames_out, int32_t* __restrict__ staged,
    int32_t* __restrict__ counts, int8_t* __restrict__ action, int32_t* __restrict__ block_info) {
  const int64_t s = (int64_t)blockIdx.x * kServeThreads + threadIdx.x;
  int count = 0, err = 0;
  if (s < n_slots) {
    const int n = n_samples[s];
    const bool fin = last[s] != 0;
    err = serve_control_error(n, fin, window_samples);
    int f = 0;
    if (err || (n == 0 && !fin)) {
      action[s] = kServeHold;                       // hold, or a rejected tick: the slot stays exactly as it was
    } else {
      const MnLayout lay(cfg);
      int32_t* st = state + s * (int64_t)lay.words;
      const int64_t cap = 2 * ((int64_t)F + lay.D) + 2;
      MnSeg g{lay, st, cfg.max_speech_frame, cfg.max_speech_frame >> 1, cfg.min_speech_frame, cfg.min_silence_frame,
              cfg.merge_silence_frame, cfg.extend_speech_frame, st[0], st[4], st[5], st[6], st[7], st[8], st[9], st[10],
              st[11], st[12], st[13], st[15], __int_as_float(st[3]), __int_as_float(st[14]),
              reinterpret_cast<int2*>(staged) + s * cap, 0, __float_as_int(cfg.threshold)};
      const int64_t samples = ((int64_t)(uint32_t)st[1] | ((int64_t)st[2] << 32)) + n;
      if (n > 0) {
        f = F;
        const float* p = probs + s * ld_probs;
        // flags of the frames u < ws - 1 (at most 63: ws <= kMaxSmooth), in a loop of their own so that the division's
        // slow-path call does not make the main loop spill
        uint64_t early = 0;
        const int n_early = min(F, lay.ws - 1 - g.t);
        float r = g.run;
        for (int k = 0; k < n_early; ++k) {
          r = __fadd_rn(r, __ldg(p + k));
          if (__fdiv_rn(r, (float)(g.t + k + 1)) >= cfg.threshold) early |= 1ull << k;
        }
        for (int k = 0; k < F; ++k) g.frame(__ldg(p + k), k < n_early && ((early >> k) & 1));
      }
      if (fin) {
        g.finish(frame_shift, samples);
        for (int i = 0; i < lay.words; ++i) st[i] = 0;   // the next stream in this slot starts fresh
        action[s] = kServeFinalize;
      } else {
        st[0] = g.t; st[1] = (int32_t)(uint32_t)samples; st[2] = (int32_t)(samples >> 32);
        st[3] = __float_as_int(g.run); st[4] = g.mode; st[5] = g.t_sp; st[6] = g.t_si; st[7] = g.prev3; st[8] = g.prev4;
        st[9] = g.gap; st[10] = g.l1; st[11] = g.in_run; st[12] = g.pos; st[13] = g.started;
        st[14] = __float_as_int(g.best); st[15] = g.best_i;
        action[s] = kServeAdvance;
      }
      count = g.count;
    }
    frames_out[s] = f;
    counts[s] = count;
  }
  serve_block_totals(count, err, block_info);
}

}  // namespace vadx

using namespace vadx;

extern "C" int vadx_stream_post_state_words(int smooth_window) {
  return kSpHeader + (smooth_window < 1 ? 1 : smooth_window);
}

extern "C" int vadx_stream_postprocess(const float* d_probs, int64_t ld_probs, const int32_t* d_n_frames,
                                       int64_t n_streams, int n_frames, const vadx_stream_post_cfg* cfg,
                                       int32_t* d_state, int32_t* d_seg_count, int32_t* d_segments, int max_segments,
                                       int32_t* d_open, void* stream) {
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "stream_postprocess_kernel", 4.0 * n_streams * n_frames);
  VADX_REQUIRE(d_probs && cfg && d_state, "vadx_stream_postprocess: null pointer");
  VADX_REQUIRE(n_streams >= 0 && n_frames >= 0 && ld_probs >= n_frames, "vadx_stream_postprocess: bad shape");
  VADX_REQUIRE(cfg->smooth_window <= kMaxSmooth, "vadx_stream_postprocess: smooth_window %d > %d", cfg->smooth_window,
               kMaxSmooth);
  VADX_REQUIRE(max_segments >= 0 && (max_segments == 0 || (d_segments && d_seg_count)),
               "vadx_stream_postprocess: segments buffer without counts");
  if (n_streams == 0) return VADX_OK;
  stream_post_kernel<<<(unsigned)ceil_div(n_streams, 128), 128, 0, (cudaStream_t)stream>>>(
      d_probs, ld_probs, d_n_frames, n_streams, n_frames, *cfg, d_state, d_seg_count, d_segments, max_segments, d_open);
  return after_launch("vadx_stream_postprocess");
}

extern "C" int vadx_stream_serve_zero_tail(int16_t* d_chunk, int64_t ld_chunk, const int32_t* d_n_samples,
                                           int64_t n_slots, int chunk_samples, int frame_len, void* stream) {
  VADX_REQUIRE(d_chunk && d_n_samples, "vadx_stream_serve_zero_tail: null pointer");
  VADX_REQUIRE(n_slots >= 0 && frame_len >= 1 && chunk_samples >= frame_len && ld_chunk >= chunk_samples,
               "vadx_stream_serve_zero_tail: bad shape");
  if (n_slots == 0) return VADX_OK;
  stream_serve_tail_kernel<<<(unsigned)ceil_div(n_slots * frame_len, 256), 256, 0, (cudaStream_t)stream>>>(
      d_chunk, ld_chunk, d_n_samples, n_slots, chunk_samples, frame_len);
  return after_launch("vadx_stream_serve_zero_tail");
}

namespace {
// Scratch of a serve step: staged events [S][cap] int32 pairs, counts [S], actions [S], block totals [blocks][2].
struct ServeScratch {
  int64_t cap, n_blocks;
  size_t o_counts, o_action, o_info, need;
  ServeScratch(int64_t n_slots, int64_t cap_) : cap(cap_), n_blocks(ceil_div(n_slots, kServeThreads)) {
    o_counts = (size_t)round_up(n_slots * cap * 8, 256);
    o_action = o_counts + (size_t)round_up(n_slots * 4, 256);
    o_info = o_action + (size_t)round_up(n_slots, 256);
    need = o_info + (size_t)round_up(n_blocks * 8, 256);
  }
  int32_t* staged(void* p) const { return static_cast<int32_t*>(p); }
  int32_t* counts(void* p) const { return reinterpret_cast<int32_t*>(static_cast<char*>(p) + o_counts); }
  int8_t* action(void* p) const { return reinterpret_cast<int8_t*>(static_cast<char*>(p) + o_action); }
  int32_t* info(void* p) const { return reinterpret_cast<int32_t*>(static_cast<char*>(p) + o_info); }
};

// The emit kernel writes the host mirror through unified addressing: it must be page-locked host memory whose device
// address is its host address.  Checked on eager calls; a capture replays the pointers an eager call checked.
int check_host_mirror(const int32_t* h_events, const int32_t* h_header, void* stream, const char* who) {
  VADX_REQUIRE((h_events == nullptr) == (h_header == nullptr), "%s: h_events and h_header go together", who);
  if (!h_events) return VADX_OK;
  cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
  cudaError_t e = cudaStreamIsCapturing((cudaStream_t)stream, &cap_status);
  if (e != cudaSuccess) return cuda_fail(e, "cudaStreamIsCapturing");
  if (cap_status != cudaStreamCaptureStatusNone) return VADX_OK;
  for (const void* h : {(const void*)h_events, (const void*)h_header}) {
    cudaPointerAttributes at{};
    e = cudaPointerGetAttributes(&at, h);
    if (e != cudaSuccess) return cuda_fail(e, "cudaPointerGetAttributes");
    VADX_REQUIRE(at.type == cudaMemoryTypeHost && at.devicePointer == h,
                 "%s: the host mirror must be pinned host memory mapped at its own address", who);
  }
  return VADX_OK;
}

// stream_serve_emit_kernel over a segmenter's staged events, plus one block per slot when there are caches
int serve_emit(const ServeScratch& sl, int64_t n_slots, void* d_scratch, int32_t* d_events, int32_t* d_header,
               int32_t* h_events, int32_t* h_header, const float* d_caches_in, float* d_caches_out, int n_cache_blocks,
               int64_t cache_row, void* stream, const char* who) {
  const int64_t grid = sl.n_blocks + (d_caches_out ? n_slots : 0);
  stream_serve_emit_kernel<<<(unsigned)grid, kServeThreads, 0, (cudaStream_t)stream>>>(
      n_slots, (int)sl.n_blocks, (int)sl.cap, sl.staged(d_scratch), sl.counts(d_scratch), sl.action(d_scratch),
      sl.info(d_scratch), d_events, d_header, h_events, h_header, d_caches_in, d_caches_out, n_cache_blocks, cache_row);
  return after_launch(who);
}
}  // namespace

extern "C" int vadx_stream_serve_step(const float* d_probs, int64_t ld_probs, int n_frames, const int32_t* d_n_samples,
                                      const uint8_t* d_last, int64_t n_slots, int chunk_samples, int frame_len,
                                      int frame_hop, const vadx_stream_post_cfg* cfg, int32_t* d_state,
                                      const float* d_caches_in, float* d_caches_out, int n_cache_blocks,
                                      int64_t cache_row, int32_t* d_frames, int32_t* d_events, int32_t* d_header,
                                      int32_t* h_events, int32_t* h_header, void* d_scratch, size_t scratch_bytes,
                                      size_t* scratch_needed, void* stream) {
  VADX_REQUIRE(n_slots >= 1 && n_frames >= 1 && frame_len >= 1 && frame_hop >= 1 && chunk_samples >= frame_len,
               "vadx_stream_serve_step: bad shape");
  VADX_REQUIRE(1 + (chunk_samples - frame_len) / frame_hop <= n_frames,
               "vadx_stream_serve_step: a full chunk gives %d frames, probs hold %d", 1 + (chunk_samples - frame_len) / frame_hop,
               n_frames);
  const ServeScratch sl(n_slots, 2 * (int64_t)n_frames + 1);
  if (scratch_needed) *scratch_needed = sl.need;
  if (!d_scratch) return VADX_OK;                   // size query
  VADX_REQUIRE(scratch_bytes >= sl.need, "vadx_stream_serve_step: scratch of %zu bytes, %zu needed", scratch_bytes, sl.need);
  VADX_REQUIRE(d_probs && d_n_samples && d_last && cfg && d_state && d_frames && d_events && d_header,
               "vadx_stream_serve_step: null pointer");
  VADX_REQUIRE(ld_probs >= n_frames, "vadx_stream_serve_step: ld_probs %lld < n_frames %d", (long long)ld_probs, n_frames);
  VADX_REQUIRE(cfg->smooth_window <= kMaxSmooth, "vadx_stream_serve_step: smooth_window %d > %d", cfg->smooth_window,
               kMaxSmooth);
  VADX_REQUIRE((d_caches_in == nullptr) == (d_caches_out == nullptr) && (!d_caches_out || (n_cache_blocks >= 1 && cache_row >= 1)),
               "vadx_stream_serve_step: caches_in and caches_out go together, with n_cache_blocks and cache_row >= 1");
  VADX_REQUIRE(!d_caches_out || d_caches_in != d_caches_out, "vadx_stream_serve_step: caches_out must not alias caches_in");
  VADX_TRY(check_host_mirror(h_events, h_header, stream, "vadx_stream_serve_step"));
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "stream_serve_seg_kernel", 4.0 * n_slots * n_frames);
  stream_serve_seg_kernel<<<(unsigned)sl.n_blocks, kServeThreads, 0, (cudaStream_t)stream>>>(
      d_probs, ld_probs, n_frames, d_n_samples, d_last, n_slots, chunk_samples, frame_len, frame_hop, *cfg, d_state,
      d_frames, sl.staged(d_scratch), sl.counts(d_scratch), sl.action(d_scratch), sl.info(d_scratch));
  VADX_TRY(after_launch("vadx_stream_serve_step"));
  return serve_emit(sl, n_slots, d_scratch, d_events, d_header, h_events, h_header, d_caches_in, d_caches_out,
                    n_cache_blocks, cache_row, stream, "vadx_stream_serve_step");
}

extern "C" int vadx_silero_serve_load(const int16_t* d_chunk, const int32_t* d_n_samples, int64_t n_slots,
                                      int windows_per_tick, float* d_x, void* stream) {
  VADX_REQUIRE(n_slots >= 1 && windows_per_tick >= 1 && windows_per_tick <= kSileroMaxWindowsPerTick,
               "vadx_silero_serve_load: bad shape");
  VADX_REQUIRE(d_chunk && d_n_samples && d_x, "vadx_silero_serve_load: null pointer");
  VADX_REQUIRE(aligned16(d_chunk) && aligned16(d_x), "vadx_silero_serve_load: d_chunk and d_x must be 16-byte aligned");
  const int chunk_samples = windows_per_tick * kSileroWindow;
  StageTimer _timer(VADX_STAGE_PREP, (cudaStream_t)stream, "silero_serve_load_kernel", 6.0 * n_slots * chunk_samples);
  silero_serve_load_kernel<<<(unsigned)ceil_div(n_slots * (chunk_samples / 8), 256), 256, 0, (cudaStream_t)stream>>>(
      d_chunk, d_n_samples, n_slots, chunk_samples, d_x);
  return after_launch("vadx_silero_serve_load");
}

extern "C" int vadx_silero_serve_step(const float* d_probs, int64_t ld_probs, const int32_t* d_n_samples,
                                      const uint8_t* d_last, int64_t n_slots, int windows_per_tick, double threshold,
                                      double min_silence_samples, int32_t* d_state, float* d_x, const float* d_state_in,
                                      float* d_state_out, int32_t* d_windows, int32_t* d_events, int32_t* d_header,
                                      int32_t* h_events, int32_t* h_header, void* d_scratch, size_t scratch_bytes,
                                      size_t* scratch_needed, void* stream) {
  VADX_REQUIRE(n_slots >= 1 && windows_per_tick >= 1 && windows_per_tick <= kSileroMaxWindowsPerTick,
               "vadx_silero_serve_step: bad shape");
  const ServeScratch sl(n_slots, (int64_t)windows_per_tick + 1);
  if (scratch_needed) *scratch_needed = sl.need;
  if (!d_scratch) return VADX_OK;                   // size query
  VADX_REQUIRE(scratch_bytes >= sl.need, "vadx_silero_serve_step: scratch of %zu bytes, %zu needed", scratch_bytes, sl.need);
  VADX_REQUIRE(d_probs && d_n_samples && d_last && d_state && d_windows && d_events && d_header,
               "vadx_silero_serve_step: null pointer");
  VADX_REQUIRE(ld_probs >= n_slots, "vadx_silero_serve_step: ld_probs %lld < n_slots %lld", (long long)ld_probs,
               (long long)n_slots);
  VADX_REQUIRE(!d_x || aligned16(d_x), "vadx_silero_serve_step: d_x must be 16-byte aligned");
  VADX_REQUIRE((d_state_in == nullptr) == (d_state_out == nullptr),
               "vadx_silero_serve_step: state_in and state_out go together");
  VADX_REQUIRE(!d_state_out || d_state_in != d_state_out, "vadx_silero_serve_step: state_out must not alias state_in");
  VADX_TRY(check_host_mirror(h_events, h_header, stream, "vadx_silero_serve_step"));
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "silero_serve_seg_kernel", 4.0 * n_slots * windows_per_tick);
  silero_serve_seg_kernel<<<(unsigned)sl.n_blocks, kServeThreads, 0, (cudaStream_t)stream>>>(
      d_probs, ld_probs, d_n_samples, d_last, n_slots, windows_per_tick, threshold, min_silence_samples, d_state, d_x,
      d_windows, sl.staged(d_scratch), sl.counts(d_scratch), sl.action(d_scratch), sl.info(d_scratch));
  VADX_TRY(after_launch("vadx_silero_serve_step"));
  return serve_emit(sl, n_slots, d_scratch, d_events, d_header, h_events, h_header, d_state_in, d_state_out, 2,
                    kSileroHidden, stream, "vadx_silero_serve_step");
}

extern "C" int vadx_fsmn_serve_state_words(int look_backward) { return fsmn_serve_words(look_backward < 0 ? 0 : look_backward); }

extern "C" int vadx_fsmn_serve_load(const int16_t* d_chunk, const int32_t* d_n_samples, const uint8_t* d_last,
                                    const int32_t* d_state, int64_t n_slots, int chunk_len, int stride, int look_backward,
                                    float noise_init, int16_t* d_window, float* d_noise_avg, void* stream) {
  VADX_REQUIRE(n_slots >= 1 && stride >= 1 && stride < chunk_len && chunk_len <= kFsmnMaxChunk && chunk_len % 8 == 0 &&
                   stride % 8 == 0 && look_backward >= 0,
               "vadx_fsmn_serve_load: bad shape");
  VADX_REQUIRE(d_chunk && d_n_samples && d_last && d_state && d_window && d_noise_avg, "vadx_fsmn_serve_load: null pointer");
  VADX_REQUIRE(aligned16(d_chunk) && aligned16(d_window), "vadx_fsmn_serve_load: d_chunk and d_window must be 16-byte aligned");
  StageTimer _timer(VADX_STAGE_PREP, (cudaStream_t)stream, "fsmn_serve_load_kernel", 2.0 * n_slots * (stride + 2.0 * chunk_len));
  fsmn_serve_load_kernel<<<(unsigned)n_slots, 256, 0, (cudaStream_t)stream>>>(
      d_chunk, d_n_samples, d_last, d_state, fsmn_serve_words(look_backward), chunk_len, stride, noise_init,
      d_window, d_noise_avg);
  return after_launch("vadx_fsmn_serve_load");
}

extern "C" int vadx_fsmn_serve_step(const uint8_t* d_score, int64_t ld_score, const float* d_noisy_dB, int n_frames,
                                    const int32_t* d_n_samples, const uint8_t* d_last, int64_t n_slots, int chunk_len,
                                    int stride, int look_backward, const vadx_fsmn_serve_cfg* cfg, int32_t* d_state,
                                    const float* d_caches_in, float* d_caches_out, int n_cache_blocks, int64_t cache_row,
                                    int32_t* d_decisions, int32_t* d_events, int32_t* d_header, int32_t* h_events,
                                    int32_t* h_header, void* d_scratch, size_t scratch_bytes, size_t* scratch_needed,
                                    void* stream) {
  VADX_REQUIRE(n_slots >= 1 && n_frames >= 1 && stride >= 1 && stride < chunk_len && chunk_len <= kFsmnMaxChunk &&
                   look_backward >= 0 && look_backward < n_frames,
               "vadx_fsmn_serve_step: bad shape");
  const ServeScratch sl(n_slots, 2 * (int64_t)n_frames + 2);
  if (scratch_needed) *scratch_needed = sl.need;
  if (!d_scratch) return VADX_OK;                   // size query
  VADX_REQUIRE(scratch_bytes >= sl.need, "vadx_fsmn_serve_step: scratch of %zu bytes, %zu needed", scratch_bytes, sl.need);
  VADX_REQUIRE(d_score && d_noisy_dB && d_n_samples && d_last && cfg && d_state && d_decisions && d_events && d_header,
               "vadx_fsmn_serve_step: null pointer");
  VADX_REQUIRE(ld_score >= n_frames, "vadx_fsmn_serve_step: ld_score %lld < n_frames %d", (long long)ld_score, n_frames);
  VADX_REQUIRE((d_caches_in == nullptr) == (d_caches_out == nullptr) && (!d_caches_out || (n_cache_blocks >= 1 && cache_row >= 1)),
               "vadx_fsmn_serve_step: caches_in and caches_out go together, with n_cache_blocks and cache_row >= 1");
  VADX_REQUIRE(!d_caches_out || d_caches_in != d_caches_out, "vadx_fsmn_serve_step: caches_out must not alias caches_in");
  VADX_TRY(check_host_mirror(h_events, h_header, stream, "vadx_fsmn_serve_step"));
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "fsmn_serve_seg_kernel", 1.0 * n_slots * n_frames);
  fsmn_serve_seg_kernel<<<(unsigned)sl.n_blocks, kServeThreads, 0, (cudaStream_t)stream>>>(
      d_score, ld_score, d_noisy_dB, n_frames, d_n_samples, d_last, n_slots, chunk_len, stride, look_backward, *cfg, d_state,
      d_decisions, sl.staged(d_scratch), sl.counts(d_scratch), sl.action(d_scratch), sl.info(d_scratch));
  VADX_TRY(after_launch("vadx_fsmn_serve_step"));
  return serve_emit(sl, n_slots, d_scratch, d_events, d_header, h_events, h_header, d_caches_in, d_caches_out,
                    n_cache_blocks, cache_row, stream, "vadx_fsmn_serve_step");
}

extern "C" int vadx_marblenet_serve_state_words(const vadx_post_cfg* cfg) {
  VADX_REQUIRE(cfg, "vadx_marblenet_serve_state_words: null pointer");
  VADX_REQUIRE(MnLayout(*cfg).D <= kMnMaxDelay, "vadx_marblenet_serve_state_words: a decision delay of %d frames > %d",
               MnLayout(*cfg).D, kMnMaxDelay);
  return MnLayout(*cfg).words;
}

extern "C" int vadx_marblenet_serve_step(const float* d_probs, int64_t ld_probs, int n_frames, const int32_t* d_n_samples,
                                         const uint8_t* d_last, int64_t n_slots, int window_samples,
                                         const vadx_post_cfg* cfg, float frame_shift, int32_t* d_state, int32_t* d_frames,
                                         int32_t* d_events, int32_t* d_header, int32_t* h_events, int32_t* h_header,
                                         void* d_scratch, size_t scratch_bytes, size_t* scratch_needed, void* stream) {
  VADX_REQUIRE(n_slots >= 1 && n_frames >= 1 && window_samples >= 1, "vadx_marblenet_serve_step: bad shape");
  VADX_REQUIRE(cfg, "vadx_marblenet_serve_step: null pointer");
  const MnLayout lay(*cfg);
  VADX_REQUIRE(lay.D <= kMnMaxDelay, "vadx_marblenet_serve_step: a decision delay of %d frames > %d", lay.D, kMnMaxDelay);
  VADX_REQUIRE(cfg->smooth_window <= kMaxSmooth, "vadx_marblenet_serve_step: smooth_window %d > %d", cfg->smooth_window,
               kMaxSmooth);
  const ServeScratch sl(n_slots, 2 * ((int64_t)n_frames + lay.D) + 2);
  if (scratch_needed) *scratch_needed = sl.need;
  if (!d_scratch) return VADX_OK;                   // size query
  VADX_REQUIRE(scratch_bytes >= sl.need, "vadx_marblenet_serve_step: scratch of %zu bytes, %zu needed", scratch_bytes,
               sl.need);
  VADX_REQUIRE(d_probs && d_n_samples && d_last && d_state && d_frames && d_events && d_header,
               "vadx_marblenet_serve_step: null pointer");
  VADX_REQUIRE(ld_probs >= n_frames, "vadx_marblenet_serve_step: ld_probs %lld < n_frames %d", (long long)ld_probs,
               n_frames);
  VADX_TRY(check_host_mirror(h_events, h_header, stream, "vadx_marblenet_serve_step"));
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "marblenet_serve_seg_kernel", 4.0 * n_slots * n_frames);
  marblenet_serve_seg_kernel<<<(unsigned)sl.n_blocks, kServeThreads, 0, (cudaStream_t)stream>>>(
      d_probs, ld_probs, n_frames, d_n_samples, d_last, n_slots, window_samples, *cfg, frame_shift, d_state, d_frames,
      sl.staged(d_scratch), sl.counts(d_scratch), sl.action(d_scratch), sl.info(d_scratch));
  VADX_TRY(after_launch("vadx_marblenet_serve_step"));
  return serve_emit(sl, n_slots, d_scratch, d_events, d_header, h_events, h_header, nullptr, nullptr, 0, 0, stream,
                    "vadx_marblenet_serve_step");
}

extern "C" int vadx_postprocess_frames(const float* d_probs, int64_t ld_probs, const int32_t* d_n_frames,
                                       int64_t n_streams, int n_frames, const vadx_post_cfg* cfg,
                                       int8_t* d_decisions, int32_t* d_seg_count, int32_t* d_segments,
                                       int max_segments, void* stream) {
  StageTimer _timer(VADX_STAGE_POSTPROC, (cudaStream_t)stream, "postprocess_frames_runs_kernel", 5.0 * n_streams * n_frames);
  VADX_REQUIRE(d_probs && cfg && d_decisions, "vadx_postprocess_frames: null pointer (d_decisions is required)");
  VADX_REQUIRE(n_streams >= 0 && n_frames >= 0 && ld_probs >= n_frames, "vadx_postprocess_frames: bad shape");
  VADX_REQUIRE(cfg->smooth_window <= kMaxSmooth, "vadx_postprocess_frames: smooth_window %d > %d", cfg->smooth_window,
               kMaxSmooth);
  VADX_REQUIRE(max_segments >= 0 && (max_segments == 0 || d_segments), "vadx_postprocess_frames: segments buffer");
  if (n_streams == 0) return VADX_OK;
  // warp-per-stream kernel when one stream (probs + running sums + decisions) fits in shared memory
  const int per_warp_floats = (int)round_up(2 * (int64_t)std::max(n_frames, 1) + 1 + (std::max(n_frames, 1) + 3) / 4 +
                                               (std::max(n_frames, 1) + 31) / 32 + 1, 4);
  const size_t smem_w = (size_t)per_warp_floats * 4 * kPpWarps;
  if (smem_w <= 200 * 1024) {
    static PerDevice per_device_w;
    VADX_TRY(per_device_w.ensure(nullptr, [] {
      cudaError_t e = cudaFuncSetAttribute(postprocess_frames_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(postprocess_frames_runs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      return e;
    }));
    // VADX_PP_LEGACY=1 (AB build only): the frame-by-frame kernel, kept as the cross-check of the run-based one
    static const int legacy = ab_env("VADX_PP_LEGACY", 0);
    if (legacy)
      postprocess_frames_warp_kernel<<<(unsigned)ceil_div(n_streams, kPpWarps), kPpWarps * 32, smem_w, (cudaStream_t)stream>>>(
          d_probs, ld_probs, d_n_frames, n_streams, n_frames, *cfg, d_decisions, d_seg_count, d_segments, max_segments,
          per_warp_floats);
    else
      postprocess_frames_runs_kernel<<<(unsigned)ceil_div(n_streams, kPpWarps), kPpWarps * 32, smem_w, (cudaStream_t)stream>>>(
          d_probs, ld_probs, d_n_frames, n_streams, n_frames, *cfg, d_decisions, d_seg_count, d_segments, max_segments,
          per_warp_floats);
    return after_launch("vadx_postprocess_frames");
  }
  const int64_t blocks = ceil_div(n_streams, 32);
  const size_t smem = (size_t)std::max(n_frames, 1) * 32;
  const int use_smem = smem <= 200 * 1024;
  static PerDevice per_device;
  VADX_TRY(per_device.ensure(nullptr, [] {
    return cudaFuncSetAttribute(postprocess_frames_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  }));
  postprocess_frames_kernel<<<(unsigned)blocks, 32, use_smem ? smem : 0, (cudaStream_t)stream>>>(
      d_probs, ld_probs, d_n_frames, n_streams, n_frames, *cfg, d_decisions, d_seg_count, d_segments, max_segments,
      use_smem);
  return after_launch("vadx_postprocess_frames");
}
