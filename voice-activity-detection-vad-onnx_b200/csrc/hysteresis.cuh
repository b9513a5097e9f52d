// hysteresis.cuh -- the look-ahead hysteresis of FSMN / DFSMN, one stream per thread (a13).  Shared by the lock-step
// kernels (fsmn_extra.cu) and the FSMN slot server (postproc.cu), which differ only in what they do with a decision.
#pragma once
#include "common.cuh"

namespace vadx {

// One decision of the final flush (FSMN/Inference_FSMN_VAD_ONNX.py:226-234): the last look_backward frames of the last
// window vote one frame at a time.
__device__ __forceinline__ bool hysteresis_tail(bool silence, bool speech_vote, bool silence_vote) {
  return silence ? !speech_vote : silence_vote;
}

// mode 0 (FSMN): `fl` is uint8 flags; a frame votes "speech" when flag != 0 and "silence" when
//                flag != 1 (FSMN/Inference_FSMN_VAD_ONNX.py:188-215).
// mode 1 (DFSMN): `pr` is fp32 probabilities; a frame votes with p >= SPEAKING_SCORE / p <= SILENCE_SCORE, the same two
//                scores the vote RATIO is then tested against (DFSMN/near_and_far_end_audio/Inference_DFSMN_VAD_ONNX.py:
//                231-273).  The per-frame test compares a numpy float32 with a Python float: under NEP 50 (numpy >= 2) the
//                Python float is the weak operand, so the comparison happens in float32; the ratio test is Python floats.
// One window of the machine for one stream: hands T - look_backward decisions (all T when is_final) to emit(silence).
template <class Emit>
__device__ __forceinline__ void hysteresis_chunk(const uint8_t* fl, const float* pr, int mode, int T, int look_backward,
                                                 double speaking_score, double silence_score, int is_final, bool& silence,
                                                 Emit&& emit) {
  const float speak_f = (float)speaking_score, sil_f = (float)silence_score;
  auto speech_vote = [&](int i) { return mode == 0 ? fl[i] != 0 : pr[i] >= speak_f; };
  auto silence_vote = [&](int i) { return mode == 0 ? fl[i] != 1 : pr[i] <= sil_f; };
  const int lb = look_backward != 0 ? look_backward : 1;
  const double inv_d = 1.0 / (double)lb;
  const int range = T - look_backward;
  for (int i = 0; i < range; ++i) {
    if (silence) {
      if (speech_vote(i)) {
        int votes = 1;
        for (int j = 1; j < lb; ++j) votes += speech_vote(i + j) ? 1 : 0;
        silence = !((double)votes * inv_d >= speaking_score);
      }
    } else {
      if (silence_vote(i)) {
        int votes = 1;
        for (int j = 1; j < lb; ++j) votes += silence_vote(i + j) ? 1 : 0;
        silence = !((double)votes * inv_d <= silence_score);
      } else {
        silence = false;
      }
    }
    emit(silence);
  }
  if (is_final) {
    for (int i = range; i < T; ++i) {
      silence = hysteresis_tail(silence, speech_vote(i), silence_vote(i));
      emit(silence);
    }
  }
}

}  // namespace vadx
