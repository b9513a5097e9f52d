"""vadx.InferenceSession -- the drop-in for `onnxruntime.InferenceSession` on the VAD hot path.

The reference scripts build a session from an .onnx file and call
``sess.run([out_name], {in_name: ndarray})`` once per chunk
(FireRedVAD/Inference_FireRed_ONNX.py:523-572).  Here the session is built from a model kind +
hyper-parameters + a state_dict of numpy weights, and the same ``run`` call goes to the CUDA
engine through the C ABI (include/vadx.h).  ``run_batch`` is the B200-native entry: S chunks
at once, device tensors in and out, asynchronous on the current stream.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import asdict

import numpy as np

from . import constants, lib, tables, weights as W


class NodeArg:
    """Mirror of onnxruntime.NodeArg: .name, .shape, .type"""

    def __init__(self, name, shape, type_):
        self.name, self.shape, self.type = name, shape, type_

    def __repr__(self):
        return f"NodeArg(name='{self.name}', type='{self.type}', shape={self.shape})"


class _Engine:
    """Owns a vadx_model handle and a growable device workspace."""

    def __init__(self, kind: str, hparams):
        import torch
        self._torch = torch
        self._lib = lib.load()
        lib.require_device()
        hp = (C.c_int32 * len(hparams))(*[int(v) for v in hparams])
        h = C.c_void_p()
        lib.check(self._lib.vadx_create(kind.encode(), hp, len(hparams), C.byref(h)))
        self._h = h
        self._ws = {}            # (device, stream handle) -> workspace: calls in flight on different streams never share scratch
        self._captured_ws = []

    def close(self):
        if getattr(self, "_h", None):
            self._lib.vadx_destroy(self._h)
            self._h = None

    __del__ = close

    def set_tensor(self, name: str, arr: np.ndarray):
        arr = np.ascontiguousarray(arr)
        dt = {np.dtype(np.int16): lib.DT_I16, np.dtype(np.float32): lib.DT_F32, np.dtype(np.int32): lib.DT_I32}[arr.dtype]
        dims = (C.c_int64 * max(arr.ndim, 1))(*(arr.shape if arr.ndim else (1,)))
        lib.check(self._lib.vadx_set_tensor(self._h, name.encode(), arr.ctypes.data, dt, dims, max(arr.ndim, 1)))

    def set_scalar(self, name: str, v: float):
        lib.check(self._lib.vadx_set_scalar(self._h, name.encode(), float(v)))

    def set_frontend(self, basis: np.ndarray, bank: np.ndarray):
        """The log-mel frontend's tensors: the interleaved DFT basis and the mel bank [n_bins, n_mels] in sparse form."""
        st, ln, w = tables.sparse_bank(bank)
        self.set_tensor("frontend.basis", basis)
        self.set_tensor("frontend.mel_start", st)
        self.set_tensor("frontend.mel_len", ln)
        self.set_tensor("frontend.mel_w", w)

    def output_frames(self, n_samples: int) -> int:
        out = C.c_int32()
        lib.check(self._lib.vadx_output_frames(self._h, n_samples, C.byref(out)))
        return out.value

    def workspace_bytes(self, n_streams: int, n_samples: int) -> int:
        out = C.c_size_t()
        lib.check(self._lib.vadx_workspace_bytes(self._h, n_streams, n_samples, C.byref(out)))
        return out.value

    def workspace(self, n_bytes: int, device, stream=None):
        """One growable scratch buffer per (device, stream): two calls enqueued on different streams may overlap on the
        GPU, so they must not share it.  A buffer that is outgrown may still be in use by work queued on ITS stream;
        record_stream keeps the caching allocator from handing the block out before that work has finished."""
        torch = self._torch
        st = stream if stream is not None else torch.cuda.current_stream(device)
        key = (device.index if device.index is not None else torch.cuda.current_device(), int(st.cuda_stream))
        ws = self._ws.get(key)
        if ws is None or ws.numel() < n_bytes:
            if ws is not None:
                ws.record_stream(st)
            with torch.cuda.device(device):
                ws = torch.empty(n_bytes, dtype=torch.uint8, device=device)
            self._ws[key] = ws
        return ws

    def forward(self, inputs, outputs, states, n_streams, n_samples, stream=None):
        dev = inputs[0].device
        need = self.workspace_bytes(n_streams, n_samples)
        ws = self.workspace(need, dev, stream)
        if self._torch.cuda.is_current_stream_capturing() and not any(ws is k for k in self._captured_ws):
            self._captured_ws.append(ws)   # a CUDA graph now holds this address: never free it (growth allocates anew)
        ins = (C.c_void_p * len(inputs))(*[None if t is None else t.data_ptr() for t in inputs])      # None = optional input absent
        outs = (C.c_void_p * len(outputs))(*[None if t is None else t.data_ptr() for t in outputs])
        sts = (C.c_void_p * max(len(states), 1))(*([t.data_ptr() for t in states] or [None]))
        lib.check(self._lib.vadx_forward(self._h, ins, outs, sts, n_streams, n_samples, ws.data_ptr(), need,
                                         lib.stream_ptr(stream)))


class FireRedSession:
    """FireRedVAD (non-stream VAD / AED) session.

    I/O contract of the reference graph (FireRedVAD/Export_FireRedVAD.py:794-807):
    ``audio`` int16 (1, 1, L) -> ``probs`` fp32 (1, odim, T), T = 1 + (L - 400) // 160.
    """
    MAX_STREAMS_PER_CALL = 32768

    def __init__(self, weights: dict, cfg: W.FireRedConfig = W.FireRedConfig(), chunk_len: int | None = 16000,
                 tensor_cores: bool = True, in_sample_rate: int = 16000):
        """tensor_cores=False keeps every contraction on the exact-fp32 FFMA kernels (debug / A-B).
        in_sample_rate != 16000 enables the wrapper's in-graph linear resampler (IN_SAMPLE_RATE,
        FireRedVAD/Export_FireRedVAD.py:389-393,431-449); chunk_len is then counted at that rate."""
        self.cfg = cfg
        self.chunk_len = chunk_len
        self.in_sample_rate = int(in_sample_rate)
        hp = [cfg.idim, cfg.R, cfg.M, cfg.H, cfg.P, cfg.N1, cfg.S1, cfg.N2 if not cfg.streaming else 0, cfg.S2,
              cfg.odim, cfg.n_fft, cfg.win_length, cfg.hop, cfg.n_mels]
        self._e = _Engine("firered", hp)
        basis, first, _ = tables.interleaved_basis(cfg.n_fft, cfg.win_length, cfg.window, "v2")
        assert first == 0
        bank = constants.kaldi_like_mel_bank(cfg.n_fft, cfg.n_mels, 16000).numpy()
        self._e.set_frontend(basis, bank)
        self._e.set_scalar("frontend.preemph", cfg.pre_emphasis)
        self._e.set_scalar("frontend.log_floor", cfg.log_floor)
        self._e.set_scalar("engine.use_tc", 1.0 if tensor_cores else 0.0)
        self._e.set_scalar("frontend.in_sample_rate", float(self.in_sample_rate))
        spec = W.firered_spec(cfg)
        for name in spec:
            if name not in weights:
                raise KeyError(f"FireRedSession: weight '{name}' missing from the state dict")
            a = np.asarray(weights[name], np.float32)
            if tuple(a.shape) != tuple(spec[name]):
                raise ValueError(f"FireRedSession: '{name}' has shape {a.shape}, expected {spec[name]}")
            self._e.set_tensor(name, a)
        L = chunk_len if chunk_len else "audio_len"
        T = self._e.output_frames(chunk_len) if chunk_len else "signal_len"
        self._inputs_meta = [NodeArg("audio", [1, 1, L], "tensor(int16)")]
        self._outputs_meta = [NodeArg("probs", [1, cfg.odim, T], "tensor(float)")]

    # ---- onnxruntime.InferenceSession surface --------------------------------------------
    def get_inputs(self):
        return list(self._inputs_meta)

    def get_outputs(self):
        return list(self._outputs_meta)

    def get_providers(self):
        return ["B200ExecutionProvider"]

    def run(self, output_names, input_feed: dict):
        """numpy in / numpy out, like ORT.  Accepts (S, 1, L) as well as the reference's (1, 1, L)."""
        import torch
        if output_names is not None and any(n != "probs" for n in output_names):
            raise ValueError(f"InvalidArgument: unknown output name in {output_names}")
        if set(input_feed) != {"audio"}:
            raise ValueError(f"InvalidArgument: expected exactly the input 'audio', got {sorted(input_feed)}")
        a = input_feed["audio"]
        if not isinstance(a, np.ndarray) or a.dtype != np.int16:
            raise ValueError("InvalidArgument: 'audio' must be a numpy int16 array (tensor(int16))")
        if a.ndim != 3 or a.shape[1] != 1:
            raise ValueError(f"InvalidArgument: 'audio' must have shape (S, 1, L), got {a.shape}")
        if self.chunk_len and a.shape[2] != self.chunk_len:
            raise ValueError(f"InvalidArgument: 'audio' length {a.shape[2]} != static axis {self.chunk_len}")
        if self.frames(a.shape[2]) < 1:
            raise ValueError(f"InvalidArgument: 'audio' length {a.shape[2]} shorter than one frame")
        d = torch.from_numpy(np.ascontiguousarray(a[:, 0, :])).cuda()
        p = self.run_batch(d)
        return [p.cpu().numpy()]

    # ---- B200-native surface ----------------------------------------------------------------
    def frames(self, n_samples: int) -> int:
        return self._e.output_frames(n_samples)

    def run_batch(self, audio, out=None, stream=None):
        """audio: cuda int16 [S, L] -> probs cuda fp32 [S, odim, T]; asynchronous on `stream`."""
        import torch
        if not (torch.is_tensor(audio) and audio.is_cuda and audio.dtype == torch.int16 and audio.dim() == 2):
            raise ValueError("run_batch: audio must be a CUDA int16 tensor of shape [S, L]")
        if not audio.is_contiguous():
            raise ValueError("run_batch: audio must be contiguous")
        S, L = audio.shape
        T = self.frames(L)
        if T < 1:
            raise ValueError(f"run_batch: {L} samples are shorter than one frame")
        if out is None:
            out = torch.empty((S, self.cfg.odim, T), dtype=torch.float32, device=audio.device)
        elif tuple(out.shape) != (S, self.cfg.odim, T) or out.dtype != torch.float32 or not out.is_contiguous():
            raise ValueError("run_batch: bad `out` tensor")
        step = self.MAX_STREAMS_PER_CALL
        for s0 in range(0, S, step):
            s1 = min(S, s0 + step)
            self._e.forward([audio[s0:s1]], [out[s0:s1]], [], s1 - s0, L, stream)
        return out


class FireRedStreamSession(FireRedSession):
    """FireRed Stream-VAD session: lookback-only DFSMN with explicit caches.

    I/O contract of the reference graph (FireRedVAD/Export_FireRedVAD.py:863-876; call site
    Inference_FireRed_ONNX.py:794-799): ``audio`` int16 (1, 1, L), ``caches_in`` fp32 (R, 1, P, (N1-1)*S1)
    -> ``probs`` fp32 (1, 1, T), ``caches_out``.  The unit axes generalise to S streams in lock-step."""

    def __init__(self, weights: dict, cfg: W.FireRedConfig | None = None, tensor_cores: bool = True):
        cfg = cfg or W.FireRedConfig(N2=0, S2=0, streaming=True)
        if not cfg.streaming:
            raise ValueError("FireRedStreamSession needs a streaming config (FireRedConfig(N2=0, streaming=True))")
        super().__init__(weights, cfg, chunk_len=None, tensor_cores=tensor_cores)
        self.lookback = (cfg.N1 - 1) * cfg.S1
        self._inputs_meta = [NodeArg("audio", [1, 1, "audio_len"], "tensor(int16)"),
                             NodeArg("caches_in", [cfg.R, 1, cfg.P, self.lookback], "tensor(float)")]
        self._outputs_meta = [NodeArg("probs", [1, cfg.odim, "T"], "tensor(float)"),
                              NodeArg("caches_out", [cfg.R, 1, cfg.P, self.lookback], "tensor(float)")]

    def new_caches(self, n_streams: int, device):
        import torch
        return torch.zeros((self.cfg.R, n_streams, self.cfg.P, self.lookback), dtype=torch.float32, device=device)

    def run_batch(self, audio, caches_in, out=None, caches_out=None, stream=None):
        """audio cuda int16 [S, L], caches_in cuda fp32 [R, S, P, Lb] -> (probs [S, odim, T], caches_out)."""
        import torch
        if not (torch.is_tensor(audio) and audio.is_cuda and audio.dtype == torch.int16 and audio.dim() == 2
                and audio.is_contiguous()):
            raise ValueError("run_batch: audio must be a contiguous CUDA int16 tensor of shape [S, L]")
        S, L = audio.shape
        shape = (self.cfg.R, S, self.cfg.P, self.lookback)
        if not (torch.is_tensor(caches_in) and caches_in.is_cuda and caches_in.dtype == torch.float32
                and tuple(caches_in.shape) == shape and caches_in.is_contiguous()):
            raise ValueError(f"run_batch: caches_in must be a contiguous CUDA fp32 tensor of shape {shape}")
        if S > self.MAX_STREAMS_PER_CALL:
            raise ValueError(f"run_batch: at most {self.MAX_STREAMS_PER_CALL} streams per call")
        T = self.frames(L)
        if T < 1:
            raise ValueError(f"run_batch: {L} samples are shorter than one frame")
        if out is None:
            out = torch.empty((S, self.cfg.odim, T), dtype=torch.float32, device=audio.device)
        if caches_out is None:
            caches_out = torch.empty_like(caches_in)
        elif caches_out.data_ptr() == caches_in.data_ptr() or tuple(caches_out.shape) != shape:
            raise ValueError("run_batch: caches_out must be a distinct tensor of the caches_in shape")
        self._e.forward([audio], [out], [caches_in, caches_out], S, L, stream)
        return out, caches_out

    def run(self, output_names, input_feed: dict):
        import torch
        names = [o.name for o in self._outputs_meta]
        if output_names is not None and any(n not in names for n in output_names):
            raise ValueError(f"InvalidArgument: unknown output name in {output_names}")
        if set(input_feed) != {"audio", "caches_in"}:
            raise ValueError(f"InvalidArgument: expected the inputs 'audio' and 'caches_in', got {sorted(input_feed)}")
        a, c = input_feed["audio"], input_feed["caches_in"]
        if not isinstance(a, np.ndarray) or a.dtype != np.int16 or a.ndim != 3 or a.shape[1] != 1:
            raise ValueError("InvalidArgument: 'audio' must be a numpy int16 array of shape (S, 1, L)")
        if a.shape[2] < self.cfg.win_length:
            raise ValueError(f"InvalidArgument: 'audio' length {a.shape[2]} shorter than one frame")
        S = a.shape[0]
        want = (self.cfg.R, S, self.cfg.P, self.lookback)
        if not isinstance(c, np.ndarray) or c.dtype != np.float32 or tuple(c.shape) != want:
            raise ValueError(f"InvalidArgument: 'caches_in' must be a numpy float32 array of shape {want}")
        d = torch.from_numpy(np.ascontiguousarray(a[:, 0, :])).cuda()
        p, co = self.run_batch(d, torch.from_numpy(np.ascontiguousarray(c)).cuda())
        res = {"probs": p, "caches_out": co}
        return [res[n].cpu().numpy() for n in (output_names or names)]


class FsmnSession:
    """FunASR FSMN-VAD session.

    I/O contract of the reference graph (FSMN/Export_FSMN_VAD.py:122-134), static audio length L:
      inputs : audio int16 (1,1,L); cache_0..3 fp32 (1,128,19,1); one_minus_speech_threshold fp32 (1,);
               noise_average_dB fp32 (1,)
      outputs: score uint8 (T,), T = L//160 + 1; cache_0..3 (new); noisy_dB fp32 ()
    `run` keeps that contract (numpy, one stream); `run_batch` is the device-resident S-stream form
    that also returns P(silence) and power_dB (the quantities the uint8 score is thresholded from).
    """
    INPUT_NAMES = ["audio", "cache_0", "cache_1", "cache_2", "cache_3", "one_minus_speech_threshold",
                   "noise_average_dB"]
    OUTPUT_NAMES = ["score", "cache_0_out", "cache_1_out", "cache_2_out", "cache_3_out", "noisy_dB"]

    def __init__(self, weights: dict, cfg: W.FsmnConfig = W.FsmnConfig(), chunk_len: int = 16000,
                 tensor_cores: bool = True, io_dtype: str = "float32"):
        """io_dtype = "float16" gives the I/O contract of the reference's fp16-optimised export (Optimize_ONNX.py
        `use_fp16`, `convert_float_to_float16(keep_io_types=False)`): caches, threshold, noise level and noisy_dB travel as
        float16 and `_inputs_meta[1].type` says so, which is what the inference script keys on (:42,:157-160).  The arithmetic
        inside stays the fp32-grade engine (the ORT fp16 kernels' own rounding is not reproducible here, DESIGN.md section 7):
        results are the fp32 graph's, rounded to float16 at the boundary."""
        if io_dtype not in ("float32", "float16"):
            raise ValueError("FsmnSession: io_dtype must be 'float32' or 'float16'")
        self.io_dtype = np.float16 if io_dtype == "float16" else np.float32
        self.cfg, self.chunk_len = cfg, int(chunk_len)
        if self.chunk_len < cfg.n_fft:
            raise ValueError(f"FsmnSession: chunk_len {chunk_len} is shorter than the {cfg.n_fft}-sample energy frame")
        hp = [cfg.input_dim, cfg.input_affine_dim, cfg.fsmn_layers, cfg.linear_dim, cfg.proj_dim, cfg.lorder,
              cfg.rorder, cfg.lstride, cfg.rstride, cfg.output_affine_dim, cfg.output_dim, cfg.n_fft, cfg.win_length,
              cfg.hop, cfg.n_mels, cfg.lfr_m, cfg.lfr_n]
        self._e = _Engine("fsmn", hp)
        basis, _first, _ = tables.interleaved_basis(cfg.n_fft, cfg.win_length, cfg.window, "v1")
        bank = constants.torchaudio_mel_bank(cfg.n_fft // 2 + 1, 20.0, 8000.0, cfg.n_mels, 16000, None, "htk").numpy()
        self._e.set_frontend(basis, bank)
        self._e.set_scalar("frontend.preemph", cfg.pre_emphasis)
        self._e.set_scalar("frontend.log_floor", cfg.log_floor)
        self._e.set_scalar("speech_2_noise_ratio", cfg.speech_2_noise_ratio)
        self._e.set_scalar("one_minus_speech_threshold", 1.0)
        self._e.set_scalar("engine.use_tc", 1.0 if tensor_cores else 0.0)
        spec = W.fsmn_spec(cfg)
        for name in spec:
            if name not in weights:
                raise KeyError(f"FsmnSession: weight '{name}' missing from the state dict")
            a = np.asarray(weights[name], np.float32)
            if tuple(a.shape) != tuple(spec[name]):
                raise ValueError(f"FsmnSession: '{name}' has shape {a.shape}, expected {spec[name]}")
            self._e.set_tensor(name, a)
        self.T = self._e.output_frames(self.chunk_len)
        self.cache_shape = (cfg.proj_dim, (cfg.lorder - 1) * cfg.lstride)
        cs = [1, cfg.proj_dim, (cfg.lorder - 1) * cfg.lstride, 1]
        ft = "tensor(float16)" if self.io_dtype == np.float16 else "tensor(float)"
        self._inputs_meta = [NodeArg("audio", [1, 1, self.chunk_len], "tensor(int16)")]
        self._inputs_meta += [NodeArg(f"cache_{i}", cs, ft) for i in range(cfg.fsmn_layers)]
        self._inputs_meta += [NodeArg("one_minus_speech_threshold", [1], ft),
                              NodeArg("noise_average_dB", [1], ft)]
        self._outputs_meta = [NodeArg("score", [self.T], "tensor(uint8)")]
        self._outputs_meta += [NodeArg(f"cache_{i}_out", cs, ft) for i in range(cfg.fsmn_layers)]
        self._outputs_meta += [NodeArg("noisy_dB", [], ft)]
        self._thr = 1.0

    def get_inputs(self):
        return list(self._inputs_meta)

    def get_outputs(self):
        return list(self._outputs_meta)

    def get_providers(self):
        return ["B200ExecutionProvider"]

    def new_caches(self, n_streams: int, device):
        import torch
        return [torch.zeros((n_streams,) + self.cache_shape, dtype=torch.float32, device=device)
                for _ in range(self.cfg.fsmn_layers)]

    def run_batch(self, audio, caches, noise_average_dB, one_minus_speech_threshold: float = 1.0, stream=None, out=None,
                  caches_out=None):
        """audio cuda int16 [S, L]; caches: list of cuda fp32 [S,128,19]; noise_average_dB cuda fp32 [S].
        -> (score u8 [S,T], new_caches, noisy_dB [S], p_silence [S,T], power_dB [S,T]); asynchronous.
        out = (score, noisy_dB, p_silence, power_dB) and caches_out (a list like caches, distinct from it) are static
        outputs to write instead of new tensors; p_silence and power_dB may be None there (not returned then)."""
        import torch
        if not (torch.is_tensor(audio) and audio.is_cuda and audio.dtype == torch.int16 and audio.dim() == 2
                and audio.is_contiguous()):
            raise ValueError("run_batch: audio must be a contiguous CUDA int16 tensor [S, L]")
        S, L = audio.shape
        if L != self.chunk_len:
            raise ValueError(f"InvalidArgument: audio length {L} != static axis {self.chunk_len}")
        n = self.cfg.fsmn_layers
        if len(caches) != n or any(tuple(c.shape) != (S,) + self.cache_shape or c.dtype != torch.float32
                                   or not c.is_cuda or not c.is_contiguous() for c in caches):
            raise ValueError(f"InvalidArgument: expected {n} contiguous CUDA fp32 caches of shape {(S,) + self.cache_shape}")
        if tuple(noise_average_dB.shape) != (S,) or noise_average_dB.dtype != torch.float32:
            raise ValueError("InvalidArgument: noise_average_dB must be fp32 [S]")
        if float(one_minus_speech_threshold) != self._thr:
            self._thr = float(one_minus_speech_threshold)
            self._e.set_scalar("one_minus_speech_threshold", self._thr)
        self._leave_window_mode()
        dev = audio.device
        if out is None:
            score = torch.empty((S, self.T), dtype=torch.uint8, device=dev)
            noisy = torch.empty((S,), dtype=torch.float32, device=dev)
            p_sil = torch.empty((S, self.T), dtype=torch.float32, device=dev)
            power = torch.empty((S, self.T), dtype=torch.float32, device=dev)
        else:
            score, noisy, p_sil, power = out
            want = ((torch.uint8, (S, self.T)), (torch.float32, (S,)), (torch.float32, (S, self.T)), (torch.float32, (S, self.T)))
            for i, (t, (dt, shape)) in enumerate(zip(out, want)):
                if (t is None and i < 2) or (t is not None and not (t.is_cuda and t.dtype == dt and tuple(t.shape) == shape
                                                                     and t.is_contiguous())):
                    raise ValueError("run_batch: out must be contiguous CUDA (score u8 [S,T], noisy_dB fp32 [S], "
                                     "p_silence fp32 [S,T] or None, power_dB fp32 [S,T] or None)")
        if caches_out is None:
            new = [torch.empty_like(c) for c in caches]
        else:
            new = list(caches_out)
            if len(new) != n or any(tuple(c.shape) != tuple(ci.shape) or c.dtype != torch.float32 or not c.is_cuda
                                    or not c.is_contiguous() or c.data_ptr() == ci.data_ptr() for c, ci in zip(new, caches)):
                raise ValueError(f"run_batch: caches_out must be {n} contiguous CUDA fp32 caches of the caches' shape, "
                                 "distinct from them")
        self._e.forward([audio, noise_average_dB], [score, noisy, p_sil, power], list(caches) + new, S, L, stream)
        return score, new, noisy, p_sil, power

    def run_windows(self, aligned, stride: int, caches, stream=None):
        """Whole-file mode: aligned cuda int16 [S, n] (chunk-aligned recordings, audio_io.align_overlapping), windows of
        chunk_len samples `stride` apart.  ONE forward covers all W = (n - chunk_len) // stride + 1 windows of every stream
        (the caches across windows are a causal FIR over the concatenated frames, see csrc/model_fsmn.cu).
        -> (p_silence [S, W, T], power_dB [S, W, T], new_caches); the gate and the look-ahead machine, which depend on the
        running background level, follow in postprocess.fsmn_gate_hysteresis_windows."""
        import torch
        if not (torch.is_tensor(aligned) and aligned.is_cuda and aligned.dtype == torch.int16 and aligned.dim() == 2
                and aligned.is_contiguous()):
            raise ValueError("run_windows: aligned must be a contiguous CUDA int16 tensor [S, n]")
        S, n = aligned.shape
        L = self.chunk_len
        if n < L or stride < 1:
            raise ValueError(f"run_windows: recordings of {n} samples are shorter than one {L}-sample window")
        Wn = (n - L) // stride + 1
        key = (Wn, int(stride), int(n))
        if getattr(self, "_win_key", None) != key:
            self._e.set_scalar("input.n_windows", float(Wn))
            self._e.set_scalar("input.window_stride", float(stride))
            self._e.set_scalar("input.stream_stride", float(n))
            self._win_key = key
        dev = aligned.device
        p_sil = torch.empty((S, Wn, self.T), dtype=torch.float32, device=dev)
        power = torch.empty((S, Wn, self.T), dtype=torch.float32, device=dev)
        new = [torch.empty_like(c) for c in caches]
        self._e.forward([aligned, None], [p_sil, None, p_sil, power], list(caches) + new, S, L, stream)
        return p_sil, power, new

    def _leave_window_mode(self):
        if getattr(self, "_win_key", None) is not None:
            self._e.set_scalar("input.n_windows", 1.0)
            self._win_key = None

    def run(self, output_names, input_feed: dict):
        import torch
        names = [o.name for o in self._outputs_meta]
        if output_names is not None and any(n not in names for n in output_names):
            raise ValueError(f"InvalidArgument: unknown output name in {output_names}")
        if set(input_feed) != set(self.INPUT_NAMES[:1] + [f"cache_{i}" for i in range(self.cfg.fsmn_layers)]
                                  + self.INPUT_NAMES[-2:]):
            raise ValueError(f"InvalidArgument: inputs must be {self.INPUT_NAMES}, got {sorted(input_feed)}")
        a = input_feed["audio"]
        if not isinstance(a, np.ndarray) or a.dtype != np.int16 or a.shape != (1, 1, self.chunk_len):
            raise ValueError(f"InvalidArgument: 'audio' must be int16 of shape (1, 1, {self.chunk_len})")
        caches = []
        for i in range(self.cfg.fsmn_layers):
            c = np.asarray(input_feed[f"cache_{i}"])
            if c.dtype != self.io_dtype or c.shape != (1,) + self.cache_shape + (1,):
                raise ValueError(f"InvalidArgument: 'cache_{i}' must be {np.dtype(self.io_dtype).name} of shape "
                                 f"{(1,) + self.cache_shape + (1,)}")
            caches.append(torch.from_numpy(np.ascontiguousarray(c[..., 0], dtype=np.float32)).cuda())
        for k in ("one_minus_speech_threshold", "noise_average_dB"):
            if np.asarray(input_feed[k]).dtype != self.io_dtype:
                raise ValueError(f"InvalidArgument: '{k}' must be {np.dtype(self.io_dtype).name}")
        thr = float(np.asarray(input_feed["one_minus_speech_threshold"], np.float32).reshape(-1)[0])
        noise = torch.from_numpy(np.asarray(input_feed["noise_average_dB"], np.float32).reshape(1)).cuda()
        score, new, noisy, _, _ = self.run_batch(torch.from_numpy(a[0]).cuda(), caches, noise, thr)
        outs = ([score[0].cpu().numpy()] + [c.cpu().numpy()[..., None].astype(self.io_dtype, copy=False) for c in new]
                + [noisy[0].cpu().numpy().astype(self.io_dtype, copy=False)])
        if output_names is None:
            return outs
        return [outs[names.index(n)] for n in output_names]


class MarbleNetSession:
    """NVIDIA Frame-VAD MarbleNet session.

    I/O contract of the reference graph (NVIDIA_Frame_VAD_Multilingual_MarbleNet/
    Export_NVIDIA_MarbleNet_VAD.py:444-457), dynamic audio axis:
      audio int16 (1,1,L) -> score_silence, score_active fp32 (1,T',1); signal_len int32 (1,) = T' - 1.
    `weights` is the NeMo state dict (un-folded); BatchNorm is folded on the host exactly like the
    reference's fold_bn_into_conv1d (:58-101).
    """
    MAX_STREAMS_PER_CALL = 32768

    def __init__(self, weights: dict, cfg: W.MarbleNetConfig = W.MarbleNetConfig(), tensor_cores: bool = True,
                 in_sample_rate: int = 16000):
        self.cfg = cfg
        hp = [cfg.feat_in, len(cfg.blocks)]
        for b in cfg.blocks:
            if not b.separable:
                raise ValueError("MarbleNetSession: only separable Jasper blocks are supported")
            hp += [b.filters, b.repeat, b.kernel, b.stride, b.dilation, 1 if b.residual else 0]
        hp += [cfg.num_classes, cfg.n_fft, cfg.win_length, cfg.hop, cfg.n_mels]
        self._e = _Engine("marblenet", hp)
        basis, _first, _ = tables.interleaved_basis(cfg.n_fft, cfg.win_length, cfg.window, "v2")
        bank = constants.torchaudio_mel_bank(cfg.n_fft // 2 + 1, 0.0, 8000.0, cfg.n_mels, 16000, "slaney", "slaney").numpy()
        self._e.set_frontend(basis, bank)
        self._e.set_scalar("frontend.preemph", cfg.pre_emphasis)
        self._e.set_scalar("frontend.log_eps", cfg.log_eps)
        self._e.set_scalar("engine.use_tc", 1.0 if tensor_cores else 0.0)
        # IN_SAMPLE_RATE != 16000: the wrapper's in-graph linear resampler (Export_NVIDIA_MarbleNet_VAD.py:180-183,236-254)
        self.in_sample_rate = int(in_sample_rate)
        self._e.set_scalar("frontend.in_sample_rate", float(self.in_sample_rate))
        spec = W.marblenet_spec(cfg)
        for name in spec:
            if name not in weights:
                raise KeyError(f"MarbleNetSession: weight '{name}' missing from the state dict")
            if tuple(np.shape(weights[name])) != tuple(spec[name]):
                raise ValueError(f"MarbleNetSession: '{name}' has shape {np.shape(weights[name])}, expected {spec[name]}")
        for name, arr in W.marblenet_fold(cfg, {k: np.asarray(v, np.float32) for k, v in weights.items()}).items():
            self._e.set_tensor(name, np.asarray(arr, np.float32))
        self._inputs_meta = [NodeArg("audio", [1, 1, "audio_len"], "tensor(int16)")]
        self._outputs_meta = [NodeArg("score_silence", [1, "signal_len", 1], "tensor(float)"),
                              NodeArg("score_active", [1, "signal_len", 1], "tensor(float)"),
                              NodeArg("signal_len", [1], "tensor(int32)")]

    def get_inputs(self):
        return list(self._inputs_meta)

    def get_outputs(self):
        return list(self._outputs_meta)

    def get_providers(self):
        return ["B200ExecutionProvider"]

    def frames(self, n_samples: int) -> int:
        """T' = frames emitted; the graph's `signal_len` output is T' - 1."""
        return self._e.output_frames(n_samples)

    def run_batch(self, audio, stream=None, out=None):
        """audio cuda int16 [S, L] -> scores cuda fp32 [2, S, T'] (plane 0 silence, plane 1 active).  out: an optional
        contiguous CUDA fp32 [2, S, T'] the scores are written to (a static output, so a call can be captured)."""
        import torch
        if not (torch.is_tensor(audio) and audio.is_cuda and audio.dtype == torch.int16 and audio.dim() == 2
                and audio.is_contiguous()):
            raise ValueError("run_batch: audio must be a contiguous CUDA int16 tensor [S, L]")
        S, L = audio.shape
        if L < 1:
            raise ValueError("InvalidArgument: empty audio")
        T = self.frames(L)
        if out is None:
            out = torch.empty((2, S, T), dtype=torch.float32, device=audio.device)
            fresh = True
        else:
            if not (torch.is_tensor(out) and out.device == audio.device and out.dtype == torch.float32
                    and tuple(out.shape) == (2, S, T) and out.is_contiguous()):
                raise ValueError(f"run_batch: out must be a contiguous fp32 tensor [2, {S}, {T}] on {audio.device}")
            fresh = False
        step = self.MAX_STREAMS_PER_CALL
        if S <= step:
            self._e.forward([audio], [out[0], out[1]], [], S, L, stream)
            return out
        for s0 in range(0, S, step):
            s1 = min(S, s0 + step)
            if fresh:
                part = torch.empty((2, s1 - s0, T), dtype=torch.float32, device=audio.device)
                self._e.forward([audio[s0:s1]], [part[0], part[1]], [], s1 - s0, L, stream)
                out[:, s0:s1] = part
            else:                                    # the planes' row ranges are contiguous: no temporary
                self._e.forward([audio[s0:s1]], [out[0, s0:s1], out[1, s0:s1]], [], s1 - s0, L, stream)
        return out

    def run(self, output_names, input_feed: dict):
        import torch
        names = [o.name for o in self._outputs_meta]
        if output_names is not None and any(n not in names for n in output_names):
            raise ValueError(f"InvalidArgument: unknown output name in {output_names}")
        if set(input_feed) != {"audio"}:
            raise ValueError(f"InvalidArgument: expected exactly the input 'audio', got {sorted(input_feed)}")
        a = input_feed["audio"]
        if not isinstance(a, np.ndarray) or a.dtype != np.int16 or a.ndim != 3 or a.shape[1] != 1:
            raise ValueError("InvalidArgument: 'audio' must be a numpy int16 array of shape (S, 1, L)")
        sc = self.run_batch(torch.from_numpy(np.ascontiguousarray(a[:, 0, :])).cuda()).cpu().numpy()
        outs = [sc[0][..., None], sc[1][..., None], np.full((a.shape[0],), sc.shape[2] - 1, np.int32)]
        if output_names is None:
            return outs
        return [outs[names.index(n)] for n in output_names]


class SileroSession:
    """Silero VAD v5 (16 kHz) -- mirrors utils_vad.OnnxWrapper (Silero/modeling_modified/utils_vad.py:10-146):
    ``model(x, sr)`` on a (B, 512) chunk keeps a 64-sample context and the (2, B, 128) LSTM state between
    calls, ``reset_states``, ``audio_forward``; plus ``run`` with the raw ORT contract
    ('input' (B,576), 'state' (2,B,128), 'sr') -> ('output' (B,1), 'stateN') and the device-resident
    ``speech_probs`` used by the batched entry point."""
    sample_rates = [16000]

    MAX_ROWS_PER_CALL = 262144      # streams x windows handled by one batched forward (bounds the workspace)

    def __init__(self, weights: dict, cfg: W.SileroConfig = W.SileroConfig(), tensor_cores: bool = True):
        import torch
        self.cfg = cfg
        spec = W.silero_spec(cfg)
        for name in spec:
            if name not in weights:
                raise KeyError(f"SileroSession: weight '{name}' missing from the state dict")
            if tuple(np.shape(weights[name])) != tuple(spec[name]):
                raise ValueError(f"SileroSession: '{name}' has shape {np.shape(weights[name])}, expected {spec[name]}")
        dense = W.silero_dense_layers(cfg, weights)
        hp = [cfg.window, cfg.context, cfg.reflect_pad, cfg.n_fft, cfg.hop, cfg.hidden, len(dense)]
        for D, _b in dense:
            hp += [D.shape[0], D.shape[1]]
        self._e = _Engine("silero", hp)
        fb = np.asarray(weights["stft.forward_basis_buffer"], np.float32)[:, 0, :]     # [2F, n_fft]
        F = cfg.n_bins
        ld = (2 * F + 3) // 4 * 4
        basis = np.zeros((cfg.n_fft, ld), np.float32)
        basis[:, 0:2 * F:2] = fb[:F].T
        basis[:, 1:2 * F:2] = fb[F:].T
        self._e.set_tensor("frontend.basis", basis)
        for i, (D, b) in enumerate(dense):
            self._e.set_tensor(f"enc.{i}.weight", D)
            self._e.set_tensor(f"enc.{i}.bias", b)
        self._e.set_tensor("rnn.weight_ih", np.asarray(weights["decoder.rnn.weight_ih"], np.float32))
        self._e.set_tensor("rnn.weight_hh", np.asarray(weights["decoder.rnn.weight_hh"], np.float32))
        self._e.set_tensor("rnn.bias", (np.asarray(weights["decoder.rnn.bias_ih"], np.float32)
                                        + np.asarray(weights["decoder.rnn.bias_hh"], np.float32)))
        self._e.set_tensor("head.weight", np.asarray(weights["decoder.decoder.2.weight"], np.float32)[:, :, 0])
        self._e.set_tensor("head.bias", np.asarray(weights["decoder.decoder.2.bias"], np.float32))
        self._e.set_scalar("engine.use_tc", 1.0 if tensor_cores else 0.0)
        self._row_stride = None
        self._dev = torch.device("cuda", torch.cuda.current_device())
        n_in = cfg.window + cfg.context
        self._inputs_meta = [NodeArg("input", [None, n_in], "tensor(float)"), NodeArg("state", [2, None, cfg.hidden], "tensor(float)"),
                             NodeArg("sr", [], "tensor(int64)")]
        self._outputs_meta = [NodeArg("output", [None, 1], "tensor(float)"), NodeArg("stateN", [2, None, cfg.hidden], "tensor(float)")]
        self.reset_states()

    # ---- ORT surface of the opaque silero_vad.onnx session the reference's OnnxWrapper holds (utils_vad.py:33-61,119-123)
    def get_inputs(self):
        return list(self._inputs_meta)

    def get_outputs(self):
        return list(self._outputs_meta)

    def get_providers(self):
        return ["B200ExecutionProvider"]

    # ---- raw graph ---------------------------------------------------------------------------
    def step(self, x, state, row_stride: int | None = None, stream=None):
        """x: CUDA fp32, S rows of 576 valid samples spaced `row_stride` apart (default: contiguous
        [S,576]); state CUDA fp32 [2,S,128] -> (out [S,1], new_state)."""
        import torch
        n_in = self.cfg.window + self.cfg.context
        S = state.shape[1]
        stride = int(row_stride) if row_stride is not None else n_in
        if stride != self._row_stride:
            self._e.set_scalar("input.row_stride", float(stride))
            self._row_stride = stride
        out = torch.empty((S, 1), dtype=torch.float32, device=state.device)
        new_state = torch.empty_like(state)
        self._e.forward([x], [out], [state, new_state], S, n_in, stream)
        return out, new_state

    def run(self, output_names, input_feed: dict):
        import torch
        if set(input_feed) != {"input", "state", "sr"}:
            raise ValueError(f"InvalidArgument: inputs must be input/state/sr, got {sorted(input_feed)}")
        x = np.asarray(input_feed["input"])
        st = np.asarray(input_feed["state"])
        if int(np.asarray(input_feed["sr"])) != 16000:
            raise ValueError("Supported sampling rates: [16000]")
        if x.dtype != np.float32 or x.ndim != 2 or x.shape[1] != self.cfg.window + self.cfg.context:
            raise ValueError(f"InvalidArgument: 'input' must be fp32 (B, {self.cfg.window + self.cfg.context})")
        if st.dtype != np.float32 or st.shape != (2, x.shape[0], self.cfg.hidden):
            raise ValueError(f"InvalidArgument: 'state' must be fp32 (2, {x.shape[0]}, {self.cfg.hidden})")
        out, new = self.step(torch.from_numpy(np.ascontiguousarray(x)).cuda(), torch.from_numpy(np.ascontiguousarray(st)).cuda())
        outs = [out.cpu().numpy(), new.cpu().numpy()]
        names = ["output", "stateN"]
        if output_names is None:
            return outs
        return [outs[names.index(n)] for n in output_names]

    # ---- OnnxWrapper surface -------------------------------------------------------------------
    def reset_states(self, batch_size=1):
        import torch
        self._state = torch.zeros((2, batch_size, self.cfg.hidden), dtype=torch.float32, device=self._dev)
        self._context = None
        self._last_sr = 0
        self._last_batch_size = 0

    def _validate_input(self, x, sr: int):
        if x.dim() == 1:
            x = x.unsqueeze(0)
        if x.dim() > 2:
            raise ValueError(f"Too many dimensions for input audio chunk {x.dim()}")
        if sr != 16000 and (sr % 16000 == 0):
            x = x[:, ::sr // 16000]
            sr = 16000
        if sr not in self.sample_rates:
            raise ValueError(f"Supported sampling rates: {self.sample_rates} (or multiply of 16000)")
        if sr / x.shape[1] > 31.25:
            raise ValueError("Input audio chunk is too short")
        return x, sr

    def __call__(self, x, sr: int = 16000):
        import torch
        x, sr = self._validate_input(x, sr)
        if x.shape[-1] != self.cfg.window:
            raise ValueError(f"Provided number of samples is {x.shape[-1]} (Supported values: 256 for 8000 sample rate, 512 for 16000)")
        b = x.shape[0]
        if not self._last_batch_size or (self._last_sr and self._last_sr != sr) or self._last_batch_size != b:
            self.reset_states(b)
        if self._context is None:
            self._context = torch.zeros((b, self.cfg.context), dtype=torch.float32, device=self._dev)
        xd = torch.cat([self._context, x.to(self._dev, torch.float32)], dim=1).contiguous()
        out, self._state = self.step(xd, self._state)
        self._context = xd[:, -self.cfg.context:]
        self._last_sr, self._last_batch_size = sr, b
        return out.cpu() if not x.is_cuda else out

    def audio_forward(self, x, sr: int = 16000):
        x, sr = self._validate_input(x, sr)
        probs = self.speech_probs(x.to(self._dev, dtype=self._state.dtype).contiguous())
        return probs.cpu()

    # ---- B200-native surface ---------------------------------------------------------------------
    def speech_probs_graph(self, audio):
        """speech_probs with the per-window kernel sequence (10 launches) captured once into a CUDA graph:
        each window costs one strided copy into a static buffer, one graph replay and one copy out.
        The static buffers and the graph are kept per (streams, device) and reused across calls."""
        import torch
        c = self.cfg
        S, n = audio.shape
        n_win = (n + c.window - 1) // c.window
        if n_win < 3:
            return self.speech_probs(audio)
        padded = torch.zeros((S, c.context + n_win * c.window), dtype=torch.float32, device=audio.device)
        padded[:, c.context:c.context + n] = audio
        n_in = c.window + c.context
        probs = torch.empty((n_win, S, 1), dtype=torch.float32, device=audio.device)
        runners = self.__dict__.setdefault("_graph_runners", {})
        r = runners.get((S, str(audio.device)))
        if r is None:
            r = {"x": torch.empty((S, n_in), dtype=torch.float32, device=audio.device),
                 "state": torch.zeros((2, S, c.hidden), dtype=torch.float32, device=audio.device),
                 "nxt": torch.empty((2, S, c.hidden), dtype=torch.float32, device=audio.device),
                 "out": torch.empty((S, 1), dtype=torch.float32, device=audio.device), "graph": None}
            runners[(S, str(audio.device))] = r
        x, state, nxt, out = r["x"], r["state"], r["nxt"], r["out"]
        state.zero_()
        if self._row_stride != n_in:
            self._e.set_scalar("input.row_stride", float(n_in))
            self._row_stride = n_in

        def step():
            self._e.forward([x], [out], [state, nxt], S, n_in, None)
            state.copy_(nxt)

        for t in range(n_win):
            x.copy_(padded[:, t * c.window:t * c.window + n_in])
            if r["graph"] is None and t == 0:
                step()                      # first ever window eager: uploads constants, sizes the workspace
            else:
                if r["graph"] is None:
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        step()
                    r["graph"] = g
                r["graph"].replay()
            probs[t].copy_(out)
        self._final_state = state.clone()
        return probs[:, :, 0].transpose(0, 1).contiguous()

    def forward_windows(self, x, out, state_in, state_out, n_windows: int, row_stride: int, stream=None):
        """One forward over n_windows consecutive 512-sample windows of S streams, read in place: x CUDA fp32 rows
        row_stride floats apart, window w of row s at columns [w*512, w*512 + 576) (64 context samples, then the
        window); out fp32 [n_windows][S][1]; state_in -> state_out fp32 [2][S][128], distinct.  It only enqueues
        library launches, so a CUDA graph can capture it: the engine scalars it sets are read on the host when the
        launches are enqueued, and input.n_windows is back at 1 on return."""
        c = self.cfg
        if row_stride != self._row_stride:
            self._e.set_scalar("input.row_stride", float(row_stride))
            self._row_stride = row_stride
        self._e.set_scalar("input.n_windows", float(n_windows))
        try:
            self._e.forward([x], [out], [state_in, state_out], state_in.shape[1], c.window + c.context, stream)
        finally:
            self._e.set_scalar("input.n_windows", 1.0)

    def speech_probs(self, audio, stream=None):
        """audio: CUDA fp32 [S, n] (already scaled by 1/32768) -> probs CUDA fp32 [S, ceil(n/512)].
        One graph step per 32 ms window for all S streams; the context is not copied: every window
        is a strided view of the zero-prefixed, zero-padded signal; the LSTM state stays in HBM."""
        import torch
        c = self.cfg
        if not (torch.is_tensor(audio) and audio.is_cuda and audio.dtype == torch.float32 and audio.dim() == 2):
            raise ValueError("speech_probs: audio must be a CUDA fp32 tensor [S, n]")
        S, n = audio.shape
        n_win = (n + c.window - 1) // c.window
        padded = torch.zeros((S, c.context + n_win * c.window), dtype=torch.float32, device=audio.device)
        padded[:, c.context:c.context + n] = audio
        probs = torch.empty((n_win, S, 1), dtype=torch.float32, device=audio.device)
        state = torch.zeros((2, S, c.hidden), dtype=torch.float32, device=audio.device)
        stride = padded.shape[1]
        nxt = torch.empty_like(state)
        # blocks of windows per call: the state-free part of the graph (STFT, encoder, input half of the gates)
        # runs once over streams x windows rows, only the recurrence runs per window (input.n_windows)
        block = max(1, min(n_win, self.MAX_ROWS_PER_CALL // max(S, 1)))
        t = 0
        while t < n_win:
            wb = min(block, n_win - t)
            self.forward_windows(padded[:, t * c.window:], probs[t:t + wb], state, nxt, wb, stride, stream)
            state, nxt = nxt, state
            t += wb
        self._final_state = state
        return probs[:, :, 0].transpose(0, 1).contiguous()


def InferenceSession(kind: str, weights: dict, config=None, **kw):
    """Factory with the reference's constructor name; `kind` replaces the .onnx path."""
    if kind == "firered":
        return FireRedSession(weights, config or W.FireRedConfig(), **kw)
    if kind == "firered_stream":
        return FireRedStreamSession(weights, config, **kw)
    if kind == "fsmn":
        return FsmnSession(weights, config or W.FsmnConfig(), **kw)
    if kind == "marblenet":
        return MarbleNetSession(weights, config or W.MarbleNetConfig(), **kw)
    if kind == "silero":
        return SileroSession(weights, config or W.SileroConfig(), **kw)
    raise ValueError(f"unknown model kind {kind!r}")
