"""Model object with the reference's duck-typed surface, backed by the CUDA engine.

Mirrors (same names, argument meaning, error types and messages):
  load_silero_vad()                       /root/reference/src/silero_vad/model.py:6-36
  model(x, sr), reset_states(),           silero_vad.jit::forward / reset_states / audio_forward and the
  audio_forward(x, sr), _validate_input   readable twin OnnxWrapper, src/silero_vad/utils_vad.py:33-110
PyTorch is used for device memory and streams only; all arithmetic happens in libsilero_vad_b200.so.
There is no CPU path: constructing the model without a CUDA device raises.
"""
from pathlib import Path

import torch

from . import _cabi

WEIGHTS = Path(__file__).resolve().parent / "data" / "silero_vad_v6.weights"


def _ptr(t):
    return 0 if t is None else t.data_ptr()


class SileroVADB200:
    sample_rates = [8000, 16000]

    def __init__(self, device=None, weights=None):
        if not torch.cuda.is_available():
            raise RuntimeError("silero_vad_b200 needs a CUDA device (B200 / sm_100a); there is no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else torch.device(device).index or 0)
        self.weights = Path(weights or WEIGHTS)   # the SVADW001 container the engine was built from (stock or save_tuned output)
        self.engine = _cabi.Engine(self.weights, self.device.index)
        self.reset_states()

    # ------------------------------------------------------------------ reference surface
    def reset_states(self, batch_size=1):
        """Forget (h, c), the audio context, the last sr and batch size (utils_vad.py:51-55)."""
        self._state = None      # f32[2, B, 128] on device
        self._context = None    # f32[B, ctx] on device
        self._last_sr = 0
        self._last_batch_size = 0

    def _validate_input(self, x, sr: int, device_decimation=False):
        """utils_vad.py:33-49.  With device_decimation the `x[:, ::step]` slice of sr = k * 16000 input is NOT taken here:
        (x, 16000, step) is returned and the kernel reads every step-th sample itself (SURVEY.md section 8(f)-2)."""
        if not torch.is_tensor(x):
            x = torch.as_tensor(x)
        if x.dim() == 1:
            x = x.unsqueeze(0)
        if x.dim() > 2:
            raise ValueError(f"Too many dimensions for input audio chunk {x.dim()}")
        step = 1
        if sr != 16000 and (sr % 16000 == 0):
            step = sr // 16000
            if not device_decimation:
                x = x[:, ::step]
            sr = 16000
        if sr not in self.sample_rates:
            raise ValueError(f"Supported sampling rates: {self.sample_rates} (or multiply of 16000)")
        n_model = -(-x.shape[1] // step) if device_decimation else x.shape[1]
        if n_model == 0 or sr / n_model > 31.25:
            raise ValueError("Input audio chunk is too short")
        if device_decimation:
            return x, sr, step
        return x, sr

    def _to_device(self, x, keep_pcm16=False):
        if keep_pcm16 and x.dtype == torch.int16:
            return x.to(device=self.device, non_blocking=True).contiguous()
        if x.dtype == torch.int16:   # PCM -> [-1, 1) like the reference's loaders (int16 / 32768)
            return x.to(device=self.device, non_blocking=True).to(torch.float32).mul_(1.0 / 32768.0).contiguous()
        return x.to(device=self.device, dtype=torch.float32, non_blocking=True).contiguous()

    def __call__(self, x, sr: int):
        x, sr, step = self._validate_input(x, sr, device_decimation=True)
        num_samples = 512 if sr == 16000 else 256
        raw = x.shape[-1]
        if -(-raw // step) != num_samples:
            raise ValueError(f"Provided number of samples is {-(-raw // step)} (Supported values: 256 for 8000 sample rate, 512 for 16000)")
        batch_size = x.shape[0]
        context_size = 64 if sr == 16000 else 32
        if self._last_sr and self._last_sr != sr:
            self.reset_states()
        if self._last_batch_size and self._last_batch_size != batch_size:
            self.reset_states()
        in_device = x.device
        with torch.cuda.device(self.device):
            xd = self._to_device(x)
            if self._state is None:
                self._state = torch.zeros(2, batch_size, 128, device=self.device)
            if self._context is None:
                self._context = torch.zeros(batch_size, context_size, device=self.device)
            out = torch.empty(batch_size, 1, device=self.device)
            st = torch.cuda.current_stream(self.device).cuda_stream
            # one chunk: state and context are read, advanced and written back in place by the kernel
            self.engine.forward_device_ex(sr, batch_size, raw, xd.stride(0), _ptr(xd), 0, step, _ptr(self._state), _ptr(self._context),
                                          _ptr(self._state), _ptr(self._context), _ptr(out), 1, st)
        self._last_sr = sr
        self._last_batch_size = batch_size
        return out if in_device == self.device else out.to(in_device)

    forward = __call__

    def audio_forward(self, x, sr: int):
        """All chunk probabilities of B streams in one fused launch -> f32[B, ceil(L/n)] on the CPU
        (utils_vad.py:94-110: validate, reset, zero-pad the tail, loop, cat, .cpu())."""
        return self.audio_forward_device(x, sr).cpu()

    # ------------------------------------------------------------------ extensions
    def audio_forward_device(self, x, sr: int, reset=True):
        """Like audio_forward but leaves the probabilities on the GPU; with reset=False continues from the
        carried state/context (long streams fed in pieces whose length is a multiple of the chunk size).
        int16 tensors are taken as PCM and read by the kernel directly (half the bytes, same probabilities)."""
        x, sr, step = self._validate_input(x, sr, device_decimation=True)
        if reset:
            self.reset_states()
        n = 512 if sr == 16000 else 256
        ctx = 64 if sr == 16000 else 32
        B, L = x.shape                      # stored samples; the model sees every step-th one
        T = (-(-L // step) + n - 1) // n
        if self._last_sr and self._last_sr != sr:
            self.reset_states()
        if self._last_batch_size and self._last_batch_size != B:
            self.reset_states()
        with torch.cuda.device(self.device):
            xd = self._to_device(x, keep_pcm16=True)
            if self._state is None:
                self._state = torch.zeros(2, B, 128, device=self.device)
            if self._context is None:
                self._context = torch.zeros(B, ctx, device=self.device)
            probs = torch.empty(B, T, device=self.device)
            st = torch.cuda.current_stream(self.device).cuda_stream
            self.engine.forward_device_ex(sr, B, L, xd.stride(0), _ptr(xd), 1 if xd.dtype == torch.int16 else 0, step, _ptr(self._state),
                                          _ptr(self._context), _ptr(self._state), _ptr(self._context), _ptr(probs), max(T, 1), st)
        self._last_sr = sr
        self._last_batch_size = B
        return probs

    def get_states(self):
        """(state f32[2,B,128], context f32[B,ctx]) clones, to park a set of streams (SURVEY.md section 5)."""
        return (None if self._state is None else self._state.clone(), None if self._context is None else self._context.clone(),
                self._last_sr, self._last_batch_size)

    def set_states(self, saved):
        """Resume streams parked with get_states().  The tensors are CLONED onto this model's device (the kernels advance
        state and context in place, so the caller's snapshot must stay what it was and can be restored again) and their
        shapes are checked against the recorded batch size / sample rate: they are handed to the kernel as raw pointers."""
        state, context, last_sr, last_bs = saved
        if (state is None) != (context is None):
            raise ValueError("state and context must both be given or both be None")
        if state is not None:
            if last_sr not in (8000, 16000) or last_bs < 1:
                raise ValueError("a saved state needs the sample rate and batch size it belongs to")
            ctx = 64 if last_sr == 16000 else 32
            if tuple(state.shape) != (2, last_bs, 128) or tuple(context.shape) != (last_bs, ctx):
                raise ValueError(f"expected state [2, {last_bs}, 128] and context [{last_bs}, {ctx}], got {tuple(state.shape)} and {tuple(context.shape)}")
            state = state.detach().to(device=self.device, dtype=torch.float32, copy=True).contiguous()
            context = context.detach().to(device=self.device, dtype=torch.float32, copy=True).contiguous()
        self._state, self._context, self._last_sr, self._last_batch_size = state, context, last_sr, last_bs

    def stream(self, sr: int = 16000, nstreams: int = 1):
        """A persistent low-latency session (svad_stream_*): a duck-typed model object for `VADIterator` and other chunk-by-chunk
        callers whose `__call__` costs one PCIe round trip instead of a launch + two copies + a sync."""
        return StreamSession(self, sr, nstreams)

    def eval(self):
        return self

    def to(self, *args, **kwargs):
        return self


class StreamSession:
    """model(chunk, sr) / reset_states() over a resident cluster kernel fed through mapped host memory.  Same protocol as the
    reference model object for streaming callers (utils_vad.py:507-549): chunks of exactly n samples, float32, [n] or [nstreams, n];
    returns a CPU tensor [nstreams, 1].  Close it (or use it as a context manager) to release its 8 SMs."""
    sample_rates = [8000, 16000]

    def __init__(self, model, sr, nstreams):
        if sr not in self.sample_rates:
            raise ValueError(f"Supported sampling rates: {self.sample_rates}")
        self.engine, self.sr, self.nstreams = model.engine, sr, nstreams
        self.n = 512 if sr == 16000 else 256
        self._h = self.engine.stream_open(sr, nstreams)

    def reset_states(self, batch_size=1):
        self.engine.stream_reset(self._h)

    def __call__(self, x, sr: int):
        if sr != self.sr:
            raise ValueError(f"this session runs at {self.sr} Hz")
        x = torch.as_tensor(x, dtype=torch.float32)
        if x.dim() == 1:
            x = x.unsqueeze(0)
        if x.dim() != 2 or x.shape[0] != self.nstreams or x.shape[1] != self.n:
            raise ValueError(f"Provided number of samples is {x.shape[-1]} (Supported values: 256 for 8000 sample rate, 512 for 16000)")
        return torch.from_numpy(self.engine.stream_push(self._h, x.contiguous().numpy())).unsqueeze(1)

    def close(self):
        if self._h is not None:
            self.engine.stream_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def load_silero_vad(onnx=False, opset_version=16, device=None):
    """Drop-in for silero_vad.load_silero_vad (model.py:6-36).  `onnx` / `opset_version` select between
    files that hold the same network in the reference; here they only keep the reference's argument
    checking (unknown opset with onnx=True raises) -- every variant runs the CUDA engine."""
    available_ops = [15, 16]
    if onnx and opset_version not in available_ops:
        raise Exception(f'Available ONNX opset_version: {available_ops}')
    model = SileroVADB200(device=device)
    if onnx and opset_version == 15:
        model.sample_rates = [16000]   # silero_vad_16k_op15.onnx is 16 kHz only (utils_vad.py:27-29)
    return model
