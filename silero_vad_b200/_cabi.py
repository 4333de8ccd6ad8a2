"""ctypes binding of include/silero_vad_b200.h (the C ABI of libsilero_vad_b200.so).

Fails loudly when the CUDA library is missing or cannot be loaded: there is no CPU fallback.
"""
import ctypes
from pathlib import Path

from .build import LIB, build

_f32p = ctypes.c_void_p  # device or host float* passed as an integer address
_lib = None

EXPORTS = ["svad_abi_version", "svad_last_error", "svad_engine_create", "svad_engine_destroy",
           "svad_engine_set_tile_rows", "svad_engine_set_kernel", "svad_engine_set_small_batch_max", "svad_engine_set_pair_mode", "svad_engine_sm_count", "svad_engine_launch_count",
           "svad_forward_device", "svad_forward_device_pcm16", "svad_forward_device_ex", "svad_step_device", "svad_forward_host",
           "svad_collect_chunks_device", "svad_stream_open", "svad_stream_push", "svad_stream_reset", "svad_stream_close",
           "svad_forward_host_pcm16", "svad_step_host",
           "svad_segment_params_default", "svad_speech_segments",
           "svad_features_device", "svad_decoder_tape_floats", "svad_decoder_workspace_bytes", "svad_decoder_forward_device",
           "svad_decoder_backward_device", "svad_threshold_grid_device"]


class SvadError(RuntimeError):
    pass


class SegmentParams(ctypes.Structure):
    """struct svad_segment_params (include/silero_vad_b200.h)."""
    _fields_ = [("sampling_rate", ctypes.c_int32), ("use_max_poss_sil_at_max_speech", ctypes.c_int32),
                ("threshold", ctypes.c_double), ("neg_threshold", ctypes.c_double),
                ("min_speech_duration_ms", ctypes.c_double), ("max_speech_duration_s", ctypes.c_double),
                ("min_silence_duration_ms", ctypes.c_double), ("speech_pad_ms", ctypes.c_double),
                ("min_silence_at_max_speech_ms", ctypes.c_double)]


def lib():
    global _lib
    if _lib is not None:
        return _lib
    # build() compares a content hash of csrc/ + include/ with the one the library was built from and recompiles on a
    # mismatch, so Python never loads a library whose ABI or weight-tape layout differs from the sources in the tree
    path = Path(build())
    L = ctypes.CDLL(str(path))
    i64, i32, vp = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p
    L.svad_abi_version.restype = i32
    L.svad_last_error.restype = ctypes.c_char_p
    L.svad_engine_create.argtypes = [ctypes.c_char_p, i32, ctypes.POINTER(vp)]
    L.svad_engine_destroy.argtypes = [vp]
    L.svad_engine_destroy.restype = None
    L.svad_engine_set_tile_rows.argtypes = [vp, i32]
    L.svad_engine_set_kernel.argtypes = [vp, i32]
    L.svad_engine_set_small_batch_max.argtypes = [vp, i32]
    L.svad_engine_set_pair_mode.argtypes = [vp, i32]
    L.svad_engine_sm_count.argtypes = [vp]
    L.svad_engine_launch_count.argtypes = [vp]
    L.svad_engine_launch_count.restype = i64
    L.svad_forward_device.argtypes = [vp, i32, i32, i64, i64, vp, vp, vp, vp, vp, vp, i64, vp]
    L.svad_forward_device_pcm16.argtypes = [vp, i32, i32, i64, i64, vp, vp, vp, vp, vp, vp, i64, vp]
    L.svad_forward_host_pcm16.argtypes = [vp, i32, i32, i64, i64, vp, vp, vp, vp, vp, vp, i64]
    L.svad_forward_device_ex.argtypes = [vp, i32, i32, i64, i64, vp, i32, i32, vp, vp, vp, vp, vp, i64, vp]
    L.svad_stream_open.argtypes = [vp, i32, i32, ctypes.POINTER(vp)]
    L.svad_stream_push.argtypes = [vp, vp, vp]
    L.svad_stream_reset.argtypes = [vp]
    L.svad_stream_close.argtypes = [vp]
    L.svad_collect_chunks_device.argtypes = [vp, vp, i32, i64, i64, vp, vp, vp, i64, i32, vp, i64, vp, vp]
    L.svad_step_device.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp]
    L.svad_forward_host.argtypes = [vp, i32, i32, i64, i64, vp, vp, vp, vp, vp, vp, i64]
    L.svad_step_host.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    L.svad_segment_params_default.argtypes = [ctypes.POINTER(SegmentParams)]
    L.svad_segment_params_default.restype = None
    L.svad_speech_segments.argtypes = [vp, i64, i64, i64, vp, ctypes.POINTER(SegmentParams), vp, vp, i64, ctypes.POINTER(i64)]
    L.svad_features_device.argtypes = [vp, i32, i32, i64, i64, vp, vp, vp, vp]
    L.svad_decoder_tape_floats.argtypes = [i32, i64]
    L.svad_decoder_tape_floats.restype = i64
    L.svad_decoder_workspace_bytes.argtypes = [i32, i64, i32]
    L.svad_decoder_workspace_bytes.restype = i64
    L.svad_decoder_forward_device.argtypes = [vp, i32, i64] + [vp] * 12
    L.svad_decoder_backward_device.argtypes = [vp, i32, i64] + [vp] * 14
    L.svad_threshold_grid_device.argtypes = [vp, vp, vp, i64, vp, vp, vp]
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


def check(rc):
    if rc != 0:
        msg = lib().svad_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError(msg)
        raise SvadError("silero_vad_b200 error %d: %s" % (rc, msg))


class Engine:
    """Owns one svad_engine (weights resident on one CUDA device)."""

    def __init__(self, weights_path, device=0):
        self._h = ctypes.c_void_p()
        check(lib().svad_engine_create(str(weights_path).encode(), int(device), ctypes.byref(self._h)))
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.svad_engine_destroy(self._h)
            self._h = ctypes.c_void_p()

    __del__ = close

    @property
    def sm_count(self):
        return lib().svad_engine_sm_count(self._h)

    @property
    def launch_count(self):
        return lib().svad_engine_launch_count(self._h)

    def set_kernel(self, kernel):
        """0 / 'fp32' = CUDA-core kernel, 1 / 'tc' = tcgen05 split-TF32 kernel, 2 / 'h16' = tcgen05 split-fp16 two-loop kernel."""
        check(lib().svad_engine_set_kernel(self._h, {"fp32": 0, "tc": 1, "h16": 2}.get(kernel, kernel)))

    def set_pair_mode(self, on):
        check(lib().svad_engine_set_pair_mode(self._h, 1 if on else 0))

    def set_small_batch_max(self, streams):
        check(lib().svad_engine_set_small_batch_max(self._h, streams))

    def set_tile_rows(self, rows):
        check(lib().svad_engine_set_tile_rows(self._h, rows))

    def forward_device(self, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp, stream=0):
        check(lib().svad_forward_device(self._h, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp, stream))

    def forward_device_pcm16(self, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp, stream=0):
        check(lib().svad_forward_device_pcm16(self._h, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp, stream))

    def forward_device_ex(self, sr, B, L, ld, audio, sample_format, sample_stride, state_in, ctx_in, state_out, ctx_out, probs, ldp, stream=0):
        """sample_format 0 = f32, 1 = int16 PCM; sample_stride k reads every k-th stored sample (sr = k * 16000 input)."""
        check(lib().svad_forward_device_ex(self._h, sr, B, L, ld, audio, sample_format, sample_stride, state_in, ctx_in, state_out,
                                           ctx_out, probs, ldp, stream))

    def collect_chunks_device(self, wav_ptr, elem_bytes, B, ld, row_len, seg_rows, seg_bounds, drop, out_ptr, out_cap, stream=0):
        """One gather launch over a segment table (svad_collect_chunks_device); returns out_offsets[B+1] (numpy int64).
        out_ptr = 0 only sizes the result."""
        import numpy as np
        row_len = np.ascontiguousarray(row_len, np.int64)
        seg_rows = np.ascontiguousarray(seg_rows, np.int64)
        seg_bounds = np.ascontiguousarray(seg_bounds, np.int64).reshape(-1, 2)
        offs = np.zeros(B + 1, np.int64)
        check(lib().svad_collect_chunks_device(self._h, wav_ptr, elem_bytes, B, ld, row_len.ctypes.data, seg_rows.ctypes.data,
                                               seg_bounds.ctypes.data, len(seg_rows), 1 if drop else 0, out_ptr, out_cap,
                                               offs.ctypes.data, stream))
        return offs

    # ---- persistent streaming session (svad_stream_*): chunk in, probability out, no launch per chunk
    def stream_open(self, sr, nstreams=1):
        h = ctypes.c_void_p()
        check(lib().svad_stream_open(self._h, sr, nstreams, ctypes.byref(h)))
        return h

    def stream_push(self, h, chunk):
        """chunk: C-contiguous float32 numpy [nstreams, n] (or [n]); returns float32 numpy [nstreams]."""
        import numpy as np
        chunk = np.ascontiguousarray(chunk, np.float32)
        prob = np.zeros(max(1, chunk.shape[0] if chunk.ndim == 2 else 1), np.float32)
        check(lib().svad_stream_push(h, chunk.ctypes.data, prob.ctypes.data))
        return prob

    def stream_reset(self, h):
        check(lib().svad_stream_reset(h))

    def stream_close(self, h):
        check(lib().svad_stream_close(h))

    def forward_host_pcm16(self, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp):
        check(lib().svad_forward_host_pcm16(self._h, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp))

    def step_device(self, sr, B, x1, state_in, prob, state_out, stream=0):
        check(lib().svad_step_device(self._h, sr, B, x1, state_in, prob, state_out, stream))

    # ---- decoder fine-tuning (silero_vad_b200.tuning)
    def features_device(self, sr, B, L, ld, audio, ctx_in, feat, stream=0):
        check(lib().svad_features_device(self._h, sr, B, L, ld, audio, ctx_in, feat, stream))

    def decoder_forward_device(self, B, T, feat, w_ih, w_hh, b_ih, b_hh, w_head, b_head, drop, probs, tape, work, stream=0):
        check(lib().svad_decoder_forward_device(self._h, B, T, feat, w_ih, w_hh, b_ih, b_hh, w_head, b_head, drop, probs, tape, work, stream))

    def decoder_backward_device(self, B, T, feat, w_hh, w_head, drop, probs, dprobs, tape, work, dw_ih, dw_hh, db, dw_head, db_head, stream=0):
        check(lib().svad_decoder_backward_device(self._h, B, T, feat, w_hh, w_head, drop, probs, dprobs, tape, work, dw_ih, dw_hh, db,
                                                 dw_head, db_head, stream))

    def forward_host(self, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp):
        check(lib().svad_forward_host(self._h, sr, B, L, ld, audio, state_in, ctx_in, state_out, ctx_out, probs, ldp))

    def step_host(self, sr, B, x1, state_in, prob, state_out):
        check(lib().svad_step_host(self._h, sr, B, x1, state_in, prob, state_out))


def speech_segments(probs, audio_lens, params):
    """probs: C-contiguous float32 numpy [B, T]; audio_lens: int64 numpy [B].  Returns a list (per stream) of
    (start, end) integer pairs in samples at the model rate."""
    import numpy as np
    probs = np.ascontiguousarray(probs, np.float32)
    lens = np.ascontiguousarray(audio_lens, np.int64)
    B, T = probs.shape
    offs = np.zeros(B + 1, np.int64)
    cap = B * (T // 2 + 2) + 1
    bounds = np.zeros((cap, 2), np.int64)
    n = ctypes.c_int64(0)
    check(lib().svad_speech_segments(probs.ctypes.data, B, T, T, lens.ctypes.data, ctypes.byref(params), offs.ctypes.data,
                                     bounds.ctypes.data, cap, ctypes.byref(n)))
    assert n.value <= cap
    return [[(int(a), int(b)) for a, b in bounds[offs[i]:offs[i + 1]]] for i in range(B)]
