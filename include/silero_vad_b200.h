/*
 * silero_vad_b200.h -- C ABI of the B200-native Silero-VAD engine (libsilero_vad_b200.so).
 *
 * The reference has no C ABI of its own: its boundary is the duck-typed Python model object
 * (src/silero_vad/utils_vad.py:10-110, silero_vad.jit::forward) and, for every native example, the
 * ONNX I/O contract   input f32[B, ctx+n], state f32[2,B,128], sr -> output f32[B,1], stateN f32[2,B,128]
 * (src/silero_vad/utils_vad.py:80-82 ; examples/cpp/silero-vad-onnx.cpp:103-112,176-195 ;
 *  examples/rust-example/src/silero.rs:42-83 ; examples/java-wav-file-example/.../SileroVadOnnxModel.java:155-215).
 * These entry points are what an FFI binding for that contract binds instead of an onnxruntime
 * session: plain pointers and sizes, no torch types.  INTEGRATION.md shows the reference-side stubs.
 *
 * Conventions: every function returns 0 on success or a negative SVAD_E* code; svad_last_error()
 * gives the message for the calling thread.  "device" pointers are CUDA device pointers on the
 * engine's device; `stream` is a cudaStream_t (NULL = legacy default stream).  sr is 16000 (n = 512,
 * ctx = 64) or 8000 (n = 256, ctx = 32).  An engine is not thread-safe (like the reference object).
 * There is no CPU fallback: without a CUDA device svad_engine_create fails.
 */
#ifndef SILERO_VAD_B200_H
#define SILERO_VAD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVAD_OK 0
#define SVAD_EINVAL (-1)   /* bad argument (shape, sr, null pointer) */
#define SVAD_EWEIGHTS (-2) /* weight container missing / malformed */
#define SVAD_ECUDA (-3)    /* CUDA runtime error (message in svad_last_error) */
#define SVAD_ENOMEM (-4)

typedef struct svad_engine svad_engine;

/* ABI version of this header (bumped on incompatible change). */
int svad_abi_version(void);
const char* svad_last_error(void);

/* Load `weights_path` (SVADW001 container holding the 28 tensors of silero_vad.jit's state_dict, both
 * branches), pack them for the kernels and upload to CUDA device `device`.
 * Replaces: load_silero_vad() (src/silero_vad/model.py:6-36) / Ort::Session construction
 * (examples/cpp/silero-vad-onnx.cpp:86-101). */
int svad_engine_create(const char* weights_path, int device, svad_engine** out);
void svad_engine_destroy(svad_engine* e);

/* Streams per CTA tile = 4*rows; rows in [4,8], 0 = choose per call (default). Testing / tuning knob. */
int svad_engine_set_tile_rows(svad_engine* e, int rows);
/* Kernel selection for batches above the small-batch limit:
 *   2 = svad_fused_h16 (default): every contraction, the STFT included (as the reference's dense DFT-basis product), on tcgen05 with
 *       fp16 split-precision operands (x.w = x_hi.w_hi + x_lo.w_hi + x_hi.w_lo, fp32 accumulate in TMEM), two software-pipelined
 *       loops per CTA;
 *   1 = svad_fused_tc: encoder + LSTM on tcgen05 with tf32 split precision, STFT as an FFT on the CUDA cores;
 *   0 = svad_fused_fp32: all-fp32 CUDA-core kernel.
 * All meet the parity bar; their probabilities differ by ~5e-6. */
int svad_engine_set_kernel(svad_engine* e, int kernel);
/* Batches of up to `streams` streams run on the small-batch cluster kernel (8-CTA clusters with the network split
 * across their shared memories; the latency path).  Default 256 (measured crossover with the tile kernels); 0 disables it. */
int svad_engine_set_small_batch_max(svad_engine* e, int streams);
/* svad_fused_h16 in CTA pairs (thread-block clusters of 2): each CTA of a pair fetches half of every weight slab and multicasts it
 * into both shared memories, which halves the bytes the kernel reads out of L2 (same probabilities, bit for bit).  Default on for
 * batches of >= 64 streams (environment SVAD_H16_PAIR=0 turns the default off); falls back to single CTAs when the device cannot
 * co-schedule pairs. */
int svad_engine_set_pair_mode(svad_engine* e, int on);
/* Number of SMs of the engine's device. */
int svad_engine_sm_count(const svad_engine* e);
/* Kernel launches issued by this engine so far (bench.py's gpu_launches). */
int64_t svad_engine_launch_count(const svad_engine* e);

/* Bulk path: probabilities of every chunk of B independent streams in one fused kernel launch.
 * Replaces: model.audio_forward(x, sr) (src/silero_vad/utils_vad.py:94-110, silero_vad.jit::audio_forward)
 * with the carried state made explicit so long streams can be fed in pieces.
 *   d_audio      f32[B][ld]   L valid samples per row; the tail is zero-padded to T*n, T = ceil(L/n)
 *   d_state_in   f32[2][B][128] or NULL (zeros = reset_states())     (h, c)
 *   d_ctx_in     f32[B][ctx]    or NULL (zeros)                      last ctx samples before d_audio[.][0]
 *   d_state_out  f32[2][B][128] or NULL ; may alias d_state_in
 *   d_ctx_out    f32[B][ctx]    or NULL ; may alias d_ctx_in
 *   d_probs      f32[B][ldp], ldp >= T */
int svad_forward_device(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const float* d_audio,
                        const float* d_state_in, const float* d_ctx_in, float* d_state_out, float* d_ctx_out,
                        float* d_probs, int64_t ldp, void* stream);

/* Same, with int16 PCM samples (scaled by 2^-15 on load = the int16/32768 convention of examples/cpp/wav.h:95-136
 * and examples/onnx_sequence/run.py:115-119): half the HBM / PCIe bytes per chunk, bit-identical probabilities. */
int svad_forward_device_pcm16(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const int16_t* d_audio,
                              const float* d_state_in, const float* d_ctx_in, float* d_state_out, float* d_ctx_out,
                              float* d_probs, int64_t ldp, void* stream);

/* General form of the two calls above.  sample_format: 0 = f32, 1 = int16 PCM.  sample_stride k >= 1: rows hold
 * sr_in = k * sr audio and the kernel reads every k-th stored sample -- the reference's `x[:, ::step]` decimation for
 * sampling rates that are a multiple of 16000 (src/silero_vad/utils_vad.py:39-42, 301-305) done by the load itself.
 * L counts STORED samples per row; the model sees ceil(L / k) of them. */
int svad_forward_device_ex(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const void* d_audio, int sample_format,
                           int sample_stride, const float* d_state_in, const float* d_ctx_in, float* d_state_out,
                           float* d_ctx_out, float* d_probs, int64_t ldp, void* stream);

/* One chunk, the stateless ONNX contract (utils_vad.py:80-82; examples/cpp/silero-vad-onnx.cpp:176-195):
 *   d_input f32[B][ctx+n] (context already prepended), d_state_in f32[2][B][128] (NULL = zeros)
 *   -> d_prob f32[B], d_state_out f32[2][B][128] (may alias d_state_in). */
int svad_step_device(svad_engine* e, int sr, int B, const float* d_input, const float* d_state_in, float* d_prob,
                     float* d_state_out, void* stream);

/* Host-buffer twins: same semantics with host pointers; the host<->device copies are part of the call
 * (pinned staging inside the engine).  These are what bench.py's `e2e` times. */
int svad_forward_host(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const float* audio, const float* state_in,
                      const float* ctx_in, float* state_out, float* ctx_out, float* probs, int64_t ldp);
int svad_forward_host_pcm16(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const int16_t* audio, const float* state_in,
                            const float* ctx_in, float* state_out, float* ctx_out, float* probs, int64_t ldp);
int svad_step_host(svad_engine* e, int sr, int B, const float* input, const float* state_in, float* prob,
                   float* state_out);

/* ---- persistent streaming session (low-latency path, BASELINE configs[1]) ------------------------------
 * Replaces the reference's per-chunk streaming call, one model invocation + `.item()` per 32 ms chunk
 * (src/silero_vad/utils_vad.py:507-549 VADIterator.__call__; examples/cpp/silero-vad-onnx.cpp:167-197 predict()): one cluster of
 * 8 CTAs stays resident on the GPU with the whole network in its shared memory and (h, c) + audio context on chip, and is fed
 * through a mailbox in mapped pinned host memory.  svad_stream_push costs one PCIe round trip plus the compute: no kernel launch,
 * no cudaMemcpy, no stream synchronisation per chunk.  Up to 4 streams per session (they advance together, one chunk each per push).
 * The session occupies 8 SMs until closed; the kernel ends by itself after ~30 s without a chunk (push then reports an error). */
typedef struct svad_stream svad_stream;
int svad_stream_open(svad_engine* e, int sr, int nstreams, svad_stream** out);
/* chunk f32[nstreams][n] (host, n = 512 @16 kHz / 256 @8 kHz) -> prob f32[nstreams]; state and context carry over between pushes */
int svad_stream_push(svad_stream* s, const float* chunk, float* prob);
/* forget (h, c) and the context before the next chunk (model.reset_states(), utils_vad.py:51-55) */
int svad_stream_reset(svad_stream* s);
int svad_stream_close(svad_stream* s);

/* ---- speech segments from probabilities (host; the automaton of get_speech_timestamps) -------------
 * Replaces: src/silero_vad/utils_vad.py:315-319,338-440 (one stream) and the native port
 * examples/cpp/silero-vad-onnx.cpp:199-331; batched over B streams here.  Units are samples at the MODEL
 * rate (after the reference's `audio[::step]` decimation); seconds / `*step` conversion stays with the caller
 * (utils_vad.py:442-450).  Field defaults = the reference's keyword defaults (utils_vad.py:212-227). */
typedef struct svad_segment_params {
    int32_t sampling_rate;                 /* 16000 or 8000 */
    int32_t use_max_poss_sil_at_max_speech; /* bool */
    double threshold;                      /* 0.5 */
    double neg_threshold;                  /* NaN = max(threshold - 0.15, 0.01) */
    double min_speech_duration_ms;         /* 250 */
    double max_speech_duration_s;          /* +inf */
    double min_silence_duration_ms;        /* 100 */
    double speech_pad_ms;                  /* 30 */
    double min_silence_at_max_speech_ms;   /* 98 */
} svad_segment_params;

void svad_segment_params_default(svad_segment_params* p);

/* probs f32[B][ldp] (T valid per row), audio_len[B] in samples.  Writes seg_offsets[B+1] (prefix sums) and up
 * to `cap` (start,end) pairs into seg_bounds[2*cap] (may be NULL to only count); *n_total = segments found. */
int svad_speech_segments(const float* probs, int64_t B, int64_t T, int64_t ldp, const int64_t* audio_len,
                         const svad_segment_params* p, int64_t* seg_offsets, int64_t* seg_bounds, int64_t cap,
                         int64_t* n_total);

/* ---- collect_chunks / drop_chunks as ONE device gather ------------------------------------------------
 * Replaces: src/silero_vad/utils_vad.py:552-646 (`torch.cat([wav[s:e] for ...])` / its complement), batched over B rows
 * so that speech-only audio stays on the GPU for a downstream stage.
 *   d_wav       [B][ld] elements of elem_bytes (4 = f32, 2 = int16 PCM); row_len[B] (host) valid samples per row
 *   seg_rows[n], seg_bounds[n][2] (host): segment k = samples [start, end) of row seg_rows[k]; rows non-decreasing; bounds
 *               are clamped to the row length like Python slices; drop != 0 gathers what lies BETWEEN the segments
 *               (wav[cur:start], cur = end, ..., wav[cur:]) exactly like drop_chunks
 *   d_out       out_cap elements or NULL (sizing pass); out_offsets[B+1] (host) = per-row prefix sums of the output */
int svad_collect_chunks_device(svad_engine* e, const void* d_wav, int elem_bytes, int64_t B, int64_t ld, const int64_t* row_len,
                               const int64_t* seg_rows, const int64_t* seg_bounds, int64_t n_seg, int drop, void* d_out,
                               int64_t out_cap, int64_t* out_offsets, void* stream);

/* ---- decoder fine-tuning --------------------------------------------------------------------------------------------------------
 * The encoder is frozen; the decoder (LSTMCell(128 -> 128) + Dropout -> ReLU -> Conv1d(128 -> 1) -> Sigmoid) is trained on the
 * encoder's outputs.  All pointers are device memory of the engine's device unless noted; work is enqueued on `stream`.
 *
 * Encoder features: d_audio f32 [B][ld], L valid samples per row, L a multiple of the chunk size n (512 @16 kHz, 256 @8 kHz);
 * d_ctx_in [B][n/8] (or NULL = zeros) are the samples that precede each row; d_feat f32 [B][L/n][128] receives the post-ReLU
 * encoder output (the LSTM input) of every chunk.  Always the fp32 tile kernel, whatever svad_engine_set_kernel selected. */
int svad_features_device(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const float* d_audio, const float* d_ctx_in,
                         float* d_feat, void* stream);
/* Decoder scans over B streams x T steps from zero state.  Parameters in torch layout: W_ih, W_hh [512][128], b_ih, b_hh [512],
 * w_head [128], b_head [1]; gate order i, f, g, o.  d_drop [B][T][128] (or NULL) multiplies h on the head path only.
 * svad_decoder_tape_floats: floats of the tape the forward pass saves for the backward pass (activated gates and c);
 * svad_decoder_workspace_bytes: scratch of the forward (backward = 0) or backward (backward = 1) pass.  Both return SVAD_EINVAL
 * for negative sizes. */
int64_t svad_decoder_tape_floats(int B, int64_t T);
int64_t svad_decoder_workspace_bytes(int B, int64_t T, int backward);
/* d_feat [B][T][128] -> d_probs [B][T]; d_tape (or NULL when no backward pass follows) receives svad_decoder_tape_floats floats. */
int svad_decoder_forward_device(svad_engine* e, int B, int64_t T, const float* d_feat, const float* d_w_ih, const float* d_w_hh,
                                const float* d_b_ih, const float* d_b_hh, const float* d_w_head, const float* d_b_head,
                                const float* d_drop, float* d_probs, float* d_tape, void* d_work, void* stream);
/* d_dprobs [B][T] = dloss / dprobs -> dW_ih, dW_hh [512][128], db [512] (the gradient of b_ih and of b_hh alike), dw_head [128],
 * db_head [1].  d_probs and d_tape are what the forward pass with the same parameters and d_drop produced.  Fixed-order
 * reductions: the result does not change from call to call. */
int svad_decoder_backward_device(svad_engine* e, int B, int64_t T, const float* d_feat, const float* d_w_hh, const float* d_w_head,
                                 const float* d_drop, const float* d_probs, const float* d_dprobs, const float* d_tape, void* d_work,
                                 float* d_dw_ih, float* d_dw_hh, float* d_db, float* d_dw_head, float* d_db_head, void* stream);
/* Threshold search: file f holds d_probs / d_targets [d_offsets[f], d_offsets[f+1]) (d_offsets int64 [files+1]); d_grid f64 [20]
 * are the candidate thresholds.  For each of the 190 pairs (enter index a, exit index e < a; a outer, e inner) the hysteresis
 * decision (p >= enter -> 1, else p <= exit -> 0, else hold; from 0) is compared with the target, in double precision;
 * d_counts int64 [files][190] receives the number of matching chunks.  Runs on the current device. */
int svad_threshold_grid_device(const float* d_probs, const float* d_targets, const int64_t* d_offsets, int64_t files,
                               const double* d_grid, int64_t* d_counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SILERO_VAD_B200_H */
