/* b200vad.h -- C ABI of the B200-native VAD inference hot path.
 *
 * The reference (arnavsshah/universal-voice-activity-detection) is pure Python and has no
 * FFI of its own: its "operator interface" for this path is the set of library calls listed
 * below.  Each entry point names the reference call site it replaces (paths relative to the
 * reference root).  Conventions for every function:
 *   - plain pointers and sizes only; device pointers unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); nothing synchronises
 *     and nothing allocates unless documented; the caller owns every buffer;
 *   - returns 0 on success, <0 on error (B200VAD_E*); b200vad_last_error() gives the message
 *     of the calling thread's last failure;
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef B200VAD_H
#define B200VAD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200VAD_OK 0
#define B200VAD_EINVAL (-1)
#define B200VAD_ECUDA (-2)
#define B200VAD_ENOMEM (-3)
#define B200VAD_ESTATE (-4)

#if defined(__GNUC__)
#define B200VAD_API __attribute__((visibility("default")))
#else
#define B200VAD_API
#endif

#define B200VAD_ABI_VERSION 1
#define B200VAD_HIDDEN 128      /* LSTM hidden size (PyanNet2.py:60-66 LSTM_DEFAULTS) */
#define B200VAD_NUM_MEL 80      /* FbankConfig.num_filters */
#define B200VAD_MAX_INPUT_DIM 768   /* widest LSTM input D (768-dim SSL features): b200vad_model_workspace_bytes sizes for it */

B200VAD_API int b200vad_abi_version(void);
B200VAD_API const char* b200vad_last_error(void);

/* Instrumentation used by bench.py: number of kernels this library has launched in this
 * process, and CUDA-event timing of the dominant kernel (the LSTM recurrence) on its own stream.
 * profile_collect synchronises on the recorded events, sums their durations and resets. */
B200VAD_API long long b200vad_launch_count(void);
B200VAD_API void b200vad_profile_enable(int on);
B200VAD_API int b200vad_profile_collect(int kind /* 0 = LSTM recurrence, 1 = input-projection GEMM, 2 = head / warp-MMA GEMMs, 3 = fbank */, double* total_ms, int* launches);
/* 2 = tcgen05 kernels (default); 1 = the warp-MMA kernels kept for cross-validation of the tcgen05 path */
B200VAD_API int b200vad_set_impl(int impl);
/* fp16 tensor-core products per k-step of the input projections of LSTM layers >= 1: 2 (default: the layer outputs
 * travel as planes y1 = fp16((1 - 2^-6) y), y2 = fp16(y - y1) and xg = y1.W_hi + y2.W' with W' = fp16(W_hi + 2^6 W_lo),
 * one accumulator) or 3 (hi / lo planes and the plain split product x_lo.W_hi + x_hi.W_lo + x_hi.W_hi; validation).
 * Layer 0 and the head always use 3. */
B200VAD_API int b200vad_set_projection_terms(int terms);
/* Kernel of the input projections with K <= 256: 2 (default) = CTA pairs (tcgen05.mma.cta_group::2: two feature blocks
 * share an activation tile, each CTA loading half of it), both weight planes in tensor memory, 2 or 3 products per
 * k-step (see above); 1 = the same on single CTAs with an 8-warp epilogue; 0 = the general K-split kernel (always 3
 * products; validation, and the path of inputs wider than 256).  In LSTM modes 1 and 2 (b200vad_set_lstm_fused) the fused
 * layer kernels compute every projection with K <= 256 themselves, so there this choice reaches no kernel: layers >= 1
 * use 2 or 3 products as b200vad_set_projection_terms says, whichever kernel is set. */
B200VAD_API int b200vad_set_projection_kernel(int which);
/* 1 (default): the head (two Linear + LeakyReLU, classifier, sigmoid -- PyanNet2.py:183-187) runs as one kernel whose hidden
 * activations stay in shared memory; 0: two GEMM launches with the hidden activations as fp16 planes in HBM (validation;
 * bit-identical probabilities). */
B200VAD_API int b200vad_set_head_fused(int on);
/* Sequences per CTA of the tcgen05 recurrence: 0 = automatic (16 while the batch fits one wave of CTAs -- low latency
 * for small batches / streaming --, else 64), or 16 / 64 to force one (validation, tuning). */
B200VAD_API int b200vad_set_lstm_tile(int sequences_per_cta);
/* LSTM layers with input width <= 256 (PyanNet2.py:95,170): 1 = one fused kernel per layer on 4-CTA clusters
 * (input projection + recurrence, W_ih and W_hh as two fp16 planes each in tensor memory, no intermediate in HBM);
 * 2 = the same layer with every product issued as tcgen05.mma.cta_group::2 by CTA pairs (each CTA holds half of every
 * operand tile: half the x and h traffic per SM; bit-identical to 1);
 * 0 = the round-1 path (projection GEMM -> xg in HBM -> recurrence with a single-plane W_hh), kept for cross-validation
 * and for wider inputs (768-dim SSL features on layer 0).  The environment variable B200VAD_LSTM_MODE sets the initial mode. */
B200VAD_API int b200vad_set_lstm_fused(int on);
/* tuning bits of mode 2 (default 3): 1 = the input-product issuers yield to a recurrent product that is ready to issue,
 * 2 = two sets of h operand tiles (no "tile free" hand-shake on the per-step chain).  Results do not depend on bits 1 and 2.
 * Bits 4, 8, 32 are timing probes of tools/lstm_modes_timing.py (one k-step of the input product, no recurrent MMAs, no x
 * loads: RESULTS ARE WRONG while set); 64 fills the wait-site table read by b200vad_lstm_fused_read_debug (tools/pair_waits.py). */
B200VAD_API int b200vad_set_lstm_pair_opt(int opt);
/* clusters of 4 CTAs of the fused LSTM kernel that are co-resident on the current device (cudaOccupancyMaxActiveClusters) */
B200VAD_API int b200vad_lstm_fused_clusters(void);
/* timing probes of the fused kernel for tools/fused_ablate.py (RESULTS ARE WRONG while flags != 0): 1 no h exchange, 2 no
 * layer-output store, 4 no cell arithmetic, 8 no recurrent MMAs, 16 no input-projection MMAs; lag >= 0 sets how many part
 * slots the input MMAs of a part trail its recurrent MMAs (default 3).  flags = 0 restores the product path. */
B200VAD_API int b200vad_set_lstm_fused_debug(int flags, int lag);
/* with flag 32 set, the last fused launch leaves per (CTA, warp, wait site) cycle totals / counts of its waits in a device
 * table; this copies the first n int64 values to host (synchronises).  Mode 1: [cta 148][warp 25][site 8][cycles, waits,
 * mbarrier polls], site 0 = [kernel cycles, steps run, -]; mode 2: the CTA-pair kernel's table (tools/pair_waits.py) */
B200VAD_API int b200vad_lstm_fused_read_debug(long long* host, int n);
/* the fused kernel's waits are bounded (a protocol bug traps instead of hanging the GPU); the first wait that timed out leaves
 * {1, block, thread, wait site, barrier address, parity, grid size} in page-locked host memory, readable after the fault */
B200VAD_API int b200vad_lstm_fused_last_timeout(int* out7);
/* Split-precision linear layer on the tcgen05 GEMM: c[M,N] = a[M,K] . w[N,K]^T + bias, fp32 in / out, operands
 * split into fp16 (hi, lo) planes in `ws` (K % 8 == 0, N % 128 == 0; weights must fit in shared memory). */
B200VAD_API int b200vad_linear_split_f32(const float* a, int64_t M, int K, const float* w, int N, const float* bias, int use_w_lo,
                             float* c, void* ws, size_t ws_bytes, void* stream);

/* Page-locked host memory for the host-facing session calls (b200vad_session_submit_host ...); the reference's DataLoaders
 * (src/datasets/data_module.py:171-206) hand Lightning pageable batches.  write_combined != 0 asks for write-combined pages: the producer writes them
 * (streaming stores), only the GPU's DMA reads them -- no CPU-cache snooping on the H2D path.  Returns NULL on failure. */
B200VAD_API void* b200vad_host_alloc(size_t bytes, int write_combined);
B200VAD_API void b200vad_host_free(void* p);

/* Build the per-device constant tables (povey window, FFT twiddles, Kaldi mel triangles).
 * Allocates a few KB of device memory once per device.  Must precede any fbank call. */
B200VAD_API int b200vad_init(int device);

/* ---- a1: lhotse Fbank(FbankConfig(sampling_rate=16000)).extract / extract_batch
 * (src/utils/helper.py:120-130, src/datasets/ami/utils.py:152-163 and siblings).
 * T = (N + 80) / 160 frames per row. */
B200VAD_API int64_t b200vad_fbank_num_frames(int64_t num_samples);
/* wav: (B, N) f32 rows `wav_stride` elements apart; lens: optional (B) i32 valid samples per
 * row (NULL = N); feats: (B, T, 80) f32, rows shorter than T are padded with lhotse's
 * LOG_EPSILON; row_sum_ws: (B) f64 scratch. */
B200VAD_API int b200vad_fbank_f32(const float* wav, const int32_t* lens, int B, int64_t N, int64_t wav_stride,
                      float* feats, int64_t T, double* row_sum_ws, void* stream);
/* the same from 16-bit PCM: samples are converted as an audio loader does (int16 / 32768 -> float32, exact), so the
 * features are identical to b200vad_fbank_f32 on the converted waveform; halves the waveform bytes */
B200VAD_API int b200vad_fbank_i16(const int16_t* wav, const int32_t* lens, int B, int64_t N, int64_t wav_stride,
                      float* feats, int64_t T, double* row_sum_ws, void* stream);

/* ---- a2: PyanNet2.forward (src/models/segmentation/PyanNet2.py:154-187): nn.LSTM stack
 * (4 x BiLSTM(128) by default) + Linear/LeakyReLU x2 + Linear(1) + Sigmoid.
 * Weights are packed once into an opaque device blob in kernel layout.  Input widths 1 <= D <= B200VAD_MAX_INPUT_DIM:
 * packed_bytes returns 0 for any other D, and the pack and forward calls refuse it with B200VAD_EINVAL. */
B200VAD_API size_t b200vad_model_packed_bytes(int D, int num_layers);
/* one call per (layer, direction); w_ih (512, D_l), w_hh (512, 128), b_ih/b_hh (512): f32 device */
B200VAD_API int b200vad_model_pack_lstm(void* packed, int D, int num_layers, int layer, int direction, const float* w_ih,
                            const float* w_hh, const float* b_ih, const float* b_hh, void* stream);
/* linear.0 (128,256)+(128), linear.1 (128,128)+(128), classifier (1,128)+(1): f32 device */
B200VAD_API int b200vad_model_pack_head(void* packed, int D, int num_layers, const float* w1, const float* b1, const float* w2,
                            const float* b2, const float* wc, const float* bc, void* stream);
B200VAD_API size_t b200vad_model_workspace_bytes(int B, int64_t T);
/* x: (B, T, D) f32 -> prob: (B, T) f32 in (0,1).  The batch is processed in chunks that fit
 * `ws_bytes` (>= b200vad_model_workspace_bytes(1, T)). */
B200VAD_API int b200vad_model_forward_f32(const void* packed, int D, int num_layers, const float* x, int B, int64_t T, float* prob,
                              void* workspace, size_t ws_bytes, void* stream);

/* ---- a3/a4: PyanNet.forward / SincNet.forward (src/models/segmentation/PyanNet.py:164-197,
 * src/models/blocks/sincnet.py:73-103).  a5: get_num_frames (src/utils/receptive_field.py:165-193). */
B200VAD_API int64_t b200vad_sincnet_num_frames(int64_t num_samples);
B200VAD_API size_t b200vad_sincnet_packed_bytes(void);
/* wav_norm (1)+(1); low_hz_, band_hz_ (40); window_ (125); n_ (125); conv1 (60,80,5)+(60);
 * conv2 (60,60,5)+(60); norm{0,1,2} weight/bias (80),(60),(60): f32 device */
B200VAD_API int b200vad_sincnet_pack(void* packed, const float* wav_norm_w, const float* wav_norm_b, const float* low_hz,
                         const float* band_hz, const float* window, const float* n, const float* conv1_w,
                         const float* conv1_b, const float* conv2_w, const float* conv2_b, const float* norm0_w,
                         const float* norm0_b, const float* norm1_w, const float* norm1_b, const float* norm2_w,
                         const float* norm2_b, void* stream);
B200VAD_API size_t b200vad_sincnet_workspace_bytes(int B, int64_t N);
/* wav: (B, N) f32 -> out: (B, Ts, 60) f32 (time-major, i.e. already "b t f" of PyanNet.py:178) */
B200VAD_API int b200vad_sincnet_forward_f32(const void* packed, const float* wav, int B, int64_t N, int64_t wav_stride, float* out,
                                void* workspace, size_t ws_bytes, void* stream);

/* ---- a6/a7: median_filter (src/utils/helper.py:66-97) as called by VadModel.predict_step
 * (src/engines/vad_engine.py:204-211): out[b,t] = median over a zero-padded window of `kernel`
 * frames of (prob < thr ? 0 : 1).  elem_bytes = 1 (uint8) or 8 (int64, the reference's dtype).
 * near_count (optional, i32, must be zeroed by the caller): number of frames with
 * |prob - thr| <= near_tol, the "near-threshold" set parity reports separately. */
B200VAD_API int b200vad_median_window(double speech_window, double window);
B200VAD_API int b200vad_threshold_median(const float* prob, int B, int64_t T, float thr, int kernel, void* out, int elem_bytes,
                             int32_t* near_count, float near_tol, void* stream);

/* ---- a8/a9: run-length segment extraction (src/scripts/predict.py:447-458, 472-490).
 * dec: flat uint8 decisions; stream r = dec[offsets[r], offsets[r+1]) (offsets: (R+1) i64,
 * NULL = R rows of T frames).  Emits (r, first_frame, last_frame_inclusive) i32 triples for
 * every run of >= min_run frames (2 = the reference's `end - start > 0`), ordered by (r, first).
 * counts: (R) i32 out; seg_off: (R+1) i64 out (seg_off[R] = total); seg: (cap, 3) i32. */
B200VAD_API int b200vad_segments(const uint8_t* dec, const int64_t* offsets, int R, int64_t T, int min_run, int32_t* counts,
                     int64_t* seg_off, int32_t* seg, int64_t cap, void* stream);

/* ---- 8f-1 scoring.  VadModel.test_step stat scores (src/engines/vad_engine.py:167-202): out4 (device, i64) =
 * tp, fp, tn, fn of dec (u8, != 0 is speech) against labels (u8) over n frames. */
B200VAD_API int b200vad_stat_scores(const uint8_t* dec, const uint8_t* labels, int64_t n, int64_t* out4, void* stream);
/* get_binary_tensor / get_false_alarm / get_missed_detection (src/scripts/predict.py:654-673) on bit masks.
 * Intervals are (recording, start_frame, end_frame_exclusive) i32 triples, already int(t / frame_shift) as the
 * reference computes them; recording r has nframes[r] = ceil(duration / frame_shift) frames and its mask starts at
 * word word_off[r] (word_off: (R+1) i64, 32 frames per word, total_words = word_off[R]).  fa / md: (R) i64 frame
 * counts (pred & ~gt, gt & ~pred); the caller divides by nframes like the reference.  All pointers device. */
B200VAD_API size_t b200vad_score_workspace_bytes(int64_t total_words);
B200VAD_API int b200vad_score_intervals(const int32_t* gt_iv, int64_t n_gt, const int32_t* pred_iv, int64_t n_pred,
                            const int64_t* word_off, const int32_t* nframes, int R, int64_t total_words, int max_words_per_rec,
                            void* workspace, int64_t* fa, int64_t* md, void* stream);

/* ---- synthetic corpus (BASELINE config 4: 1000 h sharded across GPUs; there is no network for real corpora).
 * wav (rows, N) f32 device <- utterances first_utt .. first_utt + rows - 1 of the corpus `seed`: 0.5 s segments of
 * background noise or noise + a voiced burst, a pure function of (seed, utterance id, sample index), so any sharding
 * or batching of the corpus sees identical audio. */
B200VAD_API int b200vad_synth_corpus(float* wav, int64_t first_utt, int rows, int64_t N, uint64_t seed, void* stream);

/* ---- long-form audio with OVERLAPPING windows (BASELINE config 3; the reference itself only cuts hop = window,
 * src/datasets/ami/utils.py:107, which needs no stitching): prob (num_windows, frames_per_window) f32, window w
 * starting at global frame w * hop_frames -> out (L) f32, every frame taken from the window whose centre is nearest. */
B200VAD_API int b200vad_stitch_center(const float* prob, int num_windows, int frames_per_window, int hop_frames, float* out, int64_t L,
                          void* stream);

/* ---- whole path on device buffers: fbank -> PyanNet2 -> threshold/median -> segments */
B200VAD_API size_t b200vad_pipeline_workspace_bytes(int B, int64_t N);
B200VAD_API int b200vad_pipeline_fbank_f32(const void* packed, int num_layers, const float* wav, const int32_t* lens, int B,
                               int64_t N, int64_t wav_stride, float thr, int kernel, float* prob /* (B,T) */,
                               uint8_t* dec /* (B,T) */, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap,
                               void* workspace, size_t ws_bytes, void* stream);

B200VAD_API int b200vad_pipeline_fbank_i16(const void* packed, int num_layers, const int16_t* wav, const int32_t* lens, int B,
                               int64_t N, int64_t wav_stride, float thr, int kernel, float* prob, uint8_t* dec, int32_t* counts,
                               int64_t* seg_off, int32_t* seg, int64_t cap, void* workspace, size_t ws_bytes, void* stream);

/* ---- whole path of the reference's SincNet flow (feature_extractor="sincnet", config/config.py) on device buffers:
 * SincNet -> PyanNet's LSTM stack + head (src/models/segmentation/PyanNet.py:164-197) -> threshold / median filter
 * (src/engines/vad_engine.py:204-211: kernel 49 = window 0.01 since encoding_dim != 768) -> run-length segments that keep
 * single-frame runs (src/scripts/predict_sincnet.py:348-370, min_run = 1).  The front end hands the LSTM its layer-0 operand
 * as fp16 planes directly (no fp32 (B, Ts, 60) round trip): prob / dec equal b200vad_sincnet_forward_f32 followed by
 * b200vad_model_forward_f32 and b200vad_threshold_median bit for bit.
 * packed_model: b200vad_model_pack_* blob with D = 60; packed_sincnet: b200vad_sincnet_pack blob.  Ts =
 * b200vad_sincnet_num_frames(N) frames per row; N >= 991 (one SincNet frame).  There is no lens argument: the reference pads
 * SincNet windows with zero audio, which its InstanceNorm sees.  cap: B * ceil(Ts / 2) holds every possible segment. */
B200VAD_API size_t b200vad_pipeline_sincnet_workspace_bytes(int B, int64_t N);
B200VAD_API int b200vad_pipeline_sincnet_f32(const void* packed_model, const void* packed_sincnet, int num_layers, const float* wav,
                                 int B, int64_t N, int64_t wav_stride, float thr, int kernel, float* prob /* (B,Ts) */,
                                 uint8_t* dec /* (B,Ts) */, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap,
                                 void* workspace, size_t ws_bytes, void* stream);
/* 16-bit PCM rows (int16 / 32768, exact): identical results to the f32 form on the converted waveform, half the bytes */
B200VAD_API int b200vad_pipeline_sincnet_i16(const void* packed_model, const void* packed_sincnet, int num_layers, const int16_t* wav,
                                 int B, int64_t N, int64_t wav_stride, float thr, int kernel, float* prob, uint8_t* dec,
                                 int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, void* workspace, size_t ws_bytes,
                                 void* stream);

/* ---- host-buffer session: the same path with HOST waveforms and HOST results -- what a caller holding
 * lhotse/DataLoader batches in host memory uses (src/engines/vad_engine.py:204-211 fed by
 * src/datasets/data_module.py:194-206).  The session owns device buffers for two batches in flight and three
 * CUDA streams (H2D / compute / D2H).
 *   run_host     : blocking; B rows are cut into chunks of max_chunk_rows that are pipelined internally.
 *   submit / wait: asynchronous; submit(slot) enqueues H2D + whole path + D2H of one batch (<= max_chunk_rows
 *                  rows) and returns; wait(slot) blocks until that batch's dec/prob are in the host buffers
 *                  given to submit and copies its segment triples.  Keeping both slots busy overlaps the PCIe
 *                  copies of batch i+1 / i-1 with the compute of batch i.  This is what `e2e` times in bench.py.
 * Host buffers should be pinned (cudaHostAlloc / torch pin_memory) for the copies to be asynchronous. */
typedef struct b200vad_session b200vad_session;
B200VAD_API int b200vad_session_create(int device, const void* packed_device, int num_layers, int max_chunk_rows, int64_t N,
                           b200vad_session** out);
/* the same session on the SincNet path (b200vad_pipeline_sincnet_*; the reference feeds it from
 * src/scripts/predict_sincnet.py's DataLoader): T = b200vad_sincnet_num_frames(N), up to ceil(T / 2) segments per row.
 * It is driven by the calls below, unchanged. */
B200VAD_API int b200vad_session_create_sincnet(int device, const void* packed_model, const void* packed_sincnet, int num_layers,
                                   int max_chunk_rows, int64_t N, b200vad_session** out);
/* wav_host: (B, N) f32; outputs on host: dec (B,T) u8 (optional), prob (B,T) f32 (optional),
 * seg (cap,3) i32, *nseg total segments.  Blocks until results are on the host. */
B200VAD_API int b200vad_session_run_host(b200vad_session* s, const float* wav_host, int B, float thr, int kernel, uint8_t* dec_host,
                             float* prob_host, int32_t* seg_host, int64_t cap, int64_t* nseg);
B200VAD_API int b200vad_session_submit_host(b200vad_session* s, int slot, const float* wav_host, int B, float thr, int kernel,
                                uint8_t* dec_host, float* prob_host);
/* 16-bit PCM host waveforms (B, N) i16: half the PCIe bytes of the fp32 form, identical results */
B200VAD_API int b200vad_session_submit_host_i16(b200vad_session* s, int slot, const int16_t* wav_host, int B, float thr, int kernel,
                                    uint8_t* dec_host, float* prob_host);
B200VAD_API int b200vad_session_wait(b200vad_session* s, int slot, int32_t* seg_host, int64_t cap, int64_t* nseg);
/* Device timeline of the slot's most recent batch, in ms since the session was created:
 * ms[0..4] = H2D begin, H2D end, compute begin, compute end, D2H end (CUDA events on the three streams). */
B200VAD_API int b200vad_session_slot_times(b200vad_session* s, int slot, float* ms);
B200VAD_API void b200vad_session_destroy(b200vad_session* s);

/* ---- streaming session (BASELINE config 5): num_streams ring buffers of the last window_samples samples.
 * push() appends hop_samples new samples per stream (chunk: (num_streams, hop_samples) f32, host or device),
 * runs fbank -> PyanNet2 -> threshold/median on every buffered window (one CUDA graph replay when use_graph),
 * and returns the newest hop_samples/160 frames of every stream on the host: prob_new (S, nf) f32, dec_new (S, nf)
 * u8.  These equal the batch path applied to the same window (there is no reference streaming mode: the BiLSTM is
 * non-causal).  device_ms (optional) = CUDA-event time of the push.  Blocking. */
typedef struct b200vad_stream b200vad_stream;
B200VAD_API int b200vad_stream_create(int device, const void* packed_device, int num_layers, int num_streams, int64_t window_samples,
                          int hop_samples, int use_graph, b200vad_stream** out);
/* the same on the SincNet path: SincNet -> PyanNet -> threshold / median on every buffered window (the graph covers the
 * front end too).  hop_samples must be a multiple of 270 (the SincNet frame step), window_samples >= 991; a push returns
 * the newest hop_samples / 270 frames, the last ones of the b200vad_sincnet_num_frames(window_samples) frames of the window. */
B200VAD_API int b200vad_stream_create_sincnet(int device, const void* packed_model, const void* packed_sincnet, int num_layers,
                                  int num_streams, int64_t window_samples, int hop_samples, int use_graph, b200vad_stream** out);
B200VAD_API int b200vad_stream_push(b200vad_stream* s, const float* chunk, int chunk_on_host, float thr, int kernel, float* prob_new_host,
                        uint8_t* dec_new_host, float* device_ms);
/* parity / debugging: current windows (S, window) f32 and all frame outputs (S, T) of the last push, to host buffers */
B200VAD_API int b200vad_stream_snapshot(b200vad_stream* s, float* window_host, float* prob_host, uint8_t* dec_host);
B200VAD_API void b200vad_stream_destroy(b200vad_stream* s);

#ifdef __cplusplus
}
#endif
#endif /* B200VAD_H */
