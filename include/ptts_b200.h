/* ptts_b200.h — C ABI of the B200-native Pocket-TTS generation engine (libptts_b200.so).
 *
 * This is the drop-in boundary for the reference's per-frame hot path. Every entry point below states the
 * reference interface it replaces (paths are into Codes4Fun/pocket-tts.cpp). Plain pointers and sizes only;
 * all pointers are HOST pointers unless a name says otherwise. Functions return 0 on success, a negative
 * B200_E* code on a recoverable error; unrecoverable CUDA faults abort() with a message, mirroring the
 * reference's exit(1)/assert error behaviour (src/pocket_tts.cpp:110-113,295-298).
 *
 * Two layers live in the library:
 *   b200_*        device layer: weights, per-utterance slots, batched prefill/step          (this file)
 *   ptts_*        the reference's own C++ streaming API, same signatures (include/pocket_tts/pocket_tts.h)
 *   ptts_c_*      extern "C" aliases of ptts_* for FFI users (ctypes / cgo / JNI)           (this file)
 */
#ifndef PTTS_B200_H
#define PTTS_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_API __attribute__((visibility("default")))

enum { B200_OK = 0, B200_EINVAL = -1, B200_ENOMEM = -2, B200_ESTATE = -3, B200_ENOTFOUND = -4, B200_ECAPACITY = -5 };
enum { B200_DT_F32 = 0, B200_DT_BF16 = 1, B200_DT_F16 = 2 };

typedef struct b200_engine b200_engine;

typedef struct b200_config {
    int device;           /* CUDA ordinal */
    int max_slots;        /* utterances in flight (reference: batch hard-wired to 1, models/mimi.h:55,62)          */
    int max_voices;       /* voice-conditioned prefixes resident at once                                            */
    int kv_capacity;      /* FlowLM positions per slot (reference: 1000, src/pocket_tts.cpp:367-368)                */
    int kv_f32;           /* 1 = fp32 FlowLM KV cache like the reference (modules/transformer.h:21-33), 0 = bf16    */
    int mimi_mask_mode;   /* 0 = the reference's mask incl. its offset>250 quirk (src/torch.h:168-221), 1 = causal  */
    int convt_split;      /* 1 = transposed convs see hi+lo f16 activations (~fp32; reference conv.h:282 is f32); 0 (default) = f16
                             activations like every other conv: Mimi-only SNR 63.8 vs 65.9 dB, full-pipeline SNR unchanged (46.5 dB) */
    int gemm_path;        /* 0 = auto (tcgen05 for large row counts), 1 = CUDA-core only (validation path)          */
    int max_prefill_rows; /* rows per prefill chunk (0 = default 4096; 256 paragraphs start in 9.7 / 8.1 / 7.3 ms at 2048 / 4096 / 16384) */
    int cuda_graphs;      /* 1 = replay the per-frame step as a CUDA graph (captured on second use of a shape)       */
    int pdl;              /* programmatic dependent launch (a kernel's prologue overlaps its predecessor's tail): 0 = off, 1 = for up to
                             128 utterances per step (default), 2 = always                                                      */
    int overlap;          /* 1 = two-stream pipeline: the Mimi decode of frame t overlaps the FlowLM step of frame t+1   */
    int prefix_share;     /* 1 (default) = every utterance of a voice attends to ONE resident copy of the voice-conditioned KV prefix
                             (cascade attention: prefix x all rows of the voice on tensor cores, private suffix streamed per row);
                             0 = the reference's copy_states semantics (models/flow_lm.h:70-78): each sentence start copies the
                             prefix into the slot's own cache. Results agree to rounding; tests run both. */
} b200_config;

B200_API void b200_default_config(b200_config* cfg);

/* Replaces ptts_init's allocation half (src/pocket_tts.cpp:273-287). */
B200_API int  b200_engine_create(const b200_config* cfg, b200_engine** out);
B200_API void b200_engine_destroy(b200_engine* e);

/* Replaces WeightLoader::fetch/load (src/loader.h:191-226,274-311): hand over one checkpoint tensor, by its
 * FILE key (reference name minus its first component, src/loader.h:101-105), in its file dtype and torch-order
 * shape. The engine applies the reference's per-consumer dtype policy itself (linears bf16, convs f16, ...). */
B200_API int  b200_upload_tensor(b200_engine* e, const char* key, const void* data, int dtype, const int64_t* shape, int ndim);
/* Replaces weights->load() (src/pocket_tts.cpp:306): repack + upload; precomputes the constant timestep
 * embedding (s=0,t=1; models/flow_lm.h:137-138, modules/mlp.h:92-106). */
B200_API int  b200_finalize_weights(b200_engine* e);

/* Replaces get_state_for_audio_prompt (src/pocket_tts.cpp:100-124): prefill of audio_prompt[T][1024] (f32)
 * into a resident voice prefix. Returns the voice id (>=0) or an error. */
B200_API int  b200_voice_create(b200_engine* e, const float* audio_prompt, int T);
/* Voice cloning (DESIGN.md 4.6; the reference port has no encoder). The checkpoint's encoder set (mimi.encoder.*, mimi.encoder_transformer.*,
 * mimi.downsample.*, flow_lm.speaker_proj_weight) is uploaded by b200_finalize_weights when present; b200_has_encoder tells (1 / 0).
 * pcm: n >= 1 mono float samples at sample_rate Hz, any integer in [8000, 192000]. Other rates than 24000 are resampled to 24 kHz on the
 * device (torchaudio.functional.resample with its defaults, DESIGN.md 4.6) into n24 = ceil(24000 n / sample_rate) samples; 24 kHz input
 * is used as is (n24 = n). The signal is right-padded with zeros to a multiple of 1920; T = ceil(n24 / 1920) prompt rows.
 * b200_voice_embed_audio_rate encodes on the engine stream and returns T; with out != NULL ([T][1024]) it copies the audio_prompt rows
 * out (synchronises). b200_voice_create_from_audio_rate encodes and prefills a new voice without a host round trip or wait; returns the
 * voice id. b200_voice_embed_audio / b200_voice_create_from_audio are these with sample_rate = 24000.
 * Errors: B200_ENOTFOUND no encoder weights, B200_EINVAL n < 1, a NULL pointer or a sample rate outside [8000, 192000], B200_ECAPACITY
 * T > kv_capacity or max_voices reached. */
B200_API int  b200_has_encoder(b200_engine* e);
B200_API int  b200_voice_embed_audio(b200_engine* e, const float* pcm, long long n, float* out);
B200_API int  b200_voice_create_from_audio(b200_engine* e, const float* pcm, long long n);
B200_API int  b200_voice_embed_audio_rate(b200_engine* e, const float* pcm, long long n, int sample_rate, float* out);
B200_API int  b200_voice_create_from_audio_rate(b200_engine* e, const float* pcm, long long n, int sample_rate);

/* Replaces _stream_sentence_init (src/pocket_tts.cpp:416-444): restore the voice-conditioned KV prefix
 * (copy_states, models/flow_lm.h:70-78), reset the Mimi states (models/mimi.h:71-75), prefill the text tokens,
 * arm the stop rule. tokens are SentencePiece ids (conditioners/text.h:21-27). */
B200_API int  b200_begin_sentence(b200_engine* e, int slot, int voice, const int32_t* tokens, int n_tokens,
                                  int max_gen_len, int frames_after_eos, float temp);
/* Same for many slots at once (one ragged prefill): slots[i] gets tokens[tok_off[i] .. tok_off[i+1]). */
B200_API int  b200_begin_sentences(b200_engine* e, int n, const int32_t* slots, const int32_t* voices,
                                   const int32_t* tokens, const int32_t* tok_off, const int32_t* max_gen_len,
                                   const int32_t* frames_after_eos, const float* temp);
/* Same, plus rng_stream[n]: the id that keys the device noise generator for each sentence (default = the slot). A scheduler passes the
 * sentence's global index so that its audio does not depend on the slot or GPU it lands on. Nothing in this call waits on the host:
 * uploads are staged through a pinned ring, the prefill is enqueued behind the steps already submitted (reference
 * _stream_sentence_init is synchronous, src/pocket_tts.cpp:416-444). max_gen_len is clamped to the remaining KV capacity. */
B200_API int  b200_begin_sentences_ex(b200_engine* e, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens,
                                      const int32_t* tok_off, const int32_t* max_gen_len, const int32_t* frames_after_eos,
                                      const float* temp, const uint32_t* rng_stream);
/* Per-sentence sampling controls (DESIGN.md 4.7), the knobs upstream Pocket TTS exposes per request:
 *   lsd_steps      LSD decode steps N, 1..8: x_{i+1} = x_i + v(c, i/N, (i+1)/N, x_i) / N from x_0 = noise (1 = the single-step head)
 *   noise_clamp    a >= 0: noise drawn from N(0, temp) truncated to [-a, a] (absolute bounds, torch trunc_normal_); 0 = untruncated.
 *                  Injected noise (b200_step's `noise`) is used as given.
 *   eos_threshold  EOS fires when the EOS logit > eos_threshold (the reported eos_logit stays logit + 4); finite
 * b200_default_sampling fills {1, 0, -4}: a sentence with these values runs exactly the step it runs without sampling controls. */
#define B200_LSD_MAX_STEPS 8
typedef struct b200_sampling { int lsd_steps; float noise_clamp; float eos_threshold; } b200_sampling;
B200_API void b200_default_sampling(b200_sampling* s);
/* B200_OK, or B200_EINVAL for NULL, lsd_steps outside 1..8, a negative or non-finite clamp, or a non-finite threshold. */
B200_API int  b200_sampling_check(const b200_sampling* s);
/* b200_begin_sentences_ex plus sampling[n] (NULL = defaults for every sentence). B200_EINVAL when any entry fails b200_sampling_check. */
B200_API int  b200_begin_sentences_sampling(b200_engine* e, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens,
                                            const int32_t* tok_off, const int32_t* max_gen_len, const int32_t* frames_after_eos,
                                            const float* temp, const uint32_t* rng_stream, const b200_sampling* sampling);
/* Stream-ordered: the sentences in `slots` end now. From the next enqueued step on these slots are dead rows (no KV append, no attention,
 * produced = 0) until a sentence start reuses them. Steps already enqueued are unaffected. Nothing in this call waits on the host. */
B200_API int  b200_end_sentences(b200_engine* e, int n, const int32_t* slots);
B200_API int  b200_voice_len(b200_engine* e, int voice);           /* prefix rows of a resident voice */
B200_API int  b200_kv_capacity(b200_engine* e);
B200_API int  b200_max_slots(b200_engine* e);

/* Replaces _stream_sentence_step (src/pocket_tts.cpp:446-492) for the dense slot range [slot0, slot0+n):
 * FlowLM step -> EOS/stop rule -> LSD head -> Mimi -> 1920 samples per slot.
 *   noise      [n][32] injected N(0,temp) draws, or NULL = device counter-based RNG (0 when temp == 0)
 *   pcm        [n][1920] raw float samples (only rows with produced[i] != 0 are meaningful)
 *   produced   [n]  1 = a frame was emitted (reference returns true), 0 = sentence finished / slot idle
 *   latents    [n][32] optional, eos_logit [n] optional (logit + 4, EOS when > 0)
 * Host<->device copies and one stream synchronise are inside the call. */
B200_API int  b200_step(b200_engine* e, int slot0, int n, const float* noise, float* pcm, int32_t* produced,
                        float* latents, float* eos_logit);
/* Device-resident variant: enqueue one step, no copies, no sync. Results stay in the engine's device buffers (b200_device_ptr).
 * With cfg.overlap the step is pipelined over two streams (its Mimi decode may be enqueued together with the NEXT step, see
 * DESIGN.md 4.1): call b200_join (stream-ordered) or b200_sync (host) before reading "pcm". */
B200_API int  b200_step_enqueue(b200_engine* e, int slot0, int n, int use_injected_noise);
/* `count` consecutive b200_step_enqueue(e, slot0, n, 0) calls made natively (a driver loop in an interpreted host language can starve the
 * stream: one step is ~1 ms of device time behind two graph launches). */
B200_API int  b200_steps_enqueue(b200_engine* e, int slot0, int n, int count);
/* Pipelined pair for throughput serving (up to three frames in flight): submit enqueues a frame and returns at once, collect blocks until the
   oldest submitted frame is complete and copies out its n x 1920 samples + produced flags; returns n (or a negative error).         */
B200_API int  b200_submit(b200_engine* e, int slot0, int n, const float* noise /* [n][32] or NULL */);
B200_API int  b200_collect(b200_engine* e, float* pcm, int32_t* produced);
B200_API int  b200_sync(b200_engine* e);
/* main stream waits for the Mimi stream: an event recorded on b200_stream() afterwards covers all enqueued frames incl. PCM */
B200_API int  b200_join(b200_engine* e);

/* Mimi-only path (BASELINE config 3): decode caller-provided latents [n][32] for slots [slot0, slot0+n). */
B200_API int  b200_mimi_reset(b200_engine* e, int slot0, int n);
B200_API int  b200_mimi_decode(b200_engine* e, int slot0, int n, const float* latents, float* pcm);
B200_API int  b200_mimi_decode_enqueue(b200_engine* e, int slot0, int n);

B200_API void b200_set_seed(b200_engine* e, uint64_t seed);
B200_API int  b200_slot_position(b200_engine* e, int slot);        /* FlowLM current_end of a slot (synchronises the stream and reads the device counter) */
/* Force every slot in the range to position `pos` with an active, never-ending sentence (bench: KV length control). */
B200_API int  b200_debug_set_position(b200_engine* e, int slot0, int n, int pos, int max_gen_len);
/* Unit-test hook for the GEMM family (tests/test_gpu_gemm.py): out[n_slots*T][N] = windows(A) . W^T (+bias); A is
 * [n_slots][rows_buf][C] f32 (rounded to bf16, or f16 when f16 != 0), window of output row (slot,t) = rows t..t+taps-1.
 * path 0 = dispatcher, 1 = CUDA-core. Returns 1 when the tcgen05 kernel ran, 0 for a CUDA-core kernel, <0 on error. */
B200_API int  b200_debug_gemm(b200_engine* e, int f16, const float* A, int n_slots, int rows_buf, int C, int T, int taps, const float* W, int N,
                              const float* bias, int path, float* out, float* out2_as_f32);
/* Parity helper (teacher forcing): overwrite the backbone input latent [n][32] of slots [slot0, slot0+n). */
B200_API int  b200_debug_set_latent(b200_engine* e, int slot0, int n, const float* latents);
/* Per-segment device timing with CUDA events on the engine stream (bench.py roofline leg). Categories: 0 FlowLM attention streaming
 * kernel, 1 FlowLM backbone, 2 flow head, 3 Mimi transformer, 4 SEANet, 5 whole step, 6 shared-prefix tile kernel. out_ms[7], out_count[7]. */
B200_API int  b200_profile(b200_engine* e, int on);
B200_API int  b200_profile_read(b200_engine* e, float* out_ms, int* out_count);
/* cudaProfilerStart (1) / cudaProfilerStop (0): lets `ncu --profile-from-start off` capture only a bracketed region. */
B200_API void b200_profiler_range(int start);
B200_API void* b200_stream(b200_engine* e);                        /* cudaStream_t the engine launches on */
B200_API void* b200_device_ptr(b200_engine* e, const char* name);  /* "pcm", "latent", "noise", "produced", "eos", "lat_f32", "noise_drawn" */
B200_API int  b200_debug_read_f32(b200_engine* e, const char* name, long long offset, float* out, int n); /* synchronises, copies an f32 buffer out */
B200_API long long b200_launch_count(b200_engine* e);              /* kernels launched so far by this engine */
B200_API int  b200_read_kv(b200_engine* e, int slot, int layer, int which, int n_pos, float* out); /* debug/parity */
/* Tap points for localising a parity failure (replaces GraphContext::debug, src/context.h:526-547; names follow the tests' CPU restatement):
 * "flow.layer<l>" / "flow.attn<l>" [1024] (need b200_debug_taps(e, 1): steps then run eagerly on one stream), "mimi.upsample" [16*512],
 * "mimi.transformer" [16*512], "seanet.conv0" [16*512], "seanet.convt2" [96*256], "seanet.res3" [96*256], "seanet.res6" [480*128],
 * "seanet.res9" [1920*64] of `slot` after its last step; "enc.input" [1920T] (the 24 kHz signal the encoder read), "enc.seanet" [16T*512], "enc.transformer" [16T*512], "enc.downsample" [T*512] of the
 * last clone (any valid slot). out == NULL returns the element count. */
B200_API int  b200_debug_taps(b200_engine* e, int on);
B200_API int  b200_debug_tap(b200_engine* e, const char* name, int slot, float* out, int max_elems);
/* Host-only: tile width (32/64/128) and deterministic split-K factor the GEMM dispatcher would use (cost model of gemm_tc.cuh). */
B200_API int  b200_debug_gemm_plan(int R, int N, int K, int num_sms, int want_ln, int* bn, int* splits);
/* Unit-test hooks for the FlowLM attention (tests/test_gpu_attention.py). b200_debug_write_kv writes physical cache rows [pos0, pos0+n)
 * of a slot from f32 rows [n][1024] (no prefix redirection; rounded to the cache type): the counterpart of b200_read_kv.
 * b200_debug_set_prefix makes keys [0, pfx_len) of `slot` the rows of `pfx_slot` (0 rows = private cache). */
B200_API int  b200_debug_write_kv(b200_engine* e, int slot, int layer, int which, int pos0, int n, const float* rows);
B200_API int  b200_debug_set_prefix(b200_engine* e, int slot, int pfx_slot, int pfx_len);
/* Per-call overrides of the attention switches; a negative field keeps the engine's value. */
typedef struct b200_attn_opts {
    int stream_splits;    /* KV splits of the streaming kernel, 1..16 (0 = automatic; PTTS_B200_AF_SPLITS)          */
    int tile_prec;        /* operand precision of the decode-side prefix tiles, 0..2 (PTTS_B200_TILE_PREC)           */
    int prefill_prec;     /* operand precision of the prefill tiles, 0..2 (PTTS_B200_PREFILL_PREC)                   */
    int fork_tiles;       /* 1 = prefix tiles on a forked stream + merge (PTTS_B200_FORK_TILES)                      */
    int counted_merge;    /* 1 = last-arriving CTA merges instead of attn_merge_kernel (PTTS_B200_COUNTED_MERGE)     */
    int tile_min_rows;    /* fewest decode rows that use the prefix tiles (PTTS_B200_TILE_MIN_ROWS)                  */
} b200_attn_opts;
/* Runs the attention dispatch of one FlowLM layer eagerly over q [n][1024] f32 and the keys in the cache; out [n][1024] = the bf16
 * output as f32 (NaN where nothing was written). prefill = 0: row r is slot slot0 + r at position rows_pos[r] (negative = dead row).
 * prefill = 1: rows (rows_slot[r], rows_pos[r]) slot-major with ascending positions, chunked by max_prefill_rows like a prefill.
 * Returns the number of tile work items (decode: 1 if the shared-prefix tiles ran, else 0), or a negative error. */
B200_API int  b200_debug_attention(b200_engine* e, int layer, int prefill, int slot0, int n, const int32_t* rows_slot, const int32_t* rows_pos,
                                   const float* q, const b200_attn_opts* opts, float* out);
/* Host-only: the attention work lists. prefill = 0: prefix tiles of decode rows [0, n) whose prefix is (pfx_slot[r], pfx_len[r]) on
 * num_sms SMs; aux_out[n] receives the tile row list; returns the prefix split count (0: no tiles) or B200_ECAPACITY beyond the work-list
 * capacity of n slots and max_voices prefixes. prefill = 1: tile items of rows (row_slot[r], row_pos[r]) in chunks of chunk_rows,
 * pfx_slot / pfx_len indexed by slot; aux_out[chunks + 1] receives the first item of each chunk; returns the chunk count.
 * items_out[cap][9] = {row0, nrows, a_slot, a_k0, a_k1, b_slot, b_k0, b_k1, out_split}; *n_items = the item count. */
B200_API int  b200_debug_attn_plan(int prefill, int n, const int32_t* row_slot, const int32_t* row_pos, const int32_t* pfx_slot, const int32_t* pfx_len,
                                   int num_sms, int chunk_rows, int max_voices, int32_t* items_out, int cap, int32_t* aux_out, int* n_items);
/* Unit-test hook for the voice-cloning encoder's window attention (tests/test_gpu_voice_clone.py): q, k, v [R][512] f32 (rounded to bf16;
 * q and k as the QKV epilogue leaves them, rotated), positions = row indices, key j visible to query i iff 0 <= i - j < 250, 8 heads of 64;
 * out [R][512] = the bf16 attention output as f32. Synchronises. */
B200_API int  b200_debug_window_attention(b200_engine* e, int R, const float* q, const float* k, const float* v, float* out);
B200_API const char* b200_build_info(void);

/* ---- extern "C" aliases of the reference's C++ API (include/pocket_tts/pocket_tts.h:18-42) ---- */
typedef struct ptts_context_t ptts_context_t;
typedef struct ptts_stream_t ptts_stream_t;
B200_API void ptts_c_set_seed(unsigned int seed);
B200_API unsigned int ptts_c_get_seed(void);
B200_API ptts_context_t* ptts_c_init(const char* model_path);
/* Same with an explicit engine configuration instead of the PTTS_B200_* environment variables. */
B200_API ptts_context_t* ptts_c_init_ex(const char* model_path, const b200_config* cfg);
B200_API int ptts_c_voice(ptts_stream_t* s);   /* engine voice id of a stream */
B200_API int ptts_c_slot(ptts_stream_t* s);    /* engine slot of a stream */
B200_API int ptts_c_get_sample_rate(ptts_context_t* ctx);
B200_API int ptts_c_get_frame_size(ptts_context_t* ctx);
B200_API ptts_stream_t* ptts_c_stream_from_safetensors(ptts_context_t* ctx, const char* voice, float temp);
B200_API void ptts_c_stream_reset(ptts_stream_t* s);
B200_API void ptts_c_stream_flush(ptts_stream_t* s);
B200_API void ptts_c_stream_send(ptts_stream_t* s, const char* chunk);
B200_API int ptts_c_stream_receive(ptts_stream_t* s, float* samples);
/* Sampling controls of the stream's sentences from the next sentence start on (B200_EINVAL: NULL or out of range, see b200_sampling_check). */
B200_API int ptts_c_stream_set_sampling(ptts_stream_t* s, const b200_sampling* sampling);
B200_API b200_engine* ptts_c_engine(ptts_context_t* ctx);
B200_API void ptts_c_destroy(ptts_context_t* ctx);   /* frees the engine and the context (the reference API never frees, src/pocket_tts.cpp:313) */
/* Text front end, exposed for bit-exactness tests (conditioners/text.h:21-27,81-94). */
B200_API int ptts_c_tokenize(ptts_context_t* ctx, const char* text, int32_t* ids, int max_ids);
B200_API int ptts_c_count_words(const char* text);
/* Pending sentences of a stream after send/flush (conditioners/text.h:207-251); returns count, copies the i-th. */
B200_API int ptts_c_stream_pending(ptts_stream_t* s, int index, char* buf, int buflen);
/* Voice cloning through the context. A voice argument ending in ".wav" (RIFF PCM 16 / 24 / 32-bit or float32, any channel count, mixed
 * down to mono, at its own sample rate in [8000, 192000] Hz) is cloned on first use, like a voice file is loaded. ptts_c_voice_add_audio
 * registers pcm[n] (mono, at sample_rate Hz) under `name`, which then works wherever a voice name does; returns the voice id or a B200_E*
 * error (B200_EINVAL for a sample rate outside [8000, 192000] or a name in use).
 * ptts_c_voice_export writes a cloned voice's audio_prompt [1, T, 1024] as an F32 safetensors voice file (B200_ENOTFOUND: not a clone). */
B200_API int ptts_c_voice_add_audio(ptts_context_t* ctx, const char* name, const float* pcm, long long n, int sample_rate);
B200_API int ptts_c_voice_export(ptts_context_t* ctx, const char* name, const char* path);
/* Host-only WAV reader: copies up to max mono samples into pcm (may be NULL), sets *sample_rate (may be NULL); returns the number of
 * samples in the file, or B200_EINVAL for a file that is not a readable RIFF PCM 16 / 24 / 32-bit or float32 WAV. */
B200_API int ptts_c_wav_read(const char* path, float* pcm, long long max, int* sample_rate);

/* ---- continuous batching: the batched extension of the streaming API (SURVEY 8b(3)). The reference rolls one stream to its next
 * sentence inside ptts_stream_receive (src/pocket_tts.cpp:494-519); here sentences of many utterances share the engine's slots and a
 * finished slot is refilled while the others keep generating. Utterance audio = its sentences' frames in order. ---- */
typedef struct ptts_batch_t ptts_batch_t;
typedef struct ptts_batch_stats { long long steps, frames, slot_steps, sentences, refills; double wall_ms, begin_ms, submit_ms, collect_ms; } ptts_batch_stats;
B200_API ptts_batch_t* ptts_c_batch_create(ptts_context_t* ctx, int n_slots /* 0 = all engine slots */);
B200_API void ptts_c_batch_destroy(ptts_batch_t* b);
/* refill policy: start queued sentences once refill_min slots are free or refill_every steps passed; stepped range rounded up to
 * range_quantum slots; keep_pcm 0 = count frames only. Values <= 0 (keep_pcm < 0) keep the default. */
B200_API int  ptts_c_batch_configure(ptts_batch_t* b, int refill_min, int refill_every, int range_quantum, int keep_pcm);
B200_API int  ptts_c_batch_add(ptts_batch_t* b, const char* voice, const char* text, float temp);   /* -> utterance id */
B200_API int  ptts_c_batch_add_tokens(ptts_batch_t* b, int voice_id, const int32_t* ids, int n_ids, int max_gen_len, int frames_after_eos,
                                      float temp, uint32_t rng_stream /* 0 = job index + 1 */);
/* Appends one more sentence, given as token ids, to utterance `utt` (an utterance of several sentences for callers that tokenise
 * themselves); returns utt. B200_EINVAL for a cancelled utterance. */
B200_API int  ptts_c_batch_append_tokens(ptts_batch_t* b, int utt, int voice_id, const int32_t* ids, int n_ids, int max_gen_len, int frames_after_eos,
                                         float temp, uint32_t rng_stream);
/* The same three with per-sentence sampling controls (NULL = defaults; B200_EINVAL when b200_sampling_check fails). The scheduler hands the
 * struct to the engine's sentence start unchanged. */
B200_API int  ptts_c_batch_add_sampling(ptts_batch_t* b, const char* voice, const char* text, float temp, const b200_sampling* sampling);
B200_API int  ptts_c_batch_add_tokens_sampling(ptts_batch_t* b, int voice_id, const int32_t* ids, int n_ids, int max_gen_len, int frames_after_eos,
                                               float temp, uint32_t rng_stream, const b200_sampling* sampling);
B200_API int  ptts_c_batch_append_tokens_sampling(ptts_batch_t* b, int utt, int voice_id, const int32_t* ids, int n_ids, int max_gen_len,
                                                  int frames_after_eos, float temp, uint32_t rng_stream, const b200_sampling* sampling);
B200_API long long ptts_c_batch_run(ptts_batch_t* b);                  /* runs every queued sentence to completion; frames produced */
B200_API int  ptts_c_batch_frames(ptts_batch_t* b, int utt);           /* frames generated for the utterance so far (popped ones included) */
B200_API int  ptts_c_batch_read(ptts_batch_t* b, int utt, float* pcm, int max_frames);   /* [n][1920]: the frames not popped yet */
B200_API void ptts_c_batch_stats(ptts_batch_t* b, ptts_batch_stats* out);
/* Online serving. add / add_tokens may be called at any time; utterances added since the last pump join the back of the queue, longest
 * sentence cap first. pump runs the scheduler until max_steps steps have been collected and at least one frame was produced, leaving the
 * pipeline full for the next call; once nothing is queued or running it drains the pipeline. Returns the frames produced, 0 when idle,
 * or a negative engine error. */
B200_API long long ptts_c_batch_pump(ptts_batch_t* b, int max_steps);
/* Copies up to max_frames ready frames [n][1920] of the utterance, in order, and returns n. A frame is ready once its step was collected
 * and every earlier sentence of the utterance is done. A sentence's audio is freed once it is done and fully popped. */
B200_API int  ptts_c_batch_pop(ptts_batch_t* b, int utt, float* pcm, int max_frames);
/* Drops the utterance's queued sentences and frees the slots of its running ones (their frames still in flight are discarded); its audio
 * not popped yet is freed and its frame count stops growing. A done utterance is left as it is. An open utterance is also closed. */
B200_API int  ptts_c_batch_cancel(ptts_batch_t* b, int utt);
/* 0 queued, 1 running, 2 done, 3 cancelled, 4 open and waiting for text (ptts_c_batch_open: none of its sentences queued or running; an open
 * utterance is never reported done); *ready_frames (optional) = frames ptts_c_batch_pop would return now. */
B200_API int  ptts_c_batch_status(ptts_batch_t* b, int utt, int* ready_frames);
/* Streamed text, the batched counterpart of ptts_stream_send / ptts_stream_flush: an LLM can feed its reply as it is written.
 * ptts_c_batch_open returns an utterance id that accepts text; the voice is resolved as ptts_c_batch_add resolves it (name, voice file or
 * .wav) and sampling may be NULL (defaults). ptts_c_batch_send feeds a chunk of any size to the utterance's sentence splitter; every
 * sentence it completes (once the first character after its terminator arrives, as in ptts_stream_send) becomes a sentence of the
 * utterance, queued at the next pump like any addition; returns the number of sentences added (an empty chunk adds nothing, it does not
 * flush). ptts_c_batch_close ends the text: the splitter's flush applies the final-period rule and emits the tail; returns the sentences
 * added. From then on the utterance behaves like one made by ptts_c_batch_add. Each sentence's RNG stream id is the job index + 1 when it
 * is split off, so with no other addition between the first send and the close the audio is bitwise that of ptts_c_batch_add of the same
 * text. send / close on an utterance that is not open (never opened, closed, cancelled) return B200_EINVAL. */
B200_API int  ptts_c_batch_open(ptts_batch_t* b, const char* voice, float temp, const b200_sampling* sampling);
B200_API int  ptts_c_batch_send(ptts_batch_t* b, int utt, const char* chunk);
B200_API int  ptts_c_batch_close(ptts_batch_t* b, int utt);
/* ptts_c_batch_open with an engine voice id (B200_EINVAL for an unknown voice). On a batch over caller-supplied ops it needs a tokenizer
 * from ptts_c_batch_set_text. */
B200_API int  ptts_c_batch_open_id(ptts_batch_t* b, int voice_id, float temp, const b200_sampling* sampling);
/* The same scheduler over caller-supplied engine calls (CPU tests drive it with a mock engine). */
typedef int (*ptts_batch_begin_fn)(void* user, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens, const int32_t* tok_off,
                                   const int32_t* max_gen_len, const int32_t* frames_after_eos, const float* temp, const uint32_t* rng_stream);
typedef int (*ptts_batch_submit_fn)(void* user, int slot0, int n);
typedef int (*ptts_batch_collect_fn)(void* user, float* pcm, int32_t* produced);
B200_API ptts_batch_t* ptts_c_batch_create_with_ops(void* user, ptts_batch_begin_fn begin, ptts_batch_submit_fn submit, ptts_batch_collect_fn collect,
                                                    int n_slots, int frame_size);
/* retires slots whose sentence was cancelled (b200_end_sentences); NULL = such slots stay live on the engine until refilled */
typedef int (*ptts_batch_end_fn)(void* user, int n, const int32_t* slots);
B200_API ptts_batch_t* ptts_c_batch_create_with_ops_ex(void* user, ptts_batch_begin_fn begin, ptts_batch_submit_fn submit, ptts_batch_collect_fn collect,
                                                       ptts_batch_end_fn end, int n_slots, int frame_size);
/* begin with each sentence's sampling controls (b200_begin_sentences_sampling's signature minus the engine) */
typedef int (*ptts_batch_begin_sampling_fn)(void* user, int n, const int32_t* slots, const int32_t* voices, const int32_t* tokens, const int32_t* tok_off,
                                            const int32_t* max_gen_len, const int32_t* frames_after_eos, const float* temp, const uint32_t* rng_stream,
                                            const b200_sampling* sampling);
B200_API ptts_batch_t* ptts_c_batch_create_with_ops_sampling(void* user, ptts_batch_begin_sampling_fn begin, ptts_batch_submit_fn submit,
                                                             ptts_batch_collect_fn collect, ptts_batch_end_fn end, int n_slots, int frame_size);

/* Host-only text front end (no GPU needed): tokenizer + sentence splitter objects. */
typedef struct ptts_text_t ptts_text_t;
B200_API ptts_text_t* ptts_c_text_create(const char* tokenizer_model);
B200_API void ptts_c_text_destroy(ptts_text_t* t);
B200_API int  ptts_c_text_encode(ptts_text_t* t, const char* text, int32_t* ids, int max_ids);
B200_API void ptts_c_text_send(ptts_text_t* t, const char* chunk);
B200_API void ptts_c_text_flush(ptts_text_t* t);
B200_API void ptts_c_text_reset(ptts_text_t* t);
B200_API int  ptts_c_text_pop(ptts_text_t* t, char* buf, int buflen);
/* Gives a batch without a context (ptts_c_batch_create_with_ops*) the tokenizer of t for ptts_c_batch_open_id / send / close; t is borrowed
 * and must outlive the batch. B200_EINVAL on a batch over a context, which uses the context's tokenizer. */
B200_API int  ptts_c_batch_set_text(ptts_batch_t* b, const ptts_text_t* text);

#ifdef __cplusplus
}
#endif
#endif
