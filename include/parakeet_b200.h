/* parakeet_b200.h -- the drop-in boundary: a flat C-ABI over the B200-native hot path
 *
 *     16 kHz PCM -> log-mel -> FastConformer encoder -> CTC / TDT greedy decode
 *
 * The reference (Frikallo/parakeet.cpp @ 40bbd7e) has no C API ("C API" is an
 * unchecked roadmap item, README.md:518); its boundary for this path is C++:
 * parakeet::Transcriber (include/parakeet/transcribe.hpp:55-190) calling
 * preprocess_audio (src/audio.cpp:100), FastConformerEncoder::forward
 * (src/encoder.cpp:253), CTCDecoder::forward + ctc_greedy_decode (src/ctc.cpp:12,40)
 * and tdt_greedy_decode (src/tdt.cpp:36).  Each entry point below names the
 * reference function(s) it replaces.  include/parakeet/transcribe.hpp in this
 * repository is the header-only C++ shim with the reference's class signatures
 * on top of this ABI; INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions: plain pointers and sizes only; every call returns pk_status and
 * never throws; the opaque engine owns all device memory, its CUDA stream and
 * graphs; the caller owns host buffers.  One engine per device; calls on one
 * engine are serialised on its stream (thread-compatible, not thread-safe).
 * There is no CPU fallback: without a CUDA device pk_engine_create fails.
 */
#ifndef PARAKEET_B200_H
#define PARAKEET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    PK_OK = 0,
    PK_ERR_INVALID = 1,   /* bad argument / shape */
    PK_ERR_IO = 2,        /* cannot open / parse weights */
    PK_ERR_CUDA = 3,      /* CUDA runtime / driver error */
    PK_ERR_MISSING = 4,   /* tensor missing from the state dict */
    PK_ERR_CAPACITY = 5,  /* batch exceeds the engine's configured capacity */
    PK_ERR_NCCL = 6
} pk_status;

/* PK_DECODER_RNNT is the only decoder of an RNNT engine (pk_config.n_durations == 0), and the only one it accepts;
 * TDT and CTC engines reject it.  Phrase boosting and streaming are not available on RNNT engines. */
typedef enum { PK_DECODER_CTC = 0, PK_DECODER_TDT = 1, PK_DECODER_RNNT = 2 } pk_decoder;

/* GEMM arithmetic.  PK_MATH_BF16X3 (default): tcgen05 kind::f16 MMAs on bf16
 * hi/lo operand splits, 3 MMAs per product (hi*hi + hi*lo + lo*hi), fp32
 * accumulation in TMEM: ~1e-5 relative, the parity mode.  PK_MATH_BF16X1: hi*hi only
 * (fast, ~4e-3).  PK_MATH_FP32: CUDA-core fp32 GEMM (bring-up / checker). */
typedef enum { PK_MATH_BF16X3 = 0, PK_MATH_BF16X1 = 1, PK_MATH_FP32 = 2 } pk_math;

/* Mirrors EncoderConfig / PredictionConfig / JointConfig / TDTCTCConfig
 * (include/parakeet/config.hpp:9-75).  pk_config_110m / pk_config_tdt_600m fill
 * it with make_110m_config (:77-95) / make_tdt_600m_config (:98-116). */
typedef struct {
    int32_t mel_bins;          /* 80 | 128 */
    int32_t sub_channels;      /* 256 */
    int32_t d_model;           /* 512 | 1024 */
    int32_t n_layers;          /* 17 | 24 */
    int32_t n_heads;           /* 8 */
    int32_t ff;                /* 2048 | 4096 */
    int32_t conv_kernel;       /* 9 */
    int32_t vocab;             /* 1025 | 8193, blank = vocab-1 */
    int32_t pred_hidden;       /* 640 */
    int32_t lstm_layers;       /* 1 | 2 */
    int32_t joint_hidden;      /* 640 */
    int32_t n_durations;       /* 5; 0 = RNNT joint (RNNTConfig, rnnt.hpp): one output head "out_proj_" of vocab rows */
    int32_t durations[8];      /* {0,1,2,3,4} */
    int32_t has_ctc;           /* ParakeetTDTCTC: 1, ParakeetTDT / ParakeetRNNT: 0 */
    int32_t joint_prefix_tdt;  /* 1: keys "tdt_joint_." (tdt_ctc.cpp:5-9); 0: "joint_." (tdt.cpp:28-32, rnnt.cpp:46-50) */
    int32_t max_symbols;       /* max_symbols_per_step, 10 (tdt.hpp, rnnt.hpp); observable in RNNT decoding only:
                                  an RNNT engine holds up to max_symbols tokens per encoder frame */
    /* engine capacity (not model shape) */
    int32_t max_batch;         /* utterances per call */
    int32_t max_samples;       /* per utterance */
    int32_t math;              /* pk_math */
} pk_config;

typedef struct pk_engine pk_engine;

void pk_config_110m(pk_config *cfg);      /* config.hpp:77-95  */
void pk_config_tdt_600m(pk_config *cfg);  /* config.hpp:98-116 */
void pk_config_rnnt_600m(pk_config *cfg); /* config.hpp:119-135 (nvidia/parakeet-rnnt-0.6b) */

/* Replaces Transcriber::Transcriber + to_gpu (transcribe.hpp:59-71):
 * safetensors::load (axiom io_safetensors.cpp:123-160) + load_state_dict(strict=false)
 * (axiom module.cpp:24-38) + Module::to(GPU).  Missing tensors for modules on the
 * path are an error (PK_ERR_MISSING); extra tensors are ignored. */
pk_status pk_engine_create(const pk_config *cfg, const char *safetensors_path, int device,
                           pk_engine **out);
void pk_engine_destroy(pk_engine *e);
/* Last error text of this engine (or of the failed create when e == NULL). */
const char *pk_last_error(const pk_engine *e);

/* Shape helpers (operations.cpp:3191-3196 output-length formula). */
int32_t pk_mel_frames(int64_t n_samples);           /* 1 + n/160                       */
int32_t pk_encoder_frames(int32_t n_mel_frames);    /* three stride-2 k3 p1 stages     */

/* Replaces preprocess_audio (src/audio.cpp:100-158) for a batch of utterances.
 * pcm: host fp32, utterance i = pcm[offsets[i] .. offsets[i+1]).
 * feats_out: host fp32, packed (sum_i frames_i, mel_bins); n_frames_out[n_utt]. */
pk_status pk_mel(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt,
                 float *feats_out, int32_t *n_frames_out);

/* Replaces FastConformerEncoder::forward (src/encoder.cpp:253-271).
 * feats: host fp32 packed (sum frames_i, mel_bins); enc_out: host fp32 packed
 * (sum T'_i, d_model); enc_lens_out[n_utt] = T'_i.
 * Optional debug taps (may be NULL): sub_out packed (sum T'_i, d_model) after
 * ConvSubsampling; layers_out (n_layers, sum T'_i, d_model) after each block. */
pk_status pk_encode(pk_engine *e, const float *feats, const int32_t *n_frames, int32_t n_utt,
                    float *enc_out, int32_t *enc_lens_out, float *sub_out, float *layers_out);

/* Token streams of a batch.  Row i holds len[i] entries of ids/start/end/conf
 * at stride `cap`.  start/end are encoder frames (0.08 s, timestamp.hpp:31-35),
 * conf = exp(log-prob) as in ctc.cpp:110 / tdt.cpp:165.  */
typedef struct {
    int32_t cap;        /* in: row capacity (>= max tokens per utterance)   */
    int32_t *ids;       /* [n_utt * cap] */
    int32_t *start;     /* [n_utt * cap] or NULL */
    int32_t *end;       /* [n_utt * cap] or NULL */
    float *conf;        /* [n_utt * cap] or NULL */
    int32_t *len;       /* [n_utt] */
} pk_tokens;

/* Decode-only entry points on a host encoder output (packed (sum T_i, d_model)):
 * CTCDecoder::forward + ctc_greedy_decode(_with_timestamps) (src/ctc.cpp:12-127) and
 * tdt_greedy_decode(_with_timestamps) (src/tdt.cpp:36-201). */
pk_status pk_decode(pk_engine *e, const float *enc, const int32_t *enc_lens, int32_t n_utt,
                    pk_decoder dec, pk_tokens *out);

/* CTC head log-probs (CTCDecoder::forward, src/ctc.cpp:12-25) for inspection:
 * enc packed (sum T_i, d_model) -> logprobs packed (sum T_i, vocab). */
pk_status pk_ctc_logprobs(pk_engine *e, const float *enc, int32_t total_frames, float *logprobs_out);

/* The whole path, replacing the body of Transcriber::transcribe
 * (transcribe.hpp:99-179) for a batch: host PCM in, token streams out.
 * H2D of the PCM and D2H of the tokens happen inside the call. */
pk_status pk_transcribe_batch(pk_engine *e, const float *pcm, const int64_t *offsets,
                              int32_t n_utt, pk_decoder dec, pk_tokens *out);

/* Device-resident variant for throughput measurement: stage PCM once ...
 * Buffer lifetime: when `pcm` is page-locked, the engine DMAs straight from it and pk_stage_pcm returns while
 * the copy may still be in flight -- the buffer must stay valid AND unmodified until the next pk_fetch_tokens /
 * pk_sync on this engine returns (the same holds for a buffer handed to pk_prefetch_pcm).  Pageable buffers are
 * copied before the call returns. */
pk_status pk_stage_pcm(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt);
/* Serving pipeline (no reference counterpart: the reference is synchronous and batch-1).  Starts the
 * host-to-device copy of the NEXT batch into the engine's second PCM buffer on a copy stream and
 * returns at once, so the copy runs under the current batch's kernels:
 *     pk_prefetch_pcm(b0); loop { pk_stage_pcm(b_i); pk_run_staged(); pk_prefetch_pcm(b_{i+1}); pk_fetch_tokens(); }
 * pk_stage_pcm / pk_transcribe_batch with the same (pcm, offsets, n_utt) then adopt the prefetched buffer
 * instead of copying.  The samples are read when this call is made; the buffer must be page-locked and
 * packed back to back (PK_ERR_INVALID otherwise) and must stay valid until the adopting call returns. */
pk_status pk_prefetch_pcm(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt);
/* ... then run the path on the staged batch; tokens stay on the device until
 * pk_fetch_tokens.  Asynchronous on the engine stream. */
pk_status pk_run_staged(pk_engine *e, pk_decoder dec);
pk_status pk_fetch_tokens(pk_engine *e, pk_tokens *out);
pk_status pk_sync(pk_engine *e);

/* Device token buffer of the last run for the single cross-GPU exchange:
 * int32 rows [n_utt][1 + cap] = (len, ids...).  The caller (torch.distributed /
 * NCCL) all-gathers this buffer; see INTEGRATION.md. */
pk_status pk_token_buffer(pk_engine *e, void **dev_ptr, int32_t *rows, int32_t *row_ints);

/* ---- Jobs and the single cross-GPU exchange (SURVEY.md section 8e; BASELINE configs[4]: 8192 clips over 8 GPUs).
 * The reference is single-device and batch-1 (transcribe.hpp:170-171); this is what a sharded host adds around
 * Transcriber::transcribe.  A rank owns a contiguous block of clips and runs it in micro-batches of at most
 * pk_config.max_batch; after every pk_run_staged, pk_job_append copies that micro-batch's token rows
 * (int32 [1 + cap] = len, ids...) into a device-resident job buffer of rows_local rows (asynchronous, engine
 * stream).  pk_allgather_tokens then issues ONE ncclAllGather of the job buffer on the engine stream (no host
 * synchronisation; rows a rank did not fill have len = 0), and pk_job_fetch copies local (gathered = 0) or
 * gathered (gathered = 1: rank-major [world][rows_local]) rows to the host.
 *
 * NCCL is resolved at run time (dlopen "libnccl.so.2": the copy the process already uses); without it these
 * calls return PK_ERR_NCCL.  Either pass the host's own ncclComm_t to pk_allgather_tokens, or let the engine
 * own one: rank 0 calls pk_nccl_unique_id, the host broadcasts the 128 bytes, every rank calls pk_comm_init_rank. */
#define PK_NCCL_UNIQUE_ID_BYTES 128
pk_status pk_job_begin(pk_engine *e, int64_t rows_local, int32_t world);
pk_status pk_job_append(pk_engine *e);
pk_status pk_nccl_unique_id(void *id128);
pk_status pk_comm_init_rank(pk_engine *e, const void *id128, int32_t rank, int32_t world);
pk_status pk_allgather_tokens(pk_engine *e, void *nccl_comm /* ncclComm_t, or NULL: the engine's communicator */);
pk_status pk_job_fetch(pk_engine *e, int32_t gathered, int32_t *rows_out, int64_t n_rows, int32_t *row_ints);
/* Device-resident job input for throughput measurement: copy the PCM of a whole job (any number of utterances,
 * host buffer, packed or not) to the device once, then make micro-batch [first, first + n_utt) the staged batch
 * without a copy (pk_run_staged / pk_job_append follow as usual). */
pk_status pk_job_stage_pcm(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt);
pk_status pk_job_select(pk_engine *e, int32_t first, int32_t n_utt);

/* ---- Streaming (SURVEY.md section 8f row 2; BASELINE configs[3]: eou-120m, 160 ms chunks), replacing
 * StreamingTranscriber::transcribe_chunk / reset (src/eou.cpp:111-149): StreamingAudioPreprocessor::process_chunk
 * (src/audio.cpp:195-259), StreamingFastConformerEncoder::forward_chunk (src/streaming_encoder.cpp:425-472) and
 * rnnt_streaming_decode_chunk (src/eou.cpp:17-98).  The reference advances ONE stream per call; here n_streams streams
 * advance in lock step and share every weight read.  The engine must have been created with max_batch >= n_streams and
 * max_samples large enough that its encoder-frame capacity is >= att_context_left + frames per chunk (6.4 s is plenty
 * for the eou-120m preset: left context 70).  Per-stream state (sample overlap, leftover mel frames, K/V and conv caches,
 * LSTM state, last token, frame offset) lives on the device.
 *   pk_stream_open : allocate the state of n_streams streams (att_context_left / right of StreamingEncoderConfig,
 *                    streaming_encoder.hpp:18-24; the right context / mask is inert in the reference's CPU path and is
 *                    not applied, see DESIGN.md).
 *   pk_stream_step : stream s receives pcm[offsets[s] .. offsets[s+1]) (host fp32; an empty chunk is allowed); `out` rows
 *                    (n = n_streams, may be NULL) receive the tokens emitted BY THIS STEP, start/end = absolute encoder
 *                    frames (the end frame is not clamped to the chunk, eou.cpp:81-84).  Optional taps (may be NULL):
 *                    mel_out packed (sum nf_s, mel_bins) new log-mel frames, n_mel[s] = nf_s; enc_out packed
 *                    (sum C_s, d_model) encoder rows of this step, n_enc[s] = C_s.  A first chunk of 400..511 samples
 *                    returns PK_ERR_INVALID where the reference's STFT throws (fft.cpp:1516-1521).
 *   pk_stream_reset: StreamingTranscriber::reset for one stream (-1: all). */
pk_status pk_stream_open(pk_engine *e, int32_t n_streams, int32_t max_chunk_samples, int32_t att_context_left,
                         int32_t att_context_right);
pk_status pk_stream_reset(pk_engine *e, int32_t stream);
pk_status pk_stream_step(pk_engine *e, const float *pcm, const int64_t *offsets, pk_tokens *out, float *mel_out,
                         int32_t *n_mel, float *enc_out, int32_t *n_enc);
int32_t pk_stream_count(const pk_engine *e);

/* Host-only probe of the checkpoint reader (safetensors::load, axiom io_safetensors.cpp:16-160: F32 / F16 / BF16 / F64
 * tensors, converted to fp32): opens the file (PK_ERR_IO + pk_last_error(NULL) on a malformed header), and if `name` is
 * given converts that tensor into out[0 .. cap) and reports its element count.  Needs no device. */
pk_status pk_safetensors_probe(const char *path, const char *name, float *out, int64_t cap, int64_t *numel);

/* Number of utterances of the last pk_fetch_tokens whose TDT hypothesis was cut at the engine's token capacity
 * (2 T'max + 8 per utterance; only reachable on inputs that livelock the reference's tdt_greedy_decode, which
 * never forces an advance after max_symbols_per_step, src/tdt.cpp:66-104). */
int32_t pk_truncated_count(const pk_engine *e);

/* CUDA stream of the engine (cudaStream_t as void*), for event timing. */
void *pk_stream(pk_engine *e);
/* Number of kernel launches issued by the engine since creation (the
 * `gpu_launches` claim in bench.py). */
int64_t pk_launch_count(const pk_engine *e);

/* Measurement aids (bench.py): per-kernel-class device time measured with CUDA events on
 * the engine stream between begin/end (classes in pk_profile_names() order, comma
 * separated; ms / launch counts / algorithmic GEMM flops summed per class), and an L2
 * flush (writes a 256 MiB scratch buffer on the engine stream). */
pk_status pk_profile_begin(pk_engine *e);
pk_status pk_profile_end(pk_engine *e, double *ms, int64_t *counts, double *flops, int32_t n);
const char *pk_profile_names(void);
pk_status pk_flush_l2(pk_engine *e);

/* Debug aid: cycles CTA 0 of the last TDT decode spent in {P1, B1, P2, B2, P3, B3, P4}; out8[7] =
 * number of lock-step decode steps. */
pk_status pk_debug_tdt_phases(pk_engine *e, int64_t *out8);
/* Debug aid: cycles CTA 0 spent in the sections of the decode kernel's passes since the previous call:
 * {x staging, products, partial store + cluster barrier, DSMEM gather + finalise, number of passes, 0, 0, 0}. */
pk_status pk_debug_tdt_passes(pk_engine *e, int64_t *out8);

/* GPU self-check of the tcgen05 GEMM kernel against the fp32 CUDA-core GEMM on seeded
 * random data (epi_kind: EpiKind of csrc/pk_common.cuh; math: PK_MATH_BF16X3 | PK_MATH_BF16X1). */
pk_status pk_selftest_gemm(int device, int M, int N, int K, int epi_kind, int math, uint32_t seed,
                           float *max_err, float *max_ref);
/* GPU self-check of the residual GEMM with the LayerNorm fused into its epilogue (csrc/gemm_tc_ln.cu, N = 512, run in place)
 * against the fp32 GEMM followed by the stand-alone LayerNorm kernel.  mode 0: x = resid + a(A W^T + b), planes = LN1(x);
 * 1: x = LN1(.), planes = LN2(x);  2: x = LN1(.), planes = split(x);  3: mode 0 without a residual.
 * err4 = {max |x - x_ref|, max |x_ref|, max |planes - planes_ref|, max |planes_ref|}. */
pk_status pk_selftest_gemm_ln(int device, int M, int K, int mode, int math, uint32_t seed, float *err4);
/* GPU self-check of the tcgen05 attention kernel (csrc/attention_umma.cu: head_dim 64, <= 128 frames per utterance) against the
 * fp32 CUDA-core attention kernel on seeded random inputs (d_model 512, 8 heads), utterance lengths lens[0..n).  mode bit 0:
 * zero position table; bit 1: zero keys.  err2 = {max |ctx - ctx_ref|, max |ctx_ref|}. */
pk_status pk_selftest_attention(int device, const int32_t *lens, int n, int tmax, int mode, uint32_t seed, float *err2);

/* Host-side text helpers (pure C++ host code; no device work):
 * Tokenizer::load/decode (src/vocab.cpp:10-64), group_timestamps (src/timestamp.cpp:24-75). */
typedef struct pk_vocab pk_vocab;
pk_status pk_vocab_load(const char *vocab_path, pk_vocab **out);
void pk_vocab_free(pk_vocab *v);
int32_t pk_vocab_size(const pk_vocab *v);
/* Longest piece in bytes: pk_detokenize / pk_group_words never write more than n * (that + 1) + 1 bytes for n tokens. */
int32_t pk_vocab_max_piece_bytes(const pk_vocab *v);
/* Writes NUL-terminated UTF-8 into buf (truncated to cap-1); returns full length. */
int32_t pk_detokenize(const pk_vocab *v, const int32_t *ids, int32_t n, char *buf, int32_t cap);
/* Words are written '\n'-separated into buf; returns the number of words. */
int32_t pk_group_words(const pk_vocab *v, const int32_t *ids, const int32_t *start,
                       const int32_t *end, const float *conf, int32_t n, char *buf, int32_t cap,
                       float *w_start, float *w_end, float *w_conf);

/* Tokenizer::encode (src/vocab.cpp:76-117): U+2581-prefixed, spaces -> U+2581, greedy longest piece match on
 * bytes, unknown bytes skipped.  Writes at most cap ids; returns the full count. */
int32_t pk_tokenize(const pk_vocab *v, const char *text, int32_t *ids, int32_t cap);

/* Phrase-boosted CTC greedy decode of ONE utterance on the host (widening row: SURVEY.md section 8f(3)), replacing
 * ctc_greedy_decode_boosted / ctc_greedy_decode_with_timestamps_boosted (src/phrase_boost.cpp:70-176) and the
 * ContextTrie they use (:9-66).  logprobs = (n_frames, vocab) row-major as returned by pk_ctc_logprobs; the
 * phrases are token-id sequences (pk_tokenize), phrase p = phrase_ids[phrase_off[p] .. phrase_off[p+1]).
 * Every frame takes argmax_v(logprob[v] + boost * [v continues an active phrase]) (first maximum), the trie
 * advances on emissions, confidences are exp of the UNboosted log-prob.  start / end / conf may be NULL.
 * Returns the number of tokens (at most `cap` are written) or -1 on invalid arguments. */
int32_t pk_ctc_decode_boosted(const float *logprobs, int32_t n_frames, int32_t vocab, int32_t blank,
                              const int32_t *phrase_ids, const int32_t *phrase_off, int32_t n_phrases, float boost,
                              int32_t *ids, int32_t *start, int32_t *end, float *conf, int32_t cap);

/* Phrase boosting ON THE DEVICE for both decoders (widening row: SURVEY.md section 8f(3)), replacing the decode loops of
 * ctc_greedy_decode(_with_timestamps)_boosted and tdt_greedy_decode(_with_timestamps)_boosted (src/phrase_boost.cpp:70-352)
 * as Transcriber::transcribe uses them when TranscribeOptions::boost_phrases is set (transcribe.hpp:110-137, :158-165).
 * The phrases are token-id sequences (pk_tokenize), phrase p = phrase_ids[phrase_off[p] .. phrase_off[p+1]); the engine builds the
 * ContextTrie (:9-66) and keeps it on the device.  While set, every decode of this engine (pk_transcribe_batch,
 * pk_run_staged, pk_decode; CTC and TDT) adds `boost` to the label scores of the tokens that continue an active phrase;
 * the trie state is per utterance and advances on emissions; confidences stay exp(raw log-prob).  n_phrases = 0 clears
 * it.  (Not applied by pk_stream_step.)  At most 64 simultaneously active trie states per utterance. */
pk_status pk_set_boost(pk_engine *e, const int32_t *phrase_ids, const int32_t *phrase_off, int32_t n_phrases, float boost);

/* Sample-rate conversion (widening row: SURVEY.md section 8f(4)), replacing parakeet::resample / sinc_resample
 * (src/audio_io.cpp:123-195, :238-251): 32-tap Kaiser (beta 7.857) windowed sinc in double, output length
 * ceil(n * dst / src) (pk_resample_len), implemented as a POLYPHASE filter: the weights depend only on the phase
 * (i * down) mod up, so they are tabulated once per rate pair (csrc/resample.cu).
 *   pk_stage_pcm_rate : like pk_stage_pcm for a batch recorded at `src_rate`: the raw samples go to the device and are
 *                       converted there straight into the staged 16 kHz batch (read_audio's resampling, audio_io.cpp:227-232,
 *                       without a host pass).  Utterance lengths are checked at 16 kHz.
 *   pk_resample_batch : device conversion of a batch between arbitrary rates, results back to the host
 *                       (out_offsets = prefix sums of pk_resample_len per utterance).
 *   pk_resample       : the same filter evaluated on the host for engine-less callers (parakeet::resample of the C++
 *                       shim); writes at most `cap` samples, returns the full length or -1 on invalid arguments. */
int64_t pk_resample_len(int64_t n, int32_t src_rate, int32_t dst_rate);
int64_t pk_resample(const float *in, int64_t n, int32_t src_rate, int32_t dst_rate, float *out, int64_t cap);
pk_status pk_stage_pcm_rate(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, int32_t src_rate);
pk_status pk_resample_batch(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, int32_t src_rate,
                            int32_t dst_rate, float *out, const int64_t *out_offsets);

#ifdef __cplusplus
}
#endif
#endif /* PARAKEET_B200_H */
