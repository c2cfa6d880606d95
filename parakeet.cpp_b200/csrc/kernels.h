// kernels.h -- host-callable launchers of the sm_100a kernels (one .cu per op group).
#pragma once
#include <cuda.h>

#include "pk_common.cuh"

#define PK_MAX_LSTM 4

namespace pk {

// ------------------------------------------------------------------ mel.cu (K1, K2)
struct MelTables {
    const float *window;    // [400] symmetric Hann (fp32 of the double formula)
    const float2 *tw256;    // [256] exp(-2 pi i m / 256)
    const float2 *tw512;    // [257] exp(-2 pi i k / 512)
    const float *fb_w;      // non-zero filterbank weights, filter-major
    const int32_t *fb_start, *fb_len, *fb_off;   // [n_mels]
    int fb_nnz;
};
size_t mel_smem_bytes(const MelTables &tb);
// part: scratch of mel_part_floats(n_utt, n_mels) floats (per-chunk statistics of the normalisation), one slice per utterance
size_t mel_part_floats(int n_utt, int n_mels);
void launch_mel(const float *pcm, const int64_t *pcm_off, const int32_t *frame_off, int n_utt, int max_frames,
                int n_mels, const MelTables &tb, float *logmel, float *feats, float *part, cudaStream_t st);

// streaming variant (StreamingAudioPreprocessor::process_chunk, src/audio.cpp:195-259): `sig` holds, per stream, the
// already pre-emphasised samples [overlap | chunk]; frame f = window . sig[f*160 .. f*160+512) (center = False, no
// reflection), n_frames[b] frames, log-mel WITHOUT normalisation written to logmel rows out_row[b] + f.
void launch_mel_stream(const float *sig, const int64_t *sig_off, const int32_t *n_frames, const int32_t *out_row, int n_streams,
                       int max_frames, int n_mels, const MelTables &tb, float *logmel, cudaStream_t st);

// ------------------------------------------------------------------ stream.cu (streaming eou path)
constexpr int STREAM_OVL_CAP = 512;   // overlap buffer per stream (< 400 samples are ever kept, audio.cpp:225-240)
struct StreamPlan {                   // one row per stream and step, computed on the host from the chunk sizes
    int64_t chunk_off;                // offset of this stream's chunk in the packed chunk buffer
    int64_t sig_off;                  // offset of [overlap | pre-emphasised chunk] in the signal scratch
    int32_t chunk_len, ovl_len;       // samples in the chunk / carried overlap
    int32_t consumed;                 // samples covered by the frames of this step (0: none; overlap = whole signal)
    int32_t nf;                       // new mel frames (the reference's STFT yields one fewer than its own count, DESIGN.md)
    int32_t left;                     // leftover mel frames from the previous steps (< 8)
    int32_t min_off;                  // first row of [leftover | new] frames in mel_in
    int32_t take;                     // frames consumed by the subsampling this step (multiple of 8)
    int32_t feat_off;                 // first row in the packed encoder input (valid if take > 0)
};
struct StreamState {
    float *ovl;                       // [S][STREAM_OVL_CAP]
    float *last;                      // [S] pre-emphasis carry (audio.cpp:206-213)
    float *melq;                      // [S][8][n_mels] leftover mel frames (streaming_encoder.cpp:348-385)
};
void launch_stream_prep(const float *chunk, const StreamPlan *plan, StreamState st, int n_streams, float *ssig, float *mel_in,
                        int n_mels, cudaStream_t s);
void launch_stream_post(const float *chunk, const StreamPlan *plan, StreamState st, int n_streams, const float *ssig,
                        const float *mel_in, int n_mels, float *feats, cudaStream_t s);
bool launch_stream_attention(const float *qkv, int ld_qkv, const int32_t *row_off, const int32_t *act_stream, int n_active,
                             int max_C, const int32_t *cache_len, const int32_t *ring_start, float *kc, float *vc, int L,
                             int n_heads, int hd, int d_model, const float *pp, int tmax, const float *bu, const float *bv,
                             ActBuf out, cudaStream_t s);
bool launch_stream_dwconv(const float *glu, const int32_t *row_off, const int32_t *act_stream, int n_active, float *cache, int d,
                          int ks, const float *w, const float *bias, ActBuf out, cudaStream_t s);

// ------------------------------------------------------------------ resample.cu (front-of-path rate conversion)
// utterance b: in[in_off[b] .. in_off[b+1]) at src_rate -> out[out_off[b] .. out_off[b+1]) at dst_rate (lengths = pk_resample_len)
bool launch_resample(const float *in, const int64_t *in_off, const int64_t *out_off, int n_utt, int64_t max_out, int src_rate,
                     int dst_rate, float *out, cudaStream_t st);

// ------------------------------------------------------------------ subsample.cu (K3, K4)
void launch_subsample_conv1_dw1(const float *feats, const int32_t *frame_off, const int32_t *s2_off, int n_utt,
                                int max_t2, int mel, int C, const float *w1, const float *b1, const float *wd,
                                const float *bd, ActBuf out, cudaStream_t st);
void launch_subsample_dw(const float *in, const int32_t *in_rows, const int32_t *in_off, const int32_t *out_off,
                         int n_utt, int fin, int C, const float *wd, const float *bd, ActBuf out,
                         int total_out_rows, cudaStream_t st);

// ------------------------------------------------------------------ gemm_simt.cu / gemm_tc.cu (K5)
void launch_gemm_simt(const float *A, int lda, const float *W, int ldw, int M, int N, int K,
                      const EpiParams &epi, cudaStream_t st);

// tcgen05 path (gemm_tc.cu): a K-major bf16 matrix [rows][K] as TMA tensor maps of its hi
// (and lo) split planes, box = 64 (K) x box_rows, SWIZZLE_128B.
struct TcOperand {
    CUtensorMap hi, lo;
    bool has_lo = false;
    uint32_t box_rows = 0;
};
bool make_tc_operand(TcOperand *out, const bf16 *hi, const bf16 *lo, uint64_t rows, uint64_t K, uint32_t box_rows);
// Output-side tensor map for the TMA-store epilogue: [rows][ld] matrix of bf16 (is_f32 = false: box 64 x 32) or fp32
// (box 32 x 32), 128-byte inner box, SWIZZLE_128B.
bool make_tc_out_map(CUtensorMap *out, const void *ptr, bool is_f32, uint64_t rows, uint64_t ld);
int tc_tile_n(int N);
void tc_set_2cta(bool on);   // debug/measurement switch: use the cta_group::2 kernel for N >= 256 (default off; PK_GEMM_2CTA=1)   // N-tile (= box_rows of the weight operand) chosen for an [N][K] weight
void tc_set_debug(int bits); // measurement aid (PK_GEMM_DBG): bit 0 = skip the epilogue's work, bit 1 = skip the TMA loads (results are garbage)
double tc_probe_mhz();
void tc_print_timeline(int n_tiles);
// cl = 2 | 4 with A_slice = the A operand with a 128 / cl-row box: clusters of cl CTAs along N that share (TMA multicast) the
// A tile; taken when gemm_tc_cluster_supported(N, epi.kind, cl), else the plain persistent kernel.
bool gemm_tc_cluster_supported(int N, int epi_kind, int cl);
cudaError_t launch_gemm_tc(const TcOperand &A, const TcOperand &W, int M, int N, int K, bool split3,
                           const EpiParams &epi, cudaStream_t st, int cl = 1, const TcOperand *A_slice = nullptr);

// ------------------------------------------------------------------ gemm_tc_ln.cu (K5b: residual GEMM + fused LayerNorm)
//     v = resid + alpha * (A . W^T + bias)   (resid may be null);   y1 = LN1(v);   y2 = LN2(y1) if ln2_w
//     out_f32 = out_ln1 ? y1 : v   (may alias resid);   planes = hi/lo split of the last LayerNorm's result
// N must be a full LayerNorm row of 4 x 128 columns (one 4-CTA cluster per 128-row block; statistics through DSMEM).
struct LnEpi {
    const float *bias = nullptr, *resid = nullptr;
    float alpha = 1.0f;
    float *out_f32 = nullptr;
    const float *ln1_w = nullptr, *ln1_b = nullptr, *ln2_w = nullptr, *ln2_b = nullptr;
    bool out_ln1 = false;
    ActBuf planes;
    float eps = 1e-5f;
};
bool gemm_tc_ln_supported(int N);
void gemm_tc_ln_set_debug(int on);            // measurement aid (PK_LN_DBG=1): per-tile epilogue timeline of CTA 0
void gemm_tc_ln_print_timeline(int n_tiles);
cudaError_t launch_gemm_tc_ln(const TcOperand &A, const TcOperand &W, int M, int N, int K, bool split3, const LnEpi &epi, int num_sms,
                              cudaStream_t st);

// ------------------------------------------------------------------ gemm_skinny.cu (M <= 128: the streaming path's GEMMs)
size_t gemm_skinny_ws_floats(int max_n, int max_splits);
cudaError_t launch_gemm_skinny(const bf16 *Ahi, const bf16 *Alo, int lda, const bf16 *Whi, const bf16 *Wlo, int M, int N, int K, bool split3,
                               const EpiParams &epi, float *ws, size_t ws_floats, unsigned int *tickets, int n_tickets, int num_sms,
                               cudaStream_t st);

// ------------------------------------------------------------------ norm_conv.cu (K6, K8)
// fp32 -> bf16 hi/lo operand planes (n multiple of 4)
void launch_split(const float *x, size_t n, ActBuf out, cudaStream_t st);
void launch_layernorm(const float *x, int M, int d, const float *w1, const float *b1, float *out1_f32,
                      ActBuf out1_act, const float *w2, const float *b2, ActBuf out2_act, cudaStream_t st);
bool launch_dwconv_bn_silu(const float *g, const int32_t *row_off, int n_utt, int max_T, int d, int ks,
                           const float *w, const float *bias, ActBuf out, cudaStream_t st);

// ------------------------------------------------------------------ attention.cu (K7)
bool launch_relpos_attention(const float *qkv, int ld_qkv, const int32_t *row_off, int n_utt, int max_T,
                             int n_heads, int head_dim, const float *pp, int tmax, const float *bu,
                             const float *bv, int d_model, ActBuf out, cudaStream_t st);

// tensor-core variant (attention_tc.cu, head_dim 64): pp as bf16 hi/lo planes
// From the EPI_QKV_ACT GEMM epilogue: q32 = fp32 q [M, d] (the kernel adds pos_u / pos_v), kv_hi / kv_lo = bf16 planes
// [M, ld_kv = 2 d] = [k | v].
bool launch_relpos_attention_tc(const float *q32, const float *pos_u, const float *pos_v, const bf16 *kv_hi, const bf16 *kv_lo,
                                int ld_kv, const int32_t *row_off, int n_utt, int max_T, int n_heads, int head_dim, const bf16 *pp_hi,
                                const bf16 *pp_lo, int tmax, int d_model, ActBuf out, cudaStream_t st);

// tcgen05 variant (attention_umma.cu): head_dim 64, utterances of <= 128 frames, one CTA per (utterance, head).
// kv = tensor maps of the [M][2 d] k | v planes (box 64 x 128, rows = M exactly); pp = of the [2 tmax - 1][d] planes of
// the projected position table (box 64 x 256).
bool relpos_attention_umma_supported(int head_dim, int max_T);
bool launch_relpos_attention_umma(const float *q32, const float *pos_u, const float *pos_v, const TcOperand &kv, const TcOperand &pp,
                                  const int32_t *row_off, int n_utt, int max_T, int n_heads, int head_dim, int tmax, int d_model, int num_sms, ActBuf out,
                                  cudaStream_t st);
void relpos_attention_umma_set_debug(int on);          // measurement aid (PK_AU_DBG=1): per-item timeline of CTA 0
void relpos_attention_umma_print_timeline(int n_items);

// ContextTrie (src/phrase_boost.cpp:9-66) in CSR form on the device: node 0 = root; the edges of node i are
// [first[i], first[i+1]) = (token, child node), sorted by token.
struct DeviceTrie {
    const int32_t *first = nullptr, *tok = nullptr, *child = nullptr;
    int32_t n_nodes = 0;
};

// ------------------------------------------------------------------ ctc.cu (K9)
void launch_ctc_boosted_decode(const float *logprobs, const int32_t *row_off, int n_utt, int V, int blank, int cap,
                               const DeviceTrie &trie, float boost, int32_t *tok, int32_t *t_start, int32_t *t_end, float *t_conf,
                               cudaStream_t st);
void launch_ctc_frame_argmax(const float *logits, int M, int V, int ld, int32_t *best, float *conf,
                             float *logprobs, cudaStream_t st);
void launch_ctc_collapse(const int32_t *best, const float *conf, const int32_t *row_off, int n_utt, int blank,
                         int cap, int32_t *tok, int32_t *t_start, int32_t *t_end, float *t_conf, cudaStream_t st);

// ------------------------------------------------------------------ tdt.cu (K10)
struct TdtParams {
    int P, J, V, D, L, Bpad, n_utt, cap, max_steps, n_dur;
    // RNNT mode (rnnt_greedy_decode(_with_timestamps), src/rnnt.cpp:56-177; D = 0, no duration head): blank advances one
    // frame, a symbol stays on the frame (start = end = t), and the max_symbols-th symbol on a frame moves to the next
    // frame with the state and token kept.  0 = TDT rule.
    int max_symbols;
    int out_in_smem, wih_in_smem, smem_lstm_floats;   // filled by launch_tdt_decode
    int wstage_rows;                                  // rows of the shared-memory staging tile for weights that stay in L2 (0: none)
    int durations[8];
    const float *EP;                          // [M][J] enc_proj(enc) + bias
    const int32_t *row_off;                   // [n_utt+1]
    const float *G0;                          // [V][4P] W_ih0 . E[token] + b0
    // weights pre-split for the tensor-core products (launch_tdt_split_rows): row = [hi: K][lo: K] bf16
    const bf16 *Whh[PK_MAX_LSTM];             // [P*4] rows, K = P, unit-major: row = unit*4 + gate(i,f,g,o)
    const bf16 *Wih[PK_MAX_LSTM];             // [P*4] rows, K = P, unit-major (layers >= 1)
    const float *bih[PK_MAX_LSTM];            // [4P]    (layers >= 1)
    const bf16 *Wp;                           // [J] rows, K = P
    const bf16 *Wout;                         // [V+D] rows, K = J
    const float *bout;                        // [V+D]
    float *hbuf;                              // bf16 [hi|lo][L][2][Bpad][P] LSTM h (two state planes per utterance), zeroed
    float *z;                                 // bf16 [hi|lo][Bpad][J]       joint hidden
    int32_t *overflow;                        // [Bpad]
    float *pl_max, *pl_sum;                   // [3][grid][Bpad] per-CTA (max, sum-exp) partials
    unsigned long long *key_lab, *key_dur;    // [3][Bpad] packed (value, index) arg-max keys
    unsigned int *bar;                        // grid barrier counter
    long long *dbg;                           // [8] optional: CTA-0 cycles per phase, steps
    int32_t *tok;                             // [n_utt][1+cap]
    int32_t *t_start, *t_end;                 // [n_utt][cap]
    float *t_conf;
    // Carried decode state (rnnt_streaming_decode_chunk, src/eou.cpp:17-98): the LSTM state, the last token and the
    // absolute frame number survive from chunk to chunk.  carry = 1: hbuf plane 0 holds the committed h on entry and on
    // exit, c_state [L][Bpad][P] the committed cell state, tok_state [Bpad] the last emitted token; emitted frames are
    // frame_base[b] + t and the end frame is NOT clamped to the chunk (eou.cpp:81-84); utterances with no frames idle.
    int carry;
    float *c_state;
    int32_t *tok_state;
    const int32_t *frame_base;
    // Phrase boosting (tdt_greedy_decode(_with_timestamps)_boosted, src/phrase_boost.cpp:177-352): boost_on = 1 adds `boost`
    // to the label logits of the tokens that continue an active trie state of the utterance (durations are not boosted);
    // boost_bits [Bpad][(V+31)/32] is the per-utterance bitmap of those tokens, trie_active [Bpad][64] / trie_nact [Bpad] the
    // active states; all three are maintained by the CTA that owns the utterance.  Confidence stays exp(raw log-prob).
    int boost_on;
    float boost;
    DeviceTrie trie;
    uint32_t *boost_bits;
    int32_t *trie_active, *trie_nact;
};
cudaError_t launch_tdt_decode(TdtParams p, int num_sms, cudaStream_t st);
void tdt_pass_profile(long long *out8, bool reset);   // measurement aid: section cycles of cluster_pass (CTA 0), summed since the last reset
// fp32 [rows][K] -> [rows][2 K] bf16 = [hi: K][lo: K]
void launch_tdt_split_rows(const float *src, int rows, int K, bf16 *dst, cudaStream_t st);

}  // namespace pk
