// stream_engine.cu -- the STREAMING path behind the C-ABI (SURVEY.md section 8f row 2, BASELINE configs[3]: eou-120m,
// 160 ms chunks).  Reference call stack being replaced (one stream, one chunk at a time, host round trips throughout):
//   StreamingTranscriber::transcribe_chunk                 src/eou.cpp:111-143
//   StreamingAudioPreprocessor::process_chunk              src/audio.cpp:195-259
//   StreamingFastConformerEncoder::forward_chunk           src/streaming_encoder.cpp:425-472
//     CausalConvSubsampling::forward_cached                :339-385
//     StreamingConformerAttention::forward_cached          :160-272
//     CausalConformerConvModule::forward_cached            :41-80
//   rnnt_streaming_decode_chunk                            src/eou.cpp:17-98
//
// B200 design: the reference advances ONE stream by 1-2 encoder frames per call, which is weight-bandwidth-bound (435 MB of
// fp32 weights per chunk).  Here S streams advance in LOCK STEP: a step takes one chunk of every stream, and all
// streams' frames form one packed row block M = sum_s C_s that runs through the same tcgen05 GEMMs / LayerNorm kernels as
// the offline path (weights are read once per step for all streams).  Per-stream state is resident in HBM: sample
// overlap + pre-emphasis carry, leftover mel frames, per layer a ring of the last att_context_left K / V rows and the
// last k-1 GLU outputs, the LSTM state, the last token and the absolute frame offset.  All lengths depend only on the
// chunk sizes, so the host computes them (StreamPlan) and the kernels never synchronise with it.
#include <algorithm>

#include "engine.h"

struct StreamSet {
    int S = 0, L = 70, R = 1, max_chunk = 0;
    int nf_max = 0, take_max = 0, c_max = 0;
    // host bookkeeping
    std::vector<int32_t> ovl_len, left, cache_len, ring_start, frame_base;
    std::vector<int32_t> act, take, nC;                       // this step: active stream ids, frames taken, encoder frames
    // device state
    StreamState st{};
    float *kc = nullptr, *vc = nullptr;                        // [layers][S][L][d]
    float *convc = nullptr;                                    // [layers][S][k-1][d]
    float *c_state = nullptr;                                  // [lstm][Bpad][P]
    float *hbuf = nullptr;                                     // bf16 planes [hi|lo][lstm][2][Bpad][P]
    int32_t *tok_state = nullptr;
    // per-step device scratch
    float *d_chunk = nullptr, *ssig = nullptr, *mel_in = nullptr;
    StreamPlan *d_plan = nullptr, *h_plan = nullptr;           // h_plan pinned
    int64_t *d_sig_off = nullptr, *h_sig_off = nullptr;
    int32_t *d_meta = nullptr, *h_meta = nullptr;              // nf | out_row | act | cache_len | ring_start | frame_base | row_off_S
    float *h_chunk = nullptr;                                  // pinned staging of the chunk samples
    cudaEvent_t ev_up = nullptr;                               // uploads of the previous step consumed
    size_t state_bytes = 0;
};

namespace {

inline int enc_frames(int mel_frames) { return conv_len(conv_len(conv_len(mel_frames))); }

}  // namespace

// Conformer blocks on the packed chunk rows (streaming_encoder.cpp:430-472): ffn1 -> cached attention -> cached conv ->
// ffn2 -> LayerNorm, the same GEMM / LayerNorm kernels as the offline encoder (engine.cu run_encoder).
pk_status pk_engine::run_stream_layers() {
    StreamSet &s = *ss;
    const pk_config &c = cfg;
    const int d = c.d_model, H = c.n_heads, hd = d / H;
    const int n_act = (int)s.act.size();
    int maxC = 0;
    for (int a = 0; a < n_act; ++a) maxC = std::max(maxC, s.nC[a]);
    const int32_t *d_act = s.d_meta + 2 * s.S, *d_cl = s.d_meta + 3 * s.S, *d_rs = s.d_meta + 4 * s.S;
    ActBuf none;
    auto LN = [&](const float *w1, const float *b1, float *o1, ActBuf a1, const float *w2, const float *b2, ActBuf a2) {
        Scope sc(this, CAT_LAYERNORM);
        launch_layernorm(x, M, d, w1, b1, o1, a1, w2, b2, a2, stream);
        ++launches;
    };
    LN(layers[0].ffn_ln_w[0], layers[0].ffn_ln_b[0], nullptr, ln, nullptr, nullptr, none);
    for (int i = 0; i < c.n_layers; ++i) {
        const LayerW &Lw = layers[i];
        for (int f = 0; f < 2; ++f) {
            if (f == 1) LN(Lw.ffn_ln_w[1], Lw.ffn_ln_b[1], nullptr, ln, nullptr, nullptr, none);
            EpiParams e1;
            e1.kind = EPI_BIAS_SILU_ACT;
            e1.act = ffh;
            e1.ldo = c.ff;
            gemm(ln, d, Lw.fc1[f], M, e1);
            EpiParams e2;
            e2.kind = EPI_RESID_F32;
            e2.out_f32 = x;
            e2.resid = x;
            e2.ldo = d;
            e2.alpha = 0.5f;
            gemm(ffh, c.ff, Lw.fc2[f], M, e2);
            if (f == 1) break;
            // cached attention
            LN(Lw.att_ln_w, Lw.att_ln_b, nullptr, ln, nullptr, nullptr, none);
            EpiParams eq;
            eq.kind = EPI_BIAS_F32;
            eq.out_f32 = qkv;
            eq.ldo = 3 * d;
            gemm(ln, d, Lw.qkv, M, eq);
            {
                Scope sc(this, CAT_ATTENTION);
                const size_t per_layer = (size_t)s.S * s.L * d;
                if (!launch_stream_attention(qkv, 3 * d, d_row_off, d_act, n_act, maxC, d_cl, d_rs, s.kc + (size_t)i * per_layer,
                                             s.vc + (size_t)i * per_layer, s.L, H, hd, d, Lw.pp, Tmax, Lw.pos_u, Lw.pos_v, ctx, stream))
                    return fail(PK_ERR_INVALID, "stream attention: chunk too long for one block's shared memory");
            }
            ++launches;
            EpiParams eo;
            eo.kind = EPI_RESID_F32;
            eo.out_f32 = x;
            eo.resid = x;
            eo.ldo = d;
            eo.alpha = 1.0f;
            gemm(ctx, d, Lw.out, M, eo);
            // cached causal conv module
            LN(Lw.conv_ln_w, Lw.conv_ln_b, nullptr, ln, nullptr, nullptr, none);
            EpiParams eg;
            eg.kind = EPI_GLU_F32;
            eg.out_f32 = glu;
            eg.ldo = d;
            gemm(ln, d, Lw.pw1, M, eg);
            {
                Scope sc(this, CAT_DWCONV);
                if (!launch_stream_dwconv(glu, d_row_off, d_act, n_act, s.convc + (size_t)i * s.S * (c.conv_kernel - 1) * d, d,
                                          c.conv_kernel, Lw.dw_w, Lw.dw_b, cv, stream))
                    return fail(PK_ERR_INVALID, "unsupported conv_kernel");
            }
            ++launches;
            EpiParams ec;
            ec.kind = EPI_RESID_F32;
            ec.out_f32 = x;
            ec.resid = x;
            ec.ldo = d;
            ec.alpha = 1.0f;
            gemm(cv, d, Lw.pw2, M, ec);
        }
        const bool last = (i + 1 == c.n_layers);
        if (!last)
            LN(Lw.fin_ln_w, Lw.fin_ln_b, x, none, layers[i + 1].ffn_ln_w[0], layers[i + 1].ffn_ln_b[0], ln);
        else
            LN(Lw.fin_ln_w, Lw.fin_ln_b, x, cfg.math == PK_MATH_FP32 ? none : ln, nullptr, nullptr, none);
    }
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

// rnnt_streaming_decode_chunk (eou.cpp:17-98) for all streams: the TDT decode kernel with carried state.
pk_status pk_engine::run_stream_decode() {
    StreamSet &s = *ss;
    const pk_config &c = cfg;
    EpiParams ep;
    ep.kind = EPI_BIAS_F32;
    ep.out_f32 = EP;
    ep.ldo = c.joint_hidden;
    Act encop;
    if (cfg.math == PK_MATH_FP32) encop.f32 = x; else encop = ln;
    gemm(encop, c.d_model, enc_proj, M, ep);
    int maxC = 0;
    for (size_t a = 0; a < s.act.size(); ++a) maxC = std::max(maxC, s.nC[a]);
    TdtParams p{};
    p.P = c.pred_hidden; p.J = c.joint_hidden; p.V = c.vocab; p.D = c.n_durations; p.L = c.lstm_layers;
    p.Bpad = Bpad; p.n_utt = s.S; p.cap = cap; p.n_dur = c.n_durations;
    p.max_steps = maxC + cap + 2;
    for (int i = 0; i < 8; ++i) p.durations[i] = c.durations[i];
    p.EP = EP; p.row_off = s.d_meta + 6 * s.S; p.G0 = G0;
    for (int l = 0; l < c.lstm_layers; ++l) { p.Whh[l] = Whh_s[l]; p.Wih[l] = Wih_s[l]; p.bih[l] = bih[l]; }
    p.Wp = Wp_s; p.Wout = Wout_s; p.bout = bout;
    p.hbuf = s.hbuf; p.z = zbuf;
    p.overflow = tdt_ints; p.bar = reinterpret_cast<unsigned int *>(tdt_ints + Bpad);
    p.pl_max = pl_max; p.pl_sum = pl_sum;
    p.key_lab = tdt_keys; p.key_dur = tdt_keys + 3 * (size_t)Bpad;
    p.dbg = reinterpret_cast<long long *>(tdt_keys + 6 * (size_t)Bpad);
    p.tok = tok; p.t_start = t_start; p.t_end = t_end; p.t_conf = t_conf;
    p.carry = 1; p.c_state = s.c_state; p.tok_state = s.tok_state; p.frame_base = s.d_meta + 5 * s.S;
    cudaError_t ce;
    {
        Scope sc(this, CAT_TDT);
        ce = launch_tdt_decode(p, num_sms, stream);
    }
    launches += 2;
    last_tdt = true;
    if (ce != cudaSuccess) return fail(PK_ERR_CUDA, std::string("stream decode launch: ") + cudaGetErrorString(ce));
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

extern "C" {

pk_status pk_stream_open(pk_engine *e, int32_t n_streams, int32_t max_chunk_samples, int32_t att_context_left, int32_t att_context_right) {
    if (!e || n_streams < 1 || max_chunk_samples < 1 || att_context_left < 1) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (e->ss) return e->fail(PK_ERR_INVALID, "pk_stream_open: streams are already open on this engine");
    const pk_config &c = e->cfg;
    if (c.n_durations == 0) return e->fail(PK_ERR_INVALID, "pk_stream_open: streaming is not available on an RNNT engine (n_durations = 0)");
    auto s = std::make_unique<StreamSet>();
    s->S = n_streams; s->L = att_context_left; s->R = att_context_right; s->max_chunk = max_chunk_samples;
    const int tot_max = 399 + max_chunk_samples;
    s->nf_max = tot_max >= 512 ? ((((tot_max - 400) / 160) * 160 + 400) - 512) / 160 + 1 : 0;
    s->take_max = ((7 + s->nf_max) / 8) * 8;
    s->c_max = enc_frames(std::max(s->take_max, 8));
    if (n_streams > e->Bmax) return e->fail(PK_ERR_CAPACITY, "pk_stream_open: more streams than pk_config.max_batch");
    if (s->take_max > e->Fmax || s->L + s->c_max > e->Tmax)
        return e->fail(PK_ERR_CAPACITY, "pk_stream_open: pk_config.max_samples too small (needs encoder frames >= att_context_left + frames per chunk)");
    const int S = n_streams, d = c.d_model, nl = c.n_layers, P = c.pred_hidden, LL = c.lstm_layers;
    s->ovl_len.assign(S, 0); s->left.assign(S, 0); s->cache_len.assign(S, 0); s->ring_start.assign(S, 0); s->frame_base.assign(S, 0);
    s->st.ovl = e->dalloc<float>((size_t)S * STREAM_OVL_CAP);
    s->st.last = e->dalloc<float>(S);
    s->st.melq = e->dalloc<float>((size_t)S * 8 * c.mel_bins);
    s->kc = e->dalloc<float>((size_t)nl * S * s->L * d);
    s->vc = e->dalloc<float>((size_t)nl * S * s->L * d);
    s->convc = e->dalloc<float>((size_t)nl * S * (c.conv_kernel - 1) * d);
    s->c_state = e->dalloc<float>((size_t)LL * e->Bpad * P);
    s->hbuf = e->dalloc<float>((size_t)P * e->Bpad * 2 * LL);
    s->tok_state = e->dalloc<int32_t>(e->Bpad);
    s->d_chunk = e->dalloc<float>((size_t)S * max_chunk_samples + 8);
    s->ssig = e->dalloc<float>((size_t)S * (max_chunk_samples + STREAM_OVL_CAP) + 8);
    s->mel_in = e->dalloc<float>((size_t)S * (8 + s->nf_max) * c.mel_bins);
    s->d_plan = e->dalloc<StreamPlan>(S);
    s->d_sig_off = e->dalloc<int64_t>(S + 1);
    s->d_meta = e->dalloc<int32_t>((size_t)7 * S + 8);
    if (!s->d_meta || !s->d_plan || !s->mel_in || !s->ssig || !s->kc || !s->vc || !s->convc || !s->hbuf)
        return e->fail(PK_ERR_CUDA, "cudaMalloc failed (stream state)");
    if (cudaMallocHost(&s->h_plan, sizeof(StreamPlan) * S) != cudaSuccess || cudaMallocHost(&s->h_sig_off, sizeof(int64_t) * (S + 1)) != cudaSuccess ||
        cudaMallocHost(&s->h_meta, sizeof(int32_t) * (7 * S + 8)) != cudaSuccess ||
        cudaMallocHost(&s->h_chunk, sizeof(float) * ((size_t)S * max_chunk_samples + 8)) != cudaSuccess ||
        cudaEventCreateWithFlags(&s->ev_up, cudaEventDisableTiming) != cudaSuccess)
        return e->fail(PK_ERR_CUDA, "cudaMallocHost failed (stream staging)");
    e->ss = s.release();
    return pk_stream_reset(e, -1);
}

// StreamingTranscriber::reset (eou.cpp:145-149) for one stream (or all: stream = -1)
pk_status pk_stream_reset(pk_engine *e, int32_t stream) {
    if (!e || !e->ss) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    StreamSet &s = *e->ss;
    const pk_config &c = e->cfg;
    if (stream < -1 || stream >= s.S) return e->fail(PK_ERR_INVALID, "pk_stream_reset: bad stream index");
    const int s0 = stream < 0 ? 0 : stream, s1 = stream < 0 ? s.S : stream + 1;
    const int P = c.pred_hidden, Bp = e->Bpad, LL = c.lstm_layers;
    cudaError_t ce = cudaSuccess;
    for (int i = s0; i < s1 && ce == cudaSuccess; ++i) {
        s.ovl_len[i] = s.left[i] = s.cache_len[i] = s.ring_start[i] = s.frame_base[i] = 0;
        ce = cudaMemsetAsync(s.st.last + i, 0, sizeof(float), e->stream);
        // conv caches start as zeros (streaming_encoder.cpp:52-56); K / V rings and mel queues are empty (lengths 0)
        for (int l = 0; l < c.n_layers && ce == cudaSuccess; ++l)
            ce = cudaMemsetAsync(s.convc + ((size_t)l * s.S + i) * (c.conv_kernel - 1) * c.d_model, 0,
                                 sizeof(float) * (c.conv_kernel - 1) * c.d_model, e->stream);
        // LSTM state zero, last token = blank (eou.cpp:22-33)
        for (int l = 0; l < LL && ce == cudaSuccess; ++l) {
            ce = cudaMemsetAsync(s.c_state + ((size_t)l * Bp + i) * P, 0, sizeof(float) * P, e->stream);
            bf16 *hb = reinterpret_cast<bf16 *>(s.hbuf);
            const size_t HS = (size_t)P * Bp, lo = (size_t)LL * 2 * HS;
            for (int pl = 0; pl < 2 && ce == cudaSuccess; ++pl) {
                ce = cudaMemsetAsync(hb + (size_t)(l * 2 + pl) * HS + (size_t)i * P, 0, sizeof(bf16) * P, e->stream);
                if (ce == cudaSuccess) ce = cudaMemsetAsync(hb + lo + (size_t)(l * 2 + pl) * HS + (size_t)i * P, 0, sizeof(bf16) * P, e->stream);
            }
        }
    }
    if (ce == cudaSuccess) {
        std::vector<int32_t> blank(s1 - s0, c.vocab - 1);
        ce = cudaMemcpyAsync(s.tok_state + s0, blank.data(), sizeof(int32_t) * (s1 - s0), cudaMemcpyHostToDevice, e->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    }
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_stream_reset: ") + cudaGetErrorString(ce));
    return PK_OK;
}

// One step = StreamingTranscriber::transcribe_chunk (eou.cpp:111-143) for every stream: stream s receives the samples
// pcm[offsets[s] .. offsets[s+1]) (an empty chunk is allowed).  out rows (n = n_streams) hold the tokens emitted BY THIS
// STEP with absolute frame numbers.  Optional taps (may be NULL): mel_out packed (sum nf_s, mel_bins) = the new log-mel frames
// of this step, n_mel[s] = nf_s; enc_out packed (sum C_s, d_model) = the encoder rows of this step, n_enc[s] = C_s.
pk_status pk_stream_step(pk_engine *e, const float *pcm, const int64_t *offsets, pk_tokens *out, float *mel_out, int32_t *n_mel,
                         float *enc_out, int32_t *n_enc) {
    if (!e || !e->ss || !offsets || (!pcm && offsets[e->ss->S] > offsets[0])) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    StreamSet &s = *e->ss;
    const pk_config &c = e->cfg;
    const int S = s.S;
    cudaEventSynchronize(s.ev_up);                 // the previous step has consumed the pinned staging buffers
    // ---- the plan: pure integer bookkeeping (audio.cpp:216-240, streaming_encoder.cpp:348-385, :185-208)
    int64_t coff = 0, soff = 0;
    int moff = 0, foff = 0, max_nf = 0;
    s.act.clear(); s.take.clear(); s.nC.clear();
    int32_t *m_nf = s.h_meta, *m_row = s.h_meta + S, *m_act = s.h_meta + 2 * S, *m_cl = s.h_meta + 3 * S, *m_rs = s.h_meta + 4 * S,
            *m_fb = s.h_meta + 5 * S, *m_ro = s.h_meta + 6 * S;
    m_ro[0] = 0;
    std::vector<int32_t> new_ovl(S), new_left(S);
    for (int i = 0; i < S; ++i) {
        const int64_t n64 = offsets[i + 1] - offsets[i];
        if (n64 < 0 || n64 > s.max_chunk) return e->fail(PK_ERR_CAPACITY, "pk_stream_step: chunk longer than max_chunk_samples");
        const int n = (int)n64, total = s.ovl_len[i] + n;
        StreamPlan &p = s.h_plan[i];
        p.chunk_off = coff; p.sig_off = soff; p.chunk_len = n; p.ovl_len = s.ovl_len[i];
        p.left = s.left[i]; p.min_off = moff;
        if (total < 400) {                         // audio.cpp:225-229: keep everything
            p.consumed = 0; p.nf = 0;
        } else {
            const int nfh = (total - 400) / 160 + 1;
            p.consumed = (nfh - 1) * 160 + 400;
            // fft::stft(center = false) is called with n_fft = 512 on `consumed` samples: the reference throws below 512
            // (fft.cpp:1516-1521) and otherwise returns (consumed - 512) / 160 + 1 frames -- one fewer than nfh (DESIGN.md)
            if (p.consumed < 512) return e->fail(PK_ERR_INVALID, "pk_stream_step: stft: signal length is less than n_fft (the reference throws here: first chunk of 400..511 samples)");
            p.nf = (p.consumed - 512) / 160 + 1;
        }
        new_ovl[i] = total - p.consumed;
        const int frames = p.left + p.nf;
        p.take = (frames / 8) * 8;
        new_left[i] = frames - p.take;
        p.feat_off = foff;
        m_nf[i] = p.nf; m_row[i] = p.min_off + p.left; m_cl[i] = s.cache_len[i]; m_rs[i] = s.ring_start[i]; m_fb[i] = s.frame_base[i];
        int C = 0;
        if (p.take > 0) {
            C = enc_frames(p.take);
            s.act.push_back(i); s.take.push_back(p.take); s.nC.push_back(C);
            foff += p.take;
        }
        m_ro[i + 1] = m_ro[i] + C;
        s.h_sig_off[i] = soff;
        if (n > 0) memcpy(s.h_chunk + coff, pcm + offsets[i], sizeof(float) * n);
        coff += n; soff += total; moff += frames;
        max_nf = std::max(max_nf, p.nf);
    }
    s.h_sig_off[S] = soff;
    const int n_act = (int)s.act.size();
    for (int a = 0; a < n_act; ++a) m_act[a] = s.act[a];
    cudaStream_t st = e->stream;
    cudaError_t ce = cudaMemcpyAsync(s.d_plan, s.h_plan, sizeof(StreamPlan) * S, cudaMemcpyHostToDevice, st);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(s.d_sig_off, s.h_sig_off, sizeof(int64_t) * (S + 1), cudaMemcpyHostToDevice, st);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(s.d_meta, s.h_meta, sizeof(int32_t) * (7 * S + 1), cudaMemcpyHostToDevice, st);
    if (ce == cudaSuccess && coff > 0) ce = cudaMemcpyAsync(s.d_chunk, s.h_chunk, sizeof(float) * coff, cudaMemcpyHostToDevice, st);
    if (ce == cudaSuccess) ce = cudaEventRecord(s.ev_up, st);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_stream_step upload: ") + cudaGetErrorString(ce));
    // ---- front end
    launch_stream_prep(s.d_chunk, s.d_plan, s.st, S, s.ssig, s.mel_in, c.mel_bins, st);
    {
        pk_engine::Scope sc(e, pk_engine::CAT_MEL);
        launch_mel_stream(s.ssig, s.d_sig_off, s.d_meta, s.d_meta + S, S, max_nf, c.mel_bins, e->mel_tb, s.mel_in, st);
    }
    launch_stream_post(s.d_chunk, s.d_plan, s.st, S, s.ssig, s.mel_in, c.mel_bins, e->feats, st);
    e->launches += 3;
    if (mel_out) {      // debug tap: the new frames of every stream, packed
        size_t o = 0;
        for (int i = 0; i < S && ce == cudaSuccess; ++i) {
            const StreamPlan &p = s.h_plan[i];
            if (p.nf > 0)
                ce = cudaMemcpyAsync(mel_out + o, s.mel_in + (size_t)(p.min_off + p.left) * c.mel_bins, sizeof(float) * p.nf * c.mel_bins,
                                     cudaMemcpyDeviceToHost, st);
            o += (size_t)p.nf * c.mel_bins;
        }
    }
    if (n_mel) for (int i = 0; i < S; ++i) n_mel[i] = s.h_plan[i].nf;
    if (n_enc) for (int i = 0; i < S; ++i) n_enc[i] = m_ro[i + 1] - m_ro[i];
    // ---- host state of the next step
    for (int i = 0; i < S; ++i) {
        s.ovl_len[i] = new_ovl[i];
        s.left[i] = new_left[i];
        const int C = m_ro[i + 1] - m_ro[i], kv = s.cache_len[i] + C;
        if (kv > s.L) s.ring_start[i] = (s.ring_start[i] + kv - s.L) % s.L;
        s.cache_len[i] = std::min(kv, s.L);
        s.frame_base[i] += C;
    }
    pk_status ps = PK_OK;
    if (n_act > 0) {
        // the active streams' frames as an ordinary packed batch (CausalConvSubsampling runs the plain zero-padded subsampling)
        if ((ps = e->set_batch_shapes(s.take.data(), nullptr, n_act))) return ps;
        if ((ps = e->upload_shapes())) return ps;
        auto body = [e, enc_out, st]() -> pk_status {
            pk_status q;
            if ((q = e->run_conv1())) return q;
            if ((q = e->run_subsample_tail())) return q;
            if ((q = e->run_stream_layers())) return q;
            if (enc_out) {
                cudaError_t c2 = cudaMemcpyAsync(enc_out, e->x, sizeof(float) * (size_t)e->M * e->cfg.d_model, cudaMemcpyDeviceToHost, st);
                if (c2 != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_stream_step tap: ") + cudaGetErrorString(c2));
            }
            return e->run_stream_decode();
        };
        if (enc_out) {
            ps = body();                       // (debug taps: plain launches)
        } else {
            // every kernel argument of the step depends only on which streams take how many frames: one graph per pattern
            std::string key(1, 's');
            key.append(reinterpret_cast<const char *>(s.act.data()), s.act.size() * sizeof(int32_t));
            key.append(reinterpret_cast<const char *>(s.take.data()), s.take.size() * sizeof(int32_t));
            ps = e->run_graphed(key, body);
        }
        if (ps) return ps;
        if (e->gemm_err) return e->gemm_err;
    }
    if (!out) return PK_OK;
    if (n_act == 0) {
        for (int i = 0; i < S; ++i) out->len[i] = 0;
        ce = cudaStreamSynchronize(st);
        return ce == cudaSuccess ? PK_OK : e->fail(PK_ERR_CUDA, std::string("pk_stream_step: ") + cudaGetErrorString(ce));
    }
    e->n_utt = S;                                   // the token rows cover all streams
    return e->fetch(out);
}

int32_t pk_stream_count(const pk_engine *e) { return (e && e->ss) ? e->ss->S : 0; }

}  // extern "C"

void pk_stream_free(pk_engine *e) {
    if (!e || !e->ss) return;
    StreamSet *s = e->ss;
    if (s->h_plan) cudaFreeHost(s->h_plan);
    if (s->h_sig_off) cudaFreeHost(s->h_sig_off);
    if (s->h_meta) cudaFreeHost(s->h_meta);
    if (s->h_chunk) cudaFreeHost(s->h_chunk);
    if (s->ev_up) cudaEventDestroy(s->ev_up);
    delete s;
    e->ss = nullptr;
}
