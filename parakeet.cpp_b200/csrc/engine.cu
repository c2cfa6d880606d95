// engine.cu -- the engine behind the C-ABI (include/parakeet_b200.h): weight loading and
// layout, workspace, and the orchestration of the sm_100a kernels for
//     PCM -> log-mel -> FastConformer encoder -> CTC / TDT greedy decode.
//
// Reference call stack being replaced (SURVEY.md section 3.2/3.3):
//   Transcriber::Transcriber / to_gpu        include/parakeet/transcribe.hpp:59-71
//   Transcriber::transcribe                  include/parakeet/transcribe.hpp:99-179
//   preprocess_audio                         src/audio.cpp:100-158
//   FastConformerEncoder::forward            src/encoder.cpp:253-271 (and :9-241)
//   CTCDecoder::forward + ctc_greedy_decode  src/ctc.cpp:12-127
//   tdt_greedy_decode(_with_timestamps)      src/tdt.cpp:36-201
//
// Data layout in HBM: utterances are PACKED, not padded: a batch is one row-major matrix
// whose rows are (utterance, time[, freq]) and per-utterance prefix offsets say where each
// utterance starts.  GEMMs run over all rows at once; length-aware kernels (convolutions,
// attention, decode) use the offsets, so every utterance sees exactly the zero padding /
// sequence end the batch-1 reference gives it.
#include "engine.h"

namespace pk_detail {
std::string &create_err() {
    thread_local std::string s;
    return s;
}
}  // namespace pk_detail
#define g_create_err (create_err())

// ===================================================================== weights

pk_status pk_engine::get_vec(const SafeTensors &st, const std::string &name, int n, float **out) {
    std::vector<float> h;
    std::string e;
    if (!st.read_f32(name, h, n, e)) return fail(PK_ERR_MISSING, e);
    *out = upload(h);
    return *out ? PK_OK : fail(PK_ERR_CUDA, "cudaMalloc failed for " + name);
}

pk_status pk_engine::finish_weight(std::vector<float> &w, std::vector<float> *b, int N, int K, GemmWeight &out) {
    out.N = N;
    out.K = K;
    out.w = upload(w);
    if (!out.w) return fail(PK_ERR_CUDA, "cudaMalloc failed (weight)");
    if (b) {
        out.bias = upload(*b);
        if (!out.bias) return fail(PK_ERR_CUDA, "cudaMalloc failed (bias)");
    }
    if (cfg.math != PK_MATH_FP32) {
        std::vector<bf16> hi(w.size()), lo(w.size());
        for (size_t i = 0; i < w.size(); ++i) {
            hi[i] = __float2bfloat16_rn(w[i]);
            lo[i] = __float2bfloat16_rn(w[i] - __bfloat162float(hi[i]));
        }
        out.hi = upload(hi);
        out.lo = upload(lo);
        if (!out.hi || !out.lo) return fail(PK_ERR_CUDA, "cudaMalloc failed (split weight)");
        if (K % 64 != 0) return fail(PK_ERR_INVALID, "tcgen05 GEMM needs K % 64 == 0");
        if (!make_tc_operand(&out.tc, out.hi, out.lo, N, K, tc_tile_n(N)))
            return fail(PK_ERR_CUDA, "cuTensorMapEncodeTiled failed for a weight");
    }
    return PK_OK;
}

pk_status pk_engine::make_weight(const SafeTensors &st, const std::string &wname, const std::string &bname, int N,
                                 int K, GemmWeight &out, const std::vector<int> *row_perm,
                                 const std::vector<int> *col_perm) {
    std::vector<float> w, b;
    std::string e;
    if (!st.read_f32(wname, w, (int64_t)N * K, e)) return fail(PK_ERR_MISSING, e);
    if (!bname.empty() && !st.read_f32(bname, b, N, e)) return fail(PK_ERR_MISSING, e);
    if (row_perm || col_perm) {
        std::vector<float> w2(w.size()), b2(b.size());
        for (int n = 0; n < N; ++n) {
            const int sn = row_perm ? (*row_perm)[n] : n;
            for (int k = 0; k < K; ++k) {
                const int sk = col_perm ? (*col_perm)[k] : k;
                w2[(size_t)n * K + k] = w[(size_t)sn * K + sk];
            }
            if (!b.empty()) b2[n] = b[sn];
        }
        w.swap(w2);
        if (!b.empty()) b.swap(b2);
    }
    return finish_weight(w, bname.empty() ? nullptr : &b, N, K, out);
}

pk_status pk_engine::load(const char *path) {
    SafeTensors st;
    std::string e;
    if (!st.open(path, e)) return fail(PK_ERR_IO, e);
    const pk_config &c = cfg;
    const int C = c.sub_channels, d = c.d_model, ff = c.ff, H = c.n_heads, hd = d / H;
    pk_status s;

    // ---- mel tables (host, double precision where the reference uses it)
    {
        std::vector<float> win(400);
        for (int i = 0; i < 400; ++i) win[i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * i / 399.0));  // fft.cpp:1117-1142
        std::vector<float2> tw256(256), tw512(257);
        for (int m = 0; m < 256; ++m) tw256[m] = make_float2((float)std::cos(2.0 * M_PI * m / 256.0), (float)-std::sin(2.0 * M_PI * m / 256.0));
        for (int k = 0; k <= 256; ++k) tw512[k] = make_float2((float)std::cos(2.0 * M_PI * k / 512.0), (float)-std::sin(2.0 * M_PI * k / 512.0));
        // Slaney filterbank, audio.cpp:18-94
        auto hz2mel = [](double f) { return f < 1000.0 ? f / (200.0 / 3.0) : 15.0 + std::log(f / 1000.0) / 0.06875177742094912; };
        auto mel2hz = [](double m) { return m < 15.0 ? m * (200.0 / 3.0) : 1000.0 * std::exp((m - 15.0) * 0.06875177742094912); };
        const int nm = c.mel_bins, nf = 257;
        const double mmin = hz2mel(0.0), mmax = hz2mel(8000.0);
        std::vector<double> hz(nm + 2);
        for (int i = 0; i < nm + 2; ++i) hz[i] = mel2hz(mmin + (double)i * (mmax - mmin) / (double)(nm + 1));
        std::vector<float> fbw;
        std::vector<int32_t> fstart(nm), flen(nm), foff(nm);
        for (int m = 0; m < nm; ++m) {
            const double left = hz[m], center = hz[m + 1], right = hz[m + 2], enorm = 2.0 / (right - left);
            int first = -1, last = -1;
            std::vector<float> col(nf);
            for (int f = 0; f < nf; ++f) {
                const double fr = (double)f * 16000.0 / (2.0 * (nf - 1));
                double v = 0.0;
                if (fr >= left && fr <= center && center > left) v = (fr - left) / (center - left);
                else if (fr > center && fr <= right && right > center) v = (right - fr) / (right - center);
                col[f] = (float)(v * enorm);
                if (col[f] != 0.f) {
                    if (first < 0) first = f;
                    last = f;
                }
            }
            fstart[m] = first < 0 ? 0 : first;
            flen[m] = first < 0 ? 0 : last - first + 1;
            foff[m] = (int32_t)fbw.size();
            for (int f = fstart[m]; f < fstart[m] + flen[m]; ++f) fbw.push_back(col[f]);
        }
        mel_tb.window = upload(win);
        mel_tb.tw256 = upload(tw256);
        mel_tb.tw512 = upload(tw512);
        mel_tb.fb_w = upload(fbw);
        mel_tb.fb_start = upload(fstart);
        mel_tb.fb_len = upload(flen);
        mel_tb.fb_off = upload(foff);
        mel_tb.fb_nnz = (int)fbw.size();
    }

    // ---- subsampling (encoder.cpp:208-241)
    const std::string sp = "encoder_.subsampling_.";
    if ((s = get_vec(st, sp + "conv1_.weight", C * 9, &c1_w))) return s;
    if ((s = get_vec(st, sp + "conv1_.bias", C, &c1_b))) return s;
    if ((s = get_vec(st, sp + "dw1_.weight", C * 9, &dw1_w))) return s;
    if ((s = get_vec(st, sp + "dw1_.bias", C, &dw1_b))) return s;
    if ((s = get_vec(st, sp + "dw2_.weight", C * 9, &dw2_w))) return s;
    {
        std::vector<float> w, wt((size_t)C * 9);
        if (!st.read_f32(sp + "dw2_.weight", w, (int64_t)C * 9, e)) return fail(PK_ERR_MISSING, e);
        for (int ch = 0; ch < C; ++ch)
            for (int k = 0; k < 9; ++k) wt[(size_t)k * C + ch] = w[(size_t)ch * 9 + k];
        dw2_wt = upload(wt);
    }
    if ((s = get_vec(st, sp + "dw2_.bias", C, &dw2_b))) return s;
    if ((s = make_weight(st, sp + "conv2_.weight", sp + "conv2_.bias", C, C, conv2))) return s;
    if ((s = make_weight(st, sp + "conv3_.weight", sp + "conv3_.bias", C, C, conv3))) return s;
    {
        // reference flattens (C, F') channel-major (encoder.cpp:236-238): k_ref = c*F' + f.
        // Our rows are (f, c): k = f*C + c.
        std::vector<int> colp((size_t)C * f3n);
        for (int f = 0; f < f3n; ++f)
            for (int ch = 0; ch < C; ++ch) colp[(size_t)f * C + ch] = ch * f3n + f;
        if ((s = make_weight(st, sp + "proj_.weight", sp + "proj_.bias", d, C * f3n, proj, nullptr, &colp))) return s;
    }

    // ---- relative position table input: emb(p) for p = -(Tmax-1) .. Tmax-1, fp32 math as
    // encoder.cpp:9-30 (row index here = p + Tmax - 1)
    const int NP = 2 * Tmax - 1;
    std::vector<float> emb((size_t)NP * d);
    for (int r = 0; r < NP; ++r) {
        const float position = (float)(r - (Tmax - 1));
        for (int i = 0; i < d; i += 2) {
            const float div_term = std::exp((float)i * (-std::log(10000.0f) / d));
            emb[(size_t)r * d + i] = std::sin(position * div_term);
            if (i + 1 < d) emb[(size_t)r * d + i + 1] = std::cos(position * div_term);
        }
    }
    float *d_emb = upload(emb);
    if (!d_emb) return fail(PK_ERR_CUDA, "cudaMalloc failed (pos emb)");

    layers.resize(c.n_layers);
    for (int i = 0; i < c.n_layers; ++i) {
        LayerW &L = layers[i];
        const std::string lp = "encoder_.layers_." + std::to_string(i) + ".";
        for (int f = 0; f < 2; ++f) {
            const std::string fp = lp + (f == 0 ? "ffn1_." : "ffn2_.");
            if ((s = get_vec(st, fp + "norm_.weight", d, &L.ffn_ln_w[f]))) return s;
            if ((s = get_vec(st, fp + "norm_.bias", d, &L.ffn_ln_b[f]))) return s;
            if ((s = make_weight(st, fp + "fc1_.weight", fp + "fc1_.bias", ff, d, L.fc1[f]))) return s;
            if ((s = make_weight(st, fp + "fc2_.weight", fp + "fc2_.bias", d, ff, L.fc2[f]))) return s;
        }
        const std::string ap = lp + "attn_.";
        if ((s = get_vec(st, ap + "norm_.weight", d, &L.att_ln_w))) return s;
        if ((s = get_vec(st, ap + "norm_.bias", d, &L.att_ln_b))) return s;
        {
            std::vector<float> w((size_t)3 * d * d), b((size_t)3 * d), t;
            const char *names[3] = {"q_proj", "k_proj", "v_proj"};
            for (int q = 0; q < 3; ++q) {
                if (!st.read_f32(ap + "mha_." + names[q] + ".weight", t, (int64_t)d * d, e)) return fail(PK_ERR_MISSING, e);
                memcpy(&w[(size_t)q * d * d], t.data(), t.size() * 4);
                if (!st.read_f32(ap + "mha_." + names[q] + ".bias", t, d, e)) return fail(PK_ERR_MISSING, e);
                memcpy(&b[(size_t)q * d], t.data(), t.size() * 4);
            }
            if ((s = finish_weight(w, &b, 3 * d, d, L.qkv))) return s;
        }
        if ((s = make_weight(st, ap + "mha_.out_proj.weight", ap + "mha_.out_proj.bias", d, d, L.out))) return s;
        if ((s = get_vec(st, ap + "pos_bias_u_", H * hd, &L.pos_u))) return s;
        if ((s = get_vec(st, ap + "pos_bias_v_", H * hd, &L.pos_v))) return s;
        {
            // PP = emb . Wpos^T (pos_proj_ has no bias, encoder.cpp:80), exact fp32 GEMM
            float *wpos;
            if ((s = get_vec(st, ap + "pos_proj_.weight", d * d, &wpos))) return s;
            L.pp = dalloc<float>((size_t)NP * d);
            if (!L.pp) return fail(PK_ERR_CUDA, "cudaMalloc failed (pp)");
            EpiParams ep;
            ep.kind = EPI_BIAS_F32;
            ep.out_f32 = L.pp;
            ep.ldo = d;
            launch_gemm_simt(d_emb, d, wpos, d, NP, d, d, ep, stream);
            ++launches;
            if (cfg.math != PK_MATH_FP32 && (hd == 64 || hd == 128)) {
                L.pp_hi = dalloc<bf16>((size_t)NP * d);
                L.pp_lo = dalloc<bf16>((size_t)NP * d);
                if (!L.pp_hi || !L.pp_lo) return fail(PK_ERR_CUDA, "cudaMalloc failed (pp planes)");
                ActBuf sp;
                sp.hi = L.pp_hi;
                sp.lo = L.pp_lo;
                launch_split(L.pp, (size_t)NP * d, sp, stream);
                ++launches;
                L.pp_tc_ok = hd == 64 && make_tc_operand(&L.pp_tc, L.pp_hi, L.pp_lo, (uint64_t)NP, (uint64_t)d, 256);
            }
        }
        const std::string cp = lp + "conv_.";
        if ((s = get_vec(st, cp + "norm_.weight", d, &L.conv_ln_w))) return s;
        if ((s = get_vec(st, cp + "norm_.bias", d, &L.conv_ln_b))) return s;
        {
            // GLU pairs channel j with j+d (operations.cpp:1450-1476): interleave the rows so
            // the pair sits in adjacent GEMM columns.
            std::vector<int> rowp((size_t)2 * d);
            for (int j = 0; j < d; ++j) {
                rowp[2 * j] = j;
                rowp[2 * j + 1] = d + j;
            }
            if ((s = make_weight(st, cp + "pointwise_conv1_.weight", cp + "pointwise_conv1_.bias", 2 * d, d, L.pw1, &rowp))) return s;
        }
        if ((s = make_weight(st, cp + "pointwise_conv2_.weight", cp + "pointwise_conv2_.bias", d, d, L.pw2))) return s;
        {
            // fold BatchNorm1d(eval) (normalization.cpp:48-104, eps 1e-5) into the depthwise conv
            const int ks = c.conv_kernel;
            std::vector<float> w, b, g, be, mu, var;
            if (!st.read_f32(cp + "depthwise_conv_.weight", w, (int64_t)d * ks, e)) return fail(PK_ERR_MISSING, e);
            if (!st.read_f32(cp + "depthwise_conv_.bias", b, d, e)) return fail(PK_ERR_MISSING, e);
            if (!st.read_f32(cp + "batch_norm_.weight", g, d, e)) return fail(PK_ERR_MISSING, e);
            if (!st.read_f32(cp + "batch_norm_.bias", be, d, e)) return fail(PK_ERR_MISSING, e);
            if (!st.read_f32(cp + "batch_norm_.running_mean", mu, d, e)) return fail(PK_ERR_MISSING, e);
            if (!st.read_f32(cp + "batch_norm_.running_var", var, d, e)) return fail(PK_ERR_MISSING, e);
            for (int ch = 0; ch < d; ++ch) {
                const double sc = (double)g[ch] / std::sqrt((double)var[ch] + 1e-5);
                for (int j = 0; j < ks; ++j) w[(size_t)ch * ks + j] = (float)((double)w[(size_t)ch * ks + j] * sc);
                b[ch] = (float)(((double)b[ch] - (double)mu[ch]) * sc + (double)be[ch]);
            }
            L.dw_w = upload(w);
            std::vector<float> wt((size_t)d * ks);
            for (int ch = 0; ch < d; ++ch)
                for (int j = 0; j < ks; ++j) wt[(size_t)j * d + ch] = w[(size_t)ch * ks + j];
            L.dw_wt = upload(wt);
            L.dw_b = upload(b);
        }
        if ((s = get_vec(st, lp + "final_norm_.weight", d, &L.fin_ln_w))) return s;
        if ((s = get_vec(st, lp + "final_norm_.bias", d, &L.fin_ln_b))) return s;
    }

    // ---- heads
    const int V = c.vocab, P = c.pred_hidden, J = c.joint_hidden, D = c.n_durations;
    if (c.has_ctc) {
        if ((s = make_weight(st, "ctc_decoder_.proj_.weight", "ctc_decoder_.proj_.bias", V, d, ctc_head))) return s;
    }
    const std::string jp = c.joint_prefix_tdt ? "tdt_joint_." : "joint_.";
    if ((s = make_weight(st, jp + "enc_proj_.weight", jp + "enc_proj_.bias", J, d, enc_proj))) return s;
    if ((s = get_vec(st, jp + "pred_proj_.weight", J * P, &Wp))) return s;
    if (D == 0) {   // RNNTJoint (rnnt.cpp:34-45): one output head of V rows
        if ((s = get_vec(st, jp + "out_proj_.weight", V * J, &Wout))) return s;
        if ((s = get_vec(st, jp + "out_proj_.bias", V, &bout))) return s;
    } else {
        std::vector<float> w((size_t)(V + D) * J), b((size_t)V + D), t;
        if (!st.read_f32(jp + "label_proj_.weight", t, (int64_t)V * J, e)) return fail(PK_ERR_MISSING, e);
        memcpy(w.data(), t.data(), t.size() * 4);
        if (!st.read_f32(jp + "duration_proj_.weight", t, (int64_t)D * J, e)) return fail(PK_ERR_MISSING, e);
        memcpy(&w[(size_t)V * J], t.data(), t.size() * 4);
        if (!st.read_f32(jp + "label_proj_.bias", t, V, e)) return fail(PK_ERR_MISSING, e);
        memcpy(b.data(), t.data(), t.size() * 4);
        if (!st.read_f32(jp + "duration_proj_.bias", t, D, e)) return fail(PK_ERR_MISSING, e);
        memcpy(&b[V], t.data(), t.size() * 4);
        Wout = upload(w);
        bout = upload(b);
    }
    {
        float *embed, *wih0, *b0;
        if ((s = get_vec(st, "prediction_.embed_.weight", V * P, &embed))) return s;
        for (int l = 0; l < c.lstm_layers; ++l) {
            const std::string q = "prediction_.lstm_.cells_." + std::to_string(l) + ".";
            if ((s = get_vec(st, q + "hidden_proj_.weight", 4 * P * P, &Whh[l]))) return s;
            if ((s = get_vec(st, q + "input_proj_.weight", 4 * P * P, &Wih[l]))) return s;
            // unit-major copies for the decode kernel (row = unit*4 + gate; gate order i,f,g,o of lstm.cpp:20-24)
            {
                std::vector<float> src, dst((size_t)4 * P * P);
                for (int which = 0; which < 2; ++which) {
                    if (!st.read_f32(q + (which ? "input_proj_.weight" : "hidden_proj_.weight"), src, (int64_t)4 * P * P, e)) return fail(PK_ERR_MISSING, e);
                    for (int u = 0; u < P; ++u)
                        for (int gt = 0; gt < 4; ++gt)
                            memcpy(&dst[((size_t)u * 4 + gt) * P], &src[((size_t)gt * P + u) * P], (size_t)P * sizeof(float));
                    float *d = upload(dst);
                    if (!d) return fail(PK_ERR_CUDA, "cudaMalloc failed (LSTM weights)");
                    (which ? Wih_um[l] : Whh_um[l]) = d;
                }
            }
            if ((s = get_vec(st, q + "input_proj_.bias", 4 * P, &bih[l]))) return s;
        }
        wih0 = Wih[0];
        b0 = bih[0];
        // G0[token] = W_ih0 . E[token] + b0 (lstm.cpp:17 first term, rnnt.cpp:24)
        G0 = dalloc<float>((size_t)V * 4 * P);
        if (!G0) return fail(PK_ERR_CUDA, "cudaMalloc failed (G0)");
        EpiParams ep;
        ep.kind = EPI_BIAS_F32;
        ep.bias = b0;
        ep.out_f32 = G0;
        ep.ldo = 4 * P;
        launch_gemm_simt(embed, P, wih0, P, V, 4 * P, P, ep, stream);
        ++launches;
    }
    {   // decode-kernel weights, split once into bf16 hi/lo rows
        auto split = [&](const float *src, int rows, int K, bf16 **out) {
            *out = dalloc<bf16>((size_t)rows * 2 * (K + 4));
            if (*out) launch_tdt_split_rows(src, rows, K, *out, stream);
            ++launches;
            return *out != nullptr;
        };
        bool ok = split(Wp, J, P, &Wp_s) && split(Wout, V + D, J, &Wout_s);
        for (int l = 0; l < c.lstm_layers && ok; ++l)
            ok = split(Whh_um[l], 4 * P, P, &Whh_s[l]) && split(Wih_um[l], 4 * P, P, &Wih_s[l]);
        if (!ok) return fail(PK_ERR_CUDA, "cudaMalloc failed (TDT split weights)");
    }
    PK_CUDA(cudaStreamSynchronize(stream));
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

// ===================================================================== workspace

pk_status pk_engine::alloc_workspace() {
    const pk_config &c = cfg;
    const int C = c.sub_channels, d = c.d_model;
    const size_t B = Bmax;
    const int t1 = conv_len(Fmax), t2 = conv_len(t1);
    const size_t rows2 = B * t2 * f2n, rows3 = B * (size_t)Tmax * f3n, Mx = B * (size_t)Tmax;
    d_pcm = dalloc<float>(B * (size_t)c.max_samples + 8);
    d_pcm_alt = dalloc<float>(B * (size_t)c.max_samples + 8);
    d_pcm_off = dalloc<int64_t>(B + 1);
    d_frame_off = dalloc<int32_t>(B + 1);
    d_s2_off = dalloc<int32_t>(B + 1);
    d_row_off = dalloc<int32_t>(B + 1);
    d_t2_rows = dalloc<int32_t>(B + 1);
    logmel = dalloc<float>(B * (size_t)Fmax * c.mel_bins);
    mel_part = dalloc<float>(mel_part_floats((int)B, c.mel_bins));
    feats = dalloc<float>(B * (size_t)Fmax * c.mel_bins);
    sub1 = act_alloc(rows2, C);
    sub2 = dalloc<float>(rows2 * C);
    sub3 = act_alloc(rows3, C);
    sub4 = act_alloc(rows3, C);
    if (cfg.math != PK_MATH_FP32 && sub4.hi && (!make_tc_operand(&sub4.tc, sub4.hi, sub4.lo, Mx, (size_t)C * f3n, 128) || !make_tc_operand(&sub4.tc32, sub4.hi, sub4.lo, Mx, (size_t)C * f3n, 32))) sub4.hi = nullptr;   // viewed as [M][C*F'] by proj_
    x = dalloc<float>(Mx * d);
    ln = act_alloc(Mx, d);
    ffh = act_alloc(Mx, c.ff);
    qkv = dalloc<float>(Mx * 3 * d);
    if (cfg.math != PK_MATH_FP32 && (c.d_model / c.n_heads == 64 || c.d_model / c.n_heads == 128)) {
        qkvp_hi = dalloc<bf16>(Mx * 2 * d);
        qkvp_lo = dalloc<bf16>(Mx * 2 * d);
        if (!qkvp_hi || !qkvp_lo) return fail(PK_ERR_CUDA, "cudaMalloc failed (qkv planes)");
    }
    ctx = act_alloc(Mx, d);
    glu = dalloc<float>(Mx * d);
    cv = act_alloc(Mx, d);
    const int ldv = (c.vocab + 3) & ~3;
    logits = dalloc<float>(Mx * ldv);
    EP = dalloc<float>(Mx * c.joint_hidden);
    best = dalloc<int32_t>(Mx);
    bconf = dalloc<float>(Mx);
    tok = dalloc<int32_t>(B * (1 + (size_t)cap));
    t_start = dalloc<int32_t>(B * (size_t)cap);
    t_end = dalloc<int32_t>(B * (size_t)cap);
    t_conf = dalloc<float>(B * (size_t)cap);
    Bpad = ((Bmax + 31) / 32) * 32;
    const size_t HS = (size_t)c.pred_hidden * Bpad;
    hbuf = dalloc<float>(HS * 2 * c.lstm_layers);                  // bf16 hi + lo planes
    zbuf = dalloc<float>((size_t)c.joint_hidden * Bpad);           // bf16 hi + lo planes
    tdt_ints = dalloc<int32_t>((size_t)Bpad + 512);               // overflow flags | grid-barrier counters (8 lines)
    tdt_keys = dalloc<unsigned long long>((size_t)6 * Bpad + 8);
    const size_t PG = (size_t)3 * num_sms * Bpad;
    pl_max = dalloc<float>(PG);
    pl_sum = dalloc<float>(PG);
    skinny_ws_floats = (size_t)2 << 20;                                       // 8 MB: >= (2 SMs' worth of CTAs) x 128 x 32 fp32 tiles
    skinny_ws = dalloc<float>(skinny_ws_floats);
    skinny_tickets = dalloc<unsigned int>(SKINNY_TICKETS);
    if (skinny_tickets) cudaMemsetAsync(skinny_tickets, 0, SKINNY_TICKETS * sizeof(unsigned int), stream);
    if (!pl_sum || !tdt_keys || !hbuf || !x || !sub2 || !d_pcm || !t_conf || !skinny_ws || !skinny_tickets || !mel_part) return fail(PK_ERR_CUDA, "cudaMalloc failed (workspace)");
    if (cfg.math != PK_MATH_FP32 && (!sub1.hi || !sub3.hi || !sub4.hi || !ln.hi || !ffh.hi || !ctx.hi || !cv.hi))
        return fail(PK_ERR_CUDA, "workspace: cudaMalloc or cuTensorMapEncodeTiled failed for an activation operand");
    PK_CUDA(cudaMallocHost(&h_pcm, (B * (size_t)c.max_samples + 8) * sizeof(float)));
    PK_CUDA(cudaMallocHost(&h_meta, (size_t)(8 * (B + 1)) * sizeof(int32_t)));
    PK_CUDA(cudaMallocHost(&h_tok, B * (1 + (size_t)cap) * sizeof(int32_t)));
    PK_CUDA(cudaMallocHost(&h_ts, B * (size_t)cap * sizeof(int32_t)));
    PK_CUDA(cudaMallocHost(&h_te, B * (size_t)cap * sizeof(int32_t)));
    PK_CUDA(cudaMallocHost(&h_tc, B * (size_t)cap * sizeof(float)));
    return PK_OK;
}

// Derive every per-utterance extent from either sample offsets or mel frame counts.
pk_status pk_engine::set_batch_shapes(const int32_t *n_frames, const int64_t *offsets, int n) {
    if (n <= 0) return fail(PK_ERR_INVALID, "empty batch");
    if (n > Bmax) return fail(PK_ERR_CAPACITY, "batch of " + std::to_string(n) + " exceeds max_batch " + std::to_string(Bmax));
    n_utt = n;
    pcm_off.assign(n + 1, 0);
    frame_off.assign(n + 1, 0);
    s2_off.assign(n + 1, 0);
    row_off.assign(n + 1, 0);
    t2_rows.assign(n + 1, 0);
    maxF = maxT2 = maxT = 0;
    for (int i = 0; i < n; ++i) {
        int F;
        if (offsets) {
            const int64_t ns = offsets[i + 1] - offsets[i];
            if (ns < 400) return fail(PK_ERR_INVALID, "utterance shorter than one 400-sample window");
            if (ns > cfg.max_samples) return fail(PK_ERR_CAPACITY, "utterance exceeds max_samples");
            pcm_off[i + 1] = pcm_off[i] + ns;
            F = (int)(1 + ns / 160);
        } else {
            F = n_frames[i];
            if (F < 2) return fail(PK_ERR_INVALID, "utterance needs at least 2 mel frames");
            if (F > Fmax) return fail(PK_ERR_CAPACITY, "utterance exceeds max frames");
        }
        const int t1 = conv_len(F), t2 = conv_len(t1), T = conv_len(t2);
        frame_off[i + 1] = frame_off[i] + F;
        s2_off[i + 1] = s2_off[i] + t2;
        row_off[i + 1] = row_off[i] + T;
        t2_rows[i] = t2;
        maxF = std::max(maxF, F);
        maxT2 = std::max(maxT2, t2);
        maxT = std::max(maxT, T);
    }
    M = row_off[n];
    M2 = s2_off[n] * f2n;
    return PK_OK;
}

pk_status pk_engine::upload_shapes() {
    const int n = n_utt;
    int32_t *m = h_meta;
    PK_CUDA(cudaEventSynchronize(ev_h2d));  // pinned staging of the previous batch fully consumed
    memcpy(m, frame_off.data(), (n + 1) * 4);
    memcpy(m + (n + 1), s2_off.data(), (n + 1) * 4);
    memcpy(m + 2 * (n + 1), row_off.data(), (n + 1) * 4);
    memcpy(m + 3 * (n + 1), t2_rows.data(), (n + 1) * 4);
    memcpy(m + 4 * (n + 1), pcm_off.data(), (n + 1) * 8);
    PK_CUDA(cudaMemcpyAsync(d_frame_off, m, (n + 1) * 4, cudaMemcpyHostToDevice, stream));
    PK_CUDA(cudaMemcpyAsync(d_s2_off, m + (n + 1), (n + 1) * 4, cudaMemcpyHostToDevice, stream));
    PK_CUDA(cudaMemcpyAsync(d_row_off, m + 2 * (n + 1), (n + 1) * 4, cudaMemcpyHostToDevice, stream));
    PK_CUDA(cudaMemcpyAsync(d_t2_rows, m + 3 * (n + 1), (n + 1) * 4, cudaMemcpyHostToDevice, stream));
    PK_CUDA(cudaMemcpyAsync(d_pcm_off, m + 4 * (n + 1), (n + 1) * 8, cudaMemcpyHostToDevice, stream));
    PK_CUDA(cudaEventRecord(ev_h2d, stream));
    return PK_OK;
}

// ===================================================================== pipeline

const CUtensorMap *pk_engine::out_map(const void *ptr, bool is_f32, int rows, int ld) {
    auto key = std::make_tuple(ptr, (int)is_f32, rows, ld);
    auto it = out_maps.find(key);
    if (it != out_maps.end()) return &it->second;
    CUtensorMap m;
    if (!make_tc_out_map(&m, ptr, is_f32, (uint64_t)rows, (uint64_t)ld)) return nullptr;
    if (out_maps.size() > 4096) out_maps.clear();          // (shape-varying batches: bounded; maps are rebuilt on demand)
    return &(out_maps[key] = m);
}

void pk_engine::gemm(const Act &A, int lda, const GemmWeight &W, int M_, EpiParams epi) {
    epi.bias = W.bias;
    if (tma_out && cfg.math != PK_MATH_FP32 && epi.kind != EPI_RESID_F32 && M_ > 0) {
        // results leave the SM through the TMA engine (UTMASTG) wherever the tile is interior (gemm_tc.cu: epilogue_slab64)
        const bool act_kind = epi.kind == EPI_BIAS_RELU_ACT || epi.kind == EPI_BIAS_SILU_ACT || epi.kind == EPI_BIAS_ACT || epi.kind == EPI_QKV_ACT;
        if (act_kind && epi.act.hi) {
            const CUtensorMap *m0 = out_map(epi.act.hi, false, M_, epi.ldo), *m1 = epi.act.lo ? out_map(epi.act.lo, false, M_, epi.ldo) : nullptr;
            const CUtensorMap *m2 = epi.kind == EPI_QKV_ACT ? out_map(epi.out_f32, true, M_, epi.qcols) : nullptr;
            if (m0 && (m1 || !epi.act.lo) && (m2 || epi.kind != EPI_QKV_ACT)) { epi.tma_out = 1; epi.tm_out0 = m0; epi.tm_out1 = m1; epi.tm_out2 = m2; }
        } else if (!act_kind && epi.out_f32) {
            const CUtensorMap *m0 = out_map(epi.out_f32, true, M_, epi.ldo);
            if (m0) { epi.tma_out = 1; epi.tm_out0 = m0; }
        }
    }
    Scope sc(this, CAT_GEMM, 2.0 * M_ * W.N * W.K);
    if (cfg.math == PK_MATH_FP32) {
        launch_gemm_simt(A.f32, lda, W.w, W.K, M_, W.N, W.K, epi, stream);
    } else if (skinny && M_ <= 128 && skinny_ws && W.N <= 32 * SKINNY_TICKETS) {
        // one row tile: weight-streaming bound -- split over N and K so that every SM pulls weights (gemm_skinny.cu)
        epi.tma_out = 0;
        cudaError_t ce = launch_gemm_skinny(A.hi, A.lo, lda, W.hi, W.lo, M_, W.N, W.K, cfg.math == PK_MATH_BF16X3, epi, skinny_ws, skinny_ws_floats,
                                            skinny_tickets, SKINNY_TICKETS, num_sms, stream);
        if (ce != cudaSuccess && gemm_err == PK_OK) gemm_err = fail(PK_ERR_CUDA, std::string("skinny GEMM launch: ") + cudaGetErrorString(ce));
    } else {
        const int cl = (gemm_cluster == 2 || gemm_cluster == 4) && lda == W.K ? gemm_cluster : 1;
        cudaError_t ce = launch_gemm_tc(A.tc, W.tc, M_, W.N, W.K, cfg.math == PK_MATH_BF16X3, epi, stream, cl, cl == 4 ? &A.tc32 : &A.tc64);
        if (ce != cudaSuccess && gemm_err == PK_OK) gemm_err = fail(PK_ERR_CUDA, std::string("tcgen05 GEMM launch: ") + cudaGetErrorString(ce));
    }
    ++launches;
}

// Front end of utterances [u0, u1): the offset arrays hold absolute positions in the packed
// buffers, so a sub-range is just a shifted view of them.
pk_status pk_engine::run_mel(int u0, int u1) {
    if (u1 < 0) u1 = n_utt;
    if (u1 <= u0) return PK_OK;
    Scope sc(this, CAT_MEL);
    launch_mel(pcm_src ? pcm_src : d_pcm, d_pcm_off + u0, d_frame_off + u0, u1 - u0, maxF, cfg.mel_bins, mel_tb, logmel, feats,
               mel_part + mel_part_floats(u0, cfg.mel_bins), stream);
    launches += 3;
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

// conv1_ + ReLU + dw1_ of ConvSubsampling (encoder.cpp:219-241), first kernel of the encoder
pk_status pk_engine::run_conv1(int u0, int u1) {
    if (u1 < 0) u1 = n_utt;
    if (u1 <= u0) return PK_OK;
    const pk_config &c = cfg;
    Scope sc(this, CAT_SUBSAMPLE);
    launch_subsample_conv1_dw1(feats, d_frame_off + u0, d_s2_off + u0, u1 - u0, maxT2, c.mel_bins, c.sub_channels, c1_w, c1_b,
                               dw1_w, dw1_b, sub1, stream);
    ++launches;
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

#define PK_LN(...)                              \
    do {                                        \
        Scope _sc(this, CAT_LAYERNORM);         \
        launch_layernorm(__VA_ARGS__);          \
    } while (0)

pk_status pk_engine::gemm_ln(const Act &A, int lda, const GemmWeight &W, int M_, bool resid_in_x, float alpha, const float *ln1_w,
                             const float *ln1_b, bool out_ln1, const float *ln2_w, const float *ln2_b, ActBuf planes) {
    const int d = cfg.d_model;
    const bool fused = fuse_ln && W.K >= fuse_ln_min_k && cfg.math != PK_MATH_FP32 && W.N == d && gemm_tc_ln_supported(d) && lda == W.K && W.tc.box_rows == 128 &&
                       !(skinny && M_ <= 128 && skinny_ws) && planes.hi != nullptr;
    if (fused) {
        LnEpi le;
        le.bias = W.bias;
        le.resid = resid_in_x ? x : nullptr;
        le.alpha = alpha;
        le.out_f32 = x;
        le.ln1_w = ln1_w; le.ln1_b = ln1_b; le.ln2_w = ln2_w; le.ln2_b = ln2_b;
        le.out_ln1 = out_ln1;
        le.planes = planes;
        Scope sc(this, CAT_GEMM, 2.0 * M_ * W.N * W.K);
        cudaError_t ce = launch_gemm_tc_ln(ln_mcast ? A.tc32 : A.tc, W.tc, M_, W.N, W.K, cfg.math == PK_MATH_BF16X3, le, num_sms, stream);
        if (ce != cudaSuccess && gemm_err == PK_OK) gemm_err = fail(PK_ERR_CUDA, std::string("tcgen05 GEMM+LayerNorm launch: ") + cudaGetErrorString(ce));
        ++launches;
        return PK_OK;
    }
    EpiParams ep;
    ep.kind = resid_in_x ? EPI_RESID_F32 : EPI_BIAS_F32;
    ep.out_f32 = x;
    ep.resid = resid_in_x ? x : nullptr;
    ep.ldo = d;
    ep.alpha = alpha;
    gemm(A, lda, W, M_, ep);
    ActBuf none;
    if (!out_ln1) PK_LN(x, M_, d, ln1_w, ln1_b, nullptr, planes, nullptr, nullptr, none, stream);
    else if (ln2_w) PK_LN(x, M_, d, ln1_w, ln1_b, x, none, ln2_w, ln2_b, planes, stream);
    else PK_LN(x, M_, d, ln1_w, ln1_b, x, planes, nullptr, nullptr, none, stream);
    ++launches;
    return PK_OK;
}

// conv2_ .. proj_ of ConvSubsampling (encoder.cpp:219-241) on the staged batch; conv1_/dw1_ already ran (run_conv1)
pk_status pk_engine::run_subsample_tail(bool with_first_ln) {
    const pk_config &c = cfg;
    const int C = c.sub_channels, d = c.d_model;
    {
        EpiParams ep;
        ep.kind = EPI_BIAS_RELU_F32;
        ep.out_f32 = sub2;
        ep.ldo = C;
        gemm(sub1, C, conv2, M2, ep);
    }
    {
        Scope sc(this, CAT_SUBSAMPLE);
        launch_subsample_dw(sub2, d_t2_rows, d_s2_off, d_row_off, n_utt, f2n, C, dw2_wt, dw2_b, sub3, M * f3n, stream);
    }
    ++launches;
    {
        EpiParams ep;
        ep.kind = EPI_BIAS_RELU_ACT;
        ep.act = sub4;
        ep.ldo = C;
        gemm(sub3, C, conv3, M * f3n, ep);
    }
    if (with_first_ln) {       // proj_ + the first block's ffn1_.norm_ (encoder.cpp:40)
        pk_status q = gemm_ln(sub4, C * f3n, proj, M, false, 1.0f, layers[0].ffn_ln_w[0], layers[0].ffn_ln_b[0], false, nullptr, nullptr, ln);
        if (q) return q;
    } else {
        EpiParams ep;
        ep.kind = EPI_BIAS_F32;
        ep.out_f32 = x;
        ep.ldo = d;
        gemm(sub4, C * f3n, proj, M, ep);
    }
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

pk_status pk_engine::run_encoder(float *sub_out_host, float *layers_out_host) {
    const pk_config &c = cfg;
    const int d = c.d_model, H = c.n_heads, hd = d / H;
    {
        pk_status ss = run_subsample_tail(true);
        if (ss) return ss;
    }
    PK_CUDA(cudaGetLastError());
    if (sub_out_host) {
        PK_CUDA(cudaMemcpyAsync(sub_out_host, x, (size_t)M * d * 4, cudaMemcpyDeviceToHost, stream));
        PK_CUDA(cudaStreamSynchronize(stream));
    }
    // ---- Conformer blocks (encoder.cpp:196-204).  Every residual GEMM carries the LayerNorm that consumes its result
    // (gemm_ln: one kernel when fuse_ln applies): ffn1 -> attention norm, attention out -> conv norm, conv pw2 -> ffn2 norm,
    // ffn2 -> final_norm_ chained with the next block's ffn1_.norm_.
    ActBuf none;
    // PK_DEBUG_SUBBLOCKS=n (bisecting aid): stop after n residual sub-blocks; x is returned as is.
    int dbg_stop = -1, dbg_cnt = 0;
    if (const char *ev = getenv("PK_DEBUG_SUBBLOCKS")) dbg_stop = atoi(ev);
    for (int i = 0; i < c.n_layers; ++i) {
        const LayerW &L = layers[i];
        const bool last = (i + 1 == c.n_layers);
        pk_status q;
        for (int f = 0; f < 2; ++f) {
            // FeedForward (encoder.cpp:39-46): x += 0.5 * fc2(silu(fc1(LN(x))))
            EpiParams e1;
            e1.kind = EPI_BIAS_SILU_ACT;
            e1.act = ffh;
            e1.ldo = c.ff;
            gemm(ln, d, L.fc1[f], M, e1);
            if (f == 0) {
                q = gemm_ln(ffh, c.ff, L.fc2[f], M, true, 0.5f, L.att_ln_w, L.att_ln_b, false, nullptr, nullptr, ln);
            } else if (!last) {
                // final_norm_ of this block chained with the next block's ffn1_.norm_
                q = gemm_ln(ffh, c.ff, L.fc2[f], M, true, 0.5f, L.fin_ln_w, L.fin_ln_b, true, layers[i + 1].ffn_ln_w[0], layers[i + 1].ffn_ln_b[0], ln);
            } else {
                // after the last block the normalised output is also written in GEMM-operand form for the heads
                q = gemm_ln(ffh, c.ff, L.fc2[f], M, true, 0.5f, L.fin_ln_w, L.fin_ln_b, true, nullptr, nullptr, cfg.math == PK_MATH_FP32 ? none : (ActBuf)ln);
            }
            if (q) return q;
            if (++dbg_cnt == dbg_stop) return PK_OK;
            if (f == 1) break;
            // ConformerAttention (encoder.cpp:111-186)
            const bool tc_attn = L.pp_hi && qkvp_hi && attn_tc;
            EpiParams eq;
            if (tc_attn) {   // k | v land as bf16 hi/lo planes [M, 2 d], q as fp32 [M, d] (the attention kernel adds pos_bias_u / _v)
                eq.kind = EPI_QKV_ACT;
                eq.act.hi = qkvp_hi;
                eq.act.lo = qkvp_lo;
                eq.ldo = 2 * d;
                eq.out_f32 = qkv;
                eq.qcols = d;
            } else {
                eq.kind = EPI_BIAS_F32;
                eq.out_f32 = qkv;
                eq.ldo = 3 * d;
            }
            gemm(ln, d, L.qkv, M, eq);
            {
                Scope sc(this, CAT_ATTENTION);
                bool ok = false;
                if (tc_attn && attn_umma && L.pp_tc_ok && relpos_attention_umma_supported(hd, maxT) && ctx.hi) {
                    // tcgen05 kernel: the k | v planes as a TMA operand of exactly M rows (rows past the batch read as zeros)
                    auto it = kv_maps.find(M);
                    if (it == kv_maps.end()) {
                        if (kv_maps.size() > 256) kv_maps.clear();
                        TcOperand op;
                        if (make_tc_operand(&op, qkvp_hi, qkvp_lo, (uint64_t)M, (uint64_t)2 * d, 128)) it = kv_maps.emplace(M, op).first;
                    }
                    if (it != kv_maps.end())
                        ok = launch_relpos_attention_umma(qkv, L.pos_u, L.pos_v, it->second, L.pp_tc, d_row_off, n_utt, maxT, H, hd, Tmax, d, num_sms, ctx, stream);
                }
                if (!ok)
                    ok = tc_attn
                        ? launch_relpos_attention_tc(qkv, L.pos_u, L.pos_v, qkvp_hi, qkvp_lo, 2 * d, d_row_off, n_utt, maxT, H, hd, L.pp_hi, L.pp_lo, Tmax, d, ctx, stream)
                        : launch_relpos_attention(qkv, 3 * d, d_row_off, n_utt, maxT, H, hd, L.pp, Tmax, L.pos_u, L.pos_v, d, ctx, stream);
                if (!ok) return fail(PK_ERR_INVALID, "unsupported head_dim " + std::to_string(hd));
            }
            ++launches;
            if ((q = gemm_ln(ctx, d, L.out, M, true, 1.0f, L.conv_ln_w, L.conv_ln_b, false, nullptr, nullptr, ln))) return q;
            if (++dbg_cnt == dbg_stop) return PK_OK;
            // ConformerConvModule (encoder.cpp:59-75)
            EpiParams eg;
            eg.kind = EPI_GLU_F32;
            eg.out_f32 = glu;
            eg.ldo = d;
            gemm(ln, d, L.pw1, M, eg);
            {
                Scope sc(this, CAT_DWCONV);
                if (!launch_dwconv_bn_silu(glu, d_row_off, n_utt, maxT, d, c.conv_kernel, L.dw_wt, L.dw_b, cv, stream))
                    return fail(PK_ERR_INVALID, "unsupported conv_kernel");
            }
            ++launches;
            if ((q = gemm_ln(cv, d, L.pw2, M, true, 1.0f, L.ffn_ln_w[1], L.ffn_ln_b[1], false, nullptr, nullptr, ln))) return q;
            if (++dbg_cnt == dbg_stop) return PK_OK;
        }
        if (layers_out_host) {
            PK_CUDA(cudaMemcpyAsync(layers_out_host + (size_t)i * M * d, x, (size_t)M * d * 4, cudaMemcpyDeviceToHost, stream));
        }
    }
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

// encoder output as a GEMM operand
static Act enc_operand(pk_engine *e) {
    if (e->cfg.math == PK_MATH_FP32) {
        Act a;
        a.f32 = e->x;
        return a;
    }
    return e->ln;
}

pk_status pk_engine::run_ctc(float *logprobs_dev) {
    const pk_config &c = cfg;
    if (!c.has_ctc) return fail(PK_ERR_INVALID, "this model has no CTC head");
    const int ldv = (c.vocab + 3) & ~3;
    EpiParams ep;
    ep.kind = EPI_BIAS_F32;
    ep.out_f32 = logits;
    ep.ldo = ldv;
    gemm(enc_operand(this), c.d_model, ctc_head, M, ep);
    if (boost_on && !logprobs_dev) {
        // boosted decode compares log-probs + boost (phrase_boost.cpp:94-102): they land in the (idle) qkv workspace
        if ((size_t)M * c.vocab > (size_t)Bmax * Tmax * 3 * c.d_model) return fail(PK_ERR_CAPACITY, "boosted CTC decode: workspace too small for the log-probs");
        logprobs_dev = qkv;
    }
    {
        Scope sc(this, CAT_CTC);
        launch_ctc_frame_argmax(logits, M, c.vocab, ldv, best, bconf, logprobs_dev, stream);
        if (boost_on)
            launch_ctc_boosted_decode(logprobs_dev, d_row_off, n_utt, c.vocab, c.vocab - 1, cap, trie, boost, tok, t_start, t_end, t_conf, stream);
        else
            launch_ctc_collapse(best, bconf, d_row_off, n_utt, c.vocab - 1, cap, tok, t_start, t_end, t_conf, stream);
    }
    launches += 2;
    last_tdt = false;
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

pk_status pk_engine::run_tdt() {
    const pk_config &c = cfg;
    // enc_proj for all frames at once (joint's first Linear, tdt.cpp:17)
    EpiParams ep;
    ep.kind = EPI_BIAS_F32;
    ep.out_f32 = EP;
    ep.ldo = c.joint_hidden;
    gemm(enc_operand(this), c.d_model, enc_proj, M, ep);

    const int bp = ((n_utt + 31) / 32) * 32;
    TdtParams p{};
    p.P = c.pred_hidden; p.J = c.joint_hidden; p.V = c.vocab; p.D = c.n_durations; p.L = c.lstm_layers;
    p.Bpad = bp; p.n_utt = n_utt; p.cap = cap; p.n_dur = c.n_durations;
    p.max_symbols = c.n_durations == 0 ? c.max_symbols : 0;
    p.max_steps = maxT + cap + 2;     // (RNNT: every step emits or advances, so <= maxT + maxT * max_symbols steps)
    for (int i = 0; i < 8; ++i) p.durations[i] = c.durations[i];
    p.EP = EP; p.row_off = d_row_off; p.G0 = G0;
    for (int l = 0; l < c.lstm_layers; ++l) { p.Whh[l] = Whh_s[l]; p.Wih[l] = Wih_s[l]; p.bih[l] = bih[l]; }
    p.Wp = Wp_s; p.Wout = Wout_s; p.bout = bout;
    p.hbuf = hbuf; p.z = zbuf;
    p.overflow = tdt_ints; p.bar = reinterpret_cast<unsigned int *>(tdt_ints + Bpad);
    p.pl_max = pl_max; p.pl_sum = pl_sum;
    p.key_lab = tdt_keys; p.key_dur = tdt_keys + 3 * (size_t)Bpad;
    p.dbg = reinterpret_cast<long long *>(tdt_keys + 6 * (size_t)Bpad);
    p.tok = tok; p.t_start = t_start; p.t_end = t_end; p.t_conf = t_conf;
    p.boost_on = boost_on ? 1 : 0; p.boost = boost; p.trie = trie; p.boost_bits = boost_bits; p.trie_active = trie_active; p.trie_nact = trie_nact;
    // initial state: zero LSTM state, token = blank (SOS), t = 0 (tdt.cpp:49-59)
    const size_t HS = (size_t)p.P * bp;
    PK_CUDA(cudaMemsetAsync(hbuf, 0, HS * 2 * p.L * sizeof(float), stream));
    cudaError_t ce;
    {
        Scope sc(this, CAT_TDT);
        ce = launch_tdt_decode(p, num_sms, stream);
    }
    launches += 2;
    last_tdt = true;
    if (ce != cudaSuccess) return fail(PK_ERR_CUDA, std::string("tdt_decode launch: ") + cudaGetErrorString(ce));
    PK_CUDA(cudaGetLastError());
    return PK_OK;
}

pk_status pk_engine::fetch(pk_tokens *out) {
    if (!out || !out->ids || !out->len) return fail(PK_ERR_INVALID, "pk_tokens needs ids and len");
    const size_t n = n_utt;
    PK_CUDA(cudaMemcpyAsync(h_tok, tok, n * (1 + cap) * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (out->start) PK_CUDA(cudaMemcpyAsync(h_ts, t_start, n * cap * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (out->end) PK_CUDA(cudaMemcpyAsync(h_te, t_end, n * cap * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    if (out->conf) PK_CUDA(cudaMemcpyAsync(h_tc, t_conf, n * cap * sizeof(float), cudaMemcpyDeviceToHost, stream));
    int32_t *h_ovf = h_meta + 6 * (Bmax + 1);      // (upload_shapes uses the first 6 (n+1) ints)
    if (last_tdt) PK_CUDA(cudaMemcpyAsync(h_ovf, tdt_ints, n * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    PK_CUDA(cudaStreamSynchronize(stream));
    truncated = 0;
    if (last_tdt)
        for (size_t b = 0; b < n; ++b) truncated += h_ovf[b] != 0;
    for (size_t b = 0; b < n; ++b) {
        const int32_t len = h_tok[b * (1 + cap)];
        if (len > out->cap) return fail(PK_ERR_CAPACITY, "pk_tokens.cap too small for utterance " + std::to_string(b));
        out->len[b] = len;
        memcpy(out->ids + b * out->cap, h_tok + b * (1 + cap) + 1, (size_t)len * 4);
        if (out->start) memcpy(out->start + b * out->cap, h_ts + b * cap, (size_t)len * 4);
        if (out->end) memcpy(out->end + b * out->cap, h_te + b * cap, (size_t)len * 4);
        if (out->conf) memcpy(out->conf + b * out->cap, h_tc + b * cap, (size_t)len * 4);
    }
    return PK_OK;
}

// Runs `body` (a sequence of launches on the engine stream whose kernel arguments depend only on `key`) as ONE CUDA graph
// once the key has been seen twice: first sight runs eagerly (which also completes every lazy one-time initialisation),
// second sight captures + instantiates, later sights replay.  Falls back to plain launches if capture is not possible.
pk_status pk_engine::run_graphed(const std::string &key, const std::function<pk_status()> &body) {
    if (!use_graphs || prof_on) return body();
    if (graphs.size() >= 32 && graphs.find(key) == graphs.end()) {
        // Bound the cache at INSERTION: with variable-length audio nearly every batch shape is new.  Drop the
        // entries that never got a graph first; if the instantiated graphs alone fill it, drop those too.
        for (auto it = graphs.begin(); it != graphs.end();)
            it = it->second.exec ? std::next(it) : graphs.erase(it);
        if (graphs.size() >= 24) {
            for (auto &kv : graphs) cudaGraphExecDestroy(kv.second.exec);
            graphs.clear();
        }
    }
    auto &g = graphs[key];
    if (g.exec) {
        cudaError_t ce = cudaGraphLaunch(g.exec, stream);
        if (ce != cudaSuccess) return fail(PK_ERR_CUDA, std::string("cudaGraphLaunch: ") + cudaGetErrorString(ce));
        launches += g.launches;
        return PK_OK;
    }
    if (g.seen++ == 0) return body();
    const int64_t l0 = launches;
    cudaError_t ce = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
    if (ce != cudaSuccess) return fail(PK_ERR_CUDA, std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(ce));
    pk_status s = body();
    cudaGraph_t graph = nullptr;
    ce = cudaStreamEndCapture(stream, &graph);
    if (s != PK_OK || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        use_graphs = false;     // capture not possible here: stay on plain launches
        launches = l0;
        return body();
    }
    g.launches = launches - l0;
    ce = cudaGraphInstantiate(&g.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) {
        g.exec = nullptr;
        cudaGetLastError();
        use_graphs = false;
        launches = l0;
        return body();
    }
    ce = cudaGraphLaunch(g.exec, stream);
    if (ce != cudaSuccess) return fail(PK_ERR_CUDA, std::string("cudaGraphLaunch: ") + cudaGetErrorString(ce));
    return PK_OK;
}

// ===================================================================== C-ABI

extern "C" {

void pk_config_110m(pk_config *c) {
    memset(c, 0, sizeof(*c));
    c->mel_bins = 80; c->sub_channels = 256; c->d_model = 512; c->n_layers = 17; c->n_heads = 8; c->ff = 2048;
    c->conv_kernel = 9; c->vocab = 1025; c->pred_hidden = 640; c->lstm_layers = 1; c->joint_hidden = 640;
    c->n_durations = 5;
    for (int i = 0; i < 5; ++i) c->durations[i] = i;
    c->has_ctc = 1; c->joint_prefix_tdt = 1; c->max_symbols = 10;
    c->max_batch = 64; c->max_samples = 160000; c->math = PK_MATH_BF16X3;
}

void pk_config_tdt_600m(pk_config *c) {
    pk_config_110m(c);
    c->mel_bins = 128; c->d_model = 1024; c->n_layers = 24; c->ff = 4096; c->vocab = 8193; c->lstm_layers = 2;
    c->has_ctc = 0; c->joint_prefix_tdt = 0; c->max_batch = 16; c->max_samples = 480000;
}

void pk_config_rnnt_600m(pk_config *c) {
    pk_config_110m(c);
    c->d_model = 1024; c->n_layers = 24; c->ff = 4096; c->lstm_layers = 2;
    c->n_durations = 0;
    for (int i = 0; i < 8; ++i) c->durations[i] = 0;
    c->has_ctc = 0; c->joint_prefix_tdt = 0; c->max_batch = 16; c->max_samples = 480000;
}

int32_t pk_mel_frames(int64_t n_samples) { return (int32_t)(1 + n_samples / 160); }
int32_t pk_encoder_frames(int32_t f) { return conv_len(conv_len(conv_len(f))); }

const char *pk_last_error(const pk_engine *e) { return e ? e->err.c_str() : g_create_err.c_str(); }

pk_status pk_engine_create(const pk_config *cfg, const char *path, int device, pk_engine **out) {
    if (!cfg || !path || !out) {
        g_create_err = "null argument";
        return PK_ERR_INVALID;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        g_create_err = "no CUDA device: this engine has no CPU fallback";
        return PK_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) {
        g_create_err = "bad device index";
        return PK_ERR_INVALID;
    }
    const pk_config &c = *cfg;
    if (c.d_model % 128 || c.d_model % c.n_heads || c.mel_bins % 8 || c.sub_channels % 4 || c.ff % 16 ||
        c.pred_hidden % 32 || c.joint_hidden % 32 || c.lstm_layers < 1 || c.lstm_layers > PK_MAX_LSTM ||
        c.n_durations < 0 || c.n_durations > 8 || c.max_batch < 1 || c.max_samples < 400 || c.sub_channels > 1024 ||
        (c.n_durations == 0 && (c.max_symbols < 1 || c.max_symbols > 64))) {
        g_create_err = "unsupported model shape in pk_config";
        return PK_ERR_INVALID;
    }
    if (c.math != PK_MATH_FP32 && c.math != PK_MATH_BF16X3 && c.math != PK_MATH_BF16X1) {
        g_create_err = "unknown pk_math mode";
        return PK_ERR_INVALID;
    }
    if (const char *ev = getenv("PK_GEMM_2CTA")) tc_set_2cta(atoi(ev) != 0);
    auto e = std::make_unique<pk_engine>();
    e->cfg = c;
    if (const char *ev = getenv("PK_GRAPH")) e->use_graphs = atoi(ev) != 0;
    if (const char *ev = getenv("PK_ATTN_TC")) e->attn_tc = atoi(ev) != 0;
    if (const char *ev = getenv("PK_ATTN_UMMA")) e->attn_umma = atoi(ev) != 0;
    if (const char *ev = getenv("PK_GEMM_TMA_OUT")) e->tma_out = atoi(ev) != 0;
    if (const char *ev = getenv("PK_GEMM_SKINNY")) e->skinny = atoi(ev) != 0;
    if (const char *ev = getenv("PK_FUSE_LN")) e->fuse_ln = atoi(ev) != 0;
    if (const char *ev = getenv("PK_GEMM_CLUSTER")) e->gemm_cluster = atoi(ev);
    if (const char *ev = getenv("PK_LN_MCAST")) e->ln_mcast = atoi(ev) != 0;
    if (const char *ev = getenv("PK_FUSE_LN_MINK")) e->fuse_ln_min_k = atoi(ev);
    e->device = device;
    if (cudaSetDevice(device) != cudaSuccess) {
        g_create_err = "cudaSetDevice failed";
        return PK_ERR_CUDA;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    e->num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
        g_create_err = "cudaStreamCreate failed";
        return PK_ERR_CUDA;
    }
    bool ev_ok = cudaEventCreateWithFlags(&e->ev_h2d, cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&e->ev_front, cudaEventDisableTiming) == cudaSuccess &&
                 cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < pk_engine::H2D_CHUNKS && ev_ok; ++i)
        ev_ok = cudaEventCreateWithFlags(&e->ev_chunk[i], cudaEventDisableTiming) == cudaSuccess;
    ev_ok = ev_ok && cudaEventCreateWithFlags(&e->ev_prefetch, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_pcm_free[0], cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&e->ev_pcm_free[1], cudaEventDisableTiming) == cudaSuccess;
    if (!ev_ok) {
        g_create_err = "cudaEventCreate / cudaStreamCreate failed";
        return PK_ERR_CUDA;
    }
    e->Bmax = c.max_batch;
    e->Fmax = 1 + c.max_samples / 160;
    e->Tmax = pk_encoder_frames(e->Fmax);
    e->f1n = conv_len(c.mel_bins);
    e->f2n = conv_len(e->f1n);
    e->f3n = conv_len(e->f2n);
    // RNNT emits at most max_symbols tokens per frame, so Tmax * max_symbols can never truncate
    e->cap = c.n_durations == 0 ? e->Tmax * c.max_symbols : 2 * e->Tmax + 8;
    pk_status s = e->load(path);
    if (s == PK_OK) s = e->alloc_workspace();
    if (s != PK_OK) {
        g_create_err = e->err;
        pk_engine_destroy(e.release());
        return s;
    }
    *out = e.release();
    return PK_OK;
}

void pk_engine_destroy(pk_engine *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (void *p : e->allocs) cudaFree(p);
    for (auto &kv : e->graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    for (auto &r : e->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto ev : e->ev_pool) cudaEventDestroy(ev);
    pk_stream_free(e);
    if (e->nccl_comm && nccl_api().ok) nccl_api().CommDestroy(e->nccl_comm);
    if (e->h_job) cudaFreeHost(e->h_job);
    if (e->h_pcm) cudaFreeHost(e->h_pcm);
    if (e->h_meta) cudaFreeHost(e->h_meta);
    if (e->h_tok) cudaFreeHost(e->h_tok);
    if (e->h_ts) cudaFreeHost(e->h_ts);
    if (e->h_te) cudaFreeHost(e->h_te);
    if (e->h_tc) cudaFreeHost(e->h_tc);
    if (e->ev_h2d) cudaEventDestroy(e->ev_h2d);
    if (e->ev_front) cudaEventDestroy(e->ev_front);
    for (int i = 0; i < pk_engine::H2D_CHUNKS; ++i)
        if (e->ev_chunk[i]) cudaEventDestroy(e->ev_chunk[i]);
    if (e->ev_prefetch) cudaEventDestroy(e->ev_prefetch);
    for (int i = 0; i < 2; ++i)
        if (e->ev_pcm_free[i]) cudaEventDestroy(e->ev_pcm_free[i]);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

void *pk_stream(pk_engine *e) { return e ? (void *)e->stream : nullptr; }
int64_t pk_launch_count(const pk_engine *e) { return e ? e->launches : 0; }

pk_status pk_profile_begin(pk_engine *e) {
    if (!e) return PK_ERR_INVALID;
    e->prof_on = true;
    return PK_OK;
}

pk_status pk_profile_end(pk_engine *e, double *ms, int64_t *counts, double *flops, int32_t n) {
    if (!e || !ms || !counts || n < pk_engine::CAT_N) return PK_ERR_INVALID;
    cudaStreamSynchronize(e->stream);
    for (int i = 0; i < n; ++i) { ms[i] = 0; counts[i] = 0; if (flops) flops[i] = 0; }
    for (auto &r : e->prof) {
        float t = 0.f;
        cudaEventElapsedTime(&t, r.a, r.b);
        ms[r.cat] += t;
        counts[r.cat] += 1;
        if (flops) flops[r.cat] += r.flops;
        e->ev_pool.push_back(r.a);
        e->ev_pool.push_back(r.b);
    }
    e->prof.clear();
    e->prof_on = false;
    return PK_OK;
}

const char *pk_profile_names(void) { return "mel,subsample,gemm,layernorm,attention,dwconv,ctc,tdt"; }

pk_status pk_flush_l2(pk_engine *e) {
    if (!e) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (!e->l2_scratch) {
        e->l2_scratch_bytes = (size_t)256 << 20;   // > 126 MB L2
        if (cudaMalloc(&e->l2_scratch, e->l2_scratch_bytes) != cudaSuccess) return e->fail(PK_ERR_CUDA, "cudaMalloc (L2 scratch)");
        e->allocs.push_back(e->l2_scratch);
    }
    cudaError_t ce = cudaMemsetAsync(e->l2_scratch, (int)(++e->l2_flushes & 0xff), e->l2_scratch_bytes, e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("L2 flush: ") + cudaGetErrorString(ce));
    return PK_OK;
}

// Runs one GEMM through the tcgen05 kernel and through the fp32 CUDA-core kernel on seeded
// random data and returns max |tc - fp32| and max |fp32| (GPU self-check used by the tests).
pk_status pk_selftest_gemm(int device, int M, int N, int K, int epi_kind, int math, uint32_t seed, float *max_err,
                           float *max_ref) {
    if (cudaSetDevice(device) != cudaSuccess) return PK_ERR_CUDA;
    if (const char *ev = getenv("PK_GEMM_2CTA")) tc_set_2cta(atoi(ev) != 0);
    tc_set_debug(getenv("PK_GEMM_DBG") ? atoi(getenv("PK_GEMM_DBG")) : 0);
    if (K % 64 != 0 || (epi_kind == EPI_GLU_F32 && (N & 1))) return PK_ERR_INVALID;
    const int qcols = epi_kind == EPI_QKV_ACT ? N / 3 : 0;     // fused q/k/v projection: N = 3 d -> fp32 q [M, d] + planes [M, 2 d]
    if (epi_kind == EPI_QKV_ACT && (N % 3 != 0 || qcols % 16 != 0)) return PK_ERR_INVALID;
    cudaStream_t st;
    cudaStreamCreate(&st);
    const bool act_out = epi_kind == EPI_BIAS_RELU_ACT || epi_kind == EPI_BIAS_SILU_ACT || epi_kind == EPI_BIAS_ACT ||
                         epi_kind == EPI_QKV_ACT;
    const int No = epi_kind == EPI_GLU_F32 ? N / 2 : N - qcols;
    std::vector<float> hA((size_t)M * K), hW((size_t)N * K), hb(N), hr((size_t)M * No);
    uint32_t sd = seed * 2654435761u + 12345u;
    auto rnd = [&]() { sd = sd * 1664525u + 1013904223u; return ((sd >> 8) & 0xffff) / 32768.0f - 1.0f; };
    for (auto &v : hA) v = rnd();
    for (auto &v : hW) v = rnd() * 0.1f;
    for (auto &v : hb) v = rnd();
    for (auto &v : hr) v = rnd();
    float *dA, *dW, *db, *dr, *o_ref, *o_tc, *q_ref = nullptr, *q_tc = nullptr;
    bf16 *Ah, *Al, *Wh, *Wl, *oh, *ol;
    if (qcols) { cudaMalloc(&q_ref, (size_t)M * qcols * 4); cudaMalloc(&q_tc, (size_t)M * qcols * 4); }
    cudaMalloc(&dA, hA.size() * 4); cudaMalloc(&dW, hW.size() * 4); cudaMalloc(&db, hb.size() * 4);
    cudaMalloc(&dr, hr.size() * 4); cudaMalloc(&o_ref, hr.size() * 4); cudaMalloc(&o_tc, hr.size() * 4);
    cudaMalloc(&Ah, hA.size() * 2); cudaMalloc(&Al, hA.size() * 2); cudaMalloc(&Wh, hW.size() * 2); cudaMalloc(&Wl, hW.size() * 2);
    cudaMalloc(&oh, hr.size() * 2); cudaMalloc(&ol, hr.size() * 2);
    cudaMemcpy(dA, hA.data(), hA.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dW, hW.data(), hW.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(db, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dr, hr.data(), hr.size() * 4, cudaMemcpyHostToDevice);
    cudaDeviceSynchronize();
    ActBuf sa; sa.hi = Ah; sa.lo = Al;
    ActBuf sw; sw.hi = Wh; sw.lo = Wl;
    launch_split(dA, hA.size(), sa, st);
    launch_split(dW, hW.size(), sw, st);
    EpiParams ep;
    ep.kind = epi_kind; ep.bias = db; ep.ldo = No; ep.resid = dr; ep.alpha = 0.5f;
    ep.qcols = qcols;
    ep.out_f32 = qcols ? q_ref : o_ref;
    ActBuf ref_act; ref_act.f32 = o_ref;
    ep.act = ref_act;
    launch_gemm_simt(dA, K, dW, K, M, N, K, ep, st);
    TcOperand ta, tw;
    pk_status rc = PK_OK;
    const int cl = getenv("PK_GEMM_CLUSTER") ? atoi(getenv("PK_GEMM_CLUSTER")) : 1;
    TcOperand ta_sl;
    if (!make_tc_operand(&ta, Ah, Al, M, K, 128) || !make_tc_operand(&tw, Wh, Wl, N, K, tc_tile_n(N))) rc = PK_ERR_CUDA;
    if (rc == PK_OK && (cl == 2 || cl == 4) && !make_tc_operand(&ta_sl, Ah, Al, M, K, 128 / cl)) rc = PK_ERR_CUDA;
    if (rc == PK_OK) {
        ep.out_f32 = qcols ? q_tc : o_tc;
        ActBuf tc_act; tc_act.hi = oh; tc_act.lo = ol;
        ep.act = tc_act;
        CUtensorMap om0, om1, om2;
        if (getenv("PK_GEMM_TMA_OUT") && atoi(getenv("PK_GEMM_TMA_OUT")) && epi_kind != EPI_RESID_F32) {
            const bool ok = act_out ? (make_tc_out_map(&om0, oh, false, M, No) && make_tc_out_map(&om1, ol, false, M, No))
                                    : make_tc_out_map(&om0, o_tc, true, M, No);
            if (ok && (!qcols || make_tc_out_map(&om2, q_tc, true, M, qcols))) {
                ep.tma_out = 1; ep.tm_out0 = &om0; ep.tm_out1 = act_out ? &om1 : nullptr; ep.tm_out2 = qcols ? &om2 : nullptr;
            }
        }
        const bool use_skinny = getenv("PK_SELFTEST_SKINNY") && atoi(getenv("PK_SELFTEST_SKINNY")) && M <= 128;
        float *sws = nullptr;
        unsigned int *stk = nullptr;
        if (use_skinny) {           // the few-row kernel (gemm_skinny.cu) on the same operands
            cudaMalloc(&sws, ((size_t)2 << 20) * sizeof(float));
            cudaMalloc(&stk, 1024 * sizeof(unsigned int));
            cudaMemsetAsync(stk, 0, 1024 * sizeof(unsigned int), st);
            int sms = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
            ep.tma_out = 0;
            for (int rep = 0; rep < 2 && rc == PK_OK; ++rep)      // twice: the tickets must come back to zero
                if (launch_gemm_skinny(Ah, Al, K, Wh, Wl, M, N, K, math == PK_MATH_BF16X3, ep, sws, (size_t)2 << 20, stk, 1024, sms, st) != cudaSuccess) rc = PK_ERR_CUDA;
            cudaStreamSynchronize(st);
            cudaFree(sws);
            cudaFree(stk);
        } else if (launch_gemm_tc(ta, tw, M, N, K, math == PK_MATH_BF16X3, ep, st, cl, &ta_sl) != cudaSuccess) rc = PK_ERR_CUDA;
        if (rc == PK_OK && !use_skinny && getenv("PK_SELFTEST_TIME")) {   // warm, back-to-back timing of the tcgen05 launch
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            const int reps = 20;
            cudaEventRecord(e0, st);
            for (int i = 0; i < reps; ++i) launch_gemm_tc(ta, tw, M, N, K, math == PK_MATH_BF16X3, ep, st, cl, &ta_sl);
            cudaEventRecord(e1, st);
            cudaStreamSynchronize(st);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            const double us = 1e3 * ms / reps, tf = 2.0 * M * N * K / (us * 1e-6) / 1e12;
            fprintf(stderr, "gemm_tc M=%d N=%d K=%d epi=%d math=%d: %.1f us  %.1f TFLOP/s algorithmic (x%d MMA)  [probe %.0f MHz]\n", M, N, K,
                    epi_kind, math, us, tf, math == PK_MATH_BF16X3 ? 3 : 1, tc_probe_mhz());
            cudaEventDestroy(e0); cudaEventDestroy(e1);
            if (getenv("PK_GEMM_DBG") && (atoi(getenv("PK_GEMM_DBG")) & 32)) tc_print_timeline(8);
        }
    }
    if (cudaStreamSynchronize(st) != cudaSuccess) rc = PK_ERR_CUDA;
    if (rc == PK_OK) {
        std::vector<float> r(hr.size()), t(hr.size());
        cudaMemcpy(r.data(), o_ref, r.size() * 4, cudaMemcpyDeviceToHost);
        if (act_out) {
            std::vector<bf16> h(hr.size()), l(hr.size());
            cudaMemcpy(h.data(), oh, h.size() * 2, cudaMemcpyDeviceToHost);
            cudaMemcpy(l.data(), ol, l.size() * 2, cudaMemcpyDeviceToHost);
            for (size_t i = 0; i < t.size(); ++i) t[i] = __bfloat162float(h[i]) + __bfloat162float(l[i]);
        } else {
            cudaMemcpy(t.data(), o_tc, t.size() * 4, cudaMemcpyDeviceToHost);
        }
        float me = 0.f, mr = 0.f;
        for (size_t i = 0; i < t.size(); ++i) {
            const float e = std::fabs(t[i] - r[i]);
            if (!(e <= me)) me = e;            // NaN-propagating max
            mr = std::max(mr, std::fabs(r[i]));
        }
        if (qcols) {                           // the fp32 q columns of the fused projection
            std::vector<float> qr((size_t)M * qcols), qt((size_t)M * qcols);
            cudaMemcpy(qr.data(), q_ref, qr.size() * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(qt.data(), q_tc, qt.size() * 4, cudaMemcpyDeviceToHost);
            for (size_t i = 0; i < qt.size(); ++i) {
                const float e = std::fabs(qt[i] - qr[i]);
                if (!(e <= me)) me = e;
                mr = std::max(mr, std::fabs(qr[i]));
            }
        }
        *max_err = me;
        *max_ref = mr;
    }
    for (void *p : {(void *)dA, (void *)dW, (void *)db, (void *)dr, (void *)o_ref, (void *)o_tc, (void *)Ah, (void *)Al,
                    (void *)Wh, (void *)Wl, (void *)oh, (void *)ol, (void *)q_ref, (void *)q_tc})
        cudaFree(p);
    cudaStreamDestroy(st);
    return rc;
}

// GPU self-check of the fused residual-GEMM + LayerNorm kernel (gemm_tc_ln.cu) against the fp32 CUDA-core GEMM followed by
// layernorm_kernel, N = 512.  mode 0: x = resid + a (A W^T + b), planes = LN1(x);  1: x = LN1(.), planes = LN2(x) (block end);
// 2: x = LN1(.), planes = split(x) (last block);  3: mode 0 without a residual (proj_).  The fused kernel runs IN PLACE
// (out = resid), as the encoder uses it.  err4 = {max |x - x_ref|, max |x_ref|, max |planes - planes_ref|, max |planes_ref|}.
pk_status pk_selftest_gemm_ln(int device, int M, int K, int mode, int math, uint32_t seed, float *err4) {
    if (cudaSetDevice(device) != cudaSuccess) return PK_ERR_CUDA;
    const int N = 512;
    if (K % 64 != 0 || M < 1 || mode < 0 || mode > 3 || !err4) return PK_ERR_INVALID;
    cudaStream_t st;
    cudaStreamCreate(&st);
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    std::vector<float> hA((size_t)M * K), hW((size_t)N * K), hb(N), hr((size_t)M * N), hl(4 * N);
    uint32_t sd = seed * 2654435761u + 777u;
    auto rnd = [&]() { sd = sd * 1664525u + 1013904223u; return ((sd >> 8) & 0xffff) / 32768.0f - 1.0f; };
    for (auto &v : hA) v = rnd();
    for (auto &v : hW) v = rnd() * 0.1f;
    for (auto &v : hb) v = rnd();
    for (auto &v : hr) v = rnd() + 0.25f;
    for (int i = 0; i < 4 * N; ++i) hl[i] = (i / N) % 2 == 0 ? 1.0f + 0.5f * rnd() : 0.3f * rnd();   // w1, b1, w2, b2
    float *dA, *dW, *db, *dr, *dl, *x_ref, *x_tc, *p_ref;
    bf16 *Ah, *Al, *Wh, *Wl, *ph, *pl;
    cudaMalloc(&dA, hA.size() * 4); cudaMalloc(&dW, hW.size() * 4); cudaMalloc(&db, hb.size() * 4); cudaMalloc(&dr, hr.size() * 4);
    cudaMalloc(&dl, hl.size() * 4); cudaMalloc(&x_ref, hr.size() * 4); cudaMalloc(&x_tc, hr.size() * 4); cudaMalloc(&p_ref, hr.size() * 4);
    cudaMalloc(&Ah, hA.size() * 2); cudaMalloc(&Al, hA.size() * 2); cudaMalloc(&Wh, hW.size() * 2); cudaMalloc(&Wl, hW.size() * 2);
    cudaMalloc(&ph, hr.size() * 2); cudaMalloc(&pl, hr.size() * 2);
    cudaMemcpy(dA, hA.data(), hA.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dW, hW.data(), hW.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(db, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dr, hr.data(), hr.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dl, hl.data(), hl.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(x_tc, hr.data(), hr.size() * 4, cudaMemcpyHostToDevice);      // in place: starts as the residual
    cudaMemset(ph, 0, hr.size() * 2); cudaMemset(pl, 0, hr.size() * 2);
    cudaDeviceSynchronize();
    const float *w1 = dl, *b1 = dl + N, *w2 = dl + 2 * N, *b2 = dl + 3 * N;
    const bool has_resid = mode != 3, out_ln1 = mode == 1 || mode == 2, two = mode == 1;
    ActBuf sa; sa.hi = Ah; sa.lo = Al;
    ActBuf sw; sw.hi = Wh; sw.lo = Wl;
    launch_split(dA, hA.size(), sa, st);
    launch_split(dW, hW.size(), sw, st);
    // reference: fp32 GEMM (+ residual), then the stand-alone LayerNorm kernel
    EpiParams ep;
    ep.kind = has_resid ? EPI_RESID_F32 : EPI_BIAS_F32; ep.bias = db; ep.ldo = N; ep.resid = has_resid ? dr : nullptr; ep.alpha = has_resid ? 0.5f : 1.0f;
    ep.out_f32 = x_ref;
    launch_gemm_simt(dA, K, dW, K, M, N, K, ep, st);
    ActBuf none, refp; refp.f32 = p_ref;
    if (!out_ln1) launch_layernorm(x_ref, M, N, w1, b1, nullptr, refp, nullptr, nullptr, none, st);
    else if (two) launch_layernorm(x_ref, M, N, w1, b1, x_ref, none, w2, b2, refp, st);
    else launch_layernorm(x_ref, M, N, w1, b1, x_ref, refp, nullptr, nullptr, none, st);
    TcOperand ta, tw;
    pk_status rc = PK_OK;
    const bool mcast = getenv("PK_LN_MCAST") && atoi(getenv("PK_LN_MCAST")) != 0;
    TcOperand ta128;                              // (the unfused comparison launch needs the 128-row box)
    if (!make_tc_operand(&ta, Ah, Al, M, K, mcast ? 32 : 128) || !make_tc_operand(&ta128, Ah, Al, M, K, 128) || !make_tc_operand(&tw, Wh, Wl, N, K, 128)) rc = PK_ERR_CUDA;
    gemm_tc_ln_set_debug(getenv("PK_LN_DBG") ? atoi(getenv("PK_LN_DBG")) : 0);
    LnEpi le;
    le.bias = db; le.resid = has_resid ? x_tc : nullptr; le.alpha = ep.alpha; le.out_f32 = x_tc;
    le.ln1_w = w1; le.ln1_b = b1; le.ln2_w = two ? w2 : nullptr; le.ln2_b = two ? b2 : nullptr; le.out_ln1 = out_ln1;
    le.planes.hi = ph; le.planes.lo = math == PK_MATH_BF16X3 ? pl : nullptr;
    if (rc == PK_OK && launch_gemm_tc_ln(ta, tw, M, N, K, math == PK_MATH_BF16X3, le, sms, st) != cudaSuccess) rc = PK_ERR_CUDA;
    if (rc == PK_OK && cudaStreamSynchronize(st) != cudaSuccess) rc = PK_ERR_CUDA;
    if (rc == PK_OK) {
        std::vector<float> xr(hr.size()), xt(hr.size()), pr(hr.size());
        std::vector<bf16> h(hr.size()), l(hr.size());
        cudaMemcpy(xr.data(), x_ref, xr.size() * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(xt.data(), x_tc, xt.size() * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(pr.data(), p_ref, pr.size() * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(h.data(), ph, h.size() * 2, cudaMemcpyDeviceToHost);
        cudaMemcpy(l.data(), pl, l.size() * 2, cudaMemcpyDeviceToHost);
        float e0 = 0.f, r0 = 0.f, e1 = 0.f, r1 = 0.f;
        for (size_t i = 0; i < xr.size(); ++i) {
            const float ex = std::fabs(xt[i] - xr[i]);
            if (!(ex <= e0)) e0 = ex;
            r0 = std::max(r0, std::fabs(xr[i]));
            const float pv = __bfloat162float(h[i]) + (math == PK_MATH_BF16X3 ? __bfloat162float(l[i]) : 0.f);
            const float epv = std::fabs(pv - pr[i]);
            if (!(epv <= e1)) e1 = epv;
            r1 = std::max(r1, std::fabs(pr[i]));
        }
        err4[0] = e0; err4[1] = r0; err4[2] = e1; err4[3] = r1;
    }
    if (rc == PK_OK && getenv("PK_SELFTEST_TIME")) {   // warm back-to-back: the fused kernel vs residual GEMM + layernorm_kernel
        cudaEvent_t e0, e1, e2;
        cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
        const int reps = 20;
        EpiParams er;
        er.kind = EPI_RESID_F32; er.bias = db; er.ldo = N; er.resid = x_tc; er.out_f32 = x_tc; er.alpha = 0.5f;
        ActBuf tp; tp.hi = ph; tp.lo = pl;
        for (int w = 0; w < 2; ++w) {
            cudaEventRecord(e0, st);
            for (int i = 0; i < reps; ++i) launch_gemm_tc_ln(ta, tw, M, N, K, math == PK_MATH_BF16X3, le, sms, st);
            cudaEventRecord(e1, st);
            for (int i = 0; i < reps; ++i) {
                launch_gemm_tc(ta128, tw, M, N, K, math == PK_MATH_BF16X3, er, st);
                if (two) launch_layernorm(x_tc, M, N, w1, b1, x_tc, none, w2, b2, tp, st);
                else launch_layernorm(x_tc, M, N, w1, b1, out_ln1 ? x_tc : nullptr, tp, nullptr, nullptr, none, st);
            }
            cudaEventRecord(e2, st);
            cudaStreamSynchronize(st);
        }
        float ms0 = 0.f, ms1 = 0.f;
        cudaEventElapsedTime(&ms0, e0, e1);
        cudaEventElapsedTime(&ms1, e1, e2);
        fprintf(stderr, "gemm_tc_ln M=%d N=%d K=%d mode=%d math=%d: fused %.1f us | gemm_tc + layernorm %.1f us\n", M, N, K, mode, math,
                1e3 * ms0 / reps, 1e3 * ms1 / reps);
        if (getenv("PK_LN_DBG") && atoi(getenv("PK_LN_DBG"))) gemm_tc_ln_print_timeline(2);
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    }
    for (void *p : {(void *)dA, (void *)dW, (void *)db, (void *)dr, (void *)dl, (void *)x_ref, (void *)x_tc, (void *)p_ref, (void *)Ah, (void *)Al,
                    (void *)Wh, (void *)Wl, (void *)ph, (void *)pl})
        cudaFree(p);
    cudaStreamDestroy(st);
    return rc;
}

// GPU self-check of the tcgen05 attention kernel (attention_umma.cu) against the fp32 CUDA-core attention kernel on seeded
// random q | k | v, position table and biases: d_model 512, 8 heads of 64, utterance lengths lens[0..n) (<= 128), table for
// `tmax` frames.  mode bit 0: zero position table (isolates Qu.K^T -> softmax -> P.V); bit 1: zero keys (isolates the
// rel_shift path).  err2 = {max |ctx - ctx_ref|, max |ctx_ref|}.
pk_status pk_selftest_attention(int device, const int32_t *lens, int n, int tmax, int mode, uint32_t seed, float *err2) {
    if (cudaSetDevice(device) != cudaSuccess) return PK_ERR_CUDA;
    const int d = 512, H = 8, hd = 64;
    if (!lens || n < 1 || !err2 || tmax < 1) return PK_ERR_INVALID;
    std::vector<int32_t> off(n + 1, 0);
    int maxT = 0;
    for (int i = 0; i < n; ++i) {
        if (lens[i] < 0 || lens[i] > 128 || lens[i] > tmax) return PK_ERR_INVALID;
        off[i + 1] = off[i] + lens[i];
        maxT = std::max(maxT, (int)lens[i]);
    }
    const int M = off[n], NP = 2 * tmax - 1;
    if (M < 1) return PK_ERR_INVALID;
    cudaStream_t st;
    cudaStreamCreate(&st);
    uint32_t sd = seed * 2654435761u + 4242u;
    auto rnd = [&]() { sd = sd * 1664525u + 1013904223u; return ((sd >> 8) & 0xffff) / 32768.0f - 1.0f; };
    std::vector<float> hq((size_t)M * 3 * d), hpp((size_t)NP * d), hu(d), hv(d);
    for (auto &v : hq) v = rnd();
    for (auto &v : hpp) v = (mode & 1) ? 0.f : rnd();
    for (auto &v : hu) v = 0.3f * rnd();
    for (auto &v : hv) v = 0.3f * rnd();
    if (mode & 2)
        for (int r = 0; r < M; ++r)
            for (int c = 0; c < d; ++c) hq[(size_t)r * 3 * d + d + c] = 0.f;
    std::vector<float> hq32((size_t)M * d), hkv((size_t)M * 2 * d);
    for (int r = 0; r < M; ++r) {
        memcpy(&hq32[(size_t)r * d], &hq[(size_t)r * 3 * d], (size_t)d * 4);
        memcpy(&hkv[(size_t)r * 2 * d], &hq[(size_t)r * 3 * d + d], (size_t)2 * d * 4);
    }
    float *dq, *dq32, *dkv, *dpp, *du, *dv, *c_ref;
    bf16 *kvh, *kvl, *pph, *ppl, *ch, *cl;
    int32_t *doff;
    cudaMalloc(&dq, hq.size() * 4); cudaMalloc(&dq32, hq32.size() * 4); cudaMalloc(&dkv, hkv.size() * 4); cudaMalloc(&dpp, hpp.size() * 4);
    cudaMalloc(&du, d * 4); cudaMalloc(&dv, d * 4); cudaMalloc(&c_ref, (size_t)M * d * 4);
    cudaMalloc(&kvh, hkv.size() * 2); cudaMalloc(&kvl, hkv.size() * 2); cudaMalloc(&pph, hpp.size() * 2); cudaMalloc(&ppl, hpp.size() * 2);
    cudaMalloc(&ch, (size_t)M * d * 2); cudaMalloc(&cl, (size_t)M * d * 2); cudaMalloc(&doff, (n + 1) * 4);
    cudaMemcpy(dq, hq.data(), hq.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dq32, hq32.data(), hq32.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dkv, hkv.data(), hkv.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dpp, hpp.data(), hpp.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(du, hu.data(), d * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dv, hv.data(), d * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(doff, off.data(), (n + 1) * 4, cudaMemcpyHostToDevice);
    cudaMemset(ch, 0, (size_t)M * d * 2); cudaMemset(cl, 0, (size_t)M * d * 2);
    cudaDeviceSynchronize();
    ActBuf skv; skv.hi = kvh; skv.lo = kvl;
    ActBuf spp; spp.hi = pph; spp.lo = ppl;
    launch_split(dkv, hkv.size(), skv, st);
    launch_split(dpp, hpp.size(), spp, st);
    ActBuf ref; ref.f32 = c_ref;
    pk_status rc = PK_OK;
    if (!launch_relpos_attention(dq, 3 * d, doff, n, maxT, H, hd, dpp, tmax, du, dv, d, ref, st)) rc = PK_ERR_INVALID;
    TcOperand kv, pp;
    if (rc == PK_OK && (!make_tc_operand(&kv, kvh, kvl, (uint64_t)M, (uint64_t)2 * d, 128) || !make_tc_operand(&pp, pph, ppl, (uint64_t)NP, (uint64_t)d, 256))) rc = PK_ERR_CUDA;
    ActBuf got; got.hi = ch; got.lo = cl;
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    relpos_attention_umma_set_debug(getenv("PK_AU_DBG") ? atoi(getenv("PK_AU_DBG")) : 0);
    if (rc == PK_OK && !launch_relpos_attention_umma(dq32, du, dv, kv, pp, doff, n, maxT, H, hd, tmax, d, sms, got, st)) rc = PK_ERR_INVALID;
    if (rc == PK_OK && cudaStreamSynchronize(st) != cudaSuccess) rc = PK_ERR_CUDA;
    if (rc == PK_OK) {
        std::vector<float> r((size_t)M * d);
        std::vector<bf16> h((size_t)M * d), l((size_t)M * d);
        cudaMemcpy(r.data(), c_ref, r.size() * 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(h.data(), ch, h.size() * 2, cudaMemcpyDeviceToHost);
        cudaMemcpy(l.data(), cl, l.size() * 2, cudaMemcpyDeviceToHost);
        float me = 0.f, mr = 0.f;
        for (size_t i = 0; i < r.size(); ++i) {
            const float e = std::fabs(__bfloat162float(h[i]) + __bfloat162float(l[i]) - r[i]);
            if (!(e <= me)) me = e;
            mr = std::max(mr, std::fabs(r[i]));
        }
        err2[0] = me; err2[1] = mr;
    }
    if (rc == PK_OK && getenv("PK_SELFTEST_TIME")) {
        cudaEvent_t e0, e1, e2;
        cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
        const int reps = 20;
        for (int w = 0; w < 2; ++w) {
            cudaEventRecord(e0, st);
            for (int i = 0; i < reps; ++i) launch_relpos_attention_umma(dq32, du, dv, kv, pp, doff, n, maxT, H, hd, tmax, d, sms, got, st);
            cudaEventRecord(e1, st);
            for (int i = 0; i < reps; ++i) launch_relpos_attention_tc(dq32, du, dv, kvh, kvl, 2 * d, doff, n, maxT, H, hd, pph, ppl, tmax, d, got, st);
            cudaEventRecord(e2, st);
            cudaStreamSynchronize(st);
        }
        float ms0 = 0.f, ms1 = 0.f;
        cudaEventElapsedTime(&ms0, e0, e1);
        cudaEventElapsedTime(&ms1, e1, e2);
        fprintf(stderr, "attention n_utt=%d maxT=%d: tcgen05 %.1f us | mma.sync %.1f us\n", n, maxT, 1e3 * ms0 / reps, 1e3 * ms1 / reps);
        if (getenv("PK_AU_DBG") && atoi(getenv("PK_AU_DBG"))) relpos_attention_umma_print_timeline(n < 32 ? 1 : 4);
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    }
    for (void *p : {(void *)dq, (void *)dq32, (void *)dkv, (void *)dpp, (void *)du, (void *)dv, (void *)c_ref, (void *)kvh, (void *)kvl, (void *)pph,
                    (void *)ppl, (void *)ch, (void *)cl, (void *)doff})
        cudaFree(p);
    cudaStreamDestroy(st);
    return rc;
}

// Debug aid: cycles CTA 0 of the last TDT decode spent in {P1, B1, P2, B2, P3, B3, P4} and the
// number of lock-step decode steps (out[7]).
pk_status pk_debug_tdt_phases(pk_engine *e, int64_t *out8) {
    if (!e || !out8) return PK_ERR_INVALID;
    cudaStreamSynchronize(e->stream);
    cudaMemcpy(out8, e->tdt_keys + 6 * (size_t)e->Bpad, 8 * sizeof(int64_t), cudaMemcpyDeviceToHost);
    return PK_OK;
}

// Debug aid: cycles CTA 0 spent in the sections of the decode kernel's passes since the last call
// {x staging, products, partial store + cluster barrier, DSMEM gather + finalise, number of passes}.
pk_status pk_debug_tdt_passes(pk_engine *e, int64_t *out8) {
    if (!e || !out8) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    long long v[8];
    tdt_pass_profile(v, true);
    for (int i = 0; i < 8; ++i) out8[i] = v[i];
    return PK_OK;
}

pk_status pk_sync(pk_engine *e) {
    if (!e) return PK_ERR_INVALID;
    cudaError_t ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("sync: ") + cudaGetErrorString(ce));
    return PK_OK;
}

pk_status pk_stage_pcm(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt) {
    if (!e || !pcm || !offsets) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    pk_status s = e->set_batch_shapes(nullptr, offsets, n_utt);
    if (s) return s;
    e->pcm_src = nullptr;
    const size_t total = (size_t)e->pcm_off[n_utt];
    cudaEventSynchronize(e->ev_h2d);  // previous batch's staging copies have left the pinned buffers
    // Is the caller's buffer already page-locked and packed back to back?  Then DMA straight from it.
    bool packed = true;
    for (int i = 0; i < n_utt; ++i) packed = packed && (offsets[i] - offsets[0] == e->pcm_off[i]);
    cudaPointerAttributes at;
    const bool pinned = cudaPointerGetAttributes(&at, pcm) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();   // an unregistered host pointer is not an error for us
    cudaError_t ce = cudaSuccess;
    e->front_done = false;
    if (e->pref.valid) {
        const bool same = e->pref.pcm == pcm && e->pref.n == n_utt &&
                          std::equal(e->pref.off.begin(), e->pref.off.end(), offsets);
        e->pref.valid = false;
        if (same) {      // the samples are already on their way into the second buffer: adopt it
            if ((s = e->upload_shapes())) return s;
            std::swap(e->d_pcm, e->d_pcm_alt);
            e->pcm_cur ^= 1;
            ce = cudaStreamWaitEvent(e->stream, e->ev_prefetch, 0);
            if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("prefetch wait: ") + cudaGetErrorString(ce));
            if ((s = e->run_mel())) return s;
            if ((s = e->run_conv1())) return s;
            cudaEventRecord(e->ev_pcm_free[e->pcm_cur], e->stream);
            e->front_done = true;
            return PK_OK;
        }
    }
    if (pinned && packed) {
        // DMA in utterance groups on the copy stream; mel + conv1/dw1 of a group start as soon as it has
        // landed, under the DMA of the next group (the copy of 64 x 10 s is ~0.8 ms of PCIe time).
        if ((s = e->upload_shapes())) return s;
        ce = cudaEventRecord(e->ev_front, e->stream);                  // d_pcm of the previous batch is free
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(e->copy_stream, e->ev_front, 0);
        const int nch = std::min<int>(pk_engine::H2D_CHUNKS, n_utt);
        int u0 = 0;
        for (int i = 0; i < nch && ce == cudaSuccess; ++i) {
            // group boundaries balanced by samples
            int u1 = (i == nch - 1) ? n_utt : u0 + 1;
            while (i < nch - 1 && u1 < n_utt - (nch - 1 - i) && (size_t)e->pcm_off[u1] < total * (size_t)(i + 1) / nch) ++u1;
            const size_t o0 = (size_t)e->pcm_off[u0], o1 = (size_t)e->pcm_off[u1];
            ce = cudaMemcpyAsync(e->d_pcm + o0, pcm + offsets[0] + o0, (o1 - o0) * sizeof(float), cudaMemcpyHostToDevice,
                                 e->copy_stream);
            if (ce == cudaSuccess) ce = cudaEventRecord(e->ev_chunk[i], e->copy_stream);
            if (ce == cudaSuccess) ce = cudaStreamWaitEvent(e->stream, e->ev_chunk[i], 0);
            if (ce != cudaSuccess) break;
            if ((s = e->run_mel(u0, u1))) return s;
            if ((s = e->run_conv1(u0, u1))) return s;
            u0 = u1;
        }
        if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("H2D pcm: ") + cudaGetErrorString(ce));
        cudaEventRecord(e->ev_pcm_free[e->pcm_cur], e->stream);
        e->front_done = true;
        return PK_OK;
    }
    // pageable -> pinned staging -> device, utterance by utterance so the DMA of utterance i
    // overlaps the host copy of utterance i+1; utterances are re-packed back to back
    for (int i = 0; i < n_utt && ce == cudaSuccess; ++i) {
        const size_t ns = (size_t)(offsets[i + 1] - offsets[i]);
        memcpy(e->h_pcm + e->pcm_off[i], pcm + offsets[i], ns * sizeof(float));
        ce = cudaMemcpyAsync(e->d_pcm + e->pcm_off[i], e->h_pcm + e->pcm_off[i], ns * sizeof(float),
                             cudaMemcpyHostToDevice, e->stream);
    }
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("H2D pcm: ") + cudaGetErrorString(ce));
    return e->upload_shapes();
}

pk_status pk_prefetch_pcm(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt) {
    if (!e || !pcm || !offsets) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (n_utt <= 0 || n_utt > e->Bmax) return e->fail(PK_ERR_CAPACITY, "bad batch size");
    cudaPointerAttributes at;
    const bool pinned = cudaPointerGetAttributes(&at, pcm) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const int64_t total = offsets[n_utt] - offsets[0];
    bool ok = pinned && total > 0;
    for (int i = 0; i < n_utt && ok; ++i) {
        const int64_t ns = offsets[i + 1] - offsets[i];
        ok = ns >= 400 && ns <= e->cfg.max_samples;
    }
    if (!ok) return e->fail(PK_ERR_INVALID, "pk_prefetch_pcm needs a page-locked, packed buffer of valid utterances");
    // the second buffer was last read by the front end of the batch before the current one
    cudaError_t ce = cudaStreamWaitEvent(e->copy_stream, e->ev_pcm_free[e->pcm_cur ^ 1], 0);
    if (ce == cudaSuccess)
        ce = cudaMemcpyAsync(e->d_pcm_alt, pcm + offsets[0], (size_t)total * sizeof(float), cudaMemcpyHostToDevice, e->copy_stream);
    if (ce == cudaSuccess) ce = cudaEventRecord(e->ev_prefetch, e->copy_stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_prefetch_pcm: ") + cudaGetErrorString(ce));
    e->pref.pcm = pcm;
    e->pref.n = n_utt;
    e->pref.off.assign(offsets, offsets + n_utt + 1);
    e->pref.valid = true;
    return PK_OK;
}

// Front end (mel + conv1/dw1; 3 launches, always plain launches) unless pk_stage_pcm already ran it
// group by group under the H2D copy.
static pk_status run_front(pk_engine *e) {
    if (e->front_done) return PK_OK;
    pk_status s;
    if ((s = e->run_mel())) return s;
    if ((s = e->run_conv1())) return s;
    cudaEventRecord(e->ev_pcm_free[e->pcm_cur], e->stream);
    e->front_done = true;
    return PK_OK;
}
// An RNNT engine (n_durations == 0) decodes with PK_DECODER_RNNT only, a TDT engine never does.
static pk_status check_decoder(pk_engine *e, pk_decoder dec) {
    if (dec != PK_DECODER_CTC && dec != PK_DECODER_TDT && dec != PK_DECODER_RNNT) return e->fail(PK_ERR_INVALID, "unknown pk_decoder");
    const bool rnnt = e->cfg.n_durations == 0;
    if (rnnt && dec != PK_DECODER_RNNT)
        return e->fail(PK_ERR_INVALID, "this engine holds an RNNT model (n_durations = 0): decode with PK_DECODER_RNNT");
    if (!rnnt && dec == PK_DECODER_RNNT)
        return e->fail(PK_ERR_INVALID, "PK_DECODER_RNNT needs an RNNT model (pk_config.n_durations = 0)");
    if (dec == PK_DECODER_RNNT && e->boost_on)
        return e->fail(PK_ERR_INVALID, "phrase boosting is not available for RNNT decoding: clear it with pk_set_boost(e, ..., 0, ...)");
    return PK_OK;
}
static pk_status run_decoder(pk_engine *e, pk_decoder dec) {    // the RNNT rule is a mode of the TDT decode kernel
    return dec == PK_DECODER_CTC ? e->run_ctc(nullptr) : e->run_tdt();
}
static pk_status run_pipeline(pk_engine *e, pk_decoder dec) {   // everything after the front end
    pk_status s;
    if ((s = e->run_encoder(nullptr, nullptr))) return s;
    return run_decoder(e, dec);
}

// The ~250 launches of one batch are replayed as ONE CUDA graph once a batch shape has been seen
// twice (first sight runs eagerly, which also completes every lazy one-time initialisation).
pk_status pk_run_staged(pk_engine *e, pk_decoder dec) {
    if (!e || e->n_utt <= 0) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (e->gemm_err) return e->gemm_err;
    if (pk_status ds = check_decoder(e, dec)) return ds;
    {
        pk_status fs = run_front(e);
        e->front_done = false;      // a second pk_run_staged of the same staged batch re-runs the front end
        if (fs) return fs;
    }
    std::string key(1, dec == PK_DECODER_CTC ? 'c' : dec == PK_DECODER_RNNT ? 'r' : 't');
    const int32_t bg = e->boost_on ? e->boost_gen : 0;
    key.append(reinterpret_cast<const char *>(&bg), sizeof(bg));
    key.append(reinterpret_cast<const char *>(e->frame_off.data()), e->frame_off.size() * sizeof(int32_t));
    return e->run_graphed(key, [e, dec]() { return run_pipeline(e, dec); });
}

pk_status pk_fetch_tokens(pk_engine *e, pk_tokens *out) {
    if (!e) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    return e->fetch(out);
}

pk_status pk_transcribe_batch(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, pk_decoder dec,
                              pk_tokens *out) {
    pk_status s;
    if ((s = pk_stage_pcm(e, pcm, offsets, n_utt))) return s;
    if ((s = pk_run_staged(e, dec))) return s;
    return pk_fetch_tokens(e, out);
}

pk_status pk_token_buffer(pk_engine *e, void **dev_ptr, int32_t *rows, int32_t *row_ints) {
    if (!e || !dev_ptr) return PK_ERR_INVALID;
    *dev_ptr = e->tok;
    if (rows) *rows = e->n_utt;
    if (row_ints) *row_ints = 1 + e->cap;
    return PK_OK;
}

// ===================================================================== jobs and the single exchange step
// SURVEY.md section 8e / BASELINE configs[4]: a rank transcribes its block of clips in micro-batches; the token
// rows (len, ids...) of every micro-batch are appended to a device-resident job buffer; ONE ncclAllGather of that
// buffer (on the engine stream, no host synchronisation) assembles the result of all ranks.

pk_status pk_job_begin(pk_engine *e, int64_t rows_local, int32_t world) {
    if (!e || rows_local < 1 || world < 1) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    const size_t W = 1 + (size_t)e->cap;
    if (rows_local * world > e->job_alloc_rows || !e->job_tok) {     // (grow-only; freed with the engine)
        cudaStreamSynchronize(e->stream);
        e->job_tok = e->dalloc<int32_t>((size_t)rows_local * W);
        e->job_all = e->dalloc<int32_t>((size_t)world * rows_local * W);
        if (!e->job_tok || !e->job_all) return e->fail(PK_ERR_CUDA, "cudaMalloc failed (job buffers)");
        if (e->h_job) cudaFreeHost(e->h_job);
        e->h_job_ints = (size_t)world * rows_local * W;
        if (cudaMallocHost(&e->h_job, e->h_job_ints * sizeof(int32_t)) != cudaSuccess) return e->fail(PK_ERR_CUDA, "cudaMallocHost failed (job rows)");
        e->job_alloc_rows = rows_local * world;
    }
    e->job_cap_rows = rows_local;
    e->job_world = world;
    e->job_rows = 0;
    // rows a rank does not fill (a short last block) stay (len = 0)
    cudaError_t ce = cudaMemsetAsync(e->job_tok, 0, (size_t)rows_local * W * sizeof(int32_t), e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_job_begin: ") + cudaGetErrorString(ce));
    return PK_OK;
}

pk_status pk_job_append(pk_engine *e) {
    if (!e || !e->job_tok || e->n_utt <= 0) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (e->job_rows + e->n_utt > e->job_cap_rows) return e->fail(PK_ERR_CAPACITY, "pk_job_append: job buffer full");
    const size_t W = 1 + (size_t)e->cap;
    cudaError_t ce = cudaMemcpyAsync(e->job_tok + (size_t)e->job_rows * W, e->tok, (size_t)e->n_utt * W * sizeof(int32_t),
                                     cudaMemcpyDeviceToDevice, e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_job_append: ") + cudaGetErrorString(ce));
    e->job_rows += e->n_utt;
    return PK_OK;
}

pk_status pk_job_stage_pcm(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt) {
    if (!e || !pcm || !offsets || n_utt < 1) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    const int64_t total = offsets[n_utt] - offsets[0];
    if (total <= 0) return e->fail(PK_ERR_INVALID, "pk_job_stage_pcm: empty job");
    if ((size_t)total + 8 > e->job_pcm_cap) {
        cudaStreamSynchronize(e->stream);
        e->job_pcm = e->dalloc<float>((size_t)total + 8);
        if (!e->job_pcm) return e->fail(PK_ERR_CUDA, "cudaMalloc failed (job PCM)");
        e->job_pcm_cap = (size_t)total + 8;
    }
    e->job_off.assign(n_utt + 1, 0);
    for (int i = 0; i <= n_utt; ++i) e->job_off[i] = offsets[i] - offsets[0];
    cudaError_t ce = cudaMemcpyAsync(e->job_pcm, pcm + offsets[0], (size_t)total * sizeof(float), cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_job_stage_pcm: ") + cudaGetErrorString(ce));
    return PK_OK;
}

pk_status pk_job_select(pk_engine *e, int32_t first, int32_t n_utt) {
    if (!e) return PK_ERR_INVALID;
    if (e->job_off.empty() || first < 0 || n_utt < 1 || (size_t)first + (size_t)n_utt > e->job_off.size() - 1)
        return e->fail(PK_ERR_INVALID, "pk_job_select: range outside the staged job");
    cudaSetDevice(e->device);
    pk_status s = e->set_batch_shapes(nullptr, e->job_off.data() + first, n_utt);
    if (s) return s;
    if ((s = e->upload_shapes())) return s;
    e->pcm_src = e->job_pcm + e->job_off[first];
    e->front_done = false;
    return PK_OK;
}

pk_status pk_nccl_unique_id(void *id128) {
    if (!id128) return PK_ERR_INVALID;
    const NcclApi &n = nccl_api();
    if (!n.ok) {
        g_create_err = n.why;
        return PK_ERR_NCCL;
    }
    NcclApi::UniqueId id;
    if (n.GetUniqueId(&id) != 0) {
        g_create_err = "ncclGetUniqueId failed";
        return PK_ERR_NCCL;
    }
    memcpy(id128, id.internal, sizeof(id.internal));
    return PK_OK;
}

pk_status pk_comm_init_rank(pk_engine *e, const void *id128, int32_t rank, int32_t world) {
    if (!e || !id128 || world < 1 || rank < 0 || rank >= world) return PK_ERR_INVALID;
    const NcclApi &n = nccl_api();
    if (!n.ok) return e->fail(PK_ERR_NCCL, n.why);
    cudaSetDevice(e->device);
    if (e->nccl_comm) {
        n.CommDestroy(e->nccl_comm);
        e->nccl_comm = nullptr;
    }
    NcclApi::UniqueId id;
    memcpy(id.internal, id128, sizeof(id.internal));
    const int rc = n.CommInitRank(&e->nccl_comm, world, id, rank);
    if (rc != 0) return e->fail(PK_ERR_NCCL, std::string("ncclCommInitRank: ") + n.GetErrorString(rc));
    e->nccl_rank = rank;
    e->nccl_world = world;
    return PK_OK;
}

pk_status pk_allgather_tokens(pk_engine *e, void *nccl_comm) {
    if (!e || !e->job_tok) return PK_ERR_INVALID;
    const NcclApi &n = nccl_api();
    if (!n.ok) return e->fail(PK_ERR_NCCL, n.why);
    void *comm = nccl_comm ? nccl_comm : e->nccl_comm;
    if (!comm) return e->fail(PK_ERR_NCCL, "pk_allgather_tokens: no communicator (pk_comm_init_rank or pass an ncclComm_t)");
    cudaSetDevice(e->device);
    const size_t cnt = (size_t)e->job_cap_rows * (1 + (size_t)e->cap);
    const int rc = n.AllGather(e->job_tok, e->job_all, cnt, /*ncclInt32*/ 2, comm, e->stream);
    if (rc != 0) return e->fail(PK_ERR_NCCL, std::string("ncclAllGather: ") + n.GetErrorString(rc));
    ++e->launches;
    return PK_OK;
}

pk_status pk_job_fetch(pk_engine *e, int32_t gathered, int32_t *rows_out, int64_t n_rows, int32_t *row_ints) {
    if (!e || !e->job_tok) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    const size_t W = 1 + (size_t)e->cap;
    if (row_ints) *row_ints = (int32_t)W;
    if (!rows_out) return PK_OK;
    const int64_t have = gathered ? e->job_world * e->job_cap_rows : e->job_cap_rows;
    if (n_rows < 0 || n_rows > have) return e->fail(PK_ERR_CAPACITY, "pk_job_fetch: more rows than the job holds");
    cudaError_t ce = cudaMemcpyAsync(e->h_job, gathered ? e->job_all : e->job_tok, (size_t)n_rows * W * sizeof(int32_t),
                                     cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_job_fetch: ") + cudaGetErrorString(ce));
    memcpy(rows_out, e->h_job, (size_t)n_rows * W * sizeof(int32_t));
    return PK_OK;
}

// ===================================================================== non-16 kHz input (SURVEY.md section 8f row 4)
// Raw samples at `src_rate` go to the device as they are; the polyphase kernel (resample.cu) writes the 16 kHz signal
// straight into the staged PCM buffer, so the resampled audio never exists on the host.
static pk_status stage_raw(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, std::vector<int64_t> &in_off) {
    in_off.assign(n_utt + 1, 0);
    for (int i = 0; i < n_utt; ++i) {
        if (offsets[i + 1] < offsets[i]) return e->fail(PK_ERR_INVALID, "offsets must be non-decreasing");
        in_off[i + 1] = in_off[i] + (offsets[i + 1] - offsets[i]);
    }
    const size_t total = (size_t)in_off[n_utt];
    if (total + 8 > e->d_raw_cap) {
        cudaStreamSynchronize(e->stream);
        e->d_raw = e->dalloc<float>(total + 8);
        if (!e->d_raw) return e->fail(PK_ERR_CUDA, "cudaMalloc failed (raw PCM)");
        e->d_raw_cap = total + 8;
    }
    if (!e->d_raw_off) {
        e->d_raw_off = e->dalloc<int64_t>(2 * ((size_t)e->Bmax + 1));
        if (!e->d_raw_off) return e->fail(PK_ERR_CUDA, "cudaMalloc failed (raw offsets)");
    }
    cudaError_t ce = cudaSuccess;
    for (int i = 0; i < n_utt && ce == cudaSuccess; ++i)      // (pageable or pinned; utterances need not be packed)
        if (in_off[i + 1] > in_off[i])
            ce = cudaMemcpyAsync(e->d_raw + in_off[i], pcm + offsets[i], (size_t)(in_off[i + 1] - in_off[i]) * sizeof(float),
                                 cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess)
        ce = cudaMemcpyAsync(e->d_raw_off, in_off.data(), (size_t)(n_utt + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);   // in_off / pageable sources are the caller's
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("H2D raw pcm: ") + cudaGetErrorString(ce));
    return PK_OK;
}

pk_status pk_stage_pcm_rate(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, int32_t src_rate) {
    if (!e || !pcm || !offsets || src_rate <= 0) return PK_ERR_INVALID;
    if (src_rate == 16000) return pk_stage_pcm(e, pcm, offsets, n_utt);
    cudaSetDevice(e->device);
    if (n_utt < 1 || n_utt > e->Bmax) return e->fail(PK_ERR_CAPACITY, "bad batch size");
    std::vector<int64_t> in_off, out_off(n_utt + 1, 0);
    pk_status s = stage_raw(e, pcm, offsets, n_utt, in_off);
    if (s) return s;
    int64_t max_out = 0;
    for (int i = 0; i < n_utt; ++i) {
        const int64_t m = pk_resample_len(in_off[i + 1] - in_off[i], src_rate, 16000);
        out_off[i + 1] = out_off[i] + m;
        max_out = std::max(max_out, m);
    }
    if ((s = e->set_batch_shapes(nullptr, out_off.data(), n_utt))) return s;     // (length checks at 16 kHz)
    e->pcm_src = nullptr;
    e->pref.valid = false;
    if ((s = e->upload_shapes())) return s;
    if (!launch_resample(e->d_raw, e->d_raw_off, e->d_pcm_off, n_utt, max_out, src_rate, 16000, e->d_pcm, e->stream))
        return e->fail(PK_ERR_CUDA, "resample launch failed");
    ++e->launches;
    e->front_done = false;
    return PK_OK;
}

pk_status pk_resample_batch(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, int32_t src_rate,
                            int32_t dst_rate, float *out, const int64_t *out_offsets) {
    if (!e || !pcm || !offsets || !out || !out_offsets || src_rate <= 0 || dst_rate <= 0 || n_utt < 1) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (n_utt > e->Bmax) return e->fail(PK_ERR_CAPACITY, "bad batch size");
    std::vector<int64_t> in_off, out_off(n_utt + 1, 0);
    pk_status s = stage_raw(e, pcm, offsets, n_utt, in_off);
    if (s) return s;
    int64_t max_out = 0;
    for (int i = 0; i < n_utt; ++i) {
        const int64_t m = pk_resample_len(in_off[i + 1] - in_off[i], src_rate, dst_rate);
        if (out_offsets[i + 1] - out_offsets[i] != m) return e->fail(PK_ERR_INVALID, "pk_resample_batch: out_offsets must be prefix sums of pk_resample_len");
        out_off[i + 1] = out_off[i] + m;
        max_out = std::max(max_out, m);
    }
    const size_t total = (size_t)out_off[n_utt];
    if (total > (size_t)e->Bmax * (size_t)e->cfg.max_samples) return e->fail(PK_ERR_CAPACITY, "pk_resample_batch: output exceeds the PCM workspace");
    cudaError_t ce = cudaMemcpyAsync(e->d_raw_off + e->Bmax + 1, out_off.data(), (size_t)(n_utt + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_resample_batch: ") + cudaGetErrorString(ce));
    float *dst = e->d_pcm_alt;                       // (the second PCM buffer: the staged batch stays intact)
    e->pref.valid = false;
    if (src_rate == dst_rate) {
        ce = cudaMemcpyAsync(dst, e->d_raw, total * sizeof(float), cudaMemcpyDeviceToDevice, e->stream);
    } else if (!launch_resample(e->d_raw, e->d_raw_off, e->d_raw_off + e->Bmax + 1, n_utt, max_out, src_rate, dst_rate, dst, e->stream)) {
        return e->fail(PK_ERR_CUDA, "resample launch failed");
    }
    ++e->launches;
    for (int i = 0; i < n_utt && ce == cudaSuccess; ++i)
        if (out_off[i + 1] > out_off[i])
            ce = cudaMemcpyAsync(out + out_offsets[i], dst + out_off[i], (size_t)(out_off[i + 1] - out_off[i]) * sizeof(float),
                                 cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_resample_batch: ") + cudaGetErrorString(ce));
    return PK_OK;
}

// ===================================================================== phrase boosting (SURVEY.md section 8f row 3)
// ContextTrie (src/phrase_boost.cpp:9-66) built on the host from token-id phrases, flattened to CSR (children of a node
// sorted by token) and uploaded; the decode kernels (ctc.cu: ctc_boosted_decode_kernel, tdt.cu: boost_on) walk it.
pk_status pk_set_boost(pk_engine *e, const int32_t *phrase_ids, const int32_t *phrase_off, int32_t n_phrases, float boost) {
    if (!e || n_phrases < 0 || (n_phrases > 0 && (!phrase_ids || !phrase_off))) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    ++e->boost_gen;
    if (n_phrases == 0) {
        e->boost_on = false;
        return PK_OK;
    }
    std::vector<std::map<int32_t, int32_t>> ch(1);
    for (int32_t p = 0; p < n_phrases; ++p) {
        int32_t node = 0;
        if (phrase_off[p + 1] < phrase_off[p]) return e->fail(PK_ERR_INVALID, "pk_set_boost: phrase_off must be non-decreasing");
        for (int32_t i = phrase_off[p]; i < phrase_off[p + 1]; ++i) {
            auto it = ch[node].find(phrase_ids[i]);
            if (it == ch[node].end()) {
                const int32_t nx = (int32_t)ch.size();
                ch[node][phrase_ids[i]] = nx;
                ch.emplace_back();
                node = nx;
            } else {
                node = it->second;
            }
        }
    }
    std::vector<int32_t> first(ch.size() + 1, 0), tk, cd;
    for (size_t i = 0; i < ch.size(); ++i) {
        for (auto &kv : ch[i]) {
            tk.push_back(kv.first);
            cd.push_back(kv.second);
        }
        first[i + 1] = (int32_t)tk.size();
    }
    if (tk.empty()) {       // only empty phrases
        e->boost_on = false;
        return PK_OK;
    }
    int32_t *d_first = e->upload(first), *d_tok = e->upload(tk), *d_child = e->upload(cd);
    if (!d_first || !d_tok || !d_child) return e->fail(PK_ERR_CUDA, "cudaMalloc failed (trie)");
    e->trie.first = d_first; e->trie.tok = d_tok; e->trie.child = d_child; e->trie.n_nodes = (int32_t)ch.size();
    if (!e->boost_bits) {
        const size_t W = ((size_t)e->cfg.vocab + 31) / 32;
        e->boost_bits = e->dalloc<uint32_t>((size_t)e->Bpad * W);
        e->trie_active = e->dalloc<int32_t>((size_t)e->Bpad * 64);
        e->trie_nact = e->dalloc<int32_t>(e->Bpad);
        if (!e->boost_bits || !e->trie_active || !e->trie_nact) return e->fail(PK_ERR_CUDA, "cudaMalloc failed (boost state)");
    }
    e->boost = boost;
    e->boost_on = true;
    return PK_OK;
}

// Host-only probe of the checkpoint reader (safetensors.cpp): opens `path`, converts tensor `name` to fp32.  No device.
pk_status pk_safetensors_probe(const char *path, const char *name, float *out, int64_t cap, int64_t *numel) {
    if (!path) return PK_ERR_INVALID;
    SafeTensors st;
    std::string err;
    if (!st.open(path, err)) {
        g_create_err = err;
        return PK_ERR_IO;
    }
    if (!name) return PK_OK;
    std::vector<float> v;
    if (!st.read_f32(name, v, -1, err)) {
        g_create_err = err;
        return st.find(name) ? PK_ERR_IO : PK_ERR_MISSING;
    }
    if (numel) *numel = (int64_t)v.size();
    if (out)
        for (int64_t i = 0; i < cap && i < (int64_t)v.size(); ++i) out[i] = v[i];
    return PK_OK;
}

int32_t pk_truncated_count(const pk_engine *e) { return e ? e->truncated : 0; }

pk_status pk_mel(pk_engine *e, const float *pcm, const int64_t *offsets, int32_t n_utt, float *feats_out,
                 int32_t *n_frames_out) {
    pk_status s;
    if ((s = pk_stage_pcm(e, pcm, offsets, n_utt))) return s;
    if (!e->front_done && (s = e->run_mel())) return s;     // (a pinned caller buffer: already run group by group)
    e->front_done = false;
    const size_t n = (size_t)e->frame_off[n_utt] * e->cfg.mel_bins;
    cudaError_t ce = cudaMemcpyAsync(feats_out, e->feats, n * sizeof(float), cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_mel: ") + cudaGetErrorString(ce));
    if (n_frames_out)
        for (int i = 0; i < n_utt; ++i) n_frames_out[i] = e->frame_off[i + 1] - e->frame_off[i];
    return PK_OK;
}

pk_status pk_encode(pk_engine *e, const float *feats, const int32_t *n_frames, int32_t n_utt, float *enc_out,
                    int32_t *enc_lens_out, float *sub_out, float *layers_out) {
    if (!e || !feats || !n_frames || !enc_out) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    pk_status s = e->set_batch_shapes(n_frames, nullptr, n_utt);
    if (s) return s;
    if ((s = e->upload_shapes())) return s;
    const size_t nf = (size_t)e->frame_off[n_utt] * e->cfg.mel_bins;
    cudaError_t ce = cudaMemcpyAsync(e->feats, feats, nf * sizeof(float), cudaMemcpyHostToDevice, e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("H2D feats: ") + cudaGetErrorString(ce));
    if ((s = e->run_conv1())) return s;
    if ((s = e->run_encoder(sub_out, layers_out))) return s;
    ce = cudaMemcpyAsync(enc_out, e->x, (size_t)e->M * e->cfg.d_model * sizeof(float), cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_encode: ") + cudaGetErrorString(ce));
    if (enc_lens_out)
        for (int i = 0; i < n_utt; ++i) enc_lens_out[i] = e->row_off[i + 1] - e->row_off[i];
    return PK_OK;
}

// Stage a host encoder output as the current batch (decode-only entry points).
static pk_status stage_enc(pk_engine *e, const float *enc, const int32_t *enc_lens, int32_t n_utt) {
    if (n_utt <= 0 || n_utt > e->Bmax) return e->fail(PK_ERR_CAPACITY, "bad batch size");
    e->n_utt = n_utt;
    e->row_off.assign(n_utt + 1, 0);
    e->frame_off.assign(n_utt + 1, 0);
    e->s2_off.assign(n_utt + 1, 0);
    e->t2_rows.assign(n_utt + 1, 0);
    e->pcm_off.assign(n_utt + 1, 0);
    e->maxT = 0;
    for (int i = 0; i < n_utt; ++i) {
        if (enc_lens[i] < 1 || enc_lens[i] > e->Tmax) return e->fail(PK_ERR_CAPACITY, "encoder length out of range");
        e->row_off[i + 1] = e->row_off[i] + enc_lens[i];
        e->maxT = std::max(e->maxT, enc_lens[i]);
    }
    e->M = e->row_off[n_utt];
    pk_status s = e->upload_shapes();
    if (s) return s;
    cudaError_t ce = cudaMemcpyAsync(e->x, enc, (size_t)e->M * e->cfg.d_model * sizeof(float), cudaMemcpyHostToDevice, e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("H2D enc: ") + cudaGetErrorString(ce));
    if (e->cfg.math != PK_MATH_FP32) launch_split(e->x, (size_t)e->M * e->cfg.d_model, e->ln, e->stream);
    return PK_OK;
}

pk_status pk_decode(pk_engine *e, const float *enc, const int32_t *enc_lens, int32_t n_utt, pk_decoder dec,
                    pk_tokens *out) {
    if (!e || !enc || !enc_lens) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    pk_status s;
    if ((s = check_decoder(e, dec))) return s;
    if ((s = stage_enc(e, enc, enc_lens, n_utt))) return s;
    if ((s = run_decoder(e, dec))) return s;
    return e->fetch(out);
}

pk_status pk_ctc_logprobs(pk_engine *e, const float *enc, int32_t total_frames, float *logprobs_out) {
    if (!e || !enc || !logprobs_out || total_frames < 1) return PK_ERR_INVALID;
    cudaSetDevice(e->device);
    if (total_frames > e->Tmax) return e->fail(PK_ERR_CAPACITY, "pk_ctc_logprobs: more than Tmax frames");
    pk_status s;
    int32_t len = total_frames;
    if ((s = stage_enc(e, enc, &len, 1))) return s;
    // the [M][V] log-prob matrix lands in the (idle) qkv workspace
    if ((size_t)e->M * e->cfg.vocab > (size_t)e->Bmax * e->Tmax * 3 * e->cfg.d_model)
        return e->fail(PK_ERR_CAPACITY, "pk_ctc_logprobs: workspace too small");
    if ((s = e->run_ctc(e->qkv))) return s;
    cudaError_t ce = cudaMemcpyAsync(logprobs_out, e->qkv, (size_t)e->M * e->cfg.vocab * sizeof(float), cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) return e->fail(PK_ERR_CUDA, std::string("pk_ctc_logprobs: ") + cudaGetErrorString(ce));
    return PK_OK;
}

}  // extern "C"
