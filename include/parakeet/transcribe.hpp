// include/parakeet/transcribe.hpp -- header-only C++ drop-in for the reference's high-level
// API (Frikallo/parakeet.cpp include/parakeet/transcribe.hpp:23-299, config.hpp:9-135,
// timestamp.hpp:11-35) on top of the B200 C-ABI (include/parakeet_b200.h).
//
//   parakeet::Transcriber t("model.safetensors", "vocab.txt");   // transcribe.hpp:59
//   t.to_gpu();                                                    // :68
//   auto r = t.transcribe("audio.wav");                           // :74, Decoder::TDT default
//   auto r2 = t.transcribe(samples, n, parakeet::Decoder::CTC, /*timestamps=*/true);
//
// Same class / method names, argument meaning, defaults and error behaviour
// (std::runtime_error) as the reference.  Differences, all forced by the boundary:
//   * samples are (const float*, size_t) or std::vector<float> instead of axiom::Tensor
//     (an axiom::Tensor overload is enabled when <axiom/axiom.hpp> is on the include path);
//   * the model only ever lives on the CUDA device: to_gpu() is a checked no-op and there
//     is no CPU fallback;
//   * transcribe_batch() is an addition (the reference is batch-1, transcribe.hpp:170-171);
//   * phrase boosting (TranscribeOptions::boost_phrases) runs on the device for both decoders (pk_set_boost);
//   * TDTTranscriber passes blank = vocab-1 like the reference CLI (src/main.cpp:252), not
//     the header's hard-coded 1024 (transcribe.hpp:256-261) which is wrong for 8193 tokens.
// Link with libparakeet_b200.so.
#pragma once

#include <cstdint>
#include <cstring>
#include <algorithm>
#include <fstream>
#include <functional>
#include <iterator>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../parakeet_b200.h"

#if __has_include(<axiom/axiom.hpp>)
#include <axiom/axiom.hpp>
#define PARAKEET_B200_HAS_AXIOM 1
#endif

namespace parakeet {

// ─── configs (config.hpp:9-135) ──────────────────────────────────────────────
struct EncoderConfig {
    int mel_bins = 80, subsampling_factor = 8, subsampling_channels = 256, hidden_size = 1024, num_layers = 24,
        num_heads = 8, ffn_intermediate = 4096, conv_kernel_size = 9;
    float dropout = 0.1f, layer_norm_eps = 1e-5f;
};
struct PredictionConfig { int vocab_size = 1025, pred_hidden = 640, num_lstm_layers = 2; float dropout = 0.1f; };
struct JointConfig { int encoder_hidden = 1024, pred_hidden = 640, joint_hidden = 640, vocab_size = 1025; };
struct TDTConfig { EncoderConfig encoder; PredictionConfig prediction; JointConfig joint; std::vector<int> durations = {0, 1, 2, 3, 4}; };
struct TDTCTCConfig { EncoderConfig encoder; PredictionConfig prediction; JointConfig joint; std::vector<int> durations = {0, 1, 2, 3, 4}; int ctc_vocab_size = 1025; };

inline TDTCTCConfig make_110m_config() {       // config.hpp:77-95
    TDTCTCConfig c;
    c.encoder.hidden_size = 512; c.encoder.num_layers = 17; c.encoder.num_heads = 8; c.encoder.ffn_intermediate = 2048;
    c.prediction.num_lstm_layers = 1; c.joint.encoder_hidden = 512;
    return c;
}
inline TDTConfig make_tdt_600m_config() {      // config.hpp:98-116
    TDTConfig c;
    c.encoder.mel_bins = 128;
    c.prediction.vocab_size = 8193; c.joint.vocab_size = 8193;
    return c;
}
struct RNNTConfig { EncoderConfig encoder; PredictionConfig prediction; JointConfig joint; };
inline RNNTConfig make_rnnt_600m_config() { return RNNTConfig{}; }   // config.hpp:119-135: the defaults above

// ─── timestamps (timestamp.hpp:11-35) ────────────────────────────────────────
struct TimestampedToken { int token_id; int start_frame; int end_frame; float confidence = 1.0f; };
struct WordTimestamp { std::string word; float start; float end; float confidence = 1.0f; };
constexpr float FRAME_DURATION_S = 0.08f;
inline float frame_to_seconds(int frame) { return static_cast<float>(frame) * FRAME_DURATION_S; }

// ─── result / options (transcribe.hpp:23-43) ─────────────────────────────────
struct TranscribeResult {
    std::string text;
    std::vector<int> token_ids;
    std::vector<TimestampedToken> timestamped_tokens;
    std::vector<WordTimestamp> word_timestamps;
};
enum class Decoder { CTC, TDT };
struct TranscribeOptions {
    Decoder decoder = Decoder::TDT;
    bool timestamps = false;
    std::vector<std::string> boost_phrases;
    float boost_score = 5.0f;
};

// ─── Tokenizer (vocab.hpp) over the C-ABI host helpers ───────────────────────
class Tokenizer {
  public:
    Tokenizer() = default;
    Tokenizer(const Tokenizer &) = delete;
    Tokenizer &operator=(const Tokenizer &) = delete;
    ~Tokenizer() { pk_vocab_free(v_); }
    void load(const std::string &vocab_path) {
        pk_vocab_free(v_);
        v_ = nullptr;
        if (pk_vocab_load(vocab_path.c_str(), &v_) != PK_OK) throw std::runtime_error("Cannot open vocab file: " + vocab_path);
    }
    bool loaded() const { return v_ && pk_vocab_size(v_) > 0; }
    size_t vocab_size() const { return loaded() ? (size_t)pk_vocab_size(v_) + 1 : 0; }   // +1 blank, like the reference
    std::string decode(const std::vector<int> &ids) const {
        std::vector<int32_t> a(ids.begin(), ids.end());
        std::string buf(2 + ((size_t)pk_vocab_max_piece_bytes(v_) + 1) * std::max<size_t>(a.size(), 1), '\0');
        int n = pk_detokenize(v_, a.data(), (int32_t)a.size(), &buf[0], (int32_t)buf.size());
        buf.resize(n < 0 ? 0 : std::min<size_t>((size_t)n, buf.size() - 1));
        return buf;
    }
    // Tokenizer::encode (vocab.cpp:76-117)
    std::vector<int> encode(const std::string &text) const {
        std::vector<int32_t> a(2 * text.size() + 8);
        int n = pk_tokenize(v_, text.c_str(), a.data(), (int32_t)a.size());
        return std::vector<int>(a.begin(), a.begin() + (n < 0 ? 0 : n));
    }
    std::vector<WordTimestamp> group(const std::vector<TimestampedToken> &t) const {
        const int n = (int)t.size();
        std::vector<int32_t> id(n), st(n), en(n);
        std::vector<float> cf(n), ws(n + 1), we(n + 1), wc(n + 1);
        for (int i = 0; i < n; ++i) { id[i] = t[i].token_id; st[i] = t[i].start_frame; en[i] = t[i].end_frame; cf[i] = t[i].confidence; }
        std::string buf(2 + ((size_t)pk_vocab_max_piece_bytes(v_) + 2) * std::max<size_t>((size_t)n, 1), '\0');
        int k = pk_group_words(v_, id.data(), st.data(), en.data(), cf.data(), n, &buf[0], (int32_t)buf.size(), ws.data(), we.data(), wc.data());
        std::vector<WordTimestamp> out;
        size_t pos = 0;
        for (int i = 0; i < k; ++i) {
            size_t e = buf.find('\n', pos);
            out.push_back({buf.substr(pos, e - pos), ws[i], we[i], wc[i]});
            pos = e + 1;
        }
        return out;
    }
  private:
    pk_vocab *v_ = nullptr;
};

// ─── phrase boosting (phrase_boost.hpp:22-66, CTC variants :70-176), host side ──
class ContextTrie {
  public:
    void insert(const std::vector<int> &token_ids) {
        if (token_ids.empty()) return;
        ids_.insert(ids_.end(), token_ids.begin(), token_ids.end());
        off_.push_back((int32_t)ids_.size());
    }
    void build(const std::vector<std::string> &phrases, const Tokenizer &tokenizer) {
        for (const auto &p : phrases) insert(tokenizer.encode(p));
    }
    bool empty() const { return off_.size() <= 1; }
    const std::vector<int32_t> &ids() const { return ids_; }
    const std::vector<int32_t> &offsets() const { return off_; }
  private:
    std::vector<int32_t> ids_, off_{0};
};

// log_probs: one utterance, (n_frames, vocab) row-major (e.g. from pk_ctc_logprobs)
inline std::vector<TimestampedToken> ctc_greedy_decode_with_timestamps_boosted(const float *log_probs, int n_frames, int vocab,
                                                                               const ContextTrie &trie, float boost_score = 5.0f,
                                                                               int blank_id = 1024) {
    std::vector<int32_t> id(n_frames + 1), st(n_frames + 1), en(n_frames + 1);
    std::vector<float> cf(n_frames + 1);
    static const int32_t none = 0;
    const int n = pk_ctc_decode_boosted(log_probs, n_frames, vocab, blank_id, trie.ids().empty() ? &none : trie.ids().data(),
                                        trie.offsets().data(), (int32_t)trie.offsets().size() - 1, boost_score, id.data(),
                                        st.data(), en.data(), cf.data(), n_frames + 1);
    if (n < 0) throw std::runtime_error("ctc_greedy_decode_boosted: invalid arguments");
    std::vector<TimestampedToken> out;
    for (int i = 0; i < n; ++i) out.push_back({id[i], st[i], en[i], cf[i]});
    return out;
}
inline std::vector<int> ctc_greedy_decode_boosted(const float *log_probs, int n_frames, int vocab, const ContextTrie &trie,
                                                  float boost_score = 5.0f, int blank_id = 1024) {
    std::vector<int> ids;
    for (const auto &t : ctc_greedy_decode_with_timestamps_boosted(log_probs, n_frames, vocab, trie, boost_score, blank_id))
        ids.push_back(t.token_id);
    return ids;
}

// ─── minimal read_audio (audio_io.hpp): mono-mixed PCM16 / float32 WAV ───────
// read_audio_native keeps the file's own sample rate (Transcriber::transcribe(path) converts on the DEVICE,
// pk_stage_pcm_rate); read_audio resamples to 16 kHz on the host like the reference's (audio_io.cpp:227-232).
inline std::vector<float> read_audio_native(const std::string &path, int &sample_rate) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error("Cannot open audio file: " + path);
    std::vector<char> d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    if (d.size() < 12 || std::memcmp(d.data(), "RIFF", 4) || std::memcmp(d.data() + 8, "WAVE", 4))
        throw std::runtime_error("Unsupported audio format (RIFF/WAVE only on this path): " + path);
    uint16_t tag = 0, ch = 0, bits = 0;
    uint32_t sr = 0;
    const char *pcm = nullptr;
    uint32_t pcm_bytes = 0;
    for (size_t pos = 12; pos + 8 <= d.size();) {
        uint32_t sz;
        std::memcpy(&sz, d.data() + pos + 4, 4);
        if (!std::memcmp(d.data() + pos, "fmt ", 4) && sz >= 16) {
            std::memcpy(&tag, d.data() + pos + 8, 2); std::memcpy(&ch, d.data() + pos + 10, 2);
            std::memcpy(&sr, d.data() + pos + 12, 4); std::memcpy(&bits, d.data() + pos + 22, 2);
        } else if (!std::memcmp(d.data() + pos, "data", 4)) {
            pcm = d.data() + pos + 8;
            pcm_bytes = (uint32_t)std::min<size_t>(sz, d.size() - pos - 8);
        }
        pos += 8 + sz + (sz & 1);
    }
    if (!pcm || !ch) throw std::runtime_error("malformed WAV: " + path);
    std::vector<float> mono;
    if (tag == 1 && bits == 16) {
        const size_t n = pcm_bytes / 2 / ch;
        mono.resize(n);
        for (size_t i = 0; i < n; ++i) {
            float s = 0.f;
            for (int c = 0; c < ch; ++c) { int16_t v; std::memcpy(&v, pcm + 2 * (i * ch + c), 2); s += (float)v / 32768.0f; }
            mono[i] = s / (float)ch;
        }
    } else if (tag == 3 && bits == 32) {
        const size_t n = pcm_bytes / 4 / ch;
        mono.resize(n);
        for (size_t i = 0; i < n; ++i) {
            float s = 0.f;
            for (int c = 0; c < ch; ++c) { float v; std::memcpy(&v, pcm + 4 * (i * ch + c), 4); s += v; }
            mono[i] = s / (float)ch;
        }
    } else {
        throw std::runtime_error("unsupported WAV encoding: " + path);
    }
    sample_rate = (int)sr;
    return mono;
}
inline std::vector<float> read_audio(const std::string &path) {
    int sr = 16000;
    auto mono = read_audio_native(path, sr);
    if (sr != 16000) {   // read_audio resamples to the target rate (audio_io.cpp:123-195, :227-232)
        std::vector<float> r((size_t)std::max<int64_t>(pk_resample_len((int64_t)mono.size(), (int32_t)sr, 16000), 0));
        pk_resample(mono.data(), (int64_t)mono.size(), (int32_t)sr, 16000, r.data(), (int64_t)r.size());
        return r;
    }
    return mono;
}

// parakeet::resample (audio_io.hpp:41)
inline std::vector<float> resample(const std::vector<float> &samples, int src_rate, int dst_rate) {
    std::vector<float> r((size_t)std::max<int64_t>(pk_resample_len((int64_t)samples.size(), src_rate, dst_rate), 0));
    pk_resample(samples.data(), (int64_t)samples.size(), src_rate, dst_rate, r.data(), (int64_t)r.size());
    return r;
}

namespace detail {

class EngineHolder {
  public:
    EngineHolder(const pk_config &cfg, const std::string &weights, int device) : cfg_(cfg) {
        if (pk_engine_create(&cfg, weights.c_str(), device, &e_) != PK_OK)
            throw std::runtime_error(std::string("parakeet_b200: ") + pk_last_error(nullptr));
        const int32_t tmax = pk_encoder_frames(pk_mel_frames(cfg.max_samples));
        cap_ = cfg.n_durations == 0 ? tmax * cfg.max_symbols : 2 * tmax + 8;     // (RNNT: up to max_symbols per frame)
    }
    EngineHolder(const EngineHolder &) = delete;
    EngineHolder &operator=(const EngineHolder &) = delete;
    ~EngineHolder() { pk_engine_destroy(e_); }

    std::vector<std::vector<TimestampedToken>> run(const std::vector<const float *> &pcm, const std::vector<size_t> &n, pk_decoder dec,
                                                   int sample_rate = 16000) {
        const int B = (int)pcm.size();
        std::vector<int64_t> off(B + 1, 0);
        for (int i = 0; i < B; ++i) off[i + 1] = off[i] + (int64_t)n[i];
        std::vector<float> buf((size_t)off[B]);
        for (int i = 0; i < B; ++i) std::memcpy(buf.data() + off[i], pcm[i], n[i] * sizeof(float));
        std::vector<int32_t> ids((size_t)B * cap_), st((size_t)B * cap_), en((size_t)B * cap_), len(B);
        std::vector<float> cf((size_t)B * cap_);
        pk_tokens t{cap_, ids.data(), st.data(), en.data(), cf.data(), len.data()};
        // 16 kHz: the blocking whole-path call; any other rate: raw samples to the device, polyphase conversion there
        const bool ok = sample_rate == 16000
                            ? pk_transcribe_batch(e_, buf.data(), off.data(), B, dec, &t) == PK_OK
                            : (pk_stage_pcm_rate(e_, buf.data(), off.data(), B, sample_rate) == PK_OK && pk_run_staged(e_, dec) == PK_OK &&
                               pk_fetch_tokens(e_, &t) == PK_OK);
        if (!ok) throw std::runtime_error(std::string("parakeet_b200: ") + pk_last_error(e_));
        std::vector<std::vector<TimestampedToken>> out(B);
        for (int b = 0; b < B; ++b)
            for (int i = 0; i < len[b]; ++i)
                out[b].push_back({ids[(size_t)b * cap_ + i], st[(size_t)b * cap_ + i], en[(size_t)b * cap_ + i], cf[(size_t)b * cap_ + i]});
        return out;
    }
    const pk_config &cfg() const { return cfg_; }
    pk_engine *raw() { return e_; }

  private:
    pk_config cfg_;
    pk_engine *e_ = nullptr;
    int32_t cap_ = 0;
};

inline void fill(pk_config &c, const EncoderConfig &e, const PredictionConfig &p, const JointConfig &j, const std::vector<int> &dur) {
    c.mel_bins = e.mel_bins; c.sub_channels = e.subsampling_channels; c.d_model = e.hidden_size; c.n_layers = e.num_layers;
    c.n_heads = e.num_heads; c.ff = e.ffn_intermediate; c.conv_kernel = e.conv_kernel_size;
    c.vocab = j.vocab_size; c.pred_hidden = p.pred_hidden; c.lstm_layers = p.num_lstm_layers; c.joint_hidden = j.joint_hidden;
    c.n_durations = (int)dur.size();
    for (size_t i = 0; i < dur.size() && i < 8; ++i) c.durations[i] = dur[i];
}

template <class Derived>
class TranscriberBase {
  public:
    void to_gpu() {}   // the reference moves weights to Metal here (transcribe.hpp:68-71); we are always on the device

    TranscribeResult transcribe(const std::string &audio_path, const TranscribeOptions &opts) {
        int sr = 16000;
        auto s = read_audio_native(audio_path, sr);
        return transcribe(s.data(), s.size(), opts, sr);
    }
    TranscribeResult transcribe(const std::vector<float> &samples, const TranscribeOptions &opts) { return transcribe(samples.data(), samples.size(), opts); }
    TranscribeResult transcribe(const float *samples, size_t n, const TranscribeOptions &opts, int sample_rate = 16000) {
        // phrase boosting (transcribe.hpp:110-137, :158-165): the ContextTrie and the boosted decode live on the device
        struct BoostGuard {
            pk_engine *e; bool on;
            ~BoostGuard() { if (on) pk_set_boost(e, nullptr, nullptr, 0, 0.f); }
        } guard{eng_->raw(), false};
        if (!opts.boost_phrases.empty() && tokenizer_.loaded()) {
            ContextTrie trie;
            trie.build(opts.boost_phrases, tokenizer_);
            if (!trie.empty()) {
                if (pk_set_boost(eng_->raw(), trie.ids().data(), trie.offsets().data(), (int32_t)trie.offsets().size() - 1, opts.boost_score) != PK_OK)
                    throw std::runtime_error(std::string("parakeet_b200: ") + pk_last_error(eng_->raw()));
                guard.on = true;
            }
        }
        auto toks = eng_->run({samples}, {n}, self().pick(opts.decoder), sample_rate)[0];
        return finish(toks, opts.timestamps);
    }
    // Not in the reference (batch-1 only): one call for many utterances.
    std::vector<TranscribeResult> transcribe_batch(const std::vector<std::vector<float>> &utts, Decoder decoder = Decoder::TDT, bool timestamps = false) {
        std::vector<TranscribeResult> out;
        const size_t B = (size_t)eng_->cfg().max_batch;
        for (size_t i = 0; i < utts.size(); i += B) {
            std::vector<const float *> p;
            std::vector<size_t> n;
            for (size_t k = i; k < utts.size() && k < i + B; ++k) { p.push_back(utts[k].data()); n.push_back(utts[k].size()); }
            for (auto &toks : eng_->run(p, n, self().pick(decoder))) out.push_back(finish(toks, timestamps));
        }
        return out;
    }
#ifdef PARAKEET_B200_HAS_AXIOM
    TranscribeResult transcribe(const axiom::Tensor &samples, const TranscribeOptions &opts) {
        auto c = samples.cpu().ascontiguousarray();
        return transcribe(c.template typed_data<float>(), c.size(), opts);
    }
#endif
    const Tokenizer &tokenizer() const { return tokenizer_; }
    pk_engine *engine() { return eng_->raw(); }

  protected:
    TranscribeResult finish(const std::vector<TimestampedToken> &toks, bool timestamps) {
        TranscribeResult r;
        for (auto &t : toks) r.token_ids.push_back(t.token_id);
        if (timestamps) r.timestamped_tokens = toks;
        if (tokenizer_.loaded()) {
            r.text = tokenizer_.decode(r.token_ids);
            if (timestamps) r.word_timestamps = tokenizer_.group(toks);
        }
        return r;
    }
    Derived &self() { return static_cast<Derived &>(*this); }
    std::unique_ptr<EngineHolder> eng_;
    Tokenizer tokenizer_;
};

}  // namespace detail

/// parakeet::Transcriber (reference transcribe.hpp:55-190): TDT-CTC hybrid, 110M preset by default.
class Transcriber : public detail::TranscriberBase<Transcriber> {
  public:
    Transcriber(const std::string &weights_path, const std::string &vocab_path, const TDTCTCConfig &config = make_110m_config(),
                int device = 0, int max_batch = 64, int max_samples = 30 * 16000) {
        pk_config c;
        pk_config_110m(&c);
        detail::fill(c, config.encoder, config.prediction, config.joint, config.durations);
        c.has_ctc = 1; c.joint_prefix_tdt = 1; c.max_batch = max_batch; c.max_samples = max_samples;
        eng_ = std::make_unique<detail::EngineHolder>(c, weights_path, device);
        tokenizer_.load(vocab_path);
    }
    using TranscriberBase::transcribe;
    TranscribeResult transcribe(const std::string &audio_path, Decoder decoder = Decoder::TDT, bool timestamps = false) {
        TranscribeOptions o; o.decoder = decoder; o.timestamps = timestamps;
        return TranscriberBase::transcribe(audio_path, o);
    }
    TranscribeResult transcribe(const std::vector<float> &samples, Decoder decoder = Decoder::TDT, bool timestamps = false) {
        TranscribeOptions o; o.decoder = decoder; o.timestamps = timestamps;
        return TranscriberBase::transcribe(samples, o);
    }
    TranscribeResult transcribe(const float *samples, size_t n, Decoder decoder = Decoder::TDT, bool timestamps = false) {
        TranscribeOptions o; o.decoder = decoder; o.timestamps = timestamps;
        return TranscriberBase::transcribe(samples, n, o);
    }
    pk_decoder pick(Decoder d) const { return d == Decoder::CTC ? PK_DECODER_CTC : PK_DECODER_TDT; }
};

/// parakeet::TDTTranscriber (reference transcribe.hpp:200-299): TDT-only models (600M multilingual).
class TDTTranscriber : public detail::TranscriberBase<TDTTranscriber> {
  public:
    TDTTranscriber(const std::string &weights_path, const std::string &vocab_path, const TDTConfig &config = make_tdt_600m_config(),
                   int device = 0, int max_batch = 16, int max_samples = 30 * 16000) {
        pk_config c;
        pk_config_tdt_600m(&c);
        detail::fill(c, config.encoder, config.prediction, config.joint, config.durations);
        c.has_ctc = 0; c.joint_prefix_tdt = 0; c.max_batch = max_batch; c.max_samples = max_samples;
        eng_ = std::make_unique<detail::EngineHolder>(c, weights_path, device);
        tokenizer_.load(vocab_path);
    }
    using TranscriberBase::transcribe;
    TranscribeResult transcribe(const std::string &audio_path, bool timestamps = false) {
        TranscribeOptions o; o.timestamps = timestamps;
        return TranscriberBase::transcribe(audio_path, o);
    }
    TranscribeResult transcribe(const std::vector<float> &samples, bool timestamps = false) {
        TranscribeOptions o; o.timestamps = timestamps;
        return TranscriberBase::transcribe(samples, o);
    }
    pk_decoder pick(Decoder) const { return PK_DECODER_TDT; }
};

/// RNNT models (rnnt-600m, reference config.hpp:119-135), with TDTTranscriber's surface.  The reference has no such
/// class: its CLI does the same inline in run_rnnt_600m (src/main.cpp:296-360) -- preprocess_audio, the encoder, then
/// rnnt_greedy_decode(_with_timestamps) with blank = vocab - 1.  Phrase boosting is not available for RNNT decoding.
class RNNTTranscriber : public detail::TranscriberBase<RNNTTranscriber> {
  public:
    RNNTTranscriber(const std::string &weights_path, const std::string &vocab_path, const RNNTConfig &config = make_rnnt_600m_config(),
                    int device = 0, int max_batch = 16, int max_samples = 30 * 16000) {
        pk_config c;
        pk_config_rnnt_600m(&c);
        detail::fill(c, config.encoder, config.prediction, config.joint, {});
        c.max_batch = max_batch; c.max_samples = max_samples;
        eng_ = std::make_unique<detail::EngineHolder>(c, weights_path, device);
        tokenizer_.load(vocab_path);
    }
    using TranscriberBase::transcribe;
    TranscribeResult transcribe(const std::string &audio_path, bool timestamps = false) {
        TranscribeOptions o; o.timestamps = timestamps;
        return TranscriberBase::transcribe(audio_path, o);
    }
    TranscribeResult transcribe(const std::vector<float> &samples, bool timestamps = false) {
        TranscribeOptions o; o.timestamps = timestamps;
        return TranscriberBase::transcribe(samples, o);
    }
    pk_decoder pick(Decoder) const { return PK_DECODER_RNNT; }
};


// ─── streaming (reference include/parakeet/eou.hpp:25-141, streaming_encoder.hpp:18-24) ─────────────────────────
struct StreamingEncoderConfig : EncoderConfig {
    int att_context_left = 70, att_context_right = 0, chunk_size = 20;
    bool xscaling = false;
};
struct EOUConfig {
    StreamingEncoderConfig encoder;
    PredictionConfig prediction;
    JointConfig joint;
    std::vector<int> durations = {0, 1, 2, 3, 4};
    int eou_token_id = -1;
    int ctc_vocab_size = 1025;
};
inline EOUConfig make_eou_120m_config() {      // eou.hpp:32-55
    EOUConfig c;
    c.encoder.hidden_size = 512; c.encoder.num_layers = 17; c.encoder.num_heads = 8; c.encoder.ffn_intermediate = 2048;
    c.encoder.subsampling_channels = 256; c.encoder.conv_kernel_size = 9; c.encoder.att_context_left = 70; c.encoder.att_context_right = 1;
    c.prediction.vocab_size = 1025; c.prediction.pred_hidden = 640; c.prediction.num_lstm_layers = 1;
    c.joint.encoder_hidden = 512; c.joint.pred_hidden = 640; c.joint.joint_hidden = 640; c.joint.vocab_size = 1025;
    c.eou_token_id = 1024;
    return c;
}

/// parakeet::StreamingTranscriber (reference eou.hpp:101-141, src/eou.cpp:100-155): chunk-by-chunk transcription with
/// carried state.  One object = one stream on the device (pk_stream_open with a single stream); for many concurrent
/// streams that share every weight read use StreamingBatch below -- the reference has no counterpart to it.
class StreamingBatch {
  public:
    StreamingBatch(const std::string &weights_path, const std::string &vocab_path, int n_streams, const EOUConfig &config = make_eou_120m_config(),
                   int device = 0, int max_chunk_samples = 5120)
        : n_(n_streams), tokens_(n_streams), stamped_(n_streams) {
        if (config.encoder.xscaling) throw std::runtime_error("StreamingBatch: xscaling is not supported on the B200 path");
        pk_config c;
        pk_config_110m(&c);
        detail::fill(c, config.encoder, config.prediction, config.joint, config.durations);
        c.has_ctc = 0; c.joint_prefix_tdt = 0;                 // ParakeetEOU registers "joint_" (eou.cpp:9-13)
        c.max_batch = std::max(n_streams, 8);
        c.max_samples = 102400;                                 // 6.4 s: encoder-frame capacity >= left context + frames per chunk
        eng_ = std::make_unique<detail::EngineHolder>(c, weights_path, device);
        if (pk_stream_open(eng_->raw(), n_streams, max_chunk_samples, config.encoder.att_context_left, config.encoder.att_context_right) != PK_OK)
            throw std::runtime_error(std::string("parakeet_b200: ") + pk_last_error(eng_->raw()));
        if (!vocab_path.empty()) tokenizer_.load(vocab_path);
        cap_ = 2 * pk_encoder_frames(pk_mel_frames(c.max_samples)) + 8;
    }
    /// One step: stream s receives chunks[s] (may be empty).  Returns the text each stream produced in this step.
    std::vector<std::string> transcribe_chunks(const std::vector<std::vector<float>> &chunks) {
        if ((int)chunks.size() != n_) throw std::runtime_error("StreamingBatch: one chunk per stream expected");
        std::vector<int64_t> off(n_ + 1, 0);
        for (int i = 0; i < n_; ++i) off[i + 1] = off[i] + (int64_t)chunks[i].size();
        std::vector<float> buf((size_t)off[n_] + 1);
        for (int i = 0; i < n_; ++i) std::memcpy(buf.data() + off[i], chunks[i].data(), chunks[i].size() * sizeof(float));
        std::vector<int32_t> ids((size_t)n_ * cap_), st((size_t)n_ * cap_), en((size_t)n_ * cap_), len(n_);
        std::vector<float> cf((size_t)n_ * cap_);
        pk_tokens t{cap_, ids.data(), st.data(), en.data(), cf.data(), len.data()};
        if (pk_stream_step(eng_->raw(), buf.data(), off.data(), &t, nullptr, nullptr, nullptr, nullptr) != PK_OK)
            throw std::runtime_error(std::string("parakeet_b200: ") + pk_last_error(eng_->raw()));
        std::vector<std::string> out(n_);
        for (int s = 0; s < n_; ++s) {
            std::vector<int> fresh;
            for (int i = 0; i < len[s]; ++i) {
                const size_t k = (size_t)s * cap_ + i;
                fresh.push_back(ids[k]);
                tokens_[s].push_back(ids[k]);
                stamped_[s].push_back({ids[k], st[k], en[k], cf[k]});
            }
            if (!fresh.empty() && tokenizer_.loaded()) out[s] = tokenizer_.decode(fresh);
        }
        return out;
    }
    void reset(int stream = -1) {
        if (pk_stream_reset(eng_->raw(), stream) != PK_OK) throw std::runtime_error(std::string("parakeet_b200: ") + pk_last_error(eng_->raw()));
        for (int s = 0; s < n_; ++s)
            if (stream < 0 || s == stream) { tokens_[s].clear(); stamped_[s].clear(); }
    }
    std::string get_text(int stream = 0) const { return (tokenizer_.loaded() && !tokens_[stream].empty()) ? tokenizer_.decode(tokens_[stream]) : std::string(); }
    const std::vector<TimestampedToken> &get_timestamped_tokens(int stream = 0) const { return stamped_[stream]; }
    const std::vector<int> &get_tokens(int stream = 0) const { return tokens_[stream]; }
    const Tokenizer &tokenizer() const { return tokenizer_; }
    int streams() const { return n_; }

  private:
    int n_;
    int32_t cap_ = 0;
    std::unique_ptr<detail::EngineHolder> eng_;
    Tokenizer tokenizer_;
    std::vector<std::vector<int>> tokens_;
    std::vector<std::vector<TimestampedToken>> stamped_;
};

class StreamingTranscriber {
  public:
    using PartialResultCallback = std::function<void(const std::string &partial)>;
    StreamingTranscriber(const std::string &weights_path, const std::string &vocab_path, const EOUConfig &config = make_eou_120m_config(), int device = 0)
        : batch_(weights_path, vocab_path, 1, config, device) {}
    void to_gpu() {}                                           // always on the device
    std::string transcribe_chunk(const float *data, size_t num_samples) {
        auto text = batch_.transcribe_chunks({std::vector<float>(data, data + num_samples)})[0];
        if (!text.empty() && cb_) cb_(text);                  // eou.cpp:134-139
        return text;
    }
    std::string transcribe_chunk(const std::vector<float> &samples) { return transcribe_chunk(samples.data(), samples.size()); }
    std::string transcribe_chunk(const int16_t *data, size_t num_samples) {   // eou.hpp:123-129
        std::vector<float> f(num_samples);
        for (size_t i = 0; i < num_samples; ++i) f[i] = static_cast<float>(data[i]) / 32768.0f;
        return transcribe_chunk(f.data(), f.size());
    }
    void reset() { batch_.reset(-1); }
    void set_partial_callback(PartialResultCallback cb) { cb_ = std::move(cb); }
    std::string get_text() const { return batch_.get_text(0); }
    const std::vector<TimestampedToken> &get_timestamped_tokens() const { return batch_.get_timestamped_tokens(0); }
    const Tokenizer &tokenizer() const { return batch_.tokenizer(); }

  private:
    StreamingBatch batch_;
    PartialResultCallback cb_;
};

}  // namespace parakeet
