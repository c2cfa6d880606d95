// tests/golden/ref_rnnt_harness.cpp -- TEST INFRASTRUCTURE, not product code.
//
// A thin C-ABI around the UNMODIFIED reference's RNNT model, compiled by make_golden_rnnt.py against the reference
// library oracle/_ref/libpkref.so (oracle/Makefile) to record tests/golden/golden_rnnt_v1.npz.  It only calls:
//   ParakeetRNNT(make_rnnt_600m_config())             include/parakeet/config.hpp:119-135, src/rnnt.cpp:46-52
//   FastConformerEncoder::forward                      src/encoder.cpp:253-271
//   rnnt_greedy_decode(_with_timestamps)               src/rnnt.cpp:56-177

#include <cstdint>
#include <cstring>
#include <memory>
#include <string>

#include <axiom/axiom.hpp>
#include <axiom/io/safetensors.hpp>

#include "parakeet/config.hpp"
#include "parakeet/rnnt.hpp"

using namespace parakeet;
using axiom::Shape;
using axiom::Tensor;

namespace {

struct RefRNNT {
    RNNTConfig cfg;
    std::unique_ptr<ParakeetRNNT> model;
};

thread_local std::string g_err;

}  // namespace

extern "C" {

const char *pkref_rnnt_last_error() { return g_err.c_str(); }

// preset 2 = make_rnnt_600m_config(); custom != 0 replaces the dimensions (test-only tiny shapes).
void *pkref_rnnt_load(const char *weights_path, int custom, int mel, int sub_ch, int d, int layers, int heads, int ff,
                      int vocab, int pred_hidden, int lstm_layers, int joint_hidden) {
    try {
        auto m = std::make_unique<RefRNNT>();
        m->cfg = make_rnnt_600m_config();
        if (custom) {
            auto &c = m->cfg;
            c.encoder.mel_bins = mel;
            c.encoder.subsampling_channels = sub_ch;
            c.encoder.hidden_size = d;
            c.encoder.num_layers = layers;
            c.encoder.num_heads = heads;
            c.encoder.ffn_intermediate = ff;
            c.prediction.vocab_size = vocab;
            c.prediction.pred_hidden = pred_hidden;
            c.prediction.num_lstm_layers = lstm_layers;
            c.joint.encoder_hidden = d;
            c.joint.pred_hidden = pred_hidden;
            c.joint.joint_hidden = joint_hidden;
            c.joint.vocab_size = vocab;
        }
        m->model = std::make_unique<ParakeetRNNT>(m->cfg);
        auto weights = axiom::io::safetensors::load(weights_path);
        m->model->load_state_dict(weights, "", false);
        return m.release();
    } catch (const std::exception &e) {
        g_err = e.what();
        return nullptr;
    }
}

void pkref_rnnt_free(void *h) { delete static_cast<RefRNNT *>(h); }

// feats (n_frames, n_mels) -> encoder output (T', d).  Returns T' or -1.
int pkref_rnnt_encode(void *h, const float *feats, int n_frames, int n_mels, float *out) {
    try {
        auto *m = static_cast<RefRNNT *>(h);
        auto y = m->model->encoder()(Tensor::from_data(feats, Shape{1, (size_t)n_frames, (size_t)n_mels}, true));
        auto c = y.cpu().ascontiguousarray();
        std::memcpy(out, c.typed_data<float>(), c.size() * sizeof(float));
        return (int)y.shape()[1];
    } catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

// enc (T, d) -> both reference decoders with blank = vocab - 1 (the CLI's value, main.cpp:296-360).  The timestamped
// result goes to ids/start/end/conf, the id-only result to ids_plain (cap entries each).  Returns the timestamped
// token count (*n_plain: the id-only count), or -1.
int pkref_rnnt_greedy(void *h, const float *enc, int T, int d, int cap, int *ids, int *start, int *end, float *conf,
                      int *ids_plain, int *n_plain) {
    try {
        auto *m = static_cast<RefRNNT *>(h);
        auto e = Tensor::from_data(enc, Shape{1, (size_t)T, (size_t)d}, true);
        const int blank = m->cfg.joint.vocab_size - 1;
        auto r = rnnt_greedy_decode_with_timestamps(*m->model, e, blank);
        auto r2 = rnnt_greedy_decode(*m->model, e, blank);
        const int n = (int)r[0].size();
        *n_plain = (int)r2[0].size();
        for (int i = 0; i < n && i < cap; ++i) {
            ids[i] = r[0][i].token_id;
            start[i] = r[0][i].start_frame;
            end[i] = r[0][i].end_frame;
            conf[i] = r[0][i].confidence;
        }
        for (int i = 0; i < *n_plain && i < cap; ++i) ids_plain[i] = r2[0][i];
        return n;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

}  // extern "C"
