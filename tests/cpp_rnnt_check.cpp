// RNNTTranscriber through the header-only shim (include/parakeet/transcribe.hpp), as a C++ user calls it.
//   cpp_rnnt_check <weights.safetensors> <vocab.txt> <samples.f32>     (tiny RNNT shape of tests/test_rnnt.py)
// Prints "TOK id:start:end ..." and "TEXT <text>".
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <vector>

#include "parakeet/transcribe.hpp"

int main(int argc, char **argv) {
    if (argc < 4) return 2;
    std::ifstream f(argv[3], std::ios::binary);
    std::vector<char> raw((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    std::vector<float> pcm(raw.size() / sizeof(float));
    std::memcpy(pcm.data(), raw.data(), pcm.size() * sizeof(float));
    parakeet::RNNTConfig cfg = parakeet::make_rnnt_600m_config();
    cfg.encoder.subsampling_channels = 64; cfg.encoder.hidden_size = 128; cfg.encoder.num_layers = 2;
    cfg.encoder.num_heads = 2; cfg.encoder.ffn_intermediate = 256;
    cfg.prediction.vocab_size = 33; cfg.prediction.pred_hidden = 64; cfg.prediction.num_lstm_layers = 2;
    cfg.joint.encoder_hidden = 128; cfg.joint.pred_hidden = 64; cfg.joint.joint_hidden = 64; cfg.joint.vocab_size = 33;
    parakeet::RNNTTranscriber t(argv[1], argv[2], cfg, 0, 4, 64000);
    t.to_gpu();
    auto r = t.transcribe(pcm, /*timestamps=*/true);
    std::cout << "TOK";
    for (auto &x : r.timestamped_tokens) std::cout << ' ' << x.token_id << ':' << x.start_frame << ':' << x.end_frame;
    std::cout << "\nTEXT " << r.text << "\n";
    return 0;
}
