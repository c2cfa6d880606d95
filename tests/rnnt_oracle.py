"""Numpy restatement of the reference's RNNT model (src/rnnt.cpp, include/parakeet/config.hpp:119-135) on top of
oracle/oracle.py: the presets, RNNTJoint::forward and rnnt_greedy_decode(_with_timestamps).  Test infrastructure only
(tests/ and __graft_entry__.smoke()); tests/golden/golden_rnnt_v1.npz pins it to the compiled reference."""
from __future__ import annotations

import numpy as np

import oracle as O

F32 = np.float32


def make_rnnt_600m_config() -> O.Config:       # config.hpp:119-135 (mel_bins keeps EncoderConfig's 80)
    return O.Config(mel_bins=80, d_model=1024, n_layers=24, n_heads=8, ff=4096, vocab=1025, lstm_layers=2, durations=(),
                    has_ctc=False, joint_prefix="joint_.", name="rnnt-600m")


def make_tiny_rnnt_config() -> O.Config:
    """Not a reference preset: a small RNNT shape (tiny encoder, 2 LSTM layers) for fast unit tests only."""
    return O.Config(mel_bins=80, sub_channels=64, d_model=128, n_layers=2, n_heads=2, ff=256, vocab=33, pred_hidden=64,
                    lstm_layers=2, joint_hidden=64, durations=(), has_ctc=False, joint_prefix="joint_.", name="tiny-rnnt")


def rnnt_joint(W, enc_t, pred, cfg: O.Config):
    """RNNTJoint::forward, rnnt.cpp:38-45: log_softmax(out_proj(relu(enc_proj(enc) + pred_proj(pred))))."""
    p = cfg.joint_prefix
    z = O.linear(enc_t, W[p + "enc_proj_.weight"], W[p + "enc_proj_.bias"]) + O.linear(pred, W[p + "pred_proj_.weight"])
    z = np.maximum(z, 0).astype(F32)
    return O.log_softmax(O.linear(z, W[p + "out_proj_.weight"], W[p + "out_proj_.bias"]))


def rnnt_greedy_decode(W, enc, cfg: O.Config, max_symbols=10, with_timestamps=False, gaps=None):
    """rnnt_greedy_decode(_with_timestamps), rnnt.cpp:56-177: per frame at most max_symbols emissions; blank reverts
    the LSTM state and moves to the next frame; after the max_symbols-th emission the next frame starts with the
    state and token kept.  Timestamped tokens are (id, t, t, exp(log-prob)).  gaps: a list that receives the top-2
    log-prob gap of every decision (how far each arg-max is from a tie)."""
    blank = cfg.vocab - 1
    H = cfg.pred_hidden
    states = [(np.zeros(H, F32), np.zeros(H, F32)) for _ in range(cfg.lstm_layers)]
    token, out = blank, []
    for t in range(enc.shape[0]):
        for _sym in range(max_symbols):
            pred, new = O.prediction_step(W, token, states, cfg)
            lp = rnnt_joint(W, enc[t], pred, cfg)
            k = O.first_argmax(lp)
            if gaps is not None:
                top2 = np.partition(lp, -2)[-2:]
                gaps.append(float(top2[1] - top2[0]))
            if k == blank:
                break
            states = new
            out.append((k, t, t, float(np.exp(F32(lp[k])))) if with_timestamps else k)
            token = k
    return out


def transcribe(W, pcm, cfg: O.Config, timestamps=False):
    """Transcriber path of the reference CLI's run_rnnt_600m (src/main.cpp:296-360) for one utterance."""
    feats = O.preprocess_audio(pcm, cfg.mel_bins)
    enc = O.encoder_forward(W, feats, cfg)
    return rnnt_greedy_decode(W, enc, cfg, with_timestamps=timestamps)
