"""Seeded synthetic checkpoints, vocabularies and 16 kHz audio (harness only).

There is no network here, so no real Parakeet checkpoint: both the reference
build and this engine load the SAME synthetic safetensors file whose tensor
names / shapes follow the reference's loader contract (SURVEY.md section 8a row L:
names come from AX_REGISTER_* stringification, e.g. src/tdt_ctc.cpp:5-9,
src/encoder.cpp:36,52-53,80-81,193,216,249; shapes from scripts/convert_nemo.py).

Weight statistics are chosen so the model is numerically "alive" (time-varying
encoder output, diverse CTC/TDT token streams, no TDT livelock), see
`make_weights`.  Audio follows SURVEY.md section 8d: a seeded mixture of
amplitude-modulated tones per 250 ms segment plus N(0, 0.02) noise, passed
through an int16 round trip so a WAV file and the raw fp32 hold equal samples.
"""
from __future__ import annotations

import json
import struct

import numpy as np

F32 = np.float32


def tensor_specs(cfg):
    """[(name, shape, kind)] in a fixed order.  cfg: any object with the fields of
    oracle.Config / engine.ModelConfig."""
    C, d, ff, mel = cfg.sub_channels, cfg.d_model, cfg.ff, cfg.mel_bins
    H, hd = cfg.n_heads, cfg.d_model // cfg.n_heads
    Fq = mel // 8
    s = []
    p = "encoder_.subsampling_."
    s += [(p + "conv1_.weight", (C, 1, 3, 3), "w"), (p + "conv1_.bias", (C,), "b"),
          (p + "dw1_.weight", (C, 1, 3, 3), "w"), (p + "dw1_.bias", (C,), "b"),
          (p + "conv2_.weight", (C, C, 1, 1), "w"), (p + "conv2_.bias", (C,), "b"),
          (p + "dw2_.weight", (C, 1, 3, 3), "w"), (p + "dw2_.bias", (C,), "b"),
          (p + "conv3_.weight", (C, C, 1, 1), "w"), (p + "conv3_.bias", (C,), "b"),
          (p + "proj_.weight", (d, C * Fq), "w"), (p + "proj_.bias", (d,), "b")]
    for i in range(cfg.n_layers):
        L = f"encoder_.layers_.{i}."
        for f in ("ffn1_.", "ffn2_."):
            s += [(L + f + "norm_.weight", (d,), "g"), (L + f + "norm_.bias", (d,), "b"),
                  (L + f + "fc1_.weight", (ff, d), "w"), (L + f + "fc1_.bias", (ff,), "b"),
                  (L + f + "fc2_.weight", (d, ff), "wo"), (L + f + "fc2_.bias", (d,), "bo")]
        a = L + "attn_."
        s += [(a + "norm_.weight", (d,), "g"), (a + "norm_.bias", (d,), "b")]
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            s += [(a + f"mha_.{n}.weight", (d, d),
                   "wq" if n in ("q_proj", "k_proj") else ("wo" if n == "out_proj" else "w")),
                  (a + f"mha_.{n}.bias", (d,), "bo" if n == "out_proj" else "b")]
        s += [(a + "pos_proj_.weight", (d, d), "wq"),
              (a + "pos_bias_u_", (H, hd), "pb"), (a + "pos_bias_v_", (H, hd), "pb")]
        c = L + "conv_."
        s += [(c + "norm_.weight", (d,), "g"), (c + "norm_.bias", (d,), "b"),
              (c + "pointwise_conv1_.weight", (2 * d, d, 1), "w"), (c + "pointwise_conv1_.bias", (2 * d,), "b"),
              (c + "depthwise_conv_.weight", (d, 1, cfg.conv_k), "w"), (c + "depthwise_conv_.bias", (d,), "b"),
              (c + "batch_norm_.weight", (d,), "g"), (c + "batch_norm_.bias", (d,), "b"),
              (c + "batch_norm_.running_mean", (d,), "b"), (c + "batch_norm_.running_var", (d,), "var"),
              (c + "batch_norm_.num_batches_tracked", (), "i64"),
              (c + "pointwise_conv2_.weight", (d, d, 1), "wo"), (c + "pointwise_conv2_.bias", (d,), "bo")]
        s += [(L + "final_norm_.weight", (d,), "g"), (L + "final_norm_.bias", (d,), "b")]
    V, P, J = cfg.vocab, cfg.pred_hidden, cfg.joint_hidden
    if cfg.has_ctc:
        s += [("ctc_decoder_.proj_.weight", (V, d, 1), "head"), ("ctc_decoder_.proj_.bias", (V,), "b")]
    s += [("prediction_.embed_.weight", (V, P), "emb")]
    for l in range(cfg.lstm_layers):
        q = f"prediction_.lstm_.cells_.{l}."
        s += [(q + "input_proj_.weight", (4 * P, P), "w"), (q + "input_proj_.bias", (4 * P,), "b"),
              (q + "hidden_proj_.weight", (4 * P, P), "w")]
    j = cfg.joint_prefix
    s += [(j + "enc_proj_.weight", (J, d), "w"), (j + "enc_proj_.bias", (J,), "b"),
          (j + "pred_proj_.weight", (J, P), "w")]
    if len(cfg.durations) == 0:         # RNNTJoint (rnnt.cpp:34-45): one output head, no durations
        s += [(j + "out_proj_.weight", (V, J), "head"), (j + "out_proj_.bias", (V,), "lab_b")]
    else:
        s += [(j + "label_proj_.weight", (V, J), "head"), (j + "label_proj_.bias", (V,), "lab_b"),
              (j + "duration_proj_.weight", (len(cfg.durations), J), "head"),
              (j + "duration_proj_.bias", (len(cfg.durations),), "dur_b")]
    return s


def make_weights(cfg, seed=0, gain=1.0, head_gain=4.0, out_gain=0.25, blank_bias=None, ctc_blank_bias=None):
    """dict name -> ndarray.  N(0, gain/sqrt(fan_in)) matrices; LayerNorm/BN scale
    ~1; small biases; the q/k/pos projections get a larger gain so attention is
    peaked (time-local) instead of uniform, and the classification heads get
    `head_gain` so arg-max margins sit well above fp32 re-association noise."""
    rng = np.random.default_rng(seed)
    W = {}
    if blank_bias is None:          # keeps the TDT token rate near one per 2-4 frames
        blank_bias = 5.0 if cfg.vocab > 100 else 2.5
    if ctc_blank_bias is None:
        ctc_blank_bias = 12.0 if cfg.vocab > 100 else 5.0
    for name, shape, kind in tensor_specs(cfg):
        if kind == "i64":
            W[name] = np.array(1000, dtype=np.int64)
            continue
        fan_in = int(np.prod(shape[1:])) if len(shape) > 1 else 1
        if kind == "w":
            a = rng.standard_normal(shape) * (gain / np.sqrt(fan_in))
        elif kind == "wo":
            a = rng.standard_normal(shape) * (out_gain / np.sqrt(fan_in))
        elif kind == "bo":
            a = 0.1 * out_gain * rng.standard_normal(shape)
        elif kind == "wq":
            a = rng.standard_normal(shape) * (2.0 * gain / np.sqrt(fan_in))
        elif kind == "head":
            a = rng.standard_normal(shape) * (head_gain / np.sqrt(fan_in))
            if name.startswith(cfg.joint_prefix):
                # zero-mean rows: the (positive-mean) ReLU joint activation then adds no constant
                # per-class offset, so labels/durations follow the input instead of a few classes
                a = a - a.reshape(shape[0], -1).mean(axis=1).reshape((shape[0],) + (1,) * (len(shape) - 1))
        elif kind == "emb":
            a = rng.standard_normal(shape)
            a[-1] = 0.0                      # blank/SOS row is zero in real checkpoints
        elif kind == "g":
            a = 1.0 + 0.1 * rng.standard_normal(shape)
        elif kind == "var":
            a = rng.uniform(0.5, 1.5, shape)
        elif kind == "pb":
            a = 0.5 * rng.standard_normal(shape)
        elif kind == "lab_b":
            a = 0.1 * rng.standard_normal(shape)
            a[-1] = blank_bias               # blank is the commonest TDT label
        elif kind == "dur_b":
            # duration 0 ("emit again on this frame") must stay rare: the reference never forces an
            # advance (tdt.cpp:66-104), so a zero-duration fixed point livelocks it
            a = np.array([-3.5, 1.0, 0.5, 0.0, -0.5])[: shape[0]] + 0.1 * rng.standard_normal(shape)
        else:                                # "b"
            a = 0.1 * rng.standard_normal(shape)
        W[name] = a.astype(F32)
    if "ctc_decoder_.proj_.bias" in W:
        W["ctc_decoder_.proj_.bias"][-1] = ctc_blank_bias
    return W


_ST_DTYPE = {np.dtype("float32"): "F32", np.dtype("int64"): "I64", np.dtype("float16"): "F16"}


def save_safetensors(path, tensors):
    """Minimal safetensors writer: 8-byte LE header length, JSON header, raw data
    (the layout axiom io_safetensors.cpp:123-160 parses)."""
    header, off, blobs = {}, 0, []
    for name, a in tensors.items():
        a = np.ascontiguousarray(a)
        b = a.tobytes()
        header[name] = {"dtype": _ST_DTYPE[a.dtype], "shape": list(a.shape),
                        "data_offsets": [off, off + len(b)]}
        off += len(b)
        blobs.append(b)
    header["__metadata__"] = {"format": "pt", "generator": "parakeet_b200.synth"}
    hj = json.dumps(header, separators=(",", ":")).encode()
    hj += b" " * ((8 - len(hj) % 8) % 8)
    with open(path, "wb") as f:
        f.write(struct.pack("<Q", len(hj)))
        f.write(hj)
        for b in blobs:
            f.write(b)


def load_safetensors(path):
    """Minimal reader (harness / oracle side)."""
    with open(path, "rb") as f:
        n = struct.unpack("<Q", f.read(8))[0]
        header = json.loads(f.read(n))
        base = 8 + n
        raw = np.memmap(path, dtype=np.uint8, mode="r")
    inv = {v: k for k, v in _ST_DTYPE.items()}
    out = {}
    for name, m in header.items():
        if name == "__metadata__":
            continue
        s, e = m["data_offsets"]
        out[name] = np.frombuffer(raw[base + s: base + e].tobytes(), dtype=inv[m["dtype"]]).reshape(m["shape"])
    return out


def make_vocab(n_pieces, seed=0):
    """n_pieces SentencePiece-like pieces (vocab-1 of them; the blank has none).
    ~40 % start a word (U+2581 prefix) so word grouping is exercised."""
    rng = np.random.default_rng(seed + 7)
    letters = "abcdefghijklmnopqrstuvwxyz"
    pieces, seen = [], set()
    while len(pieces) < n_pieces:
        k = int(rng.integers(1, 5))
        w = "".join(letters[int(i)] for i in rng.integers(0, 26, k))
        if rng.random() < 0.4:
            w = "▁" + w
        if w in seen:
            continue
        seen.add(w)
        pieces.append(w)
    return pieces


def save_vocab(path, pieces):
    with open(path, "w", encoding="utf-8") as f:
        for i, p in enumerate(pieces):
            f.write(f"{p}\t{-float(i)}\n")


def make_audio(n_samples, seed):
    """Seeded synthetic speech-like fp32 PCM in [-1, 1] (int16-exact)."""
    rng = np.random.default_rng(seed)
    sr = 16000
    t = np.arange(n_samples) / sr
    x = np.zeros(n_samples)
    seg = sr // 4
    for s0 in range(0, n_samples, seg):
        s1 = min(s0 + seg, n_samples)
        tt = t[s0:s1]
        for _ in range(int(rng.integers(3, 7))):
            f = rng.uniform(100.0, 4000.0)
            am = rng.uniform(1.0, 8.0)
            x[s0:s1] += rng.uniform(0.05, 0.25) * np.sin(2 * np.pi * f * tt + rng.uniform(0, 6.28)) * \
                (0.5 + 0.5 * np.sin(2 * np.pi * am * tt + rng.uniform(0, 6.28)))
    x += rng.normal(0.0, 0.02, n_samples)
    x = np.clip(x, -0.99, 0.99)
    i16 = np.round(x * 32767.0).astype(np.int16)
    return (i16.astype(F32) / F32(32768.0)).astype(F32)
