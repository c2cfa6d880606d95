"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol
include/parakeet_b200.h declares (no compute without a GPU), presets match the
reference's config.hpp, the host-side text helpers match the oracle, and the product
fails loudly without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "parakeet_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pk_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(pkg):
    L = pkg.load_library()
    syms = _declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/parakeet_b200.h but not exported"
    assert set(pkg.engine.EXPORTS) == set(syms)


def test_presets_match_reference_config(pkg):
    L = pkg.load_library()
    c = pkg.engine._PkConfig()
    L.pk_config_110m(C.byref(c))           # config.hpp:77-95
    assert (c.mel_bins, c.sub_channels, c.d_model, c.n_layers, c.n_heads, c.ff, c.conv_kernel) == (80, 256, 512, 17, 8, 2048, 9)
    assert (c.vocab, c.pred_hidden, c.lstm_layers, c.joint_hidden, c.n_durations) == (1025, 640, 1, 640, 5)
    assert list(c.durations)[:5] == [0, 1, 2, 3, 4] and c.has_ctc == 1 and c.joint_prefix_tdt == 1
    L.pk_config_tdt_600m(C.byref(c))       # config.hpp:98-116
    assert (c.mel_bins, c.d_model, c.n_layers, c.ff, c.vocab, c.lstm_layers, c.has_ctc, c.joint_prefix_tdt) == \
        (128, 1024, 24, 4096, 8193, 2, 0, 0)
    py = pkg.make_110m_config().to_c()
    L.pk_config_110m(C.byref(c))
    for f, _ in pkg.engine._PkConfig._fields_:
        if f in ("durations", "max_batch", "max_samples", "math"):
            continue
        assert getattr(py, f) == getattr(c, f), f


def test_shape_helpers(pkg, O):
    L = pkg.load_library()
    for n in (400, 401, 16000, 159999, 160000, 160001, 480000):
        assert L.pk_mel_frames(n) == O.n_mel_frames(n)
        assert L.pk_encoder_frames(L.pk_mel_frames(n)) == O.encoder_len(O.n_mel_frames(n))
    assert L.pk_encoder_frames(1001) == 126 and L.pk_encoder_frames(3001) == 376


def test_text_helpers_match_oracle(pkg, O, tiny):
    tok = pkg.engine.Tokenizer(tiny.vocab_path)
    assert tok.loaded()
    rng = np.random.default_rng(5)
    for _ in range(20):
        n = int(rng.integers(0, 30))
        ids = rng.integers(0, tiny.ocfg.vocab - 1, n).tolist()
        if n > 3:
            ids[2] = 9999        # out-of-range -> "[9999]" (vocab.cpp:33-36)
        assert tok.decode(ids) == O.detokenize(ids, tiny.pieces)
        start = np.cumsum(rng.integers(0, 4, n)).tolist()
        toks = [pkg.TimestampedToken(i, s, s + int(rng.integers(0, 3)), float(rng.random())) for i, s in zip(ids, start)]
        got = tok.group_words(toks)
        want = O.group_timestamps([(t.token_id, t.start_frame, t.end_frame, t.confidence) for t in toks], tiny.pieces)
        assert [w.word for w in got] == [w[0] for w in want]
        assert np.allclose([[w.start, w.end, w.confidence] for w in got], [[w[1], w[2], w[3]] for w in want], rtol=1e-6) or not want


def test_tokenize_and_boosted_ctc_match_reference_goldens(pkg, O, synth, tiny, golden):
    """Host code behind pk_tokenize / pk_ctc_decode_boosted (no device needed) against the compiled reference's
    fixtures (tests/golden/make_golden.py boost) and the oracle: Tokenizer::encode, ContextTrie, boosted CTC greedy."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_boost_v1.npz"))
    tok = pkg.engine.Tokenizer(tiny.vocab_path)
    for i in range(int(g["n_texts"][0])):
        text = bytes(g[f"enc.k{i}.text"]).decode()
        assert tok.encode(text) == g[f"enc.k{i}.ids"].tolist()
        assert tok.encode(text) == O.tokenizer_encode(text, tiny.pieces)
    assert tok.decode(tok.encode("")) == ""
    for n in range(int(g["n_cases"][0])):
        k = f"boost.k{n}."
        lens, ids, p, phrases = g[k + "ph_len"].tolist(), g[k + "ph_ids"].tolist(), 0, []
        for ln in lens:
            phrases.append(ids[p:p + ln])
            p += ln
        lp = O.ctc_log_probs(tiny.W, golden[f"tiny.c{int(g[k + 'clip'][0])}.enc"])
        got = pkg.engine.ctc_greedy_decode_boosted(lp, phrases, float(g[k + "boost"][0]))
        assert [[t.token_id, t.start_frame, t.end_frame] for t in got] == g[k + "ctc_tok"].tolist()
        assert np.allclose([t.confidence for t in got], g[k + "ctc_conf"], rtol=1e-3)
    # no phrases == plain greedy (ctc.cpp:79-127); random phrase sets == oracle
    lp = O.ctc_log_probs(tiny.W, golden["tiny.c0.enc"])
    plain = O.ctc_greedy_decode_with_timestamps(lp, tiny.ocfg.vocab - 1)
    assert [(t.token_id, t.start_frame, t.end_frame) for t in pkg.engine.ctc_greedy_decode_boosted(lp, [])] == [x[:3] for x in plain]
    rng = np.random.default_rng(31)
    for _ in range(10):
        phrases = [rng.integers(0, tiny.ocfg.vocab - 1, size=int(rng.integers(1, 5))).tolist() for _ in range(int(rng.integers(1, 9)))]
        boost = float(rng.uniform(0.5, 12.0))
        want = O.ctc_greedy_decode_with_timestamps_boosted(lp, O.ContextTrie(phrases), boost, tiny.ocfg.vocab - 1)
        got = pkg.engine.ctc_greedy_decode_boosted(lp, phrases, boost)
        assert [(t.token_id, t.start_frame, t.end_frame) for t in got] == [x[:3] for x in want]


def test_cpp_shim_host_functions(pkg, O, tiny, tmp_path):
    """The C++ shim's host-only pieces (Tokenizer::encode, ContextTrie, boosted CTC decode) compiled with g++ and
    run without a device; answers = the reference's BoostedCTCDecode tests and the oracle's encode."""
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "parakeet.cpp_b200")
    exe = str(tmp_path / "cpp_host_check")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "cpp_host_check.cpp"),
                    "-L", libdir, "-lparakeet_b200", "-Wl,-rpath," + libdir, "-o", exe], check=True)
    text = " ".join(p.replace(O.SP_MARK, " ").strip() for p in tiny.pieces[3:7])
    import struct
    rng = np.random.default_rng(8)
    pcm16 = (rng.standard_normal(5000) * 6000).astype(np.int16)
    wav = str(tmp_path / "a22k.wav")
    with open(wav, "wb") as f:                                    # mono PCM16 at 22.05 kHz
        f.write(b"RIFF" + struct.pack("<I", 36 + 2 * len(pcm16)) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, 22050, 44100, 2, 16))
        f.write(b"data" + struct.pack("<I", 2 * len(pcm16)) + pcm16.tobytes())
    out = subprocess.run([exe, tiny.vocab_path, text, wav], check=True, capture_output=True, text=True).stdout.splitlines()
    want = O.tokenizer_encode(text, tiny.pieces)
    assert out[0].split()[1:] == [str(i) for i in want] and len(want) >= 3
    assert out[1] == "decode " + O.detokenize(want, tiny.pieces)
    assert out[2] == "plain 42 n=1"
    assert out[3] == "boosted 43 start=0 end=2 n=1 empty=1/0"
    assert out[4] == "built %d" % len(want)
    res = O.sinc_resample(pcm16.astype(np.float32) / np.float32(32768.0), 22050, 16000)      # audio_io.cpp: PCM16 / 32768, then resample
    n_s, mid_s, acc_s = out[5].split()[1:]
    assert int(n_s) == len(res)
    assert abs(float(mid_s) - float(res[len(res) // 2])) <= 1e-7 * max(1.0, abs(float(res[len(res) // 2])))
    acc = float(np.sum(res.astype(np.float64) * ((np.arange(len(res)) % 7) + 1)))
    assert abs(float(acc_s) - acc) <= 1e-6 * max(1.0, abs(acc))


def test_resample_matches_oracle_and_reference(pkg, O, golden_refcalls):
    """pk_resample (host) == the oracle's sinc_resample == the compiled reference's parakeet::resample, bit for bit
    (double arithmetic in the same order), for down- and up-sampling, integer and fractional ratios, tiny inputs.
    The reference's outputs are stored as SHA-256 digests of their fp32 bytes."""
    import hashlib
    rng = np.random.default_rng(4)
    for sr, dr, n in [(44100, 16000, 9000), (48000, 16000, 5001), (8000, 16000, 2500), (22050, 16000, 3000), (24000, 16000, 999),
                      (96000, 16000, 6000), (16000, 16000, 50), (11025, 16000, 3), (16000, 8000, 1000), (44100, 16000, 0)]:
        x = (rng.standard_normal(n) * 0.3).astype(np.float32)
        got = pkg.engine.resample(x, sr, dr)
        want = O.sinc_resample(x, sr, dr)
        assert got.shape == want.shape == (pkg.engine.load_library().pk_resample_len(n, sr, dr),)
        assert np.array_equal(got, want), (sr, dr, n, float(np.abs(got - want).max()))
        if n > 0:
            ref_digest = golden_refcalls[f"resample_host.{sr}.{dr}.{n}.sha256"].tobytes()
            assert hashlib.sha256(np.ascontiguousarray(got, np.float32).tobytes()).digest() == ref_digest, (sr, dr, n)
    assert pkg.engine.load_library().pk_resample_len(-1, 16000, 16000) == -1
    # a resampled 1 kHz tone keeps its frequency
    t = np.arange(44100, dtype=np.float64) / 44100.0
    y = pkg.engine.resample(np.sin(2 * np.pi * 1000.0 * t).astype(np.float32), 44100, 16000)
    spec = np.abs(np.fft.rfft(y[1000:1000 + 8000]))
    assert abs(int(spec.argmax()) * 16000 / 8000 - 1000.0) <= 2.0


def test_vocab_missing_file_raises(pkg):
    with pytest.raises(RuntimeError):
        pkg.engine.Tokenizer("/nonexistent/vocab.txt")


def test_safetensors_errors_are_reported(pkg, tiny, tmp_path):
    """Loader error paths that do not need a device come back as status + message...
    but without a GPU pk_engine_create refuses first: the product has no CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises(RuntimeError, match="no CUDA device|CUDA"):
        pkg.Engine(tiny.cfg, tiny.weights_path, 0)


def test_read_wav_roundtrip(pkg, synth, tmp_path):
    import struct
    pcm = synth.make_audio(16000, 5)
    i16 = np.round(pcm * 32768.0).astype(np.int16)
    p = tmp_path / "a.wav"
    with open(p, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 36 + 2 * len(i16)) + b"WAVEfmt " +
                struct.pack("<IHHIIHH", 16, 1, 1, 16000, 32000, 2, 16) + b"data" + struct.pack("<I", 2 * len(i16)))
        f.write(i16.tobytes())
    assert np.array_equal(pkg.engine.read_wav(str(p)), pcm)


def test_synth_checkpoint_layout(O, synth):
    """705 tensors / 114.6 M parameters for 110m (SURVEY.md section 8a row L)."""
    specs = synth.tensor_specs(O.make_110m_config())
    assert len(specs) == 705
    n = sum(int(np.prod(s)) for _, s, k in specs if k != "i64")
    assert abs(n - 114.6e6) < 0.1e6


def _write_st(path, header_json: bytes, data: bytes = b""):
    import struct
    with open(path, "wb") as f:
        f.write(struct.pack("<Q", len(header_json)) + header_json + data)


def test_safetensors_reader_dtypes_and_hostile_headers(pkg, tmp_path):
    """The checkpoint reader (csrc/safetensors.cpp) on the host: F32 / F16 / BF16 / F64 tensors convert to the expected fp32
    values (safetensors::load, axiom io_safetensors.cpp:16-44), and malformed headers are refused instead of read out of
    bounds: negative or overflowing sizes, offsets past the file, an unterminated escape, bottomless nesting."""
    import json
    from parakeet_cpp_b200.engine import safetensors_probe
    rng = np.random.default_rng(2)
    x = (rng.standard_normal(37) * 3).astype(np.float32)
    import torch
    parts = {"a32": (x.tobytes(), "F32"), "a16": (x.astype(np.float16).tobytes(), "F16"),
             "ab16": (torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().tobytes(), "BF16"),
             "a64": (x.astype(np.float64).tobytes(), "F64")}
    hdr, blob = {"__metadata__": {"format": "pt", "nested": {"k": [1, 2, {"z": None}]}}}, b""
    for k, (b, dt) in parts.items():
        hdr[k] = {"dtype": dt, "shape": [37], "data_offsets": [len(blob), len(blob) + len(b)]}
        blob += b
    p = str(tmp_path / "ok.safetensors")
    _write_st(p, json.dumps(hdr).encode(), blob)
    st, msg, v = safetensors_probe(p, "a32", 37)
    assert st == 0 and np.array_equal(v, x)
    assert np.array_equal(safetensors_probe(p, "a16", 37)[2], x.astype(np.float16).astype(np.float32))
    assert np.array_equal(safetensors_probe(p, "ab16", 37)[2], torch.from_numpy(x).to(torch.bfloat16).float().numpy())
    assert np.array_equal(safetensors_probe(p, "a64", 37)[2], x)
    assert safetensors_probe(p, "nope", 1)[0] == 4                                    # PK_ERR_MISSING
    bad = {
        "neg_shape": b'{"t":{"dtype":"F32","shape":[-4],"data_offsets":[0,16]}}',
        "huge_offset": b'{"t":{"dtype":"F32","shape":[4],"data_offsets":[0,18446744073709551615]}}',
        "overflow_offset": b'{"t":{"dtype":"F32","shape":[4],"data_offsets":[0,99999999999999999999999]}}',
        "float_offset": b'{"t":{"dtype":"F32","shape":[4],"data_offsets":[0,1e30]}}',
        "end_before_begin": b'{"t":{"dtype":"F32","shape":[4],"data_offsets":[16,0]}}',
        "cut_escape": b'{"t\\u12',
        "deep": b'{"__metadata__":' + b"[" * 5000 + b"]" * 5000 + b"}",
        "not_object": b'[1,2,3]',
    }
    for name, h in bad.items():
        q = str(tmp_path / (name + ".safetensors"))
        _write_st(q, h, b"\0" * 16)
        assert safetensors_probe(q)[0] == 2, name                                     # PK_ERR_IO, no crash
    q = str(tmp_path / "shape_overflow.safetensors")
    _write_st(q, b'{"t":{"dtype":"F32","shape":[4294967296,4294967296,4],"data_offsets":[0,16]}}', b"\0" * 16)
    st, msg, _ = safetensors_probe(q, "t", 4)
    assert st == 2 and "overflow" in msg
    q = str(tmp_path / "hdr_len.safetensors")
    with open(q, "wb") as f:
        f.write(b"\xff" * 8 + b"{}")
    assert safetensors_probe(q)[0] == 2
