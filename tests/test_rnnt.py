"""RNNT greedy decoding (rnnt_greedy_decode(_with_timestamps), reference src/rnnt.cpp:56-177) and the rnnt-600m
preset (config.hpp:119-135).  CPU: the presets and the numpy oracle against tests/golden/golden_rnnt_v1.npz, which
the compiled reference recorded (make_golden_rnnt.py).  GPU: the decode kernel's RNNT mode through the C-ABI."""
import ctypes as C
import dataclasses
import os
import subprocess
from collections import Counter

import numpy as np
import pytest

import rnnt_oracle as RO

HERE = os.path.dirname(os.path.abspath(__file__))
MATH = {"bf16x3": 0, "fp32": 2}
ENC_TOL = 1e-3


@pytest.fixture(scope="module")
def grnnt():
    with np.load(os.path.join(HERE, "golden", "golden_rnnt_v1.npz"), allow_pickle=False) as z:
        return dict(z)


def _clips(g, tag):
    return [f"{tag}.c{i}." for i in range(int(g[tag + ".n_clips"][0]))]


def _tt(toks):
    return [[t.token_id, t.start_frame, t.end_frame] for t in toks]


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ------------------------------------------------------------------ CPU
def test_rnnt_600m_preset_matches_reference_config(pkg, O):
    """make_rnnt_600m_config (config.hpp:119-135): EncoderConfig's 80 mels into d 1024, 24 layers, 8 heads, ff 4096,
    256 subsampling channels, kernel 9; 2-layer LSTM of 640; joint 640; vocab 1025; no durations, no CTC head."""
    c = pkg.make_rnnt_600m_config()
    assert (c.mel_bins, c.sub_channels, c.d_model, c.n_layers, c.n_heads, c.ff, c.conv_k) == (80, 256, 1024, 24, 8, 4096, 9)
    assert (c.vocab, c.pred_hidden, c.lstm_layers, c.joint_hidden) == (1025, 640, 2, 640)
    assert c.durations == () and not c.has_ctc and c.joint_prefix == "joint_." and c.is_rnnt
    assert (c.max_batch, c.max_samples) == (16, 480000)
    o = RO.make_rnnt_600m_config()
    for f in ("mel_bins", "sub_channels", "d_model", "n_layers", "n_heads", "ff", "conv_k", "vocab", "pred_hidden",
              "lstm_layers", "joint_hidden", "durations", "has_ctc", "joint_prefix"):
        assert getattr(o, f) == getattr(c, f), f
    # the C preset fills the same struct
    L = pkg.load_library()
    want, got = c.to_c(), pkg.engine._PkConfig()
    L.pk_config_rnnt_600m(C.byref(got))
    assert bytes(got) == bytes(want)
    assert O.encoder_len(1 + 480000 // 160) == 376 and c.sub_channels * (80 // 8) == 2560    # F' = 10: proj_ is 2560 -> 1024


def test_synthetic_rnnt_checkpoint_has_the_rnnt_joint_keys(synth):
    names = {n: s for n, s, _ in synth.tensor_specs(RO.make_rnnt_600m_config())}
    assert names["joint_.out_proj_.weight"] == (1025, 640) and names["joint_.out_proj_.bias"] == (1025,)
    assert names["joint_.enc_proj_.weight"] == (640, 1024) and "joint_.pred_proj_.bias" not in names
    assert names["encoder_.subsampling_.proj_.weight"] == (1024, 2560)
    assert not any("label_proj_" in n or "duration_proj_" in n or n.startswith("ctc_") for n in names)


@pytest.mark.parametrize("tag", ["tiny", "msym"])
def test_numpy_oracle_matches_reference_golden(synth, grnnt, tag):
    cfg = RO.make_tiny_rnnt_config()
    W = synth.make_weights(cfg, seed=3, blank_bias=float(grnnt[tag + ".blank_bias"][0]))
    for k in _clips(grnnt, tag):
        got = RO.rnnt_greedy_decode(W, grnnt[k + "enc"], cfg, with_timestamps=True)
        assert [list(t[:3]) for t in got] == grnnt[k + "tok"].tolist(), k
        assert np.allclose([t[3] for t in got], grnnt[k + "conf"], rtol=1e-4, atol=1e-7), k
        assert RO.rnnt_greedy_decode(W, grnnt[k + "enc"], cfg) == grnnt[k + "ids"].tolist(), k


def test_numpy_oracle_matches_reference_golden_600m(synth, grnnt):
    cfg = RO.make_rnnt_600m_config()
    W = synth.make_weights(cfg, seed=0, blank_bias=float(grnnt["r600.blank_bias"][0]))
    k = "r600.c0."
    got = RO.rnnt_greedy_decode(W, grnnt[k + "enc"], cfg, with_timestamps=True)
    assert [list(t[:3]) for t in got] == grnnt[k + "tok"].tolist()
    assert np.allclose([t[3] for t in got], grnnt[k + "conf"], rtol=1e-4, atol=1e-7)


def test_fixture_exercises_every_branch_of_the_rule(grnnt):
    """Counted from the reference's own output: frames where blank came at once, frames with 1-9 symbols followed by a
    blank, and frames left after max_symbols = 10 symbols without a blank (forced advance), in the tiny shape and in
    the preset, and a T' = 1 clip with several symbols; timestamps are start = end = t; the id-only decoder agrees."""
    counts = {}
    for tag in ("tiny", "msym", "r600"):
        zero = some = forced = 0
        for k in _clips(grnnt, tag):
            tok = grnnt[k + "tok"]
            T = grnnt[k + "enc"].shape[0]
            assert (tok[:, 1] == tok[:, 2]).all() and (np.diff(tok[:, 1]) >= 0).all() and (tok[:, 1] < T).all()
            assert grnnt[k + "ids"].tolist() == tok[:, 0].tolist()
            per = Counter(tok[:, 1].tolist())
            assert max(per.values(), default=0) <= 10
            zero += T - len(per)
            some += sum(1 <= v <= 9 for v in per.values())
            forced += sum(v == 10 for v in per.values())
        counts[tag] = (zero, some, forced)
    assert all(z > 0 and s > 0 and f > 0 for z, s, f in counts.values()), counts
    assert counts["tiny"][1] + counts["msym"][1] >= 10, counts
    assert grnnt["tiny.c1.enc"].shape[0] == 1                         # the 400-sample clip: T' = 1
    k = f"msym.c{int(grnnt['msym.t1_multi'][0])}."
    assert grnnt[k + "enc"].shape[0] == 1 and len(grnnt[k + "tok"]) >= 2


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module", params=["bf16x3", "fp32"])
def math_mode(request):
    return request.param


class _Model:
    def __init__(self, d, synth, ocfg, seed, blank_bias, tag):
        self.W = synth.make_weights(ocfg, seed=seed, blank_bias=blank_bias)
        self.weights_path = os.path.join(d, tag + ".safetensors")
        synth.save_safetensors(self.weights_path, self.W)
        self.pieces = synth.make_vocab(ocfg.vocab - 1, seed=seed)
        self.vocab_path = os.path.join(d, tag + ".vocab.txt")
        synth.save_vocab(self.vocab_path, self.pieces)
        self.ocfg = ocfg


@pytest.fixture(scope="module")
def trnnt(tmp_path_factory, synth, grnnt):
    d = str(tmp_path_factory.mktemp("trnnt"))
    return {tag: _Model(d, synth, RO.make_tiny_rnnt_config(), 3, float(grnnt[tag + ".blank_bias"][0]), tag) for tag in ("tiny", "msym")}


@pytest.fixture(scope="module")
def r600(tmp_path_factory, synth, grnnt):
    return _Model(str(tmp_path_factory.mktemp("r600")), synth, RO.make_rnnt_600m_config(), 0, float(grnnt["r600.blank_bias"][0]), "r600")


def _engine(pkg, path, math_mode, **kw):
    return pkg.Engine(pkg.make_tiny_rnnt_config(math=MATH[math_mode], **kw), path, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["tiny", "msym"])
def test_tiny_rnnt_decode_and_transcribe_match_reference_golden(pkg, synth, trnnt, grnnt, math_mode, tag):
    e = _engine(pkg, trnnt[tag].weights_path, math_mode)
    keys = _clips(grnnt, tag)
    # pk_decode on the reference's encoder output, all clips as one ragged batch
    got = e.decode([grnnt[k + "enc"] for k in keys], pkg.Decoder.RNNT)
    assert e.truncated_count() == 0
    for k, g in zip(keys, got):
        assert _tt(g) == grnnt[k + "tok"].tolist(), k
        assert np.allclose([t.confidence for t in g], grnnt[k + "conf"], rtol=1e-3, atol=1e-6), k
    # pk_transcribe_batch from PCM
    pcms = [synth.make_audio(*(int(v) for v in grnnt[k + "n_samples"])) for k in keys]
    got = e.transcribe_batch(pcms, pkg.Decoder.RNNT)
    assert e.truncated_count() == 0
    for k, g in zip(keys, got):
        assert _tt(g) == grnnt[k + "tok"].tolist(), k
        assert np.allclose([t.confidence for t in g], grnnt[k + "conf"], rtol=1e-3, atol=1e-6), k
    e.close()


@pytest.mark.gpu
def test_tiny_rnnt_lockstep_batch_equals_singles_and_more_than_64(pkg, synth, trnnt, math_mode):
    m = trnnt["msym"]
    e = _engine(pkg, m.weights_path, math_mode, max_batch=80)
    pcms = [synth.make_audio(int(n), 500 + i) for i, n in enumerate(np.linspace(400, 64000, 70).astype(int))]
    batch = e.transcribe_batch(pcms, pkg.Decoder.RNNT)
    assert e.truncated_count() == 0
    for i in (0, 1, 17, 40, 64, 69):
        alone = e.transcribe_batch([pcms[i]], pkg.Decoder.RNNT)[0]
        assert _tt(alone) == _tt(batch[i]), i
        want = RO.transcribe(m.W, pcms[i], m.ocfg, timestamps=True)
        assert _tt(alone) == [list(w[:3]) for w in want], i
    e.close()


@pytest.mark.gpu
def test_rnnt_600m_matches_reference_golden(pkg, O, synth, r600, grnnt, math_mode):
    k = "r600.c0."
    pcm = synth.make_audio(*(int(v) for v in grnnt[k + "n_samples"]))
    cfg = pkg.make_rnnt_600m_config(max_batch=4, max_samples=80000, math=MATH[math_mode])
    e = pkg.Engine(cfg, r600.weights_path, 0)
    feats = e.mel([pcm])[0]
    assert np.abs(feats - grnnt[k + "mel"].astype(np.float32)).max() < 5e-3
    enc = e.encode([O.preprocess_audio(pcm, 80)])[0]
    assert enc.shape == grnnt[k + "enc"].shape
    assert _rel(enc, grnnt[k + "enc"]) < ENC_TOL
    toks = e.decode([grnnt[k + "enc"]], pkg.Decoder.RNNT)[0]
    assert _tt(toks) == grnnt[k + "tok"].tolist()
    assert np.allclose([t.confidence for t in toks], grnnt[k + "conf"], rtol=1e-3, atol=1e-6)
    e.close()
    t = pkg.Transcriber(r600.weights_path, r600.vocab_path, cfg)
    r = t.transcribe(pcm, timestamps=True)
    assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == grnnt[k + "tok"].tolist()
    assert r.text == pkg.engine.Tokenizer(r600.vocab_path).decode(grnnt[k + "ids"].tolist())
    t.engine.close()


@pytest.mark.gpu
def test_rnnt_600m_full_size_ragged_batch_against_oracle(pkg, synth, r600):
    """16 clips up to 30 s (T' = 376) in one batch: the decode of each row equals the numpy rnnt_greedy_decode on the
    engine's own encoder output (for rows whose decisions all sit >= 1e-3 from a tie), and single-utterance runs."""
    cfg = pkg.make_rnnt_600m_config()
    e = pkg.Engine(cfg, r600.weights_path, 0)
    lens = [480000, 400, 16000, 80000, 160000, 240000, 333333, 479999, 48000, 123456, 300000, 64000, 420000, 8000, 200000, 360000]
    pcms = [synth.make_audio(n, 4000 + i) for i, n in enumerate(lens)]
    got = e.transcribe_batch(pcms, pkg.Decoder.RNNT)
    assert e.truncated_count() == 0
    encs = e.encode(e.mel(pcms))
    checked = 0
    for i in (0, 1, 3, 8, 13):
        gaps = []
        want = RO.rnnt_greedy_decode(r600.W, encs[i], r600.ocfg, with_timestamps=True, gaps=gaps)
        if min(gaps, default=1.0) >= 1e-3:
            assert _tt(got[i]) == [list(w[:3]) for w in want], i
            assert np.allclose([t.confidence for t in got[i]], [w[3] for w in want], rtol=1e-3, atol=1e-6), i
            checked += 1
    assert checked >= 3
    for i in (0, 6, 10):
        assert _tt(e.transcribe_batch([pcms[i]], pkg.Decoder.RNNT)[0]) == _tt(got[i]), i
    e.close()


@pytest.mark.gpu
def test_rnnt_error_statuses(pkg, pkg_tiny_tdt, synth, trnnt, tmp_path):
    m = trnnt["tiny"]
    e = pkg.Engine(pkg.make_tiny_rnnt_config(), m.weights_path, 0)
    pcm = [synth.make_audio(16000, 1)]
    for dec in (pkg.Decoder.TDT, pkg.Decoder.CTC):
        with pytest.raises(RuntimeError, match="RNNT model"):
            e.transcribe_batch(pcm, dec)
        with pytest.raises(RuntimeError, match="RNNT model"):
            e.decode([np.zeros((3, 128), np.float32)], dec)
    with pytest.raises(RuntimeError, match=r"unknown pk_decoder"):
        e.transcribe_batch(pcm, 7)
    with pytest.raises(RuntimeError, match="not available on an RNNT engine"):
        e.stream_open(2, 2560)
    e.set_boost([[3, 4]], 5.0)
    with pytest.raises(RuntimeError, match="phrase boosting"):
        e.transcribe_batch(pcm, pkg.Decoder.RNNT)
    e.set_boost([], 0.0)
    assert len(e.transcribe_batch(pcm, pkg.Decoder.RNNT)) == 1
    e.close()
    # the Python Transcriber: RNNT is the default; an explicit CTC / TDT request is an error, as in the C-ABI
    t = pkg.Transcriber(m.weights_path, m.vocab_path, pkg.make_tiny_rnnt_config())
    assert t.transcribe(pcm[0]).token_ids == t.transcribe(pcm[0], pkg.Decoder.RNNT).token_ids
    for dec in (pkg.Decoder.TDT, pkg.Decoder.CTC):
        with pytest.raises(ValueError, match="RNNT model"):
            t.transcribe(pcm[0], dec)
        with pytest.raises(ValueError, match="RNNT model"):
            t.transcribe_batch(pcm, dec)
    t.engine.close()
    # a TDT engine rejects PK_DECODER_RNNT
    with pytest.raises(RuntimeError, match="needs an RNNT model"):
        pkg_tiny_tdt.transcribe_batch(pcm, pkg.Decoder.RNNT)
    # a checkpoint without the RNNT output head: PK_ERR_MISSING
    bad = dict(m.W)
    bad.pop("joint_.out_proj_.weight")
    p = str(tmp_path / "no_out_proj.safetensors")
    synth.save_safetensors(p, bad)
    L = pkg.load_library()
    h = C.c_void_p()
    cc = pkg.make_tiny_rnnt_config().to_c()
    assert L.pk_engine_create(C.byref(cc), p.encode(), 0, C.byref(h)) == 4
    assert b"out_proj_" in L.pk_last_error(None)


@pytest.fixture(scope="module")
def pkg_tiny_tdt(pkg, tiny):
    e = pkg.Engine(tiny.cfg, tiny.weights_path, 0)
    yield e
    e.close()


@pytest.mark.gpu
def test_rnnt_job_api(pkg, synth, trnnt, math_mode):
    m = trnnt["msym"]
    e = _engine(pkg, m.weights_path, math_mode)
    batches = [[synth.make_audio(n, 700 + 10 * r + i) for i, n in enumerate(ns)] for r, ns in enumerate(([32000, 400, 64000], [20000, 48000]))]
    want = [e.transcribe_batch(b, pkg.Decoder.RNNT) for b in batches]
    from parakeet_cpp_b200.engine import _pack
    buf, off = _pack(batches[0] + batches[1])
    e.job_stage(buf, off)
    e.job_begin(5, 1)
    for first, n in ((0, 3), (3, 2)):
        e.job_select(first, n)
        e.run_staged(pkg.Decoder.RNNT)
        e.job_append()
    rows = e.job_fetch(5)
    assert rows.shape[1] == 1 + e.cap == 1 + 10 * e.Tmax
    flat = [w for ws in want for w in ws]
    for i, w in enumerate(flat):
        assert rows[i, 1:1 + rows[i, 0]].tolist() == [t.token_id for t in w], i
    e.close()


@pytest.mark.gpu
def test_cpp_rnnt_transcriber(pkg, synth, trnnt, grnnt, tmp_path):
    """tests/cpp_rnnt_check.cpp: parakeet::RNNTTranscriber t(weights, vocab, config); t.transcribe(samples, true)."""
    root = os.path.dirname(HERE)
    exe = str(tmp_path / "cpp_rnnt_check")
    libdir = os.path.dirname(pkg.lib_path())
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), os.path.join(HERE, "cpp_rnnt_check.cpp"),
                    "-L" + libdir, "-lparakeet_b200", "-Wl,-rpath," + libdir, "-o", exe], check=True)
    k = "tiny.c2."
    pcm = synth.make_audio(*(int(v) for v in grnnt[k + "n_samples"]))
    raw = str(tmp_path / "a.f32")
    pcm.astype(np.float32).tofile(raw)
    m = trnnt["tiny"]
    out = subprocess.run([exe, m.weights_path, m.vocab_path, raw], check=True, capture_output=True, text=True).stdout.strip().split("\n")
    assert out[0].split()[1:] == [f"{a}:{b}:{c}" for a, b, c in grnnt[k + "tok"].tolist()]
    assert out[1] == "TEXT " + pkg.engine.Tokenizer(m.vocab_path).decode(grnnt[k + "ids"].tolist())
