"""Generates the fixtures under tests/golden/ from the UNMODIFIED reference, compiled into
oracle/_ref/libpkref.so by oracle/Makefile (REF=<path of the reference sources>).

    python tests/golden/make_golden.py [boost|stream|refcalls|600m|600m_extra|600m_long|110m_extra]

The reference ships no numeric golden vectors for mel / encoder (SURVEY.md section 4:
its tests pin shapes and decode-loop logic only), so these are produced by running
the reference itself on seeded synthetic checkpoints / audio
(parakeet.cpp_b200/synth.py; same seeds as the tests' fixtures).  The fixtures pin
oracle/oracle.py (tests/test_oracle.py, CPU) and the CUDA path (tests/test_gpu_parity.py).
The reference is not needed to *consume* the fixtures.
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import __graft_entry__ as ge  # noqa: E402
import oracle as O  # noqa: E402
import refbind as R  # noqa: E402

ge.load_package()
from parakeet_cpp_b200 import synth  # noqa: E402


def toks_arr(toks):
    return np.array([[t[0], t[1], t[2]] for t in toks], np.int32).reshape(-1, 3), \
        np.array([t[3] for t in toks], np.float32)


def run_model(out, tag, ocfg, seed, clips, td, custom, preset=0):
    W = synth.make_weights(ocfg, seed=seed)
    wp = os.path.join(td, tag + ".safetensors")
    synth.save_safetensors(wp, W)
    pieces = synth.make_vocab(ocfg.vocab - 1, seed=seed)
    vp = os.path.join(td, tag + ".vocab.txt")
    synth.save_vocab(vp, pieces)
    m = R.RefModel(wp, vp, preset, cfg=ocfg if custom else None)
    for ci, (n, aseed) in enumerate(clips):
        k = f"{tag}.c{ci}."
        pcm = synth.make_audio(n, aseed)
        feats = R.mel(pcm, ocfg.mel_bins)
        T = O.encoder_len(feats.shape[0])
        sub, lay = m.encode_layers(feats, ocfg.d_model, ocfg.n_layers, T)
        enc = m.encode(feats, ocfg.d_model)
        assert np.array_equal(enc, lay[-1])
        if ocfg.has_ctc:
            lp = m.ctc_logprobs(enc, ocfg.vocab)
            ctc = R.ctc_greedy(lp, ocfg.vocab - 1, True)[0]
        else:
            lp, ctc = np.zeros((enc.shape[0], 1), np.float32), []
        tdt = m.tdt_greedy(enc, True)
        out[k + "n_samples"] = np.array([n, aseed], np.int64)
        out[k + "mel"] = feats.astype(np.float16) if feats.size > 50000 else feats
        out[k + "mel_stats"] = np.array([feats.mean(), feats.std(), np.abs(feats).max(), feats[::7, ::3].sum()], np.float64)
        out[k + "sub"] = sub if sub.size < 70000 else sub[::8]
        out[k + "layers_first_last"] = np.stack([lay[0], lay[-1]]) if lay[0].size < 70000 else np.stack([lay[0][::8], lay[-1][::8]])
        out[k + "enc"] = enc
        out[k + "ctc_lp_max"] = lp.max(axis=1)
        out[k + "ctc_argmax"] = lp.argmax(axis=1).astype(np.int32)
        out[k + "ctc_tok"], out[k + "ctc_conf"] = toks_arr(ctc)
        out[k + "tdt_tok"], out[k + "tdt_conf"] = toks_arr(tdt)
        out[k + "ctc_text"] = np.frombuffer(m.detok([t[0] for t in ctc]).encode(), np.uint8)
        out[k + "tdt_text"] = np.frombuffer(m.detok([t[0] for t in tdt]).encode(), np.uint8)
        words = m.group_words(tdt)
        out[k + "tdt_words"] = np.frombuffer("\n".join(w[0] for w in words).encode(), np.uint8)
        out[k + "tdt_word_times"] = np.array([[w[1], w[2], w[3]] for w in words], np.float32).reshape(-1, 3)
        print(tag, ci, "frames", feats.shape[0], "T", T, "ctc", len(ctc), "tdt", len(tdt))
    m.close()


def main():
    out = {}
    out["posemb_5_4"] = R.posemb(5, 4)
    out["posemb_10_64"] = R.posemb(10, 64)
    # decode-loop vectors of the reference's own tests (tests/test_all.cpp:759-872), run
    # through the reference to record the full timestamped answers
    V = 1025
    for name, pattern in (("collapse", [10, 10, 1024, 10, 10, 20]), ("with_ts", [5, 5, 1024, 8, 8, 8]),
                          ("all_blank", [1024] * 10), ("single", [42, 42, 42, 1024, 1024])):
        lp = np.full((len(pattern), V), -10.0, np.float32)
        for t, p in enumerate(pattern):
            lp[t, p] = 0.0
        r = R.ctc_greedy(lp, 1024, True)[0]
        out[f"ctc_ka.{name}.pattern"] = np.array(pattern, np.int32)
        out[f"ctc_ka.{name}.tok"], out[f"ctc_ka.{name}.conf"] = toks_arr(r)
    with tempfile.TemporaryDirectory() as td:
        run_model(out, "tiny", O.make_tiny_config(), 3, [(32000, 11), (20000, 12), (400, 13), (64000, 14)], td, True)
        run_model(out, "m110", O.make_110m_config(), 0, [(160000, 1000)], td, False)
    # the 110m clip gets a file of its own (each fixture stays below 1 MB); its last layer is its encoder output,
    # stored once as m110.c0.enc
    k = "m110.c0."
    assert np.array_equal(out[k + "layers_first_last"][1], out[k + "enc"])
    out[k + "layer_first"] = out.pop(k + "layers_first_last")[0]
    m110 = {n: out.pop(n) for n in list(out) if n.startswith("m110.")}
    for name, d in (("golden_v1.npz", out), ("golden_110m_v1.npz", m110)):
        path = os.path.join(ROOT, "tests", "golden", name)
        np.savez_compressed(path, **d)
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main_600m():
    """tdt-600m preset (config.hpp:98-116): one 4 s clip through the compiled reference."""
    out = {}
    with tempfile.TemporaryDirectory() as td:
        run_model(out, "m600", O.make_tdt_600m_config(), 0, [(64000, 2000)], td, False, preset=1)
    for k in list(out):
        if k.endswith(".mel") or k.endswith(".sub") or k.endswith("layers_first_last"):
            out[k] = out[k].astype(np.float16) if out[k].dtype == np.float32 and out[k].size > 70000 else out[k]
    path = os.path.join(ROOT, "tests", "golden", "golden_600m_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main_110m_extra():
    """More full-size (tdt-ctc-110m) clips through the compiled reference: tokens, frames, confidences, text only
    (token exactness of the bf16x3 path is the claim these pin; activations are covered by golden_v1)."""
    out = {}
    ocfg = O.make_110m_config()
    clips = [(48000, 1101), (112000, 1102), (160000, 1103), (80000, 1107)]
    clips += [(160000, 1000 + i) for i in range(16)]      # the first 16 clips of bench.py's 64 x 10 s batch
    with tempfile.TemporaryDirectory() as td:
        W = synth.make_weights(ocfg, seed=0)
        wp = os.path.join(td, "m110.safetensors")
        synth.save_safetensors(wp, W)
        pieces = synth.make_vocab(ocfg.vocab - 1, seed=0)
        vp = os.path.join(td, "m110.vocab.txt")
        synth.save_vocab(vp, pieces)
        m = R.RefModel(wp, vp, 0)
        kept = 0
        for n, aseed in clips:
            pcm = synth.make_audio(n, aseed)
            feats = R.mel(pcm, ocfg.mel_bins)
            enc = m.encode(feats, ocfg.d_model)
            lp = m.ctc_logprobs(enc, ocfg.vocab)
            ctc = R.ctc_greedy(lp, ocfg.vocab - 1, True)[0]
            try:
                tdt = m.tdt_greedy(enc, True)
            except Exception as ex:          # the reference livelocks / throws on this input: no oracle for TDT
                print("skip", n, aseed, type(ex).__name__, ex)
                continue
            k = f"x110.c{kept}."
            kept += 1
            out[k + "n_samples"] = np.array([n, aseed], np.int64)
            out[k + "ctc_tok"], out[k + "ctc_conf"] = toks_arr(ctc)
            out[k + "tdt_tok"], out[k + "tdt_conf"] = toks_arr(tdt)
            out[k + "ctc_text"] = np.frombuffer(m.detok([t[0] for t in ctc]).encode(), np.uint8)
            out[k + "tdt_text"] = np.frombuffer(m.detok([t[0] for t in tdt]).encode(), np.uint8)
            # margin statistics: how close the argmax decisions are (smallest top-2 gap over frames)
            srt = np.sort(lp, axis=1)
            out[k + "ctc_min_gap"] = np.array([(srt[:, -1] - srt[:, -2]).min()], np.float32)
            print("x110", kept - 1, n, aseed, "ctc", len(ctc), "tdt", len(tdt), "min ctc gap", float(out[k + "ctc_min_gap"][0]))
        m.close()
    out["n_clips"] = np.array([kept], np.int64)
    path = os.path.join(ROOT, "tests", "golden", "golden_110m_extra_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main_600m_extra():
    """Three more tdt-600m clips (tokens, frames, confidences, text only)."""
    out = {}
    ocfg = O.make_tdt_600m_config()
    clips = [(40000, 2001), (72000, 2002), (56000, 2003)]
    with tempfile.TemporaryDirectory() as td:
        W = synth.make_weights(ocfg, seed=0)
        wp = os.path.join(td, "m600.safetensors")
        synth.save_safetensors(wp, W)
        pieces = synth.make_vocab(ocfg.vocab - 1, seed=0)
        vp = os.path.join(td, "m600.vocab.txt")
        synth.save_vocab(vp, pieces)
        m = R.RefModel(wp, vp, 1)
        kept = 0
        for n, aseed in clips:
            pcm = synth.make_audio(n, aseed)
            feats = R.mel(pcm, ocfg.mel_bins)
            enc = m.encode(feats, ocfg.d_model)
            try:
                tdt = m.tdt_greedy(enc, True)
            except Exception as ex:
                print("skip", n, aseed, type(ex).__name__, ex)
                continue
            k = f"x600.c{kept}."
            kept += 1
            out[k + "n_samples"] = np.array([n, aseed], np.int64)
            out[k + "tdt_tok"], out[k + "tdt_conf"] = toks_arr(tdt)
            out[k + "tdt_text"] = np.frombuffer(m.detok([t[0] for t in tdt]).encode(), np.uint8)
            print("x600", kept - 1, n, aseed, "tdt", len(tdt))
        m.close()
    out["n_clips"] = np.array([kept], np.int64)
    path = os.path.join(ROOT, "tests", "golden", "golden_600m_extra_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def main_600m_long():
    """BASELINE config 3 (tdt-600m, 30 s clips, T' = 376) through the compiled reference: one full 30 s clip
    (mel statistics, every 4th encoder row, TDT tokens + frames + confidences, text) and one 21 s clip (tokens only)
    so that the GPU test can run a RAGGED batch at the configuration's full size.  The CPU reference needs
    several minutes per clip."""
    out = {}
    ocfg = O.make_tdt_600m_config()
    clips = [(480000, 1000), (336000, 3001)]      # clip 0 = clip 0 of bench.py's 16 x 30 s batch (seed 1000 + i)
    with tempfile.TemporaryDirectory() as td:
        W = synth.make_weights(ocfg, seed=0)
        wp = os.path.join(td, "m600.safetensors")
        synth.save_safetensors(wp, W)
        pieces = synth.make_vocab(ocfg.vocab - 1, seed=0)
        vp = os.path.join(td, "m600.vocab.txt")
        synth.save_vocab(vp, pieces)
        m = R.RefModel(wp, vp, 1)
        kept = 0
        for n, aseed in clips:
            pcm = synth.make_audio(n, aseed)
            feats = R.mel(pcm, ocfg.mel_bins)
            enc = m.encode(feats, ocfg.d_model)
            try:
                tdt = m.tdt_greedy(enc, True)
            except Exception as ex:
                print("skip", n, aseed, type(ex).__name__, ex)
                continue
            k = f"l600.c{kept}."
            kept += 1
            out[k + "n_samples"] = np.array([n, aseed], np.int64)
            out[k + "mel_stats"] = np.array([feats.mean(), feats.std(), np.abs(feats).max(), feats[::7, ::3].sum()], np.float64)
            out[k + "enc_rows4"] = enc[::4].copy()
            out[k + "enc_T"] = np.array([enc.shape[0]], np.int64)
            out[k + "tdt_tok"], out[k + "tdt_conf"] = toks_arr(tdt)
            out[k + "tdt_text"] = np.frombuffer(m.detok([t[0] for t in tdt]).encode(), np.uint8)
            print("l600", kept - 1, n, aseed, "T", enc.shape[0], "tdt", len(tdt), flush=True)
        m.close()
    out["n_clips"] = np.array([kept], np.int64)
    path = os.path.join(ROOT, "tests", "golden", "golden_600m_long_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


STREAM_SCHEDULE = [2560, 2560, 2560, 1000, 4000, 2560, 2560, 2560, 2560, 5000, 2560, 2560, 2560, 2560, 2560, 2560, 2560]


def main_stream():
    """Streaming path (eou-120m; SURVEY section 8f row 2) through the compiled reference, chunk by chunk:
    StreamingAudioPreprocessor -> forward_chunk -> rnnt_streaming_decode_chunk (oracle/ref_harness_stream.cpp).
    The oracle is run FIRST on every model: the reference would hang on a livelocking decode."""
    out = {}
    with tempfile.TemporaryDirectory() as td:
        for tag, ocfg, wseed, aseed, sched in (("tstream", O.make_tiny_stream_config(), 3, 77, STREAM_SCHEDULE),
                                               ("eou120", O.make_eou_120m_config(), 0, 1200, [2560] * 14)):
            W = synth.make_weights(ocfg, seed=wseed)
            pcm = synth.make_audio(sum(sched), aseed)
            pre, cache, st = O.StreamingPreprocessor(ocfg.mel_bins), O.StreamEncoderCache(ocfg.n_layers), O.StreamDecodeState(ocfg)
            pos = 0
            for n in sched:                                   # raises RuntimeError on a livelock
                f = pre.process_chunk(pcm[pos:pos + n]); pos += n
                e = O.stream_encoder_chunk(W, f, cache, ocfg) if f is not None else None
                if e is not None:
                    O.stream_decode_chunk(W, e, st, ocfg, max_steps=5000)
            wp = os.path.join(td, tag + ".safetensors")
            synth.save_safetensors(wp, W)
            rs = R.RefStream(wp, ocfg)
            pos, ntok = 0, 0
            out[tag + ".schedule"] = np.array(sched, np.int64)
            out[tag + ".seeds"] = np.array([wseed, aseed], np.int64)
            for ci, n in enumerate(sched):
                f, e, toks = rs.chunk(pcm[pos:pos + n]); pos += n
                k = f"{tag}.k{ci}."
                out[k + "feats"] = f if f is not None else np.zeros((0, ocfg.mel_bins), np.float32)
                out[k + "enc"] = e if e is not None else np.zeros((0, ocfg.d_model), np.float32)
                out[k + "tok"], out[k + "conf"] = toks_arr(toks)
                ntok += len(toks)
            rs.close()
            print(tag, "chunks", len(sched), "tokens", ntok)
    path = os.path.join(ROOT, "tests", "golden", "golden_stream_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def sha256(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).digest(), np.uint8)


# the resampler inputs of tests/test_abi.py::test_resample_matches_oracle_and_reference (seed 4) and
# tests/test_gpu_parity.py::test_gpu_resampler_matches_oracle_and_feeds_the_path (seed 9), drawn in the same order
RESAMPLE_HOST = [(44100, 16000, 9000), (48000, 16000, 5001), (8000, 16000, 2500), (22050, 16000, 3000), (24000, 16000, 999),
                 (96000, 16000, 6000), (16000, 16000, 50), (11025, 16000, 3), (16000, 8000, 1000), (44100, 16000, 0)]
RESAMPLE_DEVICE = [(44100, 16000, [9000, 3, 20000]), (48000, 16000, [5001]), (8000, 16000, [2500, 1]), (22050, 16000, [30000, 12345]),
                   (96000, 16000, [6000]), (16000, 8000, [1000]), (11025, 16000, [4097])]
REF_STREAM_SCHEDULE = [2560, 3000, 800, 2560, 6000, 2560, 2560]


def main_refcalls():
    """What the oracle tests compare with single calls into the compiled reference: the tiny model's mel, subsampling,
    per-layer encoder output and TDT decode of one 3 s clip; one tiny streaming model chunk by chunk; boosted CTC greedy
    on random phrase sets; and parakeet::resample, stored as SHA-256 digests of its fp32 output (those comparisons
    are bit-exact)."""
    out = {}
    with tempfile.TemporaryDirectory() as td:
        ocfg = O.make_tiny_config()
        W = synth.make_weights(ocfg, seed=3)
        wp, vp = os.path.join(td, "tiny.safetensors"), os.path.join(td, "tiny.vocab.txt")
        synth.save_safetensors(wp, W)
        synth.save_vocab(vp, synth.make_vocab(ocfg.vocab - 1, seed=3))
        m = R.RefModel(wp, vp, 0, cfg=ocfg)
        n, aseed = 48000, 22
        feats = R.mel(synth.make_audio(n, aseed))
        sub, lay = m.encode_layers(feats, ocfg.d_model, ocfg.n_layers, O.encoder_len(feats.shape[0]))
        out["tiny.n_samples"] = np.array([n, aseed], np.int64)
        out["tiny.mel"], out["tiny.sub"], out["tiny.layers"] = feats, sub, lay
        out["tiny.tdt_tok"], out["tiny.tdt_conf"] = toks_arr(m.tdt_greedy(lay[-1], True))
        # boosted CTC greedy on the oracle's log-probs of golden clip 1
        g = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))
        lp = O.ctc_log_probs(W, g["tiny.c1.enc"])
        rng = np.random.default_rng(23)
        for i in range(5):
            phrases = [rng.integers(0, ocfg.vocab - 1, size=int(rng.integers(1, 5))).tolist() for _ in range(8)]
            k = f"boost.k{i}."
            out[k + "clip"], out[k + "boost"] = np.array([1], np.int64), np.array([4.0], np.float32)
            out[k + "ph_ids"] = np.array([t for ph in phrases for t in ph], np.int32)
            out[k + "ph_len"] = np.array([len(ph) for ph in phrases], np.int32)
            out[k + "ctc_tok"], _ = toks_arr(R.ctc_greedy_boosted(lp, ocfg.vocab - 1, phrases, 4.0))
        out["boost.n_cases"] = np.array([5], np.int64)
        m.close()
        # streaming: the oracle first (the reference would hang on a livelocking decode)
        scfg = O.make_tiny_stream_config()
        wseed, aseed, sched = 9, 91, REF_STREAM_SCHEDULE
        Ws = synth.make_weights(scfg, seed=wseed)
        pcm = synth.make_audio(sum(sched), aseed)
        pre, cache, st = O.StreamingPreprocessor(scfg.mel_bins), O.StreamEncoderCache(scfg.n_layers), O.StreamDecodeState(scfg)
        pos = 0
        for n in sched:
            f = pre.process_chunk(pcm[pos:pos + n]); pos += n
            e = O.stream_encoder_chunk(Ws, f, cache, scfg) if f is not None else None
            if e is not None:
                O.stream_decode_chunk(Ws, e, st, scfg, max_steps=5000)
        wps = os.path.join(td, "tstream9.safetensors")
        synth.save_safetensors(wps, Ws)
        rs = R.RefStream(wps, scfg)
        out["stream.seeds"], out["stream.schedule"] = np.array([wseed, aseed], np.int64), np.array(sched, np.int64)
        pos = 0
        for ci, n in enumerate(sched):
            f, e, toks = rs.chunk(pcm[pos:pos + n]); pos += n
            k = f"stream.k{ci}."
            out[k + "feats"] = f if f is not None else np.zeros((0, scfg.mel_bins), np.float32)
            out[k + "enc"] = e if e is not None else np.zeros((0, scfg.d_model), np.float32)
            out[k + "tok"], _ = toks_arr(toks)
        rs.close()
    rng = np.random.default_rng(4)
    for sr, dr, n in RESAMPLE_HOST:
        x = (rng.standard_normal(n) * 0.3).astype(np.float32)
        if n > 0:
            out[f"resample_host.{sr}.{dr}.{n}.sha256"] = sha256(R.resample(x, sr, dr))
    rng = np.random.default_rng(9)
    for sr, dr, lens in RESAMPLE_DEVICE:
        for n in lens:
            x = (rng.standard_normal(n) * 0.3).astype(np.float32)
            if n > 16:
                y = R.resample(x, sr, dr)
                assert np.array_equal(y, O.sinc_resample(x, sr, dr))      # the GPU test compares with the oracle's output
                out[f"resample_device.{sr}.{dr}.{n}.sha256"] = sha256(y)
    path = os.path.join(ROOT, "tests", "golden", "golden_refcalls_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def boost_cases(vocab, base_ctc, rng):
    """Phrase sets for the boosted-decode fixtures: random short phrases plus one that continues a prefix of the
    unboosted output (so that deeper trie states are visited)."""
    phrases = [rng.integers(0, vocab - 1, size=int(rng.integers(1, 4))).tolist() for _ in range(6)]
    if len(base_ctc) > 4:
        k = int(rng.integers(0, len(base_ctc) - 3))
        phrases.append([int(v) for v in base_ctc[k:k + 2]] + [int(rng.integers(0, vocab - 1))])
    return phrases, float(rng.choice([2.0, 5.0, 9.0]))


def main_boost():
    """Phrase-boosted CTC / TDT decode (src/phrase_boost.cpp; SURVEY section 8f row 3) through the compiled reference,
    on the tiny model's golden encoder outputs.  TDT cases on which the ORACLE detects the livelock are recorded as
    such and never sent to the reference (it would hang)."""
    out = {}
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))
    ocfg = O.make_tiny_config()
    with tempfile.TemporaryDirectory() as td:
        W = synth.make_weights(ocfg, seed=3)
        wp = os.path.join(td, "tiny.safetensors")
        synth.save_safetensors(wp, W)
        pieces = synth.make_vocab(ocfg.vocab - 1, seed=3)
        vp = os.path.join(td, "tiny.vocab.txt")
        synth.save_vocab(vp, pieces)
        m = R.RefModel(wp, vp, 0, cfg=ocfg)
        rng = np.random.default_rng(11)
        n = 0
        for ci in (0, 1, 3):
            enc = g[f"tiny.c{ci}.enc"]
            lp = m.ctc_logprobs(enc, ocfg.vocab)
            base = [t[0] for t in R.ctc_greedy(lp, ocfg.vocab - 1, True)[0]]
            for _ in range(4):
                phrases, boost = boost_cases(ocfg.vocab, base, rng)
                k = f"boost.k{n}."
                n += 1
                out[k + "clip"] = np.array([ci], np.int64)
                out[k + "boost"] = np.array([boost], np.float32)
                out[k + "ph_ids"] = np.array([t for ph in phrases for t in ph], np.int32)
                out[k + "ph_len"] = np.array([len(ph) for ph in phrases], np.int32)
                out[k + "ctc_tok"], out[k + "ctc_conf"] = toks_arr(R.ctc_greedy_boosted(lp, ocfg.vocab - 1, phrases, boost))
                try:
                    O.tdt_greedy_decode_with_timestamps_boosted(W, enc, ocfg, O.ContextTrie(phrases), boost, max_steps=3000)
                    tdt, live = R.tdt_greedy_boosted(m, enc, phrases, boost), 0
                except RuntimeError:
                    tdt, live = [], 1
                out[k + "tdt_tok"], out[k + "tdt_conf"] = toks_arr(tdt)
                out[k + "tdt_livelock"] = np.array([live], np.int64)
                print(k, "boost", boost, "ctc", len(out[k + "ctc_tok"]), "tdt", len(tdt), "livelock" if live else "")
        out["n_cases"] = np.array([n], np.int64)
        # Tokenizer::encode known answers on the synthetic vocabulary
        texts = [" ".join(p.replace(O.SP_MARK, " ").strip() for p in pieces[3:9]), "zz " + pieces[5].replace(O.SP_MARK, ""), ""]
        for i, tx in enumerate(texts):
            out[f"enc.k{i}.text"] = np.frombuffer(tx.encode(), np.uint8)
            out[f"enc.k{i}.ids"] = np.array(R.tok_encode(m, tx) if tx else [], np.int32)
        out["n_texts"] = np.array([len(texts)], np.int64)
        m.close()
    path = os.path.join(ROOT, "tests", "golden", "golden_boost_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "boost":
        main_boost()
    elif len(sys.argv) > 1 and sys.argv[1] == "stream":
        main_stream()
    elif len(sys.argv) > 1 and sys.argv[1] == "refcalls":
        main_refcalls()
    elif len(sys.argv) > 1 and sys.argv[1] == "600m_extra":
        main_600m_extra()
    elif len(sys.argv) > 1 and sys.argv[1] == "110m_extra":
        main_110m_extra()
    elif len(sys.argv) > 1 and sys.argv[1] == "600m_long":
        main_600m_long()
    elif len(sys.argv) > 1 and sys.argv[1] == "600m":
        main_600m()
    else:
        main()
