"""CPU tests that PIN THE ORACLE (oracle/oracle.py) before it is trusted:
  (1) the reference's own known-answer tests that apply at this boundary
      (the reference's tests/test_all.cpp: CTCDecode.* :759-872, PositionEmbedding.* :1003-1030,
       GroupTimestamps.* / TimestampTypes.* :45-129, Tokenizer.DecodeOutOfRange :470-477),
  (2) golden vectors produced by the unmodified reference
      (tests/golden/golden_*.npz <- tests/golden/make_golden.py),
  (3) recorded single calls into the compiled reference (tests/golden/golden_refcalls_v1.npz).
"""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lp_from_pattern(pattern, V=1025):
    lp = np.full((len(pattern), V), -10.0, np.float32)
    for t, p in enumerate(pattern):
        lp[t, p] = 0.0
    return lp


# ---------------------------------------------------------------- (1) reference known-answer tests
def test_ctc_all_blanks(O):                       # CTCDecode.AllBlanks
    assert O.ctc_greedy_decode(_lp_from_pattern([1024] * 10)) == []


def test_ctc_single_token(O):                     # CTCDecode.SingleToken
    assert O.ctc_greedy_decode(_lp_from_pattern([42, 42, 42, 1024, 1024])) == [42]


def test_ctc_collapse_repeats(O):                 # CTCDecode.CollapseRepeats
    assert O.ctc_greedy_decode(_lp_from_pattern([10, 10, 1024, 10, 10, 20])) == [10, 10, 20]


def test_ctc_with_timestamps(O):                  # CTCDecode.WithTimestamps
    r = O.ctc_greedy_decode_with_timestamps(_lp_from_pattern([5, 5, 1024, 8, 8, 8]))
    assert [(t[0], t[1]) for t in r] == [(5, 0), (8, 3)]


def test_ctc_batch(O):                            # CTCDecode.BatchDecode
    assert O.ctc_greedy_decode(_lp_from_pattern([5] * 4)) == [5]
    assert O.ctc_greedy_decode(_lp_from_pattern([1024] * 4)) == []


def test_ctc_first_max_wins(O):                   # strict '>' scan, ctc.cpp:59-66
    lp = np.zeros((1, 1025), np.float32)
    assert O.ctc_greedy_decode(lp) == [0]


def test_posemb_shape_values_center(O):           # PositionEmbedding.{Shape,Values,CenterRow}
    pe = O.sinusoidal_position_embedding(10, 64)
    assert pe.shape == (19, 64)
    pe = O.sinusoidal_position_embedding(5, 4)
    assert np.all(pe >= -1.001) and np.all(pe <= 1.001)
    assert abs(pe[4, 0]) < 1e-5


def test_frame_to_seconds_and_grouping(O):        # TimestampTypes.FrameToSeconds, GroupTimestamps.*
    M = O.SP_MARK
    assert O.group_timestamps([], []) == []
    w = O.group_timestamps([(0, 5, 10, 1.0)], [M + "hello"])
    assert len(w) == 1 and w[0][0] == "hello"
    assert w[0][1] == pytest.approx(np.float32(5) * np.float32(0.08)) and w[0][2] == pytest.approx(0.8)
    w = O.group_timestamps([(0, 0, 2, 1.0), (1, 5, 8, 1.0), (2, 12, 15, 1.0)], [M + "the", M + "quick", M + "fox"])
    assert [x[0] for x in w] == ["the", "quick", "fox"]
    w = O.group_timestamps([(0, 0, 3, 0.9), (1, 4, 6, 0.5)], [M + "run", "ning"])
    assert len(w) == 1 and w[0][0] == "running" and w[0][1] == 0.0
    assert w[0][2] == pytest.approx(np.float32(6) * np.float32(0.08)) and w[0][3] == pytest.approx(0.5)
    w = O.group_timestamps([(999, 0, 1, 1.0), (0, 2, 4, 1.0)], [M + "hello"])      # OutOfRangeTokenId
    assert len(w) == 1 and w[0][0] == "hello"


def test_detokenize(O):                           # Tokenizer.DecodeEmpty / DecodeOutOfRange
    M = O.SP_MARK
    assert O.detokenize([], ["a"]) == ""
    assert O.detokenize([9999], ["a"]) == "[9999]"
    assert O.detokenize([0, 1, 2], [M + "he", "llo", M + "you"]) == "hello you"


def test_preset_values(O):                        # Config.* (test_all.cpp:135-194)
    c = O.make_110m_config()
    assert (c.d_model, c.n_layers, c.n_heads, c.ff, c.vocab, c.lstm_layers, c.pred_hidden) == (512, 17, 8, 2048, 1025, 1, 640)
    c = O.make_tdt_600m_config()
    assert (c.mel_bins, c.d_model, c.n_layers, c.ff, c.vocab, c.lstm_layers) == (128, 1024, 24, 4096, 8193, 2)


# ---------------------------------------------------------------- (2) golden vectors from the compiled reference
def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def test_golden_posemb(O, golden):
    assert np.abs(O.sinusoidal_position_embedding(5, 4) - golden["posemb_5_4"]).max() < 2e-6
    assert np.abs(O.sinusoidal_position_embedding(10, 64) - golden["posemb_10_64"]).max() < 2e-6


@pytest.mark.parametrize("name", ["collapse", "with_ts", "all_blank", "single"])
def test_golden_ctc_known_answers(O, golden, name):
    lp = _lp_from_pattern(golden[f"ctc_ka.{name}.pattern"])
    r = O.ctc_greedy_decode_with_timestamps(lp)
    tok = golden[f"ctc_ka.{name}.tok"]
    assert [[t[0], t[1], t[2]] for t in r] == tok.tolist()
    assert np.allclose([t[3] for t in r], golden[f"ctc_ka.{name}.conf"], rtol=1e-6)


def _golden_clip(O, synth, golden, tag, ci, ocfg, seed):
    k = f"{tag}.c{ci}."
    n, aseed = (int(v) for v in golden[k + "n_samples"])
    W = synth.make_weights(ocfg, seed=seed)
    pcm = synth.make_audio(n, aseed)
    return k, W, pcm


@pytest.mark.parametrize("ci", [0, 1, 2, 3])
def test_golden_tiny_whole_path(O, synth, golden, ci):
    ocfg = O.make_tiny_config()
    k, W, pcm = _golden_clip(O, synth, golden, "tiny", ci, ocfg, 3)
    feats = O.preprocess_audio(pcm, ocfg.mel_bins)
    assert feats.shape == golden[k + "mel"].shape
    if feats.shape[0] > 3:   # the 3-frame clip has near-zero variance bins: 1/(sigma+1e-5) amplifies fp32 noise
        assert np.abs(feats - golden[k + "mel"]).max() < 2e-3
    enc, sub, lay = O.encoder_forward(W, golden[k + "mel"].astype(np.float32), ocfg, return_layers=True)
    assert _rel(sub, golden[k + "sub"]) < 2e-5
    assert _rel(lay[0], golden[k + "layers_first_last"][0]) < 2e-5
    assert _rel(enc, golden[k + "enc"]) < 5e-5
    genc = golden[k + "enc"]
    lp = O.ctc_log_probs(W, genc)
    assert np.array_equal(lp.argmax(1), golden[k + "ctc_argmax"])
    assert np.abs(lp.max(1) - golden[k + "ctc_lp_max"]).max() < 1e-4
    ctc = O.ctc_greedy_decode_with_timestamps(lp, ocfg.vocab - 1)
    assert [[t[0], t[1], t[2]] for t in ctc] == golden[k + "ctc_tok"].tolist()
    assert np.allclose([t[3] for t in ctc], golden[k + "ctc_conf"], rtol=1e-4)
    tdt = O.tdt_greedy_decode(W, genc, ocfg, with_timestamps=True)
    assert [[t[0], t[1], t[2]] for t in tdt] == golden[k + "tdt_tok"].tolist()
    assert np.allclose([t[3] for t in tdt], golden[k + "tdt_conf"], rtol=1e-4)
    pieces = synth.make_vocab(ocfg.vocab - 1, seed=3)
    assert O.detokenize([t[0] for t in tdt], pieces) == bytes(golden[k + "tdt_text"]).decode()
    words = O.group_timestamps(tdt, pieces)
    assert "\n".join(w[0] for w in words) == bytes(golden[k + "tdt_words"]).decode()
    if words:
        assert np.allclose(np.array([[w[1], w[2], w[3]] for w in words], np.float32), golden[k + "tdt_word_times"], rtol=1e-4)


def test_golden_110m_decode(O, synth, golden):
    """110m: decode-side check on the reference's encoder output (the encoder itself is
    covered at the tiny shape above and, when _ref is present, live below)."""
    ocfg = O.make_110m_config()
    k, W, pcm = _golden_clip(O, synth, golden, "m110", 0, ocfg, 0)
    feats = O.preprocess_audio(pcm, ocfg.mel_bins)
    assert np.abs(feats - golden[k + "mel"].astype(np.float32)).max() < 5e-3     # stored as fp16
    st = golden[k + "mel_stats"]
    assert abs(feats[::7, ::3].sum() - st[3]) < 0.5 and abs(np.abs(feats).max() - st[2]) < 1e-2
    genc = golden[k + "enc"]
    lp = O.ctc_log_probs(W, genc)
    assert np.array_equal(lp.argmax(1), golden[k + "ctc_argmax"])
    ctc = O.ctc_greedy_decode_with_timestamps(lp, ocfg.vocab - 1)
    assert [[t[0], t[1], t[2]] for t in ctc] == golden[k + "ctc_tok"].tolist()
    tdt = O.tdt_greedy_decode(W, genc, ocfg, with_timestamps=True)
    assert [[t[0], t[1], t[2]] for t in tdt] == golden[k + "tdt_tok"].tolist()
    pieces = synth.make_vocab(ocfg.vocab - 1, seed=0)
    assert O.detokenize([t[0] for t in ctc], pieces) == bytes(golden[k + "ctc_text"]).decode()


# ---------------------------------------------------------------- (3) recorded calls into the compiled reference
def test_live_reference_tiny(O, synth, tiny, golden_refcalls):
    """The reference's mel, subsampling, per-layer encoder output and TDT decode of one 3 s clip (tiny model)."""
    g = golden_refcalls
    n, aseed = (int(v) for v in g["tiny.n_samples"])
    pcm = synth.make_audio(n, aseed)
    fr = g["tiny.mel"]
    fo = O.preprocess_audio(pcm)
    assert np.abs(fr - fo).max() < 2e-3
    sub_r, lay_r = g["tiny.sub"], g["tiny.layers"]
    assert lay_r.shape[1] == O.encoder_len(fr.shape[0])
    enc_o, sub_o, lay_o = O.encoder_forward(tiny.W, fr, tiny.ocfg, return_layers=True)
    assert _rel(sub_o, sub_r) < 2e-5
    for i in range(tiny.ocfg.n_layers):
        assert _rel(lay_o[i], lay_r[i]) < 5e-5
    ref_tdt = [(int(a), int(b), int(c), float(d)) for (a, b, c), d in zip(g["tiny.tdt_tok"], g["tiny.tdt_conf"])]
    oracle_tdt = O.tdt_greedy_decode(tiny.W, lay_r[-1], tiny.ocfg, with_timestamps=True)
    assert ref_tdt[:50] == [tuple(t) for t in oracle_tdt][:50] or [t[:3] for t in ref_tdt] == [tuple(t[:3]) for t in oracle_tdt]


def test_golden_600m_decode(O, synth):
    """tdt-600m preset: the oracle's 2-layer LSTM / 8193-label TDT decode on the reference's encoder output."""
    import os
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_600m_v1.npz")
    if not os.path.exists(p):
        pytest.skip("600m golden not generated")
    g = np.load(p)
    ocfg = O.make_tdt_600m_config()
    specs = {n: s for n, s, _ in synth.tensor_specs(ocfg)}
    rng_needed = [n for n in specs if n.startswith("prediction_.") or n.startswith("joint_.")]
    W = synth.make_weights(ocfg, seed=0)
    tdt = O.tdt_greedy_decode({k: W[k] for k in rng_needed}, g["m600.c0.enc"], ocfg, with_timestamps=True)
    assert [[t[0], t[1], t[2]] for t in tdt] == g["m600.c0.tdt_tok"].tolist()
    assert np.allclose([t[3] for t in tdt], g["m600.c0.tdt_conf"], rtol=1e-4)


# ------------------------------------------------------------------ streaming path (eou-120m; SURVEY 8f row 2)
def _run_stream_oracle(O, synth, W, ocfg, pcm, sched):
    pre, cache, st = O.StreamingPreprocessor(ocfg.mel_bins), O.StreamEncoderCache(ocfg.n_layers), O.StreamDecodeState(ocfg)
    pos, out = 0, []
    for n in sched:
        f = pre.process_chunk(pcm[pos:pos + n])
        pos += n
        e = O.stream_encoder_chunk(W, f, cache, ocfg) if f is not None else None
        t = O.stream_decode_chunk(W, e, st, ocfg, max_steps=5000) if e is not None else []
        out.append((f, e, t))
    return out


def _rel(a, b):
    return float(np.abs(a - b).max() / max(float(np.abs(b).max()), 1e-9))


@pytest.mark.parametrize("tag", ["tstream", "eou120"])
def test_golden_streaming_chunks(O, synth, tag):
    """The streaming restatement (StreamingPreprocessor, stream_encoder_chunk, stream_decode_chunk) against the
    compiled reference's chunk-by-chunk outputs (tests/golden/make_golden.py stream): frame-count quirk (13/14
    frames per 2560 samples), leftover-frame cache, K/V and conv caches, un-shifted position scores, the
    ineffective CPU context mask, carried LSTM state, absolute frame numbers."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_stream_v1.npz"))
    ocfg = O.make_tiny_stream_config() if tag == "tstream" else O.make_eou_120m_config()
    wseed, aseed = (int(v) for v in g[tag + ".seeds"])
    sched = [int(v) for v in g[tag + ".schedule"]]
    W = synth.make_weights(ocfg, seed=wseed)
    pcm = synth.make_audio(sum(sched), aseed)
    n_tok = 0
    for ci, (f, e, t) in enumerate(_run_stream_oracle(O, synth, W, ocfg, pcm, sched)):
        k = f"{tag}.k{ci}."
        gf, ge_, gt, gc = g[k + "feats"], g[k + "enc"], g[k + "tok"], g[k + "conf"]
        assert (0 if f is None else f.shape[0]) == gf.shape[0]
        if gf.shape[0]:
            assert _rel(f, gf) < 1e-4
        assert (0 if e is None else e.shape[0]) == ge_.shape[0]
        if ge_.shape[0]:
            assert _rel(e, ge_) < 1e-4
        assert [list(x[:3]) for x in t] == gt.tolist()
        assert np.allclose([x[3] for x in t], gc, rtol=1e-3)
        n_tok += len(t)
    assert n_tok > 5


def test_streaming_context_mask_is_inert_in_the_reference(O, synth):
    """Documented reference quirk: on CPU the bounded-context mask of forward_cached never fills anything
    (float mask read bytewise), so the golden encoder output matches the oracle WITHOUT the mask and differs
    from the intended masked attention once a chunk has 3 frames."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_stream_v1.npz"))
    ocfg = O.make_tiny_stream_config()
    wseed, aseed = (int(v) for v in g["tstream.seeds"])
    sched = [int(v) for v in g["tstream.schedule"]]
    W = synth.make_weights(ocfg, seed=wseed)
    pcm = synth.make_audio(sum(sched), aseed)
    pre, cache = O.StreamingPreprocessor(ocfg.mel_bins), O.StreamEncoderCache(ocfg.n_layers)
    real = O.stream_attention_cached
    try:
        O.stream_attention_cached = lambda *a, **kw: real(*a, apply_context_mask=True, **kw)
        pos, worst = 0, 0.0
        for ci, n in enumerate(sched):
            f = pre.process_chunk(pcm[pos:pos + n])
            pos += n
            e = O.stream_encoder_chunk(W, f, cache, ocfg) if f is not None else None
            if e is not None:
                worst = max(worst, _rel(e, g[f"tstream.k{ci}.enc"]))
    finally:
        O.stream_attention_cached = real
    assert worst > 1e-3


def test_live_reference_streaming(O, synth, golden_refcalls):
    """The reference's streaming path chunk by chunk on a second tiny streaming model, with uneven chunk sizes."""
    g = golden_refcalls
    ocfg = O.make_tiny_stream_config()
    wseed, aseed = (int(v) for v in g["stream.seeds"])
    sched = [int(v) for v in g["stream.schedule"]]
    W = synth.make_weights(ocfg, seed=wseed)
    pcm = synth.make_audio(sum(sched), aseed)
    for ci, (f, e, t) in enumerate(_run_stream_oracle(O, synth, W, ocfg, pcm, sched)):
        k = f"stream.k{ci}."
        rf, re_, rt = g[k + "feats"], g[k + "enc"], g[k + "tok"]      # (no rows: the reference returned nothing)
        assert (len(rf) == 0) == (f is None) and (len(re_) == 0) == (e is None)
        if f is not None:
            assert _rel(f, rf) < 1e-4
        if e is not None:
            assert _rel(e, re_) < 1e-4
        assert rt.tolist() == [list(x[:3]) for x in t]


# ------------------------------------------------------------------ phrase-boosted decode (SURVEY 8f row 3)
def _boost_case(g, k):
    lens = g[k + "ph_len"].tolist()
    ids = g[k + "ph_ids"].tolist()
    phrases, p = [], 0
    for n in lens:
        phrases.append(ids[p:p + n])
        p += n
    return phrases, float(g[k + "boost"][0]), int(g[k + "clip"][0])


def test_context_trie_semantics(O):
    """ContextTrie (phrase_boost.cpp:9-66): shared prefixes share nodes, the root is always active, the boosted
    set is the union of the children of the active states."""
    t = O.ContextTrie([[1, 2, 3], [1, 2, 4], [5]])
    assert len(t.children) == 6                                   # root, 1, 1-2, 1-2-3, 1-2-4, 5
    assert t.boosted({0}) == {1, 5}
    a = t.advance({0}, 1)
    assert 0 in a and len(a) == 2 and t.boosted(a) == {1, 5, 2}
    a = t.advance(a, 2)
    assert t.boosted(a) == {1, 5, 3, 4}
    assert t.advance(a, 9) == {0}
    empty = O.ContextTrie([[]])
    assert len(empty.children) == 1 and empty.boosted({0}) == set()


def test_golden_boosted_decode(O, synth, golden):
    """ctc_/tdt_greedy_decode_with_timestamps_boosted restated in the oracle against the compiled reference
    (tests/golden/make_golden.py boost): boosted first-max argmax, trie advance on emission, raw-log-prob confidence."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_boost_v1.npz"))
    ocfg = O.make_tiny_config()
    W = synth.make_weights(ocfg, seed=3)
    changed = 0
    for n in range(int(g["n_cases"][0])):
        k = f"boost.k{n}."
        phrases, boost, ci = _boost_case(g, k)
        enc = golden[f"tiny.c{ci}.enc"]
        lp = O.ctc_log_probs(W, enc)
        trie = O.ContextTrie(phrases)
        got = O.ctc_greedy_decode_with_timestamps_boosted(lp, trie, boost, ocfg.vocab - 1)
        assert [list(x[:3]) for x in got] == g[k + "ctc_tok"].tolist()
        assert np.allclose([x[3] for x in got], g[k + "ctc_conf"], rtol=1e-3)
        changed += [x[0] for x in got] != [x[0] for x in O.ctc_greedy_decode_with_timestamps(lp, ocfg.vocab - 1)]
        if int(g[k + "tdt_livelock"][0]):
            with pytest.raises(RuntimeError):
                O.tdt_greedy_decode_with_timestamps_boosted(W, enc, ocfg, trie, boost, max_steps=3000)
        else:
            got = O.tdt_greedy_decode_with_timestamps_boosted(W, enc, ocfg, trie, boost, max_steps=3000)
            assert [list(x[:3]) for x in got] == g[k + "tdt_tok"].tolist()
            assert np.allclose([x[3] for x in got], g[k + "tdt_conf"], rtol=1e-3)
    assert changed >= 6                                           # the boosts really alter the decode
    pieces = synth.make_vocab(ocfg.vocab - 1, seed=3)
    for i in range(int(g["n_texts"][0])):                         # Tokenizer::encode (vocab.cpp:76-117)
        text = bytes(g[f"enc.k{i}.text"]).decode()
        assert O.tokenizer_encode(text, pieces) == g[f"enc.k{i}.ids"].tolist()
    assert len(g["enc.k0.ids"]) >= 4


def test_live_reference_boosted_ctc(O, synth, golden, golden_refcalls):
    """The reference's boosted CTC greedy decode with random sets of eight phrases."""
    g = golden_refcalls
    ocfg = O.make_tiny_config()
    W = synth.make_weights(ocfg, seed=3)
    for n in range(int(g["boost.n_cases"][0])):
        k = f"boost.k{n}."
        phrases, boost, ci = _boost_case(g, k)
        lp = O.ctc_log_probs(W, golden[f"tiny.c{ci}.enc"])
        got = O.ctc_greedy_decode_with_timestamps_boosted(lp, O.ContextTrie(phrases), boost, ocfg.vocab - 1)
        assert [list(x[:3]) for x in got] == g[k + "ctc_tok"].tolist()


def _boost_lp(pattern_or_none):
    V = 1025
    if pattern_or_none is not None:                      # BoostedCTCDecode.*EmptyTrie* (test_all.cpp:1369-1388, :1428-1452)
        return _lp_from_pattern(pattern_or_none, V)
    lp = np.full((3, V), -10.0, np.float32)              # BoostedCTCDecode.BoostFlipsDecision (test_all.cpp:1390-1426)
    lp[0, 42], lp[0, 43], lp[0, 1024] = -0.1, -0.2, -5.0
    lp[1, 1024] = lp[2, 1024] = 0.0
    return lp


def test_reference_known_answers_boosted_ctc_and_trie(O, pkg):
    """The reference's own phrase-boost tests (tests/test_all.cpp:1278-1452) on the oracle AND on the host C-ABI."""
    # ContextTrie.{EmptyTrie, InsertAndSize, GetBoostedTokens, Advance, AdvanceNonMatchingToken, MultiplePhrases}
    t = O.ContextTrie()
    assert len(t.children) == 1 and t.boosted({0}) == set()
    t.insert([10, 20, 30])
    assert len(t.children) == 4
    t.insert([10, 25])
    assert t.boosted({0}) == {10}
    nxt = t.advance({0}, 10)
    assert 0 in nxt and 20 in t.boosted(nxt)
    assert t.advance({0}, 999) == {0}
    m = O.ContextTrie([[10, 20], [10, 30], [40, 50]])
    assert m.boosted({0}) == {10, 40}
    assert {20, 30, 10, 40} <= m.boosted(m.advance({0}, 10))
    # BoostedCTCDecode.*
    for decode in (lambda lp, ph: [x[:2] for x in O.ctc_greedy_decode_with_timestamps_boosted(lp, O.ContextTrie(ph), 5.0, 1024)],
                   lambda lp, ph: [(x.token_id, x.start_frame) for x in pkg.engine.ctc_greedy_decode_boosted(lp, ph, 5.0, 1024)]):
        lp = _boost_lp([5, 5, 1024, 8, 8, 8])
        plain = [x[:2] for x in O.ctc_greedy_decode_with_timestamps(lp, 1024)]
        assert decode(lp, []) == plain == [(5, 0), (8, 3)]
        flip = _boost_lp(None)
        assert [x[0] for x in decode(flip, [])] == [42]
        assert [x[0] for x in decode(flip, [[43]])] == [43]
