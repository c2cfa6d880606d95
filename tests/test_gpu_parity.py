"""GPU parity tests: the CUDA path, called through the C-ABI (ctypes), against the oracle
on the same seeded inputs, against the committed golden fixtures produced by the
compiled reference, and -- at the BASELINE batch size -- through size-independent
properties (batch invariance, determinism).

Tolerances: tokens / frames / argmax are bit-exact; floating point uses the north-star
bound "encoder activations within 1e-3 rel fp32" (max-abs error / max-abs reference), and
tighter where the arithmetic is exact fp32.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ENC_TOL = 1e-3        # north_star tolerance for encoder activations
MEL_TOL = 2e-3        # abs, on unit-variance normalised features


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _tt(toks):
    return [(t.token_id, t.start_frame, t.end_frame) for t in toks]


MATH = {"bf16x3": 0, "fp32": 2}     # pk_math: the tcgen05 parity mode and the fp32 CUDA-core mode


@pytest.fixture(scope="module", params=["bf16x3", "fp32"])
def math_mode(request):
    return request.param


@pytest.fixture(scope="module")
def eng_tiny(pkg, tiny, math_mode):
    import dataclasses
    e = pkg.Engine(dataclasses.replace(tiny.cfg, math=MATH[math_mode]), tiny.weights_path, 0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def eng110(pkg, m110, math_mode):
    import dataclasses
    e = pkg.Engine(dataclasses.replace(m110.cfg, math=MATH[math_mode]), m110.weights_path, 0)
    yield e
    e.close()


# ------------------------------------------------------------------ tcgen05 GEMM kernel (K5) in isolation
EPI = dict(BIAS_F32=0, RELU_F32=1, RELU_ACT=2, SILU_ACT=3, RESID=4, GLU=5, BIAS_ACT=6, QKV=7)


@pytest.mark.parametrize("M,N,K,epi", [(128, 128, 64, "BIAS_F32"), (300, 256, 256, "RELU_F32"), (126, 1025, 512, "BIAS_F32"),
                                       (777, 2048, 512, "SILU_ACT"), (513, 512, 2048, "RESID"), (256, 1024, 512, "GLU"),
                                       (130, 64, 64, "BIAS_ACT"), (1, 640, 512, "BIAS_F32"), (8064, 512, 2560, "BIAS_F32"),
                                       (5020, 256, 256, "RELU_ACT"), (300, 384, 128, "QKV"), (8064, 1536, 512, "QKV")])
def test_tcgen05_gemm_matches_fp32_gemm(pkg, M, N, K, epi):
    from parakeet_cpp_b200.engine import selftest_gemm
    err, ref = selftest_gemm(M, N, K, EPI[epi], 0)
    assert err / ref < 5e-5, (err, ref)          # bf16 hi/lo split, 3 MMAs: ~16 mantissa bits
    err1, _ = selftest_gemm(M, N, K, EPI[epi], 1)
    assert err1 / ref < 2e-2                     # plain bf16 operands


@pytest.mark.parametrize("cl", ["2", "4"])
@pytest.mark.parametrize("M,N,K,epi", [(8064, 2048, 512, "SILU_ACT"), (8064, 1536, 512, "QKV"), (8064, 1024, 512, "GLU"), (777, 2048, 512, "SILU_ACT"),
                                       (130, 1024, 1024, "GLU"), (6016, 4096, 1024, "SILU_ACT")])
def test_tcgen05_gemm_cluster_multicast_matches_fp32_gemm(pkg, M, N, K, epi, cl, monkeypatch):
    """The wide GEMMs as clusters of 2 / 4 CTAs along N (PK_GEMM_CLUSTER): every CTA fetches a slice of the shared A tile and
    TMA-multicasts it into the stage of all CTAs of the cluster; stage release by a multicast tcgen05.commit from each of them."""
    from parakeet_cpp_b200.engine import selftest_gemm
    monkeypatch.setenv("PK_GEMM_CLUSTER", cl)
    err, ref = selftest_gemm(M, N, K, EPI[epi], 0)
    assert err / ref < 5e-5, (err, ref)


@pytest.mark.parametrize("M,N,K,epi", [(1, 640, 512, "BIAS_F32"), (2, 2048, 512, "SILU_ACT"), (64, 512, 2048, "RESID"), (128, 1536, 512, "QKV"),
                                       (100, 1024, 512, "GLU"), (126, 1025, 512, "BIAS_F32"), (17, 256, 256, "RELU_ACT"), (128, 512, 2560, "BIAS_F32"),
                                       (77, 384, 128, "QKV"), (128, 64, 64, "BIAS_ACT")])
def test_skinny_gemm_matches_fp32_gemm(pkg, M, N, K, epi, monkeypatch):
    """The few-row GEMM of the streaming path (csrc/gemm_skinny.cu: N x K-split CTAs, mma.sync bf16x3, slices reduced in
    a fixed order by the last CTA to arrive) against the fp32 CUDA-core GEMM, every epilogue kind, edge columns, two
    launches in a row (tickets reset)."""
    from parakeet_cpp_b200.engine import selftest_gemm
    monkeypatch.setenv("PK_SELFTEST_SKINNY", "1")
    err, ref = selftest_gemm(M, N, K, EPI[epi], 0)
    assert err / ref < 5e-5, (err, ref)
    err1, _ = selftest_gemm(M, N, K, EPI[epi], 1)
    assert err1 / ref < 2e-2


@pytest.mark.parametrize("M,K,mode", [(8064, 2048, 0), (8064, 512, 0), (8064, 2048, 1), (8064, 2048, 2), (8064, 2560, 3), (777, 512, 1),
                                      (129, 512, 0), (4000, 2048, 1)])
@pytest.mark.parametrize("mcast", ["1", "0"])
def test_fused_gemm_layernorm_matches_gemm_then_layernorm(pkg, M, K, mode, mcast, monkeypatch):
    """csrc/gemm_tc_ln.cu: the residual GEMM with the following LayerNorm(s) in its epilogue (4-CTA clusters along N = 512,
    row statistics exchanged through distributed shared memory, run in place on the residual stream) against the fp32
    CUDA-core GEMM followed by the stand-alone LayerNorm kernel: the residual stream and the operand planes, the chained
    block-end pair, the last block, the residual-free proj_ case, a ragged last row block; with the A tile fetched in quarters
    and TMA-multicast across the cluster (PK_LN_MCAST=1, default) and loaded whole by every CTA."""
    from parakeet_cpp_b200.engine import selftest_gemm_ln
    monkeypatch.setenv("PK_LN_MCAST", mcast)
    xe, xr, pe, pr = selftest_gemm_ln(M, K, mode, 0)
    assert xe / xr < 5e-5 and pe / pr < 5e-5, (xe, xr, pe, pr)
    xe1, _, pe1, _ = selftest_gemm_ln(M, K, mode, 1)
    assert xe1 / xr < 2e-2 and pe1 / pr < 5e-2          # plain bf16 operands, bf16 hi plane only


@pytest.mark.parametrize("lens,tmax,mode", [([126], 126, 0), ([126], 126, 1), ([126], 126, 2), ([128, 1, 77, 126, 33], 128, 0),
                                            ([50, 126, 126, 9], 501, 0), ([64] * 20, 100, 0)])
def test_tcgen05_attention_matches_fp32_attention(pkg, lens, tmax, mode):
    """csrc/attention_umma.cu (UMMA tiles in TMEM, K / position window / V by TMA, rel_shift by a register barrel shifter,
    V as an MN-major operand) against the fp32 CUDA-core attention kernel on random inputs: the content term alone (zero
    position table), the position term alone (zero keys), ragged batches, a position table longer / shorter than the tile."""
    from parakeet_cpp_b200.engine import selftest_attention
    err, ref = selftest_attention(lens, tmax, mode)
    assert err / ref < 2e-4, (err, ref)


# ------------------------------------------------------------------ mel front end (K1/K2)
@pytest.mark.parametrize("lengths", [[16000], [400], [401, 559, 560, 561], [32000, 20000, 64000, 12345, 8000, 16001]])
def test_mel_matches_oracle(eng_tiny, O, synth, lengths):
    pcms = [synth.make_audio(n, 100 + i) for i, n in enumerate(lengths)]
    got = eng_tiny.mel(pcms)
    for pcm, g in zip(pcms, got):
        want = O.preprocess_audio(pcm)
        assert g.shape == want.shape
        if want.shape[0] > 3:
            assert np.abs(g - want).max() < MEL_TOL
        else:   # 3 frames: sigma ~ 0 bins amplify fp32 noise by 1e5; compare what is stable
            assert np.isfinite(g).all()


def test_mel_matches_reference_golden(eng_tiny, synth, golden):
    for ci in (0, 1, 3):
        n, aseed = (int(v) for v in golden[f"tiny.c{ci}.n_samples"])
        got = eng_tiny.mel([synth.make_audio(n, aseed)])[0]
        assert np.abs(got - golden[f"tiny.c{ci}.mel"]).max() < MEL_TOL


def test_mel_edge_signals(eng_tiny, O):
    rng = np.random.default_rng(0)
    sil = (1e-4 * rng.standard_normal(16000)).astype(np.float32)          # near-silence
    loud = np.clip(rng.standard_normal(16000), -1, 1).astype(np.float32)  # full-scale noise
    imp = np.zeros(16000, np.float32); imp[8000] = 1.0; imp += (1e-3 * rng.standard_normal(16000)).astype(np.float32)
    for pcm in (sil, loud, imp):
        g = eng_tiny.mel([pcm])[0]
        assert np.abs(g - O.preprocess_audio(pcm)).max() < 5e-3


# ------------------------------------------------------------------ encoder
def test_encoder_tiny_layers_match_oracle_and_golden(eng_tiny, O, tiny, golden):
    for ci in (0, 1, 2, 3):
        k = f"tiny.c{ci}."
        feats = golden[k + "mel"].astype(np.float32)
        encs, subs, lays = eng_tiny.encode([feats], taps=True)
        enc_o, sub_o, lay_o = O.encoder_forward(tiny.W, feats, tiny.ocfg, return_layers=True)
        assert _rel(subs[0], sub_o) < 1e-4
        for i in range(tiny.ocfg.n_layers):
            assert _rel(lays[0][i], lay_o[i]) < ENC_TOL
        assert _rel(encs[0], golden[k + "enc"]) < ENC_TOL
        assert _rel(subs[0], golden[k + "sub"]) < 1e-4


def test_encoder_ragged_batch_equals_singles(eng_tiny, O, synth, tiny):
    """Packed batch == each utterance alone (the reference is batch-1): padding, conv edges
    and attention extents are per utterance."""
    pcms = [synth.make_audio(n, 200 + i) for i, n in enumerate([64000, 400, 20000, 33333, 8000])]
    feats = [O.preprocess_audio(p) for p in pcms]
    batch = eng_tiny.encode(feats)
    for f, b in zip(feats, batch):
        single = eng_tiny.encode([f])[0]
        assert np.array_equal(single, b)
        assert _rel(b, O.encoder_forward(tiny.W, f, tiny.ocfg)) < ENC_TOL


def test_encoder_long_utterance(pkg, O, synth, tiny, math_mode):
    """An 11 s utterance (T' = 138: three 64-key tiles, three 64-query tiles in the attention kernel)
    next to a short one."""
    import dataclasses
    cfg = dataclasses.replace(tiny.cfg, math=MATH[math_mode], max_samples=200000, max_batch=4)
    e = pkg.Engine(cfg, tiny.weights_path, 0)
    try:
        pcms = [synth.make_audio(n, 300 + i) for i, n in enumerate([176000, 30000])]
        feats = [O.preprocess_audio(p) for p in pcms]
        got = e.encode(feats)
        assert got[0].shape[0] == 138
        for f, b in zip(feats, got):
            assert _rel(b, O.encoder_forward(tiny.W, f, tiny.ocfg)) < ENC_TOL
    finally:
        e.close()


def test_bf16x1_mode_runs_within_its_looser_bound(pkg, O, synth, tiny):
    """PK_MATH_BF16X1 (plain bf16 operands, one MMA per product; opt-in, NOT the parity mode): the whole path
    runs and the encoder stays within 2e-2 of the oracle (tokens are not required to match)."""
    import dataclasses
    e = pkg.Engine(dataclasses.replace(tiny.cfg, math=1), tiny.weights_path, 0)
    try:
        pcms = [synth.make_audio(n, 700 + i) for i, n in enumerate([32000, 9000])]
        feats = [O.preprocess_audio(p) for p in pcms]
        for f, b in zip(feats, e.encode(feats)):
            assert _rel(b, O.encoder_forward(tiny.W, f, tiny.ocfg)) < 2e-2
        for dec in (0, 1):
            toks = e.transcribe_batch(pcms, dec)
            assert len(toks) == 2
    finally:
        e.close()


def test_encoder_110m_matches_reference_golden(eng110, O, m110, synth, golden):
    k = "m110.c0."
    n, aseed = (int(v) for v in golden[k + "n_samples"])
    feats = O.preprocess_audio(synth.make_audio(n, aseed))
    encs, subs, lays = eng110.encode([feats], taps=True)
    assert encs[0].shape == (126, 512)
    assert _rel(subs[0], golden[k + "sub"]) < 1e-4
    assert _rel(lays[0][0], golden[k + "layer_first"]) < ENC_TOL
    assert _rel(lays[0][-1], golden[k + "enc"]) < ENC_TOL          # (the reference's last layer is its encoder output)
    assert np.array_equal(lays[0][-1], encs[0])
    assert _rel(encs[0], golden[k + "enc"]) < ENC_TOL


# ------------------------------------------------------------------ CTC head + greedy (K9)
def test_ctc_logprobs_and_tokens(eng_tiny, eng110, O, tiny, m110, golden):
    for eng, mdl, tag, cis in ((eng_tiny, tiny, "tiny", (0, 1, 2, 3)), (eng110, m110, "m110", (0,))):
        for ci in cis:
            k = f"{tag}.c{ci}."
            enc = golden[k + "enc"]
            lp = eng.ctc_logprobs(enc)
            want = O.ctc_log_probs(mdl.W, enc)
            assert np.abs(lp - want).max() < 1e-3
            assert np.array_equal(lp.argmax(1), golden[k + "ctc_argmax"])
            toks = eng.decode([enc], 0)[0]
            assert [list(t) for t in _tt(toks)] == golden[k + "ctc_tok"].tolist()
            assert np.allclose([t.confidence for t in toks], golden[k + "ctc_conf"], rtol=1e-3)


def test_ctc_known_answer_patterns(pkg, eng_tiny, O, tiny, golden):
    """The reference's CTCDecode.* vectors need log-probs as input; the C-ABI decodes from
    encoder output, so drive it with encoder rows that make the head emit the pattern:
    checked against the oracle's collapse of the engine's own per-frame argmax."""
    rng = np.random.default_rng(1)
    enc = rng.standard_normal((40, tiny.ocfg.d_model)).astype(np.float32)
    enc[10:14] = enc[10]       # repeated frames -> repeated argmax -> collapse
    enc[20:23] = enc[5]
    lp = O.ctc_log_probs(tiny.W, enc)
    want = O.ctc_greedy_decode_with_timestamps(lp, tiny.ocfg.vocab - 1)
    got = eng_tiny.decode([enc], 0)[0]
    assert _tt(got) == [w[:3] for w in want]


# ------------------------------------------------------------------ TDT greedy (K10)
def test_tdt_tokens_match_reference_golden(eng_tiny, eng110, golden):
    for eng, tag, cis in ((eng_tiny, "tiny", (0, 1, 2, 3)), (eng110, "m110", (0,))):
        for ci in cis:
            k = f"{tag}.c{ci}."
            toks = eng.decode([golden[k + "enc"]], 1)[0]
            assert [list(t) for t in _tt(toks)] == golden[k + "tdt_tok"].tolist()
            assert np.allclose([t.confidence for t in toks], golden[k + "tdt_conf"], rtol=1e-3)


def test_tdt_batch_lockstep_equals_singles(eng_tiny, O, tiny):
    rng = np.random.default_rng(2)
    encs = [rng.standard_normal((T, tiny.ocfg.d_model)).astype(np.float32) for T in (51, 1, 7, 33, 20, 2, 40, 13)]
    got = eng_tiny.decode(encs, 1)
    for e, g in zip(encs, got):
        try:
            want = O.tdt_greedy_decode(tiny.W, e, tiny.ocfg, with_timestamps=True, max_steps=4000)
        except RuntimeError:      # the reference algorithm livelocks on this input (tdt.cpp:66-104): no oracle
            assert len(g) == eng_tiny.cap
            continue
        assert _tt(g) == [w[:3] for w in want]
        assert np.allclose([t.confidence for t in g], [w[3] for w in want], rtol=1e-3)


def test_tdt_more_than_64_utterances(pkg, O, tiny, math_mode):
    """> 64 utterances: the decode kernel walks the batch in passes of 64 (cluster partial-sum buffers are
    reused between passes); every utterance must still equal its batch-of-1 decode and the oracle."""
    import dataclasses
    cfg = dataclasses.replace(tiny.cfg, math=MATH[math_mode], max_batch=96, max_samples=40000)
    e = pkg.Engine(cfg, tiny.weights_path, 0)
    try:
        rng = np.random.default_rng(5)
        encs = [rng.standard_normal((int(T), tiny.ocfg.d_model)).astype(np.float32) for T in rng.integers(1, 30, size=75)]
        got = e.decode(encs, 1)
        for i in (0, 31, 63, 64, 70, 74):
            assert _tt(got[i]) == _tt(e.decode([encs[i]], 1)[0])
            try:
                want = O.tdt_greedy_decode(tiny.W, encs[i], tiny.ocfg, with_timestamps=True, max_steps=4000)
            except RuntimeError:
                continue
            assert _tt(got[i]) == [w[:3] for w in want]
    finally:
        e.close()


def test_prefetch_pipeline_equals_blocking_call(pkg, tiny, synth, math_mode):
    """pk_prefetch_pcm double buffering: the H2D copy of the next batch is started while the current one runs;
    every batch must give exactly the tokens of the blocking pk_transcribe_batch, also when batches alternate."""
    import dataclasses
    import torch
    e = pkg.Engine(dataclasses.replace(tiny.cfg, math=MATH[math_mode]), tiny.weights_path, 0)
    try:
        batches = []
        for k, lens in enumerate(([32000, 20000, 8000], [16000, 400, 31000, 12345])):
            pcms = [synth.make_audio(n, 500 + 10 * k + i) for i, n in enumerate(lens)]
            buf = torch.from_numpy(np.concatenate(pcms)).pin_memory().numpy()
            off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
            arrs = e.transcribe_packed(buf, off, pkg.Decoder.TDT)
            want = [arrs["ids"][b, :arrs["len"][b]].tolist() for b in range(len(lens))]
            assert sum(len(w) for w in want) > 0
            batches.append((buf, off, want))
        e.prefetch(batches[0][0], batches[0][1])
        for it in range(5):
            buf, off, want = batches[it % 2]
            nbuf, noff, _ = batches[(it + 1) % 2]
            e.stage(buf, off)
            e.run_staged(pkg.Decoder.TDT)
            e.prefetch(nbuf, noff)
            arrs = e.fetch_into(e._tokens(len(off) - 1))
            assert [arrs["ids"][b, :arrs["len"][b]].tolist() for b in range(len(off) - 1)] == want
        # a stage() that does not match the outstanding prefetch falls back to a normal copy
        buf, off, want = batches[1]
        e.stage(buf, off)
        e.run_staged(pkg.Decoder.TDT)
        arrs = e.fetch_into(e._tokens(len(off) - 1))
        assert [arrs["ids"][b, :arrs["len"][b]].tolist() for b in range(len(off) - 1)] == want
    finally:
        e.close()


# ------------------------------------------------------------------ whole path through the public API
def test_transcriber_api_matches_reference_golden(pkg, tiny, synth, golden, math_mode):
    import dataclasses
    t = pkg.Transcriber(tiny.weights_path, tiny.vocab_path, dataclasses.replace(tiny.cfg, math=MATH[math_mode]))
    t.to_gpu()
    for ci in (0, 1, 3):
        k = f"tiny.c{ci}."
        n, aseed = (int(v) for v in golden[k + "n_samples"])
        pcm = synth.make_audio(n, aseed)
        r = t.transcribe(pcm, pkg.Decoder.TDT, True)
        assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == golden[k + "tdt_tok"].tolist()
        assert r.text == bytes(golden[k + "tdt_text"]).decode()
        assert "\n".join(w.word for w in r.word_timestamps) == bytes(golden[k + "tdt_words"]).decode()
        if r.word_timestamps:
            assert np.allclose([[w.start, w.end, w.confidence] for w in r.word_timestamps], golden[k + "tdt_word_times"], rtol=1e-3)
        r2 = t.transcribe(pcm, pkg.Decoder.CTC)
        assert r2.token_ids == golden[k + "ctc_tok"][:, 0].tolist()
        assert r2.text == bytes(golden[k + "ctc_text"]).decode()
        assert r2.timestamped_tokens == []           # timestamps=false leaves them empty (transcribe.hpp:152-176)
    t.engine.close()


def test_transcribe_110m_whole_path_tokens(pkg, m110, synth, golden, math_mode):
    import dataclasses
    t = pkg.Transcriber(m110.weights_path, m110.vocab_path, dataclasses.replace(m110.cfg, math=MATH[math_mode]))
    k = "m110.c0."
    n, aseed = (int(v) for v in golden[k + "n_samples"])
    pcm = synth.make_audio(n, aseed)
    r = t.transcribe(pcm, pkg.Decoder.CTC, True)
    assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == golden[k + "ctc_tok"].tolist()
    assert r.text == bytes(golden[k + "ctc_text"]).decode()
    r = t.transcribe(pcm, pkg.Decoder.TDT, True)
    assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == golden[k + "tdt_tok"].tolist()
    t.engine.close()


def test_transcribe_110m_more_clips_tokens_match_reference(pkg, m110, synth, math_mode):
    """Twenty more full-size clips decoded by the compiled reference (tests/golden/make_golden.py 110m_extra:
    four of 3 ... 10 s plus the first 16 clips of bench.py's batch): CTC and TDT tokens + frames bit-exact,
    confidences to 1e-3, as ONE ragged batch.  The closest CTC argmax decision in these clips has a top-2
    log-prob gap of 0.0006."""
    import dataclasses
    gx = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_110m_extra_v1.npz"))
    n_clips = int(gx["n_clips"][0])
    assert n_clips >= 4
    t = pkg.Transcriber(m110.weights_path, m110.vocab_path, dataclasses.replace(m110.cfg, math=MATH[math_mode]))
    pcms = []
    for ci in range(n_clips):
        n, aseed = (int(v) for v in gx[f"x110.c{ci}.n_samples"])
        pcms.append(synth.make_audio(n, aseed))
    for dec, tag in ((pkg.Decoder.CTC, "ctc"), (pkg.Decoder.TDT, "tdt")):
        rs = t.transcribe_batch(pcms, dec, True)
        for ci, r in enumerate(rs):
            k = f"x110.c{ci}."
            assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == gx[k + tag + "_tok"].tolist(), (tag, ci)
            assert np.allclose([x.confidence for x in r.timestamped_tokens], gx[k + tag + "_conf"], rtol=1e-3, atol=1e-6)
            assert r.text == bytes(gx[k + tag + "_text"]).decode()
    t.engine.close()


@pytest.mark.parametrize("switch", ["PK_FUSE_LN", "PK_ATTN_UMMA", "PK_GEMM_CLUSTER"])
def test_alternative_kernels_engine_equals_default_and_reference(pkg, O, m110, synth, monkeypatch, switch):
    """Kernel variants behind an engine switch, each against the same engine without it -- per-layer activations of a ragged
    batch -- and against the compiled reference's tokens on the twenty full-size clips (CTC and TDT, bit-exact):
    PK_FUSE_LN: every LayerNorm inside the epilogue of the GEMM that produces its input (gemm_tc_ln.cu);
    PK_ATTN_UMMA: the tcgen05 attention (attention_umma.cu: UMMA tiles in TMEM, rel_shift by a register barrel shifter,
    V as an MN-major operand) instead of the mma.sync kernel; PK_GEMM_CLUSTER: the wide GEMMs as 2-CTA clusters with the A tile
    multicast."""
    import dataclasses
    cfg = dataclasses.replace(m110.cfg, math=MATH["bf16x3"])
    feats = [O.preprocess_audio(synth.make_audio(n, 4200 + i)) for i, n in enumerate((160000, 112000, 48000, 81234))]
    outs = {}
    on = "2" if switch == "PK_GEMM_CLUSTER" else "1"
    for flag in ("0", on):
        monkeypatch.setenv(switch, flag)
        e = pkg.Engine(cfg, m110.weights_path, 0)
        outs["1" if flag == on else "0"] = e.encode(feats, taps=True)
        e.close()
    sub_tol, lay_tol = 1e-6, 2e-5
    for b in range(len(feats)):
        assert _rel(outs["1"][1][b], outs["0"][1][b]) < sub_tol                   # subsampling output (proj_ without / with the fused norm)
        for i in range(len(outs["0"][2][b])):
            assert _rel(outs["1"][2][b][i], outs["0"][2][b][i]) < lay_tol, (b, i)  # every block's output
        assert _rel(outs["1"][0][b], outs["0"][0][b]) < lay_tol
    monkeypatch.setenv(switch, on)
    gx = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_110m_extra_v1.npz"))
    n_clips = int(gx["n_clips"][0])
    t = pkg.Transcriber(m110.weights_path, m110.vocab_path, cfg)
    pcms = []
    for ci in range(n_clips):
        n, aseed = (int(v) for v in gx[f"x110.c{ci}.n_samples"])
        pcms.append(synth.make_audio(n, aseed))
    for dec, tag in ((pkg.Decoder.CTC, "ctc"), (pkg.Decoder.TDT, "tdt")):
        rs = t.transcribe_batch(pcms, dec, True)
        for ci, r in enumerate(rs):
            k = f"x110.c{ci}."
            assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == gx[k + tag + "_tok"].tolist(), (tag, ci)
            assert np.allclose([x.confidence for x in r.timestamped_tokens], gx[k + tag + "_conf"], rtol=1e-3, atol=1e-6)
    t.engine.close()


def test_full_batch_properties(pkg, m110, synth, math_mode):
    """BASELINE size (64 x 10 s): batch invariance and determinism, no oracle needed."""
    cfg = pkg.make_110m_config(max_batch=64, math=MATH[math_mode])
    e = pkg.Engine(cfg, m110.weights_path, 0)
    pcms = [synth.make_audio(160000, 1000 + i) for i in range(64)]
    for dec in (0, 1):
        a = e.transcribe_batch(pcms, dec)
        b = e.transcribe_batch(pcms, dec)
        assert [_tt(x) for x in a] == [_tt(x) for x in b]                 # deterministic
        sub = e.transcribe_batch([pcms[5], pcms[63], pcms[0]], dec)
        assert [_tt(x) for x in sub] == [_tt(a[5]), _tt(a[63]), _tt(a[0])]  # batch-invariant
        for x in a:
            assert all(0 <= t.token_id < 1024 for t in x)
            assert all(0 <= t.start_frame <= t.end_frame <= 125 for t in x)
            assert all(x[i].start_frame <= x[i + 1].start_frame for i in range(len(x) - 1))
    e.close()


# ------------------------------------------------------------------ error behaviour
def test_error_statuses(pkg, eng_tiny, tiny, synth, tmp_path):
    with pytest.raises(RuntimeError, match="max_samples|capacity|exceeds"):
        eng_tiny.transcribe_batch([synth.make_audio(tiny.cfg.max_samples + 160, 1)], 0)
    with pytest.raises(RuntimeError, match="window|shorter"):
        eng_tiny.transcribe_batch([np.zeros(100, np.float32)], 0)
    with pytest.raises(RuntimeError, match="max_batch|exceeds"):
        eng_tiny.transcribe_batch([synth.make_audio(800, i) for i in range(tiny.cfg.max_batch + 1)], 0)
    with pytest.raises(RuntimeError, match="cannot open"):
        pkg.Engine(tiny.cfg, str(tmp_path / "nope.safetensors"), 0)
    bad = dict(tiny.W)
    bad.pop("encoder_.layers_.1.attn_.pos_bias_u_")
    p = str(tmp_path / "missing.safetensors")
    synth.save_safetensors(p, bad)
    with pytest.raises(RuntimeError, match="missing tensor"):
        pkg.Engine(tiny.cfg, p, 0)


# ------------------------------------------------------------------ the C++ drop-in shim (include/parakeet/transcribe.hpp)
def test_cpp_shim(pkg, O, tiny, synth, golden, tmp_path):
    """Builds tests/cpp_shim_check.cpp (the reference-style usage: parakeet::Transcriber t(weights, vocab);
    t.to_gpu(); t.transcribe("audio.wav", Decoder, timestamps)) against the header-only shim + the C-ABI
    library and compares its tokens / text / words with the reference goldens."""
    import os
    import struct
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "cpp_shim_check")
    libdir = os.path.dirname(pkg.lib_path())
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp_shim_check.cpp"),
                    "-L" + libdir, "-lparakeet_b200", "-Wl,-rpath," + libdir, "-o", exe], check=True)
    k = "tiny.c0."
    n, aseed = (int(v) for v in golden[k + "n_samples"])
    pcm = synth.make_audio(n, aseed)
    i16 = np.round(pcm * 32768.0).astype(np.int16)
    wav = str(tmp_path / "a.wav")
    with open(wav, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 36 + 2 * len(i16)) + b"WAVEfmt " +
                struct.pack("<IHHIIHH", 16, 1, 1, 16000, 32000, 2, 16) + b"data" + struct.pack("<I", 2 * len(i16)))
        f.write(i16.tobytes())
    # a phrase for TranscribeOptions::boost_phrases: three vocabulary pieces as text
    phrase = "".join(tiny.pieces[i] for i in (7, 11, 5)).replace(O.SP_MARK, " ").strip()
    wav22 = str(tmp_path / "b.wav")                                      # the same samples declared as 22.05 kHz
    with open(wav22, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 36 + 2 * len(i16)) + b"WAVEfmt " +
                struct.pack("<IHHIIHH", 16, 1, 1, 22050, 44100, 2, 16) + b"data" + struct.pack("<I", 2 * len(i16)))
        f.write(i16.tobytes())
    out = subprocess.run([exe, tiny.weights_path, tiny.vocab_path, wav, "tiny", phrase, wav22], check=True, capture_output=True, text=True).stdout
    lines = out.strip().split("\n")
    tdt = [[int(x) for x in t.split(":")] for t in lines[0].split()[1:]]
    assert tdt == golden[k + "tdt_tok"].tolist()
    assert lines[1] == "TEXT " + bytes(golden[k + "tdt_text"]).decode()
    assert lines[2].split()[1:] == bytes(golden[k + "tdt_words"]).decode().split("\n")
    ctc = [[int(x) for x in t.split(":")] for t in lines[3].split()[1:]]
    assert ctc == golden[k + "ctc_tok"].tolist()
    assert lines[4] == "TEXT " + bytes(golden[k + "ctc_text"]).decode()
    # boosted decode through the shim == pk_set_boost on the same phrase through the ctypes binding; then plain again
    tk = pkg.engine.Tokenizer(tiny.vocab_path)
    e = pkg.Engine(tiny.cfg, tiny.weights_path, 0)
    wav_pcm = i16.astype(np.float32) / np.float32(32768.0)
    e.set_boost([tk.encode(phrase)], 6.0)
    for li, dec in ((6, pkg.Decoder.CTC), (7, pkg.Decoder.TDT)):
        want = e.transcribe_batch([wav_pcm], dec)[0]
        assert lines[li].split()[1:] == [f"{t.token_id}:{t.start_frame}:{t.end_frame}" for t in want], li
    e.set_boost([], 0.0)
    want22 = e.transcribe_batch_rate([wav_pcm], 22050, pkg.Decoder.TDT)[0]
    e.close()
    assert lines[8].split()[1:] == lines[3].split()[1:] and lines[8].startswith("PLAIN")
    assert lines[9].startswith("RATE") and lines[9].split()[1:] == [f"{t.token_id}:{t.start_frame}:{t.end_frame}" for t in want22]
    assert lines[10].startswith("ERR Cannot open audio file")


# ------------------------------------------------------------------ tdt-600m preset (SURVEY section 8f.1, BASELINE config 3)
@pytest.fixture(scope="module")
def m600(tmp_path_factory, pkg, O, synth):
    import os
    d = str(tmp_path_factory.mktemp("m600"))
    ocfg = O.make_tdt_600m_config()
    W = synth.make_weights(ocfg, seed=0)
    wp = os.path.join(d, "m600.safetensors")
    synth.save_safetensors(wp, W)
    pieces = synth.make_vocab(ocfg.vocab - 1, seed=0)
    vp = os.path.join(d, "m600.vocab.txt")
    synth.save_vocab(vp, pieces)
    return dict(ocfg=ocfg, W=W, weights_path=wp, vocab_path=vp, pieces=pieces)


def test_tdt_600m_preset_matches_reference_golden(pkg, O, synth, m600):
    """make_tdt_600m_config: 128 mels, d=1024, 24 layers, head_dim 128, 2-layer LSTM, 8193 labels,
    'joint_.' key prefix, no CTC head -- same kernels, checked against the compiled reference."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_600m_v1.npz"))
    k = "m600.c0."
    n, aseed = (int(v) for v in g[k + "n_samples"])
    pcm = synth.make_audio(n, aseed)
    cfg = pkg.make_tdt_600m_config(max_batch=4, max_samples=80000)
    e = pkg.Engine(cfg, m600["weights_path"], 0)
    feats = e.mel([pcm])[0]
    assert feats.shape == g[k + "mel"].shape
    assert np.abs(feats - g[k + "mel"].astype(np.float32)).max() < 5e-3          # golden stored as fp16
    encs, subs, lays = e.encode([O.preprocess_audio(pcm, 128)], taps=True)
    genc = g[k + "enc"]
    assert encs[0].shape == genc.shape
    assert _rel(encs[0], genc) < ENC_TOL
    toks = e.decode([genc], 1)[0]
    assert [list(t) for t in _tt(toks)] == g[k + "tdt_tok"].tolist()
    assert np.allclose([t.confidence for t in toks], g[k + "tdt_conf"], rtol=1e-3)
    # whole path + a ragged batch through the public API
    t = pkg.Transcriber(m600["weights_path"], m600["vocab_path"], cfg)
    r = t.transcribe(pcm, pkg.Decoder.TDT, True)
    assert [[x.token_id, x.start_frame, x.end_frame] for x in r.timestamped_tokens] == g[k + "tdt_tok"].tolist()
    assert r.text == bytes(g[k + "tdt_text"]).decode()
    rs = t.transcribe_batch([pcm[:40000], pcm, pcm[:16000]], pkg.Decoder.TDT)
    assert rs[1].token_ids == r.token_ids
    # three more clips decoded by the compiled reference (make_golden.py 600m_extra), as one ragged batch
    gx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_600m_extra_v1.npz"))
    pcms = []
    for ci in range(int(gx["n_clips"][0])):
        n2, seed2 = (int(v) for v in gx[f"x600.c{ci}.n_samples"])
        pcms.append(synth.make_audio(n2, seed2))
    for ci, r2 in enumerate(t.transcribe_batch(pcms, pkg.Decoder.TDT, True)):
        kx = f"x600.c{ci}."
        assert [[x.token_id, x.start_frame, x.end_frame] for x in r2.timestamped_tokens] == gx[kx + "tdt_tok"].tolist(), ci
        assert np.allclose([x.confidence for x in r2.timestamped_tokens], gx[kx + "tdt_conf"], rtol=1e-3, atol=1e-6)
        assert r2.text == bytes(gx[kx + "tdt_text"]).decode()
    e.close()
    t.engine.close()


def test_tdt_600m_config3_full_size_ragged_batch(pkg, O, synth, m600):
    """BASELINE configs[2] at its full size: tdt-600m, 30 s clips (T' = 376: 6 x 6 attention tiles of the head_dim-128
    tensor-core kernel, 3 GEMM row tiles per utterance), as a RAGGED 16-utterance batch.  Two clips were decoded by the
    compiled reference (make_golden.py 600m_long: a 30 s and a 21 s clip; ~25 CPU-minutes each); the other rows are
    shorter cuts whose results must equal single-utterance runs (batch invariance)."""
    import os
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_600m_long_v1.npz")
    g = np.load(p)
    nclips = int(g["n_clips"][0])
    pcms = []
    for ci in range(nclips):
        n, aseed = (int(v) for v in g[f"l600.c{ci}.n_samples"])
        pcms.append(synth.make_audio(n, aseed))
    cfg = pkg.make_tdt_600m_config(max_batch=16, max_samples=480000)
    e = pkg.Engine(cfg, m600["weights_path"], 0)
    # encoder activations of the 30 s clip (every 4th row is in the fixture)
    feats = e.mel([pcms[0]])[0]
    ms = g["l600.c0.mel_stats"]
    assert abs(float(feats.mean()) - ms[0]) < 1e-4 and abs(float(feats.std()) - ms[1]) < 1e-3
    enc = e.encode([feats])[0]
    assert enc.shape[0] == int(g["l600.c0.enc_T"][0]) == 376
    assert _rel(enc[::4], g["l600.c0.enc_rows4"]) < ENC_TOL
    # the ragged 16-utterance batch through the whole path
    batch = list(pcms) + [pcms[0][:n] for n in (400, 16000, 80000, 160000, 240000, 333333, 479999)] + \
        [pcms[-1][:n] for n in (48000, 123456, 300000)] + [synth.make_audio(480000, 1001 + i) for i in range(16 - nclips - 10)]
    assert len(batch) == 16
    got = e.transcribe_batch(batch, pkg.Decoder.TDT)
    assert e.truncated_count() in range(0, 15)      # (a cut may hit the reference's livelock; the golden rows may not)
    for ci in range(nclips):
        assert len(got[ci]) < e.cap
        k = f"l600.c{ci}."
        assert [list(t) for t in _tt(got[ci])] == g[k + "tdt_tok"].tolist(), ci
        assert np.allclose([t.confidence for t in got[ci]], g[k + "tdt_conf"], rtol=1e-3, atol=1e-6)
    for i in (nclips + 3, nclips + 5, nclips + 8):          # batch invariance on three of the cuts
        alone = e.transcribe_batch([batch[i]], pkg.Decoder.TDT)[0]
        assert _tt(alone) == _tt(got[i]), i
    e.close()


def test_attention_hd128_tensor_core_equals_fp32_kernel(pkg, O, synth, m600, monkeypatch):
    """head_dim 128: the mma.sync bf16x3 attention (Q tiles in shared memory) against the fp32 SIMT attention
    (PK_ATTN_TC=0) on the same engine configuration, 9 s clip (T' = 113, two key tiles)."""
    pcm = synth.make_audio(144000, 4242)
    cfg = pkg.make_tdt_600m_config(max_batch=2, max_samples=160000)
    feats = O.preprocess_audio(pcm, 128)
    e = pkg.Engine(cfg, m600["weights_path"], 0)
    enc_tc = e.encode([feats, feats[:500]])
    e.close()
    monkeypatch.setenv("PK_ATTN_TC", "0")
    e = pkg.Engine(cfg, m600["weights_path"], 0)
    enc_f32 = e.encode([feats, feats[:500]])
    e.close()
    for a, b in zip(enc_tc, enc_f32):
        assert _rel(a, b) < 2e-4


def test_job_api_appends_microbatches_and_allgathers(pkg, tiny, synth, math_mode):
    """SURVEY section 8e behind the C-ABI: micro-batches appended to the device job buffer, ONE ncclAllGather
    (world size 1 here: NCCL resolved with dlopen, communicator owned by the engine), rows read back; and the
    device-resident job input (pk_job_stage_pcm / pk_job_select) against the host-buffer path."""
    import dataclasses
    e = pkg.Engine(dataclasses.replace(tiny.cfg, math=MATH[math_mode]), tiny.weights_path, 0)
    lens = [32000, 20000, 64000, 12345, 8000, 16001, 40000, 2000, 400, 25000, 31000]
    pcms = [synth.make_audio(n, 700 + i) for i, n in enumerate(lens)]
    want = e.transcribe_batch(pcms[:8], pkg.Decoder.TDT) + e.transcribe_batch(pcms[8:], pkg.Decoder.TDT)
    from parakeet_cpp_b200.engine import _pack
    buf, off = _pack(pcms)
    e.job_stage(buf, off)
    e.comm_init_rank(e.nccl_unique_id(), 0, 1)
    for rnd in range(2):                                     # second round: buffers are reused, rows reset
        e.job_begin(12, 1)
        for first, n in ((0, 8), (8, 3)):
            e.job_select(first, n)
            e.run_staged(pkg.Decoder.TDT)
            e.job_append()
        e.allgather_tokens()
        rows = e.job_fetch(12, gathered=True)
        assert np.array_equal(rows, e.job_fetch(12, gathered=False))
        assert rows[11, 0] == 0                              # the row nobody filled
        for i, w in enumerate(want):
            assert rows[i, 1:1 + rows[i, 0]].tolist() == [t.token_id for t in w], (rnd, i)
    with pytest.raises(RuntimeError):                        # job buffer full
        e.job_append(); e.job_append()
    e.close()


# ------------------------------------------------------------------ streaming eou path (SURVEY section 8f.2, BASELINE config 4)
def _stream_engine(pkg, O, synth, tag, S, tmpdir, math):
    import dataclasses
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_stream_v1.npz"))
    ocfg = O.make_tiny_stream_config() if tag == "tstream" else O.make_eou_120m_config()
    cfg = pkg.make_tiny_stream_config(max_batch=max(S, 8)) if tag == "tstream" else pkg.make_eou_120m_config(max_batch=max(S, 8))
    wseed, aseed = (int(v) for v in g[tag + ".seeds"])
    sched = [int(v) for v in g[tag + ".schedule"]]
    wp = os.path.join(str(tmpdir), tag + ".safetensors")
    synth.save_safetensors(wp, synth.make_weights(ocfg, seed=wseed))
    e = pkg.Engine(dataclasses.replace(cfg, math=MATH[math]), wp, 0)
    e.stream_open(S, max(sched))
    return e, g, sched, synth.make_audio(sum(sched), aseed)


@pytest.mark.parametrize("tag", ["tstream", "eou120"])
def test_streaming_chunks_match_reference_golden(pkg, O, synth, tmp_path, math_mode, tag):
    """One stream, chunk by chunk, against the compiled reference (golden_stream_v1.npz): new log-mel frames (13/14 per
    2560 samples: the reference's STFT quirk), encoder rows of the chunk (leftover-frame cache, K/V ring, conv cache,
    un-shifted position scores), tokens with absolute frames and confidences (carried LSTM state)."""
    e, g, sched, pcm = _stream_engine(pkg, O, synth, tag, 1, tmp_path, math_mode)
    pos, n_tok = 0, 0
    for ci, n in enumerate(sched):
        toks, mel, enc = e.stream_step([pcm[pos:pos + n]], taps=True)
        pos += n
        k = f"{tag}.k{ci}."
        gf, ge_, gt, gc = g[k + "feats"], g[k + "enc"], g[k + "tok"], g[k + "conf"]
        assert mel[0].shape == gf.shape, ci
        if gf.shape[0]:
            assert np.abs(mel[0] - gf).max() < 2e-3 * max(1.0, float(np.abs(gf).max())), ci      # un-normalised log-mel (|x| up to ~17)
        assert enc[0].shape == ge_.shape, ci
        if ge_.shape[0]:
            assert _rel(enc[0], ge_) < ENC_TOL, ci
        assert [list(t) for t in _tt(toks[0])] == gt.tolist(), ci
        assert np.allclose([t.confidence for t in toks[0]], gc, rtol=1e-3, atol=1e-6), ci
        n_tok += len(toks[0])
    assert n_tok > 5
    # reset, then the same stream again: identical tokens (StreamingTranscriber::reset, eou.cpp:145-149)
    e.stream_reset(0)
    pos, again = 0, []
    for n in sched:
        again += [_tt(e.stream_step([pcm[pos:pos + n]])[0])]
        pos += n
    assert [[list(t) for t in a] for a in again] == [g[f"{tag}.k{ci}.tok"].tolist() for ci in range(len(sched))]
    e.close()


def test_streaming_many_streams_lockstep(pkg, O, synth, tmp_path, math_mode):
    """S streams in lock step: copies of the golden stream started at different steps (so cache fill levels, ring
    positions and leftover-frame counts differ between the rows of one step), an always-silent stream and a stream that
    is reset half way.  Every copy must reproduce the reference's tokens of its own timeline."""
    tag, S = "tstream", 6
    e, g, sched, pcm = _stream_engine(pkg, O, synth, tag, S, tmp_path, math_mode)
    want = [g[f"{tag}.k{ci}.tok"].tolist() for ci in range(len(sched))]
    starts = [0, 1, 3, 4, None, 0]                   # stream 4 never gets samples; stream 5 is reset at step 8 and restarts
    cuts = np.concatenate([[0], np.cumsum(sched)])
    empty = np.zeros(0, np.float32)
    got = [[] for _ in range(S)]
    local = [0] * S                                  # next chunk index of each stream's own timeline
    for step in range(len(sched) + 5):
        if step == 8:
            e.stream_reset(5)
            local[5], got[5] = 0, []
        chunks = []
        for s in range(S):
            active = starts[s] is not None and step >= starts[s] and local[s] < len(sched)
            chunks.append(pcm[cuts[local[s]]:cuts[local[s] + 1]] if active else empty)
        toks = e.stream_step(chunks)
        for s in range(S):
            if len(chunks[s]):
                got[s].append([list(t) for t in _tt(toks[s])])
                local[s] += 1
            else:
                assert toks[s] == []
    for s in (0, 1, 2, 3):
        assert got[s] == want, s
    assert got[5] == want[:len(got[5])] and len(got[5]) >= 10
    e.close()


# ------------------------------------------------------------------ front-of-path rate conversion (SURVEY section 8f.4)
def test_gpu_resampler_matches_oracle_and_feeds_the_path(pkg, O, synth, tiny, golden_refcalls):
    """The polyphase kernel (csrc/resample.cu) against the oracle's sinc_resample (= the compiled reference's
    parakeet::resample, pinned on the CPU in tests/test_abi.py and here by SHA-256 digests of the reference's output):
    identical floats except where the reference's per-output rounding of i / (dst/src) differs from the exact rational
    position (bound: 1 ulp, >= 99.9 % identical); and a 22.05 kHz batch converted on the device (pk_stage_pcm_rate)
    gives the tokens of the host-converted batch."""
    import hashlib
    e = pkg.Engine(tiny.cfg, tiny.weights_path, 0)
    rng = np.random.default_rng(9)
    for sr, dr, lens in [(44100, 16000, [9000, 3, 20000]), (48000, 16000, [5001]), (8000, 16000, [2500, 1]), (22050, 16000, [30000, 12345]),
                         (96000, 16000, [6000]), (16000, 8000, [1000]), (11025, 16000, [4097])]:
        xs = [(rng.standard_normal(n) * 0.3).astype(np.float32) for n in lens]
        got = e.resample_batch(xs, sr, dr)
        for x, g in zip(xs, got):
            want = O.sinc_resample(x, sr, dr)
            assert g.shape == want.shape
            same = float(np.mean(g == want)) if len(want) else 1.0
            assert same >= 0.999, (sr, dr, len(x), same)
            assert np.all(np.abs(g - want) <= np.spacing(np.abs(want).astype(np.float32)) + 1e-45), (sr, dr, len(x))
            if len(x) > 16:      # the oracle's output is the reference's, bit for bit: `same` above compares with the reference
                ref_digest = golden_refcalls[f"resample_device.{sr}.{dr}.{len(x)}.sha256"].tobytes()
                assert hashlib.sha256(np.ascontiguousarray(want, np.float32).tobytes()).digest() == ref_digest, (sr, dr, len(x))
    # whole path from 22.05 kHz input
    pcm22 = [synth.make_audio(44100, 31)[:n] for n in (44100, 30000)]      # (any signal; treated as 22.05 kHz samples)
    host16 = [O.sinc_resample(p, 22050, 16000) for p in pcm22]
    want = e.transcribe_batch(host16, pkg.Decoder.TDT)
    got = e.transcribe_batch_rate(pcm22, 22050, pkg.Decoder.TDT)
    assert [_tt(a) for a in got] == [_tt(b) for b in want]
    e.close()


# ------------------------------------------------------------------ phrase-boosted decode on the device (SURVEY section 8f.3)
def test_boosted_decode_on_device_matches_reference_golden(pkg, eng_tiny, O, tiny, golden):
    """pk_set_boost + pk_decode (CTC and TDT) against the compiled reference's ctc_/tdt_greedy_decode_with_timestamps_boosted
    (golden_boost_v1.npz): boosted first-max argmax, trie advance on every emission, confidence = exp(raw log-prob);
    a batch of all cases' utterances at once (per-utterance trie state), the livelocking TDT cases only through their
    token capacity; and the boost is really off again after clearing it."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_boost_v1.npz"))
    changed = 0
    for n in range(int(g["n_cases"][0])):
        k = f"boost.k{n}."
        ci = int(g[k + "clip"][0])
        boost = float(g[k + "boost"][0])
        ids, lens = g[k + "ph_ids"], g[k + "ph_len"]
        offs = np.concatenate([[0], np.cumsum(lens)])
        phrases = [ids[offs[i]:offs[i + 1]].tolist() for i in range(len(lens))]
        enc = golden[f"tiny.c{ci}.enc"]
        eng_tiny.set_boost(phrases, boost)
        # the same utterance three times in one batch: every row keeps its own trie state
        ctc = eng_tiny.decode([enc, enc[:max(4, len(enc) // 2)], enc], pkg.Decoder.CTC)
        assert [list(t) for t in _tt(ctc[0])] == g[k + "ctc_tok"].tolist(), n
        assert _tt(ctc[2]) == _tt(ctc[0])
        assert np.allclose([t.confidence for t in ctc[0]], g[k + "ctc_conf"], rtol=1e-3, atol=1e-6)
        if not int(g[k + "tdt_livelock"][0]):
            tdt = eng_tiny.decode([enc, enc], pkg.Decoder.TDT)
            assert [list(t) for t in _tt(tdt[0])] == g[k + "tdt_tok"].tolist(), n
            assert _tt(tdt[1]) == _tt(tdt[0])
            assert np.allclose([t.confidence for t in tdt[0]], g[k + "tdt_conf"], rtol=1e-3, atol=1e-6)
        eng_tiny.set_boost([], 0.0)
        plain = eng_tiny.decode([enc], pkg.Decoder.CTC)[0]
        assert [list(t) for t in _tt(plain)] == golden[f"tiny.c{ci}.ctc_tok"].tolist()
        changed += _tt(plain) != _tt(ctc[0])
    assert changed >= 6
    assert [list(t) for t in _tt(eng_tiny.decode([golden["tiny.c0.enc"]], pkg.Decoder.TDT)[0])] == golden["tiny.c0.tdt_tok"].tolist()


def test_f16_and_bf16_checkpoints_load_like_their_f32_roundings(pkg, tiny, synth, tmp_path):
    """Checkpoint dtypes other than F32 (safetensors::load, axiom io_safetensors.cpp:16-44): a half-precision file must give
    exactly the engine an F32 file holding the same (rounded) values gives -- the loader converts on the way in."""
    import struct as _s
    import json as _j
    import torch
    W = tiny.W
    pcms = [synth.make_audio(32000, 11), synth.make_audio(20000, 12)]

    def save(path, conv, dtype_name):
        header, off, blobs = {}, 0, []
        for name, a in W.items():
            a = np.ascontiguousarray(a)
            if a.dtype == np.float32:
                b, dt = conv(a), dtype_name
            else:
                b, dt = a.tobytes(), "I64"
            header[name] = {"dtype": dt, "shape": list(a.shape), "data_offsets": [off, off + len(b)]}
            off += len(b)
            blobs.append(b)
        hj = _j.dumps(header).encode()
        with open(path, "wb") as f:
            f.write(_s.pack("<Q", len(hj)) + hj + b"".join(blobs))

    for tag, to_half, back in (("f16", lambda a: a.astype(np.float16).tobytes(), lambda a: a.astype(np.float16).astype(np.float32)),
                               ("bf16", lambda a: torch.from_numpy(a).to(torch.bfloat16).view(torch.int16).numpy().tobytes(),
                                lambda a: torch.from_numpy(a).to(torch.bfloat16).float().numpy())):
        ph, pf = str(tmp_path / (tag + ".safetensors")), str(tmp_path / (tag + "_as_f32.safetensors"))
        save(ph, to_half, "F16" if tag == "f16" else "BF16")
        save(pf, lambda a: back(a).tobytes(), "F32")
        outs = []
        for p in (ph, pf):
            e = pkg.Engine(tiny.cfg, p, 0)
            feats = e.mel(pcms)
            outs.append((e.encode(feats), [_tt(t) for t in e.transcribe_batch(pcms, pkg.Decoder.TDT)]))
            e.close()
        for a, b in zip(outs[0][0], outs[1][0]):
            assert np.array_equal(a, b), tag
        assert outs[0][1] == outs[1][1] and sum(len(t) for t in outs[0][1]) > 0


def test_cpp_streaming_transcriber(pkg, O, synth, tmp_path):
    """parakeet::StreamingTranscriber of the C++ drop-in (reference eou.hpp:101-141): transcribe_chunk per chunk of the golden
    stream, tokens with absolute frames per chunk, get_text, the partial-result callback, reset."""
    import subprocess
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_stream_v1.npz"))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "cpp_stream_check")
    libdir = os.path.dirname(pkg.lib_path())
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp_stream_check.cpp"),
                    "-L" + libdir, "-lparakeet_b200", "-Wl,-rpath," + libdir, "-o", exe], check=True)
    ocfg = O.make_tiny_stream_config()
    wseed, aseed = (int(v) for v in g["tstream.seeds"])
    sched = [int(v) for v in g["tstream.schedule"]]
    wp, vp, pp = str(tmp_path / "ts.safetensors"), str(tmp_path / "ts.vocab.txt"), str(tmp_path / "pcm.f32")
    synth.save_safetensors(wp, synth.make_weights(ocfg, seed=wseed))
    pieces = synth.make_vocab(ocfg.vocab - 1, seed=wseed)
    synth.save_vocab(vp, pieces)
    synth.make_audio(sum(sched), aseed).astype(np.float32).tofile(pp)
    out = subprocess.run([exe, wp, vp, pp, ",".join(str(n) for n in sched)], check=True, capture_output=True, text=True).stdout.strip().split("\n")
    all_ids = []
    for ci in range(len(sched)):
        want = g[f"tstream.k{ci}.tok"].tolist()
        assert out[ci].split()[1:] == [f"{a}:{b}:{c}" for a, b, c in want], ci
        all_ids += [w[0] for w in want]
    assert out[len(sched)] == "TEXT " + O.detokenize(all_ids, pieces)
    assert int(out[len(sched) + 1].split()[1]) == sum(1 for ci in range(len(sched)) if len(g[f"tstream.k{ci}.tok"]))
    assert out[len(sched) + 2] == "AFTER_RESET 0"


def test_cpp_sharded_example_world1(pkg, O, tiny, tmp_path):
    """examples/sharded_transcribe.cpp (a C++ host: one thread per GPU, pk_comm_init_rank + pk_job_* + ONE
    pk_allgather_tokens, NCCL by dlopen) built and run with one rank; on 2 GPUs the same job gives the same checksum
    (profiles/r02_example_sharded_cpp_2gpu.txt)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "sharded_transcribe")
    libdir = os.path.dirname(pkg.lib_path())
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), os.path.join(root, "examples", "sharded_transcribe.cpp"),
                    "-L" + libdir, "-lparakeet_b200", "-Wl,-rpath," + libdir, "-lpthread", "-o", exe], check=True)
    out = subprocess.run([exe, tiny.weights_path, "1", "12", "tiny"], check=True, capture_output=True, text=True).stdout
    assert "gathered 12 rows" in out and "identical on every rank" in out
