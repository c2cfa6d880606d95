"""Generates tests/golden/golden_rnnt_v1.npz from the UNMODIFIED reference's RNNT model:

    make -C oracle ref                       # oracle/_ref/libpkref.so (REF=<path of the reference sources>)
    python tests/golden/make_golden_rnnt.py  # REF as above; compiles tests/golden/ref_rnnt_harness.cpp against it,
                                             # with the compiler, flags and include paths of oracle/Makefile

Contents (seeded synthetic checkpoints and audio, parakeet.cpp_b200/synth.py):
  tiny.*  tiny RNNT shape (2 LSTM layers), ragged clips incl. a 400-sample one (T' = 1): encoder output, tokens
  msym.*  the same shape with a smaller blank bias, so that frames reach max_symbols_per_step emissions
  r600.*  the rnnt-600m preset (config.hpp:119-135), one 4 s clip, stored like golden_600m_v1.npz
Each clip holds the reference's rnnt_greedy_decode_with_timestamps result (tok = [id, start, end], conf) and its
rnnt_greedy_decode ids (ids).  The script counts, from the reference's own output, the frames by how many symbols the
reference emitted on them: 0 (blank at once), 1-9 (symbols, then blank) and max_symbols (forced advance); it asserts
that every kind occurs, including several symbols on a T' = 1 clip, and that every arg-max decision of the numpy
oracle (tests/rnnt_oracle.py, which must agree with the reference) is at least MIN_GAP from a tie.

The synthetic joint rarely prefers blank, and once a frame emits a symbol it tends to keep emitting up to
max_symbols; the blank logit therefore gets a large POSITIVE bias, and a smaller one for the variant that is meant to
reach max_symbols (with the default bias every frame of every clip reaches it).
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile
from collections import Counter

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import __graft_entry__ as ge  # noqa: E402
import oracle as O  # noqa: E402
import refbind as R  # noqa: E402
import rnnt_oracle as RO  # noqa: E402

ge.load_package()
from parakeet_cpp_b200 import synth  # noqa: E402

MAX_SYMBOLS = 10
MIN_GAP = 1e-3          # top-2 log-prob gap of every decision: far above the bf16x3 / fp32 re-association noise
# (blank bias, clips)
TINY = (14.0, [(20000, 22), (400, 23), (64000, 24), (48000, 26), (40000, 27), (56000, 28), (24000, 29)])
MSYM = (11.0, [(32000, 21), (20000, 22), (64000, 24), (400, 23)])
R600 = (8.0, [(64000, 3000)])


def build_harness(td):
    # one recipe: the compiler, flags and include paths are read from oracle/Makefile (the ones its harness uses)
    odir = os.path.join(ROOT, "oracle")
    extra = [f"REF={os.environ['REF']}"] if "REF" in os.environ else []
    r = subprocess.run(["make", "-s", "-C", odir, *extra, "--eval", "pk-print-%: ; @echo $($*)", "pk-print-CXX",
                        "pk-print-PK_CXXFLAGS", "pk-print-INCS"], check=True, capture_output=True, text=True)
    cxx, flags, incs = r.stdout.strip().split("\n")
    libdir = os.path.join(odir, "_ref")
    so = os.path.join(td, "librefrnnt.so")
    subprocess.run([cxx, *flags.split(), *incs.split(), "-shared", os.path.join(ROOT, "tests", "golden", "ref_rnnt_harness.cpp"),
                    f"-L{libdir}", "-lpkref", f"-Wl,-rpath,{libdir}", "-o", so], check=True)
    L = C.CDLL(so)
    vp, f32p, i32p = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32)
    L.pkref_rnnt_load.restype = vp
    L.pkref_rnnt_load.argtypes = [C.c_char_p] + [C.c_int] * 11
    L.pkref_rnnt_free.argtypes = [vp]
    L.pkref_rnnt_encode.argtypes = [vp, f32p, C.c_int, C.c_int, f32p]
    L.pkref_rnnt_greedy.argtypes = [vp, f32p, C.c_int, C.c_int, C.c_int, i32p, i32p, i32p, f32p, i32p, i32p]
    L.pkref_rnnt_last_error.restype = C.c_char_p
    return L


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def frame_events(tok, T):
    """Frames of one decode by the symbols emitted on them: (0: blank at once, 1..max_symbols-1: symbols then blank,
    max_symbols: forced advance without a blank)."""
    per = Counter(int(f) for f in tok[:, 1])
    return T - len(per), sum(1 for v in per.values() if v < MAX_SYMBOLS), sum(1 for v in per.values() if v == MAX_SYMBOLS)


def run(L, out, tag, ocfg, blank_bias, clips, td, custom, store_mel=False):
    W = synth.make_weights(ocfg, seed=0 if not custom else 3, blank_bias=blank_bias)
    wp = os.path.join(td, tag + ".safetensors")
    synth.save_safetensors(wp, W)
    c = ocfg
    h = L.pkref_rnnt_load(wp.encode(), int(custom), c.mel_bins, c.sub_channels, c.d_model, c.n_layers, c.n_heads, c.ff,
                          c.vocab, c.pred_hidden, c.lstm_layers, c.joint_hidden)
    assert h, L.pkref_rnnt_last_error().decode()
    ev = np.zeros(3, np.int64)
    for ci, (n, aseed) in enumerate(clips):
        k = f"{tag}.c{ci}."
        pcm = synth.make_audio(n, aseed)
        feats = np.ascontiguousarray(R.mel(pcm, c.mel_bins))
        T = O.encoder_len(feats.shape[0])
        enc = np.zeros((T, c.d_model), np.float32)
        assert L.pkref_rnnt_encode(h, _p(feats, C.c_float), feats.shape[0], c.mel_bins, _p(enc, C.c_float)) == T
        cap = T * MAX_SYMBOLS
        ids, st, en, ids2 = (np.zeros(cap, np.int32) for _ in range(4))
        cf = np.zeros(cap, np.float32)
        n2 = C.c_int32(0)
        m = L.pkref_rnnt_greedy(h, _p(enc, C.c_float), T, c.d_model, cap, _p(ids, C.c_int32), _p(st, C.c_int32),
                                _p(en, C.c_int32), _p(cf, C.c_float), _p(ids2, C.c_int32), C.byref(n2))
        assert m >= 0, L.pkref_rnnt_last_error().decode()
        tok = np.stack([ids[:m], st[:m], en[:m]], axis=1).astype(np.int32).reshape(-1, 3)
        gaps = []
        want = RO.rnnt_greedy_decode(W, enc, ocfg, MAX_SYMBOLS, with_timestamps=True, gaps=gaps)
        assert [list(w[:3]) for w in want] == tok.tolist(), (tag, ci, "numpy oracle and reference disagree")
        assert min(gaps) >= MIN_GAP, (tag, ci, min(gaps))
        out[k + "n_samples"] = np.array([n, aseed], np.int64)
        if store_mel:
            out[k + "mel"] = feats.astype(np.float16)
        out[k + "enc"] = enc
        out[k + "tok"], out[k + "conf"] = tok, cf[:m].copy()
        out[k + "ids"] = ids2[:n2.value].copy()
        e = frame_events(tok, T)
        ev += e
        print(tag, ci, n, "T", T, "tokens", m, "frames (0, 1-9, 10 symbols) =", e, "min gap %.4f" % min(gaps))
        if T == 1 and m > 1:
            out[tag + ".t1_multi"] = np.array([ci], np.int64)
    L.pkref_rnnt_free(h)
    out[tag + ".blank_bias"] = np.array([blank_bias], np.float32)
    out[tag + ".n_clips"] = np.array([len(clips)], np.int64)
    return ev


def main():
    out = {}
    with tempfile.TemporaryDirectory() as td:
        L = build_harness(td)
        ev = run(L, out, "tiny", RO.make_tiny_rnnt_config(), *TINY, td, True)
        ev_m = run(L, out, "msym", RO.make_tiny_rnnt_config(), *MSYM, td, True)
        ev_6 = run(L, out, "r600", RO.make_rnnt_600m_config(), *R600, td, False, store_mel=True)
    # the fixture must exercise every branch of the decode rule, in the tiny shape and in the preset
    assert min(ev + ev_m) > 0 and ev[1] >= 8, (ev, ev_m)
    assert ev_6[0] > 0 and ev_6[1] > 0 and ev_6[2] > 0, ev_6
    assert "msym.t1_multi" in out                 # a T' = 1 clip with several symbols on its only frame
    path = os.path.join(ROOT, "tests", "golden", "golden_rnnt_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")
    assert os.path.getsize(path) < 1 << 20


if __name__ == "__main__":
    main()
