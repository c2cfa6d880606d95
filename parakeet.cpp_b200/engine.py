"""ctypes binding of libparakeet_b200.so and a Python mirror of the reference's
high-level API (include/parakeet/transcribe.hpp:23-190 in the reference):

    Transcriber(weights_path, vocab_path, config=make_110m_config())
    .to_gpu()
    .transcribe(samples | path, decoder=None (the model's default), timestamps=False) -> TranscribeResult
    .transcribe(samples | path, TranscribeOptions(...))

plus `transcribe_batch`, which the reference lacks (it is batch-1 only,
transcribe.hpp:170-171).  There is no CPU path: if the CUDA library or a device
is missing, construction raises.
"""
from __future__ import annotations

import ctypes as C
import enum
import os
import struct
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path() -> str:
    # PK_LIB: a developer knob to load a variant build of the same sources (scratch/build_variant.py)
    return os.environ.get("PK_LIB") or os.path.join(_HERE, "libparakeet_b200.so")


class _PkConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "mel_bins", "sub_channels", "d_model", "n_layers", "n_heads", "ff", "conv_kernel", "vocab",
        "pred_hidden", "lstm_layers", "joint_hidden", "n_durations")] + [("durations", C.c_int32 * 8)] + \
        [(n, C.c_int32) for n in ("has_ctc", "joint_prefix_tdt", "max_symbols", "max_batch", "max_samples", "math")]


class _PkTokens(C.Structure):
    _fields_ = [("cap", C.c_int32), ("ids", C.POINTER(C.c_int32)), ("start", C.POINTER(C.c_int32)),
                ("end", C.POINTER(C.c_int32)), ("conf", C.POINTER(C.c_float)), ("len", C.POINTER(C.c_int32))]


EXPORTS = ["pk_config_110m", "pk_config_tdt_600m", "pk_config_rnnt_600m", "pk_engine_create", "pk_engine_destroy", "pk_last_error",
           "pk_mel_frames", "pk_encoder_frames", "pk_mel", "pk_encode", "pk_decode", "pk_ctc_logprobs",
           "pk_transcribe_batch", "pk_stage_pcm", "pk_prefetch_pcm", "pk_run_staged", "pk_fetch_tokens", "pk_sync",
           "pk_token_buffer", "pk_stream", "pk_launch_count", "pk_profile_begin", "pk_profile_end",
           "pk_profile_names", "pk_flush_l2", "pk_selftest_gemm", "pk_selftest_gemm_ln", "pk_selftest_attention", "pk_debug_tdt_phases", "pk_vocab_load", "pk_vocab_free", "pk_vocab_size",
           "pk_detokenize", "pk_group_words", "pk_tokenize", "pk_ctc_decode_boosted",
           "pk_resample_len", "pk_resample",
           "pk_job_begin", "pk_job_append", "pk_nccl_unique_id", "pk_comm_init_rank", "pk_allgather_tokens",
           "pk_job_fetch", "pk_job_stage_pcm", "pk_job_select", "pk_truncated_count",
           "pk_stream_open", "pk_stream_reset", "pk_stream_step", "pk_stream_count", "pk_stage_pcm_rate", "pk_resample_batch",
           "pk_set_boost", "pk_vocab_max_piece_bytes", "pk_safetensors_probe", "pk_debug_tdt_passes"]

_lib = None


def load_library():
    """Load the CUDA extension; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise RuntimeError(f"{p} is missing: build it with `python parakeet.cpp_b200/build.py` "
                           "(there is no CPU fallback)")
    L = C.CDLL(p)
    vp, i32p, f32p, i64p = C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_int64)
    L.pk_config_110m.argtypes = [C.POINTER(_PkConfig)]
    L.pk_config_tdt_600m.argtypes = [C.POINTER(_PkConfig)]
    L.pk_config_rnnt_600m.argtypes = [C.POINTER(_PkConfig)]
    L.pk_engine_create.argtypes = [C.POINTER(_PkConfig), C.c_char_p, C.c_int, C.POINTER(vp)]
    L.pk_engine_destroy.argtypes = [vp]
    L.pk_last_error.argtypes = [vp]
    L.pk_last_error.restype = C.c_char_p
    L.pk_mel_frames.argtypes = [C.c_int64]
    L.pk_encoder_frames.argtypes = [C.c_int32]
    L.pk_mel.argtypes = [vp, f32p, i64p, C.c_int32, f32p, i32p]
    L.pk_encode.argtypes = [vp, f32p, i32p, C.c_int32, f32p, i32p, f32p, f32p]
    L.pk_decode.argtypes = [vp, f32p, i32p, C.c_int32, C.c_int, C.POINTER(_PkTokens)]
    L.pk_ctc_logprobs.argtypes = [vp, f32p, C.c_int32, f32p]
    L.pk_transcribe_batch.argtypes = [vp, f32p, i64p, C.c_int32, C.c_int, C.POINTER(_PkTokens)]
    L.pk_stage_pcm.argtypes = [vp, f32p, i64p, C.c_int32]
    L.pk_resample_len.argtypes = [C.c_int64, C.c_int32, C.c_int32]
    L.pk_resample_len.restype = C.c_int64
    L.pk_resample.argtypes = [f32p, C.c_int64, C.c_int32, C.c_int32, f32p, C.c_int64]
    L.pk_resample.restype = C.c_int64
    L.pk_tokenize.argtypes = [vp, C.c_char_p, i32p, C.c_int32]
    L.pk_tokenize.restype = C.c_int32
    L.pk_ctc_decode_boosted.argtypes = [f32p, C.c_int32, C.c_int32, C.c_int32, i32p, i32p, C.c_int32, C.c_float, i32p, i32p, i32p,
                                        f32p, C.c_int32]
    L.pk_ctc_decode_boosted.restype = C.c_int32
    L.pk_prefetch_pcm.argtypes = [vp, f32p, i64p, C.c_int32]
    L.pk_run_staged.argtypes = [vp, C.c_int]
    L.pk_fetch_tokens.argtypes = [vp, C.POINTER(_PkTokens)]
    L.pk_sync.argtypes = [vp]
    L.pk_token_buffer.argtypes = [vp, C.POINTER(vp), i32p, i32p]
    L.pk_stream.argtypes = [vp]
    L.pk_stream.restype = vp
    L.pk_launch_count.argtypes = [vp]
    L.pk_launch_count.restype = C.c_int64
    L.pk_profile_begin.argtypes = [vp]
    L.pk_profile_end.argtypes = [vp, C.POINTER(C.c_double), i64p, C.POINTER(C.c_double), C.c_int32]
    L.pk_profile_names.restype = C.c_char_p
    L.pk_flush_l2.argtypes = [vp]
    L.pk_debug_tdt_phases.argtypes = [vp, i64p]
    L.pk_debug_tdt_passes.argtypes = [vp, i64p]
    L.pk_selftest_gemm.argtypes = [C.c_int] * 6 + [C.c_uint32, f32p, f32p]
    L.pk_selftest_gemm_ln.argtypes = [C.c_int] * 5 + [C.c_uint32, f32p]
    L.pk_selftest_attention.argtypes = [C.c_int, i32p, C.c_int, C.c_int, C.c_int, C.c_uint32, f32p]
    L.pk_vocab_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.pk_vocab_free.argtypes = [vp]
    L.pk_vocab_size.argtypes = [vp]
    L.pk_vocab_max_piece_bytes.argtypes = [vp]
    L.pk_detokenize.argtypes = [vp, i32p, C.c_int32, C.c_char_p, C.c_int32]
    L.pk_group_words.argtypes = [vp, i32p, i32p, i32p, f32p, C.c_int32, C.c_char_p, C.c_int32, f32p, f32p, f32p]
    L.pk_job_begin.argtypes = [vp, C.c_int64, C.c_int32]
    L.pk_job_append.argtypes = [vp]
    L.pk_nccl_unique_id.argtypes = [C.c_char_p]
    L.pk_comm_init_rank.argtypes = [vp, C.c_char_p, C.c_int32, C.c_int32]
    L.pk_allgather_tokens.argtypes = [vp, vp]
    L.pk_job_fetch.argtypes = [vp, C.c_int32, i32p, C.c_int64, i32p]
    L.pk_job_stage_pcm.argtypes = [vp, f32p, i64p, C.c_int32]
    L.pk_job_select.argtypes = [vp, C.c_int32, C.c_int32]
    L.pk_truncated_count.argtypes = [vp]
    L.pk_stream_open.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    L.pk_stream_reset.argtypes = [vp, C.c_int32]
    L.pk_stream_step.argtypes = [vp, f32p, i64p, C.POINTER(_PkTokens), f32p, i32p, f32p, i32p]
    L.pk_stream_count.argtypes = [vp]
    L.pk_set_boost.argtypes = [vp, i32p, i32p, C.c_int32, C.c_float]
    L.pk_safetensors_probe.argtypes = [C.c_char_p, C.c_char_p, f32p, C.c_int64, i64p]
    L.pk_stage_pcm_rate.argtypes = [vp, f32p, i64p, C.c_int32, C.c_int32]
    L.pk_resample_batch.argtypes = [vp, f32p, i64p, C.c_int32, C.c_int32, C.c_int32, f32p, i64p]
    _lib = L
    return L


# ------------------------------------------------------------------ configs (config.hpp)
class Math(enum.IntEnum):
    BF16X3 = 0
    BF16X1 = 1
    FP32 = 2


@dataclass
class ModelConfig:
    """EncoderConfig + PredictionConfig + JointConfig (reference config.hpp:9-75)."""
    mel_bins: int = 80
    sub_channels: int = 256
    d_model: int = 512
    n_layers: int = 17
    n_heads: int = 8
    ff: int = 2048
    conv_k: int = 9
    vocab: int = 1025
    pred_hidden: int = 640
    lstm_layers: int = 1
    joint_hidden: int = 640
    durations: tuple = (0, 1, 2, 3, 4)    # () = RNNT joint (one "out_proj_" head, decoded with Decoder.RNNT)
    max_symbols: int = 10                 # max_symbols_per_step (tdt.hpp, rnnt.hpp); an RNNT engine holds this many tokens per frame
    has_ctc: bool = True
    joint_prefix: str = "tdt_joint_."
    name: str = "tdt-ctc-110m"
    # streaming encoder only (StreamingEncoderConfig, streaming_encoder.hpp:18-24)
    att_context_left: int = 70
    att_context_right: int = 0
    # engine capacity
    max_batch: int = 64
    max_samples: int = 160000
    math: int = int(Math.BF16X3)

    def to_c(self) -> _PkConfig:
        c = _PkConfig()
        c.mel_bins, c.sub_channels, c.d_model, c.n_layers = self.mel_bins, self.sub_channels, self.d_model, self.n_layers
        c.n_heads, c.ff, c.conv_kernel, c.vocab = self.n_heads, self.ff, self.conv_k, self.vocab
        c.pred_hidden, c.lstm_layers, c.joint_hidden = self.pred_hidden, self.lstm_layers, self.joint_hidden
        c.n_durations = len(self.durations)
        for i, d in enumerate(self.durations):
            c.durations[i] = d
        c.has_ctc = int(self.has_ctc)
        c.joint_prefix_tdt = int(self.joint_prefix == "tdt_joint_.")
        c.max_symbols = self.max_symbols
        c.max_batch, c.max_samples, c.math = self.max_batch, self.max_samples, int(self.math)
        return c

    @property
    def is_rnnt(self) -> bool:
        return len(self.durations) == 0


def make_110m_config(**kw) -> ModelConfig:           # config.hpp:77-95
    return ModelConfig(**kw)


def make_tdt_600m_config(**kw) -> ModelConfig:       # config.hpp:98-116
    base = dict(mel_bins=128, d_model=1024, n_layers=24, ff=4096, vocab=8193, lstm_layers=2, has_ctc=False,
                joint_prefix="joint_.", name="tdt-600m", max_batch=16, max_samples=480000)
    base.update(kw)
    return ModelConfig(**base)


def make_rnnt_600m_config(**kw) -> ModelConfig:      # config.hpp:119-135 (80 mels into d 1024: proj_ is 2560 -> 1024)
    base = dict(d_model=1024, n_layers=24, ff=4096, vocab=1025, lstm_layers=2, durations=(), has_ctc=False,
                joint_prefix="joint_.", name="rnnt-600m", max_batch=16, max_samples=480000)
    base.update(kw)
    return ModelConfig(**base)


def make_tiny_rnnt_config(**kw) -> ModelConfig:
    """Small test-only RNNT shape (tiny encoder, 2 LSTM layers; not a reference preset)."""
    base = dict(sub_channels=64, d_model=128, n_layers=2, n_heads=2, ff=256, vocab=33, pred_hidden=64, lstm_layers=2,
                joint_hidden=64, durations=(), has_ctc=False, joint_prefix="joint_.", name="tiny-rnnt", max_batch=8,
                max_samples=64000)
    base.update(kw)
    return ModelConfig(**base)


def make_eou_120m_config(**kw) -> ModelConfig:       # eou.hpp:32-55 (streaming; ParakeetEOU registers "joint_", eou.cpp:9-13)
    base = dict(has_ctc=False, joint_prefix="joint_.", name="eou-120m", att_context_left=70, att_context_right=1,
                max_batch=64, max_samples=102400)
    base.update(kw)
    return ModelConfig(**base)


def make_tiny_stream_config(**kw) -> ModelConfig:
    """Small test-only streaming shape (mirrors oracle.make_tiny_stream_config; not a reference preset)."""
    base = dict(sub_channels=64, d_model=128, n_layers=2, n_heads=2, ff=256, vocab=33, pred_hidden=64, joint_hidden=64,
                has_ctc=False, joint_prefix="joint_.", name="tiny-stream", att_context_left=12, att_context_right=1,
                max_batch=8, max_samples=102400)
    base.update(kw)
    return ModelConfig(**base)


def make_tiny_config(**kw) -> ModelConfig:
    """Small test-only shape (not a reference preset)."""
    base = dict(sub_channels=64, d_model=128, n_layers=2, n_heads=2, ff=256, vocab=33, pred_hidden=64,
                joint_hidden=64, name="tiny", max_batch=8, max_samples=64000)
    base.update(kw)
    return ModelConfig(**base)


# ------------------------------------------------------------------ result types (timestamp.hpp, transcribe.hpp)
class Decoder(enum.IntEnum):          # transcribe.hpp:34
    CTC = 0
    TDT = 1
    RNNT = 2                          # rnnt_greedy_decode(_with_timestamps), rnnt.cpp:56-177: RNNT models only


@dataclass
class TimestampedToken:               # timestamp.hpp:11-18
    token_id: int
    start_frame: int
    end_frame: int
    confidence: float = 1.0


@dataclass
class WordTimestamp:                  # timestamp.hpp:20-27
    word: str
    start: float
    end: float
    confidence: float = 1.0


@dataclass
class TranscribeResult:               # transcribe.hpp:23-30
    text: str = ""
    token_ids: List[int] = field(default_factory=list)
    timestamped_tokens: List[TimestampedToken] = field(default_factory=list)
    word_timestamps: List[WordTimestamp] = field(default_factory=list)


@dataclass
class TranscribeOptions:              # transcribe.hpp:38-43
    decoder: Optional[Decoder] = None     # None: the model's default (TDT; RNNT for an RNNT model)
    timestamps: bool = False
    boost_phrases: List[str] = field(default_factory=list)
    boost_score: float = 5.0


def safetensors_probe(path: str, name: Optional[str] = None, cap: int = 0):
    """Host-only check of the checkpoint reader: -> (status, message, values | None)."""
    L = load_library()
    out = np.zeros(max(cap, 1), np.float32)
    n = C.c_int64(0)
    st = L.pk_safetensors_probe(path.encode(), name.encode() if name else None, _f32p(out), cap, C.byref(n))
    msg = L.pk_last_error(None).decode() if st != 0 else ""
    return st, msg, (out[:min(cap, n.value)].copy() if (st == 0 and name) else None)


def selftest_gemm(M, N, K, epi_kind, math=0, seed=1, device=0):
    """-> (max_abs_err, max_abs_ref) of the tcgen05 GEMM vs the fp32 CUDA-core GEMM."""
    L = load_library()
    e, r = C.c_float(), C.c_float()
    st = L.pk_selftest_gemm(device, M, N, K, epi_kind, math, seed, C.byref(e), C.byref(r))
    if st != 0:
        raise RuntimeError(f"pk_selftest_gemm failed ({st})")
    return e.value, r.value


def selftest_attention(lens, tmax=126, mode=0, seed=1, device=0):
    """-> (max_abs_err, max_abs_ref) of the tcgen05 attention kernel vs the fp32 attention kernel."""
    L = load_library()
    ln = np.ascontiguousarray(lens, np.int32)
    out = np.zeros(2, np.float32)
    st = L.pk_selftest_attention(device, _i32p(ln), len(ln), tmax, mode, seed, _f32p(out))
    if st != 0:
        raise RuntimeError(f"pk_selftest_attention failed ({st})")
    return float(out[0]), float(out[1])


def selftest_gemm_ln(M, K, mode, math=0, seed=1, device=0):
    """-> (x_err, x_ref, planes_err, planes_ref) of the fused residual-GEMM + LayerNorm kernel vs fp32 GEMM + LayerNorm kernel."""
    L = load_library()
    out = np.zeros(4, np.float32)
    st = L.pk_selftest_gemm_ln(device, M, K, mode, math, seed, _f32p(out))
    if st != 0:
        raise RuntimeError(f"pk_selftest_gemm_ln failed ({st})")
    return tuple(float(v) for v in out)


def _f32p(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _i32p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _i64p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


def _pack(arrs: Sequence[np.ndarray]):
    arrs = [np.ascontiguousarray(a, np.float32).reshape(-1) for a in arrs]
    off = np.zeros(len(arrs) + 1, np.int64)
    off[1:] = np.cumsum([len(a) for a in arrs])
    return (np.concatenate(arrs) if arrs else np.zeros(0, np.float32)), off


def read_wav(path: str) -> np.ndarray:
    """16 kHz mono PCM16 / float32 WAV -> fp32 in [-1, 1] (the subset of read_audio,
    src/audio_io.cpp:453-483, the configs need; int16 is divided by 32768 like dr_wav)."""
    with open(path, "rb") as f:
        data = f.read()
    if data[:4] != b"RIFF" or data[8:12] != b"WAVE":
        raise RuntimeError("Unsupported audio format (only RIFF/WAVE here): " + path)
    pos, fmt, pcm = 12, None, None
    while pos + 8 <= len(data):
        cid, size = data[pos:pos + 4], struct.unpack("<I", data[pos + 4:pos + 8])[0]
        body = data[pos + 8:pos + 8 + size]
        if cid == b"fmt ":
            fmt = struct.unpack("<HHIIHH", body[:16])
        elif cid == b"data":
            pcm = body
        pos += 8 + size + (size & 1)
    if fmt is None or pcm is None:
        raise RuntimeError("malformed WAV: " + path)
    tag, ch, sr, _, _, bits = fmt
    if sr != 16000:
        raise RuntimeError(f"Sample rate mismatch: audio={sr} expected=16000")
    if tag == 1 and bits == 16:
        x = np.frombuffer(pcm, "<i2").astype(np.float32) / np.float32(32768.0)
    elif tag == 3 and bits == 32:
        x = np.frombuffer(pcm, "<f4").astype(np.float32)
    else:
        raise RuntimeError("unsupported WAV encoding")
    if ch > 1:
        x = x.reshape(-1, ch).mean(axis=1).astype(np.float32)
    return x


class Engine:
    """Thin object wrapper over the C-ABI (one engine per device)."""

    def __init__(self, cfg: ModelConfig, weights_path: str, device: int = 0):
        self.L = load_library()
        self.cfg = cfg
        self.h = C.c_void_p()
        cc = cfg.to_c()
        st = self.L.pk_engine_create(C.byref(cc), weights_path.encode(), device, C.byref(self.h))
        if st != 0:
            raise RuntimeError(f"pk_engine_create failed ({st}): " + self.L.pk_last_error(None).decode())
        self.Tmax = self.L.pk_encoder_frames(self.L.pk_mel_frames(cfg.max_samples))
        self.cap = self.Tmax * cc.max_symbols if cfg.is_rnnt else 2 * self.Tmax + 8   # tokens per utterance, as pk_engine_create sizes them

    def close(self):
        if self.h:
            self.L.pk_engine_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, what):
        if st != 0:
            raise RuntimeError(f"{what} failed ({st}): " + self.L.pk_last_error(self.h).decode())

    # -- stage-level entry points (parity taps)
    def mel(self, pcms: Sequence[np.ndarray]) -> List[np.ndarray]:
        buf, off = _pack(pcms)
        nfr = np.zeros(len(pcms), np.int32)
        total = sum(1 + len(p) // 160 for p in pcms)
        out = np.zeros((total, self.cfg.mel_bins), np.float32)
        self._check(self.L.pk_mel(self.h, _f32p(buf), _i64p(off), len(pcms), _f32p(out), _i32p(nfr)), "pk_mel")
        res, o = [], 0
        for n in nfr:
            res.append(out[o:o + n].copy())
            o += n
        return res

    def encode(self, feats: Sequence[np.ndarray], taps: bool = False):
        nfr = np.array([f.shape[0] for f in feats], np.int32)
        buf = np.ascontiguousarray(np.concatenate([np.asarray(f, np.float32) for f in feats], axis=0))
        lens = [self.L.pk_encoder_frames(int(n)) for n in nfr]
        Mx, d = sum(lens), self.cfg.d_model
        out = np.zeros((Mx, d), np.float32)
        olen = np.zeros(len(feats), np.int32)
        sub = np.zeros((Mx, d), np.float32) if taps else None
        lay = np.zeros((self.cfg.n_layers, Mx, d), np.float32) if taps else None
        self._check(self.L.pk_encode(self.h, _f32p(buf), _i32p(nfr), len(feats), _f32p(out), _i32p(olen),
                                     _f32p(sub) if taps else None, _f32p(lay) if taps else None), "pk_encode")
        offs = np.concatenate([[0], np.cumsum(olen)])
        encs = [out[offs[i]:offs[i + 1]].copy() for i in range(len(feats))]
        if taps:
            return encs, [sub[offs[i]:offs[i + 1]].copy() for i in range(len(feats))], \
                [lay[:, offs[i]:offs[i + 1]].copy() for i in range(len(feats))]
        return encs

    def _tokens(self, n):
        cap = self.cap
        arrs = dict(ids=np.zeros((n, cap), np.int32), start=np.zeros((n, cap), np.int32),
                    end=np.zeros((n, cap), np.int32), conf=np.zeros((n, cap), np.float32), len=np.zeros(n, np.int32))
        t = _PkTokens(cap, _i32p(arrs["ids"]), _i32p(arrs["start"]), _i32p(arrs["end"]), _f32p(arrs["conf"]),
                      _i32p(arrs["len"]))
        return t, arrs

    @staticmethod
    def _unpack(arrs, n):
        out = []
        for b in range(n):
            k = int(arrs["len"][b])
            out.append([TimestampedToken(int(arrs["ids"][b, i]), int(arrs["start"][b, i]), int(arrs["end"][b, i]),
                                         float(arrs["conf"][b, i])) for i in range(k)])
        return out

    def decode(self, encs: Sequence[np.ndarray], decoder: Decoder) -> List[List[TimestampedToken]]:
        lens = np.array([e.shape[0] for e in encs], np.int32)
        buf = np.ascontiguousarray(np.concatenate([np.asarray(e, np.float32) for e in encs], axis=0))
        t, arrs = self._tokens(len(encs))
        self._check(self.L.pk_decode(self.h, _f32p(buf), _i32p(lens), len(encs), int(decoder), C.byref(t)), "pk_decode")
        return self._unpack(arrs, len(encs))

    def ctc_logprobs(self, enc: np.ndarray) -> np.ndarray:
        enc = np.ascontiguousarray(enc, np.float32)
        out = np.zeros((enc.shape[0], self.cfg.vocab), np.float32)
        self._check(self.L.pk_ctc_logprobs(self.h, _f32p(enc), enc.shape[0], _f32p(out)), "pk_ctc_logprobs")
        return out

    # -- the whole path
    def transcribe_batch(self, pcms: Sequence[np.ndarray], decoder: Decoder) -> List[List[TimestampedToken]]:
        buf, off = _pack(pcms)
        t, arrs = self._tokens(len(pcms))
        self._check(self.L.pk_transcribe_batch(self.h, _f32p(buf), _i64p(off), len(pcms), int(decoder), C.byref(t)),
                    "pk_transcribe_batch")
        return self._unpack(arrs, len(pcms))

    def transcribe_packed(self, buf: np.ndarray, off: np.ndarray, decoder: Decoder, out=None):
        """Same call on an already packed host buffer (fp32 samples back to back + int64 offsets;
        page-locked buffers are DMA'd directly).  Returns the raw token arrays
        (ids, start, end, conf, len) without building Python objects."""
        n = len(off) - 1
        if out is None:
            out = self._tokens(n)
        t, arrs = out
        self._check(self.L.pk_transcribe_batch(self.h, _f32p(buf), _i64p(off), n, int(decoder), C.byref(t)),
                    "pk_transcribe_batch")
        return arrs

    # -- device-resident variant (bench)
    def stage(self, buf: np.ndarray, off: np.ndarray):
        self._check(self.L.pk_stage_pcm(self.h, _f32p(buf), _i64p(off), len(off) - 1), "pk_stage_pcm")

    def prefetch(self, buf: np.ndarray, off: np.ndarray):
        """Start the H2D copy of the NEXT batch (page-locked packed buffer) under the current batch's kernels;
        the following stage() / transcribe_packed() with the same arguments adopts it."""
        self._check(self.L.pk_prefetch_pcm(self.h, _f32p(buf), _i64p(off), len(off) - 1), "pk_prefetch_pcm")

    def fetch_into(self, out):
        """pk_fetch_tokens into preallocated arrays (see _tokens)."""
        t, arrs = out
        self._check(self.L.pk_fetch_tokens(self.h, C.byref(t)), "pk_fetch_tokens")
        return arrs

    def run_staged(self, decoder: Decoder):
        self._check(self.L.pk_run_staged(self.h, int(decoder)), "pk_run_staged")

    def fetch(self, n) -> List[List[TimestampedToken]]:
        t, arrs = self._tokens(n)
        self._check(self.L.pk_fetch_tokens(self.h, C.byref(t)), "pk_fetch_tokens")
        return self._unpack(arrs, n)

    def sync(self):
        self._check(self.L.pk_sync(self.h), "pk_sync")

    def flush_l2(self):
        self._check(self.L.pk_flush_l2(self.h), "pk_flush_l2")

    def profile_begin(self):
        self._check(self.L.pk_profile_begin(self.h), "pk_profile_begin")

    def profile_end(self):
        """-> {class: (ms, launches, gemm_flops)} summed since profile_begin()."""
        names = self.L.pk_profile_names().decode().split(",")
        n = len(names)
        ms = (C.c_double * n)(); cnt = (C.c_int64 * n)(); fl = (C.c_double * n)()
        self._check(self.L.pk_profile_end(self.h, ms, cnt, fl, n), "pk_profile_end")
        return {names[i]: (ms[i], int(cnt[i]), fl[i]) for i in range(n)}

    def tdt_phases(self):
        a = np.zeros(8, np.int64)
        self._check(self.L.pk_debug_tdt_phases(self.h, _i64p(a)), "pk_debug_tdt_phases")
        return a

    def tdt_passes(self):
        a = np.zeros(8, np.int64)
        self._check(self.L.pk_debug_tdt_passes(self.h, _i64p(a)), "pk_debug_tdt_passes")
        return a

    def launch_count(self) -> int:
        return int(self.L.pk_launch_count(self.h))

    def stream(self) -> int:
        return int(self.L.pk_stream(self.h) or 0)

    # -- phrase boosting on the device (SURVEY.md section 8f row 3)
    def set_boost(self, phrases: Sequence[Sequence[int]], boost: float = 5.0):
        """phrases: token-id sequences; an empty list clears the boost."""
        ids = np.array([t for ph in phrases for t in ph], np.int32)
        off = np.zeros(len(phrases) + 1, np.int32)
        off[1:] = np.cumsum([len(ph) for ph in phrases])
        if len(ids) == 0:
            ids = np.zeros(1, np.int32)
        self._check(self.L.pk_set_boost(self.h, _i32p(ids), _i32p(off), len(phrases), float(boost)), "pk_set_boost")

    # -- non-16 kHz input: converted on the device (SURVEY.md section 8f row 4)
    def stage_rate(self, pcms: Sequence[np.ndarray], src_rate: int):
        buf, off = _pack(pcms)
        self._check(self.L.pk_stage_pcm_rate(self.h, _f32p(buf), _i64p(off), len(pcms), src_rate), "pk_stage_pcm_rate")

    def transcribe_batch_rate(self, pcms: Sequence[np.ndarray], src_rate: int, decoder: Decoder) -> List[List[TimestampedToken]]:
        self.stage_rate(pcms, src_rate)
        self.run_staged(decoder)
        return self.fetch(len(pcms))

    def resample_batch(self, pcms: Sequence[np.ndarray], src_rate: int, dst_rate: int) -> List[np.ndarray]:
        buf, off = _pack(pcms)
        lens = [int(self.L.pk_resample_len(len(p), src_rate, dst_rate)) for p in pcms]
        ooff = np.zeros(len(pcms) + 1, np.int64)
        ooff[1:] = np.cumsum(lens)
        out = np.zeros(int(ooff[-1]), np.float32)
        self._check(self.L.pk_resample_batch(self.h, _f32p(buf), _i64p(off), len(pcms), src_rate, dst_rate, _f32p(out), _i64p(ooff)),
                    "pk_resample_batch")
        return [out[ooff[i]:ooff[i + 1]].copy() for i in range(len(pcms))]

    # -- jobs: many micro-batches, one exchange (SURVEY.md section 8e)
    def job_begin(self, rows_local: int, world: int = 1):
        self._check(self.L.pk_job_begin(self.h, rows_local, world), "pk_job_begin")

    def job_append(self):
        self._check(self.L.pk_job_append(self.h), "pk_job_append")

    def job_stage(self, buf: np.ndarray, off: np.ndarray):
        self._check(self.L.pk_job_stage_pcm(self.h, _f32p(buf), _i64p(off), len(off) - 1), "pk_job_stage_pcm")

    def job_select(self, first: int, n: int):
        self._check(self.L.pk_job_select(self.h, first, n), "pk_job_select")

    def nccl_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        if self.L.pk_nccl_unique_id(buf) != 0:
            raise RuntimeError("pk_nccl_unique_id failed: " + self.L.pk_last_error(None).decode())
        return buf.raw

    def comm_init_rank(self, uid: bytes, rank: int, world: int):
        self._check(self.L.pk_comm_init_rank(self.h, uid, rank, world), "pk_comm_init_rank")

    def allgather_tokens(self, comm=None):
        self._check(self.L.pk_allgather_tokens(self.h, comm), "pk_allgather_tokens")

    def job_fetch(self, n_rows: int, gathered: bool = False) -> np.ndarray:
        """-> int32 [n_rows, 1 + cap] rows (len, ids...) of this rank's job (or of all ranks, rank-major)."""
        out = np.zeros((n_rows, 1 + self.cap), np.int32)
        w = C.c_int32()
        self._check(self.L.pk_job_fetch(self.h, int(gathered), _i32p(out), n_rows, C.byref(w)), "pk_job_fetch")
        assert w.value == 1 + self.cap
        return out

    # -- streaming (eou path): n_streams streams advanced in lock step, one chunk per stream and step
    def stream_open(self, n_streams: int, max_chunk_samples: int = 5120):
        self._check(self.L.pk_stream_open(self.h, n_streams, max_chunk_samples, self.cfg.att_context_left,
                                          self.cfg.att_context_right), "pk_stream_open")
        self.n_streams = n_streams

    def stream_reset(self, stream: int = -1):
        self._check(self.L.pk_stream_reset(self.h, stream), "pk_stream_reset")

    def stream_step(self, chunks: Sequence[np.ndarray], taps: bool = False, out=None, raw: bool = False):
        """chunks[s] = the samples stream s receives in this step (may be empty).  Returns the tokens each stream emitted
        in this step (absolute frames); with taps also the new log-mel frames and the encoder rows per stream."""
        S = self.n_streams
        assert len(chunks) == S
        buf, off = _pack(chunks)
        if out is None:
            out = self._tokens(S)
        t, arrs = out
        if not taps:
            self._check(self.L.pk_stream_step(self.h, _f32p(buf), _i64p(off), C.byref(t), None, None, None, None), "pk_stream_step")
            return arrs if raw else self._unpack(arrs, S)
        max_nf = 8 + max(len(c) for c in chunks) // 160 + 4
        mel = np.zeros((S * max_nf, self.cfg.mel_bins), np.float32)
        enc = np.zeros((S * (max_nf // 8 + 2), self.cfg.d_model), np.float32)
        n_mel, n_enc = np.zeros(S, np.int32), np.zeros(S, np.int32)
        self._check(self.L.pk_stream_step(self.h, _f32p(buf), _i64p(off), C.byref(t), _f32p(mel), _i32p(n_mel), _f32p(enc), _i32p(n_enc)),
                    "pk_stream_step")
        mo, eo = np.concatenate([[0], np.cumsum(n_mel)]), np.concatenate([[0], np.cumsum(n_enc)])
        return self._unpack(arrs, S), [mel[mo[i]:mo[i + 1]].copy() for i in range(S)], [enc[eo[i]:eo[i + 1]].copy() for i in range(S)]

    def truncated_count(self) -> int:
        return int(self.L.pk_truncated_count(self.h))

    def token_buffer(self):
        p, rows, ints = C.c_void_p(), C.c_int32(), C.c_int32()
        self._check(self.L.pk_token_buffer(self.h, C.byref(p), C.byref(rows), C.byref(ints)), "pk_token_buffer")
        return int(p.value), rows.value, ints.value


class Tokenizer:
    """Tokenizer::load / decode (src/vocab.cpp:10-64) via the C-ABI host helpers."""

    def __init__(self, vocab_path: Optional[str] = None):
        self.L = load_library()
        self.h = C.c_void_p()
        if vocab_path:
            self.load(vocab_path)

    def load(self, vocab_path: str):
        if self.L.pk_vocab_load(vocab_path.encode(), C.byref(self.h)) != 0:
            raise RuntimeError("Cannot open vocab file: " + vocab_path)      # vocab.cpp:13

    def loaded(self) -> bool:
        return bool(self.h) and self.L.pk_vocab_size(self.h) > 0

    def decode(self, ids: Sequence[int]) -> str:
        a = np.ascontiguousarray(ids, np.int32)
        buf = C.create_string_buffer(2 + (self.L.pk_vocab_max_piece_bytes(self.h) + 1) * max(len(a), 1))
        self.L.pk_detokenize(self.h, _i32p(a), len(a), buf, len(buf))
        return buf.value.decode("utf-8")

    def encode(self, text: str) -> List[int]:
        """Tokenizer::encode (src/vocab.cpp:76-117)."""
        raw = text.encode("utf-8")
        ids = np.zeros(2 * len(raw) + 8, np.int32)
        n = self.L.pk_tokenize(self.h, raw, _i32p(ids), len(ids))
        return ids[:n].tolist()

    def group_words(self, toks: Sequence[TimestampedToken]) -> List[WordTimestamp]:
        n = len(toks)
        ids = np.array([t.token_id for t in toks], np.int32)
        st = np.array([t.start_frame for t in toks], np.int32)
        en = np.array([t.end_frame for t in toks], np.int32)
        cf = np.array([t.confidence for t in toks], np.float32)
        buf = C.create_string_buffer(64 + 64 * max(n, 1))
        ws, we, wc = (np.zeros(max(n, 1), np.float32) for _ in range(3))
        k = self.L.pk_group_words(self.h, _i32p(ids), _i32p(st), _i32p(en), _f32p(cf), n, buf, len(buf), _f32p(ws),
                                  _f32p(we), _f32p(wc))
        words = buf.value.decode("utf-8").split("\n")[:k]
        return [WordTimestamp(words[i], float(ws[i]), float(we[i]), float(wc[i])) for i in range(k)]


def resample(samples: np.ndarray, src_rate: int, dst_rate: int = 16000) -> np.ndarray:
    """parakeet::resample (src/audio_io.cpp:238-251): Kaiser-windowed sinc, host code behind pk_resample."""
    L = load_library()
    x = np.ascontiguousarray(samples, np.float32)
    m = L.pk_resample_len(len(x), src_rate, dst_rate)
    if m < 0:
        raise ValueError("pk_resample: invalid arguments")
    out = np.zeros(max(m, 1), np.float32)
    L.pk_resample(_f32p(x if len(x) else np.zeros(1, np.float32)), len(x), src_rate, dst_rate, _f32p(out), m)
    return out[:m]


def ctc_greedy_decode_boosted(logprobs: np.ndarray, phrases: Sequence[Sequence[int]], boost_score: float = 5.0,
                              blank_id: Optional[int] = None) -> List[TimestampedToken]:
    """ctc_greedy_decode_with_timestamps_boosted (src/phrase_boost.cpp:122-176) on one utterance's log-probs
    (Engine.ctc_logprobs); phrases are token-id sequences (Tokenizer.encode).  Host code behind pk_ctc_decode_boosted."""
    L = load_library()
    lp = np.ascontiguousarray(logprobs, np.float32)
    T, V = lp.shape
    blank = V - 1 if blank_id is None else blank_id
    flat = np.array([t for ph in phrases for t in ph] or [0], np.int32)
    off = np.zeros(len(phrases) + 1, np.int32)
    off[1:] = np.cumsum([len(ph) for ph in phrases])
    ids, st, en = (np.zeros(max(T, 1), np.int32) for _ in range(3))
    cf = np.zeros(max(T, 1), np.float32)
    n = L.pk_ctc_decode_boosted(_f32p(lp), T, V, blank, _i32p(flat), _i32p(off), len(phrases), float(boost_score), _i32p(ids),
                                _i32p(st), _i32p(en), _f32p(cf), len(ids))
    if n < 0:
        raise ValueError("pk_ctc_decode_boosted: invalid arguments")
    return [TimestampedToken(int(ids[i]), int(st[i]), int(en[i]), float(cf[i])) for i in range(n)]


class Transcriber:
    """Python mirror of parakeet::Transcriber / TDTTranscriber (transcribe.hpp:55-299).  With an RNNT config
    (make_rnnt_600m_config) the default decoder is Decoder.RNNT, the model's only one; asking such a model for CTC or TDT
    raises ValueError, as the C-ABI rejects it."""

    def __init__(self, weights_path: str, vocab_path: str, config: Optional[ModelConfig] = None, device: int = 0):
        self.config = config or make_110m_config()
        self.engine = Engine(self.config, weights_path, device)
        self.tokenizer = Tokenizer(vocab_path) if vocab_path else Tokenizer()

    def to_gpu(self):
        """The reference moves the module tree to Metal here (transcribe.hpp:68-71); this
        engine only ever lives on the CUDA device, so this is a checked no-op."""
        return self

    def _result(self, toks, timestamps):
        r = TranscribeResult()
        r.token_ids = [t.token_id for t in toks]
        if timestamps:
            r.timestamped_tokens = list(toks)
        if self.tokenizer.loaded():
            r.text = self.tokenizer.decode(r.token_ids)
            if timestamps:
                r.word_timestamps = self.tokenizer.group_words(toks)
        return r

    def _decoder(self, decoder: Optional[Decoder]) -> Decoder:
        if self.config.is_rnnt:
            if decoder is not None and decoder != Decoder.RNNT:
                raise ValueError(f"{self.config.name} is an RNNT model: it decodes with Decoder.RNNT only")
            return Decoder.RNNT
        if decoder is None:
            return Decoder.TDT
        return decoder if self.config.has_ctc else Decoder.TDT

    def transcribe(self, audio, decoder: Optional[Decoder] = None, timestamps: bool = False) -> TranscribeResult:
        if isinstance(decoder, TranscribeOptions):
            opts = decoder
        else:
            opts = TranscribeOptions(decoder=decoder, timestamps=timestamps)
        if opts.boost_phrases:
            raise NotImplementedError("phrase boosting is outside the B200 hot path (SURVEY.md section 8f.3)")
        samples = read_wav(audio) if isinstance(audio, str) else np.asarray(audio, np.float32)
        dec = self._decoder(opts.decoder)
        toks = self.engine.transcribe_batch([samples], dec)[0]
        return self._result(toks, opts.timestamps)

    def transcribe_batch(self, audios, decoder: Optional[Decoder] = None, timestamps: bool = False) -> List[TranscribeResult]:
        pcms = [read_wav(a) if isinstance(a, str) else np.asarray(a, np.float32) for a in audios]
        out = []
        decoder = self._decoder(decoder) if (self.config.is_rnnt or decoder is None) else decoder
        B = self.config.max_batch
        for i in range(0, len(pcms), B):
            for toks in self.engine.transcribe_batch(pcms[i:i + B], decoder):
                out.append(self._result(toks, timestamps))
        return out


TDTTranscriber = Transcriber   # transcribe.hpp:200-299 (same surface, TDT only)
