"""rnnt-600m, 16 x 30 s clips on one GPU: one JSON line (DESIGN.md section 13).

    python scratch/bench_rnnt.py [--out profiles/r03_rnnt_600m_16x30s.json] [--steps 20] [--warmup 3]

Seeded synthetic checkpoint (the golden fixture's rnnt-600m weights: synth seed 0, blank bias 8) and 16 seeded 30 s
clips.  Records the device-resident step (audio staged in HBM, pk_run_staged + sync) and the end-to-end step
(pk_transcribe_batch from host memory), the per-class device time from pk_profile_*, the decode's lock-steps from
pk_debug_tdt_phases, the tokens of two clips against the numpy oracle run on the engine's own encoder output, the
algorithmic encoder work (SURVEY.md section 8d formula, F' = 10), and the GPU name, power limit and clocks read in the
same run.  Checkpoints go to a temporary directory."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import __graft_entry__ as ge  # noqa: E402

pkg = ge.load_package()
from parakeet_cpp_b200 import synth  # noqa: E402
import rnnt_oracle as RO  # noqa: E402

BATCH, CLIP = 16, 480000


def conv_len(n):
    return (n + 2 - 3) // 2 + 1


def f_enc(n_samples, mel, d, ff, L, C=256):
    """SURVEY.md section 8d: F_enc = F_sub + L * F_layer (pos_proj excluded), FLOP per clip."""
    t0 = 1 + n_samples // 160
    t1, f1 = conv_len(t0), conv_len(mel)
    t2, f2 = conv_len(t1), conv_len(f1)
    T, Fp = conv_len(t2), conv_len(f2)
    f_sub = 2 * C * 9 * (t1 * f1) + 2 * C * 9 * (t2 * f2) + 2 * C * C * (t2 * f2) + 2 * C * 9 * (T * Fp) + 2 * C * C * (T * Fp) + 2 * T * (C * Fp) * d
    f_layer = 8 * T * d * ff + 8 * T * d * d + 4 * T * T * d + 2 * T * (2 * T - 1) * d + (6 * T * d * d + 18 * T * d)
    return f_sub + L * f_layer, T, Fp


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"], capture_output=True, text=True)
    v = [x.strip() for x in r.stdout.strip().split(",")]
    return dict(zip(("name", "power_limit_w", "clock_sm_mhz", "clock_max_sm_mhz"), v)) if len(v) == 4 else {"error": r.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_rnnt_600m_16x30s.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    gflop_clip, T, Fp = f_enc(CLIP, 80, 1024, 4096, 24)
    gflop_clip /= 1e9
    gflop_tdt600, _, _ = f_enc(CLIP, 128, 1024, 4096, 24)      # check of the formula against SURVEY's 470.9
    ocfg = RO.make_rnnt_600m_config()
    cfg = pkg.make_rnnt_600m_config()
    with tempfile.TemporaryDirectory() as td:
        W = synth.make_weights(ocfg, seed=0, blank_bias=8.0)
        wp = os.path.join(td, "rnnt600m.safetensors")
        synth.save_safetensors(wp, W)
        e = pkg.Engine(cfg, wp, 0)
    pcms = [synth.make_audio(CLIP, 5000 + i) for i in range(BATCH)]
    buf = np.ascontiguousarray(np.concatenate(pcms))
    off = np.arange(BATCH + 1, dtype=np.int64) * CLIP
    out = e._tokens(BATCH)
    info0 = gpu_info()
    # end to end: host PCM -> tokens on the host, one blocking call per step
    for _ in range(args.warmup):
        e.transcribe_packed(buf, off, pkg.Decoder.RNNT, out)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arrs = e.transcribe_packed(buf, off, pkg.Decoder.RNNT, out)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    # device resident: audio staged once, the whole path per step, one sync at the end
    e.stage(buf, off)
    for _ in range(args.warmup):
        e.run_staged(pkg.Decoder.RNNT)
    e.sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e.run_staged(pkg.Decoder.RNNT)
    e.sync()
    dev_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    phases = e.tdt_phases()
    info1 = gpu_info()
    # per class (a separate profiled pass: events around each launch class)
    e.profile_begin()
    for _ in range(3):
        e.run_staged(pkg.Decoder.RNNT)
    e.sync()
    prof = e.profile_end()
    per_class = {k: v[0] / 3 for k, v in prof.items()}
    toks = e.fetch(BATCH)
    assert e.truncated_count() == 0
    # tokens against the numpy oracle on the engine's own encoder output (two clips; decisions >= 1e-3 from a tie)
    checked = []
    encs = e.encode(e.mel(pcms[:2]))
    for i in range(2):
        gaps = []
        want = RO.rnnt_greedy_decode(W, encs[i], ocfg, with_timestamps=True, gaps=gaps)
        got = [(t.token_id, t.start_frame, t.end_frame) for t in toks[i]]
        checked.append(dict(clip=i, tokens=len(got), identical=got == [w[:3] for w in want], min_gap=min(gaps)))
    e.close()
    audio_s = BATCH * CLIP / 16000
    dec_ms = per_class.get("tdt", 0.0)
    prof_total = sum(per_class.values())
    line = {
        "workload": f"rnnt-600m RNNT decode, batch={BATCH}x{CLIP / 16000:g}s synthetic clips, 1 GPU, bf16x3",
        "gpu": info0, "gpu_after": info1,
        "steps": args.steps, "warmup": args.warmup,
        "device_resident": {"ms_per_step": dev_ms, "rtfx": audio_s / (dev_ms / 1e3)},
        "end_to_end": {"ms_per_step": e2e_ms, "rtfx": audio_s / (e2e_ms / 1e3)},
        "per_class_ms_per_step": per_class,
        "decode_share_of_profiled_step": dec_ms / prof_total if prof_total else None,
        "decode_lock_steps_per_batch": int(phases[7]),
        "encoder_frames_per_clip": T, "f_prime": Fp,
        "tokens_per_clip_mean": float(np.mean(arrs["len"])),
        "algorithmic_encoder_gflop_per_clip": gflop_clip,
        "formula_check_tdt600m_gflop_per_clip": gflop_tdt600 / 1e9,
        "oracle_check": checked,
    }
    s = json.dumps(line)
    print(s)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
