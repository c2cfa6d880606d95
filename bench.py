#!/usr/bin/env python
"""bench.py -- the headline benchmark of the hot path (BASELINE.json):

    audio-seconds / second (RTFx), tdt-ctc-110m, 10 s clips, 1/2/4/8 x B200

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 110m-64x10s|600m-16x30s] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path (PCM -> log-mel -> FastConformer -> TDT greedy) over
one batch of 64 synthetic 10 s clips per GPU (BASELINE.json configs[1]; --config 600m-16x30s:
configs[2]).  The K timed steps form one JOB of K x 64 DISTINCT clips per GPU (weak scaling); the
only exchange is ONE all-gather of the job's token rows after the last step, issued behind the
C-ABI (pk_allgather_tokens) inside the timed region: K=16 on 8 GPUs is BASELINE configs[4].

  value  : whole-job audio-seconds per second with the PCM already resident in HBM
           (pk_stage_pcm once, then pk_run_staged per step on the engine stream).
  e2e    : same metric through the public C-ABI with HOST buffers: every step copies its 41 MB of PCM from
           page-locked memory and reads its tokens back inside the timed region, driven as a serving loop
           (pk_stage_pcm + pk_run_staged + pk_prefetch_pcm(next batch) + pk_fetch_tokens: the H2D copy of
           batch i+1 runs under the kernels of batch i); e2e.sync_call = the single blocking call
           pk_transcribe_batch per batch.
  roofline / cpu_baseline / clocks / gpu_launches: see DESIGN.md section "Measurement".

--impl reference times the reference's own CPU implementation (oracle/_ref/libpkref.so,
the unmodified reference compiled by oracle/Makefile) on this box's host cores, one 10 s
clip per step (a bounded sample of the same workload).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

METRIC = "audio-seconds/sec (RTFx) tdt-ctc-110m 10s clips"

# BASELINE.json configs[1] (the configuration the metric is quoted on) and configs[2]; SURVEY.md section 8d for the
# algorithmic encoder work per clip (excl. the input-independent pos_proj).
CONFIGS = {
    "110m-64x10s": dict(model="tdt-ctc-110m", preset=0, batch=64, clip_samples=160000, enc_gflop=28.23, metric=METRIC,
                        cpu_sample_samples=160000),
    "600m-16x30s": dict(model="tdt-600m", preset=1, batch=16, clip_samples=480000, enc_gflop=470.9,
                        metric="audio-seconds/sec (RTFx) tdt-600m 30s clips", cpu_sample_samples=16000),
    # BASELINE.json configs[3]: eou-120m streaming, 160 ms chunks over 60 s streams (SURVEY.md section 8f row 2)
    "eou-120m-stream": dict(model="eou-120m", stream=True, chunk_samples=2560, stream_seconds=60.0,
                            metric="audio-seconds/sec (RTFx) eou-120m streaming, 160 ms chunks"),
}


def valid_rows(rows):
    """(len, ids...) rows -> token lists (entries past len are not part of the row's value)."""
    return [r[1:1 + r[0]].tolist() for r in rows]


def dump_tokens(dirname, arrs, n):
    """Writes the token arrays of n utterances (what pk_fetch_tokens returns) as DIR/<name>.npy in float32, so that the
    outputs of two builds can be compared; entries past an utterance's token count are -1."""
    os.makedirs(dirname, exist_ok=True)
    lens = arrs["len"][:n]
    valid = np.arange(arrs["ids"].shape[1])[None, :] < lens[:, None]
    np.save(os.path.join(dirname, "token_count.npy"), lens.astype(np.float32))
    for name, key in (("token_ids", "ids"), ("token_start_frame", "start"), ("token_end_frame", "end"), ("token_confidence", "conf")):
        np.save(os.path.join(dirname, name + ".npy"), np.where(valid, arrs[key][:n], -1).astype(np.float32))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sus=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.rows, self.proc = dev, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.dev)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        busy = sorted(sm)[len(sm) // 2:] if sm else [0.0]     # upper half ~ samples under load
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_checkpoint(tmpdir, conf=None):
    conf = conf or CONFIGS["110m-64x10s"]
    pkg = ge.load_package()
    from parakeet_cpp_b200 import synth
    mk = pkg.make_110m_config if conf["preset"] == 0 else pkg.make_tdt_600m_config
    cfg = mk(max_batch=conf["batch"], max_samples=conf["clip_samples"])
    wp = os.path.join(tmpdir, "pk110m_seed0.safetensors" if conf["preset"] == 0 else "pk600m_seed0.safetensors")
    if not os.path.exists(wp):
        W = synth.make_weights(cfg, seed=0)
        synth.save_safetensors(wp + ".tmp", W)
        os.replace(wp + ".tmp", wp)
    return pkg, synth, cfg, wp


def omp_threads():
    """CPUs the reference's OpenMP team can really run on: the affinity mask capped by the cgroup CPU quota
    (the GPU boxes show 128 CPUs but grant 16 CPUs of time; 128 spinning threads made the reference 4.6x slower).
    The team size is applied with omp_set_num_threads on the OpenMP runtime libpkref.so uses."""
    import ctypes
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, -(-int(quota) // int(period))))
    except (OSError, ValueError):
        pass
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except OSError:
        pass
    return n


def run_reference(args, rank, world, conf):
    """The reference's own CPU path (Transcriber::transcribe, transcribe.hpp:99-179)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refbind as R
    if not R.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libpkref.so not built"}))
        return
    cores = omp_threads()
    if conf.get("stream"):
        import oracle as O
        pkg = ge.load_package()
        from parakeet_cpp_b200 import synth
        wp = os.path.join(args.tmp, "pkeou120m_seed0.safetensors")
        if not os.path.exists(wp):
            synth.save_safetensors(wp + ".tmp", synth.make_weights(pkg.make_eou_120m_config(), seed=0))
            os.replace(wp + ".tmp", wp)
        CH, nch = conf["chunk_samples"], 14      # the golden fixture's chunks of stream 0 (known not to livelock the reference)
        pcm = synth.make_audio(max(args.steps, nch) * CH, 1200)
        t0 = time.perf_counter()
        n_steps = 0
        for _ in range(max(1, min(args.steps, 3))):
            rs = R.RefStream(wp, O.make_eou_120m_config())
            for k in range(nch):
                rs.chunk(pcm[k * CH:(k + 1) * CH])
            rs.close()
            n_steps += nch
        dt = time.perf_counter() - t0
        val = n_steps * CH / 16000.0 / dt
        print(json.dumps({"impl": "reference", "metric": conf["metric"], "value": val, "unit": "x real-time", "n_gpus": args.gpus,
                          "steps": n_steps, "warmup": 0, "ms_per_step": 1e3 * dt / n_steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "eou-120m streaming, ONE stream, 2560-sample chunks (the reference is single-stream)", "streams": 1},
                          "cpu_baseline": {"value": val, "unit": "x real-time", "cores": cores, "kind": "reference",
                                           "sample": f"{n_steps} chunks of one stream, OpenMP team = {cores}"},
                          "e2e": {"value": val, "unit": "x real-time", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    pkg, synth, cfg, wp = make_checkpoint(args.tmp, conf)
    m = R.RefModel(wp, "", conf["preset"])
    n = conf["cpu_sample_samples"]
    secs = n / 16000.0
    clips = [synth.make_audio(n, 1000 + i) for i in range(2)]
    for i in range(args.warmup):
        m.transcribe(clips[i % 2], "tdt")
        if i == 0 and args.warmup > 1:
            break                                  # one warm-up pass is enough for a CPU step of seconds
    t0 = time.perf_counter()
    stage = np.zeros(3)
    for i in range(args.steps):
        _, ms = m.transcribe(clips[i % 2], "tdt")
        stage += ms
    dt = time.perf_counter() - t0
    val = args.steps * secs / dt
    line = {"impl": "reference", "metric": conf["metric"], "value": val, "unit": "x real-time", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{conf['model']} TDT decode, {secs:g} s 16 kHz synthetic clips", "clips_per_step": 1,
                       "note": f"bounded sample: 1 clip of {secs:g} s per step of the {conf['batch']}-clip batch"},
            "cpu_baseline": {"value": val, "unit": "x real-time", "cores": cores, "kind": "reference",
                             "sample": f"{args.steps} x one {secs:g} s clip, TDT, OpenMP team = {cores} threads (affinity mask capped by the cgroup CPU quota)",
                             "stage_ms_per_clip": {"mel": stage[0] / args.steps, "encoder": stage[1] / args.steps,
                                                   "decode": stage[2] / args.steps}},
            "e2e": {"value": val, "unit": "x real-time", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_stream_bench(args, conf):
    """BASELINE configs[3]: eou-120m streaming.  S streams advance in lock step; a "step" feeds one 160 ms chunk (2560 samples)
    to every stream through pk_stream_step (host PCM in, host token arrays out, every step) -- the chunks arrive from the host
    by construction, so `value` and `e2e` are the same measurement.  Also reported: the latency of one step (= per-chunk
    latency of every stream in it) and the single-stream latency (S = 1, the reference's operating point)."""
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return                                     # streams do not shard below one process: replicas only (DESIGN.md)
    pkg = ge.load_package()
    from parakeet_cpp_b200 import synth
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    S, CH = args.streams, conf["chunk_samples"]
    K = args.steps
    cfg = pkg.make_eou_120m_config(max_batch=max(S, 8))
    wp = os.path.join(args.tmp, "pkeou120m_seed0.safetensors")
    if not os.path.exists(wp):
        synth.save_safetensors(wp + ".tmp", synth.make_weights(cfg, seed=0))
        os.replace(wp + ".tmp", wp)
    eng = pkg.Engine(cfg, wp, 0)
    eng.stream_open(S, CH)
    n = K * CH
    base = [synth.make_audio(n, 1200 + i) for i in range(min(S, 8))]          # stream 0 = the golden fixture's stream
    streams = [base[i % len(base)] if i < len(base) else np.roll(base[i % len(base)], 4001 * (i // len(base))) for i in range(S)]
    out = eng._tokens(S)

    def run(steps, eng_=eng, streams_=streams, out_=out):
        ntok = 0
        for k in range(steps):
            arrs = eng_.stream_step([x[k * CH:(k + 1) * CH] for x in streams_], out=out_, raw=True)
            ntok += int(arrs["len"].sum())
        return ntok

    run(min(K, 24))                                # warm-up: both chunk patterns seen, graphs instantiated
    eng.stream_reset(-1)
    eng.sync()
    sampler = ClockSampler(0)
    sampler.start()
    time.sleep(0.2)
    l0 = eng.launch_count()
    t0 = time.perf_counter()
    ntok = run(K)
    eng.sync()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_tokens(args.dump_outputs, out[1], S)          # the tokens every stream emitted in the last timed step
    launches = eng.launch_count() - l0
    audio_s = S * K * CH / 16000.0
    value = audio_s / wall
    # single-stream latency (the reference's case)
    cfg1 = pkg.make_eou_120m_config(max_batch=8)
    e1 = pkg.Engine(cfg1, wp, 0)
    e1.stream_open(1, CH)
    o1 = e1._tokens(1)
    run(24, e1, streams[:1], o1)
    e1.stream_reset(-1)
    e1.sync()
    t0 = time.perf_counter()
    k1 = min(K, 125)
    run(k1, e1, streams[:1], o1)
    e1.sync()
    lat1 = (time.perf_counter() - t0) / k1
    e1.close()
    pk = peaks()
    weight_bytes = 4.0 * 108.8e6                   # bf16 hi + lo planes of the 108.8 M encoder parameters, read once per step
    line = {"metric": conf["metric"], "value": value, "unit": "x real-time", "n_gpus": 1, "steps": K, "warmup": min(K, 24),
            "ms_per_step": 1e3 * wall / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16x3",
            "data": "synthetic",
            "config": {"workload": f"eou-120m streaming TDT decode, {S} concurrent 16 kHz streams in lock step, {CH}-sample (160 ms) chunks, "
                                   f"{K} chunks per stream ({K * CH / 16000.0:g} s)", "streams": S, "chunk_samples": CH,
                       "tokens_emitted": ntok, "l2": "weights (435 MB of bf16 hi/lo planes) exceed the 126 MB L2: re-read from HBM every step"},
            "e2e": {"value": value, "unit": "x real-time", "h2d_bytes_per_step": S * CH * 4, "d2h_bytes_per_step": int(S * (1 + eng.cap) * 4 + 3 * S * eng.cap * 4),
                    "api": "pk_stream_step per chunk (pageable host PCM in, host token arrays out)"},
            "latency": {"ms_per_chunk_step_all_streams": 1e3 * wall / K, "ms_per_chunk_single_stream": 1e3 * lat1,
                        "real_time_budget_ms": 160.0},
            "gpu_launches": int(launches), "wall_s": wall, "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "the step's tcgen05 GEMMs stream every encoder weight once per step (M = sum of 1-2 frames per stream)",
                         "achieved": weight_bytes / (wall / K) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                         "frac": weight_bytes / (wall / K) / 1e9 / pk["hbm"], "traffic": None,
                         "note": "launch/latency-bound at this S: ~330 kernels per step replayed as one CUDA graph"}}
    if not args.no_cpu_baseline:
        import refbind as R
        import oracle as O
        if R.available():
            cores = omp_threads()
            rs = R.RefStream(wp, O.make_eou_120m_config())
            t0 = time.perf_counter()
            nch = 14                               # the golden fixture's chunks of stream 0 (known not to livelock the reference)
            for k in range(nch):
                rs.chunk(streams[0][k * CH:(k + 1) * CH])
            dt = time.perf_counter() - t0
            rs.close()
            line["cpu_baseline"] = {"value": nch * CH / 16000.0 / dt, "unit": "x real-time", "cores": cores, "kind": "reference",
                                    "sample": f"one stream, its first {nch} chunks (2.24 s) through StreamingTranscriber's pipeline, OpenMP team = {cores}",
                                    "ms_per_chunk": 1e3 * dt / nch}
    print(json.dumps(line))
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 20; eou-120m-stream: 375 = one 60 s stream)")
    ap.add_argument("--streams", type=int, default=64, help="eou-120m-stream: concurrent streams advanced in lock step")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="110m-64x10s", choices=sorted(CONFIGS))
    ap.add_argument("--decoder", default="tdt", choices=["tdt", "ctc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tmp", default=os.environ.get("PK_BENCH_TMP", os.path.join(tempfile.gettempdir(), f"pk_bench_{os.getuid()}")),
                    help="cache of the synthetic checkpoints (per user: the directory is shared by every run on the machine)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the token arrays of the last timed step as DIR/<name>.npy "
                    "(float32; with N GPUs, those of rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps what the CUDA path computed (--impl ours)")
    os.makedirs(args.tmp, exist_ok=True)
    conf = CONFIGS[args.config]
    if args.steps is None:
        args.steps = 375 if conf.get("stream") else 20
    if conf.get("stream"):
        if args.impl == "reference":
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            return run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), conf)
        return run_stream_bench(args, conf)
    BATCH, CLIP_SAMPLES = conf["batch"], conf["clip_samples"]
    CLIP_SECONDS = CLIP_SAMPLES / 16000.0
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        run_reference(args, rank, world, conf)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        pkg, synth, cfg, wp = make_checkpoint(args.tmp, conf)
    if world > 1:
        dist.barrier()
    pkg, synth, cfg, wp = make_checkpoint(args.tmp, conf)
    eng = pkg.Engine(cfg, wp, local)
    dec = pkg.Decoder.TDT if args.decoder == "tdt" else pkg.Decoder.CTC
    if dec == pkg.Decoder.CTC and not cfg.has_ctc:
        raise SystemExit("bench.py: this model has no CTC head")
    K = args.steps
    NJ = max(K, args.warmup)                       # micro-batches held by the job buffers

    # The multi-GPU exchange lives behind the C-ABI: the engine owns an NCCL communicator (rank 0 creates the
    # unique id, torch.distributed only carries its 128 bytes) and pk_allgather_tokens issues the one collective.
    if world > 1:
        uid = [eng.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init_rank(uid[0], rank, world)

    # This rank's job: K micro-batches of BATCH DISTINCT clips (weak scaling).  Micro-batch 0 holds the seeded clips
    # 1000 + rank * BATCH + i (the ones the golden fixtures pin); micro-batch k holds clip (i + k) % BATCH of that
    # set rotated by 997 k samples: different samples, mel frames and tokens in every step, at memcpy cost.
    base = [synth.make_audio(CLIP_SAMPLES, 1000 + rank * BATCH + i) for i in range(BATCH)]
    big = torch.empty(NJ * BATCH * CLIP_SAMPLES, dtype=torch.float32).pin_memory().numpy()   # PAGE-LOCKED host input
    for k in range(NJ):
        for i in range(BATCH):
            o = (k * BATCH + i) * CLIP_SAMPLES
            big[o:o + CLIP_SAMPLES] = np.roll(base[(i + k) % BATCH], 997 * k) if k else base[i]
    off = np.arange(BATCH + 1, dtype=np.int64) * CLIP_SAMPLES          # offsets of one micro-batch
    off_all = np.arange(NJ * BATCH + 1, dtype=np.int64) * CLIP_SAMPLES

    def mb(k):                                                         # host view of micro-batch k
        return big[k * BATCH * CLIP_SAMPLES:(k + 1) * BATCH * CLIP_SAMPLES]

    def barrier():
        eng.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    stream = torch.cuda.ExternalStream(eng.stream(), device=local)   # events must be recorded on the engine stream

    def timed(fn):
        """fn() runs the K steps; bracketed by barrier+sync; device time via events on the ENGINE stream."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record(stream)
        fn()
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - w0
        ms = e0.elapsed_time(e1)
        if world > 1:      # max over ranks, measured on the device
            t = torch.tensor([ms, wall * 1e3], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms, wall

    # ---- device-resident throughput ("value"): the whole job's PCM is staged in HBM once; a step selects its
    # micro-batch (no copy), runs the path and appends its token rows to the device job buffer; ONE all-gather
    # after the last step (inside the timed region).  No host synchronisation anywhere in the loop.
    eng.job_stage(big, off_all)
    eng.job_begin(NJ * BATCH, world)               # size the job buffers once, outside every timed region

    def job_resident(steps):
        eng.job_begin(steps * BATCH, world)
        for k in range(steps):
            eng.flush_l2()
            eng.job_select(k * BATCH, BATCH)
            eng.run_staged(dec)
            eng.job_append()
        if world > 1:
            eng.allgather_tokens()

    job_resident(args.warmup)
    job_resident(args.warmup)       # (second pass: CUDA graph replay of the batch shape)
    l0 = eng.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ms, wall = timed(lambda: job_resident(K))
    launches = eng.launch_count() - l0
    rows_all = eng.job_fetch(world * K * BATCH, gathered=True) if world > 1 else eng.job_fetch(K * BATCH)
    mine = rows_all[rank * K * BATCH:(rank + 1) * K * BATCH]
    assert int((rows_all[:, 0] > 0).sum()) == rows_all.shape[0], "bench: an utterance of the job decoded to nothing"
    if args.dump_outputs and rank == 0:
        last = eng.fetch_into(eng._tokens(BATCH))                  # micro-batch K - 1: the last timed step
        assert valid_rows(np.concatenate([last["len"][:, None], last["ids"]], axis=1)) == valid_rows(mine[(K - 1) * BATCH:])
        dump_tokens(args.dump_outputs, last, BATCH)
    eng.job_select(0, BATCH)
    eng.run_staged(dec)
    ref_tokens = eng.fetch(BATCH)                                  # micro-batch 0 again, through the plain token path
    assert [r[1:1 + r[0]].tolist() for r in mine[:BATCH]] == [[t.token_id for t in u] for u in ref_tokens]
    distinct = len({r[1:1 + r[0]].tobytes() for r in rows_all})
    audio_s = K * BATCH * CLIP_SECONDS * world
    value = audio_s / (max(ms, 1e-9) / 1e3)

    # ---- the former per-step variant, for the scaling curve's history: every step all-gathers its own 64 rows
    per_step = None
    if world > 1:
        def steps_with_gather():
            for k in range(K):
                eng.flush_l2()
                eng.job_begin(BATCH, world)
                eng.job_select(k * BATCH, BATCH)
                eng.run_staged(dec)
                eng.job_append()
                eng.allgather_tokens()
        steps_with_gather()
        ms_ps, _ = timed(steps_with_gather)
        per_step = {"value": audio_s / (ms_ps / 1e3), "ms_per_step": ms_ps / K,
                    "note": "one pk_allgather_tokens per step on the engine stream (no host sync)"}

    # ---- end-to-end through the public API with host buffers ("e2e"): every step copies its PCM from page-locked
    # host memory and reads its tokens back; the job's rows are all-gathered once and read back at the end.
    #   sync     : pk_transcribe_batch (one blocking call per micro-batch, like the reference's transcribe())
    #   pipelined: pk_stage_pcm + pk_run_staged + pk_prefetch_pcm(next micro-batch) + pk_fetch_tokens -- the H2D
    #              copy of micro-batch k+1 runs under the kernels of micro-batch k (double-buffered PCM on the device)
    tok_out = eng._tokens(BATCH)

    def job_sync(steps):
        eng.job_begin(steps * BATCH, world)
        for k in range(steps):
            eng.flush_l2()
            arrs = eng.transcribe_packed(mb(k), off, dec, tok_out)     # H2D of the PCM + D2H of the token arrays inside
            eng.job_append()
        if world > 1:
            eng.allgather_tokens()
        return eng.job_fetch(world * steps * BATCH if world > 1 else steps * BATCH, gathered=world > 1), arrs

    def job_pipelined(steps):
        eng.job_begin(steps * BATCH, world)
        eng.prefetch(mb(0), off)                                       # H2D of micro-batch 0: inside the timed region
        for k in range(steps):
            eng.flush_l2()
            eng.stage(mb(k), off)            # adopts the copy started by the previous step's prefetch
            eng.run_staged(dec)
            eng.job_append()
            if k + 1 < steps:
                eng.prefetch(mb(k + 1), off)
            arrs = eng.fetch_into(tok_out)   # D2H of this step's tokens
        if world > 1:
            eng.allgather_tokens()
        return eng.job_fetch(world * steps * BATCH if world > 1 else steps * BATCH, gathered=world > 1), arrs

    def time_e2e(job_fn):
        job_fn(2)
        barrier()
        w0 = time.perf_counter()
        rows, o = job_fn(K)
        barrier()
        wall_ = time.perf_counter() - w0
        assert valid_rows(rows) == valid_rows(rows_all), "bench: e2e job rows differ from the device-resident job"
        if world > 1:
            t = torch.tensor([wall_], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            wall_ = float(t[0])
        return wall_, o

    sync_wall, out = time_e2e(job_sync)
    e2e_wall, out = time_e2e(job_pipelined)
    clocks = sampler.stop()            # sampled every 20 ms across the three timed regions (value, e2e sync, e2e pipelined)
    e2e_value = audio_s / e2e_wall
    n_tok = int(mine[:, 0].sum())
    W = 1 + eng.cap
    # per step: token rows + start/end/conf (pk_fetch_tokens) + this step's share of the job rows read back at the end
    d2h = BATCH * W * 4 + 3 * BATCH * eng.cap * 4 + world * BATCH * W * 4

    # ---- per-kernel-class device time (separate profiled pass; not the timed value)
    eng.job_select(0, BATCH)
    eng.profile_begin()
    PSTEPS = 3
    for _ in range(PSTEPS):
        eng.flush_l2()
        eng.run_staged(dec)
    prof = eng.profile_end()
    pk = peaks()
    gemm_ms, gemm_n, gemm_fl = prof["gemm"]
    gemm_tflops = gemm_fl / max(gemm_ms, 1e-9) / 1e9
    enc_ms = sum(prof[k][0] for k in ("subsample", "gemm", "layernorm", "attention", "dwconv")) / PSTEPS
    math_name = {0: "bf16x3", 1: "bf16", 2: "f32"}[int(cfg.math)]
    # The timed region is seconds long at ~1 kW: the sustained bf16 peak is the denominator; the burst figure is
    # reported beside it (frac_of_burst) because short runs keep the boost clock.
    # DRAM bytes of one launch of the dominant GEMM come from the committed ncu --set full capture
    # (bench.py cannot run ncu on itself; profiles/*_traffic.json says which launch and how it was taken)
    traffic, traffic_note = None, None
    for tf in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", tf)) as f:
                tj = json.load(f)
            traffic, traffic_note = tj["dram_bytes_per_launch"], f'{tj["kernel"]}; {tj["source"]}'
            break
        except (OSError, KeyError, ValueError):
            continue
    enc_gflop = conf["enc_gflop"]
    roofline = {"bound": "tensor", "kernel": "gemm_tc kernels (tcgen05; all GEMM launches of one step)",
                "achieved": gemm_tflops, "peak": pk["bf16_sus"], "unit": "TFLOP/s",
                "frac": gemm_tflops / pk["bf16_sus"], "frac_of_burst": gemm_tflops / pk["bf16"],
                "traffic": traffic if args.config == "110m-64x10s" else None, "traffic_of": traffic_note,
                "mma_frac": (3.0 if int(cfg.math) == 0 else 1.0) * gemm_tflops / pk["bf16_sus"] if int(cfg.math) != 2 else None,
                "peak_source": pk["src"] + " bf16 sustained (kernel timed inside a long step)",
                "algorithmic_gflop_per_launch": gemm_fl / max(gemm_n, 1) / 1e9, "launches_per_step": gemm_n // PSTEPS,
                "avg_launch_ms": gemm_ms / max(gemm_n, 1),
                "encoder": {"ms_per_clip": enc_ms / BATCH, "ms_per_batch": enc_ms,
                            "algorithmic_tflops": enc_gflop * BATCH / max(enc_ms, 1e-9),
                            "frac_of_bf16_peak": enc_gflop * BATCH / max(enc_ms, 1e-9) / pk["bf16_sus"]},
                "per_class_ms_per_step": {k: v[0] / PSTEPS for k, v in prof.items()}}

    line = {"metric": conf["metric"], "value": value, "unit": "x real-time", "n_gpus": world, "steps": K,
            "warmup": args.warmup, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": math_name, "data": "synthetic",
            "config": {"workload": f"{conf['model']} {args.decoder.upper()} decode, batch={BATCH}x{CLIP_SECONDS:g}s synthetic clips per GPU per step; "
                                   f"a job = {K} steps of DISTINCT clips per GPU ({K * BATCH * world} clips in all), token rows appended on the device, "
                                   "ONE all-gather at the end (K=16, N=8 is BASELINE configs[4]: 8192 clips)",
                       "clips_per_gpu_per_step": BATCH, "global_clips_per_step": BATCH * world, "job_clips": K * BATCH * world,
                       "distinct_hypotheses_in_job": distinct,
                       "parallelism": f"utterance-sharded dp{world}; pk_allgather_tokens: one ncclAllGather of the job's token rows on the engine stream",
                       "l2": "256 MiB scratch written between steps (inside the timed region)",
                       "tokens_in_job_this_rank": n_tok},
            "e2e": {"value": e2e_value, "unit": "x real-time", "h2d_bytes_per_step": int(mb(0).nbytes),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_wall / K,
                    "api": "pk_stage_pcm + pk_run_staged + pk_job_append + pk_prefetch_pcm(next micro-batch) + pk_fetch_tokens per step, then "
                           "pk_allgather_tokens + pk_job_fetch once: pinned host PCM in, host token arrays out, H2D of micro-batch k+1 under the "
                           "kernels of micro-batch k",
                    "sync_call": {"value": audio_s / sync_wall, "ms_per_step": 1e3 * sync_wall / K,
                                  "api": "pk_transcribe_batch (one blocking call per micro-batch) + pk_job_append"}},
            "gpu_launches": int(launches), "wall_s": wall, "clocks": clocks, "roofline": roofline}
    if per_step:
        line["per_step_allgather"] = per_step

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import refbind as R
        if R.available():
            cores = omp_threads()
            m = R.RefModel(wp, "", conf["preset"])
            ns = conf["cpu_sample_samples"]
            m.transcribe(base[0][:min(ns, 32000)], args.decoder)                 # touch the weights
            t0 = time.perf_counter()
            ids, stage = m.transcribe(base[0][:ns], args.decoder)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": (ns / 16000.0) / dt, "unit": "x real-time", "cores": cores, "kind": "reference",
                                    "sample": f"the first {ns / 16000.0:g} s of clip 0 of the batch, OpenMP team = {cores} threads (cgroup CPU quota)",
                                    "stage_ms": {"mel": stage[0], "encoder": stage[1], "decode": stage[2]}}
            if ns == CLIP_SAMPLES:
                line["cpu_baseline"]["tokens_match_gpu"] = ids == [t.token_id for t in ref_tokens[0]]
            m.close()
        else:
            line["cpu_baseline"] = {"value": None, "unit": "x real-time", "cores": 0, "kind": "reference",
                                    "sample": "oracle/_ref/libpkref.so not present"}
    if rank == 0:
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
