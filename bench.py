#!/usr/bin/env python
"""bench.py — RTFx (audio-seconds transcribed per second) of the Qwen3-ASR-0.6B batch transcription path.

Workload (BASELINE.json `metric` / configs[2], extended by the decode the metric's "transcribed" implies):
64 x 30 s synthetic 16 kHz clips PER GPU (utterance-sharded, no collective on the data path, weak scaling),
random-init bf16 weights, full pipeline per step: log-mel -> audio encoder -> prompt splice + prefill -> 128 greedy
tokens over the paged KV cache.  One "step" = one pass over one such batch.

  value     whole-job RTFx with the batch already resident in HBM when the timed region starts (device time, CUDA
            events on the library's stream, max over ranks)
  e2e       the same metric through q3asr_transcribe_ids with HOST buffers: pinned staging + H2D of the samples and
            D2H of the ids inside the timed region (wall clock around the blocking call, max over ranks)
  roofline  the dominant kernel family (by device time) of the step, timed live with CUDA events around its launches
            in extra profiled steps of the same workload, against MEASURED_PEAKS.json; roofline_mel is the log-mel
            kernel against the HBM peak (the north star's "mel GB/s")
  cpu_baseline  the CPU oracle (a restatement of the reference's algorithm; the Swift/MLX reference cannot build on
            Linux) timed on this box's host cores on a bounded sample

`--impl reference` times only that CPU restatement (rank 0), for the driver's reference arm.
`--dump-outputs DIR` writes the token ids of the last device-timed step to DIR/ids.npy (float32 [clips, max_tokens]; one
DIR/ids_rank<r>.npy per rank on several GPUs).  The inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the benchmark may run from a read-only tree and writes nothing into it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "qwen3-asr-swift_b200"))

MODEL = "0.6B"
CLIPS_PER_GPU = 64
CLIP_SECONDS = 30
MAX_TOKENS = 128
SEED = 20260418
METRIC = "RTFx (audio-sec/sec) Qwen3-ASR-0.6B batched"
UNIT = "audio-seconds/second"
DUMP_LIMIT = 64 << 20  # bytes that --dump-outputs may write in all


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def clip_indices(rank, per_gpu=None):
    """Utterance sharding: rank r owns clips [r * per_gpu, (r + 1) * per_gpu) — disjoint, no data-path collective."""
    per_gpu = CLIPS_PER_GPU if per_gpu is None else per_gpu
    return list(range(rank * per_gpu, (rank + 1) * per_gpu))


def make_clips(rank):
    from q3asr import synth  # input data generator shared with the tests (not oracle arithmetic)
    n = CLIP_SECONDS * 16000
    return [synth.clip(i, n) for i in clip_indices(rank)]


def max_over_ranks_cpu(x, world):
    """The timing reduction of the N > 1 path on a CPU (gloo) group; bench.main uses the same all_reduce(MAX) on CUDA tensors."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return float(x)
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def cpu_sample(seconds, tokens, clips=1, state_dict=None, threads=None):
    """Times the CPU oracle (fp32, torch-CPU matmuls, all host threads) on `clips` clips one after the other, as the reference's
    own serial loop does (TranscribeBatchCommand.swift:82); returns (callable -> seconds, cores, description)."""
    import torch
    from oracle import mel as omel
    from oracle import model as omodel
    from oracle import weights
    from q3asr import synth
    cfg = weights.preset(MODEL)
    if state_dict is None:
        state_dict = weights.random_state_dict(cfg, SEED)
    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    orc = omodel.Oracle(cfg, state_dict, emulate_bf16=False)
    xs = [synth.clip(i, seconds * 16000) for i in range(clips)]

    def once():
        t0 = time.perf_counter()
        for x in xs:
            feats = omel.mel(x)
            emb = orc.encode(feats)
            orc.greedy(emb, tokens, stop_on_eos=False)
        return time.perf_counter() - t0
    return once, cores, (f"{clips} clip(s) x {seconds} s one after the other, mel + encoder + prefill + {tokens} greedy tokens each, "
                         f"fp32 torch-CPU, {cores} threads")


def cpu_mel_gbs(clips):
    """The reference's CPU mel path (AudioPreprocessing.swift:209-293: serial frame loop, dense 257 x 128 product) as restated in
    oracle/mel_oracle.c, timed (i) on one thread, as the reference runs it, and (ii) over clips on all host cores.  Algorithmic
    bytes as for the GPU kernel: 7.2 B per input sample."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import mel as omel
    omel.mel(clips[0][:16000])  # builds / loads the C library
    by = lambda xs: sum(4.0 * x.size + 4.0 * 128 * (x.size // 160) for x in xs)
    def best_of(fn, reps=3):
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            t.append(time.perf_counter() - t0)
        return min(t)
    one = by(clips[:1]) / best_of(lambda: omel.mel(clips[0])) / 1e9
    cores = os.cpu_count() or 1
    sample = (clips * (1 + cores // max(len(clips), 1)))[:max(1, cores)]  # one clip per thread
    with ThreadPoolExecutor(cores) as ex:  # ctypes releases the GIL for the duration of the C call
        allc = by(sample) / best_of(lambda: list(ex.map(omel.mel, sample))) / 1e9
    return {"gbs_1_thread": one, "gbs_all_cores": allc, "cores": cores, "kind": "port",
            "sample": f"1 clip on one thread; {len(sample)} clips of {CLIP_SECONDS} s over {cores} threads (oracle/mel_oracle.c)"}


def _bf16_ulp(x):
    return float(np.exp2(np.floor(np.log2(max(abs(float(x)), 2.0 ** -20))) - 7))


def parity_check(model, state_dict, clip, tokens, noise_ulps=40):
    """The bf16-emulating CPU oracle on one clip of the workload against the GPU's ids for the same clip (the checker of tests/,
    run here on the bench's own weights).  Free-running ids agree until the first step whose top-1 / top-2 margin is inside the
    bf16 noise two summation orders show (tests/golden/make_golden.py); teacher-forcing the oracle's ids compares every step."""
    from oracle import mel as omel
    from oracle import model as omodel
    from oracle import weights
    orc = omodel.Oracle(weights.preset(MODEL), state_dict, emulate_bf16=True)
    t0 = time.perf_counter()
    enc = orc.encode(omel.mel(clip))
    ids, tops, margins = orc.greedy(enc, tokens, stop_on_eos=False)
    cpu_s = time.perf_counter() - t0
    got = model.transcribe_ids([clip], max_tokens=tokens, stop_on_eos=False)[0]
    neq = np.nonzero(got != ids)[0]
    prefix = int(neq[0]) if neq.size else tokens
    f_ids, f_tops = model.decode_forced(clip, ids[:-1])
    ulps = np.array([_bf16_ulp(t) for t in tops])
    clear = margins > noise_ulps * ulps
    rec = {"clip_seconds": CLIP_SECONDS, "tokens": tokens, "distinct_ids": len(set(ids.tolist())),
           "ids_equal": bool(prefix == tokens), "ids_equal_prefix": prefix,
           "margin_ulps_at_first_mismatch": None if prefix == tokens else float(margins[prefix] / ulps[prefix]),
           "teacher_forced_equal": int((f_ids == ids).sum()), "teacher_forced_equal_where_margin_clear": int((f_ids[clear] == ids[clear]).sum()),
           "steps_with_clear_margin": int(clear.sum()), "noise_ulps": noise_ulps,
           "best_logit_max_diff_ulps": float((np.abs(f_tops - tops) / ulps).max()), "oracle_seconds": cpu_s,
           "how": "oracle/model.py (bf16-emulating restatement) vs q3asr_transcribe_ids / q3asr_decode_forced on the bench's weights"}
    return rec


def pool_extras(world, steps):
    """Rank 0, after the per-rank section: what the product's own multi-GPU scheduler (q3asr_pool_*, one process, one worker thread per
    GPU) delivers on the same box — weak and strong scaling of the headline workload, and BASELINE configs 4 and 5 (1.7B)."""
    import q3asr
    from q3asr import synth
    out = {}
    devs = tuple(range(world))
    n30 = CLIP_SECONDS * 16000

    def timed(pool, clips, tokens, per_gpu, reps):
        pool.transcribe_ids(clips, tokens, stop_on_eos=False, max_batch_per_gpu=per_gpu)  # warm-up: buffers, graphs
        t0 = time.perf_counter()
        for _ in range(reps):
            pool.transcribe_ids(clips, tokens, stop_on_eos=False, max_batch_per_gpu=per_gpu)
        return (time.perf_counter() - t0) / reps

    pool = q3asr.Pool("0.6B", devices=devs, seed=SEED)
    try:
        clips = [synth.clip(i, n30) for i in range(64 * world)]
        sec = timed(pool, clips, MAX_TOKENS, 64, steps)
        out["e2e_pool"] = {"value": len(clips) * CLIP_SECONDS / sec, "unit": UNIT, "n_gpus": world, "ms_per_step": 1000 * sec,
                           "how": f"q3asr_pool_transcribe_ids over devices 0..{world - 1} in ONE process, {len(clips)} x {CLIP_SECONDS} s host clips, "
                                  f"{MAX_TOKENS} tokens, 64 per GPU"}
        per = max(1, 64 // world)
        sec = timed(pool, clips[:64], MAX_TOKENS, per, steps)
        out["strong_scaling"] = {"value": 64 * CLIP_SECONDS / sec, "unit": UNIT, "n_gpus": world, "clips_total": 64, "clips_per_gpu": per,
                                 "ms_per_step": 1000 * sec,
                                 "how": "BASELINE config 3 as written: 64 x 30 s clips in total, 64 / N per GPU, through the pool; "
                                        "the decode step at 64 / N sequences is latency-bound, so this is far from linear by construction"}
        one = [clips[0]]  # BASELINE config 2: one 30 s clip, 128 tokens, batch 1, on GPU 0 (latency, not throughput)
        lat = []
        pool.transcribe_ids(one, MAX_TOKENS, stop_on_eos=False, max_batch_per_gpu=1)
        for _ in range(5):
            t0 = time.perf_counter()
            pool.transcribe_ids(one, MAX_TOKENS, stop_on_eos=False, max_batch_per_gpu=1)
            lat.append(time.perf_counter() - t0)
        sec = float(np.median(lat))
        out["config2"] = {"value": CLIP_SECONDS / sec, "unit": UNIT, "n_gpus": 1, "ms_per_clip": 1000 * sec, "max_tokens": MAX_TOKENS,
                          "how": "one 30 s host clip through the blocking pool call (mel, encoder, prefill, 128 greedy tokens), median of 5: the "
                                 "decode chain at batch 1 is 196 dependent phases per token, latency-bound"}
    finally:
        pool.close()
    pool = q3asr.Pool("0.6B", devices=devs + devs, seed=SEED)  # throughput mode: two workers per GPU, 256-wide sub-batches
    try:
        base = [synth.clip(i, n30) for i in range(64)]
        clips = [base[i % 64] for i in range(512 * world)]
        sec = timed(pool, clips, MAX_TOKENS, 256, 1)
        out["throughput_mode"] = {"value": len(clips) * CLIP_SECONDS / sec, "unit": UNIT, "n_gpus": world, "clips": len(clips),
                                  "sub_batch": 256, "workers_per_gpu": 2, "s_total": sec,
                                  "how": "512 x 30 s host clips per GPU through q3asr_pool_transcribe_ids with two workers per GPU and 256-wide "
                                         "sub-batches (the decode step's row capacity), 128 tokens: what a large transcription job gets, "
                                         "beside the headline's one batch of 64 per GPU at a time"}
    finally:
        pool.close()
    pool = q3asr.Pool("1.7B", devices=devs, seed=SEED)
    try:
        clips = [synth.clip(1000 + i, 15 * 16000) for i in range(64 * world)]
        sec = timed(pool, clips, 448, 64, 1)
        prompt = q3asr.encoder_tokens(1500) + 16
        kv = 64 * (prompt + 449 / 2.0) * 114688.0
        floor_ms = (3.441e9 + kv) / (peaks()["hbm"] * 1e9) * 1000.0
        out["config4"] = {"value": len(clips) * 15 / sec, "unit": UNIT, "n_gpus": world, "model": "1.7B", "utterances": len(clips),
                          "utterance_seconds": 15, "max_tokens": 448, "s_per_batch": sec, "decode_step_hbm_floor_ms": floor_ms,
                          "how": "64 concurrent 15 s utterances per GPU, paged KV, 448 greedy tokens, through the pool (host buffers in, ids out); "
                                 "s_per_batch includes mel, encoder and prefill"}
        clips = [synth.clip(2000 + i, n30) for i in range(15 * world)]
        sec = timed(pool, clips, 128, 64, 1)
        out["config5"] = {"value": len(clips) * 30 / sec, "unit": UNIT, "n_gpus": world, "model": "1.7B", "windows": len(clips),
                          "audio_minutes": len(clips) * 0.5, "max_tokens": 128, "s_total": sec,
                          "how": "long-form audio cut into 30 s windows (15 per GPU; 120 = 60 min at 8 GPUs), each an independent utterance"}
    finally:
        pool.close()
    return out


def workload_config(world):
    """The workload both arms name (the reference arm runs a bounded sample of it, described in its cpu_baseline.sample)."""
    return {"workload": f"Qwen3-ASR-{MODEL}: {CLIPS_PER_GPU} x {CLIP_SECONDS} s clips per GPU, mel -> encoder -> prefill -> "
                        f"{MAX_TOKENS} greedy tokens (fixed length), random-init weights seed {SEED}",
            "clips_per_gpu": CLIPS_PER_GPU, "clip_seconds": CLIP_SECONDS, "max_tokens": MAX_TOKENS,
            "parallelism": f"dp{world} (utterance-sharded, no collective on the data path)",
            "l2": "256 MiB flush between timed iterations; activations (>5 GB per step) exceed L2"}


def run_reference(args, rank):
    """The reference arm: the CPU restatement of the reference's algorithm (oracle/), all host threads, rank 0 only."""
    if rank != 0:
        return
    seconds, tokens, clips = CLIP_SECONDS, MAX_TOKENS, 1  # one clip of the workload per step, the full decode length
    once, cores, sample = cpu_sample(seconds, tokens, clips)
    for _ in range(args.warmup):
        once()
    t = [once() for _ in range(args.steps)]
    total = float(sum(t))
    val = clips * seconds * args.steps / total
    line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the Swift/MLX reference does not build on Linux; this is the CPU restatement in oracle/ (kind=port)"}
    _emit(line)


def main():
    global MODEL, CLIP_SECONDS, CLIPS_PER_GPU, MAX_TOKENS, METRIC
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default=MODEL, choices=["0.6B", "1.7B"], help="other BASELINE configs; the headline metric is 0.6B")
    ap.add_argument("--clip-seconds", type=int, default=CLIP_SECONDS)
    ap.add_argument("--clips-per-gpu", type=int, default=CLIPS_PER_GPU)
    ap.add_argument("--max-tokens", type=int, default=MAX_TOKENS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-pipelined", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the pool / strong-scaling / 1.7B sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the token ids of the last timed step to DIR/ids.npy (float32)")
    args = ap.parse_args()
    MODEL, CLIP_SECONDS, CLIPS_PER_GPU, MAX_TOKENS = args.model, args.clip_seconds, args.clips_per_gpu, args.max_tokens
    METRIC = f"RTFx (audio-sec/sec) Qwen3-ASR-{MODEL} batched"
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computes; the reference arm has none")
    if args.dump_outputs and world * CLIPS_PER_GPU * MAX_TOKENS * 4 > DUMP_LIMIT:
        ap.error(f"--dump-outputs: the ids of {world} x {CLIPS_PER_GPU} clips x {MAX_TOKENS} tokens exceed {DUMP_LIMIT >> 20} MB")

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # a host-side group for the one long wait of the run (rank 0's single-process section): an NCCL barrier would leave a
        # spinning kernel on every other rank's GPU, taking SMs from the very measurement it waits for
        cpu_group = dist.new_group(backend="gloo")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    import q3asr
    model = q3asr.Qwen3ASRModel.random_init(MODEL, seed=SEED, device=local_rank)
    clips = make_clips(rank)
    audio_s = CLIPS_PER_GPU * CLIP_SECONDS

    # ---- device-timed steps: batch resident in HBM ----
    model.batch_upload(clips)
    for _ in range(args.warmup):
        model.batch_run(q3asr.STAGE_ALL, MAX_TOKENS, False)
        model.sync()
    ids_ref = model.batch_download(CLIPS_PER_GPU, MAX_TOKENS)
    assert all(len(t) == MAX_TOKENS for t in ids_ref)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    l0 = model.launch_count
    dev_ms, stage = 0.0, np.zeros(4)
    for _ in range(args.steps):
        model.flush_l2()  # between timed iterations; outside the event pair
        model.timer_record(0)
        model.batch_run(q3asr.STAGE_ALL, MAX_TOKENS, False)
        model.timer_record(1)
        dev_ms += model.timer_ms(0, 1)
        ids_last = model.batch_download(CLIPS_PER_GPU, MAX_TOKENS)
        stage += model.stage_ms()
    barrier()
    clocks = sampler.stop()
    launches = model.launch_count - l0
    dev_ms = max_over_ranks(dev_ms)
    value = world * audio_s * args.steps / (dev_ms / 1000.0)
    if args.dump_outputs:
        # fixed length (stop_on_eos off), so the ids stack to [clips, max_tokens]; float32 holds every id of the vocabulary exactly
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "ids" if world == 1 else f"ids_rank{rank}"
        np.save(os.path.join(args.dump_outputs, name + ".npy"), np.stack(ids_last).astype(np.float32))

    # ---- end to end: host buffers in, ids out ----
    model.transcribe_ids(clips, MAX_TOKENS, stop_on_eos=False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = model.transcribe_ids(clips, MAX_TOKENS, stop_on_eos=False)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    assert [t.tolist() for t in out] == [t.tolist() for t in ids_ref], "greedy ids changed between runs"
    e2e = world * audio_s * args.steps / e2e_s
    h2d = int(sum(c.nbytes for c in clips))
    d2h = int(CLIPS_PER_GPU * MAX_TOKENS * 4 + CLIPS_PER_GPU * 4)

    # ---- the same K steps through the scheduler's submit / wait calls with two steps in flight per GPU (extra key, not the headline):
    #      the decode steps of two batches interleave on one GPU, and step k + 1's upload overlaps step k's compute ----
    e2e_pipe = None
    if not args.no_pipelined:
        pools = [q3asr.Pool(MODEL, devices=(local_rank,), seed=SEED) for _ in range(2)]
        try:
            for p_ in pools:
                p_.transcribe_ids(clips, MAX_TOKENS, stop_on_eos=False, max_batch_per_gpu=CLIPS_PER_GPU)  # warm-up: buffers, graphs
            barrier()
            t0 = time.perf_counter()
            jobs = [pools[k % 2].submit(clips, MAX_TOKENS, stop_on_eos=False, max_batch_per_gpu=CLIPS_PER_GPU) for k in range(args.steps)]
            outs = [j.wait() for j in jobs]
            pipe_s = max_over_ranks(time.perf_counter() - t0)
            barrier()
            assert all([t.tolist() for t in o] == [t.tolist() for t in ids_ref] for o in outs), "pipelined ids differ"
            e2e_pipe = {"value": world * audio_s * args.steps / pipe_s, "unit": UNIT, "in_flight_per_gpu": 2,
                        "how": "q3asr_pool_submit / q3asr_job_wait on two single-worker pools per GPU, steps alternating between them; "
                               "host buffers in, ids out, same K steps"}
        finally:
            for p_ in pools:
                p_.close()

    # ---- per-kernel-family timing (extra steps, CUDA events around the launches) ----
    pk = peaks()
    roof, roof_mel, roof_gemm, families = None, None, None, None
    if not args.no_profile:
        model.batch_upload(clips)
        model.profile(True)
        nprof = 2
        for _ in range(nprof):
            model.flush_l2()
            model.batch_run(q3asr.STAGE_ALL, MAX_TOKENS, False)
            model.sync()
        rep = model.profile_report()
        model.profile(False)
        families = {k: {"ms_per_step": v["ms"] / nprof, "launches_per_step": v["launches"] // nprof,
                        "tflops": (v["flops"] / max(v["ms"], 1e-9)) / 1e9 if v["flops"] else None,
                        "gbs": (v["bytes"] / max(v["ms"], 1e-9)) / 1e6 if v["bytes"] else None} for k, v in rep.items()}
        # share of the step: the profiled run executes ONE decode step eagerly (the other MAX_TOKENS - 2 are graph replays that
        # events cannot see inside), so a dec_* family stands for (MAX_TOKENS - 1) times its measured time
        def est_ms(k, v):
            if k == "lm_head":  # one call after the prefill + one in the eager decode step
                return v["ms"] / nprof / 2 * MAX_TOKENS
            return v["ms"] / nprof * ((MAX_TOKENS - 1) if k.startswith("dec_") else 1)
        kernel_of = {"dec_layers": "megastep_kernel (28 decoder layers of one decode step)", "dec_attn": "decode_attn_mma_kernel", "mel": "mel_kernel", "dec_qkv": "gemm_skinny_kernel (dec_qkv)",
                     "dec_o": "gemm_skinny_kernel (dec_o)", "dec_down": "gemm_skinny_kernel (dec_down)"}
        # "dec_attn_chain" is a measurement, not part of the step: the decode attention of all layers launched back to back (one
        # event pair around the chain, programmatic dependent launch as in the step graph) after the last decode step
        chain = rep.pop("dec_attn_chain", None)
        families.pop("dec_attn_chain", None)
        ranked = sorted(((est_ms(k, v), k) for k, v in rep.items() if k != "decode_graph_steps" and (v["flops"] or v["bytes"])), reverse=True)
        for k in families:
            families[k]["est_ms_in_step"] = est_ms(k, rep[k])
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")  # dram bytes per launch from the committed ncu --set full captures
        if os.path.exists(tpath):
            traffic = json.load(open(tpath))

        def roof_of(fam):
            v = rep[fam]
            name = kernel_of.get(fam, f"gemm_tc_kernel ({fam})" if v["flops"] else fam)
            hbm = fam.startswith("dec_") or fam in ("mel", "lm_head") or not v["flops"]  # the decode step streams weights and KV
            if hbm:
                ach, peak, unit, src = v["bytes"] / v["ms"] / 1e6, pk["hbm"], "GB/s", f"hbm_gbs, {pk['src']}"
            else:
                ach, peak, unit, src = v["flops"] / v["ms"] / 1e9, pk["tf_sustained"], "TFLOP/s", f"bf16_tflops_sustained, {pk['src']}"
            return {"bound": "hbm" if hbm else "tensor", "kernel": name, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                    "traffic": traffic.get(fam), "peak_source": src, "launches_per_step": v["launches"] // nprof,
                    "ms_per_launch": v["ms"] / v["launches"], "est_share_of_step": est_ms(fam, v) / (dev_ms / args.steps),
                    "algorithmic_per_launch": (v["bytes"] if hbm else v["flops"]) / v["launches"]}

        roof = roof_of(ranked[0][1])  # the dominant kernel of the step: the persistent decode-layers kernel (weights + KV streaming, HBM-bound)
        roof["how"] = ("CUDA events on the library's stream around each launch of the kernel in extra profiled steps of the same workload "
                       "(eager launches; the timed region replays the same launch inside a CUDA graph)")
        if chain and ranked[0][1] == "dec_attn" and chain["ms"] > 0:
            # the same kernel launched for every layer back to back behind ONE event pair (no event records and no launch ramp
            # between the launches, as inside the replayed step): its sustained duration.  `frac` is that figure; the eager
            # single-launch figure stays beside it as `standalone`.
            n_layers = rep["dec_attn"]["launches"] // nprof  # one eager launch per decoder layer and profiled step
            n_launch = (chain["launches"] or 1) * n_layers
            ms_l = chain["ms"] / n_launch
            standalone = {k: roof[k] for k in ("achieved", "frac", "ms_per_launch", "algorithmic_per_launch")}
            roof.update({"achieved": chain["bytes"] / chain["ms"] / 1e6, "ms_per_launch": ms_l,
                         "algorithmic_per_launch": chain["bytes"] / n_launch, "standalone": standalone})
            roof["frac"] = roof["achieved"] / roof["peak"]
            roof["est_share_of_step"] = ms_l * n_layers * (MAX_TOKENS - 1) / (dev_ms / args.steps)
            roof["how"] = ("one CUDA-event pair on the library's stream around the kernel launched for all decoder layers back to back "
                           "(largest context of the step sequence, programmatic dependent launch as inside the replayed step graph), "
                           "in extra profiled steps of the same workload; `standalone` = event pairs around single eager launches")
        # the top dense tensor-core family (encoder / prefill GEMMs and convolutions; the decode-step products are weight streaming)
        tens = [k for _, k in ranked if rep[k]["flops"] > 0 and not k.startswith("dec_") and k != "lm_head" and not k.endswith("attn")]
        roof_gemm = roof_of(tens[0]) if tens else None
        roof_mel = roof_of("mel") if "mel" in rep else None

    # ---- the decode stage as a whole against its HBM floor (weights of every layer + LM head once per step, the keys and values
    #      of every sequence once per layer and step): the number that governs the headline, next to the dominant kernel's ----
    roof_dec = None
    try:
        cf = q3asr.preset(MODEL)
        nq, nkv = cf.dec_heads * cf.dec_head_dim, cf.dec_kv_heads * cf.dec_head_dim
        w_bytes = 2.0 * (cf.dec_layers * (cf.dec_hidden * (nq + 2 * nkv) + nq * cf.dec_hidden + 3 * cf.dec_hidden * cf.dec_inter)
                         + cf.dec_vocab * cf.dec_hidden)
        prompt = q3asr.encoder_tokens(CLIP_SECONDS * 100) + 16  # audio tokens + the chat template around them
        kv_bytes = CLIPS_PER_GPU * (prompt + MAX_TOKENS / 2.0) * cf.dec_layers * 2 * nkv * 2.0
        dec_ms = float(stage[3]) / args.steps / (MAX_TOKENS - 1)
        ach = (w_bytes + kv_bytes) / dec_ms / 1e6
        roof_dec = {"bound": "hbm", "what": "decode stage (all kernels of a decode step)", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
                    "frac": ach / pk["hbm"], "ms_per_decode_step": dec_ms, "floor_ms_per_decode_step": (w_bytes + kv_bytes) / pk["hbm"] / 1e6,
                    "algorithmic_per_step": w_bytes + kv_bytes,
                    "how": "bytes every decode step must move (bf16 weights of all decoder layers and the tied LM head, the cached keys and "
                           "values at the mean context of the 128 steps) / the device-timed decode stage per step, timed region of `value`"}
    except Exception as e:
        roof_dec = {"error": repr(e)}

    # ---- CPU baseline (rank 0, N = 1 only) ----
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sd = model.state_dict()  # the same bf16 weights, read back through the C ABI
        n_cpu = 1  # one clip of the workload with the full decode length: 10-30 s on the box's host cores
        once, cores, sample = cpu_sample(CLIP_SECONDS, MAX_TOKENS, n_cpu, state_dict=sd)
        sec = once()
        cpu = {"value": n_cpu * CLIP_SECONDS / sec, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample + f" ({sec:.1f} s of CPU time)",
               "mel": cpu_mel_gbs(clips)}
        parity = parity_check(model, sd, clips[0], MAX_TOKENS)
    model.close()
    extras = None
    if not args.no_extras:
        barrier()  # every rank has released its handle; rank 0 now drives all N GPUs from one process
        if rank == 0:
            try:
                extras = pool_extras(world, max(1, min(args.steps, 3)))
            except Exception as e:  # the headline line must still be printed
                extras = {"error": repr(e)}
        if world > 1:
            dist.barrier(group=cpu_group)  # the other ranks wait on the host, their GPUs idle

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": workload_config(world),
            "stage_ms_per_step": {k: float(v) / args.steps for k, v in zip(("mel", "encoder", "prefill", "decode"), stage)},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "e2e_pipelined": e2e_pipe,
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_gemm": roof_gemm, "roofline_mel": roof_mel, "roofline_decode_stage": roof_dec,
            "kernel_families": families,
            "cpu_baseline": cpu, "parity": parity,
        }
        if extras:
            line.update(extras)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def _emit(line):
    """The contract is ONE JSON line on stdout: everything else this process (or NCCL, which prints its version banner to
    stdout) writes to fd 1 is diverted to stderr, and the line goes to the saved descriptor."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    main()
