#!/usr/bin/env python
"""Continuous batching against the static schedule, on the workloads where utterances stop at ragged steps.

Static: transcribe_ids in sub-batches of 256 utterances, one after the other, each compacting its finished rows.  Continuous:
q3asr_transcribe_ids_continuous with 256 resident rows, refilled from the waiting utterances.  The 0.6B random-init model gets a
token it emits at spread-out steps as its EOS token (the trick of tests/test_gpu_compaction.py), so utterances finish at ragged
steps as real speech does.  Workloads: 1024 x 30 s, 1024 mixed 5-30 s, the 30 s set without EOS (every row runs to max_tokens,
all finish together), and the pool with two workers on one GPU.  The two schedules alternate run by run (three each after a
warm-up); medians are printed with the card and its power limit, plus the histogram of utterance lengths and whether the ids of
the two schedules are equal.
Usage: python tools/continuous_batching.py [clips] [tokens] [reps]"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "qwen3-asr-swift_b200"))
import q3asr  # noqa: E402
from q3asr import synth  # noqa: E402  (input data only)

N = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
TOKENS = int(sys.argv[2]) if len(sys.argv) > 2 else 448
REPS = int(sys.argv[3]) if len(sys.argv) > 3 else 3
ROWS = 256
SEED = 20260418

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print(f"card: {card.splitlines()[0] if card else 'unknown'}", flush=True)

full = [synth.clip(i, 16000 * 30) for i in range(N)]
rng = np.random.default_rng(7)
mixed = [synth.clip(5000 + i, int(16000 * s)) for i, s in enumerate(rng.uniform(5.0, 30.0, N))]


def ragged_eos():
    """the token whose first occurrences are most spread over the steps, among those at least half of 64 clips emit"""
    m = q3asr.Qwen3ASRModel.random_init("0.6B", seed=SEED)
    free = [t.tolist() for t in m.transcribe_ids(full[:64], max_tokens=TOKENS, stop_on_eos=False)]
    m.close()
    firsts = {}
    for ids in free:
        seen = set()
        for s, t in enumerate(ids):
            if t not in seen:
                seen.add(t)
                firsts.setdefault(t, []).append(s)
    return max(firsts, key=lambda t: (len(firsts[t]) >= 32) * (np.std(firsts[t]) + 0.01 * len(firsts[t])))


cfg = q3asr.preset("0.6B")
cfg.tok_eos = int(ragged_eos())
print(f"EOS token for the ragged workloads: {cfg.tok_eos}", flush=True)
m = q3asr.Qwen3ASRModel.random_init("0.6B", seed=SEED, config=cfg)


def run_static(clips, eos):
    t0 = time.perf_counter()
    ids, steps, row_steps = [], 0, 0
    for b0 in range(0, len(clips), ROWS):
        ids += m.transcribe_ids(clips[b0:b0 + ROWS], max_tokens=TOKENS, stop_on_eos=eos)
        st = m.decode_stats()
        steps += st["steps"]
        row_steps += st["row_steps"]
    return time.perf_counter() - t0, ids, row_steps / max(steps, 1), 0, 0.0


def run_continuous(clips, eos):
    t0 = time.perf_counter()
    ids = m.transcribe_ids(clips, max_tokens=TOKENS, stop_on_eos=eos, continuous_rows=ROWS)
    dt = time.perf_counter() - t0
    st, adm, ms = m.decode_stats(), m.decode_admissions(), m.stage_ms()
    return dt, ids, st["row_steps"] / max(st["steps"], 1), adm["admissions"], float(ms[0] + ms[1] + ms[2])


def compare(name, clips, eos, runs):
    audio = sum(c.size for c in clips) / 16000.0
    res = {k: [] for k in runs}
    ids = {}
    for r in range(REPS + 1):  # run 0 of each schedule warms up
        for k in (list(runs) if r % 2 == 0 else list(runs)[::-1]):
            out = runs[k](clips, eos)
            ids[k] = [t.tolist() for t in out[1]]
            if r > 0:
                res[k].append(out)
    lens = np.array([len(t) for t in ids[list(runs)[0]]])
    hist, edges = np.histogram(lens, bins=[1, 2, 17, 65, 129, 257, TOKENS, TOKENS + 1])
    print(f"\n{name}: {len(clips)} clips, {audio:.0f} s of audio, max_tokens {TOKENS}, stop_on_eos {eos}")
    print("  utterance lengths: " + ", ".join(f"[{edges[i]},{edges[i + 1]}): {hist[i]}" for i in range(len(hist))))
    for k, rs in res.items():
        dt = np.array([x[0] for x in rs])
        med = float(np.median(dt))
        print(f"  {k:10s}: {med * 1000:9.1f} ms [{dt.min() * 1000:.1f}..{dt.max() * 1000:.1f}]  {audio / med:8.1f} audio-s/s  "
              f"{lens.sum() / med:9.1f} tokens/s  mean rows/step {np.median([x[2] for x in rs]):6.1f}  admissions {rs[-1][3]}  "
              f"mel+encoder+prefill {np.median([x[4] for x in rs]):8.1f} ms", flush=True)
    keys = list(runs)
    print(f"  ids equal: {ids[keys[0]] == ids[keys[1]]}", flush=True)


both = {"static": run_static, "continuous": run_continuous}
compare("1024 x 30 s, ragged EOS", full, True, both)
compare("1024 mixed 5-30 s, ragged EOS", mixed, True, both)
compare("1024 x 30 s, no EOS", full, False, both)
m.close()

pools = {}
for k, cont in (("pool", False), ("pool cont", True)):
    pools[k] = q3asr.Pool("0.6B", devices=(0, 0), seed=SEED, config=cfg, continuous=cont)


def pool_runner(k):
    def run(clips, eos):
        t0 = time.perf_counter()
        ids = pools[k].transcribe_ids(clips, max_tokens=TOKENS, stop_on_eos=eos, max_batch_per_gpu=ROWS)
        return time.perf_counter() - t0, ids, float("nan"), 0, float("nan")
    return run


compare("pool, two workers on one GPU, 1024 mixed 5-30 s, ragged EOS", mixed, True, {k: pool_runner(k) for k in pools})
for p in pools.values():
    p.close()
