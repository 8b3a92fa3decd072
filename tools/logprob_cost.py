#!/usr/bin/env python
"""What asking for per-token log-probabilities costs: prefill- and decode-stage device time (q3asr_stage_ms) of the same resident
batch with them off and on, the two settings alternated run by run so that drift of the shared machine hits both alike.
Prints the card and its power limit beside the numbers, the median of each setting and its spread (min..max).
Usage: python tools/logprob_cost.py [size] [clips,clips,...] [seconds] [tokens] [reps]"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "qwen3-asr-swift_b200"))
import q3asr  # noqa: E402
from q3asr import synth  # noqa: E402  (input data only)

size = sys.argv[1] if len(sys.argv) > 1 else "0.6B"
batches = [int(b) for b in (sys.argv[2] if len(sys.argv) > 2 else "64,256").split(",")]
secs = int(sys.argv[3]) if len(sys.argv) > 3 else 30
tokens = int(sys.argv[4]) if len(sys.argv) > 4 else 128
reps = int(sys.argv[5]) if len(sys.argv) > 5 else 5

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print(f"card: {card.splitlines()[0] if card else 'unknown'}", flush=True)
m = q3asr.Qwen3ASRModel.random_init(size)
for B in batches:
    clips = [synth.clip(i, 16000 * secs) for i in range(B)]
    t = {False: [], True: []}
    ids = {}
    for r in range(reps + 1):  # run 0 of each setting warms up
        for lp in (False, True) if r % 2 == 0 else (True, False):
            m.batch_upload(clips)
            if lp:
                m.batch_set_logprobs(True)
            m.batch_run(q3asr.STAGE_ALL, tokens, False)
            m.sync()
            ids[lp] = m.batch_download(B, tokens)
            if r > 0:
                t[lp].append(m.stage_ms()[2:4].astype(np.float64))
    same = all(a.tolist() == b.tolist() for a, b in zip(ids[False], ids[True]))
    off, on = np.array(t[False]), np.array(t[True])
    for k, stage in enumerate(("prefill", "decode")):
        mo, mn = np.median(off[:, k]), np.median(on[:, k])
        print(f"{size} {B:4d} x {secs} s, {tokens} tokens, {stage:7s}: off {mo:8.3f} ms [{off[:, k].min():.3f}..{off[:, k].max():.3f}]  "
              f"on {mn:8.3f} ms [{on[:, k].min():.3f}..{on[:, k].max():.3f}]  cost {100.0 * (mn - mo) / mo:+6.2f} %", flush=True)
    print(f"{size} {B:4d}: ids identical with and without log-probabilities: {same}", flush=True)
m.close()
