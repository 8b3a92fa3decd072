#!/usr/bin/env python
"""GPU vs oracle fixture, step by step (no assertions): best-logit difference in bf16 ulps, argmax agreement, margins.
Usage: python tools/parity_diag.py [fixture ...]"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "qwen3-asr-swift_b200"))
import q3asr  # noqa: E402
from oracle import mel as omel  # noqa: E402
from q3asr import synth  # noqa: E402

SIZES = {"q06b_clip30s": "0.6B", "q06b_ragged": "0.6B", "q17b_clip15s": "1.7B"}


def ulp(x):
    return np.exp2(np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -20))) - 7)


for name in (sys.argv[1:] or list(SIZES)):
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    if not os.path.exists(path):
        print(name, "missing")
        continue
    g = np.load(path)
    m = q3asr.Qwen3ASRModel.random_init(SIZES[name], seed=int(g["seed"]))
    x = synth.clip(int(g["clip_index"]), int(g["n_samples"]))
    enc = m.encode(m.extract_features(x))
    ref = (np.asarray(g["encoder_bf16"], dtype=np.uint32) << 16).view(np.float32)
    rel = np.linalg.norm(enc - ref) / np.linalg.norm(ref)
    msg = f"{name}: encoder relL2 vs bf16 oracle {rel:.3e}, max |diff| {np.abs(enc - ref).max():.3g} (max |ref| {np.abs(ref).max():.3g})"
    if "encoder_fp32_as_bf16" in g:
        r32 = (np.asarray(g["encoder_fp32_as_bf16"], dtype=np.uint32) << 16).view(np.float32)  # every sample_step-th row
        step = int(g["sample_step"])
        msg += (f", vs fp32 oracle {np.linalg.norm(enc[::step] - r32) / np.linalg.norm(r32):.3e}; bf16 oracle vs fp32 oracle "
                f"{np.linalg.norm(ref[::step] - r32) / np.linalg.norm(r32):.3e} (every {step}th row)")
    print(msg)
    streams = (("own ids", g["ids"][:-1], g["ids"], g["tops"], g["margins"]),) + (
        (("random stream", g["forced"], g["forced_ids"], g["forced_tops"], g["forced_margins"]),) if "forced" in g else ())
    for tag, forced, ids, tops, margins in [(t + " (GPU encoder)",) + tuple(r) for t, *r in streams] + [(t + " (ORACLE encoder output)",) + tuple(r) for t, *r in streams]:
        got_ids, got_tops = m.decode_forced_embeds(x, ref, forced) if "ORACLE" in tag else m.decode_forced(x, forced)
        u = ulp(tops)
        d = np.abs(got_tops - tops) / u
        same = got_ids == ids
        mu = margins / u
        print(f"  {tag}: argmax equal {int(same.sum())}/{len(ids)}; |best logit diff| ulps: median {np.median(d):.1f} p90 {np.percentile(d, 90):.1f} "
              f"max {d.max():.1f}; where equal: max {d[same].max():.1f}")
        print("    mismatching steps (step, margin ulps, diff ulps):", [(int(s), round(float(mu[s]), 1), round(float(d[s]), 1)) for s in np.nonzero(~same)[0]])
        print("    steps with diff > 8 ulps (step, margin ulps, diff ulps):", [(int(s), round(float(mu[s]), 1), round(float(d[s]), 1)) for s in np.nonzero(d > 8)[0]])
    ids = g["ids"]
    got = m.transcribe_ids([x], max_tokens=len(ids), stop_on_eos=False)[0]
    neq = np.nonzero(got != ids)[0]
    print(f"  free-running: first {int(neq[0]) if neq.size else len(ids)} of {len(ids)} ids equal (two CPU orders: {int(g['cpu_cpu_prefix'])}; "
          f"CPU-CPU best-logit noise {float(g['cpu_cpu_noise_ulps']):.1f} ulps)")
    m.close()
