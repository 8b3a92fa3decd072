"""Generates the committed golden fixtures from the CPU oracle (run here, on CPU):
    python tests/golden/make_golden.py            small fixtures (seconds)
    python tests/golden/make_golden.py --big      + the full-size fixtures below (tens of minutes: it screens clips)
mel_golden.npz      inputs + oracle log-mel for four small clips
tiny_golden.npz     encoder output + greedy ids + teacher-forced argmax of the tiny configuration
q06b_clip30s.npz    (--big) Qwen3-ASR-0.6B dims, one 30 s clip (BASELINE configs 1/2): full [390,1024] encoder output of the
                    bf16-emulating oracle and every fourth row of the plain fp32 oracle's, 128 free-running greedy ids, 128
                    teacher-forced steps on a pseudo-random token stream (ids, best logit, margin)
q06b_ragged.npz     (--big) 0.6B, a 17.3 s clip (1730 frames: ragged last chunk, windows [104,104,17]): encoder + 32 ids
q17b_clip15s.npz    (--big) Qwen3-ASR-1.7B dims, one 15 s clip (BASELINE config 4's shape): the same contents as q06b_clip30s
The reference itself cannot be imported (Swift + MLX); these are outputs of the restatement in oracle/.

Two correct bf16 implementations of a 28-layer decoder do not produce bit-identical logits: every op rounds its output to
bf16, a different fp32 summation order moves a few values across a rounding boundary, and the flips spread.  Measured here with
the oracle itself (the decoder run again with float64 accumulation, same rounding points): final hidden states differ by 1-4 %
in relative L2 and the best logit by up to ~8 bf16 ulps, for these weights and equally for the plain 0.02-scaled ones.  Greedy ids
are therefore bit-exact between implementations only where the top-1 / top-2 margin exceeds that noise.  NOISE_ULPS = 24 is the screening
bound here; the tests use 16 ulps with the decoder isolated and 40 end to end, from the measured deviations of the B200 kernels
against this oracle (tools/parity_diag.py, tests/test_gpu_golden.py).

A full-size fixture is only written when its ids are a meaningful parity target (SURVEY.md section 7): at least 32 distinct
tokens among the 128 free-running ids, at least 90 % of the steps with a margin above two bf16 ulps and at least 35 % above
NOISE_ULPS (those steps are strict equality checks in the tests; on the rest the implementation under test must pick one of the
oracle's eight best tokens whose logit is within NOISE_ULPS of the best, and may differ from the oracle's id on at most 20 % of
all steps).  The fixture also holds the logits of the prefill position (every SAMPLE_STEP-th vocabulary entry) from the bf16-emulating
and from the plain fp32 oracle: the tests require the kernels to be as close to the fp32 model as the bf16 restatement is (a
noise-calibrated bound).  Clips are screened in index order until one passes.
Each fixture also records how many leading ids the float64-accumulation run shares with the fp32 one (`cpu_cpu_prefix`): the
length over which free-running ids are determined by the arithmetic contract at all.
"""
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import mel as omel  # noqa: E402
from oracle import model as omodel  # noqa: E402
from oracle import synth, weights  # noqa: E402

SEED = 20260418


def bf16_ulp(x):
    """Spacing of bf16 numbers at |x| (8 significant bits)."""
    x = np.maximum(np.abs(np.asarray(x, dtype=np.float64)), 1e-30)
    return np.exp2(np.floor(np.log2(x)) - 7)


def to_bf16_bits(x):
    """bf16-representable float32 -> uint16 (the fixtures store encoder states this way: half the bytes, exact)."""
    return (np.ascontiguousarray(weights.bf16_round(x), dtype=np.float32).view(np.uint32) >> 16).astype(np.uint16)


NOISE_ULPS = 24
SAMPLE_STEP = 4  # stride of the stored fp32-oracle encoder rows and prefill logits


def margin_report(ids, tops, margins):
    ulp = bf16_ulp(tops)
    return dict(distinct=len(set(ids.tolist())), frac_gt2=float((margins > 2 * ulp).mean()),
                frac_gt_noise=float((margins > NOISE_ULPS * ulp).mean()), median_margin_ulps=float(np.median(margins / ulp)))


def acceptable(rep, n):
    return rep["distinct"] >= min(32, n // 4) and rep["frac_gt2"] >= 0.9 and rep["frac_gt_noise"] >= 0.35


def full_size_fixture(path, preset, n_samples, n_free, n_forced, first_clip, max_trials, fp32_weights_too=True):
    cfg = weights.preset(preset)
    t0 = time.time()
    sd = weights.random_state_dict(cfg, SEED)
    print(f"{preset}: weights in {time.time() - t0:.0f} s", flush=True)
    orc = omodel.Oracle(cfg, sd)
    orc64 = omodel.Oracle(cfg, sd, decoder_fp64=True)
    chosen = None
    for clip in range(first_clip, first_clip + max_trials):
        x = synth.clip(clip, n_samples)
        feats = omel.mel(x)
        enc = orc.encode(feats)
        ids, tops, margins = orc.greedy(enc, n_free, stop_on_eos=False)
        rep = margin_report(ids, tops, margins)
        tk_ids, tk_vals = np.stack(orc.topk_ids), np.stack(orc.topk_vals)
        print(f"  clip {clip}: {rep}", flush=True)
        if acceptable(rep, n_free):
            chosen = clip
            break
    assert chosen is not None, "no clip passed the screening: widen max_trials"
    # the same decode with float64 accumulation: how far two CPU summation orders agree, and how far apart their logits are
    ids64, tops64, _ = orc64.greedy(enc, n_free, stop_on_eos=False)
    neq = np.nonzero(ids64 != ids)[0]
    prefix = int(neq[0]) if neq.size else n_free
    f64 = orc64.greedy(enc, 0, forced=ids[:-1])  # teacher-forced on the fp32 run's ids: logits of the same contexts
    noise = float((np.abs(f64[1] - tops) / bf16_ulp(tops)).max())
    print(f"    float64 accumulation: first {prefix} of {n_free} free-running ids equal; teacher-forced best logit differs by up to "
          f"{noise:.1f} ulp, {int((f64[0] != ids).sum())} of {n_free} argmax differ", flush=True)
    out = dict(seed=SEED, clip_index=chosen, n_samples=n_samples, encoder_bf16=to_bf16_bits(enc), ids=ids, tops=tops, margins=margins,
               topk_ids=tk_ids, topk_vals=tk_vals, cpu_cpu_prefix=prefix, cpu_cpu_noise_ulps=noise, noise_ulps=NOISE_ULPS)
    if n_forced:
        forced = np.random.default_rng(1000 + chosen).integers(0, cfg["dec_vocab"] - 2000, size=n_forced).astype(np.int32)
        fids, ftops, fmargins = orc.greedy(enc, 0, forced=forced)
        ftk_ids, ftk_vals = np.stack(orc.topk_ids), np.stack(orc.topk_vals)
        frep = margin_report(fids, ftops, fmargins)
        print(f"  teacher-forced on a pseudo-random stream: {frep}", flush=True)
        assert frep["frac_gt_noise"] >= 0.3, frep
        out.update(forced=forced, forced_ids=fids, forced_tops=ftops, forced_margins=fmargins, forced_topk_ids=ftk_ids,
                   forced_topk_vals=ftk_vals)
    # the reference's encoder runs in fp32 on an fp32 mel: the plain fp32 oracle states the bf16 tolerance, for the encoder states and
    # for the logits of the prefill position (float16).  These tolerance arrays keep every SAMPLE_STEP-th encoder row and vocabulary
    # entry, so that a fixture stays under 1 MB; the bf16 encoder states above stay whole (the decoder-isolated tests feed them in).
    o32 = omodel.Oracle(cfg, sd, emulate_bf16=False)
    enc32 = o32.encode(feats)
    if fp32_weights_too:
        out["encoder_fp32_as_bf16"] = to_bf16_bits(enc32)[::SAMPLE_STEP]
    out["prefill_logits_fp32"] = o32.prefill(enc32)[0].numpy().astype(np.float16)[::SAMPLE_STEP]
    out["prefill_logits_bf16emu"] = orc.prefill(enc)[0].numpy().astype(np.float16)[::SAMPLE_STEP]
    out["sample_step"] = SAMPLE_STEP
    np.savez_compressed(path, **out)
    print(f"  wrote {os.path.basename(path)} ({os.path.getsize(path) / 1e6:.2f} MB) ids[:16] {ids[:16].tolist()}", flush=True)


def main():
    out = {}
    imp = np.zeros(4000, np.float32)
    imp[2000] = 1.0
    for name, x in (("mel_clip0_1600", synth.clip(0, 1600)), ("mel_clip1_16000", synth.clip(1, 16000)),
                    ("mel_zeros_3200", np.zeros(3200, np.float32)), ("mel_impulse_4000", imp)):
        out[name + "_x"] = x
        out[name + "_y"] = omel.mel(x)
    np.savez_compressed(os.path.join(HERE, "mel_golden.npz"), **out)

    cfg = weights.preset("tiny")
    orc = omodel.Oracle(cfg, weights.random_state_dict(cfg, SEED))
    x = synth.clip(0, 16000 * 3 + 777)
    enc = orc.encode(omel.mel(x))
    ids, tops, margins = orc.greedy(enc, 32, stop_on_eos=False)
    forced = np.random.default_rng(11).integers(0, 2000, size=24).astype(np.int32)
    fids, ftops, fmargins = orc.greedy(enc, 0, forced=forced)
    np.savez_compressed(os.path.join(HERE, "tiny_golden.npz"), seed=SEED, clip_index=0, n_samples=x.size, encoder=enc, ids=ids,
                        tops=tops, margins=margins, forced=forced, forced_ids=fids, forced_tops=ftops, forced_margins=fmargins)
    print("tiny ids", ids.tolist(), margin_report(ids, tops, margins))

    if "--big" in sys.argv:
        which = [a for a in sys.argv[1:] if not a.startswith("--")]
        if not which or "q06b_clip30s" in which:
            full_size_fixture(os.path.join(HERE, "q06b_clip30s.npz"), "0.6B", 480000, 128, 128, 0, 60)
        if not which or "q06b_ragged" in which:
            full_size_fixture(os.path.join(HERE, "q06b_ragged.npz"), "0.6B", 1730 * 160 + 57, 32, 0, 100, 40, fp32_weights_too=False)
        if not which or "q17b_clip15s" in which:
            full_size_fixture(os.path.join(HERE, "q17b_clip15s.npz"), "1.7B", 240000, 128, 128, 200, 60)


if __name__ == "__main__":
    main()
