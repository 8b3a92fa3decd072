"""Full-size parity against the committed oracle fixtures (tests/golden/make_golden.py --big), through the C ABI.

BASELINE.json north star: "encoder hidden states within a stated bf16 tolerance, greedy token IDs bit-exact for a fixed decode
length", at the sizes the configs name:
  q06b_clip30s   Qwen3-ASR-0.6B, one 30 s clip (configs 1 and 2): [390, 1024] encoder states, 128 greedy ids
  q06b_ragged    0.6B, a 17.3 s clip: ragged last chunk, attention windows [104, 104, 17]
  q17b_clip15s   Qwen3-ASR-1.7B, one 15 s clip (config 4's shape)
The fixtures are screened so that the ids are a real target (>= 32 distinct tokens in 128 steps, >= 90 % of the margins above
two bf16 ulps); every step carries the oracle's eight best tokens and logits, and the prefill position its logits from both the
bf16-emulating and the plain fp32 oracle (every `sample_step`-th vocabulary entry, which keeps a fixture under 1 MB).

Why not plain equality everywhere: two correct bf16 implementations of an 18-layer encoder + 28-layer decoder do not agree bit for
bit.  Every op rounds to bf16; a different fp32 summation order moves a few values across a rounding boundary and the flips spread.
Measured (tests/golden/make_golden.py, tools/parity_diag.py, DESIGN.md section 2):
  * the oracle against ITSELF with float64 accumulation in the decoder: best logit up to 10 ulps apart, 3-4 % of the argmaxes differ,
    free-running ids diverge after 14-28 steps;
  * the B200 decoder fed the ORACLE's encoder output (q3asr_decode_forced_embeds): best logit median 2-3 / 90th percentile 6-7 /
    largest 9-20 ulps apart, 5-8 % of the argmaxes differ, every disagreement at a margin of at most 12 ulps — the same level;
  * end to end (the kernels' own encoder output, which is 1.25e-2 in relative L2 from the bf16 oracle's — exactly as far as the bf16
    oracle is from the fp32 oracle, 1.1e-2, and the kernels are from the fp32 oracle, 1.1e-2): 90th percentile 8-10, largest
    15-44 ulps, disagreements up to a margin of 29 ulps.
An id is only determined by the arithmetic contract where its top-1 / top-2 margin exceeds that noise.  The bounds used here:
NOISE_DEC = 16 ulps with the decoder isolated, NOISE_E2E = 40 ulps end to end.

What is asserted:
  * encoder, over the FULL output: relative L2 <= 2e-2 against the bf16-emulating oracle, and against the plain fp32 oracle (on
    every `sample_step`-th row) at most 1.5 x what the bf16 oracle itself shows (noise-calibrated) and <= 3e-2;
  * prefill logits: the same noise-calibrated bound against the fp32 oracle on every `sample_step`-th vocabulary entry, and the
    argmax over the full vocabulary among the oracle's in-noise candidates;
  * teacher-forced steps (the oracle's own ids, and a pseudo-random token stream), decoder isolated and end to end, EVERY step
    constrained: the chosen id equals the oracle's wherever the oracle's margin exceeds the bound; elsewhere it is one of the
    oracle's eight best tokens whose logit is within the bound of the best; the chosen token's logit is within 2 x the bound of the
    oracle's logit for it (median <= 6 ulps); at most 15 % (decoder isolated) / 20 % (end to end) of the steps differ from the
    oracle's id;
  * free-running greedy ids: equal to the oracle's on every step before the first in-noise step; a deviation is only accepted at
    such a step, towards an in-noise candidate (nothing after it can be compared).  The test prints the length of the common
    prefix next to the prefix two CPU summation orders share (`cpu_cpu_prefix`);
  * ids do not depend on the batch a clip is decoded in (bit-exact).
"""
import os

import numpy as np
import pytest

from oracle import mel as omel
from oracle import synth

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
NOISE_DEC = 16.0   # bf16 ulps of the best logit: decoder isolated (both sides start from the oracle's audio embeddings)
NOISE_E2E = 40.0   # end to end (each side behind its own encoder)
FIXTURES = {"q06b_clip30s": "0.6B", "q06b_ragged": "0.6B", "q17b_clip15s": "1.7B"}


def _bf16_bits_to_f32(u):
    return (np.asarray(u, dtype=np.uint32) << 16).view(np.float32)


def _ulp(x):
    return float(np.exp2(np.floor(np.log2(max(abs(float(x)), 2.0 ** -20))) - 7))


def _rel_l2(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b), 1e-30))


def _load(name):
    path = os.path.join(GOLD, name + ".npz")
    if not os.path.exists(path):
        pytest.fail(f"{path} is missing: run tests/golden/make_golden.py --big")
    return np.load(path)


@pytest.fixture(scope="module")
def models(built_lib):
    cache = {}

    def get(size, seed):
        if size not in cache:
            for m in cache.values():  # one full-size model resident at a time
                m.close()
            cache.clear()
            cache[size] = built_lib.Qwen3ASRModel.random_init(size, seed=seed)
        return cache[size]
    yield get
    for m in cache.values():
        m.close()


def _allowed(tk_ids, tk_vals, noise_ulps):
    """Tokens a correct implementation may choose at this step: the oracle's best, plus any of its next three within the bound."""
    u = _ulp(tk_vals[0])
    return [int(i) for i, v in zip(tk_ids, tk_vals) if float(tk_vals[0]) - float(v) <= noise_ulps * u]  # includes every exact tie


def check_forced(got_ids, got_tops, ids, tops, margins, tk_ids, tk_vals, noise_ulps, what, max_differ=0.2, min_strict=0.05):
    """Per-step check of a teacher-forced run; returns (steps that differ from the oracle's id, strict steps)."""
    assert len(got_ids) == len(ids), (what, len(got_ids), len(ids))
    differ = strict = 0
    diffs = []
    for s in range(len(ids)):
        u = _ulp(tops[s])
        if margins[s] > noise_ulps * u:
            strict += 1
            assert got_ids[s] == ids[s], (what, s, int(got_ids[s]), int(ids[s]), float(margins[s]) / u)
        else:
            assert got_ids[s] == ids[s] or int(got_ids[s]) in _allowed(tk_ids[s], tk_vals[s], noise_ulps), (what, s, int(got_ids[s]), tk_ids[s].tolist(), tk_vals[s].tolist())
        differ += int(got_ids[s] != ids[s])
        # the oracle's logit of the token the GPU chose
        ref_val = float(tops[s]) if got_ids[s] == ids[s] else float(tk_vals[s][list(tk_ids[s]).index(int(got_ids[s]))])
        diffs.append(abs(float(got_tops[s]) - ref_val) / u)
        assert diffs[-1] <= 2 * noise_ulps, (what, s, float(got_tops[s]), ref_val, u)
    assert np.median(diffs) <= 6, (what, float(np.median(diffs)))
    assert strict >= min_strict * len(ids), (what, strict)  # the share of steps that are plain equality checks
    assert differ <= max_differ * len(ids), (what, differ)
    return differ, strict


def check_free_running(got, ids, tops, margins, tk_ids, tk_vals, noise_ulps, what):
    """Returns the length of the common prefix; a deviation is only accepted at a step whose oracle margin is within the noise
    bound, towards one of the oracle's in-noise candidates."""
    assert len(got) == len(ids), (what, len(got), len(ids))
    for s in range(len(ids)):
        if got[s] != ids[s]:
            u = _ulp(tops[s])
            assert margins[s] <= noise_ulps * u and int(got[s]) in _allowed(tk_ids[s], tk_vals[s], noise_ulps), \
                (what, s, int(got[s]), int(ids[s]), float(margins[s]) / u, tk_ids[s].tolist())
            return s
    return len(ids)


@pytest.mark.parametrize("name", list(FIXTURES))
def test_encoder_full_output(models, name):
    g = _load(name)
    m = models(FIXTURES[name], int(g["seed"]))
    x = synth.clip(int(g["clip_index"]), int(g["n_samples"]))
    mel = m.extract_features(x)
    ref_mel = omel.mel(x)
    assert (np.abs(mel - ref_mel) / np.maximum(1.0, np.abs(ref_mel))).max() <= 1e-4
    enc = m.encode(mel)
    ref = _bf16_bits_to_f32(g["encoder_bf16"])
    assert enc.shape == ref.shape
    e1 = _rel_l2(enc, ref)
    mx = np.abs(enc - ref).max()
    assert e1 <= 2e-2, (name, e1)
    assert mx <= 16 * np.abs(ref).max() * 2.0 ** -8, (name, mx)
    msg = f"{name}: encoder {enc.shape} relL2 vs bf16 oracle {e1:.2e}, max |diff| {mx:.3g}"
    if "encoder_fp32_as_bf16" in g:
        r32 = _bf16_bits_to_f32(g["encoder_fp32_as_bf16"])  # every sample_step-th row
        step = int(g["sample_step"])
        e2, e_ref = _rel_l2(enc[::step], r32), _rel_l2(ref[::step], r32)
        assert e2 <= 3e-2 and e2 <= 1.5 * e_ref, (name, e2, e_ref)
        msg += f"; vs fp32 oracle {e2:.2e} (the bf16 oracle itself: {e_ref:.2e})"
    print(msg)


@pytest.mark.parametrize("name", list(FIXTURES))
def test_prefill_logits_full_vocabulary(models, name):
    g = _load(name)
    m = models(FIXTURES[name], int(g["seed"]))
    x = synth.clip(int(g["clip_index"]), int(g["n_samples"]))
    logits = m.prefill_logits(x)
    got = logits[::int(g["sample_step"])]  # the vocabulary entries the fixture keeps
    l32 = g["prefill_logits_fp32"].astype(np.float32)
    lbf = g["prefill_logits_bf16emu"].astype(np.float32)
    assert got.shape == l32.shape == lbf.shape, (name, got.shape, l32.shape, lbf.shape)
    e_gpu, e_ref = _rel_l2(got, l32), _rel_l2(lbf, l32)
    assert e_gpu <= 1.5 * e_ref + 1e-3, (name, e_gpu, e_ref)
    assert _rel_l2(got, lbf) <= 2.0 * e_ref + 1e-3, (name, _rel_l2(got, lbf), e_ref)
    assert int(np.argmax(logits)) in _allowed(g["topk_ids"][0], g["topk_vals"][0], NOISE_E2E)
    print(f"{name}: prefill logits relL2 vs fp32 oracle {e_gpu:.2e} (the bf16 oracle itself: {e_ref:.2e}), vs bf16 oracle {_rel_l2(got, lbf):.2e}")


@pytest.mark.parametrize("name", list(FIXTURES))
def test_free_running_ids(models, name):
    g = _load(name)
    ids = g["ids"]
    assert len(set(ids.tolist())) >= min(32, len(ids) // 4)  # not an echo fixed point
    m = models(FIXTURES[name], int(g["seed"]))
    x = synth.clip(int(g["clip_index"]), int(g["n_samples"]))
    got = m.transcribe_ids([x], max_tokens=len(ids), stop_on_eos=False)[0]
    first = check_free_running(got, ids, g["tops"], g["margins"], g["topk_ids"], g["topk_vals"], NOISE_E2E, name)
    print(f"{name}: first {first} of {len(ids)} free-running ids equal to the oracle's (two CPU summation orders share {int(g['cpu_cpu_prefix'])})")
    # the same clip inside a batch (other slots: other clips), at batch position 5: ids must not depend on the neighbours
    others = [synth.clip(900 + i, int(g["n_samples"]) - 1600 * i) for i in range(7)]
    batch = others[:5] + [x] + others[5:]
    got_b = m.transcribe_ids(batch, max_tokens=len(ids), stop_on_eos=False)[5]
    assert got_b.tolist() == got.tolist()


@pytest.mark.parametrize("warps", ["8", "2", "1"])
@pytest.mark.parametrize("name", list(FIXTURES))
def test_teacher_forced(models, monkeypatch, name, warps):
    """warps: the decode-attention variant (8 warps per (sequence, kv head): what a batch of one uses by default; 2: large batches;
    1: two single-warp CTAs per item, what the bench's batches of 64 use)."""
    monkeypatch.setenv("Q3ASR_DECODE_ATTN_WARPS", warps)
    g = _load(name)
    m = models(FIXTURES[name], int(g["seed"]))
    x = synth.clip(int(g["clip_index"]), int(g["n_samples"]))
    ids = g["ids"]
    ref_enc = _bf16_bits_to_f32(g["encoder_bf16"])
    msg = f"{name} warps {warps}:"
    for tag, noise, max_differ, min_strict in (("decoder isolated", NOISE_DEC, 0.15, 0.4), ("end to end", NOISE_E2E, 0.2, 0.05)):
        run = (lambda f: m.decode_forced_embeds(x, ref_enc, f)) if tag == "decoder isolated" else (lambda f: m.decode_forced(x, f))
        got_ids, got_tops = run(ids[:-1])  # the oracle's own ids as the forced stream
        d1, s1 = check_forced(got_ids, got_tops, ids, g["tops"], g["margins"], g["topk_ids"], g["topk_vals"], noise, f"{name} own ids, {tag}",
                              max_differ, min_strict)
        msg += f" [{tag}] own ids {len(ids) - d1}/{len(ids)} equal ({s1} strict)"
        if "forced" in g:
            got_ids, got_tops = run(g["forced"])
            d2, s2 = check_forced(got_ids, got_tops, g["forced_ids"], g["forced_tops"], g["forced_margins"], g["forced_topk_ids"],
                                  g["forced_topk_vals"], noise, f"{name} random stream, {tag}", max_differ, min_strict)
            msg += f", random stream {len(got_ids) - d2}/{len(got_ids)} equal ({s2} strict)"
    print(msg)
