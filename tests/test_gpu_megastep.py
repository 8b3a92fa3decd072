"""The persistent decode-step kernel (csrc/megastep.cuh, opt-in with Q3ASR_MEGA=1) against the default multi-kernel decode step.

Both paths perform the same arithmetic in the same order (same split-K partition and k order in the products, the same
fixed-order split reductions, the same canonical key streams in the attention), so ids AND best logits must be bit-identical —
for every shape the kernel specialises on: sub-batch tiles of 16 / 32 / 64 token columns, 2 or 8 warps per attention item, one sub-batch (a single sequence) or two, both model sizes (gate|up tiles of 64 and 128 columns).
"""
import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu


def _clips(n, base):
    return [synth.clip(base + i, 16000 + 2400 * ((i * 7) % 11)) for i in range(n)]


def _run(m, monkeypatch, mega, clips, tokens):
    monkeypatch.setenv("Q3ASR_MEGA", "1" if mega else "0")
    l0 = m.launch_count
    ids = m.transcribe_ids(clips, max_tokens=tokens, stop_on_eos=False)
    return [t.tolist() for t in ids], m.launch_count - l0


@pytest.mark.parametrize("size,batches", [("0.6B", (1, 5, 40, 70, 100, 128)), ("1.7B", (3, 64))])
def test_megastep_matches_multi_kernel_path(built_lib, monkeypatch, size, batches):
    m = built_lib.Qwen3ASRModel.random_init(size, seed=20260418)
    try:
        for B in batches:
            clips = _clips(B, 300 + B)
            tokens = 40
            ref, l_ref = _run(m, monkeypatch, False, clips, tokens)
            got, l_got = _run(m, monkeypatch, True, clips, tokens)
            assert got == ref, (size, B, [i for i, (a, b) in enumerate(zip(got, ref)) if a != b][:8])
            assert l_got < l_ref, (size, B, l_got, l_ref)  # the persistent kernel really ran: far fewer launches
            assert len({tuple(t) for t in got}) > 1 or B == 1
        # teacher-forced best logits, one sequence: identical floats
        x = synth.clip(77, 16000 * 4)
        forced = np.random.default_rng(3).integers(0, 150000, size=12).astype(np.int32)
        monkeypatch.setenv("Q3ASR_MEGA", "0")
        ids0, top0 = m.decode_forced(x, forced)
        monkeypatch.setenv("Q3ASR_MEGA", "1")
        ids1, top1 = m.decode_forced(x, forced)
        assert ids0.tolist() == ids1.tolist() and top0.tolist() == top1.tolist()
    finally:
        m.close()


def test_megastep_matches_multi_kernel_path_at_long_context(built_lib, monkeypatch):
    """Contexts of 500 to 1 200 keys: every one of the 8 key streams of an attention item holds several 16-key chunks, so the
    persistent kernel's own copy of the attention body (megastep.cuh attention_item) runs its chunk walk, the online-softmax
    rescale within a stream and the stream merge at depth; the short-clip tests above stay within one or two chunks per stream.
    The multi-kernel side is pinned to a float64 reference by test_gpu_decode_attention.py."""
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418)
    try:
        clips = [synth.clip(900 + i, 16000 * 30 - 1111 * i) for i in range(6)]
        context = np.random.default_rng(11).integers(0, 150000, size=600).astype(np.int32)
        prompts = [None] * 5 + [{"context": context}]
        runs, launches = [], []
        for mega in ("0", "1"):
            monkeypatch.setenv("Q3ASR_MEGA", mega)
            l0 = m.launch_count
            runs.append([t.tolist() for t in m.transcribe_ids(clips, max_tokens=160, stop_on_eos=False, prompts=prompts)])
            launches.append(m.launch_count - l0)
        assert runs[1] == runs[0], [i for i, (a, b) in enumerate(zip(runs[0], runs[1])) if a != b]
        assert all(len(t) == 160 for t in runs[0])
        assert launches[1] < launches[0], launches  # the persistent kernel really ran
        forced = np.random.default_rng(12).integers(0, 150000, size=300).astype(np.int32)
        monkeypatch.setenv("Q3ASR_MEGA", "0")
        ids0, top0 = m.decode_forced(clips[0], forced)
        monkeypatch.setenv("Q3ASR_MEGA", "1")
        ids1, top1 = m.decode_forced(clips[0], forced)
        assert ids0.tolist() == ids1.tolist() and top0.tolist() == top1.tolist()
    finally:
        m.close()


def test_megastep_stop_on_eos_and_long_decode(built_lib, monkeypatch):
    """A longer decode (KV pages cross several page boundaries, contexts of different lengths in one batch) and the EOS path."""
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418)
    try:
        clips = [synth.clip(500 + i, 16000 * (1 + i % 4) + 777 * i) for i in range(9)]
        ref, _ = _run(m, monkeypatch, False, clips, 70)
        got, _ = _run(m, monkeypatch, True, clips, 70)
        assert got == ref
        monkeypatch.setenv("Q3ASR_MEGA", "0")
        r0 = [t.tolist() for t in m.transcribe_ids(clips, max_tokens=40, stop_on_eos=True)]
        monkeypatch.setenv("Q3ASR_MEGA", "1")
        r1 = [t.tolist() for t in m.transcribe_ids(clips, max_tokens=40, stop_on_eos=True)]
        assert r0 == r1
    finally:
        m.close()
