"""Continuous batching (q3asr_transcribe_ids_continuous): one request decoded by one resident batch of at most max_rows rows, the
rows freed by finished utterances refilled with the waiting ones.  Only the schedule changes, so every utterance must come out
with exactly the ids and log-probabilities the static path (q3asr_transcribe_ids*, sub-batches with compaction) gives it.

Workload: the 0.6B random-init model with a token it emits at spread-out steps made the EOS token (the trick of
test_gpu_compaction.py), ~100 clips of 2-6 s, some at 24 kHz, some with context / language prompts, 32 resident rows: several
admissions per call.
"""
import collections
import ctypes
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "qwen3-asr-swift_b200")
TOKENS = 80
ROWS = 32
N = 100
SEED = 20260418
INVALID = 1


def _workload():
    clips, rates, prompts = [], [], []
    for i in range(N):
        secs = 2.0 + 4.0 * ((i * 37) % 23) / 22.0
        rate = 24000 if i % 5 == 3 else 16000
        clips.append(synth.clip(900 + i, int(rate * secs)))
        rates.append(rate)
        p = {}
        if i % 7 == 2:
            p["context"] = [(31 * i + 7 * k) % 5000 + 100 for k in range(3 + i % 17)]
        if i % 11 == 5:
            p["language"] = [1500 + i % 9, 1600]
        prompts.append(p)
    return clips, rates, prompts


@pytest.fixture(scope="module")
def ragged(built_lib):
    """(model with the ragged EOS, clips, rates, prompts, static ids, static log-probabilities, static stats at 32-clip sub-batches)"""
    clips, rates, prompts = _workload()
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=SEED)
    try:
        free = [t.tolist() for t in m.transcribe_ids(clips, max_tokens=TOKENS, stop_on_eos=False, sample_rates=rates, prompts=prompts)]
    finally:
        m.close()
    firsts = collections.defaultdict(list)
    for ids in free:
        seen = set()
        for s, t in enumerate(ids):
            if t not in seen:
                seen.add(t)
                firsts[t].append(s)
    eos = max(firsts, key=lambda t: (len(firsts[t]) >= N // 2) * (np.std(firsts[t]) + 0.01 * len(firsts[t])))
    assert len(firsts[eos]) >= N // 2, "no token is emitted by at least half of the clips: pick other clips"
    cfg = built_lib.preset("0.6B")
    cfg.tok_eos = int(eos)
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=SEED, config=cfg)
    ids, lp = m.transcribe_ids(clips, max_tokens=TOKENS, stop_on_eos=True, sample_rates=rates, prompts=prompts, return_logprobs=True)
    steps = row_steps = 0
    for b0 in range(0, N, ROWS):  # the static schedule at the same row count: sub-batches of 32, one after the other
        m.transcribe_ids(clips[b0:b0 + ROWS], max_tokens=TOKENS, stop_on_eos=True, sample_rates=rates[b0:b0 + ROWS],
                         prompts=prompts[b0:b0 + ROWS])
        st = m.decode_stats()
        steps += st["steps"]
        row_steps += st["row_steps"]
    want = [ids[i].tolist() for i in range(N)]
    assert sum(len(w) < TOKENS for w in want) >= N // 3, "too few utterances stop early"
    yield dict(m=m, cfg=cfg, clips=clips, rates=rates, prompts=prompts, ids=want, lp=lp, static_rows=row_steps / steps)
    m.close()


def _first_diff(got, want):
    return [(i, next((s for s, (a, b) in enumerate(zip(g, w)) if a != b), min(len(g), len(w))), len(g), len(w))
            for i, (g, w) in enumerate(zip(got, want)) if g != w]


@pytest.mark.parametrize("mega", ["0", "1"])
def test_continuous_equals_static(ragged, mega):
    m = ragged["m"]
    old = os.environ.get("Q3ASR_MEGA")
    os.environ["Q3ASR_MEGA"] = mega
    try:
        ids, lp = m.transcribe_ids(ragged["clips"], max_tokens=TOKENS, stop_on_eos=True, sample_rates=ragged["rates"],
                                   prompts=ragged["prompts"], return_logprobs=True, continuous_rows=ROWS)
        st, adm = m.decode_stats(), m.decode_admissions()
    finally:
        if old is None:
            os.environ.pop("Q3ASR_MEGA")
        else:
            os.environ["Q3ASR_MEGA"] = old
    got = [t.tolist() for t in ids]
    bad = _first_diff(got, ragged["ids"])
    assert not bad, f"(utterance, first differing step, got length, want length): {bad[:10]}; stats {st} {adm}"
    for i in range(N):
        assert np.array_equal(lp[i], ragged["lp"][i]), i
    rows = st["row_steps"] / st["steps"]
    print(f"continuous: {st} {adm}, mean rows per step {rows:.1f} against {ragged['static_rows']:.1f} static")
    assert adm["admissions"] >= 2 and adm["admitted"] == N - ROWS
    assert rows > ragged["static_rows"]
    assert st["rows"] <= ROWS


def test_request_order_does_not_matter(ragged):
    m = ragged["m"]
    perm = np.random.default_rng(3).permutation(N)
    ids = m.transcribe_ids([ragged["clips"][i] for i in perm], max_tokens=TOKENS, stop_on_eos=True,
                           sample_rates=[ragged["rates"][i] for i in perm], prompts=[ragged["prompts"][i] for i in perm],
                           continuous_rows=ROWS)
    got = [None] * N
    for j, i in enumerate(perm):
        got[i] = ids[j].tolist()
    assert not _first_diff(got, ragged["ids"])


def _prompt_len(built_lib, cfg, n, rate, prompt):
    L = built_lib.lib()
    n16 = int(L.q3asr_resample_len(n, rate, 16000)) if rate != 16000 else n
    ntok = L.q3asr_encoder_tokens(L.q3asr_mel_frames(n16))
    return built_lib.prompt_ids(cfg, ntok, context=prompt.get("context"), language=prompt.get("language"))[0].size


def test_pages_exactly_full(built_lib, ragged):
    """The longest prompt + max_tokens fills its KV pages to the last slot, and that utterance is admitted last: a finished row that
    kept appending would write past its block into another sequence's pages."""
    m, cfg = ragged["m"], ragged["cfg"]
    clips, rates, prompts = ragged["clips"][:60], ragged["rates"][:60], ragged["prompts"][:60]
    clips = clips + [synth.clip(4242, 16000 * 5)]
    rates = rates + [16000]
    prompts = prompts + [{"context": [(13 * k) % 4000 + 300 for k in range(90)]}]
    lens = [_prompt_len(built_lib, cfg, c.size, r, p) for c, r, p in zip(clips, rates, prompts)]
    assert lens[-1] == max(lens)
    mt = 32 * ((lens[-1] + 60) // 32 + 1) - lens[-1]
    want = m.transcribe_ids(clips, max_tokens=mt, stop_on_eos=True, sample_rates=rates, prompts=prompts)
    got = m.transcribe_ids(clips, max_tokens=mt, stop_on_eos=True, sample_rates=rates, prompts=prompts, continuous_rows=16)
    assert m.decode_admissions()["admissions"] >= 2
    assert not _first_diff([t.tolist() for t in got], [t.tolist() for t in want])


def test_no_eos(ragged):
    m = ragged["m"]
    kw = dict(max_tokens=24, stop_on_eos=False, sample_rates=ragged["rates"][:70], prompts=ragged["prompts"][:70])
    want = m.transcribe_ids(ragged["clips"][:70], **kw)
    got = m.transcribe_ids(ragged["clips"][:70], continuous_rows=ROWS, **kw)
    assert all(len(t) == 24 for t in got) and m.decode_admissions()["admissions"] >= 2
    assert not _first_diff([t.tolist() for t in got], [t.tolist() for t in want])


def test_errors_and_recovery(built_lib, ragged):
    m = ragged["m"]
    L = built_lib.lib()
    clips = [np.ascontiguousarray(c, dtype=np.float32) for c in ragged["clips"][:4]]
    n = np.array([c.size for c in clips], dtype=np.uint64)
    arr = (ctypes.c_void_p * 4)(*[c.ctypes.data for c in clips])
    ids = np.zeros((4, 8), np.int32)
    lens = np.zeros(4, np.int32)
    args = lambda batch, rows: (m._h, ctypes.cast(arr, ctypes.c_void_p), n.ctypes.data, None, batch, None, 8, 1, rows, ids.ctypes.data,
                                lens.ctypes.data, None)
    assert L.q3asr_transcribe_ids_continuous(*args(4, 257)) == INVALID
    assert L.q3asr_transcribe_ids_continuous(*args(0, 32)) == INVALID
    # the same handle still serves the static path and the resident batch
    k = 6
    sub = dict(sample_rates=ragged["rates"][:k], prompts=ragged["prompts"][:k])
    got = m.transcribe_ids(ragged["clips"][:k], max_tokens=TOKENS, stop_on_eos=True, **sub)
    assert [t.tolist() for t in got] == ragged["ids"][:k]
    plain = [c for c, r, p in zip(ragged["clips"], ragged["rates"], ragged["prompts"]) if r == 16000 and not p][:3]
    want = m.transcribe_ids(plain, max_tokens=12, stop_on_eos=False)
    m.batch_upload(plain)
    m.batch_run(max_tokens=12)
    res = m.batch_download(3, 12)
    assert [res[i].tolist() for i in range(3)] == [w.tolist() for w in want]
    assert m.decode_admissions() == dict(admissions=0, admitted=0)


def test_pool_continuous(built_lib, ragged):
    clips = ragged["clips"][:48]
    cfg = ragged["cfg"]
    pool = built_lib.Pool("0.6B", devices=(0, 0), seed=SEED, config=cfg)
    try:
        want = pool.transcribe_ids(clips, max_tokens=TOKENS, stop_on_eos=True, max_batch_per_gpu=8)
    finally:
        pool.close()
    pool = built_lib.Pool("0.6B", devices=(0, 0), seed=SEED, config=cfg, continuous=True)
    try:
        got, lp = pool.transcribe_ids(clips, max_tokens=TOKENS, stop_on_eos=True, max_batch_per_gpu=8, return_logprobs=True)
        job = pool.submit(clips, max_tokens=TOKENS, stop_on_eos=True, max_batch_per_gpu=8)
        j_got = job.wait()
        for g in (got, j_got):
            assert [t.tolist() for t in g] == [t.tolist() for t in want]
        with pytest.raises(built_lib.Q3Error) as e:
            pool.transcribe_ids(clips[:4], max_tokens=8, options=built_lib.Qwen3DecodingOptions(temperature=0.7))
        assert e.value.code == INVALID
    finally:
        pool.close()


def _wav(path, x, rate):
    pcm = np.clip(np.round(x * 32767.0), -32768, 32767).astype("<i2")
    hdr = struct.pack("<4sI4s4sIHHIIHH4sI", b"RIFF", 36 + pcm.nbytes, b"WAVE", b"fmt ", 16, 1, 1, rate, 2 * rate, 2, 16, b"data", pcm.nbytes)
    path.write_bytes(hdr + pcm.tobytes())


def test_transcribe_batch_continuous(tmp_path):
    exe = os.path.join(PKG, "build", "transcribe_batch_cont")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-o", exe, os.path.join(PKG, "host", "transcribe_batch.cpp"),
                    "-L" + os.path.join(PKG, "lib"), "-lq3asr", "-Wl,-rpath," + os.path.join(PKG, "lib")], check=True)
    for i in range(9):
        _wav(tmp_path / f"f{i}.wav", synth.clip(70 + i, 16000 + 6000 * i), 16000)
    out = []
    for extra in ([], ["--continuous"]):
        r = subprocess.run([exe, str(tmp_path), "--jsonl", "--confidence", "--batch", "4", "--max-tokens", "10", "--devices", "0",
                            "--workers-per-gpu", "1"] + extra, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout + r.stderr
        recs = [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]
        out.append([{k: v for k, v in rec.items() if k not in ("time", "rtf")} for rec in recs])
    assert len(out[0]) == 9 and out[0] == out[1]
