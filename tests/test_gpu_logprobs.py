"""Per-token log-probabilities (q3asr_transcribe_ids_lp and friends, definition in include/q3asr.h):
logprob = z[t] - logsumexp(z) over the bf16-rounded logits, the log-sum-exp reduced in the LM head's epilogue on the device.

Checked:
  1. the kernels alone (q3asr_debug_gemm 8 = LM-head kernel, 9 = general GEMM EPI_ARGMAX) on operands whose logits are exact
     integers on both sides: ids equal the host's first maximum, log-probabilities within 2e-5 of float64 log_softmax;
  2. the tiny model against the live oracle (free-running greedy, and the decoder knobs against generate_slow's RAW logits);
  3. every LM-head path agrees (fused, Q3ASR_LM_GENERAL, device sampler with greedy options, Q3ASR_NO_SKINNY); the persistent step
     (Q3ASR_MEGA) is bit-identical to the multi-kernel step;
  4. asking for log-probabilities changes no id, length or teacher-forced logit;
  5. batch invariance, bit for bit: request sizes, 0.6B at 64 x 30 s, compaction with ragged EOS;
  6. 0.6B self-consistency against the float64 log-softmax of the prefill logits;
  7. the pool (blocking, submit / wait) and the transcribe_batch --confidence front end.
The oracle is used unchanged: a subclass records the float64 log_softmax of every step's bf16-emulated logits.
"""
import collections
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import mel as omel
from oracle import model as omodel
from oracle import synth, weights

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "qwen3-asr-swift_b200")


class LpOracle(omodel.Oracle):
    """The oracle, recording log_softmax (float64) of the logits of every prefill / decode step it computes."""

    def _logits(self, last):
        z = super()._logits(last)
        self.lsm.append(torch.log_softmax(z.double(), dim=-1).numpy())
        self.zmax.append(float(z.max()))
        return z

    def greedy_lp(self, emb, max_tokens):
        self.lsm, self.zmax = [], []
        ids, tops, margins = self.greedy(emb, max_tokens, stop_on_eos=False)
        return ids, np.array([self.lsm[s][t] for s, t in enumerate(ids)]), tops, margins

    def slow_lp(self, emb, max_tokens, **kw):
        self.lsm, self.zmax = [], []
        ids, margins, _ = self.generate_slow(emb, max_tokens, stop_on_eos=False, **kw)
        return ids, np.array([self.lsm[s][t] for s, t in enumerate(ids)]), margins, np.array(self.zmax[:len(ids)])


@pytest.fixture(scope="module")
def lp_oracle():
    cfg = weights.preset("tiny")
    return LpOracle(cfg, weights.random_state_dict(cfg, 20260418))


def _ulp(x):
    return np.exp2(np.floor(np.log2(np.maximum(np.abs(np.asarray(x, dtype=np.float64)), 2.0 ** -6))) - 7)


# ---- 1. kernel exactness ---------------------------------------------------------------------------------------------------------
def _exact_weights(N, K, seed):
    """W [N, K] with 4 distinct nonzero columns per row, values in [-4, 4], as bf16 bit patterns, plus (columns, values)."""
    rng = np.random.default_rng(seed)
    cols = np.argsort(rng.random((N, 16)), axis=1)[:, :4] * (K // 16) + rng.integers(0, K // 16, size=(N, 1))
    vals = rng.integers(-4, 5, size=(N, 4)).astype(np.float32)
    W = np.zeros((N, K), dtype=np.uint16)
    W[np.repeat(np.arange(N), 4), cols.reshape(-1)] = (vals.view(np.uint32) >> 16).astype(np.uint16).reshape(-1)
    return W, cols, vals


def _exact_logits(A, cols, vals):
    """A [M, K] integers in [-8, 8]: every logit is an integer of magnitude <= 128, exact in fp32 and bf16 whatever the summation
    order; returned in float64"""
    z = np.zeros((A.shape[0], cols.shape[0]), dtype=np.float64)
    for j in range(4):
        z += A[:, cols[:, j]].astype(np.float64) * vals[:, j][None, :]
    return z


def _debug_lp(lib, h, a_bits, w_bits, M, N, K, epi):
    out = np.zeros(2 * M, dtype=np.int32)
    rc = lib.lib().q3asr_debug_gemm(h, a_bits.ctypes.data, w_bits.ctypes.data, None, None, M, N, K, epi, 0, 0, 0, out.ctypes.data)
    assert rc == 0, lib.lib().q3asr_last_error(h)
    return out[:M].copy(), out[M:].view(np.float32).copy()


@pytest.mark.parametrize("N,K", [(151936, 1024), (151936, 2048), (2048, 1024), (2048, 2048), (1000, 1024), (1000, 2048)])
def test_kernel_logprobs_exact(built_lib, tiny_model, N, K):
    W, cols, vals = _exact_weights(N, K, seed=N + K)
    rng = np.random.default_rng(K)
    for M in (1, 7, 16, 64, 129, 256):
        A = rng.integers(-8, 9, size=(M, K)).astype(np.float32)
        a = (A.view(np.uint32) >> 16).astype(np.uint16)
        z = _exact_logits(A, cols, vals)
        want_ids = z.argmax(axis=1)  # numpy: first maximum
        mx = z.max(axis=1, keepdims=True)
        want_lp = (z - mx - np.log(np.exp(z - mx).sum(axis=1, keepdims=True)))[np.arange(M), want_ids]
        for epi in ((8, 9) if N % 32 == 0 else (8,)):  # the general GEMM takes whole tiles only
            ids, lp = _debug_lp(built_lib, tiny_model._h, a, W, M, N, K, epi)
            assert (ids == want_ids).all(), (epi, M, N, K, np.nonzero(ids != want_ids)[0][:8])
            err = np.abs(lp.astype(np.float64) - want_lp)
            assert err.max() <= 2e-5, (epi, M, N, K, float(err.max()))


# ---- 2. tiny model against the oracle ----------------------------------------------------------------------------------------------
def test_free_running_logprobs_match_oracle(tiny_model, lp_oracle):
    for seed, n in [(0, 16000 * 2 + 123), (1, 40000)]:
        x = synth.clip(seed, n)
        emb = lp_oracle.encode(omel.mel(x))
        ref_ids, ref_lp, ref_top, _ = lp_oracle.greedy_lp(emb, 16)
        ids, lp = tiny_model.transcribe_ids([x], max_tokens=16, stop_on_eos=False, return_logprobs=True)
        same = int(np.argmin(np.append(ids[0] == ref_ids, False)))  # common prefix (ids are bit-exact: all 16 in practice)
        assert same >= 8, (ids[0].tolist(), ref_ids.tolist())
        err = np.abs(lp[0][:same].astype(np.float64) - ref_lp[:same])
        assert (err <= 8 * _ulp(ref_top[:same])).all(), (seed, err.tolist())
        assert np.isfinite(lp[0]).all() and (lp[0] <= 0).all()


def test_decoder_knob_logprobs_are_raw_model_logprobs(built_lib, tiny_model, lp_oracle):
    """Penalty + n-gram mask at temperature 0: the log-probability is the one of the UNMODIFIED logits (Whisper's convention)."""
    x = synth.clip(3, 16000 * 3)
    emb = lp_oracle.encode(omel.mel(x))
    ref_ids, ref_lp, margins, ref_top = lp_oracle.slow_lp(emb, 16, repetition_penalty=1.3, no_repeat_ngram_size=2)
    opts = built_lib.Qwen3DecodingOptions(repetition_penalty=1.3, no_repeat_ngram_size=2)
    ids, lp = tiny_model.transcribe_ids([x], max_tokens=16, stop_on_eos=False, options=opts, return_logprobs=True)
    ids, lp = ids[0], lp[0].astype(np.float64)
    checked = 0
    for s in range(len(ref_ids)):  # up to the first step whose choice is inside the bf16 noise
        if ids[s] != ref_ids[s] or margins[s] <= 8 * _ulp(ref_top[s]):
            break
        assert abs(lp[s] - ref_lp[s]) <= 8 * _ulp(ref_top[s]), (s, lp[s], ref_lp[s])
        checked += 1
    assert checked >= 4, checked
    plain_ids, plain_lp = tiny_model.transcribe_ids([x], max_tokens=16, stop_on_eos=False, return_logprobs=True)
    assert plain_ids[0].tolist() != ids.tolist()  # the knobs really changed the run


# ---- 3. / 4. paths agree, nothing else changes ------------------------------------------------------------------------------------
PATHS = {"fused": {}, "general": {"Q3ASR_LM_GENERAL": "1"}, "no_skinny": {"Q3ASR_NO_SKINNY": "1"}, "sampler": None}


def _run(built_lib, m, monkeypatch, path, clips, tokens, lp, stop_on_eos=False):
    env = PATHS[path] or {}
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    try:
        opts = built_lib.Qwen3DecodingOptions() if path == "sampler" else None
        return m.transcribe_ids(clips, max_tokens=tokens, stop_on_eos=stop_on_eos, options=opts, force_device_sampler=path == "sampler",
                                return_logprobs=lp)
    finally:
        for k in env:
            monkeypatch.delenv(k)


def test_paths_agree_and_logprobs_change_nothing(built_lib, tiny_model, monkeypatch):
    clips = [synth.clip(20 + i, 16000 + 5000 * i) for i in range(5)]
    forced = np.random.default_rng(9).integers(0, 2000, size=12).astype(np.int32)
    f_ids0, f_top0 = tiny_model.decode_forced(clips[0], forced)
    runs = {}
    for path in PATHS:
        plain = _run(built_lib, tiny_model, monkeypatch, path, clips, 24, False)
        ids, lp = _run(built_lib, tiny_model, monkeypatch, path, clips, 24, True)
        assert [t.tolist() for t in ids] == [t.tolist() for t in plain], path  # 4: ids and lengths unchanged
        runs[path] = (ids, lp)
    f_ids1, f_top1 = tiny_model.decode_forced(clips[0], forced)
    assert np.array_equal(f_ids0, f_ids1) and np.array_equal(f_top0, f_top1)
    ref_ids, ref_lp = runs["fused"]
    for i, x in enumerate(clips):  # the top logit of every step, from teacher forcing on the run's own ids
        _, tops = tiny_model.decode_forced(x, ref_ids[i][:-1])
        for path, (ids, lp) in runs.items():
            # the LM-head variants see the same hidden states; the plain decoder layers (no_skinny) are another summation order of
            # the whole step, whose logits differ by a few bf16 ulps (tests/test_gpu_model.py test_decode_paths_agree)
            tol = (8 if path == "no_skinny" else 1) * _ulp(tops) + 1e-4
            assert ids[i].tolist() == ref_ids[i].tolist(), path
            err = np.abs(lp[i].astype(np.float64) - ref_lp[i])
            assert (err <= tol).all(), (path, i, err.max())


def test_megastep_logprobs_bit_identical(built_lib, monkeypatch):
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418)
    try:
        for B in (1, 40):
            clips = [synth.clip(300 + B + i, 16000 + 2400 * ((i * 7) % 11)) for i in range(B)]
            out = {}
            for mega in ("0", "1"):
                monkeypatch.setenv("Q3ASR_MEGA", mega)
                plain = m.transcribe_ids(clips, max_tokens=24, stop_on_eos=False)
                ids, lp = m.transcribe_ids(clips, max_tokens=24, stop_on_eos=False, return_logprobs=True)
                assert [t.tolist() for t in ids] == [t.tolist() for t in plain]
                out[mega] = (ids, lp)
            assert [t.tolist() for t in out["0"][0]] == [t.tolist() for t in out["1"][0]]
            for a, b in zip(out["0"][1], out["1"][1]):
                assert np.array_equal(a, b)
    finally:
        monkeypatch.delenv("Q3ASR_MEGA", raising=False)
        m.close()


# ---- 5. batch invariance ---------------------------------------------------------------------------------------------------------
def test_tiny_logprobs_do_not_depend_on_request_size(tiny_model):
    clips = [synth.clip(1000 + i, 8000 + 1600 * (i % 9)) for i in range(300)]
    ref_ids, ref_lp = tiny_model.transcribe_ids(clips, max_tokens=12, stop_on_eos=False, return_logprobs=True)
    for n in (1, 8, 20, 40, 70, 128, 140, 256):
        ids, lp = tiny_model.transcribe_ids(clips[:n], max_tokens=12, stop_on_eos=False, return_logprobs=True)
        for i in range(n):
            assert ids[i].tolist() == ref_ids[i].tolist(), (n, i)
            assert np.array_equal(lp[i], ref_lp[i]), (n, i, np.abs(lp[i] - ref_lp[i]).max())


def test_full_size_logprobs_batch_invariant_and_self_consistent(built_lib):
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418)
    try:
        clips = [synth.clip(500 + i, 16000 * 30) for i in range(64)]
        one_ids, one_lp = m.transcribe_ids(clips[:1], max_tokens=32, stop_on_eos=False, return_logprobs=True)
        ids, lp = m.transcribe_ids(clips, max_tokens=32, stop_on_eos=False, return_logprobs=True)
        assert ids[0].tolist() == one_ids[0].tolist() and np.array_equal(lp[0], one_lp[0])
        for t in lp:
            assert np.isfinite(t).all() and (t <= 0).all()
        # 6. step 0 against the float64 log-softmax of the prefill logits, rounded to bf16 like the LM head rounds them
        z = torch.from_numpy(m.prefill_logits(clips[0])).to(torch.bfloat16).double()
        t0 = int(ids[0][0])
        want = float(torch.log_softmax(z, dim=-1)[t0])
        assert t0 == int(torch.argmax(z)) or z[t0] == z.max()
        assert abs(float(lp[0][0]) - want) <= _ulp(float(z[t0])) + 1e-4, (float(lp[0][0]), want)
    finally:
        m.close()


def test_compaction_logprobs_are_prefixes(built_lib):
    n, tokens = 40, 80
    clips = [synth.clip(700 + i, 16000 * 2 + 3200 * (i % 7)) for i in range(n)]
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418)
    try:
        free_ids, free_lp = m.transcribe_ids(clips, max_tokens=tokens, stop_on_eos=False, return_logprobs=True)
    finally:
        m.close()
    free = [t.tolist() for t in free_ids]
    firsts = collections.defaultdict(list)
    for ids in free:
        seen = set()
        for s, t in enumerate(ids):
            if t not in seen:
                seen.add(t)
                firsts[t].append(s)
    eos = max(firsts, key=lambda t: (len(firsts[t]) >= n // 2) * (np.std(firsts[t]) + 0.01 * len(firsts[t])))
    cfg = built_lib.preset("0.6B")
    cfg.tok_eos = int(eos)
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418, config=cfg)
    try:
        ids, lp = m.transcribe_ids(clips, max_tokens=tokens, stop_on_eos=True, return_logprobs=True)
        assert m.decode_stats()["compactions"] >= 1
    finally:
        m.close()
    for i in range(n):
        L = free[i].index(eos) + 1 if eos in free[i] else tokens
        assert ids[i].tolist() == free[i][:L]
        assert np.array_equal(lp[i], free_lp[i][:L]), (i, L)


# ---- 7. front ends ---------------------------------------------------------------------------------------------------------------
def test_pool_logprobs_match_single_handle(built_lib, tiny_model):
    clips = [synth.clip(40 + i, 16000 + 900 * i) for i in range(7)]
    want_ids, want_lp = tiny_model.transcribe_ids(clips, max_tokens=10, stop_on_eos=True, return_logprobs=True)
    pool = built_lib.Pool("tiny", devices=(0, 0), seed=20260418)
    try:
        ids, lp = pool.transcribe_ids(clips, max_tokens=10, stop_on_eos=True, max_batch_per_gpu=3, return_logprobs=True)
        job = pool.submit(clips, max_tokens=10, stop_on_eos=True, max_batch_per_gpu=2, return_logprobs=True)
        j_ids, j_lp = job.wait()
        for got_ids, got_lp in ((ids, lp), (j_ids, j_lp)):
            assert [t.tolist() for t in got_ids] == [t.tolist() for t in want_ids]
            for a, b in zip(got_lp, want_lp):
                assert np.array_equal(a, b)
        # a job submitted without log-probabilities refuses to give them
        L = built_lib.lib()
        cl = [np.ascontiguousarray(c, dtype=np.float32) for c in clips[:2]]
        nn = np.array([c.size for c in cl], dtype=np.uint64)
        arr = (ctypes.c_void_p * 2)(*[c.ctypes.data for c in cl])
        j = ctypes.c_void_p()
        assert L.q3asr_pool_submit(pool._p, ctypes.cast(arr, ctypes.c_void_p), nn.ctypes.data, None, 2, None, None, 6, 1, 0,
                                   ctypes.byref(j)) == 0
        ids_buf = np.zeros((2, 6), np.int32)
        lens_buf = np.zeros(2, np.int32)
        out = np.zeros((2, 6), np.float32)
        assert L.q3asr_job_wait(j, ids_buf.ctypes.data, lens_buf.ctypes.data) == 0
        assert L.q3asr_job_logprobs(j, out.ctypes.data) == 1  # Q3ASR_ERR_INVALID
        L.q3asr_job_free(j)
    finally:
        pool.close()


def test_resident_batch_logprobs(built_lib, tiny_model):
    clips = [synth.clip(60 + i, 20000 + 3000 * i) for i in range(3)]
    want_ids, want_lp = tiny_model.transcribe_ids(clips, max_tokens=9, stop_on_eos=False, return_logprobs=True)
    tiny_model.batch_upload(clips)
    with pytest.raises(built_lib.Q3Error):  # not requested for this batch
        tiny_model.batch_download_logprobs(3, 9)
    tiny_model.batch_set_logprobs(True)
    tiny_model.batch_run(max_tokens=9)
    ids = tiny_model.batch_download(3, 9)
    lp = tiny_model.batch_download_logprobs(3, 9)
    with pytest.raises(built_lib.Q3Error):  # too late: the first token has been chosen
        tiny_model.batch_set_logprobs(False)
    for i in range(3):
        assert ids[i].tolist() == want_ids[i].tolist() and np.array_equal(lp[i], want_lp[i])


def test_transcribe_batch_confidence(built_lib, tmp_path):
    import struct
    exe = os.path.join(PKG, "build", "transcribe_batch_lp")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-o", exe, os.path.join(PKG, "host", "transcribe_batch.cpp"),
                    "-L" + os.path.join(PKG, "lib"), "-lq3asr", "-Wl,-rpath," + os.path.join(PKG, "lib")], check=True)
    x = synth.clip(0, 16000 * 2)
    pcm = np.clip(np.round(x * 32767.0), -32768, 32767).astype("<i2")
    hdr = struct.pack("<4sI4s4sIHHIIHH4sI", b"RIFF", 36 + pcm.nbytes, b"WAVE", b"fmt ", 16, 1, 1, 16000, 32000, 2, 16, b"data", pcm.nbytes)
    (tmp_path / "a.wav").write_bytes(hdr + pcm.tobytes())
    r = subprocess.run([exe, str(tmp_path), "--jsonl", "--confidence", "--max-tokens", "6", "--devices", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    recs = [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]
    assert len(recs) == 1 and "avg_logprob" in recs[0]
    samples = built_lib.AudioFileLoader.load_wav(str(tmp_path / "a.wav"))[0]
    m = built_lib.Qwen3ASRModel.random_init("0.6B", seed=20260418)  # the weights the command uses without --model-dir
    try:
        _, lp = m.transcribe_ids([samples], max_tokens=6, stop_on_eos=True, return_logprobs=True)
    finally:
        m.close()
    assert abs(recs[0]["avg_logprob"] - built_lib.avg_logprob(lp[0])) <= 1e-4, (recs[0]["avg_logprob"], built_lib.avg_logprob(lp[0]))
