"""The decode-step attention kernels (csrc/ops.cu) against a float64 paged-KV reference, through q3asr_debug_decode_attention.

Every variant the decode step can run is built from the same inputs (the fp32 split-K partials of the QKV product, the q/k norm
weights, the cache lengths, a page table and the paged pool) and checked element by element:

    0         the decode step's own choice for the batch size and SM count
    1, 2, 8   decode_attn_mma_kernel: the split variant (two single-warp CTAs per item), 2 warps, 8 warps
    4, 16     decode_attn_fused_kernel<2, 4> / <2, 16>, the SIMT kernels
    -1        the general path: qknorm_rope_kv_kernel + decode_attn_kernel<G> (above 256 decode rows, and under Q3ASR_NO_SKINNY)

Memory.  A sequence's pages are a random, non-monotonic choice of pool pages; the page-table entries past its last page name a page
that holds nothing but bf16 NaN, and so does every other byte a kernel must not read: the pages no sequence references, the rows
past the new token in a sequence's last page, and the new token's own slot before the call.  A kernel that reads a wrong page, row,
layer or head, or misses the patch of the new token's row into its prefetched last chunk, produces NaN or a wrong value, not a fault.

Reference.
  1. v = bf16(the fp32 sum of the partials in split order 0, 1, 2, ...): the kernels' rounding point, bit for bit.
  2. q, k: per-head RMSNorm rounded to bf16, then split-half RoPE, whose angle is the fp32 product pos * inv_freq
     (oracle/model.py _rope) with cos / sin in float64, rounded to bf16.
  3. softmax(q K^T * scale) V in float64 over the keys and values read back from the returned pool.

Tolerances.
  * The appended v row is bit-exact, and every other uint16 of the pool is unchanged (NaN poison, other layers, other heads).
  * q and k: the kernels compute the norm in fp32 with rsqrtf, so a normalised element n_i may round to the bf16 neighbour of the
    reference's (one ulp).  The rotation moves such a difference into both elements of its pair, and the result is rounded again:
    |k_kernel_i - k_ref_i| <= ulp(k_ref_i) + ulp(n_i)|cos_i| + ulp(n_partner)|sin_i|  (the same allowance a_i for q).
  * Output, element-wise: |got - ref| <= 2^-8 mag + 2^-8 |ref| + 2 delta mag + 1e-4, with mag = sum_j p_j |v_j| / sum_j p_j.
      - the kernels round every p_j to bf16 (2^-9 relative) before the PV product but not in the denominator: at most
        2^-9 mag each way, 2^-8 mag with room for the fp32 accumulation;
      - the output is rounded to bf16: 2^-9 |ref|, taken as 2^-8;
      - the kernel's q may differ from the reference's by a_i per element, so every score moves by at most
        delta = scale * max_j sum_i a_i |k_ji|; a score shift that lies in [-delta, delta] moves the softmax average of v by at
        most (max shift - min shift) * mag <= 2 delta mag (first order);
      - 1e-4 absolute for the fp32 sums.
  * Relative RMS error over the batch <= 4e-3.
Random keys give a near-uniform softmax, in which one wrong key hides in these bounds; the sensitivity cases (spike, dominant new
token, ramps, kv_len 1) make single keys decide the output.

Bit identity: the tensor-core variants (0, 1, 2, 8) share one key partition (8 canonical streams merged in a fixed tree), so they
agree bit for bit with each other, with the same sequence at another row of a batch of 1, 40 or 200 on other physical pages
(DESIGN.md section 2: batch invariance), and from one launch to the next on the same buffers.  The SIMT kernels and the general path
partition the keys differently and are held to the reference tolerance only (and to launch-to-launch identity).
"""
import numpy as np
import pytest

HD = 128
PAGE = 32
NAN_BITS = 0x7FC0
EPS = 1e-6
SCALE = 1.0 / np.sqrt(HD)
THETA = 1000000.0  # dec_rope_theta of every preset (the hook takes the loaded model's frequencies)
VARIANTS = (0, 1, 2, 8, 4, 16, -1)
MMA = (0, 1, 2, 8)

SHORT = [1, 2, 15, 16, 17, 31, 32, 33, 127, 128, 129, 255, 256, 257, 1000]
LONG = [2047, 2048, 4097, 1, 33]
ALL = [1, 2, 15, 16, 17, 31, 32, 33, 127, 128, 129, 255, 256, 257, 1000, 2047, 2048, 4097]


# ---- float64 reference ----------------------------------------------------------------------------------------------------------
def _bf16(x):
    """float64 -> the nearest-even bf16 value (as float64), exactly: no double rounding through float32."""
    m, e = np.frexp(np.asarray(x, dtype=np.float64))
    return np.ldexp(np.rint(np.ldexp(m, 8)), e - 8)


def _ulp(x):
    """One bf16 ulp at |x| (x holding bf16 values)."""
    _, e = np.frexp(np.abs(np.asarray(x, dtype=np.float64)))
    return np.where(x == 0, 2.0 ** -133, np.ldexp(1.0, e - 8))


def _bits(x):
    """bf16 values -> uint16 bits."""
    return (np.asarray(x, dtype=np.float32).view(np.uint32) >> 16).astype(np.uint16)


def _val(b):
    """uint16 bf16 bits -> float64 values."""
    return (np.asarray(b, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def _rand_bits(rng, shape, scale=1.0):
    x = rng.standard_normal(shape, dtype=np.float32) * np.float32(scale)
    u = x.view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def _inv_freq():
    return np.power(THETA, -np.arange(HD // 2, dtype=np.float64) * 2.0 / HD).astype(np.float32)


def _rmsnorm(x, w, eps=EPS):
    """Per-head RMSNorm over the last axis (x: bf16 values), rounded to bf16."""
    x = np.asarray(x, dtype=np.float64)
    return _bf16(x / np.sqrt((x * x).mean(axis=-1, keepdims=True) + eps) * np.asarray(w, dtype=np.float64))


def _cos_sin(pos):
    ang = (np.asarray(pos, dtype=np.float32)[:, None] * _inv_freq()[None, :]).astype(np.float32)  # the fp32 product
    return np.cos(ang.astype(np.float64))[:, None, :], np.sin(ang.astype(np.float64))[:, None, :]


def _rope(x, pos):
    """Split-half RoPE of x [n, heads, 128] (bf16 values) at positions pos [n], rounded to bf16."""
    c, s = _cos_sin(pos)
    a, b = x[..., :HD // 2], x[..., HD // 2:]
    return _bf16(np.concatenate([a * c - b * s, b * c + a * s], axis=-1))


def _rope_allowance(n, out, pos):
    """What a one-ulp difference of the normalised input n moves the rotated, rounded result by, plus its own rounding."""
    c, s = (np.abs(t) for t in _cos_sin(pos))
    ua, ub = _ulp(n[..., :HD // 2]), _ulp(n[..., HD // 2:])
    return _ulp(out) + np.concatenate([ua * c + ub * s, ub * c + ua * s], axis=-1)


def _new_token(inp):
    """q [n, heads, 128], k and v [n, kv_heads, 128] of the new tokens (bf16 values) and the allowances of q and k."""
    acc = np.zeros(inp.part.shape[1:], dtype=np.float32)
    for p in inp.part:  # split order 0, 1, 2, ... in fp32
        acc += p
    x = _bf16(acc.astype(np.float64)).reshape(len(inp.lens), inp.heads + 2 * inp.kvh, HD)
    pos = inp.lens - 1
    nq, nk = _rmsnorm(x[:, :inp.heads], inp.qw), _rmsnorm(x[:, inp.heads:inp.heads + inp.kvh], inp.kw)
    q, k = _rope(nq, pos), _rope(nk, pos)
    return q, k, x[:, inp.heads + inp.kvh:], _rope_allowance(nq, q, pos), _rope_allowance(nk, k, pos)


def _attend_one(q, K, V, q_allow):
    """q [heads, 128], K / V [kv_heads, S, 128] (float64) -> out, mag [heads, 128], delta [heads]."""
    heads, group = q.shape[0], q.shape[0] // K.shape[0]
    out, mag, delta = np.zeros_like(q), np.zeros_like(q), np.zeros(heads)
    for h in range(heads):
        Kh, Vh = K[h // group], V[h // group]
        s = Kh @ q[h] * SCALE
        p = np.exp(s - s.max())
        out[h] = p @ Vh / p.sum()
        mag[h] = p @ np.abs(Vh) / p.sum()
        delta[h] = SCALE * (np.abs(Kh) @ q_allow[h]).max()
    return out, mag, delta


def _attend(inp, pool, q, q_allow):
    """The reference attention of every sequence over the keys and values of the returned pool."""
    out, mag = np.zeros_like(q), np.zeros_like(q)
    delta = np.zeros(q.shape[:2])
    for s, L in enumerate(inp.lens):
        npg = -(-L // PAGE)
        kv = _val(pool[inp.pt[s, :npg], inp.layer])  # [pages, 2, kv_heads, 32, 128]
        kv = kv.transpose(1, 2, 0, 3, 4).reshape(2, inp.kvh, npg * PAGE, HD)[:, :, :L]
        out[s], mag[s], delta[s] = _attend_one(q[s], kv[0], kv[1], q_allow[s])
    return out, mag, delta


# ---- inputs -----------------------------------------------------------------------------------------------------------------------
class _Inputs:
    pass


def _build(rng, lens, heads, kvh, splits, layers=3, layer=1, n_nan=4):
    """Random partials and norm weights; random pages holding random keys / values for every cached position, NaN elsewhere."""
    inp = _Inputs()
    inp.lens = np.asarray(lens, dtype=np.int32)
    inp.heads, inp.kvh, inp.layers, inp.layer = heads, kvh, layers, layer
    n = len(lens)
    inp.part = (rng.standard_normal((splits, n, (heads + 2 * kvh) * HD), dtype=np.float32) / np.float32(np.sqrt(splits)))
    inp.qw = _bf16(1.0 + 0.25 * rng.standard_normal(HD)).astype(np.float32)
    inp.kw = _bf16(1.0 + 0.25 * rng.standard_normal(HD)).astype(np.float32)
    need = -(-inp.lens // PAGE)
    max_pages = int(need.max()) + 1  # every sequence has table entries past its last page
    perm = rng.permutation(int(need.sum()) + n_nan)
    nan_pages = perm[need.sum():]
    inp.pt = np.empty((n, max_pages), dtype=np.int32)
    inp.pool = np.full((perm.size, layers, 2, kvh, PAGE, HD), NAN_BITS, dtype=np.uint16)
    o = 0
    for s in range(n):
        pages = perm[o:o + need[s]]
        o += need[s]
        if pages.size > 1 and (np.diff(pages) > 0).all():
            pages = pages[::-1]
        inp.pt[s, :need[s]] = pages
        inp.pt[s, need[s]:] = rng.choice(nan_pages, max_pages - need[s])
        for i, pg in enumerate(pages):
            rows = min(PAGE, int(inp.lens[s]) - 1 - i * PAGE)  # the new token's slot and the rows past it stay NaN
            if rows > 0:
                inp.pool[pg, :, :, :, :rows] = _rand_bits(rng, (layers, 2, kvh, rows, HD))
    return inp


def _cached(inp, s):
    """(pages, rows) of the cached positions 0 .. kv_len - 2 of sequence s."""
    j = np.arange(int(inp.lens[s]) - 1)
    return inp.pt[s, j // PAGE], j % PAGE


def _product_splits(K):
    """gemm_skinny_splits of the decode step's QKV product (N = 4096 for both presets) on this GPU."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles_n, num_kb = 4096 // 128, K // 64
    per = -(-num_kb // min(num_kb, max(1, sms // tiles_n)))
    return -(-num_kb // per)


# ---- running and checking ---------------------------------------------------------------------------------------------------------
def _run(m, inp, variant, launches=2):
    out, pool = m.debug_decode_attention(inp.part, inp.heads, inp.kvh, inp.qw, inp.kw, inp.lens, inp.pt, inp.pool, inp.layer,
                                         variant=variant, launches=launches, eps=EPS, scale=SCALE)
    for i in range(1, launches):  # the append is idempotent and the split counters return to zero: every launch gives the same bits
        assert np.array_equal(out[i].view(np.uint32), out[0].view(np.uint32)), (variant, "launch", i)
    return out[0].reshape(len(inp.lens), inp.heads, HD), pool


def _check_append(inp, pool, k_ref, k_allow, v_ref, variant):
    n = len(inp.lens)
    pos = inp.lens - 1
    pg, row = inp.pt[np.arange(n), pos // PAGE], pos % PAGE
    got_k = _val(pool[pg, inp.layer, 0, :, row])
    err = np.abs(got_k - k_ref)
    assert (err <= k_allow).all(), (variant, "appended k", np.argwhere(err > k_allow)[:5].tolist())
    want = inp.pool.copy()
    want[pg, inp.layer, 1, :, row] = _bits(v_ref)
    want[pg, inp.layer, 0, :, row] = pool[pg, inp.layer, 0, :, row]
    bad = np.argwhere(want != pool)
    assert bad.size == 0, (variant, "pool bytes changed (or v row differs) at [page, layer, k/v, head, row, dim]", bad[:5].tolist())


def _check_out(got, ref, mag, delta, what):
    assert not np.isnan(got).any(), (what, "NaN at [seq, head, dim]", np.argwhere(np.isnan(got))[:5].tolist())
    err = np.abs(got - ref)
    tol = 2.0 ** -8 * mag + 2.0 ** -8 * np.abs(ref) + 2.0 * delta[..., None] * mag + 1e-4
    assert (err <= tol).all(), (what, float(err.max()), np.argwhere(err > tol)[:5].tolist())
    rel = np.sqrt((err ** 2).sum() / (ref ** 2).sum())
    assert rel <= 4e-3, (what, rel)


def _check_case(m, inp, exact=(), variants=VARIANTS):
    """All variants on one input set; exact: (seq, head, bf16 values) the output must equal bit for bit.  Returns the outputs."""
    q, k, v, q_allow, k_allow = _new_token(inp)
    exact = list(exact) + [(s, h, v[s, h // (inp.heads // inp.kvh)]) for s in np.flatnonzero(inp.lens == 1) for h in range(inp.heads)]
    refs, outs = {}, {}
    for var in variants:
        if var != -1 and inp.heads != 2 * inp.kvh:
            continue
        got, pool = _run(m, inp, var)
        _check_append(inp, pool, k, k_allow, v, var)
        key = pool[inp.pt[np.arange(len(inp.lens)), (inp.lens - 1) // PAGE], inp.layer, 0, :, (inp.lens - 1) % PAGE].tobytes()
        # the reference reads the appended k back (the rest of the pool is checked unchanged): recomputed only when k differs
        if key not in refs:
            refs.clear()
            refs[key] = _attend(inp, pool, q, q_allow)
        _check_out(got, *refs[key], f"variant {var}")
        for s, h, want in exact:
            assert np.array_equal(got[s, h], want), (var, "seq", s, "len", int(inp.lens[s]), "head", h, np.abs(got[s, h] - want).max())
        outs[var] = got
    for var in MMA[1:]:
        if var in outs and 0 in outs:
            assert np.array_equal(outs[var].view(np.uint32), outs[0].view(np.uint32)), ("variant", var, "differs from variant 0")
    return outs


# ---- random inputs at every length, layout and split count -----------------------------------------------------------------------
RANDOM = [  # id, heads, kv_heads, lengths, splits ("qkv0.6B" / "qkv1.7B": the decode step's own count), layer
    ("16x8-short-qkv0.6B", 16, 8, SHORT, "qkv0.6B", 1),
    ("16x8-long-s8", 16, 8, LONG, 8, 1),
    ("16x8-short-s3-layer2", 16, 8, SHORT, 3, 2),
    ("16x8-long-qkv1.7B", 16, 8, LONG, "qkv1.7B", 1),
    ("4x2-all-s1", 4, 2, ALL, 1, 1),
    ("4x2-all-s3", 4, 2, ALL, 3, 1),
    ("8x8-short-s3-general", 8, 8, SHORT, 3, 1),  # one query head per kv head: the general path only
]


@pytest.mark.gpu
@pytest.mark.parametrize("heads,kvh,lens,splits,layer", [c[1:] for c in RANDOM], ids=[c[0] for c in RANDOM])
def test_decode_attention_matches_reference(tiny_model, heads, kvh, lens, splits, layer):
    if isinstance(splits, str):
        splits = _product_splits(1024 if splits == "qkv0.6B" else 2048)
    rng = np.random.default_rng(heads * 7919 + kvh * 31 + len(lens) * 7 + splits + layer)
    _check_case(tiny_model, _build(rng, lens, heads, kvh, splits, layer=layer))


# ---- sensitivity: single keys decide the output -----------------------------------------------------------------------------------
def _spike_rows(lens):
    rows = []
    for L in lens:
        for p in sorted({0, 15, 16, 31, 32, 33, L - 2}):
            if p <= L - 2:
                rows.append((L, p))
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("heads,kvh,lens", [(4, 2, [34, 257, 2048]), (16, 8, [40, 300])], ids=["4x2", "16x8"])
def test_spike_key_decides_the_output(tiny_model, heads, kvh, lens):
    """At cached position p (0, 15, 16, 31, 32, 33, kv_len - 2: chunk and page edges, the first and the last cached key) every kv
    head holds c * q_ref of one of its query heads, about 40 nats above the other keys, which are scaled down, with a distinctive v:
    that query head's output is that v, bit for bit.  A key read from a wrong page or row, or masked away, changes it."""
    rng = np.random.default_rng(101 + heads)
    rows = _spike_rows(lens)
    inp = _build(rng, [L for L, _ in rows], heads, kvh, 4)
    q = _new_token(inp)[0]
    group = heads // kvh
    exact = []
    for s, (L, p) in enumerate(rows):
        pages, rr = _cached(inp, s)
        inp.pool[pages, inp.layer, 0, :, rr] = _bits(_val(inp.pool[pages, inp.layer, 0, :, rr]) / 8)  # exact in bf16
        for g in range(kvh):
            h = g * group + (s + g) % group
            c = 40.0 / (SCALE * (q[s, h] @ q[s, h]))
            vs = _bf16(8.0 + rng.standard_normal(HD))
            inp.pool[pages[p], inp.layer, 0, g, rr[p]] = _bits(_bf16(c * q[s, h]))
            inp.pool[pages[p], inp.layer, 1, g, rr[p]] = _bits(vs)
            exact.append((s, h, vs))
    _check_case(tiny_model, inp, exact)


@pytest.mark.gpu
@pytest.mark.parametrize("heads,kvh,lens", [(16, 8, SHORT), (4, 2, ALL)], ids=["16x8", "4x2"])
def test_dominant_new_token(tiny_model, heads, kvh, lens):
    """The k partials equal the q partials of one query head per kv head and q_norm = k_norm = 3, so that head's score against the
    new key is about 100 nats, and the cached keys are small: its output is v_new bit for bit.  The new token's slot is NaN before
    the call, so a kernel that attends over its prefetched copy of that row without patching the new k / v in returns NaN."""
    rng = np.random.default_rng(202 + heads)
    inp = _build(rng, lens, heads, kvh, 4)
    group = heads // kvh
    for g in range(kvh):
        kc, qc = (heads + g) * HD, g * group * HD
        inp.part[:, :, kc:kc + HD] = inp.part[:, :, qc:qc + HD]
    inp.qw = np.full(HD, 3.0, dtype=np.float32)
    inp.kw = inp.qw.copy()
    for s in range(len(lens)):
        pages, rr = _cached(inp, s)
        inp.pool[pages, inp.layer, 0, :, rr] = _bits(_val(inp.pool[pages, inp.layer, 0, :, rr]) / 64)
    v = _new_token(inp)[2]
    _check_case(tiny_model, inp, [(s, g * group, v[s, g]) for s in range(len(lens)) for g in range(kvh)])


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["up", "down"])
@pytest.mark.parametrize("heads,kvh,lens", [(4, 2, [1000, 1500, 2048, 4097]), (16, 8, [1000, 2048])], ids=["4x2", "16x8"])
def test_score_ramps(tiny_model, heads, kvh, lens, direction):
    """Cached keys a_j u, u along q_ref of one query head per kv head.  up: the scores climb 60 nats over the context, so the running
    maximum moves with every chunk and every earlier partial is rescaled; down: they fall 120 nats, so the exponentials of the later
    chunks and of whole streams underflow to zero in the merges."""
    rng = np.random.default_rng(303 + heads + len(direction))
    inp = _build(rng, lens, heads, kvh, 4)
    q = _new_token(inp)[0]
    group = heads // kvh
    for s, L in enumerate(lens):
        pages, rr = _cached(inp, s)
        t = np.linspace(0.0, 1.0, L - 1)
        nats = -30.0 + 60.0 * t if direction == "up" else 60.0 - 120.0 * t
        for g in range(kvh):
            qh = q[s, g * group]
            inp.pool[pages, inp.layer, 0, g, rr] = _bits(_bf16((nats / (SCALE * (qh @ qh)))[:, None] * qh[None, :]))
    _check_case(tiny_model, inp)


# ---- batch and page invariance ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_batch_row_and_page_invariance(tiny_model):
    """The same three sequences (2048, 257 and 33 keys) decoded alone, then at other rows of batches of 40 and 200 on other physical
    pages (so variant 0 switches from 8 to 2 warps): every tensor-core variant returns the same bits everywhere."""
    rng = np.random.default_rng(404)
    heads, kvh, layers, splits = 16, 8, 3, 4
    targets = [2048, 257, 33]
    t_in = _build(rng, targets, heads, kvh, splits, layers=layers)
    t_pages = [t_in.pool[t_in.pt[i, :-(-L // PAGE)]] for i, L in enumerate(targets)]
    want = {}
    for B in (1, 40, 200):
        placements = [[i] for i in range(len(targets))] if B == 1 else [list(rng.choice(B, len(targets), replace=False))]
        for rows in placements:
            if B == 1:
                lens = [targets[rows[0]]]
                where = {0: rows[0]}
            else:
                lens = list(rng.integers(1, PAGE + 1, size=B))
                where = {}
                for i, r in enumerate(rows):
                    lens[r] = targets[i]
                    where[int(r)] = i
            inp = _build(rng, lens, heads, kvh, splits, layers=layers)
            inp.qw, inp.kw = t_in.qw, t_in.kw
            for r, i in where.items():
                inp.part[:, r] = t_in.part[:, i]
                inp.pool[inp.pt[r, :t_pages[i].shape[0]]] = t_pages[i]
            if B == 1:
                outs = _check_case(tiny_model, inp, variants=MMA)
            else:
                outs = {var: _run(tiny_model, inp, var)[0] for var in MMA}
            for var, got in outs.items():
                for r, i in where.items():
                    bits = got[r].view(np.uint32).copy()
                    if i not in want:
                        want[i] = bits
                    assert np.array_equal(bits, want[i]), ("batch", B, "row", r, "variant", var, "sequence", targets[i])
    assert len(want) == len(targets)


# ---- the hook's argument checks ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_debug_hook_rejects_bad_arguments(built_lib, tiny_model):
    rng = np.random.default_rng(505)
    inp = _build(rng, [40, 3], 4, 2, 2)

    def call(m=tiny_model, **kw):
        args = dict(qkv_part=inp.part, heads=4, kv_heads=2, q_norm=inp.qw, k_norm=inp.kw, kv_len=inp.lens, page_table=inp.pt,
                    pool=inp.pool, layer=1, variant=0)
        args.update(kw)
        return m.debug_decode_attention(**args)

    bad_pt = inp.pt.copy()
    bad_pt[1, -1] = inp.pool.shape[0]
    for kw in (dict(page_table=bad_pt), dict(kv_len=np.array([40, 0])), dict(kv_len=np.array([40, 3 * PAGE + 1])), dict(variant=3),
               dict(layer=3), dict(launches=0)):
        with pytest.raises(built_lib.Q3Error) as e:
            call(**kw)
        assert e.value.code == 1, kw
    q8 = rng.standard_normal((2, 2, (8 + 2 * 2) * HD)).astype(np.float32)
    with pytest.raises(built_lib.Q3Error) as e:  # the fused kernels are built for two query heads per kv head
        call(qkv_part=q8, heads=8)
    assert e.value.code == 1
    empty = built_lib.Qwen3ASRModel("tiny")
    try:
        with pytest.raises(built_lib.Q3Error) as e:  # the RoPE frequencies come from a loaded model
            call(m=empty)
        assert e.value.code == 2
    finally:
        empty.close()
    out, pool = call()  # the handle still works
    assert not np.isnan(out).any()


# ---- the reference against the oracle (no GPU) ------------------------------------------------------------------------------------
def test_reference_helpers_match_the_oracle(tiny_oracle):
    """_rmsnorm / _rope / _attend_one against oracle.model.Oracle's _rmsnorm / _rope / _attention (bf16-rounding float32 and float64
    code) on a small case, so that the reference the kernels are held to is itself pinned."""
    import torch
    rng = np.random.default_rng(606)
    heads, kvh, n = 4, 2, 5
    pos = np.array([0, 1, 31, 1000, 4096])
    x = _bf16(rng.standard_normal((n, heads, HD)) * 3)
    w = _bf16(1 + 0.25 * rng.standard_normal(HD))
    o = tiny_oracle
    mine = _rmsnorm(x, w)
    theirs = o._rmsnorm(torch.from_numpy(x.astype(np.float32)), torch.from_numpy(w.astype(np.float32)), EPS).double().numpy()
    assert (np.abs(mine - theirs) <= _ulp(mine)).all() and (mine == theirs).mean() > 0.99
    mine_r = _rope(mine, pos)
    theirs_r = o._rope(torch.from_numpy(mine.reshape(n, heads * HD).astype(np.float32)), pos, heads).double().numpy().reshape(n, heads, HD)
    allow = _rope_allowance(mine, mine_r, pos)
    assert (np.abs(mine_r - theirs_r) <= allow).all() and (mine_r == theirs_r).mean() > 0.99
    assert np.array_equal(mine_r[0], mine[0])  # position 0 is the identity
    S = 300
    K = _bf16(rng.standard_normal((kvh, S, HD)))
    V = _bf16(rng.standard_normal((kvh, S, HD)))
    q = mine_r[3]
    out, mag, _ = _attend_one(q, K, V, np.zeros_like(q))
    kt = torch.from_numpy(K.transpose(1, 0, 2).reshape(S, kvh * HD).astype(np.float32))
    vt = torch.from_numpy(V.transpose(1, 0, 2).reshape(S, kvh * HD).astype(np.float32))
    qt = torch.from_numpy(q.reshape(1, heads * HD).astype(np.float32))
    theirs_a = o._attention(qt, kt, vt, heads, kvh, float(SCALE), False, fp64=True).double().numpy().reshape(heads, HD)
    assert (np.abs(out - theirs_a) <= 2.0 ** -8 * mag + 2.0 ** -8 * np.abs(out) + 1e-6).all()
    # and the exact bf16 rounding agrees with the project's float32 one
    y = rng.standard_normal(10000).astype(np.float32)
    from oracle.weights import bf16_round
    assert np.array_equal(_bf16(y.astype(np.float64)), bf16_round(y).astype(np.float64))
