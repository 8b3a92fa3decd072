"""The prefill's attention block (csrc/forward.cu prefill_attention) against a float64 reference on scrambled paged KV, through
q3asr_debug_prefill_attention, which runs the same host function as the prefill with the caller's buffers:

    q‖k‖v product  ->  EPI_QKV (gemm.cuh: per-head RMSNorm + split-half RoPE of q and k, k copied to a contiguous buffer, k and v
                       written into the paged cache, v left in the q‖k‖v buffer)
                       or, as its checker, the plain product + qknorm_rope_kv_kernel (ops.cu)
                   ->  causal attention: fa_tc_kernel<128, true, 2 or 1> (attention_tc.cu) or the mma.sync checker (attention.cu),
                       v read from inside the q‖k‖v buffer with leading dimension (heads + 2 kv_heads) * 128

Memory.  Each prompt's pages are a random, non-monotonic choice of pool pages, and its page-table row is not its index (rows 5, 0, 3
of a table of 8, say).  Table entries past a prompt's last page, the table rows no prompt uses and page 0 (where a row past the end
of the product would land if the epilogue's guards failed) name pages that hold bf16 NaN.  The layer under test is NaN everywhere
before the call, the other layers of the 3-layer pool are random: the call must write exactly the slots of the prompts' positions.

Exact-integer operands.  x holds integers in [-4, 4] times 2^e per row (e in -6 .. 3, some rows all zero), every row of w has at
most 31 non-zeros, integers in [-2, 2].  So every partial sum of a product element is an integer times 2^e with magnitude at most
31 * 4 * 2 = 248 times 2^e: exact in fp32 in any summation order, and bf16(acc) = acc.  The sum of squares over a head is at most
128 * 248^2 < 2^24 (times 2^2e): exact as well, in the sequential order of EPI_QKV and in the shuffle tree of qknorm_rope_kv_kernel.
Realistic operands (one case): x ~ N(0, 1), w ~ 0.08 N(0, 1) in bf16, the random-init decoder's scale.  There the fp32
accumulation of the tensor cores (exact products, each 16-deep MMA step added with alignment to the largest addend) is off the exact
sum by at most e = K 2^-23 sum_i |x_i w_i|, which matters where the sum cancels to near zero.

Reference.
  1. The product in float32 (exact operands: exact) or float64, rounded to bf16: v, and under the checker all of q‖k‖v.
  2. q, k: per-head RMSNorm in float64 rounded to bf16, then split-half RoPE at the fp32 angle pos * inv_freq with cos / sin in
     float64, rounded (the helpers of test_gpu_decode_attention.py, pinned there and below to oracle/model.py).
  3. The causal softmax(q k^T scale) v in float64 per prompt over the kernel's own returned q, k and v, so that the attention check
     does not depend on (2).

Tolerances.
  * v is bit-exact on exact operands.  On realistic ones bf16(acc) and bf16(exact) differ by at most ulp(v_ref) + 2e (one ulp while
    e < ulp / 2, and e + 1.5 ulp above).
  * Pool: every written slot holds the returned k / v row bit for bit, every other uint16 is unchanged.
  * q, k: the kernels compute the norm in fp32 with rsqrtf, so a normalised element n_i may round to the bf16 neighbour of the
    reference's (one ulp).  The rotation moves such a difference into both elements of its pair, and the result is rounded again:
    |q_kernel_i - q_ref_i| <= ulp(q_ref_i) + ulp(n_i)|cos_i| + ulp(n_partner)|sin_i|.  On realistic operands the product element
    itself may be off by its allowance above, which the norm scales into r |w_i| (ulp(x_i) + 2e_i) more on n_i, moved through the
    rotation the same way.
  * Attention, element-wise: |got - ref| <= 2^-8 mag + 2^-8 |ref| + 1e-4, mag = sum_j p_j |v_j| / sum_j p_j (the kernels round
    every p_j to bf16 before the PV product but not in the row sum: 2^-9 mag each way; the output is rounded: 2^-9 |ref|; 1e-4 for
    the fp32 sums), and a relative RMS error of at most 4e-3: the tolerance of test_gpu_attention.py.  Norm weights near 1 give
    soft scores; near 3 the scores have a standard deviation of about 10, so single keys decide rows.

Bit identity.  A single CTA or a CTA pair, tiles of 128 or 256 columns (one or two heads per epilogue pass): per element the
arithmetic is the same, so q, k, v and the pool are identical on all operands.  EPI_QKV and the checker kernel differ only in the
order of the sum of squares, which is exact on the exact operands, so there they agree bit for bit as well.  A prompt's rows do
not depend on where it is packed, on which pages or at which table row (DESIGN.md section 2: batch invariance).
"""
import numpy as np
import pytest

from test_gpu_decode_attention import EPS, HD, NAN_BITS, PAGE, SCALE, _bf16, _bits, _cos_sin, _rand_bits, _rmsnorm, _rope, _rope_allowance, _ulp, _val

LAYERS = 3
ALL = [1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 406, 1100, 2049]  # 4 804 rows: 38 M tiles
# Q3ASR_2CTA (None: unset), qkv_variant, bn, attn_variant.  The first run is the checker path, the last the prefill's own choice.
RUNS = [(None, -1, 0, 1), ("0", 0, 128, 0), ("0", 0, 256, 0), ("1", 0, 128, 0), ("1", 0, 256, 0), (None, 0, 0, 0)]


# ---- inputs -----------------------------------------------------------------------------------------------------------------------
class _Inputs:
    pass


def _layout(rng, lens, kvh, layer, n_nan=4):
    """Packing, table rows, page table and pool for prompts of these lengths (in this order)."""
    lens = np.asarray(lens)
    n = len(lens)
    need = -(-lens // PAGE)
    n_pages = int(need.sum()) + n_nan
    perm = rng.permutation(n_pages)
    perm[perm == 0], perm[-1] = perm[-1], 0  # page 0 is a NaN page
    nan_pages = perm[need.sum():]
    table_rows = n + 3
    trow = rng.permutation(table_rows)[:n]
    if (trow == np.arange(n)).all():
        trow = trow[::-1].copy()
    pt = rng.choice(nan_pages, (table_rows, int(need.max()) + 1)).astype(np.int32)
    o = 0
    for s in range(n):
        pages = perm[o:o + need[s]].copy()
        o += need[s]
        d = np.diff(pages)
        if pages.size > 2 and ((d > 0).all() or (d < 0).all()):
            pages[[0, 1]] = pages[[1, 0]]
        pt[trow[s], :need[s]] = pages
    pool = rng.integers(0, 1 << 16, size=(n_pages, LAYERS, 2, kvh, PAGE, HD), dtype=np.uint16)
    pool[:, layer] = NAN_BITS
    row0 = np.concatenate([[0], np.cumsum(lens)[:-1]])
    return [(int(r), int(L)) for r, L in zip(row0, lens)], trow.astype(np.int32), pt, pool


def _build(rng, lens, heads, kvh, hidden, layer, wn, exact=True):
    inp = _Inputs()
    inp.heads, inp.kvh, inp.hidden, inp.layer, inp.exact = heads, kvh, hidden, layer, exact
    inp.segs, inp.trow, inp.pt, inp.pool = _layout(rng, rng.permutation(lens), kvh, layer)
    rows, nqkv = sum(L for _, L in inp.segs), (heads + 2 * kvh) * HD
    inp.rows = rows
    inp.pos = np.concatenate([np.arange(L) for _, L in inp.segs])
    inp.row_seq = np.concatenate([np.full(L, inp.trow[s]) for s, (_, L) in enumerate(inp.segs)])
    if exact:
        x = rng.integers(-4, 5, size=(rows, hidden)).astype(np.float32)
        x *= np.exp2(rng.integers(-6, 4, size=rows)).astype(np.float32)[:, None]
        zero = [r0 for r0, _ in inp.segs[:2]] + [r0 + L - 1 for r0, L in inp.segs[-2:]] + list(rng.choice(rows, rows // 50))
        x[zero] = 0
        w = np.zeros((nqkv, hidden), dtype=np.float32)
        w[np.arange(nqkv)[:, None], rng.integers(0, hidden, size=(nqkv, 31))] = rng.integers(-2, 3, size=(nqkv, 31))
        inp.zero = np.unique(zero)
    else:
        x = _val(_rand_bits(rng, (rows, hidden))).astype(np.float32)
        w = _val(_rand_bits(rng, (nqkv, hidden), 0.08)).astype(np.float32)
        inp.zero = np.zeros(0, dtype=int)
    inp.x, inp.w = x, w
    inp.qw = _bf16(wn + 0.25 * rng.standard_normal(HD)).astype(np.float32)
    inp.kw = _bf16(wn + 0.25 * rng.standard_normal(HD)).astype(np.float32)
    return inp


# ---- float64 reference ------------------------------------------------------------------------------------------------------------
def _product(inp, lo, hi):
    """bf16 of columns [lo, hi) of x w^T as [rows, heads, 128] and how far the kernel's bf16 may be from it (0 on exact operands,
    where the float32 product is exact too)."""
    shape = (inp.rows, -1, HD)
    if inp.exact:
        acc = (inp.x @ inp.w[lo:hi].T).astype(np.float64)
        return _bf16(acc).reshape(shape), np.zeros(acc.shape).reshape(shape)
    acc = inp.x.astype(np.float64) @ inp.w[lo:hi].T.astype(np.float64)
    e = inp.hidden * 2.0 ** -23 * (np.abs(inp.x).astype(np.float64) @ np.abs(inp.w[lo:hi]).T.astype(np.float64))
    ref = _bf16(acc)
    return ref.reshape(shape), (_ulp(ref) + 2 * e).reshape(shape)


def _norm_rope(xh, x_allow, w, pos):
    """RMSNorm + RoPE of xh [rows, heads, 128] and its allowance, given the allowance of the product xh itself."""
    n = _rmsnorm(xh, w)
    out = _rope(n, pos)
    allow = _rope_allowance(n, out, pos)
    if x_allow.any():
        e = np.abs(np.asarray(w, np.float64)) * x_allow / np.sqrt((xh * xh).mean(axis=-1, keepdims=True) + EPS)
        c, s = (np.abs(t) for t in _cos_sin(pos))
        ea, eb = e[..., :HD // 2], e[..., HD // 2:]
        allow = allow + np.concatenate([ea * c + eb * s, eb * c + ea * s], axis=-1)
    return out, allow


def _reference(inp):
    nq, nkv = inp.heads * HD, inp.kvh * HD
    ref = _Inputs()
    (ref.qx, qx_allow), (ref.kx, kx_allow) = _product(inp, 0, nq), _product(inp, nq, nq + nkv)
    ref.v, ref.v_allow = _product(inp, nq + nkv, nq + 2 * nkv)
    ref.q, ref.q_allow = _norm_rope(ref.qx, qx_allow, inp.qw, inp.pos)
    ref.k, ref.k_allow = _norm_rope(ref.kx, kx_allow, inp.kw, inp.pos)
    return ref


def _attention(q, k, v, segs):
    """Causal softmax(q k^T * SCALE) v of every segment in float64; q [rows, heads, 128], k / v [rows, kv_heads, 128] -> out, mag."""
    heads, group = q.shape[1], q.shape[1] // k.shape[1]
    out, mag = np.empty(q.shape), np.empty(q.shape)
    for r0, L in segs:
        future = np.triu(np.ones((L, L), dtype=bool), 1)
        step = max(1, (1 << 24) // (L * L))  # heads per batch: at most 16 M scores at a time
        for h0 in range(0, heads, step):
            hh = np.arange(h0, min(heads, h0 + step))
            Q = q[r0:r0 + L, hh].transpose(1, 0, 2)
            K = k[r0:r0 + L, hh // group].transpose(1, 0, 2)
            V = v[r0:r0 + L, hh // group].transpose(1, 0, 2)
            s = Q @ K.transpose(0, 2, 1) * SCALE
            s[:, future] = -np.inf
            p = np.exp(s - s.max(axis=-1, keepdims=True))
            l = p.sum(axis=-1, keepdims=True)
            out[r0:r0 + L, hh] = ((p @ V) / l).transpose(1, 0, 2)
            mag[r0:r0 + L, hh] = ((p @ np.abs(V)) / l).transpose(1, 0, 2)
    return out, mag


# ---- running and checking ---------------------------------------------------------------------------------------------------------
def _gemm_choice(rows, nqkv):
    """gemm()'s choice for the EPI_QKV product with bn = 0 and Q3ASR_2CTA unset on this GPU (gemm.cu): (tile width, CTA pair)."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    m_tiles = -(-rows // 128)
    bn = 256 if nqkv % 256 == 0 and m_tiles * (nqkv // 256) >= sms else 128
    return bn, m_tiles * (nqkv // bn) >= 4 * sms


def _run(m, inp, monkeypatch, pair, qkv_variant, bn, attn):
    if pair is None:
        monkeypatch.delenv("Q3ASR_2CTA", raising=False)
    else:
        monkeypatch.setenv("Q3ASR_2CTA", pair)
    try:
        q, k, qkv, att, pool = m.debug_prefill_attention(inp.x, inp.w, inp.heads, inp.kvh, inp.qw, inp.kw, inp.segs, inp.trow, inp.pt,
                                                         inp.pool, inp.layer, qkv_variant=qkv_variant, bn=bn, attn_variant=attn, eps=EPS,
                                                         scale=SCALE)
    finally:
        monkeypatch.delenv("Q3ASR_2CTA", raising=False)
    r = _Inputs()
    nq, nkv = inp.heads * HD, inp.kvh * HD
    r.q, r.k = q.reshape(inp.rows, inp.heads, HD), k.reshape(inp.rows, inp.kvh, HD)
    r.qkv, r.att, r.pool = qkv, att.reshape(inp.rows, inp.heads, HD), pool
    r.v = qkv[:, nq + nkv:].reshape(inp.rows, inp.kvh, HD)
    return r


def _slots(inp):
    """(page, slot) of every packed row's position."""
    return inp.pt[inp.row_seq, inp.pos // PAGE], inp.pos % PAGE


def _check_block(inp, ref, got, what):
    """v, the pool, q and k of one run against the reference."""
    if inp.exact:
        assert np.array_equal(got.v, ref.v), (what, "v at [row, head, dim]", np.argwhere(got.v != ref.v)[:5].tolist())
    else:
        err = np.abs(got.v - ref.v)
        assert (err <= ref.v_allow).all(), (what, "v at [row, head, dim]", np.argwhere(~(err <= ref.v_allow))[:5].tolist())
    pg, sl = _slots(inp)
    want = inp.pool.copy()
    want[pg, inp.layer, 0, :, sl] = _bits(got.k)
    want[pg, inp.layer, 1, :, sl] = _bits(got.v)
    bad = np.argwhere(want != got.pool)
    assert bad.size == 0, (what, "pool differs at [page, layer, k/v, head, slot, dim]", bad[:5].tolist())
    for name, g, r, allow in (("q", got.q, ref.q, ref.q_allow), ("k", got.k, ref.k, ref.k_allow)):
        err = np.abs(g - r)
        assert (err <= allow).all(), (what, name, "at [row, head, dim]", np.argwhere(~(err <= allow))[:5].tolist())
    for name, g in (("q", got.q), ("k", got.k), ("v", got.v)):  # an all-zero row of x gives zeros
        assert (g[inp.zero] == 0).all(), (what, name, "of an all-zero row")


def _check_attention(inp, got, what, cache):
    key = got.q.tobytes() + got.k.tobytes() + got.v.tobytes()
    if key not in cache:
        cache.clear()
        cache[key] = _attention(got.q.astype(np.float64), got.k.astype(np.float64), got.v.astype(np.float64), inp.segs)
    ref, mag = cache[key]
    att = got.att.astype(np.float64)
    assert not np.isnan(att).any(), (what, "NaN attention at [row, head, dim]", np.argwhere(np.isnan(att))[:5].tolist())
    err = np.abs(att - ref)
    tol = 2.0 ** -8 * mag + 2.0 ** -8 * np.abs(ref) + 1e-4
    assert (err <= tol).all(), (what, "attention", float(err.max()), np.argwhere(err > tol)[:5].tolist())
    rel = np.sqrt((err ** 2).sum() / (ref ** 2).sum())
    assert rel <= 4e-3, (what, "attention relative RMS", rel)


def _same(a, b, what):
    for name in ("q", "k", "v"):
        assert np.array_equal(_bits(getattr(a, name)), _bits(getattr(b, name))), (what, name)
    assert np.array_equal(a.pool, b.pool), (what, "pool")


# ---- every head layout, prompt length, layer and tile configuration ---------------------------------------------------------------
CASES = [  # id, heads, kv_heads, hidden, prompt lengths, layer, norm-weight scale, operands
    ("16x8-h1024", 16, 8, 1024, ALL, 1, 1.0, "exact"),              # both presets' shape; 38 M tiles: bn 0 picks gemm_tc2_kernel<256>
    ("16x8-h2048", 16, 8, 2048, [1, 33, 129, 406, 1100], 2, 3.0, "exact"),  # the 1.7B product's K
    ("4x2-h128", 4, 2, 128, ALL, 0, 3.0, "exact"),                  # the tiny model the model tests run
    ("6x3-h1024", 6, 3, 1024, [33, 128, 256, 406, 2049], 2, 1.0, "exact"),  # a 256-wide tile holds k2 and v0; 23 M tiles
    ("2x2-h256", 2, 2, 256, ALL, 1, 1.0, "exact"),                  # group 1: fa_tc_kernel<128, true, 1>
    ("16x8-h1024-realistic", 16, 8, 1024, [1, 127, 129, 406, 1100], 0, 1.0, "realistic"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("heads,kvh,hidden,lens,layer,wn,operands", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_prefill_attention_matches_reference(tiny_model, monkeypatch, heads, kvh, hidden, lens, layer, wn, operands):
    rng = np.random.default_rng(heads * 7919 + kvh * 131 + hidden + len(lens) + layer)
    inp = _build(rng, lens, heads, kvh, hidden, layer, wn, exact=operands == "exact")
    nqkv = (heads + 2 * kvh) * HD
    if (heads, kvh, hidden) == (16, 8, 1024) and lens == ALL:  # the bench's configuration: the prefill's own choice is the 256-wide CTA-pair kernel
        assert _gemm_choice(inp.rows, nqkv) == (256, True), _gemm_choice(inp.rows, nqkv)
    if heads == 6:  # the odd CTA of the last pair holds no M tile
        assert -(-inp.rows // 128) % 2 == 1
    ref = _reference(inp)
    cache, first, first_tc = {}, None, None
    for pair, qkv_variant, bn, attn in RUNS:
        what = f"2CTA={pair} qkv_variant={qkv_variant} bn={bn} attn={attn}"
        got = _run(tiny_model, inp, monkeypatch, pair, qkv_variant, bn, attn)
        _check_block(inp, ref, got, what)
        if qkv_variant == -1 and inp.exact:  # the checker returns the whole bf16 product
            assert np.array_equal(got.qkv[:, :heads * HD].reshape(ref.qx.shape), ref.qx), what
            assert np.array_equal(got.qkv[:, heads * HD:(heads + kvh) * HD].reshape(ref.kx.shape), ref.kx), what
        if qkv_variant == 0 or inp.exact:  # the checker's sum of squares is exact, and so bit-identical, on exact operands only
            if first is None:
                first = got
            else:
                _same(got, first, what)
        if attn == 0 and first_tc is not None:  # the same q, k and v bits (just checked) give the same attention bits
            assert np.array_equal(got.att.view(np.uint32), first_tc.att.view(np.uint32)), (what, "attention differs from the first tcgen05 run")
        else:
            _check_attention(inp, got, what, cache)
            if attn == 0:
                first_tc = got


# ---- batch invariance -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pair,bn,attn", [(None, 0, 0), ("1", 128, 1)], ids=["own-choice-tc", "pair-bn128-mma"])
def test_prompt_rows_do_not_depend_on_the_packing(tiny_model, monkeypatch, pair, bn, attn):
    """Prompts of 406 and 129 rows alone, then inside a batch of six at other rows (so at other offsets within the 128-row M tiles),
    on other pages and at other table rows: their q, k, v, attention rows and pool slots are the same bits."""
    rng = np.random.default_rng(707)
    heads, kvh, hidden, layer = 16, 8, 1024, 1
    a = _build(rng, [406, 129], heads, kvh, hidden, layer, 1.0, exact=False)
    b = _build(rng, [33, 406, 257, 1, 129, 1100], heads, kvh, hidden, layer, 1.0, exact=False)
    b.qw, b.kw, b.w = a.qw, a.kw, a.w
    where = []  # (row0 in a, row0 in b, length) of every target prompt
    for ra, La in a.segs:
        rb = next(r for r, L in b.segs if L == La)
        b.x[rb:rb + La] = a.x[ra:ra + La]
        where.append((ra, rb, La))
    ga, gb = (_run(tiny_model, t, monkeypatch, pair, 0, bn, attn) for t in (a, b))
    pa, sa = _slots(a)
    pb, sb = _slots(b)
    for ra, rb, L in where:
        for name in ("q", "k", "v", "att"):
            x, y = getattr(ga, name)[ra:ra + L], getattr(gb, name)[rb:rb + L]
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), (name, "prompt of", L)
        x = ga.pool[pa[ra:ra + L], layer, :, :, sa[ra:ra + L]]
        y = gb.pool[pb[rb:rb + L], layer, :, :, sb[rb:rb + L]]
        assert np.array_equal(x, y), ("pool slots of the prompt of", L)
    for g, t in ((ga, a), (gb, b)):
        _check_attention(t, g, "packing", {})


# ---- the hook's argument checks ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_debug_hook_rejects_bad_arguments(built_lib, tiny_model):
    rng = np.random.default_rng(808)
    inp = _build(rng, [40, 3], 4, 2, 128, 1, 1.0)

    def call(m=tiny_model, **kw):
        args = dict(x=inp.x, w=inp.w, heads=4, kv_heads=2, q_norm=inp.qw, k_norm=inp.kw, segs=inp.segs, seg_table_rows=inp.trow,
                    page_table=inp.pt, pool=inp.pool, layer=1)
        args.update(kw)
        return m.debug_prefill_attention(**args)

    (r0, L0), (r1, L1) = inp.segs
    bad_pt = inp.pt.copy()
    bad_pt[-1, -1] = inp.pool.shape[0]
    for kw in (dict(segs=[(r0, L0), (r1 + 1, L1 - 1)]),                   # a gap between the segments
               dict(segs=[(r0, L0), (r1, L1 - 1)]),                       # rows no segment covers
               dict(page_table=inp.pt[:, :1]),                            # 40 positions, 32 in the table
               dict(page_table=bad_pt), dict(seg_table_rows=np.array([inp.pt.shape[0], 0])), dict(seg_table_rows=np.array([0, -1])),
               dict(qkv_variant=1), dict(bn=64), dict(bn=512), dict(attn_variant=2), dict(layer=LAYERS)):
        with pytest.raises(built_lib.Q3Error) as e:
            call(**kw)
        assert e.value.code == 1, kw
    empty = built_lib.Qwen3ASRModel("tiny")
    try:
        with pytest.raises(built_lib.Q3Error) as e:  # the RoPE frequencies come from a loaded model
            call(m=empty)
        assert e.value.code == 2
    finally:
        empty.close()
    q, k, qkv, att, pool = call()  # the handle still works
    assert not np.isnan(att).any()


# ---- the reference against the oracle (no GPU) ------------------------------------------------------------------------------------
def test_reference_helpers_match_the_oracle(tiny_oracle):
    """_attention (and the imported _rmsnorm / _rope, at prefill positions) against oracle.model.Oracle's _attention(causal=True,
    fp64=True), _rmsnorm and _rope, so that the reference the kernels are held to is itself pinned."""
    import torch
    rng = np.random.default_rng(909)
    heads, kvh, S = 4, 2, 150
    o = tiny_oracle
    x = _bf16(rng.standard_normal((S, heads, HD)) * 3)
    w = _bf16(1 + 0.25 * rng.standard_normal(HD))
    pos = np.arange(S)
    mine = _rmsnorm(x, w)
    theirs = o._rmsnorm(torch.from_numpy(x.astype(np.float32)), torch.from_numpy(w.astype(np.float32)), EPS).double().numpy()
    assert (np.abs(mine - theirs) <= _ulp(mine)).all() and (mine == theirs).mean() > 0.99
    mine_r = _rope(mine, pos)
    theirs_r = o._rope(torch.from_numpy(mine.reshape(S, heads * HD).astype(np.float32)), pos, heads).double().numpy().reshape(S, heads, HD)
    assert (np.abs(mine_r - theirs_r) <= _rope_allowance(mine, mine_r, pos)).all() and (mine_r == theirs_r).mean() > 0.99
    q = mine_r
    k = _bf16(rng.standard_normal((S, kvh, HD)))
    v = _bf16(rng.standard_normal((S, kvh, HD)))
    segs = [(0, 1), (1, 60), (61, S - 61)]
    out, mag = _attention(q, k, v, segs)
    for r0, L in segs:
        t = [torch.from_numpy(a[r0:r0 + L].reshape(L, -1).astype(np.float32)) for a in (q, k, v)]
        theirs_a = o._attention(*t, heads, kvh, float(SCALE), True, fp64=True).double().numpy().reshape(L, heads, HD)
        sl = slice(r0, r0 + L)
        assert (np.abs(out[sl] - theirs_a) <= 2.0 ** -8 * mag[sl] + 2.0 ** -8 * np.abs(out[sl]) + 1e-6).all(), (r0, L)
    assert np.array_equal(out[0], np.repeat(v[0], heads // kvh, axis=0))  # a prompt of one row attends to itself only
