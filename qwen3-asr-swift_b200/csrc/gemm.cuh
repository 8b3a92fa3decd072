// gemm.cuh — bf16 tensor-core GEMM / implicit-GEMM convolution for sm_100a.
//
//   C[rows, N] = A[rows, K] · W[N, K]^T      (both operands K-major, fp32 accumulation in TMEM)
//
// Replaces the reference's MLX `Linear`, `Conv2d` and tied-embedding `asLinear` calls on the hot path:
//   Sources/Qwen3ASR/AudioEncoder.swift:117-124,157-159,409-427,506-508
//   Sources/Qwen3ASR/FloatTextDecoder.swift:77-79,107,128-132
//   Sources/MLXCommon/PreQuantizedEmbedding.swift:45-49 (LM head, fused argmax)
//
// Structure (persistent, one CTA per SM, 256 threads):
//   warp 0    TMA producer     cp.async.bulk.tensor (4-D A boxes, 2-D W boxes), 128B swizzle, mbarrier ring
//   warp 1    MMA issuer       one lane issues tcgen05.mma (M=128, N=BN, K=16), commits to mbarriers
//   warp 2    TMEM allocator
//   warps 4-11 epilogue        tcgen05.ld 32x32b -> registers -> bias/PE/GELU/residual/SwiGLU/argmax -> global; two warps
//                              share each TMEM lane quadrant and take alternate 32-column chunks (GELU / SwiGLU epilogues
//                              of wide tiles are otherwise slower than the tile's MMAs)
// The accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// The A operand is always described by a 4-D tensor map {c, w, h, b}.  A plain GEMM is the degenerate
// case {K, M, 1, 1}.  A convolution (NHWC activations, [O][kh][kw][I] weights) is run as an implicit GEMM:
// the M tile is a box of output positions (Wb x Hb x Bb <= 128), each k-block is (tap, 64-channel chunk),
// and the producer shifts the box origin by the tap offset; out-of-image taps are zero-filled by TMA,
// the input stride (2) is the tensor map's element stride.  Channel counts that are not multiples of
// 64 (480) are handled by issuing fewer K=16 MMA steps for the last chunk of a tap.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace q3 {

enum GemmEpi : int {
    EPI_NORMAL = 0,  // out(bf16) = [resid +] bf16( act(acc + bias + row_add) ), optional zero mask / row map
    EPI_SWIGLU = 1,  // columns alternate 32 gate / 32 up (GU_UNIT): out = bf16( bf16(silu(bf16 g)) * bf16 u ), N/2 outputs
    EPI_F32 = 2,     // out(fp32) = acc + bias
    EPI_ARGMAX = 3,  // per (row, n-tile): max / lowest index of bf16(acc)
    EPI_QKV = 4,     // decoder prefill: columns are q | k | v heads of 128; per-head RMSNorm + split-half RoPE on q and k, q -> its own
                     // buffer, k -> a contiguous buffer + the paged cache, v -> out (as is) + the paged cache (FloatTextDecoder.swift:77-102)
};

// what EPI_QKV needs besides the accumulator (by value inside GemmDev)
struct QkvRope {
    const int* pos;        // [rows] position of every packed row
    const int* row_seq;    // [rows] sequence (page-table row) of every packed row
    const float2* rope;    // [64][rope_n] (cos, sin), dimension-major: lane = token row, so a warp's 32 loads of one dimension fall on
                           // consecutive positions (2-3 cache lines instead of 32 with the [pos][64] table of the decode kernels)
    int rope_n;
    const bf16 *qw, *kw;   // per-head norm weights [128]
    bf16 *q, *kc;          // q [rows, heads*128], k [rows, kv_heads*128]
    bf16* pool;            // paged cache [pages][layers][2][kv_heads][32][128]
    const int* page_table; // [seqs][max_pages]
    int max_pages, layers, layer, heads, kv_heads;
    float eps;
};

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 384;  // 4 control warps + 8 epilogue warps (two per TMEM lane quadrant)
constexpr int GEMM_MAX_TAPS = 16;
constexpr int GU_UNIT = 32;  // fused gate/up weights: 32 gate rows, then the matching 32 up rows, repeating

struct GemmDev {  // by-value kernel parameter
    int N, num_kb, kb_per_tap, C;
    int tiles_n, tiles_w, tiles_h, tiles_b;
    int Wb, Hb, Bb;
    int OW, OH, OB;
    int sw, sh;
    signed char tap_dw[GEMM_MAX_TAPS], tap_dh[GEMM_MAX_TAPS];
    void* out;
    int ldo;
    const bf16* bias;      // [N] or null
    const bf16* resid;     // [rows, ldr] or null (indexed by the destination row)
    int ldr;
    const float* row_add;  // [OW, N] fp32 or null (sinusoidal positions, indexed by w)
    const int* row_map;    // [rows] destination row or -1, or null (identity)
    const int* valid_w;    // [OB] columns w >= valid_w[b] are stored as zero, or null
    int gelu;
    int stages;            // smem ring depth actually used (<= gemm_stages(BN))
    int tma_out;           // EPI_NORMAL: output tiles are staged in shared memory and written with TMA stores (tmC is valid)
    float* amax_val;       // [rows, tiles_n]
    int* amax_idx;
    float* amax_sum;       // [rows, tiles_n] sum of exp(bf16(acc) - tile max) over the tile, or null (EPI_ARGMAX)
    QkvRope rp;            // EPI_QKV only
};

__host__ __device__ constexpr int gemm_acc_stride(int BN) { return BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256; }
__host__ __device__ constexpr int gemm_stage_bytes(int BN) { return GEMM_BM * 128 + BN * 128; }
__host__ __device__ constexpr int gemm_stages(int BN) {
    return (196 * 1024) / gemm_stage_bytes(BN) > 8 ? 8 : (196 * 1024) / gemm_stage_bytes(BN);
}
// Output staging of the plain epilogue: per group of four epilogue warps (one per TMEM lane quadrant) two buffers of 128 rows x 32
// columns bf16 (64-byte rows, 64-byte swizzle), written row-per-thread and drained by one TMA store per 32-column chunk.
constexpr int EPI_STAGE_BUF = GEMM_BM * 64;
constexpr int EPI_STAGE_BYTES = 2 * 2 * EPI_STAGE_BUF;  // 32 KB
__host__ __device__ constexpr int gemm_smem_bytes(int BN) { return gemm_stages(BN) * gemm_stage_bytes(BN) + EPI_STAGE_BYTES + 1024 + 256; }

__device__ __forceinline__ float epi_swiglu(float g_acc, float u_acc) {
    const float g = bf16_round(g_acc);
    const float s = bf16_round(silu(g));
    const float u = bf16_round(u_acc);
    return s * u;  // caller rounds to bf16 on store
}

struct TileCoord {
    int tn, w0, h0, b0;
};
__device__ __forceinline__ TileCoord gemm_tile_coord(const GemmDev& p, int tile) {
    TileCoord t;
    t.tn = tile % p.tiles_n;
    int r = tile / p.tiles_n;
    t.w0 = (r % p.tiles_w) * p.Wb;
    r /= p.tiles_w;
    t.h0 = (r % p.tiles_h) * p.Hb;
    t.b0 = (r / p.tiles_h) * p.Bb;
    return t;
}

// One tile's epilogue for one thread: TMEM row -> registers -> bias / PE / GELU / residual / SwiGLU / argmax -> global.
// `tfull` is the barrier the accumulator's completion is committed to (waited on here, after the index arithmetic).
// Shared-memory staging of the plain epilogue's TMA stores: `buf` = this warp group's two buffers, `ctr` counts its stores.
struct EpiStage {
    const CUtensorMap* tmC;
    uint8_t* buf;
    uint32_t ctr;
};

template <int BN, int EPI>
__device__ __forceinline__ void gemm_epilogue_tile(const GemmDev& p, const TileCoord tc, uint32_t tmem_acc, uint64_t* tfull, uint32_t aphase,
                                                   int q, int lane, int chalf, int tile_rows, EpiStage& es) {
    const int n0 = tc.tn * BN;
    const int r = q * 32 + lane;
    const int w = tc.w0 + r % p.Wb;
    const int h = tc.h0 + (r / p.Wb) % p.Hb;
    const int b = tc.b0 + r / (p.Wb * p.Hb);
    bool row_ok = r < tile_rows && w < p.OW && h < p.OH && b < p.OB;
    long row = row_ok ? ((long)b * p.OH + h) * p.OW + w : 0;
    bool zero = false;
    if (row_ok && p.valid_w != nullptr) zero = w >= __ldg(p.valid_w + b);
    if (row_ok && p.row_map != nullptr) {
        row = __ldg(p.row_map + row);
        row_ok = row >= 0;
    }
    const uint32_t t_row = tmem_acc + (uint32_t(q * 32) << 16);
    int qkv_pos = 0, qkv_page = 0;  // EPI_QKV: the row's position and KV page, fetched under the wait for the accumulator
    if constexpr (EPI == EPI_QKV) {
        if (row_ok) {
            qkv_pos = __ldg(p.rp.pos + row);
            qkv_page = __ldg(p.rp.page_table + (size_t)__ldg(p.rp.row_seq + row) * p.rp.max_pages + qkv_pos / 32);
        }
    }
    if constexpr (EPI != EPI_NORMAL && EPI != EPI_F32) {  // (the plain epilogue prefetches its bias / residual rows before it waits)
        ptx::mbar_wait(tfull, aphase);
        ptx::tc_fence_after();
    }

    if constexpr (EPI == EPI_SWIGLU) {
        // weight rows alternate GU_UNIT gate rows / GU_UNIT up rows, so every 64 accumulator columns hold 32 outputs
        if constexpr (BN % (2 * GU_UNIT) == 0) {
            bf16* out = reinterpret_cast<bf16*>(p.out) + (size_t)row * p.ldo + tc.tn * (BN / 2);
            const bool gu32 = (reinterpret_cast<uintptr_t>(p.out) & 31) == 0 && p.ldo % 16 == 0;
#pragma unroll 1
            for (int c = chalf; c < BN / 32; c += 2) {  // 16 outputs per step
                const int col = (c >> 1) * (2 * GU_UNIT) + (c & 1) * 16;
                uint32_t g[16], u[16];
                ptx::tmem_ld_32x16(t_row + col, g);
                ptx::tmem_ld_32x16(t_row + col + GU_UNIT, u);
                ptx::tmem_ld_wait();
                if (row_ok) {
                    uint32_t pk[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float a = epi_swiglu(__uint_as_float(g[2 * j]), __uint_as_float(u[2 * j]));
                        const float bb = epi_swiglu(__uint_as_float(g[2 * j + 1]), __uint_as_float(u[2 * j + 1]));
                        pk[j] = pack_bf16x2(a, bb);
                    }
                    if (gu32) {
                        st_global_v8(out + c * 16, pk[0], pk[1], pk[2], pk[3], pk[4], pk[5], pk[6], pk[7]);
                    } else {
                        uint4* dst = reinterpret_cast<uint4*>(out + c * 16);
                        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
                    }
                }
            }
        }
    } else if constexpr (EPI == EPI_QKV) {
        // One head (128 accumulator columns) at a time per thread = per token row; the two warps of a lane quadrant take alternate
        // heads of the tile.  The raw product is rounded to bf16 first (the reference's Linear output), then normed, rounded,
        // rotated, rounded — the rounding points of qknorm_rope_kv_kernel (ops.cu), which this epilogue replaces in the prefill:
        // the QKV product is no longer written, re-read and re-written (436 MB per layer at 64 x 30 s).
        if constexpr (BN % 128 == 0) {
            const QkvRope& R = p.rp;
            const int pos = qkv_pos, page = qkv_page;
            bf16* page_base = R.pool + (((size_t)page * R.layers + R.layer) * 2) * R.kv_heads * (32 * 128) + (pos % 32) * 128;
#pragma unroll 1
            for (int hh = chalf; hh < BN / 128; hh += 2) {
                const int slot = tc.tn * (BN / 128) + hh;  // [0, heads) q, [heads, heads + kv_heads) k, then v
                const uint32_t t_head = t_row + hh * 128;
                const bool is_q = slot < R.heads, is_v = slot >= R.heads + R.kv_heads;
                const int kvh = is_v ? slot - R.heads - R.kv_heads : slot - R.heads;
                if (is_v) {
#pragma unroll 1
                    for (int c = 0; c < 4; c++) {
                        uint32_t v[32];
                        ptx::tmem_ld_32x32(t_head + c * 32, v);
                        ptx::tmem_ld_wait();
                        if (row_ok) {
                            uint4 pk[4];
#pragma unroll
                            for (int j = 0; j < 4; j++)
                                pk[j] = make_uint4(pack_bf16x2(__uint_as_float(v[8 * j]), __uint_as_float(v[8 * j + 1])),
                                                   pack_bf16x2(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3])),
                                                   pack_bf16x2(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5])),
                                                   pack_bf16x2(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7])));
                            bf16* d0 = reinterpret_cast<bf16*>(p.out) + (size_t)row * p.ldo + slot * 128 + c * 32;
                            bf16* d1 = page_base + ((size_t)R.kv_heads + kvh) * (32 * 128) + c * 32;
#pragma unroll
                            for (int j = 0; j < 4; j += 2) {  // 256-bit stores (all these rows are 256-byte aligned)
                                st_global_v8(d0 + j * 8, pk[j].x, pk[j].y, pk[j].z, pk[j].w, pk[j + 1].x, pk[j + 1].y, pk[j + 1].z, pk[j + 1].w);
                                st_global_v8(d1 + j * 8, pk[j].x, pk[j].y, pk[j].z, pk[j].w, pk[j + 1].x, pk[j + 1].y, pk[j + 1].z, pk[j + 1].w);
                            }
                        }
                    }
                    continue;
                }
                float ss = 0.f;
#pragma unroll 1
                for (int c = 0; c < 4; c++) {
                    uint32_t v[32];
                    ptx::tmem_ld_32x32(t_head + c * 32, v);
                    ptx::tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        const float x = bf16_round(__uint_as_float(v[j]));
                        ss = fmaf(x, x, ss);
                    }
                }
                const float r = rsqrtf(ss * (1.0f / 128.0f) + R.eps);
                const bf16* nw = is_q ? R.qw : R.kw;
                bf16* dst = is_q ? R.q + (size_t)row * R.heads * 128 + slot * 128 : R.kc + (size_t)row * R.kv_heads * 128 + kvh * 128;
                bf16* dst2 = page_base + (size_t)kvh * (32 * 128);  // K half of the page (k heads only)
#pragma unroll 1
                for (int c = 0; c < 2; c++) {  // dims [32c, 32c + 32) pair with [64 + 32c, ...)
                    uint32_t a[32], b[32];
                    ptx::tmem_ld_32x32(t_head + c * 32, a);
                    ptx::tmem_ld_32x32(t_head + 64 + c * 32, b);
                    ptx::tmem_ld_wait();
                    if (row_ok) {
                        const float2* tp = R.rope + (size_t)(c * 32) * R.rope_n + pos;  // (cos, sin) of dimension 32 c of this row's position
                        const uint4* wa = reinterpret_cast<const uint4*>(nw + c * 32);
                        const uint4* wb = reinterpret_cast<const uint4*>(nw + 64 + c * 32);
                        uint32_t oa[16], ob[16];
#pragma unroll
                        for (int j4 = 0; j4 < 4; j4++) {
                            const uint4 wua = __ldg(wa + j4), wub = __ldg(wb + j4);
                            const uint32_t wwa[4] = {wua.x, wua.y, wua.z, wua.w}, wwb[4] = {wub.x, wub.y, wub.z, wub.w};
#pragma unroll
                            for (int j2 = 0; j2 < 4; j2++) {
                                const int j = 8 * j4 + 2 * j2;
                                const float2 t0 = __ldg(tp + (size_t)j * R.rope_n), t1 = __ldg(tp + (size_t)(j + 1) * R.rope_n);
                                const float4 t = make_float4(t0.x, t0.y, t1.x, t1.y);  // cos, sin of dims j and j + 1
                                const float2 fa = unpack_bf16x2(wwa[j2]), fb = unpack_bf16x2(wwb[j2]);
                                const float xa0 = bf16_round(bf16_round(__uint_as_float(a[j])) * r * fa.x);
                                const float xa1 = bf16_round(bf16_round(__uint_as_float(a[j + 1])) * r * fa.y);
                                const float xb0 = bf16_round(bf16_round(__uint_as_float(b[j])) * r * fb.x);
                                const float xb1 = bf16_round(bf16_round(__uint_as_float(b[j + 1])) * r * fb.y);
                                oa[j >> 1] = pack_bf16x2(fmaf(xa0, t.x, -1.f * xb0 * t.y), fmaf(xa1, t.z, -1.f * xb1 * t.w));
                                ob[j >> 1] = pack_bf16x2(fmaf(xb0, t.x, xa0 * t.y), fmaf(xb1, t.z, xa1 * t.w));
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 2; j++) {  // 256-bit stores
                            st_global_v8(dst + c * 32 + j * 16, oa[8 * j], oa[8 * j + 1], oa[8 * j + 2], oa[8 * j + 3], oa[8 * j + 4], oa[8 * j + 5],
                                         oa[8 * j + 6], oa[8 * j + 7]);
                            st_global_v8(dst + 64 + c * 32 + j * 16, ob[8 * j], ob[8 * j + 1], ob[8 * j + 2], ob[8 * j + 3], ob[8 * j + 4],
                                         ob[8 * j + 5], ob[8 * j + 6], ob[8 * j + 7]);
                        }
                        if (!is_q) {
#pragma unroll
                            for (int j = 0; j < 2; j++) {
                                st_global_v8(dst2 + c * 32 + j * 16, oa[8 * j], oa[8 * j + 1], oa[8 * j + 2], oa[8 * j + 3], oa[8 * j + 4],
                                             oa[8 * j + 5], oa[8 * j + 6], oa[8 * j + 7]);
                                st_global_v8(dst2 + 64 + c * 32 + j * 16, ob[8 * j], ob[8 * j + 1], ob[8 * j + 2], ob[8 * j + 3], ob[8 * j + 4],
                                             ob[8 * j + 5], ob[8 * j + 6], ob[8 * j + 7]);
                            }
                        }
                    }
                }
            }
        }
    } else if constexpr (EPI == EPI_ARGMAX) {
        float best = -INFINITY;
        int best_i = 0;
#pragma unroll 1
        for (int c = 0; c < (chalf == 0 ? BN / 32 : 0); c++) {  // one warp per quadrant scans the whole row (weight-streaming bound)
            uint32_t v[32];
            ptx::tmem_ld_32x32(t_row + c * 32, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const float x = bf16_round(__uint_as_float(v[j]));
                if (x > best) { best = x; best_i = n0 + c * 32 + j; }
            }
        }
        float sum = 0.f;
#pragma unroll 1
        for (int c = 0; c < (chalf == 0 && p.amax_sum != nullptr ? BN / 32 : 0); c++) {  // second pass, columns in order
            uint32_t v[32];
            ptx::tmem_ld_32x32(t_row + c * 32, v);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; j++) sum += __expf(bf16_round(__uint_as_float(v[j])) - best);
        }
        if (row_ok && chalf == 0) {
            p.amax_val[(size_t)row * p.tiles_n + tc.tn] = best;
            p.amax_idx[(size_t)row * p.tiles_n + tc.tn] = best_i;
            if (p.amax_sum != nullptr) p.amax_sum[(size_t)row * p.tiles_n + tc.tn] = sum;
        }
    } else {
        // Bias and residual do not depend on the accumulator: the loads of chunk c + 2 are issued before chunk c is processed (and
        // those of the first chunk before the wait for the accumulator, see the top of the function), so their L2 / HBM latency
        // (~1 us for a residual row that was written a layer ago) is not paid once per chunk.  Products with a short K loop
        // (K = 896: 14 k-blocks, 4.5 us of MMAs per tile) were bound by exactly that: out-proj 35 % tensor-active (ncu, round 1).
        uint4 bnx[4], rnx[4];
        const bool resid32 = EPI == EPI_NORMAL && p.resid != nullptr && (reinterpret_cast<uintptr_t>(p.resid) & 31) == 0 && p.ldr % 16 == 0;
        const bool out32 = EPI == EPI_NORMAL && (reinterpret_cast<uintptr_t>(p.out) & 31) == 0 && p.ldo % 16 == 0;
        auto fetch = [&](int c) {
            if (EPI == EPI_NORMAL || EPI == EPI_F32) {
                const int col = n0 + c * 32;
                if (row_ok && p.bias != nullptr) {
                    const uint4* bp = reinterpret_cast<const uint4*>(p.bias + col);
#pragma unroll
                    for (int j = 0; j < 4; j++) bnx[j] = __ldg(bp + j);
                }
                if (EPI == EPI_NORMAL && row_ok && p.resid != nullptr) {
                    const bf16* rp = p.resid + (size_t)row * p.ldr + col;
                    if (resid32) {  // 32-byte aligned rows: two 256-bit loads per row instead of four 128-bit ones
                        const U8 lo = ld_global_nc_v8(rp), hi = ld_global_nc_v8(rp + 16);
                        rnx[0] = make_uint4(lo.v[0], lo.v[1], lo.v[2], lo.v[3]); rnx[1] = make_uint4(lo.v[4], lo.v[5], lo.v[6], lo.v[7]);
                        rnx[2] = make_uint4(hi.v[0], hi.v[1], hi.v[2], hi.v[3]); rnx[3] = make_uint4(hi.v[4], hi.v[5], hi.v[6], hi.v[7]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; j++) rnx[j] = __ldg(reinterpret_cast<const uint4*>(rp) + j);
                    }
                }
            }
        };
        if (chalf < BN / 32) fetch(chalf);
        ptx::mbar_wait(tfull, aphase);
        ptx::tc_fence_after();
#pragma unroll 1
        for (int c = chalf; c < BN / 32; c += 2) {
            const int col = n0 + c * 32;
            uint4 bvv[4], rvv[4];
#pragma unroll
            for (int j = 0; j < 4; j++) { bvv[j] = bnx[j]; rvv[j] = rnx[j]; }
            if (c + 2 < BN / 32) fetch(c + 2);
            uint32_t v[32];
            ptx::tmem_ld_32x32(t_row + c * 32, v);
            ptx::tmem_ld_wait();
            if (row_ok) {
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; j++) f[j] = __uint_as_float(v[j]);
                if (p.bias != nullptr) {
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint4 bv = bvv[j];
                        float2 t;
                        t = unpack_bf16x2(bv.x); f[8 * j + 0] += t.x; f[8 * j + 1] += t.y;
                        t = unpack_bf16x2(bv.y); f[8 * j + 2] += t.x; f[8 * j + 3] += t.y;
                        t = unpack_bf16x2(bv.z); f[8 * j + 4] += t.x; f[8 * j + 5] += t.y;
                        t = unpack_bf16x2(bv.w); f[8 * j + 6] += t.x; f[8 * j + 7] += t.y;
                    }
                }
                if constexpr (EPI == EPI_F32) {
                    float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (size_t)row * p.ldo + col);
#pragma unroll
                    for (int j = 0; j < 8; j++) dst[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                } else {
                    if (p.row_add != nullptr) {
                        const float4* ap = reinterpret_cast<const float4*>(p.row_add + (size_t)w * p.N + col);
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const float4 a = __ldg(ap + j);
                            f[4 * j] += a.x; f[4 * j + 1] += a.y; f[4 * j + 2] += a.z; f[4 * j + 3] += a.w;
                        }
                    }
                    if (p.gelu) {  // two values per instruction on the packed fp32 pipe (common.cuh)
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const float2 gg = gelu_erf2(make_float2(f[j], f[j + 1]));
                            f[j] = gg.x;
                            f[j + 1] = gg.y;
                        }
                    }
                    if (zero) {
#pragma unroll
                        for (int j = 0; j < 32; j++) f[j] = 0.f;
                    }
                    if (p.resid != nullptr) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const uint4 rv = rvv[j];
                            float2 t;
                            t = unpack_bf16x2(rv.x); f[8 * j + 0] = t.x + bf16_round(f[8 * j + 0]); f[8 * j + 1] = t.y + bf16_round(f[8 * j + 1]);
                            t = unpack_bf16x2(rv.y); f[8 * j + 2] = t.x + bf16_round(f[8 * j + 2]); f[8 * j + 3] = t.y + bf16_round(f[8 * j + 3]);
                            t = unpack_bf16x2(rv.z); f[8 * j + 4] = t.x + bf16_round(f[8 * j + 4]); f[8 * j + 5] = t.y + bf16_round(f[8 * j + 5]);
                            t = unpack_bf16x2(rv.w); f[8 * j + 6] = t.x + bf16_round(f[8 * j + 6]); f[8 * j + 7] = t.y + bf16_round(f[8 * j + 7]);
                        }
                    }
                    bf16* dst = reinterpret_cast<bf16*>(p.out) + (size_t)row * p.ldo + col;
                    uint32_t pk[16];
#pragma unroll
                    for (int j = 0; j < 16; j++) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
                    if (p.tma_out) {
                        // this thread's row of the chunk: 64 bytes at row pitch 64, 16-byte pieces XOR-swizzled with bits 1-2 of the
                        // row (the TMA 64-byte swizzle): the 32 lanes' stores spread over all banks
                        uint8_t* srow = es.buf + (es.ctr & 1) * EPI_STAGE_BUF + r * 64;
                        const int sw = (r >> 1) & 3;
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            *reinterpret_cast<uint4*>(srow + ((j ^ sw) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                    } else if (out32) {
                        st_global_v8(dst, pk[0], pk[1], pk[2], pk[3], pk[4], pk[5], pk[6], pk[7]);
                        st_global_v8(dst + 16, pk[8], pk[9], pk[10], pk[11], pk[12], pk[13], pk[14], pk[15]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            reinterpret_cast<uint4*>(dst)[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                    }
                }
            }
            if constexpr (EPI == EPI_NORMAL) {
                if (p.tma_out) {
                    // One store per (warp group, chunk): 128 rows x 32 columns leave as ONE bulk tensor copy instead of 256 row-strided
                    // 32-byte stores.  The elected thread first makes sure the group's previous store has finished reading the
                    // OTHER buffer (the next chunk will be written there), so the barrier below says both "this chunk is staged" and
                    // "the other buffer is free".
                    ptx::fence_proxy_async();
                    const bool elected = q == 0 && lane == 0;
                    if (elected) ptx::bulk_wait_group_read<0>();
                    ptx::named_bar_sync(1 + chalf, 128);
                    if (elected && tc.w0 < p.OW && tc.h0 < p.OH && tc.b0 < p.OB) {  // (the odd CTA of a pair may hold a tile past the end)
                        ptx::tma_store_4d(es.tmC, col, tc.w0, tc.h0, tc.b0, es.buf + (es.ctr & 1) * EPI_STAGE_BUF);
                        ptx::bulk_commit_group();
                    }
                    es.ctr++;
                }
            }
        }
    }
}

template <int BN, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
               const GemmDev p) {
    constexpr int MAX_STAGES = gemm_stages(BN);
    const int STAGES = p.stages;  // <= MAX_STAGES; the decode step asks for a shallow ring so the next kernel's CTAs fit beside this one
    constexpr int STAGE_BYTES = gemm_stage_bytes(BN);
    constexpr int ACC_STRIDE = gemm_acc_stride(BN);
    constexpr int TMEM_COLS = 2 * ACC_STRIDE;
    constexpr uint32_t IDESC = ptx::umma_idesc_bf16(GEMM_BM, BN);
    static_assert(BN % 32 == 0 && BN <= 256, "BN");
    static_assert(TMEM_COLS >= 32 && TMEM_COLS <= 512, "tmem");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* epi_stage = smem + STAGES * STAGE_BYTES;  // [2 warp groups][2 buffers], only when p.tma_out
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(epi_stage + (p.tma_out ? EPI_STAGE_BYTES : 0));
    uint64_t* empty_bar = full_bar + MAX_STAGES;
    uint64_t* tfull_bar = empty_bar + MAX_STAGES;  // [2]
    uint64_t* tempty_bar = tfull_bar + 2;      // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_tiles = p.tiles_n * p.tiles_w * p.tiles_h * p.tiles_b;
    const int tile_rows = p.Wb * p.Hb * p.Bb;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmA);
        ptx::prefetch_tmap(&tmB);
        if (p.tma_out) ptx::prefetch_tmap(&tmC);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; s++) {
            ptx::mbar_init(&tfull_bar[s], 1);
            ptx::mbar_init(&tempty_bar[s], 256);
        }
        ptx::fence_barrier_init();
    }
    if (warp == 2) ptx::tmem_alloc<TMEM_COLS>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            ptx::grid_dep_launch();
            const uint32_t tx_bytes = (uint32_t)(tile_rows * 128 + BN * 128);
            // The weight (B) tiles do not depend on the previous kernel: start the first tile's ring with them, then wait for
            // the producer of A (programmatic dependent launch; a no-op for ordinary launches).
            int pre = 0;
            if ((int)blockIdx.x < num_tiles) {
                const int n0 = gemm_tile_coord(p, blockIdx.x).tn * BN;
                pre = min(STAGES, p.num_kb);
                int tap = 0, cc = 0;
                for (int i = 0; i < pre; i++) {
                    ptx::mbar_arrive_expect_tx(&full_bar[i], tx_bytes);
                    ptx::tma_load_2d(smem + i * STAGE_BYTES + GEMM_BM * 128, &tmB, tap * p.C + cc * GEMM_BK, n0, &full_bar[i]);
                    if (++cc == p.kb_per_tap) { cc = 0; tap++; }
                }
            }
            ptx::grid_dep_wait();  // A (and everything the epilogue reads) comes from the previous kernel
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const TileCoord tc = gemm_tile_coord(p, tile);
                const int n0 = tc.tn * BN;
                int tap = 0, cc = 0;
                for (int kb = 0; kb < p.num_kb; kb++) {
                    uint8_t* sa = smem + stage * STAGE_BYTES;
                    uint8_t* sb = sa + GEMM_BM * 128;
                    if (pre > 0) {
                        pre--;  // slot already armed and its B tile in flight
                    } else {
                        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                        ptx::mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
                        ptx::tma_load_2d(sb, &tmB, tap * p.C + cc * GEMM_BK, n0, &full_bar[stage]);
                    }
                    ptx::tma_load_4d(sa, &tmA, cc * GEMM_BK, tc.w0 * p.sw + p.tap_dw[tap], tc.h0 * p.sh + p.tap_dh[tap],
                                     tc.b0, &full_bar[stage]);
                    if (++cc == p.kb_per_tap) { cc = 0; tap++; }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            const int last_steps = (p.C - (p.kb_per_tap - 1) * GEMM_BK + 15) >> 4;  // K=16 steps in a tap's last chunk
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
                const int as = it & 1;
                const uint32_t aphase = (it >> 1) & 1;
                ptx::mbar_wait(&tempty_bar[as], aphase ^ 1);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + as * ACC_STRIDE;
                int cc = 0;
                for (int kb = 0; kb < p.num_kb; kb++) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t sa = ptx::smem_u32(smem + stage * STAGE_BYTES);
                    const uint32_t sb = sa + GEMM_BM * 128;
                    const int steps = (cc == p.kb_per_tap - 1) ? last_steps : GEMM_BK / 16;
#pragma unroll
                    for (int k = 0; k < GEMM_BK / 16; k++) {
                        if (k < steps) {
                            const uint64_t da = ptx::umma_desc_sw128(sa + k * 32);
                            const uint64_t db = ptx::umma_desc_sw128(sb + k * 32);
                            ptx::mma_bf16_ss(d_tmem, da, db, IDESC, (kb | k) != 0 ? 1u : 0u);
                        }
                    }
                    ptx::mma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs retire
                    if (++cc == p.kb_per_tap) cc = 0;
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                ptx::mma_commit(&tfull_bar[as]);  // accumulator complete -> epilogue
            }
        }
    } else if (warp >= 4) {
        // ===== epilogue =====
        const int q = warp & 3;          // TMEM lane quadrant this warp may access
        const int chalf = (warp - 4) >> 2;  // which of the quadrant's two warps: takes chunks chalf, chalf + 2, ...
        int it = 0;
        ptx::grid_dep_wait();  // the epilogue prefetches residual rows (the previous kernel's output) before it sees the accumulator
        EpiStage es{&tmC, epi_stage + chalf * 2 * EPI_STAGE_BUF, 0u};
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            gemm_epilogue_tile<BN, EPI>(p, gemm_tile_coord(p, tile), tmem_base + as * ACC_STRIDE, &tfull_bar[as], aphase, q, lane, chalf, tile_rows, es);
            ptx::tc_fence_before();
            ptx::mbar_arrive(&tempty_bar[as]);
        }
        if (p.tma_out && q == 0 && lane == 0) ptx::bulk_wait_group<0>();  // the staged tiles have reached memory before the CTA leaves
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

// ---------------------------------------------------------------------------------------------
// Host API (gemm.cu)
// ---------------------------------------------------------------------------------------------
struct GemmA {               // activation operand as a 4-D {c, w, h, b} view, element strides (bf16 units)
    const bf16* ptr = nullptr;
    int C = 0, W = 1, H = 1, B = 1;
    long sW = 0, sH = 0, sB = 0;   // strides of w, h, b in elements (c is contiguous)
};
struct GemmShape {           // how output rows map onto the view, and the k-block program
    int Wb = 128, Hb = 1, Bb = 1;  // M-tile box in output positions
    int OW = 0, OH = 1, OB = 1;    // output extents
    int sw = 1, sh = 1;            // input step per output step
    int taps = 1;
    signed char tap_dw[GEMM_MAX_TAPS] = {0}, tap_dh[GEMM_MAX_TAPS] = {0};
};
struct GemmEpiArgs {
    int epi = EPI_NORMAL;
    void* out = nullptr;
    int ldo = 0;
    const bf16* bias = nullptr;
    const bf16* resid = nullptr;
    int ldr = 0;
    const float* row_add = nullptr;
    const int* row_map = nullptr;
    const int* valid_w = nullptr;
    int gelu = 0;
    int max_stages = 0;  // 0: as deep as shared memory allows
    float* amax_val = nullptr;
    int* amax_idx = nullptr;
    float* amax_sum = nullptr;  // EPI_ARGMAX: also the per-(row, n-tile) sum of exp(bf16(acc) - tile max), for log-probabilities
    QkvRope rp = {};  // EPI_QKV
};

void gemm_init(int device);  // resolves cuTensorMapEncodeTiled, sets smem attributes, reads the SM count
int gemm_pick_bn(int N, int epi);
int gemm_pick_bn(int N, int epi, long m_tiles);
// General form.  W is [N, taps*C] row-major bf16.  `simt` runs the CUDA-core checker kernel instead
// (tests only: bisects tensor-core bugs; never used by the model code).
void gemm_conv(const GemmA& a, const GemmShape& s, const bf16* W, int N, const GemmEpiArgs& e, cudaStream_t st,
               bool simt = false, int bn = 0);
// Plain C[M,N] = A[M,K](lda) W[N,K]^T
void gemm(const bf16* A, int lda, int M, int K, const bf16* W, int N, const GemmEpiArgs& e, cudaStream_t st,
          bool simt = false, int bn = 0);
unsigned long long gemm_launch_count();

// ---- decode-step weight-streaming GEMM (skinny.cuh): Y[Mtok, N] = X[Mtok, K](ldx) W[N, K]^T, Mtok <= SKINNY_MAX_ROWS (256) per launch ----
constexpr int SKINNY_MAX_ROWS = 256;  // token rows of the weight-streaming decode step: the UMMA N operand (<= 256)
enum SkinnyEpi : int {
    SK_PARTIAL = 0,  // out(fp32)[split][m][n] = acc
    SK_STORE = 1,    // out(bf16)[m][n] = bf16(acc)                       (splits must be 1)
};

// number of K splits the launch will use for this shape (1 for SK_STORE)
int gemm_skinny_splits(int N, int K, int epi);
// SK_PARTIAL: out = fp32 [splits][Mtok][N] (split_stride = Mtok * N); SK_STORE: bf16 [Mtok, ldo]
void gemm_skinny(const bf16* X, int ldx, int Mtok, int K, const bf16* W, int N, int epi, void* out, int ldo, cudaStream_t st);
// Decode-step LM head (lmhead.cuh): per 128-row vocabulary tile the (value, index) of the first maximum of bf16(X E^T) for every token
// row, amax_val / amax_idx [Mtok, lmhead_tiles(N)], to be merged by argmax_reduce.  Mtok <= SKINNY_MAX_ROWS.
int lmhead_tiles(int N);
// amax_sum (may be null): also sum over the tile's rows of exp(z - tile max) per token, for log-probabilities (a second instantiation).
void lmhead_argmax(const bf16* X, int ldx, int Mtok, int K, const bf16* W, int N, float* amax_val, int* amax_idx, cudaStream_t st,
                   float* amax_sum = nullptr);
// final reduce of EPI_ARGMAX partials: out[row] = index of the maximum (lowest index on ties)
void argmax_reduce(const float* val, const int* idx, int rows, int tiles, int32_t* out, float* out_val, cudaStream_t st);
// the same plus out_lp[row] = z[out[row]] - logsumexp(z) from the per-tile sums of exp(z - tile max) (tile_sum) and per-tile maxima
// (tile_max, or val itself when null).  raw (may be null): bf16 logits [rows, ld] to read z[out[row]] from (decoder knobs, where the
// chosen token need not be the maximum of the raw logits); else z[out[row]] is the maximum.
void argmax_lse_reduce(const float* val, const int* idx, const float* tile_sum, const float* tile_max, const bf16* raw, int ld, int rows,
                       int tiles, int32_t* out, float* out_val, float* out_lp, cudaStream_t st);

}  // namespace q3
