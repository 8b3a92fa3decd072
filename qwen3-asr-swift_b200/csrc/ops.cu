// ops.cu — CUDA-core kernels around the GEMMs: conv2d1, LayerNorm, RMSNorm, embedding gather/splice,
// q/k-norm + RoPE + KV-cache write, paged decode attention, greedy bookkeeping, dtype/init helpers.
// Reductions are warp-shuffle based (one warp per row / per head).
#include <stdlib.h>

#include <algorithm>

#include "ops.cuh"
#include "ptx.cuh"

namespace q3 {

namespace {

__device__ __forceinline__ uint2 ld8(const bf16* p) { return *reinterpret_cast<const uint2*>(p); }
__device__ __forceinline__ void st8(bf16* p, float a, float b, float c, float d) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(a, b), pack_bf16x2(c, d));
}

// ------------------------------------------------------------------------------------------
// conv2d1 + GELU.  grid (64 output rows, chunks); thread = one output-channel pair, loops over columns.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv1_kernel(const float* __restrict__ mel, const Conv1Chunk* __restrict__ chunks,
                                                    const bf16* __restrict__ w, const bf16* __restrict__ bias, int C, int chunk_w,
                                                    bf16* __restrict__ out) {
    extern __shared__ float2 s_in[];  // [3][chunk_w + 2] as (x, x) pairs: the packed multiply-adds below take them as they are
    const int oh = blockIdx.x, g = blockIdx.y;
    const Conv1Chunk c = chunks[g];
    const int pitch = chunk_w + 2;
    for (int i = threadIdx.x; i < 3 * pitch; i += blockDim.x) {
        const int r = i / pitch, j = i % pitch - 1;  // input column j in [-1, chunk_w]
        const int ih = 2 * oh + r - 1;
        float v = 0.f;
        if (ih >= 0 && ih < 128 && j >= 0 && j < c.len) v = __ldg(mel + c.mel_off + (long long)ih * c.T + c.f0 + j);
        s_in[i] = make_float2(v, v);
    }
    __syncthreads();
    const int OW = chunk_w / 2;
    const int w1 = (c.w0 - 1) / 2 + 1;  // valid output columns of this chunk
    bf16* orow = out + ((size_t)g * 64 + oh) * OW * C;
    for (int cp = threadIdx.x; cp < C / 2; cp += blockDim.x) {
        // the thread's two output channels ride the two lanes of the packed fp32 pipe: 9 FFMA2 + one packed GELU per output pair
        float2 wab[9];
#pragma unroll
        for (int t = 0; t < 9; t++) wab[t] = make_float2(__bfloat162float(w[(2 * cp) * 9 + t]), __bfloat162float(w[(2 * cp + 1) * 9 + t]));
        const float2 bab = make_float2(__bfloat162float(bias[2 * cp]), __bfloat162float(bias[2 * cp + 1]));
        for (int ow = 0; ow < OW; ow++) {
            float2 ab = make_float2(0.f, 0.f);
            if (ow < w1) {
                ab = bab;
#pragma unroll
                for (int r = 0; r < 3; r++)
#pragma unroll
                    for (int q = 0; q < 3; q++) ab = f2_fma(s_in[r * pitch + 2 * ow + q], wab[r * 3 + q], ab);  // column 2*ow + q - 1, stored at +1
                ab = gelu_erf2(ab);
            }
            *reinterpret_cast<uint32_t*>(orow + (size_t)ow * C + 2 * cp) = pack_bf16x2(ab.x, ab.y);
        }
    }
}

// ------------------------------------------------------------------------------------------
// LayerNorm / RMSNorm: one warp per row, 4 elements per lane per step (8-byte loads).
// ------------------------------------------------------------------------------------------
template <int MAXV>
__global__ void __launch_bounds__(256) layernorm_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w,
                                                        const bf16* __restrict__ b, bf16* __restrict__ y, int rows, int d, float eps) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const int nv = d >> 7;
    const bf16* xr = x + (size_t)row * d;
    float v[MAXV][4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; i++)
        if (i < nv) {
            const uint2 u = ld8(xr + i * 128 + lane * 4);
            const float2 a = unpack_bf16x2(u.x), c = unpack_bf16x2(u.y);
            v[i][0] = a.x; v[i][1] = a.y; v[i][2] = c.x; v[i][3] = c.y;
            s += (a.x + a.y) + (c.x + c.y);
        }
    const float mean = warp_sum(s) / (float)d;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; i++)
        if (i < nv) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float t = v[i][j] - mean;
                q = fmaf(t, t, q);
            }
        }
    const float rstd = rsqrtf(warp_sum(q) / (float)d + eps);
    bf16* yr = y + (size_t)row * d;
#pragma unroll
    for (int i = 0; i < MAXV; i++)
        if (i < nv) {
            const int c0 = i * 128 + lane * 4;
            const uint2 wu = ld8(w + c0), bu = ld8(b + c0);
            const float2 w0 = unpack_bf16x2(wu.x), w1 = unpack_bf16x2(wu.y), b0 = unpack_bf16x2(bu.x), b1 = unpack_bf16x2(bu.y);
            st8(yr + c0, fmaf((v[i][0] - mean) * rstd, w0.x, b0.x), fmaf((v[i][1] - mean) * rstd, w0.y, b0.y),
                fmaf((v[i][2] - mean) * rstd, w1.x, b1.x), fmaf((v[i][3] - mean) * rstd, w1.y, b1.y));
        }
}

template <int MAXV>
__global__ void __launch_bounds__(256) rmsnorm_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w, bf16* __restrict__ y,
                                                      int rows, int d, float eps, const int* __restrict__ row_index) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const int nv = d >> 7;
    const int src = row_index ? row_index[row] : row;
    const bf16* xr = x + (size_t)src * d;
    float v[MAXV][4];
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; i++)
        if (i < nv) {
            const uint2 u = ld8(xr + i * 128 + lane * 4);
            const float2 a = unpack_bf16x2(u.x), c = unpack_bf16x2(u.y);
            v[i][0] = a.x; v[i][1] = a.y; v[i][2] = c.x; v[i][3] = c.y;
            q = fmaf(a.x, a.x, q); q = fmaf(a.y, a.y, q); q = fmaf(c.x, c.x, q); q = fmaf(c.y, c.y, q);
        }
    const float r = rsqrtf(warp_sum(q) / (float)d + eps);
    bf16* yr = y + (size_t)row * d;
#pragma unroll
    for (int i = 0; i < MAXV; i++)
        if (i < nv) {
            const int c0 = i * 128 + lane * 4;
            const uint2 wu = ld8(w + c0);
            const float2 w0 = unpack_bf16x2(wu.x), w1 = unpack_bf16x2(wu.y);
            st8(yr + c0, v[i][0] * r * w0.x, v[i][1] * r * w0.y, v[i][2] * r * w1.x, v[i][3] * r * w1.y);
        }
}

// ------------------------------------------------------------------------------------------
__global__ void embed_splice_kernel(const int32_t* __restrict__ ids, const int* __restrict__ audio_src, const bf16* __restrict__ embed,
                                    const bf16* __restrict__ audio, bf16* __restrict__ x, int rows, int h) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    const int vec = h >> 3;  // 16-byte vectors per row
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long)rows * vec) return;
    const int r = (int)(idx / vec), c = (int)(idx % vec);
    const int a = audio_src ? audio_src[r] : -1;
    const bf16* src = a >= 0 ? audio + (size_t)a * h : embed + (size_t)ids[r] * h;
    reinterpret_cast<uint4*>(x + (size_t)r * h)[c] = __ldg(reinterpret_cast<const uint4*>(src) + c);
}

// ------------------------------------------------------------------------------------------
// q/k RMSNorm + RoPE + KV write.  One warp per (row, head slot); head_dim == 128 (4 dims per lane).
// slots [0, heads) = q, [heads, heads+kvh) = k, [heads+kvh, heads+2kvh) = v.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) qknorm_rope_kv_kernel(const bf16* __restrict__ qkv, int ld, const bf16* __restrict__ qw,
                                                            const bf16* __restrict__ kw, const int* __restrict__ pos,
                                                            const int* __restrict__ row_seq, int rows, int heads, int kv_heads, float eps,
                                                            const float2* __restrict__ rope_tab, bf16* __restrict__ qout,
                                                            bf16* __restrict__ kc, bf16* __restrict__ vc, KvCache cache, int layer) {
    // one CTA per row, 8 warps; warp w takes head slots w, w + 8, ... so the row's position, page and table entries are
    // fetched once per warp (the kernel is instruction-bound when every (row, slot) pair recomputes them)
    const int row = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slots = heads + 2 * kv_heads;
    const int d0 = lane * 4;
    const int p = pos[row];
    const int seq = row_seq[row];
    const int page = cache.page_table[(size_t)seq * cache.max_pages + p / KV_PAGE];
    bf16* page_base = cache.pool + (((size_t)page * cache.layers + layer) * 2) * cache.kv_heads * (KV_PAGE * 128) + (p % KV_PAGE) * 128 + d0;
    const float4* tp = reinterpret_cast<const float4*>(rope_tab + (size_t)p * 64 + (d0 & 63));  // (cos, sin) pairs of 4 dims
    const float4 t0 = __ldg(tp), t1 = __ldg(tp + 1);
    const float cs[4] = {t0.x, t0.z, t1.x, t1.z}, sn[4] = {t0.y, t0.w, t1.y, t1.w};
    const float sgn = lane < 16 ? -1.f : 1.f;
    const uint2 qwu = ld8(qw + d0), kwu = ld8(kw + d0);
    const bf16* src = qkv + (size_t)row * ld + d0;
    for (int slot = warp; slot < slots; slot += 8) {
        const uint2 u = ld8(src + slot * 128);
        const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
        float x[4] = {a.x, a.y, b.x, b.y};
        const bool is_v = slot >= heads + kv_heads;
        if (!is_v) {
            float q = fmaf(x[0], x[0], fmaf(x[1], x[1], fmaf(x[2], x[2], x[3] * x[3])));
            const float r = rsqrtf(warp_sum(q) * (1.0f / 128.0f) + eps);
            const uint2 wu = slot < heads ? qwu : kwu;
            const float2 w0 = unpack_bf16x2(wu.x), w1 = unpack_bf16x2(wu.y);
            x[0] = bf16_round(x[0] * r * w0.x);
            x[1] = bf16_round(x[1] * r * w0.y);
            x[2] = bf16_round(x[2] * r * w1.x);
            x[3] = bf16_round(x[3] * r * w1.y);
            // split-half rotation: dims (i, i+64); the partner values live in lane ^ 16
            float y[4];
#pragma unroll
            for (int j = 0; j < 4; j++) y[j] = __shfl_xor_sync(0xffffffffu, x[j], 16);
#pragma unroll
            for (int j = 0; j < 4; j++) x[j] = fmaf(x[j], cs[j], sgn * y[j] * sn[j]);
        }
        if (slot < heads) {
            st8(qout + (size_t)row * heads * 128 + slot * 128 + d0, x[0], x[1], x[2], x[3]);
            continue;
        }
        const int kvh = is_v ? slot - heads - kv_heads : slot - heads;
        bf16* cont = is_v ? vc : kc;
        if (cont) st8(cont + (size_t)row * kv_heads * 128 + kvh * 128 + d0, x[0], x[1], x[2], x[3]);
        st8(page_base + ((size_t)(is_v ? 1 : 0) * cache.kv_heads + kvh) * (KV_PAGE * 128), x[0], x[1], x[2], x[3]);
    }
}

// ------------------------------------------------------------------------------------------
// Paged decode attention: one CTA per (sequence, kv head), 4 warps; a warp scores 4 keys at a time
// (8 lanes x 16 dims each), online softmax per lane group, groups merged through shared memory.
// ------------------------------------------------------------------------------------------
template <int GROUP>
__global__ void __launch_bounds__(128) decode_attn_kernel(const bf16* __restrict__ q, KvCache cache, int layer,
                                                         const int* __restrict__ kv_len, int heads, float scale_log2,
                                                         bf16* __restrict__ out) {
    const int seq = blockIdx.x, kvh = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane >> 3, sub = lane & 7;  // key slot within the warp, 16-dim slice
    const int len = kv_len[seq];
    float qf[GROUP][16];
#pragma unroll
    for (int g = 0; g < GROUP; g++) {
        const bf16* qp = q + ((size_t)seq * heads + kvh * GROUP + g) * 128 + sub * 16;
        const uint4 u0 = *reinterpret_cast<const uint4*>(qp), u1 = *reinterpret_cast<const uint4*>(qp + 8);
        const uint32_t w[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const float2 f = unpack_bf16x2(w[j]);
            qf[g][2 * j] = f.x;
            qf[g][2 * j + 1] = f.y;
        }
    }
    float m[GROUP], l[GROUP], acc[GROUP][16];
#pragma unroll
    for (int g = 0; g < GROUP; g++) {
        m[g] = -INFINITY;
        l[g] = 0.f;
#pragma unroll
        for (int j = 0; j < 16; j++) acc[g][j] = 0.f;
    }
    const int* pt = cache.page_table + (size_t)seq * cache.max_pages;
    for (int j0 = warp * 4; j0 < len; j0 += 16) {
        const int j = j0 + grp;
        const bool ok = j < len;
        float kf[16], vf[16];
        if (ok) {
            const int page = pt[j / KV_PAGE];
            const bf16* kp = cache.pool + ((((size_t)page * cache.layers + layer) * 2) * cache.kv_heads + kvh) * (KV_PAGE * 128) +
                             (j % KV_PAGE) * 128 + sub * 16;
            const bf16* vp = kp + (size_t)cache.kv_heads * (KV_PAGE * 128);
            const uint4 k0 = *reinterpret_cast<const uint4*>(kp), k1 = *reinterpret_cast<const uint4*>(kp + 8);
            const uint4 v0 = *reinterpret_cast<const uint4*>(vp), v1 = *reinterpret_cast<const uint4*>(vp + 8);
            const uint32_t kw[8] = {k0.x, k0.y, k0.z, k0.w, k1.x, k1.y, k1.z, k1.w};
            const uint32_t vw[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
            for (int t = 0; t < 8; t++) {
                const float2 a = unpack_bf16x2(kw[t]), b = unpack_bf16x2(vw[t]);
                kf[2 * t] = a.x; kf[2 * t + 1] = a.y;
                vf[2 * t] = b.x; vf[2 * t + 1] = b.y;
            }
        } else {
#pragma unroll
            for (int t = 0; t < 16; t++) { kf[t] = 0.f; vf[t] = 0.f; }
        }
#pragma unroll
        for (int g = 0; g < GROUP; g++) {
            float s = 0.f;
#pragma unroll
            for (int t = 0; t < 16; t++) s = fmaf(qf[g][t], kf[t], s);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            s = ok ? s * scale_log2 : -INFINITY;
            const float mn = fmaxf(m[g], s);
            const float alpha = mn == -INFINITY ? 1.f : exp2f(m[g] - mn);
            const float pj = mn == -INFINITY ? 0.f : exp2f(s - mn);
            l[g] = l[g] * alpha + pj;
            const float pb = bf16_round(pj);
#pragma unroll
            for (int t = 0; t < 16; t++) acc[g][t] = fmaf(pb, vf[t], acc[g][t] * alpha);
            m[g] = mn;
        }
    }
    // merge the 16 (warp, group) partials per head
    __shared__ float s_m[GROUP][16], s_l[GROUP][16];
    __shared__ float s_acc[GROUP][16][128];
#pragma unroll
    for (int g = 0; g < GROUP; g++) {
        if (sub == 0) { s_m[g][warp * 4 + grp] = m[g]; s_l[g][warp * 4 + grp] = l[g]; }
#pragma unroll
        for (int t = 0; t < 16; t++) s_acc[g][warp * 4 + grp][sub * 16 + t] = acc[g][t];
    }
    __syncthreads();
    for (int g = 0; g < GROUP; g++) {
        const int d = threadIdx.x;  // 128 threads = 128 dims
        float mm = -INFINITY;
#pragma unroll
        for (int i = 0; i < 16; i++) mm = fmaxf(mm, s_m[g][i]);
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const float f = s_m[g][i] == -INFINITY ? 0.f : exp2f(s_m[g][i] - mm);
            num = fmaf(f, s_acc[g][i][d], num);
            den = fmaf(f, s_l[g][i], den);
        }
        out[((size_t)seq * heads + kvh * GROUP + g) * 128 + d] = __float2bfloat16_rn(num / den);
    }
}

// ------------------------------------------------------------------------------------------
// Fused decode-step attention: one CTA per (sequence, kv head), NW warps.
//   1. q (GROUP heads), k, v of the new token = fixed-order sum of the split-K fp32 partials of the QKV
//      product, rounded to bf16 (the oracle's rounding point); per-head RMSNorm + split-half RoPE on q and k
//      (same arithmetic as qknorm_rope_kv_kernel); k and v are appended to the paged cache.
//   2. the query heads attend over kv_len keys (the new one included): a warp scores 8 keys per iteration
//      (4 lane groups x 2 keys in flight, 8 lanes x 16 dims each), online softmax per lane group.
//   3. lane groups are merged with shuffles, warps through shared memory.
// FloatTextDecoder.swift:77-107 (q/k/v, q_norm/k_norm, rope, cache update, attention) for seqLen == 1.
// ------------------------------------------------------------------------------------------
constexpr int DA_CHUNK = 8;   // keys per warp step
constexpr int DA_STAGES = 3;  // cp.async ring depth per warp
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "r"(src_bytes)
                 : "memory");
}
constexpr int decode_attn_smem(int nw) { return nw * DA_STAGES * 2 * DA_CHUNK * 128 * 2; }

template <int GROUP, int NW>
__global__ void __launch_bounds__(NW * 32, NW == 4 ? 4 : 1) decode_attn_fused_kernel(const float* __restrict__ qkv_part, int splits, long long split_stride,
                                                                    int nqkv, const bf16* __restrict__ qw, const bf16* __restrict__ kw,
                                                                    const int* __restrict__ pos, float eps,
                                                                    const float2* __restrict__ rope_tab, KvCache cache, int layer,
                                                                    const int* __restrict__ kv_len, int heads, float scale_log2,
                                                                    bf16* __restrict__ out) {
    ptx::grid_dep_launch();
    const int seq = blockIdx.x, kvh = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ float s_q[GROUP][128];
    __shared__ __align__(16) bf16 s_new[2][128];  // the new token's k and v rows
    __shared__ float s_m[GROUP][NW], s_l[GROUP][NW];
    __shared__ float s_acc[GROUP][NW][128];
    const int* pt = cache.page_table + (size_t)seq * cache.max_pages;

    // ---- 0. start streaming the cached keys/values: each warp owns a cp.async ring of 8-key chunks (K and V rows are
    //         contiguous inside a page).  Nothing here depends on the previous kernel, so it runs ahead of the
    //         programmatic-dependency wait; the row of the new token (position len - 1) is patched in from shared memory. ----
    const int len = kv_len[seq];
    extern __shared__ uint4 da_smem[];
    bf16* ring = reinterpret_cast<bf16*>(da_smem) + (size_t)warp * DA_STAGES * 2 * DA_CHUNK * 128;
    const size_t head_off = (((size_t)layer * 2) * cache.kv_heads + kvh) * (KV_PAGE * 128);
    const size_t page_elems = (size_t)cache.layers * 2 * cache.kv_heads * (KV_PAGE * 128);
    const size_t v_off = (size_t)cache.kv_heads * (KV_PAGE * 128);
    const int n_chunks = (len + DA_CHUNK - 1) / DA_CHUNK;
    auto issue = [&](int chunk, int stage) {
        if (chunk < n_chunks) {
            const int j0 = chunk * DA_CHUNK;
            const bf16* kb = cache.pool + (size_t)pt[j0 / KV_PAGE] * page_elems + head_off + (j0 % KV_PAGE) * 128;
            bf16* sk = ring + (size_t)stage * 2 * DA_CHUNK * 128;
#pragma unroll
            for (int i = 0; i < DA_CHUNK * 16 / 32; i++) {
                const int seg = i * 32 + lane;  // 16-byte segment of the chunk; key = seg / 16
                const uint32_t n = j0 + (seg >> 4) < len ? 16u : 0u;  // rows past the end are zero-filled
                cp_async16(sk + seg * 8, kb + seg * 8, n);
                cp_async16(sk + DA_CHUNK * 128 + seg * 8, kb + v_off + seg * 8, n);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
#pragma unroll
    for (int s = 0; s < DA_STAGES - 1; s++) issue(warp + s * NW, s);

    ptx::grid_dep_wait();

    // ---- 1. new-token q / k / v ----
    if (warp < GROUP + 2) {
        const int slot = warp;  // 0..GROUP-1 = q heads, GROUP = k, GROUP+1 = v
        const int d0 = lane * 4;
        const int col = slot < GROUP ? (kvh * GROUP + slot) * 128
                                     : slot == GROUP ? heads * 128 + kvh * 128 : (heads + cache.kv_heads) * 128 + kvh * 128;
        const float* src = qkv_part + (size_t)seq * nqkv + col + d0;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int s0 = 0; s0 < splits; s0 += 4) {  // fixed summation order, four loads in flight
            float4 b[4];
#pragma unroll
            for (int i = 0; i < 4; i++)
                b[i] = s0 + i < splits ? *reinterpret_cast<const float4*>(src + (size_t)(s0 + i) * split_stride) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; i++) { a.x += b[i].x; a.y += b[i].y; a.z += b[i].z; a.w += b[i].w; }
        }
        float x[4] = {bf16_round(a.x), bf16_round(a.y), bf16_round(a.z), bf16_round(a.w)};
        const int p = pos[seq];
        if (slot <= GROUP) {
            float q = fmaf(x[0], x[0], fmaf(x[1], x[1], fmaf(x[2], x[2], x[3] * x[3])));
            const float r = rsqrtf(warp_sum(q) * (1.0f / 128.0f) + eps);
            const uint2 wu = ld8((slot < GROUP ? qw : kw) + d0);
            const float2 w0 = unpack_bf16x2(wu.x), w1 = unpack_bf16x2(wu.y);
            x[0] = bf16_round(x[0] * r * w0.x);
            x[1] = bf16_round(x[1] * r * w0.y);
            x[2] = bf16_round(x[2] * r * w1.x);
            x[3] = bf16_round(x[3] * r * w1.y);
            float y[4];
#pragma unroll
            for (int j = 0; j < 4; j++) y[j] = __shfl_xor_sync(0xffffffffu, x[j], 16);
            const int i0 = d0 & 63;
            const float sgn = lane < 16 ? -1.f : 1.f;
            const float4* tp = reinterpret_cast<const float4*>(rope_tab + (size_t)p * 64 + i0);  // (cos, sin) pairs of 4 dims
            const float4 t0 = __ldg(tp), t1 = __ldg(tp + 1);
            const float cs[4] = {t0.x, t0.z, t1.x, t1.z}, sn[4] = {t0.y, t0.w, t1.y, t1.w};
#pragma unroll
            for (int j = 0; j < 4; j++) x[j] = bf16_round(fmaf(x[j], cs[j], sgn * y[j] * sn[j]));
        }
        if (slot < GROUP) {
#pragma unroll
            for (int j = 0; j < 4; j++) s_q[slot][d0 + j] = x[j];
        } else {
            const int page = pt[p / KV_PAGE];
            bf16* dst = cache.pool + ((((size_t)page * cache.layers + layer) * 2 + (slot == GROUP ? 0 : 1)) * cache.kv_heads + kvh) * (KV_PAGE * 128) +
                        (p % KV_PAGE) * 128 + d0;
            st8(dst, x[0], x[1], x[2], x[3]);
            st8(&s_new[slot - GROUP][d0], x[0], x[1], x[2], x[3]);
        }
    }
    __syncthreads();  // s_q and s_new ready

    // ---- 2. attention ----
    const int grp = lane >> 3, sub = lane & 7;
    // lane `sub` owns dims [8 sub, 8 sub + 8) and [64 + 8 sub, 64 + 8 sub + 8): a lane group reads 128 contiguous bytes
    float qf[GROUP][16];
#pragma unroll
    for (int g = 0; g < GROUP; g++)
#pragma unroll
        for (int t = 0; t < 16; t++) qf[g][t] = s_q[g][(t >> 3) * 64 + sub * 8 + (t & 7)];
    float m[GROUP], l[GROUP], acc[GROUP][16];
#pragma unroll
    for (int g = 0; g < GROUP; g++) {
        m[g] = -INFINITY;
        l[g] = 0.f;
#pragma unroll
        for (int t = 0; t < 16; t++) acc[g][t] = 0.f;
    }
    int stage = 0;
    for (int chunk = warp; chunk < n_chunks; chunk += NW) {
        issue(chunk + (DA_STAGES - 1) * NW, (stage + DA_STAGES - 1) % DA_STAGES);
        asm volatile("cp.async.wait_group %0;" ::"n"(DA_STAGES - 1) : "memory");
        __syncwarp();
        bf16* sk = ring + (size_t)stage * 2 * DA_CHUNK * 128;
        const int j0 = chunk * DA_CHUNK;
        if (chunk == n_chunks - 1) {  // the prefetch may have read the new token's row before it was written
            const int row = (len - 1) - j0;
            reinterpret_cast<uint4*>(sk + (lane >> 4) * DA_CHUNK * 128 + row * 128)[lane & 15] = reinterpret_cast<const uint4*>(s_new[lane >> 4])[lane & 15];
            __syncwarp();
        }
        // scores of the chunk's two keys per lane group, then one running-max update for both
        float sc[GROUP][2];
        uint32_t vraw[2][8];
#pragma unroll
        for (int u = 0; u < DA_CHUNK / 4; u++) {
            const int key = u * 4 + grp;
            const bool ok = j0 + key < len;
            const uint4 k0 = *reinterpret_cast<const uint4*>(sk + key * 128 + sub * 8);
            const uint4 k1 = *reinterpret_cast<const uint4*>(sk + key * 128 + 64 + sub * 8);
            const uint4 v0 = *reinterpret_cast<const uint4*>(sk + DA_CHUNK * 128 + key * 128 + sub * 8);
            const uint4 v1 = *reinterpret_cast<const uint4*>(sk + DA_CHUNK * 128 + key * 128 + 64 + sub * 8);
            const uint32_t kw32[8] = {k0.x, k0.y, k0.z, k0.w, k1.x, k1.y, k1.z, k1.w};
            vraw[u][0] = v0.x; vraw[u][1] = v0.y; vraw[u][2] = v0.z; vraw[u][3] = v0.w;
            vraw[u][4] = v1.x; vraw[u][5] = v1.y; vraw[u][6] = v1.z; vraw[u][7] = v1.w;
            float s[GROUP];
#pragma unroll
            for (int g = 0; g < GROUP; g++) s[g] = 0.f;
#pragma unroll
            for (int t = 0; t < 8; t++) {
                const float2 kk = unpack_bf16x2(kw32[t]);
#pragma unroll
                for (int g = 0; g < GROUP; g++) s[g] = fmaf(qf[g][2 * t + 1], kk.y, fmaf(qf[g][2 * t], kk.x, s[g]));
            }
#pragma unroll
            for (int g = 0; g < GROUP; g++) {
                s[g] += __shfl_xor_sync(0xffffffffu, s[g], 1);
                s[g] += __shfl_xor_sync(0xffffffffu, s[g], 2);
                s[g] += __shfl_xor_sync(0xffffffffu, s[g], 4);
                sc[g][u] = ok ? s[g] * scale_log2 : -INFINITY;
            }
        }
        float b0[GROUP], b1[GROUP];
#pragma unroll
        for (int g = 0; g < GROUP; g++) {
            const float mn = fmaxf(m[g], fmaxf(sc[g][0], sc[g][1]));
            const float alpha = mn == -INFINITY ? 1.f : exp2f(m[g] - mn);
            const float p0 = mn == -INFINITY ? 0.f : exp2f(sc[g][0] - mn);
            const float p1 = mn == -INFINITY ? 0.f : exp2f(sc[g][1] - mn);
            l[g] = l[g] * alpha + (p0 + p1);
            b0[g] = bf16_round(p0);
            b1[g] = bf16_round(p1);
            m[g] = mn;
#pragma unroll
            for (int t = 0; t < 16; t++) acc[g][t] *= alpha;
        }
#pragma unroll
        for (int t = 0; t < 8; t++) {
            const float2 va = unpack_bf16x2(vraw[0][t]), vb = unpack_bf16x2(vraw[1][t]);
#pragma unroll
            for (int g = 0; g < GROUP; g++) {
                acc[g][2 * t] = fmaf(b1[g], vb.x, fmaf(b0[g], va.x, acc[g][2 * t]));
                acc[g][2 * t + 1] = fmaf(b1[g], vb.y, fmaf(b0[g], va.y, acc[g][2 * t + 1]));
            }
        }
        __syncwarp();  // the slot is refilled by the next iteration's issue
        stage = (stage + 1) % DA_STAGES;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    // ---- 3. merge the four lane groups of the warp, then the warps ----
#pragma unroll
    for (int g = 0; g < GROUP; g++) {
#pragma unroll
        for (int off = 8; off <= 16; off <<= 1) {
            const float mo = __shfl_xor_sync(0xffffffffu, m[g], off);
            const float lo = __shfl_xor_sync(0xffffffffu, l[g], off);
            const float mn = fmaxf(m[g], mo);
            const float a = mn == -INFINITY ? 1.f : exp2f(m[g] - mn);
            const float b = mn == -INFINITY ? 0.f : exp2f(mo - mn);
            l[g] = l[g] * a + lo * b;
#pragma unroll
            for (int t = 0; t < 16; t++) {
                const float ao = __shfl_xor_sync(0xffffffffu, acc[g][t], off);
                acc[g][t] = acc[g][t] * a + ao * b;
            }
            m[g] = mn;
        }
        if (grp == 0) {
            if (sub == 0) { s_m[g][warp] = m[g]; s_l[g][warp] = l[g]; }
#pragma unroll
            for (int t = 0; t < 16; t++) s_acc[g][warp][(t >> 3) * 64 + sub * 8 + (t & 7)] = acc[g][t];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < GROUP * 128; i += NW * 32) {
        const int g = i >> 7, d = i & 127;
        float mm = -INFINITY;
#pragma unroll
        for (int w = 0; w < NW; w++) mm = fmaxf(mm, s_m[g][w]);
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int w = 0; w < NW; w++) {
            const float f = s_m[g][w] == -INFINITY ? 0.f : exp2f(s_m[g][w] - mm);
            num = fmaf(f, s_acc[g][w][d], num);
            den = fmaf(f, s_l[g][w], den);
        }
        out[((size_t)seq * heads + kvh * GROUP + g) * 128 + d] = __float2bfloat16_rn(num / den);
    }
}

// ------------------------------------------------------------------------------------------
// Fused decode-step attention, tensor-core version (the default): same contract as decode_attn_fused_kernel, but the
// two query heads of a kv head form rows 0 and 1 of an m16n8k16 tile, so a warp scores a 16-key chunk with 16 mma.sync
// and accumulates P V with 16 more — about a fifth of the CUDA-core instruction count, which leaves the kernel bound by
// the KV stream.  Each warp owns a 3-deep cp.async ring of 16-key chunks (K and V rows are contiguous in a page); rows are
// stored with a 16-byte XOR swizzle so ldmatrix is conflict-free without padding.
// ------------------------------------------------------------------------------------------
constexpr int DM_CHUNK = 16;
constexpr int DM_STAGES = 3;
constexpr int DM_STREAMS = 8;  // canonical number of key streams (see the kernel)

// scales of the online-softmax merge of two partials with maxima am, bm: returns max(am, bm), *fa = 2^(am - m), *fb = 2^(bm - m)
// (0 for an empty partial, whose maximum is -inf)
__device__ __forceinline__ float dm_merge_scales(float am, float bm, float* fa, float* fb) {
    const float m = fmaxf(am, bm);
    *fa = am == -INFINITY ? 0.f : exp2f(am - m);
    *fb = bm == -INFINITY ? 0.f : exp2f(bm - m);
    return m;
}
constexpr int decode_attn_mma_smem(int nw) { return nw * DM_STAGES * 2 * DM_CHUNK * 128 * 2; }

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* smem_ptr) {
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(smem_ptr));
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const void* smem_ptr) {
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(smem_ptr));
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(a));
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// element offset of 16-byte segment `seg` of row `key` in a swizzled [16 keys][128] tile
__device__ __forceinline__ int dm_off(int key, int seg) { return key * 128 + ((seg ^ (key & 7)) << 3); }

// SPLIT (NW == 1, opt-in: Q3ASR_DECODE_ATTN_WARPS=1): the (sequence, kv head) item is shared by the two single-warp CTAs blockIdx.z = 0 / 1,
// which walk the even / the odd key streams — exactly what warps 0 and 1 of the two-warp variant do — and meet through global
// memory: each stores its partial (maximum, sum, accumulator), bumps the item's counter, and whichever arrives second merges
// even + odd in that fixed order, so the result is bit-identical to the other variants and independent of the arrival order.
// Built to even out the tail (two-warp CTAs at four per SM leave 3 or 4 items per SM at 64 sequences); measured slower, see the launcher.
constexpr int DM_PART_STRIDE = 264;  // floats per stored partial: [2][128] accumulators, 2 maxima, 2 sums, padding
template <int NW, bool SPLIT>
__global__ void __launch_bounds__(NW * 32, SPLIT ? 8 : NW == 2 ? 4 : 1) decode_attn_mma_kernel(const float* __restrict__ qkv_part, int splits, long long split_stride,
                                                                  int nqkv, const bf16* __restrict__ qw, const bf16* __restrict__ kw,
                                                                  const int* __restrict__ pos, float eps,
                                                                  const float2* __restrict__ rope_tab, KvCache cache, int layer,
                                                                  const int* __restrict__ kv_len, int heads, float scale_log2,
                                                                  bf16* __restrict__ out, float* __restrict__ split_part, int* __restrict__ split_cnt) {
    static_assert(!SPLIT || NW == 1, "the split variant is one warp per CTA");
    constexpr int GROUP = 2;
    constexpr int SW = SPLIT ? 2 : NW;  // this CTA's warps walk the streams sw0, sw0 + SW, ...
    ptx::grid_dep_launch();
    const int seq = blockIdx.x, kvh = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int half = SPLIT ? (int)blockIdx.z : 0;
    const int sw0 = SPLIT ? half : warp;
    __shared__ __align__(16) bf16 s_qb[GROUP][128];  // the two query heads (bf16, after norm + RoPE)
    __shared__ __align__(16) bf16 s_new[2][128];     // the new token's k and v rows
    __shared__ float s_m[GROUP][NW], s_l[GROUP][NW];
    __shared__ float s_acc[GROUP][NW][128];
    const int* pt = cache.page_table + (size_t)seq * cache.max_pages;

    // ---- 0. start streaming cached keys/values (independent of the previous kernel) ----
    const int len = kv_len[seq];
    extern __shared__ uint4 da_smem[];
    bf16* ring = reinterpret_cast<bf16*>(da_smem) + (size_t)warp * DM_STAGES * 2 * DM_CHUNK * 128;
    const size_t head_off = (((size_t)layer * 2) * cache.kv_heads + kvh) * (KV_PAGE * 128);
    const size_t page_elems = (size_t)cache.layers * 2 * cache.kv_heads * (KV_PAGE * 128);
    const size_t v_off = (size_t)cache.kv_heads * (KV_PAGE * 128);
    const int n_chunks = (len + DM_CHUNK - 1) / DM_CHUNK;
    auto issue = [&](int chunk, int stage) {
        if (chunk < n_chunks) {
            const int j0 = chunk * DM_CHUNK;
            const bf16* kb = cache.pool + (size_t)pt[j0 / KV_PAGE] * page_elems + head_off + (j0 % KV_PAGE) * 128;
            bf16* sk = ring + (size_t)stage * 2 * DM_CHUNK * 128;
#pragma unroll
            for (int i = 0; i < DM_CHUNK * 16 / 32; i++) {
                const int lin = i * 32 + lane, key = lin >> 4, seg = lin & 15;
                const uint32_t n = j0 + key < len ? 16u : 0u;  // rows past the end are zero-filled
                cp_async16(sk + dm_off(key, seg), kb + lin * 8, n);
                cp_async16(sk + DM_CHUNK * 128 + dm_off(key, seg), kb + v_off + lin * 8, n);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // Canonical key partition (independent of NW, so a sequence's result does not depend on the batch it is decoded in): chunk c
    // belongs to stream c % DM_STREAMS; a stream is accumulated in chunk order; streams are merged by dm_merge as
    // ((s0 + s2) + s4) + s6, ((s1 + s3) + s5) + s7, then even + odd.  Warp w walks the streams w, w + NW, ... one after the other.
    auto seq_next = [&](int& sj, int& sc) {  // next chunk of this warp's sequence after (stream sj, chunk sc); sc >= n_chunks: done
        sc += DM_STREAMS;
        while (sc >= n_chunks && sj + SW < DM_STREAMS) {
            sj += SW;
            sc = sj;
        }
    };
    int ij = sw0, ic = sw0;  // issue cursor
    while (ic >= n_chunks && ij + SW < DM_STREAMS) { ij += SW; ic = ij; }
#pragma unroll
    for (int s = 0; s < DM_STAGES - 1; s++) {
        issue(ic, s);  // chunks >= n_chunks are skipped inside issue (the group is still committed)
        seq_next(ij, ic);
    }

    ptx::grid_dep_wait();

    // ---- 1. new-token q / k / v (slots 0,1 = q heads, 2 = k, 3 = v): one half-warp per slot, 8 dims per lane, so all four
    //         are done in one pass by the first two warps (the other warps keep their prefetches in flight) ----
    // (split variant: 32 threads, two passes — the queries, then k and v, which only the CTA that appends them to the cache (half 0)
    // or owns the last chunk needs)
    const bool need_kv = !SPLIT || half == 0 || (((n_chunks - 1) % DM_STREAMS) & 1) == half;
    for (int vt = threadIdx.x; vt < 16 * (GROUP + 2) && (vt < 16 * GROUP || need_kv); vt += NW * 32) {
        const int slot = vt >> 4, hl = vt & 15;
        const unsigned half_mask = 0xffffu << (threadIdx.x & 16);  // the two halves of a warp hold different slots and diverge (v skips the norm)
        const int d0 = hl * 8;
        const int col = slot < GROUP ? (kvh * GROUP + slot) * 128
                                     : slot == GROUP ? heads * 128 + kvh * 128 : (heads + cache.kv_heads) * 128 + kvh * 128;
        const float* src = qkv_part + (size_t)seq * nqkv + col + d0;
        float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int s0 = 0; s0 < splits; s0 += 4) {  // fixed summation order, eight loads in flight
            float4 b[4][2];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const bool on = s0 + i < splits;
                const float4* sp = reinterpret_cast<const float4*>(src + (size_t)(s0 + i) * split_stride);
                b[i][0] = on ? sp[0] : make_float4(0.f, 0.f, 0.f, 0.f);
                b[i][1] = on ? sp[1] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                x[0] += b[i][0].x; x[1] += b[i][0].y; x[2] += b[i][0].z; x[3] += b[i][0].w;
                x[4] += b[i][1].x; x[5] += b[i][1].y; x[6] += b[i][1].z; x[7] += b[i][1].w;
            }
        }
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = bf16_round(x[j]);
        const int p = pos[seq];
        if (slot <= GROUP) {
            float q = 0.f;
#pragma unroll
            for (int j = 0; j < 8; j++) q = fmaf(x[j], x[j], q);
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) q += __shfl_xor_sync(half_mask, q, o);  // stays inside the half-warp
            const float r = rsqrtf(q * (1.0f / 128.0f) + eps);
            const uint4 wu = *reinterpret_cast<const uint4*>((slot < GROUP ? qw : kw) + d0);
            const uint32_t ww[4] = {wu.x, wu.y, wu.z, wu.w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float2 wf = unpack_bf16x2(ww[j]);
                x[2 * j] = bf16_round(x[2 * j] * r * wf.x);
                x[2 * j + 1] = bf16_round(x[2 * j + 1] * r * wf.y);
            }
            // split-half rotation: dims (i, i+64); the partner values live 8 lanes away
            float y[8];
#pragma unroll
            for (int j = 0; j < 8; j++) y[j] = __shfl_xor_sync(half_mask, x[j], 8);
            const float sgn = hl < 8 ? -1.f : 1.f;
            const float4* tp = reinterpret_cast<const float4*>(rope_tab + (size_t)p * 64 + (d0 & 63));  // (cos, sin) pairs
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float4 t = __ldg(tp + j);
                x[2 * j] = fmaf(x[2 * j], t.x, sgn * y[2 * j] * t.y);
                x[2 * j + 1] = fmaf(x[2 * j + 1], t.z, sgn * y[2 * j + 1] * t.w);
            }
        }
        const uint4 packed = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
        if (slot < GROUP) {
            *reinterpret_cast<uint4*>(&s_qb[slot][d0]) = packed;
        } else {
            const int page = pt[p / KV_PAGE];
            bf16* dst = cache.pool + ((((size_t)page * cache.layers + layer) * 2 + (slot == GROUP ? 0 : 1)) * cache.kv_heads + kvh) * (KV_PAGE * 128) +
                        (p % KV_PAGE) * 128 + d0;
            if (half == 0) *reinterpret_cast<uint4*>(dst) = packed;
            *reinterpret_cast<uint4*>(&s_new[slot - GROUP][d0]) = packed;
        }
    }
    __syncthreads();  // s_qb and s_new ready

    // ---- 2. attention on the tensor cores ----
    const int g = lane >> 2, t = lane & 3;  // accumulator row (query head when < 2) and column pair
    uint32_t qa[8][2];                      // A fragments of Q: rows 0,1 real, the rest zero
#pragma unroll
    for (int ks = 0; ks < 8; ks++) {
        qa[ks][0] = lane < 8 ? *reinterpret_cast<const uint32_t*>(&s_qb[g & 1][ks * 16 + t * 2]) : 0u;
        qa[ks][1] = lane < 8 ? *reinterpret_cast<const uint32_t*>(&s_qb[g & 1][ks * 16 + 8 + t * 2]) : 0u;
    }
    float o[16][4];
    float m_run = -INFINITY, l_run = 0.f;
    const int mi = lane >> 3, r8 = lane & 7;
    int stage = 0;
    int cj = sw0, chunk = sw0;  // consume cursor
    while (chunk >= n_chunks && cj + SW < DM_STREAMS) { cj += SW; chunk = cj; }
    int cur_stream = -1;
    bool first_stream = true;
    // folds the finished stream (m_run, l_run, o) into this warp's running partial in shared memory (lanes 0-7 hold the two rows)
    auto flush_stream = [&]() {
        float l = l_run;
        l += __shfl_xor_sync(0xffffffffu, l, 1);
        l += __shfl_xor_sync(0xffffffffu, l, 2);
        if (lane < 8) {
            float am = first_stream ? -INFINITY : s_m[g][warp], al = first_stream ? 0.f : s_l[g][warp];
            float fa, fb;
            const float mm = dm_merge_scales(am, m_run, &fa, &fb);
#pragma unroll
            for (int nt = 0; nt < 16; nt++) {
                float* dst = &s_acc[g][warp][nt * 8 + t * 2];
                const float a0 = first_stream ? 0.f : dst[0], a1 = first_stream ? 0.f : dst[1];
                dst[0] = fmaf(fb, o[nt][0], fa * a0);
                dst[1] = fmaf(fb, o[nt][1], fa * a1);
            }
            __syncwarp(0xffu);
            if (t == 0) { s_m[g][warp] = mm; s_l[g][warp] = fmaf(fb, l, fa * al); }
        }
        first_stream = false;
    };
    for (; chunk < n_chunks; seq_next(cj, chunk)) {
        if (cj != cur_stream) {  // a new stream starts: fold the previous one away, start from an empty accumulator
            if (cur_stream >= 0) flush_stream();
            cur_stream = cj;
#pragma unroll
            for (int i = 0; i < 16; i++) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
            m_run = -INFINITY;
            l_run = 0.f;
        }
        issue(ic, (stage + DM_STAGES - 1) % DM_STAGES);
        seq_next(ij, ic);
        asm volatile("cp.async.wait_group %0;" ::"n"(DM_STAGES - 1) : "memory");
        __syncwarp();
        bf16* sk = ring + (size_t)stage * 2 * DM_CHUNK * 128;
        bf16* sv = sk + DM_CHUNK * 128;
        const int j0 = chunk * DM_CHUNK;
        if (chunk == n_chunks - 1) {  // the prefetch may have read the new token's row before it was written
            const int row = (len - 1) - j0;
            *reinterpret_cast<uint4*>((lane < 16 ? sk : sv) + dm_off(row, lane & 15)) = reinterpret_cast<const uint4*>(s_new[lane >> 4])[lane & 15];
            __syncwarp();
        }
        // S = Q K^T: 16 (2 real) x 16 keys
        float s[2][4];
#pragma unroll
        for (int i = 0; i < 2; i++) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 8; ks++) {
            uint32_t b[4];
            const int key = (mi >> 1) * 8 + r8;
            ldsm_x4(b, sk + dm_off(key, ks * 2 + (mi & 1)));
            const uint32_t a[4] = {qa[ks][0], 0u, qa[ks][1], 0u};
            mma16816(s[0], a, b[0], b[1]);
            mma16816(s[1], a, b[2], b[3]);
        }
        float mx = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 2; nt++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const bool ok = j0 + nt * 8 + t * 2 + e < len;
                s[nt][e] = ok ? s[nt][e] * scale_log2 : -INFINITY;
                mx = fmaxf(mx, s[nt][e]);
            }
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        const float mn = fmaxf(m_run, mx);  // finite: every chunk holds at least one valid key
        const float alpha = exp2f(m_run - mn);
        m_run = mn;
        const float p00 = exp2f(s[0][0] - mn), p01 = exp2f(s[0][1] - mn), p10 = exp2f(s[1][0] - mn), p11 = exp2f(s[1][1] - mn);
        l_run = l_run * alpha + ((p00 + p01) + (p10 + p11));
        const uint32_t pa[4] = {pack_bf16x2(p00, p01), 0u, pack_bf16x2(p10, p11), 0u};
#pragma unroll
        for (int i = 0; i < 16; i++) { o[i][0] *= alpha; o[i][1] *= alpha; }
        // O += P V
#pragma unroll
        for (int np = 0; np < 8; np++) {
            uint32_t b[4];
            const int key = r8 + (mi & 1) * 8;
            ldsm_x4_t(b, sv + dm_off(key, np * 2 + (mi >> 1)));
            mma16816(o[2 * np], pa, b[0], b[1]);
            mma16816(o[2 * np + 1], pa, b[2], b[3]);
        }
        __syncwarp();  // the slot is refilled by the next iteration's issue
        stage = (stage + 1) % DM_STAGES;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");

    // ---- 3. merge the streams: each warp's partial already holds its streams folded in order; across warps the same fixed tree ----
    if (cur_stream >= 0) {
        flush_stream();
    } else if (lane < 8) {  // a warp whose streams are all empty (very short contexts) contributes the neutral element
        if (t == 0) { s_m[g][warp] = -INFINITY; s_l[g][warp] = 0.f; }
#pragma unroll
        for (int nt = 0; nt < 16; nt++) s_acc[g][warp][nt * 8 + t * 2] = s_acc[g][warp][nt * 8 + t * 2 + 1] = 0.f;
    }
    __syncthreads();
    if constexpr (SPLIT) {
        const size_t item = (size_t)seq * gridDim.y + kvh;
        float* mine = split_part + (item * 2 + half) * DM_PART_STRIDE;
        for (int i = lane; i < GROUP * 128; i += 32) mine[i] = s_acc[i >> 7][0][i & 127];
        if (lane < 2 * GROUP) mine[GROUP * 128 + lane] = lane < GROUP ? s_m[lane][0] : s_l[lane - GROUP][0];
        __threadfence();
        __syncwarp();
        int arrived = 0;
        if (lane == 0) arrived = atomicAdd(split_cnt + item, 1);
        arrived = __shfl_sync(0xffffffffu, arrived, 0);
        if (arrived == 0) return;  // the other half finishes the item
        __threadfence();
        const float* other = split_part + (item * 2 + (half ^ 1)) * DM_PART_STRIDE;
        for (int i = lane; i < GROUP * 128; i += 32) {
            const int gg = i >> 7, d = i & 127;
            const float om = __ldcg(other + GROUP * 128 + gg), ol = __ldcg(other + GROUP * 128 + GROUP + gg), oa = __ldcg(other + i);
            // even = half 0, odd = half 1 (the chains of the other variants: a chain of one partial is that partial)
            const float em = half == 0 ? s_m[gg][0] : om, el = half == 0 ? s_l[gg][0] : ol, ea = half == 0 ? s_acc[gg][0][d] : oa;
            const float dm = half == 0 ? om : s_m[gg][0], dl = half == 0 ? ol : s_l[gg][0], da = half == 0 ? oa : s_acc[gg][0][d];
            float fa, fb;
            dm_merge_scales(em, dm, &fa, &fb);
            const float num = fmaf(fb, da, fa * ea), den = fmaf(fb, dl, fa * el);
            out[((size_t)seq * heads + kvh * GROUP + gg) * 128 + d] = __float2bfloat16_rn(num / den);
        }
        if (lane == 0) split_cnt[item] = 0;  // ready for the next launch
    } else
    for (int i = threadIdx.x; i < GROUP * 128; i += NW * 32) {
        const int gg = i >> 7, d = i & 127;
        // even chain (warps 0, 2, ...), odd chain (warps 1, 3, ...), then even + odd: for NW == 2 that is just warp 0 + warp 1
        float cm[2] = {-INFINITY, -INFINITY}, cl[2] = {0.f, 0.f}, ca[2] = {0.f, 0.f};
#pragma unroll
        for (int w = 0; w < NW; w++) {
            float fa, fb;
            const float mm = dm_merge_scales(cm[w & 1], s_m[gg][w], &fa, &fb);
            ca[w & 1] = fmaf(fb, s_acc[gg][w][d], fa * ca[w & 1]);
            cl[w & 1] = fmaf(fb, s_l[gg][w], fa * cl[w & 1]);
            cm[w & 1] = mm;
        }
        float fa, fb;
        dm_merge_scales(cm[0], cm[1], &fa, &fb);
        const float num = fmaf(fb, ca[1], fa * ca[0]), den = fmaf(fb, cl[1], fa * cl[0]);
        out[((size_t)seq * heads + kvh * GROUP + gg) * 128 + d] = __float2bfloat16_rn(num / den);
    }
}

// ------------------------------------------------------------------------------------------
// Split-K consumer of the decode step: x[r] = bf16(x[r] + bf16(sum_s part[s][r])) (residual stream, in place),
// y[r] = RMSNorm(x[r]) * w  (the next block's input).  One CTA per row, 4 columns per thread.
// FloatTextDecoder.swift:144-147 (residual adds) + :139, :146 (the norms that follow them).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) reduce_resid_rmsnorm_kernel(const float* __restrict__ part, int splits, long long split_stride,
                                                                    bf16* __restrict__ x, const bf16* __restrict__ w, bf16* __restrict__ y,
                                                                    int d, float eps) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    // blockDim.x = (d / 4) * SG: thread (cg, sg) sums the splits sg, sg + SG, ... of four columns (all loads in flight at once);
    // the SG partial sums are then added in a fixed order, so the result does not depend on scheduling.
    __shared__ float4 s_part[1024];
    __shared__ float s_red[32];
    const int ncg = d >> 2, sg_count = blockDim.x / ncg;
    const int row = blockIdx.x, cg = threadIdx.x % ncg, sg = threadIdx.x / ncg, c0 = cg * 4;
    const float* src = part + (size_t)row * d + c0;
    float4 b[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int sp = sg + i * sg_count;
        b[i] = sp < splits ? *reinterpret_cast<const float4*>(src + (size_t)sp * split_stride) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float4 a = b[0];
#pragma unroll
    for (int i = 1; i < 4; i++) { a.x += b[i].x; a.y += b[i].y; a.z += b[i].z; a.w += b[i].w; }
    for (int sp = sg + 4 * sg_count; sp < splits; sp += sg_count) {  // more than 4 * SG splits: rare, serial tail
        const float4 t = *reinterpret_cast<const float4*>(src + (size_t)sp * split_stride);
        a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
    }
    s_part[threadIdx.x] = a;
    __syncthreads();
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    float q = 0.f;
    if (sg == 0) {
        for (int g = 1; g < sg_count; g++) {
            const float4 t = s_part[g * ncg + cg];
            a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
        }
        const uint2 u = ld8(x + (size_t)row * d + c0);
        const float2 x0 = unpack_bf16x2(u.x), x1 = unpack_bf16x2(u.y);
        v[0] = bf16_round(x0.x + bf16_round(a.x));
        v[1] = bf16_round(x0.y + bf16_round(a.y));
        v[2] = bf16_round(x1.x + bf16_round(a.z));
        v[3] = bf16_round(x1.y + bf16_round(a.w));
        st8(x + (size_t)row * d + c0, v[0], v[1], v[2], v[3]);
        q = fmaf(v[0], v[0], fmaf(v[1], v[1], fmaf(v[2], v[2], v[3] * v[3])));
    }
    q = warp_sum(q);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = q;
    __syncthreads();
    if (sg == 0) {
        float tot = 0.f;
        for (int i = 0; i < (ncg >> 5); i++) tot += s_red[i];  // the sg == 0 threads are the first ncg / 32 warps
        const float r = rsqrtf(tot / (float)d + eps);
        const uint2 wu = ld8(w + c0);
        const float2 w0 = unpack_bf16x2(wu.x), w1 = unpack_bf16x2(wu.y);
        st8(y + (size_t)row * d + c0, v[0] * r * w0.x, v[1] * r * w0.y, v[2] * r * w1.x, v[3] * r * w1.y);
    }
}

// ------------------------------------------------------------------------------------------
// PER_SEQ (continuous batching): every sequence counts its own steps (out_len), because an admitted utterance starts at step 0 in
// the middle of the loop; it finishes on EOS or at max_tokens, and a finished row stays where it is (pos / kv_len frozen) until a
// partition takes it out, so it never appends past the last page of its block.
template <bool PER_SEQ>
__global__ void decode_advance_kernel(DecodeState s, int n_seqs) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // decode row
    const int step = *s.step;
    if (PER_SEQ) {
        if (i < n_seqs) {
            const int q = s.slot_seq[i];
            if (!s.finished[q]) {
                const int32_t tok = s.next_tok[i];
                const int t = s.out_len[q];
                s.out_ids[(size_t)q * s.max_tokens + t] = tok;
                if (s.out_val && s.next_val) s.out_val[(size_t)q * s.max_tokens + t] = s.next_val[i];
                if (s.out_lp && s.next_lp) s.out_lp[(size_t)q * s.max_tokens + t] = s.next_lp[i];
                s.out_len[q] = t + 1;
                if ((s.stop_on_eos && tok == s.eos) || t + 1 >= s.max_tokens) {
                    s.finished[q] = 1;
                    atomicSub(s.n_active, 1);
                }
                s.cur_tok[i] = tok;
                s.pos[i] += 1;
                s.kv_len[i] += 1;
            }
        }
        __syncthreads();
        if (i == 0) *s.step = step + 1;
        return;
    }
    if (i < n_seqs) {
        const int32_t tok = s.next_tok[i];
        const int q = s.slot_seq ? s.slot_seq[i] : i;  // the sequence this row decodes
        if (!s.finished[q] && step < s.max_tokens) {
            s.out_ids[(size_t)q * s.max_tokens + step] = tok;
            if (s.out_val && s.next_val) s.out_val[(size_t)q * s.max_tokens + step] = s.next_val[i];
            if (s.out_lp && s.next_lp) s.out_lp[(size_t)q * s.max_tokens + step] = s.next_lp[i];
            s.out_len[q] = step + 1;
            if (s.stop_on_eos && tok == s.eos) {
                s.finished[q] = 1;
                atomicSub(s.n_active, 1);
            }
        }
        s.cur_tok[i] = s.forced ? s.forced[step] : tok;
        s.pos[i] += 1;
        s.kv_len[i] += 1;
    }
    __syncthreads();
    if (i == 0) *s.step = step + 1;
}

// ------------------------------------------------------------------------------------------
// Compaction of the decode rows: see decode_compact_launch (ops.cuh).  PARTITION: the finished rows' page-table rows follow the live
// ones (stable), and the rows [rows, cap) are carried over, so every page block stays named in the new table.
template <bool PARTITION>
__global__ void __launch_bounds__(1024) decode_compact_kernel(int rows, const int* __restrict__ finished, int* slot_seq, int32_t* cur_tok, int* pos,
                                                              int* kv_len, const int* __restrict__ page_in, int* __restrict__ page_out,
                                                              int max_pages, int cap) {
    __shared__ int s_warp[32];
    const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
    int q = 0, tok = 0, p = 0, kl = 0, alive = 0;
    if (i < rows) {
        q = slot_seq[i];
        tok = cur_tok[i];
        p = pos[i];
        kl = kv_len[i];
        alive = finished[q] ? 0 : 1;
    }
    // exclusive prefix sum of `alive` over the CTA: warp ballots, then the warp totals
    const unsigned bal = __ballot_sync(0xffffffffu, alive);
    const int in_warp = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();  // also: every row has been read before any is overwritten
    int base = 0;
    for (int w = 0; w < warp; w++) base += s_warp[w];
    if (alive) {
        const int j = base + in_warp;
        slot_seq[j] = q;
        cur_tok[j] = tok;
        pos[j] = p;
        kv_len[j] = kl;
        for (int k = 0; k < max_pages; k++) page_out[(size_t)j * max_pages + k] = page_in[(size_t)i * max_pages + k];
    }
    if (PARTITION) {
        int live = base;
        for (int w = warp; w < 32; w++) live += s_warp[w];
        if (i < rows && !alive) {
            const int j = live + (i - base - in_warp);  // live rows first, then the finished ones in row order
            for (int k = 0; k < max_pages; k++) page_out[(size_t)j * max_pages + k] = page_in[(size_t)i * max_pages + k];
        } else if (i >= rows && i < cap) {
            for (int k = 0; k < max_pages; k++) page_out[(size_t)i * max_pages + k] = page_in[(size_t)i * max_pages + k];
        }
    }
}

// Step 0 of an admitted group (continuous batching), written straight into the resident decode state at rows [row0, row0 + k):
// group member j is request sequence seq0 + j, its first token comes from the group's prefill LM head (tok / val / lp [k]).
__global__ void decode_admit_kernel(DecodeState s, const int32_t* __restrict__ tok, const float* __restrict__ val, const float* __restrict__ lp,
                                    const int* __restrict__ prompt_len, int row0, int k, int seq0) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    __shared__ int s_alive;
    const int j = threadIdx.x;
    if (j == 0) s_alive = 0;
    __syncthreads();
    if (j < k) {
        const int q = seq0 + j, r = row0 + j;
        const int32_t t = tok[j];
        const size_t o = (size_t)q * s.max_tokens;
        const_cast<int*>(s.slot_seq)[r] = q;  // (the step kernels only read the map; the admission extends it)
        s.cur_tok[r] = t;
        s.pos[r] = prompt_len[j];
        s.kv_len[r] = prompt_len[j] + 1;
        s.out_ids[o] = t;
        if (s.out_val && val) s.out_val[o] = val[j];
        if (s.out_lp && lp) s.out_lp[o] = lp[j];
        s.out_len[q] = 1;
        const int fin = (s.stop_on_eos && t == s.eos) || s.max_tokens <= 1;
        s.finished[q] = fin;
        if (!fin) atomicAdd(&s_alive, 1);
    }
    __syncthreads();
    if (j == 0 && s_alive) atomicAdd(s.n_active, s_alive);
}

// ------------------------------------------------------------------------------------------
// pickNextToken on the device (Qwen3ASR.swift:449-520).  Order of the edits as in the reference: penalty, n-gram mask,
// temperature + Gumbel noise, then the first maximum (lowest index on ties; index 0 when every score is -inf).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64_dev(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// (max, sum of exp(x - max)) pairs: the merge of two partial log-sum-exps (an empty side has max -inf and sum 0)
__device__ __forceinline__ void lse_merge(float& m, float& s, float om, float os) {
    const float M = fmaxf(m, om);
    s = (m == -INFINITY ? 0.f : s * __expf(m - M)) + (om == -INFINITY ? 0.f : os * __expf(om - M));
    m = M;
}

// LP: also the (max, sum of exp(x - max)) of the slice's RAW logits (before penalty / mask / noise) to part_rmax / part_rsum, for the
// log-probability of the chosen token (argmax_lse_reduce); every thread walks its indices in ascending order and the merge tree is
// fixed, so the sums depend on the vocabulary and the slice count only.
template <typename T, bool LP>
__global__ void __launch_bounds__(1024) sample_kernel(const T* __restrict__ logits, int ld, int vocab, const int32_t* __restrict__ gen_ids,
                                                       int gen_stride, const int* __restrict__ gen_len, SamplingParams sp,
                                                       const int* __restrict__ step, float* __restrict__ part_val,
                                                       int* __restrict__ part_idx, float* __restrict__ part_rmax, float* __restrict__ part_rsum) {
    // grid (sequence, slice): gridDim.y CTAs share a row's vocabulary scan (the bitmaps are rebuilt by each, they are tiny);
    // argmax_reduce_kernel merges the slices (first maximum)
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    extern __shared__ unsigned int s_bits[];
    const int words = (vocab + 31) / 32;
    unsigned int* seen = s_bits;            // tokens generated so far
    unsigned int* forbidden = s_bits + words;  // tokens that would complete a repeated n-gram
    __shared__ float s_best[32];
    __shared__ int s_idx[32];
    const int seq = blockIdx.x, tid = threadIdx.x;
    const int32_t* gen = gen_ids + (size_t)seq * gen_stride;
    const int g = gen_len[seq];
    const bool penal = sp.repetition_penalty > 1.0f && g > 0;
    const int n = sp.no_repeat_ngram;
    for (int i = tid; i < 2 * words; i += blockDim.x) s_bits[i] = 0u;
    __syncthreads();
    if (penal)
        for (int i = tid; i < g; i += blockDim.x) {
            const int t = gen[i];
            if (t >= 0 && t < vocab) atomicOr(&seen[t >> 5], 1u << (t & 31));
        }
    if (n > 0 && g >= n) {
        const int32_t* last = gen + g - (n - 1);  // the n-1 most recent tokens
        for (int i = tid; i <= g - n; i += blockDim.x) {
            bool same = true;
            for (int k = 0; k < n - 1 && same; k++) same = gen[i + k] == last[k];
            if (same) {
                const int t = gen[i + n - 1];
                if (t >= 0 && t < vocab) atomicOr(&forbidden[t >> 5], 1u << (t & 31));
            }
        }
    }
    __syncthreads();
    const T* row = logits + (size_t)seq * ld;
    const float inv_t = sp.temperature > 0.f ? 1.0f / sp.temperature : 1.0f;
    const unsigned long long key = splitmix64_dev(sp.seed ^ ((unsigned long long)(step ? *step : 0) << 32) ^ (unsigned long long)seq);
    float best = -INFINITY;
    int bidx = 0x7fffffff;
    const int per = (vocab + gridDim.y - 1) / gridDim.y;
    const int i_end = min(vocab, ((int)blockIdx.y + 1) * per);
    float rm = -INFINITY, rs = 0.f;  // LP: running (max, sum) of the raw logits
    for (int i = blockIdx.y * per + tid; i < i_end; i += blockDim.x) {
        float v = (float)row[i];
        if constexpr (LP) {
            if (v > rm) {
                rs = (rm == -INFINITY ? 0.f : rs * __expf(rm - v)) + 1.f;
                rm = v;
            } else {
                rs += __expf(v - rm);
            }
        }
        const unsigned int bit = 1u << (i & 31);
        if (seen[i >> 5] & bit) v = v > 0.f ? v / sp.repetition_penalty : v * sp.repetition_penalty;
        if (forbidden[i >> 5] & bit) v = -INFINITY;
        if (sp.temperature > 0.f) {
            const unsigned int r = (unsigned int)(splitmix64_dev(key + (unsigned long long)i) >> 40);  // 24 bits
            const float u = 1e-6f + (float)r * (1.0f / 16777216.0f) * (1.0f - 1e-6f);                  // [1e-6, 1)
            v = v * inv_t - __logf(-__logf(u));
        }
        if (v > best) { best = v; bidx = i; }  // ascending i per thread: the first maximum is kept
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
    }
    __shared__ float s_rm[32], s_rs[32];
    if constexpr (LP) {
        for (int o = 16; o > 0; o >>= 1) lse_merge(rm, rs, __shfl_xor_sync(0xffffffffu, rm, o), __shfl_xor_sync(0xffffffffu, rs, o));
        if ((tid & 31) == 0) { s_rm[tid >> 5] = rm; s_rs[tid >> 5] = rs; }
    }
    if ((tid & 31) == 0) { s_best[tid >> 5] = best; s_idx[tid >> 5] = bidx; }
    __syncthreads();
    if (tid < 32) {
        const int nw = blockDim.x >> 5;
        best = tid < nw ? s_best[tid] : -INFINITY;
        bidx = tid < nw ? s_idx[tid] : 0x7fffffff;
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
            if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
        }
        if constexpr (LP) {
            rm = tid < nw ? s_rm[tid] : -INFINITY;
            rs = tid < nw ? s_rs[tid] : 0.f;
            for (int o = 16; o > 0; o >>= 1) lse_merge(rm, rs, __shfl_xor_sync(0xffffffffu, rm, o), __shfl_xor_sync(0xffffffffu, rs, o));
            if (tid == 0) {
                part_rmax[(size_t)seq * gridDim.y + blockIdx.y] = rm;
                part_rsum[(size_t)seq * gridDim.y + blockIdx.y] = rs;
            }
        }
        if (tid == 0) {  // an all -inf slice reports index 0 of ITS slice start only through the value: the reducer keeps the first maximum
            part_val[(size_t)seq * gridDim.y + blockIdx.y] = best;
            part_idx[(size_t)seq * gridDim.y + blockIdx.y] = bidx == 0x7fffffff ? 0 : bidx;
        }
    }
}

__global__ void fill_i32_kernel(int* p, int v, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void bf16_to_f32_kernel(const bf16* in, float* out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __bfloat162float(in[i]);
}
__global__ void f32_to_bf16_kernel(const float* in, bf16* out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __float2bfloat16_rn(in[i]);
}
__global__ void f16_to_bf16_kernel(const uint16_t* in, bf16* out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __float2bfloat16_rn(__half2float(__ushort_as_half(in[i])));
}
__global__ void fill_bf16_kernel(bf16* out, size_t n, float v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __float2bfloat16_rn(v);
}
__device__ __forceinline__ unsigned long long splitmix(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
// row_len > 0: "loud rows" — row r of the matrix is multiplied by 2^min(ctz(splitmix(row_seed + r)) / 4, 4) after the bf16
// rounding (exact), i.e. one row in 16 is twice as large, one in 256 four times, ...: a heavy-tailed logit distribution
// through the tied head, so that greedy ids on random weights have margins well above bf16 noise (DESIGN.md §2)
__global__ void random_init_kernel(bf16* out, size_t n, unsigned long long seed, float mult, unsigned long long row_seed, int row_len) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long z = splitmix(seed + (unsigned long long)i * 0x9E3779B97F4A7C15ULL);
    const int s = (int)(z & 0xFFFF) + (int)((z >> 16) & 0xFFFF) + (int)((z >> 32) & 0xFFFF) + (int)(z >> 48) - 131070;
    float v = __bfloat162float(__float2bfloat16_rn(__fmul_rn(__int2float_rn(s), mult)));
    if (row_len > 0) {
        const unsigned long long hz = splitmix(row_seed + (unsigned long long)(i / (size_t)row_len));
        const int tz = hz ? __ffsll((long long)hz) - 1 : 64;
        v *= (float)(1 << min(tz >> 2, 4));
    }
    out[i] = __float2bfloat16_rn(v);
}

// (cos, sin)(pos * inv_freq[i]) for pos < n_pos, i < 64: the fp32 product and sincosf of the per-element kernels, tabulated
__global__ void rope_table_kernel(const float* __restrict__ inv_freq, int n_pos, float2* __restrict__ tab, float2* __restrict__ tab_t) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_pos * 64) return;
    float sn, cs;
    sincosf((float)(idx >> 6) * inv_freq[idx & 63], &sn, &cs);
    tab[idx] = make_float2(cs, sn);
    if (tab_t != nullptr) tab_t[(size_t)(idx & 63) * n_pos + (idx >> 6)] = make_float2(cs, sn);  // the same values, [64][n_pos]
}

inline unsigned blocks_for(size_t n, int t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

void conv1_launch(const float* mel, const Conv1Chunk* chunks, int n_chunks, const bf16* w, const bf16* bias, int C, int chunk_w,
                  bf16* out, cudaStream_t st) {
    if (n_chunks <= 0) return;
    dim3 grid(64, n_chunks);
    conv1_kernel<<<grid, 256, sizeof(float2) * 3 * (chunk_w + 2), st>>>(mel, chunks, w, bias, C, chunk_w, out);
    Q3_CUDA(cudaGetLastError());
}

void layernorm_launch(const bf16* x, const bf16* w, const bf16* b, bf16* y, int rows, int d, float eps, cudaStream_t st) {
    if (rows <= 0) return;
    Q3_CHECK(d % 128 == 0 && d <= 2048, 1, "layernorm: d must be a multiple of 128, <= 2048");
    const unsigned grid = blocks_for(rows, 8);
    if (d <= 1024) layernorm_kernel<8><<<grid, 256, 0, st>>>(x, w, b, y, rows, d, eps);
    else layernorm_kernel<16><<<grid, 256, 0, st>>>(x, w, b, y, rows, d, eps);
    Q3_CUDA(cudaGetLastError());
}

void rmsnorm_launch(const bf16* x, const bf16* w, bf16* y, int rows, int d, float eps, const int* row_index, cudaStream_t st) {
    if (rows <= 0) return;
    Q3_CHECK(d % 128 == 0 && d <= 2048, 1, "rmsnorm: d must be a multiple of 128, <= 2048");
    const unsigned grid = blocks_for(rows, 8);
    if (d <= 1024) launch_kernel(rmsnorm_kernel<8>, grid, 256, 0, st, x, w, y, rows, d, eps, row_index);
    else launch_kernel(rmsnorm_kernel<16>, grid, 256, 0, st, x, w, y, rows, d, eps, row_index);
}

void embed_splice_launch(const int32_t* ids, const int* audio_src, const bf16* embed, const bf16* audio, bf16* x, int rows, int h,
                         cudaStream_t st) {
    if (rows <= 0) return;
    launch_kernel(embed_splice_kernel, blocks_for((size_t)rows * (h / 8), 256), 256, 0, st, ids, audio_src, embed, audio, x, rows, h);
}

void qknorm_rope_kv_launch(const bf16* qkv, int ld, const bf16* qw, const bf16* kw, const int* pos, const int* row_seq, int rows,
                           int heads, int kv_heads, float eps, const float2* rope_tab, bf16* qout, bf16* kc, bf16* vc,
                           const KvCache& cache, int layer, cudaStream_t st) {
    if (rows <= 0) return;
    Q3_CHECK(cache.head_dim == 128, 1, "decoder head_dim must be 128");
    qknorm_rope_kv_kernel<<<rows, 256, 0, st>>>(qkv, ld, qw, kw, pos, row_seq, rows, heads, kv_heads, eps, rope_tab, qout,
                                                                kc, vc, cache, layer);
    Q3_CUDA(cudaGetLastError());
}

void rope_table_launch(const float* inv_freq, int n_pos, float2* tab, float2* tab_t, cudaStream_t st) {
    if (n_pos > 0) rope_table_kernel<<<blocks_for((size_t)n_pos * 64, 256), 256, 0, st>>>(inv_freq, n_pos, tab, tab_t);
    Q3_CUDA(cudaGetLastError());
}

void decode_attn_launch(const bf16* q, const KvCache& cache, int layer, const int* kv_len, int n_seqs, int heads, float scale, bf16* out,
                        cudaStream_t st) {
    if (n_seqs <= 0) return;
    const int group = heads / cache.kv_heads;
    const float sl2 = scale * 1.4426950408889634f;
    dim3 grid(n_seqs, cache.kv_heads);
    switch (group) {
        case 1: decode_attn_kernel<1><<<grid, 128, 0, st>>>(q, cache, layer, kv_len, heads, sl2, out); break;
        case 2: decode_attn_kernel<2><<<grid, 128, 0, st>>>(q, cache, layer, kv_len, heads, sl2, out); break;
        default: throw Error(1, "decode attention: only 1 or 2 query heads per kv head are built");
    }
    Q3_CUDA(cudaGetLastError());
}

void decode_attn_fused_launch(const float* qkv_part, int splits, long long split_stride, int nqkv, const bf16* qw, const bf16* kw,
                              const int* pos, float eps, const float2* rope_tab, const KvCache& cache, int layer, const int* kv_len,
                              int n_seqs, int heads, float scale, bf16* out, int num_sms, cudaStream_t st, float* split_part, int* split_cnt,
                              int force) {
    if (n_seqs <= 0) return;
    Q3_CHECK(cache.head_dim == 128, 1, "decoder head_dim must be 128");
    Q3_CHECK(heads == 2 * cache.kv_heads, 1, "fused decode attention is built for 2 query heads per kv head");
    Q3_CHECK(force == 0 || force == 2 || force == 4 || force == 8 || force == 16 || (force == 1 && split_part != nullptr && split_cnt != nullptr), 1,
             "fused decode attention: unknown variant");
    const float sl2 = scale * 1.4426950408889634f;
    dim3 grid(n_seqs, cache.kv_heads);
    // few (sequence, head) pairs: more warps per CTA so that short batches still spread the key loop
    static PerDeviceOnce attr_once;
    attr_once([] {
        Q3_CUDA(cudaFuncSetAttribute(decode_attn_fused_kernel<2, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, decode_attn_smem(4)));
        Q3_CUDA(cudaFuncSetAttribute(decode_attn_fused_kernel<2, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, decode_attn_smem(16)));
        Q3_CUDA(cudaFuncSetAttribute(decode_attn_mma_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, decode_attn_mma_smem(1)));
        Q3_CUDA(cudaFuncSetAttribute(decode_attn_mma_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, decode_attn_mma_smem(2)));
        Q3_CUDA(cudaFuncSetAttribute(decode_attn_mma_kernel<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, decode_attn_mma_smem(8)));
    });
    const long items = (long)n_seqs * cache.kv_heads;
    // eight warps per item below two items per SM, two above.  The split variant (two single-warp CTAs per item, all 1024 half-items
    // of the bench batch resident at once, 6.9 per SM instead of 3 or 4 items) is opt-in: bit-identical, but measured SLOWER on B200,
    // 63.2 against 55.2 us per layer at 64 sequences — the second pass of the prologue and the meeting through global memory
    // (fence, atomic, 1 KB read back) add more to every item's dependent chain than the even spread takes off the tail.
    int warps = items >= 2L * num_sms ? 2 : 8;
    if (const char* f = getenv("Q3ASR_DECODE_ATTN_WARPS")) {  // tests force a variant on small batches (1 = split, 2 or 8 warps)
        const int w = atoi(f);
        if (w == 2 || w == 8 || (w == 1 && split_part != nullptr && split_cnt != nullptr)) warps = w;
    }
    static const bool simt_env = getenv("Q3ASR_DECODE_ATTN_SIMT") != nullptr && atoi(getenv("Q3ASR_DECODE_ATTN_SIMT")) != 0;
    bool simt = simt_env;
    if (force != 0) {  // the kernel test hook names the variant: 1, 2, 8 = the tensor-core kernel's warps, 4, 16 = the SIMT kernel's
        simt = force == 4 || force == 16;
        warps = force == 16 ? 8 : force == 4 ? 2 : force;
    }
    if (!simt) {
        if (warps == 1)
            launch_kernel(decode_attn_mma_kernel<1, true>, dim3(n_seqs, cache.kv_heads, 2), 32, decode_attn_mma_smem(1), st, qkv_part, splits,
                          split_stride, nqkv, qw, kw, pos, eps, rope_tab, cache, layer, kv_len, heads, sl2, out, split_part, split_cnt);
        else if (warps == 2)
            launch_kernel(decode_attn_mma_kernel<2, false>, grid, 64, decode_attn_mma_smem(2), st, qkv_part, splits, split_stride, nqkv, qw, kw, pos, eps,
                          rope_tab, cache, layer, kv_len, heads, sl2, out, split_part, split_cnt);
        else
            launch_kernel(decode_attn_mma_kernel<8, false>, grid, 256, decode_attn_mma_smem(8), st, qkv_part, splits, split_stride, nqkv, qw, kw, pos, eps,
                          rope_tab, cache, layer, kv_len, heads, sl2, out, split_part, split_cnt);
    } else if (warps <= 2) {
        launch_kernel(decode_attn_fused_kernel<2, 4>, grid, 128, decode_attn_smem(4), st, qkv_part, splits, split_stride, nqkv, qw, kw, pos, eps,
                      rope_tab, cache, layer, kv_len, heads, sl2, out);
    } else {
        launch_kernel(decode_attn_fused_kernel<2, 16>, grid, 512, decode_attn_smem(16), st, qkv_part, splits, split_stride, nqkv, qw, kw, pos,
                      eps, rope_tab, cache, layer, kv_len, heads, sl2, out);
    }
}

void reduce_resid_rmsnorm_launch(const float* part, int splits, long long split_stride, bf16* x, const bf16* w, bf16* y, int rows, int d,
                                 float eps, cudaStream_t st) {
    if (rows <= 0) return;
    Q3_CHECK(d % 128 == 0 && d <= 2048, 1, "reduce_resid_rmsnorm: d must be a multiple of 128, <= 2048");
    const int ncg = d / 4;
    int sg = std::max(1, std::min(1024 / ncg, (splits + 3) / 4 > 0 ? 1024 / ncg : 1));
    while (sg > 1 && sg > splits) sg >>= 1;  // no more split groups than splits
    launch_kernel(reduce_resid_rmsnorm_kernel, rows, ncg * sg, 0, st, part, splits, split_stride, x, w, y, d, eps);
}

void decode_advance_launch(const DecodeState& s, int n_seqs, cudaStream_t st, bool per_seq) {
    Q3_CHECK(n_seqs <= 1024, 1, "decode_advance: at most 1024 sequences per handle");
    Q3_CHECK(!per_seq || s.slot_seq != nullptr, 1, "decode_advance: per-sequence steps need the row -> sequence map");
    if (per_seq) launch_kernel(decode_advance_kernel<true>, 1, 1024, 0, st, s, n_seqs);
    else launch_kernel(decode_advance_kernel<false>, 1, 1024, 0, st, s, n_seqs);
}

void decode_compact_launch(int rows, const int* finished, int* slot_seq, int32_t* cur_tok, int* pos, int* kv_len, const int* page_in,
                           int* page_out, int max_pages, cudaStream_t st, int partition_cap) {
    Q3_CHECK(rows >= 1 && rows <= 1024 && partition_cap <= 1024, 1, "decode_compact: 1..1024 rows");
    if (partition_cap > 0)
        decode_compact_kernel<true><<<1, 1024, 0, st>>>(rows, finished, slot_seq, cur_tok, pos, kv_len, page_in, page_out, max_pages,
                                                        partition_cap);
    else
        decode_compact_kernel<false><<<1, 1024, 0, st>>>(rows, finished, slot_seq, cur_tok, pos, kv_len, page_in, page_out, max_pages, 0);
    Q3_CUDA(cudaGetLastError());
}

void decode_admit_launch(const DecodeState& s, const int32_t* tok, const float* val, const float* lp, const int* prompt_len, int row0, int k,
                         int seq0, cudaStream_t st) {
    Q3_CHECK(k >= 1 && k <= 1024 && s.slot_seq != nullptr, 1, "decode_admit: 1..1024 rows and a row -> sequence map");
    launch_kernel(decode_admit_kernel, 1, 1024, 0, st, s, tok, val, lp, prompt_len, row0, k, seq0);
}

int sample_parts(int vocab) { return vocab >= 32768 ? 4 : 1; }

void sample_launch(const bf16* logits_bf16, const float* logits_f32, int ld, int vocab, const int32_t* gen_ids, int gen_stride,
                   const int* gen_len, const SamplingParams& sp, const int* step, int n_seqs, float* part_val, int* part_idx,
                   cudaStream_t st, float* part_rmax, float* part_rsum) {
    if (n_seqs <= 0) return;
    Q3_CHECK(vocab > 0 && vocab <= 160 * 1024, 1, "sample: vocabulary too large for the shared-memory bitmaps");
    Q3_CHECK((logits_bf16 != nullptr) != (logits_f32 != nullptr), 1, "sample: exactly one logits pointer");
    Q3_CHECK(part_val != nullptr && part_idx != nullptr, 1, "sample: null scratch");
    const size_t smem = (size_t)2 * ((vocab + 31) / 32) * sizeof(unsigned int);
    const int parts = sample_parts(vocab);
    const dim3 grid(n_seqs, parts);
    Q3_CHECK((part_rmax != nullptr) == (part_rsum != nullptr) && (part_rmax == nullptr || logits_bf16 != nullptr), 1,
             "sample: raw (max, sum) outputs come in pairs, bf16 logits only");
    if (part_rmax)
        launch_kernel(sample_kernel<bf16, true>, grid, 1024, smem, st, logits_bf16, ld, vocab, gen_ids, gen_stride, gen_len, sp, step, part_val,
                      part_idx, part_rmax, part_rsum);
    else if (logits_bf16)
        launch_kernel(sample_kernel<bf16, false>, grid, 1024, smem, st, logits_bf16, ld, vocab, gen_ids, gen_stride, gen_len, sp, step, part_val,
                      part_idx, nullptr, nullptr);
    else
        launch_kernel(sample_kernel<float, false>, grid, 1024, smem, st, logits_f32, ld, vocab, gen_ids, gen_stride, gen_len, sp, step, part_val,
                      part_idx, nullptr, nullptr);
}

void fill_i32_launch(int* p, int v, size_t n, cudaStream_t st) {
    if (n) fill_i32_kernel<<<blocks_for(n, 256), 256, 0, st>>>(p, v, n);
}
void bf16_to_f32_launch(const bf16* in, float* out, size_t n, cudaStream_t st) {
    if (n) bf16_to_f32_kernel<<<blocks_for(n, 256), 256, 0, st>>>(in, out, n);
}
void f32_to_bf16_launch(const float* in, bf16* out, size_t n, cudaStream_t st) {
    if (n) f32_to_bf16_kernel<<<blocks_for(n, 256), 256, 0, st>>>(in, out, n);
}
void f16_to_bf16_launch(const uint16_t* in, bf16* out, size_t n, cudaStream_t st) {
    if (n) f16_to_bf16_kernel<<<blocks_for(n, 256), 256, 0, st>>>(in, out, n);
}
void random_init_launch(bf16* out, size_t n, uint64_t seed, float scale, cudaStream_t st, uint64_t row_seed, int row_len) {
    // std of the 4x16-bit Irwin-Hall sum is sqrt((65536^2 - 1) / 3)
    const float mult = (float)((double)scale / 37837.22668596909);
    if (n) random_init_kernel<<<blocks_for(n, 256), 256, 0, st>>>(out, n, (unsigned long long)seed, mult, (unsigned long long)row_seed, row_len);
}
void fill_bf16_launch(bf16* out, size_t n, float v, cudaStream_t st) {
    if (n) fill_bf16_kernel<<<blocks_for(n, 256), 256, 0, st>>>(out, n, v);
}

}  // namespace q3
