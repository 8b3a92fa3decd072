// lmhead.cuh — tied LM head + argmax for the decode step (few token rows, the whole embedding matrix streamed once).
//
//   logits[m, n] = sum_k X[m, k] E[n, k];  token[m] = first maximum of bf16(logits[m, :])
//   (PreQuantizedEmbedding.asLinear + argMax, MLXCommon/PreQuantizedEmbedding.swift:45-49, Qwen3ASR.swift:254-256, 360)
//
// Same operand roles as skinny.cuh: 128 vocabulary rows are the UMMA M operand, the <= NB token rows the N operand, so neither the
// tensor core nor the shared-memory fill path carries the padding a 128-row token tile would.  Persistent: CTA c owns a contiguous
// range of 128-row vocabulary tiles, an 8-stage ring keeps >= 128 KB of the matrix in flight per SM, and the accumulator is
// double-buffered in TMEM so the argmax of tile t overlaps the products of tile t + 1.  The epilogue holds one vocabulary row per
// thread (TMEM lane): the per-token maximum over the 32 rows of a warp is a transpose-reduce (31 exchanges per 32 tokens instead
// of 160), the four warps are merged through shared memory, and each tile writes (value, index) per token for argmax_reduce.
//
// LSE = true (log-probabilities, q3asr_batch_set_logprobs) also writes amax_sum[token, tile] = sum over the tile's valid rows of
// exp(z_r - tile max), z = bf16(logits).  Formulation: the max transpose-reduce already leaves lane l with token l's maximum over the
// warp's 32 rows; it is broadcast back with one shuffle per token, each lane takes one exponential per value against it (rows >= N
// contribute 0, never exp(-inf - -inf)), a second transpose-reduce sums them, and the four warps' (max, sum) pairs are merged in
// warp order with s = sum_w s_w exp(m_w - M).  Carrying (max, sum) pairs through the first reduce instead would take two exponentials
// per exchange; broadcasting the TILE maximum is not possible, because it is known only after the four-warp merge, when the
// accumulator has been handed back to the tensor core.  Every token's sum has one fixed tree (lane butterfly, then warps 0..3), so it
// does not depend on NB, on the token count or on which CTA owns the tile.
//
// CTA = 256 threads: warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue.
#pragma once
#include "skinny.cuh"

namespace q3 {

struct LmHeadDev {
    int N, Mtok, num_kb, tiles;
    float* amax_val;  // [Mtok, tiles]
    int* amax_idx;
    float* amax_sum;  // [Mtok, tiles], LSE instantiations only
};

constexpr int LMH_STAGES = 8;
__host__ __device__ constexpr int lmh_stages(int NB) { return (200 * 1024) / sk_stage_bytes(NB) < LMH_STAGES ? (200 * 1024) / sk_stage_bytes(NB) : LMH_STAGES; }
__host__ __device__ constexpr int lmh_smem_bytes(int NB, bool LSE = false) {
    return lmh_stages(NB) * sk_stage_bytes(NB) + 1024 + 512 + 4 * NB * (LSE ? 12 : 8);
}

// (value, index) maximum with the first index on ties
__device__ __forceinline__ void amax_merge(float& v, int& i, float ov, int oi) {
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
}

// 32 tokens per lane, one vocabulary row per lane: afterwards lane l holds token l's maximum over the warp's 32 rows
__device__ __forceinline__ void transpose_reduce32(float (&v)[32], int (&ix)[32], int lane) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; i++) {
            const float sv = up ? v[i] : v[i + off];
            const int si = up ? ix[i] : ix[i + off];
            float kv = up ? v[i + off] : v[i];
            int ki = up ? ix[i + off] : ix[i];
            amax_merge(kv, ki, __shfl_xor_sync(0xffffffffu, sv, off), __shfl_xor_sync(0xffffffffu, si, off));
            v[i] = kv;
            ix[i] = ki;
        }
    }
}

// the same butterfly as transpose_reduce32, summing: afterwards lane l holds sum over the warp's 32 lanes of v[l]
__device__ __forceinline__ void transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; i++) {
            const float sv = up ? v[i] : v[i + off];
            const float kv = up ? v[i + off] : v[i];
            v[i] = kv + __shfl_xor_sync(0xffffffffu, sv, off);
        }
    }
}

template <int NB, bool LSE = false>
__global__ void __launch_bounds__(256, 1)
lmhead_argmax_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmX, const LmHeadDev p) {
    constexpr int STAGES = lmh_stages(NB);
    constexpr int STAGE_BYTES = sk_stage_bytes(NB);
    constexpr int ACC_COLS = NB < 32 ? 32 : NB;
    constexpr int TMEM_COLS = 2 * ACC_COLS < 32 ? 32 : 2 * ACC_COLS;
    constexpr uint32_t IDESC = ptx::umma_idesc_bf16(SK_BM, NB);
    constexpr int CH = NB < 32 ? NB : 32;
    static_assert(NB % 16 == 0 && NB >= 16 && NB <= 256, "NB");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;   // [2]
    uint64_t* tempty_bar = tfull_bar + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* s_val = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + 512);  // [4 warps][NB]
    int* s_idx = reinterpret_cast<int*>(s_val + 4 * NB);
    float* s_sum = reinterpret_cast<float*>(s_idx + 4 * NB);  // [4 warps][NB], LSE only

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t0 = (int)(((long long)blockIdx.x * p.tiles) / gridDim.x), t1 = (int)(((long long)(blockIdx.x + 1) * p.tiles) / gridDim.x);
    const int total_kb = (t1 - t0) * p.num_kb;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmW);
        ptx::prefetch_tmap(&tmX);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; s++) {
            ptx::mbar_init(&full_bar[s], 1);
            ptx::mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; b++) {
            ptx::mbar_init(&tfull_bar[b], 1);
            ptx::mbar_init(&tempty_bar[b], 128);
        }
        ptx::fence_barrier_init();
    }
    if (warp == 2) ptx::tmem_alloc<TMEM_COLS>(tmem_slot);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            ptx::grid_dep_launch();
            // the embedding tiles do not depend on the previous kernel: fill the ring with them, then wait for the producer of X
            const int pre = min(STAGES, total_kb);
            for (int i = 0; i < pre; i++) {
                ptx::mbar_arrive_expect_tx(&full_bar[i], (uint32_t)STAGE_BYTES);
                ptx::tma_load_2d(smem + i * STAGE_BYTES, &tmW, (i % p.num_kb) * SK_BK, (t0 + i / p.num_kb) * SK_BM, &full_bar[i]);
            }
            ptx::grid_dep_wait();
            for (int i = 0; i < pre; i++)
                ptx::tma_load_2d(smem + i * STAGE_BYTES + SK_BM * 128, &tmX, (i % p.num_kb) * SK_BK, 0, &full_bar[i]);
            int stage = 0;
            uint32_t phase = 1;
            for (int i = pre; i < total_kb; i++) {
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + stage * STAGE_BYTES;
                const int kb = i % p.num_kb, tile = t0 + i / p.num_kb;
                ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)STAGE_BYTES);
                ptx::tma_load_2d(sa, &tmW, kb * SK_BK, tile * SK_BM, &full_bar[stage]);
                ptx::tma_load_2d(sa + SK_BM * 128, &tmX, kb * SK_BK, 0, &full_bar[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = t0, it = 0; t < t1; t++, it++) {
                const int ab = it & 1;
                ptx::mbar_wait(&tempty_bar[ab], ((it >> 1) & 1) ^ 1);  // the epilogue has drained this accumulator
                ptx::tc_fence_after();
                const uint32_t acc = tmem_base + (uint32_t)(ab * ACC_COLS);
                for (int kb = 0; kb < p.num_kb; kb++) {
                    ptx::mbar_wait(&full_bar[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t sa = ptx::smem_u32(smem + stage * STAGE_BYTES);
                    const uint32_t sb = sa + SK_BM * 128;
#pragma unroll
                    for (int k = 0; k < SK_BK / 16; k++)
                        ptx::mma_bf16_ss(acc, ptx::umma_desc_sw128(sa + k * 32), ptx::umma_desc_sw128(sb + k * 32), IDESC, (kb > 0 || k > 0) ? 1u : 0u);
                    ptx::mma_commit(&empty_bar[stage]);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                ptx::mma_commit(&tfull_bar[ab]);
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3;
        const int r = q * 32 + lane;  // vocabulary row within the tile = TMEM lane
        for (int t = t0, it = 0; t < t1; t++, it++) {
            const int ab = it & 1;
            ptx::mbar_wait(&tfull_bar[ab], (it >> 1) & 1);
            ptx::tc_fence_after();
            const uint32_t t_row = tmem_base + (uint32_t)(ab * ACC_COLS) + (uint32_t(q * 32) << 16);
            const int row = t * SK_BM + r;
            const bool row_ok = row < p.N;
#pragma unroll 1
            for (int c = 0; c < NB / CH; c++) {
                uint32_t u[CH];
                if constexpr (CH == 32) ptx::tmem_ld_32x32(t_row + c * CH, u); else ptx::tmem_ld_32x16(t_row + c * CH, reinterpret_cast<uint32_t(&)[16]>(u));
                ptx::tmem_ld_wait();
                if (c == NB / CH - 1) {  // everything of this accumulator is in registers: hand it back to the tensor core
                    ptx::tc_fence_before();
                    ptx::mbar_arrive(&tempty_bar[ab]);
                }
                float v[32];
                int ix[32];
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    v[j] = (j < CH && row_ok) ? bf16_round(__uint_as_float(u[j < CH ? j : 0])) : -INFINITY;
                    ix[j] = row;
                }
                transpose_reduce32(v, ix, lane);  // lane l: token c * CH + l over this warp's 32 rows
                if (lane < CH) {
                    s_val[q * NB + c * CH + lane] = v[0];
                    s_idx[q * NB + c * CH + lane] = ix[0];
                }
                if constexpr (LSE) {
                    const float wmax = v[0];
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        const float mj = __shfl_sync(0xffffffffu, wmax, j);
                        v[j] = (j < CH && row_ok) ? __expf(bf16_round(__uint_as_float(u[j < CH ? j : 0])) - mj) : 0.f;
                    }
                    transpose_sum32(v, lane);
                    if (lane < CH) s_sum[q * NB + c * CH + lane] = v[0];
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");  // the four epilogue warps
            for (int m = threadIdx.x - 128; m < NB && m < p.Mtok; m += 128) {  // 128 epilogue threads, up to 256 tokens
                float bv = s_val[m];
                int bi = s_idx[m];
#pragma unroll
                for (int w = 1; w < 4; w++) amax_merge(bv, bi, s_val[w * NB + m], s_idx[w * NB + m]);
                p.amax_val[(size_t)m * p.tiles + t] = bv;
                p.amax_idx[(size_t)m * p.tiles + t] = bi;
                if constexpr (LSE) {  // a warp without valid rows has max -inf and sum 0
                    float sum = 0.f;
#pragma unroll
                    for (int w = 0; w < 4; w++) {
                        const float mw = s_val[w * NB + m];
                        sum += mw == -INFINITY ? 0.f : s_sum[w * NB + m] * __expf(mw - bv);
                    }
                    p.amax_sum[(size_t)m * p.tiles + t] = sum;
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");  // s_val / s_idx are reused by the next tile
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

}  // namespace q3
