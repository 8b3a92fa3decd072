// gemm.cu — host side of the tcgen05 GEMM: tensor-map construction, tile selection, dispatch, plus the
// CUDA-core checker kernels used by the GPU tests to bisect tensor-core bugs (never by the model code).
#include <cudaTypedefs.h>
#include <stdlib.h>

#include <atomic>
#include <vector>

#include "gemm2.cuh"
#include "lmhead.cuh"
#include "skinny.cuh"

namespace q3 {

namespace {

PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
int g_num_sms = 148;
// per host thread: a handle is driven by one thread (pool workers each own theirs), so differencing the counter around a region
// (forward.cu: the captured decode step) counts that handle's launches only
thread_local unsigned long long g_launches = 0;

void make_tmap(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
               const cuuint32_t* box, const cuuint32_t* estr, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
    Q3_CHECK(g_encode != nullptr, 2, "gemm_init() has not been called");
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides_bytes, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        std::string s = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + "): rank " + std::to_string(rank) + " dims";
        for (int i = 0; i < rank; i++) s += " " + std::to_string((unsigned long long)dims[i]);
        s += " strides";
        for (int i = 0; i + 1 < rank; i++) s += " " + std::to_string((unsigned long long)strides_bytes[i]);
        s += " box";
        for (int i = 0; i < rank; i++) s += " " + std::to_string(box[i]);
        s += " estr";
        for (int i = 0; i < rank; i++) s += " " + std::to_string(estr[i]);
        throw Error(3, s);
    }
}

template <int BN, int EPI>
void launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, GemmDev p, int max_stages, int grid, cudaStream_t st) {
    static PerDeviceOnce attr_once;
    attr_once([] {
        Q3_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes(BN)));
    });
    p.stages = max_stages > 0 ? std::min(max_stages, gemm_stages(BN)) : gemm_stages(BN);
    const int smem = p.stages * gemm_stage_bytes(BN) + (p.tma_out ? EPI_STAGE_BYTES : 0) + 1024 + 256;
    launch_kernel(gemm_tc_kernel<BN, EPI>, grid, GEMM_THREADS, smem, st, ta, tb, tc, p);
}

template <int BN>
void launch_bn(int epi, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmDev& p, int ms, int grid, cudaStream_t st) {
    switch (epi) {
        case EPI_NORMAL: launch_tc<BN, EPI_NORMAL>(ta, tb, tc, p, ms, grid, st); break;
        case EPI_SWIGLU: launch_tc<BN, EPI_SWIGLU>(ta, tb, tc, p, ms, grid, st); break;
        case EPI_F32: launch_tc<BN, EPI_F32>(ta, tb, tc, p, ms, grid, st); break;
        case EPI_ARGMAX: launch_tc<BN, EPI_ARGMAX>(ta, tb, tc, p, ms, grid, st); break;
        case EPI_QKV:
            if constexpr (BN % 128 == 0) launch_tc<BN, EPI_QKV>(ta, tb, tc, p, ms, grid, st);
            else throw Error(1, "gemm: the fused q/k/v epilogue needs tiles of whole heads (128 or 256 columns)");
            break;
        default: throw Error(1, "gemm: bad epilogue");
    }
}

template <int BN, int EPI>
void launch_tc2(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmDev& p, int grid, cudaStream_t st) {
    static PerDeviceOnce attr_once;
    attr_once([] {
        Q3_CUDA(cudaFuncSetAttribute(gemm_tc2_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm2_smem_bytes(BN)));
    });
    launch_kernel(gemm_tc2_kernel<BN, EPI>, grid, GEMM_THREADS, gemm2_smem_bytes(BN) - (p.tma_out ? 0 : EPI_STAGE_BYTES), st, ta, tb, tc, p);
}
template <int BN>
void launch_bn2(int epi, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmDev& p, int grid, cudaStream_t st) {
    if (epi == EPI_SWIGLU) launch_tc2<BN, EPI_SWIGLU>(ta, tb, tc, p, grid, st);
    else if (epi == EPI_QKV) {
        if constexpr (BN % 128 == 0) launch_tc2<BN, EPI_QKV>(ta, tb, tc, p, grid, st);
        else throw Error(1, "gemm: the fused q/k/v epilogue needs tiles of whole heads (128 or 256 columns)");
    } else launch_tc2<BN, EPI_NORMAL>(ta, tb, tc, p, grid, st);
}

// ------------------------------------------------------------------------------------------
// CUDA-core checker: same operand views, same epilogue arithmetic, no tensor cores, no TMA.
// ------------------------------------------------------------------------------------------
struct SimtView {
    const bf16* A;
    int C, W, H, B;
    long sW, sH, sB;
    int OW, OH, OB, sw, sh, taps;
    signed char tap_dw[GEMM_MAX_TAPS], tap_dh[GEMM_MAX_TAPS];
    const bf16* Wt;
    int N;
};

__global__ void simt_acc_kernel(SimtView v, float* acc, long rows) {
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * v.N) return;
    const int n = (int)(idx % v.N);
    const long row = idx / v.N;
    const int w = (int)(row % v.OW);
    const int h = (int)((row / v.OW) % v.OH);
    const int b = (int)(row / ((long)v.OW * v.OH));
    const long K = (long)v.taps * v.C;
    float s = 0.f;
    for (int t = 0; t < v.taps; t++) {
        const int iw = w * v.sw + v.tap_dw[t], ih = h * v.sh + v.tap_dh[t];
        if (iw < 0 || iw >= v.W || ih < 0 || ih >= v.H) continue;
        const bf16* ap = v.A + (long)b * v.sB + (long)ih * v.sH + (long)iw * v.sW;
        const bf16* wp = v.Wt + (long)n * K + (long)t * v.C;
        for (int c = 0; c < v.C; c++) s = fmaf(__bfloat162float(ap[c]), __bfloat162float(wp[c]), s);
    }
    acc[idx] = s;
}

__global__ void simt_epi_kernel(const float* acc, long rows, GemmDev p, int epi, int BN) {
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (epi == EPI_ARGMAX) {
        if (idx >= rows * p.tiles_n) return;
        const int tn = (int)(idx % p.tiles_n);
        const long row = idx / p.tiles_n;
        float best = -INFINITY;
        int bi = 0;
        for (int j = 0; j < BN; j++) {
            const float x = bf16_round(acc[row * p.N + tn * BN + j]);
            if (x > best) { best = x; bi = tn * BN + j; }
        }
        p.amax_val[idx] = best;
        p.amax_idx[idx] = bi;
        if (p.amax_sum) {
            float sum = 0.f;
            for (int j = 0; j < BN; j++) sum += __expf(bf16_round(acc[row * p.N + tn * BN + j]) - best);
            p.amax_sum[idx] = sum;
        }
        return;
    }
    if (epi == EPI_SWIGLU) {
        const int half = p.N / 2;
        if (idx >= rows * half) return;
        const int oc = (int)(idx % half);
        const long row = idx / half;
        const int blk = oc / GU_UNIT, j = oc % GU_UNIT;
        const float g = acc[row * p.N + blk * 2 * GU_UNIT + j], u = acc[row * p.N + blk * 2 * GU_UNIT + GU_UNIT + j];
        reinterpret_cast<bf16*>(p.out)[row * p.ldo + oc] = __float2bfloat16_rn(epi_swiglu(g, u));
        return;
    }
    if (idx >= rows * p.N) return;
    const int n = (int)(idx % p.N);
    long row = idx / p.N;
    const int w = (int)(row % p.OW);
    const int b = (int)(row / ((long)p.OW * p.OH));
    float f = acc[idx];
    if (p.bias) f += __bfloat162float(p.bias[n]);
    if (epi == EPI_F32) {
        reinterpret_cast<float*>(p.out)[row * p.ldo + n] = f;
        return;
    }
    if (p.row_add) f += p.row_add[(long)w * p.N + n];
    if (p.gelu) f = gelu_erf(f);
    if (p.valid_w && w >= p.valid_w[b]) f = 0.f;
    if (p.row_map) {
        row = p.row_map[row];
        if (row < 0) return;
    }
    if (p.resid) f = __bfloat162float(p.resid[row * p.ldr + n]) + bf16_round(f);
    reinterpret_cast<bf16*>(p.out)[row * p.ldo + n] = __float2bfloat16_rn(f);
}

__global__ void argmax_reduce_kernel(const float* val, const int* idx, int rows, int tiles, int32_t* out, float* out_val) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    const int row = blockIdx.x;
    if (row >= rows) return;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int t = threadIdx.x; t < tiles; t += blockDim.x) {
        const float v = val[(size_t)row * tiles + t];
        const int i = idx[(size_t)row * tiles + t];
        if (v > best || (v == best && i < bi)) { best = v; bi = i; }
    }
    __shared__ float sv[32];
    __shared__ int si[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sv[warp] = best; si[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        best = lane < nw ? sv[lane] : -INFINITY;
        bi = lane < nw ? si[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) {
            out[row] = bi;
            if (out_val) out_val[row] = best;
        }
    }
}

// argmax_reduce_kernel plus the log-probability of the chosen token: lse = M + log sum_t s_t exp(m_t - M) over the per-tile maxima
// m_t (tile_max, or val when null) and sums s_t = sum exp(z - m_t) of the tile's logits; out_lp = z[chosen] - lse, with z[chosen]
// read from the raw bf16 logits when given (decoder knobs: the chosen index need not be the raw maximum), else the maximum itself.
// Every thread walks its tiles in ascending order and the 256 threads are merged by a fixed tree, so the result depends only on
// `tiles`, never on the row count.
__global__ void __launch_bounds__(256) argmax_lse_reduce_kernel(const float* val, const int* idx, const float* tile_sum, const float* tile_max,
                                                                const bf16* raw, int ld, int rows, int tiles, int32_t* out, float* out_val,
                                                                float* out_lp) {
    ptx::grid_dep_launch();
    ptx::grid_dep_wait();
    const int row = blockIdx.x;
    if (row >= rows) return;
    const float* mx = (tile_max ? tile_max : val) + (size_t)row * tiles;
    const float* sm = tile_sum + (size_t)row * tiles;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ float sv[8];
    __shared__ int si[8];
    __shared__ float s_m;
    float best = -INFINITY, m = -INFINITY;
    int bi = 0x7fffffff;
    for (int t = threadIdx.x; t < tiles; t += blockDim.x) {
        const float v = val[(size_t)row * tiles + t];
        const int i = idx[(size_t)row * tiles + t];
        if (v > best || (v == best && i < bi)) { best = v; bi = i; }
        m = fmaxf(m, mx[t]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    if (lane == 0) { sv[warp] = best; si[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        best = lane < 8 ? sv[lane] : -INFINITY;
        bi = lane < 8 ? si[lane] : 0x7fffffff;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
    }
    __syncthreads();
    if (lane == 0) sv[warp] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float mm = sv[0];
        for (int w = 1; w < 8; w++) mm = fmaxf(mm, sv[w]);
        s_m = mm;
    }
    __syncthreads();
    const float M = s_m;
    float s = 0.f;
    for (int t = threadIdx.x; t < tiles; t += blockDim.x) {
        const float mt = mx[t];
        if (mt != -INFINITY) s += sm[t] * __expf(mt - M);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __syncthreads();  // sv is reused
    if (lane == 0) sv[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
        for (int w = 0; w < 8; w++) tot += sv[w];
        const float z = raw ? __bfloat162float(raw[(size_t)row * ld + bi]) : best;
        out[row] = bi;
        if (out_val) out_val[row] = best;
        out_lp[row] = (z - M) - logf(tot);  // z - M first: both are logits of similar size, the difference is exact
    }
}

}  // namespace

void make_tmap_2d_bf16(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint64_t row_stride_elems, uint32_t box_cols,
                       uint32_t box_rows) {
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t str[1] = {(cuuint64_t)row_stride_elems * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t es[2] = {1, 1};
    make_tmap(m, ptr, 2, dims, str, box, es);
}

void gemm_init(int device) {
    if (g_encode == nullptr) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        Q3_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        Q3_CHECK(qres == cudaDriverEntryPointSuccess && fn != nullptr, 3, "cuTensorMapEncodeTiled not available in this driver");
        g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    }
    cudaDeviceProp prop;
    Q3_CUDA(cudaGetDeviceProperties(&prop, device));
    Q3_CHECK(prop.major == 10, 3, std::string("q3asr kernels are built for sm_100a only; device is sm_") + std::to_string(prop.major) +
                                      std::to_string(prop.minor));
    g_num_sms = prop.multiProcessorCount;
}

int gemm_pick_bn(int N, int epi, long m_tiles) {
    // wide tiles first: a 128-row M tile with N <= 128 is bound by shared-memory operand reads, not by the tensor pipe
    static const int cand[] = {256, 224, 160, 128, 64, 32};
    int smallest = 0;
    for (int bn : cand) {
        if (N % bn) continue;
        if (epi == EPI_SWIGLU && bn % (2 * GU_UNIT)) continue;
        smallest = bn;
        if (m_tiles * (N / bn) >= 2L * g_num_sms) return bn;
    }
    Q3_CHECK(smallest != 0, 1, "gemm: N = " + std::to_string(N) + " is not a multiple of 32");
    // small problems: the narrowest tile gives the most CTAs to stream the weights
    return smallest;
}
int gemm_pick_bn(int N, int epi) { return gemm_pick_bn(N, epi, 1L << 20); }

void gemm_conv(const GemmA& a, const GemmShape& s, const bf16* W, int N, const GemmEpiArgs& e, cudaStream_t st, bool simt, int bn) {
    Q3_CHECK(a.C % 8 == 0 && a.C > 0, 1, "gemm: channel count must be a positive multiple of 8");
    Q3_CHECK(s.taps >= 1 && s.taps <= GEMM_MAX_TAPS, 1, "gemm: taps");
    Q3_CHECK(s.Wb * s.Hb * s.Bb <= GEMM_BM && s.Wb * s.sw <= 256 && s.Hb * s.sh <= 256, 1, "gemm: M-tile box");
    const long rows = (long)s.OW * s.OH * s.OB;
    if (rows == 0) return;
    GemmDev p;
    memset(&p, 0, sizeof(p));
    p.N = N;
    p.C = a.C;
    p.kb_per_tap = (a.C + GEMM_BK - 1) / GEMM_BK;
    p.num_kb = p.kb_per_tap * s.taps;
    p.Wb = s.Wb; p.Hb = s.Hb; p.Bb = s.Bb;
    p.OW = s.OW; p.OH = s.OH; p.OB = s.OB;
    p.sw = s.sw; p.sh = s.sh;
    p.tiles_w = cdiv(s.OW, s.Wb);
    p.tiles_h = cdiv(s.OH, s.Hb);
    p.tiles_b = cdiv(s.OB, s.Bb);
    for (int t = 0; t < GEMM_MAX_TAPS; t++) { p.tap_dw[t] = s.tap_dw[t]; p.tap_dh[t] = s.tap_dh[t]; }
    p.out = e.out; p.ldo = e.ldo; p.bias = e.bias; p.resid = e.resid; p.ldr = e.ldr;
    p.row_add = e.row_add; p.row_map = e.row_map; p.valid_w = e.valid_w; p.gelu = e.gelu;
    p.amax_val = e.amax_val; p.amax_idx = e.amax_idx; p.amax_sum = e.amax_sum;
    p.rp = e.rp;
    const long m_tiles = (long)p.tiles_w * p.tiles_h * p.tiles_b;
    if (bn == 0 && e.epi == EPI_QKV) bn = (N % 256 == 0 && m_tiles * (N / 256) >= g_num_sms) ? 256 : 128;  // tiles of whole heads
    if (bn == 0) bn = gemm_pick_bn(N, e.epi, m_tiles);
    Q3_CHECK(e.epi != EPI_QKV || ((bn == 128 || bn == 256) && N % bn == 0 && e.rp.q != nullptr), 1, "gemm: fused q/k/v epilogue arguments");
    Q3_CHECK(e.epi != EPI_QKV || (((reinterpret_cast<uintptr_t>(e.out) | reinterpret_cast<uintptr_t>(e.rp.q) | reinterpret_cast<uintptr_t>(e.rp.kc) |
                                    reinterpret_cast<uintptr_t>(e.rp.pool)) & 31) == 0 && e.ldo % 16 == 0),
             1, "gemm: the fused q/k/v epilogue stores 32 bytes at a time: buffers must be 32-byte aligned");
    Q3_CHECK(N % bn == 0, 1, "gemm: N must be a multiple of the tile width");
    Q3_CHECK(e.epi != EPI_SWIGLU || bn % (2 * GU_UNIT) == 0, 1, "gemm: SwiGLU tiles must be multiples of 64 columns");
    p.tiles_n = N / bn;
    Q3_CHECK(e.epi == EPI_ARGMAX || e.out != nullptr, 1, "gemm: null output");

    if (simt) {
        SimtView v;
        v.A = a.ptr; v.C = a.C; v.W = a.W; v.H = a.H; v.B = a.B; v.sW = a.sW; v.sH = a.sH; v.sB = a.sB;
        v.OW = s.OW; v.OH = s.OH; v.OB = s.OB; v.sw = s.sw; v.sh = s.sh; v.taps = s.taps;
        for (int t = 0; t < GEMM_MAX_TAPS; t++) { v.tap_dw[t] = s.tap_dw[t]; v.tap_dh[t] = s.tap_dh[t]; }
        v.Wt = W; v.N = N;
        float* acc = nullptr;
        Q3_CUDA(cudaMallocAsync(&acc, sizeof(float) * rows * N, st));
        const long total = rows * N;
        simt_acc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(v, acc, rows);
        simt_epi_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(acc, rows, p, e.epi, bn);
        Q3_CUDA(cudaGetLastError());
        Q3_CUDA(cudaFreeAsync(acc, st));
        return;
    }

    CUtensorMap ta, tb;
    {
        const long sW = a.sW ? a.sW : a.C;
        const long sH = a.sH ? a.sH : sW * a.W;
        const long sB = a.sB ? a.sB : sH * a.H;
        cuuint64_t dims[4] = {(cuuint64_t)a.C, (cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)a.B};
        cuuint64_t str[3] = {(cuuint64_t)sW * 2, (cuuint64_t)sH * 2, (cuuint64_t)sB * 2};
        cuuint32_t box[4] = {(cuuint32_t)GEMM_BK, (cuuint32_t)(s.Wb * s.sw), (cuuint32_t)(s.Hb * s.sh), (cuuint32_t)s.Bb};
        cuuint32_t es[4] = {1, (cuuint32_t)s.sw, (cuuint32_t)s.sh, 1};
        make_tmap(&ta, a.ptr, 4, dims, str, box, es);
    }
    // CTA pairs (gemm2.cuh) for the big dense products: each CTA stages half of the weight tile
    const char* env2 = getenv("Q3ASR_2CTA");  // "0" never, "1" whenever the tile shape allows (tests), unset: large problems only
    const int mode2 = env2 && *env2 ? atoi(env2) : -1;
    // measured (profiles/): pairing lifts the plain products (q/k/v, o, down, fc2, conv_out: +9..19 %, 1.2-1.3 PFLOP/s) to the cuBLAS
    // ceiling; SwiGLU tiles are bound by their epilogues and the stride-2 convolutions by their TMA boxes, where it does not pay
    // (round 2: with the packed-fp32 GELU the fc1 tiles are no longer epilogue-bound and pairing pays there too: 3.20 -> 3.08 ms)
    const bool plain = (e.epi == EPI_NORMAL || e.epi == EPI_QKV) && s.sw == 1 && s.sh == 1;
    const bool pair = mode2 != 0 && !simt && (e.epi == EPI_NORMAL || e.epi == EPI_SWIGLU || e.epi == EPI_QKV) && (bn == 128 || bn == 160 || bn == 224 || bn == 256) &&
                      (mode2 == 1 || (plain && m_tiles * p.tiles_n >= 4L * g_num_sms)) && (e.epi != EPI_SWIGLU || bn % (2 * GU_UNIT) == 0);
    {
        const long K = (long)s.taps * a.C;
        cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
        cuuint64_t str[1] = {(cuuint64_t)K * 2};
        cuuint32_t box[2] = {(cuuint32_t)GEMM_BK, (cuuint32_t)(pair ? bn / 2 : bn)};
        cuuint32_t es[2] = {1, 1};
        make_tmap(&tb, W, 2, dims, str, box, es);
    }
    // Output tensor map of the plain epilogue (gemm.cuh: tiles staged in shared memory, one TMA store per 128 x 32 chunk): the
    // output rows are (b, h, w) positions in that order, so the map has the shape of the A map with N as the contiguous dimension
    // and the M-tile box {32 columns, Wb, Hb, Bb}; rows outside the tensor are clipped by the copy.  Not for scattered rows.
    CUtensorMap tc = ta;
    // Opt-in (Q3ASR_TMA_STORE=1): measured on the bench batch against the default, row-per-thread 256-bit stores, it is no faster
    // (encoder out-proj 0.89 vs 0.85 ms, fc1 3.11 vs 2.92, conv2 6.40 vs 6.22): once the stores are 32 bytes wide the epilogue is
    // no longer what bounds these products, and the staging costs a barrier of four warps per chunk.
    const char* env_ts = getenv("Q3ASR_TMA_STORE");
    const bool want_tma_out = env_ts != nullptr && atoi(env_ts) != 0;
    p.tma_out = 0;
    if (e.epi == EPI_NORMAL && e.row_map == nullptr && want_tma_out && (reinterpret_cast<uintptr_t>(e.out) & 15) == 0 && e.ldo % 8 == 0 &&
        (e.max_stages == 0 || pair)) {
        cuuint64_t dims[4] = {(cuuint64_t)N, (cuuint64_t)s.OW, (cuuint64_t)s.OH, (cuuint64_t)s.OB};
        cuuint64_t str[3] = {(cuuint64_t)e.ldo * 2, (cuuint64_t)e.ldo * 2 * s.OW, (cuuint64_t)e.ldo * 2 * s.OW * s.OH};
        cuuint32_t box[4] = {32u, (cuuint32_t)s.Wb, (cuuint32_t)s.Hb, (cuuint32_t)s.Bb};
        cuuint32_t es[4] = {1, 1, 1, 1};
        make_tmap(&tc, e.out, 4, dims, str, box, es, CU_TENSOR_MAP_SWIZZLE_64B);
        p.tma_out = 1;
    }
    if (pair) {
        const long super = ((m_tiles + 1) / 2) * p.tiles_n;
        const int grid2 = 2 * (int)std::min<long>(super, g_num_sms / 2);
        switch (bn) {
            case 128: launch_bn2<128>(e.epi, ta, tb, tc, p, grid2, st); break;
            case 160: launch_bn2<160>(e.epi, ta, tb, tc, p, grid2, st); break;
            case 224: launch_bn2<224>(e.epi, ta, tb, tc, p, grid2, st); break;
            default: launch_bn2<256>(e.epi, ta, tb, tc, p, grid2, st); break;
        }
        Q3_CUDA(cudaGetLastError());
        g_launches++;
        return;
    }
    const long tiles = m_tiles * p.tiles_n;
    const int grid = (int)std::min<long>(tiles, g_num_sms);
    switch (bn) {
        case 32: launch_bn<32>(e.epi, ta, tb, tc, p, e.max_stages, grid, st); break;
        case 64: launch_bn<64>(e.epi, ta, tb, tc, p, e.max_stages, grid, st); break;
        case 128: launch_bn<128>(e.epi, ta, tb, tc, p, e.max_stages, grid, st); break;
        case 160: launch_bn<160>(e.epi, ta, tb, tc, p, e.max_stages, grid, st); break;
        case 224: launch_bn<224>(e.epi, ta, tb, tc, p, e.max_stages, grid, st); break;
        case 256: launch_bn<256>(e.epi, ta, tb, tc, p, e.max_stages, grid, st); break;
        default: throw Error(1, "gemm: unsupported tile width " + std::to_string(bn));
    }
    Q3_CUDA(cudaGetLastError());
    g_launches++;
}

void gemm(const bf16* A, int lda, int M, int K, const bf16* W, int N, const GemmEpiArgs& e, cudaStream_t st, bool simt, int bn) {
    GemmA a;
    a.ptr = A; a.C = K; a.W = M; a.H = 1; a.B = 1; a.sW = lda;
    GemmShape s;
    s.Wb = GEMM_BM; s.OW = M;
    gemm_conv(a, s, W, N, e, st, simt, bn);
}

unsigned long long gemm_launch_count() { return g_launches; }

// ------------------------------------------------------------------------------------------
// decode-step weight-streaming GEMM
// ------------------------------------------------------------------------------------------
namespace {
template <int NB, int EPI, bool DEEP>
void launch_skinny(const CUtensorMap& tw, const CUtensorMap& tx, const SkinnyDev& p, dim3 grid, cudaStream_t st) {
    static PerDeviceOnce attr_once;
    attr_once([] {
        Q3_CUDA(cudaFuncSetAttribute(gemm_skinny_kernel<NB, EPI, DEEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, sk_smem_bytes(NB, DEEP)));
    });
    launch_kernel(gemm_skinny_kernel<NB, EPI, DEEP>, grid, 256, sk_smem_bytes(NB, DEEP), st, tw, tx, p);
}
template <int NB>
void launch_skinny_nb(int epi, bool deep, const CUtensorMap& tw, const CUtensorMap& tx, const SkinnyDev& p, dim3 grid, cudaStream_t st) {
    switch (epi) {
        case SK_PARTIAL:
            if (deep) launch_skinny<NB, SK_PARTIAL, true>(tw, tx, p, grid, st); else launch_skinny<NB, SK_PARTIAL, false>(tw, tx, p, grid, st);
            break;
        case SK_STORE:
            if (deep) launch_skinny<NB, SK_STORE, true>(tw, tx, p, grid, st); else launch_skinny<NB, SK_STORE, false>(tw, tx, p, grid, st);
            break;
        default: throw Error(1, "gemm_skinny: bad epilogue");
    }
}
}  // namespace

int gemm_skinny_splits(int N, int K, int epi) {
    if (epi == SK_STORE) return 1;
    const int tiles_n = cdiv(N, SK_BM), num_kb = cdiv(K, SK_BK);
    int splits = std::min(num_kb, std::max(1, g_num_sms / tiles_n));
    const int per = cdiv(num_kb, splits);
    return cdiv(num_kb, per);  // no empty slices
}

void gemm_skinny(const bf16* X, int ldx, int Mtok, int K, const bf16* W, int N, int epi, void* out, int ldo, cudaStream_t st) {
    Q3_CHECK(Mtok > 0 && Mtok <= SKINNY_MAX_ROWS, 1, "gemm_skinny: 1..256 token rows per launch");
    Q3_CHECK(K % 8 == 0 && ldx % 8 == 0 && N > 0, 1, "gemm_skinny: K and ldx must be multiples of 8");
    const int nb = Mtok <= 16 ? 16 : Mtok <= 32 ? 32 : Mtok <= 64 ? 64 : Mtok <= 128 ? 128 : 256;
    SkinnyDev p;
    memset(&p, 0, sizeof(p));
    p.N = N;
    p.Mtok = Mtok;
    p.num_kb = cdiv(K, SK_BK);
    const int splits = gemm_skinny_splits(N, K, epi);
    p.kb_per_split = cdiv(p.num_kb, splits);
    // ring depth: see skinny.cuh.  A long K slice is bandwidth-bound: half as many bytes again in flight (measured on 1.7B, 64
    // sequences: 63.3 -> 60.8 us per layer; 0.6B, whose slices are 2-4 blocks, is fastest with the 96 KB ring)
    static const int deep_kb = getenv("Q3ASR_SK_DEEP_KB") ? atoi(getenv("Q3ASR_SK_DEEP_KB")) : 8;
    const bool deep = p.kb_per_split >= deep_kb;
    p.out = out;
    p.ldo = ldo;
    p.split_stride = (long long)Mtok * N;
    CUtensorMap tw, tx;
    {
        cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
        cuuint64_t str[1] = {(cuuint64_t)K * 2};
        cuuint32_t box[2] = {(cuuint32_t)SK_BK, (cuuint32_t)SK_BM};
        cuuint32_t es[2] = {1, 1};
        make_tmap(&tw, W, 2, dims, str, box, es);
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Mtok};
        cuuint64_t str[1] = {(cuuint64_t)ldx * 2};
        cuuint32_t box[2] = {(cuuint32_t)SK_BK, (cuuint32_t)nb};
        cuuint32_t es[2] = {1, 1};
        make_tmap(&tx, X, 2, dims, str, box, es);
    }
    const dim3 grid(cdiv(N, SK_BM), splits);
    switch (nb) {
        case 16: launch_skinny_nb<16>(epi, deep, tw, tx, p, grid, st); break;
        case 32: launch_skinny_nb<32>(epi, deep, tw, tx, p, grid, st); break;
        case 64: launch_skinny_nb<64>(epi, deep, tw, tx, p, grid, st); break;
        case 128: launch_skinny_nb<128>(epi, deep, tw, tx, p, grid, st); break;
        default: launch_skinny_nb<256>(epi, deep, tw, tx, p, grid, st); break;
    }
    Q3_CUDA(cudaGetLastError());
    g_launches++;
}

namespace {
template <int NB, bool LSE>
void launch_lmhead_k(const CUtensorMap& tw, const CUtensorMap& tx, const LmHeadDev& p, int grid, cudaStream_t st) {
    static PerDeviceOnce attr_once;
    attr_once([] {
        Q3_CUDA(cudaFuncSetAttribute(lmhead_argmax_kernel<NB, LSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, lmh_smem_bytes(NB, LSE)));
    });
    launch_kernel(lmhead_argmax_kernel<NB, LSE>, grid, 256, lmh_smem_bytes(NB, LSE), st, tw, tx, p);
}
template <int NB>
void launch_lmhead(const CUtensorMap& tw, const CUtensorMap& tx, const LmHeadDev& p, int grid, cudaStream_t st) {
    if (p.amax_sum) launch_lmhead_k<NB, true>(tw, tx, p, grid, st);
    else launch_lmhead_k<NB, false>(tw, tx, p, grid, st);
}
}  // namespace

int lmhead_tiles(int N) { return cdiv(N, SK_BM); }

void lmhead_argmax(const bf16* X, int ldx, int Mtok, int K, const bf16* W, int N, float* amax_val, int* amax_idx, cudaStream_t st,
                   float* amax_sum) {
    Q3_CHECK(Mtok > 0 && Mtok <= SKINNY_MAX_ROWS, 1, "lmhead_argmax: 1..256 token rows per launch");
    Q3_CHECK(K % 8 == 0 && ldx % 8 == 0 && N > 0 && amax_val && amax_idx, 1, "lmhead_argmax: bad argument");
    const int nb = Mtok <= 16 ? 16 : Mtok <= 32 ? 32 : Mtok <= 64 ? 64 : Mtok <= 128 ? 128 : 256;
    LmHeadDev p;
    memset(&p, 0, sizeof(p));
    p.N = N;
    p.Mtok = Mtok;
    p.num_kb = cdiv(K, SK_BK);
    p.tiles = lmhead_tiles(N);
    p.amax_val = amax_val;
    p.amax_idx = amax_idx;
    p.amax_sum = amax_sum;
    CUtensorMap tw, tx;
    {
        cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
        cuuint64_t str[1] = {(cuuint64_t)K * 2};
        cuuint32_t box[2] = {(cuuint32_t)SK_BK, (cuuint32_t)SK_BM};
        cuuint32_t es[2] = {1, 1};
        make_tmap(&tw, W, 2, dims, str, box, es);
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Mtok};
        cuuint64_t str[1] = {(cuuint64_t)ldx * 2};
        cuuint32_t box[2] = {(cuuint32_t)SK_BK, (cuuint32_t)nb};
        cuuint32_t es[2] = {1, 1};
        make_tmap(&tx, X, 2, dims, str, box, es);
    }
    const int grid = std::min(p.tiles, g_num_sms);
    switch (nb) {
        case 16: launch_lmhead<16>(tw, tx, p, grid, st); break;
        case 32: launch_lmhead<32>(tw, tx, p, grid, st); break;
        case 64: launch_lmhead<64>(tw, tx, p, grid, st); break;
        case 128: launch_lmhead<128>(tw, tx, p, grid, st); break;
        default: launch_lmhead<256>(tw, tx, p, grid, st); break;
    }
    Q3_CUDA(cudaGetLastError());
    g_launches++;
}

void argmax_reduce(const float* val, const int* idx, int rows, int tiles, int32_t* out, float* out_val, cudaStream_t st) {
    if (rows <= 0) return;
    launch_kernel(argmax_reduce_kernel, rows, 256, 0, st, val, idx, rows, tiles, out, out_val);
}

void argmax_lse_reduce(const float* val, const int* idx, const float* tile_sum, const float* tile_max, const bf16* raw, int ld, int rows,
                       int tiles, int32_t* out, float* out_val, float* out_lp, cudaStream_t st) {
    if (rows <= 0) return;
    Q3_CHECK(tile_sum != nullptr && out_lp != nullptr, 1, "argmax_lse_reduce: null sums / output");
    launch_kernel(argmax_lse_reduce_kernel, rows, 256, 0, st, val, idx, tile_sum, tile_max, raw, ld, rows, tiles, out, out_val, out_lp);
}

}  // namespace q3
