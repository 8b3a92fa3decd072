// ops.cuh — the non-GEMM kernels of the encoder and decoder (ops.cu, attention.cu).
#pragma once
#include "common.cuh"

namespace q3 {

constexpr int KV_PAGE = 32;  // tokens per KV-cache page

// ---- encoder ----
// conv2d1 (1 -> C channels, 3x3, stride 2, pad 1) + exact GELU, fp32 math on the fp32 mel, bf16 NHWC output.
// AudioEncoder.swift:380-410 (chunk extraction, zero padding of the last chunk, conv2d1, gelu).
struct Conv1Chunk {
    long long mel_off;  // start of the clip's [128, T] block
    int T;              // frames of the clip (row pitch)
    int f0;             // first frame of the chunk
    int len;            // valid frames in the chunk
    int w0;             // padded chunk width (frames >= w0 are convolution padding)
};
void conv1_launch(const float* mel, const Conv1Chunk* chunks, int n_chunks, const bf16* w /*[C,3,3,1]*/, const bf16* bias, int C,
                  int chunk_w /*100*/, bf16* out /*[n_chunks,64,chunk_w/2,C]*/, cudaStream_t st);

// LayerNorm over the last dim (biased variance, fp32 statistics), bf16 in/out.  d % 128 == 0, d <= 2048.
void layernorm_launch(const bf16* x, const bf16* w, const bf16* b, bf16* y, int rows, int d, float eps, cudaStream_t st);
// RMSNorm; row_index (optional) gathers input rows: y[r] = norm(x[row_index[r]]).
void rmsnorm_launch(const bf16* x, const bf16* w, bf16* y, int rows, int d, float eps, const int* row_index, cudaStream_t st);

// ---- attention (attention.cu) ----
// Multi-head attention over independent segments of a packed row list (encoder windows, decoder prompts).
// q/k/v/o are row-major with the given leading dimensions; head h of q lives at columns [h*HD, (h+1)*HD),
// kv head h/group likewise in k and v.  causal: key j visible to query i iff j <= i (same segment).
struct AttnSegs {
    const int* row0;  // [n_segs] first row of each segment
    const int* len;   // [n_segs]
    int n_segs;
    int max_len;
};
void flash_attn_launch(const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv, bf16* o, int ldo, const AttnSegs& segs,
                       int heads, int group, int head_dim, bool causal, float scale, cudaStream_t st);

// The same contract on tcgen05 / TMEM / TMA (attention_tc.cu); total_rows = rows of the packed q/k/v buffers.
void flash_attn_tc_launch(const bf16* q, int ldq, const bf16* k, int ldk, const bf16* v, int ldv, bf16* o, int ldo, const AttnSegs& segs,
                          int total_rows, int heads, int group, int head_dim, bool causal, float scale, cudaStream_t st);

// ---- decoder ----
// x[r] = audio_src[r] >= 0 ? audio[audio_src[r]] : embed[ids[r]]   (Qwen3ASR.swift:236-244)
void embed_splice_launch(const int32_t* ids, const int* audio_src, const bf16* embed, const bf16* audio, bf16* x, int rows, int h,
                         cudaStream_t st);

struct KvCache {
    bf16* pool;             // [pages][layers][2][kv_heads][KV_PAGE][head_dim]
    const int* page_table;  // [n_seqs][max_pages]
    int max_pages;
    int layers, kv_heads, head_dim;
};
// rope_tab[pos][i] = (cos, sin)(pos * theta^(-2i/128)), i < 64 (head_dim 128), for pos < n_pos
// tab_t (optional): the same table dimension-major, [64][n_pos]
void rope_table_launch(const float* inv_freq, int n_pos, float2* tab, float2* tab_t, cudaStream_t st);
// Per (row, head): q/k RMSNorm over head_dim, split-half RoPE at pos[row], v passthrough; writes q to qout
// [rows, heads*hd], k/v to the paged cache (slot pos[row] of sequence row_seq[row]) and, if kc/vc != null, to
// contiguous [rows, kv_heads*hd] buffers for the prefill attention.  FloatTextDecoder.swift:85-102.
void qknorm_rope_kv_launch(const bf16* qkv, int ld, const bf16* qw, const bf16* kw, const int* pos, const int* row_seq, int rows,
                           int heads, int kv_heads, float eps, const float2* rope_tab, bf16* qout, bf16* kc, bf16* vc,
                           const KvCache& cache, int layer, cudaStream_t st);
// One query token per sequence against its paged cache (kv_len[seq] keys, the new token included), GQA.
void decode_attn_launch(const bf16* q /*[n_seqs, heads*hd]*/, const KvCache& cache, int layer, const int* kv_len, int n_seqs, int heads,
                        float scale, bf16* out, cudaStream_t st);

// Decode step, fused: sums the split-K partials of the QKV product (fp32 [splits][n_seqs][nqkv]), applies q/k-norm + RoPE,
// appends k/v to the cache and attends (one launch instead of qknorm_rope_kv + decode_attn).
// force (kernel tests): 0 = the choice for this batch and SM count (environment switches included); 1 = the split tensor-core variant
// (needs split_part / split_cnt), 2 / 8 = the tensor-core kernel with 2 / 8 warps, 4 / 16 = the SIMT kernel with 4 / 16 warps.
void decode_attn_fused_launch(const float* qkv_part, int splits, long long split_stride, int nqkv, const bf16* qw, const bf16* kw,
                              const int* pos, float eps, const float2* rope_tab, const KvCache& cache, int layer, const int* kv_len,
                              int n_seqs, int heads, float scale, bf16* out, int num_sms, cudaStream_t st, float* split_part = nullptr,
                              int* split_cnt = nullptr, int force = 0);
// scratch of the split variant (two single-warp CTAs per (sequence, kv head)): floats for the partials, counters (zero before the first launch)
constexpr size_t decode_attn_split_floats(size_t n_seqs, size_t kv_heads) { return n_seqs * kv_heads * 2 * 264; }
// x += bf16(sum of split-K partials) (in place), y = RMSNorm(x) * w.  d % 128 == 0, d <= 2048.
void reduce_resid_rmsnorm_launch(const float* part, int splits, long long split_stride, bf16* x, const bf16* w, bf16* y, int rows, int d,
                                 float eps, cudaStream_t st);

// Greedy bookkeeping after each LM-head argmax (Qwen3ASR.swift:344-389): appends the token, handles EOS,
// advances positions, selects the next input token (the argmax, or forced[step] when teacher forcing).
struct DecodeState {
    int32_t* next_tok;    // [n_seqs] argmax of this step (input)
    float* next_val;      // [n_seqs] its logit (input, may be null)
    int32_t* cur_tok;     // [n_seqs] token fed to the next step (output)
    int* pos;             // [n_seqs] position of the next token
    int* kv_len;          // [n_seqs]
    int32_t* out_ids;     // [n_seqs, max_tokens]
    float* out_val;       // [n_seqs, max_tokens] or null
    float* next_lp = nullptr;  // [n_seqs] log-probability of this step's token (input, may be null)
    float* out_lp = nullptr;   // [n_seqs, max_tokens] or null
    int* out_len;         // [n_seqs]
    int* finished;        // [n_seqs]
    int* n_active;        // [1]
    const int* slot_seq;  // [rows] sequence of every decode row, or null (identity): after a compaction the rows are the still-active sequences
    const int32_t* forced;  // [n_seqs? no: steps] or null
    int* step;            // [1] device-side step counter
    int max_tokens;
    int eos;
    int stop_on_eos;
};
// per_seq (continuous batching): out_ids / out_lp are indexed by each sequence's own out_len instead of the batch step; a sequence also
// finishes at max_tokens (stop_on_eos or not), and a finished row no longer advances pos / kv_len.  Needs slot_seq.
void decode_advance_launch(const DecodeState& s, int n_seqs, cudaStream_t st, bool per_seq = false);
// Drops the finished sequences from the decode rows (Qwen3ASR.swift:378-379 stops an utterance at EOS; a batched loop has to take it
// out of the batch, or its KV pages and a column of every product keep being streamed): the rows whose sequence is still active
// move to the front, in order, together with their token / position / cache length / page-table row.  One CTA; rows <= 1024.
// page_in / page_out: [rows][max_pages] (distinct buffers).  slot_seq is updated in place (identity on entry if it was never set).
// partition_cap > 0 (continuous batching): a stable partition of the page table instead — the finished rows' page-table rows follow
// the live ones and rows [rows, partition_cap) are copied as they are, so rows [live, partition_cap) of page_out name free blocks.
void decode_compact_launch(int rows, const int* finished, int* slot_seq, int32_t* cur_tok, int* pos, int* kv_len, const int* page_in,
                           int* page_out, int max_pages, cudaStream_t st, int partition_cap = 0);
// Continuous batching: step 0 of a freshly prefilled group of k utterances (request sequences seq0 ..), appended to the resident decode
// state at rows [row0, row0 + k): slot_seq, cur_tok = tok[j], pos = prompt_len[j], kv_len = prompt_len[j] + 1, out_ids / out_val /
// out_lp [q][0], out_len[q] = 1, finished[q] on EOS (stop_on_eos) or max_tokens <= 1; n_active grows by the rows still alive.
void decode_admit_launch(const DecodeState& s, const int32_t* tok, const float* val, const float* lp, const int* prompt_len, int row0, int k,
                         int seq0, cudaStream_t st);

// Decoder knobs of Qwen3DecodingOptions (Qwen3ASR.swift:13-51) applied on the device: the reference pulls the [vocab] logits to
// the CPU every token (pickNextToken, Qwen3ASR.swift:449-520); here one CTA per sequence applies the same three edits while it
// scans the row for the argmax — sign-aware repetition penalty over the tokens generated so far, the no-repeat-n-gram mask,
// logits / T + Gumbel(0,1) — with the generated set and the forbidden set as vocabulary bitmaps in shared memory.
struct SamplingParams {
    float repetition_penalty = 1.0f;
    int no_repeat_ngram = 0;
    float temperature = 0.0f;
    unsigned long long seed = 0;
};
// logits: [n_seqs, ld] (bf16 or fp32); gen_ids: [n_seqs, gen_stride] with gen_len[seq] valid entries; step: device counter that
// varies the noise per decode step (may be null).  A row's vocabulary is scanned by sample_parts(vocab) CTAs; each writes its best
// adjusted score and index to part_val / part_idx [n_seqs, sample_parts(vocab)], to be merged by argmax_reduce (gemm.cuh), which
// keeps the first maximum.  part_rmax / part_rsum (bf16 logits only, may be null): per slice also the maximum and the sum of
// exp(x - maximum) of the raw logits, for argmax_lse_reduce.
int sample_parts(int vocab);
void sample_launch(const bf16* logits_bf16, const float* logits_f32, int ld, int vocab, const int32_t* gen_ids, int gen_stride,
                   const int* gen_len, const SamplingParams& sp, const int* step, int n_seqs, float* part_val, int* part_idx,
                   cudaStream_t st, float* part_rmax = nullptr, float* part_rsum = nullptr);

void fill_i32_launch(int* p, int v, size_t n, cudaStream_t st);
void bf16_to_f32_launch(const bf16* in, float* out, size_t n, cudaStream_t st);
void f32_to_bf16_launch(const float* in, bf16* out, size_t n, cudaStream_t st);
void f16_to_bf16_launch(const uint16_t* in, bf16* out, size_t n, cudaStream_t st);
// deterministic random init (see model.cu / oracle/weights.py): out[i] = bf16(scale * irwin_hall4(seed, i))
void random_init_launch(bf16* out, size_t n, uint64_t seed, float scale, cudaStream_t st, uint64_t row_seed = 0, int row_len = 0);
void fill_bf16_launch(bf16* out, size_t n, float v, cudaStream_t st);

}  // namespace q3
