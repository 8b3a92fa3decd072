// model.h — kernel-ready weights and the resident-batch state of one handle.
#pragma once
#include <atomic>
#include <memory>
#include <thread>

#include "gemm.cuh"
#include "handle.h"
#include "megastep_params.h"
#include "ops.cuh"

namespace q3 {

struct EncLayerW {
    bf16 *ln1_w, *ln1_b, *qkv_w, *qkv_b, *o_w, *o_b, *ln2_w, *ln2_b, *fc1_w, *fc1_b, *fc2_w, *fc2_b;
};
struct DecLayerW {
    bf16 *in_ln, *qkv_w, *q_norm, *k_norm, *o_w, *post_ln, *gu_w, *down_w;
};

struct Model {
    // encoder
    bf16 *conv1_w, *conv1_b, *conv2_w, *conv2_b, *conv3_w, *conv3_b, *conv_out_w;
    std::vector<EncLayerW> enc;
    bf16 *ln_post_w, *ln_post_b, *proj1_w, *proj1_b, *proj2_w, *proj2_b;
    float* pe = nullptr;  // [tokens per chunk][d_model] sinusoidal positions, fp32
    // decoder
    bf16* embed;
    std::vector<DecLayerW> dec;
    bf16* final_norm;
    // forced aligner: classification head padded with zero rows to a multiple of 64 classes (GEMM tile width)
    bf16 *cls_w = nullptr, *cls_b = nullptr;
    int cls_pad = 0;
    float* inv_freq = nullptr;  // [head_dim/2]
    std::vector<void*> owned;   // derived device buffers
    size_t owned_bytes = 0;
};

// geometry derived from the config
struct Geom {
    int chunk;       // frames per conv chunk (2 * n_window = 100)
    int w1, w2, w3;  // conv output widths of a full chunk (50, 25, 13)
    int tpc;         // tokens per full chunk (= w3)
    int win_mult;    // n_window_infer / chunk (8)
    int C;           // conv channels
    explicit Geom(const q3asr_config& c) {
        chunk = 2 * c.enc_n_window;
        w1 = (chunk - 1) / 2 + 1;
        w2 = (w1 - 1) / 2 + 1;
        w3 = (w2 - 1) / 2 + 1;
        tpc = w3;
        win_mult = c.enc_n_window_infer / chunk;
        C = c.enc_conv_ch;
    }
};
inline int conv_len(int x) { return (x - 1) / 2 + 1; }
inline int conv_len3(int x) { return conv_len(conv_len(conv_len(x))); }

struct ClipInfo {
    int n = 0, frames = 0;
    int chunk0 = 0, nchunks = 0;
    int tok0 = 0, ntok = 0;
    int win_size = 0;
    int row0 = 0, prompt_len = 0, audio_at = 0;
};

// Host side of a batch upload that is still running (forward.cu batch_upload): worker threads copy the caller's clips into the
// pinned staging area and queue their host -> device copies; `recorded[b]` turns 1 once clip b's copy is queued and its event
// recorded (-1: it failed).  The threads borrow the caller's sample buffers, so the job is always joined before the API call that
// started it returns (finish_upload / the destructor).
struct UploadJob {
    std::vector<std::thread> workers;
    std::vector<cudaError_t> werr;
    std::unique_ptr<std::atomic<int>[]> recorded;
    std::vector<const float*> pcm;
    std::vector<size_t> n_in, n16, raw_off;
    std::vector<long long> in_off;
    std::vector<int> rates;  // empty: every clip is 16 kHz
    ~UploadJob() {
        for (auto& t : workers)
            if (t.joinable()) t.join();
    }
};

struct BatchState {
    std::unique_ptr<UploadJob> upload;  // non-null while the staging threads of the current batch may still be running
    int B = 0;
    MelPlan mel;
    std::vector<ClipInfo> clips;
    std::vector<int32_t> prompt_ids;  // packed
    int n_chunks = 0, n_tok = 0, n_win = 0, max_win = 0;
    int mel_next = 0;              // clips [0, mel_next) have had their mel kernel launched in this run
    bool copy_events = false;      // the clips of this batch were uploaded on the copy stream (one event per clip in Handle::copy_ev)
    std::vector<char> copy_waited; // the compute stream already waits for this clip's copy
    int R = 0, max_prompt = 0;
    int max_tokens = 0;      // decode capacity the KV pages were reserved for
    int pages_per_seq = 0;
    bool has_audio = false, mel_done = false, enc_done = false, prefill_done = false;
    bool sampler_on = false;   // decoder knobs active: full logits + sample_kernel instead of the fused argmax epilogue
    SamplingParams sampling;
    bool logprobs_on = false;  // per-token log-probabilities: the LM head also reduces the log-sum-exp (q3asr_batch_set_logprobs)
    int steps_done = 0;
    // decode rows: the sequences still being decoded (B until a compaction drops the finished ones; stop_on_eos only)
    int dec_rows = 0;
    int page_cur = 0;             // which of page_tab / page_tab2 the decode rows index through
    bool slot_map_on = false;     // st_slot_seq holds the row -> sequence map (identity until the first compaction)
    unsigned long long stat_row_steps = 0, stat_steps = 0, stat_compactions = 0;  // q3asr_decode_stats
    // continuous batching (transcribe_continuous): the resident state decodes a whole request of n_seqs utterances through its B rows
    int n_seqs = 0;               // sequences the outputs (out_ids / out_lp / out_len / finished) are sized and indexed for; B otherwise
    int page_prompt = 0;          // prompt length the KV pages are planned for when it exceeds max_prompt (the request's longest prompt)
    bool per_seq_steps = false;   // decode_advance counts steps per sequence (admitted sequences start mid-loop)
    unsigned long long stat_admissions = 0, stat_admitted = 0;  // q3asr_decode_admissions
    // an admission group's state borrows the resident state's KV pool: its prefill writes through the resident page table from row
    // kv_row0 on (the freed rows' blocks)
    BatchState* kv_from = nullptr;
    int kv_row0 = 0;
    std::vector<int> plan_ints;   // host plan of a staged group, uploaded when it is admitted
    std::vector<int> up_rates;    // sample rates of a staged group (empty: all 16 kHz), converted when it is admitted
    std::vector<size_t> up_n, up_raw_off;

    // device buffers
    DevBuf pcm, mel_out, mel_clips, mel_gmax, mel_tmin;
    DevBuf raw_pcm;  // clips at other sample rates, before the conversion to 16 kHz
    DevBuf ints;  // all small int arrays, one upload
    // offsets into `ints` (in ints)
    size_t o_conv_chunks = 0;  // Conv1Chunk[] (as bytes, see model.cu)
    size_t o_vw1 = 0, o_vw2 = 0, o_vw3 = 0, o_rowmap = 0, o_win_row0 = 0, o_win_len = 0;
    size_t o_ids = 0, o_audio_src = 0, o_pos = 0, o_row_seq = 0, o_seq_row0 = 0, o_seq_len = 0, o_last_row = 0,
           o_ident = 0, o_pos0 = 0;
    DevBuf a1, a2, a3, ex, exn, eqkv, eatt, effn, audio;        // encoder activations
    DevBuf dx, dxn, dqkv, dq, dkc, datt, dact, dlast, dws; // decoder activations (dws: fp32 split-K partials of the decode step)
    DevBuf dattn_part, dattn_cnt;        // decode attention, split variant: stored partials and per-item arrival counters
    DevBuf mega_tab, dws2, mega_trace;   // persistent decode-step kernel (megastep.cu): tables + the second sub-batch's split-K partials
    HostBuf h_mega;
    MegaParams mega;
    int mega_nb = 0, mega_gu = 0;
    bool mega_ready = false;
    DevBuf kv_pool, rope_tab, rope_tab_t, page_tab, page_tab2, st_slot_seq;  // rope_tab_t: the table dimension-major (EPI_QKV)
     // page_tab: [B][pages_per_seq] (plan_pages)
    int rope_n = 0;          // positions tabulated in rope_tab
    DevBuf amax_val, amax_idx, amax_sum, logits, logits_bf;  // amax_sum: per-tile sums of exp(z - tile max) (logprobs_on only)
    // decode state (device); st_next_lp / st_out_lp: logprobs_on only
    DevBuf st_next_tok, st_next_val, st_cur_tok, st_pos, st_kv_len, st_out_ids, st_out_val, st_out_len, st_finished, st_scalars, st_forced;
    DevBuf st_next_lp, st_out_lp;
    HostBuf h_stage, h_ints, h_out, h_pages;
    cudaGraphExec_t step_graph = nullptr;
    int graph_B = 0;
    cudaEvent_t ev[5] = {nullptr};

    void bind(size_t* total) {
        for (DevBuf* b : all()) b->total = total;
    }
    std::vector<DevBuf*> all() {
        return {&pcm, &raw_pcm, &mel_out, &mel_clips, &mel_gmax, &mel_tmin, &ints, &a1, &a2, &a3, &ex, &exn, &eqkv, &eatt, &effn, &audio,
                &dx, &dxn, &dqkv, &dq, &dkc, &datt, &dact, &dlast, &dws, &dattn_part, &dattn_cnt, &dws2, &mega_tab, &mega_trace, &kv_pool, &rope_tab, &rope_tab_t, &page_tab, &page_tab2, &st_slot_seq, &amax_val, &amax_idx, &amax_sum, &logits, &logits_bf,
                &st_next_tok, &st_next_val, &st_cur_tok, &st_pos, &st_kv_len, &st_out_ids, &st_out_val, &st_out_len, &st_finished,
                &st_scalars, &st_forced, &st_next_lp, &st_out_lp};
    }
    ~BatchState() {
        for (DevBuf* b : all()) b->release();
        h_stage.release();
        h_ints.release();
        h_out.release();
        h_pages.release();
        h_mega.release();
        if (step_graph) cudaGraphExecDestroy(step_graph);
        for (auto& e : ev)
            if (e) cudaEventDestroy(e);
    }
};

// One decoder layer's prefill attention block (forward.cu, FloatTextDecoder.swift:77-117): the q‖k‖v product of the normed rows,
// per-head RMSNorm + split-half RoPE of q and k, k and v written into the paged cache, then the causal attention of every prompt.
// decoder_layers runs it on the batch's buffers and q3asr_debug_prefill_attention on the caller's, so the kernel tests see the
// product's own launches.
struct PrefillAttn {
    const bf16* xn;                       // [rows, hidden] normed hidden states
    const bf16 *w_qkv, *q_norm, *k_norm;  // [(heads + 2 kv_heads) * 128, hidden] in q | k | v row order; [128]; [128]
    int rows, hidden, heads, kv_heads;
    float eps, scale;
    const int *pos, *row_seq;             // [rows] position and page-table row of every packed row
    AttnSegs segs;                        // the prompts
    const float2 *rope, *rope_t;          // (cos, sin) tables [rope_n][64] and [64][rope_n]
    int rope_n;
    KvCache kc;
    int layer;
    bf16 *qkv, *q, *k, *att;              // [rows, nqkv] (the attention reads v from it), [rows, nq], [rows, nkv], [rows, nq]
};
// fuse_qkv: norm, RoPE and the cache write in the product's epilogue (EPI_QKV), else the plain product + qknorm_rope_kv_kernel;
// bn: the product's tile width (0: gemm's choice); attn: 0 the tcgen05 kernel, 1 the mma.sync kernel, -1 none.
// causal_pairs (sum over prompts of S(S+1)/2) only feeds the profile.
void prefill_attention(Handle* h, const PrefillAttn& a, bool fuse_qkv, int bn, int attn, double causal_pairs);

// persistent decode-step kernel (megastep.cu)
bool megastep_supported(const Handle* h, const BatchState* bs);
void megastep_prepare(Handle* h, BatchState* bs);
void megastep_launch(Handle* h, BatchState* bs);

}  // namespace q3
