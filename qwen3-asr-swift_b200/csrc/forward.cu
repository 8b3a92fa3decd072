// forward.cu — the batched transcription pipeline behind q3asr_batch_* / q3asr_transcribe_ids:
// host-side planning (chunks, audio tokens, attention windows, prompts, KV pages) and the kernel
// sequence  mel -> conv stack -> encoder layers -> prompt splice -> prefill -> greedy decode.
//
// Follows (paths relative to /root/reference/Sources/Qwen3ASR):
//   AudioEncoder.swift:362-511   chunking, conv stack, conv_out + positions, valid-token gather, windows, layers, projector
//   Qwen3ASR.swift:181-256       prompt layout, audio splice, prefill, tied LM head on the last position
//   Qwen3ASR.swift:317-390       greedy loop (token appended, then EOS check)
//   FloatTextDecoder.swift:35-226 decoder block
// B200 design notes: all utterances of a batch are packed row-wise (no padding to the longest one);
// every dense product is one launch of the persistent tcgen05 GEMM; the conv stack is walked in
// L2-sized groups of chunks; a decode step is a CUDA graph replayed max_tokens-1 times with the
// per-sequence state (positions, cache lengths, EOS flags) living on the device.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <thread>

#include "model.h"

namespace q3 {

void build_prompt(const q3asr_config& c, const q3asr_prompt* pr, int ntok, std::vector<int32_t>* ids, int* audio_at) {
    // Qwen3ASR.swift:196-233
    ids->insert(ids->end(), {c.tok_im_start, c.tok_system, c.tok_newline});
    if (pr && pr->context_ids && pr->n_context > 0) ids->insert(ids->end(), pr->context_ids, pr->context_ids + pr->n_context);
    ids->insert(ids->end(), {c.tok_im_end, c.tok_newline, c.tok_im_start, c.tok_user, c.tok_newline, c.tok_audio_start});
    *audio_at = (int)ids->size();
    ids->insert(ids->end(), (size_t)ntok, c.tok_audio_pad);
    ids->insert(ids->end(), {c.tok_audio_end, c.tok_im_end, c.tok_newline, c.tok_im_start, c.tok_assistant, c.tok_newline});
    if (pr && pr->language_ids && pr->n_language > 0) ids->insert(ids->end(), pr->language_ids, pr->language_ids + pr->n_language);
    if (!(pr && pr->raw_suffix)) ids->push_back(c.tok_asr_text);  // the aligner's template ends with the slotted text (ForcedAligner.swift:338-378)
}

namespace {

int env_int(const char* name, int def) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : def;
}

template <typename T>
size_t push_ints(std::vector<int>& buf, const std::vector<T>& v) {
    static_assert(sizeof(T) % sizeof(int) == 0, "int-multiple types only");
    // 16-byte aligned sub-arrays
    while (buf.size() % 4) buf.push_back(0);
    const size_t off = buf.size();
    const size_t n = v.size() * sizeof(T) / sizeof(int);
    buf.resize(off + n);
    if (n) memcpy(buf.data() + off, v.data(), n * sizeof(int));
    return off;
}

BatchState* fresh_state(Handle* h, std::unique_ptr<BatchState>& slot) {
    if (!slot) {
        slot.reset(new BatchState());
        slot->bind(&h->dev_bytes);
        for (auto& e : slot->ev) Q3_CUDA(cudaEventCreate(&e));
    }
    return slot.get();
}
BatchState* fresh_batch(Handle* h) { return fresh_state(h, h->batch); }

// outputs (out_ids, out_lp, out_len, finished) are sized for this many sequences
int seq_count(const BatchState* bs) { return std::max(bs->n_seqs, bs->B); }

// Plans the encoder side for clips with the given frame counts (mel already known or to be computed).
void plan_encoder(Handle* h, BatchState* bs, const std::vector<int>& frames, const std::vector<long long>& mel_off,
                  std::vector<int>* ints) {
    const Geom g(h->cfg);
    const int B = (int)frames.size();
    bs->clips.assign(B, ClipInfo());
    std::vector<Conv1Chunk> chunks;
    std::vector<int> vw1, vw2, vw3, rowmap, win_row0, win_len;
    int tok = 0, max_win = 0;
    for (int b = 0; b < B; b++) {
        ClipInfo& ci = bs->clips[b];
        const int T = frames[b];
        ci.frames = T;
        ci.chunk0 = (int)chunks.size();
        ci.nchunks = (T + g.chunk - 1) / g.chunk;
        ci.tok0 = tok;
        int maxv = 0;
        const int w0 = ci.nchunks > 1 ? g.chunk : T;  // max chunk length of this clip (AudioEncoder.swift:380)
        for (int k = 0; k < ci.nchunks; k++) {
            Conv1Chunk cc;
            cc.mel_off = mel_off[b];
            cc.T = T;
            cc.f0 = k * g.chunk;
            cc.len = std::min(g.chunk, T - cc.f0);
            cc.w0 = w0;
            chunks.push_back(cc);
            const int a1 = conv_len(w0), a2 = conv_len(a1), a3 = conv_len(a2);
            vw1.push_back(a1);
            vw2.push_back(a2);
            vw3.push_back(a3);
            const int v = conv_len3(cc.len);  // valid tokens of this chunk (:441-448)
            maxv = std::max(maxv, v);
            for (int t = 0; t < g.tpc; t++) rowmap.push_back(t < v ? tok + t : -1);
            tok += v;
        }
        ci.ntok = tok - ci.tok0;
        ci.win_size = maxv * g.win_mult;  // :463-465
        for (int s = 0; s < ci.ntok; s += ci.win_size) {
            win_row0.push_back(ci.tok0 + s);
            win_len.push_back(std::min(ci.win_size, ci.ntok - s));
            max_win = std::max(max_win, win_len.back());
        }
    }
    bs->n_chunks = (int)chunks.size();
    bs->n_tok = tok;
    bs->n_win = (int)win_row0.size();
    bs->max_win = max_win;
    bs->o_conv_chunks = push_ints(*ints, chunks);
    bs->o_vw1 = push_ints(*ints, vw1);
    bs->o_vw2 = push_ints(*ints, vw2);
    bs->o_vw3 = push_ints(*ints, vw3);
    bs->o_rowmap = push_ints(*ints, rowmap);
    bs->o_win_row0 = push_ints(*ints, win_row0);
    bs->o_win_len = push_ints(*ints, win_len);
}

void plan_decoder(Handle* h, BatchState* bs, const q3asr_prompt* prompts, int max_tokens, std::vector<int>* ints) {
    const q3asr_config& c = h->cfg;
    const int B = bs->B;
    std::vector<int> ids, audio_src, pos, row_seq, seq_row0, seq_len, last_row, ident, pos0;
    int row = 0, max_prompt = 0;
    for (int b = 0; b < B; b++) {
        ClipInfo& ci = bs->clips[b];
        std::vector<int32_t> p;
        build_prompt(c, prompts ? &prompts[b] : nullptr, ci.ntok, &p, &ci.audio_at);
        ci.row0 = row;
        ci.prompt_len = (int)p.size();
        for (int i = 0; i < ci.prompt_len; i++) {
            Q3_CHECK(p[i] >= 0 && p[i] < c.dec_vocab, Q3ASR_ERR_INVALID, "prompt token id out of range");
            ids.push_back(p[i]);
            const int a = i - ci.audio_at;
            audio_src.push_back(a >= 0 && a < ci.ntok ? ci.tok0 + a : -1);
            pos.push_back(i);
            row_seq.push_back(b);
        }
        seq_row0.push_back(row);
        seq_len.push_back(ci.prompt_len);
        pos0.push_back(ci.prompt_len - 1);
        row += ci.prompt_len;
        last_row.push_back(row - 1);
        ident.push_back(b);
        max_prompt = std::max(max_prompt, ci.prompt_len);
    }
    bs->R = row;
    bs->max_prompt = max_prompt;
    (void)max_tokens;  // the KV pages are planned separately (plan_pages): the decode capacity may grow until the prefill runs
    bs->o_ids = push_ints(*ints, ids);
    bs->o_audio_src = push_ints(*ints, audio_src);
    bs->o_pos = push_ints(*ints, pos);
    bs->o_row_seq = push_ints(*ints, row_seq);
    bs->o_seq_row0 = push_ints(*ints, seq_row0);
    bs->o_seq_len = push_ints(*ints, seq_len);
    bs->o_last_row = push_ints(*ints, last_row);
    bs->o_ident = push_ints(*ints, ident);
    bs->o_pos0 = push_ints(*ints, pos0);
}

// KV page table for a decode capacity of max_tokens per sequence: pages are handed out in order and freed with the batch.
// Its own device buffer, so that batch_run can re-plan for a larger max_tokens than the upload reserved (the reference's
// transcribe(maxTokens:) takes any value, Qwen3ASR.swift:131-136) as long as the prefill has not written any page yet.
void plan_pages(Handle* h, BatchState* bs, int max_tokens) {
    bs->max_tokens = max_tokens;
    bs->pages_per_seq = (std::max(bs->max_prompt, bs->page_prompt) + max_tokens + KV_PAGE - 1) / KV_PAGE;
    const size_t n = (size_t)bs->B * bs->pages_per_seq;
    bs->page_tab.reserve(n * sizeof(int));
    bs->page_tab2.reserve(n * sizeof(int));  // target of the next compaction of the decode rows
    bs->page_cur = 0;
    bs->h_pages.reserve(n * sizeof(int));
    int* t = bs->h_pages.as<int>();
    for (size_t i = 0; i < n; i++) t[i] = (int)i;
    Q3_CUDA(cudaMemcpyAsync(bs->page_tab.p, t, n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    Q3_CUDA(cudaStreamSynchronize(h->stream));  // h_pages is reused by the next plan
}

void upload_ints(Handle* h, BatchState* bs, const std::vector<int>& ints) {
    bs->ints.reserve(ints.size() * sizeof(int) + 16);
    bs->h_ints.reserve(ints.size() * sizeof(int) + 16);  // its own pinned buffer: sample copies from h_stage may still be in flight
    memcpy(bs->h_ints.p, ints.data(), ints.size() * sizeof(int));
    Q3_CUDA(cudaMemcpyAsync(bs->ints.p, bs->h_ints.p, ints.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    Q3_CUDA(cudaStreamSynchronize(h->stream));  // the staging buffers are reused by the next upload
}

void reserve_encoder(Handle* h, BatchState* bs) {
    const q3asr_config& c = h->cfg;
    const Geom g(c);
    const int grp = std::min(bs->n_chunks, std::max(1, env_int("Q3ASR_CONV_GROUP", 30)));
    const size_t d = c.enc_d_model;
    bs->a1.reserve((size_t)grp * 64 * g.w1 * g.C * 2);
    bs->a2.reserve((size_t)bs->n_chunks * 32 * g.w2 * g.C * 2);  // conv3 runs once over all chunks
    bs->a3.reserve((size_t)bs->n_chunks * 16 * g.w3 * g.C * 2);
    const size_t T = std::max(bs->n_tok, 1);
    bs->ex.reserve(T * d * 2);
    bs->exn.reserve(T * d * 2);
    bs->eqkv.reserve(T * 3 * d * 2);
    bs->eatt.reserve(T * d * 2);
    bs->effn.reserve(T * c.enc_ffn * 2);
    bs->audio.reserve(T * c.enc_out_dim * 2);
}

void reserve_decoder(Handle* h, BatchState* bs) {
    const q3asr_config& c = h->cfg;
    const size_t R = std::max(bs->R, bs->B), hd = c.dec_head_dim;
    const size_t nq = c.dec_heads * hd, nkv = c.dec_kv_heads * hd, H = c.dec_hidden;
    bs->dx.reserve(R * H * 2);
    bs->dxn.reserve(R * H * 2);
    bs->dqkv.reserve(R * (nq + 2 * nkv) * 2);
    bs->dq.reserve(R * nq * 2);
    bs->dkc.reserve(R * nkv * 2);
    {  // RoPE table for every position the KV pages can hold
        const int n_pos = bs->pages_per_seq * KV_PAGE;
        if (bs->rope_n < n_pos) {
            bs->rope_tab.reserve((size_t)n_pos * 64 * sizeof(float2));
            bs->rope_tab_t.reserve((size_t)n_pos * 64 * sizeof(float2));
            rope_table_launch(h->model->inv_freq, n_pos, bs->rope_tab.as<float2>(), bs->rope_tab_t.as<float2>(), h->stream);
            h->launches++;
            bs->rope_n = n_pos;
        }
    }
    bs->datt.reserve(R * nq * 2);
    bs->dact.reserve(R * c.dec_inter * 2);
    bs->dlast.reserve((size_t)bs->B * H * 2);
    if (bs->B <= SKINNY_MAX_ROWS) {  // split-K partials of the decode-step GEMMs
        const size_t Bq = bs->B;
        const size_t w1 = (size_t)gemm_skinny_splits((int)(nq + 2 * nkv), (int)H, SK_PARTIAL) * Bq * (nq + 2 * nkv);
        const size_t w2 = (size_t)gemm_skinny_splits((int)H, (int)nq, SK_PARTIAL) * Bq * H;
        const size_t w3 = (size_t)gemm_skinny_splits((int)H, c.dec_inter, SK_PARTIAL) * Bq * H;
        bs->dws.reserve(std::max(w1, std::max(w2, w3)) * 4);
        bs->dattn_part.reserve(decode_attn_split_floats(Bq, c.dec_kv_heads) * 4);
        const size_t cnt_bytes = Bq * c.dec_kv_heads * sizeof(int);
        if (cnt_bytes > bs->dattn_cnt.cap) {  // the counters return to zero after every launch: cleared when (re)allocated only
            bs->dattn_cnt.reserve(cnt_bytes);
            Q3_CUDA(cudaMemsetAsync(bs->dattn_cnt.p, 0, bs->dattn_cnt.cap, h->stream));
        }
    }
    const size_t page_elems = (size_t)c.dec_layers * 2 * c.dec_kv_heads * KV_PAGE * hd;
    if (!bs->kv_from) bs->kv_pool.reserve((size_t)bs->B * bs->pages_per_seq * page_elems * 2);  // an admission group writes the resident pool
    const size_t tiles = c.dec_vocab / 32;  // upper bound on LM-head n-tiles
    bs->amax_val.reserve((size_t)bs->B * tiles * 4);
    bs->amax_idx.reserve((size_t)bs->B * tiles * 4);
    const size_t B = bs->B, S = seq_count(bs), mt = std::max(bs->max_tokens, 1);
    bs->st_next_tok.reserve(B * 4);
    bs->st_next_val.reserve(B * 4);
    bs->st_cur_tok.reserve(B * 4);
    bs->st_pos.reserve(B * 4);
    bs->st_kv_len.reserve(B * 4);
    bs->st_out_ids.reserve(S * mt * 4);
    bs->st_out_val.reserve(S * mt * 4);
    bs->st_out_len.reserve(S * 4);
    bs->st_finished.reserve(S * 4);
    bs->st_slot_seq.reserve(B * 4);
    bs->st_scalars.reserve(64);
    if (bs->logprobs_on) {
        bs->amax_sum.reserve((size_t)bs->B * tiles * 4);
        bs->st_next_lp.reserve(B * 4);
        bs->st_out_lp.reserve(S * mt * 4);
    }
    bs->h_out.reserve(S * mt * 8 + S * 8 + 64);
}

// ---------------------------------------------------------------------------------------------
// stages
// ---------------------------------------------------------------------------------------------
}  // namespace

// Joins the staging threads of the current upload (if any) and reports their first error.
void finish_upload(BatchState* bs) {
    if (bs == nullptr || !bs->upload) return;
    std::unique_ptr<UploadJob> job = std::move(bs->upload);
    for (auto& t : job->workers)
        if (t.joinable()) t.join();
    for (cudaError_t e : job->werr) Q3_CUDA(e);
}

namespace {

// Host-side wait until clip b's copy has been queued on the copy stream and its event recorded.
void wait_recorded(BatchState* bs, int b) {
    if (!bs->upload) return;
    std::atomic<int>& f = bs->upload->recorded[(size_t)b];
    while (f.load(std::memory_order_acquire) == 0) std::this_thread::yield();
    if (f.load(std::memory_order_acquire) < 0) {
        finish_upload(bs);  // throws the worker's error
        throw Error(Q3ASR_ERR_CUDA, "batch_upload: a sample copy failed");
    }
}
// true while some clip's host -> device copy (batch_upload, copy stream) has not been queued or has not landed yet
bool copies_pending(Handle* h, BatchState* bs) {
    if (!bs->copy_events || bs->B <= 0) return false;
    if (bs->upload)
        for (int b = 0; b < bs->B; b++)
            if (bs->upload->recorded[(size_t)b].load(std::memory_order_acquire) == 0) return true;
    return cudaEventQuery(h->copy_ev[(size_t)bs->B - 1]) == cudaErrorNotReady;
}

// Log-mel of the clips [bs->mel_next, upto) (upto < 0: all that remain).  While the upload is still in flight the batch is taken in
// (up to) four groups of clips, each launch waiting only for its own clips' copies, so the caller (run_encoder) can interleave
// the convolution stack of a group with the copies of the next; with the samples resident it is one launch for the whole batch.
void run_mel(Handle* h, BatchState* bs, int upto = -1) {
    const int B = bs->B;
    if (upto < 0 || upto > B) upto = B;
    const int gsz = copies_pending(h, bs) ? (B + 3) / 4 : B;
    while (bs->mel_next < upto) {
        const int c0 = bs->mel_next, c1 = std::min(B, (c0 / gsz + 1) * gsz);
        if (bs->copy_events)
            for (int b = c0; b < c1; b++)
                if (!bs->copy_waited[(size_t)b]) {
                    wait_recorded(bs, b);
                    Q3_CUDA(cudaStreamWaitEvent(h->stream, h->copy_ev[(size_t)b], 0));
                    bs->copy_waited[(size_t)b] = 1;
                }
        double mel_bytes = 0;
        for (int b = c0; b < c1; b++) mel_bytes += 4.0 * bs->mel.clips[(size_t)b].n + 4.0 * MEL_BINS * bs->mel.clips[(size_t)b].frames;
        const int tile_lo = bs->mel.clips[(size_t)c0].tile0;
        const int tile_hi = c1 < B ? bs->mel.clips[(size_t)c1].tile0 : bs->mel.total_tiles;
        ProfScope ps(h, "mel", 0, mel_bytes);
        mel_launch_range(h->mel_tables, bs->pcm.as<float>(), bs->mel_out.as<float>(), bs->mel_clips.as<MelClip>(), c0, c1, tile_lo, tile_hi,
                         bs->mel.total_tiles, bs->mel_gmax.as<int>(), bs->mel_tmin.as<float>(), h->num_sms, h->stream);
        h->launches += 3;
        bs->mel_next = c1;
    }
    bs->mel_done = bs->mel_next >= B;
}

GemmEpiArgs epi_store(void* out, int ldo, const bf16* bias, int gelu = 0, const bf16* resid = nullptr, int ldr = 0) {
    GemmEpiArgs e;
    e.out = out; e.ldo = ldo; e.bias = bias; e.gelu = gelu; e.resid = resid; e.ldr = ldr;
    return e;
}

void run_encoder(Handle* h, BatchState* bs, const float* d_mel) {
    const q3asr_config& c = h->cfg;
    const Geom g(c);
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    const int* ints = bs->ints.as<int>();
    const int d = c.enc_d_model;
    if (bs->n_tok == 0) { bs->enc_done = true; return; }

    // ---- conv stack, walked in groups of chunks so conv1/conv2 activations stay L2-resident ----
    const int grp = std::min(bs->n_chunks, std::max(1, env_int("Q3ASR_CONV_GROUP", 30)));
    const Conv1Chunk* chunks = reinterpret_cast<const Conv1Chunk*>(ints + bs->o_conv_chunks);
    GemmShape s2, s3;
    s2.Wb = g.w2; s2.Hb = 1; s2.Bb = std::max(1, GEMM_BM / g.w2);
    s2.OW = g.w2; s2.OH = 32; s2.sw = 2; s2.sh = 2; s2.taps = 9;
    s3.Wb = g.w3; s3.Hb = 1; s3.Bb = std::max(1, GEMM_BM / g.w3);
    s3.OW = g.w3; s3.OH = 16; s3.sw = 2; s3.sh = 2; s3.taps = 9;
    for (int t = 0; t < 9; t++) {
        s2.tap_dw[t] = s3.tap_dw[t] = (signed char)(t % 3 - 1);
        s2.tap_dh[t] = s3.tap_dh[t] = (signed char)(t / 3 - 1);
    }
    for (int c0 = 0; c0 < bs->n_chunks; c0 += grp) {
        const int n = std::min(grp, bs->n_chunks - c0);
        if (d_mel == bs->mel_out.as<float>() && bs->mel_next < bs->B) {  // the mel stage was deferred: the upload is still in flight
            int hi = bs->mel_next;
            while (hi < bs->B && bs->clips[(size_t)hi].chunk0 < c0 + n) hi++;  // clips with a chunk in this group
            run_mel(h, bs, hi);
        }
        {
            ProfScope ps(h, "conv1", 2.0 * 9 * n * 64.0 * g.w1 * g.C, n * (128.0 * g.chunk * 4 + 64.0 * g.w1 * g.C * 2));
            conv1_launch(d_mel, chunks + c0, n, m.conv1_w, m.conv1_b, g.C, g.chunk, bs->a1.as<bf16>(), st);
        }
        h->launches++;
        GemmA a;
        a.ptr = bs->a1.as<bf16>(); a.C = g.C; a.W = g.w1; a.H = 64; a.B = n;
        a.sW = g.C; a.sH = (long)g.w1 * g.C; a.sB = 64L * g.w1 * g.C;
        s2.OB = n;
        GemmEpiArgs e2 = epi_store(bs->a2.as<bf16>() + (size_t)c0 * 32 * g.w2 * g.C, g.C, m.conv2_b, 1);
        e2.valid_w = ints + bs->o_vw2 + c0;
        {
            ProfScope ps(h, "conv2", 2.0 * n * 32.0 * g.w2 * g.C * 9.0 * g.C, 0);
            gemm_conv(a, s2, m.conv2_w, g.C, e2, st);
        }
    }
    if (d_mel == bs->mel_out.as<float>() && bs->mel_next < bs->B) run_mel(h, bs);
    // conv3 in one launch over every chunk: per group it would be 192 tiles on 148 SMs (two waves, the second 30 % full);
    // the conv2 output (24 MB per 32 chunks) is read back from HBM instead of L2, which costs far less than the idle SMs did.
    {
        GemmA a;
        a.ptr = bs->a2.as<bf16>(); a.C = g.C; a.W = g.w2; a.H = 32; a.B = bs->n_chunks;
        a.sW = g.C; a.sH = (long)g.w2 * g.C; a.sB = 32L * g.w2 * g.C;
        s3.OB = bs->n_chunks;
        GemmEpiArgs e3 = epi_store(bs->a3.p, g.C, m.conv3_b, 1);
        e3.valid_w = ints + bs->o_vw3;
        ProfScope ps(h, "conv3", 2.0 * bs->n_chunks * 16.0 * g.w3 * g.C * 9.0 * g.C, 0);
        gemm_conv(a, s3, m.conv3_w, g.C, e3, st);
    }
    // ---- conv_out over the [chunk, t, (f, c)] view of the conv3 output, + positions, gather valid tokens ----
    {
        GemmA a;
        a.ptr = bs->a3.as<bf16>(); a.C = g.C; a.W = g.w3; a.H = 16; a.B = bs->n_chunks;
        a.sW = g.C; a.sH = (long)g.w3 * g.C; a.sB = 16L * g.w3 * g.C;
        GemmShape s;
        s.Wb = g.w3; s.Hb = 1; s.Bb = std::max(1, GEMM_BM / g.w3);
        s.OW = g.w3; s.OH = 1; s.OB = bs->n_chunks;
        s.sw = 1; s.sh = 1; s.taps = 16;
        for (int f = 0; f < 16; f++) { s.tap_dw[f] = 0; s.tap_dh[f] = (signed char)f; }
        GemmEpiArgs e = epi_store(bs->ex.p, d, nullptr);
        e.row_add = m.pe;
        e.row_map = ints + bs->o_rowmap;
        ProfScope ps(h, "conv_out", 2.0 * bs->n_tok * (double)d * 16.0 * g.C, 0);
        gemm_conv(a, s, m.conv_out_w, d, e, st);
    }
    // ---- transformer layers over the packed tokens ----
    const int T = bs->n_tok;
    AttnSegs segs{ints + bs->o_win_row0, ints + bs->o_win_len, bs->n_win, bs->max_win};
    bf16 *x = bs->ex.as<bf16>(), *xn = bs->exn.as<bf16>(), *qkv = bs->eqkv.as<bf16>(), *att = bs->eatt.as<bf16>(),
         *ffn = bs->effn.as<bf16>();
    const bool attn_tc = env_int("Q3ASR_ATTN_MMASYNC", 0) == 0;  // tcgen05 attention unless the mma.sync checker kernel is asked for
    double win_pairs = 0;  // sum over windows of len^2 (attention work)
    for (const ClipInfo& ci : bs->clips)
        for (int s0 = 0; s0 < ci.ntok; s0 += ci.win_size) {
            const double L = std::min(ci.win_size, ci.ntok - s0);
            win_pairs += L * L;
        }
    for (int l = 0; l < c.enc_layers; l++) {
        const EncLayerW& w = m.enc[l];
        const double Td = T, dd = d, fd = c.enc_ffn;
        { ProfScope ps(h, "enc_ln", 0, 4.0 * Td * dd); layernorm_launch(x, w.ln1_w, w.ln1_b, xn, T, d, c.enc_ln_eps, st); }
        { ProfScope ps(h, "enc_qkv", 6.0 * Td * dd * dd, 0); gemm(xn, d, T, d, w.qkv_w, 3 * d, epi_store(qkv, 3 * d, w.qkv_b), st); }
        {
            ProfScope ps(h, "enc_attn", 4.0 * win_pairs * dd, 8.0 * Td * dd);
            if (attn_tc)
                flash_attn_tc_launch(qkv, 3 * d, qkv + d, 3 * d, qkv + 2 * d, 3 * d, att, d, segs, T, c.enc_heads, 1, 64, false, 0.125f, st);
            else
                flash_attn_launch(qkv, 3 * d, qkv + d, 3 * d, qkv + 2 * d, 3 * d, att, d, segs, c.enc_heads, 1, 64, false, 0.125f, st);
        }
        { ProfScope ps(h, "enc_out", 2.0 * Td * dd * dd, 0); gemm(att, d, T, d, w.o_w, d, epi_store(x, d, w.o_b, 0, x, d), st); }
        { ProfScope ps(h, "enc_ln", 0, 4.0 * Td * dd); layernorm_launch(x, w.ln2_w, w.ln2_b, xn, T, d, c.enc_ln_eps, st); }
        { ProfScope ps(h, "enc_fc1", 2.0 * Td * dd * fd, 0); gemm(xn, d, T, d, w.fc1_w, c.enc_ffn, epi_store(ffn, c.enc_ffn, w.fc1_b, 1), st); }
        { ProfScope ps(h, "enc_fc2", 2.0 * Td * dd * fd, 0); gemm(ffn, c.enc_ffn, T, c.enc_ffn, w.fc2_w, d, epi_store(x, d, w.fc2_b, 0, x, d), st); }
        h->launches += 3;
    }
    {
        ProfScope ps(h, "enc_proj", 2.0 * T * (double)d * (d + c.enc_out_dim), 0);
        layernorm_launch(x, m.ln_post_w, m.ln_post_b, xn, T, d, c.enc_ln_eps, st);
        gemm(xn, d, T, d, m.proj1_w, d, epi_store(att, d, m.proj1_b, 1), st);
        gemm(att, d, T, d, m.proj2_w, c.enc_out_dim, epi_store(bs->audio.p, c.enc_out_dim, m.proj2_b), st);
    }
    h->launches++;
    bs->enc_done = true;
}

KvCache kv_cache(Handle* h, BatchState* bs) {
    KvCache kc;
    if (bs->kv_from) {  // admission group: the resident pool, through the resident page table's rows from kv_row0 on
        const BatchState* r = bs->kv_from;
        kc.pool = r->kv_pool.as<bf16>();
        kc.page_table = (r->page_cur ? r->page_tab2 : r->page_tab).as<int>() + (size_t)bs->kv_row0 * r->pages_per_seq;
        kc.max_pages = r->pages_per_seq;
    } else {
        kc.pool = bs->kv_pool.as<bf16>();
        kc.page_table = (bs->page_cur ? bs->page_tab2 : bs->page_tab).as<int>();
        kc.max_pages = bs->pages_per_seq;
    }
    kc.layers = h->cfg.dec_layers;
    kc.kv_heads = h->cfg.dec_kv_heads;
    kc.head_dim = h->cfg.dec_head_dim;
    return kc;
}

// rows: packed token rows in bs->dx.  prefill: segs describe the prompts; decode: one row per sequence.
void decoder_layers(Handle* h, BatchState* bs, int rows, bool prefill) {
    const q3asr_config& c = h->cfg;
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    const int* ints = bs->ints.as<int>();
    const int H = c.dec_hidden, hd = c.dec_head_dim, nq = c.dec_heads * hd, nkv = c.dec_kv_heads * hd, nqkv = nq + 2 * nkv;
    const float scale = 1.0f / sqrtf((float)hd);
    bf16 *x = bs->dx.as<bf16>(), *xn = bs->dxn.as<bf16>(), *qkv = bs->dqkv.as<bf16>(), *q = bs->dq.as<bf16>(),
         *att = bs->datt.as<bf16>(), *act = bs->dact.as<bf16>();
    const KvCache kc = kv_cache(h, bs);
    const int* pos = prefill ? ints + bs->o_pos : bs->st_pos.as<int>();
    const int* row_seq = prefill ? ints + bs->o_row_seq : ints + bs->o_ident;
    AttnSegs segs{ints + bs->o_seq_row0, ints + bs->o_seq_len, bs->B, bs->max_prompt};
    const bool fuse_qkv = hd == 128 && env_int("Q3ASR_NO_QKV_FUSE", 0) == 0;  // "1": the separate norm + RoPE kernel (the checker)
    const int attn = env_int("Q3ASR_ATTN_MMASYNC", 0) == 0 ? 0 : 1;  // tcgen05 attention unless the mma.sync checker kernel is asked for
    double causal_pairs = 0;  // sum over prompts of S(S+1)/2
    for (const ClipInfo& ci : bs->clips) causal_pairs += 0.5 * ci.prompt_len * (ci.prompt_len + 1.0);
    for (int l = 0; l < c.dec_layers; l++) {
        const DecLayerW& w = m.dec[l];
        const double Rd = rows;
        ProfScope* ps = nullptr;
        auto tag = [&](const char* pre, const char* dec, double fl, double by) {
            delete ps;
            ps = new ProfScope(h, prefill ? pre : dec, fl, by);
        };
        tag("pre_norm", "dec_norm", 0, 4.0 * Rd * H);
        rmsnorm_launch(x, w.in_ln, xn, rows, H, c.dec_rms_eps, nullptr, st);
        if (prefill) {
            delete ps;
            ps = nullptr;
            const PrefillAttn pa{xn, w.qkv_w, w.q_norm, w.k_norm, rows, H, c.dec_heads, c.dec_kv_heads, c.dec_rms_eps, scale, pos, row_seq,
                                 segs, bs->rope_tab.as<float2>(), bs->rope_tab_t.as<float2>(), bs->rope_n, kc, l, qkv, q,
                                 bs->dkc.as<bf16>(), att};
            prefill_attention(h, pa, fuse_qkv, 0, attn, causal_pairs);
        } else {
            tag("pre_qkv", "dec_qkv", 2.0 * Rd * H * nqkv, 2.0 * H * nqkv);
            gemm(xn, H, rows, H, w.qkv_w, nqkv, epi_store(qkv, nqkv, nullptr), st);
            tag("pre_rope", "dec_rope", 0, 4.0 * Rd * nqkv);
            qknorm_rope_kv_launch(qkv, nqkv, w.q_norm, w.k_norm, pos, row_seq, rows, c.dec_heads, c.dec_kv_heads, c.dec_rms_eps,
                                  bs->rope_tab.as<float2>(), q, nullptr, nullptr, kc, l, st);
            tag("pre_attn", "dec_attn", 0, 0);
            decode_attn_launch(q, kc, l, bs->st_kv_len.as<int>(), rows, c.dec_heads, scale, att, st);
        }
        tag("pre_o", "dec_o", 2.0 * Rd * nq * H, 2.0 * nq * H);
        gemm(att, nq, rows, nq, w.o_w, H, epi_store(x, H, nullptr, 0, x, H), st);
        tag("pre_norm", "dec_norm", 0, 4.0 * Rd * H);
        rmsnorm_launch(x, w.post_ln, xn, rows, H, c.dec_rms_eps, nullptr, st);
        tag("pre_gateup", "dec_gateup", 4.0 * Rd * H * c.dec_inter, 4.0 * H * c.dec_inter);
        GemmEpiArgs eg;
        eg.epi = EPI_SWIGLU; eg.out = act; eg.ldo = c.dec_inter;
        gemm(xn, H, rows, H, w.gu_w, 2 * c.dec_inter, eg, st);
        tag("pre_down", "dec_down", 2.0 * Rd * H * c.dec_inter, 2.0 * H * c.dec_inter);
        gemm(act, c.dec_inter, rows, c.dec_inter, w.down_w, H, epi_store(x, H, nullptr, 0, x, H), st);
        delete ps;
        h->launches += 4;
    }
}

// RAII: kernels launched while this is alive may overlap their prologue with the previous kernel's tail (PDL)
struct PdlScope {
    bool prev;
    explicit PdlScope(bool on) : prev(pdl_enabled()) { pdl_enabled() = on; }
    ~PdlScope() { pdl_enabled() = prev; }
};

// Decode step for B <= SKINNY_MAX_ROWS sequences: weight-streaming split-K GEMMs (skinny.cuh) whose fp32 partials are
// consumed by fused kernels — 7 launches per layer.  On entry bs->dx holds the new token embeddings; on exit bs->dlast
// holds the final-norm hidden states (the LM-head input).
void decoder_layers_decode(Handle* h, BatchState* bs) {
    const q3asr_config& c = h->cfg;
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    const int B = bs->dec_rows;  // decode rows: the sequences still active
    const int H = c.dec_hidden, hd = c.dec_head_dim, nq = c.dec_heads * hd, nkv = c.dec_kv_heads * hd, nqkv = nq + 2 * nkv;
    const float scale = 1.0f / sqrtf((float)hd);
    bf16 *x = bs->dx.as<bf16>(), *xn = bs->dxn.as<bf16>(), *att = bs->datt.as<bf16>(), *act = bs->dact.as<bf16>();
    float* ws = bs->dws.as<float>();
    const KvCache kc = kv_cache(h, bs);
    const int s_qkv = gemm_skinny_splits(nqkv, H, SK_PARTIAL), s_o = gemm_skinny_splits(H, nq, SK_PARTIAL),
              s_dn = gemm_skinny_splits(H, c.dec_inter, SK_PARTIAL);
#ifdef Q3ASR_ABLATION  // `make ablation` only (tools/decode_ablation.py): the shipped library has no switch that changes results
    const int skip = env_int("Q3ASR_DEC_SKIP", 0);  // bit i drops kernel i of the layer
#else
    constexpr int skip = 0;
#endif
    double kv_bytes = 0;  // keys + values read by one layer's attention
    for (const ClipInfo& ci : bs->clips) kv_bytes += 2.0 * 2.0 * nkv * (ci.prompt_len + bs->steps_done);
    {
        ProfScope ps(h, "dec_norm", 0, 4.0 * B * H);
        rmsnorm_launch(x, m.dec[0].in_ln, xn, B, H, c.dec_rms_eps, nullptr, st);
        h->launches++;
    }
    if (bs->mega_ready) {  // all layers in one persistent kernel (megastep.cuh); the loop below is the multi-kernel path it replaces
        PdlScope no_pdl(false);
        // algorithmic bytes of the launch: every layer's weights once + the keys and values its attention reads
        const double w_bytes = 2.0 * ((double)H * nqkv + (double)nq * H + 3.0 * H * c.dec_inter);
        ProfScope ps(h, "dec_layers", 2.0 * B * c.dec_layers * w_bytes / 2.0, c.dec_layers * (w_bytes + kv_bytes));
        megastep_launch(h, bs);
        return;
    }
    for (int l = 0; l < c.dec_layers; l++) {
        const DecLayerW& w = m.dec[l];
        const bool last = l + 1 == c.dec_layers;
        {
            ProfScope ps(h, "dec_qkv", 2.0 * B * H * nqkv, 2.0 * H * nqkv);
            if (!(skip & 1)) gemm_skinny(xn, H, B, H, w.qkv_w, nqkv, SK_PARTIAL, ws, 0, st);
        }
        {
            ProfScope ps(h, "dec_attn", 0, kv_bytes);
            if (!(skip & 2)) decode_attn_fused_launch(ws, s_qkv, (long long)B * nqkv, nqkv, w.q_norm, w.k_norm, bs->st_pos.as<int>(), c.dec_rms_eps, bs->rope_tab.as<float2>(),
                                     kc, l, bs->st_kv_len.as<int>(), B, c.dec_heads, scale, att, h->num_sms, st, bs->dattn_part.as<float>(),
                                     bs->dattn_cnt.as<int>());
        }
        {
            ProfScope ps(h, "dec_o", 2.0 * B * nq * H, 2.0 * nq * H);
            if (!(skip & 4)) gemm_skinny(att, nq, B, nq, w.o_w, H, SK_PARTIAL, ws, 0, st);
        }
        {
            ProfScope ps(h, "dec_norm", 0, 4.0 * B * H);
            if (!(skip & 8)) reduce_resid_rmsnorm_launch(ws, s_o, (long long)B * H, x, w.post_ln, xn, B, H, c.dec_rms_eps, st);
        }
        {
            ProfScope ps(h, "dec_gateup", 4.0 * B * H * c.dec_inter, 4.0 * H * c.dec_inter);
            // M = B <= 128 fits one M tile of the general kernel (two above, up to 256 rows); 64-column tiles give N/64 CTAs per M tile,
            // each streaming its weight rows once
            GemmEpiArgs eg;
            eg.epi = EPI_SWIGLU; eg.out = act; eg.ldo = c.dec_inter;
            // narrowest 64-multiple tile that still gives one CTA per SM at most (0.6B: 96 tiles of 64, 1.7B: 96 tiles of 128)
            int gu_bn = 64;
            while ((2 * c.dec_inter) / gu_bn > h->num_sms && gu_bn < 256 && (2 * c.dec_inter) % (2 * gu_bn) == 0) gu_bn *= 2;
            if (!(skip & 16)) gemm(xn, H, B, H, w.gu_w, 2 * c.dec_inter, eg, st, false, gu_bn);
        }
        {
            ProfScope ps(h, "dec_down", 2.0 * B * H * c.dec_inter, 2.0 * H * c.dec_inter);
            if (!(skip & 32)) gemm_skinny(act, c.dec_inter, B, c.dec_inter, w.down_w, H, SK_PARTIAL, ws, 0, st);
        }
        {
            ProfScope ps(h, "dec_norm", 0, 4.0 * B * H);
            if (!(skip & 64)) reduce_resid_rmsnorm_launch(ws, s_dn, (long long)B * H, x, last ? m.final_norm : m.dec[l + 1].in_ln,
                                        last ? bs->dlast.as<bf16>() : xn, B, H, c.dec_rms_eps, st);
        }
        h->launches += 3;
    }
}

// final norm of the given rows + tied LM head + argmax -> st_next_tok / st_next_val (+ st_next_lp with logprobs_on: every branch
// also reduces the log-sum-exp of the bf16 logits).  normed: bs->dlast already holds the final-norm hidden states (fused decode path).
void lm_head_argmax(Handle* h, BatchState* bs, const int* row_index, bool normed = false) {
    const q3asr_config& c = h->cfg;
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    const int H = c.dec_hidden, B = bs->prefill_done ? bs->dec_rows : bs->B;
    ProfScope ps(h, "lm_head", 2.0 * B * (double)H * c.dec_vocab, 2.0 * H * c.dec_vocab);
    if (!normed) {
        rmsnorm_launch(bs->dx.as<bf16>(), m.final_norm, bs->dlast.as<bf16>(), B, H, c.dec_rms_eps, row_index, st);
        h->launches++;
    }
    if (bs->sampler_on) {
        // decoder knobs (Qwen3ASR.swift:396-520): bf16 logits of every sequence, then penalty / n-gram mask / Gumbel noise / argmax
        // in one kernel over the tokens decode_advance has recorded so far
        bs->logits_bf.reserve((size_t)B * c.dec_vocab * sizeof(bf16));
        GemmEpiArgs e;
        e.epi = EPI_NORMAL;
        e.out = bs->logits_bf.p;
        e.ldo = c.dec_vocab;
        gemm(bs->dlast.as<bf16>(), H, B, H, m.embed, c.dec_vocab, e, st);
        const int parts = sample_parts(c.dec_vocab);
        if (bs->logprobs_on) {  // raw (max, sum) per slice: amax_sum = [sums | maxima], [B, parts] each
            float* rsum = bs->amax_sum.as<float>();
            float* rmax = rsum + (size_t)B * parts;
            sample_launch(bs->logits_bf.as<bf16>(), nullptr, c.dec_vocab, c.dec_vocab, bs->st_out_ids.as<int32_t>(), bs->max_tokens,
                          bs->st_out_len.as<int>(), bs->sampling, bs->st_scalars.as<int>() + 1, B, bs->amax_val.as<float>(),
                          bs->amax_idx.as<int>(), st, rmax, rsum);
            argmax_lse_reduce(bs->amax_val.as<float>(), bs->amax_idx.as<int>(), rsum, rmax, bs->logits_bf.as<bf16>(), c.dec_vocab, B, parts,
                              bs->st_next_tok.as<int32_t>(), bs->st_next_val.as<float>(), bs->st_next_lp.as<float>(), st);
        } else {
            sample_launch(bs->logits_bf.as<bf16>(), nullptr, c.dec_vocab, c.dec_vocab, bs->st_out_ids.as<int32_t>(), bs->max_tokens,
                          bs->st_out_len.as<int>(), bs->sampling, bs->st_scalars.as<int>() + 1, B, bs->amax_val.as<float>(),
                          bs->amax_idx.as<int>(), st);
            argmax_reduce(bs->amax_val.as<float>(), bs->amax_idx.as<int>(), B, parts, bs->st_next_tok.as<int32_t>(), bs->st_next_val.as<float>(),
                          st);
        }
        h->launches += 2;
        return;
    }
    float* sums = bs->logprobs_on ? bs->amax_sum.as<float>() : nullptr;
    int tiles = 0;
    if (B <= SKINNY_MAX_ROWS && env_int("Q3ASR_LM_GENERAL", 0) == 0) {
        // decode-step shape (few token rows): the persistent weight-streaming kernel of lmhead.cuh
        lmhead_argmax(bs->dlast.as<bf16>(), H, B, H, m.embed, c.dec_vocab, bs->amax_val.as<float>(), bs->amax_idx.as<int>(), st, sums);
        tiles = lmhead_tiles(c.dec_vocab);
    } else {
        const int bn = gemm_pick_bn(c.dec_vocab, EPI_ARGMAX, 1);
        GemmEpiArgs e;
        e.epi = EPI_ARGMAX;
        e.amax_val = bs->amax_val.as<float>();
        e.amax_idx = bs->amax_idx.as<int>();
        e.amax_sum = sums;
        gemm(bs->dlast.as<bf16>(), H, B, H, m.embed, c.dec_vocab, e, st, false, bn);
        tiles = c.dec_vocab / bn;
    }
    if (sums)
        argmax_lse_reduce(bs->amax_val.as<float>(), bs->amax_idx.as<int>(), sums, nullptr, nullptr, 0, B, tiles, bs->st_next_tok.as<int32_t>(),
                          bs->st_next_val.as<float>(), bs->st_next_lp.as<float>(), st);
    else
        argmax_reduce(bs->amax_val.as<float>(), bs->amax_idx.as<int>(), B, tiles, bs->st_next_tok.as<int32_t>(), bs->st_next_val.as<float>(), st);
    h->launches++;
}

DecodeState decode_state(Handle* h, BatchState* bs, int stop_on_eos, bool forced) {
    DecodeState s;
    s.next_tok = bs->st_next_tok.as<int32_t>();
    s.next_val = bs->st_next_val.as<float>();
    s.cur_tok = bs->st_cur_tok.as<int32_t>();
    s.pos = bs->st_pos.as<int>();
    s.kv_len = bs->st_kv_len.as<int>();
    s.out_ids = bs->st_out_ids.as<int32_t>();
    s.out_val = bs->st_out_val.as<float>();
    if (bs->logprobs_on) {
        s.next_lp = bs->st_next_lp.as<float>();
        s.out_lp = bs->st_out_lp.as<float>();
    }
    s.out_len = bs->st_out_len.as<int>();
    s.finished = bs->st_finished.as<int>();
    s.n_active = bs->st_scalars.as<int>();
    s.step = bs->st_scalars.as<int>() + 1;
    s.slot_seq = bs->slot_map_on ? bs->st_slot_seq.as<int>() : nullptr;
    s.forced = forced ? bs->st_forced.as<int32_t>() : nullptr;
    s.max_tokens = bs->max_tokens;
    s.eos = h->cfg.tok_eos;
    s.stop_on_eos = stop_on_eos;
    return s;
}

void run_prefill(Handle* h, BatchState* bs, int stop_on_eos, bool forced) {
    const q3asr_config& c = h->cfg;
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    const int* ints = bs->ints.as<int>();
    const int B = bs->B;
    if (bs->page_cur != 0 || bs->stat_compactions != 0) plan_pages(h, bs, bs->max_tokens);  // a previous run of this batch compacted its rows
    bs->dec_rows = B;
    embed_splice_launch(ints + bs->o_ids, ints + bs->o_audio_src, m.embed, bs->audio.as<bf16>(), bs->dx.as<bf16>(), bs->R, c.dec_hidden,
                        st);
    h->launches++;
    decoder_layers(h, bs, bs->R, true);
    // decode state: positions / cache lengths start at the prompt length
    Q3_CUDA(cudaMemcpyAsync(bs->st_pos.p, ints + bs->o_pos0, sizeof(int) * B, cudaMemcpyDeviceToDevice, st));
    Q3_CUDA(cudaMemcpyAsync(bs->st_kv_len.p, ints + bs->o_seq_len, sizeof(int) * B, cudaMemcpyDeviceToDevice, st));
    const size_t S = seq_count(bs);
    Q3_CUDA(cudaMemsetAsync(bs->st_out_len.p, 0, sizeof(int) * S, st));
    Q3_CUDA(cudaMemsetAsync(bs->st_finished.p, 0, sizeof(int) * S, st));
    Q3_CUDA(cudaMemcpyAsync(bs->st_slot_seq.p, ints + bs->o_ident, sizeof(int) * B, cudaMemcpyDeviceToDevice, st));
    bs->dec_rows = B;
    bs->slot_map_on = bs->per_seq_steps;  // per-sequence steps index the outputs through the map from the start (identity here)
    bs->stat_row_steps = bs->stat_steps = bs->stat_compactions = 0;
    bs->stat_admissions = bs->stat_admitted = 0;
    Q3_CUDA(cudaMemsetAsync(bs->st_out_ids.p, 0, sizeof(int32_t) * S * std::max(bs->max_tokens, 1), st));
    if (bs->logprobs_on) Q3_CUDA(cudaMemsetAsync(bs->st_out_lp.p, 0, sizeof(float) * S * std::max(bs->max_tokens, 1), st));
    const int scal[2] = {B, 0};
    memcpy(bs->h_out.p, scal, sizeof(scal));
    Q3_CUDA(cudaMemcpyAsync(bs->st_scalars.p, bs->h_out.p, sizeof(scal), cudaMemcpyHostToDevice, st));
    lm_head_argmax(h, bs, ints + bs->o_last_row);
    // step 0 records the first token.  decode_advance increments pos and kv_len, so they start at
    // prompt_len - 1 / prompt_len and come out as prompt_len (position of the first generated token) and
    // prompt_len + 1 (keys visible to the first decode step).
    DecodeState s = decode_state(h, bs, stop_on_eos, forced);
    decode_advance_launch(s, B, st, bs->per_seq_steps);
    h->launches++;
    bs->prefill_done = true;
    bs->steps_done = 1;
}

void decode_step_kernels(Handle* h, BatchState* bs, int stop_on_eos, bool forced) {
    const q3asr_config& c = h->cfg;
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    // the first kernel of a step is fully serialised against the previous step; the rest chain programmatically
    const int rows = bs->dec_rows;
    embed_splice_launch(bs->st_cur_tok.as<int32_t>(), nullptr, m.embed, nullptr, bs->dx.as<bf16>(), rows, c.dec_hidden, st);
    h->launches++;
    PdlScope pdl(env_int("Q3ASR_NO_PDL", 0) == 0 && !h->prof_on);
    if (rows <= SKINNY_MAX_ROWS && c.dec_heads == 2 * c.dec_kv_heads && env_int("Q3ASR_NO_SKINNY", 0) == 0) {
        decoder_layers_decode(h, bs);
        lm_head_argmax(h, bs, nullptr, true);
    } else {
        decoder_layers(h, bs, rows, false);
        lm_head_argmax(h, bs, nullptr);
    }
    decode_advance_launch(decode_state(h, bs, stop_on_eos, forced), rows, st, bs->per_seq_steps);
    h->launches++;
}

// Captures one decode step for the current decode rows into bs->step_graph; returns the launches one replay stands for.
unsigned long long capture_step_graph(Handle* h, BatchState* bs, int stop_on_eos, bool forced) {
    cudaStream_t st = h->stream;
    if (bs->step_graph) {  // the graph bakes in buffer addresses, row counts and flags: rebuilt per batch and per compaction (~1 ms)
        cudaGraphExecDestroy(bs->step_graph);
        bs->step_graph = nullptr;
    }
    cudaGraph_t graph = nullptr;
    const unsigned long long l0 = h->launches, g0 = gemm_launch_count();
    const bool prof_was = h->prof_on;
    h->prof_on = false;  // event records inside a captured graph cannot be read back per replay
    Q3_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    try {
        decode_step_kernels(h, bs, stop_on_eos, forced);
    } catch (...) {
        h->prof_on = prof_was;
        cudaStreamEndCapture(st, &graph);
        if (graph) cudaGraphDestroy(graph);
        throw;
    }
    Q3_CUDA(cudaStreamEndCapture(st, &graph));
    h->prof_on = prof_was;
    const unsigned long long gper = gemm_launch_count() - g0;  // captured, not executed
    const unsigned long long per_step = (h->launches - l0) + gper;
    h->launches = l0;
    h->gemm_base += gper;
    Q3_CUDA(cudaGraphInstantiate(&bs->step_graph, graph, 0));
    Q3_CUDA(cudaGraphDestroy(graph));
    bs->graph_B = bs->dec_rows;
    return per_step;
}

// Profiling only (q3asr_profile): the decode attention of every layer launched back to back, chained with programmatic dependent
// launch as inside the step graph, bracketed by ONE pair of events ("dec_attn_chain": one entry per call, bytes = the keys and
// values all the launches read).  A single eager launch between two event records also pays the launch ramp and the records
// (bench.py reports that figure as `standalone`); the chain is the kernel's sustained duration, the state it runs in inside the
// step.  Called after the last decode step of a batch: the launches re-read the cache and write the (by then meaningless) new-token
// row of the next position, which nothing reads any more.
void profile_attn_chain(Handle* h, BatchState* bs) {
    const q3asr_config& c = h->cfg;
    const Model& m = *h->model;
    cudaStream_t st = h->stream;
    const int B = bs->dec_rows;
    const int hd = c.dec_head_dim, nq = c.dec_heads * hd, nkv = c.dec_kv_heads * hd, nqkv = nq + 2 * nkv;
    const KvCache kc = kv_cache(h, bs);
    const int s_qkv = gemm_skinny_splits(nqkv, c.dec_hidden, SK_PARTIAL);
    const float scale = 1.0f / sqrtf((float)hd);
    double kv_bytes = 0;
    for (const ClipInfo& ci : bs->clips) kv_bytes += 2.0 * 2.0 * nkv * (ci.prompt_len + bs->steps_done);
    ProfScope ps(h, "dec_attn_chain", 0, c.dec_layers * kv_bytes);
    PdlScope pdl(env_int("Q3ASR_NO_PDL", 0) == 0);
    for (int l = 0; l < c.dec_layers; l++)
        decode_attn_fused_launch(bs->dws.as<float>(), s_qkv, (long long)B * nqkv, nqkv, m.dec[l].q_norm, m.dec[l].k_norm, bs->st_pos.as<int>(),
                                 c.dec_rms_eps, bs->rope_tab.as<float2>(), kc, l, bs->st_kv_len.as<int>(), B, c.dec_heads, scale,
                                 bs->datt.as<bf16>(), h->num_sms, st, bs->dattn_part.as<float>(), bs->dattn_cnt.as<int>());
}

bool mega_wanted(Handle* h, BatchState* bs) {
    return bs->dec_rows <= SKINNY_MAX_ROWS && h->cfg.dec_heads == 2 * h->cfg.dec_kv_heads && env_int("Q3ASR_NO_SKINNY", 0) == 0 &&
           megastep_supported(h, bs);
}

// Takes the finished sequences out of the decode rows (continuous-batching half of the scheduler: the reference stops an
// utterance at EOS, Qwen3ASR.swift:378-379; here its KV pages and its column of every product stop being streamed).
// n_active: the number of unfinished sequences the host has just read back.
void compact_decode_rows(Handle* h, BatchState* bs, int n_active) {
    cudaStream_t st = h->stream;
    int* cur = (bs->page_cur ? bs->page_tab2 : bs->page_tab).as<int>();
    int* nxt = (bs->page_cur ? bs->page_tab : bs->page_tab2).as<int>();
    decode_compact_launch(bs->dec_rows, bs->st_finished.as<int>(), bs->st_slot_seq.as<int>(), bs->st_cur_tok.as<int32_t>(), bs->st_pos.as<int>(),
                          bs->st_kv_len.as<int>(), cur, nxt, bs->pages_per_seq, st);
    h->launches++;
    bs->page_cur ^= 1;
    bs->slot_map_on = true;
    bs->dec_rows = n_active;
    bs->stat_compactions++;
    if (bs->mega_ready) megastep_prepare(h, bs);
}

void run_decode(Handle* h, BatchState* bs, int max_tokens, int stop_on_eos, bool forced) {
    cudaStream_t st = h->stream;
    const bool use_graph = env_int("Q3ASR_NO_GRAPH", 0) == 0;
    // rows are compacted when a quarter of them has finished (and at least four): each compaction costs a graph capture (~1 ms),
    // each finished row a share of the step's KV and activation traffic.  Not with the decoder knobs (the sampler indexes the
    // generated ids by row) nor when teacher forcing.
    const bool may_compact = stop_on_eos && !forced && !bs->sampler_on && env_int("Q3ASR_NO_COMPACT", 0) == 0;
    int* h_active = reinterpret_cast<int*>(bs->h_out.p);
    int step = bs->steps_done;
    bs->mega_ready = false;
    if (mega_wanted(h, bs)) megastep_prepare(h, bs);
    auto account = [&]() { bs->stat_steps++; bs->stat_row_steps += (unsigned long long)bs->dec_rows; };
    // after every 16th step with stop_on_eos: how many sequences are still active?  Returns false when the batch is done.
    auto poll = [&](bool* recapture) {
        Q3_CUDA(cudaMemcpyAsync(h_active, bs->st_scalars.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        Q3_CUDA(cudaStreamSynchronize(st));
        const int n = *h_active;
        if (n <= 0) return false;
        if (may_compact && n < bs->dec_rows && bs->dec_rows - n >= std::max(4, bs->dec_rows / 4)) {
            compact_decode_rows(h, bs, n);
            *recapture = true;
        }
        return true;
    };
    // One eager step the first time a handle decodes (it sets the kernels' function attributes, which must not happen inside a
    // stream capture) or when the graph is off / profiling brackets the launches; afterwards the first step is a graph replay too
    // (eager: ~2.5 ms for the 201 launches of a step against 1.5 ms replayed).
    if (step < max_tokens && (!h->decode_warm || !use_graph || h->prof_on)) {
        decode_step_kernels(h, bs, stop_on_eos, forced);
        h->decode_warm = true;
        account();
        step++;
    }
    if (step < max_tokens && use_graph) {
        unsigned long long per_step = capture_step_graph(h, bs, stop_on_eos, forced);
        ProfScope ps(h, "decode_graph_steps", 0, 0);
        for (; step < max_tokens; step++) {
            Q3_CUDA(cudaGraphLaunch(bs->step_graph, st));
            h->launches += per_step;
            account();
            if (stop_on_eos && (step & 15) == 15) {
                bool recapture = false;
                if (!poll(&recapture)) { step++; break; }
                if (recapture && step + 1 < max_tokens) per_step = capture_step_graph(h, bs, stop_on_eos, forced);
            }
        }
    } else {
        for (; step < max_tokens; step++) {
            decode_step_kernels(h, bs, stop_on_eos, forced);
            account();
            if (stop_on_eos && (step & 15) == 15) {
                bool recapture = false;
                if (!poll(&recapture)) { step++; break; }
            }
        }
    }
    bs->steps_done = step;
    if (h->prof_on && step >= max_tokens && !stop_on_eos && !bs->mega_ready && bs->dec_rows > 0 && bs->dec_rows <= SKINNY_MAX_ROWS &&
        h->cfg.dec_heads == 2 * h->cfg.dec_kv_heads && env_int("Q3ASR_NO_SKINNY", 0) == 0)
        profile_attn_chain(h, bs);
}

}  // namespace

void prefill_attention(Handle* h, const PrefillAttn& a, bool fuse_qkv, int bn, int attn, double causal_pairs) {
    cudaStream_t st = h->stream;
    const int hd = 128, nq = a.heads * hd, nkv = a.kv_heads * hd, nqkv = nq + 2 * nkv;
    const double Rd = a.rows;
    {
        ProfScope ps(h, "pre_qkv", 2.0 * Rd * a.hidden * nqkv, 2.0 * a.hidden * nqkv);
        if (fuse_qkv) {
            // per-head RMSNorm + RoPE + the paged-KV write happen in the product's epilogue (gemm.cuh EPI_QKV): q, k and the cache
            // are written once, the raw product never reaches memory (v does, as is: the attention reads it from there)
            GemmEpiArgs e;
            e.epi = EPI_QKV;
            e.out = a.qkv;
            e.ldo = nqkv;
            e.rp = QkvRope{a.pos, a.row_seq, a.rope_t, a.rope_n, a.q_norm, a.k_norm, a.q, a.k, a.kc.pool, a.kc.page_table, a.kc.max_pages,
                           a.kc.layers, a.layer, a.heads, a.kv_heads, a.eps};
            gemm(a.xn, a.hidden, a.rows, a.hidden, a.w_qkv, nqkv, e, st, false, bn);
        } else {
            gemm(a.xn, a.hidden, a.rows, a.hidden, a.w_qkv, nqkv, epi_store(a.qkv, nqkv, nullptr), st, false, bn);
        }
    }
    if (!fuse_qkv) {
        ProfScope ps(h, "pre_rope", 0, 4.0 * Rd * nqkv);
        // v is not transformed: the attention reads it straight from the QKV product, only k needs a contiguous copy
        qknorm_rope_kv_launch(a.qkv, nqkv, a.q_norm, a.k_norm, a.pos, a.row_seq, a.rows, a.heads, a.kv_heads, a.eps, a.rope, a.q, a.k,
                              nullptr, a.kc, a.layer, st);
    }
    ProfScope ps(h, "pre_attn", 4.0 * causal_pairs * nq, 0);
    if (attn == 0)
        flash_attn_tc_launch(a.q, nq, a.k, nkv, a.qkv + nq + nkv, nqkv, a.att, nq, a.segs, a.rows, a.heads, a.heads / a.kv_heads, hd, true,
                             a.scale, st);
    else if (attn == 1)
        flash_attn_launch(a.q, nq, a.k, nkv, a.qkv + nq + nkv, nqkv, a.att, nq, a.segs, a.heads, a.heads / a.kv_heads, hd, true, a.scale, st);
}

int encoder_tokens_for(int frames) {
    // AudioEncoder.swift:287-303 with chunk = 100
    if (frames <= 0) return 0;
    const int full = frames / 100, rem = frames % 100;
    return full * 13 + (rem > 0 ? std::max(conv_len3(rem), 1) : 0);
}

namespace {

// The clips at another rate, converted to 16 kHz on the compute stream once their copy has landed (their event).
void resample_clips(Handle* h, BatchState* bs, const int* rates, const size_t* n_in, const size_t* raw_off) {
    for (int b = 0; b < bs->B; b++)
        if (rates[b] != 16000) {
            wait_recorded(bs, b);
            Q3_CUDA(cudaStreamWaitEvent(h->stream, h->copy_ev[(size_t)b], 0));
            bs->copy_waited[(size_t)b] = 1;
            resample_device(h, bs->raw_pcm.as<float>() + raw_off[b], n_in[b], rates[b], 16000, bs->pcm.as<float>() + bs->mel.clips[b].in_off,
                            (size_t)bs->mel.clips[b].n, h->stream);
        }
}

// Upload into a given state.  staged (continuous batching's next group): only the host side runs now — the staging threads copy
// the samples on the copy stream while the decode goes on, and the plan is kept on the host; nothing is queued on the compute
// stream and nothing waits for it.  upload_staged finishes the upload when the group is admitted.
void batch_upload_into(Handle* h, BatchState* bs, const float* const* pcm, const size_t* n_in, int batch, const q3asr_prompt* prompts,
                       const int* rates, bool defer_join, bool staged) {
    finish_upload(bs);  // (a previous upload whose caller never ran it to the end)
    Q3_CHECK(pcm != nullptr && n_in != nullptr && batch > 0, Q3ASR_ERR_INVALID, "batch_upload: null argument / empty batch");
    Q3_CHECK(batch <= 1024, Q3ASR_ERR_INVALID, "batch_upload: at most 1024 utterances per call");
    // clips at another rate are converted to 16 kHz on the device (Qwen3ASRModel.transcribe resamples first,
    // AudioPreprocessing.swift:323-337): n16[b] samples reach the mel kernel
    std::vector<size_t> n16(n_in, n_in + batch);
    size_t raw_floats = 0;
    std::vector<size_t> raw_off((size_t)batch, 0);
    for (int b = 0; b < batch; b++) {
        Q3_CHECK(pcm[b] != nullptr && n_in[b] < (size_t)1 << 30, Q3ASR_ERR_INVALID, "batch_upload: null clip / clip too long");
        if (rates != nullptr && rates[b] != 16000) {
            Q3_CHECK(rates[b] > 0, Q3ASR_ERR_INVALID, "batch_upload: bad sample rate");
            n16[b] = resample_len(n_in[b], rates[b], 16000);
            raw_off[(size_t)b] = raw_floats;
            raw_floats += (n_in[b] + 3) & ~size_t(3);
        }
        Q3_CHECK(n16[b] >= (size_t)MEL_HOP && n16[b] < (size_t)1 << 30, Q3ASR_ERR_INVALID,
                 "batch_upload: every clip needs at least 160 samples at 16 kHz (one mel frame)");
    }
    const size_t* n = n16.data();
    bs->B = batch;
    bs->n_seqs = batch;
    bs->page_prompt = 0;
    bs->per_seq_steps = false;
    bs->kv_from = nullptr;
    bs->kv_row0 = 0;
    bs->stat_admissions = bs->stat_admitted = 0;
    bs->mel = mel_plan(n, batch);
    bs->mel_done = bs->enc_done = bs->prefill_done = false;
    bs->steps_done = 0;
    bs->has_audio = true;
    bs->sampler_on = false;  // every batch starts greedy; batch_set_sampling turns the decoder knobs on
    bs->logprobs_on = false;  // batch_set_logprobs turns them on
    // samples: pinned staging -> device
    bs->pcm.reserve(sizeof(float) * (bs->mel.pcm_floats + 64));
    bs->mel_out.reserve(sizeof(float) * std::max<long long>(bs->mel.out_floats, 1));
    bs->mel_clips.reserve(sizeof(MelClip) * batch);
    bs->mel_gmax.reserve(sizeof(int) * batch);
    bs->mel_tmin.reserve(sizeof(float) * 2 * bs->mel.total_tiles);  // per-tile minimum + per-tile clip
    bs->h_stage.reserve(sizeof(float) * (bs->mel.pcm_floats + raw_floats));
    float* stage = bs->h_stage.as<float>();
    float* stage_raw = stage + bs->mel.pcm_floats;  // clips awaiting conversion
    if (raw_floats) bs->raw_pcm.reserve(sizeof(float) * raw_floats);
    // The caller's buffers are pageable: copy each clip into the pinned staging area and queue its H2D copy at once, from a
    // few host threads (4: as fast as 6 or 8 for one rank, and 8 ranks x 4 do not oversubscribe a 32-core box), so the staging memcpy
    // (the slow leg, ~10 GB/s per thread) overlaps the PCIe transfers and the planning
    // below.  Clips are independent, so the order of the copies on the stream does not matter.
    const int n_workers = std::max(1, std::min({batch, env_int("Q3ASR_UPLOAD_THREADS", 4), (int)std::thread::hardware_concurrency() / 2}));
    // the copies go on the copy stream, one event per clip (waited for by the mel launch of the clip's group, run_mel)
    while (h->copy_ev.size() < (size_t)batch) {
        cudaEvent_t e = nullptr;
        Q3_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->copy_ev.push_back(e);
    }
    bs->copy_events = true;
    bs->copy_waited.assign((size_t)batch, 0);
    bs->mel_next = 0;
    Q3_CUDA(cudaEventRecord(bs->ev[0], h->stream));  // (any earlier work on the compute stream that still reads the sample buffer)
    Q3_CUDA(cudaStreamWaitEvent(h->copy_stream, bs->ev[0], 0));
    // The staging threads outlive this function when `defer_join` (q3asr_transcribe_ids*: the caller's buffers stay borrowed until
    // the call returns): the planning below, the mel kernels and the convolution stack of the first clips then run while the last
    // clips are still being copied into the staging area — the staging memcpy (123 MB at ~27 GB/s from four threads for 64 x 30 s)
    // is the slow leg of an upload, not PCIe.  Everything the threads read lives in the job.
    bs->upload.reset(new UploadJob());
    UploadJob* J = bs->upload.get();
    J->werr.assign((size_t)n_workers, cudaSuccess);
    J->recorded.reset(new std::atomic<int>[(size_t)batch]);
    for (int b = 0; b < batch; b++) J->recorded[(size_t)b].store(0, std::memory_order_relaxed);
    J->pcm.assign(pcm, pcm + batch);
    J->n_in.assign(n_in, n_in + batch);
    J->n16 = n16;
    J->raw_off = raw_off;
    J->in_off.resize((size_t)batch);
    for (int b = 0; b < batch; b++) J->in_off[(size_t)b] = bs->mel.clips[(size_t)b].in_off;
    if (rates != nullptr) J->rates.assign(rates, rates + batch);
    {
        float* d_pcm = bs->pcm.as<float>();
        float* d_raw = raw_floats ? bs->raw_pcm.as<float>() : nullptr;
        const int device = h->device;
        cudaStream_t cs = h->copy_stream;
        const cudaEvent_t* evs = h->copy_ev.data();  // not resized while the job runs
        J->workers.reserve((size_t)n_workers);
        for (int w = 0; w < n_workers; w++)
            J->workers.emplace_back([J, w, n_workers, batch, stage, stage_raw, d_pcm, d_raw, device, cs, evs]() {
                cudaError_t e = cudaSetDevice(device);
                for (int b = w; b < batch; b += n_workers) {
                    if (e == cudaSuccess) {
                        const bool raw = !J->rates.empty() && J->rates[(size_t)b] != 16000;
                        float* sp = raw ? stage_raw + J->raw_off[(size_t)b] : stage + J->in_off[(size_t)b];
                        float* dp = raw ? d_raw + J->raw_off[(size_t)b] : d_pcm + J->in_off[(size_t)b];
                        const size_t bytes = sizeof(float) * (raw ? J->n_in[(size_t)b] : J->n16[(size_t)b]);
                        memcpy(sp, J->pcm[(size_t)b], bytes);
                        e = cudaMemcpyAsync(dp, sp, bytes, cudaMemcpyHostToDevice, cs);
                        if (e == cudaSuccess) e = cudaEventRecord(evs[b], cs);
                    }
                    J->recorded[(size_t)b].store(e == cudaSuccess ? 1 : -1, std::memory_order_release);
                }
                J->werr[(size_t)w] = e;
            });
    }
    if (!staged) Q3_CUDA(cudaMemcpyAsync(bs->mel_clips.p, bs->mel.clips.data(), sizeof(MelClip) * batch, cudaMemcpyHostToDevice, h->stream));
    // plan
    std::vector<int> frames(batch);
    std::vector<long long> mel_off(batch);
    for (int b = 0; b < batch; b++) {
        frames[b] = bs->mel.clips[b].frames;
        mel_off[b] = bs->mel.clips[b].out_off;
    }
    std::vector<int> ints;
    plan_encoder(h, bs, frames, mel_off, &ints);
    for (int b = 0; b < batch; b++) bs->clips[b].n = (int)n[b];
    // the KV pages are reserved for the reference's default decode length (maxTokens = 448, Qwen3ASR.swift:135); batch_run
    // re-plans them when a larger value is asked for
    const int reserve_tokens = std::max(1, env_int("Q3ASR_RESERVE_TOKENS", 448));
    plan_decoder(h, bs, prompts, reserve_tokens, &ints);
    if (staged) {
        bs->plan_ints = std::move(ints);
        bs->up_rates.clear();
        if (raw_floats) bs->up_rates.assign(rates, rates + batch);
        bs->up_n.assign(n_in, n_in + batch);
        bs->up_raw_off = raw_off;
        return;
    }
    if (!defer_join) finish_upload(bs);
    if (raw_floats) resample_clips(h, bs, rates, n_in, raw_off.data());  // the conversions follow their clip's copy (its event)
    upload_ints(h, bs, ints);  // (synchronises the COMPUTE stream; the sample copies may still be in flight on the copy stream: the
                               // caller's buffers are free — they were copied to the staging area — and run_mel waits per clip)
    plan_pages(h, bs, reserve_tokens);
    bs->prompt_ids.clear();
}

// The compute-stream half of a staged upload: clip table, sample-rate conversions, plan.
void upload_staged(Handle* h, BatchState* bs) {
    Q3_CUDA(cudaMemcpyAsync(bs->mel_clips.p, bs->mel.clips.data(), sizeof(MelClip) * bs->B, cudaMemcpyHostToDevice, h->stream));
    if (!bs->up_rates.empty()) resample_clips(h, bs, bs->up_rates.data(), bs->up_n.data(), bs->up_raw_off.data());
    upload_ints(h, bs, bs->plan_ints);
}

}  // namespace

void batch_upload(Handle* h, const float* const* pcm, const size_t* n_in, int batch, const q3asr_prompt* prompts, const int* rates,
                  bool defer_join) {
    batch_upload_into(h, fresh_batch(h), pcm, n_in, batch, prompts, rates, defer_join, false);
}

// Qwen3ForcedAligner.align (ForcedAligner.swift:226-331), batched: mel -> encoder -> one causal prefill over the aligner template ->
// final RMSNorm of the requested rows only -> classification head (+bias, bf16 logits) -> first-maximum class per row.
void align_indices(Handle* h, const float* const* pcm, const size_t* n, const int* rates, int batch, const int32_t* const* slotted_ids,
                   const int* n_slotted, const int* const* positions, const int* n_positions, int32_t* const* raw_out) {
    const q3asr_config& c = h->cfg;
    Q3_CHECK(c.classify_num > 0, Q3ASR_ERR_STATE, "align: this configuration has no classification head (classify_num == 0)");
    Q3_CHECK(h->loaded && h->model, Q3ASR_ERR_STATE, "weights are not loaded");
    Q3_CHECK(slotted_ids && n_slotted && positions && n_positions && raw_out && batch > 0, Q3ASR_ERR_INVALID, "align: null argument");
    std::vector<q3asr_prompt> prompts((size_t)batch);
    for (int b = 0; b < batch; b++) {
        Q3_CHECK(slotted_ids[b] != nullptr && n_slotted[b] > 0 && n_positions[b] >= 0 && (n_positions[b] == 0 || (positions[b] && raw_out[b])),
                 Q3ASR_ERR_INVALID, "align: empty slotted text / null positions");
        for (int i = 0; i < n_positions[b]; i++)
            Q3_CHECK(positions[b][i] >= 0 && positions[b][i] < n_slotted[b], Q3ASR_ERR_INVALID, "align: position outside the slotted text");
        prompts[(size_t)b] = q3asr_prompt{nullptr, 0, slotted_ids[b], n_slotted[b], 1};
    }
    batch_upload(h, pcm, n, batch, prompts.data(), rates);
    BatchState* bs = h->batch.get();
    cudaStream_t st = h->stream;
    run_mel(h, bs);
    reserve_encoder(h, bs);
    run_encoder(h, bs, bs->mel_out.as<float>());
    reserve_decoder(h, bs);
    const Model& m = *h->model;
    embed_splice_launch(bs->ints.as<int>() + bs->o_ids, bs->ints.as<int>() + bs->o_audio_src, m.embed, bs->audio.as<bf16>(), bs->dx.as<bf16>(),
                        bs->R, c.dec_hidden, st);
    h->launches++;
    decoder_layers(h, bs, bs->R, true);
    // rows of the requested positions: prompt row0 + (prompt_len - n_slotted) + position
    std::vector<int> rows;
    for (int b = 0; b < batch; b++)
        for (int i = 0; i < n_positions[b]; i++) rows.push_back(bs->clips[b].row0 + bs->clips[b].prompt_len - n_slotted[b] + positions[b][i]);
    const int P = (int)rows.size();
    if (P == 0) {
        Q3_CUDA(cudaStreamSynchronize(st));
        return;
    }
    const int H = c.dec_hidden, NP = m.cls_pad;
    // scratch: [rows | gen_len zeros | tokens] ints, normed rows, bf16 logits
    const int parts = sample_parts(c.classify_num);
    bs->amax_idx.reserve(sizeof(int) * (size_t)((3 + 2 * parts) * P + 4));
    int* d_rows = bs->amax_idx.as<int>();
    int* d_zero = d_rows + P;
    int32_t* d_tok = reinterpret_cast<int32_t*>(d_zero + P);
    int* d_pidx = reinterpret_cast<int*>(d_tok + P);
    float* d_pval = reinterpret_cast<float*>(d_pidx + (size_t)parts * P);
    bs->h_ints.reserve(sizeof(int) * (size_t)(3 * P + 4));
    int* hrows = bs->h_ints.as<int>();
    for (int i = 0; i < P; i++) { hrows[i] = rows[(size_t)i]; hrows[P + i] = 0; }
    Q3_CUDA(cudaMemcpyAsync(d_rows, hrows, sizeof(int) * 2 * P, cudaMemcpyHostToDevice, st));
    bs->dlast.reserve((size_t)P * H * sizeof(bf16));
    bs->logits_bf.reserve((size_t)P * NP * sizeof(bf16));
    rmsnorm_launch(bs->dx.as<bf16>(), m.final_norm, bs->dlast.as<bf16>(), P, H, c.dec_rms_eps, d_rows, st);
    h->launches++;
    GemmEpiArgs e;
    e.epi = EPI_NORMAL;
    e.out = bs->logits_bf.p;
    e.ldo = NP;
    e.bias = m.cls_b;
    gemm(bs->dlast.as<bf16>(), H, P, H, m.cls_w, NP, e, st);
    SamplingParams greedy;
    sample_launch(bs->logits_bf.as<bf16>(), nullptr, NP, c.classify_num, d_tok, 1, d_zero, greedy, nullptr, P, d_pval, d_pidx, st);
    argmax_reduce(d_pval, d_pidx, P, parts, d_tok, nullptr, st);
    h->launches += 2;
    Q3_CUDA(cudaMemcpyAsync(hrows + 2 * P, d_tok, sizeof(int32_t) * P, cudaMemcpyDeviceToHost, st));
    Q3_CUDA(cudaStreamSynchronize(st));
    int k = 0;
    for (int b = 0; b < batch; b++)
        for (int i = 0; i < n_positions[b]; i++) raw_out[b][i] = hrows[2 * P + k++];
}

void batch_set_sampling(Handle* h, const q3asr_sampling* opts) {
    BatchState* bs = h->batch.get();
    Q3_CHECK(bs != nullptr && bs->B > 0, Q3ASR_ERR_STATE, "batch_set_sampling: no batch uploaded");
    Q3_CHECK(!bs->prefill_done, Q3ASR_ERR_STATE, "batch_set_sampling: the first token of this batch has already been chosen");
    if (opts == nullptr) {
        bs->sampler_on = false;
        return;
    }
    Q3_CHECK(opts->repetition_penalty > 0.f && opts->no_repeat_ngram_size >= 0 && opts->temperature >= 0.f, Q3ASR_ERR_INVALID,
             "sampling: repetition_penalty > 0, no_repeat_ngram_size >= 0, temperature >= 0");
    // Qwen3ASRModel.isGreedyFastPath (Qwen3ASR.swift:300-304): the default configuration keeps the fused argmax epilogue
    const bool greedy = opts->repetition_penalty == 1.0f && opts->no_repeat_ngram_size == 0 && opts->temperature == 0.0f;
    bs->sampler_on = !greedy || opts->force_device_sampler != 0;
    bs->sampling.repetition_penalty = opts->repetition_penalty;
    bs->sampling.no_repeat_ngram = opts->no_repeat_ngram_size;
    bs->sampling.temperature = opts->temperature;
    bs->sampling.seed = opts->seed;
}

void batch_set_logprobs(Handle* h, int enable) {
    BatchState* bs = h->batch.get();
    Q3_CHECK(bs != nullptr && bs->B > 0 && bs->has_audio, Q3ASR_ERR_STATE, "batch_set_logprobs: no batch uploaded");
    Q3_CHECK(!bs->prefill_done, Q3ASR_ERR_STATE, "batch_set_logprobs: the first token of this batch has already been chosen");
    bs->logprobs_on = enable != 0;
}

void pick_next_token(Handle* h, const float* logits, int vocab, const int32_t* generated, int n_generated, const q3asr_sampling* opts,
                     int draw, int32_t* token) {
    Q3_CHECK(logits != nullptr && vocab > 0 && n_generated >= 0 && (generated != nullptr || n_generated == 0) && opts != nullptr &&
                 token != nullptr,
             Q3ASR_ERR_INVALID, "pick_next_token: bad argument");
    SamplingParams sp;
    sp.repetition_penalty = opts->repetition_penalty;
    sp.no_repeat_ngram = opts->no_repeat_ngram_size;
    sp.temperature = opts->temperature;
    sp.seed = opts->seed;
    float* d_logits = nullptr;
    int32_t* d_gen = nullptr;
    int* d_small = nullptr;  // [gen_len, step, token, -, slice indices (8), slice values (8)]
    cudaStream_t st = h->stream;
    auto release = [&]() { cudaFree(d_logits); cudaFree(d_gen); cudaFree(d_small); };
    try {
        Q3_CUDA(cudaMalloc(&d_logits, sizeof(float) * vocab));
        Q3_CUDA(cudaMalloc(&d_gen, sizeof(int32_t) * std::max(n_generated, 1)));
        Q3_CUDA(cudaMalloc(&d_small, sizeof(int) * 20));
        const int small[4] = {n_generated, draw, 0, 0};
        Q3_CUDA(cudaMemcpyAsync(d_logits, logits, sizeof(float) * vocab, cudaMemcpyHostToDevice, st));
        if (n_generated) Q3_CUDA(cudaMemcpyAsync(d_gen, generated, sizeof(int32_t) * n_generated, cudaMemcpyHostToDevice, st));
        Q3_CUDA(cudaMemcpyAsync(d_small, small, sizeof(small), cudaMemcpyHostToDevice, st));
        sample_launch(nullptr, d_logits, vocab, vocab, d_gen, std::max(n_generated, 1), d_small, sp, d_small + 1, 1,
                      reinterpret_cast<float*>(d_small + 12), d_small + 4, st);
        argmax_reduce(reinterpret_cast<float*>(d_small + 12), d_small + 4, 1, sample_parts(vocab), d_small + 2, nullptr, st);
        h->launches += 2;
        Q3_CUDA(cudaMemcpyAsync(token, d_small + 2, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        Q3_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        release();
        throw;
    }
    release();
}

void batch_run(Handle* h, int stages, int max_tokens, int stop_on_eos) {
    BatchState* bs = h->batch.get();
    Q3_CHECK(bs != nullptr && bs->B > 0 && bs->has_audio, Q3ASR_ERR_STATE, "batch_run: no batch uploaded");
    Q3_CHECK(max_tokens >= 0 && max_tokens <= (1 << 20), Q3ASR_ERR_INVALID, "batch_run: max_tokens out of range");
    if (max_tokens > bs->max_tokens) {
        Q3_CHECK(!bs->prefill_done, Q3ASR_ERR_STATE,
                 "batch_run: max_tokens exceeds the decode capacity this batch was prefilled with (pass the larger value to the prefill stage)");
        plan_pages(h, bs, max_tokens);
    }
    if (stages & (Q3ASR_STAGE_ENCODER | Q3ASR_STAGE_PREFILL | Q3ASR_STAGE_DECODE))
        Q3_CHECK(h->loaded && h->model, Q3ASR_ERR_STATE, "weights are not loaded (q3asr_init_random / q3asr_load_safetensors)");
    cudaStream_t st = h->stream;
    Q3_CUDA(cudaEventRecord(bs->ev[0], st));
    if (stages & Q3ASR_STAGE_MEL) {
        bs->mel_next = 0;
        bs->mel_done = false;
        // with the upload still in flight and the encoder to follow, the mel launches are interleaved with the convolution stack
        // (run_encoder), group of clips by group of clips, as their copies land
        if ((stages & Q3ASR_STAGE_ENCODER) && copies_pending(h, bs) && bs->n_tok > 0) bs->mel_done = true;
        else run_mel(h, bs);
    }
    Q3_CUDA(cudaEventRecord(bs->ev[1], st));
    if (stages & Q3ASR_STAGE_ENCODER) {
        Q3_CHECK(bs->mel_done, Q3ASR_ERR_STATE, "batch_run: encoder stage needs the mel stage first");
        reserve_encoder(h, bs);
        run_encoder(h, bs, bs->mel_out.as<float>());
        finish_upload(bs);  // every clip's copy has been queued by now (run_mel waited for each): the staging threads are done
    }
    Q3_CUDA(cudaEventRecord(bs->ev[2], st));
    if (stages & Q3ASR_STAGE_PREFILL) {
        Q3_CHECK(bs->enc_done, Q3ASR_ERR_STATE, "batch_run: prefill stage needs the encoder stage first");
        reserve_decoder(h, bs);
        if (max_tokens > 0) run_prefill(h, bs, stop_on_eos, false);
    }
    Q3_CUDA(cudaEventRecord(bs->ev[3], st));
    if ((stages & Q3ASR_STAGE_DECODE) && max_tokens > 1) {
        Q3_CHECK(bs->prefill_done, Q3ASR_ERR_STATE, "batch_run: decode stage needs the prefill stage first");
        run_decode(h, bs, max_tokens, stop_on_eos, false);
    }
    Q3_CUDA(cudaEventRecord(bs->ev[4], st));
}

void batch_download(Handle* h, int32_t* ids, int max_tokens, int* lens) {
    BatchState* bs = h->batch.get();
    Q3_CHECK(bs != nullptr && bs->B > 0, Q3ASR_ERR_STATE, "batch_download: no batch");
    Q3_CHECK(ids != nullptr && lens != nullptr && max_tokens >= 0, Q3ASR_ERR_INVALID, "batch_download: bad argument");
    const int B = seq_count(bs), mt = bs->max_tokens;
    cudaStream_t st = h->stream;
    if (!bs->prefill_done) {
        Q3_CUDA(cudaStreamSynchronize(st));
        for (int b = 0; b < B; b++) lens[b] = 0;
    } else {
        int32_t* h_ids = reinterpret_cast<int32_t*>(bs->h_out.p) + 16;
        int* h_len = reinterpret_cast<int*>(h_ids + (size_t)B * mt);
        Q3_CUDA(cudaMemcpyAsync(h_ids, bs->st_out_ids.p, sizeof(int32_t) * B * mt, cudaMemcpyDeviceToHost, st));
        Q3_CUDA(cudaMemcpyAsync(h_len, bs->st_out_len.p, sizeof(int) * B, cudaMemcpyDeviceToHost, st));
        Q3_CUDA(cudaStreamSynchronize(st));
        for (int b = 0; b < B; b++) {
            const int L = std::min(std::min(h_len[b], max_tokens), mt);
            lens[b] = L;
            memcpy(ids + (size_t)b * max_tokens, h_ids + (size_t)b * mt, sizeof(int32_t) * L);
        }
    }
    for (int i = 0; i < 4; i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, bs->ev[i], bs->ev[i + 1]) == cudaSuccess) h->stage_ms[i] = ms;
    }
}

void batch_download_logprobs(Handle* h, float* out, int max_tokens) {
    BatchState* bs = h->batch.get();
    Q3_CHECK(bs != nullptr && bs->B > 0, Q3ASR_ERR_STATE, "batch_download_logprobs: no batch");
    Q3_CHECK(out != nullptr && max_tokens >= 0, Q3ASR_ERR_INVALID, "batch_download_logprobs: bad argument");
    Q3_CHECK(bs->logprobs_on, Q3ASR_ERR_STATE, "batch_download_logprobs: log-probabilities were not requested for this batch");
    const int B = seq_count(bs), mt = bs->max_tokens;
    cudaStream_t st = h->stream;
    std::fill(out, out + (size_t)B * max_tokens, 0.f);
    if (!bs->prefill_done) {
        Q3_CUDA(cudaStreamSynchronize(st));
        return;
    }
    float* h_lp = reinterpret_cast<float*>(bs->h_out.p) + 16;  // (the staging area of batch_download: ids [B, mt] + lens fit)
    Q3_CUDA(cudaMemcpyAsync(h_lp, bs->st_out_lp.p, sizeof(float) * B * mt, cudaMemcpyDeviceToHost, st));
    Q3_CUDA(cudaStreamSynchronize(st));
    const int L = std::min(max_tokens, mt);
    for (int b = 0; b < B; b++) memcpy(out + (size_t)b * max_tokens, h_lp + (size_t)b * mt, sizeof(float) * L);
}

void encode_one(Handle* h, const float* mel, int frames, float* out, int* tokens) {
    Q3_CHECK(mel != nullptr && out != nullptr && frames > 0 && frames <= MEL_MAX_FRAMES, Q3ASR_ERR_INVALID, "encode: bad argument");
    Q3_CHECK(h->loaded && h->model, Q3ASR_ERR_STATE, "weights are not loaded");
    BatchState* bs = fresh_batch(h);
    bs->B = 1;
    bs->has_audio = false;
    bs->mel_done = bs->enc_done = bs->prefill_done = false;
    bs->copy_events = false;  // the features come from the caller: no sample copies to wait for, no mel launch pending
    bs->mel_next = 1;
    const size_t nmel = (size_t)MEL_BINS * frames;
    bs->mel_out.reserve(nmel * 4);
    bs->h_stage.reserve(nmel * 4);
    memcpy(bs->h_stage.p, mel, nmel * 4);
    Q3_CUDA(cudaMemcpyAsync(bs->mel_out.p, bs->h_stage.p, nmel * 4, cudaMemcpyHostToDevice, h->stream));
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    std::vector<int> ints;
    plan_encoder(h, bs, {frames}, {0}, &ints);
    upload_ints(h, bs, ints);
    reserve_encoder(h, bs);
    run_encoder(h, bs, bs->mel_out.as<float>());
    const size_t n = (size_t)bs->n_tok * h->cfg.enc_out_dim;
    bs->logits.reserve(std::max<size_t>(n, 1) * 4);
    bf16_to_f32_launch(bs->audio.as<bf16>(), bs->logits.as<float>(), n, h->stream);
    h->launches++;
    bs->h_stage.reserve(std::max<size_t>(n, 1) * 4);
    Q3_CUDA(cudaMemcpyAsync(bs->h_stage.p, bs->logits.p, n * 4, cudaMemcpyDeviceToHost, h->stream));
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(out, bs->h_stage.p, n * 4);
    if (tokens) *tokens = bs->n_tok;
}

void decode_forced(Handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, const int32_t* forced, int n_forced,
                   int32_t* argmax_out, float* top_out, const float* audio_embeds, int n_audio_tokens) {
    Q3_CHECK(forced != nullptr && n_forced >= 0 && argmax_out != nullptr, Q3ASR_ERR_INVALID, "decode_forced: bad argument");
    Q3_CHECK(h->loaded && h->model, Q3ASR_ERR_STATE, "weights are not loaded");
    const float* pp[1] = {pcm};
    batch_upload(h, pp, &n, 1, prompt);
    BatchState* bs = h->batch.get();
    const int steps = n_forced + 1;
    Q3_CHECK(steps <= (1 << 20), Q3ASR_ERR_INVALID, "decode_forced: too many forced tokens");
    if (steps > bs->max_tokens) plan_pages(h, bs, steps);
    for (int i = 0; i < n_forced; i++) Q3_CHECK(forced[i] >= 0 && forced[i] < h->cfg.dec_vocab, Q3ASR_ERR_INVALID, "forced id out of range");
    cudaStream_t st = h->stream;
    run_mel(h, bs);
    reserve_encoder(h, bs);
    run_encoder(h, bs, bs->mel_out.as<float>());
    if (audio_embeds != nullptr) {  // parity hook: the caller's audio embeddings replace the encoder's (rounded to bf16 like the splice does)
        Q3_CHECK(n_audio_tokens == bs->n_tok, Q3ASR_ERR_INVALID, "decode_forced_embeds: token count differs from the clip's encoder_tokens");
        const size_t ne = (size_t)bs->n_tok * h->cfg.enc_out_dim;
        bs->logits.reserve(ne * sizeof(float));
        Q3_CUDA(cudaMemcpyAsync(bs->logits.p, audio_embeds, ne * sizeof(float), cudaMemcpyHostToDevice, st));
        f32_to_bf16_launch(bs->logits.as<float>(), bs->audio.as<bf16>(), ne, st);
        h->launches++;
        Q3_CUDA(cudaStreamSynchronize(st));  // the caller's buffer is borrowed for the call only
    }
    reserve_decoder(h, bs);
    std::vector<int32_t> f(forced, forced + n_forced);
    f.push_back(0);
    bs->st_forced.reserve(f.size() * 4);
    Q3_H2D_SYNC(bs->st_forced.p, f.data(), f.size() * 4);
    run_prefill(h, bs, 0, true);
    run_decode(h, bs, steps, 0, true);
    std::vector<int32_t> ids((size_t)bs->max_tokens);
    std::vector<float> vals((size_t)bs->max_tokens);
    Q3_CUDA(cudaStreamSynchronize(st));
    Q3_CUDA(cudaMemcpy(ids.data(), bs->st_out_ids.p, ids.size() * 4, cudaMemcpyDeviceToHost));
    Q3_CUDA(cudaMemcpy(vals.data(), bs->st_out_val.p, vals.size() * 4, cudaMemcpyDeviceToHost));
    for (int i = 0; i < steps; i++) {
        argmax_out[i] = ids[i];
        if (top_out) top_out[i] = vals[i];
    }
}

void prefill_logits(Handle* h, const float* pcm, size_t n, const q3asr_prompt* prompt, float* logits) {
    Q3_CHECK(logits != nullptr, Q3ASR_ERR_INVALID, "prefill_logits: null output");
    Q3_CHECK(h->loaded && h->model, Q3ASR_ERR_STATE, "weights are not loaded");
    const float* pp[1] = {pcm};
    batch_upload(h, pp, &n, 1, prompt);
    BatchState* bs = h->batch.get();
    const q3asr_config& c = h->cfg;
    cudaStream_t st = h->stream;
    run_mel(h, bs);
    reserve_encoder(h, bs);
    run_encoder(h, bs, bs->mel_out.as<float>());
    reserve_decoder(h, bs);
    run_prefill(h, bs, 0, false);
    // dlast holds the normed last hidden state; full-vocabulary fp32 logits through the same GEMM
    bs->logits.reserve((size_t)c.dec_vocab * 4);
    GemmEpiArgs e;
    e.epi = EPI_F32;
    e.out = bs->logits.p;
    e.ldo = c.dec_vocab;
    gemm(bs->dlast.as<bf16>(), c.dec_hidden, 1, c.dec_hidden, h->model->embed, c.dec_vocab, e, st);
    Q3_CUDA(cudaStreamSynchronize(st));
    Q3_CUDA(cudaMemcpy(logits, bs->logits.p, (size_t)c.dec_vocab * 4, cudaMemcpyDeviceToHost));
}

// ---------------------------------------------------------------------------------------------
// Continuous batching: one request decoded by one resident batch of at most max_rows rows.  The first max_rows utterances are
// prefilled as usual; whenever a poll finds enough rows finished, the finished rows are partitioned out of the decode rows and the
// next waiting utterances (request order) go through mel -> encoder -> prefill as a group whose KV lands directly in the freed page
// blocks, then join the decode rows.  Every utterance runs the same kernels on the same rows as in a static batch, so its ids and
// log-probabilities do not depend on the schedule.
// ---------------------------------------------------------------------------------------------
namespace {

struct ContinuousRun {
    Handle* h;
    BatchState* bs;  // the resident state
    const float* const* pcm;
    const size_t* n;
    const int* rates;
    const q3asr_prompt* prompts;
    int batch, max_rows, stop_on_eos;
    int next_stage = 0;              // first utterance not yet staged
    int staged = -1, staged_k = 0, staged_seq0 = 0, next_adm = 0;  // the staged group (h->adm[staged])
    std::vector<cudaEvent_t> ev;     // four per admission: start, encoder, prefill, end
    float adm_ms[3] = {0.f, 0.f, 0.f};

    ~ContinuousRun() {
        for (std::unique_ptr<BatchState>* s : {&h->batch, &h->adm[0], &h->adm[1]}) {  // the staging threads borrow the caller's buffers
            try {
                finish_upload(s->get());
            } catch (...) {
            }
        }
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
    }

    // the next group's samples go to the copy stream now; its size is the rows that will be free when it is admitted, at least
    // the admission threshold
    void stage(int threshold) {
        if (staged >= 0 || next_stage >= batch) return;
        const int k = std::min(batch - next_stage, std::max(threshold, max_rows - bs->dec_rows));
        BatchState* a = fresh_state(h, h->adm[next_adm]);
        batch_upload_into(h, a, pcm + next_stage, n + next_stage, k, prompts ? prompts + next_stage : nullptr, rates ? rates + next_stage : nullptr,
                          true, true);
        staged = next_adm;
        staged_k = k;
        staged_seq0 = next_stage;
        next_stage += k;
        next_adm ^= 1;
    }

    // Rows [n_live, B) of the resident page table become the finished rows' blocks (and those of rows already free).
    void partition(int n_live) {
        cudaStream_t st = h->stream;
        int* cur = (bs->page_cur ? bs->page_tab2 : bs->page_tab).as<int>();
        int* nxt = (bs->page_cur ? bs->page_tab : bs->page_tab2).as<int>();
        decode_compact_launch(bs->dec_rows, bs->st_finished.as<int>(), bs->st_slot_seq.as<int>(), bs->st_cur_tok.as<int32_t>(), bs->st_pos.as<int>(),
                              bs->st_kv_len.as<int>(), cur, nxt, bs->pages_per_seq, st, bs->B);
        h->launches++;
        bs->page_cur ^= 1;
        bs->dec_rows = n_live;
        bs->stat_compactions++;
    }

    // The staged group: mel -> encoder -> prefill with its KV written into the resident rows [dec_rows, dec_rows + k), then step 0
    // straight into the resident decode state.
    void admit() {
        cudaStream_t st = h->stream;
        BatchState* a = h->adm[staged].get();
        const int k = staged_k, row0 = bs->dec_rows;
        Q3_CHECK(row0 + k <= bs->B, Q3ASR_ERR_STATE, "continuous: admission beyond the resident rows");
        a->kv_from = bs;
        a->kv_row0 = row0;
        a->pages_per_seq = bs->pages_per_seq;
        a->max_tokens = bs->max_tokens;
        a->logprobs_on = bs->logprobs_on;
        a->sampler_on = false;
        while (ev.size() < stat_events() + 4) {
            cudaEvent_t e = nullptr;
            Q3_CUDA(cudaEventCreate(&e));
            ev.push_back(e);
        }
        cudaEvent_t* e = ev.data() + stat_events();
        Q3_CUDA(cudaEventRecord(e[0], st));
        upload_staged(h, a);
        if (!(copies_pending(h, a) && a->n_tok > 0)) run_mel(h, a);  // else interleaved with the convolution stack, as in batch_run
        Q3_CUDA(cudaEventRecord(e[1], st));
        reserve_encoder(h, a);
        run_encoder(h, a, a->mel_out.as<float>());
        finish_upload(a);
        Q3_CUDA(cudaEventRecord(e[2], st));
        reserve_decoder(h, a);
        const int* ints = a->ints.as<int>();
        embed_splice_launch(ints + a->o_ids, ints + a->o_audio_src, h->model->embed, a->audio.as<bf16>(), a->dx.as<bf16>(), a->R, h->cfg.dec_hidden, st);
        h->launches++;
        decoder_layers(h, a, a->R, true);
        lm_head_argmax(h, a, ints + a->o_last_row);
        {
            PdlScope pdl(env_int("Q3ASR_NO_PDL", 0) == 0 && !h->prof_on);  // a programmatic dependent of the LM head's reduction
            decode_admit_launch(decode_state(h, bs, stop_on_eos, false), a->st_next_tok.as<int32_t>(), a->st_next_val.as<float>(),
                                bs->logprobs_on ? a->st_next_lp.as<float>() : nullptr, ints + a->o_seq_len, row0, k, staged_seq0, st);
            h->launches++;
        }
        Q3_CUDA(cudaEventRecord(e[3], st));
        bs->dec_rows = row0 + k;
        bs->stat_admissions++;
        bs->stat_admitted += (unsigned long long)k;
        staged = -1;
    }
    size_t stat_events() const { return (size_t)bs->stat_admissions * 4; }

    void decode() {
        cudaStream_t st = h->stream;
        const bool use_graph = env_int("Q3ASR_NO_GRAPH", 0) == 0;
        const int threshold = std::min(max_rows, std::max(4, max_rows / 4));  // today's compaction threshold at max_rows rows
        int* h_active = reinterpret_cast<int*>(bs->h_out.p);
        bool graph_ok = false;
        unsigned long long per_step = 0;
        auto rows_changed = [&]() {
            graph_ok = false;
            bs->mega_ready = false;
            if (bs->dec_rows > 0 && mega_wanted(h, bs)) megastep_prepare(h, bs);
        };
        rows_changed();
        stage(threshold);
        // every utterance needs at most max_tokens steps; a poll window without an active row always ends in an admission or the end
        const long long max_steps = (long long)batch * (bs->max_tokens + 32) + 64;
        long long steps = 0;
        for (;;) {
            for (int i = 0; i < 16 && bs->dec_rows > 0; i++, steps++) {
                if (!use_graph || h->prof_on || !h->decode_warm) {
                    decode_step_kernels(h, bs, stop_on_eos, false);
                    h->decode_warm = true;
                } else {
                    if (!graph_ok) {
                        per_step = capture_step_graph(h, bs, stop_on_eos, false);
                        graph_ok = true;
                    }
                    Q3_CUDA(cudaGraphLaunch(bs->step_graph, st));
                    h->launches += per_step;
                }
                bs->stat_steps++;
                bs->stat_row_steps += (unsigned long long)bs->dec_rows;
            }
            Q3_CHECK(steps <= max_steps, Q3ASR_ERR_STATE, "continuous: the decode loop did not finish");
            Q3_CUDA(cudaMemcpyAsync(h_active, bs->st_scalars.p, sizeof(int), cudaMemcpyDeviceToHost, st));
            Q3_CUDA(cudaStreamSynchronize(st));
            const int n_live = *h_active;
            if (n_live <= 0 && staged < 0 && next_stage >= batch) break;
            if (staged >= 0 && max_rows - n_live >= staged_k) {
                if (bs->dec_rows > n_live) partition(n_live);
                admit();
                rows_changed();
                stage(threshold);
            } else if (staged < 0 && n_live < bs->dec_rows && bs->dec_rows - n_live >= std::max(4, bs->dec_rows / 4)) {
                partition(n_live);  // nothing waits any more: shrink the batch as a static run does
                rows_changed();
            }
        }
        bs->steps_done = (int)std::min<long long>(steps, 1 << 30);
    }
};

}  // namespace

void transcribe_continuous(Handle* h, const float* const* pcm, const size_t* n, const int* rates, int batch, const q3asr_prompt* prompts,
                           int max_tokens, int stop_on_eos, int max_rows, int32_t* ids_out, int* lens_out, float* lp_out) {
    if (max_rows <= 0) max_rows = SKINNY_MAX_ROWS;
    Q3_CHECK(max_rows <= SKINNY_MAX_ROWS, Q3ASR_ERR_INVALID, "transcribe_continuous: max_rows > 256");
    Q3_CHECK(pcm != nullptr && n != nullptr && ids_out != nullptr && lens_out != nullptr && batch > 0 && batch <= (1 << 16), Q3ASR_ERR_INVALID,
             "transcribe_continuous: null argument, empty batch or more than 65536 utterances");
    Q3_CHECK(max_tokens >= 1 && max_tokens <= (1 << 20), Q3ASR_ERR_INVALID, "transcribe_continuous: max_tokens out of range");
    Q3_CHECK(h->loaded && h->model, Q3ASR_ERR_STATE, "weights are not loaded (q3asr_init_random / q3asr_load_safetensors)");
    // every utterance is checked up front (a later group must not fail mid-decode), and the KV pages are planned for the longest
    // prompt of the whole request: an utterance with a long context admitted late still fits its block
    int max_prompt = 0;
    for (int b = 0; b < batch; b++) {
        Q3_CHECK(pcm[b] != nullptr && n[b] < (size_t)1 << 30 && (rates == nullptr || rates[b] > 0), Q3ASR_ERR_INVALID,
                 "transcribe_continuous: null clip, clip too long or bad sample rate");
        const size_t n16 = rates != nullptr && rates[b] != 16000 ? resample_len(n[b], rates[b], 16000) : n[b];
        Q3_CHECK(n16 >= (size_t)MEL_HOP && n16 < (size_t)1 << 30, Q3ASR_ERR_INVALID,
                 "transcribe_continuous: every clip needs at least 160 samples at 16 kHz (one mel frame)");
        std::vector<int32_t> ids;
        int at = 0;
        build_prompt(h->cfg, prompts ? &prompts[b] : nullptr, encoder_tokens_for(mel_frames_for(n16)), &ids, &at);
        max_prompt = std::max(max_prompt, (int)ids.size());
    }
    const int rows = std::min(batch, max_rows);
    BatchState* bs = fresh_batch(h);
    ContinuousRun run{h, bs, pcm, n, rates, prompts, batch, max_rows, stop_on_eos};
    run.next_stage = rows;
    cudaStream_t st = h->stream;
    batch_upload_into(h, bs, pcm, n, rows, prompts, rates, true, false);
    bs->n_seqs = batch;
    bs->page_prompt = max_prompt;
    bs->per_seq_steps = true;
    bs->logprobs_on = lp_out != nullptr;
    plan_pages(h, bs, max_tokens);
    Q3_CUDA(cudaEventRecord(bs->ev[0], st));
    if (!(copies_pending(h, bs) && bs->n_tok > 0)) run_mel(h, bs);
    Q3_CUDA(cudaEventRecord(bs->ev[1], st));
    reserve_encoder(h, bs);
    run_encoder(h, bs, bs->mel_out.as<float>());
    finish_upload(bs);
    Q3_CUDA(cudaEventRecord(bs->ev[2], st));
    reserve_decoder(h, bs);
    run_prefill(h, bs, stop_on_eos, false);
    Q3_CUDA(cudaEventRecord(bs->ev[3], st));
    run.decode();
    Q3_CUDA(cudaEventRecord(bs->ev[4], st));
    batch_download(h, ids_out, max_tokens, lens_out);  // (synchronises; stage times of the first group)
    if (lp_out) batch_download_logprobs(h, lp_out, max_tokens);
    float adm[3] = {0.f, 0.f, 0.f};
    for (size_t i = 0; i + 3 < run.ev.size() && i < run.stat_events(); i += 4)
        for (int s = 0; s < 3; s++) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, run.ev[i + s], run.ev[i + s + 1]) == cudaSuccess) adm[s] += ms;
        }
    for (int s = 0; s < 3; s++) {
        h->stage_ms[s] += adm[s];
        h->stage_ms[3] -= adm[s];  // the admissions ran inside the decode window
    }
}

}  // namespace q3
