// weights.cu — named weight tensors (the reference's safetensors keys), deterministic random
// initialisation, and the kernel-ready derived layouts.
//
// Key contract: /root/reference/Sources/Qwen3ASR/WeightLoading.swift:17-126 (audio_tower.* / model.*
// prefixes), :235-323 (per-module names).  Linear.weight is [out, in]; Conv2d.weight is MLX layout
// [O, kH, kW, I] (:54-56).  The ASR model has no lm_head: the embedding is tied (Qwen3ASR.swift:253-256).
#include <stdlib.h>
#include <string.h>

#include "model.h"

namespace q3 {

namespace {

uint64_t fnv1a(const std::string& s) {
    uint64_t h = 0xcbf29ce484222325ULL;
    for (unsigned char c : s) {
        h ^= c;
        h *= 0x100000001b3ULL;
    }
    return h;
}
uint64_t splitmix_host(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

bool is_norm_weight(const std::string& n) {
    auto ends = [&](const char* s) {
        const size_t l = strlen(s);
        return n.size() >= l && n.compare(n.size() - l, l, s) == 0;
    };
    return ends("layer_norm.weight") || ends("ln_post.weight") || ends("layernorm.weight") || ends("_norm.weight") ||
           n == "model.norm.weight";
}

// dst[r, :] (ld_dst) = src[r, :] for `rows` rows of `cols` bf16
void copy_rows(bf16* dst, size_t ld_dst, const bf16* src, size_t ld_src, size_t rows, size_t cols, cudaStream_t st) {
    Q3_CUDA(cudaMemcpy2DAsync(dst, ld_dst * 2, src, ld_src * 2, cols * 2, rows, cudaMemcpyDeviceToDevice, st));
}

__global__ void permute_conv_out_kernel(const bf16* w, bf16* out, int d, int C) {
    // out[n][f*C + c] = w[n][c*16 + f]
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long K = (long)C * 16;
    if (idx >= (long)d * K) return;
    const int n = (int)(idx / K);
    const int k = (int)(idx % K);
    const int f = k / C, c = k % C;
    out[idx] = w[(long)n * K + c * 16 + f];
}

__global__ void pe_kernel(float* pe, int tpc, int d) {
    // AudioEncoder.swift:171-199: [sin | cos], increment ln(10000)/(d/2 - 1), Float arithmetic
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= tpc * d) return;
    const int t = idx / d, j = idx % d, half = d / 2;
    const float inc = logf(10000.0f) / (float)(half - 1);
    const int i = j < half ? j : j - half;
    const float inv = expf((float)i * -inc);
    const float a = (float)t * inv;
    pe[idx] = j < half ? sinf(a) : cosf(a);
}

template <typename T>
T* dev_alloc(Model* m, size_t n, size_t* total) {
    T* p = nullptr;
    const size_t bytes = (n * sizeof(T) + 255) & ~size_t(255);
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) throw Error(Q3ASR_ERR_NOMEM, std::string("cudaMalloc(weights): ") + cudaGetErrorString(e));
    m->owned.push_back(p);
    m->owned_bytes += bytes;
    *total += bytes;
    return p;
}

const Tensor& need(const Handle* h, const std::string& name) {
    auto it = h->tensor_index.find(name);
    Q3_CHECK(it != h->tensor_index.end() && h->tensors[it->second].d != nullptr, Q3ASR_ERR_STATE, "missing weight tensor: " + name);
    return h->tensors[it->second];
}

void ensure_tensor_table(Handle* h) {
    if (!h->tensors.empty()) return;
    std::vector<std::pair<std::string, std::vector<int64_t>>> specs;
    model_tensor_specs(h->cfg, &specs);
    h->tensors.reserve(specs.size());
    for (auto& s : specs) {
        Tensor t;
        t.name = s.first;
        t.shape = s.second;
        t.numel = 1;
        for (int64_t v : t.shape) t.numel *= (size_t)v;
        h->tensor_index[t.name] = (int)h->tensors.size();
        h->tensors.push_back(std::move(t));
    }
}

void alloc_tensor(Handle* h, Tensor& t) {
    if (t.d) return;
    const size_t bytes = (t.numel * 2 + 255) & ~size_t(255);
    cudaError_t e = cudaMalloc(&t.d, bytes);
    if (e != cudaSuccess) throw Error(Q3ASR_ERR_NOMEM, "cudaMalloc(" + t.name + "): " + cudaGetErrorString(e));
    h->dev_bytes += bytes;
}

}  // namespace

void config_validate(const q3asr_config& c) {
    Q3_CHECK(c.enc_d_model > 0 && c.enc_d_model % 128 == 0 && c.enc_d_model <= 2048, Q3ASR_ERR_INVALID, "enc_d_model must be a multiple of 128");
    Q3_CHECK(c.enc_heads > 0 && c.enc_d_model == c.enc_heads * 64, Q3ASR_ERR_INVALID, "encoder head dim must be 64");
    Q3_CHECK(c.enc_ffn % 128 == 0 && c.enc_out_dim % 128 == 0 && c.enc_layers > 0, Q3ASR_ERR_INVALID, "encoder dims must be multiples of 128");
    Q3_CHECK(c.enc_conv_ch % 32 == 0 && c.enc_conv_ch > 0, Q3ASR_ERR_INVALID, "enc_conv_ch must be a multiple of 32");
    Q3_CHECK(c.enc_n_window > 0 && c.enc_n_window_infer % (2 * c.enc_n_window) == 0, Q3ASR_ERR_INVALID, "window configuration");
    Q3_CHECK(conv_len3(2 * c.enc_n_window) * (c.enc_n_window_infer / (2 * c.enc_n_window)) <= 128, Q3ASR_ERR_INVALID,
             "attention window larger than 128 tokens");
    Q3_CHECK(c.dec_head_dim == 128, Q3ASR_ERR_INVALID, "decoder head dim must be 128");
    Q3_CHECK(c.dec_hidden % 128 == 0 && c.dec_hidden <= 2048 && c.dec_inter % 64 == 0, Q3ASR_ERR_INVALID, "decoder dims");
    Q3_CHECK(c.dec_hidden == c.enc_out_dim, Q3ASR_ERR_INVALID, "encoder output dim must equal decoder hidden size");
    Q3_CHECK(c.dec_heads % c.dec_kv_heads == 0 && (c.dec_heads / c.dec_kv_heads) <= 2, Q3ASR_ERR_INVALID, "GQA group must be 1 or 2");
    Q3_CHECK(c.dec_vocab % 128 == 0 && c.dec_layers > 0, Q3ASR_ERR_INVALID, "vocab must be a multiple of 128");
    Q3_CHECK(c.classify_num >= 0 && c.classify_num <= 65536, Q3ASR_ERR_INVALID, "classify_num out of range");
}

void model_tensor_specs(const q3asr_config& c, std::vector<std::pair<std::string, std::vector<int64_t>>>* out) {
    auto add = [&](const std::string& n, std::vector<int64_t> s) { out->emplace_back(n, std::move(s)); };
    const int64_t C = c.enc_conv_ch, d = c.enc_d_model, f = c.enc_ffn;
    const std::string a = "audio_tower.";
    add(a + "conv2d1.weight", {C, 3, 3, 1});
    add(a + "conv2d1.bias", {C});
    add(a + "conv2d2.weight", {C, 3, 3, C});
    add(a + "conv2d2.bias", {C});
    add(a + "conv2d3.weight", {C, 3, 3, C});
    add(a + "conv2d3.bias", {C});
    add(a + "conv_out.weight", {d, C * 16});
    for (int l = 0; l < c.enc_layers; l++) {
        const std::string p = a + "layers." + std::to_string(l) + ".";
        for (const char* nm : {"q_proj", "k_proj", "v_proj", "out_proj"}) {
            add(p + "self_attn." + nm + ".weight", {d, d});
            add(p + "self_attn." + nm + ".bias", {d});
        }
        add(p + "self_attn_layer_norm.weight", {d});
        add(p + "self_attn_layer_norm.bias", {d});
        add(p + "fc1.weight", {f, d});
        add(p + "fc1.bias", {f});
        add(p + "fc2.weight", {d, f});
        add(p + "fc2.bias", {d});
        add(p + "final_layer_norm.weight", {d});
        add(p + "final_layer_norm.bias", {d});
    }
    add(a + "ln_post.weight", {d});
    add(a + "ln_post.bias", {d});
    add(a + "proj1.weight", {d, d});
    add(a + "proj1.bias", {d});
    add(a + "proj2.weight", {(int64_t)c.enc_out_dim, d});
    add(a + "proj2.bias", {(int64_t)c.enc_out_dim});
    const int64_t h = c.dec_hidden, hd = c.dec_head_dim, I = c.dec_inter;
    add("model.embed_tokens.weight", {(int64_t)c.dec_vocab, h});
    for (int l = 0; l < c.dec_layers; l++) {
        const std::string p = "model.layers." + std::to_string(l) + ".";
        add(p + "self_attn.q_proj.weight", {c.dec_heads * hd, h});
        add(p + "self_attn.k_proj.weight", {c.dec_kv_heads * hd, h});
        add(p + "self_attn.v_proj.weight", {c.dec_kv_heads * hd, h});
        add(p + "self_attn.o_proj.weight", {h, c.dec_heads * hd});
        add(p + "self_attn.q_norm.weight", {hd});
        add(p + "self_attn.k_norm.weight", {hd});
        add(p + "input_layernorm.weight", {h});
        add(p + "post_attention_layernorm.weight", {h});
        add(p + "mlp.gate_proj.weight", {I, h});
        add(p + "mlp.up_proj.weight", {I, h});
        add(p + "mlp.down_proj.weight", {h, I});
    }
    add("model.norm.weight", {h});
    if (c.classify_num > 0) {  // WeightLoading.swift:177-179, 229: the aligner's head keeps the lm_head.* keys
        add("lm_head.weight", {(int64_t)c.classify_num, h});
        add("lm_head.bias", {(int64_t)c.classify_num});
    }
}

// Random initialisation (weights are not available offline; SURVEY.md section 8d): bf16(scale * approx-normal) per tensor,
// norm scales constant.  scale = 0.02 for the audio tower and the aligner's head; for the text decoder 0.08 (o_proj 0.04), the
// tied embedding 0.15 with "loud" rows (x 2^k for one row in 16^k, k <= 4), and q_norm / k_norm scales of 2 (other norms 1).
// Why not 0.02 everywhere: the decoder's hidden state is then an average over the (nearly identical) audio rows that ignores
// the last token, greedy ids collapse to one repeated id and id parity is vacuous (SURVEY.md section 7).  With these values
// the token path carries weight, the attention is peaked (scores ~ N(0, 4^2)) so that it picks out individual earlier tokens
// (history and position dependence: no short cycles), and the heavy-tailed rows of the tied head keep the top-1 / top-2 margins of
// the bf16 logits above rounding noise; tests/golden/make_golden.py measures and asserts all three on the oracle.
// The generator is integer-only up to one fp32 multiply and one exact power-of-two scale, so the NumPy twin
// (oracle/weights.py) reproduces it bit for bit.
void model_init_random(Handle* h, uint64_t seed) {
    ensure_tensor_table(h);
    for (Tensor& t : h->tensors) {
        alloc_tensor(h, t);
        if (is_norm_weight(t.name)) {
            const bool qk = t.name.find("self_attn.q_norm.") != std::string::npos || t.name.find("self_attn.k_norm.") != std::string::npos;
            fill_bf16_launch(t.d, t.numel, qk ? 2.0f : 1.0f, h->stream);
        } else {
            const uint64_t s = splitmix_host(seed ^ fnv1a(t.name));
            const bool embed = t.name == "model.embed_tokens.weight";
            const bool text = t.name.rfind("model.", 0) == 0;
            const bool oproj = text && t.name.find("self_attn.o_proj.") != std::string::npos;
            random_init_launch(t.d, t.numel, s, embed ? 0.15f : oproj ? 0.04f : text ? 0.08f : 0.02f, h->stream,
                               embed ? splitmix_host(seed ^ fnv1a(t.name + "#loud")) : 0, embed ? (int)t.shape.back() : 0);
        }
        h->launches++;
    }
    Q3_CUDA(cudaGetLastError());
    model_commit(h);
}

void model_set_tensor(Handle* h, const char* name, const void* data, int dtype, const int64_t* shape, int ndim) {
    Q3_CHECK(name && data && shape && ndim > 0 && ndim <= 4, Q3ASR_ERR_INVALID, "set_tensor: bad argument");
    ensure_tensor_table(h);
    auto it = h->tensor_index.find(name);
    Q3_CHECK(it != h->tensor_index.end(), Q3ASR_ERR_INVALID, std::string("set_tensor: unknown tensor ") + name);
    Tensor& t = h->tensors[it->second];
    size_t n = 1;
    for (int i = 0; i < ndim; i++) n *= (size_t)shape[i];
    bool same = (int)t.shape.size() == ndim;
    for (int i = 0; same && i < ndim; i++) same = t.shape[i] == shape[i];
    // PyTorch conv layout [O, I, kH, kW] is accepted for the conv weights and transposed to [O, kH, kW, I]
    // (WeightLoading.swift:185-187, 289-291)
    const bool is_conv = ndim == 4 && t.shape.size() == 4;
    const bool torch_layout = is_conv && !same && shape[0] == t.shape[0] && shape[1] == t.shape[3] && shape[2] == 3 && shape[3] == 3;
    Q3_CHECK(same || torch_layout, Q3ASR_ERR_INVALID, std::string("set_tensor: shape mismatch for ") + name);
    alloc_tensor(h, t);
    std::vector<float> f(n);
    if (dtype == 0) {
        memcpy(f.data(), data, n * 4);
    } else if (dtype == 1) {
        const uint16_t* s = (const uint16_t*)data;
        for (size_t i = 0; i < n; i++) {
            uint32_t u = (uint32_t)s[i] << 16;
            memcpy(&f[i], &u, 4);
        }
    } else if (dtype == 2) {
        const uint16_t* s = (const uint16_t*)data;
        for (size_t i = 0; i < n; i++) {
            const uint32_t hbits = s[i], sign = (hbits >> 15) & 1, ex = (hbits >> 10) & 31, man = hbits & 1023;
            float v;
            if (ex == 0) v = ldexpf((float)man, -24);
            else if (ex == 31) v = man ? NAN : INFINITY;
            else v = ldexpf((float)(man | 1024), (int)ex - 25);
            f[i] = sign ? -v : v;
        }
    } else {
        throw Error(Q3ASR_ERR_INVALID, "set_tensor: dtype must be 0 (fp32), 1 (bf16) or 2 (fp16)");
    }
    if (torch_layout) {
        std::vector<float> g(n);
        const int64_t O = shape[0], I = shape[1];
        for (int64_t o = 0; o < O; o++)
            for (int64_t i = 0; i < I; i++)
                for (int64_t k = 0; k < 9; k++) g[(o * 9 + k) * I + i] = f[(o * I + i) * 9 + k];
        f.swap(g);
    }
    std::vector<uint16_t> b(n);
    for (size_t i = 0; i < n; i++) {  // round to nearest even
        uint32_t u;
        memcpy(&u, &f[i], 4);
        if ((u & 0x7fffffffu) > 0x7f800000u) b[i] = (uint16_t)((u >> 16) | 0x40);
        else b[i] = (uint16_t)((u + 0x7fffu + ((u >> 16) & 1)) >> 16);
    }
    Q3_H2D_SYNC(t.d, b.data(), n * 2);
    h->loaded = false;  // derived layouts are stale until q3asr_commit_weights
}

void model_get_tensor(const Handle* h, const char* name, float* out, size_t n) {
    Q3_CHECK(name && out, Q3ASR_ERR_INVALID, "get_tensor: bad argument");
    const Tensor& t = need(h, name);
    Q3_CHECK(n >= t.numel, Q3ASR_ERR_INVALID, "get_tensor: output buffer too small");
    std::vector<uint16_t> b(t.numel);
    Q3_CUDA(cudaStreamSynchronize(h->stream));
    Q3_CUDA(cudaMemcpy(b.data(), t.d, t.numel * 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < t.numel; i++) {
        const uint32_t u = (uint32_t)b[i] << 16;
        memcpy(&out[i], &u, 4);
    }
}

static void free_model(Handle* h) {
    if (!h->model) return;
    for (void* p : h->model->owned) cudaFree(p);
    h->dev_bytes -= h->model->owned_bytes;
    h->model.reset();
}

void model_commit(Handle* h) {
    ensure_tensor_table(h);
    free_model(h);
    const q3asr_config& c = h->cfg;
    const Geom g(c);
    std::unique_ptr<Model> mp(new Model());
    Model* m = mp.get();
    h->model = std::move(mp);  // owned buffers are released through the handle if anything below throws
    cudaStream_t st = h->stream;
    const std::string a = "audio_tower.";
    auto W = [&](const std::string& n) { return need(h, n).d; };
    m->conv1_w = W(a + "conv2d1.weight");
    m->conv1_b = W(a + "conv2d1.bias");
    m->conv2_w = W(a + "conv2d2.weight");
    m->conv2_b = W(a + "conv2d2.bias");
    m->conv3_w = W(a + "conv2d3.weight");
    m->conv3_b = W(a + "conv2d3.bias");
    const int d = c.enc_d_model;
    {
        const long K = (long)g.C * 16;
        m->conv_out_w = dev_alloc<bf16>(m, (size_t)d * K, &h->dev_bytes);
        permute_conv_out_kernel<<<(unsigned)(((long)d * K + 255) / 256), 256, 0, st>>>(W(a + "conv_out.weight"), m->conv_out_w, d, g.C);
        h->launches++;
    }
    m->enc.resize(c.enc_layers);
    for (int l = 0; l < c.enc_layers; l++) {
        const std::string p = a + "layers." + std::to_string(l) + ".";
        EncLayerW& e = m->enc[l];
        e.ln1_w = W(p + "self_attn_layer_norm.weight");
        e.ln1_b = W(p + "self_attn_layer_norm.bias");
        e.ln2_w = W(p + "final_layer_norm.weight");
        e.ln2_b = W(p + "final_layer_norm.bias");
        e.qkv_w = dev_alloc<bf16>(m, (size_t)3 * d * d, &h->dev_bytes);
        e.qkv_b = dev_alloc<bf16>(m, (size_t)3 * d, &h->dev_bytes);
        const char* nm[3] = {"q_proj", "k_proj", "v_proj"};
        for (int i = 0; i < 3; i++) {
            Q3_CUDA(cudaMemcpyAsync(e.qkv_w + (size_t)i * d * d, W(p + "self_attn." + nm[i] + ".weight"), (size_t)d * d * 2,
                                    cudaMemcpyDeviceToDevice, st));
            Q3_CUDA(cudaMemcpyAsync(e.qkv_b + (size_t)i * d, W(p + "self_attn." + nm[i] + ".bias"), (size_t)d * 2,
                                    cudaMemcpyDeviceToDevice, st));
        }
        e.o_w = W(p + "self_attn.out_proj.weight");
        e.o_b = W(p + "self_attn.out_proj.bias");
        e.fc1_w = W(p + "fc1.weight");
        e.fc1_b = W(p + "fc1.bias");
        e.fc2_w = W(p + "fc2.weight");
        e.fc2_b = W(p + "fc2.bias");
    }
    m->ln_post_w = W(a + "ln_post.weight");
    m->ln_post_b = W(a + "ln_post.bias");
    m->proj1_w = W(a + "proj1.weight");
    m->proj1_b = W(a + "proj1.bias");
    m->proj2_w = W(a + "proj2.weight");
    m->proj2_b = W(a + "proj2.bias");
    m->pe = dev_alloc<float>(m, (size_t)g.tpc * d, &h->dev_bytes);
    pe_kernel<<<(g.tpc * d + 255) / 256, 256, 0, st>>>(m->pe, g.tpc, d);
    h->launches++;

    // decoder
    const int hdim = c.dec_hidden, hd = c.dec_head_dim, I = c.dec_inter;
    const int nq = c.dec_heads * hd, nkv = c.dec_kv_heads * hd;
    m->embed = W("model.embed_tokens.weight");
    m->final_norm = W("model.norm.weight");
    Q3_CHECK(I % GU_UNIT == 0, Q3ASR_ERR_INVALID, "dec_inter must be a multiple of 32");
    m->dec.resize(c.dec_layers);
    for (int l = 0; l < c.dec_layers; l++) {
        const std::string p = "model.layers." + std::to_string(l) + ".";
        DecLayerW& e = m->dec[l];
        e.in_ln = W(p + "input_layernorm.weight");
        e.post_ln = W(p + "post_attention_layernorm.weight");
        e.q_norm = W(p + "self_attn.q_norm.weight");
        e.k_norm = W(p + "self_attn.k_norm.weight");
        e.o_w = W(p + "self_attn.o_proj.weight");
        e.down_w = W(p + "mlp.down_proj.weight");
        e.qkv_w = dev_alloc<bf16>(m, (size_t)(nq + 2 * nkv) * hdim, &h->dev_bytes);
        Q3_CUDA(cudaMemcpyAsync(e.qkv_w, W(p + "self_attn.q_proj.weight"), (size_t)nq * hdim * 2, cudaMemcpyDeviceToDevice, st));
        Q3_CUDA(cudaMemcpyAsync(e.qkv_w + (size_t)nq * hdim, W(p + "self_attn.k_proj.weight"), (size_t)nkv * hdim * 2,
                                cudaMemcpyDeviceToDevice, st));
        Q3_CUDA(cudaMemcpyAsync(e.qkv_w + (size_t)(nq + nkv) * hdim, W(p + "self_attn.v_proj.weight"), (size_t)nkv * hdim * 2,
                                cudaMemcpyDeviceToDevice, st));
        // gate/up interleaved in units of GU_UNIT rows: [g 0..31 | u 0..31 | g 32..63 | u 32..63 | ...], so any tile that is a
        // multiple of 64 rows (columns of the accumulator) holds matching gate and up values for the SwiGLU epilogue
        e.gu_w = dev_alloc<bf16>(m, (size_t)2 * I * hdim, &h->dev_bytes);
        const int half = GU_UNIT;
        const bf16* gw = W(p + "mlp.gate_proj.weight");
        const bf16* uw = W(p + "mlp.up_proj.weight");
        // rows of tile t: a 2-D copy with destination pitch 2*half rows
        copy_rows(e.gu_w, (size_t)2 * half * hdim, gw, (size_t)half * hdim, I / half, (size_t)half * hdim, st);
        copy_rows(e.gu_w + (size_t)half * hdim, (size_t)2 * half * hdim, uw, (size_t)half * hdim, I / half, (size_t)half * hdim, st);
    }
    if (c.classify_num > 0) {
        m->cls_pad = (c.classify_num + 63) / 64 * 64;
        m->cls_w = dev_alloc<bf16>(m, (size_t)m->cls_pad * hdim, &h->dev_bytes);
        m->cls_b = dev_alloc<bf16>(m, (size_t)m->cls_pad, &h->dev_bytes);
        Q3_CUDA(cudaMemsetAsync(m->cls_w, 0, (size_t)m->cls_pad * hdim * 2, st));
        Q3_CUDA(cudaMemsetAsync(m->cls_b, 0, (size_t)m->cls_pad * 2, st));
        Q3_CUDA(cudaMemcpyAsync(m->cls_w, W("lm_head.weight"), (size_t)c.classify_num * hdim * 2, cudaMemcpyDeviceToDevice, st));
        Q3_CUDA(cudaMemcpyAsync(m->cls_b, W("lm_head.bias"), (size_t)c.classify_num * 2, cudaMemcpyDeviceToDevice, st));
    }
    {
        std::vector<float> inv(hd / 2);
        for (int i = 0; i < hd / 2; i++) inv[i] = (float)pow((double)c.dec_rope_theta, -(double)(2 * i) / (double)hd);
        m->inv_freq = dev_alloc<float>(m, hd / 2, &h->dev_bytes);
        Q3_CUDA(cudaMemcpyAsync(m->inv_freq, inv.data(), sizeof(float) * inv.size(), cudaMemcpyHostToDevice, st));
        Q3_CUDA(cudaStreamSynchronize(st));  // inv is a stack-lifetime host buffer
    }
    Q3_CUDA(cudaStreamSynchronize(st));
    Q3_CUDA(cudaGetLastError());
    h->loaded = true;
}

void model_unload(Handle* h) {
    h->batch.reset();
    h->adm[0].reset();
    h->adm[1].reset();
    free_model(h);
    for (Tensor& t : h->tensors) {
        if (t.d) {
            cudaFree(t.d);
            h->dev_bytes -= (t.numel * 2 + 255) & ~size_t(255);
            t.d = nullptr;
        }
    }
    h->loaded = false;
}

}  // namespace q3
