// mrd_ctx: the per-device forward engine behind the C ABI.
//
// Owns (a) the packed weights (BN-folded NHWC conv filters, fused QKV, pre-multiplied cross-attention
// projections; bf16 matrices + fp32 vectors), (b) the activation workspace, sized for one micro-batch
// so the ResNet / BERT intermediates of a chunk stay L2-resident between producer and consumer
// kernels, and (c) launch plans: every GEMM/conv launch of a forward has its TMA descriptors and tile
// schedule built once per shape and then replayed, so a forward is a straight sequence of kernel
// launches on the caller's stream with no host-side descriptor work and no synchronisation.
//
// Reference path replaced: MultimodalClassifier.forward and the module forwards it calls
// (src/multimodal_classifier.py:131-177, src/cnn_encoder.py:168-184, src/text_encoder.py:95-127,
// src/fusion_model.py:245-291) plus torchvision ResNet (TV:models/resnet.py:266-282) and HF BertModel
// (HF:models/bert/modeling_bert.py:628-691).

#include <mrd_b200.h>

#include <stdio.h>
#include <string.h>

#include <map>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "attention.h"
#include "conv_chain.h"
#include "dgrad.h"
#include "elementwise.h"
#include "fp32_check.h"
#include "gemm_conv.h"
#include "simt_gemm.h"
#include "tail_fused.h"
#include "tma_host.h"
#include "train_kernels.h"

using namespace mrd;
typedef __nv_bfloat16 bf16;

namespace {

struct Tensor {
    const float* p = nullptr;
    long long d[4] = {0, 0, 0, 0};
    long long numel() const {
        long long n = 1;
        for (int i = 0; i < 4; ++i)
            if (d[i] > 0) n *= d[i];
        return n;
    }
};

struct ConvW {
    bf16* w = nullptr;
    float* b = nullptr;
    int cin = 0, cout = 0, k = 0, stride = 1;
};

struct Bottleneck {
    ConvW c1, c2, c3, ds;
    bool has_ds = false;
    // conv3 and the downsample branch as one K-concatenated 1x1 convolution: [Cout][c3.cin + ds.cin] bf16, bias
    // = the two folded BatchNorm shifts added (plan_conv1x1_dual)
    bf16* c3ds_w = nullptr;
    float* c3ds_b = nullptr;
};

struct LinearW {
    bf16* w = nullptr;
    float* b = nullptr;
    int in = 0, out = 0;
};

struct BertLayerW {
    LinearW qkv, o, f1, f2;
    float *ln1g = nullptr, *ln1b = nullptr, *ln2g = nullptr, *ln2b = nullptr;
};

struct CnnPlan {
    int B = 0, H = 0, W = 0;
    GemmLaunch stem;   // conv + BN + ReLU + maxpool in one launch (plan_stem_pool)
    struct BlockPlan {
        GemmLaunch c1, c2, c3, ds;
        bool has_ds = false;
        bool fused_ds = false;   // c3 = conv3 + downsample + add (plan_conv1x1_dual); ds is not launched
        // conv3 (+downsample) + add of THIS block and conv1 of the NEXT block as one launch (conv_chain.h): c3 / ds
        // of this block and c1 of the next one are then not launched
        bool chained = false, c1_in_prev_chain = false;
        ChainLaunch chain;
    };
    std::vector<BlockPlan> blocks;
    const bf16* final_act = nullptr;  // layer4 output [B, H/32*W/32, 2048]
    int final_hw = 0;
};

struct TextPlan {
    int B = 0, S = 0;
    int blocked_qkv = 0;  // QKV written as [36][T][64] for the tcgen05 attention (S <= 128)
    struct LayerPlan {
        GemmLaunch qkv, o, f1, f2;
        GemmLaunch f2_ln;   // FFN2 + residual + LayerNorm in one launch (plan_gemm_ln)
        bool f2_fused = false;
    };
    std::vector<LayerPlan> layers;
    // last layer, CLS rows only (M = B): everything after its attention feeds nothing but the CLS row
    // (src/text_encoder.py:118), so the out-projection, both LayerNorms and the FFN run on B rows
    GemmLaunch o_cls, f1_cls, f2_cls;
    GemmLaunch f2_cls_ln;      // the same fused LayerNorm kernel as the full layers' FFN2 (identical arithmetic per row)
    bool f2_cls_fused = false;
};

struct BatchPlan {
    int B = 0;
    bool has_proj = false, has_fusion = false, has_head = false;
    GemmLaunch proj1, proj2;
    GemmLaunch ip, tp, i2t, t2i, f1, f2;
    std::vector<GemmLaunch> head;
    bool has_tail = false;   // fusion + head + softmax as ONE launch (tail_fused.h); the launches above stay planned
    TailLaunch tail;         // for the module-level entry points (mrd_fusion_fwd, mrd_head_fwd)
};

}  // namespace

namespace {
struct TrainState;  // engine_train.cuh
}

struct ProfRecord {
    const char* label = "";
    int cat = 0;
    double flops = 0, bytes = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

struct mrd_ctx {
    int device = 0;
    long long launches = 0;
    bool profiling = false;
    std::vector<ProfRecord> prof;
    std::vector<int> block_stage;          // ResNet stage (1..4) of each bottleneck
    std::map<std::string, std::string> label_pool;
    const char* label(const char* a, const char* b) {  // interned "a" + "b"
        std::string k = std::string(a) + b;
        auto it = label_pool.find(k);
        if (it == label_pool.end()) it = label_pool.emplace(k, k).first;
        return it->second.c_str();
    }
    long long dev_bytes = 0;
    std::vector<void*> weight_allocs;
    std::unordered_map<const void*, size_t> weight_bytes;

    // options
    // images per ResNet pass / tokens per BERT pass: larger passes are faster (more tiles per SM in every launch;
    // measured at 4096 samples, r02: 512 / 131072 -> 1024 / 262144 -> 2048 / 524288 = 36.5 -> 36.7 -> 37.2 k
    // samples/s) and the workspaces are sized by the batch that actually arrives (28 GB at 4096 samples)
    int img_chunk = 2048;
    int tok_chunk = 524288;
    int bert_heads = 12;
    float bert_ln_eps = 1e-12f;
    float bn_eps = 1e-5f;
    float fusion_ln_eps = 1e-5f;
    int fusion_heads = 8;
    int fusion_residual = 1;
    int head_act = MRD_ACT_RELU;
    // fp32 check mode (fp32_check.h): forwards run the plain-fp32 SIMT kernels on the caller's raw fp32
    // tensors; `raw` keeps the name table of the last load_weights (the host keeps the tensors alive)
    TrainState* train = nullptr;   // training step state (engine_train.cuh), created on first use
    long long text_ws_epoch = 0;   // bumped when the text workspace is re-carved (pointers change)
    long long cnn_ws_epoch = 0;    // same for the ResNet workspace
    long long text_run_epoch = 0;  // bumped by every eval-mode BERT pass (overwrites the packing tables)
    bool fp32_check = false;
    // load_weights synchronises the device before re-packing and the stream afterwards (safe for callers
    // that use several streams or free their tensors right away); "load_sync" = 0 drops both when the
    // caller keeps its tensors alive and works on one stream (the training loop: no host stall per step)
    bool load_sync = true;
    RawTable raw;
    Fp32Arena f32_ws;
    Fp32TrainSave f32_train;   // fp32 check of the training step: saved activations of the text encoder
    Fp32Opts f32_opts() const {
        Fp32Opts o;
        o.bert_heads = bert_heads; o.bert_ln_eps = bert_ln_eps; o.bn_eps = bn_eps;
        o.fusion_ln_eps = fusion_ln_eps; o.fusion_heads = fusion_heads;
        o.fusion_residual = fusion_residual; o.head_act = head_act;
        return o;
    }

    // ---- weights
    bool has_cnn = false, has_text = false, has_fusion = false, has_head = false;
    bool has_backbone = false, has_proj = false;   // has_cnn = both (they are handed over as separate groups)
    bf16* stem_w = nullptr;
    float* stem_b = nullptr;
    std::vector<Bottleneck> blocks;
    LinearW proj1, proj2;
    int feat_dim = 2048, img_emb_dim = 512;

    bf16* word_emb = nullptr;
    float *pos_type = nullptr, *emb_g = nullptr, *emb_b = nullptr;
    int vocab = 0, hidden = 768, max_pos = 512, ffn = 3072;
    std::vector<BertLayerW> layers;

    LinearW f_ip, f_tp, f_i2t, f_t2i, f_1, f_2;
    float *ln_i_g = nullptr, *ln_i_b = nullptr, *ln_t_g = nullptr, *ln_t_b = nullptr;
    int fusion_dim = 512, fusion_img_in = 512, fusion_txt_in = 768;

    bf16* tail_wbig = nullptr;        // [2F][img_in + txt_in]: both LayerNorm inputs straight from the embeddings
    float *tail_bbig = nullptr, *tail_scratch = nullptr;
    int tail_residual = -1;           // fusion_residual the packed tail weights were built with
    std::vector<LinearW> head_hidden;
    float *head_out_w = nullptr, *head_out_b = nullptr;
    int head_in = 0, head_last = 0, num_classes = 0;

    // ---- workspaces
    struct Arena {
        void* base = nullptr;
        size_t bytes = 0, used = 0;
    };
    Arena cnn_ws, text_ws, batch_ws;
    int cnn_ws_B = 0, cnn_ws_H = 0, cnn_ws_W = 0;
    int text_ws_tokens = 0, text_ws_seqs = 0;
    int batch_ws_B = 0;

    // cnn chunk buffers
    bf16 *xpad = nullptr, *stem_out = nullptr, *act0 = nullptr, *act1 = nullptr, *mid0 = nullptr,
         *mid1 = nullptr, *dsb = nullptr;
    struct PadBuf {  // zero-bordered [Bc][h+2][w+2][c] input of a flat-mode 3x3 convolution
        int h = 0, w = 0, c = 0;
        bf16* p = nullptr;
    };
    std::vector<PadBuf> pads;
    // text chunk buffers
    bf16 *t_h = nullptr, *t_h2 = nullptr, *t_qkv = nullptr, *t_ctx = nullptr, *t_tmp = nullptr,
         *t_ffn = nullptr;
    bf16 *t_cls_ctx = nullptr, *t_cls_h = nullptr, *t_cls_h2 = nullptr, *t_cls_tmp = nullptr,
         *t_cls_ffn = nullptr;  // CLS-row tail of the last layer
    float* t_bias = nullptr;   // key bias per packed row
    int *t_seq_off = nullptr, *t_row_tok = nullptr, *t_nrows = nullptr, *t_scratch = nullptr;
    void* t_ln_ws = nullptr;   // statistics exchange of the LayerNorm GEMMs (gemm_ln_ws_bytes; zero between launches)
    // batch buffers
    bf16 *b_pooled = nullptr, *b_projh = nullptr, *b_img = nullptr, *b_txt = nullptr, *b_ip = nullptr,
         *b_tp = nullptr, *b_prei = nullptr, *b_pret = nullptr, *b_cat = nullptr, *b_fh = nullptr,
         *b_fused = nullptr, *b_h[2] = {nullptr, nullptr};
    float* b_scratch_f32 = nullptr;  // [B, 1024] scratch for optional fp32 outputs nobody asked for

    std::map<std::pair<int, std::pair<int, int>>, CnnPlan> cnn_plans;
    std::map<std::pair<int, int>, TextPlan> text_plans;
    std::map<int, BatchPlan> batch_plans;
};

namespace {

#define MRD_TRY(expr)            \
    do {                         \
        int rc__ = (expr);       \
        if (rc__ != 0) return rc__; \
    } while (0)

int cuda_fail(cudaError_t e, const char* what) {
    set_last_error("%s: %s", what, cudaGetErrorString(e));
    return -static_cast<int>(e);
}

int dev_alloc(mrd_ctx* c, void** out, size_t bytes, bool track_weight) {
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
    c->dev_bytes += static_cast<long long>(bytes);
    if (track_weight) c->weight_allocs.push_back(*out);
    return 0;
}

template <typename T>
int walloc(mrd_ctx* c, T** out, long long n) {
    const size_t bytes = static_cast<size_t>(n) * sizeof(T);
    if (*out) {  // reload: repack in place when the tensor still fits
        auto it = c->weight_bytes.find(*out);
        if (it != c->weight_bytes.end() && it->second >= bytes) return 0;
        set_last_error("load_weights: a tensor grew since the previous load; create a new context");
        return -2;
    }
    void* p = nullptr;
    MRD_TRY(dev_alloc(c, &p, bytes, true));
    c->weight_bytes[p] = bytes;
    *out = static_cast<T*>(p);
    return 0;
}

int arena_reset(mrd_ctx* c, mrd_ctx::Arena* a, size_t bytes) {
    if (a->base && a->bytes >= bytes) {
        a->used = 0;
        return 0;
    }
    if (a->base) {
        // plans referencing this arena are cleared by the caller; wait for in-flight work first
        cudaDeviceSynchronize();
        cudaFree(a->base);
        c->dev_bytes -= static_cast<long long>(a->bytes);
        a->base = nullptr;
    }
    MRD_TRY(dev_alloc(c, &a->base, bytes, false));
    a->bytes = bytes;
    a->used = 0;
    return 0;
}

template <typename T>
T* arena_take(mrd_ctx::Arena* a, long long n) {
    size_t bytes = (static_cast<size_t>(n) * sizeof(T) + 1023) & ~static_cast<size_t>(1023);
    T* p = reinterpret_cast<T*>(static_cast<char*>(a->base) + a->used);
    a->used += bytes;
    return p;
}
inline size_t pad1k(long long n, size_t elt) {
    return (static_cast<size_t>(n) * elt + 1023) & ~static_cast<size_t>(1023);
}

// ------------------------------------------------------------------ weight table
struct Table {
    std::unordered_map<std::string, Tensor> m;
    const Tensor* find(const std::string& k) const {
        auto it = m.find(k);
        return it == m.end() ? nullptr : &it->second;
    }
    int need(const std::string& k, const Tensor** out) const {
        *out = find(k);
        if (!*out) {
            set_last_error("load_weights: missing tensor '%s'", k.c_str());
            return -2;
        }
        return 0;
    }
};

int load_conv_bn(mrd_ctx* c, const Table& t, const std::string& conv, const std::string& bn,
                 int stride, ConvW* out, cudaStream_t s) {
    const Tensor *w, *g, *b, *mu, *var;
    MRD_TRY(t.need(conv + ".weight", &w));
    MRD_TRY(t.need(bn + ".weight", &g));
    MRD_TRY(t.need(bn + ".bias", &b));
    MRD_TRY(t.need(bn + ".running_mean", &mu));
    MRD_TRY(t.need(bn + ".running_var", &var));
    out->cout = static_cast<int>(w->d[0]);
    out->cin = static_cast<int>(w->d[1]);
    out->k = static_cast<int>(w->d[2]);
    out->stride = stride;
    if (w->d[2] != w->d[3] || g->numel() != out->cout) {
        set_last_error("load_weights: bad conv/bn shapes at %s", conv.c_str());
        return -2;
    }
    MRD_TRY(walloc(c, &out->w, w->numel()));
    MRD_TRY(walloc(c, &out->b, out->cout));
    return pack_conv_bn(w->p, g->p, b->p, mu->p, var->p, c->bn_eps, out->cout, out->cin, out->k,
                        out->w, out->b, s);
}

int load_linear(mrd_ctx* c, const Table& t, const std::string& name, LinearW* out, cudaStream_t s) {
    const Tensor *w, *b;
    MRD_TRY(t.need(name + ".weight", &w));
    MRD_TRY(t.need(name + ".bias", &b));
    out->out = static_cast<int>(w->d[0]);
    out->in = static_cast<int>(w->d[1]);
    MRD_TRY(walloc(c, &out->w, w->numel()));
    MRD_TRY(walloc(c, &out->b, out->out));
    return pack_linear(w->p, b->p, out->out, out->in, 1.0f, out->w, out->b, s);
}

int load_vec(mrd_ctx* c, const Table& t, const std::string& name, float** out, cudaStream_t s) {
    const Tensor* v;
    MRD_TRY(t.need(name, &v));
    MRD_TRY(walloc(c, out, v->numel()));
    cudaError_t e = cudaMemcpyAsync(*out, v->p, static_cast<size_t>(v->numel()) * sizeof(float),
                                    cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(weight vector)");
    return 0;
}

int load_cnn_projection(mrd_ctx* c, const Table& t, cudaStream_t s) {
    MRD_TRY(load_linear(c, t, "cnn_encoder.projection.0", &c->proj1, s));
    MRD_TRY(load_linear(c, t, "cnn_encoder.projection.3", &c->proj2, s));
    c->img_emb_dim = c->proj2.out;
    c->has_proj = true;
    c->has_cnn = c->has_backbone && c->has_proj;
    return 0;
}

int load_cnn(mrd_ctx* c, const Table& t, cudaStream_t s) {
    const std::string bb = "cnn_encoder.backbone.";
    {
        const Tensor *w, *g, *b, *mu, *var;
        MRD_TRY(t.need(bb + "conv1.weight", &w));
        MRD_TRY(t.need(bb + "bn1.weight", &g));
        MRD_TRY(t.need(bb + "bn1.bias", &b));
        MRD_TRY(t.need(bb + "bn1.running_mean", &mu));
        MRD_TRY(t.need(bb + "bn1.running_var", &var));
        if (w->d[0] != 64 || w->d[1] != 3 || w->d[2] != 7 || w->d[3] != 7) {
            set_last_error("load_weights: stem must be Conv2d(3,64,7) (ResNet50 backbone only)");
            return -2;
        }
        MRD_TRY(walloc(c, &c->stem_w, 64 * 7 * 32));
        MRD_TRY(walloc(c, &c->stem_b, 64));
        MRD_TRY(pack_stem_bn(w->p, g->p, b->p, mu->p, var->p, c->bn_eps, c->stem_w, c->stem_b, s));
    }
    // stages are discovered from the names: layer{L}.{i}.conv{1,2,3}, stride on conv2 + downsample
    // of the first block of layers 2..4 (ResNet v1.5, TV:models/resnet.py:109-113)
    size_t bi = 0;
    for (int L = 1; L <= 4; ++L) {
        for (int i = 0;; ++i) {
            char pre[96];
            snprintf(pre, sizeof(pre), "%slayer%d.%d.", bb.c_str(), L, i);
            const std::string p(pre);
            if (!t.find(p + "conv1.weight")) break;
            if (c->blocks.size() <= bi) c->blocks.emplace_back();
            if (c->block_stage.size() <= bi) c->block_stage.push_back(L);
            c->block_stage[bi] = L;
            Bottleneck& b = c->blocks[bi++];
            const int stride = (i == 0 && L > 1) ? 2 : 1;
            MRD_TRY(load_conv_bn(c, t, p + "conv1", p + "bn1", 1, &b.c1, s));
            MRD_TRY(load_conv_bn(c, t, p + "conv2", p + "bn2", stride, &b.c2, s));
            MRD_TRY(load_conv_bn(c, t, p + "conv3", p + "bn3", 1, &b.c3, s));
            b.has_ds = t.find(p + "downsample.0.weight") != nullptr;
            if (b.has_ds) {
                MRD_TRY(load_conv_bn(c, t, p + "downsample.0", p + "downsample.1", stride, &b.ds, s));
                if (b.ds.k == 1 && b.c3.k == 1 && b.ds.cout == b.c3.cout) {
                    MRD_TRY(walloc(c, &b.c3ds_w, 1LL * b.c3.cout * (b.c3.cin + b.ds.cin)));
                    MRD_TRY(walloc(c, &b.c3ds_b, b.c3.cout));
                    MRD_TRY(pack_concat_k(b.c3.w, b.c3.cin, b.ds.w, b.ds.cin, b.c3.b, b.ds.b, b.c3.cout,
                                          b.c3ds_w, b.c3ds_b, s));
                }
            }
        }
    }
    if (bi == 0) {
        set_last_error("load_weights: no cnn_encoder.backbone.layer*.conv1.weight tensors");
        return -2;
    }
    c->blocks.resize(bi);
    c->feat_dim = c->blocks.back().c3.cout;
    c->has_backbone = true;
    c->has_cnn = c->has_backbone && c->has_proj;
    return 0;
}

int load_text(mrd_ctx* c, const Table& t, cudaStream_t s) {
    const std::string e = "text_encoder.encoder.embeddings.";
    const Tensor *we, *pe, *te;
    MRD_TRY(t.need(e + "word_embeddings.weight", &we));
    MRD_TRY(t.need(e + "position_embeddings.weight", &pe));
    MRD_TRY(t.need(e + "token_type_embeddings.weight", &te));
    c->vocab = static_cast<int>(we->d[0]);
    c->hidden = static_cast<int>(we->d[1]);
    c->max_pos = static_cast<int>(pe->d[0]);
    if (c->hidden != 768 || c->bert_heads * 64 != c->hidden) {
        set_last_error("load_weights: text encoder must be BERT-base shaped (hidden 768, 12x64 heads)");
        return -2;
    }
    MRD_TRY(walloc(c, &c->word_emb, we->numel()));
    MRD_TRY(pack_linear(we->p, nullptr, c->vocab, c->hidden, 1.0f, c->word_emb, nullptr, s));
    MRD_TRY(walloc(c, &c->pos_type, pe->numel()));
    MRD_TRY(pack_pos_type(pe->p, te->p, c->max_pos, c->hidden, c->pos_type, s));
    MRD_TRY(load_vec(c, t, e + "LayerNorm.weight", &c->emb_g, s));
    MRD_TRY(load_vec(c, t, e + "LayerNorm.bias", &c->emb_b, s));
    size_t li = 0;
    for (int i = 0;; ++i) {
        char pre[96];
        snprintf(pre, sizeof(pre), "text_encoder.encoder.encoder.layer.%d.", i);
        const std::string p(pre);
        const Tensor *wq, *wk, *wv, *bq, *bk, *bv;
        if (!t.find(p + "attention.self.query.weight")) break;
        if (c->layers.size() <= li) c->layers.emplace_back();
        BertLayerW& L = c->layers[li++];
        MRD_TRY(t.need(p + "attention.self.query.weight", &wq));
        MRD_TRY(t.need(p + "attention.self.key.weight", &wk));
        MRD_TRY(t.need(p + "attention.self.value.weight", &wv));
        MRD_TRY(t.need(p + "attention.self.query.bias", &bq));
        MRD_TRY(t.need(p + "attention.self.key.bias", &bk));
        MRD_TRY(t.need(p + "attention.self.value.bias", &bv));
        const int Hd = c->hidden;
        L.qkv.in = Hd;
        L.qkv.out = 3 * Hd;
        MRD_TRY(walloc(c, &L.qkv.w, 3LL * Hd * Hd));
        MRD_TRY(walloc(c, &L.qkv.b, 3LL * Hd));
        // softmax scale 1/sqrt(64) = 0.125 folded into the query projection (exact in bf16)
        MRD_TRY(pack_linear(wq->p, bq->p, Hd, Hd, 0.125f, L.qkv.w, L.qkv.b, s));
        MRD_TRY(pack_linear(wk->p, bk->p, Hd, Hd, 1.0f, L.qkv.w + 1LL * Hd * Hd, L.qkv.b + Hd, s));
        MRD_TRY(pack_linear(wv->p, bv->p, Hd, Hd, 1.0f, L.qkv.w + 2LL * Hd * Hd, L.qkv.b + 2 * Hd, s));
        MRD_TRY(load_linear(c, t, p + "attention.output.dense", &L.o, s));
        MRD_TRY(load_vec(c, t, p + "attention.output.LayerNorm.weight", &L.ln1g, s));
        MRD_TRY(load_vec(c, t, p + "attention.output.LayerNorm.bias", &L.ln1b, s));
        MRD_TRY(load_linear(c, t, p + "intermediate.dense", &L.f1, s));
        MRD_TRY(load_linear(c, t, p + "output.dense", &L.f2, s));
        MRD_TRY(load_vec(c, t, p + "output.LayerNorm.weight", &L.ln2g, s));
        MRD_TRY(load_vec(c, t, p + "output.LayerNorm.bias", &L.ln2b, s));
        c->ffn = L.f1.out;
    }
    if (li == 0) {
        set_last_error("load_weights: no text_encoder.encoder.encoder.layer.* tensors");
        return -2;
    }
    c->layers.resize(li);
    c->has_text = true;
    return 0;
}

int load_cross(mrd_ctx* c, const Table& t, const std::string& p, LinearW* out, cudaStream_t s) {
    const Tensor *wv, *bv, *wo, *bo;
    MRD_TRY(t.need(p + "value_proj.weight", &wv));
    MRD_TRY(t.need(p + "value_proj.bias", &bv));
    MRD_TRY(t.need(p + "output_proj.weight", &wo));
    MRD_TRY(t.need(p + "output_proj.bias", &bo));
    const int D = static_cast<int>(wo->d[0]);
    if (wo->d[1] != D || wv->d[0] != D || wv->d[1] != D) {
        set_last_error("load_weights: cross attention projections must be square (%s)", p.c_str());
        return -2;
    }
    out->in = D;
    out->out = D;
    MRD_TRY(walloc(c, &out->w, 1LL * D * D));
    MRD_TRY(walloc(c, &out->b, D));
    return pack_premul_linear(wo->p, bo->p, wv->p, bv->p, D, out->w, out->b, s);
}

int load_fusion(mrd_ctx* c, const Table& t, cudaStream_t s) {
    const std::string f = "fusion.fusion_layer.";
    MRD_TRY(load_linear(c, t, f + "image_proj", &c->f_ip, s));
    MRD_TRY(load_linear(c, t, f + "text_proj", &c->f_tp, s));
    MRD_TRY(load_cross(c, t, f + "image_to_text_attention.", &c->f_i2t, s));
    MRD_TRY(load_cross(c, t, f + "text_to_image_attention.", &c->f_t2i, s));
    MRD_TRY(load_vec(c, t, f + "layer_norm_image.weight", &c->ln_i_g, s));
    MRD_TRY(load_vec(c, t, f + "layer_norm_image.bias", &c->ln_i_b, s));
    MRD_TRY(load_vec(c, t, f + "layer_norm_text.weight", &c->ln_t_g, s));
    MRD_TRY(load_vec(c, t, f + "layer_norm_text.bias", &c->ln_t_b, s));
    MRD_TRY(load_linear(c, t, f + "fusion.0", &c->f_1, s));
    MRD_TRY(load_linear(c, t, f + "fusion.3", &c->f_2, s));
    c->fusion_dim = c->f_ip.out;
    c->fusion_img_in = c->f_ip.in;
    c->fusion_txt_in = c->f_tp.in;
    if (c->fusion_dim != 256 && c->fusion_dim != 512) {
        set_last_error("load_weights: fusion hidden_dim %d unsupported (256 or 512)", c->fusion_dim);
        return -2;
    }
    {
        // operands of the fused tail (tail_fused.h): K-concatenated pre-LayerNorm weights from the raw parameters
        const Tensor *wip, *bip, *wtp, *btp;
        MRD_TRY(t.need(f + "image_proj.weight", &wip));
        MRD_TRY(t.need(f + "image_proj.bias", &bip));
        MRD_TRY(t.need(f + "text_proj.weight", &wtp));
        MRD_TRY(t.need(f + "text_proj.bias", &btp));
        CrossRaw cr[2];
        const char* names[2] = {"image_to_text_attention.", "text_to_image_attention."};
        for (int i = 0; i < 2; ++i) {
            const Tensor *wv, *bv, *wo, *bo;
            MRD_TRY(t.need(f + names[i] + "value_proj.weight", &wv));
            MRD_TRY(t.need(f + names[i] + "value_proj.bias", &bv));
            MRD_TRY(t.need(f + names[i] + "output_proj.weight", &wo));
            MRD_TRY(t.need(f + names[i] + "output_proj.bias", &bo));
            cr[i] = CrossRaw{wv->p, bv->p, wo->p, bo->p};
        }
        const int F = c->fusion_dim, Ii = c->fusion_img_in, Ti = c->fusion_txt_in;
        MRD_TRY(walloc(c, &c->tail_wbig, 2LL * F * (Ii + Ti)));
        MRD_TRY(walloc(c, &c->tail_bbig, 2LL * F));
        MRD_TRY(walloc(c, &c->tail_scratch, 2LL * F * F + 2LL * F));
        MRD_TRY(pack_tail_big(wip->p, bip->p, wtp->p, btp->p, cr[0], cr[1], F, Ii, Ti, c->fusion_residual,
                              c->tail_scratch, c->tail_wbig, c->tail_bbig, s));
        c->tail_residual = c->fusion_residual;
    }
    c->has_fusion = true;
    return 0;
}

int load_head(mrd_ctx* c, const Table& t, cudaStream_t s) {
    // classifier.classifier.{0,3,6,...}: Linear every third slot (Linear, act, Dropout)*, Linear
    std::vector<int> idx;
    for (int i = 0; i < 64; i += 3) {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%d.weight", i);
        if (!t.find(nm)) break;
        idx.push_back(i);
    }
    if (idx.empty()) {
        set_last_error("load_weights: no classifier.classifier.*.weight tensors");
        return -2;
    }
    if (c->head_hidden.size() < idx.size() - 1) c->head_hidden.resize(idx.size() - 1);
    for (size_t j = 0; j + 1 < idx.size(); ++j) {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%d", idx[j]);
        MRD_TRY(load_linear(c, t, nm, &c->head_hidden[j], s));
    }
    c->head_hidden.resize(idx.size() - 1);
    char nm[64];
    snprintf(nm, sizeof(nm), "classifier.classifier.%d", idx.back());
    const Tensor *w, *b;
    MRD_TRY(t.need(std::string(nm) + ".weight", &w));
    MRD_TRY(t.need(std::string(nm) + ".bias", &b));
    c->num_classes = static_cast<int>(w->d[0]);
    c->head_last = static_cast<int>(w->d[1]);
    MRD_TRY(load_vec(c, t, std::string(nm) + ".weight", &c->head_out_w, s));
    MRD_TRY(load_vec(c, t, std::string(nm) + ".bias", &c->head_out_b, s));
    c->head_in = c->head_hidden.empty() ? c->head_last : c->head_hidden[0].in;
    if (c->num_classes > 32 || c->head_last % 32 != 0 || c->head_last > 1024) {
        set_last_error("load_weights: head output layer %dx%d unsupported", c->num_classes,
                       c->head_last);
        return -2;
    }
    c->has_head = true;
    return 0;
}

// ------------------------------------------------------------------ workspaces and plans
// 3x3 stride-1 convolutions on mid-sized feature maps run in flat-shift mode (plan_conv3x3_flat): the
// tile is th = 128/(w+2) whole padded rows, so the M efficiency is th*w/128; below ~20 columns the
// classic per-tap boxes (which can pack several rows/images per tile) win.
inline bool flat3_eligible(const ConvW& cv, int h, int w) {
    return cv.k == 3 && cv.stride == 1 && w >= 20 && conv3x3_flat_supported(h, w, cv.cin, cv.cout);
}

// Activation workspace of the ResNet passes, sized for the images one pass really holds: min(img_chunk, batch rounded
// up to a power of two), grown when a larger batch arrives (10.5 MB per 224 x 224 image).
int ensure_cnn_ws(mrd_ctx* c, int B, int H, int W) {
    int want = 16;
    while (want < B && want < c->img_chunk) want *= 2;
    if (want > c->img_chunk) want = c->img_chunk;
    const bool same_hw = c->cnn_ws.base && c->cnn_ws_H == H && c->cnn_ws_W == W;
    if (same_hw && c->cnn_ws_B >= want) return 0;
    const int Bc = (same_hw && c->cnn_ws_B > want) ? c->cnn_ws_B : want;
    c->cnn_plans.clear();
    c->pads.clear();
    ++c->cnn_ws_epoch;
    {
        int h = H / 4, w = W / 4;
        for (const Bottleneck& b : c->blocks) {
            if (flat3_eligible(b.c2, h, w)) {
                bool have = false;
                for (auto& pb : c->pads) have |= (pb.h == h && pb.w == w && pb.c == b.c2.cin);
                if (!have) {
                    mrd_ctx::PadBuf pb;
                    pb.h = h; pb.w = w; pb.c = b.c2.cin;
                    c->pads.push_back(pb);
                }
            }
            h /= b.c2.stride;
            w /= b.c2.stride;
        }
    }
    const long long q = 1LL * (H / 4) * (W / 4);  // pixels after stem + maxpool
    const long long n_xpad = 1LL * Bc * (H + 6) * (W + 8) * 4;
    const long long n_stem = 1LL * Bc * (H / 2) * (W / 2) * 64;
    const long long n_act = 1LL * Bc * q * 256;   // largest block output (layer1)
    const long long n_mid = 1LL * Bc * q * 128;   // largest bottleneck intermediate (layer2.0.conv1)
    size_t total = pad1k(n_xpad, 2) + pad1k(n_stem, 2) + 3 * pad1k(n_act, 2) + 2 * pad1k(n_mid, 2);
    size_t pad_bytes = 0;
    for (auto& pb : c->pads) pad_bytes += pad1k(1LL * Bc * (pb.h + 2) * (pb.w + 2) * pb.c, 2);
    total += pad_bytes;
    MRD_TRY(arena_reset(c, &c->cnn_ws, total));
    c->xpad = arena_take<bf16>(&c->cnn_ws, n_xpad);
    c->stem_out = arena_take<bf16>(&c->cnn_ws, n_stem);
    c->act0 = arena_take<bf16>(&c->cnn_ws, n_act);
    c->act1 = arena_take<bf16>(&c->cnn_ws, n_act);
    c->dsb = arena_take<bf16>(&c->cnn_ws, n_act);
    c->mid0 = arena_take<bf16>(&c->cnn_ws, n_mid);
    c->mid1 = arena_take<bf16>(&c->cnn_ws, n_mid);
    if (!c->pads.empty()) {
        bf16* first = nullptr;
        for (auto& pb : c->pads) {
            pb.p = arena_take<bf16>(&c->cnn_ws, 1LL * Bc * (pb.h + 2) * (pb.w + 2) * pb.c);
            if (!first) first = pb.p;
        }
        // borders must be (and stay) zero: the producing 1x1 convolution only writes the interior
        cudaError_t e = cudaMemset(first, 0, pad_bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemset(padded conv inputs)");
    }
    c->cnn_ws_B = Bc;
    c->cnn_ws_H = H;
    c->cnn_ws_W = W;
    return 0;
}

int get_cnn_plan(mrd_ctx* c, int B, int H, int W, CnnPlan** out) {
    auto key = std::make_pair(B, std::make_pair(H, W));
    auto it = c->cnn_plans.find(key);
    if (it != c->cnn_plans.end()) {
        *out = &it->second;
        return 0;
    }
    CnnPlan p;
    p.B = B; p.H = H; p.W = W;
    // stem + BN + ReLU + maxpool in one launch: the pooled map goes straight to act0
    MRD_TRY(plan_stem_pool(&p.stem, c->xpad, B, H, W, c->stem_w, c->stem_b, c->act0));
    int h = H / 4, w = W / 4;
    const bf16* x = c->act0;  // maxpool output goes to act0
    bf16* bufs[2] = {c->act0, c->act1};
    int cur = 0;
    p.blocks.resize(c->blocks.size());
    for (size_t i = 0; i < c->blocks.size(); ++i) {
        const Bottleneck& b = c->blocks[i];
        CnnPlan::BlockPlan& bp = p.blocks[i];
        const int ho = h / b.c2.stride, wo = w / b.c2.stride;
        if (h % b.c2.stride || w % b.c2.stride) {
            set_last_error("cnn plan: feature map %dx%d not divisible by stride at block %zu", h, w, i);
            return -1;
        }
        bf16* y = bufs[cur ^ 1];
        bf16* pad = nullptr;
        if (flat3_eligible(b.c2, h, w))
            for (auto& pb : c->pads)
                if (pb.h == h && pb.w == w && pb.c == b.c2.cin) pad = pb.p;
        if (pad) {
            // conv1 writes the interior of the zero-bordered buffer; conv2 reads it in flat-shift mode
            MRD_TRY(plan_conv(&bp.c1, x, B, h, w, b.c1.cin, b.c1.w, b.c1.cout, b.c1.k, 1, b.c1.b, pad,
                              nullptr, ACT_RELU, 1));
            MRD_TRY(plan_conv3x3_flat(&bp.c2, pad, B, h, w, b.c2.cin, b.c2.w, b.c2.cout, b.c2.b,
                                      c->mid1, ACT_RELU));
        } else {
            MRD_TRY(plan_conv(&bp.c1, x, B, h, w, b.c1.cin, b.c1.w, b.c1.cout, b.c1.k, 1, b.c1.b,
                              c->mid0, nullptr, ACT_RELU));
            MRD_TRY(plan_conv(&bp.c2, c->mid0, B, h, w, b.c2.cin, b.c2.w, b.c2.cout, b.c2.k,
                              b.c2.stride, b.c2.b, c->mid1, nullptr, ACT_RELU));
        }
        const bf16* identity = x;
        bp.has_ds = b.has_ds;
        bp.fused_ds = false;
        if (b.has_ds && b.c3ds_w) {
            // conv3 + downsample + add in one accumulator: the downsample output is never written or re-read
            MRD_TRY(plan_conv1x1_dual(&bp.c3, c->mid1, b.c3.cin, x, b.ds.cin, b.ds.stride, B, ho, wo, b.c3ds_w,
                                      b.c3.cout, b.c3ds_b, y, ACT_RELU));
            bp.fused_ds = true;
        } else {
            if (b.has_ds) {
                MRD_TRY(plan_conv(&bp.ds, x, B, h, w, b.ds.cin, b.ds.w, b.ds.cout, b.ds.k, b.ds.stride,
                                  b.ds.b, c->dsb, nullptr, ACT_NONE));
                identity = c->dsb;
            }
            MRD_TRY(plan_conv(&bp.c3, c->mid1, B, ho, wo, b.c3.cin, b.c3.w, b.c3.cout, b.c3.k, 1,
                              b.c3.b, y, identity, ACT_RELU));
        }
        // ---- chain this block's tail with the next block's conv1 (same pixels, one launch, y re-read from L2).
        // Layer1 only: for layers 2-4 the weights no longer stay resident and the chain measured slower than the two
        // launches it replaces (DESIGN.md section 10).
        if (i + 1 < c->blocks.size() && c->block_stage[i] == 1) {
            const Bottleneck& nx = c->blocks[i + 1];
            const bool dual = b.has_ds && b.c3ds_w != nullptr;
            const bool ok = b.c3.k == 1 && nx.c1.k == 1 && nx.c1.stride == 1 && nx.c1.cin == b.c3.cout &&
                            (!b.has_ds || dual) &&
                            conv_chain_supported(b.c3.cin, dual ? b.ds.cin : 0, b.c3.cout, nx.c1.cout);
            if (ok) {
                bf16* npad = nullptr;   // the next block's conv1 writes into its flat-3x3 input when it has one
                if (flat3_eligible(nx.c2, ho, wo))
                    for (auto& pb : c->pads)
                        if (pb.h == ho && pb.w == wo && pb.c == nx.c2.cin) npad = pb.p;
                MRD_TRY(plan_conv_chain(&bp.chain, c->mid1, b.c3.cin, dual ? x : nullptr, dual ? b.ds.cin : 0,
                                        b.ds.stride, dual ? nullptr : x, B, ho, wo, dual ? b.c3ds_w : b.c3.w,
                                        b.c3.cout, dual ? b.c3ds_b : b.c3.b, y, nx.c1.w, nx.c1.cout, nx.c1.b,
                                        npad ? npad : c->mid0, npad ? 1 : 0));
                bp.chained = true;
                p.blocks[i + 1].c1_in_prev_chain = true;
            }
        }
        x = y;
        cur ^= 1;
        h = ho;
        w = wo;
    }
    p.final_act = x;
    p.final_hw = h * w;
    auto ins = c->cnn_plans.emplace(key, std::move(p));
    *out = &ins.first->second;
    return 0;
}

int ensure_text_ws(mrd_ctx* c, int tokens, int seqs) {
    if (c->text_ws.base && c->text_ws_tokens >= tokens && c->text_ws_seqs >= seqs) return 0;
    c->text_plans.clear();
    ++c->text_ws_epoch;
    if (tokens < c->text_ws_tokens) tokens = c->text_ws_tokens;
    if (seqs < c->text_ws_seqs) seqs = c->text_ws_seqs;
    c->text_ws_seqs = seqs;
    const long long T = tokens;
    const int Hd = c->hidden;
    const long long Sq = c->text_ws_seqs;  // most sequences one pass can hold
    size_t total = 4 * pad1k(T * Hd, 2) + pad1k(T * 3 * Hd, 2) + pad1k(T * c->ffn, 2) +
                   4 * pad1k(T + 2, 4) + pad1k(1, 4) + 4 * pad1k(Sq * Hd, 2) + pad1k(Sq * c->ffn, 2) +
                   pad1k(static_cast<long long>(gemm_ln_ws_bytes(tokens)), 1);
    MRD_TRY(arena_reset(c, &c->text_ws, total));
    c->t_h = arena_take<bf16>(&c->text_ws, T * Hd);
    c->t_h2 = arena_take<bf16>(&c->text_ws, T * Hd);
    c->t_ctx = arena_take<bf16>(&c->text_ws, T * Hd);
    c->t_tmp = arena_take<bf16>(&c->text_ws, T * Hd);
    c->t_qkv = arena_take<bf16>(&c->text_ws, T * 3 * Hd);
    c->t_ffn = arena_take<bf16>(&c->text_ws, T * c->ffn);
    c->t_cls_ctx = arena_take<bf16>(&c->text_ws, Sq * Hd);
    c->t_cls_h = arena_take<bf16>(&c->text_ws, Sq * Hd);
    c->t_cls_h2 = arena_take<bf16>(&c->text_ws, Sq * Hd);
    c->t_cls_tmp = arena_take<bf16>(&c->text_ws, Sq * Hd);
    c->t_cls_ffn = arena_take<bf16>(&c->text_ws, Sq * c->ffn);
    c->t_bias = arena_take<float>(&c->text_ws, T + 2);
    c->t_seq_off = arena_take<int>(&c->text_ws, T + 2);
    c->t_row_tok = arena_take<int>(&c->text_ws, T + 2);
    c->t_scratch = arena_take<int>(&c->text_ws, T + 2);
    c->t_nrows = arena_take<int>(&c->text_ws, 1);
    c->t_ln_ws = arena_take<char>(&c->text_ws, static_cast<long long>(gemm_ln_ws_bytes(tokens)));
    c->text_ws_tokens = tokens;
    // rows beyond the live token count are read (never used) by tile-granular kernels: keep every
    // byte of the workspace a finite number from the start
    cudaError_t e = cudaMemset(c->text_ws.base, 0, c->text_ws.bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemset(text workspace)");
    return 0;
}

int get_text_plan(mrd_ctx* c, int B, int S, TextPlan** out) {
    auto key = std::make_pair(B, S);
    auto it = c->text_plans.find(key);
    if (it != c->text_plans.end()) {
        *out = &it->second;
        return 0;
    }
    TextPlan p;
    p.B = B; p.S = S;
    const int T = B * S, Hd = c->hidden;
    p.blocked_qkv = attention_prefers_blocked_qkv(S) ? 1 : 0;
    p.layers.resize(c->layers.size());
    for (size_t i = 0; i < c->layers.size(); ++i) {
        const BertLayerW& L = c->layers[i];
        TextPlan::LayerPlan& lp = p.layers[i];
        MRD_TRY(plan_gemm(&lp.qkv, c->t_h, Hd, T, Hd, L.qkv.w, 3 * Hd, L.qkv.b, c->t_qkv, 3 * Hd,
                          nullptr, 0, nullptr, 0, ACT_NONE, p.blocked_qkv));
        MRD_TRY(plan_gemm(&lp.o, c->t_ctx, Hd, T, Hd, L.o.w, Hd, L.o.b, c->t_tmp, Hd, c->t_h, Hd,
                          nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&lp.f1, c->t_h2, Hd, T, Hd, L.f1.w, c->ffn, L.f1.b, c->t_ffn, c->ffn,
                          nullptr, 0, nullptr, 0, ACT_GELU));
        MRD_TRY(plan_gemm(&lp.f2, c->t_ffn, c->ffn, T, c->ffn, L.f2.w, Hd, L.f2.b, c->t_tmp, Hd,
                          c->t_h2, Hd, nullptr, 0, ACT_NONE));
        // rows are token-packed: the live count is produced on the device by compact_tokens
        lp.qkv.p.dyn_rows = lp.o.p.dyn_rows = lp.f1.p.dyn_rows = lp.f2.p.dyn_rows = c->t_nrows;
        // FFN2 + residual + LayerNorm as one launch (Hd/256 CTAs per 128-token stripe, statistics exchanged through
        // L2): the normalised rows go straight to the buffer the separate LayerNorm launch would have written.  The
        // attention output keeps its separate LayerNorm: its two-pass epilogue hides under FFN2's K = 3072 main loop
        // (-25 us per launch) but not under the K = 768 one (153 vs 140 us, DESIGN.md section 10).  Widths the
        // kernel does not cover (plan_gemm_ln returns 1) take the GEMM + layernorm_residual launches.
        int r2 = plan_gemm_ln(&lp.f2_ln, c->t_ffn, c->ffn, T, c->ffn, L.f2.w, Hd, L.f2.b, c->t_h, Hd, c->t_h2, Hd,
                              L.ln2g, L.ln2b, c->bert_ln_eps, c->t_ln_ws);
        if (r2 < 0) return r2;
        lp.f2_fused = r2 == 0;
        lp.f2_ln.p.dyn_rows = c->t_nrows;
    }
    {
        const BertLayerW& L = c->layers.back();
        MRD_TRY(plan_gemm(&p.o_cls, c->t_cls_ctx, Hd, B, Hd, L.o.w, Hd, L.o.b, c->t_cls_tmp, Hd,
                          c->t_cls_h, Hd, nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.f1_cls, c->t_cls_h2, Hd, B, Hd, L.f1.w, c->ffn, L.f1.b, c->t_cls_ffn,
                          c->ffn, nullptr, 0, nullptr, 0, ACT_GELU));
        MRD_TRY(plan_gemm(&p.f2_cls, c->t_cls_ffn, c->ffn, B, c->ffn, L.f2.w, Hd, L.f2.b,
                          c->t_cls_tmp, Hd, c->t_cls_h2, Hd, nullptr, 0, ACT_NONE));
        // output = this chunk's rows of b_txt: patched at run time (run_bert), planned on a placeholder
        int r = plan_gemm_ln(&p.f2_cls_ln, c->t_cls_ffn, c->ffn, B, c->ffn, L.f2.w, Hd, L.f2.b, c->t_cls_tmp, Hd,
                             c->t_cls_h2, Hd, L.ln2g, L.ln2b, c->bert_ln_eps, c->t_ln_ws);
        if (r < 0) return r;
        p.f2_cls_fused = r == 0;
    }
    auto ins = c->text_plans.emplace(key, std::move(p));
    *out = &ins.first->second;
    return 0;
}

int ensure_batch_ws(mrd_ctx* c, int B) {
    if (c->batch_ws.base && c->batch_ws_B >= B) return 0;
    c->batch_plans.clear();
    // round up so slowly growing batches do not reallocate every call
    int cap = 64;
    while (cap < B) cap *= 2;
    const long long n = cap;
    const long long wmax = 2048;  // widest row any batch-level buffer holds
    if (c->feat_dim > wmax) {
        set_last_error("backbone feature width %d unsupported", c->feat_dim);
        return -1;
    }
    size_t total = 14 * pad1k(n * wmax, 2) + pad1k(n * wmax, 4);
    MRD_TRY(arena_reset(c, &c->batch_ws, total));
    c->b_pooled = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_projh = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_img = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_txt = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_ip = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_tp = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_prei = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_pret = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_fh = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_fused = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_cat = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_h[0] = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_h[1] = arena_take<bf16>(&c->batch_ws, n * wmax);
    c->b_scratch_f32 = arena_take<float>(&c->batch_ws, n * wmax);
    c->batch_ws_B = cap;
    return 0;
}

int get_batch_plan(mrd_ctx* c, int B, BatchPlan** out) {
    auto it = c->batch_plans.find(B);
    if (it != c->batch_plans.end()) {
        *out = &it->second;
        return 0;
    }
    BatchPlan p;
    p.B = B;
    if (c->has_cnn) {
        if (c->proj1.out > 1024 || c->proj2.out > 1024) {
            set_last_error("batch plan: projection width > 1024 unsupported");
            return -1;
        }
        MRD_TRY(plan_gemm(&p.proj1, c->b_pooled, c->feat_dim, B, c->feat_dim, c->proj1.w,
                          c->proj1.out, c->proj1.b, c->b_projh, c->proj1.out, nullptr, 0, nullptr, 0,
                          ACT_RELU));
        MRD_TRY(plan_gemm(&p.proj2, c->b_projh, c->proj1.out, B, c->proj1.out, c->proj2.w,
                          c->proj2.out, c->proj2.b, c->b_img, c->proj2.out, nullptr, 0,
                          nullptr, 0, ACT_NONE));
        p.has_proj = true;
    }
    if (c->has_fusion) {
        const int F = c->fusion_dim;
        MRD_TRY(plan_gemm(&p.ip, c->b_img, c->fusion_img_in, B, c->fusion_img_in, c->f_ip.w, F,
                          c->f_ip.b, c->b_ip, F, nullptr, 0, nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.tp, c->b_txt, c->fusion_txt_in, B, c->fusion_txt_in, c->f_tp.w, F,
                          c->f_tp.b, c->b_tp, F, nullptr, 0, nullptr, 0, ACT_NONE));
        // image attends to text: attended = O(V(text_proj)); + image_proj residual
        const bf16* res_i = c->fusion_residual ? c->b_ip : nullptr;
        const bf16* res_t = c->fusion_residual ? c->b_tp : nullptr;
        MRD_TRY(plan_gemm(&p.i2t, c->b_tp, F, B, F, c->f_i2t.w, F, c->f_i2t.b, c->b_prei, F, res_i, F,
                          nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.t2i, c->b_ip, F, B, F, c->f_t2i.w, F, c->f_t2i.b, c->b_pret, F, res_t, F,
                          nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.f1, c->b_cat, 2 * F, B, 2 * F, c->f_1.w, F, c->f_1.b, c->b_fh, F,
                          nullptr, 0, nullptr, 0, ACT_RELU));
        MRD_TRY(plan_gemm(&p.f2, c->b_fh, F, B, F, c->f_2.w, F, c->f_2.b, c->b_fused, F, nullptr, 0,
                          nullptr, 0, ACT_NONE));
        p.has_fusion = true;
    }
    if (c->has_head) {
        const bf16* x = c->b_fused;
        int ld = c->head_in;
        p.head.resize(c->head_hidden.size());
        for (size_t j = 0; j < c->head_hidden.size(); ++j) {
            const LinearW& L = c->head_hidden[j];
            if (L.out > 1024 || L.in != ld) {
                set_last_error("batch plan: head layer %zu has unsupported shape %dx%d", j, L.out,
                               L.in);
                return -1;
            }
            bf16* y = c->b_h[j & 1];
            MRD_TRY(plan_gemm(&p.head[j], x, ld, B, L.in, L.w, L.out, L.b, y, L.out, nullptr, 0,
                              nullptr, 0, c->head_act));
            x = y;
            ld = L.out;
        }
        p.has_head = true;
    }
    if (c->has_fusion && c->has_head && c->tail_residual == c->fusion_residual &&
        c->fusion_dim == c->head_in && !c->head_hidden.empty() &&
        c->head_hidden.size() <= 3) {
        TailWeights w = {};
        w.w_big = c->tail_wbig; w.b_big = c->tail_bbig;
        w.ln_i_g = c->ln_i_g; w.ln_i_b = c->ln_i_b; w.ln_t_g = c->ln_t_g; w.ln_t_b = c->ln_t_b;
        w.w1 = c->f_1.w; w.b1 = c->f_1.b; w.w2 = c->f_2.w; w.b2 = c->f_2.b;
        w.num_hidden = static_cast<int>(c->head_hidden.size());
        for (int j = 0; j < w.num_hidden; ++j) {
            w.wh[j] = c->head_hidden[j].w;
            w.bh[j] = c->head_hidden[j].b;
            w.hdim[j] = c->head_hidden[j].out;
        }
        w.head_act = c->head_act;
        w.out_w = c->head_out_w; w.out_b = c->head_out_b;
        w.F = c->fusion_dim; w.img_in = c->fusion_img_in; w.txt_in = c->fusion_txt_in; w.C = c->num_classes;
        w.ln_eps = c->fusion_ln_eps;
        bool chain = c->f_1.in == 2 * w.F && c->f_1.out == w.F && c->f_2.in == w.F && c->f_2.out == w.F;
        int in_dim = w.F;
        for (int j = 0; j < w.num_hidden; ++j) {
            chain = chain && c->head_hidden[j].in == in_dim;
            in_dim = w.hdim[j];
        }
        chain = chain && in_dim == c->head_last;
        if (chain && tail_supported(w.F, w.img_in, w.txt_in, w.num_hidden, w.hdim, w.C)) {
            MRD_TRY(plan_tail(&p.tail, w, c->b_img, c->b_txt, B));
            p.has_tail = true;
        }
    }
    auto ins = c->batch_plans.emplace(B, std::move(p));
    *out = &ins.first->second;
    return 0;
}

// ------------------------------------------------------------------ launch accounting / profiling
// Every kernel launch of a forward goes through one ProfScope: it counts the launch and, when the
// context is in profile mode (mrd_ctx_profile), brackets it with CUDA events on the launching stream
// so bench.py can attribute device time, algorithmic FLOPs and bytes to each kernel family.
enum Cat : int { CAT_TENSOR = 0, CAT_ATTN = 1, CAT_MEM = 2 };

struct ProfScope {
    mrd_ctx* c;
    cudaStream_t s;
    ProfRecord r;
    ProfScope(mrd_ctx* c_, cudaStream_t s_, const char* label, int cat, double flops, double bytes)
        : c(c_), s(s_) {
        ++c->launches;
        if (!c->profiling) return;
        r.label = label;
        r.cat = cat;
        r.flops = flops;
        r.bytes = bytes;
        cudaEventCreate(&r.e0);
        cudaEventCreate(&r.e1);
        cudaEventRecord(r.e0, s);
    }
    ~ProfScope() {
        if (!c->profiling) return;
        cudaEventRecord(r.e1, s);
        c->prof.push_back(r);
    }
};

inline int run(mrd_ctx* c, const char* label, const GemmLaunch& g, cudaStream_t s) {
    ProfScope ps(c, s, label, CAT_TENSOR, g.flops, g.bytes);
    return launch_gemm(&g, s);
}
inline int run_f32(mrd_ctx* c, const char* label, const GemmLaunch& g, float* out_f32, long long ld,
                   cudaStream_t s) {
    GemmLaunch t = g;
    t.p.out_f32 = out_f32;
    t.p.ld_f32 = ld;
    ProfScope ps(c, s, label, CAT_TENSOR, g.flops, g.bytes);
    return launch_gemm(&t, s);
}

// ------------------------------------------------------------------ input checks
// images of every backbone forward (eval, batch-statistics BatchNorm, saving forward for data gradients)
int check_images(int img_dtype, int H, int W) {
    if (img_dtype != MRD_DT_F32 && img_dtype != MRD_DT_BF16) {
        set_last_error("images must be f32 or bf16 (dtype code %d)", img_dtype);
        return -1;
    }
    if (H % 32 != 0 || W % 32 != 0 || H <= 0 || W <= 0) {
        set_last_error("image size %dx%d unsupported: H and W must be multiples of 32", H, W);
        return -1;
    }
    return 0;
}

int fp32_images_only(int img_dtype) {
    if (img_dtype != MRD_DT_F32) {
        set_last_error("fp32 check mode takes fp32 images (dtype code %d given)", img_dtype);
        return -1;
    }
    return 0;
}

// the attention mask is optional; when given, its dtype code must be one the token compaction reads
int check_mask_dtype(const void* mask, int mask_dtype) {
    if (mask && (mask_dtype < MRD_DT_I64 || mask_dtype > MRD_DT_BF16)) {
        set_last_error("unknown mask dtype code %d", mask_dtype);
        return -1;
    }
    return 0;
}

// ------------------------------------------------------------------ stage runners
// ResNet50 backbone over the whole batch in micro-batches; leaves pooled features in b_pooled.
int run_backbone(mrd_ctx* c, const void* images, int img_dtype, int B, int H, int W,
                 float* feat_pooled, float* feat_map, cudaStream_t s) {
    if (!c->has_cnn) {
        set_last_error("cnn_encoder weights are not loaded in this context");
        return -3;
    }
    MRD_TRY(check_images(img_dtype, H, W));
    MRD_TRY(ensure_cnn_ws(c, B, H, W));
    const size_t esz = img_dtype == MRD_DT_BF16 ? 2 : 4;
    static const char* const kStage[5] = {"", "layer1", "layer2", "layer3", "layer4"};
    for (int b0 = 0; b0 < B; b0 += c->img_chunk) {
        const int nb = B - b0 < c->img_chunk ? B - b0 : c->img_chunk;
        CnnPlan* p;
        MRD_TRY(get_cnn_plan(c, nb, H, W, &p));
        const char* img = static_cast<const char*>(images) + static_cast<size_t>(b0) * 3 * H * W * esz;
        {
            ProfScope ps(c, s, "repack_images", CAT_MEM, 0,
                         1.0 * nb * (3.0 * H * W * esz + (H + 6.0) * (W + 8) * 8));
            MRD_TRY(repack_images(img, img_dtype == MRD_DT_BF16, nb, H, W, c->xpad, s));
        }
        {
            // the epilogue folds partial window maxima into act0 with red.global.max: start from zero (= the padding
            // value and the identity of the maximum of post-ReLU values)
            const size_t pooled_bytes = static_cast<size_t>(nb) * (H / 4) * (W / 4) * 64 * sizeof(bf16);
            ProfScope ps(c, s, "zero_pooled", CAT_MEM, 0, 1.0 * pooled_bytes);
            cudaError_t e = cudaMemsetAsync(c->act0, 0, pooled_bytes, s);
            if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(pooled stem output)");
        }
        MRD_TRY(run(c, "conv_stem7x7+maxpool", p->stem, s));
        for (size_t i = 0; i < p->blocks.size(); ++i) {
            auto& bp = p->blocks[i];
            const char* st = kStage[c->block_stage[i]];
            if (!bp.c1_in_prev_chain) MRD_TRY(run(c, c->label(st, ".conv1_1x1"), bp.c1, s));
            MRD_TRY(run(c, c->label(st, c->blocks[i].c2.stride == 2 ? ".conv2_3x3s2" : ".conv2_3x3"),
                        bp.c2, s));
            if (bp.chained) {
                ProfScope ps(c, s, c->label(st, bp.has_ds ? ".conv3+ds+next_conv1" : ".conv3+res+next_conv1"),
                             CAT_TENSOR, bp.chain.flops, bp.chain.bytes);
                MRD_TRY(launch_conv_chain(&bp.chain, s));
                continue;
            }
            if (bp.fused_ds) {
                MRD_TRY(run(c, c->label(st, ".conv3+downsample"), bp.c3, s));
                continue;
            }
            if (bp.has_ds) MRD_TRY(run(c, c->label(st, ".downsample"), bp.ds, s));
            MRD_TRY(run(c, c->label(st, ".conv3_1x1+res"), bp.c3, s));
        }
        {
            ProfScope ps(c, s, "global_avgpool", CAT_MEM, 0,
                         1.0 * nb * c->feat_dim * (p->final_hw * 2.0 + 2.0));
            MRD_TRY(global_avgpool(p->final_act, nb, p->final_hw, c->feat_dim,
                                   c->b_pooled + 1LL * b0 * c->feat_dim,
                                   feat_pooled ? feat_pooled + 1LL * b0 * c->feat_dim : nullptr, s));
        }
        if (feat_map) {
            ProfScope ps(c, s, "nhwc_to_nchw_f32", CAT_MEM, 0, 6.0 * nb * c->feat_dim * p->final_hw);
            MRD_TRY(nhwc_bf16_to_nchw_f32(p->final_act, nb, p->final_hw, c->feat_dim,
                                          feat_map + 1LL * b0 * c->feat_dim * p->final_hw, s));
        }
    }
    return 0;
}

int run_projection(mrd_ctx* c, BatchPlan* bp, float* emb_f32, cudaStream_t s) {
    MRD_TRY(run(c, "cnn_proj1", bp->proj1, s));
    MRD_TRY(run_f32(c, "cnn_proj2", bp->proj2, emb_f32, emb_f32 ? c->proj2.out : 0, s));
    return 0;
}

// BERT encoder over the whole batch in micro-batches; leaves CLS rows in b_txt (+ optional fp32).
// attn_probs (optional): f32 [layers,B,heads,S,S], every layer's attention probabilities.
int run_bert(mrd_ctx* c, const long long* ids, const void* mask, int mask_dtype, int B, int S,
             float* cls_f32, float* last_hidden, float* all_hidden, float* attn_probs, cudaStream_t s) {
    if (!c->has_text) {
        set_last_error("text_encoder weights are not loaded in this context");
        return -3;
    }
    if (S <= 0 || S > c->max_pos || S > 512) {
        set_last_error("sequence length %d unsupported (1..%d)", S, c->max_pos < 512 ? c->max_pos : 512);
        return -1;
    }
    ++c->text_run_epoch;
    int seqs = c->tok_chunk / S;
    if (seqs < 1) seqs = 1;
    if (seqs > B) seqs = B;
    MRD_TRY(ensure_text_ws(c, seqs * S, seqs));
    static const size_t msz[5] = {8, 4, 4, 1, 2};
    const int Hd = c->hidden;
    for (int b0 = 0; b0 < B; b0 += seqs) {
        const int nb = B - b0 < seqs ? B - b0 : seqs;
        const int T = nb * S;
        TextPlan* p;
        MRD_TRY(get_text_plan(c, nb, S, &p));
        const void* m = mask ? static_cast<const char*>(mask) + static_cast<size_t>(b0) * S * msz[mask_dtype]
                             : nullptr;
        // token packing: padded positions are dropped (they influence nothing TextEncoder.forward
        // returns); every later kernel reads the live row count from the device, so no host sync
        if (all_hidden && !last_hidden) {
            set_last_error("all_hidden requires last_hidden (both keep every token)");
            return -1;
        }
        // the probabilities are returned for every query row, padded ones included: they need every token too
        const int keep_all = last_hidden != nullptr || attn_probs != nullptr;
        // hidden_states[l] of HF BertModel: l = 0 is the embedding output, l = i+1 the output of layer i;
        // layout [L+1, B, S, Hd] fp32 (src/text_encoder.py:129-149)
        auto export_hidden = [&](size_t l) -> int {
            if (!all_hidden) return 0;
            ProfScope ps(c, s, "hidden_to_f32", CAT_MEM, 0, 6.0 * T * Hd);
            return cast_bf16_to_f32(c->t_h, Hd, T, Hd,
                                    all_hidden + (static_cast<long long>(l) * B + b0) * S * Hd, Hd, s);
        };
        {
            ProfScope ps(c, s, "compact_tokens", CAT_MEM, 0, 1.0 * T * (msz[mask_dtype] + 8));
            MRD_TRY(compact_tokens(m, mask_dtype, nb, S, keep_all, c->t_seq_off, c->t_row_tok,
                                   c->t_bias, c->t_nrows, c->t_scratch, s));
            c->launches += 2;
        }
        {
            ProfScope ps(c, s, "bert_embed_ln", CAT_MEM, 0, 1.0 * T * (8 + Hd * 2.0 * 2 + Hd * 4.0));
            MRD_TRY(bert_embed_layernorm(ids + 1LL * b0 * S, nb, S, c->word_emb, c->pos_type, c->emb_g,
                                         c->emb_b, c->bert_ln_eps, c->vocab, c->t_h, s, c->t_row_tok,
                                         c->t_nrows));
        }
        MRD_TRY(export_hidden(0));
        const double ln_bytes = 1.0 * T * Hd * 2 * 2;
        const double attn_flops = 4.0 * nb * c->bert_heads * S * 1.0 * S * 64;
        for (size_t i = 0; i < p->layers.size(); ++i) {
            const BertLayerW& L = c->layers[i];
            auto& lp = p->layers[i];
            MRD_TRY(run(c, "bert.qkv", lp.qkv, s));
            {
                ProfScope ps(c, s, "bert.attention", CAT_ATTN, attn_flops, 1.0 * T * Hd * 2 * 4);
                // blocked layout: block stride = the M the QKV plan was built with (T rows)
                MRD_TRY(attention_forward(c->t_qkv, c->t_bias, c->t_seq_off, nb, S, c->bert_heads,
                                          c->t_ctx, s, p->blocked_qkv ? T : c->text_ws_tokens,
                                          p->blocked_qkv));
            }
            if (attn_probs) {
                // keep_all: the packed layout is the dense one, t_bias is the [nb,S] key bias
                const int H = c->bert_heads;
                ProfScope ps(c, s, "bert.attn_probs", CAT_MEM, 0,
                             4.0 * nb * H * S * S + 2.0 * T * Hd * (1 + (S + 127) / 128));
                MRD_TRY(attention_probs(c->t_qkv, c->t_bias, nb, S, H,
                                        attn_probs + (static_cast<long long>(i) * B + b0) * H * S * S, s,
                                        p->blocked_qkv ? T : c->text_ws_tokens, p->blocked_qkv));
            }
            if (i + 1 == p->layers.size() && !last_hidden) {
                // ---- last layer: only the CLS row of each sequence is consumed downstream
                {
                    ProfScope ps(c, s, "gather_cls", CAT_MEM, 0, 8.0 * nb * Hd);
                    MRD_TRY(gather_cls_rows(c->t_ctx, c->t_seq_off, nb, Hd, c->t_cls_ctx, nullptr, s));
                    MRD_TRY(gather_cls_rows(c->t_h, c->t_seq_off, nb, Hd, c->t_cls_h, nullptr, s));
                    ++c->launches;
                }
                MRD_TRY(run(c, "bert.cls.attn_out+res", p->o_cls, s));
                {
                    ProfScope ps(c, s, "bert.cls.layernorm", CAT_MEM, 0, 4.0 * nb * Hd);
                    MRD_TRY(layernorm_residual(c->t_cls_tmp, Hd, nullptr, 0, L.ln1g, L.ln1b,
                                               c->bert_ln_eps, nb, Hd, c->t_cls_h2, Hd, nullptr, 0, s));
                }
                MRD_TRY(run(c, "bert.cls.ffn1+gelu", p->f1_cls, s));
                if (p->f2_cls_fused) {
                    MRD_TRY(run(c, "bert.cls.ffn2+res+ln", p->f2_cls_ln, s));
                    // the plan's output is a workspace row block: copy to this chunk's rows of the embedding buffer
                    ProfScope ps(c, s, "cls_copy", CAT_MEM, 0, 4.0 * nb * Hd);
                    cudaError_t e = cudaMemcpyAsync(c->b_txt + 1LL * b0 * Hd, c->t_cls_tmp, sizeof(bf16) * nb * Hd,
                                                    cudaMemcpyDeviceToDevice, s);
                    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(CLS rows)");
                } else {
                    MRD_TRY(run(c, "bert.cls.ffn2+res", p->f2_cls, s));
                    ProfScope ps(c, s, "bert.cls.layernorm", CAT_MEM, 0, 4.0 * nb * Hd);
                    MRD_TRY(layernorm_residual(c->t_cls_tmp, Hd, nullptr, 0, L.ln2g, L.ln2b,
                                               c->bert_ln_eps, nb, Hd, c->b_txt + 1LL * b0 * Hd, Hd,
                                               nullptr, 0, s));
                }
                if (cls_f32) {
                    ProfScope ps(c, s, "cls_to_f32", CAT_MEM, 0, 6.0 * nb * Hd);
                    MRD_TRY(cast_bf16_to_f32(c->b_txt + 1LL * b0 * Hd, Hd, nb, Hd,
                                             cls_f32 + 1LL * b0 * Hd, Hd, s));
                }
                break;
            }
            MRD_TRY(run(c, "bert.attn_out+res", lp.o, s));
            {
                ProfScope ps(c, s, "bert.layernorm", CAT_MEM, 0, ln_bytes);
                MRD_TRY(layernorm_residual(c->t_tmp, Hd, nullptr, 0, L.ln1g, L.ln1b, c->bert_ln_eps, T,
                                           Hd, c->t_h2, Hd, nullptr, 0, s, c->t_nrows));
            }
            MRD_TRY(run(c, "bert.ffn1+gelu", lp.f1, s));
            if (lp.f2_fused) {
                MRD_TRY(run(c, "bert.ffn2+res+ln", lp.f2_ln, s));
            } else {
                MRD_TRY(run(c, "bert.ffn2+res", lp.f2, s));
                ProfScope ps(c, s, "bert.layernorm", CAT_MEM, 0, ln_bytes);
                MRD_TRY(layernorm_residual(c->t_tmp, Hd, nullptr, 0, L.ln2g, L.ln2b, c->bert_ln_eps, T,
                                           Hd, c->t_h, Hd, nullptr, 0, s, c->t_nrows));
            }
            MRD_TRY(export_hidden(i + 1));
        }
        if (last_hidden) {
            // full last layer was computed: CLS rows (src/text_encoder.py:118) = first packed row of
            // every sequence
            ProfScope ps(c, s, "gather_cls", CAT_MEM, 0, 8.0 * nb * Hd);
            MRD_TRY(gather_cls_rows(c->t_h, c->t_seq_off, nb, Hd, c->b_txt + 1LL * b0 * Hd,
                                    cls_f32 ? cls_f32 + 1LL * b0 * Hd : nullptr, s));
        }
        if (last_hidden) {  // keep_all: packed layout == dense [nb,S,Hd]
            ProfScope ps(c, s, "hidden_to_f32", CAT_MEM, 0, 6.0 * T * Hd);
            MRD_TRY(cast_bf16_to_f32(c->t_h, Hd, T, Hd, last_hidden + 1LL * b0 * S * Hd, Hd, s));
        }
    }
    return 0;
}

int run_fusion(mrd_ctx* c, BatchPlan* bp, int B, float* fused_f32, float* attn_i2t, float* attn_t2i,
               cudaStream_t s) {
    const int F = c->fusion_dim;
    MRD_TRY(run(c, "fusion.image_proj", bp->ip, s));
    MRD_TRY(run(c, "fusion.text_proj", bp->tp, s));
    MRD_TRY(run(c, "fusion.img2txt_attn", bp->i2t, s));
    MRD_TRY(run(c, "fusion.txt2img_attn", bp->t2i, s));
    {
        ProfScope ps(c, s, "fusion.layernorm", CAT_MEM, 0, 4.0 * B * F);
        MRD_TRY(layernorm_residual(c->b_prei, F, nullptr, 0, c->ln_i_g, c->ln_i_b, c->fusion_ln_eps, B,
                                   F, c->b_cat, 2 * F, nullptr, 0, s));
    }
    {
        ProfScope ps(c, s, "fusion.layernorm", CAT_MEM, 0, 4.0 * B * F);
        MRD_TRY(layernorm_residual(c->b_pret, F, nullptr, 0, c->ln_t_g, c->ln_t_b, c->fusion_ln_eps, B,
                                   F, c->b_cat + F, 2 * F, nullptr, 0, s));
    }
    MRD_TRY(run(c, "fusion.mlp1", bp->f1, s));
    MRD_TRY(run_f32(c, "fusion.mlp2", bp->f2, fused_f32, fused_f32 ? F : 0, s));
    // softmax over a single key: the weights are exactly 1 (src/fusion_model.py:138-164)
    if (attn_i2t) {
        ProfScope ps(c, s, "fill_ones", CAT_MEM, 0, 4.0 * B * c->fusion_heads);
        MRD_TRY(fill_f32(attn_i2t, 1LL * B * c->fusion_heads, 1.0f, s));
    }
    if (attn_t2i) {
        ProfScope ps(c, s, "fill_ones", CAT_MEM, 0, 4.0 * B * c->fusion_heads);
        MRD_TRY(fill_f32(attn_t2i, 1LL * B * c->fusion_heads, 1.0f, s));
    }
    return 0;
}

int run_head(mrd_ctx* c, BatchPlan* bp, int B, float* logits, float* probs, cudaStream_t s) {
    const bf16* x = c->b_fused;
    int ld = c->head_in;
    for (size_t j = 0; j < bp->head.size(); ++j) {
        MRD_TRY(run(c, "head.hidden", bp->head[j], s));
        x = c->b_h[j & 1];
        ld = c->head_hidden[j].out;
    }
    ProfScope ps(c, s, "head.logits_softmax", CAT_MEM, 0,
                 1.0 * B * (c->head_last * 2.0 + c->num_classes * 8.0));
    MRD_TRY(head_logits_softmax(x, ld, c->head_out_w, c->head_out_b, B, c->head_last, c->num_classes,
                                logits, probs, s));
    return 0;
}

int check_ctx(mrd_ctx* c) {
    if (!c) {
        set_last_error("null context");
        return -1;
    }
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
    if (dev != c->device) {
        e = cudaSetDevice(c->device);
        if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    }
    return 0;
}

#include "engine_train.cuh"
#include "engine_dgrad.cuh"

// mrd_train_forward_ex and mrd_train_forward_dg (save = true: the saving forward for data gradients)
int train_forward_entry(mrd_ctx* c, const void* images, int img_dtype, const long long* ids, const void* mask,
                        int mask_dtype, int B, int H, int W, int S, unsigned long long seed, float* logits,
                        float* feat_map, bool save, float* const* block_out, float* img_emb, float* txt_emb,
                        float* fused, cudaStream_t s) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    MRD_TRY(check_mask_dtype(mask, mask_dtype));
    MRD_TRY(train_forward(c, images, img_dtype, ids, mask, mask_dtype, B, H, W, S, seed, logits, feat_map, save,
                          block_out, s));
    return train_export_embeddings(c, B, img_emb, txt_emb, fused, s);
}

}  // namespace

// ====================================================================== C ABI
extern "C" {

int mrd_abi_version(void) { return MRD_ABI_VERSION; }

int mrd_ctx_create(mrd_ctx** out) {
    if (!out) return -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e, "mrd_ctx_create: cudaGetDevice (no CUDA device?)");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) return cuda_fail(e, "mrd_ctx_create: cudaGetDeviceProperties");
    if (prop.major != 10) {
        set_last_error("mrd_ctx_create: device %d is sm_%d%d; this library only runs on sm_100 (B200)",
                       dev, prop.major, prop.minor);
        return -4;
    }
    mrd_ctx* c = new mrd_ctx();
    c->device = dev;
    *out = c;
    return 0;
}

int mrd_ctx_destroy(mrd_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (void* p : c->weight_allocs) cudaFree(p);
    if (c->cnn_ws.base) cudaFree(c->cnn_ws.base);
    if (c->text_ws.base) cudaFree(c->text_ws.base);
    if (c->batch_ws.base) cudaFree(c->batch_ws.base);
    fp32_arena_free(&c->f32_ws);
    fp32_arena_free(&c->f32_train.ws);
    train_free(c);
    delete c;
    return 0;
}

int mrd_ctx_configure(mrd_ctx* c, int img_chunk, int seq_chunk_tokens) {
    MRD_TRY(check_ctx(c));
    if (img_chunk > 0 && img_chunk != c->img_chunk) {
        c->img_chunk = img_chunk;
        c->cnn_plans.clear();
        c->cnn_ws_B = 0;  // forces a re-carve on next use
    }
    if (seq_chunk_tokens > 0) c->tok_chunk = seq_chunk_tokens;
    return 0;
}

int mrd_ctx_set_option(mrd_ctx* c, const char* key, double v) {
    MRD_TRY(check_ctx(c));
    const std::string k(key ? key : "");
    if (k == "bert_heads") c->bert_heads = static_cast<int>(v);
    else if (k == "bert_ln_eps") c->bert_ln_eps = static_cast<float>(v);
    else if (k == "bn_eps") c->bn_eps = static_cast<float>(v);
    else if (k == "fusion_ln_eps") c->fusion_ln_eps = static_cast<float>(v);
    else if (k == "fusion_heads") c->fusion_heads = static_cast<int>(v);
    else if (k == "fusion_residual") { c->fusion_residual = v != 0.0; c->batch_plans.clear(); }
    else if (k == "head_act") { c->head_act = static_cast<int>(v); c->batch_plans.clear(); }
    else if (k == "fp32_check") c->fp32_check = v != 0.0;
    else if (k == "load_sync") c->load_sync = v != 0.0;
    else if (k.rfind("train.", 0) == 0) return train_set_option(c, k, v);
    else {
        set_last_error("mrd_ctx_set_option: unknown option '%s'", k.c_str());
        return -1;
    }
    return 0;
}

int mrd_ctx_load_weights(mrd_ctx* c, int n, const char* const* names, const void* const* ptrs,
                         const long long* shapes, void* stream) {
    MRD_TRY(check_ctx(c));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Table t;
    t.m.reserve(static_cast<size_t>(n) * 2);
    bool any_cnn = false, any_proj = false, any_text = false, any_fusion = false, any_head = false;
    for (int i = 0; i < n; ++i) {
        Tensor x;
        x.p = static_cast<const float*>(ptrs[i]);
        for (int j = 0; j < 4; ++j) x.d[j] = shapes[i * 4 + j];
        const std::string nm(names[i]);
        t.m.emplace(nm, x);
        RawTensor rt;
        rt.p = x.p;
        for (int j = 0; j < 4; ++j) rt.d[j] = x.d[j];
        c->raw[nm] = rt;
        any_cnn |= nm.rfind("cnn_encoder.backbone.", 0) == 0;
        any_proj |= nm.rfind("cnn_encoder.projection.", 0) == 0;
        any_text |= nm.rfind("text_encoder.", 0) == 0;
        any_fusion |= nm.rfind("fusion.", 0) == 0;
        any_head |= nm.rfind("classifier.", 0) == 0;
    }
    // weights are rewritten in place: nothing may still be reading them
    cudaError_t e = c->load_sync ? cudaDeviceSynchronize() : cudaSuccess;
    if (e != cudaSuccess) return cuda_fail(e, "mrd_ctx_load_weights: device sync");
    const size_t n_blocks = c->blocks.size(), n_layers = c->layers.size(), n_head = c->head_hidden.size();
    if (c->train) train_invalidate_packs(c, any_text, any_cnn);
    if (any_cnn) MRD_TRY(load_cnn(c, t, s));
    if (any_proj) MRD_TRY(load_cnn_projection(c, t, s));
    if (any_text) MRD_TRY(load_text(c, t, s));
    if (any_fusion) MRD_TRY(load_fusion(c, t, s));
    if (any_head) MRD_TRY(load_head(c, t, s));
    // a different architecture than the one the plans were built for invalidates them
    if (n_blocks != c->blocks.size() || n_layers != c->layers.size() || n_head != c->head_hidden.size()) {
        c->cnn_plans.clear();
        c->text_plans.clear();
        c->batch_plans.clear();
    }
    e = c->load_sync ? cudaStreamSynchronize(s) : cudaSuccess;  // the caller may free or mutate its fp32 tensors after return
    if (e != cudaSuccess) return cuda_fail(e, "mrd_ctx_load_weights: packing kernels");
    return 0;
}

int mrd_cnn_encoder_fwd(mrd_ctx* c, const void* images, int img_dtype, int B, int H, int W,
                        float* emb, float* feat_pooled, float* feat_map, void* stream) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (c->fp32_check) {
        MRD_TRY(fp32_images_only(img_dtype));
        ++c->launches;
        return fp32_cnn_encoder(c->raw, c->f32_opts(), &c->f32_ws, static_cast<const float*>(images), B, H,
                                W, emb, feat_pooled, feat_map, s);
    }
    MRD_TRY(ensure_batch_ws(c, B));
    MRD_TRY(run_backbone(c, images, img_dtype, B, H, W, feat_pooled, feat_map, s));
    BatchPlan* bp;
    MRD_TRY(get_batch_plan(c, B, &bp));
    return run_projection(c, bp, emb, s);
}

int mrd_text_encoder_fwd(mrd_ctx* c, const long long* ids, const void* mask, int mask_dtype, int B,
                         int S, float* cls, float* last_hidden, float* all_hidden, void* stream) {
    return mrd_text_encoder_fwd_ex(c, ids, mask, mask_dtype, B, S, cls, last_hidden, all_hidden, nullptr, stream);
}

int mrd_text_encoder_fwd_ex(mrd_ctx* c, const long long* ids, const void* mask, int mask_dtype, int B, int S,
                            float* cls, float* last_hidden, float* all_hidden, float* attn_probs, void* stream) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    MRD_TRY(check_mask_dtype(mask, mask_dtype));
    if (c->fp32_check) {
        ++c->launches;
        return fp32_text_encoder(c->raw, c->f32_opts(), &c->f32_ws, ids, mask, mask_dtype, B, S, cls,
                                 last_hidden, all_hidden, attn_probs, static_cast<cudaStream_t>(stream));
    }
    MRD_TRY(ensure_batch_ws(c, B));
    return run_bert(c, ids, mask, mask_dtype, B, S, cls, last_hidden, all_hidden, attn_probs,
                    static_cast<cudaStream_t>(stream));
}

int mrd_fusion_fwd(mrd_ctx* c, const float* img_emb, const float* txt_emb, int B, float* fused,
                   float* attn_i2t, float* attn_t2i, void* stream) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    if (!c->has_fusion) {
        set_last_error("fusion weights are not loaded in this context");
        return -3;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (c->fp32_check) {
        ++c->launches;
        return fp32_fusion(c->raw, c->f32_opts(), &c->f32_ws, img_emb, txt_emb, B, fused, attn_i2t, attn_t2i, s);
    }
    MRD_TRY(ensure_batch_ws(c, B));
    BatchPlan* bp;
    MRD_TRY(get_batch_plan(c, B, &bp));
    {
        ProfScope ps(c, s, "cast_f32_to_bf16", CAT_MEM, 0, 6.0 * B * c->fusion_img_in);
        MRD_TRY(cast_f32_to_bf16(img_emb, c->fusion_img_in, B, c->fusion_img_in, c->b_img,
                                 c->fusion_img_in, s));
    }
    {
        ProfScope ps(c, s, "cast_f32_to_bf16", CAT_MEM, 0, 6.0 * B * c->fusion_txt_in);
        MRD_TRY(cast_f32_to_bf16(txt_emb, c->fusion_txt_in, B, c->fusion_txt_in, c->b_txt,
                                 c->fusion_txt_in, s));
    }
    return run_fusion(c, bp, B, fused, attn_i2t, attn_t2i, s);
}

namespace {
// fusion -> head -> softmax from the bf16 embeddings in b_img / b_txt: one launch when the plan has the fused tail
int run_tail(mrd_ctx* c, BatchPlan* bp, int B, float* fused, float* attn_i2t, float* attn_t2i, float* logits,
             float* probs, cudaStream_t s) {
    if (!bp->has_tail) {
        MRD_TRY(run_fusion(c, bp, B, fused, attn_i2t, attn_t2i, s));
        return run_head(c, bp, B, logits, probs, s);
    }
    {
        ProfScope ps(c, s, "fusion+head (one launch)", CAT_TENSOR, bp->tail.flops, bp->tail.bytes);
        MRD_TRY(launch_tail(&bp->tail, logits, probs, fused, c->fusion_dim, s));
    }
    // softmax over a single key: the weights are exactly 1 (src/fusion_model.py:138-164)
    for (float* a : {attn_i2t, attn_t2i})
        if (a) {
            ProfScope ps(c, s, "fill_ones", CAT_MEM, 0, 4.0 * B * c->fusion_heads);
            MRD_TRY(fill_f32(a, 1LL * B * c->fusion_heads, 1.0f, s));
        }
    return 0;
}
}  // namespace

int mrd_fusion_head_fwd(mrd_ctx* c, const float* img_emb, const float* txt_emb, int B, float* fused, float* logits,
                        float* probs, void* stream) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    if (!c->has_fusion || !c->has_head) {
        set_last_error("mrd_fusion_head_fwd needs fusion and classifier weights");
        return -3;
    }
    if (c->fp32_check) {
        set_last_error("mrd_fusion_head_fwd has no fp32 check mode: call mrd_fusion_fwd and mrd_head_fwd");
        return -1;
    }
    if (c->fusion_dim != c->head_in) {
        set_last_error("fusion / head dimensions do not chain (%d->%d)", c->fusion_dim, c->head_in);
        return -1;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    MRD_TRY(ensure_batch_ws(c, B));
    BatchPlan* bp;
    MRD_TRY(get_batch_plan(c, B, &bp));
    {
        ProfScope ps(c, s, "cast_f32_to_bf16", CAT_MEM, 0, 6.0 * B * c->fusion_img_in);
        MRD_TRY(cast_f32_to_bf16(img_emb, c->fusion_img_in, B, c->fusion_img_in, c->b_img, c->fusion_img_in, s));
    }
    {
        ProfScope ps(c, s, "cast_f32_to_bf16", CAT_MEM, 0, 6.0 * B * c->fusion_txt_in);
        MRD_TRY(cast_f32_to_bf16(txt_emb, c->fusion_txt_in, B, c->fusion_txt_in, c->b_txt, c->fusion_txt_in, s));
    }
    return run_tail(c, bp, B, fused, nullptr, nullptr, logits, probs, s);
}

int mrd_head_fwd(mrd_ctx* c, const float* x, int B, float* logits, float* probs, void* stream) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    if (!c->has_head) {
        set_last_error("classifier weights are not loaded in this context");
        return -3;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (c->fp32_check) {
        ++c->launches;
        return fp32_head(c->raw, c->f32_opts(), &c->f32_ws, x, B, logits, probs, s);
    }
    MRD_TRY(ensure_batch_ws(c, B));
    BatchPlan* bp;
    MRD_TRY(get_batch_plan(c, B, &bp));
    {
        ProfScope ps(c, s, "cast_f32_to_bf16", CAT_MEM, 0, 6.0 * B * c->head_in);
        MRD_TRY(cast_f32_to_bf16(x, c->head_in, B, c->head_in, c->b_fused, c->head_in, s));
    }
    return run_head(c, bp, B, logits, probs, s);
}

int mrd_multimodal_fwd(mrd_ctx* c, const void* images, int img_dtype, const long long* ids,
                       const void* mask, int mask_dtype, int B, int H, int W, int S, float* logits,
                       float* probs, float* img_emb, float* txt_emb, float* fused, float* attn_i2t,
                       float* attn_t2i, void* stream) {
    MRD_TRY(check_ctx(c));
    if (B <= 0) return 0;
    if (!(c->has_cnn && c->has_text && c->has_fusion && c->has_head)) {
        set_last_error("mrd_multimodal_fwd needs cnn_encoder, text_encoder, fusion and classifier weights");
        return -3;
    }
    if (c->img_emb_dim != c->fusion_img_in || c->hidden != c->fusion_txt_in ||
        c->fusion_dim != c->head_in) {
        set_last_error("encoder / fusion / head dimensions do not chain (%d->%d, %d->%d, %d->%d)",
                       c->img_emb_dim, c->fusion_img_in, c->hidden, c->fusion_txt_in, c->fusion_dim,
                       c->head_in);
        return -1;
    }
    MRD_TRY(check_mask_dtype(mask, mask_dtype));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    MRD_TRY(ensure_batch_ws(c, B));
    if (c->fp32_check) {
        // every stage in plain fp32 on the raw parameters; embeddings nobody asked for live in scratch
        MRD_TRY(fp32_images_only(img_dtype));
        float* sc = c->b_scratch_f32;
        float* ie = img_emb ? img_emb : sc;
        float* te = txt_emb ? txt_emb : sc + 1LL * B * c->img_emb_dim;
        float* fe = fused ? fused : sc + 1LL * B * (c->img_emb_dim + c->hidden);
        if (c->img_emb_dim + c->hidden + c->fusion_dim > 2048) {
            set_last_error("fp32 check: embedding widths exceed the scratch row");
            return -1;
        }
        const Fp32Opts o = c->f32_opts();
        c->launches += 4;
        MRD_TRY(fp32_cnn_encoder(c->raw, o, &c->f32_ws, static_cast<const float*>(images), B, H, W, ie,
                                 nullptr, nullptr, s));
        MRD_TRY(fp32_text_encoder(c->raw, o, &c->f32_ws, ids, mask, mask_dtype, B, S, te, nullptr, nullptr, nullptr, s));
        MRD_TRY(fp32_fusion(c->raw, o, &c->f32_ws, ie, te, B, fe, attn_i2t, attn_t2i, s));
        return fp32_head(c->raw, o, &c->f32_ws, fe, B, logits, probs, s);
    }
    BatchPlan* bp;
    MRD_TRY(get_batch_plan(c, B, &bp));
    MRD_TRY(run_backbone(c, images, img_dtype, B, H, W, nullptr, nullptr, s));
    MRD_TRY(run_projection(c, bp, img_emb, s));
    MRD_TRY(run_bert(c, ids, mask, mask_dtype, B, S, txt_emb, nullptr, nullptr, nullptr, s));
    return run_tail(c, bp, B, fused, attn_i2t, attn_t2i, logits, probs, s);
}

int mrd_ctx_profile(mrd_ctx* c, int enable) {
    MRD_TRY(check_ctx(c));
    for (auto& r : c->prof) {
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    c->prof.clear();
    c->profiling = enable != 0;
    gemm_set_pdl(!c->profiling);
    return 0;
}

int mrd_ctx_profile_report(mrd_ctx* c, char* buf, int cap) {
    MRD_TRY(check_ctx(c));
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return cuda_fail(e, "mrd_ctx_profile_report: sync");
    struct Agg {
        int cat = 0;
        long long n = 0;
        double ms = 0, flops = 0, bytes = 0;
    };
    std::map<std::string, Agg> agg;
    for (auto& r : c->prof) {
        float ms = 0;
        cudaEventElapsedTime(&ms, r.e0, r.e1);
        Agg& a = agg[r.label];
        a.cat = r.cat;
        ++a.n;
        a.ms += ms;
        a.flops += r.flops;
        a.bytes += r.bytes;
    }
    int off = 0;
    for (auto& kv : agg) {
        int w = snprintf(buf + off, off < cap ? cap - off : 0, "%s,%d,%lld,%.6f,%.6e,%.6e\n",
                         kv.first.c_str(), kv.second.cat, kv.second.n, kv.second.ms, kv.second.flops,
                         kv.second.bytes);
        if (w < 0 || off + w >= cap) {
            set_last_error("mrd_ctx_profile_report: buffer too small");
            return -1;
        }
        off += w;
    }
    return 0;
}

int mrd_train_forward_ex(mrd_ctx* c, const void* images, int img_dtype, const long long* ids, const void* mask,
                         int mask_dtype, int B, int H, int W, int S, unsigned long long seed, float* logits,
                         float* feat_map, float* img_emb, float* txt_emb, float* fused, void* stream) {
    return train_forward_entry(c, images, img_dtype, ids, mask, mask_dtype, B, H, W, S, seed, logits, feat_map, false,
                               nullptr, img_emb, txt_emb, fused, static_cast<cudaStream_t>(stream));
}

int mrd_train_forward(mrd_ctx* c, const void* images, int img_dtype, const long long* ids, const void* mask,
                      int mask_dtype, int B, int H, int W, int S, unsigned long long seed, float* logits,
                      void* stream) {
    return mrd_train_forward_ex(c, images, img_dtype, ids, mask, mask_dtype, B, H, W, S, seed, logits, nullptr, nullptr,
                                nullptr, nullptr, stream);
}

int mrd_train_backward_ex(mrd_ctx* c, const float* dlogits, int n, const char* const* names, float* const* grads,
                          float* d_pooled, void* stream) {
    MRD_TRY(check_ctx(c));
    return train_backward(c, dlogits, grad_table(n, names, grads), d_pooled, static_cast<cudaStream_t>(stream));
}

int mrd_train_backward_begin(mrd_ctx* c, const float* dlogits, int n, const char* const* names,
                             float* const* grads, float* d_pooled) {
    MRD_TRY(check_ctx(c));
    return train_backward_begin(c, dlogits, grad_table(n, names, grads), d_pooled);
}

int mrd_train_backward_stages(mrd_ctx* c, int first, int last, void* stream) {
    MRD_TRY(check_ctx(c));
    return train_backward_run(c, first, last, static_cast<cudaStream_t>(stream));
}

int mrd_train_backward_num_stages(mrd_ctx* c) {
    if (!c) return -1;
    return train_backward_stages(c);
}

int mrd_train_backward(mrd_ctx* c, const float* dlogits, int n, const char* const* names, float* const* grads,
                       void* stream) {
    return mrd_train_backward_ex(c, dlogits, n, names, grads, nullptr, stream);
}

int mrd_train_forward_dg(mrd_ctx* c, const void* images, int img_dtype, const long long* ids, const void* mask,
                         int mask_dtype, int B, int H, int W, int S, unsigned long long seed, float* logits,
                         float* const* block_out, float* img_emb, float* txt_emb, float* fused, void* stream) {
    return train_forward_entry(c, images, img_dtype, ids, mask, mask_dtype, B, H, W, S, seed, logits, nullptr, true,
                               block_out, img_emb, txt_emb, fused, static_cast<cudaStream_t>(stream));
}

int mrd_train_backward_dg(mrd_ctx* c, const float* dlogits, int n, const char* const* names, float* const* grads,
                          float* d_pooled, float* const* block_grads, int first_block, float* d_block_in,
                          float* d_images, void* stream) {
    MRD_TRY(check_ctx(c));
    DgradCnn* d = c->train ? c->train->dg : nullptr;
    if (!d || !d->valid) {
        set_last_error("mrd_train_backward_dg: the pending forward was not a mrd_train_forward_dg");
        return -1;
    }
    float* dp = d_pooled ? d_pooled : d->d_pooled;
    if (!d_pooled) {
        cudaError_t e = cudaMemsetAsync(dp, 0, sizeof(float) * d->B * c->feat_dim, static_cast<cudaStream_t>(stream));
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(d_pooled)");
    }
    MRD_TRY(mrd_train_backward_ex(c, dlogits, n, names, grads, dp, stream));
    static float* const kNone[16] = {};
    return dgrad_backbone(c, dp, block_grads ? block_grads : kNone, first_block, d_block_in, d_images,
                          static_cast<cudaStream_t>(stream));
}

int mrd_dropout_mask(unsigned long long seed, unsigned int site, double p, long long n, float* out, void* stream) {
    return dropout_mask_f32(make_drop(seed, site, p), n, out, static_cast<cudaStream_t>(stream));
}

int mrd_attention_bwd_bf16(const void* qkv, const void* ctx, const void* dctx, const float* mask_bias,
                           const int* seq_off, int B, int S, int heads, unsigned long long seed,
                           unsigned int site, double p, void* dqkv, float* dkv_acc, long long rows, void* stream) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    MRD_TRY(attention_backward(static_cast<const bf16*>(qkv), static_cast<const bf16*>(ctx),
                               static_cast<const bf16*>(dctx), mask_bias, seq_off, B, S, heads,
                               make_drop(seed, site, p), static_cast<bf16*>(dqkv), s, dkv_acc));
    if (S > 128) {   // fold the fp32 dK | dV accumulators into dqkv's K / V columns
        const int Hd = heads * 64;
        if (rows <= 0 || rows > 0x7fffffffLL) {
            set_last_error("mrd_attention_bwd_bf16: rows (of qkv / dqkv / dkv_acc) is required when S > 128");
            return -1;
        }
        return cast_f32_to_bf16(dkv_acc, 2 * Hd, static_cast<int>(rows), 2 * Hd, static_cast<bf16*>(dqkv) + Hd, 3 * Hd, s);
    }
    return 0;
}

int mrd_attention_train_bf16(const void* qkv, const float* mask_bias, int B, int S, int heads,
                             unsigned long long seed, unsigned int site, double p, void* out, void* stream) {
    const DropCfg d = make_drop(seed, site, p);
    return attention_forward(static_cast<const bf16*>(qkv), mask_bias, nullptr, B, S, heads,
                             static_cast<bf16*>(out), static_cast<cudaStream_t>(stream), 0, 0, &d);
}

int mrd_attention_train_varlen_bf16(const void* qkv, const float* row_bias, const int* seq_off, int B, int S_max,
                                    int heads, long long rows, unsigned long long seed, unsigned int site, double p,
                                    void* out, void* stream) {
    if (!seq_off) {
        set_last_error("mrd_attention_train_varlen_bf16: seq_off is required");
        return -1;
    }
    if (rows <= 0) {
        set_last_error("mrd_attention_train_varlen_bf16: rows must be the row count of qkv / out");
        return -1;
    }
    const DropCfg d = make_drop(seed, site, p);
    return attention_forward(static_cast<const bf16*>(qkv), row_bias, seq_off, B, S_max, heads, static_cast<bf16*>(out),
                             static_cast<cudaStream_t>(stream), rows, 0, &d);
}

int mrd_layernorm_bwd_bf16(const void* s_in, const void* dy, const float* gamma, float eps, int rows, int width,
                           void* dx, float* dgamma, float* dbeta, void* stream) {
    return ln_bwd_bf16(static_cast<const bf16*>(s_in), static_cast<const bf16*>(dy), gamma, eps, rows, width,
                       nullptr, static_cast<bf16*>(dx), dgamma, dbeta, static_cast<cudaStream_t>(stream));
}

long long mrd_ctx_launch_count(const mrd_ctx* c) { return c ? c->launches : 0; }
long long mrd_ctx_device_bytes(const mrd_ctx* c) { return c ? c->dev_bytes : 0; }

}  // extern "C"
