// Training step of the engine: forward with saved activations + backward (SURVEY.md 8(f).1; reference:
// autograd through MultimodalClassifier.forward in src/train.py:247-321 / src/train_multimodal.py:508-543).
// Included by engine.cu inside its anonymous namespace (it uses the context, arenas and plan helpers
// defined there); the C ABI wrappers are at the end of engine.cu.
//
// What runs where
//   * ResNet50 backbone: forward only - the reference freezes it by default (src/config.py:64,
//     src/cnn_encoder.py:102-106), so no gradient flows into it; BatchNorm uses running statistics
//     when the backbone modules are in eval mode, batch statistics otherwise (run_backbone_train).
//   * BERT: forward = the tcgen05 GEMMs / tcgen05 attention of the inference path on token-packed rows,
//     with every tensor the backward needs kept (layer input, QKV, context, pre-LayerNorm sums, FFN
//     pre-activation and activation).  Backward per layer: LayerNorm backward -> dropout mask ->
//     dW = dY^T X and dX = dY W on the SAME tcgen05 kernel (operands transposed by a staging kernel /
//     transposed bf16 weight copies, fp32 outputs written straight into the caller's gradient
//     tensors) -> GELU' -> attention backward (mma.sync) -> QKV.
//   * projection / fusion / head (rows = batch size): fp32 SIMT GEMMs (simt_gemm.cu) both ways.
// Dropout masks are counter-based (rng.cuh) and recomputed in the backward pass.

// a non-GEMM kernel of the training step: counted, and timed when the context is in profile mode
#define TRK(label, cat, call)                        \
    do {                                             \
        ProfScope ps__(c, s, label, cat, 0.0, 0.0);  \
        MRD_TRY(call);                               \
    } while (0)

struct TrainOpts {
    double p_bert_hidden = 0.1, p_bert_attn = 0.1, p_text_out = 0.1, p_cnn_proj = 0.5, p_fusion = 0.3,
           p_head = 0.5;
    int pad_idx = 0;
    int bn_train = 0;
    double bn_momentum = 0.1;
};

struct TrainLayerBuf {
    bf16 *x = nullptr, *qkv = nullptr, *ctx = nullptr, *s1 = nullptr, *h1 = nullptr, *u = nullptr,
         *g = nullptr, *s2 = nullptr;
};
struct TrainLayerWt {
    bf16 *qkv_t = nullptr, *o_t = nullptr, *f1_t = nullptr, *f2_t = nullptr;  // [in][out] bf16
};
struct TrainLayerPlan {
    GemmLaunch qkv, o, f1, f2;            // forward
    GemmLaunch d_g, d_h1, d_ctx, d_x;     // dX = dY W
    GemmLaunch d_g0, d_ctx0;              // the same with A = d_s (no dropout mask between LayerNorm and dense)
};

struct TrainCnn;
struct DgradCnn;

struct TrainState {
    TrainOpts o;
    TrainCnn* cnn = nullptr;              // batch-statistics backbone (created when bn_train is first used)
    DgradCnn* dg = nullptr;               // data gradients through the backbone (engine_dgrad.cuh), created on first use
    std::vector<TrainLayerWt> wt;
    bool packs_valid = false;
    // plan / workspace for one (B, S)
    int B = 0, S = 0, Ta = 0, Tp = 0;
    long long text_ws_epoch = -1;         // c->text_ws_epoch the plans were built against
    long long text_run_epoch = -1;        // c->text_run_epoch right after the pending forward
    mrd_ctx::Arena ws;
    std::vector<TrainLayerBuf> L;
    std::vector<TrainLayerPlan> P;
    GemmLaunch w_f2, w_f1, w_o, w_qkv;    // dW = dY^T X on the shared staging buffers
    bf16 *x_final = nullptr, *z = nullptr, *dxa = nullptr, *dxb = nullptr, *d_s = nullptr, *dz = nullptr,
         *dh1 = nullptr, *dctx = nullptr, *dbig = nullptr, *dqkv = nullptr, *At = nullptr, *Bt = nullptr;
    float* dkv_acc = nullptr;             // [Ta, 2*Hd] fp32: dK / dV accumulator of the tiled attention backward (S > 128)
    float* wq_scratch = nullptr;          // [3*Hd, Hd] fp32: QKV weight gradient before it is split
    float* bq_scratch = nullptr;          // [3*Hd]
    // batch-level fp32 activations
    float *pooled = nullptr, *a1 = nullptr, *p1 = nullptr, *img = nullptr, *cls = nullptr, *txt = nullptr,
          *ip = nullptr, *tp = nullptr, *v1 = nullptr, *v1d = nullptr, *v2 = nullptr, *v2d = nullptr,
          *pre_i = nullptr, *pre_t = nullptr, *cat = nullptr, *fh = nullptr, *fused = nullptr;
    std::vector<float*> hh;               // head hidden activations (post dropout)
    float *g0 = nullptr, *g1 = nullptr, *g2 = nullptr, *g3 = nullptr, *g4 = nullptr;  // [B, 2048] gradient scratch
    // staged backward (train_backward_begin / train_backward_run)
    bool bw_active = false, bw_want_text = false;
    int bw_next = 0;
    const float* bw_dlogits = nullptr;
    float* bw_d_pooled = nullptr;
    std::unordered_map<std::string, float*> bw_grads;
    // forward bookkeeping
    bool fwd_done = false;
    unsigned long long seed = 0;
    const long long* ids = nullptr;
};

enum : unsigned { SITE_EMB = 1000, SITE_TEXT_OUT = 1001, SITE_CNN_PROJ = 1002, SITE_I2T = 1003,
                  SITE_T2I = 1004, SITE_FUSION_MLP = 1005, SITE_HEAD = 1010 };
inline unsigned site_attn(size_t l) { return static_cast<unsigned>(16 * l); }
inline unsigned site_attn_out(size_t l) { return static_cast<unsigned>(16 * l + 1); }
inline unsigned site_ffn_out(size_t l) { return static_cast<unsigned>(16 * l + 2); }

TrainState* train_state(mrd_ctx* c) {
    if (!c->train) c->train = new TrainState();
    return c->train;
}

void train_cnn_invalidate(TrainState* t);
void train_cnn_free(TrainState* t);
void dgrad_invalidate(TrainState* t);
void dgrad_forget(TrainState* t);
void dgrad_free(TrainState* t);
int run_backbone_save(mrd_ctx* c, const void* images, int img_dtype, int B, int H, int W, float* pooled_f32,
                      float* const* block_out, cudaStream_t s);

void train_invalidate_packs(mrd_ctx* c, bool text, bool backbone) {
    if (!c->train) return;
    if (text) c->train->packs_valid = false;
    if (backbone) train_cnn_invalidate(c->train);
}

void train_free(mrd_ctx* c) {
    if (!c->train) return;
    if (c->train->ws.base) cudaFree(c->train->ws.base);
    train_cnn_free(c->train);
    delete c->train;
    c->train = nullptr;
}

int train_set_option(mrd_ctx* c, const std::string& k, double v) {
    TrainOpts& o = train_state(c)->o;
    if (k == "train.p_bert_hidden") o.p_bert_hidden = v;
    else if (k == "train.p_bert_attn") o.p_bert_attn = v;
    else if (k == "train.p_text_out") o.p_text_out = v;
    else if (k == "train.p_cnn_proj") o.p_cnn_proj = v;
    else if (k == "train.p_fusion") o.p_fusion = v;
    else if (k == "train.p_head") o.p_head = v;
    else if (k == "train.pad_idx") o.pad_idx = static_cast<int>(v);
    else if (k == "train.bn_train") o.bn_train = v != 0.0;
    else if (k == "train.bn_momentum") o.bn_momentum = v;
    else {
        set_last_error("mrd_ctx_set_option: unknown option '%s'", k.c_str());
        return -1;
    }
    return 0;
}

int raw_need(mrd_ctx* c, const std::string& k, const RawTensor** out) {
    auto it = c->raw.find(k);
    if (it == c->raw.end()) {
        set_last_error("training step: tensor '%s' was not handed over by load_weights", k.c_str());
        return -2;
    }
    *out = &it->second;
    return 0;
}

// Transposed bf16 copies of the BERT linears: the B operand of dX = dY W.  Rebuilt after every
// load_weights (the optimizer changed the parameters).
int train_ensure_packs(mrd_ctx* c, cudaStream_t s) {
    TrainState* t = train_state(c);
    if (t->packs_valid) return 0;
    const int Hd = c->hidden, F = c->ffn;
    t->wt.resize(c->layers.size());
    for (size_t i = 0; i < c->layers.size(); ++i) {
        TrainLayerWt& w = t->wt[i];
        char pre[96];
        snprintf(pre, sizeof(pre), "text_encoder.encoder.encoder.layer.%zu.", i);
        const std::string p(pre);
        MRD_TRY(walloc(c, &w.qkv_t, 3LL * Hd * Hd));
        MRD_TRY(walloc(c, &w.o_t, 1LL * Hd * Hd));
        MRD_TRY(walloc(c, &w.f1_t, 1LL * Hd * F));
        MRD_TRY(walloc(c, &w.f2_t, 1LL * Hd * F));
        // transposed ([in][out]) copies of the PACKED bf16 weights (the query block already carries the folded
        // 1/sqrt(64)): word-wise transposes, two matrices per launch
        const BertLayerW& W = c->layers[i];
        TRK("train.pack", CAT_MEM, transpose_pad2_bf16(W.qkv.w, Hd, Hd, w.qkv_t, nullptr, 0, 0, nullptr, 3 * Hd, nullptr,
                                                      3 * Hd, s));
        TRK("train.pack", CAT_MEM, transpose_pad2_bf16(W.o.w, Hd, Hd, w.o_t, nullptr, 0, 0, nullptr, Hd, nullptr, Hd, s));
        TRK("train.pack", CAT_MEM, transpose_pad2_bf16(W.f1.w, Hd, Hd, w.f1_t, nullptr, 0, 0, nullptr, F, nullptr, F, s));
        TRK("train.pack", CAT_MEM, transpose_pad2_bf16(W.f2.w, F, F, w.f2_t, nullptr, 0, 0, nullptr, Hd, nullptr, Hd, s));
    }
    t->packs_valid = true;
    return 0;
}

int train_ensure_plan(mrd_ctx* c, int B, int S) {
    TrainState* t = train_state(c);
    if (t->ws.base && t->B == B && t->S == S && t->P.size() == c->layers.size() &&
        t->text_ws_epoch == c->text_ws_epoch)
        return 0;
    const int Hd = c->hidden, F = c->ffn;
    const long long Ta = 1LL * B * S;
    const long long Tp = (Ta + 63) / 64 * 64;
    const size_t nl = c->layers.size();
    const int wide = F > 3 * Hd ? F : 3 * Hd;
    size_t total = 0;
    total += nl * (5 * pad1k(Ta * Hd, 2) + pad1k(Ta * 3 * Hd, 2) + 2 * pad1k(Ta * F, 2));  // saved per layer
    total += 8 * pad1k(Ta * Hd, 2) + pad1k(Ta * F, 2) + pad1k(Ta * 3 * Hd, 2);             // x_final + temporaries
    total += 2 * pad1k(1LL * wide * Tp, 2);                                                 // At, Bt
    total += pad1k(3LL * Hd * Hd, 4) + pad1k(3LL * Hd, 4) + (S > 128 ? pad1k(Ta * 2 * Hd, 4) : 0);
    const long long bw = 2048;
    const size_t n_head = c->head_hidden.size();
    total += (17 + n_head + 5) * pad1k(1LL * B * bw, 4);
    MRD_TRY(arena_reset(c, &t->ws, total));
    cudaError_t e = cudaMemset(t->ws.base, 0, t->ws.bytes);  // rows beyond the live count stay finite
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemset(training workspace)");
    t->L.assign(nl, TrainLayerBuf());
    for (size_t i = 0; i < nl; ++i) {
        TrainLayerBuf& b = t->L[i];
        b.x = arena_take<bf16>(&t->ws, Ta * Hd);
        b.qkv = arena_take<bf16>(&t->ws, Ta * 3 * Hd);
        b.ctx = arena_take<bf16>(&t->ws, Ta * Hd);
        b.s1 = arena_take<bf16>(&t->ws, Ta * Hd);
        b.h1 = arena_take<bf16>(&t->ws, Ta * Hd);
        b.u = arena_take<bf16>(&t->ws, Ta * F);
        b.g = arena_take<bf16>(&t->ws, Ta * F);
        b.s2 = arena_take<bf16>(&t->ws, Ta * Hd);
    }
    t->x_final = arena_take<bf16>(&t->ws, Ta * Hd);
    t->z = arena_take<bf16>(&t->ws, Ta * Hd);
    t->dxa = arena_take<bf16>(&t->ws, Ta * Hd);
    t->dxb = arena_take<bf16>(&t->ws, Ta * Hd);
    t->d_s = arena_take<bf16>(&t->ws, Ta * Hd);
    t->dz = arena_take<bf16>(&t->ws, Ta * Hd);
    t->dh1 = arena_take<bf16>(&t->ws, Ta * Hd);
    t->dctx = arena_take<bf16>(&t->ws, Ta * Hd);
    t->dbig = arena_take<bf16>(&t->ws, Ta * F);
    t->dqkv = arena_take<bf16>(&t->ws, Ta * 3 * Hd);
    t->At = arena_take<bf16>(&t->ws, 1LL * wide * Tp);
    t->Bt = arena_take<bf16>(&t->ws, 1LL * wide * Tp);
    t->dkv_acc = S > 128 ? arena_take<float>(&t->ws, Ta * 2 * Hd) : nullptr;
    t->wq_scratch = arena_take<float>(&t->ws, 3LL * Hd * Hd);
    t->bq_scratch = arena_take<float>(&t->ws, 3LL * Hd);
    float** fb[] = {&t->pooled, &t->a1, &t->p1, &t->img, &t->cls, &t->txt, &t->ip, &t->tp, &t->v1, &t->v1d,
                    &t->v2, &t->v2d, &t->pre_i, &t->pre_t, &t->cat, &t->fh, &t->fused};
    for (float** p : fb) *p = arena_take<float>(&t->ws, 1LL * B * bw);
    t->hh.assign(n_head, nullptr);
    for (size_t j = 0; j < n_head; ++j) t->hh[j] = arena_take<float>(&t->ws, 1LL * B * bw);
    t->g0 = arena_take<float>(&t->ws, 1LL * B * bw);
    t->g1 = arena_take<float>(&t->ws, 1LL * B * bw);
    t->g2 = arena_take<float>(&t->ws, 1LL * B * bw);
    t->g3 = arena_take<float>(&t->ws, 1LL * B * bw);
    t->g4 = arena_take<float>(&t->ws, 1LL * B * bw);

    const int T = static_cast<int>(Ta);
    t->P.assign(nl, TrainLayerPlan());
    for (size_t i = 0; i < nl; ++i) {
        const BertLayerW& W = c->layers[i];
        const TrainLayerWt& Wt = t->wt[i];
        const TrainLayerBuf& b = t->L[i];
        TrainLayerPlan& p = t->P[i];
        MRD_TRY(plan_gemm(&p.qkv, b.x, Hd, T, Hd, W.qkv.w, 3 * Hd, W.qkv.b, b.qkv, 3 * Hd, nullptr, 0, nullptr, 0,
                          ACT_NONE));
        MRD_TRY(plan_gemm(&p.o, b.ctx, Hd, T, Hd, W.o.w, Hd, W.o.b, t->z, Hd, nullptr, 0, nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.f1, b.h1, Hd, T, Hd, W.f1.w, F, W.f1.b, b.u, F, nullptr, 0, nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.f2, b.g, F, T, F, W.f2.w, Hd, W.f2.b, t->z, Hd, nullptr, 0, nullptr, 0, ACT_NONE));
        // dG = dZ2 W2 ; dH1 = dU W1 + dS2 ; dCtx = dZ1 Wo ; dX = dQKV Wqkv + dS1
        MRD_TRY(plan_gemm(&p.d_g, t->dz, Hd, T, Hd, Wt.f2_t, F, nullptr, t->dbig, F, nullptr, 0, nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.d_h1, t->dbig, F, T, F, Wt.f1_t, Hd, nullptr, t->dh1, Hd, t->d_s, Hd, nullptr, 0,
                          ACT_NONE));
        MRD_TRY(plan_gemm(&p.d_ctx, t->dz, Hd, T, Hd, Wt.o_t, Hd, nullptr, t->dctx, Hd, nullptr, 0, nullptr, 0,
                          ACT_NONE));
        MRD_TRY(plan_gemm(&p.d_g0, t->d_s, Hd, T, Hd, Wt.f2_t, F, nullptr, t->dbig, F, nullptr, 0, nullptr, 0, ACT_NONE));
        MRD_TRY(plan_gemm(&p.d_ctx0, t->d_s, Hd, T, Hd, Wt.o_t, Hd, nullptr, t->dctx, Hd, nullptr, 0, nullptr, 0,
                          ACT_NONE));
        // layer i reads its output gradient from dx[(i+1)&1] and writes its input gradient to dx[i&1]
        bf16* dx_out = (i & 1) ? t->dxb : t->dxa;
        MRD_TRY(plan_gemm(&p.d_x, t->dqkv, 3 * Hd, T, 3 * Hd, Wt.qkv_t, Hd, nullptr, dx_out, Hd, t->d_s, Hd, nullptr,
                          0, ACT_NONE));
        GemmLaunch* all[] = {&p.qkv, &p.o, &p.f1, &p.f2, &p.d_g, &p.d_h1, &p.d_ctx, &p.d_x, &p.d_g0, &p.d_ctx0};
        for (GemmLaunch* g : all) g->p.dyn_rows = c->t_nrows;
    }
    // dW[out,in] += dY^T[out,Tp] * (X^T[in,Tp])^T : split-K over the live tokens, fp32 partial sums added
    // into the (zeroed) destination, which is patched per launch
    const int K = static_cast<int>(Tp);
    MRD_TRY(plan_gemm_splitk(&t->w_f2, t->At, Tp, Hd, K, t->Bt, F, t->wq_scratch, F, c->t_nrows));
    MRD_TRY(plan_gemm_splitk(&t->w_f1, t->At, Tp, F, K, t->Bt, Hd, t->wq_scratch, Hd, c->t_nrows));
    MRD_TRY(plan_gemm_splitk(&t->w_o, t->At, Tp, Hd, K, t->Bt, Hd, t->wq_scratch, Hd, c->t_nrows));
    MRD_TRY(plan_gemm_splitk(&t->w_qkv, t->At, Tp, 3 * Hd, K, t->Bt, Hd, t->wq_scratch, Hd, c->t_nrows));
    t->B = B; t->S = S; t->Ta = T; t->Tp = K;
    t->text_ws_epoch = c->text_ws_epoch;
    return 0;
}

// ---- frozen backbone under model.train(): BatchNorm on batch statistics --------------------------------
// The reference's default training configuration freezes the backbone's parameters but leaves its
// BatchNorm layers in train mode (src/cnn_encoder.py:102-106 only clears requires_grad), so every
// convolution is followed by batch statistics, normalisation and a running-stat update
// (TV:models/resnet.py:143-163 under nn.Module.train()).  Convolutions run on the same tcgen05 implicit-GEMM
// kernel with un-folded weights; statistics / normalise+residual+ReLU are two HBM-bound passes.
struct TrainCnn {
    bool packed = false;
    bf16* stem_w = nullptr;
    float *ones = nullptr, *zeros = nullptr;     // [2048] identity BatchNorm for the packers / zero bias
    float* dummy_bias = nullptr;                 // [2048] bias output of the packers (always zero, unused)
    std::vector<Bottleneck> blocks;              // raw (un-folded) filters
    float* stats = nullptr;                      // [sites][4][2048]: sum, sumsq, shift, (1 spare)
    BnSite* site_table = nullptr;                // device: one entry per BatchNorm layer (running-stat update)
    std::vector<BnSite> site_host;
    std::vector<std::string> bn_names;           // site -> "cnn_encoder.backbone....bnX"
    int B = 0, H = 0, W = 0;
    long long ws_epoch = -1;
    CnnPlan plan;
};

TrainCnn* train_cnn(mrd_ctx* c) {
    TrainState* t = train_state(c);
    if (!t->cnn) t->cnn = new TrainCnn();
    return t->cnn;
}

int train_cnn_pack(mrd_ctx* c, cudaStream_t s) {
    TrainCnn* tc = train_cnn(c);
    if (tc->packed) return 0;
    const std::string bb = "cnn_encoder.backbone.";
    if (!tc->ones) {
        MRD_TRY(walloc(c, &tc->ones, 2048));
        MRD_TRY(walloc(c, &tc->zeros, 2048));
        MRD_TRY(fill_f32(tc->ones, 2048, 1.0f, s));
        MRD_TRY(fill_f32(tc->zeros, 2048, 0.0f, s));
    }
    const RawTensor* w;
    MRD_TRY(raw_need(c, bb + "conv1.weight", &w));
    MRD_TRY(walloc(c, &tc->stem_w, 64 * 7 * 32));
    MRD_TRY(walloc(c, &tc->dummy_bias, 2048));
    float* dummy_bias = tc->dummy_bias;
    TRK("train.pack", CAT_MEM, pack_stem_bn(w->p, tc->ones, tc->zeros, tc->zeros, tc->ones, 0.0f, tc->stem_w, dummy_bias, s));
    tc->bn_names.clear();
    tc->bn_names.push_back(bb + "bn1");
    tc->blocks.resize(c->blocks.size());
    size_t bi = 0;
    for (int L = 1; L <= 4 && bi < c->blocks.size(); ++L) {
        for (int i = 0; bi < c->blocks.size(); ++i) {
            char pre[96];
            snprintf(pre, sizeof(pre), "%slayer%d.%d.", bb.c_str(), L, i);
            const std::string p(pre);
            if (c->raw.find(p + "conv1.weight") == c->raw.end()) break;
            const Bottleneck& src = c->blocks[bi];
            Bottleneck& dst = tc->blocks[bi];
            // keep previously allocated filters (re-pack in place)
            ConvW keep1 = dst.c1, keep2 = dst.c2, keep3 = dst.c3, keepd = dst.ds;
            auto pack_keep = [&](const std::string& conv, const ConvW& shape, ConvW* out, const ConvW& keep) -> int {
                const RawTensor* cw;
                MRD_TRY(raw_need(c, conv + ".weight", &cw));
                bf16* wbuf = keep.w;
                *out = ConvW(shape);
                out->w = wbuf;
                out->b = tc->zeros;
                MRD_TRY(walloc(c, &out->w, cw->numel()));
                return pack_conv_bn(cw->p, tc->ones, tc->zeros, tc->zeros, tc->ones, 0.0f, shape.cout, shape.cin,
                                    shape.k, out->w, dummy_bias, s);
            };
            MRD_TRY(pack_keep(p + "conv1", src.c1, &dst.c1, keep1));
            MRD_TRY(pack_keep(p + "conv2", src.c2, &dst.c2, keep2));
            MRD_TRY(pack_keep(p + "conv3", src.c3, &dst.c3, keep3));
            dst.has_ds = src.has_ds;
            tc->bn_names.push_back(p + "bn1");
            tc->bn_names.push_back(p + "bn2");
            tc->bn_names.push_back(p + "bn3");
            if (src.has_ds) {
                MRD_TRY(pack_keep(p + "downsample.0", src.ds, &dst.ds, keepd));
                tc->bn_names.push_back(p + "downsample.1");
            }
            ++bi;
        }
    }
    if (!tc->stats) MRD_TRY(walloc(c, &tc->stats, static_cast<long long>(tc->bn_names.size()) * 4 * 2048));
    tc->packed = true;
    tc->B = 0;  // filters may have moved: re-plan
    return 0;
}

int train_cnn_plan(mrd_ctx* c, int B, int H, int W) {
    TrainCnn* tc = train_cnn(c);
    if (tc->B == B && tc->H == H && tc->W == W && tc->ws_epoch == c->cnn_ws_epoch) return 0;
    CnnPlan p;
    p.B = B; p.H = H; p.W = W;
    MRD_TRY(plan_stem(&p.stem, c->xpad, B, H, W, tc->stem_w, tc->zeros, c->stem_out, ACT_NONE));
    int h = H / 4, w = W / 4;
    const bf16* x = c->act0;
    bf16* bufs[2] = {c->act0, c->act1};
    int cur = 0;
    p.blocks.resize(tc->blocks.size());
    for (size_t i = 0; i < tc->blocks.size(); ++i) {
        const Bottleneck& b = tc->blocks[i];
        CnnPlan::BlockPlan& bp = p.blocks[i];
        const int ho = h / b.c2.stride, wo = w / b.c2.stride;
        bf16* y = bufs[cur ^ 1];
        MRD_TRY(plan_conv(&bp.c1, x, B, h, w, b.c1.cin, b.c1.w, b.c1.cout, b.c1.k, 1, b.c1.b, c->mid0, nullptr, ACT_NONE));
        MRD_TRY(plan_conv(&bp.c2, c->mid0, B, h, w, b.c2.cin, b.c2.w, b.c2.cout, b.c2.k, b.c2.stride, b.c2.b, c->mid1,
                          nullptr, ACT_NONE));
        bp.has_ds = b.has_ds;
        if (b.has_ds)
            MRD_TRY(plan_conv(&bp.ds, x, B, h, w, b.ds.cin, b.ds.w, b.ds.cout, b.ds.k, b.ds.stride, b.ds.b, c->dsb,
                              nullptr, ACT_NONE));
        MRD_TRY(plan_conv(&bp.c3, c->mid1, B, ho, wo, b.c3.cin, b.c3.w, b.c3.cout, b.c3.k, 1, b.c3.b, y, nullptr, ACT_NONE));
        x = y;
        cur ^= 1;
        h = ho;
        w = wo;
    }
    p.final_act = x;
    p.final_hw = h * w;
    tc->plan = std::move(p);
    tc->site_host.clear();   // row counts / buffer addresses of the running-stat table belong to this plan
    tc->B = B; tc->H = H; tc->W = W;
    tc->ws_epoch = c->cnn_ws_epoch;
    return 0;
}

int run_backbone_train(mrd_ctx* c, const void* images, int img_dtype, int B, int H, int W, float* pooled_f32,
                       cudaStream_t s) {
    MRD_TRY(check_images(img_dtype, H, W));
    TrainState* t = train_state(c);
    MRD_TRY(ensure_cnn_ws(c, B, H, W));
    MRD_TRY(train_cnn_pack(c, s));
    MRD_TRY(train_cnn_plan(c, B, H, W));
    TrainCnn* tc = t->cnn;
    const size_t n_sites = tc->bn_names.size();
    cudaError_t e = cudaMemsetAsync(tc->stats, 0, sizeof(float) * n_sites * 4 * 2048, s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(bn stats)");
    size_t site = 0;
    const bool fill_table = tc->site_host.empty();
    if (fill_table) tc->site_host.assign(n_sites, BnSite());
    auto bn = [&](bf16* y, long long rows, int C, const bf16* identity, int relu) -> int {
        const std::string& nm = tc->bn_names[site];
        float* st = tc->stats + site * 4 * 2048;
        const RawTensor *g, *b, *rm, *rv;
        MRD_TRY(raw_need(c, nm + ".weight", &g));
        MRD_TRY(raw_need(c, nm + ".bias", &b));
        if (fill_table) {
            MRD_TRY(raw_need(c, nm + ".running_mean", &rm));
            MRD_TRY(raw_need(c, nm + ".running_var", &rv));
            BnSite& e = tc->site_host[site];
            e.sum = st; e.sumsq = st + 2048; e.shift = st + 2 * 2048;
            e.running_mean = const_cast<float*>(rm->p);
            e.running_var = const_cast<float*>(rv->p);
            e.n = static_cast<float>(rows);
            e.C = C;
        }
        ++site;
        TRK("train.bn_stats", CAT_MEM, bn_stats_bf16(y, rows, C, st, st + 2048, st + 2 * 2048, s));
        // scale / shift are derived from the sums inside the normalise pass; the running buffers of all layers
        // are updated by one launch at the end of the backbone
        TRK("train.bn_apply", CAT_MEM, bn_apply_stats_bf16(y, rows, C, st, st + 2048, st + 2 * 2048, g->p, b->p, c->bn_eps,
                                                           identity, relu, s));
        return 0;
    };
    const CnnPlan& p = tc->plan;
    TRK("train.repack_images", CAT_MEM, repack_images(images, img_dtype == MRD_DT_BF16, B, H, W, c->xpad, s));
    MRD_TRY(run(c, "train.conv_stem", p.stem, s));
    MRD_TRY(bn(c->stem_out, 1LL * B * (H / 2) * (W / 2), 64, nullptr, 1));
    TRK("train.maxpool", CAT_MEM, maxpool3x3s2(c->stem_out, B, H / 2, W / 2, 64, c->act0, s));
    int h = H / 4, w = W / 4;
    bf16* bufs[2] = {c->act0, c->act1};
    int cur = 0;
    for (size_t i = 0; i < p.blocks.size(); ++i) {
        const Bottleneck& b = tc->blocks[i];
        const CnnPlan::BlockPlan& bp = p.blocks[i];
        const int ho = h / b.c2.stride, wo = w / b.c2.stride;
        bf16* x = bufs[cur];
        bf16* y = bufs[cur ^ 1];
        MRD_TRY(run(c, "train.conv", bp.c1, s));
        MRD_TRY(bn(c->mid0, 1LL * B * h * w, b.c1.cout, nullptr, 1));
        MRD_TRY(run(c, "train.conv", bp.c2, s));
        MRD_TRY(bn(c->mid1, 1LL * B * ho * wo, b.c2.cout, nullptr, 1));
        MRD_TRY(run(c, "train.conv", bp.c3, s));
        // bn_names order per block: bn1, bn2, bn3, downsample.1 - run bn3's statistics before the downsample
        // branch but apply it after (it needs the identity)
        const bf16* identity = x;
        if (bp.has_ds) {
            const size_t site_bn3 = site;
            ++site;   // reserve bn3, do the downsample site first
            MRD_TRY(run(c, "train.conv", bp.ds, s));
            MRD_TRY(bn(c->dsb, 1LL * B * ho * wo, b.ds.cout, nullptr, 0));
            const size_t after = site;
            site = site_bn3;
            MRD_TRY(bn(y, 1LL * B * ho * wo, b.c3.cout, c->dsb, 1));
            site = after;
        } else {
            MRD_TRY(bn(y, 1LL * B * ho * wo, b.c3.cout, identity, 1));
        }
        cur ^= 1;
        h = ho;
        w = wo;
    }
    TRK("train.avgpool", CAT_MEM, global_avgpool(p.final_act, B, p.final_hw, c->feat_dim, c->b_pooled, pooled_f32, s));
    if (fill_table) {
        MRD_TRY(walloc(c, reinterpret_cast<char**>(&tc->site_table), static_cast<long long>(n_sites * sizeof(BnSite))));
        cudaError_t ce = cudaMemcpyAsync(tc->site_table, tc->site_host.data(), n_sites * sizeof(BnSite),
                                         cudaMemcpyHostToDevice, s);
        if (ce != cudaSuccess) return cuda_fail(ce, "cudaMemcpyAsync(bn site table)");
    }
    TRK("train.bn_running", CAT_MEM, bn_update_running(tc->site_table, static_cast<int>(n_sites), 2048,
                                                      static_cast<float>(t->o.bn_momentum), s));
    return 0;
}

void train_cnn_invalidate(TrainState* t) {
    if (t->cnn) t->cnn->packed = false;
    dgrad_invalidate(t);
}
void train_cnn_free(TrainState* t) {
    delete t->cnn;   // device buffers are weight allocations of the context (freed with it)
    t->cnn = nullptr;
    dgrad_free(t);
}

typedef std::unordered_map<std::string, float*> GradTable;
// the parameters of the C ABI's (names, grads) arrays that have a gradient slot
GradTable grad_table(int n, const char* const* names, float* const* grads) {
    GradTable gt;
    gt.reserve(static_cast<size_t>(n) * 2);
    for (int i = 0; i < n; ++i)
        if (grads[i]) gt.emplace(names[i], grads[i]);
    return gt;
}
inline float* grad_of(const GradTable& g, const std::string& k) {
    auto it = g.find(k);
    return it == g.end() ? nullptr : it->second;
}

// ---- fp32 linear helpers for the batch-level layers (rows = batch) -----------------------------------
int lin_fwd(mrd_ctx* c, const std::string& name, const float* x, long long ldx, int M, float* y, long long ldy,
            int act, const float* res, long long ldr, cudaStream_t s) {
    const RawTensor *w, *b;
    MRD_TRY(raw_need(c, name + ".weight", &w));
    MRD_TRY(raw_need(c, name + ".bias", &b));
    SimtGemm g;
    g.A = x; g.a_rs = ldx; g.a_cs = 1;
    g.B = w->p; g.b_rs = w->d[1]; g.b_cs = 1;
    g.M = M; g.N = static_cast<int>(w->d[0]); g.K = static_cast<int>(w->d[1]);
    g.C = y; g.ldc = ldy;
    g.bias = b->p; g.act = act; g.res = res; g.ldr = ldr;
    TRK("train.simt_gemm", CAT_TENSOR, simt_gemm(g, s));
    return 0;
}

// y = x W^T + b.  dW += dy^T x, db += colsum(dy) (when the parameter has a gradient slot);
// dx = dy W (+ dx_res) when dx != null.
int lin_bwd(mrd_ctx* c, const GradTable& gt, const std::string& name, const float* x, long long ldx,
            const float* dy, long long lddy, int M, float* dx, long long lddx, const float* dx_res,
            long long ld_res, cudaStream_t s) {
    const RawTensor* w;
    MRD_TRY(raw_need(c, name + ".weight", &w));
    const int N = static_cast<int>(w->d[0]), K = static_cast<int>(w->d[1]);
    if (float* gw = grad_of(gt, name + ".weight")) {
        SimtGemm g;  // C[n_out, k_in] = sum_m dy[m, n_out] * x[m, k_in]
        g.A = dy; g.a_rs = 1; g.a_cs = lddy;
        g.B = x; g.b_rs = 1; g.b_cs = ldx;
        g.M = N; g.N = K; g.K = M;
        g.C = gw; g.ldc = K; g.accumulate = 1;
        TRK("train.simt_gemm", CAT_TENSOR, simt_gemm(g, s));
    }
    if (float* gb = grad_of(gt, name + ".bias")) {
        TRK("train.colsum", CAT_MEM, colsum_f32(dy, lddy, M, N, gb, s));
    }
    if (dx) {
        SimtGemm g;  // C[m, k_in] = sum_n dy[m, n] * W[n, k_in]
        g.A = dy; g.a_rs = lddy; g.a_cs = 1;
        g.B = w->p; g.b_rs = 1; g.b_cs = K;
        g.M = M; g.N = K; g.K = N;
        g.C = dx; g.ldc = lddx;
        g.res = dx_res; g.ldr = ld_res;
        TRK("train.simt_gemm", CAT_TENSOR, simt_gemm(g, s));
    }
    return 0;
}

// ---- forward -------------------------------------------------------------------------------------
// Refusals that depend on the loaded weights and the shapes: checked before any workspace is resized.
int train_check_shapes(mrd_ctx* c, int B, int S) {
    if (!(c->has_cnn && c->has_text && c->has_fusion && c->has_head)) {
        set_last_error("training step needs cnn_encoder, text_encoder, fusion and classifier weights");
        return -3;
    }
    if (S > 512 || S <= 0 || S > c->max_pos) {
        set_last_error("training step: sequence length %d unsupported (1..%d)", S, c->max_pos < 512 ? c->max_pos : 512);
        return -1;
    }
    if (B > c->img_chunk || 1LL * B * S > c->tok_chunk) {
        set_last_error("training step: batch %d x %d tokens exceeds one pass (%d images, %d tokens)", B, S,
                       c->img_chunk, c->tok_chunk);
        return -1;
    }
    if (c->head_act != MRD_ACT_RELU) {
        set_last_error("training step: classifier activation must be relu");
        return -1;
    }
    return 0;
}

// Refusals that depend on the mode: fp32 check, batch-statistics BatchNorm, the layer4 map, a saving forward.
int train_check_mode(mrd_ctx* c, int img_dtype, const float* feat_map, bool save) {
    const TrainOpts& o = c->train->o;
    if (save && (c->fp32_check || o.bn_train || feat_map)) {
        set_last_error("data gradients: need the bf16 path (no fp32 check) and the backbone's BatchNorm on running "
                       "statistics (train.bn_train = 0); the layer4 map is block output 15");
        return -1;
    }
    if (c->fp32_check) {
        if (o.p_bert_hidden != 0.0 || o.p_bert_attn != 0.0 || o.p_text_out != 0.0 || o.p_cnn_proj != 0.0 ||
            o.p_fusion != 0.0 || o.p_head != 0.0) {
            set_last_error("fp32 check (train): every dropout probability must be 0 (the check compares with the "
                           "reference's autograd, whose Philox masks cannot be reproduced)");
            return -1;
        }
        if (o.bn_train) {
            set_last_error("fp32 check (train): the frozen backbone must be in eval mode (running statistics)");
            return -1;
        }
        return fp32_images_only(img_dtype);
    }
    if (o.bn_train && feat_map) {
        set_last_error("training step: the layer4 feature map is exported with the backbone in eval mode only");
        return -1;
    }
    return 0;
}

// Image branch: the frozen backbone (forward only; fp32 check, batch-statistics BatchNorm, saving forward for data
// gradients, or the eval forward) into t->pooled, then the trainable projection in fp32 into t->img.
int train_forward_image(mrd_ctx* c, const void* images, int img_dtype, int B, int H, int W, float* feat_map, bool save,
                        float* const* block_out, cudaStream_t s) {
    TrainState* t = c->train;
    const TrainOpts& o = t->o;
    if (c->fp32_check) {
        ++c->launches;
        MRD_TRY(fp32_cnn_encoder(c->raw, c->f32_opts(), &c->f32_ws, static_cast<const float*>(images), B, H, W, t->g4,
                                 t->pooled, feat_map, s));
    } else if (o.bn_train) {
        MRD_TRY(run_backbone_train(c, images, img_dtype, B, H, W, t->pooled, s));
    } else if (save) {
        MRD_TRY(run_backbone_save(c, images, img_dtype, B, H, W, t->pooled, block_out, s));
    } else {
        MRD_TRY(run_backbone(c, images, img_dtype, B, H, W, t->pooled, feat_map, s));
    }
    MRD_TRY(lin_fwd(c, "cnn_encoder.projection.0", t->pooled, c->feat_dim, B, t->a1, c->proj1.out, MRD_ACT_NONE,
                    nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, relu_dropout_f32(t->a1, B, c->proj1.out, make_drop(t->seed, SITE_CNN_PROJ, o.p_cnn_proj), t->p1, s));
    MRD_TRY(lin_fwd(c, "cnn_encoder.projection.3", t->p1, c->proj1.out, B, t->img, c->proj2.out, MRD_ACT_NONE,
                    nullptr, 0, s));
    return 0;
}

// Text branch: BERT with every activation the backward needs kept (plain fp32 in the fp32 check), its CLS row
// (src/text_encoder.py:118) into t->cls, then TextEncoder.dropout into t->txt.
int train_forward_text(mrd_ctx* c, const long long* ids, const void* mask, int mask_dtype, int B, int S,
                       cudaStream_t s) {
    TrainState* t = c->train;
    const TrainOpts& o = t->o;
    const unsigned long long seed = t->seed;
    const int Hd = c->hidden, F = c->ffn, T = B * S;
    if (c->fp32_check) {
        ++c->launches;
        MRD_TRY(fp32_bert_train_forward(c->raw, c->f32_opts(), &c->f32_train, ids, mask, mask_dtype, B, S, t->cls, s));
    } else {
        TRK("train.compact_tokens", CAT_MEM, compact_tokens(mask, mask_dtype, B, S, 0, c->t_seq_off, c->t_row_tok, c->t_bias, c->t_nrows,
                               c->t_scratch, s));
        TRK("train.embed_ln", CAT_MEM, bert_embed_layernorm(ids, B, S, c->word_emb, c->pos_type, c->emb_g, c->emb_b, c->bert_ln_eps, c->vocab,
                                     t->L[0].x, s, c->t_row_tok, c->t_nrows));
        TRK("train.dropout", CAT_MEM, dropout_bf16(t->L[0].x, Hd, T, Hd, c->t_nrows, make_drop(seed, SITE_EMB, o.p_bert_hidden), t->L[0].x,
                             Hd, s));
        const size_t nl = c->layers.size();
        for (size_t i = 0; i < nl; ++i) {
            const BertLayerW& Lw = c->layers[i];
            const TrainLayerBuf& b = t->L[i];
            TrainLayerPlan& p = t->P[i];
            bf16* x_next = i + 1 < nl ? t->L[i + 1].x : t->x_final;
            MRD_TRY(run(c, "train.qkv", p.qkv, s));
            const DropCfg da = make_drop(seed, site_attn(i), o.p_bert_attn);
            TRK("train.attention", CAT_ATTN, attention_forward(b.qkv, c->t_bias, c->t_seq_off, B, S, c->bert_heads, b.ctx, s, T, 0, &da));
            MRD_TRY(run(c, "train.attn_out", p.o, s));
            TRK("train.drop_add_ln", CAT_MEM, drop_add_ln_fwd(t->z, b.x, T, Hd, c->t_nrows, make_drop(seed, site_attn_out(i), o.p_bert_hidden),
                                    Lw.ln1g, Lw.ln1b, c->bert_ln_eps, b.s1, b.h1, s));
            MRD_TRY(run(c, "train.ffn1", p.f1, s));
            TRK("train.gelu", CAT_MEM, gelu_fwd_bf16(b.u, T, F, c->t_nrows, b.g, s));
            MRD_TRY(run(c, "train.ffn2", p.f2, s));
            TRK("train.drop_add_ln", CAT_MEM, drop_add_ln_fwd(t->z, b.h1, T, Hd, c->t_nrows, make_drop(seed, site_ffn_out(i), o.p_bert_hidden),
                                    Lw.ln2g, Lw.ln2b, c->bert_ln_eps, b.s2, x_next, s));
        }
        TRK("train.cls", CAT_MEM, gather_cls_rows_f32(t->x_final, c->t_seq_off, B, Hd, t->cls, s));
    }
    TRK("train.dropout", CAT_MEM, dropout_f32(t->cls, B, Hd, make_drop(seed, SITE_TEXT_OUT, o.p_text_out), t->txt, s));
    return 0;
}

// Fusion (src/fusion_model.py:245-291 in train mode) and head (src/multimodal_classifier.py:73-83) on t->img, t->txt.
int train_forward_tail(mrd_ctx* c, int B, float* logits, cudaStream_t s) {
    TrainState* t = c->train;
    const TrainOpts& o = t->o;
    const unsigned long long seed = t->seed;
    const int Fd = c->fusion_dim;
    const std::string f = "fusion.fusion_layer.";
    const int hd = Fd / c->fusion_heads;
    MRD_TRY(lin_fwd(c, f + "image_proj", t->img, c->fusion_img_in, B, t->ip, Fd, MRD_ACT_NONE, nullptr, 0, s));
    MRD_TRY(lin_fwd(c, f + "text_proj", t->txt, c->fusion_txt_in, B, t->tp, Fd, MRD_ACT_NONE, nullptr, 0, s));
    MRD_TRY(lin_fwd(c, f + "image_to_text_attention.value_proj", t->tp, Fd, B, t->v1, Fd, MRD_ACT_NONE, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, head_dropout_f32(t->v1, B, c->fusion_heads, hd, make_drop(seed, SITE_I2T, o.p_fusion), t->v1d, nullptr, s));
    MRD_TRY(lin_fwd(c, f + "image_to_text_attention.output_proj", t->v1d, Fd, B, t->pre_i, Fd, MRD_ACT_NONE,
                    c->fusion_residual ? t->ip : nullptr, Fd, s));
    MRD_TRY(lin_fwd(c, f + "text_to_image_attention.value_proj", t->ip, Fd, B, t->v2, Fd, MRD_ACT_NONE, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, head_dropout_f32(t->v2, B, c->fusion_heads, hd, make_drop(seed, SITE_T2I, o.p_fusion), t->v2d, nullptr, s));
    MRD_TRY(lin_fwd(c, f + "text_to_image_attention.output_proj", t->v2d, Fd, B, t->pre_t, Fd, MRD_ACT_NONE,
                    c->fusion_residual ? t->tp : nullptr, Fd, s));
    TRK("train.ln_f32", CAT_MEM, ln_fwd_f32(t->pre_i, Fd, c->ln_i_g, c->ln_i_b, c->fusion_ln_eps, B, Fd, t->cat, 2 * Fd, s));
    TRK("train.ln_f32", CAT_MEM, ln_fwd_f32(t->pre_t, Fd, c->ln_t_g, c->ln_t_b, c->fusion_ln_eps, B, Fd, t->cat + Fd, 2 * Fd, s));
    MRD_TRY(lin_fwd(c, f + "fusion.0", t->cat, 2 * Fd, B, t->g0, Fd, MRD_ACT_NONE, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, relu_dropout_f32(t->g0, B, Fd, make_drop(seed, SITE_FUSION_MLP, o.p_fusion), t->fh, s));
    MRD_TRY(lin_fwd(c, f + "fusion.3", t->fh, Fd, B, t->fused, Fd, MRD_ACT_NONE, nullptr, 0, s));

    const float* x = t->fused;
    int ld = c->head_in;
    for (size_t j = 0; j < c->head_hidden.size(); ++j) {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%zu", 3 * j);
        const int n = c->head_hidden[j].out;
        MRD_TRY(lin_fwd(c, nm, x, ld, B, t->g0, n, MRD_ACT_NONE, nullptr, 0, s));
        TRK("train.dropout", CAT_MEM, relu_dropout_f32(t->g0, B, n, make_drop(seed, SITE_HEAD + static_cast<unsigned>(j), o.p_head), t->hh[j], s));
        x = t->hh[j];
        ld = n;
    }
    char nm[64];
    snprintf(nm, sizeof(nm), "classifier.classifier.%zu", 3 * c->head_hidden.size());
    return lin_fwd(c, nm, x, ld, B, logits, c->num_classes, MRD_ACT_NONE, nullptr, 0, s);
}

// The training forward.  save: keep what the backbone's data-gradient backward needs (dgrad_backbone), and write the
// output of bottleneck k into block_out[k] where that slot is given.  In the fp32 check the backbone and BERT run in
// plain fp32 (fp32_check.cu) with dropout off; the batch-level layers are fp32 in either mode.
int train_forward(mrd_ctx* c, const void* images, int img_dtype, const long long* ids, const void* mask,
                  int mask_dtype, int B, int H, int W, int S, unsigned long long seed, float* logits,
                  float* feat_map, bool save, float* const* block_out, cudaStream_t s) {
    TrainState* t = train_state(c);
    MRD_TRY(train_check_shapes(c, B, S));
    MRD_TRY(ensure_batch_ws(c, B));
    MRD_TRY(ensure_text_ws(c, B * S, B));
    MRD_TRY(train_ensure_packs(c, s));
    MRD_TRY(train_ensure_plan(c, B, S));
    t->fwd_done = false;
    t->seed = seed;
    t->ids = ids;
    dgrad_forget(t);   // a saving forward re-validates its activations
    MRD_TRY(train_check_mode(c, img_dtype, feat_map, save));
    MRD_TRY(train_forward_image(c, images, img_dtype, B, H, W, feat_map, save, block_out, s));
    MRD_TRY(train_forward_text(c, ids, mask, mask_dtype, B, S, s));
    MRD_TRY(train_forward_tail(c, B, logits, s));
    t->fwd_done = true;
    t->text_run_epoch = c->text_run_epoch;
    return 0;
}

// image / text / fused embeddings of the pending forward (fp32 activations of the batch-level layers)
int train_export_embeddings(mrd_ctx* c, int B, float* img_emb, float* txt_emb, float* fused, cudaStream_t s) {
    TrainState* t = train_state(c);
    const struct { float* dst; const float* src; int w; } out[3] = {
        {img_emb, t->img, c->proj2.out}, {txt_emb, t->txt, c->hidden}, {fused, t->fused, c->fusion_dim}};
    for (const auto& o : out) {
        if (!o.dst) continue;
        cudaError_t e = cudaMemcpyAsync(o.dst, o.src, sizeof(float) * static_cast<size_t>(B) * o.w,
                                        cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(embedding export)");
    }
    return 0;
}

// dW = dY^T X through the tcgen05 GEMM: stage both operands token-minor (the bias gradient = column sums of dY
// is taken by the same staging kernel), fp32 result into `dst`.  Either destination may be null.
int train_wgrad(mrd_ctx* c, TrainState* t, const GemmLaunch& plan, const bf16* dY, int n_out, const bf16* X, int n_in,
                float* dst, float* bias_dst, cudaStream_t s) {
    if (!dst) {
        if (bias_dst) TRK("train.colsum", CAT_MEM, colsum_bf16(dY, n_out, t->Ta, n_out, c->t_nrows, 1.0f, bias_dst, s));
        return 0;
    }
    TRK("train.transpose", CAT_MEM, transpose_pad2_bf16(dY, n_out, n_out, t->At, X, n_in, n_in, t->Bt, t->Ta, c->t_nrows,
                                                        t->Tp, s, bias_dst));
    return run_f32(c, "train.wgrad", plan, dst, n_in, s);
}

// The backward is cut into stages so that a data-parallel host can start the all-reduce of a gradient bucket as
// soon as the stage that completes it has been enqueued (SURVEY.md 8(e): bucketed, overlapped with backward):
//   stage 0                head, fusion, image projection, TextEncoder.dropout, CLS scatter
//   stage 1 + k            BERT layer (layers-1-k), k = 0 .. layers-1  (reverse order)
//   stage layers + 1       embeddings
int train_backward_stages(mrd_ctx* c) { return static_cast<int>(c->layers.size()) + 2; }

int train_backward_begin(mrd_ctx* c, const float* dlogits, const GradTable& gt, float* d_pooled) {
    TrainState* t = train_state(c);
    t->bw_active = false;
    if (!t->fwd_done) {
        set_last_error("mrd_train_backward: no forward is pending on this context");
        return -1;
    }
    t->fwd_done = false;
    if (t->text_run_epoch != c->text_run_epoch) {
        set_last_error("mrd_train_backward: another forward ran on this context after mrd_train_forward (the "
                       "token-packing tables it saved were overwritten)");
        return -1;
    }
    t->bw_dlogits = dlogits;
    t->bw_grads = gt;
    t->bw_d_pooled = d_pooled;
    t->bw_want_text = false;
    for (const auto& kv : gt) t->bw_want_text |= kv.first.rfind("text_encoder.", 0) == 0;
    t->bw_next = 0;
    t->bw_active = true;
    return 0;
}

// ---- stage 0: head, fusion, image projection, TextEncoder.dropout, CLS scatter
// Head (src/multimodal_classifier.py:73-83): dlogits -> *d_fused [B, head_in], one of the ping-pong buffers g1 / g2.
int bw_head(mrd_ctx* c, TrainState* t, float** d_fused, cudaStream_t s) {
    const GradTable& gt = t->bw_grads;
    const TrainOpts& o = t->o;
    const int B = t->B;
    const size_t nh = c->head_hidden.size();
    {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%zu", 3 * nh);
        const float* x = nh ? t->hh[nh - 1] : t->fused;
        const int ldx = nh ? c->head_hidden[nh - 1].out : c->head_in;
        MRD_TRY(lin_bwd(c, gt, nm, x, ldx, t->bw_dlogits, c->num_classes, B, t->g1, ldx, nullptr, 0, s));
    }
    float* ping[2] = {t->g1, t->g2};
    int cur = 0;
    for (size_t jj = nh; jj-- > 0;) {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%zu", 3 * jj);
        const int n = c->head_hidden[jj].out;
        // ping[cur] is the gradient of the post-dropout activation hh[jj]
        TRK("train.dropout", CAT_MEM, dropout_f32(ping[cur], B, n, make_drop(t->seed, SITE_HEAD + static_cast<unsigned>(jj), o.p_head), t->g0, s));
        TRK("train.relu_bwd", CAT_MEM, relu_bwd_f32(t->hh[jj], t->g0, 1LL * B * n, t->g0, s));
        const float* x = jj ? t->hh[jj - 1] : t->fused;
        const int ldx = jj ? c->head_hidden[jj - 1].out : c->head_in;
        MRD_TRY(lin_bwd(c, gt, nm, x, ldx, t->g0, n, B, ping[cur ^ 1], ldx, nullptr, 0, s));
        cur ^= 1;
    }
    *d_fused = ping[cur];
    return 0;
}

// Fusion (src/fusion_model.py:245-291): d(fused) -> d(image embedding) in g1, d(text embedding) in g2.
int bw_fusion(mrd_ctx* c, TrainState* t, const float* d_fused, cudaStream_t s) {
    const GradTable& gt = t->bw_grads;
    const TrainOpts& o = t->o;
    const unsigned long long seed = t->seed;
    const int B = t->B, Fd = c->fusion_dim, hd = Fd / c->fusion_heads;
    const std::string f = "fusion.fusion_layer.";
    float* d_fh = d_fused == t->g1 ? t->g2 : t->g1;   // the head's other ping-pong buffer
    MRD_TRY(lin_bwd(c, gt, f + "fusion.3", t->fh, Fd, d_fused, c->head_in, B, d_fh, Fd, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, dropout_f32(d_fh, B, Fd, make_drop(seed, SITE_FUSION_MLP, o.p_fusion), t->g0, s));
    TRK("train.relu_bwd", CAT_MEM, relu_bwd_f32(t->fh, t->g0, 1LL * B * Fd, t->g0, s));
    float* d_cat = t->g3;  // [B, 2*Fd]
    MRD_TRY(lin_bwd(c, gt, f + "fusion.0", t->cat, 2 * Fd, t->g0, Fd, B, d_cat, 2 * Fd, nullptr, 0, s));
    float* d_pre_i = t->g1;
    float* d_pre_t = t->g2;
    TRK("train.ln_f32", CAT_MEM, ln_bwd_f32(t->pre_i, Fd, d_cat, 2 * Fd, c->ln_i_g, c->fusion_ln_eps, B, Fd, d_pre_i, Fd,
                       grad_of(gt, f + "layer_norm_image.weight"), grad_of(gt, f + "layer_norm_image.bias"), s));
    TRK("train.ln_f32", CAT_MEM, ln_bwd_f32(t->pre_t, Fd, d_cat + Fd, 2 * Fd, c->ln_t_g, c->fusion_ln_eps, B, Fd, d_pre_t, Fd,
                       grad_of(gt, f + "layer_norm_text.weight"), grad_of(gt, f + "layer_norm_text.bias"), s));
    // pre_i = ip + O1(headdrop(V1(tp)));  pre_t = tp + O2(headdrop(V2(ip)))
    float* d_v = t->g0;      // gradient of the dropped value vector, then of the value vector
    float* d_ip = t->g3;     // d_cat is dead after the two LayerNorm backwards
    float* d_tp = t->g4;
    MRD_TRY(lin_bwd(c, gt, f + "image_to_text_attention.output_proj", t->v1d, Fd, d_pre_i, Fd, B, d_v, Fd, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, head_dropout_f32(d_v, B, c->fusion_heads, hd, make_drop(seed, SITE_I2T, o.p_fusion), d_v, nullptr, s));
    MRD_TRY(lin_bwd(c, gt, f + "image_to_text_attention.value_proj", t->tp, Fd, d_v, Fd, B, d_tp, Fd,
                    c->fusion_residual ? d_pre_t : nullptr, Fd, s));
    MRD_TRY(lin_bwd(c, gt, f + "text_to_image_attention.output_proj", t->v2d, Fd, d_pre_t, Fd, B, d_v, Fd, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, head_dropout_f32(d_v, B, c->fusion_heads, hd, make_drop(seed, SITE_T2I, o.p_fusion), d_v, nullptr, s));
    MRD_TRY(lin_bwd(c, gt, f + "text_to_image_attention.value_proj", t->ip, Fd, d_v, Fd, B, d_ip, Fd,
                    c->fusion_residual ? d_pre_i : nullptr, Fd, s));
    // d_pre_i / d_pre_t are dead now
    MRD_TRY(lin_bwd(c, gt, f + "image_proj", t->img, c->fusion_img_in, d_ip, Fd, B, t->g1, c->fusion_img_in, nullptr, 0, s));
    MRD_TRY(lin_bwd(c, gt, f + "text_proj", t->txt, c->fusion_txt_in, d_tp, Fd, B, t->g2, c->fusion_txt_in, nullptr, 0, s));
    return 0;
}

// Image projection (the backbone below it is frozen): d(image embedding) -> optional d_pooled, the gradient of the
// backbone's pooled output - what Grad-CAM spreads over the layer4 map.
int bw_image_projection(mrd_ctx* c, TrainState* t, const float* d_img, cudaStream_t s) {
    const GradTable& gt = t->bw_grads;
    const int B = t->B;
    MRD_TRY(lin_bwd(c, gt, "cnn_encoder.projection.3", t->p1, c->proj1.out, d_img, c->proj2.out, B, t->g0,
                    c->proj1.out, nullptr, 0, s));
    TRK("train.dropout", CAT_MEM, dropout_f32(t->g0, B, c->proj1.out, make_drop(t->seed, SITE_CNN_PROJ, t->o.p_cnn_proj), t->g0, s));
    TRK("train.relu_bwd", CAT_MEM, relu_bwd_f32(t->p1, t->g0, 1LL * B * c->proj1.out, t->g0, s));
    return lin_bwd(c, gt, "cnn_encoder.projection.0", t->pooled, c->feat_dim, t->g0, c->proj1.out, B, t->bw_d_pooled,
                   c->feat_dim, nullptr, 0, s);
}

int bw_batch_layers(mrd_ctx* c, TrainState* t, cudaStream_t s) {
    float* d_fused = nullptr;
    MRD_TRY(bw_head(c, t, &d_fused, s));
    MRD_TRY(bw_fusion(c, t, d_fused, s));
    MRD_TRY(bw_image_projection(c, t, t->g1, s));
    if (!t->bw_want_text) return 0;   // nothing below the text embedding is differentiated (frozen text encoder)

    // ---- TextEncoder.dropout, then the CLS scatter into the input gradient of the top BERT layer
    const int B = t->B, Hd = c->hidden;
    float* d_txt = t->g2;
    TRK("train.dropout", CAT_MEM, dropout_f32(d_txt, B, Hd, make_drop(t->seed, SITE_TEXT_OUT, t->o.p_text_out), d_txt, s));
    if (c->fp32_check) {
        ++c->launches;
        return fp32_bert_train_backward(c->raw, c->f32_opts(), &c->f32_train, d_txt, t->bw_grads, t->o.pad_idx, s);
    }
    bf16* dx_top = (c->layers.size() & 1) ? t->dxb : t->dxa;   // layer nl-1 reads dx[nl & 1]
    cudaError_t e = cudaMemsetAsync(dx_top, 0, sizeof(bf16) * static_cast<size_t>(t->Ta) * Hd, s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(dX)");
    TRK("train.cls", CAT_MEM, scatter_cls_rows_bf16(d_txt, c->t_seq_off, B, Hd, dx_top, s));
    return 0;
}

// ---- stages 1 .. layers: one BERT layer each, in reverse
// QKV weight gradient of layer input x: one [3*Hd, Hd] product into zeroed scratch, split into the three parameters.
// The query block carries the folded 1/sqrt(64): d/dWq = 0.125 * d/dWq'.
int bw_qkv_wgrad(mrd_ctx* c, TrainState* t, const bf16* x, const std::string& pre, cudaStream_t s) {
    const GradTable& gt = t->bw_grads;
    const int Hd = c->hidden;
    const std::string sa = pre + "attention.self.";
    struct Part {
        float* scratch;
        long long n;       // elements per parameter
        float* dst[3];     // query, key, value
        bool want() const { return dst[0] || dst[1] || dst[2]; }
    };
    const Part parts[2] = {
        {t->wq_scratch, 1LL * Hd * Hd,
         {grad_of(gt, sa + "query.weight"), grad_of(gt, sa + "key.weight"), grad_of(gt, sa + "value.weight")}},
        {t->bq_scratch, Hd, {grad_of(gt, sa + "query.bias"), grad_of(gt, sa + "key.bias"), grad_of(gt, sa + "value.bias")}}};
    if (!parts[0].want() && !parts[1].want()) return 0;
    for (const Part& p : parts) {
        if (!p.want()) continue;
        cudaError_t e = cudaMemsetAsync(p.scratch, 0, sizeof(float) * 3 * static_cast<size_t>(p.n), s);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(QKV gradient scratch)");
    }
    MRD_TRY(train_wgrad(c, t, t->w_qkv, t->dqkv, 3 * Hd, x, Hd, parts[0].want() ? t->wq_scratch : nullptr,
                        parts[1].want() ? t->bq_scratch : nullptr, s));
    for (const Part& p : parts) {
        if (p.dst[0]) TRK("train.scale", CAT_MEM, scale_f32(p.scratch, p.n, 0.125f, s));
        for (int k = 0; k < 3; ++k) {
            if (!p.dst[k]) continue;
            cudaError_t e = cudaMemcpyAsync(p.dst[k], p.scratch + k * p.n, sizeof(float) * static_cast<size_t>(p.n),
                                            cudaMemcpyDeviceToDevice, s);
            if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpyAsync(QKV gradient split)");
        }
    }
    return 0;
}

// Layer i reads its output gradient from dx[(i+1)&1] and writes its input gradient to dx[i&1] (the d_x plan).
int bw_bert_layer(mrd_ctx* c, TrainState* t, size_t i, cudaStream_t s) {
    const GradTable& gt = t->bw_grads;
    const TrainOpts& o = t->o;
    const unsigned long long seed = t->seed;
    const int B = t->B, S = t->S, T = t->Ta, Hd = c->hidden, F = c->ffn;
    const BertLayerW& Lw = c->layers[i];
    const TrainLayerBuf& b = t->L[i];
    TrainLayerPlan& p = t->P[i];
    const std::string pre = "text_encoder.encoder.encoder.layer." + std::to_string(i) + ".";
    const bf16* dx_in = ((i + 1) & 1) ? t->dxb : t->dxa;
    const DropCfg d_ffn = make_drop(seed, site_ffn_out(i), o.p_bert_hidden);
    const DropCfg d_att = make_drop(seed, site_attn_out(i), o.p_bert_hidden);
    // x_{i+1} = LN2(s2), s2 = h1 + drop(W2 g + b2)
    TRK("train.ln_bwd", CAT_MEM, ln_bwd_bf16(b.s2, dx_in, Lw.ln2g, c->bert_ln_eps, T, Hd, c->t_nrows, t->d_s,
                        grad_of(gt, pre + "output.LayerNorm.weight"), grad_of(gt, pre + "output.LayerNorm.bias"), s));
    const bf16* dz = t->d_s;
    if (d_ffn.thresh) {
        TRK("train.dropout", CAT_MEM, dropout_bf16(t->d_s, Hd, T, Hd, c->t_nrows, d_ffn, t->dz, Hd, s));
        dz = t->dz;
    }
    MRD_TRY(train_wgrad(c, t, t->w_f2, dz, Hd, b.g, F, grad_of(gt, pre + "output.dense.weight"),
                        grad_of(gt, pre + "output.dense.bias"), s));
    MRD_TRY(run(c, "train.dgrad", dz == t->dz ? p.d_g : p.d_g0, s));
    TRK("train.gelu_bwd", CAT_MEM, gelu_bwd_bf16(b.u, t->dbig, T, F, c->t_nrows, t->dbig, s));
    MRD_TRY(train_wgrad(c, t, t->w_f1, t->dbig, F, b.h1, Hd, grad_of(gt, pre + "intermediate.dense.weight"),
                        grad_of(gt, pre + "intermediate.dense.bias"), s));
    MRD_TRY(run(c, "train.dgrad", p.d_h1, s));   // dh1 = du W1 + d_s2
    // h1 = LN1(s1), s1 = x + drop(Wo ctx + bo)
    TRK("train.ln_bwd", CAT_MEM, ln_bwd_bf16(b.s1, t->dh1, Lw.ln1g, c->bert_ln_eps, T, Hd, c->t_nrows, t->d_s,
                        grad_of(gt, pre + "attention.output.LayerNorm.weight"),
                        grad_of(gt, pre + "attention.output.LayerNorm.bias"), s));
    dz = t->d_s;
    if (d_att.thresh) {
        TRK("train.dropout", CAT_MEM, dropout_bf16(t->d_s, Hd, T, Hd, c->t_nrows, d_att, t->dz, Hd, s));
        dz = t->dz;
    }
    MRD_TRY(train_wgrad(c, t, t->w_o, dz, Hd, b.ctx, Hd, grad_of(gt, pre + "attention.output.dense.weight"),
                        grad_of(gt, pre + "attention.output.dense.bias"), s));
    MRD_TRY(run(c, "train.dgrad", dz == t->dz ? p.d_ctx : p.d_ctx0, s));
    if (t->dkv_acc) {
        cudaError_t e = cudaMemsetAsync(t->dkv_acc, 0, sizeof(float) * static_cast<size_t>(T) * 2 * Hd, s);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(dK/dV accumulator)");
    }
    TRK("train.attention_bwd", CAT_ATTN, attention_backward(b.qkv, b.ctx, t->dctx, c->t_bias, c->t_seq_off, B, S, c->bert_heads,
                               make_drop(seed, site_attn(i), o.p_bert_attn), t->dqkv, s, t->dkv_acc));
    if (t->dkv_acc)   // fp32 dK | dV accumulators -> the K / V columns of dqkv
        TRK("train.attention_bwd", CAT_MEM, cast_f32_to_bf16(t->dkv_acc, 2 * Hd, T, 2 * Hd, t->dqkv + Hd, 3 * Hd, s));
    MRD_TRY(bw_qkv_wgrad(c, t, b.x, pre, s));
    return run(c, "train.dgrad", p.d_x, s);    // dx_i = dqkv Wqkv + d_s1
}

// ---- stage layers + 1: embeddings: dropout, LayerNorm backward, scatter-add into the three tables
int bw_embeddings(mrd_ctx* c, TrainState* t, cudaStream_t s) {
    const GradTable& gt = t->bw_grads;
    const int T = t->Ta, Hd = c->hidden;
    bf16* dx0 = t->dxa;   // layer 0 wrote dx[0]
    TRK("train.dropout", CAT_MEM, dropout_bf16(dx0, Hd, T, Hd, c->t_nrows, make_drop(t->seed, SITE_EMB, t->o.p_bert_hidden), dx0, Hd, s));
    const std::string em = "text_encoder.encoder.embeddings.";
    float* g_word = grad_of(gt, em + "word_embeddings.weight");
    float* g_pos = grad_of(gt, em + "position_embeddings.weight");
    float* g_type = grad_of(gt, em + "token_type_embeddings.weight");
    float* g_lg = grad_of(gt, em + "LayerNorm.weight");
    float* g_lb = grad_of(gt, em + "LayerNorm.bias");
    if (g_word || g_pos || g_type || g_lg || g_lb)
        TRK("train.embed_bwd", CAT_MEM, embed_ln_bwd(t->ids, c->t_row_tok, T, c->t_nrows, t->S, c->word_emb, c->pos_type, c->emb_g,
                             c->bert_ln_eps, c->vocab, t->o.pad_idx, dx0, g_word, g_pos, g_type, g_lg, g_lb, s));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "training backward");
    return 0;
}

// Runs stages [lo, hi) of the pending backward; stages must be run in order, each exactly once.  Without a text
// encoder gradient, and in the fp32 check, stage 0 does everything there is to do and the later stages are no-ops.
int train_backward_run(mrd_ctx* c, int lo, int hi, cudaStream_t s) {
    TrainState* t = train_state(c);
    const int n_stages = train_backward_stages(c);
    if (!t->bw_active || lo != t->bw_next || hi <= lo || hi > n_stages) {
        set_last_error("mrd_train_backward_stage: stages [%d, %d) out of order (next %d of %d, %s)", lo, hi,
                       t->bw_next, n_stages, t->bw_active ? "active" : "no backward begun");
        return -1;
    }
    t->bw_next = hi;
    if (hi == n_stages) t->bw_active = false;
    const int nl = n_stages - 2;
    for (int st = lo; st < hi; ++st) {
        if (st == 0) MRD_TRY(bw_batch_layers(c, t, s));
        else if (!t->bw_want_text || c->fp32_check) break;
        else if (st <= nl) MRD_TRY(bw_bert_layer(c, t, static_cast<size_t>(nl - st), s));
        else MRD_TRY(bw_embeddings(c, t, s));
    }
    return 0;
}

int train_backward(mrd_ctx* c, const float* dlogits, const GradTable& gt, float* d_pooled, cudaStream_t s) {
    MRD_TRY(train_backward_begin(c, dlogits, gt, d_pooled));
    return train_backward_run(c, 0, train_backward_stages(c), s);
}
