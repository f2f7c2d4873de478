// Data gradients through the frozen ResNet50 backbone: input saliency (images.grad) and forward / backward hooks on
// every stage and bottleneck (Grad-CAM below layer4).  Included by engine.cu after engine_train.cuh, inside its
// anonymous namespace; the C ABI wrappers are at the end of engine.cu.
//
// Forward ("saving forward", only when data gradients are requested): the eval-BatchNorm backbone with every ReLU
// output the backward needs kept, bf16 NHWC, in an arena sized for the batch:
//   stem output before the max-pool, the max-pool output, and per bottleneck a1 = relu(bn1(conv1 x)),
//   a2 = relu(bn2(conv2 a1)) and the block output.
// At 224 x 224 that is 9,809,408 elements = 19.6 MB per image (stem 802,816, pool 200,704, blocks 8,805,888); the
// backward's scratch (two block-gradient buffers, the masked gradient, d_a1, d_a2 and the stem gradient) adds
// 3,813,376 elements = 7.6 MB.  The launches are those of the training step's eval backbone (plan_stem, the max-pool
// kernel, plan_conv, plan_conv1x1_dual) without the layer1 chain and the flat-shift 3x3 mode, which do not keep
// a1 / a2 (the flat mode writes a1 into a zero-bordered buffer and the chain never writes it).
//
// Backward, from d_pooled (the training step's backward) down to the lowest tensor anything asks for.  g = d/d(block
// output), gz = g * [out > 0]; per block, on the tcgen05 GEMM (plan_conv_dgrad):
//   d_a2 = conv3^T gz * [a2 > 0]                       1x1, ReLU-mask epilogue
//   d_a1 = conv2^T d_a2 * [a1 > 0]                     3x3: flipped filter (stride 1) or four parity phases (stride 2)
//   g_in = conv1^T d_a1 + gz                           identity block: residual epilogue
//   g_in = conv1^T d_a1, then += downsample^T gz       at the even pixels of a stride-2 view, in place
// then max-pool backward fused with the stem ReLU mask, and the stem's data gradient to fp32 NCHW (CUDA cores).
// Samples are independent (BatchNorm on running statistics): a row of the batch never reads another row.

struct DgradBlockW {
    bf16 *c1t = nullptr, *c2t = nullptr, *c3t = nullptr, *dst = nullptr;   // [Cin][taps][Cout] (pack_dgrad_weights)
};
struct DgradBlock {
    bf16 *a1 = nullptr, *a2 = nullptr, *out = nullptr;
    int h = 0, w = 0, ho = 0, wo = 0;
    GemmLaunch f1, f2, f3;        // forward: conv1, conv2, conv3 (+ downsample + add)
    GemmLaunch b3, b1, bds;       // backward: conv3^T (masked), conv1^T (+ identity), downsample^T (scatter-add)
    GemmLaunch b2[4];             // conv2^T: one launch (stride 1) or one per parity phase (stride 2)
    int n_b2 = 0;
};
struct DgradCnn {
    bool packed = false;
    std::vector<DgradBlockW> wt;
    float* stem_wf = nullptr;     // [7][7][64][3] fp32, BatchNorm folded (pack_stem_dgrad)
    mrd_ctx::Arena ws;
    int B = 0, H = 0, W = 0;
    long long cnn_epoch = -1;     // c->cnn_ws_epoch the stem plan was built against (it reads c->xpad)
    bf16 *stem_out = nullptr, *pool_out = nullptr, *gz = nullptr, *da1 = nullptr, *da2 = nullptr, *dstem = nullptr;
    bf16* g[2] = {nullptr, nullptr};
    float* d_pooled = nullptr;
    GemmLaunch stem;
    std::vector<DgradBlock> blk;
    bool valid = false;           // the pending training forward was a saving forward of this plan
};

// images per saving forward: the training step's batch limit (27 MB of arena per 224 x 224 image)
constexpr int kDgradMaxBatch = 512;

// stride-2 conv2 data gradient: taps of the four output parity phases (ph, pw), in pack order
struct PhaseTaps {
    int n, first;                 // taps, index of the first one in the pack
    TapDesc t[4];
};
const int kS2Order[9] = {4, 5, 3, 7, 1, 8, 6, 2, 0};   // forward tap (kh*3 + kw) of each pack slot
const PhaseTaps kS2Phase[4] = {
    {1, 0, {{0, 0, 0, 0}}},                                             // even row, even column: (1,1)
    {2, 1, {{0, 0, 0, 0}, {0, 0, 1, 0}}},                               // even, odd: (1,2) (1,0)
    {2, 3, {{0, 0, 0, 0}, {0, 1, 0, 0}}},                               // odd, even: (2,1) (0,1)
    {4, 5, {{0, 0, 0, 0}, {0, 0, 1, 0}, {0, 1, 0, 0}, {0, 1, 1, 0}}},   // odd, odd: (2,2) (2,0) (0,2) (0,0)
};

DgradCnn* dgrad_state(mrd_ctx* c) {
    TrainState* t = train_state(c);
    if (!t->dg) t->dg = new DgradCnn();
    return t->dg;
}

void dgrad_invalidate(TrainState* t) {
    if (t->dg) {
        t->dg->packed = false;
        t->dg->valid = false;
    }
}
void dgrad_forget(TrainState* t) {
    if (t->dg) t->dg->valid = false;
}
void dgrad_free(TrainState* t) {
    if (!t->dg) return;
    if (t->dg->ws.base) cudaFree(t->dg->ws.base);
    delete t->dg;   // packed weights are weight allocations of the context (freed with it)
    t->dg = nullptr;
}

int dgrad_pack(mrd_ctx* c, cudaStream_t s) {
    DgradCnn* d = dgrad_state(c);
    if (d->packed) return 0;
    const std::string bb = "cnn_encoder.backbone.";
    const RawTensor *w, *g, *v;
    MRD_TRY(raw_need(c, bb + "conv1.weight", &w));
    MRD_TRY(raw_need(c, bb + "bn1.weight", &g));
    MRD_TRY(raw_need(c, bb + "bn1.running_var", &v));
    MRD_TRY(walloc(c, &d->stem_wf, 7 * 7 * 64 * 3));
    TRK("dgrad.pack", CAT_MEM, pack_stem_dgrad(w->p, g->p, v->p, c->bn_eps, d->stem_wf, s));
    d->wt.resize(c->blocks.size());
    const TapList one = {1, {0}};
    TapList flip = {9, {0}}, s2 = {9, {0}};
    for (int t = 0; t < 9; ++t) {
        flip.tap[t] = 8 - t;
        s2.tap[t] = kS2Order[t];
    }
    for (size_t i = 0; i < c->blocks.size(); ++i) {
        const Bottleneck& b = c->blocks[i];
        DgradBlockW& o = d->wt[i];
        if (b.c1.k != 1 || b.c2.k != 3 || b.c3.k != 1 || b.c1.stride != 1 || (b.has_ds && b.ds.k != 1)) {
            set_last_error("data gradients: block %zu is not a ResNet50 bottleneck (1x1, 3x3, 1x1)", i);
            return -1;
        }
        MRD_TRY(walloc(c, &o.c1t, 1LL * b.c1.cin * b.c1.cout));
        MRD_TRY(walloc(c, &o.c2t, 9LL * b.c2.cin * b.c2.cout));
        MRD_TRY(walloc(c, &o.c3t, 1LL * b.c3.cin * b.c3.cout));
        TRK("dgrad.pack", CAT_MEM, pack_dgrad_weights(b.c1.w, b.c1.cout, b.c1.cin, 1, one, o.c1t, s));
        TRK("dgrad.pack", CAT_MEM, pack_dgrad_weights(b.c2.w, b.c2.cout, b.c2.cin, 9, b.c2.stride == 2 ? s2 : flip,
                                                      o.c2t, s));
        TRK("dgrad.pack", CAT_MEM, pack_dgrad_weights(b.c3.w, b.c3.cout, b.c3.cin, 1, one, o.c3t, s));
        if (b.has_ds) {
            MRD_TRY(walloc(c, &o.dst, 1LL * b.ds.cin * b.ds.cout));
            TRK("dgrad.pack", CAT_MEM, pack_dgrad_weights(b.ds.w, b.ds.cout, b.ds.cin, 1, one, o.dst, s));
        }
    }
    d->packed = true;
    d->B = 0;   // re-plan against the (possibly moved) filters
    return 0;
}

int dgrad_plan(mrd_ctx* c, int B, int H, int W) {
    DgradCnn* d = dgrad_state(c);
    if (d->B == B && d->H == H && d->W == W && d->cnn_epoch == c->cnn_ws_epoch) return 0;
    d->valid = false;
    const long long q = 1LL * (H / 4) * (W / 4);
    const long long n_stem = 1LL * B * (H / 2) * (W / 2) * 64;
    long long n_g = 1LL * B * q * 64, n_da1 = 0, n_da2 = 0;
    size_t total = 2 * pad1k(n_stem, 2) + pad1k(1LL * B * q * 64, 2) + pad1k(1LL * B * c->feat_dim, 4);
    d->blk.assign(c->blocks.size(), DgradBlock());
    {
        int h = H / 4, w = W / 4;
        for (size_t i = 0; i < c->blocks.size(); ++i) {
            const Bottleneck& b = c->blocks[i];
            DgradBlock& k = d->blk[i];
            if (h % b.c2.stride || w % b.c2.stride) {
                set_last_error("data gradients: feature map %dx%d not divisible by the stride of block %zu", h, w, i);
                return -1;
            }
            k.h = h; k.w = w; k.ho = h / b.c2.stride; k.wo = w / b.c2.stride;
            const long long n1 = 1LL * B * h * w * b.c1.cout, n2 = 1LL * B * k.ho * k.wo * b.c2.cout,
                            n3 = 1LL * B * k.ho * k.wo * b.c3.cout;
            total += pad1k(n1, 2) + pad1k(n2, 2) + pad1k(n3, 2);
            n_g = n3 > n_g ? n3 : n_g;
            n_da1 = n1 > n_da1 ? n1 : n_da1;
            n_da2 = n2 > n_da2 ? n2 : n_da2;
            h = k.ho;
            w = k.wo;
        }
    }
    total += 3 * pad1k(n_g, 2) + pad1k(n_da1, 2) + pad1k(n_da2, 2);
    MRD_TRY(arena_reset(c, &d->ws, total));
    d->stem_out = arena_take<bf16>(&d->ws, n_stem);
    d->dstem = arena_take<bf16>(&d->ws, n_stem);
    d->pool_out = arena_take<bf16>(&d->ws, 1LL * B * q * 64);
    d->d_pooled = arena_take<float>(&d->ws, 1LL * B * c->feat_dim);
    for (size_t i = 0; i < c->blocks.size(); ++i) {
        const Bottleneck& b = c->blocks[i];
        DgradBlock& k = d->blk[i];
        k.a1 = arena_take<bf16>(&d->ws, 1LL * B * k.h * k.w * b.c1.cout);
        k.a2 = arena_take<bf16>(&d->ws, 1LL * B * k.ho * k.wo * b.c2.cout);
        k.out = arena_take<bf16>(&d->ws, 1LL * B * k.ho * k.wo * b.c3.cout);
    }
    d->g[0] = arena_take<bf16>(&d->ws, n_g);
    d->g[1] = arena_take<bf16>(&d->ws, n_g);
    d->gz = arena_take<bf16>(&d->ws, n_g);
    d->da1 = arena_take<bf16>(&d->ws, n_da1);
    d->da2 = arena_take<bf16>(&d->ws, n_da2);

    MRD_TRY(plan_stem(&d->stem, c->xpad, B, H, W, c->stem_w, c->stem_b, d->stem_out, ACT_RELU));
    const TapDesc tap0[1] = {{0, 0, 0, 0}};
    TapDesc tap9[9];
    for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) tap9[r * 3 + s] = TapDesc{0, (int8_t)(r - 1), (int8_t)(s - 1), 0};
    const bf16* x = d->pool_out;
    for (size_t i = 0; i < c->blocks.size(); ++i) {
        const Bottleneck& b = c->blocks[i];
        const DgradBlockW& wt = d->wt[i];
        DgradBlock& k = d->blk[i];
        const int st = b.c2.stride;
        // ---- forward
        MRD_TRY(plan_conv(&k.f1, x, B, k.h, k.w, b.c1.cin, b.c1.w, b.c1.cout, 1, 1, b.c1.b, k.a1, nullptr, ACT_RELU));
        MRD_TRY(plan_conv(&k.f2, k.a1, B, k.h, k.w, b.c2.cin, b.c2.w, b.c2.cout, 3, st, b.c2.b, k.a2, nullptr,
                          ACT_RELU));
        if (b.has_ds) {
            if (!b.c3ds_w) {
                set_last_error("data gradients: block %zu's downsample is not a 1x1 convolution to conv3's width", i);
                return -1;
            }
            MRD_TRY(plan_conv1x1_dual(&k.f3, k.a2, b.c3.cin, x, b.ds.cin, b.ds.stride, B, k.ho, k.wo, b.c3ds_w,
                                      b.c3.cout, b.c3ds_b, k.out, ACT_RELU));
        } else {
            MRD_TRY(plan_conv(&k.f3, k.a2, B, k.ho, k.wo, b.c3.cin, b.c3.w, b.c3.cout, 1, 1, b.c3.b, k.out, x,
                              ACT_RELU));
        }
        // ---- backward: block i reads its output gradient gz, writes its input gradient to g[(i + 1) & 1]
        bf16* g_in = d->g[(i + 1) & 1];
        MRD_TRY(plan_conv_dgrad(&k.b3, d->gz, B, k.ho, k.wo, b.c3.cout, wt.c3t, b.c3.cout, 1, tap0, b.c3.cin, d->da2,
                                1, 1, 0, 0, k.a2, 2));
        if (st == 1) {
            k.n_b2 = 1;
            MRD_TRY(plan_conv_dgrad(&k.b2[0], d->da2, B, k.ho, k.wo, b.c2.cout, wt.c2t, 9LL * b.c2.cout, 9, tap9,
                                    b.c2.cin, d->da1, 1, 1, 0, 0, k.a1, 2));
        } else {
            k.n_b2 = 4;
            for (int ph = 0; ph < 4; ++ph) {
                const PhaseTaps& pt = kS2Phase[ph];
                MRD_TRY(plan_conv_dgrad(&k.b2[ph], d->da2, B, k.ho, k.wo, b.c2.cout,
                                        wt.c2t + 1LL * pt.first * b.c2.cout, 9LL * b.c2.cout, pt.n, pt.t, b.c2.cin,
                                        d->da1, 2, 2, ph >> 1, ph & 1, k.a1, 2));
            }
        }
        MRD_TRY(plan_conv_dgrad(&k.b1, d->da1, B, k.h, k.w, b.c1.cout, wt.c1t, b.c1.cout, 1, tap0, b.c1.cin, g_in, 1,
                                1, 0, 0, b.has_ds ? nullptr : d->gz, b.has_ds ? 0 : 1));
        if (b.has_ds)
            MRD_TRY(plan_conv_dgrad(&k.bds, d->gz, B, k.ho, k.wo, b.ds.cout, wt.dst, b.ds.cout, 1, tap0, b.ds.cin,
                                    g_in, b.ds.stride, b.ds.stride, 0, 0, g_in, 1));
        x = k.out;
    }
    d->B = B; d->H = H; d->W = W;
    d->cnn_epoch = c->cnn_ws_epoch;
    return 0;
}

// The saving forward: pooled features (fp32 [B, feat_dim]) as run_backbone computes them, every activation the
// backward needs kept, and block_out[k] (optional, f32 NCHW) = the output of bottleneck k.
int run_backbone_save(mrd_ctx* c, const void* images, int img_dtype, int B, int H, int W, float* pooled_f32,
                      float* const* block_out, cudaStream_t s) {
    MRD_TRY(check_images(img_dtype, H, W));
    if (B > kDgradMaxBatch) {
        set_last_error("data gradients: batch %d exceeds %d images per forward (27 MB of saved activations and "
                       "gradient scratch per 224 x 224 image)", B, kDgradMaxBatch);
        return -1;
    }
    MRD_TRY(ensure_cnn_ws(c, B, H, W));
    MRD_TRY(dgrad_pack(c, s));
    MRD_TRY(dgrad_plan(c, B, H, W));
    DgradCnn* d = train_state(c)->dg;
    d->valid = false;
    TRK("dgrad_fwd.repack_images", CAT_MEM, repack_images(images, img_dtype == MRD_DT_BF16, B, H, W, c->xpad, s));
    MRD_TRY(run(c, "dgrad_fwd.conv_stem", d->stem, s));
    TRK("dgrad_fwd.maxpool", CAT_MEM, maxpool3x3s2(d->stem_out, B, H / 2, W / 2, 64, d->pool_out, s));
    for (size_t i = 0; i < d->blk.size(); ++i) {
        const DgradBlock& k = d->blk[i];
        MRD_TRY(run(c, "dgrad_fwd.conv1", k.f1, s));
        MRD_TRY(run(c, "dgrad_fwd.conv2", k.f2, s));
        MRD_TRY(run(c, "dgrad_fwd.conv3", k.f3, s));
        if (block_out && block_out[i])
            TRK("dgrad.nhwc_to_nchw_f32", CAT_MEM, nhwc_bf16_to_nchw_f32(k.out, B, k.ho * k.wo, c->blocks[i].c3.cout,
                                                                        block_out[i], s));
    }
    const DgradBlock& top = d->blk.back();
    TRK("dgrad_fwd.avgpool", CAT_MEM, global_avgpool(top.out, B, top.ho * top.wo, c->feat_dim, c->b_pooled, pooled_f32, s));
    d->valid = true;
    return 0;
}

// Backward of the saving forward from d_pooled (f32 [B, feat_dim]).  Blocks 15 .. first_block run (first_block = 16:
// none); block_grads[k] (optional, f32 NCHW) receives d/d(output of block k) for first_block - 1 <= k < 15 (slot 15 is
// d_pooled / (h*w) at every position and is not written); d_block_in (optional) = d/d(input of block first_block);
// d_images (optional, first_block == 0) = d/d(images) f32 [B,3,H,W].  The caller has checked that the pending forward
// was a saving forward (DgradCnn::valid).
int dgrad_backbone(mrd_ctx* c, const float* d_pooled, float* const* block_grads, int first_block, float* d_block_in,
                   float* d_images, cudaStream_t s) {
    DgradCnn* d = c->train->dg;
    d->valid = false;
    const int nb = static_cast<int>(d->blk.size());
    if (first_block < 0 || first_block > nb || (d_images && first_block != 0) || (d_block_in && first_block == nb)) {
        set_last_error("data gradients: first_block %d outside [0, %d] or inconsistent with the outputs asked for",
                       first_block, nb);
        return -1;
    }
    const int B = d->B;
    if (first_block == nb) return 0;
    {
        const DgradBlock& top = d->blk.back();
        TRK("dgrad.avgpool_bwd", CAT_MEM, avgpool_bwd_mask_bf16(d_pooled, B, top.ho * top.wo, c->feat_dim, top.out,
                                                                d->gz, s));
    }
    for (int i = nb - 1; i >= first_block; --i) {
        const Bottleneck& b = c->blocks[i];
        const DgradBlock& k = d->blk[i];
        if (i < nb - 1)
            TRK("dgrad.relu_mask", CAT_MEM, relu_mask_bf16(d->g[i & 1], k.out, 1LL * B * k.ho * k.wo * b.c3.cout,
                                                           d->gz, s));
        MRD_TRY(run(c, "dgrad.conv3", k.b3, s));
        for (int j = 0; j < k.n_b2; ++j) MRD_TRY(run(c, k.n_b2 == 1 ? "dgrad.conv2" : "dgrad.conv2_s2", k.b2[j], s));
        MRD_TRY(run(c, b.has_ds ? "dgrad.conv1" : "dgrad.conv1+identity", k.b1, s));
        if (b.has_ds) MRD_TRY(run(c, b.ds.stride == 2 ? "dgrad.downsample_s2" : "dgrad.downsample", k.bds, s));
        const bf16* g_in = d->g[(i + 1) & 1];
        float* dst = i > 0 ? block_grads[i - 1] : nullptr;
        if (i == first_block && d_block_in) dst = d_block_in;
        if (dst) TRK("dgrad.nhwc_to_nchw_f32", CAT_MEM, nhwc_bf16_to_nchw_f32(g_in, B, k.h * k.w, b.c1.cin, dst, s));
        if (i > 0 && i == first_block && d_block_in && block_grads[i - 1])
            TRK("dgrad.nhwc_to_nchw_f32", CAT_MEM, nhwc_bf16_to_nchw_f32(g_in, B, k.h * k.w, b.c1.cin,
                                                                        block_grads[i - 1], s));
    }
    if (!d_images) return 0;
    const int H = d->H, W = d->W;
    TRK("dgrad.maxpool_bwd", CAT_MEM, maxpool3x3s2_bwd_relu(d->g[1], d->stem_out, B, H / 2, W / 2, 64, d->dstem, s));
    TRK("dgrad.stem", CAT_MEM, stem_dgrad_nchw(d->dstem, d->stem_wf, B, H, W, d_images, s));
    return 0;
}
