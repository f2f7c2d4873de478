// fp32 check mode (see fp32_check.h): a plain-fp32 CUDA forward of the reference's modules, written for
// exactness rather than speed.  Contractions go through simt_gemm.cu; the rest are the small kernels
// below.  Reference code followed: src/multimodal_classifier.py:131-177, src/cnn_encoder.py:168-184,
// TV:models/resnet.py:143-163,266-282, src/text_encoder.py:95-127, HF:models/bert/modeling_bert.py:72-112,
// 168-207,294-298,339-356, src/fusion_model.py:116-182,245-291, src/multimodal_classifier.py:73-83.

#include "fp32_check.h"

#include <math.h>
#include <stdio.h>

#include <mrd_b200.h>

#include "elementwise.h"
#include "simt_gemm.h"
#include "tma_host.h"
#include "train_kernels.h"

namespace mrd {

namespace {

#define F32_TRY(expr)               \
    do {                            \
        int rc__ = (expr);          \
        if (rc__ != 0) return rc__; \
    } while (0)

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("%s launch: %s", what, cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// MaxPool2d(3, stride 2, padding 1) on NCHW fp32 (TV:models/resnet.py:200)
__global__ void maxpool_nchw_kernel(const float* __restrict__ x, long long planes, int H, int W,
                                    float* __restrict__ y) {
    const int Ho = H / 2, Wo = W / 2;
    const long long total = planes * Ho * Wo;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int wo = static_cast<int>(i % Wo), ho = static_cast<int>((i / Wo) % Ho);
    const long long pl = i / (static_cast<long long>(Wo) * Ho);
    const float* src = x + pl * H * W;
    float m = -INFINITY;
    for (int dh = -1; dh <= 1; ++dh)
        for (int dw = -1; dw <= 1; ++dw) {
            const int h = ho * 2 + dh, w = wo * 2 + dw;
            if (h >= 0 && h < H && w >= 0 && w < W) m = fmaxf(m, src[h * W + w]);
        }
    y[i] = m;
}

// AdaptiveAvgPool2d(1): one warp per (image, channel) plane
__global__ void avgpool_nchw_kernel(const float* __restrict__ x, long long planes, int HW,
                                    float* __restrict__ y) {
    const long long pl = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pl >= planes) return;
    const int lane = threadIdx.x & 31;
    float a = 0.0f;
    for (int i = lane; i < HW; i += 32) a += x[pl * HW + i];
    a = wsum(a);
    if (lane == 0) y[pl] = a / static_cast<float>(HW);
}

// y = LayerNorm(x (+ r)) * g + b, biased variance, one warp per row (torch.nn.functional.layer_norm)
__global__ void layernorm_f32_kernel(const float* __restrict__ x, long long ldx,
                                     const float* __restrict__ r, long long ldr,
                                     const float* __restrict__ g, const float* __restrict__ b, float eps,
                                     int rows, int width, float* __restrict__ y, long long ldy) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* xr = x + row * ldx;
    const float* rr = r ? r + row * ldr : nullptr;
    float s = 0.0f;
    for (int i = lane; i < width; i += 32) s += xr[i] + (rr ? rr[i] : 0.0f);
    const float mean = wsum(s) / width;
    float v = 0.0f;
    for (int i = lane; i < width; i += 32) {
        const float d = xr[i] + (rr ? rr[i] : 0.0f) - mean;
        v += d * d;
    }
    const float rstd = 1.0f / sqrtf(wsum(v) / width + eps);
    for (int i = lane; i < width; i += 32)
        y[row * ldy + i] = (xr[i] + (rr ? rr[i] : 0.0f) - mean) * rstd * g[i] + b[i];
}

// word[ids] + position[j] + token_type[0] (HF:models/bert/modeling_bert.py:72-112, before LayerNorm)
__global__ void embed_sum_kernel(const long long* __restrict__ ids, const float* __restrict__ word,
                                 const float* __restrict__ pos, const float* __restrict__ type0, int S,
                                 int Hd, int vocab, long long total, float* __restrict__ y) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int h = static_cast<int>(i % Hd);
    const long long tok = i / Hd;
    const int j = static_cast<int>(tok % S);
    long long id = ids[tok];
    if (id < 0) id = 0;
    if (id >= vocab) id = vocab - 1;
    y[i] = word[id * Hd + h] + type0[h] + pos[static_cast<long long>(j) * Hd + h];
}

// softmax(q k^T / sqrt(d) + key_bias) v for one head; one warp per query row, scores in shared memory.
// qkv: [T, 3*Hd] fp32 (columns Q | K | V), d = 64.  probs (optional): the probabilities, [B,heads,S,S]; a row
// without any attended key is written as zeros (attention_probs does the same).
__global__ void attention_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ key_bias,
                                     int S, int heads, float scale, float* __restrict__ out,
                                     float* __restrict__ probs) {
    extern __shared__ float sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int b = blockIdx.x / heads, h = blockIdx.x % heads;
    const int q = blockIdx.y * nw + warp;
    float* sc = sm + warp * (S + 64);
    float* qs = sc + S;
    if (q >= S) return;
    const int Hd = heads * 64;
    const long long row0 = static_cast<long long>(b) * S;
    const float* qp = qkv + (row0 + q) * 3 * Hd + h * 64;
    qs[lane] = qp[lane];
    qs[lane + 32] = qp[lane + 32];
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) {
        const float* kp = qkv + (row0 + j) * 3 * Hd + Hd + h * 64;
        float a = 0.0f;
#pragma unroll 16
        for (int d = 0; d < 64; ++d) a = fmaf(qs[d], kp[d], a);
        a = a * scale + (key_bias ? key_bias[row0 + j] : 0.0f);
        sc[j] = a;
        mx = fmaxf(mx, a);
    }
    mx = wmax(mx);
    float sum = 0.0f;
    for (int j = lane; j < S; j += 32) {
        const float e = expf(sc[j] - mx);
        sc[j] = e;
        sum += e;
    }
    sum = wsum(sum);
    __syncwarp();
    if (probs) {
        float* pr = probs + (static_cast<long long>(blockIdx.x) * S + q) * S;
        for (int j = lane; j < S; j += 32) pr[j] = mx == -INFINITY ? 0.0f : sc[j] / sum;
    }
    float o0 = 0.0f, o1 = 0.0f;
    for (int j = 0; j < S; ++j) {
        const float* vp = qkv + (row0 + j) * 3 * Hd + 2 * Hd + h * 64;
        const float p = sc[j];
        o0 = fmaf(p, vp[lane], o0);
        o1 = fmaf(p, vp[lane + 32], o1);
    }
    float* op = out + (row0 + q) * Hd + h * 64;
    op[lane] = o0 / sum;
    op[lane + 32] = o1 / sum;
}

__global__ void softmax_rows_kernel(const float* __restrict__ x, int rows, int C, float* __restrict__ y) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float mx = -INFINITY;
    for (int i = 0; i < C; ++i) mx = fmaxf(mx, x[r * C + i]);
    float s = 0.0f;
    for (int i = 0; i < C; ++i) s += expf(x[r * C + i] - mx);
    for (int i = 0; i < C; ++i) y[r * C + i] = expf(x[r * C + i] - mx) / s;
}

__global__ void gather_rows_kernel(const float* __restrict__ x, long long row_stride, int rows, int width,
                                   float* __restrict__ y) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(rows) * width) return;
    y[i] = x[(i / width) * row_stride + i % width];
}

inline unsigned nblk(long long n, int per) { return static_cast<unsigned>((n + per - 1) / per); }

int need(const RawTable& t, const std::string& k, const RawTensor** out) {
    auto it = t.find(k);
    if (it == t.end()) {
        set_last_error("fp32 check: missing tensor '%s'", k.c_str());
        return -2;
    }
    *out = &it->second;
    return 0;
}

int arena_prepare(Fp32Arena* a, size_t bytes, cudaStream_t s) {
    a->used = 0;
    if (a->base && a->bytes >= bytes) return 0;
    cudaStreamSynchronize(s);
    cudaDeviceSynchronize();
    if (a->base) cudaFree(a->base);
    a->base = nullptr;
    a->bytes = 0;
    cudaError_t e = cudaMalloc(&a->base, bytes);
    if (e != cudaSuccess) {
        set_last_error("fp32 check: cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    a->bytes = bytes;
    return 0;
}
inline size_t pad256(long long n) { return (static_cast<size_t>(n) * 4 + 255) & ~static_cast<size_t>(255); }
float* take(Fp32Arena* a, long long n) {
    float* p = reinterpret_cast<float*>(static_cast<char*>(a->base) + a->used);
    a->used += pad256(n);
    return p;
}

int linear(const RawTable& t, const std::string& name, const float* x, long long ldx, int M, float* y,
           long long ldy, int act, const float* res, long long ldr, cudaStream_t s) {
    const RawTensor *w, *b;
    F32_TRY(need(t, name + ".weight", &w));
    F32_TRY(need(t, name + ".bias", &b));
    SimtGemm g;
    g.A = x; g.a_rs = ldx; g.a_cs = 1;
    g.B = w->p; g.b_rs = w->d[1]; g.b_cs = 1;
    g.M = M; g.N = static_cast<int>(w->d[0]); g.K = static_cast<int>(w->d[1]);
    g.C = y; g.ldc = ldy;
    g.bias = b->p;
    g.act = act;
    g.res = res; g.ldr = ldr;
    g.ksplit = 1;   // check mode: one CTA owns each output element (bit-reproducible, no atomics)
    return simt_gemm(g, s);
}

int layernorm(const RawTable& t, const std::string& name, const float* x, long long ldx, const float* r,
              long long ldr, float eps, int rows, int width, float* y, long long ldy, cudaStream_t s) {
    const RawTensor *g, *b;
    F32_TRY(need(t, name + ".weight", &g));
    F32_TRY(need(t, name + ".bias", &b));
    layernorm_f32_kernel<<<nblk(rows, 8), 256, 0, s>>>(x, ldx, r, ldr, g->p, b->p, eps, rows, width, y, ldy);
    return check_launch("layernorm_f32");
}

int conv_bn(const RawTable& t, const std::string& conv, const std::string& bn, const float* x, int B,
            int Cin, int H, int W, int stride, float eps, const float* residual, int act, float* y,
            int* Cout, int* Ho, int* Wo, cudaStream_t s) {
    const RawTensor *w, *g, *b, *mu, *var;
    F32_TRY(need(t, conv + ".weight", &w));
    F32_TRY(need(t, bn + ".weight", &g));
    F32_TRY(need(t, bn + ".bias", &b));
    F32_TRY(need(t, bn + ".running_mean", &mu));
    F32_TRY(need(t, bn + ".running_var", &var));
    if (w->d[1] != Cin) {
        set_last_error("fp32 check: %s expects %lld input channels, got %d", conv.c_str(), w->d[1], Cin);
        return -1;
    }
    SimtConv cv{};
    cv.Cin = Cin; cv.H = H; cv.W = W;
    cv.ks = static_cast<int>(w->d[2]);
    cv.stride = stride;
    cv.pad = cv.ks / 2;
    cv.Ho = (H + 2 * cv.pad - cv.ks) / stride + 1;
    cv.Wo = (W + 2 * cv.pad - cv.ks) / stride + 1;
    cv.mean = mu->p; cv.var = var->p; cv.gamma = g->p; cv.beta = b->p; cv.eps = eps;
    cv.residual = residual;
    *Cout = static_cast<int>(w->d[0]);
    *Ho = cv.Ho;
    *Wo = cv.Wo;
    return simt_conv_bn(x, B, cv, w->p, *Cout, act, y, s);
}

}  // namespace

void fp32_arena_free(Fp32Arena* ws) {
    if (ws->base) cudaFree(ws->base);
    ws->base = nullptr;
    ws->bytes = ws->used = 0;
}

int fp32_cnn_encoder(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const float* images, int B,
                     int H, int W, float* emb, float* pooled_out, float* fmap, cudaStream_t s) {
    if (H % 32 || W % 32) {
        set_last_error("fp32 check: image size %dx%d must be a multiple of 32", H, W);
        return -1;
    }
    const long long big = 1LL * B * 64 * (H / 2) * (W / 2);  // = B*256*(H/4)*(W/4): the largest tensor
    F32_TRY(arena_prepare(ws, 3 * pad256(big) + 2 * pad256(big / 2) + pad256(1LL * B * 2048) +
                                  pad256(1LL * B * 1024), s));
    float* bufs[2] = {take(ws, big), take(ws, big)};
    float* dsb = take(ws, big);
    float* mid0 = take(ws, big / 2);
    float* mid1 = take(ws, big / 2);
    float* pooled = take(ws, 1LL * B * 2048);
    float* projh = take(ws, 1LL * B * 1024);
    const std::string bb = "cnn_encoder.backbone.";
    int C, h, w;
    F32_TRY(conv_bn(t, bb + "conv1", bb + "bn1", images, B, 3, H, W, 2, o.bn_eps, nullptr, MRD_ACT_RELU,
                    bufs[1], &C, &h, &w, s));
    maxpool_nchw_kernel<<<nblk(1LL * B * C * (h / 2) * (w / 2), 256), 256, 0, s>>>(bufs[1], 1LL * B * C, h, w,
                                                                                bufs[0]);
    F32_TRY(check_launch("maxpool_nchw"));
    h /= 2; w /= 2;
    int cur = 0;
    for (int L = 1; L <= 4; ++L) {
        for (int i = 0;; ++i) {
            char pre[96];
            snprintf(pre, sizeof(pre), "%slayer%d.%d.", bb.c_str(), L, i);
            const std::string p(pre);
            if (t.find(p + "conv1.weight") == t.end()) break;
            const int stride = (i == 0 && L > 1) ? 2 : 1;  // ResNet v1.5: stride on conv2 (TV:109-113)
            const float* x = bufs[cur];
            float* y = bufs[cur ^ 1];
            int c1, c2, c3, h1, w1, h2, w2, h3, w3;
            F32_TRY(conv_bn(t, p + "conv1", p + "bn1", x, B, C, h, w, 1, o.bn_eps, nullptr, MRD_ACT_RELU, mid0,
                            &c1, &h1, &w1, s));
            F32_TRY(conv_bn(t, p + "conv2", p + "bn2", mid0, B, c1, h1, w1, stride, o.bn_eps, nullptr,
                            MRD_ACT_RELU, mid1, &c2, &h2, &w2, s));
            const float* identity = x;
            if (t.find(p + "downsample.0.weight") != t.end()) {
                int cd, hd, wd;
                F32_TRY(conv_bn(t, p + "downsample.0", p + "downsample.1", x, B, C, h, w, stride, o.bn_eps,
                                nullptr, MRD_ACT_NONE, dsb, &cd, &hd, &wd, s));
                identity = dsb;
            }
            F32_TRY(conv_bn(t, p + "conv3", p + "bn3", mid1, B, c2, h2, w2, 1, o.bn_eps, identity,
                            MRD_ACT_RELU, y, &c3, &h3, &w3, s));
            C = c3; h = h3; w = w3;
            cur ^= 1;
        }
    }
    if (C > 2048) {
        set_last_error("fp32 check: backbone feature width %d unsupported", C);
        return -1;
    }
    const float* feat = bufs[cur];
    if (fmap) {
        cudaError_t e = cudaMemcpyAsync(fmap, feat, sizeof(float) * B * C * h * w, cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) {
            set_last_error("fp32 check: feature map copy: %s", cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
    }
    float* pl = pooled_out ? pooled_out : pooled;
    avgpool_nchw_kernel<<<nblk(1LL * B * C, 8), 256, 0, s>>>(feat, 1LL * B * C, h * w, pl);
    F32_TRY(check_launch("avgpool_nchw"));
    const RawTensor* w1;
    F32_TRY(need(t, "cnn_encoder.projection.0.weight", &w1));
    const int E1 = static_cast<int>(w1->d[0]);
    if (E1 > 1024) {
        set_last_error("fp32 check: projection width %d unsupported", E1);
        return -1;
    }
    F32_TRY(linear(t, "cnn_encoder.projection.0", pl, C, B, projh, E1, MRD_ACT_RELU, nullptr, 0, s));
    const RawTensor* w2;
    F32_TRY(need(t, "cnn_encoder.projection.3.weight", &w2));
    return linear(t, "cnn_encoder.projection.3", projh, E1, B, emb, w2->d[0], MRD_ACT_NONE, nullptr, 0, s);
}

int fp32_text_encoder(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const long long* ids,
                      const void* mask, int mask_dtype, int B, int S, float* cls, float* last_hidden,
                      float* all_hidden, float* attn_probs, cudaStream_t s) {
    const std::string e = "text_encoder.encoder.embeddings.";
    const RawTensor *we, *pe, *te;
    F32_TRY(need(t, e + "word_embeddings.weight", &we));
    F32_TRY(need(t, e + "position_embeddings.weight", &pe));
    F32_TRY(need(t, e + "token_type_embeddings.weight", &te));
    const int Hd = static_cast<int>(we->d[1]), vocab = static_cast<int>(we->d[0]);
    const int heads = o.bert_heads;
    if (Hd != heads * 64 || S > pe->d[0] || S <= 0) {
        set_last_error("fp32 check: text encoder shape unsupported (hidden %d, heads %d, S %d)", Hd, heads, S);
        return -1;
    }
    const long long T = 1LL * B * S;
    const RawTensor* wf;
    F32_TRY(need(t, "text_encoder.encoder.encoder.layer.0.intermediate.dense.weight", &wf));
    const int F = static_cast<int>(wf->d[0]);
    F32_TRY(arena_prepare(ws, 4 * pad256(T * Hd) + pad256(T * 3 * Hd) + pad256(T * F) + pad256(T), s));
    float* h = take(ws, T * Hd);
    float* h2 = take(ws, T * Hd);
    float* ctx = take(ws, T * Hd);
    float* tmp = take(ws, T * Hd);
    float* qkv = take(ws, T * 3 * Hd);
    float* ffn = take(ws, T * F);
    float* bias = take(ws, T);
    if (mask) F32_TRY(mask_to_bias(mask, mask_dtype, B, S, bias, s));
    embed_sum_kernel<<<nblk(T * Hd, 256), 256, 0, s>>>(ids, we->p, pe->p, te->p, S, Hd, vocab, T * Hd, tmp);
    F32_TRY(check_launch("embed_sum"));
    F32_TRY(layernorm(t, e + "LayerNorm", tmp, Hd, nullptr, 0, o.bert_ln_eps, static_cast<int>(T), Hd, h, Hd, s));
    auto export_hidden = [&](int l) -> int {
        if (!all_hidden) return 0;
        cudaError_t ce = cudaMemcpyAsync(all_hidden + l * T * Hd, h, sizeof(float) * T * Hd,
                                         cudaMemcpyDeviceToDevice, s);
        if (ce != cudaSuccess) {
            set_last_error("fp32 check: hidden export: %s", cudaGetErrorString(ce));
            return -static_cast<int>(ce);
        }
        return 0;
    };
    F32_TRY(export_hidden(0));
    const int nw = 4;
    for (int i = 0;; ++i) {
        char pre[96];
        snprintf(pre, sizeof(pre), "text_encoder.encoder.encoder.layer.%d.", i);
        const std::string p(pre);
        if (t.find(p + "attention.self.query.weight") == t.end()) break;
        F32_TRY(linear(t, p + "attention.self.query", h, Hd, static_cast<int>(T), qkv, 3 * Hd, MRD_ACT_NONE,
                       nullptr, 0, s));
        F32_TRY(linear(t, p + "attention.self.key", h, Hd, static_cast<int>(T), qkv + Hd, 3 * Hd, MRD_ACT_NONE,
                       nullptr, 0, s));
        F32_TRY(linear(t, p + "attention.self.value", h, Hd, static_cast<int>(T), qkv + 2 * Hd, 3 * Hd,
                       MRD_ACT_NONE, nullptr, 0, s));
        attention_f32_kernel<<<dim3(B * heads, (S + nw - 1) / nw), nw * 32, nw * (S + 64) * sizeof(float), s>>>(
            qkv, mask ? bias : nullptr, S, heads, 0.125f, ctx,
            attn_probs ? attn_probs + static_cast<long long>(i) * B * heads * S * S : nullptr);
        F32_TRY(check_launch("attention_f32"));
        // BertSelfOutput: LayerNorm(dense(ctx) + hidden) (HF:294-298)
        F32_TRY(linear(t, p + "attention.output.dense", ctx, Hd, static_cast<int>(T), tmp, Hd, MRD_ACT_NONE,
                       nullptr, 0, s));
        F32_TRY(layernorm(t, p + "attention.output.LayerNorm", tmp, Hd, h, Hd, o.bert_ln_eps,
                          static_cast<int>(T), Hd, h2, Hd, s));
        // BertIntermediate + BertOutput (HF:339-356)
        F32_TRY(linear(t, p + "intermediate.dense", h2, Hd, static_cast<int>(T), ffn, F, MRD_ACT_GELU, nullptr,
                       0, s));
        F32_TRY(linear(t, p + "output.dense", ffn, F, static_cast<int>(T), tmp, Hd, MRD_ACT_NONE, nullptr, 0, s));
        F32_TRY(layernorm(t, p + "output.LayerNorm", tmp, Hd, h2, Hd, o.bert_ln_eps, static_cast<int>(T), Hd,
                          h, Hd, s));
        F32_TRY(export_hidden(i + 1));
    }
    if (last_hidden) {
        cudaError_t ce = cudaMemcpyAsync(last_hidden, h, sizeof(float) * T * Hd, cudaMemcpyDeviceToDevice, s);
        if (ce != cudaSuccess) {
            set_last_error("fp32 check: last_hidden copy: %s", cudaGetErrorString(ce));
            return -static_cast<int>(ce);
        }
    }
    // CLS row of every sequence (src/text_encoder.py:118); eval-mode dropout is the identity
    gather_rows_kernel<<<nblk(1LL * B * Hd, 256), 256, 0, s>>>(h, 1LL * S * Hd, B, Hd, cls);
    return check_launch("gather_rows");
}

int fp32_fusion(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const float* img, const float* txt,
                int B, float* fused, float* attn_i2t, float* attn_t2i, cudaStream_t s) {
    const std::string f = "fusion.fusion_layer.";
    const RawTensor* wi;
    F32_TRY(need(t, f + "image_proj.weight", &wi));
    const int F = static_cast<int>(wi->d[0]);
    const RawTensor* wt;
    F32_TRY(need(t, f + "text_proj.weight", &wt));
    F32_TRY(arena_prepare(ws, 8 * pad256(1LL * B * F) + pad256(2LL * B * F), s));
    float* ip = take(ws, 1LL * B * F);
    float* tp = take(ws, 1LL * B * F);
    float* v = take(ws, 1LL * B * F);
    float* ia = take(ws, 1LL * B * F);
    float* ta = take(ws, 1LL * B * F);
    float* fh = take(ws, 1LL * B * F);
    float* cat = take(ws, 2LL * B * F);
    F32_TRY(linear(t, f + "image_proj", img, wi->d[1], B, ip, F, MRD_ACT_NONE, nullptr, 0, s));
    F32_TRY(linear(t, f + "text_proj", txt, wt->d[1], B, tp, F, MRD_ACT_NONE, nullptr, 0, s));
    // CrossModalAttention with one key (src/fusion_model.py:138-176): softmax over a single score is 1,
    // so attended = output_proj(value_proj(kv)); the residual is added in the GEMM epilogue
    const float* res_i = o.fusion_residual ? ip : nullptr;
    const float* res_t = o.fusion_residual ? tp : nullptr;
    F32_TRY(linear(t, f + "image_to_text_attention.value_proj", tp, F, B, v, F, MRD_ACT_NONE, nullptr, 0, s));
    F32_TRY(linear(t, f + "image_to_text_attention.output_proj", v, F, B, ia, F, MRD_ACT_NONE, res_i, F, s));
    F32_TRY(linear(t, f + "text_to_image_attention.value_proj", ip, F, B, v, F, MRD_ACT_NONE, nullptr, 0, s));
    F32_TRY(linear(t, f + "text_to_image_attention.output_proj", v, F, B, ta, F, MRD_ACT_NONE, res_t, F, s));
    F32_TRY(layernorm(t, f + "layer_norm_image", ia, F, nullptr, 0, o.fusion_ln_eps, B, F, cat, 2 * F, s));
    F32_TRY(layernorm(t, f + "layer_norm_text", ta, F, nullptr, 0, o.fusion_ln_eps, B, F, cat + F, 2 * F, s));
    F32_TRY(linear(t, f + "fusion.0", cat, 2 * F, B, fh, F, MRD_ACT_RELU, nullptr, 0, s));
    F32_TRY(linear(t, f + "fusion.3", fh, F, B, fused, F, MRD_ACT_NONE, nullptr, 0, s));
    if (attn_i2t) F32_TRY(fill_f32(attn_i2t, 1LL * B * o.fusion_heads, 1.0f, s));
    if (attn_t2i) F32_TRY(fill_f32(attn_t2i, 1LL * B * o.fusion_heads, 1.0f, s));
    return 0;
}

int fp32_head(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const float* x, int B, float* logits,
              float* probs, cudaStream_t s) {
    F32_TRY(arena_prepare(ws, 2 * pad256(1LL * B * 4096), s));
    float* buf[2] = {take(ws, 1LL * B * 4096), take(ws, 1LL * B * 4096)};
    std::string last;
    int last_idx = -1;
    for (int i = 0; i < 64; i += 3) {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%d", i);
        if (t.find(std::string(nm) + ".weight") == t.end()) break;
        last = nm;
        last_idx = i;
    }
    if (last_idx < 0) {
        set_last_error("fp32 check: no classifier.classifier.*.weight tensors");
        return -2;
    }
    const float* cur = x;
    long long ld = 0;
    {
        const RawTensor* w0;
        F32_TRY(need(t, "classifier.classifier.0.weight", &w0));
        ld = w0->d[1];
    }
    int j = 0;
    for (int i = 0; i < last_idx; i += 3, ++j) {
        char nm[64];
        snprintf(nm, sizeof(nm), "classifier.classifier.%d", i);
        const RawTensor* w;
        F32_TRY(need(t, std::string(nm) + ".weight", &w));
        if (w->d[0] > 4096) {
            set_last_error("fp32 check: head layer width %lld unsupported", w->d[0]);
            return -1;
        }
        F32_TRY(linear(t, nm, cur, ld, B, buf[j & 1], w->d[0], o.head_act, nullptr, 0, s));
        cur = buf[j & 1];
        ld = w->d[0];
    }
    const RawTensor* wl;
    F32_TRY(need(t, last + ".weight", &wl));
    const int C = static_cast<int>(wl->d[0]);
    F32_TRY(linear(t, last, cur, ld, B, logits, C, MRD_ACT_NONE, nullptr, 0, s));
    if (probs) {
        softmax_rows_kernel<<<nblk(B, 128), 128, 0, s>>>(logits, B, C, probs);
        F32_TRY(check_launch("softmax_rows"));
    }
    return 0;
}

// ====================================================================== fp32 check of the training step
namespace {

__global__ void gelu_f32_kernel(const float* __restrict__ u, long long n, float* __restrict__ g) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) g[i] = 0.5f * u[i] * (1.0f + erff(u[i] * 0.70710678118654752f));
}
// du = dg * gelu'(u), gelu'(u) = Phi(u) + u * phi(u)
__global__ void gelu_bwd_f32_kernel(const float* __restrict__ u, const float* __restrict__ dg, long long n,
                                    float* __restrict__ du) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = u[i];
    du[i] = dg[i] * (0.5f * (1.0f + erff(v * 0.70710678118654752f)) + v * 0.3989422804014327f * expf(-0.5f * v * v));
}

// dst[b*S*width + c] = src[b*width + c] (dst zeroed): gradient of last_hidden_state[:, 0, :]
__global__ void scatter_first_rows_kernel(const float* __restrict__ src, int B, long long row_stride, int width,
                                          float* __restrict__ dst) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(B) * width) return;
    dst[(i / width) * row_stride + i % width] = src[i];
}

// Attention backward, pass 1: one warp per (sample, head, query).  Recomputes the probabilities of the row, stores
// them and dS = P o (dP - rowsum(P o dP)) and produces dQ = scale * dS K.
__global__ void attention_bwd_q_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ key_bias,
                                           const float* __restrict__ dctx, int S, int heads, float scale,
                                           float* __restrict__ P, float* __restrict__ dS,
                                           float* __restrict__ dqkv) {
    extern __shared__ float sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int b = blockIdx.x / heads, h = blockIdx.x % heads;
    const int q = blockIdx.y * nw + warp;
    if (q >= S) return;
    float* pr = sm + warp * (2 * S + 128);
    float* ds = pr + S;
    float* qs = ds + S;      // 64
    float* dos = qs + 64;    // 64
    const int Hd = heads * 64;
    const long long row0 = static_cast<long long>(b) * S;
    const float* qp = qkv + (row0 + q) * 3 * Hd + h * 64;
    const float* dop = dctx + (row0 + q) * Hd + h * 64;
    qs[lane] = qp[lane]; qs[lane + 32] = qp[lane + 32];
    dos[lane] = dop[lane]; dos[lane + 32] = dop[lane + 32];
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) {
        const float* kp = qkv + (row0 + j) * 3 * Hd + Hd + h * 64;
        float a = 0.0f;
#pragma unroll 16
        for (int d = 0; d < 64; ++d) a = fmaf(qs[d], kp[d], a);
        a = a * scale + (key_bias ? key_bias[row0 + j] : 0.0f);
        pr[j] = a;
        mx = fmaxf(mx, a);
    }
    mx = wmax(mx);
    float sum = 0.0f;
    for (int j = lane; j < S; j += 32) {
        const float e = expf(pr[j] - mx);
        pr[j] = e;
        sum += e;
    }
    sum = wsum(sum);
    float delta = 0.0f;
    for (int j = lane; j < S; j += 32) {
        const float* vp = qkv + (row0 + j) * 3 * Hd + 2 * Hd + h * 64;
        float dp = 0.0f;
#pragma unroll 16
        for (int d = 0; d < 64; ++d) dp = fmaf(dos[d], vp[d], dp);
        const float p = pr[j] / sum;
        pr[j] = p;
        ds[j] = dp;
        delta += p * dp;
    }
    delta = wsum(delta);
    const long long prow = (static_cast<long long>(blockIdx.x) * S + q) * S;
    for (int j = lane; j < S; j += 32) {
        const float v = pr[j] * (ds[j] - delta);
        ds[j] = v;
        P[prow + j] = pr[j];
        dS[prow + j] = v;
    }
    __syncwarp();
    float g0 = 0.0f, g1 = 0.0f;
    for (int j = 0; j < S; ++j) {
        const float* kp = qkv + (row0 + j) * 3 * Hd + Hd + h * 64;
        g0 = fmaf(ds[j], kp[lane], g0);
        g1 = fmaf(ds[j], kp[lane + 32], g1);
    }
    float* dq = dqkv + (row0 + q) * 3 * Hd + h * 64;
    dq[lane] = g0 * scale;
    dq[lane + 32] = g1 * scale;
}

// pass 2: one warp per (sample, head, key): dK = scale * dS^T Q, dV = P^T dO
__global__ void attention_bwd_kv_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ dctx,
                                            const float* __restrict__ P, const float* __restrict__ dS, int S,
                                            int heads, float scale, float* __restrict__ dqkv) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int b = blockIdx.x / heads, h = blockIdx.x % heads;
    const int j = blockIdx.y * nw + warp;
    if (j >= S) return;
    const int Hd = heads * 64;
    const long long row0 = static_cast<long long>(b) * S;
    const long long pbase = static_cast<long long>(blockIdx.x) * S * S;
    float k0 = 0.0f, k1 = 0.0f, v0 = 0.0f, v1 = 0.0f;
    for (int q = 0; q < S; ++q) {
        const float d = dS[pbase + static_cast<long long>(q) * S + j];
        const float p = P[pbase + static_cast<long long>(q) * S + j];
        const float* qp = qkv + (row0 + q) * 3 * Hd + h * 64;
        const float* dop = dctx + (row0 + q) * Hd + h * 64;
        k0 = fmaf(d, qp[lane], k0);
        k1 = fmaf(d, qp[lane + 32], k1);
        v0 = fmaf(p, dop[lane], v0);
        v1 = fmaf(p, dop[lane + 32], v1);
    }
    float* dk = dqkv + (row0 + j) * 3 * Hd + Hd + h * 64;
    float* dv = dqkv + (row0 + j) * 3 * Hd + 2 * Hd + h * 64;
    dk[lane] = k0 * scale;
    dk[lane + 32] = k1 * scale;
    dv[lane] = v0;
    dv[lane + 32] = v1;
}

// scatter-add of the embedding-sum gradient into the three tables (nn.Embedding backward; the word row of
// padding_idx receives nothing, HF:models/bert/modeling_bert.py:76)
__global__ void embed_bwd_f32_kernel(const long long* __restrict__ ids, const float* __restrict__ de, int S,
                                     int Hd, int vocab, int pad_idx, long long total, float* __restrict__ dword,
                                     float* __restrict__ dpos, float* __restrict__ dtype0) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int hh = static_cast<int>(i % Hd);
    const long long tok = i / Hd;
    const int j = static_cast<int>(tok % S);
    long long id = ids[tok];
    if (id < 0) id = 0;
    if (id >= vocab) id = vocab - 1;
    const float v = de[i];
    if (v == 0.0f) return;
    if (dword && id != pad_idx) atomicAdd(dword + id * Hd + hh, v);
    if (dpos) atomicAdd(dpos + static_cast<long long>(j) * Hd + hh, v);
    if (dtype0) atomicAdd(dtype0 + hh, v);
}

// C[M,N] (+)= A * B^T with arbitrary element strides; one CTA per output element group (no split-K atomics)
int gemm_f32(const float* A, long long a_rs, long long a_cs, const float* B, long long b_rs, long long b_cs, int M,
             int N, int K, float* C, long long ldc, int accumulate, const float* res, long long ldr, cudaStream_t s) {
    SimtGemm g;
    g.A = A; g.a_rs = a_rs; g.a_cs = a_cs;
    g.B = B; g.b_rs = b_rs; g.b_cs = b_cs;
    g.M = M; g.N = N; g.K = K;
    g.C = C; g.ldc = ldc;
    g.accumulate = accumulate;
    g.res = res; g.ldr = ldr;
    g.ksplit = 1;
    return simt_gemm(g, s);
}

inline float* grad_of(const Fp32GradTable& g, const std::string& k) {
    auto it = g.find(k);
    return it == g.end() ? nullptr : it->second;
}

// y = x W^T + b: dW += dy^T x, db += colsum(dy), dx = dy W (+ dx_res) when dx != null
int linear_bwd(const RawTable& t, const Fp32GradTable& gt, const std::string& name, const float* x, long long ldx,
               const float* dy, long long lddy, int M, float* dx, long long lddx, const float* dx_res,
               long long ld_res, cudaStream_t s) {
    const RawTensor* w;
    F32_TRY(need(t, name + ".weight", &w));
    const int N = static_cast<int>(w->d[0]), K = static_cast<int>(w->d[1]);
    if (float* gw = grad_of(gt, name + ".weight"))
        F32_TRY(gemm_f32(dy, 1, lddy, x, 1, ldx, N, K, M, gw, K, 1, nullptr, 0, s));
    if (float* gb = grad_of(gt, name + ".bias")) F32_TRY(colsum_f32(dy, lddy, M, N, gb, s));
    if (dx) F32_TRY(gemm_f32(dy, lddy, 1, w->p, 1, K, M, K, N, dx, lddx, 0, dx_res, ld_res, s));
    return 0;
}

}  // namespace

int fp32_bert_train_forward(const RawTable& t, const Fp32Opts& o, Fp32TrainSave* sv, const long long* ids,
                            const void* mask, int mask_dtype, int B, int S, float* cls, cudaStream_t s) {
    sv->valid = false;
    const std::string e = "text_encoder.encoder.embeddings.";
    const RawTensor *we, *pe, *te, *wf;
    F32_TRY(need(t, e + "word_embeddings.weight", &we));
    F32_TRY(need(t, e + "position_embeddings.weight", &pe));
    F32_TRY(need(t, e + "token_type_embeddings.weight", &te));
    F32_TRY(need(t, "text_encoder.encoder.encoder.layer.0.intermediate.dense.weight", &wf));
    const int Hd = static_cast<int>(we->d[1]), vocab = static_cast<int>(we->d[0]);
    const int F = static_cast<int>(wf->d[0]), heads = o.bert_heads;
    int L = 0;
    while (L < 48 && t.find("text_encoder.encoder.encoder.layer." + std::to_string(L) + ".attention.self.query.weight") != t.end())
        ++L;
    if (Hd != heads * 64 || S > pe->d[0] || S <= 0 || S > 512 || L == 0) {
        set_last_error("fp32 check (train): text encoder shape unsupported (hidden %d, heads %d, S %d, layers %d)", Hd,
                       heads, S, L);
        return -1;
    }
    const long long T = 1LL * B * S;
    const long long att = 1LL * B * heads * S * S;
    const size_t per_layer = 6 * pad256(T * Hd) + pad256(T * 3 * Hd) + 2 * pad256(T * F);   // x ctx s1 h1 s2 (+1 spare), qkv, u g
    const size_t total = L * per_layer + pad256(T) + 2 * pad256(T * Hd) /* emb_sum, x_final */ +
                         5 * pad256(T * Hd) + pad256(T * F) + pad256(T * 3 * Hd) + 2 * pad256(att);
    F32_TRY(arena_prepare(&sv->ws, total, s));
    sv->B = B; sv->S = S; sv->Hd = Hd; sv->F = F; sv->L = L; sv->ids = ids;
    sv->bias = take(&sv->ws, T);
    sv->emb_sum = take(&sv->ws, T * Hd);
    sv->x_final = take(&sv->ws, T * Hd);
    for (int i = 0; i < L; ++i) {
        sv->x[i] = take(&sv->ws, T * Hd);
        sv->qkv[i] = take(&sv->ws, T * 3 * Hd);
        sv->ctx[i] = take(&sv->ws, T * Hd);
        sv->s1[i] = take(&sv->ws, T * Hd);
        sv->h1[i] = take(&sv->ws, T * Hd);
        sv->u[i] = take(&sv->ws, T * F);
        sv->g[i] = take(&sv->ws, T * F);
        sv->s2[i] = take(&sv->ws, T * Hd);
    }
    sv->dxa = take(&sv->ws, T * Hd);
    sv->dxb = take(&sv->ws, T * Hd);
    sv->d_s = take(&sv->ws, T * Hd);
    sv->d_h1 = take(&sv->ws, T * Hd);
    sv->d_ctx = take(&sv->ws, T * Hd);
    sv->d_big = take(&sv->ws, T * F);
    sv->d_qkv = take(&sv->ws, T * 3 * Hd);
    sv->P = take(&sv->ws, att);
    sv->dS = take(&sv->ws, att);

    const int Ti = static_cast<int>(T);
    if (mask) F32_TRY(mask_to_bias(mask, mask_dtype, B, S, sv->bias, s));
    const float* kb = mask ? sv->bias : nullptr;
    sv->has_mask = mask != nullptr;
    embed_sum_kernel<<<nblk(T * Hd, 256), 256, 0, s>>>(ids, we->p, pe->p, te->p, S, Hd, vocab, T * Hd, sv->emb_sum);
    F32_TRY(check_launch("embed_sum"));
    F32_TRY(layernorm(t, e + "LayerNorm", sv->emb_sum, Hd, nullptr, 0, o.bert_ln_eps, Ti, Hd, sv->x[0], Hd, s));
    const int nw = 4;
    for (int i = 0; i < L; ++i) {
        const std::string p = "text_encoder.encoder.encoder.layer." + std::to_string(i) + ".";
        float* x_next = i + 1 < L ? sv->x[i + 1] : sv->x_final;
        F32_TRY(linear(t, p + "attention.self.query", sv->x[i], Hd, Ti, sv->qkv[i], 3 * Hd, MRD_ACT_NONE, nullptr, 0, s));
        F32_TRY(linear(t, p + "attention.self.key", sv->x[i], Hd, Ti, sv->qkv[i] + Hd, 3 * Hd, MRD_ACT_NONE, nullptr, 0, s));
        F32_TRY(linear(t, p + "attention.self.value", sv->x[i], Hd, Ti, sv->qkv[i] + 2 * Hd, 3 * Hd, MRD_ACT_NONE, nullptr, 0, s));
        attention_f32_kernel<<<dim3(B * heads, (S + nw - 1) / nw), nw * 32, nw * (S + 64) * sizeof(float), s>>>(
            sv->qkv[i], kb, S, heads, 0.125f, sv->ctx[i], nullptr);
        F32_TRY(check_launch("attention_f32"));
        // s1 = dense(ctx) + x ; h1 = LayerNorm(s1)   (HF:294-298)
        F32_TRY(linear(t, p + "attention.output.dense", sv->ctx[i], Hd, Ti, sv->s1[i], Hd, MRD_ACT_NONE, sv->x[i], Hd, s));
        F32_TRY(layernorm(t, p + "attention.output.LayerNorm", sv->s1[i], Hd, nullptr, 0, o.bert_ln_eps, Ti, Hd,
                          sv->h1[i], Hd, s));
        // u = dense(h1) ; g = gelu(u) ; s2 = dense(g) + h1 ; x' = LayerNorm(s2)   (HF:339-356)
        F32_TRY(linear(t, p + "intermediate.dense", sv->h1[i], Hd, Ti, sv->u[i], F, MRD_ACT_NONE, nullptr, 0, s));
        gelu_f32_kernel<<<nblk(T * F, 256), 256, 0, s>>>(sv->u[i], T * F, sv->g[i]);
        F32_TRY(check_launch("gelu_f32"));
        F32_TRY(linear(t, p + "output.dense", sv->g[i], F, Ti, sv->s2[i], Hd, MRD_ACT_NONE, sv->h1[i], Hd, s));
        F32_TRY(layernorm(t, p + "output.LayerNorm", sv->s2[i], Hd, nullptr, 0, o.bert_ln_eps, Ti, Hd, x_next, Hd, s));
    }
    gather_rows_kernel<<<nblk(1LL * B * Hd, 256), 256, 0, s>>>(sv->x_final, 1LL * S * Hd, B, Hd, cls);
    F32_TRY(check_launch("gather_rows"));
    sv->valid = true;
    return 0;
}

int fp32_bert_train_backward(const RawTable& t, const Fp32Opts& o, Fp32TrainSave* sv, const float* d_cls,
                             const Fp32GradTable& gt, int pad_idx, cudaStream_t s) {
    if (!sv->valid) {
        set_last_error("fp32 check (train): no forward is pending");
        return -1;
    }
    sv->valid = false;
    const int B = sv->B, S = sv->S, Hd = sv->Hd, F = sv->F, L = sv->L, heads = o.bert_heads;
    const long long T = 1LL * B * S;
    const int Ti = static_cast<int>(T);
    const float* kb = sv->has_mask ? sv->bias : nullptr;
    auto get = [&](const std::string& k) -> const float* {
        auto it = t.find(k);
        return it == t.end() ? nullptr : it->second.p;
    };
    float* dx_in = (L & 1) ? sv->dxb : sv->dxa;   // layer i reads dx[(i+1)&1], writes dx[i&1]
    cudaError_t ce = cudaMemsetAsync(dx_in, 0, sizeof(float) * T * Hd, s);
    if (ce != cudaSuccess) {
        set_last_error("fp32 check (train): memset: %s", cudaGetErrorString(ce));
        return -static_cast<int>(ce);
    }
    scatter_first_rows_kernel<<<nblk(1LL * B * Hd, 256), 256, 0, s>>>(d_cls, B, 1LL * S * Hd, Hd, dx_in);
    F32_TRY(check_launch("scatter_first_rows"));
    const int nw = 4;
    for (int i = L - 1; i >= 0; --i) {
        const std::string p = "text_encoder.encoder.encoder.layer." + std::to_string(i) + ".";
        const float* dxi = ((i + 1) & 1) ? sv->dxb : sv->dxa;
        float* dxo = (i & 1) ? sv->dxb : sv->dxa;
        const float* g2 = get(p + "output.LayerNorm.weight");
        const float* g1 = get(p + "attention.output.LayerNorm.weight");
        if (!g1 || !g2) {
            set_last_error("fp32 check (train): LayerNorm weights of layer %d missing", i);
            return -2;
        }
        // x' = LN2(s2), s2 = h1 + W2 g + b2
        F32_TRY(ln_bwd_f32(sv->s2[i], Hd, dxi, Hd, g2, o.bert_ln_eps, Ti, Hd, sv->d_s, Hd,
                           grad_of(gt, p + "output.LayerNorm.weight"), grad_of(gt, p + "output.LayerNorm.bias"), s));
        F32_TRY(linear_bwd(t, gt, p + "output.dense", sv->g[i], F, sv->d_s, Hd, Ti, sv->d_big, F, nullptr, 0, s));
        gelu_bwd_f32_kernel<<<nblk(T * F, 256), 256, 0, s>>>(sv->u[i], sv->d_big, T * F, sv->d_big);
        F32_TRY(check_launch("gelu_bwd_f32"));
        // dh1 = du W1 + d_s2 (residual path)
        F32_TRY(linear_bwd(t, gt, p + "intermediate.dense", sv->h1[i], Hd, sv->d_big, F, Ti, sv->d_h1, Hd, sv->d_s, Hd, s));
        // h1 = LN1(s1), s1 = x + Wo ctx + bo
        F32_TRY(ln_bwd_f32(sv->s1[i], Hd, sv->d_h1, Hd, g1, o.bert_ln_eps, Ti, Hd, sv->d_s, Hd,
                           grad_of(gt, p + "attention.output.LayerNorm.weight"),
                           grad_of(gt, p + "attention.output.LayerNorm.bias"), s));
        F32_TRY(linear_bwd(t, gt, p + "attention.output.dense", sv->ctx[i], Hd, sv->d_s, Hd, Ti, sv->d_ctx, Hd, nullptr, 0, s));
        attention_bwd_q_f32_kernel<<<dim3(B * heads, (S + nw - 1) / nw), nw * 32, nw * (2 * S + 128) * sizeof(float), s>>>(
            sv->qkv[i], kb, sv->d_ctx, S, heads, 0.125f, sv->P, sv->dS, sv->d_qkv);
        F32_TRY(check_launch("attention_bwd_q_f32"));
        attention_bwd_kv_f32_kernel<<<dim3(B * heads, (S + nw - 1) / nw), nw * 32, 0, s>>>(
            sv->qkv[i], sv->d_ctx, sv->P, sv->dS, S, heads, 0.125f, sv->d_qkv);
        F32_TRY(check_launch("attention_bwd_kv_f32"));
        // dx = dq Wq + dk Wk + dv Wv + d_s1
        F32_TRY(linear_bwd(t, gt, p + "attention.self.query", sv->x[i], Hd, sv->d_qkv, 3 * Hd, Ti, dxo, Hd, sv->d_s, Hd, s));
        F32_TRY(linear_bwd(t, gt, p + "attention.self.key", sv->x[i], Hd, sv->d_qkv + Hd, 3 * Hd, Ti, sv->d_h1, Hd, dxo, Hd, s));
        F32_TRY(linear_bwd(t, gt, p + "attention.self.value", sv->x[i], Hd, sv->d_qkv + 2 * Hd, 3 * Hd, Ti, dxo, Hd, sv->d_h1, Hd, s));
    }
    // embeddings: x0 = LayerNorm(word[id] + position[j] + token_type[0])
    const std::string e = "text_encoder.encoder.embeddings.";
    const float* ge = get(e + "LayerNorm.weight");
    const RawTensor* we;
    F32_TRY(need(t, e + "word_embeddings.weight", &we));
    if (!ge) {
        set_last_error("fp32 check (train): embedding LayerNorm weight missing");
        return -2;
    }
    F32_TRY(ln_bwd_f32(sv->emb_sum, Hd, sv->dxa, Hd, ge, o.bert_ln_eps, Ti, Hd, sv->d_s, Hd,
                       grad_of(gt, e + "LayerNorm.weight"), grad_of(gt, e + "LayerNorm.bias"), s));
    float* gw = grad_of(gt, e + "word_embeddings.weight");
    float* gp = grad_of(gt, e + "position_embeddings.weight");
    float* gty = grad_of(gt, e + "token_type_embeddings.weight");
    if (gw || gp || gty) {
        embed_bwd_f32_kernel<<<nblk(T * Hd, 256), 256, 0, s>>>(sv->ids, sv->d_s, S, Hd, static_cast<int>(we->d[0]),
                                                               pad_idx, T * Hd, gw, gp, gty);
        F32_TRY(check_launch("embed_bwd_f32"));
    }
    return 0;
}

}  // namespace mrd
