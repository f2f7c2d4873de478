// fp32 check mode: the whole MultimodalClassifier forward in plain fp32 CUDA (SIMT FFMA, no bf16
// storage anywhere, BatchNorm un-folded), driven from the caller's raw fp32 parameters.  It is the
// "fp32 check mode" of BASELINE.json's north_star (logits within 1e-4 of the reference's own fp32
// forward): slow by design - a verification instrument for the fast bf16/tcgen05 path, selected with
// mrd_ctx_set_option(ctx, "fp32_check", 1).
#pragma once

#include <cuda_runtime.h>

#include <string>
#include <unordered_map>

namespace mrd {

struct RawTensor {
    const float* p = nullptr;
    long long d[4] = {0, 0, 0, 0};
    long long numel() const {
        long long n = 1;
        for (int i = 0; i < 4; ++i)
            if (d[i] > 0) n *= d[i];
        return n;
    }
};
typedef std::unordered_map<std::string, RawTensor> RawTable;

struct Fp32Opts {
    int bert_heads = 12;
    float bert_ln_eps = 1e-12f, bn_eps = 1e-5f, fusion_ln_eps = 1e-5f;
    int fusion_heads = 8, fusion_residual = 1, head_act = 1;
};

struct Fp32Arena {
    void* base = nullptr;
    size_t bytes = 0, used = 0;
};

// Each stage mirrors one module forward of the reference; outputs are fp32 device buffers owned by
// the caller.  Stages return 0 or a negative code (message via mrd_last_error()).
int fp32_cnn_encoder(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const float* images, int B,
                     int H, int W, float* emb, float* pooled, float* fmap, cudaStream_t s);
int fp32_text_encoder(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const long long* ids,
                      const void* mask, int mask_dtype, int B, int S, float* cls, float* last_hidden,
                      float* all_hidden, float* attn_probs, cudaStream_t s);
int fp32_fusion(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const float* img, const float* txt,
                int B, float* fused, float* attn_i2t, float* attn_t2i, cudaStream_t s);
int fp32_head(const RawTable& t, const Fp32Opts& o, Fp32Arena* ws, const float* x, int B, float* logits,
              float* probs, cudaStream_t s);
void fp32_arena_free(Fp32Arena* ws);

// ---- fp32 check of the TRAINING step (text encoder) ------------------------------------------------------
// The BERT encoder forward in plain fp32 with every tensor its backward needs kept, and the matching backward
// (autograd through HF:models/bert/modeling_bert.py:72-112,168-207,294-298,339-356 restated by hand: LayerNorm,
// exact-erf GELU, softmax attention, embeddings), all dropout probabilities 0.  Dense [B*S] rows exactly as the
// reference computes them (padded rows included; they receive and propagate zero gradients).  Together with the
// fp32 batch-level layers of the training step this gives per-parameter gradients that agree with the reference's
// autograd to fp32 rounding: the instrument that separates structural errors of the bf16 step from rounding.
struct Fp32TrainSave {
    Fp32Arena ws;
    int B = 0, S = 0, Hd = 0, F = 0, L = 0;
    bool valid = false, has_mask = false;
    const long long* ids = nullptr;
    float *bias = nullptr, *emb_sum = nullptr, *x_final = nullptr;
    float *x[48], *qkv[48], *ctx[48], *s1[48], *h1[48], *u[48], *g[48], *s2[48];
    float *dxa = nullptr, *dxb = nullptr, *d_s = nullptr, *d_big = nullptr, *d_h1 = nullptr, *d_ctx = nullptr,
          *d_qkv = nullptr, *P = nullptr, *dS = nullptr;
};
typedef std::unordered_map<std::string, float*> Fp32GradTable;

// cls: f32 [B, hidden] = last hidden state of the first token (src/text_encoder.py:118)
int fp32_bert_train_forward(const RawTable& t, const Fp32Opts& o, Fp32TrainSave* sv, const long long* ids,
                            const void* mask, int mask_dtype, int B, int S, float* cls, cudaStream_t s);
// d_cls: f32 [B, hidden].  Gradients are ACCUMULATED into the (zeroed) buffers of `grads`, keyed by state_dict name;
// absent names are treated as frozen.
int fp32_bert_train_backward(const RawTable& t, const Fp32Opts& o, Fp32TrainSave* sv, const float* d_cls,
                             const Fp32GradTable& grads, int pad_idx, cudaStream_t s);

}  // namespace mrd
