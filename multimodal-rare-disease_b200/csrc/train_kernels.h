// Kernels of the training step that are not contractions (SURVEY.md 8(f).1; reference:
// src/train.py:247-321, i.e. autograd through MultimodalClassifier.forward).  HBM-bound: 16-byte
// accesses, one warp per row for the row-wise ops.  The contractions of the backward pass reuse the
// tcgen05 GEMM (gemm_conv.cu) on transposed operands, see engine_train.cuh.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "rng.cuh"

namespace mrd {

// ---- dropout -------------------------------------------------------------------------------------
// y[r,c] = keep(r*width + c) ? x[r,c] * scale : 0   (nn.Dropout in train mode).  In place allowed.
// The same call is its own backward (apply it to the gradient).  rows bounded by *dyn_rows if given.
int dropout_bf16(const __nv_bfloat16* x, long long ldx, int rows, int width, const int* dyn_rows,
                 DropCfg d, __nv_bfloat16* y, long long ldy, cudaStream_t s);
int dropout_f32(const float* x, int rows, int width, DropCfg d, float* y, cudaStream_t s);
// y = dropout(relu(x)): Linear -> ReLU -> Dropout of the projection / fusion MLP / head, on the GEMM's output
int relu_dropout_f32(const float* x, int rows, int width, DropCfg d, float* y, cudaStream_t s);
// Dropout of the length-1 cross-attention weights (src/fusion_model.py:164-165): the softmax over one
// key is 1, so after dropout head h of row r carries weight w = keep(r*heads + h) ? scale : 0 and
// y[r, h*hd + j] = w * x[r, h*hd + j].  w_out (optional): [rows, heads].  Its own backward as well.
int head_dropout_f32(const float* x, int rows, int heads, int head_dim, DropCfg d, float* y,
                     float* w_out, cudaStream_t s);
// out[i] = keep(i) ? 1 : 0 for i < n (materialises a mask; tests and debugging)
int dropout_mask_f32(DropCfg d, long long n, float* out, cudaStream_t s);

// ---- LayerNorm -----------------------------------------------------------------------------------
// s = res + dropout(z);  y = LayerNorm(s) * gamma + beta   (HF:models/bert/modeling_bert.py:294-298,
// 352-356 in train mode).  s is stored (bf16) for the backward pass; statistics are taken from the
// stored (rounded) values so forward and backward agree.  width in {256,512,768,1024}.
int drop_add_ln_fwd(const __nv_bfloat16* z, const __nv_bfloat16* res, int rows, int width,
                    const int* dyn_rows, DropCfg d, const float* gamma, const float* beta, float eps,
                    __nv_bfloat16* s_out, __nv_bfloat16* y, cudaStream_t s);
// Backward of y = LayerNorm(s_in)*gamma + beta: dx = rstd * (g - mean(g) - xhat * mean(g*xhat)), g = dy*gamma;
// dgamma += sum_r dy*xhat, dbeta += sum_r dy (atomic accumulation into fp32; either may be null).
int ln_bwd_bf16(const __nv_bfloat16* s_in, const __nv_bfloat16* dy, const float* gamma, float eps,
                int rows, int width, const int* dyn_rows, __nv_bfloat16* dx, float* dgamma,
                float* dbeta, cudaStream_t s);
// fp32 variants for the batch-level layers (src/fusion_model.py:274-276); any width.
int ln_fwd_f32(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int rows,
               int width, float* y, long long ldy, cudaStream_t s);
int ln_bwd_f32(const float* x, long long ldx, const float* dy, long long lddy, const float* gamma,
               float eps, int rows, int width, float* dx, long long lddx, float* dgamma, float* dbeta,
               cudaStream_t s);

// ---- GELU (exact erf, HF:activations.py:70-90) -------------------------------------------------------
int gelu_fwd_bf16(const __nv_bfloat16* u, int rows, int width, const int* dyn_rows, __nv_bfloat16* g,
                  cudaStream_t s);
int gelu_bwd_bf16(const __nv_bfloat16* u, const __nv_bfloat16* dg, int rows, int width,
                  const int* dyn_rows, __nv_bfloat16* du, cudaStream_t s);

// ---- operand staging for the weight-gradient GEMMs ---------------------------------------------------
// y[c][r] = r < live ? x[r][c] : 0 for r < Kp; x: [rows, width] bf16 (row stride ldx), y: [width][Kp].
// dW = dY^T X contracts over tokens, so both operands are needed token-minor; columns beyond the live
// row count are zero-filled so stale rows of the token-packed buffers contribute nothing.
// two operands (same rows / Kp) in one launch (x1 may be null); colsum0 (optional): colsum0[c] += sum_r x0[r][c] over the live
// rows - the bias gradient of the dY operand, taken while the tile is in flight anyway
int transpose_pad2_bf16(const __nv_bfloat16* x0, long long ldx0, int width0, __nv_bfloat16* y0,
                        const __nv_bfloat16* x1, long long ldx1, int width1, __nv_bfloat16* y1, int rows,
                        const int* dyn_rows, int Kp, cudaStream_t s, float* colsum0 = nullptr);
// out[c] += scale * sum_r x[r,c]   (bias gradients)
int colsum_bf16(const __nv_bfloat16* x, long long ldx, int rows, int width, const int* dyn_rows,
                float scale, float* out, cudaStream_t s);
int colsum_f32(const float* x, long long ldx, int rows, int width, float* out, cudaStream_t s);
int scale_f32(float* x, long long n, float a, cudaStream_t s);
// dx = y > 0 ? dy : 0
int relu_bwd_f32(const float* y, const float* dy, long long n, float* dx, cudaStream_t s);
// dst (bf16 [*, width], already zero) row seq_off[b] = src[b] (fp32 [B, width]): the gradient of
// last_hidden_state[:, 0, :] (src/text_encoder.py:118) on the token-packed layout
int scatter_cls_rows_bf16(const float* src, const int* seq_off, int B, int width, __nv_bfloat16* dst,
                          cudaStream_t s);
// y[b] = x[seq_off[b]] as fp32
int gather_cls_rows_f32(const __nv_bfloat16* x, const int* seq_off, int B, int width, float* y,
                        cudaStream_t s);

// ---- embeddings ------------------------------------------------------------------------------------
// Backward of BertEmbeddings (HF:models/bert/modeling_bert.py:72-112): LayerNorm backward on the
// recomputed sum word[id] + position[j] + token_type[0], then scatter-add into the three tables
// (word rows with id == pad_idx receive no gradient, as nn.Embedding(padding_idx=...) does).
int embed_ln_bwd(const long long* ids, const int* row_tok, int rows, const int* dyn_rows, int S,
                 const __nv_bfloat16* word, const float* pos_type, const float* gamma, float eps,
                 int vocab, int pad_idx, const __nv_bfloat16* dy, float* dword, float* dpos,
                 float* dtype0, float* dgamma, float* dbeta, cudaStream_t s);

// ---- attention backward --------------------------------------------------------------------------
// Backward of softmax(Q K^T + key_bias) V with optional dropout on the probabilities (mma.sync m16n8k16).
// Sequences of at most 128 tokens: one 128x128 tile per (sample, head).  qkv / dqkv: [rows, 3*heads*64]
// bf16 token-major (Q already scaled by 1/sqrt(64): dQ is the gradient of the scaled Q); ctx = forward
// output O, dctx = its gradient: [rows, heads*64].  Layout arguments as attention_forward.
// S > 128 (up to 512): tiled over 128-query x 128-key blocks with the softmax statistics recomputed in a first
// pass; dK / dV are ACCUMULATED in fp32 into dkv_acc [rows, 2*heads*64] (K then V; zeroed by the caller) because
// several query blocks contribute to one key block - the caller converts them into dqkv's K / V columns; dQ is
// written to dqkv directly.  dkv_acc may be null when S <= 128.
int attention_backward(const __nv_bfloat16* qkv, const __nv_bfloat16* ctx, const __nv_bfloat16* dctx,
                       const float* mask_bias, const int* seq_off, int B, int S, int heads, DropCfg d,
                       __nv_bfloat16* dqkv, cudaStream_t s, float* dkv_acc = nullptr);

// ---- BatchNorm with batch statistics (frozen backbone under model.train(), TV:models/resnet.py:143-163) --
// Shifted sums over an NHWC bf16 tensor viewed as [rows, C] (C % 2 == 0): shift[c] = the mean of y[0..7, c]
// rounded to bf16 (written),
// sum[c] += sum_r (y[r,c] - shift[c]), sumsq[c] += sum_r (y[r,c] - shift[c])^2.  The shift keeps the variance
// free of the cancellation of sumsq/n - mean^2 when a channel's |mean| is large against its spread.
int bn_stats_bf16(const __nv_bfloat16* y, long long rows, int C, float* sum, float* sumsq, float* shift,
                  cudaStream_t s);
// y = act(y*scale[c] + shift[c] (+ identity)) in place on [rows, C] bf16 (C % 8 == 0), scale / shift derived per
// block from bn_stats_bf16's sums: d = sum/n, mean = shift + d, var = sumsq/n - d^2 (biased),
// scale = gamma*rsqrt(var+eps), shift = beta - mean*scale.
int bn_apply_stats_bf16(__nv_bfloat16* y, long long rows, int C, const float* sum, const float* sumsq,
                        const float* shift, const float* gamma, const float* beta, float eps,
                        const __nv_bfloat16* identity, int relu, cudaStream_t s);
// Running-statistics update of every BatchNorm layer of a forward in ONE launch (what nn.BatchNorm2d does in
// train mode: running <- (1-m)*running + m*(mean, var*n/(n-1))), from bn_stats_bf16's sums.  table: device
// array, one entry per layer.  Mirrored by mrd_bn_site (include/mrd_b200.h).
struct BnSite {
    const float* sum;
    const float* sumsq;
    const float* shift;
    float* running_mean;
    float* running_var;
    float n;
    int C;
};
int bn_update_running(const BnSite* table, int sites, int max_C, float momentum, cudaStream_t s);

}  // namespace mrd
