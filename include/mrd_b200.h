/* mrd_b200.h — C ABI of libmrd_b200.so: hand-written sm_100a kernels for the batched
 * MultimodalClassifier forward of ArshvirSk/Multimodal-Rare-Disease.
 *
 * The reference has no FFI (it is pure Python on top of torch/torchvision/transformers); this header
 * defines the boundary a host binds instead of the reference's nn.Module.forward bodies.  Each entry
 * point names the reference code it replaces (paths relative to the reference repo; TV: = torchvision
 * 0.26 models/resnet.py, HF: = transformers 5.5 models/bert/modeling_bert.py).
 *
 * Conventions
 *   - every function returns 0 on success or a negative code; mrd_last_error() gives the message
 *     (thread-local, valid until the next failing call on that thread);
 *   - all data pointers are DEVICE pointers on the context's device; nothing here allocates, frees or
 *     retains caller memory (a context owns only its packed weights, workspace and TMA descriptors);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - there is no CPU path: calls fail (or the process faults) without an sm_100 GPU.
 */
#ifndef MRD_B200_H_
#define MRD_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define MRD_ABI_VERSION 1

/* activation codes for the GEMM / conv epilogues */
#define MRD_ACT_NONE 0
#define MRD_ACT_RELU 1
#define MRD_ACT_GELU 2 /* exact erf GELU, HF:activations.py:70-90 */

/* element type codes for inputs whose dtype the reference API leaves open */
#define MRD_DT_I64 0
#define MRD_DT_I32 1
#define MRD_DT_F32 2
#define MRD_DT_U8 3 /* also torch.bool */
#define MRD_DT_BF16 4

const char* mrd_last_error(void);
int mrd_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * Context: packed weights + workspace + launch plans for one device.
 * ---------------------------------------------------------------------------------------------- */
typedef struct mrd_ctx mrd_ctx;

/* Creates a context on the CURRENT CUDA device. */
int mrd_ctx_create(mrd_ctx** out);
int mrd_ctx_destroy(mrd_ctx* ctx);

/* Micro-batch sizes the forward is tiled into (activations of one micro-batch are sized to stay in
 * L2).  img_chunk: images per ResNet pass; seq_chunk_tokens: tokens (B*S) per BERT pass.  <=0 keeps
 * the default. */
int mrd_ctx_configure(mrd_ctx* ctx, int img_chunk, int seq_chunk_tokens);

/* Scalar options: "bert_heads" (12), "bert_ln_eps" (1e-12), "bn_eps" (1e-5), "fusion_ln_eps" (1e-5),
 * "fusion_heads" (8), "fusion_residual" (1), "head_act" (MRD_ACT_RELU).  Set before load_weights.
 * "fp32_check" (0): forwards run the plain-fp32 reference kernels.  "load_sync" (1): load_weights synchronises
 * the device before re-packing and the stream afterwards; 0 drops both.  "train.*": options of the training step.
 * Any other key returns -1 ("unknown option"). */
int mrd_ctx_set_option(mrd_ctx* ctx, const char* key, double value);

/* Hands the context the model's fp32 parameters/buffers by their state_dict names
 * (cnn_encoder.backbone.*, cnn_encoder.projection.{0,3}.*, text_encoder.encoder.*,
 * fusion.fusion_layer.*, classifier.classifier.{0,3,6}.*).  shapes[i*4..i*4+3] holds up to 4 dims
 * (unused = 0).  The context converts them into its own packed bf16/fp32 device buffers (BN folded
 * into the conv weights: TV:143-163; QKV concatenated, 1/sqrt(d) folded into Wq: HF:177-179;
 * value_proj/output_proj of the length-1 cross attention pre-multiplied: src/fusion_model.py:149-176).
 * Groups that are absent (e.g. no text_encoder.* names) are simply not loaded; a forward that needs
 * a missing group fails.  May be called again after the parameters change. */
int mrd_ctx_load_weights(mrd_ctx* ctx, int n, const char* const* names, const void* const* ptrs,
                         const long long* shapes, void* stream);

/* CNNEncoder.forward (src/cnn_encoder.py:168-184): ResNet50 backbone (TV:266-282) + projection
 * (src/cnn_encoder.py:46-51, eval mode).  images: [B,3,H,W] NCHW, img_dtype MRD_DT_F32 or MRD_DT_BF16.
 * emb: f32 [B,E].  feat_pooled (optional): f32 [B,2048] backbone output after global average pooling.
 * feat_map (optional): f32 [B,2048,H/32,W/32] NCHW layer4 output (src/cnn_encoder.py:200-226). */
int mrd_cnn_encoder_fwd(mrd_ctx* ctx, const void* images, int img_dtype, int B, int H, int W,
                        float* emb, float* feat_pooled, float* feat_map, void* stream);

/* TextEncoder.forward (src/text_encoder.py:95-127): BertModel (HF:628-691) -> CLS row of the last
 * hidden state (eval mode, pooler skipped: its output is unused with use_pooler_output=False).
 * ids: i64 [B,S]; mask: [B,S] of mask_dtype, key j of sample b is attended iff mask[b,j] != 0
 * (HF:masking_utils.py:1001-1088); mask may be NULL (= all ones).  cls: f32 [B,768].
 * last_hidden (optional): f32 [B,S,768]; requesting it keeps every token (no packing) so padded rows
 * are computed as the reference computes them.  all_hidden (optional, needs last_hidden): f32
 * [layers+1,B,S,768], HF's hidden_states tuple (src/text_encoder.py:129-149). */
int mrd_text_encoder_fwd(mrd_ctx* ctx, const long long* ids, const void* mask, int mask_dtype, int B,
                         int S, float* cls, float* last_hidden, float* all_hidden, void* stream);

/* MultimodalFusion.forward with fusion_type="attention" (src/fusion_model.py:245-291).
 * img_emb f32 [B,Di], txt_emb f32 [B,Dt] -> fused f32 [B,Hd].  attn_i2t / attn_t2i (optional):
 * f32 [B,heads,1,1], the cross-attention weights (identically 1: softmax over one key). */
int mrd_fusion_fwd(mrd_ctx* ctx, const float* img_emb, const float* txt_emb, int B, float* fused,
                   float* attn_i2t, float* attn_t2i, void* stream);

/* ClassificationHead.forward + softmax (src/multimodal_classifier.py:73-83,166-167).
 * x f32 [B,Din] -> logits f32 [B,C], probs f32 [B,C] (probs optional). */
int mrd_head_fwd(mrd_ctx* ctx, const float* x, int B, float* logits, float* probs, void* stream);

/* The batch-level tail of MultimodalClassifier.forward as ONE launch (tail_fused_kernel): AttentionFusion
 * (src/fusion_model.py:245-291) -> ClassificationHead -> softmax (src/multimodal_classifier.py:73-83,166-167).
 * img_emb f32 [B,Di], txt_emb f32 [B,Dt] -> logits f32 [B,C]; probs f32 [B,C] and fused f32 [B,Hd] optional.
 * Falls back to the per-layer launches of mrd_fusion_fwd + mrd_head_fwd when the shapes are outside the fused
 * kernel's range. */
int mrd_fusion_head_fwd(mrd_ctx* ctx, const float* img_emb, const float* txt_emb, int B, float* fused,
                        float* logits, float* probs, void* stream);

/* MultimodalClassifier.forward (src/multimodal_classifier.py:131-177).  Outputs other than logits
 * are optional (NULL to skip): probs [B,C], img_emb [B,512], txt_emb [B,768], fused [B,512],
 * attn_i2t / attn_t2i [B,heads,1,1]. */
int mrd_multimodal_fwd(mrd_ctx* ctx, const void* images, int img_dtype, const long long* ids,
                       const void* mask, int mask_dtype, int B, int H, int W, int S, float* logits,
                       float* probs, float* img_emb, float* txt_emb, float* fused, float* attn_i2t,
                       float* attn_t2i, void* stream);

/* Profile mode: while enabled every kernel launch of a forward is bracketed by CUDA events on the
 * launching stream.  mrd_ctx_profile(ctx, 1) clears earlier records and starts; _report synchronises
 * and writes one CSV line per kernel label into buf: label,category(0 tensor|1 attention|2 memory),
 * launches,total_ms,algorithmic_flops,algorithmic_bytes.  Used by bench.py for the roofline object. */
int mrd_ctx_profile(mrd_ctx* ctx, int enable);
int mrd_ctx_profile_report(mrd_ctx* ctx, char* buf, int cap);

/* Kernel launches issued by this context since creation (for the bench's gpu_launches claim). */
long long mrd_ctx_launch_count(const mrd_ctx* ctx);
/* Bytes of device memory the context currently owns (weights + workspace). */
long long mrd_ctx_device_bytes(const mrd_ctx* ctx);

/* ------------------------------------------------------------------------------------------------
 * Individual kernels (unit tests, ncu captures, other hosts).  bf16 tensors are passed as void*.
 * ---------------------------------------------------------------------------------------------- */

/* C[M,N] = act(A[M,K] * W[N,K]^T + bias (+ residual)); nn.Linear (HF:177-179,295,340,353;
 * src/cnn_encoder.py:46-51; src/fusion_model.py:212-240; src/multimodal_classifier.py:44-58).
 * tcgen05/TMEM tiles fed by TMA.  K % 64 == 0, N % 64 == 0; lda/ldc/ld_res in elements (% 8 == 0).
 * C (bf16) and out_f32 are each optional. */
int mrd_gemm_bf16(const void* A, long long lda, int M, int K, const void* W, int N,
                  const float* bias, void* C, long long ldc, const void* residual,
                  long long ld_res, float* out_f32, long long ld_f32, int act, void* stream);

/* C = LayerNorm(A W^T + bias + residual) * gamma + beta over whole rows (HF:models/bert/modeling_bert.py:294-298,
 * 352-356: BertSelfOutput / BertOutput) in ONE launch: N/256 CTAs own a 128-row stripe and exchange the row
 * statistics through stats_ws.  N in {512, 768, 1024}, otherwise -1.  residual may be NULL.
 * stats_ws (required): a device buffer of mrd_gemm_ln_ws_bytes(M) bytes, zeroed once by the caller (the kernel leaves
 * it zero again); NULL returns -1. */
int mrd_gemm_ln_bf16(const void* A, long long lda, int M, int K, const void* W, int N, const float* bias, void* C,
                     long long ldc, const void* residual, long long ld_res, const float* gamma, const float* beta,
                     float eps, void* stats_ws, void* stream);
long long mrd_gemm_ln_ws_bytes(int M);

/* out_f32[M,N] += A[M,K] * W[N,K]^T on the same tcgen05 kernel with split-K: 128x256 output tiles whose K loop is
 * cut into work items (one per SM), fp32 partial sums added into out_f32 (which the caller ZEROES first) with
 * red.global.add.v4.f32.  The weight gradients dW = dY^T X of the training step (few output tiles, K = tokens).
 * dyn_k (optional, device int): live part of K; the operands must be zero between it and the next multiple of 64. */
int mrd_gemm_splitk_f32(const void* A, long long lda, int M, int K, const void* W, int N, float* out_f32,
                        long long ld_f32, const int* dyn_k, void* stream);

/* Conv2d(k in {1,3}, stride in {1,2}, pad k/2, no bias) + folded BatchNorm + optional residual +
 * activation on NHWC bf16 (TV:143-163).  Wt: [Cout][k][k][Cin] bf16 with the BN scale folded in,
 * bias: f32 [Cout] = beta - mean*scale.  Cin % 64 == 0, Cout % 64 == 0.
 * out_pad = 1: Y is a zero-bordered [N][H/stride+2][W/stride+2][Cout] tensor and only its interior is
 * written (the input layout of mrd_conv3x3_flat_bf16). */
int mrd_conv2d_nhwc_bf16(const void* X, int N, int H, int W, int Cin, const void* Wt, int Cout,
                         int ksize, int stride, const float* bias, void* Y, const void* residual,
                         int act, int out_pad, void* stream);

/* conv3 + downsample + residual add + ReLU of a bottleneck's FIRST block (TV:143-163 with self.downsample) as one
 * GEMM over the concatenated K: Y = act(X0 * Wcat[:, :C0]^T + X1[:, ::stride, ::stride] * Wcat[:, C0:]^T + bias).
 * X0: [N,Ho,Wo,C0] bf16 (conv2 output), X1: [N,Ho*stride,Wo*stride,C1] bf16 (block input), stride in {1,2};
 * Wcat: [Cout][C0+C1] bf16 (both BN scales folded), bias: f32 [Cout] = sum of the two folded BN shifts.
 * The downsample branch's output is never written to memory.  C0, C1, Cout % 64 == 0. */
int mrd_conv1x1_dual_bf16(const void* X0, int C0, const void* X1, int C1, int stride, int N, int Ho, int Wo,
                          const void* Wcat, int Cout, const float* bias, void* Y, int act, void* stream);

/* Tail of bottleneck i and head of bottleneck i+1 in one launch (TV:143-163 across two blocks):
 *   Y = relu(X0 * W1[:, :C0]^T (+ X1[:, ::stride, ::stride] * W1[:, C0:]^T) + bias1 (+ identity))
 *   Z = relu(Y * W2^T + bias2)
 * X0: [N,Ho,Wo,C0] bf16; X1 (optional, downsample fused; then identity must be NULL): [N,Ho*stride,Wo*stride,C1];
 * identity (optional): [N,Ho,Wo,Cout]; W1: [Cout][C0(+C1)], W2: [C2][Cout]; Y: [N,Ho,Wo,Cout];
 * Z: [N,Ho,Wo,C2], or with out_pad = 1 the interior of a zero-bordered [N][Ho+2][Wo+2][C2] tensor.
 * Y is written once and re-read by the second product while the tile is still in L2: per block one read of the
 * block's largest tensor from HBM is saved.  Cout % 128 == 0, C2 in {64,128,256}, C0 / C1 % 64 == 0. */
int mrd_conv_chain_bf16(const void* X0, int C0, const void* X1, int C1, int stride, const void* identity, int N,
                        int Ho, int Wo, const void* W1, int Cout, const float* bias1, void* Y, const void* W2,
                        int C2, const float* bias2, void* Z, int out_pad, void* stream);

/* Conv2d(3, stride 1, pad 1) + folded BN + activation in flat-shift mode: Xpad is the zero-bordered
 * [N][H+2][W+2][Cin] bf16 input; the halo span of each tile is fetched once per 64-channel chunk and
 * the 9 taps are row-shifted tcgen05 views of it (TV:143-163 conv2 of layer1/layer2).  W <= 62. */
int mrd_conv3x3_flat_bf16(const void* Xpad, int N, int H, int W, int Cin, const void* Wt, int Cout,
                          const float* bias, void* Y, int act, void* stream);

/* ResNet stem: Conv2d(3,64,7,stride 2,pad 3) + BN + ReLU (TV:197-199,268-270) on the repacked image
 * Xpad [N][H+6][W+8][4] bf16; Wst [64][7][32] bf16; Y [N,H/2,W/2,64] bf16. */
int mrd_stem_conv_bf16(const void* Xpad, int N, int H, int W, const void* Wst, const float* bias,
                       void* Y, int act, void* stream);

/* The stem with MaxPool2d(3, stride 2, pad 1) (TV:200,271) fused into its epilogue: P [N,H/4,W/4,64] bf16.
 * P must be ZERO when the launch starts (window maxima are folded into it with red.global.max); the 112 x 112 stem
 * output is never written.  H % 32 == 0, W % 32 == 0. */
int mrd_stem_pool_bf16(const void* Xpad, int N, int H, int W, const void* Wst, const float* bias, void* P,
                       void* stream);

/* [N,3,H,W] (f32 or bf16) -> Xpad [N][H+6][W+8][4] bf16, pixel (h,w) at (h+3,w+3), zero elsewhere. */
int mrd_repack_images(const void* x_nchw, int img_dtype, int N, int H, int W, void* xpad,
                      void* stream);

/* MaxPool2d(3, stride 2, pad 1) on NHWC bf16 (TV:200,271). */
int mrd_maxpool3x3s2(const void* x, int N, int H, int W, int C, void* y, void* stream);

/* AdaptiveAvgPool2d(1)+flatten on NHWC bf16 (TV:205,278-279): [N,HW,C] -> [N,C] (bf16 and/or f32). */
int mrd_global_avgpool(const void* x, int N, int HW, int C, void* y_bf16, float* y_f32,
                       void* stream);

/* y = LayerNorm(x (+ residual)) (HF:294-298,352-356; src/fusion_model.py:274-276); one warp per row,
 * fp32 statistics.  width in {256,512,768,1024}. */
int mrd_layernorm_residual(const void* x, long long ldx, const void* residual, long long ldr,
                           const float* gamma, const float* beta, float eps, int rows, int width,
                           void* y_bf16, long long ldy, float* y_f32, long long ldy32,
                           void* stream);

/* BertEmbeddings (HF:72-112): word[ids] + position + token_type[0] -> LayerNorm -> bf16 [B*S,768].
 * word_emb bf16 [vocab,768]; pos_type_emb f32 [>=S,768] = position + token_type[0]. */
int mrd_bert_embed_layernorm(const long long* ids, int B, int S, const void* word_emb,
                             const float* pos_type_emb, const float* gamma, const float* beta,
                             float eps, int vocab, void* y_bf16, void* stream);

/* Fused masked-softmax self-attention (HF:168-207 + integrations/sdpa_attention.py:92).
 * qkv: bf16 [B*S, 3*heads*64] rows = tokens, columns = [Q | K | V], Q already scaled by 1/sqrt(64).
 * mask_bias: f32 [B,S], 0 for attended keys and -inf for padded keys, or NULL.  out: bf16
 * [B*S, heads*64]. */
int mrd_attention_bf16(const void* qkv, const float* mask_bias, int B, int S, int heads, void* out,
                       void* stream);

/* Token packing for BERT ("unpadding"): keeps token (b,j) iff mask[b,j] != 0 or j == 0 (or all tokens
 * when keep_all).  Outputs (device): seq_off[B+1] first packed row of each sequence, row_tok[r] =
 * b*S+j of packed row r, row_bias[r] = 0 / -inf key bias, n_rows[0] = number of packed rows.
 * scratch: B ints.  Padded positions are masked as keys (HF:masking_utils.py:1001-1088) and only the
 * CLS row is read downstream (src/text_encoder.py:118), so dropping them changes no output. */
int mrd_compact_tokens(const void* mask, int mask_dtype, int B, int S, int keep_all, int* seq_off,
                       int* row_tok, float* row_bias, int* n_rows, int* scratch, void* stream);

/* mrd_attention_bf16 on the token-packed layout: sample b owns rows [seq_off[b], seq_off[b+1]) of qkv,
 * row_bias and out; max_len bounds the sequence lengths; total_rows = rows of qkv / out. */
int mrd_attention_varlen_bf16(const void* qkv, const float* row_bias, const int* seq_off, int B,
                              int max_len, int heads, long long total_rows, void* out, void* stream);

/* Attention with max length <= 128 runs on tcgen05 (TMEM scores, TMA tiles); 0 forces the mma.sync
 * kernel that serves longer sequences (process-wide test switch). */
int mrd_attention_use_tcgen05(int on);

/* attention_mask [B,S] -> additive key bias (0 / -inf). */
int mrd_mask_to_bias(const void* mask, int mask_dtype, int B, int S, float* bias, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training step (SURVEY.md 8(f).1): what autograd does around MultimodalClassifier.forward in the
 * reference's trainers (src/train.py:247-321, src/train_multimodal.py:508-543).  The loss, gradient
 * clipping and the optimizer stay with the caller, exactly as in the reference (criterion(logits,
 * labels).backward(); clip_grad_norm_; optimizer.step()): the library provides the forward in train
 * mode and the backward from d(loss)/d(logits) to every trainable parameter.
 * ---------------------------------------------------------------------------------------------- */

/* Train-mode forward (dropout active with the probabilities set through mrd_ctx_set_option:
 * "train.p_bert_hidden" 0.1, "train.p_bert_attn" 0.1, "train.p_text_out" 0.1, "train.p_cnn_proj" 0.5,
 * "train.p_fusion" 0.3, "train.p_head" 0.5, "train.pad_idx" 0; masks are a pure function of `seed`).
 * Keeps the activations the backward needs inside the context; one forward may be pending at a time.
 * The ResNet50 backbone must be frozen (the reference default, src/config.py:64) and is run forward
 * only.  S <= 512, B <= one pass.  logits: f32 [B,C]. */
int mrd_train_forward(mrd_ctx* ctx, const void* images, int img_dtype, const long long* ids,
                      const void* mask, int mask_dtype, int B, int H, int W, int S,
                      unsigned long long seed, float* logits, void* stream);

/* Backward of the pending mrd_train_forward.  dlogits: f32 [B,C].  names/grads: state_dict names of the
 * parameters that want a gradient and their f32 gradient buffers (same shapes as the parameters,
 * ZEROED by the caller: gradients are accumulated into them); parameters that are absent or NULL are
 * treated as frozen.  query_proj / key_proj of the length-1 cross attention receive exactly zero
 * (softmax over one key, src/fusion_model.py:138-165), the BERT pooler is unused. */
int mrd_train_backward(mrd_ctx* ctx, const float* dlogits, int n, const char* const* names,
                       float* const* grads, void* stream);

/* The same two calls with the extra tensors Grad-CAM needs (notebooks/explainability.ipynb cell 3 hooks
 * cnn_encoder.get_attention_layer() = backbone.layer4, src/cnn_encoder.py:186-198, and back-propagates one logit):
 * feat_map (optional): f32 [B,2048,H/32,W/32] NCHW, the layer4 output of this forward (BatchNorm on running
 * statistics only); img_emb / txt_emb / fused (optional): the three embeddings of this forward as
 * MultimodalClassifier.forward(return_embeddings=True) returns them (src/multimodal_classifier.py:168-175), f32
 * [B,512] / [B,768] / [B,512]; d_pooled (optional): f32 [B,2048] = d(loss)/d(backbone output after global average pooling), from
 * which d(loss)/d(layer4 output) = d_pooled / (H/32 * W/32) at every position.  With every dropout probability 0
 * this is the eval-mode forward made differentiable.  When no text_encoder.* gradient is requested the text branch
 * of the backward is skipped. */
int mrd_train_forward_ex(mrd_ctx* ctx, const void* images, int img_dtype, const long long* ids,
                         const void* mask, int mask_dtype, int B, int H, int W, int S,
                         unsigned long long seed, float* logits, float* feat_map, float* img_emb,
                         float* txt_emb, float* fused, void* stream);
int mrd_train_backward_ex(mrd_ctx* ctx, const float* dlogits, int n, const char* const* names,
                          float* const* grads, float* d_pooled, void* stream);

/* The backward in stages, for data-parallel hosts that overlap the gradient all-reduce with the rest of the backward
 * (SURVEY.md 8(e)): _begin takes what mrd_train_backward_ex takes and enqueues nothing; _stages runs stages
 * [first, last) on `stream` - they must be run in order, each once.  Stage 0 = head + fusion + image projection (all
 * their gradients are complete when it returns), stage 1 + k = BERT layer (layers - 1 - k), the last stage = the
 * embeddings; mrd_train_backward_num_stages = layers + 2.  The gradient buffers handed to _begin must stay valid
 * until the last stage has been enqueued. */
int mrd_train_backward_begin(mrd_ctx* ctx, const float* dlogits, int n, const char* const* names,
                             float* const* grads, float* d_pooled);
int mrd_train_backward_stages(mrd_ctx* ctx, int first, int last, void* stream);
int mrd_train_backward_num_stages(mrd_ctx* ctx);

/* out[i] = 1 if element i of dropout site `site` is kept under (seed, p), else 0 (i < n).  The masks
 * of mrd_train_forward are reproducible with this (tests; csrc/rng.cuh documents the site ids and the
 * element indexing). */
int mrd_dropout_mask(unsigned long long seed, unsigned int site, double p, long long n, float* out,
                     void* stream);

/* mrd_attention_bf16 with dropout on the probabilities (train mode); element index of (b,h,q,k) is
 * ((b*heads + h)*S + q)*S + k. */
int mrd_attention_train_bf16(const void* qkv, const float* mask_bias, int B, int S, int heads,
                             unsigned long long seed, unsigned int site, double p, void* out,
                             void* stream);

/* Backward of the fused attention: qkv / dqkv bf16 [rows, 3*heads*64], ctx (forward output) / dctx bf16
 * [rows, heads*64]; dQ is the gradient of the pre-scaled Q.  seq_off as mrd_attention_varlen_bf16 or
 * NULL for the dense layout.  S <= 128: one 128x128 tile per (sample, head), dkv_acc may be NULL.
 * 128 < S <= 512: tiled over 128x128 blocks; dkv_acc = ZEROED f32 scratch [rows, 2*heads*64] (dK | dV are
 * accumulated there across query blocks and then converted into dqkv), rows = row count of the tensors. */
int mrd_attention_bwd_bf16(const void* qkv, const void* ctx, const void* dctx, const float* mask_bias,
                           const int* seq_off, int B, int S, int heads, unsigned long long seed,
                           unsigned int site, double p, void* dqkv, float* dkv_acc, long long rows,
                           void* stream);

/* Backward of y = LayerNorm(s)*gamma + beta on bf16 rows: dx (bf16), dgamma / dbeta accumulated into
 * f32 buffers (either may be NULL).  width in {256,512,768,1024}. */
int mrd_layernorm_bwd_bf16(const void* s_in, const void* dy, const float* gamma, float eps, int rows,
                           int width, void* dx, float* dgamma, float* dbeta, void* stream);

/* The other non-GEMM kernels of the training step, one entry each (unit tests, captures of one kernel).  Each
 * calls the kernel's host wrapper in csrc/train_kernels.h with the same arguments; the semantics are documented
 * there.  bf16 tensors are void*, dropout is given as (seed, site, p) as in mrd_dropout_mask, and dyn_rows
 * (optional, device int) bounds the row count on the device as in the engine's token-packed buffers. */
int mrd_dropout_bf16(const void* x, long long ldx, int rows, int width, const int* dyn_rows,
                     unsigned long long seed, unsigned int site, double p, void* y, long long ldy, void* stream);
int mrd_dropout_f32(const float* x, int rows, int width, unsigned long long seed, unsigned int site, double p,
                    float* y, void* stream);
int mrd_relu_dropout_f32(const float* x, int rows, int width, unsigned long long seed, unsigned int site,
                         double p, float* y, void* stream);
int mrd_head_dropout_f32(const float* x, int rows, int heads, int head_dim, unsigned long long seed,
                         unsigned int site, double p, float* y, float* w_out, void* stream);
/* s_out = res + dropout(z) (bf16), y = LayerNorm(s_out)*gamma + beta (bf16); width in {256,512,768,1024}. */
int mrd_drop_add_layernorm_bf16(const void* z, const void* res, int rows, int width, const int* dyn_rows,
                                unsigned long long seed, unsigned int site, double p, const float* gamma,
                                const float* beta, float eps, void* s_out, void* y, void* stream);
int mrd_layernorm_f32(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int rows,
                      int width, float* y, long long ldy, void* stream);
int mrd_layernorm_bwd_f32(const float* x, long long ldx, const float* dy, long long lddy, const float* gamma,
                          float eps, int rows, int width, float* dx, long long lddx, float* dgamma, float* dbeta,
                          void* stream);
int mrd_gelu_fwd_bf16(const void* u, int rows, int width, const int* dyn_rows, void* g, void* stream);
int mrd_gelu_bwd_bf16(const void* u, const void* dg, int rows, int width, const int* dyn_rows, void* du,
                      void* stream);
/* y0 [width0][Kp] = x0^T, y1 [width1][Kp] = x1^T (x1 may be NULL), zero-filled past the live rows; colsum0
 * (optional) += the column sums of x0 over the live rows. */
int mrd_transpose_pad2_bf16(const void* x0, long long ldx0, int width0, void* y0, const void* x1, long long ldx1,
                            int width1, void* y1, int rows, const int* dyn_rows, int Kp, void* stream,
                            float* colsum0);
int mrd_colsum_bf16(const void* x, long long ldx, int rows, int width, const int* dyn_rows, float scale,
                    float* out, void* stream);
int mrd_colsum_f32(const float* x, long long ldx, int rows, int width, float* out, void* stream);
int mrd_relu_bwd_f32(const float* y, const float* dy, long long n, float* dx, void* stream);
int mrd_scatter_cls_rows_bf16(const float* src, const int* seq_off, int B, int width, void* dst, void* stream);
int mrd_gather_cls_rows_f32(const void* x, const int* seq_off, int B, int width, float* y, void* stream);
/* Backward of the BERT embeddings (word[id] + pos_type[pos] -> LayerNorm, width 768) into the three tables and
 * the LayerNorm parameters (each output optional, all accumulated); word rows of pad_idx get nothing. */
int mrd_embed_layernorm_bwd(const long long* ids, const int* row_tok, int rows, const int* dyn_rows, int S,
                            const void* word, const float* pos_type, const float* gamma, float eps, int vocab,
                            int pad_idx, const void* dy, float* dword, float* dpos, float* dtype0, float* dgamma,
                            float* dbeta, void* stream);
/* BatchNorm with batch statistics on bf16 [rows, C]: sums about a per-channel shift (the mean of the first 8
 * rows, written to shift[C]; mean = shift + sum/rows, var = sumsq/rows - (sum/rows)^2), the in-place normalise
 * (+ identity, + ReLU), and the running-statistics update of several layers from one table of mrd_bn_site. */
int mrd_bn_stats_bf16(const void* y, long long rows, int C, float* sum, float* sumsq, float* shift, void* stream);
int mrd_bn_apply_stats_bf16(void* y, long long rows, int C, const float* sum, const float* sumsq,
                            const float* shift, const float* gamma, const float* beta, float eps,
                            const void* identity, int relu, void* stream);
typedef struct {
    const float* sum;    /* mrd_bn_stats_bf16's outputs for this layer */
    const float* sumsq;
    const float* shift;
    float* running_mean; /* updated in place */
    float* running_var;
    float n;             /* rows the sums cover */
    int C;
} mrd_bn_site;
int mrd_bn_update_running(const mrd_bn_site* table_dev, int sites, int max_C, float momentum, void* stream);

/* clip_grad_norm_(parameters, max_norm) + torch.optim.AdamW.step() of the reference's loop (src/train.py:307-320,
 * :193-198) as two multi-tensor launches without a host synchronisation: the global L2 norm of all gradients is
 * reduced into sqnorm_dev[0] (its square; zeroed inside), the clip coefficient min(1, max_norm / (norm + 1e-6)) is
 * derived on the device (max_norm <= 0: no clipping) and applied to the gradient as it is read (the gradient
 * tensors themselves are NOT rescaled).  Decoupled weight decay, bias correction with the common `step` (1-based)
 * exactly as torch.optim.AdamW (amsgrad = False).  All arrays are DEVICE arrays: tensors_dev[n_tensors] (g may be
 * NULL: parameter skipped), and a chunk table - chunk c covers elements [chunk_off_dev[c], + chunk_elems) of tensor
 * chunk_tensor_dev[c]; chunk_elems % 4 == 0. */
typedef struct {
    float* p;        /* parameter, updated in place */
    const float* g;  /* gradient */
    float* m;        /* exp_avg */
    float* v;        /* exp_avg_sq */
    long long n;     /* elements */
    float lr;
    float wd;
} mrd_adamw_tensor;
int mrd_adamw_step(const mrd_adamw_tensor* tensors_dev, int n_tensors, const int* chunk_tensor_dev,
                   const long long* chunk_off_dev, int n_chunks, int chunk_elems, float beta1, float beta2,
                   float eps, long long step, float max_norm, float* sqnorm_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MRD_B200_H_ */
