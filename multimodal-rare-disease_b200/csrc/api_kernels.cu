// C-ABI entry points for the individual kernels (unit tests, ncu captures, other hosts).
// All pointers are device pointers; `stream` is a cudaStream_t passed as void*.

#include <mrd_b200.h>

#include "elementwise.h"
#include "attention.h"
#include "conv_chain.h"
#include "gemm_conv.h"
#include "tma_host.h"
#include "train_kernels.h"
#include "rng.cuh"

using namespace mrd;

typedef __nv_bfloat16 bf16;

static_assert(sizeof(BnSite) == sizeof(mrd_bn_site), "layout");

extern "C" {

const char* mrd_last_error(void) { return get_last_error(); }

int mrd_gemm_bf16(const void* A, long long lda, int M, int K, const void* W, int N,
                  const float* bias, void* C, long long ldc, const void* residual,
                  long long ld_res, float* out_f32, long long ld_f32, int act, void* stream) {
    GemmLaunch g;
    int rc = plan_gemm(&g, static_cast<const __nv_bfloat16*>(A), lda, M, K,
                       static_cast<const __nv_bfloat16*>(W), N, bias,
                       static_cast<__nv_bfloat16*>(C), ldc,
                       static_cast<const __nv_bfloat16*>(residual), ld_res, out_f32, ld_f32, act);
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_gemm_ln_bf16(const void* A, long long lda, int M, int K, const void* W, int N, const float* bias, void* C,
                     long long ldc, const void* residual, long long ld_res, const float* gamma, const float* beta,
                     float eps, void* stats_ws, void* stream) {
    GemmLaunch g;
    int rc = plan_gemm_ln(&g, static_cast<const __nv_bfloat16*>(A), lda, M, K, static_cast<const __nv_bfloat16*>(W), N,
                          bias, static_cast<__nv_bfloat16*>(C), ldc, static_cast<const __nv_bfloat16*>(residual), ld_res,
                          gamma, beta, eps, stats_ws);
    if (rc > 0) {
        set_last_error("mrd_gemm_ln_bf16: N=%d outside the fused LayerNorm kernel's range (512 / 768 / 1024)", N);
        return -1;
    }
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

long long mrd_gemm_ln_ws_bytes(int M) { return static_cast<long long>(gemm_ln_ws_bytes(M)); }

int mrd_gemm_splitk_f32(const void* A, long long lda, int M, int K, const void* W, int N, float* out_f32,
                        long long ld_f32, const int* dyn_k, void* stream) {
    GemmLaunch g;
    int rc = plan_gemm_splitk(&g, static_cast<const __nv_bfloat16*>(A), lda, M, K,
                              static_cast<const __nv_bfloat16*>(W), N, out_f32, ld_f32, dyn_k);
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_conv2d_nhwc_bf16(const void* X, int N, int H, int W, int Cin, const void* Wt, int Cout,
                         int ksize, int stride, const float* bias, void* Y, const void* residual,
                         int act, int out_pad, void* stream) {
    GemmLaunch g;
    int rc = plan_conv(&g, static_cast<const __nv_bfloat16*>(X), N, H, W, Cin,
                       static_cast<const __nv_bfloat16*>(Wt), Cout, ksize, stride, bias,
                       static_cast<__nv_bfloat16*>(Y), static_cast<const __nv_bfloat16*>(residual),
                       act, out_pad);
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_conv1x1_dual_bf16(const void* X0, int C0, const void* X1, int C1, int stride, int N, int Ho, int Wo,
                          const void* Wcat, int Cout, const float* bias, void* Y, int act, void* stream) {
    GemmLaunch g;
    int rc = plan_conv1x1_dual(&g, static_cast<const __nv_bfloat16*>(X0), C0, static_cast<const __nv_bfloat16*>(X1),
                               C1, stride, N, Ho, Wo, static_cast<const __nv_bfloat16*>(Wcat), Cout, bias,
                               static_cast<__nv_bfloat16*>(Y), act);
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_conv_chain_bf16(const void* X0, int C0, const void* X1, int C1, int stride, const void* identity, int N,
                        int Ho, int Wo, const void* W1, int Cout, const float* bias1, void* Y, const void* W2,
                        int C2, const float* bias2, void* Z, int out_pad, void* stream) {
    typedef const __nv_bfloat16* cb;
    ChainLaunch g;
    int rc = plan_conv_chain(&g, static_cast<cb>(X0), C0, static_cast<cb>(X1), C1, stride, static_cast<cb>(identity), N,
                             Ho, Wo, static_cast<cb>(W1), Cout, bias1, static_cast<__nv_bfloat16*>(Y),
                             static_cast<cb>(W2), C2, bias2, static_cast<__nv_bfloat16*>(Z), out_pad);
    if (rc) return rc;
    return launch_conv_chain(&g, static_cast<cudaStream_t>(stream));
}

int mrd_conv3x3_flat_bf16(const void* Xpad, int N, int H, int W, int Cin, const void* Wt, int Cout,
                          const float* bias, void* Y, int act, void* stream) {
    GemmLaunch g;
    int rc = plan_conv3x3_flat(&g, static_cast<const __nv_bfloat16*>(Xpad), N, H, W, Cin,
                               static_cast<const __nv_bfloat16*>(Wt), Cout, bias,
                               static_cast<__nv_bfloat16*>(Y), act);
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_stem_conv_bf16(const void* Xpad, int N, int H, int W, const void* Wst, const float* bias,
                       void* Y, int act, void* stream) {
    GemmLaunch g;
    int rc = plan_stem(&g, static_cast<const __nv_bfloat16*>(Xpad), N, H, W,
                       static_cast<const __nv_bfloat16*>(Wst), bias,
                       static_cast<__nv_bfloat16*>(Y), act);
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_stem_pool_bf16(const void* Xpad, int N, int H, int W, const void* Wst, const float* bias, void* P,
                       void* stream) {
    GemmLaunch g;
    int rc = plan_stem_pool(&g, static_cast<const __nv_bfloat16*>(Xpad), N, H, W,
                            static_cast<const __nv_bfloat16*>(Wst), bias, static_cast<__nv_bfloat16*>(P));
    if (rc) return rc;
    return launch_gemm(&g, static_cast<cudaStream_t>(stream));
}

int mrd_repack_images(const void* x_nchw, int img_dtype, int N, int H, int W, void* xpad,
                      void* stream) {
    if (img_dtype != MRD_DT_F32 && img_dtype != MRD_DT_BF16) {
        set_last_error("mrd_repack_images: images must be f32 or bf16");
        return -1;
    }
    return repack_images(x_nchw, img_dtype == MRD_DT_BF16, N, H, W,
                         static_cast<__nv_bfloat16*>(xpad), static_cast<cudaStream_t>(stream));
}

int mrd_maxpool3x3s2(const void* x, int N, int H, int W, int C, void* y, void* stream) {
    return maxpool3x3s2(static_cast<const __nv_bfloat16*>(x), N, H, W, C,
                        static_cast<__nv_bfloat16*>(y), static_cast<cudaStream_t>(stream));
}

int mrd_global_avgpool(const void* x, int N, int HW, int C, void* y_bf16, float* y_f32,
                       void* stream) {
    return global_avgpool(static_cast<const __nv_bfloat16*>(x), N, HW, C,
                          static_cast<__nv_bfloat16*>(y_bf16), y_f32,
                          static_cast<cudaStream_t>(stream));
}

int mrd_layernorm_residual(const void* x, long long ldx, const void* residual, long long ldr,
                           const float* gamma, const float* beta, float eps, int rows, int width,
                           void* y_bf16, long long ldy, float* y_f32, long long ldy32,
                           void* stream) {
    return layernorm_residual(static_cast<const __nv_bfloat16*>(x), ldx,
                              static_cast<const __nv_bfloat16*>(residual), ldr, gamma, beta, eps,
                              rows, width, static_cast<__nv_bfloat16*>(y_bf16), ldy, y_f32, ldy32,
                              static_cast<cudaStream_t>(stream));
}

int mrd_bert_embed_layernorm(const long long* ids, int B, int S, const void* word_emb,
                             const float* pos_type_emb, const float* gamma, const float* beta,
                             float eps, int vocab, void* y_bf16, void* stream) {
    return bert_embed_layernorm(ids, B, S, static_cast<const __nv_bfloat16*>(word_emb),
                                pos_type_emb, gamma, beta, eps, vocab,
                                static_cast<__nv_bfloat16*>(y_bf16),
                                static_cast<cudaStream_t>(stream));
}

int mrd_attention_bf16(const void* qkv, const float* mask_bias, int B, int S, int heads,
                       void* out, void* stream) {
    return attention_forward(static_cast<const __nv_bfloat16*>(qkv), mask_bias, nullptr, B, S, heads,
                             static_cast<__nv_bfloat16*>(out), static_cast<cudaStream_t>(stream));
}

int mrd_attention_varlen_bf16(const void* qkv, const float* row_bias, const int* seq_off, int B,
                              int max_len, int heads, long long total_rows, void* out, void* stream) {
    if (!seq_off) {
        set_last_error("mrd_attention_varlen_bf16: seq_off is required");
        return -1;
    }
    if (total_rows <= 0) {
        set_last_error("mrd_attention_varlen_bf16: total_rows must be the row count of qkv / out");
        return -1;
    }
    return attention_forward(static_cast<const __nv_bfloat16*>(qkv), row_bias, seq_off, B, max_len,
                             heads, static_cast<__nv_bfloat16*>(out),
                             static_cast<cudaStream_t>(stream), total_rows);
}

int mrd_attention_use_tcgen05(int on) {
    attention_set_tc(on != 0);
    return 0;
}

int mrd_compact_tokens(const void* mask, int mask_dtype, int B, int S, int keep_all, int* seq_off,
                       int* row_tok, float* row_bias, int* n_rows, int* scratch, void* stream) {
    return compact_tokens(mask, mask_dtype, B, S, keep_all, seq_off, row_tok, row_bias, n_rows,
                          scratch, static_cast<cudaStream_t>(stream));
}

int mrd_mask_to_bias(const void* mask, int mask_dtype, int B, int S, float* bias, void* stream) {
    return mask_to_bias(mask, mask_dtype, B, S, bias, static_cast<cudaStream_t>(stream));
}

// ---- training-step kernels (train_kernels.h)

int mrd_dropout_bf16(const void* x, long long ldx, int rows, int width, const int* dyn_rows,
                     unsigned long long seed, unsigned int site, double p, void* y, long long ldy, void* stream) {
    return dropout_bf16(static_cast<const bf16*>(x), ldx, rows, width, dyn_rows, make_drop(seed, site, p),
                        static_cast<bf16*>(y), ldy, static_cast<cudaStream_t>(stream));
}

int mrd_dropout_f32(const float* x, int rows, int width, unsigned long long seed, unsigned int site, double p,
                    float* y, void* stream) {
    return dropout_f32(x, rows, width, make_drop(seed, site, p), y, static_cast<cudaStream_t>(stream));
}

int mrd_relu_dropout_f32(const float* x, int rows, int width, unsigned long long seed, unsigned int site,
                         double p, float* y, void* stream) {
    return relu_dropout_f32(x, rows, width, make_drop(seed, site, p), y, static_cast<cudaStream_t>(stream));
}

int mrd_head_dropout_f32(const float* x, int rows, int heads, int head_dim, unsigned long long seed,
                         unsigned int site, double p, float* y, float* w_out, void* stream) {
    return head_dropout_f32(x, rows, heads, head_dim, make_drop(seed, site, p), y, w_out,
                            static_cast<cudaStream_t>(stream));
}

int mrd_drop_add_layernorm_bf16(const void* z, const void* res, int rows, int width, const int* dyn_rows,
                                unsigned long long seed, unsigned int site, double p, const float* gamma,
                                const float* beta, float eps, void* s_out, void* y, void* stream) {
    return drop_add_ln_fwd(static_cast<const bf16*>(z), static_cast<const bf16*>(res), rows, width, dyn_rows,
                           make_drop(seed, site, p), gamma, beta, eps, static_cast<bf16*>(s_out),
                           static_cast<bf16*>(y), static_cast<cudaStream_t>(stream));
}

int mrd_layernorm_f32(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int rows,
                      int width, float* y, long long ldy, void* stream) {
    return ln_fwd_f32(x, ldx, gamma, beta, eps, rows, width, y, ldy, static_cast<cudaStream_t>(stream));
}

int mrd_layernorm_bwd_f32(const float* x, long long ldx, const float* dy, long long lddy, const float* gamma,
                          float eps, int rows, int width, float* dx, long long lddx, float* dgamma, float* dbeta,
                          void* stream) {
    return ln_bwd_f32(x, ldx, dy, lddy, gamma, eps, rows, width, dx, lddx, dgamma, dbeta,
                      static_cast<cudaStream_t>(stream));
}

int mrd_gelu_fwd_bf16(const void* u, int rows, int width, const int* dyn_rows, void* g, void* stream) {
    return gelu_fwd_bf16(static_cast<const bf16*>(u), rows, width, dyn_rows, static_cast<bf16*>(g),
                         static_cast<cudaStream_t>(stream));
}

int mrd_gelu_bwd_bf16(const void* u, const void* dg, int rows, int width, const int* dyn_rows, void* du,
                      void* stream) {
    return gelu_bwd_bf16(static_cast<const bf16*>(u), static_cast<const bf16*>(dg), rows, width, dyn_rows,
                         static_cast<bf16*>(du), static_cast<cudaStream_t>(stream));
}

int mrd_transpose_pad2_bf16(const void* x0, long long ldx0, int width0, void* y0, const void* x1, long long ldx1,
                            int width1, void* y1, int rows, const int* dyn_rows, int Kp, void* stream,
                            float* colsum0) {
    return transpose_pad2_bf16(static_cast<const bf16*>(x0), ldx0, width0, static_cast<bf16*>(y0),
                               static_cast<const bf16*>(x1), ldx1, width1, static_cast<bf16*>(y1), rows, dyn_rows, Kp,
                               static_cast<cudaStream_t>(stream), colsum0);
}

int mrd_colsum_bf16(const void* x, long long ldx, int rows, int width, const int* dyn_rows, float scale,
                    float* out, void* stream) {
    return colsum_bf16(static_cast<const bf16*>(x), ldx, rows, width, dyn_rows, scale, out,
                       static_cast<cudaStream_t>(stream));
}

int mrd_colsum_f32(const float* x, long long ldx, int rows, int width, float* out, void* stream) {
    return colsum_f32(x, ldx, rows, width, out, static_cast<cudaStream_t>(stream));
}

int mrd_relu_bwd_f32(const float* y, const float* dy, long long n, float* dx, void* stream) {
    return relu_bwd_f32(y, dy, n, dx, static_cast<cudaStream_t>(stream));
}

int mrd_scatter_cls_rows_bf16(const float* src, const int* seq_off, int B, int width, void* dst, void* stream) {
    return scatter_cls_rows_bf16(src, seq_off, B, width, static_cast<bf16*>(dst), static_cast<cudaStream_t>(stream));
}

int mrd_gather_cls_rows_f32(const void* x, const int* seq_off, int B, int width, float* y, void* stream) {
    return gather_cls_rows_f32(static_cast<const bf16*>(x), seq_off, B, width, y, static_cast<cudaStream_t>(stream));
}

int mrd_embed_layernorm_bwd(const long long* ids, const int* row_tok, int rows, const int* dyn_rows, int S,
                            const void* word, const float* pos_type, const float* gamma, float eps, int vocab,
                            int pad_idx, const void* dy, float* dword, float* dpos, float* dtype0, float* dgamma,
                            float* dbeta, void* stream) {
    return embed_ln_bwd(ids, row_tok, rows, dyn_rows, S, static_cast<const bf16*>(word), pos_type, gamma, eps, vocab,
                        pad_idx, static_cast<const bf16*>(dy), dword, dpos, dtype0, dgamma, dbeta,
                        static_cast<cudaStream_t>(stream));
}

int mrd_bn_stats_bf16(const void* y, long long rows, int C, float* sum, float* sumsq, float* shift, void* stream) {
    return bn_stats_bf16(static_cast<const bf16*>(y), rows, C, sum, sumsq, shift, static_cast<cudaStream_t>(stream));
}

int mrd_bn_apply_stats_bf16(void* y, long long rows, int C, const float* sum, const float* sumsq,
                            const float* shift, const float* gamma, const float* beta, float eps,
                            const void* identity, int relu, void* stream) {
    return bn_apply_stats_bf16(static_cast<bf16*>(y), rows, C, sum, sumsq, shift, gamma, beta, eps,
                               static_cast<const bf16*>(identity), relu, static_cast<cudaStream_t>(stream));
}

int mrd_bn_update_running(const mrd_bn_site* table_dev, int sites, int max_C, float momentum, void* stream) {
    return bn_update_running(reinterpret_cast<const BnSite*>(table_dev), sites, max_C, momentum,
                             static_cast<cudaStream_t>(stream));
}

}  // extern "C"
