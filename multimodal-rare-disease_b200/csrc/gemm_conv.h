// Implicit-GEMM launch plans.  One kernel family (conv_gemm_kernel) serves
//   * plain GEMMs              C[M,N] = act(A[M,K] * W[N,K]^T + bias (+ residual))      (BERT, heads)
//   * 1x1 / 3x3 convolutions   on NHWC bf16 activations, stride 1 or 2, BN folded       (ResNet50)
//   * the 7x7/2 stem           through an overlapping-window 5-D tensor map             (ResNet50)
// The A operand is always fetched by TMA from a (<=5)-D view of the activation tensor; im2col is
// never materialised.  See DESIGN.md "K1/K2".
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mrd {

enum Act : int { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2 };

struct TapDesc {
    int8_t map;  // which A tensor map (stride-2 convs read one of 4 parity phases)
    int8_t dh;   // row shift of the box, in (phase-)rows
    int8_t dw;   // column shift of the box
    int8_t pad_;
};

struct alignas(64) ConvGemmParams {
    CUtensorMap a_map[4];
    CUtensorMap b_map;
    CUtensorMap c_map;
    CUtensorMap r_map;              // residual, same logical shape / boxes as the output
    const float* bias;              // [Cout] fp32
    float* out_f32;                 // optional fp32 copy of the output, or null
    long long ld_f32;               // out_f32 row stride in elements
    const int* dyn_rows;            // optional (device): live GEMM rows <= M; tiles beyond are skipped
    int has_res;                    // 1: add the residual tile fetched through r_map
    int c_blocked;                  // 1: C is stored as [N/64][M][64] (one contiguous block per 64 columns)
    int stages, ring;               // operand pipeline depth, residual ring depth (16 KB sub-tiles)
    int w_shift;                    // added to the tile's first column (flat 3x3 mode: -1)
    int span_rows, a_stage_bytes, b_res_bytes;  // weights-resident modes: halo span rows, A stage / weight panel bytes
    int num_taps;                   // 1, 7 (stem) or 9
    int kc_per_tap;                 // K chunks (of BLOCK_K) per tap
    TapDesc taps[9];
    int tw, th, nb;                      // tile box: columns, rows, images  (tw*th*nb <= 128)
    int tiles_w, tiles_h, tiles_img;     // tiles per output row / column / batch
    int Wo, Ho, Nimg, Cout;              // logical output extent
    int n_tiles_n;                       // Cout / BLOCK_N
    int total_tiles;
    int act;
    int store_bf16;                      // 1: write bf16 output through c_map
    // split-K (generic mode only; weight gradients dW = dY^T X contract over the tokens, few output tiles):
    // the K loop of every output tile is cut into `ksplit` work items whose fp32 results are ADDED into
    // out_f32 (f32_accum = 1; the destination must be zeroed by the caller).  dyn_k (device, optional):
    // live contraction length in elements (token-packed operands), rounded up to 64 inside the kernel.
    int ksplit;
    int f32_accum;
    const int* dyn_k;
    // K-concatenated 1x1 convolutions (plan_conv1x1_dual: conv3 + downsample of a bottleneck's first block summed in
    // one accumulator): K chunks [0, kc_split) come from taps[0], the rest from taps[1]; 0 = every tap has
    // kc_per_tap chunks.  num_k_total = total K chunks in that mode.
    int kc_split;
    int num_k_total;
    // stem only: fused MaxPool2d(3, 2, 1) (TV:models/resnet.py:200,271).  When pool_out is set the epilogue does not
    // store the stem tile; it pools it in shared memory and folds the partial maxima into pool_out
    // [N, pool_h, pool_w, 64] bf16 with red.global.max (pool_out must be ZERO before the launch: post-ReLU values are
    // >= 0, so 0 is the identity of the max and doubles as the padding value).
    __nv_bfloat16* pool_out;
    int pool_h, pool_w;
    // LayerNorm in the epilogue (plan_gemm_ln): the n_tiles_n CTAs that hold one 128-row stripe of the whole output
    // row between them exchange per-row partial statistics through global memory (ln_stats) and store
    // LayerNorm(A W^T + bias + residual) * ln_g + ln_b.
    const float* ln_g;
    const float* ln_b;
    float ln_eps;
    // one record per 128-row stripe = [128][8] (mean, M2) partials + arrival / departure counters (zero between
    // launches: the last warp to leave a stripe resets them)
    float2* ln_stats;
};

struct GemmLaunch {
    ConvGemmParams p;
    int block_n;  // 64, 128 or 256
    int stem;     // 1: 5-D overlapping-window A map, BLOCK_K = 32
    int flat3;    // 1: flat-shift 3x3 stride-1 mode (halo span in smem, taps = row-shifted views)
    int lnc;      // 1: LayerNorm epilogue across the n_tiles_n CTAs of a stripe (plan_gemm_ln)
    int pair;     // 1: two-CTA clusters sharing each weight tile by TMA multicast (b_map's box is half a tile)
    int grid;
    double flops;  // algorithmic FLOPs (2*M*N*K, un-padded), for reporting
    double bytes;  // algorithmic bytes: A + W read once, C written once (+ residual read)
};

// Plain GEMM.  A: [M,K] bf16 with row stride lda; W: [N,K] bf16 (nn.Linear layout); C: [M,N] bf16
// with row stride ldc (may be null when only out_f32 is wanted).  K % 64 == 0, N % 64 == 0.
// c_blocked = 1: C is written as [N/64][M][64] instead of row-major [M][N] (ldc ignored): every
// 64-column block (one attention head of Q, K or V) becomes one contiguous [M,64] matrix.
int plan_gemm(GemmLaunch* out, const __nv_bfloat16* A, long long lda, int M, int K,
              const __nv_bfloat16* W, int N, const float* bias, __nv_bfloat16* C, long long ldc,
              const __nv_bfloat16* residual, long long ld_res, float* out_f32, long long ld_f32,
              int act, int c_blocked = 0);

// C = LayerNorm(A W^T + bias + residual) over the whole row (nn.LayerNorm(N), eps), gamma / beta fp32 [N]:
// HF:models/bert/modeling_bert.py:294-298,352-356 (dense -> dropout -> LayerNorm(x + input)) as ONE launch.
// N = c * 256 with c in [2, 4] (BERT-base: 3): c CTAs own a 128-row stripe.  Returns 1 (no error message) when N
// is outside that range - the caller then plans the GEMM and a LayerNorm launch.
// stats_ws (required, device, gemm_ln_ws_bytes(M) bytes, zeroed once by the caller): the CTAs of a stripe exchange
// the statistics through it in global memory.  Null returns -1.
size_t gemm_ln_ws_bytes(int M);
int plan_gemm_ln(GemmLaunch* out, const __nv_bfloat16* A, long long lda, int M, int K, const __nv_bfloat16* W, int N,
                 const float* bias, __nv_bfloat16* C, long long ldc, const __nv_bfloat16* residual, long long ld_res,
                 const float* gamma, const float* beta, float eps, void* stats_ws);

// ksize in {1,3}, stride in {1,2}, padding = ksize/2.  X: [N,H,W,Cin] bf16, Wt: [Cout][k][k][Cin]
// bf16 (BN already folded), Y: [N,H/stride,W/stride,Cout] bf16.  Cin % 64 == 0, Cout % 64 == 0.
// out_pad = 1: Y is a zero-bordered [N][Ho+2][Wo+2][Cout] tensor whose interior is written (feeds
// plan_conv3x3_flat).
int plan_conv(GemmLaunch* out, const __nv_bfloat16* X, int N, int H, int W, int Cin,
              const __nv_bfloat16* Wt, int Cout, int ksize, int stride, const float* bias,
              __nv_bfloat16* Y, const __nv_bfloat16* residual, int act, int out_pad = 0);

// Two 1x1 convolutions summed into one output: Y = act(X0 * W[:, :C0]^T + subsample_s(X1) * W[:, C0:]^T + bias).
// X0: [N,Ho,Wo,C0] (the bottleneck's conv2 output), X1: [N,Ho*s,Wo*s,C1] read at stride s in {1,2} (the block
// input), Wcat: [Cout][C0+C1] bf16, bias = the two folded BatchNorm shifts added.  This is conv3 + downsample +
// residual add of a bottleneck's first block (TV:models/resnet.py:143-163 with a downsample branch) as ONE GEMM
// over the concatenated K, so the downsample output never exists in memory.
int plan_conv1x1_dual(GemmLaunch* out, const __nv_bfloat16* X0, int C0, const __nv_bfloat16* X1, int C1,
                      int stride1, int N, int Ho, int Wo, const __nv_bfloat16* Wcat, int Cout,
                      const float* bias, __nv_bfloat16* Y, int act);

// 3x3 stride-1 pad-1 convolution in flat-shift mode.  Xpad: zero-bordered [N][H+2][W+2][Cin] bf16;
// Wt: [Cout][3][3][Cin]; Y: [N,H,W,Cout] (unpadded).  The halo span of a tile is loaded once per
// 64-channel chunk and the 9 taps are row-shifted UMMA views of it.  W <= 62.
// (Cin/64) * 9 weight tiles must fit in shared memory next to two halo spans: see conv3x3_flat_supported.
bool conv3x3_flat_supported(int H, int W, int Cin, int Cout);
int plan_conv3x3_flat(GemmLaunch* out, const __nv_bfloat16* Xpad, int N, int H, int W, int Cin,
                      const __nv_bfloat16* Wt, int Cout, const float* bias, __nv_bfloat16* Y, int act);

// 7x7 stride-2 pad-3 stem.  Xpad: [N][H+6][W+8][4] bf16 (zero border, channel 3 zero),
// Wst: [64][7][32] bf16 (tap row r, then 8 pixels x 4 channels; BN folded), Y: [N,H/2,W/2,64].
int plan_stem(GemmLaunch* out, const __nv_bfloat16* Xpad, int N, int H, int W,
              const __nv_bfloat16* Wst, const float* bias, __nv_bfloat16* Y, int act);
// The stem with the 3x3 / stride-2 / pad-1 max pooling fused into its epilogue: P [N,H/4,W/4,64] bf16 must be zeroed
// before every launch; the 112 x 112 stem output itself is never written.  act must be ReLU.
int plan_stem_pool(GemmLaunch* out, const __nv_bfloat16* Xpad, int N, int H, int W,
                   const __nv_bfloat16* Wst, const float* bias, __nv_bfloat16* P);

// Weight-gradient GEMM: out_f32[M,N] += A[M,K] * W[N,K]^T with fp32 accumulation across split-K work
// items (wide 128x256 tiles for operand reuse, K cut so that every SM gets a work item).  out_f32 must be
// zero before the launch.  dyn_k: optional device int, the live part of K (<= K).
int plan_gemm_splitk(GemmLaunch* out, const __nv_bfloat16* A, long long lda, int M, int K,
                     const __nv_bfloat16* W, int N, float* out_f32, long long ld_f32, const int* dyn_k);

int launch_gemm(const GemmLaunch* g, cudaStream_t stream);

int gemm_num_sms();

// Programmatic dependent launch for the GEMM/conv kernels (on by default; the engine turns it off
// while profiling so that per-launch event timings do not overlap).
void gemm_set_pdl(bool on);

}  // namespace mrd
