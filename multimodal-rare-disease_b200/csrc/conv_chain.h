// Bottleneck tail + next head in ONE persistent kernel (ResNet50 layer1 / layer2 are HBM-bound under per-conv
// fusion, SURVEY.md section 7): for every 128-pixel tile a CTA computes
//     y = relu(conv3_1x1(mid) [+ downsample_1x1(x)] + identity)          (TV:models/resnet.py:155-163, block i)
//     z = relu(conv1_1x1(y))                                              (TV:models/resnet.py:146-148, block i+1)
// with two tcgen05 pipelines side by side.  y is written once (the next block needs it as its identity) and the
// second pipeline reads the tile back a few microseconds later, while it is still in L2: the block's largest
// tensor is read from HBM once instead of twice.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mrd {

struct ChainPhase {
    CUtensorMap a_map[2];   // phase 0: conv2 output (+ block input when the downsample branch is fused); phase 1: y
    CUtensorMap b_map;      // weights [N][K] bf16, box {64, BLOCK_N}
    CUtensorMap c_map;      // output, box {64, tw, th, nb}
    CUtensorMap r_map;      // phase 0: identity, same boxes as the output
    const float* bias;      // [N] fp32
    int num_k;              // K chunks of 64
    int kc_split;           // > 0: chunks [0, kc_split) come from a_map[0], the rest from a_map[1]
    int n_tiles;            // N / BLOCK_N
    int act;
    int has_res;
};

struct alignas(64) ChainParams {
    ChainPhase ph[2];
    int tw, th, nb;                     // tile box: columns, rows, images (tw*th*nb <= 128)
    int tiles_w, tiles_h, tiles_img;
    int m_tiles;
    int stages1, stages2, ring;         // operand pipeline depths, residual ring depth (16 KB sub-tiles)
};

struct ChainLaunch {
    ChainParams p;
    int block_n2;   // 64 or 128 (phase 0 always uses 128-column tiles)
    int grid;
    int smem;
    double flops, bytes;
};

// X0: [N,Ho,Wo,C0] bf16 (conv2 output of block i).  X1 (optional): block input [N,Ho*s1,Wo*s1,C1] read at stride s1
// (downsample branch fused, W1cat = [Cout][C0+C1]); otherwise `identity` [N,Ho,Wo,Cout] is added.
// Y: [N,Ho,Wo,Cout] (block output).  W2: [C2][Cout], Z: [N,Ho,Wo,C2] or, with out_pad = 1, the interior of a
// zero-bordered [N][Ho+2][Wo+2][C2] tensor (input of the flat 3x3 convolution).  Both activations are ReLU.
// C0, C1 % 64 == 0, Cout % 128 == 0, C2 in {64, 128, 256}.
bool conv_chain_supported(int C0, int C1, int Cout, int C2);
int plan_conv_chain(ChainLaunch* out, const __nv_bfloat16* X0, int C0, const __nv_bfloat16* X1, int C1, int s1,
                    const __nv_bfloat16* identity, int N, int Ho, int Wo, const __nv_bfloat16* W1, int Cout,
                    const float* bias1, __nv_bfloat16* Y, const __nv_bfloat16* W2, int C2, const float* bias2,
                    __nv_bfloat16* Z, int out_pad);
int launch_conv_chain(const ChainLaunch* g, cudaStream_t stream);

}  // namespace mrd
