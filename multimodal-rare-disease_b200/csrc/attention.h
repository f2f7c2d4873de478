// K3: fused masked-softmax self-attention for BERT (S <= 512, head dim 64).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace mrd {

struct DropCfg;

// qkv: [B*S, 3*heads*64] bf16 (columns [Q | K | V], Q pre-scaled by 1/sqrt(64));
// mask_bias: [B,S] fp32 additive key bias (0 / -inf) or null; out: [B*S, heads*64] bf16.
// Replaces BertSelfAttention's SDPA call (HF:models/bert/modeling_bert.py:168-207,
// HF:integrations/sdpa_attention.py:92) without materialising the [B,1,S,S] mask.
// seq_off (optional, device, B+1 ints): token-packed layout - sample b owns rows
// [seq_off[b], seq_off[b+1]) of qkv/out and of mask_bias; S is then the maximum sequence length.
// rows_alloc: rows of the qkv / out allocations (>= the last row any sample touches; default B*S).
// S <= 128 runs on tcgen05 (TMA-fed 128x128 tiles, S and O in TMEM); longer sequences on mma.sync.
int attention_forward(const __nv_bfloat16* qkv, const float* mask_bias, const int* seq_off, int B,
                      int S, int heads, __nv_bfloat16* out, cudaStream_t stream,
                      long long rows_alloc = 0, int blocked = 0, const struct DropCfg* drop = nullptr);
// drop (train mode): dropout on the attention probabilities, element index ((b*heads + h)*S + q)*S + k
// (rng.cuh); attention_backward (train_kernels.h) recomputes the same mask.
// blocked = 1: qkv is [3*heads][rows_alloc][64] (what plan_gemm(c_blocked=1) writes): each head's Q, K
// and V tile is one contiguous block - streaming-friendly for the TMA loads of the tcgen05 path.
bool attention_prefers_blocked_qkv(int S);

// The attention probabilities themselves (what HF's eager attention returns with output_attentions=True,
// HF:models/bert/modeling_bert.py:115-140 in eval mode): probs[b,h,q,k] = softmax_k(q.k + mask_bias[b,k]) in fp32,
// [B,heads,S,S], for EVERY query row (padded ones included).  Dense layout: sample b owns rows [b*S, (b+1)*S) of
// qkv and mask_bias is [B,S] or null; rows_alloc / blocked as for attention_forward.  A masked key gets exactly 0;
// a sample without any attended key gets all-zero rows (attention_forward gives it a zero context).  S <= 512.
// attention_probs.cu: one tcgen05 product S = Q K^T per (sample, head, 128-query block), softmax from TMEM, and a
// write stream staged through shared memory (TMA stores when S % 4 == 0).
int attention_probs(const __nv_bfloat16* qkv, const float* mask_bias, int B, int S, int heads, float* probs,
                    cudaStream_t stream, long long rows_alloc = 0, int blocked = 0);
// 3-D TMA views {64 dims, rows, 3*heads blocks} of qkv with row boxes of 32 / 64 / 96 / 128 (attention.cu)
int encode_qkv_maps(CUtensorMap* maps, const __nv_bfloat16* qkv, int heads, long long rows_alloc, int blocked);

// test hook: force the mma.sync path for every S
void attention_set_tc(bool on);

}  // namespace mrd
