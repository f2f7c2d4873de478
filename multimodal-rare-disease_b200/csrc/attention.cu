// K3: fused masked-softmax self-attention (flash-style, one pass over the keys).
//
// One CTA = one (sample, head, BLOCK_M query rows); each warp owns 16 query rows.  Keys/values are
// streamed in blocks of 64 through a cp.async double buffer in 128B-XOR-swizzled shared memory;
// QK^T and PV run on mma.sync m16n8k16 (bf16 in, fp32 accumulate) with the probabilities kept in
// registers between the two products; softmax statistics are fp32 and online.  The key-padding mask
// is a per-key additive bias ([B,S], 0 / -inf) staged once in shared memory: the [B,1,S,S] mask of
// HF:masking_utils.py:1001-1088 is never built, and 64-key blocks whose keys are all padded are
// skipped outright.  At BERT-base sizes attention is 2.7 % (S=128) to 10 % (S=512) of the forward's
// FLOPs, which is why it stays on the legacy tensor path while the GEMMs/convs use tcgen05.

#include "attention.h"

#include <math.h>
#include <stdint.h>

#include "ptx.cuh"
#include "rng.cuh"
#include "tma_host.h"

namespace mrd {

namespace {

bool g_attention_tc = true;

constexpr int kHeadDim = 64;
constexpr int kBlockN = 64;
constexpr int kMaxS = 512;
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() {
    asm volatile("cp.async.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                            uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1,
                                                  uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0,
                                         uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, "
        "{%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// rows x 64 bf16 tile, global row stride ld (elements) -> swizzled smem (128 B per row).  NT threads:
// thread t always moves 16-byte chunk (t & 7) of rows (t >> 3) + k * NT/8, so the address arithmetic
// is one pointer increment per row.
template <int NT>
__device__ __forceinline__ void load_tile(uint32_t dst, const __nv_bfloat16* base, long long ld,
                                          int row0, int rows, int S, int tid) {
    const int c = tid & 7;
    int r = tid >> 3;
    const __nv_bfloat16* src = base + static_cast<long long>(row0 + r) * ld + c * 8;
    uint32_t d = dst + r * 128 + ((c ^ (r & 7)) << 4);   // (r & 7) is invariant: rows advance by NT/8 = 16 or 32
#pragma unroll
    for (; r < rows; r += NT / 8) {
        const bool ok = row0 + r < S;
        cp_async16(d, ok ? src : base, ok);
        src += static_cast<long long>(NT / 8) * ld;
        d += (NT / 8) * 128;
    }
}

// bar.sync with an OR reduction of one predicate over the participating threads
__device__ __forceinline__ bool named_bar_or(int id, int nthreads, bool pred) {
    uint32_t r;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.u32 q, %1, 0;\n\t"
        "barrier.cta.red.or.pred p, %2, %3, q;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(r)
        : "r"(static_cast<uint32_t>(pred)), "r"(id), "r"(nthreads)
        : "memory");
    return r != 0;
}

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// seq_off == null: dense layout, sample b owns rows [b*S_max, (b+1)*S_max) and mask_bias is [B,S_max].
// seq_off != null: token-packed layout, sample b owns rows [seq_off[b], seq_off[b+1]) and mask_bias is
// indexed by packed row.
// One CTA = one (sample, BLOCK_M query rows, group of `hpg` heads).  The CTA walks its heads and their
// 64-key blocks as one flat item list with a two-deep cp.async pipeline (the next item's K/V - and the
// next head's Q - stream in while the current item is computed), so the global-load latency is paid
// once per CTA instead of once per head.
template <int BLOCK_M, bool DROP>
__global__ void __launch_bounds__(BLOCK_M * 2, BLOCK_M == 64 ? 4 : 2)
attention_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ mask_bias,
                 const int* __restrict__ seq_off, int S_max, int heads, int hpg,
                 __nv_bfloat16* __restrict__ out, DropCfg drop) {
    constexpr int NT = BLOCK_M * 2;
    constexpr int QBYTES = BLOCK_M * 128, KVBYTES = kBlockN * 128;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t q_s = smem_u32(smem);            // 2 Q buffers
    const uint32_t k_s = q_s + 2 * QBYTES;          // 2 K buffers
    const uint32_t v_s = k_s + 2 * KVBYTES;         // 2 V buffers
    float* bias_s = reinterpret_cast<float*>(smem + 2 * QBYTES + 4 * KVBYTES);
    int* kb_list = reinterpret_cast<int*>(bias_s + kMaxS);
    int* nkb_s = kb_list + 8;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tq = lane & 3;
    const int q0 = blockIdx.x * BLOCK_M, b = blockIdx.z;
    const int h_begin = blockIdx.y * hpg;
    const int nh = min(hpg, heads - h_begin);
    long long off;
    int S;
    if (seq_off) {
        off = __ldg(seq_off + b);
        S = __ldg(seq_off + b + 1) - static_cast<int>(off);
    } else {
        off = static_cast<long long>(b) * S_max;
        S = S_max;
    }
    if (q0 >= S || nh <= 0) return;  // uniform for the whole CTA
    const long long ld = 3LL * heads * kHeadDim;
    const long long ldo = static_cast<long long>(heads) * kHeadDim;
    const __nv_bfloat16* row0 = qkv + off * ld;

    // item = (head, key block); block 0 is always visited (it holds the CLS key), later blocks only
    // when they contain an attended key
    const int nkb_total = (S + kBlockN - 1) / kBlockN;
    auto issue = [&](int item, int nkb) {
        const int hh = item / nkb, ki = item - hh * nkb;
        const __nv_bfloat16* q_base = row0 + (h_begin + hh) * kHeadDim;
        const int kb = ki == 0 ? 0 : kb_list[ki];
        if (ki == 0) load_tile<NT>(q_s + (hh & 1) * QBYTES, q_base, ld, q0, BLOCK_M, S, tid);
        load_tile<NT>(k_s + (item & 1) * KVBYTES, q_base + heads * kHeadDim, ld, kb * kBlockN, kBlockN, S, tid);
        load_tile<NT>(v_s + (item & 1) * KVBYTES, q_base + 2 * heads * kHeadDim, ld, kb * kBlockN, kBlockN, S, tid);
        cp_async_commit();
    };
    issue(0, 1 << 30);  // (head 0, block 0): does not depend on the bias pass below

    for (int i = tid; i < nkb_total * kBlockN; i += NT)
        bias_s[i] = i < S ? (mask_bias ? __ldg(mask_bias + off + i) : 0.0f) : -INFINITY;
    __syncthreads();
    if (warp == 0) {
        int cnt = 1;
        if (lane == 0) kb_list[0] = 0;
        for (int kb = 1; kb < nkb_total; ++kb) {
            const bool v = bias_s[kb * kBlockN + lane] > -INFINITY ||
                           bias_s[kb * kBlockN + 32 + lane] > -INFINITY;
            if (__any_sync(0xffffffffu, v)) {
                if (lane == 0) kb_list[cnt] = kb;
                ++cnt;
            }
        }
        if (lane == 0) *nkb_s = cnt;
    }
    __syncthreads();
    const int nkb = *nkb_s;
    const int items = nh * nkb;

    // a warp whose 16 query rows all lie beyond the sequence only helps with the loads
    const bool warp_active = q0 + warp * 16 < S;

    float o[8][4];
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.0f, l1 = 0.0f;
    uint32_t qf[4][4];

    // per-lane ldmatrix offsets (swizzled), computed once: K tiles are read as [key][d] 8x8 blocks,
    // V tiles transposed
    const int mi = lane >> 3, x7 = lane & 7;
    const uint32_t k_row = static_cast<uint32_t>(((mi >> 1) * 8 + x7) * 128);
    const uint32_t v_row = static_cast<uint32_t>(((mi & 1) * 8 + x7) * 128);
    uint32_t k_col[4], v_col[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        k_col[i] = static_cast<uint32_t>(((i * 2 + (mi & 1)) ^ x7) << 4);
        v_col[i] = static_cast<uint32_t>(((i * 2 + (mi >> 1)) ^ x7) << 4);
    }

    for (int item = 0; item < items; ++item) {
        const int buf = item & 1;
        if (item + 1 < items) {
            issue(item + 1, nkb);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();

        if (!warp_active) {
            __syncthreads();
            continue;
        }
        const int hh = item / nkb, ki = item - hh * nkb;
        const int kb = kb_list[ki];
        const uint32_t qbuf = q_s + (hh & 1) * QBYTES;
        // keys of this block that exist: 8-key MMA tiles beyond them are skipped (their scores stay
        // 0 + (-inf) bias, their probabilities 0)
        const int nvalid = min(kBlockN, S - kb * kBlockN);
        if (ki == 0) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const int r = warp * 16 + (lane & 15);
                const int c = kk * 2 + (lane >> 4);
                ldmatrix_x4(qbuf + r * 128 + ((c ^ (r & 7)) << 4), qf[kk][0], qf[kk][1], qf[kk][2],
                            qf[kk][3]);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.0f;
            m0 = m1 = -INFINITY;
            l0 = l1 = 0.0f;
        }

        // ---- S = Q K^T (16 x 64 per warp)
        float s[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.0f;
        const uint32_t kt = k_s + buf * KVBYTES;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
            for (int np = 0; np < 4; ++np) {
                if (np * 16 >= nvalid) break;
                uint32_t b0, b1, b2, b3;
                ldmatrix_x4(kt + np * 2048 + k_row + k_col[kk], b0, b1, b2, b3);
                mma_bf16(s[np * 2], qf[kk], b0, b1);
                mma_bf16(s[np * 2 + 1], qf[kk], b2, b3);
            }
        }

        // ---- online softmax (rows g and g+8 of this warp's 16)
        const float* bb = bias_s + kb * kBlockN + tq * 2;
        float mx0 = m0, mx1 = m1;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j * 8 >= nvalid) {  // no key in this 8-wide tile: probabilities are exactly 0
                s[j][0] = s[j][1] = s[j][2] = s[j][3] = -INFINITY;
                continue;
            }
            const float2 b01 = *reinterpret_cast<const float2*>(bb + j * 8);
            const float b0 = b01.x, b1 = b01.y;
            s[j][0] += b0; s[j][1] += b1; s[j][2] += b0; s[j][3] += b1;
            mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
            mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float mu0 = mx0 == -INFINITY ? 0.0f : mx0;
        const float mu1 = mx1 == -INFINITY ? 0.0f : mx1;
        const float corr0 = fast_exp2((m0 - mu0) * kLog2e);
        const float corr1 = fast_exp2((m1 - mu1) * kLog2e);
        m0 = mx0; m1 = mx1;
        l0 *= corr0; l1 *= corr1;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            o[j][0] *= corr0; o[j][1] *= corr0; o[j][2] *= corr1; o[j][3] *= corr1;
        }
        const float ms0 = mu0 * kLog2e, ms1 = mu1 * kLog2e;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j * 8 >= nvalid) {
                s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.0f;
                continue;
            }
            s[j][0] = fast_exp2(fmaf(s[j][0], kLog2e, -ms0));
            s[j][1] = fast_exp2(fmaf(s[j][1], kLog2e, -ms0));
            s[j][2] = fast_exp2(fmaf(s[j][2], kLog2e, -ms1));
            s[j][3] = fast_exp2(fmaf(s[j][3], kLog2e, -ms1));
            l0 += s[j][0] + s[j][1];
            l1 += s[j][2] + s[j][3];
        }

        if (DROP) {
            // train mode: the probabilities that feed P V are dropped / rescaled; l0 / l1 above stay undropped
            const unsigned long long row_idx =
                (static_cast<unsigned long long>(b * heads + h_begin + hh) * S_max + (q0 + warp * 16 + g)) * S_max;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const unsigned long long k0 = static_cast<unsigned long long>(kb * kBlockN + j * 8 + tq * 2);
                s[j][0] = drop_keep(drop, row_idx + k0) ? s[j][0] * drop.scale : 0.0f;
                s[j][1] = drop_keep(drop, row_idx + k0 + 1) ? s[j][1] * drop.scale : 0.0f;
                s[j][2] = drop_keep(drop, row_idx + 8ull * S_max + k0) ? s[j][2] * drop.scale : 0.0f;
                s[j][3] = drop_keep(drop, row_idx + 8ull * S_max + k0 + 1) ? s[j][3] * drop.scale : 0.0f;
            }
        }
        // ---- O += P V
        const uint32_t vt = v_s + buf * KVBYTES;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            if (kk * 16 >= nvalid) break;
            uint32_t a[4];
            a[0] = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
            a[1] = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
            a[2] = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
            a[3] = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
            for (int dp = 0; dp < 4; ++dp) {
                uint32_t b0, b1, b2, b3;
                ldmatrix_x4_trans(vt + kk * 2048 + v_row + v_col[dp], b0, b1, b2, b3);
                mma_bf16(o[dp * 2], a, b0, b1);
                mma_bf16(o[dp * 2 + 1], a, b2, b3);
            }
        }

        if (ki == nkb - 1) {
            // ---- head finished: normalise, stage through this warp's own rows of the head's Q
            // buffer (already consumed into registers), 16-byte coalesced stores
            float t0 = l0, t1 = l1;
            t0 += __shfl_xor_sync(0xffffffffu, t0, 1);
            t0 += __shfl_xor_sync(0xffffffffu, t0, 2);
            t1 += __shfl_xor_sync(0xffffffffu, t1, 1);
            t1 += __shfl_xor_sync(0xffffffffu, t1, 2);
            const float inv0 = t0 > 0.0f ? 1.0f / t0 : 0.0f;
            const float inv1 = t1 > 0.0f ? 1.0f / t1 : 0.0f;
            uint8_t* q_gen = smem + (hh & 1) * QBYTES;
            const int r0 = warp * 16 + g, r1 = r0 + 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                *reinterpret_cast<uint32_t*>(q_gen + r0 * 128 + ((j ^ (r0 & 7)) << 4) + tq * 4) =
                    pack_bf16(o[j][0] * inv0, o[j][1] * inv0);
                *reinterpret_cast<uint32_t*>(q_gen + r1 * 128 + ((j ^ (r1 & 7)) << 4) + tq * 4) =
                    pack_bf16(o[j][2] * inv1, o[j][3] * inv1);
            }
            __syncwarp();
            __nv_bfloat16* o_base = out + off * ldo + (h_begin + hh) * kHeadDim;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int idx = i * 32 + lane;
                const int r = warp * 16 + (idx >> 3), c = idx & 7;
                const int q = q0 + r;
                if (q < S) {
                    const uint4 v = *reinterpret_cast<const uint4*>(q_gen + r * 128 + ((c ^ (r & 7)) << 4));
                    *reinterpret_cast<uint4*>(o_base + q * ldo + c * 8) = v;
                }
            }
        }
        __syncthreads();
    }
}

template <int BLOCK_M, bool DROP>
int launch(const __nv_bfloat16* qkv, const float* mask_bias, const int* seq_off, int B, int S,
           int heads, __nv_bfloat16* out, cudaStream_t stream, DropCfg drop = DropCfg{0ull, 0u, 0u, 1.0f}) {
    constexpr int SMEM = 2 * BLOCK_M * 128 + 4 * kBlockN * 128 + kMaxS * 4 + 64;
    static bool attr_set = false;
    auto kfn = attention_kernel<BLOCK_M, DROP>;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) {
            set_last_error("attention: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
        attr_set = true;
    }
    // heads per CTA: enough CTAs to fill the machine a few times over, as few pipeline ramps as possible
    const long long base = static_cast<long long>((S + BLOCK_M - 1) / BLOCK_M) * B;
    int hpg = heads;
    while (hpg > 1 && base * ((heads + hpg - 1) / hpg) < 148LL * 8) hpg = (hpg + 1) / 2;
    if (hpg > 4) hpg = 4;
    dim3 grid((S + BLOCK_M - 1) / BLOCK_M, (heads + hpg - 1) / hpg, B);
    kfn<<<grid, BLOCK_M * 2, SMEM, stream>>>(qkv, mask_bias, seq_off, S, heads, hpg, out, drop);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("attention_kernel<%d> launch: %s", BLOCK_M, cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

// ====================================================================== tcgen05 path (S <= 128)
// One work item = one (sample, head); all queries and keys of the sample fit one 128x128 tile.
//   control warp (lane 0): TMA loads Q | K | V tiles (128 rows x 64 dims each, 128B-swizzled) straight
//       from the [rows, 3*heads*64] qkv matrix, issues S = Q K^T (tcgen05.mma, N = keys rounded up to 16)
//       into TMEM and later O = P V (V is the MN-major B operand exactly as TMA wrote it);
//   4 softmax warps (thread = query row = TMEM lane): read their score row with tcgen05.ld, apply the
//       key bias / length mask, exponentiate, write the bf16 probabilities as the K-major A operand of
//       the second product over the (already consumed) Q/K tiles, then read O back, scale by 1/sum and
//       store the row.
// A CTA is strictly sequential per item; four CTAs share an SM (48 KB smem, 128 TMEM columns each), so
// one CTA's softmax overlaps the other CTAs' loads and MMAs.
constexpr int kTcThreads = 160;

struct TcParams {
    CUtensorMap qkv_map[4];  // boxes of 32 / 64 / 96 / 128 rows: fetch only the rows the sample has
    const float* bias;     // per row (packed) or [B,S] (dense); may be null
    const int* seq_off;    // packed layout or null
    __nv_bfloat16* out;
    int S_max, heads, items;
    DropCfg drop;          // train mode: dropout on the probabilities (DROP instantiation only)
};

// DROP: the probabilities that feed P V are dropped / rescaled (attention_probs_dropout_prob in train
// mode, HF:models/bert/modeling_bert.py:168-207); the softmax normaliser stays the undropped sum.
template <bool DROP>
__global__ void __launch_bounds__(kTcThreads, 4)
attention_tc_kernel(const __grid_constant__ TcParams p) {
    extern __shared__ uint8_t raw[];
    const uint32_t base = (smem_u32(raw) + 1023u) & ~1023u;
    uint8_t* gen = raw + (base - smem_u32(raw));
    const uint32_t q_s = base, k_s = base + 16384, v_s = base + 32768;  // P overlays Q and K
    float* bias_s = reinterpret_cast<float*>(gen + 49152);
    const uint32_t bars = base + 49152 + 512;
    const uint32_t full_bar = bars, s_bar = bars + 8, p_bar = bars + 16, o_bar = bars + 24, t_bar = bars + 32;
    volatile uint32_t* tslot = reinterpret_cast<volatile uint32_t*>(gen + 49152 + 512 + 64);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // rows a short sample does not fetch keep whatever the previous item left there (finite values
    // that are masked or multiplied by zero); make the very first contents finite as well
    for (int i = tid; i < 49152 / 16; i += kTcThreads) reinterpret_cast<uint4*>(gen)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.qkv_map[i]);
        mbar_init(full_bar, 1);
        mbar_init(s_bar, 1);
        mbar_init(p_bar, 128);
        mbar_init(o_bar, 1);
        mbar_init(t_bar, 128);
        fence_mbar_init();
    }
    if (warp == 4) tmem_alloc<128>(bars + 64);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = *tslot;
    const long long ldo = static_cast<long long>(p.heads) * kHeadDim;

    uint32_t phase = 0;
    for (int item = blockIdx.x; item < p.items; item += gridDim.x, phase ^= 1u) {
        const int b = item / p.heads, h = item - b * p.heads;
        int off, len;
        if (p.seq_off) {
            off = __ldg(p.seq_off + b);
            len = __ldg(p.seq_off + b + 1) - off;
        } else {
            off = b * p.S_max;
            len = p.S_max;
        }
        len = len > 128 ? 128 : len;
        const int n16 = len > 0 ? (len + 15) & ~15 : 16;  // keys rounded up to the MMA granule

        if (warp == 4) {
            // ------------------------------------------------ control: TMA + MMA issue
            if (lane == 0) {
                if (item != static_cast<int>(blockIdx.x)) mbar_wait(o_bar, phase ^ 1u);  // smem of the previous item consumed
                const int bi = (len - 1) >> 5;  // box of 32 * (bi + 1) rows
                const CUtensorMap* map = &p.qkv_map[bi];
                mbar_expect_tx(full_bar, 3u * 4096u * static_cast<uint32_t>(bi + 1));
                tma_load_3d(map, full_bar, q_s, 0, off, h);
                tma_load_3d(map, full_bar, k_s, 0, off, p.heads + h);
                tma_load_3d(map, full_bar, v_s, 0, off, 2 * p.heads + h);
                mbar_wait(full_bar, phase);
                if (item != static_cast<int>(blockIdx.x)) mbar_wait(t_bar, phase ^ 1u);  // O of the previous item read out
                tc_fence_after();
                {   // S[128 x n16] = Q K^T
                    const uint32_t idesc = make_idesc_bf16(128, n16, 0, 0);
                    const uint64_t adesc = make_smem_desc(q_s, 0, 1024, 2);
                    const uint64_t bdesc = make_smem_desc(k_s, 0, 1024, 2);
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_bf16(tm, adesc + 2 * k, bdesc + 2 * k, idesc, k != 0);
                    umma_commit(s_bar);
                }
                mbar_wait(p_bar, phase);
                tc_fence_after();
                {   // O[128 x 64] = P[128 x n16] V[n16 x 64]; V rows are keys: MN-major B, 2 KB per 16 keys
                    const uint32_t idesc = make_idesc_bf16(128, 64, 0, 1);
                    for (int k = 0; k < n16 / 16; ++k) {
                        const uint64_t adesc = make_smem_desc(q_s + (k >> 2) * 16384 + (k & 3) * 32, 0, 1024, 2);
                        const uint64_t bdesc = make_smem_desc(v_s + k * 2048, 0, 1024, 2);
                        umma_bf16(tm, adesc, bdesc, idesc, k != 0);
                    }
                    umma_commit(o_bar);
                }
            }
            __syncwarp();
        } else {
            // ------------------------------------------------ softmax warps: thread = query row
            const int row = tid;  // 0..127 == TMEM lane
            const float my_bias = row < len ? (p.bias ? __ldg(p.bias + off + row) : 0.0f) : -INFINITY;
            bias_s[row] = my_bias;
            // token-packed batches carry no key bias at all except on a masked [CLS] row: when every key of the
            // item is plain (bias 0) the inner loops skip the per-key bias (one shared-memory load, one add and one
            // select per score) and only bound the columns by the length
            const bool biased = named_bar_or(1, 128, row < len && my_bias != 0.0f);
            const uint32_t t_row = tm + (static_cast<uint32_t>(warp * 32) << 16);
            mbar_wait(s_bar, phase);
            tc_fence_after();
            // pass 1: row maximum over the attended keys
            float mx = -INFINITY;
            for (int c0 = 0; c0 < n16; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(t_row + c0, v);
                tmem_ld_wait();
                if (!biased && c0 + 32 <= len) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]) + bias_s[c0 + j]);
                }
            }
            const float ms = (mx == -INFINITY ? 0.0f : mx) * kLog2e;
            // pass 2: probabilities -> bf16 A operand (K-major, two 64-key swizzle atoms over Q|K)
            float sum = 0.0f;
            for (int c0 = 0; c0 < n16; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(t_row + c0, v);
                tmem_ld_wait();
                float e[32];
                if (!biased && c0 + 32 <= len) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        e[j] = fast_exp2(fmaf(__uint_as_float(v[j]), kLog2e, -ms));
                        sum += e[j];
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        e[j] = fast_exp2(fmaf(__uint_as_float(v[j]) + bias_s[c0 + j], kLog2e, -ms));
                        sum += e[j];
                    }
                }
                if (DROP) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const unsigned long long idx =
                            (static_cast<unsigned long long>(item) * p.S_max + row) * p.S_max + (c0 + j);
                        e[j] = drop_keep(p.drop, idx) ? e[j] * p.drop.scale : 0.0f;
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (c0 + q * 8 >= n16) break;
                    uint4 o;
                    o.x = pack_bf16(e[q * 8 + 0], e[q * 8 + 1]);
                    o.y = pack_bf16(e[q * 8 + 2], e[q * 8 + 3]);
                    o.z = pack_bf16(e[q * 8 + 4], e[q * 8 + 5]);
                    o.w = pack_bf16(e[q * 8 + 6], e[q * 8 + 7]);
                    const int c8 = (c0 >> 3) + q;  // 8-key chunk index 0..15
                    *reinterpret_cast<uint4*>(gen + (c8 >> 3) * 16384 + row * 128 + (((c8 & 7) ^ (row & 7)) << 4)) = o;
                }
            }
            fence_proxy_async_smem();
            tc_fence_before();
            mbar_arrive(p_bar);
            // O row back from TMEM, normalise, store
            mbar_wait(o_bar, phase);
            tc_fence_after();
            uint32_t o0[32], o1[32];
            tmem_ld32(t_row, o0);
            tmem_ld32(t_row + 32, o1);
            tmem_ld_wait();
            tc_fence_before();
            mbar_arrive(t_bar);
            if (row < len) {
                const float inv = sum > 0.0f ? 1.0f / sum : 0.0f;
                uint4* dst = reinterpret_cast<uint4*>(p.out + (static_cast<long long>(off) + row) * ldo + h * kHeadDim);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    uint4 w;
                    w.x = pack_bf16(__uint_as_float(o0[q * 8 + 0]) * inv, __uint_as_float(o0[q * 8 + 1]) * inv);
                    w.y = pack_bf16(__uint_as_float(o0[q * 8 + 2]) * inv, __uint_as_float(o0[q * 8 + 3]) * inv);
                    w.z = pack_bf16(__uint_as_float(o0[q * 8 + 4]) * inv, __uint_as_float(o0[q * 8 + 5]) * inv);
                    w.w = pack_bf16(__uint_as_float(o0[q * 8 + 6]) * inv, __uint_as_float(o0[q * 8 + 7]) * inv);
                    dst[q] = w;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    uint4 w;
                    w.x = pack_bf16(__uint_as_float(o1[q * 8 + 0]) * inv, __uint_as_float(o1[q * 8 + 1]) * inv);
                    w.y = pack_bf16(__uint_as_float(o1[q * 8 + 2]) * inv, __uint_as_float(o1[q * 8 + 3]) * inv);
                    w.z = pack_bf16(__uint_as_float(o1[q * 8 + 4]) * inv, __uint_as_float(o1[q * 8 + 5]) * inv);
                    w.w = pack_bf16(__uint_as_float(o1[q * 8 + 6]) * inv, __uint_as_float(o1[q * 8 + 7]) * inv);
                    dst[4 + q] = w;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<128>(tm);
    }
}

// ====================================================================== tcgen05 path (128 < S <= 512)
// One work item = one (sample, head, block of 128 queries).  The keys are walked in blocks of 128; per block
//   control warp (lane 0): S_j = Q K_j^T into TMEM; K_{j+1} | V_{j+1} (also across items) are already on their
//       way into the other shared-memory buffer, and the next item's Q is fetched as soon as the last S of this
//       item has been consumed, so no TMA latency sits on the per-block chain;
//   softmax warps (thread = query row = TMEM lane): block maximum, running maximum m, P_j = exp(S_j - m) as the
//       bf16 K-major A operand over the consumed K_j tile (+16 KB), running sum l;
//   control warp: O_j = P_j V_j into the TMEM columns S_j occupied;
//   softmax warps: acc = acc * exp(m_old - m) + O_j with the 64 accumulators of the row in REGISTERS (the flash
//       recurrence; HF:integrations/sdpa_attention.py:92 computes the same softmax(QK^T + mask) V in one piece),
// and the row is normalised by 1/l and stored after the last block.  Nothing but Q, K, V is read and nothing but
// the output written: scores and probabilities never leave the SM.  Every barrier completes one phase per key
// block (counted in `it` by every role alike); two CTAs share an SM (99 KB smem, 128 TMEM columns each) so one
// CTA's softmax overlaps the other's MMAs.
struct TcLongParams {
    CUtensorMap qkv_map[4];  // boxes of 32 / 64 / 96 / 128 rows
    const float* bias;       // per row (packed) or [B,S] (dense); may be null
    const int* seq_off;      // packed layout or null
    __nv_bfloat16* out;
    int S_max, heads, qblocks, items;
    DropCfg drop;
};

constexpr int kTcLongData = 6 * 16384;   // Q | K0 | V0 | K1 | V1 | second P atom
constexpr int kTcLongSmem = kTcLongData + 2048 + 256 + 1024;

struct TcLongBlock {   // one (item, key block) of a CTA's work list
    int item, j, nkv, off, len, q0, qlen, h, bh;
    bool valid;
};

__device__ __forceinline__ bool tc_long_item(const TcLongParams& p, int item, TcLongBlock* o) {
    o->item = item;
    o->bh = item / p.qblocks;
    const int qb = item - o->bh * p.qblocks;
    const int b = o->bh / p.heads;
    o->h = o->bh - b * p.heads;
    int off, len;
    if (p.seq_off) {
        off = __ldg(p.seq_off + b);
        len = __ldg(p.seq_off + b + 1) - off;
    } else {
        off = b * p.S_max;
        len = p.S_max;
    }
    len = len > kMaxS ? kMaxS : len;
    o->off = off;
    o->len = len;
    o->q0 = qb * 128;
    o->j = 0;
    if (o->q0 >= len) return false;   // query block beyond the sequence: nothing to do
    o->qlen = len - o->q0 < 128 ? len - o->q0 : 128;
    o->nkv = (len + 127) >> 7;
    return true;
}
// first block of the first non-empty item at or after `item` (items are strided by the grid size)
__device__ __forceinline__ TcLongBlock tc_long_first(const TcLongParams& p, int item, int stride) {
    TcLongBlock b;
    b.valid = false;
    for (; item < p.items; item += stride)
        if (tc_long_item(p, item, &b)) {
            b.valid = true;
            return b;
        }
    return b;
}
__device__ __forceinline__ TcLongBlock tc_long_next(const TcLongParams& p, const TcLongBlock& c, int stride) {
    if (c.j + 1 < c.nkv) {
        TcLongBlock n = c;
        ++n.j;
        return n;
    }
    return tc_long_first(p, c.item + stride, stride);
}

template <bool DROP>
__global__ void __launch_bounds__(kTcThreads, 2)
attention_tc_long_kernel(const __grid_constant__ TcLongParams p) {
    extern __shared__ uint8_t raw[];
    const uint32_t base = (smem_u32(raw) + 1023u) & ~1023u;
    uint8_t* gen = raw + (base - smem_u32(raw));
    const uint32_t q_s = base;
    const uint32_t x_s = base + 5 * 16384;                 // second 64-key atom of P
    auto k_smem = [&](int buf) { return base + 16384u + static_cast<uint32_t>(buf) * 32768u; };
    auto v_smem = [&](int buf) { return base + 32768u + static_cast<uint32_t>(buf) * 32768u; };
    float* bias_s = reinterpret_cast<float*>(gen + kTcLongData);          // [512]
    const uint32_t bars = base + kTcLongData + 2048;
    const uint32_t s_bar = bars + 16, p_bar = bars + 24, o_bar = bars + 32, t_bar = bars + 40, q_bar = bars + 48;
    auto full_bar = [&](int buf) { return bars + 8u * buf; };
    volatile uint32_t* tslot = reinterpret_cast<volatile uint32_t*>(gen + kTcLongData + 2048 + 64);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // rows a short block does not fetch keep the previous contents (finite, masked or multiplied by zero)
    for (int i = tid; i < kTcLongData / 16; i += kTcThreads) reinterpret_cast<uint4*>(gen)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.qkv_map[i]);
        mbar_init(full_bar(0), 1);
        mbar_init(full_bar(1), 1);
        mbar_init(s_bar, 1);
        mbar_init(p_bar, 128);
        mbar_init(o_bar, 1);
        mbar_init(t_bar, 128);
        mbar_init(q_bar, 1);
        fence_mbar_init();
    }
    if (warp == 4) tmem_alloc<128>(bars + 64);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = *tslot;
    const long long ldo = static_cast<long long>(p.heads) * kHeadDim;
    const int stride = static_cast<int>(gridDim.x);

    if (warp == 4) {
        // ------------------------------------------------ control: TMA + MMA issue (one thread)
        if (lane == 0) {
            auto load_kv = [&](const TcLongBlock& blk, int buf) {
                const int klen = blk.len - blk.j * 128 < 128 ? blk.len - blk.j * 128 : 128;
                const int bk = (klen - 1) >> 5;
                mbar_expect_tx(full_bar(buf), 2u * 4096u * static_cast<uint32_t>(bk + 1));
                tma_load_3d(&p.qkv_map[bk], full_bar(buf), k_smem(buf), 0, blk.off + blk.j * 128, p.heads + blk.h);
                tma_load_3d(&p.qkv_map[bk], full_bar(buf), v_smem(buf), 0, blk.off + blk.j * 128, 2 * p.heads + blk.h);
            };
            auto load_q = [&](const TcLongBlock& blk) {
                const int bq = (blk.qlen - 1) >> 5;
                mbar_expect_tx(q_bar, 4096u * static_cast<uint32_t>(bq + 1));
                tma_load_3d(&p.qkv_map[bq], q_bar, q_s, 0, blk.off + blk.q0, blk.h);
            };
            TcLongBlock cur = tc_long_first(p, static_cast<int>(blockIdx.x), stride);
            uint32_t q_phase = 0;
            if (cur.valid) {
                load_q(cur);
                load_kv(cur, 0);
            }
            for (int it = 0; cur.valid; ++it) {
                const int buf = it & 1;
                const uint32_t ph = it & 1u, prev = ph ^ 1u;
                const TcLongBlock nxt = tc_long_next(p, cur, stride);
                const int klen = cur.len - cur.j * 128 < 128 ? cur.len - cur.j * 128 : 128;
                const int n16 = (klen + 15) & ~15;
                // the other buffer (K, V and the P atom over K) was last read by the P V product of block it-1
                if (it > 0) mbar_wait(o_bar, prev);
                if (nxt.valid) load_kv(nxt, buf ^ 1);
                mbar_wait(full_bar(buf), static_cast<uint32_t>(it >> 1) & 1u);
                if (cur.j == 0) {
                    mbar_wait(q_bar, q_phase);
                    q_phase ^= 1u;
                }
                if (it > 0) mbar_wait(t_bar, prev);   // O of the previous block read out of TMEM
                tc_fence_after();
                {   // S[128 x n16] = Q K_j^T
                    const uint32_t idesc = make_idesc_bf16(128, n16, 0, 0);
                    const uint64_t adesc = make_smem_desc(q_s, 0, 1024, 2);
                    const uint64_t bdesc = make_smem_desc(k_smem(buf), 0, 1024, 2);
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_bf16(tm, adesc + 2 * k, bdesc + 2 * k, idesc, k != 0);
                    umma_commit(s_bar);
                }
                mbar_wait(p_bar, ph);   // every softmax thread has read S and written P: S (and Q, if last) is consumed
                tc_fence_after();
                if (nxt.valid && nxt.j == 0) load_q(nxt);   // Q of the next item streams in under P V and the O read-out
                {   // O_j[128 x 64] = P_j[128 x n16] V_j[n16 x 64]; V rows are keys: MN-major B
                    const uint32_t idesc = make_idesc_bf16(128, 64, 0, 1);
                    for (int k = 0; k < n16 / 16; ++k) {
                        const uint32_t pa = (k < 4 ? k_smem(buf) : x_s) + (k & 3) * 32;
                        const uint64_t adesc = make_smem_desc(pa, 0, 1024, 2);
                        const uint64_t bdesc = make_smem_desc(v_smem(buf) + k * 2048, 0, 1024, 2);
                        umma_bf16(tm, adesc, bdesc, idesc, k != 0);
                    }
                    umma_commit(o_bar);
                }
                cur = nxt;
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------ softmax warps: thread = query row
        const int row = tid;  // 0..127 == TMEM lane
        const uint32_t t_row = tm + (static_cast<uint32_t>(warp * 32) << 16);
        int it = 0;
        for (TcLongBlock cur = tc_long_first(p, static_cast<int>(blockIdx.x), stride); cur.valid;
             cur = tc_long_first(p, cur.item + stride, stride)) {
            // all 128 threads are past the previous item's last P write (its o_bar needed every p_bar arrival)
#pragma unroll
            for (int i = 0; i < kMaxS / 128; ++i) {
                const int key = i * 128 + row;
                bias_s[key] = key < cur.len ? (p.bias ? __ldg(p.bias + cur.off + key) : 0.0f) : -INFINITY;
            }
            bool nz = false;
#pragma unroll
            for (int i = 0; i < kMaxS / 128; ++i) nz |= (i * 128 + row < cur.len) && bias_s[i * 128 + row] != 0.0f;
            // no key of the item carries a bias (the normal case of a token-packed batch): the inner loops then
            // skip the per-key bias and only bound the columns by the block's key count
            const bool biased = named_bar_or(1, 128, nz);
            float acc[64];
#pragma unroll
            for (int i = 0; i < 64; ++i) acc[i] = 0.0f;
            float m_run = -INFINITY, l_run = 0.0f;
            for (int j = 0; j < cur.nkv; ++j, ++it) {
                const uint32_t ph = it & 1u;
                uint8_t* p0 = gen + 16384 + (it & 1) * 32768;   // first P atom: over K_j
                uint8_t* p1 = gen + 5 * 16384;                  // second P atom
                const int klen = cur.len - j * 128 < 128 ? cur.len - j * 128 : 128;
                const int n16 = (klen + 15) & ~15;
                const float* bj = bias_s + j * 128;
                mbar_wait(s_bar, ph);
                tc_fence_after();
                // pass 1: block maximum over the attended keys
                float mx = -INFINITY;
                for (int c0 = 0; c0 < n16; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(t_row + c0, v);
                    tmem_ld_wait();
                    if (!biased && c0 + 32 <= klen) {
#pragma unroll
                        for (int jj = 0; jj < 32; ++jj) mx = fmaxf(mx, __uint_as_float(v[jj]));
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 32; ++jj) {
                            const float bb = bj[c0 + jj];
                            mx = fmaxf(mx, bb == -INFINITY ? -INFINITY : __uint_as_float(v[jj]) + bb);
                        }
                    }
                }
                const float m_new = fmaxf(m_run, mx);
                const float ms = (m_new == -INFINITY ? 0.0f : m_new) * kLog2e;
                const float corr = m_run == -INFINITY ? 0.0f : fast_exp2(fmaf(m_run, kLog2e, -ms));
                // pass 2: probabilities relative to the running maximum -> bf16 A operand (two 64-key atoms)
                float sum = 0.0f;
                for (int c0 = 0; c0 < n16; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(t_row + c0, v);
                    tmem_ld_wait();
                    float e[32];
                    if (!biased && c0 + 32 <= klen) {
#pragma unroll
                        for (int jj = 0; jj < 32; ++jj) {
                            e[jj] = fast_exp2(fmaf(__uint_as_float(v[jj]), kLog2e, -ms));
                            sum += e[jj];
                        }
                    } else {
#pragma unroll
                        for (int jj = 0; jj < 32; ++jj) {
                            const float bb = bj[c0 + jj];
                            e[jj] = bb == -INFINITY ? 0.0f : fast_exp2(fmaf(__uint_as_float(v[jj]) + bb, kLog2e, -ms));
                            sum += e[jj];
                        }
                    }
                    if (DROP) {
#pragma unroll
                        for (int jj = 0; jj < 32; ++jj) {
                            const unsigned long long idx =
                                (static_cast<unsigned long long>(cur.bh) * p.S_max + (cur.q0 + row)) * p.S_max +
                                (j * 128 + c0 + jj);
                            e[jj] = drop_keep(p.drop, idx) ? e[jj] * p.drop.scale : 0.0f;
                        }
                    }
                    uint8_t* pa = c0 < 64 ? p0 : p1;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (c0 + q * 8 >= n16) break;
                        uint4 o;
                        o.x = pack_bf16(e[q * 8 + 0], e[q * 8 + 1]);
                        o.y = pack_bf16(e[q * 8 + 2], e[q * 8 + 3]);
                        o.z = pack_bf16(e[q * 8 + 4], e[q * 8 + 5]);
                        o.w = pack_bf16(e[q * 8 + 6], e[q * 8 + 7]);
                        const int c8 = ((c0 & 63) >> 3) + q;  // 8-key chunk inside the 64-key atom
                        *reinterpret_cast<uint4*>(pa + row * 128 + ((c8 ^ (row & 7)) << 4)) = o;
                    }
                }
                l_run = fmaf(l_run, corr, sum);
                m_run = m_new;
                fence_proxy_async_smem();
                tc_fence_before();
                mbar_arrive(p_bar);
                // O_j back from TMEM into the row's running accumulators
                mbar_wait(o_bar, ph);
                tc_fence_after();
                {
                    uint32_t o0[32];
                    tmem_ld32(t_row, o0);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) acc[i] = fmaf(acc[i], corr, __uint_as_float(o0[i]));
                    tmem_ld32(t_row + 32, o0);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) acc[32 + i] = fmaf(acc[32 + i], corr, __uint_as_float(o0[i]));
                }
                tc_fence_before();
                mbar_arrive(t_bar);
            }
            if (row < cur.qlen) {
                const float inv = l_run > 0.0f ? 1.0f / l_run : 0.0f;
                uint4* dst = reinterpret_cast<uint4*>(p.out + (static_cast<long long>(cur.off) + cur.q0 + row) * ldo +
                                                      cur.h * kHeadDim);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    uint4 w;
                    w.x = pack_bf16(acc[q * 8 + 0] * inv, acc[q * 8 + 1] * inv);
                    w.y = pack_bf16(acc[q * 8 + 2] * inv, acc[q * 8 + 3] * inv);
                    w.z = pack_bf16(acc[q * 8 + 4] * inv, acc[q * 8 + 5] * inv);
                    w.w = pack_bf16(acc[q * 8 + 6] * inv, acc[q * 8 + 7] * inv);
                    dst[q] = w;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<128>(tm);
    }
}

}  // namespace

int encode_qkv_maps(CUtensorMap* maps, const __nv_bfloat16* qkv, int heads, long long rows_alloc, int blocked) {
    // 3-D view {64 dims, rows, 3*heads column blocks}: token-major rows are 3*heads*64 elements apart
    // with the blocks side by side; in the blocked layout every block is a contiguous [rows,64] matrix
    const uint64_t nblk = static_cast<uint64_t>(3) * heads;
    uint64_t dims[3] = {64, static_cast<uint64_t>(rows_alloc), nblk};
    uint64_t str_tok[2] = {nblk * 128, 128};
    uint64_t str_blk[2] = {128, static_cast<uint64_t>(rows_alloc) * 128};
    for (int i = 0; i < 4; ++i) {
        uint32_t box[3] = {64, static_cast<uint32_t>(32 * (i + 1)), 1};
        int rc = encode_tensor_map(&maps[i], qkv, 2, 3, dims, blocked ? str_blk : str_tok, box, 128);
        if (rc) return rc;
    }
    return 0;
}

namespace {

int launch_tc_long(const __nv_bfloat16* qkv, const float* mask_bias, const int* seq_off, int B, int S,
                   int heads, long long rows_alloc, int blocked, __nv_bfloat16* out, cudaStream_t stream,
                   const DropCfg* drop) {
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(attention_tc_long_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             kTcLongSmem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(attention_tc_long_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     kTcLongSmem);
        if (e != cudaSuccess) {
            set_last_error("attention_tc_long: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
        attr_set = true;
    }
    TcLongParams p;
    const bool dropping = drop != nullptr && drop->thresh != 0u;
    p.drop = dropping ? *drop : DropCfg{0ull, 0u, 0u, 1.0f};
    int rc = encode_qkv_maps(p.qkv_map, qkv, heads, rows_alloc, blocked);
    if (rc) return rc;
    p.bias = mask_bias;
    p.seq_off = seq_off;
    p.out = out;
    p.S_max = S;
    p.heads = heads;
    p.qblocks = (S + 127) / 128;
    const long long items = static_cast<long long>(B) * heads * p.qblocks;
    p.items = static_cast<int>(items);
    const int grid = p.items < 148 * 2 ? p.items : 148 * 2;
    if (dropping)
        attention_tc_long_kernel<true><<<grid, kTcThreads, kTcLongSmem, stream>>>(p);
    else
        attention_tc_long_kernel<false><<<grid, kTcThreads, kTcLongSmem, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("attention_tc_long_kernel launch: %s", cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

int launch_tc(const __nv_bfloat16* qkv, const float* mask_bias, const int* seq_off, int B, int S,
              int heads, long long rows_alloc, int blocked, __nv_bfloat16* out, cudaStream_t stream,
              const DropCfg* drop) {
    constexpr int SMEM = 49152 + 1024 + 1024;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(attention_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(attention_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) {
            set_last_error("attention_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
        attr_set = true;
    }
    TcParams p;
    const bool dropping = drop != nullptr && drop->thresh != 0u;
    p.drop = dropping ? *drop : DropCfg{0ull, 0u, 0u, 1.0f};
    // 3-D view {64 dims, rows, 3*heads column blocks}: token-major rows are 3*heads*64 elements apart
    // with the blocks side by side; in the blocked layout every block is a contiguous [rows,64] matrix
    const uint64_t nblk = static_cast<uint64_t>(3) * heads;
    uint64_t dims[3] = {64, static_cast<uint64_t>(rows_alloc), nblk};
    uint64_t str_tok[2] = {nblk * 128, 128};
    uint64_t str_blk[2] = {128, static_cast<uint64_t>(rows_alloc) * 128};
    for (int i = 0; i < 4; ++i) {
        uint32_t box[3] = {64, static_cast<uint32_t>(32 * (i + 1)), 1};
        int rc = encode_tensor_map(&p.qkv_map[i], qkv, 2, 3, dims, blocked ? str_blk : str_tok, box, 128);
        if (rc) return rc;
    }
    p.bias = mask_bias;
    p.seq_off = seq_off;
    p.out = out;
    p.S_max = S;
    p.heads = heads;
    p.items = B * heads;
    const int grid = p.items < 148 * 4 ? p.items : 148 * 4;
    if (dropping)
        attention_tc_kernel<true><<<grid, kTcThreads, SMEM, stream>>>(p);
    else
        attention_tc_kernel<false><<<grid, kTcThreads, SMEM, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("attention_tc_kernel launch: %s", cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

}  // namespace

void attention_set_tc(bool on) { g_attention_tc = on; }

bool attention_prefers_blocked_qkv(int S) { return S <= kMaxS && g_attention_tc; }

int attention_forward(const __nv_bfloat16* qkv, const float* mask_bias, const int* seq_off, int B,
                      int S, int heads, __nv_bfloat16* out, cudaStream_t stream, long long rows_alloc,
                      int blocked, const DropCfg* drop) {
    if (B <= 0 || S <= 0) return 0;
    const bool dropping = drop && drop->thresh != 0u;
    if (blocked && !g_attention_tc) {
        set_last_error("attention_forward: the blocked qkv layout is only read by the tcgen05 kernels");
        return -1;
    }
    if (S > kMaxS || heads <= 0 || heads > 65535 || B > 65535) {
        set_last_error("attention_forward: unsupported B=%d S=%d heads=%d (S <= %d)", B, S, heads,
                       kMaxS);
        return -1;
    }
    // 64-row query blocks when sequences are short (or packed to short lengths): a block whose rows
    // all lie beyond the sequence exits immediately; 128-row blocks halve the K/V re-reads otherwise
    // whole sequences fit one 128x128 tile: tcgen05 path (rows_alloc bounds the TMA view of qkv)
    if (S <= 128 && g_attention_tc && static_cast<long long>(B) * heads < 0x7fffffffLL)
        return launch_tc(qkv, mask_bias, seq_off, B, S, heads,
                         rows_alloc > 0 ? rows_alloc : static_cast<long long>(B) * S, blocked, out, stream, drop);
    // longer sequences: 128-query blocks against key blocks of 128, running softmax, O accumulated in registers
    if (g_attention_tc && static_cast<long long>(B) * heads * ((S + 127) / 128) < 0x7fffffffLL)
        return launch_tc_long(qkv, mask_bias, seq_off, B, S, heads,
                              rows_alloc > 0 ? rows_alloc : static_cast<long long>(B) * S, blocked, out, stream, drop);
    if (dropping) {
        if (S > 64) return launch<128, true>(qkv, mask_bias, seq_off, B, S, heads, out, stream, *drop);
        return launch<64, true>(qkv, mask_bias, seq_off, B, S, heads, out, stream, *drop);
    }
    if (S > 64)
        return launch<128, false>(qkv, mask_bias, seq_off, B, S, heads, out, stream);
    return launch<64, false>(qkv, mask_bias, seq_off, B, S, heads, out, stream);
}

}  // namespace mrd
