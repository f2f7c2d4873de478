// K3 companion: the attention probabilities of BERT self-attention as an output (TextEncoder.get_attention_weights
// with HF's eager attention, HF:models/bert/modeling_bert.py:115-140).  A kernel of its own rather than an epilogue
// branch of attention_tc_kernel / attention_tc_long_kernel (extra branches cost those, DESIGN.md section 10): it
// recomputes Q K^T, which is cheap next to writing B*heads*S*S floats.
//
// One work item = one (sample, head, block of 128 queries); a CTA walks items grid-strided.
//   control warp (lane 0): TMA loads the Q block and ALL of the sample's keys (<= 512 rows, 64 KB, the 3-D views of
//       encode_qkv_maps, so both qkv layouts of the engine are read), issues S = Q K^T (tcgen05.mma kind::f16, N <= 256
//       per instruction) into TMEM, and prefetches the next item's Q / K as soon as the product has read them;
//   4 softmax warps (thread = query row = TMEM lane): row maximum with the key bias, exp(s - m) written back into
//       TMEM with the row sum, then exp / sum in fp32 staged per warp as 32 x 32 tiles in shared memory and written
//       with TMA stores (S % 4 == 0: the row stride is a multiple of 16 bytes) or with row-coalesced plain stores.
// TMEM: the smallest power of two >= the keys rounded to 32 (the product covers the last TMA box), so short sequences keep several CTAs
// per SM; S = 512 takes all 512 columns of an SM.

#include "attention.h"

#include <math.h>
#include <stdint.h>

#include "ptx.cuh"
#include "tma_host.h"

namespace mrd {

namespace {

constexpr int kPrThreads = 160;                       // 4 softmax warps + 1 control warp
constexpr int kPrMaxS = 512;
constexpr int kPrStageBufs = 2;                       // 4 KB staging tiles per softmax warp
constexpr int kPrStageBytes = 4 * kPrStageBufs * 4096;
constexpr float kPrLog2e = 1.4426950408889634f;

struct ProbsParams {
    CUtensorMap qkv_map[4];   // boxes of 32 / 64 / 96 / 128 rows
    CUtensorMap out_map;      // {S keys, S queries, B*heads} fp32, box {32, 32, 1}, 128B swizzle (tma_out only)
    const float* bias;        // [B,S] or null
    float* out;               // [B,heads,S,S]
    int S, heads, qblocks, items, tmem_cols, tma_out;
};

__host__ __device__ constexpr int probs_smem_bytes(int S) {
    return 1024 + 16384 + ((S + 127) / 128) * 16384 + kPrStageBytes + 2 * kPrMaxS * 4 + 64;
}

__device__ __forceinline__ void tmem_alloc_cols(uint32_t smem_result_addr, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cols(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ float probs_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__global__ void __launch_bounds__(kPrThreads, 1)
attention_probs_kernel(const __grid_constant__ ProbsParams p) {
    extern __shared__ uint8_t raw[];
    const uint32_t base = (smem_u32(raw) + 1023u) & ~1023u;
    uint8_t* gen = raw + (base - smem_u32(raw));
    const int S = p.S;
    const int nkc = (S + 127) >> 7;                    // 128-key chunks of K, back to back: key r at k_s + r * 128
    const uint32_t q_s = base, k_s = base + 16384u;
    const uint32_t st_off = 16384u + static_cast<uint32_t>(nkc) * 16384u;
    float* bias_s = reinterpret_cast<float*>(gen + st_off + kPrStageBytes);   // 2 x 512, alternating per item
    const uint32_t bars = base + st_off + kPrStageBytes + 2 * kPrMaxS * 4;
    const uint32_t full_bar = bars, s_bar = bars + 8, t_bar = bars + 16;
    volatile uint32_t* tslot = reinterpret_cast<volatile uint32_t*>(gen + st_off + kPrStageBytes + 2 * kPrMaxS * 4 + 32);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.qkv_map[i]);
        if (p.tma_out) tma_prefetch_desc(&p.out_map);
        mbar_init(full_bar, 1);
        mbar_init(s_bar, 1);
        mbar_init(t_bar, 128);
        fence_mbar_init();
    }
    if (warp == 4) tmem_alloc_cols(bars + 32, static_cast<uint32_t>(p.tmem_cols));
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = *tslot;
    const int stride = static_cast<int>(gridDim.x);

    if (warp == 4) {
        // ------------------------------------------------ control: TMA + MMA issue (one thread)
        if (lane == 0) {
            const int n32 = (S + 31) & ~31;   // the K rows the TMA boxes fetch: every column read below is written
            int it = 0;
            for (int item = blockIdx.x; item < p.items; item += stride, ++it) {
                const int bh = item / p.qblocks, q0 = (item - bh * p.qblocks) * 128;
                const int b = bh / p.heads, h = bh - b * p.heads;
                const int qlen = S - q0 < 128 ? S - q0 : 128;
                const uint32_t ph = static_cast<uint32_t>(it) & 1u;
                if (it > 0) mbar_wait(s_bar, ph ^ 1u);   // the previous product has read Q and K
                const int bq = (qlen - 1) >> 5;
                uint32_t bytes = 4096u * static_cast<uint32_t>(bq + 1);
                for (int j = 0; j < nkc; ++j) {
                    const int klen = S - j * 128 < 128 ? S - j * 128 : 128;
                    bytes += 4096u * static_cast<uint32_t>(((klen - 1) >> 5) + 1);
                }
                mbar_expect_tx(full_bar, bytes);
                tma_load_3d(&p.qkv_map[bq], full_bar, q_s, 0, b * S + q0, h);
                for (int j = 0; j < nkc; ++j) {
                    const int klen = S - j * 128 < 128 ? S - j * 128 : 128;
                    tma_load_3d(&p.qkv_map[(klen - 1) >> 5], full_bar, k_s + j * 16384u, 0, b * S + j * 128,
                                p.heads + h);
                }
                mbar_wait(full_bar, ph);
                if (it > 0) mbar_wait(t_bar, ph ^ 1u);   // the previous item's scores are read out of TMEM
                tc_fence_after();
                // S[128 x n32] = Q K^T, at most 256 columns per instruction
                const uint64_t adesc = make_smem_desc(q_s, 0, 1024, 2);
                for (int n0 = 0; n0 < n32; n0 += 256) {
                    const int n = n32 - n0 < 256 ? n32 - n0 : 256;
                    const uint32_t idesc = make_idesc_bf16(128, n, 0, 0);
                    const uint64_t bdesc = make_smem_desc(k_s + static_cast<uint32_t>(n0) * 128u, 0, 1024, 2);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_bf16(tm + static_cast<uint32_t>(n0), adesc + 2 * k, bdesc + 2 * k, idesc, k != 0);
                }
                umma_commit(s_bar);
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------ softmax warps: thread = query row = TMEM lane
        const uint32_t t_row = tm + (static_cast<uint32_t>(warp * 32) << 16);
        uint8_t* stage = gen + st_off + static_cast<uint32_t>(warp) * (kPrStageBufs * 4096);
        const uint32_t stage_s = base + st_off + static_cast<uint32_t>(warp) * (kPrStageBufs * 4096);
        const int n32 = (S + 31) & ~31;
        int tile = 0;   // staging tiles this warp has used (ring position)
        int it = 0;
        for (int item = blockIdx.x; item < p.items; item += stride, ++it) {
            const int bh = item / p.qblocks, q0 = (item - bh * p.qblocks) * 128;
            const int b = bh / p.heads;
            const uint32_t ph = static_cast<uint32_t>(it) & 1u;
            // the bias buffer of this parity was last read by item it-2, which every softmax thread finished
            // before the barrier of item it-1
            // keys S..n32-1 exist only as padding of the last TMA box: -inf makes them exactly 0
            float* bs = bias_s + (it & 1) * kPrMaxS;
            for (int k = tid; k < n32; k += 128)
                bs[k] = k >= S ? -INFINITY : p.bias ? __ldg(p.bias + static_cast<long long>(b) * S + k) : 0.0f;
            named_bar_sync(1, 128);
            const int r0 = q0 + warp * 32;   // first query row of this warp
            mbar_wait(s_bar, ph);
            tc_fence_after();
            if (r0 < S) {
                // pass 1: row maximum over the attended keys (scores are finite: s + (-inf) = -inf)
                float mx = -INFINITY;
                {
                    uint32_t nx[32];
                    tmem_ld32(t_row, nx);
                    for (int c0 = 0; c0 < n32; c0 += 32) {
                        tmem_ld_wait();
                        uint32_t v[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = nx[j];
                        if (c0 + 32 < n32) tmem_ld32(t_row + c0 + 32, nx);
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 bb = *reinterpret_cast<const float4*>(bs + c0 + j);
                            mx = fmaxf(mx, fmaxf(fmaxf(__uint_as_float(v[j]) + bb.x, __uint_as_float(v[j + 1]) + bb.y),
                                                 fmaxf(__uint_as_float(v[j + 2]) + bb.z, __uint_as_float(v[j + 3]) + bb.w)));
                        }
                    }
                }
                const float ms = (mx == -INFINITY ? 0.0f : mx) * kPrLog2e;
                // pass 2: exp(s - m) back into TMEM (exactly 0 for a masked key), row sum
                float sum = 0.0f;
                for (int c0 = 0; c0 < n32; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(t_row + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 bb = *reinterpret_cast<const float4*>(bs + c0 + j);
                        const float b4[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float e = probs_exp2(fmaf(__uint_as_float(v[j + u]) + b4[u], kPrLog2e, -ms));
                            sum += e;
                            v[j + u] = __float_as_uint(e);
                        }
                    }
                    tmem_st32(t_row + c0, v);
                }
                tmem_st_wait();
                const float inv = sum > 0.0f ? 1.0f / sum : 0.0f;   // no attended key: zero rows
                // pass 3: normalise, stage 32 rows x 32 keys per tile (128B-swizzled rows), store
                float* out = p.out + static_cast<long long>(bh) * S * S;
                uint32_t nx[32];
                tmem_ld32(t_row, nx);
                for (int c0 = 0; c0 < n32; c0 += 32, ++tile) {
                    tmem_ld_wait();
                    uint32_t v[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = nx[j];
                    if (c0 + 32 < n32) tmem_ld32(t_row + c0 + 32, nx);
                    const int buf = tile % kPrStageBufs;
                    uint8_t* sb = stage + buf * 4096;
                    if (p.tma_out) {
                        if (lane == 0) tma_store_wait_read<kPrStageBufs - 1>();   // this buffer's last store has read it
                    }
                    __syncwarp();
#pragma unroll
                    for (int ch = 0; ch < 8; ++ch) {
                        float4 w;
                        w.x = __uint_as_float(v[ch * 4 + 0]) * inv;
                        w.y = __uint_as_float(v[ch * 4 + 1]) * inv;
                        w.z = __uint_as_float(v[ch * 4 + 2]) * inv;
                        w.w = __uint_as_float(v[ch * 4 + 3]) * inv;
                        *reinterpret_cast<float4*>(sb + lane * 128 + ((ch ^ (lane & 7)) << 4)) = w;
                    }
                    if (p.tma_out) {
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_3d(&p.out_map, stage_s + buf * 4096u, c0, r0, bh);
                            tma_store_commit();
                        }
                    } else {
                        __syncwarp();
                        // lane = key: every store instruction writes 32 consecutive floats of one row
                        const int c = c0 + lane;
#pragma unroll 4
                        for (int r = 0; r < 32; ++r) {
                            if (r0 + r < S && c < S)
                                out[static_cast<long long>(r0 + r) * S + c] = *reinterpret_cast<const float*>(
                                    sb + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + (lane & 3) * 4);
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(t_bar);
        }
        if (p.tma_out && lane == 0) tma_store_wait_all<0>();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc_cols(tm, static_cast<uint32_t>(p.tmem_cols));
    }
}

}  // namespace

int attention_probs(const __nv_bfloat16* qkv, const float* mask_bias, int B, int S, int heads, float* probs,
                    cudaStream_t stream, long long rows_alloc, int blocked) {
    if (B <= 0 || S <= 0) return 0;
    if (S > kPrMaxS || heads <= 0) {
        set_last_error("attention_probs: unsupported B=%d S=%d heads=%d (S <= %d)", B, S, heads, kPrMaxS);
        return -1;
    }
    const long long qblocks = (S + 127) / 128;
    const long long items = static_cast<long long>(B) * heads * qblocks;
    if (items >= 0x7fffffffLL || static_cast<long long>(B) * S >= 0x7fffffffLL) {
        set_last_error("attention_probs: B=%d heads=%d S=%d exceeds the 32-bit item / row index", B, heads, S);
        return -1;
    }
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(attention_probs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             probs_smem_bytes(kPrMaxS));
        if (e != cudaSuccess) {
            set_last_error("attention_probs: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
        attr_set = true;
    }
    ProbsParams p;
    int rc = encode_qkv_maps(p.qkv_map, qkv, heads, rows_alloc > 0 ? rows_alloc : static_cast<long long>(B) * S,
                             blocked);
    if (rc) return rc;
    // TMA stores need 16-byte row and plane strides and a 16-byte aligned base
    p.tma_out = S % 4 == 0 && (reinterpret_cast<uintptr_t>(probs) & 15u) == 0;
    if (p.tma_out) {
        uint64_t dims[3] = {static_cast<uint64_t>(S), static_cast<uint64_t>(S), static_cast<uint64_t>(B) * heads};
        uint64_t strides[2] = {static_cast<uint64_t>(S) * 4, static_cast<uint64_t>(S) * S * 4};
        uint32_t box[3] = {32, 32, 1};
        rc = encode_tensor_map(&p.out_map, probs, 4, 3, dims, strides, box, 128);
        if (rc) return rc;
    }
    p.bias = mask_bias;
    p.out = probs;
    p.S = S;
    p.heads = heads;
    p.qblocks = static_cast<int>(qblocks);
    p.items = static_cast<int>(items);
    int cols = 32;
    while (cols < S) cols *= 2;
    p.tmem_cols = cols;
    const int smem = probs_smem_bytes(S);
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, attention_probs_kernel, kPrThreads, smem);
    if (e != cudaSuccess) {
        set_last_error("attention_probs: occupancy query: %s", cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    if (per_sm > 512 / cols) per_sm = 512 / cols;   // co-resident CTAs must fit the SM's TMEM together
    if (per_sm < 1) per_sm = 1;
    const int grid = p.items < 148 * per_sm ? p.items : 148 * per_sm;
    attention_probs_kernel<<<grid, kPrThreads, smem, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("attention_probs_kernel launch: %s", cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

}  // namespace mrd
