// conv_chain_kernel: conv3 (+downsample) + identity + ReLU of bottleneck i and conv1 + ReLU of bottleneck i+1 for
// the same 128-pixel tiles inside one persistent CTA (see conv_chain.h), with the y tile handed from the first
// product to the second ON CHIP:
//
//   warp 0        TMA producer          once: the whole W1 and W2 into shared memory (resident for the CTA's life);
//                                       then per tile the conv2-output rows (and the block input when the downsample
//                                       branch is fused): one stage = the tile's whole K
//   warp 1        product-1 MMA issuer  per tile and 128-column half: 128 x 128 x 16 tcgen05.mma into TMEM columns
//                                       [0, 256) (two accumulators); owns the TMEM allocation (512 columns)
//   warps 2..9    epilogue of BOTH products (TMEM lane quarter = warp % 4, two warps per quarter split 64 columns):
//                                       +bias (+identity) -> ReLU -> bf16 -> 128B-swizzled staging -> TMA store
//   warp 10       identity loader       TMA ring ahead of the product-1 epilogue
//   warp 11       product-2 MMA issuer  every staged 64-column sub-tile of y IS a K-major A operand chunk: as soon as
//                                       the epilogue has written it, 128 x BN2 x 16 MMAs against the matching W2
//                                       chunk accumulate z into TMEM columns [256, 256 + 2*BN2)
//
// y is written to memory once (the next block needs it as its identity) and never read back: neither DRAM nor the
// SM<->L2 fabric sees the second product's operand.  (Measured first, r02: reading y back through L2 - a hit, DRAM
// traffic 2.0 instead of 2.8 GB per launch - was no faster than two launches; ncu showed all of these layers moving
// ~7.2 TB/s between the SMs and L2, weights re-fetched per tile included.  Hence resident weights and the on-chip
// hand-off.)
// Staging ring protocol (kStg slots, every sub-tile of either product takes the next slot): the epilogue may
// overwrite a slot when the TMA store that read it has drained (bulk-group wait) AND product 2 is done with it
// (s_done); it arrives on s_full after writing; the product-2 issuer walks the same slot sequence, issuing MMAs for
// y sub-tiles and passing z sub-tiles through.
// Reference ops replaced: TV:models/resnet.py:143-163 (Bottleneck.forward) across two consecutive blocks.

#include "conv_chain.h"

#include <stdio.h>
#include <string.h>

#include "gemm_conv.h"
#include "ptx.cuh"
#include "tma_host.h"

namespace mrd {

namespace {

constexpr int kBN1 = 128;
constexpr int kThreads = 12 * 32;
constexpr int kEpi = 256;
constexpr int kSub = 128 * 128;      // one 128-row x 64-column bf16 sub-tile
constexpr int kSmemMax = 232448;
constexpr int kBars = 1024;
constexpr int kAcc2Col = 256;        // first TMEM column of the product-2 accumulators
constexpr int kStg = 4;              // staging slots: the product-2 MMAs add latency before a slot can be reused

struct Tile {
    int w0, h0, n0;
};
__device__ __forceinline__ Tile decode(const ChainParams& p, int m) {
    Tile t;
    const int tw_i = m % p.tiles_w;
    const int r = m / p.tiles_w;
    t.w0 = tw_i * p.tw;
    t.h0 = (r % p.tiles_h) * p.th;
    t.n0 = (r / p.tiles_h) * p.nb;
    return t;
}

template <int BN2>
__global__ void __launch_bounds__(kThreads, 1) conv_chain_kernel(const __grid_constant__ ChainParams p) {
    constexpr int kW2Chunk = BN2 * 128;              // W2 rows x 64 K
    constexpr int NSUB1 = kBN1 / 64, NSUB2 = BN2 / 64;
    const ChainPhase& P1 = p.ph[0];
    const ChainPhase& P2 = p.ph[1];
    const int SA = p.stages1, RING = p.ring;
    const int K1c = P1.num_k;                        // K chunks of product 1 (whole K per A stage)
    const int n1 = P1.n_tiles;                       // 128-column halves of y
    const int K2c = P2.num_k;                        // = y sub-tiles per tile = n1 * NSUB1
    const int a_stage = K1c * kSub;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t w1_s = base;                                    // [n1][K1c] blocks of 128 x 64
    const uint32_t w2_s = w1_s + n1 * K1c * kSub;                  // [K2c] blocks of BN2 x 64
    const uint32_t a_s = w2_s + K2c * kW2Chunk;                    // [SA] stages of K1c x (128 x 64)
    const uint32_t st_s = a_s + SA * a_stage;                      // [kStg] staging slots
    const uint32_t ring_s = st_s + kStg * kSub;
    const uint32_t bar = ring_s + RING * kSub;
    uint8_t* st_gen = gen + (st_s - base);
    uint8_t* ring_gen = gen + (ring_s - base);
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen + (bar - base) + 480);

    auto fullA = [&](int s) { return bar + 8u * s; };
    auto emptyA = [&](int s) { return bar + 64u + 8u * s; };
    auto sfull = [&](int s) { return bar + 128u + 8u * s; };
    auto sdone = [&](int s) { return bar + 192u + 8u * s; };
    auto rfull = [&](int s) { return bar + 256u + 8u * s; };
    auto rempty = [&](int s) { return bar + 320u + 8u * s; };
    auto tfull1 = [&](int a) { return bar + 384u + 8u * a; };
    auto tempty1 = [&](int a) { return bar + 400u + 8u * a; };
    auto tfull2 = [&](int a) { return bar + 416u + 8u * a; };
    auto tempty2 = [&](int a) { return bar + 432u + 8u * a; };
    const uint32_t wres = bar + 448u;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&P1.a_map[0]);
        tma_prefetch_desc(&P1.a_map[1]);
        tma_prefetch_desc(&P1.b_map);
        tma_prefetch_desc(&P1.c_map);
        tma_prefetch_desc(&P1.r_map);
        tma_prefetch_desc(&P2.b_map);
        tma_prefetch_desc(&P2.c_map);
        for (int s = 0; s < 8; ++s) {
            mbar_init(fullA(s), 1);
            mbar_init(emptyA(s), 1);
            mbar_init(sfull(s), 1);
            mbar_init(sdone(s), 1);
            mbar_init(rfull(s), 1);
            mbar_init(rempty(s), 1);   // one arrival per consumed sub-tile, by the group's leader (see sub_tile)
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull1(a), 1);
            mbar_init(tempty1(a), 4 * (kBN1 / 64));   // 4 warps per 64-column sub-tile
            mbar_init(tfull2(a), 1);
            mbar_init(tempty2(a), 4 * (BN2 / 64));
        }
        mbar_init(wres, 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<512>(bar + 480);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const int bid = static_cast<int>(blockIdx.x), nblk = static_cast<int>(gridDim.x);
    const int n_my = p.m_tiles > bid ? (p.m_tiles - bid + nblk - 1) / nblk : 0;
    const int box_rows = p.tw * p.th * p.nb;
    const uint32_t a_bytes = static_cast<uint32_t>(box_rows) * 128u;

    if (warp == 0) {
        // ------------------------------------------------------------ producer: resident weights, then A tiles
        if (lane == 0) {
            mbar_expect_tx(wres, static_cast<uint32_t>(n1 * K1c * kSub + K2c * kW2Chunk));
            for (int n = 0; n < n1; ++n)
                for (int kc = 0; kc < K1c; ++kc)
                    tma_load_2d(&P1.b_map, wres, w1_s + (n * K1c + kc) * kSub, kc * 64, n * kBN1);
            for (int kc = 0; kc < K2c; ++kc) tma_load_2d(&P2.b_map, wres, w2_s + kc * kW2Chunk, kc * 64, 0);
        }
        __syncwarp();
        int stage = 0;
        uint32_t phase = 0;
        for (int j = 0; j < n_my; ++j) {
            const Tile t = decode(p, bid + j * nblk);
            mbar_wait(emptyA(stage), phase ^ 1u);
            if (lane == 0) {
                mbar_expect_tx(fullA(stage), a_bytes * static_cast<uint32_t>(K1c));
                for (int kc = 0; kc < K1c; ++kc) {
                    const int second = (P1.kc_split && kc >= P1.kc_split) ? 1 : 0;
                    const int c = kc - (second ? P1.kc_split : 0);
                    tma_load_4d(&P1.a_map[second], fullA(stage), a_s + stage * a_stage + kc * kSub, c * 64, t.w0, t.h0,
                                t.n0);
                }
            }
            __syncwarp();
            if (++stage == SA) { stage = 0; phase ^= 1u; }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ product-1 MMA issuer
        constexpr uint32_t idesc = make_idesc_bf16(128, kBN1, 0, 0);
        int stage = 0, it = 0;
        uint32_t phase = 0;
        mbar_wait(wres, 0);
        for (int j = 0; j < n_my; ++j) {
            mbar_wait(fullA(stage), phase);
            for (int n = 0; n < n1; ++n, ++it) {
                const int acc = it & 1;
                mbar_wait(tempty1(acc), ((it >> 1) & 1) ^ 1u);
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t d = tmem + acc * kBN1;
                    for (int kc = 0; kc < K1c; ++kc) {
                        const uint64_t ad = make_smem_desc(a_s + stage * a_stage + kc * kSub, 0, 1024, 2);
                        const uint64_t bd = make_smem_desc(w1_s + (n * K1c + kc) * kSub, 0, 1024, 2);
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_bf16(d, ad + 2 * k, bd + 2 * k, idesc, (kc | k) != 0 ? 1u : 0u);
                    }
                    umma_commit(tfull1(acc));
                    if (n == n1 - 1) umma_commit(emptyA(stage));   // the tile's A rows are free once these MMAs are done
                }
                __syncwarp();
            }
            if (++stage == SA) { stage = 0; phase ^= 1u; }
        }
    } else if (warp == 10) {
        // ------------------------------------------------------------ identity loader (product 1)
        if (P1.has_res) {
            int slot = 0;
            uint32_t phase = 0;
            for (int j = 0; j < n_my; ++j) {
                const Tile t = decode(p, bid + j * nblk);
                for (int n = 0; n < n1; ++n)
                    for (int sub = 0; sub < NSUB1; ++sub) {
                        mbar_wait(rempty(slot), phase ^ 1u);
                        if (lane == 0) {
                            mbar_expect_tx(rfull(slot), a_bytes);
                            tma_load_4d(&P1.r_map, rfull(slot), ring_s + slot * kSub, n * kBN1 + sub * 64, t.w0, t.h0,
                                        t.n0);
                        }
                        __syncwarp();
                        if (++slot == RING) { slot = 0; phase ^= 1u; }
                    }
            }
        }
    } else if (warp == 11) {
        // ------------------------------------------------------------ product-2 MMA issuer
        // walks the staging slots in the order the epilogue fills them: K2c y sub-tiles of tile j (each one a K chunk
        // of z = relu(y W2^T + b2)), then - from the second tile on - the NSUB2 z sub-tiles of tile j-1, which only
        // pass through
        constexpr uint32_t idesc = make_idesc_bf16(128, BN2, 0, 0);
        mbar_wait(wres, 0);
        if (lane == 0) {
            int q = 0;
            auto pass_through = [&](int count) {
                for (int i = 0; i < count; ++i, ++q) {
                    const int slot = q % kStg;
                    mbar_wait(sfull(slot), static_cast<uint32_t>(q / kStg) & 1u);
                    mbar_arrive(sdone(slot));
                }
            };
            for (int j = 0; j < n_my; ++j) {
                const int acc = j & 1;
                mbar_wait(tempty2(acc), ((j >> 1) & 1) ^ 1u);
                tc_fence_after();
                const uint32_t d = tmem + kAcc2Col + acc * BN2;
                for (int kc = 0; kc < K2c; ++kc, ++q) {
                    const int slot = q % kStg;
                    mbar_wait(sfull(slot), static_cast<uint32_t>(q / kStg) & 1u);
                    tc_fence_after();
                    const uint64_t ad = make_smem_desc(st_s + slot * kSub, 0, 1024, 2);
                    const uint64_t bd = make_smem_desc(w2_s + kc * kW2Chunk, 0, 1024, 2);
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_bf16(d, ad + 2 * k, bd + 2 * k, idesc, (kc | k) != 0 ? 1u : 0u);
                    umma_commit(sdone(slot));
                    if (kc == K2c - 1) umma_commit(tfull2(acc));
                }
                if (j >= 1) pass_through(NSUB2);
            }
            if (n_my > 0) pass_through(NSUB2);
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------ epilogue of both products (warps 2..9)
        // Two independent groups of four warps (one warp per TMEM lane quarter each): group g takes the sub-tiles
        // with q % 2 == g of the common sequence, a thread owns one row and all 64 columns of its sub-tile.  A
        // sub-tile is a latency chain (TMEM load -> identity -> pack -> fence -> barrier -> TMA store); two of
        // them in flight per SM hide it.
        const int grp = (warp - 2) >> 2;
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        const bool leader = (warp - 2) % 4 == 0 && lane == 0;   // issues this group's TMA stores
        const int bar_a = 1 + 2 * grp, bar_b = 2 + 2 * grp;     // this group's named barriers (128 threads)
        int q = 0;                       // position in the common sub-tile sequence (staging slot = q % kStg)

        // one 64-column sub-tile: TMEM columns [acc_col, acc_col + 64) -> global columns [col0, col0 + 64)
        auto sub_tile = [&](const ChainPhase& P, const Tile& t, int col0, uint32_t acc_col, uint32_t tfull,
                            uint32_t tphase, uint32_t tempty, int yq) {
            const int slot = q % kStg;
            mbar_wait(tfull, tphase);
            tc_fence_after();
            uint32_t v0[32], v1[32];
            tmem_ld32(tmem + (static_cast<uint32_t>(quarter * 32) << 16) + acc_col, v0);
            tmem_ld32(tmem + (static_cast<uint32_t>(quarter * 32) << 16) + acc_col + 32, v1);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);   // 4 warps x sub-tiles of the accumulator = its arrival count
            float f[64];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                const float4 b0 = __ldg(reinterpret_cast<const float4*>(P.bias + col0 + j));
                const float4 b1 = __ldg(reinterpret_cast<const float4*>(P.bias + col0 + 32 + j));
                f[j + 0] = __uint_as_float(v0[j + 0]) + b0.x;
                f[j + 1] = __uint_as_float(v0[j + 1]) + b0.y;
                f[j + 2] = __uint_as_float(v0[j + 2]) + b0.z;
                f[j + 3] = __uint_as_float(v0[j + 3]) + b0.w;
                f[32 + j + 0] = __uint_as_float(v1[j + 0]) + b1.x;
                f[32 + j + 1] = __uint_as_float(v1[j + 1]) + b1.y;
                f[32 + j + 2] = __uint_as_float(v1[j + 2]) + b1.z;
                f[32 + j + 3] = __uint_as_float(v1[j + 3]) + b1.w;
            }
            if (yq >= 0) {   // identity of a y sub-tile: ring slot in the order the loader fetched them
                const int rslot = yq % RING;
                mbar_wait(rfull(rslot), static_cast<uint32_t>(yq / RING) & 1u);
                const uint8_t* r_row = ring_gen + rslot * kSub + row * 128;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const uint4 r4 = *reinterpret_cast<const uint4*>(r_row + ((c ^ (row & 7)) << 4));
                    const float2 r0 = unpack_bf16(r4.x), r1 = unpack_bf16(r4.y), r2 = unpack_bf16(r4.z),
                                 r3 = unpack_bf16(r4.w);
                    f[c * 8 + 0] += r0.x; f[c * 8 + 1] += r0.y;
                    f[c * 8 + 2] += r1.x; f[c * 8 + 3] += r1.y;
                    f[c * 8 + 4] += r2.x; f[c * 8 + 5] += r2.y;
                    f[c * 8 + 6] += r3.x; f[c * 8 + 7] += r3.y;
                }
            }
            if (P.act == ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 64; ++j) f[j] = fmaxf(f[j], 0.0f);
            }
            // the slot was last used kStg sub-tiles ago (by this same group: kStg is even): its TMA store must
            // have read it and product 2 must be done with it
            if (leader) {
                tma_store_wait_read<kStg / 2 - 1>();
                if (q >= kStg) mbar_wait(sdone(slot), static_cast<uint32_t>(q / kStg - 1) & 1u);
            }
            named_bar_sync(bar_b, 128);
            uint8_t* st_row = st_gen + slot * kSub + row * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint4 o;
                o.x = pack_bf16(f[c * 8 + 0], f[c * 8 + 1]);
                o.y = pack_bf16(f[c * 8 + 2], f[c * 8 + 3]);
                o.z = pack_bf16(f[c * 8 + 4], f[c * 8 + 5]);
                o.w = pack_bf16(f[c * 8 + 6], f[c * 8 + 7]);
                *reinterpret_cast<uint4*>(st_row + ((c ^ (row & 7)) << 4)) = o;
            }
            fence_proxy_async_smem();
            named_bar_sync(bar_a, 128);
            if (leader) {
                // The identity slot is released only here, after every thread of the group has stored values that
                // depend on its ld.shared of the slot: an arrive right after the loads does not wait for them, and
                // the loader's next TMA write overtook loads still in flight (tools/stress_patterns.py, r02).
                if (yq >= 0) mbar_arrive(rempty(yq % RING));
                tma_store_4d(&P.c_map, st_s + slot * kSub, col0, t.w0, t.h0, t.n0);
                tma_store_commit();
                mbar_arrive(sfull(slot));
            }
        };
        auto product2_tile = [&](int j) {
            const Tile t = decode(p, bid + j * nblk);
            const int acc = j & 1;
            for (int sub = 0; sub < NSUB2; ++sub, ++q)
                if ((q & 1) == grp)
                    sub_tile(P2, t, sub * 64, kAcc2Col + acc * BN2 + sub * 64, tfull2(acc), (j >> 1) & 1u, tempty2(acc),
                             -1);
        };
        for (int j = 0; j < n_my; ++j) {
            const Tile t = decode(p, bid + j * nblk);
            for (int n = 0; n < n1; ++n) {
                const int it1 = j * n1 + n, acc = it1 & 1;
                for (int sub = 0; sub < NSUB1; ++sub, ++q)
                    if ((q & 1) == grp)
                        sub_tile(P1, t, n * kBN1 + sub * 64, acc * kBN1 + sub * 64, tfull1(acc), (it1 >> 1) & 1u,
                                 tempty1(acc), P1.has_res ? j * K2c + n * NSUB1 + sub : -1);
            }
            if (j >= 1) product2_tile(j - 1);   // its MMAs finished while this tile's y was being produced
        }
        if (n_my > 0) product2_tile(n_my - 1);
        if (leader) tma_store_wait_all<0>();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem);
    }
}

template <int BN2>
int launch_bn2(const ChainLaunch* g, cudaStream_t stream) {
    static bool attr_set = false;
    auto kfn = conv_chain_kernel<BN2>;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
        if (e != cudaSuccess) {
            set_last_error("conv_chain: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
        attr_set = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g->grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = g->smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kfn, g->p);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("conv_chain_kernel<%d> launch: %s", BN2, cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

// 4-D view of an NHWC activation seen through (stride s) sampling, boxes of tw x th x nb output pixels
int map_nhwc(CUtensorMap* m, const __nv_bfloat16* x, int C, int N, int Ho, int Wo, int s, int pad, int tw, int th,
             int nb) {
    const int W = Wo * s + 2 * pad, H = Ho * s + 2 * pad;
    const __nv_bfloat16* x0 = x + (static_cast<long long>(pad) * W + pad) * C;
    uint64_t dims[4] = {(uint64_t)C, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
    uint64_t str[3] = {(uint64_t)s * C * 2, (uint64_t)s * W * C * 2, (uint64_t)H * W * C * 2};
    uint32_t box[4] = {64, (uint32_t)tw, (uint32_t)th, (uint32_t)nb};
    return encode_tensor_map(m, x0, 2, 4, dims, str, box, 128);
}
// the same tensor as a flat [M, C] matrix, boxes of 128 rows
int map_flat(CUtensorMap* m, const __nv_bfloat16* x, int C, long long M) {
    uint64_t dims[4] = {(uint64_t)C, (uint64_t)M, 1, 1};
    uint64_t str[3] = {(uint64_t)C * 2, (uint64_t)C * 2 * M, (uint64_t)C * 2 * M};
    uint32_t box[4] = {64, 128, 1, 1};
    return encode_tensor_map(m, x, 2, 4, dims, str, box, 128);
}
int map_weights(CUtensorMap* m, const __nv_bfloat16* w, int N, int K, int bn) {
    uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
    uint64_t str[1] = {(uint64_t)K * 2};
    uint32_t box[2] = {64, (uint32_t)bn};
    return encode_tensor_map(m, w, 2, 2, dims, str, box, 128);
}

// shared memory of one launch: resident W1 + W2, A stages (whole K each), staging slots, identity ring, barriers
int chain_smem(int C0, int C1, int Cout, int C2, bool identity, int* stages, int* ring) {
    const int K1c = (C0 + C1) / 64;
    const int w_bytes = Cout * (C0 + C1) * 2 + C2 * Cout * 2;
    const int a_stage = K1c * kSub;
    const int avail = kSmemMax - 1024 - kBars - kStg * kSub - w_bytes;
    int sa = 2, r = identity ? 2 : 0;
    int left = avail - sa * a_stage - r * kSub;
    if (left < 0) {   // a single A stage still works (the tile's loads then wait for the previous tile's MMAs)
        sa = 1;
        left = avail - sa * a_stage - r * kSub;
        if (left < 0 && identity) { r = 1; left = avail - sa * a_stage - r * kSub; }
    }
    if (left < 0) return -1;
    while (identity && left >= kSub && r < 6) { ++r; left -= kSub; }
    while (left >= a_stage && sa < 4) { ++sa; left -= a_stage; }
    *stages = sa;
    *ring = r;
    return 1024 + w_bytes + sa * a_stage + kStg * kSub + r * kSub + kBars;
}

}  // namespace

bool conv_chain_supported(int C0, int C1, int Cout, int C2) {
    if (!(C0 > 0 && C0 % 64 == 0 && C1 >= 0 && C1 % 64 == 0 && Cout % 128 == 0 && (C2 == 64 || C2 == 128))) return false;
    int sa, r;
    return chain_smem(C0, C1, Cout, C2, C1 == 0, &sa, &r) > 0;
}

int plan_conv_chain(ChainLaunch* g, const __nv_bfloat16* X0, int C0, const __nv_bfloat16* X1, int C1, int s1,
                    const __nv_bfloat16* identity, int N, int Ho, int Wo, const __nv_bfloat16* W1, int Cout,
                    const float* bias1, __nv_bfloat16* Y, const __nv_bfloat16* W2, int C2, const float* bias2,
                    __nv_bfloat16* Z, int out_pad) {
    memset(g, 0, sizeof(*g));
    if (!X1) C1 = 0;
    if (!conv_chain_supported(C0, C1, Cout, C2) || (X1 && s1 != 1 && s1 != 2) || (X1 && identity) || N <= 0 ||
        Ho <= 0 || Wo <= 0) {
        set_last_error("plan_conv_chain: unsupported shape C0=%d C1=%d Cout=%d C2=%d stride=%d (both weight matrices "
                       "must fit in shared memory next to the pipeline)", C0, C1, Cout, C2, s1);
        return -1;
    }
    ChainParams& p = g->p;
    const long long M = static_cast<long long>(N) * Ho * Wo;
    if (M > 0x7fffffffLL) {
        set_last_error("plan_conv_chain: M too large");
        return -1;
    }
    const int bn2 = C2;
    g->block_n2 = bn2;
    const bool boxes = out_pad != 0 || (X1 && s1 == 2);   // tiles must be pixel boxes; otherwise flat 128-row tiles
    if (boxes) {
        p.tw = Wo < 128 ? Wo : 128;
        p.th = 128 / p.tw;
        if (p.th > Ho) p.th = Ho;
        if (p.th < 1) p.th = 1;
        p.nb = 1;
        if (p.th == Ho && p.tw == Wo) {
            p.nb = 128 / (p.tw * p.th);
            if (p.nb < 1) p.nb = 1;
            if (p.nb > N) p.nb = N;
        }
        p.tiles_w = (Wo + p.tw - 1) / p.tw;
        p.tiles_h = (Ho + p.th - 1) / p.th;
        p.tiles_img = (N + p.nb - 1) / p.nb;
    } else {
        p.tw = 128; p.th = 1; p.nb = 1;
        p.tiles_w = static_cast<int>((M + 127) / 128); p.tiles_h = 1; p.tiles_img = 1;
    }
    const long long mt = static_cast<long long>(p.tiles_w) * p.tiles_h * p.tiles_img;
    p.m_tiles = static_cast<int>(mt);
    auto act_map = [&](CUtensorMap* m, const __nv_bfloat16* x, int C, int s, int pad) -> int {
        if (boxes) return map_nhwc(m, x, C, N, Ho, Wo, s, pad, p.tw, p.th, p.nb);
        return map_flat(m, x, C, M);
    };
    ChainPhase& a = p.ph[0];
    ChainPhase& b = p.ph[1];
    int rc = act_map(&a.a_map[0], X0, C0, 1, 0);
    if (rc) return rc;
    a.a_map[1] = a.a_map[0];
    if (X1) {
        rc = act_map(&a.a_map[1], X1, C1, s1, 0);
        if (rc) return rc;
    }
    rc = map_weights(&a.b_map, W1, Cout, C0 + C1, kBN1);
    if (rc) return rc;
    rc = act_map(&a.c_map, Y, Cout, 1, 0);
    if (rc) return rc;
    a.r_map = a.c_map;
    if (identity) {
        rc = act_map(&a.r_map, identity, Cout, 1, 0);
        if (rc) return rc;
    }
    a.bias = bias1;
    a.num_k = (C0 + C1) / 64;
    a.kc_split = X1 ? C0 / 64 : 0;
    a.n_tiles = Cout / kBN1;
    a.act = ACT_RELU;
    a.has_res = identity ? 1 : 0;

    b.a_map[0] = b.a_map[1] = a.c_map;   // unused: product 2 reads y from the staging slots
    rc = map_weights(&b.b_map, W2, C2, Cout, bn2);
    if (rc) return rc;
    rc = act_map(&b.c_map, Z, C2, 1, out_pad);
    if (rc) return rc;
    b.r_map = b.c_map;
    b.bias = bias2;
    b.num_k = Cout / 64;
    b.kc_split = 0;
    b.n_tiles = 1;
    b.act = ACT_RELU;
    b.has_res = 0;

    g->smem = chain_smem(C0, C1, Cout, C2, identity != nullptr, &p.stages1, &p.ring);
    p.stages2 = 0;
    const int sms = gemm_num_sms();
    g->grid = p.m_tiles < sms ? p.m_tiles : sms;
    g->flops = 2.0 * M * (static_cast<double>(Cout) * (C0 + C1) + static_cast<double>(C2) * Cout);
    g->bytes = 2.0 * (1.0 * M * C0 + (X1 ? 1.0 * M * C1 : 0.0) + (identity ? 1.0 * M * Cout : 0.0) + 1.0 * M * Cout +
                      1.0 * M * C2 + 1.0 * Cout * (C0 + C1) + 1.0 * C2 * Cout);
    return 0;
}

int launch_conv_chain(const ChainLaunch* g, cudaStream_t stream) {
    if (g->block_n2 == 64) return launch_bn2<64>(g, stream);
    return launch_bn2<128>(g, stream);
}

}  // namespace mrd
