// K1/K2: persistent, warp-specialised tcgen05 implicit-GEMM kernel for sm_100a.
//
//   warp 0      TMA producer  : A boxes from a 4-D/5-D view of the NHWC activation (one box per
//                               (tap, 64-channel chunk)), B boxes from the [Cout][K] weight matrix
//   warp 1      MMA issuer    : tcgen05.mma (128 x BLOCK_N x 16, bf16 -> fp32) into a double-buffered
//                               TMEM accumulator; also owns the TMEM allocation
//   warps 2..9  epilogue      : per 64-column sub-tile: residual sub-tile prefetched by TMA into the
//                               (swizzled) store staging buffer; tcgen05.ld -> +bias (+residual, in
//                               place) -> ReLU/GELU -> bf16 -> staging -> TMA store (clipped by the
//                               tensor map); optional fp32 side output.  8 warps: TMEM lane quarter =
//                               warp % 4, two warps per quarter split the 64 columns.
//
// The epilogue of tile i overlaps the main loop of tile i+1 (two accumulator stages in TMEM).
// Reference ops replaced: torchvision Bottleneck conv+bn+relu(+add) (TV:models/resnet.py:143-163),
// ResNet stem (TV:models/resnet.py:268-270), nn.Linear in BertSelfAttention/BertSelfOutput/
// BertIntermediate/BertOutput (HF:models/bert/modeling_bert.py:177-179,295,340,353), and the
// Linear layers of src/cnn_encoder.py:46-51, src/fusion_model.py:108-111,212-240,
// src/multimodal_classifier.py:44-58.

#include "gemm_conv.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "ptx.cuh"
#include "tma_host.h"

namespace mrd {

namespace {

bool g_use_pdl = true;

// Debugging overrides (tools/stress_kernels.py): MRD_DEBUG_PDL, MRD_DEBUG_RING, read once.
int g_debug_ring = -1;
void apply_debug_env() {
    static bool done = false;
    if (done) return;
    done = true;
    if (const char* e = getenv("MRD_DEBUG_PDL")) g_use_pdl = atoi(e) != 0;
    if (const char* e = getenv("MRD_DEBUG_RING")) g_debug_ring = atoi(e);
}

constexpr int kBlockM = 128;
constexpr int kNumThreads = 352;  // TMA warp + MMA warp + 8 epilogue warps + residual-loader warp
constexpr int kEpiThreads = 256;
constexpr int kStageBufBytes = 128 * 128;  // one 128-row x 64-column bf16 sub-tile (store / residual)
constexpr int kSmemLimit = 232448;         // 227 KB opt-in limit per CTA
constexpr int kMaxStages = 8;
constexpr int kMaxRing = 8;
constexpr int kBarBytes = 1024;

constexpr int MODE_GENERIC = 0, MODE_STEM = 1, MODE_FLAT3 = 2;

template <int BLOCK_N, int MODE>
struct Cfg {
    static constexpr bool STEM = MODE == MODE_STEM;
    static constexpr int BLOCK_K = STEM ? 32 : 64;
    static constexpr int ROW_BYTES = BLOCK_K * 2;
    static constexpr int A_STAGE = kBlockM * ROW_BYTES;
    static constexpr int B_STAGE = BLOCK_N * ROW_BYTES;
    static constexpr int STAGE = A_STAGE + B_STAGE;
    static constexpr int FIXED = 2 * kStageBufBytes + kBarBytes + 1024;  // staging + barriers + alignment
    static constexpr int TMEM_COLS = 2 * BLOCK_N;  // 128 / 256 / 512: powers of two
    static constexpr uint32_t LAYOUT = STEM ? 4u : 2u;  // SWIZZLE_64B : SWIZZLE_128B
    static constexpr uint32_t SBO = 8 * ROW_BYTES;      // 8-row core-matrix group pitch
};

struct TileCoord {
    int n_idx, w0, h0, n0;
};

__device__ __forceinline__ TileCoord decode_tile(const ConvGemmParams& p, int tile) {
    TileCoord t;
    int m_idx = tile / p.n_tiles_n;
    t.n_idx = tile - m_idx * p.n_tiles_n;
    int tw_i = m_idx % p.tiles_w;
    int r = m_idx / p.tiles_w;
    int th_i = r % p.tiles_h;
    int img_i = r / p.tiles_h;
    t.w0 = tw_i * p.tw + p.w_shift;
    t.h0 = th_i * p.th;
    t.n0 = img_i * p.nb;
    return t;
}

// Shared-memory map (all offsets from a 1024-byte aligned base; stage / ring counts are runtime so
// one binary serves the compute-bound GEMMs (deep operand pipeline, no residual ring) and the
// memory-bound short-K convolutions with residual (shallow operand pipeline, deep residual ring)):
//   [stages x A_STAGE][stages x B_STAGE][2 x 16 KB store staging][ring x 16 KB residual][barriers]
// MASK (generic mode, single-group epilogue; plan_conv_dgrad): the tile fetched through r_map is not added but used as
// a ReLU mask - out = acc * [r > 0] - the backward of a ReLU whose output r was saved by the forward.  Separate
// instantiations for the same reason as SPLITK: a run-time branch in the shared epilogue costs the forward's kernels.
// SPLITK (generic mode only) is a separate instantiation so that the forward's kernels compile exactly as they
// did before split-K existed: measured, the merged version cost the forward 3 % (different epilogue schedule).
// EPI2: the eight epilogue warps work as two independent groups of four (one warp per TMEM lane quarter each); group g
// takes the 64-column sub-tiles with q % 2 == g of the CTA's sub-tile sequence and a thread owns one row and all 64
// columns.  A sub-tile is a latency chain (TMEM load -> residual -> activation -> pack -> proxy fence -> barrier ->
// TMA store, ~1500 cycles measured on the chained bottleneck kernel of conv_chain.cu): with one sub-tile in flight
// per CTA that chain bounds every launch whose main loop is shorter than it.
// Stem patch geometry (MODE_STEM): a tile is 8 output pixels x 16 output rows; its raw input patch is 37 rows x 24
// pixels x 4 channels bf16 of the padded image.
constexpr int kStemRow = 192;    // bytes per patch row (24 pixels x 8 B)
constexpr int kStemRows = 37;

// LNC: LayerNorm over the whole output row in the epilogue.  The n_tiles_n CTAs that hold the column tiles of one
// 128-row stripe are neighbours in the persistent tile order.  Epilogue pass 1: accumulator + bias + residual ->
// per-row partial (mean, M2) of this CTA's columns, the fp32 sums go BACK into TMEM (tcgen05.st); the partials are
// exchanged through L2 (ln_stats) and counted on the stripe's arrival counter.  Pass 2: combine the partials (Chan),
// normalise the TMEM values, store.  HF:models/bert/modeling_bert.py:294-298,352-356.
// One ln_stats record per 128-row stripe = 128 rows x 8 partials x (mean, M2), then the arrival / departure counters.
// The layout does not depend on the row count, so plans of different sizes can share one workspace.
constexpr int kLnStripeBytes = 128 * 8 * 8 + 64;

// PAIR (generic mode, flat GEMMs): tcgen05.mma.cta_group::2.  A cluster of two CTAs takes the 128-row stripes 2j and
// 2j+1 of the SAME column tile as ONE 256 x 256 tile: each CTA's producer loads its own 128 x 64 A block and HALF of
// the 256 x 64 weight block per K step (32 KB instead of 48 KB into each SM: a single-CTA 128 x 256 tile needs
// 94 B/clk of L2 -> SM ingest at full tensor rate, which the SM port does not deliver - the BERT GEMMs sat at ~62 % of
// the tensor rate, r02), the leader CTA's MMA warp issues 256 x 256 x 16 instructions that read both CTAs' shared
// memory and write both CTAs' TMEM, and its tcgen05.commit arrives on the barriers of both CTAs (.multicast::cluster).
// The peer CTA's warp 1 forwards "my stage has landed" to the leader (remote mbarrier arrive); both CTAs' epilogue
// warps hand an accumulator back by arriving on the LEADER's `tempty` barrier.  (Measured first: only multicasting the
// weight tile into both CTAs, each still issuing its own 128 x 256 MMAs, changed nothing - the bytes into each SM
// stayed the same.)
template <int BLOCK_N, int MODE, bool SPLITK = false, bool EPI2 = false, bool LNC = false, bool PAIR = false,
          bool MASK = false>
__global__ void __launch_bounds__(kNumThreads, 1)
conv_gemm_kernel(const __grid_constant__ ConvGemmParams p) {
    using C = Cfg<BLOCK_N, MODE>;
    constexpr bool STEM = MODE == MODE_STEM;
    constexpr bool FLAT = MODE == MODE_FLAT3;
    constexpr bool WRES = STEM || FLAT;  // weights-resident modes
    const int STAGES = p.stages;      // operand stages (WRES: A stages, one per tile / channel chunk)
    const int RING = p.ring;
    // WRES: the whole weight panel of this CTA's output channels stays in shared memory for the
    // lifetime of the (persistent) CTA and an A stage holds everything one tile needs - the 7 tap-row
    // boxes of the stem, or one halo span of a flat 3x3 tile - so the MMA warp waits on ONE barrier
    // per stage and then issues 14 / 36 back-to-back tcgen05.mma.  With N = 64 an MMA occupies the
    // tensor core for only 32 cycles; a barrier round trip per 64-wide K block (the generic path)
    // makes such layers issue-bound.
    const int a_stage_bytes = WRES ? p.a_stage_bytes : C::A_STAGE;
    constexpr int B_STAGE = PAIR ? C::B_STAGE / 2 : C::B_STAGE;   // PAIR: each CTA holds half of the weight block
    const int b_region = WRES ? p.b_res_bytes : STAGES * B_STAGE;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

    const uint32_t a_smem = smem_base;
    const uint32_t b_smem = a_smem + STAGES * a_stage_bytes;
    const uint32_t st_smem = b_smem + b_region;
    const uint32_t ring_smem = st_smem + 2 * kStageBufBytes;
    const uint32_t bar_smem = ring_smem + RING * kStageBufBytes;
    uint8_t* st_gen = smem_gen + (st_smem - smem_base);
    uint8_t* ring_gen = smem_gen + (ring_smem - smem_base);
    volatile uint32_t* tmem_slot =
        reinterpret_cast<volatile uint32_t*>(smem_gen + (bar_smem - smem_base) + 320);
    const uint32_t bres_bar = bar_smem + 384u;  // WRES: resident weights have landed

    auto full_bar = [&](int s) { return bar_smem + 8u * s; };
    auto empty_bar = [&](int s) { return bar_smem + 64u + 8u * s; };
    auto rfull_bar = [&](int s) { return bar_smem + 128u + 8u * s; };
    auto rempty_bar = [&](int s) { return bar_smem + 192u + 8u * s; };
    auto tfull_bar = [&](int a) { return bar_smem + 256u + 8u * a; };
    auto tempty_bar = [&](int a) { return bar_smem + 272u + 8u * a; };
    // hand accumulator stage a back to the MMA issuer (PAIR: the leader CTA's barrier counts both CTAs' warps)
    auto release_acc = [&](int a) {
        if constexpr (PAIR)
            mbar_arrive_remote(mapa_shared(tempty_bar(a), 0));
        else
            mbar_arrive(tempty_bar(a));
    };

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_map[i]);
        tma_prefetch_desc(&p.b_map);
        tma_prefetch_desc(&p.c_map);
        tma_prefetch_desc(&p.r_map);
        for (int s = 0; s < kMaxStages; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
            if constexpr (PAIR) mbar_init(bar_smem + 448u + 8u * s, 1);   // leader: the peer's stage s has landed
            if constexpr (PAIR) mbar_init(bar_smem + 440u, 1);            // leader: the peer's resident weights have landed
            mbar_init(rfull_bar(s), 1);
            // ONE arrival per consumed sub-tile, made by the thread that issues the sub-tile's TMA store, i.e. after
            // every consumer thread has turned the residual into shared-memory stores behind a barrier.  An arrival
            // per warp right after the ld.shared instructions released the slot while loads were still in flight
            // (nothing orders an mbarrier arrive behind earlier ld.shared of the warp): under load the loader's next
            // TMA write overtook them - a few rows of a 16-byte chunk took the residual of sub-tile q + RING
            // (tools/stress_patterns.py, r02).
            mbar_init(rempty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull_bar(a), 1);
            // one arrival per epilogue warp and accumulator (EPI2: four warps per 64-column sub-tile)
            mbar_init(tempty_bar(a), (PAIR ? 2 : 1) * (EPI2 ? 4 * (BLOCK_N / 64) : 8));
        }
        mbar_init(bres_bar, 1);
        fence_mbar_init();
    }
    if (warp == 1) {
        if constexpr (PAIR)
            tmem_alloc_pair<C::TMEM_COLS>(bar_smem + 320);
        else
            tmem_alloc<C::TMEM_COLS>(bar_smem + 320);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if constexpr (PAIR) cluster_sync_all();   // the peer's barriers exist before anyone arrives on them

    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor
    // prefetch) overlaps the tail of the previous kernel in the stream; nothing below may touch
    // global memory before the previous grid has completed and flushed.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    constexpr int NSUB = BLOCK_N / 64;
    int num_k = p.kc_split ? p.num_k_total : p.num_taps * p.kc_per_tap;
    if constexpr (SPLITK) {
        if (p.dyn_k) {   // token-packed contraction (weight gradients): only the live K blocks
            int live_k = (__ldg(p.dyn_k) + C::BLOCK_K - 1) / C::BLOCK_K;
            live_k = live_k < 1 ? 1 : live_k;
            num_k = live_k < num_k ? live_k : num_k;
        }
    }
    const int box_rows = p.tw * p.th * p.nb;
    const uint32_t a_box_bytes = static_cast<uint32_t>(box_rows) * C::ROW_BYTES;
    const uint32_t stage_tx = a_box_bytes + B_STAGE;
    const int bid = static_cast<int>(blockIdx.x), nblk = static_cast<int>(gridDim.x);
    // token-packed BERT: the live row count is only known on the device
    int total_tiles = p.total_tiles;
    if (p.dyn_rows) {
        const int live = (__ldg(p.dyn_rows) + kBlockM - 1) / kBlockM * p.n_tiles_n;
        total_tiles = live < total_tiles ? live : total_tiles;
    }
    // split-K: work item = (output tile, K slice); item i covers tile i % total_tiles, slice i / total_tiles.
    // ksplit == 1 (every launch of the forward) makes items and tiles the same thing.
    int ksplit = 1;
    if constexpr (SPLITK) {
        ksplit = p.ksplit > 1 ? p.ksplit : 1;
        ksplit = ksplit < num_k ? ksplit : num_k;
    }
    const int total_items = SPLITK ? total_tiles * ksplit : total_tiles;
    int my_tiles = total_items > bid ? (total_items - bid + nblk - 1) / nblk : 0;
    // work item `it` of this CTA -> tile.  PAIR: cluster c of P takes pair-tiles j = c + it * P of
    // ceil(stripes / 2) x n_tiles_n; j = (stripe pair, column tile); CTA rank r works on stripe 2 * pair + r.  With an
    // odd stripe count the last pair's second tile lies outside the matrix: its loads are zero-filled, its stores
    // clipped by the tensor maps, and it still forwards its half of the weight tiles.
    uint32_t pair_rank = 0;
    if constexpr (PAIR) {
        pair_rank = cluster_ctarank();
        const int pair_total = (total_tiles / p.n_tiles_n + 1) / 2 * p.n_tiles_n;
        const int c = bid >> 1, P = nblk >> 1;
        my_tiles = pair_total > c ? (pair_total - c + P - 1) / P : 0;
    }
    auto tile_at = [&](int it) -> int {
        if constexpr (PAIR) {
            const int j = (bid >> 1) + it * (nblk >> 1);
            const int pm = j / p.n_tiles_n;
            return (2 * pm + static_cast<int>(pair_rank)) * p.n_tiles_n + (j - pm * p.n_tiles_n);
        } else {
            return bid + it * nblk;
        }
    };

    if (warp == 0 && WRES) {
        // ------------------------------------------------------------ TMA producer, weights-resident modes
        // FLAT: the activation is a zero-bordered [N][H+2][W+2][Cin] tensor seen as a flat list of
        // pixel rows.  One 2-D box per 64-channel chunk brings in the whole halo span of the tile; the
        // 9 taps are then row-shifted views of that span (UMMA descriptors may start at any 128-byte
        // row of a swizzled region), so every input byte crosses L2->SMEM once instead of 9 times.
        // STEM: the 7 tap-row boxes of a tile land in one stage under one barrier.
        // grid is a multiple of n_tiles_n: constant per CTA.  PAIR (flat mode, one column tile): each CTA keeps its
        // HALF of the weight panel's rows resident (b_map's box is BLOCK_N / 2 rows)
        const int n_fixed = PAIR ? 0 : bid % p.n_tiles_n;
        if (lane == 0) {
            mbar_expect_tx(bres_bar, static_cast<uint32_t>(p.b_res_bytes));
            if constexpr (FLAT) {
                for (int kc = 0; kc < p.kc_per_tap; ++kc)
                    for (int tap = 0; tap < 9; ++tap)
                        tma_load_2d(&p.b_map, bres_bar, b_smem + (kc * 9 + tap) * B_STAGE,
                                    (tap * p.kc_per_tap + kc) * 64,
                                    n_fixed * BLOCK_N + (PAIR ? static_cast<int>(pair_rank) * (BLOCK_N / 2) : 0));
            } else {
                for (int tap = 0; tap < 7; ++tap)
                    tma_load_2d(&p.b_map, bres_bar, b_smem + tap * C::B_STAGE, tap * C::BLOCK_K, 0);
            }
        }
        __syncwarp();
        int sa = 0;
        uint32_t pa = 0;
        const uint32_t span_bytes = static_cast<uint32_t>(p.span_rows) * 128u;
        // With whole-tile stages only 2-3 loads are in flight per SM, too few to cover HBM latency:
        // the tiles kPrefetch iterations ahead are pulled into L2 with bulk prefetches (no smem).
        constexpr int kPrefetch = 0;  // measured: no gain for the flat mode, a loss for the stem (r01)
        auto prefetch_tile = [&](int tile) {
            if (tile >= total_tiles || lane != 0) return;
            const TileCoord t = decode_tile(p, tile);
            if constexpr (FLAT) {
                const int f_start = (t.n0 * (p.Ho + 2) + t.h0) * p.tw;
                for (int kc = 0; kc < p.kc_per_tap; ++kc) tma_prefetch_2d(&p.a_map[0], kc * 64, f_start);
            } else {
                for (int tap = 0; tap < 7; ++tap) tma_prefetch_5d(&p.a_map[0], 0, t.w0, t.h0, tap, t.n0);
            }
        };
        if (kPrefetch > 0)
            for (int i = 1; i < kPrefetch; ++i) prefetch_tile(bid + i * nblk);
        for (int pit = 0; pit < my_tiles; ++pit) {
            const int tile = tile_at(pit);
            const TileCoord t = decode_tile(p, tile);
            if (kPrefetch > 0) prefetch_tile(tile + kPrefetch * nblk);
            if constexpr (FLAT) {
                // tile row i = padded pixel (h0+1, 1) + i in flat order; its halo span starts one padded
                // row and one pixel earlier, i.e. at padded pixel (h0, 0)  (tw == W+2)
                const int f_start = (t.n0 * (p.Ho + 2) + t.h0) * p.tw;
                for (int kc = 0; kc < p.kc_per_tap; ++kc) {
                    mbar_wait(empty_bar(sa), pa ^ 1u);
                    if (lane == 0) {
                        mbar_expect_tx(full_bar(sa), span_bytes);
                        tma_load_2d(&p.a_map[0], full_bar(sa), a_smem + sa * a_stage_bytes, kc * 64, f_start);
                    }
                    __syncwarp();
                    if (++sa == STAGES) { sa = 0; pa ^= 1u; }
                }
            } else {
                // the raw input patch of the tile, fetched ONCE (7 KB): the MMA reads its im2col rows straight out of
                // it through an overlapping un-swizzled descriptor (see the issuer).  An im2col matrix fetched
                // through an overlapping-window tensor map instead moved 57 KB per tile across the SM<->L2 fabric.
                mbar_wait(empty_bar(sa), pa ^ 1u);
                if (lane == 0) {
                    mbar_expect_tx(full_bar(sa), static_cast<uint32_t>(kStemRows * kStemRow));
                    tma_load_3d(&p.a_map[0], full_bar(sa), a_smem + sa * a_stage_bytes, 8 * t.w0, 2 * t.h0, t.n0);
                }
                __syncwarp();
                if (++sa == STAGES) { sa = 0; pa ^= 1u; }
            }
        }
    } else if (warp == 1 && WRES) {
        // ------------------------------------------------------------ MMA issuer, weights-resident modes
        constexpr uint32_t idesc = make_idesc_bf16(PAIR ? 2 * kBlockM : kBlockM, BLOCK_N, 0, 0);
        int sa = 0;
        uint32_t pa = 0;
        mbar_wait(bres_bar, 0);
        if (PAIR && pair_rank != 0) {
            // peer CTA of a pair: forwards "my weight panel / my halo span has landed" to the leader, which issues
            // the 256 x BLOCK_N x 16 MMAs for both (see the generic-mode issuer)
            if (lane == 0) mbar_arrive_remote(mapa_shared(bar_smem + 440u, 0));
            __syncwarp();
            if constexpr (FLAT) {
                for (int it = 0; it < my_tiles; ++it)
                    for (int kc = 0; kc < p.kc_per_tap; ++kc) {
                        mbar_wait(full_bar(sa), pa);
                        if (lane == 0) mbar_arrive_remote(mapa_shared(bar_smem + 448u + 8u * sa, 0));
                        __syncwarp();
                        if (++sa == STAGES) { sa = 0; pa ^= 1u; }
                    }
            }
        } else
        for (int it = 0; it < my_tiles; ++it) {
            const int acc = it & 1;
            if (PAIR && it == 0) mbar_wait(bar_smem + 440u, 0);   // the peer's half of the weight panel is resident
            mbar_wait(tempty_bar(acc), ((it >> 1) & 1) ^ 1u);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
            if constexpr (FLAT) {
                for (int kc = 0; kc < p.kc_per_tap; ++kc) {
                    mbar_wait(full_bar(sa), pa);
                    if constexpr (PAIR) mbar_wait(bar_smem + 448u + 8u * sa, pa);
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t a0 = a_smem + sa * a_stage_bytes;
                        const uint32_t b0 = b_smem + kc * 9 * B_STAGE;
#pragma unroll
                        for (int tap = 0; tap < 9; ++tap) {
                            const int tap_row = (tap / 3) * p.tw + (tap % 3);  // row shift of this tap's view
                            const uint64_t adesc = make_smem_desc(a0 + tap_row * 128, 0, C::SBO, C::LAYOUT);
                            const uint64_t bdesc = make_smem_desc(b0 + tap * B_STAGE, 0, C::SBO, C::LAYOUT);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if constexpr (PAIR)
                                    umma_bf16_pair(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc,
                                                   (kc | tap | k) != 0 ? 1u : 0u);
                                else
                                    umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc,
                                              (kc | tap | k) != 0 ? 1u : 0u);
                            }
                        }
                        if constexpr (PAIR) {
                            umma_commit_pair(empty_bar(sa), 3);
                            if (kc == p.kc_per_tap - 1) umma_commit_pair(tfull_bar(acc), 3);
                        } else {
                            umma_commit(empty_bar(sa));
                            if (kc == p.kc_per_tap - 1) umma_commit(tfull_bar(acc));
                        }
                    }
                    __syncwarp();
                    if (++sa == STAGES) { sa = 0; pa ^= 1u; }
                }
            } else {
                mbar_wait(full_bar(sa), pa);
                tc_fence_after();
                if (lane == 0) {
#pragma unroll
                    // GEMM row m = (output row m / 8, output pixel m % 8) of the 8 x 16 tile; its K = 32 slice for tap
                    // row r is 8 pixels x 4 channels = 64 contiguous bytes at pixel 2*(m % 8) of patch row
                    // 2*(m / 8) + r.  In the un-swizzled K-major layout a core matrix is 8 rows 16 bytes apart, K
                    // chunks are LBO apart and 8-row groups SBO apart: LBO = 16 B (chunk c of row m IS chunk 0 of
                    // row m + c: the windows overlap) and SBO = 2 patch rows describe exactly that matrix, so no
                    // im2col copy exists anywhere (tools/exp_hankel_desc.cu verifies the addressing).
                    for (int tap = 0; tap < 7; ++tap) {
                        const uint64_t bdesc = make_smem_desc(b_smem + tap * C::B_STAGE, 0, C::SBO, C::LAYOUT);
#pragma unroll
                        for (int k = 0; k < C::BLOCK_K / 16; ++k) {
                            const uint64_t adesc = make_smem_desc(
                                a_smem + sa * a_stage_bytes + tap * kStemRow + k * 32, 16, 2 * kStemRow, 0);
                            umma_bf16(d_tmem, adesc, bdesc + 2 * k, idesc, (tap | k) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(empty_bar(sa));
                    umma_commit(tfull_bar(acc));
                }
                __syncwarp();
                if (++sa == STAGES) { sa = 0; pa ^= 1u; }
            }
        }
    } else if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        int stage = 0;
        uint32_t phase = 0;
        for (int pit = 0; pit < my_tiles; ++pit) {
            const int item = tile_at(pit);
            const int split = SPLITK ? item / total_tiles : 0;
            const TileCoord t = decode_tile(p, SPLITK ? item - split * total_tiles : item);
            const int k_begin = SPLITK ? split * num_k / ksplit : 0;
            const int k_end = SPLITK ? (split + 1) * num_k / ksplit : num_k;
            for (int ks = k_begin; ks < k_end; ++ks) {
                mbar_wait(empty_bar(stage), phase ^ 1u);
                if (lane == 0) {
                    mbar_expect_tx(full_bar(stage), stage_tx);
                    const uint32_t a_dst = a_smem + stage * C::A_STAGE;
                    const uint32_t b_dst = b_smem + stage * B_STAGE;
                    // K-concatenated pair of 1x1 convolutions: chunks [0, kc_split) read taps[0], the rest taps[1]
                    const int tap = p.kc_split ? (ks >= p.kc_split ? 1 : 0) : ks / p.kc_per_tap;
                    const int kc = ks - tap * (p.kc_split ? p.kc_split : p.kc_per_tap);
                    const TapDesc td = p.taps[tap];
                    tma_load_4d(&p.a_map[td.map], full_bar(stage), a_dst, kc * C::BLOCK_K,
                                t.w0 + td.dw, t.h0 + td.dh, t.n0);
                    // PAIR: my half of the weight block (b_map's box is BLOCK_N / 2 rows)
                    tma_load_2d(&p.b_map, full_bar(stage), b_dst, ks * C::BLOCK_K,
                                t.n_idx * BLOCK_N + (PAIR ? static_cast<int>(pair_rank) * (BLOCK_N / 2) : 0));
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        constexpr uint32_t idesc = make_idesc_bf16(PAIR ? 2 * kBlockM : kBlockM, BLOCK_N, 0, 0);
        int stage = 0;
        uint32_t phase = 0;
        if (PAIR && pair_rank != 0) {
            // peer CTA: no MMAs of its own - tell the leader when each of my stages has landed (the TMA's bytes are
            // visible to me through the barrier wait, to the leader through the release / acquire pair at cluster scope)
            for (int it = 0; it < my_tiles; ++it)
                for (int ks = 0; ks < num_k; ++ks) {
                    mbar_wait(full_bar(stage), phase);
                    if (lane == 0) mbar_arrive_remote(mapa_shared(bar_smem + 448u + 8u * stage, 0));
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
        } else
        for (int it = 0; it < my_tiles; ++it) {
            const int item = tile_at(it);
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait(tempty_bar(acc), acc_phase ^ 1u);   // PAIR: both CTAs' epilogues have drained it
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
            const int split = SPLITK ? item / total_tiles : 0;
            const int k_begin = SPLITK ? split * num_k / ksplit : 0;
            const int k_end = SPLITK ? (split + 1) * num_k / ksplit : num_k;
            for (int ks = k_begin; ks < k_end; ++ks) {
                mbar_wait(full_bar(stage), phase);
                // (plain waits on the remotely-arrived barriers, as for any cluster barrier: an acquire at cluster scope
                // per K step cost more than the step's 512 tensor cycles and held the pair at 700 TFLOP/s)
                if constexpr (PAIR) mbar_wait(bar_smem + 448u + 8u * stage, phase);
                tc_fence_after();
                if (lane == 0) {
                    const uint64_t adesc =
                        make_smem_desc(a_smem + stage * C::A_STAGE, 0, C::SBO, C::LAYOUT);
                    const uint64_t bdesc =
                        make_smem_desc(b_smem + stage * B_STAGE, 0, C::SBO, C::LAYOUT);
#pragma unroll
                    for (int k = 0; k < C::BLOCK_K / 16; ++k) {
                        // +32 bytes (encoded >>4) per 16-element K slice inside the swizzle span
                        if constexpr (PAIR)
                            umma_bf16_pair(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc,
                                           (ks != k_begin || k != 0) ? 1u : 0u);
                        else
                            umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc,
                                      (ks != k_begin || k != 0) ? 1u : 0u);
                    }
                    if constexpr (PAIR) {   // the stage is free, the accumulator ready: in BOTH CTAs
                        umma_commit_pair(empty_bar(stage), 3);
                        if (ks == k_end - 1) umma_commit_pair(tfull_bar(acc), 3);
                    } else {
                        umma_commit(empty_bar(stage));
                        if (ks == k_end - 1) umma_commit(tfull_bar(acc));
                    }
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 10) {
        // ------------------------------------------------------------ residual loader
        // Runs up to RING sub-tiles ahead of the epilogue so the residual (an HBM read the epilogue
        // would otherwise wait ~2 us for) is already in shared memory when its sub-tile is due.
        if (p.has_res) {
            const uint32_t res_bytes = static_cast<uint32_t>(box_rows) * 128u;
            int slot = 0;
            uint32_t phase = 0;
            for (int it = 0; it < my_tiles; ++it) {
                const TileCoord t = decode_tile(p, SPLITK ? tile_at(it) % total_tiles : tile_at(it));
                for (int sub = 0; sub < NSUB; ++sub) {
                    mbar_wait(rempty_bar(slot), phase ^ 1u);
                    if (lane == 0) {
                        mbar_expect_tx(rfull_bar(slot), res_bytes);
                        tma_load_4d(&p.r_map, rfull_bar(slot), ring_smem + slot * kStageBufBytes,
                                    t.n_idx * BLOCK_N + sub * 64, t.w0, t.h0, t.n0);
                    }
                    __syncwarp();
                    if (++slot == RING) { slot = 0; phase ^= 1u; }
                }
            }
        }
    } else if (LNC) {
        // ------------------------------------------------------------ epilogue with LayerNorm across the row's CTAs
        const int quarter = warp & 3;
        const int half = (warp - 2) >> 2;
        const int row = quarter * 32 + lane;
        const int epi_tid = threadIdx.x - 64;
        const bool has_res = p.has_res != 0;
        const int csize = p.n_tiles_n;
        const int npart = 2 * csize;                     // partials per row: (CTA, column half)
        constexpr float kPartN = static_cast<float>(NSUB * 32);   // columns behind one partial
        const float inv_n = 1.0f / (static_cast<float>(csize) * BLOCK_N);
        int rslot = 0;
        uint32_t rphase = 0;
        int q = 0;
        for (int it = 0; it < my_tiles; ++it) {
            const int acc = it & 1;
            const TileCoord t = decode_tile(p, tile_at(it));
            const uint32_t tbase =
                tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BLOCK_N + half * 32;
            mbar_wait(tfull_bar(acc), (it >> 1) & 1u);
            tc_fence_after();
            // ---- pass 1: x = acc + bias + residual back into TMEM, running sum / sum of squares of this thread's columns
            float sum = 0.0f, ssq = 0.0f;
            for (int sub = 0; sub < NSUB; ++sub) {
                const int col0 = t.n_idx * BLOCK_N + sub * 64 + half * 32;
                uint32_t v[32];
                tmem_ld32(tbase + sub * 64, v);
                tmem_ld_wait();
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j));
                    f[j + 0] = __uint_as_float(v[j + 0]) + b4.x;
                    f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
                    f[j + 2] = __uint_as_float(v[j + 2]) + b4.z;
                    f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
                }
                if (has_res) {
                    mbar_wait(rfull_bar(rslot), rphase);
                    const uint8_t* r_row = ring_gen + rslot * kStageBufBytes + row * 128;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const int chunk = (half * 4 + c) ^ (row & 7);
                        const uint4 r4 = *reinterpret_cast<const uint4*>(r_row + chunk * 16);
                        const float2 r0 = unpack_bf16(r4.x), r1 = unpack_bf16(r4.y),
                                     r2 = unpack_bf16(r4.z), r3 = unpack_bf16(r4.w);
                        f[c * 8 + 0] += r0.x; f[c * 8 + 1] += r0.y;
                        f[c * 8 + 2] += r1.x; f[c * 8 + 3] += r1.y;
                        f[c * 8 + 4] += r2.x; f[c * 8 + 5] += r2.y;
                        f[c * 8 + 6] += r3.x; f[c * 8 + 7] += r3.y;
                    }
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    sum += f[j];
                    ssq = fmaf(f[j], f[j], ssq);
                    v[j] = __float_as_uint(f[j]);
                }
                tmem_st32(tbase + sub * 64, v);
                tmem_st_wait();
                if (has_res) {
                    // the stores above consumed every residual load of this thread: behind the barrier the slot is free
                    named_bar_sync(2, kEpiThreads);
                    if (epi_tid == 0) mbar_arrive(rempty_bar(rslot));
                    if (++rslot == RING) { rslot = 0; rphase ^= 1u; }
                }
            }
            // ---- publish (mean, M2) of these kPartN columns to the CTAs that hold the rest of the row
            const float mean_p = sum * (1.0f / kPartN);
            const float m2_p = fmaxf(ssq - sum * mean_p, 0.0f);
            // through L2: the csize CTAs of a stripe are neighbours in the persistent tile order, so all of them are
            // resident (grid <= SM count) and a spin on the stripe's arrival counter cannot deadlock
            float2 part[8];
            const int stripe = tile_at(it) / csize;
            char* rec = reinterpret_cast<char*>(p.ln_stats) + static_cast<long long>(stripe) * kLnStripeBytes;
            float2* srow = reinterpret_cast<float2*>(rec) + row * 8;
            __stcg(srow + t.n_idx * 2 + half, make_float2(mean_p, m2_p));
            __threadfence();
            __syncwarp();
            unsigned int* cnt = reinterpret_cast<unsigned int*>(rec + 128 * 8 * 8);
            const unsigned int want = 8u * csize;
            if (lane == 0) {
                asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(cnt) : "memory");
                unsigned int seen;
                const long long t0 = clock64();
                do {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(cnt) : "memory");
                    if (clock64() - t0 > 4000000000LL) __trap();
                } while (seen < want);
            }
            __syncwarp();
            for (int i = 0; i < npart; ++i) part[i] = __ldcg(srow + i);
            __syncwarp();
            if (lane == 0) {   // the last warp to have read the stripe's partials re-arms both counters
                unsigned int left;
                asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(left) : "l"(cnt + 1) : "memory");
                if (left == want - 1) {
                    cnt[1] = 0;
                    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(cnt), "r"(0u) : "memory");
                }
            }
            float mean = 0.0f;
            for (int i = 0; i < npart; ++i) mean += part[i].x;
            mean *= 1.0f / static_cast<float>(npart);
            float m2 = 0.0f;
            for (int i = 0; i < npart; ++i) {
                const float d = part[i].x - mean;
                m2 += part[i].y + kPartN * d * d;
            }
            const float rstd = rsqrtf(m2 * inv_n + p.ln_eps);
            // ---- pass 2: normalise, store
            for (int sub = 0; sub < NSUB; ++sub, ++q) {
                const uint32_t buf = q & 1u;
                const int col0 = t.n_idx * BLOCK_N + sub * 64 + half * 32;
                uint32_t v[32];
                tmem_ld32(tbase + sub * 64, v);
                tmem_ld_wait();
                if (sub == NSUB - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) release_acc(acc);
                }
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.ln_g + col0 + j));
                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.ln_b + col0 + j));
                    f[j + 0] = fmaf((__uint_as_float(v[j + 0]) - mean) * rstd, g4.x, b4.x);
                    f[j + 1] = fmaf((__uint_as_float(v[j + 1]) - mean) * rstd, g4.y, b4.y);
                    f[j + 2] = fmaf((__uint_as_float(v[j + 2]) - mean) * rstd, g4.z, b4.z);
                    f[j + 3] = fmaf((__uint_as_float(v[j + 3]) - mean) * rstd, g4.w, b4.w);
                }
                if (epi_tid == 0) tma_store_wait_read<1>();
                named_bar_sync(2, kEpiThreads);
                uint8_t* st_row = st_gen + buf * kStageBufBytes + row * 128;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint4 o;
                    o.x = pack_bf16(f[c * 8 + 0], f[c * 8 + 1]);
                    o.y = pack_bf16(f[c * 8 + 2], f[c * 8 + 3]);
                    o.z = pack_bf16(f[c * 8 + 4], f[c * 8 + 5]);
                    o.w = pack_bf16(f[c * 8 + 6], f[c * 8 + 7]);
                    const int chunk = (half * 4 + c) ^ (row & 7);
                    *reinterpret_cast<uint4*>(st_row + chunk * 16) = o;
                }
                fence_proxy_async_smem();
                named_bar_sync(1, kEpiThreads);
                if (epi_tid == 0) {
                    tma_store_4d(&p.c_map, st_smem + buf * kStageBufBytes, t.n_idx * BLOCK_N + sub * 64, t.w0, t.h0,
                                 t.n0);
                    tma_store_commit();
                }
            }
        }
        if (epi_tid == 0) tma_store_wait_all<0>();
    } else if (EPI2) {
        // ------------------------------------------------------------ epilogue, two groups of four warps
        const int grp = (warp - 2) >> 2;
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        const bool leader = ((warp - 2) & 3) == 0 && lane == 0;   // issues this group's TMA stores
        const int bar_a = 1 + 2 * grp, bar_b = 2 + 2 * grp;        // this group's named barriers (128 threads)
        const int wi = row % p.tw;
        const int hi = (row / p.tw) % p.th;
        const int ni = row / (p.tw * p.th);
        const bool has_res = p.has_res != 0;
        const int nq = my_tiles * NSUB;
        uint8_t* st_row = st_gen + grp * kStageBufBytes + row * 128;   // one staging buffer per group
        for (int q = grp; q < nq; q += 2) {
            const int sub = q % NSUB;
            const int it = q / NSUB;
            const int acc = it & 1;
            const TileCoord t = decode_tile(p, tile_at(it));
            const int col0 = t.n_idx * BLOCK_N + sub * 64;
            mbar_wait(tfull_bar(acc), (it >> 1) & 1u);
            tc_fence_after();
            uint32_t v0[32], v1[32];
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BLOCK_N + sub * 64;
            tmem_ld32(taddr, v0);
            tmem_ld32(taddr + 32, v1);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) release_acc(acc);
            float f[64];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
                if (p.bias) {
                    b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j));
                    b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + 32 + j));
                }
                f[j + 0] = __uint_as_float(v0[j + 0]) + b0.x;
                f[j + 1] = __uint_as_float(v0[j + 1]) + b0.y;
                f[j + 2] = __uint_as_float(v0[j + 2]) + b0.z;
                f[j + 3] = __uint_as_float(v0[j + 3]) + b0.w;
                f[32 + j + 0] = __uint_as_float(v1[j + 0]) + b1.x;
                f[32 + j + 1] = __uint_as_float(v1[j + 1]) + b1.y;
                f[32 + j + 2] = __uint_as_float(v1[j + 2]) + b1.z;
                f[32 + j + 3] = __uint_as_float(v1[j + 3]) + b1.w;
            }
            if (has_res) {   // the loader fetched the residual sub-tiles in q order
                const int rslot = q % RING;
                mbar_wait(rfull_bar(rslot), static_cast<uint32_t>(q / RING) & 1u);
                const uint8_t* r_row = ring_gen + rslot * kStageBufBytes + row * 128;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const uint4 r4 = *reinterpret_cast<const uint4*>(r_row + ((c ^ (row & 7)) << 4));
                    const float2 r0 = unpack_bf16(r4.x), r1 = unpack_bf16(r4.y),
                                 r2 = unpack_bf16(r4.z), r3 = unpack_bf16(r4.w);
                    f[c * 8 + 0] += r0.x; f[c * 8 + 1] += r0.y;
                    f[c * 8 + 2] += r1.x; f[c * 8 + 3] += r1.y;
                    f[c * 8 + 4] += r2.x; f[c * 8 + 5] += r2.y;
                    f[c * 8 + 6] += r3.x; f[c * 8 + 7] += r3.y;
                }
            }
            if (p.act == ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 64; ++j) f[j] = fmaxf(f[j], 0.0f);
            } else if (p.act == ACT_GELU) {
#pragma unroll
                for (int j = 0; j < 64; ++j) f[j] = gelu_erf_fast(f[j]);
            }
            if (p.out_f32) {
                const bool row_ok = (row < box_rows) && (t.n0 + ni < p.Nimg) && (t.h0 + hi < p.Ho) &&
                                    (t.w0 + wi < p.Wo);
                if (row_ok) {
                    const long long pix =
                        (static_cast<long long>(t.n0 + ni) * p.Ho + (t.h0 + hi)) * p.Wo + (t.w0 + wi);
                    float* f32_row = p.out_f32 + pix * p.ld_f32 + col0;
#pragma unroll
                    for (int j = 0; j < 64; j += 4)
                        *reinterpret_cast<float4*>(f32_row + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                }
            }
            // this group's staging buffer was the source of its previous TMA store: it must have been read
            if (leader) tma_store_wait_read<0>();
            named_bar_sync(bar_b, 128);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint4 o;
                o.x = pack_bf16(f[c * 8 + 0], f[c * 8 + 1]);
                o.y = pack_bf16(f[c * 8 + 2], f[c * 8 + 3]);
                o.z = pack_bf16(f[c * 8 + 4], f[c * 8 + 5]);
                o.w = pack_bf16(f[c * 8 + 6], f[c * 8 + 7]);
                *reinterpret_cast<uint4*>(st_row + ((c ^ (row & 7)) << 4)) = o;
            }
            if constexpr (STEM) {
                if (p.pool_out) {
                    // ---- fused MaxPool2d(3, 2, 1): the tile (8 x 16 stem pixels, rows of 64 channels) is in this
                    // group's staging buffer.  Pooled pixel (pr, pc) of the 9 x 5 it touches takes the maximum over
                    // the part of its 3 x 3 window that lies inside the tile; neighbouring tiles add theirs with the
                    // same reduction.  One item = one pooled pixel x 8 channels (16 bytes).
                    named_bar_sync(bar_a, 128);
                    const uint8_t* tile = st_gen + grp * kStageBufBytes;
                    const int gt = threadIdx.x - 64 - grp * 128;   // 0..127 inside the group
                    for (int item = gt; item < 45 * 8; item += 128) {
                        const int ch = item & 7, pp = item >> 3;
                        const int pr = pp / 5, pc = pp - pr * 5;
                        const int ph = (t.h0 >> 1) + pr, pw = (t.w0 >> 1) + pc;
                        if (ph >= p.pool_h || pw >= p.pool_w) continue;
                        __nv_bfloat162 m0 = __floats2bfloat162_rn(0.f, 0.f), m1 = m0, m2 = m0, m3 = m0;
                        // window positions outside the tile are clamped onto the tile's edge: every pooled pixel of the
                        // 9 x 5 has at least its centre row / column inside, so a clamped position is a duplicate of
                        // an in-window element (max is idempotent) and the loop has no thread-dependent branch - with
                        // per-thread `continue`s the four pooled pixels of a warp diverged and every ld.shared was
                        // issued up to four times (ncu, r02: 15.5 M extra shared-load wavefronts per launch)
#pragma unroll
                        for (int dr = -1; dr <= 1; ++dr) {
                            const int hr = min(max(2 * pr + dr, 0), 15);
#pragma unroll
                            for (int dc = -1; dc <= 1; ++dc) {
                                const int wc = min(max(2 * pc + dc, 0), 7);
                                const int m = hr * 8 + wc;
                                const uint4 v = *reinterpret_cast<const uint4*>(tile + m * 128 + ((ch ^ (m & 7)) << 4));
                                m0 = __hmax2(m0, *reinterpret_cast<const __nv_bfloat162*>(&v.x));
                                m1 = __hmax2(m1, *reinterpret_cast<const __nv_bfloat162*>(&v.y));
                                m2 = __hmax2(m2, *reinterpret_cast<const __nv_bfloat162*>(&v.z));
                                m3 = __hmax2(m3, *reinterpret_cast<const __nv_bfloat162*>(&v.w));
                            }
                        }
                        uint4 o;
                        o.x = *reinterpret_cast<uint32_t*>(&m0);
                        o.y = *reinterpret_cast<uint32_t*>(&m1);
                        o.z = *reinterpret_cast<uint32_t*>(&m2);
                        o.w = *reinterpret_cast<uint32_t*>(&m3);
                        __nv_bfloat16* dst = p.pool_out +
                            ((static_cast<long long>(t.n0) * p.pool_h + ph) * p.pool_w + pw) * 64 + ch * 8;
                        red_max_bf16x8(dst, o);
                    }
                    continue;   // the next write of this staging buffer is behind the bar_b barrier of the next tile
                }
            }
            fence_proxy_async_smem();
            named_bar_sync(bar_a, 128);
            // every thread of the group has stored values that depend on its residual loads: the ring slot is free
            if (leader && has_res) mbar_arrive(rempty_bar(q % RING));
            if (leader && p.store_bf16) {
                if (p.c_blocked)
                    tma_store_4d(&p.c_map, st_smem + grp * kStageBufBytes, 0, t.w0, t.n_idx * NSUB + sub, 0);
                else
                    tma_store_4d(&p.c_map, st_smem + grp * kStageBufBytes, col0, t.w0, t.h0, t.n0);
                tma_store_commit();
            }
        }
        if (leader) tma_store_wait_all<0>();
    } else {
        // ------------------------------------------------------------ epilogue (warps 2..9)
        const int quarter = warp & 3;           // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;       // which 32 of the sub-tile's 64 columns
        const int row = quarter * 32 + lane;    // accumulator row == smem staging row
        const int epi_tid = threadIdx.x - 64;   // 0..255
        const int wi = row % p.tw;
        const int hi = (row / p.tw) % p.th;
        const int ni = row / (p.tw * p.th);
        const bool has_res = p.has_res != 0;
        const int nq = my_tiles * NSUB;  // sub-tiles this CTA produces
        int rslot = 0;
        uint32_t rphase = 0;

        TileCoord t = decode_tile(p, SPLITK ? (total_tiles > 0 ? bid % total_tiles : 0) : tile_at(0));
        for (int q = 0; q < nq; ++q) {
            const int sub = q % NSUB;
            const int it = q / NSUB;
            const int acc = it & 1;
            const uint32_t buf = q & 1u;
            if (sub == 0) t = decode_tile(p, SPLITK ? tile_at(it) % total_tiles : tile_at(it));
            const int col0 = t.n_idx * BLOCK_N + sub * 64 + half * 32;  // first global column of this thread

            if (sub == 0) {
                mbar_wait(tfull_bar(acc), (it >> 1) & 1u);
                tc_fence_after();
            }
            uint32_t v[32];
            tmem_ld32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BLOCK_N + sub * 64 +
                          half * 32,
                      v);
            tmem_ld_wait();
            if (sub == NSUB - 1) {
                // accumulator stage fully read by this warp: hand it back to the MMA warp early
                tc_fence_before();
                __syncwarp();
                if (lane == 0) release_acc(acc);
            }
            float f[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j));
                f[j + 0] = __uint_as_float(v[j + 0]) + b4.x;
                f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
                f[j + 2] = __uint_as_float(v[j + 2]) + b4.z;
                f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
            }
            if (has_res) {
                mbar_wait(rfull_bar(rslot), rphase);
                const uint8_t* r_row = ring_gen + rslot * kStageBufBytes + row * 128;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int chunk = (half * 4 + c) ^ (row & 7);
                    const uint4 r4 = *reinterpret_cast<const uint4*>(r_row + chunk * 16);
                    const float2 r0 = unpack_bf16(r4.x), r1 = unpack_bf16(r4.y),
                                 r2 = unpack_bf16(r4.z), r3 = unpack_bf16(r4.w);
                    if constexpr (MASK) {   // ReLU backward: keep the positions whose saved activation is > 0
                        f[c * 8 + 0] = r0.x > 0.0f ? f[c * 8 + 0] : 0.0f; f[c * 8 + 1] = r0.y > 0.0f ? f[c * 8 + 1] : 0.0f;
                        f[c * 8 + 2] = r1.x > 0.0f ? f[c * 8 + 2] : 0.0f; f[c * 8 + 3] = r1.y > 0.0f ? f[c * 8 + 3] : 0.0f;
                        f[c * 8 + 4] = r2.x > 0.0f ? f[c * 8 + 4] : 0.0f; f[c * 8 + 5] = r2.y > 0.0f ? f[c * 8 + 5] : 0.0f;
                        f[c * 8 + 6] = r3.x > 0.0f ? f[c * 8 + 6] : 0.0f; f[c * 8 + 7] = r3.y > 0.0f ? f[c * 8 + 7] : 0.0f;
                    } else {
                        f[c * 8 + 0] += r0.x; f[c * 8 + 1] += r0.y;
                        f[c * 8 + 2] += r1.x; f[c * 8 + 3] += r1.y;
                        f[c * 8 + 4] += r2.x; f[c * 8 + 5] += r2.y;
                        f[c * 8 + 6] += r3.x; f[c * 8 + 7] += r3.y;
                    }
                }
            }
            if (p.act == ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.0f);
            } else if (p.act == ACT_GELU) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = gelu_erf_fast(f[j]);
            }
            if (p.out_f32) {
                const bool row_ok = (row < box_rows) && (t.n0 + ni < p.Nimg) && (t.h0 + hi < p.Ho) &&
                                    (t.w0 + wi < p.Wo);
                if (row_ok) {
                    const long long pix =
                        (static_cast<long long>(t.n0 + ni) * p.Ho + (t.h0 + hi)) * p.Wo + (t.w0 + wi);
                    float* f32_row = p.out_f32 + pix * p.ld_f32 + col0;
                    if constexpr (SPLITK) {   // split-K partial result: reduce in L2
#pragma unroll
                        for (int j = 0; j < 32; j += 4)
                            atomicAdd(reinterpret_cast<float4*>(f32_row + j),
                                      make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j += 4)
                            *reinterpret_cast<float4*>(f32_row + j) =
                                make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                    }
                }
            }
            // staging buffer `buf` was the source of TMA store q-2: it must have been read out
            if (epi_tid == 0) tma_store_wait_read<1>();
            named_bar_sync(2, kEpiThreads);
            // bf16 pack into the 128B-swizzled staging tile (matches the C tensor map)
            uint8_t* st_row = st_gen + buf * kStageBufBytes + row * 128;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint4 o;
                o.x = pack_bf16(f[c * 8 + 0], f[c * 8 + 1]);
                o.y = pack_bf16(f[c * 8 + 2], f[c * 8 + 3]);
                o.z = pack_bf16(f[c * 8 + 4], f[c * 8 + 5]);
                o.w = pack_bf16(f[c * 8 + 6], f[c * 8 + 7]);
                const int chunk = (half * 4 + c) ^ (row & 7);
                *reinterpret_cast<uint4*>(st_row + chunk * 16) = o;
            }
            fence_proxy_async_smem();
            named_bar_sync(1, kEpiThreads);
            if (has_res) {
                // every epilogue thread has stored values that depend on its residual loads: the ring slot is free
                if (epi_tid == 0) mbar_arrive(rempty_bar(rslot));
                if (++rslot == RING) { rslot = 0; rphase ^= 1u; }
            }
            if (epi_tid == 0 && p.store_bf16) {
                if (p.c_blocked)
                    tma_store_4d(&p.c_map, st_smem + buf * kStageBufBytes, 0, t.w0, t.n_idx * NSUB + sub, 0);
                else
                    tma_store_4d(&p.c_map, st_smem + buf * kStageBufBytes, t.n_idx * BLOCK_N + sub * 64,
                                 t.w0, t.h0, t.n0);
                tma_store_commit();
            }
        }
        if (epi_tid == 0) tma_store_wait_all<0>();
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();   // no CTA leaves while its peer may still arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        if constexpr (PAIR)
            tmem_dealloc_pair<C::TMEM_COLS>(tmem_base);
        else
            tmem_dealloc<C::TMEM_COLS>(tmem_base);
    }
}

template <int BLOCK_N, int MODE, bool SPLITK = false, bool EPI2 = false, bool LNC = false, bool PAIR = false,
          bool MASK = false>
int launch_variant(const GemmLaunch* g, cudaStream_t stream) {
    using C = Cfg<BLOCK_N, MODE>;
    static bool attr_set = false;
    auto kfn = conv_gemm_kernel<BLOCK_N, MODE, SPLITK, EPI2, LNC, PAIR, MASK>;
    if (!attr_set) {
        cudaError_t e =
            cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
        if (e != cudaSuccess) {
            set_last_error("cudaFuncSetAttribute(smem=%d): %s", kSmemLimit, cudaGetErrorString(e));
            return -static_cast<int>(e);
        }
        attr_set = true;
    }
    const int smem = MODE != MODE_GENERIC
                         ? C::FIXED + g->p.stages * g->p.a_stage_bytes + g->p.b_res_bytes
                         : C::FIXED + g->p.stages * (PAIR ? C::A_STAGE + C::B_STAGE / 2 : C::STAGE) +
                               g->p.ring * kStageBufBytes;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g->grid);
    cfg.blockDim = dim3(kNumThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = g_use_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (PAIR) {
        // one cluster = two stripes of one column tile; as many clusters as are co-resident
        constexpr int cs = 2;
        attr[1].id = cudaLaunchAttributeClusterDimension;
        attr[1].val.clusterDim.x = cs;
        attr[1].val.clusterDim.y = 1;
        attr[1].val.clusterDim.z = 1;
        cfg.numAttrs = 2;
        static int max_clusters = 0;
        if (max_clusters == 0) {
            cfg.gridDim = dim3(cs * 16);
            int n = 0;
            cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kfn, &cfg);
            if (e != cudaSuccess || n <= 0) {
                set_last_error("cudaOccupancyMaxActiveClusters(cluster of %d): %s", cs, cudaGetErrorString(e));
                return e != cudaSuccess ? -static_cast<int>(e) : -1;
            }
            max_clusters = n;
            if (getenv("MRD_DEBUG_PRINT"))
                fprintf(stderr, "[mrd] conv_gemm_kernel<%d,%d,%d,%d,%d,%d>: %d co-resident clusters of %d CTAs\n", BLOCK_N,
                        MODE, SPLITK, EPI2, LNC, PAIR, n, cs);
        }
        int clusters = g->grid / cs;
        if (clusters > max_clusters) clusters = max_clusters;
        if (clusters < 1) clusters = 1;
        cfg.gridDim = dim3(clusters * cs);
    }
    cudaError_t e = cudaLaunchKernelEx(&cfg, kfn, g->p);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("conv_gemm_kernel<%d,%d> launch: %s", BLOCK_N, MODE,
                       cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

// Pipeline depths for one launch: operand stages vs residual ring (both live in the same 227 KB).
void pick_pipeline(ConvGemmParams* p, int block_n, bool stem, bool pair = false) {
    const int stage = stem ? (128 * 64 + 64 * 64) : (128 * 128 + (pair ? block_n / 2 : block_n) * 128);
    const int fixed = 2 * kStageBufBytes + kBarBytes + 1024;
    const int avail = kSmemLimit - fixed;
    const int num_k = p->num_taps * p->kc_per_tap;
    if (!p->has_res) {
        int s = avail / stage;
        p->stages = s > kMaxStages ? kMaxStages : s;
        if (const char* e = getenv("MRD_DEBUG_STAGES")) {   // timing experiments: a shallower operand pipeline
            const int v = atoi(e);
            if (v >= 2 && v < p->stages) p->stages = v;
        }
        p->ring = 0;
        return;
    }
    // with a residual: short-K launches are memory-bound -> few operand stages (each already covers
    // a whole tile), many residual sub-tiles in flight; long-K launches keep >= 3 operand stages
    int s = num_k <= 2 ? 2 : 3;
    while (s > 2 && (avail - s * stage) / kStageBufBytes < 2) --s;
    int r = (avail - s * stage) / kStageBufBytes;
    if (r > kMaxRing) {
        r = kMaxRing;
        int extra = (avail - r * kStageBufBytes) / stage;  // leftover smem back to the operand pipeline
        if (extra > s) s = extra > kMaxStages ? kMaxStages : extra;
    }
    if (num_k > 6 && r > 4) {   // long K: one tile's residual sub-tiles in flight are enough, the rest feeds the operands
        r = 4;
        int more = (avail - r * kStageBufBytes) / stage;
        if (more > s) s = more > kMaxStages ? kMaxStages : more;
    }
    apply_debug_env();
    if (g_debug_ring > 0 && g_debug_ring < r) r = g_debug_ring;
    p->stages = s;
    p->ring = r;
}

#define MRD_GEMM_TRY(expr)          \
    do {                            \
        int rc__ = (expr);          \
        if (rc__ != 0) return rc__; \
    } while (0)

int pick_block_n(int n, long long m_tiles, int sms) {
    // widest N tile that divides N and still gives every SM at least one tile
    if (n % 256 == 0 && m_tiles * (n / 256) >= sms) return 256;
    if (n % 128 == 0 && m_tiles * (n / 128) >= sms) return 128;
    if (n % 64 == 0 && (n % 128 != 0 || m_tiles * (n / 128) < sms)) return 64;
    if (n % 128 == 0) return 128;
    return 64;
}

int finish_plan(GemmLaunch* g, int block_n) {
    ConvGemmParams& p = g->p;
    g->block_n = block_n;
    p.n_tiles_n = p.Cout / block_n;
    const long long m_tiles = static_cast<long long>(p.tiles_w) * p.tiles_h * p.tiles_img;
    const long long total = m_tiles * p.n_tiles_n;
    if (total <= 0 || total > 0x7fffffffLL) {
        set_last_error("gemm plan: bad tile count %lld", total);
        return -1;
    }
    p.total_tiles = static_cast<int>(total);
    const int sms = gemm_num_sms();
    g->grid = p.total_tiles < sms ? p.total_tiles : sms;
    if (g->flat3 || g->stem) {
        // weights-resident: every CTA keeps one n-tile's weights, so its tiles must share n_idx
        g->grid = g->grid / p.n_tiles_n * p.n_tiles_n;
        if (g->grid < p.n_tiles_n) g->grid = p.n_tiles_n;
    } else {
        pick_pipeline(&p, block_n, false, g->pair != 0);
    }
    return 0;
}

}  // namespace

void gemm_set_pdl(bool on) { g_use_pdl = on; }

int gemm_num_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            sms <= 0)
            sms = 148;
    }
    return sms;
}

namespace {
int plan_gemm_impl(GemmLaunch* g, const __nv_bfloat16* A, long long lda, int M, int K,
                   const __nv_bfloat16* W, int N, const float* bias, __nv_bfloat16* Cout, long long ldc,
                   const __nv_bfloat16* residual, long long ld_res, float* out_f32, long long ld_f32,
                   int act, int c_blocked, int force_bn);
}

int plan_gemm(GemmLaunch* g, const __nv_bfloat16* A, long long lda, int M, int K,
              const __nv_bfloat16* W, int N, const float* bias, __nv_bfloat16* Cout, long long ldc,
              const __nv_bfloat16* residual, long long ld_res, float* out_f32, long long ld_f32,
              int act, int c_blocked) {
    return plan_gemm_impl(g, A, lda, M, K, W, N, bias, Cout, ldc, residual, ld_res, out_f32, ld_f32, act, c_blocked, 0);
}

namespace {
int plan_gemm_impl(GemmLaunch* g, const __nv_bfloat16* A, long long lda, int M, int K,
                   const __nv_bfloat16* W, int N, const float* bias, __nv_bfloat16* Cout, long long ldc,
                   const __nv_bfloat16* residual, long long ld_res, float* out_f32, long long ld_f32,
                   int act, int c_blocked, int force_bn) {
    memset(g, 0, sizeof(*g));
    if (M <= 0 || K <= 0 || N <= 0 || K % 64 != 0 || N % 64 != 0 || lda % 8 != 0 ||
        (Cout && ldc % 8 != 0)) {
        set_last_error("plan_gemm: unsupported shape M=%d N=%d K=%d lda=%lld ldc=%lld", M, N, K,
                       lda, ldc);
        return -1;
    }
    ConvGemmParams& p = g->p;
    g->stem = 0;
    p.bias = bias;
    p.has_res = residual != nullptr;
    p.out_f32 = out_f32;
    p.ld_f32 = ld_f32;
    p.num_taps = 1;
    p.kc_per_tap = K / 64;
    p.taps[0] = TapDesc{0, 0, 0, 0};
    p.tw = 128; p.th = 1; p.nb = 1;
    p.tiles_w = (M + 127) / 128; p.tiles_h = 1; p.tiles_img = 1;
    p.Wo = M; p.Ho = 1; p.Nimg = 1; p.Cout = N;
    p.act = act;
    p.store_bf16 = Cout != nullptr;
    g->flops = 2.0 * M * static_cast<double>(N) * K;
    g->bytes = 2.0 * (1.0 * M * K + 1.0 * N * K + (Cout ? 1.0 * M * N : 0.0) + (residual ? 1.0 * M * N : 0.0)) +
               (out_f32 ? 4.0 * M * N : 0.0);

    const int bn = force_bn ? force_bn : pick_block_n(N, p.tiles_w, gemm_num_sms());
    // at least two tiles per SM: below that the pairing has nothing to amortise
    g->pair = (bn == 256 && static_cast<long long>(p.tiles_w) * (N / 256) >= 2LL * gemm_num_sms()) ? 1 : 0;
    {
        uint64_t dims[4] = {(uint64_t)K, (uint64_t)M, 1, 1};
        uint64_t str[3] = {(uint64_t)lda * 2, (uint64_t)lda * 2 * M, (uint64_t)lda * 2 * M};
        uint32_t box[4] = {64, 128, 1, 1};
        int rc = encode_tensor_map(&p.a_map[0], A, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        for (int i = 1; i < 4; ++i) p.a_map[i] = p.a_map[0];
    }
    {
        uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
        uint64_t str[1] = {(uint64_t)K * 2};
        uint32_t box[2] = {64, (uint32_t)(g->pair ? bn / 2 : bn)};   // PAIR: each CTA fetches half a weight tile
        int rc = encode_tensor_map(&p.b_map, W, 2, 2, dims, str, box, 128);
        if (rc) return rc;
    }
    p.c_blocked = (Cout && c_blocked) ? 1 : 0;
    if (Cout && c_blocked) {
        uint64_t dims[4] = {64, (uint64_t)M, (uint64_t)(N / 64), 1};
        uint64_t str[3] = {128, (uint64_t)M * 128, (uint64_t)M * 128 * (N / 64)};
        uint32_t box[4] = {64, 128, 1, 1};
        int rc = encode_tensor_map(&p.c_map, Cout, 2, 4, dims, str, box, 128);
        if (rc) return rc;
    } else if (Cout) {
        uint64_t dims[4] = {(uint64_t)N, (uint64_t)M, 1, 1};
        uint64_t str[3] = {(uint64_t)ldc * 2, (uint64_t)ldc * 2 * M, (uint64_t)ldc * 2 * M};
        uint32_t box[4] = {64, 128, 1, 1};
        int rc = encode_tensor_map(&p.c_map, Cout, 2, 4, dims, str, box, 128);
        if (rc) return rc;
    } else {
        p.c_map = p.a_map[0];  // never dereferenced (store_bf16 == 0)
    }
    if (residual) {
        if (ld_res % 8 != 0) {
            set_last_error("plan_gemm: residual row stride must be a multiple of 8 elements");
            return -1;
        }
        uint64_t dims[4] = {(uint64_t)N, (uint64_t)M, 1, 1};
        uint64_t str[3] = {(uint64_t)ld_res * 2, (uint64_t)ld_res * 2 * M, (uint64_t)ld_res * 2 * M};
        uint32_t box[4] = {64, 128, 1, 1};
        int rc = encode_tensor_map(&p.r_map, residual, 2, 4, dims, str, box, 128);
        if (rc) return rc;
    } else {
        p.r_map = p.a_map[0];  // never dereferenced (has_res == 0)
    }
    return finish_plan(g, bn);
}
}  // namespace

int plan_gemm_ln(GemmLaunch* g, const __nv_bfloat16* A, long long lda, int M, int K, const __nv_bfloat16* W, int N,
                 const float* bias, __nv_bfloat16* Cout, long long ldc, const __nv_bfloat16* residual,
                 long long ld_res, const float* gamma, const float* beta, float eps, void* stats_ws) {
    if (N % 256 != 0 || N / 256 < 2 || N / 256 > 4 || !Cout || !bias || !gamma || !beta) return 1;
    if (!stats_ws) {
        set_last_error("gemm + LayerNorm: stats_ws is required (a zeroed device buffer of mrd_gemm_ln_ws_bytes(M) bytes)");
        return -1;
    }
    // always 256-wide tiles, however few rows there are: which kernel (and so which rounding) a row goes through
    // must not depend on the batch it arrives in - sub-batches reproduce the rows of the full batch bit for bit
    MRD_GEMM_TRY(plan_gemm_impl(g, A, lda, M, K, W, N, bias, Cout, ldc, residual, ld_res, nullptr, 0, ACT_NONE, 0, 256));
    ConvGemmParams& p = g->p;
    p.ln_g = gamma;
    p.ln_b = beta;
    p.ln_eps = eps;
    p.ln_stats = static_cast<float2*>(stats_ws);   // records of kLnStripeBytes
    g->lnc = 1;
    // three operand stages (four of the pair's smaller ones), two residual sub-tiles in flight
    if (p.has_res) {
        p.stages = g->pair ? 4 : 3;
        p.ring = 2;
    } else if (p.stages > (g->pair ? 5 : 3)) {
        p.stages = g->pair ? 5 : 3;
    }
    g->bytes += 8.0 * N;   // gamma / beta
    return 0;
}

size_t gemm_ln_ws_bytes(int M) {
    const size_t stripes = ((static_cast<size_t>(M) + 127) / 128 + 1) & ~static_cast<size_t>(1);
    return stripes * kLnStripeBytes;   // (even stripe count: the pair's second stripe may lie outside the matrix)
}

int plan_gemm_splitk(GemmLaunch* g, const __nv_bfloat16* A, long long lda, int M, int K,
                     const __nv_bfloat16* W, int N, float* out_f32, long long ld_f32, const int* dyn_k) {
    if (!out_f32) {
        set_last_error("plan_gemm_splitk: an fp32 destination is required");
        return -1;
    }
    MRD_GEMM_TRY(plan_gemm(g, A, lda, M, K, W, N, nullptr, nullptr, 0, nullptr, 0, out_f32, ld_f32, ACT_NONE));
    // plan_gemm sized the N tile for a single pass (64 wide when there are few tiles); with split-K the SMs
    // are filled by K slices instead, so take the widest tile (best operand reuse) and rebuild the B map
    const int bn = N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 64);
    g->pair = 0;
    {
        uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
        uint64_t str[1] = {(uint64_t)K * 2};
        uint32_t box[2] = {64, (uint32_t)bn};
        int rc = encode_tensor_map(&g->p.b_map, W, 2, 2, dims, str, box, 128);
        if (rc) return rc;
    }
    MRD_GEMM_TRY(finish_plan(g, bn));
    const int sms = gemm_num_sms();
    int ks = sms / g->p.total_tiles;
    const int num_k = K / 64;
    if (ks > num_k / 4) ks = num_k / 4;   // at least 4 K blocks per work item
    if (ks < 1) ks = 1;
    g->p.ksplit = ks;
    g->p.f32_accum = 1;
    g->p.dyn_k = dyn_k;
    const long long items = static_cast<long long>(g->p.total_tiles) * ks;
    g->grid = items < sms ? static_cast<int>(items) : sms;
    return 0;
}

int plan_conv(GemmLaunch* g, const __nv_bfloat16* X, int N, int H, int W, int Cin,
              const __nv_bfloat16* Wt, int Cout, int ksize, int stride, const float* bias,
              __nv_bfloat16* Y, const __nv_bfloat16* residual, int act, int out_pad) {
    if (ksize == 1 && stride == 1 && out_pad == 0) {
        const long long M = static_cast<long long>(N) * H * W;
        if (M > 0x7fffffffLL) {
            set_last_error("plan_conv: M too large");
            return -1;
        }
        return plan_gemm(g, X, Cin, static_cast<int>(M), Cin, Wt, Cout, bias, Y, Cout, residual,
                         Cout, nullptr, 0, act);
    }
    memset(g, 0, sizeof(*g));
    if ((ksize != 1 && ksize != 3) || (stride != 1 && stride != 2) || Cin % 64 != 0 ||
        Cout % 64 != 0 || H % stride != 0 || W % stride != 0 || N <= 0) {
        set_last_error("plan_conv: unsupported conv k=%d s=%d Cin=%d Cout=%d H=%d W=%d", ksize,
                       stride, Cin, Cout, H, W);
        return -1;
    }
    ConvGemmParams& p = g->p;
    g->stem = 0;
    const int Ho = H / stride, Wo = W / stride;
    p.bias = bias;
    p.has_res = residual != nullptr;
    p.out_f32 = nullptr;
    p.ld_f32 = 0;
    p.num_taps = ksize * ksize;
    p.kc_per_tap = Cin / 64;
    p.Wo = Wo; p.Ho = Ho; p.Nimg = N; p.Cout = Cout;
    p.act = act;
    p.store_bf16 = 1;
    g->flops = 2.0 * N * Ho * Wo * static_cast<double>(Cout) * Cin * ksize * ksize;
    g->bytes = 2.0 * (1.0 * N * H * W * Cin + 1.0 * Cout * Cin * ksize * ksize +
                      1.0 * N * Ho * Wo * Cout * (residual ? 2.0 : 1.0));

    // tile box: as many whole output rows (then whole images) as fit in 128 GEMM rows
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

    // taps and A maps
    if (stride == 1) {
        int t = 0;
        for (int r = 0; r < ksize; ++r)
            for (int s = 0; s < ksize; ++s)
                p.taps[t++] = TapDesc{0, (int8_t)(r - ksize / 2), (int8_t)(s - ksize / 2), 0};
        uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
        uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, (uint32_t)p.nb};
        int rc = encode_tensor_map(&p.a_map[0], X, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        for (int i = 1; i < 4; ++i) p.a_map[i] = p.a_map[0];
    } else {
        // stride 2: input row 2*ho + r - pad lives in parity phase a = (r - pad) & 1 at phase-row
        // ho + floor((r - pad) / 2); same for columns.  Four phase views of the same tensor.
        const int pad = ksize / 2;
        int t = 0;
        for (int r = 0; r < ksize; ++r)
            for (int s = 0; s < ksize; ++s) {
                const int dr = r - pad, ds = s - pad;
                const int a = dr & 1, b = ds & 1;
                const int qh = (dr - a) / 2, qw = (ds - b) / 2;  // floor division
                p.taps[t++] = TapDesc{(int8_t)(a * 2 + b), (int8_t)qh, (int8_t)qw, 0};
            }
        for (int a = 0; a < 2; ++a)
            for (int b = 0; b < 2; ++b) {
                const __nv_bfloat16* base = X + (static_cast<long long>(a) * W + b) * Cin;
                uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)(W / 2), (uint64_t)(H / 2), (uint64_t)N};
                uint64_t str[3] = {(uint64_t)2 * Cin * 2, (uint64_t)2 * W * Cin * 2,
                                   (uint64_t)H * W * Cin * 2};
                uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, (uint32_t)p.nb};
                int rc = encode_tensor_map(&p.a_map[a * 2 + b], base, 2, 4, dims, str, box, 128);
                if (rc) return rc;
            }
    }
    const long long m_tiles = static_cast<long long>(p.tiles_w) * p.tiles_h * p.tiles_img;
    const int bn = pick_block_n(Cout, m_tiles, gemm_num_sms());
    // CTA pairs (cta_group::2) for the tensor-bound 3x3 / strided convolutions of layers 3 and 4 as well: two tiles of
    // 128 output pixels share each weight block
    g->pair = (bn == 256 && m_tiles * (Cout / 256) >= 2LL * gemm_num_sms()) ? 1 : 0;
    {
        const uint64_t Kt = static_cast<uint64_t>(Cin) * ksize * ksize;
        uint64_t dims[2] = {Kt, (uint64_t)Cout};
        uint64_t str[1] = {Kt * 2};
        uint32_t box[2] = {64, (uint32_t)(g->pair ? bn / 2 : bn)};
        int rc = encode_tensor_map(&p.b_map, Wt, 2, 2, dims, str, box, 128);
        if (rc) return rc;
    }
    {
        // out_pad: Y is a zero-bordered [N][Ho+2p][Wo+2p][Cout] tensor; only its interior is written
        const int Wy = Wo + 2 * out_pad, Hy = Ho + 2 * out_pad;
        __nv_bfloat16* y0 = Y + (static_cast<long long>(out_pad) * Wy + out_pad) * Cout;
        uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Wy * Cout * 2,
                           (uint64_t)Hy * Wy * Cout * 2};
        uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, (uint32_t)p.nb};
        int rc = encode_tensor_map(&p.c_map, y0, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        p.r_map = p.c_map;
        if (residual) {
            if (out_pad) {
                set_last_error("plan_conv: residual with a padded output is not supported");
                return -1;
            }
            rc = encode_tensor_map(&p.r_map, residual, 2, 4, dims, str, box, 128);
            if (rc) return rc;
        }
    }
    return finish_plan(g, bn);
}

int plan_conv1x1_dual(GemmLaunch* g, const __nv_bfloat16* X0, int C0, const __nv_bfloat16* X1, int C1,
                      int stride1, int N, int Ho, int Wo, const __nv_bfloat16* Wcat, int Cout,
                      const float* bias, __nv_bfloat16* Y, int act) {
    memset(g, 0, sizeof(*g));
    if (C0 % 64 != 0 || C1 % 64 != 0 || Cout % 64 != 0 || (stride1 != 1 && stride1 != 2) || N <= 0 || Ho <= 0 ||
        Wo <= 0) {
        set_last_error("plan_conv1x1_dual: unsupported shape C0=%d C1=%d Cout=%d stride=%d", C0, C1, Cout, stride1);
        return -1;
    }
    ConvGemmParams& p = g->p;
    const long long M = static_cast<long long>(N) * Ho * Wo;
    if (M > 0x7fffffffLL) {
        set_last_error("plan_conv1x1_dual: M too large");
        return -1;
    }
    p.bias = bias;
    p.has_res = 0;
    p.num_taps = 2;
    p.kc_per_tap = C0 / 64;
    p.kc_split = C0 / 64;
    p.num_k_total = (C0 + C1) / 64;
    p.taps[0] = TapDesc{0, 0, 0, 0};
    p.taps[1] = TapDesc{1, 0, 0, 0};
    p.Cout = Cout;
    p.act = act;
    p.store_bf16 = 1;
    g->flops = 2.0 * M * static_cast<double>(Cout) * (C0 + C1);
    g->bytes = 2.0 * (1.0 * M * C0 + 1.0 * M * C1 + 1.0 * Cout * (C0 + C1) + 1.0 * M * Cout);
    if (stride1 == 1) {
        // both operands are plain [M, C] matrices: flat 128-row tiles as in plan_gemm
        p.tw = 128; p.th = 1; p.nb = 1;
        p.tiles_w = static_cast<int>((M + 127) / 128); p.tiles_h = 1; p.tiles_img = 1;
        p.Wo = static_cast<int>(M); p.Ho = 1; p.Nimg = 1;
        const __nv_bfloat16* xs[2] = {X0, X1};
        const int cs[2] = {C0, C1};
        for (int i = 0; i < 2; ++i) {
            uint64_t dims[4] = {(uint64_t)cs[i], (uint64_t)M, 1, 1};
            uint64_t str[3] = {(uint64_t)cs[i] * 2, (uint64_t)cs[i] * 2 * M, (uint64_t)cs[i] * 2 * M};
            uint32_t box[4] = {64, 128, 1, 1};
            int rc = encode_tensor_map(&p.a_map[i], xs[i], 2, 4, dims, str, box, 128);
            if (rc) return rc;
        }
        uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)M, 1, 1};
        uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Cout * 2 * M, (uint64_t)Cout * 2 * M};
        uint32_t box[4] = {64, 128, 1, 1};
        int rc = encode_tensor_map(&p.c_map, Y, 2, 4, dims, str, box, 128);
        if (rc) return rc;
    } else {
        // X1 is read at every second row / column: tiles are boxes of output pixels (as in plan_conv)
        p.Wo = Wo; p.Ho = Ho; p.Nimg = N;
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
        const int H = Ho * 2, W = Wo * 2;
        uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, (uint32_t)p.nb};
        {
            uint64_t dims[4] = {(uint64_t)C0, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
            uint64_t str[3] = {(uint64_t)C0 * 2, (uint64_t)Wo * C0 * 2, (uint64_t)Ho * Wo * C0 * 2};
            int rc = encode_tensor_map(&p.a_map[0], X0, 2, 4, dims, str, box, 128);
            if (rc) return rc;
        }
        {
            uint64_t dims[4] = {(uint64_t)C1, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
            uint64_t str[3] = {(uint64_t)2 * C1 * 2, (uint64_t)2 * W * C1 * 2, (uint64_t)H * W * C1 * 2};
            int rc = encode_tensor_map(&p.a_map[1], X1, 2, 4, dims, str, box, 128);
            if (rc) return rc;
        }
        uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Wo * Cout * 2, (uint64_t)Ho * Wo * Cout * 2};
        int rc = encode_tensor_map(&p.c_map, Y, 2, 4, dims, str, box, 128);
        if (rc) return rc;
    }
    p.a_map[2] = p.a_map[3] = p.a_map[0];
    p.r_map = p.c_map;  // never dereferenced (has_res == 0)
    const long long m_tiles = static_cast<long long>(p.tiles_w) * p.tiles_h * p.tiles_img;
    const int bn = pick_block_n(Cout, m_tiles, gemm_num_sms());
    {
        const uint64_t Kt = static_cast<uint64_t>(C0 + C1);
        uint64_t dims[2] = {Kt, (uint64_t)Cout};
        uint64_t str[1] = {Kt * 2};
        uint32_t box[2] = {64, (uint32_t)bn};
        int rc = encode_tensor_map(&p.b_map, Wcat, 2, 2, dims, str, box, 128);
        if (rc) return rc;
    }
    return finish_plan(g, bn);
}

bool conv3x3_flat_supported(int H, int W, int Cin, int Cout) {
    const int Wp = W + 2;
    if (H < 1 || W < 1 || Wp > 128 || Cin % 64 != 0 || Cout % 64 != 0) return false;
    const int th = 128 / Wp;
    if ((th + 2) * Wp + 2 > 256) return false;
    int rows_alloc = 2 * Wp + 2 + 128;
    if (rows_alloc < (th + 2) * Wp + 2) rows_alloc = (th + 2) * Wp + 2;
    const int a_stage = ((rows_alloc * 128) + 1023) / 1024 * 1024;
    const int fixed = 2 * kStageBufBytes + kBarBytes + 1024;
    return fixed + 2 * a_stage + 9 * (Cin / 64) * 64 * 128 <= kSmemLimit;
}

int plan_conv3x3_flat(GemmLaunch* g, const __nv_bfloat16* Xpad, int N, int H, int W, int Cin,
                      const __nv_bfloat16* Wt, int Cout, const float* bias, __nv_bfloat16* Y, int act) {
    memset(g, 0, sizeof(*g));
    const int Wp = W + 2, Hp = H + 2;
    const int th = 128 / Wp;
    if (th < 1 || Cin % 64 != 0 || Cout % 64 != 0 || N <= 0) {
        set_last_error("plan_conv3x3_flat: unsupported shape H=%d W=%d Cin=%d Cout=%d", H, W, Cin, Cout);
        return -1;
    }
    ConvGemmParams& p = g->p;
    g->flat3 = 1;
    int rows_alloc = 2 * Wp + 2 + 128;  // the MMA reads 128 rows from any tap offset (<= 2*Wp + 2)
    if (rows_alloc < (th + 2) * Wp + 2) rows_alloc = (th + 2) * Wp + 2;
    const int a_stage = ((rows_alloc * 128) + 1023) / 1024 * 1024;
    const int fixed = 2 * kStageBufBytes + kBarBytes + 1024;
    // widest N tile whose whole 3x3 weight panel fits next to two halo-span stages
    int bn = 0;
    for (int cand : {128, 64})
        if (Cout % cand == 0 && bn == 0 &&
            fixed + 2 * a_stage + 9 * (Cin / 64) * cand * 128 <= kSmemLimit)
            bn = cand;
    // CTA pairs (cta_group::2): when only a 64-wide panel fits a single CTA (N = 64 MMAs run at half rate), two CTAs
    // keep half of a 128-wide panel each and the pair issues 256 x 128 x 16 MMAs at the full rate (layer2 conv2:
    // 4.70 -> 2.2-2.7 ms per 4096 images).  A 64-channel layer gains too (layer1 conv2: 4.4 -> 3.7 ms): a
    // 256 x 64 x 16 pair instruction takes ~45-58 cycles against 62 for 128 x 64 x 16 on one SM
    // (tools/exp_pair_rate.cu).  One column tile only (the resident panel fixes a CTA's column tile).
    const long long flat_tiles = static_cast<long long>((H + th - 1) / th) * N;
    if (bn == 64 && (Cout == 128 || Cout == 64) &&
        flat_tiles >= 2LL * gemm_num_sms() && fixed + 2 * a_stage + 9 * (Cin / 64) * (Cout / 2) * 128 <= kSmemLimit) {
        g->pair = 1;
        bn = Cout;
    }
    if (bn == 0) {
        set_last_error("plan_conv3x3_flat: weight panel of Cin=%d does not fit in shared memory", Cin);
        return -1;
    }
    p.bias = bias;
    p.has_res = 0;
    p.num_taps = 9;
    p.kc_per_tap = Cin / 64;
    p.tw = Wp; p.th = th; p.nb = 1;
    // tile row i is output pixel (h0 + i / (W+2), i % (W+2)): columns W and W+1 of every row are the
    // right/left border positions of the flat order; the TMA store clips them (w >= W is out of bounds)
    p.w_shift = 0;
    p.tiles_w = 1; p.tiles_h = (H + th - 1) / th; p.tiles_img = N;
    p.Wo = W; p.Ho = H; p.Nimg = N; p.Cout = Cout;
    p.act = act;
    p.store_bf16 = 1;
    p.span_rows = (th + 2) * Wp + 2;
    p.a_stage_bytes = a_stage;
    if (p.span_rows > 256) {
        set_last_error("plan_conv3x3_flat: halo span of %d rows exceeds the TMA box limit", p.span_rows);
        return -1;
    }
    g->flops = 2.0 * N * H * W * static_cast<double>(Cout) * Cin * 9;
    g->bytes = 2.0 * (1.0 * N * Hp * Wp * Cin + 9.0 * Cout * Cin + 1.0 * N * H * W * Cout);
    {
        const uint64_t R = static_cast<uint64_t>(N) * Hp * Wp;
        uint64_t dims[2] = {(uint64_t)Cin, R};
        uint64_t str[1] = {(uint64_t)Cin * 2};
        uint32_t box[2] = {64, (uint32_t)p.span_rows};
        int rc = encode_tensor_map(&p.a_map[0], Xpad, 2, 2, dims, str, box, 128);
        if (rc) return rc;
        for (int i = 1; i < 4; ++i) p.a_map[i] = p.a_map[0];
    }
    {
        const uint64_t Kt = static_cast<uint64_t>(Cin) * 9;
        uint64_t dims[2] = {Kt, (uint64_t)Cout};
        uint64_t str[1] = {Kt * 2};
        uint32_t box[2] = {64, (uint32_t)(g->pair ? bn / 2 : bn)};
        int rc = encode_tensor_map(&p.b_map, Wt, 2, 2, dims, str, box, 128);
        if (rc) return rc;
    }
    {
        uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)W, (uint64_t)H, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)W * Cout * 2, (uint64_t)H * W * Cout * 2};
        uint32_t box[4] = {64, (uint32_t)Wp, (uint32_t)th, 1};
        int rc = encode_tensor_map(&p.c_map, Y, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        p.r_map = p.c_map;
    }
    // pipeline: resident weight panel + as many halo-span stages as fit
    p.b_res_bytes = 9 * (Cin / 64) * (g->pair ? bn / 2 : bn) * 128;   // per CTA
    p.ring = 0;
    int st = (kSmemLimit - fixed - p.b_res_bytes) / a_stage;
    p.stages = st > kMaxStages ? kMaxStages : st;
    return finish_plan(g, bn);
}

int plan_stem(GemmLaunch* g, const __nv_bfloat16* Xpad, int N, int H, int W,
              const __nv_bfloat16* Wst, const float* bias, __nv_bfloat16* Y, int act) {
    memset(g, 0, sizeof(*g));
    if (H % 2 != 0 || W % 2 != 0 || N <= 0) {
        set_last_error("plan_stem: H, W must be even (got %d x %d)", H, W);
        return -1;
    }
    ConvGemmParams& p = g->p;
    g->stem = 1;
    const int Ho = H / 2, Wo = W / 2;
    const int Hp = H + 6, Wp = W + 8;  // 3 rows/cols of zero padding before, 3/5 after
    p.bias = bias;
    p.has_res = 0;
    p.out_f32 = nullptr;
    p.num_taps = 7;
    p.kc_per_tap = 1;
    p.Wo = Wo; p.Ho = Ho; p.Nimg = N; p.Cout = 64;
    p.act = act;
    p.store_bf16 = 1;
    g->flops = 2.0 * N * Ho * Wo * 64.0 * 147.0;
    g->bytes = 2.0 * (1.0 * N * (H + 6) * (W + 8) * 4 + 64.0 * 7 * 32 + 1.0 * N * Ho * Wo * 64);
    if (Wo % 8 != 0 || Ho % 16 != 0) {
        set_last_error("plan_stem: output %dx%d must be a multiple of the 8 x 16 tile", Wo, Ho);
        return -1;
    }
    p.tw = 8;
    p.th = 16;
    p.nb = 1;
    p.tiles_w = Wo / 8;
    p.tiles_h = Ho / 16;
    p.tiles_img = N;
    {
        // the padded image as rows of (W+8)*4 bf16; one box = the raw patch of an 8 x 16 output tile: 37 rows
        // (2*15 + 7 taps) x 24 pixels (2*7 + 7 taps, rounded up to a 16-byte multiple), un-swizzled
        uint64_t dims[3] = {(uint64_t)Wp * 4, (uint64_t)Hp, (uint64_t)N};
        uint64_t str[2] = {(uint64_t)Wp * 8, (uint64_t)Hp * Wp * 8};
        uint32_t box[3] = {kStemRow / 2, kStemRows, 1};
        int rc = encode_tensor_map(&p.a_map[0], Xpad, 2, 3, dims, str, box, 0);
        if (rc) return rc;
        for (int i = 1; i < 4; ++i) p.a_map[i] = p.a_map[0];
    }
    {
        uint64_t dims[2] = {7 * 32, 64};
        uint64_t str[1] = {7 * 32 * 2};
        uint32_t box[2] = {32, 64};
        int rc = encode_tensor_map(&p.b_map, Wst, 2, 2, dims, str, box, 64);
        if (rc) return rc;
    }
    {
        uint64_t dims[4] = {64, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
        uint64_t str[3] = {64 * 2, (uint64_t)Wo * 64 * 2, (uint64_t)Ho * Wo * 64 * 2};
        uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, 1};
        int rc = encode_tensor_map(&p.c_map, Y, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        p.r_map = p.c_map;
    }
    // weights-resident: one raw patch (7 KB) per A stage, the 7 x 4 KB weight tiles resident
    p.a_stage_bytes = 7168;
    p.b_res_bytes = 7 * 64 * 64;
    p.ring = 0;
    p.stages = kMaxStages;
    return finish_plan(g, 64);
}

int plan_stem_pool(GemmLaunch* g, const __nv_bfloat16* Xpad, int N, int H, int W,
                   const __nv_bfloat16* Wst, const float* bias, __nv_bfloat16* P) {
    // the C map is never used (nothing is stored through it): any valid tensor of the output's shape class will do
    int rc = plan_stem(g, Xpad, N, H, W, Wst, bias, P, ACT_RELU);
    if (rc) return rc;
    g->p.pool_out = P;
    g->p.pool_h = H / 4;
    g->p.pool_w = W / 4;
    g->p.store_bf16 = 0;
    g->bytes = 2.0 * (1.0 * N * (H + 6) * (W + 8) * 4 + 64.0 * 7 * 32 + 1.0 * N * (H / 4) * (W / 4) * 64);
    return 0;
}

int plan_conv_dgrad(GemmLaunch* g, const __nv_bfloat16* dY, int N, int Ho, int Wo, int Cy, const __nv_bfloat16* Wt,
                    long long ldw, int ntaps, const TapDesc* taps, int Cx, __nv_bfloat16* dX, int sh, int sw, int ph,
                    int pw, const __nv_bfloat16* aux, int aux_mode) {
    memset(g, 0, sizeof(*g));
    if (N <= 0 || Ho <= 0 || Wo <= 0 || Cy % 64 != 0 || Cx % 64 != 0 || ntaps < 1 || ntaps > 9 || sh < 1 ||
        sh > 2 || sw < 1 || sw > 2 || ph < 0 || ph >= sh || pw < 0 || pw >= sw || ldw % 8 != 0 ||
        ldw < 1LL * ntaps * Cy || aux_mode < 0 || aux_mode > 2 || (aux_mode != 0) != (aux != nullptr)) {
        set_last_error("plan_conv_dgrad: unsupported N=%d %dx%d Cy=%d Cx=%d taps=%d stride %dx%d phase (%d,%d) aux %d",
                       N, Ho, Wo, Cy, Cx, ntaps, sh, sw, ph, pw, aux_mode);
        return -1;
    }
    for (int t = 0; t < ntaps; ++t)
        if (taps[t].dh < -1 || taps[t].dh > 1 || taps[t].dw < -1 || taps[t].dw > 1) {
            set_last_error("plan_conv_dgrad: tap shifts must lie in [-1, 1]");
            return -1;
        }
    ConvGemmParams& p = g->p;
    const int Hx = sh * Ho, Wx = sw * Wo;
    p.bias = nullptr;
    p.has_res = aux != nullptr;
    p.num_taps = ntaps;
    p.kc_per_tap = Cy / 64;
    for (int t = 0; t < ntaps; ++t) p.taps[t] = TapDesc{0, taps[t].dh, taps[t].dw, 0};
    p.Wo = Wo; p.Ho = Ho; p.Nimg = N; p.Cout = Cx;
    p.act = ACT_NONE;
    p.store_bf16 = 1;
    g->relu_mask = aux_mode == 2;
    g->flops = 2.0 * N * Ho * Wo * static_cast<double>(Cx) * Cy * ntaps;
    g->bytes = 2.0 * (1.0 * N * Ho * Wo * Cy + 1.0 * Cx * Cy * ntaps + 1.0 * N * Ho * Wo * Cx * (aux ? 2.0 : 1.0));
    // tile box as plan_conv: whole rows, then whole images, of the dY grid
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
    {   // dY rows / columns shifted outside the grid are zero-filled by TMA (the far edge of a transposed convolution)
        uint64_t dims[4] = {(uint64_t)Cy, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)Cy * 2, (uint64_t)Wo * Cy * 2, (uint64_t)Ho * Wo * Cy * 2};
        uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, (uint32_t)p.nb};
        int rc = encode_tensor_map(&p.a_map[0], dY, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        for (int i = 1; i < 4; ++i) p.a_map[i] = p.a_map[0];
    }
    const long long m_tiles = static_cast<long long>(p.tiles_w) * p.tiles_h * p.tiles_img;
    const int bn = pick_block_n(Cx, m_tiles, gemm_num_sms());
    g->pair = (bn == 256 && m_tiles * (Cx / 256) >= 2LL * gemm_num_sms()) ? 1 : 0;
    {
        uint64_t dims[2] = {(uint64_t)ntaps * Cy, (uint64_t)Cx};
        uint64_t str[1] = {(uint64_t)ldw * 2};
        uint32_t box[2] = {64, (uint32_t)(g->pair ? bn / 2 : bn)};
        int rc = encode_tensor_map(&p.b_map, Wt, 2, 2, dims, str, box, 128);
        if (rc) return rc;
    }
    {   // the (ph, pw) phase of dX as a [N][Ho][Wo][Cx] view; the mask / addend through the same view
        const long long off = (static_cast<long long>(ph) * Wx + pw) * Cx;
        uint64_t dims[4] = {(uint64_t)Cx, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
        uint64_t str[3] = {(uint64_t)sw * Cx * 2, (uint64_t)sh * Wx * Cx * 2, (uint64_t)Hx * Wx * Cx * 2};
        uint32_t box[4] = {64, (uint32_t)p.tw, (uint32_t)p.th, (uint32_t)p.nb};
        int rc = encode_tensor_map(&p.c_map, dX + off, 2, 4, dims, str, box, 128);
        if (rc) return rc;
        p.r_map = p.c_map;
        if (aux) {
            rc = encode_tensor_map(&p.r_map, aux + off, 2, 4, dims, str, box, 128);
            if (rc) return rc;
        }
    }
    return finish_plan(g, bn);
}

int launch_gemm(const GemmLaunch* g, cudaStream_t stream) {
    apply_debug_env();
    if (g->stem) {
        // the fused pooling lives in the two-group epilogue
        if (g->p.pool_out) return launch_variant<64, MODE_STEM, false, true>(g, stream);
        return launch_variant<64, MODE_STEM>(g, stream);
    }
    if (g->lnc)
        return g->pair ? launch_variant<256, MODE_GENERIC, false, false, true, true>(g, stream)
                       : launch_variant<256, MODE_GENERIC, false, false, true>(g, stream);
    if (g->flat3 && g->pair)
        return g->block_n == 128 ? launch_variant<128, MODE_FLAT3, false, true, false, true>(g, stream)
                                 : launch_variant<64, MODE_FLAT3, false, true, false, true>(g, stream);
    if (g->flat3) {
        switch (g->block_n) {
            case 64: return launch_variant<64, MODE_FLAT3, false, true>(g, stream);
            case 128: return launch_variant<128, MODE_FLAT3, false, true>(g, stream);
        }
        set_last_error("launch_gemm: bad flat3 block_n %d", g->block_n);
        return -1;
    }
    if (g->relu_mask) {   // plan_conv_dgrad with a ReLU mask: single-group epilogue only
        if (g->pair && g->block_n == 256) return launch_variant<256, MODE_GENERIC, false, false, false, true, true>(g, stream);
        switch (g->block_n) {
            case 64: return launch_variant<64, MODE_GENERIC, false, false, false, false, true>(g, stream);
            case 128: return launch_variant<128, MODE_GENERIC, false, false, false, false, true>(g, stream);
            case 256: return launch_variant<256, MODE_GENERIC, false, false, false, false, true>(g, stream);
        }
        set_last_error("launch_gemm: bad masked block_n %d", g->block_n);
        return -1;
    }
    if (g->p.f32_accum) {   // plan_gemm_splitk
        switch (g->block_n) {
            case 64: return launch_variant<64, MODE_GENERIC, true>(g, stream);
            case 128: return launch_variant<128, MODE_GENERIC, true>(g, stream);
            case 256: return launch_variant<256, MODE_GENERIC, true>(g, stream);
        }
    }
    // Two-group epilogue where the per-sub-tile latency chain bounds the launch (measured, r02: GELU epilogue -5 %,
    // short-K residual convolutions -7..-12 %); long-K GEMMs without activation are main-loop-bound and keep the
    // single-group epilogue with its two shared staging buffers (QKV lost 5 % with the split).
    const bool chain_bound = g->p.act == ACT_GELU || g->p.num_taps * g->p.kc_per_tap <= 6 ||
                             (g->p.kc_split && g->p.num_k_total <= 6);
    const bool epi2 = chain_bound && !(g->p.kc_split && g->p.num_k_total > 6);
    if (g->pair && g->block_n == 256) {
        if (epi2) return launch_variant<256, MODE_GENERIC, false, true, false, true>(g, stream);
        return launch_variant<256, MODE_GENERIC, false, false, false, true>(g, stream);
    }
    if (epi2) {
        switch (g->block_n) {
            case 64: return launch_variant<64, MODE_GENERIC, false, true>(g, stream);
            case 128: return launch_variant<128, MODE_GENERIC, false, true>(g, stream);
            case 256: return launch_variant<256, MODE_GENERIC, false, true>(g, stream);
        }
    }
    switch (g->block_n) {
        case 64: return launch_variant<64, MODE_GENERIC>(g, stream);
        case 128: return launch_variant<128, MODE_GENERIC>(g, stream);
        case 256: return launch_variant<256, MODE_GENERIC>(g, stream);
    }
    set_last_error("launch_gemm: bad block_n %d", g->block_n);
    return -1;
}

}  // namespace mrd
