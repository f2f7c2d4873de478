// Thin inline-PTX wrappers for the Blackwell (sm_100a) primitives the kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and fences.
// Nothing here is architecture-portable on purpose: this library targets B200 only.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace mrd {

// ------------------------------------------------------------------ misc
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile(
        "{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar)
        : "memory");
}

__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}

// Spin on an mbarrier phase.  A wait that lasts longer than ~4e9 SM cycles (seconds) means a
// protocol bug; trap instead of hanging the GPU so the host sees a launch failure.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}

// ------------------------------------------------------------------ fences / barriers
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tma_load_2d(const void* map, uint32_t bar, uint32_t dst, int c0,
                                            int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}

__device__ __forceinline__ void tma_load_3d(const void* map, uint32_t bar, uint32_t dst, int c0,
                                            int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

__device__ __forceinline__ void tma_load_4d(const void* map, uint32_t bar, uint32_t dst, int c0,
                                            int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

__device__ __forceinline__ void tma_load_5d(const void* map, uint32_t bar, uint32_t dst, int c0,
                                            int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
        "r"(c4)
        : "memory");
}

// L2 eviction-priority hints for TMA traffic: streaming operands (read once) should not push out a tile that is
// about to be re-read; a tile that WILL be re-read soon is stored with evict_last.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_load_4d_hint(const void* map, uint32_t bar, uint32_t dst, int c0, int c1,
                                                 int c2, int c3, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tma_store_4d_hint(const void* map, uint32_t src, int c0, int c1, int c2, int c3,
                                                  uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4, %5}], [%1], %6;" ::
            "l"(reinterpret_cast<uint64_t>(map)),
        "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(policy)
        : "memory");
}

// 8 bf16 maxima folded into global memory in one reduction (REDG.E.MAX.BF16x8)
__device__ __forceinline__ void red_max_bf16x8(void* gptr, uint4 v) {
    asm volatile("red.global.v4.bf16x2.max.noftz [%0], {%1, %2, %3, %4};" ::"l"(gptr), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// L2 prefetch of a tensor box (no shared-memory destination, no barrier): used by producers that
// hold only a few large stages to pull the tiles they will need next from HBM into L2.
__device__ __forceinline__ void tma_prefetch_2d(const void* map, int c0, int c1) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::
                     "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_prefetch_5d(const void* map, int c0, int c1, int c2, int c3,
                                                int c4) {
    asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global.tile [%0, {%1, %2, %3, %4, %5}];" ::
                     "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}

__device__ __forceinline__ void tma_store_4d(const void* map, uint32_t src, int c0, int c1,
                                             int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::
            "l"(reinterpret_cast<uint64_t>(map)),
        "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

__device__ __forceinline__ void tma_store_commit() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------ tcgen05 / TMEM
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_result_addr),
                 "n"(NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS)
                 : "memory");
}

// cta_group::2: TMEM columns in BOTH CTAs of a pair (one warp of each CTA executes these)
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_result_addr) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr),
                 "n"(NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// One 256 x N x 16 product over the CTA pair, issued by ONE thread of the leader CTA: each CTA's shared memory holds
// 128 rows of A and N/2 rows of B at the offsets the descriptors name, each CTA's TMEM gets its 128 accumulator rows
// (verified by tools/exp_cta_pair.cu).
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the mbarrier at this offset in every CTA of cta_mask when the pair's MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"(cta_mask)
        : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> f32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// mbarrier arrive when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::
                     "r"(bar)
                 : "memory");
}

// 32 lanes x 32 columns of fp32: thread t of the warp gets lane (base_lane + t), 32 columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
          "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
          "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 32 lanes x 32 columns of fp32 back into TMEM (same lane / column mapping as tmem_ld32)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
        "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
        "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ------------------------------------------------------------------ thread-block clusters / distributed shared memory
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {   // every thread of every CTA of the cluster
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> the same offset in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
// TMA load delivered to the same shared-memory offset (and counted on the same mbarrier offset) of every CTA of the
// cluster whose bit is set in cta_mask
__device__ __forceinline__ void tma_load_2d_multicast(const void* map, uint32_t bar, uint32_t dst, int c0, int c1,
                                                      uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "h"(cta_mask)
        : "memory");
}
// tcgen05.commit that arrives on the mbarrier at this offset in every CTA of cta_mask
__device__ __forceinline__ void umma_commit_multicast(uint32_t bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"(cta_mask)
        : "memory");
}
// arrive on an mbarrier of another CTA of the cluster (address from mapa_shared) with the default (CTA-scope release)
// ordering: for barriers that only pace hardware-tracked work - a TMA landing, accumulator columns drained with
// tcgen05.ld - and publish no data written by ordinary stores.  (A cluster-scope release costs the arriving thread on
// the order of a thousand cycles per call.)
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}

// ------------------------------------------------------------------ descriptors
// Shared-memory matrix descriptor (sm_100 "version 1").  layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= 1ull << 46;  // descriptor version for Blackwell
    d |= static_cast<uint64_t>(layout & 7) << 61;
    return d;
}

// Instruction descriptor for kind::f16 with bf16 inputs and fp32 accumulation.
// a_mn / b_mn: 0 = K-major operand, 1 = MN-major operand.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) |
           (static_cast<uint32_t>(b_mn) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}

// ------------------------------------------------------------------ small math helpers
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t u) {
    __nv_bfloat162 t = *reinterpret_cast<__nv_bfloat162*>(&u);
    return __bfloat1622float2(t);
}
__device__ __forceinline__ float gelu_erf(float x) {
    return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f));
}
// Exact-erf GELU (HF:activations.py:70-90) with erf from Abramowitz & Stegun 7.1.26
// (|error| <= 1.5e-7, far below the bf16 rounding of the result), written against the raw fast-math
// units: one MUFU.RCP, one MUFU.EX2 and 11 FP32 issue slots per element, so the FFN1 epilogue keeps pace with the
// tensor core (erff(), or __fdividef/__expf with their range fix-ups, cost 2-3x as many).
//   z = |x|/sqrt(2), t = 1/(1 + p z), h = 0.5 (a1 t + ... + a5 t^5) exp(-z^2) = 0.5 erfc(z)
//   gelu(x) = x (x >= 0 ? 1 - h : h) = max(x, 0) - |x| h
// with w = |x| sqrt(log2(e)/2): exp(-z^2) = 2^(-w^2) and p z = (p sqrt(2/log2(e)) / sqrt(2)) w, so |x| is scaled once.
__device__ __forceinline__ float gelu_erf_fast(float x) {
    float t, e;
    const float ax = fabsf(x);
    const float w = ax * 0.84932180028801904f;                 // sqrt(0.5 * log2(e))
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.27273748f, w, 1.0f)));   // p / sqrt(log2(e))
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(w * -w));
    float poly = fmaf(0.5f * 1.061405429f, t, 0.5f * -1.453152027f);
    poly = fmaf(poly, t, 0.5f * 1.421413741f);
    poly = fmaf(poly, t, 0.5f * -0.284496736f);
    poly = fmaf(poly, t, 0.5f * 0.254829592f);
    const float h = poly * t * e;
    return fmaf(-ax, h, fmaxf(x, 0.0f));
}

}  // namespace mrd
