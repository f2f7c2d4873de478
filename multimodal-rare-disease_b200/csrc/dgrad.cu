// Non-GEMM kernels of the backbone's data-gradient backward (see dgrad.h).

#include "dgrad.h"

#include <math.h>
#include <stdint.h>

#include <mrd_b200.h>

#include "ptx.cuh"
#include "tma_host.h"

namespace mrd {

namespace {

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("%s launch: %s", what, cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}

inline unsigned blocks_for(long long n, int per_block) {
    return static_cast<unsigned>((n + per_block - 1) / per_block);
}

__global__ void pack_dgrad_weights_kernel(const __nv_bfloat16* __restrict__ w, int Cout, int Cin, int kk, TapList src,
                                          __nv_bfloat16* __restrict__ out) {
    const long long total = static_cast<long long>(Cin) * src.n * Cout;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int co = static_cast<int>(i % Cout);
    const long long r = i / Cout;
    const int t = static_cast<int>(r % src.n);
    const int ci = static_cast<int>(r / src.n);
    out[i] = w[(static_cast<long long>(co) * kk + src.tap[t]) * Cin + ci];
}

__global__ void relu_mask_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y, long long n8,
                                 uint4* __restrict__ gz) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n8) return;
    uint4 gv = __ldg(g + i);
    const uint4 yv = __ldg(y + i);
    const uint32_t* yw = reinterpret_cast<const uint32_t*>(&yv);
    uint32_t* gw = reinterpret_cast<uint32_t*>(&gv);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 yf = unpack_bf16(yw[k]);
        // a bf16 is > 0 iff its sign bit is clear and it is not +0 (no NaN in a ReLU output)
        const uint32_t keep = (yf.x > 0.0f ? 0x0000ffffu : 0u) | (yf.y > 0.0f ? 0xffff0000u : 0u);
        gw[k] &= keep;
    }
    gz[i] = gv;
}

__global__ void avgpool_bwd_mask_kernel(const float* __restrict__ dp, int HW, int C8, float inv_hw,
                                        const uint4* __restrict__ y, long long total, uint4* __restrict__ gz) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c8 = static_cast<int>(i % C8);
    const long long n = i / C8 / HW;
    const float4 a = __ldg(reinterpret_cast<const float4*>(dp + (n * C8 + c8) * 8));
    const float4 b = __ldg(reinterpret_cast<const float4*>(dp + (n * C8 + c8) * 8 + 4));
    const float gv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    const uint4 yv = __ldg(y + i);
    const uint32_t* yw = reinterpret_cast<const uint32_t*>(&yv);
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 yf = unpack_bf16(yw[k]);
        o[k] = pack_bf16(yf.x > 0.0f ? gv[2 * k] * inv_hw : 0.0f, yf.y > 0.0f ? gv[2 * k + 1] * inv_hw : 0.0f);
    }
    gz[i] = make_uint4(o[0], o[1], o[2], o[3]);
}

// one thread = one input pixel x 8 channels; the (at most 2 x 2) windows containing it are re-evaluated
__global__ void maxpool_bwd_relu_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y, int N, int H, int W,
                                        int C8, uint4* __restrict__ dx) {
    const int Hp = H / 2, Wp = W / 2;
    const long long total = static_cast<long long>(N) * H * W * C8;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = static_cast<int>(i % C8);
    long long r = i / C8;
    const int x = static_cast<int>(r % W);
    r /= W;
    const int yy = static_cast<int>(r % H);
    const int n = static_cast<int>(r / H);
    const uint4* yimg = y + static_cast<long long>(n) * H * W * C8;
    const uint4 self = __ldg(yimg + (static_cast<long long>(yy) * W + x) * C8 + c);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int py0 = yy >> 1, py1 = (yy + 1) >> 1;   // windows 2p-1 .. 2p+1 that contain row yy
    const int px0 = x >> 1, px1 = (x + 1) >> 1;
    for (int py = py0; py <= py1 && py < Hp; ++py) {
        for (int px = px0; px <= px1 && px < Wp; ++px) {
            float best[8];
            int arg[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { best[j] = -INFINITY; arg[j] = -1; }
            for (int dh = -1; dh <= 1; ++dh) {
                const int h = 2 * py + dh;
                if (h < 0 || h >= H) continue;
                for (int dw = -1; dw <= 1; ++dw) {
                    const int w = 2 * px + dw;
                    if (w < 0 || w >= W) continue;
                    const uint4 v = __ldg(yimg + (static_cast<long long>(h) * W + w) * C8 + c);
                    const uint32_t* vw = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float2 f = unpack_bf16(vw[k]);
                        if (f.x > best[2 * k]) { best[2 * k] = f.x; arg[2 * k] = h * W + w; }
                        if (f.y > best[2 * k + 1]) { best[2 * k + 1] = f.y; arg[2 * k + 1] = h * W + w; }
                    }
                }
            }
            const int me = yy * W + x;
            bool any = false;
#pragma unroll
            for (int j = 0; j < 8; ++j) any |= arg[j] == me;
            if (!any) continue;
            const uint4 gv = __ldg(g + ((static_cast<long long>(n) * Hp + py) * Wp + px) * C8 + c);
            const uint32_t* gw = reinterpret_cast<const uint32_t*>(&gv);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 f = unpack_bf16(gw[k]);
                if (arg[2 * k] == me) acc[2 * k] += f.x;
                if (arg[2 * k + 1] == me) acc[2 * k + 1] += f.y;
            }
        }
    }
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(&self);
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 f = unpack_bf16(sw[k]);
        o[k] = pack_bf16(f.x > 0.0f ? acc[2 * k] : 0.0f, f.y > 0.0f ? acc[2 * k + 1] : 0.0f);
    }
    dx[i] = make_uint4(o[0], o[1], o[2], o[3]);
}

__global__ void pack_stem_dgrad_kernel(const float* __restrict__ w, const float* __restrict__ gamma,
                                       const float* __restrict__ var, float eps, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;   // [kh][kw][co][c]
    if (i >= 7 * 7 * 64 * 3) return;
    const int c = i % 3, co = (i / 3) % 64, kw = (i / 192) % 7, kh = i / (192 * 7);
    out[i] = w[((co * 3 + c) * 7 + kh) * 7 + kw] * (gamma[co] / sqrtf(var[co] + eps));
}

constexpr int kStemRowsPerBlock = 4;

// block = kStemRowsPerBlock image rows of one image; the folded filter (37.6 KB) sits in shared memory.  Thread t of a
// row takes column 2t (first half of the row's threads) or 2t+1: threads of one parity share their tap set.
__global__ void __launch_bounds__(256) stem_dgrad_kernel(const __nv_bfloat16* __restrict__ d,
                                                         const float* __restrict__ wf, int H, int W,
                                                         float* __restrict__ out) {
    __shared__ float ws[7 * 7 * 64 * 3];
    for (int i = threadIdx.x; i < 7 * 7 * 64 * 3; i += blockDim.x) ws[i] = __ldg(wf + i);
    __syncthreads();
    const int Ho = H / 2, Wo = W / 2;
    const int n = blockIdx.y;
    const uint4* dimg = reinterpret_cast<const uint4*>(d) + static_cast<long long>(n) * Ho * Wo * 8;
    const int half = W / 2;
    for (int item = threadIdx.x; item < kStemRowsPerBlock * W; item += blockDim.x) {
        const int ih = blockIdx.x * kStemRowsPerBlock + item / W;
        if (ih >= H) break;
        const int t = item % W;
        const int iw = t < half ? 2 * t : 2 * (t - half) + 1;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        for (int kh = (ih + 3) & 1; kh < 7; kh += 2) {   // ih = 2*oh + kh - 3
            const int oh = (ih + 3 - kh) >> 1;
            if (oh < 0 || oh >= Ho) continue;
            for (int kw = (iw + 3) & 1; kw < 7; kw += 2) {
                const int ow = (iw + 3 - kw) >> 1;
                if (ow < 0 || ow >= Wo) continue;
                const uint4* dp = dimg + (static_cast<long long>(oh) * Wo + ow) * 8;
                const float* wp = ws + (kh * 7 + kw) * 192;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const uint4 v = __ldg(dp + q);
                    const uint32_t* vw = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float2 f = unpack_bf16(vw[k]);
                        const float* w0 = wp + (q * 8 + 2 * k) * 3;
                        a0 = fmaf(f.x, w0[0], a0); a1 = fmaf(f.x, w0[1], a1); a2 = fmaf(f.x, w0[2], a2);
                        a0 = fmaf(f.y, w0[3], a0); a1 = fmaf(f.y, w0[4], a1); a2 = fmaf(f.y, w0[5], a2);
                    }
                }
            }
        }
        float* o = out + static_cast<long long>(n) * 3 * H * W + static_cast<long long>(ih) * W + iw;
        o[0] = a0;
        o[static_cast<long long>(H) * W] = a1;
        o[2LL * H * W] = a2;
    }
}

}  // namespace

int pack_dgrad_weights(const __nv_bfloat16* w, int Cout, int Cin, int kk, TapList src, __nv_bfloat16* out,
                       cudaStream_t s) {
    if ((kk != 1 && kk != 9) || src.n < 1 || src.n > 9) {
        set_last_error("pack_dgrad_weights: kk=%d taps=%d", kk, src.n);
        return -1;
    }
    for (int t = 0; t < src.n; ++t)
        if (src.tap[t] < 0 || src.tap[t] >= kk) {
            set_last_error("pack_dgrad_weights: tap %d outside the filter", src.tap[t]);
            return -1;
        }
    const long long total = static_cast<long long>(Cin) * src.n * Cout;
    pack_dgrad_weights_kernel<<<blocks_for(total, 256), 256, 0, s>>>(w, Cout, Cin, kk, src, out);
    return check_launch("pack_dgrad_weights");
}

int relu_mask_bf16(const __nv_bfloat16* g, const __nv_bfloat16* y, long long n, __nv_bfloat16* gz, cudaStream_t s) {
    if (n % 8 != 0) {
        set_last_error("relu_mask_bf16: n %% 8 != 0 (n=%lld)", n);
        return -1;
    }
    if (n == 0) return 0;
    relu_mask_kernel<<<blocks_for(n / 8, 256), 256, 0, s>>>(reinterpret_cast<const uint4*>(g),
                                                            reinterpret_cast<const uint4*>(y), n / 8,
                                                            reinterpret_cast<uint4*>(gz));
    return check_launch("relu_mask_bf16");
}

int avgpool_bwd_mask_bf16(const float* d_pooled, int N, int HW, int C, const __nv_bfloat16* y, __nv_bfloat16* gz,
                          cudaStream_t s) {
    if (C % 8 != 0 || HW <= 0) {
        set_last_error("avgpool_bwd_mask_bf16: C %% 8 != 0 or HW <= 0 (C=%d HW=%d)", C, HW);
        return -1;
    }
    const long long total = static_cast<long long>(N) * HW * (C / 8);
    if (total == 0) return 0;
    avgpool_bwd_mask_kernel<<<blocks_for(total, 256), 256, 0, s>>>(d_pooled, HW, C / 8, 1.0f / HW,
                                                                   reinterpret_cast<const uint4*>(y), total,
                                                                   reinterpret_cast<uint4*>(gz));
    return check_launch("avgpool_bwd_mask_bf16");
}

int maxpool3x3s2_bwd_relu(const __nv_bfloat16* g, const __nv_bfloat16* y, int N, int H, int W, int C,
                          __nv_bfloat16* dx, cudaStream_t s) {
    if (C % 8 != 0 || H % 2 != 0 || W % 2 != 0) {
        set_last_error("maxpool3x3s2_bwd_relu: need C %% 8 == 0 and even H, W (C=%d H=%d W=%d)", C, H, W);
        return -1;
    }
    const long long total = static_cast<long long>(N) * H * W * (C / 8);
    if (total == 0) return 0;
    maxpool_bwd_relu_kernel<<<blocks_for(total, 256), 256, 0, s>>>(reinterpret_cast<const uint4*>(g),
                                                                   reinterpret_cast<const uint4*>(y), N, H, W, C / 8,
                                                                   reinterpret_cast<uint4*>(dx));
    return check_launch("maxpool3x3s2_bwd_relu");
}

int pack_stem_dgrad(const float* w, const float* gamma, const float* var, float eps, float* out, cudaStream_t s) {
    pack_stem_dgrad_kernel<<<blocks_for(7 * 7 * 64 * 3, 256), 256, 0, s>>>(w, gamma, var, eps, out);
    return check_launch("pack_stem_dgrad");
}

int stem_dgrad_nchw(const __nv_bfloat16* d, const float* wf, int N, int H, int W, float* out, cudaStream_t s) {
    if (H % 2 != 0 || W % 2 != 0 || N > 65535) {
        set_last_error("stem_dgrad_nchw: need even H, W and N <= 65535 (N=%d H=%d W=%d)", N, H, W);
        return -1;
    }
    if (N == 0) return 0;
    const dim3 grid((H + kStemRowsPerBlock - 1) / kStemRowsPerBlock, N);
    stem_dgrad_kernel<<<grid, 256, 0, s>>>(d, wf, H, W, out);
    return check_launch("stem_dgrad_nchw");
}

}  // namespace mrd
