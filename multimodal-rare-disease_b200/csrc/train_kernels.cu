// Non-contraction kernels of the training step (see train_kernels.h).

#include "train_kernels.h"

#include <math.h>
#include <stdint.h>

#include <mrd_b200.h>

#include "ptx.cuh"
#include "tma_host.h"

namespace mrd {

namespace {

typedef __nv_bfloat16 bf16;

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_last_error("%s launch: %s", what, cudaGetErrorString(e));
        return -static_cast<int>(e);
    }
    return 0;
}
inline unsigned nblk(long long n, int per) { return static_cast<unsigned>((n + per - 1) / per); }

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
    float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y;
    f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint4 u;
    u.x = pack_bf16(f[0], f[1]);
    u.y = pack_bf16(f[2], f[3]);
    u.z = pack_bf16(f[4], f[5]);
    u.w = pack_bf16(f[6], f[7]);
    return u;
}
// values as the stored bf16 would read back
__device__ __forceinline__ void round8(float (&f)[8]) {
    const uint4 u = pack8(f);
    unpack8(u, f);
}

// ------------------------------------------------------------------ dropout
__global__ void dropout_bf16_kernel(const bf16* __restrict__ x, long long ldx, int rows, int width,
                                    const int* __restrict__ dyn_rows, DropCfg d, bf16* __restrict__ y,
                                    long long ldy) {
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    const int w8 = width >> 3;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(rows) * w8) return;
    const long long r = i / w8;
    const int c = static_cast<int>(i - r * w8) * 8;
    float v[8];
    unpack8(*reinterpret_cast<const uint4*>(x + r * ldx + c), v);
    const unsigned long long base = static_cast<unsigned long long>(r) * width + c;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = drop_keep(d, base + j) ? v[j] * d.scale : 0.0f;
    *reinterpret_cast<uint4*>(y + r * ldy + c) = pack8(v);
}

__global__ void dropout_f32_kernel(const float* __restrict__ x, long long n, DropCfg d, float* __restrict__ y) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    y[i] = drop_keep(d, static_cast<unsigned long long>(i)) ? x[i] * d.scale : 0.0f;
}

__global__ void relu_dropout_f32_kernel(const float* __restrict__ x, long long n, DropCfg d, float* __restrict__ y) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    y[i] = drop_keep(d, static_cast<unsigned long long>(i)) ? fmaxf(x[i], 0.0f) * d.scale : 0.0f;
}

__global__ void head_dropout_f32_kernel(const float* __restrict__ x, int rows, int heads, int hd, DropCfg d,
                                        float* __restrict__ y, float* __restrict__ w_out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long n = static_cast<long long>(rows) * heads * hd;
    if (i >= n) return;
    const long long rh = i / hd;  // r*heads + h
    const float w = drop_keep(d, static_cast<unsigned long long>(rh)) ? d.scale : 0.0f;
    y[i] = x[i] * w;
    if (w_out && i % hd == 0) w_out[rh] = w;
}

__global__ void dropout_mask_kernel(DropCfg d, long long n, float* __restrict__ out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = drop_keep(d, static_cast<unsigned long long>(i)) ? 1.0f : 0.0f;
}

// ------------------------------------------------------------------ LayerNorm forward (train)
template <int NCH>
__global__ void __launch_bounds__(256)
drop_add_ln_kernel(const bf16* __restrict__ z, const bf16* __restrict__ res, int rows,
                   const int* __restrict__ dyn_rows, DropCfg d, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float eps, bf16* __restrict__ s_out, bf16* __restrict__ y) {
    constexpr int WIDTH = NCH * 256;
    const int lane = threadIdx.x & 31;
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    if (row >= rows) return;
    float v[NCH][8];
    float sum = 0.0f;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const int col = (c * 32 + lane) * 8;
        float zz[8], rr[8];
        unpack8(*reinterpret_cast<const uint4*>(z + row * WIDTH + col), zz);
        unpack8(*reinterpret_cast<const uint4*>(res + row * WIDTH + col), rr);
        const unsigned long long base = static_cast<unsigned long long>(row) * WIDTH + col;
#pragma unroll
        for (int j = 0; j < 8; ++j) v[c][j] = rr[j] + (drop_keep(d, base + j) ? zz[j] * d.scale : 0.0f);
        round8(v[c]);
        *reinterpret_cast<uint4*>(s_out + row * WIDTH + col) = pack8(v[c]);
#pragma unroll
        for (int j = 0; j < 8; ++j) sum += v[c][j];
    }
    const float mean = wsum(sum) * (1.0f / WIDTH);
    float sq = 0.0f;
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float t = v[c][j] - mean;
            sq += t * t;
        }
    const float rstd = rsqrtf(wsum(sq) * (1.0f / WIDTH) + eps);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const int col = (c * 32 + lane) * 8;
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = (v[c][j] - mean) * rstd * __ldg(gamma + col + j) + __ldg(beta + col + j);
        *reinterpret_cast<uint4*>(y + row * WIDTH + col) = pack8(o);
    }
}

// ------------------------------------------------------------------ LayerNorm backward
// One warp per row, rows strided over the grid; per-lane partial dgamma/dbeta live in registers and are
// reduced once per block through shared memory before the atomics.
template <int NCH>
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const bf16* __restrict__ s_in, const bf16* __restrict__ dy, const float* __restrict__ gamma,
              float eps, int rows, const int* __restrict__ dyn_rows, bf16* __restrict__ dx,
              float* __restrict__ dgamma, float* __restrict__ dbeta) {
    constexpr int WIDTH = NCH * 256;
    __shared__ float red[8][WIDTH];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    float ag[NCH][8], ab[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) ag[c][j] = ab[c][j] = 0.0f;
    for (long long row = static_cast<long long>(blockIdx.x) * 8 + warp; row < rows;
         row += static_cast<long long>(gridDim.x) * 8) {
        float x[NCH][8], g[NCH][8];
        float sum = 0.0f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int col = (c * 32 + lane) * 8;
            unpack8(*reinterpret_cast<const uint4*>(s_in + row * WIDTH + col), x[c]);
            unpack8(*reinterpret_cast<const uint4*>(dy + row * WIDTH + col), g[c]);
#pragma unroll
            for (int j = 0; j < 8; ++j) sum += x[c][j];
        }
        const float mean = wsum(sum) * (1.0f / WIDTH);
        float sq = 0.0f;
#pragma unroll
        for (int c = 0; c < NCH; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                x[c][j] -= mean;
                sq += x[c][j] * x[c][j];
            }
        const float rstd = rsqrtf(wsum(sq) * (1.0f / WIDTH) + eps);
        float m1 = 0.0f, m2 = 0.0f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int col = (c * 32 + lane) * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float xh = x[c][j] * rstd;
                x[c][j] = xh;
                ag[c][j] += g[c][j] * xh;
                ab[c][j] += g[c][j];
                const float gg = g[c][j] * __ldg(gamma + col + j);
                g[c][j] = gg;
                m1 += gg;
                m2 += gg * xh;
            }
        }
        m1 = wsum(m1) * (1.0f / WIDTH);
        m2 = wsum(m2) * (1.0f / WIDTH);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int col = (c * 32 + lane) * 8;
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = rstd * (g[c][j] - m1 - x[c][j] * m2);
            *reinterpret_cast<uint4*>(dx + row * WIDTH + col) = pack8(o);
        }
    }
    for (int pass = 0; pass < 2; ++pass) {
        float* dst = pass == 0 ? dgamma : dbeta;
        if (!dst) continue;  // uniform
        __syncthreads();
#pragma unroll
        for (int c = 0; c < NCH; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j) red[warp][(c * 32 + lane) * 8 + j] = pass == 0 ? ag[c][j] : ab[c][j];
        __syncthreads();
        for (int col = threadIdx.x; col < WIDTH; col += 256) {
            float t = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; ++w) t += red[w][col];
            atomicAdd(dst + col, t);
        }
    }
}

__global__ void ln_fwd_f32_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ g,
                                  const float* __restrict__ b, float eps, int rows, int width,
                                  float* __restrict__ y, long long ldy) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* xr = x + row * ldx;
    float s = 0.0f;
    for (int i = lane; i < width; i += 32) s += xr[i];
    const float mean = wsum(s) / width;
    float v = 0.0f;
    for (int i = lane; i < width; i += 32) {
        const float t = xr[i] - mean;
        v += t * t;
    }
    const float rstd = 1.0f / sqrtf(wsum(v) / width + eps);
    for (int i = lane; i < width; i += 32) y[row * ldy + i] = (xr[i] - mean) * rstd * g[i] + b[i];
}

// one warp per row; dgamma/dbeta through atomics (rows = batch size: a few hundred at most)
__global__ void ln_bwd_f32_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ dy,
                                  long long lddy, const float* __restrict__ g, float eps, int rows, int width,
                                  float* __restrict__ dx, long long lddx, float* __restrict__ dgamma,
                                  float* __restrict__ dbeta) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* xr = x + row * ldx;
    const float* dr = dy + row * lddy;
    float s = 0.0f;
    for (int i = lane; i < width; i += 32) s += xr[i];
    const float mean = wsum(s) / width;
    float v = 0.0f;
    for (int i = lane; i < width; i += 32) {
        const float t = xr[i] - mean;
        v += t * t;
    }
    const float rstd = 1.0f / sqrtf(wsum(v) / width + eps);
    float m1 = 0.0f, m2 = 0.0f;
    for (int i = lane; i < width; i += 32) {
        const float xh = (xr[i] - mean) * rstd, gg = dr[i] * g[i];
        m1 += gg;
        m2 += gg * xh;
    }
    m1 = wsum(m1) / width;
    m2 = wsum(m2) / width;
    for (int i = lane; i < width; i += 32) {
        const float xh = (xr[i] - mean) * rstd, gg = dr[i] * g[i];
        dx[row * lddx + i] = rstd * (gg - m1 - xh * m2);
        if (dgamma) atomicAdd(dgamma + i, dr[i] * xh);
        if (dbeta) atomicAdd(dbeta + i, dr[i]);
    }
}

// ------------------------------------------------------------------ GELU
__device__ __forceinline__ float gelu_f(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad_f(float v) {
    return 0.5f * (1.0f + erff(v * 0.70710678118654752f)) + v * 0.3989422804014327f * __expf(-0.5f * v * v);
}

template <bool BWD>
__global__ void gelu_kernel(const bf16* __restrict__ u, const bf16* __restrict__ dg, int rows, int width,
                            const int* __restrict__ dyn_rows, bf16* __restrict__ out) {
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    const long long n8 = static_cast<long long>(rows) * width / 8;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float a[8], o[8];
        unpack8(reinterpret_cast<const uint4*>(u)[i], a);
        if (BWD) {
            float g[8];
            unpack8(reinterpret_cast<const uint4*>(dg)[i], g);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = g[j] * gelu_grad_f(a[j]);
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = gelu_f(a[j]);
        }
        reinterpret_cast<uint4*>(out)[i] = pack8(o);
    }
}

// ------------------------------------------------------------------ transposes / reductions
// 64 rows x 64 columns per block.  Works on 32-bit words (bf16 pairs): a thread reads the same word of two
// adjacent rows, re-pairs them ([x(r,c) x(r,c+1)], [x(r+1,c) x(r+1,c+1)] -> [x(r,c) x(r+1,c)], [x(r,c+1)
// x(r+1,c+1)]) and the block transposes the words through a padded shared tile: every global access is a
// 128-byte warp row, every shared access conflict-free or 2-way.  blockIdx.z selects one of two operands
// so the dY^T and X^T of a weight gradient are staged by one launch.
struct TransposeJob {
    const bf16* x;
    long long ldx;
    int width;
    bf16* y;
    float* colsum;   // optional: colsum[c] += sum over the live rows of x[r][c] (bias gradient of a dY operand)
};

__global__ void __launch_bounds__(256)
transpose_pad_kernel(TransposeJob j0, TransposeJob j1, int rows, const int* __restrict__ dyn_rows, int Kp) {
    __shared__ uint32_t tile[64][33];
    __shared__ float csum[8][64];
    const TransposeJob job = blockIdx.z ? j1 : j0;
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    const int r0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
    if (c0 >= job.width) return;
    // the consumer (split-K GEMM with dyn_k) reads K blocks below round_up(live, 64) only
    if (dyn_rows && r0 >= ((rows + 63) & ~63)) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = c0 + 2 * lane;
    float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int rp = warp * 4 + i;          // row pair 0..31
        const int r = r0 + 2 * rp;
        uint32_t a = 0u, b = 0u;
        if (c < job.width) {
            if (r < rows) a = *reinterpret_cast<const uint32_t*>(job.x + r * job.ldx + c);
            if (r + 1 < rows) b = *reinterpret_cast<const uint32_t*>(job.x + (r + 1) * job.ldx + c);
        }
        tile[2 * lane][rp] = (a & 0xffffu) | (b << 16);
        tile[2 * lane + 1][rp] = (a >> 16) | (b & 0xffff0000u);
        s0 += __uint_as_float(a << 16) + __uint_as_float(b << 16);
        s1 += __uint_as_float(a & 0xffff0000u) + __uint_as_float(b & 0xffff0000u);
    }
    if (job.colsum) {
        csum[warp][2 * lane] = s0;
        csum[warp][2 * lane + 1] = s1;
    }
    __syncthreads();
    if (job.colsum && threadIdx.x < 64 && c0 + threadIdx.x < job.width) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += csum[w][threadIdx.x];
        atomicAdd(job.colsum + c0 + threadIdx.x, t);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int cc = warp * 8 + i;          // output row (= input column) within the tile
        const int r = r0 + 2 * lane;
        if (c0 + cc < job.width && r < Kp)
            *reinterpret_cast<uint32_t*>(job.y + static_cast<long long>(c0 + cc) * Kp + r) = tile[cc][lane];
    }
}

__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const bf16* __restrict__ x, long long ldx, int rows, int width,
                   const int* __restrict__ dyn_rows, float scale, float* __restrict__ out) {
    __shared__ float red[8][64];
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * 64 + lane * 2;
    float a0 = 0.0f, a1 = 0.0f;
    if (c < width) {
        for (long long r = static_cast<long long>(blockIdx.y) * 8 + warp; r < rows;
             r += static_cast<long long>(gridDim.y) * 8) {
            const float2 v = unpack_bf16(*reinterpret_cast<const uint32_t*>(x + r * ldx + c));
            a0 += v.x;
            a1 += v.y;
        }
    }
    red[warp][lane * 2] = a0;
    red[warp][lane * 2 + 1] = a1;
    __syncthreads();
    if (threadIdx.x < 64) {
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += red[w][threadIdx.x];
        const int cc = blockIdx.x * 64 + threadIdx.x;
        if (cc < width) atomicAdd(out + cc, t * scale);
    }
}

__global__ void colsum_f32_kernel(const float* __restrict__ x, long long ldx, int rows, int width,
                                  float* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= width) return;
    float a = 0.0f;
    for (int r = 0; r < rows; ++r) a += x[r * ldx + c];
    out[c] += a;
}

__global__ void scale_f32_kernel(float* __restrict__ x, long long n, float a) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) x[i] *= a;
}
__global__ void relu_bwd_f32_kernel(const float* __restrict__ y, const float* __restrict__ dy, long long n,
                                    float* __restrict__ dx) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) dx[i] = y[i] > 0.0f ? dy[i] : 0.0f;
}

__global__ void scatter_cls_kernel(const float* __restrict__ src, const int* __restrict__ seq_off, int B,
                                   int width, bf16* __restrict__ dst) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(B) * width) return;
    const int b = static_cast<int>(i / width), c = static_cast<int>(i % width);
    dst[static_cast<long long>(__ldg(seq_off + b)) * width + c] = __float2bfloat16(src[i]);
}
__global__ void gather_cls_f32_kernel(const bf16* __restrict__ x, const int* __restrict__ seq_off, int B,
                                      int width, float* __restrict__ y) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(B) * width) return;
    const int b = static_cast<int>(i / width), c = static_cast<int>(i % width);
    y[i] = __bfloat162float(x[static_cast<long long>(__ldg(seq_off + b)) * width + c]);
}

// ------------------------------------------------------------------ embeddings backward
__global__ void __launch_bounds__(256)
embed_ln_bwd_kernel(const long long* __restrict__ ids, const int* __restrict__ row_tok, int rows,
                    const int* __restrict__ dyn_rows, int S, const bf16* __restrict__ word,
                    const float* __restrict__ pos_type, const float* __restrict__ gamma, float eps, int vocab,
                    int pad_idx, const bf16* __restrict__ dy, float* __restrict__ dword,
                    float* __restrict__ dpos, float* __restrict__ dtype0, float* __restrict__ dgamma,
                    float* __restrict__ dbeta) {
    constexpr int WIDTH = 768, NCH = 3;
    __shared__ float red[8][WIDTH];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (dyn_rows) rows = min(rows, __ldg(dyn_rows));
    // column sums that every row feeds (LayerNorm weight / bias, token_type row 0): registers, one block
    // reduction and one atomic per column and block at the end
    float ag[NCH][8], ab[NCH][8], at[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) ag[c][j] = ab[c][j] = at[c][j] = 0.0f;
    for (long long row = static_cast<long long>(blockIdx.x) * 8 + warp; row < rows;
         row += static_cast<long long>(gridDim.x) * 8) {
        const long long tok = row_tok ? __ldg(row_tok + row) : row;
        long long id = __ldg(ids + tok);
        const bool live_word = id >= 0 && id < vocab && id != pad_idx;
        id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
        const int pos = static_cast<int>(tok % S);
        float x[NCH][8], g[NCH][8];
        float sum = 0.0f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int col = (c * 32 + lane) * 8;
            unpack8(__ldg(reinterpret_cast<const uint4*>(word + id * WIDTH + col)), x[c]);
            const float4 p0 = __ldg(reinterpret_cast<const float4*>(pos_type + pos * WIDTH + col));
            const float4 p1 = __ldg(reinterpret_cast<const float4*>(pos_type + pos * WIDTH + col + 4));
            x[c][0] += p0.x; x[c][1] += p0.y; x[c][2] += p0.z; x[c][3] += p0.w;
            x[c][4] += p1.x; x[c][5] += p1.y; x[c][6] += p1.z; x[c][7] += p1.w;
            unpack8(*reinterpret_cast<const uint4*>(dy + row * WIDTH + col), g[c]);
#pragma unroll
            for (int j = 0; j < 8; ++j) sum += x[c][j];
        }
        const float mean = wsum(sum) * (1.0f / WIDTH);
        float sq = 0.0f;
#pragma unroll
        for (int c = 0; c < NCH; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                x[c][j] -= mean;
                sq += x[c][j] * x[c][j];
            }
        const float rstd = rsqrtf(wsum(sq) * (1.0f / WIDTH) + eps);
        float m1 = 0.0f, m2 = 0.0f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int col = (c * 32 + lane) * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float xh = x[c][j] * rstd;
                x[c][j] = xh;
                ag[c][j] += g[c][j] * xh;
                ab[c][j] += g[c][j];
                const float gg = g[c][j] * __ldg(gamma + col + j);
                g[c][j] = gg;
                m1 += gg;
                m2 += gg * xh;
            }
        }
        m1 = wsum(m1) * (1.0f / WIDTH);
        m2 = wsum(m2) * (1.0f / WIDTH);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int col = (c * 32 + lane) * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float d = rstd * (g[c][j] - m1 - x[c][j] * m2);
                at[c][j] += d;
                if (dword && live_word) atomicAdd(dword + id * WIDTH + col + j, d);
                if (dpos) atomicAdd(dpos + static_cast<long long>(pos) * WIDTH + col + j, d);
            }
        }
    }
    for (int pass = 0; pass < 3; ++pass) {
        float* dst = pass == 0 ? dgamma : (pass == 1 ? dbeta : dtype0);
        if (!dst) continue;  // uniform
        __syncthreads();
#pragma unroll
        for (int c = 0; c < NCH; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j)
                red[warp][(c * 32 + lane) * 8 + j] = pass == 0 ? ag[c][j] : (pass == 1 ? ab[c][j] : at[c][j]);
        __syncthreads();
        for (int col = threadIdx.x; col < WIDTH; col += 256) {
            float t = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; ++w) t += red[w][col];
            atomicAdd(dst + col, t);
        }
    }
}

// ------------------------------------------------------------------ BatchNorm (batch statistics)
// The sums are taken about a per-channel shift k, the mean of the first (up to) 8 rows, so |mean - k| is of the
// order of the spread: var = E[(y-k)^2] - E[y-k]^2 does not cancel when |mean| >> std, as E[y^2] - mean^2 would.
// Every block derives the same k from the same 8 rows; the blocks of the first row slice store it.
__global__ void __launch_bounds__(256)
bn_stats_kernel(const bf16* __restrict__ y, long long rows, int C, float* __restrict__ sum,
                float* __restrict__ sumsq, float* __restrict__ shift) {
    __shared__ float red[2][8][64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x * 64 + lane * 2;
    float a0 = 0.0f, a1 = 0.0f, q0 = 0.0f, q1 = 0.0f;
    if (c < C) {
        const int nk = rows < 8 ? static_cast<int>(rows) : 8;
        float k0 = 0.0f, k1 = 0.0f;
#pragma unroll
        for (int r = 0; r < 8; ++r) {   // unrolled: the 8 loads are in flight together
            if (r < nk) {
                const float2 v = unpack_bf16(__ldg(reinterpret_cast<const uint32_t*>(y + static_cast<long long>(r) * C + c)));
                k0 += v.x; k1 += v.y;
            }
        }
        // rounded to bf16 like y, so that y - k is exact in fp32 across the channel's range
        const float2 k = unpack_bf16(pack_bf16(k0 / nk, k1 / nk));
        if (blockIdx.y == 0 && warp == 0) {
            shift[c] = k.x;
            shift[c + 1] = k.y;
        }
        for (long long r = static_cast<long long>(blockIdx.y) * 8 + warp; r < rows;
             r += static_cast<long long>(gridDim.y) * 8) {
            const float2 v = unpack_bf16(*reinterpret_cast<const uint32_t*>(y + r * C + c));
            const float d0 = v.x - k.x, d1 = v.y - k.y;
            a0 += d0; a1 += d1;
            q0 = fmaf(d0, d0, q0); q1 = fmaf(d1, d1, q1);
        }
    }
    red[0][warp][lane * 2] = a0; red[0][warp][lane * 2 + 1] = a1;
    red[1][warp][lane * 2] = q0; red[1][warp][lane * 2 + 1] = q1;
    __syncthreads();
    if (threadIdx.x < 128) {
        const int which = threadIdx.x >> 6, col = threadIdx.x & 63;
        float t = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += red[which][w][col];
        const int cc = blockIdx.x * 64 + col;
        if (cc < C) atomicAdd((which ? sumsq : sum) + cc, t);
    }
}

// scale / shift of all C channels are derived once per block into shared memory (2*C floats), then applied
__global__ void bn_apply_stats_kernel(bf16* __restrict__ y, long long n8, int C, const float* __restrict__ sum,
                                      const float* __restrict__ sumsq, const float* __restrict__ shift, float inv_n,
                                      const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                      const bf16* __restrict__ identity, int relu) {
    extern __shared__ float ss[];   // [C] scale, [C] shift
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float md = __ldg(sum + c) * inv_n;   // mean - shift
        const float var = fmaxf(__ldg(sumsq + c) * inv_n - md * md, 0.0f);
        const float sc = __ldg(gamma + c) * rsqrtf(var + eps);
        ss[c] = sc;
        ss[C + c] = __ldg(beta + c) - (__ldg(shift + c) + md) * sc;
    }
    __syncthreads();
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n8;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>((i * 8) % C);
        float v[8];
        unpack8(reinterpret_cast<const uint4*>(y)[i], v);
        const float4 s0 = *reinterpret_cast<const float4*>(ss + c), s1 = *reinterpret_cast<const float4*>(ss + c + 4);
        const float4 h0 = *reinterpret_cast<const float4*>(ss + C + c), h1 = *reinterpret_cast<const float4*>(ss + C + c + 4);
        v[0] = fmaf(v[0], s0.x, h0.x); v[1] = fmaf(v[1], s0.y, h0.y); v[2] = fmaf(v[2], s0.z, h0.z); v[3] = fmaf(v[3], s0.w, h0.w);
        v[4] = fmaf(v[4], s1.x, h1.x); v[5] = fmaf(v[5], s1.y, h1.y); v[6] = fmaf(v[6], s1.z, h1.z); v[7] = fmaf(v[7], s1.w, h1.w);
        if (identity) {
            float r[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(identity) + i), r);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] += r[j];
        }
        if (relu) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.0f);
        }
        reinterpret_cast<uint4*>(y)[i] = pack8(v);
    }
}

__global__ void bn_update_running_kernel(const BnSite* __restrict__ table, float momentum) {
    const BnSite st = table[blockIdx.y];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= st.C) return;
    const float md = st.sum[c] / st.n;   // mean - shift
    const float mean = st.shift[c] + md;
    const float var = fmaxf(st.sumsq[c] / st.n - md * md, 0.0f);
    st.running_mean[c] = (1.0f - momentum) * st.running_mean[c] + momentum * mean;
    st.running_var[c] = (1.0f - momentum) * st.running_var[c] + momentum * var * (st.n / fmaxf(st.n - 1.0f, 1.0f));
}

}  // namespace

// ====================================================================== host wrappers
int dropout_bf16(const bf16* x, long long ldx, int rows, int width, const int* dyn_rows, DropCfg d, bf16* y,
                 long long ldy, cudaStream_t s) {
    if (rows <= 0) return 0;
    if (width % 8) {
        set_last_error("dropout_bf16: width %% 8 != 0");
        return -1;
    }
    dropout_bf16_kernel<<<nblk(static_cast<long long>(rows) * (width / 8), 256), 256, 0, s>>>(x, ldx, rows, width,
                                                                                          dyn_rows, d, y, ldy);
    return check_launch("dropout_bf16");
}
int dropout_f32(const float* x, int rows, int width, DropCfg d, float* y, cudaStream_t s) {
    const long long n = static_cast<long long>(rows) * width;
    if (n <= 0) return 0;
    dropout_f32_kernel<<<nblk(n, 256), 256, 0, s>>>(x, n, d, y);
    return check_launch("dropout_f32");
}
int relu_dropout_f32(const float* x, int rows, int width, DropCfg d, float* y, cudaStream_t s) {
    const long long n = static_cast<long long>(rows) * width;
    if (n <= 0) return 0;
    relu_dropout_f32_kernel<<<nblk(n, 256), 256, 0, s>>>(x, n, d, y);
    return check_launch("relu_dropout_f32");
}
int head_dropout_f32(const float* x, int rows, int heads, int head_dim, DropCfg d, float* y, float* w_out,
                     cudaStream_t s) {
    const long long n = static_cast<long long>(rows) * heads * head_dim;
    if (n <= 0) return 0;
    head_dropout_f32_kernel<<<nblk(n, 256), 256, 0, s>>>(x, rows, heads, head_dim, d, y, w_out);
    return check_launch("head_dropout_f32");
}
int dropout_mask_f32(DropCfg d, long long n, float* out, cudaStream_t s) {
    if (n <= 0) return 0;
    dropout_mask_kernel<<<nblk(n, 256), 256, 0, s>>>(d, n, out);
    return check_launch("dropout_mask_f32");
}

int drop_add_ln_fwd(const bf16* z, const bf16* res, int rows, int width, const int* dyn_rows, DropCfg d,
                    const float* gamma, const float* beta, float eps, bf16* s_out, bf16* y, cudaStream_t s) {
    if (rows <= 0) return 0;
    const unsigned grid = nblk(rows, 8);
#define MRD_K(NC) drop_add_ln_kernel<NC><<<grid, 256, 0, s>>>(z, res, rows, dyn_rows, d, gamma, beta, eps, s_out, y)
    switch (width) {
        case 256: MRD_K(1); break;
        case 512: MRD_K(2); break;
        case 768: MRD_K(3); break;
        case 1024: MRD_K(4); break;
        default:
            set_last_error("drop_add_ln_fwd: unsupported width %d", width);
            return -1;
    }
#undef MRD_K
    return check_launch("drop_add_ln_fwd");
}

int ln_bwd_bf16(const bf16* s_in, const bf16* dy, const float* gamma, float eps, int rows, int width,
                const int* dyn_rows, bf16* dx, float* dgamma, float* dbeta, cudaStream_t s) {
    if (rows <= 0) return 0;
    unsigned grid = nblk(rows, 8);
    if (grid > 148u * 2u) grid = 148u * 2u;
#define MRD_K(NC) ln_bwd_kernel<NC><<<grid, 256, 0, s>>>(s_in, dy, gamma, eps, rows, dyn_rows, dx, dgamma, dbeta)
    switch (width) {
        case 256: MRD_K(1); break;
        case 512: MRD_K(2); break;
        case 768: MRD_K(3); break;
        case 1024: MRD_K(4); break;
        default:
            set_last_error("ln_bwd_bf16: unsupported width %d", width);
            return -1;
    }
#undef MRD_K
    return check_launch("ln_bwd_bf16");
}

int ln_fwd_f32(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int rows,
               int width, float* y, long long ldy, cudaStream_t s) {
    if (rows <= 0) return 0;
    ln_fwd_f32_kernel<<<nblk(rows, 8), 256, 0, s>>>(x, ldx, gamma, beta, eps, rows, width, y, ldy);
    return check_launch("ln_fwd_f32");
}
int ln_bwd_f32(const float* x, long long ldx, const float* dy, long long lddy, const float* gamma, float eps,
               int rows, int width, float* dx, long long lddx, float* dgamma, float* dbeta, cudaStream_t s) {
    if (rows <= 0) return 0;
    ln_bwd_f32_kernel<<<nblk(rows, 8), 256, 0, s>>>(x, ldx, dy, lddy, gamma, eps, rows, width, dx, lddx,
                                                    dgamma, dbeta);
    return check_launch("ln_bwd_f32");
}

int gelu_fwd_bf16(const bf16* u, int rows, int width, const int* dyn_rows, bf16* g, cudaStream_t s) {
    if (rows <= 0) return 0;
    unsigned grid = nblk(static_cast<long long>(rows) * width / 8, 256);
    if (grid > 148u * 16u) grid = 148u * 16u;
    gelu_kernel<false><<<grid, 256, 0, s>>>(u, nullptr, rows, width, dyn_rows, g);
    return check_launch("gelu_fwd_bf16");
}
int gelu_bwd_bf16(const bf16* u, const bf16* dg, int rows, int width, const int* dyn_rows, bf16* du,
                  cudaStream_t s) {
    if (rows <= 0) return 0;
    unsigned grid = nblk(static_cast<long long>(rows) * width / 8, 256);
    if (grid > 148u * 16u) grid = 148u * 16u;
    gelu_kernel<true><<<grid, 256, 0, s>>>(u, dg, rows, width, dyn_rows, du);
    return check_launch("gelu_bwd_bf16");
}

int transpose_pad2_bf16(const bf16* x0, long long ldx0, int width0, bf16* y0, const bf16* x1, long long ldx1,
                        int width1, bf16* y1, int rows, const int* dyn_rows, int Kp, cudaStream_t s,
                        float* colsum0) {
    if (Kp <= 0 || width0 <= 0) return 0;
    if (Kp % 2 || width0 % 2 || width1 % 2 || ldx0 % 2 || ldx1 % 2) {
        set_last_error("transpose_pad_bf16: odd extent");
        return -1;
    }
    const int wmax = width0 > width1 ? width0 : width1;
    dim3 grid((Kp + 63) / 64, (wmax + 63) / 64, x1 ? 2 : 1);
    TransposeJob j0{x0, ldx0, width0, y0, colsum0}, j1{x1, ldx1, width1, y1, nullptr};
    transpose_pad_kernel<<<grid, 256, 0, s>>>(j0, j1, rows, dyn_rows, Kp);
    return check_launch("transpose_pad_bf16");
}
int colsum_bf16(const bf16* x, long long ldx, int rows, int width, const int* dyn_rows, float scale, float* out,
                cudaStream_t s) {
    if (rows <= 0 || width <= 0) return 0;
    if (width % 2) {
        set_last_error("colsum_bf16: odd width");
        return -1;
    }
    int split = (rows + 255) / 256;
    if (split > 64) split = 64;
    if (split < 1) split = 1;
    dim3 grid((width + 63) / 64, split);
    colsum_bf16_kernel<<<grid, 256, 0, s>>>(x, ldx, rows, width, dyn_rows, scale, out);
    return check_launch("colsum_bf16");
}
int colsum_f32(const float* x, long long ldx, int rows, int width, float* out, cudaStream_t s) {
    if (rows <= 0 || width <= 0) return 0;
    colsum_f32_kernel<<<nblk(width, 128), 128, 0, s>>>(x, ldx, rows, width, out);
    return check_launch("colsum_f32");
}
int scale_f32(float* x, long long n, float a, cudaStream_t s) {
    if (n <= 0) return 0;
    scale_f32_kernel<<<nblk(n, 256), 256, 0, s>>>(x, n, a);
    return check_launch("scale_f32");
}
int relu_bwd_f32(const float* y, const float* dy, long long n, float* dx, cudaStream_t s) {
    if (n <= 0) return 0;
    relu_bwd_f32_kernel<<<nblk(n, 256), 256, 0, s>>>(y, dy, n, dx);
    return check_launch("relu_bwd_f32");
}
int scatter_cls_rows_bf16(const float* src, const int* seq_off, int B, int width, bf16* dst, cudaStream_t s) {
    if (B <= 0) return 0;
    scatter_cls_kernel<<<nblk(static_cast<long long>(B) * width, 256), 256, 0, s>>>(src, seq_off, B, width, dst);
    return check_launch("scatter_cls_rows_bf16");
}
int gather_cls_rows_f32(const bf16* x, const int* seq_off, int B, int width, float* y, cudaStream_t s) {
    if (B <= 0) return 0;
    gather_cls_f32_kernel<<<nblk(static_cast<long long>(B) * width, 256), 256, 0, s>>>(x, seq_off, B, width, y);
    return check_launch("gather_cls_rows_f32");
}

int embed_ln_bwd(const long long* ids, const int* row_tok, int rows, const int* dyn_rows, int S, const bf16* word,
                 const float* pos_type, const float* gamma, float eps, int vocab, int pad_idx, const bf16* dy,
                 float* dword, float* dpos, float* dtype0, float* dgamma, float* dbeta, cudaStream_t s) {
    if (rows <= 0) return 0;
    unsigned grid = nblk(rows, 8);
    if (grid > 148u) grid = 148u;
    embed_ln_bwd_kernel<<<grid, 256, 0, s>>>(ids, row_tok, rows, dyn_rows, S, word, pos_type, gamma, eps, vocab,
                                             pad_idx, dy, dword, dpos, dtype0, dgamma, dbeta);
    return check_launch("embed_ln_bwd");
}

int bn_stats_bf16(const bf16* y, long long rows, int C, float* sum, float* sumsq, float* shift, cudaStream_t s) {
    if (rows <= 0 || C <= 0) return 0;
    if (C % 2) {
        set_last_error("bn_stats_bf16: odd channel count");
        return -1;
    }
    long long split = (rows + 127) / 128;   // 16 rows per warp: short serial loops, more CTAs in flight
    if (split > 148 * 8) split = 148 * 8;
    if (split < 1) split = 1;
    dim3 grid((C + 63) / 64, static_cast<unsigned>(split));
    bn_stats_kernel<<<grid, 256, 0, s>>>(y, rows, C, sum, sumsq, shift);
    return check_launch("bn_stats_bf16");
}
int bn_apply_stats_bf16(bf16* y, long long rows, int C, const float* sum, const float* sumsq, const float* shift,
                        const float* gamma, const float* beta, float eps, const bf16* identity, int relu,
                        cudaStream_t s) {
    if (rows <= 0 || C <= 0) return 0;
    if (C % 8) {
        set_last_error("bn_apply_stats_bf16: C %% 8 != 0");
        return -1;
    }
    const long long n8 = rows * C / 8;
    if (C > 4096) {
        set_last_error("bn_apply_stats_bf16: C > 4096");
        return -1;
    }
    // every block first derives the C scale/shift pairs: keep the grid to a few blocks per SM
    unsigned grid = nblk(n8, 256 * 4);
    if (grid > 148u * 4u) grid = 148u * 4u;
    if (grid < 1u) grid = 1u;
    bn_apply_stats_kernel<<<grid, 256, 2 * C * sizeof(float), s>>>(y, n8, C, sum, sumsq, shift,
                                                                   1.0f / static_cast<float>(rows), gamma, beta, eps,
                                                                   identity, relu);
    return check_launch("bn_apply_stats_bf16");
}
int bn_update_running(const BnSite* table, int sites, int max_C, float momentum, cudaStream_t s) {
    if (sites <= 0) return 0;
    dim3 grid((max_C + 127) / 128, sites);
    bn_update_running_kernel<<<grid, 128, 0, s>>>(table, momentum);
    return check_launch("bn_update_running");
}

}  // namespace mrd
