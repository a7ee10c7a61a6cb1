// K5 / K6 and layout plumbing — the HBM-bound kernels around the tensor-core GEMMs and the recurrence.
//
//   pack_lstm_weights   fp32 nn.LSTM parameters -> bf16 operand layouts (row-permuted so that a CTA of the
//                       recurrent kernel owns all four gates of 32 units; transposed copies for BPTT / dX)
//   cast_transpose      fp32 [R,C] (optionally (t,n)-strided, optionally with a per-column affine = the
//                       BatchNorm apply) -> bf16 [R,C] and/or bf16 [C,R]; feeds every GEMM operand
//   bn_stats/finalize   training-mode BatchNorm1d statistics over T*N rows (model_ctc.py:29-32,136)
//   bn_bwd_reduce/apply BatchNorm backward
//   log_softmax fwd/bwd nn.LogSoftmax(dim=-1) (model_ctc.py:140,168)
//
// All are grid-stride / tiled streaming kernels: coalesced 128-byte rows, 32x33 shared-memory tiles
// for the transposes, grids sized in multiples of the SM count.
#include "common.cuh"
#include "ctcb200.h"

namespace ctcb200 {
namespace {

// part 0: the bf16 rounding of v; part 1: the bf16 rounding of what part 0 lost (split-operand "x3" mode)
__device__ __forceinline__ __nv_bfloat16 bf16_part(float v, int part) {
    const __nv_bfloat16 hi = __float2bfloat16(v);
    return part ? __float2bfloat16(v - __bfloat162float(hi)) : hi;
}
__device__ __forceinline__ __nv_bfloat162 bf16x2_part(float a, float b, int part) {
    __nv_bfloat162 r;
    r.x = bf16_part(a, part);
    r.y = bf16_part(b, part);
    return r;
}

__device__ __forceinline__ int packed_to_orig_row(int p, int H) {
    // packed gate row p = j*128 + ul*4 + q  ->  torch row q*H + 32 j + ul
    const int j = p >> 7, ul = (p & 127) >> 2, q = p & 3;
    return q * H + j * 32 + ul;
}

__global__ void pack_lstm_weights_kernel(const float* __restrict__ wih_f, const float* __restrict__ whh_f,
                                         const float* __restrict__ wih_r, const float* __restrict__ whh_r,
                                         __nv_bfloat16* __restrict__ wih_p, __nv_bfloat16* __restrict__ wihT_p,
                                         __nv_bfloat16* __restrict__ whh_p, __nv_bfloat16* __restrict__ whhT_p, int H,
                                         int I, int Ipad, int part, int gates) {
    // gates = rows / H of the torch weights: 4 (LSTM: i,f,g,o), 3 (GRU: r,z,n), 1 (vanilla RNN); the operand layouts always
    // have four gate slots per unit, slots >= gates are zero
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    const int G4 = 4 * H, G8 = 8 * H;
    // wih_p [8H, Ipad]
    for (long long e = tid; e < static_cast<long long>(G8) * Ipad; e += stride) {
        const int R = static_cast<int>(e / Ipad), i = static_cast<int>(e % Ipad);
        const int dir = R / G4, orow = packed_to_orig_row(R % G4, H);
        const float* w = dir ? wih_r : wih_f;
        wih_p[e] = bf16_part((i < I && orow < gates * H) ? w[static_cast<size_t>(orow) * I + i] : 0.0f, part);
    }
    // wihT_p [I, 8H]
    for (long long e = tid; e < static_cast<long long>(I) * G8; e += stride) {
        const int i = static_cast<int>(e / G8), R = static_cast<int>(e % G8);
        const int dir = R / G4, orow = packed_to_orig_row(R % G4, H);
        const float* w = dir ? wih_r : wih_f;
        wihT_p[e] = bf16_part(orow < gates * H ? w[static_cast<size_t>(orow) * I + i] : 0.0f, part);
    }
    // whh_p [8H, H]
    for (long long e = tid; e < static_cast<long long>(G8) * H; e += stride) {
        const int R = static_cast<int>(e / H), k = static_cast<int>(e % H);
        const int dir = R / G4, orow = packed_to_orig_row(R % G4, H);
        const float* w = dir ? whh_r : whh_f;
        whh_p[e] = bf16_part(orow < gates * H ? w[static_cast<size_t>(orow) * H + k] : 0.0f, part);
    }
    // whhT_p [(dir,q,m), k] = whh_dir[q*H + k][m]
    for (long long e = tid; e < static_cast<long long>(G8) * H; e += stride) {
        const int R = static_cast<int>(e / H), k = static_cast<int>(e % H);
        const int dir = R / G4, q = (R % G4) / H, m = R % H;
        const float* w = dir ? whh_r : whh_f;
        whhT_p[e] = bf16_part(q < gates ? w[(static_cast<size_t>(q) * H + k) * H + m] : 0.0f, part);
    }
}

// torch row of packed gate row p of a layer run at Hp >= H units (units >= H are zero padding), or -1 for a zero row
__device__ __forceinline__ int padded_src_row(int p, int H, int Hp, int gates) {
    const int orow = packed_to_orig_row(p, Hp), q = orow / Hp, u = orow % Hp;
    return (u < H && q < gates) ? q * H + u : -1;
}
// torch input column of device input column i: blocks of i_blk real columns spread i_blk_p apart (-1: zero padding)
__device__ __forceinline__ int padded_src_col(int i, int i_blk, int i_blk_p) {
    const int off = i % i_blk_p;
    return off < i_blk ? (i / i_blk_p) * i_blk + off : -1;
}

// The same operand layouts as pack_lstm_weights_kernel for a layer run at Hp = 128 * ceil(H / 128) units: the Hp - H extra units
// get zero rows in every matrix and zero columns in the recurrent ones, and the input columns are spread the way the layer below
// leaves its output (I_dev = (I / i_blk) * i_blk_p device columns). Those units then stay exactly zero (DESIGN.md §3.2).
__global__ void pack_lstm_weights_padded_kernel(const float* __restrict__ wih_f, const float* __restrict__ whh_f,
                                                const float* __restrict__ wih_r, const float* __restrict__ whh_r,
                                                __nv_bfloat16* __restrict__ wih_p, __nv_bfloat16* __restrict__ wihT_p,
                                                __nv_bfloat16* __restrict__ whh_p, __nv_bfloat16* __restrict__ whhT_p, int H,
                                                int Hp, int I, int i_blk, int i_blk_p, int I_dev, int Ipad, int part, int gates) {
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    const int G4 = 4 * Hp, G8 = 8 * Hp;
    // wih_p [8Hp, Ipad]
    for (long long e = tid; e < static_cast<long long>(G8) * Ipad; e += stride) {
        const int R = static_cast<int>(e / Ipad), i = static_cast<int>(e % Ipad);
        const int orow = padded_src_row(R % G4, H, Hp, gates), ic = i < I_dev ? padded_src_col(i, i_blk, i_blk_p) : -1;
        const float* w = R >= G4 ? wih_r : wih_f;
        wih_p[e] = bf16_part((orow >= 0 && ic >= 0) ? w[static_cast<size_t>(orow) * I + ic] : 0.0f, part);
    }
    // wihT_p [I_dev, 8Hp]
    for (long long e = tid; e < static_cast<long long>(I_dev) * G8; e += stride) {
        const int i = static_cast<int>(e / G8), R = static_cast<int>(e % G8);
        const int orow = padded_src_row(R % G4, H, Hp, gates), ic = padded_src_col(i, i_blk, i_blk_p);
        const float* w = R >= G4 ? wih_r : wih_f;
        wihT_p[e] = bf16_part((orow >= 0 && ic >= 0) ? w[static_cast<size_t>(orow) * I + ic] : 0.0f, part);
    }
    // whh_p [8Hp, Hp]
    for (long long e = tid; e < static_cast<long long>(G8) * Hp; e += stride) {
        const int R = static_cast<int>(e / Hp), k = static_cast<int>(e % Hp);
        const int orow = padded_src_row(R % G4, H, Hp, gates);
        const float* w = R >= G4 ? whh_r : whh_f;
        whh_p[e] = bf16_part((orow >= 0 && k < H) ? w[static_cast<size_t>(orow) * H + k] : 0.0f, part);
    }
    // whhT_p [(dir,q,m), k] = whh_dir[q*H + k][m]
    for (long long e = tid; e < static_cast<long long>(G8) * Hp; e += stride) {
        const int R = static_cast<int>(e / Hp), k = static_cast<int>(e % Hp);
        const int q = (R % G4) / Hp, m = R % Hp;
        const float* w = R >= G4 ? whh_r : whh_f;
        whhT_p[e] = bf16_part((q < gates && k < H && m < H) ? w[(static_cast<size_t>(q) * H + k) * H + m] : 0.0f, part);
    }
}

// src element (r, c) lives at src[(r / n_inner) * s_outer + (r % n_inner) * s_inner + c].
__global__ void __launch_bounds__(256)
cast_transpose_kernel(const float* __restrict__ src, long long s_outer, long long s_inner, int n_inner,
                      const float* __restrict__ scale, const float* __restrict__ shift,
                      __nv_bfloat16* __restrict__ dst, long long dst_pitch, __nv_bfloat16* __restrict__ dstT,
                      long long dstT_pitch, int n_pad, int R, int C, int part) {
    __shared__ float tile[32][33];
    const int tiles_c = (C + 31) / 32, tiles_r = (R + 31) / 32;
    const long long tiles = static_cast<long long>(tiles_c) * tiles_r;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    for (long long tile_id = blockIdx.x; tile_id < tiles; tile_id += gridDim.x) {
        const int r0 = static_cast<int>(tile_id / tiles_c) * 32, c0 = static_cast<int>(tile_id % tiles_c) * 32;
        const int c = c0 + tx;
        float sc = 1.0f, sh = 0.0f;
        if (scale && c < C) { sc = scale[c]; sh = shift[c]; }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = r0 + ty + 8 * k;
            float v = 0.0f;
            if (r < R && c < C) {
                v = src[static_cast<long long>(r / n_inner) * s_outer + static_cast<long long>(r % n_inner) * s_inner + c];
                v = v * sc + sh;
                if (dst) dst[static_cast<long long>(r) * dst_pitch + c] = bf16_part(v, part);
            }
            tile[ty + 8 * k][tx] = v;
        }
        if (dstT) {
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int cc = c0 + ty + 8 * k, rr = r0 + tx;
                // transposed column of row (t, n) is t * n_pad + n: the batch axis is padded so that a shift by
                // one time step stays 16-byte aligned for TMA
                if (cc < C && rr < R)
                    dstT[static_cast<long long>(cc) * dstT_pitch + static_cast<long long>(rr / n_inner) * n_pad + rr % n_inner] =
                        bf16_part(tile[tx][ty + 8 * k], part);
            }
            __syncthreads();
        }
    }
}

// Vectorised variant for even C and even strides: 64 x 64 tiles, float2 loads (256-byte rows), bf16x2 stores
// (128-byte rows) for both the straight and the transposed output.
__global__ void __launch_bounds__(256)
cast_transpose_v2_kernel(const float* __restrict__ src, long long s_outer, long long s_inner, int n_inner,
                         const float* __restrict__ scale, const float* __restrict__ shift,
                         __nv_bfloat16* __restrict__ dst, long long dst_pitch, __nv_bfloat16* __restrict__ dstT,
                         long long dstT_pitch, int n_pad, int R, int C, int part) {
    __shared__ __nv_bfloat16 tile[64][66];
    const int tiles_c = (C + 63) / 64, tiles_r = (R + 63) / 64;
    const long long tiles = static_cast<long long>(tiles_c) * tiles_r;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const bool fast_rows = (n_inner == n_pad) && (R % 2 == 0);
    for (long long tile_id = blockIdx.x; tile_id < tiles; tile_id += gridDim.x) {
        const int r0 = static_cast<int>(tile_id / tiles_c) * 64, c0 = static_cast<int>(tile_id % tiles_c) * 64;
        const int c = c0 + 2 * tx;
        float sc0 = 1.0f, sc1 = 1.0f, sh0 = 0.0f, sh1 = 0.0f;
        if (scale && c < C) { sc0 = scale[c]; sc1 = scale[c + 1]; sh0 = shift[c]; sh1 = shift[c + 1]; }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int r = r0 + ty + 8 * k;
            __nv_bfloat162 b = __floats2bfloat162_rn(0.0f, 0.0f);
            if (r < R && c < C) {
                const float2 v = *reinterpret_cast<const float2*>(
                    src + static_cast<long long>(r / n_inner) * s_outer + static_cast<long long>(r % n_inner) * s_inner + c);
                b = bf16x2_part(v.x * sc0 + sh0, v.y * sc1 + sh1, part);
                if (dst) *reinterpret_cast<__nv_bfloat162*>(dst + static_cast<long long>(r) * dst_pitch + c) = b;
            }
            tile[ty + 8 * k][2 * tx] = b.x;
            tile[ty + 8 * k][2 * tx + 1] = b.y;
        }
        if (dstT) {
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int cc = c0 + ty + 8 * k, rr = r0 + 2 * tx;
                if (cc < C) {
                    __nv_bfloat16* orow = dstT + static_cast<long long>(cc) * dstT_pitch;
                    if (fast_rows) {
                        if (rr < R) {
                            __nv_bfloat162 v;
                            v.x = tile[2 * tx][ty + 8 * k];
                            v.y = tile[2 * tx + 1][ty + 8 * k];
                            *reinterpret_cast<__nv_bfloat162*>(orow + rr) = v;
                        }
                    } else {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const int r = rr + h;
                            if (r < R) orow[static_cast<long long>(r / n_inner) * n_pad + r % n_inner] = tile[2 * tx + h][ty + 8 * k];
                        }
                    }
                }
            }
            __syncthreads();
        }
    }
}


// ---- BatchNorm ------------------------------------------------------------------------------------
// partial column sums over a slab of rows; double atomics into ws[0..C) (sum) and ws[C..2C) (sum of squares)
__global__ void __launch_bounds__(256)
bn_stats_kernel(const float* __restrict__ x, double* __restrict__ ws, int R, int C, int rows_per_block) {
    __shared__ float s1[8][32], s2[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    const int r_begin = blockIdx.y * rows_per_block;
    const int r_end = min(R, r_begin + rows_per_block);
    float a = 0.0f, b = 0.0f;
    if (c < C)
        for (int r = r_begin + ty; r < r_end; r += 8) {
            const float v = x[static_cast<long long>(r) * C + c];
            a += v;
            b += v * v;
        }
    s1[ty][tx] = a;
    s2[ty][tx] = b;
    __syncthreads();
    if (ty == 0 && c < C) {
        double da = 0.0, db = 0.0;
        for (int k = 0; k < 8; ++k) { da += s1[k][tx]; db += s2[k][tx]; }
        atomicAdd(&ws[c], da);
        atomicAdd(&ws[C + c], db);
    }
}

// float4 variant (C % 4 == 0): 128 columns per block, 8 rows in flight per block, 4 rows unrolled per thread
__global__ void __launch_bounds__(256)
bn_stats4_kernel(const float* __restrict__ x, double* __restrict__ ws, int R, int C, int rows_per_block) {
    __shared__ float4 s1[8][32], s2[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + tx) * 4;
    const int r_begin = blockIdx.y * rows_per_block;
    const int r_end = min(R, r_begin + rows_per_block);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (c < C) {
        int r = r_begin + ty;
        for (; r + 24 < r_end; r += 32) {
            float4 v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = *reinterpret_cast<const float4*>(x + static_cast<long long>(r + 8 * k) * C + c);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a.x += v[k].x; a.y += v[k].y; a.z += v[k].z; a.w += v[k].w;
                b.x += v[k].x * v[k].x; b.y += v[k].y * v[k].y; b.z += v[k].z * v[k].z; b.w += v[k].w * v[k].w;
            }
        }
        for (; r < r_end; r += 8) {
            const float4 v = *reinterpret_cast<const float4*>(x + static_cast<long long>(r) * C + c);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
            b.x += v.x * v.x; b.y += v.y * v.y; b.z += v.z * v.z; b.w += v.w * v.w;
        }
    }
    s1[ty][tx] = a;
    s2[ty][tx] = b;
    __syncthreads();
    if (ty == 0 && c < C) {
        double da[4] = {0, 0, 0, 0}, db[4] = {0, 0, 0, 0};
        for (int k = 0; k < 8; ++k) {
            da[0] += s1[k][tx].x; da[1] += s1[k][tx].y; da[2] += s1[k][tx].z; da[3] += s1[k][tx].w;
            db[0] += s2[k][tx].x; db[1] += s2[k][tx].y; db[2] += s2[k][tx].z; db[3] += s2[k][tx].w;
        }
        for (int k = 0; k < 4; ++k) {
            atomicAdd(&ws[c + k], da[k]);
            atomicAdd(&ws[C + c + k], db[k]);
        }
    }
}

__global__ void bn_finalize_kernel(const double* __restrict__ ws, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float momentum, float eps, float* __restrict__ mean,
                                   float* __restrict__ rstd, float* __restrict__ scale, float* __restrict__ shift, int R,
                                   int C) {
    // R = number of rows the statistics are over (the valid-frame count in packed mode: zero padding rows add nothing to the sums)
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double m = ws[c] / R;
    double var = ws[C + c] / R - m * m;
    if (var < 0.0) var = 0.0;
    const float rs = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    mean[c] = static_cast<float>(m);
    rstd[c] = rs;
    const float g = gamma ? gamma[c] : 1.0f, b = beta ? beta[c] : 0.0f;
    scale[c] = g * rs;
    shift[c] = b - static_cast<float>(m) * g * rs;
    if (running_mean) {
        const double unbiased = R > 1 ? var * R / (R - 1) : var;
        running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * static_cast<float>(m);
        running_var[c] = (1.0f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
    }
}

// inference: scale/shift from running statistics
__global__ void bn_eval_affine_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                      const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                      float eps, float* __restrict__ scale, float* __restrict__ shift, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float rs = rsqrtf(running_var[c] + eps);
    const float g = gamma ? gamma[c] : 1.0f, b = beta ? beta[c] : 0.0f;
    scale[c] = g * rs;
    shift[c] = b - running_mean[c] * g * rs;
}

// sums over rows of dy and dy * xhat (xhat = (x - mean) * rstd)
__global__ void __launch_bounds__(256)
bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ mean,
                     const float* __restrict__ rstd, double* __restrict__ ws, int R, int C, int rows_per_block) {
    __shared__ float s1[8][32], s2[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    const int r_begin = blockIdx.y * rows_per_block;
    const int r_end = min(R, r_begin + rows_per_block);
    float a = 0.0f, b = 0.0f;
    if (c < C) {
        const float m = mean[c], rs = rstd[c];
        for (int r = r_begin + ty; r < r_end; r += 8) {
            const long long o = static_cast<long long>(r) * C + c;
            const float g = dy[o];
            a += g;
            b += g * (x[o] - m) * rs;
        }
    }
    s1[ty][tx] = a;
    s2[ty][tx] = b;
    __syncthreads();
    if (ty == 0 && c < C) {
        double da = 0.0, db = 0.0;
        for (int k = 0; k < 8; ++k) { da += s1[k][tx]; db += s2[k][tx]; }
        atomicAdd(&ws[c], da);
        atomicAdd(&ws[C + c], db);
    }
}

// dx = gamma*rstd * (dy - sum_dy/R - xhat * sum_dy_xhat/R); also emits dgamma / dbeta (block 0)
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ mean,
                    const float* __restrict__ rstd, const float* __restrict__ gamma, const double* __restrict__ ws,
                    float* __restrict__ dx, float* __restrict__ dgamma, float* __restrict__ dbeta, int R, int C, int Rv) {
    const long long total = static_cast<long long>(R) * C;
    const float invR = 1.0f / Rv;   // Rv = rows the statistics were taken over (packed mode: valid frames only)
    for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
         e += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(e % C);
        const float rs = rstd[c], g = gamma ? gamma[c] : 1.0f;
        const float xh = (x[e] - mean[c]) * rs;
        const float sdy = static_cast<float>(ws[c]), sdyx = static_cast<float>(ws[C + c]);
        dx[e] = g * rs * (dy[e] - sdy * invR - xh * sdyx * invR);
    }
    if (blockIdx.x == 0)
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            if (dbeta) dbeta[c] = static_cast<float>(ws[c]);
            if (dgamma) dgamma[c] = static_cast<float>(ws[C + c]);
        }
}

// float4 variant of the reduction (C % 4 == 0): 128 columns per block, 8 rows in flight per block, 4 rows unrolled
__global__ void __launch_bounds__(256)
bn_bwd_reduce4_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ mean,
                      const float* __restrict__ rstd, double* __restrict__ ws, int R, int C, int rows_per_block) {
    __shared__ float4 s1[8][32], s2[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + tx) * 4;
    const int r_begin = blockIdx.y * rows_per_block;
    const int r_end = min(R, r_begin + rows_per_block);
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (c < C) {
        const float4 m = *reinterpret_cast<const float4*>(mean + c), rs = *reinterpret_cast<const float4*>(rstd + c);
        int r = r_begin + ty;
        for (; r + 24 < r_end; r += 32) {
            float4 g[4], v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const long long o = static_cast<long long>(r + 8 * k) * C + c;
                g[k] = __ldcs(reinterpret_cast<const float4*>(dy + o));
                v[k] = __ldcs(reinterpret_cast<const float4*>(x + o));
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a.x += g[k].x; a.y += g[k].y; a.z += g[k].z; a.w += g[k].w;
                b.x += g[k].x * (v[k].x - m.x) * rs.x; b.y += g[k].y * (v[k].y - m.y) * rs.y;
                b.z += g[k].z * (v[k].z - m.z) * rs.z; b.w += g[k].w * (v[k].w - m.w) * rs.w;
            }
        }
        for (; r < r_end; r += 8) {
            const long long o = static_cast<long long>(r) * C + c;
            const float4 g = *reinterpret_cast<const float4*>(dy + o), v = *reinterpret_cast<const float4*>(x + o);
            a.x += g.x; a.y += g.y; a.z += g.z; a.w += g.w;
            b.x += g.x * (v.x - m.x) * rs.x; b.y += g.y * (v.y - m.y) * rs.y;
            b.z += g.z * (v.z - m.z) * rs.z; b.w += g.w * (v.w - m.w) * rs.w;
        }
    }
    s1[ty][tx] = a;
    s2[ty][tx] = b;
    __syncthreads();
    if (ty == 0 && c < C) {
        double da[4] = {0, 0, 0, 0}, db[4] = {0, 0, 0, 0};
        for (int k = 0; k < 8; ++k) {
            da[0] += s1[k][tx].x; da[1] += s1[k][tx].y; da[2] += s1[k][tx].z; da[3] += s1[k][tx].w;
            db[0] += s2[k][tx].x; db[1] += s2[k][tx].y; db[2] += s2[k][tx].z; db[3] += s2[k][tx].w;
        }
        for (int k = 0; k < 4; ++k) {
            atomicAdd(&ws[c + k], da[k]);
            atomicAdd(&ws[C + c + k], db[k]);
        }
    }
}

// Per-column coefficients of the input gradient, dx = A*dy + B*x + D, for consumers that apply BatchNorm's backward on the
// fly (the BPTT kernel of the layer below): A = g rstd, B = -g rstd^2 S2/R, D = g rstd (mean rstd S2 - S1)/R with
// S1 = sum dy, S2 = sum dy*xhat. Also emits dgamma = S2, dbeta = S1.
__global__ void bn_bwd_coef_kernel(const double* __restrict__ ws, const float* __restrict__ mean, const float* __restrict__ rstd,
                                   const float* __restrict__ gamma, float* __restrict__ coef, float* __restrict__ dgamma,
                                   float* __restrict__ dbeta, int R, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double s1 = ws[c], s2 = ws[C + c];
    const double g = gamma ? static_cast<double>(gamma[c]) : 1.0, rs = rstd[c], m = mean[c];
    coef[c] = static_cast<float>(g * rs);
    coef[C + c] = static_cast<float>(-g * rs * rs * s2 / R);
    coef[2 * C + c] = static_cast<float>(g * rs * (m * rs * s2 - s1) / R);
    if (dbeta) dbeta[c] = static_cast<float>(s1);
    if (dgamma) dgamma[c] = static_cast<float>(s2);
}

// ---- log-softmax ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
log_softmax_fwd_kernel(const float* __restrict__ x, long long x_pitch, float* __restrict__ y, int R, int C) {
    const int lane = threadIdx.x & 31;
    const long long wpb = blockDim.x >> 5;
    for (long long r = blockIdx.x * wpb + (threadIdx.x >> 5); r < R; r += gridDim.x * wpb) {
        const float* p = x + r * x_pitch;
        float m = -INFINITY;
        for (int c = lane; c < C; c += 32) m = fmaxf(m, p[c]);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float s = 0.0f;
        for (int c = lane; c < C; c += 32) s += expf(p[c] - m);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float lse = m + logf(s);
        float* q = y + r * C;
        for (int c = lane; c < C; c += 32) q[c] = p[c] - lse;
    }
}

// dx = g - exp(y) * sum_c g
__global__ void __launch_bounds__(256)
log_softmax_bwd_kernel(const float* __restrict__ g, const float* __restrict__ y, float* __restrict__ dx, int R, int C) {
    const int lane = threadIdx.x & 31;
    const long long wpb = blockDim.x >> 5;
    for (long long r = blockIdx.x * wpb + (threadIdx.x >> 5); r < R; r += gridDim.x * wpb) {
        const float* gp = g + r * C;
        const float* yp = y + r * C;
        float s = 0.0f;
        for (int c = lane; c < C; c += 32) s += gp[c];
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        float* d = dx + r * C;
        for (int c = lane; c < C; c += 32) d[c] = gp[c] - expf(yp[c]) * s;
    }
}

// out[r, c] = a[r, c] * mask[r, c] * inv_keep (dropout apply; the mask comes from the host framework's RNG)
__global__ void scale_mask_kernel(float* __restrict__ a, const uint8_t* __restrict__ mask, float inv_keep, long long n) {
    for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < n;
         e += static_cast<long long>(gridDim.x) * blockDim.x)
        a[e] = mask[e] ? a[e] * inv_keep : 0.0f;
}

// Packed-sequence support (my_863_corpus/steps/model.py:37-56,93-141): the recurrent kernels always scan all T rows of a padded
// [T, N, W] tensor, so packed semantics come from ALIGNMENT — the forward direction sees the left-aligned batch, the reverse
// direction a right-aligned copy (frame k of utterance n at row T - len_n + k) whose scan T-1 -> 0 meets the last valid frame
// first. This kernel moves data between the two alignments and zeroes the padding rows:
//   columns [0, split)  : dst[t, n] = t < len_n ? src[t, n] : 0                                  (mask only)
//   columns [split, W)  : dir = +1 (right -> left): dst[t, n] = t < len_n ? src[t + T - len_n, n] : 0
//                         dir = -1 (left -> right): dst[t, n] = t >= T - len_n ? src[t - (T - len_n), n] : 0
// accumulate = 1 adds into dst instead of overwriting it (dX of the reverse direction joining that of the forward direction).
__global__ void __launch_bounds__(256)
realign_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, const long long* __restrict__ lengths, int T, int N,
                    int W, int split, int dir, int accumulate) {
    const long long total = static_cast<long long>(T) * N * W;
    for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
         e += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(e % W);
        const long long rn = e / W;
        const int n = static_cast<int>(rn % N), t = static_cast<int>(rn / N);
        int len = static_cast<int>(lengths[n]);
        len = len < 0 ? 0 : (len > T ? T : len);
        float v = 0.0f;
        if (c < split) {
            if (t < len) v = src[e];
        } else if (dir > 0) {
            if (t < len) v = src[(static_cast<long long>(t + T - len) * N + n) * W + c];
        } else {
            if (t >= T - len) v = src[(static_cast<long long>(t - (T - len)) * N + n) * W + c];
        }
        dst[e] = accumulate ? dst[e] + v : v;
    }
}

int stream_grid(long long work_items, int per_block) {
    long long b = (work_items + per_block - 1) / per_block;
    const long long cap = static_cast<long long>(device_sm_count()) * 8;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return static_cast<int>(b);
}

}  // namespace
}  // namespace ctcb200

using namespace ctcb200;

extern "C" CTCB200_API int ctcb200_pack_lstm_weights(const float* wih_f, const float* whh_f, const float* wih_r,
                                                     const float* whh_r, void* wih_p, void* wihT_p, void* whh_p,
                                                     void* whhT_p, int H, int I, int Ipad, int part, int gates,
                                                     ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(H % 32 == 0 && I > 0 && Ipad >= I && Ipad % 8 == 0, "pack_lstm_weights: bad sizes H=%d I=%d Ipad=%d", H, I, Ipad);
    CTCB_REQUIRE(gates == 4 || gates == 3 || gates == 1, "pack_lstm_weights: gates %d not in {4 LSTM, 3 GRU, 1 RNN}", gates);
    const long long work = static_cast<long long>(8) * H * (Ipad > H ? Ipad : H);
    pack_lstm_weights_kernel<<<stream_grid(work, 1024), 256, 0, stream>>>(
        wih_f, whh_f, wih_r, whh_r, static_cast<__nv_bfloat16*>(wih_p), static_cast<__nv_bfloat16*>(wihT_p),
        static_cast<__nv_bfloat16*>(whh_p), static_cast<__nv_bfloat16*>(whhT_p), H, I, Ipad, part, gates);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_pack_lstm_weights_padded(const float* wih_f, const float* whh_f, const float* wih_r,
                                                            const float* whh_r, void* wih_p, void* wihT_p, void* whh_p,
                                                            void* whhT_p, int H, int Hp, int I, int i_blk, int i_blk_p, int Ipad,
                                                            int part, int gates, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(H >= 1 && Hp >= H && Hp % 32 == 0, "pack_lstm_weights_padded: bad hidden sizes H=%d Hp=%d", H, Hp);
    CTCB_REQUIRE(I > 0 && i_blk >= 1 && i_blk_p >= i_blk && I % i_blk == 0,
                 "pack_lstm_weights_padded: bad input map I=%d i_blk=%d i_blk_p=%d", I, i_blk, i_blk_p);
    const int I_dev = (I / i_blk) * i_blk_p;
    CTCB_REQUIRE(Ipad >= I_dev && Ipad % 8 == 0, "pack_lstm_weights_padded: Ipad=%d below the %d device columns", Ipad, I_dev);
    CTCB_REQUIRE(gates == 4 || gates == 3 || gates == 1, "pack_lstm_weights_padded: gates %d not in {4 LSTM, 3 GRU, 1 RNN}", gates);
    const long long work = static_cast<long long>(8) * Hp * (Ipad > Hp ? Ipad : Hp);
    pack_lstm_weights_padded_kernel<<<stream_grid(work, 1024), 256, 0, stream>>>(
        wih_f, whh_f, wih_r, whh_r, static_cast<__nv_bfloat16*>(wih_p), static_cast<__nv_bfloat16*>(wihT_p),
        static_cast<__nv_bfloat16*>(whh_p), static_cast<__nv_bfloat16*>(whhT_p), H, Hp, I, i_blk, i_blk_p, I_dev, Ipad, part,
        gates);
    CTCB_LAUNCH_CHECK();
    return OK;
}

namespace ctcb200 {
namespace {
// dst only (no transposed copy): pure streaming cast, float4 in / 4 x bf16 out, optional per-column affine (BatchNorm apply)
__global__ void __launch_bounds__(256)
cast_rows4_kernel(const float* __restrict__ src, long long s_outer, long long s_inner, int n_inner,
                  const float* __restrict__ scale, const float* __restrict__ shift, __nv_bfloat16* __restrict__ dst,
                  long long dst_pitch, int R, int C, int part) {
    const int c4 = C >> 2;
    const long long total = static_cast<long long>(R) * c4;
    for (long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
         e += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int r = static_cast<int>(e / c4), c = static_cast<int>(e - static_cast<long long>(r) * c4) * 4;
        float4 v = __ldcs(reinterpret_cast<const float4*>(src + static_cast<long long>(r / n_inner) * s_outer +
                                                           static_cast<long long>(r % n_inner) * s_inner + c));
        if (scale) {
            const float4 sc = *reinterpret_cast<const float4*>(scale + c), sh = *reinterpret_cast<const float4*>(shift + c);
            v.x = v.x * sc.x + sh.x; v.y = v.y * sc.y + sh.y; v.z = v.z * sc.z + sh.z; v.w = v.w * sc.w + sh.w;
        }
        __nv_bfloat162 lo = bf16x2_part(v.x, v.y, part), hi = bf16x2_part(v.z, v.w, part);
        uint2 o = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        *reinterpret_cast<uint2*>(dst + static_cast<long long>(r) * dst_pitch + c) = o;
    }
}
}  // namespace
}  // namespace ctcb200

extern "C" CTCB200_API int ctcb200_cast_transpose(const float* src, int64_t s_outer, int64_t s_inner, int n_inner,
                                                  const float* scale, const float* shift, void* dst, int64_t dst_pitch,
                                                  void* dstT, int64_t dstT_pitch, int n_pad, int R, int C, int part,
                                                  ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(R > 0 && C > 0 && n_inner > 0, "cast_transpose: empty R=%d C=%d", R, C);
    CTCB_REQUIRE(dst || dstT, "cast_transpose: no output requested");
    CTCB_REQUIRE(n_pad >= n_inner, "cast_transpose: n_pad %d < n_inner %d", n_pad, n_inner);
    const bool vec = (C % 2 == 0) && (s_outer % 2 == 0) && (s_inner % 2 == 0) && (dst_pitch % 2 == 0) &&
                     (dstT_pitch % 2 == 0) && ((reinterpret_cast<uintptr_t>(src) & 7) == 0);
    const bool rows4 = dst && !dstT && (C % 4 == 0) && (s_outer % 4 == 0) && (s_inner % 4 == 0) && (dst_pitch % 4 == 0) &&
                       dst_pitch == C && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dst) & 7) == 0) &&
                       (!scale || ((reinterpret_cast<uintptr_t>(scale) | reinterpret_cast<uintptr_t>(shift)) & 15) == 0);
    if (rows4) {
        ctcb200::cast_rows4_kernel<<<stream_grid(static_cast<long long>(R) * (C / 4), 2048), 256, 0, stream>>>(
            src, s_outer, s_inner, n_inner, scale, shift, static_cast<__nv_bfloat16*>(dst), dst_pitch, R, C, part);
    } else if (vec) {
        const long long tiles = static_cast<long long>((R + 63) / 64) * ((C + 63) / 64);
        cast_transpose_v2_kernel<<<stream_grid(tiles, 1), 256, 0, stream>>>(
            src, s_outer, s_inner, n_inner, scale, shift, static_cast<__nv_bfloat16*>(dst), dst_pitch,
            static_cast<__nv_bfloat16*>(dstT), dstT_pitch, n_pad, R, C, part);
    } else {
        const long long tiles = static_cast<long long>((R + 31) / 32) * ((C + 31) / 32);
        cast_transpose_kernel<<<stream_grid(tiles, 1), 256, 0, stream>>>(
            src, s_outer, s_inner, n_inner, scale, shift, static_cast<__nv_bfloat16*>(dst), dst_pitch,
            static_cast<__nv_bfloat16*>(dstT), dstT_pitch, n_pad, R, C, part);
    }
    CTCB_LAUNCH_CHECK();
    return OK;
}


// ws: 2*C doubles of scratch. Training statistics over R rows; writes mean/rstd (saved for backward),
// scale/shift (the affine cast_transpose applies) and updates the running statistics like nn.BatchNorm1d.
extern "C" CTCB200_API int ctcb200_bn_train_stats(const float* x, int R, int C, const float* gamma, const float* beta,
                                                  float* running_mean, float* running_var, float momentum, float eps,
                                                  float* mean, float* rstd, float* scale, float* shift, void* ws,
                                                  int n_valid, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(R > 0 && C > 0, "bn_train_stats: empty R=%d C=%d", R, C);
    CTCB_REQUIRE(n_valid >= 0 && n_valid <= R, "bn_train_stats: n_valid %d outside [0, R=%d]", n_valid, R);
    const int Rv = n_valid > 0 ? n_valid : R;
    CTCB_CUDA(cudaMemsetAsync(ws, 0, static_cast<size_t>(2) * C * sizeof(double), stream));
    const bool vec = (C % 4 == 0) && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    const int cols_per_block = vec ? 128 : 32;
    const int col_blocks = (C + cols_per_block - 1) / cols_per_block;
    int row_blocks = (device_sm_count() * 4 + col_blocks - 1) / col_blocks;
    int rows_per_block = (R + row_blocks - 1) / row_blocks;
    if (rows_per_block < 64) rows_per_block = 64;
    row_blocks = (R + rows_per_block - 1) / rows_per_block;
    if (vec) bn_stats4_kernel<<<dim3(col_blocks, row_blocks), 256, 0, stream>>>(x, static_cast<double*>(ws), R, C, rows_per_block);
    else bn_stats_kernel<<<dim3(col_blocks, row_blocks), 256, 0, stream>>>(x, static_cast<double*>(ws), R, C, rows_per_block);
    CTCB_LAUNCH_CHECK();
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, stream>>>(static_cast<const double*>(ws), gamma, beta, running_mean,
                                                          running_var, momentum, eps, mean, rstd, scale, shift, Rv, C);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean,
                                                  const float* running_var, float eps, float* scale, float* shift,
                                                  int C, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    bn_eval_affine_kernel<<<(C + 127) / 128, 128, 0, stream>>>(gamma, beta, running_mean, running_var, eps, scale, shift, C);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_bn_bwd(const float* dy, const float* x, const float* mean, const float* rstd,
                                          const float* gamma, float* dx, float* dgamma, float* dbeta, int R, int C,
                                          void* ws, int n_valid, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(R > 0 && C > 0, "bn_bwd: empty R=%d C=%d", R, C);
    CTCB_CUDA(cudaMemsetAsync(ws, 0, static_cast<size_t>(2) * C * sizeof(double), stream));
    const int col_blocks = (C + 31) / 32;
    int row_blocks = (device_sm_count() * 4 + col_blocks - 1) / col_blocks;
    int rows_per_block = (R + row_blocks - 1) / row_blocks;
    if (rows_per_block < 64) rows_per_block = 64;
    row_blocks = (R + rows_per_block - 1) / rows_per_block;
    bn_bwd_reduce_kernel<<<dim3(col_blocks, row_blocks), 256, 0, stream>>>(dy, x, mean, rstd, static_cast<double*>(ws), R, C,
                                                                         rows_per_block);
    CTCB_LAUNCH_CHECK();
    bn_bwd_apply_kernel<<<stream_grid(static_cast<long long>(R) * C, 1024), 256, 0, stream>>>(
        dy, x, mean, rstd, gamma, static_cast<const double*>(ws), dx, dgamma, dbeta, R, C, n_valid > 0 ? n_valid : R);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_bn_bwd_coef(const float* dy, const float* x, const float* mean, const float* rstd,
                                               const float* gamma, float* coef, float* dgamma, float* dbeta, int R, int C,
                                               void* ws, int n_valid, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(R > 0 && C > 0, "bn_bwd_coef: empty R=%d C=%d", R, C);
    CTCB_CUDA(cudaMemsetAsync(ws, 0, static_cast<size_t>(2) * C * sizeof(double), stream));
    const bool vec = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) |
                                       reinterpret_cast<uintptr_t>(mean) | reinterpret_cast<uintptr_t>(rstd)) & 15) == 0;
    const int cols_per_block = vec ? 128 : 32;
    const int col_blocks = (C + cols_per_block - 1) / cols_per_block;
    int row_blocks = (device_sm_count() * 4 + col_blocks - 1) / col_blocks;
    int rows_per_block = (R + row_blocks - 1) / row_blocks;
    if (rows_per_block < 64) rows_per_block = 64;
    row_blocks = (R + rows_per_block - 1) / rows_per_block;
    if (vec)
        bn_bwd_reduce4_kernel<<<dim3(col_blocks, row_blocks), 256, 0, stream>>>(dy, x, mean, rstd, static_cast<double*>(ws), R, C,
                                                                              rows_per_block);
    else
        bn_bwd_reduce_kernel<<<dim3(col_blocks, row_blocks), 256, 0, stream>>>(dy, x, mean, rstd, static_cast<double*>(ws), R, C,
                                                                             rows_per_block);
    CTCB_LAUNCH_CHECK();
    bn_bwd_coef_kernel<<<(C + 127) / 128, 128, 0, stream>>>(static_cast<const double*>(ws), mean, rstd, gamma, coef, dgamma, dbeta,
                                                          n_valid > 0 ? n_valid : R, C);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_log_softmax_fwd(const float* x, int64_t x_pitch, float* y, int R, int C,
                                                   ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(R > 0 && C > 0, "log_softmax_fwd: empty R=%d C=%d", R, C);
    log_softmax_fwd_kernel<<<stream_grid(R, 8), 256, 0, stream>>>(x, x_pitch, y, R, C);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_log_softmax_bwd(const float* g, const float* y, float* dx, int R, int C,
                                                   ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(R > 0 && C > 0, "log_softmax_bwd: empty R=%d C=%d", R, C);
    log_softmax_bwd_kernel<<<stream_grid(R, 8), 256, 0, stream>>>(g, y, dx, R, C);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_dropout_apply(float* a, const void* mask_u8, float inv_keep, int64_t n,
                                                 ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(n > 0, "dropout_apply: empty");
    scale_mask_kernel<<<stream_grid(n, 1024), 256, 0, stream>>>(a, static_cast<const uint8_t*>(mask_u8), inv_keep, n);
    CTCB_LAUNCH_CHECK();
    return OK;
}

extern "C" CTCB200_API int ctcb200_realign_rows(const float* src, float* dst, const void* lengths_i64, int T, int N, int W,
                                                int split, int dir, int accumulate, ctcb200_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CTCB_REQUIRE(T > 0 && N > 0 && W > 0 && split >= 0 && split <= W, "realign_rows: bad sizes T=%d N=%d W=%d split=%d", T, N, W, split);
    CTCB_REQUIRE(src != dst || split == W, "realign_rows: in-place use is only valid when every column is mask-only (split == W)");
    realign_rows_kernel<<<stream_grid(static_cast<long long>(T) * N * W, 1024), 256, 0, stream>>>(
        src, dst, static_cast<const long long*>(lengths_i64), T, N, W, split, dir, accumulate);
    CTCB_LAUNCH_CHECK();
    return OK;
}
