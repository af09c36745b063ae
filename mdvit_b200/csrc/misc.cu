// Small HBM-bound kernels: 1-channel heads (commuted 1x1 conv), bias-gradient column sums, casts / weight
// preparation, the fused segmentation + MKD losses, fused AdamW.
#include "../../include/mdvit_b200.h"
#include <stdlib.h>

#include "common.cuh"

namespace {

// ---------------------------------------------------------------------------------- rowdot: logits[m] = sum_c x[m,c] w[c] m(b,c) + bias
// The reference applies the C->1 1x1 conv AFTER a bilinear upsample (mdvit.py:699-700, Decoders.py:336-337); bilinear
// weights sum to 1 per channel so conv and resize commute exactly and the conv runs at 1/16 of the pixels.
// Optional Dropout2d (Decoders.py:334): whole (sample, channel) planes are dropped, mask = f(rng, stream, b*C+c).
template <typename TI>
__global__ void __launch_bounds__(256) rowdot_fwd_kernel(const TI* __restrict__ x, const float* __restrict__ w,
                                                          const float* __restrict__ bias, float* __restrict__ out, int M, int C,
                                                          int rows_per_sample, float drop_p, const unsigned long long* __restrict__ rng,
                                                          uint32_t stream) {
    MDV_PDL_SYNC();
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= M) return;
    uint32_t thr = 0, key = 0;
    float inv = 1.f;
    if (drop_p > 0.f) {
        thr = drop_thresh(drop_p);
        inv = 1.f / (1.f - drop_p);
        key = rng_key(rng, stream);
    }
    const int b = row / rows_per_sample;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) {
        float wv = __ldg(w + c);
        if (thr) wv *= drop_scale(key, (unsigned long long)b * C + c, thr, inv);
        s += ldf(x + (size_t)row * C + c) * wv;
    }
    s = warp_sum(s);
    if (lane == 0) out[row] = s + (bias ? bias[0] : 0.f);
}

// dx[m,c] = dlog[m] w[c] mask;  dw[c] += sum_m dlog[m] x[m,c] mask;  db += sum_m dlog[m]
template <typename TI>
__global__ void __launch_bounds__(256) rowdot_bwd_kernel(const float* __restrict__ dlog, const TI* __restrict__ x,
                                                          const float* __restrict__ w, float* __restrict__ dx, float* __restrict__ dw,
                                                          float* __restrict__ db, int M, int C, int rows_per_sample, float drop_p,
                                                          const unsigned long long* __restrict__ rng, uint32_t stream, int rows_per_block) {
    MDV_PDL_SYNC();
    // thread = channel (strided), block = chunk of rows of ONE sample
    uint32_t thr = 0, key = 0;
    float inv = 1.f;
    if (drop_p > 0.f) {
        thr = drop_thresh(drop_p);
        inv = 1.f / (1.f - drop_p);
        key = rng_key(rng, stream);
    }
    const int r0 = blockIdx.x * rows_per_block, r1 = min(M, r0 + rows_per_block);
    float dbacc = 0.f;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float acc = 0.f;
        const float wv = __ldg(w + c);
        int r = r0;
        while (r < r1) {       // rows of one sample share the Dropout2d mask of (sample, channel): hash once per segment
            const int b = r / rows_per_sample;
            const int rend = min(r1, (b + 1) * rows_per_sample);
            const float m = thr ? drop_scale(key, (unsigned long long)b * C + c, thr, inv) : 1.f;
            const float wm = wv * m;
#pragma unroll 4
            for (; r < rend; ++r) {
                const float d = __ldg(dlog + r);
                if (dx) dx[(size_t)r * C + c] = d * wm;
                acc += d * ldf(x + (size_t)r * C + c);
            }
            if (dw) atomicAdd(dw + c, acc * m);      // dw[c] += sum_m dlog[m] x[m,c] mask(b,c)
            acc = 0.f;
        }
    }
    if (db && threadIdx.x == 0) {
        for (int r = r0; r < r1; ++r) dbacc += dlog[r];
        atomicAdd(db, dbacc);
    }
}

// ---- vectorised versions (C a multiple of the 16-byte chunk, power-of-two chunks per row): the kernels above move 2-4 bytes per
// load, re-hash the Dropout2d mask of every (row, channel), and the backward ran 64-thread blocks at C = 64 (5x their HBM time)
template <typename TI> struct Chunk;
template <> struct Chunk<float> { static constexpr int E = 4; };
template <> struct Chunk<bf16> { static constexpr int E = 8; };
template <typename TI>
__device__ __forceinline__ void load_chunk(const TI* p, float (&v)[Chunk<TI>::E]) {
    if constexpr (sizeof(TI) == 4) {
        const float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
        const uint4 t = *reinterpret_cast<const uint4*>(p);
        const float2 a = bf2_to_f2(t.x), b = bf2_to_f2(t.y), c = bf2_to_f2(t.z), d = bf2_to_f2(t.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    }
}

// forward: LPR = min(32, chunks per row) lanes share a row (32 / LPR rows per warp pass), a warp owns a contiguous band of rows and
// keeps w * mask of its chunks in registers, re-evaluated only when the sample changes
template <typename TI, int NCH>      // NCH = chunks per lane (chunks per row / LPR)
__global__ void __launch_bounds__(256) rowdot_fwd_v_kernel(const TI* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ bias, float* __restrict__ out, int M, int C,
                                                            int rows_per_sample, float drop_p, const unsigned long long* __restrict__ rng,
                                                            uint32_t stream, int rows_per_warp) {
    MDV_PDL_SYNC();
    constexpr int E = Chunk<TI>::E;
    const int cpr = C / E;
    const int lpr = cpr < 32 ? cpr : 32, rpw = 32 / lpr;
    const int lane = threadIdx.x & 31, wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int cl = lane % lpr, rsub = lane / lpr;
    uint32_t thr = 0, key = 0;
    float inv = 1.f;
    if (drop_p > 0.f) {
        thr = drop_thresh(drop_p);
        inv = 1.f / (1.f - drop_p);
        key = rng_key(rng, stream);
    }
    const float b0 = bias ? bias[0] : 0.f;
    float wm[NCH][E];
    int cur_b = -1;
    const int r0 = wid * rows_per_warp, r1 = min(M, r0 + rows_per_warp);
    for (int r = r0 + rsub; r < r1 + rsub; r += rpw) {      // (all lanes of a row group iterate together: shuffles below)
        const bool ok = r < r1;
        const int rr = ok ? r : r1 - 1;
        const int b = rr / rows_per_sample;
        if (b != cur_b) {
            cur_b = b;
#pragma unroll
            for (int n = 0; n < NCH; ++n)
#pragma unroll
                for (int j = 0; j < E; ++j) {
                    const int c = (cl + n * lpr) * E + j;
                    wm[n][j] = __ldg(w + c) * (thr ? drop_scale(key, (unsigned long long)b * C + c, thr, inv) : 1.f);
                }
        }
        float s = 0.f;
#pragma unroll
        for (int n = 0; n < NCH; ++n) {
            float v[E];
            load_chunk<TI>(x + (size_t)rr * C + (cl + n * lpr) * E, v);
#pragma unroll
            for (int j = 0; j < E; ++j) s = fmaf(v[j], wm[n][j], s);
        }
        for (int o = lpr >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (ok && cl == 0) out[r] = s + b0;
    }
}

// backward: thread = one 16-byte chunk column, rows strided over the block's row lanes (4 in flight); dw partial sums in
// registers, reduced over the row lanes in shared memory, one atomic per channel and block
template <typename TI>
__global__ void __launch_bounds__(256) rowdot_bwd_v_kernel(const float* __restrict__ dlog, const TI* __restrict__ x,
                                                            const float* __restrict__ w, float* __restrict__ dx, float* __restrict__ dw,
                                                            float* __restrict__ db, int M, int C, int rows_per_sample, float drop_p,
                                                            const unsigned long long* __restrict__ rng, uint32_t stream, int rows_per_block) {
    MDV_PDL_SYNC();
    constexpr int E = Chunk<TI>::E;
    __shared__ float sh[256 * 8];
    const int tpr = C / E, rpi = 256 / tpr;
    const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr;
    uint32_t thr = 0, key = 0;
    float inv = 1.f;
    if (drop_p > 0.f) {
        thr = drop_thresh(drop_p);
        inv = 1.f / (1.f - drop_p);
        key = rng_key(rng, stream);
    }
    const int r0 = blockIdx.x * rows_per_block, r1 = min(M, r0 + rows_per_block);
    float acc[E], wv[E], mk[E], dbacc = 0.f;
#pragma unroll
    for (int j = 0; j < E; ++j) {
        acc[j] = 0.f;
        mk[j] = 1.f;
        wv[j] = rl < rpi ? __ldg(w + cl * E + j) : 0.f;
    }
    if (rl < rpi) {
        int cur_b = -1;
        constexpr int U = 4;
        for (int r = r0 + rl; r < r1; r += rpi * U) {
            float v[U][E], d[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int rr = r + u * rpi;
                d[u] = rr < r1 ? __ldg(dlog + rr) : 0.f;
                if (dw && rr < r1) load_chunk<TI>(x + (size_t)rr * C + cl * E, v[u]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int rr = r + u * rpi;
                if (rr >= r1) break;
                const int b = rr / rows_per_sample;
                if (b != cur_b) {      // rows of one sample share the Dropout2d mask of (sample, channel): flush, then re-hash
                    if (dw && cur_b >= 0) {
#pragma unroll
                        for (int j = 0; j < E; ++j) {
                            atomicAdd(dw + cl * E + j, acc[j] * mk[j]);
                            acc[j] = 0.f;
                        }
                    }
                    cur_b = b;
#pragma unroll
                    for (int j = 0; j < E; ++j) mk[j] = thr ? drop_scale(key, (unsigned long long)b * C + cl * E + j, thr, inv) : 1.f;
                }
                if (cl == 0) dbacc += d[u];
                if (dw) {
#pragma unroll
                    for (int j = 0; j < E; ++j) acc[j] = fmaf(d[u], v[u][j], acc[j]);
                }
                if (dx) {
                    float* o = dx + (size_t)rr * C + cl * E;
#pragma unroll
                    for (int j = 0; j < E; j += 4)
                        *reinterpret_cast<float4*>(o + j) = make_float4(d[u] * wv[j] * mk[j], d[u] * wv[j + 1] * mk[j + 1], d[u] * wv[j + 2] * mk[j + 2],
                                                                        d[u] * wv[j + 3] * mk[j + 3]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < E; ++j) acc[j] *= mk[j];
    }
    // reduce the row lanes: sh[rl][cl][j]
    if (dw) {
#pragma unroll
        for (int j = 0; j < E; ++j) sh[threadIdx.x * E + j] = rl < rpi ? acc[j] : 0.f;
        __syncthreads();
        for (int e = threadIdx.x; e < tpr * E; e += 256) {
            float t = 0.f;
            for (int q = 0; q < rpi; ++q) t += sh[(q * tpr) * E + e];
            atomicAdd(dw + e, t);
        }
    }
    if (db) {
        // (cl == 0 threads hold the dlog sums of their rows)
        __syncthreads();
        float* shb = sh;
        if (threadIdx.x < 32) shb[threadIdx.x] = 0.f;
        __syncthreads();
        if (rl < rpi && cl == 0) atomicAdd(shb + (rl & 31), dbacc);
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int q = 0; q < 32; ++q) t += shb[q];
            atomicAdd(db, t);
        }
    }
}

// ---------------------------------------------------------------------------------- column sums (bias gradients)
template <typename TI>
__global__ void __launch_bounds__(256) colsum_kernel(const TI* __restrict__ x, int ld, float* __restrict__ out, int M, int C,
                                                      int rows_per_block) {
    MDV_PDL_SYNC();
    __shared__ float sh[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    const int r0 = blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
    float s = 0.f;
    if (c < C)
        for (int r = r0 + ty; r < r1; r += 8) s += ldf(x + (size_t)r * ld + c);
    sh[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && c < C) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += sh[i][tx];
        atomicAdd(out + c, t);
    }
}

// ---------------------------------------------------------------------------------- casts
// out[m, c] (bf16, pitch ld_out) = in[m, c] (fp32, pitch ld_in) * rowscale[m / rps] * dropout_mask(m*C + c)
__global__ void __launch_bounds__(256) cast_bf16_kernel(const float* __restrict__ in, int ld_in, bf16* __restrict__ out, int ld_out,
                                                         long long M, int C, const float* __restrict__ rowscale, int rps, float drop_p,
                                                         const unsigned long long* __restrict__ rng, uint32_t stream) {
    MDV_PDL_SYNC();
    const int c4n = C >> 2;
    const int total = (int)(M * c4n);             // 32-bit element indices: the host checks M*C < 2^31
    uint32_t thr = 0, key = 0;
    float inv = 1.f;
    if (drop_p > 0.f) {
        thr = drop_thresh(drop_p);
        inv = 1.f / (1.f - drop_p);
        key = rng_key(rng, stream);
    }
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int c = (idx % c4n) * 4;
        const int m = idx / c4n;
        float4 v = *reinterpret_cast<const float4*>(in + (size_t)m * ld_in + c);
        float s = rowscale ? __ldg(rowscale + m / rps) : 1.f;
        float s0 = s, s1 = s, s2 = s, s3 = s;
        if (thr) {
            const uint32_t pr = (uint32_t)(((unsigned long long)m * C + c) >> 1);    // C, c multiples of 4: even index
            const uint32_t h0 = drop_hash(key, pr), h1 = drop_hash(key, pr + 1);
            s0 *= drop_lo(h0, thr, inv);
            s1 *= drop_hi(h0, thr, inv);
            s2 *= drop_lo(h1, thr, inv);
            s3 *= drop_hi(h1, thr, inv);
        }
        *reinterpret_cast<uint2*>(out + (size_t)m * ld_out + c) = make_uint2(f2_to_bf2(v.x * s0, v.y * s1), f2_to_bf2(v.z * s2, v.w * s3));
    }
}

// Same cast, plus column sums of the values written (the bias gradient of the Linear whose output gradient this is).
// block = (C/4 column groups) x (256 / (C/4) row lanes) over a chunk of rows; one atomic per column per block.
__global__ void __launch_bounds__(256) cast_bf16_colsum_kernel(const float* __restrict__ in, int ld_in, bf16* __restrict__ out,
                                                                int ld_out, int M, int C, const float* __restrict__ rowscale, int rps,
                                                                float drop_p, const unsigned long long* __restrict__ rng,
                                                                uint32_t stream, float* __restrict__ colsum, int rows_per_block) {
    MDV_PDL_SYNC();
    __shared__ float4 sh[256];
    const int cg = C >> 2;
    const int nty = 256 / cg;
    const int tx = threadIdx.x % cg, ty = threadIdx.x / cg;
    uint32_t thr = 0, key = 0;
    float inv = 1.f;
    if (drop_p > 0.f) {
        thr = drop_thresh(drop_p);
        inv = 1.f / (1.f - drop_p);
        key = rng_key(rng, stream);
    }
    const int r0 = blockIdx.x * rows_per_block, r1 = min(M, r0 + rows_per_block);
    const int c = tx * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ty < nty) {
#pragma unroll 4
        for (int m = r0 + ty; m < r1; m += nty) {
            const float4 v = *reinterpret_cast<const float4*>(in + (size_t)m * ld_in + c);
            const float s = rowscale ? __ldg(rowscale + m / rps) : 1.f;
            float s0 = s, s1 = s, s2 = s, s3 = s;
            if (thr) {
                const uint32_t pr = (uint32_t)(((unsigned long long)m * C + c) >> 1);
                const uint32_t h0 = drop_hash(key, pr), h1 = drop_hash(key, pr + 1);
                s0 *= drop_lo(h0, thr, inv);
                s1 *= drop_hi(h0, thr, inv);
                s2 *= drop_lo(h1, thr, inv);
                s3 *= drop_hi(h1, thr, inv);
            }
            const float o0 = v.x * s0, o1 = v.y * s1, o2 = v.z * s2, o3 = v.w * s3;
            acc.x += o0; acc.y += o1; acc.z += o2; acc.w += o3;
            *reinterpret_cast<uint2*>(out + (size_t)m * ld_out + c) = make_uint2(f2_to_bf2(o0, o1), f2_to_bf2(o2, o3));
        }
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (ty == 0) {
        for (int k = 1; k < nty; ++k) {
            const float4 o = sh[k * cg + tx];
            acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
        }
        atomicAdd(colsum + c, acc.x);
        atomicAdd(colsum + c + 1, acc.y);
        atomicAdd(colsum + c + 2, acc.z);
        atomicAdd(colsum + c + 3, acc.w);
    }
}

// out fp32 [M,C] (pitch ld_out) (+)= bf16/fp32 in (pitch ld_in)
template <typename TI>
__global__ void __launch_bounds__(256) add_f32_kernel(const TI* __restrict__ in, int ld_in, float* __restrict__ out, int ld_out,
                                                       long long M, int C, int accumulate) {
    MDV_PDL_SYNC();
    const long long total = M * C;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int c = (int)(idx % C);
        const long long m = idx / C;
        const float v = ldf(in + m * ld_in + c);
        float* o = out + m * ld_out + c;
        *o = accumulate ? *o + v : v;
    }
}

// Grouped fp32 FFMA products C[M,N] (=|+=) op(A)[M,K] . op(B)[K,N] (+ u[m] v[n]): the weight-sized products of the collapsed aux
// decoder.  Every problem of a group is independent (distinct C), so one grid covers them all: each is only 16-256 tiles and K <= 512,
// i.e. latency-bound, and launched one by one they ran back to back.  32 x 32 output tile per block, 2 x 2 per thread, k-steps of
// 32 staged in shared memory; the staging loads walk whichever index is contiguous in memory, so both orientations are coalesced.
constexpr int MM_T = 32;
constexpr int MM_MAX = 16;

struct MatmulGroup {
    MdvMatmulDesc d[MM_MAX];
    int tile0[MM_MAX + 1];      // first block of each problem
    int n;
};

__global__ void __launch_bounds__(256) matmul_f32_kernel(const __grid_constant__ MatmulGroup g) {
    MDV_PDL_SYNC();
    __shared__ float As[MM_T][MM_T + 1], Bs[MM_T][MM_T + 1];    // [k][m], [k][n]
    int p = 0;
    while (p + 1 < g.n && (int)blockIdx.x >= g.tile0[p + 1]) ++p;
    const MdvMatmulDesc& d = g.d[p];
    const int t = blockIdx.x - g.tile0[p], ntn = (d.N + MM_T - 1) / MM_T;
    const int m0 = (t / ntn) * MM_T, n0 = (t % ntn) * MM_T;
    const int M = d.M, N = d.N, K = d.K, ta = d.trans_a, tb = d.trans_b, lda = d.lda, ldb = d.ldb;
    const float* __restrict__ A = d.A;
    const float* __restrict__ B = d.B;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[2][2] = {};
    for (int k0 = 0; k0 < K; k0 += MM_T) {
        for (int e = threadIdx.x; e < MM_T * MM_T; e += 256) {
            const int r = e / MM_T, q = e % MM_T;       // q: the index contiguous in memory
            {
                const int m = ta ? q : r, k = ta ? r : q, gm = m0 + m, gk = k0 + k;
                As[k][m] = (gm < M && gk < K) ? A[ta ? (size_t)gk * lda + gm : (size_t)gm * lda + gk] : 0.f;
            }
            {
                const int n = tb ? r : q, k = tb ? q : r, gn = n0 + n, gk = k0 + k;
                Bs[k][n] = (gn < N && gk < K) ? B[tb ? (size_t)gn * ldb + gk : (size_t)gk * ldb + gn] : 0.f;
            }
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < MM_T; ++k) {
            const float a0 = As[k][ty], a1 = As[k][ty + 16], b0 = Bs[k][tx], b1 = Bs[k][tx + 16];
            acc[0][0] = fmaf(a0, b0, acc[0][0]);
            acc[0][1] = fmaf(a0, b1, acc[0][1]);
            acc[1][0] = fmaf(a1, b0, acc[1][0]);
            acc[1][1] = fmaf(a1, b1, acc[1][1]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int m = m0 + ty + 16 * i, n = n0 + tx + 16 * j;
            if (m < M && n < N) {
                float v = acc[i][j];
                if (d.u) v = fmaf(d.u[m], d.v[n], v);
                float* c = d.C + (size_t)m * d.ldc + n;
                *c = d.accumulate ? *c + v : v;
            }
        }
}

// Weight preparation: dst[r, c] = bf16(src[...]) with optional transpose / 3x3-conv permutation.
//  mode 0: src [R, Cc] row-major                       -> dst [R, ld]        (Linear / 1x1 conv weight)
//  mode 1: src [R, Cc] row-major                       -> dst [Cc, ld] = src^T (for input gradients)
//  mode 2: src [R, Cin, 3, 3] (PyTorch conv)           -> dst [R, ld], column (i*3+j)*Cin + ci    (im2col order)
//  mode 3: src [R, Cin, 3, 3]                          -> dst [9*Cin (pad to rows), ld] transposed of mode 2
//  mode 4: src [R, Cin, 3, 3]                          -> dst [Cin, ld], column t*R + r            (operand of the implicit-GEMM input gradient)
//  mode | 8: the same layouts with an fp32 destination (operands of the TF32 GEMMs of the conv trunk)
template <typename TO>
__global__ void __launch_bounds__(256) prep_weight_kernel(const float* __restrict__ src, TO* __restrict__ dst, int R, int Cc,
                                                           int ld, int mode, int cin) {
    MDV_PDL_SYNC();
    const long long total = (long long)R * Cc;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(idx / Cc), c = (int)(idx % Cc);
        TO v;
        stf(&v, src[idx]);
        if (mode == 0) {
            dst[(size_t)r * ld + c] = v;
        } else if (mode == 1) {
            dst[(size_t)c * ld + r] = v;
        } else if (mode == 4) {      // conv [R, Cin, 3, 3] -> [Cin, ld >= 9*R]: dst[ci, t*R + r] (input-gradient operand of mdv_conv3_gemm)
            const int ci = c / 9, t = c % 9;
            dst[(size_t)ci * ld + t * R + r] = v;
        } else {
            const int ci = c / 9, t = c % 9;
            const int col = t * cin + ci;
            if (mode == 2) dst[(size_t)r * ld + col] = v;
            else dst[(size_t)col * ld + r] = v;
        }
    }
}

// All bf16 operand copies of a model in ONE launch: blockIdx.y walks a device-resident table of (src, dst, shape, mode)
// descriptors (same modes as prep_weight_kernel).  Replaces ~200 tiny launches per training step.
__global__ void __launch_bounds__(256) prep_weights_batched_kernel(const MdvPrepDesc* __restrict__ descs) {
    MDV_PDL_SYNC();
    const MdvPrepDesc d = descs[blockIdx.y];
    const float* __restrict__ src = d.src;
    const int total = d.rows * d.cols;
    const int mode = d.mode & 7;
    const bool f32 = (d.mode & 8) != 0;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int r = idx / d.cols, c = idx % d.cols;
        size_t o;
        if (mode == 0) {
            o = (size_t)r * d.ld + c;
        } else if (mode == 1) {
            o = (size_t)c * d.ld + r;
        } else if (mode == 4) {
            o = (size_t)(c / 9) * d.ld + (size_t)(c % 9) * d.rows + r;
        } else {
            const int ci = c / 9, t = c % 9;
            const int col = t * d.cin + ci;
            o = mode == 2 ? (size_t)r * d.ld + col : (size_t)col * d.ld + r;
        }
        if (f32) ((float*)d.dst)[o] = src[idx];
        else ((bf16*)d.dst)[o] = __float2bfloat16_rn(src[idx]);
    }
}

// d(conv weight [R,Cin,3,3]) += dW_im2col[R, ld] (column (i*3+j)*Cin+ci)
__global__ void __launch_bounds__(256) unperm_conv_grad_kernel(const float* __restrict__ g, int ld, float* __restrict__ dw, int R,
                                                                int cin) {
    MDV_PDL_SYNC();
    const long long total = (long long)R * cin * 9;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(idx / (cin * 9)), c = (int)(idx % (cin * 9));
        const int ci = c / 9, t = c % 9;
        dw[idx] += g[(size_t)r * ld + t * cin + ci];
    }
}

// ---------------------------------------------------------------------------------- losses
// multi_train_MDViT.py:147-169 + Utils/losses.py:8-16.  p = sigmoid(out), q = sigmoid(aux), y = label.
// sums[0..7] = sum bce(p,y), sum bce(q,y), sum p*y, sum p*p, sum y*y, sum q*y, sum q*q, sum q*p     (double)
__device__ __forceinline__ float bce_term(float p, float y) {
    const float lp = fmaxf(logf(p), -100.f), l1p = fmaxf(logf(1.f - p), -100.f);
    return -(y * lp + (1.f - y) * l1p);
}

// labels travel as fp32 (the reference's label.cuda().float(), multi_train_MDViT.py:136) or as uint8 {0,1} (a quarter of
// the host->device bytes; same values)
template <typename LT>
__global__ void __launch_bounds__(256) loss_sums_kernel(const float* __restrict__ out, const float* __restrict__ aux,
                                                         const LT* __restrict__ label, double* __restrict__ sums, long long n) {
    MDV_PDL_SYNC();
    __shared__ float red[32];
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float y = (float)label[i];
        const float p = 1.f / (1.f + expf(-out[i]));
        const float q = aux ? 1.f / (1.f + expf(-aux[i])) : 0.f;
        a[0] += bce_term(p, y);
        a[2] += p * y;
        a[3] += p * p;
        a[4] += y * y;
        if (aux) {
            a[1] += bce_term(q, y);
            a[5] += q * y;
            a[6] += q * q;
            a[7] += q * p;
        }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float t = block_sum(a[k], red);
        if (threadIdx.x == 0) atomicAdd(sums + k, (double)t);
    }
}

// losses[0..2] = L_seg, L_aux, L_kt  (fp32), from (possibly all-reduced) sums;  n_total = global element count.
__global__ void loss_finalize_kernel(const double* __restrict__ sums, double n_total, float* __restrict__ losses) {
    MDV_PDL_SYNC();
    const double eps = 1e-5;
    const double bce_p = sums[0] / n_total, bce_q = sums[1] / n_total;
    const double dice_p = 1.0 - (2.0 * sums[2] + eps) / (sums[3] + sums[4] + eps);
    const double dice_q = 1.0 - (2.0 * sums[5] + eps) / (sums[6] + sums[4] + eps);
    const double dice_kt = 1.0 - (2.0 * sums[7] + eps) / (sums[6] + sums[3] + eps);
    losses[0] = (float)(bce_p + dice_p);
    losses[1] = (float)(bce_q + dice_q);
    losses[2] = (float)dice_kt;
}

// Gradients w.r.t. the logits for  L = c_seg*L_seg + c_aux*L_aux + c_kt*L_kt  (coef[0..2]); see SURVEY.md App. E.
// PyTorch's BCELoss backward: (p - y) / max(p(1-p), 1e-12) / n, times sigmoid' = p(1-p).
template <typename LT>
__global__ void __launch_bounds__(256) loss_bwd_kernel(const float* __restrict__ out, const float* __restrict__ aux,
                                                        const LT* __restrict__ label, const double* __restrict__ sums,
                                                        double n_total, const float* __restrict__ coef, float* __restrict__ dout,
                                                        float* __restrict__ daux, long long n) {
    MDV_PDL_SYNC();
    const double eps = 1e-5;
    const float c_seg = coef[0], c_aux = coef[1], c_kt = coef[2];
    const float inv_n = (float)(1.0 / n_total);
    // dice(s,t): dD/ds_i = -(2 t_i den - 2 s_i num) / den^2, num = 2I+eps, den = Z+Y+eps
    const double den_p = sums[3] + sums[4] + eps, num_p = 2.0 * sums[2] + eps;
    const double den_q = sums[6] + sums[4] + eps, num_q = 2.0 * sums[5] + eps;
    const double den_k = sums[6] + sums[3] + eps, num_k = 2.0 * sums[7] + eps;
    const float ap = (float)(2.0 / den_p), bp = (float)(2.0 * num_p / (den_p * den_p));
    const float aq = (float)(2.0 / den_q), bq = (float)(2.0 * num_q / (den_q * den_q));
    const float ak = (float)(2.0 / den_k), bk = (float)(2.0 * num_k / (den_k * den_k));
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float y = (float)label[i];
        const float p = 1.f / (1.f + expf(-out[i]));
        const float sp = p * (1.f - p);
        float gp = c_seg * ((p - y) / fmaxf(sp, 1e-12f) * inv_n + (-ap * y + bp * p));
        if (aux) {
            const float q = 1.f / (1.f + expf(-aux[i]));
            const float sq = q * (1.f - q);
            float gq = c_aux * ((q - y) / fmaxf(sq, 1e-12f) * inv_n + (-aq * y + bq * q));
            gq += c_kt * (-ak * p + bk * q);
            gp += c_kt * (-ak * q + bk * p);
            daux[i] = gq * sq;
        }
        dout[i] = gp * sp;
    }
}

// Dice / Jaccard counts of the thresholded prediction (multi_train_MDViT.py:172-177: medpy dc/jc of sigmoid(out) > 0.5 vs
// label > 0.5, on the host in the reference — one .cpu() sync per domain per step): counts[0..2] += |P&L|, |P|, |L|.
template <typename LT>
__global__ void __launch_bounds__(256) seg_counts_kernel(const float* __restrict__ logits, const LT* __restrict__ label,
                                                          unsigned long long* __restrict__ counts, long long n) {
    MDV_PDL_SYNC();
    unsigned int c0 = 0, c1 = 0, c2 = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const bool p = logits[i] > 0.f;            // sigmoid(x) > 0.5  <=>  x > 0
        const bool l = (float)label[i] > 0.5f;
        c0 += p && l;
        c1 += p;
        c2 += l;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c0 += __shfl_xor_sync(0xffffffffu, c0, o);
        c1 += __shfl_xor_sync(0xffffffffu, c1, o);
        c2 += __shfl_xor_sync(0xffffffffu, c2, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(counts + 0, (unsigned long long)c0);
        atomicAdd(counts + 1, (unsigned long long)c1);
        atomicAdd(counts + 2, (unsigned long long)c2);
    }
}

// ---------------------------------------------------------------------------------- AdamW (torch.optim.AdamW semantics)
// hyper (device fp64[8]): lr, beta1, beta2, eps, weight_decay, t (steps taken so far), unused, grad_scale
__global__ void adamw_tick_kernel(double* hyper) {
    MDV_PDL_SYNC();
    hyper[5] += 1.0;
}

__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                     float* __restrict__ v, const double* __restrict__ hyper, long long n) {
    MDV_PDL_SYNC();
    // the step count lives on the device (bumped by adamw_tick_kernel just before this kernel), so a CUDA-graph replay
    // needs no per-step host->device parameter traffic; bias corrections in double, as torch.optim.AdamW computes them
    const double t = hyper[5];
    const float lr = (float)hyper[0], b1 = (float)hyper[1], b2 = (float)hyper[2], eps = (float)hyper[3], wd = (float)hyper[4],
                gs = (float)hyper[7];
    const double bc1 = 1.0 - pow(hyper[1], t), bc2 = 1.0 - pow(hyper[2], t);
    const float step = (float)(hyper[0] / bc1), isb2 = (float)(1.0 / sqrt(bc2));
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += (long long)gridDim.x * blockDim.x * 4) {
        if (i + 3 < n) {
            float4 pp = *reinterpret_cast<float4*>(p + i), gg = *reinterpret_cast<const float4*>(g + i);
            float4 mm = *reinterpret_cast<float4*>(m + i), vv = *reinterpret_cast<float4*>(v + i);
            float pa[4] = {pp.x, pp.y, pp.z, pp.w}, ga[4] = {gg.x, gg.y, gg.z, gg.w}, ma[4] = {mm.x, mm.y, mm.z, mm.w},
                  va[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float gk = ga[k] * gs;
                pa[k] *= 1.f - lr * wd;
                ma[k] = b1 * ma[k] + (1.f - b1) * gk;
                va[k] = b2 * va[k] + (1.f - b2) * gk * gk;
                pa[k] -= step * ma[k] / (sqrtf(va[k]) * isb2 + eps);
            }
            *reinterpret_cast<float4*>(p + i) = make_float4(pa[0], pa[1], pa[2], pa[3]);
            *reinterpret_cast<float4*>(m + i) = make_float4(ma[0], ma[1], ma[2], ma[3]);
            *reinterpret_cast<float4*>(v + i) = make_float4(va[0], va[1], va[2], va[3]);
        } else {
            for (long long j = i; j < n; ++j) {
                const float gk = g[j] * gs;
                float pj = p[j] * (1.f - lr * wd);
                const float mj = b1 * m[j] + (1.f - b1) * gk, vj = b2 * v[j] + (1.f - b2) * gk * gk;
                pj -= step * mj / (sqrtf(vj) * isb2 + eps);
                p[j] = pj; m[j] = mj; v[j] = vj;
            }
        }
    }
}

__global__ void rng_bump_kernel(unsigned long long* rng) {
    MDV_PDL_SYNC(); rng[1] += 1ull; }

// DropPath per-sample scale: scale[b] = Bernoulli(1-p)/(1-p)   (timm DropPath, mdvit.py:339)
__global__ void droppath_scale_kernel(float* __restrict__ scale, int B, float p, const unsigned long long* __restrict__ rng,
                                      uint32_t stream) {
    MDV_PDL_SYNC();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    scale[b] = drop_scale(rng_key(rng, stream), (unsigned long long)b, drop_thresh(p), 1.f / (1.f - p));
}

inline int grid_for(long long total_threads) {
    long long b = (total_threads + 255) / 256;
    const long long cap = (long long)MDV_NUM_SMS * 16;
    return (int)(b < cap ? (b > 0 ? b : 1) : cap);
}

}  // namespace

long long g_mdv_launches = 0;
int g_mdv_pdl = []() {
    const char* e = getenv("MDV_NO_PDL");
    return (e && e[0] == '1') ? 0 : 1;
}();

extern "C" int mdv_set_pdl(int enabled) {
    g_mdv_pdl = enabled ? 1 : 0;
    return MDV_OK;
}

extern "C" int mdv_version(void) { return 100; }

extern "C" long long mdv_launch_count(void) { return g_mdv_launches; }

extern "C" int mdv_rowdot_fwd(const void* x, int x_bf16, const float* w, const float* bias, float* out, int M, int C,
                              int rows_per_sample, float drop_p, const void* rng, uint32_t drop_stream, void* stream) {
    if (!x || !w || !out || M <= 0 || rows_per_sample <= 0) return MDV_ERR_ARG;
    {   // vectorised path: 16-byte chunks, power-of-two chunks per row
        const int E = x_bf16 ? 8 : 4;
        const int cpr = C / E;
        const bool pow2 = cpr > 0 && (cpr & (cpr - 1)) == 0;
        if (!(C % E) && pow2 && cpr <= 128 && !(reinterpret_cast<uintptr_t>(x) & 15)) {
            const int nch = cpr <= 32 ? 1 : cpr / 32;
            int rpw = mdv_cdiv(M, 8 * 8 * MDV_NUM_SMS);      // ~8 blocks of 8 warps per SM
            const int rows_pass = cpr < 32 ? 32 / cpr : 1;
            rpw = mdv_cdiv(rpw < 16 ? 16 : rpw, rows_pass) * rows_pass;
            const int nb = mdv_cdiv(mdv_cdiv(M, rpw), 8);
            cudaStream_t st = (cudaStream_t)stream;
#define MDV_RDF(TI, N) mdv_launch((rowdot_fwd_v_kernel<TI, N>), dim3(nb), dim3(256), 0, st, (const TI*)x, w, bias, out, M, C, rows_per_sample, drop_p, \
                                  (const unsigned long long*)rng, drop_stream, rpw)
            if (x_bf16) { if (nch == 1) MDV_RDF(bf16, 1); else if (nch == 2) MDV_RDF(bf16, 2); else MDV_RDF(bf16, 4); }
            else { if (nch == 1) MDV_RDF(float, 1); else if (nch == 2) MDV_RDF(float, 2); else MDV_RDF(float, 4); }
#undef MDV_RDF
            MDV_CHECK_LAUNCH();
            return MDV_OK;
        }
    }
    const int blocks = mdv_cdiv(M, 8);
    if (x_bf16)
        mdv_launch(rowdot_fwd_kernel<bf16>, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (const bf16*)x, w, bias, out, M, C, rows_per_sample, drop_p, (const unsigned long long*)rng, drop_stream);
    else
        mdv_launch(rowdot_fwd_kernel<float>, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, (const float*)x, w, bias, out, M, C, rows_per_sample, drop_p, (const unsigned long long*)rng, drop_stream);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_rowdot_bwd(const float* dlog, const void* x, int x_bf16, const float* w, float* dx, float* dw, float* db, int M,
                              int C, int rows_per_sample, float drop_p, const void* rng, uint32_t drop_stream, void* stream) {
    if (!dlog || !x || !w || M <= 0 || rows_per_sample <= 0) return MDV_ERR_ARG;
    {
        const int E = x_bf16 ? 8 : 4;
        const int tpr = C / E;
        if (!(C % E) && tpr >= 1 && tpr <= 256 && !(reinterpret_cast<uintptr_t>(x) & 15) && (!dx || !(reinterpret_cast<uintptr_t>(dx) & 15))) {
            const int rpi = 256 / tpr;
            int rpbv = mdv_cdiv(M, 8 * MDV_NUM_SMS);
            if (rpbv < rpi * 16) rpbv = rpi * 16;
            const int nb = mdv_cdiv(M, rpbv);
            if (x_bf16)
                mdv_launch(rowdot_bwd_v_kernel<bf16>, dim3(nb), dim3(256), 0, (cudaStream_t)stream, dlog, (const bf16*)x, w, dx, dw, db, M, C, rows_per_sample,
                           drop_p, (const unsigned long long*)rng, drop_stream, rpbv);
            else
                mdv_launch(rowdot_bwd_v_kernel<float>, dim3(nb), dim3(256), 0, (cudaStream_t)stream, dlog, (const float*)x, w, dx, dw, db, M, C, rows_per_sample,
                           drop_p, (const unsigned long long*)rng, drop_stream, rpbv);
            MDV_CHECK_LAUNCH();
            return MDV_OK;
        }
    }
    int rpb = mdv_cdiv(M, 4 * MDV_NUM_SMS);
    if (rpb < 8) rpb = 8;
    const int blocks = mdv_cdiv(M, rpb);
    const int threads = C >= 256 ? 256 : (C >= 128 ? 128 : 64);
    if (x_bf16)
        mdv_launch(rowdot_bwd_kernel<bf16>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, dlog, (const bf16*)x, w, dx, dw, db, M, C, rows_per_sample, drop_p, (const unsigned long long*)rng, drop_stream, rpb);
    else
        mdv_launch(rowdot_bwd_kernel<float>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, dlog, (const float*)x, w, dx, dw, db, M, C, rows_per_sample, drop_p, (const unsigned long long*)rng, drop_stream, rpb);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_colsum(const void* x, int x_bf16, int ld, float* out, int M, int C, void* stream) {
    if (!x || !out || M <= 0 || C <= 0) return MDV_ERR_ARG;
    const int cb = mdv_cdiv(C, 32);
    int want = (8 * MDV_NUM_SMS) / cb;
    if (want < 1) want = 1;
    int rpb = mdv_cdiv(M, want);
    if (rpb < 64) rpb = 64;
    dim3 grid(cb, mdv_cdiv(M, rpb));
    if (x_bf16) mdv_launch(colsum_kernel<bf16>, dim3(grid), dim3(256), 0, (cudaStream_t)stream, (const bf16*)x, ld, out, M, C, rpb);
    else mdv_launch(colsum_kernel<float>, dim3(grid), dim3(256), 0, (cudaStream_t)stream, (const float*)x, ld, out, M, C, rpb);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_cast_bf16(const float* in, int ld_in, void* out_bf16, int ld_out, long long M, int C, const float* rowscale,
                             int rows_per_scale, float drop_p, const void* rng, uint32_t drop_stream, float* colsum, void* stream) {
    if (!in || !out_bf16 || (C & 3) || (ld_in & 3) || (ld_out & 3)) return MDV_ERR_ARG;
    if (M * C >= 0x7fffffffLL) return MDV_ERR_UNSUPPORTED;
    if (colsum) {
        if (C > 1024 || M > 0x7fffffffLL) return MDV_ERR_UNSUPPORTED;
        int rpb = mdv_cdiv(M, 4 * MDV_NUM_SMS);
        const int nty = 256 / (C / 4);
        if (rpb < 4 * nty) rpb = 4 * nty;
        mdv_launch(cast_bf16_colsum_kernel, dim3(mdv_cdiv(M, rpb)), dim3(256), 0, (cudaStream_t)stream, in, ld_in, (bf16*)out_bf16, ld_out, (int)M, C, rowscale,
                                                                                    rows_per_scale > 0 ? rows_per_scale : 1, drop_p,
                                                                                    (const unsigned long long*)rng, drop_stream, colsum, rpb);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    mdv_launch(cast_bf16_kernel, dim3(grid_for(M * (C / 4))), dim3(256), 0, (cudaStream_t)stream, in, ld_in, (bf16*)out_bf16, ld_out, M, C, rowscale,
                                                                               rows_per_scale > 0 ? rows_per_scale : 1, drop_p,
                                                                               (const unsigned long long*)rng, drop_stream);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_add_f32(const void* in, int in_bf16, int ld_in, float* out, int ld_out, long long M, int C, int accumulate,
                           void* stream) {
    if (!in || !out) return MDV_ERR_ARG;
    if (in_bf16) mdv_launch(add_f32_kernel<bf16>, dim3(grid_for(M * C)), dim3(256), 0, (cudaStream_t)stream, (const bf16*)in, ld_in, out, ld_out, M, C, accumulate);
    else mdv_launch(add_f32_kernel<float>, dim3(grid_for(M * C)), dim3(256), 0, (cudaStream_t)stream, (const float*)in, ld_in, out, ld_out, M, C, accumulate);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_matmul_f32_grouped(const MdvMatmulDesc* descs, int n, void* stream) {
    if (!descs || n <= 0 || n > MM_MAX) return MDV_ERR_ARG;
    MatmulGroup g = {};
    g.n = n;
    for (int i = 0; i < n; ++i) {
        const MdvMatmulDesc& d = descs[i];
        if (!d.A || !d.B || !d.C || d.M <= 0 || d.N <= 0 || d.K <= 0 || d.lda < (d.trans_a ? d.M : d.K) || d.ldb < (d.trans_b ? d.K : d.N) ||
            d.ldc < d.N || (!d.u != !d.v))
            return MDV_ERR_ARG;
        g.d[i] = d;
        g.tile0[i + 1] = g.tile0[i] + mdv_cdiv(d.M, MM_T) * mdv_cdiv(d.N, MM_T);
    }
    mdv_launch(matmul_f32_kernel, dim3(g.tile0[n]), dim3(256), 0, (cudaStream_t)stream, g);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_prep_weight(const float* src, void* dst, int R, int Cc, int ld, int mode, int cin, void* stream) {
    if (!src || !dst || mode < 0 || (mode & 7) > 4 || mode > 12) return MDV_ERR_ARG;
    if (mode & 8)
        mdv_launch(prep_weight_kernel<float>, dim3(grid_for((long long)R * Cc)), dim3(256), 0, (cudaStream_t)stream, src, (float*)dst, R, Cc, ld, mode & 7, cin);
    else
        mdv_launch(prep_weight_kernel<bf16>, dim3(grid_for((long long)R * Cc)), dim3(256), 0, (cudaStream_t)stream, src, (bf16*)dst, R, Cc, ld, mode, cin);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_prep_weights_batched(const MdvPrepDesc* descs_dev, int n, void* stream) {
    if (!descs_dev || n <= 0) return MDV_ERR_ARG;
    mdv_launch(prep_weights_batched_kernel, dim3(MDV_NUM_SMS, n), dim3(256), 0, (cudaStream_t)stream, descs_dev);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_unperm_conv_grad(const float* g, int ld, float* dw, int R, int cin, void* stream) {
    if (!g || !dw) return MDV_ERR_ARG;
    mdv_launch(unperm_conv_grad_kernel, dim3(grid_for((long long)R * cin * 9)), dim3(256), 0, (cudaStream_t)stream, g, ld, dw, R, cin);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

// sums: 8 doubles (zeroed here).  aux may be NULL (BASE model: only L_seg is meaningful).
extern "C" int mdv_loss_sums(const float* out, const float* aux, const void* label, int label_u8, void* sums, long long n, void* stream) {
    if (!out || !label || !sums || n <= 0) return MDV_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(sums, 0, 8 * sizeof(double), st);
    if (e != cudaSuccess) return (int)e;
    if (label_u8) mdv_launch(loss_sums_kernel<uint8_t>, dim3(grid_for(n)), dim3(256), 0, st, out, aux, (const uint8_t*)label, (double*)sums, n);
    else mdv_launch(loss_sums_kernel<float>, dim3(grid_for(n)), dim3(256), 0, st, out, aux, (const float*)label, (double*)sums, n);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_loss_finalize(const void* sums, double n_total, float* losses, void* stream) {
    if (!sums || !losses) return MDV_ERR_ARG;
    mdv_launch(loss_finalize_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, (const double*)sums, n_total, losses);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_loss_bwd(const float* out, const float* aux, const void* label, int label_u8, const void* sums, double n_total,
                            const float* coef, float* dout, float* daux, long long n, void* stream) {
    if (!out || !label || !sums || !coef || !dout || (aux && !daux)) return MDV_ERR_ARG;
    if (label_u8)
        mdv_launch(loss_bwd_kernel<uint8_t>, dim3(grid_for(n)), dim3(256), 0, (cudaStream_t)stream, out, aux, (const uint8_t*)label, (const double*)sums, n_total, coef, dout, daux, n);
    else
        mdv_launch(loss_bwd_kernel<float>, dim3(grid_for(n)), dim3(256), 0, (cudaStream_t)stream, out, aux, (const float*)label, (const double*)sums, n_total, coef, dout, daux, n);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_seg_counts(const float* logits, const void* label, int label_u8, void* counts, long long n, void* stream) {
    if (!logits || !label || !counts || n <= 0) return MDV_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (label_u8) mdv_launch(seg_counts_kernel<uint8_t>, dim3(grid_for(n)), dim3(256), 0, st, logits, (const uint8_t*)label, (unsigned long long*)counts, n);
    else mdv_launch(seg_counts_kernel<float>, dim3(grid_for(n)), dim3(256), 0, st, logits, (const float*)label, (unsigned long long*)counts, n);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_adamw(float* p, const float* g, float* m, float* v, void* hyper_, long long n, void* stream) {
    double* hyper = (double*)hyper_;
    if (!p || !g || !m || !v || !hyper || n <= 0) return MDV_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15)
        return MDV_ERR_ARG;
    mdv_launch(adamw_tick_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, hyper);
    MDV_CHECK_LAUNCH();
    mdv_launch(adamw_kernel, dim3(grid_for((n + 3) / 4)), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, (const double*)hyper, n);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_rng_bump(void* rng, void* stream) {
    if (!rng) return MDV_ERR_ARG;
    mdv_launch(rng_bump_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, (unsigned long long*)rng);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_droppath_scale(float* scale, int B, float p, const void* rng, uint32_t drop_stream, void* stream) {
    if (!scale || B <= 0 || p < 0.f || p >= 1.f) return MDV_ERR_ARG;
    mdv_launch(droppath_scale_kernel, dim3(mdv_cdiv(B, 128)), dim3(128), 0, (cudaStream_t)stream, scale, B, p, (const unsigned long long*)rng, drop_stream);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}
