// LayerNorm (token-wise) and BatchNorm (channel-wise, train + eval) kernels — HBM-bound, warp-shuffle reduced.
// LayerNorm: reference mdvit.py:349,357 (nn.LayerNorm eps=1e-6).  BatchNorm2d (+Hardswish/ReLU): mpvit.py:119-122,
// mdvit.py:120-121,559-563, Decoders.py:60-61,306-307.
#include "../../include/mdvit_b200.h"
#include "common.cuh"

#include <initializer_list>

namespace {

constexpr int LN_MAXV = 8;  // float2 per lane -> C <= 512

// ---------------------------------------------------------------------------------- LayerNorm forward
// one warp owns R rows per iteration (all loads issued before any arithmetic: at C = 64 a row is only 256 B, and one
// row per warp leaves HBM latency exposed); a row lives in registers, NV float2 per lane.
// blockIdx.y is the row group (M rows); its gamma / beta are gtab.p[blockIdx.y] / btab.p[blockIdx.y].  With a sample_set
// (per-sample sets, one group) row `row` uses gtab.p[s] / btab.p[s], s = sample_set[row / rows_per_sample]; an s outside
// [0, nsets) reads no table entry and the row is written as NaN.  mean_out / rstd_out may be NULL.
template <int NV, int R>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, const __grid_constant__ MdvPtrTable gtab,
                                                      const __grid_constant__ MdvPtrTable btab, float eps, bf16* __restrict__ y,
                                                      float* __restrict__ mean_out, float* __restrict__ rstd_out, int M,
                                                      const int* __restrict__ sample_set, int rows_per_sample, int nsets) {
    MDV_PDL_SYNC();
    constexpr int C = NV * 64;
    const int lane = threadIdx.x & 31;
    const int lo = blockIdx.y * M, hi = lo + M;
    const int row0 = lo + (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * R;
    if (row0 >= hi) return;
    float2 v[R][NV];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const bool ok = row0 + r < hi;
        const float* xr = x + (size_t)(ok ? row0 + r : row0) * C;
#pragma unroll
        for (int i = 0; i < NV; ++i) v[r][i] = *reinterpret_cast<const float2*>(xr + i * 64 + lane * 2);
    }
    // the set of the parameters in g / b: the row group, or (per-sample sets) the set of the warp's first row; a row of
    // another sample reloads them (-1: an out-of-range index, whose row reads no table entry)
    auto set_of = [&](int row) {
        const int k = __ldg(sample_set + row / rows_per_sample);
        return (unsigned)k < (unsigned)nsets ? k : -1;
    };
    int kcur = sample_set ? set_of(row0) : (int)blockIdx.y;
    float2 g[NV], b[NV];
    auto load_set = [&](int k) {
        const float* __restrict__ gamma = (const float*)gtab.p[k];
        const float* __restrict__ beta = (const float*)btab.p[k];
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            g[i] = *reinterpret_cast<const float2*>(gamma + i * 64 + lane * 2);
            b[i] = *reinterpret_cast<const float2*>(beta + i * 64 + lane * 2);
        }
    };
    if (kcur >= 0) load_set(kcur);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int row = row0 + r;
        if (row >= hi) break;
        if (sample_set && r > 0) {
            const int k = set_of(row);
            if (k != kcur && k >= 0) load_set(k);
            kcur = k;
        }
        const bool bad = kcur < 0;
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) s += v[r][i].x + v[r][i].y;
        const float mean = warp_sum(s) * (1.f / C);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const float a0 = v[r][i].x - mean, a1 = v[r][i].y - mean;
            q += a0 * a0 + a1 * a1;
        }
        const float rstd = rsqrtf(warp_sum(q) * (1.f / C) + eps);
        bf16* yr = y + (size_t)row * C;
#pragma unroll
        for (int i = 0; i < NV; ++i)
            *reinterpret_cast<uint32_t*>(yr + i * 64 + lane * 2) =
                bad ? 0x7fc07fc0u : f2_to_bf2((v[r][i].x - mean) * rstd * g[i].x + b[i].x, (v[r][i].y - mean) * rstd * g[i].y + b[i].y);
        if (lane == 0 && mean_out) {
            mean_out[row] = mean;
            rstd_out[row] = rstd;
        }
    }
}

// ---------------------------------------------------------------------------------- LayerNorm backward
// dx = dres + rstd * (gy - mean(gy) - xhat * mean(gy*xhat)),  gy = dy*gamma;  dgamma += sum dy*xhat; dbeta += sum dy.
// Optional dx_masked = bf16(dx * rowscale[row / rows_per_scale] * dropout_mask) feeds the previous Linear's dgrad/wgrad,
// and its column sums (that Linear's bias gradient) are accumulated into dbias_masked.
// One warp owns R rows per iteration (all of their loads are issued before any arithmetic: with C = 64 a row is only
// 256 B, so a single row per warp leaves HBM latency exposed); a row lives in registers, NV float2 per lane.
// blockIdx.y is the row group (M rows) and gamma, dgamma, dbeta come from the tables — a block never crosses a group boundary,
// so its column partials belong to one group's dgamma / dbeta.
template <int NV, int R>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                      const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                                                      const __grid_constant__ MdvPtrTable gtab, const float* __restrict__ dres,
                                                      float* __restrict__ dx, bf16* __restrict__ dx_masked,
                                                      const float* __restrict__ rowscale, int rows_per_scale, float drop_p,
                                                      const unsigned long long* __restrict__ rng, uint32_t drop_stream,
                                                      const __grid_constant__ MdvPtrTable dgtab, const __grid_constant__ MdvPtrTable dbtab,
                                                      float* __restrict__ dbias_masked, int M) {
    MDV_PDL_SYNC();
    constexpr int C = NV * 64;
    __shared__ float red[8][64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int lo = blockIdx.y * M, hi = lo + M;
    const float* __restrict__ gamma = (const float*)gtab.p[blockIdx.y];
    float* __restrict__ dgamma = (float*)dgtab.p[blockIdx.y];
    float* __restrict__ dbeta = (float*)dbtab.p[blockIdx.y];
    float2 ag[NV], ab[NV], am[NV], gm[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        ag[i] = make_float2(0.f, 0.f);
        ab[i] = make_float2(0.f, 0.f);
        am[i] = make_float2(0.f, 0.f);
        gm[i] = *reinterpret_cast<const float2*>(gamma + i * 64 + lane * 2);
    }
    uint32_t dthr = 0, dkey = 0;
    float dinv = 1.f;
    if (dx_masked && drop_p > 0.f) {
        dthr = drop_thresh(drop_p);
        dinv = 1.f / (1.f - drop_p);
        dkey = rng_key(rng, drop_stream);
    }
    for (int row0 = lo + (blockIdx.x * nwarp + warp) * R; row0 < hi; row0 += gridDim.x * nwarp * R) {
        float2 d[R][NV], xh[R][NV], rr[R][NV];
        float mean[R], rstd[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int row = row0 + r;
            const bool ok = row < hi;
            const size_t off = (size_t)(ok ? row : 0) * C;
            mean[r] = ok ? mean_in[row] : 0.f;
            rstd[r] = ok ? rstd_in[row] : 0.f;
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int c = i * 64 + lane * 2;
                d[r][i] = ok ? *reinterpret_cast<const float2*>(dy + off + c) : make_float2(0.f, 0.f);
                xh[r][i] = ok ? *reinterpret_cast<const float2*>(x + off + c) : make_float2(0.f, 0.f);
                rr[r][i] = (ok && dres) ? *reinterpret_cast<const float2*>(dres + off + c) : make_float2(0.f, 0.f);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int row = row0 + r;
            if (row >= hi) break;
            const size_t off = (size_t)row * C;
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                xh[r][i] = make_float2((xh[r][i].x - mean[r]) * rstd[r], (xh[r][i].y - mean[r]) * rstd[r]);
                ag[i].x += d[r][i].x * xh[r][i].x;
                ag[i].y += d[r][i].y * xh[r][i].y;
                ab[i].x += d[r][i].x;
                ab[i].y += d[r][i].y;
                d[r][i].x *= gm[i].x;
                d[r][i].y *= gm[i].y;
                s1 += d[r][i].x + d[r][i].y;
                s2 += d[r][i].x * xh[r][i].x + d[r][i].y * xh[r][i].y;
            }
            s1 = warp_sum(s1) * (1.f / C);
            s2 = warp_sum(s2) * (1.f / C);
            const float rs = rowscale ? rowscale[row / rows_per_scale] : 1.f;
#pragma unroll
            for (int i = 0; i < NV; ++i) {
                const int c = i * 64 + lane * 2;
                const float o0 = rstd[r] * (d[r][i].x - s1 - xh[r][i].x * s2) + rr[r][i].x;
                const float o1 = rstd[r] * (d[r][i].y - s1 - xh[r][i].y * s2) + rr[r][i].y;
                *reinterpret_cast<float2*>(dx + off + c) = make_float2(o0, o1);
                if (dx_masked) {
                    float m0 = rs, m1 = rs;
                    if (dthr) {
                        const uint32_t h = drop_hash(dkey, (uint32_t)((off + c) >> 1));   // off + c is even
                        m0 *= drop_lo(h, dthr, dinv);
                        m1 *= drop_hi(h, dthr, dinv);
                    }
                    m0 *= o0;
                    m1 *= o1;
                    am[i].x += m0;
                    am[i].y += m1;
                    *reinterpret_cast<uint32_t*>(dx_masked + off + c) = f2_to_bf2(m0, m1);
                }
            }
        }
    }
    // column reductions across the block's warps, then one atomic per column per block
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        for (int pass = 0; pass < 3; ++pass) {
            float* base = pass == 0 ? dgamma : (pass == 1 ? dbeta : dbias_masked);
            if (!base) continue;   // block-uniform
            const float2 val = pass == 0 ? ag[i] : (pass == 1 ? ab[i] : am[i]);
            __syncthreads();
            red[warp][lane * 2] = val.x;
            red[warp][lane * 2 + 1] = val.y;
            __syncthreads();
            if (warp == 0) {
                float t0 = 0.f, t1 = 0.f;
                for (int w = 0; w < nwarp; ++w) {
                    t0 += red[w][lane * 2];
                    t1 += red[w][lane * 2 + 1];
                }
                float* dst = base + i * 64 + lane * 2;
                atomicAdd(dst, t0);
                atomicAdd(dst + 1, t1);
            }
        }
    }
}

// ---------------------------------------------------------------------------------- BatchNorm
__device__ __forceinline__ float act_fwd(float v, int act) {
    if (act == MDV_ACT_RELU) return fmaxf(v, 0.f);
    if (act == MDV_ACT_HSWISH) return hardswish_f(v);
    return v;
}
__device__ __forceinline__ float act_bwd(float v, int act) {
    if (act == MDV_ACT_RELU) return v > 0.f ? 1.f : 0.f;
    if (act == MDV_ACT_HSWISH) return hardswish_grad(v);
    return 1.f;
}

// eval: mean/rstd from the running buffers
__global__ void bn_eval_stats_kernel(const float* __restrict__ running_mean, const float* __restrict__ running_var, float eps,
                                     float* __restrict__ mean, float* __restrict__ rstd, int C) {
    MDV_PDL_SYNC();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    mean[c] = running_mean[c];
    rstd[c] = rsqrtf(running_var[c] + eps);
}

template <typename TO>
__global__ void __launch_bounds__(256) bn_act_fwd_kernel(const float* __restrict__ z, const float* __restrict__ mean,
                                                          const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, int act, TO* __restrict__ y,
                                                          int total, int C) {
    MDV_PDL_SYNC();
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;      // 32-bit: the host checks M*C < 2^31
    if (i >= total) return;
    const int c = i % C;
    float4 v = *reinterpret_cast<const float4*>(z + i);
    float o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int cc = c + j;
        o[j] = act_fwd((o[j] - __ldg(mean + cc)) * __ldg(rstd + cc) * __ldg(gamma + cc) + __ldg(beta + cc), act);
    }
    if (sizeof(TO) == 4) {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + i) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
        uint2 pk = make_uint2(f2_to_bf2(o[0], o[1]), f2_to_bf2(o[2], o[3]));
        *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(y) + i) = pk;
    }
}

// Rank-1 output gradient (the commuted 1-channel head, Decoders.py:334-337): dy[m,c] = dlog[m] * wrow[c] * dropout2d_mask(m / rps, c)
// is generated on the fly instead of being materialised as an [M, C] fp32 tensor.
struct Rank1Dy {
    const float* dlog;      // [M] or NULL (then the dense dy is used)
    const float* wrow;      // [C]
    const unsigned long long* rng;
    int rps;                // rows per sample
    float drop_p;
    uint32_t stream;
    const float* wtab;      // [samples, C] = wrow[c] * dropout2d_mask(b, c), precomputed once per call (vectorised kernels)
};

// ------------------------------------------------------------------------------------------------ train-mode BatchNorm
// The fused multi-domain forward stacks G single-domain mini-batches along the rows; BatchNorm statistics are per group of
// Mg consecutive rows (one reference forward each).  These kernels handle all groups in ONE launch (grid.z = group) with
// float4 loads and 4 rows in flight per thread; a single BatchNorm call is the case G = 1.  Group g's gamma / beta are
// gt.p[g] / bt.p[g]: one parameter set repeated G times, or one set per group (domain-specific norms).
// Thread layout: C/4 threads per row (one float4 of channels each), RPI = 256 / (C/4) rows per block iteration.
// (b*C + c) is a multiple of 4: two pair-hashes give the four Dropout2d masks of a float4 of channels
__device__ __forceinline__ float4 rank1_w4(const Rank1Dy& r1, int b, int c, int C) {
    float4 w = *reinterpret_cast<const float4*>(r1.wrow + c);
    if (r1.drop_p > 0.f) {
        const uint32_t key = rng_key(r1.rng, r1.stream), thr = drop_thresh(r1.drop_p);
        const float inv = 1.f / (1.f - r1.drop_p);
        const uint32_t pr = (uint32_t)(b * C + c) >> 1;
        const uint32_t h0 = drop_hash(key, pr), h1 = drop_hash(key, pr + 1);
        w.x *= drop_lo(h0, thr, inv); w.y *= drop_hi(h0, thr, inv); w.z *= drop_lo(h1, thr, inv); w.w *= drop_hi(h1, thr, inv);
    }
    return w;
}

__global__ void rank1_table_kernel(Rank1Dy r1, float* __restrict__ wtab, int samples, int C) {
    MDV_PDL_SYNC();
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= samples * C) return;
    *reinterpret_cast<float4*>(wtab + i) = rank1_w4(r1, i / C, i % C, C);
}

template <bool BWD, bool RANK1 = false>
__global__ void __launch_bounds__(256) bn_reduce_g_kernel(const float* __restrict__ a, const float* __restrict__ z,
                                                           const float* __restrict__ mean, const float* __restrict__ rstd, int act,
                                                           double* __restrict__ sums, int Mg, int C, int rows_per_block,
                                                           Rank1Dy rk, const __grid_constant__ MdvPtrTable gt, const __grid_constant__ MdvPtrTable bt) {
    MDV_PDL_SYNC();
    __shared__ float4 sh[2][256];
    const int tpr = C >> 2;                       // threads per row
    const int rpi = 256 / tpr;                    // rows per block iteration
    const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr;
    const int g = blockIdx.z;
    const float* __restrict__ gamma = (const float*)gt.p[g];
    const float* __restrict__ beta = (const float*)bt.p[g];
    const int r0 = blockIdx.x * rows_per_block, r1 = min(Mg, r0 + rows_per_block);
    const size_t base = (size_t)g * Mg * C;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
    if (rl < rpi) {
        float4 mu = s, rs = s, ga = s, be = s;
        if (BWD) {
            mu = *reinterpret_cast<const float4*>(mean + (size_t)g * C + 4 * cl);
            rs = *reinterpret_cast<const float4*>(rstd + (size_t)g * C + 4 * cl);
            ga = *reinterpret_cast<const float4*>(gamma + 4 * cl);
            be = *reinterpret_cast<const float4*>(beta + 4 * cl);
        }
        constexpr int U = 4;
        int cur_b = -1;
        float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = r0 + rl; r < r1; r += rpi * U) {
            float4 zv[U], dv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int rr = r + u * rpi;
                const bool ok = rr < r1;
                const size_t o = base + (size_t)rr * C + 4 * cl;
                zv[u] = ok ? *reinterpret_cast<const float4*>(z + o) : make_float4(0.f, 0.f, 0.f, 0.f);
                if (BWD && !RANK1) dv[u] = ok ? *reinterpret_cast<const float4*>(a + o) : make_float4(0.f, 0.f, 0.f, 0.f);
                if (BWD && RANK1) {
                    // dy[m, c] = dlog[m] * wrow[c] * dropout2d_mask(m / rps, c), generated on the fly (G == 1)
                    dv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ok) {
                        const int bb = rr / rk.rps;
                        if (bb != cur_b) {
                            cur_b = bb;
                            wm = *reinterpret_cast<const float4*>(rk.wtab + (size_t)bb * C + 4 * cl);
                        }
                        const float dl = __ldg(rk.dlog + rr);
                        dv[u] = make_float4(dl * wm.x, dl * wm.y, dl * wm.z, dl * wm.w);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (r + u * rpi >= r1) break;
                if (!BWD) {
                    s.x += zv[u].x; s.y += zv[u].y; s.z += zv[u].z; s.w += zv[u].w;
                    q.x += zv[u].x * zv[u].x; q.y += zv[u].y * zv[u].y; q.z += zv[u].z * zv[u].z; q.w += zv[u].w * zv[u].w;
                } else {
                    const float xh0 = (zv[u].x - mu.x) * rs.x, xh1 = (zv[u].y - mu.y) * rs.y, xh2 = (zv[u].z - mu.z) * rs.z,
                                xh3 = (zv[u].w - mu.w) * rs.w;
                    const float g0 = dv[u].x * act_bwd(xh0 * ga.x + be.x, act), g1 = dv[u].y * act_bwd(xh1 * ga.y + be.y, act),
                                g2 = dv[u].z * act_bwd(xh2 * ga.z + be.z, act), g3 = dv[u].w * act_bwd(xh3 * ga.w + be.w, act);
                    s.x += g0; s.y += g1; s.z += g2; s.w += g3;
                    q.x += g0 * xh0; q.y += g1 * xh1; q.z += g2 * xh2; q.w += g3 * xh3;
                }
            }
        }
    }
    sh[0][threadIdx.x] = s;
    sh[1][threadIdx.x] = q;
    __syncthreads();
    for (int tid = threadIdx.x; tid < 2 * tpr; tid += 256) {
        const int which = tid / tpr, c4 = tid % tpr;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int i = 0; i < rpi; ++i) {
            const float4 v = sh[which][i * tpr + c4];
            t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
        }
        double* dst = sums + (size_t)g * 2 * C + which * C + 4 * c4;
        atomicAdd(dst, (double)t.x);
        atomicAdd(dst + 1, (double)t.y);
        atomicAdd(dst + 2, (double)t.z);
        atomicAdd(dst + 3, (double)t.w);
    }
}

// y = act(gamma (z - mean) rstd + beta): row-walking like the backward apply kernel (parameters once per thread, 4 rows in flight)
template <typename TO>
__global__ void __launch_bounds__(256) bn_act_fwd_g_kernel(const float* __restrict__ z, const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, int act, TO* __restrict__ y, int Mg,
                                                            int C, int rows_per_block, const __grid_constant__ MdvPtrTable gt, const __grid_constant__ MdvPtrTable bt) {
    MDV_PDL_SYNC();
    const int tpr = C >> 2, rpi = 256 / tpr;
    const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr;
    if (rl >= rpi) return;
    const int g = blockIdx.z, c = 4 * cl;
    const float* __restrict__ gamma = (const float*)gt.p[g];
    const float* __restrict__ beta = (const float*)bt.p[g];
    const int r0 = blockIdx.x * rows_per_block, r1e = min(Mg, r0 + rows_per_block);
    const size_t base = (size_t)g * Mg * C;
    const float4 mu = *reinterpret_cast<const float4*>(mean + (size_t)g * C + c), rs = *reinterpret_cast<const float4*>(rstd + (size_t)g * C + c);
    const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
    // y = z * a + b with a = gamma rstd, b = beta - mean a
    const float4 sa = make_float4(rs.x * ga.x, rs.y * ga.y, rs.z * ga.z, rs.w * ga.w);
    constexpr int U = 4;
    for (int r = r0 + rl; r < r1e; r += rpi * U) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int rr = r + u * rpi;
            v[u] = rr < r1e ? *reinterpret_cast<const float4*>(z + base + (size_t)rr * C + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int rr = r + u * rpi;
            if (rr >= r1e) break;
            const float o0 = act_fwd((v[u].x - mu.x) * sa.x + be.x, act), o1 = act_fwd((v[u].y - mu.y) * sa.y + be.y, act),
                        o2 = act_fwd((v[u].z - mu.z) * sa.z + be.z, act), o3 = act_fwd((v[u].w - mu.w) * sa.w + be.w, act);
            const size_t o = base + (size_t)rr * C + c;
            if (sizeof(TO) == 4) *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + o) = make_float4(o0, o1, o2, o3);
            else *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(y) + o) = make_uint2(f2_to_bf2(o0, o1), f2_to_bf2(o2, o3));
        }
    }
}

// Train-mode statistics of G groups; group g updates the running buffers of table entry g (one nn.BatchNorm2d step).  The thread of
// channel c walks the groups in order, so groups that name the same buffers update them in group order, exactly as consecutive
// nn.BatchNorm2d forwards would (the momentum update does not commute).
__global__ void bn_finalize_kernel(const double* __restrict__ sums, int G, int Mg, int C, float eps, float momentum, const __grid_constant__ MdvPtrTable rmt,
                                      const __grid_constant__ MdvPtrTable rvt, const __grid_constant__ MdvPtrTable nbt, float* __restrict__ mean, float* __restrict__ rstd) {
    MDV_PDL_SYNC();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0)
        for (int g = 0; g < G; ++g)
            if (nbt.p[g]) *(long long*)nbt.p[g] += 1;
    if (c >= C) return;
    float rm = 0.f, rv = 0.f;
    for (int g = 0; g < G; ++g) {
        const double mu = sums[(size_t)g * 2 * C + c] / Mg;
        double var = sums[(size_t)g * 2 * C + C + c] / Mg - mu * mu;
        if (var < 0) var = 0;
        mean[(size_t)g * C + c] = (float)mu;
        rstd[(size_t)g * C + c] = (float)(1.0 / sqrt(var + (double)eps));
        // a run of consecutive groups naming the same buffer updates it in a register: one load and one store per run
        float* rmp = (float*)rmt.p[g];
        float* rvp = (float*)rvt.p[g];
        if (rmp) {
            if (g == 0 || rmt.p[g - 1] != rmp) rm = rmp[c];
            rm = (1.f - momentum) * rm + momentum * (float)mu;
            if (g + 1 == G || rmt.p[g + 1] != rmp) rmp[c] = rm;
        }
        if (rvp) {
            if (g == 0 || rvt.p[g - 1] != rvp) rv = rvp[c];
            const double unb = Mg > 1 ? var * Mg / (Mg - 1) : var;
            rv = (1.f - momentum) * rv + momentum * (float)unb;
            if (g + 1 == G || rvt.p[g + 1] != rvp) rvp[c] = rv;
        }
    }
}

// coef[g][c] = sum_g / Mg, coef[g][C+c] = sum_gxhat / Mg;  dgamma[g] += group g's sum_gxhat, dbeta[g] += its sum_g.  Consecutive
// groups that name the same target are summed in double and added with one atomic: one set repeated G times gets the sum over
// all groups added once.
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ sums, int G, int Mg, int C, float* __restrict__ coef,
                                       const __grid_constant__ MdvPtrTable dgt, const __grid_constant__ MdvPtrTable dbt) {
    MDV_PDL_SYNC();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double sg = 0.0, sq = 0.0;
    for (int g = 0; g < G; ++g) {
        const double a = sums[(size_t)g * 2 * C + c], b = sums[(size_t)g * 2 * C + C + c];
        coef[(size_t)g * 2 * C + c] = (float)(a / Mg);
        coef[(size_t)g * 2 * C + C + c] = (float)(b / Mg);
        sg += a;
        sq += b;
        const bool last = g + 1 == G;
        if (last || dbt.p[g + 1] != dbt.p[g]) {
            if (dbt.p[g]) atomicAdd((float*)dbt.p[g] + c, (float)sg);
            sg = 0.0;
        }
        if (last || dgt.p[g + 1] != dgt.p[g]) {
            if (dgt.p[g]) atomicAdd((float*)dgt.p[g] + c, (float)sq);
            sq = 0.0;
        }
    }
}

// dz = gamma rstd (g - c0 - xhat c1), g = dy act'(.).  Same thread mapping as bn_reduce_g_kernel: a thread owns 4 channels and walks
// the rows of its block's band, 4 rows in flight — the per-channel parameters (7 float4) are loaded once instead of once per 16
// bytes of z, and there is no index arithmetic per element.
template <typename TO, bool RANK1 = false>
__global__ void __launch_bounds__(256) bn_bwd_apply_g_kernel(const float* __restrict__ dy, const float* __restrict__ z,
                                                              const float* __restrict__ mean, const float* __restrict__ rstd, int act,
                                                              const float* __restrict__ coef, TO* __restrict__ dz, int Mg, int C,
                                                              int rows_per_block, Rank1Dy r1, const __grid_constant__ MdvPtrTable gt, const __grid_constant__ MdvPtrTable bt) {
    MDV_PDL_SYNC();
    const int tpr = C >> 2;                       // threads per row
    const int rpi = 256 / tpr;                    // rows per block iteration
    const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr;
    if (rl >= rpi) return;
    const int g = blockIdx.z;
    const float* __restrict__ gamma = (const float*)gt.p[g];
    const float* __restrict__ beta = (const float*)bt.p[g];
    const int r0 = blockIdx.x * rows_per_block, r1e = min(Mg, r0 + rows_per_block);
    const size_t base = (size_t)g * Mg * C;
    const int c = 4 * cl;
    const float4 mu = *reinterpret_cast<const float4*>(mean + (size_t)g * C + c), rs = *reinterpret_cast<const float4*>(rstd + (size_t)g * C + c);
    const float4 ga = *reinterpret_cast<const float4*>(gamma + c), be = *reinterpret_cast<const float4*>(beta + c);
    const float4 k0 = *reinterpret_cast<const float4*>(coef + (size_t)g * 2 * C + c), k1 = *reinterpret_cast<const float4*>(coef + (size_t)g * 2 * C + C + c);
    const float m4[4] = {mu.x, mu.y, mu.z, mu.w}, r4[4] = {rs.x, rs.y, rs.z, rs.w}, g4[4] = {ga.x, ga.y, ga.z, ga.w},
                b4[4] = {be.x, be.y, be.z, be.w}, c0[4] = {k0.x, k0.y, k0.z, k0.w}, c1[4] = {k1.x, k1.y, k1.z, k1.w};
    constexpr int U = 4;
    int cur_b = -1;
    float4 wm = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = r0 + rl; r < r1e; r += rpi * U) {
        float4 zv[U], dv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int rr = r + u * rpi;
            const bool ok = rr < r1e;
            const size_t o = base + (size_t)rr * C + c;
            zv[u] = ok ? *reinterpret_cast<const float4*>(z + o) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (!RANK1) {
                dv[u] = ok ? *reinterpret_cast<const float4*>(dy + o) : make_float4(0.f, 0.f, 0.f, 0.f);
            } else {
                dv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok) {      // dy[m, c] = dlog[m] * wrow[c] * dropout2d_mask(m / rps, c), from the per-sample factor table (G == 1)
                    const int bb = rr / r1.rps;
                    if (bb != cur_b) {
                        cur_b = bb;
                        wm = *reinterpret_cast<const float4*>(r1.wtab + (size_t)bb * C + c);
                    }
                    const float dl = __ldg(r1.dlog + rr);
                    dv[u] = make_float4(dl * wm.x, dl * wm.y, dl * wm.z, dl * wm.w);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int rr = r + u * rpi;
            if (rr >= r1e) break;
            const float zz[4] = {zv[u].x, zv[u].y, zv[u].z, zv[u].w}, dd[4] = {dv[u].x, dv[u].y, dv[u].z, dv[u].w};
            float o4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float xh = (zz[j] - m4[j]) * r4[j];
                const float gg = dd[j] * act_bwd(xh * g4[j] + b4[j], act);
                o4[j] = g4[j] * r4[j] * (gg - c0[j] - xh * c1[j]);
            }
            const size_t o = base + (size_t)rr * C + c;
            if (sizeof(TO) == 4) *reinterpret_cast<float4*>(reinterpret_cast<float*>(dz) + o) = make_float4(o4[0], o4[1], o4[2], o4[3]);
            else *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(dz) + o) = make_uint2(f2_to_bf2(o4[0], o4[1]), f2_to_bf2(o4[2], o4[3]));
        }
    }
}

int grouped_rows_per_block(int Mg, int C, int G) {
    const int rpi = 256 / (C / 4);
    int want = (6 * MDV_NUM_SMS) / G;                     // ~6 blocks per SM over all groups
    if (want < 1) want = 1;
    int rpb = mdv_cdiv(Mg, want);
    const int minr = rpi * 16;
    if (rpb < minr) rpb = minr;
    return rpb;
}

// streaming apply pass: ~16 blocks per SM over all groups, at least 4 iterations of 4 rows per thread
int apply_rows_per_block(int Mg, int C, int G) {
    const int rpi = 256 / (C / 4);
    int want = (16 * MDV_NUM_SMS) / G;
    if (want < 1) want = 1;
    int rpb = mdv_cdiv(Mg, want);
    const int minr = rpi * 16;
    if (rpb < minr) rpb = minr;
    return rpb;
}

}  // namespace

// Rows per warp iteration by width: C = 64 * NV.
#define MDV_LN_DISPATCH(X)      \
    switch (C >> 6) {           \
        case 1: X(1, 4)         \
        case 2: X(2, 4)         \
        case 3: X(3, 2)         \
        case 4: X(4, 2)         \
        case 5: X(5, 2)         \
        case 6: X(6, 1)         \
        case 7: X(7, 1)         \
        default: X(8, 1)        \
    }

// sample_set != NULL: per-sample sets (G = 1, nsets table entries); else row group g of G uses table entry g
static int ln_fwd_launch(const float* x, MdvPtrTable gt, MdvPtrTable bt, float eps, void* y_bf16, float* mean, float* rstd, int G, int Mg,
                         int C, cudaStream_t st, const int* sample_set = nullptr, int rows_per_sample = 1, int nsets = 0) {
#define MDV_LN_FWD(NV, R)                                                                                                        \
    mdv_launch((ln_fwd_kernel<NV, R>), dim3(mdv_cdiv(Mg, 8 * R), G), dim3(256), 0, st, x, gt, bt, eps, (bf16*)y_bf16, mean, rstd, Mg, \
               sample_set, rows_per_sample, nsets);                                                                             \
    break;
    MDV_LN_DISPATCH(MDV_LN_FWD)
#undef MDV_LN_FWD
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

static int ln_bwd_launch(const float* dy, const float* x, const float* mean, const float* rstd, MdvPtrTable gt, const float* dres, float* dx,
                         void* dx_masked_bf16, const float* rowscale, int rows_per_scale, float drop_p, const void* rng, uint32_t drop_stream,
                         MdvPtrTable dgt, MdvPtrTable dbt, float* dbias_masked, int G, int Mg, int C, cudaStream_t st) {
    const int rps = rows_per_scale > 0 ? rows_per_scale : 1;
    const int max_blocks = (4 * MDV_NUM_SMS + G - 1) / G;      // ~4 blocks per SM over all groups
#define MDV_LN_BWD(NV, R)                                                                                                        \
    {                                                                                                                            \
        int blocks = mdv_cdiv(Mg, 8 * R);                                                                                        \
        if (blocks > max_blocks) blocks = max_blocks;                                                                            \
        mdv_launch((ln_bwd_kernel<NV, R>), dim3(blocks, G), dim3(256), 0, st, dy, x, mean, rstd, gt, dres, dx, (bf16*)dx_masked_bf16, \
                   rowscale, rps, drop_p, (const unsigned long long*)rng, drop_stream, dgt, dbt, dbias_masked, Mg);              \
    }                                                                                                                            \
    break;
    MDV_LN_DISPATCH(MDV_LN_BWD)
#undef MDV_LN_BWD
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

// The table of the single-set entry points: one parameter set, G = 1.
static MdvPtrTable one_set(const void* p) {
    MdvPtrTable t = MdvPtrTable();
    t.p[0] = const_cast<void*>(p);
    return t;
}

static bool tables_set(int G, std::initializer_list<const MdvPtrTable*> tabs) {
    for (const MdvPtrTable* t : tabs)
        for (int g = 0; g < G; ++g)
            if (!t->p[g]) return false;
    return true;
}

static bool ln_shape_ok(int M, int C) { return M > 0 && !(C & 63) && C <= 64 * LN_MAXV; }

extern "C" int mdv_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y_bf16, float* mean,
                                 float* rstd, int M, int C, void* stream) {
    if (!x || !y_bf16 || !gamma || !beta || !ln_shape_ok(M, C)) return MDV_ERR_ARG;
    return ln_fwd_launch(x, one_set(gamma), one_set(beta), eps, y_bf16, mean, rstd, 1, M, C, (cudaStream_t)stream);
}

extern "C" int mdv_layernorm_fwd_gp(const float* x, MdvPtrTable gamma, MdvPtrTable beta, float eps, void* y_bf16, float* mean, float* rstd,
                                    int G, int Mg, int C, void* stream) {
    if (G < 1 || G > MDV_MAX_GROUPS || !x || !y_bf16 || !mean || !rstd || !ln_shape_ok(Mg, C)) return MDV_ERR_ARG;
    if (!tables_set(G, {&gamma, &beta}) || (long long)G * Mg >= 0x7fffffffLL) return MDV_ERR_ARG;
    return ln_fwd_launch(x, gamma, beta, eps, y_bf16, mean, rstd, G, Mg, C, (cudaStream_t)stream);
}

extern "C" int mdv_layernorm_fwd_sets(const float* x, MdvPtrTable gamma, MdvPtrTable beta, float eps, void* y_bf16, float* mean, float* rstd,
                                      const int* sample_set, int rows_per_sample, int S, int M, int C, void* stream) {
    if (S < 1 || S > MDV_MAX_GROUPS || !x || !y_bf16 || !sample_set || rows_per_sample < 1 || !ln_shape_ok(M, C)) return MDV_ERR_ARG;
    if (!tables_set(S, {&gamma, &beta})) return MDV_ERR_ARG;
    return ln_fwd_launch(x, gamma, beta, eps, y_bf16, mean, rstd, 1, M, C, (cudaStream_t)stream, sample_set, rows_per_sample, S);
}

extern "C" int mdv_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                                 const float* dres, float* dx, void* dx_masked_bf16, const float* rowscale,
                                 int rows_per_scale, float drop_p, const void* rng, uint32_t drop_stream, float* dgamma,
                                 float* dbeta, float* dbias_masked, int M, int C, void* stream) {
    if (!dy || !x || !dx || !gamma || !ln_shape_ok(M, C)) return MDV_ERR_ARG;
    if (dbias_masked && !dx_masked_bf16) return MDV_ERR_ARG;
    return ln_bwd_launch(dy, x, mean, rstd, one_set(gamma), dres, dx, dx_masked_bf16, rowscale, rows_per_scale, drop_p, rng, drop_stream,
                         one_set(dgamma), one_set(dbeta), dbias_masked, 1, M, C, (cudaStream_t)stream);
}

extern "C" int mdv_layernorm_bwd_gp(const float* dy, const float* x, const float* mean, const float* rstd, MdvPtrTable gamma,
                                    const float* dres, float* dx, void* dx_masked_bf16, const float* rowscale, int rows_per_scale,
                                    float drop_p, const void* rng, uint32_t drop_stream, MdvPtrTable dgamma, MdvPtrTable dbeta,
                                    float* dbias_masked, int G, int Mg, int C, void* stream) {
    if (G < 1 || G > MDV_MAX_GROUPS || !dy || !x || !mean || !rstd || !dx || !ln_shape_ok(Mg, C)) return MDV_ERR_ARG;
    if (dbias_masked && !dx_masked_bf16) return MDV_ERR_ARG;
    if (!tables_set(G, {&gamma}) || (long long)G * Mg >= 0x7fffffffLL) return MDV_ERR_ARG;
    return ln_bwd_launch(dy, x, mean, rstd, gamma, dres, dx, dx_masked_bf16, rowscale, rows_per_scale, drop_p, rng, drop_stream, dgamma, dbeta,
                         dbias_masked, G, Mg, C, (cudaStream_t)stream);
}

// ---- train-mode BatchNorm (+activation): one call = G consecutive nn.BatchNorm2d forwards on [G*Mg, C]
static bool bn_grouped_ok(int G, int Mg, int C) { return G >= 1 && Mg >= 1 && C >= 32 && C <= 1024 && (C & 3) == 0 && (long long)G * Mg * C < 0x7fffffffLL; }

// Batch statistics of the G row groups -> mean/rstd [G, C]; updates the running buffers of the tables.  ws: 2*C*G doubles.
static int bn_train_stats(const float* z, int G, int Mg, int C, float eps, float momentum, MdvPtrTable rmt, MdvPtrTable rvt, MdvPtrTable nbt,
                          float* mean, float* rstd, void* ws, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(ws, 0, sizeof(double) * 2 * C * G, st);
    if (e != cudaSuccess) return (int)e;
    const int rpb = grouped_rows_per_block(Mg, C, G);
    mdv_launch(bn_reduce_g_kernel<false>, dim3(mdv_cdiv(Mg, rpb), 1, G), dim3(256), 0, st, (const float*)nullptr, z, (const float*)nullptr,
               (const float*)nullptr, 0, (double*)ws, Mg, C, rpb, Rank1Dy(), MdvPtrTable(), MdvPtrTable());
    MDV_CHECK_LAUNCH();
    mdv_launch(bn_finalize_kernel, dim3(mdv_cdiv(C, 128)), dim3(128), 0, st, (const double*)ws, G, Mg, C, eps, momentum, rmt, rvt, nbt, mean, rstd);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

// ws: >= 2*C doubles (zeroed here).  Writes mean[C], rstd[C]; in training also updates the running buffers.
extern "C" int mdv_bn_stats(const float* z, int M, int C, float eps, float momentum, int training, float* running_mean,
                            float* running_var, long long* num_batches_tracked, float* mean, float* rstd, void* ws,
                            void* stream) {
    if (!mean || !rstd || M <= 0 || C <= 0) return MDV_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (training) {
        if (!z || !ws) return MDV_ERR_ARG;
        if (!bn_grouped_ok(1, M, C)) return MDV_ERR_UNSUPPORTED;
        return bn_train_stats(z, 1, M, C, eps, momentum, one_set(running_mean), one_set(running_var), one_set(num_batches_tracked), mean, rstd,
                              ws, st);
    }
    if (!running_mean || !running_var) return MDV_ERR_ARG;
    mdv_launch(bn_eval_stats_kernel, dim3(mdv_cdiv(C, 128)), dim3(128), 0, st, (const float*)running_mean, (const float*)running_var, eps, mean,
               rstd, C);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

// Eval-mode BatchNorm folds of S parameter sets (blockIdx.y = set): scale / shift are [S, C]; the conv bias is shared.
__global__ void bn_fold_kernel(const __grid_constant__ MdvPtrTable gt, const __grid_constant__ MdvPtrTable bt,
                               const __grid_constant__ MdvPtrTable rmt, const __grid_constant__ MdvPtrTable rvt,
                               const float* __restrict__ cbias, float eps, float* __restrict__ scale, float* __restrict__ shift, int C) {
    MDV_PDL_SYNC();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const int k = blockIdx.y;
    const float* __restrict__ gamma = (const float*)gt.p[k];
    const float* __restrict__ beta = (const float*)bt.p[k];
    const float* __restrict__ rm = (const float*)rmt.p[k];
    const float* __restrict__ rv = (const float*)rvt.p[k];
    const float s = gamma[c] * rsqrtf(rv[c] + eps);
    scale[(size_t)k * C + c] = s;
    shift[(size_t)k * C + c] = beta[c] + ((cbias ? cbias[c] : 0.f) - rm[c]) * s;
}

static int bn_fold_launch(MdvPtrTable gt, MdvPtrTable bt, MdvPtrTable rmt, MdvPtrTable rvt, const float* conv_bias, float eps, float* scale,
                          float* shift, int S, int C, cudaStream_t st) {
    mdv_launch(bn_fold_kernel, dim3(mdv_cdiv(C, 128), S), dim3(128), 0, st, gt, bt, rmt, rvt, conv_bias, eps, scale, shift, C);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                           const float* conv_bias, float eps, float* scale, float* shift, int C, void* stream) {
    if (!gamma || !beta || !running_mean || !running_var || !scale || !shift || C <= 0) return MDV_ERR_ARG;
    return bn_fold_launch(one_set(gamma), one_set(beta), one_set(running_mean), one_set(running_var), conv_bias, eps, scale, shift, 1, C,
                          (cudaStream_t)stream);
}

extern "C" int mdv_bn_fold_sets(MdvPtrTable gamma, MdvPtrTable beta, MdvPtrTable running_mean, MdvPtrTable running_var, const float* conv_bias,
                                float eps, float* scale, float* shift, int S, int C, void* stream) {
    if (S < 1 || S > MDV_MAX_GROUPS || !scale || !shift || C <= 0) return MDV_ERR_ARG;
    if (!tables_set(S, {&gamma, &beta, &running_mean, &running_var})) return MDV_ERR_ARG;
    return bn_fold_launch(gamma, beta, running_mean, running_var, conv_bias, eps, scale, shift, S, C, (cudaStream_t)stream);
}

extern "C" int mdv_bn_act_fwd(const float* z, const float* mean, const float* rstd, const float* gamma, const float* beta,
                              int act, void* y, int y_bf16, int M, int C, void* stream) {
    if (!z || !y || M <= 0 || (C & 3)) return MDV_ERR_ARG;
    if ((long long)M * C >= 0x7fffffffLL) return MDV_ERR_UNSUPPORTED;
    const int total = M * C;
    const int blocks = mdv_cdiv(total / 4, 256);
    if (y_bf16)
        mdv_launch(bn_act_fwd_kernel<bf16>, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, z, mean, rstd, gamma, beta, act, (bf16*)y, total, C);
    else
        mdv_launch(bn_act_fwd_kernel<float>, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, z, mean, rstd, gamma, beta, act, (float*)y, total, C);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

// dz for y = act(BN_train(z)) on G row groups; dgamma/dbeta accumulate through the tables.  With a rank-1 output gradient (r1.dlog,
// G == 1) the per-(sample, channel) factor wrow[c] * dropout2d mask is tabulated once.
// ws: 2*C*G doubles of sums, 2*C*G floats of coefficients, then (rank-1) the (Mg / rps) x C factor table.
static int bn_act_bwd_impl(const float* dy, const Rank1Dy& r1, const float* z, const float* mean, const float* rstd, MdvPtrTable gt,
                           MdvPtrTable bt, int act, void* dz, int dz_bf16, MdvPtrTable dgt, MdvPtrTable dbt, int G, int Mg, int C, void* ws,
                           cudaStream_t st) {
    double* sums = (double*)ws;
    float* coef = (float*)(sums + (size_t)2 * C * G);
    cudaError_t e = cudaMemsetAsync(ws, 0, sizeof(double) * 2 * C * G, st);
    if (e != cudaSuccess) return (int)e;
    Rank1Dy rt = r1;
    if (r1.dlog) {
        float* wtab = (float*)(sums + (size_t)3 * C * G);
        const int samples = Mg / r1.rps;
        rt.wtab = wtab;
        mdv_launch(rank1_table_kernel, dim3(mdv_cdiv(samples * C / 4, 256)), dim3(256), 0, st, r1, wtab, samples, C);
        MDV_CHECK_LAUNCH();
    }
    const int rpb = grouped_rows_per_block(Mg, C, G);
    const dim3 rgrid(mdv_cdiv(Mg, rpb), 1, G);
    if (r1.dlog)
        mdv_launch((bn_reduce_g_kernel<true, true>), rgrid, dim3(256), 0, st, dy, z, mean, rstd, act, sums, Mg, C, rpb, rt, gt, bt);
    else
        mdv_launch(bn_reduce_g_kernel<true>, rgrid, dim3(256), 0, st, dy, z, mean, rstd, act, sums, Mg, C, rpb, rt, gt, bt);
    MDV_CHECK_LAUNCH();
    mdv_launch(bn_bwd_finalize_kernel, dim3(mdv_cdiv(C, 128)), dim3(128), 0, st, (const double*)sums, G, Mg, C, coef, dgt, dbt);
    MDV_CHECK_LAUNCH();
    const int rpa = apply_rows_per_block(Mg, C, G);
    const dim3 agrid(mdv_cdiv(Mg, rpa), 1, G);
    if (dz_bf16 && r1.dlog)
        mdv_launch((bn_bwd_apply_g_kernel<bf16, true>), agrid, dim3(256), 0, st, dy, z, mean, rstd, act, (const float*)coef, (bf16*)dz, Mg, C,
                   rpa, rt, gt, bt);
    else if (dz_bf16)
        mdv_launch(bn_bwd_apply_g_kernel<bf16>, agrid, dim3(256), 0, st, dy, z, mean, rstd, act, (const float*)coef, (bf16*)dz, Mg, C, rpa, rt,
                   gt, bt);
    else if (r1.dlog)
        mdv_launch((bn_bwd_apply_g_kernel<float, true>), agrid, dim3(256), 0, st, dy, z, mean, rstd, act, (const float*)coef, (float*)dz, Mg, C,
                   rpa, rt, gt, bt);
    else
        mdv_launch(bn_bwd_apply_g_kernel<float>, agrid, dim3(256), 0, st, dy, z, mean, rstd, act, (const float*)coef, (float*)dz, Mg, C, rpa, rt,
                   gt, bt);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_bn_act_bwd(const float* dy, const float* z, const float* mean, const float* rstd, const float* gamma,
                              const float* beta, int act, void* dz, int dz_bf16, float* dgamma, float* dbeta, int M, int C,
                              void* ws, void* stream) {
    if (!dy || !z || !mean || !rstd || !gamma || !beta || !dz || !ws || M <= 0 || (C & 3)) return MDV_ERR_ARG;
    if (!bn_grouped_ok(1, M, C)) return MDV_ERR_UNSUPPORTED;
    return bn_act_bwd_impl(dy, Rank1Dy(), z, mean, rstd, one_set(gamma), one_set(beta), act, dz, dz_bf16, one_set(dgamma), one_set(dbeta), 1, M,
                           C, ws, (cudaStream_t)stream);
}

// Same, with the output gradient given in rank-1 form dy[m,c] = dlog[m] * wrow[c] * dropout2d_mask(m / rows_per_sample, c).
extern "C" int mdv_bn_act_bwd_rank1(const float* dlog, const float* wrow, int rows_per_sample, float drop_p, const void* rng,
                                    uint32_t drop_stream, const float* z, const float* mean, const float* rstd, const float* gamma,
                                    const float* beta, int act, void* dz, int dz_bf16, float* dgamma, float* dbeta, int M, int C,
                                    void* ws, void* stream) {
    if (!dlog || !wrow || !z || !mean || !rstd || !gamma || !beta || !dz || !ws || M <= 0 || (C & 3) || rows_per_sample <= 0)
        return MDV_ERR_ARG;
    if (!bn_grouped_ok(1, M, C) || M % rows_per_sample || (long long)(M / rows_per_sample + 1) * C >= 0x7fffffffLL) return MDV_ERR_UNSUPPORTED;
    Rank1Dy r1 = {dlog, wrow, (const unsigned long long*)rng, rows_per_sample, drop_p, drop_stream, nullptr};
    return bn_act_bwd_impl(nullptr, r1, z, mean, rstd, one_set(gamma), one_set(beta), act, dz, dz_bf16, one_set(dgamma), one_set(dbeta), 1, M, C,
                           ws, (cudaStream_t)stream);
}

extern "C" int mdv_bn_train_fwd_gp(const float* z, int G, int Mg, int C, float eps, float momentum, MdvPtrTable running_mean,
                                   MdvPtrTable running_var, MdvPtrTable num_batches_tracked, MdvPtrTable gamma, MdvPtrTable beta, int act,
                                   float* mean, float* rstd, void* y, int y_bf16, void* ws, void* stream) {
    if (G < 1 || G > MDV_MAX_GROUPS || !z || !mean || !rstd || !y || !ws || !tables_set(G, {&gamma, &beta})) return MDV_ERR_ARG;
    if (!bn_grouped_ok(G, Mg, C)) return MDV_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const int rc = bn_train_stats(z, G, Mg, C, eps, momentum, running_mean, running_var, num_batches_tracked, mean, rstd, ws, st);
    if (rc != MDV_OK) return rc;
    const int rpa = apply_rows_per_block(Mg, C, G);
    const dim3 grid(mdv_cdiv(Mg, rpa), 1, G);
    if (y_bf16)
        mdv_launch(bn_act_fwd_g_kernel<bf16>, grid, dim3(256), 0, st, z, (const float*)mean, (const float*)rstd, act, (bf16*)y, Mg, C, rpa, gamma,
                   beta);
    else
        mdv_launch(bn_act_fwd_g_kernel<float>, grid, dim3(256), 0, st, z, (const float*)mean, (const float*)rstd, act, (float*)y, Mg, C, rpa, gamma,
                   beta);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_bn_act_bwd_gp(const float* dy, const float* z, const float* mean, const float* rstd, MdvPtrTable gamma, MdvPtrTable beta,
                                 int act, void* dz, int dz_bf16, MdvPtrTable dgamma, MdvPtrTable dbeta, int G, int Mg, int C, void* ws,
                                 void* stream) {
    if (G < 1 || G > MDV_MAX_GROUPS || !dy || !z || !mean || !rstd || !dz || !ws || !tables_set(G, {&gamma, &beta})) return MDV_ERR_ARG;
    if (!bn_grouped_ok(G, Mg, C)) return MDV_ERR_UNSUPPORTED;
    return bn_act_bwd_impl(dy, Rank1Dy(), z, mean, rstd, gamma, beta, act, dz, dz_bf16, dgamma, dbeta, G, Mg, C, ws, (cudaStream_t)stream);
}
