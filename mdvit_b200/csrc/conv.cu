// Token-major (NHWC) stencil kernels: depthwise 3x3 (ConvPosEnc / patch-embed), the decoder's 2-in-per-group 3x3,
// im2col / col2im for the dense 3x3 convs (stem, bridge -> tcgen05 GEMM), bilinear resize (align_corners=False).
// All HBM/L2-bound; one thread owns 4 consecutive channels of one pixel so every access is a coalesced 16-byte vector.
// Reference: mpvit.py:239-248 (ConvPosEnc), mdvit.py:114-123 (DWConv2d_BN), Decoders.py:54-63,194-199,315-336,
// mdvit.py:509-526,557-564,699.
#include "../../include/mdvit_b200.h"
#include "common.cuh"

namespace {

// element / pixel indices of the stencil and resize kernels are 32-bit (64-bit divisions made these kernels issue-bound);
// every entry point checks that the tensor has fewer than 2^31 elements
typedef int idx_t;

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(bf16* p, float4 v) {
    *reinterpret_cast<uint2*>(p) = make_uint2(f2_to_bf2(v.x, v.y), f2_to_bf2(v.z, v.w));
}
__device__ __forceinline__ float4 ld4(const bf16* p) {
    uint2 u = *reinterpret_cast<const uint2*>(p);
    float2 a = bf2_to_f2(u.x), b = bf2_to_f2(u.y);
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void fma4(float4& a, const float4& w, const float4& x) {
    a.x += w.x * x.x; a.y += w.y * x.y; a.z += w.z * x.z; a.w += w.w * x.w;
}

// ---------------------------------------------------------------------------------- depthwise 3x3
// forward:    out[b,yo,xo,c] = bias[c] + sum_ij w[c,i,j] * in[b, yo*s-1+i, xo*s-1+j, c]   (+ in[b,yo,xo,c] if residual)
// transposed: out[b,y,x,c]   = sum_ij w[c,i,j] * in[b, (y+1-i)/s, (x+1-j)/s, c]           (+ in[b,y,x,c] if residual)
//             (input-gradient of the forward; `in` is then the output-gradient on the Ho x Wo grid)
// Weights are staged in shared memory as [9][C].
// STRIDE = 1 / 2 at compile time (0: runtime `stride_rt`): the transposed form divides and takes remainders by the stride for
// every tap — with a runtime stride the stride-2 input gradients of the patch embeddings were instruction bound at 6x their HBM time.
template <typename TO, int STRIDE>
__global__ void __launch_bounds__(256) dwconv3_kernel(const float* __restrict__ in, const float* __restrict__ w,
                                                       const float* __restrict__ bias, TO* __restrict__ out, int B, int Hi,
                                                       int Wi, int Ho, int Wo, int C, int stride_rt, int transposed, int residual) {
    MDV_PDL_SYNC();
    const int stride = STRIDE ? STRIDE : stride_rt;
    extern __shared__ float sw[];  // [9][C] then bias [C]
    for (int i = threadIdx.x; i < 9 * C; i += blockDim.x) sw[(i % 9) * C + i / 9] = w[i];
    for (int i = threadIdx.x; i < C; i += blockDim.x) sw[9 * C + i] = bias ? bias[i] : 0.f;
    __syncthreads();
    const int c4n = C >> 2;
    const idx_t total = (idx_t)B * Ho * Wo * c4n;
    for (idx_t idx = (idx_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (idx_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % c4n) * 4;
        idx_t pix = idx / c4n;
        const int xo = (int)(pix % Wo);
        pix /= Wo;
        const int yo = (int)(pix % Ho);
        const int b = (int)(pix / Ho);
        float4 acc = transposed ? make_float4(0.f, 0.f, 0.f, 0.f) : ld4(sw + 9 * C + c);
        const float* inb = in + (size_t)b * Hi * Wi * C;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            int yi;
            if (!transposed) {
                yi = yo * stride - 1 + i;
            } else {
                int t = yo + 1 - i;
                if (t < 0 || (t % stride)) continue;
                yi = t / stride;
            }
            if (yi < 0 || yi >= Hi) continue;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                int xi;
                if (!transposed) {
                    xi = xo * stride - 1 + j;
                } else {
                    int t = xo + 1 - j;
                    if (t < 0 || (t % stride)) continue;
                    xi = t / stride;
                }
                if (xi < 0 || xi >= Wi) continue;
                fma4(acc, ld4(sw + (i * 3 + j) * C + c), ld4(inb + ((size_t)yi * Wi + xi) * C + c));
            }
        }
        if (residual) {
            float4 r = ld4(inb + ((size_t)yo * Wi + xo) * C + c);
            acc.x += r.x; acc.y += r.y; acc.z += r.z; acc.w += r.w;
        }
        st4(out + ((size_t)(b * Ho + yo) * Wo + xo) * C + c, acc);
    }
}

// Stride-1 fast path (ConvPosEnc forward and backward, first patch embedding).  An image row of an NHWC tensor is one
// contiguous vector of W*C floats and a horizontal shift is +-C floats, so a thread owns 4 consecutive floats of the row
// (4 channels of one pixel) and walks down a segment of rows with a 3-row sliding window in registers: 3 coalesced
// 16-byte loads per output instead of 9, weights in registers, no per-element index arithmetic.
// flip = 1 gives the transposed convolution (input gradient): same stencil with the taps reversed.
struct Row3 {
    float4 l, m, r;
};
__device__ __forceinline__ Row3 load_row3(const float* __restrict__ row, int p, int C, bool ok, bool left_ok, bool right_ok) {
    Row3 t;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    t.m = ok ? ld4(row + p) : z;
    t.l = (ok && left_ok) ? ld4(row + p - C) : z;
    t.r = (ok && right_ok) ? ld4(row + p + C) : z;
    return t;
}
template <typename TO>
__global__ void __launch_bounds__(256) dwconv3_s1_kernel(const float* __restrict__ in, const float* __restrict__ w,
                                                          const float* __restrict__ bias, TO* __restrict__ out, int H, int W, int C,
                                                          int flip, int residual, int seg) {
    MDV_PDL_SYNC();
    const int L = W * C;
    const int p = (blockIdx.x * 256 + threadIdx.x) * 4;
    if (p >= L) return;
    const int c = p % C, x = p / C;
    const bool left_ok = x > 0, right_ok = x < W - 1;
    float4 wv[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const int tt = flip ? 8 - t : t;
        wv[t] = make_float4(__ldg(w + (c + 0) * 9 + tt), __ldg(w + (c + 1) * 9 + tt), __ldg(w + (c + 2) * 9 + tt), __ldg(w + (c + 3) * 9 + tt));
    }
    const float4 bv = bias ? ld4(bias + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int y0 = blockIdx.y * seg, y1 = min(H, y0 + seg);
    const float* img = in + (size_t)blockIdx.z * H * L;
    TO* oimg = out + (size_t)blockIdx.z * H * L;
    Row3 r0 = load_row3(img + (size_t)(y0 - 1) * L, p, C, y0 > 0, left_ok, right_ok);
    Row3 r1 = load_row3(img + (size_t)y0 * L, p, C, true, left_ok, right_ok);
#pragma unroll 4
    for (int y = y0; y < y1; ++y) {      // (unrolled: the loads of the next rows are independent of the arithmetic: more bytes in flight)
        const Row3 r2 = load_row3(img + (size_t)(y + 1) * L, p, C, y + 1 < H, left_ok, right_ok);
        float4 acc = bv;
        fma4(acc, wv[0], r0.l); fma4(acc, wv[1], r0.m); fma4(acc, wv[2], r0.r);
        fma4(acc, wv[3], r1.l); fma4(acc, wv[4], r1.m); fma4(acc, wv[5], r1.r);
        fma4(acc, wv[6], r2.l); fma4(acc, wv[7], r2.m); fma4(acc, wv[8], r2.r);
        if (residual) {
            acc.x += r1.m.x; acc.y += r1.m.y; acc.z += r1.m.z; acc.w += r1.m.w;
        }
        st4(oimg + (size_t)y * L + p, acc);
        r0 = r1;
        r1 = r2;
    }
}

// weight / bias gradient, stride 1: dw[c,i,j] += sum dy[y,x,c] * x[y-1+i, x-1+j, c];  db[c] += sum dy.  Same thread
// mapping; 10 float4 accumulators per thread, summed per block in shared memory, one global atomic per (channel, tap).
__global__ void __launch_bounds__(256) dwconv3_s1_wgrad_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                                float* __restrict__ dw, float* __restrict__ db, int H, int W, int C,
                                                                int seg) {
    MDV_PDL_SYNC();
    extern __shared__ float sacc[];     // [C][10]
    for (int i = threadIdx.x; i < C * 10; i += 256) sacc[i] = 0.f;
    __syncthreads();
    const int L = W * C;
    const int p = (blockIdx.x * 256 + threadIdx.x) * 4;
    if (p < L) {
        const int c = p % C, xx = p / C;
        const bool left_ok = xx > 0, right_ok = xx < W - 1;
        const int y0 = blockIdx.y * seg, y1 = min(H, y0 + seg);
        const float* img = x + (size_t)blockIdx.z * H * L;
        const float* gimg = dy + (size_t)blockIdx.z * H * L;
        float4 acc[10];
#pragma unroll
        for (int t = 0; t < 10; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        Row3 r0 = load_row3(img + (size_t)(y0 - 1) * L, p, C, y0 > 0, left_ok, right_ok);
        Row3 r1 = load_row3(img + (size_t)y0 * L, p, C, true, left_ok, right_ok);
#pragma unroll 4
        for (int y = y0; y < y1; ++y) {
            const Row3 r2 = load_row3(img + (size_t)(y + 1) * L, p, C, y + 1 < H, left_ok, right_ok);
            const float4 g = ld4(gimg + (size_t)y * L + p);
            fma4(acc[0], g, r0.l); fma4(acc[1], g, r0.m); fma4(acc[2], g, r0.r);
            fma4(acc[3], g, r1.l); fma4(acc[4], g, r1.m); fma4(acc[5], g, r1.r);
            fma4(acc[6], g, r2.l); fma4(acc[7], g, r2.m); fma4(acc[8], g, r2.r);
            acc[9].x += g.x; acc[9].y += g.y; acc[9].z += g.z; acc[9].w += g.w;
            r0 = r1;
            r1 = r2;
        }
#pragma unroll
        for (int t = 0; t < 10; ++t) {
            atomicAdd(sacc + (c + 0) * 10 + t, acc[t].x);
            atomicAdd(sacc + (c + 1) * 10 + t, acc[t].y);
            atomicAdd(sacc + (c + 2) * 10 + t, acc[t].z);
            atomicAdd(sacc + (c + 3) * 10 + t, acc[t].w);
        }
    }
    __syncthreads();
    // channels this block touched: the 1024-float span [blockIdx.x*1024, +1024) modulo C
    const int span = min(C, 1024);
    const int cfirst = (blockIdx.x * 1024) % C;
    for (int o = threadIdx.x; o < span * 10; o += 256) {
        const int cc = (cfirst + o / 10) % C, t = o % 10;
        const float v = sacc[cc * 10 + t];
        if (v != 0.f) {
            if (t < 9) atomicAdd(dw + cc * 9 + t, v);
            else if (db) atomicAdd(db + cc, v);
        }
    }
}

// weight / bias gradient of the forward above: dw[c,i,j] += sum dy[b,yo,xo,c] * x[b,yo*s-1+i,xo*s-1+j,c]; db[c] += sum dy
// block = 32 channels x 8 pixel lanes over a chunk of output pixels.
__global__ void __launch_bounds__(256) dwconv3_wgrad_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                             float* __restrict__ dw, float* __restrict__ db, int B, int Hi, int Wi,
                                                             int Ho, int Wo, int C, int stride, int pix_per_block) {
    MDV_PDL_SYNC();
    __shared__ float sh[8][32][11];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    const idx_t npix = (idx_t)B * Ho * Wo;
    const idx_t p0 = (idx_t)blockIdx.y * pix_per_block;
    const idx_t p1 = min(npix, p0 + pix_per_block);
    float acc[10];
#pragma unroll
    for (int t = 0; t < 10; ++t) acc[t] = 0.f;
    if (c < C)
        for (idx_t p = p0 + ty; p < p1; p += 8) {
            const int xo = (int)(p % Wo);
            const int yo = (int)((p / Wo) % Ho);
            const int b = (int)(p / ((idx_t)Wo * Ho));
            const float g = __ldg(dy + (size_t)p * C + c);
            acc[9] += g;
            const float* xb = x + (size_t)b * Hi * Wi * C + c;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int yi = yo * stride - 1 + i;
                if (yi < 0 || yi >= Hi) continue;
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int xi = xo * stride - 1 + j;
                    if (xi < 0 || xi >= Wi) continue;
                    acc[i * 3 + j] += g * __ldg(xb + ((size_t)yi * Wi + xi) * C);
                }
            }
        }
#pragma unroll
    for (int t = 0; t < 10; ++t) sh[ty][tx][t] = acc[t];
    __syncthreads();
    // 320 (channel, tap) sums per block, reduced over the 8 pixel lanes
    for (int o = threadIdx.x; o < 320; o += 256) {
        const int cc = o / 10, t = o % 10;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += sh[k][cc][t];
        const int cg = blockIdx.x * 32 + cc;
        if (cg < C) {
            if (t < 9) atomicAdd(dw + cg * 9 + t, s);
            else if (db) atomicAdd(db + cg, s);
        }
    }
}

// ---------------------------------------------------------------------------------- decoder grouped 3x3 (2 inputs / group)
// cat = concat(skip[C], up[C]) along channels; out[g] = sum_{t<2} sum_ij w[g,t,i,j] * cat[2g+t] shifted.  Decoders.py:30-38,198-205.
// cat channel k lives in skip if k < C else in up (k - C).  Forward and input gradient: sliding-window kernels further below.

// weight gradient: dw[g,t,i,j] += sum dout[p,g] * cat[p shifted, 2g+t].  block = 32 groups x 8 pixel lanes.
__global__ void __launch_bounds__(256) gconv2_wgrad_kernel(const float* __restrict__ dout, const float* __restrict__ skip,
                                                            const float* __restrict__ up, float* __restrict__ dw, int B, int H, int W,
                                                            int C, int pix_per_block) {
    MDV_PDL_SYNC();
    __shared__ float sh[8][32][19];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int g = blockIdx.x * 32 + tx;
    const idx_t npix = (idx_t)B * H * W;
    const idx_t p0 = (idx_t)blockIdx.y * pix_per_block, p1 = min(npix, p0 + pix_per_block);
    float acc[18];
#pragma unroll
    for (int t = 0; t < 18; ++t) acc[t] = 0.f;
    if (g < C) {
        const int k = 2 * g;
        const float* srcbase = (k < C ? skip + k : up + (k - C));
        for (idx_t p = p0 + ty; p < p1; p += 8) {
            const int x0 = (int)(p % W);
            const int y0 = (int)((p / W) % H);
            const int b = (int)(p / ((idx_t)W * H));
            const float d = __ldg(dout + (size_t)p * C + g);
            const float* src = srcbase + (size_t)b * H * W * C;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int yi = y0 - 1 + i;
                if (yi < 0 || yi >= H) continue;
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int xi = x0 - 1 + j;
                    if (xi < 0 || xi >= W) continue;
                    const float2 v = *reinterpret_cast<const float2*>(src + ((size_t)yi * W + xi) * C);
                    acc[i * 3 + j] += d * v.x;
                    acc[9 + i * 3 + j] += d * v.y;
                }
            }
        }
    }
#pragma unroll
    for (int t = 0; t < 18; ++t) sh[ty][tx][t] = acc[t];
    __syncthreads();
    for (int o = threadIdx.x; o < 32 * 18; o += 256) {
        const int gg = o / 18, t = o % 18;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += sh[k][gg][t];
        const int gi = blockIdx.x * 32 + gg;
        if (gi < C) atomicAdd(dw + (size_t)gi * 18 + t, s);
    }
}

// ---------------------------------------------------------------------------------- grouped 3x3, sliding-window versions
// Same scheme as dwconv3_s1_kernel: a thread owns one pixel column x and 4 consecutive "cat" channels 4q..4q+3 (= output
// channels g = 2q, 2q+1; cat = concat(skip, up), so the 4 channels are one float4 of `skip` (4q < C) or of `up`), walks
// down a segment of rows with a 3-row register window: 3 coalesced 16-byte loads per output row instead of 9.
struct GRow3 {
    float4 l, m, r;
};
__device__ __forceinline__ GRow3 gload_row3(const float* __restrict__ row, int p, int C, bool ok, bool left_ok, bool right_ok) {
    GRow3 t;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    t.m = ok ? ld4(row + p) : z;
    t.l = (ok && left_ok) ? ld4(row + p - C) : z;
    t.r = (ok && right_ok) ? ld4(row + p + C) : z;
    return t;
}
// taps of the two output channels g, g+1 as float4 (w[g,0,t], w[g,1,t], w[g+1,0,t], w[g+1,1,t]);  w layout [C][2][3][3]
__device__ __forceinline__ void gload_taps(const float* __restrict__ w, int g, bool flip, float4 (&wv)[9]) {
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const int tt = flip ? 8 - t : t;
        wv[t] = make_float4(__ldg(w + g * 18 + tt), __ldg(w + g * 18 + 9 + tt), __ldg(w + (g + 1) * 18 + tt), __ldg(w + (g + 1) * 18 + 9 + tt));
    }
}
__device__ __forceinline__ void gfma(float2& a, const float4& w, const float4& v) {
    a.x += w.x * v.x + w.y * v.y;
    a.y += w.z * v.z + w.w * v.w;
}

template <typename TO>
__global__ void __launch_bounds__(256) gconv2_s_fwd_kernel(const float* __restrict__ skip, const float* __restrict__ up,
                                                            const float* __restrict__ w, TO* __restrict__ out, int H, int W, int C,
                                                            int seg) {
    MDV_PDL_SYNC();
    const int half = C >> 1;                        // float4 groups per pixel of the concatenated input
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= W * half) return;
    const int x = t / half, q = t % half;
    const int k0 = 4 * q, g = 2 * q;
    const float* src = (k0 < C ? skip + k0 : up + (k0 - C)) + (size_t)blockIdx.z * H * W * C;
    const int p = x * C;                            // offset of pixel x inside an image row of the source
    const int L = W * C;
    const bool left_ok = x > 0, right_ok = x < W - 1;
    float4 wv[9];
    gload_taps(w, g, false, wv);
    const int y0 = blockIdx.y * seg, y1 = min(H, y0 + seg);
    TO* oimg = out + (size_t)blockIdx.z * H * L;
    GRow3 r0 = gload_row3(src + (size_t)(y0 - 1) * L, p, C, y0 > 0, left_ok, right_ok);
    GRow3 r1 = gload_row3(src + (size_t)y0 * L, p, C, true, left_ok, right_ok);
    for (int y = y0; y < y1; ++y) {
        const GRow3 r2 = gload_row3(src + (size_t)(y + 1) * L, p, C, y + 1 < H, left_ok, right_ok);
        float2 a = make_float2(0.f, 0.f);
        gfma(a, wv[0], r0.l); gfma(a, wv[1], r0.m); gfma(a, wv[2], r0.r);
        gfma(a, wv[3], r1.l); gfma(a, wv[4], r1.m); gfma(a, wv[5], r1.r);
        gfma(a, wv[6], r2.l); gfma(a, wv[7], r2.m); gfma(a, wv[8], r2.r);
        if (sizeof(TO) == 2) *reinterpret_cast<uint32_t*>(oimg + (size_t)y * L + p + g) = f2_to_bf2(a.x, a.y);
        else *reinterpret_cast<float2*>(oimg + (size_t)y * L + p + g) = a;
        r0 = r1;
        r1 = r2;
    }
}

// input gradient: dcat[4q..4q+3][y,x] = sum_ij w[.,.,i,j] * dout[g(.)][y+1-i, x+1-j]   (flipped taps), written to dskip / dup
__global__ void __launch_bounds__(256) gconv2_s_dgrad_kernel(const float* __restrict__ dout, const float* __restrict__ w,
                                                              float* __restrict__ dskip, float* __restrict__ dup, int H, int W, int C,
                                                              int seg) {
    MDV_PDL_SYNC();
    const int half = C >> 1;
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= W * half) return;
    const int x = t / half, q = t % half;
    const int k0 = 4 * q, g = 2 * q;
    const int L = W * C;
    const float* dimg = dout + (size_t)blockIdx.z * H * L + g;
    float* dst = (k0 < C ? dskip + k0 : dup + (k0 - C)) + (size_t)blockIdx.z * H * L;
    const int p = x * C;
    const bool left_ok = x > 0, right_ok = x < W - 1;
    float4 wv[9];
    gload_taps(w, g, true, wv);
    const int y0 = blockIdx.y * seg, y1 = min(H, y0 + seg);
    auto ldrow = [&](int y, float2& l, float2& m, float2& r) {
        const bool ok = y >= 0 && y < H;
        const float* row = dimg + (size_t)y * L + p;
        const float2 z = make_float2(0.f, 0.f);
        m = ok ? *reinterpret_cast<const float2*>(row) : z;
        l = (ok && left_ok) ? *reinterpret_cast<const float2*>(row - C) : z;
        r = (ok && right_ok) ? *reinterpret_cast<const float2*>(row + C) : z;
    };
    float2 a0l, a0m, a0r, a1l, a1m, a1r;
    ldrow(y0 - 1, a0l, a0m, a0r);
    ldrow(y0, a1l, a1m, a1r);
    for (int y = y0; y < y1; ++y) {
        float2 a2l, a2m, a2r;
        ldrow(y + 1, a2l, a2m, a2r);
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        auto acc = [&](const float4& ww, const float2& d) {
            a.x += ww.x * d.x; a.y += ww.y * d.x; a.z += ww.z * d.y; a.w += ww.w * d.y;
        };
        acc(wv[0], a0l); acc(wv[1], a0m); acc(wv[2], a0r);
        acc(wv[3], a1l); acc(wv[4], a1m); acc(wv[5], a1r);
        acc(wv[6], a2l); acc(wv[7], a2m); acc(wv[8], a2r);
        st4(dst + (size_t)y * L + p, a);
        a0l = a1l; a0m = a1m; a0r = a1r;
        a1l = a2l; a1m = a2m; a1r = a2r;
    }
}

// weight gradient: dw[g,t,i,j] += sum dout[g][y,x] * cat[2g+t][y-1+i, x-1+j]
__global__ void __launch_bounds__(256) gconv2_s_wgrad_kernel(const float* __restrict__ dout, const float* __restrict__ skip,
                                                              const float* __restrict__ up, float* __restrict__ dw, int H, int W, int C,
                                                              int seg) {
    MDV_PDL_SYNC();
    extern __shared__ float sacc[];     // [C/2][36]
    const int half = C >> 1;
    for (int i = threadIdx.x; i < half * 36; i += 256) sacc[i] = 0.f;
    __syncthreads();
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t < W * half) {
        const int x = t / half, q = t % half;
        const int k0 = 4 * q, g = 2 * q;
        const int L = W * C;
        const float* src = (k0 < C ? skip + k0 : up + (k0 - C)) + (size_t)blockIdx.z * H * L;
        const float* dimg = dout + (size_t)blockIdx.z * H * L + g;
        const int p = x * C;
        const bool left_ok = x > 0, right_ok = x < W - 1;
        const int y0 = blockIdx.y * seg, y1 = min(H, y0 + seg);
        float4 acc[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        GRow3 r0 = gload_row3(src + (size_t)(y0 - 1) * L, p, C, y0 > 0, left_ok, right_ok);
        GRow3 r1 = gload_row3(src + (size_t)y0 * L, p, C, true, left_ok, right_ok);
        for (int y = y0; y < y1; ++y) {
            const GRow3 r2 = gload_row3(src + (size_t)(y + 1) * L, p, C, y + 1 < H, left_ok, right_ok);
            const float2 d = *reinterpret_cast<const float2*>(dimg + (size_t)y * L + p);
            auto upd = [&](float4& a, const float4& v) {
                a.x += d.x * v.x; a.y += d.x * v.y; a.z += d.y * v.z; a.w += d.y * v.w;
            };
            upd(acc[0], r0.l); upd(acc[1], r0.m); upd(acc[2], r0.r);
            upd(acc[3], r1.l); upd(acc[4], r1.m); upd(acc[5], r1.r);
            upd(acc[6], r2.l); upd(acc[7], r2.m); upd(acc[8], r2.r);
            r0 = r1;
            r1 = r2;
        }
        // sacc[q][36]: (g,0,tap) at tap, (g,1,tap) at 9+tap, (g+1,0,tap) at 18+tap, (g+1,1,tap) at 27+tap == dw + g*18 layout
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            atomicAdd(sacc + q * 36 + k, acc[k].x);
            atomicAdd(sacc + q * 36 + 9 + k, acc[k].y);
            atomicAdd(sacc + q * 36 + 18 + k, acc[k].z);
            atomicAdd(sacc + q * 36 + 27 + k, acc[k].w);
        }
    }
    __syncthreads();
    for (int o = threadIdx.x; o < half * 36; o += 256) {
        const float v = sacc[o];
        if (v != 0.f) atomicAdd(dw + o, v);      // q*36 + r == g*18 + r: the same linear layout as dw [C][2][3][3]
    }
}

// ---------------------------------------------------------------------------------- im2col / col2im (3x3, pad 1)
// col[(b,yo,xo), (i*3+j)*C + c] = in[b, yo*s+(i-1)*d, xo*s+(j-1)*d, c]  (0 outside; d = dilation, padding = d); row pitch
// ldc >= 9*C (extra columns zeroed).
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) im2col3_kernel(const TI* __restrict__ in, TO* __restrict__ col, int B, int Hi, int Wi,
                                                       int Ho, int Wo, int C, int stride, int ldc, int dil) {
    MDV_PDL_SYNC();
    const int c4n = C >> 2;
    const int per_row = 9 * c4n;
    const idx_t total = (idx_t)B * Ho * Wo * per_row;
    for (idx_t idx = (idx_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (idx_t)gridDim.x * blockDim.x) {
        const int r = (int)(idx % per_row);
        const idx_t pix = idx / per_row;
        const int t = r / c4n, c = (r % c4n) * 4;
        const int xo = (int)(pix % Wo);
        const int yo = (int)((pix / Wo) % Ho);
        const int b = (int)(pix / ((idx_t)Wo * Ho));
        const int yi = yo * stride + (t / 3 - 1) * dil, xi = xo * stride + (t % 3 - 1) * dil;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (yi >= 0 && yi < Hi && xi >= 0 && xi < Wi) v = ld4(in + (((size_t)b * Hi + yi) * Wi + xi) * C + c);
        st4(col + (size_t)pix * ldc + t * C + c, v);
    }
}

// first stem conv: NCHW fp32 image [B,3,H,W] -> col [B*Ho*Wo, LD] (LD = 64 bf16, or 32 fp32 for the TF32 GEMM), column =
// (i*3+j)*3 + ci for < 27, zero elsewhere.
template <typename TO, int LD>
__global__ void __launch_bounds__(256) im2col_stem_kernel(const float* __restrict__ img, TO* __restrict__ col, int B, int Hi,
                                                           int Wi, int Ho, int Wo) {
    MDV_PDL_SYNC();
    const idx_t total = (idx_t)B * Ho * Wo * (LD / 2);  // one thread = 2 columns
    for (idx_t idx = (idx_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (idx_t)gridDim.x * blockDim.x) {
        const int k = (int)(idx % (LD / 2)) * 2;
        const idx_t pix = idx / (LD / 2);
        const int xo = (int)(pix % Wo);
        const int yo = (int)((pix / Wo) % Ho);
        const int b = (int)(pix / ((idx_t)Wo * Ho));
        float v[2] = {0.f, 0.f};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int kk = k + u;
            if (kk < 27) {
                const int t = kk / 3, ci = kk % 3;
                const int yi = yo * 2 - 1 + t / 3, xi = xo * 2 - 1 + t % 3;
                if (yi >= 0 && yi < Hi && xi >= 0 && xi < Wi) v[u] = __ldg(img + (((size_t)b * 3 + ci) * Hi + yi) * Wi + xi);
            }
        }
        if (sizeof(TO) == 2) *reinterpret_cast<uint32_t*>(col + (size_t)pix * LD + k) = f2_to_bf2(v[0], v[1]);
        else *reinterpret_cast<float2*>(col + (size_t)pix * LD + k) = make_float2(v[0], v[1]);
    }
}

// dx[b,y,x,c] (+)= sum_ij dcol[(b,(y-(i-1)d)/s,(x-(j-1)d)/s), (i*3+j)*C + c]   (gather form of the im2col transpose)
__global__ void __launch_bounds__(256) col2im3_kernel(const float* __restrict__ dcol, float* __restrict__ dx, int B, int Hi, int Wi,
                                                       int Ho, int Wo, int C, int stride, int ldc, int dil, int accumulate) {
    MDV_PDL_SYNC();
    const int c4n = C >> 2;
    const idx_t total = (idx_t)B * Hi * Wi * c4n;
    for (idx_t idx = (idx_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (idx_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % c4n) * 4;
        const idx_t pix = idx / c4n;
        const int x = (int)(pix % Wi);
        const int y = (int)((pix / Wi) % Hi);
        const int b = (int)(pix / ((idx_t)Wi * Hi));
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            int t = y - (i - 1) * dil;
            if (t < 0 || (t % stride)) continue;
            const int yo = t / stride;
            if (yo >= Ho) continue;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                int u = x - (j - 1) * dil;
                if (u < 0 || (u % stride)) continue;
                const int xo = u / stride;
                if (xo >= Wo) continue;
                const float4 v = ld4(dcol + (((size_t)b * Ho + yo) * Wo + xo) * ldc + (i * 3 + j) * C + c);
                a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
            }
        }
        if (accumulate) {
            const float4 o = ld4(dx + (size_t)pix * C + c);
            a.x += o.x; a.y += o.y; a.z += o.z; a.w += o.w;
        }
        st4(dx + (size_t)pix * C + c, a);
    }
}

// ---------------------------------------------------------------------------------- bilinear resize, align_corners=False
__device__ __forceinline__ void bil_src(int d, float scale, int n_in, int& i0, int& i1, float& lam) {
    float s = ((float)d + 0.5f) * scale - 0.5f;
    if (s < 0.f) s = 0.f;
    i0 = (int)s;
    if (i0 > n_in - 1) i0 = n_in - 1;
    i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    lam = s - (float)i0;
}

// Column-walking version: a thread owns one output column x and 4 channels and walks down a band of output rows; the
// horizontally interpolated values of the two source rows are kept in registers and only re-loaded when the source row
// index changes (every `scale` output rows), so an upsample by S costs ~4/S loads per output instead of 4.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) upsample_fwd_walk_kernel(const TI* __restrict__ in, int ld_in, TO* __restrict__ out, int ld_out,
                                                                 int Hi, int Wi, int Ho, int Wo, int C, int seg) {
    MDV_PDL_SYNC();
    const int c4n = C >> 2;
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= Wo * c4n) return;
    const int x = t / c4n, c = (t % c4n) * 4;
    const float sy = (float)Hi / Ho, sx = (float)Wi / Wo;
    int x0, x1;
    float lx;
    bil_src(x, sx, Wi, x0, x1, lx);
    const TI* base = in + (size_t)blockIdx.z * Hi * Wi * ld_in + c;
    TO* obase = out + ((size_t)blockIdx.z * Ho * Wo + x) * ld_out + c;
    auto hload = [&](int ys) {
        const float4 a = ld4(base + ((size_t)ys * Wi + x0) * ld_in), b = ld4(base + ((size_t)ys * Wi + x1) * ld_in);
        return make_float4(a.x + lx * (b.x - a.x), a.y + lx * (b.y - a.y), a.z + lx * (b.z - a.z), a.w + lx * (b.w - a.w));
    };
    int i0 = -1, i1 = -1;
    float4 h0 = make_float4(0.f, 0.f, 0.f, 0.f), h1 = h0;
    const int y0 = blockIdx.y * seg, y1 = min(Ho, y0 + seg);
    for (int y = y0; y < y1; ++y) {
        int ys0, ys1;
        float ly;
        bil_src(y, sy, Hi, ys0, ys1, ly);
        if (ys0 != i0) {
            if (ys0 == i1) h0 = h1; else h0 = hload(ys0);
            i0 = ys0;
        }
        if (ys1 != i1) {
            if (ys1 == i0) h1 = h0; else h1 = hload(ys1);
            i1 = ys1;
        }
        // same evaluation order as the reference formula: (1-ly)*((1-lx) a + lx b) + ly*(...)
        st4(obase + (size_t)y * Wo * ld_out,
            make_float4(h0.x + ly * (h1.x - h0.x), h0.y + ly * (h1.y - h0.y), h0.z + ly * (h1.z - h0.z), h0.w + ly * (h1.w - h0.w)));
    }
}

// bf16 -> bf16 with 8 channels (16 bytes) per thread: the aux decoder's 512-channel maps written into the concat buffer
__global__ void __launch_bounds__(256) upsample_fwd_walk8_kernel(const bf16* __restrict__ in, int ld_in, bf16* __restrict__ out, int ld_out,
                                                                  int Hi, int Wi, int Ho, int Wo, int C, int seg) {
    MDV_PDL_SYNC();
    const int c8n = C >> 3;
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= Wo * c8n) return;
    const int x = t / c8n, c = (t % c8n) * 8;
    const float sy = (float)Hi / Ho, sx = (float)Wi / Wo;
    int x0, x1;
    float lx;
    bil_src(x, sx, Wi, x0, x1, lx);
    const bf16* base = in + (size_t)blockIdx.z * Hi * Wi * ld_in + c;
    bf16* obase = out + ((size_t)blockIdx.z * Ho * Wo + x) * ld_out + c;
    struct F8 { float v[8]; };
    auto hload = [&](int ys) {
        const uint4 a = *reinterpret_cast<const uint4*>(base + ((size_t)ys * Wi + x0) * ld_in), b = *reinterpret_cast<const uint4*>(base + ((size_t)ys * Wi + x1) * ld_in);
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
        F8 r;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const float2 fa = bf2_to_f2(aw[w]), fb = bf2_to_f2(bw[w]);
            r.v[2 * w] = fa.x + lx * (fb.x - fa.x);
            r.v[2 * w + 1] = fa.y + lx * (fb.y - fa.y);
        }
        return r;
    };
    int i0 = -1, i1 = -1;
    F8 h0 = {}, h1 = {};
    const int y0 = blockIdx.y * seg, y1 = min(Ho, y0 + seg);
    for (int y = y0; y < y1; ++y) {
        int ys0, ys1;
        float ly;
        bil_src(y, sy, Hi, ys0, ys1, ly);
        if (ys0 != i0) {
            if (ys0 == i1) h0 = h1; else h0 = hload(ys0);
            i0 = ys0;
        }
        if (ys1 != i1) {
            if (ys1 == i0) h1 = h0; else h1 = hload(ys1);
            i1 = ys1;
        }
        uint32_t o[4];
#pragma unroll
        for (int w = 0; w < 4; ++w)
            o[w] = f2_to_bf2(h0.v[2 * w] + ly * (h1.v[2 * w] - h0.v[2 * w]), h0.v[2 * w + 1] + ly * (h1.v[2 * w + 1] - h0.v[2 * w + 1]));
        *reinterpret_cast<uint4*>(obase + (size_t)y * Wo * ld_out) = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// out[b, y, x, :] += sum_k resize(in_k)[b, y, x, :] for up to three fp32 maps of different sizes, one read-modify-write of
// `out`: the stage-2..4 terms of the collapsed aux decoder (ops.AuxFn).  Same column walk as upsample_fwd_walk_kernel, with
// the two horizontally interpolated source rows of every input kept in registers.
struct UpIn3 {
    const float* p[3];
    int H[3], W[3];
};

__global__ void __launch_bounds__(256) upsample_add_kernel(UpIn3 in, int n_in, float* __restrict__ out, int ld_out, int Ho, int Wo, int C,
                                                           int seg) {
    MDV_PDL_SYNC();
    const int c4n = C >> 2;
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= Wo * c4n) return;
    const int x = t / c4n, c = (t % c4n) * 4;
    const float* base[3];
    int x0[3], x1[3], i0[3], i1[3];
    float lx[3];
    float4 h0[3], h1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (k < n_in) {
            bil_src(x, (float)in.W[k] / Wo, in.W[k], x0[k], x1[k], lx[k]);
            base[k] = in.p[k] + (size_t)blockIdx.z * in.H[k] * in.W[k] * C + c;
        }
        i0[k] = i1[k] = -1;
        h0[k] = h1[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float* obase = out + ((size_t)blockIdx.z * Ho * Wo + x) * ld_out + c;
    const int y0 = blockIdx.y * seg, y1 = min(Ho, y0 + seg);
    // four rows of `out` in flight per thread: the pass is HBM-bound, one outstanding 16-byte load per thread is not enough
    for (int yb = y0; yb < y1; yb += 4) {
        float4 o[4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (yb + r < y1) o[r] = ld4(obase + (size_t)(yb + r) * Wo * ld_out);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int y = yb + r;
            if (y >= y1) break;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                if (k >= n_in) break;
                const int Wi = in.W[k];
                auto hload = [&](int ys) {
                    const float4 a = ld4(base[k] + ((size_t)ys * Wi + x0[k]) * C), b = ld4(base[k] + ((size_t)ys * Wi + x1[k]) * C);
                    return make_float4(a.x + lx[k] * (b.x - a.x), a.y + lx[k] * (b.y - a.y), a.z + lx[k] * (b.z - a.z), a.w + lx[k] * (b.w - a.w));
                };
                int ys0, ys1;
                float ly;
                bil_src(y, (float)in.H[k] / Ho, in.H[k], ys0, ys1, ly);
                if (ys0 != i0[k]) {
                    h0[k] = ys0 == i1[k] ? h1[k] : hload(ys0);
                    i0[k] = ys0;
                }
                if (ys1 != i1[k]) {
                    h1[k] = ys1 == i0[k] ? h0[k] : hload(ys1);
                    i1[k] = ys1;
                }
                o[r].x += h0[k].x + ly * (h1[k].x - h0[k].x);
                o[r].y += h0[k].y + ly * (h1[k].y - h0[k].y);
                o[r].z += h0[k].z + ly * (h1[k].z - h0[k].z);
                o[r].w += h0[k].w + ly * (h1[k].w - h0[k].w);
            }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
            if (yb + r < y1) st4(obase + (size_t)(yb + r) * Wo * ld_out, o[r]);
    }
}

// single-channel variant (the commuted segmentation heads): in [B,Hi,Wi] fp32 -> out [B,Ho,Wo] fp32
__global__ void __launch_bounds__(256) upsample1_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int Hi,
                                                             int Wi, int Ho, int Wo) {
    MDV_PDL_SYNC();
    const float sy = (float)Hi / Ho, sx = (float)Wi / Wo;
    const idx_t total = (idx_t)B * Ho * Wo;
    for (idx_t idx = (idx_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (idx_t)gridDim.x * blockDim.x) {
        const int x = (int)(idx % Wo);
        const int y = (int)((idx / Wo) % Ho);
        const int b = (int)(idx / ((idx_t)Wo * Ho));
        int y0, y1, x0, x1;
        float ly, lx;
        bil_src(y, sy, Hi, y0, y1, ly);
        bil_src(x, sx, Wi, x0, x1, lx);
        const float* base = in + (size_t)b * Hi * Wi;
        out[idx] = (1.f - ly) * ((1.f - lx) * __ldg(base + y0 * Wi + x0) + lx * __ldg(base + y0 * Wi + x1)) +
                   ly * ((1.f - lx) * __ldg(base + y1 * Wi + x0) + lx * __ldg(base + y1 * Wi + x1));
    }
}

// Transposed resize in gather form.  For input pixel (yi,xi) the contributing output rows are found by scanning the
// candidate window [ (yi-1)/scale , (yi+2)/scale ) and re-evaluating the forward's (i0,i1,lam) — an exact mirror.
template <typename TI, int VEC>
__global__ void __launch_bounds__(256) upsample_bwd_kernel(const TI* __restrict__ dout, int ld_out, float* __restrict__ din,
                                                            int ld_in, int B, int Hi, int Wi, int Ho, int Wo, int C) {
    MDV_PDL_SYNC();
    const int cvn = C / VEC;
    const float sy = (float)Hi / Ho, sx = (float)Wi / Wo;
    const float iy = (float)Ho / Hi, ix = (float)Wo / Wi;
    const idx_t total = (idx_t)B * Hi * Wi * cvn;
    for (idx_t idx = (idx_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (idx_t)gridDim.x * blockDim.x) {
        const int c = (int)(idx % cvn) * VEC;
        const idx_t pix = idx / cvn;
        const int xi = (int)(pix % Wi);
        const int yi = (int)((pix / Wi) % Hi);
        const int b = (int)(pix / ((idx_t)Wi * Hi));
        // outputs whose source coordinate falls in (i-1, i+1):  x in ((i-0.5)*inv - 0.5, (i+1.5)*inv - 0.5), padded by one
        int ya = (int)floorf(((float)yi - 0.5f) * iy - 0.5f) - 1, yb = (int)ceilf(((float)yi + 1.5f) * iy - 0.5f) + 2;
        int xa = (int)floorf(((float)xi - 0.5f) * ix - 0.5f) - 1, xb = (int)ceilf(((float)xi + 1.5f) * ix - 0.5f) + 2;
        ya = max(ya, 0); xa = max(xa, 0); yb = min(yb, Ho); xb = min(xb, Wo);
        float acc[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[v] = 0.f;
        {
            for (int y = ya; y < yb; ++y) {
                int y0, y1;
                float ly;
                bil_src(y, sy, Hi, y0, y1, ly);
                const float wy = (y0 == yi ? 1.f - ly : 0.f) + (y1 == yi ? ly : 0.f);
                if (wy == 0.f) continue;
                for (int x = xa; x < xb; ++x) {
                    int x0, x1;
                    float lx;
                    bil_src(x, sx, Wi, x0, x1, lx);
                    const float wx = (x0 == xi ? 1.f - lx : 0.f) + (x1 == xi ? lx : 0.f);
                    if (wx == 0.f) continue;
                    const TI* p = dout + (((size_t)b * Ho + y) * Wo + x) * ld_out + c;
                    const float wgt = wy * wx;
                    if (VEC == 4) {
                        const float4 v = ld4(p);
                        acc[0] += wgt * v.x; acc[1] += wgt * v.y; acc[2] += wgt * v.z; acc[3] += wgt * v.w;
                    } else {
                        acc[0] += wgt * ldf(p);
                    }
                }
            }
        }
        float* o = din + (size_t)pix * ld_in + c;
        if (VEC == 4) st4(o, make_float4(acc[0], acc[1], acc[2], acc[3]));
        else *o = acc[0];
    }
}

// Integer scale factors S (every resize of the 256x256 configuration: 2, 4, 8): input pixel i receives exactly the 2S
// outputs [S*i - S/2, S*i + 3S/2), so the window is a compile-time constant: no scanning, fully unrolled loads.  The
// weights are still evaluated with the forward's own index/lambda arithmetic (bil_src), which keeps the edge clamping
// (src < 0, i1 == i0 at the far edge) an exact mirror of F.interpolate(align_corners=False).
template <typename TI, int S>
__global__ void __launch_bounds__(256) upsample_bwd_int_kernel(const TI* __restrict__ dout, int ld_out, float* __restrict__ din,
                                                                int ld_in, int B, int Hi, int Wi, int C) {
    MDV_PDL_SYNC();
    const int Ho = Hi * S, Wo = Wi * S;
    const int cvn = C >> 2;
    const float sc = 1.f / S;
    const int total = B * Hi * Wi * cvn;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int c = (idx % cvn) * 4;
        const int pix = idx / cvn;
        const int xi = pix % Wi;
        const int yi = (pix / Wi) % Hi;
        const int b = pix / (Wi * Hi);
        const int xa = S * xi - S / 2, ya = S * yi - S / 2;
        float wx[2 * S];
#pragma unroll
        for (int k = 0; k < 2 * S; ++k) {
            const int x = xa + k;
            int x0, x1;
            float lx;
            bil_src(x, sc, Wi, x0, x1, lx);
            wx[k] = (x >= 0 && x < Wo) ? (x0 == xi ? 1.f - lx : 0.f) + (x1 == xi ? lx : 0.f) : 0.f;
        }
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int r = 0; r < 2 * S; ++r) {
            const int y = ya + r;
            if (y < 0 || y >= Ho) continue;
            int y0, y1;
            float ly;
            bil_src(y, sc, Hi, y0, y1, ly);
            const float wy = (y0 == yi ? 1.f - ly : 0.f) + (y1 == yi ? ly : 0.f);
            const TI* prow = dout + ((size_t)(b * Ho + y) * Wo) * ld_out + c;
#pragma unroll
            for (int k = 0; k < 2 * S; ++k) {
                const int x = xa + k;
                if (x < 0 || x >= Wo) continue;
                const float4 v = ld4(prow + (size_t)x * ld_out);
                const float wgt = wy * wx[k];
                acc.x += wgt * v.x; acc.y += wgt * v.y; acc.z += wgt * v.z; acc.w += wgt * v.w;
            }
        }
        st4(din + (size_t)pix * ld_in + c, acc);
    }
}

// Separable form of the same transposed resize for the larger factors: a horizontal pass into an fp32 scratch
// tmp[B, Ho, Wi, C] (every output pixel read by 2 input columns instead of the 2x2 = 4 input pixels of the one-pass kernel,
// which was L2-bandwidth bound on its 4x re-reads), then a vertical pass over the S-times smaller scratch.
template <typename TI, int S>
__global__ void __launch_bounds__(256) upsample_bwd_h_kernel(const TI* __restrict__ dout, int ld_out, float* __restrict__ tmp, int B,
                                                              int Ho, int Wi, int C) {
    MDV_PDL_SYNC();
    const int Wo = Wi * S;
    const int cvn = C >> 2;
    const float sc = 1.f / S;
    const int total = B * Ho * Wi * cvn;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int c = (idx % cvn) * 4;
        const int pix = idx / cvn;            // (b, y, xi)
        const int xi = pix % Wi;
        const int row = pix / Wi;             // b * Ho + y
        const int xa = S * xi - S / 2;
        const TI* prow = dout + (size_t)row * Wo * ld_out + c;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 2 * S; ++k) {
            const int x = xa + k;
            if (x < 0 || x >= Wo) continue;
            int x0, x1;
            float lx;
            bil_src(x, sc, Wi, x0, x1, lx);
            const float wgt = (x0 == xi ? 1.f - lx : 0.f) + (x1 == xi ? lx : 0.f);
            const float4 v = ld4(prow + (size_t)x * ld_out);
            acc.x += wgt * v.x; acc.y += wgt * v.y; acc.z += wgt * v.z; acc.w += wgt * v.w;
        }
        st4(tmp + (size_t)pix * C + c, acc);
    }
}

// bf16 gradients, 8 channels (16 bytes) per thread, tap weights from a per-block table: the scalar versions above spent more
// instructions on bil_src per tap than on the 4 multiply-adds and moved 8 bytes per load (0.3-0.4 of HBM at the aux decoder's
// 512-channel maps).  wtab[i][k] = weight of output pixel S*i - S/2 + k in input pixel i (0 outside the image).
template <int S>
__device__ __forceinline__ void upsample_wtab(float* wtab, int n_in) {
    const int n_out = n_in * S;
    const float sc = 1.f / S;
    for (int e = threadIdx.x; e < n_in * 2 * S; e += blockDim.x) {
        const int i = e / (2 * S), k = e - i * 2 * S;
        const int x = S * i - S / 2 + k;
        float w = 0.f;
        if (x >= 0 && x < n_out) {
            int x0, x1;
            float lx;
            bil_src(x, sc, n_in, x0, x1, lx);
            w = (x0 == i ? 1.f - lx : 0.f) + (x1 == i ? lx : 0.f);
        }
        wtab[e] = w;
    }
}
__device__ __forceinline__ void fma8(float (&acc)[8], float w, uint4 v) {
    const float2 a = bf2_to_f2(v.x), b = bf2_to_f2(v.y), c = bf2_to_f2(v.z), d = bf2_to_f2(v.w);
    acc[0] += w * a.x; acc[1] += w * a.y; acc[2] += w * b.x; acc[3] += w * b.y;
    acc[4] += w * c.x; acc[5] += w * c.y; acc[6] += w * d.x; acc[7] += w * d.y;
}

template <int S>
__global__ void __launch_bounds__(256) upsample_bwd_h8_kernel(const bf16* __restrict__ dout, int ld_out, float* __restrict__ tmp, int B,
                                                               int Ho, int Wi, int C) {
    MDV_PDL_SYNC();
    extern __shared__ float wtab[];      // [Wi][2S]
    upsample_wtab<S>(wtab, Wi);
    __syncthreads();
    const int Wo = Wi * S;
    const int cvn = C >> 3;
    const int total = B * Ho * Wi * cvn;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int c = (idx % cvn) * 8;
        const int pix = idx / cvn;            // (b, y, xi)
        const int xi = pix % Wi;
        const int row = pix / Wi;             // b * Ho + y
        const int xa = S * xi - S / 2;
        const bf16* prow = dout + (size_t)row * Wo * ld_out + c;
        uint4 v[2 * S];
#pragma unroll
        for (int k = 0; k < 2 * S; ++k) {
            const int x = min(max(xa + k, 0), Wo - 1);          // (clamped address; the table holds weight 0 outside)
            v[k] = *reinterpret_cast<const uint4*>(prow + (size_t)x * ld_out);
        }
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 2 * S; ++k) fma8(acc, wtab[xi * 2 * S + k], v[k]);
        float* o = tmp + (size_t)pix * C + c;
        st4(o, make_float4(acc[0], acc[1], acc[2], acc[3]));
        st4(o + 4, make_float4(acc[4], acc[5], acc[6], acc[7]));
    }
}

// one-pass 2x version (window 4 x 4)
__global__ void __launch_bounds__(256) upsample_bwd_int8x2_kernel(const bf16* __restrict__ dout, int ld_out, float* __restrict__ din,
                                                                   int ld_in, int B, int Hi, int Wi, int C) {
    MDV_PDL_SYNC();
    constexpr int S = 2;
    extern __shared__ float wtab[];      // [Wi][4] then [Hi][4]
    float* wty = wtab + Wi * 2 * S;
    upsample_wtab<S>(wtab, Wi);
    upsample_wtab<S>(wty, Hi);
    __syncthreads();
    const int Ho = Hi * S, Wo = Wi * S;
    const int cvn = C >> 3;
    const int total = B * Hi * Wi * cvn;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int c = (idx % cvn) * 8;
        const int pix = idx / cvn;
        const int xi = pix % Wi;
        const int yi = (pix / Wi) % Hi;
        const int b = pix / (Wi * Hi);
        const int xa = S * xi - S / 2, ya = S * yi - S / 2;
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int r = 0; r < 2 * S; ++r) {
            const int y = min(max(ya + r, 0), Ho - 1);
            const float wy = wty[yi * 2 * S + r];
            const bf16* prow = dout + ((size_t)(b * Ho + y) * Wo) * ld_out + c;
            uint4 v[2 * S];
#pragma unroll
            for (int k = 0; k < 2 * S; ++k) v[k] = *reinterpret_cast<const uint4*>(prow + (size_t)min(max(xa + k, 0), Wo - 1) * ld_out);
#pragma unroll
            for (int k = 0; k < 2 * S; ++k) fma8(acc, wy * wtab[xi * 2 * S + k], v[k]);
        }
        float* o = din + (size_t)pix * ld_in + c;
        st4(o, make_float4(acc[0], acc[1], acc[2], acc[3]));
        st4(o + 4, make_float4(acc[4], acc[5], acc[6], acc[7]));
    }
}

// single-channel maps (the gradients of the commuted segmentation heads' logits): integer factor, table weights — the generic
// gather kernel scanned a (3S)^2 candidate window with two bil_src evaluations per candidate
template <int S>
__global__ void __launch_bounds__(256) upsample_bwd_int1_kernel(const float* __restrict__ dout, float* __restrict__ din, int B, int Hi,
                                                                 int Wi) {
    MDV_PDL_SYNC();
    extern __shared__ float wtab[];      // [Wi][2S] then [Hi][2S]
    float* wty = wtab + Wi * 2 * S;
    upsample_wtab<S>(wtab, Wi);
    upsample_wtab<S>(wty, Hi);
    __syncthreads();
    const int Ho = Hi * S, Wo = Wi * S;
    const int total = B * Hi * Wi;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int xi = idx % Wi;
        const int yi = (idx / Wi) % Hi;
        const int b = idx / (Wi * Hi);
        const int xa = S * xi - S / 2, ya = S * yi - S / 2;
        float wx[2 * S];
#pragma unroll
        for (int k = 0; k < 2 * S; ++k) wx[k] = wtab[xi * 2 * S + k];
        float acc = 0.f;
#pragma unroll 2
        for (int r = 0; r < 2 * S; ++r) {
            const int y = min(max(ya + r, 0), Ho - 1);
            const float* prow = dout + (size_t)(b * Ho + y) * Wo;
            float rs = 0.f;
#pragma unroll
            for (int k = 0; k < 2 * S; ++k) rs = fmaf(wx[k], __ldg(prow + min(max(xa + k, 0), Wo - 1)), rs);
            acc = fmaf(wty[yi * 2 * S + r], rs, acc);
        }
        din[idx] = acc;
    }
}

template <int S>
__global__ void __launch_bounds__(256) upsample_bwd_v_kernel(const float* __restrict__ tmp, float* __restrict__ din, int ld_in, int B,
                                                              int Hi, int Wi, int C) {
    MDV_PDL_SYNC();
    const int Ho = Hi * S;
    const int cvn = C >> 2;
    const float sc = 1.f / S;
    const int total = B * Hi * Wi * cvn;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int c = (idx % cvn) * 4;
        const int pix = idx / cvn;
        const int xi = pix % Wi;
        const int yi = (pix / Wi) % Hi;
        const int b = pix / (Wi * Hi);
        const int ya = S * yi - S / 2;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int r = 0; r < 2 * S; ++r) {
            const int y = ya + r;
            if (y < 0 || y >= Ho) continue;
            int y0, y1;
            float ly;
            bil_src(y, sc, Hi, y0, y1, ly);
            const float wgt = (y0 == yi ? 1.f - ly : 0.f) + (y1 == yi ? ly : 0.f);
            const float4 v = ld4(tmp + ((size_t)(b * Ho + y) * Wi + xi) * C + c);
            acc.x += wgt * v.x; acc.y += wgt * v.y; acc.z += wgt * v.z; acc.w += wgt * v.w;
        }
        st4(din + (size_t)pix * ld_in + c, acc);
    }
}

inline int grid_for(long long total_threads) {
    long long b = (total_threads + 255) / 256;
    const long long cap = (long long)MDV_NUM_SMS * 16;
    return (int)(b < cap ? (b > 0 ? b : 1) : cap);
}
inline bool fits_i32(long long n) { return n > 0 && n < 0x7fffffffLL; }
inline int pix_per_block_for(long long npix, int col_blocks) {
    int want = (8 * MDV_NUM_SMS) / (col_blocks > 0 ? col_blocks : 1);
    if (want < 1) want = 1;
    long long ppb = (npix + want - 1) / want;
    if (ppb < 64) ppb = 64;
    return (int)ppb;
}

}  // namespace

extern "C" int mdv_dwconv3(const float* in, const float* w, const float* bias, void* out, int out_bf16, int B, int Hi, int Wi,
                           int Ho, int Wo, int C, int stride, int transposed, int residual, void* stream) {
    if (!in || !w || !out || (C & 3) || B <= 0) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * (Hi > Ho ? Hi : Ho) * (Wi > Wo ? Wi : Wo) * C)) return MDV_ERR_UNSUPPORTED;
    const long long total = (long long)B * Ho * Wo * (C / 4);
    const size_t smem = (size_t)10 * C * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    if (stride == 1 && Hi == Ho && Wi == Wo) {
        // rows per thread: long segments amortise the 36 weight loads and the 2 halo rows, as long as the grid still fills the SMs
        int seg = Hi >= 64 ? 16 : (Hi >= 16 ? 8 : Hi);
        while (seg < Hi && seg < 64 && (long long)mdv_cdiv((long long)Wi * C, 1024) * mdv_cdiv(Hi, 2 * seg) * B >= 4 * MDV_NUM_SMS) seg *= 2;
        dim3 grid(mdv_cdiv((long long)Wi * C, 1024), mdv_cdiv(Hi, seg), B);
        if (out_bf16) mdv_launch(dwconv3_s1_kernel<bf16>, dim3(grid), dim3(256), 0, st, in, w, bias, (bf16*)out, Hi, Wi, C, transposed, residual, seg);
        else mdv_launch(dwconv3_s1_kernel<float>, dim3(grid), dim3(256), 0, st, in, w, bias, (float*)out, Hi, Wi, C, transposed, residual, seg);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
#define MDV_DW(TO_, S_) mdv_launch((dwconv3_kernel<TO_, S_>), dim3(grid_for(total)), dim3(256), smem, st, in, w, bias, (TO_*)out, B, Hi, Wi, Ho, Wo, C, stride, transposed, residual)
    if (out_bf16) {
        if (stride == 2) MDV_DW(bf16, 2); else if (stride == 1) MDV_DW(bf16, 1); else MDV_DW(bf16, 0);
    } else {
        if (stride == 2) MDV_DW(float, 2); else if (stride == 1) MDV_DW(float, 1); else MDV_DW(float, 0);
    }
#undef MDV_DW
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_dwconv3_wgrad(const float* dy, const float* x, float* dw, float* db, int B, int Hi, int Wi, int Ho, int Wo,
                                 int C, int stride, void* stream) {
    if (!dy || !x || !dw || B <= 0) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * Hi * Wi * C)) return MDV_ERR_UNSUPPORTED;
    if (stride == 1 && Hi == Ho && Wi == Wo && !(C & 3) && C * 40 <= 48 * 1024) {
        // long row segments: the per-thread tail (40 shared + the block's global atomics) is amortised over more rows
        int seg = Hi >= 64 ? 16 : (Hi >= 16 ? 8 : Hi);
        while (seg < Hi && seg < 64 && (long long)mdv_cdiv((long long)Wi * C, 1024) * mdv_cdiv(Hi, 2 * seg) * B >= 4 * MDV_NUM_SMS) seg *= 2;
        dim3 grid(mdv_cdiv((long long)Wi * C, 1024), mdv_cdiv(Hi, seg), B);
        mdv_launch(dwconv3_s1_wgrad_kernel, dim3(grid), dim3(256), (size_t)C * 10 * sizeof(float), (cudaStream_t)stream, dy, x, dw, db, Hi, Wi, C, seg);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    const long long npix = (long long)B * Ho * Wo;
    const int cb = mdv_cdiv(C, 32);
    const int ppb = pix_per_block_for(npix, cb);
    dim3 grid(cb, mdv_cdiv(npix, ppb));
    mdv_launch(dwconv3_wgrad_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, dy, x, dw, db, B, Hi, Wi, Ho, Wo, C, stride, ppb);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_gconv2_fwd(const float* skip, const float* up, const float* w, void* out, int out_bf16, int B, int H, int W, int C,
                              void* stream) {
    if (!skip || !up || !w || !out || (C & 3)) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * H * W * C)) return MDV_ERR_UNSUPPORTED;
    {
        const int seg = H >= 64 ? 16 : (H >= 16 ? 8 : H);
        if (out_bf16)
            mdv_launch(gconv2_s_fwd_kernel<bf16>, dim3(mdv_cdiv(W * (C / 2), 256), mdv_cdiv(H, seg), B), dim3(256), 0, (cudaStream_t)stream, skip, up, w,
                       (bf16*)out, H, W, C, seg);
        else
            mdv_launch(gconv2_s_fwd_kernel<float>, dim3(mdv_cdiv(W * (C / 2), 256), mdv_cdiv(H, seg), B), dim3(256), 0, (cudaStream_t)stream, skip, up, w,
                       (float*)out, H, W, C, seg);
    }
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_gconv2_bwd(const float* dout, const float* skip, const float* up, const float* w, float* dskip, float* dup,
                              float* dw, int B, int H, int W, int C, void* stream) {
    if (!dout || !skip || !up || !w || !dskip || !dup || (C & 3)) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * H * W * C)) return MDV_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const int seg = H >= 64 ? 16 : (H >= 16 ? 8 : H);
    mdv_launch(gconv2_s_dgrad_kernel, dim3(mdv_cdiv(W * (C / 2), 256), mdv_cdiv(H, seg), B), dim3(256), 0, st, dout, w, dskip, dup, H, W, C, seg);
    MDV_CHECK_LAUNCH();
    if (!dw) return MDV_OK;   // weight gradient not wanted in this pass
    if ((size_t)(C / 2) * 36 * sizeof(float) <= 48 * 1024) {
        mdv_launch(gconv2_s_wgrad_kernel, dim3(mdv_cdiv(W * (C / 2), 256), mdv_cdiv(H, seg), B), dim3(256), (size_t)(C / 2) * 36 * sizeof(float), st,
                   dout, skip, up, dw, H, W, C, seg);
    } else {
        const long long npix = (long long)B * H * W;
        const int cb = mdv_cdiv(C, 32);
        const int ppb = pix_per_block_for(npix, cb);
        dim3 grid(cb, mdv_cdiv(npix, ppb));
        mdv_launch(gconv2_wgrad_kernel, dim3(grid), dim3(256), 0, st, dout, skip, up, dw, B, H, W, C, ppb);
    }
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_im2col3(const void* in, int in_bf16, void* col, int col_bf16, int B, int Hi, int Wi, int Ho, int Wo, int C, int stride,
                           int ldc, void* stream) {
    if (!in || !col || (C & 3) || ldc < 9 * C || (ldc & 7)) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * Ho * Wo * ldc)) return MDV_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (ldc > 9 * C) {
        cudaError_t e = cudaMemsetAsync(col, 0, (size_t)B * Ho * Wo * ldc * (col_bf16 ? 2 : 4), st);
        if (e != cudaSuccess) return (int)e;
    }
    const long long total = (long long)B * Ho * Wo * 9 * (C / 4);
    if (in_bf16 && col_bf16)
        mdv_launch((im2col3_kernel<bf16, bf16>), dim3(grid_for(total)), dim3(256), 0, st, (const bf16*)in, (bf16*)col, B, Hi, Wi, Ho, Wo, C, stride, ldc, 1);
    else if (!in_bf16 && col_bf16)
        mdv_launch((im2col3_kernel<float, bf16>), dim3(grid_for(total)), dim3(256), 0, st, (const float*)in, (bf16*)col, B, Hi, Wi, Ho, Wo, C, stride, ldc, 1);
    else if (!in_bf16 && !col_bf16)
        mdv_launch((im2col3_kernel<float, float>), dim3(grid_for(total)), dim3(256), 0, st, (const float*)in, (float*)col, B, Hi, Wi, Ho, Wo, C, stride, ldc, 1);
    else
        return MDV_ERR_UNSUPPORTED;
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_im2col_stem(const float* img_nchw, void* col, int col_bf16, int B, int Hi, int Wi, void* stream) {
    if (!img_nchw || !col || (Hi & 1) || (Wi & 1)) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * Hi * Wi * 16)) return MDV_ERR_UNSUPPORTED;
    const int Ho = Hi / 2, Wo = Wi / 2;
    if (col_bf16)
        mdv_launch((im2col_stem_kernel<bf16, 64>), dim3(grid_for((long long)B * Ho * Wo * 32)), dim3(256), 0, (cudaStream_t)stream, img_nchw, (bf16*)col, B, Hi, Wi, Ho, Wo);
    else
        mdv_launch((im2col_stem_kernel<float, 32>), dim3(grid_for((long long)B * Ho * Wo * 16)), dim3(256), 0, (cudaStream_t)stream, img_nchw, (float*)col, B, Hi, Wi, Ho, Wo);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_col2im3(const float* dcol, float* dx, int B, int Hi, int Wi, int Ho, int Wo, int C, int stride, int ldc,
                           void* stream) {
    if (!dcol || !dx || (C & 3)) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * Ho * Wo * ldc)) return MDV_ERR_UNSUPPORTED;
    mdv_launch(col2im3_kernel, dim3(grid_for((long long)B * Hi * Wi * (C / 4))), dim3(256), 0, (cudaStream_t)stream, dcol, dx, B, Hi, Wi, Ho, Wo, C, stride, ldc, 1, 0);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_im2col3_dil(const void* in, int in_bf16, void* col, int B, int H, int W, int C, int dil, int ldc, void* stream) {
    if (!in || !col || (C & 3) || ldc != 9 * C || dil < 1) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * H * W * ldc)) return MDV_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)B * H * W * 9 * (C / 4);
    if (in_bf16)
        mdv_launch((im2col3_kernel<bf16, bf16>), dim3(grid_for(total)), dim3(256), 0, st, (const bf16*)in, (bf16*)col, B, H, W, H, W, C, 1, ldc, dil);
    else
        mdv_launch((im2col3_kernel<float, bf16>), dim3(grid_for(total)), dim3(256), 0, st, (const float*)in, (bf16*)col, B, H, W, H, W, C, 1, ldc, dil);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_col2im3_dil(const float* dcol, float* dx, int B, int H, int W, int C, int dil, int ldc, int accumulate, void* stream) {
    if (!dcol || !dx || (C & 3) || dil < 1) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * H * W * ldc)) return MDV_ERR_UNSUPPORTED;
    mdv_launch(col2im3_kernel, dim3(grid_for((long long)B * H * W * (C / 4))), dim3(256), 0, (cudaStream_t)stream, dcol, dx, B, H, W, H, W, C, 1, ldc, dil,
               accumulate);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_upsample_fwd(const void* in, int in_bf16, int ld_in, void* out, int out_bf16, int ld_out, int B, int Hi, int Wi,
                                int Ho, int Wo, int C, void* stream) {
    if (!in || !out || B <= 0) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * Ho * Wo * (ld_out > C ? ld_out : C))) return MDV_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (C == 1) {
        if (in_bf16 || out_bf16) return MDV_ERR_UNSUPPORTED;
        mdv_launch(upsample1_fwd_kernel, dim3(grid_for((long long)B * Ho * Wo)), dim3(256), 0, st, (const float*)in, (float*)out, B, Hi, Wi, Ho, Wo);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    if ((C & 3) || (ld_in & 3) || (ld_out & 3)) return MDV_ERR_ARG;
    const int seg = Ho >= 64 ? 32 : Ho;
    const dim3 grid(mdv_cdiv(Wo * (C / 4), 256), mdv_cdiv(Ho, seg), B);
    if (in_bf16 && out_bf16 && !(C & 7) && !(ld_in & 7) && !(ld_out & 7) && !((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15))
        mdv_launch(upsample_fwd_walk8_kernel, dim3(mdv_cdiv(Wo * (C / 8), 256), mdv_cdiv(Ho, seg), B), dim3(256), 0, st, (const bf16*)in, ld_in, (bf16*)out,
                   ld_out, Hi, Wi, Ho, Wo, C, seg);
    else if (in_bf16 && out_bf16)
        mdv_launch((upsample_fwd_walk_kernel<bf16, bf16>), grid, dim3(256), 0, st, (const bf16*)in, ld_in, (bf16*)out, ld_out, Hi, Wi, Ho, Wo, C, seg);
    else if (!in_bf16 && out_bf16)
        mdv_launch((upsample_fwd_walk_kernel<float, bf16>), grid, dim3(256), 0, st, (const float*)in, ld_in, (bf16*)out, ld_out, Hi, Wi, Ho, Wo, C, seg);
    else if (!in_bf16 && !out_bf16)
        mdv_launch((upsample_fwd_walk_kernel<float, float>), grid, dim3(256), 0, st, (const float*)in, ld_in, (float*)out, ld_out, Hi, Wi, Ho, Wo, C, seg);
    else
        return MDV_ERR_UNSUPPORTED;
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

extern "C" int mdv_upsample_add(float* out, int ld_out, int B, int Ho, int Wo, int C, const float* in0, int H0, int W0, const float* in1,
                                int H1, int W1, const float* in2, int H2, int W2, void* stream) {
    if (!out || B <= 0 || Ho <= 0 || Wo <= 0 || C <= 0 || (C & 3) || (ld_out & 3) || ld_out < C || (reinterpret_cast<uintptr_t>(out) & 15))
        return MDV_ERR_ARG;
    UpIn3 in = {};
    int n = 0;
    const float* ps[3] = {in0, in1, in2};
    const int hs[3] = {H0, H1, H2}, ws[3] = {W0, W1, W2};
    for (int k = 0; k < 3; ++k) {
        if (!ps[k]) continue;
        if (hs[k] <= 0 || ws[k] <= 0 || (reinterpret_cast<uintptr_t>(ps[k]) & 15)) return MDV_ERR_ARG;
        if (!fits_i32((long long)B * hs[k] * ws[k] * C)) return MDV_ERR_UNSUPPORTED;
        in.p[n] = ps[k]; in.H[n] = hs[k]; in.W[n] = ws[k];
        ++n;
    }
    if (!n) return MDV_OK;
    const int seg = Ho >= 64 ? 32 : Ho;
    mdv_launch(upsample_add_kernel, dim3(mdv_cdiv(Wo * (C / 4), 256), mdv_cdiv(Ho, seg), B), dim3(256), 0, (cudaStream_t)stream, in, n, out,
               ld_out, Ho, Wo, C, seg);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

// din[B,Hi,Wi,C] (fp32, overwritten) = resize^T(dout[B,Ho,Wo,C])
extern "C" int mdv_upsample_bwd(const void* dout, int dout_bf16, int ld_out, float* din, int ld_in, int B, int Hi, int Wi, int Ho,
                                int Wo, int C, float* ws, void* stream) {
    if (!dout || !din || B <= 0) return MDV_ERR_ARG;
    if (!fits_i32((long long)B * Ho * Wo * (ld_out > C ? ld_out : C))) return MDV_ERR_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (C == 1) {
        if (dout_bf16) return MDV_ERR_UNSUPPORTED;
        const int S1 = (Ho % Hi == 0 && Wo % Wi == 0 && Ho / Hi == Wo / Wi) ? Ho / Hi : 0;
        if ((S1 == 2 || S1 == 4 || S1 == 8) && (size_t)(Wi + Hi) * 2 * S1 * sizeof(float) <= 40 * 1024) {
            const dim3 g1(grid_for((long long)B * Hi * Wi));
            const size_t sm = (size_t)(Wi + Hi) * 2 * S1 * sizeof(float);
            if (S1 == 2) mdv_launch(upsample_bwd_int1_kernel<2>, g1, dim3(256), sm, st, (const float*)dout, din, B, Hi, Wi);
            else if (S1 == 4) mdv_launch(upsample_bwd_int1_kernel<4>, g1, dim3(256), sm, st, (const float*)dout, din, B, Hi, Wi);
            else mdv_launch(upsample_bwd_int1_kernel<8>, g1, dim3(256), sm, st, (const float*)dout, din, B, Hi, Wi);
            MDV_CHECK_LAUNCH();
            return MDV_OK;
        }
        mdv_launch((upsample_bwd_kernel<float, 1>), dim3(grid_for((long long)B * Hi * Wi)), dim3(256), 0, st, (const float*)dout, 1, din, 1, B, Hi, Wi, Ho, Wo, 1);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    if ((C & 3) || (ld_in & 3) || (ld_out & 3)) return MDV_ERR_ARG;
    const int g = grid_for((long long)B * Hi * Wi * (C / 4));
    const int S = (Ho % Hi == 0 && Wo % Wi == 0 && Ho / Hi == Wo / Wi) ? Ho / Hi : 0;
    if (ws && (S == 4 || S == 8) && fits_i32((long long)B * Ho * Wi * C)) {
        // separable two-pass form (scratch: B*Ho*Wi*C floats)
        const int gh = grid_for((long long)B * Ho * Wi * (C / 4));
        const bool v8 = dout_bf16 && !(C & 7) && !(ld_out & 7) && !(reinterpret_cast<uintptr_t>(dout) & 15);
        const int gh8 = grid_for((long long)B * Ho * Wi * (C / 8));
#define MDV_UPH(SS)                                                                                                                  \
    if (v8) mdv_launch((upsample_bwd_h8_kernel<SS>), dim3(gh8), dim3(256), (size_t)Wi * 2 * SS * sizeof(float), st, (const bf16*)dout, ld_out, ws, B, Ho, Wi, C); \
    else if (dout_bf16) mdv_launch((upsample_bwd_h_kernel<bf16, SS>), dim3(gh), dim3(256), 0, st, (const bf16*)dout, ld_out, ws, B, Ho, Wi, C);     \
    else mdv_launch((upsample_bwd_h_kernel<float, SS>), dim3(gh), dim3(256), 0, st, (const float*)dout, ld_out, ws, B, Ho, Wi, C);             \
    MDV_CHECK_LAUNCH();                                                                                                              \
    mdv_launch((upsample_bwd_v_kernel<SS>), dim3(g), dim3(256), 0, st, (const float*)ws, din, ld_in, B, Hi, Wi, C);
        if (S == 4) { MDV_UPH(4) } else { MDV_UPH(8) }
#undef MDV_UPH
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    if (S == 2 && dout_bf16 && !(C & 7) && !(ld_out & 7) && !(ld_in & 3) && !(reinterpret_cast<uintptr_t>(dout) & 15)) {
        mdv_launch(upsample_bwd_int8x2_kernel, dim3(grid_for((long long)B * Hi * Wi * (C / 8))), dim3(256), (size_t)(Wi + Hi) * 4 * sizeof(float), st,
                   (const bf16*)dout, ld_out, din, ld_in, B, Hi, Wi, C);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    if ((S == 2 || S == 4 || S == 8) && (long long)B * Hi * Wi * (C / 4) < 0x7fffffffLL) {
#define MDV_UPB(SS)                                                                                                              \
    if (dout_bf16) mdv_launch((upsample_bwd_int_kernel<bf16, SS>), dim3(g), dim3(256), 0, st, (const bf16*)dout, ld_out, din, ld_in, B, Hi, Wi, C);     \
    else mdv_launch((upsample_bwd_int_kernel<float, SS>), dim3(g), dim3(256), 0, st, (const float*)dout, ld_out, din, ld_in, B, Hi, Wi, C);
        if (S == 2) { MDV_UPB(2) } else if (S == 4) { MDV_UPB(4) } else { MDV_UPB(8) }
#undef MDV_UPB
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    if (dout_bf16)
        mdv_launch((upsample_bwd_kernel<bf16, 4>), dim3(g), dim3(256), 0, st, (const bf16*)dout, ld_out, din, ld_in, B, Hi, Wi, Ho, Wo, C);
    else
        mdv_launch((upsample_bwd_kernel<float, 4>), dim3(g), dim3(256), 0, st, (const float*)dout, ld_out, din, ld_in, B, Hi, Wi, Ho, Wo, C);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}
