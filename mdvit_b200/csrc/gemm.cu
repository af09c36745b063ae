// Persistent, warp-specialised tcgen05 / TMEM / TMA GEMM for sm_100a.
//
//   mdv_gemm_nt : C[M,N] = epilogue( A[M,K] . W[N,K]^T )      (both operands K-major; Linear / 1x1 conv fwd + dgrad)
//   mdv_gemm_tn : C[P,Q] += A[R,P]^T . B[R,Q]                 (both operands MN-major; weight gradients; the reduction
//                                                              is split over CTAs and summed with TMA reduce-add)
//
// One CTA per SM loops over 128 x BN output tiles (tile = blockIdx.x, += gridDim.x; BN is a runtime multiple of 32).
//   warp 0      TMA producer: 128B-swizzled operand tiles into an mbarrier ring of `stages` buffers; runs ahead across tiles
//   warp 1      single-thread tcgen05.mma issuer; fp32 accumulators live in TMEM, double-buffered (2 x 256 columns)
//   warp 2      TMEM allocator
//   warps 4..11 epilogue: tcgen05.ld (32 lanes x 32 columns) -> bias / GELU / dropout / DropPath / residual in registers ->
//               swizzled shared-memory slab -> TMA store (bf16 or fp32), overlapping the next tile's loads and MMAs
// PAIR (large NT GEMMs): the kernel is launched as 2-CTA clusters and a CTA pair works on one 256 x BN tile with
//   tcgen05.mma.cta_group::2 — each CTA loads its own 128 rows of A and HALF of the B tile, so the operand bytes an SM pulls
//   from L2 per flop drop by 30-40% (these GEMMs are L2->SM bandwidth bound: K is short, see DESIGN.md).
// Replaces the aten::addmm / cudnn 1x1-conv calls behind nn.Linear / nn.Conv2d(k=1) in the reference
// (Models/Transformer/mdvit.py:288,310, mpvit.py:72-76, Decoders.py:197,59,317-333) and their backward passes.
#include <cuda.h>

#include <cstdlib>

#include "../../include/mdvit_b200.h"
#include "common.cuh"
#include "tc.cuh"

namespace {
using namespace tc;
#ifdef MDV_GEMM_SPIN_EPILOGUE
#define mbar_wait mbar_wait_spin
#endif

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int MAX_STAGES = 8;
constexpr int A_BYTES = BM * BK * 2;       // 16 KB
// NEPI epilogue warps (template parameter): NEPI/4 warps per TMEM lane quarter, interleaving 32-column chunks.  8 for
// MMA-bound shapes; 16 when the epilogue does real arithmetic (GELU / gelu' / dropout): those epilogues are issue-bound
// and 2 warps per scheduler cannot hide the ALU/MUFU latencies (profiles/r1_ncu_gemm_fc1_epilogue.txt: IPC 2.0).

struct GemmParams {
    int M, N, K;          // NT: output M x N, reduce K.  TN: output P(=M) x Q(=N), reduce R(=K)
    int BN;               // tile width (multiple of 32, <= 256; TN: multiple of 64)
    int stages;
    int n_tiles, m_tiles, splits, kb_per_split;
    int has_preact;
    int exp;              // development experiments (MDV_GEMM_EXP): 1 = skip the output stores
    int pair;             // NT only: 2-CTA clusters, one 256 x BN tile per CTA pair (tcgen05 cta_group::2)
    int tf32;             // NT only: operands are fp32, multiplied as TF32 (kind::tf32, 32-element k-blocks); else bf16 (64)
    int bk;               // elements per k-block: 128 bytes of K per row of a stage
    int nbuf;             // staging buffers per epilogue warp (2 or 4)
    int out_slab, buf_bytes;   // bytes of the output slab (2 KB bf16 / 4 KB fp32) and of one buffer (out [+ 2 KB preact])
    // NT only, implicit-GEMM 3x3 convolution (mdv_conv3_gemm): A is an NHWC activation read through a 4-D tensor map; k-block kc
    // belongs to tap kc / conv_cin and channels kc % conv_cin.., and its A tile is the output tile's pixels shifted by that tap
    int conv_cin, conv_w, conv_hw, conv_flip;
    // NT only, per-sample norm sets (mdv_gemm_nt_tf32_sets): epi.colscale / epi.bias are [nsets, N] tables and row m uses
    // table row sample_set[m / rows_per_sample]; NULL = the plain [N] vectors
    const int* sample_set;
    int rows_per_sample, nsets;
    MdvGemmEpi epi;
};

struct TileCoord {
    int m_tile, n_tile, kb0, num_kb;
};
template <bool TN>
__device__ __forceinline__ TileCoord tile_coord(const GemmParams& p, int t) {
    TileCoord c;
    c.n_tile = t % p.n_tiles;
    const int r = t / p.n_tiles;
    c.m_tile = r % p.m_tiles;
    const int total_kb = (p.K + p.bk - 1) / p.bk;
    if (TN) {
        c.kb0 = (r / p.m_tiles) * p.kb_per_split;
        c.num_kb = min(p.kb_per_split, total_kb - c.kb0);
    } else {
        c.kb0 = 0;
        c.num_kb = total_kb;
    }
    return c;
}

// LIGHT: the epilogue only adds a bias, sums columns and stores (no activation / multiplier / dropout / row scale / residual /
// second output): the feature tests of the general epilogue cost ~220 instructions per 32 x 32 chunk even when every feature is
// off, and the chunk chain of an epilogue warp is latency bound (profiles/r2_ncu_gemm_linear_fuse_dgrad.txt).
template <bool TN, int NEPI, bool PAIR, bool LIGHT>
__global__ void __launch_bounds__(32 * (4 + NEPI), 1)
    gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmP, const GemmParams p) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // PDL: let the next kernel start launching right away
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t tfull_bar[2];
    __shared__ __align__(8) uint64_t tempty_bar[2];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int BN = p.BN;
    const int stages = p.stages;
    // PAIR: this CTA's half of the B tile; its rows of the 256-row tile; the pair's position in the persistent tile walk
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const int cta_id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, cta_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    constexpr int TM = PAIR ? 2 * BM : BM;          // rows of an output tile
    const int bn_cta = PAIR ? BN / 2 : BN;          // B rows held by this CTA
    const uint32_t b_bytes = (uint32_t)bn_cta * BK * 2;
    const uint32_t stage_bytes = A_BYTES + b_bytes;
    uint8_t* slabs = smem + (size_t)stages * stage_bytes;          // [8 warps][nbuf][out (+ preact)]
    float* cs_all = reinterpret_cast<float*>(slabs + (size_t)NEPI * p.nbuf * p.buf_bytes);   // [NEPI warps][4 chunks][32]
    const int total_tiles = p.n_tiles * p.m_tiles * p.splits;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmC)) : "memory");
        if (p.has_preact) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmP)) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], PAIR ? 2 * NEPI : NEPI);      // PAIR: the epilogue warps of both CTAs arrive at the leader's
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(512u)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(512u)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();      // the peer's barriers are initialised before anything can arrive on them
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;
    // PDL: barrier init, TMEM allocation and tensor-map prefetch above overlap the previous kernel's tail; nothing before
    // this point reads or writes memory the previous kernel may still be producing / consuming
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int it = 0;
            for (int t = cta_id; t < total_tiles; t += cta_step) {
                const TileCoord tc = tile_coord<TN>(p, t);
                for (int kb = 0; kb < tc.num_kb; ++kb, ++it) {
                    const int s = it % stages;
                    const uint32_t ph = (it / stages) & 1;
                    mbar_wait_spin(&empty_bar[s], ph ^ 1);
                    uint8_t* sa = smem + (size_t)s * stage_bytes;
                    uint8_t* sb = sa + A_BYTES;
                    const int kc = (tc.kb0 + kb) * p.bk;
                    if (p.exp == 4) {       // experiment: no operand loads (MMA + epilogue alone)
                        if (rank == 0) mbar_arrive(&full_bar[s]);
                        continue;
                    }
                    // implicit 3x3 convolution: the A tile of this k-block = the tile's 128 pixels (whole image rows) moved by the tap
                    int cv_c = 0, cv_x = 0, cv_y = 0, cv_b = 0;
                    if (!TN && p.conv_cin) {
                        const int tap = kc / p.conv_cin;
                        cv_c = kc - tap * p.conv_cin;
                        int di = tap / 3 - 1, dj = tap - (tap / 3) * 3 - 1;
                        if (p.conv_flip) { di = -di; dj = -dj; }
                        const int p0 = tc.m_tile * TM + (int)rank * BM;
                        cv_b = p0 / p.conv_hw;
                        cv_y = (p0 - cv_b * p.conv_hw) / p.conv_w + di;
                        cv_x = dj;
                    }
                    if (PAIR) {
                        // the bytes of both CTAs are counted on the leader's barrier (a complete_tx that overtakes the
                        // leader's expect_tx only drives the transaction count negative within the same phase)
                        if (rank == 0) mbar_expect_tx(&full_bar[s], 2 * stage_bytes);
                        const uint32_t fb = mapa_u32(smem_u32(&full_bar[s]), 0);
                        if (p.conv_cin) tma_load_4d_pair(sa, &tmA, cv_c, cv_x, cv_y, cv_b, fb);
                        else tma_load_2d_pair(sa, &tmA, kc, tc.m_tile * TM + (int)rank * BM, fb);
                        tma_load_2d_pair(sb, &tmB, kc, tc.n_tile * BN + (int)rank * bn_cta, fb);
                        continue;
                    }
                    mbar_expect_tx(&full_bar[s], stage_bytes);
                    if (!TN) {
                        if (p.conv_cin) tma_load_4d(sa, &tmA, cv_c, cv_x, cv_y, cv_b, &full_bar[s]);
                        else tma_load_2d(sa, &tmA, kc, tc.m_tile * BM, &full_bar[s]);
                        tma_load_2d(sb, &tmB, kc, tc.n_tile * BN, &full_bar[s]);
                    } else {
                        for (int c = 0; c < BM / 64; ++c) tma_load_2d(sa + c * 8192, &tmA, tc.m_tile * BM + c * 64, kc, &full_bar[s]);
                        if (p.conv_cin) {
                            // implicit 3x3 weight gradient: column q of B is (tap, channel) = (q / Cin, q % Cin); the 64 reduction
                            // rows of this k-block are 64 consecutive pixels (whole image rows) moved by the tap
                            const int cb = kc / p.conv_hw, cy = (kc - cb * p.conv_hw) / p.conv_w;
                            for (int c = 0; c < BN / 64; ++c) {
                                const int q = tc.n_tile * BN + c * 64;
                                const int tap = q / p.conv_cin;
                                const int di = tap / 3 - 1, dj = tap - (tap / 3) * 3 - 1;
                                // (chunks past the last tap: an image index beyond the batch = all zeros)
                                tma_load_4d(sb + c * 8192, &tmB, q - tap * p.conv_cin, dj, cy + di, tap < 9 ? cb : 0x3fffffff, &full_bar[s]);
                            }
                        } else {
                            for (int c = 0; c < BN / 64; ++c) tma_load_2d(sb + c * 8192, &tmB, tc.n_tile * BN + c * 64, kc, &full_bar[s]);
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        // The WHOLE warp walks the loops (uniform control flow) and one elected lane issues: tcgen05.mma / commit take their
        // operands from uniform registers, and inside an `if (lane == 0)` region the compiler has to move every descriptor
        // there with ELECT / R2UR.BROADCAST waterfall loops — ~270 cycles per MMA, twice the 96-128 cycles the MMA itself takes
        // (the loop was issue-bound: same time with the operand loads removed, see DESIGN.md).
        if (rank == 0) {
            // TF32: same descriptor with a/b format 2 instead of 1 (cute::UMMA::F16F32Format); one MMA consumes K=8 fp32 = 32 B,
            // exactly the +32 B per step of the bf16 path (K=16), so the k-loop is shared
            const uint32_t idesc = p.tf32 ? (make_idesc(TM, BN, TN) + (1u << 7) + (1u << 10)) : make_idesc(TM, BN, TN);
            const bool is_tf32 = p.tf32 != 0;
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);      // (a value the compiler knows to be warp-uniform)
            // descriptors of stage 0, k-step 0: a stage / k-step only moves the start-address field (16-byte units, bits 0-13)
            //   K-major : 8-row groups 1024B apart; +32B per K=16 step inside the 128B swizzle span
            //   MN-major: 64-element MN chunks 8192B apart (LBO), 8 k-rows = 1024B (SBO); K=16 -> +2048B
            const uint32_t smem0 = smem_u32(smem);
            const uint64_t adesc0 = TN ? make_desc(smem0, 8192, 1024) : make_desc(smem0, 16, 1024);
            const uint64_t bdesc0 = TN ? make_desc(smem0 + A_BYTES, 8192, 1024) : make_desc(smem0 + A_BYTES, 16, 1024);
            constexpr uint32_t KSTEP16 = (TN ? 2048 : 32) >> 4;
            const uint32_t sstep16 = stage_bytes >> 4;
            const bool no_mma = p.exp == 3;      // experiment: no MMAs (loads + epilogue alone)
            int lt = 0, s = 0;
            uint32_t ph = 0;
            for (int t = cta_id; t < total_tiles; t += cta_step, ++lt) {
                const TileCoord tc = tile_coord<TN>(p, t);
                const int as = lt & 1;
                mbar_wait_spin(&tempty_bar[as], ((lt >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tacc = tmem_u + (uint32_t)as * 256u;
                for (int kb = 0; kb < tc.num_kb; ++kb) {
                    mbar_wait_spin(&full_bar[s], ph);
                    tc_fence_after();
                    const uint64_t ad = adesc0 + (uint64_t)((uint32_t)s * sstep16), bd = bdesc0 + (uint64_t)((uint32_t)s * sstep16);
                    if (elect_one()) {
                        if (!no_mma) {
#pragma unroll
                            for (int k = 0; k < BK / 16; ++k) {
                                const uint32_t acc = (kb | k) != 0 ? 1u : 0u;
                                if (PAIR) {
                                    if (is_tf32) tc_mma2_tf32(tacc, ad + k * KSTEP16, bd + k * KSTEP16, idesc, acc);
                                    else tc_mma2_bf16(tacc, ad + k * KSTEP16, bd + k * KSTEP16, idesc, acc);
                                } else if (!TN && is_tf32) tc_mma_tf32(tacc, ad + k * KSTEP16, bd + k * KSTEP16, idesc, acc);
                                else tc_mma_bf16(tacc, ad + k * KSTEP16, bd + k * KSTEP16, idesc, acc);
                            }
                        }
                        if (PAIR) tc_commit_pair(&empty_bar[s]);
                        else tc_commit(&empty_bar[s]);
                    }
                    __syncwarp();
                    if (++s == stages) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
                if (elect_one()) {
                    if (PAIR) tc_commit_pair(&tfull_bar[as]);
                    else tc_commit(&tfull_bar[as]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue
        const MdvGemmEpi& e = p.epi;
        const int q = warp & 3;                 // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;       // which interleaved 32-column chunks it owns (0 .. NEPI/4-1)
        constexpr int CSTEP = 8 * NEPI;         // column distance between two chunks of one warp
        uint8_t* myslab = slabs + (size_t)(warp - 4) * (p.nbuf * p.buf_bytes);
        const int nbuf_mask = p.nbuf - 1;
        uint32_t dthr = 0, dkey = 0;
        float dinv = 1.0f;
        if (!LIGHT && e.dropout_p > 0.0f) {
            dthr = drop_thresh(e.dropout_p);
            dinv = 1.0f / (1.0f - e.dropout_p);
            dkey = rng_key((const unsigned long long*)e.rng, e.drop_stream);
        }
        const bool out_bf16 = e.out_bf16 != 0;
        const float* const bias_p = e.bias;
        float* const colsum_p = e.colsum;
        // bias-gradient by-product: per-lane column sums of the stored tile, kept in shared memory across this CTA's
        // tiles while they share an n_tile and flushed with one atomic per column when it changes / at the end
        float* cs = cs_all + (warp - 4) * 128;
        int cs_n0 = -1;
        if (colsum_p) {
#pragma unroll
            for (int i = 0; i < 4; ++i) cs[i * 32 + lane] = 0.f;
        }
        int lt = 0, nstore = 0;
        for (int t = cta_id; t < total_tiles; t += cta_step, ++lt) {
            const TileCoord tc = tile_coord<TN>(p, t);
            const int as = lt & 1;
            if (colsum_p && tc.n_tile * BN != cs_n0) {
                if (cs_n0 >= 0) {
                    for (int i = 0; i < 4; ++i) {
                        const int col = cs_n0 + half * 32 + CSTEP * i + lane;
                        if (half * 32 + CSTEP * i < BN && col < p.N) atomicAdd(colsum_p + col, cs[i * 32 + lane]);
                        cs[i * 32 + lane] = 0.f;
                    }
                }
                cs_n0 = tc.n_tile * BN;
            }
            mbar_wait(&tfull_bar[as], (lt >> 1) & 1);
            tc_fence_after();
            const int row0 = tc.m_tile * TM + (int)rank * BM + q * 32;     // first row of this warp's slab
            const int row = row0 + lane;
            const bool row_ok = row < p.M;
            const int n0 = tc.n_tile * BN;
            float rs = 1.0f;
            if (!LIGHT && e.rowscale && row_ok) rs = __ldg(e.rowscale + row / e.rows_per_scale);
            for (int c0 = half * 32; c0 < BN; c0 += CSTEP) {
                const int col0 = n0 + c0;
                const bool full_cols = col0 + 32 <= p.N;
                // the multiplier tile (fc2 dgrad: gelu'(.)*mask saved by the forward) is read row-per-lane from global memory:
                // issue those loads BEFORE the TMEM load so their latency overlaps it (profiles/r2_ncu_gemm_fc2_dgrad_before_hoist.txt:
                // long-scoreboard stall 8.6 issue slots per instruction when they were issued at the point of use)
                uint4 uq[4];
                const bool pre_u = !LIGHT && e.mul_gelu_grad && row_ok && full_cols;
                if (pre_u) {
                    const bf16* up = (const bf16*)e.mul_gelu_grad + (size_t)row * e.ld_mul + col0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) uq[j] = *reinterpret_cast<const uint4*>(up + 8 * j);
                }
                uint32_t v[32];
                tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 256 + c0), v);
                tc_wait_ld();
                if (col0 >= p.N || row0 >= p.M) continue;   // tile overhang: nothing to store (warp-uniform)
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                int sset = 0;
                if (!LIGHT && e.colscale) {
                    // eval-mode BatchNorm folded into the GEMM: v = acc * scale[n] + shift[n] (shift arrives as `bias`)
                    // per-sample norm sets: this row's table row; an index outside [0, nsets) reads no table row (set 0 stands
                    // in) and the row is stored as NaN
                    if (p.sample_set && row_ok) {
                        sset = __ldg(p.sample_set + row / p.rows_per_sample);
                        if ((unsigned)sset >= (unsigned)p.nsets) sset = -1;
                    }
                    const int soff = sset > 0 ? sset * p.N : 0;
                    const float* const sc_p = e.colscale + soff;
                    const float* const sh_p = e.bias ? e.bias + soff : nullptr;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (col0 + j < p.N) f[j] = fmaf(f[j], __ldg(sc_p + col0 + j), sh_p ? __ldg(sh_p + col0 + j) : 0.f);
                } else if (bias_p) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        if (full_cols) {
                            const float4 b = __ldg(reinterpret_cast<const float4*>(bias_p + col0 + j));
                            f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
                        } else {
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                if (col0 + j + u < p.N) f[j + u] += __ldg(bias_p + col0 + j + u);
                        }
                    }
                }
                const int buf = nstore & nbuf_mask;
                // make sure the TMA store that last read this buffer has drained (one bulk group per chunk)
                if (lane == 0) {
                    if (p.nbuf == 4) tma_wait_read<3>();
                    else if (p.nbuf == 2) tma_wait_read<1>();
                    else tma_wait_read<0>();
                }
                __syncwarp();
                uint8_t* s_out = myslab + (size_t)buf * p.buf_bytes;
                uint8_t* s_pre = s_out + p.out_slab;
                const uint32_t s_out_u = smem_u32(s_out);
                const bool fused_act = !LIGHT && p.has_preact && e.preact_mode == 1 && e.act == MDV_ACT_GELU;
                if (fused_act) {
                    // one pass per pair: GELU, its derivative and the dropout scale share Phi(x), exp(-x^2/2) and the hash;
                    // out_preact receives gelu'(x) * mask/(1-p) — the factor the backward multiplies the gradient by
                    const uint32_t pbase = (uint32_t)(((unsigned long long)row * (unsigned)p.N + (unsigned)col0) >> 1);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        uint32_t pk[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int j = 8 * j4 + 2 * u;
                            const float2 x = make_float2(f[j], f[j + 1]);
                            float2 gl, gr;
                            gelu_pair<true>(x, &gl, &gr);
                            if (dthr) {
                                const uint32_t h = drop_hash(dkey, pbase + (j >> 1));
                                const float2 sc = make_float2(drop_lo(h, dthr, dinv), drop_hi(h, dthr, dinv));
                                gl = __fmul2_rn(gl, sc);
                                gr = __fmul2_rn(gr, sc);
                            }
                            f[j] = gl.x;
                            f[j + 1] = gl.y;
                            pk[u] = f2_to_bf2(gr.x, gr.y);
                        }
                        *reinterpret_cast<uint4*>(s_pre + lane * 64 + ((j4 ^ ((lane >> 1) & 3)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                } else if (!LIGHT) {
                if (p.has_preact) {
                    // bf16 rows of 64 B, SWIZZLE_64B: 16B-chunk index ^= (row >> 1) & 3
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 pk = make_uint4(f2_to_bf2(f[8 * j], f[8 * j + 1]), f2_to_bf2(f[8 * j + 2], f[8 * j + 3]),
                                              f2_to_bf2(f[8 * j + 4], f[8 * j + 5]), f2_to_bf2(f[8 * j + 6], f[8 * j + 7]));
                        *reinterpret_cast<uint4*>(s_pre + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)) = pk;
                    }
                }
                if (e.act == MDV_ACT_GELU) {
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                        const float2 r = gelu_erf2(make_float2(f[j], f[j + 1]));
                        f[j] = r.x;
                        f[j + 1] = r.y;
                    }
                } else if (e.act == MDV_ACT_RELU) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
                } else if (e.act == MDV_ACT_HSWISH) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = hardswish_f(f[j]);
                }
                }
                if (!LIGHT && e.mul_gelu_grad && row_ok) {
                    const bf16* up = (const bf16*)e.mul_gelu_grad + (size_t)row * e.ld_mul + col0;
#pragma unroll
                    for (int j = 0; j < 32; j += 8) {
                        if (full_cols) {
                            const uint4 u4 = uq[j >> 3];
                            const uint32_t uu[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const float2 uf = bf2_to_f2(uu[u]);
                                const float2 r = __fmul2_rn(make_float2(f[j + 2 * u], f[j + 2 * u + 1]), e.mul_mode == 1 ? uf : gelu_erf_grad2(uf));
                                f[j + 2 * u] = r.x;
                                f[j + 2 * u + 1] = r.y;
                            }
                        } else {
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (col0 + j + u < p.N) f[j + u] *= e.mul_mode == 1 ? __bfloat162float(up[j + u]) : gelu_erf_grad(__bfloat162float(up[j + u]));
                        }
                    }
                }
                if (!LIGHT && dthr && !fused_act) {
                    // N and col0 are even: elements (2j, 2j+1) of this chunk share one hash
                    const uint32_t pbase = (uint32_t)(((unsigned long long)row * (unsigned)p.N + (unsigned)col0) >> 1);
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const uint32_t h = drop_hash(dkey, pbase + j);
                        const float2 r = __fmul2_rn(make_float2(f[2 * j], f[2 * j + 1]), make_float2(drop_lo(h, dthr, dinv), drop_hi(h, dthr, dinv)));
                        f[2 * j] = r.x;
                        f[2 * j + 1] = r.y;
                    }
                }
                if (!LIGHT && e.rowscale) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] *= rs;
                }
                if (!LIGHT && e.residual && row_ok) {
                    const float* rp = e.residual + (size_t)row * e.ld_res + col0;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        if (full_cols) {
                            const float4 r4 = *reinterpret_cast<const float4*>(rp + j);
                            f[j] += r4.x; f[j + 1] += r4.y; f[j + 2] += r4.z; f[j + 3] += r4.w;
                        } else {
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                if (col0 + j + u < p.N) f[j + u] += rp[j + u];
                        }
                    }
                }
                if (!LIGHT && sset < 0) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = __int_as_float(0x7fffffff);      // out-of-range set index (after the
                }                                                                      // activation: ReLU would drop a NaN)
                if (colsum_p && !row_ok) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = 0.f;      // rows past M are clipped by the TMA store; keep them out of the sums
                }
                if (out_bf16) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 pk = make_uint4(f2_to_bf2(f[8 * j], f[8 * j + 1]), f2_to_bf2(f[8 * j + 2], f[8 * j + 3]),
                                              f2_to_bf2(f[8 * j + 4], f[8 * j + 5]), f2_to_bf2(f[8 * j + 6], f[8 * j + 7]));
                        sts128(s_out_u + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4), pk);
                    }
                } else {
                    // fp32 rows of 128 B, SWIZZLE_128B: 16B-chunk index ^= row & 7
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        sts128(s_out_u + lane * 128 + ((j ^ (lane & 7)) << 4),
                               make_uint4(__float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]), __float_as_uint(f[4 * j + 2]), __float_as_uint(f[4 * j + 3])));
                }
                fence_async_smem();
                __syncwarp();
                if (colsum_p) {
                    // lane = column: walk the 32 rows of the staged (swizzled) tile
                    float s = 0.f;
                    if (out_bf16) {
#pragma unroll 8
                        for (int r = 0; r < 32; ++r)
                            s += __bfloat162float(*reinterpret_cast<const bf16*>(s_out + r * 64 + (((lane >> 3) ^ ((r >> 1) & 3)) << 4) + (lane & 7) * 2));
                    } else {
#pragma unroll 8
                        for (int r = 0; r < 32; ++r)
                            s += *reinterpret_cast<const float*>(s_out + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + (lane & 3) * 4);
                    }
                    cs[((c0 - half * 32) / CSTEP) * 32 + lane] += s;
                }
                if (lane == 0 && p.exp != 1) {
                    if (TN) tma_reduce_add_2d(&tmC, s_out, col0, row0);
                    else tma_store_2d(&tmC, s_out, col0, row0);
                    if (!LIGHT && p.has_preact) tma_store_2d(&tmP, s_pre, col0, row0);
                    tma_commit();
                }
                ++nstore;
            }
            // all of this warp's tcgen05.ld for the tile have completed -> hand the accumulator stage back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (PAIR) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[as]), 0));
                else mbar_arrive(&tempty_bar[as]);
            }
        }
        if (colsum_p && cs_n0 >= 0) {
            for (int i = 0; i < 4; ++i) {
                const int col = cs_n0 + half * 32 + CSTEP * i + lane;
                if (half * 32 + CSTEP * i < BN && col < p.N) atomicAdd(colsum_p + col, cs[i * 32 + lane]);
            }
        }
        if (lane == 0) tma_wait_all();
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();      // neither CTA leaves (or frees TMEM) while the other can still signal it / write into it
    if (warp == 2) {
        tc_fence_after();
        if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ----------------------------------------------------------------------------- host side
int g_force_bn = 0, g_force_stages = 0, g_force_split = 0, g_force_grid = 0;
int g_force_light = [] {
    const char* e = getenv("MDV_GEMM_LIGHT");
    return e ? atoi(e) : 1;
}();
int g_force_pair = [] {
    const char* e = getenv("MDV_GEMM_PAIR");
    return e ? atoi(e) : -1;
}();

// Tile width (multiple of `step`, <= 256).  Measured with the operand loads switched off (scripts/dev_gemm_bn.py, MDV_GEMM_EXP=4),
// a K=16 MMA of width BN costs ~(224 + BN) units — a large width-independent part — so a wide tile that overhangs N by a few
// percent beats a narrower exact fit: minimise n_tiles * (224 + BN); ties go to the wider tile.
int pick_bn(int N, int step) {
    if (g_force_bn) return g_force_bn;
    int best = step;
    long long best_c = -1;
    for (int bn = 256; bn >= step; bn -= step) {
        const long long c = (long long)mdv_cdiv(N, bn) * (224 + bn);
        if (best_c < 0 || c < best_c) {
            best_c = c;
            best = bn;
        }
    }
    return best;
}

template <bool TN, int NEPI, bool PAIR, bool LIGHT>
int launch_n(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tp, GemmParams& p, cudaStream_t st) {
    const size_t stage_bytes = (size_t)A_BYTES + (size_t)(PAIR ? p.BN / 2 : p.BN) * BK * 2;
    p.out_slab = (TN || !p.epi.out_bf16) ? 4096 : 2048;
    p.buf_bytes = p.out_slab + (p.has_preact ? 2048 : 0);
    // short-K tiles are epilogue-bound (deep store buffering); long-K tiles are MMA-bound (spend smem on operand stages)
    const int kbt = TN ? p.kb_per_split : mdv_cdiv(p.K, p.bk);
    p.nbuf = kbt <= 2 ? 4 : (kbt <= 8 ? 2 : 1);
    if (p.exp == 2) p.nbuf = 4;
    if (NEPI > 8 && p.nbuf > 2) p.nbuf = 2;      // twice the warps: the same number of stores in flight
    const size_t cs_bytes = p.epi.colsum ? NEPI * 128 * sizeof(float) : 0;
    const size_t budget = 226 * 1024 - 1024 - 512;
    size_t slab_bytes;
    int stages;
    for (;;) {
        slab_bytes = (size_t)NEPI * p.nbuf * p.buf_bytes + cs_bytes;
        stages = (int)((budget - slab_bytes) / stage_bytes);
        if (stages >= 2 || p.nbuf == 1) break;
        p.nbuf >>= 1;      // trade store buffering for operand stages
    }
    if (stages > MAX_STAGES) stages = MAX_STAGES;
    if (g_force_stages && g_force_stages < stages) stages = g_force_stages;
    if (stages < 2) return MDV_ERR_UNSUPPORTED;
    p.stages = stages;
    const size_t smem = stages * stage_bytes + slab_bytes + 1024;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(gemm_kernel<TN, NEPI, PAIR, LIGHT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(226 * 1024));
        if (e != cudaSuccess) return (int)e;
        configured = true;
    }
    const int total_tiles = p.n_tiles * p.m_tiles * p.splits;
    if (PAIR) {
        // one cluster of two CTAs (a TPC) per tile walker
        int pairs = total_tiles < MDV_NUM_SMS / 2 ? total_tiles : MDV_NUM_SMS / 2;
        if (g_force_grid && g_force_grid / 2 < pairs && g_force_grid >= 2) pairs = g_force_grid / 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * pairs);
        cfg.blockDim = dim3(32 * (4 + NEPI));
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[2];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = g_mdv_pdl ? 2 : 1;
        cudaLaunchKernelEx(&cfg, gemm_kernel<TN, NEPI, PAIR, LIGHT>, ta, tb, tc, tp, p);
        MDV_CHECK_LAUNCH();
        return MDV_OK;
    }
    int grid = total_tiles < MDV_NUM_SMS ? total_tiles : MDV_NUM_SMS;
    if (g_force_grid && g_force_grid < grid) grid = g_force_grid;
    mdv_launch((gemm_kernel<TN, NEPI, PAIR, LIGHT>), dim3(grid), dim3(32 * (4 + NEPI)), smem, st, ta, tb, tc, tp, p);
    MDV_CHECK_LAUNCH();
    return MDV_OK;
}

int g_force_nepi = 0;

template <bool TN>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& tp, GemmParams& p, cudaStream_t st) {
    const MdvGemmEpi& e = p.epi;
    bool heavy = !TN && (e.act != MDV_ACT_NONE || e.mul_gelu_grad != nullptr || e.dropout_p > 0.f);
    if (g_force_nepi) heavy = g_force_nepi == 16;
    // LIGHT: nothing but (bias,) column sums and the store
    const bool light = !heavy && !e.rowscale && !e.residual && !e.colscale && !p.has_preact && g_force_light != 0;
    if constexpr (TN) {
        return launch_n<true, 8, false, true>(ta, tb, tc, tp, p, st);
    } else {
        if (p.pair) {
            if (heavy) {
                const int rc = launch_n<false, 16, true, false>(ta, tb, tc, tp, p, st);
                if (rc != MDV_ERR_UNSUPPORTED) return rc;
            }
            return light ? launch_n<false, 8, true, true>(ta, tb, tc, tp, p, st) : launch_n<false, 8, true, false>(ta, tb, tc, tp, p, st);
        }
        if (heavy) {
            const int rc = launch_n<false, 16, false, false>(ta, tb, tc, tp, p, st);
            if (rc != MDV_ERR_UNSUPPORTED) return rc;
        }
        return light ? launch_n<false, 8, false, true>(ta, tb, tc, tp, p, st) : launch_n<false, 8, false, false>(ta, tb, tc, tp, p, st);
    }
}

}  // namespace

extern "C" int mdv_gemm_tune(int force_bn, int force_stages, int force_split) {
    g_force_bn = force_bn;
    g_force_stages = force_stages & 0xff;
    g_force_nepi = (force_stages >> 8) & 0xff;      // debug: bits 8..15 of force_stages force the epilogue warp count (8 / 16)
    g_force_split = force_split;
    return MDV_OK;
}

extern "C" int mdv_gemm_force_pair(int mode) {
    g_force_pair = mode < 0 ? -1 : (mode != 0);
    return MDV_OK;
}

struct ConvGeom {      // implicit 3x3 convolution mode of gemm_nt_impl (mdv_conv3_gemm)
    int B, H, W, Cin, flip;
};

struct SampleSets {      // per-sample norm sets of mdv_gemm_nt_tf32_sets
    const int* idx;
    int rows_per_sample, S;
};

static int gemm_nt_impl(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi, int tf32, void* stream,
                        const ConvGeom* cv = nullptr, const SampleSets* sets = nullptr) {
    if (!A || !W || !epi || !epi->out || M <= 0 || N <= 0 || K <= 0) return MDV_ERR_ARG;
    if ((N & 3) || (K & (tf32 ? 3 : 7)) || epi->accumulate) return MDV_ERR_ARG;
    GemmParams p = {};
    p.M = M; p.N = N; p.K = K;
    if (cv) {
        p.conv_cin = cv->Cin; p.conv_w = cv->W; p.conv_hw = cv->H * cv->W; p.conv_flip = cv->flip;
    }
    if (sets) {
        p.sample_set = sets->idx; p.rows_per_sample = sets->rows_per_sample; p.nsets = sets->S;
    }
    p.epi = *epi;
    p.tf32 = tf32;
    p.bk = tf32 ? 32 : 64;
    p.BN = pick_bn(N, 32);
    p.n_tiles = mdv_cdiv(N, p.BN);
    {
        static const int exp = getenv("MDV_GEMM_EXP") ? atoi(getenv("MDV_GEMM_EXP")) : 0;
        p.exp = exp;
    }
    // CTA pairs for long-K problems with enough 256-row tiles for every pair (they are bound by operand traffic and power: a
    // pair moves 30-40% fewer operand bytes per flop).  Short-K tiles are epilogue bound and lose to the cross-CTA
    // accumulator hand-shake (K=64: 31 -> 43 us), narrow tiles have no B half worth sharing (N=64: 55 -> 63 us), small problems
    // would leave SMs idle.  MDV_GEMM_PAIR=0/1 overrides (A/B runs).
    p.pair = g_force_pair >= 0 ? g_force_pair
                               : (mdv_cdiv(K, p.bk) >= 8 && p.BN >= 128 && (long long)mdv_cdiv(M, 2 * BM) * p.n_tiles >= 2 * (MDV_NUM_SMS / 2));
    if (M < 2 * BM) p.pair = 0;
    p.m_tiles = mdv_cdiv(M, p.pair ? 2 * BM : BM);
    p.splits = 1;
    p.kb_per_split = mdv_cdiv(K, p.bk);
    p.has_preact = epi->out_preact != nullptr;
    CUtensorMap ta, tb, tc, tp;
    const int es = tf32 ? 4 : 2;
    int rc = cv ? make_map_nhwc(&ta, A, es, cv->Cin, cv->W, cv->H, cv->B, lda, p.bk, cv->W, BM / cv->W, CU_TENSOR_MAP_SWIZZLE_128B)
                : make_map(&ta, A, es, K, M, lda, p.bk, BM, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_map(&tb, W, es, K, N, ldw, p.bk, p.pair ? p.BN / 2 : p.BN, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    if (epi->out_bf16) rc = make_map(&tc, epi->out, 2, N, M, epi->ldc, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
    else rc = make_map(&tc, epi->out, 4, N, M, epi->ldc, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    tp = tc;
    if (p.has_preact) {
        rc = make_map(&tp, epi->out_preact, 2, N, M, epi->ld_preact, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B);
        if (rc) return rc;
    }
    return launch<false>(ta, tb, tc, tp, p, (cudaStream_t)stream);
}

extern "C" int mdv_gemm_nt(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi,
                           void* stream) {
    return gemm_nt_impl(A, lda, W, ldw, M, N, K, epi, 0, stream);
}

extern "C" int mdv_gemm_nt_tf32(const float* A, int lda, const float* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi,
                                void* stream) {
    return gemm_nt_impl(A, lda, W, ldw, M, N, K, epi, 1, stream);
}

extern "C" int mdv_gemm_nt_tf32_sets(const float* A, int lda, const float* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi,
                                     const int* sample_set, int rows_per_sample, int S, void* stream) {
    if (!epi || !epi->colscale || !sample_set || rows_per_sample < 1 || S < 1 || S > MDV_MAX_GROUPS) return MDV_ERR_ARG;
    const SampleSets sets = {sample_set, rows_per_sample, S};
    return gemm_nt_impl(A, lda, W, ldw, M, N, K, epi, 1, stream, nullptr, &sets);
}

// out[(b,y,x), n] = epi( sum_{tap=(i,j), c} x[b, y + s(i-1), x + s(j-1), c] . Wm[n, tap*Cin + c] ),  s = flip ? -1 : +1, zero outside
// the image: a 3x3 / stride 1 / padding 1 convolution as ONE tcgen05 GEMM with K = 9*Cin whose A tiles are fetched straight from
// the NHWC activation by 4-D TMA boxes (no im2col matrix).  flip = 1 with x := dz and Wm[ci, tap*Cout + co] = w[co, ci, tap] is the
// convolution's input gradient.
extern "C" int mdv_conv3_gemm(const void* x, int x_f32, int ldx, const void* Wm, int ldw, int B, int H, int W, int Cin, int N, int flip,
                              const MdvGemmEpi* epi, void* stream) {
    if (!x || !Wm || !epi || B <= 0 || H <= 0 || W <= 0 || Cin <= 0) return MDV_ERR_ARG;
    const int bk = x_f32 ? 32 : 64;
    if ((Cin % bk) || W > BM || (BM % W) || ((long long)H * W) % BM) return MDV_ERR_UNSUPPORTED;
    if ((long long)B * H * W >= 2147483647LL) return MDV_ERR_UNSUPPORTED;
    ConvGeom cv = {B, H, W, Cin, flip ? 1 : 0};
    return gemm_nt_impl(x, ldx, Wm, ldw, B * H * W, N, 9 * Cin, epi, x_f32 ? 1 : 0, stream, &cv);
}

static int gemm_tn_impl(const void* A, int lda, const void* B, int ldb, int R, int P, int Q, float* C, int ldc, void* stream,
                        const ConvGeom* cv = nullptr) {
    if (!A || !B || !C || R <= 0 || P <= 0 || Q <= 0) return MDV_ERR_ARG;
    if ((P & 7) || (Q & 7) || (ldc & 3)) return MDV_ERR_ARG;
    GemmParams p = {};
    p.M = P; p.N = Q; p.K = R;
    if (cv) {
        p.conv_cin = cv->Cin; p.conv_w = cv->W; p.conv_hw = cv->H * cv->W;
    }
    p.bk = BK;
    p.BN = pick_bn(Q, 64);
    p.n_tiles = mdv_cdiv(Q, p.BN);
    p.m_tiles = mdv_cdiv(P, BM);
    const int kb = mdv_cdiv(R, BK);
    // split the reduction so that every SM gets ~2 tiles; at least 4 k-blocks per split
    int want = (2 * MDV_NUM_SMS) / (p.n_tiles * p.m_tiles);
    if (want < 1) want = 1;
    int splits = kb / 4 < want ? (kb / 4 > 0 ? kb / 4 : 1) : want;
    if (g_force_split) splits = g_force_split;
    if (splits > kb) splits = kb;
    p.kb_per_split = mdv_cdiv(kb, splits);
    p.splits = mdv_cdiv(kb, p.kb_per_split);
    MdvGemmEpi e = {};
    e.out = C;
    e.ldc = ldc;
    p.epi = e;
    CUtensorMap ta, tb, tc;
    int rc = make_map(&ta, A, 2, P, R, lda, 64, BK, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = cv ? make_map_nhwc(&tb, B, 2, cv->Cin, cv->W, cv->H, cv->B, ldb, 64, cv->W, BK / cv->W, CU_TENSOR_MAP_SWIZZLE_128B)
            : make_map(&tb, B, 2, Q, R, ldb, 64, BK, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_map(&tc, C, 4, Q, P, ldc, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    return launch<true>(ta, tb, tc, tc, p, (cudaStream_t)stream);
}

extern "C" int mdv_gemm_tn(const void* A, int lda, const void* B, int ldb, int R, int P, int Q, float* C, int ldc,
                           void* stream) {
    return gemm_tn_impl(A, lda, B, ldb, R, P, Q, C, ldc, stream);
}

// dWm[p, tap*Cin + c] += sum_{(b,y,x)} dz[(b,y,x), p] . x[b, y + i - 1, x + j - 1, c]: the weight gradient of the 3x3 / stride 1 /
// padding 1 convolution in the im2col column order of mdv_prep_weight mode 2 (mdv_unperm_conv_grad turns it into [P, Cin, 3, 3]),
// as one TN GEMM whose B tiles come straight from the NHWC activation (4-D TMA boxes; no im2col matrix).
extern "C" int mdv_conv3_wgrad(const void* dz_bf16, int ldz, const void* x_bf16, int ldx, int B, int H, int W, int Cin, int P, float* dWm,
                               int ldc, void* stream) {
    if (!dz_bf16 || !x_bf16 || !dWm || B <= 0 || H <= 0 || W <= 0 || Cin <= 0) return MDV_ERR_ARG;
    if ((Cin % 64) || W > BK || (BK % W) || ((long long)H * W) % BK) return MDV_ERR_UNSUPPORTED;
    if ((long long)B * H * W >= 2147483647LL) return MDV_ERR_UNSUPPORTED;
    ConvGeom cv = {B, H, W, Cin, 0};
    return gemm_tn_impl(dz_bf16, ldz, x_bf16, ldx, B * H * W, P, 9 * Cin, dWm, ldc, stream, &cv);
}
