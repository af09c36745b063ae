/* mdvit_b200 — C ABI of the B200 (sm_100a) kernels behind the MDViT hot path.
 *
 * The reference (siyi-wind/MDViT) is pure PyTorch and has no FFI layer of its own; its drop-in
 * boundary is the nn.Module contract (Models/Transformer/mdvit.py:484-504 ctor, :667 forward).
 * This library sits underneath that module: every entry point replaces the aten op(s) the reference
 * module launches at the cited line.  The Python host (mdvit_b200/_lib.py) binds it with ctypes.
 *
 * Conventions: all pointers are DEVICE pointers unless noted; activations are token-major
 * ([B, H*W, C] == NHWC); `stream` is a cudaStream_t passed as void*; every function returns
 * 0 on success, a positive cudaError_t on a CUDA failure, or a negative MDV_ERR_* code on bad
 * arguments.  Nothing is allocated or freed by the library; workspaces are caller-owned.
 * Functions are re-entrant (no global mutable state apart from the debug knobs mdv_gemm_tune / mdv_gemm_force_pair).
 */
#ifndef MDVIT_B200_H
#define MDVIT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDV_ACT_NONE 0
#define MDV_ACT_GELU 1
#define MDV_ACT_RELU 2
#define MDV_ACT_HSWISH 3

int mdv_version(void);
long long mdv_launch_count(void); /* kernels launched by this library so far (host-side counter) */
/* Programmatic dependent launch for every kernel of the library (default on; env MDV_NO_PDL=1 disables): each kernel's
 * launch and prologue overlap the tail of its predecessor on the stream; results are unchanged. */
int mdv_set_pdl(int enabled);

/* ------------------------------------------------------------------ GEMM (tcgen05 / TMEM / TMA) */
/* Epilogue applied to acc = A.W^T, in this order:
 *   v = acc + bias[n];  out_preact[m,n] = bf16(v) (see preact_mode);  v = act(v);  v *= gelu'(mul_gelu_grad[m,n]) (see mul_mode);
 *   v *= dropout_mask(rng, drop_stream, m*N+n)/(1-p);  v *= rowscale[m / rows_per_scale];
 *   v += residual[m,n];  out[m,n] = v;  colsum[n] += sum_m v   (bias gradient of the producing layer) */
typedef struct MdvGemmEpi {
    const float* bias;          /* [N] fp32 or NULL */
    const float* residual;      /* [M, ld_res] fp32 or NULL */
    const void* mul_gelu_grad;  /* [M, ld_mul] bf16 pre-activation u, or NULL */
    void* out_preact;           /* [M, ld_preact] bf16 or NULL */
    void* out;                  /* [M, ldc] bf16 or fp32 */
    const float* rowscale;      /* [ceil(M / rows_per_scale)] fp32 or NULL (DropPath per-sample scale) */
    const void* rng;            /* device uint64[2] {seed, step}; may be NULL when dropout_p == 0 */
    float* colsum;              /* [N] fp32 or NULL: column sums of the stored values are ADDED here (atomics) */
    const float* colscale;      /* [N] fp32 or NULL: v = acc * colscale[n] + bias[n] instead of acc + bias[n] (eval-mode BatchNorm folded
                                   into the producing GEMM: colscale = gamma / sqrt(running_var + eps), bias = beta - mean * colscale) */
    int ld_res, ld_mul, ld_preact, ldc;
    int rows_per_scale;
    int out_bf16;               /* 1: out is bf16, 0: fp32 */
    int act;                    /* MDV_ACT_NONE | MDV_ACT_GELU | MDV_ACT_RELU | MDV_ACT_HSWISH */
    int accumulate;             /* fp32 out only: out += v */
    int preact_mode;            /* what out_preact receives: 0 = v before the activation; 1 = act'(v) * dropout_mask/(1-p), i.e. the
                                   exact factor the backward pass multiplies the incoming gradient by (saves recomputing it there) */
    int mul_mode;               /* how mul_gelu_grad is used: 0 = v *= gelu'(u[m,n]);  1 = v *= u[m,n] (u holds a preact_mode-1 factor) */
    float dropout_p;
    uint32_t drop_stream;
} MdvGemmEpi;

/* C[M,N] = epi(A[M,K] . W[N,K]^T); A, W bf16 row-major with pitches lda, ldw (elements, multiples of 8).
 * nn.Linear / 1x1 Conv2d forward (mdvit.py:288,310; mpvit.py:72-76; Decoders.py:59,197,317-333) and,
 * with W := W^T, their input gradients. */
int mdv_gemm_nt(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi, void* stream);

/* The same with fp32 operands multiplied as TF32 (tcgen05 kind::tf32: 10 mantissa bits instead of bf16's 7, fp32
 * accumulate); pitches in elements, multiples of 4.  Used for the convolutional trunk (stem, patch embeddings, bridge,
 * decoder 1x1 convs): every one of them rewrites the whole residual stream, so their operand rounding is what the logits
 * see — bf16 there put the logits 1.0-1.4e-2 from the reference at its random init, TF32 puts them at ~3e-3 (DESIGN.md
 * section 7); the transformer blocks' GEMMs, whose outputs are small additive branches, stay bf16. */
int mdv_gemm_nt_tf32(const float* A, int lda, const float* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi, void* stream);

/* mdv_gemm_nt_tf32 with one folded eval-mode BatchNorm set per SAMPLE (mixed-domain inference of the domain-specific-norm
 * models): epi->colscale and epi->bias are [S, N] tables, and row m uses row s = sample_set[m / rows_per_sample] of both,
 *   v = acc * colscale[s*N + n] + bias[s*N + n],  then the activation and the rest of the epilogue as above.
 * sample_set is a DEVICE int32 vector read by the kernel, so a captured CUDA graph serves any domain mix.  A row whose index is
 * outside [0, S) reads no table entry and is written as NaN.  S outside 1..8, rows_per_sample < 1, or a NULL sample_set /
 * colscale returns MDV_ERR_ARG before any CUDA call. */
int mdv_gemm_nt_tf32_sets(const float* A, int lda, const float* W, int ldw, int M, int N, int K, const MdvGemmEpi* epi,
                          const int* sample_set, int rows_per_sample, int S, void* stream);

/* 3x3 / stride 1 / padding 1 convolution of an NHWC activation as ONE implicit GEMM (no im2col matrix): the A tiles of the K = 9*Cin
 * reduction are fetched straight from x [B,H,W,Cin] (pixel pitch ldx) by 4-D TMA boxes, whose out-of-range zero fill is the padding:
 *   out[(b,y,x), n] = epi( sum_{tap=(i,j), c} x[b, y + s(i-1), x + s(j-1), c] . Wm[n, tap*Cin + c] ),   s = flip ? -1 : +1.
 * x fp32 (x_f32 = 1: TF32 math, Cin % 32 == 0) or bf16 (Cin % 64 == 0); Wm the same type, [N, ldw].  W <= 128 must divide 128 and
 * H*W must be a multiple of 128 (a 128-row tile = whole image rows), else MDV_ERR_UNSUPPORTED (callers fall back to mdv_im2col3).
 * Forward of the dense 3x3 convs of TransFuse_S_adapt (torchvision BasicBlock, DoubleConv / Conv, TransFuse.py:574-650) with
 * Wm = mdv_prep_weight mode 2; with flip = 1, x := dz and Wm = mdv_prep_weight mode 4 it is their input gradient. */
int mdv_conv3_gemm(const void* x, int x_f32, int ldx, const void* Wm, int ldw, int B, int H, int W, int Cin, int N, int flip,
                   const MdvGemmEpi* epi, void* stream);

/* Weight gradient of the same convolution, in the column order of mdv_prep_weight mode 2 (apply mdv_unperm_conv_grad):
 *   dWm[p, tap*Cin + c] += sum_{(b,y,x)} dz[(b,y,x), p] . x[b, y + i - 1, x + j - 1, c]
 * one TN GEMM whose B tiles are 4-D TMA boxes of x (bf16 NHWC, pixel pitch ldx); dz bf16 [B*H*W, P].  Cin % 64 == 0, W <= 64 must
 * divide 64, H*W % 64 == 0, else MDV_ERR_UNSUPPORTED. */
int mdv_conv3_wgrad(const void* dz_bf16, int ldz, const void* x_bf16, int ldx, int B, int H, int W, int Cin, int P, float* dWm, int ldc,
                    void* stream);

/* C[P,Q] += A[R,P]^T . B[R,Q]  (fp32 atomics; A, B bf16 row-major).  Weight gradients of the above. */
int mdv_gemm_tn(const void* A, int lda, const void* B, int ldb, int R, int P, int Q, float* C, int ldc, void* stream);

/* ------------------------------------------------------------------ fused MLP (two chained tcgen05 GEMMs, hidden tile on chip) */
/* 1 if mdv_mlp_fwd / mdv_mlp_bwd support this width (C in {64, 128}, hidden a multiple of 64, <= 2048). */
int mdv_mlp_supported(int C, int hidden);
/* Mlp.forward + the block's residual add (mpvit.py:71-78, mdvit.py:357-359) in ONE kernel:
 *   h = dropout1(GELU(a W1^T + b1));  out = residual + rowscale[m / rows_per_scale] * dropout2(h W2^T + b2)
 * a [M,C] bf16 (the LayerNorm output), w1 [hidden,C] bf16, w2 [C,hidden] bf16, residual/out [M,C] fp32.
 * hact_out / u_out ([M,hidden] bf16, both or neither may be NULL): h, and u = GELU'(.) * dropout1 mask/(1-p) — the tensors
 * the backward pass needs; NULL for inference, where the hidden activation then never leaves the SM. */
int mdv_mlp_fwd(const void* a_bf16, const void* w1_bf16, const float* b1, const void* w2_bf16, const float* b2, const float* residual,
                float* out, void* hact_out, void* u_out, int M, int C, int hidden, float drop_p, const void* rng, uint32_t drop_stream1,
                uint32_t drop_stream2, const float* rowscale, int rows_per_scale, void* stream);
/* Input gradient of the same: du = (dy W2) * u;  dx = du W1.   dy [M,C] bf16 (gradient of the fc2 output, masks applied),
 * w2t [hidden,C] bf16 (= W2^T), u [M,hidden] bf16 from mdv_mlp_fwd, w1t [C,hidden] bf16 (= W1^T), dx [M,C] fp32.
 * du_out ([M,hidden] bf16) and colsum1 ([hidden] += column sums of du = fc1 bias gradient) are needed only when weight
 * gradients are; both may be NULL (then du never leaves the SM). */
int mdv_mlp_bwd(const void* dy_bf16, const void* w2t_bf16, const void* u_bf16, const void* w1t_bf16, void* du_out, float* dx_out,
                float* colsum1, int M, int C, int hidden, void* stream);

/* Debug/tuning knob (0 = automatic): force tile N, pipeline stages, TN split count. */
int mdv_gemm_tune(int force_bn, int force_stages, int force_split);
/* Debug/test knob: -1 = automatic choice of the CTA-pair (tcgen05 cta_group::2) instantiation of mdv_gemm_nt, 0 / 1 = never / always
   (the automatic rule only picks pairs for large long-K problems; tests force them on small and ragged shapes as well). */
int mdv_gemm_force_pair(int mode);

/* ------------------------------------------------------------------ LayerNorm (mdvit.py:349,357; eps 1e-6) */
/* y = bf16(LN(x)); mean/rstd [M] are saved for backward.  C % 64 == 0, C <= 512. */
int mdv_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, void* y_bf16, float* mean,
                      float* rstd, int M, int C, void* stream);
/* dx = dres + LN'(dy); optional dx_masked = bf16(dx * rowscale[m/rows_per_scale] * dropout_mask) (the gradient of the
 * preceding Linear's output when proj_drop/DropPath sit between it and the residual add, mdvit.py:311,354);
 * dgamma/dbeta accumulate (+=). */
int mdv_layernorm_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                      const float* dres, float* dx, void* dx_masked_bf16, const float* rowscale, int rows_per_scale,
                      float drop_p, const void* rng, uint32_t drop_stream, float* dgamma, float* dbeta,
                      float* dbias_masked /* [C] += column sums of dx_masked, or NULL */, int M, int C, void* stream);

/* ------------------------------------------------------------------ row groups with norm parameter tables */
/* The stacked multi-domain pass runs G single-domain mini-batches as one [G*Mg, C] tensor; row group g = rows
 * [g*Mg, (g+1)*Mg) uses norm parameter set g.  A table names one tensor per group (p[g], g < G); it is passed by value, so a
 * captured CUDA graph holds the addresses and no host-to-device copy is needed.  1 <= G <= 8, else MDV_ERR_ARG before any
 * CUDA call.  Entries may repeat: one set named G times is a shared set (MDViT's stacked pass, TransFuse's dataset
 * groups), G distinct sets are domain-specific norms (MDViT_DSN / BASE_DSN).  Groups that name the same running buffers
 * update them in group order, and groups that name the same gradient target add to it, exactly as consecutive
 * single-set calls would. */
#define MDV_MAX_GROUPS 8
typedef struct MdvPtrTable {
    void* p[MDV_MAX_GROUPS];
} MdvPtrTable;

/* mdv_layernorm_fwd / mdv_layernorm_bwd with gamma[g], beta[g] for row group g.  dgamma[g] / dbeta[g] accumulate (+=) the
 * sums over group g only and may each be NULL; dbias_masked (a shared bias) is one [C] sum over all rows. */
int mdv_layernorm_fwd_gp(const float* x, MdvPtrTable gamma, MdvPtrTable beta, float eps, void* y_bf16, float* mean, float* rstd,
                         int G, int Mg, int C, void* stream);
/* mdv_layernorm_fwd with one parameter set per SAMPLE (mixed-domain inference): row m uses gamma[s], beta[s] with
 * s = sample_set[m / rows_per_sample], read on the device (DEVICE int32 vector).  A row whose index is outside [0, S) reads no
 * table entry and is written as NaN.  mean / rstd may be NULL (inference needs neither).  1 <= S <= 8, a gamma / beta for every
 * set, rows_per_sample >= 1 and a non-NULL sample_set, else MDV_ERR_ARG before any CUDA call. */
int mdv_layernorm_fwd_sets(const float* x, MdvPtrTable gamma, MdvPtrTable beta, float eps, void* y_bf16, float* mean, float* rstd,
                           const int* sample_set, int rows_per_sample, int S, int M, int C, void* stream);
int mdv_layernorm_bwd_gp(const float* dy, const float* x, const float* mean, const float* rstd, MdvPtrTable gamma,
                         const float* dres, float* dx, void* dx_masked_bf16, const float* rowscale, int rows_per_scale,
                         float drop_p, const void* rng, uint32_t drop_stream, MdvPtrTable dgamma, MdvPtrTable dbeta,
                         float* dbias_masked, int G, int Mg, int C, void* stream);
/* Train-mode BatchNorm2d (+act) on G row groups: group g normalises with its own batch statistics, gamma[g] and beta[g],
 * and updates running_mean[g], running_var[g] (momentum, unbiased variance) and *num_batches_tracked[g] += 1, as
 * nn.BatchNorm2d would on that mini-batch; dgamma[g] / dbeta[g] accumulate (+=) group g's sums.  Buffer and gradient entries
 * may be NULL.  mean/rstd: [G, C].  C % 4 == 0, 32 <= C <= 1024, G*Mg*C < 2^31, else MDV_ERR_UNSUPPORTED.
 * fwd ws >= 2*C*G doubles; bwd ws >= 2*C*G doubles + 2*C*G floats. */
int mdv_bn_train_fwd_gp(const float* z, int G, int Mg, int C, float eps, float momentum, MdvPtrTable running_mean,
                        MdvPtrTable running_var, MdvPtrTable num_batches_tracked, MdvPtrTable gamma, MdvPtrTable beta, int act,
                        float* mean, float* rstd, void* y, int y_bf16, void* ws, void* stream);
int mdv_bn_act_bwd_gp(const float* dy, const float* z, const float* mean, const float* rstd, MdvPtrTable gamma, MdvPtrTable beta,
                      int act, void* dz, int dz_bf16, MdvPtrTable dgamma, MdvPtrTable dbeta, int G, int Mg, int C, void* ws,
                      void* stream);

/* ------------------------------------------------------------------ BatchNorm2d (+act) on [M=B*H*W, C] (mpvit.py:119-122 ...) */
/* training: batch mean / biased var -> mean,rstd; running stats updated with momentum (unbiased var) and
 * *num_batches_tracked += 1 (mdv_bn_train_fwd_gp's statistics with G = 1: shapes outside its limits return
 * MDV_ERR_UNSUPPORTED).  eval: mean,rstd from the running buffers.  ws >= 2*C doubles. */
int mdv_bn_stats(const float* z, int M, int C, float eps, float momentum, int training, float* running_mean,
                 float* running_var, long long* num_batches_tracked, float* mean, float* rstd, void* ws, void* stream);
/* Eval-mode BatchNorm as a per-channel affine map folded into the GEMM that produces its input (MdvGemmEpi.colscale/bias):
 * scale[c] = gamma[c] / sqrt(running_var[c] + eps);  shift[c] = beta[c] + (conv_bias[c] - running_mean[c]) * scale[c]. */
int mdv_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var, const float* conv_bias,
                float eps, float* scale, float* shift, int C, void* stream);
/* mdv_bn_fold for S parameter sets in one launch: scale / shift are [S, C], row s from gamma[s], beta[s], running_mean[s],
 * running_var[s]; conv_bias ([C] or NULL) is shared by all sets.  mdv_bn_fold is the S = 1 call.  1 <= S <= 8 and every table
 * entry set, else MDV_ERR_ARG before any CUDA call. */
int mdv_bn_fold_sets(MdvPtrTable gamma, MdvPtrTable beta, MdvPtrTable running_mean, MdvPtrTable running_var, const float* conv_bias,
                     float eps, float* scale, float* shift, int S, int C, void* stream);
int mdv_bn_act_fwd(const float* z, const float* mean, const float* rstd, const float* gamma, const float* beta, int act,
                   void* y, int y_bf16, int M, int C, void* stream);
/* dz for y = act(BN_train(z)); ws >= 2*C doubles + 2*C floats; dgamma/dbeta accumulate.  mdv_bn_act_bwd_gp with G = 1:
 * shapes outside its limits return MDV_ERR_UNSUPPORTED. */
int mdv_bn_act_bwd(const float* dy, const float* z, const float* mean, const float* rstd, const float* gamma,
                   const float* beta, int act, void* dz, int dz_bf16, float* dgamma, float* dbeta, int M, int C, void* ws,
                   void* stream);
/* mdv_bn_act_bwd with a rank-1 output gradient dy[m,c] = dlog[m] * wrow[c] * dropout2d_mask(m / rows_per_sample, c) generated
 * on the fly: the backward of Dropout2d + the 1-channel `linear_out` head of MLPDecoderFM (Decoders.py:334-337) never
 * materialises the [M, C] gradient of the BatchNorm output.  M % rows_per_sample != 0 returns MDV_ERR_UNSUPPORTED.
 * (ws here: >= 3*C doubles + (M / rows_per_sample)*C floats) */
int mdv_bn_act_bwd_rank1(const float* dlog, const float* wrow, int rows_per_sample, float drop_p, const void* rng,
                         uint32_t drop_stream, const float* z, const float* mean, const float* rstd, const float* gamma,
                         const float* beta, int act, void* dz, int dz_bf16, float* dgamma, float* dbeta, int M, int C, void* ws,
                         void* stream);

/* ------------------------------------------------------------------ stencils (token-major / NHWC) */
/* depthwise 3x3, pad 1 (ConvPosEnc mpvit.py:244-246 with residual=1; patch-embed dwconv mdvit.py:118).
 * transposed=1 computes the input gradient of the same conv (in = output gradient on the Ho x Wo grid). */
int mdv_dwconv3(const float* in, const float* w, const float* bias, void* out, int out_bf16, int B, int Hi, int Wi, int Ho,
                int Wo, int C, int stride, int transposed, int residual, void* stream);
int mdv_dwconv3_wgrad(const float* dy, const float* x, float* dw, float* db, int B, int Hi, int Wi, int Ho, int Wo, int C,
                      int stride, void* stream);
/* decoder conv_after.dwconv: 3x3, groups=C over cat(skip, up) (2 inputs per group), Decoders.py:30-38,198-205 */
int mdv_gconv2_fwd(const float* skip, const float* up, const float* w, void* out, int out_bf16, int B, int H, int W, int C,
                   void* stream);
int mdv_gconv2_bwd(const float* dout, const float* skip, const float* up, const float* w, float* dskip, float* dup, float* dw,
                   int B, int H, int W, int C, void* stream);
/* im2col for dense 3x3 convs (stem mdvit.py:509-526, bridge :557-564): col[(b,yo,xo), (i*3+j)*C + c] */
int mdv_im2col3(const void* in, int in_bf16, void* col, int col_bf16, int B, int Hi, int Wi, int Ho, int Wo, int C, int stride,
                int ldc, void* stream);
/* col: [B*Ho*Wo, 64] bf16 (col_bf16 = 1) or [B*Ho*Wo, 32] fp32 (col_bf16 = 0), 27 columns used, the rest zero */
int mdv_im2col_stem(const float* img_nchw, void* col, int col_bf16, int B, int Hi, int Wi, void* stream);
int mdv_col2im3(const float* dcol, float* dx, int B, int Hi, int Wi, int Ho, int Wo, int C, int stride, int ldc, void* stream);
/* dilated 3x3 convs of the DeepLabV3 auxiliary decoder's ASPP (Utils/_deeplab.py:115-122, Decoders.py:218-235): stride 1,
   padding = dilation, same size; col is bf16 [B*H*W, 9*C]; the transpose optionally accumulates into dx */
int mdv_im2col3_dil(const void* in, int in_bf16, void* col, int B, int H, int W, int C, int dil, int ldc, void* stream);
int mdv_col2im3_dil(const float* dcol, float* dx, int B, int H, int W, int C, int dil, int ldc, int accumulate, void* stream);
/* bilinear resize, align_corners=False (mdvit.py:699; Decoders.py:196,319-336) and its exact transpose */
int mdv_upsample_fwd(const void* in, int in_bf16, int ld_in, void* out, int out_bf16, int ld_out, int B, int Hi, int Wi, int Ho,
                     int Wo, int C, void* stream);
/* out[b,y,x,c] += sum_k resize(in_k)[b,y,x,c] (align_corners=False) for up to three fp32 maps in_k [B,Hk,Wk,C] (NULL: skipped),
 * one pass over out [B,Ho,Wo] with pixel pitch ld_out: the upsampled stage-2..4 terms of the collapsed MLPDecoderFM
 * (Decoders.py:317-333, see ops.AuxFn).  C, ld_out % 4 == 0, pointers 16-byte aligned. */
int mdv_upsample_add(float* out, int ld_out, int B, int Ho, int Wo, int C, const float* in0, int H0, int W0, const float* in1, int H1,
                     int W1, const float* in2, int H2, int W2, void* stream);
/* ws: optional scratch of B*Ho*Wi*C floats; with it, integer factors 4 and 8 use the separable two-pass form */
int mdv_upsample_bwd(const void* dout, int dout_bf16, int ld_out, float* din, int ld_in, int B, int Hi, int Wi, int Ho, int Wo,
                     int C, float* ws, void* stream);

/* ------------------------------------------------------------------ factorized attention + CRPE + DA gate */
long long mdv_attn_stats_floats(int B, int C, int heads); /* floats of `stats` (column max, softmax denominators, K^T V): kept for backward */
long long mdv_attn_ws_floats(int B, int C, int heads);    /* floats of scratch `ws` one forward or backward call needs */
/* FactorAtt_ConvRelPosEnc(_Sup).forward between the qkv and proj Linears (mdvit.py:288-304, mpvit.py:296-318).
 * qkv bf16 [B,N,3C]; gate fp32 [B,C] or NULL (non-'Sup' attention, mpvit.py:347-373); out bf16 [B,N,C]. */
int mdv_attn_fwd(const void* qkv_bf16, const float* gate, const float* crpe_w3, const float* crpe_b3, const float* crpe_w5,
                 const float* crpe_b5, const float* crpe_w7, const float* crpe_b7, float* stats, float* ws, void* out_bf16,
                 void* e_out_bf16 /* [B,N,C] bf16 or NULL: dwconv(V)+b, kept for mdv_attn_bwd */, int B, int H, int W, int C, int heads,
                 void* stream);
/* dqkv and dgate are overwritten; the CRPE gradients accumulate (the six CRPE gradient pointers may all be NULL: skipped). */
int mdv_attn_bwd(const void* qkv_bf16, const void* dy_bf16, const void* y_bf16, const void* e_bf16, const float* gate, const float* crpe_w3,
                 const float* crpe_b3, const float* crpe_w5, const float* crpe_b5, const float* crpe_w7, const float* crpe_b7,
                 const float* stats, void* dqkv_bf16, float* dgate, float* dcrpe_w3, float* dcrpe_b3, float* dcrpe_w5,
                 float* dcrpe_b5, float* dcrpe_w7, float* dcrpe_b7,
                 float* dbias_qkv /* [3C] += column sums of dqkv (bias gradient of the qkv Linear), or NULL */, float* ws, int B,
                 int H, int W, int C, int heads,
                 void* stream);
/* DA: gate[b,h,v] = softmax_h( W2 relu(W1 label_b + b1) + b2 )  (mdvit.py:272-276,301-303) */
int mdv_da_gate_fwd(const float* label, const float* w1, const float* b1, const float* w2, const float* b2, float* hid_out,
                    float* gate, int B, int nd, int hid, int C, int heads, void* stream);
int mdv_da_gate_bwd(const float* label, const float* w2, const float* hid_in, const float* gate, const float* dgate, float* dw1,
                    float* db1, float* dw2, float* db2, float* ws /* B*(C+hid) floats */, int B, int nd, int hid, int C, int heads,
                    void* stream);

/* ------------------------------------------------------------------ softmax(Q K^T) V attention + DA gate (TransFuse_S_adapt's DeiT branch) */
/* Attention_Sup.forward between its qkv and proj Linears (Models/Hybrid_models/TransFuseFolder/vision_transformer.py:149-169):
 *   out[b,n,h*64+v] = gate[b,h*64+v] * sum_m softmax_m(scale * q[b,h,n,:].k[b,h,m,:]) v[b,h,m,v]
 * qkv bf16 [B,N,3C] (rows q | k | v, heads contiguous inside each, as nn.Linear(dim, 3*dim) lays them out), gate fp32 [B,C]
 * from mdv_da_gate_fwd (softmax over heads) or NULL (plain Attention, vision_transformer.py:110-122), out bf16 [B,N,C].
 * lse (optional, [B,heads,N] fp32) receives the row log-sum-exp for a backward pass.  head_dim 64, N in {128, 256}. */
int mdv_sdpa_fwd(const void* qkv_bf16, const float* gate, void* out_bf16, float* lse, int B, int N, int C, int heads, float scale,
                 void* stream);
/* Its backward (what autograd runs for vision_transformer.py:155-166): dqkv bf16 [B,N,3C] (rows dq | dk | dv) from dout bf16
 * [B,N,C], the forward's out and lse; dgate fp32 [B,C] (optional, written: feed it to mdv_da_gate_bwd).  P is recomputed. */
int mdv_sdpa_bwd(const void* qkv_bf16, const float* gate, const void* out_bf16, const float* lse, const void* dout_bf16,
                 void* dqkv_bf16, float* dgate, int B, int N, int C, int heads, float scale, void* stream);

/* ------------------------------------------------------------------ TransFuse_S_adapt: CNN branch, fusion and decoder (Models/Hybrid_models/TransFuseFolder/TransFuse.py:182-283) */
/* Generic k x k im2col of an fp32 NHWC tensor (in_nchw = 1: the NCHW input image, resnet.conv1 TransFuse.py:231):
 *   col[(b,yo,xo), c*k*k + i*k + j] = in[b, yo*stride - pad + i, xo*stride - pad + j, c], zero outside the image and in the
 * columns [C*k*k, ldc).  The column order is that of the flattened nn.Conv2d weight, so the GEMM's W operand is the parameter.
 * Used for the 7x7 stride-2 stem, the 1x1 stride-2 downsample convs (torchvision resnet34) and BiFusion_block.spatial (7x7 on 2
 * channels, TransFuse.py:38); the 3x3 convs use mdv_im2col3. */
int mdv_im2col_k(const float* in, int in_nchw, void* col, int col_bf16, int B, int Hi, int Wi, int Ho, int Wo, int C, int k, int stride,
                 int pad, int ldc, void* stream);
/* its transpose (input gradient): dx NHWC fp32 [B,Hi,Wi,C], overwritten */
int mdv_col2im_k(const float* dcol, float* dx, int B, int Hi, int Wi, int Ho, int Wo, int C, int k, int stride, int pad, int ldc,
                 void* stream);
/* nn.MaxPool2d(3, stride 2, padding 1) on NHWC fp32 (resnet.maxpool, TransFuse.py:234); tap_u8 [B,Ho,Wo,C] keeps which of the 9
 * taps won (first maximum in scan order, where nn.MaxPool2d sends the gradient).  Ho = (Hi-1)/2 + 1.  C % 4 == 0. */
int mdv_maxpool3s2_fwd(const float* in, float* out, void* tap_u8, int B, int Hi, int Wi, int C, void* stream);
int mdv_maxpool3s2_bwd(const float* dout, const void* tap_u8, float* din, int B, int Hi, int Wi, int C, void* stream);
/* out = act(a + b), act in {NONE, RELU}: `out += identity; relu(out)` of the ResNet BasicBlock, DoubleConv (TransFuse.py:589) and
 * Attention_block (TransFuse.py:617).  n % 4 == 0. */
int mdv_add_act(const float* a, const float* b, float* out, long long n, int act, void* stream);
/* dx = dy * [y > 0] with y the ReLU's OUTPUT */
int mdv_relu_bwd(const float* dy, const float* y, float* dx, long long n, void* stream);
/* bilinear resize with align_corners=True on NHWC fp32 (nn.Upsample in Up, TransFuse.py:559; the three output maps,
 * TransFuse.py:262-264) and its exact transpose (gather form, deterministic) */
int mdv_resize_ac_fwd(const float* in, float* out, int B, int Hi, int Wi, int Ho, int Wo, int C, void* stream);
int mdv_resize_ac_bwd(const float* dout, float* din, int B, int Hi, int Wi, int Ho, int Wo, int C, void* stream);
/* Gates of BiFusion_block / Attention_block and the concat that follows them, one pass (TransFuse.py:63-73,620):
 *   out[m, :] = [ g[m, :C1] * pgate[m]  |  x[m, :C2] * vgate[m / rows_per_sample, :C2]  |  bp[m, :C3] ]
 * pgate [M] (spatial / psi gate) and vgate [B, C2] (squeeze-and-excitation gate) are the values AFTER their sigmoids.  C2 = C3 = 0
 * (x, vgate, bp NULL) is Attention_block's `x * psi`.  Channel counts % 4 == 0, C2 <= 512.
 * _bwd: dg = dout1 * pgate, dp[m] = sum_c dout1 g, dx = dout2 * vgate, dv[b, c] = sum_{m in b} dout2 x (written), dbp = dout3. */
int mdv_gate_cat_fwd(const float* g, const float* pgate, const float* x, const float* vgate, const float* bp, float* out, int M, int C1,
                     int C2, int C3, int rows_per_sample, void* stream);
int mdv_gate_cat_bwd(const float* dout, const float* g, const float* pgate, const float* x, const float* vgate, float* dg, float* dp, float* dx,
                     float* dv, float* dbp, int M, int C1, int C2, int C3, int rows_per_sample, void* stream);
/* ChannelPool (TransFuse.py:20-22): out[m] = (max_c x[m,c], mean_c x[m,c]); arg_i32 [M] = first maximal channel (torch.max's gradient
 * routing).  _bwd: dx[m,c] = dout[m,1] / C + (c == arg[m]) dout[m,0]. */
int mdv_channel_pool_fwd(const float* x, float* out, void* arg_i32, int M, int C, void* stream);
int mdv_channel_pool_bwd(const float* dout, const void* arg_i32, float* dx, int M, int C, void* stream);
/* nn.Dropout2d (TransFuse.py:217,226-245) on an NHWC map: out = x * mask(b, c) / (1 - p), mask a function of (rng, drop_stream, b*C + c);
 * the backward is the same call on the gradient.  C % 4 == 0. */
int mdv_dropout2d(const float* x, float* out, int M, int C, int rows_per_sample, float p, const void* rng, uint32_t drop_stream, void* stream);
/* structure_loss (multi_train_TransFuse.py:29-38): weit = 1 + 5 |avg_pool2d(mask, 31, 1, 15) - mask| (ws: B*H*W floats);
 * loss = mean_b( sum(weit*bce)/sum(weit) + 1 - (I+1)/(U-I+1) ), I = sum(sigmoid(pred)*mask*weit), U = sum((sigmoid(pred)+mask)*weit).
 * sums: DEVICE double[4*B] (per sample: sum weit, sum weit*bce, I, U), written by _fwd, read by _bwd;
 * dpred (=|+=) gout[0] * coef * dloss/dpred  (gout may be NULL = 1). */
int mdv_structure_weit(const float* mask, float* weit, float* ws, int B, int H, int W, void* stream);
int mdv_structure_loss_fwd(const float* pred, const float* mask, const float* weit, void* sums, float* loss, int B, int HW, void* stream);
int mdv_structure_loss_bwd(const float* pred, const float* mask, const float* weit, const void* sums, const float* gout, float coef,
                           float* dpred, int B, int HW, int accumulate, void* stream);

/* ------------------------------------------------------------------ heads, reductions, casts */
/* logits[m] = sum_c x[m,c] w[c] dropout2d(b,c) + bias  — the C->1 1x1 conv commuted in front of the final resize */
int mdv_rowdot_fwd(const void* x, int x_bf16, const float* w, const float* bias, float* out, int M, int C, int rows_per_sample,
                   float drop_p, const void* rng, uint32_t drop_stream, void* stream);
int mdv_rowdot_bwd(const float* dlog, const void* x, int x_bf16, const float* w, float* dx, float* dw, float* db, int M, int C,
                   int rows_per_sample, float drop_p, const void* rng, uint32_t drop_stream, void* stream);
int mdv_colsum(const void* x, int x_bf16, int ld, float* out, int M, int C, void* stream);  /* out[c] += sum_m x[m,c] */
/* out = bf16(in * rowscale[m / rows_per_scale] * dropout_mask(m*C + c)); colsum (optional, C <= 1024): [C] += column sums of out */
int mdv_cast_bf16(const float* in, int ld_in, void* out_bf16, int ld_out, long long M, int C, const float* rowscale,
                  int rows_per_scale, float drop_p, const void* rng, uint32_t drop_stream, float* colsum, void* stream);
int mdv_add_f32(const void* in, int in_bf16, int ld_in, float* out, int ld_out, long long M, int C, int accumulate, void* stream);
/* Up to 16 independent fp32 FFMA products in one launch (`descs`: HOST array of n descriptors, distinct C):
 *   C[M,N] = (accumulate ? C : 0) + op(A)[M,K] . op(B)[K,N] (+ u[m] v[n] when u, v are not NULL),
 * op(A)[m,k] = trans_a ? A[k*lda + m] : A[m*lda + k], op(B) likewise.  The weight-sized products of the collapsed MLPDecoderFM
 * (ops.AuxFn): Wf_i W_i and Wf_i b_i in the forward; E_i W_i^T + s b_i^T, Wf_i^T E_i and Wf_i^T s for the weight gradients. */
typedef struct MdvMatmulDesc {
    const float* A;
    const float* B;
    float* C;
    const float* u;
    const float* v;
    int lda, ldb, ldc, M, N, K, trans_a, trans_b, accumulate, pad_;
} MdvMatmulDesc;
int mdv_matmul_f32_grouped(const MdvMatmulDesc* descs, int n, void* stream);
/* fp32 master weight -> GEMM operand.  mode 0 copy, 1 transpose, 2 conv3x3 -> im2col order, 3 = transpose of 2, 4 = conv3x3 ->
 * [Cin, tap*Cout + co] (input-gradient operand of mdv_conv3_gemm); dst is bf16, or
 * fp32 (TF32 GEMM operand) when 8 is added to the mode */
int mdv_prep_weight(const float* src, void* dst, int R, int Cc, int ld, int mode, int cin, void* stream);
/* The same for a whole model in one launch: `descs_dev` is a DEVICE array of n descriptors (zero-padded dst regions are
 * the caller's job, as with mdv_prep_weight). */
typedef struct MdvPrepDesc {
    const float* src;
    void* dst;
    int rows, cols, ld, mode, cin, pad_;
} MdvPrepDesc;
int mdv_prep_weights_batched(const MdvPrepDesc* descs_dev, int n, void* stream);
int mdv_unperm_conv_grad(const float* g, int ld, float* dw, int R, int cin, void* stream);

/* ------------------------------------------------------------------ losses (multi_train_MDViT.py:147-169, Utils/losses.py:8-16) */
/* sums: 8 doubles {bce(p,y), bce(q,y), p.y, p.p, y.y, q.y, q.q, q.p}; all-reduce them across ranks for the global Dice. */
/* label: fp32 [n] (label_u8 = 0; the reference's label.cuda().float(), multi_train_MDViT.py:136) or uint8 {0,1} (label_u8 = 1) */
int mdv_loss_sums(const float* out, const float* aux, const void* label, int label_u8, void* sums, long long n, void* stream);
int mdv_loss_finalize(const void* sums, double n_total, float* losses /* seg, aux, kt */, void* stream);
int mdv_loss_bwd(const float* out, const float* aux, const void* label, int label_u8, const void* sums, double n_total,
                 const float* coef, float* dout, float* daux, long long n, void* stream);

/* Dice / Jaccard metrics of the trainer (multi_train_MDViT.py:172-177 calls medpy dc/jc on output.cpu().numpy() > 0.5, one
 * host sync per domain per step): counts (DEVICE uint64[3]) += {|P & L|, |P|, |L|} with P = logits > 0 (== sigmoid > 0.5),
 * L = label > 0.5.  dc = 2 c0 / (c1 + c2), jc = c0 / (c1 + c2 - c0); integer counts: bit-exact vs the host metric. */
int mdv_seg_counts(const float* logits, const void* label, int label_u8, void* counts, long long n, void* stream);

/* ------------------------------------------------------------------ optimizer / RNG */
/* One torch.optim.AdamW step (multi_train_MDViT.py:93-94,213) over a flat fp32 buffer.  hyper: DEVICE fp64[8] = {lr, beta1,
 * beta2, eps, weight_decay, t, unused, grad_scale}; the call first bumps t (steps taken) on the device, then applies step t:
 * the bias corrections 1-beta^t are computed on the device, so a captured CUDA graph replays correctly with no host input. */
int mdv_adamw(float* p, const float* g, float* m, float* v, void* hyper, long long n, void* stream);
int mdv_rng_bump(void* rng /* device uint64[2] {seed, step} */, void* stream);
int mdv_droppath_scale(float* scale, int B, float p, const void* rng, uint32_t drop_stream, void* stream);

#ifdef __cplusplus
}
#endif
#endif
