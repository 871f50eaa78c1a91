/* libgalerkin_b200 -- C ABI of the B200-native (sm_100a) Galerkin/Fourier attention encoder and
 * spectral-convolution decoder operators.
 *
 * The reference (scaomath/galerkin-transformer) has no FFI: its hot path is eager PyTorch.  Each
 * entry point below therefore cites the reference Python lines it replaces; INTEGRATION.md
 * shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to fp32 data unless the name says otherwise; the
 *     caller (PyTorch) owns every buffer including outputs and workspaces; the library never
 *     allocates device memory and never synchronises the host;
 *   - `device` is the CUDA ordinal the buffers live on, `stream` a cudaStream_t passed as void*;
 *     all work is enqueued on that stream and is CUDA-graph capturable;
 *   - return value: 0 (GB200_OK) on success, non-zero otherwise with a human-readable message
 *     from gb200_last_error() (thread-local); no exception ever crosses the boundary;
 *   - matrices are row-major; `ld*` are row strides in floats;
 *   - split reductions are two-stage with a fixed summation order: results are run-to-run
 *     deterministic.
 */
#ifndef GALERKIN_B200_H_
#define GALERKIN_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GB200_OK 0
#define GB200_ERR_INVALID 1
#define GB200_ERR_CUDA 2

#define GB200_ACT_NONE 0
#define GB200_ACT_RELU 1
#define GB200_ACT_SILU 2

int gb200_version(void);
const char* gb200_last_error(void);
/* Number of kernels this library has launched since load (all threads). */
unsigned long long gb200_launch_count(void);
/* Graph-safe dropout: every fused-dropout kernel adds *device_counter (read on the device at run time) to
 * its Philox seed.  Bumping the counter with a kernel inside a captured CUDA graph gives every replay fresh
 * masks while forward and backward of one step still agree.  NULL (default) disables the offset. */
int gb200_set_rng_offset_ptr(const unsigned long long* device_counter);

/* dst = concat(srcs[0..n)) in one launch (n <= 64; srcs / sizes are HOST arrays of device pointers / element counts).
 * Assembles W_qkv, b_qkv and the per-head LayerNorm tables from the reference's separate parameters
 * (libs/layers.py:810-811, 945-946) without torch.cat / torch.stack kernels. */
int gb200_pack(int device, float* dst, const float* const* srcs, const long long* sizes, int n, void* stream);

/* ------------------------------------------------------------------ dense layers ------------
 * C[b] = R[b] + rscale * dropout_p( act( alpha * op(A[b]) . op(B[b]) + bias ) )   (+= C if accumulate)
 *   op(A): transA ? A stored [K,M] : A stored [M,K];  op(B): transB ? B stored [N,K] : B stored [K,N]
 *   Zout (optional): receives the pre-activation (alpha*AB + bias), needed by SiLU backward
 *   dropout: Philox4x32-10 keyed by (seed, element index); the same key in backward regenerates
 *            the mask, no mask tensor exists
 * Replaces nn.Linear forward/backward on the hot path: libs/layers.py:837-839 (Q,K,V), :896-897
 * (fc), :980-986 (FeedForward), :1083 and :1172 (SpectralConv residual), libs/model.py:615-617,
 * :629 (SpectralRegressor fc / regressor), and the residual adds of libs/model.py:124-132. */
size_t gb200_gemm_workspace_bytes(int M, int N, int K, int nbatch, int ksplit);
int gb200_gemm_suggest_ksplit(int M, int N, int K, int nbatch);
int gb200_gemm(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB,
               float* C, int ldc, int M, int N, int K, int nbatch, long long strideA,
               long long strideB, long long strideC, float alpha, const float* bias, int act,
               float* Zout, int ldz, float drop_p, unsigned long long seed, const float* R, int ldr,
               float rscale, int accumulate, int ksplit, float* workspace, size_t workspace_bytes,
               void* stream);

/* Same contract as gb200_gemm (single batch), executed on the 5th-generation tensor cores:
 * TMA-staged SWIZZLE_128B tiles, tcgen05.mma kind::tf32 (fp32 operands read as TF32, fp32 accumulate in
 * TMEM), all four operand layouts without transpose copies, deterministic split-K.  Requires 16-byte
 * aligned operands with lda, ldb multiples of 4 and N, K >= 8 (gb200_gemm_tc_supported); otherwise call
 * gb200_gemm.  Relative error ~4e-4 per contraction (TF32), see DESIGN.md. */
int gb200_gemm_tc_supported(const float* A, int lda, const float* B, int ldb, int M, int N, int K);
int gb200_gemm_tc_suggest_ksplit(int M, int N, int K);
/* Diagnostics: when `device_buffer` is non-null every CTA of subsequent gb200_gemm_tc launches writes eight
 * %globaltimer stamps (entry, setup done, first/last tile landed, last tile rounded, accumulator complete,
 * TMEM drained, stores issued) to device_buffer[8 * linear_cta + slot].  Null (default) disables it. */
int gb200_gemm_tc_set_trace(unsigned long long* device_buffer);
/* split != 0 runs the GEMM in split ("3xTF32") arithmetic -- each product is hi.hi + hi.lo + lo.hi of the two-term TF32
 * split of its fp32 operands (~2^-22 relative error): the tensor-core path of the forward / input-gradient GEMMs in 'x3'
 * precision mode where no fused kernel applies.  Same for gb200_gemm_tc_gated. */
int gb200_gemm_tc(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB,
                  float* C, int ldc, int M, int N, int K, float alpha, const float* bias, int act,
                  float* Zout, int ldz, float drop_p, unsigned long long seed, const float* R, int ldr,
                  float rscale, int accumulate, int ksplit, float* workspace, size_t workspace_bytes,
                  int split, void* stream);

/* Grouped weight gradients: dW_i (M_i, N_i) = G_i^T X_i, i < n <= 6, each a contraction over all T_i rows (tokens), as ONE
 * tcgen05 TF32 split-K grid plus ONE fixed-order reduction -- the four weight gradients of an encoder layer
 * (libs/layers.py:837-839, :896-897, :980-986 in backward) fill the GPU together instead of queueing as eight launches. */
typedef struct gb200_wgrad_problem {
    const float* G; int ldg;        /* (T, M) gradient w.r.t. the layer output */
    const float* X; int ldx;        /* (T, N) layer input */
    float* dW; int ldw;             /* (M, N) */
    int M, N; long long T;
} gb200_wgrad_problem;
size_t gb200_gemm_tc_wgrad_group_workspace_bytes(int n, const gb200_wgrad_problem* probs);
int gb200_gemm_tc_wgrad_group(int device, int n, const gb200_wgrad_problem* probs, float* workspace, size_t workspace_bytes,
                              void* stream);

/* Gated GEMM: C = rscale * dropout_p( (alpha * op(A).op(B)) * act'(gate) ), gate_act = GB200_ACT_RELU (keep where
 * gate > 0; `gate` may be the stored post-activation/post-dropout output) or GB200_ACT_SILU (times silu'(gate), `gate`
 * = stored pre-activation).  With (seed, drop_p, rscale) of the forward layer this is "input gradient of layer i+1,
 * pushed through the activation and dropout of layer i" in one launch -- the elementwise backward between
 * lr2 and lr1 of FeedForward (libs/layers.py:980-986) and between `out` and the hidden layer of the regressor
 * (libs/model.py:629).  gb200_gemm_gated is the exact-fp32 / odd-shape path (N = 1 head: a rank-1 streaming kernel). */
int gb200_gemm_tc_gated(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB,
                        float* C, int ldc, int M, int N, int K, float alpha, float drop_p, unsigned long long seed,
                        float rscale, const float* gate, int ldg, int gate_act, int ksplit, float* workspace,
                        size_t workspace_bytes, int split, void* stream);
int gb200_gemm_gated(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB,
                     float* C, int ldc, int M, int N, int K, float alpha, float drop_p, unsigned long long seed,
                     float rscale, const float* gate, int ldg, int gate_act, int ksplit, float* workspace,
                     size_t workspace_bytes, void* stream);

/* out[n] (+)= scale * sum_m X[m,n]            (bias gradients) */
size_t gb200_colsum_workspace_bytes(long long M, int N);
int gb200_colsum(int device, const float* X, int ld, long long M, int N, float scale, int accumulate,
                 float* out, float* workspace, size_t workspace_bytes, void* stream);

/* g = dy * rscale * dropmask(p, seed) * act'(.)   -- backward of the gb200_gemm epilogue.
 * ReLU uses z if given, else the stored output y; SiLU needs z. */
int gb200_epilogue_bwd(int device, const float* dy, int lddy, const float* z, int ldz, const float* y,
                       int ldy, float* g, int ldg, long long M, int N, int act, float rscale,
                       float drop_p, unsigned long long seed, void* stream);

/* same, fused with the bias gradient dbias[n] = sum_m g[m,n] (one pass over g instead of three) */
size_t gb200_epilogue_bwd_bias_workspace_bytes(long long M, int N);
int gb200_epilogue_bwd_bias(int device, const float* dy, int lddy, const float* z, int ldz, const float* y, int ldy,
                            float* g, int ldg, long long M, int N, int act, float rscale, float drop_p,
                            unsigned long long seed, float* dbias, float* workspace, size_t workspace_bytes,
                            void* stream);

/* row LayerNorm over the last dimension (post-LN encoder variant, libs/model.py:128-129, 134-135) */
int gb200_layernorm_fwd(int device, const float* x, long long rows, int width, const float* gamma,
                        const float* beta, float eps, float* y, float* mean, float* rstd, void* stream);
size_t gb200_layernorm_bwd_workspace_bytes(long long rows, int width);
int gb200_layernorm_bwd(int device, const float* dy, const float* x, const float* mean, const float* rstd,
                        const float* gamma, long long rows, int width, float* dx, float* dgamma,
                        float* dbeta, int accumulate, float* workspace, size_t workspace_bytes,
                        void* stream);

/* ------------------------------------------------------------------ attention core ----------
 * Token-major "augmented head operand": row t, head h reads
 *     [ pos[t,0..p) , gamma[h,:] * X[t, col0 + h*dk + :] + beta[h,:] ]      (augmented == 0)
 *     X[t, col0 + h*(p+dk) + :]                                              (augmented == 1)
 * which is what libs/layers.py:846-874 builds with per-head LayerNorm modules, torch.stack,
 * pos.repeat and torch.cat -- here nothing of that is materialised. */
typedef struct gb200_head_operand {
    const float* ptr;
    int ld;
    int col0;
    int augmented;
    const float* gamma; /* (H, dk) or NULL */
    const float* beta;  /* (H, dk) or NULL */
} gb200_head_operand;

/* per-head LayerNorm statistics: x[t, col0 + h*dk + :] <- (x - mean) * rstd in place; rstd (T,H).
 * A second operand block (col0b >= 0, rstd_b) is normalised by the same launch: Galerkin normalises K and V,
 * Fourier Q and K.  libs/layers.py:846-851, 859-864 (the affine part is applied on load by the kernels below) */
int gb200_headnorm_fwd(int device, float* x, int ld, int col0, int col0b, long long T, int H, int dk, float eps,
                       float* rstd, float* rstd_b, void* stream);
size_t gb200_headnorm_bwd_workspace_bytes(long long T, int H, int dk);
/* dy (grad w.r.t. gamma*xhat+beta) is overwritten by the grad w.r.t. the un-normalised rows; *_b = second block
 * (dcol0b < 0: absent) */
int gb200_headnorm_bwd(int device, float* dy, int lddy, int dcol0, int dcol0b, const float* xhat, int ldx, int xcol0,
                       int xcol0b, const float* rstd, const float* rstd_b, const float* gamma, const float* gamma_b,
                       long long T, int H, int dk, float* dgamma, float* dbeta, float* dgamma_b, float* dbeta_b,
                       int accumulate, float* workspace, size_t workspace_bytes, void* stream);

/* tensor_cores != 0 (and d_k+p <= 64): operands rounded to TF32 (cvt.rna) and contracted with warp-level
 * mma.sync.m16n8k8 (fp32 accumulate), tiles right-sized to d; 0: exact-fp32 SIMT FMAs.
 * out[b,h,i,j] = scale * drop[b,h,i,j] * sum_t L~[b,t,h,i] * R~[b,t,h,j], where drop is
 *   2*keep_mask (explicit uint8 keep-mask), else the in-kernel Philox draw with keep-probability 1-mask_p scaled
 *   by 1/(1-mask_p) (mask_p = 0.5 reproduces F.dropout(p_attn), libs/layers.py:730-731; the same mask_seed in
 *   backward regenerates the same mask), else 1 (mask_p = 0).
 * forward: A = K~^T V~ / n with the reference's always-on p=0.5 dropout as an explicit keep-mask
 * (libs/layers.py:723, 728, 730-731); backward: dA = Q~^T dO. */
int gb200_attn_suggest_nsplit(int B, int H, int n);
size_t gb200_attn_xty_workspace_bytes(int B, int H, int d, int nsplit);
int gb200_attn_xty(int device, const gb200_head_operand* L, const gb200_head_operand* R, const float* pos,
                   int B, int H, int n, int dk, int p, float scale, const unsigned char* keep_mask, float mask_p,
                   unsigned long long mask_seed, float* out, int nsplit, float* workspace,
                   size_t workspace_bytes, int tensor_cores, void* stream);
/* out[e] = 0 or 1/(1-p): the scale tensor of the in-kernel dropout stream (seed, element index) */
int gb200_philox_scale(int device, float* out, long long total, float p, unsigned long long seed, void* stream);

/* out[b,t,h,:] = out_scale * L~[b,t,h,:] . (transM ? M[b,h]^T : M[b,h])
 * out_augmented: written head-merged as (T, H*(p+dk)) -- libs/layers.py:733, 892-894;
 * else the p position columns are dropped and (T, ldo) is written at ocol0 + h*dk (gradients). */
int gb200_attn_xm(int device, const gb200_head_operand* L, const float* pos, const float* M, int transM,
                  int B, int H, int n, int dk, int p, float* out, int ldo, int ocol0, int out_augmented,
                  float out_scale, int tensor_cores, void* stream);

/* Quadratic-form Fourier-type attention, out = drop(Q~ K~^T * scale) V~ with scale = 1/(sqrt(d) n), flash-style
 * (the (B,H,n,n) matrix is only written if attn_or_null is given).  Used when an n x n dropout sits between the
 * products: explicit uint8 keep-mask (B,H,n,n) or the in-kernel Philox draw (mask_p, mask_seed), which reproduces
 * F.dropout(p_attn) of libs/layers.py:698-703; backward regenerates the same mask.  d_k + p <= 64.
 * fwd: out (T, H*(p+dk)) head-merged;  bwd: dqkv (T, ld) receives dQ~, dK~, dV~ (position columns dropped) at the
 * given column offsets, given dO in the head-merged layout. */
int gb200_fourier_quad_fwd(int device, const gb200_head_operand* q, const gb200_head_operand* k,
                           const gb200_head_operand* v, const float* pos, int B, int H, int n, int dk, int p,
                           float scale, const unsigned char* keep_mask, float mask_p, unsigned long long mask_seed,
                           float* out, float* attn_or_null, void* stream);
int gb200_fourier_quad_bwd(int device, const gb200_head_operand* q, const gb200_head_operand* k,
                           const gb200_head_operand* v, const gb200_head_operand* dO, const float* pos, int B, int H,
                           int n, int dk, int p, float scale, const unsigned char* keep_mask, float mask_p,
                           unsigned long long mask_seed, float* dqkv, int ld, int qcol0, int kcol0, int vcol0,
                           void* stream);

/* ------------------------------------------------------------------ spectral convolution ----
 * Mode-truncated DFT pipeline replacing rfft/rfft2 -> mode slice -> complex einsum -> zero pad ->
 * irfft/irfft2 (libs/layers.py:1086-1101, 1175-1189).  Complex buffers are interleaved (re,im).
 * twY: (m, n, 2) = (cos, sin)(2 pi ky Y / n);  twX: (2m, n, 2) for kx(r) = r (r<m) | n-2m+r.
 * tensor_cores != 0: the two grid-sized stages (ydft, yidft_epilogue) run as per-row TF32 products against the
 * twiddle matrix on warp-level mma.sync (operands rounded with cvt.rna, fp32 accumulate); 0: exact fp32 FMAs. */
int gb200_spectral_suggest_ysplit(long long R, int C, int n);
size_t gb200_spectral_ydft_workspace_bytes(long long R, int C, int m, int nsplit);
/* out[R,ky,c] = scale * (hermitian ? c_ky : 1) * sum_Y x[R,Y,c] e^{-i 2pi ky Y/n} */
int gb200_spectral_ydft(int device, const float* x, long long R, int n, int C, int m, const float* twY,
                        float scale, int hermitian, float* out, int nsplit, float* workspace,
                        size_t workspace_bytes, int tensor_cores, void* stream);
/* inverse == 0: out[b,r,ky,c] = scale * sum_X in[b,X,ky,c] e^{-i 2pi kx(r) X/n}
 * inverse == 1: out[b,X,ky,c] = scale * sum_r in[b,r,ky,c] e^{+i 2pi kx(r) X/n} */
int gb200_spectral_xdft(int device, const float* in, int B, int n, int m, int C, const float* twX,
                        float scale, int inverse, float* out, void* stream);
/* O[b,q,o] = sum_i X[b,q,i] * W_half(q)[i,o,q']   complex_matmul_{1d,2d}: libs/layers.py:1068-1075,
 * 1144-1151.  halves = 1 (1-D, W0 only) or 2 (2-D, W0 = fourier_weight[0], W1 = fourier_weight[1]);
 * M2 = modes per half (m or m*m). */
int gb200_spectral_mix_fwd(int device, const float* Xf, const float* W0, const float* W1, int B, int halves,
                           int M2, int Ci, int Co, float* Of, void* stream);
/* dX = dO . conj(W) (skipped if NULL);  dW (+)= sum_b conj(X) . dO (skipped if dW0 NULL) */
int gb200_spectral_mix_bwd(int device, const float* Xf, const float* dO, const float* W0, const float* W1,
                           int B, int halves, int M2, int Ci, int Co, float* dX, float* dW0, float* dW1,
                           int accumulate_dw, void* stream);
/* y[R,Y,o] = act( scale * sum_ky c_ky Re(Z[R,ky,o] e^{+i 2pi ky Y/n}) + sum_i x2[R,Y,i] Wm[i,o] + bias[o] )
 * i.e. irfft along the last axis fused with the residual nn.Linear, bias and SiLU
 * (libs/layers.py:1083, 1098-1101 / 1172, 1187-1189).  zout (optional) receives the pre-activation. */
int gb200_spectral_yidft_epilogue(int device, const float* Z, long long R, int n, int m, int Co,
                                  const float* twY, float scale, int hermitian, const float* x2, int Ci,
                                  const float* Wm, const float* bias, int act, float* y, float* zout,
                                  int tensor_cores, void* stream);

/* ------------------------------------------------------------------ grid resize ---------------
 * Bilinear resize with align_corners = True of a channel-last grid (B, Hin, Win, C) -> (B, Hout, Wout, C): the
 * F.interpolate(mode='bilinear', align_corners=True) steps of the interpolation scalers
 * (libs/layers.py:431-512 Interp2dEncoder, :624-670 Interp2dUpsample), which the reference runs on (B, C, H, W).
 * _bwd: din (B, Hin, Win, C) = adjoint applied to dout (B, Hout, Wout, C); gather formulation, deterministic. */
int gb200_interp_bilinear_fwd(int device, const float* in, int B, int Hin, int Win, int C, float* out, int Hout, int Wout,
                              void* stream);
int gb200_interp_bilinear_bwd(int device, const float* dout, int B, int Hin, int Win, int C, float* din, int Hout,
                              int Wout, void* stream);

/* ------------------------------------------------------------------ fused encoder layer --------
 * SimpleTransformerEncoderLayer.forward (libs/model.py:104-140) = SimpleAttention.forward (libs/layers.py:829-899:
 * Q/K/V projections :837-839, per-head LayerNorm loop :846-851, position concat :869-874, K^T V / n + dropout + Q.(.)
 * :723-733, head merge + fc :892-897) + residual (:124-127) + FeedForward (libs/layers.py:979-987) + residual (:131-132),
 * Galerkin type, as three tcgen05 kernels per 128-token tile (csrc/encoder_fwd.cu):
 *     1. x -> [Q | LN(K) | LN(V)] and the tile's partial K~^T V~ (the LayerNorm is fused into the first of the two
 *        back-to-back contractions; both run on TMA-staged tiles and tcgen05.mma with TMEM accumulators)
 *     2. A = mask * sum(partials) * scale ; heads = Q~ A ; x1 = x + sign * dropout(heads W_fc^T + b_fc)
 *     3. x2 = x1 + dropout( dropout(relu(x1 W1^T + b1)) W2^T + b2 )       (hidden tile never leaves the SM)
 * Arithmetic: "bf16x3" -- every product is a_hi.b_hi + a_hi.b_lo + a_lo.b_hi with (hi, lo) the two-term bf16 split of
 * the fp32 operand, fp32 accumulation: ~2^-17 relative error per product, 30x tighter than TF32 (DESIGN.md).
 * Supported shape: d_model 128, 4 heads, d_ff 256, pos_dim <= 2 (BASELINE config 3); gb200_encoder_supported() says so
 * and the Python layer falls back to the per-operator kernels otherwise.
 *
 * gb200_encoder_pack: once per step, parameters -> bf16 (hi, lo) operand tile images in streaming order for the
 * forward and backward kernels plus one fp32 block of biases / LayerNorm tables (`packed`: 128-byte aligned,
 * gb200_encoder_pack_bytes() bytes).  Buffers saved by _fwd are exactly those the per-operator backward consumes:
 * qkv (B n, 3 d_model) = [Q | x^_K | x^_V], rstd_k / rstd_v (B n, heads), attn (B, heads, d, d), heads (B n, heads d),
 * x1 (B n, d_model), hidden (B n, d_ff) post-ReLU post-dropout, x2 (B n, d_model).  Dropout masks are Philox streams
 * keyed exactly like the unfused epilogues (seed, flat element index), so either backward regenerates them.
 * `stages`: bit 0/1/2 = run kernel 1/2/3 (7 = whole layer; tests run them one at a time). */
#define GB200_ENC_TILES 70
#define GB200_ENC_MAX_HEADS 8
typedef struct gb200_encoder_params {
    const float *wq, *wk, *wv, *bq, *bk, *bv;                 /* attn.linears.{0,1,2} */
    const float *gamma_k[GB200_ENC_MAX_HEADS], *beta_k[GB200_ENC_MAX_HEADS];   /* attn.norm_K.{h}; NULL without norm */
    const float *gamma_v[GB200_ENC_MAX_HEADS], *beta_v[GB200_ENC_MAX_HEADS];   /* attn.norm_V.{h} */
    const float *wfc, *bfc;                                   /* attn.fc (d_model, d_model + heads * pos_dim) */
    const float *w1, *b1, *w2, *b2;                           /* ff.lr1, ff.lr2 */
    int d_model, n_head, pos_dim, d_ff;
} gb200_encoder_params;
int gb200_encoder_supported(int d_model, int n_head, int pos_dim, int d_ff);
/* Diagnostics: non-null = every CTA of the fused encoder kernels writes clock64 stamps of its pipeline milestones to
 * device_buffer[32 * blockIdx.x + slot] (slot 31: %globaltimer at entry); tools/trace_fused.py prints the timeline. */
int gb200_encoder_set_trace(unsigned long long* device_buffer);
size_t gb200_encoder_pack_bytes(int d_model, int n_head, int pos_dim, int d_ff);
int gb200_encoder_pack(int device, const gb200_encoder_params* params, void* packed, void* stream);
size_t gb200_encoder_workspace_bytes(int B, int n, int n_head, int d_k, int pos_dim);
int gb200_encoder_layer_fwd(int device, const void* packed, int d_model, int n_head, int pos_dim, int d_ff,
                            const float* x, const float* pos, int B, int n, int has_norm, float eps, float attn_scale,
                            const unsigned char* keep_mask, float mask_p, unsigned long long mask_seed,
                            float p_attn_out, unsigned long long seed_attn_out, float res_sign, float p_ffn,
                            unsigned long long seed_ffn, float p_out, unsigned long long seed_out, float* qkv,
                            float* rstd_k, float* rstd_v, float* attn, float* heads, float* x1, float* hidden, float* x2,
                            float* workspace, size_t workspace_bytes, int stages, void* stream);

/* Backward of the fused layer (csrc/encoder_bwd.cu): four tcgen05 kernels + one reduction carry every input-gradient
 * GEMM (bf16x3), the activation / dropout / per-head LayerNorm backward passes and all bias / LayerNorm-parameter
 * gradients; the caller runs the four weight-gradient GEMMs (dW2 = g2^T hidden, dW1 = g1^T x1, dW_fc = gfc^T heads,
 * dW_qkv = dqkv^T x) on gb200_gemm_tc from the buffers written here.
 *   g2 (B n, d_model) = dy * mask_out      (written only when p_out > 0; otherwise dy itself)
 *   g1 (B n, d_ff), dx1 (B n, d_model), gfc (B n, d_model) = sign * dx1 * mask_attn_out (only when it differs from dx1),
 *   dqkv (B n, 3 d_model), dx (B n, d_model), dvec (1408 floats, the layout of the packed vector block:
 *   d b_q | d b_k | d b_v | d gamma_K | d beta_K | d gamma_V | d beta_V | d b_fc | d b_1 | d b_2).
 * `stages`: bit 0 ffn, 1 attention-out, 2 K/V + LayerNorm, 3 dx, 4 reduction (31 = everything). */
size_t gb200_encoder_bwd_workspace_bytes(int B, int n, int n_head, int d_k, int pos_dim);
int gb200_encoder_bwd_set_trace(unsigned long long* device_buffer);
int gb200_encoder_layer_bwd(int device, const void* packed, int d_model, int n_head, int pos_dim, int d_ff,
                            const float* dy, const float* pos, int B, int n, int has_norm, float attn_scale,
                            const unsigned char* keep_mask, float mask_p, unsigned long long mask_seed, float p_attn_out,
                            unsigned long long seed_attn_out, float res_sign, float p_ffn, float p_out,
                            unsigned long long seed_out, const float* qkv, const float* rstd_k, const float* rstd_v,
                            const float* attn, const float* hidden, float* g2, float* g1, float* dx1, float* gfc,
                            float* dqkv, float* dx, float* dvec, float* workspace, size_t workspace_bytes, int stages,
                            void* stream);

/* ------------------------------------------------------------------ scaler convolutions --------
 * y = act( dropout( conv3x3(x) ) ), stride 1, padding 1, no bias, channel-last (B, H, W, C) fp32: Conv2dResBlock
 * (libs/layers.py:88-150) as used by Interp2dEncoder (:431-512) and Interp2dUpsample (:624-670).  csrc/conv.cu:
 * implicit GEMM on tcgen05 in bf16x3 arithmetic; the nine taps are nine shifted 4-D TMA tile loads of the (hi, lo) bf16
 * images of the input (TMA's out-of-bounds zero fill is the padding).  gb200_conv_split makes the images (and, in
 * backward mode, applies the activation / dropout derivative first); gb200_conv3x3_pack lays the weights out as operand
 * tiles for the forward (dgrad = 0) or the input-gradient pass (dgrad = 1: transposed and flipped), which is the same
 * kernel.  The 1 -> C first convolution is a streaming stencil (gb200_conv1_*; backward for the ReLU block).
 * The weight gradient of the multi-channel blocks is left to the caller (a library convolution-backward call). */
int gb200_conv3x3_supported(int Cin, int Cout);
size_t gb200_conv3x3_pack_bytes(int Cin, int Cout, int dgrad);
int gb200_conv3x3_pack(int device, const float* w, int Cin, int Cout, int dgrad, void* tiles, void* stream);
int gb200_conv_split(int device, const float* x, int ldx, int c0, int C, long long npix, void* hi, void* lo, const float* yz,
                     int ldyz, int yz_c0, int act, float p, unsigned long long seed, float* gout, void* stream);
int gb200_conv3x3(int device, const void* in_hi, const void* in_lo, int Cin, const void* wtiles, int Cout, int B, int H, int W,
                  float* out, int ldo, int co0, float* zout, const float* resid, int ldr, int r0, int act, float p,
                  unsigned long long seed, void* stream);
int gb200_conv1_fwd(int device, const float* x, const float* w, float* y, int B, int H, int W, int C, int act, float p,
                    unsigned long long seed, void* stream);
size_t gb200_conv1_bwd_workspace_bytes(int C);
int gb200_conv1_bwd(int device, const float* dy, const float* y, const float* x, const float* w, float* dx, float* dw, int B,
                    int H, int W, int C, float p, float* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ training-step tail ---------
 * SURVEY.md 8(f) row 3.  csrc/train.cu.
 *
 * gb200_weighted_l2_loss2d: WeightedL2Loss2d.forward(preds, targets, targets_prime=..., K=...) of libs/ft.py:1035-1101
 * for preds / targets (B, n, n), targets_prime (B, n, n, 2) or NULL, K (B, n, n) or NULL (K = 1):
 *   loss_b = beta * mean((p - t)^2) / (mean(t^2) + eps);  loss = mean_b sqrt(loss_b)   (return_norm; else mean_b loss_b)
 *   reg_b  = gamma * h * mean((K (tp - D_h p))^2) / (2 mean(K tp^2) + eps) over the interior (regularizer != 0 and
 *            targets_prime given; D_h = central differences with the given even dilation), reduced like the loss
 *   out4   = { loss, regularizer, 'L1' metric = mean_b sqrt(loss_b), loss + regularizer }         (device floats)
 *   dloss / dreg (either may be NULL) = the gradients of out4[0] / out4[1] with respect to preds -- what autograd through
 *   the reference's ~40 elementwise launches produces.  Two launches, fixed-order reductions, no host synchronisation.
 *
 * gb200_adam_clip_step: nn.utils.clip_grad_norm_(params, max_norm) followed by torch.optim.Adam.step()
 * (libs/utils_ft.py:676-681) over FLAT fp32 buffers of n elements: total = |grad|_2, g *= min(1, max_norm / (total + 1e-6))
 * (max_norm <= 0: no clipping), m = lerp(m, g, 1 - beta1), v = beta2 v + (1 - beta2) g^2,
 * p -= lr / bias_correction1 * m / (sqrt(v) / sqrt(bias_correction2) + eps).
 * hyper = DEVICE array { lr, beta1, bias_correction1, bias_correction2 } (changes every step under OneCycleLR, which also
 * cycles beta1; a device array keeps the launches graph-capturable).  grad_norm_out (device float or NULL) receives the
 * pre-clip norm.  Two launches. */
size_t gb200_weighted_l2_loss2d_workspace_bytes(int B, int n);
int gb200_weighted_l2_loss2d(int device, const float* preds, const float* targets, const float* targets_prime,
                             const float* K, int B, int n, float h, float beta, float gamma, float eps, int dilation,
                             int regularizer, int return_norm, float* out4, float* dloss, float* dreg, float* workspace,
                             size_t workspace_bytes, void* stream);
size_t gb200_adam_clip_step_workspace_bytes(long long n);
int gb200_adam_clip_step(int device, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n,
                         const float* hyper, float beta2, float eps, float weight_decay, float max_norm,
                         float* grad_norm_out, float* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GALERKIN_B200_H_ */
