/*
 * b200_imagen.h -- C-ABI of libb200imagen.so: the sm_100a kernels behind the
 * imagen-pytorch sampling hot path (U-Net forward x denoising loop).
 *
 * The reference (lucidrains/imagen-pytorch v2.0.0) has NO native/FFI interface:
 * every FLOP goes through ATen (SURVEY.md section 2.2).  The boundary a
 * maintainer would bind is therefore "one entry point per fused ATen op group
 * of Unet.forward / p_sample / one_unet_sample".  Each declaration below cites
 * the reference lines (relative to /root/reference/imagen_pytorch/) whose
 * arithmetic it replaces.  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - extern "C", POD arguments only: device pointers, sizes, strides, a
 *     cudaStream_t passed as void*.  No torch types.
 *   - every function returns 0 on success or a negative b200_status; the text
 *     of the last error of the calling thread is b200_last_error().
 *   - nothing here allocates, frees or synchronises: all functions are
 *     CUDA-graph-capture safe.  The caller owns every buffer.
 *   - activations are NHWC bf16 ("pixel rows": [B*H*W, C] row-major with an
 *     explicit row stride ld, in elements); sampler state is fp32 NCHW exactly
 *     as the reference keeps it.
 */
#ifndef B200_IMAGEN_H_
#define B200_IMAGEN_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_ABI_VERSION 2

typedef enum {
  B200_OK = 0,
  B200_ERR_INVALID = -1,   /* bad argument / unsupported shape */
  B200_ERR_CUDA = -2,      /* a CUDA runtime / driver call failed */
  B200_ERR_NO_DEVICE = -3, /* no sm_100 device */
} b200_status;

const char* b200_last_error(void);
int b200_abi_version(void);
/* sizeof() of the ABI structs as compiled: 0 b200_src, 1 b200_seg, 2 b200_epilogue, 3 b200_timerow_job,
 * 4 b200_ddpm_coef, 5 b200_edm_coef (lets a binding verify its struct mirrors). */
int b200_sizeof(int which);
/* 0 if device `dev` is compute capability 10.x, else B200_ERR_NO_DEVICE. */
int b200_check_device(int dev);

/* ------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution / linear layer on the 5th-gen tensor cores
 * (TMA-staged NHWC tiles -> 128B-swizzled smem -> tcgen05.mma -> TMEM -> fused epilogue).
 * Replaces: nn.Conv2d 3x3/1x1 in Block.project (imagen_pytorch.py:681,691), res_conv (:732,757),
 * Downsample 1x1 (:639), PixelShuffleUpsample conv+SiLU+PixelShuffle (:611-617), Parallel (:1366),
 * final_conv (:1436,1725), and every nn.Linear on pixel rows: to_q/to_kv/to_out (:521-532,539,591;
 * :782-791,799,834), FeedForward (:976-979), time_mlp (:711-714,739).
 *
 *   out[m, n] = epilogue( sum_seg sum_c  A_seg[pixel(m) + (dh,dw), c] * Wp[n, k(seg,c)] )
 * ------------------------------------------------------------------------------------------ */

#define B200_MAX_SRC 4
#define B200_MAX_SEG 24

typedef struct {
  const void* ptr; /* bf16, [B*H*W, C] pixel rows, row stride ld elements (ld % 8 == 0) */
  int32_t C;       /* channels read from this source */
  int32_t ld;
} b200_src;

typedef struct {
  int32_t src; /* index into srcs[] */
  int32_t dh;  /* tap offset, rows   (-1..1 for 3x3 pad 1, 0 for 1x1) */
  int32_t dw;  /* tap offset, columns */
} b200_seg;

enum { B200_ACT_NONE = 0, B200_ACT_SILU = 1, B200_ACT_GELU = 2 };
enum {
  B200_OUT_BF16 = 0,         /* out[row, n] bf16, row stride ldc                                   */
  B200_OUT_PIXEL_SHUFFLE = 1,/* N = 4*ps_C ordered (r1, r2, c'): out[b, 2h+r1, 2w+r2, c'] bf16     */
  B200_OUT_F32_NCHW = 2,     /* out[b, n, h, w] fp32 (final conv -> sampler)                        */
  B200_OUT_F32 = 3,          /* out[row, n] fp32, row stride ldc                                    */
};

typedef struct {
  const float* bias;      /* [N] or NULL */
  int32_t act;            /* B200_ACT_* applied after bias */
  float out_scale;        /* multiplies the activated value (1.0 = none) */
  const void* residual;   /* bf16 [M, ldr] added last, or NULL */
  int32_t ldr;
  int32_t out_mode;       /* B200_OUT_* */
  void* out;
  int32_t ldc;
  /* columns >= split_col go to out2 (column n - split_col), bf16 row-major; 0 = off */
  void* out2;
  int32_t ldc2;
  int32_t split_col;
  /* row remap for out/out2: row' = (m / rows_per_group) * group_stride + row_offset + m % rows_per_group;
     rows_per_group == 0 -> identity */
  int32_t rows_per_group;
  int32_t group_stride;
  int32_t row_offset;
  /* cosine-sim attention: L2-normalise each 64-column group of the first l2_cols columns
     (F.normalize eps 1e-12) and multiply by l2_scale[n % 64]  (imagen_pytorch.py:559-561, 812-814) */
  int32_t l2_cols;
  const float* l2_scale;  /* [64] */
  int32_t ps_C;           /* C' for B200_OUT_PIXEL_SHUFFLE */
  /* also store rows at +dup_rows (classifier-free-guidance batch duplication); 0 = off */
  int32_t dup_rows;
  /* ---- per-row normalisations fused into the epilogue (ABI v2).  Available when one N tile spans all channels
   *      (64 <= N <= 256, N % 32 == 0), out_mode == B200_OUT_BF16 and none of split_col / rows_per_group / l2_cols / dup_rows:
   *        v  = act(acc + bias) * out_scale
   *        v  = norm1 ? LayerNorm(v) * norm1_g : v                     (custom gain-only LayerNorm, eps 1e-5, imagen_pytorch.py:331-349)
   *        w  = v + residual                                           -> out (bf16; may be NULL when only out_norm is wanted)
   *        y  = norm2 == 1 ? LayerNorm(w) * norm2_g                    (the next pre-norm: imagen_pytorch.py:516, :775, :975)
   *           : norm2 == 2 ? SiLU( w / |w|_2 * norm2_g [* (scale+1) + shift] )   (Block: ChanRMSNorm -> FiLM -> SiLU, :683-691;
   *                          norm2_g = gamma * sqrt(N) folded by the caller)
   *        y -> out_norm (bf16)
   *      Statistics are taken on the fp32 values (the reference's arithmetic), not on bf16-rounded ones. */
  int32_t norm1;
  const float* norm1_g;     /* [N] */
  int32_t norm2;
  const float* norm2_g;     /* [N] */
  const float* film;        /* norm2 == 2: fp32 rows [scale (N) | shift (N)] per sample, row pitch film_ld; NULL = no FiLM */
  int32_t film_ld;
  int32_t rows_per_sample;  /* output rows per sample (selects the film row) */
  void* out_norm;
  int32_t ld_norm;
} b200_epilogue;

/* Packed weight layout: bf16 [Npad, Ktot], Npad = N rounded up to the N tile, K ordered by
 * segment, each segment padded to a multiple of 64 channels with zeros.
 * b200_conv_gemm_npad() tells the packer the N padding used for a given N. */
int b200_conv_gemm_npad(int N);

/* K-split factor the library will use for this shape WHEN a workspace is passed (1 = none): the caller then provides
 * f32_scratch of >= factor * B*H*W * b200_conv_gemm_npad(N) floats to b200_conv_gemm (impl 0).  Ktot = sum over segments of the
 * channel count rounded up to 64.  Without a workspace the GEMM runs unsplit. */
int b200_conv_gemm_splitk(int B, int H, int W, int N, int Ktot);
int b200_conv_gemm(const b200_src* srcs, int nsrc, const b200_seg* segs, int nseg,
                   int B, int H, int W,              /* pixel grid of the OUTPUT rows: M = B*H*W */
                   const void* w_packed, int N,
                   const b200_epilogue* epi,
                   int impl,                         /* 0 = tcgen05 (product); 1 = SIMT checker used by tests */
                   void* f32_scratch,                /* impl 1: >= M*Npad floats; impl 0: optional split-K workspace (b200_conv_gemm_splitk) */
                   void* stream);

/* ------------------------------------------------------------------------------------------
 * Flash-style cosine-sim attention (no N x M score matrix).  Q rows are already L2-normalised
 * and pre-multiplied by q_scale * 8 * log2(e) by the to_q epilogue; K rows by k_scale.
 * Replaces: Attention.forward einsum/softmax/einsum (imagen_pytorch.py:565-588) with the multi-query
 * layout (n_heads = 1, rows = 8*n, q_row_stride = 64) and CrossAttention.forward (:818-833)
 * (n_heads = 8, rows = n, q_row_stride = 512, per-head K/V).
 * problem (b, h): q + b*q_bs + h*q_hs (row stride q_rs), k/v + b*kv_bs + h*kv_hs (row stride kv_rs),
 * o like q.  Head dim = 64.  All strides in elements.
 * max_logit: an upper bound of |q.k| in log2 units (8*log2e*max_d|q_scale_d*k_scale_d| for cosine-sim attention,
 * by Cauchy-Schwarz).  0 < max_logit <= 40 selects the tcgen05 kernel (TMA -> tcgen05.mma S/P.V with TMEM
 * accumulators, softmax without running max); <= 0 selects the online-softmax mma.sync kernel.
 * ------------------------------------------------------------------------------------------ */
int b200_attention(const void* q, void* o, int64_t q_bs, int64_t q_hs, int32_t q_rs, int32_t rows,
                   const void* k, const void* v, int64_t kv_bs, int64_t kv_hs, int32_t kv_rs, int32_t n_keys,
                   int B, int n_heads, float max_logit, void* stream);

/* ------------------------------------------------------------------------------------------
 * Linear cross-attention (LinearCrossAttention.forward, imagen_pytorch.py:836-874; Unet(use_linear_cross_attn=...)):
 *   out = softmax_d(q) @ C,  C[d, e] = 8 * sum_j softmax_j(k)[j, d] * v[j, e]   per (sample b, head h).
 * Two steps, both per denoising step (the time-token K/V rows change every step):
 * b200_linear_xattn_context: raw (not normalised) bf16 k / v of problem (b, h) at k + b*kv_bs + h*64, row stride kv_rs,
 *   n_keys >= 1 rows (the null key/value included) -> ctx, bf16 [B][n_heads][64][64] (row d, column e), rows d >= dim_head zero.
 * b200_linear_cross_attention: q bf16 rows (problem (b, h) at q + b*q_bs + h*64, row stride q_rs, `rows` pixels), the softmax
 *   over its first dim_head channels (channels dim_head..63 are zero padding and get weight 0) times ctx -> o, same layout as q.
 *   tcgen05 kernel: q through a TMA ring, P in tensor memory, O = P C as one M128 x N64 x K64 MMA per 128-row tile.
 * n_heads <= 8, dim_head <= 64, strides in elements (multiples of 8 for q / o).
 * ------------------------------------------------------------------------------------------ */
int b200_linear_xattn_context(const void* k, const void* v, int64_t kv_bs, int32_t kv_rs, int32_t n_keys, int B, int n_heads,
                              int32_t dim_head, void* ctx, void* stream);
int b200_linear_cross_attention(const void* q, void* o, int64_t q_bs, int32_t q_rs, int32_t rows, const void* ctx, int B, int n_heads,
                                int32_t dim_head, void* stream);

/* ------------------------------------------------------------------------------------------
 * Row-wise normalisation kernels on pixel rows (HBM-bound).
 * ------------------------------------------------------------------------------------------ */

/* ChanRMSNorm -> FiLM -> SiLU over the channel concat of up to 2 sources
 * (Block.forward imagen_pytorch.py:683-690, ChanRMSNorm :322-329, skip concat+scale :1694).
 *   y = silu( x / max(||x||_2, 1e-12) * gamma_sqrtC[c] * (scale[b,c] + 1) + shift[b,c] )
 * x = cat(src0, src1 * src1_scale).  film: fp32 [B, film_ld], scale at [c], shift at [Ctot + c]; NULL = none. */
int b200_rmsnorm_film_silu(const b200_src* srcs, int nsrc, float src1_scale, const float* gamma_sqrtC,
                           const float* film, int32_t film_ld, int32_t rows_per_sample,
                           void* out, int32_t ldo, int64_t M, void* stream);

/* LayerNorm over C (biased variance, eps): y = (x-mean)*rsqrt(var+eps)*g (+ beta) (+ residual).
 * Custom gain-only LayerNorm imagen_pytorch.py:331-349 (eps 1e-5) and the "+ x" of Residual-style
 * callers (:749, :1017-1018). */
int b200_layernorm(const void* x, int32_t ldx, const float* g, const float* beta, float eps,
                   const void* residual, int32_t ldr, void* out, int32_t ldo, int64_t M, int32_t C, void* stream);

/* GlobalContext (imagen_pytorch.py:945-970): gate[b, c] = sigmoid(W2 silu(W1 pool + b1) + b2),
 * pool[c] = sum_p softmax_p(x[p,:].wk + bk) x[p, c].  scratch: fp32 [B*nchunk*(C + 2) + B*C + B*hidden + B*rows_per_sample]
 * (softmax partials | pooled | hidden | per-pixel logits). */
int b200_gca_gate(const void* x, int32_t ldx, int B, int32_t rows_per_sample, int32_t C,
                  const float* wk, float bk, const float* w1, const float* b1, int32_t hidden,
                  const float* w2, const float* b2, float* scratch, int32_t nchunk, float* gate, void* stream);
/* Chained per-row kernel: the per-pixel ops that sit between two GEMMs when the GEMM epilogue cannot host them (more than 256
 * channels, or a producer that is not a GEMM), in ONE pass over the row:
 *     v = x [* gate[row / rows_per_sample, :]]                      (GlobalContext gate, imagen_pytorch.py:754)
 *     v = norm1 ? LayerNorm(v) * norm1_g : v                         (:331-349)
 *     w = v + residual                         -> out  (bf16, may be NULL)
 *     y = norm2 == 1 ? LayerNorm(w) * norm2_g : norm2 == 2 ? SiLU(RMSNorm(w) * norm2_g [* (scale+1) + shift])   -> out_norm
 * The struct is read at launch time, so a consumer discovered later can attach its norm2 to an already recorded call.
 * Replaces b200_layernorm (+ residual) / b200_gate_residual followed by b200_layernorm / b200_rmsnorm_film_silu. */
typedef struct {
  const void* x; int32_t ldx;
  const float* gate;        /* fp32 [B, C] or NULL */
  int32_t rows_per_sample;  /* rows per sample (selects the gate / film row) */
  int32_t norm1; const float* norm1_g;
  const void* residual; int32_t ldr;
  void* out; int32_t ldo;
  int32_t norm2; const float* norm2_g;
  const float* film; int32_t film_ld;
  void* out_norm; int32_t ld_norm;
  int64_t M; int32_t C;
} b200_rowchain;
int b200_row_chain(const b200_rowchain* p, void* stream);

int b200_gca_nchunk(int32_t rows_per_sample);
/* chunk count for which b200_gca_gate takes its 2-launch path (fused logits + pooling with the pixel chunk staged in shared memory, then
 * one cluster kernel for combine + MLP + gate); the scratch layout is the same with this nchunk */
int b200_gca_chunks(int32_t rows_per_sample, int32_t C);

/* out = x * gate[b, c] + residual  (ResnetBlock.forward imagen_pytorch.py:755-757). */
int b200_gate_residual(const void* x, int32_t ldx, const float* gate, const void* residual, int32_t ldr,
                       void* out, int32_t ldo, int64_t M, int32_t C, int32_t rows_per_sample, void* stream);

/* Patch gather for the initial cross-embed convolution (CrossEmbedLayer imagen_pytorch.py:1051-1076,
 * used at :1564): fp32 NCHW image(s) -> bf16 [B*H*W, Kpad] rows ordered (kh, kw, c), zero padded.
 * c runs over cat(img0, img1) (lowres concat :1551). */
int b200_im2col_init(const float* img0, int C0, const float* img1, int C1, int B, int H, int W, int ksize,
                     void* out, int32_t Kpad, void* stream);
/* the same with a third NCHW source (channel order img0 | img1 | img2): x | self_cond | lowres_cond_img (imagen_pytorch.py:1541-1551) */
int b200_im2col_init3(const float* img0, int C0, const float* img1, int C1, const float* img2, int C2, int B, int H, int W,
                      int ksize, void* out, int32_t Kpad, void* stream);
/* the same with a fourth image (Unet(cond_images_channels > 0): cat((cond_images, x [, self_cond] [, lowres_cond_img])),
 * imagen_pytorch.py:1553-1560) */
int b200_im2col_init4(const float* img0, int C0, const float* img1, int C1, const float* img2, int C2,
                      const float* img3, int C3, int B, int H, int W, int ksize, void* out, int32_t Kpad, void* stream);

/* Pixel-unshuffle gather of Downsample (imagen_pytorch.py:638): out[b,h,w,(s1,s2,c)] = x[b,2h+s1,2w+s2,c]. */
int b200_pixel_unshuffle(const void* x, int32_t ldx, int B, int H, int W, int C, void* out, void* stream);

/* fp32 NCHW [B,C,H,W] -> bf16 NHWC rows with Cpad channels (zero padded). Used for the low-res
 * conditioning image concatenated before final_conv (imagen_pytorch.py:1722-1723). */
int b200_nchw_to_rows(const float* img, int B, int C, int H, int W, void* out, int32_t Cpad, void* stream);

/* ------------------------------------------------------------------------------------------
 * Per-step conditioning plumbing (time-dependent rows only; everything text-dependent is
 * hoisted out of the loop, SURVEY.md fact 6).
 * ------------------------------------------------------------------------------------------ */

/* t_silu[r, :] = silu(time_cond_table[slot[r], :] + text_hiddens[r, :])   bf16 out.
 * (Unet.forward :1578,1588,1652 and the nn.SiLU at the head of every time_mlp :711-713.) */
int b200_make_time_cond(const float* table, const float* text_hiddens, const int32_t* slots,
                        int R, int32_t D, void* out, void* stream);

typedef struct {
  const void* table; /* bf16 [S, rows, width] : time-token K or V rows for every schedule slot */
  void* dst;         /* bf16, row r of sample b at dst + b*sample_stride + r*width */
  int64_t sample_stride;
  int32_t rows;
  int32_t width;
} b200_timerow_job;

/* For every job and sample: copy table[slot[b]] into the K/V buffers. jobs is a DEVICE array. */
int b200_update_time_rows(const b200_timerow_job* jobs_dev, int njobs, const int32_t* slots, int R,
                          int32_t max_elems, void* stream);

/* ------------------------------------------------------------------------------------------
 * fp32 conditioning head (runs once per sample() call, not per step): time MLPs, text_to_cond,
 * PerceiverResampler, to_text_non_attn_cond, norm_cond, per-layer context K/V.
 * Unet.forward imagen_pytorch.py:1573-1660; PerceiverAttention :408-445; LearnedSinusoidalPosEmb :664-669.
 * ------------------------------------------------------------------------------------------ */

/* y[M,N] = out_act( in_act(x)[M,K] @ W[N,K]^T + b ) (+ residual), all fp32. */
int b200_linear_f32(const float* x, int32_t ldx, const float* W, const float* b, int in_act, int out_act,
                    const float* residual, int32_t ldr, float* y, int32_t ldy, int64_t M, int32_t N, int32_t K,
                    void* stream);
int b200_layernorm_f32(const float* x, int32_t ldx, const float* g, const float* beta, float eps,
                       float* y, int32_t ldy, int64_t M, int32_t C, void* stream);
/* [x, sin(2 pi x w), cos(2 pi x w)] -> out[M, 2*half+1] */
int b200_sinu_pos_emb(const float* x, const float* w, int M, int half, float* out, void* stream);
/* multi-head cosine-sim attention, fp32: q [B, nq, H*64], k/v [B, nk, H*64] (ld = row strides). */
int b200_attn_f32(const float* q, int32_t ldq, const float* k, const float* v, int32_t ldkv,
                  const float* q_scale, const float* k_scale, float* o, int32_t ldo,
                  int B, int H, int nq, int nk, void* stream);
/* per 64-wide head group: optional F.normalize, optional * scale[64], cast to bf16 and scatter:
 * dst[(row / rpg) * s_grp + (row % rpg) * s_row + g * s_head + d]. */
int b200_headnorm_store(const float* x, int32_t ldx, int32_t col0, int32_t ngroups, int normalize,
                        const float* scale, void* dst, int32_t rpg, int64_t s_grp, int64_t s_row, int64_t s_head,
                        int64_t M, void* stream);

/* ------------------------------------------------------------------------------------------
 * Sampler steps (fp32 state, exact torch.quantile dynamic thresholding inside).
 * ------------------------------------------------------------------------------------------ */

/* Per-step scalars of the continuous-time DDPM posterior, tabulated on the host with the same
 * torch ops as GaussianDiffusionContinuousTimes (imagen_pytorch.py:245-270, 314-318). */
typedef struct {
  float sigma;          /* sqrt(sigmoid(-log_snr(t)))           */
  float alpha;          /* sqrt(sigmoid( log_snr(t)))           */
  float inv_alpha_clamped; /* 1 / max(alpha, 1e-8)              */
  float alpha_next;
  float c;              /* -expm1(log_snr - log_snr_next)        */
  float noise_std;      /* [t_next != 0] * exp(0.5*log(max(sigma_next^2 c, 1e-20))) */
  float pad0, pad1;
} b200_ddpm_coef;

/* One ancestral DDPM step, in place on x (Imagen.p_sample imagen_pytorch.py:2112-2165,
 * p_mean_variance :2085-2110, CFG combine :1522).  pred: fp32 [R, C, H, W] with the conditional rows
 * first and (if cond_scale != 1) the null rows at +B.  objective 0 noise, 1 x_start, 2 v.
 * thresholding: 1 = dynamic (quantile q_lo/q_hi/q_w as torch.quantile computes them), 0 = clamp(-1,1).
 * Increments slots[0..R) by one at the end (the device-side step counter). */
int b200_ddpm_step(float* x, const float* pred, const float* noise, const b200_ddpm_coef* coefs,
                   int32_t* slots, int R, int B, int64_t chw, float cond_scale, int objective,
                   int thresholding, int32_t q_lo, int32_t q_hi, float q_w, void* stream);
/* the same; additionally writes the thresholded x_start [B, chw] (the next step's self-conditioning input, imagen_pytorch.py:2252)
 * when x_start_out != NULL. */
int b200_ddpm_step_sc(float* x, const float* pred, const float* noise, const b200_ddpm_coef* coefs,
                      int32_t* slots, int R, int B, int64_t chw, float cond_scale, int objective,
                      int thresholding, int32_t q_lo, int32_t q_hi, float q_w, float* x_start_out, void* stream);

typedef struct {
  float s_noise;     /* S_noise: eps = s_noise * z                                        */
  float noise_coef;  /* fp32(sqrt(sigma_hat^2 - sigma^2)) (python double math, then cast) */
  float sigma_hat, sigma_next;               /* fp32 casts of the python doubles          */
  float dt, half_dt; /* fp32(sigma_next - sigma_hat), fp32(0.5 * (sigma_next - sigma_hat)) */
  float c_in_hat, c_skip_hat, c_out_hat;     /* preconditioning at sigma_hat (torch fp32 ops) */
  float c_in_next, c_skip_next, c_out_next;  /* at sigma_next (unused on the last step)   */
  float has_second;  /* sigma_next != 0 */
  float pad0, pad1, pad2;
} b200_edm_coef;

/* EDM stochastic Heun sampler (ElucidatedImagen.one_unet_sample elucidated_imagen.py:481-531,
 * preconditioned_network_forward :340-369, threshold_x_start :309-321), split at the two network
 * evaluations.  phase 0: x_hat = x + noise_coef*(s_noise*z) ; net_in = c_in_hat * x_hat.
 * phase 1: D = thr(c_skip x_hat + c_out F); d = (x_hat - D)/sigma_hat; x1 = x_hat + (sn - sh) d;
 *          net_in = c_in_next * x1 (if has_second) else x = x1.
 * phase 2: D' = thr(...x1...); d' = (x1 - D')/sn; x = x_hat + 0.5 (sn - sh)(d + d').
 * The step index into coefs is read from the device counter step_ctr[0] (step_ctr is int32[2], both
 * zero-initialised by the caller); the last phase of a step (2, or 1 when !has_second) stages the
 * increment in step_ctr[1] and the next phase-0 launch commits it.  Phases 1 and 2 bump slots (one slot per network
 * evaluation) so the whole step is CUDA-graph capturable. */
int b200_edm_phase(int phase, float* x, float* x_hat, float* x1, float* d, float* net_in,
                   const float* pred, const float* eps, const b200_edm_coef* coefs, int32_t* step_ctr,
                   int32_t* slots, int R, int B, int64_t chw, float cond_scale, int thresholding,
                   int32_t q_lo, int32_t q_hi, float q_w, void* stream);
/* the same; phases 1 and 2 additionally write the thresholded denoiser output D [B, chw] (self-conditioning input of the next
 * network evaluation, elucidated_imagen.py:518, :538) when denoised_out != NULL. */
int b200_edm_phase_sc(int phase, float* x, float* x_hat, float* x1, float* d, float* net_in,
                      const float* pred, const float* eps, const b200_edm_coef* coefs, int32_t* step_ctr,
                      int32_t* slots, int R, int B, int64_t chw, float cond_scale, int thresholding,
                      int32_t q_lo, int32_t q_hi, float q_w, float* denoised_out, void* stream);

/* RePaint inpainting conditioning (imagen_pytorch.py:2248-2250, :2285-2286): where mask[b, p] != 0 (uint8 [B, HW], shared by the C
 * channels) x <- alpha * known + sigma * noise (q_sample :272-284; noise may be NULL with sigma == 0 for the final paste). */
int b200_inpaint_mix(float* x, const float* known, const uint8_t* mask, const float* noise, float alpha, float sigma,
                     int B, int C, int64_t hw, void* stream);
/* q_sample_from_to (imagen_pytorch.py:286-306), the RePaint re-noising between resamples:
 * x <- x * c1 + (noise * c2) / alpha, c1 = alpha_to / alpha, c2 = sigma_to * alpha - sigma * alpha_to (tabulated on the host). */
int b200_renoise(float* x, const float* noise, float c1, float c2, float alpha, int64_t n, void* stream);

/* flags bit 0: out = (v + 1) * 0.5 (unnormalize_zero_to_one, imagen_pytorch.py:2288); bit 1: skip the clamp(x, -1, 1) of :2281
 * (the caller already clamped, then pasted the inpainting pixels). */
int b200_finalize_images(const float* x, float* out, int64_t n, int flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_IMAGEN_H_ */
