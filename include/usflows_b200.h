/* usflows_b200 -- C ABI of the B200 (sm_100a) flow-evaluation library  (libusflows_b200.so)
 *
 * Drop-in boundary for the hot path of aai-institute/USFlows: the per-layer forward (sample) and
 * backward (log_prob) passes of a `Flow`/`USFlow` layer stack and the base-distribution log-density.
 * The reference is pure Python/PyTorch and has no FFI of its own; each entry point below names the
 * reference call site(s) (file:line under /root/reference/src/usflows) whose arithmetic it replaces.
 * The Python host package `usflows_b200` binds these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in `_host`; buffers are caller-owned
 *  - matrices are row-major; `ld*` are leading dimensions in ELEMENTS
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream)
 *  - every function returns USF_OK (0) or a negative USF_ERR_* code; the message is in usf_last_error()
 *  - no CPU fallback exists: without a CUDA device every compute entry point returns USF_ERR_CUDA
 */
#ifndef USFLOWS_B200_H
#define USFLOWS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define USF_ABI_VERSION 10  /* ABI 10: the accumulation / pixel-plane tuning setters and the GEMM timeline hook are gone; usf_debug_set_store_path */

#define USF_OK 0
#define USF_ERR_INVALID (-1)     /* bad argument (shape, alignment, null pointer) */
#define USF_ERR_CUDA (-2)        /* CUDA runtime / driver error, no device, launch failure */
#define USF_ERR_UNSUPPORTED (-3) /* valid request this build cannot serve */
#define USF_ERR_INFEASIBLE (-4)  /* a layer is not invertible (zero on diag(U) or in scale) */

/* contraction engines (usf_linear_args.engine) */
#define USF_ENGINE_SIMT 0      /* fp32 FFMA, CUDA cores; any shape / alignment                         */
#define USF_ENGINE_TC_3XTF32 1 /* tcgen05 kind::tf32, 3-term split (hi*hi + lo*hi + hi*lo): ~fp32 accuracy */
#define USF_ENGINE_TC_TF32 2   /* tcgen05 kind::tf32, single pass                                      */
#define USF_ENGINE_TC_BF16 3   /* tcgen05 kind::f16 (bf16 operands), fp32 accumulate                   */
#define USF_ENGINE_TC_3XF16 4  /* tcgen05 kind::f16, fp16 split x = hi + lo'*2^-11 (3 products, the cross terms rescaled
                                  in the accumulator by scale-input-d): ~fp32 accuracy at twice the tf32 rate; values
                                  with |x| > 65000 raise the caller's overflow flag (re-run with TC_3XTF32)           */

/* base distributions (distributions.py:199-238) */
#define USF_BASE_LAPLACE 0
#define USF_BASE_NORMAL 1

/* Lp-radial base distribution (distributions.py:327-372): the norm and the distribution of the radius */
#define USF_LP_INF 0
#define USF_LP_1 1
#define USF_LP_2 2
#define USF_NORM_LOGNORMAL 0     /* params = [mu, sigma]                                  (distributions.py:181-197) */
#define USF_NORM_GAMMA_MIXTURE 1 /* params = [logits (K) | concentration (K) | rate (K)]  (distributions.py:674-707) */
#define USF_NORM_GENGAMMA_MIXTURE 2 /* R = scale_k * S^(1 / power_k), S ~ Gamma(concentration_k, rate_k), mixed with softmax(logits):
                                       params = [logits (K) | concentration (K) | rate (K) | scale (K) | power (K)].  One kind for the
                                       reference's Chi(df, scale) (distributions.py:55-116: a = df / 2, b = 1 / 2, power 2), torch's
                                       HalfNormal, Weibull(scale, concentration) (a = b = 1, power = concentration) and WeibullMM
                                       (distributions.py:835-848)  (ABI 6; the per-component scale / power layout is ABI 8) */
#define USF_NORM_LOGNORMAL_MIXTURE 3 /* params = [logits (K) | mu (K) | sigma (K)]: LogNormalMM (distributions.py:821-833)  (ABI 8) */

/* output planes of an activation in the operand format(s) of an engine mode; unused planes are NULL */
typedef struct usf_planes {
  float* f32;  int64_t ld_f32;
  float* hi;   float* lo;  int64_t ld_split;   /* tf32 split  */
  void* bf16;  int64_t ld_bf16;
  void* h16;   void* l16;  int64_t ld_16;      /* fp16 split (x = h16 + l16 * 2^-11) */
} usf_planes;

const char* usf_last_error(void);
int usf_abi_version(void);
/* device properties of the current CUDA device; any pointer may be NULL */
int usf_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes);

/* ------------------------------------------------------------------------------------------------
 * usf_linear: out[M,N] = epilogue( A[M,K] . W[N,K]^T )
 *   v = acc + bias[n]; if relu: v = max(v,0); if resid: v = resid[m,n] + resid_sign * v;
 *   if colscale: v *= colscale[n]; if postsub: v -= postsub[n]; stored to every non-NULL output plane.
 * Replaces: F.linear in BlockAffineTransform.forward/backward (transforms.py:934, 960-961),
 *           LUTransform.forward/backward (:1255, :1267-1268), pyro.nn.DenseNN's Linear+ReLU stack,
 *           the masked residual add/sub of MaskedCoupling.forward/backward (:284-290, :301-306) and
 *           ScaleTransform.forward (:105-114) when fused as `colscale`.
 * Operand planes by engine:
 *   SIMT      a (fp32) [+ a_lo added to it], w (fp32) [+ w_lo]; trans_w=1 reads w as [K,N]
 *   TC_3XTF32 a, a_lo, w, w_lo: fp32 storage holding tf32-representable values (x = hi + lo)
 *   TC_TF32   a, w fp32 (low 13 mantissa bits ignored by the tensor core)
 *   TC_BF16   a, w bf16
 *   TC_3XF16  a, a_lo, w, w_lo: fp16 planes (hi, lo' = (x - hi) * 2^11); outputs in out_h16/out_l16, residual
 *             from resid_h16/resid_l16 (or the fp32 `resid`)
 * tcgen05 engines need 16-byte aligned operand pointers and lda/ldw multiples of 4 (8 for bf16 / fp16).
 */
typedef struct usf_linear_args {
  int64_t M;
  int32_t N;
  int32_t K;
  int32_t engine;
  int32_t trans_w;
  const void* a;
  const void* a_lo;
  int64_t lda;
  const void* w;
  const void* w_lo;
  int64_t ldw;
  const float* bias;
  int32_t relu;
  float resid_sign;
  const float* resid;
  const float* resid_lo;
  int64_t ldr;
  const float* colscale;
  const float* postsub;
  float* out_f32;
  int64_t ld_f32;
  float* out_hi;
  float* out_lo;
  int64_t ld_split;
  void* out_bf16;
  int64_t ld_bf16;
  /* fp16 split planes (any engine may write them; TC_3XF16 reads them) */
  const void* resid_h16;
  const void* resid_l16;
  int64_t ldr_16;
  void* out_h16;
  void* out_l16;
  int64_t ld_16;
  int32_t* overflow_flag; /* device int, set to 1 if a value written to out_h16 exceeds the fp16 range */
  /* ABI 4.  split_k > 1 (the fp16-split engine TC_3XF16 only; ignored elsewhere): the contraction over K is cut into up to
   * split_k pieces that run on different CTA pairs and are summed into out_f32 with vector reductions -- for products
   * with a small output and a long K, i.e. the weight gradients dW[N_w, K_w] = dY^T . X of the training pass
   * (reference: autograd of F.linear, flows.py:199).  Requires out_f32 (16-byte aligned, ld_f32 % 4 == 0, N % 8 == 0)
   * as the only output and no bias / relu / residual / colscale / postsub; the library zero-fills out_f32 first. */
  int32_t split_k;
  int32_t reserved0;
} usf_linear_args;

int usf_linear(const usf_linear_args* args, void* stream);

/* test hook: force the tcgen05 tile width BLOCK_N (0 = automatic) */
int usf_debug_set_block_n(int block_n);
/* test hook: 1 (default) = the kernels of an evaluation are chained with programmatic dependent launch, 0 = plain
 * stream order */
int usf_debug_set_pdl(int on);
/* test hook for the CTA-pair tcgen05 kernel: force the store / residual paths that automatic choice takes only on other
 * shapes or configurations (0 = automatic; results are bit-identical on every path).  `flags` combines 4 = outputs leave
 * through the generic register/patch store path instead of the staged coalesced one, 32 = the epilogue warps copy their
 * staged boxes out themselves instead of issuing TMA stores, 256 = the coupling residual is read lane-per-row instead of
 * coalesced through the epilogue warp's in-box.  Any other bit: USF_ERR_INVALID. */
int usf_debug_set_store_path(int flags);

/* ------------------------------------------------------------------------------------------------
 * whole layer stack in one launch for tiny event sizes (d <= 8, conditioner width <= 64): replaces the per-layer loop
 * of Flow.log_prob / Flow.sample (flows.py:234-245, 258-265) where a layer is far below one MMA tile (BASELINE config C1:
 * d = 2, H = 32).  Rows and hidden activations live in registers, the weights of all layers in shared memory.
 *   prog : n_ops pairs (code, offset): code = 0 affine `x <- W x + c` (W [D,D] row-major then c [D] at blob + offset) or
 *          1 | (n_mid << 8) coupling `x <- x + W_last relu(.. relu(W_0 x + b_0) ..) + b_last` with blocks
 *          W_0 [H,D], b_0 [H], n_mid x (W [H,H], b [H]), W_last [D,H], b_last [D]; mask and sign folded into W_0 / W_last.
 *   blob : fp32 weights, 16-byte aligned, every op block starting at a multiple of 4 floats; d padded to D in {2,4,8}
 *          (identity / zero padding), hidden widths padded to H in {32,64} with zeros.
 * out [rows, d] receives the transformed rows (the base density runs through usf_base_logprob). */
int usf_flow_small(const float* x, int64_t ldx, int64_t rows, int32_t d, const int32_t* prog, int32_t n_ops,
                   const float* blob, int32_t blob_floats, int32_t D, int32_t H, float* out, int64_t ldo, void* stream);

/* ------------------------------------------------------------------------------------------------
 * elementwise / reduction kernels over [N_rows, d] activations (HBM-bound, 128-bit accesses)
 */

/* out = ((x / div[j]) * mul[j]) - sub[j]  (each vector optional), written to any of the planes.
 * Replaces ScaleTransform.backward (transforms.py:116-125), ScaleTransform.forward (:105-114), the
 * `y - b` of BlockAffineTransform.backward (:959) for the first layer, and the fp32 -> operand-format
 * conversion of user input. */
int usf_ingest(const float* x, int64_t ldx, int64_t rows, int32_t d, const float* div, const float* mul,
               const float* sub, float* out_f32, int64_t ld_f32, float* out_hi, float* out_lo,
               int64_t ld_split, void* out_bf16, int64_t ld_bf16, void* stream);
/* same, writing the fp16 split planes of the TC_3XF16 engine (+ overflow flag, may be NULL) */
int usf_ingest_f16(const float* x, int64_t ldx, int64_t rows, int32_t d, const float* div, const float* mul,
                   const float* sub, void* out_h16, void* out_l16, int64_t ld_16, int32_t* overflow_flag,
                   void* stream);

/* 8-bit inputs (dequantisation of image data, the reference's DequantizedDataset: x = pixel / 256 + U(0, 1/256)).
 * Value k in 0..255 at flat event index j (row-major over the event, e.g. c*H*W + h*W + w) of GLOBAL row r becomes
 *   USF_DEQUANT_UNIFORM:  x = (k + u) / 256,  u = (2m + 1) / 2^16,  m = Philox4x32-10(key = seed, counter = (r, j >> 2))[j & 3] >> 17
 *   USF_DEQUANT_MIDPOINT: x = (k + 0.5) / 256
 * (counter words and rounds as usf_base_sample's).  Every x is exact in fp32 and lies strictly inside (k/256, (k+1)/256); the
 * noise depends on (seed, r, j) only.  r = row0 + the row's index in the call; when dev_params (device memory, 2 x int64) is
 * given, the kernel reads {seed, row base} there at run time: seed is replaced, row base is added to row0 (a captured graph
 * can then be replayed with new values). */
#define USF_DEQUANT_UNIFORM 0
#define USF_DEQUANT_MIDPOINT 1
typedef struct usf_dequant {
  int32_t mode;
  int32_t reserved0;
  uint64_t seed;
  int64_t row0;
  const int64_t* dev_params;
} usf_dequant;
/* usf_ingest / usf_ingest_f16 reading 8-bit rows x [rows, ldx] (bytes): out = ((dequant(x) / div) * mul) - sub into every
 * non-NULL plane of `out` (+ the fp16 range flag, may be NULL).  With only the fp32 plane it is the plain dequantisation. */
int usf_ingest_u8(const uint8_t* x, int64_t ldx, int64_t rows, int32_t d, const usf_dequant* dq, const float* div,
                  const float* mul, const float* sub, const usf_planes* out, int32_t* overflow_flag, void* stream);

/* out[r] = sum_j logpdf_base(z[r,j]; loc[j], scale[j]) + add_const  (z = z_hi [+ z_lo]).
 * Replaces DistributionModule.log_prob (distributions.py:150-151; torch Laplace/Normal.log_prob +
 * Independent sum) and the `+ log_det` of Flow.log_prob (flows.py:234-245). */
int usf_base_logprob(const float* z, const float* z_lo, int64_t ldz, int64_t rows, int32_t d,
                     const float* loc, const float* scale, int32_t base_kind, float add_const,
                     float* out, void* stream);

/* Affine coupling update (EXTENSION: the reference's MaskedCoupling, transforms.py:254-347, is additive only; this is
 * the scale-and-shift form named by the task).  st [rows, 2h]: conditioner outputs of the h updated features, log-scale s
 * in columns [0,h), shift t in [h,2h).  direction +1: x <- x*exp(s) + t, -1: x <- (x - t)*exp(-s), s clamped to
 * [s_min, s_max]; x is given in the planes of the engine mode (any of f32 / hi+lo / bf16 / h16+l16) and updated in place;
 * row_ladj[r] += sum_j s[r,j] (the layer's forward log|det J| of that row; may be NULL). */
int usf_affine_couple(const float* st, int64_t ld_st, int64_t rows, int32_t h, float* x_f32, int64_t ld_f32, float* x_hi,
                      float* x_lo, int64_t ld_split, void* x_bf16, int64_t ld_bf16, void* x_h16, void* x_l16, int64_t ld_16,
                      int32_t* overflow_flag, float direction, float s_min, float s_max, float* row_ladj, void* stream);
/* out[i] -= v[i]: per-row log-determinants leave the log-density (flows.py:234-245 with data-dependent layers) */
int usf_sub_rows(float* out, const float* v, int64_t n, void* stream);

/* z[r,j] = loc[j] + scale[j] * eps with eps ~ Laplace(0,1) or N(0,1) from Philox4x32-10(seed, offset).
 * Replaces DistributionModule.sample (distributions.py:147-148) in Flow.sample (flows.py:258). */
int usf_base_sample(int64_t rows, int32_t d, const float* loc, const float* scale, int32_t base_kind,
                    uint64_t seed, uint64_t offset, float* out_f32, int64_t ld_f32, float* out_hi,
                    float* out_lo, int64_t ld_split, void* out_bf16, int64_t ld_bf16, void* stream);

/* Philox key and counter base of one sampling call (usf_base_sample_at / usf_radial_sample_at).  Every counter that the
 * plain entries key by the row index r within the call is keyed by the GLOBAL row row0 + r instead: counter
 * ((row0 + r) * ceil(d / 4) + g, offset) for the 4-column group g of the coordinates, and (row0 + r, offset ^ tag [+ k]) for
 * the radius, mixture component, rejection rounds and extremal coordinate of the radial sampler.  Rows [r0, r1) of one call
 * therefore equal a call over r1 - r0 rows with row0 = r0, and usf_base_sample / usf_radial_sample are the row0 = 0 calls.
 * When dev_params (device memory, 2 x int64) is given, the kernel reads {seed, row base} there at run time: seed is
 * replaced, row base is added to row0 (a captured graph can then be replayed for the next chunk). */
typedef struct usf_draw {
  uint64_t seed;
  uint64_t offset;
  int64_t row0;
  const int64_t* dev_params;
} usf_draw;
/* usf_base_sample with the draws of global rows draw->row0 .. draw->row0 + rows - 1 (row0 >= 0) */
int usf_base_sample_at(int64_t rows, int32_t d, const float* loc, const float* scale, int32_t base_kind,
                       const usf_draw* draw, float* out_f32, int64_t ld_f32, float* out_hi, float* out_lo,
                       int64_t ld_split, void* out_bf16, int64_t ld_bf16, void* stream);

/* 8-bit output, the inverse of usf_ingest_u8: out[r, j] = min(255, max(0, floor(256 y[r, j]))), NaN -> 0.  256 y is exact
 * in fp32, so every value usf_ingest_u8 makes of k (either mode) quantises back to k. */
int usf_quantize_u8(const float* y, int64_t ldy, int64_t rows, int32_t d, uint8_t* out, int64_t ldo, void* stream);

/* Lp-radial base density:  out[r] = log f_R(r_r) - [dv_const + (d-1) log r_r] + add_const,  r_r = ||z[r,:] - loc||_p
 * (z = z [+ z_lo]); f_R is LogNormal(mu, sigma) or a K-component mixture (K <= 128) of Gammas, generalised Gammas or
 * log-normals, `norm_params` as listed at USF_NORM_*, already constrained (sigma, concentration, rate, scale, power > 0;
 * logits raw).  dv_const = the r-independent part of
 * log dV_p^d/dr.  Replaces RadialDistribution.log_prob + log_delta_volume (distributions.py:501-549), the norm
 * distributions' log_prob (torch LogNormal / MixtureSameFamily(Categorical, Gamma)) and the `+ log_det` of Flow.log_prob. */
int usf_radial_logprob(const float* z, const float* z_lo, int64_t ldz, int64_t rows, int32_t d, const float* loc,
                       int32_t p_kind, int32_t norm_kind, const float* norm_params, int32_t n_comp, float dv_const,
                       float add_const, float* out, void* stream);
/* z[r,:] = loc + R_r * u_r,  R_r ~ f_R,  u_r uniform on the unit Lp sphere (p = 2: normalised Gaussian, p = 1: signed
 * Dirichlet(1..1), p = inf: uniform cube face with one coordinate pinned to +1, as UniformUnitLpBall.sample,
 * distributions.py:286-316); Philox4x32-10(seed, offset).  Replaces RadialDistribution.sample (distributions.py:478-499). */
int usf_radial_sample(int64_t rows, int32_t d, const float* loc, int32_t p_kind, int32_t norm_kind,
                      const float* norm_params, int32_t n_comp, uint64_t seed, uint64_t offset, float* out, int64_t ldo,
                      void* stream);
/* usf_radial_sample with the draws of global rows draw->row0 .. draw->row0 + rows - 1 (usf_draw) */
int usf_radial_sample_at(int64_t rows, int32_t d, const float* loc, int32_t p_kind, int32_t norm_kind,
                         const float* norm_params, int32_t n_comp, const usf_draw* draw, float* out, int64_t ldo,
                         void* stream);

/* Row-wise glue of networks.ConvNet's vector branch (networks.py:205-245, 287-307) between two usf_linear calls:
 *   v = gated ? xres[r,j] + o[r,j] * sigmoid(o[r,n+j]) : o[r,j]        (GatedMLP: o = [val | gate], xres = x or proj(x))
 *   v = pre_relu ? max(v, 0) : v                                        (ConvNet2D: GatedConv -> ReLU -> LayerNormChannels)
 *   v = gamma ? LayerNorm_row(v; gamma, beta, eps) : v                  (LayerNormVector / LayerNormChannels, biased variance)
 *   y_f32 <- v (may alias xres);  act <- act_relu ? max(v,0) : v;  raw <- v     (each of y_f32 / act / raw may be NULL)
 * n <= 6144.  overflow_flag: set when a value written to fp16 split planes leaves the fp16 range (may be NULL). */
int usf_gate_norm(const float* o, int64_t ldo, const float* xres, int64_t ldx, int64_t rows, int32_t n, int32_t gated,
                  int32_t pre_relu, const float* gamma, const float* beta, float eps, float* y_f32, int64_t ldy, const usf_planes* act,
                  int32_t act_relu, const usf_planes* raw, int32_t* overflow_flag, void* stream);

/* ---- image-shaped flows (in_dims = [C, H, W]): channels-last rows [N*H*W, C] inside the layer stack ----------------
 * out[n, b, a] = f(in[n, a, b]) for in [N, A, B] (NCHW -> channels-last rows with A = C, B = H*W, and back with A = H*W,
 * B = C); f multiplies (scale_mode 1) or divides (2) by `scale`, indexed in the order of the NCHW side (scale_on_input:
 * the input is the NCHW side).  Replaces the layout the reference's conv calls imply and ScaleTransform.forward/backward
 * over [C, H, W] (transforms.py:105-125). */
int usf_layout_transpose(const float* in, int64_t n, int32_t a, int32_t b, const float* scale, int32_t scale_mode,
                         int32_t scale_on_input, float* out, void* stream);
/* the channels-last -> NCHW direction of usf_layout_transpose (scale_on_input = 0: `scale` indexed in NCHW order on the
 * output side) writing 8-bit images: each fp32 value it would write is quantised as usf_quantize_u8 does */
int usf_layout_transpose_to_u8(const float* in, int64_t n, int32_t a, int32_t b, const float* scale, int32_t scale_mode,
                               uint8_t* out, void* stream);
/* the NCHW -> channels-last direction of usf_layout_transpose (A = c, B = hw, scale on the input side) reading 8-bit images
 * in [n, c, hw], dequantised as usf_ingest_u8 does (j = c_index * hw + pixel, r = dq->row0 + image index) */
int usf_layout_transpose_u8(const uint8_t* in, int64_t n, int32_t c, int32_t hw, const usf_dequant* dq, const float* scale,
                            int32_t scale_mode, float* out, void* stream);
/* Operand rows of a k x k convolution (stride 1, zero padding 'same', dilation) over channels-last rows:
 *   out[r, (kh*k + kw)*C + c] = g(in[pixel (h + (kh - k/2) dil, w + (kw - k/2) dil) of r's image, c]), 0 outside;
 *   g = optional multiply by mask[(h'*W + w')*C + c] (the coupling's x * mask, transforms.py:286), then optional ReLU.
 * With usf_linear over K = k*k*C this replaces nn.Conv2d in ConvNet2D / GatedConv (networks.py:61-121, 405-510); the
 * weight is the conv weight permuted to [C_out, kh, kw, C_in]. */
int usf_im2col(const float* in, int64_t ld_in, int64_t n_images, int32_t h, int32_t w, int32_t c, int32_t k, int32_t dilation,
               const float* mask, int32_t relu, const usf_planes* out, int32_t* overflow_flag, void* stream);
/* The same convolution WITHOUT the materialised operand rows (implicit GEMM on tcgen05): out = epilogue(conv(g(act)))
 * over channels-last rows act [n*h*w, c_in]; `a` describes the contraction part as for usf_linear -- M = n*h*w,
 * K = k*k*c_in, N <= 64, w / w_lo = tf32 hi / lo planes of the weight [N, K] in the usf_im2col column order (a->a, a->a_lo,
 * a->engine are ignored), bias, relu and the output planes; no residual / colscale / postsub.  fp32-accurate (3-term tf32
 * split).  c_in % 16 == 0.  The whole weight stays resident in shared memory: USF_ERR_UNSUPPORTED when
 * 3 * 32 KB + ceil(K/32) * 2 * (N <= 32 ? 32 : 64) * 128 B exceeds 227 KB (use usf_im2col + usf_linear then). */
int usf_conv2d_rows(const usf_linear_args* a, const float* act, int64_t ld_act, int64_t n_images, int32_t h, int32_t w,
                    int32_t c_in, int32_t k, int32_t dilation, const float* mask, int32_t relu_in, void* stream);
/* ---- pixel planes (ABI 5): the ConvNet2D conditioner without gather threads (csrc/conv_pix.cuh) ------------------------
 * An activation with <= 32 channels as [n*h*w, 64] fp16: per pixel 32 high halves | 32 low halves' (x = hi + lo' 2^-11,
 * missing channels zero) = one 128-byte operand row; a k x k tap of 256 pixels is ONE 4-D TMA box (zero padding 'same' by
 * the hardware's out-of-bounds fill).
 * usf_pix_encode: fp32 channels-last rows x [rows, c] (c <= 32) -> pixel planes, times mask[(r mod hw)*c + ch] when mask is
 * given (the coupling's x * mask, transforms.py:286), then optional ReLU. */
int usf_pix_encode(const float* x, int64_t ldx, int64_t rows, int32_t c, int32_t hw, const float* mask, int32_t relu,
                   void* out16, int32_t* overflow_flag, void* stream);
typedef struct usf_conv_pix_args {
  const void* a16;       /* input pixel planes [n*h*w, 64] fp16 */
  int64_t n_images;
  int32_t h, w, ksize, dilation;   /* odd ksize, stride 1, padding 'same' */
  const void* w1;        /* [32, k*k*64] fp16: row = output channel (rows >= n1 zero), per tap 32 hi | 32 lo' input channels */
  const float* bias1;    /* [32], entries >= n1 zero */
  int32_t n1;            /* output channels of the k x k convolution (<= 32, multiple of 4; gated: 32) */
  int32_t relu1;         /* plain: ReLU on conv + bias */
  int32_t gated;         /* 0 = plain, 1 = GatedConv block (networks.py:100-121) */
  int32_t post_relu;     /* gated: ReLU after the gate (ConvNet2D applies its nonlinearity to the GatedConv output) */
  const void* w2;        /* gated: [64, 64] fp16, rows = val (32) | gate (32) channels of the 1 x 1 convolution, 32 hi | 32 lo' */
  const float* bias2;    /* gated: [64] */
  const float* gamma;    /* LayerNormChannels over the n1 channels, after relu1 / post_relu (NULL: none; networks.py:40-58) */
  const float* beta;
  float eps;
  float sign;            /* plain + x: sign of the coupling update */
  float* out_f32;        /* plain: result rows [n*h*w, n1] (optional); gated: residual stream y [n*h*w, 32], updated in place */
  int64_t ld_f32;
  void* out16;           /* pixel planes of the result (optional) */
  int32_t relu_planes;   /* the planes hold max(result, 0) (the ReLU in front of the next convolution) */
  int32_t c_x;           /* plain + x: channels of x (<= n1) */
  float* x;              /* plain: x[r, c] += sign * inv_mask[(r mod h*w)*c_x + c] * result[r, c] (transforms.py:284-290) */
  int64_t ldx;
  const float* inv_mask;
  int32_t* overflow_flag;   /* set when a value written to fp16 planes leaves the fp16 range (may be NULL) */
} usf_conv_pix_args;
/* Plain: result = [LayerNorm]([ReLU](conv_kxk(a16) + bias1)) -> out_f32 / out16 / the coupling update of x.
 * Gated: u = relu(conv_kxk(a16) + bias1); [val | gate] = w2 u + bias2 (same kernel, second TMEM accumulator);
 *        y <- [LayerNorm]([ReLU](y + val * sigmoid(gate))) in place, + its pixel planes.  fp32-accurate (fp16 split, 3 products).
 * Replaces nn.Conv2d, GatedConv.forward, the ReLU and LayerNormChannels of ConvNet2D (networks.py:40-121, 405-494) and, for the
 * last convolution, MaskedCoupling's update.  USF_ERR_UNSUPPORTED when w > 256 or the k*k*4 KB weight leaves no room for two
 * 32 KB pipeline stages in 227 KB of shared memory. */
int usf_conv2d_pix(const usf_conv_pix_args* a, void* stream);

/* x[r, c] += sign * g[(r mod hw)*c_dim + c] * t[r, c]: MaskedCoupling.forward/backward with a mask over [C, H, W]
 * (transforms.py:284-290, 301-306; g = 1 - mask in channels-last order). */
int usf_masked_add(float* x, int64_t ldx, const float* t, int64_t ldt, int64_t rows, int32_t c, int32_t hw, const float* g,
                   float sign, void* stream);

/* y = x >= 0 ? x : slope * x ; optional per-row count of negative inputs (for log|det J| = log(slope)*count).
 * Replaces LeakyReLUTransform.forward/backward (transforms.py:434-454). */
int usf_leaky_relu(const float* x, int64_t ldx, int64_t rows, int32_t d, float slope, float* y,
                   int64_t ldy, float* neg_count, void* stream);

/* y[r,j] = x[r,perm[j]].  Replaces Permute._call/_inverse (transforms.py:213-232). */
int usf_permute(const float* x, int64_t ldx, int64_t rows, int32_t d, const int32_t* perm, float* y,
                int64_t ldy, void* stream);

/* ------------------------------------------------------------------------------------------------
 * weight preparation (runs once per weight version; all matrices [d,d] fp32 with leading dim ld)
 */

/* L = tril(L_raw,-1) + I  and  U = triu(U_raw)  (transforms.py:1271-1279); either output may be NULL.
 * `transpose_u` writes U^T instead (operand layout for L @ U as A . B^T). */
int usf_lu_assemble(const float* L_raw, const float* U_raw, int32_t d, int64_t ld_raw, float* L, float* U,
                    int64_t ld_out, int32_t transpose_u, void* stream);

/* out[0] = sum_i log|U_raw[i,i]| (transforms.py:1303-1320), out[1] = number of zero diagonal entries
 * (LUTransform.is_feasible, :1347-1349).  `out` is 2 floats on the device. */
int usf_lu_logabsdet(const float* U_raw, int32_t d, int64_t ld, float* out, void* stream);

/* out[0] = sum log|v_j| , out[1] = number of zeros (ScaleTransform.log_abs_det_jacobian / is_feasible,
 * transforms.py:135-152). */
int usf_vec_logabs(const float* v, int64_t n, float* out, void* stream);

/* X = T^-1 for a triangular T (lower != 0: lower triangular, else upper); unit_diag != 0 takes the
 * diagonal as 1.  Replaces torch.inverse(self.L) / torch.inverse(self.U) (transforms.py:1264-1265,
 * 1291-1292).  `work` is a device scratch of usf_tri_inverse_work_floats(d) floats. */
int64_t usf_tri_inverse_work_floats(int32_t d);
int usf_tri_inverse(const float* T, int32_t d, int64_t ldt, int32_t lower, int32_t unit_diag, float* X,
                    int64_t ldx, float* work, void* stream);

/* out[c,r] = in[r,c] */
int usf_transpose(const float* in, int32_t rows, int32_t cols, int64_t ld_in, float* out, int64_t ld_out,
                  void* stream);

/* out[r,c] = in[r,c] * rowf[r] * colf[c]   (either factor vector optional) -- folds the coupling mask
 * into the conditioner's first / last Linear (transforms.py:284-289). */
int usf_scale_rows_cols(const float* in, int32_t rows, int32_t cols, int64_t ld_in, const float* rowf,
                        const float* colf, float* out, int64_t ld_out, void* stream);

/* tf32 split planes / bf16 copy of an fp32 matrix (operand formats of the tcgen05 engines) */
int usf_split_tf32(const float* in, int64_t rows, int32_t cols, int64_t ld_in, float* hi, float* lo,
                   int64_t ld_out, void* stream);
int usf_to_bf16(const float* in, int64_t rows, int32_t cols, int64_t ld_in, void* out, int64_t ld_out,
                void* stream);
/* fp16 split planes of an fp32 matrix: hi = fp16(x), lo = fp16((x - hi) * 2^11); flag as in usf_ingest_f16 */
int usf_split_f16(const float* in, int64_t rows, int32_t cols, int64_t ld_in, void* hi, void* lo, int64_t ld_out,
                  int32_t* overflow_flag, void* stream);

/* W <- W @ (I - 2 v v^T / v.v) in place (one Householder reflection, transforms.py:795-809);
 * `work` = d floats. */
int usf_householder_right(float* W, int32_t d, int64_t ld, const float* v, float* work, void* stream);

/* C[M,N] = A[M,K] . B[K,N], row-major fp64 (leading dimensions in elements).  Composition of neighbouring
 * affine layers into one operator (SequentialAffineTransform.matrix/inverse_matrix, transforms.py:1457-1469,
 * and the products across Aff_i^-1 / Aff_{i+1} boundaries) in higher precision than the layers run in. */
int usf_matmul_f64(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int32_t M,
                   int32_t N, int32_t K, void* stream);

/* The same product for the triangular factors of an LU layer (ABI 7): `USF_TRI_LOWER_UPPER` C = L . U (the layer's matrix,
 * transforms.py:1281-1283), `USF_TRI_UPPER_LOWER` C = U^-1 . L^-1 (its inverse, :1291-1293).  A and B are dense d x d
 * arrays WITH their zeros stored; the kind only lets a tile skip the k range in which one factor is zero (a third of
 * the work of the dense product).  The result is the full dense d x d matrix. */
#define USF_TRI_NONE 0
#define USF_TRI_LOWER_UPPER 1
#define USF_TRI_UPPER_LOWER 2
int usf_matmul_f64_tri(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int32_t d,
                       int32_t tri, void* stream);

/* out[j] = softplus(in[j])  (distributions.py:211-215, base scale parameterisation) */
int usf_softplus(const float* in, int64_t n, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Whole-stack evaluation (ABI 4).  A plan is the launch sequence of ONE direction of a layer stack whose steps are all
 * contractions (every USFlow with DenseNN conditioners): ingest -> usf_linear chain -> base density.  Replaces the
 * per-layer loops of Flow.log_prob (flows.py:225-245), Flow.backward (:57-67) and Flow._forward (:45-55) with one call
 * per batch; the host that builds the plan passes prepared operands (the same ones usf_linear takes).  The plan owns
 * its device workspaces (allocated by usf_plan_finalize for `max_rows` rows, freed by usf_plan_destroy) and keeps
 * POINTERS to the operands, biases and base parameters it was given: they must stay alive and unchanged while it is used.
 * One plan per device and stream at a time.
 * ------------------------------------------------------------------------------------------------ */
typedef struct usf_plan usf_plan;
enum usf_mode { USF_MODE_FP32 = 0, USF_MODE_FP32_TF32 = 1, USF_MODE_FP32_SIMT = 2, USF_MODE_TF32 = 3, USF_MODE_BF16 = 4 };
enum usf_plan_src { USF_PLAN_SRC_STREAM = 0, USF_PLAN_SRC_HIDDEN = 1 };
enum usf_plan_dst { USF_PLAN_DST_STREAM = 0,   /* new stream activation (the LAST step writes the fp32 result instead) */
                    USF_PLAN_DST_HIDDEN = 1,   /* conditioner hidden activation */
                    USF_PLAN_DST_SEGMENT = 2   /* coupling output: stream[:, out_col0 : out_col0 + N] += resid_sign * value, in place */ };
typedef struct usf_plan_linear {
  int32_t N, K, engine, relu;
  const void* w; const void* w_lo; int64_t ldw;     /* operand planes of the engine, [N, K] */
  const float* bias;
  int32_t src, dst;
  int32_t in_col0, in_width;                         /* src = stream: columns read as A (in_width = 0: all) */
  int32_t out_col0;
  float resid_sign;
} usf_plan_linear;
int usf_plan_create(usf_plan** plan, int32_t d_in, int32_t mode, int64_t max_rows);
int usf_plan_add_linear(usf_plan* plan, const usf_plan_linear* step);
/* base density of the latent (Laplace / Normal, prepared loc / scale as for usf_base_logprob); add_const = -sum of the
 * weight-only log-determinants */
int usf_plan_set_base(usf_plan* plan, int32_t base_kind, const float* loc, const float* scale, float add_const);
int usf_plan_finalize(usf_plan* plan);
int64_t usf_plan_workspace_bytes(const usf_plan* plan);
/* z[rows, width] (fp32) = the stack applied to x[rows, d_in] */
int usf_flow_apply(const usf_plan* plan, const float* x, int64_t ldx, int64_t rows, float* z, int64_t ldz,
                   int32_t* overflow_flag, void* stream);
/* out[r] = log p(x[r, :]) = base.log_prob(stack(x[r, :])) + add_const   (Flow.log_prob, flows.py:225-245) */
int usf_flow_logprob(const usf_plan* plan, const float* x, int64_t ldx, int64_t rows, float* out, int32_t* overflow_flag,
                     void* stream);
/* the same for 8-bit rows x [rows, ldx] (bytes), dequantised as usf_ingest_u8 does by the plan's first ingest */
int usf_flow_logprob_u8(const usf_plan* plan, const uint8_t* x, int64_t ldx, int64_t rows, const usf_dequant* dq, float* out,
                        int32_t* overflow_flag, void* stream);
int usf_plan_destroy(usf_plan* plan);

/* ------------------------------------------------------------------------------------------------
 * Training step (ABI 4).  Replaces what torch autograd does behind Flow.fit's loss.backward() (flows.py:199):
 * the batch-side products dX = dY . W and dW = dY^T . X are usf_linear calls (dW with split_k); these entries are the
 * passes between them and the weight-side algebra of LUTransform (transforms.py:1271-1293 and its derivative).
 * ------------------------------------------------------------------------------------------------ */
/* One pass over a [rows, n] matrix given as fp16 split planes (h, l) or as fp32 (src_f32, when h == NULL):
 *   value <- 0 where mask_h[r, j] <= 0 (ReLU backward: mask_h = hi plane of the saved post-ReLU activation);
 *   value <- sign * value;  out planes [rows, n] (may alias the input);  t planes = the TRANSPOSE [n, rows] (the K-major
 *   operand of dW = dY^T . X);  colsum[j] += sum_r value (bias gradient);  colsum2[j] += sum_r value * mul[r, j].
 * Every output is optional.  n % 8 == 0, 16-byte aligned planes, pitches multiples of 16 bytes. */
typedef struct usf_glue_args {
  const void* h; const void* l; int64_t ld;
  const float* src_f32; int64_t ld_src;
  int64_t rows; int32_t n; int32_t reserved0;
  const void* mask_h; int64_t ld_mask;
  float sign; int32_t reserved1;
  void* out_h; void* out_l; int64_t ld_out;
  void* t_h; void* t_l; int64_t ld_t;
  float* colsum;
  const float* mul; int64_t ld_mul;
  float* colsum2;
  int32_t* overflow_flag;
} usf_glue_args;
int usf_planes_glue(const usf_glue_args* args, void* stream);

/* g = d(-log p(z)) / dz of the Laplace / Normal base density (distributions.py:199-238), un-normalised, as fp16 split
 * planes g [rows, d] and (optional) transposed planes t [d, rows]; dloc[j] += sum_r d(-log p)/dloc_j,
 * dscale[j] += sum_r d(-log p)/dscale_j (scale = softplus'ed).  d % 8 == 0. */
int usf_base_backward(const float* z, int64_t ldz, int64_t rows, int32_t d, const float* loc, const float* scale,
                      int32_t kind, void* g_h, void* g_l, int64_t ld_g, void* t_h, void* t_l, int64_t ld_t,
                      float* dloc, float* dscale, void* stream);

/* Weight-side copy: out[i, j] = scale * S[ri(i), cj(j)] with S = src (transpose = 0) or src^T (1); row_idx / col_idx are
 * optional int32 gather indices; written as fp32 (out_f32) and / or fp16 split operand planes (out_h, out_l) and / or the
 * TRANSPOSED operand planes outT [cols, rows] of the same matrix (the operand of dX = dY . M next to the one of x . M^T). */
int usf_mat_prep(const float* src, int64_t ld_src, int32_t rows, int32_t cols, int32_t transpose, const int32_t* row_idx,
                 const int32_t* col_idx, float scale, float* out_f32, int64_t ld_f32, void* out_h, void* out_l,
                 int64_t ld_16, void* outT_h, void* outT_l, int64_t ld_T, int32_t* overflow_flag, void* stream);

/* The bias path of an inverse affine layer, y = (x - b) W^-T = x W^-T + c with c = -W^-1 b (transforms.py:936-962):
 *   usf_rowdot:  out[i] = alpha * sum_k W[row_idx ? row_idx[i] : i, k] * v[k]        (c = rowdot(W^-1, b, -1))
 *   usf_colcomb: out[j] += alpha * sum_i v[i] * W[i, j]                               (db -= dc . W^-1)
 *   usf_rank1:   A[i, j] += alpha * u[i] * v[j]                                       (dW^-1 -= dc (x) b) */
int usf_rowdot(const float* W, int64_t ld, int32_t n_rows, int32_t K, const int32_t* row_idx, const float* v, float alpha,
               float* out, void* stream);
int usf_colcomb(const float* W, int64_t ld, int32_t rows, int32_t cols, const float* v, float alpha, float* out,
                void* stream);
int usf_rank1(float* A, int64_t ld, int32_t rows, int32_t cols, const float* u, const float* v, float alpha, void* stream);

/* out = scale * (strict lower part of src, mode 0 | upper part incl. diagonal, mode 1) [+ coef / diag_src[i, i] on the
 * diagonal, mode 1]: the gradient masks of LUTransform (transforms.py:1209-1213) and d(sum log|diag U|)/dU. */
int usf_tri_mask(const float* src, int64_t ld_src, int32_t d, int32_t mode, float scale, const float* diag_src,
                 int64_t ld_diag, float coef, float* out, int64_t ld_out, void* stream);

/* Inverses of a stack of n_mats (<= 32) lower-triangular [d, d] matrices (pitch ld, matrix stride mat_stride floats) by
 * recursive block doubling; bit m of unit_mask: matrix m has an implicit unit diagonal (L of LUTransform).  X and tmp are
 * stacks of the same geometry (tmp: scratch).  Replaces torch.inverse(L) / torch.inverse(U) (transforms.py:1291-1292) for
 * all layers of a flow in 1 + 2 log2(d / 64) launches. */
int usf_tri_inverse_batched(const float* T, float* X, float* tmp, int32_t d, int64_t ld, int64_t mat_stride,
                            int32_t n_mats, uint32_t unit_mask, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* USFLOWS_B200_H */
