/*
 * whvi_b200 -- C ABI of the B200-native WHVI hot path (libwhvi_b200.so, sm_100a).
 *
 * This is the drop-in boundary: the entry points below are what the reference's
 * Python layer binds instead of its two torch C++/CUDA extensions.  Every function
 *   - takes plain device pointers and sizes (no torch types),
 *   - is stream-ordered on the cudaStream_t passed as `stream` (NULL = legacy default
 *     stream), never synchronises, never allocates or frees device memory (the caller
 *     owns every buffer, including workspaces sized by the *_workspace_bytes calls),
 *   - returns 0 on success, a negative WHVI_E_* code for an invalid argument, or a
 *     positive cudaError_t for a CUDA failure (launch errors ARE checked, unlike the
 *     reference, src/fwht/cuda/fwht_cuda_kernel.cu:169-178); whvi_last_error() gives the
 *     thread-local message.  The Python side turns non-zero into RuntimeError, which is
 *     what the reference's TORCH_CHECKs raise (src/fwht/cuda/fwht_cuda.cpp:6-10).
 * All matrices are row-major contiguous fp32; device pointers must be 16-byte aligned.
 *
 * Reference interfaces replaced (file:line in ltdung/WHVI):
 *   whvi_fwht_f32            fwht_cuda.fwht            src/fwht/cuda/fwht_cuda.cpp:5-18
 *                            fwht_cuda_frontend        src/fwht/cuda/fwht_cuda_kernel.cu:156-181
 *                            fwht_cpp.forward/backward src/fwht/cpp/fwht.cpp:23-34
 *   whvi_layer_fwd_f32       WHVISquarePow2Matrix.sample_lrt / w_bar  src/weights.py:66-93
 *   whvi_layer_bwd_f32       autograd of the above (FWHTFunction.backward, src/fwht/cuda/fwht.py:14-16)
 *   whvi_reparam_*_f32       g_sigma + reparameterisation               src/weights.py:43-50, :82-83, :92-93
 *   whvi_kl_f32              WHVISquarePow2Matrix.kl -> kl_diag_normal  src/weights.py:52-64, src/utils.py:49-71
 */
#ifndef WHVI_B200_H
#define WHVI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WHVI_ABI_VERSION 1

#if defined(WHVI_BUILDING) && defined(__GNUC__)
#define WHVI_API __attribute__((visibility("default")))
#else
#define WHVI_API
#endif

#define WHVI_OK 0
#define WHVI_E_NULL (-1)      /* a required pointer is NULL                      */
#define WHVI_E_SHAPE (-2)     /* negative size, D not a power of two, D too big  */
#define WHVI_E_ALIGN (-3)     /* pointer not 16-byte aligned                     */
#define WHVI_E_MODE (-4)      /* unknown mode / flag                             */
#define WHVI_E_WORKSPACE (-5) /* workspace missing or too small                  */

typedef void* whvi_stream_t; /* a cudaStream_t */

/* Library / ABI identification. */
WHVI_API int whvi_abi_version(void);
/* Message for the last non-zero return on this thread ("" if none). */
WHVI_API const char* whvi_last_error(void);
/* Largest D (power of two) the FWHT accepts (single pass in shared memory up to 2^15,
 * multi-pass through global memory beyond).  The fused layer kernels state their own limits. */
WHVI_API int64_t whvi_max_dim(void);

/*
 * Batched fast Walsh-Hadamard transform, natural (Sylvester) order, unnormalised:
 *   out[r, :] = H_D . in[r, :]      for r in [0, rows)
 * D is a power of two, 1 <= D <= whvi_max_dim().  in == out (in place) is allowed;
 * partial overlap is not.  rows == 0 is a no-op.  fwd and bwd are the same call
 * (H is symmetric: src/fwht/cuda/fwht.py:14-16).
 */
WHVI_API int whvi_fwht_f32(const float* in, float* out, int64_t rows, int64_t D, whvi_stream_t stream);
/* The same transform in double precision (the reference dispatches double too,
 * src/fwht/cuda/fwht_cuda_kernel.cu:170, and its gradient check runs in double,
 * src/fwht/grad_check.py:26).  Parity tooling: correct for every D the fp32 entry accepts, not
 * tuned for bandwidth.  in == out allowed. */
/* out[r, :] = H_D . (scale * in[r, :]) with a (D) vector broadcast over the rows: the sample-independent first transform
 * t2 = H(s2 * x) of the layer (SURVEY 8d C5; feeds WHVI_LAYER_FROM_T2 / whvi_layer_moments_f32) in one pass.  4 <= D <= 2^15. */
WHVI_API int whvi_fwht_scaled_f32(const float* in, const float* scale, float* out, int64_t rows, int64_t D, whvi_stream_t stream);
/* bf16 activations in HBM (SURVEY 8f N4, not in the reference): the same transform with fp32 butterflies in registers and ONE
 * rounding (to nearest even) at the store, i.e. out = bf16( whvi_fwht_f32( float(in) ) ); 4 B/element of HBM traffic instead
 * of 8.  D <= 2^15 (single pass); pointers 8-byte aligned. */
WHVI_API int whvi_fwht_bf16(const void* in, void* out, int64_t rows, int64_t D, whvi_stream_t stream);
WHVI_API int whvi_fwht_f64(const double* in, double* out, int64_t rows, int64_t D, whvi_stream_t stream);

/*
 * Fused WHVILinear forward, PAPER semantics (docstring src/weights.py:77):
 *   y[s,b,:] = s1 * H( g[s,:] * H( s2 * x[s,b,:] ) ) (+ bias)
 * x: rows (s,b) at x + s*x_sample_stride + b*D; x_sample_stride is B*D for a contiguous
 *    (S,B,D) tensor or 0 when all samples share one (B,D) block (first layer of a net).
 * g: (S,D), one reparameterised vector per MC sample; s1, s2: (D); bias: (D) or NULL;
 * y: (S,B,D) contiguous.  4 <= D <= 32768, power of two (the backward supports D <= 8192).  Replaces the chain of ~20 torch
 * ops and the B x D x D GEMM of WHVISquarePow2Matrix.sample_lrt (src/weights.py:87-93).
 */
WHVI_API int whvi_layer_fwd_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1,
                                const float* s2, const float* bias, float* y, int64_t S, int64_t B, int64_t D,
                                whvi_stream_t stream);

/* The forward with bf16 activations in HBM (x, y bf16; g, s1, s2, bias fp32; arithmetic fp32, one rounding at the store):
 * y = bf16( whvi_layer_fwd_fused_f32( float(x) ) ).  Inference-side variant (SURVEY 8f N4): flags as the fused forward's
 * (WHVI_LAYER_RELU_OUT, WHVI_LAYER_FROM_T2), no target. */
WHVI_API int whvi_layer_fwd_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                 const float* bias, void* y, int64_t S, int64_t B, int64_t D, int flags, whvi_stream_t stream);

/* Bytes of device workspace whvi_layer_bwd_f32 needs for this shape. */
WHVI_API int whvi_layer_bwd_workspace_bytes(int64_t S, int64_t B, int64_t D, size_t* bytes);

/*
 * Fused WHVILinear backward (SURVEY Appendix A), recomputing the two forward transforms:
 *   dx[s,b,:] = s2 * H( g[s] * H( s1 * dy[s,b,:] ) )           (S,B,D), or NULL to skip
 *   dg[s,:]   = sum_b H(s1*dy) * H(s2*x)                        (S,D)
 *   ds1 = sum_{s,b} dy * H(g*H(s2*x));  ds2 = sum_{s,b} H(g*H(s1*dy)) * x     (D) each
 *   dbias = sum_{s,b} dy                                         (D), or NULL to skip
 * All outputs are overwritten (not accumulated).  Reductions use a fixed order, so results
 * are bit-reproducible run to run.  When x_sample_stride == 0 and dx != NULL, dx still has
 * the (S,B,D) shape; the caller sums it over s.
 */
WHVI_API int whvi_layer_bwd_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g,
                                const float* s1, const float* s2, float* dx, float* dg, float* ds1, float* ds2,
                                float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B,
                                int64_t D, whvi_stream_t stream);

/*
 * Fused variants (SURVEY 8f N1/N2: the steps either side of the layer folded into it).
 *  forward:  flags & WHVI_LAYER_RELU_OUT  -> y = max(y, 0) before the store (the nn.ReLU
 *            that follows the layer in the reference's networks);
 *            target != NULL ((B,D), broadcast over samples) -> additionally
 *            sq_partials[i] = partial sums of (y - target)^2, i < whvi_layer_fwd_partials();
 *            their plain sum is the data term of GaussianLikelihood.mnll_batch_estimate
 *            (src/likelihoods.py:18-29).
 *  backward: flags & WHVI_LAYER_RELU_IN   -> x is the output of a fused ReLU; dx is
 *            multiplied by (x > 0), i.e. it is the gradient w.r.t. the producer's
 *            pre-activation;
 *            target != NULL -> `dy` points at the layer's saved OUTPUT and the upstream
 *            gradient is formed on the fly as coef[0] * (output - target) (coef: device
 *            scalar), the gradient of the Gaussian MNLL, so it never exists in HBM.
 *  forward:  flags & WHVI_LAYER_FROM_T2   -> `x` already holds t2 = H(s2 * x) (one whvi_fwht_f32 of
 *            the scaled inputs, shared by all samples: the first transform is sample-independent,
 *            SURVEY 8d C5), so only y = s1 * H(g_s * t2) (+ bias) is left; s2 is not read.
 *            Not combinable with `target`.
 */
#define WHVI_LAYER_RELU_OUT 1
#define WHVI_LAYER_FROM_T2 2
#define WHVI_LAYER_RELU_IN 1
#define WHVI_LAYER_ACCUMULATE 4   /* whvi_layer_moments_f32: add to the existing contents of sum_y / sum_y2 */
#define WHVI_LAYER_RESERVE_SMS(n) (((n) & 0xFF) << 8)   /* whvi_layer_moments_f32: leave n SMs free (for a concurrent collective) */
WHVI_API int whvi_layer_fwd_partials(int64_t S, int64_t B, int64_t D, int64_t* count);
WHVI_API int whvi_layer_fwd_fused_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1,
                                      const float* s2, const float* bias, float* y, int64_t S, int64_t B, int64_t D,
                                      int flags, const float* target, float* sq_partials, whvi_stream_t stream);
WHVI_API int whvi_layer_bwd_fused_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g,
                                      const float* s1, const float* s2, float* dx, float* dg, float* ds1, float* ds2,
                                      float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B,
                                      int64_t D, int flags, const float* target, const float* coef,
                                      whvi_stream_t stream);

/* whvi_layer_bwd_f32 with the upstream gradient taken as dy_scale[0] * dy (dy_scale: device
 * scalar).  Lets a producer that computed its dx for a unit loss coefficient (whvi_layer_loss_f32)
 * hand it on without a separate scaling pass over the activations. */
WHVI_API int whvi_layer_bwd_scaled_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* dy_scale,
                                       const float* g, const float* s1, const float* s2, float* dx, float* dg,
                                       float* ds1, float* ds2, float* dbias, void* workspace, size_t workspace_bytes,
                                       int64_t S, int64_t B, int64_t D, int flags, whvi_stream_t stream);

/*
 * Fused LAST layer of a regression network: forward + Gaussian-MNLL residual + backward in one
 * pass over x (the predictions never touch HBM):
 *   y_hat = s1*H(g[s]*H(s2*x)) (+bias);  r = y_hat - target (target (B,D), shared by the samples)
 *   sq_partials[i], i < sq_count: partial sums of r^2 (their sum is the data term of
 *       GaussianLikelihood.mnll_batch_estimate, src/likelihoods.py:18-29).  The caller ZERO-FILLS the array:
 *       sq_count is an upper bound over the kernel variants (with / without bias), entries a variant does
 *       not use stay zero
 *   dx, dg, ds1, ds2, dbias: the layer's gradients for the upstream gradient dy = r, i.e. for a
 *       unit coefficient; the caller multiplies by 2 * dLoss/d(sum r^2) (the small vectors
 *       directly, dx through whvi_layer_bwd_scaled_f32 of the previous layer).
 * 128 <= D <= 4096.  flags: WHVI_LAYER_RELU_IN.  dx may be NULL; dbias is required iff bias.
 */
WHVI_API int whvi_layer_loss_sizes(int64_t S, int64_t B, int64_t D, size_t* workspace_bytes, int64_t* sq_count);
WHVI_API int whvi_layer_loss_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1,
                                 const float* s2, const float* bias, const float* target, float* dx, float* dg,
                                 float* ds1, float* ds2, float* dbias, float* sq_partials, void* workspace,
                                 size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int flags,
                                 whvi_stream_t stream);

/*
 * Training with bf16 activations in HBM (x, dy, dx bf16; parameters, their gradients, the target, the workspace and all
 * arithmetic fp32).  Each call is its fp32 counterpart on the widened inputs with the same plan, so
 *   dx = bf16( dx of the fp32 call on float(x), float(dy) ), rounded once at the store, and
 *   dg, ds1, ds2, dbias (and sq_partials) are bit-identical to the fp32 call's for float(x), float(dy).
 * The workspace is the fp32 call's: whvi_layer_bwd_workspace_bytes / whvi_layer_loss_sizes.
 * whvi_layer_bwd_bf16 is whvi_layer_bwd_scaled_f32 (dy_scale: device scalar, NULL = 1; flags: WHVI_LAYER_RELU_IN;
 * D = 4 ... 8192); the saved-output + target mode of whvi_layer_bwd_fused_f32 is fp32 only.
 * whvi_layer_loss_bf16 is whvi_layer_loss_f32 (128 <= D <= 4096; target fp32).
 * Alignment: fp32 pointers 16 bytes; x and dy 16 bytes (they are fetched by bulk async copies), dx 8 bytes.  The bulk copies
 * also need B * D % 8 == 0 (whole 16-byte units per sample); the only shape that breaks it, D = 4 with an odd B, is
 * rejected with WHVI_E_SHAPE -- a caller can pad B with a zero row of x and dy, which adds zero to every gradient.
 */
WHVI_API int whvi_layer_bwd_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* dy_scale, const float* g,
                                 const float* s1, const float* s2, void* dx, float* dg, float* ds1, float* ds2, float* dbias,
                                 void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int flags,
                                 whvi_stream_t stream);
WHVI_API int whvi_layer_loss_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                  const float* bias, const float* target, void* dx, float* dg, float* ds1, float* ds2, float* dbias,
                                  float* sq_partials, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                                  int flags, whvi_stream_t stream);

/*
 * Reparameterisation (src/weights.py:43-50, :82-83, :92-93), one eps row per MC sample:
 *   mode 0:  g[s,:] = mu + softplus(rho) * eps[s,:]              (diagonal; the reference)
 *   mode 1:  reserved -- the dense form g[s,:] = mu + L eps[s,:] is whvi_reparam_dense_f32 below (it needs a workspace).
 * eps, g: (S,D); mu, rho: (D).
 */
#define WHVI_REPARAM_DIAG 0
#define WHVI_REPARAM_DENSE 1
WHVI_API int whvi_reparam_f32(const float* mu, const float* rho, const float* eps, float* g, int64_t S, int64_t D,
                              int mode, whvi_stream_t stream);
/*
 * Dense-covariance superset of the reference's diagonal posterior (SURVEY F5; north-star kernel (4) as a tensor-core
 * GEMM, kernel (5) with the log-determinant).  L: (D, D) row-major lower triangular (entries above the diagonal are
 * ignored), D a multiple of 128.  All three products run on tcgen05 (kind::tf32, 3xTF32 operand split for fp32-level
 * accuracy, TMA-fed 128-byte-swizzled tiles, TMEM accumulators):
 *   whvi_reparam_dense_f32      g[s,:] = mu + L eps[s,:]            eps, g: (S, D); workspace from ..._workspace_bytes
 *   whvi_reparam_dense_bwd_f32  dL = tril( dgT epsT^T )             dgT, epsT: (D, S_padded) = the TRANSPOSES of dg and eps,
 *                               zero-padded to S_padded % 32 == 0; dL: (D, D), the caller zero-fills it (tiles above the
 *                               diagonal are not written); dmu = sum_s dg[s] is a column sum the caller does
 *   whvi_kl_dense_f32           KL( N(mu, L L^T) || N(0, lambda I) ) = 0.5 ( D ln lambda - 2 sum ln L_ii - D + |L|_F^2 / lambda
 *                               + |mu|^2 / lambda ) into out_kl[0]; dmu = grad_scale mu / lambda, dL = grad_scale ( L / lambda -
 *                               diag(1 / L_ii) ) (zero above the diagonal), both or neither; workspace: D doubles
 */
WHVI_API int whvi_reparam_dense_workspace_bytes(int64_t S, int64_t D, size_t* bytes);
WHVI_API int whvi_reparam_dense_f32(const float* mu, const float* L, const float* eps, float* g, int64_t S, int64_t D,
                                    void* workspace, size_t workspace_bytes, whvi_stream_t stream);
WHVI_API int whvi_reparam_dense_bwd_f32(const float* dgT, const float* epsT, float* dL, int64_t S_padded, int64_t D,
                                        whvi_stream_t stream);
WHVI_API int whvi_kl_dense_f32(const float* mu, const float* L, float lambda_, int64_t D, float* out_kl, float* dmu, float* dL,
                               float grad_scale, void* workspace, size_t workspace_bytes, whvi_stream_t stream);

/*
 * Grouped dense reparameterisation and KL: G blocks at once (the square blocks of a Stacked layer; G = 1 is a square or
 * Column layer), D <= 64 or a multiple of 128 (every power of two).  Block k's mu is read at + k * mu_stride floats and its L (D, D) at + k * L_stride
 * (strides >= D and D * D; multiples of 4 at D >= 128); entries of L above the diagonal are ignored.  eps, g, dg: (G, S, D);
 * dmu (G, D) and dL (G, D, D) are written densely, dL zero above the diagonal.
 *   D <= 64   one CUDA-core launch per direction for all blocks; L_k in shared memory; fixed-order fp32 sums (j ascending
 *             forward, s ascending backward): bit-reproducible.  No workspace.
 *   D >= 128  the tcgen05 kernels of whvi_reparam_dense_f32 / whvi_reparam_dense_bwd_f32, one launch (sequence) per block, so
 *             g and dL equal those calls' bit for bit; the backward writes the transposed, zero-padded GEMM operands into the
 *             workspace itself, and dmu is a device column sum (samples ascending).
 *   whvi_reparam_dense_grouped_workspace_bytes   bytes for either direction at (S, D) (0 below 128), reused block after block
 *   whvi_kl_dense_grouped_f32   sum over the blocks of the whvi_kl_dense_f32 term (fp64 accumulation, fixed order); dmu (G, D),
 *                               dL (G, D, D), both or neither; workspace: G * D doubles
 */
WHVI_API int whvi_reparam_dense_grouped_workspace_bytes(int64_t S, int64_t D, size_t* bytes);
WHVI_API int whvi_reparam_dense_grouped_f32(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, const float* eps, float* g,
                                            int64_t S, int64_t D, int64_t G, void* workspace, size_t workspace_bytes, whvi_stream_t stream);
WHVI_API int whvi_reparam_dense_grouped_bwd_f32(const float* eps, const float* dg, float* dmu, float* dL, int64_t S, int64_t D, int64_t G,
                                                void* workspace, size_t workspace_bytes, whvi_stream_t stream);
WHVI_API int whvi_kl_dense_grouped_f32(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, float lambda_, int64_t D,
                                       int64_t G, float* out_kl, float* dmu, float* dL, float grad_scale, void* workspace,
                                       size_t workspace_bytes, whvi_stream_t stream);

/*
 * WHVIStackedMatrix (src/weights.py:111-208) as ONE call per direction: the G = ceil(n_out / D) square blocks of a
 * non-square layer run as a second sample axis of the fused layer kernels instead of G launches + torch.cat (:179-180),
 * with the reparameterisation (:82-83), the bias add (:204-205), the ReLU that follows the layer, the concatenation and
 * the drop of the padded output columns (:207) inside the call.
 *   x      (B, D) [x_sample_stride = 0] or (S, B, D): the input, zero-padded to D = next_pow2(n_in) columns
 *          (whvi_pad_rows_f32 does src/weights.py:197-198)
 *   mu, rho, s1, s2: block k's (D) vectors at + k * param_stride floats (param_stride >= D, multiple of 4): the blocks'
 *          separate parameters are used where they lie when they are evenly spaced
 *   eps    (G, S, D) noise, block-major;  bias (G * D) or NULL;  g (G, S, D) out: the reparameterised vectors (kept for backward)
 *   y_blocks (G, S, B, D) scratch;  y (S, B, n_out) out, (G - 1) D < n_out <= G D
 * Backward: dy (S, B, n_out) -> dmu, drho, ds1, ds2 (G, D) each, dbias (G * D) or NULL, dx (S, B, n_in) or NULL (the sum over
 * the blocks, already un-padded; with a shared input the caller sums it over s).  Reductions are fixed-order.
 */
WHVI_API int whvi_pad_rows_f32(const float* in, float* out, int64_t rows, int64_t n_in, int64_t D, whvi_stream_t stream);
WHVI_API int whvi_stacked_fwd_f32(const float* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1,
                                  const float* s2, int64_t param_stride, const float* eps, const float* bias, float* g,
                                  float* y_blocks, float* y, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags,
                                  whvi_stream_t stream);
WHVI_API int whvi_stacked_bwd_workspace_bytes(int64_t S, int64_t B, int64_t D, int64_t G, int want_dx, size_t* bytes);
WHVI_API int whvi_stacked_bwd_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* rho,
                                  const float* s1, const float* s2, int64_t param_stride, const float* eps, float* dx, int64_t n_in,
                                  float* dmu, float* drho, float* ds1, float* ds2, float* dbias, void* workspace,
                                  size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags,
                                  whvi_stream_t stream);
/* The same layer from g (G, S, D) given, however it was drawn (e.g. whvi_reparam_dense_grouped_f32): the forward without the
 * reparameterisation, the backward returning dg (G, S, D) in place of dmu, drho (workspace from whvi_stacked_bwd_workspace_bytes).
 * whvi_stacked_fwd_f32 / whvi_stacked_bwd_f32 are the diagonal reparameterisation around these two. */
WHVI_API int whvi_stacked_fwd_g_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                    int64_t param_stride, const float* bias, float* y_blocks, float* y, int64_t S, int64_t B, int64_t D,
                                    int64_t G, int64_t n_out, int flags, whvi_stream_t stream);
WHVI_API int whvi_stacked_bwd_g_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* s1,
                                    const float* s2, int64_t param_stride, float* dx, int64_t n_in, float* dg, float* ds1, float* ds2,
                                    float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G,
                                    int64_t n_out, int flags, whvi_stream_t stream);
/*
 * bf16 activations for the Stacked layer: the same arguments with x, y_blocks, y, dy and dx bf16 (void*); g, the parameters,
 * their gradients, the workspace and all arithmetic stay fp32.  Each call is its fp32 twin on the widened inputs:
 *   forward   y = bf16(y of the fp32 call on float(x)), bit for bit;
 *   backward  dmu, drho (dg), ds1, ds2, dbias bit-identical to the fp32 call on float(x), float(dy); dx = bf16(dx_f32), rounded
 *             ONCE: the per-block dx are kept fp32, summed in the fp32 call's block order, then rounded.
 * whvi_pad_rows_bf16 is whvi_pad_rows_f32 on bf16 rows.  The workspace is the fp32 call's (whvi_stacked_bwd_workspace_bytes: the
 * bf16 dy blocks use the first half of its dy-block region).  Alignment: fp32 pointers as the fp32 twins; forward x and y_blocks
 * 8 bytes; backward x 16 bytes and B * D % 8 == 0 (the padded x and the block-layout dy reach the layer kernel by bulk copy, as
 * in whvi_layer_bwd_bf16; D = 4 with an odd B is rejected with WHVI_E_SHAPE, pad B with a zero row of x and dy); other bf16
 * pointers 2 bytes.
 */
WHVI_API int whvi_pad_rows_bf16(const void* in, void* out, int64_t rows, int64_t n_in, int64_t D, whvi_stream_t stream);
WHVI_API int whvi_stacked_fwd_bf16(const void* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1,
                                   const float* s2, int64_t param_stride, const float* eps, const float* bias, float* g,
                                   void* y_blocks, void* y, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags,
                                   whvi_stream_t stream);
WHVI_API int whvi_stacked_fwd_g_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                     int64_t param_stride, const float* bias, void* y_blocks, void* y, int64_t S, int64_t B, int64_t D,
                                     int64_t G, int64_t n_out, int flags, whvi_stream_t stream);
WHVI_API int whvi_stacked_bwd_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* g, const float* rho,
                                   const float* s1, const float* s2, int64_t param_stride, const float* eps, void* dx, int64_t n_in,
                                   float* dmu, float* drho, float* ds1, float* ds2, float* dbias, void* workspace,
                                   size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags,
                                   whvi_stream_t stream);
WHVI_API int whvi_stacked_bwd_g_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* g, const float* s1,
                                     const float* s2, int64_t param_stride, void* dx, int64_t n_in, float* dg, float* ds1, float* ds2,
                                     float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G,
                                     int64_t n_out, int flags, whvi_stream_t stream);
/* sum of the G blocks' KL terms (WHVIStackedMatrix.kl, src/weights.py:162-164) and their gradients (G, D), one launch */
WHVI_API int whvi_kl_grouped_f32(const float* mu, const float* rho, float lambda_, int64_t D, int64_t G, int64_t param_stride,
                                 int mode, float* out_kl, float* dmu, float* drho, float grad_scale, whvi_stream_t stream);

/*
 * WHVIColumnMatrix (src/weights.py:211-251), PAPER semantics, as ONE call per direction.  The reference samples the whole
 * D x D matrix and keeps the first n entries of its flattening (:239-245), i.e. of row 0:
 *     w[s, j] = s1[0] * s2[j] * (H g_s)[j], j < n,  g_s = mu + softplus(rho) * eps_s,  D = next_pow2(n) <= 32768
 *   transposed != 0  (n_in = n, n_out = 1):  x (B, n) or (S, B, n);  y[s, b]    = sum_j x[s, b, j] w[s, j] + bias[0]
 *   transposed == 0  (n_in = 1, n_out = n):  x (B, 1) or (S, B, 1);  y[s, b, j] = x[s, b] w[s, j] + bias[j]   (RELU_OUT allowed)
 * mu, rho, s1, s2: (D); eps: (S, D); g: (S, D) scratch; hg: (S, D) out = H g, kept for the backward.
 * Backward: dy as y; dx as x per sample (or NULL; RELU_IN masks it by x > 0, transposed form only); dmu, drho, ds1, ds2: (D);
 * dbias: (1) / (n) or NULL.  Fixed-order reductions.
 */
WHVI_API int whvi_column_fwd_f32(const float* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1,
                                 const float* s2, const float* eps, const float* bias, float* g, float* hg, float* y, int64_t S,
                                 int64_t B, int64_t D, int64_t n, int transposed, int flags, whvi_stream_t stream);
WHVI_API int whvi_column_bwd_workspace_bytes(int64_t S, int64_t D, int64_t n, size_t* bytes);
WHVI_API int whvi_column_bwd_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* hg, const float* rho,
                                 const float* s1, const float* s2, const float* eps, float* dx, float* dmu, float* drho, float* ds1,
                                 float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                                 int64_t n, int transposed, int flags, whvi_stream_t stream);
/* The same layer from g (S, D) given: the forward without the reparameterisation (g is read, hg = H g written), the backward
 * returning dg (S, D) in place of dmu, drho (workspace from whvi_column_bwd_workspace_bytes).  whvi_column_fwd_f32 /
 * whvi_column_bwd_f32 are the diagonal reparameterisation around these two. */
WHVI_API int whvi_column_fwd_g_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                   const float* bias, float* hg, float* y, int64_t S, int64_t B, int64_t D, int64_t n, int transposed,
                                   int flags, whvi_stream_t stream);
WHVI_API int whvi_column_bwd_g_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* hg, const float* s1,
                                   const float* s2, float* dx, float* dg, float* ds1, float* ds2, float* dbias, void* workspace,
                                   size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags,
                                   whvi_stream_t stream);
/*
 * bf16 activations for the Column layer: the same arguments with the activations bf16 (void*): x and dx always; y and dy in the
 * plain form (1 -> n) only.  The transposed form (n -> 1) keeps y (S, B, 1) and dy fp32: they are 1/n of the input's bytes, they
 * hold the predictions of a regression network, and rounding them to 8 significant bits would put that error straight into the
 * loss.  g, hg, the parameters, their gradients, the workspace (whvi_column_bwd_workspace_bytes) and all arithmetic stay fp32.
 * Each call is its fp32 twin on the widened inputs with the same reduction orders: the parameter gradients (and dg) are
 * bit-identical to the fp32 call's, and every bf16 output is the fp32 output rounded once.  bf16 pointers: 2-byte aligned.
 */
WHVI_API int whvi_column_fwd_bf16(const void* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1,
                                  const float* s2, const float* eps, const float* bias, float* g, float* hg, void* y, int64_t S,
                                  int64_t B, int64_t D, int64_t n, int transposed, int flags, whvi_stream_t stream);
WHVI_API int whvi_column_fwd_g_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                    const float* bias, float* hg, void* y, int64_t S, int64_t B, int64_t D, int64_t n, int transposed,
                                    int flags, whvi_stream_t stream);
WHVI_API int whvi_column_bwd_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* hg, const float* rho,
                                  const float* s1, const float* s2, const float* eps, void* dx, float* dmu, float* drho, float* ds1,
                                  float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                                  int64_t n, int transposed, int flags, whvi_stream_t stream);
WHVI_API int whvi_column_bwd_g_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* hg, const float* s1,
                                    const float* s2, void* dx, float* dg, float* ds1, float* ds2, float* dbias, void* workspace,
                                    size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags,
                                    whvi_stream_t stream);

/* dmu = sum_s dg[s];  drho = (sum_s dg[s]*eps[s]) * sigmoid(rho).  accumulate != 0: += */
WHVI_API int whvi_reparam_bwd_f32(const float* rho, const float* eps, const float* dg, float* dmu, float* drho,
                                  int64_t S, int64_t D, int mode, int accumulate, whvi_stream_t stream);

/*
 * Gaussian KL of N(mu, diag) against N(0, lambda I) with sigma = softplus(rho), value and
 * gradient in one pass (src/weights.py:52-64 -> src/utils.py:49-71):
 *   mode 0 (reference, sigma used as a variance):
 *        0.5*( D ln(lambda) - sum ln(sigma) - D + sum sigma/lambda + sum mu^2/lambda )
 *   mode 1 (statistically consistent): sigma -> sigma^2 in the log and ratio terms.
 * out_kl: device float[1].  dmu/drho: (D) or both NULL; they receive grad_scale * dKL/d.
 * (accumulate != 0: added to the existing contents).
 */
/*
 * MC predictive moments (SURVEY 8f N1; the reduction WHVIRegression.eval_model does over the
 * sample axis of WHVINetwork.forward's (B, out, S) output, src/networks.py:36-54, :131-132):
 *   sum_y[i] (+)= sum_s y[s*n + i],  sum_y2[i] (+)= sum_s y[s*n + i]^2,   i < n (= B*D), n % 4 == 0.
 * accumulate != 0 adds to the existing contents (sample chunks); s ascending, so results are
 * bit-reproducible.  sum_y2 may be NULL.
 */
WHVI_API int whvi_mc_moments_f32(const float* y, float* sum_y, float* sum_y2, int64_t S, int64_t n, int accumulate,
                                 whvi_stream_t stream);
/*
 * The same two sums WITHOUT the (S, B, D) predictions ever existing (8192 <= D <= 32768; BASELINE config 5): the layer
 * forward over all S samples of the call with the reduction fused in -- one CTA per input row loops over the samples
 * and keeps sum_s t4 and sum_s t4^2 (t4 = H(g_s * t2)) in tensor memory; s1 and bias are applied once per row in
 * closed form.  HBM traffic: each input row once, 8*D bytes of sums per row.
 *   x: (B, D) shared by all samples (x_sample_stride = 0) or (S, B, D) (x_sample_stride = B*D);
 *   flags & WHVI_LAYER_FROM_T2: x holds t2 = H(s2 * x) already (shared input only; sample-independent by linearity,
 *       one whvi_fwht_f32 per input chunk), so one transform per (sample, row) pair is left;
 *   flags & WHVI_LAYER_ACCUMULATE: sum_y / sum_y2 are added to (sample chunks, or per-rank partial sums).
 *   flags | WHVI_LAYER_RESERVE_SMS(n): the persistent grid leaves n SMs unoccupied -- its CTAs take whole SMs (all
 *       registers or all shared memory), so a collective kernel launched next to it (multi-GPU evaluation: the exchange of
 *       partial sums overlaps the next chunk) would otherwise wait for it to finish.
 * sum_y2 may be NULL; bias may be NULL; g: (S, D).
 */
WHVI_API int whvi_layer_moments_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                    const float* bias, float* sum_y, float* sum_y2, int64_t S, int64_t B, int64_t D,
                                    int flags, whvi_stream_t stream);
/* The same with a starting value: sum_y = in_sum_y + sum_s y, sum_y2 = in_sum_y2 + sum_s y^2 (either may be NULL = 0).  The
 * multi-GPU evaluation uses it for the exchange inside a sample-group pair without a collective kernel: a rank runs the
 * rows its PARTNER owns first, with sum_y / sum_y2 pointing into the partner's (NVLink-mapped) staging buffer -- the partial
 * sums travel as the kernel's own stores -- and then its own rows with in_sum_y / in_sum_y2 = what the partner stored. */
WHVI_API int whvi_layer_moments_add_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                                        const float* bias, const float* in_sum_y, const float* in_sum_y2, float* sum_y,
                                        float* sum_y2, int64_t S, int64_t B, int64_t D, int flags, whvi_stream_t stream);
/*
 * The same reduction with separate inputs and outputs and a sample stride (so `y` may be a block of
 * rows of a larger (S, B, D) tensor):  out_sum_y[i] = in_sum_y[i] + sum_s y[s*y_sample_stride + i]
 * (likewise y^2); in_* may be NULL (zero), out_sum_y2 may be NULL.  The outputs may point into a PEER
 * GPU's memory mapped over NVLink (one process per GPU, MC samples sharded over the ranks,
 * SURVEY 8e): the kernel then reduces this rank's samples and delivers the partial sums to the rank
 * that owns those rows in one pass -- the evaluation path's reduce-scatter fused into its producer.
 */
WHVI_API int whvi_mc_moments_strided_f32(const float* y, int64_t y_sample_stride, const float* in_sum_y,
                                         const float* in_sum_y2, float* out_sum_y, float* out_sum_y2, int64_t S,
                                         int64_t n, whvi_stream_t stream);

/*
 * Categorical (softmax) likelihood of a classifier (not in the reference, whose networks only regress).  logits: (S, B, K)
 * sample-major rows r = s * B + b, fp32 or bf16 (the _bf16 calls: the fp32 calls on the widened logits, same plan and order, so
 * bit-identical; a bf16 dz is the fp32 dz rounded once).  labels: (B) int64, shared by the samples.  2 <= K <= 65536, any K.
 *   whvi_categorical_sizes       bytes of workspace whvi_categorical_nll_* needs for R = S * B rows of K classes
 *   whvi_categorical_nll_*       lse[r] = log sum_k exp(z[r, k]) (max-subtracted; lse may be NULL) and
 *                                total[0] = sum_r (lse[r] - z[r, y_b]): fp64 per-CTA partials in the workspace, summed in a fixed
 *                                order.  The caller applies the estimator's coefficient n / (m S).
 *   whvi_categorical_nll_bwd_*   dz[r, k] = c[0] (exp(z[r, k] - lse[r]) - [k = y_b]), c a device scalar (NULL = 1), lse the forward's
 *   whvi_categorical_predictive_*  prob_sum[b, k] (+)= sum_s softmax(z[s, b])[k] and, with labels, loglik_sum[b] (+)=
 *                                sum_s log softmax(z[s, b])[y_b]; (B, K) and (B) fp32, s ascending.  Sample s's rows are read at
 *                                logits + s * sample_stride (>= B * K, so a sample chunk may be a slice of a larger tensor);
 *                                flags & WHVI_CATEGORICAL_ACCUMULATE adds to the existing sums in the order one call over all
 *                                samples would (chunks give that call's bits).  labels and loglik_sum both or neither.
 * A label outside [0, K) is never used as an index: that row's loss (so the total), its log p and its dz row are NaN.
 * Every reduction has a fixed order: repeated calls are bit-identical.  Alignment: the element size of each pointer's type
 * (rows need no more: the loads are element-wise); workspace 8 bytes.
 */
#define WHVI_CATEGORICAL_ACCUMULATE 1
WHVI_API int whvi_categorical_sizes(int64_t R, int64_t K, size_t* workspace_bytes);
WHVI_API int whvi_categorical_nll_f32(const float* logits, const int64_t* labels, float* lse, float* total, void* workspace,
                                      size_t workspace_bytes, int64_t S, int64_t B, int64_t K, whvi_stream_t stream);
WHVI_API int whvi_categorical_nll_bf16(const void* logits, const int64_t* labels, float* lse, float* total, void* workspace,
                                       size_t workspace_bytes, int64_t S, int64_t B, int64_t K, whvi_stream_t stream);
WHVI_API int whvi_categorical_nll_bwd_f32(const float* logits, const int64_t* labels, const float* lse, const float* c, float* dz,
                                          int64_t S, int64_t B, int64_t K, whvi_stream_t stream);
WHVI_API int whvi_categorical_nll_bwd_bf16(const void* logits, const int64_t* labels, const float* lse, const float* c, void* dz,
                                           int64_t S, int64_t B, int64_t K, whvi_stream_t stream);
WHVI_API int whvi_categorical_predictive_f32(const float* logits, int64_t sample_stride, const int64_t* labels, float* prob_sum,
                                             float* loglik_sum, int64_t S, int64_t B, int64_t K, int flags, whvi_stream_t stream);
WHVI_API int whvi_categorical_predictive_bf16(const void* logits, int64_t sample_stride, const int64_t* labels, float* prob_sum,
                                              float* loglik_sum, int64_t S, int64_t B, int64_t K, int flags, whvi_stream_t stream);

/*
 * Patch gather and scatter of a convolutional WHVI layer (WHVIConv2d; not in the reference).  Activations are channels-last:
 * x and dx are (S|1, B, H, W, C), the patch matrix is (S|1, B * Ho * Wo, ld) with its rows in (b, oh, ow) order, i.e. the rows a
 * layer call takes.  Column order: tap (i, j) and channel c go to column (i * kw + j) * C + c (channels fastest), so a WHVI
 * weight W (C_out, C * kh * kw) is the torch filter W.reshape(C_out, kh, kw, C).permute(0, 3, 1, 2).
 *   Ho = (H + 2 pad_h - dil_h (kh - 1) - 1) / stride_h + 1, Wo likewise (floor); Ho <= 0 or Wo <= 0 is WHVI_E_SHAPE.
 *   whvi_im2col_*   patches[s, (b, oh, ow), (i kw + j) C + c] = x[s, b, oh stride_h - pad_h + i dil_h, ow stride_w - pad_w + j dil_w, c]
 *                   and 0 for taps outside the image and for the columns n_in ... ld - 1 (n_in = C kh kw <= ld, else
 *                   WHVI_E_SHAPE): every element of the (S, B Ho Wo, ld) output is written, so ld = D of a Stacked or square
 *                   layer gives that call's padded input directly.  x_sample_stride: 0 (one (B, H, W, C) image batch for all S
 *                   samples; patches are still written per sample) or B H W C.  A copy: the bf16 call moves the same bits.
 *   whvi_col2im_*   the adjoint: dx[s, b, h, w, c] = sum of the dpatches elements that im2col took from x[s, b, h, w, c], taps
 *                   i ascending then j ascending, fp32 accumulation (a bf16 dx is rounded once).  No atomics: bit-reproducible.
 *                   flags & WHVI_COL2IM_SUM_SAMPLES: dx is ONE (B, H, W, C) block, the per-sample sums added over s ascending
 *                   (the gradient of an input shared by the samples; S = 0 writes zeros); otherwise dx is (S, B, H, W, C).
 * Limits: H, W, C, kernel, stride, dilation in [1, 2^24), padding in [0, 2^24), dil (k - 1) + 1 < 2^24, C kh kw and ld below
 * 2^31, elements below 2^62 (int64 indexing: rows may exceed 65535 and elements 2^31).  Alignment: the element size of each
 * pointer's type; 16-byte aligned pointers with C and ld multiples of 4 (fp32) or 8 (bf16) take 16-byte moves.
 */
#define WHVI_COL2IM_SUM_SAMPLES 1
WHVI_API int whvi_im2col_f32(const float* x, int64_t x_sample_stride, float* patches, int64_t S, int64_t B, int64_t H, int64_t W,
                             int64_t C, int64_t kh, int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w,
                             int64_t dil_h, int64_t dil_w, int64_t ld, whvi_stream_t stream);
WHVI_API int whvi_im2col_bf16(const void* x, int64_t x_sample_stride, void* patches, int64_t S, int64_t B, int64_t H, int64_t W,
                              int64_t C, int64_t kh, int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w,
                              int64_t dil_h, int64_t dil_w, int64_t ld, whvi_stream_t stream);
WHVI_API int whvi_col2im_f32(const float* dpatches, int64_t ld, float* dx, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C,
                             int64_t kh, int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w, int64_t dil_h,
                             int64_t dil_w, int flags, whvi_stream_t stream);
WHVI_API int whvi_col2im_bf16(const void* dpatches, int64_t ld, void* dx, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C,
                              int64_t kh, int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w, int64_t dil_h,
                              int64_t dil_w, int flags, whvi_stream_t stream);

/*
 * One Adam step over a flat fp32 parameter buffer (the optimizer.step() of the reference's training loop,
 * src/networks.py:80-82, :92-94, which the reference runs as torch.optim.Adam: src/evaluation.py:15-27), in
 * torch.optim.Adam's arithmetic (weight_decay = 0, amsgrad = False):
 *   m += (1-beta1)(g-m);  v = beta2 v + (1-beta2) g^2;  p -= lr/(1-beta1^t) * m / (sqrt(v)/sqrt(1-beta2^t) + eps)
 * with g = grad_scale * grad.  step_dev: device float[1] holding t >= 1 (the caller increments it before the
 * call); lr_dev: device float[1] or NULL (then `lr` is used) -- device-resident so that a captured CUDA graph
 * follows learning-rate schedules and step counts.  All four buffers have n elements; in place.
 */
WHVI_API int whvi_adam_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                           const float* lr_dev, const float* step_dev, float beta1, float beta2, float eps,
                           float grad_scale, whvi_stream_t stream);

#define WHVI_KL_REFERENCE 0
#define WHVI_KL_CONSISTENT 1
WHVI_API int whvi_kl_f32(const float* mu, const float* rho, float lambda_, int64_t D, int mode, float* out_kl,
                         float* dmu, float* drho, float grad_scale, int accumulate, whvi_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* WHVI_B200_H */
