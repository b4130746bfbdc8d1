/*
 * psld_b200.h — C ABI of libpsld_b200.so: hand-written sm_100a CUDA kernels for the
 * reverse-time sampling hot path of PSLD (mandt-lab/PSLD).
 *
 * Boundary being replaced (reference file:line, relative to the reference repo):
 *   - the only native boundary the reference has is a pybind11 torch extension that is
 *     JIT-compiled at import: `Tensor upfirdn2d(const Tensor& input, const Tensor& kernel,
 *     int up_x, up_y, down_x, down_y, pad_x0, pad_x1, pad_y0, pad_y1)`
 *     (main/models/score_fn/song_sde/op/upfirdn2d.cpp:12-23, kernel in
 *     op/upfirdn2d_kernel.cu:107-369)  ->  psld_upfirdn2d / PSLD_OP_FIR below;
 *   - everything else on the path is PyTorch-eager code that this library replaces
 *     kernel by kernel; each entry point cites the reference lines it computes.
 *
 * Conventions (SURVEY.md §8b): plain `extern "C"`, no torch/C++ types in signatures.
 * Every function returns 0 on success or a negative PSLD_E* code and never throws;
 * psld_last_error() returns a thread-local message for the last failure.  All data
 * pointers are DEVICE pointers owned by the caller unless a parameter says "host".
 * Every launch goes to the explicit `stream` (a cudaStream_t passed as void*).  The
 * library allocates no device memory; scratch buffers are passed in by the caller.
 */
#ifndef PSLD_B200_H_
#define PSLD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSLD_B200_VERSION 100

/* error codes */
#define PSLD_OK 0
#define PSLD_EINVAL (-1)      /* bad argument / unsupported shape             */
#define PSLD_ECUDA (-2)       /* CUDA runtime / driver error                  */
#define PSLD_EUNSUPPORTED (-3)/* op not eligible for the requested engine     */
#define PSLD_ENUMERIC (-4)    /* NaN in the 2x2 factorisation (psld.py:171)   */

/* element types */
#define PSLD_F32 0
#define PSLD_BF16 1
#define PSLD_F64 2
/* "split bf16": every value is stored as hi + lo, two bf16 numbers (hi = rn_bf16(x), lo =
 * rn_bf16(x - hi): 16 significand bits, fp32 range).  NHWC activations keep both halves in the
 * pixel row: [C hi | C lo] (row stride 2C bf16 = 4C bytes, lo at +C); weights as two planes
 * [2][Cout, K].  It is the operand format of the fp32-tolerance tensor-core tier ("bf16x3":
 * a*w ~= a_hi*w_hi + a_hi*w_lo + a_lo*w_hi, three bf16 tcgen05 MMAs into one fp32 accumulator) */
#define PSLD_BF16S 3

/* tensor layouts */
#define PSLD_NHWC 0
#define PSLD_NCHW 1

typedef void* psld_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define PSLD_API __attribute__((visibility("default")))
#else
#define PSLD_API
#endif

PSLD_API int psld_version(void);
PSLD_API const char* psld_last_error(void);
/* sm count / compute capability of the current device */
PSLD_API int psld_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------
 * 1. Fused phase-space update (SSCS / Euler-Maruyama / denoise)
 *
 * State u = [x; m], NCHW [B, 2C, H, W]; one "pair" = (x[b,j], m[b,j]), j in [0, C*H*W).
 * Coefficients are identical for every batch element (SURVEY.md Appendix A) and are
 * computed once on the host in float64 (psld_b200/schedule.py).
 * ---------------------------------------------------------------------------------- */

/* u' = A u + L z   — SSCSSampler.analytical_dynamics (main/samplers/sde.py:294-312):
 * A from _mean (sde.py:236-263), L = get_coeff(_var) (sde.py:265-292, psld.py:154-186) */
typedef struct {
  double a_xx, a_xm, a_mx, a_mm; /* x' = a_xx x + a_xm m ;  m' = a_mx x + a_mm m      */
  double c11, c12, c21, c22;     /* x' += c11 zx + c12 zm ; m' += c21 zx + c22 zm     */
} psld_half_step;

/* score = -L^{-T} eps with L^{-T} rounded to fp32 (main/models/sde/psld.py:230-260);
 * SSCS:  x += k_x (s_x + x) ; m += k_m (s_m + m_inv m)     (sde.py:314-329)
 * EM  :  u += fbar dt + g sqrt(dt) z,  fbar = -f + g^2 score (psld.py:330-364, sde.py:16-26)
 * mode: 0 = score_xm (eps has 2C channels), 1 = score_m (eps has C channels, s_x = 0),
 *       2 = score_x  (eps has C channels, s_m = 0)                                     */
typedef struct {
  float li11, li12, li21, li22;  /* L^{-T} entries, already rounded to fp32             */
  int32_t mode;
  int32_t _pad;
  double k_x;      /* SSCS: dt*gamma*beta(tau)          EM: unused                      */
  double k_m;      /* SSCS: dt*M*nu*beta(tau)           EM: unused                      */
  double m_inv;
  /* EM / denoise (reverse_sde): */
  double half_beta, gamma, nu;   /* f_x = hb (m_inv m - gamma x); f_m = hb (-nu m - x) */
  double g2_x, g2_m;             /* g_x^2, g_m^2                                        */
  double dt;                     /* EM: dt ; denoise: eps                               */
  double gs_x, gs_m;             /* g_x sqrt(dt), g_m sqrt(dt)  (0 for denoise)         */
} psld_score_step;

/* stage bits for psld_sscs_update */
#define PSLD_STAGE_HALF_A 1 /* u <- A_a u + L_a z_a            (first half of a step) */
#define PSLD_STAGE_SCORE 2  /* Euler score step with eps                              */
#define PSLD_STAGE_HALF_B 4 /* second half of the step                                */
#define PSLD_STAGE_HALF_C 8 /* first half of the NEXT step, fused into the same pass  */

typedef struct {
  psld_half_step half_a, half_b, half_c;
  psld_score_step score;
} psld_sscs_coeffs;

/*
 * One pass over HBM applying the selected stages in order A -> SCORE -> B -> C.
 *   u_in / u_out : state, `state_dtype` PSLD_F64 (reference-faithful) or PSLD_F32; may alias.
 *   net_in       : optional fp32 copy of u_out (the next score_fn input, sde.py:320), or NULL.
 *   eps          : fp32 NCHW network output [B, 2C or C, H, W]; required with STAGE_SCORE.
 *   z_a/z_b/z_c  : pre-drawn fp32 N(0,1) noise [B,2C,H,W] per stage (parity mode).  When a
 *                  needed pointer is NULL the kernel draws from Philox4x32-10 keyed by
 *                  (seed, stream id = stage slot of `step`, pair index)  (throughput mode).
 *   B, chw       : batch and C*H*W (pairs per sample); chw % 4 == 0.
 * Algorithmic HBM bytes per pair (fp32 state): 8 (u in) + 8 (u out) + 8 (eps) + 8 per
 * pre-drawn noise tensor [+ 8 net_in]; Philox mode drops the noise reads.
 */
PSLD_API int psld_sscs_update(void* u_out, const void* u_in, int state_dtype, float* net_in,
                     const float* eps, const float* z_a, const float* z_b, const float* z_c,
                     const psld_sscs_coeffs* coeffs /* host */, int stages,
                     uint64_t seed, uint64_t step, int64_t B, int64_t chw,
                     psld_stream_t stream);

/* EulerMaruyamaSampler.predictor_update_fn (sde.py:16-26) and both samplers'
 * denoising_fn (sde.py:28-36, 338-348; pass z = NULL and use_philox = 0, gs_* = 0). */
PSLD_API int psld_em_update(void* u_out, const void* u_in, int state_dtype, float* net_in,
                   const float* eps, const float* z, int use_philox,
                   const psld_score_step* coeffs /* host */, uint64_t seed, uint64_t step,
                   int64_t B, int64_t chw, psld_stream_t stream);

/* Classifier-guided Euler-Maruyama step, ClassCondEulerMaruyamaSampler.predictor_update_fn
 * (main/samplers/sde.py:73-100): fbar = -f + g^2 score + g^2 (guide * guide_scale), where guide is
 * d/du log p(y | u, t) as fp32 [B,2C,H,W] (the caller's classifier gradient) and guide_scale the
 * classifier temperature clf_temp; guide = NULL is psld_em_update.  z = NULL and use_philox = 0
 * gives the guided mean x + fbar dt the reference uses for its denoising call (sde.py:112-117). */
PSLD_API int psld_em_update_guided(void* u_out, const void* u_in, int state_dtype, float* net_in,
                          const float* eps, const float* guide, double guide_scale, const float* z,
                          int use_philox, const psld_score_step* coeffs /* host */, uint64_t seed,
                          uint64_t step, int64_t B, int64_t chw, psld_stream_t stream);

/* One Split-Perturb-Combine step of the inpainting sampler ES3EulerMaruyamaInpainter
 * (main/samplers/sde.py:134-186; perturbation kernel PSLD._mean / cond_marginal_prob /
 * perturb_data, main/models/sde/psld.py:62-84,222-228,262-287), fused into one pass:
 *   m0   = m0_std * z_m0                      (DSM; HSM passes m0_std = 0, sde.py:137-143)
 *   mu_x = a_xx x0 + a_xm m0 ;  mu_m = a_mx x0 + a_mm m0
 *   x_k  = mu_x + c11 e_x + c12 e_m ;  m_k = mu_m + c21 e_x + c22 e_m   (mean_only: x_k = mu_x, ...)
 *   x    = x (1 - mask) + x_k mask ;  m = m (1 - mask) + m_k mask        (sde.py:175-178)
 * u: [B,2C,H,W] state (in place, f64 or f32); x0, mask: fp32 [B,C,H,W]; z_m0 [B,C,H,W] and
 * z_eps [B,2C,H,W] are pre-drawn N(0,1) tensors or NULL (both NULL: Philox4x32-10 keyed by
 * (seed, step)); net_in (optional): fp32 copy of the new state for the next score_fn call. */
typedef struct psld_inpaint_step {
  double a_xx, a_xm, a_mx, a_mm;
  double c11, c12, c21, c22;
  double m0_std;
  int32_t mean_only;
  int32_t _pad;
} psld_inpaint_step;

PSLD_API int psld_inpaint_combine(void* u, int state_dtype, float* net_in, const float* x0,
                                  const float* mask, const float* z_m0, const float* z_eps,
                                  const psld_inpaint_step* coeffs /* host */, uint64_t seed,
                                  uint64_t step, int64_t B, int64_t chw, psld_stream_t stream);

/* Euler-Maruyama step of the VP-SDE baseline (reference main/models/sde/vpsde.py:42-74 under
 * EulerMaruyamaSampler, main/samplers/sde.py:16-36):
 *   score = eps * neg_inv_std ;  x' = x + (half_beta x + g2 score) dt + gs z
 * x: [n] elements (f64 or f32, may be updated in place), eps fp32, z pre-drawn N(0,1) or NULL
 * (use_philox: in-kernel Philox; neither: no noise = the denoising step), net_in (optional): fp32
 * copy of x'.  n must be a multiple of 4. */
typedef struct psld_vp_step {
  double half_beta, g2, neg_inv_std, dt, gs;
} psld_vp_step;

PSLD_API int psld_vp_em_update(void* x_out, const void* x_in, int state_dtype, float* net_in,
                               const float* eps, const float* z, int use_philox,
                               const psld_vp_step* coeffs /* host */, uint64_t seed, uint64_t step,
                               int64_t n, psld_stream_t stream);

/* ------------------------------------------------------------------------------------
 * 1b. Probability-flow ODE sampler BBODESampler (main/samplers/ode.py:41-76): the reference hands
 * ode_fn = reverse_sde(..., probability_flow=True) (psld.py:345-364) to torchdiffeq==0.2.3
 * odeint(method="scipy_solver") = scipy.integrate.solve_ivp(RK45) (Dormand-Prince 5(4) with scipy's
 * step-size control), which is absent from the reference tree; psld_b200/ode.py restates that driver
 * on the host and runs every vector operation on the device through these three kernels.
 * ---------------------------------------------------------------------------------- */
/* fbar = -f + g^2 (score_scale * score), float64 out [B,2C,H,W]; u in state_dtype (f64 | f32). */
PSLD_API int psld_reverse_drift(double* out, const void* u, int state_dtype, const float* eps,
                                const psld_score_step* coeffs /* host */, double score_scale,
                                int64_t B, int64_t chw, psld_stream_t stream);
/* The same drift for the VP-SDE baseline (vpsde.py:42-67; scripts_psld/ablations/uncond/cifar10/
 * sample_uncond_vpsde_ode.sh): fbar = 0.5 beta x + g^2 score_scale (eps * neg_inv_std), x: [n] elements
 * (n % 4 == 0) in state_dtype, coefficients = the psld_vp_step of this time (dt, gs unused). */
PSLD_API int psld_vp_reverse_drift(double* out, const void* x, int state_dtype, const float* eps,
                                   const psld_vp_step* coeffs /* host */, double score_scale, int64_t n,
                                   psld_stream_t stream);
/* out = y + h * sum_{j < terms} coef[j] K[j]; K = [terms, n] float64, coef on the HOST (terms <= 8);
 * out32 (optional) receives the float32 rounding of the same values (the float32-batch view of the
 * state = the next network input); out may be NULL when only out32 is wanted. */
PSLD_API int psld_rk_combine(double* out, float* out32, const double* y, const double* K,
                             const double* coef /* host */, int terms, double h, int64_t n,
                             psld_stream_t stream);
/* *sum_out += sum_i ((h sum_j e[j] K[j][i]) / (atol + max(|y_i|, |y_new_i|) rtol))^2  (the RK error
 * norm of scipy's RungeKutta._estimate_error_norm is sqrt(sum / n)); sum_out zeroed by the caller. */
PSLD_API int psld_rk_error(const double* y, const double* y_new, const double* K,
                           const double* e /* host */, int terms, double h, double atol, double rtol,
                           int64_t n, double* sum_out, psld_stream_t stream);

/* PSLD.prior_sampling (psld.py:366-370) on device: x ~ N(0,1), m ~ N(0, M); fp32 NCHW. */
PSLD_API int psld_prior_sample(float* u, double m_std, uint64_t seed, int64_t B, int64_t chw,
                      psld_stream_t stream);

/* Caller-side epilogue of sampling, fused (SimpleImageWriter.write_on_batch_end,
 * main/callbacks.py:103-107 + save_as_images, main/util.py:147-158): drop the momentum half,
 * x*0.5+0.5, *255, clip, truncate to uint8; state NCHW [B,2C,H,W] -> images NHWC [B,H,W,C]. */
PSLD_API int psld_quantize_images(const void* state, int state_dtype, uint8_t* out_nhwc, int64_t B,
                                  int C, int HW, psld_stream_t stream);

/* ------------------------------------------------------------------------------------
 * 2. NCSN++ score network ops.  Activations are NHWC inside the network, element type
 *    PSLD_F32 (reference-faithful path) or PSLD_BF16 (tensor-core path).
 *    A network forward is a "program": a flat array of psld_op records built once by the
 *    host (psld_b200/ncsnpp.py) and replayed by psld_program_run.
 * ---------------------------------------------------------------------------------- */
#define PSLD_OP_LAYOUT 1 /* NCHW f32 <-> NHWC T                                        */
#define PSLD_OP_TEMB 2   /* Fourier/positional embedding + MLP + all Dense_0 projections */
#define PSLD_OP_GN 3     /* GroupNorm (+SiLU) over a virtual channel-concat of 2 inputs  */
#define PSLD_OP_FIR 4    /* upfirdn2d                                                   */
#define PSLD_OP_CONV 5   /* conv3x3 / conv1x1 / NIN / strided conv as implicit GEMM     */
#define PSLD_OP_ATTN 6   /* softmax(q k^T / sqrt(C)) v                                  */
#define PSLD_OP_ZERO 7   /* out[0] = buffer, i[0] | i[1] << 31 = bytes: cudaMemsetAsync(0).  Clears
                            the GroupNorm statistics accumulators at the top of a program   */
#define PSLD_OP_AXPBY 8  /* out[0] = f[0] * in[0] + f[1] * in[1] over i[0] | i[1] << 31 floats (in[1] may be
                            NULL: out = f[0] * in[0]).  Classifier-free guidance: a guided program is
                            [cond program | copy net_in | uncond program | eps = (1+w) eps_c - w eps_u]  */

#define PSLD_ENGINE_SIMT 0 /* fp32 FFMA implicit GEMM (any shape)                       */
#define PSLD_ENGINE_TC 1   /* tcgen05.mma + TMEM + TMA implicit GEMM (bf16, Cin%64==0;
                              stride 1 'same' padding, or 3x3 stride 2 without padding)     */

#define PSLD_ENGINE_TC_GN 2 /* PSLD_OP_CONV only: tensor-core 3x3 conv with GroupNorm(+SiLU) applied
                              to the input inside the kernel (in[6] = per-(n,channel) affine)  */

#define PSLD_OP_NI 28
#define PSLD_OP_NF 24
#define PSLD_OP_NP 10

/* Generic op record.  Slot meaning per kind is documented next to each PSLD_*_ index
 * enum below; unused slots must be zero.                                              */
typedef struct {
  int32_t kind;
  int32_t engine;
  int32_t i[PSLD_OP_NI];
  float f[PSLD_OP_NF];
  const void* in[PSLD_OP_NP];
  void* out[PSLD_OP_NP];
  void* aux; /* library-owned per-op host state (TMA descriptors); set by psld_op_prepare */
} psld_op;

/* --- PSLD_OP_LAYOUT: in[0] -> out[0].  i: N, C, HW, dir (0: NCHW f32 -> NHWC T, 1: NHWC T
 *     -> NCHW f32), dtype (T), CPAD (dir 0 only: NHWC channel count >= C, zero padded; 0 = C),
 *     CWRITE (dir 0 only: channels [0, CWRITE) are written, C <= CWRITE <= CPAD; 0 = CPAD: the
 *     caller zeroed the remaining padding channels once)                                   */
enum { PSLD_LAYOUT_N = 0, PSLD_LAYOUT_C, PSLD_LAYOUT_HW, PSLD_LAYOUT_DIR, PSLD_LAYOUT_DTYPE,
       PSLD_LAYOUT_CPAD, PSLD_LAYOUT_CWRITE };

/* --- PSLD_OP_TEMB (ncsnpp.py:292-311, layerspp.py:32-41,262-263, layers.py:500-514):
 *   in[0] = time [nt] f32 (forward time tau, or log(tau) when i[LOGGED]=1)
 *   in[1] = Fourier W [nf] ; in[2],in[3] = Linear0 W [4nf, E], b ; in[4],in[5] = Linear1 W,b
 *   in[6],in[7] = concatenated Dense_0 W [totalC, 4nf], b [totalC]
 *   out[0] = proj [nt, totalC] f32 (Dense_0(SiLU(temb)) of every resblock)
 *   out[1] = scratch f32 [nt, E + 8nf]
 *   out[2] = optional device int32 step counter: the time row used is in[0][*out[2] + r]
 *            (lets a captured CUDA graph of one sampler step be replayed for every step)
 *   i: NT, NF, EMB (0 fourier, 1 positional), TOTALC, LOGGED                           */
enum { PSLD_TEMB_NT = 0, PSLD_TEMB_NF, PSLD_TEMB_EMB, PSLD_TEMB_TOTALC, PSLD_TEMB_LOGGED };

/* --- PSLD_OP_GN (nn.GroupNorm(min(C/4,32), C, eps=1e-6) [+ SiLU]; layerspp.py:219,231,67):
 *   in[0] = x1 [N,HW,C1], in[1] = x2 [N,HW,C2] or NULL (virtual torch.cat([x1,x2],1),
 *   ncsnpp.py:374), in[2] = gamma [C], in[3] = beta [C];  out[0] = y [N,HW,C1+C2],
 *   out[1] = scratch, >= N*NCHUNK*G*2 doubles
 *   in[4], in[5] = optional producer-side statistics of x1 / x2: f64 [N, C/4, 2] holding
 *   (sum, sum of squares) per sample x 4 channels, accumulated by the PSLD_OP_CONV that produced
 *   the tensor (its out[1]).  When every source has them there is no statistics pass at all:
 *   the apply (or affine) kernel sums the C/G/4 entries of each group itself.
 *   i: N, HW, C1, C2, G, SILU, IN_DTYPE, OUT_DTYPE, NCHUNK, AFFINE_ONLY ; f[0] = eps
 *   AFFINE_ONLY = 1: no apply pass; out[0] receives fp32 [N, C, 2] = (rstd*gamma,
 *   beta - mean*rstd*gamma) for a PSLD_ENGINE_TC_GN convolution to apply on load.            */
enum { PSLD_GN_N = 0, PSLD_GN_HW, PSLD_GN_C1, PSLD_GN_C2, PSLD_GN_G, PSLD_GN_SILU,
       PSLD_GN_IN_DTYPE, PSLD_GN_OUT_DTYPE, PSLD_GN_NCHUNK, PSLD_GN_AFFINE_ONLY };

/* --- PSLD_OP_FIR (upfirdn2d, op/upfirdn2d.py:159-200; callers up_or_down_sampling.py:195-257):
 *   in[0] = x [N,H,W,C] ; out[0] = y [N,OH,OW,C]
 *   i: N, H, W, C, UP, DOWN, PAD0, PAD1, KH (== KW <= 4), DTYPE, CACT ; f[0..KH*KW) = taps (unflipped)
 *   CACT > 0: only channels [0, CACT) are filtered and written (C and CACT multiples of 8): for the
 *   channel-padded network input, whose padding channels stay at the zeros they were allocated with */
enum { PSLD_FIR_N = 0, PSLD_FIR_H, PSLD_FIR_W, PSLD_FIR_C, PSLD_FIR_UP, PSLD_FIR_DOWN,
       PSLD_FIR_PAD0, PSLD_FIR_PAD1, PSLD_FIR_KH, PSLD_FIR_DTYPE, PSLD_FIR_CACT };

/* --- PSLD_OP_CONV: y = scale * (conv(cat(x1,x2), W) + bias + temb[n,:] + residual)
 *   (ddpm_conv3x3/conv1x1 layers.py:85-109; NIN layers.py:531-540; F.conv2d(stride=2)
 *   up_or_down_sampling.py:178; epilogue terms layerspp.py:262-274,88-91, ncsnpp.py:353-356)
 *   in[0] = x1, in[1] = x2 or NULL, in[2] = residual [N,OH,OW,Cout] or NULL,
 *   in[3] = temb proj (f32) or NULL, in[4] = weight, in[5] = bias f32 [Cout] or NULL
 *   in[8], in[9] = (tensor-core engines, i[EXT_C1] > 0) a second input cat(e1, e2) [N,OH,OW,EXT_C1+EXT_C2]
 *           whose 1x1 convolution is accumulated into the same output tile: y = scale*(conv(x,W) +
 *           conv1x1(e, We) + bias + ...); the weight is then [Cout, K + EXT_C1 + EXT_C2] with the
 *           1x1 part appended along K (ResnetBlockBigGANpp's Conv_2 shortcut, layerspp.py:269-274)
 *   in[6] = (engine PSLD_ENGINE_TC_GN) fp32 [N, Cin, 2] (scale, shift) produced by a PSLD_OP_GN
 *           in affine-only mode: the conv input is silu?(x * scale + shift), applied in-kernel
 *           (i[GN_SILU] selects the SiLU); x1/x2 are then the RAW, un-normalised tensors (the
 *           extension input e, if any, is never normalised)
 *   out[0] = y
 *   out[1] = optional f64 [N, Cout/4, 2] (sum, sum of squares) of y per sample x 4 channels for the
 *            GroupNorms that consume it: ACCUMULATED with atomics by the epilogue, so the caller
 *            zeroes it before the launch (PSLD_OP_ZERO) (TC engines, bf16 NHWC output,
 *            OH*OW % 32 == 0), or NULL
 *   weight layout: SIMT engine f32 [K, Cout] ; TC engine bf16 [Cout, K], K = (ky*KW+kx)*Cin + c
 *   OUT_LAYOUT = NCHW (the network's output head): y is fp32 [N, V, OH, OW] with V = Cout (SIMT) or
 *           V = f[1] valid channels of a zero-padded Cout (TC engines); the residual, if any, is then
 *           fp32 NCHW of the same shape (RES_DTYPE = PSLD_F32) and is added to those V channels
 *           (progressive=output_skip: the upsampled output pyramid, ncsnpp.py:414-418)
 *   PSLD_ENGINE_TC output widths: OW a power of two in 4..128, or 256 for stride 1 (half-row tiles)
 *   i: N, H, W, C1, C2, COUT, KS (1|3), STRIDE, PAD, OH, OW, IN_LAYOUT, OUT_LAYOUT,
 *      IN_DTYPE, OUT_DTYPE, RES_DTYPE, TEMB_OFF, TEMB_BSTRIDE ; f[0] = scale            */
enum { PSLD_CONV_N = 0, PSLD_CONV_H, PSLD_CONV_W, PSLD_CONV_C1, PSLD_CONV_C2, PSLD_CONV_COUT,
       PSLD_CONV_KS, PSLD_CONV_STRIDE, PSLD_CONV_PAD, PSLD_CONV_OH, PSLD_CONV_OW,
       PSLD_CONV_IN_LAYOUT, PSLD_CONV_OUT_LAYOUT, PSLD_CONV_IN_DTYPE, PSLD_CONV_OUT_DTYPE,
       PSLD_CONV_RES_DTYPE, PSLD_CONV_TEMB_OFF, PSLD_CONV_TEMB_BSTRIDE, PSLD_CONV_GN_SILU,
       PSLD_CONV_EXT_C1, PSLD_CONV_EXT_C2 };

/* --- PSLD_OP_ATTN (AttnBlockpp core, layerspp.py:82-86): single head over HW tokens.
 *   in[0] = qkv [N, HW, 3C] (q | k | v along the last axis) ; out[0] = o [N, HW, C]
 *   i: N, HW, C, DTYPE, PROJ ; f[0] = softmax scale (C^-0.5)
 *   PROJ = 1 (PSLD_ENGINE_TC, HW % 128 == 0): the block's output projection and skip connection are
 *   fused (layerspp.py:87-91): out[0] = (NIN_3(o) + x) * f[1] with in[1] = NIN_3 weight bf16
 *   [C out, C in], in[2] = bias f32 [C] or NULL, in[3] = x [N, HW, C]; out[1] = optional GroupNorm
 *   statistics accumulator of out[0] (as for PSLD_OP_CONV)                                 */
enum { PSLD_ATTN_N = 0, PSLD_ATTN_HW, PSLD_ATTN_C, PSLD_ATTN_DTYPE, PSLD_ATTN_PROJ };

/* Standalone PSLD_OP_AXPBY: out = a * x + b * y over n floats (y may be NULL). */
PSLD_API int psld_axpby(float* out, float a, const float* x, float b, const float* y, int64_t n,
                        psld_stream_t stream);

/* Validate an op and build its per-op host state (TMA descriptors for PSLD_ENGINE_TC).
 * Returns PSLD_EUNSUPPORTED when the shape is not eligible for op->engine. */
PSLD_API int psld_op_prepare(psld_op* op);
PSLD_API int psld_op_release(psld_op* op);
/* Launch one op / a whole program on `stream`. */
PSLD_API int psld_op_run(const psld_op* op, psld_stream_t stream);
PSLD_API int psld_program_run(const psld_op* ops, int n_ops, psld_stream_t stream);
/* Number of kernel launches psld_program_run issues for this program (bench accounting). */
PSLD_API int psld_program_launches(const psld_op* ops, int n_ops);

/* Standalone drop-in for the reference's native op (op/upfirdn2d.cpp:12-23): NCHW fp32
 * input [N*C, H, W] planes, taps [kh, kw] on the HOST, same argument meaning. */
PSLD_API int psld_upfirdn2d(const float* input, float* output, const float* taps_host, int kh, int kw,
                   int64_t planes, int in_h, int in_w, int up_x, int up_y, int down_x,
                   int down_y, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                   psld_stream_t stream);

/* ------------------------------------------------------------------------------------
 * 3. Native sampling loop: runs all n predictor steps (+ denoise) without returning to
 *    the host interpreter.  SSCSSampler.sample / EulerMaruyamaSampler.sample
 *    (main/samplers/sde.py:38-58, 350-370).
 * ---------------------------------------------------------------------------------- */
typedef struct {
  int32_t sampler;      /* 0 = sscs_sde, 1 = em_sde                                     */
  int32_t n_steps;      /* predictor steps n                                            */
  int32_t denoise;      /* 1: final denoising step (one more network call)              */
  int32_t state_dtype;  /* PSLD_F64 | PSLD_F32                                          */
  int32_t fuse_halves;  /* SSCS: 0 = A | net | SCORE+B per step (3 state passes / 2 steps);
                           1 = SCORE+B+C in one pass (C = half A of step i+1, own draw);
                           2 = same, with B and C pre-merged by the host into half_b (one
                               Gaussian draw, exact in law; only without pre-drawn noise)    */
  int32_t temb_op;      /* index of the (first) PSLD_OP_TEMB op in the program; EVERY PSLD_OP_TEMB op of
                           the program receives the call's time (a classifier-free-guidance program
                           holds two networks)                                           */
  int64_t B, chw;
  uint64_t seed;
  void* state;          /* [B,2C,H,W] state_dtype, in: prior, out: samples              */
  float* net_in;        /* [B,2C,H,W] fp32 : program input buffer                       */
  const float* eps;     /* program output buffer (fp32 NCHW)                            */
  const float* time_table; /* device f32 [n_steps+1]: log(tau) (fourier) or tau per call */
  const float* noise;   /* pre-drawn fp32 noise [draws, B,2C,H,W] in reference draw order,
                           or NULL for in-kernel Philox                                 */
  const psld_sscs_coeffs* sscs; /* host [n_steps]  (sampler 0)                          */
  const psld_score_step* em;    /* host [n_steps]  (sampler 1)                          */
  const psld_score_step* den;   /* host, denoise step coefficients                      */
  void* record;         /* optional: state after every step [n_steps, B,2C,H,W] or NULL */
  /* CUDA-graph replay (optional; all three non-NULL enables it, Philox noise only, no record):
   * ONE predictor step (program + fused update + counter increment) is stream-captured and the
   * instantiated graph is launched n_steps times; per-step scalars are read on the device from
   * these tables at row *step_counter.  `stream` must not be the legacy default stream.        */
  const psld_sscs_coeffs* sscs_dev; /* device copy of sscs[n_steps]                            */
  const psld_score_step* em_dev;    /* device copy of em[n_steps]                              */
  int32_t* step_counter;            /* device int32, zeroed by the caller                      */
} psld_sampler_desc;

PSLD_API int psld_sampler_run(const psld_op* ops, int n_ops, const psld_sampler_desc* d,
                     psld_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PSLD_B200_H_ */
