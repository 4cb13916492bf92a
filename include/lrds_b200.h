/*
 * lrds_b200.h - C ABI of the B200-native batched trajectory rollout of sde_sampler_lrds.
 *
 * The reference has no FFI: its seam is the Python method contract of the loss objects in
 * sde_sampler/losses/oc.py (SURVEY.md 8b).  Every entry point below names the reference
 * interface it replaces.  All pointers are DEVICE pointers unless stated otherwise, all
 * matrices row-major float32, `stream` is a cudaStream_t.  Calls are asynchronous on `stream`,
 * never allocate, never throw; they return LRDS_OK or a negative lrds_status (message via
 * lrds_last_error()).  One call per GPU; re-entrant across streams and devices.
 */
#ifndef LRDS_B200_H
#define LRDS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRDS_ABI_VERSION 10 /* 10: lrds_adjoint; 9: lrds_gmm.layout (full-covariance Gaussian / mixture references) */
#define LRDS_CHANNELS 64 /* FourierMLP / TimeEmbed width, conf/model/base/fouriermlp.yaml:4 */
#define LRDS_MAX_DIM_PAD 1024 /* largest d_pad the operand packers accept */

typedef enum {
  LRDS_OK = 0,
  LRDS_ERR_INVALID = -1,     /* bad argument / inconsistent spec */
  LRDS_ERR_UNSUPPORTED = -2, /* valid in the reference but not built here (no silent fallback) */
  LRDS_ERR_CUDA = -3,        /* CUDA runtime error, see lrds_last_error() */
  LRDS_ERR_RESOURCES = -4    /* per-particle state does not fit in shared memory */
} lrds_status;

/* Which loop of losses/oc.py runs. */
typedef enum {
  LRDS_ROLLOUT_LINEAR = 0,     /* EM/EI/DDPM-like/DDS simulate: oc.py:218-296, 444-510, 584-651, 1319-1397 */
  LRDS_ROLLOUT_CMCD = 1,       /* ControlledLangevinSDELoss.simulate, oc.py:666-755 */
  LRDS_ROLLOUT_EUBO_LINEAR = 2,/* EM/EI compute_eubo, oc.py:298-362, 512-568 */
  LRDS_ROLLOUT_EUBO_CMCD = 3   /* ControlledLangevinSDELoss.compute_eubo, oc.py:757-828 */
} lrds_rollout_kind;

/* State update of one LINEAR step (u = control, r = reference score, z ~ N(0,I)). */
typedef enum {
  LRDS_UPDATE_AXPY = 0, /* x' = (a x + b (r + u)) + c z       EI/DDPM: eq/sdes.py:532-555, 658-678; DDS: oc.py:1373-1377 */
  LRDS_UPDATE_EM = 1    /* x' = x + ((-(f x) + s2 r) + sig u) dt + sig (z sqrt_dt)   oc.py:277-281 */
} lrds_update_form;

/* Ito (martingale) term of one LINEAR step. */
typedef enum {
  LRDS_ITO_NONE = 0,   /* DDS with compute_ito_int=False, oc.py:1380 */
  LRDS_ITO_SCALED = 1, /* rnd += w_ito * sum(u z)                 oc.py:499, 639 */
  LRDS_ITO_EM = 2,     /* rnd += sum(u * (z * sqrt_dt))           oc.py:277, 284 */
  LRDS_ITO_DDS = 3     /* rnd += sum(((sig u) z) * beta_k)        oc.py:1381-1383 (sig in A, beta_k in W_ITO) */
} lrds_ito_form;

typedef enum {
  LRDS_CTRL_CLIPPED = 0, /* ClippedCtrl.forward, models/reparam.py:33-43 (base_zero_init) */
  LRDS_CTRL_SCORE = 1,   /* ScoreCtrl.forward, models/reparam.py:112-117 (target_informed_zero_init) */
  /* The two DIS parametrisations (LINEAR simulate and lrds_ctrl_forward only; they run the run-time-switched kernels): */
  LRDS_CTRL_CANCEL_DRIFT = 2, /* CancelDriftCtrl.forward, models/reparam.py:131-147 (target_informed_langevin_init):
                               * u = (clip(net) + CX x) + GSCALE ((scale_score clip(target_score)) gamma),  CX = f(t)/sigma(t),
                               * GSCALE = sigma(t)/2 */
  LRDS_CTRL_LERP = 3     /* LerpCtrl.forward, models/reparam.py:189-199 (target_informed_lerp_tempering, hard_constrain=False):
                          * u = clip(net) + GSCALE ((scale_score clip(lerp(prior_score, target_score, LERP))) gamma),
                          * GSCALE = sigma(t), LERP = t / terminal_t, prior_score from ref_0 (a diagonal Gaussian: the prior) */
} lrds_ctrl_kind;

typedef enum {
  LRDS_DISTR_NONE = 0,
  LRDS_DISTR_GMM = 1,   /* Gaussian / mixture, diagonal (distr/gauss.py:67-73, 97-107, 124-126, 202-221) or full (gmm.layout) */
  LRDS_DISTR_PHI4 = 2,  /* PhiFour U / grad_U, distr/phi_four.py:45-96 (dim_phys=1, Dirichlet-0) */
  LRDS_DISTR_LOGREG = 3 /* LogisticRegression.posterior_log_prob + its autograd score, distr/logistic_regression.py:41-61 */
} lrds_distr_kind;

typedef enum {
  LRDS_PRECISION_FP32_SIMT = 0, /* FFMA everywhere (parity anchor) */
  LRDS_PRECISION_TF32X3 = 1,    /* tcgen05 kind::tf32, 3-pass (hi, lo) split: fp32-grade drift MLP on tensor cores */
  LRDS_PRECISION_BF16 = 2,      /* tcgen05 kind::f16 single pass: reduced-precision fast mode, reported separately */
  LRDS_PRECISION_TF32 = 3,      /* tcgen05 kind::tf32 single pass: reduced-precision fast mode, reported separately */
  LRDS_PRECISION_F16X3 = 4      /* tcgen05 kind::f16, 3-pass (hi, lo) fp16 split of power-of-two scaled operands: fp32-grade
                                 * like TF32X3 (22 mantissa bits per operand) at half its shared-memory / TMEM footprint and
                                 * twice its tensor rate; operands must stay below 65504 (particle coordinates) resp. 1023
                                 * (hidden activations) in magnitude, beyond that they saturate */
} lrds_precision;

/* Per-step table: one row of `step_stride` floats per grid time (K rows; K+1 for the CMCD kinds, whose
 * row k describes time ts[k]).  The host fills it with the reference's own float32 scalar formulas
 * (eq/sdes.py) so that schedules agree bit for bit.  Offsets into a row: */
enum {
  LRDS_STEP_A = 0,       /* AXPY: a          | EM: drift coefficient f(tau)      | DDS ito: see LRDS_ITO_DDS */
  LRDS_STEP_B = 1,       /* AXPY: b          | EM: sigma(tau)                                              */
  LRDS_STEP_C = 2,       /* AXPY: c          | EM: sigma(tau)^2                                            */
  LRDS_STEP_DT = 3,      /* t - s                                                                         */
  LRDS_STEP_SQRT_DT = 4, /* sqrt(t - s)                                                                   */
  LRDS_STEP_W_COST = 5,  /* rnd += W_COST * sum(u^2): 0.5*omega (EI), 0.5*dt (EM), 0.5*beta_k^2 sigma^2 (DDS) */
  LRDS_STEP_W_ITO = 6,   /* sqrt(omega) (EI/DDPM), beta_k (DDS)                                            */
  LRDS_STEP_GAMMA = 7,   /* clip(score_model(tau)) of ScoreCtrl, models/reparam.py:101-110                 */
  LRDS_STEP_FRAC = 8,    /* CMCD: t / terminal_t, eq/sdes.py:103                                           */
  LRDS_STEP_SIGU = 9,    /* DDS ito: sigma                                                                 */
  LRDS_STEP_EU_A = 10,   /* EUBO: mean factor                                                              */
  LRDS_STEP_EU_B = 11,   /* EUBO: std factor                                                               */
  LRDS_STEP_EU_C = 12,   /* EUBO-EM: 1/mean - 1 + f(tau) dt ; EUBO ito weight in W_ITO                      */
  LRDS_STEP_CX = 13,     /* LRDS_CTRL_CANCEL_DRIFT: sde.drift_coeff_t(t) / sde.diff(t)                         */
  LRDS_STEP_LERP = 14,   /* LRDS_CTRL_LERP: t / sde.terminal_t                                                */
  LRDS_STEP_GSCALE = 15, /* LRDS_CTRL_CANCEL_DRIFT: sde.diff(t) / 2 ; LRDS_CTRL_LERP: sde.diff(t)              */
  LRDS_STEP_BIAS1 = 16,  /* 64 floats: input_embed.bias + TimeEmbed_2(tau), models/mlp.py:136-139           */
  LRDS_STEP_STRIDE = 80
};

/* Drift backbone FourierMLP (models/mlp.py:99-143), weights pre-transposed so that the 64 outputs of one
 * input feature are contiguous. */
typedef struct {
  int32_t d;            /* particle dimension */
  int32_t d_pad;        /* d rounded up to a multiple of 8 */
  int32_t num_hidden;   /* hidden 64x64 layers (num_layers - 2) */
  int32_t reserved;
  const float* w_in_t;  /* [d][64]            input_embed.weight^T */
  const float* w_hid_t; /* [num_hidden][64][64] hidden_layer[i].weight^T */
  const float* b_hid;   /* [num_hidden][64] */
  const float* w_out_t; /* [64][d_pad]        out_layer.weight^T, zero padded */
  const float* b_out;   /* [d_pad] */
  const void* tc_image; /* weight image written by lrds_pack_mlp_tc for spec.precision (tensor-core precisions only) */
} lrds_mlp;

/* Storage layout of a lrds_gmm block. */
typedef enum {
  LRDS_GMM_DIAG = 0, /* diagonal covariances: logc, mu, ivar, sn (and optionally mix_tc) as described below */
  LRDS_GMM_FULL = 1  /* full covariances (eq/sdes.py:232-239, distr/gauss.py:76-121): logc and mu as below, and
                      * sn = the precision matrices [M][d_pad][d_pad] (row-major, zero in the padded rows and columns,
                      * step_stride_sn = M d_pad^2 for a per-step block); ivar and mix_tc are unused (NULL).
                      * logc_m = log w_m - d/2 log(2 pi) - 1/2 log det(Sigma_m).  Accepted as spec.ref_t / spec.ref_0 of
                      * the LINEAR and EUBO_LINEAR kinds and by lrds_distr_eval; LRDS_ERR_UNSUPPORTED everywhere else
                      * (targets, CMCD / DIS priors, lrds_mala, lrds_score_cot_sums). */
} lrds_gmm_layout;

/* Gaussian mixture with M >= 1 components.  `step_stride_*` = 0 for a static distribution; for the
 * time-marginal reference p_t^ref (eq/sdes.py:208-248, 281-345) the arrays hold one block per step and the
 * strides are the element distance between consecutive steps.  The fields below describe the diagonal layout
 * (layout = LRDS_GMM_DIAG); see lrds_gmm_layout for the full one. */
typedef struct {
  int32_t M;
  int32_t layout; /* lrds_gmm_layout; 0 (a zero-initialised block) = diagonal */
  const float* logc; /* [4 ceil(M/4)]  log w_m - d/2 log(2 pi) - 1/2 sum_j log var_mj (w normalised); padding = -inf; 16-byte aligned */
  const float* mu;   /* [M][d_pad]  rows padded with 0 to d_pad = 8 ceil(d / 8) floats, 16-byte aligned */
  const float* ivar; /* [M][d_pad]  1 / var, padded with 0 */
  const float* sn;   /* [ceil(M/4)][d_pad/4][4][8]  operands of the mixture kernels (M > 1): for mode block b, dim group c
                      * and mode i = 4 b + i': {1/sigma_{i,4c..4c+3}, -mu/sigma_{i,4c..4c+3}}, zero for padded dims and modes, so
                      * that (x - mu)/sigma = x * (1/sigma) + (-mu/sigma) is one FMA and every load has an immediate offset */
  int64_t step_stride_logc;  /* floats between consecutive steps of logc (4 ceil(M/4)) */
  int64_t step_stride_param; /* floats between consecutive steps of mu / ivar (M * d_pad) */
  int64_t step_stride_sn;    /* floats between consecutive steps of sn (8 ceil(M/4) * d_pad) */
  const void* mix_tc;        /* optional (M > 1; NULL = evaluate the score contraction on the SIMT pipes): tensor-core operand
                              * of  score_j = x_j sum_m r_m (-1/var_mj) + sum_m r_m mu_mj/var_mj.  Per step one block of
                              * lrds_gmm_mix_tc_bytes(M, d_pad) bytes: the matrix B[n][m], rows n = 16 c + i over the 8-dim
                              * chunks c (i < 8: -1/var_{m,8c+i}; i >= 8: mu/var_{m,8c+i-8}), multiplied by the power of two
                              * that puts its largest entry into [2^14, 2^15) and split into fp16 hi | lo parts, each in the
                              * K-major no-swizzle tcgen05 layout [m/8][n][m%8] with m padded to a multiple of 16; then 16
                              * bytes whose first float is the un-scale.  Behind it the LOGIT image of the block: the
                              * responsibilities r = softmax_m(logc_m - q_m / 2) of a mixture whose modes share their
                              * variances need only  logit_m = c_m + x . wc_m  (the x^2 term is mode-independent), with
                              * wc_mj = mu_mj/var_mj - mean_m(mu_mj/var_mj),  c_m = logc_m - sum_j mu_mj^2/var_mj / 2 - max over the modes:
                              * wc as a power-of-two scaled fp16 hi | lo matrix [j/8][m][j%8] (rows m padded to a multiple
                              * of 16, K = j padded to a multiple of 16), then c_m (fp32, -inf for padded modes), then four
                              * floats {un-scale, max_m |wc_m|_2, max_m |c_m|, 1.0 if the variances are shared else 0.0}.
                              * The kernels use it only when that flag is set and a per-particle error bound allows;
                              * otherwise they evaluate the quadratic forms exactly (sn).  16-byte aligned. */
  int64_t step_stride_mix_tc;/* BYTES between consecutive steps of mix_tc */
} lrds_gmm;

typedef struct {
  float a, b, beta; /* conf/target/phi_four.yaml; coef = a * d */
  float reserved;
} lrds_phi4;

typedef struct {
  int32_t N, p;       /* data rows, features; d = p + 1 (intercept last) */
  int32_t n_pad;      /* N rounded up to a multiple of 4 */
  int32_t reserved;
  const float* X;     /* [N][d_pad]   rows zero padded beyond p (for the gradient pass) */
  const float* Xt;    /* [p][n_pad]   transposed, zero padded (for the logit pass) */
  const float* y;     /* [n_pad] */
  float weight_scale, intercept_mean, intercept_scale;
  float threshold;    /* 1e-8, logistic_regression.py:27,56 */
  float eps;          /* float32 machine eps used by probs_to_logits (2^-23) */
  float reserved2;
  const void* x_tc;   /* optional (NULL = both passes on the SIMT pipes): tensor-core operand of the logit GEMM z = X w + b and
                       * of the gradient GEMM sum_n g_n X_n.  Img[n][k] = X[n][k] (k < p), 1 (k = p), 0 beyond, n padded to
                       * N16 = 16 ceil(N/16) and k to K16 = 16 ceil((p+1)/16), times the power of two that puts its largest
                       * entry into [2^14, 2^15), as fp16 hi | lo parts, each K-major no-swizzle [k/8][n][k%8] (the gradient
                       * GEMM reads the same bytes MN-major); then 16 bytes whose first float is the un-scale; then y as N16
                       * floats.  16-byte aligned; 4 N16 K16 + 16 + 4 N16 bytes. */
} lrds_logreg;

typedef struct {
  int32_t kind; /* lrds_distr_kind */
  int32_t reserved;
  lrds_gmm gmm;
  lrds_phi4 phi4;
  lrds_logreg logreg;
} lrds_distr;

typedef struct {
  int32_t abi_version; /* LRDS_ABI_VERSION */
  int32_t kind;        /* lrds_rollout_kind */
  int32_t update_form; /* lrds_update_form (LINEAR kinds) */
  int32_t ito_form;    /* lrds_ito_form    (LINEAR kinds) */
  int32_t ctrl_kind;   /* lrds_ctrl_kind */
  int32_t precision;   /* lrds_precision */
  int32_t B, d, K;     /* particles on this GPU, dimension, steps */
  int32_t has_ref_ctrl;/* LINEAR: reference_ctrl is not None (RDS yes, PIS/DDS no) */
  float clip_model;    /* <= 0: no clip (models/reparam.py:25) */
  float clip_score;    /* <= 0: no clip (models/reparam.py:79) */
  float scale_score;   /* ScoreCtrl.scale_score */
  float clip_target;   /* <= 0: none (TrainableDiff.clip_target, solver/oc.py:33,80-87) */
  float cmcd_diff;     /* ControlledLangevinSDE.diff_coeff, eq/sdes.py:93 */
  float cmcd_clip;     /* ControlledLangevinSDE.clip_score, <= 0: none */
  int32_t init_cost;   /* LINEAR (simulate only): 0 = rnd starts at 0 and ends with + reference_log_prob(x_T), ref_0 being the
                        * reference (RDS / PIS / DDS: oc.py:245, 290, 1389); 1 = rnd starts at initial_log_prob(x_0) + rnd_offset,
                        * ref_0 being the PRIOR, and ends with the target term alone (DIS: TimeReversalLoss.simulate,
                        * oc.py:1164-1168, 1230; DiscreteTimeReversalLossEI.simulate, oc.py:925-973).  EUBO_LINEAR with
                        * init_cost = DiscreteTimeReversalLossEI.compute_eubo (oc.py:980-1036): no reference control, rnd
                        * starts at -target(x) and ends with + initial_log_prob(x) at the noised state */
  float rnd_offset;    /* init_cost: state-independent part of the log-weight, -sum_k sde.drift_div_int(s_k, t_k, x)
                        * (OU.drift_div_int = d * int_drift_coeff_t, eq/sdes.py:137-141; oc.py:1217-1218, train=False) */
  const float* steps;  /* per-step table, LRDS_STEP_STRIDE floats per row */
  lrds_mlp mlp;
  lrds_distr target;   /* terminal_unnorm_log_prob + ScoreCtrl.target_score */
  lrds_gmm ref_t;      /* time-marginal reference score (has_ref_ctrl), one block per step */
  lrds_gmm ref_0;      /* reference_log_prob at the end of the rollout (LINEAR) / prior = initial_log_prob (CMCD) */
  uint32_t* status;    /* optional (NULL = not counted): two device counters the rollout ADDS to.  [0] += particle threads
                        * of an F16X3 launch whose fp16 tensor-core operands saturated at least once (a coordinate beyond
                        * 65504 or a hidden pre-activation beyond 1023: the results of such a particle are not fp32-grade -
                        * rerun with TF32X3, which has no magnitude limit); [1] += particles whose final log-weight or
                        * state is not finite.  The two-threads-per-particle kernels count every thread that saw a
                        * saturating value, so [0] can reach twice the number of affected particles. */
} lrds_spec;

/* ---- the rollout: replaces loss.simulate / loss.compute_eubo (losses/oc.py, callers solver/oc.py:305-632,
 * additions/hacking.py:14-33).
 *   x0       [B][d]   prior samples (EUBO kinds: target samples)
 *   noise    [K][B][d] standard normals to consume (validation mode: the reference's own increments), or NULL
 *            for production mode = in-kernel Philox4x32-10 keyed by (seed, particle_offset + b, step, j/4)
 *   x_out    [B][d]   final states (may alias x0)          rnd_out [B] log-weights
 *   traj_out [K+1][B][d] or NULL (return_traj)
 */
int lrds_rollout(const lrds_spec* spec, const float* x0, const float* noise, uint64_t seed,
                 uint64_t particle_offset, float* x_out, float* rnd_out, float* traj_out, void* stream);

/* ---- the pathwise (method 'kl' / 'kl_ito') gradient of the LINEAR simulate loop: the reverse-time recursion that
 * autograd runs through the K steps when the SDE follows the non-detached control (generative_and_sde_ctrl,
 * oc.py:83-103) and loss = mean(rnd[mask]) (compute_loss, oc.py:105-131).  With g_k = clip(net(t_k, x_k)) and
 * e_k = the Ito weight of lrds_ito_form times z_k (0 for LRDS_ITO_NONE), the adjoint of particle b is
 *   lambda_K = w_b (grad ref_0(x_K) - [|target(x_K)| <= clip_target] grad target(x_K))        (init_cost: no ref_0 term)
 *   gbar_k   = w_b (2 W_COST g_k + e_k) + (d x_{k+1} / d g) lambda_{k+1}                        (B for AXPY, B dt for EM)
 *   lambda_k = a_k lambda_{k+1} + c_k J_r(x_k) lambda_{k+1} + J_net^T ([|net| <= clip_model] gbar_k)
 *              (a_k, c_k) = (A, B) for AXPY, (1 - A dt, C dt) for EM; J_r = the Jacobian of the reference score
 * and d loss / d theta = sum_k <gbar_k, d g_k / d theta>: lrds_mlp_grad with cot = gbar (step_w = row_w = NULL).
 *   traj    [K+1][B][d] the trajectory lrds_rollout wrote for this spec
 *   noise   [K][B][d] the increments that rollout consumed, or NULL: the kernel regenerates the production-mode Philox
 *           increments of (seed, particle_offset)
 *   row_w   [B] w_b = d loss / d rnd_b
 *   cot_out [K][B][d] gbar_k = d loss / d g_k
 * Built for the LRDS_ROLLOUT_LINEAR kind, LRDS_CTRL_CLIPPED, a diagonal reference (or none), every target kind, and the
 * precisions F16X3 / TF32X3 / FP32_SIMT; LRDS_ERR_UNSUPPORTED for the score-family controls, full-covariance ref_t /
 * ref_0, the CMCD and EUBO kinds and BF16 / TF32 (their network is not the one the adjoint would linearise).  F16X3 inside
 * lrds_mlp_grad's envelope (d <= 64, num_hidden <= 2; mlp.tc_image = the F16X3 image) runs the network on tcgen05 with the
 * rollout's weight image and adds to spec.status like the rollout: [0] += threads (four per particle) whose fp16 operands
 * saturated (a coordinate or cotangent beyond 65504, a hidden pre-activation beyond 1023), [1] += particles with a
 * non-finite cotangent.  Every other accepted spec recomputes the network with fp32 FFMA and never touches [0]. */
int lrds_adjoint(const lrds_spec* spec, const float* traj, const float* noise, uint64_t seed, uint64_t particle_offset,
                 const float* row_w, float* cot_out, void* stream);

/* ---- tensor-core weight image: the FourierMLP weights in the shared-memory operand layout of tcgen05.mma (plus
 * the fp32 biases), staged once per CTA by a bulk TMA copy.  `image_out` (device, 16-byte aligned) must hold
 * lrds_tc_image_bytes(d, num_hidden, precision) bytes; set mlp.tc_image to it before lrds_rollout.  Repack after
 * every weight update. */
int64_t lrds_tc_image_bytes(int32_t d, int32_t num_hidden, int32_t precision);
int64_t lrds_gmm_mix_tc_bytes(int32_t M, int32_t d_pad); /* one block of lrds_gmm.mix_tc */
/* Builds lrds_gmm.mix_tc from gmm->logc / mu / ivar (M > 1): `steps` consecutive blocks (1 for a static mixture, K for
 * the time-marginal reference, read with step_stride_logc / step_stride_param) of lrds_gmm_mix_tc_bytes(M, d_pad) bytes
 * each; `d` = the number of real dims (<= d_pad). */
int lrds_pack_gmm_mix_tc(const lrds_gmm* gmm, int32_t d, int32_t d_pad, int32_t steps, void* image_out, void* stream);
/* Builds lrds_logreg.x_tc (lrds_logreg_tc_bytes(N, p) bytes) from logreg->X ([N][d_pad]) and logreg->y. */
int64_t lrds_logreg_tc_bytes(int32_t N, int32_t p);
int lrds_pack_logreg_tc(const lrds_logreg* logreg, int32_t d_pad, void* image_out, void* stream);
int lrds_pack_mlp_tc(const lrds_mlp* mlp, int32_t precision, void* image_out, void* stream);

/* ---- estimator partials: replaces BaseOCLoss.compute_results (oc.py:134-173), ESS (eval/metrics.py:134-140)
 * and evaluate_eubo (additions/hacking.py:24-32).  Writes 8 doubles to `partials` (device):
 *   [0] m = max(-rnd)  [1] sum exp(-rnd - m)  [2] sum exp(2(-rnd - m))  [3] sum rnd  [4] sum rnd^2
 *   [5] count          [6] m' = max(rnd)      [7] sum exp(rnd - m')
 * Partials of several GPUs merge associatively (the only cross-GPU exchange of the path).
 * `scratch` must hold at least 8 * (blocks + 1) doubles where blocks = lrds_estimator_blocks(B). */
int lrds_estimator_blocks(int32_t B);
int lrds_estimator_partials(const float* rnd, int32_t B, double* partials, double* scratch, void* stream);
/* Merge of n partial records parts[n][8] (the all_gather result) into out[8], on the device. */
int lrds_estimator_merge(const double* parts, int32_t n, double* out, void* stream);

/* ---- drop-in pieces of the same arithmetic, for the reference's smaller public interfaces.
 * control u = generative_ctrl(t, x) for the time of table row `row` (models/reparam.py:33-43, 112-117). */
int lrds_ctrl_forward(const lrds_spec* spec, int32_t row, const float* x, int32_t B, float* u_out, void* stream);

/* Parameter gradient of the drift backbone over S x B stored states: the vector-Jacobian product that autograd takes
 * through FourierMLP.forward (models/mlp.py:135-143) under the clip of ClippedCtrl (models/reparam.py:33-43) when
 * loss.backward() runs after BaseOCLoss.compute_loss with method 'lv' / 'lv_traj' (losses/oc.py:105-131; the SDE follows
 * the detached control there, so the states are constants and the gradient is one batched pass, see train.py).
 *   x     [S][B][d]  states (e.g. the trajectory lrds_rollout wrote), time row s is shared by the B rows of slice s
 *   bias1 [S][64]    input_embed.bias + TimeEmbed(t_s)  (the rows of LRDS_STEP_BIAS1)
 *   cot   [S][B][d]  cotangent of the clipped network output; multiplied by step_w[s] and row_w[b] when given
 *                    (log-variance loss: cot = z, step_w = the Ito weights, row_w = d loss / d rnd_b)
 *   clip             bound of the output clip (<= 0: none): rows/columns with |net| > clip receive no gradient
 *   cot_scale        power of two applied to the cotangents before their fp16 operands are formed and removed from the
 *                    results: choose it so that max |cot * step_w * row_w| * cot_scale is of order 1 .. 10;
 *   cot_scale_dev    optional device copy of that scalar (used instead when non-NULL: a caller whose bound lives on the
 *                    device, e.g. max |d loss / d rnd|, avoids the host round trip)
 * Outputs: grads_out = lrds_mlp_grad_floats(d, num_hidden) floats laid out like the weight blocks of lrds_mlp
 * ([d][64] w_in_t, [nh][64][64] w_hid_t, [nh][64] b_hid, [64][d_pad] w_out_t, [d_pad] b_out) and dbias1_out [S][64] (the
 * cotangent of bias1: its column sums are the gradient of input_embed.bias, and TimeEmbed's backward takes it from
 * there).  mlp->tc_image must be the LRDS_PRECISION_F16X3 image.  Built for d <= 64 and num_hidden <= 2 (the
 * reference's FourierMLP default, num_layers = 4); LRDS_ERR_UNSUPPORTED otherwise.  Sums run in a fixed order
 * (deterministic).  `scratch` holds lrds_mlp_grad_scratch_floats(d, num_hidden, S, B) floats. */
/* out[s][j] = sum_b step_w[s] row_w[b] cot[s][b][j] * clip(score(x[s][b]))[j]: the cotangent of the time-only factor
 * clip(TimeEmbed_score(t)) of ScoreCtrl / CancelDriftCtrl (models/reparam.py:112-117, 131-147) in the same batched
 * gradient pass (clip <= 0: none; step_w / row_w may be NULL).  Fixed summation order.  `scratch` holds
 * lrds_score_cot_scratch_floats(distr, d, S, B) floats. */
int64_t lrds_score_cot_scratch_floats(const lrds_distr* distr, int32_t d, int32_t S, int32_t B);
int lrds_score_cot_sums(const lrds_distr* distr, int32_t d, const float* x, const float* cot, const float* step_w,
                        const float* row_w, float clip, int32_t S, int32_t B, float* out, float* scratch, void* stream);
int64_t lrds_mlp_grad_floats(int32_t d, int32_t num_hidden);
int64_t lrds_mlp_grad_scratch_floats(int32_t d, int32_t num_hidden, int32_t S, int32_t B);
int lrds_mlp_grad(const lrds_mlp* mlp, const float* bias1, const float* x, const float* cot, const float* step_w,
                  const float* row_w, float clip, float cot_scale, const float* cot_scale_dev, int32_t S, int32_t B,
                  float* grads_out, float* dbias1_out, float* scratch, void* stream);
/* Distribution.unnorm_log_prob / score (distr/base.py:128-157); either output may be NULL. */
int lrds_distr_eval(const lrds_distr* distr, int32_t d, const float* x, int32_t B, float* logp_out,
                    float* score_out, void* stream);
/* out = (a x + b s) + c z : VP/PinnedBM.ei_integration_step / ddpm_integration_step (eq/sdes.py:532-555, 658-678)
 * and EulerIntegrator.integrate's update (eq/integrator.py:116-120) with a=1. */
int lrds_axpy_step(const float* x, const float* s, const float* z, float a, float b, float c, float* out,
                   int64_t n, void* stream);
/* z[K][B][d] of the production-mode generator (stream_id 0 = Brownian increments, 1 = prior draws). */
int lrds_normals(uint64_t seed, uint64_t particle_offset, int32_t stream_id, int32_t K, int32_t B, int32_t d,
                 float* out, void* stream);

/* ---- MALA chains: replaces the loop of mcmc_sample(mcmc_type='mala') (experiments/benchmark_utils.py:268-333) around
 * mala_step and heuristics_step_size (sde_sampler/additions/mcmc.py:75-134, 54-72) - the sampler that produces the data the
 * GMM reference is fitted to.  One launch runs n_warmup + n_steps Metropolis-adjusted Langevin steps of C chains
 * (one thread per chain), with the per-chain step-size heuristic (target acceptance 0.75, factor 1.01, tolerance 0.05)
 * after every step when `adapt` is set.
 *   y0 [C][d] initial states        step_size [C] in / out
 *   noise [n_warmup + n_steps][C][d] standard normals or NULL (in-kernel Philox, stream 0)
 *   unif  [n_warmup + n_steps][C] uniforms in (0, 1] of the accept test or NULL (Philox, stream 2)
 *   ys_out [n_steps][C][d] the chains after the warm-up      log_acc_out [n_warmup + n_steps][C] or NULL
 *   sampler: LRDS_MCMC_MALA, or LRDS_MCMC_RWMH = the other branch of mcmc_sample: rwmh_step (additions/mcmc.py:258-290),
 *   proposal y + step_size * z, acceptance on the log-density difference alone (no score is evaluated) */
typedef enum { LRDS_MCMC_MALA = 0, LRDS_MCMC_RWMH = 1 } lrds_mcmc_sampler;
int lrds_mala(const lrds_distr* target, int32_t d, int32_t C, int32_t n_warmup, int32_t n_steps, int32_t adapt,
              int32_t sampler, const float* y0, float* step_size, const float* noise, const float* unif, uint64_t seed,
              float* ys_out, float* log_acc_out, void* stream);

const char* lrds_last_error(void);
int lrds_abi_version(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches claim) */
int64_t lrds_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LRDS_B200_H */
