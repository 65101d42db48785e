/*
 * bean_b200.h -- C-ABI of the B200-native SVI hot path of `bean run` (pinellolab/crispr-bean).
 *
 * The reference has NO FFI / plugin interface for this path (pure Python on pyro + eager torch), so
 * these entry points replace Python-level op chains; each one cites the reference interface it
 * replaces (paths relative to the reference root).  See INTEGRATION.md for the ctypes binding a
 * maintainer would add to bean/model/model.py.
 *
 * Conventions
 *  - plain C: raw DEVICE pointers + sizes + a CUDA stream handle (void*, i.e. cudaStream_t);
 *    no torch / C++ types cross the boundary.
 *  - the caller owns every buffer (inputs, outputs, workspace); the library never allocates,
 *    frees or retains a pointer past the call.
 *  - every call is asynchronous on `stream`, never synchronises, never prints, never exits.
 *  - return value: BEAN_OK or a negative BEAN_E* code; `bean_last_error()` gives the message of the
 *    last failure on the calling thread.
 *  - there is NO CPU fallback: without a CUDA device every compute call returns BEAN_ECUDA.
 *  - `_f32` entry points take float buffers, `_f64` double buffers (the struct fields typed `void*`
 *    below are `real*`); count tensors hold integer-valued reals exactly as the reference stores them
 *    (`.float()`, bean/preprocessing/data_class.py:220-228).
 *
 * Layout (device): count rows are REPLICATE-MAJOR, re-tiled once at tensorisation from the reference's
 * (R, B, G) tensors:  x[layer][r][g][b],  allele_counts[r][g][a],  row_mask[r][g]  -- a kernel thread owns a guide,
 * so the rows the 32 threads of a warp read for replicate r are contiguous (one 128-bit load per thread at B = 4);
 * per-guide allele vectors stay guide-major:  pi[g][r][a],  mu_allele[g][a].
 */
#ifndef BEAN_B200_H_
#define BEAN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEAN_ABI_VERSION 16

enum {
  BEAN_OK = 0,
  BEAN_EINVAL = -1,   /* null pointer / bad shape / unsupported size */
  BEAN_ECUDA = -2,    /* CUDA runtime error (message in bean_last_error) */
  BEAN_EALIGN = -3    /* a buffer is not aligned for 128-bit access */
};

enum { BEAN_MODE_SORTING = 0, BEAN_MODE_SURVIVAL = 1 };

#define BEAN_MAX_BINS 8        /* n_condits incl. the control pseudo-bin (SURVEY App. B1) */
#define BEAN_MAX_RB 64         /* n_reps * n_bins per guide */
#define BEAN_MAX_ALLELES 4096  /* alleles per guide incl. wild type (raw tiling allele tables reach hundreds) */
#define BEAN_MAX_LAYERS 2
#define BEAN_SURV_FOLD_ROWS 1024 /* spare rows of BeanSurvivalState.abund_partial (second level of the abundance sums) */
#define BEAN_MAX_PEERS 8        /* GPUs of one box */
#define BEAN_PEER_MAX_VALS 72   /* >= n_reps + 1 */

int bean_abi_version(void);
const char* bean_last_error(void);
/* number of SMs of the current device (grid sizing), <0 on error */
int bean_device_sm_count(void);

/* ------------------------------------------------------------------------------------------------
 * Screen constants: everything the *ScreenData object holds that the likelihood reads every step.
 * Replaces the attribute reads of bean/model/model.py:123-165, :484-547 (data.X_masked,
 * data.X_bcmatch_masked, data.size_factor(_bcmatch), data.sample_mask, data.a0(_bcmatch),
 * data.repguide_mask, data.upper_bounds / lower_bounds | data.timepoints).
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanScreen {
  int32_t n_guides;            /* G */
  int32_t n_reps;              /* R */
  int32_t n_bins;              /* B = n_condits */
  int32_t n_layers;            /* 1 = guide counts, 2 = + barcode-matched counts (use_bcmatch) */
  int32_t mode;                /* BEAN_MODE_SORTING | BEAN_MODE_SURVIVAL */
  int32_t mask_thres;          /* row kept iff sum_b x > mask_thres (model.py:132-137; 10) */
  const void* x;               /* real [L][R][G][B]   X_masked / X_bcmatch_masked               */
  const void* a0;              /* real [L][G]         a0 / a0_bcmatch                           */
  const uint8_t* row_mask;     /* u8   [R][G]         repguide_mask (the reference's own layout)        */
  const double* row_const;     /* f64  [L][R][G] or NULL: data-only part of each row's log-pmf,
                                  lgamma(N+1) - sum_b lgamma(x_b+1) + sum_{x_b>0} x_b ln(x_b/N)   */
  /* small per-sample tables, HOST pointers (copied into kernel arguments):                      */
  const double* size_factor;   /* [L][R][B]           size_factor / size_factor_bcmatch         */
  const double* sample_mask;   /* [R][B]                                                        */
  const double* upper_thres;   /* [B] sorting: Phi^-1(upper_quantile), +inf where quantile == 1  */
  const double* lower_thres;   /* [B] sorting: Phi^-1(lower_quantile), -inf where quantile == 0  */
  const double* timepoints;    /* [B] survival: normalised time of each condition               */
} BeanScreen;

/* ------------------------------------------------------------------------------------------------
 * bean_ll_{f32,f64}: count log-likelihood forward + local gradients in one pass.
 *
 * Replaces, for every model of bean/model/model.py and bean/model/survival_model.py, the op chain
 *   get_std_normal_prob (model/utils.py:34-76) | exp(mu * t) (survival_model.py:358-361)
 *   -> mixture over alleles (model.py:495-499) -> get_alpha x L (model/utils.py:10-25)
 *   -> DirichletMultinomial(a).log_prob(X) under poutine.mask (model.py:526-547)
 * and its autograd backward.
 *
 * in : mu_allele, sd_allele  real [G][A]   per-guide allele mean / sd (sd ignored for survival)
 *      pi                    real [G][R][A] allele weights, or NULL for "all ones" (A must be 1)
 *      allele_mask           u8   [G][A]   or NULL (tiling: 0 = allele does not exist, P := 0)
 * out: ll_row                real [L][R][G] masked per-row log-prob (0 where masked), may be NULL
 *      ll_partial            double [bean_ll_num_partials(G, A)] per-CTA partial sums of the masked ll
 *      d_mu, d_sd            real [G][A]   d(sum ll)/d(mu_allele, sd_allele)
 *      d_pi                  real [G][R][A] d(sum ll)/d(pi), may be NULL when pi is NULL
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanLLArgs {
  int32_t n_alleles;           /* A */
  const void* mu_allele;
  const void* sd_allele;
  const void* pi;
  const uint8_t* allele_mask;
  void* ll_row;
  double* ll_partial;
  void* d_mu;
  void* d_sd;
  void* d_pi;
} BeanLLArgs;

int bean_ll_num_partials(int32_t n_guides, int32_t n_alleles);
int bean_ll_f32(const BeanScreen* screen, const BeanLLArgs* args, void* stream);
int bean_ll_f64(const BeanScreen* screen, const BeanLLArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bean_allele_gather / bean_allele_scatter: allele <- edit contraction of the tiling models.
 *
 * Replaces `torch.matmul(data.allele_to_edit, mu_edits)`, `torch.linalg.norm(data.allele_to_edit *
 * sd_edits, dim=-1)` and the prepended WT column (0, 1) (bean/model/model.py:618-625, :907-918;
 * survival_model.py:484-493) plus their autograd backward.  The dense 0/1 (G, A-1, E) tensor becomes
 * CSR (slot -> edits) for the forward and CSC (edit -> slots) for the deterministic backward.
 *   gather : mu_allele[g][0] = 0, sd_allele[g][0] = 1;  a >= 1: mu = sum_e mu_edit[e], sd = sqrt(sum_e sd_edit[e]^2)
 *   scatter: d_mu_edit[e] = sum_slots d_mu_allele;  d_sd_edit[e] = sum_slots d_sd_allele * sd_edit[e] / sd_allele
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanAlleleMap {
  int32_t n_guides;            /* G */
  int32_t n_alleles;           /* A = n_max_alleles, wild type included */
  int32_t n_edits;             /* E */
  int32_t nnz;
  const int32_t* allele_ptr;   /* i32 [G*(A-1)+1]  CSR over slots, slot = g*(A-1) + (a-1) */
  const int32_t* allele_edit;  /* i32 [nnz]        edit ids of each slot                  */
  const int32_t* edit_ptr;     /* i32 [E+1]        CSC over edits                         */
  const int32_t* edit_slot;    /* i32 [nnz]        slots containing each edit             */
} BeanAlleleMap;

int bean_allele_gather_f32(const BeanAlleleMap* map, const void* mu_edit, const void* sd_edit, void* mu_allele,
                           void* sd_allele, void* stream);
int bean_allele_gather_f64(const BeanAlleleMap* map, const void* mu_edit, const void* sd_edit, void* mu_allele,
                           void* sd_allele, void* stream);
int bean_allele_scatter_f32(const BeanAlleleMap* map, const void* sd_edit, const void* sd_allele, const void* d_mu_allele,
                            const void* d_sd_allele, void* d_mu_edit, void* d_sd_edit, void* stream);
int bean_allele_scatter_f64(const BeanAlleleMap* map, const void* sd_edit, const void* sd_allele, const void* d_mu_allele,
                            const void* d_sd_allele, void* d_mu_edit, void* d_sd_edit, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bean_svi_run_{f32,f64}: n_steps complete SVI steps on the device, no host round trip per step.
 *
 * One step = what `svi.step(data)` does in bean/model/run.py:376-380 for the variant sorting models:
 *   guide program  (model.py:754-782 Normal, :785-858 MixtureNormal, :861-875 ControlNormal):
 *       reparameterised draws  mu_targets ~ Normal, sd_targets ~ LogNormal, pi ~ Dirichlet
 *   model program  (model.py:19-165, :168-252, :378-547): priors, Dirichlet / Multinomial editing-rate
 *       sites, Normal-CDF bin probabilities, allele mixture, get_alpha, Dirichlet-Multinomial sites
 *   Trace_ELBO (1 particle) loss and its gradient (pyro.infer; pathwise Dirichlet derivative as
 *       torch._dirichlet_grad), then pyro.optim.ClippedAdam on the unconstrained parameters.
 * Kernels per step: a per-guide kernel (sampling, likelihood, editing-rate sites, per-guide d/d(mu, sd)), for the mixture
 * model a second per-guide kernel (pathwise Dirichlet derivative of every draw, alpha_pi gradient and its Adam update;
 * folded into the first when BeanSviState.pw / dconc are NULL) and a per-variant kernel (segmented reduction of the
 * guide gradients over the CSR variant ranges, prior / entropy terms, Adam on the variant parameters, loss).
 *
 * Randomness is counter-based (Philox4x32-10 keyed by `seed`, indexed by (entity, replicate, step)),
 * so a run is reproducible and independent of the launch geometry.  For parity tests the noise can be
 * injected instead (BeanSviNoise), and `apply_update = 0` returns the loss gradient w.r.t. the
 * unconstrained parameters without touching them.
 * ---------------------------------------------------------------------------------------------- */
enum { BEAN_MODEL_NORMAL = 0, BEAN_MODEL_MIXTURE_NORMAL = 1 };

typedef struct BeanSviConfig {
  int32_t model;            /* BEAN_MODEL_* (ControlNormal = NORMAL with one variant, sd_is_sqrt = 0) */
  int32_t sd_is_sqrt;       /* NormalModel feeds sqrt(sd_targets) to the CDF (model.py:92-98)        */
  int32_t mu_prior_normal;  /* 0: Laplace(0,1) (model.py:43); 1: Normal(mu_prior_loc, mu_prior_scale) */
  int32_t apply_update;     /* 1: ClippedAdam step; 0: only write gradients                          */
  int32_t phases;           /* 0: the whole step; otherwise a bit mask -- 1 guide kernel, 2 variant kernel, 4 alpha kernel
                               (split guide step only) -- so a benchmark can time each kernel with CUDA events */
  int32_t fit_noise;        /* --scale-by-acc only: 1 = guide Normal(noise_loc, noise_scale) on logit_pi_noise
                               (utils.py:145-155), 0 = drawn from the prior Normal(0, 0.655)           */
  int32_t force_generic;    /* 1: never pick the specialised kernels (exactly 4 / 5 bins, no masked sample); tests use it
                               to check that both code paths give the same numbers                      */
  int32_t reserved_;
  double mu_prior_loc, mu_prior_scale;
  double sd_prior_loc, sd_prior_scale; /* LogNormal prior on sd_targets: (0, 0.01); ControlNormal (0, 1) */
  double lr0, lrd;          /* ClippedAdam: lr_t = lr0 * lrd^t, lrd = gamma^(1/num_steps) (run.py:367) */
  double beta1, beta2, adam_eps, clip;
  double ll_const;          /* data-only part of the ELBO (sum of masked lgamma(1+N) - sum lgamma(1+x)) */
  double prob_clamp_eps;    /* torch.distributions.Multinomial clamps probs to [eps, 1 - eps] of THEIR dtype; in the reference
                               pi inherits pi_a0's dtype (float64 from the fit, float32 with the fallback coefficients,
                               get_pi_alpha0.py:109-143): 2.2e-16 or 1.19e-7.  0 selects the eps of the entry point's real */
  uint64_t seed;
  uint32_t guide_offset;    /* global index of this shard's first guide / variant: the Philox counters   */
  uint32_t variant_offset;  /* use GLOBAL ids, so a variant-sharded run draws exactly the unsharded noise */
} BeanSviConfig;

typedef struct BeanSviState {
  int32_t n_variants;            /* T */
  int32_t loss_capacity;
  const int32_t* guide_variant;  /* i32 [G]   variant of each guide (guides of a variant contiguous)  */
  const int32_t* variant_ptr;    /* i32 [T+1] CSR: guides of variant v are [ptr[v], ptr[v+1])          */
  const void* allele_counts;     /* real [R][G][2] control-condition reporter allele counts (MIXTURE)  */
  const void* pi_a0;             /* real [G]                                                            */
  void* var_params;              /* real [4][T]: mu_loc, log mu_scale, sd_loc, log sd_scale             */
  void* var_m;                   /* real [4][T] Adam first moments                                      */
  void* var_v;                   /* real [4][T] Adam second moments                                     */
  void* alpha_u;                 /* real [G][2] log alpha_pi (MIXTURE)                                  */
  void* alpha_m;
  void* alpha_v;
  void* d_guide;                 /* real [2][G] scratch: d ELBO / d(mu, sd) of each guide's edited allele */
  void* var_grad;                /* real [4][T] out (loss gradient, unconstrained) or NULL              */
  void* alpha_grad;              /* real [G][2] out or NULL                                             */
  double* partial;               /* f64 [bean_svi_num_partials(G, T)] scratch                           */
  uint32_t* counter;             /* u32 [1], zero before the first call                                 */
  double* loss;                  /* f64 [loss_capacity]: loss[t] = -ELBO of step t                      */
  /* --scale-by-acc (bean/model/utils.py:79-178); acc_k == NULL switches the whole block off           */
  const void* acc_k;             /* real [G]    exp(b) * accessibility^a  (a = 0.2513, b = -1.9458)     */
  void* noise_u;                 /* real [2][G] noise_loc, log noise_scale (fit_noise)                  */
  void* noise_m;
  void* noise_v;
  void* noise_grad;              /* real [2][G] out or NULL                                             */
  /* per-variant priors (`bean run --prior-params`, bean/model/run.py:480-542: tensors written by `bean build-prior`);
     each may be NULL -> the scalar of BeanSviConfig applies.  mu_prior_* are read only when mu_prior_normal = 1.  */
  const void* mu_prior_loc_v;    /* real [T] */
  const void* mu_prior_scale_v;  /* real [T] */
  const void* sd_prior_loc_v;    /* real [T] */
  const void* sd_prior_scale_v;  /* real [T] */
  /* optional scratch of the split guide step (MIXTURE): when both are non-NULL the pathwise Dirichlet derivative and
     the alpha_pi update run in a second kernel that reads what the first one leaves here                          */
  void* pw;                      /* real [R][G][4]: (pi0, pi1, w0, w1) of every draw (replicate-major: coalesced)    */
  void* dconc;                   /* real [G][4]:    concentration gradients without the pathwise part               */
  /* device i32 [1] or NULL (off): first non-finite step.  A step t that runs with apply_update = 1 and whose loss[t] or any
     ClippedAdam input is NaN / inf does atomicMin(nonfinite_step, t); the caller initialises the word to INT32_MAX.  The update
     of step t is still applied (the clip turns a NaN gradient into -clip): the caller discards what follows t.              */
  int32_t* nonfinite_step;
} BeanSviState;

typedef struct BeanSviNoise {    /* all optional (NULL = draw with Philox) */
  const void* eps_mu;            /* real [T] */
  const void* eps_sd;            /* real [T] */
  const void* pi;                /* real [G][R][2] */
  const void* eps_noise;         /* real [G]  standard-normal draw behind logit_pi_noise (--scale-by-acc) */
  void* eps_out;                 /* real [2][T]    out: the (eps_mu, eps_sd) the step used, or NULL */
  void* pi_out;                  /* real [G][R][2] out: the pi draws the step used, or NULL         */
} BeanSviNoise;

int bean_svi_num_partials(int32_t n_guides, int32_t n_variants);
int bean_svi_run_f32(const BeanScreen* screen, const BeanSviState* state, const BeanSviConfig* cfg,
                     const BeanSviNoise* noise, int32_t first_step, int32_t n_steps, void* stream);
int bean_svi_run_f64(const BeanScreen* screen, const BeanSviState* state, const BeanSviConfig* cfg,
                     const BeanSviNoise* noise, int32_t first_step, int32_t n_steps, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bean_svi_survival_run_{f32,f64}: n_steps complete SVI steps of the SURVIVAL MixtureNormal program on the device.
 *
 * One step = `svi.step(data)` (bean/model/run.py:376-380) for bean/model/survival_model.py:215-424 (MixtureNormalModel) and
 * :651-739 (MixtureNormalGuide): guide draws (`initial_abundance` ~ Dirichlet(q0) over ALL guides per replicate, `mu_targets`,
 * `pi`), the model-only latent `mu_negctrl`, exp(mu t) allele masses, allele mixture, get_alpha + Dirichlet-Multinomial
 * sites of the count layers, the observed `initial_abundance` Dirichlet, `pi` Dirichlet and `control_allele_count`
 * Multinomial on pi exp(mu t_c), Trace_ELBO loss and gradient, ClippedAdam.  Three launches per step: a per-guide kernel,
 * the alpha_pi kernel and the per-variant kernel of bean_svi_run_* (BeanSviState is shared: var_params rows 2, 3 -- the
 * sd site -- are unused, d_guide is [G]).  The screen must be in BEAN_MODE_SURVIVAL.
 *
 * The Dirichlet over all guides needs, per replicate, sum_g gamma[r][g] of the gamma draws and sum_g q0[g]: `sums`.  They
 * are produced on the device (per-warp partials by the guide kernel of the step before, reduced by the last CTA of the
 * per-variant kernel).  With guides SHARDED over GPUs these R + 1 doubles are the one exchange step of the path: call with
 * n_steps = 1 and all-reduce `sums[(t + 1) & 1]` between steps (prime = BEAN_SURV_PRIME_ONLY first, all-reduce
 * `sums[t & 1]`, then prime = BEAN_SURV_PRIME_NONE).
 * ---------------------------------------------------------------------------------------------- */
/* Device-side exchange of those sums (guides sharded over the GPUs of one box, one process per GPU): every rank owns one
 * BeanPeerBuffer in its own GPU memory (bean_peer_alloc) and maps the other ranks' through CUDA IPC (bean_peer_open of the
 * handles, exchanged by the host once).  The last CTA of step t's per-variant kernel stores its rank's partial sums for step
 * t + 1 into slot (t + 1) & 1 of EVERY rank's buffer over NVLink and then raises flag[(t + 1) & 1][rank] = t + 2 there; the
 * guide kernel of step t + 1 waits in its own memory until all `world` flags have arrived and adds the partials in rank order.
 * With `peers` set, bean_svi_survival_run runs n_steps > 1 steps in one call without the host (the first step of a call still
 * reads `sums`, all-reduced by the host after the previous call).  A wait gives up after 30 s (bean_peer_timeouts). */
typedef struct BeanPeerBuffer {
  double vals[2][BEAN_MAX_PEERS][BEAN_PEER_MAX_VALS];
  unsigned long long flag[2][BEAN_MAX_PEERS];
  unsigned long long timeouts;
} BeanPeerBuffer;
typedef struct BeanPeerExchange {
  int32_t world, rank;
  void* buf[BEAN_MAX_PEERS];     /* BeanPeerBuffer of every rank, as mapped in THIS process (buf[rank]: its own) */
} BeanPeerExchange;
int bean_peer_exchange_bytes(void);
int bean_peer_alloc(void** ptr, unsigned char* handle64);        /* cudaMalloc + zero; handle64: 64-byte CUDA IPC handle */
int bean_peer_open(const unsigned char* handle64, void** ptr);   /* map another rank's buffer */
int bean_peer_close(void* ptr);
int bean_peer_free(void* ptr);
int bean_peer_timeouts(const void* own, unsigned long long* out);
int bean_peer_reset_flags(void* own);                           /* zero own flags (a fit set back to an earlier step) */
enum { BEAN_SURV_PRIME_NONE = 0, BEAN_SURV_PRIME_AND_RUN = 1, BEAN_SURV_PRIME_ONLY = 2 };
typedef struct BeanSurvivalState {
  int32_t n_controls;            /* C: control conditions of the reporter Multinomial (BeanSviState.allele_counts is [R][C][G][2]) */
  int32_t prime;                 /* BEAN_SURV_PRIME_*: draw the abundance gammas of `first_step` from the current q0 first
                                    (first call of a run, or after q0 was changed from outside) */
  int64_t n_guides_total;        /* guides of ALL shards (0 = n_guides) */
  const double* control_time;    /* HOST double [C]: normalised timepoints of the control conditions */
  double negctrl_loc, negctrl_scale; /* mu_negctrl ~ Normal(loc, scale) (cli/run.py:258-268; default (0, 0.1)) */
  const void* log_obs;           /* real [R][G] log((X[r][0][g] + 1) / sum over ALL guides) (survival_model.py:306-311) */
  void* q0_u;                    /* real [G] log q0 */
  void* q0_m;
  void* q0_v;
  void* q0_grad;                 /* real [G] out or NULL */
  void* gamma[2];                /* real [R][G] x 2: unnormalised abundance draws of even / odd steps */
  double* sums[2];               /* f64 [R + 1] x 2: sum_g gamma[r][g] (r < R), sum_g q0[g] */
  double* abund_partial;         /* f64 [ceil(G / 128) * 4 + BEAN_SURV_FOLD_ROWS][R + 1] scratch */
  const BeanPeerExchange* peers; /* device-side exchange of `sums` between the ranks of a sharded run, or NULL */
  int32_t* nonfinite_step;       /* as BeanSviState.nonfinite_step (q0 included); NULL: BeanSviState's is used */
} BeanSurvivalState;
typedef struct BeanSurvivalNoise { /* optional injected noise of the survival-only sites (parity runs) */
  const void* eps_negctrl;       /* real [G] standard-normal draw behind mu_negctrl */
  const void* q0;                /* real [R][G] the guide's abundance draw (on the simplex over all guides) */
} BeanSurvivalNoise;
int bean_svi_survival_run_f32(const BeanScreen* screen, const BeanSviState* state, const BeanSurvivalState* survival,
                              const BeanSviConfig* cfg, const BeanSviNoise* noise, const BeanSurvivalNoise* survival_noise,
                              int32_t first_step, int32_t n_steps, void* stream);
int bean_svi_survival_run_f64(const BeanScreen* screen, const BeanSviState* state, const BeanSurvivalState* survival,
                              const BeanSviConfig* cfg, const BeanSviNoise* noise, const BeanSurvivalNoise* survival_noise,
                              int32_t first_step, int32_t n_steps, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bean_row_const_{f32,f64}: the data-only part of each row's count log-pmf, once per screen (the reference recomputes it inside
 * every step: the lgamma(N + 1) - sum lgamma(x + 1) of pyro's DirichletMultinomial.log_prob, model.py:531-547, and the
 * Multinomial coefficient of the reporter counts, model.py:464-474).
 *   row_const[i] = lgamma(N_i + 1) - sum_b lgamma(x[i][b] + 1)  [+ sum_{x > 0} x[i][b] ln(x[i][b] / max(N_i, 1)) with_xlogx]
 *   row_total[i] = N_i = sum_b x[i][b]   (optional)
 * x: real [n_rows][n_bins] (device); log_factorial: f64 [table_size] (device), log_factorial[k] = ln k!: integer entries below
 * table_size are looked up, everything else takes lgamma.  Feeds BeanScreen.row_const and BeanSviConfig.ll_const.
 * ---------------------------------------------------------------------------------------------- */
int bean_row_const_f32(const void* x, int64_t n_rows, int32_t n_bins, int32_t with_xlogx, const double* log_factorial, int32_t table_size,
                       double* row_const, double* row_total, void* stream);
int bean_row_const_f64(const void* x, int64_t n_rows, int32_t n_bins, int32_t with_xlogx, const double* log_factorial, int32_t table_size,
                       double* row_const, double* row_total, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bean_svi_tiling_run_{f32,f64}: n_steps complete SVI steps of the TILING sorting program (MultiMixtureNormal) on the device.
 *
 * One step = `svi.step(data)` (bean/model/run.py:376-380) for bean/model/model.py:550-751 (MultiMixtureNormalModel) and
 * :878-962 (MultiMixtureNormalGuide): per-edit draws `mu_alleles`, `sd_alleles`; allele mean / sd from its edits
 * (`allele_to_edit @ mu_edits`, norm of `allele_to_edit * sd_edits`, wild type (0, 1)); Normal-CDF bin masses per allele with
 * non-existent alleles forced to 0; `pi` ~ Dirichlet over the alleles of a guide; allele mixture; get_alpha +
 * Dirichlet-Multinomial sites; `pi` Dirichlet prior with the epsilon-regularised concentration, guide Dirichlet and
 * `bulk_allele_count` Multinomial under repguide_mask; Trace_ELBO loss and gradient; ClippedAdam.  Three launches per step:
 * per-edit draws, a warp-per-guide kernel with one lane per allele (so n_alleles <= 32: filtered allele tables; wider raw
 * tables stay on the site-kernel engine), and the per-edit kernel that reduces the allele slots over the CSC map.
 * Without --scale-by-acc.  Layouts: alpha_u / alpha_m / alpha_v / allele_mask [G][A]; counts [R][C][G][A]; pi [R][G][A].
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanTilingState {
  const BeanAlleleMap* map;      /* CSR slot -> edits, CSC edit -> slots (bean_allele_gather) */
  int32_t n_controls;            /* C */
  int32_t loss_capacity;
  const uint8_t* allele_mask;    /* u8 [G][A]: 0 = the guide has no such allele */
  const double* pi_a0;           /* f64 [G] */
  const void* counts;            /* real [R][C][G][A] allele_counts_control */
  void* edit_params;             /* real [4][E]: mu_loc, log mu_scale, sd_loc, log sd_scale */
  void* edit_m;
  void* edit_v;
  void* edit_grad;               /* real [4][E] out or NULL */
  void* alpha_u;                 /* real [G][A] log alpha_pi (entries of non-existent alleles are ignored: epsilon) */
  void* alpha_m;
  void* alpha_v;
  void* alpha_grad;              /* real [G][A] out or NULL */
  void* mu_e;                    /* real [E] scratch: this step's draws */
  void* sd_e;
  void* d_slot;                  /* real [2][G * (A - 1)] scratch */
  double* partial;               /* f64 [bean_svi_tiling_num_partials(G, E)] scratch */
  uint32_t* counter;             /* u32 [1], zero before the first call */
  double* loss;                  /* f64 [loss_capacity] */
  const void* mu_prior_loc_v;    /* real [E] per-edit priors or NULL (BeanSviConfig scalars apply) */
  const void* mu_prior_scale_v;
  const void* sd_prior_loc_v;
  const void* sd_prior_scale_v;
  double epsilon;                /* the model's epsilon (1e-5) */
  double pi_tiny;                /* lower clamp of the pi draws = smallest normal number of the dtype pi has in the reference */
  /* Guides sharded over ranks (every rank holds ALL edits: an edit's alleles sit in guides of several shards).  With edit_sum
   * set, BeanSviConfig.phases splits the step: bit 0 = draws + guide kernel + per-edit sums of this shard's allele-slot
   * gradients into edit_sum (no update); the host all-reduces edit_sum over the ranks; bit 1 = priors, guide densities and
   * ClippedAdam of every edit from the reduced sums (identical on every rank) + loss[t].  edit_term_weight scales the
   * per-edit ELBO terms in loss[t] (1 on one rank, 0 on the others, so that the ranks' losses add up). */
  void* edit_sum;                /* real [2][E] or NULL (not sharded) */
  const int32_t* edit_iota;      /* i32 [E + 1] = 0, 1, ..., E (needed with edit_sum) */
  double edit_term_weight;
  int32_t* nonfinite_step;       /* as BeanSviState.nonfinite_step (alpha_pi and the per-edit parameters) */
} BeanTilingState;
typedef struct BeanTilingNoise { /* all optional */
  const void* eps_mu;            /* real [E] */
  const void* eps_sd;            /* real [E] */
  const double* pi;              /* f64 [R][G][A] */
  void* eps_out;                 /* real [2][E] out */
  double* pi_out;                /* f64 [R][G][A] out */
} BeanTilingNoise;
int bean_svi_tiling_num_partials(int32_t n_guides, int32_t n_edits);
int bean_svi_tiling_run_f32(const BeanScreen* screen, const BeanTilingState* state, const BeanSviConfig* cfg, const BeanTilingNoise* noise,
                            int32_t first_step, int32_t n_steps, void* stream);
int bean_svi_tiling_run_f64(const BeanScreen* screen, const BeanTilingState* state, const BeanSviConfig* cfg, const BeanTilingNoise* noise,
                            int32_t first_step, int32_t n_steps, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Editing-rate sites of the MultiMixtureNormal (tiling) and survival MixtureNormal programs: forward value and local
 * gradients in one launch.  Replaces the op chains
 *   pyro.sample("pi", Dirichlet(pi_a_scaled))            model.py:652-661, survival_model.py:313-322 / :515-524
 *   pyro.sample("control_allele_count", Multinomial(probs=pi * exp(mu t_c)), obs=allele_counts_control)
 *                                                         model.py:662-670, survival_model.py:323-346 / :525-548
 *   guide: pyro.sample("pi", Dirichlet(...))              model.py:938-950, survival_model.py:699-712 / :822-833
 * and their autograd backward (torch.distributions.Dirichlet / Multinomial.log_prob).
 *   V = sum m[r,g] log Dir(pi[r,g,:]; conc_model[g,:]) + sum m[r,g] [sum_a x[r,c,g,a] log clamp(q_a / sum q, eps, 1 - eps)]
 *       - sum m'[r,g] log Dir(pi[r,g,:]; conc_guide[g,:]),   q_a = pi[r,g,a] exp(growth[g,a] control_time[c])
 *   m = rep_guide_mask; m' = m if mask_guide_site else 1.  The data-only Multinomial constant is left to the caller.
 * in : conc_guide, conc_model real [G][A]; pi real [R][G][A]; counts real [R][C][G][A]; rep_guide_mask u8 [R][G];
 *      growth real [G][A] or NULL (q = pi); control_time HOST double [C] (needed with growth)
 * out: partial double [G] (V = sum of it); d_conc_guide, d_conc_model real [G][A]; d_pi real [R][G][A];
 *      d_growth real [G][A] (NULL iff growth is NULL) -- all d(V)/d(input)
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanPiSitesArgs {
  int32_t n_guides, n_reps, n_alleles, n_controls;
  int32_t mask_guide_site;
  const void* conc_guide;
  const void* conc_model;
  const void* pi;
  const void* counts;
  const uint8_t* rep_guide_mask;
  const void* growth;
  const double* control_time;
  double prob_eps;             /* eps of the dtype the reference evaluates the Multinomial probabilities in */
  double* partial;
  void* d_conc_guide;
  void* d_conc_model;
  void* d_pi;
  void* d_growth;
} BeanPiSitesArgs;
int bean_pi_sites_f32(const BeanPiSitesArgs* args, void* stream);
int bean_pi_sites_f64(const BeanPiSitesArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Per-variant / per-edit latent sites `mu_targets` (and `sd_targets`) of the programs that run on torch autograd around
 * bean_ll_*: reparameterised draws, prior and guide log-densities, closed-form gradients.
 * Replaces  guide: pyro.sample("mu_targets", Normal(mu_loc, mu_scale)), pyro.sample("sd_targets", LogNormal(sd_loc, sd_scale))
 *                  (model.py:893-921, survival_model.py:640-652 / :770-789)
 *           model: pyro.sample("mu_targets", Laplace(0, 1) | Normal(prior)), pyro.sample("sd_targets", LogNormal(prior))
 *                  (model.py:579-610, survival_model.py:37-56 / :246-274 / :440-468)
 * and their autograd backward.  Forward: mu = mu_loc + exp(mu_log_scale) eps_mu, sd = exp(sd_loc + exp(sd_log_scale) eps_sd),
 *   V = sum_i [log p(mu_i) - log q(mu_i)] + [log p(sd_i) - log q(sd_i)]  (what the sites add to the ELBO),
 *   dv[4][n] = dV/d(mu_loc, mu_log_scale, sd_loc, sd_log_scale) including the path through the draws.
 * Backward (bean_latent_sites_grad_*): grad[4][n] = d L/d(the four parameters) from the upstream d L/d(mu, sd, V).
 * Prior hyper-parameters: scalar, or per element where the *_v pointer is non-NULL (`bean build-prior` tensors).
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanLatentSitesArgs {
  int64_t n;
  int32_t has_sd;              /* 0: survival programs (no sd_targets site) */
  int32_t mu_prior_normal;     /* 0: Laplace(0, 1); 1: Normal(mu_prior_loc, mu_prior_scale) */
  const void* mu_loc;          /* real [n] */
  const void* mu_log_scale;    /* real [n] */
  const void* sd_loc;          /* real [n] or NULL */
  const void* sd_log_scale;    /* real [n] or NULL */
  const void* eps_mu;          /* real [n] standard-normal noise */
  const void* eps_sd;          /* real [n] or NULL */
  double mu_prior_loc, mu_prior_scale, sd_prior_loc, sd_prior_scale;
  const void* mu_prior_loc_v;  /* real [n] or NULL */
  const void* mu_prior_scale_v;
  const void* sd_prior_loc_v;
  const void* sd_prior_scale_v;
  void* mu;                    /* out real [n] */
  void* sd;                    /* out real [n] or NULL */
  double* partial;             /* out f64 [bean_latent_sites_num_partials(n)], V = sum */
  void* dv;                    /* out real [4][n] (rows 2, 3 untouched without sd) */
} BeanLatentSitesArgs;
typedef struct BeanLatentSitesGradArgs {
  int64_t n;
  int32_t has_sd;
  const void* mu_log_scale;
  const void* sd_log_scale;
  const void* eps_mu;
  const void* eps_sd;
  const void* sd;              /* the forward's sd draws */
  const void* dv;              /* the forward's dv */
  const void* g_mu;            /* real [n] upstream d L/d mu, or NULL (= 0) */
  const void* g_sd;            /* real [n] upstream d L/d sd, or NULL */
  const void* g_v;             /* real [1] DEVICE scalar d L/d V, or NULL */
  void* grad;                  /* out real [4][n] */
} BeanLatentSitesGradArgs;
int bean_latent_sites_num_partials(int64_t n);
int bean_latent_sites_f32(const BeanLatentSitesArgs* args, void* stream);
int bean_latent_sites_f64(const BeanLatentSitesArgs* args, void* stream);
int bean_latent_sites_grad_f32(const BeanLatentSitesGradArgs* args, void* stream);
int bean_latent_sites_grad_f64(const BeanLatentSitesGradArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * pyro.optim.ClippedAdam on every parameter tensor of a model in one launch.
 * Replaces the optimiser half of `svi.step` (bean/model/run.py:368-380: ClippedAdam({"lr", "lrd", "clip_norm": 10}))
 * for the models whose ELBO is assembled by torch autograd around `bean_ll_*` (tiling, survival, covariates).
 * Per element of the unconstrained tensors (SURVEY App. A.6):
 *   g = clamp(grad, -clip, clip); m = b1 m + (1 - b1) g; v = b2 v + (1 - b2) g^2;
 *   theta -= step_sizes[min(*step, n_steps - 1)] * m / (sqrt(v) + eps)
 * with step_sizes[t] = lr lrd^(t+1) sqrt(1 - b2^(t+1)) / (1 - b1^(t+1)) precomputed by the caller.  `step_sizes` and
 * `step` are DEVICE pointers: nothing about the launch depends on the host, so it can be captured in a CUDA graph.
 * ---------------------------------------------------------------------------------------------- */
#define BEAN_ADAM_MAX_TENSORS 16
typedef struct BeanAdamTensor {
  void* theta;        /* real [n] unconstrained parameter, updated in place */
  const void* grad;   /* real [n] d(-ELBO)/d theta                          */
  void* m;            /* real [n] first-moment state                        */
  void* v;            /* real [n] second-moment state                       */
  int64_t n;
} BeanAdamTensor;
typedef struct BeanAdamArgs {
  int32_t n_tensors;
  BeanAdamTensor tensors[BEAN_ADAM_MAX_TENSORS];
  const double* step_sizes;  /* device f64 [n_steps] */
  const int64_t* step;       /* device i64 [1]: 0-based index of this step */
  int64_t n_steps;
  double beta1, beta2, eps, clip;
  /* first non-finite step, as BeanSviState.nonfinite_step: step *step is recorded when a gradient is NaN / inf or, with
     `loss` set, when loss[*step] is (the caller writes it before this launch).  NULL: off                          */
  const double* loss;        /* device f64 [n_steps] or NULL */
  int32_t* nonfinite_step;   /* device i32 [1] or NULL */
} BeanAdamArgs;
int bean_clipped_adam_f32(const BeanAdamArgs* args, void* stream);
int bean_clipped_adam_f64(const BeanAdamArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * bean_dirichlet_rsample_{f32,f64} / bean_dirichlet_rsample_grad_{f32,f64}: reparameterised draws of the editing-rate
 * site `pi` and their pathwise derivative.
 * Replaces  dist.Dirichlet(concentration).rsample()  in the guides of the programs that run on torch autograd around
 * bean_ll_* (bean/model/model.py:942-950 MultiMixtureNormalGuide; bean/model/survival_model.py:699-712, :822-833), i.e.
 * torch._sample_dirichlet forward and torch._dirichlet_grad (`_Dirichlet_backward`) backward:
 *   forward : x[r][g][:] ~ Dirichlet(conc[g][:])  (gamma draws normalised, clamped to [tiny, 1 - eps/2])
 *   backward: d_conc[g][a] = sum_r D(x[r][g][a]; conc[g][a], sum_b conc[g][b]) * (grad_x[r][g][a] - sum_b x[r][g][b] grad_x[r][g][b])
 * Counter-based noise (Philox4x32-10 keyed by `seed`; counter = (guide_offset + g, r | a << 8, step, site)): reproducible,
 * independent of launch geometry and of how guides are sharded over GPUs.  `step` is a DEVICE pointer (or NULL: then
 * `step_value` is used), so the launch can be captured in a CUDA graph whose replays advance the step on the device.
 * ---------------------------------------------------------------------------------------------- */
typedef struct BeanDirichletArgs {
  int32_t n_guides, n_reps, n_alleles;
  uint32_t site;             /* distinguishes several Dirichlet sites of one program (separate noise streams) */
  const void* conc;          /* real [G][A] concentrations (> 0) */
  void* x;                   /* real [R][G][A]: out (forward), in (backward) */
  const void* grad_x;        /* real [R][G][A] upstream d L / d x (backward only) */
  void* d_conc;              /* real [G][A] out (backward only) */
  uint64_t seed;
  uint32_t guide_offset;     /* global index of this shard's first guide */
  const int64_t* step;       /* device i64 [1] or NULL */
  int64_t step_value;
} BeanDirichletArgs;
int bean_dirichlet_rsample_f32(const BeanDirichletArgs* args, void* stream);
int bean_dirichlet_rsample_f64(const BeanDirichletArgs* args, void* stream);
int bean_dirichlet_rsample_grad_f32(const BeanDirichletArgs* args, void* stream);
int bean_dirichlet_rsample_grad_f64(const BeanDirichletArgs* args, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Measurement aid (no reference counterpart): register-only evaluation of the Dirichlet-Multinomial row
 * maths of `n_rows_per_guide` rows of `n_bins` bins for `n_guides` guides -- the empirical FP32/SFU ceiling
 * bench.py quotes next to the HBM roofline (SURVEY 8d).  out: float [ceil(n_guides / 128)] (checksum sink).
 * ---------------------------------------------------------------------------------------------- */
int bean_row_ceiling_f32(int32_t n_guides, int32_t n_rows_per_guide, int32_t n_bins, void* out, void* stream);
/* the same maths (4 bins) with one lane per (row, bin) cell and 4-lane shuffle reductions -- the mapping of the north_star,
 * timed against the thread-per-guide mapping above; out: float [4 * number of SMs] */
int bean_row_ceiling_lanes_f32(int32_t n_guides, int32_t n_rows_per_guide, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BEAN_B200_H_ */
