// bean_svi_shared.cuh -- what the fused SVI steps of the sorting (bean_svi.cu) and survival (bean_svi_survival.cu) programs share:
// the kernel argument block, ClippedAdam, the variant draw, the alpha_pi kernel (pathwise Dirichlet derivative + update) and
// the per-variant kernel (segmented reduction, prior / entropy terms, update, loss).
#pragma once
#include "bean_common.cuh"
#include "bean_math.cuh"
#include "bean_rng.cuh"
#include "bean_row.cuh"

#define BEAN_SURV_MAX_CTRL 4

namespace bean {

constexpr int SVI_THREADS = 128;
constexpr int SVI_MIN_CTAS = 4;        // fused guide step: <= 128 registers, 16 warps/SM (more CTAs measured +-2 %)
#ifndef BEAN_GUIDE_MIN_CTAS
#define BEAN_GUIDE_MIN_CTAS 7  // with the cp.async-staged rows: 6: 0.4243, 7: 0.4132, 8: 0.4235 ms per launch at c5 (profiles/r2h_phase_times.jsonl)
#endif
constexpr int SVI_MIN_CTAS_SPLIT = BEAN_GUIDE_MIN_CTAS;  // split guide step and the Normal models: 72 registers, 28 warps/SM
                                       // (MixtureNormal 4: 1.17, 6: 1.11, 8: 1.08 ms/step; Normal 4: 0.64, 8: 0.58; final kernel 7: 0.650, 8: 0.640 ms)
// ELBO partials are per WARP (no CTA barrier: per-guide cost varies with the Dirichlet-gradient regime of its draws,
// so the warps of a CTA finish far apart).  1-warp CTAs were tried and were 4 % slower.
constexpr int SVI_WARP = 32;
#ifndef BEAN_VAR_THREADS
#define BEAN_VAR_THREADS 256
#endif
constexpr int VAR_THREADS = BEAN_VAR_THREADS;
constexpr int VAR_PER_CTA = VAR_THREADS;  // one thread per variant

template <typename real>
struct SviParams {
  int G, R, B, L, T;
  int mixture, sd_is_sqrt, mu_prior_normal, apply_update, fit_noise;
  uint32_t step, guide_offset, variant_offset;
  uint64_t seed;
  PhiloxKeys rk;  // Philox round keys of `seed` (philox_round_keys)
  real mask_thres;
  // screen
  const real* x;
  const real* a0;
  const uint8_t* row_mask;
  const int32_t* guide_variant;
  const int32_t* variant_ptr;
  const real* allele_counts;
  const real* pi_a0;
  // parameters + Adam state
  real* var_params;
  real* var_m;
  real* var_v;
  real* alpha_u;
  real* alpha_m;
  real* alpha_v;
  const real* acc_k;
  real* noise_u;
  real* noise_m;
  real* noise_v;
  real* noise_grad;
  // scratch / outputs
  real* d_guide;
  real* var_grad;
  real* alpha_grad;
  real* pw;      // split path: [R][G][4] = (pi0, pi1, w0, w1) of every draw, written by the guide kernel
  real* dconc;   // split path: [G][4]    = (dcm0, dcm1, dcg0, dcg1) without the pathwise part
  double* partial;
  uint32_t* counter;
  double* loss;
  int32_t* nonfinite;  // first non-finite step (include/bean_b200.h: BeanSviState.nonfinite_step) or NULL
  int n_partial_guide, n_partial_var;
  // injected noise (parity runs)
  const real* eps_mu;
  const real* eps_sd;
  const real* pi_in;
  const real* eps_noise;
  real* eps_out;
  real* pi_out;
  // priors / optimiser scalars of this step
  real mu_prior_loc, mu_prior_scale, sd_prior_loc, sd_prior_scale;
  const real* mu_prior_loc_v;
  const real* mu_prior_scale_v;
  const real* sd_prior_loc_v;
  const real* sd_prior_scale_v;
  real step_size, beta1, beta2, adam_eps, clip, prob_eps;
  double ll_const;
  real p_wt[BEAN_MAX_BINS];  // bin masses of the wild-type allele N(0, 1)
  SampleTables<real> t;
  // ---- survival MixtureNormal step (bean_svi_survival.cu); has_sd = 0 there (no sd_targets site) ----
  int has_sd;
  int n_ctrl;                           // control conditions of the reporter Multinomial
  real t_ctrl[BEAN_SURV_MAX_CTRL];      // their (normalised) timepoints
  real negctrl_loc, negctrl_scale;      // mu_negctrl ~ Normal(loc, scale): parameter-free prior draw per guide
  double n_guides_total;                // guides of ALL shards (the abundance Dirichlet spans the whole library)
  const real* log_obs;                  // [R][G] log of the observed initial abundance
  real* q0_u; real* q0_m; real* q0_v; real* q0_grad;   // [G] log q0 + Adam state (+ gradient out)
  const real* gamma_cur;                // [R][G] unnormalised gamma draws of THIS step's abundance sample
  real* gamma_next;                     // [R][G] ... of the next step's (drawn after the q0 update)
  const double* sums_cur;               // [R + 1] sum_g gamma[r][g] (r < R), sum_g q0[g]
  double* sums_next;
  double* abund_partial;                // [warps][R + 1] per-warp partial sums behind sums_next
  int n_abund_partial;
  // device-side exchange of the sums between the ranks of a sharded run (include/bean_b200.h: BeanPeerBuffer)
  int peer_world, peer_rank;            // peer_world <= 1: none
  int peer_consume;                     // this step's guide kernel takes its sums from the exchange buffer, not from sums_cur
  BeanPeerBuffer* peer_buf[BEAN_MAX_PEERS];
  const real* eps_negctrl;              // injected noise (parity runs)
  const real* q0_in;                    // [R][G] injected abundance draw (already normalised)
  // ---- tiling step (bean_svi_tiling.cu): the "variants" are edits, whose gradient entries sit in allele slots ----
  const int32_t* gather_idx;            // [nnz] CSC: d_guide index of the j-th entry of a segment (NULL: j itself)
  real* seg_sum_out;                    // [2][T] sharded tiling step: write the segment sums here and do nothing else
  int variant_terms_off;                // the per-variant ELBO terms stay out of loss[t] (another rank counts them)
  int dsd_times_sd;                     // d_guide's second row holds d/d(sd_allele) / sd_allele: multiply the sum by the edit's sd
};

// Step `step` is non-finite: keep the smallest such step in *word (atomicMin; the caller initialised it to INT32_MAX).  Skips
// the atomic while the word already holds this step or an earlier one.
__device__ __forceinline__ void record_nonfinite(int32_t* word, uint32_t step) {
  if (*(volatile int32_t*)word > (int32_t)step) atomicMin(word, (int32_t)step);
}
// The same from a warp: every lane of `mask` calls with its own verdict, one lane of a warp that has any bad one records.
__device__ __forceinline__ void note_nonfinite(int32_t* word, uint32_t step, unsigned mask, bool bad) {
  if (word == nullptr) return;  // kernel-uniform
  const unsigned any = __ballot_sync(mask, bad);
  if (any != 0u && (int)(threadIdx.x & 31u) == __ffs(any) - 1) record_nonfinite(word, step);
}

// pyro.optim.ClippedAdam on one unconstrained scalar (SURVEY App. A.6); step_size carries
// lr_t * sqrt(1 - beta2^t) / (1 - beta1^t).  `bad` collects whether an input was NaN / inf (the clip below maps NaN to -clip).
template <typename real>
__device__ __forceinline__ void clipped_adam(const SviParams<real>& p, real grad, real& theta, real& m, real& v, bool& bad) {
  bad |= !isfinite(grad);
  const real g = Num<real>::fmin(Num<real>::fmax(grad, -p.clip), p.clip);
  m = p.beta1 * m + (real(1) - p.beta1) * g;
  v = p.beta2 * v + (real(1) - p.beta2) * g * g;
  theta -= p.step_size * m / (Num<real>::sqrt(v) + p.adam_eps);
}

// reparameterised draw of the variant's (mu, sd) -- recomputed wherever needed instead of stored
template <typename real>
__device__ __forceinline__ void variant_draw(const SviParams<real>& p, int v, real& mu_t, real& sd_t, real& eps_mu,
                                             real& eps_sd, real& mu_scale, real& sd_scale, real& log_sd) {
  const real mu_loc = p.var_params[v];
  mu_scale = Num<real>::exp(p.var_params[p.T + v]);
  const real sd_loc = p.var_params[2 * p.T + v];
  sd_scale = Num<real>::exp(p.var_params[3 * p.T + v]);
  if (p.eps_mu) {
    eps_mu = p.eps_mu[v];
    eps_sd = p.eps_sd ? p.eps_sd[v] : real(0);
  } else {
    float e0, e1;
    variant_noise(p.seed, (uint32_t)v + p.variant_offset, p.step, e0, e1);
    eps_mu = real(e0);
    eps_sd = real(e1);
  }
  mu_t = mu_loc + mu_scale * eps_mu;   // Normal(mu_loc, mu_scale).rsample()          model.py:810
  log_sd = sd_loc + sd_scale * eps_sd;  // LogNormal(sd_loc, sd_scale).rsample()       model.py:811
  sd_t = Num<real>::exp(log_sd);
}

// concentration gradients -> log alpha_pi gradient -> ClippedAdam (alpha_pi is per guide)
template <typename real>
__device__ __forceinline__ void alpha_update(const SviParams<real>& p, int g, real al0, real al1, real pa0, real cm0, real cm1,
                                             real dcm0, real dcm1, real dcg0, real dcg1, bool& bad) {
  const real eps = real(1e-5);
  const real asum = al0 + al1;
  // clamp(min) passes the gradient where its input >= 1e-5
  const real dC0 = dcm0 + (cm0 >= eps ? dcg0 : real(0));
  const real dC1 = dcm1 + (cm1 >= eps ? dcg1 : real(0));
  const real k = pa0 / (asum * asum);
  const real dal0 = k * (dC0 * (asum - al0) - dC1 * al1);
  const real dal1 = k * (dC1 * (asum - al1) - dC0 * al0);
  const real gl0 = -dal0 * al0, gl1 = -dal1 * al1;  // loss = -ELBO, unconstrained (log) space
  if (p.alpha_grad) {
    p.alpha_grad[2 * (size_t)g] = gl0;
    p.alpha_grad[2 * (size_t)g + 1] = gl1;
  }
  if (p.apply_update) {
    real th0 = p.alpha_u[2 * (size_t)g], th1 = p.alpha_u[2 * (size_t)g + 1];
    real m0 = p.alpha_m[2 * (size_t)g], m1 = p.alpha_m[2 * (size_t)g + 1];
    real v0 = p.alpha_v[2 * (size_t)g], v1 = p.alpha_v[2 * (size_t)g + 1];
    clipped_adam(p, gl0, th0, m0, v0, bad);
    clipped_adam(p, gl1, th1, m1, v1, bad);
    p.alpha_u[2 * (size_t)g] = th0; p.alpha_u[2 * (size_t)g + 1] = th1;
    p.alpha_m[2 * (size_t)g] = m0;  p.alpha_m[2 * (size_t)g + 1] = m1;
    p.alpha_v[2 * (size_t)g] = v0;  p.alpha_v[2 * (size_t)g + 1] = v1;
  }
}

template <typename real> struct SaddleOf;
template <> struct SaddleOf<float> { typedef SaddlePairF type; };
template <> struct SaddleOf<double> { typedef SaddlePair type; };

// Programmatic dependent launch (sm_90+): a kernel launched with `launch_after` may have its CTAs scheduled while the kernel
// before it on the stream is still draining; it must call `grid_dependency_wait()` before it touches anything that kernel wrote
// (here: first thing).  What this buys is the launch latency and ramp-up of three dependent kernels per step -- a few
// microseconds each, which is what a step is made of once a screen is split over eight GPUs.
#ifndef BEAN_NO_PDL
#define BEAN_PDL 1
#endif
__device__ __forceinline__ void grid_dependency_wait() {
#ifdef BEAN_PDL
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}
template <typename Kernel, typename Params>
static inline void launch_after(Kernel kernel, int grid, int block, cudaStream_t st, const Params& p) {
#ifdef BEAN_PDL
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = 0; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, p);
#else
  kernel<<<grid, block, 0, st>>>(p);
#endif
}

// Second half of the split guide step: pathwise Dirichlet derivative of every draw (saddle-point pairs in place, the other
// regimes through the per-warp queue), alpha_pi gradient and its ClippedAdam update.  One thread per guide.
// one warp per CTA: the work per draw differs by regime, and small CTAs hand their SM slot on as soon as their own 32 guides are
// done (128 / 64 / 32 threads: 0.161 / 0.160 / 0.155 ms at c5, 0.057 / 0.055 / 0.054 at a quarter of it; profiles/r2p_variants.jsonl)
#ifndef BEAN_ALPHA_THREADS
#define BEAN_ALPHA_THREADS 32
#endif
constexpr int ALPHA_THREADS = BEAN_ALPHA_THREADS;
#ifndef BEAN_ALPHA_MIN_CTAS
#define BEAN_ALPHA_MIN_CTAS (768 / BEAN_ALPHA_THREADS)
#endif
template <typename real>
__global__ void __launch_bounds__(ALPHA_THREADS, BEAN_ALPHA_MIN_CTAS) svi_alpha_kernel(const SviParams<real> p) {
  __shared__ TailQueue<real> tail_queues[ALPHA_THREADS / SVI_WARP];
  __shared__ float s_near_mean[6][ALPHA_THREADS];
  grid_dependency_wait();
  const int g = blockIdx.x * ALPHA_THREADS + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const real eps = real(1e-5);
  const unsigned wmask = __ballot_sync(0xffffffffu, g < p.G);
  if (g >= p.G) return;
  TailQueue<real>& tq = tail_queues[threadIdx.x / SVI_WARP];
  const real al0 = Num<real>::exp(p.alpha_u[2 * (size_t)g]), al1 = Num<real>::exp(p.alpha_u[2 * (size_t)g + 1]);
  const real asum = al0 + al1, pa0 = p.pi_a0[g];
  const real cm0 = al0 / asum * pa0, cm1 = al1 / asum * pa0;
  const real cg0 = Num<real>::fmax(cm0, eps), cg1 = Num<real>::fmax(cm1, eps);
  const typename Vec4<real>::type dc = reinterpret_cast<const typename Vec4<real>::type*>(p.dconc)[g];
  real dcg0 = dc.z, dcg1 = dc.w;
  int n_tail = 0;
  // saddle-point regime: float kernels use the cancellation-free single-precision form, double kernels torch's expression
  typename SaddleOf<real>::type sp;
  sp.init(cg0, cg1);
  sp.prepare_near_mean(&s_near_mean[0][threadIdx.x], ALPHA_THREADS);
  const typename Vec4<real>::type* pw = reinterpret_cast<const typename Vec4<real>::type*>(p.pw) + g;
  typename Vec4<real>::type nxt = pw[0];
  for (int r = 0; r < p.R; ++r) {
    const typename Vec4<real>::type rec = nxt;
    if (r + 1 < p.R) nxt = pw[(size_t)(r + 1) * p.G];  // the next draw's record is in flight while this one is evaluated
    const bool saddle = dirichlet_pair_is_saddle((double)rec.x, (double)rec.y, (double)cg0, (double)cg1);
    if (saddle) {
      real dg0, dg1;
      sp.eval(rec.x, rec.y, dg0, dg1);
      dcg0 += dg0 * rec.z;
      dcg1 += dg1 * rec.w;
    }
    n_tail = tail_queue_push(tq, n_tail, wmask, lane, !saddle, rec.x, rec.y, cg0, cg1, rec.z, rec.w);
    if (n_tail >= 32) {
      tail_queue_flush(tq, n_tail, wmask, lane, dcg0, dcg1);
      n_tail = 0;
    }
  }
  if (n_tail > 0) tail_queue_flush(tq, n_tail, wmask, lane, dcg0, dcg1);
  bool bad = false;
  alpha_update(p, g, al0, al1, pa0, cm0, cm1, dc.x, dc.y, dcg0, dcg1, bad);
  note_nonfinite(p.nonfinite, p.step, wmask, bad);
}

// This step's library-wide sums into shared memory: from `sums_cur` (single GPU, or the first step of a call: all-reduced by the
// host), or from the exchange buffer in this rank's own memory once the flags of all ranks for this step have arrived -- added in
// rank order (deterministic).  Every thread of the CTA calls; n_vals <= BEAN_PEER_MAX_VALS.
#ifndef BEAN_PEER_TIMEOUT_NS
#define BEAN_PEER_TIMEOUT_NS 30000000000ull
#endif
template <typename real>
__device__ __forceinline__ void load_library_sums(const SviParams<real>& p, int n_vals, double* s_sums) {
  if (p.peer_world > 1 && p.peer_consume) {
    BeanPeerBuffer* own = p.peer_buf[p.peer_rank];
    const int slot = (int)(p.step & 1u);
    if ((int)threadIdx.x < p.peer_world) {
      volatile unsigned long long* f = &own->flag[slot][threadIdx.x];
      const unsigned long long want = (unsigned long long)p.step + 1ull;
      unsigned long long t0 = 0ull;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      volatile unsigned long long* gave_up = &own->timeouts;
      while (*f < want && *gave_up == 0ull) {  // once one wait has timed out nobody waits again: the run is lost, not hung
        __nanosleep(200);
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > BEAN_PEER_TIMEOUT_NS) {  // a peer died or never ran this step: give up (counted; the host reports it)
          atomicAdd(&own->timeouts, 1ull);
          break;
        }
      }
      __threadfence_system();
    }
    __syncthreads();
    if ((int)threadIdx.x < n_vals) {
      double a = 0.0;
      for (int k = 0; k < p.peer_world; ++k) a += *(volatile const double*)&own->vals[slot][k][threadIdx.x];
      s_sums[threadIdx.x] = a;
    }
  } else if ((int)threadIdx.x < n_vals) {
    s_sums[threadIdx.x] = p.sums_cur[threadIdx.x];
  }
  __syncthreads();
}

// Column sums of rows first, first + stride, ... (< n_rows) of a row-major [n_rows][C] array of doubles, C <= VAR_THREADS, by
// one CTA of VAR_THREADS threads: thread t accumulates column t % C over every (VAR_THREADS / C)-th row of the set, the partial
// sums meet in shared memory in a fixed order.  Every thread calls; thread j < C receives column j.
__device__ __forceinline__ double column_sums(const double* a, int n_rows, int C, int first, int stride, double* s_cs) {
  const int slots = VAR_THREADS / C, col = threadIdx.x % C, slot = threadIdx.x / C;
  double acc = 0.0;
  if (slot < slots)
    for (long long row = first + (long long)slot * stride; row < n_rows; row += (long long)slots * stride) acc += __ldcg(a + row * C + col);
  s_cs[threadIdx.x] = acc;
  __syncthreads();
  double tot = 0.0;
  if ((int)threadIdx.x < C)
    for (int m = 0; m < slots; ++m) tot += s_cs[m * C + threadIdx.x];
  __syncthreads();
  return tot;
}

// One step's per-variant work, ONE THREAD PER VARIANT: the segmented sum of the guides' (d mu, d sd) over the variant's guide
// range, then the draw, priors, entropy and ClippedAdam of the variant.  A variant has a handful of guides (5 at c5), whose
// gradients sit in L2: one thread walking them in order beats 8 cooperating lanes by 3 x (0.042 -> 0.013 ms at c5, measured
// for 8 / 4 / 2 / 1 lanes: profiles/r2aa_, r2ab_variants.jsonl) because every lane then also has a variant to update.  Segments
// longer than VAR_SHORT_SEG (a variant with hundreds of guides; the tiling step's edits shared by many alleles) are summed by
// the whole warp instead, strided and tree-reduced -- both orders are fixed, the result is deterministic.  Every CTA also folds
// its slice of the guide kernel's ELBO partials into its own partial, so the last CTA's fixed-order reduction reads
// n_partial_var numbers, not n_partial_guide + n_partial_var.
constexpr int VAR_SHORT_SEG = 32;
template <typename real>
__global__ void __launch_bounds__(VAR_THREADS) svi_variant_kernel(const SviParams<real> p) {
  __shared__ double red[32];
  __shared__ bool is_last;
  __shared__ double s_cs[VAR_THREADS];
  grid_dependency_wait();
  const int v = blockIdx.x * VAR_PER_CTA + threadIdx.x;
  const int lane = threadIdx.x & 31;
  real dmu = real(0), dsd = real(0);
  {
    int beg = 0, end = 0;
    if (v < p.T) {
      beg = p.variant_ptr[v];
      end = p.variant_ptr[v + 1];
    }
    const bool is_long = end - beg > VAR_SHORT_SEG;
    if (!is_long) {
      for (int j = beg; j < end; ++j) {
        const int k = p.gather_idx ? p.gather_idx[j] : j;
        dmu += p.d_guide[k];
        if (p.has_sd) dsd += p.d_guide[(size_t)p.G + k];
      }
    }
    unsigned todo = __ballot_sync(0xffffffffu, is_long);
    while (todo) {  // warp-uniform
      const int src = __ffs(todo) - 1;
      todo &= todo - 1u;
      const int b0 = __shfl_sync(0xffffffffu, beg, src), e0 = __shfl_sync(0xffffffffu, end, src);
      real a = real(0), c = real(0);
      for (int j = b0 + lane; j < e0; j += 32) {
        const int k = p.gather_idx ? p.gather_idx[j] : j;
        a += p.d_guide[k];
        if (p.has_sd) c += p.d_guide[(size_t)p.G + k];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
      }
      if (lane == src) {
        dmu = a;
        dsd = c;
      }
    }
    if (p.seg_sum_out && v < p.T) {
      p.seg_sum_out[v] = dmu;
      p.seg_sum_out[(size_t)p.T + v] = dsd;
    }
  }
  if (p.seg_sum_out) return;  // reduce-only launch (grid-uniform)
  // this CTA's slice of the guide kernel's partials (fixed assignment: deterministic)
  double elbo = 0.0;
  for (int i = blockIdx.x * VAR_THREADS + threadIdx.x; i < p.n_partial_guide; i += gridDim.x * VAR_THREADS) elbo += p.partial[i];
  bool bad = false;
  if (v < p.T) {
    real mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, y;
    variant_draw(p, v, mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, y);
    if (p.eps_out) {
      p.eps_out[v] = e_mu;
      p.eps_out[p.T + v] = e_sd;
    }
    const real HL2PI = real(0.91893853320467274178);
    // model priors (model.py:41-65 / :405-428; ControlNormal :178-179)
    real lp_mu, dlp_mu;
    if (p.mu_prior_normal) {
      const real loc = p.mu_prior_loc_v ? p.mu_prior_loc_v[v] : p.mu_prior_loc;
      const real scale = p.mu_prior_scale_v ? p.mu_prior_scale_v[v] : p.mu_prior_scale;
      const real z = (mu_t - loc) / scale;
      lp_mu = -Num<real>::log(scale) - HL2PI - real(0.5) * z * z;
      dlp_mu = -z / scale;
    } else {  // Laplace(0, 1)
      lp_mu = -real(0.69314718055994530942) - (mu_t < real(0) ? -mu_t : mu_t);
      dlp_mu = mu_t > real(0) ? real(-1) : (mu_t < real(0) ? real(1) : real(0));
    }
    const real sloc = p.sd_prior_loc_v ? p.sd_prior_loc_v[v] : p.sd_prior_loc;
    const real sscale = p.sd_prior_scale_v ? p.sd_prior_scale_v[v] : p.sd_prior_scale;
    const real zs = (y - sloc) / sscale;
    const real lp_sd = -y - Num<real>::log(sscale) - HL2PI - real(0.5) * zs * zs;
    const real dlp_sd = (-real(1) - zs / sscale) / sd_t;
    // guide densities (entropy side)
    const real lq_mu = -Num<real>::log(mu_scale) - HL2PI - real(0.5) * e_mu * e_mu;
    const real lq_sd = -y - Num<real>::log(sd_scale) - HL2PI - real(0.5) * e_sd * e_sd;
    if (!p.variant_terms_off) elbo += (double)lp_mu - (double)lq_mu + (p.has_sd ? (double)lp_sd - (double)lq_sd : 0.0);
    if (p.dsd_times_sd) dsd *= sd_t;  // sd_allele = sqrt(sum sd_edit^2): d sd_allele / d sd_edit = sd_edit / sd_allele
    const real dE_mu = dmu + dlp_mu;
    const real dE_sd = dsd + dlp_sd;
    // gradient of the LOSS (-ELBO) w.r.t. the unconstrained parameters
    real grad[4];
    grad[0] = -dE_mu;
    grad[1] = -(dE_mu * e_mu * mu_scale + real(1));
    grad[2] = -(dE_sd * sd_t + real(1));
    grad[3] = -((dE_sd * sd_t * e_sd + e_sd) * sd_scale + real(1));
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (k >= 2 && !p.has_sd) break;
      const size_t i = (size_t)k * p.T + v;
      if (p.var_grad) p.var_grad[i] = grad[k];
      if (p.apply_update) {
        real th = p.var_params[i], m = p.var_m[i], vv = p.var_v[i];
        clipped_adam(p, grad[k], th, m, vv, bad);
        p.var_params[i] = th;
        p.var_m[i] = m;
        p.var_v[i] = vv;
      }
    }
  }
  // survival: the library-wide sums of the NEXT step's abundance draw (sum_g gamma[r][g], sum_g q0[g]) from the per-warp
  // partials [n_abund_partial][R + 1] the guide kernel left, in two fixed-order levels: CTA b < M folds rows b, b + M, ...
  // into row n_abund_partial + b (the buffer's BEAN_SURV_FOLD_ROWS spare rows), the last CTA sums those M rows.  With guides
  // sharded over GPUs the host all-reduces these R + 1 numbers.
  const int C = p.R + 1;
  const int M = p.sums_next ? min(min((int)gridDim.x, BEAN_SURV_FOLD_ROWS), p.n_abund_partial) : 0;
  if ((int)blockIdx.x < M) {
    const double tot_j = column_sums(p.abund_partial, p.n_abund_partial, C, (int)blockIdx.x, M, s_cs);
    if ((int)threadIdx.x < C) {
      p.abund_partial[((size_t)p.n_abund_partial + blockIdx.x) * C + threadIdx.x] = tot_j;
      __threadfence();
    }
  }
  note_nonfinite(p.nonfinite, p.step, 0xffffffffu, bad);
  const double tot = block_sum(elbo, red);  // (its barriers also order the row written above before thread 0's fence)
  if (threadIdx.x == 0) {
    p.partial[p.n_partial_guide + blockIdx.x] = tot;
    __threadfence();
    const uint32_t done = atomicAdd(p.counter, 1u);
    is_last = (done == (uint32_t)gridDim.x - 1u);
  }
  __syncthreads();
  if (is_last) {
    // last CTA: fixed-order reduction of every CTA's partial of this step -> loss[t] = -ELBO
    __threadfence();
    const double* pv = p.partial + p.n_partial_guide;
    const int n = p.n_partial_var;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;  // four loads in flight per thread
    int i = threadIdx.x;
    for (; i + 3 * VAR_THREADS < n; i += 4 * VAR_THREADS) {
      a0 += __ldcg(pv + i);
      a1 += __ldcg(pv + i + VAR_THREADS);
      a2 += __ldcg(pv + i + 2 * VAR_THREADS);
      a3 += __ldcg(pv + i + 3 * VAR_THREADS);
    }
    for (; i < n; i += VAR_THREADS) a0 += __ldcg(pv + i);
    const double all = block_sum((a0 + a1) + (a2 + a3), red);
    if (threadIdx.x == 0) {
      const double loss = -(all + p.ll_const);
      p.loss[p.step] = loss;
      *p.counter = 0u;
      if (p.apply_update && p.nonfinite && !isfinite(loss)) record_nonfinite(p.nonfinite, p.step);
    }
    if (p.sums_next) {
      const double tot_j = column_sums(p.abund_partial + (size_t)p.n_abund_partial * C, M, C, 0, 1, s_cs);
      if ((int)threadIdx.x < C) p.sums_next[threadIdx.x] = tot_j;
      if (p.peer_world > 1) {
        // publish this rank's partial sums of step t + 1 into every rank's exchange buffer (remote stores over NVLink), then --
        // after a system-scope fence on every writer and the barrier -- the flag that tells that rank they are there
        const int slot = (int)((p.step + 1u) & 1u);
        if ((int)threadIdx.x < C) {
          for (int k = 0; k < p.peer_world; ++k) {
            volatile double* dst = &p.peer_buf[k]->vals[slot][p.peer_rank][threadIdx.x];
            *dst = tot_j;
          }
          __threadfence_system();
        }
        __syncthreads();
        if ((int)threadIdx.x < p.peer_world) {
          __threadfence_system();
          volatile unsigned long long* f = &p.peer_buf[threadIdx.x]->flag[slot][p.peer_rank];
          *f = (unsigned long long)p.step + 2ull;
        }
      }
    }
  }
}

}  // namespace bean
