// bean_svi_tiling.cu -- the fused SVI step of the tiling sorting program (MultiMixtureNormal over filtered alleles).
//
// One `svi.step` of bean/model/run.py:376-380 for bean/model/model.py:550-751 (MultiMixtureNormalModel) and :878-962
// (MultiMixtureNormalGuide) in three launches, every value and gradient in closed form (pinned beforehand in
// oracle/tiling_closed_form.py):
//
//   tiling_draw_kernel   one thread per edit: reparameterised draws mu_e ~ Normal, sd_e ~ LogNormal (counter-based noise).
//   tiling_guide_kernel  one CTA per guide, one WARP per replicate (+ one for the Dirichlet normalisers), one LANE per allele
//       (wild type + up to 31 edited alleles): allele mean / sd from
//       its edits through the CSR map (the reference's dense (G, A-1, E) matmul / norm, model.py:618-625), Normal-CDF bin masses
//       per allele, per replicate: pi ~ Dirichlet draw (one gamma per lane, normalised by a warp sum), allele mixture by warp
//       reductions over the alleles, get_alpha + Dirichlet-Multinomial rows of the count layers (evaluated identically by all
//       lanes), editing-rate sites (model Dirichlet with the epsilon-regularised concentration, guide Dirichlet, reporter
//       Multinomial -- all under repguide_mask, model.py:632-670 / :938-950), pathwise Dirichlet derivative, then per lane the
//       alpha_pi gradient and its ClippedAdam update, and d ELBO / d (allele mean, sd) into the allele's slot.
//   svi_variant_kernel   (shared) with the edits as "variants": per-edit reduction of the slot gradients over the CSC map
//       (deterministic, no atomics), Laplace / Normal and LogNormal priors, guide densities, ClippedAdam, loss[t].
//
// The concentrations, the pi draws and the editing-rate sites are evaluated in DOUBLE in both builds: in the reference they
// carry pi_a0's dtype (float64 out of the a0 fit) even on its float32 path, draws of non-existent alleles underflow float32,
// and they are O(R A) work per guide beside the O(R L B) special-function rows.
#include <string.h>

#include "bean_svi_shared.cuh"

namespace bean {

constexpr int TILING_MAX_REP_WARPS = 8;  // replicate warps per guide (CTA = these + one site warp)
enum : uint32_t { STREAM_TILING_PI = 96 };

template <typename real>
struct TilingParams {
  int G, R, B, L, A, C;
  int apply_update;
  uint32_t step, guide_offset;
  uint64_t seed;
  real mask_thres;
  const real* x;             // [L][R][G][B]
  const real* a0;            // [L][G]
  const uint8_t* row_mask;   // [R][G]
  const uint8_t* allele_mask;  // [G][A]
  const int32_t* allele_ptr;   // CSR over slots g * (A - 1) + (a - 1)
  const int32_t* allele_edit;
  const double* pi_a0;       // [G]
  const real* counts;        // [R][C][G][A] reporter allele counts of the control condition(s)
  const real* mu_e;          // [E] this step's draws (tiling_draw_kernel)
  const real* sd_e;
  real* alpha_u; real* alpha_m; real* alpha_v; real* alpha_grad;  // [G][A]
  real* d_slot;              // [2][G * (A - 1)]: d ELBO / d mu_allele, (d ELBO / d sd_allele) / sd_allele
  double* partial;           // per-warp ELBO partials
  int32_t* nonfinite;        // first non-finite step or NULL (BeanTilingState.nonfinite_step)
  const double* pi_in;       // [R][G][A] injected draws (parity) or NULL
  double* pi_out;
  double epsilon, prob_eps, pi_tiny;
  real step_size, beta1, beta2, adam_eps, clip;
  SampleTables<real> t;
};

__device__ __forceinline__ double warp_all_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <typename real>
__device__ __forceinline__ real warp_all_sum_r(real v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Gamma(alpha) in double for (guide g, replicate r, allele a) at `step`
__device__ __forceinline__ double tiling_gamma(uint64_t seed, uint32_t g, uint32_t r, uint32_t a, uint32_t step, double alpha) {
  GammaMT<double> mt;
  mt.init(alpha);
  const uint2 key = seed_key(seed);
  const uint32_t cy = r | (a << 8);
  double boost = 1.0;
  if (mt.inv_alpha != 0.0) {
    const uint4 w = philox4x32_10(make_uint4(g, cy, step, STREAM_TILING_PI), key);
    const double lb = ::log(1.0 - (double)u01(w.x)) * mt.inv_alpha;
    if (lb < -720.0) return 0.0;  // below the smallest double: clamped by the caller
    boost = ::exp(lb);
  }
  double out = 0.0;
  bool ok = false;
  for (uint32_t k = 0; k < 16u && !ok; ++k) {
    const uint4 w = philox4x32_10(make_uint4(g, cy, step, STREAM_TILING_PI + 8u * (k + 1u)), key);
    float n0, n1;
    box_muller(w.x, w.y, n0, n1);
    ok = mt.attempt(n0, 1.0f - u01(w.z), out);
    if (!ok) ok = mt.attempt(n1, 1.0f - u01(w.w), out);
  }
  return out * boost;
}

template <typename real>
__global__ void __launch_bounds__(VAR_THREADS) tiling_draw_kernel(const SviParams<real> p, real* mu_e, real* sd_e) {
  grid_dependency_wait();
  const int e = blockIdx.x * VAR_THREADS + threadIdx.x;
  if (e >= p.T) return;
  real mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, log_sd;
  variant_draw(p, e, mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, log_sd);
  mu_e[e] = mu_t;
  sd_e[e] = sd_t;
}

// One CTA per guide, NW = blockDim / 32 warps: warp w takes replicates w, w + NW, ... (draw, allele mixture, count rows,
// editing-rate sites, pathwise derivative); the last warp then adds the replicate-independent normalisers of the two Dirichlet
// sites (lgamma / digamma of the model's concentrations).  The kernel is bound by the LATENCY of its double-precision chains
// (800 guides = 5 warps per SM with a warp per guide: 78 us at c3), so the host picks the largest NW whose warps are all
// resident at once (tiling_run) and the replicates run side by side instead of one after the other.  The warps' accumulators
// meet in shared memory and warp 0 adds them in a fixed order (deterministic), then does the per-allele epilogue.  Every warp
// repeats the cheap prologue (concentrations, allele mean / sd, bin masses).
template <typename real, int NB>
__global__ void __launch_bounds__(TILING_MAX_REP_WARPS * 32) tiling_guide_kernel(const TilingParams<real> p) {
  grid_dependency_wait();
  __shared__ double s_elbo[TILING_MAX_REP_WARPS][32], s_slp[TILING_MAX_REP_WARPS][32], s_path[TILING_MAX_REP_WARPS][32];
  __shared__ real s_dP[TILING_MAX_REP_WARPS][NB][32];
  __shared__ int s_nin[TILING_MAX_REP_WARPS];
  __shared__ double s_dgd_m[32], s_norm_diff;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int NW = (int)(blockDim.x >> 5);
  const int g = blockIdx.x;
  const int R = p.R, B = p.B, A = p.A, C = p.C;
  const bool has = lane < A;
  const bool exists = has && p.allele_mask[(size_t)g * A + lane] != 0;
  const double eps = p.epsilon;
  // ---- editing-rate concentrations (model.py:645-651 model, :937-938 guide; entries of non-existent alleles are epsilon)
  const double al = has ? (exists ? ::exp((double)p.alpha_u[(size_t)g * A + lane]) : eps) : 0.0;
  const double asum = warp_all_sum(al);
  const double pa0 = p.pi_a0[g];
  const double cg = has ? al / asum * pa0 : 1.0;  // guide: neither clamped nor regularised
  const double S1 = asum + eps;
  const double cm_raw = has ? (al + eps / A) / S1 * pa0 : 1.0;
  const bool cm_live = cm_raw >= eps;              // `pi_a_scaled[pi_a_scaled < eps] = eps` (model.py:651): no gradient there
  const double cm = cm_live ? cm_raw : eps;
  const double sum_g = warp_all_sum(has ? cg : 0.0);
  const double dgd_g = digamma_f64(sum_g) - digamma_f64(cg);  // psi(sum) - psi(c_a): Dirichlet site and pathwise derivative
  // ---- allele mean / sd from its edits (model.py:618-625): wild type (0, 1)
  real mu_a = real(0), sd_a = real(1);
  long long slot = -1;
  if (has && lane > 0) {
    slot = (long long)g * (A - 1) + (lane - 1);
    real m = real(0), v = real(0);
    for (int k = p.allele_ptr[slot]; k < p.allele_ptr[slot + 1]; ++k) {
      const int e = p.allele_edit[k];
      m += p.mu_e[e];
      v += p.sd_e[e] * p.sd_e[e];
    }
    mu_a = m;
    sd_a = Num<real>::sqrt(v);
  }
  real P[NB], dP[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    dP[b] = real(0);
    P[b] = (b < B && exists) ? bin_mass_sorting(p.t.thr_u[b], p.t.thr_l[b], mu_a, sd_a) : real(0);  // utils.py:73-74: absent -> 0
  }
  double elbo = 0.0, slp = 0.0, path = 0.0;  // sum of log pi over the masked replicates; sum of the pathwise terms
  int n_in = 0;
  const real epsr = real(1e-5);
  for (int r = warp; r < R; r += NW) {
    const bool rmask = p.row_mask[(size_t)r * p.G + g] != 0;
    // ---- pi ~ Dirichlet(cg): one gamma per lane, normalised over the warp, clamped like torch's sampler
    double pi_a = 0.0;
    if (p.pi_in) {
      pi_a = has ? p.pi_in[((size_t)r * p.G + g) * A + lane] : 0.0;
    } else {
      const double gam = has ? ::fmax(tiling_gamma(p.seed, (uint32_t)g + p.guide_offset, (uint32_t)r, (uint32_t)lane, p.step, cg), 2.2250738585072014e-308) : 0.0;
      const double tot = warp_all_sum(gam);
      pi_a = has ? ::fmin(::fmax(gam / tot, p.pi_tiny), 1.0 - 1.1102230246251565e-16) : 0.0;
    }
    if (p.pi_out && has) p.pi_out[((size_t)r * p.G + g) * A + lane] = pi_a;
    // ---- allele mixture (model.py:699-703): e[b] = sum_a pi_a P_a[b]
    real e[NB], de[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      e[b] = b < B ? warp_all_sum_r<real>(real(pi_a) * P[b]) : real(0);
      de[b] = real(0);
    }
    // ---- Dirichlet-Multinomial rows (model.py:706-751): every lane evaluates the same numbers
    for (int l = 0; l < p.L; ++l) {
      const real* xr = p.x + (((size_t)l * R + r) * p.G + g) * B;
      real xb[NB], pb[NB], ab[NB], frac[NB], gb[NB];
      bool live[NB];
      real N = real(0), S = real(0);
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        xb[b] = b < B ? xr[b] : real(0);
        N += xb[b];
        pb[b] = b < B ? e[b] * p.t.sf[l][r * B + b] : real(0);
        S += pb[b];
      }
      if (!(rmask && N > p.mask_thres)) continue;  // poutine.mask
      const real a0 = p.a0[(size_t)l * p.G + g];
      const real inv = Num<real>::rcp(S + epsr);
      real Asum = real(0);
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        frac[b] = (pb[b] + epsr / real(B)) * inv;
        const real raw = frac[b] * a0 * p.t.smask[r * B + b];
        live[b] = raw >= epsr;
        ab[b] = (b < B) ? (live[b] ? raw : epsr) : real(0);
        Asum += ab[b];
      }
      const real V = dm_row_kl<real, NB>(B, xb, ab, N, Asum, gb);
      if (lane == 0) elbo += (double)V;
      real dot = real(0);
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        gb[b] = (b < B && live[b]) ? gb[b] * p.t.smask[r * B + b] : real(0);
        dot += gb[b] * frac[b];
      }
      const real cc = a0 * inv;
#pragma unroll
      for (int b = 0; b < NB; ++b)
        if (b < B) de[b] += p.t.sf[l][r * B + b] * cc * (gb[b] - dot);
    }
    double go = 0.0;  // d ELBO / d pi_a
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      go += (double)(de[b] * P[b]);
      dP[b] += de[b] * real(pi_a);
    }
    if (!has) go = 0.0;
    if (rmask) {
      // ---- editing-rate sites under repguide_mask: model Dirichlet(cm) - guide Dirichlet(cg), reporter Multinomial
      ++n_in;
      const double lp = has ? ::log(pi_a) : 0.0;
      if (has) {
        elbo += (cm - cg) * lp;
        go += (cm - cg) / pi_a;
        slp += lp;
      }
      const double Sp = warp_all_sum(has ? pi_a : 0.0);
      const double n = has ? pi_a / Sp : 0.5;
      const bool inside = n >= p.prob_eps && n <= 1.0 - p.prob_eps;
      const double lcl = ::log(::fmin(::fmax(n, p.prob_eps), 1.0 - p.prob_eps));
      for (int c = 0; c < C; ++c) {
        const double xc = has ? (double)p.counts[(((size_t)r * C + c) * p.G + g) * A + lane] : 0.0;
        if (xc != 0.0) elbo += xc * lcl;
        const double h = (has && inside) ? xc / n : 0.0;
        const double hbar = warp_all_sum(h * n);
        if (has) go += (h - hbar) / Sp;
      }
    }
    // ---- pathwise derivative of the draw w.r.t. the guide concentration (torch _Dirichlet_backward)
    const double dot = warp_all_sum(has ? pi_a * go : 0.0);
    if (has) path += dirichlet_grad_one_f64_psi(pi_a, cg, sum_g, dgd_g) * (go - dot);
  }
  if (warp == NW - 1) {  // the model site's psi(sum) - psi(c_a) and the difference of the two Dirichlet normalisers
    const double sum_m = warp_all_sum(has ? cm : 0.0);
    s_dgd_m[lane] = digamma_f64(sum_m) - digamma_f64(cm);
    const double nd = (::lgamma(sum_m) - warp_all_sum(has ? ::lgamma(cm) : 0.0)) - (::lgamma(sum_g) - warp_all_sum(has ? ::lgamma(cg) : 0.0));
    if (lane == 0) s_norm_diff = nd;
  }
  s_elbo[warp][lane] = elbo;
  s_slp[warp][lane] = slp;
  s_path[warp][lane] = path;
#pragma unroll
  for (int b = 0; b < NB; ++b) s_dP[warp][b][lane] = dP[b];
  if (lane == 0) s_nin[warp] = n_in;
  __syncthreads();
  if (warp != 0) return;
  // ---- warp 0: the replicate warps' sums in warp order, then the per-allele epilogue
  elbo = 0.0; slp = 0.0; path = 0.0; n_in = 0;
#pragma unroll
  for (int b = 0; b < NB; ++b) dP[b] = real(0);
  for (int w = 0; w < NW; ++w) {
    elbo += s_elbo[w][lane];
    slp += s_slp[w][lane];
    path += s_path[w][lane];
    n_in += s_nin[w];
#pragma unroll
    for (int b = 0; b < NB; ++b) dP[b] += s_dP[w][b][lane];
  }
  const double dcm = has ? (double)n_in * s_dgd_m[lane] + slp : 0.0;   // d / d cm: n_in (psi(sum) - psi(cm)) + sum log pi
  const double dcg = has ? path - ((double)n_in * dgd_g + slp) : 0.0;  // d / d cg: pathwise - [n_in (psi(sum) - psi(cg)) + sum log pi]
  elbo += lane == 0 ? (double)n_in * s_norm_diff : 0.0;
  // ---- d ELBO / d (allele mean, sd) into the allele's slot; the per-edit kernel reduces the slots over the CSC map
  if (slot >= 0) {
    real dmu = real(0), dsd = real(0);
    if (exists) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        if (b < B) {
          real dPm, dPs;
          bin_mass_grad_sorting(p.t.thr_u[b], p.t.thr_l[b], mu_a, sd_a, dPm, dPs);
          dmu += dP[b] * dPm;
          dsd += dP[b] * dPs;
        }
      }
    }
    const size_t n_slots = (size_t)p.G * (A - 1);
    p.d_slot[slot] = dmu;
    p.d_slot[n_slots + slot] = (exists && sd_a > real(0)) ? dsd / sd_a : real(0);
  }
  // ---- concentrations -> log alpha_pi (tiling_closed_form.py), ClippedAdam per existing allele
  const double dm = cm_live ? dcm : 0.0;
  const double sum_cg = warp_all_sum(has ? dcg * al : 0.0), sum_cm = warp_all_sum(has ? dm * (al + eps / A) : 0.0);
  bool bad = false;
  if (has) {
    const double d_al = pa0 / (asum * asum) * (dcg * asum - sum_cg) + pa0 / S1 * (dm - sum_cm / S1);
    const real gl = exists ? real(-d_al * al) : real(0);
    const size_t i = (size_t)g * A + lane;
    if (p.alpha_grad) p.alpha_grad[i] = gl;
    if (p.apply_update) {
      real th = p.alpha_u[i], m = p.alpha_m[i], v = p.alpha_v[i];
      bad = !isfinite(gl);
      const real gc = Num<real>::fmin(Num<real>::fmax(gl, -p.clip), p.clip);
      m = p.beta1 * m + (real(1) - p.beta1) * gc;
      v = p.beta2 * v + (real(1) - p.beta2) * gc * gc;
      th -= p.step_size * m / (Num<real>::sqrt(v) + p.adam_eps);
      p.alpha_u[i] = th; p.alpha_m[i] = m; p.alpha_v[i] = v;
    }
  }
  note_nonfinite(p.nonfinite, p.step, 0xffffffffu, bad);
  const double tot = warp_all_sum(elbo);
  if (lane == 0) p.partial[g] = tot;
}

template <typename real>
static int tiling_run(const BeanScreen* s, const BeanTilingState* ts, const BeanSviConfig* cfg, const BeanTilingNoise* noise,
                      int32_t first_step, int32_t n_steps, void* stream) {
  int rc = validate_screen(s);
  if (rc != BEAN_OK) return rc;
  BEAN_REQUIRE(ts && cfg, BEAN_EINVAL, "state / cfg is NULL");
  BEAN_REQUIRE(s->mode == BEAN_MODE_SORTING, BEAN_EINVAL, "bean_svi_tiling_run needs a sorting screen");
  BEAN_REQUIRE(ts->map && ts->map->n_guides == s->n_guides, BEAN_EINVAL, "allele map missing or of another screen");
  const int A = ts->map->n_alleles, E = ts->map->n_edits;
  BEAN_REQUIRE(A >= 2 && A <= 32, BEAN_EINVAL, "the fused tiling step takes 2..32 alleles per guide (got %d): one lane per allele", A);
  BEAN_REQUIRE(E > 0, BEAN_EINVAL, "n_edits must be > 0");
  BEAN_REQUIRE(ts->n_controls >= 1, BEAN_EINVAL, "n_controls must be >= 1");
  BEAN_REQUIRE(ts->allele_mask && ts->pi_a0 && ts->counts, BEAN_EINVAL, "allele_mask / pi_a0 / counts must be non-NULL");
  BEAN_REQUIRE(ts->edit_params && ts->edit_m && ts->edit_v && ts->alpha_u && ts->alpha_m && ts->alpha_v, BEAN_EINVAL, "parameter buffers must be non-NULL");
  BEAN_REQUIRE(ts->mu_e && ts->sd_e && ts->d_slot && ts->partial && ts->counter && ts->loss, BEAN_EINVAL, "scratch buffers must be non-NULL");
  if ((rc = check_step_range(first_step, n_steps, ts->loss_capacity)) != BEAN_OK) return rc;
  if (noise && (rc = check_eps_pair(noise->eps_mu, noise->eps_sd)) != BEAN_OK) return rc;

  const int G = s->n_guides;
  const int n_slots = G * (A - 1);
  // ---- the per-edit kernels: SviParams with the edits as variants
  SviParams<real> v;
  memset(&v, 0, sizeof(v));
  fill_common(v, s, cfg);
  v.G = n_slots; v.T = E;
  v.has_sd = 1;
  v.variant_ptr = ts->map->edit_ptr; v.gather_idx = ts->map->edit_slot; v.dsd_times_sd = 1;
  v.var_params = static_cast<real*>(ts->edit_params); v.var_m = static_cast<real*>(ts->edit_m); v.var_v = static_cast<real*>(ts->edit_v);
  v.var_grad = static_cast<real*>(ts->edit_grad);
  v.d_guide = static_cast<real*>(ts->d_slot);
  v.partial = ts->partial; v.counter = ts->counter; v.loss = ts->loss; v.nonfinite = ts->nonfinite_step;
  v.n_partial_guide = G;  // one ELBO partial per guide (warp)
  v.n_partial_var = (E + VAR_PER_CTA - 1) / VAR_PER_CTA;
  v.eps_mu = noise ? static_cast<const real*>(noise->eps_mu) : nullptr;
  v.eps_sd = noise ? static_cast<const real*>(noise->eps_sd) : nullptr;
  v.eps_out = noise ? static_cast<real*>(noise->eps_out) : nullptr;
  v.mu_prior_loc_v = static_cast<const real*>(ts->mu_prior_loc_v); v.mu_prior_scale_v = static_cast<const real*>(ts->mu_prior_scale_v);
  v.sd_prior_loc_v = static_cast<const real*>(ts->sd_prior_loc_v); v.sd_prior_scale_v = static_cast<const real*>(ts->sd_prior_scale_v);
  // ---- the per-guide kernel
  TilingParams<real> p;
  memset(&p, 0, sizeof(p));
  p.G = G; p.R = s->n_reps; p.B = s->n_bins; p.L = s->n_layers; p.A = A; p.C = ts->n_controls;
  p.apply_update = cfg->apply_update; p.guide_offset = cfg->guide_offset; p.seed = cfg->seed;
  p.mask_thres = real(s->mask_thres);
  p.x = static_cast<const real*>(s->x); p.a0 = static_cast<const real*>(s->a0); p.row_mask = s->row_mask;
  p.allele_mask = ts->allele_mask; p.allele_ptr = ts->map->allele_ptr; p.allele_edit = ts->map->allele_edit;
  p.pi_a0 = ts->pi_a0; p.counts = static_cast<const real*>(ts->counts);
  p.mu_e = static_cast<const real*>(ts->mu_e); p.sd_e = static_cast<const real*>(ts->sd_e);
  p.alpha_u = static_cast<real*>(ts->alpha_u); p.alpha_m = static_cast<real*>(ts->alpha_m); p.alpha_v = static_cast<real*>(ts->alpha_v);
  p.alpha_grad = static_cast<real*>(ts->alpha_grad);
  p.d_slot = static_cast<real*>(ts->d_slot);
  p.partial = ts->partial;
  p.nonfinite = ts->nonfinite_step;
  p.pi_in = noise ? noise->pi : nullptr; p.pi_out = noise ? noise->pi_out : nullptr;
  p.epsilon = ts->epsilon > 0.0 ? ts->epsilon : 1e-5;
  p.prob_eps = cfg->prob_clamp_eps > 0.0 ? cfg->prob_clamp_eps : 2.220446049250313e-16;
  p.pi_tiny = ts->pi_tiny > 0.0 ? ts->pi_tiny : 2.2250738585072014e-308;
  p.beta1 = v.beta1; p.beta2 = v.beta2; p.adam_eps = v.adam_eps; p.clip = v.clip;
  fill_tables(s, p.t);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // warps per guide: as many as stay resident all at once (one wave), at most one per replicate
  int n_rep_warps = 1;
  {
    cudaFuncAttributes fa;
    BEAN_CUDA(s->n_bins <= 4 ? cudaFuncGetAttributes(&fa, tiling_guide_kernel<real, 4>) : cudaFuncGetAttributes(&fa, tiling_guide_kernel<real, BEAN_MAX_BINS>));
    int sms = bean_device_sm_count();
    if (sms <= 0) sms = 148;
    const int regs = ((fa.numRegs + 7) / 8) * 8;
    const long long resident_warps = (long long)sms * (65536 / (regs * 32));
    const int cap = s->n_reps < TILING_MAX_REP_WARPS ? s->n_reps : TILING_MAX_REP_WARPS;
    while (n_rep_warps * 2 <= cap && (long long)G * (n_rep_warps * 2) <= resident_warps) n_rep_warps *= 2;
  }
  // guides sharded over ranks: phase 1 leaves this shard's per-edit sums in edit_sum, phase 2 (after the host's all-reduce)
  // updates every edit from them -- `u` = the per-edit kernel's parameters with the reduced sums as a one-entry-per-edit CSR
  const bool sharded = ts->edit_sum != nullptr;
  SviParams<real> u = v;
  if (sharded) {
    BEAN_REQUIRE(ts->edit_iota != nullptr, BEAN_EINVAL, "edit_sum needs edit_iota");
    BEAN_REQUIRE(cfg->phases == 1 || cfg->phases == 2, BEAN_EINVAL, "sharded tiling step: phases must be 1 (reduce) or 2 (update), got %d", cfg->phases);
    v.seg_sum_out = static_cast<real*>(ts->edit_sum);
    u.G = E; u.d_guide = static_cast<real*>(ts->edit_sum); u.variant_ptr = ts->edit_iota; u.gather_idx = nullptr;
    u.variant_terms_off = ts->edit_term_weight == 0.0 ? 1 : 0;
  }
  for (int i = 0; i < n_steps; ++i) {
    const int t = first_step + i;
    v.step = u.step = p.step = (uint32_t)t;
    v.step_size = u.step_size = p.step_size = adam_step_size<real>(cfg, t);
    if (sharded && cfg->phases == 2) {
      launch_after(svi_variant_kernel<real>, u.n_partial_var, VAR_THREADS, st, u);
      continue;
    }
    tiling_draw_kernel<real><<<(E + VAR_THREADS - 1) / VAR_THREADS, VAR_THREADS, 0, st>>>(v, static_cast<real*>(ts->mu_e), static_cast<real*>(ts->sd_e));
    if (s->n_bins <= 4)  // bin arrays of 4 instead of BEAN_MAX_BINS registers: more guides resident per SM
      launch_after(tiling_guide_kernel<real, 4>, G, n_rep_warps * 32, st, p);
    else
      launch_after(tiling_guide_kernel<real, BEAN_MAX_BINS>, G, n_rep_warps * 32, st, p);
    launch_after(svi_variant_kernel<real>, v.n_partial_var, VAR_THREADS, st, v);
  }
  BEAN_CUDA(cudaPeekAtLastError());
  return BEAN_OK;
}

}  // namespace bean

extern "C" {
int bean_svi_tiling_num_partials(int32_t n_guides, int32_t n_edits) { return n_guides + (n_edits + bean::VAR_PER_CTA - 1) / bean::VAR_PER_CTA; }
int bean_svi_tiling_run_f32(const BeanScreen* s, const BeanTilingState* ts, const BeanSviConfig* c, const BeanTilingNoise* n, int32_t first_step,
                            int32_t n_steps, void* stream) {
  return bean::tiling_run<float>(s, ts, c, n, first_step, n_steps, stream);
}
int bean_svi_tiling_run_f64(const BeanScreen* s, const BeanTilingState* ts, const BeanSviConfig* c, const BeanTilingNoise* n, int32_t first_step,
                            int32_t n_steps, void* stream) {
  return bean::tiling_run<double>(s, ts, c, n, first_step, n_steps, stream);
}
}
