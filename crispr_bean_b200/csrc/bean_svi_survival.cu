// bean_svi_survival.cu -- the fused SVI step of the survival (proliferation) MixtureNormal program.
//
// One `svi.step` of bean/model/run.py:376-380 for bean/model/survival_model.py:215-424 (MixtureNormalModel) and :651-739
// (MixtureNormalGuide) in three launches and no host round trip; every site's value and gradient in closed form
// (pinned beforehand in oracle/survival_closed_form.py and oracle/survival_guide_row.c):
//
//   surv_guide_kernel   one thread per guide.  Parameter-free growth draw of the unedited allele u ~ N(m0, s0)
//       (`mu_negctrl`, a model-only latent: fresh prior noise every step); allele growth rates (u, u + mu_variant);
//       abundance sites: x[r][g] = gamma[r][g] / sum_g gamma[r][.] is the guide's Dirichlet(q0) draw over ALL guides,
//       the model observes (X[:, 0] + 1) / sum under the same Dirichlet(q0), so the normalisers cancel and the pair adds
//       sum (q0 - 1)(log obs - log x); pathwise derivative D(x, q0, sum q0) with sum_h x_h gout_h = -(sum q0 - G) in closed
//       form -- two library-wide sums per replicate are all that crosses guides; per replicate: pi ~ Beta draw, model /
//       guide Dirichlet sites, reporter Multinomial on pi exp(mu t_c), Dirichlet-Multinomial rows of both count layers on
//       e[b] = sum_a pi_a exp(mu_a t_b) with their digamma differences; q0 gradient AND its ClippedAdam update, then the
//       NEXT step's gamma draws from the updated q0 with their per-warp partial sums.
//   svi_alpha_kernel    (shared with the sorting step) pathwise Dirichlet derivative of the pi draws, alpha_pi update.
//   svi_variant_kernel  (shared) segmented reduction of d ELBO / d (edited growth rate) per variant, Laplace / Normal prior,
//       Normal guide entropy, update of (mu_loc, mu_scale); last CTA: loss[t] and the library-wide sums of the next step.
#include <string.h>

#include "bean_svi_shared.cuh"

namespace bean {

enum : uint32_t { STREAM_NEGCTRL = 48, STREAM_ABUND = 52 };  // bean_rng.cuh uses 0 .. 47, bean_dirichlet.cu 64 ..

// Gamma(c) draw behind the abundance sample of guide g, replicate r at `step` (Marsaglia-Tsang + boost; c = q0[g] is
// ~1/G, so nearly every draw underflows to `tiny` -- exactly what torch's sampler does with such a concentration)
template <typename real>
__device__ __forceinline__ real abundance_gamma(uint64_t seed, uint32_t g, uint32_t r, uint32_t step, real c) {
  GammaMT<real> mt;
  mt.init(c);
  const uint2 key = seed_key(seed);
  real boost = real(1);
  if (mt.inv_alpha != real(0)) {
    // alpha < 1: Gamma(a) = Gamma(a + 1) U^(1/a).  With a = q0 ~ 1/G the factor underflows for all but ~1e-4 of the draws:
    // its logarithm is looked at FIRST, and a draw that cannot reach `tiny` (Gamma(a + 1) < e^12 with probability
    // 1 - 1e-5 ... it is clamped to tiny either way) skips the Marsaglia-Tsang loop altogether
    const uint4 w = philox4x32_10(make_uint4(g, r, step, STREAM_ABUND), key);
    const real lb = Num<real>::flog(real(1) - real(u01(w.x))) * mt.inv_alpha;
    if (lb < real(sizeof(real) == 4 ? -100.0 : -720.0)) return Lim<real>::tiny();
    boost = Num<real>::exp(lb);
  }
  real out = real(0);
  bool ok = false;
  for (uint32_t k = 0; k < 16u && !ok; ++k) {
    const uint4 w = philox4x32_10(make_uint4(g, r, step, STREAM_ABUND + 64u * (k + 1u)), key);
    float n0, n1;
    box_muller(w.x, w.y, n0, n1);
    ok = mt.attempt(n0, 1.0f - u01(w.z), out);
    if (!ok) ok = mt.attempt(n1, 1.0f - u01(w.w), out);
  }
  return Num<real>::fmax(out * boost, Lim<real>::tiny());
}

// standard normal behind mu_negctrl of guide g at `step`
__device__ __forceinline__ float negctrl_noise(uint64_t seed, uint32_t g, uint32_t step) {
  const uint4 w = philox4x32_10(make_uint4(g, 0u, step, STREAM_NEGCTRL), seed_key(seed));
  float e0, e1;
  box_muller(w.x, w.y, e0, e1);
  return e0;
}

// gamma draws of `step` from the CURRENT q0 + per-warp partial sums (first step of a run; later steps get theirs from the
// guide kernel of the step before)
template <typename real>
__device__ __forceinline__ void draw_abundance(const SviParams<real>& p, int g, bool owns, real c, uint32_t step) {
  const int R = p.R;
  for (int r = 0; r < R; ++r) {
    real gam = real(0);
    if (owns) {
      gam = abundance_gamma<real>(p.seed, (uint32_t)g + p.guide_offset, (uint32_t)r, step, c);
      p.gamma_next[(size_t)r * p.G + g] = gam;
    }
    const double tot = warp_sum((double)gam);
    if ((threadIdx.x & 31) == 0) p.abund_partial[(size_t)((blockIdx.x * SVI_THREADS + threadIdx.x) / SVI_WARP) * (R + 1) + r] = tot;
  }
  const double totc = warp_sum(owns ? (double)c : 0.0);
  if ((threadIdx.x & 31) == 0) p.abund_partial[(size_t)((blockIdx.x * SVI_THREADS + threadIdx.x) / SVI_WARP) * (R + 1) + R] = totc;
}

template <typename real>
__global__ void __launch_bounds__(SVI_THREADS) surv_prime_kernel(const SviParams<real> p) {
  const int g = blockIdx.x * SVI_THREADS + threadIdx.x;
  const bool owns = g < p.G;
  const real c = owns ? Num<real>::exp(p.q0_u[g]) : real(0);
  draw_abundance(p, g, owns, c, p.step);
}

// sums_next[j] = sum of the per-warp partials (one CTA; fixed order)
template <typename real>
__global__ void __launch_bounds__(VAR_THREADS) surv_sums_kernel(const SviParams<real> p) {
  __shared__ double red[32];
  for (int j = 0; j <= p.R; ++j) {
    double a = 0.0;
    for (int i = threadIdx.x; i < p.n_abund_partial; i += VAR_THREADS) a += p.abund_partial[(size_t)i * (p.R + 1) + j];
    const double tot = block_sum(a, red);
    if (threadIdx.x == 0) p.sums_next[j] = tot;
  }
}

// EXACT: the screen has exactly NB timepoints (no `b < B` predicates in the bin loops).
#ifndef BEAN_SURV_MIN_CTAS
#define BEAN_SURV_MIN_CTAS 6
#endif
template <typename real, int NB, bool EXACT>
__global__ void __launch_bounds__(SVI_THREADS, sizeof(real) == 4 ? BEAN_SURV_MIN_CTAS : 3) surv_guide_kernel(const SviParams<real> p) {
  grid_dependency_wait();
  const int g = blockIdx.x * SVI_THREADS + threadIdx.x;
  const int R = p.R, B = EXACT ? NB : p.B;
  const real eps = real(1e-5);
  const bool owns = g < p.G;
  double elbo = 0.0;
  bool bad = false;  // q0's ClippedAdam input was NaN / inf
  real c_next = real(0);
  __shared__ double s_sums[BEAN_PEER_MAX_VALS];
  load_library_sums(p, R + 1, s_sums);
  if (owns) {
    const int v = p.guide_variant[g];
    real mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, log_sd;
    variant_draw(p, v, mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, log_sd);
    // mu_negctrl: u = m0 + s0 eps, density Normal(m0, s0) without parameters (survival_model.py:271-274)
    const real e_u = p.eps_negctrl ? p.eps_negctrl[g] : real(negctrl_noise(p.seed, (uint32_t)g + p.guide_offset, p.step));
    const real u = p.negctrl_loc + p.negctrl_scale * e_u;
    real elbo_g = -Num<real>::log(p.negctrl_scale) - real(0.5) * e_u * e_u - real(0.91893853320467274178);
    const real mu0 = u, mu1 = u + mu_t;  // growth rate of (unedited, edited) allele (survival_model.py:276-285)
    real P0[NB], P1[NB], dP1[NB];        // exp(mu_a t_b) (survival_model.py:358-361); dP1 accumulates d ELBO / d P1
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      P0[b] = b < B ? Num<real>::exp(mu0 * p.t.tp[b]) : real(0);
      P1[b] = b < B ? Num<real>::exp(mu1 * p.t.tp[b]) : real(0);
      dP1[b] = real(0);
    }
    // editing-rate concentrations (survival_model.py:300-302 / :690-698): model = alpha/sum*pi_a0, guide = clamp(model, 1e-5)
    real al[2], cm[2], cg[2], lg_cm, lg_cg, dgd_cm[2], dgd_cg[2], dcm[2] = {}, dcg[2] = {};
    al[0] = Num<real>::exp(p.alpha_u[2 * (size_t)g]);
    al[1] = Num<real>::exp(p.alpha_u[2 * (size_t)g + 1]);
    const real asum = al[0] + al[1], pa0 = p.pi_a0[g];
    {
      real lg0, lg1, lgs, d0, d1, ds;
      cm[0] = al[0] / asum * pa0;
      cm[1] = al[1] / asum * pa0;
      lgamma_digamma(cm[0], lg0, d0);
      lgamma_digamma(cm[1], lg1, d1);
      lgamma_digamma(cm[0] + cm[1], lgs, ds);
      lg_cm = lgs - lg0 - lg1;
      dgd_cm[0] = ds - d0; dgd_cm[1] = ds - d1;
      cg[0] = Num<real>::fmax(cm[0], eps);
      cg[1] = Num<real>::fmax(cm[1], eps);
      if (cg[0] == cm[0] && cg[1] == cm[1]) {
        lg_cg = lg_cm;
        dgd_cg[0] = dgd_cm[0]; dgd_cg[1] = dgd_cm[1];
      } else {
        lgamma_digamma(cg[0], lg0, d0);
        lgamma_digamma(cg[1], lg1, d1);
        lgamma_digamma(cg[0] + cg[1], lgs, ds);
        lg_cg = lgs - lg0 - lg1;
        dgd_cg[0] = ds - d0; dgd_cg[1] = ds - d1;
      }
    }
    GammaMT<real> mt0, mt1;
    if (!p.pi_in) {
      mt0.init(cg[0]);
      mt1.init(cg[1]);
    }
    // abundance sites: q0[g] and the library-wide sums
    const real c = Num<real>::exp(p.q0_u[g]);
    const double Csum = s_sums[R];
    real d_c = real(0), dmu1 = real(0);
    // float: psi(c + 1) - psi(sum q0), the guide-only part of the pathwise derivative of a draw at the lower clamp (below)
    real psi_diff = real(0);
    if (sizeof(real) == 4) psi_diff = digamma_full(c + real(1)) - digamma_full(real(Csum));
    // growth of the two alleles up to each control condition (survival_model.py:326-333): per guide, not per replicate
    real wc0[BEAN_SURV_MAX_CTRL], wc1[BEAN_SURV_MAX_CTRL];
#pragma unroll
    for (int ci = 0; ci < BEAN_SURV_MAX_CTRL; ++ci) {
      wc0[ci] = ci < p.n_ctrl ? Num<real>::exp(mu0 * p.t_ctrl[ci]) : real(0);
      wc1[ci] = ci < p.n_ctrl ? Num<real>::exp(mu1 * p.t_ctrl[ci]) : real(0);
    }
    for (int r = 0; r < R; ++r) {
      const bool rmask = p.row_mask[(size_t)r * p.G + g] != 0;
      // ---- initial abundance: guide draw x ~ Dirichlet(q0) over all guides, model observes `obs` under the same Dirichlet
      {
        real xq;
        if (p.q0_in) {
          xq = p.q0_in[(size_t)r * p.G + g];
        } else {
          xq = real((double)p.gamma_cur[(size_t)r * p.G + g] / s_sums[r]);
          xq = Num<real>::fmin(Num<real>::fmax(xq, Lim<real>::tiny()), Lim<real>::one_minus());
        }
        const real lx = log_pos(xq);
        const real dl = p.log_obs[(size_t)r * p.G + g] - lx;
        elbo_g += (c - real(1)) * dl;
        // pathwise derivative of the draw w.r.t. q0 (torch _Dirichlet_backward with sum_h x_h gout_h = -(C - G)).  With q0 ~ 1/G
        // nearly every draw sits at the sampler's lower clamp (1.2e-38): torch's small-x series then reduces to its first term,
        // x / c (psi(c + 1) - psi(C) - ln x) to 1e-12 relative, whose guide-only part is hoisted (float path; the double
        // kernels evaluate torch's expression as written)
        double D;
        if (sizeof(real) == 4 && xq < real(1e-12) && Csum * (double)xq < 2.5)
          D = (double)(xq / c * (psi_diff - lx));
        else
          D = dirichlet_grad_any<false>((double)xq, (double)c, Csum - (double)c);
        d_c += dl + real(D * (-(double)(c - real(1)) / (double)xq + (Csum - p.n_guides_total)));
      }
      // ---- pi ~ Dirichlet(cg) (a Beta draw)
      real pi0, pi1;
      if (p.pi_in) {
        pi0 = p.pi_in[((size_t)g * R + r) * 2];
        pi1 = p.pi_in[((size_t)g * R + r) * 2 + 1];
      } else {
        sample_pi2(p.seed, (uint32_t)g + p.guide_offset, (uint32_t)r, p.step, mt0, mt1, pi0, pi1, &p.rk);
      }
      if (p.pi_out) {
        p.pi_out[((size_t)g * R + r) * 2] = pi0;
        p.pi_out[((size_t)g * R + r) * 2 + 1] = pi1;
      }
      real e[NB], de[NB];
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        e[b] = pi0 * P0[b] + pi1 * P1[b];  // survival_model.py:364-367
        de[b] = real(0);
      }
      // ---- Dirichlet-Multinomial rows of the count layers (survival_model.py:376-424)
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
        const real inv = Num<real>::rcp(S + eps);
        real Asum = real(0);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          frac[b] = (pb[b] + eps / real(B)) * inv;
          const real raw = frac[b] * a0 * p.t.smask[r * B + b];
          live[b] = raw >= eps;
          ab[b] = (b < B) ? (live[b] ? raw : eps) : real(0);
          Asum += ab[b];
        }
        elbo_g += dm_row_kl<real, NB>(B, xb, ab, N, Asum, gb);
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
      real go0 = real(0), go1 = real(0);
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        go0 += de[b] * P0[b];
        go1 += de[b] * P1[b];
        dP1[b] += de[b] * pi1;
      }
      // the guide's Dirichlet(pi; cg) (unmasked, survival_model.py:699-712) and the model's Dirichlet(pi; cm) (under repguide_mask,
      // :313-322) as their DIFFERENCE: identically zero -- value and gradients -- for an unclamped guide inside the mask
      if (!(rmask && cg[0] == cm[0] && cg[1] == cm[1])) {
        const real lp0 = log_pos(pi0), lp1 = log_pos(pi1);
        const real ip0 = Num<real>::rcp(pi0), ip1 = Num<real>::rcp(pi1);
        elbo_g -= lg_cg + (cg[0] - real(1)) * lp0 + (cg[1] - real(1)) * lp1;
        go0 -= (cg[0] - real(1)) * ip0;
        go1 -= (cg[1] - real(1)) * ip1;
        dcg[0] -= dgd_cg[0] + lp0;
        dcg[1] -= dgd_cg[1] + lp1;
        if (rmask) {
          elbo_g += lg_cm + (cm[0] - real(1)) * lp0 + (cm[1] - real(1)) * lp1;
          go0 += (cm[0] - real(1)) * ip0;
          go1 += (cm[1] - real(1)) * ip1;
          dcm[0] += dgd_cm[0] + lp0;
          dcm[1] += dgd_cm[1] + lp1;
        }
      }
      if (rmask) {
        // Multinomial on pi exp(mu t_c) under repguide_mask (survival_model.py:323-346)
        const real lo = p.prob_eps, hi = real(1) - p.prob_eps;
#pragma unroll
        for (int ci = 0; ci < BEAN_SURV_MAX_CTRL; ++ci) {
          if (ci >= p.n_ctrl) break;
          const typename Vec2<real>::type ac =
              reinterpret_cast<const typename Vec2<real>::type*>(p.allele_counts)[((size_t)r * p.n_ctrl + ci) * p.G + g];
          const real q0 = pi0 * wc0[ci], q1 = pi1 * wc1[ci];
          const real iSq = Num<real>::rcp(q0 + q1), n0 = q0 * iSq, n1 = q1 * iSq;
          const real c0 = Num<real>::fmin(Num<real>::fmax(n0, lo), hi), c1 = Num<real>::fmin(Num<real>::fmax(n1, lo), hi);
          if (ac.x != real(0)) elbo_g += ac.x * log_unit(c0);
          if (ac.y != real(0)) elbo_g += ac.y * log_unit(c1);
          const real h0 = (n0 >= lo && n0 <= hi) ? Num<real>::div(ac.x, n0) : real(0), h1 = (n1 >= lo && n1 <= hi) ? Num<real>::div(ac.y, n1) : real(0);
          const real hbar = h0 * n0 + h1 * n1;
          const real dq0 = (h0 - hbar) * iSq, dq1 = (h1 - hbar) * iSq;
          go0 += dq0 * wc0[ci];
          go1 += dq1 * wc1[ci];
          dmu1 += dq1 * q1 * p.t_ctrl[ci];
        }
      }
      // hand the draw with its upstream weights to svi_alpha_kernel (pathwise derivative w.r.t. the guide concentration)
      const double gbar = (double)pi0 * (double)go0 + (double)pi1 * (double)go1;
      typename Vec4<real>::type rec;
      rec.x = pi0; rec.y = pi1; rec.z = real((double)go0 - gbar); rec.w = real((double)go1 - gbar);
      reinterpret_cast<typename Vec4<real>::type*>(p.pw)[(size_t)r * p.G + g] = rec;
    }
    // d ELBO / d (edited growth rate): through exp(mu1 t_b) of the likelihood + the Multinomial part above
#pragma unroll
    for (int b = 0; b < NB; ++b)
      if (b < B) dmu1 += dP1[b] * P1[b] * p.t.tp[b];
    p.d_guide[g] = dmu1;
    {
      typename Vec4<real>::type rec;
      rec.x = dcm[0]; rec.y = dcm[1]; rec.z = dcg[0]; rec.w = dcg[1];
      reinterpret_cast<typename Vec4<real>::type*>(p.dconc)[g] = rec;
    }
    // q0: gradient of the loss w.r.t. log q0, ClippedAdam, then the next step's draws from the updated value
    const real gq = -(d_c * c);
    if (p.q0_grad) p.q0_grad[g] = gq;
    c_next = c;
    if (p.apply_update) {
      real th = p.q0_u[g], m = p.q0_m[g], vv = p.q0_v[g];
      clipped_adam(p, gq, th, m, vv, bad);
      p.q0_u[g] = th; p.q0_m[g] = m; p.q0_v[g] = vv;
      c_next = Num<real>::exp(th);
    }
    elbo = (double)elbo_g;
  }
  note_nonfinite(p.nonfinite, p.step, 0xffffffffu, bad);
  const double tot = warp_sum(elbo);
  if ((threadIdx.x & 31) == 0) p.partial[(blockIdx.x * SVI_THREADS + threadIdx.x) / SVI_WARP] = tot;
  if (p.apply_update && p.gamma_next) draw_abundance(p, g, owns, c_next, p.step + 1u);
}

template <typename real>
static int survival_run(const BeanScreen* s, const BeanSviState* state, const BeanSurvivalState* sv, const BeanSviConfig* cfg,
                        const BeanSviNoise* noise, const BeanSurvivalNoise* snoise, int32_t first_step, int32_t n_steps, void* stream) {
  int rc = validate_screen(s);
  if (rc != BEAN_OK) return rc;
  BEAN_REQUIRE(state && sv && cfg, BEAN_EINVAL, "state / survival state / cfg is NULL");
  BEAN_REQUIRE(s->mode == BEAN_MODE_SURVIVAL, BEAN_EINVAL, "bean_svi_survival_run needs a survival screen");
  BEAN_REQUIRE(state->n_variants > 0 && state->guide_variant && state->variant_ptr, BEAN_EINVAL, "variant CSR missing");
  BEAN_REQUIRE(state->var_params && state->var_m && state->var_v && state->d_guide && state->partial && state->counter && state->loss,
               BEAN_EINVAL, "variant parameter / scratch buffers must be non-NULL");
  BEAN_REQUIRE(state->allele_counts && state->pi_a0 && state->alpha_u && state->alpha_m && state->alpha_v && state->pw && state->dconc,
               BEAN_EINVAL, "alpha_pi buffers / hand-over scratch must be non-NULL");
  BEAN_REQUIRE(sv->q0_u && sv->q0_m && sv->q0_v && sv->log_obs && sv->gamma[0] && sv->gamma[1] && sv->sums[0] && sv->sums[1] && sv->abund_partial,
               BEAN_EINVAL, "abundance buffers must be non-NULL");
  BEAN_REQUIRE(sv->n_controls >= 1 && sv->n_controls <= BEAN_SURV_MAX_CTRL, BEAN_EINVAL, "n_controls %d out of range [1, %d]", sv->n_controls,
               BEAN_SURV_MAX_CTRL);
  BEAN_REQUIRE(sv->control_time != nullptr, BEAN_EINVAL, "control_time is NULL");
  BEAN_REQUIRE(aligned16(state->pw) && aligned16(state->dconc), BEAN_EALIGN, "pw / dconc are not 16-byte aligned");
  BEAN_REQUIRE(first_step >= 0 && n_steps >= 0 && first_step + n_steps <= state->loss_capacity, BEAN_EINVAL, "bad step range %d + %d (capacity %d)",
               first_step, n_steps, state->loss_capacity);

  SviParams<real> p{};  // zero: every optional pointer NULL, every mode flag off
  memset(&p, 0, sizeof(p));
  p.G = s->n_guides; p.R = s->n_reps; p.B = s->n_bins; p.L = s->n_layers; p.T = state->n_variants;
  p.mixture = 1; p.has_sd = 0; p.mu_prior_normal = cfg->mu_prior_normal; p.apply_update = cfg->apply_update;
  p.seed = cfg->seed; p.guide_offset = cfg->guide_offset; p.variant_offset = cfg->variant_offset;
  philox_round_keys(p.seed, p.rk);
  p.mask_thres = real(s->mask_thres);
  p.x = static_cast<const real*>(s->x);
  p.a0 = static_cast<const real*>(s->a0);
  p.row_mask = s->row_mask;
  p.guide_variant = state->guide_variant; p.variant_ptr = state->variant_ptr;
  p.allele_counts = static_cast<const real*>(state->allele_counts);
  p.pi_a0 = static_cast<const real*>(state->pi_a0);
  p.var_params = static_cast<real*>(state->var_params); p.var_m = static_cast<real*>(state->var_m); p.var_v = static_cast<real*>(state->var_v);
  p.alpha_u = static_cast<real*>(state->alpha_u); p.alpha_m = static_cast<real*>(state->alpha_m); p.alpha_v = static_cast<real*>(state->alpha_v);
  p.d_guide = static_cast<real*>(state->d_guide);
  p.var_grad = static_cast<real*>(state->var_grad);
  p.alpha_grad = static_cast<real*>(state->alpha_grad);
  p.pw = static_cast<real*>(state->pw); p.dconc = static_cast<real*>(state->dconc);
  p.partial = state->partial; p.counter = state->counter; p.loss = state->loss;
  p.nonfinite = sv->nonfinite_step ? sv->nonfinite_step : state->nonfinite_step;
  p.n_partial_guide = (p.G + SVI_THREADS - 1) / SVI_THREADS * (SVI_THREADS / SVI_WARP);
  p.n_partial_var = (p.T + VAR_PER_CTA - 1) / VAR_PER_CTA;
  p.eps_mu = noise ? static_cast<const real*>(noise->eps_mu) : nullptr;
  p.eps_sd = nullptr;
  p.pi_in = noise ? static_cast<const real*>(noise->pi) : nullptr;
  p.eps_out = noise ? static_cast<real*>(noise->eps_out) : nullptr;
  p.pi_out = noise ? static_cast<real*>(noise->pi_out) : nullptr;
  p.eps_negctrl = snoise ? static_cast<const real*>(snoise->eps_negctrl) : nullptr;
  p.q0_in = snoise ? static_cast<const real*>(snoise->q0) : nullptr;
  p.mu_prior_loc = real(cfg->mu_prior_loc); p.mu_prior_scale = real(cfg->mu_prior_scale);
  p.sd_prior_loc = real(0); p.sd_prior_scale = real(1);
  p.mu_prior_loc_v = static_cast<const real*>(state->mu_prior_loc_v);
  p.mu_prior_scale_v = static_cast<const real*>(state->mu_prior_scale_v);
  p.beta1 = real(cfg->beta1); p.beta2 = real(cfg->beta2); p.adam_eps = real(cfg->adam_eps); p.clip = real(cfg->clip);
  p.ll_const = cfg->ll_const;
  p.prob_eps = cfg->prob_clamp_eps > 0.0 ? real(cfg->prob_clamp_eps) : Lim<real>::eps();
  fill_tables(s, p.t);
  p.n_ctrl = sv->n_controls;
  for (int c = 0; c < BEAN_SURV_MAX_CTRL; ++c) p.t_ctrl[c] = c < sv->n_controls ? real(sv->control_time[c]) : real(0);
  p.negctrl_loc = real(sv->negctrl_loc); p.negctrl_scale = real(sv->negctrl_scale);
  p.n_guides_total = sv->n_guides_total > 0 ? (double)sv->n_guides_total : (double)p.G;
  p.log_obs = static_cast<const real*>(sv->log_obs);
  p.q0_u = static_cast<real*>(sv->q0_u); p.q0_m = static_cast<real*>(sv->q0_m); p.q0_v = static_cast<real*>(sv->q0_v);
  p.q0_grad = static_cast<real*>(sv->q0_grad);
  p.abund_partial = sv->abund_partial;
  p.n_abund_partial = p.n_partial_guide;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = (p.G + SVI_THREADS - 1) / SVI_THREADS;
  // device-side exchange of the sums (sharded guides): whole, updating steps only; the first step of a call reads `sums`
  p.peer_world = 0; p.peer_rank = 0; p.peer_consume = 0;
  for (int k = 0; k < BEAN_MAX_PEERS; ++k) p.peer_buf[k] = nullptr;
  if (sv->peers && sv->peers->world > 1 && cfg->phases == 0 && cfg->apply_update && sv->prime == BEAN_SURV_PRIME_NONE) {
    BEAN_REQUIRE(sv->peers->world <= BEAN_MAX_PEERS && sv->peers->rank >= 0 && sv->peers->rank < sv->peers->world, BEAN_EINVAL,
                 "peer exchange: world %d / rank %d out of range", sv->peers->world, sv->peers->rank);
    BEAN_REQUIRE(s->n_reps + 1 <= BEAN_PEER_MAX_VALS, BEAN_EINVAL, "peer exchange: n_reps + 1 > %d", BEAN_PEER_MAX_VALS);
    p.peer_world = sv->peers->world; p.peer_rank = sv->peers->rank;
    for (int k = 0; k < p.peer_world; ++k) {
      BEAN_REQUIRE(sv->peers->buf[k] != nullptr, BEAN_EINVAL, "peer exchange: buffer of rank %d is NULL", k);
      p.peer_buf[k] = static_cast<BeanPeerBuffer*>(sv->peers->buf[k]);
    }
  }
  for (int i = 0; i < n_steps; ++i) {
    const int t = first_step + i;
    p.step = (uint32_t)t;
    p.peer_consume = i > 0 ? 1 : 0;
    const double lr = cfg->lr0 * pow(cfg->lrd, (double)(t + 1));
    p.step_size = real(lr * sqrt(1.0 - pow(cfg->beta2, (double)(t + 1))) / (1.0 - pow(cfg->beta1, (double)(t + 1))));
    // the abundance draw of step t lives in buffer t & 1 (written by the step before, or primed here)
    const int cur = t & 1;
    if (sv->prime != BEAN_SURV_PRIME_NONE && i == 0) {
      p.gamma_next = static_cast<real*>(sv->gamma[cur]);
      p.sums_next = sv->sums[cur];
      surv_prime_kernel<real><<<grid, SVI_THREADS, 0, st>>>(p);
      surv_sums_kernel<real><<<1, VAR_THREADS, 0, st>>>(p);
      if (sv->prime == BEAN_SURV_PRIME_ONLY) break;  // sharded guides: the host all-reduces sums[cur] before the step runs
    }
    p.gamma_cur = static_cast<const real*>(sv->gamma[cur]);
    p.sums_cur = sv->sums[cur];
    p.gamma_next = cfg->apply_update ? static_cast<real*>(sv->gamma[cur ^ 1]) : nullptr;
    p.sums_next = cfg->apply_update ? sv->sums[cur ^ 1] : nullptr;
    // phases: 0 = the whole step; otherwise a bit mask (1 guide kernel, 2 variant kernel, 4 alpha kernel) so that a benchmark
    // can time each kernel alone with CUDA events
    const int ph = cfg->phases == 0 ? 7 : cfg->phases;
    if (ph & 1) {
      if (p.B == 3)
        launch_after(surv_guide_kernel<real, 3, true>, grid, SVI_THREADS, st, p);
      else if (p.B <= 4)
        launch_after(surv_guide_kernel<real, 4, false>, grid, SVI_THREADS, st, p);
      else
        launch_after(surv_guide_kernel<real, BEAN_MAX_BINS, false>, grid, SVI_THREADS, st, p);
    }
    if (ph & 4) launch_after(svi_alpha_kernel<real>, (p.G + ALPHA_THREADS - 1) / ALPHA_THREADS, ALPHA_THREADS, st, p);
    if (ph & 2) launch_after(svi_variant_kernel<real>, p.n_partial_var, VAR_THREADS, st, p);
  }
  BEAN_CUDA(cudaPeekAtLastError());
  return BEAN_OK;
}

}  // namespace bean

extern "C" {
int bean_svi_survival_run_f32(const BeanScreen* s, const BeanSviState* st, const BeanSurvivalState* sv, const BeanSviConfig* c,
                              const BeanSviNoise* n, const BeanSurvivalNoise* sn, int32_t first_step, int32_t n_steps, void* stream) {
  return bean::survival_run<float>(s, st, sv, c, n, sn, first_step, n_steps, stream);
}
int bean_svi_survival_run_f64(const BeanScreen* s, const BeanSviState* st, const BeanSurvivalState* sv, const BeanSviConfig* c,
                              const BeanSviNoise* n, const BeanSurvivalNoise* sn, int32_t first_step, int32_t n_steps, void* stream) {
  return bean::survival_run<double>(s, st, sv, c, n, sn, first_step, n_steps, stream);
}
}
