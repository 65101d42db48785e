// bean_svi.cu -- the fused SVI step of the variant sorting models (Normal / ControlNormal / MixtureNormal).
//
// Per step, three kernels (two for the Normal models) and no host round trip (reference: one `svi.step`,
// bean/model/run.py:376-380, ~2,500 eager torch op dispatches):
//
//   svi_guide_kernel   one thread per guide, looping over its replicates with everything in registers:
//       draw (mu, sd) of its variant and pi[r] ~ Dirichlet (counter-based Philox), Normal-CDF bin masses,
//       allele mixture, get_alpha + Dirichlet-Multinomial of both count layers with their digamma
//       differences, the Dirichlet / Multinomial editing-rate sites, per-guide d ELBO / d(mu, sd), ELBO partial
//       per warp; hands every draw (pi0, pi1) with its upstream weights to the alpha kernel.
//   svi_alpha_kernel   (MixtureNormal) one thread per guide: the pathwise Dirichlet derivative of each draw
//       (saddle-point pairs in double, the other regimes through a per-warp queue), the alpha_pi gradient AND
//       its ClippedAdam update (alpha_pi is per-guide, so it never leaves the thread).
//   svi_variant_kernel 8 lanes per variant: segmented reduction of the per-guide gradients over the CSR
//       variant range (no atomics; guides of a variant are contiguous, data_class.py:511-532), prior and
//       entropy terms, ClippedAdam on (mu_loc, mu_scale, sd_loc, sd_scale), and -- in the last CTA to
//       finish -- the deterministic reduction of all ELBO partials into loss[t].
#include "bean_svi_shared.cuh"

namespace bean {

// MixtureNormal: the pathwise Dirichlet derivative and the alpha_pi update run in `svi_alpha_kernel`; this kernel hands
// over every draw with its upstream weights (16 B per replicate) and the rest of the concentration gradient.  Two small
// instruction footprints instead of one large one (the I-cache is 32 KB per SM), at +0.26 GB of HBM traffic per step:
// 0.68 ms per step against 1.20 for the single kernel that did both (DESIGN section 5).
//
// FAST: the screen has exactly NB bins and no masked sample (sample_mask all ones: every screen without `bean qc` sample
// drops).  The bin loops then carry no `b < B` predicates, the per-sample size factors come from a shared-memory table as
// one 128-bit load per row instead of NB constant-bank loads with computed addresses, and the sample-mask multiplies are
// gone -- together a third of the instructions of the get_alpha section (profiles/r2b_guide_source_top.txt: that section,
// not the special functions, was the largest single block of the kernel after the round-2 instruction diet).
template <typename real, int NB, bool MIXTURE, bool ACC, int FAST>
__global__ void __launch_bounds__(SVI_THREADS, sizeof(real) == 4 ? SVI_GUIDE_MIN_CTAS_F32 : SVI_GUIDE_MIN_CTAS_F64) svi_guide_kernel(const SviParams<real> p) {
  __shared__ __align__(16) real s_sf[FAST ? BEAN_MAX_LAYERS * BEAN_MAX_RB : 1];  // [l][r][b] size factors
  // STAGE (float, 4 bins, mixture): the count rows and reporter counts of replicate r + 1 are copied global -> shared with
  // cp.async while replicate r is evaluated, double-buffered per thread; a row is then one LDS.128 (~30 cycles) instead of an
  // LDG.128 whose ~600-cycle latency sat in the middle of the replicate's dependency chain (ncu r2f: long-scoreboard stalls
  // 3.0 per issue, the largest stall reason, with only 32 warps per SM to hide them)
#ifdef BEAN_NO_STAGE
  constexpr bool STAGE = false;
#else
  constexpr bool STAGE = FAST && MIXTURE && NB == 4 && sizeof(real) == 4;
#endif
  __shared__ __align__(16) float4 s_x[STAGE ? 2 * BEAN_MAX_LAYERS * SVI_THREADS : 1];  // [buffer][layer][thread]
  __shared__ __align__(8) float2 s_ac[STAGE ? 2 * SVI_THREADS : 1];                    // [buffer][thread]
  grid_dependency_wait();
  const int g = blockIdx.x * SVI_THREADS + threadIdx.x;
  const int R = p.R, B = FAST ? NB : p.B;
  constexpr bool LFIX = FAST == 2;  // both count layers present (all reads + barcode-matched reads): L is a constant
  const int L = LFIX ? 2 : p.L;
  const real eps = real(1e-5);
  double elbo = 0.0;
  bool bad = false;  // a ClippedAdam input of this thread was NaN / inf
  if (FAST) {
    for (int i = threadIdx.x; i < L * R * NB; i += SVI_THREADS) s_sf[i] = p.t.sf[i / (R * NB)][i % (R * NB)];
    __syncthreads();
  }
  if (g < p.G) {
    const int v = p.guide_variant[g];
    real mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, log_sd;
    variant_draw(p, v, mu_t, sd_t, e_mu, e_sd, mu_scale, sd_scale, log_sd);
    const real sigma = p.sd_is_sqrt ? Num<real>::sqrt(sd_t) : sd_t;  // model.py:92-98
    // bin masses of the edited allele now; their (mu, sd) derivatives are recomputed in the epilogue (two exp per bin)
    // instead of being carried through the replicate loop in 2 NB registers
    real P1[NB], dP[NB];
    {
      BinMasses<real> bm(mu_t, sigma);
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        P1[b] = dP[b] = real(0);
        if (b < B) P1[b] = bm.next(p.t.thr_u[b], p.t.thr_l[b], b > 0 && p.t.thr_l[b] == p.t.thr_u[b > 0 ? b - 1 : 0]);
      }
    }
    // editing-rate concentrations (model.py:449 / :835): model = alpha/sum*pi_a0, guide = clamp(model, 1e-5)
    real al[2] = {real(1), real(1)}, cm[2] = {real(1), real(1)}, cg[2] = {real(1), real(1)};
    real lg_cm = real(0), lg_cg = real(0), dgd_cm[2] = {}, dgd_cg[2] = {}, dcm[2] = {}, dcg[2] = {};  // dgd = psi(sum) - psi(c_a)
    real asum = real(2), pa0 = real(0);
    if (MIXTURE) {
      al[0] = Num<real>::exp(p.alpha_u[2 * (size_t)g]);
      al[1] = Num<real>::exp(p.alpha_u[2 * (size_t)g + 1]);
      asum = al[0] + al[1];
      pa0 = p.pi_a0[g];
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
    // --scale-by-acc: per-guide logit-space noise (utils.py:133-178)
    constexpr bool acc = MIXTURE && ACC;  // compiled out of the plain kernels (code size)
    const real PI_NOISE_SD = real(0.655);
    real kacc = real(1), n_eps = real(0), n_loc = real(0), n_scale = PI_NOISE_SD, n_val = real(0), dnoise = real(0);
    if (acc) {
      kacc = p.acc_k[g];
      n_eps = p.eps_noise ? p.eps_noise[g] : real(guide_noise(p.seed, (uint32_t)g + p.guide_offset, p.step));
      if (p.fit_noise) {
        n_loc = p.noise_u[g];
        n_scale = Num<real>::exp(p.noise_u[(size_t)p.G + g]);
      }
      n_val = n_loc + n_scale * n_eps;
    }
    GammaMT<real> mt0, mt1;
    if (MIXTURE && !p.pi_in) {
      mt0.init(cg[0]);
      mt1.init(cg[1]);
    }
    real elbo_g = real(0);
    constexpr bool HOIST = LFIX;  // (-1 % of the kernel's time at c5, A/B in profiles/r2j_variants.jsonl)
    real a0h0 = real(0), a0h1 = real(0);  // prior precision of the guide's two rows: replicate-independent
    if (HOIST) {
      a0h0 = p.a0[g];
      a0h1 = p.a0[(size_t)p.G + g];
    }
    auto stage = [&](int r) {  // rows of both layers + reporter counts of replicate r -> buffer r & 1
      const int buf = r & 1;
#pragma unroll(LFIX ? 2 : 1)
      for (int l = 0; l < L; ++l)
        cp_async_16(&s_x[(buf * BEAN_MAX_LAYERS + l) * SVI_THREADS + threadIdx.x], p.x + (((size_t)l * R + r) * p.G + g) * 4);
      cp_async_8(&s_ac[buf * SVI_THREADS + threadIdx.x], p.allele_counts + ((size_t)r * p.G + g) * 2);
    };
    if (STAGE) {
      stage(0);
      cp_async_commit();
    }
    for (int r = 0; r < R; ++r) {
      // (all R mask bytes loaded up front into a bit mask was tried: +1 %, profiles/r2l_variants.jsonl)
      const bool rmask = p.row_mask[(size_t)r * p.G + g] != 0;  // replicate-major: a warp reads 32 consecutive bytes
      if (STAGE) {
        if (r + 1 < R) stage(r + 1);
        cp_async_commit();   // one group per iteration (possibly empty), so that "all but the newest" = replicate r has landed
        cp_async_wait<1>();
      }
      real pi0 = real(0), pi1 = real(1);
      if (MIXTURE) {
        if (p.pi_in) {
          pi0 = p.pi_in[((size_t)g * R + r) * 2];
          pi1 = p.pi_in[((size_t)g * R + r) * 2 + 1];
        } else {
          // first proposal through the inlined Philox with host-made round keys: -3 % of the kernel's time at c5
          // (profiles/r2k_variants.jsonl)
          sample_pi2(p.seed, (uint32_t)g + p.guide_offset, (uint32_t)r, p.step, mt0, mt1, pi0, pi1, &p.rk);
        }
        if (p.pi_out) {
          p.pi_out[((size_t)g * R + r) * 2] = pi0;
          p.pi_out[((size_t)g * R + r) * 2 + 1] = pi1;
        }
      }
      // allele weights seen by the likelihood: pi itself, or its accessibility-scaled, noised version
      real q0 = pi0, q1 = pi1, dq1_dpi1 = real(1), dq1_dnoise = real(0);
      if (acc) {
        const real lo3 = real(1e-3), hi3 = real(1) - real(1e-3);
        const real scaled = pi1 * kacc;                       // _scale_edited_pi
        const real den = Num<real>::fmax((real(1) - scaled) + scaled, real(1));
        const real s1 = scaled / den;
        const real c1 = Num<real>::fmin(Num<real>::fmax(s1, lo3), hi3);
        const real logit = Num<real>::log(c1 / (real(1) - c1)) + n_val;
        const real ex = Num<real>::exp(logit);
        const real praw = ex / (real(1) + ex);
        q1 = Num<real>::fmin(Num<real>::fmax(praw, lo3), hi3);
        q0 = real(1) - q1;
        dq1_dnoise = (praw >= lo3 && praw <= hi3) ? praw * (real(1) - praw) : real(0);
        dq1_dpi1 = (s1 >= lo3 && s1 <= hi3) ? dq1_dnoise * kacc / (den * c1 * (real(1) - c1)) : real(0);
      }
      real e[NB], de[NB];
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        e[b] = MIXTURE ? q0 * p.p_wt[b] + q1 * P1[b] : P1[b];  // model.py:495-499
        de[b] = real(0);
      }
#ifdef BEAN_UNROLL_LAYERS
#pragma unroll(LFIX ? 2 : 1)
#else
#pragma unroll 1
#endif
      for (int l = 0; l < L; ++l) {
        // x[l][r][g][b]: the rows of 32 consecutive guides are contiguous, so a warp's loads coalesce; with B = 4 a row
        // is one 128-bit load
        const real* xr = p.x + (((size_t)l * R + r) * p.G + g) * B;
        real xb[NB], sfb[NB], smb[NB], pb[NB], ab[NB], frac[NB], gb[NB];
        bool live[NB];
        real N = real(0), S = real(0);
        if (STAGE) {
          const float4 q = s_x[((r & 1) * BEAN_MAX_LAYERS + l) * SVI_THREADS + threadIdx.x];
          xb[0] = q.x; xb[1] = q.y; xb[2] = q.z; xb[3] = q.w;
        } else if (NB == 4 && B == 4) {
          const typename Vec4<real>::type q = *reinterpret_cast<const typename Vec4<real>::type*>(xr);
          xb[0] = q.x; xb[1] = q.y; xb[2] = q.z; xb[3] = q.w;
        } else {
#pragma unroll
          for (int b = 0; b < NB; ++b) xb[b] = b < B ? xr[b] : real(0);
        }
        if (FAST && NB == 4) {
          const typename Vec4<real>::type q = reinterpret_cast<const typename Vec4<real>::type*>(s_sf)[l * R + r];
          sfb[0] = q.x; sfb[1] = q.y; sfb[2] = q.z; sfb[3] = q.w;
        } else {
#pragma unroll
          for (int b = 0; b < NB; ++b) sfb[b] = FAST ? s_sf[(l * R + r) * NB + b] : (b < B ? p.t.sf[l][r * B + b] : real(0));
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          smb[b] = FAST ? real(1) : (b < B ? p.t.smask[r * B + b] : real(0));
          N += xb[b];
          pb[b] = e[b] * sfb[b];
          S += pb[b];
        }
        if (!(rmask && N > p.mask_thres)) continue;  // poutine.mask: the row contributes nothing
        const real a0 = HOIST ? (l == 0 ? a0h0 : a0h1) : p.a0[(size_t)l * p.G + g];
        const real inv = Num<real>::rcp(S + eps);
        real Asum = real(0);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          frac[b] = (pb[b] + eps / real(B)) * inv;  // utils.py:19-23
          const real raw = FAST ? frac[b] * a0 : frac[b] * a0 * smb[b];
          live[b] = raw >= eps;
          ab[b] = (b < B) ? (live[b] ? raw : eps) : real(0);
          Asum += ab[b];
        }
        elbo_g += dm_row_kl<real, NB>(B, xb, ab, N, Asum, gb);
        real dot = real(0);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          gb[b] = (b < B && live[b]) ? (FAST ? gb[b] : gb[b] * smb[b]) : real(0);
          dot += gb[b] * frac[b];
        }
        const real c = a0 * inv;
#pragma unroll
        for (int b = 0; b < NB; ++b)
          if (b < B) de[b] += sfb[b] * c * (gb[b] - dot);
      }
      if (MIXTURE) {
        // d ELBO / d pi from the likelihood
        real go0 = real(0), go1 = real(0);
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          go0 += de[b] * p.p_wt[b];
          go1 += de[b] * P1[b];
          dP[b] += de[b] * q1;
        }
        if (acc) {  // chain through q1(pi1, noise), q0 = 1 - q1; pi0 does not reach the likelihood
          const real gq = go1 - go0;
          dnoise += gq * dq1_dnoise;
          go1 = gq * dq1_dpi1;
          go0 = real(0);
        }
        // The two Dirichlet sites on pi -- the guide's, unmasked, with concentration cg = clamp(cm, 1e-5) (model.py:837-847),
        // and the model's prior under poutine.mask(repguide_mask) with cm (model.py:454-463) -- are accumulated as their
        // DIFFERENCE: for an unclamped guide inside the mask (nearly all) they cancel identically, value and gradients, so
        // nothing is computed and no rounding residue of two large equal terms reaches the alpha_pi gradient.
        const bool same_conc = cg[0] == cm[0] && cg[1] == cm[1];
        real lp0 = real(0), lp1 = real(0);
        if (!(rmask && same_conc)) {
          lp0 = Num<real>::log(pi0);
          lp1 = Num<real>::log(pi1);
          const real ip0 = Num<real>::rcp(pi0), ip1 = Num<real>::rcp(pi1);
          // guide site: -log Dirichlet(pi; cg)
          elbo_g -= lg_cg + (cg[0] - real(1)) * lp0 + (cg[1] - real(1)) * lp1;
          go0 -= (cg[0] - real(1)) * ip0;
          go1 -= (cg[1] - real(1)) * ip1;
          dcg[0] -= dgd_cg[0] + lp0;
          dcg[1] -= dgd_cg[1] + lp1;
          if (rmask) {  // model site (clamped guide: the two concentrations differ)
            elbo_g += lg_cm + (cm[0] - real(1)) * lp0 + (cm[1] - real(1)) * lp1;
            go0 += (cm[0] - real(1)) * ip0;
            go1 += (cm[1] - real(1)) * ip1;
            dcm[0] += dgd_cm[0] + lp0;
            dcm[1] += dgd_cm[1] + lp1;
          }
        }
        if (rmask) {
          // Multinomial reporter counts under the mask (model.py:464-474); torch Multinomial normalises probs and clamps
          // them to [eps, 1-eps]
          real x0, x1;
          if (STAGE) {
            const float2 ac = s_ac[(r & 1) * SVI_THREADS + threadIdx.x];
            x0 = ac.x; x1 = ac.y;
          } else {
            const typename Vec2<real>::type ac = reinterpret_cast<const typename Vec2<real>::type*>(p.allele_counts)[(size_t)r * p.G + g];
            x0 = ac.x; x1 = ac.y;
          }
          const real Sp = pi0 + pi1, iSp = Num<real>::rcp(Sp), pn0 = pi0 * iSp, pn1 = pi1 * iSp;
          // torch clamps Multinomial probs to [eps, 1 - eps] of THEIR dtype; in the reference pi inherits pi_a0's dtype
          // (float64 out of the fit even on the float32 path): the host passes the eps that applies (BeanSviConfig)
          const real lo = p.prob_eps, hi = real(1) - p.prob_eps;
          const real c0 = Num<real>::fmin(Num<real>::fmax(pn0, lo), hi), c1 = Num<real>::fmin(Num<real>::fmax(pn1, lo), hi);
          const real l0 = log_unit(c0), l1 = log_unit(c1);
          elbo_g += x0 * l0 + x1 * l1;
          const real h0 = (pn0 >= lo && pn0 <= hi) ? Num<real>::div(x0, c0) : real(0), h1 = (pn1 >= lo && pn1 <= hi) ? Num<real>::div(x1, c1) : real(0);
          const real hbar = h0 * pn0 + h1 * pn1;
          go0 += (h0 - hbar) * iSp;
          go1 += (h1 - hbar) * iSp;
        }
        // pathwise derivative of pi w.r.t. the guide concentration (torch _Dirichlet_backward)
        // evaluated in double even on the float path, as torch's CPU kernel does (accscalar_t = double):
        // the saddle-point branch cancels badly in float
        if (sizeof(real) == 4) {
          // go_a - (pi0 go0 + pi1 go1) without forming the weighted mean: with s = 1 - pi0 - pi1 (a few ulp: pi is a clamped,
          // rounded normalisation) it equals s go_a + pi_b (go_a - go_b), where nothing cancels -- as accurate as the double
          // evaluation rounded to float, in 6 FP32 instructions instead of 4 conversions + 4 FP64 operations
          const real s = (real(1) - pi0) - pi1, dgo = go0 - go1;
          typename Vec4<real>::type rec;
          rec.x = pi0; rec.y = pi1; rec.z = fma(pi1, dgo, s * go0); rec.w = fma(pi0, -dgo, s * go1);
          reinterpret_cast<typename Vec4<real>::type*>(p.pw)[(size_t)r * p.G + g] = rec;
          continue;
        }
        const double gbar = (double)pi0 * (double)go0 + (double)pi1 * (double)go1;
        const double w0 = (double)go0 - gbar, w1 = (double)go1 - gbar;
        typename Vec4<real>::type rec;
        rec.x = pi0; rec.y = pi1; rec.z = real(w0); rec.w = real(w1);
        reinterpret_cast<typename Vec4<real>::type*>(p.pw)[(size_t)r * p.G + g] = rec;  // replicate-major: a warp's stores coalesce
      } else {
#pragma unroll
        for (int b = 0; b < NB; ++b) dP[b] += de[b];
      }
    }
    // per-guide gradient w.r.t. the edited allele's (mu, sd_targets); reduced per variant by the next kernel
    real dmu = real(0), dsg = real(0);
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      if (b < B) {
        real dPm, dPs;
        bin_mass_grad_sorting(p.t.thr_u[b], p.t.thr_l[b], mu_t, sigma, dPm, dPs);
        dmu += dP[b] * dPm;
        dsg += dP[b] * dPs;
      }
    }
    if (p.sd_is_sqrt) dsg *= real(0.5) / sigma;
    p.d_guide[g] = dmu;
    p.d_guide[(size_t)p.G + g] = dsg;
    if (MIXTURE) {
      typename Vec4<real>::type rec;
      rec.x = dcm[0]; rec.y = dcm[1]; rec.z = dcg[0]; rec.w = dcg[1];
      reinterpret_cast<typename Vec4<real>::type*>(p.dconc)[g] = rec;
    }
    if (acc) {
      // logit_pi_noise site: model Normal(0, 0.655); guide Normal(noise_loc, noise_scale) or the prior itself
      if (p.fit_noise) {
        const real z0 = n_val / PI_NOISE_SD;
        elbo_g += (-Num<real>::log(PI_NOISE_SD) - real(0.5) * z0 * z0) - (-Num<real>::log(n_scale) - real(0.5) * n_eps * n_eps);
        const real dE = dnoise - n_val / (PI_NOISE_SD * PI_NOISE_SD);
        const real gl = -dE, gs = -(dE * n_eps * n_scale + real(1));
        if (p.noise_grad) {
          p.noise_grad[g] = gl;
          p.noise_grad[(size_t)p.G + g] = gs;
        }
        if (p.apply_update) {
          real th = p.noise_u[g], m = p.noise_m[g], v = p.noise_v[g];
          clipped_adam(p, gl, th, m, v, bad);
          p.noise_u[g] = th; p.noise_m[g] = m; p.noise_v[g] = v;
          const size_t j = (size_t)p.G + g;
          th = p.noise_u[j]; m = p.noise_m[j]; v = p.noise_v[j];
          clipped_adam(p, gs, th, m, v, bad);
          p.noise_u[j] = th; p.noise_m[j] = m; p.noise_v[j] = v;
        }
      }
    }
    elbo = (double)elbo_g;
  }
  if (MIXTURE && ACC) note_nonfinite(p.nonfinite, p.step, 0xffffffffu, bad);
  const double tot = warp_sum(elbo);
  if ((threadIdx.x & 31) == 0) p.partial[(blockIdx.x * SVI_THREADS + threadIdx.x) / SVI_WARP] = tot;
}

template <typename real, bool MIXTURE, bool ACC>
static void launch_guide(const SviParams<real>& p, cudaStream_t st, bool guide, bool alpha, bool fast) {
  const int grid = (p.G + SVI_THREADS - 1) / SVI_THREADS;
  if (!guide) {
  } else if (fast && p.B == 4 && p.L == 2)
    launch_after(svi_guide_kernel<real, 4, MIXTURE, ACC, 2>, grid, SVI_THREADS, st, p);
  else if (fast && p.B == 4)
    launch_after(svi_guide_kernel<real, 4, MIXTURE, ACC, 1>, grid, SVI_THREADS, st, p);
  else if (fast && p.B == 5)
    launch_after(svi_guide_kernel<real, 5, MIXTURE, ACC, 1>, grid, SVI_THREADS, st, p);
  else if (p.B <= 4)
    launch_after(svi_guide_kernel<real, 4, MIXTURE, ACC, 0>, grid, SVI_THREADS, st, p);
  else if (p.B == 5)
    launch_after(svi_guide_kernel<real, 5, MIXTURE, ACC, 0>, grid, SVI_THREADS, st, p);
  else
    launch_after(svi_guide_kernel<real, BEAN_MAX_BINS, MIXTURE, ACC, 0>, grid, SVI_THREADS, st, p);
  // (one thread per (guide, replicate) with a shuffle reduction was tried for this kernel: 0.42 vs 0.27 ms)
  if (MIXTURE && alpha) launch_after(svi_alpha_kernel<real>, (p.G + ALPHA_THREADS - 1) / ALPHA_THREADS, ALPHA_THREADS, st, p);
}

template <typename real>
static int svi_run(const BeanScreen* s, const BeanSviState* state, const BeanSviConfig* cfg, const BeanSviNoise* noise,
                   int32_t first_step, int32_t n_steps, void* stream) {
  int rc = validate_screen(s);
  if (rc != BEAN_OK) return rc;
  BEAN_REQUIRE(state && cfg, BEAN_EINVAL, "state / cfg is NULL");
  BEAN_REQUIRE(s->mode == BEAN_MODE_SORTING, BEAN_EINVAL, "bean_svi_run supports the sorting models only");
  BEAN_REQUIRE(cfg->model == BEAN_MODEL_NORMAL || cfg->model == BEAN_MODEL_MIXTURE_NORMAL, BEAN_EINVAL, "bad model %d", cfg->model);
  BEAN_REQUIRE(state->n_variants > 0, BEAN_EINVAL, "n_variants must be > 0");
  BEAN_REQUIRE(state->guide_variant && state->variant_ptr, BEAN_EINVAL, "guide_variant / variant_ptr must be non-NULL");
  BEAN_REQUIRE(state->var_params && state->var_m && state->var_v, BEAN_EINVAL, "variant parameter buffers must be non-NULL");
  BEAN_REQUIRE(state->d_guide && state->partial && state->counter && state->loss, BEAN_EINVAL, "scratch buffers must be non-NULL");
  const bool mix = cfg->model == BEAN_MODEL_MIXTURE_NORMAL;
  if (mix) {
    BEAN_REQUIRE(state->allele_counts && state->pi_a0, BEAN_EINVAL, "MixtureNormal needs allele_counts / pi_a0");
    BEAN_REQUIRE(state->alpha_u && state->alpha_m && state->alpha_v, BEAN_EINVAL, "MixtureNormal needs alpha_u / alpha_m / alpha_v");
    BEAN_REQUIRE(state->pw && state->dconc, BEAN_EINVAL, "MixtureNormal needs the hand-over scratch pw / dconc");
    BEAN_REQUIRE(aligned16(state->pw) && aligned16(state->dconc), BEAN_EALIGN, "pw / dconc are not 16-byte aligned");
  }
  if (mix && state->acc_k && cfg->fit_noise)
    BEAN_REQUIRE(state->noise_u && state->noise_m && state->noise_v, BEAN_EINVAL, "fit_noise needs noise_u / noise_m / noise_v");
  if ((rc = check_step_range(first_step, n_steps, state->loss_capacity)) != BEAN_OK) return rc;
  if (noise && (rc = check_eps_pair(noise->eps_mu, noise->eps_sd)) != BEAN_OK) return rc;

  SviParams<real> p{};  // zero: every optional pointer NULL, every mode flag off
  fill_common(p, s, cfg);
  p.T = state->n_variants;
  p.mixture = mix; p.sd_is_sqrt = cfg->sd_is_sqrt; p.has_sd = 1;
  p.guide_variant = state->guide_variant;
  p.variant_ptr = state->variant_ptr;
  p.allele_counts = static_cast<const real*>(state->allele_counts);
  p.pi_a0 = static_cast<const real*>(state->pi_a0);
  p.var_params = static_cast<real*>(state->var_params);
  p.var_m = static_cast<real*>(state->var_m);
  p.var_v = static_cast<real*>(state->var_v);
  p.alpha_u = static_cast<real*>(state->alpha_u);
  p.alpha_m = static_cast<real*>(state->alpha_m);
  p.alpha_v = static_cast<real*>(state->alpha_v);
  p.acc_k = mix ? static_cast<const real*>(state->acc_k) : nullptr;
  p.noise_u = static_cast<real*>(state->noise_u);
  p.noise_m = static_cast<real*>(state->noise_m);
  p.noise_v = static_cast<real*>(state->noise_v);
  p.noise_grad = static_cast<real*>(state->noise_grad);
  p.fit_noise = cfg->fit_noise;
  p.d_guide = static_cast<real*>(state->d_guide);
  p.var_grad = static_cast<real*>(state->var_grad);
  p.alpha_grad = static_cast<real*>(state->alpha_grad);
  p.pw = static_cast<real*>(state->pw);
  p.dconc = static_cast<real*>(state->dconc);
  p.partial = state->partial;
  p.counter = state->counter;
  p.loss = state->loss;
  p.nonfinite = state->nonfinite_step;
  p.n_partial_guide = (p.G + SVI_THREADS - 1) / SVI_THREADS * (SVI_THREADS / SVI_WARP);
  p.n_partial_var = (p.T + VAR_PER_CTA - 1) / VAR_PER_CTA;
  p.eps_mu = noise ? static_cast<const real*>(noise->eps_mu) : nullptr;
  p.eps_sd = noise ? static_cast<const real*>(noise->eps_sd) : nullptr;
  p.pi_in = noise ? static_cast<const real*>(noise->pi) : nullptr;
  p.eps_noise = noise ? static_cast<const real*>(noise->eps_noise) : nullptr;
  p.eps_out = noise ? static_cast<real*>(noise->eps_out) : nullptr;
  p.pi_out = noise ? static_cast<real*>(noise->pi_out) : nullptr;
  p.mu_prior_loc_v = static_cast<const real*>(state->mu_prior_loc_v);
  p.mu_prior_scale_v = static_cast<const real*>(state->mu_prior_scale_v);
  p.sd_prior_loc_v = static_cast<const real*>(state->sd_prior_loc_v);
  p.sd_prior_scale_v = static_cast<const real*>(state->sd_prior_scale_v);
  for (int b = 0; b < BEAN_MAX_BINS; ++b) {
    double m = 0.0;
    if (b < s->n_bins) {  // wild-type allele N(0, 1): Phi(t_u) - Phi(t_l), as get_std_normal_prob does in float64
      const double cu = isinf(s->upper_thres[b]) ? 1.0 : 0.5 * (1.0 + erf(s->upper_thres[b] * 0.70710678118654752440));
      const double cl = isinf(s->lower_thres[b]) ? 0.0 : 0.5 * (1.0 + erf(s->lower_thres[b] * 0.70710678118654752440));
      m = cu - cl;
    }
    p.p_wt[b] = real(m);
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // FAST kernels: exactly 4 or 5 bins and no masked sample
  bool fast = (s->n_bins == 4 || s->n_bins == 5) && !cfg->force_generic;
  for (int i = 0; i < s->n_reps * s->n_bins; ++i) fast = fast && s->sample_mask[i] == 1.0;
  for (int i = 0; i < n_steps; ++i) {
    const int t = first_step + i;
    p.step = (uint32_t)t;
    p.step_size = adam_step_size<real>(cfg, t);
    const int ph = step_phases(cfg);
    const bool do_guide = ph & 1, do_alpha = ph & 4;
    if (mix && p.acc_k) launch_guide<real, true, true>(p, st, do_guide, do_alpha, fast);
    else if (mix) launch_guide<real, true, false>(p, st, do_guide, do_alpha, fast);
    else launch_guide<real, false, false>(p, st, do_guide, false, fast);
    if (ph & 2) launch_after(svi_variant_kernel<real>, p.n_partial_var, VAR_THREADS, st, p);
  }
  BEAN_CUDA(cudaPeekAtLastError());
  return BEAN_OK;
}

}  // namespace bean

extern "C" {

int bean_svi_num_partials(int32_t n_guides, int32_t n_variants) {
  return (n_guides + bean::SVI_THREADS - 1) / bean::SVI_THREADS * (bean::SVI_THREADS / bean::SVI_WARP) + (n_variants + bean::VAR_PER_CTA - 1) / bean::VAR_PER_CTA;
}
int bean_svi_run_f32(const BeanScreen* s, const BeanSviState* st, const BeanSviConfig* c, const BeanSviNoise* n,
                     int32_t first_step, int32_t n_steps, void* stream) {
  return bean::svi_run<float>(s, st, c, n, first_step, n_steps, stream);
}
int bean_svi_run_f64(const BeanScreen* s, const BeanSviState* st, const BeanSviConfig* c, const BeanSviNoise* n,
                     int32_t first_step, int32_t n_steps, void* stream) {
  return bean::svi_run<double>(s, st, c, n, first_step, n_steps, stream);
}

}  // extern "C"
