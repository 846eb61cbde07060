/* oracle/cf_hbtq.c -- CPU restatement of the HBT Fourier sums of the linear-delta-f emission function.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/ and tools may load this library (oracle/cf_hbtq.py compiles it on first use); the product never links or calls it.
 * It is one translation unit with cf_hbt.c and cf_oracle.c (included below): the cell set-up and the weight are those of
 * cfo_hbt_moments, statement for statement, so Re[d][0] equals its S0 (and cfo_smooth_vh) bin for bin, bit for bit.
 * Per evaluation (cell, slot), with the weight w and the LCMS coordinates (o, s, l) of cfo_hbt_moments, and per ray d, q point k:
 *   q = k dq d,   theta = (q_o o + q_s s + q_l l) / hbarC   (= -q.x with q^0 = beta_perp q_o),   direct cos / sin, no recurrence
 * Re[d][k][bin] += prefactor * degeneracy * sum_slots w cos(theta), Im likewise with sin, arrays [n_dir][n_q][n_bins].
 * W_abs (optional) [n_bins] receives the same sum of the weight's |terms| magnitude (cfo_smooth_vh's conditioning): the floor of the
 * rounding noise of every Re and Im sum of the bin.
 * dir: [n_dir][3] (o, s, l).  Returns #cells skipped (u.dsigma <= 0) or a negative error code. */
#include "cf_hbt.c"

int64_t cfo_hbt_fourier(const cfo_flags *fl, const cfo_cells *c, const double *xpos, const double *ypos, const cfo_species *sp,
                        const cfo_grid *g, const cfo_df_tables *tab, int n_dir, int n_q, double dq, const double *dir,
                        double *Re, double *Im, double *W_abs)
{
  if (fl->df_mode != 1 && fl->df_mode != 2) return -1;
  if (fl->include_baryon) return -2;
  if (n_dir < 1 || n_q < 1) return -4;
  const double prefactor = pow(2.0 * M_PI * hbarC, -3);
  const int npart = sp->n, npT = g->n_pT, nphi = g->n_phi;
  int y_pts, eta_pts; grid_dims(fl, g, &y_pts, &eta_pts);
  const int64_t n = c->n_cells, n_bins = (int64_t)npart * npT * nphi * g->n_y;
  const int nq = n_dir * n_q;
  spline_cache sc; cache_build(&sc, tab);
  cell_setup *cs = (cell_setup *)malloc(sizeof(cell_setup) * (size_t)(n > 0 ? n : 1));
  int64_t skipped = 0; int bad = 0;
  for (int64_t i = 0; i < n; i++) {                      /* the set-up loop of cfo_smooth_vh */
    cell_setup *s = &cs[i];
    cell_common(fl, c, i, s);
    if (s->skip) { skipped++; continue; }
    if (df_eval(&sc, fl->df_mode, s->T, s->E, s->P, s->bulkPi, &s->df)) bad = 1;
    if (fl->df_mode == 1) {
      s->shear_coeff = 0.5 / (s->T * s->T * (s->E + s->P));
      s->bulk0_coeff = s->df.c0 - s->df.c2;
      s->bulk1_coeff = s->df.c1;
      s->bulk2_coeff = 4.0 * s->df.c2 - s->df.c0;
    } else {
      s->shear_coeff = 0.5 / (s->df.betapi * s->T);
      s->bulk0_coeff = s->df.F / (s->T * s->T * s->df.betabulk);
      s->bulk1_coeff = s->df.G / s->df.betabulk;
      s->bulk2_coeff = 1.0 / (3.0 * s->T * s->df.betabulk);
    }
  }
  cache_free(&sc);
  if (bad) { free(cs); return -3; }
  double *cosphi = (double *)malloc(sizeof(double) * nphi), *sinphi = (double *)malloc(sizeof(double) * nphi);
  for (int k = 0; k < nphi; k++) { cosphi[k] = cos(g->phi[k]); sinphi[k] = sin(g->phi[k]); }

  /* (species, pT) pairs in parallel: every bin's sum still runs over the cells in order, as in cfo_hbt_moments */
#pragma omp parallel for schedule(dynamic, 1) collapse(2)
  for (int ipart = 0; ipart < npart; ipart++) {
    for (int ipT = 0; ipT < npT; ipT++) {
      double mass = sp->mass[ipart], mass2 = mass * mass, sign = sp->sign[ipart];
      double degeneracy = sp->degeneracy[ipart], baryon = sp->baryon[ipart];
      double *fre = (double *)malloc(sizeof(double) * nq), *fim = (double *)malloc(sizeof(double) * nq);
      for (int64_t icell = 0; icell < n; icell++) {
        const cell_setup *s = &cs[icell];
        if (s->skip) continue;
        double chem = baryon * s->alphaB;
        const double xc = xpos[icell], yc = ypos[icell];
        double pT = g->pT[ipT];
        double mT = sqrt(mass2 + pT * pT);
        double mT_over_tau = mT / s->tau;
        const double beta = pT / mT;
        for (int iphip = 0; iphip < nphi; iphip++) {
          double px = pT * cosphi[iphip], py = pT * sinphi[iphip];
          const double so = xc * cosphi[iphip] + yc * sinphi[iphip], ss = -xc * sinphi[iphip] + yc * cosphi[iphip];
          for (int iy = 0; iy < y_pts; iy++) {
            double y = (fl->dimension == 2) ? 0.0 : g->y[iy];
            double sa = 0.0;
            for (int j = 0; j < nq; j++) { fre[j] = 0.0; fim[j] = 0.0; }
            for (int ieta = 0; ieta < eta_pts; ieta++) {
              double eta = (fl->dimension == 2) ? g->eta[ieta] : s->eta;
              double eta_weight = (fl->dimension == 2) ? g->eta_weight[ieta] : 1.0;
              double pt = mT * cosh(y - eta);
              double pn = mT_over_tau * sinh(y - eta);
              double tau2_pn = s->tau2 * pn;
              double pdotdsigma = eta_weight * (pt * s->dat + px * s->dax + py * s->day + pn * s->dan);
              if (fl->outflow && pdotdsigma <= 0.0) continue;
              double pdotu = pt * s->ut - px * s->ux - py * s->uy - tau2_pn * s->un;
              double feq = 1.0 / (exp(pdotu / s->T - chem) + sign);
              double mag = 0.0;
              double feqbar = 1.0 - sign * feq;
              double pimunu_pmu_pnu = s->pitt * pt * pt + s->pixx * px * px + s->piyy * py * py + s->pinn * tau2_pn * tau2_pn
                + 2.0 * (-(s->pitx * px + s->pity * py) * pt + s->pixy * px * py + tau2_pn * (s->pixn * px + s->piyn * py - s->pitn * pt));
              double Vmu_pmu = s->Vt * pt - s->Vx * px - s->Vy * py - s->Vn * tau2_pn;
              double df;
              if (fl->df_mode == 1) {
                double df_shear = s->shear_coeff * pimunu_pmu_pnu;
                double df_bulk = (s->bulk0_coeff * mass2 + (s->bulk1_coeff * baryon + s->bulk2_coeff * pdotu) * pdotu) * s->bulkPi;
                double df_diff = (s->df.c3 * baryon + s->df.c4 * pdotu) * Vmu_pmu;
                df = feqbar * (df_shear + df_bulk + df_diff);
                mag = fabs(s->shear_coeff) * (fabs(s->pitt) * pt * pt + fabs(s->pixx) * px * px + fabs(s->piyy) * py * py + fabs(s->pinn) * tau2_pn * tau2_pn
                      + 2.0 * ((fabs(s->pitx * px) + fabs(s->pity * py)) * pt + fabs(s->pixy * px * py) + fabs(tau2_pn) * (fabs(s->pixn * px) + fabs(s->piyn * py) + fabs(s->pitn) * pt)))
                      + (fabs(s->bulk0_coeff) * mass2 + fabs(s->bulk2_coeff) * pdotu * pdotu) * fabs(s->bulkPi) + fabs(df_diff);
              } else {
                double df_shear = s->shear_coeff * pimunu_pmu_pnu / pdotu;
                double df_bulk = (s->bulk0_coeff * pdotu + s->bulk1_coeff * baryon + s->bulk2_coeff * (pdotu - mass2 / pdotu)) * s->bulkPi;
                double df_diff = (s->baryon_enthalpy_ratio - baryon / pdotu) * Vmu_pmu / s->df.betaV;
                df = feqbar * (df_shear + df_bulk + df_diff);
                mag = fabs(s->shear_coeff) / pdotu * (fabs(s->pitt) * pt * pt + fabs(s->pixx) * px * px + fabs(s->piyy) * py * py + fabs(s->pinn) * tau2_pn * tau2_pn
                      + 2.0 * ((fabs(s->pitx * px) + fabs(s->pity * py)) * pt + fabs(s->pixy * px * py) + fabs(tau2_pn) * (fabs(s->pixn * px) + fabs(s->piyn * py) + fabs(s->pitn) * pt)))
                      + (fabs(s->bulk0_coeff) * pdotu + fabs(s->bulk2_coeff) * (pdotu + mass2 / pdotu)) * fabs(s->bulkPi) + fabs(df_diff);
              }
              int clamped = 0;
              if (fl->regulate_deltaf) { clamped = (df <= -1.0 || df >= 1.0); df = fmax(-1.0, fmin(df, 1.0)); }
              double f = feq * (1.0 + df);
              /* the weight and its |terms| magnitude, then the LCMS coordinates and the phases of this evaluation */
              const double w = pdotdsigma * f;
              const double wa = fabs(pdotdsigma) * feq * (1.0 + (clamped ? 1.0 : fabs(feqbar) * mag));
              const double tstar = s->tau * cosh(eta - y), zstar = s->tau * sinh(eta - y);
              const double o = so - beta * tstar, l = zstar;
              sa += wa;
              for (int d = 0; d < n_dir; d++)
                for (int k = 0; k < n_q; k++) {
                  const double qo = k * dq * dir[3 * d], qs = k * dq * dir[3 * d + 1], ql = k * dq * dir[3 * d + 2];
                  const double theta = (qo * o + qs * ss + ql * l) / hbarC;
                  fre[d * n_q + k] += w * cos(theta);
                  fim[d * n_q + k] += w * sin(theta);
                }
            }
            int64_t iS3D = (int64_t)ipart + (int64_t)npart * ((int64_t)ipT + (int64_t)npT * ((int64_t)iphip + (int64_t)nphi * (int64_t)iy));
            for (int j = 0; j < nq; j++) {
              Re[j * n_bins + iS3D] += prefactor * degeneracy * fre[j];
              Im[j * n_bins + iS3D] += prefactor * degeneracy * fim[j];
            }
            if (W_abs) W_abs[iS3D] += prefactor * degeneracy * sa;
          }
        }
      }
      free(fre); free(fim);
    }
  }
  free(cs); free(cosphi); free(sinphi);
  return skipped;
}
