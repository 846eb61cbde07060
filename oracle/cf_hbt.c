/* oracle/cf_hbt.c -- CPU restatement of the HBT moments of the linear-delta-f emission function.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/ and tools may load this library (oracle/cf_hbt.py compiles it on first use); the product never links or calls it.
 * It is one translation unit with cf_oracle.c (included below), so that the per-cell set-up, the coefficient lookup and the
 * per-evaluation weight are those of cfo_smooth_vh, statement for statement: S0 equals cfo_smooth_vh bin for bin, bit for bit.
 * Per evaluation (cell, slot) of the spectra, with the weight w = pdotdsigma * f of cfo_smooth_vh and the LCMS coordinates of the bin
 *   t* = tau cosh(eta - y),  z* = tau sinh(eta - y),  o = x cos phi + y sin phi - (pT / mT) t*,  s = -x sin phi + y cos phi,  l = z*
 * the ten raw sums S0 = sum w, S_i = sum w x_i, S_ij = sum w x_i x_j (x = (o, s, l)) are formed per (cell, bin) over the slots and
 * then added into S[10][n_bins] (order S0 So Ss Sl Soo Sss Sll Sos Sol Ssl) as prefactor * degeneracy * sum, like dN.
 * S_abs (optional) [10][n_bins] receives the same sums with the weight replaced by cfo_smooth_vh's |terms| magnitude and every
 * coordinate by the sum of the absolute values of its terms: the floor of the rounding noise of a cancelling sum.
 * x, y: transverse cell positions [n_cells].  Returns #cells skipped (u.dsigma <= 0) or a negative error code. */
#include "cf_oracle.c"

int64_t cfo_hbt_moments(const cfo_flags *fl, const cfo_cells *c, const double *xpos, const double *ypos, const cfo_species *sp,
                        const cfo_grid *g, const cfo_df_tables *tab, double *S, double *S_abs)
{
  if (fl->df_mode != 1 && fl->df_mode != 2) return -1;
  if (fl->include_baryon) return -2;
  const double prefactor = pow(2.0 * M_PI * hbarC, -3);
  const int npart = sp->n, npT = g->n_pT, nphi = g->n_phi;
  int y_pts, eta_pts; grid_dims(fl, g, &y_pts, &eta_pts);
  const int64_t n = c->n_cells, n_bins = (int64_t)npart * npT * nphi * g->n_y;
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

#pragma omp parallel for schedule(dynamic, 1)
  for (int ipart = 0; ipart < npart; ipart++) {
    double mass = sp->mass[ipart], mass2 = mass * mass, sign = sp->sign[ipart];
    double degeneracy = sp->degeneracy[ipart], baryon = sp->baryon[ipart];
    for (int64_t icell = 0; icell < n; icell++) {
      const cell_setup *s = &cs[icell];
      if (s->skip) continue;
      double chem = baryon * s->alphaB;
      const double xc = xpos[icell], yc = ypos[icell];
      for (int ipT = 0; ipT < npT; ipT++) {
        double pT = g->pT[ipT];
        double mT = sqrt(mass2 + pT * pT);
        double mT_over_tau = mT / s->tau;
        const double beta = pT / mT;
        for (int iphip = 0; iphip < nphi; iphip++) {
          double px = pT * cosphi[iphip], py = pT * sinphi[iphip];
          const double so = xc * cosphi[iphip] + yc * sinphi[iphip], ss = -xc * sinphi[iphip] + yc * cosphi[iphip];
          const double ao = fabs(xc * cosphi[iphip]) + fabs(yc * sinphi[iphip]), as = fabs(xc * sinphi[iphip]) + fabs(yc * cosphi[iphip]);
          for (int iy = 0; iy < y_pts; iy++) {
            double y = (fl->dimension == 2) ? 0.0 : g->y[iy];
            double sum = 0.0, sq[10] = {0}, sa[10] = {0};
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
              sum += (pdotdsigma * f);
              /* the weight and its |terms| magnitude, then the LCMS coordinates of this evaluation */
              const double w = pdotdsigma * f;
              const double wa = fabs(pdotdsigma) * feq * (1.0 + (clamped ? 1.0 : fabs(feqbar) * mag));
              const double tstar = s->tau * cosh(eta - y), zstar = s->tau * sinh(eta - y);
              const double o = so - beta * tstar, l = zstar;
              const double oa = ao + beta * tstar, la = fabs(zstar);
              const double v[3] = {o, ss, l}, va[3] = {oa, as, la};
              sq[0] += w; sa[0] += wa;
              for (int i = 0; i < 3; i++) { sq[1 + i] += w * v[i]; sa[1 + i] += wa * va[i]; }
              for (int i = 0; i < 3; i++) { sq[4 + i] += w * v[i] * v[i]; sa[4 + i] += wa * va[i] * va[i]; }
              const int pi_[3][2] = {{0, 1}, {0, 2}, {1, 2}};
              for (int k = 0; k < 3; k++) {
                sq[7 + k] += w * v[pi_[k][0]] * v[pi_[k][1]];
                sa[7 + k] += wa * va[pi_[k][0]] * va[pi_[k][1]];
              }
            }
            int64_t iS3D = (int64_t)ipart + (int64_t)npart * ((int64_t)ipT + (int64_t)npT * ((int64_t)iphip + (int64_t)nphi * (int64_t)iy));
            S[iS3D] += (prefactor * degeneracy * sum);           /* S0: the statement of cfo_smooth_vh */
            for (int q = 1; q < 10; q++) S[q * n_bins + iS3D] += prefactor * degeneracy * sq[q];
            if (S_abs)
              for (int q = 0; q < 10; q++) S_abs[q * n_bins + iS3D] += prefactor * degeneracy * sa[q];
          }
        }
      }
    }
  }
  free(cs); free(cosphi); free(sinphi);
  return skipped;
}
