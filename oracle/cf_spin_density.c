/* oracle/cf_spin_density.c -- CPU restatement of the spin density matrix from thermal vorticity (mode 5 surfaces).  TEST
 * INFRASTRUCTURE ONLY.
 *
 * Only tests/ and tools may load this library (oracle/cf_spin_density.py compiles it on first use); the product never links or calls it.
 * It is one translation unit with cf_polzn.c (included below), so cfo_spin_polarization is in the same library.  Over the cells, slots,
 * weights, skip and outflow rules of cfo_spin_polarization it sums, as a plain loop nest, the local-equilibrium distribution with the
 * spin term exponentiated (Becattini, Chandra, Del Zanna, Grossi 2013):
 *   theta^mu = -(1/(2m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau     (the eps contraction of cf_polzn.c, eps^{txyz} = +1)
 *   theta*_i = theta^i - theta^t p^i / (E + m),  theta = |theta*|,  that = theta* / theta (0 at theta = 0)
 *   f_m      = 1 / (exp(u.p/T - m theta) + sign),  an explicit sum over the levels m = -J .. J, J = (g - 1)/2, in long double
 *   Snorm = K sum W sum_m f_m,  P_i = K sum W sum_m m f_m that_i,  Q_ij = K sum W sum_m f_m (3m^2 - J(J+1))/2 (that_i that_j - delta_ij/3)
 * with K = 1/(2 pi hbar c)^3 and W = eta weight x p.dsigma.  Each level enters as its deviation d_m = f_m - f_ref from f_ref = f_0 (m = 0
 * formally), formed with expm1l: sum_m m = sum_m (3m^2 - J(J+1)) = 0, so P and Q are sums of d_m alone and the O(theta^2) tensor keeps
 * its relative accuracy down to theta ~ 1e-6.  An evaluation whose exp(u.p/T) overflows in double contributes 0, as in cf_polzn.c.
 * out is [9][n_bins] (Snorm, Px, Py, Pz, Qxx, Qxy, Qxz, Qyy, Qyz), ADDED into; cond (optional) [9][n_bins] receives per-bin sums of
 * |terms|: for Snorm sum |W| sum_m f_m; for P and Q the same sums with every level term and every component of theta* taken in absolute
 * value, the components as the sums of |products| of the eps contraction and of the rest-frame projection (the rounding floor of a
 * cancelling component).
 * Returns #cells skipped (u.dsigma <= 0), or a negative error code: -2 include_baryon, -4 m <= 0, -6 a degeneracy that is not an
 * integer in [1, 16], -5 a boson evaluation with u.p/T - J theta <= 0 (no valid occupation of the top level). */
#include "cf_polzn.c"

int64_t cfo_spin_density(const cfo_flags *fl, const cfo_cells *c, const cfo_vorticity *w, const cfo_species *sp, const cfo_grid *g,
                         double *out, double *cond)
{
  if (fl->include_baryon) return -2;
  const double prefactor = pow(2.0 * M_PI * hbarC, -3);
  const int npart = sp->n, npT = g->n_pT, nphi = g->n_phi;
  const int y_pts = (fl->dimension == 2) ? 1 : g->n_y, eta_pts = (fl->dimension == 2) ? g->n_eta : 1;
  const int64_t n = c->n_cells, n_bins = (int64_t)npart * npT * nphi * g->n_y;
  for (int s = 0; s < npart; s++) if (!(sp->mass[s] > 0.0)) return -4;
  for (int s = 0; s < npart; s++) {
    const double d = sp->degeneracy[s];
    if (!(d >= 1.0 && d <= 16.0 && d == floor(d))) return -6;
  }
  int perm[24][4], psgn[24], np = 0;
  for (int a = 0; a < 4; a++) for (int b = 0; b < 4; b++) for (int d = 0; d < 4; d++) for (int e = 0; e < 4; e++) {
    if (a == b || a == d || a == e || b == d || b == e || d == e) continue;
    int q[4] = {a, b, d, e}, inv = 0;
    for (int i = 0; i < 4; i++) for (int j = i + 1; j < 4; j++) inv += q[i] > q[j];
    perm[np][0] = a; perm[np][1] = b; perm[np][2] = d; perm[np][3] = e; psgn[np] = (inv & 1) ? -1 : 1; np++;
  }
  const int qi[5] = {0, 0, 0, 1, 1}, qj[5] = {0, 1, 2, 1, 2};     /* xx xy xz yy yz */
  int64_t skipped = 0;
  for (int64_t i = 0; i < n; i++) {
    const double tau = c->tau[i], ux = c->ux[i], uy = c->uy[i], un = c->un[i];
    const double ut = sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un);
    if (ut * c->dat[i] + ux * c->dax[i] + uy * c->day[i] + un * c->dan[i] <= 0.0) skipped++;
  }
  int bad = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(| : bad)
  for (int ipart = 0; ipart < npart; ipart++) {
    const double mass = sp->mass[ipart], sign = sp->sign[ipart];
    const int two_j = (int)sp->degeneracy[ipart] - 1;
    const long double J = 0.5L * two_j, JJ1 = J * (J + 1.0L);
    for (int64_t icell = 0; icell < n; icell++) {
      const double tau = c->tau[icell], tau2 = tau * tau, ux = c->ux[icell], uy = c->uy[icell], un = c->un[icell], T = c->T[icell];
      const double ut = sqrt(1.0 + ux * ux + uy * uy + tau2 * un * un);
      const double dat = c->dat[icell], dax = c->dax[icell], day = c->day[icell], dan = c->dan[icell];
      if (ut * dat + ux * dax + uy * day + un * dan <= 0.0) continue;
      const double wtx = w->wtx[icell], wty = w->wty[icell], wtn = w->wtn[icell], wxy = w->wxy[icell], wxn = w->wxn[icell], wyn = w->wyn[icell];
      for (int ipT = 0; ipT < npT; ipT++) {
        const double pT = g->pT[ipT], mT = sqrt(mass * mass + pT * pT);
        for (int iphip = 0; iphip < nphi; iphip++) {
          const double px = pT * cos(g->phi[iphip]), py = pT * sin(g->phi[iphip]);
          for (int iy = 0; iy < y_pts; iy++) {
            const double y = (fl->dimension == 2) ? 0.0 : g->y[iy];
            const double E = mT * cosh(y), pup[3] = {px, py, mT * sinh(y)};
            long double s[9] = {0}, sa[9] = {0};
            for (int ieta = 0; ieta < eta_pts; ieta++) {
              const double eta = (fl->dimension == 2) ? g->eta[ieta] : c->eta[icell];
              const double eta_weight = (fl->dimension == 2) ? g->eta_weight[ieta] : 1.0;
              const double pt = mT * cosh(y - eta), pn = mT / tau * sinh(y - eta);
              const double pdotdsigma = eta_weight * (pt * dat + px * dax + py * day + pn * dan);
              if (fl->outflow && pdotdsigma <= 0.0) continue;
              const double pdotu = pt * ut - px * ux - py * uy - tau2 * pn * un;
              const double x = pdotu / T;
              if (!(x <= 709.782712893384)) continue;            /* exp(u.p/T) overflows: f = 0 exactly, nothing to add */
              const double ch = cosh(eta), sh = sinh(eta);
              double Wv[4][4] = {{0}};
              Wv[0][1] = ch * wtx + sh / tau * wxn;  Wv[0][2] = ch * wty + sh / tau * wyn;  Wv[0][3] = wtn / tau;
              Wv[1][3] = sh * wtx + ch / tau * wxn;  Wv[2][3] = sh * wty + ch / tau * wyn;  Wv[1][2] = wxy;
              for (int a = 0; a < 4; a++) for (int b = a + 1; b < 4; b++) Wv[b][a] = -Wv[a][b];
              const double plow[4] = {E, -px, -py, -mT * sinh(y)};
              long double A[4] = {0, 0, 0, 0}, mag[4] = {0, 0, 0, 0};
              for (int k = 0; k < 24; k++) {
                const long double v = (long double)psgn[k] * Wv[perm[k][1]][perm[k][2]] * plow[perm[k][3]];
                A[perm[k][0]] += v; mag[perm[k][0]] += fabsl(v);
              }
              /* theta^mu = -A^mu / (2m); rest-frame part and its |terms| */
              long double th[3], tha[3], t2 = 0.0L, ta2 = 0.0L;
              for (int k = 0; k < 3; k++) {
                th[k] = (-A[k + 1] + A[0] * pup[k] / (E + mass)) / (2.0L * mass);
                tha[k] = (mag[k + 1] + mag[0] * fabs(pup[k]) / (E + mass)) / (2.0L * mass);
                t2 += th[k] * th[k]; ta2 += tha[k] * tha[k];
              }
              const long double theta = sqrtl(t2);
              if (sign < 0.0 && (long double)x - J * theta <= 0.0L) { bad = 1; continue; }
              const long double that[3] = {theta > 0 ? th[0] / theta : 0, theta > 0 ? th[1] / theta : 0, theta > 0 ? th[2] / theta : 0};
              const long double ex = expl((long double)x), fref = 1.0L / (ex + sign);
              long double sn = 0.0L, sP = 0.0L, sQ = 0.0L, aP = 0.0L, aQ = 0.0L;
              for (int k2 = -two_j; k2 <= two_j; k2 += 2) {             /* m = k2 / 2 */
                const long double m = 0.5L * k2, cq = 0.5L * (3.0L * m * m - JJ1);
                /* f_m - f_ref = ex (1 - e^{-m theta}) / ((ex e^{-m theta} + sign)(ex + sign)) */
                const long double em = expl(-m * theta), d = -ex * expm1l(-m * theta) / ((ex * em + sign) * (ex + sign));
                const long double fm = fref + d;
                sn += fm; sP += m * d; sQ += cq * d;
                aP += fabsl(m) * fm; aQ += fabsl(cq) * fm;
              }
              const long double W = pdotdsigma, aW = fabsl(W);
              s[0] += W * sn; sa[0] += aW * sn;
              for (int k = 0; k < 3; k++) {
                s[1 + k] += W * sP * that[k];
                if (theta > 0) sa[1 + k] += aW * aP * tha[k] / theta;
              }
              for (int q = 0; q < 5; q++) {
                const int a = qi[q], b = qj[q];
                s[4 + q] += W * sQ * (that[a] * that[b] - (a == b ? 1.0L / 3.0L : 0.0L));
                if (theta > 0) sa[4 + q] += aW * aQ * (tha[a] * tha[b] + (a == b ? ta2 / 3.0L : 0.0L)) / t2;
              }
            }
            const int64_t iS3D = (int64_t)ipart + (int64_t)npart * ((int64_t)ipT + (int64_t)npT * ((int64_t)iphip + (int64_t)nphi * (int64_t)iy));
            for (int q = 0; q < 9; q++) {
              out[q * n_bins + iS3D] += (double)(prefactor * s[q]);
              if (cond) cond[q * n_bins + iS3D] += (double)(prefactor * sa[q]);
            }
          }
        }
      }
    }
  }
  return bad ? -5 : skipped;
}
