/* oracle/cf_polzn.c -- CPU restatement of the spin polarization from thermal vorticity (mode 5 surfaces).  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/ and tools may load this library (oracle/cf_polzn.py compiles it on first use); the product never links or calls it.
 * It restates the published formula (Becattini et al. 2013; Karpenko & Becattini 2017) as a plain loop nest over
 * cells x species x bins x slots, over the cells and slots of the ideal-f spectra (df off, cfo_smooth_vh of cf_oracle.c):
 *   Snorm = g/(2 pi hbar c)^3 sum w p.dsigma f,
 *   N^mu  = g/(2 pi hbar c)^3 sum w p.dsigma f (1 - sign f) (-1/(8m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau
 * in Cartesian lab components (eps^{txyz} = +1), varpi converted from the covariant Milne columns (tau x, tau y, tau eta, xy, x eta,
 * y eta) at the cell's (2+1D: the slot's) eta.  The reference's own calculate_spin_polzn has not been read; its conventions are not
 * pinned here.
 * N is [4][n_bins] (t, x, y, z), Snorm [n_bins], both ADDED into; N_abs (optional) [4][n_bins] receives the sums of |terms| of each
 * N^mu, every product of the eps contraction taken in absolute value (the floor of the rounding noise of a cancelling N^mu).
 * Returns #cells skipped (u.dsigma <= 0) or a negative error code. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include "cf_oracle.h"

static const double hbarC = 0.197327053; /* iS3D.h:9 */

typedef struct { const double *wtx, *wty, *wtn, *wxy, *wxn, *wyn; } cfo_vorticity;

int64_t cfo_spin_polarization(const cfo_flags *fl, const cfo_cells *c, const cfo_vorticity *w, const cfo_species *sp, const cfo_grid *g,
                              double *N, double *Snorm, double *N_abs)
{
  if (fl->include_baryon) return -2;
  const double prefactor = pow(2.0 * M_PI * hbarC, -3);
  const int npart = sp->n, npT = g->n_pT, nphi = g->n_phi;
  const int y_pts = (fl->dimension == 2) ? 1 : g->n_y, eta_pts = (fl->dimension == 2) ? g->n_eta : 1;
  const int64_t n = c->n_cells, n_bins = (int64_t)npart * npT * nphi * g->n_y;
  for (int s = 0; s < npart; s++) if (!(sp->mass[s] > 0.0)) return -4;
  /* the 24 non-zero entries of eps^{mu rho sigma tau}, eps^{0123} = +1 */
  int perm[24][4], psgn[24], np = 0;
  for (int a = 0; a < 4; a++) for (int b = 0; b < 4; b++) for (int d = 0; d < 4; d++) for (int e = 0; e < 4; e++) {
    if (a == b || a == d || a == e || b == d || b == e || d == e) continue;
    int q[4] = {a, b, d, e}, inv = 0;
    for (int i = 0; i < 4; i++) for (int j = i + 1; j < 4; j++) inv += q[i] > q[j];
    perm[np][0] = a; perm[np][1] = b; perm[np][2] = d; perm[np][3] = e; psgn[np] = (inv & 1) ? -1 : 1; np++;
  }
  int64_t skipped = 0;
  for (int64_t i = 0; i < n; i++) {
    const double tau = c->tau[i], ux = c->ux[i], uy = c->uy[i], un = c->un[i];
    const double ut = sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un);
    if (ut * c->dat[i] + ux * c->dax[i] + uy * c->day[i] + un * c->dan[i] <= 0.0) skipped++;
  }
#pragma omp parallel for schedule(dynamic, 1)
  for (int ipart = 0; ipart < npart; ipart++) {
    const double mass = sp->mass[ipart], sign = sp->sign[ipart], degeneracy = sp->degeneracy[ipart];
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
            double sn = 0.0, sN[4] = {0, 0, 0, 0}, sA[4] = {0, 0, 0, 0};
            for (int ieta = 0; ieta < eta_pts; ieta++) {
              const double eta = (fl->dimension == 2) ? g->eta[ieta] : c->eta[icell];
              const double eta_weight = (fl->dimension == 2) ? g->eta_weight[ieta] : 1.0;
              const double pt = mT * cosh(y - eta), pn = mT / tau * sinh(y - eta);
              const double pdotdsigma = eta_weight * (pt * dat + px * dax + py * day + pn * dan);
              if (fl->outflow && pdotdsigma <= 0.0) continue;
              const double pdotu = pt * ut - px * ux - py * uy - tau2 * pn * un;
              const double feq = 1.0 / (exp(pdotu / T) + sign);
              /* covariant Cartesian varpi_{mu nu} at eta from the Milne columns (tau x, tau y, tau eta, xy, x eta, y eta) */
              const double ch = cosh(eta), sh = sinh(eta);
              double W[4][4] = {{0}};
              W[0][1] = ch * wtx + sh / tau * wxn;  W[0][2] = ch * wty + sh / tau * wyn;  W[0][3] = wtn / tau;
              W[1][3] = sh * wtx + ch / tau * wxn;  W[2][3] = sh * wty + ch / tau * wyn;  W[1][2] = wxy;    /* varpi_xz = -varpi_zx */
              for (int a = 0; a < 4; a++) for (int b = a + 1; b < 4; b++) W[b][a] = -W[a][b];
              /* lower-index Cartesian momentum */
              const double plow[4] = {mT * cosh(y), -px, -py, -mT * sinh(y)};
              double A[4] = {0, 0, 0, 0}, mag[4] = {0, 0, 0, 0};
              for (int k = 0; k < 24; k++) {
                const double v = psgn[k] * W[perm[k][1]][perm[k][2]] * plow[perm[k][3]];
                A[perm[k][0]] += v; mag[perm[k][0]] += fabs(v);
              }
              const double t = pdotdsigma * feq, wf = t * (1.0 - sign * feq);
              sn += t;
              /* |terms| before the contraction's own cancellation (E omega against e x p at large rapidities) */
              for (int mu = 0; mu < 4; mu++) { sN[mu] += wf * (-A[mu] / (8.0 * mass)); sA[mu] += fabs(wf) * mag[mu] / (8.0 * mass); }
            }
            const int64_t iS3D = (int64_t)ipart + (int64_t)npart * ((int64_t)ipT + (int64_t)npT * ((int64_t)iphip + (int64_t)nphi * (int64_t)iy));
            Snorm[iS3D] += prefactor * degeneracy * sn;
            for (int mu = 0; mu < 4; mu++) {
              N[mu * n_bins + iS3D] += prefactor * degeneracy * sN[mu];
              if (N_abs) N_abs[mu * n_bins + iS3D] += prefactor * degeneracy * sA[mu];
            }
          }
        }
      }
    }
  }
  return skipped;
}
