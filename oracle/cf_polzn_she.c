/* oracle/cf_polzn_she.c -- CPU restatement of the spin Hall (SHE) spin polarization of baryons.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/ and tools may load this library (oracle/cf_polzn_she.py compiles it on first use); the product never links or calls it.
 * It is one translation unit with cf_polzn.c (included below), so cfo_spin_polarization is in the same library and the Snorm of
 * cfo_spin_polarization_spin_hall, formed statement for statement like cfo_spin_polarization's, is bit-identical to it.
 * It restates the formula as a plain loop nest over cells x species x bins x slots: the vorticity formula with the replacement
 *   varpi_{rho sigma} -> -2 q_B that_rho zeta_sigma / E,   zeta_sigma = hbar c d_sigma alpha_B (GeV), alpha_B = muB/T,
 *   N_she^mu = g/(2 pi hbar c)^3 sum w p.dsigma f (1 - sign f) (-1/(8m)) eps^{mu rho sigma tau} p_tau (-2 q_B that_rho zeta_sigma / E)
 * in Cartesian lab components (eps^{txyz} = +1, that = (1, 0, 0, 0), E = p^t, q_B = species baryon), d alpha_B converted from the four
 * covariant Milne columns (tau, x, y, eta) at the cell's (2+1D: the slot's) eta by cfo_cart_gradient.
 * N is [4][n_bins] (t, x, y, z), Snorm [n_bins], both ADDED into; N_abs (optional) [4][n_bins] receives the sums of |terms| of each
 * N^mu, every product of the eps contraction taken in absolute value.
 * Returns #cells skipped (u.dsigma <= 0) or a negative error code. */
#include "cf_polzn.c"

typedef struct { const double *d[4]; } cfo_baryon_gradient;

/* the oracle's copy of cart_gradient() (is3d_b200/csrc/cf_polzn.cuh), with the time component it leaves out: covariant Milne
 * (d_tau, d_x, d_y, d_eta) at eta -> covariant Cartesian (d_t, d_x, d_y, d_z), by the Jacobian dtau/dt = ch, dtau/dz = -sh,
 * deta/dt = -sh/tau, deta/dz = ch/tau */
void cfo_cart_gradient(const double d[4], double tau, double eta, double c[4])
{
  const double ch = cosh(eta), sh = sinh(eta);
  c[0] = ch * d[0] - sh / tau * d[3];
  c[1] = d[1];
  c[2] = d[2];
  c[3] = -sh * d[0] + ch / tau * d[3];
}

int64_t cfo_spin_polarization_spin_hall(const cfo_flags *fl, const cfo_cells *c, const cfo_baryon_gradient *gb, const cfo_species *sp,
                                        const cfo_grid *g, double *N, double *Snorm, double *N_abs)
{
  if (fl->include_baryon) return -2;
  if (!sp->baryon) return -5;
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
  const double that[4] = {1.0, 0.0, 0.0, 0.0};   /* lab time direction, lower index */
  int64_t skipped = 0;
  for (int64_t i = 0; i < n; i++) {
    const double tau = c->tau[i], ux = c->ux[i], uy = c->uy[i], un = c->un[i];
    const double ut = sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un);
    if (ut * c->dat[i] + ux * c->dax[i] + uy * c->day[i] + un * c->dan[i] <= 0.0) skipped++;
  }
#pragma omp parallel for schedule(dynamic, 1)
  for (int ipart = 0; ipart < npart; ipart++) {
    const double mass = sp->mass[ipart], sign = sp->sign[ipart], degeneracy = sp->degeneracy[ipart], qB = sp->baryon[ipart];
    for (int64_t icell = 0; icell < n; icell++) {
      const double tau = c->tau[icell], tau2 = tau * tau, ux = c->ux[icell], uy = c->uy[icell], un = c->un[icell], T = c->T[icell];
      const double ut = sqrt(1.0 + ux * ux + uy * uy + tau2 * un * un);
      const double dat = c->dat[icell], dax = c->dax[icell], day = c->day[icell], dan = c->dan[icell];
      if (ut * dat + ux * dax + uy * day + un * dan <= 0.0) continue;
      double dm[4];
      for (int k = 0; k < 4; k++) dm[k] = gb->d[k][icell];
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
              double zc[4];
              cfo_cart_gradient(dm, tau, eta, zc);
              for (int k = 0; k < 4; k++) zc[k] *= hbarC;
              /* lower-index Cartesian momentum, E = p^t */
              const double E = mT * cosh(y);
              const double plow[4] = {E, -px, -py, -mT * sinh(y)};
              double A[4] = {0, 0, 0, 0}, mag[4] = {0, 0, 0, 0};
              for (int k = 0; k < 24; k++) {
                const int mu = perm[k][0], rho = perm[k][1], sg = perm[k][2], ta = perm[k][3];
                const double w = -2.0 * qB * that[rho] * zc[sg] / E;          /* the replacement of varpi_{rho sigma} */
                const double v = psgn[k] * w * plow[ta];
                A[mu] += v; mag[mu] += fabs(v);
              }
              const double t = pdotdsigma * feq, wf = t * (1.0 - sign * feq);
              sn += t;
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
