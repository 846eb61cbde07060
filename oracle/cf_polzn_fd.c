/* oracle/cf_polzn_fd.c -- CPU restatement of the feed-down of the spin-polarization sums through 2-body resonance decays
 * (is3d_b200_polarization_decays).  TEST INFRASTRUCTURE ONLY.
 *
 * One translation unit with oracle/cf_decays.c: Snorm runs through that file's own two_body_decay / three_body_decay in the order of
 * cfo_resonance_decays, so it is the decay oracle bit for bit.  The spin term is a separate loop over the same (v, zeta, azimuth) points
 * with explicit 4x4 Lorentz matrices: L(P) maps the parent's rest frame to the lab, L(p*) the daughter's rest frame to the parent's.
 * Every point's |contribution| x (1 + |log dN|) is summed per bin and component as conditioning.
 */
#include "cf_decays.c"

typedef double mat4[4][4];

/* pure boost taking the rest frame of a particle of mass m to the frame where its four-momentum is k (k[0] = energy) */
static void boost_matrix(const double k[4], double m, mat4 L)
{
  L[0][0] = k[0] / m;
  for (int i = 1; i < 4; i++) { L[0][i] = k[i] / m; L[i][0] = k[i] / m; }
  for (int i = 1; i < 4; i++)
    for (int j = 1; j < 4; j++) L[i][j] = (i == j ? 1.0 : 0.0) + k[i] * k[j] / (m * (k[0] + m));
}
static void inverse_boost_matrix(const double k[4], double m, mat4 L)
{
  const double kk[4] = {k[0], -k[1], -k[2], -k[3]};
  boost_matrix(kk, m, L);
}
static void mat_vec(const mat4 L, const double v[4], double out[4])
{
  for (int i = 0; i < 4; i++) { double s = 0.0; for (int j = 0; j < 4; j++) s += L[i][j] * v[j]; out[i] = s; }
}

/* the Lorentz chain of one integrand point (exported for the numpy restatement test): parent P (mass M), rest-frame spin Sp (2+1D:
 * the y = 0 value at (MT, Phi), boosted longitudinally by Y), daughter p (mass mD), law (a, b) -> S_D [4] */
void cfo_fd_chain(const double P[4], double M, const double Sp_in[3], int dim2, const double p[4], double mD, double a, double b, double out[4])
{
  double Sp[3] = {Sp_in[0], Sp_in[1], Sp_in[2]};
  mat4 L, Li;
  inverse_boost_matrix(P, M, Li);
  if (dim2) {
    const double MT = sqrt(P[0] * P[0] - P[3] * P[3]), Y = atanh(P[3] / P[0]);
    const double P0[4] = {MT, P[1], P[2], 0.0};
    mat4 L0, Bz; double S0[4], S[4], r[4];
    boost_matrix(P0, M, L0);
    const double s4[4] = {0.0, Sp[0], Sp[1], Sp[2]};
    mat_vec(L0, s4, S0);
    memset(Bz, 0, sizeof(Bz));
    Bz[0][0] = cosh(Y); Bz[0][3] = sinh(Y); Bz[3][0] = sinh(Y); Bz[3][3] = cosh(Y); Bz[1][1] = 1.0; Bz[2][2] = 1.0;
    mat_vec(Bz, S0, S);
    mat_vec(Li, S, r);
    Sp[0] = r[1]; Sp[1] = r[2]; Sp[2] = r[3];
  }
  double ps[4];
  mat_vec(Li, p, ps);
  const double norm = sqrt(ps[1] * ps[1] + ps[2] * ps[2] + ps[3] * ps[3]);
  const double n[3] = {ps[1] / norm, ps[2] / norm, ps[3] / norm};
  const double Sn = Sp[0] * n[0] + Sp[1] * n[1] + Sp[2] * n[2];
  const double s4[4] = {0.0, a * Sp[0] + b * Sn * n[0], a * Sp[1] + b * Sn * n[1], a * Sp[2] + b * Sn * n[2]};
  mat4 Ld; double q[4];
  boost_matrix(ps, mD, Ld);
  mat_vec(Ld, s4, q);
  boost_matrix(P, M, L);
  mat_vec(L, q, out);
}

/* the transfer law of include/is3d_b200.h; returns 0 when the channel has none */
static int fd_law(const cfo_particles *pdg, const int32_t *spin2, const int32_t *parity, int parent, int daughter, int partner, double *a, double *b)
{
  if (spin2[daughter] != 1) return 0;
  const int jp2 = spin2[parent];
  if (abs(pdg->mcid[partner]) == 22) { if (jp2 != 1) return 0; *a = 0.0; *b = -1.0; return 1; }
  if (spin2[partner] != 0 || jp2 % 2 != 1) return 0;
  if (!parity[parent] || !parity[daughter] || !parity[partner]) return 0;
  const double eta = -((((jp2 - 1) / 2) % 2 == 0) ? 1.0 : -1.0) * parity[parent] * parity[daughter] * parity[partner];
  *a = -eta * (jp2 + 1) / 2.0; *b = 1.0 - *a;
  return 1;
}

/* linear interpolation cell of the log spectrum: log dN and S*_P at (MT, Phi[, Y]) with the weights of parent_2d / parent_3d */
static void fd_interp(const ctx_t *c, const double *Sstar, double MT, double Phip, int iYL, int iYR, double YL, double YR, double Y, double MTmax,
                      double *logdN, double S[3])
{
  int iL, iR; double PL, PR;
  const long npT = c->n_pT, nphi = c->n_phi;
  phi_points(c, &Phip, &iL, &iR, &PL, &PR);
  const double dPhi = PR - PL, wL = PR - Phip, wR = Phip - PL;
  if (c->dim == 2) { iYL = iYR = 0; }
  const double dY = (c->dim == 2) ? 1.0 : YR - YL, yL = (c->dim == 2) ? 1.0 : YR - Y, yR = (c->dim == 2) ? 0.0 : Y - YL;
#define IX(im, ip, iy) ((im) + npT * ((ip) + nphi * (iy)))
  if (MT <= MTmax) {
    int iMTR = 1;
    while (MT > c->MTValues[iMTR]) iMTR++;
    const int iMTL = iMTR - 1;
    const double MTL = c->MTValues[iMTL], MTR = c->MTValues[iMTR], dMT = MTR - MTL;
    const long ix[8] = {IX(iMTL, iL, iYL), IX(iMTL, iL, iYR), IX(iMTL, iR, iYL), IX(iMTL, iR, iYR),
                        IX(iMTR, iL, iYL), IX(iMTR, iL, iYR), IX(iMTR, iR, iYL), IX(iMTR, iR, iYR)};
    const double w[8] = {(MTR - MT) * wL * yL, (MTR - MT) * wL * yR, (MTR - MT) * wR * yL, (MTR - MT) * wR * yR,
                         (MT - MTL) * wL * yL, (MT - MTL) * wL * yR, (MT - MTL) * wR * yL, (MT - MTL) * wR * yR};
    const double den = dY * dPhi * dMT;
    double l = 0.0, s[3] = {0.0, 0.0, 0.0};
    for (int k = 0; k < 8; k++) { l += w[k] * c->logdN[ix[k]]; for (int j = 0; j < 3; j++) s[j] += w[k] * Sstar[3 * ix[k] + j]; }
    *logdN = l / den;
    for (int j = 0; j < 3; j++) S[j] = s[j] / den;
  } else {
    const int im = c->n_pT - 1;
    const int fx[4] = {iYL * c->n_phi + iL, iYR * c->n_phi + iL, iYL * c->n_phi + iR, iYR * c->n_phi + iR};
    const long ix[4] = {IX(im, iL, iYL), IX(im, iL, iYR), IX(im, iR, iYL), IX(im, iR, iYR)};
    const double w[4] = {wL * yL, wL * yR, wR * yL, wR * yR};
    const double den = dY * dPhi;
    double l = 0.0, s[3] = {0.0, 0.0, 0.0};
    for (int k = 0; k < 4; k++) {
      l += w[k] * (c->fit[fx[k]].constant + c->fit[fx[k]].slope * MT);
      for (int j = 0; j < 3; j++) s[j] += w[k] * Sstar[3 * ix[k] + j];
    }
    *logdN = l / den;
    for (int j = 0; j < 3; j++) S[j] = s[j] / den;
  }
#undef IX
}

/* spin part of one 2-body channel; c->MTValues / c->fit hold the tables two_body_decay set up for this channel's mass_parent */
static void two_body_spin(ctx_t *c, double *S4, long n_total, double *A4, const double *Sstar, const int32_t *spin2, const int32_t *parity,
                          double branch_ratio, int ipart, int particle_1, int particle_2, double mass_parent)
{
  const cfo_particles *pd = c->pdg;
  const int prod[2] = {particle_1, particle_2};
  int groups[2], members[2];
  const int ng = group_daughters(c, prod, 2, groups, members);
  const double Ymax = fabs(c->dim == 2 ? 0.0 : c->y[c->y_pts - 1]);
  const double MTmax = c->MTValues[c->n_pT - 1];
  const double two_Pi = 2.0 * M_PI, M = mass_parent, M2 = M * M;
  for (int gi = 0; gi < ng; gi++) {
    double a, b;
    if (!fd_law(pd, spin2, parity, ipart, groups[gi], particle_1 == groups[gi] ? particle_2 : particle_1, &a, &b)) continue;
    int err = 0;
    const int dchosen = particle_chosen_index(c, groups[gi], &err);
    const double mD = pd->mass[groups[gi]], mD2 = mD * mD, W = pd->mass[particle_2];
    const double Estar = (M2 + mD2 - W * W) / (2.0 * M), pstar = sqrt(Estar * Estar - mD2);
    const double prefactor = (double)members[gi] * M * branch_ratio / (8.0 * pstar);
    /* the integration points are computed with the statements of two_body_decay, so that a point next to a branch of the
     * interpolation (M_T = MTmax, the azimuthal wrap) falls on the same side as in the spectra feed-down */
    const double Estar2 = Estar * Estar, Estar_M = Estar * M;
    for (int ipT = 0; ipT < c->n_pT; ipT++)
      for (int iphip = 0; iphip < c->n_phi; iphip++)
        for (int iy = 0; iy < c->y_pts; iy++) {
          const double pT = c->pT[ipT], pT2 = pT * pT, mT2 = pT2 + mD2, mT = sqrt(mT2);
          const double M_pT = M * pT, Estar_M_mT = Estar_M * mT, Estar_M_over_pT = Estar_M / pT, Estar2_plus_pT2 = Estar2 + pT2;
          const double phip = c->phi[iphip], y = (c->dim == 2) ? 0.0 : c->y[iy];
          const double p[4] = {mT * cosh(y), pT * cos(phip), pT * sin(phip), mT * sinh(y)};
          const double DeltaY = log((pstar + sqrt(Estar2_plus_pT2)) / mT);
          double acc[4] = {0, 0, 0, 0}, cond[4] = {0, 0, 0, 0};
          for (int iv = 0; iv < GP; iv++) {
            const double v = GL_ROOT[iv], Y = y + v * DeltaY;
            int iYL = 0, iYR = 0; double YL = 0.0, YR = 0.0;
            if (c->dim == 3 && y_points(c, Y, Ymax, &iYL, &iYR, &YL, &YR)) continue;
            const double coshvDeltaY = cosh(v * DeltaY);
            const double mT2_coshvDeltaY2 = mT2 * coshvDeltaY * coshvDeltaY;
            const double den = mT2_coshvDeltaY2 - pT2;
            const double MTbar = Estar_M_mT * coshvDeltaY / den;
            const double DeltaMT = M_pT * sqrt(fabs(Estar2_plus_pT2 - mT2_coshvDeltaY2)) / den;
            const double mTc = mT * coshvDeltaY / pT;
            const double vw = DeltaY * GL_WEIGHT[iv] / sqrt(fabs(den));
            for (int iz = 0; iz < GP; iz++) {
              const double coszeta = cos((M_PI / 2.0) * (1.0 + GL_ROOT[iz]));
              const double MT = MTbar + (DeltaMT * coszeta);
              const double PT = sqrt(MT * MT - M2);
              const double tilde = acos((MT * mTc - Estar_M_over_pT) / PT);
              for (int side = 0; side < 2; side++) {
                double Phi = fmod((side ? -tilde : tilde) + phip, two_Pi);
                if (Phi < 0.0) Phi += two_Pi;
                double logdN, Sp[3], SD[4];
                fd_interp(c, Sstar, MT, Phi, iYL, iYR, YL, YR, Y, MTmax, &logdN, Sp);
                const double P[4] = {MT * cosh(Y), PT * cos(Phi), PT * sin(Phi), MT * sinh(Y)};
                cfo_fd_chain(P, M, Sp, c->dim == 2, p, mD, a, b, SD);
                const double w = prefactor * vw * GL_WEIGHT[iz] * MT * exp(logdN);
                /* conditioning: |term| x (1 + |log dN|): the weight is exp of an interpolated log, and an ulp of log dN (the GPU's and
                 * the C library's log / exp differ by about one) is |log dN| ulps of the weight */
                for (int mu = 0; mu < 4; mu++) { acc[mu] += w * SD[mu]; cond[mu] += fabs(w * SD[mu]) * (1.0 + fabs(logdN)); }
              }
            }
          }
          const long k = dchosen + (long)c->n_chosen * (ipT + (long)c->n_pT * (iphip + (long)c->n_phi * iy));
          for (int mu = 0; mu < 4; mu++) { S4[mu * n_total + k] += acc[mu]; if (A4) A4[mu * n_total + k] += cond[mu]; }
        }
  }
}

/* S: [St | Sx | Sy | Sz | Snorm], n_total = n_chosen * n_pT * n_phi * n_y each, amended in place; A (optional): [4][n_total] conditioning */
int cfo_polarization_decays(const cfo_particles *pdg, const int32_t *spin2, const int32_t *parity, int32_t n_chosen, const int32_t *chosen_pdg_index,
                            const cfo_grid *g, int32_t dimension, double *S, double *A)
{
  if (n_chosen - 1 <= 0) return -10;
  if (g->n_pT > 512) return -15;
  const long n_total = (long)n_chosen * g->n_pT * g->n_phi * g->n_y;
  ctx_t c; memset(&c, 0, sizeof(c));
  c.pdg = pdg; c.n_chosen = n_chosen; c.chosen = chosen_pdg_index;
  c.n_pT = g->n_pT; c.n_phi = g->n_phi; c.n_y_tab = g->n_y; c.dim = dimension; c.y_pts = (dimension == 2) ? 1 : g->n_y;
  c.pT = g->pT; c.phi = g->phi; c.y = g->y; c.dN = S + 4 * n_total;
  const long n_tab = (long)c.n_pT * c.n_phi * c.n_y_tab;
  c.logdN = (double *)calloc((size_t)n_tab, sizeof(double));
  c.fit = (mt_fit *)calloc((size_t)c.y_pts * c.n_phi, sizeof(mt_fit));
  double *Sstar = (double *)calloc((size_t)n_tab * 3, sizeof(double));
  for (int ichosen = n_chosen - 1; ichosen > 0 && !c.err; ichosen--) {
    const int ipart = chosen_pdg_index[ichosen];
    if (pdg->stable[ipart]) continue;
    const double m = pdg->mass[ipart];
    for (int ipT = 0; ipT < c.n_pT; ipT++)
      for (int iphip = 0; iphip < c.n_phi; iphip++)
        for (int iy = 0; iy < c.y_pts; iy++) {
          const long it = ipT + (long)c.n_pT * (iphip + (long)c.n_phi * iy);
          const long iS3D = ichosen + (long)n_chosen * it;
          c.logdN[it] = log(c.dN[iS3D]);
          /* the parent's rest-frame spin on its own bins, physical mass */
          const double sn = c.dN[iS3D];
          double st[3] = {0.0, 0.0, 0.0};
          if (isfinite(log(sn))) {
            const double pT = c.pT[ipT], phi = c.phi[iphip], y = (dimension == 2) ? 0.0 : c.y[iy];
            const double mT = sqrt(pT * pT + m * m), E = mT * cosh(y);
            const double pv[3] = {pT * cos(phi), pT * sin(phi), mT * sinh(y)};
            for (int j = 0; j < 3; j++) st[j] = (S[(j + 1) * n_total + iS3D] - S[iS3D] * pv[j] / (E + m)) / sn;
          }
          for (int j = 0; j < 3; j++) Sstar[3 * it + j] = st[j];
        }
    for (int ich = 0; ich < pdg->decays[ipart] && !c.err; ich++) {
      const int row = pdg->dec_first[ipart] + ich;
      const int decay_products = abs(pdg->dec_npart[row]);
      int idx[5];
      for (int k = 0; k < decay_products && k < 5; k++) idx[k] = particle_index(pdg, pdg->dec_part[row * 5 + k], &c.err);
      if (c.err) break;
      if (decay_products == 1) continue;
      const double branch_ratio = pdg->dec_br[row];
      if (decay_products == 2) {
        double mass_parent = pdg->mass[ipart], mass_1 = pdg->mass[idx[0]], mass_2 = pdg->mass[idx[1]];
        while ((mass_1 + mass_2) > mass_parent) {
          mass_parent += 0.25 * pdg->width[ipart];
          mass_1 -= 0.5 * pdg->width[idx[0]];
          mass_2 -= 0.5 * pdg->width[idx[1]];
          if (mass_1 < 0.0 || mass_2 < 0.0) { c.err = -16; break; }
        }
        if (!c.err) two_body_decay(&c, branch_ratio, ichosen, idx[0], idx[1], mass_parent);
        if (!c.err) two_body_spin(&c, S, n_total, A, Sstar, spin2, parity, branch_ratio, ipart, idx[0], idx[1], mass_parent);
      } else if (decay_products == 3) {
        three_body_decay(&c, branch_ratio, idx[0], idx[1], idx[2], pdg->mass[ipart]);
      } else if (decay_products == 4) {
      } else c.err = -17;
    }
  }
  free(c.logdN); free(c.fit); free(Sstar);
  return c.err;
}
