/* oracle/cf_polzn_fdw.c -- CPU restatement of the feed-down of the spin-polarization sums through weak 2-body decays
 * (is3d_b200_polarization_weak_decays).  TEST INFRASTRUCTURE ONLY.
 *
 * One translation unit with oracle/cf_polzn_fd.c and oracle/cf_decays.c (included below), so cfo_polarization_decays is exported from
 * the same library.  Every row is a plain loop over the integration points of two_body_decay (12 x 12 (v, zeta) nodes, both parent
 * azimuths), with the interpolation of cf_polzn_fd.c.  The Lee-Yang law is written out with an explicit cross product in the parent's
 * rest frame, reached with explicit 4x4 boosts; its numerator is carried to the lab by cfo_fd_chain with the law (a, b) = (1, 0).
 * Every point's |contribution| x (1 + |log dN|) is summed per bin and array as conditioning (for St..Sz the largest |component| of the
 * point's four-vector, since the boosts mix them).
 */
#include "cf_polzn_fd.c"

/* the daughter's lab spin numerator four-vector (out) and yield 1 + 2 alpha S.n at one integrand point: parent P (mass M), rest-frame spin
 * Sp (2+1D: the y = 0 value at (MT, Phi), boosted longitudinally by Y), daughter p (mass mD), decay parameters (alpha, beta, gamma) */
void cfo_fdw_chain(const double P[4], double M, const double Sp_in[3], int dim2, const double p[4], double mD, double alpha, double beta,
                   double gamma, double out[4], double *yield)
{
  double Sp[3] = {Sp_in[0], Sp_in[1], Sp_in[2]};
  mat4 Li;
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
  double cross[3];                                         /* S x n */
  cross[0] = Sp[1] * n[2] - Sp[2] * n[1];
  cross[1] = Sp[2] * n[0] - Sp[0] * n[2];
  cross[2] = Sp[0] * n[1] - Sp[1] * n[0];
  double num[3];
  for (int k = 0; k < 3; k++) num[k] = (0.5 * alpha + Sn) * n[k] + beta * cross[k] + gamma * (Sp[k] - Sn * n[k]);
  *yield = 1.0 + 2.0 * alpha * Sn;
  /* num is a rest-frame vector of the parent frame: the chain of cf_polzn_fd.c with s* = 1 x num (no 2+1D step: num is already there) */
  cfo_fd_chain(P, M, num, 0, p, mD, 1.0, 0.0, out);
}

/* one weak row: the daughter (a chosen species) gains Snorm and, with the law, N; c holds the parent's log spectrum and Sstar its spin */
static void weak_row(ctx_t *c, double *S, long n_total, double *A, const double *Sstar, int has_law, double alpha, double beta, double gamma,
                     double branch_ratio, int daughter, int partner, double M)
{
  const cfo_particles *pd = c->pdg;
  int err = 0;
  const int dchosen = particle_chosen_index(c, daughter, &err);
  const double members = (partner == daughter) ? 2.0 : 1.0;
  const double mD = pd->mass[daughter], mD2 = mD * mD, W = pd->mass[partner];
  const double Estar = (M * M + mD2 - W * W) / (2.0 * M), pstar = sqrt(Estar * Estar - mD2);
  const double prefactor = members * M * branch_ratio / (8.0 * pstar);
  setup_parent_tables(c, M);
  const double Ymax = fabs(c->dim == 2 ? 0.0 : c->y[c->y_pts - 1]);
  const double MTmax = c->MTValues[c->n_pT - 1];
  const double two_Pi = 2.0 * M_PI, M2 = M * M, Estar2 = Estar * Estar, Estar_M = Estar * M;
  for (int ipT = 0; ipT < c->n_pT; ipT++)
    for (int iphip = 0; iphip < c->n_phi; iphip++)
      for (int iy = 0; iy < c->y_pts; iy++) {
        const double pT = c->pT[ipT], pT2 = pT * pT, mT2 = pT2 + mD2, mT = sqrt(mT2);
        const double M_pT = M * pT, Estar_M_mT = Estar_M * mT, Estar_M_over_pT = Estar_M / pT, Estar2_plus_pT2 = Estar2 + pT2;
        const double phip = c->phi[iphip], y = (c->dim == 2) ? 0.0 : c->y[iy];
        const double p[4] = {mT * cosh(y), pT * cos(phip), pT * sin(phip), mT * sinh(y)};
        const double DeltaY = log((pstar + sqrt(Estar2_plus_pT2)) / mT);
        double acc[5] = {0, 0, 0, 0, 0}, cond[5] = {0, 0, 0, 0, 0};
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
              double logdN, Sp[3], SD[4] = {0, 0, 0, 0}, yield = 1.0;
              fd_interp(c, Sstar, MT, Phi, iYL, iYR, YL, YR, Y, MTmax, &logdN, Sp);
              const double P[4] = {MT * cosh(Y), PT * cos(Phi), PT * sin(Phi), MT * sinh(Y)};
              if (has_law) cfo_fdw_chain(P, M, Sp, c->dim == 2, p, mD, alpha, beta, gamma, SD, &yield);
              const double w = prefactor * vw * GL_WEIGHT[iz] * MT * exp(logdN);
              const double term[5] = {w * SD[0], w * SD[1], w * SD[2], w * SD[3], w * yield};
              /* the boosts mix the components, so a component's rounding scales with the largest one (e.g. the helicity part alpha/2 n,
               * which the lab frame turns into a large four-vector whose small components are differences) */
              const double big = fmax(fmax(fabs(term[0]), fabs(term[1])), fmax(fabs(term[2]), fabs(term[3])));
              for (int r = 0; r < 5; r++) { acc[r] += term[r]; cond[r] += (r < 4 ? big : fabs(term[r])) * (1.0 + fabs(logdN)); }
            }
          }
        }
        const long k = dchosen + (long)c->n_chosen * (ipT + (long)c->n_pT * (iphip + (long)c->n_phi * iy));
        for (int r = 0; r < 5; r++) { if (r < 4 && !has_law) continue; S[r * n_total + k] += acc[r]; if (A) A[r * n_total + k] += cond[r]; }
      }
}

/* S: [St | Sx | Sy | Sz | Snorm] amended in place; A (optional): [5][n_total] conditioning.  Rows: MC ids, branching ratio, alpha, phi.
 * Returns 0, or < 0 for a table the library rejects (-20: id not in the list, -21: parent / daughter not stable, -22: branching ratio,
 * -23: alpha / phi, -24: masses), or the tail-fit error of cf_decays.c. */
int cfo_polarization_weak_decays(const cfo_particles *pdg, const int32_t *spin2, int32_t n_rows, const int32_t *parent_id, const int32_t *daughter_id,
                                 const int32_t *partner_id, const double *branching, const double *alpha_in, const double *phi_in, int32_t n_chosen,
                                 const int32_t *chosen_pdg_index, const cfo_grid *g, int32_t dimension, double *S, double *A)
{
  if (g->n_pT > 512) return -15;
  const long n_total = (long)n_chosen * g->n_pT * g->n_phi * g->n_y;
  int *rp = (int *)calloc((size_t)n_rows + 1, sizeof(int)), *rd = (int *)calloc((size_t)n_rows + 1, sizeof(int)), *rm = (int *)calloc((size_t)n_rows + 1, sizeof(int));
  double *brsum = (double *)calloc((size_t)pdg->n_particles, sizeof(double));
  int rc = 0;
  for (int r = 0; r < n_rows && !rc; r++) {
    int e = 0;
    rp[r] = particle_index(pdg, parent_id[r], &e); rd[r] = particle_index(pdg, daughter_id[r], &e); rm[r] = particle_index(pdg, partner_id[r], &e);
    if (e) { rc = -20; break; }
    if (!pdg->stable[rp[r]] || !pdg->stable[rd[r]]) { rc = -21; break; }
    if (!(branching[r] >= 0.0 && branching[r] <= 1.0)) { rc = -22; break; }
    brsum[rp[r]] += branching[r];
    if (brsum[rp[r]] > 1.0 + 1e-9) { rc = -22; break; }
    if (!isfinite(alpha_in[r]) || !isfinite(phi_in[r]) || fabs(alpha_in[r]) > 1.0) { rc = -23; break; }
    if (pdg->mass[rd[r]] + pdg->mass[rm[r]] >= pdg->mass[rp[r]]) { rc = -24; break; }
  }
  ctx_t c; memset(&c, 0, sizeof(c));
  c.pdg = pdg; c.n_chosen = n_chosen; c.chosen = chosen_pdg_index;
  c.n_pT = g->n_pT; c.n_phi = g->n_phi; c.n_y_tab = g->n_y; c.dim = dimension; c.y_pts = (dimension == 2) ? 1 : g->n_y;
  c.pT = g->pT; c.phi = g->phi; c.y = g->y; c.dN = S + 4 * n_total;
  const long n_tab = (long)c.n_pT * c.n_phi * c.n_y_tab;
  c.logdN = (double *)calloc((size_t)n_tab, sizeof(double));
  c.fit = (mt_fit *)calloc((size_t)c.y_pts * c.n_phi, sizeof(mt_fit));
  double *Sstar = (double *)calloc((size_t)n_tab * 3, sizeof(double));
  /* weak parents among the chosen species (a row with a chosen daughter), by descending mass, ties by descending chosen index */
  int *order = (int *)calloc((size_t)n_chosen + 1, sizeof(int)), n_order = 0;
  for (int ic = 0; ic < n_chosen && !rc; ic++) {
    int any = 0;
    for (int r = 0; r < n_rows; r++) {
      int e = 0;
      if (rp[r] == chosen_pdg_index[ic]) { particle_chosen_index(&c, rd[r], &e); if (!e) any = 1; }
    }
    if (any) order[n_order++] = ic;
  }
  for (int i = 1; i < n_order; i++)                        /* insertion sort: heavier first, then higher chosen index */
    for (int j = i; j > 0; j--) {
      const double ma = pdg->mass[chosen_pdg_index[order[j - 1]]], mb = pdg->mass[chosen_pdg_index[order[j]]];
      if (mb > ma || (mb == ma && order[j] > order[j - 1])) { const int t = order[j]; order[j] = order[j - 1]; order[j - 1] = t; }
      else break;
    }
  for (int o = 0; o < n_order && !rc && !c.err; o++) {
    const int ichosen = order[o], ipart = chosen_pdg_index[ichosen];
    const double m = pdg->mass[ipart];
    for (int ipT = 0; ipT < c.n_pT; ipT++)
      for (int iphip = 0; iphip < c.n_phi; iphip++)
        for (int iy = 0; iy < c.y_pts; iy++) {
          const long it = ipT + (long)c.n_pT * (iphip + (long)c.n_phi * iy);
          const long iS3D = ichosen + (long)n_chosen * it;
          c.logdN[it] = log(c.dN[iS3D]);
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
    for (int r = 0; r < n_rows && !c.err; r++) {
      if (rp[r] != ipart) continue;
      int e = 0;
      particle_chosen_index(&c, rd[r], &e);
      if (e) continue;
      const int law = spin2[ipart] == 1 && spin2[rd[r]] == 1 && spin2[rm[r]] == 0;
      const double t = sqrt(1.0 - alpha_in[r] * alpha_in[r]);
      weak_row(&c, S, n_total, A, Sstar, law, alpha_in[r], t * sin(phi_in[r]), t * cos(phi_in[r]), branching[r], rd[r], rm[r], m);
    }
  }
  if (!rc) rc = c.err;
  free(rp); free(rd); free(rm); free(brsum); free(order); free(c.logdN); free(c.fit); free(Sstar);
  return rc;
}
