// cf_kernels.cu -- the smooth Cooper-Frye hot kernels (sm_100a), replacing the loop nest of
// EmissionFunctionArray::calculate_dN_pTdpTdphidy (reference src/cpp/emissionfunction_smooth_kernels.cpp:246-347).
//
// Work decomposition
//   lane  <-> one (species, pT) pair: idx = ipart * n_pT + ipT, 32 consecutive idx per warp.  Everything that
//             depends on the cell is then warp-uniform, so cell records are read from shared memory as broadcasts.
//   thread    keeps a register tile of NYT x NPT accumulators (rapidity slots x phi points) and walks the cells.
//   block     up to 4 warps (128 (species,pT) pairs) sharing one (y-tile, phi-tile) and one contiguous cell chunk;
//             cell tiles (CT cells x (NYT + NPT) records x 48 B + scalars) are streamed global -> shared with
//             cp.async.bulk (TMA) through a kStages-deep mbarrier pipeline.
//   grid      bin tiles x cell chunks; every block writes its partial spectra to partial[chunk][bin] (no atomics),
//             reduce_kernel sums the chunks in a fixed order and adds the result into the caller's array.
//
// Per evaluation (df_mode 1): ~22 FP64-pipe instructions in a fully alive group (u.p 1, p.dsigma 1, delta-f polynomial 4,
// exp(-x) 9 with the shared-memory table, Bose/Fermi factor 3 (dilute) or 5, df, f, accumulate 3, + ~1 of amortised hoists)
// against the 85 flops of the reference's inner loop (SURVEY.md 8d) -- cosh/sinh, the divisions and the tensor contraction
// are hoisted into the per-cell records by cf_prepare.cu, the lane-independent shear cross term into a per-tile pair table.
#include "cf_internal.h"
#include <algorithm>
#include "cf_device.cuh"
#include "cf_epilogue.cuh"

namespace is3d {

// SB selects how the NPT evaluations of a (cell, slot) are scheduled:
//   0  one divergent region per evaluation (distribution());
//   1  the NPT evaluations form one staged group (distribution_group()): their exp / reciprocal chains interleave (ILP); the
//      price is that a group is evaluated as soon as one member is alive (group_flags() in cf_device.cuh: how dead members
//      end up contributing an exact 0);
//   3  like 1 with e^{-x} = e^{-mT Ax} e^{+pT Bx} factored into one exponential per slot and one per phi point (2+1D default);
//   4  like 1 with the classification of slot j + 1 issued before slot j is evaluated (3+1D default).
// exp_neg_group: e^{-x[i]} for a group of N arguments, the slow branch (sub-normal results, dead members) taken once per group
template <int N>
__device__ __forceinline__ void exp_neg_group(const double (&x)[N], bool maybe_rare, double (&a)[N])
{
  double p[N]; int n[N];
#pragma unroll
  for (int i = 0; i < N; i++) exp_neg_poly(x[i], p[i], n[i]);
  if (__builtin_expect(maybe_rare, 0)) {              // both sides define a[]: no register shuffling on the fast side
#pragma unroll
    for (int i = 0; i < N; i++) a[i] = exp_neg_slow(x[i], p[i], n[i]);
  } else {
#pragma unroll
    for (int i = 0; i < N; i++) a[i] = exp_neg_fast(p[i], n[i]);
  }
}

// f_eq (1 + df) from a = e^{-x} (already evaluated) and the delta-f polynomial
template <int MODEL>
__device__ __forceinline__ double distribution_from_a(double a, double x, double s, double K2, double K3, double sign, int reg_thr, int one_hi,
                                                      bool dilute)
{
  double feqbar, feq;
  if (dilute) feq = occupation_bar_dilute(a, sign, feqbar);
  else feq = occupation_bar(a, sign, feqbar);
  if (MODEL == M_IDEAL) return feq;
  double dfs;
  if (MODEL == M_LIN14) dfs = fma(K2 * x, x, s);
  else dfs = fma(s, rcp_fast(x), K2 * x);
  double df = (MODEL == M_JONAHLIN) ? fma(feqbar, dfs, K3) : feqbar * dfs;
  df = clamp_unit(df, reg_thr, one_hi);
  return fma(feq, df, feq);
}

// The same stages for a group whose a[i] = e^{-x[i]} are already known (shifted-factor exponential, SB >= 5): the dilute / full
// occupation branch wraps the whole group, so that it stays a branch (a per-member `if` gets if-converted: both sides executed)
template <int MODEL, int N>
__device__ __forceinline__ void distribution_group_from_a(const double (&a)[N], const double (&x)[N], bool all_dilute, const double (&s)[N], double K2,
                                                          double K3, double sign, int reg_thr, int one_hi, double (&f)[N])
{
  double dfs[N], feq[N], feqbar[N];
#pragma unroll
  for (int i = 0; i < N; i++) {
    if (MODEL == M_IDEAL) dfs[i] = 0.0;
    else if (MODEL == M_LIN14) dfs[i] = fma(K2 * x[i], x[i], s[i]);
    else dfs[i] = fma(s[i], rcp_fast(x[i]), K2 * x[i]);
  }
  if (all_dilute) {
#pragma unroll
    for (int i = 0; i < N; i++) feq[i] = occupation_bar_dilute(a[i], sign, feqbar[i]);
  } else {
#pragma unroll
    for (int i = 0; i < N; i++) feq[i] = occupation_bar(a[i], sign, feqbar[i]);
  }
#pragma unroll
  for (int i = 0; i < N; i++) {
    if (MODEL == M_IDEAL) { f[i] = feq[i]; continue; }
    double df = (MODEL == M_JONAHLIN) ? fma(feqbar[i], dfs[i], K3) : feqbar[i] * dfs[i];
    df = clamp_unit(df, reg_thr, one_hi);
    f[i] = fma(feq[i], df, feq[i]);
  }
}

template <int MODEL, int NYT, int NPT, bool DIM2, int MINB, int SB>
__global__ void __launch_bounds__(block_warps(MINB) * 32, MINB)
cf_kernel(const HotParams hp)
{
  constexpr int RY = (MODEL == M_VAH) ? kRecVah : kRec;       // doubles per slot record
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const Layout &L = hp.L;
  const int nst = DIM2 ? L.nst : NYT;                         // slots per cell in this block's tile
  const int CT = L.ct;
  const int y_doubles = CT * nst * RY, p_doubles = CT * NPT * kRec, s_doubles = CT * kScal;
  const int stage_doubles = y_doubles + p_doubles + s_doubles;
  double *stage_base = reinterpret_cast<double *>(smem_raw);
  uint64_t *full = reinterpret_cast<uint64_t *>(stage_base + (size_t)kStages * stage_doubles);
  // linear models, 3+1D: per-tile table of the lane-independent part of the shear term (see "pair table" below)
  constexpr bool PAIR = !DIM2 && (MODEL == M_LIN14 || MODEL == M_LINCE || MODEL == M_JONAHLIN || MODEL == M_VAH);
  // modified equilibrium, 3+1D: the same table holds 2 v[slot].w[phi] for the expanded form of |p'|^2 (well-conditioned cells)
  constexpr bool PAIRF = !DIM2 && MODEL == M_FEQMOD;
  double *pair_tab = reinterpret_cast<double *>(full + kStages);

  // ---- task decode: blockIdx -> (group block, y tile, phi tile, cell chunk)
  const int n_bintiles = hp.n_groupblocks * L.n_ytiles * L.n_ptiles;
  const int chunk = blockIdx.x / n_bintiles;
  int bt = blockIdx.x - chunk * n_bintiles;
  const int tp = bt % L.n_ptiles; bt /= L.n_ptiles;
  const int ty = bt % L.n_ytiles; bt /= L.n_ytiles;
  const int gb = bt;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // ---- this lane's (species, pT)
  const int idx = (gb * hp.n_warps + warp) * 32 + lane;
  const bool lane_valid = idx < L.n_species * L.n_pT;
  const int ipart = lane_valid ? idx / L.n_pT : 0;
  const int ipT = lane_valid ? idx - ipart * L.n_pT : 0;
  const double mass = hp.mass[ipart], sign = hp.sign[ipart], pT = hp.pT[ipT];
  const double m2 = mass * mass, pT2 = pT * pT;
  const double mT2 = m2 + pT2;
  const double mT = sqrt(mT2);
  const double mTpT = mT * pT;
  const int reg_thr = hp.regulate_thr;
  const int one_hi = hp.one_hi;                               // high word of 1.0, kept in a register (see clamp_unit)
  const long long thr = hp.outflow_thr;
  const int thr_hi = (int)(thr >> 32);                       // grouped paths test the high word of p.dsigma only
  const double *renorm = (MODEL == M_FEQMOD && hp.renorm) ? hp.renorm + (int64_t)ipart * L.n_cells_pad : nullptr;

  // ---- cell tiles of this chunk: balanced contiguous split of [0, n_tiles), or the caller's table ((tau, r) bins)
  const int64_t t_begin = hp.chunk_tiles ? hp.chunk_tiles[chunk] : (L.n_tiles * (int64_t)chunk) / hp.n_chunks;
  const int64_t t_end = hp.chunk_tiles ? hp.chunk_tiles[chunk + 1] : (L.n_tiles * (int64_t)(chunk + 1)) / hp.n_chunks;
  const int n_my_tiles = (int)(t_end - t_begin);

  const double *Yg = hp.Y + ((int64_t)ty * L.n_cells_pad) * nst * RY;
  const double *Pg = hp.P + ((int64_t)tp * L.n_cells_pad) * NPT * kRec;
  const double *Sg = hp.S;
  const uint32_t stage_bytes = (uint32_t)stage_doubles * 8u;

  exp_table_init();
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  auto issue = [&](int t_local) {
    const int st = t_local % kStages;
    const int64_t cell = (t_begin + t_local) * CT;
    double *dst = stage_base + (size_t)st * stage_doubles;
    mbar_arrive_expect_tx(&full[st], stage_bytes);
    bulk_g2s(dst, Yg + cell * nst * RY, (uint32_t)y_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles, Pg + cell * NPT * kRec, (uint32_t)p_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles + p_doubles, Sg + cell * kScal, (uint32_t)s_doubles * 8u, &full[st]);
  };
  if (threadIdx.x == 0)
    for (int t = 0; t < kStages && t < n_my_tiles; t++) issue(t);

  constexpr int NACC = DIM2 ? NPT : NYT * NPT;
  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; i++) acc[i] = 0.0;

  for (int t = 0; t < n_my_tiles; t++) {
    const int st = t % kStages;
    mbar_wait(&full[st], (uint32_t)((t / kStages) & 1));
    const double *Ys = stage_base + (size_t)st * stage_doubles;
    const double *Ps = Ys + y_doubles;
    const double *Ss = Ps + p_doubles;
    const int64_t cell_base = (t_begin + t) * CT;

    // Pair table: coef pi^{mu nu} p_mu p_nu contains mT pT (R2[phi] U2[slot] - R1[phi] U1[slot]); the bracket does not depend on
    // the lane, so the block computes it once per (cell, slot, phi) of the tile (2 FP64 ops) instead of every thread spending
    // 2 DFMA + 2 hoisted DMUL on it per evaluation.  It also frees the registers of g1, g2, h1, h2.
    if (PAIR || PAIRF) {
      for (int w = threadIdx.x; w < CT * NYT * NPT; w += blockDim.x) {
        const int c = w / (NYT * NPT), r = w - c * (NYT * NPT), j = r / NPT, k = r - j * NPT;
        const double *yr = Ys + (c * nst + j) * RY, *pr = Ps + (c * NPT + k) * kRec;
        double t;
        if (PAIRF) {
          t = 2.0 * fma(pr[2], yr[2], fma(pr[1], yr[1], pr[0] * yr[0]));      // 2 v.w
        } else {
          t = fma(pr[4], yr[4], -(pr[3] * yr[3]));
          if (MODEL == M_VAH) t = fma(-pr[5], yr[5], t);            // - c3 (z.p) W_perp.p, the third mixed term of the anisotropic df
        }
        pair_tab[w] = t;
      }
      __syncthreads();
    }

    for (int c = 0; c < CT; c++) {
      const double2 k01 = *reinterpret_cast<const double2 *>(Ss + c * kScal);
      const double K2 = k01.y;                                   // linear / vah: coefficient of x^2 (or x); feqmod: per-cell renorm
      const double K3 = (MODEL == M_JONAHLIN) ? Ss[c * kScal + 2] : 0.0;
      // K0m: term proportional to m^2 (linear: Pi bulk0 m^2; feqmod: (m / T_mod)^2)
      const double K0m = k01.x * m2;
      double rn = 0.0;
      if (MODEL == M_FEQMOD) rn = renorm ? __ldg(renorm + cell_base + c) : K2;
      // feqmod: |p'|^2 = mT^2 |v|^2 + pT^2 |w|^2 + 2 mT pT v.w may be used where A^-1 does not amplify (flag set by the prepare
      // kernel, warp-uniform); elsewhere p' is formed component-wise, which keeps the rounding of ill-conditioned cells in parity
      const bool expanded = PAIRF && Ss[c * kScal + 2] != 0.0;

      // phi hoists: a few multiplies per (cell, phi), reused by every slot
      double q[NPT], pd[NPT], g0[NPT], g1[NPT], g2[NPT], g3[NPT];
      double fq[NPT]; int fm[NPT];                    // SB == 3: e^{+q[k]} = fq 2^fm (factored exponential)
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const double2 *pr = reinterpret_cast<const double2 *>(Ps + (c * NPT + k) * kRec);
        const double2 v0 = pr[0], v1 = pr[1], v2 = pr[2];
        if (MODEL == M_FEQMOD) {
          // p'/T_mod = mT v + pT w is formed component-wise and then squared: expanding |p'|^2 into |v|^2, v.w, |w|^2 would
          // amplify rounding by the square of A^-1's largest eigenvalue (cells with detA << 1)
          g1[k] = pT * v0.x; g2[k] = pT * v0.y; g3[k] = pT * v1.x;         // pT w
          g0[k] = K0m;                                                     // (m/T_mod)^2
          if (PAIRF) fq[k] = fma(pT2, v1.y, K0m);                          // pT^2 |w|^2 + (m/T_mod)^2 (expanded form; fq is free here)
          pd[k] = pT * v2.x; q[k] = 0.0;
        } else {
          q[k] = pT * v0.x;                 // pT * (cos ux + sin uy)/T
          pd[k] = pT * v0.y;                // pT * (cos dsigma_x + sin dsigma_y)
          g0[k] = fma(pT2, v1.x, K0m);      // pT^2 Qpp + (..) m^2
          g1[k] = PAIR ? 0.0 : pT * v1.y;
          g2[k] = PAIR ? 0.0 : pT * v2.x;
          g3[k] = (MODEL == M_VAH && !PAIR) ? pT * v2.y : 0.0;             // pT (Wx cos + Wy sin)
          if (SB == 3) exp_neg_poly(-q[k], fq[k], fm[k]);
        }
      }
      // SB >= 5 (linear models, 3+1D): shifted factorisation of the exponential.  With qm = max_k q[k] and d[k] = qm - q[k] >= 0,
      //   e^{-x_jk} = e^{-(a_j - qm)} e^{-d[k]}:  one exponential per slot (of the group's SMALLEST argument xm_j = a_j - qm) and
      // one per phi point and cell, a DMUL per evaluation.  Both factors lie in (0, 1], so -- unlike e^{-a_j} e^{+q_k} -- neither
      // can overflow or underflow before the product does: whenever xm_j + max d < 707.7 both factors and the product are normal
      // numbers; every other slot takes the per-member path below, which is the SB == 1 evaluation.  The group's aliveness and
      // diluteness follow from xm_j alone.
      double sd[NPT], eB[NPT]; int rare_hi = 0;
      if (SB >= 5 && MODEL != M_FEQMOD && MODEL != M_VAH) {
        double qm = q[0], qn = q[0];
#pragma unroll
        for (int k = 1; k < NPT; k++) { qm = fmax(qm, q[k]); qn = fmin(qn, q[k]); }
#pragma unroll
        for (int k = 0; k < NPT; k++) { sd[k] = qm - q[k]; double pp; int nn; exp_neg_poly(sd[k], pp, nn); eB[k] = exp_neg_fast(pp, nn); }
        // slot j is "rare" when xm_j >= 707.7 - (qm - qn); compared on the high words (negative threshold: always)
        rare_hi = __double2hiint(__hiloint2double(kRareHi, 0) - (qm - qn));
#pragma unroll
        for (int k = 0; k < NPT; k++) q[k] = qm;         // q[] is not needed any more; keep one live value
      }
      // delta-f polynomial without its (u.p)^2 part, linear models: mT^2 Qyy + pT^2 Qpp + (..) m^2 + mT pT (R2 U2 - R1 U1)
      auto sterm = [&](int j, int k, double h0, double h1, double h2) -> double {
        if (PAIR) return fma(mTpT, pair_tab[(c * NYT + j) * NPT + k], h0 + g0[k]);
        double s = h0 + g0[k];
        s = fma(g2[k], h2, s);
        return fma(-g1[k], h1, s);
      };
      auto slot = [&](int j, double *accj) {
        const double2 *yr = reinterpret_cast<const double2 *>(Ys + (c * nst + j) * RY);
        const double2 v0 = yr[0], v1 = yr[1], v2 = yr[2];
        if (MODEL == M_FEQMOD) {
          const double e1 = mT * v0.x, e2 = mT * v0.y, e3 = mT * v1.x, cpm = mT * v2.x, w = v2.y;
          if (SB == 0) {
#pragma unroll
            for (int k = 0; k < NPT; k++) {
              const double p1 = e1 + g1[k], p2 = e2 + g2[k], p3 = e3 + g3[k];
              double E2 = fma(p1, p1, g0[k]); E2 = fma(p2, p2, E2); E2 = fma(p3, p3, E2);   // (E'/T_mod)^2
              const double x = sqrt_fast(E2);
              const double pds = fma(w, pd[k], cpm);
              if (exp_finite(x)) {
                const double f = rn * occupation(exp_neg(x), sign);
                accumulate_outflow(accj[k], pds, f, thr);
              }
            }
          } else {
            double xv[NPT], pv[NPT], av[NPT]; bool any, rare, dilute;
            if (expanded) {
              const double Aj = mT2 * v1.y;                                // mT^2 |v|^2
#pragma unroll
              for (int k = 0; k < NPT; k++) xv[k] = sqrt_fast(fma(mTpT, pair_tab[(c * NYT + j) * NPT + k], Aj + fq[k]));
            } else {
#pragma unroll
              for (int k = 0; k < NPT; k++) {
                const double p1 = e1 + g1[k], p2 = e2 + g2[k], p3 = e3 + g3[k];
                double E2 = fma(p1, p1, g0[k]); E2 = fma(p2, p2, E2); E2 = fma(p3, p3, E2);
                xv[k] = sqrt_fast(E2);
              }
            }
#pragma unroll
            for (int k = 0; k < NPT; k++) pv[k] = fma(w, pd[k], cpm);
            group_flags<NPT>(xv, any, rare, dilute);
            if (DIM2) dilute = false;              // 2+1D groups are wide (light species, all eta): the extra branch costs more than it saves
            if (any) {
              exp_neg_group<NPT>(xv, rare, av);
              double fo[NPT], unused;
              if (dilute) {
#pragma unroll
                for (int k = 0; k < NPT; k++) fo[k] = occupation_bar_dilute(av[k], sign, unused);
              } else {
#pragma unroll
                for (int k = 0; k < NPT; k++) fo[k] = occupation(av[k], sign);
              }
#pragma unroll
              for (int k = 0; k < NPT; k++) accumulate_pos(accj[k], pv[k], rn * fo[k], thr_hi);
            }
          }
        } else if (MODEL == M_VAH) {
          const double2 v3 = yr[3];
          const double a = mT * v0.x, cpm = mT * v0.y, h0 = mT2 * v1.x, h1 = mT * v1.y, h2 = mT * v2.x, h3 = mT * v2.y;
          const double hz = mT2 * v3.x, w = v3.y;
          if (SB == 0) {
#pragma unroll
            for (int k = 0; k < NPT; k++) {
              const double u = a - q[k];                                   // u.p / Lambda
              const double x = sqrt_fast(fma(u, u, hz));                   // E_a / Lambda
              const double pds = fma(w, pd[k], cpm);
              if (exp_finite(x)) {
                double s;
                if (PAIR) s = fma(mTpT, pair_tab[(c * NYT + j) * NPT + k], h0 + g0[k]);
                else { s = h0 + g0[k]; s = fma(g2[k], h2, s); s = fma(-g1[k], h1, s); s = fma(-g3[k], h3, s); }
                s = fma(K2 * u, u, s);
                const double fa = occupation(exp_neg(x), sign);
                const double fabar = fma(-sign, fa, 1.0);
                const double df = clamp_unit(fabar * s, reg_thr, one_hi);
                accumulate_outflow(accj[k], pds, fma(fa, df, fa), thr);
              }
            }
          } else {
            double xv[NPT], pv[NPT], sv[NPT], av[NPT]; bool any, rare, dilute;
#pragma unroll
            for (int k = 0; k < NPT; k++) {
              const double u = a - q[k];
              xv[k] = sqrt_fast(fma(u, u, hz));
              pv[k] = fma(w, pd[k], cpm);
              double s;
              if (PAIR) s = fma(mTpT, pair_tab[(c * NYT + j) * NPT + k], h0 + g0[k]);
              else { s = h0 + g0[k]; s = fma(g2[k], h2, s); s = fma(-g1[k], h1, s); s = fma(-g3[k], h3, s); }
              sv[k] = fma(K2 * u, u, s);
            }
            group_flags<NPT>(xv, any, rare, dilute);
            if (DIM2) dilute = false;              // 2+1D groups are wide (light species, all eta): the extra branch costs more than it saves
            if (any) {
              exp_neg_group<NPT>(xv, rare, av);
              double fav[NPT], fbv[NPT];
              if (dilute) {
#pragma unroll
                for (int k = 0; k < NPT; k++) fav[k] = occupation_bar_dilute(av[k], sign, fbv[k]);
              } else {
#pragma unroll
                for (int k = 0; k < NPT; k++) fav[k] = occupation_bar(av[k], sign, fbv[k]);
              }
#pragma unroll
              for (int k = 0; k < NPT; k++) {
                const double fa = fav[k], fabar = fbv[k];
                const double df = clamp_unit(fabar * sv[k], reg_thr, one_hi);
                accumulate_pos(accj[k], pv[k], fma(fa, df, fa), thr_hi);
              }
            }
          }
        } else {
          const double a = mT * v0.x, cpm = mT * v0.y, h0 = mT2 * v1.x, h1 = mT * v1.y, h2 = mT * v2.x, w = v2.y;
          if (SB == 0) {
#pragma unroll
            for (int k = 0; k < NPT; k++) {
              const double x = a - q[k];
              const double pds = fma(w, pd[k], cpm);
              if (exp_finite(x)) {                           // else exp(x) overflows: f = 0 exactly
                const double s = sterm(j, k, h0, h1, h2);
                const double f = distribution<MODEL>(x, s, K2, K3, sign, reg_thr, one_hi);
                accumulate_outflow(accj[k], pds, f, thr);
              }
            }
          } else if (SB >= 5) {
            // shifted factorisation (see the per-cell hoists above): q[0] holds qm, sd[k] = qm - q_k, eB[k] = e^{-sd[k]}
            const double xm = a - q[0];                                     // smallest argument of the group
            const int xh = __double2hiint(xm);
            if (xh <= kAliveHi) {
              double xs[NPT], sv[NPT], pv[NPT];
#pragma unroll
              for (int k = 0; k < NPT; k++) {
                xs[k] = xm + sd[k];
                pv[k] = fma(w, pd[k], cpm);
                sv[k] = sterm(j, k, h0, h1, h2);
              }
              double fv[NPT];
              if (__builtin_expect(xh >= rare_hi, 0)) {                       // some member may be sub-normal or dead: per-member path
                distribution_group<MODEL, NPT>(xs, true, false, sv, K2, K3, sign, reg_thr, one_hi, fv);
              } else {
                double pe, av[NPT]; int ne;
                exp_neg_poly(xm, pe, ne);
                const double eA = exp_neg_fast(pe, ne);
#pragma unroll
                for (int k = 0; k < NPT; k++) av[k] = eA * eB[k];
                // a_k <= e^{-xm} < 2^-18 for every member once xm >= 12.5
                distribution_group_from_a<MODEL, NPT>(av, xs, xh >= kDiluteHi, sv, K2, K3, sign, reg_thr, one_hi, fv);
              }
#pragma unroll
              for (int k = 0; k < NPT; k++) accumulate_pos(accj[k], pv[k], fv[k], thr_hi);
            }
          } else if (SB == 3) {
            // e^{-x} = e^{-mT Ax} e^{+pT Bx}: one exponential per slot and one per phi point instead of one per evaluation
            double xs[NPT]; bool any, rare, dilute;
#pragma unroll
            for (int k = 0; k < NPT; k++) xs[k] = a - q[k];
            group_flags<NPT>(xs, any, rare, dilute);
            if (DIM2) dilute = false;
            if (any) {
              double pe; int ne;
              exp_neg_poly(a, pe, ne);
              double av[NPT];
              if (__builtin_expect(rare, 0)) {
#pragma unroll
                for (int k = 0; k < NPT; k++) av[k] = exp_neg_slow(xs[k], pe * fq[k], ne + fm[k]);
              } else {
#pragma unroll
                for (int k = 0; k < NPT; k++) av[k] = exp_neg_fast(pe * fq[k], ne + fm[k]);
              }
#pragma unroll
              for (int k = 0; k < NPT; k++) {
                const double pds = fma(w, pd[k], cpm);
                const double s = sterm(j, k, h0, h1, h2);
                accumulate_pos(accj[k], pds, distribution_from_a<MODEL>(av[k], xs[k], s, K2, K3, sign, reg_thr, one_hi, dilute), thr_hi);
              }
            }
          } else {
            double xs[NPT]; bool any, rare, dilute;
#pragma unroll
            for (int k = 0; k < NPT; k++) xs[k] = a - q[k];
            group_flags<NPT>(xs, any, rare, dilute);
            if (DIM2) dilute = false;
            if (any) {
              double sv[NPT], pv[NPT], fv[NPT];
#pragma unroll
              for (int k = 0; k < NPT; k++) {
                pv[k] = fma(w, pd[k], cpm);
                sv[k] = sterm(j, k, h0, h1, h2);
              }
              distribution_group<MODEL, NPT>(xs, rare, dilute, sv, K2, K3, sign, reg_thr, one_hi, fv);
#pragma unroll
              for (int k = 0; k < NPT; k++) accumulate_pos(accj[k], pv[k], fv[k], thr_hi);
            }
          }
        }
      };
      // SB == 4 (linear models, 3+1D): like SB == 1, but the aliveness test of slot j + 1 is issued before slot j is
      // evaluated, so that the skip branch of the next slot never waits for its predicate chain (DMUL, DADD, 2 ISETP)
      auto probe = [&](int j, double (&x)[NPT], bool &any, bool &rare, bool &dilute) {
        const double a = mT * Ys[(c * nst + j) * RY];
#pragma unroll
        for (int k = 0; k < NPT; k++) x[k] = a - q[k];
        group_flags<NPT>(x, any, rare, dilute);
      };
      auto eval_probed = [&](int j, const double (&x)[NPT], bool rare, bool dilute, double *accj) {
        const double2 *yr = reinterpret_cast<const double2 *>(Ys + (c * nst + j) * RY);
        const double2 v0 = yr[0], v1 = yr[1], v2 = yr[2];
        const double cpm = mT * v0.y, h0 = mT2 * v1.x, h1 = mT * v1.y, h2 = mT * v2.x, w = v2.y;
        double sv[NPT], pv[NPT], fv[NPT];
#pragma unroll
        for (int k = 0; k < NPT; k++) {
          pv[k] = fma(w, pd[k], cpm);
          sv[k] = sterm(j, k, h0, h1, h2);
        }
        distribution_group<MODEL, NPT>(x, rare, dilute, sv, K2, K3, sign, reg_thr, one_hi, fv);
#pragma unroll
        for (int k = 0; k < NPT; k++) accumulate_pos(accj[k], pv[k], fv[k], thr_hi);
      };
      if (DIM2) {
#pragma unroll 2
        for (int j = 0; j < nst; j++) slot(j, acc);
      } else if (SB == 4 && MODEL != M_FEQMOD && MODEL != M_VAH) {
        double xa[NPT], xb[NPT]; bool anya, rarea, dila, anyb = false, rareb = false, dilb = false;
        probe(0, xa, anya, rarea, dila);
#pragma unroll
        for (int j = 0; j < NYT; j++) {
          if (j + 1 < NYT) probe(j + 1, xb, anyb, rareb, dilb);
          if (anya) eval_probed(j, xa, rarea, dila, acc + j * NPT);
#pragma unroll
          for (int k = 0; k < NPT; k++) xa[k] = xb[k];
          anya = anyb; rarea = rareb; dila = dilb;
        }
      } else {
#pragma unroll
        for (int j = 0; j < NYT; j++) slot(j, acc + j * NPT);
      }
    }
    __syncthreads();                                   // every warp is done with stage st
    if (threadIdx.x == 0 && t + kStages < n_my_tiles) issue(t + kStages);
  }

  // ---- epilogue (cf_epilogue.cuh): spectra bins of this chunk, or the momentum-integrated numbers of operation = 0;
  //      every stage has been consumed, so the stage area doubles as the block scratch (launch_one sizes it for that)
  hot_epilogue<NYT, NPT, DIM2>(hp, acc, stage_base, chunk, gb, ty, tp, lane_valid, ipart, ipT);
}

// ------------------------------------------------------------------------------------------------ reduce
// n_active <= n_bins: only the bins the hot kernel writes (2+1D fills the iy = 0 plane, the first n_bins / n_y entries)
__global__ void reduce_kernel(const double *__restrict__ partial, int n_chunks, int64_t n_bins, int64_t n_active, double *__restrict__ out)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_active) return;
  double s = 0.0;
  for (int c = 0; c < n_chunks; c++) s += partial[(int64_t)c * n_bins + i];
  out[i] += s;
}

// integ -> out[unit][species]: fixed summation order (chunk, y tile, phi tile, group block), no atomics
__global__ void integ_reduce_kernel(const HotParams hp, int n_units, int nj, int block_lanes, double *__restrict__ out)
{
  const Layout &L = hp.L;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_units * L.n_species) return;
  const int unit = (int)(i / L.n_species), sidx = (int)(i - (int64_t)unit * L.n_species);
  const int gb_lo = (sidx * L.n_pT) / block_lanes, gb_hi = ((sidx + 1) * L.n_pT - 1) / block_lanes;
  double v = 0.0;
  auto add = [&](int64_t row) {                          // row = index of a [ptile][groupblock][sl] slab
    for (int tp = 0; tp < L.n_ptiles; tp++)
      for (int gb = gb_lo; gb <= gb_hi; gb++) {
        const int sl = sidx - (gb * block_lanes) / L.n_pT;
        v += hp.integ[((row * L.n_ptiles + tp) * hp.n_groupblocks + gb) * hp.integ_sl + sl];
      }
  };
  if (hp.integ_mode == 1) {                              // unit = chunk: sum the y tiles
    for (int ty = 0; ty < L.n_ytiles; ty++) add((int64_t)unit * L.n_ytiles + ty);
  } else {                                               // unit = slot: sum the chunks
    for (int c = 0; c < hp.n_chunks; c++) add((int64_t)c * (L.n_ytiles * nj) + unit);
  }
  out[i] = v;
}

cudaError_t launch_integ_reduce(const HotParams &hp, int n_units, double *out, cudaStream_t st)
{
  const int64_t n = (int64_t)n_units * hp.L.n_species;
  if (n == 0) return cudaSuccess;
  const bool summed = hp.L.dim2 && !hp.L.per_slot;
  const int nj = summed ? 1 : hp.L.nst;
  integ_reduce_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(hp, n_units, nj, hp.n_warps * 32, out);
  return cudaGetLastError();
}

// y[i] += x[i]
__global__ void axpy_kernel(const double *__restrict__ x, double *__restrict__ y, int64_t n)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] += x[i];
}

cudaError_t launch_axpy(const double *x, double *y, int64_t n, cudaStream_t st)
{
  if (n == 0) return cudaSuccess;
  axpy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, y, n);
  return cudaGetLastError();
}

cudaError_t launch_reduce(const double *partial, int n_chunks, int64_t n_bins, int64_t n_active, double *out, cudaStream_t st)
{
  if (n_active == 0) return cudaSuccess;
  reduce_kernel<<<(unsigned)((n_active + 255) / 256), 256, 0, st>>>(partial, n_chunks, n_bins, n_active, out);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------ dispatch
// Register-tile variants: (slots per tile, phi points per tile, cells per TMA tile, min blocks per SM, grouping SB).
// is3d_options.tile_variant = k selects entry k - 1 (0 = the tuned default of the model, chosen in cf_api.cu); every entry is
// compiled for every model and covered by tests/test_gpu_parity.py::test_every_tile_variant.  minb >= 7 means 2-warp blocks.
struct Shape { int nyt, npt, ct, minb, sb; };
static const Shape kShapes3D[] = {
  {7, 3, 8, 7, 4}, {7, 3, 8, 7, 1}, {7, 3, 16, 5, 4}, {7, 4, 16, 3, 4}, {7, 2, 16, 6, 4}, {3, 6, 16, 3, 0}, {7, 6, 16, 2, 4}, {7, 3, 16, 4, 0},
  {7, 3, 16, 4, 3}, {7, 3, 16, 3, 4}, {7, 3, 16, 3, 3}, {7, 3, 16, 4, 1}, {7, 3, 16, 3, 5}, {7, 4, 16, 3, 5}, {7, 2, 16, 6, 1}, {7, 3, 16, 4, 5}};
static const Shape kShapes2D[] = {
  {1, 3, 1, 4, 0}, {1, 4, 1, 4, 0}, {1, 6, 1, 3, 0}, {1, 8, 1, 3, 0}, {1, 2, 1, 5, 0}, {1, 12, 1, 2, 0}, {1, 4, 1, 3, 0}, {1, 1, 1, 6, 0},
  {1, 6, 1, 3, 3}, {1, 3, 1, 4, 1}, {1, 4, 1, 4, 3}, {1, 4, 1, 3, 1}, {1, 6, 1, 3, 1}, {1, 8, 1, 3, 3}, {1, 3, 1, 5, 1}, {1, 12, 1, 2, 3}};

void hot_variant_shape(int variant, int dim2, int *nyt, int *npt, int *ct, int *max_warps)
{
  if (variant < 0 || variant >= kNumVariants) variant = 0;
  const Shape &s = dim2 ? kShapes2D[variant] : kShapes3D[variant];
  *nyt = s.nyt; *npt = s.npt; *ct = s.ct; *max_warps = block_warps(s.minb);
}

template <int MODEL, int NYT, int NPT, bool DIM2, int MINB, int SB>
static cudaError_t launch_one(const HotParams &hp, cudaStream_t st, size_t *smem_out)
{
  const Layout &L = hp.L;
  constexpr int RY = (MODEL == M_VAH) ? kRecVah : kRec;
  const int nst = DIM2 ? L.nst : NYT;
  const size_t stage_doubles = (size_t)L.ct * nst * RY + (size_t)L.ct * NPT * kRec + (size_t)L.ct * kScal;
  constexpr bool PAIR = !DIM2 && (MODEL == M_LIN14 || MODEL == M_LINCE || MODEL == M_JONAHLIN || MODEL == M_VAH || MODEL == M_FEQMOD);
  // operation = 0: the epilogue reuses the stage area as [per_slot][threads] scratch -- make sure it is large enough
  const size_t stage_bytes = std::max(kStages * stage_doubles * 8, (hot_epilogue_scratch_bytes(hp, NYT, DIM2, hp.n_warps * 32) + 15) & ~(size_t)15);
  const size_t smem = stage_bytes + kStages * sizeof(uint64_t) + (PAIR ? (size_t)L.ct * NYT * NPT * 8 : 0);
  if (smem_out) *smem_out = smem;
  auto kern = cf_kernel<MODEL, NYT, NPT, DIM2, MINB, SB>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)hp.n_groupblocks * L.n_ytiles * L.n_ptiles * hp.n_chunks;
  if (grid == 0) return cudaSuccess;
  kern<<<(unsigned)grid, hp.n_warps * 32, smem, st>>>(hp);
  return cudaGetLastError();
}

template <int MODEL>
static cudaError_t launch_model(const HotParams &hp, int variant, cudaStream_t st, size_t *smem_out)
{
  constexpr bool TUNE = true;
  if (hp.L.dim2 && !hp.L.per_slot) {
    switch (variant) {
      case 1: return launch_one<MODEL, 1, 4, true, 4, 0>(hp, st, smem_out);
      case 2: return launch_one<MODEL, 1, 6, true, 3, 0>(hp, st, smem_out);
      case 3: return launch_one<MODEL, 1, 8, true, 3, 0>(hp, st, smem_out);
      case 4: return launch_one<MODEL, 1, 2, true, 5, 0>(hp, st, smem_out);
      case 5: return launch_one<MODEL, 1, 12, true, 2, 0>(hp, st, smem_out);
      case 6: return launch_one<MODEL, 1, 4, true, 3, 0>(hp, st, smem_out);
      case 7: return launch_one<MODEL, 1, 1, true, 6, 0>(hp, st, smem_out);
      default: break;
    }
    if constexpr (TUNE) {
      switch (variant) {
        case 8: return launch_one<MODEL, 1, 6, true, 3, 3>(hp, st, smem_out);
        case 9: return launch_one<MODEL, 1, 3, true, 4, 1>(hp, st, smem_out);
        case 10: return launch_one<MODEL, 1, 4, true, 4, 3>(hp, st, smem_out);
        case 11: return launch_one<MODEL, 1, 4, true, 3, 1>(hp, st, smem_out);
        case 12: return launch_one<MODEL, 1, 6, true, 3, 1>(hp, st, smem_out);
        case 13: return launch_one<MODEL, 1, 8, true, 3, 3>(hp, st, smem_out);
        case 14: return launch_one<MODEL, 1, 3, true, 5, 1>(hp, st, smem_out);
        case 15: return launch_one<MODEL, 1, 12, true, 2, 3>(hp, st, smem_out);
        default: break;
      }
    }
    return launch_one<MODEL, 1, 3, true, 4, 0>(hp, st, smem_out);
  }
  switch (variant) {
    case 1: return launch_one<MODEL, 7, 3, false, 7, 1>(hp, st, smem_out);
    case 2: return launch_one<MODEL, 7, 3, false, 5, 4>(hp, st, smem_out);
    case 3: return launch_one<MODEL, 7, 4, false, 3, 4>(hp, st, smem_out);
    case 4: return launch_one<MODEL, 7, 2, false, 6, 4>(hp, st, smem_out);
    case 5: return launch_one<MODEL, 3, 6, false, 3, 0>(hp, st, smem_out);
    case 6: return launch_one<MODEL, 7, 6, false, 2, 4>(hp, st, smem_out);
    case 7: return launch_one<MODEL, 7, 3, false, 4, 0>(hp, st, smem_out);
    default: break;
  }
  if constexpr (TUNE) {
    switch (variant) {
      case 8: return launch_one<MODEL, 7, 3, false, 4, 3>(hp, st, smem_out);
      case 9: return launch_one<MODEL, 7, 3, false, 3, 4>(hp, st, smem_out);
      case 10: return launch_one<MODEL, 7, 3, false, 3, 3>(hp, st, smem_out);
      case 11: return launch_one<MODEL, 7, 3, false, 4, 1>(hp, st, smem_out);
      case 12: return launch_one<MODEL, 7, 3, false, 3, 5>(hp, st, smem_out);
      case 13: return launch_one<MODEL, 7, 4, false, 3, 5>(hp, st, smem_out);
      case 14: return launch_one<MODEL, 7, 2, false, 6, 1>(hp, st, smem_out);
      case 15: return launch_one<MODEL, 7, 3, false, 4, 5>(hp, st, smem_out);
      default: break;
    }
  }
  return launch_one<MODEL, 7, 3, false, 7, 4>(hp, st, smem_out);
}

cudaError_t launch_hot(int model, const HotParams &hp, int variant, cudaStream_t st, size_t *smem_out)
{
  switch (model) {
    case M_LIN14: return launch_model<M_LIN14>(hp, variant, st, smem_out);
    case M_LINCE: return launch_model<M_LINCE>(hp, variant, st, smem_out);
    case M_FEQMOD: return launch_model<M_FEQMOD>(hp, variant, st, smem_out);
    case M_JONAHLIN: return launch_model<M_JONAHLIN>(hp, variant, st, smem_out);
    case M_VAH: return launch_model<M_VAH>(hp, variant, st, smem_out);
    case M_IDEAL: return launch_model<M_IDEAL>(hp, variant, st, smem_out);
    default: return cudaErrorInvalidValue;
  }
}

// ------------------------------------------------------------------------------------------------ FP64 peak probe
// 8 independent DFMA chains per thread, no memory traffic: measures the FP64-pipe roof used as roofline denominator.
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *sink, int iters)
{
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 123.456) sink[0] = s;
}

cudaError_t launch_fp64_peak(double *sink, int iters, cudaStream_t st, int *blocks, int *threads, long long *dfma_per_thread)
{
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  *blocks = sms * 8; *threads = 256; *dfma_per_thread = (long long)iters * 64;
  fp64_peak_kernel<<<*blocks, *threads, 0, st>>>(sink, iters);
  return cudaGetLastError();
}

}  // namespace is3d
