// cf_spin_density.cu -- spin density matrix of the emitted hadrons from a thermal-vorticity (mode 5) surface, to all orders in the
// thermal vorticity (sm_100a).
//
// Per momentum bin p and species (m, g = 2J + 1, Theta = sign), over the cells, rapidity slots and weights of cf_polzn.cu, with the
// spin term of the local-equilibrium distribution exponentiated, [exp(beta.p - (1/2) varpi:Sigma) + Theta]^-1 (Becattini, Chandra,
// Del Zanna, Grossi 2013):
//   theta^mu = -(1/(2m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau = (1/m) (omega.p, E omega - e x p)
//   theta*_i = theta^i - theta^t p^i / (E + m)        (rest frame of the pure boost along p),  theta = |theta*|,  that = theta* / theta
//   f_m      = 1 / (exp(u.p/T - m theta) + Theta),    m = -J .. J along that
//   Snorm = K sum W sum_m f_m,   P_i = K sum W sum_m m f_m that_i,   Q_ij = K sum W sum_m f_m (3m^2 - J(J+1))/2 (that_i that_j - delta_ij/3)
// with K = 1/(2 pi hbar c)^3 and W = slot weight x p.dsigma.  Only the varpi term is exponentiated: rho00 - 1/3 from Q is the second
// order of that exponent, not a complete second-order gradient expansion (shear-induced alignment and other terms are not included).
//
// The level sums pair +m with -m.  With e = exp(-u.p/T), D_m = (1 + Theta e)^2 + 2 Theta e (cosh m theta - 1):
//   f_m - f_-m           = 2 e sinh(m theta) / D_m
//   f_m + f_-m - 2 f_ref = 2 e (1 - Theta e) / (1 + Theta e) (cosh m theta - 1) / D_m,    f_ref = e / (1 + Theta e)
// and sum_m (3m^2 - J(J+1)) = 0, so Q sees only the paired excess, which is O(theta^2) and formed without cancellation: sinh(m theta)
// and cosh(m theta) - 1 come from sinh(theta/2) by a recurrence of positive terms.  Everything is in powers of e = exp(-x) <= 1, so no
// level overflows, and an evaluation whose exp(u.p/T) overflows contributes exact zeros, as in cf_polzn.cu.  P and Q are summed as
// W (sum_m ...)/theta * theta*_i and W (sum_m ...)/theta^2 * (theta*_i theta*_j - theta^2 delta_ij/3): finite, and exactly 0, at theta = 0.
//
// Bosons: f_J is no occupation when u.p/T - J theta <= 0.  Such evaluations are not added; each block counts them and adds its count
// to one device counter with one atomic, and the caller refuses the call.
//
// cf_spin_density_kernel: the decomposition of cf_polzn_kernel on the unchanged records of prepare_polzn_kernel (lanes = (species, pT)
//                         pairs, cell tiles streamed through the TMA / mbarrier pipeline, a register tile of NYT x NPT bins x 9 sums),
//                         one partial row per cell chunk and array, summed by launch_reduce in a fixed order: no atomics on the sums,
//                         results are bit-reproducible.  The ideal-f statements (u.p/T, p.dsigma, the outflow test, f) are those of
//                         cf_polzn_kernel, so at theta = 0 every evaluation adds to Snorm exactly what the vorticity kernel adds.
#include "cf_internal.h"
#include "cf_device.cuh"

namespace is3d {

// pT b^mu for (omega.p, E omega - e x p) at phi = (pc, ps) / pT (the b of cf_polzn.cu)
__device__ __forceinline__ void sd_b(double ex, double ey, double ez, double ox, double oy, double pc, double ps, double b[4])
{
  b[0] = fma(ox, pc, oy * ps);
  b[1] = ez * ps;
  b[2] = -ez * pc;
  b[3] = fma(ey, pc, -ex * ps);
}

// sinh(h), h >= 0, to a few ulp: Taylor series below 1/4 (truncation < 1e-17 relative), exp above (cancellation <= 4 ulp there)
__device__ __forceinline__ double sinh_pos(double h)
{
  if (h < 0.25) {
    const double h2 = h * h;
    double s = fma(h2, 1.0 / 39916800.0, 1.0 / 362880.0);
    s = fma(s, h2, 1.0 / 5040.0);
    s = fma(s, h2, 1.0 / 120.0);
    s = fma(s, h2, 1.0 / 6.0);
    return fma(s * h2, h, h);
  }
  const double E = exp(h);
  return 0.5 * (E - 1.0 / E);
}

// Register tile: NYT rapidity slots (3+1D; 2+1D sums every eta slot into one) x NPT phi points x 9 sums
// (Snorm, P_x, P_y, P_z, Q_xx, Q_xy, Q_xz, Q_yy, Q_yz)
template <int NYT, int NPT, bool DIM2>
__global__ void __launch_bounds__(kPolWarps * 32, kSdMinBlocks)
cf_spin_density_kernel(const SpinDensityParams prm)
{
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ unsigned long long blk_bad;
  const HotParams &hp = prm.hp;
  const Layout &L = hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const int CT = L.ct;
  const int y_doubles = CT * nst * kPolRecY, p_doubles = CT * NPT * kPolRecP;
  const int stage_doubles = y_doubles + p_doubles;
  double *stage_base = reinterpret_cast<double *>(smem_raw);
  uint64_t *full = reinterpret_cast<uint64_t *>(stage_base + (size_t)kStages * stage_doubles);

  const int n_bintiles = hp.n_groupblocks * L.n_ytiles * L.n_ptiles;
  const int chunk = blockIdx.x / n_bintiles;
  int bt = blockIdx.x - chunk * n_bintiles;
  const int tp = bt % L.n_ptiles; bt /= L.n_ptiles;
  const int ty = bt % L.n_ytiles; bt /= L.n_ytiles;
  const int gb = bt;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int idx = (gb * hp.n_warps + warp) * 32 + lane;
  const bool lane_valid = idx < L.n_species * L.n_pT;
  const int ipart = lane_valid ? idx / L.n_pT : 0;
  const int ipT = lane_valid ? idx - ipart * L.n_pT : 0;
  const double mass = hp.mass[ipart], sign = hp.sign[ipart], pT = hp.pT[ipT];
  const double mT = sqrt(fma(mass, mass, pT * pT));
  const long long thr = hp.outflow_thr;
  const double g = hp.degeneracy[ipart];
  const int n_pairs = (int)g >> 1;                     // levels m > 0: J, J - 1, .. down to 1/2 or 1
  const bool half_int = ((int)g & 1) == 0;
  const double J = 0.5 * (g - 1.0), JJ1 = J * (J + 1.0);
  const double inv_m = 1.0 / mass, inv_g = 1.0 / g;
  // the bin's p^z and 1 / (E + m): theta*_i = inv_m (v^i - v^t p^i c), c = 1 / (E + m); 2+1D bins have y = 0
  double cE[DIM2 ? 1 : NYT], pzc[DIM2 ? 1 : NYT];
#pragma unroll
  for (int j = 0; j < (DIM2 ? 1 : NYT); j++) {
    const int iy = ty * NYT + j;
    const double yv = (DIM2 || iy >= L.n_slots) ? 0.0 : prm.y[iy];
    cE[j] = 1.0 / fma(mT, cosh(yv), mass);
    pzc[j] = mT * sinh(yv) * cE[j];
  }

  const int64_t t_begin = (L.n_tiles * (int64_t)chunk) / hp.n_chunks;
  const int64_t t_end = (L.n_tiles * (int64_t)(chunk + 1)) / hp.n_chunks;
  const int n_my_tiles = (int)(t_end - t_begin);
  const double *Yg = hp.Y + ((int64_t)ty * L.n_cells_pad) * nst * kPolRecY;
  const double *Pg = hp.P + ((int64_t)tp * L.n_cells_pad) * NPT * kPolRecP;
  const uint32_t stage_bytes = (uint32_t)stage_doubles * 8u;

  exp_table_init();
  if (threadIdx.x == 0) {
    blk_bad = 0;
    for (int s = 0; s < kStages; s++) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  auto issue = [&](int t_local) {
    const int st = t_local % kStages;
    const int64_t cell = (t_begin + t_local) * CT;
    double *dst = stage_base + (size_t)st * stage_doubles;
    mbar_arrive_expect_tx(&full[st], stage_bytes);
    bulk_g2s(dst, Yg + cell * nst * kPolRecY, (uint32_t)y_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles, Pg + cell * NPT * kPolRecP, (uint32_t)p_doubles * 8u, &full[st]);
  };
  if (threadIdx.x == 0)
    for (int t = 0; t < kStages && t < n_my_tiles; t++) issue(t);

  constexpr int NB = DIM2 ? NPT : NYT * NPT;          // bins of the register tile
  double acc[NB][kSdSums];
#pragma unroll
  for (int i = 0; i < NB; i++)
#pragma unroll
    for (int q = 0; q < kSdSums; q++) acc[i][q] = 0.0;
  unsigned bad = 0;                                    // boson evaluations with u.p/T - J theta <= 0

  for (int t = 0; t < n_my_tiles; t++) {
    const int st = t % kStages;
    mbar_wait(&full[st], (uint32_t)((t / kStages) & 1));
    const double *Ys = stage_base + (size_t)st * stage_doubles;
    const double *Ps = Ys + y_doubles;
    for (int c = 0; c < CT; c++) {
      double q[NPT], pd[NPT], pc[NPT], ps[NPT], pb[NPT][4];
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const double2 *pr = reinterpret_cast<const double2 *>(Ps + (c * NPT + k) * kPolRecP);
        const double2 v0 = pr[0], v1 = pr[1];
        q[k] = pT * v0.x; pd[k] = pT * v0.y; pc[k] = pT * v1.x; ps[k] = pT * v1.y;
      }
      if (!DIM2) {                                      // 3+1D: varpi is the cell's, b^mu is hoisted per (cell, phi)
        const double *y0 = Ys + (c * nst) * kPolRecY;
#pragma unroll
        for (int k = 0; k < NPT; k++) sd_b(y0[7], y0[8], y0[9], y0[10], y0[11], pc[k], ps[k], pb[k]);
      }
      auto slot = [&](int j, int jb, double (*accj)[kSdSums]) {
        const double *yr = Ys + (c * nst + j) * kPolRecY;
        const double x0 = mT * yr[0];
        bool any = false;                                            // padding, skipped cells, far tails: nothing to add
#pragma unroll
        for (int k = 0; k < NPT; k++) any |= exp_finite(x0 - q[k]);
        if (!any) return;
        const double cpm = mT * yr[1], w = yr[2];
        const double a0 = mT * yr[3], a1 = mT * yr[4], a2 = mT * yr[5], a3 = mT * yr[6];
#pragma unroll
        for (int k = 0; k < NPT; k++) {
          const double x = x0 - q[k];
          const double pds = fma(w, pd[k], cpm);
          if (exp_finite(x) && __double_as_longlong(pds) > thr) {
            const double a = exp_neg(x);
            const double fbar = rcp_fast(fma(sign, a, 1.0));       // 1 / (1 + Theta e) = 1 - Theta f
            const double t0 = pds * (a * fbar);                      // p.dsigma f
            double b[4];
            if (DIM2) sd_b(yr[7], yr[8], yr[9], yr[10], yr[11], pc[k], ps[k], b);
            else { b[0] = pb[k][0]; b[1] = pb[k][1]; b[2] = pb[k][2]; b[3] = pb[k][3]; }
            const double vt = (a0 + b[0]) * cE[jb];
            const double tx = inv_m * fma(-vt, pc[k], a1 + b[1]);
            const double ty_ = inv_m * fma(-vt, ps[k], a2 + b[2]);
            const double tz = inv_m * fma(-(a0 + b[0]), pzc[jb], a3 + b[3]);
            const double th2 = fma(tx, tx, fma(ty_, ty_, tz * tz));
            const double th = th2 > 0.0 ? sqrt(th2) : 0.0;
            if (sign < 0.0 && x - J * th <= 0.0) { bad++; continue; }
            double sP = 0.0, sE = 0.0, sQ = 0.0;                     // sum_m m S_m / D_m, sum (C_m - 1) / D_m, sum cq_m (C_m - 1) / D_m
            if (n_pairs > 0 && th > 0.0) {
              const double s1 = sinh_pos(0.5 * th), c1 = sqrt(fma(s1, s1, 1.0));
              const double sT = 2.0 * s1 * c1, cT1 = 2.0 * s1 * s1, cT = 1.0 + cT1;     // sinh theta, cosh theta - 1, cosh theta
              double S = half_int ? s1 : sT;                         // sinh m theta, cosh m theta - 1 at the smallest m > 0
              double Cm1 = half_int ? s1 * s1 / (1.0 + c1) : cT1;
              double mm = half_int ? 0.5 : 1.0;
              const double op = fma(sign, a, 1.0), op2 = op * op, tte = 2.0 * sign * a;
              for (int l = 0; l < n_pairs; l++) {
                const double rD = rcp_fast(fma(tte, Cm1, op2));
                sP = fma(mm * S, rD, sP);
                const double e1 = Cm1 * rD;
                sE += e1;
                sQ = fma(0.5 * fma(3.0 * mm, mm, -JJ1), e1, sQ);
                const double Sn = fma(S, cT, fma(Cm1, sT, sT));      // sinh, cosh - 1 of (m + 1) theta: sums of positive terms
                Cm1 = fma(Cm1, cT, fma(S, sT, cT1));
                S = Sn;
                mm += 1.0;
              }
              const double ce = 2.0 * a * (1.0 - sign * a) * fbar;  // 2 e (1 - Theta e) / (1 + Theta e)
              const double ith = 1.0 / th;
              sP *= 2.0 * a * ith;
              sE *= ce;
              sQ *= ce * ith * ith;
            }
            const double wp = pds * sP, wq = pds * sQ, th2_3 = th2 * (1.0 / 3.0);
            double *A = accj[k];
            A[0] = fma(pds, sE * inv_g, A[0] + t0);
            A[1] = fma(wp, tx, A[1]);
            A[2] = fma(wp, ty_, A[2]);
            A[3] = fma(wp, tz, A[3]);
            A[4] = fma(wq, fma(tx, tx, -th2_3), A[4]);
            A[5] = fma(wq, tx * ty_, A[5]);
            A[6] = fma(wq, tx * tz, A[6]);
            A[7] = fma(wq, fma(ty_, ty_, -th2_3), A[7]);
            A[8] = fma(wq, ty_ * tz, A[8]);
          }
        }
      };
      if (DIM2) {
        for (int j = 0; j < nst; j++) slot(j, 0, acc);
      } else {
#pragma unroll
        for (int j = 0; j < NYT; j++) slot(j, j, acc + j * NPT);
      }
    }
    __syncthreads();                                   // every warp is done with stage st
    if (threadIdx.x == 0 && t + kStages < n_my_tiles) issue(t + kStages);
  }

  if (bad) atomicAdd(&blk_bad, (unsigned long long)bad);
  __syncthreads();
  if (threadIdx.x == 0 && blk_bad) atomicAdd(prm.boson_bad, blk_bad);

  // partial[array][chunk][bin], array = Snorm, P_x, P_y, P_z, Q_xx, Q_xy, Q_xz, Q_yy, Q_yz
  if (lane_valid) {
    const double scale = hp.prefactor * g;
    const int64_t n_bins = (int64_t)L.n_species * L.n_pT * L.n_phi * L.n_y_out;
#pragma unroll
    for (int j = 0; j < (DIM2 ? 1 : NYT); j++) {
      const int iy = DIM2 ? 0 : ty * NYT + j;
      if (iy >= (DIM2 ? 1 : L.n_slots)) continue;
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const int iphi = tp * NPT + k;
        if (iphi >= L.n_phi) continue;
        const int64_t bin = (int64_t)ipart + (int64_t)L.n_species * ((int64_t)ipT + (int64_t)L.n_pT * ((int64_t)iphi + (int64_t)L.n_phi * iy));
        const double *a = acc[(DIM2 ? 0 : j * NPT) + k];
#pragma unroll
        for (int q = 0; q < kSdSums; q++)
          hp.partial[((int64_t)q * hp.n_chunks + chunk) * n_bins + bin] = (q == 0 ? scale : hp.prefactor) * a[q];
      }
    }
  }
}

// (slots per tile, phi points per tile, cells per TMA tile): 9 sums per bin, register tile sized for kSdMinBlocks blocks per SM
void spin_density_shape(int dim2, int *nyt, int *npt, int *ct)
{
  if (dim2) { *nyt = 1; *npt = kSdNpt2D; *ct = 1; }
  else { *nyt = kSdNyt3D; *npt = kSdNpt3D; *ct = 8; }
}

template <int NYT, int NPT, bool DIM2>
static cudaError_t launch_spin_density_one(const SpinDensityParams &prm, cudaStream_t st)
{
  const Layout &L = prm.hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const size_t stage_doubles = (size_t)L.ct * nst * kPolRecY + (size_t)L.ct * NPT * kPolRecP;
  const size_t smem = kStages * stage_doubles * 8 + kStages * sizeof(uint64_t);
  auto kern = cf_spin_density_kernel<NYT, NPT, DIM2>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)prm.hp.n_groupblocks * L.n_ytiles * L.n_ptiles * prm.hp.n_chunks;
  if (grid == 0) return cudaSuccess;
  kern<<<(unsigned)grid, prm.hp.n_warps * 32, smem, st>>>(prm);
  return cudaGetLastError();
}

cudaError_t launch_spin_density(const SpinDensityParams &prm, cudaStream_t st)
{
  if (prm.hp.L.dim2) return launch_spin_density_one<1, kSdNpt2D, true>(prm, st);
  return launch_spin_density_one<kSdNyt3D, kSdNpt3D, false>(prm, st);
}

}  // namespace is3d
