// cf_polzn.cu -- mean spin (polarization) vector of the emitted hadrons from a thermal-vorticity (mode 5) surface (sm_100a).
//
// Per momentum bin p and species (m, g, Theta = sign), over the cells and rapidity slots of the ideal-f spectra:
//   Snorm(p) = g/(2 pi hbar c)^3 sum w p.dsigma f                          f = 1 / (exp(p.u/T) + Theta)
//   N^mu(p)  = g/(2 pi hbar c)^3 sum w p.dsigma f (1 - Theta f) (-1/(8m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau
// in Cartesian lab components, eps^{txyz} = +1 (Becattini et al. 2013).  With e_i = varpi_{ti} and omega_i = (1/2) eps_{ijk} varpi_{jk}
// the contraction is (1/(4m)) (omega.p, E omega - e x p): linear in p = (mT cosh y, pT cos phi, pT sin phi, mT sinh y), so it splits
// into mT a^mu[cell, slot] + pT b^mu[cell, phi] (3+1D; in 2+1D the Cartesian varpi depends on the slot's eta, b is formed per slot).
//
// prepare_polzn_kernel: per-cell set-up, the u.dsigma <= 0 skip, the Milne -> Cartesian conversion of varpi (cart_vorticity(), the
//                       one place that fixes the input convention) and the records
//     slot record [A, Cp, W, a^t, a^x, a^y, a^z, e_x, e_y, e_z, omega_x, omega_y]     (kPolRecY doubles)
//     phi  record [Bx, Dp, cos phi, sin phi]                                             (kPolRecP doubles)
//   with u.p / T = mT A - pT Bx and p.dsigma = mT Cp + W pT Dp as in cf_prepare.cu.
// cf_polzn_kernel:      the decomposition of cf_kernel (cf_kernels.cu): lanes = (species, pT) pairs, cell tiles streamed through a
//                       TMA / mbarrier pipeline, a register tile of NYT x NPT bins x 5 sums, one partial row per cell chunk and array.
//                       The chunks are summed by launch_reduce in a fixed order: no atomics, results are bit-reproducible.
#include "cf_internal.h"
#include "cf_device.cuh"

namespace is3d {

// Covariant Milne components (varpi_{tau x}, varpi_{tau y}, varpi_{tau eta}, varpi_{xy}, varpi_{x eta}, varpi_{y eta}) at space-time
// rapidity eta -> e = (varpi_tx, varpi_ty, varpi_tz) and omega = (varpi_yz, varpi_zx, varpi_xy), Cartesian lab components:
//   varpi_tx = ch varpi_taux + (sh/tau) varpi_xeta    varpi_zx = -sh varpi_taux - (ch/tau) varpi_xeta    varpi_tz = varpi_taueta / tau
// This is the single place to change if a surface writer uses another convention.
__device__ __forceinline__ void cart_vorticity(const double w[6], double tau, double eta, double e[3], double om[3])
{
  const double ch = cosh(eta), sh = sinh(eta), inv_tau = 1.0 / tau;
  e[0] = ch * w[0] + sh * inv_tau * w[4];
  e[1] = ch * w[1] + sh * inv_tau * w[5];
  e[2] = w[2] * inv_tau;
  const double wzx = -sh * w[0] - ch * inv_tau * w[4];
  const double wzy = -sh * w[1] - ch * inv_tau * w[5];
  om[0] = -wzy;              // varpi_yz
  om[1] = wzx;               // varpi_zx
  om[2] = w[3];              // varpi_xy
}

struct CellPol {
  double tau, eta, invT, ut, ux, uy, un, dat, dax, day, dan, w[6];
  int valid;
};

constexpr int kPolPrepCells = 16;
constexpr int kPolPrepThreads = 128;

__global__ void __launch_bounds__(kPolPrepThreads)
prepare_polzn_kernel(RawCells cells, VortCells vort, PrepTables tab, Layout L, double *__restrict__ Y, double *__restrict__ P,
                     PrepCounters *counters)
{
  __shared__ CellPol sc_[kPolPrepCells];
  const int64_t cell0 = (int64_t)blockIdx.x * kPolPrepCells;
  if (threadIdx.x < kPolPrepCells) {
    const int64_t i = cell0 + threadIdx.x;
    CellPol c;
    c.valid = 0;
    if (i < cells.n) {
      const double tau = cells.tau[i];
      const double ux = cells.ux[i], uy = cells.uy[i], un = cells.un[i];
      const double ut = sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un);
      const double dat = cells.dat[i], dax = cells.dax[i], day = cells.day[i], dan = cells.dan[i];
      if (ut * dat + ux * dax + uy * day + un * dan <= 0.0) {
        atomicAdd(&counters->skipped, 1ULL);
      } else {
        c.valid = 1;
        c.tau = tau; c.eta = cells.eta[i]; c.invT = 1.0 / cells.T[i];
        c.ut = ut; c.ux = ux; c.uy = uy; c.un = un; c.dat = dat; c.dax = dax; c.day = day; c.dan = dan;
        c.w[0] = vort.wtx[i]; c.w[1] = vort.wty[i]; c.w[2] = vort.wtn[i]; c.w[3] = vort.wxy[i]; c.w[4] = vort.wxn[i]; c.w[5] = vort.wyn[i];
      }
    }
    sc_[threadIdx.x] = c;
  }
  __syncthreads();

  const int slots_pad = L.n_ytiles * L.nst;
  for (int w = threadIdx.x; w < kPolPrepCells * slots_pad; w += kPolPrepThreads) {
    const int lc = w / slots_pad, j = w - lc * slots_pad;
    const int64_t i = cell0 + lc;
    if (i >= L.n_cells_pad) continue;
    const int ty = j / L.nst, jj = j - ty * L.nst;
    double *r = Y + (((int64_t)ty * L.n_cells_pad + i) * L.nst + jj) * kPolRecY;
    const CellPol &c = sc_[lc];
    if (!c.valid || j >= L.n_slots) {
      r[0] = kDeadSlotA;
      for (int q = 1; q < kPolRecY; q++) r[q] = 0.0;
      continue;
    }
    double yv, eta, wgt;
    if (L.dim2) { yv = 0.0; eta = tab.slot_y[j]; wgt = tab.slot_w[j]; }
    else        { yv = tab.slot_y[j]; eta = c.eta; wgt = 1.0; }
    const double ch = cosh(yv - eta), sh = sinh(yv - eta);
    r[0] = (ch * c.ut - c.tau * sh * c.un) * c.invT;
    r[1] = wgt * (ch * c.dat + (sh / c.tau) * c.dan);
    r[2] = wgt;
    double e[3], om[3];
    cart_vorticity(c.w, c.tau, eta, e, om);
    const double cy = cosh(yv), sy = sinh(yv);
    r[3] = om[2] * sy;                  // (omega.p)        mT part
    r[4] = cy * om[0] - sy * e[1];      // (E omega - e x p) mT part
    r[5] = cy * om[1] + sy * e[0];
    r[6] = cy * om[2];
    r[7] = e[0]; r[8] = e[1]; r[9] = e[2]; r[10] = om[0]; r[11] = om[1];
  }

  const int phis_pad = L.n_ptiles * L.npt;
  for (int w = threadIdx.x; w < kPolPrepCells * phis_pad; w += kPolPrepThreads) {
    const int lc = w / phis_pad, k = w - lc * phis_pad;
    const int64_t i = cell0 + lc;
    if (i >= L.n_cells_pad) continue;
    const int tp = k / L.npt, kk = k - tp * L.npt;
    double *r = P + (((int64_t)tp * L.n_cells_pad + i) * L.npt + kk) * kPolRecP;
    const CellPol &c = sc_[lc];
    if (!c.valid || k >= L.n_phi) { r[0] = 0.0; r[1] = 0.0; r[2] = 0.0; r[3] = 0.0; continue; }
    const double cs = tab.cosphi[k], sn = tab.sinphi[k];
    r[0] = (cs * c.ux + sn * c.uy) * c.invT;
    r[1] = cs * c.dax + sn * c.day;
    r[2] = cs;
    r[3] = sn;
  }
}

cudaError_t launch_prepare_polzn(const RawCells &cells, const VortCells &vort, const PrepTables &tab, const Layout &L, double *Y, double *P,
                                 PrepCounters *counters, cudaStream_t st)
{
  const int64_t nblk = (L.n_cells_pad + kPolPrepCells - 1) / kPolPrepCells;
  if (nblk == 0) return cudaSuccess;
  prepare_polzn_kernel<<<(unsigned)nblk, kPolPrepThreads, 0, st>>>(cells, vort, tab, L, Y, P, counters);
  return cudaGetLastError();
}

// pT b^mu for (omega.p, E omega - e x p) at phi = (pc, ps) / pT: 6 FP64 operations
__device__ __forceinline__ void pol_b(double ex, double ey, double ez, double ox, double oy, double pc, double ps, double b[4])
{
  b[0] = fma(ox, pc, oy * ps);
  b[1] = ez * ps;
  b[2] = -ez * pc;
  b[3] = fma(ey, pc, -ex * ps);
}

// Register tile: NYT rapidity slots (3+1D; 2+1D sums every eta slot into one) x NPT phi points x 5 sums (Snorm, N^t, N^x, N^y, N^z)
template <int NYT, int NPT, bool DIM2>
__global__ void __launch_bounds__(kPolWarps * 32, DIM2 ? 2 : 3)
cf_polzn_kernel(const HotParams hp)
{
  extern __shared__ __align__(128) unsigned char smem_raw[];
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

  const int64_t t_begin = (L.n_tiles * (int64_t)chunk) / hp.n_chunks;
  const int64_t t_end = (L.n_tiles * (int64_t)(chunk + 1)) / hp.n_chunks;
  const int n_my_tiles = (int)(t_end - t_begin);
  const double *Yg = hp.Y + ((int64_t)ty * L.n_cells_pad) * nst * kPolRecY;
  const double *Pg = hp.P + ((int64_t)tp * L.n_cells_pad) * NPT * kPolRecP;
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
    bulk_g2s(dst, Yg + cell * nst * kPolRecY, (uint32_t)y_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles, Pg + cell * NPT * kPolRecP, (uint32_t)p_doubles * 8u, &full[st]);
  };
  if (threadIdx.x == 0)
    for (int t = 0; t < kStages && t < n_my_tiles; t++) issue(t);

  constexpr int NB = DIM2 ? NPT : NYT * NPT;          // bins of the register tile
  double acc[NB][5];
#pragma unroll
  for (int i = 0; i < NB; i++)
#pragma unroll
    for (int q = 0; q < 5; q++) acc[i][q] = 0.0;

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
        for (int k = 0; k < NPT; k++) pol_b(y0[7], y0[8], y0[9], y0[10], y0[11], pc[k], ps[k], pb[k]);
      }
      auto slot = [&](int j, double (*accj)[5]) {
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
            const double fbar = rcp_fast(fma(sign, a, 1.0));       // 1 - Theta f
            const double t0 = pds * (a * fbar);                      // p.dsigma f
            const double wf = t0 * fbar;                             // p.dsigma f (1 - Theta f)
            double b[4];
            if (DIM2) pol_b(yr[7], yr[8], yr[9], yr[10], yr[11], pc[k], ps[k], b);
            else { b[0] = pb[k][0]; b[1] = pb[k][1]; b[2] = pb[k][2]; b[3] = pb[k][3]; }
            accj[k][0] += t0;
            accj[k][1] = fma(wf, a0 + b[0], accj[k][1]);
            accj[k][2] = fma(wf, a1 + b[1], accj[k][2]);
            accj[k][3] = fma(wf, a2 + b[2], accj[k][3]);
            accj[k][4] = fma(wf, a3 + b[3], accj[k][4]);
          }
        }
      };
      if (DIM2) {
        for (int j = 0; j < nst; j++) slot(j, acc);
      } else {
#pragma unroll
        for (int j = 0; j < NYT; j++) slot(j, acc + j * NPT);
      }
    }
    __syncthreads();                                   // every warp is done with stage st
    if (threadIdx.x == 0 && t + kStages < n_my_tiles) issue(t + kStages);
  }

  // partial[array][chunk][bin], array = Snorm, N^t, N^x, N^y, N^z (the order of is3d_polarization_result after the spin part)
  if (lane_valid) {
    const double scale = hp.prefactor * hp.degeneracy[ipart];
    const double scale_n = scale / (4.0 * mass);
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
        for (int q = 0; q < 5; q++)
          hp.partial[((int64_t)q * hp.n_chunks + chunk) * n_bins + bin] = (q == 0 ? scale : scale_n) * a[q];
      }
    }
  }
}

// (slots per tile, phi points per tile, cells per TMA tile) of the two instantiations; blocks are kPolWarps warps or fewer
void polzn_shape(int dim2, int *nyt, int *npt, int *ct)
{
  if (dim2) { *nyt = 1; *npt = kPolNpt2D; *ct = 1; }
  else { *nyt = kPolNyt3D; *npt = kPolNpt3D; *ct = 8; }
}

template <int NYT, int NPT, bool DIM2>
static cudaError_t launch_polzn_one(const HotParams &hp, cudaStream_t st)
{
  const Layout &L = hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const size_t stage_doubles = (size_t)L.ct * nst * kPolRecY + (size_t)L.ct * NPT * kPolRecP;
  const size_t smem = kStages * stage_doubles * 8 + kStages * sizeof(uint64_t);
  auto kern = cf_polzn_kernel<NYT, NPT, DIM2>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)hp.n_groupblocks * L.n_ytiles * L.n_ptiles * hp.n_chunks;
  if (grid == 0) return cudaSuccess;
  kern<<<(unsigned)grid, hp.n_warps * 32, smem, st>>>(hp);
  return cudaGetLastError();
}

cudaError_t launch_polzn(const HotParams &hp, cudaStream_t st)
{
  if (hp.L.dim2) return launch_polzn_one<1, kPolNpt2D, true>(hp, st);
  return launch_polzn_one<kPolNyt3D, kPolNpt3D, false>(hp, st);
}

}  // namespace is3d
