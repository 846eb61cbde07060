// cf_polzn_she.cu -- spin Hall (SHE) part of the mean spin vector of the emitted baryons: the term of the gradient of alpha_B = muB/T
// (sm_100a).
//
// Per momentum bin p and species (m, g, Theta = sign, q_B = baryon), over the cells, rapidity slots and weights of cf_polzn.cu (ideal f,
// no muB in f: the term is first order in d alpha_B around the weight of the vorticity term, whose Snorm it shares bit for bit):
//   N_she^mu(p) = g/(2 pi hbar c)^3 sum w p.dsigma f (1 - Theta f) (-1/(8m)) eps^{mu rho sigma tau} p_tau (-2 q_B that_rho d_sigma alpha_B / E)
// with that = (1, 0, 0, 0) the lab time direction and E = p^t, i.e. the thermal-shear term of cf_polzn_xi.cu with xi_{sigma lambda} p^lambda
// replaced by -q_B d_sigma alpha_B.  In Cartesian lab components N_she^t = 0 and N_she = +(q_B hbar c / (4 m E)) (Z x p), Z_j = sum W
// zeta_j, zeta the Cartesian covariant gradient in 1/fm (cart_gradient()), W the weight above.  zeta does not depend on p, so the kernel
// sums Z (3 numbers per bin) and applies q_B, hbar c, 1/(4 m E) and the cross product once per bin, in the epilogue.
//
// prepare_polzn_she_kernel: the cells and slots of prepare_polzn_kernel (same A, Cp, W and phi records, the u.dsigma <= 0 skip), the
//                           Milne -> Cartesian conversion of d alpha_B (cart_gradient()) and the slot record
//     [A, Cp, W, zeta_x, zeta_y, zeta_z, 0, 0, 0, 0, 0, 0]                               (kPolRecY doubles)
// cf_polzn_she_kernel:      the decomposition and register tile of cf_polzn_kernel with 4 sums per bin (Snorm, Z_x, Z_y, Z_z), one
//                           partial row per cell chunk and array (Snorm, N^x, N^y, N^z), summed by launch_reduce in a fixed order.
// Same layout, chunks and per-evaluation Snorm arithmetic as cf_polzn.cu: Snorm is bit-identical to the vorticity path's.
#include "cf_internal.h"
#include "cf_device.cuh"
#include "cf_polzn.cuh"

namespace is3d {

struct CellShe {
  double tau, eta, invT, ut, ux, uy, un, dat, dax, day, dan, d[4];
  int valid;
};

constexpr int kShePrepCells = 16;
constexpr int kShePrepThreads = 128;

__global__ void __launch_bounds__(kShePrepThreads)
prepare_polzn_she_kernel(RawCells cells, GradientCells grad, PrepTables tab, Layout L, double *__restrict__ Y, double *__restrict__ P,
                         PrepCounters *counters)
{
  __shared__ CellShe sc_[kShePrepCells];
  const int64_t cell0 = (int64_t)blockIdx.x * kShePrepCells;
  if (threadIdx.x < kShePrepCells) {
    const int64_t i = cell0 + threadIdx.x;
    CellShe c;
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
        for (int q = 0; q < 4; q++) c.d[q] = grad.d[q][i];
      }
    }
    sc_[threadIdx.x] = c;
  }
  __syncthreads();

  const int slots_pad = L.n_ytiles * L.nst;
  for (int w = threadIdx.x; w < kShePrepCells * slots_pad; w += kShePrepThreads) {
    const int lc = w / slots_pad, j = w - lc * slots_pad;
    const int64_t i = cell0 + lc;
    if (i >= L.n_cells_pad) continue;
    const int ty = j / L.nst, jj = j - ty * L.nst;
    double *r = Y + (((int64_t)ty * L.n_cells_pad + i) * L.nst + jj) * kPolRecY;
    const CellShe &c = sc_[lc];
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
    double z[3];
    cart_gradient(c.d, c.tau, eta, z);
    r[3] = z[0]; r[4] = z[1]; r[5] = z[2];
    for (int q = 6; q < kPolRecY; q++) r[q] = 0.0;
  }

  const int phis_pad = L.n_ptiles * L.npt;
  for (int w = threadIdx.x; w < kShePrepCells * phis_pad; w += kShePrepThreads) {
    const int lc = w / phis_pad, k = w - lc * phis_pad;
    const int64_t i = cell0 + lc;
    if (i >= L.n_cells_pad) continue;
    const int tp = k / L.npt, kk = k - tp * L.npt;
    double *r = P + (((int64_t)tp * L.n_cells_pad + i) * L.npt + kk) * kPolRecP;
    const CellShe &c = sc_[lc];
    if (!c.valid || k >= L.n_phi) { r[0] = 0.0; r[1] = 0.0; r[2] = 0.0; r[3] = 0.0; continue; }
    const double cs = tab.cosphi[k], sn = tab.sinphi[k];
    r[0] = (cs * c.ux + sn * c.uy) * c.invT;
    r[1] = cs * c.dax + sn * c.day;
    r[2] = cs;
    r[3] = sn;
  }
}

cudaError_t launch_prepare_polzn_she(const RawCells &cells, const GradientCells &grad, const PrepTables &tab, const Layout &L, double *Y,
                                     double *P, PrepCounters *counters, cudaStream_t st)
{
  const int64_t nblk = (L.n_cells_pad + kShePrepCells - 1) / kShePrepCells;
  if (nblk == 0) return cudaSuccess;
  prepare_polzn_she_kernel<<<(unsigned)nblk, kShePrepThreads, 0, st>>>(cells, grad, tab, L, Y, P, counters);
  return cudaGetLastError();
}

// Register tile: NYT rapidity slots (3+1D; 2+1D sums every eta slot into one) x NPT phi points x 4 sums (Snorm, Z_x, Z_y, Z_z)
template <int NYT, int NPT, bool DIM2>
__global__ void __launch_bounds__(kPolWarps * 32, DIM2 ? 2 : 3)
cf_polzn_she_kernel(const PolSheParams prm)
{
  extern __shared__ __align__(128) unsigned char smem_raw[];
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
  double acc[NB][4];
#pragma unroll
  for (int i = 0; i < NB; i++)
#pragma unroll
    for (int q = 0; q < 4; q++) acc[i][q] = 0.0;

  for (int t = 0; t < n_my_tiles; t++) {
    const int st = t % kStages;
    mbar_wait(&full[st], (uint32_t)((t / kStages) & 1));
    const double *Ys = stage_base + (size_t)st * stage_doubles;
    const double *Ps = Ys + y_doubles;
    for (int c = 0; c < CT; c++) {
      double q[NPT], pd[NPT];
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const double2 v0 = *reinterpret_cast<const double2 *>(Ps + (c * NPT + k) * kPolRecP);
        q[k] = pT * v0.x; pd[k] = pT * v0.y;
      }
      double z0[3] = {0.0, 0.0, 0.0};
      if (!DIM2) {                                      // 3+1D: zeta is the cell's, the same in every slot record
        const double *y0 = Ys + (c * nst) * kPolRecY;
        z0[0] = y0[3]; z0[1] = y0[4]; z0[2] = y0[5];
      }
      auto slot = [&](int j, double (*accj)[4]) {
        const double *yr = Ys + (c * nst + j) * kPolRecY;
        const double x0 = mT * yr[0];
        bool any = false;                                            // padding, skipped cells, far tails: nothing to add
#pragma unroll
        for (int k = 0; k < NPT; k++) any |= exp_finite(x0 - q[k]);
        if (!any) return;
        const double cpm = mT * yr[1], w = yr[2];
        const double zx = DIM2 ? yr[3] : z0[0], zy = DIM2 ? yr[4] : z0[1], zz = DIM2 ? yr[5] : z0[2];
#pragma unroll
        for (int k = 0; k < NPT; k++) {
          const double x = x0 - q[k];
          const double pds = fma(w, pd[k], cpm);
          if (exp_finite(x) && __double_as_longlong(pds) > thr) {
            const double a = exp_neg(x);
            const double fbar = rcp_fast(fma(sign, a, 1.0));       // 1 - Theta f
            const double t0 = pds * (a * fbar);                      // p.dsigma f
            const double wf = t0 * fbar;                             // p.dsigma f (1 - Theta f)
            accj[k][0] += t0;
            accj[k][1] = fma(wf, zx, accj[k][1]);
            accj[k][2] = fma(wf, zy, accj[k][2]);
            accj[k][3] = fma(wf, zz, accj[k][3]);
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

  // partial[array][chunk][bin], array = Snorm, N^x, N^y, N^z; N = q_B (scale hbar c / (4 m E)) Z x p with the bin's p
  if (lane_valid) {
    const double scale = prm.hp.prefactor * hp.degeneracy[ipart];
    const double qB = prm.baryon[ipart];
    const int64_t n_bins = (int64_t)L.n_species * L.n_pT * L.n_phi * L.n_y_out;
#pragma unroll
    for (int j = 0; j < (DIM2 ? 1 : NYT); j++) {
      const int iy = DIM2 ? 0 : ty * NYT + j;
      if (iy >= (DIM2 ? 1 : L.n_slots)) continue;
      const double yv = DIM2 ? 0.0 : prm.y[iy];
      const double E = mT * cosh(yv), pz = mT * sinh(yv);
      const double s = qB * (scale * kHbarC / (4.0 * mass * E));   // q_B = -1 gives exactly minus the q_B = +1 value
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const int iphi = tp * NPT + k;
        if (iphi >= L.n_phi) continue;
        const double px = pT * prm.cosphi[iphi], py = pT * prm.sinphi[iphi];
        const int64_t bin = (int64_t)ipart + (int64_t)L.n_species * ((int64_t)ipT + (int64_t)L.n_pT * ((int64_t)iphi + (int64_t)L.n_phi * iy));
        const double *a = acc[(DIM2 ? 0 : j * NPT) + k];
        const double out[4] = {scale * a[0], s * (a[2] * pz - a[3] * py), s * (a[3] * px - a[1] * pz), s * (a[1] * py - a[2] * px)};
#pragma unroll
        for (int q = 0; q < 4; q++) hp.partial[((int64_t)q * hp.n_chunks + chunk) * n_bins + bin] = out[q];
      }
    }
  }
}

template <int NYT, int NPT, bool DIM2>
static cudaError_t launch_polzn_she_one(const PolSheParams &prm, cudaStream_t st)
{
  const Layout &L = prm.hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const size_t stage_doubles = (size_t)L.ct * nst * kPolRecY + (size_t)L.ct * NPT * kPolRecP;
  const size_t smem = kStages * stage_doubles * 8 + kStages * sizeof(uint64_t);
  auto kern = cf_polzn_she_kernel<NYT, NPT, DIM2>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)prm.hp.n_groupblocks * L.n_ytiles * L.n_ptiles * prm.hp.n_chunks;
  if (grid == 0) return cudaSuccess;
  kern<<<(unsigned)grid, prm.hp.n_warps * 32, smem, st>>>(prm);
  return cudaGetLastError();
}

// the shapes of polzn_shape(): the layout (and so the chunk split) is the vorticity path's
cudaError_t launch_polzn_she(const PolSheParams &prm, cudaStream_t st)
{
  if (prm.hp.L.dim2) return launch_polzn_she_one<1, kPolNpt2D, true>(prm, st);
  return launch_polzn_she_one<kPolNyt3D, kPolNpt3D, false>(prm, st);
}

}  // namespace is3d
