// cf_hbt.cu -- space-time moments of the Cooper-Frye emission function in the out-side-long frame (HBT radii, sm_100a).
//
// Per momentum bin (species, pT, phi, y) and over the cells and rapidity slots of the linear-delta-f spectra, ten raw sums
//   S0 = sum w,  S_i = sum w x_i,  S_ij = sum w x_i x_j   (x = (o, s, l), i <= j)
// with w = g/(2 pi hbar c)^3 (slot weight) p.dsigma f_eq (1 + df), the summand of the spectra, and the LCMS coordinates
//   t* = tau cosh(eta - y) = tau U1,   z* = tau sinh(eta - y) = -U2     (U1 = ch, U2 = tsh of the cf_prepare.cu slot records)
//   o  = x cos phi + y sin phi - beta_perp t*,   s = -x sin phi + y cos phi,   l = z*,   beta_perp = pT / mT.
// The radii R^2_ij = S_ij / S0 - S_i S_j / S0^2 are formed by the writers (host_run.cpp) and api.hbt_radii().
//
// prepare_hbt_cells_kernel: per-cell record [tau, x, y, 0] (kHbtRecC doubles, 16-byte aligned) beside the records of
//                           prepare_vh_kernel (cf_prepare.cu), which this path uses unchanged: slot [A, Cp, Qyy, ch, tsh, W],
//                           phi [Bx, Dp, Qpp, R1, R2, 0], scalars [K0, K2, 0, 0] -- so the delta-f arithmetic and the skip rules
//                           (u.dsigma <= 0, padding) are literally those of the spectra.
// cf_hbt_kernel:            the decomposition of cf_kernel (cf_kernels.cu): lanes = (species, pT) pairs, cell tiles streamed through
//                           the TMA / mbarrier pipeline, a register tile of NYT x NPT bins x 10 sums, one partial row per cell chunk
//                           and array, summed by launch_reduce in a fixed order: no atomics, results are bit-reproducible.
//   Per evaluation: f_eq (1 + df) by distribution<MODEL>() (cf_device.cuh, the per-evaluation function of cf_kernel), then
//   w = p.dsigma f, o = X[phi] - beta t*[slot] and the ten accumulations (3 DMUL, 1 DADD, 10 DADD / DFMA).
#include "cf_internal.h"
#include "cf_device.cuh"

namespace is3d {

constexpr int kHbtPrepThreads = 256;

__global__ void __launch_bounds__(kHbtPrepThreads)
prepare_hbt_cells_kernel(const double *__restrict__ tau, const double *__restrict__ x, const double *__restrict__ y, int64_t n,
                         int64_t n_pad, double *__restrict__ C)
{
  const int64_t i = (int64_t)blockIdx.x * kHbtPrepThreads + threadIdx.x;
  if (i >= n_pad) return;
  double2 *r = reinterpret_cast<double2 *>(C + i * kHbtRecC);
  r[0] = i < n ? make_double2(tau[i], x[i]) : make_double2(0.0, 0.0);
  r[1] = make_double2(i < n ? y[i] : 0.0, 0.0);
}

cudaError_t launch_prepare_hbt_cells(const double *tau, const double *x, const double *y, int64_t n, int64_t n_pad, double *C, cudaStream_t st)
{
  const int64_t nblk = (n_pad + kHbtPrepThreads - 1) / kHbtPrepThreads;
  if (nblk == 0) return cudaSuccess;
  prepare_hbt_cells_kernel<<<(unsigned)nblk, kHbtPrepThreads, 0, st>>>(tau, x, y, n, n_pad, C);
  return cudaGetLastError();
}

// Register tile: NYT rapidity slots (3+1D; 2+1D sums every eta slot into one bin) x NPT phi points x 10 sums
template <int MODEL, int NYT, int NPT, bool DIM2>
__global__ void __launch_bounds__(kHbtWarps * 32, kHbtMinBlocks)
cf_hbt_kernel(const HbtParams prm)
{
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const HotParams &hp = prm.hp;
  const Layout &L = hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const int CT = L.ct;
  const int y_doubles = CT * nst * kRec, p_doubles = CT * NPT * kRec, s_doubles = CT * kScal, c_doubles = CT * kHbtRecC;
  const int stage_doubles = y_doubles + p_doubles + s_doubles + c_doubles;
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
  const double m2 = mass * mass, pT2 = pT * pT, mT2 = m2 + pT2;
  const double mT = sqrt(mT2);
  const double beta = pT / mT;                                  // beta_perp of the LCMS
  const int reg_thr = hp.regulate_thr, one_hi = hp.one_hi;
  const long long thr = hp.outflow_thr;
  double cs[NPT], sn[NPT];                                      // cos, sin of this block's phi points (padding: the last one)
#pragma unroll
  for (int k = 0; k < NPT; k++) {
    const int iphi = min(tp * NPT + k, L.n_phi - 1);
    cs[k] = prm.cosphi[iphi]; sn[k] = prm.sinphi[iphi];
  }

  const int64_t t_begin = (L.n_tiles * (int64_t)chunk) / hp.n_chunks;
  const int64_t t_end = (L.n_tiles * (int64_t)(chunk + 1)) / hp.n_chunks;
  const int n_my_tiles = (int)(t_end - t_begin);
  const double *Yg = hp.Y + ((int64_t)ty * L.n_cells_pad) * nst * kRec;
  const double *Pg = hp.P + ((int64_t)tp * L.n_cells_pad) * NPT * kRec;
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
    bulk_g2s(dst, Yg + cell * nst * kRec, (uint32_t)y_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles, Pg + cell * NPT * kRec, (uint32_t)p_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles + p_doubles, hp.S + cell * kScal, (uint32_t)s_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles + p_doubles + s_doubles, prm.C + cell * kHbtRecC, (uint32_t)c_doubles * 8u, &full[st]);
  };
  if (threadIdx.x == 0)
    for (int t = 0; t < kStages && t < n_my_tiles; t++) issue(t);

  constexpr int NB = DIM2 ? NPT : NYT * NPT;          // bins of the register tile
  double acc[NB][kHbtSums];
#pragma unroll
  for (int i = 0; i < NB; i++)
#pragma unroll
    for (int q = 0; q < kHbtSums; q++) acc[i][q] = 0.0;

  for (int t = 0; t < n_my_tiles; t++) {
    const int st = t % kStages;
    mbar_wait(&full[st], (uint32_t)((t / kStages) & 1));
    const double *Ys = stage_base + (size_t)st * stage_doubles;
    const double *Ps = Ys + y_doubles;
    const double *Ss = Ps + p_doubles;
    const double *Cs = Ss + s_doubles;
    for (int c = 0; c < CT; c++) {
      const double2 k01 = *reinterpret_cast<const double2 *>(Ss + c * kScal);
      const double K0m = k01.x * m2, K2 = k01.y;
      const double2 c01 = *reinterpret_cast<const double2 *>(Cs + c * kHbtRecC);
      const double xc = c01.y, yc = Cs[c * kHbtRecC + 2];
      const double btau = beta * c01.x;
      // phi hoists, reused by every slot: u.p, p.dsigma and delta-f pieces as in cf_kernel, the transverse out / side positions
      double q[NPT], pd[NPT], g0[NPT], g1[NPT], g2[NPT], X[NPT], sd[NPT];
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const double2 *pr = reinterpret_cast<const double2 *>(Ps + (c * NPT + k) * kRec);
        const double2 v0 = pr[0], v1 = pr[1], v2 = pr[2];
        q[k] = pT * v0.x;
        pd[k] = pT * v0.y;
        g0[k] = fma(pT2, v1.x, K0m);
        g1[k] = pT * v1.y;
        g2[k] = pT * v2.x;
        X[k] = fma(xc, cs[k], yc * sn[k]);
        sd[k] = fma(-xc, sn[k], yc * cs[k]);
      }
      auto slot = [&](int j, double (*accj)[kHbtSums]) {
        const double2 *yr = reinterpret_cast<const double2 *>(Ys + (c * nst + j) * kRec);
        const double2 v0 = yr[0];
        const double a = mT * v0.x;
        bool any = false;                                            // padding, skipped cells, far tails: nothing to add
#pragma unroll
        for (int k = 0; k < NPT; k++) any |= exp_finite(a - q[k]);
        if (!any) return;
        const double2 v1 = yr[1], v2 = yr[2];
        const double cpm = mT * v0.y, h0 = mT2 * v1.x, h1 = mT * v1.y, h2 = mT * v2.x, w = v2.y;
        const double bts = btau * v1.y;                              // beta_perp t*
        const double l = -v2.x;                                      // z*
#pragma unroll
        for (int k = 0; k < NPT; k++) {
          const double x = a - q[k];
          const double pds = fma(w, pd[k], cpm);
          if (exp_finite(x) && __double_as_longlong(pds) > thr) {
            double s = h0 + g0[k];
            s = fma(g2[k], h2, s);
            s = fma(-g1[k], h1, s);
            const double wt = pds * distribution<MODEL>(x, s, K2, 0.0, sign, reg_thr, one_hi);
            const double o = X[k] - bts;
            const double wo = wt * o, ws = wt * sd[k], wl = wt * l;
            double *r = accj[k];
            r[0] += wt;
            r[1] += wo;
            r[2] += ws;
            r[3] += wl;
            r[4] = fma(wo, o, r[4]);
            r[5] = fma(ws, sd[k], r[5]);
            r[6] = fma(wl, l, r[6]);
            r[7] = fma(wo, sd[k], r[7]);
            r[8] = fma(wo, l, r[8]);
            r[9] = fma(ws, l, r[9]);
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

  // partial[array][chunk][bin], arrays in the order of is3d_hbt_result
  if (lane_valid) {
    const double scale = hp.prefactor * hp.degeneracy[ipart];
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
        for (int q = 0; q < kHbtSums; q++) hp.partial[((int64_t)q * hp.n_chunks + chunk) * n_bins + bin] = scale * a[q];
      }
    }
  }
}

// (slots per tile, phi points per tile, cells per TMA tile) of the two instantiations; blocks are kHbtWarps warps or fewer
void hbt_shape(int dim2, int *nyt, int *npt, int *ct)
{
  if (dim2) { *nyt = 1; *npt = kHbtNpt2D; *ct = 1; }
  else { *nyt = kHbtNyt3D; *npt = kHbtNpt3D; *ct = 8; }
}

template <int MODEL, int NYT, int NPT, bool DIM2>
static cudaError_t launch_hbt_one(const HbtParams &prm, cudaStream_t st)
{
  const Layout &L = prm.hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const size_t stage_doubles = (size_t)L.ct * (nst * kRec + NPT * kRec + kScal + kHbtRecC);
  const size_t smem = kStages * stage_doubles * 8 + kStages * sizeof(uint64_t);
  auto kern = cf_hbt_kernel<MODEL, NYT, NPT, DIM2>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)prm.hp.n_groupblocks * L.n_ytiles * L.n_ptiles * prm.hp.n_chunks;
  if (grid == 0) return cudaSuccess;
  kern<<<(unsigned)grid, prm.hp.n_warps * 32, smem, st>>>(prm);
  return cudaGetLastError();
}

template <int MODEL>
static cudaError_t launch_hbt_model(const HbtParams &prm, cudaStream_t st)
{
  if (prm.hp.L.dim2) return launch_hbt_one<MODEL, 1, kHbtNpt2D, true>(prm, st);
  return launch_hbt_one<MODEL, kHbtNyt3D, kHbtNpt3D, false>(prm, st);
}

cudaError_t launch_hbt(int model, const HbtParams &prm, cudaStream_t st)
{
  switch (model) {
    case M_LIN14: return launch_hbt_model<M_LIN14>(prm, st);
    case M_LINCE: return launch_hbt_model<M_LINCE>(prm, st);
    case M_IDEAL: return launch_hbt_model<M_IDEAL>(prm, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace is3d
