// cf_hbtq.cu -- Fourier transform of the Cooper-Frye emission function in the out-side-long frame (HBT correlation functions, sm_100a).
//
// Per momentum bin (species, pT, phi, y) and per q point q_k = k dq d (ray d = (d_o, d_s, d_l), k = 0 .. n_q - 1), over the cells and
// rapidity slots of the linear-delta-f spectra, the raw sums
//   Re[d][k] = sum w cos(theta),  Im[d][k] = sum w sin(theta),   theta = k dq (d_o o + d_s s + d_l l) / hbar c
// with the weight w and the LCMS coordinates (o, s, l) of cf_hbt.cu (o already holds -beta_perp t*): the on-shell phase q.x of K = p,
// q^0 = beta_perp q_o.  Re[d][0] = S0 is the spectrum; C = 1 - sign (Re^2 + Im^2) / (g S0^2) is formed by the writers (host_run.cpp)
// and api.hbt_correlation().
//
// cf_hbt_fourier_kernel: the decomposition of cf_hbt_kernel (lanes = (species, pT) pairs, the records of prepare_vh_kernel and
//   prepare_hbt_cells_kernel streamed through the TMA / mbarrier pipeline) with the q grid in the blocks: a block is one
//   (bin tile, ray, q tile of KQ points, cell chunk) and keeps 2 KQ sums per bin of its register tile, so the weight is evaluated once
//   per q tile.  Per evaluation: f_eq (1 + df) by distribution<MODEL>(), w = p.dsigma f, the phase step
//     dtheta = T[phi] + el l - eo beta_perp t*      (eo, es, el = d dq / hbar c;  T = eo (x cos phi + y sin phi) + es s per (cell, phi);
//                                                    beta_perp t* is the only per-lane part)
//   seeds sincos(dtheta) and sincos(k0 dtheta) (k0 = first k of the tile; k0 = 0 seeds with (1, 0) exactly, so Re[d][0] is the same
//   sum for every ray), then KQ steps of the rotation (c, s) <- (c c1 - s s1, s c1 + c s1), 4 FP64 operations, and 2 FMAs into the
//   sums.  The recurrence restarts from sincos every KQ points: its drift is bounded by KQ steps whatever n_q is.
//   One partial row per cell chunk and array, summed by launch_reduce in a fixed order: no atomics, results are bit-reproducible.
#include "cf_internal.h"
#include "cf_device.cuh"

namespace is3d {

// Register tile: NYT rapidity slots (3+1D; 2+1D sums every eta slot into one bin) x NPT phi points x KQ q points x (Re, Im)
template <int MODEL, int NYT, int NPT, int KQ, bool DIM2>
__global__ void __launch_bounds__(kHbtWarps * 32, kHbtqMinBlocks)
cf_hbt_fourier_kernel(const HbtqParams prm)
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

  // block = ((chunk * n_dir + ray) * n_qtiles + q tile) * bin tiles + bin tile: the blocks of a chunk share its records in L2
  const int n_bintiles = hp.n_groupblocks * L.n_ytiles * L.n_ptiles;
  const int per_chunk = n_bintiles * prm.n_dir * prm.n_qtiles;
  const int chunk = blockIdx.x / per_chunk;
  int bt = blockIdx.x - chunk * per_chunk;
  const int tp = bt % L.n_ptiles; bt /= L.n_ptiles;
  const int ty = bt % L.n_ytiles; bt /= L.n_ytiles;
  const int gb = bt % hp.n_groupblocks; bt /= hp.n_groupblocks;
  const int qt = bt % prm.n_qtiles;
  const int ray = bt / prm.n_qtiles;
  const int k0 = qt * KQ;
  const double eo = prm.dir[3 * ray], es = prm.dir[3 * ray + 1], el = prm.dir[3 * ray + 2];
  const double k0d = (double)k0;
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
  double acc[NB][2 * KQ];                             // per bin: Re, Im of q points k0 .. k0 + KQ - 1
#pragma unroll
  for (int i = 0; i < NB; i++)
#pragma unroll
    for (int m = 0; m < 2 * KQ; m++) acc[i][m] = 0.0;

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
      // phi hoists, reused by every slot: u.p, p.dsigma and delta-f pieces as in cf_kernel, the transverse part of the phase step
      double q[NPT], pd[NPT], g0[NPT], g1[NPT], g2[NPT], T[NPT];
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const double2 *pr = reinterpret_cast<const double2 *>(Ps + (c * NPT + k) * kRec);
        const double2 v0 = pr[0], v1 = pr[1], v2 = pr[2];
        q[k] = pT * v0.x;
        pd[k] = pT * v0.y;
        g0[k] = fma(pT2, v1.x, K0m);
        g1[k] = pT * v1.y;
        g2[k] = pT * v2.x;
        const double X = fma(xc, cs[k], yc * sn[k]), sd = fma(-xc, sn[k], yc * cs[k]);
        T[k] = fma(eo, X, es * sd);
      }
      auto slot = [&](int j, double (*accj)[2 * KQ]) {
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
        const double Ls = -el * v2.x;                                // el z*
#pragma unroll
        for (int k = 0; k < NPT; k++) {
          const double x = a - q[k];
          const double pds = fma(w, pd[k], cpm);
          if (exp_finite(x) && __double_as_longlong(pds) > thr) {
            double s = h0 + g0[k];
            s = fma(g2[k], h2, s);
            s = fma(-g1[k], h1, s);
            const double wt = pds * distribution<MODEL>(x, s, K2, 0.0, sign, reg_thr, one_hi);
            const double dth = fma(-eo, bts, T[k] + Ls);
            double s1, c1, sk, ck;
            sincos(dth, &s1, &c1);
            if (k0 == 0) { ck = 1.0; sk = 0.0; }
            else sincos(k0d * dth, &sk, &ck);
            double *r = accj[k];
#pragma unroll
            for (int m = 0; m < KQ; m++) {
              r[2 * m] = fma(wt, ck, r[2 * m]);
              r[2 * m + 1] = fma(wt, sk, r[2 * m + 1]);
              const double cn = fma(ck, c1, -sk * s1);
              sk = fma(sk, c1, ck * s1);
              ck = cn;
            }
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

  // partial[array][chunk][bin], arrays Re (ray, k) then Im (ray, k)
  if (lane_valid) {
    const double scale = hp.prefactor * hp.degeneracy[ipart];
    const int64_t n_bins = (int64_t)L.n_species * L.n_pT * L.n_phi * L.n_y_out;
    const int64_t re_row = (int64_t)ray * prm.n_q, im_row = (int64_t)(prm.n_dir + ray) * prm.n_q;
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
        for (int m = 0; m < KQ; m++) {
          const int kq = k0 + m;
          if (kq >= prm.n_q) break;
          hp.partial[((re_row + kq) * hp.n_chunks + chunk) * n_bins + bin] = scale * a[2 * m];
          hp.partial[((im_row + kq) * hp.n_chunks + chunk) * n_bins + bin] = scale * a[2 * m + 1];
        }
      }
    }
  }
}

// (slots per tile, phi points per tile, cells per TMA tile) of the two instantiations; blocks are kHbtWarps warps or fewer
void hbtq_shape(int dim2, int *nyt, int *npt, int *ct)
{
  if (dim2) { *nyt = 1; *npt = kHbtqNpt2D; *ct = 1; }
  else { *nyt = kHbtqNyt3D; *npt = kHbtqNpt3D; *ct = 8; }
}

template <int MODEL, int NYT, int NPT, bool DIM2>
static cudaError_t launch_hbtq_one(const HbtqParams &prm, cudaStream_t st)
{
  const Layout &L = prm.hp.L;
  const int nst = DIM2 ? L.nst : NYT;
  const size_t stage_doubles = (size_t)L.ct * (nst * kRec + NPT * kRec + kScal + kHbtRecC);
  const size_t smem = kStages * stage_doubles * 8 + kStages * sizeof(uint64_t);
  auto kern = cf_hbt_fourier_kernel<MODEL, NYT, NPT, kHbtqKQ, DIM2>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t grid = (int64_t)prm.hp.n_groupblocks * L.n_ytiles * L.n_ptiles * prm.n_dir * prm.n_qtiles * prm.hp.n_chunks;
  if (grid == 0) return cudaSuccess;
  kern<<<(unsigned)grid, prm.hp.n_warps * 32, smem, st>>>(prm);
  return cudaGetLastError();
}

template <int MODEL>
static cudaError_t launch_hbtq_model(const HbtqParams &prm, cudaStream_t st)
{
  if (prm.hp.L.dim2) return launch_hbtq_one<MODEL, 1, kHbtqNpt2D, true>(prm, st);
  return launch_hbtq_one<MODEL, kHbtqNyt3D, kHbtqNpt3D, false>(prm, st);
}

cudaError_t launch_hbt_fourier(int model, const HbtqParams &prm, cudaStream_t st)
{
  switch (model) {
    case M_LIN14: return launch_hbtq_model<M_LIN14>(prm, st);
    case M_LINCE: return launch_hbtq_model<M_LINCE>(prm, st);
    case M_IDEAL: return launch_hbtq_model<M_IDEAL>(prm, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace is3d
