// host_run.cpp -- the drop-in driver behind the iS3D file interface: is3d_b200_run_workdir().
//
// Call order follows IS3D::run_particlization(1) for operation = 1 (reference src/cpp/iS3D.cpp:73-191):
// parameters -> surface (+ averages side file) -> particle list -> delta-f tables (+ Jonah tables) -> chosen species ->
// momentum tables -> spectra (GPU, through the C ABI) -> result files.  Species bookkeeping mirrors the
// EmissionFunctionArray constructor (emissionfunction.cpp:310-369, 1293-1307); the writers reproduce the text formats of
// write_dN_pTdpTdphidy_toFile (:381-450), write_continuous_vn_toFile (:1053-1136) and write_dN_dy_toFile (:729-772),
// including append mode and the requirement that results/ already exists.
#include "../../include/is3d_b200.h"
#include "host_io.h"
#include "host_math.h"
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <string>
#include <vector>

namespace is3d {

static std::string g_host_error;

struct Grids {
  BlockTable pT, phi, y, eta;
};

static inline long long bin_index(int ipart, int npart, int ipT, int npT, int iphi, int nphi, int iy)
{ return (long long)ipart + (long long)npart * ((long long)ipT + (long long)npT * ((long long)iphi + (long long)nphi * (long long)iy)); }

static bool write_spectra_files(const std::string &wd, const std::vector<double> &dN, const std::vector<int> &mcid,
                                const Grids &g, int dimension, std::string *err)
{
  const int npart = (int)mcid.size(), npT = (int)g.pT.rows, nphi = (int)g.phi.rows;
  const int y_pts = (dimension == 2) ? 1 : (int)g.y.rows;
  auto rapidity = [&](int iy) { return (dimension == 2) ? 0.0 : g.y.at(1, iy + 1); };
  // one block per (species, y, phi): rows "y \t phi \t pT \t dN", blank line after each phi block
  auto dump = [&](std::ostream &os, int ipart) {
    for (int iy = 0; iy < y_pts; iy++)
      for (int iphi = 0; iphi < nphi; iphi++) {
        for (int ipT = 0; ipT < npT; ipT++)
          os << std::scientific << std::setw(5) << std::setprecision(8) << rapidity(iy) << "\t" << g.phi.at(1, iphi + 1) << "\t"
             << g.pT.at(1, ipT + 1) << "\t" << dN[(size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy)] << "\n";
        os << "\n";
      }
  };
  {
    std::ofstream all((wd + "/results/dN_pTdpTdphidy.dat").c_str(), std::ios_base::app);
    if (!all) { *err = "cannot open results/dN_pTdpTdphidy.dat (does results/ exist?)"; return false; }
    for (int ipart = 0; ipart < npart; ipart++) dump(all, ipart);
  }
  for (int ipart = 0; ipart < npart; ipart++) {
    char name[255];
    std::snprintf(name, sizeof(name), "%s/results/dN_pTdpTdphidy_%d.dat", wd.c_str(), mcid[ipart]);
    std::ofstream one(name, std::ios_base::app);
    if (!one) { *err = std::string("cannot open ") + name; return false; }
    one << "y" << "\t" << "phip" << "\t" << "pT" << "\t" << "dN_pTdpTdphidy" << "\n";
    dump(one, ipart);
  }

  // continuous v_n(pT, y), n = 1..7: |sum_phi w e^{i n phi} dN| / sum_phi w dN
  const int k_max = 7;
  for (int ipart = 0; ipart < npart; ipart++) {
    char name[255];
    std::snprintf(name, sizeof(name), "%s/results/vn_continuous/vn_%d.dat", wd.c_str(), mcid[ipart]);
    std::ofstream vf(name, std::ios_base::app);
    if (!vf) { *err = std::string("cannot open ") + name; return false; }
    for (int iy = 0; iy < y_pts; iy++) {
      const double y = (dimension == 2) ? 0.0 : g.y.at(1, iy + 1);
      for (int ipT = 0; ipT < npT; ipT++) {
        double re[k_max], im[k_max], den = 0.0;
        for (int k = 0; k < k_max; k++) { re[k] = 0.0; im[k] = 0.0; }
        for (int iphi = 0; iphi < nphi; iphi++) {
          const double phip = g.phi.at(1, iphi + 1), w = g.phi.at(2, iphi + 1);
          const double v = dN[(size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy)];
          for (int k = 0; k < k_max; k++) {
            re[k] += std::cos(((double)k + 1.0) * phip) * w * v;
            im[k] += std::sin(((double)k + 1.0) * phip) * w * v;
          }
          den += w * v;
        }
        vf << std::scientific << std::setw(5) << std::setprecision(8) << y << "\t" << g.pT.at(1, ipT + 1);
        for (int k = 0; k < k_max; k++) {
          double vn = std::abs(std::complex<double>(re[k], im[k])) / den;
          if (den < 1.e-15) vn = 0.0;
          vf << "\t" << vn;
        }
        vf << "\n";
      }
      vf << "\n";
    }
  }

  // dN/dy = sum_phi sum_pT w_phi w_pT dN  (default float format, 8 significant digits)
  for (int ipart = 0; ipart < npart; ipart++) {
    char name[255];
    std::snprintf(name, sizeof(name), "%s/results/dN_dy_%d.dat", wd.c_str(), mcid[ipart]);
    std::ofstream yf(name, std::ios_base::app);
    if (!yf) { *err = std::string("cannot open ") + name; return false; }
    for (int iy = 0; iy < y_pts; iy++) {
      double y = g.y.at(1, iy + 1);
      if (dimension == 2) y = 0.0;
      double dN_dy = 0.0;
      for (int iphi = 0; iphi < nphi; iphi++) {
        const double w_phi = g.phi.at(2, iphi + 1);
        for (int ipT = 0; ipT < npT; ipT++)
          dN_dy += w_phi * g.pT.at(2, ipT + 1) * dN[(size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy)];
      }
      yf << std::setw(5) << std::setprecision(8) << y << "\t" << dN_dy << "\n";
    }
  }
  return true;
}

// results/dN_pTdpTdphidy_resonance_decays.dat and results/dN_dpTdphidy_resonance_decays.dat (append mode), as
// write_dN_pTdpTdphidy_with_resonance_decays_toFile / write_dN_dpTdphidy_with_resonance_decays_toFile write them
// (emissionfunction.cpp:452-488, 555-590): all species concatenated, the second file with a header and the values times pT
static bool write_decay_files(const std::string &wd, const std::vector<double> &dN, int npart, const Grids &g, int dimension, std::string *err)
{
  const int npT = (int)g.pT.rows, nphi = (int)g.phi.rows, y_pts = (dimension == 2) ? 1 : (int)g.y.rows;
  for (int which = 0; which < 2; which++) {
    const std::string path = wd + (which == 0 ? "/results/dN_pTdpTdphidy_resonance_decays.dat" : "/results/dN_dpTdphidy_resonance_decays.dat");
    std::ofstream f(path.c_str(), std::ios_base::app);
    if (!f) { *err = "cannot open " + path; return false; }
    if (which == 1) f << "y" << "\t" << "phip" << "\t" << "pT" << "\t" << "dN_dpTdphidy" << "\n";
    for (int ipart = 0; ipart < npart; ipart++)
      for (int iy = 0; iy < y_pts; iy++) {
        const double y = (dimension == 2) ? 0.0 : g.y.at(1, iy + 1);
        for (int iphi = 0; iphi < nphi; iphi++) {
          for (int ipT = 0; ipT < npT; ipT++) {
            const double pT = g.pT.at(1, ipT + 1);
            double value = dN[(size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy)];
            if (which == 1) value = value * pT;
            f << std::scientific << std::setw(5) << std::setprecision(8) << y << "\t" << g.phi.at(1, iphi + 1) << "\t" << pT << "\t" << value << "\n";
          }
          f << "\n";
        }
      }
  }
  return true;
}

// results/spacetime_distribution/*.dat exactly as calculate_dN_dX{,_feqmod} write them (smooth_kernels.cpp:1112-1126, 1404-1435):
// truncating opens, `setprecision(6) << scientific`, bin midpoints, sums divided by the bin volumes.
static bool write_spacetime_files(const std::string &wd, const std::vector<int> &mcid, const is3d_spacetime_bins &b, int eta_pts,
                                  const std::vector<double> &eta_values, const std::vector<double> &dN_tau, const std::vector<double> &dN_r,
                                  const std::vector<double> &dN_taur, const std::vector<double> &dN_dydeta, std::string *err)
{
  const int nt = b.tau_bins, nr = b.r_bins;
  const double tw = (b.tau_max - b.tau_min) / (double)nt, rw = (b.r_max - b.r_min) / (double)nr;
  std::vector<double> tau_mid(nt), r_mid(nr);
  for (int i = 0; i < nt; i++) tau_mid[i] = b.tau_min + tw * ((double)i + 0.5);
  for (int i = 0; i < nr; i++) r_mid[i] = b.r_min + rw * ((double)i + 0.5);
  const std::string dir = wd + "/results/spacetime_distribution/";
  for (size_t s = 0; s < mcid.size(); s++) {
    char n1[64], n2[64], n3[64], n4[96];
    std::snprintf(n1, sizeof(n1), "dN_taudtaudy_%d.dat", mcid[s]);
    std::snprintf(n2, sizeof(n2), "dN_twopirdrdy_%d.dat", mcid[s]);
    std::snprintf(n3, sizeof(n3), "dN_twopitaurdtaudrdy_%d.dat", mcid[s]);
    std::snprintf(n4, sizeof(n4), "dN_dydeta_%d_%dpt.dat", mcid[s], eta_pts);
    std::ofstream ft(dir + n1, std::ios_base::out), fr(dir + n2, std::ios_base::out), ftr(dir + n3, std::ios_base::out), fe(dir + n4, std::ios_base::out);
    if (!ft || !fr || !ftr || !fe) { *err = "cannot write into " + dir + " (the directory must exist, cleanMakeCPU.sh)"; return false; }
    const double *ht = &dN_tau[s * nt], *hr = &dN_r[s * nr], *htr = &dN_taur[s * (size_t)nt * nr], *he = &dN_dydeta[s * (size_t)eta_pts];
    for (int ir = 0; ir < nr; ir++) {
      fr << std::setprecision(6) << std::scientific << r_mid[ir] << "\t" << hr[ir] / (2.0 * M_PI * r_mid[ir] * rw) << "\n";
      for (int it = 0; it < nt; it++)
        ftr << std::setprecision(6) << std::scientific << tau_mid[it] << "\t" << r_mid[ir] << "\t"
            << htr[(size_t)it * nr + ir] / (2.0 * M_PI * tau_mid[it] * r_mid[ir] * tw * rw) << "\n";
    }
    for (int it = 0; it < nt; it++) ft << std::setprecision(6) << std::scientific << tau_mid[it] << "\t" << ht[it] / (tau_mid[it] * tw) << "\n";
    for (int j = 0; j < eta_pts; j++) fe << std::setprecision(6) << std::scientific << eta_values[j] << "\t" << he[j] << "\n";
  }
  return true;
}

// results/polarization/S_<mcid>.dat: mean spin vector S^mu = N^mu / Snorm (lab frame, Cartesian t, x, y, z; 0 where Snorm = 0) and its
// rest-frame spatial part S*_i = S^i - S^t p^i / (E + m), one row per (y, phi, pT) in the loop order, number format and blank line per
// phi block of write_spectra_files; truncating opens, results/polarization/ must exist.
// With the sums of one more term xi (St | Sx | Sy | Sz | Snorm of is3d_b200_spin_polarization_shear or _spin_hall, non-NULL) it writes
// S_<stem>_<mcid>.dat instead: Snorm, that term's part N_xi / Snorm (columns S?_<stem>), the total S = (N + N_xi) / Snorm and the
// rest-frame part of the total.
// stem: the file name stem of the plain form ("S"; "S_fd" for the sums after the feed-down through decays, "S_fdw" after the weak decays
// too), or the tag of the term
// ("xi" for the thermal shear, "she" for the spin Hall term).
static bool write_polarization_files(const std::string &wd, const std::vector<double> &sums, const std::vector<double> *xi,
                                     const std::vector<int> &mcid, const std::vector<double> &mass, const Grids &g, int dimension,
                                     std::string *err, const char *stem = "S")
{
  const int npart = (int)mcid.size(), npT = (int)g.pT.rows, nphi = (int)g.phi.rows, ny = (int)g.y.rows;
  const int y_pts = (dimension == 2) ? 1 : ny;
  const size_t n_bins = (size_t)npart * npT * nphi * ny;
  const double *St = &sums[0], *Sx = St + n_bins, *Sy = Sx + n_bins, *Sz = Sy + n_bins, *Sn = Sz + n_bins;
  const double *Xx = xi ? &(*xi)[n_bins] : nullptr, *Xy = xi ? Xx + n_bins : nullptr, *Xz = xi ? Xy + n_bins : nullptr;
  for (int ipart = 0; ipart < npart; ipart++) {
    char name[255];
    if (xi) std::snprintf(name, sizeof(name), "%s/results/polarization/S_%s_%d.dat", wd.c_str(), stem, mcid[ipart]);
    else std::snprintf(name, sizeof(name), "%s/results/polarization/%s_%d.dat", wd.c_str(), stem, mcid[ipart]);
    std::ofstream f(name, std::ios_base::out);
    if (!f) { *err = std::string("cannot open ") + name + " (the directory results/polarization/ must exist)"; return false; }
    if (xi) f << "y\tphip\tpT\tSnorm\tSx_" << stem << "\tSy_" << stem << "\tSz_" << stem << "\tSx\tSy\tSz\tSx_rest\tSy_rest\tSz_rest\n";
    else f << "y\tphip\tpT\tSnorm\tSt\tSx\tSy\tSz\tSx_rest\tSy_rest\tSz_rest\n";
    const double m = mass[ipart];
    for (int iy = 0; iy < y_pts; iy++) {
      const double y = (dimension == 2) ? 0.0 : g.y.at(1, iy + 1);
      for (int iphi = 0; iphi < nphi; iphi++) {
        const double phi = g.phi.at(1, iphi + 1);
        for (int ipT = 0; ipT < npT; ipT++) {
          const double pT = g.pT.at(1, ipT + 1), mT = std::sqrt(m * m + pT * pT);
          const double E = mT * std::cosh(y), p[3] = {pT * std::cos(phi), pT * std::sin(phi), mT * std::sinh(y)};
          const size_t b = (size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy);
          double S[4] = {0.0, 0.0, 0.0, 0.0}, X[3] = {0.0, 0.0, 0.0};
          if (Sn[b] != 0.0) { S[0] = St[b] / Sn[b]; S[1] = Sx[b] / Sn[b]; S[2] = Sy[b] / Sn[b]; S[3] = Sz[b] / Sn[b]; }
          if (xi && Sn[b] != 0.0) {
            X[0] = Xx[b] / Sn[b]; X[1] = Xy[b] / Sn[b]; X[2] = Xz[b] / Sn[b];
            S[1] = (Sx[b] + Xx[b]) / Sn[b]; S[2] = (Sy[b] + Xy[b]) / Sn[b]; S[3] = (Sz[b] + Xz[b]) / Sn[b];
          }
          f << std::scientific << std::setw(5) << std::setprecision(8) << y << "\t" << phi << "\t" << pT << "\t" << Sn[b];
          if (xi) for (int k = 0; k < 3; k++) f << "\t" << X[k];
          for (int k = xi ? 1 : 0; k < 4; k++) f << "\t" << S[k];
          for (int k = 0; k < 3; k++) f << "\t" << S[k + 1] - S[0] * p[k] / (E + m);
          f << "\n";
        }
        f << "\n";
      }
    }
  }
  return true;
}

// results/polarization/spin_<mcid>.dat, for every chosen species with degeneracy g >= 2: Snorm, the all-order rest-frame mean spin
// <S*_i> = P_i / Snorm and the rank-2 spin tensor T_ij = Q_ij / Snorm (T_zz = -T_xx - T_yy; all 0 where Snorm = 0) of the nine raw sums
// of is3d_b200_spin_density (Snorm | Px | Py | Pz | Qxx | Qxy | Qxz | Qyy | Qyz), one row per (y, phi, pT) in the loop order, number
// format and blank line per phi block of write_spectra_files; truncating opens, results/polarization/ must exist
static bool write_spin_density_files(const std::string &wd, const std::vector<double> &sums, const std::vector<int> &mcid,
                                     const std::vector<double> &degen, const Grids &g, int dimension, std::string *err)
{
  const int npart = (int)mcid.size(), npT = (int)g.pT.rows, nphi = (int)g.phi.rows, ny = (int)g.y.rows;
  const int y_pts = (dimension == 2) ? 1 : ny;
  const size_t n_bins = (size_t)npart * npT * nphi * ny;
  const double *Sn = &sums[0];
  for (int ipart = 0; ipart < npart; ipart++) {
    if (degen[ipart] < 2.0) continue;
    char name[255];
    std::snprintf(name, sizeof(name), "%s/results/polarization/spin_%d.dat", wd.c_str(), mcid[ipart]);
    std::ofstream f(name, std::ios_base::out);
    if (!f) { *err = std::string("cannot open ") + name + " (the directory results/polarization/ must exist)"; return false; }
    f << "y\tphip\tpT\tSnorm\tSx\tSy\tSz\tTxx\tTxy\tTxz\tTyy\tTyz\tTzz\n";
    for (int iy = 0; iy < y_pts; iy++) {
      const double y = (dimension == 2) ? 0.0 : g.y.at(1, iy + 1);
      for (int iphi = 0; iphi < nphi; iphi++) {
        const double phi = g.phi.at(1, iphi + 1);
        for (int ipT = 0; ipT < npT; ipT++) {
          const double pT = g.pT.at(1, ipT + 1);
          const size_t b = (size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy);
          double v[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};    // Sx Sy Sz Txx Txy Txz Tyy Tyz Tzz
          if (Sn[b] != 0.0) {
            for (int q = 0; q < 8; q++) v[q] = sums[(q + 1) * n_bins + b] / Sn[b];
            v[8] = -(sums[4 * n_bins + b] + sums[7 * n_bins + b]) / Sn[b];
          }
          f << std::scientific << std::setw(5) << std::setprecision(8) << y << "\t" << phi << "\t" << pT << "\t" << Sn[b];
          for (int q = 0; q < 9; q++) f << "\t" << v[q];
          f << "\n";
        }
        f << "\n";
      }
    }
  }
  return true;
}

// results/hbt/R2_<mcid>.dat: S0 and the HBT radii R^2_ij = S_ij / S0 - (S_i / S0)(S_j / S0) [fm^2] (all 0 where S0 = 0) of the raw sums of
// is3d_b200_hbt_moments, one row per (y, phi, pT) in the loop order, number format and blank line per phi block of write_spectra_files;
// truncating opens, results/hbt/ must exist
static bool write_hbt_files(const std::string &wd, const std::vector<double> &sums, const std::vector<int> &mcid, const Grids &g,
                            int dimension, std::string *err)
{
  const int npart = (int)mcid.size(), npT = (int)g.pT.rows, nphi = (int)g.phi.rows, ny = (int)g.y.rows;
  const int y_pts = (dimension == 2) ? 1 : ny;
  const size_t n_bins = (size_t)npart * npT * nphi * ny;
  auto S = [&](int q, size_t b) { return sums[(size_t)q * n_bins + b]; };     // S0 So Ss Sl Soo Sss Sll Sos Sol Ssl
  static const int pairs[6][3] = {{4, 1, 1}, {5, 2, 2}, {6, 3, 3}, {7, 1, 2}, {8, 1, 3}, {9, 2, 3}};   // (S_ij, i, j): out side long os ol sl
  for (int ipart = 0; ipart < npart; ipart++) {
    char name[255];
    std::snprintf(name, sizeof(name), "%s/results/hbt/R2_%d.dat", wd.c_str(), mcid[ipart]);
    std::ofstream f(name, std::ios_base::out);
    if (!f) { *err = std::string("cannot open ") + name + " (the directory results/hbt/ must exist)"; return false; }
    f << "y\tphip\tpT\tS0\tR2_out\tR2_side\tR2_long\tR2_outside\tR2_outlong\tR2_sidelong\n";
    for (int iy = 0; iy < y_pts; iy++) {
      const double y = (dimension == 2) ? 0.0 : g.y.at(1, iy + 1);
      for (int iphi = 0; iphi < nphi; iphi++) {
        for (int ipT = 0; ipT < npT; ipT++) {
          const size_t b = (size_t)bin_index(ipart, npart, ipT, npT, iphi, nphi, iy);
          const double s0 = S(0, b);
          f << std::scientific << std::setw(5) << std::setprecision(8) << y << "\t" << g.phi.at(1, iphi + 1) << "\t" << g.pT.at(1, ipT + 1) << "\t" << s0;
          for (const int *pr : pairs) f << "\t" << (s0 != 0.0 ? S(pr[0], b) / s0 - (S(pr[1], b) / s0) * (S(pr[2], b) / s0) : 0.0);
          f << "\n";
        }
        f << "\n";
      }
    }
  }
  return true;
}

// results/hbt/C_<mcid>.dat: the correlation functions C = 1 - sign (Re^2 + Im^2) / (g S0^2) (C = 1 where S0 = 0) along the out, side and long
// rays of is3d_b200_hbt_fourier for one species (re, im: [3][n_q][n_bins] of the one-species call), one row per (y, phi, pT, q) in that loop
// order, the number format and blank line per phi block of write_hbt_files; truncating open, results/hbt/ must exist
static bool write_correlation_file(const std::string &wd, const std::vector<double> &re, const std::vector<double> &im, int mcid, double sign,
                                   double degeneracy, int n_q, double dq, const Grids &g, int dimension, std::string *err)
{
  const int npT = (int)g.pT.rows, nphi = (int)g.phi.rows, ny = (int)g.y.rows;
  const int y_pts = (dimension == 2) ? 1 : ny;
  const size_t n_bins = (size_t)npT * nphi * ny;
  char name[255];
  std::snprintf(name, sizeof(name), "%s/results/hbt/C_%d.dat", wd.c_str(), mcid);
  std::ofstream f(name, std::ios_base::out);
  if (!f) { *err = std::string("cannot open ") + name + " (the directory results/hbt/ must exist)"; return false; }
  f << "y\tphip\tpT\tq\tS0\tC_out\tC_side\tC_long\n";
  for (int iy = 0; iy < y_pts; iy++) {
    const double y = (dimension == 2) ? 0.0 : g.y.at(1, iy + 1);
    for (int iphi = 0; iphi < nphi; iphi++) {
      for (int ipT = 0; ipT < npT; ipT++) {
        const size_t b = (size_t)bin_index(0, 1, ipT, npT, iphi, nphi, iy);
        const double s0 = re[b];
        for (int k = 0; k < n_q; k++) {
          f << std::scientific << std::setw(5) << std::setprecision(8) << y << "\t" << g.phi.at(1, iphi + 1) << "\t" << g.pT.at(1, ipT + 1) << "\t"
            << k * dq << "\t" << s0;
          for (int d = 0; d < 3; d++) {
            const size_t i = ((size_t)d * n_q + k) * n_bins + b;
            const double r = re[i] / s0, m = im[i] / s0;                 // ratios first: S0^2 underflows in the far tails
            f << "\t" << (s0 != 0.0 ? 1.0 - sign * (r * r + m * m) / degeneracy : 1.0);
          }
          f << "\n";
        }
      }
      f << "\n";
    }
  }
  return true;
}

// everything the host layer derives from the input files
struct Problem {
  Params par;
  is3d_flags fl;
  int operation = 0, hrg_eos = 0, group_particles = 0, do_resonance_decays = 0;
  int spin_polarization = 0;               // optional key (absent: 0): mode-5 spin polarization after the spectra
  int thermal_shear_polarization = 0;      // optional key (absent: 0): add the thermal-shear term (input/thermal_shear.dat)
  int spin_hall_polarization = 0;          // optional key (absent: 0): add the spin Hall term (input/muB_over_T_gradient.dat)
  int polarization_feed_down = 0;          // optional key (absent: 0): feed the polarization sums down through the decay tables
  int polarization_weak_decays = 0;        // optional key (absent: 0): then through the weak decays of PDG/weak_decays.dat
  WeakTable weak;                          // that table
  int spin_density = 0;                    // optional key (absent: 0): mode-5 spin density matrix (all-order spin, rank-2 tensor)
  std::map<long, int> box_parity;          // its parities by |MC id| (PDG/pdg_box.dat)
  int hbt_radii = 0;                       // optional key (absent: 0): HBT radii of the linear-delta-f spectra after the spectra
  int hbt_correlation = 0;                 // optional key (absent: 0): MC id of the species whose HBT correlation functions are written
  int hbt_species = -1;                    // its index among the chosen species
  double hbt_dq = 0.005;                   // optional key: q step of the out, side and long rays [GeV]
  int hbt_q_points = 41;                   // optional key: q points per ray (q = 0 included)
  std::vector<int> pick;                   // particle-list index of every chosen species (chosen_particles_sampling_table)
  SurfaceData sf;
  std::vector<Particle> pdg;
  DfTables dft;
  Laguerre gla;
  std::vector<double> mass, sign, degen, baryon;
  std::vector<int> mcid;
  Grids g;
};

static int load_problem(const std::string &wd, bool need_surface, Problem *p, std::string *err_out)
{
  std::string &err = *err_out;
  Params &par = p->par;
  if (!par.load(wd + "/iS3D_parameters.dat", &err)) return IS3D_ERR_IO;
  // the reference constructor reads every key, sampler ones included, and a missing key is fatal
  // (emissionfunction.cpp:170-222); keep that contract so that a file accepted here is accepted there
  static const char *required[] = {"operation", "mode", "hrg_eos", "set_FO_temperature", "T_switch", "dimension", "df_mode",
    "include_baryon", "include_bulk_deltaf", "include_shear_deltaf", "include_baryondiff_deltaf", "regulate_deltaf", "outflow",
    "deta_min", "group_particles", "particle_diff_tolerance", "mass_pion0", "do_resonance_decays", "lightest_particle",
    "oversample", "max_num_samples", "fast", "min_num_hadrons", "sampler_seed", "test_sampler", "pT_lower_cut", "pT_upper_cut",
    "pT_bins", "y_cut", "y_bins", "eta_cut", "eta_bins", "tau_min", "tau_max", "tau_bins", "r_min", "r_max", "r_bins"};
  for (const char *k : required) par.get(k, &err);
  if (!err.empty()) return IS3D_ERR_IO;
  p->operation = (int)par.get("operation", &err); p->hrg_eos = (int)par.get("hrg_eos", &err);
  p->group_particles = (int)par.get("group_particles", &err);
  is3d_flags &fl = p->fl; std::memset(&fl, 0, sizeof(fl));
  fl.mode = (int)par.get("mode", &err); fl.df_mode = (int)par.get("df_mode", &err); fl.dimension = (int)par.get("dimension", &err);
  fl.include_baryon = (int)par.get("include_baryon", &err);
  fl.include_bulk_deltaf = (int)par.get("include_bulk_deltaf", &err);
  fl.include_shear_deltaf = (int)par.get("include_shear_deltaf", &err);
  fl.include_baryondiff_deltaf = (int)par.get("include_baryondiff_deltaf", &err);
  fl.regulate_deltaf = (int)par.get("regulate_deltaf", &err);
  fl.outflow = (int)par.get("outflow", &err);
  fl.deta_min = par.get("deta_min", &err); fl.mass_pion0 = par.get("mass_pion0", &err);
  if (p->operation != 1 && p->operation != 0) { err = "this drop-in covers operation = 1 (smooth momentum spectra) and operation = 0 (spacetime distributions); the sampler (operation = 2) is out of scope"; return IS3D_ERR_UNSUPPORTED; }
  if (p->operation == 0 && fl.mode == 2) { err = "operation = 0 has no anisotropic-hydro routine in the reference (emissionfunction.cpp:1644-1673)"; return IS3D_ERR_UNSUPPORTED; }
  p->do_resonance_decays = (int)par.get("do_resonance_decays", &err);
  if (p->do_resonance_decays && p->operation != 1) { err = "do_resonance_decays = 1 applies to operation = 1 (the reference runs it after the spectra, emissionfunction.cpp:1689)"; return IS3D_ERR_UNSUPPORTED; }
  p->spin_polarization = par.has("spin_polarization") ? (int)par.get("spin_polarization", &err) : 0;
  if (p->spin_polarization && (p->operation != 1 || fl.mode != 5)) { err = "spin_polarization = 1 needs operation = 1 and a mode 5 surface (the thermal vorticity columns)"; return IS3D_ERR_UNSUPPORTED; }
  p->thermal_shear_polarization = par.has("thermal_shear_polarization") ? (int)par.get("thermal_shear_polarization", &err) : 0;
  if (p->thermal_shear_polarization && (p->operation != 1 || fl.mode != 5 || !p->spin_polarization)) {
    err = "thermal_shear_polarization = 1 needs operation = 1, a mode 5 surface and spin_polarization = 1"; return IS3D_ERR_UNSUPPORTED;
  }
  p->spin_hall_polarization = par.has("spin_hall_polarization") ? (int)par.get("spin_hall_polarization", &err) : 0;
  if (p->spin_hall_polarization && (p->operation != 1 || fl.mode != 5 || !p->spin_polarization)) {
    err = "spin_hall_polarization = 1 needs operation = 1, a mode 5 surface and spin_polarization = 1"; return IS3D_ERR_UNSUPPORTED;
  }
  p->polarization_feed_down = par.has("polarization_feed_down") ? (int)par.get("polarization_feed_down", &err) : 0;
  if (p->polarization_feed_down && (p->operation != 1 || fl.mode != 5 || !p->spin_polarization || (p->hrg_eos != 1 && p->hrg_eos != 2))) {
    err = "polarization_feed_down = 1 needs operation = 1, a mode 5 surface, spin_polarization = 1 and a particle list with decay tables "
          "(hrg_eos = 1, 2)";
    return IS3D_ERR_UNSUPPORTED;
  }
  p->polarization_weak_decays = par.has("polarization_weak_decays") ? (int)par.get("polarization_weak_decays", &err) : 0;
  if (p->polarization_weak_decays && !p->polarization_feed_down) {
    err = "polarization_weak_decays = 1 needs polarization_feed_down = 1 (it amends the fed-down sums)"; return IS3D_ERR_UNSUPPORTED;
  }
  p->spin_density = par.has("spin_density") ? (int)par.get("spin_density", &err) : 0;
  if (p->spin_density && (p->operation != 1 || fl.mode != 5)) { err = "spin_density = 1 needs operation = 1 and a mode 5 surface (the thermal vorticity columns)"; return IS3D_ERR_UNSUPPORTED; }
  p->hbt_radii = par.has("hbt_radii") ? (int)par.get("hbt_radii", &err) : 0;
  if (p->hbt_radii && (p->operation != 1 || fl.mode == 2 || (fl.df_mode != 1 && fl.df_mode != 2) || fl.include_baryon)) {
    err = "hbt_radii = 1 needs operation = 1, a viscous-hydro surface (mode != 2), df_mode 1 or 2 and include_baryon = 0"; return IS3D_ERR_UNSUPPORTED;
  }
  p->hbt_correlation = par.has("hbt_correlation") ? (int)par.get("hbt_correlation", &err) : 0;
  if (p->hbt_correlation && (p->operation != 1 || fl.mode == 2 || (fl.df_mode != 1 && fl.df_mode != 2) || fl.include_baryon)) {
    err = "hbt_correlation needs operation = 1, a viscous-hydro surface (mode != 2), df_mode 1 or 2 and include_baryon = 0"; return IS3D_ERR_UNSUPPORTED;
  }
  if (par.has("hbt_dq")) p->hbt_dq = par.get("hbt_dq", &err);
  if (par.has("hbt_q_points")) p->hbt_q_points = (int)par.get("hbt_q_points", &err);
  if (p->hbt_correlation && (!std::isfinite(p->hbt_dq) || p->hbt_dq <= 0.0 || p->hbt_q_points < 1)) {
    err = "hbt_dq must be > 0 and hbt_q_points >= 1"; return IS3D_ERR_ARGUMENT;
  }
  if (p->do_resonance_decays && p->hrg_eos == 3) { err = "do_resonance_decays = 1 needs a particle list with decay tables (hrg_eos = 1, 2); pdg_box.dat has none"; return IS3D_ERR_UNSUPPORTED; }

  // ---- surface (+ averages side file)
  if (need_surface) {
    SurfaceFlags sfl{fl.mode, fl.dimension, fl.df_mode, fl.include_baryon, fl.include_baryondiff_deltaf};
    if (!read_surface(wd, sfl, &p->sf, &err)) return IS3D_ERR_IO;
    if (p->thermal_shear_polarization && !read_thermal_shear(wd, &p->sf, &err)) return IS3D_ERR_IO;
    if (p->spin_hall_polarization && !read_baryon_gradient(wd, &p->sf, &err)) return IS3D_ERR_IO;
  }
  // ---- particle list, delta-f tables
  if (!read_pdg(wd, p->hrg_eos, &p->pdg, &err)) return IS3D_ERR_IO;
  if (p->polarization_feed_down && !read_box_parities(wd, &p->box_parity, &err)) return IS3D_ERR_IO;
  if (p->polarization_weak_decays && !read_weak_decays(wd, &p->weak, &err)) return IS3D_ERR_IO;
  if ((int)p->pdg.size() > 600) { err = "number of particles exceeds Maxparticle = 600"; return IS3D_ERR_IO; }
  if (!read_df_tables(wd, p->hrg_eos, &p->dft, &err)) return IS3D_ERR_IO;
  if (!read_laguerre(wd + "/tables/gla_roots_weights_32_points.txt", &p->gla, &err)) return IS3D_ERR_IO;
  if (p->gla.alpha < 3) { err = "Gauss-Laguerre table needs alpha = 0..2"; return IS3D_ERR_IO; }
  if (need_surface) {
    if (fl.mode != 2 && fl.df_mode == 4) compute_jonah_tables(p->pdg, p->sf.avg[0], p->gla, &p->dft);
    if (fl.mode == 2 && !fill_vah_coefficients(wd, &p->sf, &err)) return IS3D_ERR_IO;
  }
  // ---- chosen species in file order (first match in the particle list), optional mass bubble sort
  BlockTable chosen;
  if (!chosen.load(wd + "/PDG/chosen_particles.dat", &err)) return IS3D_ERR_IO;
  const int npart = (int)chosen.rows;
  std::vector<int> pick;
  for (int m = 0; m < npart; m++) {
    const int id = (int)chosen.at(1, m + 1);
    int found = -1;
    for (size_t n = 0; n < p->pdg.size(); n++) if (p->pdg[n].mcid == id) { found = (int)n; break; }
    if (found < 0) { err = "chosen particle " + std::to_string(id) + " is not in the particle list (the reference leaves that slot uninitialised)"; return IS3D_ERR_IO; }
    pick.push_back(found);
  }
  if (p->group_particles == 1)
    for (int m = 0; m < npart; m++)
      for (int n = 0; n < npart - m - 1; n++)
        if (p->pdg[pick[n]].mass > p->pdg[pick[n + 1]].mass) std::swap(pick[n], pick[n + 1]);
  p->pick = pick;
  p->mass.resize(npart); p->sign.resize(npart); p->degen.resize(npart); p->baryon.resize(npart); p->mcid.resize(npart);
  for (int i = 0; i < npart; i++) {
    const Particle &h = p->pdg[pick[i]];
    p->mass[i] = h.mass; p->sign[i] = h.sign; p->degen[i] = h.gspin; p->baryon[i] = h.baryon; p->mcid[i] = (int)h.mcid;
  }
  if (p->hbt_correlation) {
    for (int i = 0; i < npart && p->hbt_species < 0; i++) if (p->mcid[i] == p->hbt_correlation) p->hbt_species = i;
    if (p->hbt_species < 0) { err = "hbt_correlation = " + std::to_string(p->hbt_correlation) + " is not among the chosen particles"; return IS3D_ERR_ARGUMENT; }
  }
  // ---- momentum tables (iS3D.cpp:161-167)
  Grids &g = p->g;
  if (!g.pT.load(wd + "/tables/pT_gauss_legendre_table.dat", &err) || !g.phi.load(wd + "/tables/phi_gauss_legendre_table.dat", &err) ||
      !g.y.load(wd + "/tables/y_trapezoid_table_21pt.dat", &err) || !g.eta.load(wd + "/tables/eta/eta_trapezoid_table_241pt.dat", &err))
    return IS3D_ERR_IO;
  if (g.pT.cols.size() < 2 || g.phi.cols.size() < 2 || g.eta.cols.size() < 2) { err = "momentum tables need a weight column"; return IS3D_ERR_IO; }
  return IS3D_OK;
}

// the particle list with its decay channels flattened for is3d_b200_resonance_decays / is3d_b200_polarization_decays
struct FlatList {
  std::vector<int32_t> mcid, stable, decays, first, npart, parts;
  std::vector<double> mass, width, br;
  explicit FlatList(const std::vector<Particle> &pdg)
  {
    for (const Particle &h : pdg) {
      mcid.push_back((int32_t)h.mcid); mass.push_back(h.mass); width.push_back(h.width); stable.push_back(h.stable);
      decays.push_back((int32_t)h.channels.size()); first.push_back((int32_t)npart.size());
      for (const DecayChannel &ch : h.channels) {
        npart.push_back(ch.npart); br.push_back(ch.branch_ratio);
        for (int k = 0; k < 5; k++) parts.push_back((int32_t)ch.part[k]);
      }
    }
  }
  is3d_particle_list view()
  {
    return is3d_particle_list{(int32_t)mcid.size(), mcid.data(), mass.data(), width.data(), stable.data(), decays.data(), first.data(),
                              npart.data(), br.data(), parts.data()};
  }
};

static int run_problem(const std::string &wd, Problem &P, const is3d_surface &s, const is3d_vorticity *vort, const is3d_thermal_shear *shear,
                       const is3d_baryon_gradient *grad, double *dN_raw, int64_t n_raw, int32_t *mcid_out, int32_t n_mcid_max, is3d_stats *stats,
                       std::string *err_out)
{
  std::string &err = *err_out;
  const Grids &g = P.g; const DfTables &dft = P.dft; const Laguerre &gla = P.gla;
  const int npart = (int)P.mcid.size();
  // the file-level drop-in uses every visible GPU (or IS3D_B200_GPUS of them): cells are sharded inside the C ABI
  {
    const int rc_dev = is3d_b200_init_devices(0);
    if (rc_dev != IS3D_OK) { err = is3d_b200_last_error(); return rc_dev; }
  }
  is3d_species sp{npart, P.mass.data(), P.sign.data(), P.degen.data(), P.baryon.data()};
  is3d_grid gr{(int32_t)g.pT.rows, (int32_t)g.phi.rows, (int32_t)g.y.rows, (int32_t)g.eta.rows,
               g.pT.cols[0].data(), g.phi.cols[0].data(), g.y.cols[0].data(), g.eta.cols[0].data(), g.eta.cols[1].data()};
  is3d_df_tables dt; std::memset(&dt, 0, sizeof(dt));
  dt.n_T = dft.n_T; dt.T = dft.T.data(); dt.c0 = dft.c0.data(); dt.c1 = dft.c1.data(); dt.c2 = dft.c2.data(); dt.c3 = dft.c3.data();
  dt.c4 = dft.c4.data(); dt.F = dft.F.data(); dt.G = dft.G.data(); dt.betabulk = dft.betabulk.data(); dt.betaV = dft.betaV.data();
  dt.betapi = dft.betapi.data();
  if (!dft.jonah_x.empty()) {
    dt.n_jonah = (int32_t)dft.jonah_x.size(); dt.jonah_x = dft.jonah_x.data(); dt.jonah_lambda2 = dft.jonah_lambda2.data();
    dt.jonah_z = dft.jonah_z.data(); dt.bulkPi_over_Peq_max = dft.bulkPi_over_Peq_max;
  }
  is3d_laguerre la{gla.points, gla.root[1].data(), gla.weight[1].data(), gla.root[2].data(), gla.weight[2].data()};
  if (P.operation == 0) {
    // spacetime distributions (emissionfunction.cpp:1512-1516, 1577-1581): nothing else is written for this operation
    is3d_spacetime_bins b; std::memset(&b, 0, sizeof(b));
    std::string e2;
    b.tau_min = P.par.get("tau_min", &e2); b.tau_max = P.par.get("tau_max", &e2); b.tau_bins = (int32_t)P.par.get("tau_bins", &e2);
    b.r_min = P.par.get("r_min", &e2); b.r_max = P.par.get("r_max", &e2); b.r_bins = (int32_t)P.par.get("r_bins", &e2);
    b.pT_weight = g.pT.cols[1].data(); b.phi_weight = g.phi.cols[1].data();
    if (b.tau_bins <= 0 || b.r_bins <= 0) { err = "tau_bins and r_bins must be positive"; return IS3D_ERR_ARGUMENT; }
    const int eta_pts = (P.fl.dimension == 2) ? (int)g.eta.rows : 1;
    const size_t nt = (size_t)b.tau_bins, nr = (size_t)b.r_bins;
    std::vector<double> h_tau(npart * nt), h_r(npart * nr), h_taur(npart * nt * nr), h_eta((size_t)npart * eta_pts), h_y((size_t)npart);
    is3d_spacetime_result res{h_tau.data(), h_r.data(), h_taur.data(), h_eta.data(), h_y.data()};
    is3d_stats st0; std::memset(&st0, 0, sizeof(st0));
    const int rc0 = is3d_b200_spacetime_distributions_multi(&P.fl, &s, &sp, &gr, &dt, &la, &b, nullptr, &res, &st0);
    if (stats) *stats = st0;
    if (rc0 != IS3D_OK) { err = std::string("spacetime kernel failed: ") + is3d_b200_last_error(); return rc0; }
    std::vector<double> eta_values(eta_pts, 0.0);
    if (P.fl.dimension == 2) for (int j = 0; j < eta_pts; j++) eta_values[j] = g.eta.at(1, j + 1);
    else if (s.n_cells > 0) eta_values[0] = s.eta[s.n_cells - 1];          // the reference's etaValues[0] still holds the last cell's eta (:1154)
    for (int i = 0; i < npart; i++) std::printf("dN_dy = %lf\n", h_y[i]);   // :1439-1442
    if (dN_raw) {                                                          // [dN_tau | dN_r | dN_taur | dN_dydeta | dN_dy]
      std::vector<double> all;
      for (const std::vector<double> *v : {&h_tau, &h_r, &h_taur, &h_eta, &h_y}) all.insert(all.end(), v->begin(), v->end());
      std::memcpy(dN_raw, all.data(), sizeof(double) * (size_t)std::min<int64_t>(n_raw, (int64_t)all.size()));
    }
    if (mcid_out) for (int i = 0; i < npart && i < n_mcid_max; i++) mcid_out[i] = P.mcid[i];
    if (!write_spacetime_files(wd, P.mcid, b, eta_pts, eta_values, h_tau, h_r, h_taur, h_eta, &err)) return IS3D_ERR_IO;
    return IS3D_OK;
  }
  const size_t n_bins = (size_t)npart * g.pT.rows * g.phi.rows * g.y.rows;
  std::vector<double> dN(n_bins, 0.0);
  is3d_stats st; std::memset(&st, 0, sizeof(st));
  const int rc = is3d_b200_smooth_spectra_multi(&P.fl, &s, &sp, &gr, &dt, &la, nullptr, dN.data(), &st);
  if (stats) *stats = st;
  if (rc != IS3D_OK) { err = std::string("spectra kernel failed: ") + is3d_b200_last_error(); return rc; }
  if (P.fl.mode != 2 && (P.fl.df_mode == 3 || P.fl.df_mode == 4))
    std::cout << std::setw(5) << std::setprecision(4) << "\nfeqmod breaks down for " << st.cells_feqmod_breakdown << " cells\n" << std::endl;
  if (mcid_out) for (int i = 0; i < npart && i < n_mcid_max; i++) mcid_out[i] = P.mcid[i];
  if (!write_spectra_files(wd, dN, P.mcid, g, P.fl.dimension, &err)) return IS3D_ERR_IO;
  if (P.spin_polarization) {
    std::vector<double> sums(5 * n_bins, 0.0);                   // St | Sx | Sy | Sz | Snorm
    is3d_polarization_result r{&sums[0], &sums[n_bins], &sums[2 * n_bins], &sums[3 * n_bins], &sums[4 * n_bins]};
    is3d_stats sp_st; std::memset(&sp_st, 0, sizeof(sp_st));
    const int rcp = is3d_b200_spin_polarization_multi(&P.fl, &s, vort, &sp, &gr, nullptr, &r, &sp_st);
    if (rcp != IS3D_OK) { err = std::string("spin polarization failed: ") + is3d_b200_last_error(); return rcp; }
    if (stats) { stats->gpu_launches += sp_st.gpu_launches; stats->total_ms += sp_st.total_ms; }
    if (!write_polarization_files(wd, sums, nullptr, P.mcid, P.mass, g, P.fl.dimension, &err)) return IS3D_ERR_IO;
    if (P.thermal_shear_polarization) {
      std::vector<double> xi(5 * n_bins, 0.0);                   // St (zeros) | Sx | Sy | Sz | Snorm
      is3d_polarization_result rx{&xi[0], &xi[n_bins], &xi[2 * n_bins], &xi[3 * n_bins], &xi[4 * n_bins]};
      std::memset(&sp_st, 0, sizeof(sp_st));
      const int rcx = is3d_b200_spin_polarization_shear_multi(&P.fl, &s, shear, &sp, &gr, nullptr, &rx, &sp_st);
      if (rcx != IS3D_OK) { err = std::string("thermal-shear polarization failed: ") + is3d_b200_last_error(); return rcx; }
      if (stats) { stats->gpu_launches += sp_st.gpu_launches; stats->total_ms += sp_st.total_ms; }
      if (!write_polarization_files(wd, sums, &xi, P.mcid, P.mass, g, P.fl.dimension, &err, "xi")) return IS3D_ERR_IO;
      for (size_t k = 0; k < 4 * n_bins; k++) sums[k] += xi[k];  // the feed-down below runs on the total (vorticity + shear)
    }
    if (P.spin_hall_polarization) {
      std::vector<double> she(5 * n_bins, 0.0);                  // St (zeros) | Sx | Sy | Sz | Snorm
      is3d_polarization_result rh{&she[0], &she[n_bins], &she[2 * n_bins], &she[3 * n_bins], &she[4 * n_bins]};
      std::memset(&sp_st, 0, sizeof(sp_st));
      const int rch = is3d_b200_spin_polarization_spin_hall_multi(&P.fl, &s, grad, &sp, &gr, nullptr, &rh, &sp_st);
      if (rch != IS3D_OK) { err = std::string("spin Hall polarization failed: ") + is3d_b200_last_error(); return rch; }
      if (stats) { stats->gpu_launches += sp_st.gpu_launches; stats->total_ms += sp_st.total_ms; }
      if (!write_polarization_files(wd, sums, &she, P.mcid, P.mass, g, P.fl.dimension, &err, "she")) return IS3D_ERR_IO;
      for (size_t k = 0; k < 4 * n_bins; k++) sums[k] += she[k]; // the feed-down below runs on the total (vorticity (+ shear) + spin Hall)
    }
    if (P.polarization_feed_down) {
      // 2J = gspin - 1 of the list, parities by |MC id| from pdg_box.dat (0, unknown: the channel only dilutes)
      std::vector<int32_t> spin2, parity, chosen(P.pick.begin(), P.pick.end());
      for (const Particle &h : P.pdg) {
        spin2.push_back(h.gspin - 1);
        const auto it = P.box_parity.find(std::labs(h.mcid));
        parity.push_back(it == P.box_parity.end() ? 0 : it->second);
      }
      FlatList flat(P.pdg);
      const is3d_particle_list pl = flat.view();
      const is3d_spin_parity spp{spin2.data(), parity.data()};
      is3d_polarization_result r{&sums[0], &sums[n_bins], &sums[2 * n_bins], &sums[3 * n_bins], &sums[4 * n_bins]};
      is3d_stats fd_st; std::memset(&fd_st, 0, sizeof(fd_st));
      const int rcf = is3d_b200_polarization_decays(&pl, &spp, npart, chosen.data(), &gr, P.fl.dimension, nullptr, &r, &fd_st);
      if (rcf != IS3D_OK) { err = std::string("polarization feed-down failed: ") + is3d_b200_last_error(); return rcf; }
      if (stats) { stats->gpu_launches += fd_st.gpu_launches; stats->total_ms += fd_st.total_ms; }
      if (!write_polarization_files(wd, sums, nullptr, P.mcid, P.mass, g, P.fl.dimension, &err, "S_fd")) return IS3D_ERR_IO;
      if (P.polarization_weak_decays) {               // the weak pass on a copy of the fed-down sums: S_fd_ stays as it is
        std::vector<double> fdw(sums);
        is3d_polarization_result rw{&fdw[0], &fdw[n_bins], &fdw[2 * n_bins], &fdw[3 * n_bins], &fdw[4 * n_bins]};
        const is3d_weak_decays wt{(int32_t)P.weak.parent.size(), P.weak.parent.data(), P.weak.daughter.data(), P.weak.partner.data(),
                                  P.weak.branching.data(), P.weak.alpha.data(), P.weak.phi.data()};
        std::memset(&fd_st, 0, sizeof(fd_st));
        const int rcw = is3d_b200_polarization_weak_decays(&pl, &spp, &wt, npart, chosen.data(), &gr, P.fl.dimension, nullptr, &rw, &fd_st);
        if (rcw != IS3D_OK) { err = std::string("weak-decay polarization feed-down failed: ") + is3d_b200_last_error(); return rcw; }
        if (stats) { stats->gpu_launches += fd_st.gpu_launches; stats->total_ms += fd_st.total_ms; }
        if (!write_polarization_files(wd, fdw, nullptr, P.mcid, P.mass, g, P.fl.dimension, &err, "S_fdw")) return IS3D_ERR_IO;
      }
    }
  }
  if (P.spin_density) {
    std::vector<double> sums(9 * n_bins, 0.0);                   // Snorm | Px | Py | Pz | Qxx | Qxy | Qxz | Qyy | Qyz
    double *b = sums.data();
    is3d_spin_density_result r{b, b + n_bins, b + 2 * n_bins, b + 3 * n_bins, b + 4 * n_bins, b + 5 * n_bins, b + 6 * n_bins,
                               b + 7 * n_bins, b + 8 * n_bins};
    is3d_stats sd_st; std::memset(&sd_st, 0, sizeof(sd_st));
    const int rcs = is3d_b200_spin_density_multi(&P.fl, &s, vort, &sp, &gr, nullptr, &r, &sd_st);
    if (rcs != IS3D_OK) { err = std::string("spin density failed: ") + is3d_b200_last_error(); return rcs; }
    if (stats) { stats->gpu_launches += sd_st.gpu_launches; stats->total_ms += sd_st.total_ms; }
    if (!write_spin_density_files(wd, sums, P.mcid, P.degen, g, P.fl.dimension, &err)) return IS3D_ERR_IO;
  }
  if (P.hbt_radii) {
    std::vector<double> sums(10 * n_bins, 0.0);                  // S0 | So | Ss | Sl | Soo | Sss | Sll | Sos | Sol | Ssl
    double *b = sums.data();
    is3d_hbt_result r{b, b + n_bins, b + 2 * n_bins, b + 3 * n_bins, b + 4 * n_bins, b + 5 * n_bins, b + 6 * n_bins, b + 7 * n_bins,
                      b + 8 * n_bins, b + 9 * n_bins};
    is3d_stats hb_st; std::memset(&hb_st, 0, sizeof(hb_st));
    const int rch = is3d_b200_hbt_moments_multi(&P.fl, &s, &sp, &gr, &dt, nullptr, &r, &hb_st);
    if (rch != IS3D_OK) { err = std::string("HBT moments failed: ") + is3d_b200_last_error(); return rch; }
    if (stats) { stats->gpu_launches += hb_st.gpu_launches; stats->total_ms += hb_st.total_ms; }
    if (!write_hbt_files(wd, sums, P.mcid, g, P.fl.dimension, &err)) return IS3D_ERR_IO;
  }
  if (P.hbt_correlation) {
    const int i = P.hbt_species, n_q = P.hbt_q_points;
    is3d_species one{1, &P.mass[i], &P.sign[i], &P.degen[i], &P.baryon[i]};
    static const double rays[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};        // out, side, long
    is3d_hbt_qrays qr{3, n_q, P.hbt_dq, rays};
    const size_t n = (size_t)3 * n_q * (n_bins / npart);
    std::vector<double> re(n, 0.0), im(n, 0.0);
    is3d_hbt_fourier_result r{re.data(), im.data()};
    is3d_stats hq_st; std::memset(&hq_st, 0, sizeof(hq_st));
    const int rcq = is3d_b200_hbt_fourier_multi(&P.fl, &s, &one, &gr, &dt, &qr, nullptr, &r, &hq_st);
    if (rcq != IS3D_OK) { err = std::string("HBT correlation failed: ") + is3d_b200_last_error(); return rcq; }
    if (stats) { stats->gpu_launches += hq_st.gpu_launches; stats->total_ms += hq_st.total_ms; }
    if (!write_correlation_file(wd, re, im, P.mcid[i], P.sign[i], P.degen[i], n_q, P.hbt_dq, g, P.fl.dimension, &err)) return IS3D_ERR_IO;
  }
  if (P.do_resonance_decays) {
    // feed-down on the GPU, then the two amended-spectra files (emissionfunction.cpp:1689-1698)
    std::printf("Starting resonance decays: \n\n");
    std::vector<int32_t> chosen(P.pick.begin(), P.pick.end());
    FlatList flat(P.pdg);
    const is3d_particle_list pl = flat.view();
    is3d_stats sd; std::memset(&sd, 0, sizeof(sd));
    const int rcd = is3d_b200_resonance_decays(&pl, npart, chosen.data(), &gr, P.fl.dimension, nullptr, dN.data(), &sd);
    if (rcd != IS3D_OK) { err = std::string("resonance decays failed: ") + is3d_b200_last_error(); return rcd; }
    std::printf("\n\nResonance decays took %f seconds.\n", sd.total_ms * 1e-3);
    if (stats) { stats->gpu_launches += sd.gpu_launches; stats->total_ms += sd.total_ms; }
    if (!write_decay_files(wd, dN, npart, g, P.fl.dimension, &err)) return IS3D_ERR_IO;
  }
  if (dN_raw) std::memcpy(dN_raw, dN.data(), sizeof(double) * (size_t)std::min<int64_t>(n_raw, (int64_t)n_bins));
  return IS3D_OK;
}

}  // namespace is3d

using namespace is3d;

extern "C" int is3d_b200_run_workdir(const char *workdir, double *dN_raw, int64_t n_raw, int32_t *mcid_out, int32_t n_mcid_max,
                                     is3d_stats *stats)
{
  const std::string wd = (workdir && *workdir) ? workdir : ".";
  std::string err;
  auto fail = [&](int code) { g_host_error = err; std::fprintf(stderr, "is3d_b200: %s\n", err.c_str()); return code; };
  Problem P;
  int rc = load_problem(wd, true, &P, &err);
  if (rc != IS3D_OK) return fail(rc);
  const SurfaceData &sf = P.sf;
  is3d_surface s; std::memset(&s, 0, sizeof(s));
  s.n_cells = sf.n;
  s.tau = sf.tau.data(); s.eta = sf.eta.data(); s.dat = sf.dat.data(); s.dax = sf.dax.data(); s.day = sf.day.data(); s.dan = sf.dan.data();
  s.ux = sf.ux.data(); s.uy = sf.uy.data(); s.un = sf.un.data(); s.T = sf.T.data(); s.P = sf.P.data(); s.E = sf.E.data();
  s.pixx = sf.pixx.data(); s.pixy = sf.pixy.data(); s.pixn = sf.pixn.data(); s.piyy = sf.piyy.data(); s.piyn = sf.piyn.data();
  s.bulkPi = sf.bulkPi.data(); s.muB = sf.muB.data(); s.nB = sf.nB.data(); s.Vx = sf.Vx.data(); s.Vy = sf.Vy.data(); s.Vn = sf.Vn.data();
  s.x = sf.x.data(); s.y = sf.y.data();
  if (P.fl.mode == 2) {
    s.pitt = sf.pitt.data(); s.pitx = sf.pitx.data(); s.pity = sf.pity.data(); s.pitn = sf.pitn.data(); s.pinn = sf.pinn.data();
    s.Wx = sf.Wx.data(); s.Wy = sf.Wy.data(); s.Lambda = sf.Lambda.data(); s.aL = sf.aL.data();
    s.c0 = sf.c0.data(); s.c1 = sf.c1.data(); s.c2 = sf.c2.data(); s.c3 = sf.c3.data(); s.c4 = sf.c4.data();
  }
  const is3d_vorticity vort{sf.wtx.data(), sf.wty.data(), sf.wtn.data(), sf.wxy.data(), sf.wxn.data(), sf.wyn.data()};
  const is3d_thermal_shear shear{sf.xtt.data(), sf.xtx.data(), sf.xty.data(), sf.xtn.data(), sf.xxx.data(), sf.xxy.data(), sf.xxn.data(),
                                 sf.xyy.data(), sf.xyn.data(), sf.xnn.data()};
  const is3d_baryon_gradient grad{sf.gbt.data(), sf.gbx.data(), sf.gby.data(), sf.gbn.data()};
  rc = run_problem(wd, P, s, P.fl.mode == 5 ? &vort : nullptr, P.thermal_shear_polarization ? &shear : nullptr,
                   P.spin_hall_polarization ? &grad : nullptr, dN_raw, n_raw, mcid_out, n_mcid_max, stats, &err);
  return rc == IS3D_OK ? rc : fail(rc);
}

// In-memory surface (the reference's IS3D::read_fo_surf_from_memory + run_particlization(0), iS3D.cpp:26-71, 99-134):
// the freeze-out cells come from the caller, everything else (parameters, particle list, tables) from `workdir`.
// Unlike the reference -- which leaves the averages side file stale on this path -- the df_mode 4 tables are built from
// the surface that was actually passed in.
extern "C" int is3d_b200_run_surface(const char *workdir, const is3d_surface *surface, double *dN_raw, int64_t n_raw,
                                     int32_t *mcid_out, int32_t n_mcid_max, is3d_stats *stats)
{
  const std::string wd = (workdir && *workdir) ? workdir : ".";
  std::string err;
  auto fail = [&](int code) { g_host_error = err; std::fprintf(stderr, "is3d_b200: %s\n", err.c_str()); return code; };
  if (!surface) { err = "NULL surface"; return fail(IS3D_ERR_ARGUMENT); }
  Problem P;
  int rc = load_problem(wd, false, &P, &err);
  if (rc != IS3D_OK) return fail(rc);
  if (P.fl.mode != 2 && P.fl.df_mode == 4) {
    double avg[5];
    rc = is3d_b200_surface_averages(surface, avg);
    if (rc != IS3D_OK) { err = "cannot average an empty surface"; return fail(rc); }
    compute_jonah_tables(P.pdg, avg[0], P.gla, &P.dft);
  }
  rc = run_problem(wd, P, *surface, nullptr, nullptr, nullptr, dN_raw, n_raw, mcid_out, n_mcid_max, stats, &err);
  return rc == IS3D_OK ? rc : fail(rc);
}

// Writers only: takes a spectra array (reference layout) and produces the results/ files for `workdir`.
extern "C" int is3d_b200_write_results(const char *workdir, const double *dN, int64_t n)
{
  const std::string wd = (workdir && *workdir) ? workdir : ".";
  std::string err;
  Problem P;
  int rc = load_problem(wd, false, &P, &err);
  if (rc != IS3D_OK) { g_host_error = err; return rc; }
  const size_t n_bins = (size_t)P.mcid.size() * P.g.pT.rows * P.g.phi.rows * P.g.y.rows;
  if (!dN || (size_t)n != n_bins) { g_host_error = "spectra array has the wrong length"; return IS3D_ERR_ARGUMENT; }
  std::vector<double> v(dN, dN + n);
  if (!write_spectra_files(wd, v, P.mcid, P.g, P.fl.dimension, &err)) { g_host_error = err; return IS3D_ERR_IO; }
  return IS3D_OK;
}

// Host-layer inspection (no GPU work): parses every input file of `workdir` and writes what it derived -- species
// arrays, surface SoA, coefficient tables -- as named records [int32 name_len][name][int64 n][n doubles] to `out_path`.
extern "C" int is3d_b200_host_dump(const char *workdir, const char *out_path)
{
  const std::string wd = (workdir && *workdir) ? workdir : ".";
  std::string err;
  Problem P;
  int rc = load_problem(wd, true, &P, &err);
  if (rc != IS3D_OK) { g_host_error = err; return rc; }
  FILE *f = std::fopen(out_path, "wb");
  if (!f) { g_host_error = "cannot write dump"; return IS3D_ERR_IO; }
  auto put = [&](const char *name, const std::vector<double> &v) {
    int32_t len = (int32_t)std::strlen(name); int64_t n = (int64_t)v.size();
    std::fwrite(&len, 4, 1, f); std::fwrite(name, 1, len, f); std::fwrite(&n, 8, 1, f);
    if (n) std::fwrite(v.data(), 8, (size_t)n, f);
  };
  std::vector<double> tmp;
  tmp.assign(P.mcid.begin(), P.mcid.end()); put("mcid", tmp);
  put("mass", P.mass); put("sign", P.sign); put("degeneracy", P.degen); put("baryon", P.baryon);
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back((double)h.mcid); put("pdg_mcid", tmp);
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back(h.mass); put("pdg_mass", tmp);
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back(h.gspin); put("pdg_gspin", tmp);
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back(h.sign); put("pdg_sign", tmp);
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back(h.baryon); put("pdg_baryon", tmp);
  // decay tables (resonance-decay feed-down): stable flag, channels per particle, flattened channel rows
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back(h.stable); put("pdg_stable", tmp);
  tmp.clear(); for (auto &h : P.pdg) tmp.push_back((double)h.channels.size()); put("pdg_decays", tmp);
  tmp.clear(); for (auto &h : P.pdg) for (auto &ch : h.channels) tmp.push_back(ch.npart); put("pdg_dec_npart", tmp);
  tmp.clear(); for (auto &h : P.pdg) for (auto &ch : h.channels) tmp.push_back(ch.branch_ratio); put("pdg_dec_br", tmp);
  tmp.clear(); for (auto &h : P.pdg) for (auto &ch : h.channels) for (int k = 0; k < 5; k++) tmp.push_back((double)ch.part[k]); put("pdg_dec_part", tmp);
  const SurfaceData &s = P.sf;
  put("tau", s.tau); put("eta", s.eta); put("dat", s.dat); put("dax", s.dax); put("day", s.day); put("dan", s.dan);
  put("ux", s.ux); put("uy", s.uy); put("un", s.un); put("E", s.E); put("T", s.T); put("P", s.P);
  put("pixx", s.pixx); put("pixy", s.pixy); put("pixn", s.pixn); put("piyy", s.piyy); put("piyn", s.piyn); put("bulkPi", s.bulkPi);
  put("pitt", s.pitt); put("pitx", s.pitx); put("pity", s.pity); put("pitn", s.pitn); put("pinn", s.pinn);
  put("Wx", s.Wx); put("Wy", s.Wy); put("Lambda", s.Lambda); put("aL", s.aL);
  put("c0", s.c0); put("c1", s.c1); put("c2", s.c2); put("c3", s.c3); put("c4", s.c4);
  put("wtx", s.wtx); put("wty", s.wty); put("wtn", s.wtn); put("wxy", s.wxy); put("wxn", s.wxn); put("wyn", s.wyn);
  if (P.thermal_shear_polarization) {
    put("xtt", s.xtt); put("xtx", s.xtx); put("xty", s.xty); put("xtn", s.xtn); put("xxx", s.xxx);
    put("xxy", s.xxy); put("xxn", s.xxn); put("xyy", s.xyy); put("xyn", s.xyn); put("xnn", s.xnn);
  }
  if (P.spin_hall_polarization) { put("gbt", s.gbt); put("gbx", s.gbx); put("gby", s.gby); put("gbn", s.gbn); }
  if (P.polarization_feed_down) {        // what the feed-down passes as is3d_spin_parity: 2J = gspin - 1, parity by |MC id| (0 unknown)
    tmp.clear(); for (auto &h : P.pdg) tmp.push_back(h.gspin - 1); put("pdg_spin2", tmp);
    tmp.clear();
    for (auto &h : P.pdg) { const auto it = P.box_parity.find(std::labs(h.mcid)); tmp.push_back(it == P.box_parity.end() ? 0 : it->second); }
    put("pdg_parity", tmp);
  }
  if (P.polarization_weak_decays) {      // the weak-decay table as read: one record per column
    tmp.assign(P.weak.parent.begin(), P.weak.parent.end()); put("weak_parent", tmp);
    tmp.assign(P.weak.daughter.begin(), P.weak.daughter.end()); put("weak_daughter", tmp);
    tmp.assign(P.weak.partner.begin(), P.weak.partner.end()); put("weak_partner", tmp);
    put("weak_branching", P.weak.branching); put("weak_alpha", P.weak.alpha); put("weak_phi", P.weak.phi);
  }
  tmp.assign(s.avg, s.avg + 5); put("avg", tmp);
  put("df_T", P.dft.T); put("df_c0", P.dft.c0); put("df_c2", P.dft.c2); put("df_F", P.dft.F); put("df_betabulk", P.dft.betabulk);
  put("df_betapi", P.dft.betapi); put("jonah_x", P.dft.jonah_x); put("jonah_lambda2", P.dft.jonah_lambda2); put("jonah_z", P.dft.jonah_z);
  tmp.assign(1, P.dft.bulkPi_over_Peq_max); put("jonah_max", tmp);
  put("pT", P.g.pT.cols[0]); put("phi", P.g.phi.cols[0]); put("y", P.g.y.cols[0]); put("eta_tab", P.g.eta.cols[0]); put("eta_weight", P.g.eta.cols[1]);
  put("gla_root1", P.gla.root[1]); put("gla_weight2", P.gla.weight[2]);
  tmp = {(double)P.fl.mode, (double)P.fl.df_mode, (double)P.fl.dimension, (double)P.fl.include_baryon, (double)P.fl.include_bulk_deltaf,
         (double)P.fl.include_shear_deltaf, (double)P.fl.include_baryondiff_deltaf, (double)P.fl.regulate_deltaf, (double)P.fl.outflow,
         P.fl.deta_min, P.fl.mass_pion0};
  put("flags", tmp);
  std::fclose(f);
  return IS3D_OK;
}

extern "C" int is3d_b200_surface_averages(const is3d_surface *sf, double *out5)
{
  if (!sf || !out5 || sf->n_cells <= 0) return IS3D_ERR_ARGUMENT;
  double Tavg = 0, Eavg = 0, Pavg = 0, muBavg = 0, nBavg = 0, volume = 0;
  for (int64_t i = 0; i < sf->n_cells; i++) {
    const double tau = sf->tau[i], ux = sf->ux[i], uy = sf->uy[i], un = sf->un[i];
    const double ut = std::sqrt(1.0 + ux * ux + uy * uy + tau * tau * un * un);
    const double dat = sf->dat[i], dax = sf->dax[i], day = sf->day[i], dan = sf->dan[i];
    const double udsigma = ut * dat + ux * dax + uy * day + un * dan;
    const double dsds = dat * dat - dax * dax - day * day - dan * dan / (tau * tau);
    const double mag = std::fabs(udsigma) + std::sqrt(std::fabs(udsigma * udsigma - dsds));
    const double muB = sf->muB ? sf->muB[i] : 0.0, nB = sf->nB ? sf->nB[i] : 0.0;
    volume += mag;
    Eavg += (sf->E[i] * mag); Tavg += (sf->T[i] * mag); Pavg += (sf->P[i] * mag); muBavg += (muB * mag); nBavg += (nB * mag);
  }
  const double v[5] = {Tavg / volume, Eavg / volume, Pavg / volume, muBavg / volume, nBavg / volume};
  for (int k = 0; k < 5; k++) {                  // the reference writes these with 15 digits and reads them back
    char buf[64];
    std::snprintf(buf, sizeof(buf), "%.15g", v[k]);
    out5[k] = std::strtod(buf, nullptr);
  }
  return IS3D_OK;
}

// Anisotropic-hydro helpers for in-memory callers: (alpha_L, Lambda) from (T, P, PL) in the file's fm units as
// FO_data_reader::read_surf_VAH_PLMatch infers them (readindata.cpp:905-918), and the per-cell c0..c4 lookup.
extern "C" int is3d_b200_vah_anisotropy(int64_t n, const double *T_fm, const double *P_fm, const double *PL_fm, double *aL_out, double *Lambda_GeV_out)
{
  if (n < 0 || !T_fm || !P_fm || !PL_fm || !aL_out || !Lambda_GeV_out) return IS3D_ERR_ARGUMENT;
  for (int64_t i = 0; i < n; i++) {
    if (!((PL_fm[i] / P_fm[i]) < 3.0)) { g_host_error = "pl is too large, stopping anisotropic variables"; return IS3D_ERR_TABLE_RANGE; }
    const double a = aL_fit(PL_fm[i] / P_fm[i]);
    aL_out[i] = a;
    Lambda_GeV_out[i] = (T_fm[i] / std::pow(0.5 * a * R200(a), 0.25)) * 0.197327053;
  }
  return IS3D_OK;
}

extern "C" int is3d_b200_vah_coefficients(int32_t nL, int32_t naL, const double *L_fm, const double *aL_grid, const double *c0, const double *c1,
                                          const double *c2, const double *c3, const double *c4, int64_t n, const double *Lambda_GeV,
                                          const double *aL, double *o0, double *o1, double *o2, double *o3, double *o4)
{
  if (nL < 2 || naL < 2 || !L_fm || !aL_grid || !c0 || !c1 || !c2 || !c3 || !c4 || n < 0 || !Lambda_GeV || !aL) return IS3D_ERR_ARGUMENT;
  const double *c[5] = {c0, c1, c2, c3, c4};
  double *o[5] = {o0, o1, o2, o3, o4};
  for (int64_t i = 0; i < n; i++) {
    double out[5];
    if (!vah_lookup(nL, naL, L_fm, aL_grid, c, Lambda_GeV[i] / 0.197327053, aL[i], out)) {
      g_host_error = "cell " + std::to_string(i) + ": (Lambda, alpha_L) outside the vah coefficient table";
      return IS3D_ERR_TABLE_RANGE;
    }
    for (int k = 0; k < 5; k++) o[k][i] = out[k];
  }
  return IS3D_OK;
}

extern "C" int is3d_b200_jonah_tables(int32_t n_particles, const double *mass, const double *degeneracy, const double *sign, double T_avg,
                                      int32_t n_points, const double *root2, const double *weight2,
                                      double *x301, double *lambda2_301, double *z301, double *mx)
{
  if (n_particles <= 0 || !mass || !degeneracy || !sign || n_points <= 0 || !root2 || !weight2 || !x301 || !lambda2_301 || !z301)
    return IS3D_ERR_ARGUMENT;
  std::vector<Particle> pdg((size_t)n_particles);
  for (int i = 0; i < n_particles; i++) { pdg[i].mass = mass[i]; pdg[i].gspin = (int)degeneracy[i]; pdg[i].sign = (int)sign[i]; }
  Laguerre gla; gla.alpha = 3; gla.points = n_points;
  gla.root.assign(3, std::vector<double>(root2, root2 + n_points)); gla.weight.assign(3, std::vector<double>(weight2, weight2 + n_points));
  DfTables t;
  compute_jonah_tables(pdg, T_avg, gla, &t);
  std::memcpy(x301, t.jonah_x.data(), 301 * sizeof(double));
  std::memcpy(lambda2_301, t.jonah_lambda2.data(), 301 * sizeof(double));
  std::memcpy(z301, t.jonah_z.data(), 301 * sizeof(double));
  if (mx) *mx = t.bulkPi_over_Peq_max;
  return IS3D_OK;
}

// Per-species equilibrium density and bulk / diffusion corrections at the surface-average T, E, P: what
// Deltaf_Data::compute_particle_densities (deltafReader.cpp:536-650) stores in particle_info and the sampler's yield
// estimate consumes.  avg5 = (T, E, P, muB, nB) as is3d_b200_surface_averages returns them; include_baryon = 0 (muB = nB = 0).
extern "C" int is3d_b200_particle_densities(int32_t n, const double *mass, const double *degeneracy, const double *baryon,
                                            const double *sign, const double *avg5, int32_t df_mode, const is3d_df_tables *df,
                                            int32_t n_points, const double *root1, const double *weight1, const double *root2,
                                            const double *weight2, const double *root3, const double *weight3,
                                            double *neq_out, double *dn_bulk_out, double *dn_diff_out)
{
  if (n <= 0 || !mass || !degeneracy || !baryon || !sign || !avg5 || !df || n_points <= 0 || !root1 || !weight1 || !neq_out || !dn_bulk_out || !dn_diff_out)
    return IS3D_ERR_ARGUMENT;
  if (df_mode < 1 || df_mode > 4) return IS3D_ERR_ARGUMENT;
  if ((df_mode == 1 && (!root2 || !weight2 || !root3 || !weight3 || !df->c0 || !df->c2)) ||
      ((df_mode == 2 || df_mode == 3) && (!root2 || !weight2 || !df->F || !df->betabulk))) return IS3D_ERR_ARGUMENT;
  const double hbarC = 0.197327053, two_pi2_hbarC3 = 2.0 * std::pow(M_PI, 2) * std::pow(hbarC, 3);
  const double T = avg5[0], E = avg5[1], P = avg5[2], muB = avg5[3], nB = avg5[4];
  // Deltaf_Data::cubic_spline at (T, bulkPi = 0), deltafReader.cpp:325-395: T-scalings undone, G = c1 = c3 = c4 = 0, betaV = 1
  auto coef = [&](const double *y, double *out) {
    if (!y || df->n_T < 3) return false;
    std::vector<double> c(df->n_T);
    host_spline_init(df->T, y, df->n_T, c.data());
    return host_spline_eval(df->T, y, c.data(), df->n_T, T, out);
  };
  const double T4 = T * T * T * T;
  double c0 = 0, c2 = 0, F = 0, betabulk = 1;
  if (df_mode == 1) {
    if (!coef(df->c0, &c0) || !coef(df->c2, &c2)) { g_host_error = "average temperature outside the delta-f coefficient table"; return IS3D_ERR_TABLE_RANGE; }
    c0 /= T4; c2 /= T4;
  } else if (df_mode == 2 || df_mode == 3) {
    if (!coef(df->F, &F) || !coef(df->betabulk, &betabulk)) { g_host_error = "average temperature outside the delta-f coefficient table"; return IS3D_ERR_TABLE_RANGE; }
    F *= T; betabulk *= T4;
  }
  const double c1 = 0.0, c3 = 0.0, c4 = 0.0, G = 0.0, betaV = 1.0;
  const double alphaB = muB / T, baryon_enthalpy_ratio = nB / (E + P);
  auto sum = [&](double (*f)(double, double, double, double, double), const double *root, const double *w, double mbar, double b, double sg) {
    double acc = 0.0;
    for (int k = 0; k < n_points; k++) acc += w[k] * f(root[k], mbar, alphaB, b, sg);
    return acc;
  };
  // integrands of gaussThermal.cpp:19-90
  auto neq_i = [](double p, double m, double a, double b, double s) { const double Eb = std::sqrt(p * p + m * m); return p * std::exp(p) / (std::exp(Eb - b * a) + s); };
  auto J10_i = [](double p, double m, double a, double b, double s) { const double Eb = std::sqrt(p * p + m * m), q = std::exp(Eb - b * a) + s; return p * std::exp(p + Eb - b * a) / (q * q); };
  auto J11_i = [](double p, double m, double a, double b, double s) { const double Eb = std::sqrt(p * p + m * m), q = std::exp(Eb - b * a) + s; return p * p * p / (Eb * Eb) * std::exp(p + Eb - b * a) / (q * q); };
  auto J20_i = [](double p, double m, double a, double b, double s) { const double Eb = std::sqrt(p * p + m * m), q = std::exp(Eb - b * a) + s; return Eb * std::exp(p + Eb - b * a) / (q * q); };
  auto J30_i = [](double p, double m, double a, double b, double s) { const double Eb = std::sqrt(p * p + m * m), q = std::exp(Eb - b * a) + s; return Eb * Eb / p * std::exp(p + Eb - b * a) / (q * q); };
  auto J31_i = [](double p, double m, double a, double b, double s) { const double Eb = std::sqrt(p * p + m * m), q = std::exp(Eb - b * a) + s; return p * std::exp(p + Eb - b * a) / (q * q); };
  for (int i = 0; i < n; i++) {
    const double m = mass[i], g = degeneracy[i], b = baryon[i], sg = sign[i], mbar = m / T;
    const double neq_fact = g * std::pow(T, 3) / two_pi2_hbarC3;
    const double neq = neq_fact * sum(neq_i, root1, weight1, mbar, b, sg);
    double dn_bulk = 0.0, dn_diff = 0.0;
    if (df_mode == 1) {
      const double J10_fact = g * std::pow(T, 3) / two_pi2_hbarC3, J20_fact = g * std::pow(T, 4) / two_pi2_hbarC3;
      const double J30_fact = g * std::pow(T, 5) / two_pi2_hbarC3, J31_fact = g * std::pow(T, 5) / two_pi2_hbarC3 / 3.0;
      const double J10 = J10_fact * sum(J10_i, root1, weight1, mbar, b, sg), J20 = J20_fact * sum(J20_i, root2, weight2, mbar, b, sg);
      const double J30 = J30_fact * sum(J30_i, root3, weight3, mbar, b, sg), J31 = J31_fact * sum(J31_i, root3, weight3, mbar, b, sg);
      dn_bulk = ((c0 - c2) * m * m * J10 + c1 * b * J20 + (4.0 * c2 - c0) * J30);
      dn_diff = b * c3 * neq * T + c4 * J31;
    } else if (df_mode == 2 || df_mode == 3) {
      const double J10_fact = g * std::pow(T, 3) / two_pi2_hbarC3, J11_fact = g * std::pow(T, 3) / two_pi2_hbarC3 / 3.0;
      const double J20_fact = g * std::pow(T, 4) / two_pi2_hbarC3;
      const double J10 = J10_fact * sum(J10_i, root1, weight1, mbar, b, sg), J11 = J11_fact * sum(J11_i, root1, weight1, mbar, b, sg);
      const double J20 = J20_fact * sum(J20_i, root2, weight2, mbar, b, sg);
      dn_bulk = (neq + (b * J10 * G) + (J20 * F / std::pow(T, 2))) / betabulk;
      dn_diff = (neq * T * baryon_enthalpy_ratio - b * J11) / betaV;
    }
    neq_out[i] = neq; dn_bulk_out[i] = dn_bulk; dn_diff_out[i] = dn_diff;
  }
  return IS3D_OK;
}

extern "C" const char *is3d_b200_host_error(void) { return g_host_error.c_str(); }
