// cf_decays.cu -- resonance-decay feed-down of the smooth spectra on the GPU (SURVEY 8f, row N3; sm_100a).
//
// Replaces EmissionFunctionArray::do_resonance_decays and the routines below it (reference
// src/cpp/emissionfunction_resonance_decays.cpp:124-2158): parents are taken from the last chosen species down to the second; for
// every unstable parent the logarithm of its (already amended) spectrum is tabulated, and each 2- / 3-body channel adds, for every
// daughter that is a chosen species, the phase-space integral of the parent spectrum -- 12-point Gauss-Legendre in (v, zeta)
// [and s], bi- / tri-linear interpolation of log dN in (M_T, Phi[, Y]), exponential extrapolation in M_T beyond the table -- to
// the daughter's bins.  NOTE: in the reference snapshot the routine is disabled by an exit(-1) at entry (":126-129, I need to change
// the linear interpolation's MTmax ..."); what is implemented here is the body behind it, checked against that body (oracle/).
//
// B200 mapping: the spectra array stays in HBM (39 MB at 305 species); the work per parent is (channels x daughter groups) "terms" x
// momentum bins, one thread per (term, bin) for 2-body terms (144 integrand points each) and 12 threads -- one per s node -- for
// 3-body terms (1728 points), whose partial sums are folded in node order.  Terms write prefactor x integral to a scratch array
// and a second kernel adds them to the daughters in (channel, group) order, so the result does not depend on the launch geometry
// and follows the reference's accumulation order.  The parent's log table (129 KB) is read through L1/L2.  Parents are inherently
// sequential (a parent's spectrum must have received its own feed-down first).
// The same driver feeds the spin-polarization sums down (is3d_b200_polarization_decays, DESIGN §17): Snorm through exactly these
// launches, and N^mu through decay2_spin_kernel, which shares the 2-body points and interpolation with decay2_kernel.
// Compiled with -fmad=false: products and sums round one by one like the reference's scalar C++.
#include "cf_internal.h"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

namespace is3d {

namespace {

constexpr int GP = 12;                  // Gauss-Legendre points of every decay integral (:493-498, 1001-1006)
__constant__ double kGLRoot[GP] = {-0.98156063424672, -0.90411725637048, -0.76990267419431, -0.58731795428662, -0.3678314989982, -0.12523340851147,
   0.12523340851147, 0.36783149899818, 0.58731795428662, 0.76990267419431, 0.90411725637048, 0.98156063424672};
__constant__ double kGLWeight[GP] = {0.04717533638651, 0.1069393259953, 0.16007832854335, 0.20316742672307, 0.23349253653836, 0.2491470458134,
   0.2491470458134, 0.23349253653836, 0.20316742672307, 0.1600783285433, 0.10693932599532, 0.04717533638651};

struct DecayTerm {
  int body;                 // 2 or 3
  int daughter;             // chosen index of the daughter species the term adds to
  double mass_parent;       // (for 2-body channels possibly shifted to satisfy energy conservation, :241-256)
  double prefactor;
  double mass2, Estar, pstar;                  // 2-body: daughter mass^2, energy and momentum in the parent rest frame
  double m1sq, s_plus, s_minus, d;             // 3-body: daughter mass^2 and the invariant-mass range of the other pair
};

struct DecayGrid {
  int n_species, n_pT, n_phi, n_y_tab, y_pts, dim;
  const double *pT, *phi, *y;
};

struct Fit { double constant, slope; };

// ---- per-term tables: parent transverse masses and the exponential M_T fits
__device__ void lup2_solve(double A[2][2], double b[2])                        // arsenal.cpp:1072-1207 for n = 2
{
  const int n = 2;
  int pvector[2] = {0, 1}, imax = 0;
  double implicit_scale[2] = {0.0, 0.0}, big, sum, temp;
  for (int i = 0; i < n; i++) {
    big = 0.0;
    for (int j = 0; j < n; j++) { temp = fabs(A[i][j]); if (temp > big) big = temp; }
    if (big == 0.0) break;
    implicit_scale[i] = 1.0 / big;
  }
  for (int j = 0; j < n; j++) {
    for (int i = 0; i < j; i++) { sum = A[i][j]; for (int k = 0; k < i; k++) sum -= A[i][k] * A[k][j]; A[i][j] = sum; }
    big = 0.0;
    for (int i = j; i < n; i++) {
      sum = A[i][j];
      for (int k = 0; k < j; k++) sum -= A[i][k] * A[k][j];
      A[i][j] = sum;
      temp = implicit_scale[i] * fabs(sum);
      if (temp >= big) { big = temp; imax = i; }
    }
    if (j != imax) {
      for (int k = 0; k < n; k++) { temp = A[imax][k]; A[imax][k] = A[j][k]; A[j][k] = temp; }
      implicit_scale[imax] = implicit_scale[j];
    }
    pvector[j] = imax;
    if (A[j][j] == 0.0) A[j][j] = 1.0e-16;
    if (j != n - 1) { temp = 1.0 / A[j][j]; for (int i = j + 1; i < n; i++) A[i][j] *= temp; }
  }
  for (int i = 0; i < n; i++) {
    const int ip = pvector[i];
    sum = b[ip]; b[ip] = b[i];
    for (int j = 0; j < i; j++) sum -= A[i][j] * b[j];
    b[i] = sum;
  }
  for (int i = n - 1; i >= 0; i--) {
    sum = b[i];
    for (int j = i + 1; j < n; j++) sum -= A[i][j] * b[j];
    b[i] = sum / A[i][i];
  }
}

__global__ void log_parent_kernel(DecayGrid G, const double *__restrict__ dN, int parent, double *__restrict__ logdN)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = G.n_pT * G.n_phi * G.y_pts;
  if (i >= n) return;
  logdN[i] = log(dN[(int64_t)parent + (int64_t)G.n_species * i]);               // :163-171; i = ipT + n_pT (iphi + n_phi iy)
}

// one block per term: MT[ipT] and, per (iy, iphi), the least-squares line through (mT, log dN) for mT > sqrt(2.73) M (:2032-2158)
__global__ void decay_setup_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const double *__restrict__ logdN,
                                   double *__restrict__ MT_all, Fit *__restrict__ fit_all, int *__restrict__ error)
{
  const DecayTerm T = terms[blockIdx.x];
  double *MT = MT_all + (size_t)blockIdx.x * G.n_pT;
  Fit *fit = fit_all + (size_t)blockIdx.x * G.y_pts * G.n_phi;
  const double M = T.mass_parent;
  for (int ipT = threadIdx.x; ipT < G.n_pT; ipT += blockDim.x) MT[ipT] = sqrt(fabs(G.pT[ipT] * G.pT[ipT] + M * M));
  for (int w = threadIdx.x; w < G.y_pts * G.n_phi; w += blockDim.x) {
    const int iy = w / G.n_phi, iphip = w - iy * G.n_phi;
    double f[2] = {0.0, 0.0}, A[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
    int n = 0;
    // the reference collects the points first and then forms A^T y and A^T A with sums in point order; accumulating them here in
    // the same order gives the same sums
    for (int ipT = 0; ipT < G.n_pT; ipT++) {
      const double l = logdN[ipT + G.n_pT * (iphip + G.n_phi * iy)];
      if (!isfinite(l)) break;
      const double pT = G.pT[ipT];
      const double mT = sqrt(M * M + pT * pT);
      if (mT > sqrt(2.73) * M) {
        f[0] += (1.0 * l); f[1] += (mT * l);
        A[0][0] += (1.0 * 1.0); A[0][1] += (1.0 * mT); A[1][0] += (mT * 1.0); A[1][1] += (mT * mT);
        n++;
      }
    }
    if (n < 2) { atomicExch(error, 1); fit[w].constant = 0.0; fit[w].slope = 0.0; continue; }    // the reference exits here (:2078-2082)
    lup2_solve(A, f);
    fit[w].constant = f[0]; fit[w].slope = f[1];
  }
}

// ---- interpolation of the parent's log spectrum
struct ParentView {
  const double *logdN, *MT; const Fit *fit; const double *phi, *y;
  int n_pT, n_phi; double MTmax;
};

// left / right points in the azimuthal table; angles outside [phi_0, phi_last] wrap around 2 pi (:1439-1489 and its three copies)
__device__ __forceinline__ void phi_points(const ParentView &P, double &Phip, int &iL, int &iR, double &PL, double &PR)
{
  if (Phip >= P.phi[0] && Phip <= P.phi[P.n_phi - 1]) {
    int r = 1;
    while (Phip > P.phi[r]) r++;
    iR = r; iL = r - 1; PL = P.phi[iL]; PR = P.phi[iR];
  } else {
    iL = P.n_phi - 1; iR = 0;
    PL = P.phi[iL] - 2.0 * M_PI; PR = P.phi[iR];
    Phip -= floor(Phip / M_PI) * (2.0 * M_PI);
  }
}

// Polarization feed-down (is3d_b200_polarization_decays): the parent's rest-frame mean spin S*_P, tabulated like logdN ([3][bins]),
// is interpolated LINEARLY at the cell and with the weights of the log spectrum; above MTmax it is held at the last M_T point.
// SpinOut receives, per parent azimuth, exp(log dN) and S*_P there.  The plain feed-down instantiates everything with SPIN = false.
struct SpinOut { double e1, e2, S1[3], S2[3]; };

template <bool SPIN>
__device__ double parent_2d(const ParentView &P, double MT, double Phip1, double Phip2, const double *Sstar = nullptr, SpinOut *so = nullptr)   // :1413-1676
{
  double logdN1, logdN2;
  int i1L, i1R, i2L, i2R; double P1L, P1R, P2L, P2R;
  phi_points(P, Phip1, i1L, i1R, P1L, P1R);
  phi_points(P, Phip2, i2L, i2R, P2L, P2R);
  const double dPhip1 = P1R - P1L, dPhip2 = P2R - P2L;
  if (MT <= P.MTmax) {
    int iMTR = 1;
    while (MT > P.MT[iMTR]) iMTR++;
    const int iMTL = iMTR - 1, npT = P.n_pT;
    const double MTL = P.MT[iMTL], MTR = P.MT[iMTR], dMT = MTR - MTL;
    const double a_LL = P.logdN[iMTL + npT * i1L], a_RL = P.logdN[iMTL + npT * i1R], a_LR = P.logdN[iMTR + npT * i1L], a_RR = P.logdN[iMTR + npT * i1R];
    const double b_LL = P.logdN[iMTL + npT * i2L], b_RL = P.logdN[iMTL + npT * i2R], b_LR = P.logdN[iMTR + npT * i2L], b_RR = P.logdN[iMTR + npT * i2R];
    logdN1 = ((a_LL * (P1R - Phip1) + a_RL * (Phip1 - P1L)) * (MTR - MT) + (a_LR * (P1R - Phip1) + a_RR * (Phip1 - P1L)) * (MT - MTL)) / (dPhip1 * dMT);
    logdN2 = ((b_LL * (P2R - Phip2) + b_RL * (Phip2 - P2L)) * (MTR - MT) + (b_LR * (P2R - Phip2) + b_RR * (Phip2 - P2L)) * (MT - MTL)) / (dPhip2 * dMT);
    if constexpr (SPIN) {
      for (int c = 0; c < 3; c++) {
#define SG(im, ip) Sstar[3 * ((im) + npT * (ip)) + c]
        so->S1[c] = ((SG(iMTL, i1L) * (P1R - Phip1) + SG(iMTL, i1R) * (Phip1 - P1L)) * (MTR - MT)
                   + (SG(iMTR, i1L) * (P1R - Phip1) + SG(iMTR, i1R) * (Phip1 - P1L)) * (MT - MTL)) / (dPhip1 * dMT);
        so->S2[c] = ((SG(iMTL, i2L) * (P2R - Phip2) + SG(iMTL, i2R) * (Phip2 - P2L)) * (MTR - MT)
                   + (SG(iMTR, i2L) * (P2R - Phip2) + SG(iMTR, i2R) * (Phip2 - P2L)) * (MT - MTL)) / (dPhip2 * dMT);
#undef SG
      }
    }
  } else {
    const Fit f1L = P.fit[i1L], f1R = P.fit[i1R], f2L = P.fit[i2L], f2R = P.fit[i2R];
    const double a_L = f1L.constant + f1L.slope * MT, a_R = f1R.constant + f1R.slope * MT;
    const double b_L = f2L.constant + f2L.slope * MT, b_R = f2R.constant + f2R.slope * MT;
    logdN1 = (a_L * (P1R - Phip1) + a_R * (Phip1 - P1L)) / dPhip1;
    logdN2 = (b_L * (P2R - Phip2) + b_R * (Phip2 - P2L)) / dPhip2;
    if constexpr (SPIN) {
      const int im = P.n_pT - 1, npT = P.n_pT;
      for (int c = 0; c < 3; c++) {
        so->S1[c] = (Sstar[3 * (im + npT * i1L) + c] * (P1R - Phip1) + Sstar[3 * (im + npT * i1R) + c] * (Phip1 - P1L)) / dPhip1;
        so->S2[c] = (Sstar[3 * (im + npT * i2L) + c] * (P2R - Phip2) + Sstar[3 * (im + npT * i2R) + c] * (Phip2 - P2L)) / dPhip2;
      }
    }
  }
  if constexpr (SPIN) { so->e1 = exp(logdN1); so->e2 = exp(logdN2); return 0.0; }
  return (exp(logdN1) + exp(logdN2));
}

template <bool SPIN>
__device__ double parent_3d(const ParentView &P, int iYL, int iYR, double YL, double YR, double MT, double Phip1, double Phip2, double Y,   // :1680-2028
                            const double *Sstar = nullptr, SpinOut *so = nullptr)
{
  double logdN1, logdN2;
  int i1L, i1R, i2L, i2R; double P1L, P1R, P2L, P2R;
  const int npT = P.n_pT, nphi = P.n_phi;
  phi_points(P, Phip1, i1L, i1R, P1L, P1R);
  phi_points(P, Phip2, i2L, i2R, P2L, P2R);
  const double dY = YR - YL, dPhip1 = P1R - P1L, dPhip2 = P2R - P2L;
  if (MT <= P.MTmax) {
    int iMTR = 1;
    while (MT > P.MT[iMTR]) iMTR++;
    const int iMTL = iMTR - 1;
    const double MTL = P.MT[iMTL], MTR = P.MT[iMTR], dMT = MTR - MTL;
#define LG(im, ip, iy) P.logdN[(im) + npT * ((ip) + nphi * (iy))]
    const double a_LLL = LG(iMTL, i1L, iYL), a_RLL = LG(iMTL, i1L, iYR), a_LRL = LG(iMTL, i1R, iYL), a_RRL = LG(iMTL, i1R, iYR);
    const double a_LLR = LG(iMTR, i1L, iYL), a_RLR = LG(iMTR, i1L, iYR), a_LRR = LG(iMTR, i1R, iYL), a_RRR = LG(iMTR, i1R, iYR);
    const double b_LLL = LG(iMTL, i2L, iYL), b_RLL = LG(iMTL, i2L, iYR), b_LRL = LG(iMTL, i2R, iYL), b_RRL = LG(iMTL, i2R, iYR);
    const double b_LLR = LG(iMTR, i2L, iYL), b_RLR = LG(iMTR, i2L, iYR), b_LRR = LG(iMTR, i2R, iYL), b_RRR = LG(iMTR, i2R, iYR);
#undef LG
    logdN1 = (MTR - MT) * ((a_LLL * (YR - Y) + a_RLL * (Y - YL)) * (P1R - Phip1) + (a_LRL * (YR - Y) + a_RRL * (Y - YL)) * (Phip1 - P1L))
           + (MT - MTL) * ((a_LLR * (YR - Y) + a_RLR * (Y - YL)) * (P1R - Phip1) + (a_LRR * (YR - Y) + a_RRR * (Y - YL)) * (Phip1 - P1L));
    logdN1 /= (dY * dPhip1 * dMT);
    logdN2 = (MTR - MT) * ((b_LLL * (YR - Y) + b_RLL * (Y - YL)) * (P2R - Phip2) + (b_LRL * (YR - Y) + b_RRL * (Y - YL)) * (Phip2 - P2L))
           + (MT - MTL) * ((b_LLR * (YR - Y) + b_RLR * (Y - YL)) * (P2R - Phip2) + (b_LRR * (YR - Y) + b_RRR * (Y - YL)) * (Phip2 - P2L));
    logdN2 /= (dY * dPhip2 * dMT);
    if constexpr (SPIN) {
      for (int c = 0; c < 3; c++) {
#define SG(im, ip, iy) Sstar[3 * ((im) + npT * ((ip) + nphi * (iy))) + c]
        so->S1[c] = ((MTR - MT) * ((SG(iMTL, i1L, iYL) * (YR - Y) + SG(iMTL, i1L, iYR) * (Y - YL)) * (P1R - Phip1) + (SG(iMTL, i1R, iYL) * (YR - Y) + SG(iMTL, i1R, iYR) * (Y - YL)) * (Phip1 - P1L))
                   + (MT - MTL) * ((SG(iMTR, i1L, iYL) * (YR - Y) + SG(iMTR, i1L, iYR) * (Y - YL)) * (P1R - Phip1) + (SG(iMTR, i1R, iYL) * (YR - Y) + SG(iMTR, i1R, iYR) * (Y - YL)) * (Phip1 - P1L)))
                   / (dY * dPhip1 * dMT);
        so->S2[c] = ((MTR - MT) * ((SG(iMTL, i2L, iYL) * (YR - Y) + SG(iMTL, i2L, iYR) * (Y - YL)) * (P2R - Phip2) + (SG(iMTL, i2R, iYL) * (YR - Y) + SG(iMTL, i2R, iYR) * (Y - YL)) * (Phip2 - P2L))
                   + (MT - MTL) * ((SG(iMTR, i2L, iYL) * (YR - Y) + SG(iMTR, i2L, iYR) * (Y - YL)) * (P2R - Phip2) + (SG(iMTR, i2R, iYL) * (YR - Y) + SG(iMTR, i2R, iYR) * (Y - YL)) * (Phip2 - P2L)))
                   / (dY * dPhip2 * dMT);
#undef SG
      }
    }
  } else {
    const Fit f1LL = P.fit[iYL * nphi + i1L], f1RL = P.fit[iYR * nphi + i1L], f1LR = P.fit[iYL * nphi + i1R], f1RR = P.fit[iYR * nphi + i1R];
    const Fit f2LL = P.fit[iYL * nphi + i2L], f2RL = P.fit[iYR * nphi + i2L], f2LR = P.fit[iYL * nphi + i2R], f2RR = P.fit[iYR * nphi + i2R];
    const double a_LL = f1LL.constant + f1LL.slope * MT, a_LR = f1LR.constant + f1LR.slope * MT, a_RL = f1RL.constant + f1RL.slope * MT, a_RR = f1RR.constant + f1RR.slope * MT;
    const double b_LL = f2LL.constant + f2LL.slope * MT, b_LR = f2LR.constant + f2LR.slope * MT, b_RL = f2RL.constant + f2RL.slope * MT, b_RR = f2RR.constant + f2RR.slope * MT;
    logdN1 = (a_LL * (YR - Y) + a_RL * (Y - YL)) * (P1R - Phip1) + (a_LR * (YR - Y) + a_RR * (Y - YL)) * (Phip1 - P1L);
    logdN1 /= (dY * dPhip1);
    logdN2 = (b_LL * (YR - Y) + b_RL * (Y - YL)) * (P2R - Phip2) + (b_LR * (YR - Y) + b_RR * (Y - YL)) * (Phip2 - P2L);
    logdN2 /= (dY * dPhip2);
    if constexpr (SPIN) {
      const int im = npT - 1;
      for (int c = 0; c < 3; c++) {
#define SG(ip, iy) Sstar[3 * (im + npT * ((ip) + nphi * (iy))) + c]
        so->S1[c] = ((SG(i1L, iYL) * (YR - Y) + SG(i1L, iYR) * (Y - YL)) * (P1R - Phip1) + (SG(i1R, iYL) * (YR - Y) + SG(i1R, iYR) * (Y - YL)) * (Phip1 - P1L)) / (dY * dPhip1);
        so->S2[c] = ((SG(i2L, iYL) * (YR - Y) + SG(i2L, iYR) * (Y - YL)) * (P2R - Phip2) + (SG(i2R, iYL) * (YR - Y) + SG(i2R, iYR) * (Y - YL)) * (Phip2 - P2L)) / (dY * dPhip2);
#undef SG
      }
    }
  }
  if constexpr (SPIN) { so->e1 = exp(logdN1); so->e2 = exp(logdN2); return 0.0; }
  return (exp(logdN1) + exp(logdN2));
}

// Polarization feed-down: per-thread context of the daughter spin at a point of the 2-body integral (see daughter_spin)
struct SpinCtx {
  const double *Sstar;           // parent rest-frame spin table [bins][3]
  double M, mD, a, b;            // mass_parent of the term, daughter mass, transfer law s* = a S*_P + b (S*_P.n) n
  double E, px, py, pz;          // the bin's four-momentum (daughter)
  double Y;                      // parent rapidity at the current v node (y + v DeltaY; 2+1D: v DeltaY)
  int dim;
};

// Weak-decay feed-down (is3d_b200_polarization_weak_decays): the Lee-Yang law of 1/2 -> 1/2 + 0 in place of (a, b).  a and b are unused.
struct WeakCtx : SpinCtx {
  double alpha, beta, gamma;     // decay parameters of the term
};

// Spin four-vector S_D (lab) of the daughter at one integrand point: parent P = (MT cosh Y, PT cos Phi, PT sin Phi, MT sinh Y) with
// rest-frame spin Sp (2+1D: Sp is the y = 0 table value, its four-vector is boosted longitudinally by Y first), p* = L(P)^-1 p,
// n = p*/|p*|, s* = a Sp + b (Sp.n) n in the daughter's rest frame, then back through L(P).  All boosts are pure boosts.
// WeakCtx: s* is the Lee-Yang numerator (alpha/2 + Sp.n) n + beta Sp x n + gamma (Sp - (Sp.n) n), and *yield = 1 + 2 alpha Sp.n.
template <class Ctx>
__device__ __forceinline__ void daughter_spin(const Ctx &c, double MT, double PT, double Phi, const double Sp[3], double out[4], double *yield = nullptr)
{
  const double M = c.M, chY = cosh(c.Y), shY = sinh(c.Y);
  const double Px = PT * cos(Phi), Py = PT * sin(Phi), Pz = MT * shY, EP = MT * chY;
  double S[3] = {Sp[0], Sp[1], Sp[2]};
  if (c.dim == 2) {                                  // four-vector at (MT, Px, Py, 0), boost by Y, rest-frame part w.r.t. L(P)
    const double P0S = Px * Sp[0] + Py * Sp[1];
    const double s0t = P0S / M, k = P0S / (M * (MT + M));
    const double sx = Sp[0] + k * Px, sy = Sp[1] + k * Py;
    const double st = s0t * chY + Sp[2] * shY, sz = s0t * shY + Sp[2] * chY;
    const double r = st / (EP + M);
    S[0] = sx - r * Px; S[1] = sy - r * Py; S[2] = sz - r * Pz;
  }
  const double Pp = Px * c.px + Py * c.py + Pz * c.pz;
  const double pst = (EP * c.E - Pp) / M, kp = Pp / (M * (EP + M)) - c.E / M;
  const double ps[3] = {c.px + kp * Px, c.py + kp * Py, c.pz + kp * Pz};
  const double ip = 1.0 / sqrt(ps[0] * ps[0] + ps[1] * ps[1] + ps[2] * ps[2]);
  const double n[3] = {ps[0] * ip, ps[1] * ip, ps[2] * ip};
  const double Sn = S[0] * n[0] + S[1] * n[1] + S[2] * n[2];
  double s[3];
  if constexpr (std::is_same<Ctx, WeakCtx>::value) {
    const double l = 0.5 * c.alpha + Sn;
    const double x[3] = {S[1] * n[2] - S[2] * n[1], S[2] * n[0] - S[0] * n[2], S[0] * n[1] - S[1] * n[0]};    // Sp x n
    for (int k = 0; k < 3; k++) s[k] = l * n[k] + c.beta * x[k] + c.gamma * (S[k] - Sn * n[k]);
    *yield = 1.0 + 2.0 * c.alpha * Sn;
  } else {
    s[0] = c.a * S[0] + c.b * Sn * n[0]; s[1] = c.a * S[1] + c.b * Sn * n[1]; s[2] = c.a * S[2] + c.b * Sn * n[2];
  }
  const double pss = ps[0] * s[0] + ps[1] * s[1] + ps[2] * s[2];
  const double q0 = pss / c.mD, kq = pss / (c.mD * (pst + c.mD));
  const double q[3] = {s[0] + kq * ps[0], s[1] + kq * ps[1], s[2] + kq * ps[2]};
  const double Pq = Px * q[0] + Py * q[1] + Pz * q[2];
  const double kk = Pq / (M * (EP + M)) + q0 / M;
  out[0] = (EP * q0 + Pq) / M;
  out[1] = q[0] + kk * Px; out[2] = q[1] + kk * Py; out[3] = q[2] + kk * Pz;
}

// zeta integral at fixed (v [, s]): the innermost loop of the four integration routines (:588-628, 753-784, 1183-1213, 1352-1380).
// SPIN: instead, zs[mu] += w_zeta MT (exp(log dN_1) S_D^mu(Phi_1) + exp(log dN_2) S_D^mu(Phi_2)) at the same points; with a WeakCtx also
// zs[4] += w_zeta MT (exp(log dN_1) yield(Phi_1) + exp(log dN_2) yield(Phi_2)).
template <bool SPIN, class Ctx = SpinCtx>
__device__ double zeta_integral_at(const ParentView &P, double MTbar, double DeltaMT, double mTc_over_pT, double Estar_M_over_pT, double parent_mass2,
                                   double phip, int dim, bool cutoff_Y, int iYL, int iYR, double YL, double YR, double Y,
                                   const Ctx *sc = nullptr, double *zs = nullptr)
{
  const double two_Pi = 2.0 * M_PI;
  double zeta_integral = 0.0;
  if (cutoff_Y) return zeta_integral;
  for (int izeta = 0; izeta < GP; izeta++) {
    const double coszeta = cos((M_PI / 2.0) * (1.0 + kGLRoot[izeta]));
    const double MT = MTbar + (DeltaMT * coszeta);
    const double PT = sqrt(MT * MT - parent_mass2);
    const double cosPhip_tilde = (MT * mTc_over_pT - Estar_M_over_pT) / PT;
    const double Phip_tilde = acos(cosPhip_tilde);
    double Phip_1 = fmod(Phip_tilde + phip, two_Pi), Phip_2 = fmod(-Phip_tilde + phip, two_Pi);
    if (Phip_1 < 0.0) Phip_1 += two_Pi;
    if (Phip_2 < 0.0) Phip_2 += two_Pi;
    if constexpr (SPIN) {
      SpinOut so;
      if (dim == 2) parent_2d<true>(P, MT, Phip_1, Phip_2, sc->Sstar, &so);
      else parent_3d<true>(P, iYL, iYR, YL, YR, MT, Phip_1, Phip_2, Y, sc->Sstar, &so);
      double S1[4], S2[4];
      if constexpr (std::is_same<Ctx, WeakCtx>::value) {
        double y1, y2;
        daughter_spin(*sc, MT, PT, Phip_1, so.S1, S1, &y1);
        daughter_spin(*sc, MT, PT, Phip_2, so.S2, S2, &y2);
        const double w1 = MT * so.e1, w2 = MT * so.e2;
        for (int mu = 0; mu < 4; mu++) zs[mu] += (kGLWeight[izeta] * (w1 * S1[mu] + w2 * S2[mu]));
        zs[4] += (kGLWeight[izeta] * (w1 * y1 + w2 * y2));
      } else {
        daughter_spin(*sc, MT, PT, Phip_1, so.S1, S1);
        daughter_spin(*sc, MT, PT, Phip_2, so.S2, S2);
        const double w1 = MT * so.e1, w2 = MT * so.e2;
        for (int mu = 0; mu < 4; mu++) zs[mu] += (kGLWeight[izeta] * (w1 * S1[mu] + w2 * S2[mu]));
      }
    } else {
      const double integrand = MT * (dim == 2 ? parent_2d<false>(P, MT, Phip_1, Phip_2) : parent_3d<false>(P, iYL, iYR, YL, YR, MT, Phip_1, Phip_2, Y));
      zeta_integral += (kGLWeight[izeta] * integrand);
    }
  }
  return zeta_integral;
}

__device__ __forceinline__ bool y_points(const DecayGrid &G, double Y, double Ymax, int &iYL, int &iYR, double &YL, double &YR)
{
  if (fabs(Y) <= Ymax) {
    int r = 1;
    while (Y > G.y[r]) r++;
    iYR = r; iYL = r - 1; YL = G.y[iYL]; YR = G.y[iYR];
    return false;
  }
  return true;                                           // parent rapidity outside the table: cut off (:735-738)
}

__device__ __forceinline__ ParentView parent_view(const DecayGrid &G, const double *logdN, const double *MT_all, const Fit *fit_all, int term)
{
  ParentView P;
  P.logdN = logdN; P.MT = MT_all + (size_t)term * G.n_pT; P.fit = fit_all + (size_t)term * G.y_pts * G.n_phi;
  P.phi = G.phi; P.y = G.y; P.n_pT = G.n_pT; P.n_phi = G.n_phi; P.MTmax = P.MT[G.n_pT - 1];
  return P;
}

// The per-bin set-up and the kinematics of one v node of the 2-body integral (:521-806), shared by decay2_kernel and
// decay2_spin_kernel.  Macros rather than functions: the statements then compile in decay2_kernel exactly as they always have.
#define TWO_BODY_BIN_SETUP                                                                                                             \
  const double mass_parent = T.mass_parent, parent_mass2 = mass_parent * mass_parent;                                                 \
  const double Estar = T.Estar, Estar2 = Estar * Estar, pstar = T.pstar, Estar_M = Estar * mass_parent;                              \
  const double pT = G.pT[ipT], pT2 = pT * pT, mT2 = pT2 + T.mass2, mT = sqrt(mT2);                                                    \
  const double M_pT = mass_parent * pT, Estar_M_mT = Estar_M * mT, Estar_M_over_pT = Estar_M / pT, Estar2_plus_pT2 = Estar2 + pT2;  \
  const double DeltaY = log((pstar + sqrt(Estar2_plus_pT2)) / mT);                                                                    \
  const double phip = G.phi[iphip], y = (G.dim == 2) ? 0.0 : G.y[iy];                                                                 \
  const double Ymax = (G.dim == 2) ? 0.0 : fabs(G.y[G.y_pts - 1]);
#define TWO_BODY_V_NODE                                                                                                                \
    const double v = kGLRoot[iv];                                                                                                      \
    int iYL = 0, iYR = 0; double YL = 0.0, YR = 0.0, Y = 0.0; bool cutoff_Y = false;                                                  \
    if (G.dim == 3) { Y = y + v * DeltaY; cutoff_Y = y_points(G, Y, Ymax, iYL, iYR, YL, YR); }                                         \
    const double coshvDeltaY = cosh(v * DeltaY);                                                                                       \
    const double mT2_coshvDeltaY2 = mT2 * coshvDeltaY * coshvDeltaY;                                                                   \
    const double den = mT2_coshvDeltaY2 - pT2;                                                                                         \
    const double MTbar = Estar_M_mT * coshvDeltaY / den;                                                                               \
    const double DeltaMT = M_pT * sqrt(fabs(Estar2_plus_pT2 - mT2_coshvDeltaY2)) / den;                                                \
    const double mTc = mT * coshvDeltaY / pT;                                                                                          \
    const double vw = DeltaY * kGLWeight[iv] / sqrt(fabs(den));

// EmissionFunctionArray::two_body_decay, integration part (:521-806): one thread per (term, bin)
__global__ void __launch_bounds__(128) decay2_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const int *__restrict__ term_ids, int n_terms2,
                                                    const double *__restrict__ logdN, const double *__restrict__ MT_all, const Fit *__restrict__ fit_all,
                                                    double *__restrict__ scratch)
{
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)n_terms2 * n_bins) return;
  const int it = (int)(gid / n_bins), bin = (int)(gid - (int64_t)it * n_bins);
  const int term = term_ids[it];
  const DecayTerm T = terms[term];
  const int ipT = bin % G.n_pT, iphip = (bin / G.n_pT) % G.n_phi, iy = bin / (G.n_pT * G.n_phi);
  const ParentView P = parent_view(G, logdN, MT_all, fit_all, term);
  TWO_BODY_BIN_SETUP
  double decay2D_integral = 0.0;
  for (int iv = 0; iv < GP; iv++) {
    TWO_BODY_V_NODE
    const double zi = zeta_integral_at<false>(P, MTbar, DeltaMT, mTc, Estar_M_over_pT, parent_mass2, phip, G.dim, cutoff_Y, iYL, iYR, YL, YR, Y);
    decay2D_integral += (vw * zi);
  }
  scratch[(size_t)term * n_bins + bin] = T.prefactor * decay2D_integral;
}

// ---- polarization feed-down (is3d_b200_polarization_decays)
struct SpinLaw { double a, b; };       // per term; only 2-body terms listed in spin_ids have one

// the parent's rest-frame mean spin S*_P = (N^i - N^t p^i / (E + m)) / Snorm on its own bins, physical mass m; 0 where log Snorm is not
// finite.  S: the five arrays [St | Sx | Sy | Sz | Snorm], each n_total long.  Sstar[3 * i + c], i = ipT + n_pT (iphi + n_phi iy).
__global__ void spin_table_kernel(DecayGrid G, const double *__restrict__ S, int64_t n_total, int parent, double mass, double *__restrict__ Sstar)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = G.n_pT * G.n_phi * G.y_pts;
  if (i >= n) return;
  const int ipT = i % G.n_pT, iphi = (i / G.n_pT) % G.n_phi, iy = i / (G.n_pT * G.n_phi);
  const int64_t k = (int64_t)parent + (int64_t)G.n_species * i;
  const double sn = S[4 * n_total + k];
  double out[3] = {0.0, 0.0, 0.0};
  if (isfinite(log(sn))) {
    const double pT = G.pT[ipT], phi = G.phi[iphi], y = (G.dim == 2) ? 0.0 : G.y[iy];
    const double mT = sqrt(pT * pT + mass * mass), E = mT * cosh(y);
    const double p[3] = {pT * cos(phi), pT * sin(phi), mT * sinh(y)};
    const double r = S[k] / (E + mass);
    for (int c = 0; c < 3; c++) out[c] = (S[(c + 1) * n_total + k] - r * p[c]) / sn;
  }
  for (int c = 0; c < 3; c++) Sstar[3 * i + c] = out[c];
}

// one thread per (term with a transfer law, bin): spin_scratch[term][mu][bin] = prefactor x integral of spectrum x S_D^mu
__global__ void __launch_bounds__(128) decay2_spin_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const SpinLaw *__restrict__ laws,
                                                         const int *__restrict__ spin_ids, int n_spin, const double *__restrict__ logdN,
                                                         const double *__restrict__ MT_all, const Fit *__restrict__ fit_all,
                                                         const double *__restrict__ Sstar, double *__restrict__ spin_scratch)
{
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)n_spin * n_bins) return;
  const int it = (int)(gid / n_bins), bin = (int)(gid - (int64_t)it * n_bins);
  const int term = spin_ids[it];
  const DecayTerm T = terms[term];
  const int ipT = bin % G.n_pT, iphip = (bin / G.n_pT) % G.n_phi, iy = bin / (G.n_pT * G.n_phi);
  const ParentView P = parent_view(G, logdN, MT_all, fit_all, term);
  TWO_BODY_BIN_SETUP
  SpinCtx sc;
  sc.Sstar = Sstar; sc.a = laws[term].a; sc.b = laws[term].b; sc.M = mass_parent; sc.mD = sqrt(T.mass2); sc.dim = G.dim;
  sc.E = mT * cosh(y); sc.px = pT * cos(phip); sc.py = pT * sin(phip); sc.pz = mT * sinh(y);
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int iv = 0; iv < GP; iv++) {
    TWO_BODY_V_NODE
    sc.Y = y + v * DeltaY;
    double zs[4] = {0.0, 0.0, 0.0, 0.0};
    zeta_integral_at<true>(P, MTbar, DeltaMT, mTc, Estar_M_over_pT, parent_mass2, phip, G.dim, cutoff_Y, iYL, iYR, YL, YR, Y, &sc, zs);
    for (int mu = 0; mu < 4; mu++) acc[mu] += (vw * zs[mu]);
  }
  for (int mu = 0; mu < 4; mu++) spin_scratch[((size_t)term * 4 + mu) * n_bins + bin] = T.prefactor * acc[mu];
}

// N^mu[daughter] += spin_scratch[term][mu], terms with a law in (channel, group) order
__global__ void spin_add_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const int *__restrict__ has_law, int n_terms,
                                const double *__restrict__ spin_scratch, double *__restrict__ S, int64_t n_total)
{
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int bin = blockIdx.x * blockDim.x + threadIdx.x;
  if (bin >= n_bins) return;
  for (int t = 0; t < n_terms; t++) {
    if (!has_law[t]) continue;
    const int64_t k = (int64_t)terms[t].daughter + (int64_t)G.n_species * bin;
    for (int mu = 0; mu < 4; mu++) S[mu * n_total + k] += spin_scratch[((size_t)t * 4 + mu) * n_bins + bin];
  }
}

// ---- weak-decay feed-down (is3d_b200_polarization_weak_decays)
struct WeakLaw { double alpha, beta, gamma; };     // per term; only terms listed in weak_ids have one

// one thread per (weak term with the Lee-Yang law, bin): weak_scratch[term][r][bin], r = N^t, N^x, N^y, N^z, Snorm: prefactor x the
// integral of spectrum x (Lee-Yang numerator carried to the lab, and the yield 1 + 2 alpha S*_P.n)
__global__ void __launch_bounds__(128) decay2_weak_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const WeakLaw *__restrict__ laws,
                                                         const int *__restrict__ weak_ids, int n_weak, const double *__restrict__ logdN,
                                                         const double *__restrict__ MT_all, const Fit *__restrict__ fit_all,
                                                         const double *__restrict__ Sstar, double *__restrict__ weak_scratch)
{
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)n_weak * n_bins) return;
  const int it = (int)(gid / n_bins), bin = (int)(gid - (int64_t)it * n_bins);
  const int term = weak_ids[it];
  const DecayTerm T = terms[term];
  const int ipT = bin % G.n_pT, iphip = (bin / G.n_pT) % G.n_phi, iy = bin / (G.n_pT * G.n_phi);
  const ParentView P = parent_view(G, logdN, MT_all, fit_all, term);
  TWO_BODY_BIN_SETUP
  WeakCtx sc;
  sc.Sstar = Sstar; sc.a = 0.0; sc.b = 0.0; sc.M = mass_parent; sc.mD = sqrt(T.mass2); sc.dim = G.dim;
  sc.alpha = laws[term].alpha; sc.beta = laws[term].beta; sc.gamma = laws[term].gamma;
  sc.E = mT * cosh(y); sc.px = pT * cos(phip); sc.py = pT * sin(phip); sc.pz = mT * sinh(y);
  double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  for (int iv = 0; iv < GP; iv++) {
    TWO_BODY_V_NODE
    sc.Y = y + v * DeltaY;
    double zs[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    zeta_integral_at<true, WeakCtx>(P, MTbar, DeltaMT, mTc, Estar_M_over_pT, parent_mass2, phip, G.dim, cutoff_Y, iYL, iYR, YL, YR, Y, &sc, zs);
    for (int r = 0; r < 5; r++) acc[r] += (vw * zs[r]);
  }
  for (int r = 0; r < 5; r++) weak_scratch[((size_t)term * 5 + r) * n_bins + bin] = T.prefactor * acc[r];
}

// terms in row order: a term with the law adds its five rows to [St | Sx | Sy | Sz | Snorm] of the daughter, any other term its
// plain integral (scratch, decay2_kernel) to Snorm
__global__ void weak_add_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const int *__restrict__ has_law, int n_terms,
                                const double *__restrict__ scratch, const double *__restrict__ weak_scratch, double *__restrict__ S, int64_t n_total)
{
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int bin = blockIdx.x * blockDim.x + threadIdx.x;
  if (bin >= n_bins) return;
  for (int t = 0; t < n_terms; t++) {
    const int64_t k = (int64_t)terms[t].daughter + (int64_t)G.n_species * bin;
    if (has_law[t]) for (int r = 0; r < 5; r++) S[r * n_total + k] += weak_scratch[((size_t)t * 5 + r) * n_bins + bin];
    else S[4 * n_total + k] += scratch[(size_t)t * n_bins + bin];
  }
}

// EmissionFunctionArray::three_body_decay, integration part (:1048-1398): 12 threads per (term, bin), one per s node
constexpr int kBins3 = 8;               // bins per block of decay3_kernel
__global__ void __launch_bounds__(GP * kBins3) decay3_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, const int *__restrict__ term_ids, int n_terms3,
                                                            const double *__restrict__ logdN, const double *__restrict__ MT_all, const Fit *__restrict__ fit_all,
                                                            double *__restrict__ scratch)
{
  __shared__ double part[kBins3][GP];
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int is = threadIdx.x, lb = threadIdx.y;
  const int64_t gid = (int64_t)blockIdx.x * kBins3 + lb;
  const bool valid = gid < (int64_t)n_terms3 * n_bins;
  int term = 0, bin = 0;
  double contrib = 0.0, prefactor = 0.0;
  if (valid) {
    const int it = (int)(gid / n_bins);
    bin = (int)(gid - (int64_t)it * n_bins);
    term = term_ids[it];
    const DecayTerm T = terms[term];
    prefactor = T.prefactor;
    const int ipT = bin % G.n_pT, iphip = (bin / G.n_pT) % G.n_phi, iy = bin / (G.n_pT * G.n_phi);
    const ParentView P = parent_view(G, logdN, MT_all, fit_all, term);
    const double mass_parent = T.mass_parent, parent_mass2 = mass_parent * mass_parent, mass_1_squared = T.m1sq;
    const double s = T.s_minus + (T.s_plus - T.s_minus) * (1.0 + kGLRoot[is]) / 2.0;
    const double s_integrand_weight = kGLWeight[is] * sqrt(fabs((s - T.s_minus) * (s - T.d))) / s;
    const double Estar = (parent_mass2 + mass_1_squared - s) / (2.0 * mass_parent), Estar2 = Estar * Estar;
    const double pstar = sqrt(Estar * Estar - mass_1_squared);
    const double pT = G.pT[ipT], pT2 = pT * pT, mT2 = pT2 + mass_1_squared, mT = sqrt(mT2);
    const double M_pT = mass_parent * pT, M_mT = mass_parent * mT, M_over_pT = mass_parent / pT, mT_over_pT = mT / pT;
    const double Estar_M_mT = Estar * M_mT, Estar2_plus_pT2 = Estar2 + pT2, Estar_M_over_pT = Estar * M_over_pT;
    const double DeltaY = log((pstar + sqrt(Estar2_plus_pT2)) / mT);
    const double phip = G.phi[iphip], y = (G.dim == 2) ? 0.0 : G.y[iy];
    const double Ymax = (G.dim == 2) ? 0.0 : fabs(G.y[G.y_pts - 1]);
    double v_integral = 0.0;
    for (int iv = 0; iv < GP; iv++) {
      const double v = kGLRoot[iv];
      int iYL = 0, iYR = 0; double YL = 0.0, YR = 0.0, Y = 0.0; bool cutoff_Y = false;
      if (G.dim == 3) { Y = y + v * DeltaY; cutoff_Y = y_points(G, Y, Ymax, iYL, iYR, YL, YR); }
      const double coshvDeltaY = cosh(v * DeltaY);
      // the boost-invariant branch multiplies mT^2 cosh cosh left to right (:1167), the 3+1D branch squares cosh first (:1329-1330)
      const double mT2_coshvDeltaY2 = (G.dim == 2) ? mT2 * coshvDeltaY * coshvDeltaY : mT2 * (coshvDeltaY * coshvDeltaY);
      const double den = mT2_coshvDeltaY2 - pT2;
      const double mTc = mT_over_pT * coshvDeltaY;
      const double MTbar = Estar_M_mT * coshvDeltaY / den;
      const double DeltaMT = M_pT * sqrt(fabs(Estar2_plus_pT2 - mT2_coshvDeltaY2)) / den;
      const double vw = DeltaY * kGLWeight[iv] / sqrt(fabs(den));
      const double zi = zeta_integral_at<false>(P, MTbar, DeltaMT, mTc, Estar_M_over_pT, parent_mass2, phip, G.dim, cutoff_Y, iYL, iYR, YL, YR, Y);
      v_integral += vw * zi;
    }
    contrib = s_integrand_weight * v_integral;
  }
  part[lb][is] = contrib;
  __syncthreads();
  if (valid && is == 0) {
    double decay3D_integral = 0.0;
    for (int k = 0; k < GP; k++) decay3D_integral += part[lb][k];          // s nodes in order, like the reference's loop
    scratch[(size_t)term * n_bins + bin] = prefactor * decay3D_integral;
  }
}

// dN[daughter] += scratch[term], terms in (channel, group) order
__global__ void decay_add_kernel(DecayGrid G, const DecayTerm *__restrict__ terms, int n_terms, const double *__restrict__ scratch, double *__restrict__ dN)
{
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  const int bin = blockIdx.x * blockDim.x + threadIdx.x;
  if (bin >= n_bins) return;
  for (int t = 0; t < n_terms; t++) dN[(int64_t)terms[t].daughter + (int64_t)G.n_species * bin] += scratch[(size_t)t * n_bins + bin];
}

// calculate_Q_factor, :99-121
double q_factor(double mass_parent, double mass_1, double mass_2, double mass_3)
{
  static const double x_root[24] = {-0.99518721999702,-0.97472855597131,-0.93827455200273,-0.8864155270044,-0.8200019859739,-0.74012419157855,-0.64809365193698,-0.54542147138884,-0.43379350762605,-0.31504267969616,-0.19111886747362,-0.064056892862606,0.06405689286261,0.19111886747362,0.31504267969616,0.43379350762605,0.54542147138884,0.64809365193698,0.74012419157855,0.8200019859739,0.8864155270044,0.93827455200273,0.97472855597131,0.99518721999702};
  static const double x_weight[24] = {0.01234122979999,0.02853138862893,0.0442774388174,0.059298584915437,0.0733464814111,0.08619016153195,0.0976186521041,0.107444270116,0.11550566805373,0.1216704729278,0.12583745634683,0.1279381953468,0.1279381953468,0.1258374563468,0.1216704729278,0.1155056680537,0.107444270116,0.09761865210411,0.08619016153195,0.07334648141108,0.05929858491544,0.04427743881742,0.02853138862893,0.01234122979999};
  const double a = (mass_parent + mass_1) * (mass_parent + mass_1), b = (mass_parent - mass_1) * (mass_parent - mass_1);
  const double c = (mass_2 + mass_3) * (mass_2 + mass_3), d = (mass_2 - mass_3) * (mass_2 - mass_3);
  double Q = 0.0;
  for (int i = 0; i < 24; i++) {
    const double s = c + (b - c) * (1.0 + x_root[i]) / 2.0;
    Q += x_weight[i] * (b - c) * std::sqrt(std::fabs((a - s) * (b - s) * (s - c) * (s - d))) / (2.0 * s);
  }
  return Q;
}

struct Host {                       // bookkeeping helpers, all on the host and in integers / the reference's scalar order
  const is3d_particle_list *pdg; int n_chosen; const int32_t *chosen;
  int particle_index(int mc_id, std::string *err) const                           // :59-79
  {
    if (mc_id == 0) { *err = "a decay product has mc_id 0 (null particle in the particle list)"; return -1; }
    for (int i = 0; i < pdg->n_particles; i++) if (pdg->mcid[i] == mc_id) return i;
    *err = "decay product " + std::to_string(mc_id) + " is not in the particle list"; return -1;
  }
  int chosen_index(int pdg_index, std::string *err) const                          // :82-97
  {
    for (int i = 0; i < n_chosen; i++) if (chosen[i] == pdg_index) return i;
    *err = "daughter is not a chosen particle"; return -1;
  }
  // daughters that are chosen species, grouped by type in order of first appearance (:307-371, 828-899)
  int group(const int *prod, int nprod, int *groups, int *members) const
  {
    bool found[3] = {false, false, false};
    for (int ic = 0; ic < n_chosen; ic++) {
      bool all = true;
      for (int k = 0; k < nprod; k++) { if (prod[k] == chosen[ic] && !found[k]) found[k] = true; all = all && found[k]; }
      if (all) break;
    }
    int ng = 0;
    for (int k = 0; k < nprod; k++) {
      if (!found[k]) continue;
      bool put = false;
      for (int gi = 0; gi < ng; gi++) if (prod[k] == groups[gi]) { members[gi] += 1; put = true; break; }
      if (!put) { groups[ng] = prod[k]; members[ng] = 1; ng++; }
    }
    return ng;
  }
};

// Transfer law (a', b') of a 2-body channel parent -> daughter + partner for the spin-1/2-normalised arrays (include/is3d_b200.h):
// s*_D = a' S*_P + b' (S*_P.n) n.  false: no law (the channel only dilutes).
bool transfer_law(const is3d_particle_list *pdg, const int32_t *spin2, const int32_t *parity, int parent, int daughter, int partner,
                  double *a, double *b)
{
  if (spin2[daughter] != 1) return false;
  const int jp2 = spin2[parent];
  if (std::abs(pdg->mcid[partner]) == 22) {                  // 1/2 -> 1/2 + photon: only the longitudinal part survives
    if (jp2 != 1) return false;
    *a = 0.0; *b = -1.0; return true;
  }
  if (spin2[partner] != 0 || jp2 % 2 != 1) return false;
  const int pp = parity[parent], pd = parity[daughter], pm = parity[partner];
  if (pp == 0 || pd == 0 || pm == 0) return false;
  const int sign_j = (((jp2 - 1) / 2) % 2 == 0) ? 1 : -1;     // (-1)^(J_P - 1/2)
  const double eta = (double)(-sign_j * pp * pd * pm);
  *a = -eta * (double)(jp2 + 1) / 2.0;
  *b = 1.0 - *a;
  return true;
}

// the set-up half of two_body_decay for one daughter group (:296-460): daughter = its chosen index, members = its multiplicity in the
// channel, mass_secondary = the mass of the channel's second product (the recoil mass for either daughter, :411-413)
DecayTerm two_body_term(int daughter, int members, double mass_parent, double mass, double mass_secondary, double branch_ratio)
{
  DecayTerm T; memset(&T, 0, sizeof(T));
  T.body = 2; T.daughter = daughter;
  const double W2 = mass_secondary * mass_secondary;
  const double Estar = (mass_parent * mass_parent + mass * mass - W2) / (2.0 * mass_parent);
  T.mass_parent = mass_parent; T.mass2 = mass * mass; T.Estar = Estar; T.pstar = std::sqrt(Estar * Estar - mass * mass);
  T.prefactor = (double)members * mass_parent * branch_ratio / (8.0 * T.pstar);
  return T;
}

bool ck(cudaError_t e, const char *what, std::string *err)
{
  if (e != cudaSuccess) { *err = std::string(what) + ": " + cudaGetErrorString(e); return false; }
  return true;
}

// device buffers of one feed-down call, freed on every path out of the driver
struct DecayBuffers {
  double *tables = nullptr, *logdN = nullptr, *MT = nullptr, *scratch = nullptr; Fit *fit = nullptr; DecayTerm *terms = nullptr; int *ids = nullptr, *error = nullptr;
  double *Sstar = nullptr, *spin_scratch = nullptr; SpinLaw *laws = nullptr; int *spin_ids = nullptr;
  WeakLaw *weak_laws = nullptr; double *weak_scratch = nullptr;
  ~DecayBuffers() { cudaFree(tables); cudaFree(logdN); cudaFree(MT); cudaFree(scratch); cudaFree(fit); cudaFree(terms); cudaFree(ids); cudaFree(error);
                    cudaFree(Sstar); cudaFree(spin_scratch); cudaFree(laws); cudaFree(spin_ids); cudaFree(weak_laws); cudaFree(weak_scratch); }
};

// G from the grid, the buffers every driver needs for up to max_terms terms per parent, the momentum tables uploaded and the tail-fit
// flag cleared on st
int decay_setup(const is3d_grid *gr, int dimension, int n_chosen, int max_terms, DecayGrid *Gp, DecayBuffers *B, cudaStream_t st, std::string *err)
{
  DecayGrid &G = *Gp; memset(&G, 0, sizeof(G));
  G.n_species = n_chosen; G.n_pT = gr->n_pT; G.n_phi = gr->n_phi; G.n_y_tab = gr->n_y; G.dim = dimension;
  G.y_pts = (dimension == 2) ? 1 : gr->n_y;
  if (G.n_pT < 2 || G.n_phi < 2 || (dimension == 3 && G.y_pts < 2)) { *err = "momentum tables too short for the interpolation"; return IS3D_ERR_ARGUMENT; }
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  if (!ck(cudaMalloc(&B->tables, sizeof(double) * (size_t)(G.n_pT + G.n_phi + G.n_y_tab + 8)), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->logdN, sizeof(double) * (size_t)n_bins), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->MT, sizeof(double) * (size_t)max_terms * G.n_pT), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->fit, sizeof(Fit) * (size_t)max_terms * G.y_pts * G.n_phi), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->scratch, sizeof(double) * (size_t)max_terms * n_bins), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->terms, sizeof(DecayTerm) * (size_t)max_terms), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->ids, sizeof(int) * (size_t)max_terms * 2), "cudaMalloc", err) ||
      !ck(cudaMalloc(&B->error, sizeof(int)), "cudaMalloc", err)) return IS3D_ERR_CUDA;
  if (!ck(cudaMemcpyAsync(B->tables, gr->pT, sizeof(double) * G.n_pT, cudaMemcpyHostToDevice, st), "H2D", err) ||
      !ck(cudaMemcpyAsync(B->tables + G.n_pT, gr->phi, sizeof(double) * G.n_phi, cudaMemcpyHostToDevice, st), "H2D", err) ||
      !ck(cudaMemcpyAsync(B->tables + G.n_pT + G.n_phi, gr->y, sizeof(double) * G.n_y_tab, cudaMemcpyHostToDevice, st), "H2D", err) ||
      !ck(cudaMemsetAsync(B->error, 0, sizeof(int), st), "memset", err)) return IS3D_ERR_CUDA;
  G.pT = B->tables; G.phi = B->tables + G.n_pT; G.y = B->tables + G.n_pT + G.n_phi;
  return IS3D_OK;
}

// the tail-fit flag of decay_setup_kernel, read after the stream is done
int decay_tail_fit_status(const DecayBuffers &B, cudaStream_t st, std::string *err)
{
  int flag = 0;
  if (!ck(cudaMemcpyAsync(&flag, B.error, sizeof(int), cudaMemcpyDeviceToHost, st), "D2H", err) || !ck(cudaStreamSynchronize(st), "sync", err)) return IS3D_ERR_CUDA;
  if (flag) { *err = "not enough positive points of a parent spectrum beyond mT = 1.65 M to fit its large-mT tail (the reference exits here)"; return IS3D_ERR_ARGUMENT; }
  return IS3D_OK;
}

// the rows of a weak-decay table with particle-list indices and (alpha, beta, gamma), or IS3D_ERR_ARGUMENT for a table the entry point rejects
struct WeakRow { int parent, daughter, partner; double br; WeakLaw law; };
int weak_rows(const is3d_particle_list *pdg, const is3d_weak_decays *weak, std::vector<WeakRow> *out, std::string *err)
{
  const int n_rows = weak->n;
  std::vector<WeakRow> &rows = *out;
  rows.assign((size_t)n_rows, WeakRow());
  std::vector<double> br_sum((size_t)pdg->n_particles, 0.0);
  for (int r = 0; r < n_rows; r++) {
    WeakRow &R = rows[r];
    const int32_t ids[3] = {weak->parent[r], weak->daughter[r], weak->partner[r]};
    int *const idx[3] = {&R.parent, &R.daughter, &R.partner};
    for (int k = 0; k < 3; k++) {
      *idx[k] = -1;
      for (int i = 0; i < pdg->n_particles && ids[k] != 0; i++) if (pdg->mcid[i] == ids[k]) { *idx[k] = i; break; }
      if (*idx[k] < 0) { *err = "weak decay row " + std::to_string(r) + ": MC id " + std::to_string(ids[k]) + " is not in the particle list"; return IS3D_ERR_ARGUMENT; }
    }
    const std::string at = "weak decay row " + std::to_string(r) + ": ";
    if (!pdg->stable[R.parent] || !pdg->stable[R.daughter]) { *err = at + "parent and daughter must be stable in the particle list"; return IS3D_ERR_ARGUMENT; }
    const double br = weak->branching[r], alpha = weak->alpha[r], phi = weak->phi[r];
    if (!(br >= 0.0 && br <= 1.0)) { *err = at + "branching ratio outside [0, 1]"; return IS3D_ERR_ARGUMENT; }
    if (!std::isfinite(alpha) || !std::isfinite(phi) || std::fabs(alpha) > 1.0) { *err = at + "alpha must be finite with |alpha| <= 1, phi finite"; return IS3D_ERR_ARGUMENT; }
    if (pdg->mass[R.daughter] + pdg->mass[R.partner] >= pdg->mass[R.parent]) { *err = at + "m_daughter + m_partner >= m_parent"; return IS3D_ERR_ARGUMENT; }
    R.br = br;
    br_sum[R.parent] += br;
    if (br_sum[R.parent] > 1.0 + 1e-9) { *err = at + "the branching ratios of its parent sum to more than 1"; return IS3D_ERR_ARGUMENT; }
    const double t = std::sqrt(1.0 - alpha * alpha);
    R.law = WeakLaw{alpha, t * std::sin(phi), t * std::cos(phi)};
  }
  return IS3D_OK;
}

}  // namespace

// Polarization feed-down inputs of decays_core: 2J and parity per particle-list entry, and the length of each of the five arrays.
struct SpinFeedDown { const int32_t *spin2, *parity; int64_t n_total; };

// Host driver.  Without spin, dN_dev is the spectra [y][phi][pT][species], amended in place.  With spin, dN_dev holds the five arrays
// [St | Sx | Sy | Sz | Snorm] (n_total each); Snorm goes through exactly the launches of the spectra feed-down, and the 2-body terms with
// a transfer law add their spin integrals to St..Sz.
static int decays_core(const is3d_particle_list *pdg, int n_chosen, const int32_t *chosen, const is3d_grid *gr, int dimension,
                       double *dN_dev, const SpinFeedDown *spin, cudaStream_t st, int *launches, std::string *err)
{
  if (n_chosen - 1 <= 0) { *err = "need at least two chosen particles for the resonance decay routine"; return IS3D_ERR_ARGUMENT; }
  const int max_terms = 50 * 3;                       // <= 50 channels per particle (readindata.h Maxdecaychannel) x 3 daughter groups
  DecayGrid G; DecayBuffers B;
  { const int rc = decay_setup(gr, dimension, n_chosen, max_terms, &G, &B, st, err); if (rc != IS3D_OK) return rc; }
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  Host H{pdg, n_chosen, chosen};
  auto ck = [&](cudaError_t e, const char *what) { return is3d::ck(e, what, err); };
  if (spin && (!ck(cudaMalloc(&B.Sstar, sizeof(double) * 3 * (size_t)n_bins), "cudaMalloc") ||
               !ck(cudaMalloc(&B.spin_scratch, sizeof(double) * 4 * (size_t)max_terms * n_bins), "cudaMalloc") ||
               !ck(cudaMalloc(&B.laws, sizeof(SpinLaw) * (size_t)max_terms), "cudaMalloc") ||
               !ck(cudaMalloc(&B.spin_ids, sizeof(int) * (size_t)max_terms * 2), "cudaMalloc"))) return IS3D_ERR_CUDA;
  double *const dN_spec = spin ? dN_dev + 4 * spin->n_total : dN_dev;       // the array the spectra feed-down amends

  for (int ichosen = n_chosen - 1; ichosen > 0; ichosen--) {
    const int ipart = chosen[ichosen];
    if (pdg->stable[ipart]) continue;
    // ---- the parent's channels -> terms (host; resonance_decay_channel + the set-up halves of two_/three_body_decay)
    std::vector<DecayTerm> terms;
    std::vector<SpinLaw> laws;
    std::vector<int> has_law;
    for (int ich = 0; ich < pdg->decays[ipart]; ich++) {
      const int row = pdg->dec_first[ipart] + ich;
      const int decay_products = std::abs(pdg->dec_npart[row]);
      if (decay_products > 5) { *err = "a decay channel lists more than five products"; return IS3D_ERR_ARGUMENT; }
      int idx[5];
      for (int k = 0; k < decay_products; k++) { idx[k] = H.particle_index(pdg->dec_part[row * 5 + k], err); if (idx[k] < 0) return IS3D_ERR_ARGUMENT; }
      if (decay_products == 1 || decay_products == 4) continue;              // trivial; 4-body channels are skipped by the reference (:279-282)
      if (decay_products != 2 && decay_products != 3) { *err = "number of decay products = 0 or > 4"; return IS3D_ERR_ARGUMENT; }
      const double branch_ratio = pdg->dec_br[row];
      int groups[3], members[3];
      if (decay_products == 2) {
        double mass_parent = pdg->mass[ipart], mass_1 = pdg->mass[idx[0]], mass_2 = pdg->mass[idx[1]];
        while ((mass_1 + mass_2) > mass_parent) {                             // :241-256
          mass_parent += 0.25 * pdg->width[ipart];
          mass_1 -= 0.5 * pdg->width[idx[0]];
          mass_2 -= 0.5 * pdg->width[idx[1]];
          if (mass_1 < 0.0 || mass_2 < 0.0) { *err = "one daughter mass went negative while enforcing energy conservation"; return IS3D_ERR_ARGUMENT; }
        }
        const int ng = H.group(idx, 2, groups, members);
        for (int gi = 0; gi < ng; gi++) {
          const int daughter = H.chosen_index(groups[gi], err);
          if (daughter < 0) return IS3D_ERR_ARGUMENT;
          terms.push_back(two_body_term(daughter, members[gi], mass_parent, pdg->mass[groups[gi]], pdg->mass[idx[1]], branch_ratio));
          SpinLaw L{0.0, 0.0};
          has_law.push_back(spin && transfer_law(pdg, spin->spin2, spin->parity, ipart, groups[gi], idx[0] == groups[gi] ? idx[1] : idx[0], &L.a, &L.b));
          laws.push_back(L);
        }
      } else {
        const double mass_parent = pdg->mass[ipart];
        const int ng = H.group(idx, 3, groups, members);
        for (int gi = 0; gi < ng; gi++) {
          DecayTerm T; memset(&T, 0, sizeof(T));
          T.body = 3; T.daughter = H.chosen_index(groups[gi], err);
          if (T.daughter < 0) return IS3D_ERR_ARGUMENT;
          int rest[2], nr = 0; bool removed = false;
          for (int k = 0; k < 3; k++) { if (!removed && idx[k] == groups[gi]) { removed = true; continue; } rest[nr++] = idx[k]; }
          const double mass_1 = pdg->mass[groups[gi]], mass_2 = pdg->mass[rest[0]], mass_3 = pdg->mass[rest[1]];
          const double Q_norm = q_factor(mass_parent, mass_1, mass_2, mass_3);
          T.mass_parent = mass_parent; T.m1sq = mass_1 * mass_1;
          T.s_plus = (mass_parent - mass_1) * (mass_parent - mass_1); T.s_minus = (mass_2 + mass_3) * (mass_2 + mass_3);
          T.d = (mass_2 - mass_3) * (mass_2 - mass_3);
          T.prefactor = (double)members[gi] * (mass_parent * mass_parent) * (T.s_plus - T.s_minus) * branch_ratio / (8.0 * Q_norm);
          terms.push_back(T);
          laws.push_back(SpinLaw{0.0, 0.0}); has_law.push_back(0);                // 3-body channels only dilute
        }
      }
    }
    if (terms.empty()) continue;
    if ((int)terms.size() > max_terms) { *err = "too many decay terms for one parent"; return IS3D_ERR_ARGUMENT; }
    std::vector<int> ids2, ids3;
    for (int t = 0; t < (int)terms.size(); t++) (terms[t].body == 2 ? ids2 : ids3).push_back(t);
    std::vector<int> ids(ids2); ids.insert(ids.end(), ids3.begin(), ids3.end());
    std::vector<int> spin_ids;                                                // 2-body terms with a law, then the has_law flags
    for (int t : ids2) if (has_law[t]) spin_ids.push_back(t);
    const int n_spin = (int)spin_ids.size();
    spin_ids.insert(spin_ids.end(), has_law.begin(), has_law.end());
    // pageable host memory: these copies complete before cudaMemcpyAsync returns, so the vectors may go out of scope
    if (!ck(cudaMemcpyAsync(B.terms, terms.data(), sizeof(DecayTerm) * terms.size(), cudaMemcpyHostToDevice, st), "H2D") ||
        !ck(cudaMemcpyAsync(B.ids, ids.data(), sizeof(int) * ids.size(), cudaMemcpyHostToDevice, st), "H2D")) return IS3D_ERR_CUDA;
    if (spin && (!ck(cudaMemcpyAsync(B.laws, laws.data(), sizeof(SpinLaw) * laws.size(), cudaMemcpyHostToDevice, st), "H2D") ||
                 !ck(cudaMemcpyAsync(B.spin_ids, spin_ids.data(), sizeof(int) * spin_ids.size(), cudaMemcpyHostToDevice, st), "H2D"))) return IS3D_ERR_CUDA;
    log_parent_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, dN_spec, ichosen, B.logdN);
    decay_setup_kernel<<<(unsigned)terms.size(), 128, 0, st>>>(G, B.terms, B.logdN, B.MT, B.fit, B.error);
    *launches += 2;
    if (n_spin > 0) {                                 // the parent's arrays are final here: its own feed-down came from heavier parents
      spin_table_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, dN_dev, spin->n_total, ichosen, pdg->mass[ipart], B.Sstar);
      (*launches)++;
    }
    if (!ids2.empty()) {
      const int64_t n = (int64_t)ids2.size() * n_bins;
      decay2_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(G, B.terms, B.ids, (int)ids2.size(), B.logdN, B.MT, B.fit, B.scratch);
      (*launches)++;
    }
    if (!ids3.empty()) {
      const int64_t n = (int64_t)ids3.size() * n_bins;
      decay3_kernel<<<(unsigned)((n + kBins3 - 1) / kBins3), dim3(GP, kBins3), 0, st>>>(G, B.terms, B.ids + ids2.size(), (int)ids3.size(), B.logdN, B.MT, B.fit, B.scratch);
      (*launches)++;
    }
    if (n_spin > 0) {
      const int64_t n = (int64_t)n_spin * n_bins;
      decay2_spin_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(G, B.terms, B.laws, B.spin_ids, n_spin, B.logdN, B.MT, B.fit, B.Sstar, B.spin_scratch);
      (*launches)++;
    }
    decay_add_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, B.terms, (int)terms.size(), B.scratch, dN_spec);
    (*launches)++;
    if (n_spin > 0) {
      spin_add_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, B.terms, B.spin_ids + n_spin, (int)terms.size(), B.spin_scratch, dN_dev, spin->n_total);
      (*launches)++;
    }
    if (!ck(cudaGetLastError(), "decay kernels")) return IS3D_ERR_CUDA;
    // the term list of the next parent reuses B.terms: the stream must be done with it (also surfaces kernel faults per parent)
    if (!ck(cudaStreamSynchronize(st), "decay kernels")) return IS3D_ERR_CUDA;
  }
  return decay_tail_fit_status(B, st, err);
}

int resonance_decays_device(const is3d_particle_list *pdg, int n_chosen, const int32_t *chosen, const is3d_grid *gr, int dimension,
                            double *dN_dev, cudaStream_t st, int *launches, std::string *err)
{
  return decays_core(pdg, n_chosen, chosen, gr, dimension, dN_dev, nullptr, st, launches, err);
}

// S_dev: the five arrays [St | Sx | Sy | Sz | Snorm] on the device, n_total doubles each, amended in place
int polarization_decays_device(const is3d_particle_list *pdg, const int32_t *spin2, const int32_t *parity, int n_chosen, const int32_t *chosen,
                               const is3d_grid *gr, int dimension, double *S_dev, int64_t n_total, cudaStream_t st, int *launches, std::string *err)
{
  const SpinFeedDown spin{spin2, parity, n_total};
  return decays_core(pdg, n_chosen, chosen, gr, dimension, S_dev, &spin, st, launches, err);
}

int check_weak_decays(const is3d_particle_list *pdg, const is3d_weak_decays *weak, std::string *err)
{
  std::vector<WeakRow> rows;
  return weak_rows(pdg, weak, &rows, err);
}

// Weak-decay feed-down of the five arrays (is3d_b200_polarization_weak_decays, DESIGN §20): the rows of `weak` (rejected as by
// check_weak_decays before any device work); weak parents that are chosen species in descending mass (ties: descending chosen index), each with the 2-body set-up,
// tables and fixed-order add of decays_core.  Terms with the Lee-Yang law (2J = 1, 1, 0) go through decay2_weak_kernel, the others feed
// Snorm through decay2_kernel.
int polarization_weak_decays_device(const is3d_particle_list *pdg, const int32_t *spin2, const is3d_weak_decays *weak, int n_chosen,
                                    const int32_t *chosen, const is3d_grid *gr, int dimension, double *S_dev, int64_t n_total, cudaStream_t st,
                                    int *launches, std::string *err)
{
  Host H{pdg, n_chosen, chosen};
  std::vector<WeakRow> rows;
  { const int rc = weak_rows(pdg, weak, &rows, err); if (rc != IS3D_OK) return rc; }
  // weak parents among the chosen species, heaviest first: a parent's arrays are final when its turn comes
  std::vector<int> order;
  int max_terms = 1;
  for (int ic = 0; ic < n_chosen; ic++) {
    int nt = 0;
    for (const WeakRow &R : rows) if (R.parent == chosen[ic] && H.chosen_index(R.daughter, err) >= 0) nt++;
    if (nt > 0) { order.push_back(ic); max_terms = std::max(max_terms, nt); }
  }
  err->clear();
  if (order.empty()) return IS3D_OK;
  std::sort(order.begin(), order.end(), [&](int a, int b) {
    const double ma = pdg->mass[chosen[a]], mb = pdg->mass[chosen[b]];
    return ma != mb ? ma > mb : a > b;
  });
  DecayGrid G; DecayBuffers B;
  { const int rc = decay_setup(gr, dimension, n_chosen, max_terms, &G, &B, st, err); if (rc != IS3D_OK) return rc; }
  const int n_bins = G.n_pT * G.n_phi * G.y_pts;
  auto ck = [&](cudaError_t e, const char *what) { return is3d::ck(e, what, err); };
  if (!ck(cudaMalloc(&B.Sstar, sizeof(double) * 3 * (size_t)n_bins), "cudaMalloc") ||
      !ck(cudaMalloc(&B.weak_scratch, sizeof(double) * 5 * (size_t)max_terms * n_bins), "cudaMalloc") ||
      !ck(cudaMalloc(&B.weak_laws, sizeof(WeakLaw) * (size_t)max_terms), "cudaMalloc") ||
      !ck(cudaMalloc(&B.spin_ids, sizeof(int) * (size_t)max_terms * 2), "cudaMalloc")) return IS3D_ERR_CUDA;
  double *const Snorm = S_dev + 4 * n_total;
  for (const int ichosen : order) {
    const int ipart = chosen[ichosen];
    std::vector<DecayTerm> terms;
    std::vector<WeakLaw> laws;
    std::vector<int> has_law, plain_ids, law_ids;
    for (const WeakRow &R : rows) {
      if (R.parent != ipart) continue;
      const int daughter = H.chosen_index(R.daughter, err);
      if (daughter < 0) { err->clear(); continue; }
      const int t = (int)terms.size();
      terms.push_back(two_body_term(daughter, R.partner == R.daughter ? 2 : 1, pdg->mass[ipart], pdg->mass[R.daughter], pdg->mass[R.partner], R.br));
      laws.push_back(R.law);
      const bool law = spin2[ipart] == 1 && spin2[R.daughter] == 1 && spin2[R.partner] == 0;
      has_law.push_back(law);
      (law ? law_ids : plain_ids).push_back(t);
    }
    const int n_law = (int)law_ids.size();
    law_ids.insert(law_ids.end(), has_law.begin(), has_law.end());          // the terms with the law, then the has_law flags
    if (!ck(cudaMemcpyAsync(B.terms, terms.data(), sizeof(DecayTerm) * terms.size(), cudaMemcpyHostToDevice, st), "H2D") ||
        !ck(cudaMemcpyAsync(B.weak_laws, laws.data(), sizeof(WeakLaw) * laws.size(), cudaMemcpyHostToDevice, st), "H2D") ||
        !ck(cudaMemcpyAsync(B.spin_ids, law_ids.data(), sizeof(int) * law_ids.size(), cudaMemcpyHostToDevice, st), "H2D") ||
        (!plain_ids.empty() && !ck(cudaMemcpyAsync(B.ids, plain_ids.data(), sizeof(int) * plain_ids.size(), cudaMemcpyHostToDevice, st), "H2D")))
      return IS3D_ERR_CUDA;
    log_parent_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, Snorm, ichosen, B.logdN);
    decay_setup_kernel<<<(unsigned)terms.size(), 128, 0, st>>>(G, B.terms, B.logdN, B.MT, B.fit, B.error);
    spin_table_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, S_dev, n_total, ichosen, pdg->mass[ipart], B.Sstar);
    *launches += 3;
    if (!plain_ids.empty()) {
      const int64_t n = (int64_t)plain_ids.size() * n_bins;
      decay2_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(G, B.terms, B.ids, (int)plain_ids.size(), B.logdN, B.MT, B.fit, B.scratch);
      (*launches)++;
    }
    if (n_law > 0) {
      const int64_t n = (int64_t)n_law * n_bins;
      decay2_weak_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(G, B.terms, B.weak_laws, B.spin_ids, n_law, B.logdN, B.MT, B.fit, B.Sstar,
                                                                     B.weak_scratch);
      (*launches)++;
    }
    weak_add_kernel<<<(n_bins + 255) / 256, 256, 0, st>>>(G, B.terms, B.spin_ids + n_law, (int)terms.size(), B.scratch, B.weak_scratch, S_dev, n_total);
    (*launches)++;
    if (!ck(cudaGetLastError(), "weak decay kernels")) return IS3D_ERR_CUDA;
    if (!ck(cudaStreamSynchronize(st), "weak decay kernels")) return IS3D_ERR_CUDA;
  }
  return decay_tail_fit_status(B, st, err);
}

}  // namespace is3d
