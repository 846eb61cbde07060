// cf_polzn.cuh -- Milne -> Cartesian conversion of the spin-polarization inputs (cf_polzn.cu, cf_polzn_xi.cu, cf_polzn_she.cu).
//
// The functions read covariant Milne components (an eta index carries a factor tau) at space-time rapidity eta and return covariant
// Cartesian lab components, with the Jacobian d tau/dt = ch, d tau/dz = -sh, d eta/dt = -sh/tau, d eta/dz = ch/tau (ch = cosh eta,
// sh = sinh eta).  They are the single place to change if a surface writer uses another convention.
#pragma once

namespace is3d {

constexpr double kHbarC = 0.197327053;     // GeV fm

// Covariant Milne components (varpi_{tau x}, varpi_{tau y}, varpi_{tau eta}, varpi_{xy}, varpi_{x eta}, varpi_{y eta}) at space-time
// rapidity eta -> e = (varpi_tx, varpi_ty, varpi_tz) and omega = (varpi_yz, varpi_zx, varpi_xy), Cartesian lab components:
//   varpi_tx = ch varpi_taux + (sh/tau) varpi_xeta    varpi_zx = -sh varpi_taux - (ch/tau) varpi_xeta    varpi_tz = varpi_taueta / tau
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

// Covariant Milne components of the symmetric thermal shear (xi_{tau tau}, xi_{tau x}, xi_{tau y}, xi_{tau eta}, xi_{xx}, xi_{xy},
// xi_{x eta}, xi_{yy}, xi_{y eta}, xi_{eta eta}) at space-time rapidity eta -> the ten Cartesian lab components
// c = (xi_tt, xi_tx, xi_ty, xi_tz, xi_xx, xi_xy, xi_xz, xi_yy, xi_yz, xi_zz):
//   xi_tt = ch^2 xi_tautau - 2 (ch sh/tau) xi_taueta + (sh/tau)^2 xi_etaeta     xi_tx = ch xi_taux - (sh/tau) xi_xeta
//   xi_tz = -ch sh xi_tautau + ((ch^2 + sh^2)/tau) xi_taueta - (ch sh/tau^2) xi_etaeta   xi_xz = -sh xi_taux + (ch/tau) xi_xeta
//   xi_zz = sh^2 xi_tautau - 2 (ch sh/tau) xi_taueta + (ch/tau)^2 xi_etaeta     (xi_ty, xi_yz as xi_tx, xi_xz; xi_xx, xi_xy, xi_yy unchanged)
__device__ __forceinline__ void cart_shear(const double x[10], double tau, double eta, double c[10])
{
  const double ch = cosh(eta), sh = sinh(eta), inv_tau = 1.0 / tau;
  const double cht = ch * inv_tau, sht = sh * inv_tau;
  c[0] = ch * ch * x[0] - 2.0 * ch * sht * x[3] + sht * sht * x[9];
  c[1] = ch * x[1] - sht * x[6];
  c[2] = ch * x[2] - sht * x[8];
  c[3] = -ch * sh * x[0] + (ch * cht + sh * sht) * x[3] - cht * sht * x[9];
  c[4] = x[4];
  c[5] = x[5];
  c[6] = -sh * x[1] + cht * x[6];
  c[7] = x[7];
  c[8] = -sh * x[2] + cht * x[8];
  c[9] = sh * sh * x[0] - 2.0 * sh * cht * x[3] + cht * cht * x[9];
}

// Covariant Milne components of a scalar gradient (d_tau, d_x, d_y, d_eta; 1/fm, d_eta dimensionless) at space-time rapidity eta -> its
// Cartesian spatial components z = (d_x, d_y, d_z) in 1/fm (the time component never enters the spin Hall term):
//   d_z = -sh d_tau + (ch/tau) d_eta
__device__ __forceinline__ void cart_gradient(const double d[4], double tau, double eta, double z[3])
{
  z[0] = d[1];
  z[1] = d[2];
  z[2] = -sinh(eta) * d[0] + cosh(eta) / tau * d[3];
}

}  // namespace is3d
