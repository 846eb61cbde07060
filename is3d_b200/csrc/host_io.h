// host_io.h -- C++ host layer: readers for the iS3D input files (parameter file, block tables, freeze-out surface,
// particle lists, delta-f coefficient tables, Gauss-Laguerre nodes).  Each reader states the reference routine whose
// file format and corner-case behaviour it reproduces; none of them calls exit() -- errors come back as text.
#pragma once
#include <cstdint>
#include <map>
#include <string>
#include <vector>

namespace is3d {

// iS3D_parameters.dat: `name = value  # comment`, names case-insensitive, values stored as double
// (reference ParameterReader.cpp:38-98, 142-155).
struct Params {
  std::map<std::string, double> kv;
  std::vector<std::string> order;
  bool load(const std::string &path, std::string *err);
  bool has(const std::string &name) const;
  // a missing key is fatal in the reference (ParameterReader.cpp:150-154); here it sets *err and returns 0
  double get(const std::string &name, std::string *err) const;
};

// Whitespace-separated block file -> columns.  Row count = number of newline-terminated lines, column count = number
// of values on the first line (reference arsenal.cpp:406-453 via Table.cpp:179-195).
struct BlockTable {
  std::vector<std::vector<double>> cols;
  long rows = 0;
  bool load(const std::string &path, std::string *err);
  double at(int col1, long row1) const { return cols[col1 - 1][row1 - 1]; }   // 1-based like Table::get
};

struct DecayChannel { int npart = 0; double branch_ratio = 0; long part[5] = {0, 0, 0, 0, 0}; };
struct Particle {
  long mcid = 0;
  std::string name;
  double mass = 0, width = 0;
  int gspin = 0, baryon = 0, strange = 0, charm = 0, bottom = 0, gisospin = 0, charge = 0, decays = 0, sign = 0;
  int stable = 0;                          // first channel has a single product (readindata.cpp:1487-1488)
  int parity = 0;                          // pdg_box.dat only: intrinsic parity +1 / -1 (0 for the conventional lists)
  std::vector<DecayChannel> channels;      // conventional lists only (pdg_box.dat carries no decay table)
};
// PDG/pdg-urqmd_v3.3+.dat, PDG/pdg_smash.dat (readindata.cpp:1440-1568) and PDG/pdg_box.dat (:1571-1684)
bool read_pdg(const std::string &workdir, int hrg_eos, std::vector<Particle> *out, std::string *err);
// intrinsic parities by |MC id| from the PARITY column of PDG/pdg_box.dat (the polarization feed-down reads them next to a conventional
// list); a missing file is an error, an id the file lacks is simply absent from the map
bool read_box_parities(const std::string &workdir, std::map<long, int> *out, std::string *err);
// PDG/weak_decays.dat (this project's own format): one weak channel per line, `parent_mcid daughter_mcid partner_mcid branching alpha phi`
// (phi in radians), `#` starts a comment, blank lines are skipped.  A missing file or a line without exactly those six numbers is an error.
struct WeakTable { std::vector<int32_t> parent, daughter, partner; std::vector<double> branching, alpha, phi; };
bool read_weak_decays(const std::string &workdir, WeakTable *out, std::string *err);

struct SurfaceData {
  int64_t n = 0;
  std::vector<double> tau, x, y, eta, dat, dax, day, dan, ux, uy, un, E, T, P;
  std::vector<double> pitt, pitx, pity, pitn, pixx, pixy, pixn, piyy, piyn, pinn, bulkPi;
  std::vector<double> muB, nB, Vx, Vy, Vn;
  std::vector<double> PL, Wx, Wy, Lambda, aL, c0, c1, c2, c3, c4;     // anisotropic hydro (mode 2)
  std::vector<double> wtx, wty, wtn, wxy, wxn, wyn;                    // thermal vorticity, covariant Milne components (mode 5)
  std::vector<double> xtt, xtx, xty, xtn, xxx, xxy, xxn, xyy, xyn, xnn;   // thermal shear, covariant Milne components (input/thermal_shear.dat)
  std::vector<double> gbt, gbx, gby, gbn;   // gradient of alpha_B = muB/T, covariant Milne components (input/muB_over_T_gradient.dat)
  bool averages_written = false;
  double avg[5] = {0, 0, 0, 0, 0};   // T, E, P, muB, nB after the 15-digit text round trip of the side file
};
struct SurfaceFlags { int mode, dimension, df_mode, include_baryon, include_baryondiff_deltaf; };
// input/surface.dat, formats of FO_data_reader::read_surf_VH_old / read_surf_VH / read_surf_VAH_PLMatch
// (readindata.cpp:148-468, 813-928); also writes and re-reads average_thermodynamic_quantities.dat like the reference.
bool read_surface(const std::string &workdir, const SurfaceFlags &fl, SurfaceData *out, std::string *err);
// input/thermal_shear.dat (this project's own format): one newline-terminated line per surface cell, in surface order, with the ten
// covariant Milne components xi_{tau tau} xi_{tau x} xi_{tau y} xi_{tau eta} xi_{xx} xi_{xy} xi_{x eta} xi_{yy} xi_{y eta} xi_{eta eta}
// (dimensionless).  A missing file, a line count other than out->n or a line with fewer than ten numbers is an error.
bool read_thermal_shear(const std::string &workdir, SurfaceData *out, std::string *err);
// input/muB_over_T_gradient.dat (this project's own format): one newline-terminated line per surface cell, in surface order, with the four
// covariant Milne components d_tau alpha_B, d_x alpha_B, d_y alpha_B (1/fm), d_eta alpha_B (dimensionless) of alpha_B = muB/T.  A missing
// file, a line count other than out->n or a line with fewer than four numbers is an error.
bool read_baryon_gradient(const std::string &workdir, SurfaceData *out, std::string *err);

struct DfTables {
  int n_T = 0, n_muB_file = 0;
  std::vector<double> T, c0, c1, c2, c3, c4, F, G, betabulk, betaV, betapi;    // muB = 0 rows
  std::vector<double> jonah_x, jonah_lambda2, jonah_z;
  double bulkPi_over_Peq_max = -1.0;
};
// deltaf_coefficients/vh/<eos>/*.dat (deltafReader.cpp:65-219)
bool read_df_tables(const std::string &workdir, int hrg_eos, DfTables *out, std::string *err);

struct Laguerre { int alpha = 0, points = 0; std::vector<std::vector<double>> root, weight; };
// tables/gla_roots_weights_32_points.txt (readindata.cpp:23-54)
bool read_laguerre(const std::string &path, Laguerre *out, std::string *err);

// Jonah lambda(Pi/P), z(Pi/P) tables from a hadron-resonance-gas sum at temperature T
// (Deltaf_Data::compute_jonah_coefficients, deltafReader.cpp:222-297)
void compute_jonah_tables(const std::vector<Particle> &pdg, double T, const Laguerre &gla, DfTables *tab);

// anisotropic-hydro per-cell coefficients: bilinear lookup in deltaf_coefficients/vah/c{0..4}_vah1.dat
// (only specification: reference src/cuda/deltafReader.cu:192-277)
struct VahTables { int nL = 0, naL = 0; std::vector<double> L, aL, c[5]; };     // c[k][iL * naL + iaL]
bool read_vah_tables(const std::string &workdir, VahTables *out, std::string *err);
bool vah_lookup(int nL, int naL, const double *L, const double *aL_grid, const double *const c[5], double Lambda_fm, double aL, double out[5]);
bool fill_vah_coefficients(const std::string &workdir, SurfaceData *surf, std::string *err);
double aL_fit(double pl_over_peq);    // arsenal.cpp:999-1028
double R200(double aL);               // arsenal.cpp:1031-1066

}  // namespace is3d
