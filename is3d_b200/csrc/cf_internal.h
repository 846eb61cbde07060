// cf_internal.h -- structures shared by the prepare kernels, the hot kernels and the C-ABI glue.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <string>
#include "../../include/is3d_b200.h"

namespace is3d {

constexpr int kRec = 6;          // doubles per phi record (and per slot record, except the anisotropic model)
constexpr int kRecVah = 8;       // doubles per slot record of the anisotropic model
constexpr int kScal = 4;         // doubles per per-cell scalar record
constexpr int kMaxWarps = 4;     // warps per hot-kernel block (each warp = 32 consecutive (species, pT) pairs)
// variants with MINB >= 7 run 2-warp blocks (register cap 144 at 7 blocks/SM = 14 warps/SM instead of 12)
constexpr int block_warps(int minb) { return minb >= 7 ? 2 : kMaxWarps; }
constexpr int kStages = 4;       // TMA pipeline depth

// Device-side view of the raw surface (GeV/fm units), NULL where switched off
struct RawCells {
  int64_t n;
  const int64_t *gather;      // NULL: record position = cell index; else source cell of every padded record position, -1 = padding
  const double *tau, *eta, *dat, *dax, *day, *dan, *ux, *uy, *un, *T, *P, *E;
  const double *pixx, *pixy, *pixn, *piyy, *piyn, *bulkPi;
  const double *pitt, *pitx, *pity, *pitn, *pinn, *Wx, *Wy, *Lambda, *aL, *c0, *c1, *c2, *c3, *c4;
};

// natural cubic spline table on the device: knots x[n], values y[n], second-derivative coefficients c[n]
struct Spline { const double *x, *y, *c; int n; };

struct PrepTables {
  Spline c0, c2, F, betabulk, betapi, lam2, z;
  double bulkPi_over_Peq_max;
  const double *cosphi, *sinphi;        // [n_phi]
  const double *slot_y;                 // 3+1D: y values [n_y];  2+1D: eta values [n_eta]
  const double *slot_w;                 // 2+1D: eta weights [n_eta]; 3+1D: NULL
  const double *gla_root1, *gla_w1, *gla_root2, *gla_w2; int gla_n;   // feqmod
  double deta_min, mass_pion0, eta_delta;                              // eta_delta: spacing of the eta table (anisotropic 2+1D weights)
};

// Geometry of the tiled record arrays
//   Y[n_ytiles][n_cells_pad][nst][kRec]   slot records (nst = slots per tile)
//   P[n_ptiles][n_cells_pad][npt][kRec]   phi records
//   S[n_cells_pad][kScal]                 per-cell scalars
struct Layout {
  int n_species, n_pT, n_phi, n_y_out;   // output array dims (n_y_out = y table length)
  int n_slots;                           // rapidity slots per cell: n_y (3+1D) or n_eta (2+1D)
  int dim2;                              // dimension == 2: slots are the eta table (y = 0), else the y table at the cell's eta
  int per_slot;                          // dim2 only: keep the eta slots apart (3+1D-shaped tiles) instead of summing them
  int dx;                                // feqmod set-up follows calculate_dN_dX_feqmod (operation = 0) where it differs from the spectra routine
  int nst, n_ytiles, npt, n_ptiles;
  int rec_y;                             // doubles per slot record (kRec or kRecVah)
  int ct;                                // cells per TMA tile
  int64_t n_cells, n_cells_pad, n_tiles;
};

struct PrepCounters { unsigned long long skipped, breakdown, range_error, linear_items; };

// distribution-function models of the hot kernel
enum Model {
  M_LIN14 = 1,      // f_eq (1 + df), 14-moment            (smooth_kernels.cpp:303-312)
  M_LINCE = 2,      // f_eq (1 + df), Chapman-Enskog       (:313-321, also the df_mode 3 breakdown branch :835-857)
  M_FEQMOD = 3,     // modified equilibrium, Mike / Jonah  (:878-928)
  M_JONAHLIN = 4,   // Jonah's linearised df, breakdown branch of df_mode 4 (:858-876)
  M_VAH = 5,        // anisotropic f_a (1 + df~), PL matching (:2297-2349)
  M_IDEAL = 6       // f_eq only: df_mode 1/2 with include_shear_deltaf = include_bulk_deltaf = 0 (df = 0 exactly, BASELINE cfg2)
};

struct HotParams {
  Layout L;
  const double *Y, *P, *S;
  const double *mass, *sign, *degeneracy, *pT;    // species / pT tables on device
  double *partial;                                 // [n_chunks][n_bins]
  const double *renorm;                            // feqmod, df_mode 3: [n_species][n_cells_pad]; NULL -> per-cell value in S[1]
  int n_chunks, n_groupblocks, n_warps;
  long long outflow_thr;                           // bit pattern threshold of the p.dsigma > 0 test
  double prefactor;
  double pT_max;                                   // largest entry of the pT table (factored kernel: range check of pT B)
  int regulate_thr;                                // high-word threshold of |df| >= 1, see clamp_unit()
  int reg_lo, reg_hi;                              // factored kernel: bounds of the high word of g = 1 + df (0, 0x40000000 | INT_MIN, INT_MAX)
  unsigned reg_chk;                                // ... and the unsigned high word above which a member needs the clamp
  double ec[8];                                    // cf_shift.cu: constants of exp_neg_poly (kExpR[0..3], kExpC[0..2]) as kernel-parameter
                                                   // operands: c[0x0][..] feeds a DFMA directly, no register and no LDC
  int one_hi;                                      // 0x3ff00000 (high word of 1.0) as a run-time value, see clamp_unit()
  // operation = 0 (spacetime distributions): momentum-integrated epilogue instead of the spectra bins
  int integ_mode;                                  // 0 spectra; 1 sum over (slot, phi, pT) per chunk; 2 per slot, sum over (phi, pT)
  int integ_sl;                                    // species slots per block: (block lanes - 1) / n_pT + 2
  const int64_t *chunk_tiles;                      // [n_chunks + 1] first cell tile of every chunk (NULL: balanced split)
  const double *pT_weight, *phi_weight;            // quadrature weights of the pT and phi tables
  double *integ;                                   // mode 1: [chunk][ytile][ptile][groupblock][sl]; mode 2: [chunk][slot][ptile][groupblock][sl]
  // cf_shift.cu: e^{-pT (Bmax - B_k)} table of one window of consecutive chunks, [n_ptiles][e_cells][shift_table_record(L)]
  double *E;
  int64_t e_cells;                                 // cells per phi tile the table holds
  int chunk0;                                      // first chunk of the launch: block b works on chunk chunk0 + b / (blocks per chunk)
};

// launchers (cf_prepare.cu / cf_kernels.cu)
cudaError_t launch_prepare_vh(const is3d_flags &fl, const RawCells &cells, const PrepTables &tab, const Layout &L,
                              double *Y, double *P, double *S, PrepCounters *counters, cudaStream_t st);
cudaError_t launch_prepare_feqmod(const is3d_flags &fl, const RawCells &cells, const PrepTables &tab, const Layout &L,
                                  double *YF, double *PF, double *SF, double *YL, double *PL, double *SL,
                                  const double *mass, const double *sign, const double *degeneracy, const double *baryon,
                                  double *renorm, PrepCounters *counters, cudaStream_t st);
cudaError_t launch_prepare_vah(const is3d_flags &fl, const RawCells &cells, const PrepTables &tab, const Layout &L,
                               double *Y, double *P, double *S, PrepCounters *counters, cudaStream_t st);
cudaError_t launch_hot(int model, const HotParams &hp, int variant, cudaStream_t st, size_t *smem_out);
cudaError_t launch_reduce(const double *partial, int n_chunks, int64_t n_bins, int64_t n_active, double *out, cudaStream_t st);
cudaError_t launch_axpy(const double *x, double *y, int64_t n, cudaStream_t st);      // y += x
// integ -> out[unit][species], unit = chunk (mode 1) or slot (mode 2, summed over chunks)
cudaError_t launch_integ_reduce(const HotParams &hp, int n_units, double *out, cudaStream_t st);
// sampler mean yield: per-block triples (sum u.dsigma, sum u.dsigma Pi, sum u.dsigma z) in partial[3 * n_blocks]
cudaError_t launch_yield(const RawCells &cells, const PrepTables &tab, int df_mode, int include_bulk, double *partial, int *n_blocks,
                         PrepCounters *counters, cudaStream_t st);
cudaError_t launch_fp64_peak(double *sink, int iters, cudaStream_t st, int *blocks, int *threads, long long *dfma_per_thread);
// resonance-decay feed-down on device-resident spectra (cf_decays.cu)
int resonance_decays_device(const is3d_particle_list *pdg, int n_chosen, const int32_t *chosen, const is3d_grid *gr, int dimension,
                            double *dN_dev, cudaStream_t st, int *launches, std::string *err);
// polarization feed-down (cf_decays.cu): S_dev = [St | Sx | Sy | Sz | Snorm], n_total doubles each, amended in place; spin2 / parity
// (host) per particle-list entry
int polarization_decays_device(const is3d_particle_list *pdg, const int32_t *spin2, const int32_t *parity, int n_chosen, const int32_t *chosen,
                               const is3d_grid *gr, int dimension, double *S_dev, int64_t n_total, cudaStream_t st, int *launches, std::string *err);
// weak-decay feed-down of the same five arrays (cf_decays.cu); check_weak_decays: the table's argument errors (host only, no device work)
int check_weak_decays(const is3d_particle_list *pdg, const is3d_weak_decays *weak, std::string *err);
int polarization_weak_decays_device(const is3d_particle_list *pdg, const int32_t *spin2, const is3d_weak_decays *weak, int n_chosen,
                                    const int32_t *chosen, const is3d_grid *gr, int dimension, double *S_dev, int64_t n_total, cudaStream_t st,
                                    int *launches, std::string *err);
// strict (reference-order) diagnostic variant, df_mode 1 / 2 (cf_strict.cu); cell_scratch: n_cells * strict_cell_bytes()
size_t strict_cell_bytes();
cudaError_t launch_strict(const is3d_flags &fl, const RawCells &cells, const PrepTables &tab, const Layout &L, const double *mass, const double *sign,
                          const double *degeneracy, const double *pT, int n_eta, double prefactor, void *cell_scratch, double *dN_dev,
                          PrepCounters *counters, cudaStream_t st);
constexpr int kStrictVariant = 99;           // is3d_options.tile_variant value that selects it
void hot_variant_shape(int variant, int dim2, int *nyt, int *npt, int *ct, int *max_warps);
// factored kernel (cf_factored.cu): linear-df models, 3+1D tiles only
constexpr int kNumVariants = 16;             // register-tile variants of cf_kernel (is3d_options.tile_variant 1..16)
constexpr int kNumFactoredVariants = 5;      // shapes of cf_factored_kernel (tile_variant 17..21)
bool factored_supported(int model, const Layout &L);
void factored_variant_shape(int fvariant, int *nyt, int *npt, int *ct, int *max_warps);
int factored_match(int nyt, int npt);        // factored shape with this register tile, or -1
constexpr int kFactoredMinSpecies = 16;      // its lanes are species: shorter lists run on cf_kernel (lanes = (species, pT))
// warps = phi tiles of a block; n_groupblocks = blocks per (cell chunk, y tile) = species groups x pT points x phi blocks
void factored_blocking(int n_species, int n_pT, int n_ptiles, int *n_warps, int *n_groupblocks);
cudaError_t launch_factored(int model, const HotParams &hp, int fvariant, cudaStream_t st, size_t *smem_out);
// shifted-factor kernel (cf_shift.cu): linear-df models, 3+1D tiles, <= 64 pT points; 4-warp blocks, lane <-> (species class, pT)
constexpr int kNumShiftVariants = 4;         // tile_variant 22..25
bool shift_supported(int model, const Layout &L);
void shift_variant_shape(int model, int v, int n_pT, int *nyt, int *npt, int *ct, int *max_warps);   // ct fitted to n_pT
int shift_table_record(const Layout &L);     // doubles per (phi tile, cell) of HotParams::E
// Species of bit-equal (mass, sign) have bit-equal accumulators on the shifted-factor path (degeneracy enters only in the
// epilogue), so its lanes run over these classes and each class's result is stored for every member species.  A kernel
// argument of its own: HotParams is embedded in the parameter structs of other kernels and keeps its layout.
struct SpeciesClasses {
  int n;                                     // classes (lanes = n x n_pT)
  const int32_t *first, *members;            // device, CSR: species of class c are members[first[c] .. first[c + 1])
};
// per window of win_chunks chunks: the table kernel, then cf_shift_kernel on the window's chunks; *launches = kernels launched.
// hp.mass / hp.sign are the class tables [cls.n], hp.degeneracy the species table [L.n_species]
cudaError_t launch_shift(int model, const HotParams &hp, const SpeciesClasses &cls, int v, int win_chunks, cudaStream_t st, size_t *smem_out,
                         int *launches);
// slot records of padding / skipped cells carry this A = u.p / (mT T): every evaluation is dead (exp overflows, f = 0 exactly)
constexpr double kDeadSlotA = 1.0e6;
// spin polarization from thermal vorticity (cf_polzn.cu): ideal-f cells and slots, 5 sums per bin (Snorm, N^t, N^x, N^y, N^z)
struct VortCells { const double *wtx, *wty, *wtn, *wxy, *wxn, *wyn; };    // device pointers, covariant Milne components
constexpr int kPolRecY = 12;     // doubles per slot record
constexpr int kPolRecP = 4;      // doubles per phi record
constexpr int kPolWarps = 4;     // warps per block (at most)
constexpr int kPolNyt3D = 7, kPolNpt3D = 1, kPolNpt2D = 4;
void polzn_shape(int dim2, int *nyt, int *npt, int *ct);
cudaError_t launch_prepare_polzn(const RawCells &cells, const VortCells &vort, const PrepTables &tab, const Layout &L, double *Y, double *P,
                                 PrepCounters *counters, cudaStream_t st);
// partial: [5][n_chunks][n_bins]
cudaError_t launch_polzn(const HotParams &hp, cudaStream_t st);
// thermal-shear part of the spin polarization (cf_polzn_xi.cu): the layout, records sizes and chunks of cf_polzn.cu, 4 sums per bin
struct ShearCells { const double *x[10]; };    // device pointers, covariant Milne components tautau taux tauy taueta xx xy xeta yy yeta etaeta
struct PolXiParams {
  HotParams hp;                  // layout, records Y / P, species and pT tables, partial [4][n_chunks][n_bins] (Snorm, N^x, N^y, N^z)
  const double *cosphi, *sinphi; // [n_phi]
  const double *y;               // 3+1D: the y table [n_y]; 2+1D: unused (y = 0)
};
cudaError_t launch_prepare_polzn_xi(const RawCells &cells, const ShearCells &shear, const PrepTables &tab, const Layout &L, double *Y,
                                    double *P, PrepCounters *counters, cudaStream_t st);
cudaError_t launch_polzn_xi(const PolXiParams &prm, cudaStream_t st);
// spin Hall part of the spin polarization (cf_polzn_she.cu): the layout, records sizes and chunks of cf_polzn.cu, 4 sums per bin
struct GradientCells { const double *d[4]; };  // device pointers, covariant Milne components of d alpha_B: tau x y eta
struct PolSheParams {
  HotParams hp;                  // layout, records Y / P, species and pT tables, partial [4][n_chunks][n_bins] (Snorm, N^x, N^y, N^z)
  const double *cosphi, *sinphi; // [n_phi]
  const double *y;               // 3+1D: the y table [n_y]; 2+1D: unused (y = 0)
  const double *baryon;          // [n_species] baryon number q_B
};
cudaError_t launch_prepare_polzn_she(const RawCells &cells, const GradientCells &grad, const PrepTables &tab, const Layout &L, double *Y,
                                     double *P, PrepCounters *counters, cudaStream_t st);
cudaError_t launch_polzn_she(const PolSheParams &prm, cudaStream_t st);
// spin density matrix from thermal vorticity (cf_spin_density.cu): the records of prepare_polzn_kernel, its own register tile,
// 9 sums per bin (Snorm, P_x, P_y, P_z, Q_xx, Q_xy, Q_xz, Q_yy, Q_yz)
constexpr int kSdSums = 9;
constexpr int kSdMinBlocks = 3;  // blocks per SM of kPolWarps warps the register budget is sized for (__launch_bounds__)
constexpr int kSdNyt3D = 3, kSdNpt3D = 1, kSdNpt2D = 2;
struct SpinDensityParams {
  HotParams hp;                  // layout, records Y / P, species and pT tables, partial [9][n_chunks][n_bins]
  const double *y;               // 3+1D: the y table [n_y]; 2+1D: unused (y = 0)
  unsigned long long *boson_bad; // device counter: boson evaluations with u.p/T - J theta <= 0 (one atomic per block that has any)
};
void spin_density_shape(int dim2, int *nyt, int *npt, int *ct);
cudaError_t launch_spin_density(const SpinDensityParams &prm, cudaStream_t st);
// HBT moments (cf_hbt.cu): the records of prepare_vh_kernel plus a per-cell record [tau, x, y, 0]; 10 sums per bin
constexpr int kHbtRecC = 4;      // doubles per per-cell position record
constexpr int kHbtSums = 10;     // S0, So, Ss, Sl, Soo, Sss, Sll, Sos, Sol, Ssl
constexpr int kHbtWarps = 4;     // warps per block (at most)
constexpr int kHbtMinBlocks = 3; // blocks per SM the register budget is sized for (__launch_bounds__)
constexpr int kHbtNyt3D = 3, kHbtNpt3D = 1, kHbtNpt2D = 2;
struct HbtParams {
  HotParams hp;                  // layout, records Y / P / S, species and pT tables, partial [10][n_chunks][n_bins], flags
  const double *C;               // [n_cells_pad][kHbtRecC]
  const double *cosphi, *sinphi; // [n_phi]
};
void hbt_shape(int dim2, int *nyt, int *npt, int *ct);
cudaError_t launch_prepare_hbt_cells(const double *tau, const double *x, const double *y, int64_t n, int64_t n_pad, double *C, cudaStream_t st);
cudaError_t launch_hbt(int model, const HbtParams &prm, cudaStream_t st);
// HBT Fourier sums (cf_hbtq.cu): the records of cf_hbt_kernel; per bin and q point q_k = k dq d of every ray, sum w cos and sum w sin
constexpr int kHbtqKQ = 21;       // q points per block (register tile of 2 KQ sums per bin); the phase recurrence restarts every KQ
constexpr int kHbtqMinBlocks = 3; // blocks per SM of kHbtWarps warps the register budget is sized for (__launch_bounds__)
constexpr int kHbtqNyt3D = 1, kHbtqNpt3D = 1, kHbtqNpt2D = 1;
struct HbtqParams {
  HotParams hp;                  // layout, records Y / P / S, species and pT tables, partial [2 n_dir n_q][n_chunks][n_bins], flags
  const double *C;               // [n_cells_pad][kHbtRecC]
  const double *cosphi, *sinphi; // [n_phi]
  const double *dir;             // [n_dir][3]: d dq / hbar c [1/fm], (o, s, l)
  int n_dir, n_q, n_qtiles;      // n_qtiles = ceil(n_q / kHbtqKQ)
};
void hbtq_shape(int dim2, int *nyt, int *npt, int *ct);
cudaError_t launch_hbt_fourier(int model, const HbtqParams &prm, cudaStream_t st);

}  // namespace is3d
