/* include/is3d_b200.h -- C ABI of the B200-native smooth Cooper-Frye spectra path.
 *
 * The reference (derekeverett/iS3D) has no FFI/plugin interface; the hot path sits behind the C++ member functions
 *   EmissionFunctionArray::calculate_dN_pTdpTdphidy          src/cpp/emissionfunction.h:179, emissionfunction_smooth_kernels.cpp:28
 *   EmissionFunctionArray::calculate_dN_ptdptdphidy_feqmod   src/cpp/emissionfunction.h:182, emissionfunction_smooth_kernels.cpp:396
 *   EmissionFunctionArray::calculate_dN_pTdpTdphidy_VAH_PL   src/cpp/emissionfunction.h:(VAH_PL), emissionfunction_smooth_kernels.cpp:2140
 * called from EmissionFunctionArray::calculate_spectra (src/cpp/emissionfunction.cpp:1519, 1584, 1650).  The entry
 * points below take what those calls take -- the per-species arrays, the structure-of-arrays freeze-out surface, the
 * momentum tables and the delta-f coefficient tables -- as plain pointers and sizes, and add the result into a
 * caller-owned spectra array with the reference's layout.  INTEGRATION.md shows the few lines that replace the three
 * call sites.  No C++/torch types cross this boundary; all functions return 0 or an IS3D_ERR_* code, never exit().
 * Further down: operation = 0 (calculate_dN_dX{,_feqmod}, smooth_kernels.cpp:1000-2135), the sampler's mean-yield pass
 * (calculate_total_yield, emissionfunction_sampling_kernels.cpp:653-831) and the file-level host layer.
 *
 * Threading: every entry point works on the CUDA device that is current in the calling thread and keeps one workspace per
 * device, so different host threads may drive different devices concurrently (calls on the same device are serialised).
 * Multi-GPU: either one process per GPU, each calling with its own contiguous shard of cells and all-reducing the spectra
 * itself (is3d_b200/distributed.py under torchrun), or ONE process calling the *_multi entry points below.
 */
#ifndef IS3D_B200_H
#define IS3D_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  IS3D_OK = 0,
  IS3D_ERR_ARGUMENT = 1,      /* NULL / inconsistent argument */
  IS3D_ERR_UNSUPPORTED = 2,   /* flag combination outside the path (e.g. include_baryon = 1, see DESIGN.md) */
  IS3D_ERR_TABLE_RANGE = 3,   /* a cell's T (or Pi/P for df_mode 4) lies outside the coefficient table; the reference aborts here */
  IS3D_ERR_CUDA = 4,          /* CUDA runtime failure; is3d_b200_last_error() has the text */
  IS3D_ERR_NO_DEVICE = 5,     /* no CUDA device: there is deliberately no CPU fallback */
  IS3D_ERR_IO = 6,            /* host layer: missing / malformed input file */
  IS3D_ERR_NCCL = 7           /* multi-GPU: libnccl.so.2 could not be loaded, or an NCCL call failed */
};

/* Freeze-out surface, structure of arrays, GeV / fm units exactly as EmissionFunctionArray::calculate_spectra packs
 * them (emissionfunction.cpp:1327-1499).  Pointers for switched-off terms may be NULL.  Read-only, caller-owned. */
typedef struct {
  int64_t n_cells;
  const double *tau, *eta, *dat, *dax, *day, *dan, *ux, *uy, *un, *T, *P, *E;
  const double *pixx, *pixy, *pixn, *piyy, *piyn, *bulkPi;
  const double *muB, *nB, *Vx, *Vy, *Vn;
  /* anisotropic hydro (mode 2) only: all ten pi_perp components, W_perp, Lambda, alpha_L and per-cell c0..c4 */
  const double *pitt, *pitx, *pity, *pitn, *pinn, *Wx, *Wy, *Lambda, *aL, *c0, *c1, *c2, *c3, *c4;
  /* transverse cell positions: read by operation = 0 (spacetime distributions) and the HBT paths only, NULL otherwise */
  const double *x, *y;
} is3d_surface;

/* Chosen species in output order (emissionfunction.cpp:1293-1307). */
typedef struct {
  int32_t n;
  const double *mass, *sign, *degeneracy, *baryon;
} is3d_species;

/* Momentum / rapidity tables (iS3D.cpp:161-167).  eta/eta_weight are used when dimension = 2, y when dimension = 3. */
typedef struct {
  int32_t n_pT, n_phi, n_y, n_eta;
  const double *pT, *phi, *y, *eta, *eta_weight;
} is3d_grid;

/* Switches captured by the EmissionFunctionArray constructor (emissionfunction.cpp:170-191). */
typedef struct {
  int32_t mode;              /* surface type: 0,1,4,5,6,7 = viscous hydro; 2 = anisotropic hydro, PL matching */
  int32_t df_mode;           /* 1 14-moment, 2 Chapman-Enskog, 3 feqmod (Mike), 4 feqmod (Jonah) */
  int32_t dimension;         /* 2 boost invariant (y = 0, eta quadrature) or 3 */
  int32_t include_baryon, include_bulk_deltaf, include_shear_deltaf, include_baryondiff_deltaf;
  int32_t regulate_deltaf, outflow;
  double deta_min, mass_pion0;
} is3d_flags;

/* muB = 0 rows of deltaf_coefficients/vh/<eos>/{c0..c4,F,G,betabulk,betaV,betapi}.dat as stored in the files
 * (T-scaled; deltafReader.cpp:65-219), plus the Jonah lambda^2 / z tables (deltafReader.cpp:222-297). */
typedef struct {
  int32_t n_T;
  const double *T, *c0, *c1, *c2, *c3, *c4, *F, *G, *betabulk, *betaV, *betapi;
  int32_t n_jonah;
  const double *jonah_x, *jonah_lambda2, *jonah_z;
  double bulkPi_over_Peq_max;
} is3d_df_tables;

/* generalized Gauss-Laguerre nodes alpha = 1, 2 (tables/gla_roots_weights_32_points.txt), feqmod only */
typedef struct {
  int32_t n_points;
  const double *root1, *weight1, *root2, *weight2;
} is3d_laguerre;

typedef struct {
  int32_t memory;            /* 0: surface arrays and dN live in host memory; 1: they are device pointers on the current device */
  void *stream;              /* cudaStream_t to launch on (NULL = default stream) */
  int32_t n_chunks;          /* cell-range split used for load balance; 0 = choose */
  int32_t tile_variant;      /* kernel variant: 0 = tuned default for the model (df_mode 1 / 2 and ideal f_eq on 3+1D tiles with <= 64 pT
                                points: shifted-factor kernel 23; everything else: cf_kernel); 1..16 = register-tile table of cf_kernel;
                                17..21 = shapes of the factored kernel (df_mode 1/2, 3+1D, >= 16 species); 22..25 = shapes of the
                                shifted-factor kernel (df_mode 1/2, 3+1D, <= 64 pT points; slots x phi points 7 x 3, 3 x 6 (the
                                default), 3 x 8, 7 x 6 for df_mode 1 and ideal f_eq; 7 x 2, 7 x 3 (the default), 7 x 4, 7 x 6
                                for df_mode 2); 99 = strict diagnostic kernel (df_mode 1/2 in
                                the reference's own operation order, one thread per bin: ~50x slower, tests only).  A variant that does
                                not apply to the call returns IS3D_ERR_ARGUMENT. */
  int32_t reserved[4];
} is3d_options;

typedef struct {
  int64_t cells_skipped_udsigma;   /* cells with u.dsigma <= 0 (smooth_kernels.cpp:137) */
  int64_t cells_feqmod_breakdown;  /* the reference's `breakdown` counter (smooth_kernels.cpp:721, 992) */
  int64_t evaluations;             /* cells x species x pT x phi x y x eta */
  double h2d_ms, prepare_ms, kernel_ms, reduce_ms, d2h_ms, total_ms;   /* CUDA-event times on the launch stream */
  int32_t gpu_launches;            /* kernels launched by this call */
  int32_t n_chunks, tile_variant;
  int32_t n_gpus;                  /* devices that worked on this call (times above: slowest device) */
  double allreduce_ms;             /* multi-GPU: the NCCL all-reduce of the spectra array */
  int32_t n_chunks_wanted;         /* chunks the load-balance rule asked for; > n_chunks when the 4 GiB cap on the partial-sum buffer cut it down */
  int32_t reserved;
} is3d_stats;

/* Bind to the current CUDA device and create its workspace (one per CUDA ordinal).  Safe to call more than once. */
int is3d_b200_init(void);
/* ---- one process, several GPUs (SURVEY 8b / 8e: the reference has ONE entry, IS3D::run_particlization, src/cpp/iS3D.cpp:73-191;
 * a drop-in for it has to use the whole box by itself).  is3d_b200_init_devices(n) selects the first n visible devices (n <= 0: all
 * of them, or the number in the environment variable IS3D_B200_GPUS) and creates one NCCL communicator over them (libnccl.so.2 is
 * loaded at run time).  is3d_b200_smooth_spectra_multi() then takes HOST arrays, splits the cells into contiguous shards of
 * ceil(n_cells / n) (species, grids and coefficient tables are replicated), runs one host thread and one stream per device, combines
 * the per-device spectra with a single ncclAllReduce(sum, double) and adds device 0's copy into dN_out.  With one device it is
 * is3d_b200_smooth_spectra().  is3d_b200_run_workdir / is3d_b200_run_surface and the IS3D class use it, so the file-level
 * drop-in runs on every visible GPU.  Results differ from the 1-GPU result by summation order only (non-negative terms: ~1e-15). */
int is3d_b200_init_devices(int n_gpus);
int is3d_b200_device_count(void);     /* devices the *_multi entry points use (1 before is3d_b200_init_devices) */
int is3d_b200_shutdown(void);
const char *is3d_b200_strerror(int code);
const char *is3d_b200_last_error(void);
int is3d_b200_version(void);

/* dN_out has n_species * n_pT * n_phi * n_y doubles, index ipart + n_species*(ipT + n_pT*(iphi + n_phi*iy))
 * (emissionfunction_smooth_kernels.cpp:363); the result is ADDED into it (reference: `+=` into a zeroed array).
 * Dispatch follows calculate_spectra: mode 2 -> anisotropic kernel; df_mode 1,2 -> linear delta-f; 3,4 -> feqmod. */
int is3d_b200_smooth_spectra(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species,
                             const is3d_grid *grid, const is3d_df_tables *df, const is3d_laguerre *laguerre,
                             const is3d_options *options, double *dN_out, is3d_stats *stats);

int is3d_b200_smooth_spectra_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species,
                                   const is3d_grid *grid, const is3d_df_tables *df, const is3d_laguerre *laguerre,
                                   const is3d_options *options, double *dN_out, is3d_stats *stats);

/* ---- operation = 0: spacetime distributions of the momentum-integrated yield (SURVEY 8f, row N2) -------------------
 * Replaces EmissionFunctionArray::calculate_dN_dX (emissionfunction_smooth_kernels.cpp:1000-1446, df_mode 1, 2) and
 * calculate_dN_dX_feqmod (:1449-2135, df_mode 3, 4), called from calculate_spectra (emissionfunction.cpp:1514, 1579).
 * Every cell's yield  sum_{pT, phi, y} w_pT w_phi g/(2 pi hbar c)^3 sum_eta p.dsigma f  (3+1D: all y points, unweighted,
 * like the reference) is binned by the cell's tau and r = sqrt(x^2 + y^2) (is3d_surface.x, .y):
 *    itau = floor((tau - tau_min) / ((tau_max - tau_min) / tau_bins)),  ir likewise (:1376-1400).
 * Results are the RAW sums the reference accumulates; its writers divide by the bin volumes (:1404-1435), see
 * is3d_b200_write_spacetime().  Arrays are caller-allocated host memory and are OVERWRITTEN:
 *    dN_tau [n_species][tau_bins]   dN_r [n_species][r_bins]   dN_taur [n_species][tau_bins][r_bins]
 *    dN_dydeta [n_species][eta_pts] (eta_pts = 1 in 3+1D, n_eta in 2+1D)   dN_dy [n_species]                      */
typedef struct {
  double tau_min, tau_max, r_min, r_max;   /* iS3D_parameters.dat: tau_min, tau_max, r_min, r_max */
  int32_t tau_bins, r_bins;                /* tau_bins, r_bins */
  const double *pT_weight, *phi_weight;    /* host: second column of the pT and phi tables */
} is3d_spacetime_bins;
typedef struct { double *dN_tau, *dN_r, *dN_taur, *dN_dydeta, *dN_dy; } is3d_spacetime_result;
int is3d_b200_spacetime_distributions(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species,
                                      const is3d_grid *grid, const is3d_df_tables *df, const is3d_laguerre *laguerre,
                                      const is3d_spacetime_bins *bins, const is3d_options *options,
                                      is3d_spacetime_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, one thread per device; the histograms are
 * linear in the cells, so the per-device raw sums (a few MB) are added on the host in device order. */
int is3d_b200_spacetime_distributions_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species,
                                            const is3d_grid *grid, const is3d_df_tables *df, const is3d_laguerre *laguerre,
                                            const is3d_spacetime_bins *bins, const is3d_options *options,
                                            is3d_spacetime_result *result, is3d_stats *stats);

/* ---- resonance-decay feed-down of the smooth spectra (SURVEY 8f, row N3) ------------------------------------------------
 * Replaces EmissionFunctionArray::do_resonance_decays and the routines below it (src/cpp/emissionfunction_resonance_decays.cpp:
 * 124-2158, called from calculate_spectra, emissionfunction.cpp:1689-1698).  The particle list is the reference's particle_info
 * array (readindata.cpp:1440-1568: anti-baryons right behind their baryon, `stable` = first channel has one product) with the
 * decay channels flattened: channel rows dec_first[i] .. dec_first[i] + decays[i] - 1 of dec_npart / dec_br / dec_part[row * 5 + k].
 * chosen_pdg_index is the reference's chosen_particles_sampling_table (particle-list index of every chosen species).
 * dN [y][phi][pT][species] (host memory, or device memory with options->memory = 1) is amended in place: parents from the last
 * chosen species down to the second, 2- and 3-body channels, daughters that are chosen species.
 * NOTE: the reference snapshot disables its own routine with an exit(-1) at entry (:126-129, the author's note on the MTmax
 * handling of the interpolation); this entry point implements the body behind that guard and is checked against it. */
typedef struct {
  int32_t n_particles;
  const int32_t *mcid;
  const double *mass, *width;
  const int32_t *stable, *decays, *dec_first;
  const int32_t *dec_npart;
  const double *dec_br;
  const int32_t *dec_part;
} is3d_particle_list;
int is3d_b200_resonance_decays(const is3d_particle_list *particles, int32_t n_chosen, const int32_t *chosen_pdg_index,
                               const is3d_grid *grid, int32_t dimension, const is3d_options *options, double *dN, is3d_stats *stats);

/* ---- spin polarization of hadrons from thermal vorticity (mode 5 surfaces) -------------------------------------------
 * Mean spin vector of the emitted hadrons at freeze-out (Becattini et al. 2013; Karpenko & Becattini 2017), f_eq only (no delta-f):
 *    Snorm(p) = g/(2 pi hbar c)^3 sum_cells sum_slots w p.dsigma f,                      f = 1 / (exp(p.u/T) + sign)
 *    N^mu(p)  = g/(2 pi hbar c)^3 sum_cells sum_slots w p.dsigma f (1 - sign f) (-1/(8m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau
 *    S^mu(p)  = N^mu / Snorm (mean spin vector; rest frame S*_i = S^i - S^t p^i / (E + m), for spin 1/2 P* = 2 S*)
 * Cells, slots and weights w are those of the ideal-f spectra (u.dsigma <= 0 skipped, Theta(p.dsigma) with outflow = 1, 3+1D: y table at
 * the cell's eta, 2+1D: y = 0 and the eta quadrature), so Snorm is bin for bin the ideal spectrum.  Components are Cartesian lab
 * components (t, x, y, z), p^mu = (mT cosh y, pT cos phi, pT sin phi, mT sinh y), eps^{txyz} = +1.
 * Input: the six vorticity columns of a mode-5 surface, in file order the covariant Milne components varpi_{tau x}, varpi_{tau y},
 * varpi_{tau eta}, varpi_{xy}, varpi_{x eta}, varpi_{y eta} of varpi_{mu nu} = -(1/2)(d_mu beta_nu - d_nu beta_mu), beta = u/T
 * (dimensionless); they are converted to Cartesian components at the cell's eta (2+1D: the slot's eta) in cf_polzn.cuh, cart_vorticity().
 * The five result arrays have the spectra layout ipart + n_species*(ipT + n_pT*(iphi + n_phi*iy)), hold the RAW sums N^mu and Snorm
 * (they add across cell shards and devices; the ratio S^mu does not) and are ADDED into; host or device memory per options->memory.
 * Errors: IS3D_ERR_UNSUPPORTED for mode = 2 and include_baryon = 1; IS3D_ERR_ARGUMENT for a NULL vorticity or a species with m <= 0.
 * Only the surface arrays tau, eta, dat, dax, day, dan, ux, uy, un, T are read; df_mode and the delta-f switches do not enter. */
typedef struct { const double *wtx, *wty, *wtn, *wxy, *wxn, *wyn; } is3d_vorticity;
typedef struct { double *St, *Sx, *Sy, *Sz, *Snorm; } is3d_polarization_result;
int is3d_b200_spin_polarization(const is3d_flags *flags, const is3d_surface *surface, const is3d_vorticity *vorticity,
                                const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                is3d_polarization_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, the five arrays summed on the host. */
int is3d_b200_spin_polarization_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_vorticity *vorticity,
                                      const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                      is3d_polarization_result *result, is3d_stats *stats);

/* ---- spin polarization of hadrons from thermal shear (shear-induced polarization) --------------------------------------------
 * The second first-order term of the local-equilibrium mean spin vector (Becattini, Buzzegoli, Palermo 2021; Becattini, Buzzegoli,
 * Inghirami, Karpenko, Palermo 2021), over the cells, slots, weights, species and bins of is3d_b200_spin_polarization:
 *    N_xi^mu(p) = g/(2 pi hbar c)^3 sum_cells sum_slots w p.dsigma f (1 - sign f) (-1/(8m)) eps^{mu rho sigma tau} p_tau 2 that_rho xi_{sigma lambda} p^lambda / E
 * with the thermal shear xi_{mu nu} = (1/2)(d_mu beta_nu + d_nu beta_mu), beta = u/T, that = (1, 0, 0, 0) the lab time direction,
 * E = p^t = mT cosh y, and the prefactor and eps^{txyz} = +1 of the vorticity term, so that S^mu = (N^mu + N_xi^mu) / Snorm.
 * In Cartesian lab components N_xi^t = 0 exactly and N_xi = -(1/(4 m E)) sum W (v x p), v_j = xi_jt E + xi_jl p^l (p.N_xi = 0).
 * Input: the ten covariant Milne components xi_{tau tau}, xi_{tau x}, xi_{tau y}, xi_{tau eta}, xi_{xx}, xi_{xy}, xi_{x eta}, xi_{yy},
 * xi_{y eta}, xi_{eta eta} (dimensionless, the convention of the mode-5 vorticity columns), converted to Cartesian components at the
 * cell's eta (2+1D: the slot's eta) in cf_polzn.cuh, cart_shear().
 * Results go into an is3d_polarization_result: St receives exact zeros, Sx, Sy, Sz the RAW sums N_xi, Snorm the ideal spectrum (bit for
 * bit what is3d_b200_spin_polarization returns on the same device with the same options).  All are ADDED into; host or device memory
 * per options->memory.  Errors: IS3D_ERR_UNSUPPORTED for mode = 2 and include_baryon = 1; IS3D_ERR_ARGUMENT for a NULL shear or shear
 * array or a species with m <= 0. */
typedef struct { const double *xtt, *xtx, *xty, *xtn, *xxx, *xxy, *xxn, *xyy, *xyn, *xnn; } is3d_thermal_shear;
int is3d_b200_spin_polarization_shear(const is3d_flags *flags, const is3d_surface *surface, const is3d_thermal_shear *shear,
                                      const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                      is3d_polarization_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, the five arrays summed on the host. */
int is3d_b200_spin_polarization_shear_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_thermal_shear *shear,
                                            const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                            is3d_polarization_result *result, is3d_stats *stats);

/* ---- spin polarization of baryons from the spin Hall effect (gradient of alpha_B = muB/T) ------------------------------------
 * The baryonic spin Hall term of the first-order local-equilibrium mean spin vector (Liu & Yin, JHEP 07 (2021) 188; Ryu, Jupic, Shen,
 * PRC 104 (2021) 054908), in the lab-frame (that) form of the thermal-shear term, over the cells, slots, weights, species and bins of
 * is3d_b200_spin_polarization:
 *    N_she^mu(p) = g/(2 pi hbar c)^3 sum_cells sum_slots w p.dsigma f (1 - sign f) (-1/(8m)) eps^{mu rho sigma tau} p_tau (-2 q_B that_rho d_sigma alpha_B / E)
 * with q_B = species->baryon, that = (1, 0, 0, 0), E = p^t = mT cosh y, and the prefactor and eps^{txyz} = +1 of the vorticity term, so
 * that S^mu = (N^mu + N_xi^mu + N_she^mu) / Snorm.  It is the shear term with xi_{sigma lambda} p^lambda -> xi_{sigma lambda} p^lambda -
 * q_B d_sigma alpha_B, the gradient of the argument beta.p - q_B alpha_B of f.  In Cartesian lab components N_she^t = 0 exactly and
 * N_she = +(q_B / (4 m E)) sum W (zeta x p), zeta_j = hbar c d_j alpha_B (GeV); mesons (q_B = 0) give exact zeros.
 * f is the muB-free weight of the other polarization terms (include_baryon = 1 is rejected): the term is exact at first order in
 * d alpha_B around that weight, and Snorm is the Snorm of the vorticity call, so the three N arrays add.
 * Input: the covariant Milne components d_tau alpha_B, d_x alpha_B, d_y alpha_B (1/fm) and d_eta alpha_B (dimensionless), converted to
 * Cartesian components at the cell's eta (2+1D: the slot's eta) in cf_polzn.cuh, cart_gradient().
 * Results go into an is3d_polarization_result: St receives exact zeros, Sx, Sy, Sz the RAW sums N_she, Snorm the ideal spectrum (bit for
 * bit what is3d_b200_spin_polarization returns on the same device with the same options).  All are ADDED into; host or device memory
 * per options->memory.  Errors: IS3D_ERR_UNSUPPORTED for mode = 2 and include_baryon = 1; IS3D_ERR_ARGUMENT for a NULL gradient or
 * gradient array, a NULL species->baryon or a species with m <= 0. */
typedef struct { const double *dt, *dx, *dy, *dn; } is3d_baryon_gradient;
int is3d_b200_spin_polarization_spin_hall(const is3d_flags *flags, const is3d_surface *surface, const is3d_baryon_gradient *gradient,
                                          const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                          is3d_polarization_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, the five arrays summed on the host. */
int is3d_b200_spin_polarization_spin_hall_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_baryon_gradient *gradient,
                                                const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                                is3d_polarization_result *result, is3d_stats *stats);

/* ---- spin density matrix of hadrons from thermal vorticity: all-order mean spin, rank-2 spin tensor, vector-meson rho00 ---------
 * The local-equilibrium distribution with the spin term exponentiated, [exp(beta.p - (1/2) varpi:Sigma) + Theta]^-1 (Becattini, Chandra,
 * Del Zanna, Grossi, Ann. Phys. 338 (2013) 32), for any spin J = (g - 1)/2, over the cells, slots, weights, u.dsigma <= 0 skip, outflow
 * rule, species and bins of is3d_b200_spin_polarization (the same vorticity input and conventions).  Per evaluation:
 *    theta^mu = -(1/(2m)) eps^{mu rho sigma tau} varpi_{rho sigma} p_tau = (1/m)(omega.p, E omega - e x p)   (4 x the vector of the N^mu
 *               sum, without (1 - Theta f)),  theta*_i = theta^i - theta^t p^i/(E + m) (rest frame of the pure boost along p),
 *    theta = |theta* |, that = theta* / theta,  f_m = 1/(exp(u.p/T - m theta) + Theta) for the levels m = -J .. J along that.
 * Nine RAW sums per bin (K = 1/(2 pi hbar c)^3, W = slot weight x p.dsigma), which add across cell shards and devices:
 *    Snorm = K sum W sum_m f_m
 *    P_i   = K sum W sum_m m f_m that_i                                          i = x, y, z
 *    Q_ij  = K sum W sum_m f_m (3m^2 - J(J+1))/2 (that_i that_j - delta_ij/3)    ij = xx, xy, xz, yy, yz  (Q_zz = -Q_xx - Q_yy)
 * Ratios: <S*_i> = P_i/Snorm; T_ij = <S*_i S*_j> - J(J+1) delta_ij/3 = Q_ij/Snorm; for J = 1, rho00 along a rest-frame unit axis n is
 * 1/3 - n.T.n.  At theta = 0 (varpi = 0, or J = 0) P and Q are exactly 0 and Snorm is the Snorm of is3d_b200_spin_polarization; at
 * linear order P_i/Snorm = (J(J+1)/3)(1 - Theta f) theta*_i, i.e. 4J(J+1)/3 times its rest-frame S*.
 * Only the varpi term is exponentiated: rho00 - 1/3 is the second order of that exponent, not a complete second-order gradient expansion
 * (shear-induced alignment and other second-order terms are not included).
 * All nine arrays are ADDED into; host or device memory per options->memory.
 * Errors: IS3D_ERR_UNSUPPORTED for mode = 2 and include_baryon = 1; IS3D_ERR_ARGUMENT for a NULL vorticity, a NULL result array, a
 * species with m <= 0 or with a degeneracy that is not an integer in [1, 16], and for a boson (Theta = -1) evaluation with
 * u.p/T - J theta <= 0, where the top level has no valid occupation (the count is in is3d_b200_last_error()).  On any error every result
 * array is left untouched. */
typedef struct { double *Snorm, *Px, *Py, *Pz, *Qxx, *Qxy, *Qxz, *Qyy, *Qyz; } is3d_spin_density_result;
int is3d_b200_spin_density(const is3d_flags *flags, const is3d_surface *surface, const is3d_vorticity *vorticity,
                           const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                           is3d_spin_density_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, the nine arrays summed on the host in device
 * order. */
int is3d_b200_spin_density_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_vorticity *vorticity,
                                 const is3d_species *species, const is3d_grid *grid, const is3d_options *options,
                                 is3d_spin_density_result *result, is3d_stats *stats);

/* ---- feed-down of the spin polarization through resonance decays ------------------------------------------------------------
 * Amends, in place, the five raw-sum arrays of is3d_b200_spin_polarization (or vorticity + shear sums added component by component) so
 * that they describe all hadrons of a species, primary and from decays.  Parents, order, channels, daughter groups, kernels and
 * arithmetic are those of is3d_b200_resonance_decays, and:
 *  - Snorm receives exactly the spectra feed-down: bit for bit is3d_b200_resonance_decays applied to the input Snorm;
 *  - St, Sx, Sy, Sz of a daughter gain, at every point of the 2-body integral (12 x 12 (v, zeta) nodes, both parent azimuths), the
 *    point's weight times the daughter's spin four-vector S_D there.  The parent's rest-frame spin S*_P = (N^i - N^t p^i/(E + m))/Snorm
 *    (its physical mass; 0 where log Snorm is not finite) is interpolated linearly in (M_T, Phi[, Y]) at the cell and with the weights
 *    of the log spectrum, held at the last M_T point beyond the table.  With p* = L(P)^-1 p (L(P) the pure boost to the parent's rest
 *    frame) and n = p* / |p*|, the daughter's rest-frame spin is s* = a' S*_P + b' (S*_P.n) n; its four-vector is carried back by L(P).
 *    2+1D: the parent's spin four-vector at rapidity Y is the longitudinal boost by Y of the one at (M_T, Phi, 0).
 *  - 3-body channels and 2-body channels without a transfer law feed Snorm only: their daughters are diluted, not polarized.
 * Normalisation: the arrays carry the spin-1/2 prefactor -1/(8m) for every species; a spin-J parent's true mean spin is 4J(J+1)/3 times
 * S*_P (Becattini et al. 2013), and that factor is folded into (a', b').  Laws, for a daughter with J_D = 1/2 (C = <S*_D>/S*_P of the true
 * spins):
 *    J_P = 1/2 -> 1/2 + photon (partner MC id 22)                     a' = 0                 b' = -1       C = -1/3
 *    J_P -> 1/2 + spin-0 meson, the three parities known             a' = -eta (2J_P+1)/2   b' = 1 - a'   C = (1 - eta (2J_P+1)) / (4J_P(J_P+1))
 *    with eta = -(-1)^(J_P - 1/2) P_P P_D P_meson.  Any other 2-body channel has no law.
 * is3d_spin_parity has one entry per particle-list entry: spin2 = 2J >= 0, parity = +1 / -1, or 0 when unknown.
 * Arrays: spectra layout ipart + n_species*(ipT + n_pT*(iphi + n_phi*iy)); host or device memory per options->memory.
 * Errors: those of is3d_b200_resonance_decays (a parent whose tail fit has fewer than 2 points is IS3D_ERR_ARGUMENT, and all five arrays
 * stay untouched); IS3D_ERR_ARGUMENT also for a NULL spin / parity table or array, a NULL result array, spin2 < 0 or a parity outside
 * {-1, 0, 1}. */
typedef struct { const int32_t *spin2, *parity; } is3d_spin_parity;
int is3d_b200_polarization_decays(const is3d_particle_list *particles, const is3d_spin_parity *spin_parity, int32_t n_chosen,
                                  const int32_t *chosen_pdg_index, const is3d_grid *grid, int32_t dimension, const is3d_options *options,
                                  is3d_polarization_result *sums, is3d_stats *stats);

/* ---- feed-down of the spin polarization through weak decays (Xi -> Lambda pi, Omega -> Lambda K, Omega -> Xi pi) -----------------
 * Amends, in place, the five arrays with the weak channels of the caller's table only.  Meant for the output of
 * is3d_b200_polarization_decays (it does not call it): weak daughters are stable hadrons and no strong decay follows a weak one, so the
 * two passes in this order are exact.  One row per channel: parent -> daughter + partner (MC ids looked up in the particle list, where
 * an antiparticle is its own row), branching ratio and the PDG decay parameters (alpha, phi):
 *    beta = sqrt(1 - alpha^2) sin phi,   gamma = sqrt(1 - alpha^2) cos phi.
 * Weak parents that are chosen species are processed in descending mass (ties: descending chosen index), so Omega -> Xi comes before
 * Xi -> Lambda and each parent's arrays are final when its turn comes.  A row whose parent or daughter is not a chosen species does
 * nothing; only the daughter is fed (not the partner).  The 2-body integration points, the interpolation of the parent's log spectrum
 * and of S*_P, and the Lorentz chain are those of is3d_b200_polarization_decays; no width shift is applied.  At every integration point,
 * with S = S*_P and n the daughter's direction in the parent's rest frame, a row whose spins are 2J = 1 -> 1 + 0 (spin_parity->spin2 of
 * parent, daughter, partner; parities are not used) follows the Lee-Yang law, exact in S:
 *    Snorm_D += w (1 + 2 alpha S.n)
 *    N_D^mu  += w x the four-vector of  s* = (alpha/2 + S.n) n + beta S x n + gamma (S - (S.n) n)
 * (s* is the daughter's rest-frame spin times the yield 1 + 2 alpha S.n, in the frame of the pure boost along n from the parent's rest
 * frame), w = the point's weight of the spectra feed-down.  Averaged over n: yield 1, <s*> = (1 + 2 gamma)/3 S (the transfer coefficient
 * C_XiLambda of the Xi polarization measured through its Lambda); alpha = beta = 0, gamma = -1 is the 1/2+ -> 1/2+ 0- law of
 * is3d_b200_polarization_decays and gamma = +1 its S-wave law.  Any other row (e.g. Omega-, J = 3/2) has no law: it feeds Snorm with the
 * plain 2-body integral and only dilutes.  With N = 0 everywhere (S = 0), the Snorm returned is the weak feed-down of the plain
 * spectrum, and N_D receives w x (alpha/2) n carried to the lab: the helicity of the daughters of unpolarised parents.  The library
 * ships no decay parameters: their values change between PDG editions.
 * n = 0 is a valid no-op.  Arrays: spectra layout; host or device memory per options->memory.  Results are bit-reproducible.
 * Errors: IS3D_ERR_ARGUMENT, with every array untouched, for those of is3d_b200_polarization_decays, a NULL table or row array, n < 0, an
 * MC id that is not in the list, a parent or daughter that is not `stable` in the list, a branching ratio outside [0, 1], a parent whose
 * branching ratios sum to more than 1 (beyond 1e-9 of rounding), |alpha| > 1, a non-finite alpha or phi, m_daughter + m_partner >= m_parent,
 * and a parent whose tail fit has fewer than 2 points. */
typedef struct {
  int32_t n;                                   /* rows; 0 is a valid no-op */
  const int32_t *parent, *daughter, *partner;  /* MC ids, looked up in the particle list (antiparticles are their own rows) */
  const double *branching, *alpha, *phi;       /* PDG parametrisation: beta = sqrt(1-alpha^2) sin phi, gamma = sqrt(1-alpha^2) cos phi */
} is3d_weak_decays;
int is3d_b200_polarization_weak_decays(const is3d_particle_list *particles, const is3d_spin_parity *spin_parity,
                                       const is3d_weak_decays *weak, int32_t n_chosen, const int32_t *chosen_pdg_index,
                                       const is3d_grid *grid, int32_t dimension, const is3d_options *options,
                                       is3d_polarization_result *sums, is3d_stats *stats);

/* ---- HBT radii: space-time variances of the Cooper-Frye emission function ---------------------------------------------
 * Gaussian (moment) approximation with pair momentum K = p (Wiedemann & Heinz, Phys. Rept. 319 (1999) 145).  For every spectra bin
 * (species, pT, phi, y; 2+1D: y = 0) the frame is the bin's longitudinally co-moving frame (LCMS): a longitudinal boost by the bin's
 * y, out = (cos phi, sin phi, 0), side = (-sin phi, cos phi, 0), long = beam axis, beta_perp = pT / mT.  Each evaluation (cell, slot)
 * of the spectra contributes at the LCMS coordinates, with (x_c, y_c) = is3d_surface.x, .y [fm] and eta the cell's eta (3+1D) or the
 * slot's eta (2+1D):
 *    t* = tau cosh(eta - y)          z* = tau sinh(eta - y)
 *    o  = x_c cos phi + y_c sin phi - beta_perp t*        s = -x_c sin phi + y_c cos phi        l = z*
 * and the weight w = g/(2 pi hbar c)^3 (slot weight) p.dsigma f_eq (1 + df), exactly the summand of is3d_b200_smooth_spectra with the
 * same flags (cells with u.dsigma <= 0 skipped, Theta(p.dsigma) with outflow = 1, regulate_deltaf as there), so S0 is bin for bin the
 * spectrum.  The ten result arrays hold the RAW sums (they add across cell shards and devices):
 *    S0 = sum w, So = sum w o, Ss = sum w s, Sl = sum w l, Soo = sum w o^2, Sss, Sll, Sos = sum w o s, Sol, Ssl
 * The radii are R^2_ij = S_ij / S0 - (S_i / S0)(S_j / S0), i, j in {o, s, l} [fm^2]; a bin with S0 = 0 has radii 0.  Negative
 * weights (outflow = 0, delta-f without regulate_deltaf) are summed as they are, never clamped, so such radii may be unphysical.
 * Arrays have the spectra layout ipart + n_species*(ipT + n_pT*(iphi + n_phi*iy)) and are ADDED into; host or device memory per
 * options->memory.  Weights: df_mode 1 (14-moment) and 2 (Chapman-Enskog), ideal f_eq when both delta-f switches are off; 3+1D and
 * 2+1D; every viscous-hydro surface mode.
 * Errors: IS3D_ERR_UNSUPPORTED for df_mode 3 / 4, mode = 2 and include_baryon = 1; IS3D_ERR_ARGUMENT for NULL x or y;
 * IS3D_ERR_TABLE_RANGE as is3d_b200_smooth_spectra. */
typedef struct { double *S0, *So, *Ss, *Sl, *Soo, *Sss, *Sll, *Sos, *Sol, *Ssl; } is3d_hbt_result;
int is3d_b200_hbt_moments(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species, const is3d_grid *grid,
                          const is3d_df_tables *df, const is3d_options *options, is3d_hbt_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, the ten arrays summed on the host in device
 * order. */
int is3d_b200_hbt_moments_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species, const is3d_grid *grid,
                                const is3d_df_tables *df, const is3d_options *options, is3d_hbt_result *result, is3d_stats *stats);

/* ---- HBT correlation functions: Fourier transform of the Cooper-Frye emission function --------------------------------------
 * Smoothness and on-shell approximation with pair momentum K = p (Wiedemann & Heinz, Phys. Rept. 319 (1999) 145), the frame, the
 * coordinates (o, s, l) and the weight w of is3d_b200_hbt_moments (same flags, skip rules and errors).  q is given in each bin's LCMS,
 * q = (q_o, q_s, q_l) [GeV], with q^0 = beta_perp q_o from q.K = 0, so that q.x = -(q_o o + q_s s + q_l l) exactly.  q is sampled on
 * rays: the caller's n_dir direction vectors d = (d_o, d_s, d_l) (host memory, not normalised by the library) and the points
 * q_k = k dq d, k = 0 .. n_q - 1.  The result arrays hold the RAW sums (they add across cell shards and devices)
 *    Re[d][k][bin] = sum w cos(theta),   Im[d][k][bin] = sum w sin(theta),   theta = k dq (d_o o + d_s s + d_l l) / hbar c
 * with hbar c = 0.197327053 GeV fm; Re[d][0] is S0 (the spectrum) for every d and Im[d][0] = 0, exactly.  The correlation function of
 * identical particles of an unpolarised source is C = 1 - sign (Re^2 + Im^2) / (g Re[d][0]^2) (sign = -1 bosons, +1 fermions,
 * g = degeneracy; C = 1 where S0 = 0).  Negative weights are summed as they are.  Not included: final-state interactions, resonance-
 * decay halos, K != p, non-identical pairs, the modified-equilibrium, anisotropic and baryon weights.
 * Arrays are [n_dir][n_q][n_bins] with the spectra bin layout inside, ADDED into; host or device memory per options->memory.
 * Errors: as is3d_b200_hbt_moments; IS3D_ERR_ARGUMENT also for NULL Re, Im, q rays or dir, n_dir < 1, n_q < 1, dq <= 0 or not finite,
 * a direction component that is not finite, and 2 n_dir n_q n_bins partial sums beyond 4 GiB (one cell chunk). */
typedef struct {
  int32_t n_dir, n_q;   /* rays and q points per ray */
  double dq;            /* step along every ray [GeV] */
  const double *dir;    /* [n_dir][3] (o, s, l), host memory */
} is3d_hbt_qrays;
typedef struct { double *Re, *Im; /* [n_dir][n_q][n_bins] */ } is3d_hbt_fourier_result;
int is3d_b200_hbt_fourier(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species, const is3d_grid *grid,
                          const is3d_df_tables *df, const is3d_hbt_qrays *qrays, const is3d_options *options,
                          is3d_hbt_fourier_result *result, is3d_stats *stats);
/* Same over the devices of is3d_b200_init_devices(): HOST arrays, contiguous cell shards, Re and Im summed on the host in device order. */
int is3d_b200_hbt_fourier_multi(const is3d_flags *flags, const is3d_surface *surface, const is3d_species *species, const is3d_grid *grid,
                                const is3d_df_tables *df, const is3d_hbt_qrays *qrays, const is3d_options *options,
                                is3d_hbt_fourier_result *result, is3d_stats *stats);

/* FP64 FMA peak of the current device measured with a dependency-free DFMA chain (the roofline denominator;
 * MEASURED_PEAKS.json carries no FP64 figure).  Returns TFLOP/s in *tflops, SM clock not touched. */
int is3d_b200_measure_fp64_peak(double *tflops, double *ms);
/* Same probe launched back to back for `seconds` of device time: the sustained (power-capped) FP64 roof. */
int is3d_b200_measure_fp64_sustained(double seconds, double *tflops);

/* ---- host layer: the drop-in behind iS3D_parameters.dat / input/surface.dat / PDG / deltaf_coefficients / tables ----
 * Equivalent of IS3D::run_particlization(1) with operation = 1 (src/cpp/iS3D.cpp:73-191): reads the CWD-relative input
 * files under `workdir`, runs the spectra on the GPU, writes results/dN_pTdpTdphidy*.dat, results/vn_continuous/ and
 * results/dN_dy_*.dat with the reference's formats; with do_resonance_decays = 1 it then runs the feed-down and writes
 * results/dN_pTdpTdphidy_resonance_decays.dat and results/dN_dpTdphidy_resonance_decays.dat (emissionfunction.cpp:452-488, 555-590),
 * and dN_raw receives the amended spectra.  If dN_raw != NULL it receives the spectra (n_raw doubles max).
 * operation = 0 runs the spacetime distributions instead and writes results/spacetime_distribution/dN_taudtaudy_<mcid>.dat,
 * dN_twopirdrdy_<mcid>.dat, dN_twopitaurdtaudrdy_<mcid>.dat, dN_dydeta_<mcid>_<eta_pts>pt.dat (smooth_kernels.cpp:1112-1126,
 * 1404-1435); dN_raw then receives the raw sums concatenated as [dN_tau | dN_r | dN_taur | dN_dydeta | dN_dy]. */
int is3d_b200_run_workdir(const char *workdir, double *dN_raw, int64_t n_raw, int32_t *mcid_out, int32_t n_mcid_max,
                          is3d_stats *stats);
/* Same with the freeze-out cells passed in memory (reference: IS3D::read_fo_surf_from_memory + run_particlization(0),
 * src/cpp/iS3D.cpp:26-71): parameters, particle list and tables still come from `workdir`. */
int is3d_b200_run_surface(const char *workdir, const is3d_surface *surface, double *dN_raw, int64_t n_raw,
                          int32_t *mcid_out, int32_t n_mcid_max, is3d_stats *stats);

/* Host-side table builders for callers that drive is3d_b200_smooth_spectra() directly (no working directory):
 *  - surface averages T, E, P, muB, nB weighted as in FO_data_reader::read_surf_VH (readindata.cpp:423-466), passed through
 *    the reference's 15-significant-digit side file round trip (average_thermodynamic_quantities.dat);
 *  - the Jonah lambda^2(Pi/P), z(Pi/P) tables of Deltaf_Data::compute_jonah_coefficients (deltafReader.cpp:222-297):
 *    301 points each, built from the full particle list at temperature T_avg with the alpha = 2 Gauss-Laguerre nodes. */
int is3d_b200_surface_averages(const is3d_surface *surface, double *out5);
int is3d_b200_jonah_tables(int32_t n_particles, const double *mass, const double *degeneracy, const double *sign, double T_avg,
                           int32_t n_points, const double *root2, const double *weight2,
                           double *x301, double *lambda2_301, double *z301, double *bulkPi_over_Peq_max);
/* Anisotropic hydro, in-memory callers: alpha_L and Lambda [GeV] from the surface file's T, P, PL columns [fm units]
 * (readindata.cpp:905-918), and the per-cell c0..c4 from the (Lambda [fm^-1], alpha_L) tables, each table given as
 * c[iL * naL + iaL] with the values of deltaf_coefficients/vah/c{k}_vah1.dat (src/cuda/deltafReader.cu:192-277). */
int is3d_b200_vah_anisotropy(int64_t n, const double *T_fm, const double *P_fm, const double *PL_fm, double *aL_out, double *Lambda_GeV_out);
int is3d_b200_vah_coefficients(int32_t nL, int32_t naL, const double *L_fm, const double *aL_grid, const double *c0, const double *c1,
                               const double *c2, const double *c3, const double *c4, int64_t n, const double *Lambda_GeV,
                               const double *aL, double *o0, double *o1, double *o2, double *o3, double *o4);
/* ---- sampler mean yield (SURVEY 8f, row N4) -----------------------------------------------------------------------
 * is3d_b200_particle_densities: n_eq, dn_bulk, dn_diff per species at the surface averages avg5 = (T, E, P, muB, nB) -- what
 * Deltaf_Data::compute_particle_densities (deltafReader.cpp:536-650) stores in particle_info.  Host computation; rootK/weightK are
 * the alpha = K rows of tables/gla_roots_weights_32_points.txt (alpha = 3 only for df_mode 1).
 * is3d_b200_mean_yield: EmissionFunctionArray::calculate_total_yield (emissionfunction_sampling_kernels.cpp:653-831) for the
 * chosen species' densities: sum over cells with u.dsigma > 0 of u.dsigma (n_eq + Pi dn_bulk) (df_mode 1-3) or
 * u.dsigma z(Pi/P) n_eq (df_mode 4), times 2 y_cut in 2+1D.  include_baryon = 0 only.  The surface reduction runs on the GPU. */
int is3d_b200_particle_densities(int32_t n, const double *mass, const double *degeneracy, const double *baryon, const double *sign,
                                 const double *avg5, int32_t df_mode, const is3d_df_tables *df, int32_t n_points,
                                 const double *root1, const double *weight1, const double *root2, const double *weight2,
                                 const double *root3, const double *weight3, double *neq, double *dn_bulk, double *dn_diff);
int is3d_b200_mean_yield(const is3d_flags *flags, const is3d_surface *surface, int32_t n_species, const double *neq,
                         const double *dn_bulk, const is3d_df_tables *df, double y_cut, const is3d_options *options,
                         double *Ntot, is3d_stats *stats);

/* Writers only: produce the results/ files of `workdir` from a spectra array in the reference layout. */
int is3d_b200_write_results(const char *workdir, const double *dN, int64_t n);
/* Host-layer inspection without GPU work: dumps what the readers derived (named double records) to out_path. */
int is3d_b200_host_dump(const char *workdir, const char *out_path);
const char *is3d_b200_host_error(void);

#ifdef __cplusplus
}
#endif
#endif
