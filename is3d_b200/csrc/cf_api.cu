// cf_api.cu -- the extern "C" boundary (include/is3d_b200.h): workspace management, host<->device staging, kernel
// sequencing and CUDA-event timing.  There is no CPU fallback: without a CUDA device every entry point fails.
#include "cf_internal.h"
#include "host_math.h"
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstddef>
#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace is3d {

// Per-device state: one grow-only workspace, its events and a lock per CUDA ordinal.  A call works on the device that is
// current in the calling thread; the multi-GPU entry points run one host thread per device.
static thread_local std::string g_last_error;       // text of the calling thread's last failure
constexpr int kMaxDevices = 64;

#define CU_CHECK(call)                                                                          \
  do {                                                                                          \
    cudaError_t e__ = (call);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      char buf__[512];                                                                          \
      snprintf(buf__, sizeof(buf__), "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      g_last_error = buf__;                                                                     \
      return IS3D_ERR_CUDA;                                                                     \
    }                                                                                           \
  } while (0)

// a grow-only device buffer
struct DevBuf {
  void *p = nullptr; size_t cap = 0;
  cudaError_t reserve(size_t bytes)
  {
    if (bytes <= cap) return cudaSuccess;
    if (p) { cudaFree(p); p = nullptr; cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

struct Workspace {
  DevBuf raw, small, Y, P, S, Y2, P2, S2, partial, dN, counters, extra, gather, integ, integ_out;
  DevBuf E;                       // cf_shift_kernel's e^{-pT (Bmax - B_k)} table, one window of chunks
  cudaEvent_t ev[8];
  bool events = false;
  void release()
  {
    raw.release(); small.release(); Y.release(); P.release(); S.release(); Y2.release(); P2.release(); S2.release();
    partial.release(); dN.release();
    counters.release(); extra.release(); gather.release(); integ.release(); integ_out.release(); E.release();
    if (events) { for (auto &e : ev) cudaEventDestroy(e); events = false; }
  }
};
struct Device {
  std::mutex mu;                   // one call at a time per device
  Workspace ws;
  int sm_count = 0;
  int l2_bytes = 0;
  bool init = false;
};
static Device g_dev[kMaxDevices];

// bump allocator over the `small` buffer for tables; all offsets 256-byte aligned
struct SmallArena {
  std::vector<unsigned char> host;
  template <class T> size_t put(const T *src, size_t n)
  {
    size_t off = (host.size() + 255) & ~(size_t)255;
    host.resize(off + n * sizeof(T));
    if (n) memcpy(host.data() + off, src, n * sizeof(T));
    return off;
  }
};

static int fail(int code, const char *msg) { g_last_error = msg; return code; }

// operation = 0: what the core returns instead of spectra bins (see HotParams::integ_mode)
struct IntegRequest {
  int mode = 1;                               // 1: per (tau, r) category of cells;  2: per eta slot (2+1D rapidity distribution)
  const double *pT_weight = nullptr, *phi_weight = nullptr;    // host
  const int32_t *category = nullptr;          // mode 1, host: category of every cell, 0 <= category < n_categories
  int n_categories = 0;
  std::vector<int32_t> unit_category;         // out, mode 1: category of every unit (= cell chunk)
  std::vector<double> result;                 // out: [n_units][n_species]
  int n_units = 0;
};

// keep_dev != NULL: the spectra stay in the device workspace (*keep_dev receives the pointer, valid until the next call on that
// device) instead of being added into dN_out -- used by the multi-GPU entry point, which all-reduces them first
static int smooth_core(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                       const is3d_df_tables *df, const is3d_laguerre *gla, const is3d_options *opt_in,
                       double *dN_out, is3d_stats *stats, IntegRequest *iq, double **keep_dev = nullptr);
static void multi_shutdown();

}  // namespace is3d

using namespace is3d;

extern "C" {

int is3d_b200_version(void) { return 100; }

const char *is3d_b200_strerror(int code)
{
  switch (code) {
    case IS3D_OK: return "ok";
    case IS3D_ERR_ARGUMENT: return "invalid argument";
    case IS3D_ERR_UNSUPPORTED: return "flag combination not supported by the smooth Cooper-Frye path";
    case IS3D_ERR_TABLE_RANGE: return "cell temperature or Pi/P outside the delta-f coefficient table";
    case IS3D_ERR_CUDA: return "CUDA runtime error";
    case IS3D_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    case IS3D_ERR_IO: return "input/output error in the host layer";
    case IS3D_ERR_NCCL: return "NCCL unavailable or failed (multi-GPU entry points)";
    default: return "unknown error";
  }
}

const char *is3d_b200_last_error(void) { return g_last_error.c_str(); }

// the calling thread's current device, initialised on first use
static int current_device(Device **out)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return fail(IS3D_ERR_NO_DEVICE, "no CUDA device visible");
  int dev = 0;
  CU_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) return fail(IS3D_ERR_ARGUMENT, "CUDA device ordinal out of range");
  Device &D = g_dev[dev];
  std::lock_guard<std::mutex> lk(D.mu);
  if (!D.init) {
    CU_CHECK(cudaDeviceGetAttribute(&D.sm_count, cudaDevAttrMultiProcessorCount, dev));
    CU_CHECK(cudaDeviceGetAttribute(&D.l2_bytes, cudaDevAttrL2CacheSize, dev));
    if (!D.ws.events) {
      for (auto &e : D.ws.ev) CU_CHECK(cudaEventCreate(&e));
      D.ws.events = true;
    }
    D.init = true;
  }
  *out = &D;
  return IS3D_OK;
}

int is3d_b200_init(void)
{
  Device *D = nullptr;
  return current_device(&D);
}

int is3d_b200_shutdown(void)
{
  multi_shutdown();
  int n = 0, prev = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return IS3D_OK;
  cudaGetDevice(&prev);
  for (int d = 0; d < n && d < kMaxDevices; d++) {
    Device &D = g_dev[d];
    std::lock_guard<std::mutex> lk(D.mu);
    if (!D.init) continue;
    cudaSetDevice(d);
    D.ws.release();
    D.init = false;
  }
  cudaSetDevice(prev);
  return IS3D_OK;
}

int is3d_b200_measure_fp64_peak(double *tflops, double *ms_out)
{
  Device *Dp = nullptr;
  int rc = current_device(&Dp);
  if (rc) return rc;
  Workspace &ws = Dp->ws;
  std::lock_guard<std::mutex> lk(Dp->mu);
  CU_CHECK(ws.counters.reserve(256));
  int blocks = 0, threads = 0; long long per_thread = 0;
  const int iters = 20000;
  CU_CHECK(launch_fp64_peak(ws.counters.as<double>(), 2000, 0, &blocks, &threads, &per_thread));   // warm-up
  float best = 1e30f;
  for (int rep = 0; rep < 3; rep++) {
    CU_CHECK(cudaEventRecord(ws.ev[0], 0));
    CU_CHECK(launch_fp64_peak(ws.counters.as<double>(), iters, 0, &blocks, &threads, &per_thread));
    CU_CHECK(cudaEventRecord(ws.ev[1], 0));
    CU_CHECK(cudaEventSynchronize(ws.ev[1]));
    float ms = 0;
    CU_CHECK(cudaEventElapsedTime(&ms, ws.ev[0], ws.ev[1]));
    if (ms < best) best = ms;
  }
  const double flops = 2.0 * (double)per_thread * blocks * threads;
  if (tflops) *tflops = flops / (best * 1e-3) * 1e-12;
  if (ms_out) *ms_out = best;
  return IS3D_OK;
}

int is3d_b200_measure_fp64_sustained(double seconds, double *tflops)
{
  Device *Dp = nullptr;
  int rc = current_device(&Dp);
  if (rc) return rc;
  Workspace &ws = Dp->ws;
  std::lock_guard<std::mutex> lk(Dp->mu);
  CU_CHECK(ws.counters.reserve(256));
  int blocks = 0, threads = 0; long long per_thread = 0;
  const int iters = 20000;                       // ~21 ms per launch at the burst clock
  CU_CHECK(launch_fp64_peak(ws.counters.as<double>(), 2000, 0, &blocks, &threads, &per_thread));
  CU_CHECK(cudaDeviceSynchronize());
  int launches = (int)(seconds / 0.021) + 1;
  CU_CHECK(cudaEventRecord(ws.ev[0], 0));
  for (int i = 0; i < launches; i++) CU_CHECK(launch_fp64_peak(ws.counters.as<double>(), iters, 0, &blocks, &threads, &per_thread));
  CU_CHECK(cudaEventRecord(ws.ev[1], 0));
  CU_CHECK(cudaEventSynchronize(ws.ev[1]));
  float ms = 0;
  CU_CHECK(cudaEventElapsedTime(&ms, ws.ev[0], ws.ev[1]));
  const double flops = 2.0 * (double)per_thread * blocks * threads * launches;
  if (tflops) *tflops = flops / (ms * 1e-3) * 1e-12;
  return IS3D_OK;
}

int is3d_b200_smooth_spectra(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                             const is3d_df_tables *df, const is3d_laguerre *gla, const is3d_options *opt_in,
                             double *dN_out, is3d_stats *stats)
{
  if (!dN_out) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  return smooth_core(fl, sf, sp, gr, df, gla, opt_in, dN_out, stats, nullptr);
}

}  // extern "C"

namespace is3d {

static int smooth_core(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                       const is3d_df_tables *df, const is3d_laguerre *gla, const is3d_options *opt_in,
                       double *dN_out, is3d_stats *stats, IntegRequest *iq, double **keep_dev)
{
  if (!fl || !sf || !sp || !gr || (!dN_out && !iq && !keep_dev)) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  Device *Dp = nullptr;
  { int rc = current_device(&Dp); if (rc) return rc; }
  Workspace &g_ws = Dp->ws;
  const int g_sm_count = Dp->sm_count;
  std::lock_guard<std::mutex> lk(Dp->mu);
  is3d_options opt; memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  cudaStream_t st = (cudaStream_t)opt.stream;
  is3d_stats stt; memset(&stt, 0, sizeof(stt));

  // ---- validation / dispatch (emissionfunction.cpp:1503-1673)
  const bool vah = (fl->mode == 2);
  if (fl->dimension != 2 && fl->dimension != 3) return fail(IS3D_ERR_ARGUMENT, "dimension must be 2 or 3");
  if (sp->n <= 0 || gr->n_pT <= 0 || gr->n_phi <= 0 || gr->n_y <= 0) return fail(IS3D_ERR_ARGUMENT, "empty species list or momentum table");
  if (!sp->mass || !sp->sign || !sp->degeneracy || !gr->pT || !gr->phi || !gr->y) return fail(IS3D_ERR_ARGUMENT, "NULL species or momentum table");
  if (fl->dimension == 2 && (gr->n_eta <= 0 || !gr->eta || !gr->eta_weight)) return fail(IS3D_ERR_ARGUMENT, "dimension = 2 needs the eta table");
  if (fl->include_baryon) return fail(IS3D_ERR_UNSUPPORTED, "include_baryon = 1 (the reference's (T, muB) lookup reads out of bounds, SURVEY R8)");
  if (!vah && (fl->df_mode < 1 || fl->df_mode > 4)) return fail(IS3D_ERR_ARGUMENT, "df_mode must be 1..4");
  if (!vah && (!df || df->n_T < 3 || !df->T)) return fail(IS3D_ERR_ARGUMENT, "delta-f coefficient tables missing");
  const bool feqmod = !vah && (fl->df_mode == 3 || fl->df_mode == 4);
  const bool ideal = !vah && (fl->df_mode == 1 || fl->df_mode == 2) && !fl->include_shear_deltaf && !fl->include_bulk_deltaf;
  const int model = vah ? M_VAH : ideal ? M_IDEAL : (fl->df_mode == 1 ? M_LIN14 : fl->df_mode == 2 ? M_LINCE : M_FEQMOD);
  if (!vah) {
    if (fl->df_mode == 1 && (!df->c0 || !df->c2)) return fail(IS3D_ERR_ARGUMENT, "df_mode 1 needs the c0 and c2 tables");
    if ((fl->df_mode == 2 || fl->df_mode == 3) && (!df->F || !df->betabulk || !df->betapi)) return fail(IS3D_ERR_ARGUMENT, "df_mode 2/3 need the F, betabulk and betapi tables");
    if (fl->df_mode == 4 && (!df->betapi || df->n_jonah < 3 || !df->jonah_x || !df->jonah_lambda2 || !df->jonah_z))
      return fail(IS3D_ERR_ARGUMENT, "df_mode 4 needs betapi and the Jonah lambda/z tables");
    if (fl->df_mode == 3 && (!gla || gla->n_points <= 0 || !gla->root1 || !gla->weight1 || !gla->root2 || !gla->weight2))
      return fail(IS3D_ERR_ARGUMENT, "df_mode 3 needs the Gauss-Laguerre nodes");
  }
  const int64_t n_cells = sf->n_cells;
  if (n_cells < 0) return fail(IS3D_ERR_ARGUMENT, "negative cell count");
  const bool dim2 = (fl->dimension == 2);
  const int64_t n_bins = (int64_t)sp->n * gr->n_pT * gr->n_phi * gr->n_y;

  // ---- layout
  Layout L; memset(&L, 0, sizeof(L));
  L.n_species = sp->n; L.n_pT = gr->n_pT; L.n_phi = gr->n_phi; L.n_y_out = gr->n_y;
  L.dim2 = dim2 ? 1 : 0;
  L.per_slot = (iq && iq->mode == 2) ? 1 : 0;
  L.dx = iq ? 1 : 0;
  L.n_slots = dim2 ? gr->n_eta : gr->n_y;
  L.rec_y = vah ? kRecVah : kRec;
  const bool sum_slots = dim2 && !L.per_slot;               // the hot kernel folds the eta slots into one accumulator
  if (iq && vah) return fail(IS3D_ERR_UNSUPPORTED, "spacetime distributions exist for mode 1 surfaces only");
  if (iq && iq->mode == 2 && !dim2) return fail(IS3D_ERR_ARGUMENT, "per-slot integration is a 2+1D pass");
  if (iq && (!iq->pT_weight || !iq->phi_weight)) return fail(IS3D_ERR_ARGUMENT, "pT / phi quadrature weights missing");
  // tile_variant: 0 = model default (tuned on B200, see profiles/), k > 0 = table entry k - 1 (tuning / tests).
  // Defaults: linear-df models (and ideal f_eq) on 3+1D tiles with <= 64 pT points run cf_shift_kernel (tile_variant 23: 3 slots x
  // 6 phi points at 3 blocks/SM for 14-moment delta-f and ideal f_eq, 7 x 3 for Chapman-Enskog and Jonah linear);
  // modified equilibrium, the anisotropic model, 2+1D and operation = 0 run cf_kernel.
  // 17..21 = shapes of the factored kernel (cf_factored.cu; linear-df models on 3+1D tiles, >= 16 species): opt-in for the main
  // pass (measured within +-10 % of cf_kernel on B200, DESIGN.md section 6), always used for the sparse linear-branch pass of
  // df_mode 3 / 4, where its per-cell skip of dead records makes that pass nearly free
  // 99 = strict diagnostic variant (cf_strict.cu): df_mode 1 / 2 spectra in the reference's operation order, one thread per bin
  int variant, fvariant = -1;
  const bool f_ok = factored_supported(model, L) && !iq;      // operation = 0 integrates over the pT lanes of a block (cf_kernel)
  const bool strict = (opt.tile_variant == kStrictVariant);
  // 22..25 = shapes of the shifted-factor kernel (cf_shift.cu; linear-df models on 3+1D tiles, <= 64 pT points), slots x phi points:
  // 7 x 3, 3 x 6, 3 x 8 at 3 blocks/SM and 7 x 6 at 2 (14 moment, ideal); 7 x 2 at 4, 7 x 3 at 3, 7 x 4 and 7 x 6 at 2 (CE, Jonah)
  // (16-cell tiles, halved where the pipeline would not fit that many blocks per SM: 3 x 8 at 32 pT points runs 8-cell tiles)
  int svariant = -1;
  const int first_shift = kNumVariants + kNumFactoredVariants + 1;
  const bool s_ok = shift_supported(model, L) && !iq;
  if (strict && (iq || vah || feqmod)) return fail(IS3D_ERR_ARGUMENT, "tile_variant 99 (strict diagnostic kernel) needs df_mode 1/2, mode 1 and operation 1");
  if (opt.tile_variant < 0 || (opt.tile_variant >= first_shift + kNumShiftVariants && !strict)) return fail(IS3D_ERR_ARGUMENT, "unknown tile_variant");
  if (opt.tile_variant >= first_shift && !strict) {
    if (!s_ok) return fail(IS3D_ERR_ARGUMENT, "tile_variant 22..25 (shifted-factor kernel) needs df_mode 1/2, dimension 3, operation 1 and <= 64 pT points");
    svariant = opt.tile_variant - first_shift;
  }
  if (opt.tile_variant >= 1 && opt.tile_variant <= kNumVariants) variant = opt.tile_variant - 1;
  else if (opt.tile_variant > kNumVariants && opt.tile_variant <= kNumVariants + kNumFactoredVariants) {
    if (!f_ok) return fail(IS3D_ERR_ARGUMENT, "tile_variant 17..21 (factored kernel) needs df_mode 1/2, dimension 3, operation 1 and >= 16 species");
    variant = opt.tile_variant - 1; fvariant = variant - kNumVariants;
  }
  else if (svariant >= 0) variant = opt.tile_variant - 1;
  else if (sum_slots) variant = (model == M_FEQMOD || model == M_VAH) ? 12 : (model == M_IDEAL ? 13 : 10);
  else if (s_ok) { svariant = 1; variant = first_shift - 1 + svariant; }   // linear-df models, 3+1D: cf_shift_kernel, 3 x 6 (14 moment) / 7 x 3 (CE)
  else variant = (model == M_VAH || model == M_FEQMOD) ? 11 : 9;
  int nyt, npt, ct, max_warps;
  if (fvariant >= 0) factored_variant_shape(fvariant, &nyt, &npt, &ct, &max_warps);
  else if (svariant >= 0) shift_variant_shape(model, svariant, gr->n_pT, &nyt, &npt, &ct, &max_warps);
  else hot_variant_shape(variant, sum_slots ? 1 : 0, &nyt, &npt, &ct, &max_warps);
  L.nst = sum_slots ? L.n_slots : nyt;
  L.n_ytiles = sum_slots ? 1 : (L.n_slots + nyt - 1) / nyt;
  L.npt = npt; L.n_ptiles = (L.n_phi + npt - 1) / npt;
  L.ct = ct;
  L.n_cells = n_cells;
  // cells grouped by category ((tau, r) bin): every category starts on a tile boundary
  std::vector<int64_t> cat_tiles;                           // tiles per category
  if (iq && iq->mode == 1) {
    if ((!iq->category && n_cells > 0) || iq->n_categories <= 0) return fail(IS3D_ERR_ARGUMENT, "cell categories missing");
    std::vector<int64_t> count((size_t)iq->n_categories, 0);
    for (int64_t i = 0; i < n_cells; i++) {
      const int32_t c = iq->category[i];
      if (c < 0 || c >= iq->n_categories) return fail(IS3D_ERR_ARGUMENT, "cell category out of range");
      count[(size_t)c]++;
    }
    // small categories: shorter TMA tiles keep the padding (on average (ct - 1) / 2 cells per category) below ~5 %
    if (!sum_slots) {
      int64_t nonempty = 0;
      for (int64_t v : count) nonempty += (v > 0);
      const int64_t avg = nonempty ? n_cells / nonempty : 0;
      if (avg < 40) ct = 2; else if (avg < 80) ct = 4; else if (avg < 160) ct = 8;
      L.ct = ct;
    }
    cat_tiles.resize(count.size());
    L.n_tiles = 0;
    for (size_t c = 0; c < count.size(); c++) { cat_tiles[c] = (count[c] + ct - 1) / ct; L.n_tiles += cat_tiles[c]; }
  } else {
    L.n_tiles = (n_cells + ct - 1) / ct;
  }
  L.n_cells_pad = L.n_tiles * ct;

  // cf_shift_kernel: one lane per (species class, pT) -- classes of bit-equal (mass, sign) in order of first appearance, members
  // in species order (see SpeciesClasses); the partial layout, n_bins and the evaluation count stay per species
  std::vector<double> cls_mass, cls_sign;
  std::vector<int32_t> cls_first, cls_members;
  if (svariant >= 0) {
    std::map<std::pair<uint64_t, uint64_t>, int> key_cls;
    std::vector<int> cls_of(sp->n);
    for (int i = 0; i < sp->n; i++) {
      uint64_t km, ks;
      memcpy(&km, &sp->mass[i], 8); memcpy(&ks, &sp->sign[i], 8);
      auto it = key_cls.emplace(std::make_pair(km, ks), (int)cls_mass.size()).first;
      if (it->second == (int)cls_mass.size()) { cls_mass.push_back(sp->mass[i]); cls_sign.push_back(sp->sign[i]); }
      cls_of[i] = it->second;
    }
    cls_first.assign(cls_mass.size() + 1, 0);
    for (int i = 0; i < sp->n; i++) cls_first[cls_of[i] + 1]++;
    for (size_t c = 0; c < cls_mass.size(); c++) cls_first[c + 1] += cls_first[c];
    cls_members.resize(sp->n);
    std::vector<int32_t> fill(cls_first.begin(), cls_first.end() - 1);
    for (int i = 0; i < sp->n; i++) cls_members[fill[cls_of[i]]++] = i;
  }
  const int n_lane_species = svariant >= 0 ? (int)cls_mass.size() : sp->n;
  const int n_pairs = n_lane_species * gr->n_pT;
  const int n_groups = (n_pairs + 31) / 32;
  int n_warps = max_warps;                                  // widest block whose padding wastes <= 4 % of the warps
  {
    int best = 1 << 30;
    for (int w = max_warps; w >= 1; w--) {
      const int launched = ((n_groups + w - 1) / w) * w;
      if ((launched - n_groups) * 25 <= launched) { n_warps = w; break; }
      if (launched < best) { best = launched; n_warps = w; }
    }
  }
  if (svariant >= 0) n_warps = 4;                           // cf_shift_kernel blocks are always 4 warps
  int n_groupblocks = (n_groups + n_warps - 1) / n_warps;
  if (fvariant >= 0) factored_blocking(sp->n, gr->n_pT, L.n_ptiles, &n_warps, &n_groupblocks);   // lanes = species, warps = phi tiles
  const int64_t n_bintiles = (int64_t)n_groupblocks * L.n_ytiles * (fvariant >= 0 ? 1 : L.n_ptiles);      // blocks per cell chunk
  int n_chunks = opt.n_chunks;
  int n_chunks_wanted = n_chunks;
  if (n_chunks <= 0) {
    // >= 64 waves at 3 blocks/SM: the last, partly filled wave costs < 1 % (a block lasts tens of ms, its fixed cost is us; at
    // 96 blocks per SM the 125 k-cell shards of an 8-GPU run lost 1.5 % to the tail)
    const int64_t target_blocks = (int64_t)g_sm_count * 192;
    n_chunks = (int)((target_blocks + n_bintiles - 1) / n_bintiles);
    // the blocks of one chunk run together (the grid is chunk-major) and each record is read by every block with that y / phi
    // tile: keep a chunk's records within a third of L2, or the blocks drift apart and re-read them from HBM
    // (measured at 90 k cells = 199 MB per chunk: 519 GB of DRAM reads for 2.2 GB of records, profiles/r2_traffic.json)
    const int64_t rec_per_cell = ((int64_t)L.n_ytiles * L.nst * L.rec_y + (int64_t)L.n_ptiles * L.npt * kRec + kScal) * 8;
    const int64_t l2_target = std::max<int64_t>((int64_t)Dp->l2_bytes / 3, (int64_t)8 << 20);
    const int64_t n_chunks_l2 = (n_cells * rec_per_cell + l2_target - 1) / l2_target;
    if (!iq && n_chunks_l2 > n_chunks) n_chunks = (int)std::min<int64_t>(n_chunks_l2, 1 << 20);
    n_chunks_wanted = n_chunks;                                         // reported next to the capped value (is3d_stats)
    const int64_t max_partial_bytes = (int64_t)4 << 30;                 // keep the partial buffer <= 4 GiB (8 GiB with the second feqmod set)
    int64_t cap = max_partial_bytes / (n_bins * 8 > 0 ? n_bins * 8 : 1);
    if (cap < 1) cap = 1;
    if (n_chunks > cap) n_chunks = (int)cap;
  }
  if ((int64_t)n_chunks > L.n_tiles) n_chunks = (int)(L.n_tiles > 0 ? L.n_tiles : 1);
  if (n_chunks < 1) n_chunks = 1;
  if ((int64_t)n_chunks_wanted > L.n_tiles) n_chunks_wanted = n_chunks;   // fewer cell tiles than chunks is not a cap
  // operation = 0, mode 1: a chunk never crosses a category; large categories are split into chunks of ~ n_tiles / n_chunks tiles
  std::vector<int64_t> gather_h, chunk_tiles_h;
  const int integ_sl = (n_warps * 32 - 1) / gr->n_pT + 2;
  if (iq && iq->mode == 1) {
    const int64_t per_chunk = std::max<int64_t>(1, (L.n_tiles + n_chunks - 1) / n_chunks);
    std::vector<int64_t> cat_first(cat_tiles.size() + 1, 0);              // first record position of every category
    for (size_t c = 0; c < cat_tiles.size(); c++) cat_first[c + 1] = cat_first[c] + cat_tiles[c] * ct;
    gather_h.assign((size_t)L.n_cells_pad, -1);
    {
      std::vector<int64_t> fill(cat_first.begin(), cat_first.end() - 1);
      for (int64_t i = 0; i < n_cells; i++) gather_h[(size_t)fill[(size_t)iq->category[i]]++] = i;     // stable: cell order kept inside a category
    }
    iq->unit_category.clear();
    chunk_tiles_h.push_back(0);
    for (size_t c = 0; c < cat_tiles.size(); c++) {
      const int64_t t0 = cat_first[c] / ct;
      for (int64_t t = 0; t < cat_tiles[c]; t += per_chunk) {
        chunk_tiles_h.push_back(t0 + std::min(cat_tiles[c], t + per_chunk));
        iq->unit_category.push_back((int32_t)c);
      }
    }
    n_chunks = (int)iq->unit_category.size();
    iq->n_units = n_chunks;
  } else if (iq) {
    iq->n_units = L.n_ytiles * L.nst;
  }
  if (n_bintiles * (int64_t)n_chunks > 2147483647LL) return fail(IS3D_ERR_ARGUMENT, "grid too large");
  const int64_t integ_rows = iq ? (int64_t)n_chunks * L.n_ytiles * (iq->mode == 2 ? L.nst : 1) : 0;
  const size_t integ_bytes = (size_t)integ_rows * L.n_ptiles * n_groupblocks * integ_sl * 8;
  if (iq && integ_bytes > ((size_t)8 << 30)) return fail(IS3D_ERR_ARGUMENT, "too many (tau, r) bins for the integration workspace");

  // ---- small tables -> one staging buffer
  SmallArena ar;
  std::vector<double> cosphi(gr->n_phi), sinphi(gr->n_phi);
  for (int k = 0; k < gr->n_phi; k++) { cosphi[k] = cos(gr->phi[k]); sinphi[k] = sin(gr->phi[k]); }   // smooth_kernels.cpp:43-48
  std::vector<double> zero_baryon(sp->n, 0.0);
  const size_t o_mass = ar.put(sp->mass, sp->n), o_sign = ar.put(sp->sign, sp->n), o_deg = ar.put(sp->degeneracy, sp->n);
  const size_t o_bar = ar.put(sp->baryon ? sp->baryon : zero_baryon.data(), sp->n);
  size_t o_cmass = 0, o_csign = 0, o_cfirst = 0, o_cmembers = 0;
  if (svariant >= 0) {
    o_cmass = ar.put(cls_mass.data(), cls_mass.size()); o_csign = ar.put(cls_sign.data(), cls_sign.size());
    o_cfirst = ar.put(cls_first.data(), cls_first.size()); o_cmembers = ar.put(cls_members.data(), cls_members.size());
  }
  const size_t o_pT = ar.put(gr->pT, gr->n_pT), o_cos = ar.put(cosphi.data(), gr->n_phi), o_sin = ar.put(sinphi.data(), gr->n_phi);
  const size_t o_sloty = dim2 ? ar.put(gr->eta, gr->n_eta) : ar.put(gr->y, gr->n_y);
  const size_t o_slotw = dim2 ? ar.put(gr->eta_weight, gr->n_eta) : 0;
  struct SplineOff { size_t x, y, c; int n; };
  auto put_spline = [&](const double *x, const double *y, int n) {
    SplineOff o{0, 0, 0, 0};
    if (!x || !y || n < 3) return o;
    std::vector<double> c(n);
    host_spline_init(x, y, n, c.data());
    o.x = ar.put(x, n); o.y = ar.put(y, n); o.c = ar.put(c.data(), n); o.n = n;
    return o;
  };
  SplineOff s_c0{}, s_c2{}, s_F{}, s_bb{}, s_bp{}, s_l2{}, s_z{};
  size_t o_r1 = 0, o_w1 = 0, o_r2 = 0, o_w2 = 0;
  if (!vah) {
    s_c0 = put_spline(df->T, df->c0, df->n_T); s_c2 = put_spline(df->T, df->c2, df->n_T); s_F = put_spline(df->T, df->F, df->n_T);
    s_bb = put_spline(df->T, df->betabulk, df->n_T); s_bp = put_spline(df->T, df->betapi, df->n_T);
    if (fl->df_mode == 4) { s_l2 = put_spline(df->jonah_x, df->jonah_lambda2, df->n_jonah); s_z = put_spline(df->jonah_x, df->jonah_z, df->n_jonah); }
    if (fl->df_mode == 3) {
      o_r1 = ar.put(gla->root1, gla->n_points); o_w1 = ar.put(gla->weight1, gla->n_points);
      o_r2 = ar.put(gla->root2, gla->n_points); o_w2 = ar.put(gla->weight2, gla->n_points);
    }
  }

  // ---- raw surface arrays
  const bool sh = fl->include_shear_deltaf != 0, bk = fl->include_bulk_deltaf != 0;
  struct RawItem { const double *src; bool need; const double **dst; };
  RawCells rc; memset(&rc, 0, sizeof(rc));
  rc.n = n_cells;
  RawItem items[] = {
    {sf->tau, true, &rc.tau}, {sf->eta, true, &rc.eta}, {sf->dat, true, &rc.dat}, {sf->dax, true, &rc.dax}, {sf->day, true, &rc.day},
    {sf->dan, true, &rc.dan}, {sf->ux, true, &rc.ux}, {sf->uy, true, &rc.uy}, {sf->un, true, &rc.un},
    {sf->T, !vah, &rc.T}, {sf->P, !vah, &rc.P}, {sf->E, !vah, &rc.E},
    {sf->pixx, vah || sh, &rc.pixx}, {sf->pixy, vah || sh, &rc.pixy}, {sf->pixn, vah || sh, &rc.pixn}, {sf->piyy, vah || sh, &rc.piyy},
    {sf->piyn, vah || sh, &rc.piyn}, {sf->bulkPi, bk, &rc.bulkPi},
    {sf->pitt, vah, &rc.pitt}, {sf->pitx, vah, &rc.pitx}, {sf->pity, vah, &rc.pity}, {sf->pitn, vah, &rc.pitn}, {sf->pinn, vah, &rc.pinn},
    {sf->Wx, vah, &rc.Wx}, {sf->Wy, vah, &rc.Wy}, {sf->Lambda, vah, &rc.Lambda}, {sf->aL, vah, &rc.aL},
    {sf->c0, vah, &rc.c0}, {sf->c1, vah, &rc.c1}, {sf->c2, vah, &rc.c2}, {sf->c3, vah, &rc.c3}, {sf->c4, vah, &rc.c4}};
  const int n_raw = (int)(sizeof(items) / sizeof(items[0]));
  for (int a = 0; a < n_raw; a++)
    if (items[a].need && !items[a].src && n_cells > 0) return fail(IS3D_ERR_ARGUMENT, "a required surface array is NULL");

  const size_t rec_Y = (size_t)L.n_ytiles * L.n_cells_pad * L.nst * L.rec_y * 8;
  const size_t rec_P = (size_t)L.n_ptiles * L.n_cells_pad * L.npt * kRec * 8;
  const size_t rec_S = (size_t)L.n_cells_pad * kScal * 8;
  const int partial_sets = feqmod ? 2 : 1;
  CU_CHECK(g_ws.small.reserve(ar.host.size() + 256));
  CU_CHECK(g_ws.Y.reserve(rec_Y + 256));
  CU_CHECK(g_ws.P.reserve(rec_P + 256));
  CU_CHECK(g_ws.S.reserve(rec_S + 256));
  if (feqmod) {
    CU_CHECK(g_ws.Y2.reserve(rec_Y + 256));
    CU_CHECK(g_ws.P2.reserve(rec_P + 256));
    CU_CHECK(g_ws.S2.reserve(rec_S + 256));
    if (fl->df_mode == 3) CU_CHECK(g_ws.extra.reserve(((size_t)L.n_species + 8) * L.n_cells_pad * 8 + 256));
  }
  if (!iq) CU_CHECK(g_ws.partial.reserve((size_t)partial_sets * n_chunks * n_bins * 8 + 256));
  // cf_shift_kernel reads e^{-pT (Bmax - B_k)} from a table that is formed for a window of consecutive chunks at a time (the
  // table kernel, then the hot kernel on those chunks): at ~3x the records per cell, a window is kept <= 4 GiB like the
  // partial buffer.  The chunk count above deliberately ignores the table.
  int win_chunks = n_chunks;
  int64_t e_cells = 0;
  if (svariant >= 0) {
    const int64_t chunk_cells = (L.n_tiles + n_chunks - 1) / n_chunks * L.ct;        // most cells a chunk holds
    const int64_t chunk_bytes = chunk_cells * L.n_ptiles * shift_table_record(L) * 8;
    const int64_t max_table_bytes = (int64_t)4 << 30;
    win_chunks = (int)std::max<int64_t>(1, std::min<int64_t>(n_chunks, chunk_bytes > 0 ? max_table_bytes / chunk_bytes : n_chunks));
    e_cells = win_chunks * chunk_cells;
    CU_CHECK(g_ws.E.reserve((size_t)e_cells * L.n_ptiles * shift_table_record(L) * 8 + 256));
  }
  if (iq) {
    CU_CHECK(g_ws.integ.reserve((size_t)partial_sets * integ_bytes + 256));
    CU_CHECK(g_ws.integ_out.reserve((size_t)partial_sets * iq->n_units * sp->n * 8 + 256));
    CU_CHECK(g_ws.gather.reserve((gather_h.size() + chunk_tiles_h.size() + (size_t)gr->n_pT + gr->n_phi) * 8 + 1024));
  }
  CU_CHECK(g_ws.counters.reserve(256));
  const size_t cell_stride = ((size_t)n_cells * 8 + 255) & ~(size_t)255;
  if (opt.memory == 0) {
    CU_CHECK(g_ws.raw.reserve(cell_stride * n_raw + 256));
    if (!iq) CU_CHECK(g_ws.dN.reserve((size_t)n_bins * 8 + 256));
  }

  cudaEvent_t *ev = g_ws.ev;
  CU_CHECK(cudaEventRecord(ev[0], st));
  // ---- host -> device
  unsigned char *small_d = g_ws.small.as<unsigned char>();
  CU_CHECK(cudaMemcpyAsync(small_d, ar.host.data(), ar.host.size(), cudaMemcpyHostToDevice, st));
  for (int a = 0; a < n_raw; a++) {
    *items[a].dst = nullptr;
    if (!items[a].need || n_cells == 0) continue;
    if (opt.memory == 0) {
      double *dst = reinterpret_cast<double *>(g_ws.raw.as<unsigned char>() + cell_stride * a);
      CU_CHECK(cudaMemcpyAsync(dst, items[a].src, (size_t)n_cells * 8, cudaMemcpyHostToDevice, st));
      *items[a].dst = dst;
    } else *items[a].dst = items[a].src;
  }
  const int64_t *gather_d = nullptr, *chunk_tiles_d = nullptr;
  const double *wpT_d = nullptr, *wphi_d = nullptr;
  if (iq) {
    unsigned char *g = g_ws.gather.as<unsigned char>();
    size_t off = 0;
    auto up = [&](const void *src, size_t bytes) -> const void * {
      const void *d = g + off;
      if (bytes) cudaMemcpyAsync(g + off, src, bytes, cudaMemcpyHostToDevice, st);
      off = (off + bytes + 255) & ~(size_t)255;
      return d;
    };
    if (iq->mode == 1) {
      gather_d = (const int64_t *)up(gather_h.data(), gather_h.size() * 8);
      chunk_tiles_d = (const int64_t *)up(chunk_tiles_h.data(), chunk_tiles_h.size() * 8);
    }
    wpT_d = (const double *)up(iq->pT_weight, (size_t)gr->n_pT * 8);
    wphi_d = (const double *)up(iq->phi_weight, (size_t)gr->n_phi * 8);
    CU_CHECK(cudaGetLastError());
    rc.gather = gather_d;
  }
  // memory == 1: the chunk sums go to a scratch buffer first, so that an error leaves the caller's array untouched
  const bool dev_scratch = !iq && opt.memory != 0 && !keep_dev;
  if (dev_scratch || (keep_dev && opt.memory != 0)) CU_CHECK(g_ws.dN.reserve((size_t)n_bins * 8 + 256));
  double *dN_dev = iq ? nullptr : g_ws.dN.as<double>();
  if (!iq) CU_CHECK(cudaMemsetAsync(dN_dev, 0, (size_t)n_bins * 8, st));
  CU_CHECK(cudaMemsetAsync(g_ws.counters.p, 0, sizeof(PrepCounters), st));
  CU_CHECK(cudaEventRecord(ev[1], st));

  // ---- prepare
  auto dptr = [&](size_t off) { return reinterpret_cast<const double *>(small_d + off); };
  PrepTables tab; memset(&tab, 0, sizeof(tab));
  auto mk = [&](const SplineOff &o) { Spline s; s.x = dptr(o.x); s.y = dptr(o.y); s.c = dptr(o.c); s.n = o.n; return s; };
  tab.c0 = mk(s_c0); tab.c2 = mk(s_c2); tab.F = mk(s_F); tab.betabulk = mk(s_bb); tab.betapi = mk(s_bp); tab.lam2 = mk(s_l2); tab.z = mk(s_z);
  tab.bulkPi_over_Peq_max = df ? df->bulkPi_over_Peq_max : 0.0;
  tab.cosphi = dptr(o_cos); tab.sinphi = dptr(o_sin); tab.slot_y = dptr(o_sloty); tab.slot_w = dim2 ? dptr(o_slotw) : nullptr;
  tab.gla_root1 = dptr(o_r1); tab.gla_w1 = dptr(o_w1); tab.gla_root2 = dptr(o_r2); tab.gla_w2 = dptr(o_w2); tab.gla_n = gla ? gla->n_points : 0;
  tab.deta_min = fl->deta_min; tab.mass_pion0 = fl->mass_pion0;
  tab.eta_delta = (dim2 && gr->n_eta > 1) ? gr->eta[1] - gr->eta[0] : 0.0;                    // smooth_kernels.cpp:2175
  PrepCounters *cnt_d = g_ws.counters.as<PrepCounters>();
  if (strict) {
    CU_CHECK(g_ws.Y.reserve((size_t)n_cells * strict_cell_bytes() + 256));
    CU_CHECK(launch_strict(*fl, rc, tab, L, dptr(o_mass), dptr(o_sign), dptr(o_deg), dptr(o_pT), dim2 ? gr->n_eta : 1,
                           pow(2.0 * M_PI * 0.197327053, -3), g_ws.Y.p, dN_dev, cnt_d, st));
    stt.gpu_launches += 2;
  } else if (vah) {
    CU_CHECK(launch_prepare_vah(*fl, rc, tab, L, g_ws.Y.as<double>(), g_ws.P.as<double>(), g_ws.S.as<double>(), cnt_d, st));
    stt.gpu_launches++;
  } else if (feqmod) {
    CU_CHECK(launch_prepare_feqmod(*fl, rc, tab, L, g_ws.Y.as<double>(), g_ws.P.as<double>(), g_ws.S.as<double>(),
                                   g_ws.Y2.as<double>(), g_ws.P2.as<double>(), g_ws.S2.as<double>(),
                                   dptr(o_mass), dptr(o_sign), dptr(o_deg), dptr(o_bar),
                                   fl->df_mode == 3 ? g_ws.extra.as<double>() : nullptr, cnt_d, st));
    stt.gpu_launches += (fl->df_mode == 3) ? 2 : 1;
  } else {
    CU_CHECK(launch_prepare_vh(*fl, rc, tab, L, g_ws.Y.as<double>(), g_ws.P.as<double>(), g_ws.S.as<double>(), cnt_d, st));
    stt.gpu_launches++;
  }
  CU_CHECK(cudaEventRecord(ev[2], st));
  // a cell outside the coefficient tables: the reference aborts without spectra -- stop before anything is added to the result
  PrepCounters cnt; memset(&cnt, 0, sizeof(cnt));
  CU_CHECK(cudaMemcpyAsync(&cnt, cnt_d, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  CU_CHECK(cudaStreamSynchronize(st));
  if (cnt.range_error) return fail(IS3D_ERR_TABLE_RANGE, "a cell's T or Pi/P lies outside the delta-f coefficient table (or T_mod <= 0)");

  // ---- hot kernel(s)
  HotParams hp; memset(&hp, 0, sizeof(hp));
  hp.L = L; hp.Y = g_ws.Y.as<double>(); hp.P = g_ws.P.as<double>(); hp.S = g_ws.S.as<double>();
  hp.mass = dptr(o_mass); hp.sign = dptr(o_sign); hp.degeneracy = dptr(o_deg); hp.pT = dptr(o_pT);
  hp.partial = g_ws.partial.as<double>();
  hp.renorm = (feqmod && fl->df_mode == 3) ? g_ws.extra.as<double>() : nullptr;
  hp.n_chunks = n_chunks; hp.n_groupblocks = n_groupblocks; hp.n_warps = n_warps;
  hp.regulate_thr = fl->regulate_deltaf ? 0x3ff00000 : 0x7ff80000;
  hp.one_hi = 0x3ff00000;
  hp.reg_lo = fl->regulate_deltaf ? 0 : (int)0x80000000; hp.reg_hi = fl->regulate_deltaf ? 0x40000000 : 0x7fffffff;
  hp.reg_chk = fl->regulate_deltaf ? 0x3fffffffu : 0xffffffffu;
  { const double ec[8] = {-369.3299304675746, 6755399441055744.0, -0.00270760617331689, -7.453964567463233e-13,      // = kExpR, kExpC (cf_device.cuh)
                          4.1666666666666664e-02, 1.6666666666666666e-01, 0.5, 0.0};
    for (int i = 0; i < 8; i++) hp.ec[i] = ec[i]; }
  hp.outflow_thr = (fl->outflow && !vah) ? 0LL : (long long)0x8000000000000000ULL;   // the anisotropic kernel has no Theta(p.dsigma)
  const double hbarC = 0.197327053;
  hp.pT_max = *std::max_element(gr->pT, gr->pT + gr->n_pT);
  hp.prefactor = vah ? 1.0 / (8.0 * (M_PI * M_PI * M_PI)) / hbarC / hbarC / hbarC      // smooth_kernels.cpp:2146
                     : pow(2.0 * M_PI * hbarC, -3);                                      // :36, :400
  if (iq) {
    hp.integ_mode = iq->mode; hp.integ_sl = integ_sl; hp.chunk_tiles = chunk_tiles_d;
    hp.pT_weight = wpT_d; hp.phi_weight = wphi_d; hp.integ = g_ws.integ.as<double>();
  }
  hp.E = g_ws.E.as<double>(); hp.e_cells = e_cells;
  int hot_launches = 1;
  if (strict) {}                                              // the bins were summed by launch_strict above
  else if (fvariant >= 0) CU_CHECK(launch_factored(model, hp, fvariant, st, nullptr));
  else if (svariant >= 0) {
    HotParams hs = hp;
    hs.mass = dptr(o_cmass); hs.sign = dptr(o_csign);
    SpeciesClasses cls;
    cls.n = n_lane_species;
    cls.first = reinterpret_cast<const int32_t *>(small_d + o_cfirst); cls.members = reinterpret_cast<const int32_t *>(small_d + o_cmembers);
    CU_CHECK(launch_shift(model, hs, cls, svariant, win_chunks, st, nullptr, &hot_launches));
  }
  else CU_CHECK(launch_hot(model, hp, variant, st, nullptr));
  if (!strict) stt.gpu_launches += hot_launches;
  int reduce_sets = 1;
  if (feqmod) {
    // cells where feqmod breaks down (and narrow-rapidity slots) take the linear-df branch: second pass, only if any
    if (cnt.linear_items > 0) {
      HotParams hl = hp;
      hl.Y = g_ws.Y2.as<double>(); hl.P = g_ws.P2.as<double>(); hl.S = g_ws.S2.as<double>();
      hl.partial = hp.partial + (size_t)n_chunks * n_bins; hl.renorm = nullptr;
      if (iq) hl.integ = hp.integ + integ_bytes / 8;
      // the linear branch runs on the factored kernel when one of its shapes has this register tile
      const int lin_model = fl->df_mode == 3 ? M_LINCE : M_JONAHLIN;
      const int lin_f = (factored_supported(lin_model, L) && !iq) ? factored_match(nyt, npt) : -1;
      if (lin_f >= 0) {
        factored_blocking(sp->n, gr->n_pT, L.n_ptiles, &hl.n_warps, &hl.n_groupblocks);
        if ((int64_t)hl.n_groupblocks * L.n_ytiles * n_chunks > 2147483647LL) return fail(IS3D_ERR_ARGUMENT, "grid too large");
        CU_CHECK(launch_factored(lin_model, hl, lin_f, st, nullptr));
      }
      else CU_CHECK(launch_hot(lin_model, hl, variant, st, nullptr));
      stt.gpu_launches++;
      reduce_sets = 2;
    }
  }
  CU_CHECK(cudaEventRecord(ev[3], st));

  // ---- reduce chunks, add into the result
  const size_t unit_vals = iq ? (size_t)iq->n_units * sp->n : 0;
  if (iq) {
    CU_CHECK(launch_integ_reduce(hp, iq->n_units, g_ws.integ_out.as<double>(), st));
    stt.gpu_launches++;
    if (reduce_sets == 2) {
      HotParams hl = hp; hl.integ = hp.integ + integ_bytes / 8;
      CU_CHECK(launch_integ_reduce(hl, iq->n_units, g_ws.integ_out.as<double>() + unit_vals, st));
      stt.gpu_launches++;
    }
  } else if (!strict) {
    CU_CHECK(launch_reduce(hp.partial, n_chunks * reduce_sets, n_bins, dim2 ? n_bins / gr->n_y : n_bins, dN_dev, st));
    stt.gpu_launches++;
  }
  CU_CHECK(cudaEventRecord(ev[4], st));

  // ---- device -> host / add into the caller's array
  std::vector<double> host_dN;
  if (iq) {
    iq->result.assign(unit_vals * reduce_sets, 0.0);
    if (unit_vals) CU_CHECK(cudaMemcpyAsync(iq->result.data(), g_ws.integ_out.p, unit_vals * reduce_sets * 8, cudaMemcpyDeviceToHost, st));
  } else if (keep_dev) {
    *keep_dev = dN_dev;
  } else if (opt.memory == 0) {
    host_dN.resize((size_t)n_bins);
    CU_CHECK(cudaMemcpyAsync(host_dN.data(), dN_dev, (size_t)n_bins * 8, cudaMemcpyDeviceToHost, st));
  } else {
    CU_CHECK(launch_axpy(dN_dev, dN_out, dim2 ? n_bins / gr->n_y : n_bins, st));       // dN_out += scratch (device pointers)
    stt.gpu_launches++;
  }
  CU_CHECK(cudaEventRecord(ev[5], st));
  CU_CHECK(cudaEventSynchronize(ev[5]));
  if (iq) {
    if (reduce_sets == 2) for (size_t i = 0; i < unit_vals; i++) iq->result[i] += iq->result[unit_vals + i];
    iq->result.resize(unit_vals);
  } else if (!keep_dev && opt.memory == 0)
    for (int64_t i = 0; i < n_bins; i++) dN_out[i] += host_dN[(size_t)i];

  float ms;
  cudaEventElapsedTime(&ms, ev[0], ev[1]); stt.h2d_ms = ms;
  cudaEventElapsedTime(&ms, ev[1], ev[2]); stt.prepare_ms = ms;
  cudaEventElapsedTime(&ms, ev[2], ev[3]); stt.kernel_ms = ms;
  cudaEventElapsedTime(&ms, ev[3], ev[4]); stt.reduce_ms = ms;
  cudaEventElapsedTime(&ms, ev[4], ev[5]); stt.d2h_ms = ms;
  cudaEventElapsedTime(&ms, ev[0], ev[5]); stt.total_ms = ms;
  stt.cells_skipped_udsigma = (int64_t)cnt.skipped;
  stt.cells_feqmod_breakdown = (int64_t)cnt.breakdown;
  stt.evaluations = n_cells * (int64_t)sp->n * gr->n_pT * gr->n_phi * (dim2 ? (int64_t)gr->n_eta : (int64_t)gr->n_y);
  stt.n_chunks = n_chunks; stt.tile_variant = strict ? kStrictVariant - 1 : variant;
  stt.n_chunks_wanted = n_chunks_wanted;
  stt.n_gpus = 1;
  if (stats) *stats = stt;
  return IS3D_OK;
}

}  // namespace is3d

extern "C" int is3d_b200_spacetime_distributions(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp,
                                                 const is3d_grid *gr, const is3d_df_tables *df, const is3d_laguerre *gla,
                                                 const is3d_spacetime_bins *bins, const is3d_options *opt_in,
                                                 is3d_spacetime_result *res, is3d_stats *stats)
{
  if (!fl || !sf || !sp || !gr || !bins || !res) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (!res->dN_tau || !res->dN_r || !res->dN_taur || !res->dN_dydeta || !res->dN_dy) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
  if (bins->tau_bins <= 0 || bins->r_bins <= 0 || !(bins->tau_max > bins->tau_min) || !(bins->r_max > bins->r_min))
    return fail(IS3D_ERR_ARGUMENT, "empty tau or r binning");
  if ((int64_t)(bins->tau_bins + 1) * (bins->r_bins + 1) > (1 << 24)) return fail(IS3D_ERR_ARGUMENT, "too many (tau, r) bins");
  const int64_t n = sf->n_cells;
  if (n < 0) return fail(IS3D_ERR_ARGUMENT, "negative cell count");
  if (n > 0 && (!sf->tau || !sf->x || !sf->y)) return fail(IS3D_ERR_ARGUMENT, "tau, x, y arrays are required");
  if (fl->mode == 2) return fail(IS3D_ERR_UNSUPPORTED, "spacetime distributions exist for mode 1 surfaces only");
  const bool device_mem = opt_in && opt_in->memory == 1;
  { Device *D0 = nullptr; int rc = current_device(&D0); if (rc) return rc; }

  // ---- (tau, r) category of every cell on the host (:1376-1379); index tau_bins / r_bins = outside the histogram
  std::vector<double> hbuf;
  const double *tau = sf->tau, *x = sf->x, *y = sf->y;
  if (device_mem && n > 0) {
    hbuf.resize((size_t)n * 3);
    cudaStream_t cs = (cudaStream_t)opt_in->stream;          // ordered after whatever produced the arrays on the caller's stream
    if (cudaMemcpyAsync(hbuf.data(), sf->tau, (size_t)n * 8, cudaMemcpyDeviceToHost, cs) != cudaSuccess ||
        cudaMemcpyAsync(hbuf.data() + n, sf->x, (size_t)n * 8, cudaMemcpyDeviceToHost, cs) != cudaSuccess ||
        cudaMemcpyAsync(hbuf.data() + 2 * n, sf->y, (size_t)n * 8, cudaMemcpyDeviceToHost, cs) != cudaSuccess ||
        cudaStreamSynchronize(cs) != cudaSuccess)
      return fail(IS3D_ERR_CUDA, "device -> host copy of tau, x, y failed");
    tau = hbuf.data(); x = tau + n; y = x + n;
  }
  const int nt = bins->tau_bins, nr = bins->r_bins;
  const double tau_width = (bins->tau_max - bins->tau_min) / (double)nt, r_width = (bins->r_max - bins->r_min) / (double)nr;
  auto bin_of = [](double v, int nb) { return (v >= 0.0 && v < (double)nb) ? (int)v : nb; };   // NaN, negative, beyond the range -> nb
  std::vector<int32_t> cat((size_t)n);
  for (int64_t i = 0; i < n; i++) {
    const double r = sqrt(x[i] * x[i] + y[i] * y[i]);
    const int itau = bin_of(floor((tau[i] - bins->tau_min) / tau_width), nt), ir = bin_of(floor((r - bins->r_min) / r_width), nr);
    cat[(size_t)i] = itau * (nr + 1) + ir;
  }

  const int ns = sp->n;
  const bool dim2 = (fl->dimension == 2);
  const int eta_pts = dim2 ? gr->n_eta : 1;
  IntegRequest iq;
  iq.mode = 1; iq.pT_weight = bins->pT_weight; iq.phi_weight = bins->phi_weight;
  iq.category = cat.data(); iq.n_categories = (nt + 1) * (nr + 1);
  is3d_stats st1; memset(&st1, 0, sizeof(st1));
  int rc = smooth_core(fl, sf, sp, gr, df, gla, opt_in, nullptr, &st1, &iq);
  if (rc) return rc;
  std::fill(res->dN_tau, res->dN_tau + (size_t)ns * nt, 0.0);
  std::fill(res->dN_r, res->dN_r + (size_t)ns * nr, 0.0);
  std::fill(res->dN_taur, res->dN_taur + (size_t)ns * nt * nr, 0.0);
  std::fill(res->dN_dydeta, res->dN_dydeta + (size_t)ns * eta_pts, 0.0);
  std::fill(res->dN_dy, res->dN_dy + (size_t)ns, 0.0);
  for (int u = 0; u < iq.n_units; u++) {                    // units come in (itau, ir) order: fixed summation order
    const int itau = iq.unit_category[(size_t)u] / (nr + 1), ir = iq.unit_category[(size_t)u] % (nr + 1);
    for (int s = 0; s < ns; s++) {
      const double v = iq.result[(size_t)u * ns + s];
      res->dN_dy[s] += v;
      if (itau < nt) {
        res->dN_tau[(size_t)s * nt + itau] += v;
        if (ir < nr) res->dN_taur[((size_t)s * nt + itau) * nr + ir] += v;
      }
      if (ir < nr) res->dN_r[(size_t)s * nr + ir] += v;
    }
  }
  if (!dim2) {
    for (int s = 0; s < ns; s++) res->dN_dydeta[s] = res->dN_dy[s];          // eta_weight = 1: the same sum (:1352 vs :1357)
  } else {
    // rapidity distribution: a second pass that keeps the eta slots apart and integrates over (pT, phi) only
    IntegRequest iq2;
    iq2.mode = 2; iq2.pT_weight = bins->pT_weight; iq2.phi_weight = bins->phi_weight;
    is3d_stats st2; memset(&st2, 0, sizeof(st2));
    rc = smooth_core(fl, sf, sp, gr, df, gla, opt_in, nullptr, &st2, &iq2);
    if (rc) return rc;
    for (int j = 0; j < eta_pts; j++) {
      const double w = gr->eta_weight[j];
      for (int s = 0; s < ns; s++) {
        const double v = iq2.result[(size_t)j * ns + s];
        res->dN_dydeta[(size_t)s * eta_pts + j] = (v == 0.0 && w == 0.0) ? 0.0 : v / w;
      }
    }
    st1.h2d_ms += st2.h2d_ms; st1.prepare_ms += st2.prepare_ms; st1.kernel_ms += st2.kernel_ms; st1.reduce_ms += st2.reduce_ms;
    st1.d2h_ms += st2.d2h_ms; st1.total_ms += st2.total_ms; st1.gpu_launches += st2.gpu_launches; st1.evaluations += st2.evaluations;
  }
  if (stats) *stats = st1;
  return IS3D_OK;
}

// Sampler mean yield (calculate_total_yield, emissionfunction_sampling_kernels.cpp:653-831) from per-species densities
extern "C" int is3d_b200_mean_yield(const is3d_flags *fl, const is3d_surface *sf, int32_t n_species, const double *neq,
                                    const double *dn_bulk, const is3d_df_tables *df, double y_cut, const is3d_options *opt_in,
                                    double *Ntot_out, is3d_stats *stats)
{
  if (!fl || !sf || !neq || !Ntot_out || n_species <= 0) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (fl->df_mode < 1 || fl->df_mode > 4) return fail(IS3D_ERR_ARGUMENT, "df_mode must be 1..4");
  if (fl->mode == 2) return fail(IS3D_ERR_UNSUPPORTED, "the sampler has no anisotropic-hydro yield estimate");
  if (fl->include_baryon) return fail(IS3D_ERR_UNSUPPORTED, "include_baryon = 1 (SURVEY R8)");
  if (fl->df_mode != 4 && !dn_bulk) return fail(IS3D_ERR_ARGUMENT, "df_mode 1-3 need the bulk density corrections");
  if (fl->df_mode == 4 && (!df || df->n_jonah < 3 || !df->jonah_x || !df->jonah_z)) return fail(IS3D_ERR_ARGUMENT, "df_mode 4 needs the Jonah z table");
  Device *Dp = nullptr;
  { int rc = current_device(&Dp); if (rc) return rc; }
  Workspace &g_ws = Dp->ws;
  std::lock_guard<std::mutex> lk(Dp->mu);
  is3d_options opt; memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  cudaStream_t st = (cudaStream_t)opt.stream;
  const int64_t n = sf->n_cells;
  if (n < 0) return fail(IS3D_ERR_ARGUMENT, "negative cell count");
  const bool bk = fl->include_bulk_deltaf != 0;
  const double *src[10] = {sf->tau, sf->ux, sf->uy, sf->un, sf->dat, sf->dax, sf->day, sf->dan, sf->bulkPi, sf->P};
  const bool need[10] = {true, true, true, true, true, true, true, true, bk, fl->df_mode == 4};
  for (int a = 0; a < 10; a++) if (need[a] && !src[a] && n > 0) return fail(IS3D_ERR_ARGUMENT, "a required surface array is NULL");

  SmallArena ar;
  size_t o_x = 0, o_y = 0, o_c = 0; int nz = 0;
  if (fl->df_mode == 4) {
    nz = df->n_jonah;
    std::vector<double> c(nz);
    host_spline_init(df->jonah_x, df->jonah_z, nz, c.data());
    o_x = ar.put(df->jonah_x, nz); o_y = ar.put(df->jonah_z, nz); o_c = ar.put(c.data(), nz);
  }
  const int n_blocks_max = (int)((n + 8191) / 8192) + 1;
  const size_t cell_stride = ((size_t)n * 8 + 255) & ~(size_t)255;
  CU_CHECK(g_ws.small.reserve(ar.host.size() + 256));
  CU_CHECK(g_ws.counters.reserve(256));
  CU_CHECK(g_ws.integ_out.reserve((size_t)n_blocks_max * 24 + 256));
  if (opt.memory == 0) CU_CHECK(g_ws.raw.reserve(cell_stride * 10 + 256));
  cudaEvent_t *ev = g_ws.ev;
  CU_CHECK(cudaEventRecord(ev[0], st));
  unsigned char *small_d = g_ws.small.as<unsigned char>();
  if (!ar.host.empty()) CU_CHECK(cudaMemcpyAsync(small_d, ar.host.data(), ar.host.size(), cudaMemcpyHostToDevice, st));
  const double *dev[10];
  for (int a = 0; a < 10; a++) {
    dev[a] = nullptr;
    if (!need[a] || n == 0) continue;
    if (opt.memory == 0) {
      double *d = reinterpret_cast<double *>(g_ws.raw.as<unsigned char>() + cell_stride * a);
      CU_CHECK(cudaMemcpyAsync(d, src[a], (size_t)n * 8, cudaMemcpyHostToDevice, st));
      dev[a] = d;
    } else dev[a] = src[a];
  }
  RawCells rc; memset(&rc, 0, sizeof(rc));
  rc.n = n; rc.tau = dev[0]; rc.ux = dev[1]; rc.uy = dev[2]; rc.un = dev[3]; rc.dat = dev[4]; rc.dax = dev[5]; rc.day = dev[6];
  rc.dan = dev[7]; rc.bulkPi = dev[8]; rc.P = dev[9];
  PrepTables tab; memset(&tab, 0, sizeof(tab));
  if (fl->df_mode == 4) {
    tab.z.x = reinterpret_cast<const double *>(small_d + o_x); tab.z.y = reinterpret_cast<const double *>(small_d + o_y);
    tab.z.c = reinterpret_cast<const double *>(small_d + o_c); tab.z.n = nz;
    tab.bulkPi_over_Peq_max = df->bulkPi_over_Peq_max;
  }
  CU_CHECK(cudaMemsetAsync(g_ws.counters.p, 0, sizeof(PrepCounters), st));
  CU_CHECK(cudaEventRecord(ev[1], st));
  int n_blocks = 0;
  CU_CHECK(launch_yield(rc, tab, fl->df_mode, bk ? 1 : 0, g_ws.integ_out.as<double>(), &n_blocks, g_ws.counters.as<PrepCounters>(), st));
  CU_CHECK(cudaEventRecord(ev[2], st));
  std::vector<double> part((size_t)n_blocks * 3, 0.0);
  PrepCounters cnt; memset(&cnt, 0, sizeof(cnt));
  if (n_blocks) CU_CHECK(cudaMemcpyAsync(part.data(), g_ws.integ_out.p, part.size() * 8, cudaMemcpyDeviceToHost, st));
  CU_CHECK(cudaMemcpyAsync(&cnt, g_ws.counters.p, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  CU_CHECK(cudaEventRecord(ev[3], st));
  CU_CHECK(cudaEventSynchronize(ev[3]));
  double S[3] = {0.0, 0.0, 0.0};
  for (int b = 0; b < n_blocks; b++) for (int q = 0; q < 3; q++) S[q] += part[(size_t)b * 3 + q];
  double Neq = 0.0, Nbulk = 0.0;
  for (int s = 0; s < n_species; s++) { Neq += neq[s]; if (dn_bulk) Nbulk += dn_bulk[s]; }
  double Ntot = (fl->df_mode == 4) ? S[2] * Neq : S[0] * Neq + S[1] * Nbulk;     // estimate_mean_particle_number, :200-236
  if (fl->dimension == 2) Ntot *= (2.0 * y_cut);                                  // :822-826
  *Ntot_out = Ntot;
  if (stats) {
    is3d_stats stt; memset(&stt, 0, sizeof(stt));
    float ms;
    cudaEventElapsedTime(&ms, ev[0], ev[1]); stt.h2d_ms = ms;
    cudaEventElapsedTime(&ms, ev[1], ev[2]); stt.kernel_ms = ms;
    cudaEventElapsedTime(&ms, ev[2], ev[3]); stt.d2h_ms = ms;
    cudaEventElapsedTime(&ms, ev[0], ev[3]); stt.total_ms = ms;
    stt.cells_skipped_udsigma = (int64_t)cnt.skipped; stt.gpu_launches = n_blocks ? 1 : 0;
    stt.evaluations = n * (int64_t)n_species;
    *stats = stt;
  }
  if (cnt.range_error) return fail(IS3D_ERR_TABLE_RANGE, "a cell's Pi/P lies outside the Jonah z table");
  return IS3D_OK;
}


// Resonance-decay feed-down (SURVEY 8f, row N3): see cf_decays.cu
static int check_decay_args(const is3d_particle_list *pdg, int32_t n_chosen, const int32_t *chosen, const is3d_grid *gr, int32_t dimension)
{
  if (!pdg || !chosen || !gr || n_chosen <= 0) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (dimension != 2 && dimension != 3) return fail(IS3D_ERR_ARGUMENT, "dimension must be 2 or 3");
  if (!pdg->mcid || !pdg->mass || !pdg->width || !pdg->stable || !pdg->decays || !pdg->dec_first || !pdg->dec_npart || !pdg->dec_br || !pdg->dec_part)
    return fail(IS3D_ERR_ARGUMENT, "incomplete particle list");
  if (!gr->pT || !gr->phi || !gr->y || gr->n_pT <= 0 || gr->n_phi <= 0 || gr->n_y <= 0) return fail(IS3D_ERR_ARGUMENT, "momentum tables missing");
  for (int i = 0; i < n_chosen; i++) if (chosen[i] < 0 || chosen[i] >= pdg->n_particles) return fail(IS3D_ERR_ARGUMENT, "chosen particle index out of range");
  return IS3D_OK;
}

extern "C" int is3d_b200_resonance_decays(const is3d_particle_list *pdg, int32_t n_chosen, const int32_t *chosen, const is3d_grid *gr,
                                          int32_t dimension, const is3d_options *opt_in, double *dN, is3d_stats *stats)
{
  if (!dN) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  { const int rc = check_decay_args(pdg, n_chosen, chosen, gr, dimension); if (rc) return rc; }
  Device *Dp = nullptr;
  { int rc = current_device(&Dp); if (rc) return rc; }
  Workspace &ws = Dp->ws;
  std::lock_guard<std::mutex> lk(Dp->mu);
  is3d_options opt; memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  cudaStream_t st = (cudaStream_t)opt.stream;
  const int64_t n_bins = (int64_t)n_chosen * gr->n_pT * gr->n_phi * gr->n_y;
  // the feed-down works on a scratch copy: an error (the reference exits there) leaves the caller's array untouched
  cudaEvent_t *ev = ws.ev;
  CU_CHECK(cudaEventRecord(ev[0], st));
  CU_CHECK(ws.dN.reserve((size_t)n_bins * 8 + 256));
  double *dev = ws.dN.as<double>();
  CU_CHECK(cudaMemcpyAsync(dev, dN, (size_t)n_bins * 8, opt.memory == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st));
  CU_CHECK(cudaEventRecord(ev[1], st));
  int launches = 0; std::string err;
  const int rc = resonance_decays_device(pdg, n_chosen, chosen, gr, dimension, dev, st, &launches, &err);
  if (rc != IS3D_OK) { cudaStreamSynchronize(st); return fail(rc, err.c_str()); }
  CU_CHECK(cudaEventRecord(ev[2], st));
  CU_CHECK(cudaMemcpyAsync(dN, dev, (size_t)n_bins * 8, opt.memory == 0 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
  CU_CHECK(cudaEventRecord(ev[3], st));
  CU_CHECK(cudaEventSynchronize(ev[3]));
  if (stats) {
    is3d_stats stt; memset(&stt, 0, sizeof(stt));
    float ms;
    cudaEventElapsedTime(&ms, ev[0], ev[1]); stt.h2d_ms = ms;
    cudaEventElapsedTime(&ms, ev[1], ev[2]); stt.kernel_ms = ms;
    cudaEventElapsedTime(&ms, ev[2], ev[3]); stt.d2h_ms = ms;
    cudaEventElapsedTime(&ms, ev[0], ev[3]); stt.total_ms = ms;
    stt.gpu_launches = launches; stt.n_gpus = 1;
    *stats = stt;
  }
  return IS3D_OK;
}

static int check_polarization_feed_down_args(const is3d_particle_list *pdg, const is3d_spin_parity *spin_parity, int32_t n_chosen,
                                             const int32_t *chosen, const is3d_grid *gr, int32_t dimension, const is3d_polarization_result *sums)
{
  if (!sums || !sums->St || !sums->Sx || !sums->Sy || !sums->Sz || !sums->Snorm) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
  { const int rc = check_decay_args(pdg, n_chosen, chosen, gr, dimension); if (rc) return rc; }
  if (!spin_parity || !spin_parity->spin2 || !spin_parity->parity) return fail(IS3D_ERR_ARGUMENT, "NULL spin / parity table");
  for (int i = 0; i < pdg->n_particles; i++) {
    if (spin_parity->spin2[i] < 0) return fail(IS3D_ERR_ARGUMENT, "negative 2J in the spin / parity table");
    if (spin_parity->parity[i] < -1 || spin_parity->parity[i] > 1) return fail(IS3D_ERR_ARGUMENT, "parity must be -1, 0 (unknown) or +1");
  }
  return IS3D_OK;
}

// The five arrays copied to the device workspace, run(dev, n_bins, st, &launches, &err) amending them there, and copied back only when it
// succeeds: an error leaves the caller's arrays untouched.
template <class Run>
static int polarization_feed_down_call(const is3d_grid *gr, int32_t n_chosen, const is3d_options *opt_in, is3d_polarization_result *sums,
                                       is3d_stats *stats, Run run)
{
  Device *Dp = nullptr;
  { int rc = current_device(&Dp); if (rc) return rc; }
  Workspace &ws = Dp->ws;
  std::lock_guard<std::mutex> lk(Dp->mu);
  is3d_options opt; memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  cudaStream_t st = (cudaStream_t)opt.stream;
  const int64_t n_bins = (int64_t)n_chosen * gr->n_pT * gr->n_phi * gr->n_y;
  double *const arr[5] = {sums->St, sums->Sx, sums->Sy, sums->Sz, sums->Snorm};
  const cudaMemcpyKind in = opt.memory == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const cudaMemcpyKind out = opt.memory == 0 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  cudaEvent_t *ev = ws.ev;
  CU_CHECK(cudaEventRecord(ev[0], st));
  CU_CHECK(ws.dN.reserve((size_t)n_bins * 8 * 5 + 256));
  double *dev = ws.dN.as<double>();
  for (int k = 0; k < 5; k++) CU_CHECK(cudaMemcpyAsync(dev + k * n_bins, arr[k], (size_t)n_bins * 8, in, st));
  CU_CHECK(cudaEventRecord(ev[1], st));
  int launches = 0; std::string err;
  const int rc = run(dev, n_bins, st, &launches, &err);
  if (rc != IS3D_OK) { cudaStreamSynchronize(st); return fail(rc, err.c_str()); }
  CU_CHECK(cudaEventRecord(ev[2], st));
  for (int k = 0; k < 5; k++) CU_CHECK(cudaMemcpyAsync(arr[k], dev + k * n_bins, (size_t)n_bins * 8, out, st));
  CU_CHECK(cudaEventRecord(ev[3], st));
  CU_CHECK(cudaEventSynchronize(ev[3]));
  if (stats) {
    is3d_stats stt; memset(&stt, 0, sizeof(stt));
    float ms;
    cudaEventElapsedTime(&ms, ev[0], ev[1]); stt.h2d_ms = ms;
    cudaEventElapsedTime(&ms, ev[1], ev[2]); stt.kernel_ms = ms;
    cudaEventElapsedTime(&ms, ev[2], ev[3]); stt.d2h_ms = ms;
    cudaEventElapsedTime(&ms, ev[0], ev[3]); stt.total_ms = ms;
    stt.gpu_launches = launches; stt.n_gpus = 1;
    *stats = stt;
  }
  return IS3D_OK;
}

// Feed-down of the spin-polarization sums through weak 2-body decays (cf_decays.cu), on the output of is3d_b200_polarization_decays.
extern "C" int is3d_b200_polarization_weak_decays(const is3d_particle_list *pdg, const is3d_spin_parity *spin_parity, const is3d_weak_decays *weak,
                                                  int32_t n_chosen, const int32_t *chosen, const is3d_grid *gr, int32_t dimension,
                                                  const is3d_options *opt_in, is3d_polarization_result *sums, is3d_stats *stats)
{
  { const int rc = check_polarization_feed_down_args(pdg, spin_parity, n_chosen, chosen, gr, dimension, sums); if (rc) return rc; }
  if (!weak) return fail(IS3D_ERR_ARGUMENT, "NULL weak decay table");
  if (weak->n < 0) return fail(IS3D_ERR_ARGUMENT, "weak decay table with n < 0");
  if (weak->n > 0 && (!weak->parent || !weak->daughter || !weak->partner || !weak->branching || !weak->alpha || !weak->phi))
    return fail(IS3D_ERR_ARGUMENT, "NULL row array in the weak decay table");
  { std::string err; const int rc = check_weak_decays(pdg, weak, &err); if (rc) return fail(rc, err.c_str()); }
  return polarization_feed_down_call(gr, n_chosen, opt_in, sums, stats, [&](double *dev, int64_t n_bins, cudaStream_t st, int *launches, std::string *err) {
    return polarization_weak_decays_device(pdg, spin_parity->spin2, weak, n_chosen, chosen, gr, dimension, dev, n_bins, st, launches, err);
  });
}

// Feed-down of the spin-polarization sums through 2-body decays (cf_decays.cu).  Like is3d_b200_resonance_decays it works on a device
// copy of all five arrays, so an error leaves the caller's arrays untouched.
extern "C" int is3d_b200_polarization_decays(const is3d_particle_list *pdg, const is3d_spin_parity *spin_parity, int32_t n_chosen,
                                             const int32_t *chosen, const is3d_grid *gr, int32_t dimension, const is3d_options *opt_in,
                                             is3d_polarization_result *sums, is3d_stats *stats)
{
  { const int rc = check_polarization_feed_down_args(pdg, spin_parity, n_chosen, chosen, gr, dimension, sums); if (rc) return rc; }
  return polarization_feed_down_call(gr, n_chosen, opt_in, sums, stats, [&](double *dev, int64_t n_bins, cudaStream_t st, int *launches, std::string *err) {
    return polarization_decays_device(pdg, spin_parity->spin2, spin_parity->parity, n_chosen, chosen, gr, dimension, dev, n_bins, st, launches, err);
  });
}

// =====================================================================================================================
// One process, several GPUs: contiguous cell shards, one host thread + stream per device, one NCCL all-reduce
// =====================================================================================================================
#include <dlfcn.h>
#include <thread>
#include <cstdlib>

namespace is3d {

// The handful of NCCL entry points used, resolved from libnccl.so.2 at run time (no link-time dependency; the ABI of these
// calls is stable across NCCL 2.x).  Declarations restate nccl.h.
typedef struct ncclComm *ncclComm_t;
enum { kNcclSuccess = 0, kNcclSum = 0, kNcclDouble = 8 };
struct Nccl {
  void *so = nullptr;
  int (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  bool load(std::string *err)
  {
    if (so) return true;
    const char *names[] = {getenv("IS3D_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char *n : names) { if (n && *n && (so = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break; }
    if (!so) { *err = std::string("cannot load libnccl.so.2 (set IS3D_B200_NCCL_LIB): ") + dlerror(); return false; }
    CommInitAll = (decltype(CommInitAll))dlsym(so, "ncclCommInitAll");
    CommDestroy = (decltype(CommDestroy))dlsym(so, "ncclCommDestroy");
    AllReduce = (decltype(AllReduce))dlsym(so, "ncclAllReduce");
    GroupStart = (decltype(GroupStart))dlsym(so, "ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))dlsym(so, "ncclGroupEnd");
    GetErrorString = (decltype(GetErrorString))dlsym(so, "ncclGetErrorString");
    if (!CommInitAll || !CommDestroy || !AllReduce || !GroupStart || !GroupEnd) { *err = "libnccl.so.2 lacks an expected symbol"; return false; }
    return true;
  }
};

static std::mutex g_multi_mutex;
static Nccl g_nccl;
static int g_ngpus = 1;
static std::vector<ncclComm_t> g_comms;
static std::vector<cudaStream_t> g_streams;

static void multi_shutdown()
{
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  int prev = 0; cudaGetDevice(&prev);
  for (size_t d = 0; d < g_comms.size(); d++) if (g_comms[d] && g_nccl.CommDestroy) g_nccl.CommDestroy(g_comms[d]);
  for (size_t d = 0; d < g_streams.size(); d++) if (g_streams[d]) { cudaSetDevice((int)d); cudaStreamDestroy(g_streams[d]); }
  g_comms.clear(); g_streams.clear(); g_ngpus = 1;
  cudaSetDevice(prev);
}

// cell shard of device d: contiguous, ceil(n / n_dev) cells (is3d_b200/distributed.py::shard_bounds)
static void shard_bounds(int64_t n, int d, int n_dev, int64_t *lo, int64_t *hi)
{
  const int64_t per = (n + n_dev - 1) / n_dev;
  *lo = std::min<int64_t>(n, per * d); *hi = std::min<int64_t>(n, per * (d + 1));
}

static is3d_surface shard_surface(const is3d_surface &s, int64_t lo, int64_t hi)
{
  is3d_surface o = s;
  o.n_cells = hi - lo;
  const double **src = reinterpret_cast<const double **>(reinterpret_cast<char *>(&o) + offsetof(is3d_surface, tau));
  const size_t n_ptr = (sizeof(is3d_surface) - offsetof(is3d_surface, tau)) / sizeof(double *);
  for (size_t a = 0; a < n_ptr; a++) if (src[a]) src[a] += lo;
  return o;
}

static void merge_stats(is3d_stats *acc, const is3d_stats &s)
{
  acc->cells_skipped_udsigma += s.cells_skipped_udsigma; acc->cells_feqmod_breakdown += s.cells_feqmod_breakdown;
  acc->evaluations += s.evaluations; acc->gpu_launches += s.gpu_launches;
  acc->h2d_ms = std::max(acc->h2d_ms, s.h2d_ms); acc->prepare_ms = std::max(acc->prepare_ms, s.prepare_ms);
  acc->kernel_ms = std::max(acc->kernel_ms, s.kernel_ms); acc->reduce_ms = std::max(acc->reduce_ms, s.reduce_ms);
  acc->d2h_ms = std::max(acc->d2h_ms, s.d2h_ms); acc->total_ms = std::max(acc->total_ms, s.total_ms);
  acc->n_chunks = s.n_chunks; acc->tile_variant = s.tile_variant; acc->n_chunks_wanted = s.n_chunks_wanted;
}

}  // namespace is3d

extern "C" int is3d_b200_device_count(void) { return g_ngpus; }

extern "C" int is3d_b200_init_devices(int n_gpus)
{
  int visible = 0;
  if (cudaGetDeviceCount(&visible) != cudaSuccess || visible == 0) return fail(IS3D_ERR_NO_DEVICE, "no CUDA device visible");
  if (n_gpus <= 0) {
    const char *e = getenv("IS3D_B200_GPUS");
    n_gpus = (e && atoi(e) > 0) ? atoi(e) : visible;
  }
  if (n_gpus > visible) return fail(IS3D_ERR_ARGUMENT, "more GPUs requested than visible");
  if (n_gpus > kMaxDevices) n_gpus = kMaxDevices;
  {
    std::lock_guard<std::mutex> lk(g_multi_mutex);
    if (n_gpus == g_ngpus && (n_gpus == 1 || !g_comms.empty())) return IS3D_OK;
  }
  multi_shutdown();
  int prev = 0; cudaGetDevice(&prev);
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  if (n_gpus > 1) {
    std::string err;
    if (!g_nccl.load(&err)) return fail(IS3D_ERR_NCCL, err.c_str());
    std::vector<int> devs(n_gpus);
    for (int d = 0; d < n_gpus; d++) devs[d] = d;
    g_comms.assign(n_gpus, nullptr);
    const int rc = g_nccl.CommInitAll(g_comms.data(), n_gpus, devs.data());
    if (rc != kNcclSuccess) { g_comms.clear(); return fail(IS3D_ERR_NCCL, g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "ncclCommInitAll failed"); }
    g_streams.assign(n_gpus, nullptr);
    for (int d = 0; d < n_gpus; d++) {
      CU_CHECK(cudaSetDevice(d));
      CU_CHECK(cudaStreamCreateWithFlags(&g_streams[d], cudaStreamNonBlocking));
      Device *D = nullptr;
      const int r2 = current_device(&D);
      if (r2) { cudaSetDevice(prev); return r2; }
    }
    CU_CHECK(cudaSetDevice(prev));
  }
  g_ngpus = n_gpus;
  return IS3D_OK;
}

extern "C" int is3d_b200_smooth_spectra_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                                              const is3d_df_tables *df, const is3d_laguerre *gla, const is3d_options *opt_in,
                                              double *dN_out, is3d_stats *stats)
{
  if (!fl || !sf || !sp || !gr || !dN_out) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  const int G = g_ngpus;
  if (G <= 1) return is3d_b200_smooth_spectra(fl, sf, sp, gr, df, gla, opt_in, dN_out, stats);
  if (opt_in && opt_in->memory != 0) return fail(IS3D_ERR_ARGUMENT, "the multi-GPU entry point takes host arrays");
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  const int64_t n_bins = (int64_t)sp->n * gr->n_pT * gr->n_phi * gr->n_y;
  struct DeviceGuard {            // whatever path leaves this function, the caller's current device is restored
    int prev = 0;
    DeviceGuard() { cudaGetDevice(&prev); }
    ~DeviceGuard() { cudaSetDevice(prev); }
  } guard;
  struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
  } ev;
  std::vector<int> rcs(G, IS3D_OK);
  std::vector<std::string> errs(G);
  std::vector<is3d_stats> sts(G);
  std::vector<double *> dev_dN(G, nullptr);
  std::vector<std::thread> workers;
  for (int d = 0; d < G; d++) {
    workers.emplace_back([&, d]() {
      memset(&sts[d], 0, sizeof(is3d_stats));
      if (cudaSetDevice(d) != cudaSuccess) { rcs[d] = IS3D_ERR_CUDA; errs[d] = "cudaSetDevice failed"; return; }
      int64_t lo, hi;
      shard_bounds(sf->n_cells, d, G, &lo, &hi);
      const is3d_surface shard = shard_surface(*sf, lo, hi);
      is3d_options opt; memset(&opt, 0, sizeof(opt));
      if (opt_in) opt = *opt_in;
      opt.memory = 0; opt.stream = g_streams[d];
      rcs[d] = smooth_core(fl, &shard, sp, gr, df, gla, &opt, nullptr, &sts[d], nullptr, &dev_dN[d]);
      if (rcs[d]) errs[d] = g_last_error;
    });
  }
  for (auto &w : workers) w.join();
  for (int d = 0; d < G; d++) if (rcs[d]) return fail(rcs[d], errs[d].c_str());

  // ---- the one collective of the path: sum of the spectra arrays over NVLink
  CU_CHECK(cudaSetDevice(0));
  CU_CHECK(cudaEventCreate(&ev.a)); CU_CHECK(cudaEventCreate(&ev.b));
  const cudaEvent_t e0 = ev.a, e1 = ev.b;
  CU_CHECK(cudaEventRecord(e0, g_streams[0]));
  int nrc = g_nccl.GroupStart();
  for (int d = 0; d < G && nrc == kNcclSuccess; d++)
    nrc = g_nccl.AllReduce(dev_dN[d], dev_dN[d], (size_t)n_bins, kNcclDouble, kNcclSum, g_comms[d], g_streams[d]);
  const int nrc2 = g_nccl.GroupEnd();
  if (nrc == kNcclSuccess) nrc = nrc2;
  if (nrc != kNcclSuccess) { return fail(IS3D_ERR_NCCL, g_nccl.GetErrorString ? g_nccl.GetErrorString(nrc) : "ncclAllReduce failed"); }
  CU_CHECK(cudaEventRecord(e1, g_streams[0]));
  std::vector<double> host((size_t)n_bins);
  CU_CHECK(cudaMemcpyAsync(host.data(), dev_dN[0], (size_t)n_bins * 8, cudaMemcpyDeviceToHost, g_streams[0]));
  for (int d = 0; d < G; d++) { CU_CHECK(cudaSetDevice(d)); CU_CHECK(cudaStreamSynchronize(g_streams[d])); }
  for (int64_t i = 0; i < n_bins; i++) dN_out[i] += host[(size_t)i];
  float ms = 0;
  CU_CHECK(cudaSetDevice(0));
  cudaEventElapsedTime(&ms, e0, e1);
  if (stats) {
    is3d_stats tot; memset(&tot, 0, sizeof(tot));
    for (int d = 0; d < G; d++) merge_stats(&tot, sts[d]);
    tot.n_gpus = G; tot.allreduce_ms = ms; tot.total_ms += ms;
    *stats = tot;
  }
  return IS3D_OK;
}

extern "C" int is3d_b200_spacetime_distributions_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp,
                                                       const is3d_grid *gr, const is3d_df_tables *df, const is3d_laguerre *gla,
                                                       const is3d_spacetime_bins *bins, const is3d_options *opt_in,
                                                       is3d_spacetime_result *res, is3d_stats *stats)
{
  const int G = g_ngpus;
  if (G <= 1) return is3d_b200_spacetime_distributions(fl, sf, sp, gr, df, gla, bins, opt_in, res, stats);
  if (!fl || !sf || !sp || !gr || !bins || !res) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (opt_in && opt_in->memory != 0) return fail(IS3D_ERR_ARGUMENT, "the multi-GPU entry point takes host arrays");
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  const int ns = sp->n, nt = bins->tau_bins, nr = bins->r_bins, eta_pts = fl->dimension == 2 ? gr->n_eta : 1;
  if (ns <= 0 || nt <= 0 || nr <= 0) return fail(IS3D_ERR_ARGUMENT, "empty species list or binning");
  const size_t sizes[5] = {(size_t)ns * nt, (size_t)ns * nr, (size_t)ns * nt * nr, (size_t)ns * eta_pts, (size_t)ns};
  size_t total = 0; for (size_t v : sizes) total += v;
  int prev = 0; cudaGetDevice(&prev);
  std::vector<int> rcs(G, IS3D_OK);
  std::vector<std::string> errs(G);
  std::vector<is3d_stats> sts(G);
  std::vector<std::vector<double>> bufs(G, std::vector<double>(total, 0.0));
  std::vector<std::thread> workers;
  for (int d = 0; d < G; d++) {
    workers.emplace_back([&, d]() {
      memset(&sts[d], 0, sizeof(is3d_stats));
      if (cudaSetDevice(d) != cudaSuccess) { rcs[d] = IS3D_ERR_CUDA; errs[d] = "cudaSetDevice failed"; return; }
      int64_t lo, hi;
      shard_bounds(sf->n_cells, d, G, &lo, &hi);
      const is3d_surface shard = shard_surface(*sf, lo, hi);
      is3d_options opt; memset(&opt, 0, sizeof(opt));
      if (opt_in) opt = *opt_in;
      opt.memory = 0; opt.stream = g_streams[d];
      double *b = bufs[d].data();
      is3d_spacetime_result r{b, b + sizes[0], b + sizes[0] + sizes[1], b + sizes[0] + sizes[1] + sizes[2], b + sizes[0] + sizes[1] + sizes[2] + sizes[3]};
      rcs[d] = is3d_b200_spacetime_distributions(fl, &shard, sp, gr, df, gla, bins, &opt, &r, &sts[d]);
      if (rcs[d]) errs[d] = g_last_error;
    });
  }
  for (auto &w : workers) w.join();
  cudaSetDevice(prev);
  for (int d = 0; d < G; d++) if (rcs[d]) return fail(rcs[d], errs[d].c_str());
  double *out[5] = {res->dN_tau, res->dN_r, res->dN_taur, res->dN_dydeta, res->dN_dy};
  size_t off = 0;
  for (int q = 0; q < 5; q++) {
    if (!out[q]) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
    for (size_t i = 0; i < sizes[q]; i++) { double v = 0.0; for (int d = 0; d < G; d++) v += bufs[d][off + i]; out[q][i] = v; }
    off += sizes[q];
  }
  // 2+1D: dN_dydeta is a quotient by the eta weight per device shard; the quotients add because the weight is the same
  if (stats) {
    is3d_stats tot; memset(&tot, 0, sizeof(tot));
    for (int d = 0; d < G; d++) merge_stats(&tot, sts[d]);
    tot.n_gpus = G;
    *stats = tot;
  }
  return IS3D_OK;
}

// =====================================================================================================================
// Spin polarization from thermal vorticity (cf_polzn.cu), thermal shear (cf_polzn_xi.cu) and the spin Hall effect (cf_polzn_she.cu): raw
// sums N^mu and Snorm, added into the caller's five arrays; spin density matrix from thermal vorticity (cf_spin_density.cu): nine raw sums
// =====================================================================================================================
namespace is3d {

enum PolTerm { kPolVorticity, kPolShear, kPolSpinDensity, kPolSpinHall };

// result arrays per term, in the order of the kernel's partial rows; the fifth array (St) of the shear and spin Hall terms must be
// non-NULL but is left alone (N_xi^t = N_she^t = 0 exactly)
static int pol_n_out(PolTerm term) { return term == kPolSpinDensity ? kSdSums : 5; }

// tensor: the 6 vorticity columns (vorticity, spin density), the 10 thermal-shear columns (shear) or the 4 columns of d alpha_B (spin
// Hall), NULL for a NULL struct.  out: the pol_n_out(term) result arrays, NULL for a NULL result struct.  The vorticity, shear and spin
// Hall terms run on the same layout and chunk split, so their Snorm is bit-identical.  The spin-density kernel has its own register tile but the same cell chunks, so at varpi = 0 its Snorm is
// bit-identical too (unless the 4 GiB cap on its nine partial arrays lowers the chunk count).
static int polzn_core(const is3d_flags *fl, const is3d_surface *sf, const double *const *tensor, PolTerm term, const is3d_species *sp,
                      const is3d_grid *gr, const is3d_options *opt_in, double *const *out, is3d_stats *stats)
{
  const bool shear = (term == kPolShear), she = (term == kPolSpinHall);
  const int n_tensor = shear ? 10 : she ? 4 : 6;
  if (!fl || !sf || !sp || !gr || !out) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (!tensor) return fail(IS3D_ERR_ARGUMENT, shear ? "NULL thermal shear" : she ? "NULL baryon gradient" : "NULL vorticity");
  for (int q = 0; q < pol_n_out(term); q++) if (!out[q]) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
  if (fl->mode == 2) return fail(IS3D_ERR_UNSUPPORTED, "spin polarization needs a viscous-hydro surface with thermal vorticity (mode 5), not mode 2");
  if (fl->include_baryon) return fail(IS3D_ERR_UNSUPPORTED, "include_baryon = 1 (the reference's (T, muB) lookup reads out of bounds, SURVEY R8)");
  if (fl->dimension != 2 && fl->dimension != 3) return fail(IS3D_ERR_ARGUMENT, "dimension must be 2 or 3");
  if (sp->n <= 0 || gr->n_pT <= 0 || gr->n_phi <= 0 || gr->n_y <= 0) return fail(IS3D_ERR_ARGUMENT, "empty species list or momentum table");
  if (!sp->mass || !sp->sign || !sp->degeneracy || !gr->pT || !gr->phi || !gr->y) return fail(IS3D_ERR_ARGUMENT, "NULL species or momentum table");
  if (she && !sp->baryon) return fail(IS3D_ERR_ARGUMENT, "the spin Hall term needs the species' baryon numbers (NULL species table)");
  for (int s = 0; s < sp->n; s++) if (!(sp->mass[s] > 0.0)) return fail(IS3D_ERR_ARGUMENT, "spin polarization needs species with mass > 0");
  if (term == kPolSpinDensity)
    for (int s = 0; s < sp->n; s++) {
      const double g = sp->degeneracy[s];
      if (!(g >= 1.0 && g <= 16.0 && g == std::floor(g)))
        return fail(IS3D_ERR_ARGUMENT, "the spin density needs species whose degeneracy 2J + 1 is an integer in [1, 16]");
    }
  const bool dim2 = (fl->dimension == 2);
  if (dim2 && (gr->n_eta <= 0 || !gr->eta || !gr->eta_weight)) return fail(IS3D_ERR_ARGUMENT, "dimension = 2 needs the eta table");
  const int64_t n_cells = sf->n_cells;
  if (n_cells < 0) return fail(IS3D_ERR_ARGUMENT, "negative cell count");
  const double *srcs[20] = {sf->tau, sf->eta, sf->dat, sf->dax, sf->day, sf->dan, sf->ux, sf->uy, sf->un, sf->T};
  for (int a = 0; a < n_tensor; a++) srcs[10 + a] = tensor[a];
  const int n_src = 10 + n_tensor;
  for (int a = 0; a < n_src; a++)
    if (!srcs[a] && n_cells > 0)
      return fail(IS3D_ERR_ARGUMENT, shear ? "a required surface or thermal-shear array is NULL"
                                     : she ? "a required surface or baryon-gradient array is NULL" : "a required surface or vorticity array is NULL");
  Device *Dp = nullptr;
  { int rc = current_device(&Dp); if (rc) return rc; }
  Workspace &ws = Dp->ws;
  std::lock_guard<std::mutex> lk(Dp->mu);
  is3d_options opt; memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  cudaStream_t st = (cudaStream_t)opt.stream;
  const int64_t n_bins = (int64_t)sp->n * gr->n_pT * gr->n_phi * gr->n_y;
  const int64_t n_active = dim2 ? n_bins / gr->n_y : n_bins;        // 2+1D fills the y = 0 plane (index iy = 0)

  // ---- layout: the cf_kernel decomposition with the register tile of the term's kernel
  Layout L; memset(&L, 0, sizeof(L));
  L.n_species = sp->n; L.n_pT = gr->n_pT; L.n_phi = gr->n_phi; L.n_y_out = gr->n_y;
  L.dim2 = dim2 ? 1 : 0;
  L.n_slots = dim2 ? gr->n_eta : gr->n_y;
  L.rec_y = kPolRecY;
  int nyt, npt, ct, vnyt, vnpt, vct;
  polzn_shape(L.dim2, &vnyt, &vnpt, &vct);
  if (term == kPolSpinDensity) spin_density_shape(L.dim2, &nyt, &npt, &ct);
  else { nyt = vnyt; npt = vnpt; ct = vct; }
  L.nst = dim2 ? L.n_slots : nyt;
  L.n_ytiles = dim2 ? 1 : (L.n_slots + nyt - 1) / nyt;
  L.npt = npt; L.n_ptiles = (L.n_phi + npt - 1) / npt;
  L.ct = ct; L.n_cells = n_cells;
  L.n_tiles = (n_cells + ct - 1) / ct;
  L.n_cells_pad = L.n_tiles * ct;
  const int n_groups = (sp->n * gr->n_pT + 31) / 32;
  const int n_warps = std::min(kPolWarps, n_groups);
  const int n_groupblocks = (n_groups + n_warps - 1) / n_warps;
  const int64_t n_bintiles = (int64_t)n_groupblocks * L.n_ytiles * L.n_ptiles;
  // chunks: the rule of smooth_core (>= 192 blocks per SM, a chunk's records within a third of L2, partial sums <= 4 GiB), evaluated
  // on the tile of cf_polzn_kernel for every term (same cells per TMA tile), so that all terms split the cells alike
  const int64_t v_ytiles = dim2 ? 1 : (L.n_slots + vnyt - 1) / vnyt, v_ptiles = (L.n_phi + vnpt - 1) / vnpt;
  const int64_t v_bintiles = (int64_t)n_groupblocks * v_ytiles * v_ptiles;
  int64_t n_chunks = ((int64_t)Dp->sm_count * 192 + v_bintiles - 1) / v_bintiles;
  const int64_t rec_per_cell = (v_ytiles * (dim2 ? L.n_slots : vnyt) * kPolRecY + v_ptiles * vnpt * kPolRecP) * 8;
  const int64_t l2_target = std::max<int64_t>((int64_t)Dp->l2_bytes / 3, (int64_t)8 << 20);
  n_chunks = std::max<int64_t>(n_chunks, (n_cells * rec_per_cell + l2_target - 1) / l2_target);
  const int64_t n_chunks_wanted = n_chunks;
  const int n_part = (term == kPolSpinDensity) ? kSdSums : 5;       // partial arrays the 4 GiB cap counts (shear, spin Hall keep 5)
  n_chunks = std::min<int64_t>(n_chunks, std::max<int64_t>(1, ((int64_t)4 << 30) / (n_part * n_bins * 8)));
  if (opt.n_chunks > 0) n_chunks = opt.n_chunks;
  n_chunks = std::max<int64_t>(1, std::min<int64_t>(n_chunks, std::max<int64_t>(L.n_tiles, 1)));
  if (n_bintiles * n_chunks > 2147483647LL) return fail(IS3D_ERR_ARGUMENT, "grid too large");

  // ---- tables and surface to the device
  SmallArena ar;
  std::vector<double> cosphi(gr->n_phi), sinphi(gr->n_phi);
  for (int k = 0; k < gr->n_phi; k++) { cosphi[k] = cos(gr->phi[k]); sinphi[k] = sin(gr->phi[k]); }
  const size_t o_mass = ar.put(sp->mass, sp->n), o_sign = ar.put(sp->sign, sp->n), o_deg = ar.put(sp->degeneracy, sp->n);
  const size_t o_pT = ar.put(gr->pT, gr->n_pT), o_cos = ar.put(cosphi.data(), gr->n_phi), o_sin = ar.put(sinphi.data(), gr->n_phi);
  const size_t o_sloty = dim2 ? ar.put(gr->eta, gr->n_eta) : ar.put(gr->y, gr->n_y);
  const size_t o_slotw = dim2 ? ar.put(gr->eta_weight, gr->n_eta) : 0;
  const size_t o_bar = she ? ar.put(sp->baryon, sp->n) : 0;
  const size_t cell_stride = ((size_t)n_cells * 8 + 255) & ~(size_t)255;
  CU_CHECK(ws.small.reserve(ar.host.size() + 256));
  CU_CHECK(ws.Y.reserve((size_t)L.n_ytiles * L.n_cells_pad * L.nst * kPolRecY * 8 + 256));
  CU_CHECK(ws.P.reserve((size_t)L.n_ptiles * L.n_cells_pad * L.npt * kPolRecP * 8 + 256));
  CU_CHECK(ws.partial.reserve((size_t)n_part * n_chunks * n_bins * 8 + 256));
  CU_CHECK(ws.dN.reserve((size_t)n_part * n_bins * 8 + 256));
  CU_CHECK(ws.counters.reserve(256));
  if (opt.memory == 0) CU_CHECK(ws.raw.reserve(cell_stride * n_src + 256));

  cudaEvent_t *ev = ws.ev;
  CU_CHECK(cudaEventRecord(ev[0], st));
  unsigned char *small_d = ws.small.as<unsigned char>();
  CU_CHECK(cudaMemcpyAsync(small_d, ar.host.data(), ar.host.size(), cudaMemcpyHostToDevice, st));
  const double *dev[20];
  for (int a = 0; a < n_src; a++) {
    dev[a] = srcs[a];
    if (opt.memory == 0) {
      double *d = reinterpret_cast<double *>(ws.raw.as<unsigned char>() + cell_stride * a);
      if (n_cells > 0) CU_CHECK(cudaMemcpyAsync(d, srcs[a], (size_t)n_cells * 8, cudaMemcpyHostToDevice, st));
      dev[a] = d;
    }
  }
  RawCells rc; memset(&rc, 0, sizeof(rc));
  rc.n = n_cells; rc.tau = dev[0]; rc.eta = dev[1]; rc.dat = dev[2]; rc.dax = dev[3]; rc.day = dev[4]; rc.dan = dev[5];
  rc.ux = dev[6]; rc.uy = dev[7]; rc.un = dev[8]; rc.T = dev[9];
  const int n_arr = (shear || she) ? 4 : pol_n_out(term);
  double *sums_d = ws.dN.as<double>();                         // [n_arr][n_bins] in the order of out
  CU_CHECK(cudaMemsetAsync(sums_d, 0, (size_t)n_arr * n_bins * 8, st));
  CU_CHECK(cudaMemsetAsync(ws.counters.p, 0, sizeof(PrepCounters), st));
  CU_CHECK(cudaEventRecord(ev[1], st));

  auto dptr = [&](size_t off) { return reinterpret_cast<const double *>(small_d + off); };
  PrepTables tab; memset(&tab, 0, sizeof(tab));
  tab.cosphi = dptr(o_cos); tab.sinphi = dptr(o_sin); tab.slot_y = dptr(o_sloty); tab.slot_w = dim2 ? dptr(o_slotw) : nullptr;
  PrepCounters *cnt_d = ws.counters.as<PrepCounters>();
  if (shear) {
    ShearCells xc;
    for (int a = 0; a < 10; a++) xc.x[a] = dev[10 + a];
    CU_CHECK(launch_prepare_polzn_xi(rc, xc, tab, L, ws.Y.as<double>(), ws.P.as<double>(), cnt_d, st));
  } else if (she) {
    const GradientCells gc{{dev[10], dev[11], dev[12], dev[13]}};
    CU_CHECK(launch_prepare_polzn_she(rc, gc, tab, L, ws.Y.as<double>(), ws.P.as<double>(), cnt_d, st));
  } else {
    const VortCells vc{dev[10], dev[11], dev[12], dev[13], dev[14], dev[15]};
    CU_CHECK(launch_prepare_polzn(rc, vc, tab, L, ws.Y.as<double>(), ws.P.as<double>(), cnt_d, st));
  }
  CU_CHECK(cudaEventRecord(ev[2], st));

  HotParams hp; memset(&hp, 0, sizeof(hp));
  hp.L = L; hp.Y = ws.Y.as<double>(); hp.P = ws.P.as<double>();
  hp.mass = dptr(o_mass); hp.sign = dptr(o_sign); hp.degeneracy = dptr(o_deg); hp.pT = dptr(o_pT);
  hp.partial = ws.partial.as<double>();
  hp.n_chunks = (int)n_chunks; hp.n_groupblocks = n_groupblocks; hp.n_warps = n_warps;
  hp.outflow_thr = fl->outflow ? 0LL : (long long)0x8000000000000000ULL;
  hp.prefactor = pow(2.0 * M_PI * 0.197327053, -3);
  if (shear) {
    const PolXiParams prm{hp, dptr(o_cos), dptr(o_sin), dim2 ? nullptr : dptr(o_sloty)};
    CU_CHECK(launch_polzn_xi(prm, st));
  } else if (she) {
    const PolSheParams prm{hp, dptr(o_cos), dptr(o_sin), dim2 ? nullptr : dptr(o_sloty), dptr(o_bar)};
    CU_CHECK(launch_polzn_she(prm, st));
  } else if (term == kPolSpinDensity) {
    // the prepare kernel never touches range_error: here it counts the boson evaluations without a valid occupation
    const SpinDensityParams prm{hp, dim2 ? nullptr : dptr(o_sloty), &cnt_d->range_error};
    CU_CHECK(launch_spin_density(prm, st));
  } else {
    CU_CHECK(launch_polzn(hp, st));
  }
  CU_CHECK(cudaEventRecord(ev[3], st));
  for (int q = 0; q < n_arr; q++)
    CU_CHECK(launch_reduce(hp.partial + (size_t)q * n_chunks * n_bins, (int)n_chunks, n_bins, n_active, sums_d + (size_t)q * n_bins, st));
  CU_CHECK(cudaEventRecord(ev[4], st));
  if (term == kPolSpinDensity) {
    // decided before anything is added to the caller's arrays, like the table-range errors of smooth_core
    PrepCounters c0; memset(&c0, 0, sizeof(c0));
    CU_CHECK(cudaMemcpyAsync(&c0, cnt_d, sizeof(c0), cudaMemcpyDeviceToHost, st));
    CU_CHECK(cudaStreamSynchronize(st));
    if (c0.range_error) {
      char msg[256];
      snprintf(msg, sizeof(msg), "%llu boson evaluations have u.p/T - J theta <= 0: the spin level m = J has no valid occupation "
               "(thermal vorticity too large for this surface)", c0.range_error);
      return fail(IS3D_ERR_ARGUMENT, msg);
    }
  }

  std::vector<double> host;
  if (opt.memory == 0) {
    host.resize((size_t)n_arr * n_bins);
    CU_CHECK(cudaMemcpyAsync(host.data(), sums_d, (size_t)n_arr * n_bins * 8, cudaMemcpyDeviceToHost, st));
  } else {
    for (int q = 0; q < n_arr; q++) CU_CHECK(launch_axpy(sums_d + (size_t)q * n_bins, out[q], n_active, st));
  }
  PrepCounters cnt; memset(&cnt, 0, sizeof(cnt));
  CU_CHECK(cudaMemcpyAsync(&cnt, cnt_d, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  CU_CHECK(cudaEventRecord(ev[5], st));
  CU_CHECK(cudaEventSynchronize(ev[5]));
  if (opt.memory == 0)
    for (int q = 0; q < n_arr; q++)
      for (int64_t i = 0; i < n_bins; i++) out[q][i] += host[(size_t)q * n_bins + i];

  is3d_stats stt; memset(&stt, 0, sizeof(stt));
  float ms;
  cudaEventElapsedTime(&ms, ev[0], ev[1]); stt.h2d_ms = ms;
  cudaEventElapsedTime(&ms, ev[1], ev[2]); stt.prepare_ms = ms;
  cudaEventElapsedTime(&ms, ev[2], ev[3]); stt.kernel_ms = ms;
  cudaEventElapsedTime(&ms, ev[3], ev[4]); stt.reduce_ms = ms;
  cudaEventElapsedTime(&ms, ev[4], ev[5]); stt.d2h_ms = ms;
  cudaEventElapsedTime(&ms, ev[0], ev[5]); stt.total_ms = ms;
  stt.cells_skipped_udsigma = (int64_t)cnt.skipped;
  stt.evaluations = n_cells * (int64_t)sp->n * gr->n_pT * gr->n_phi * (int64_t)L.n_slots;
  stt.gpu_launches = (n_cells > 0 ? 1 : 0) + 1 + n_arr + (opt.memory == 0 ? 0 : n_arr);
  stt.n_chunks = (int)n_chunks; stt.n_chunks_wanted = (int)n_chunks_wanted;
  stt.n_gpus = 1;
  if (stats) *stats = stt;
  return IS3D_OK;
}

}  // namespace is3d

namespace is3d {

// Several devices: HOST arrays, contiguous cell shards, one thread per device; the raw sums are added on the host in device order
static int polzn_multi(const is3d_flags *fl, const is3d_surface *sf, const double *const *tensor, PolTerm term, const is3d_species *sp,
                       const is3d_grid *gr, const is3d_options *opt_in, double *const *out, is3d_stats *stats)
{
  const int G = g_ngpus;
  const bool shear = (term == kPolShear), she = (term == kPolSpinHall);
  if (G <= 1) return polzn_core(fl, sf, tensor, term, sp, gr, opt_in, out, stats);
  if (!fl || !sf || !tensor || !sp || !gr || !out)
    return fail(IS3D_ERR_ARGUMENT, tensor ? "NULL argument" : shear ? "NULL thermal shear" : she ? "NULL baryon gradient" : "NULL vorticity");
  if (opt_in && opt_in->memory != 0) return fail(IS3D_ERR_ARGUMENT, "the multi-GPU entry point takes host arrays");
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  const int n_tensor = shear ? 10 : she ? 4 : 6, n_out = pol_n_out(term);
  const size_t n_bins = (size_t)std::max(sp->n, 0) * std::max(gr->n_pT, 0) * std::max(gr->n_phi, 0) * std::max(gr->n_y, 0);
  int prev = 0; cudaGetDevice(&prev);
  std::vector<int> rcs(G, IS3D_OK);
  std::vector<std::string> errs(G);
  std::vector<is3d_stats> sts(G);
  std::vector<std::vector<double>> bufs(G, std::vector<double>(n_out * n_bins, 0.0));
  std::vector<std::thread> workers;
  for (int d = 0; d < G; d++) {
    workers.emplace_back([&, d]() {
      memset(&sts[d], 0, sizeof(is3d_stats));
      if (cudaSetDevice(d) != cudaSuccess) { rcs[d] = IS3D_ERR_CUDA; errs[d] = "cudaSetDevice failed"; return; }
      int64_t lo, hi;
      shard_bounds(sf->n_cells, d, G, &lo, &hi);
      const is3d_surface shard = shard_surface(*sf, lo, hi);
      const double *ts[10];
      for (int a = 0; a < n_tensor; a++) ts[a] = tensor[a] ? tensor[a] + lo : tensor[a];
      is3d_options opt; memset(&opt, 0, sizeof(opt));
      if (opt_in) opt = *opt_in;
      opt.memory = 0; opt.stream = g_streams[d];
      double *r[kSdSums];
      for (int q = 0; q < n_out; q++) r[q] = bufs[d].data() + q * n_bins;
      rcs[d] = polzn_core(fl, &shard, ts, term, sp, gr, &opt, r, &sts[d]);
      if (rcs[d]) errs[d] = g_last_error;
    });
  }
  for (auto &w : workers) w.join();
  cudaSetDevice(prev);
  for (int d = 0; d < G; d++) if (rcs[d]) return fail(rcs[d], errs[d].c_str());
  for (int q = 0; q < n_out; q++)
    for (size_t i = 0; i < n_bins; i++) { double v = 0.0; for (int d = 0; d < G; d++) v += bufs[d][q * n_bins + i]; out[q][i] += v; }
  if (stats) {
    is3d_stats tot; memset(&tot, 0, sizeof(tot));
    for (int d = 0; d < G; d++) merge_stats(&tot, sts[d]);
    tot.n_gpus = G;
    *stats = tot;
  }
  return IS3D_OK;
}

// the columns of the input structs in the order of the prepare kernels, or NULL for a NULL struct
static const double *const *vort_columns(const is3d_vorticity *vo, const double **c)
{
  if (!vo) return nullptr;
  const double *v[6] = {vo->wtx, vo->wty, vo->wtn, vo->wxy, vo->wxn, vo->wyn};
  for (int a = 0; a < 6; a++) c[a] = v[a];
  return c;
}
static const double *const *shear_columns(const is3d_thermal_shear *xi, const double **c)
{
  if (!xi) return nullptr;
  const double *v[10] = {xi->xtt, xi->xtx, xi->xty, xi->xtn, xi->xxx, xi->xxy, xi->xxn, xi->xyy, xi->xyn, xi->xnn};
  for (int a = 0; a < 10; a++) c[a] = v[a];
  return c;
}
static const double *const *gradient_columns(const is3d_baryon_gradient *gd, const double **c)
{
  if (!gd) return nullptr;
  c[0] = gd->dt; c[1] = gd->dx; c[2] = gd->dy; c[3] = gd->dn;
  return c;
}
// the result arrays of the terms in the order of pol_n_out() (shear_arrays serves the spin Hall term too), or NULL for a NULL struct
static double *const *vort_arrays(is3d_polarization_result *r, double **a)
{
  if (!r) return nullptr;
  a[0] = r->Snorm; a[1] = r->St; a[2] = r->Sx; a[3] = r->Sy; a[4] = r->Sz;
  return a;
}
static double *const *shear_arrays(is3d_polarization_result *r, double **a)
{
  if (!r) return nullptr;
  a[0] = r->Snorm; a[1] = r->Sx; a[2] = r->Sy; a[3] = r->Sz; a[4] = r->St;
  return a;
}
static double *const *spin_density_arrays(is3d_spin_density_result *r, double **a)
{
  if (!r) return nullptr;
  double *v[kSdSums] = {r->Snorm, r->Px, r->Py, r->Pz, r->Qxx, r->Qxy, r->Qxz, r->Qyy, r->Qyz};
  for (int q = 0; q < kSdSums; q++) a[q] = v[q];
  return a;
}

}  // namespace is3d

extern "C" int is3d_b200_spin_polarization(const is3d_flags *fl, const is3d_surface *sf, const is3d_vorticity *vo, const is3d_species *sp,
                                           const is3d_grid *gr, const is3d_options *opt, is3d_polarization_result *res, is3d_stats *stats)
{
  const double *c[6]; double *a[5];
  return polzn_core(fl, sf, vort_columns(vo, c), kPolVorticity, sp, gr, opt, vort_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_polarization_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_vorticity *vo, const is3d_species *sp,
                                                 const is3d_grid *gr, const is3d_options *opt, is3d_polarization_result *res, is3d_stats *stats)
{
  const double *c[6]; double *a[5];
  return polzn_multi(fl, sf, vort_columns(vo, c), kPolVorticity, sp, gr, opt, vort_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_polarization_shear(const is3d_flags *fl, const is3d_surface *sf, const is3d_thermal_shear *xi,
                                                 const is3d_species *sp, const is3d_grid *gr, const is3d_options *opt,
                                                 is3d_polarization_result *res, is3d_stats *stats)
{
  const double *c[10]; double *a[5];
  return polzn_core(fl, sf, shear_columns(xi, c), kPolShear, sp, gr, opt, shear_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_polarization_shear_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_thermal_shear *xi,
                                                       const is3d_species *sp, const is3d_grid *gr, const is3d_options *opt,
                                                       is3d_polarization_result *res, is3d_stats *stats)
{
  const double *c[10]; double *a[5];
  return polzn_multi(fl, sf, shear_columns(xi, c), kPolShear, sp, gr, opt, shear_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_polarization_spin_hall(const is3d_flags *fl, const is3d_surface *sf, const is3d_baryon_gradient *gd,
                                                     const is3d_species *sp, const is3d_grid *gr, const is3d_options *opt,
                                                     is3d_polarization_result *res, is3d_stats *stats)
{
  const double *c[4]; double *a[5];
  return polzn_core(fl, sf, gradient_columns(gd, c), kPolSpinHall, sp, gr, opt, shear_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_polarization_spin_hall_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_baryon_gradient *gd,
                                                           const is3d_species *sp, const is3d_grid *gr, const is3d_options *opt,
                                                           is3d_polarization_result *res, is3d_stats *stats)
{
  const double *c[4]; double *a[5];
  return polzn_multi(fl, sf, gradient_columns(gd, c), kPolSpinHall, sp, gr, opt, shear_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_density(const is3d_flags *fl, const is3d_surface *sf, const is3d_vorticity *vo, const is3d_species *sp,
                                      const is3d_grid *gr, const is3d_options *opt, is3d_spin_density_result *res, is3d_stats *stats)
{
  const double *c[6]; double *a[kSdSums];
  return polzn_core(fl, sf, vort_columns(vo, c), kPolSpinDensity, sp, gr, opt, spin_density_arrays(res, a), stats);
}

extern "C" int is3d_b200_spin_density_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_vorticity *vo, const is3d_species *sp,
                                            const is3d_grid *gr, const is3d_options *opt, is3d_spin_density_result *res, is3d_stats *stats)
{
  const double *c[6]; double *a[kSdSums];
  return polzn_multi(fl, sf, vort_columns(vo, c), kPolSpinDensity, sp, gr, opt, spin_density_arrays(res, a), stats);
}

// =====================================================================================================================
// HBT moments (cf_hbt.cu): the ten raw space-time sums of the linear-delta-f emission function, added into the caller's arrays
// =====================================================================================================================
namespace is3d {

// What hbt_setup leaves for the kernel of an HBT entry point: the records of prepare_vh_kernel and prepare_hbt_cells_kernel on the
// device, the HotParams both HBT kernels read, a zeroed sums buffer [n_arrays][n_bins], and the device's call lock, held until the
// caller returns.  Events ev[0..2] are recorded (H2D, prepare); the caller launches its kernel and calls hbt_finish.
struct HbtSetup {
  std::unique_lock<std::mutex> lk;
  Workspace *ws = nullptr;
  is3d_options opt;
  cudaStream_t st = nullptr;
  int model = 0;
  int64_t n_cells = 0, n_bins = 0, n_active = 0, n_chunks_wanted = 0, n_arrays = 0;
  HotParams hp;
  const double *C = nullptr, *cosphi = nullptr, *sinphi = nullptr;
  const double *table = nullptr;         // the caller's extra table on the device
  double *sums = nullptr;                // [n_arrays][n_bins]
  PrepCounters cnt;
};

// Validation, layout, chunking, tables and surface to the device, prepare kernels and the table-range stop of every HBT entry point.
//   what:               the path's name in error messages
//   nyt, npt, ct:       register tile and TMA tile of the caller's kernel
//   n_arrays:           partial rows per chunk and bin (the 4 GiB cap on the partial sums divides by it)
//   blocks_per_bintile: blocks of the caller's grid per (group block, y tile, phi tile) and chunk
//   table:              doubles the caller's kernel reads beside the species and momentum tables (may be empty)
// The result arrays and any argument of the caller's own are checked by the caller first.
static int hbt_setup(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr, const is3d_df_tables *df,
                     const is3d_options *opt_in, const char *what, int nyt, int npt, int ct, int64_t n_arrays, int64_t blocks_per_bintile,
                     const std::vector<double> &table, HbtSetup *S)
{
  const std::string name(what);
  if (fl->mode == 2) return fail(IS3D_ERR_UNSUPPORTED, (name + " need a viscous-hydro surface, not mode 2 (anisotropic hydro)").c_str());
  if (fl->include_baryon) return fail(IS3D_ERR_UNSUPPORTED, "include_baryon = 1 (the reference's (T, muB) lookup reads out of bounds, SURVEY R8)");
  if (fl->df_mode == 3 || fl->df_mode == 4) return fail(IS3D_ERR_UNSUPPORTED, (name + " cover the linear delta-f models (df_mode 1, 2), not the modified equilibrium").c_str());
  if (fl->df_mode != 1 && fl->df_mode != 2) return fail(IS3D_ERR_ARGUMENT, "df_mode must be 1..4");
  if (!sf->x || !sf->y) return fail(IS3D_ERR_ARGUMENT, (name + " need the transverse cell positions (surface x, y)").c_str());
  if (fl->dimension != 2 && fl->dimension != 3) return fail(IS3D_ERR_ARGUMENT, "dimension must be 2 or 3");
  if (sp->n <= 0 || gr->n_pT <= 0 || gr->n_phi <= 0 || gr->n_y <= 0) return fail(IS3D_ERR_ARGUMENT, "empty species list or momentum table");
  if (!sp->mass || !sp->sign || !sp->degeneracy || !gr->pT || !gr->phi || !gr->y) return fail(IS3D_ERR_ARGUMENT, "NULL species or momentum table");
  const bool dim2 = (fl->dimension == 2);
  if (dim2 && (gr->n_eta <= 0 || !gr->eta || !gr->eta_weight)) return fail(IS3D_ERR_ARGUMENT, "dimension = 2 needs the eta table");
  if (!df || df->n_T < 3 || !df->T) return fail(IS3D_ERR_ARGUMENT, "delta-f coefficient tables missing");
  if (fl->df_mode == 1 && (!df->c0 || !df->c2)) return fail(IS3D_ERR_ARGUMENT, "df_mode 1 needs the c0 and c2 tables");
  if (fl->df_mode == 2 && (!df->F || !df->betabulk || !df->betapi)) return fail(IS3D_ERR_ARGUMENT, "df_mode 2 needs the F, betabulk and betapi tables");
  const int64_t n_cells = sf->n_cells;
  if (n_cells < 0) return fail(IS3D_ERR_ARGUMENT, "negative cell count");
  const bool sh = fl->include_shear_deltaf != 0, bk = fl->include_bulk_deltaf != 0;
  const int model = (!sh && !bk) ? M_IDEAL : (fl->df_mode == 1 ? M_LIN14 : M_LINCE);
  // the surface arrays prepare_vh_kernel reads, then the positions
  constexpr int kRaw = 20;
  const double *srcs[kRaw] = {sf->tau, sf->eta, sf->dat, sf->dax, sf->day, sf->dan, sf->ux, sf->uy, sf->un, sf->T, sf->P, sf->E,
                              sf->pixx, sf->pixy, sf->pixn, sf->piyy, sf->piyn, sf->bulkPi, sf->x, sf->y};
  const bool need[kRaw] = {true, true, true, true, true, true, true, true, true, true, true, true, sh, sh, sh, sh, sh, bk, true, true};
  for (int a = 0; a < kRaw; a++) if (need[a] && !srcs[a] && n_cells > 0) return fail(IS3D_ERR_ARGUMENT, "a required surface array is NULL");
  Device *Dp = nullptr;
  { int rc = current_device(&Dp); if (rc) return rc; }
  Workspace &ws = Dp->ws;
  S->lk = std::unique_lock<std::mutex>(Dp->mu);
  is3d_options opt; memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  cudaStream_t st = (cudaStream_t)opt.stream;
  const int64_t n_bins = (int64_t)sp->n * gr->n_pT * gr->n_phi * gr->n_y;
  const int64_t n_active = dim2 ? n_bins / gr->n_y : n_bins;        // 2+1D fills the y = 0 plane (index iy = 0)

  // ---- layout: the cf_kernel decomposition with the caller's register tile; records of prepare_vh_kernel
  Layout L; memset(&L, 0, sizeof(L));
  L.n_species = sp->n; L.n_pT = gr->n_pT; L.n_phi = gr->n_phi; L.n_y_out = gr->n_y;
  L.dim2 = dim2 ? 1 : 0;
  L.n_slots = dim2 ? gr->n_eta : gr->n_y;
  L.rec_y = kRec;
  L.nst = dim2 ? L.n_slots : nyt;
  L.n_ytiles = dim2 ? 1 : (L.n_slots + nyt - 1) / nyt;
  L.npt = npt; L.n_ptiles = (L.n_phi + npt - 1) / npt;
  L.ct = ct; L.n_cells = n_cells;
  L.n_tiles = (n_cells + ct - 1) / ct;
  L.n_cells_pad = L.n_tiles * ct;
  const int n_groups = (sp->n * gr->n_pT + 31) / 32;
  const int n_warps = std::min(kHbtWarps, n_groups);
  const int n_groupblocks = (n_groups + n_warps - 1) / n_warps;
  const int64_t n_bintiles = (int64_t)n_groupblocks * L.n_ytiles * L.n_ptiles * blocks_per_bintile;
  // chunks: the rule of smooth_core (>= 192 blocks per SM, a chunk's records within a third of L2, partial sums <= 4 GiB)
  int64_t n_chunks = ((int64_t)Dp->sm_count * 192 + n_bintiles - 1) / n_bintiles;
  const int64_t rec_per_cell = ((int64_t)L.n_ytiles * L.nst * kRec + (int64_t)L.n_ptiles * L.npt * kRec + kScal + kHbtRecC) * 8;
  const int64_t l2_target = std::max<int64_t>((int64_t)Dp->l2_bytes / 3, (int64_t)8 << 20);
  n_chunks = std::max<int64_t>(n_chunks, (n_cells * rec_per_cell + l2_target - 1) / l2_target);
  const int64_t n_chunks_wanted = n_chunks;
  n_chunks = std::min<int64_t>(n_chunks, std::max<int64_t>(1, ((int64_t)4 << 30) / (n_arrays * n_bins * 8)));
  if (opt.n_chunks > 0) n_chunks = opt.n_chunks;
  n_chunks = std::max<int64_t>(1, std::min<int64_t>(n_chunks, std::max<int64_t>(L.n_tiles, 1)));
  if (n_bintiles * n_chunks > 2147483647LL) return fail(IS3D_ERR_ARGUMENT, "grid too large");

  // ---- tables and surface to the device
  SmallArena ar;
  std::vector<double> cosphi(gr->n_phi), sinphi(gr->n_phi);
  for (int k = 0; k < gr->n_phi; k++) { cosphi[k] = cos(gr->phi[k]); sinphi[k] = sin(gr->phi[k]); }
  const size_t o_mass = ar.put(sp->mass, sp->n), o_sign = ar.put(sp->sign, sp->n), o_deg = ar.put(sp->degeneracy, sp->n);
  const size_t o_pT = ar.put(gr->pT, gr->n_pT), o_cos = ar.put(cosphi.data(), gr->n_phi), o_sin = ar.put(sinphi.data(), gr->n_phi);
  const size_t o_sloty = dim2 ? ar.put(gr->eta, gr->n_eta) : ar.put(gr->y, gr->n_y);
  const size_t o_slotw = dim2 ? ar.put(gr->eta_weight, gr->n_eta) : 0;
  const size_t o_table = ar.put(table.data(), table.size());
  struct SplineOff { size_t x, y, c; int n; };
  auto put_spline = [&](const double *x, const double *y, int n) {
    SplineOff o{0, 0, 0, 0};
    if (!x || !y || n < 3) return o;
    std::vector<double> c(n);
    host_spline_init(x, y, n, c.data());
    o.x = ar.put(x, n); o.y = ar.put(y, n); o.c = ar.put(c.data(), n); o.n = n;
    return o;
  };
  const SplineOff s_c0 = put_spline(df->T, df->c0, df->n_T), s_c2 = put_spline(df->T, df->c2, df->n_T), s_F = put_spline(df->T, df->F, df->n_T);
  const SplineOff s_bb = put_spline(df->T, df->betabulk, df->n_T), s_bp = put_spline(df->T, df->betapi, df->n_T);
  const size_t cell_stride = ((size_t)n_cells * 8 + 255) & ~(size_t)255;
  CU_CHECK(ws.small.reserve(ar.host.size() + 256));
  CU_CHECK(ws.Y.reserve((size_t)L.n_ytiles * L.n_cells_pad * L.nst * kRec * 8 + 256));
  CU_CHECK(ws.P.reserve((size_t)L.n_ptiles * L.n_cells_pad * L.npt * kRec * 8 + 256));
  CU_CHECK(ws.S.reserve((size_t)L.n_cells_pad * kScal * 8 + 256));
  CU_CHECK(ws.extra.reserve((size_t)L.n_cells_pad * kHbtRecC * 8 + 256));          // per-cell [tau, x, y, 0]
  CU_CHECK(ws.partial.reserve((size_t)n_arrays * n_chunks * n_bins * 8 + 256));
  CU_CHECK(ws.dN.reserve((size_t)n_arrays * n_bins * 8 + 256));
  CU_CHECK(ws.counters.reserve(256));
  if (opt.memory == 0) CU_CHECK(ws.raw.reserve(cell_stride * kRaw + 256));

  cudaEvent_t *ev = ws.ev;
  CU_CHECK(cudaEventRecord(ev[0], st));
  unsigned char *small_d = ws.small.as<unsigned char>();
  CU_CHECK(cudaMemcpyAsync(small_d, ar.host.data(), ar.host.size(), cudaMemcpyHostToDevice, st));
  const double *dev[kRaw];
  for (int a = 0; a < kRaw; a++) {
    dev[a] = need[a] ? srcs[a] : nullptr;
    if (opt.memory == 0 && need[a]) {
      double *d = reinterpret_cast<double *>(ws.raw.as<unsigned char>() + cell_stride * a);
      if (n_cells > 0) CU_CHECK(cudaMemcpyAsync(d, srcs[a], (size_t)n_cells * 8, cudaMemcpyHostToDevice, st));
      dev[a] = d;
    }
  }
  RawCells rc; memset(&rc, 0, sizeof(rc));
  rc.n = n_cells; rc.tau = dev[0]; rc.eta = dev[1]; rc.dat = dev[2]; rc.dax = dev[3]; rc.day = dev[4]; rc.dan = dev[5];
  rc.ux = dev[6]; rc.uy = dev[7]; rc.un = dev[8]; rc.T = dev[9]; rc.P = dev[10]; rc.E = dev[11];
  rc.pixx = dev[12]; rc.pixy = dev[13]; rc.pixn = dev[14]; rc.piyy = dev[15]; rc.piyn = dev[16]; rc.bulkPi = dev[17];
  double *sums_d = ws.dN.as<double>();                         // [n_arrays][n_bins]
  CU_CHECK(cudaMemsetAsync(sums_d, 0, (size_t)n_arrays * n_bins * 8, st));
  CU_CHECK(cudaMemsetAsync(ws.counters.p, 0, sizeof(PrepCounters), st));
  CU_CHECK(cudaEventRecord(ev[1], st));

  // ---- prepare: the spectra's records, then the positions
  auto dptr = [&](size_t off) { return reinterpret_cast<const double *>(small_d + off); };
  PrepTables tab; memset(&tab, 0, sizeof(tab));
  auto mk = [&](const SplineOff &o) { Spline s; s.x = dptr(o.x); s.y = dptr(o.y); s.c = dptr(o.c); s.n = o.n; return s; };
  tab.c0 = mk(s_c0); tab.c2 = mk(s_c2); tab.F = mk(s_F); tab.betabulk = mk(s_bb); tab.betapi = mk(s_bp);
  tab.bulkPi_over_Peq_max = df->bulkPi_over_Peq_max;
  tab.cosphi = dptr(o_cos); tab.sinphi = dptr(o_sin); tab.slot_y = dptr(o_sloty); tab.slot_w = dim2 ? dptr(o_slotw) : nullptr;
  tab.deta_min = fl->deta_min; tab.mass_pion0 = fl->mass_pion0;
  PrepCounters *cnt_d = ws.counters.as<PrepCounters>();
  CU_CHECK(launch_prepare_vh(*fl, rc, tab, L, ws.Y.as<double>(), ws.P.as<double>(), ws.S.as<double>(), cnt_d, st));
  CU_CHECK(launch_prepare_hbt_cells(dev[0], dev[18], dev[19], n_cells, L.n_cells_pad, ws.extra.as<double>(), st));
  CU_CHECK(cudaEventRecord(ev[2], st));
  // a cell outside the coefficient tables: stop before anything is added to the result, as the spectra do
  PrepCounters cnt; memset(&cnt, 0, sizeof(cnt));
  CU_CHECK(cudaMemcpyAsync(&cnt, cnt_d, sizeof(cnt), cudaMemcpyDeviceToHost, st));
  CU_CHECK(cudaStreamSynchronize(st));
  if (cnt.range_error) return fail(IS3D_ERR_TABLE_RANGE, "a cell's T lies outside the delta-f coefficient table");

  HotParams &hp = S->hp;
  memset(&hp, 0, sizeof(hp));
  hp.L = L; hp.Y = ws.Y.as<double>(); hp.P = ws.P.as<double>(); hp.S = ws.S.as<double>();
  hp.mass = dptr(o_mass); hp.sign = dptr(o_sign); hp.degeneracy = dptr(o_deg); hp.pT = dptr(o_pT);
  hp.partial = ws.partial.as<double>();
  hp.n_chunks = (int)n_chunks; hp.n_groupblocks = n_groupblocks; hp.n_warps = n_warps;
  hp.regulate_thr = fl->regulate_deltaf ? 0x3ff00000 : 0x7ff80000;        // as smooth_core
  hp.one_hi = 0x3ff00000;
  hp.outflow_thr = fl->outflow ? 0LL : (long long)0x8000000000000000ULL;
  hp.prefactor = pow(2.0 * M_PI * 0.197327053, -3);
  S->ws = &ws; S->opt = opt; S->st = st; S->model = model;
  S->n_cells = n_cells; S->n_bins = n_bins; S->n_active = n_active; S->n_chunks_wanted = n_chunks_wanted; S->n_arrays = n_arrays;
  S->C = ws.extra.as<double>(); S->cosphi = dptr(o_cos); S->sinphi = dptr(o_sin); S->table = dptr(o_table);
  S->sums = sums_d; S->cnt = cnt;
  return IS3D_OK;
}

// After the caller's kernel: fold the partial rows [n_arrays][n_chunks][n_bins] in a fixed order, add array q into out[q] (host or
// device per options->memory), fill the stats.
static int hbt_finish(HbtSetup &S, double *const *out, is3d_stats *stats)
{
  const HotParams &hp = S.hp;
  const int64_t n_arrays = S.n_arrays, n_bins = S.n_bins, n_chunks = hp.n_chunks;
  cudaStream_t st = S.st;
  cudaEvent_t *ev = S.ws->ev;
  CU_CHECK(cudaEventRecord(ev[3], st));
  for (int64_t q = 0; q < n_arrays; q++)
    CU_CHECK(launch_reduce(hp.partial + (size_t)q * n_chunks * n_bins, (int)n_chunks, n_bins, S.n_active, S.sums + (size_t)q * n_bins, st));
  CU_CHECK(cudaEventRecord(ev[4], st));

  std::vector<double> host;
  if (S.opt.memory == 0) {
    host.resize((size_t)n_arrays * n_bins);
    CU_CHECK(cudaMemcpyAsync(host.data(), S.sums, (size_t)n_arrays * n_bins * 8, cudaMemcpyDeviceToHost, st));
  } else {
    for (int64_t q = 0; q < n_arrays; q++) CU_CHECK(launch_axpy(S.sums + (size_t)q * n_bins, out[q], S.n_active, st));
  }
  CU_CHECK(cudaEventRecord(ev[5], st));
  CU_CHECK(cudaEventSynchronize(ev[5]));
  if (S.opt.memory == 0)
    for (int64_t q = 0; q < n_arrays; q++)
      for (int64_t i = 0; i < n_bins; i++) out[q][i] += host[(size_t)q * n_bins + i];

  const Layout &L = hp.L;
  is3d_stats stt; memset(&stt, 0, sizeof(stt));
  float ms;
  cudaEventElapsedTime(&ms, ev[0], ev[1]); stt.h2d_ms = ms;
  cudaEventElapsedTime(&ms, ev[1], ev[2]); stt.prepare_ms = ms;
  cudaEventElapsedTime(&ms, ev[2], ev[3]); stt.kernel_ms = ms;
  cudaEventElapsedTime(&ms, ev[3], ev[4]); stt.reduce_ms = ms;
  cudaEventElapsedTime(&ms, ev[4], ev[5]); stt.d2h_ms = ms;
  cudaEventElapsedTime(&ms, ev[0], ev[5]); stt.total_ms = ms;
  stt.cells_skipped_udsigma = (int64_t)S.cnt.skipped;
  stt.evaluations = S.n_cells * (int64_t)L.n_species * L.n_pT * L.n_phi * (int64_t)L.n_slots;
  stt.gpu_launches = (int)((S.n_cells > 0 ? 2 : 0) + 1 + n_arrays + (S.opt.memory == 0 ? 0 : n_arrays));
  stt.n_chunks = (int)n_chunks; stt.n_chunks_wanted = (int)S.n_chunks_wanted;
  stt.n_gpus = 1;
  if (stats) *stats = stt;
  return IS3D_OK;
}

static int hbt_core(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr, const is3d_df_tables *df,
                    const is3d_options *opt_in, is3d_hbt_result *res, is3d_stats *stats)
{
  if (!fl || !sf || !sp || !gr || !res) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  double *out[kHbtSums] = {res->S0, res->So, res->Ss, res->Sl, res->Soo, res->Sss, res->Sll, res->Sos, res->Sol, res->Ssl};
  for (double *p : out) if (!p) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
  int nyt, npt, ct;
  hbt_shape(fl->dimension == 2, &nyt, &npt, &ct);
  HbtSetup S;
  { int rc = hbt_setup(fl, sf, sp, gr, df, opt_in, "HBT moments", nyt, npt, ct, kHbtSums, 1, std::vector<double>(), &S); if (rc) return rc; }
  HbtParams prm; memset(&prm, 0, sizeof(prm));
  prm.hp = S.hp; prm.C = S.C; prm.cosphi = S.cosphi; prm.sinphi = S.sinphi;
  CU_CHECK(launch_hbt(S.model, prm, S.st));
  return hbt_finish(S, out, stats);
}

// HBT Fourier sums (cf_hbtq.cu): the arguments of their own, checked before any set-up (the _multi entry point sizes its buffers by them)
static int hbtq_check(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr, const is3d_hbt_qrays *qr,
                      const is3d_hbt_fourier_result *res)
{
  if (!fl || !sf || !sp || !gr || !res || !qr) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (!res->Re || !res->Im) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
  if (qr->n_dir < 1 || qr->n_q < 1) return fail(IS3D_ERR_ARGUMENT, "the q rays need n_dir >= 1 and n_q >= 1");
  if (!qr->dir) return fail(IS3D_ERR_ARGUMENT, "NULL q-ray directions");
  if (!std::isfinite(qr->dq) || qr->dq <= 0.0) return fail(IS3D_ERR_ARGUMENT, "the q step dq must be finite and > 0");
  for (int64_t i = 0; i < 3 * (int64_t)qr->n_dir; i++)
    if (!std::isfinite(qr->dir[i])) return fail(IS3D_ERR_ARGUMENT, "a q-ray direction component is not finite");
  // the partial sums of one chunk: 2 n_dir n_q rows of n_bins doubles within the 4 GiB cap
  const double n_arrays = 2.0 * qr->n_dir * (double)qr->n_q;
  const double n_bins = (double)std::max(sp->n, 0) * std::max(gr->n_pT, 0) * std::max(gr->n_phi, 0) * std::max(gr->n_y, 0);
  if (n_arrays * n_bins * 8.0 > (double)((int64_t)4 << 30))
    return fail(IS3D_ERR_ARGUMENT, "2 n_dir n_q x n_bins sums exceed the 4 GiB partial-sum buffer even in one chunk: fewer q points, rays or bins per call");
  return IS3D_OK;
}

// HBT Fourier sums (cf_hbtq.cu): Re / Im [n_dir][n_q][n_bins] of sum w e^{i theta}, added into the caller's arrays
static int hbt_fourier_core(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr, const is3d_df_tables *df,
                            const is3d_hbt_qrays *qr, const is3d_options *opt_in, is3d_hbt_fourier_result *res, is3d_stats *stats)
{
  { int rc = hbtq_check(fl, sf, sp, gr, qr, res); if (rc) return rc; }
  const int64_t n_arrays = 2 * (int64_t)qr->n_dir * qr->n_q;
  const int n_qtiles = (qr->n_q + kHbtqKQ - 1) / kHbtqKQ;
  const double step = qr->dq / 0.197327053;                      // [1/fm per GeV of q]
  std::vector<double> dir(3 * (size_t)qr->n_dir);
  for (size_t i = 0; i < dir.size(); i++) dir[i] = qr->dir[i] * step;
  int nyt, npt, ct;
  hbtq_shape(fl->dimension == 2, &nyt, &npt, &ct);
  HbtSetup S;
  { int rc = hbt_setup(fl, sf, sp, gr, df, opt_in, "HBT Fourier sums", nyt, npt, ct, n_arrays, (int64_t)qr->n_dir * n_qtiles, dir, &S); if (rc) return rc; }
  HbtqParams prm; memset(&prm, 0, sizeof(prm));
  prm.hp = S.hp; prm.C = S.C; prm.cosphi = S.cosphi; prm.sinphi = S.sinphi;
  prm.dir = S.table; prm.n_dir = qr->n_dir; prm.n_q = qr->n_q; prm.n_qtiles = n_qtiles;
  CU_CHECK(launch_hbt_fourier(S.model, prm, S.st));
  const int64_t half = (int64_t)qr->n_dir * qr->n_q;
  std::vector<double *> out((size_t)n_arrays);
  for (int64_t a = 0; a < half; a++) { out[a] = res->Re + a * S.n_bins; out[half + a] = res->Im + a * S.n_bins; }
  return hbt_finish(S, out.data(), stats);
}

}  // namespace is3d

extern "C" int is3d_b200_hbt_moments(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                                     const is3d_df_tables *df, const is3d_options *opt, is3d_hbt_result *res, is3d_stats *stats)
{
  return hbt_core(fl, sf, sp, gr, df, opt, res, stats);
}

// Several devices: HOST arrays, contiguous cell shards, one thread per device; the ten raw sums are added on the host in device order
extern "C" int is3d_b200_hbt_moments_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                                           const is3d_df_tables *df, const is3d_options *opt_in, is3d_hbt_result *res, is3d_stats *stats)
{
  const int G = g_ngpus;
  if (G <= 1) return is3d_b200_hbt_moments(fl, sf, sp, gr, df, opt_in, res, stats);
  if (!fl || !sf || !sp || !gr || !res) return fail(IS3D_ERR_ARGUMENT, "NULL argument");
  if (opt_in && opt_in->memory != 0) return fail(IS3D_ERR_ARGUMENT, "the multi-GPU entry point takes host arrays");
  double *out[kHbtSums] = {res->S0, res->So, res->Ss, res->Sl, res->Soo, res->Sss, res->Sll, res->Sos, res->Sol, res->Ssl};
  for (double *p : out) if (!p) return fail(IS3D_ERR_ARGUMENT, "NULL result array");
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  const size_t n_bins = (size_t)std::max(sp->n, 0) * std::max(gr->n_pT, 0) * std::max(gr->n_phi, 0) * std::max(gr->n_y, 0);
  int prev = 0; cudaGetDevice(&prev);
  std::vector<int> rcs(G, IS3D_OK);
  std::vector<std::string> errs(G);
  std::vector<is3d_stats> sts(G);
  std::vector<std::vector<double>> bufs(G, std::vector<double>(kHbtSums * n_bins, 0.0));
  std::vector<std::thread> workers;
  for (int d = 0; d < G; d++) {
    workers.emplace_back([&, d]() {
      memset(&sts[d], 0, sizeof(is3d_stats));
      if (cudaSetDevice(d) != cudaSuccess) { rcs[d] = IS3D_ERR_CUDA; errs[d] = "cudaSetDevice failed"; return; }
      int64_t lo, hi;
      shard_bounds(sf->n_cells, d, G, &lo, &hi);
      const is3d_surface shard = shard_surface(*sf, lo, hi);
      is3d_options opt; memset(&opt, 0, sizeof(opt));
      if (opt_in) opt = *opt_in;
      opt.memory = 0; opt.stream = g_streams[d];
      double *b = bufs[d].data();
      is3d_hbt_result r{b, b + n_bins, b + 2 * n_bins, b + 3 * n_bins, b + 4 * n_bins, b + 5 * n_bins, b + 6 * n_bins, b + 7 * n_bins,
                        b + 8 * n_bins, b + 9 * n_bins};
      rcs[d] = hbt_core(fl, &shard, sp, gr, df, &opt, &r, &sts[d]);
      if (rcs[d]) errs[d] = g_last_error;
    });
  }
  for (auto &w : workers) w.join();
  cudaSetDevice(prev);
  for (int d = 0; d < G; d++) if (rcs[d]) return fail(rcs[d], errs[d].c_str());
  for (int q = 0; q < kHbtSums; q++)
    for (size_t i = 0; i < n_bins; i++) { double v = 0.0; for (int d = 0; d < G; d++) v += bufs[d][q * n_bins + i]; out[q][i] += v; }
  if (stats) {
    is3d_stats tot; memset(&tot, 0, sizeof(tot));
    for (int d = 0; d < G; d++) merge_stats(&tot, sts[d]);
    tot.n_gpus = G;
    *stats = tot;
  }
  return IS3D_OK;
}

extern "C" int is3d_b200_hbt_fourier(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                                     const is3d_df_tables *df, const is3d_hbt_qrays *qr, const is3d_options *opt, is3d_hbt_fourier_result *res,
                                     is3d_stats *stats)
{
  return hbt_fourier_core(fl, sf, sp, gr, df, qr, opt, res, stats);
}

// Several devices: HOST arrays, contiguous cell shards, one thread per device; Re and Im are added on the host in device order
extern "C" int is3d_b200_hbt_fourier_multi(const is3d_flags *fl, const is3d_surface *sf, const is3d_species *sp, const is3d_grid *gr,
                                           const is3d_df_tables *df, const is3d_hbt_qrays *qr, const is3d_options *opt_in,
                                           is3d_hbt_fourier_result *res, is3d_stats *stats)
{
  const int G = g_ngpus;
  if (G <= 1) return is3d_b200_hbt_fourier(fl, sf, sp, gr, df, qr, opt_in, res, stats);
  { int rc = hbtq_check(fl, sf, sp, gr, qr, res); if (rc) return rc; }
  if (opt_in && opt_in->memory != 0) return fail(IS3D_ERR_ARGUMENT, "the multi-GPU entry point takes host arrays");
  std::lock_guard<std::mutex> lk(g_multi_mutex);
  const size_t n_bins = (size_t)std::max(sp->n, 0) * std::max(gr->n_pT, 0) * std::max(gr->n_phi, 0) * std::max(gr->n_y, 0);
  const size_t n = (size_t)qr->n_dir * qr->n_q * n_bins;          // doubles per array (Re or Im)
  int prev = 0; cudaGetDevice(&prev);
  std::vector<int> rcs(G, IS3D_OK);
  std::vector<std::string> errs(G);
  std::vector<is3d_stats> sts(G);
  std::vector<std::vector<double>> bufs(G, std::vector<double>(2 * n, 0.0));
  std::vector<std::thread> workers;
  for (int d = 0; d < G; d++) {
    workers.emplace_back([&, d]() {
      memset(&sts[d], 0, sizeof(is3d_stats));
      if (cudaSetDevice(d) != cudaSuccess) { rcs[d] = IS3D_ERR_CUDA; errs[d] = "cudaSetDevice failed"; return; }
      int64_t lo, hi;
      shard_bounds(sf->n_cells, d, G, &lo, &hi);
      const is3d_surface shard = shard_surface(*sf, lo, hi);
      is3d_options opt; memset(&opt, 0, sizeof(opt));
      if (opt_in) opt = *opt_in;
      opt.memory = 0; opt.stream = g_streams[d];
      is3d_hbt_fourier_result r{bufs[d].data(), bufs[d].data() + n};
      rcs[d] = hbt_fourier_core(fl, &shard, sp, gr, df, qr, &opt, &r, &sts[d]);
      if (rcs[d]) errs[d] = g_last_error;
    });
  }
  for (auto &w : workers) w.join();
  cudaSetDevice(prev);
  for (int d = 0; d < G; d++) if (rcs[d]) return fail(rcs[d], errs[d].c_str());
  double *out[2] = {res->Re, res->Im};
  for (int q = 0; q < 2; q++)
    for (size_t i = 0; i < n; i++) { double v = 0.0; for (int d = 0; d < G; d++) v += bufs[d][q * n + i]; out[q][i] += v; }
  if (stats) {
    is3d_stats tot; memset(&tot, 0, sizeof(tot));
    for (int d = 0; d < G; d++) merge_stats(&tot, sts[d]);
    tot.n_gpus = G;
    *stats = tot;
  }
  return IS3D_OK;
}
