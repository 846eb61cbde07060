// cf_shift.cu -- "shifted-factor" hot kernel for the linear-delta-f models on 3+1D tiles (M_LIN14, M_LINCE, M_JONAHLIN, M_IDEAL).
//
// Same decomposition as cf_kernel (cf_kernels.cu), thread = register tile of NYT slots x NPT phi points, block = 4 warps on one
// (y tile, phi tile, cell chunk), records streamed by TMA through an mbarrier pipeline, pair table for the lane-independent shear
// cross term -- except that a lane is a (species class, pT) pair rather than a (species, pT) pair:
//
//  * a lane's accumulators depend on the species through its mass and statistics only (degeneracy is a factor of the epilogue;
//    baryon number enters delta-f only with include_baryon, which the library rejects).  Species with bit-equal (mass, sign) --
//    every antibaryon and its baryon, the members of an isospin multiplet in the UrQMD list: 75 classes for its 305 species --
//    form one class (SpeciesClasses, built on the host), and the epilogue stores a class's tile once for each member species,
//    scaled by that species' degeneracy.  At 32 pT points a warp is one class, as it was one species, so its votes see the same
//    lanes and every stored value is the one a per-species lane would store, bit for bit.
//
// What changes against cf_kernel is how the NPT evaluations of a (cell, slot) get their exponentials and how the per-evaluation
// integer work (regulation, outflow) is paid:
//
//  * e^{-x_jk} with x_jk = mT A_j - pT B_k is split as e^{-(mT A_j - pT Bmax)} . e^{-pT (Bmax - B_k)}, Bmax = max_k B_k over the
//    tile's phi points.  Both factors lie in (0, 1]: neither can overflow or underflow before the product does, so no exponent
//    bookkeeping is needed (compare the mantissa / exponent pairs of cf_factored.cu).  The first factor is ONE exponential per
//    (cell, slot) and thread -- of the group's smallest argument xm, which also classifies the whole group (dead / dilute /
//    possibly sub-normal) -- the second does not depend on the slot or the species: cf_shift_table_kernel tabulates it once per
//    (phi tile, cell, phi point, pT) in global memory, together with Bmax and Bmax - Bmin, and the hot kernel streams each cell
//    tile's slice with its records (formed inside every block, the table took ~14 % of the hot kernel's instructions at cfg3,
//    counted from the SASS: the n_groupblocks x n_ytiles blocks that read a cell tile each computed the same values).
//    Per evaluation that leaves a DMUL where cf_kernel spends 9 FP64 instructions.
//  * regulation and outflow cost 5 integer instructions per evaluation instead of 8: g = 1 + df is clamped to [0, 2] (the
//    reference's max(-1, min(df, 1)), smooth_kernels.cpp:328) on its high word and zeroed where p.dsigma <= 0 (:285) by the same
//    selects (clamp_mask_g), followed by an unconditional accumulate.
//  * 14-moment delta-f and ideal f_eq: the group is wide in phi (default 3 slots x 6 phi points), so the per-(cell, slot) work --
//    the exponential of xm, the votes, the slot record -- is shared by 6 evaluations.  The slot body forms each member's values
//    inside its class branch and consumes them at once (shift_slot), which keeps the 3 x 6 and 3 x 8 tiles within 168 registers
//    (3 blocks/SM) without spills.  Groups whose largest argument may reach the sub-normal range (xm + pT (Bmax - Bmin) >= 707.7)
//    take the same product with e^{-xm} scaled by 2^64 and each member scaled back (one rounding to a sub-normal); members whose
//    exp(x) overflows in the reference are set to exact zeros, so the zero pattern and gradual underflow are the reference's.
//  * Chapman-Enskog and Jonah linear keep the staged body on 7 x 3 groups (with the member-by-member body they measured slower at
//    every shape); there groups that may touch the sub-normal range are evaluated member by member with the exact routines of
//    cf_kernel (distribution_group).
//
// On B200 a warp-wide FP64 instruction holds the scheduler for ~2 cycles and every other instruction for ~1.7 more without
// overlap (profiles/r2_ubench_mix_issue.txt): the kernel time follows the TOTAL instruction count, which is what this kernel cuts.
#include "cf_internal.h"
#include <algorithm>
#include <type_traits>
#include "cf_device.cuh"

namespace is3d {

namespace {

constexpr int kShiftMaxPT = 64;           // pT points the e^{-pT dB} table is laid out for
constexpr int kUltraHi = 0x4042C000;      // high word of 37.5: e^{-x} < 2^-54
// TMA pipeline depth.  A stage holds a 16-cell tile's records and table slice (32 KB at 3 x 6 and 32 pT points): two stages
// keep 3 blocks/SM; a tile lasts tens of us against ~1 us of copy latency, so the second stage is enough to hide it.
constexpr int kShiftStages = 2;

// doubles per (phi tile, cell) record of the table: Bmax, Bmax - Bmin, then e^{-pT (Bmax - B_k)} as [NPT][n_pT], padded to
// whole 16-byte units (the bulk copies need them)
__host__ __device__ __forceinline__ int shift_erec(int npt, int n_pT) { return (2 + npt * n_pT + 1) & ~1; }

// g = 1 + df clamped to [0, 2] (regulate_deltaf, smooth_kernels.cpp:328) and zeroed where p.dsigma fails the outflow test (:285),
// all on the integer pipe from the high words: 6 instructions (2 VIMNMX, 2 ISETP, 2 SEL) for both features.
//   reg_lo / reg_hi / reg_chk = 0 / 0x40000000 / 0x3fffffff with regulation on (g keeps its low word iff its high word read as
//   unsigned is <= reg_chk), INT_MIN / INT_MAX / 0xffffffff off;  thr_hi = 0 with outflow on, INT_MIN off.
// A masked member contributes p.dsigma f_eq 0 = +-0 to the accumulator, i.e. nothing.
__device__ __forceinline__ double clamp_mask_g(double g, double pds, int reg_lo, int reg_hi, unsigned reg_chk, int thr_hi)
{
  int hi = __double2hiint(g), lo = __double2loint(g), hc, ho, lw;
  asm("{\n\t.reg .pred pass, keep;\n\t"
      "setp.gt.s32 pass, %3, %4;\n\t"                 // p.dsigma passes the outflow test
      "setp.le.and.u32 keep, %5, %6, pass;\n\t"       // ... and g lies in [0, 2): keeps its low word
      "max.s32 %0, %5, %7;\n\t"
      "min.s32 %0, %0, %8;\n\t"                       // (VIMNMX3)
      "selp.b32 %1, %0, 0, pass;\n\t"
      "selp.b32 %2, %9, 0, keep;\n\t}"
      : "=&r"(hc), "=r"(ho), "=r"(lw) : "r"(__double2hiint(pds)), "r"(thr_hi), "r"(hi), "r"(reg_chk), "r"(reg_lo), "r"(reg_hi), "r"(lo));
  return __hiloint2double(ho, lw);
}

// e^{-x} = p 2^n like exp_neg_poly(); the table is read through a precomputed shared-memory address (the generic form rebuilds
// the shared window base with uniform-datapath instructions per use) and the constants come from the kernel parameters, which
// an FP64 instruction can take as a direct operand (from __constant__ arrays they are re-loaded with LDC under register pressure)
__device__ __forceinline__ void exp_neg_poly_at(double x, uint32_t tab_addr, const double (&ec)[8], double &p_out, int &n_out)
{
  const double fk = fma(x, ec[0], ec[1]);
  const int k = __double2loint(fk);
  const double kf = fk - ec[1];
  double r = fma(kf, ec[2], -x);
  r = fma(kf, ec[3], r);
  double T;
  asm("ld.shared.f64 %0, [%1];" : "=d"(T) : "r"(tab_addr + ((k & (kExpTabSize - 1)) << 3)));
  n_out = k >> kExpTabBits;
  double q = fma(ec[4], r, ec[5]);
  q = fma(q, r, ec[6]);
  q = fma(q, r, 1.0);
  p_out = fma(T * r, q, T);
}

// 14-moment delta-f and ideal f_eq run the member-by-member slot body (shift_slot) on wide phi groups; Chapman-Enskog and Jonah
// linear keep the staged body on 7 x 3 groups: with the member-by-member body CE measured 1.5 % slower at its best shape (3 x 6)
// and 17 % slower at 7 x 3 than the staged 7 x 3 (DESIGN.md section 6, profiles/r3_sweep.json)
__host__ __device__ constexpr bool shift_lean(int model) { return model == M_LIN14 || model == M_IDEAL; }

template <int V> using IntC = std::integral_constant<int, V>;
constexpr int kRareShift = 64;            // e^{-xm} 2^64 is a normal number for every alive xm (<= 709.79)

// The NPT members of one (cell, slot) group, one member at a time: every value a member needs is formed inside the class
// branch and consumed right away, so only the per-(cell, phi) operands q, pd, g0, eB and the accumulators stay live across
// members (the independent members give the scheduler enough parallelism).
//   RARE: e^{-xm} arrives scaled by 2^kRareShift; each product is scaled back (rounding once to a sub-normal where the
//         reference's 1 / (exp(x) + Theta) is one) and members whose exp(x) overflows in the reference are exact zeros.
//   CLS : 0 ultra-dilute (every xm >= 37.5: 1 / (1 + Theta a) = 1), 1 dilute (xm >= 12.5), 2 full Bose / Fermi factor.
// In the ultra-dilute class g = 1 + df is formed with the 1 folded into h0: one FP64 instruction less per member.
template <int MODEL, int NPT, int RARE, int CLS>
__device__ __forceinline__ void shift_slot(double a, double cpm, double h0, const double *prj, const double (&q)[NPT], const double (&pd)[NPT],
                                           const double (&g0)[NPT], const double (&eB)[NPT], double eA, double mTpT, double K2, double sign, int reg_lo, int reg_hi, unsigned reg_chk, int thr_hi, double *accj)
{
  static_assert(shift_lean(MODEL), "member-by-member slot body: 14-moment delta-f and ideal f_eq");
  constexpr bool DF = MODEL != M_IDEAL;
  const double hK = (DF && CLS == 0) ? h0 + 1.0 : h0;
#pragma unroll
  for (int k2 = 0; k2 < NPT; k2 += 2) {
    double2 t2 = make_double2(0.0, 0.0);
    if (DF) t2 = *reinterpret_cast<const double2 *>(prj + k2);                 // pair-table row padded to whole 16-byte loads
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int k = k2 + h;
      if (k >= NPT) break;
      const double xs = a - q[k];
      const double pv = pd[k] + cpm;
      double av = eA * eB[k];
      if (RARE) av = exp_finite(xs) ? av * __hiloint2double((1023 - kRareShift) << 20, 0) : 0.0;
      double f = av, g = 1.0;
      if (CLS == 0) {
        if (DF) g = fma(K2 * xs, xs, fma(mTpT, h ? t2.y : t2.x, hK + g0[k]));
      } else {
        double fb;
        f = (CLS == 1) ? occupation_bar_dilute(av, sign, fb) : occupation_bar(av, sign, fb);
        if (DF) {
          const double sv = fma(mTpT, h ? t2.y : t2.x, hK + g0[k]);
          g = fma(fb, fma(K2 * xs, xs, sv), 1.0);
        }
      }
      // f = f_eq g with g clamped to [0, 2]; members failing the outflow test get g = 0.  (A warp holds all pT values of a
      // species and the largest ones are always clamped: a "nobody needs it" shortcut would never fire.)
      if (DF) accj[k] = fma(pv, f * clamp_mask_g(g, pv, reg_lo, reg_hi, reg_chk, thr_hi), accj[k]);
      else accumulate_pos(accj[k], pv, f, thr_hi);
    }
  }
}

// E[tp][cell - cell0] = {Bmax, Bmax - Bmin, e^{-pT (Bmax - B_k)} [k][pT]} for the cells [cell0, cell0 + n_win), padded phi
// records included; one thread per (phi tile, cell, pT point)
template <int NPT, bool LEAN>
__global__ void __launch_bounds__(128)
cf_shift_table_kernel(const HotParams hp, double *E, int64_t cell0, int64_t n_win)
{
  const Layout &L = hp.L;
  exp_table_init();
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.n_ptiles * n_win * L.n_pT) return;
  const int ip = (int)(i % L.n_pT);
  const int64_t r = i / L.n_pT, cl = r % n_win;
  const int tp = (int)(r / n_win);
  const double *pr = hp.P + ((int64_t)tp * L.n_cells_pad + cell0 + cl) * NPT * kRec;
  double *er = E + ((int64_t)tp * hp.e_cells + cl) * shift_erec(NPT, L.n_pT);
  double b[NPT];
#pragma unroll
  for (int k = 0; k < NPT; k++) b[k] = pr[k * kRec];
  double bmax = b[0], bmin = b[0];
#pragma unroll
  for (int k = 1; k < NPT; k++) { bmax = b[k] > bmax ? b[k] : bmax; bmin = b[k] < bmin ? b[k] : bmin; }
  if (ip == 0) { er[0] = bmax; er[1] = bmax - bmin; }
  const double pTi = hp.pT[ip];
  const uint32_t tab_addr = smem_u32(g_exp_tab);
#pragma unroll
  for (int k = 0; k < NPT; k++) {
    double pp; int nn;
    const double dd = pTi * (bmax - b[k]);
    exp_neg_poly_at(dd, tab_addr, hp.ec, pp, nn);
    // beyond 707.7 the factor leaves the normal range: such members are only reached on the scaled path of the member-by-
    // member body, which needs the sub-normal value and 0 beyond ln(DBL_MAX) (a member with pT (Bmax - B_k) > 709.78 has
    // x_k > 709.78 and is an exact zero there), and on the per-member path of the staged body, which does not read the
    // table (0 keeps the lanes that merely ride along finite)
    if constexpr (LEAN) er[2 + k * L.n_pT + ip] = exp_neg_slow(dd, pp, nn);
    else er[2 + k * L.n_pT + ip] = __double2hiint(dd) < kRareHi ? exp_neg_fast(pp, nn) : 0.0;
  }
}

template <int MODEL, int NYT, int NPT, int MINB>
__global__ void __launch_bounds__(128, MINB)
cf_shift_kernel(const HotParams hp, const SpeciesClasses cls)
{
  constexpr int RY = kRec;
  constexpr bool DF = MODEL != M_IDEAL;
  constexpr bool LEAN = shift_lean(MODEL);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const Layout &L = hp.L;
  const int CT = L.ct;
  const int RE = shift_erec(NPT, L.n_pT);
  const int y_doubles = CT * NYT * RY, p_doubles = CT * NPT * kRec, s_doubles = CT * kScal, e_doubles = CT * RE;
  const int stage_doubles = y_doubles + p_doubles + s_doubles + e_doubles;
  double *stage_base = reinterpret_cast<double *>(smem_raw);
  uint64_t *full = reinterpret_cast<uint64_t *>(stage_base + (size_t)kShiftStages * stage_doubles);
  constexpr int NPP = (NPT + 1) & ~1;                                            // pair-table row padded to whole 16-byte loads
  double *pair_tab = reinterpret_cast<double *>(full + kShiftStages);            // [CT][NYT][NPP]
  double *pT_s = pair_tab + CT * NYT * NPP;                                      // [n_pT]

  const int n_bintiles = hp.n_groupblocks * L.n_ytiles * L.n_ptiles;
  const int chunk_w = blockIdx.x / n_bintiles;                                   // chunk within the launch's window
  const int chunk = hp.chunk0 + chunk_w;
  int bt = blockIdx.x - chunk_w * n_bintiles;
  const int tp = bt % L.n_ptiles; bt /= L.n_ptiles;
  const int ty = bt % L.n_ytiles; bt /= L.n_ytiles;
  const int gb = bt;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int idx = (gb * hp.n_warps + warp) * 32 + lane;
  const bool lane_valid = idx < cls.n * L.n_pT;
  const int icls = lane_valid ? idx / L.n_pT : 0;
  const int ipT = lane_valid ? idx - icls * L.n_pT : 0;
  const double mass = hp.mass[icls], sign = hp.sign[icls], pT = hp.pT[ipT];
  const double m2 = mass * mass, pT2 = pT * pT;
  const double mT2 = m2 + pT2;
  const double mT = sqrt(mT2);
  const double mTpT = mT * pT;
  const unsigned reg_chk = hp.reg_chk;
  const int reg_lo = hp.reg_lo, reg_hi = hp.reg_hi;
  const int thr_hi = (int)(hp.outflow_thr >> 32);
  const int reg_thr = hp.regulate_thr, one_hi = hp.one_hi;

  const int64_t t_begin = (L.n_tiles * (int64_t)chunk) / hp.n_chunks;
  const int64_t t_end = (L.n_tiles * (int64_t)(chunk + 1)) / hp.n_chunks;
  const int n_my_tiles = (int)(t_end - t_begin);

  const double *Yg = hp.Y + ((int64_t)ty * L.n_cells_pad) * NYT * RY;
  const double *Pg = hp.P + ((int64_t)tp * L.n_cells_pad) * NPT * kRec;
  const double *Sg = hp.S;
  // the window's table starts at the first cell of chunk chunk0
  const int64_t e_off = (int64_t)tp * hp.e_cells - (L.n_tiles * (int64_t)hp.chunk0) / hp.n_chunks * CT;
  const uint32_t stage_bytes = (uint32_t)stage_doubles * 8u;

  exp_table_init();
  for (int i = threadIdx.x; i < L.n_pT; i += blockDim.x) pT_s[i] = hp.pT[i];
  if (threadIdx.x == 0) {
    for (int s = 0; s < kShiftStages; s++) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  auto issue = [&](int t_local) {
    const int st = t_local % kShiftStages;
    const int64_t cell = (t_begin + t_local) * CT;
    double *dst = stage_base + (size_t)st * stage_doubles;
    mbar_arrive_expect_tx(&full[st], stage_bytes);
    bulk_g2s(dst, Yg + cell * NYT * RY, (uint32_t)y_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles, Pg + cell * NPT * kRec, (uint32_t)p_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles + p_doubles, Sg + cell * kScal, (uint32_t)s_doubles * 8u, &full[st]);
    bulk_g2s(dst + y_doubles + p_doubles + s_doubles, hp.E + (e_off + cell) * RE, (uint32_t)e_doubles * 8u, &full[st]);
  };
  if (threadIdx.x == 0)
    for (int t = 0; t < kShiftStages && t < n_my_tiles; t++) issue(t);

  double acc[NYT * NPT];
#pragma unroll
  for (int i = 0; i < NYT * NPT; i++) acc[i] = 0.0;
  const uint32_t tab_addr = smem_u32(g_exp_tab);
  const double rare_x = __hiloint2double(kRareHi, 0);                            // 707.6997...: below it e^{-x} is a normal number

  // the block-uniform tile count is read back from shared memory: a register holding it across the cell loop would be spilled
  // at 3 x 8 (member-by-member body) and 7 x 6 (staged body)
  __shared__ int my_tiles_s;
  if (threadIdx.x == 0) my_tiles_s = n_my_tiles;
  __syncthreads();
  for (int t = 0; t < my_tiles_s; t++) {
    const int st = t % kShiftStages;
    mbar_wait(&full[st], (uint32_t)((t / kShiftStages) & 1));
    const double *Ys = stage_base + (size_t)st * stage_doubles;
    const double *Ps = Ys + y_doubles;
    const double *Ss = Ps + p_doubles;
    const double *Es = Ss + s_doubles;                                           // [CT][RE]  Bmax, Bmax - Bmin, e^{-pT (Bmax - B_k)}

    // ---- block phase: the pair table does not depend on the species
    if constexpr (DF) {
      for (int w = threadIdx.x; w < CT * NYT * NPT; w += blockDim.x) {             // as in cf_kernel
        const int c = w / (NYT * NPT), r = w - c * (NYT * NPT), j = r / NPT, k = r - j * NPT;
        const double *yr = Ys + (c * NYT + j) * RY, *pr = Ps + (c * NPT + k) * kRec;
        pair_tab[(c * NYT + j) * NPP + k] = fma(pr[4], yr[4], -(pr[3] * yr[3]));
      }
      __syncthreads();
    }

    for (int c = 0; c < CT; c++) {
      const double2 k01 = *reinterpret_cast<const double2 *>(Ss + c * kScal);
      const double K2 = k01.y;
      const double K3 = (MODEL == M_JONAHLIN) ? Ss[c * kScal + 2] : 0.0;
      const double K31 = (MODEL == M_JONAHLIN) ? K3 + 1.0 : 1.0;
      const double K0m = k01.x * m2;
      // (member-by-member body: pT re-read per cell, two registers fewer in the slots)
      const double pTc = LEAN ? pT_s[ipT] : pT, pT2c = LEAN ? pTc * pTc : pT2;
      const double2 bb = *reinterpret_cast<const double2 *>(Es + c * RE);
      const double qm = pTc * bb.x;                                               // largest pT B_k of the tile
      const int rare_hi = __double2hiint(fma(-pTc, bb.y, rare_x));                 // xm >= 707.7 - pT (Bmax - Bmin): scaled path
      double q[NPT], pd[NPT], g0[NPT], eB[NPT];
#pragma unroll
      for (int k = 0; k < NPT; k++) {
        const double2 *pr = reinterpret_cast<const double2 *>(Ps + (c * NPT + k) * kRec);
        const double2 v0 = pr[0];
        q[k] = pTc * v0.x;
        pd[k] = pTc * v0.y;
        g0[k] = DF ? fma(pT2c, pr[1].x, K0m) : 0.0;
        eB[k] = Es[c * RE + 2 + k * L.n_pT + ipT];
      }
#pragma unroll
      for (int j = 0; j < NYT; j++) {
        const double2 *yr = reinterpret_cast<const double2 *>(Ys + (c * NYT + j) * RY);
        const double2 v0 = yr[0];
        const double a = mT * v0.x;
        const double xm = a - qm;                                                // smallest argument of the group
        const int xh = __double2hiint(xm);
        // Control flow is WARP-uniform (votes): a lane whose group is dead (every member's exp(x) overflows: exact zeros) rides
        // along with e^{-xm} := 0, which makes its f_eq and therefore its contribution an exact 0.
        const bool alive = xh <= kAliveHi;
        if (!__any_sync(0xffffffffu, alive)) continue;
        const double cpm = mT * v0.y;
        const double h0 = DF ? mT2 * yr[1].x : 0.0;
        // (the eta weight of a 3+1D slot record is 1: p.dsigma = pT Dp + mT Cp)
        const double *prj = pair_tab + (c * NYT + j) * NPP;
        double *accj = acc + j * NPT;
        if constexpr (!LEAN) {
          // staged slot body: the NPT members' arguments, p.dsigma and delta-f polynomials are formed together, then the group
          double pr2[NPP], xs[NPT], pv[NPT], sv[NPT];
#pragma unroll
          for (int k = 0; k < NPP; k += 2) {
            const double2 t2 = *reinterpret_cast<const double2 *>(prj + k);
            pr2[k] = t2.x; pr2[k + 1] = t2.y;
          }
#pragma unroll
          for (int k = 0; k < NPT; k++) {
            xs[k] = a - q[k];
            pv[k] = pd[k] + cpm;
            sv[k] = fma(mTpT, pr2[k], h0 + g0[k]);
          }
          if (__builtin_expect(__any_sync(0xffffffffu, alive && xh >= rare_hi), 0)) {
            // some member of some lane may be sub-normal, or dead inside an alive group: member by member, exactly as cf_kernel
            double fv[NPT];
            distribution_group<MODEL, NPT>(xs, true, false, sv, K2, K3, sign, reg_thr, one_hi, fv);
#pragma unroll
            for (int k = 0; k < NPT; k++) accumulate_pos(accj[k], pv[k], fv[k], thr_hi);
            continue;
          }
          double pe; int ne;
          exp_neg_poly_at(xm, tab_addr, hp.ec, pe, ne);
          const double eA = alive ? exp_neg_fast(pe, ne) : 0.0;
          double av[NPT], dfs[NPT], feq[NPT], fb[NPT], g[NPT];
#pragma unroll
          for (int k = 0; k < NPT; k++) {
            av[k] = eA * eB[k];
            dfs[k] = fma(sv[k], rcp_fast(xs[k]), K2 * xs[k]);
          }
          if (__all_sync(0xffffffffu, xh >= kUltraHi)) {
#pragma unroll
            for (int k = 0; k < NPT; k++) { feq[k] = av[k]; g[k] = dfs[k] + K31; }
          } else if (__all_sync(0xffffffffu, xh >= kDiluteHi)) {
#pragma unroll
            for (int k = 0; k < NPT; k++) { feq[k] = occupation_bar_dilute(av[k], sign, fb[k]); g[k] = fma(fb[k], dfs[k], K31); }
          } else {
#pragma unroll
            for (int k = 0; k < NPT; k++) { feq[k] = occupation_bar(av[k], sign, fb[k]); g[k] = fma(fb[k], dfs[k], K31); }
          }
#pragma unroll
          for (int k = 0; k < NPT; k++)
            accj[k] = fma(pv[k], feq[k] * clamp_mask_g(g[k], pv[k], reg_lo, reg_hi, reg_chk, thr_hi), accj[k]);
        } else {
          double pe; int ne;
          exp_neg_poly_at(xm, tab_addr, hp.ec, pe, ne);
          // some member of some lane may be sub-normal, or dead inside an alive group: e^{-xm} is formed 2^kRareShift too large
          // (a normal number for every alive xm) and each member is scaled back after the product (one rounding to sub-normal)
          const bool rare = __builtin_expect(__any_sync(0xffffffffu, alive && xh >= rare_hi), 0);
          const double eA = alive ? exp_neg_fast(pe, ne + (rare ? kRareShift : 0)) : 0.0;
          // a_k <= e^{-xm} for every member: 1 / (1 + Theta a) is 1 to half an ulp once xm >= 37.5 (a < 2^-54; 57 % of the alive
          // groups of a whole warp on the cfg3 surface), 1 - Theta a + a^2 to 5e-17 once xm >= 12.5 (a < 2^-18; 35 %), else MUFU + 3 DFMA
          // (dead lanes have xh > kAliveHi and pass every test)
          const int cls = __all_sync(0xffffffffu, xh >= kUltraHi) ? 0 : __all_sync(0xffffffffu, xh >= kDiluteHi) ? 1 : 2;
          auto slot = [&](auto rare_c, auto cls_c) {
            shift_slot<MODEL, NPT, decltype(rare_c)::value, decltype(cls_c)::value>(a, cpm, h0, prj, q, pd, g0, eB, eA, mTpT, K2, sign,
                                                                                 reg_lo, reg_hi, reg_chk, thr_hi, accj);
          };
          if (rare) {
            if (cls == 0) slot(IntC<1>(), IntC<0>()); else if (cls == 1) slot(IntC<1>(), IntC<1>()); else slot(IntC<1>(), IntC<2>());
          } else {
            if (cls == 0) slot(IntC<0>(), IntC<0>()); else if (cls == 1) slot(IntC<0>(), IntC<1>()); else slot(IntC<0>(), IntC<2>());
          }
        }
      }
    }
    __syncthreads();                                   // every warp is done with stage st and with the pair table
    if (threadIdx.x == 0 && t + kShiftStages < my_tiles_s) issue(t + kShiftStages);
  }

  // the class index is derived again rather than kept live across the cell loop, where its register would be spilled
  int tid = threadIdx.x;
  asm volatile("" : "+r"(tid));
  const int icls_e = ((gb * hp.n_warps + (tid >> 5)) * 32 + (tid & 31)) / L.n_pT;
  // partial[chunk][species + n_species (ipT + n_pT (iphi + n_phi iy))] for every member species of the class, with the scale of
  // hot_epilogue (operation = 1; the shifted-factor path has no momentum-integrated epilogue).  Members innermost: with the
  // bins innermost the compiler keeps all NYT x NPT bin offsets live across the member loop.
  if (!lane_valid) return;
  const int64_t n_bins = (int64_t)L.n_species * L.n_pT * L.n_phi * L.n_y_out;
  double *out = hp.partial + (int64_t)chunk * n_bins;
  const int m0 = cls.first[icls_e], m1 = cls.first[icls_e + 1];
#pragma unroll
  for (int j = 0; j < NYT; j++) {
    const int iy = ty * NYT + j;
    if (iy >= L.n_slots) continue;
#pragma unroll
    for (int k = 0; k < NPT; k++) {
      const int iphi = tp * NPT + k;
      if (iphi >= L.n_phi) continue;
      double *o = out + (int64_t)L.n_species * ((int64_t)ipT + (int64_t)L.n_pT * ((int64_t)iphi + (int64_t)L.n_phi * iy));
      for (int m = m0; m < m1; m++) {
        const int sp = cls.members[m];
        o[sp] = (hp.prefactor * hp.degeneracy[sp]) * acc[j * NPT + k];
      }
    }
  }
}

// ct: the longest tile; shift_variant_shape shortens it where the pipeline would not fit minb blocks per SM
struct ShiftShape { int nyt, npt, ct, minb; };
const ShiftShape kShiftShapesLean[kNumShiftVariants] = {{7, 3, 16, 3}, {3, 6, 16, 3}, {3, 8, 16, 3}, {7, 6, 16, 2}};
const ShiftShape kShiftShapesStaged[kNumShiftVariants] = {{7, 2, 16, 4}, {7, 3, 16, 3}, {7, 4, 16, 2}, {7, 6, 16, 2}};

// dynamic shared memory of cf_shift_kernel: kShiftStages stages of a ct-cell tile (Y, P, S records and the table slice), their
// mbarriers, the pair table and the pT table
size_t shift_pipe_bytes(int nyt, int npt, int ct, int n_pT)
{
  const size_t stage_doubles = (size_t)ct * (nyt * kRec + npt * kRec + kScal + shift_erec(npt, n_pT));
  return kShiftStages * stage_doubles * 8 + kShiftStages * 8 + ((size_t)ct * nyt * ((npt + 1) & ~1) + n_pT) * 8;
}

template <int MODEL, int NYT, int NPT, int MINB>
cudaError_t launch_shift_one(const HotParams &hp, const SpeciesClasses &cls, int win_chunks, cudaStream_t st, size_t *smem_out, int *launches)
{
  const Layout &L = hp.L;
  const size_t smem = shift_pipe_bytes(NYT, NPT, L.ct, L.n_pT);
  if (smem_out) *smem_out = smem;
  *launches = 0;
  auto kern = cf_shift_kernel<MODEL, NYT, NPT, MINB>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t n_bintiles = (int64_t)hp.n_groupblocks * L.n_ytiles * L.n_ptiles;
  if (n_bintiles == 0) return cudaSuccess;
  // the grid is chunk-major: a window of chunks is a contiguous range of blocks, and its cells a contiguous range of tiles
  for (int c0 = 0; c0 < hp.n_chunks; c0 += win_chunks) {
    const int c1 = std::min(hp.n_chunks, c0 + win_chunks);
    const int64_t cell0 = (L.n_tiles * (int64_t)c0) / hp.n_chunks * L.ct, cell1 = (L.n_tiles * (int64_t)c1) / hp.n_chunks * L.ct;
    const int64_t n_threads = L.n_ptiles * (cell1 - cell0) * L.n_pT;
    if (n_threads > 0) {
      cf_shift_table_kernel<NPT, shift_lean(MODEL)><<<(unsigned)((n_threads + 127) / 128), 128, 0, st>>>(hp, hp.E, cell0, cell1 - cell0);
      ++*launches;
    }
    HotParams hw = hp;
    hw.chunk0 = c0;
    kern<<<(unsigned)(n_bintiles * (c1 - c0)), 128, smem, st>>>(hw, cls);
    ++*launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

template <int MODEL>
cudaError_t launch_shift_model(const HotParams &hp, const SpeciesClasses &cls, int v, int win_chunks, cudaStream_t st, size_t *smem_out, int *launches)
{
  if constexpr (shift_lean(MODEL)) {
    switch (v) {
      case 0: return launch_shift_one<MODEL, 7, 3, 3>(hp, cls, win_chunks, st, smem_out, launches);
      case 1: return launch_shift_one<MODEL, 3, 6, 3>(hp, cls, win_chunks, st, smem_out, launches);
      case 2: return launch_shift_one<MODEL, 3, 8, 3>(hp, cls, win_chunks, st, smem_out, launches);
      case 3: return launch_shift_one<MODEL, 7, 6, 2>(hp, cls, win_chunks, st, smem_out, launches);
      default: return cudaErrorInvalidValue;
    }
  } else {
    switch (v) {
      case 0: return launch_shift_one<MODEL, 7, 2, 4>(hp, cls, win_chunks, st, smem_out, launches);
      case 1: return launch_shift_one<MODEL, 7, 3, 3>(hp, cls, win_chunks, st, smem_out, launches);
      case 2: return launch_shift_one<MODEL, 7, 4, 2>(hp, cls, win_chunks, st, smem_out, launches);
      case 3: return launch_shift_one<MODEL, 7, 6, 2>(hp, cls, win_chunks, st, smem_out, launches);
      default: return cudaErrorInvalidValue;
    }
  }
}

}  // namespace

bool shift_supported(int model, const Layout &L)
{
  return !L.dim2 && L.n_pT <= kShiftMaxPT && (model == M_LIN14 || model == M_LINCE || model == M_JONAHLIN || model == M_IDEAL);
}

// The table slice makes a stage grow with n_pT (16 x (2 + NPT n_pT) doubles): where the 16-cell pipeline would not leave room
// for the shape's blocks/SM (3 x 8 at 32 pT points, 3 x 6 beyond 36), the tile is halved until it does: a shorter tile only
// adds per-tile synchronisation, while a block less per SM leaves fewer warps to hide the latency of the FP64 chains.
void shift_variant_shape(int model, int v, int n_pT, int *nyt, int *npt, int *ct, int *max_warps)
{
  if (v < 0 || v >= kNumShiftVariants) v = 0;
  const ShiftShape &s = shift_lean(model) ? kShiftShapesLean[v] : kShiftShapesStaged[v];
  int dev = 0, sm_bytes = 0, reserved = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sm_bytes, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev) != cudaSuccess) {
    cudaGetLastError();
    sm_bytes = 228 << 10; reserved = 1 << 10;                                  // B200
  }
  // per block: the SM's share, less the runtime's reservation and the static exp table (+ a few block-wide scalars)
  const int64_t budget = (int64_t)sm_bytes / s.minb - reserved - (kExpTabSize * 8 + 128);
  int c = s.ct;
  while (c > 2 && (int64_t)shift_pipe_bytes(s.nyt, s.npt, c, n_pT) > budget) c /= 2;
  *nyt = s.nyt; *npt = s.npt; *ct = c; *max_warps = 4;
}

int shift_table_record(const Layout &L) { return shift_erec(L.npt, L.n_pT); }

// the block is always 4 warps: hp.n_warps must be 4 and hp.n_groupblocks = ceil(cls.n n_pT / 128); hp.E holds the table of
// win_chunks chunks (hp.e_cells >= cells of any win_chunks consecutive chunks)
cudaError_t launch_shift(int model, const HotParams &hp, const SpeciesClasses &cls, int v, int win_chunks, cudaStream_t st, size_t *smem_out,
                         int *launches)
{
  switch (model) {
    case M_LIN14: return launch_shift_model<M_LIN14>(hp, cls, v, win_chunks, st, smem_out, launches);
    case M_LINCE: return launch_shift_model<M_LINCE>(hp, cls, v, win_chunks, st, smem_out, launches);
    case M_JONAHLIN: return launch_shift_model<M_JONAHLIN>(hp, cls, v, win_chunks, st, smem_out, launches);
    case M_IDEAL: return launch_shift_model<M_IDEAL>(hp, cls, v, win_chunks, st, smem_out, launches);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace is3d
