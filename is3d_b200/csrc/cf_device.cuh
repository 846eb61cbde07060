// cf_device.cuh -- device-side helpers for the Cooper-Frye kernels (sm_100a only).
//
//  * mbarrier + 1-D TMA bulk copy wrappers (cp.async.bulk, SASS: UBLKCP / SYNCS) used to stream cell tiles
//    from HBM/L2 into shared memory;
//  * exp_neg(): exp(-x) = 2^n T[j] e^r with -x = (256 n + j) ln2/256 + r: Cody-Waite reduction, a 256-entry table of 2^{j/256}
//    in shared memory, degree-4 polynomial -- 9 FP64-pipe instructions (the table-free degree-11 form needs 15), integer
//    exponent insertion on the ALU pipe, and the IEEE overflow semantics of the reference's
//    `1.0 / (exp(x) + sign)` (smooth_kernels.cpp:289): exactly 0 once exp(x) would overflow, gradual underflow below;
//  * rcp_fast(): MUFU.RCP64H seed + one cubically convergent correction (3 DFMA), relative error < 1e-15;
//  * distribution<MODEL>() / distribution_group<MODEL, N>(): f_eq (1 + df) of the linear-df models per evaluation / per group,
//    shared by cf_kernel and the kernels built on its records (cf_hbt.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "cf_internal.h"

namespace is3d {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{ asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }

__device__ __forceinline__ void mbar_fence_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{ asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory"); }

__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{ while (!mbar_try_wait(bar, parity)) { } }

// global -> shared bulk copy (TMA, non-tensor form); bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double rcp_fast(double b)
{
  double y0;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(b));
  double e = fma(-b, y0, 1.0);
  e = fma(e, e, e);
  return fma(y0, e, y0);
}

// sqrt(v), v > 0: MUFU.RSQ64H seed + two Goldschmidt steps (7 FP64-pipe instructions), relative error < 1e-15
__device__ __forceinline__ double sqrt_fast(double v)
{
  double y0;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(v));
  double g = v * y0, h = 0.5 * y0;
  double r = fma(-g, h, 0.5);
  g = fma(g, r, g); h = fma(h, r, h);
  r = fma(-g, h, 0.5);
  return fma(g, r, g);
}

// exp(x) overflows to +inf in the reference for x > ln(DBL_MAX); there 1/(inf + sign) = 0 exactly
#define IS3D_EXP_OVERFLOW_X 709.782712893384

// Constants live in constant memory so that DFMA reads them as c[bank][offset] operands (a literal costs two UMOV issue
// slots per use, which makes the loop issue-bound instead of FP64-bound).
//   kExpC: 1/4!, 1/3!, 1/2!          kExpR: -256/ln2, 1.5 * 2^52, -ln2_hi/256, -ln2_lo/256 (ln2_hi has 20 trailing zero bits:
//                                           k * ln2_hi/256 is exact for |k| < 2^20; here |k| <= 709.8 * 256 / ln2 < 2^18.01)
constexpr int kExpTabBits = 8, kExpTabSize = 1 << kExpTabBits;
__constant__ double kExpC[3] = {4.1666666666666664e-02, 1.6666666666666666e-01, 0.5};
__constant__ double kExpR[4] = {-369.3299304675746, 6755399441055744.0, -0.00270760617331689, -7.453964567463233e-13};
// 2^{j/256}, j = 0..255, correctly rounded
__constant__ double kExpT[kExpTabSize] = {
  0x1.0000000000000p+0, 0x1.00b1afa5abcbfp+0, 0x1.0163da9fb3335p+0, 0x1.02168143b0281p+0,
  0x1.02c9a3e778061p+0, 0x1.037d42e11bbccp+0, 0x1.04315e86e7f85p+0, 0x1.04e5f72f654b1p+0,
  0x1.059b0d3158574p+0, 0x1.0650a0e3c1f89p+0, 0x1.0706b29ddf6dep+0, 0x1.07bd42b72a836p+0,
  0x1.0874518759bc8p+0, 0x1.092bdf66607e0p+0, 0x1.09e3ecac6f383p+0, 0x1.0a9c79b1f3919p+0,
  0x1.0b5586cf9890fp+0, 0x1.0c0f145e46c85p+0, 0x1.0cc922b7247f7p+0, 0x1.0d83b23395decp+0,
  0x1.0e3ec32d3d1a2p+0, 0x1.0efa55fdfa9c5p+0, 0x1.0fb66affed31bp+0, 0x1.1073028d7233ep+0,
  0x1.11301d0125b51p+0, 0x1.11edbab5e2ab6p+0, 0x1.12abdc06c31ccp+0, 0x1.136a814f204abp+0,
  0x1.1429aaea92de0p+0, 0x1.14e95934f312ep+0, 0x1.15a98c8a58e51p+0, 0x1.166a45471c3c2p+0,
  0x1.172b83c7d517bp+0, 0x1.17ed48695bbc0p+0, 0x1.18af9388c8deap+0, 0x1.1972658375d2fp+0,
  0x1.1a35beb6fcb75p+0, 0x1.1af99f8138a1cp+0, 0x1.1bbe084045cd4p+0, 0x1.1c82f95281c6bp+0,
  0x1.1d4873168b9aap+0, 0x1.1e0e75eb44027p+0, 0x1.1ed5022fcd91dp+0, 0x1.1f9c18438ce4dp+0,
  0x1.2063b88628cd6p+0, 0x1.212be3578a819p+0, 0x1.21f49917ddc96p+0, 0x1.22bdda27912d1p+0,
  0x1.2387a6e756238p+0, 0x1.2451ffb82140ap+0, 0x1.251ce4fb2a63fp+0, 0x1.25e85711ece75p+0,
  0x1.26b4565e27cddp+0, 0x1.2780e341ddf29p+0, 0x1.284dfe1f56381p+0, 0x1.291ba7591bb70p+0,
  0x1.29e9df51fdee1p+0, 0x1.2ab8a66d10f13p+0, 0x1.2b87fd0dad990p+0, 0x1.2c57e39771b2fp+0,
  0x1.2d285a6e4030bp+0, 0x1.2df961f641589p+0, 0x1.2ecafa93e2f56p+0, 0x1.2f9d24abd886bp+0,
  0x1.306fe0a31b715p+0, 0x1.31432edeeb2fdp+0, 0x1.32170fc4cd831p+0, 0x1.32eb83ba8ea32p+0,
  0x1.33c08b26416ffp+0, 0x1.3496266e3fa2dp+0, 0x1.356c55f929ff1p+0, 0x1.36431a2de883bp+0,
  0x1.371a7373aa9cbp+0, 0x1.37f26231e754ap+0, 0x1.38cae6d05d866p+0, 0x1.39a401b7140efp+0,
  0x1.3a7db34e59ff7p+0, 0x1.3b57fbfec6cf4p+0, 0x1.3c32dc313a8e5p+0, 0x1.3d0e544ede173p+0,
  0x1.3dea64c123422p+0, 0x1.3ec70df1c5175p+0, 0x1.3fa4504ac801cp+0, 0x1.40822c367a024p+0,
  0x1.4160a21f72e2ap+0, 0x1.423fb2709468ap+0, 0x1.431f5d950a897p+0, 0x1.43ffa3f84b9d4p+0,
  0x1.44e086061892dp+0, 0x1.45c2042a7d232p+0, 0x1.46a41ed1d0057p+0, 0x1.4786d668b3237p+0,
  0x1.486a2b5c13cd0p+0, 0x1.494e1e192aed2p+0, 0x1.4a32af0d7d3dep+0, 0x1.4b17dea6db7d7p+0,
  0x1.4bfdad5362a27p+0, 0x1.4ce41b817c114p+0, 0x1.4dcb299fddd0dp+0, 0x1.4eb2d81d8abffp+0,
  0x1.4f9b2769d2ca7p+0, 0x1.508417f4531eep+0, 0x1.516daa2cf6642p+0, 0x1.5257de83f4eefp+0,
  0x1.5342b569d4f82p+0, 0x1.542e2f4f6ad27p+0, 0x1.551a4ca5d920fp+0, 0x1.56070dde910d2p+0,
  0x1.56f4736b527dap+0, 0x1.57e27dbe2c4cfp+0, 0x1.58d12d497c7fdp+0, 0x1.59c0827ff07ccp+0,
  0x1.5ab07dd485429p+0, 0x1.5ba11fba87a03p+0, 0x1.5c9268a5946b7p+0, 0x1.5d84590998b93p+0,
  0x1.5e76f15ad2148p+0, 0x1.5f6a320dceb71p+0, 0x1.605e1b976dc09p+0, 0x1.6152ae6cdf6f4p+0,
  0x1.6247eb03a5585p+0, 0x1.633dd1d1929fdp+0, 0x1.6434634ccc320p+0, 0x1.652b9febc8fb7p+0,
  0x1.6623882552225p+0, 0x1.671c1c70833f6p+0, 0x1.68155d44ca973p+0, 0x1.690f4b19e9538p+0,
  0x1.6a09e667f3bcdp+0, 0x1.6b052fa75173ep+0, 0x1.6c012750bdabfp+0, 0x1.6cfdcddd47645p+0,
  0x1.6dfb23c651a2fp+0, 0x1.6ef9298593ae5p+0, 0x1.6ff7df9519484p+0, 0x1.70f7466f42e87p+0,
  0x1.71f75e8ec5f74p+0, 0x1.72f8286ead08ap+0, 0x1.73f9a48a58174p+0, 0x1.74fbd35d7cbfdp+0,
  0x1.75feb564267c9p+0, 0x1.77024b1ab6e09p+0, 0x1.780694fde5d3fp+0, 0x1.790b938ac1cf6p+0,
  0x1.7a11473eb0187p+0, 0x1.7b17b0976cfdbp+0, 0x1.7c1ed0130c132p+0, 0x1.7d26a62ff86f0p+0,
  0x1.7e2f336cf4e62p+0, 0x1.7f3878491c491p+0, 0x1.80427543e1a12p+0, 0x1.814d2add106d9p+0,
  0x1.82589994cce13p+0, 0x1.8364c1eb941f7p+0, 0x1.8471a4623c7adp+0, 0x1.857f4179f5b21p+0,
  0x1.868d99b4492edp+0, 0x1.879cad931a436p+0, 0x1.88ac7d98a6699p+0, 0x1.89bd0a478580fp+0,
  0x1.8ace5422aa0dbp+0, 0x1.8be05bad61778p+0, 0x1.8cf3216b5448cp+0, 0x1.8e06a5e0866d9p+0,
  0x1.8f1ae99157736p+0, 0x1.902fed0282c8ap+0, 0x1.9145b0b91ffc6p+0, 0x1.925c353aa2fe2p+0,
  0x1.93737b0cdc5e5p+0, 0x1.948b82b5f98e5p+0, 0x1.95a44cbc8520fp+0, 0x1.96bdd9a7670b3p+0,
  0x1.97d829fde4e50p+0, 0x1.98f33e47a22a2p+0, 0x1.9a0f170ca07bap+0, 0x1.9b2bb4d53fe0dp+0,
  0x1.9c49182a3f090p+0, 0x1.9d674194bb8d5p+0, 0x1.9e86319e32323p+0, 0x1.9fa5e8d07f29ep+0,
  0x1.a0c667b5de565p+0, 0x1.a1e7aed8eb8bbp+0, 0x1.a309bec4a2d33p+0, 0x1.a42c980460ad8p+0,
  0x1.a5503b23e255dp+0, 0x1.a674a8af46052p+0, 0x1.a799e1330b358p+0, 0x1.a8bfe53c12e59p+0,
  0x1.a9e6b5579fdbfp+0, 0x1.ab0e521356ebap+0, 0x1.ac36bbfd3f37ap+0, 0x1.ad5ff3a3c2774p+0,
  0x1.ae89f995ad3adp+0, 0x1.afb4ce622f2ffp+0, 0x1.b0e07298db666p+0, 0x1.b20ce6c9a8952p+0,
  0x1.b33a2b84f15fbp+0, 0x1.b468415b749b1p+0, 0x1.b59728de5593ap+0, 0x1.b6c6e29f1c52ap+0,
  0x1.b7f76f2fb5e47p+0, 0x1.b928cf22749e4p+0, 0x1.ba5b030a1064ap+0, 0x1.bb8e0b79a6f1fp+0,
  0x1.bcc1e904bc1d2p+0, 0x1.bdf69c3f3a207p+0, 0x1.bf2c25bd71e09p+0, 0x1.c06286141b33dp+0,
  0x1.c199bdd85529cp+0, 0x1.c2d1cd9fa652cp+0, 0x1.c40ab5fffd07ap+0, 0x1.c544778fafb22p+0,
  0x1.c67f12e57d14bp+0, 0x1.c7ba88988c933p+0, 0x1.c8f6d9406e7b5p+0, 0x1.ca3405751c4dbp+0,
  0x1.cb720dcef9069p+0, 0x1.ccb0f2e6d1675p+0, 0x1.cdf0b555dc3fap+0, 0x1.cf3155b5bab74p+0,
  0x1.d072d4a07897cp+0, 0x1.d1b532b08c968p+0, 0x1.d2f87080d89f2p+0, 0x1.d43c8eacaa1d6p+0,
  0x1.d5818dcfba487p+0, 0x1.d6c76e862e6d3p+0, 0x1.d80e316c98398p+0, 0x1.d955d71ff6075p+0,
  0x1.da9e603db3285p+0, 0x1.dbe7cd63a8315p+0, 0x1.dd321f301b460p+0, 0x1.de7d5641c0658p+0,
  0x1.dfc97337b9b5fp+0, 0x1.e11676b197d17p+0, 0x1.e264614f5a129p+0, 0x1.e3b333b16ee12p+0,
  0x1.e502ee78b3ff6p+0, 0x1.e653924676d76p+0, 0x1.e7a51fbc74c83p+0, 0x1.e8f7977cdb740p+0,
  0x1.ea4afa2a490dap+0, 0x1.eb9f4867cca6ep+0, 0x1.ecf482d8e67f1p+0, 0x1.ee4aaa2188510p+0,
  0x1.efa1bee615a27p+0, 0x1.f0f9c1cb6412ap+0, 0x1.f252b376bba97p+0, 0x1.f3ac948dd7274p+0,
  0x1.f50765b6e4540p+0, 0x1.f6632798844f8p+0, 0x1.f7bfdad9cbe14p+0, 0x1.f91d802243c89p+0,
  0x1.fa7c1819e90d8p+0, 0x1.fbdba3692d514p+0, 0x1.fd3c22b8f71f1p+0, 0x1.fe9d96b2a23d9p+0};

// Per-block copy of kExpT in shared memory: the index differs from lane to lane, which constant memory would serialise.
// Every kernel that calls exp_neg*() must run exp_table_init() and a __syncthreads() first.
__shared__ double g_exp_tab[kExpTabSize];
__device__ __forceinline__ void exp_table_init()
{ for (int i = threadIdx.x; i < kExpTabSize; i += blockDim.x) g_exp_tab[i] = kExpT[i]; }

// Mantissa p in [0.998, 1.998] and binary exponent n with e^{-x} = p 2^n, for |x| < 2^19 ln2/256.
//   k = round(-256 x / ln2) = 256 n + j,  r = -x - k ln2/256 (|r| <= ln2/512),  e^r = 1 + r Q(r),  p = T_j + (T_j r) Q
// truncation r^5/5! < 3.8e-17; total error ~1 ulp (table entry, T r, final fma).  9 FP64-pipe instructions.
__device__ __forceinline__ void exp_neg_poly(double x, double &p_out, int &n_out)
{
  const double MAGIC = kExpR[1];                       // 1.5 * 2^52: round-to-nearest integer lands in the low word
  const double fk = fma(x, kExpR[0], MAGIC);
  const int k = __double2loint(fk);
  const double kf = fk - MAGIC;
  double r = fma(kf, kExpR[2], -x);                    // hi / lo split of ln2/256
  r = fma(kf, kExpR[3], r);
  const double T = g_exp_tab[k & (kExpTabSize - 1)];
  n_out = k >> kExpTabBits;
  double q = fma(kExpC[0], r, kExpC[1]);
  q = fma(q, r, kExpC[2]);
  q = fma(q, r, 1.0);
  p_out = fma(T * r, q, T);
}
// normal result: add n to the exponent field (ALU pipe, no FP64 slot)
__device__ __forceinline__ double exp_neg_fast(double p, int n)
{ return __hiloint2double(__double2hiint(p) + (n << 20), __double2loint(p)); }
__device__ __forceinline__ bool exp_neg_is_rare(int n) { return (unsigned)(n + 1021) > 2044u; }
// rare: subnormal result (708.4 < x <= 709.78).  Two-step scaling keeps the gradual-underflow rounding.
__device__ __forceinline__ double exp_neg_rare(double p, int n)
{
  const int n1 = n >> 1, n2 = n - n1;
  return (p * __hiloint2double((n1 + 1023) << 20, 0)) * __hiloint2double((n2 + 1023) << 20, 0);
}

// exp(-x) for x <= ln(DBL_MAX) (callers skip larger x: the reference's exp(x) overflows there and the term is 0).
// The staged pieces above let groups of evaluations interleave their chains and test the sub-normal case once per group.
__device__ __forceinline__ double exp_neg(double x)
{
  double p; int n;
  exp_neg_poly(x, p, n);
  return __builtin_expect(exp_neg_is_rare(n), 0) ? exp_neg_rare(p, n) : exp_neg_fast(p, n);
}

// true when the reference's exp(x) stays finite, i.e. x <= ln(DBL_MAX) = 0x40862E42FEFA39EF; integer compare on
// the ALU pipe (negative x has the sign bit set and passes).
__device__ __forceinline__ bool exp_finite(double x)
{ return __double_as_longlong(x) <= 0x40862E42FEFA39EFLL; }

// Grouped evaluation paths classify a whole group from the HIGH WORDS of its exponent arguments (integer min / max, one
// VIMNMX3 + ISETP each):
//   any_alive : some x <= 709.78271484375, the upper end of the high word of ln(DBL_MAX) -- otherwise every member's exp(x)
//               overflows in the reference, all terms are exactly 0 and the group is skipped;
//   maybe_rare: some x >= 707.70, where e^{-x} may be sub-normal.  The slow branch then re-tests each member exactly:
//               sub-normal results get the two-step scaling, arguments beyond ln(DBL_MAX) (dead members of a partly alive
//               group, including the sliver the high-word test lets through) get a = 0 and contribute an exact +0.
// So no per-member aliveness predicate and no select is needed on the fast path.
//   all_dilute: every x >= 12.5, i.e. a = e^{-x} < 2^-18: the quantum-statistics denominator 1 / (1 + Theta a) is then
//               1 - Theta a + a^2 to 5e-17 (2 DFMA instead of MUFU + 4).
constexpr int kAliveHi = 0x40862E42;
constexpr int kRareHi = 0x40861D99;
constexpr int kDiluteHi = 0x40290000;
template <int N>
__device__ __forceinline__ void group_flags(const double (&x)[N], bool &any_alive, bool &maybe_rare, bool &all_dilute)
{
  int lo = __double2hiint(x[0]), hi = lo;
#pragma unroll
  for (int i = 1; i < N; i++) { const int h = __double2hiint(x[i]); lo = min(lo, h); hi = max(hi, h); }
  any_alive = lo <= kAliveHi; maybe_rare = hi >= kRareHi; all_dilute = lo >= kDiluteHi;
}

// Slow branch of a group, per member: decided from x itself (n may have wrapped for absurdly large arguments)
__device__ __forceinline__ double exp_neg_slow(double x, double p, int n)
{
  if (__double2hiint(x) < kRareHi) return exp_neg_fast(p, n);  // ordinary member of a group that has a late one
  if (!exp_finite(x)) return 0.0;                              // the reference's exp(x) overflows: f = 0 exactly
  return exp_neg_is_rare(n) ? exp_neg_rare(p, n) : exp_neg_fast(p, n);
}

// acc += pds * f when p.dsigma passes the outflow test; the test looks at the high word only (thr_hi = 0: p.dsigma > 0,
// values below 2^-1042 count as 0;  thr_hi = INT_MIN: outflow off)
__device__ __forceinline__ void accumulate_pos(double &acc, double pds, double f, int thr_hi)
{
  asm("{\n\t.reg .pred p;\n\tsetp.gt.s32 p, %1, %2;\n\t@p fma.rn.f64 %0, %3, %4, %0;\n\t}"
      : "+d"(acc) : "r"(__double2hiint(pds)), "r"(thr_hi), "d"(pds), "d"(f));
}

// acc += pds * f when pds > thr (thr = +0 with outflow on: the reference skips p.dsigma <= 0, smooth_kernels.cpp:285;
// thr = LLONG_MIN with outflow off).  Sign/zero test on the integer pipe, predicated DFMA -- no select.
__device__ __forceinline__ void accumulate_outflow(double &acc, double pds, double f, long long thr)
{
  asm("{\n\t.reg .pred p;\n\tsetp.gt.s64 p, %1, %3;\n\t@p fma.rn.f64 %0, %2, %4, %0;\n\t}"
      : "+d"(acc) : "l"(__double_as_longlong(pds)), "d"(pds), "l"(thr), "d"(f));
}

// |v| >= 1 -> copysign(1, v), done on the integer pipe (regulate_deltaf, smooth_kernels.cpp:328).
// thr_hi = 0x3ff00000 when regulation is on, 0x7ff80000 (never reached by finite values) when off.
// one_hi = 0x3ff00000 handed in as a run-time value: with a register operand (hi & sign) | one is a single LOP3.
__device__ __forceinline__ double clamp_unit(double v, int thr_hi, int one_hi)
{
  const int hi = __double2hiint(v);
  const bool big = (hi & 0x7fffffff) >= thr_hi;
  const int hi2 = big ? ((hi & 0x80000000) | one_hi) : hi;
  const int lo2 = big ? 0 : __double2loint(v);
  return __hiloint2double(hi2, lo2);
}

// Bose/Fermi factor 1 / (e^x + Theta) from a = e^{-x}
__device__ __forceinline__ double occupation(double a, double sign) { return a * rcp_fast(fma(sign, a, 1.0)); }
// The same plus 1 - Theta f_eq, which equals 1 / (1 + Theta e^{-x}) exactly: the reciprocal itself (one DFMA less, and more
// accurate than the reference's 1 - sign * feq where that cancels)
__device__ __forceinline__ double occupation_bar(double a, double sign, double &feqbar)
{ feqbar = rcp_fast(fma(sign, a, 1.0)); return a * feqbar; }
// dilute form, a < 2^-18: 1 / (1 + Theta a) = 1 - Theta a + a^2 - ... truncated after a^2 (|error| < a^3 < 5.2e-17)
__device__ __forceinline__ double occupation_bar_dilute(double a, double sign, double &feqbar)
{ feqbar = fma(a, a, fma(-sign, a, 1.0)); return a * feqbar; }

// f_eq (1 + df) of the linear-df models; x = u.p/T, s = partial delta-f polynomial (see cf_prepare.cu)
template <int MODEL>
__device__ __forceinline__ double distribution(double x, double s, double K2, double K3, double sign, int reg_thr, int one_hi)
{
  if (MODEL == M_IDEAL) return occupation(exp_neg(x), sign);      // df = 0: f = f_eq (1 + 0)
  double dfs;
  if (MODEL == M_LIN14) dfs = fma(K2 * x, x, s);               // + Pi bulk2 (u.p)^2
  else dfs = fma(s, rcp_fast(x), K2 * x);                      // [..]/(u.p) + (..)(u.p)
  const double feq = occupation(exp_neg(x), sign);
  const double feqbar = fma(-sign, feq, 1.0);
  double df = (MODEL == M_JONAHLIN) ? fma(feqbar, dfs, K3) : feqbar * dfs;
  df = clamp_unit(df, reg_thr, one_hi);                                // regulate_deltaf
  return fma(feq, df, feq);
}

// f_eq (1 + df) of the linear-df models (x = u.p/T, s = partial delta-f polynomial, see cf_prepare.cu) for a group of N evaluations, staged so that the N dependency chains can be interleaved
template <int MODEL, int N>
__device__ __forceinline__ void distribution_group(const double (&x)[N], bool maybe_rare, bool all_dilute, const double (&s)[N], double K2, double K3,
                                                   double sign, int reg_thr, int one_hi, double (&f)[N])
{
  double p[N], a[N], dfs[N]; int n[N];
#pragma unroll
  for (int i = 0; i < N; i++) {
    exp_neg_poly(x[i], p[i], n[i]);
    if (MODEL == M_IDEAL) dfs[i] = 0.0;
    else if (MODEL == M_LIN14) dfs[i] = fma(K2 * x[i], x[i], s[i]);
    else dfs[i] = fma(s[i], rcp_fast(x[i]), K2 * x[i]);
  }
  if (__builtin_expect(maybe_rare, 0)) {              // both sides define a[]: no register shuffling on the fast side
#pragma unroll
    for (int i = 0; i < N; i++) a[i] = exp_neg_slow(x[i], p[i], n[i]);
  } else {
#pragma unroll
    for (int i = 0; i < N; i++) a[i] = exp_neg_fast(p[i], n[i]);
  }
  double feq[N], feqbar[N];
  if (all_dilute) {                                    // warp-divergent only where light species meet central rapidities
#pragma unroll
    for (int i = 0; i < N; i++) feq[i] = occupation_bar_dilute(a[i], sign, feqbar[i]);
  } else {
#pragma unroll
    for (int i = 0; i < N; i++) feq[i] = occupation_bar(a[i], sign, feqbar[i]);
  }
#pragma unroll
  for (int i = 0; i < N; i++) {
    if (MODEL == M_IDEAL) { f[i] = feq[i]; continue; }
    double df = (MODEL == M_JONAHLIN) ? fma(feqbar[i], dfs[i], K3) : feqbar[i] * dfs[i];
    df = clamp_unit(df, reg_thr, one_hi);
    f[i] = fma(feq[i], df, feq[i]);
  }
}

}  // namespace is3d
