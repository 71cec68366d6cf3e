// Per-slice, per-dimension Gaussian-process fit and prediction.
//
// Replaces NNGP_p.get_preds (models.py:185-226): for every output dimension j the 9*R
// Nelder-Mead searches (models.py:228-260, SciPy _minimize_neldermead) of the negative log
// marginal likelihood (models.py:240-252) of a squared-exponential GP on the m nearest
// neighbours (models.py:86-92, 145-155), the selection rule (models.py:212-215) and the
// posterior mean (models.py:162-168) -- one launch per predict instead of d*9*R pickled
// tasks through pool.map.
//
// Mapping.  One WARP per Nelder-Mead search.  The searches of a launch (nq*d*9*R tasks, or one rank's
// block of output dimensions) sit in a queue ordered by gp_order_kernel; a persistent grid of
// independent warps pulls them with an atomic counter, so a warp that finishes a short search
// immediately starts another one (search lengths vary from ~10 to 400 objective evaluations).  The
// warp that completes the last search of an (query, dimension) pair applies the selection rule and
// computes the posterior mean (no block barrier, no second launch).  A launch with fewer searches than
// warp slots (a rank's share of the dimension-sharded sweep) lasts as long as its longest search: there
// gp_fit_spec_kernel gives a search the four warps of a CTA, which evaluate the points an iteration
// can ask for side by side (same decisions, same bits).  Inside a warp the M(M-1)/2
// kernel entries are spread over the lanes, exchanged through a per-warp shared-memory tile, and
// lane r owns row r of the m x m kernel matrix (m <= 32) in registers: square-root-free
// right-looking LDL^T, pivot broadcast by shuffle, column broadcast through the tile with
// warp-uniform 16-byte loads, forward solve fused into the factorisation (gp_core).  The m x m
// squared-distance matrix of the neighbours is computed once per query (gp_prep_kernel); a lane keeps
// the distances of its entries in registers for the whole search.
//
// Arithmetic.  The simplex arithmetic uses explicitly rounded (non-fused) operations in SciPy's
// order.  The objective is the reference's  0.5 y^T K^-1 y + sum log L_ii + (m/2) log 2 pi  evaluated
// as 0.5 (sum_k z_k^2 / d_k + log prod_k d_k) with the LDL^T pivots d_k = L_kk^2 and z = L'^-1 y
// (identical in exact arithmetic; the reference's own optimiser trajectories are not reproducible
// below 1 ulp of the objective, see DESIGN.md "ties").  A pivot that is <= `guard` ulp of the diagonal
// (default 1 ulp, the threshold at which the failure set agrees with LAPACK's potrf without bias in either
// direction -- oracle/experiments/pivot_rule_study.py, DESIGN.md section 2), <= 0 or NaN fails and makes the
// objective +inf exactly as the reference does on a failed factorisation (NaN -> inf, models.py:250-251).
#include "common.cuh"

#include <cmath>
#include <cstdlib>

static constexpr int GP_WARPS = 4;  // warps per CTA of the persistent fit kernel
static constexpr unsigned FULL = 0xffffffffu;

// 10**jitter for jitter = -20..-12 (models.py:186, :88)
__constant__ double c_jit10[NNGP_N_JITTER] = {1e-20, 1e-19, 1e-18, 1e-17, 1e-16,
                                              1e-15, 1e-14, 1e-13, 1e-12};

__device__ __forceinline__ double shfl(double v, int src) { return __shfl_sync(FULL, v, src); }
__device__ __forceinline__ double dinf() { return __longlong_as_double(0x7ff0000000000000LL); }
__device__ __forceinline__ double dnan() { return __longlong_as_double(0x7ff8000000000000LL); }

// ---------------------------------------------------------------------------------------
// Elementary functions of the GP kernels, written for short dependency chains (a Nelder-Mead
// search is a serial chain of objective evaluations, so latency, not throughput, bounds a launch)
// and so that every constant is a constant-bank operand of the FP64 instruction.
//   exp: x = k ln2 + r, |r| <= ln2/2; exp(r) = 1 + r (1 + r Q(r)), Q = E(r^2) + r O(r^2) the even / odd
//        halves of the rest of the degree-13 Taylor polynomial (remainder < 5e-18), result 2^k p(r); NaN propagates, x < -708.39
//        (subnormal results) returns 0.  The *_vec forms interleave NV independent evaluations.
//   10**x: x = k log10(2) + r, 10**r = exp(r ln 10), same polynomial; library routine outside |x| <= 300.
//   1/p: MUFU.RCP64H seed + one cubically convergent correction.
//   log: fdlibm's algorithm (s = f/(2+f), degree-14 even polynomial) with the reciprocal above.
// All are within ~1 ulp of the correctly rounded value (tests/test_gpu_kernels.py).
// ---------------------------------------------------------------------------------------
__constant__ double c_ev[6] = {2.08767569878681e-09,   // 1/12!
                               2.755731922398589e-07,  // 1/10!
                               2.48015873015873e-05,   // 1/8!
                               0.001388888888888889,   // 1/6!
                               0.041666666666666664,   // 1/4!
                               0.5};
__constant__ double c_od[6] = {1.6059043836821613e-10,  // 1/13!
                               2.505210838544172e-08,   // 1/11!
                               2.7557319223985893e-06,  // 1/9!
                               0.0001984126984126984,   // 1/7!
                               0.008333333333333333,    // 1/5!
                               0.16666666666666666};
__constant__ double c_exp[12] = {
    1.4426950408889634,           // [0] log2(e)
    6755399441055744.0,           // [1] 1.5 * 2^52: adding it rounds to the nearest integer
    -6.93147180369123816490e-01,  // [2] -ln2_hi
    -1.90821492927058770002e-10,  // [3] -ln2_lo
    -708.39,                      // [4] below this the result is subnormal: return 0
    3.321928094887362,            // [5] log2(10)
    -0.3010299955494702,          // [6] -log10(2) hi (21 trailing zero bits)
    -1.1451100898021838e-10,      // [7] -log10(2) lo
    2.302585092994046,            // [8] ln(10) hi
    -2.1707562233822494e-16,      // [9] ln(10) lo
    0.0, 0.0};                    // [10], [11] unused
__constant__ double c_log[9] = {6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01,
                                2.222219843214978396e-01, 1.818357216161805012e-01, 1.531383769920937332e-01,
                                1.479819860511658591e-01,
                                6.93147180369123816490e-01,   // [7] ln2_hi
                                1.90821492927058770002e-10};  // [8] ln2_lo

// 2^k[i] * exp(r[i]) for |r| <= ln2/2, k in [-1022, 1023]
template <int NV>
__device__ __forceinline__ void exp_reduced_vec(const double (&r)[NV], const int (&k)[NV], double (&out)[NV]) {
  double z[NV], e[NV], o[NV];
#pragma unroll
  for (int i = 0; i < NV; i++) z[i] = r[i] * r[i];
#pragma unroll
  for (int i = 0; i < NV; i++) {
    e[i] = fma(z[i], c_ev[0], c_ev[1]);
    o[i] = fma(z[i], c_od[0], c_od[1]);
  }
#pragma unroll
  for (int s = 2; s < 6; s++) {
#pragma unroll
    for (int i = 0; i < NV; i++) {
      e[i] = fma(e[i], z[i], c_ev[s]);
      o[i] = fma(o[i], z[i], c_od[s]);
    }
  }
  // exp(r) = 1 + r (1 + r Q(r)),  Q = e + r o: the last two steps in Horner form (one rounding each)
#pragma unroll
  for (int i = 0; i < NV; i++) e[i] = fma(r[i], o[i], e[i]);
#pragma unroll
  for (int i = 0; i < NV; i++) e[i] = fma(e[i], r[i], 1.0);
#pragma unroll
  for (int i = 0; i < NV; i++) out[i] = fma(e[i], r[i], 1.0) * __hiloint2double((k[i] + 1023) << 20, 0);
}

template <int NV>
__device__ __forceinline__ void exp_neg_vec(const double (&x)[NV], double (&out)[NV]) {
  double t[NV], r[NV];
  int k[NV];
#pragma unroll
  for (int i = 0; i < NV; i++) t[i] = fma(x[i], c_exp[0], c_exp[1]);
#pragma unroll
  for (int i = 0; i < NV; i++) {
    k[i] = __double2loint(t[i]);
    t[i] = t[i] - c_exp[1];
  }
#pragma unroll
  for (int i = 0; i < NV; i++) r[i] = fma(t[i], c_exp[2], x[i]);
#pragma unroll
  for (int i = 0; i < NV; i++) r[i] = fma(t[i], c_exp[3], r[i]);
  exp_reduced_vec<NV>(r, k, out);
#pragma unroll
  for (int i = 0; i < NV; i++) out[i] = (x[i] < c_exp[4]) ? 0.0 : out[i];  // false for NaN: NaN propagates
}

__device__ __forceinline__ double exp_neg(double x) {
  double xi[1] = {x}, o[1];
  exp_neg_vec<1>(xi, o);
  return o[0];
}

// 10**x (hyper-parameters are log10, models.py:145-148) for two arguments at once
__device__ __forceinline__ void exp10_pair(double x0, double x1, double& o0, double& o1) {
  if (!(fabs(x0) <= 300.0 && fabs(x1) <= 300.0)) {  // never reached by a search in practice
    o0 = exp10(x0);
    o1 = exp10(x1);
    return;
  }
  const double x[2] = {x0, x1};
  double t[2], r[2], y[2], o[2];
  int k[2];
#pragma unroll
  for (int i = 0; i < 2; i++) t[i] = fma(x[i], c_exp[5], c_exp[1]);
#pragma unroll
  for (int i = 0; i < 2; i++) {
    k[i] = __double2loint(t[i]);
    t[i] = t[i] - c_exp[1];
  }
#pragma unroll
  for (int i = 0; i < 2; i++) r[i] = fma(t[i], c_exp[6], x[i]);
#pragma unroll
  for (int i = 0; i < 2; i++) r[i] = fma(t[i], c_exp[7], r[i]);
#pragma unroll
  for (int i = 0; i < 2; i++) y[i] = fma(r[i], c_exp[8], r[i] * c_exp[9]);
  exp_reduced_vec<2>(y, k, o);
  o0 = o[0];
  o1 = o[1];
}

// 1/p for p > 0: seed relative error e0 ~ 2^-20; y (1 + e + e^2) has error e0^3
__device__ __forceinline__ double rcp_pos(double p) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(p));
  const double e = fma(-p, y, 1.0);
  const double t = fma(e, e, e);
  return fma(y, t, y);
}

// log(x) for positive normal x, plus kadd*ln2 (kadd an integer held as int)
__device__ __forceinline__ double log_pos_plus(double x, int kadd) {
  int hi = __double2hiint(x);
  const int lo = __double2loint(x);
  int k = (hi >> 20) - 1023 + kadd;
  hi = (hi & 0x000fffff) | 0x3ff00000;
  double mnt = __hiloint2double(hi, lo);  // [1, 2)
  if (mnt > 1.4142135623730951) {
    mnt = mnt * 0.5;
    k++;
  }
  const double f = mnt - 1.0;
  const double s = f * rcp_pos(2.0 + f);
  const double z = s * s;
  const double w = z * z;
  const double t1 = w * fma(w, fma(w, c_log[5], c_log[3]), c_log[1]);
  const double t2 = z * fma(w, fma(w, fma(w, c_log[6], c_log[4]), c_log[2]), c_log[0]);
  const double R = t1 + t2;
  const double hfsq = 0.5 * f * f;
  const double dk = (double)k;
  return dk * c_log[7] - ((hfsq - fma(s, hfsq + R, dk * c_log[8])) - f);
}

__global__ void selftest_math_kernel(const double* x, int n, double* out_exp, double* out_rcp,
                                     double* out_exp10) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out_exp[i] = exp_neg(-fabs(x[i]));
  out_rcp[i] = rcp_pos(fabs(x[i]));
  if (out_exp10) {
    double a, b;
    exp10_pair(x[i], -x[i], a, b);
    out_exp10[i] = a;
    // log hook: log(|x|) + 3 ln2 in the second half of the buffer when n is even (test convention)
    out_exp10[n + i] = log_pos_plus(fabs(x[i]), 3);
  }
}

int selftest_math_launch(nngp_handle_t h, const double* d_x, int n, double* d_exp, double* d_rcp,
                         double* d_exp10, cudaStream_t st) {
  if (n <= 0) return 0;
  selftest_math_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_x, n, d_exp, d_rcp, d_exp10);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------
// GP core for one warp (models.py:86-92): the objective of the Nelder-Mead searches (ALPHA =
// false: returns the negative log marginal likelihood, +inf on failure) and the refit at the
// selected hyper-parameters (ALPHA = true: returns alpha_lane = (K^-1 y)_lane).  ONE factorisation
// code for both, so a hyper-parameter whose objective was finite always refits successfully -- as
// in the reference, where both go through the same _fit_gp_jit.  Written for latency:
//   * the kernel matrix is symmetric: the M(M-1)/2 off-diagonal entries are spread over the 32
//     lanes (NP = ceil(M(M-1)/64) exponentials per lane instead of M), written to a per-warp
//     shared tile and read back as rows; the squared distances of a lane's entries stay in
//     registers for the whole search (no global loads per evaluation);
//   * no branch inside the factorisation: a failed pivot only clears a warp-uniform flag, so the
//     shuffles stay convergent and the critical path is  broadcast -> reciprocal -> 2 FMAs;
//   * hyper-parameter transforms 10**x with the same polynomial as the kernel entries.
// ---------------------------------------------------------------------------------------
template <int M>
struct Tri {
  static constexpr int NPAIR = M * (M - 1) / 2;
  static constexpr int NP = (NPAIR + 31) / 32;
  // row stride of the tile in doubles: LD/2 odd, so the 16-byte row reads of 8 consecutive lanes
  // fall into distinct bank groups
  static constexpr int LD = ((M / 2) & 1) ? M : M + 2;
  static constexpr int TILE = M * LD;
};

// which entries of the strict lower triangle a lane computes: e = lane + 32 t -> (i > j)
template <int M>
struct PairSlots {
  int oij[Tri<M>::NP];  // i*LD + j; an empty slot points at the unused diagonal element 0
  double r2[Tri<M>::NP];
  double r2_10;  // squared distance of neighbours 1 and 0 (every lane): decides pivot 1
  bool pad[Tri<M>::NP];  // entry touches a padding row (m <= i < M) or slot empty: stored as 0
};

template <int M>
__device__ __forceinline__ void pair_slots_init(PairSlots<M>& P, int lane, int m) {
#pragma unroll
  for (int t = 0; t < Tri<M>::NP; t++) {
    const int e = lane + 32 * t;
    int i = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)e)) * 0.5f);
    while (i * (i - 1) / 2 > e) i--;
    while ((i + 1) * i / 2 <= e) i++;
    const int j = e - i * (i - 1) / 2;
    const bool valid = e < Tri<M>::NPAIR;
    // an empty slot stores (zero) to the unused diagonal element K_00 instead of branching
    P.oij[t] = valid ? i * Tri<M>::LD + j : 0;
    P.pad[t] = !valid || (i >= m);
    P.r2[t] = 0.0;
  }
  P.r2_10 = 0.0;
}

// squared distances of the lane's entries for one query: r2 global [m*m] row-major
template <int M>
__device__ __forceinline__ void pair_slots_load(PairSlots<M>& P, const double* __restrict__ r2, int m) {
#pragma unroll
  for (int t = 0; t < Tri<M>::NP; t++) {
    double v = 0.0;
    if (!P.pad[t]) {
      const int i = P.oij[t] / Tri<M>::LD, j = P.oij[t] - i * Tri<M>::LD;
      v = __ldg(r2 + i * m + j);
    }
    P.r2[t] = v;
  }
  P.r2_10 = (m > 1) ? __ldg(r2 + m) : 0.0;
}

// Hyper-parameter transforms, scaling and the first two pivots -- everything that depends on (theta, jitter)
// and the single squared distance r2_10 only.  Arguments may differ from lane to lane (the Nelder-Mead loop
// evaluates the heads of four candidate points at once); gp_core calls it with warp-uniform arguments.
struct GpHead {
  double amp, c, sc, amp_s, dd0, pmin;
  bool fail01;  // pivot 0 or pivot 1 fails: the objective is +inf whatever the rest of the matrix holds
};

__device__ __forceinline__ GpHead gp_head(double th0, double th1, double jit10, double r2_10, int m, double guard) {
  GpHead g;
  double inv;  // amp = 10**sigma_y, inv = 1/(10**sigma_x)
  exp10_pair(th1, -th0, g.amp, inv);
  g.c = -0.5 * inv;
  // The matrix is factorised as K' = 2^-e0 K with e0 = the larger binary exponent of amp and jitter
  // (an exact scaling: every pivot is scaled by the same power of two), so that the product of up to
  // 16 pivots, each in (4 ulp, 4) after scaling, stays a normal number and log det K needs no
  // per-pivot exponent bookkeeping.
  const int e0 = min(1022, max((__double2hiint(g.amp) >> 20) & 0x7ff, (__double2hiint(jit10) >> 20) & 0x7ff) - 1023);
  g.sc = __hiloint2double((1023 - e0) << 20, 0);
  g.amp_s = g.amp * g.sc;
  // the diagonal exp(c*0) (NaN when c is not finite, as in NumPy) and the entry K_10
  const double x2[2] = {g.c * r2_10, g.c * 0.0};
  double e2[2];
  exp_neg_vec<2>(x2, e2);
  g.dd0 = fma(g.amp_s, e2[1], jit10 * g.sc);  // K'_rr;  K_rr = amp*exp(c*0) + 10**jitter
  // A pivot that is not above `guard` (= ulps * 2^-52, default 1 ulp) of the diagonal it was subtracted
  // from is rounding noise of an exactly singular matrix (e.g. identical neighbour rows at a steady
  // state, jitter below one ulp of the amplitude).  LAPACK's potf2 tests pivot <= 0, but it forms the
  // pivot as K_jj - (sum of squares): the sum is rounded at ulp(K_jj), so its pivots are multiples of
  // ulp(K_jj) carrying a few ulp of noise and a singular matrix fails with probability ~1/2 per
  // duplicated row.  The fused right-looking update below keeps the residue to full relative accuracy:
  // with a literal "<= 0" test it stays positive and cascades (d_k ~ eps^k), passing as a "valid" factor
  // with an absurdly small determinant where LAPACK fails.  Measured against np.linalg.cholesky on
  // steady-state neighbour sets (oracle/experiments/pivot_rule_study.py): at 1 ulp the two failure sets
  // differ on 1.3 % of the evaluations, evenly in both directions (a literal potf2 restatement differs
  // from the installed LAPACK on 1-4 %); at 4 ulp (round 1) the device failed 3.3 % more often.
  g.pmin = g.dd0 * guard;
  // pivots 0 and 1 with exactly the operations of the factorisation in gp_core
  const double k10 = (m > 1) ? g.amp_s * e2[0] : 0.0;
  const double d1 = fma(-(k10 * rcp_pos(g.dd0)), k10, g.dd0);
  g.fail01 = !(g.dd0 > g.pmin) || !(d1 > g.pmin);
  return g;
}

// Pivots 1..4 of the leading 5 x 5 block  b_ij = K'_ij (i > j, diagonal dd0)  with exactly the operations the
// factorisation in gp_core performs on these entries: true if one of them is not above pmin.  ip: the reciprocals
// of pivots 0..3, which the factorisation reuses.  Called warp-wide by gp_core and per lane by nm_screen_fails, so the
// two decide every point alike.
__device__ __forceinline__ bool block5_fails(double b10, double b20, double b30, double b40, double b21, double b31,
                                             double b32, double b41, double b42, double b43, double dd0, double pmin,
                                             double (&ip)[4]) {
  const double ip0 = rcp_pos(dd0);
  double w1 = b10 * ip0, w2 = b20 * ip0, w3 = b30 * ip0, w4 = b40 * ip0;
  const double d1 = fma(-w1, b10, dd0);
  double d2 = fma(-w2, b20, dd0), d3 = fma(-w3, b30, dd0), d4 = fma(-w4, b40, dd0);
  b21 = fma(-w2, b10, b21); b31 = fma(-w3, b10, b31); b41 = fma(-w4, b10, b41);
  b32 = fma(-w3, b20, b32); b42 = fma(-w4, b20, b42);
  b43 = fma(-w4, b30, b43);
  const double ip1 = rcp_pos(d1);
  w2 = b21 * ip1; w3 = b31 * ip1; w4 = b41 * ip1;
  d2 = fma(-w2, b21, d2); d3 = fma(-w3, b31, d3); d4 = fma(-w4, b41, d4);
  b32 = fma(-w3, b21, b32); b42 = fma(-w4, b21, b42);
  b43 = fma(-w4, b31, b43);
  const double ip2 = rcp_pos(d2);
  w3 = b32 * ip2; w4 = b42 * ip2;
  d3 = fma(-w3, b32, d3); d4 = fma(-w4, b42, d4);
  b43 = fma(-w4, b32, b43);
  const double ip3 = rcp_pos(d3);
  w4 = b43 * ip3;
  d4 = fma(-w4, b43, d4);
  ip[0] = ip0; ip[1] = ip1; ip[2] = ip2; ip[3] = ip3;
  // a failed pivot makes the later ones meaningless, exactly as in the factorisation (ok stays false)
  return !(d1 > pmin) || !(d2 > pmin) || !(d3 > pmin) || !(d4 > pmin);
}

struct GpOut {
  double val, amp, c;
  bool ok;
#ifdef NNGP_FIT_STATS
  int stage;  // 1: failed at pivots 0 / 1 (head), 2: at pivots 2..4 (leading block), 3: factorised further
#endif
};

template <int M, bool ALPHA>
__device__ __forceinline__ GpOut gp_core(double th0, double th1, double jit10, const PairSlots<M>& P,
                                         double y, int m, int lane, double* __restrict__ Kt,
                                         double hml, double guard) {
  static_assert(M % 2 == 0, "M even: 16-byte loads of column pairs");
  constexpr int LD = Tri<M>::LD;
  constexpr int NP = Tri<M>::NP;
  // A search that starts where the kernel matrix is numerically singular sees +inf at every vertex;
  // |inf - inf| = NaN never satisfies SciPy's fatol test, so it runs all maxfev = 400 evaluations (at the
  // FHN target, whose neighbour rows become identical at the steady state, 14 % of the searches and 57 % of
  // the evaluations), and nearly all of those fail at pivot 1: decided by the head alone, before the
  // matrix is built (every lane holds the same values: uniform branch).
  const GpHead hd = gp_head(th0, th1, jit10, P.r2_10, m, guard);
  const double amp = hd.amp, c = hd.c, sc = hd.sc, amp_s = hd.amp_s, dd0 = hd.dd0, pmin = hd.pmin;
  if (!ALPHA) {
    if (__any_sync(FULL, hd.fail01)) {
      GpOut bad;
      bad.amp = amp;
      bad.c = c;
      bad.ok = false;
      bad.val = dinf();
#ifdef NNGP_FIT_STATS
      bad.stage = 1;
#endif
      return bad;
    }
  }
  // kernel entries of this lane.  Slot 0 first: the pairs are numbered e = i(i-1)/2 + j and lane l owns e = l + 32 t,
  // so slot 0 of lanes 0..9 is the leading 5 x 5 block of the matrix.
  double v[NP];
  v[0] = exp_neg(c * P.r2[0]);
  bool fail5 = false;
  double ipb[4] = {0.0, 0.0, 0.0, 0.0};  // reciprocals of pivots 0..3, reused by the first four steps of the factorisation
  if (!ALPHA) {
    // Pivots 1..4 decided from the leading block alone, with exactly the operations the factorisation below
    // performs on these entries (same fused multiply-adds in the same order: the decision is only anticipated).
    // At a steady state 91 % of the failing evaluations fail here (first failing pivot 2: 40 %, 3: 37 %, 4: 13 %,
    // profiles/r02/fit_failing_pivots.log) and they are 44 % of all evaluations: such an evaluation now costs
    // one exponential and a 5 x 5 elimination instead of the whole kernel matrix, and the searches that run to
    // SciPy's 400-evaluation limit on failing points -- the chain that ends a launch -- shrink by 3-4x.
    const double k0 = P.pad[0] ? 0.0 : amp_s * v[0];
    fail5 = block5_fails(shfl(k0, 0), shfl(k0, 1), shfl(k0, 3), shfl(k0, 6), shfl(k0, 2), shfl(k0, 4), shfl(k0, 5),
                         shfl(k0, 7), shfl(k0, 8), shfl(k0, 9), dd0, pmin, ipb);
  }
  if constexpr (NP > 1) {
    constexpr int NV = NP - 1;
    constexpr int G = (NV <= 8) ? NV : (NV + 1) / 2;
    double xin[NV];
#pragma unroll
    for (int t = 0; t < NV; t++) xin[t] = c * P.r2[t + 1];
    {
      double xa[G], oa[G];
#pragma unroll
      for (int t = 0; t < G; t++) xa[t] = xin[t];
      exp_neg_vec<G>(xa, oa);
#pragma unroll
      for (int t = 0; t < G; t++) v[t + 1] = oa[t];
    }
    if constexpr (NV > G) {
      constexpr int G2 = NV - G;
      double xa[G2], oa[G2];
#pragma unroll
      for (int t = 0; t < G2; t++) xa[t] = xin[G + t];
      exp_neg_vec<G2>(xa, oa);
#pragma unroll
      for (int t = 0; t < G2; t++) v[G + t + 1] = oa[t];
    }
  }
  // the decision of the block above: its dependency chain (ten shuffles, four reciprocals) runs beside the
  // polynomial evaluation of the other slots, which are independent of it
  if (!ALPHA) {
    if (__any_sync(FULL, fail5)) {
      GpOut bad;
      bad.amp = amp;
      bad.c = c;
      bad.ok = false;
      bad.val = dinf();
#ifdef NNGP_FIT_STATS
      bad.stage = 2;
#endif
      return bad;
    }
  }
#pragma unroll
  for (int t = 0; t < NP; t++) {  // unconditional stores: the exponentials above stay interleaved
    // only the lower triangle is stored: lane r never uses the entries right of its diagonal
    Kt[P.oij[t]] = P.pad[t] ? 0.0 : amp_s * v[t];
  }
  __syncwarp();
  const bool rowvalid = lane < m;
  double a[M];
  {
    const double2* rowp = reinterpret_cast<const double2*>(Kt + ((lane < M) ? lane : 0) * LD);
#pragma unroll
    for (int j = 0; j < M; j += 2) {
      const double2 t2 = rowp[j >> 1];
      a[j] = t2.x;
      a[j + 1] = t2.y;
    }
  }
  __syncwarp();  // the tile is reused for the column broadcasts below
  // Square-root-free right-looking factorisation K = L' D L'^T, software-pipelined: the critical
  // path of a step is  pivot broadcast -> reciprocal -> w = a_rk/d_k -> diagonal update ; the updates
  // of the lanes that own the next pivot come first, the next broadcast and column store are issued
  // before the remaining trailing updates, and a column is read from shared memory into registers in
  // one batch.  Every lane sees every pivot d_k and (L'^-1 y)_k, so  y^T K^-1 y = sum w_k^2 / d_k  and
  // log det K = log prod d_k (mantissa product + exponent sum) are accumulated redundantly in all
  // lanes: no warp reduction, one logarithm.
  auto load_col = [&](int k, double (&u)[M]) {
    // u[j] = column k entry of row j (unscaled), j > k; uniform addresses -> broadcast loads
    int j = k + 1;
    if (j < M && (j & 1)) {
      u[j] = Kt[k * LD + j];
      j++;
    }
#pragma unroll
    for (; j + 1 < M; j += 2) {
      const double2 u2 = *reinterpret_cast<const double2*>(&Kt[k * LD + j]);
      u[j] = u2.x;
      u[j + 1] = u2.y;
    }
  };
  double dd = dd0;
  double z = rowvalid ? y : 0.0;
  double quad = 0.0, prod0 = 1.0, prod1 = 1.0;
  double inv_own = 1.0, w_own = 0.0;  // ALPHA: 1/d_r and (L'^-1 y)_r of the own row
  bool ok = true;
  double u[M];
  double p = dd0, zk = shfl(z, 0);
  if (lane > 0 && lane < M) Kt[lane] = a[0];
  __syncwarp();
  load_col(0, u);
#pragma unroll
  for (int k = 0; k < M; k++) {
    ok = ok && (p > pmin);  // failed factorisation (potf2: pivot <= 0 or NaN) -> +inf
    // A search that starts where the kernel matrix is numerically singular sees +inf at every vertex;
    // |inf - inf| = NaN never satisfies SciPy's fatol test, so it runs all maxfev = 400 evaluations
    // (at the FHN target 14 % of the searches, 57 % of the evaluations, and the serial chain that ends
    // the launch).  Near-duplicate neighbours fail at the first pivots: leave early at a few fixed
    // steps (warp-uniform vote, so the shuffles below stay convergent).
    if (!ALPHA && (k == 6 || k == 8 || k == 11 || k == 14) && k < M - 1) {
      if (__any_sync(FULL, !ok)) {
        GpOut bad;
        bad.amp = amp;
        bad.c = c;
        bad.ok = false;
        bad.val = dinf();
#ifdef NNGP_FIT_STATS
        bad.stage = 3;
#endif
        __syncwarp();  // the next evaluation overwrites the tile
        return bad;
      }
    }
    // pivots 0..3 are the bits the leading-block check already inverted: take its reciprocals off the critical path
    const double ip = (!ALPHA && k < 4) ? ipb[k] : rcp_pos(p);
    const double w = a[k] * ip;  // l'_rk
    const double pk = p, zkk = zk;
    if (ALPHA && lane == k) {
      inv_own = ip;
      w_own = zk;
    }
    dd = fma(-w, a[k], dd);
    z = fma(-w, zk, z);
    if (k + 1 < M) {
      a[k + 1] = fma(-w, u[k + 1], a[k + 1]);
      p = shfl(dd, k + 1);
      zk = shfl(z, k + 1);
      if (k + 2 < M) {
        if (lane > k + 1 && lane < M) Kt[(k + 1) * LD + lane] = a[k + 1];
        __syncwarp();
      }
#pragma unroll
      for (int j = k + 2; j < M; j++) a[j] = fma(-w, u[j], a[j]);
      if (k + 2 < M) load_col(k + 1, u);
    }
    if (!ALPHA) {  // off the critical path; a padding row has z = 0 and contributes nothing to the sum
      quad = fma(zkk * zkk, ip, quad);
      if (k < M / 2) prod0 = prod0 * pk; else prod1 = prod1 * pk;
    }
  }
  // a padding row (m odd: one) keeps the untouched diagonal dd0 as its pivot: take it out of the determinant
  if (!ALPHA && m < M) {
    const double id0 = rcp_pos(dd0);
    for (int r = m; r < M; r++) {
      if (r < M / 2) prod0 = prod0 * id0; else prod1 = prod1 * id0;
    }
  }
  GpOut o;
  o.amp = amp;
  o.c = c;
  o.ok = ok;
#ifdef NNGP_FIT_STATS
  o.stage = 3;
#endif
  if (!ALPHA) {
    __syncwarp();  // the next evaluation overwrites the tile
    // -(-0.5*y@alpha - sum(log(diag L)) - (N/2) log(2 pi)),  sum log L_rr = 0.5 log det K,
    // log det K = log(prod0 prod1) + m e0 ln 2,  y^T K^-1 y = 2^-e0 sum z_k^2 / d'_k
    const int h0 = __double2hiint(prod0), h1 = __double2hiint(prod1);
    const double m0 = __hiloint2double((h0 & 0x000fffff) | 0x3ff00000, __double2loint(prod0));
    const double m1 = __hiloint2double((h1 & 0x000fffff) | 0x3ff00000, __double2loint(prod1));
    const int e0 = 1023 - ((__double2hiint(sc) >> 20) & 0x7ff);  // sc = 2^-e0
    const int esum = (h0 >> 20) + (h1 >> 20) - 2046 + m * e0;
    const double res = fma(0.5, fma(quad, sc, log_pos_plus(m0 * m1, esum)), hml);
    o.val = (ok && res == res) ? res : dinf();
    return o;
  }
  // alpha = L'^-T D^-1 L'^-1 y.  Backward solve column oriented: lane k needs column k of L',
  // l'_rk = u_rk / d_k = Kt[k*LD + r] * inv_own  (r > k; the tile still holds every unscaled column)
  __syncwarp();
  const int col = (lane < M) ? lane : 0;
#pragma unroll
  for (int r = 1; r < M; r++) a[r] = Kt[col * LD + r] * inv_own;
  double alpha = 0.0, vb = w_own * inv_own;
#pragma unroll
  for (int r = M - 1; r >= 0; r--) {
    const double ar = shfl(vb, r);
    if (lane == r) alpha = ar;
    vb = fma(-a[r], ar, vb);  // meaningful for lane < r only
  }
  __syncwarp();
  o.val = alpha * sc;  // K^-1 = 2^-e0 K'^-1
  return o;
}

// ---------------------------------------------------------------------------------------
// Nelder-Mead, SciPy semantics (non-adaptive, N=2): see oracle/nelder_mead.py for the
// restatement this is tested against.  All lanes carry the same simplex.  Written as a state
// machine around ONE objective call site (every branch of an iteration only chooses the next
// point to evaluate), which keeps the code small.
// ---------------------------------------------------------------------------------------
struct NMOut {
  double x0, x1, f;
  int nfev;
  // budget > 0 and the search was still running after `budget` evaluations at the start of an iteration: the sorted
  // simplex is handed to gp_fit_spec_kernel, which continues it with the candidate points of an iteration evaluated
  // side by side on the four warps of a CTA
  bool unfinished;
  double sx[3][2], sf[3];
  int it;
};

__device__ __forceinline__ void sort3(double (&sx)[3][2], double (&sf)[3]) {
  // stable insertion sort, ascending fsim (np.argsort on 3 elements is an insertion sort)
  auto swp = [&](int a, int b) {
    double t = sf[a]; sf[a] = sf[b]; sf[b] = t;
    t = sx[a][0]; sx[a][0] = sx[b][0]; sx[b][0] = t;
    t = sx[a][1]; sx[a][1] = sx[b][1]; sx[b][1] = t;
  };
  if (sf[1] < sf[0]) swp(0, 1);
  if (sf[2] < sf[1]) {
    swp(1, 2);
    if (sf[1] < sf[0]) swp(0, 1);
  }
}

enum { PH_INIT0 = 0, PH_INIT1 = 1, PH_INIT2 = 2, PH_REFLECT, PH_EXPAND, PH_OUTC, PH_INC, PH_SHRINK1, PH_SHRINK2 };

// sim[j] = sim[0] + sigma*(sim[j] - sim[0]), sigma = 1/2
__device__ __forceinline__ double shrink_to(double x0, double xj) {
  return __dadd_rn(x0, __dmul_rn(0.5, __dsub_rn(xj, x0)));
}

// Look-ahead of a search whose sorted simplex is all +inf.  While every value stays +inf, every comparison of the state
// machine is false: an iteration evaluates the reflection, the inside contraction and the two shrunk vertices, then
// keeps the best vertex, moves the other two halfway towards it, and the sort leaves the order as it is.  So the next
// 8 iterations' 32 points are known in advance; lane l computes point l (iteration l / 4, in SciPy's order) with the
// state machine's own operations.
__device__ __forceinline__ void nm_lookahead_point(const double (&sx)[3][2], int lane, double& t0, double& t1) {
  const int k = lane >> 2, s = lane & 3;
  double a0 = sx[1][0], a1 = sx[1][1], b0 = sx[2][0], b1 = sx[2][1];
#pragma unroll
  for (int i = 0; i < 7; i++) {
    if (i < k) {
      a0 = shrink_to(sx[0][0], a0); a1 = shrink_to(sx[0][1], a1);
      b0 = shrink_to(sx[0][0], b0); b1 = shrink_to(sx[0][1], b1);
    }
  }
  const double xb0 = __dmul_rn(__dadd_rn(sx[0][0], a0), 0.5), xb1 = __dmul_rn(__dadd_rn(sx[0][1], a1), 0.5);
  if (s == 0) {  // reflection
    t0 = __dsub_rn(__dmul_rn(2.0, xb0), b0); t1 = __dsub_rn(__dmul_rn(2.0, xb1), b1);
  } else if (s == 1) {  // inside contraction
    t0 = __dadd_rn(__dmul_rn(0.5, xb0), __dmul_rn(0.5, b0)); t1 = __dadd_rn(__dmul_rn(0.5, xb1), __dmul_rn(0.5, b1));
  } else if (s == 2) {  // shrunk second vertex
    t0 = shrink_to(sx[0][0], a0); t1 = shrink_to(sx[0][1], a1);
  } else {  // shrunk worst vertex
    t0 = shrink_to(sx[0][0], b0); t1 = shrink_to(sx[0][1], b1);
  }
}

// The leading whole iterations of a window whose four points all fail the screen, skipped in one step: each ends with
// the two shrunk vertices (points 4k-2 and 4k-1 of the window) and +inf values, so after k of them the simplex is
// (sx[0], point 4k-2, point 4k-1), fcalls has grown by 4k and it by k.  k stops before maxfun / maxiter would end
// the search, so the state machine applies those ends itself.  Returns k; the caller forms the next reflection.
__device__ __forceinline__ int nm_skip_iterations(unsigned fails, double t0, double t1, double (&sx)[3][2], int& fcalls,
                                                  int& it, int maxfun, int maxiter) {
  int k = (fails == FULL) ? 8 : (__ffs(~fails) - 1) >> 2;
  k = min(k, min((maxfun - 1 - fcalls) >> 2, maxiter - 1 - it));
  if (k > 0) {
    sx[1][0] = shfl(t0, 4 * k - 2); sx[1][1] = shfl(t1, 4 * k - 2);
    sx[2][0] = shfl(t0, 4 * k - 1); sx[2][1] = shfl(t1, 4 * k - 1);
    fcalls += 4 * k;
    it += k;
  }
  return k;
}

// Does the objective at this lane's point fail at pivots 0..4?  gp_head and the leading-block check of gp_core, with
// the lane's own arguments: the ten block entries, which gp_core gathers by shuffle from lanes 0..9, are computed
// here from their squared distances (slot 0 of lanes 0..9) with the same operations, so both decide alike.
template <int M>
__device__ __noinline__ bool nm_screen_fails(double th0, double th1, double jit10, const PairSlots<M>& P, int m,
                                             double guard) {
  const GpHead hd = gp_head(th0, th1, jit10, P.r2_10, m, guard);
  double x[10], v[10];
  bool pad[10];
#pragma unroll
  for (int e = 0; e < 10; e++) {
    x[e] = hd.c * shfl(P.r2[0], e);
    pad[e] = __shfl_sync(FULL, (int)P.pad[0], e) != 0;
  }
  {
    double xa[5], oa[5];
#pragma unroll
    for (int e = 0; e < 5; e++) xa[e] = x[e];
    exp_neg_vec<5>(xa, oa);
#pragma unroll
    for (int e = 0; e < 5; e++) v[e] = oa[e];
#pragma unroll
    for (int e = 0; e < 5; e++) xa[e] = x[5 + e];
    exp_neg_vec<5>(xa, oa);
#pragma unroll
    for (int e = 0; e < 5; e++) v[5 + e] = oa[e];
  }
  double k[10];
#pragma unroll
  for (int e = 0; e < 10; e++) k[e] = pad[e] ? 0.0 : hd.amp_s * v[e];
  double ip[4];
  const bool fail5 = block5_fails(k[0], k[1], k[3], k[6], k[2], k[4], k[5], k[7], k[8], k[9], hd.dd0, hd.pmin, ip);
  return hd.fail01 || fail5;
}

#ifdef NNGP_FIT_STATS
// statistics build only (scripts/fit_inf_share_probe.py): evaluations of nelder_mead by where they were decided,
// [0..3] in iterations that start with every vertex +inf, [4..7] in the others (and the three initial ones):
// not evaluated (look-ahead), failed at pivots 0 / 1, failed at pivots 2..4, factorised further;
// [8] / [9] warp cycles spent in the two kinds of iteration; [10] searches, [11] searches with an all-inf iteration,
// [12] their warp cycles, [13] the longest search in cycles
__device__ unsigned long long g_nm_stats[16];
#endif

template <int M>
__device__ __forceinline__ NMOut nelder_mead(double s0, double s1, double jit10, double fatol, double xatol,
                                             const PairSlots<M>& P, double y, int m, int lane,
                                             double* __restrict__ Lt, double hml, bool head_batch, double guard,
                                             int budget = 0) {
  const int maxfun = 400, maxiter = 400;  // 200 * N
  bool unfinished = false;
  double sx[3][2], sf[3];
  sx[0][0] = s0; sx[0][1] = s1;
  sx[1][0] = (s0 != 0.0) ? __dmul_rn(1.05, s0) : 0.00025; sx[1][1] = s1;
  sx[2][0] = s0; sx[2][1] = (s1 != 0.0) ? __dmul_rn(1.05, s1) : 0.00025;
  sf[0] = sf[1] = sf[2] = dinf();
  int fcalls = 0, it = 1, phase = PH_INIT0;
  double p0 = s0, p1 = s1;
  double xb0 = 0, xb1 = 0, xr0 = 0, xr1 = 0, fxr = 0;
  // When every vertex is +inf (head_batch), the next 32 points are screened at once, one per lane (nm_lookahead_point,
  // nm_screen_fails).  The leading whole iterations whose points all fail are skipped in one step (nm_skip_iterations);
  // for the other screened-out points the state machine consumes +inf without evaluating them, so the decisions and
  // the maxfun / aborted rules of a partial iteration are its own.  A point that passes the screen is evaluated; while
  // its value is +inf the rest of the window still applies, a finite one ends it.
  double la0 = 0.0, la1 = 0.0;  // this lane's point of the window
  unsigned lfail = 0;           // bit l: point l fails at pivots 0..4
  int lpos = 32;                // position of the next evaluation in the window; 32: no window
#ifdef NNGP_FIT_STATS
  unsigned long long st_n[8] = {0, 0, 0, 0, 0, 0, 0, 0}, st_cyc[2] = {0, 0};
  const long long st_begin = clock64();
  long long st_last = st_begin;
  int st_inf = 0, st_any_inf = 0;
#endif
  for (;;) {
#ifdef NNGP_FIT_STATS
    {
      const long long now = clock64();
      st_cyc[st_inf] += (unsigned long long)(now - st_last);
      st_last = now;
    }
#endif
    bool hit = false;
    if (lpos < 32) {
      if (p0 == shfl(la0, lpos) && p1 == shfl(la1, lpos)) {
        hit = (lfail >> lpos) & 1u;
        lpos++;
      } else {
        lpos = 32;
      }
    }
#ifdef NNGP_FIT_STATS
    double f = dinf();
    if (hit) {
      st_n[st_inf ? 0 : 4]++;
    } else {
      const GpOut g = gp_core<M, false>(p0, p1, jit10, P, y, m, lane, Lt, hml, guard);
      f = g.val;
      st_n[(st_inf ? 0 : 4) + g.stage]++;
    }
#else
    const double f = hit ? dinf() : gp_core<M, false>(p0, p1, jit10, P, y, m, lane, Lt, hml, guard).val;
#endif
    if (f != dinf()) lpos = 32;  // a finite value changes the trajectory
    fcalls++;
    bool aborted = false, do_shrink = false;
    if (phase == PH_INIT0) {
      sf[0] = f; phase = PH_INIT1; p0 = sx[1][0]; p1 = sx[1][1];
      continue;
    }
    if (phase == PH_INIT1) {
      sf[1] = f; phase = PH_INIT2; p0 = sx[2][0]; p1 = sx[2][1];
      continue;
    }
    const bool initial = (phase == PH_INIT2);
    if (initial) {
      sf[2] = f;
    } else if (phase == PH_REFLECT) {
      fxr = f;
      int nphase = -1;
      double q0 = 0, q1 = 0;
      const double w0 = sx[2][0], w1 = sx[2][1];
      if (fxr < sf[0]) {  // expansion: (1+rho*chi)*xbar - rho*chi*worst
        q0 = __dsub_rn(__dmul_rn(3.0, xb0), __dmul_rn(2.0, w0));
        q1 = __dsub_rn(__dmul_rn(3.0, xb1), __dmul_rn(2.0, w1));
        nphase = PH_EXPAND;
      } else if (fxr < sf[1]) {
        sx[2][0] = xr0; sx[2][1] = xr1; sf[2] = fxr;
      } else if (fxr < sf[2]) {  // outside contraction: (1+psi*rho)*xbar - psi*rho*worst
        q0 = __dsub_rn(__dmul_rn(1.5, xb0), __dmul_rn(0.5, w0));
        q1 = __dsub_rn(__dmul_rn(1.5, xb1), __dmul_rn(0.5, w1));
        nphase = PH_OUTC;
      } else {  // inside contraction: (1-psi)*xbar + psi*worst
        q0 = __dadd_rn(__dmul_rn(0.5, xb0), __dmul_rn(0.5, w0));
        q1 = __dadd_rn(__dmul_rn(0.5, xb1), __dmul_rn(0.5, w1));
        nphase = PH_INC;
      }
      if (nphase >= 0) {
        if (fcalls >= maxfun) {
          aborted = true;  // SciPy raises inside func(): the iteration's update is dropped
        } else {
          phase = nphase; p0 = q0; p1 = q1;
          continue;
        }
      }
    } else if (phase == PH_EXPAND) {
      if (f < fxr) { sx[2][0] = p0; sx[2][1] = p1; sf[2] = f; }
      else { sx[2][0] = xr0; sx[2][1] = xr1; sf[2] = fxr; }
    } else if (phase == PH_OUTC) {
      if (f <= fxr) { sx[2][0] = p0; sx[2][1] = p1; sf[2] = f; }
      else do_shrink = true;
    } else if (phase == PH_INC) {
      if (f < sf[2]) { sx[2][0] = p0; sx[2][1] = p1; sf[2] = f; }
      else do_shrink = true;
    } else if (phase == PH_SHRINK1) {
      sf[1] = f;
      sx[2][0] = shrink_to(sx[0][0], sx[2][0]);
      sx[2][1] = shrink_to(sx[0][1], sx[2][1]);
      if (fcalls >= maxfun) {
        aborted = true;  // vertex moved, value kept
      } else {
        phase = PH_SHRINK2; p0 = sx[2][0]; p1 = sx[2][1];
        continue;
      }
    } else {  // PH_SHRINK2
      sf[2] = f;
    }
    if (do_shrink) {
      sx[1][0] = shrink_to(sx[0][0], sx[1][0]);
      sx[1][1] = shrink_to(sx[0][1], sx[1][1]);
      if (fcalls >= maxfun) {
        aborted = true;
      } else {
        phase = PH_SHRINK1; p0 = sx[1][0]; p1 = sx[1][1];
        continue;
      }
    }
    // end of an iteration (or of the three initial evaluations)
    if (!initial && !aborted) it++;
    sort3(sx, sf);
    if (!(fcalls < maxfun && it < maxiter)) break;
    {
      const double d10 = fabs(__dsub_rn(sx[1][0], sx[0][0])), d11 = fabs(__dsub_rn(sx[1][1], sx[0][1]));
      const double d20 = fabs(__dsub_rn(sx[2][0], sx[0][0])), d21 = fabs(__dsub_rn(sx[2][1], sx[0][1]));
      const double f1 = fabs(__dsub_rn(sf[0], sf[1])), f2 = fabs(__dsub_rn(sf[0], sf[2]));
      // np.max(...) <= tol is false as soon as any term is NaN
      if (d10 <= xatol && d11 <= xatol && d20 <= xatol && d21 <= xatol && f1 <= fatol && f2 <= fatol)
        break;
    }
    xb0 = __dmul_rn(__dadd_rn(sx[0][0], sx[1][0]), 0.5);
    xb1 = __dmul_rn(__dadd_rn(sx[0][1], sx[1][1]), 0.5);
    xr0 = __dsub_rn(__dmul_rn(2.0, xb0), sx[2][0]);
    xr1 = __dsub_rn(__dmul_rn(2.0, xb1), sx[2][1]);
    phase = PH_REFLECT; p0 = xr0; p1 = xr1;
#ifdef NNGP_FIT_STATS
    st_inf = (sf[0] == dinf()) ? 1 : 0;
    st_any_inf |= st_inf;
#endif
    // iteration boundary: sorted simplex, nothing pending.  Searches whose vertices are all +inf stay here: their
    // iterations are screened 32 points at a time (below), cheaper than a CTA round of the continuation kernel
    if (budget > 0 && fcalls >= budget && sf[0] != dinf()) {
      unfinished = true;
      break;
    }
    // sorted: the best vertex is +inf, so all are.  An unfinished window still holds this iteration's points.
    if (head_batch && sf[0] == dinf() && lpos >= 32) {
      nm_lookahead_point(sx, lane, la0, la1);
      lfail = __ballot_sync(FULL, nm_screen_fails<M>(la0, la1, jit10, P, m, guard));
      const int k = nm_skip_iterations(lfail, la0, la1, sx, fcalls, it, maxfun, maxiter);
      if (k > 0) {
        xb0 = __dmul_rn(__dadd_rn(sx[0][0], sx[1][0]), 0.5);
        xb1 = __dmul_rn(__dadd_rn(sx[0][1], sx[1][1]), 0.5);
        xr0 = __dsub_rn(__dmul_rn(2.0, xb0), sx[2][0]);
        xr1 = __dsub_rn(__dmul_rn(2.0, xb1), sx[2][1]);
        p0 = xr0; p1 = xr1;
#ifdef NNGP_FIT_STATS
        st_n[0] += 4 * k;
#endif
      }
      lpos = 4 * k;
    }
  }
#ifdef NNGP_FIT_STATS
  {
    const long long now = clock64();
    st_cyc[st_inf] += (unsigned long long)(now - st_last);
    if (lane == 0) {
      for (int i = 0; i < 8; i++) atomicAdd(g_nm_stats + i, st_n[i]);
      atomicAdd(g_nm_stats + 8, st_cyc[1]);
      atomicAdd(g_nm_stats + 9, st_cyc[0]);
      atomicAdd(g_nm_stats + 10, 1ULL);
      atomicAdd(g_nm_stats + 11, (unsigned long long)st_any_inf);
      if (st_any_inf) atomicAdd(g_nm_stats + 12, (unsigned long long)(now - st_begin));
      atomicMax(g_nm_stats + 13, (unsigned long long)(now - st_begin));
    }
  }
#endif
  NMOut o;
  o.x0 = sx[0][0];
  o.x1 = sx[0][1];
  o.f = fmin(fmin(sf[0], sf[1]), sf[2]);
  o.nfev = fcalls;
  o.unfinished = unfinished;
  o.it = it;
#pragma unroll
  for (int v = 0; v < 3; v++) {
    o.sx[v][0] = sx[v][0];
    o.sx[v][1] = sx[v][1];
    o.sf[v] = sf[v];
  }
  return o;
}

// ---------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------
struct FitArgs {
  const long long* idx;   // [nq,m]
  const double* dist;     // [nq,m]
  const double* r2;       // [nq,m,m]
  const double* Y;        // dataset targets [rows,d]
  const signed char* starts;  // [nq,d,9,R,2]
  const double* add;      // optional [nq,d] added to the prediction (sweep: uG_next)
  double* pred;           // [nq,d]
  double* theta_opt;      // [nq,d,2]
  double* jitter_opt;     // [nq,d]
  double* fval_opt;       // [nq,d]
  int* nfev;              // [nq,d,9,R]
  double* fvals;          // [nq,d,9,R]
  double* thetas;         // [nq,d,9,R,2]
  unsigned long long* counters;  // [0] NM runs, [1] nll evaluations
  double* res;            // workspace [ntasks,3]: fval, theta0, theta1 of every search
  unsigned int* done;     // workspace [nq*d]: searches finished per (query, dim); zero on entry and exit
  unsigned int* queue;    // next task to hand out; zero on entry
  const int* order;       // optional [ntasks]: queue position -> task (longest searches first)
  int d, m, R, ntasks;
  int head_batch;         // 1: screen the points of all-inf Nelder-Mead iterations ahead, in lanes (0: one by one, tests)
  int j0, dl;             // output dimensions [j0, j0+dl) handled by this launch (a rank's share; dl = d: all)
  long long ld_pred;      // row stride of pred / add
  double fatol, xatol;
  double guard;           // failed-pivot threshold relative to the diagonal (ulps * 2^-52)
  // long searches: after `budget` evaluations a search parks its simplex in saves[task] (12 doubles) and its id in
  // cont_list[atomicAdd(cont_count)]; gp_fit_spec_kernel continues them (queue2 hands them out)
  int budget;
  double* saves;
  int* cont_list;
  unsigned int* cont_count;
  unsigned int* queue2;
  int quad_all;           // 1: gp_fit_spec_kernel runs whole searches, four warps each (no first kernel)
};

template <int M>
__device__ __noinline__ double posterior_mean(double th0, double th1, double jit10, const PairSlots<M>& P,
                                              double y, double kq, int m, int lane, double* Lt, double guard) {
  const GpOut g = gp_core<M, true>(th0, th1, jit10, P, y, m, lane, Lt, 0.0, guard);
  if (!g.ok) return dnan();
  // K_star = kernel(x, new_x); post_mean = K_star.T @ alph  (models.py:165-167)
  const double ks = g.amp * exp_neg(g.c * kq);
  return warp_sum((lane < m) ? ks * g.val : 0.0);
}

#include "gpfit_group.cuh"
#include "gpfit_big.cuh"

// results of a finished search; the warp that completes the last search of its (query, dimension) applies the selection
// rule (models.py:212-215) and computes the posterior mean (models.py:162-168)
template <int M>
__device__ __forceinline__ void finish_search(const FitArgs& A, int task, double x0, double x1, double f, int nfev,
                                              const PairSlots<M>& P, double y, int lane, double* Lt) {
  const int m = A.m, d = A.d, R = A.R, nruns = NNGP_N_JITTER * R;
  const int qj = task / nruns, run = task - qj * nruns;
  const int q = qj / A.dl, j = A.j0 + (qj - q * A.dl);
  const long long gqj = (long long)q * d + j, gtask = gqj * nruns + run;
  unsigned int prior = 0;
  if (lane == 0) {
    A.res[(long long)task * 3] = f;
    A.res[(long long)task * 3 + 1] = x0;
    A.res[(long long)task * 3 + 2] = x1;
    atomicAdd(A.counters, 1ULL);
    atomicAdd(A.counters + 1, (unsigned long long)nfev);
    if (A.nfev) A.nfev[gtask] = nfev;
    if (A.fvals) A.fvals[gtask] = f;
    if (A.thetas) {
      A.thetas[gtask * 2] = x0;
      A.thetas[gtask * 2 + 1] = x1;
    }
    __threadfence();
    prior = atomicAdd(A.done + qj, 1u);
  }
  prior = __shfl_sync(FULL, prior, 0);
  if (prior != (unsigned)(nruns - 1)) return;
  // this warp finished the last search of (q, j): selection + posterior mean
  __threadfence();
  const volatile double* rf = A.res + (long long)qj * nruns * 3;
  double fmin_all = rf[0];
  for (int r = 1; r < nruns; r++) {
    const double v = rf[3 * r];
    fmin_all = (v < fmin_all) ? v : fmin_all;
  }
  const double thr = fmin_all * 0.9;
  bool any = false;
  for (int r = 0; r < nruns; r++) any |= (rf[3 * r] < thr);
  int best = -1;
  double fb = 0.0;
  for (int r = 0; r < nruns; r++) {
    const double v = rf[3 * r];
    if (any && !(v < thr)) continue;
    if (best < 0 || v < fb) {
      best = r;
      fb = v;
    }
  }
  const int ab = best / R;
  const double th0 = rf[3 * best + 1], th1 = rf[3 * best + 2];
  const double kq = (lane < m) ? A.dist[(long long)q * m + lane] : 0.0;
  double mean = posterior_mean<M>(th0, th1, c_jit10[ab], P, y, kq, m, lane, Lt, A.guard);
  __syncwarp();
  if (lane == 0) {
    A.done[qj] = 0;  // leave the counters clean for the next launch
    const long long op = (long long)q * A.ld_pred + j;
    if (A.add) mean = mean + A.add[op];
    A.pred[op] = mean;
    if (A.theta_opt) {
      A.theta_opt[gqj * 2] = th0;
      A.theta_opt[gqj * 2 + 1] = th1;
    }
    if (A.jitter_opt) A.jitter_opt[gqj] = (double)(ab - 20);
    if (A.fval_opt) A.fval_opt[gqj] = fb;
  }
}

// registers per thread: 4-warp CTAs, fit_occ(m) CTAs per SM
static constexpr int fit_occ(int m) { return (m <= 12) ? 4 : ((m <= 20) ? 3 : 2); }

template <int M>
__global__ void __launch_bounds__(GP_WARPS * 32, fit_occ(M))
gp_fit_predict_kernel(FitArgs A) {
  extern __shared__ double sm[];
  const int m = A.m, d = A.d, R = A.R, nruns = NNGP_N_JITTER * R;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double* Lt = sm + w * (M * (M + 2));
  const double hml = (m / 2.0) * 1.8378770664093453;  // (N/2)*np.log(2*np.pi)
  PairSlots<M> P;
  pair_slots_init<M>(P, lane, m);
  int q_loaded = -1;
  for (;;) {
    int task = 0;
    if (lane == 0) {
      const unsigned pos = atomicAdd(A.queue, 1u);
      task = (pos < (unsigned)A.ntasks) ? (A.order ? A.order[pos] : (int)pos) : A.ntasks;
    }
    task = __shfl_sync(FULL, task, 0);
    if (task >= A.ntasks) break;
    // task and qj number the searches / (query, dim) pairs of THIS launch; gtask, gqj are their positions
    // in the full [nq, d, 9, R] arrays (identical when the launch covers every dimension)
    const int qj = task / nruns, run = task - qj * nruns;
    const int q = qj / A.dl, j = A.j0 + (qj - q * A.dl);
    const long long gqj = (long long)q * d + j, gtask = gqj * nruns + run;
    const int a = run / R;
    const double* r2 = A.r2 + (long long)q * m * m;
    if (q != q_loaded) {
      pair_slots_load<M>(P, r2, m);
      q_loaded = q;
    }
    const double y = (lane < m) ? A.Y[A.idx[(long long)q * m + lane] * d + j] : 0.0;
    const signed char* st = A.starts + gtask * 2;
    const NMOut o = nelder_mead<M>((double)st[0], (double)st[1], c_jit10[a], A.fatol, A.xatol, P, y, m,
                                   lane, Lt, hml, A.head_batch != 0, A.guard, A.budget);
    if (o.unfinished) {
      if (lane == 0) {
        double* sv = A.saves + (long long)task * 12;
#pragma unroll
        for (int v = 0; v < 3; v++) {
          sv[2 * v] = o.sx[v][0];
          sv[2 * v + 1] = o.sx[v][1];
          sv[6 + v] = o.sf[v];
        }
        sv[9] = (double)o.it;
        sv[10] = (double)o.nfev;
        A.cont_list[atomicAdd(A.cont_count, 1u)] = task;
      }
      continue;
    }
    finish_search<M>(A, task, o.x0, o.x1, o.f, o.nfev, P, y, lane, Lt);
  }
}

// ---------------------------------------------------------------------------------------
// Continuation of the long searches.  A launch lasts as long as its longest serial chain of objective evaluations
// (at the FHN target: a handful of searches with 200-300 evaluations of ~3 300 cycles each, and -- when the fits of a
// predict are sharded over 8 GPUs -- nothing else to hide them behind).  gp_fit_predict_kernel parks every search
// that is still running after `budget` evaluations; here ONE CTA continues one search and its four warps evaluate,
// side by side, the points the iteration can ask for: reflection, expansion, outside and inside contraction (all
// vertices +inf: reflection, inside contraction and the two shrunk vertices).  The Nelder-Mead state machine
// (nm_step) then consumes the values in SciPy's order, so decisions, evaluation counts and results are bit-identical
// to the sequential search; an iteration costs one evaluation latency instead of two (four when it shrinks).
// ---------------------------------------------------------------------------------------
template <int M>
__global__ void __launch_bounds__(GP_WARPS * 32, fit_occ(M))
gp_fit_spec_kernel(FitArgs A) {
  static_assert(GP_WARPS == 4, "four candidate points per iteration");
  extern __shared__ double sm[];
  __shared__ double s_f[GP_WARPS];
  __shared__ int s_task;
  const int m = A.m, d = A.d, R = A.R, nruns = NNGP_N_JITTER * R;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double* Lt = sm + w * (M * (M + 2));
  const double hml = (m / 2.0) * 1.8378770664093453;
  const bool scratch = A.quad_all != 0;  // whole searches (queue / order / starts) instead of parked ones
  PairSlots<M> P;
  pair_slots_init<M>(P, lane, m);
  int q_loaded = -1;
  for (;;) {
    if (threadIdx.x == 0) {
      if (scratch) {
        const unsigned pos = atomicAdd(A.queue, 1u);
        s_task = (pos < (unsigned)A.ntasks) ? (A.order ? A.order[pos] : (int)pos) : -1;
      } else {
        const unsigned pos = atomicAdd(A.queue2, 1u);
        s_task = (pos < *A.cont_count) ? A.cont_list[pos] : -1;
      }
    }
    __syncthreads();
    const int task = s_task;
    __syncthreads();
    if (task < 0) break;
    const int qj = task / nruns, run = task - qj * nruns;
    const int q = qj / A.dl, j = A.j0 + (qj - q * A.dl);
    const double jit10 = c_jit10[run / R];
    if (q != q_loaded) {
      pair_slots_load<M>(P, A.r2 + (long long)q * m * m, m);
      q_loaded = q;
    }
    const double y = (lane < m) ? A.Y[A.idx[(long long)q * m + lane] * d + j] : 0.0;
    NMState S;
    if (scratch) {
      const signed char* st = A.starts + (((long long)q * d + j) * nruns + run) * 2;
      nm_init(S, (double)st[0], (double)st[1]);
    } else {
      nm_init(S, -1.0, -1.0);
      const double* sv = A.saves + (long long)task * 12;
#pragma unroll
      for (int v = 0; v < 3; v++) {
        S.sx[v][0] = sv[2 * v];
        S.sx[v][1] = sv[2 * v + 1];
        S.sf[v] = sv[6 + v];
      }
      S.it = (int)sv[9];
      S.fcalls = (int)sv[10];
      // the start of an iteration, as nelder_mead / nm_step leave it
      S.xb0 = __dmul_rn(__dadd_rn(S.sx[0][0], S.sx[1][0]), 0.5);
      S.xb1 = __dmul_rn(__dadd_rn(S.sx[0][1], S.sx[1][1]), 0.5);
      S.xr0 = __dsub_rn(__dmul_rn(2.0, S.xb0), S.sx[2][0]);
      S.xr1 = __dsub_rn(__dmul_rn(2.0, S.xb1), S.sx[2][1]);
      S.phase = PH_REFLECT;
      S.p0 = S.xr0;
      S.p1 = S.xr1;
    }
    bool fin = false;
    // The previous iteration contracted inside or shrank: the searches that last (a collapsing simplex in the
    // rounding noise of a singular kernel matrix) do so in long runs, and such an iteration asks for the
    // reflection, the inside contraction and the two shrunk vertices -- all four known when it starts.
    bool shrinking = false;
    auto eval_round = [&](const double (&c0)[4], const double (&c1)[4], int navail, double (&fc)[4]) {
      const double t0 = (w == 0) ? c0[0] : (w == 1) ? c0[1] : (w == 2) ? c0[2] : c0[3];
      const double t1 = (w == 0) ? c1[0] : (w == 1) ? c1[1] : (w == 2) ? c1[2] : c1[3];
      if (w < navail) {
        const double f = gp_core<M, false>(t0, t1, jit10, P, y, m, lane, Lt, hml, A.guard).val;
        if (lane == 0) s_f[w] = f;
      }
      __syncthreads();
#pragma unroll
      for (int v = 0; v < 4; v++) fc[v] = s_f[v];
      __syncthreads();
    };
    while (!fin) {
      double c0[4], c1[4], fc[4];
      int navail = 4;
      const double w0 = S.sx[2][0], w1 = S.sx[2][1];
      const double s10 = shrink_to(S.sx[0][0], S.sx[1][0]), s11 = shrink_to(S.sx[0][1], S.sx[1][1]);
      const double s20 = shrink_to(S.sx[0][0], w0), s21 = shrink_to(S.sx[0][1], w1);
      if (S.phase == PH_INIT0) {  // the three vertices of the initial simplex
        c0[0] = S.sx[0][0]; c1[0] = S.sx[0][1];
        c0[1] = S.sx[1][0]; c1[1] = S.sx[1][1];
        c0[2] = S.sx[2][0]; c1[2] = S.sx[2][1];
        c0[3] = c0[0]; c1[3] = c1[0];
        navail = 3;
      } else {
        c0[0] = S.xr0; c1[0] = S.xr1;
        // inside contraction (1-psi)*xbar + psi*worst
        const double i0 = __dadd_rn(__dmul_rn(0.5, S.xb0), __dmul_rn(0.5, w0)), i1 = __dadd_rn(__dmul_rn(0.5, S.xb1), __dmul_rn(0.5, w1));
        if (S.sf[0] == dinf() || shrinking) {  // reflection, inside contraction, the two shrunk vertices
          c0[1] = i0; c1[1] = i1;
          c0[2] = s10; c1[2] = s11;
          c0[3] = s20; c1[3] = s21;
        } else {                  // reflection, expansion, outside contraction, inside contraction
          c0[1] = __dsub_rn(__dmul_rn(3.0, S.xb0), __dmul_rn(2.0, w0)); c1[1] = __dsub_rn(__dmul_rn(3.0, S.xb1), __dmul_rn(2.0, w1));
          c0[2] = __dsub_rn(__dmul_rn(1.5, S.xb0), __dmul_rn(0.5, w0)); c1[2] = __dsub_rn(__dmul_rn(1.5, S.xb1), __dmul_rn(0.5, w1));
          c0[3] = i0; c1[3] = i1;
        }
      }
      shrinking = false;
      eval_round(c0, c1, navail, fc);
      for (;;) {  // consume in the order the state machine asks (uniform over the CTA: every warp holds the same state)
        int hit = -1;
#pragma unroll
        for (int v = 3; v >= 0; v--)
          if (v < navail && S.p0 == c0[v] && S.p1 == c1[v]) hit = v;
        if (hit < 0) {
          // not among the evaluated points: evaluate it now, together with the points that can follow it in this
          // iteration (the shrunk vertices after a contraction; s10/s20 still describe them: the simplex only
          // changes when the iteration ends)
          c0[0] = S.p0; c1[0] = S.p1;
          navail = 1;
          if (S.phase == PH_SHRINK1) {
            c0[1] = s20; c1[1] = s21;
            navail = 2;
          } else if (S.phase == PH_OUTC) {
            c0[1] = s10; c1[1] = s11;
            c0[2] = s20; c1[2] = s21;
            navail = 3;
          }
          for (int v = navail; v < 4; v++) { c0[v] = c0[0]; c1[v] = c1[0]; }
          eval_round(c0, c1, navail, fc);
          continue;
        }
        if (S.phase == PH_INC || S.phase == PH_SHRINK1 || S.phase == PH_SHRINK2) shrinking = true;
        fin = nm_step(S, fc[hit], A.fatol, A.xatol, false);
        if (fin || S.phase == PH_REFLECT) break;  // search over, or the next iteration starts
      }
    }
    if (w == 0)
      finish_search<M>(A, task, S.sx[0][0], S.sx[0][1], fmin(fmin(S.sf[0], S.sf[1]), S.sf[2]), S.fcalls, P, y, lane, Lt);
    __syncthreads();
  }
}

// objective at given hyper-parameters: one warp per (q, j), loops over t
template <int M>
__global__ void __launch_bounds__(GP_WARPS * 32)
gp_nll_kernel(const long long* idx, const double* r2all, const double* Y, int d, int m, int nq, int nt,
              const double* theta, const double* jitter10, double* out, double guard) {
  extern __shared__ double sm[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double* Lt = sm + w * (M * (M + 2));
  const int qj = blockIdx.x * GP_WARPS + w;
  if (qj >= nq * d) return;
  const int q = qj / d, j = qj - q * d;
  const double* r2 = r2all + (long long)q * m * m;
  const double y = (lane < m) ? Y[idx[(long long)q * m + lane] * d + j] : 0.0;
  const double hml = (m / 2.0) * 1.8378770664093453;
  const long long base = (long long)qj * nt;
  PairSlots<M> P;
  pair_slots_init<M>(P, lane, m);
  pair_slots_load<M>(P, r2, m);
  for (int t = 0; t < nt; t++) {
    const double v = gp_core<M, false>(theta[(base + t) * 2], theta[(base + t) * 2 + 1], jitter10[base + t], P, y,
                                       m, lane, Lt, hml, guard).val;
    if (lane == 0) out[base + t] = v;
  }
}

// posterior mean at given hyper-parameters: one warp per (q, j)
template <int M>
__global__ void __launch_bounds__(GP_WARPS * 32)
gp_mean_kernel(const long long* idx, const double* dist, const double* r2all, const double* Y, int d,
               int m, int nq, const double* theta, const double* jitter, double* pred, double guard) {
  extern __shared__ double sm[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double* Lt = sm + w * (M * (M + 2));
  const int qj = blockIdx.x * GP_WARPS + w;
  if (qj >= nq * d) return;
  const int q = qj / d, j = qj - q * d;
  const double* r2 = r2all + (long long)q * m * m;
  const double y = (lane < m) ? Y[idx[(long long)q * m + lane] * d + j] : 0.0;
  const double kq = (lane < m) ? dist[(long long)q * m + lane] : 0.0;
  const double jit10 = exp10(jitter[qj]);
  PairSlots<M> P;
  pair_slots_init<M>(P, lane, m);
  pair_slots_load<M>(P, r2, m);
  const double mean = posterior_mean<M>(theta[(long long)qj * 2], theta[(long long)qj * 2 + 1], jit10, P, y, kq,
                                        m, lane, Lt, guard);
  if (lane == 0) pred[qj] = mean;
}

// pairwise squared distances of the m neighbours of each query: r2[q,a,b] = ||x_a - x_b||^2,
// summed strictly left to right (cdist arithmetic; this file allows FMA, so use intrinsics).
__global__ void __launch_bounds__(256)
gp_prep_kernel(const long long* __restrict__ idx, const double* __restrict__ X, int d, int m,
               double* __restrict__ r2) {
  constexpr int JC = 64;
  __shared__ double tile[NNGP_MAX_NEIGHBOURS][JC + 1];
  const int q = blockIdx.x;
  const int npairs = m * (m + 1) / 2;
  // up to 3 pairs per thread (m=32 -> 528 pairs on 256 threads)
  int pa[3], pb[3];
  double acc[3] = {0.0, 0.0, 0.0};
#pragma unroll
  for (int u = 0; u < 3; u++) {
    const int pidx = threadIdx.x + u * 256;
    int a = 0, b = 0;
    if (pidx < npairs) {
      a = (int)((sqrt(8.0 * pidx + 1.0) - 1.0) * 0.5);
      while ((a + 1) * (a + 2) / 2 <= pidx) a++;
      while (a * (a + 1) / 2 > pidx) a--;
      b = pidx - a * (a + 1) / 2;
    }
    pa[u] = a;
    pb[u] = b;
  }
  for (int j0 = 0; j0 < d; j0 += JC) {
    const int jn = min(JC, d - j0);
    __syncthreads();
    for (int e = threadIdx.x; e < m * JC; e += 256) {
      const int r = e / JC, jj = e - r * JC;
      if (jj < jn) tile[r][jj] = X[idx[(long long)q * m + r] * d + j0 + jj];
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 3; u++) {
      if (threadIdx.x + u * 256 < npairs) {
        double s = acc[u];
        for (int jj = 0; jj < jn; jj++) {
          const double diff = __dsub_rn(tile[pa[u]][jj], tile[pb[u]][jj]);
          s = __dadd_rn(s, __dmul_rn(diff, diff));
        }
        acc[u] = s;
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 3; u++) {
    if (threadIdx.x + u * 256 < npairs) {
      r2[((long long)q * m + pa[u]) * m + pb[u]] = acc[u];
      r2[((long long)q * m + pb[u]) * m + pa[u]] = acc[u];
    }
  }
}

// The GP inputs of host-chosen neighbour lists (position-based rules, models_alt.py), one CTA per ListedQuery:
// distances to the query and the neighbour matrix, both summed strictly left to right without FMA, so dist has the
// bits of NumPy's `dist + diff * diff` and r2 those of gp_prep_kernel / gp_prep_big_kernel on the same list.  m <= 32
// stages the listed rows and the query through shared memory in column chunks (gp_prep_kernel's pair mapping);
// larger m reads them from global memory, one thread per distance or pair (gp_prep_big_kernel's).
__global__ void __launch_bounds__(256)
listed_prep_kernel(const ListedQuery* __restrict__ lq, const double* __restrict__ X, int d) {
  constexpr int JC = 64;
  __shared__ double tile[NNGP_MAX_NEIGHBOURS][JC + 1];
  __shared__ double qt[JC];
  const ListedQuery L = lq[blockIdx.x];
  const int m = L.m, ld = L.ld, npairs = m * (m + 1) / 2;
  if (m == 0) {
    for (int j = threadIdx.x; j < d; j += 256) L.q_copy[j] = L.q[j];
    return;
  }
  if (L.idx)
    for (int a = threadIdx.x; a < m; a += 256) L.idx[a] = L.rows[a];
  auto pair_of = [](int pidx, int& a, int& b) {
    a = (int)((sqrt(8.0 * pidx + 1.0) - 1.0) * 0.5);
    while ((a + 1) * (a + 2) / 2 <= pidx) a++;
    while (a * (a + 1) / 2 > pidx) a--;
    b = pidx - a * (a + 1) / 2;
  };
  if (m > NNGP_MAX_NEIGHBOURS) {
    for (int a = threadIdx.x; a < m; a += 256) {
      const double* xa = X + L.rows[a] * d;
      double s = 0.0;
      for (int j = 0; j < d; j++) {
        const double diff = __dsub_rn(xa[j], L.q[j]);
        s = __dadd_rn(s, __dmul_rn(diff, diff));
      }
      L.dist[a] = s;
    }
    for (int pidx = threadIdx.x; pidx < npairs; pidx += 256) {
      int a, b;
      pair_of(pidx, a, b);
      const double* xa = X + L.rows[a] * d;
      const double* xb = X + L.rows[b] * d;
      double s = 0.0;
      for (int j = 0; j < d; j++) {
        const double diff = __dsub_rn(xa[j], xb[j]);
        s = __dadd_rn(s, __dmul_rn(diff, diff));
      }
      L.r2[(long long)a * ld + b] = s;
      L.r2[(long long)b * ld + a] = s;
    }
    return;
  }
  int pa[3], pb[3];
  double acc[3] = {0.0, 0.0, 0.0}, dq = 0.0;
#pragma unroll
  for (int u = 0; u < 3; u++) {
    pa[u] = pb[u] = 0;
    if (threadIdx.x + u * 256 < npairs) pair_of(threadIdx.x + u * 256, pa[u], pb[u]);
  }
  for (int j0 = 0; j0 < d; j0 += JC) {
    const int jn = min(JC, d - j0);
    __syncthreads();
    for (int e = threadIdx.x; e < m * JC; e += 256) {
      const int r = e / JC, jj = e - r * JC;
      if (jj < jn) tile[r][jj] = X[L.rows[r] * d + j0 + jj];
    }
    if (threadIdx.x < jn) qt[threadIdx.x] = L.q[j0 + threadIdx.x];
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 3; u++) {
      if (threadIdx.x + u * 256 < npairs) {
        double s = acc[u];
        for (int jj = 0; jj < jn; jj++) {
          const double diff = __dsub_rn(tile[pa[u]][jj], tile[pb[u]][jj]);
          s = __dadd_rn(s, __dmul_rn(diff, diff));
        }
        acc[u] = s;
      }
    }
    if (threadIdx.x < m) {
      for (int jj = 0; jj < jn; jj++) {
        const double diff = __dsub_rn(tile[threadIdx.x][jj], qt[jj]);
        dq = __dadd_rn(dq, __dmul_rn(diff, diff));
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 3; u++) {
    if (threadIdx.x + u * 256 < npairs) {
      L.r2[(long long)pa[u] * ld + pb[u]] = acc[u];
      L.r2[(long long)pb[u] * ld + pa[u]] = acc[u];
    }
  }
  if (threadIdx.x < m) L.dist[threadIdx.x] = dq;
}

// Queue order of the searches (longest first).  A search that starts at a large log-amplitude
// sigma_y runs to the evaluation limit far more often than one that starts at a small one (measured
// on the FHN target: >= 400 evaluations for about half of the starts with sigma_y = -1, never for
// sigma_y <= -5), and the launch ends with its longest search, so the queue hands out the searches
// by descending second start coordinate.  Any order gives the same results; this one shortens the tail.
// One CTA per segment of seg_len consecutive tasks: counting sort with 8 buckets in shared memory.
__global__ void __launch_bounds__(256)
gp_order_kernel(const signed char* __restrict__ starts, int seg_len, int global_ids, int* __restrict__ order) {
  __shared__ int cnt[8], cur[8];
  const long long base = (long long)blockIdx.x * seg_len;
  if (threadIdx.x < 8) cnt[threadIdx.x] = 0;
  __syncthreads();
  for (int t = threadIdx.x; t < seg_len; t += blockDim.x) {
    const int s1 = starts[(base + t) * 2 + 1];
    atomicAdd(&cnt[min(7, max(0, -1 - s1))], 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int run = 0;
    for (int b = 0; b < 8; b++) {
      cur[b] = run;
      run += cnt[b];
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < seg_len; t += blockDim.x) {
    const int s1 = starts[(base + t) * 2 + 1];
    const int pos = atomicAdd(&cur[min(7, max(0, -1 - s1))], 1);
    order[base + pos] = global_ids ? (int)(base + t) : t;
  }
}

int gp_order_launch(nngp_handle_t h, const signed char* d_starts, int nseg, int seg_len, int global_ids,
                    int* d_order, cudaStream_t st) {
  if (nseg <= 0 || seg_len <= 0) return 0;
  ProfScope prof(h, 4, st);
  gp_order_kernel<<<nseg, 256, 0, st>>>(d_starts, seg_len, global_ids, d_order);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
static inline size_t pad256(size_t b) { return ((b + 255) / 256) * 256; }

// workspace of a fit: [r2 nq*m*m | res ntasks*3 | done nq*d]
size_t gp_prep_bytes(int nq, int m) { return sizeof(double) * (size_t)nq * m * m; }
size_t gp_fit_ws_bytes(int nq, int d, int m, int R) {
  const size_t nt = (size_t)nq * d * NNGP_N_JITTER * R;
  return pad256(gp_prep_bytes(nq, m)) + pad256(sizeof(double) * 3 * nt) + pad256(sizeof(unsigned int) * (size_t)nq * d) +
         pad256(sizeof(double) * 12 * nt) + pad256(sizeof(int) * nt);  // + parked simplices and ids of the long searches
}
size_t gp_fit_done_offset(int nq, int d, int m, int R) {
  return pad256(gp_prep_bytes(nq, m)) + pad256(sizeof(double) * 3 * (size_t)nq * d * NNGP_N_JITTER * R);
}

int gp_prep_launch(nngp_handle_t h, const long long* d_idx, int nq, int m, double* d_r2,
                   cudaStream_t st) {
  if (nq <= 0) return 0;
  ProfScope prof(h, 2, st);
  if (m > NNGP_MAX_NEIGHBOURS) {
    const long long total = (long long)nq * (m * (m + 1) / 2);
    gp_prep_big_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_idx, h->ds_x, h->ds_d, m, nq, d_r2);
    h->launches++;
    NNGP_CUDA(h, cudaGetLastError());
    return 0;
  }
  gp_prep_kernel<<<nq, 256, 0, st>>>(d_idx, h->ds_x, h->ds_d, m, d_r2);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

int listed_prep_launch(nngp_handle_t h, const ListedQuery* d_lq, int n, cudaStream_t st) {
  if (n <= 0) return 0;
  ProfScope prof(h, 2, st);
  listed_prep_kernel<<<n, 256, 0, st>>>(d_lq, h->ds_x, h->ds_d);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

template <int M>
static size_t warp_tile_bytes() { return sizeof(double) * (size_t)GP_WARPS * M * (M + 2); }

template <int M>
static int fit_launch_m(nngp_handle_t h, const FitArgs& A, cudaStream_t st) {
  int& ctas_per_sm = h->occ_fit[M / 2];
  const size_t smem = warp_tile_bytes<M>();
  if (ctas_per_sm == 0) {
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_fit_predict_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NNGP_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, gp_fit_predict_kernel<M>,
                                                               GP_WARPS * 32, smem));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
  }
  const int sms = h->sm_count;
  // persistent grid: every resident warp slot pulls searches from the queue
  long long blocks = (long long)sms * ctas_per_sm;
  const long long need = (A.ntasks + GP_WARPS - 1) / GP_WARPS;
  if (blocks > need) blocks = need;
  ProfScope prof(h, 3, st);
  if (A.quad_all) {
    bool& set2 = h->attr_spec[M / 2];
    if (!set2) {
      NNGP_CUDA(h, cudaFuncSetAttribute(gp_fit_spec_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      set2 = true;
    }
    long long blocks2 = (long long)sms * ctas_per_sm;
    if (blocks2 > A.ntasks) blocks2 = A.ntasks;
    gp_fit_spec_kernel<M><<<(unsigned)blocks2, GP_WARPS * 32, smem, st>>>(A);
    h->launches++;
    NNGP_CUDA(h, cudaGetLastError());
    return 0;
  }
  gp_fit_predict_kernel<M><<<(unsigned)blocks, GP_WARPS * 32, smem, st>>>(A);
  h->launches++;
  if (A.budget > 0) {
    bool& set2 = h->attr_spec[M / 2];
    if (!set2) {
      NNGP_CUDA(h, cudaFuncSetAttribute(gp_fit_spec_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      set2 = true;
    }
    long long blocks2 = (long long)sms * ctas_per_sm;
    if (blocks2 > A.ntasks) blocks2 = A.ntasks;
    gp_fit_spec_kernel<M><<<(unsigned)blocks2, GP_WARPS * 32, smem, st>>>(A);
    h->launches++;
  }
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// grouped searches (gpfit_group.cuh) + selection / mean kernel
template <int M>
static int fit_grouped_launch_m(nngp_handle_t h, const FitArgs& A, int nqj, cudaStream_t st) {
  const size_t smem = sizeof(double) * (size_t)GP_WARPS * Grp<M>::PER_WARP;
  const size_t smem2 = warp_tile_bytes<M>();
  int& occ = h->occ_fit_grouped[M / 2];
  if (occ == 0) {
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_fit_grouped_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_select_mean_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    NNGP_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gp_fit_grouped_kernel<M>, GP_WARPS * 32, smem));
    if (occ < 1) occ = 1;
  }
  long long blocks = (long long)h->sm_count * occ;
  const long long per_cta = GP_WARPS * Grp<M>::NG;
  const long long need = (A.ntasks + per_cta - 1) / per_cta;
  if (blocks > need) blocks = need;
  ProfScope prof(h, 3, st);
  gp_fit_grouped_kernel<M><<<(unsigned)blocks, GP_WARPS * 32, smem, st>>>(A);
  gp_select_mean_kernel<M><<<(nqj + GP_WARPS - 1) / GP_WARPS, GP_WARPS * 32, smem2, st>>>(A, nqj);
  h->launches += 2;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// 32 < m <= NNGP_MAX_NEIGHBOURS_BIG: one CTA per search, matrix in shared memory (gpfit_big.cuh)
static int fit_big_launch(nngp_handle_t h, const FitArgs& A, int nqj, cudaStream_t st) {
  const int m = A.m, ld = m | 1;
  const size_t smem = sizeof(double) * ((size_t)m * ld + 3 * (size_t)m + 8);
  if (!h->attr_big) {
    const int maxs = (int)(sizeof(double) * ((size_t)NNGP_MAX_NEIGHBOURS_BIG * (NNGP_MAX_NEIGHBOURS_BIG | 1) + 3 * NNGP_MAX_NEIGHBOURS_BIG + 8));
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_fit_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, maxs));
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_select_mean_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, maxs));
    h->attr_big = true;
  }
  int occ = 1;
  NNGP_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gp_fit_big_kernel, BIG_THREADS, smem));
  long long blocks = (long long)h->sm_count * (occ < 1 ? 1 : occ);
  if (blocks > A.ntasks) blocks = A.ntasks;
  ProfScope prof(h, 3, st);
  gp_fit_big_kernel<<<(unsigned)blocks, BIG_THREADS, smem, st>>>(A);
  gp_select_mean_big_kernel<<<nqj, BIG_THREADS, smem, st>>>(A, nqj);
  h->launches += 2;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

#define DISPATCH_CASE(MMV, CALL) else if ((m) <= MMV) { constexpr int MM = MMV; CALL; }
#define DISPATCH_M(m, CALL)                                                   \
  do {                                                                        \
    if ((m) <= 6) { constexpr int MM = 6; CALL; }                             \
    DISPATCH_CASE(8, CALL) DISPATCH_CASE(10, CALL) DISPATCH_CASE(12, CALL)    \
    DISPATCH_CASE(14, CALL) DISPATCH_CASE(16, CALL) DISPATCH_CASE(18, CALL)   \
    DISPATCH_CASE(20, CALL) DISPATCH_CASE(22, CALL) DISPATCH_CASE(24, CALL)   \
    DISPATCH_CASE(26, CALL) DISPATCH_CASE(28, CALL) DISPATCH_CASE(30, CALL)   \
    else { constexpr int MM = 32; CALL; }                                     \
  } while (0)

// `ws` = gp_fit_ws_bytes() block whose first part already holds r2 (gp_prep_launch) and whose
// `done` part is zero (it is left zero by the kernel); `queue` = a zeroed counter.
int gp_fit_predict_launch(nngp_handle_t h, const long long* d_idx, const double* d_dist, void* ws,
                          unsigned int* queue, const int* order, int nq, int m, int R, const signed char* d_starts,
                          double fatol, double xatol, double* d_pred, const double* d_add,
                          long long ld_pred, double* d_theta_opt, double* d_jitter_opt,
                          double* d_fval_opt, int* d_nfev, double* d_fvals, double* d_thetas,
                          cudaStream_t st, int j0, int dl) {
  if (nq <= 0) return 0;
  if (m < 1 || m > NNGP_MAX_NEIGHBOURS_BIG) return nngp_fail(h, "fit: m=%d outside [1,%d]", m, NNGP_MAX_NEIGHBOURS_BIG);
  if (R < 1) return nngp_fail(h, "fit: n_restarts=%d < 1", R);
  const int d = h->ds_d;
  if (dl < 0) dl = d;
  if (j0 < 0 || dl < 1 || j0 + dl > d) return nngp_fail(h, "fit: dimension block [%d,%d) outside [0,%d)", j0, j0 + dl, d);
  const long long ntasks = (long long)nq * dl * NNGP_N_JITTER * R;
  if (ntasks > 0x7fffffffLL) return nngp_fail(h, "fit: %lld searches in one launch (limit 2^31)", ntasks);
  char* base = (char*)ws;
  FitArgs A;
  A.idx = d_idx; A.dist = d_dist; A.Y = h->ds_y; A.starts = d_starts; A.add = d_add;
  A.r2 = (const double*)base;
  A.res = (double*)(base + pad256(gp_prep_bytes(nq, m)));
  A.done = (unsigned int*)(base + gp_fit_done_offset(nq, d, m, R));
  {
    const size_t nt = (size_t)nq * d * NNGP_N_JITTER * R;
    char* after = base + gp_fit_done_offset(nq, d, m, R) + pad256(sizeof(unsigned int) * (size_t)nq * d);
    A.saves = (double*)after;
    A.cont_list = (int*)(after + pad256(sizeof(double) * 12 * nt));
  }
  A.queue = queue;
  A.order = order;
  A.pred = d_pred; A.theta_opt = d_theta_opt; A.jitter_opt = d_jitter_opt; A.fval_opt = d_fval_opt;
  A.nfev = d_nfev; A.fvals = d_fvals; A.thetas = d_thetas; A.counters = h->d_counters;
  A.d = d; A.m = m; A.R = R; A.ntasks = (int)ntasks; A.j0 = j0; A.dl = dl;
  A.head_batch = (getenv("NNGP_FIT_NO_HEAD_BATCH") == nullptr) ? 1 : 0; A.ld_pred = ld_pred; A.fatol = fatol; A.xatol = xatol; A.guard = h->pivot_guard;
  A.budget = 0; A.cont_count = nullptr; A.queue2 = nullptr; A.quad_all = 0;
  if (m > NNGP_MAX_NEIGHBOURS) return fit_big_launch(h, A, nq * dl, st);
  int rc = 0;
  const bool grouped = (h->fit_mode == 2) || (h->fit_mode == 0 && nq >= 4 && m <= 20);
  if (!grouped) {
    // Few searches per launch (a rank's share of the dimension-sharded sweep): the launch lasts as long as its
    // longest search, most warp slots idle -> four warps per search.  Measured per predict at the FHN target
    // (profiles/r02/fit_kernel_variants.log): 576 searches 388 -> 266 us, 1152: 429 -> 375 us, 2304: 504 -> 654 us.
    const long long quad_limit = 3LL * h->sm_count * fit_occ(m);
    if (h->fit_mode == 3 || (h->fit_mode == 0 && ntasks <= quad_limit)) {
      A.quad_all = 1;
    } else if (h->fit_budget >= 3) {
      A.budget = h->fit_budget;
      A.cont_count = queue + 1;
      A.queue2 = queue + 2;
    }
    DISPATCH_M(m, rc = fit_launch_m<MM>(h, A, st));
  } else {
    const int nqj = nq * dl;
    DISPATCH_M(m, rc = fit_grouped_launch_m<MM>(h, A, nqj, st));
  }
  return rc;
}

template <int M>
static int nll_launch_m(nngp_handle_t h, const long long* idx, const double* r2, int nq, int m,
                        int nt, const double* theta, const double* j10, double* out,
                        cudaStream_t st) {
  const size_t smem = warp_tile_bytes<M>();
  bool& attr_set = h->attr_nll[M / 2];
  if (!attr_set) {
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_nll_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  const int d = h->ds_d;
  gp_nll_kernel<M><<<(nq * d + GP_WARPS - 1) / GP_WARPS, GP_WARPS * 32, smem, st>>>(idx, r2, h->ds_y, d, m, nq, nt, theta, j10, out, h->pivot_guard);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

int gp_nll_launch(nngp_handle_t h, const long long* d_idx, const double* d_r2, int nq, int m,
                  int nt, const double* d_theta, const double* d_jitter10, double* d_nll,
                  cudaStream_t st) {
  if (nq <= 0 || nt <= 0) return 0;
  if (m < 1 || m > NNGP_MAX_NEIGHBOURS) return nngp_fail(h, "nll: m=%d outside [1,%d]", m, NNGP_MAX_NEIGHBOURS);
  int rc = 0;
  DISPATCH_M(m, rc = nll_launch_m<MM>(h, d_idx, d_r2, nq, m, nt, d_theta, d_jitter10, d_nll, st));
  return rc;
}

template <int M>
static int mean_launch_m(nngp_handle_t h, const long long* idx, const double* dist,
                         const double* r2, int nq, int m, const double* theta,
                         const double* jitter, double* pred, cudaStream_t st) {
  const size_t smem = warp_tile_bytes<M>();
  bool& attr_set = h->attr_mean[M / 2];
  if (!attr_set) {
    NNGP_CUDA(h, cudaFuncSetAttribute(gp_mean_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  const int d = h->ds_d;
  gp_mean_kernel<M><<<(nq * d + GP_WARPS - 1) / GP_WARPS, GP_WARPS * 32, smem, st>>>(idx, dist, r2, h->ds_y, d, m, nq, theta, jitter, pred, h->pivot_guard);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

int gp_mean_launch(nngp_handle_t h, const long long* d_idx, const double* d_dist,
                   const double* d_r2, int nq, int m, const double* d_theta,
                   const double* d_jitter, double* d_pred, cudaStream_t st) {
  if (nq <= 0) return 0;
  if (m < 1 || m > NNGP_MAX_NEIGHBOURS) return nngp_fail(h, "mean: m=%d outside [1,%d]", m, NNGP_MAX_NEIGHBOURS);
  int rc = 0;
  DISPATCH_M(m, rc = mean_launch_m<MM>(h, d_idx, d_dist, d_r2, nq, m, d_theta, d_jitter, d_pred, st));
  return rc;
}

#ifdef NNGP_FIT_STATS
extern "C" void nngp_fit_stats_dump(void) {
  unsigned long long hst[18];
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(hst, g_fail_hist, sizeof(hst));
  fprintf(stderr, "first failing pivot of wanted evaluations:");
  for (int k = 0; k < 16; k++) fprintf(stderr, " %d:%llu", k, hst[k]);
  fprintf(stderr, " | head fail01 %llu of wanted %llu\n", hst[16], hst[17]);
  unsigned long long z[18] = {0};
  cudaMemcpyToSymbol(g_fail_hist, z, sizeof(z));
  unsigned long long s[16];
  cudaMemcpyFromSymbol(s, g_nm_stats, sizeof(s));
  fprintf(stderr, "nelder_mead evaluations, all-inf iterations: look-ahead %llu head %llu block %llu further %llu | "
          "other: look-ahead %llu head %llu block %llu further %llu | cycles all-inf %llu other %llu | searches %llu "
          "with all-inf iterations %llu (cycles %llu) | longest search %llu cycles\n",
          s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7], s[8], s[9], s[10], s[11], s[12], s[13]);
  cudaMemcpyToSymbol(g_nm_stats, z, sizeof(s));
}
#endif
