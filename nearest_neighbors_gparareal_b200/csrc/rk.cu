// Batched explicit Runge-Kutta propagators and the vector fields of the named systems.
//
// Replaces, for all N time slices in one launch, the reference's per-slice task
//   SolverRK.run_F / run_G -> RK.run_get_last -> _RK_numpy_   (solver.py:86-107, RK.py:101-137)
// and the vector fields ODE.get_vector_field() (systems.py:32-44) with the Normalize affine
// map (utils.py:14-33) fused into the right-hand side.
//
// Arithmetic contract: this file is compiled with -fmad=false.  The closed-form ODE systems
// mirror the reference's NumPy operation order (k_i = h*f(u + sum_j a_ij k_j) accumulated left to
// right from 0, u += np.sum(b*k) in NumPy's 8-lane pairwise order) and reproduce the NumPy path
// bit for bit.  The PDE systems use the 3/5-point periodic stencil form of the reference's dense
// difference matrices -- already not bit-comparable with a BLAS mat-vec -- and explicit fused
// multiply-adds in the stage combinations (ulp-level differences, tests: 1e-11 scaled).
//
// Layouts: small ODEs (d<=4) one THREAD per slice, everything in registers.  PDE systems one
// CTA per slice, the stage input staged in (double-buffered) shared memory for the neighbour
// exchange, the k stages in registers, one barrier per stage: rk_pde_kernel with one thread per
// grid point (any PDE system / normalisation), rk_fhn_tile_kernel with a 2x2 block of points per
// thread for the FHN target (less shared-memory traffic; bit-identical results).  A long fine
// step over more than two slices per SM runs as a sequence of balanced launches over
// (chunk of steps, slice) tasks (launch_fhn_tile_s).  With A.traj set the kernels also store the
// state after every step (run_F_full).
#include "common.cuh"

#include <cmath>
#include <cstdlib>

struct Tableau {
  int S;
  double a[NNGP_MAX_STAGES * NNGP_MAX_STAGES];
  double b[NNGP_MAX_STAGES];
  double c[NNGP_MAX_STAGES];
};

__constant__ Tableau c_tab[4];

static int method_slot(int method) {
  switch (method) {
    case 1: return 0;
    case 2: return 1;
    case 4: return 2;
    case 8: return 3;
    default: return -1;
  }
}

// RK.py:30-48, same expressions evaluated in IEEE double.
static void build_tableau(int method, Tableau* T) {
  for (double& v : T->a) v = 0.0;
  for (double& v : T->b) v = 0.0;
  for (double& v : T->c) v = 0.0;
  auto A = [&](int i, int j) -> double& { return T->a[i * NNGP_MAX_STAGES + j]; };
  if (method == 1) {
    T->S = 1;
    T->b[0] = 1.0;
  } else if (method == 2) {
    T->S = 2;
    A(1, 0) = 0.5;
    T->b[1] = 1.0;
    T->c[1] = 0.5;
  } else if (method == 4) {
    T->S = 4;
    A(1, 0) = 0.5;
    A(2, 1) = 0.5;
    A(3, 2) = 1.0;
    T->b[0] = 1.0 / 6;
    T->b[1] = 1.0 / 3;
    T->b[2] = 1.0 / 3;
    T->b[3] = 1.0 / 6;
    T->c[1] = 0.5;
    T->c[2] = 0.5;
    T->c[3] = 1.0;
  } else {
    T->S = 11;
    volatile double s21 = 21.0;
    const double s = std::sqrt(s21);
    A(1, 0) = 1.0 / 2;
    A(2, 0) = 1.0 / 4;
    A(2, 1) = 1.0 / 4;
    A(3, 0) = 1.0 / 7;
    A(3, 1) = (-7 - 3 * s) / 98;
    A(3, 2) = (21 + 5 * s) / 49;
    A(4, 0) = (11 + s) / 84;
    A(4, 2) = (18 + 4 * s) / 63;
    A(4, 3) = (21 - s) / 252;
    A(5, 0) = (5 + s) / 48;
    A(5, 2) = (9 + s) / 36;
    A(5, 3) = (-231 + 14 * s) / 360;
    A(5, 4) = (63 - 7 * s) / 80;
    A(6, 0) = (10 - s) / 42;
    A(6, 2) = (-432 + 92 * s) / 315;
    A(6, 3) = (633 - 145 * s) / 90;
    A(6, 4) = (-504 + 115 * s) / 70;
    A(6, 5) = (63 - 13 * s) / 35;
    A(7, 0) = 1.0 / 14;
    A(7, 4) = (14 - 3 * s) / 126;
    A(7, 5) = (13 - 3 * s) / 63;
    A(7, 6) = 1.0 / 9;
    A(8, 0) = 1.0 / 32;
    A(8, 4) = (91 - 21 * s) / 576;
    A(8, 5) = 11.0 / 72;
    A(8, 6) = (-385 - 75 * s) / 1152;
    A(8, 7) = (63 + 13 * s) / 128;
    A(9, 0) = 1.0 / 14;
    A(9, 4) = 1.0 / 9;
    A(9, 5) = (-733 - 147 * s) / 2205;
    A(9, 6) = (515 + 111 * s) / 504;
    A(9, 7) = (-51 - 11 * s) / 56;
    A(9, 8) = (132 + 28 * s) / 245;
    A(10, 4) = (-42 + 7 * s) / 18;
    A(10, 5) = (-18 + 28 * s) / 45;
    A(10, 6) = (-273 - 53 * s) / 72;
    A(10, 7) = (301 + 53 * s) / 72;
    A(10, 8) = (28 - 28 * s) / 45;
    A(10, 9) = (49 - 7 * s) / 18;
    T->b[0] = 1.0 / 20;
    T->b[7] = 49.0 / 180;
    T->b[8] = 16.0 / 45;
    T->b[9] = 49.0 / 180;
    T->b[10] = 1.0 / 20;
    const double cp = (7 + s) / 14, cm = (7 - s) / 14;
    const double cc[11] = {0, 1.0 / 2, 1.0 / 2, cp, cp, 1.0 / 2, cm, cm, 1.0 / 2, cp, 1};
    for (int i = 0; i < 11; i++) T->c[i] = cc[i];
  }
}

void rk_host_tableau(int method, int* S, double* a, double* b, double* c) {
  Tableau T;
  build_tableau(method, &T);
  *S = T.S;
  for (int i = 0; i < T.S; i++) {
    for (int j = 0; j < T.S; j++) a[i * T.S + j] = T.a[i * NNGP_MAX_STAGES + j];
    b[i] = T.b[i];
    c[i] = T.c[i];
  }
}

int rk_set_tableaus(nngp_handle_t h) {
  Tableau T[4];
  const int methods[4] = {1, 2, 4, 8};
  for (int i = 0; i < 4; i++) build_tableau(methods[i], &T[i]);
  NNGP_CUDA(h, cudaMemcpyToSymbol(c_tab, T, sizeof(T)));
  return 0;
}

// ---------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------
// x**3 as NumPy computes it (libm pow, correctly rounded in practice): product with the
// rounding error of x*x carried along.
__device__ __forceinline__ double cube_cr(double x) {
  const double p = x * x;
  const double e = fma(x, x, -p);
  const double r = p * x;
  const double re = fma(p, x, -r);
  return r + (re + e * x);
}

// node time of np.linspace(t0, t1, steps+1)[n]  (RK.py:93)
__device__ __forceinline__ double linspace_node(double t0, double t1, double step, long long n,
                                                long long steps) {
  return (n == steps) ? t1 : ((double)n * step + t0);
}

__device__ __forceinline__ double step_size(int h_mode, double t0, double t1, double step,
                                            long long n, long long steps) {
  if (h_mode == NNGP_H_CONST) return step;
  return linspace_node(t0, t1, step, n + 1, steps) - linspace_node(t0, t1, step, n, steps);
}

// np.sum(b*k, axis=1) over S stage terms: NumPy's pairwise_sum (8 lanes, then the tail)
template <int S>
__device__ __forceinline__ double numpy_sum_bk(const double (&k)[S], const double* b) {
  if constexpr (S < 8) {
    double r = 0.0;
#pragma unroll
    for (int i = 0; i < S; i++) r = r + b[i] * k[i];
    return r;
  } else {
    double r[8];
#pragma unroll
    for (int i = 0; i < 8; i++) r[i] = b[i] * k[i];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
    for (int i = 8; i < S; i++) res = res + b[i] * k[i];
    return res;
  }
}

// ---------------------------------------------------------------------------------------
// closed-form ODE systems (systems.py:80-288), evaluated on de-normalised v[D]
// ---------------------------------------------------------------------------------------
template <int SYS>
struct SmallDim;
template <> struct SmallDim<NNGP_SYS_FHN_ODE> { static constexpr int D = 2; };
template <> struct SmallDim<NNGP_SYS_ROSSLER> { static constexpr int D = 3; };
template <> struct SmallDim<NNGP_SYS_HOPF> { static constexpr int D = 3; };
template <> struct SmallDim<NNGP_SYS_DBLPEND> { static constexpr int D = 4; };
template <> struct SmallDim<NNGP_SYS_BRUSSELATOR> { static constexpr int D = 2; };
template <> struct SmallDim<NNGP_SYS_LORENZ> { static constexpr int D = 3; };
template <> struct SmallDim<NNGP_SYS_THOMAS> { static constexpr int D = 3; };

template <int SYS, int D>
__device__ __forceinline__ void small_field(const double* P, const double (&u)[D], double (&o)[D]) {
  if constexpr (SYS == NNGP_SYS_FHN_ODE) {  // systems.py:97-106
    const double a = 0.2, b = 0.2, c = 3.0;
    o[0] = c * ((u[0] - (cube_cr(u[0]) / 3.0)) + u[1]);
    o[1] = (-(1.0 / c)) * ((u[0] - a) + b * u[1]);
  } else if constexpr (SYS == NNGP_SYS_ROSSLER) {  // systems.py:128-137
    const double a = 0.2, b = 0.2, c = 5.7;
    o[0] = (-u[1]) - u[2];
    o[1] = u[0] + (a * u[1]);
    o[2] = b + u[2] * (u[0] - c);
  } else if constexpr (SYS == NNGP_SYS_HOPF) {  // systems.py:157-163, P[0] = maxtime
    const double g = ((u[2] / P[0]) - u[0] * u[0]) - u[1] * u[1];
    o[0] = (-u[1]) + u[0] * g;
    o[1] = u[0] + u[1] * g;
    o[2] = 1.0;
  } else if constexpr (SYS == NNGP_SYS_DBLPEND) {  // systems.py:191-199
    const double dl = u[0] - u[2];
    const double cd = cos(dl), sd = sin(dl);
    const double pre = -1.0 / (2.0 - cd * cd);
    o[0] = u[1];
    o[1] = pre * (((((u[1] * u[1]) * cd) * sd + (u[3] * u[3]) * sd) + 2.0 * sin(u[0])) - cd * sin(u[2]));
    o[2] = u[3];
    o[3] = pre * (((((-2.0 * (u[1] * u[1])) * sd) - ((u[3] * u[3]) * sd) * cd) - (2.0 * cd) * sin(u[0])) + 2.0 * sin(u[2]));
  } else if constexpr (SYS == NNGP_SYS_BRUSSELATOR) {  // systems.py:217-222
    o[0] = (1.0 + (u[0] * u[0]) * u[1]) - 4.0 * u[0];
    o[1] = 3.0 * u[0] - (u[0] * u[0]) * u[1];
  } else if constexpr (SYS == NNGP_SYS_LORENZ) {  // systems.py:241-247
    o[0] = 10.0 * (u[1] - u[0]);
    o[1] = (28.0 * u[0] - u[1]) - u[0] * u[2];
    o[2] = u[0] * u[1] - (8.0 / 3.0) * u[2];
  } else {  // NNGP_SYS_THOMAS, systems.py:273-288
    const double a = 0.5, b = 10.0;
    o[0] = (-a) * u[0] + b * sin(u[1]);
    o[1] = (-a) * u[1] + b * sin(u[2]);
    o[2] = (-a) * u[2] + b * sin(u[0]);
  }
}

// normalised field systems.py:36-40: f(inverse(u)) * scale
template <int SYS, int D>
__device__ __forceinline__ void small_field_n(const SysArgs& A, const double (&mn)[D],
                                              const double (&rg)[D], const double (&sc)[D],
                                              const double (&u)[D], double (&o)[D]) {
  if (A.normalize) {
    double v[D];
#pragma unroll
    for (int i = 0; i < D; i++) v[i] = ((u[i] + 1.0) / 2.0) * rg[i] + mn[i];
    small_field<SYS, D>(A.p, v, o);
#pragma unroll
    for (int i = 0; i < D; i++) o[i] = o[i] * sc[i];
  } else {
    small_field<SYS, D>(A.p, u, o);
  }
}

template <int S>
struct SlotOf { static constexpr int value = (S == 1) ? 0 : (S == 2) ? 1 : (S == 4) ? 2 : 3; };

// structural non-zeros of the Butcher matrices of RK.py:30-48 (a term a_ij*k_j with a_ij = 0 adds
// exactly nothing, so skipping it is bit-identical to the reference's dense accumulation)
template <int S>
__host__ __device__ constexpr bool a_nonzero(int i, int j) {
  if (S == 2) return i == 1 && j == 0;
  if (S == 4) return j == i - 1;
  if (S == 11) {
    if (i <= 3) return true;
    if (i <= 6) return j != 1;
    if (i <= 9) return j == 0 || j >= 4;
    return j >= 4;
  }
  return false;
}
template <int S>
__host__ __device__ constexpr bool b_nonzero(int i) {
  if (S == 2) return i == 1;
  if (S == 11) return i == 0 || i >= 7;
  return true;
}

template <int SYS, int S>
__global__ void __launch_bounds__(32)
rk_small_kernel(SysArgs A, int h_mode, long long steps, int n_slices,
                const double* __restrict__ t0s, const double* __restrict__ t1s,
                const double* __restrict__ u0, long long ld0, double* __restrict__ u1,
                long long ld1) {
  constexpr int D = SmallDim<SYS>::D;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slices) return;
  const Tableau& T = c_tab[SlotOf<S>::value];
  double mn[D], rg[D], sc[D], u[D];
#pragma unroll
  for (int i = 0; i < D; i++) {
    mn[i] = A.normalize ? A.mn[i] : 0.0;
    rg[i] = A.normalize ? (A.mx[i] - A.mn[i]) : 2.0;
    sc[i] = 2.0 / rg[i];
    u[i] = u0[s * ld0 + i];
  }
  const double t0 = t0s[s], t1 = t1s[s];
  const double step = (t1 - t0) / (double)steps;
  double k[D][S];
  double* traj = A.traj ? A.traj + (long long)s * (steps + 1) * D : nullptr;
  if (traj) {
#pragma unroll
    for (int i = 0; i < D; i++) traj[i] = u[i];
  }
  for (long long n = 0; n < steps; n++) {
    const double h = step_size(h_mode, t0, t1, step, n, steps);
#pragma unroll
    for (int i = 0; i < S; i++) {
      double w[D], f[D];
#pragma unroll
      for (int c = 0; c < D; c++) {
        double tmp = 0.0;
#pragma unroll
        for (int j = 0; j < i; j++)
          if (a_nonzero<S>(i, j)) tmp = tmp + T.a[i * NNGP_MAX_STAGES + j] * k[c][j];
        w[c] = (i == 0) ? u[c] : (u[c] + tmp);
      }
      small_field_n<SYS, D>(A, mn, rg, sc, w, f);
#pragma unroll
      for (int c = 0; c < D; c++) k[c][i] = h * f[c];
    }
#pragma unroll
    for (int c = 0; c < D; c++) u[c] = u[c] + numpy_sum_bk<S>(k[c], T.b);
    if (traj) {
#pragma unroll
      for (int c = 0; c < D; c++) traj[(n + 1) * D + c] = u[c];
    }
  }
#pragma unroll
  for (int i = 0; i < D; i++) u1[s * ld1 + i] = u[i];
}

template <int SYS>
__global__ void rhs_small_kernel(SysArgs A, int n, const double* __restrict__ u,
                                 double* __restrict__ out) {
  constexpr int D = SmallDim<SYS>::D;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  double mn[D], rg[D], sc[D], w[D], f[D];
#pragma unroll
  for (int i = 0; i < D; i++) {
    mn[i] = A.normalize ? A.mn[i] : 0.0;
    rg[i] = A.normalize ? (A.mx[i] - A.mn[i]) : 2.0;
    sc[i] = 2.0 / rg[i];
    w[i] = u[(long long)s * D + i];
  }
  small_field_n<SYS, D>(A, mn, rg, sc, w, f);
#pragma unroll
  for (int i = 0; i < D; i++) out[(long long)s * D + i] = f[i];
}

// ---------------------------------------------------------------------------------------
// PDE systems: one CTA per slice, one thread per grid point
// ---------------------------------------------------------------------------------------
// FitzHugh-Nagumo on a periodic d_x x d_x grid (systems.py:291-383).  State = [u1 | u2],
// point p = iy*d_x + ix; DXX = kron(I, Dxx) couples ix+-1, DYY = kron(Dyy, I) couples iy+-1.
// params: [d_x, a*diag, a*off, b*diag, b*off, k, 1/tau] -- the entries of a*(DXX+DYY) and
// b*(DXX+DYY) computed on the host exactly as the reference builds its dense matrices.
struct FhnPde {
  static constexpr int NC = 2;
  int pl, pr, pd, pu, npts;
  __device__ void setup(const SysArgs& A, int p) {
    const int dx = (int)A.p[0];
    npts = dx * dx;
    const int ix = p % dx, iy = p / dx;
    pl = iy * dx + (ix == 0 ? dx - 1 : ix - 1);
    pr = iy * dx + (ix == dx - 1 ? 0 : ix + 1);
    pd = (iy == 0 ? dx - 1 : iy - 1) * dx + ix;
    pu = (iy == dx - 1 ? 0 : iy + 1) * dx + ix;
  }
  __device__ static int points(const SysArgs& A) { return (int)A.p[0] * (int)A.p[0]; }
  // buf holds the de-normalised stage input of every point: [u1 (npts) | u2 (npts)]
  __device__ void eval(const SysArgs& A, const double* buf, int p, const double (&v)[2],
                       double (&f)[2]) const {
    const double* b1 = buf;
    const double* b2 = buf + npts;
    const double s1 = (b1[pd] + b1[pl]) + (b1[pr] + b1[pu]);
    const double s2 = (b2[pd] + b2[pl]) + (b2[pr] + b2[pu]);
    const double m1 = fma(A.p[2], s1, A.p[1] * v[0]);  // a*(DXX+DYY)@u1 as a 5-point stencil
    const double m2 = fma(A.p[4], s2, A.p[3] * v[1]);
    // U = a*(DXX+DYY)@u1 + u1 - u1**3 - u2 + k ;  V = (1/tau)*(b*(DXX+DYY)@u2 + u1 - u2)
    f[0] = (((m1 + v[0]) - (v[0] * v[0]) * v[0]) - v[1]) + A.p[5];
    f[1] = A.p[6] * ((m2 + v[0]) - v[1]);
  }
  // Stage increment k_c = hs_c * f_c in 14 FP64 instructions per grid point and stage, coefficients
  // from the constant bank (q = derived parameters filled in by nngp_sys_args):
  //   hs0 U = hs0 (a_off S1 + u1 ((a_diag + 1) - u1^2) + (k - u2)),   S = sum of the four neighbours
  //   hs1 V = (hs1 b_off/tau) S2 + (hs1 (b_diag - 1)/tau) u2 + (hs1/tau) u1   (hv = the three products, once per step)
  __device__ static void step_coeffs(const SysArgs& A, double hs1, double (&hv)[3]) {
    hv[0] = hs1 * A.q[1];
    hv[1] = hs1 * A.q[2];
    hv[2] = hs1 * A.p[6];
  }
  __device__ void eval_k(const SysArgs& A, const double* buf, int p, const double (&v)[2],
                         const double (&hs)[2], const double (&hv)[3], double (&k)[2]) const {
    const double* b1 = buf;
    const double* b2 = buf + npts;
    const double s1 = (b1[pd] + b1[pl]) + (b1[pr] + b1[pu]);
    const double s2 = (b2[pd] + b2[pl]) + (b2[pr] + b2[pu]);
    const double t1 = fma(-v[0], v[0], A.q[0]);
    const double t2 = A.p[5] - v[1];
    k[0] = hs[0] * fma(A.p[2], s1, fma(v[0], t1, t2));
    k[1] = fma(hv[0], s2, fma(hv[1], v[1], hv[2] * v[0]));
  }
};

// Viscous Burgers, periodic central differences (systems.py:402-450).
// params: [Dxx_off, Dxx_diag, Dx_off]
struct BurgersPde {
  static constexpr int NC = 1;
  int pl, pr, npts;
  __device__ void setup(const SysArgs& A, int p) {
    npts = A.d;
    pl = (p == 0) ? npts - 1 : p - 1;
    pr = (p == npts - 1) ? 0 : p + 1;
  }
  __device__ static int points(const SysArgs& A) { return A.d; }
  __device__ void eval(const SysArgs& A, const double* buf, int p, const double (&v)[1],
                       double (&f)[1]) const {
    const double ul = buf[pl], ur = buf[pr];
    const double lap = fma(A.p[0], ul + ur, A.p[1] * v[0]);
    const double adv = A.p[2] * (ur - ul);
    f[0] = fma(-v[0], adv, lap);  // Dxx@u - u*(Dx@u)
  }
  // k = hs (Dxx_off (ul + ur) + u (Dxx_diag - Dx_off (ur - ul)))
  __device__ static void step_coeffs(const SysArgs&, double, double (&)[3]) {}
  __device__ void eval_k(const SysArgs& A, const double* buf, int p, const double (&v)[1],
                         const double (&hs)[1], const double (&)[3], double (&k)[1]) const {
    const double ul = buf[pl], ur = buf[pr];
    k[0] = hs[0] * fma(A.p[0], ul + ur, v[0] * fma(-A.p[2], ur - ul, A.p[1]));
  }
};

// CTAs per SM the PDE kernel is compiled for: 256-thread CTAs x 4 = all 512 slices of the FHN
// target resident in one wave on 148 SMs (64 registers per thread; the RK8 stage values that are
// live at the same time -- at most 8 of the 11 per component -- just fit)
template <int TB> struct PdeOcc { static constexpr int value = (TB <= 256) ? 4 : 1; };

// The stage combination and the final update use fused multiply-adds here: the PDE fields are not
// bit-comparable with the reference anyway (stencil vs dense BLAS mat-vec), and FMA halves the FP64
// instruction count of the step.
template <class RHS, int S, int TB, bool NORM>
__global__ void __launch_bounds__(TB, PdeOcc<TB>::value)
rk_pde_kernel(SysArgs A, int h_mode, long long steps, const double* __restrict__ t0s,
              const double* __restrict__ t1s, const double* __restrict__ u0, long long ld0,
              double* __restrict__ u1, long long ld1) {
  constexpr int NC = RHS::NC;
  extern __shared__ double sm[];
  const Tableau& T = c_tab[SlotOf<S>::value];
  const int npts = RHS::points(A);
  const int p = threadIdx.x;
  const bool active = p < npts;
  const int pp = active ? p : 0;
  const long long s = blockIdx.x;
  RHS rhs;
  rhs.setup(A, pp);
  double u[NC], mn[NC], hrg[NC], sc[NC], k[NC][S];
#pragma unroll
  for (int c = 0; c < NC; c++) {
    u[c] = u0[s * ld0 + c * npts + pp];
    mn[c] = NORM ? A.mn[c * npts + pp] : 0.0;
    const double rg = NORM ? (A.mx[c * npts + pp] - A.mn[c * npts + pp]) : 2.0;
    hrg[c] = 0.5 * rg;
    sc[c] = 2.0 / rg;
  }
  const double t0 = t0s[s], t1 = t1s[s];
  const double step = (t1 - t0) / (double)steps;
  int par = 0;
  double* traj = A.traj ? A.traj + s * (steps + 1) * A.d : nullptr;
  if (traj && active) {
#pragma unroll
    for (int c = 0; c < NC; c++) traj[c * npts + p] = u[c];
  }
  for (long long n = 0; n < steps; n++) {
    const double h = step_size(h_mode, t0, t1, step, n, steps);
    double hs[NC], hv[3];
#pragma unroll
    for (int c = 0; c < NC; c++) hs[c] = NORM ? h * sc[c] : h;
    RHS::step_coeffs(A, hs[NC - 1], hv);
#pragma unroll
    for (int i = 0; i < S; i++) {
      double v[NC], f[NC];
      double* buf = sm + par * (NC * npts);
      par ^= 1;
#pragma unroll
      for (int c = 0; c < NC; c++) {
        double w = u[c];
#pragma unroll
        for (int j = 0; j < i; j++)
          if (a_nonzero<S>(i, j)) w = fma(T.a[i * NNGP_MAX_STAGES + j], k[c][j], w);
        v[c] = NORM ? fma(w + 1.0, hrg[c], mn[c]) : w;  // utils.py:24-27
        if (active) buf[c * npts + p] = v[c];
      }
      __syncthreads();
      rhs.eval_k(A, buf, pp, v, hs, hv, f);
#pragma unroll
      for (int c = 0; c < NC; c++) k[c][i] = f[c];
    }
#pragma unroll
    for (int c = 0; c < NC; c++) {
#pragma unroll
      for (int i = 0; i < S; i++)
        if (b_nonzero<S>(i)) u[c] = fma(T.b[i], k[c][i], u[c]);
    }
    if (traj && active) {
#pragma unroll
      for (int c = 0; c < NC; c++) traj[(n + 1) * A.d + c * npts + p] = u[c];
    }
  }
  if (active) {
#pragma unroll
    for (int c = 0; c < NC; c++) u1[s * ld1 + c * npts + p] = u[c];
  }
}

// ---------------------------------------------------------------------------------------
// FHN, identity normalisation, even d_x: one thread owns a TY x 2 block of grid points (both fields).
// ncu (profiles/r01/rk_r1d.summary.csv) shows rk_pde_kernel bound by the shared-memory pipe
// (8 neighbour loads + 2 stores per point and stage); with 2x2 blocks half of the neighbours are the
// thread's own registers and the vertical ones come as aligned 16-byte pairs: 12 instead of 20
// shared-memory accesses per point pair, and 4x fewer threads per barrier.  Per-point arithmetic and
// summation order are those of FhnPde::eval_k, so all kernels return identical bits.
//   TY = 2 (64 threads per 16x16 slice): least shared-memory traffic -- the throughput shape, used
//          when every SM holds several slices (one GPU: 512 slices on 148 SMs);
//   TY = 1 (128 threads per slice): a slice spreads over all four SM sub-partitions, each warp
//          issuing half the FP64 work -- the latency shape, used when a GPU holds at most two slices
//          per SM (a rank of a multi-GPU run), where a slice's own step time is what counts.
// ---------------------------------------------------------------------------------------
template <int TY, int TB>
struct TileOcc { static constexpr int value = (TY == 2) ? ((TB <= 64) ? 4 : 1) : ((TB <= 128) ? 2 : 1); };

template <int S, int TY, int TB, bool TRAJ, bool SHX>
__global__ void __launch_bounds__(TB, TileOcc<TY, TB>::value)
rk_fhn_tile_kernel(SysArgs A, int h_mode, long long steps, int n_slices, long long task0, int n_chunks,
                   const double* __restrict__ t0s, const double* __restrict__ t1s,
                   const double* __restrict__ u0, long long ld0, double* __restrict__ u1, long long ld1) {
  constexpr int NV = 2 * TY;  // points per thread, row-major inside the block
  // task = (chunk of the step range, slice): chunk c of a slice continues from u1 where chunk c-1 (an
  // earlier launch) left it -- see launch_fhn_tile
  const long long task = task0 + blockIdx.x;
  if (task >= (long long)n_slices * n_chunks) return;
  const int chunk = (int)(task / n_slices);
  const long long s = task - (long long)chunk * n_slices;
  const long long n_begin = (steps * chunk) / n_chunks, n_end = (steps * (chunk + 1)) / n_chunks;
  extern __shared__ double sm[];
  const Tableau& T = c_tab[SlotOf<S>::value];
  const int dx = (int)A.p[0], npts = dx * dx, hx = dx >> 1, ntile = hx * (dx / TY);
  const bool active = (int)threadIdx.x < ntile;
  const int tt = active ? threadIdx.x : 0;
  const int ix0 = 2 * (tt % hx), iy0 = TY * (tt / hx);
  const int o00 = iy0 * dx + ix0;
  const int oup = ((iy0 == 0 ? dx : iy0) - 1) * dx + ix0;        // row iy0-1, columns ix0, ix0+1
  const int odn = ((iy0 + TY == dx) ? 0 : iy0 + TY) * dx + ix0;  // row iy0+TY
  const int xl = (ix0 == 0 ? dx : ix0) - 1, xr = (ix0 + 2 == dx) ? 0 : ix0 + 2;
  // Column loads: a left neighbour sits in an odd column, a right one in an even column, and a 128-byte line holds
  // 16 doubles, so if every thread fetched its left (or right) neighbour in the same instruction, the 16 threads of a
  // half-warp would share 8 eight-byte bank pairs: 2 wavefronts per 64-bit load instead of 1 (16 of the 64 shared-memory
  // wavefronts per warp and stage at d_x = 16, profiles/r01/rk_tile_r1.summary.csv).  Instead, threads with flip set
  // fetch the right neighbour first.  flip alternates between the block rows of a half-warp at d_x = 16 (and between
  // the two halves of a row at d_x = 32), so each half-warp reads 8 odd and 8 even columns: conflict-free, 48 wavefronts
  // (scripts/rk_shared_wavefronts.py).  The two loaded values trade places in registers: 16 FSEL per thread and stage,
  // 222 registers for <11, 2, 64>.  Same values, same arithmetic: the same bits.  (A swizzled buffer -- the pairs of
  // alternate block rows stored swapped -- is conflict-free too, but has to undo the swap for the own and the upper and
  // lower pairs: 32 FSEL per stage and 226 registers with 128-bit accesses, or 239 registers with 64-bit ones.)
  const bool flip = (((iy0 / TY) ^ (ix0 >> 4)) & 1) != 0;
  const int oc0 = iy0 * dx + (flip ? xr : xl), oc1 = iy0 * dx + (flip ? xl : xr);
  // shx: the left / right neighbour columns come from the neighbouring lanes of the same block row by shuffle instead
  // of shared memory (the threads of a block row are hx consecutive lanes; hx a power of two <= 32).
  const int lane = threadIdx.x & 31;
  const int lsrc = (lane & ~(hx - 1)) | ((lane - 1) & (hx - 1)), rsrc = (lane & ~(hx - 1)) | ((lane + 1) & (hx - 1));
  double u[2][NV], k[2][NV][S];
#pragma unroll
  for (int c = 0; c < 2; c++) {
    const double* src = ((chunk == 0) ? u0 + s * ld0 : u1 + s * ld1) + c * npts;
#pragma unroll
    for (int r = 0; r < TY; r++) {
      u[c][2 * r] = src[o00 + r * dx];
      u[c][2 * r + 1] = src[o00 + r * dx + 1];
    }
  }
  const double t0 = t0s[s], t1 = t1s[s];
  const double step = (t1 - t0) / (double)steps;
  int par = 0;
  double* traj = TRAJ ? A.traj + s * (steps + 1) * (2 * npts) : nullptr;  // TRAJ: run_F_full, every step stored
  auto put = [&](long long row) {
#pragma unroll
    for (int c = 0; c < 2; c++)
#pragma unroll
      for (int r = 0; r < TY; r++) {
        traj[row * (2 * npts) + c * npts + o00 + r * dx] = u[c][2 * r];
        traj[row * (2 * npts) + c * npts + o00 + r * dx + 1] = u[c][2 * r + 1];
      }
  };
  if (TRAJ && active && n_begin == 0) put(0);
  for (long long n = n_begin; n < n_end; n++) {
    const double h = step_size(h_mode, t0, t1, step, n, steps);
    double hv[3];
    FhnPde::step_coeffs(A, h, hv);
    // xn: the next stage's input without its newest term, u + sum_{j<i} a_{i+1,j} k_j -- formed while the
    // neighbour loads of stage i are in flight (same ascending order of the terms: same bits)
    double xn[2][NV];
#pragma unroll
    for (int c = 0; c < 2; c++)
#pragma unroll
      for (int q = 0; q < NV; q++) xn[c][q] = u[c][q];
#pragma unroll
    for (int i = 0; i < S; i++) {
      double* buf = sm + par * (2 * npts);
      par ^= 1;
      double w[2][NV], sn[2][NV];
#pragma unroll
      for (int c = 0; c < 2; c++) {
#pragma unroll
        for (int q = 0; q < NV; q++) {
          double x = xn[c][q];
          if (i > 0 && a_nonzero<S>(i, i - 1)) x = fma(T.a[i * NNGP_MAX_STAGES + i - 1], k[c][q][i - 1], x);
          w[c][q] = x;
        }
        if (active) {
#pragma unroll
          for (int r = 0; r < TY; r++)
            *reinterpret_cast<double2*>(buf + c * npts + o00 + r * dx) = make_double2(w[c][2 * r], w[c][2 * r + 1]);
        }
      }
      double lf[2][TY], rt[2][TY];
      if (SHX) {
#pragma unroll
        for (int c = 0; c < 2; c++)
#pragma unroll
          for (int r = 0; r < TY; r++) {
            lf[c][r] = __shfl_sync(0xffffffffu, w[c][2 * r + 1], lsrc);
            rt[c][r] = __shfl_sync(0xffffffffu, w[c][2 * r], rsrc);
          }
      }
      __syncthreads();
      double2 up[2], dn[2];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        const double* b = buf + c * npts;
        up[c] = *reinterpret_cast<const double2*>(b + oup);
        dn[c] = *reinterpret_cast<const double2*>(b + odn);
        if (!SHX) {
#pragma unroll
          for (int r = 0; r < TY; r++) {
            const double c0 = b[oc0 + r * dx], c1 = b[oc1 + r * dx];
            lf[c][r] = flip ? c1 : c0;
            rt[c][r] = flip ? c0 : c1;
          }
        }
      }
      if (i + 1 < S) {
#pragma unroll
        for (int c = 0; c < 2; c++)
#pragma unroll
          for (int q = 0; q < NV; q++) {
            double x = u[c][q];
#pragma unroll
            for (int j = 0; j < i; j++)
              if (a_nonzero<S>(i + 1, j)) x = fma(T.a[(i + 1) * NNGP_MAX_STAGES + j], k[c][q][j], x);
            xn[c][q] = x;
          }
      }
#pragma unroll
      for (int c = 0; c < 2; c++) {
        const double2 up_c = up[c], dn_c = dn[c];
#pragma unroll
        for (int r = 0; r < TY; r++) {
          const double l = lf[c][r], rr = rt[c][r];
          const double ax = (r == 0) ? up_c.x : w[c][2 * (r - 1)], ay = (r == 0) ? up_c.y : w[c][2 * (r - 1) + 1];
          const double bx = (r == TY - 1) ? dn_c.x : w[c][2 * (r + 1)], by = (r == TY - 1) ? dn_c.y : w[c][2 * (r + 1) + 1];
          // (v[iy-1] + v[ix-1]) + (v[ix+1] + v[iy+1]) as in FhnPde::eval_k
          sn[c][2 * r] = (ax + l) + (w[c][2 * r + 1] + bx);
          sn[c][2 * r + 1] = (ay + w[c][2 * r]) + (rr + by);
        }
      }
#pragma unroll
      for (int q = 0; q < NV; q++) {
        const double v0 = w[0][q], v1 = w[1][q];
        const double e1 = fma(-v0, v0, A.q[0]);
        const double e2 = A.p[5] - v1;
        k[0][q][i] = h * fma(A.p[2], sn[0][q], fma(v0, e1, e2));
        k[1][q][i] = fma(hv[0], sn[1][q], fma(hv[1], v1, hv[2] * v0));
      }
    }
#pragma unroll
    for (int c = 0; c < 2; c++)
#pragma unroll
      for (int q = 0; q < NV; q++)
#pragma unroll
        for (int i = 0; i < S; i++)
          if (b_nonzero<S>(i)) u[c][q] = fma(T.b[i], k[c][q][i], u[c][q]);
    if (TRAJ && active) put(n + 1);
  }
  if (active) {
#pragma unroll
    for (int c = 0; c < 2; c++) {
      double* dst = u1 + s * ld1 + c * npts;
#pragma unroll
      for (int r = 0; r < TY; r++) {
        dst[o00 + r * dx] = u[c][2 * r];
        dst[o00 + r * dx + 1] = u[c][2 * r + 1];
      }
    }
  }
}

// Time-chunked launch.  Measured (profiles/r01/rk_sweep.log; again with conflict-free column loads,
// profiles/r04/rk_layout_sweep.log): an SM reaches nearly its full fine-step throughput with TWO resident slices (one
// warp per sub-partition); 3 slices per SM are slower than 2 (two sub-partitions hold two warps: 3 per SM chunked,
// 512 slices, 625 ms against 507), 4 gain 4 % per slice (one launch of 592 slices: 560 ms against 2 x 291), and 512
// slices in one launch leave 80 SMs a slice short (560 ms).  So when a GPU holds more than 2 slices per SM the step
// range is cut into chunks and the (chunk, slice) tasks are executed chunk-major by a sequence of launches of
// exactly 2 CTAs per SM (forced by the shared-memory request): every launch is perfectly balanced, a slice's state
// passes from chunk to chunk through u1, and task (c, s) always falls into a later launch than (c-1, s) because a
// launch is smaller than the number of slices.  Results are bit-identical to the single launch.
template <int S, int TY, int TB, bool SHX>
static int launch_fhn_tile_x(const SysArgs& A, int npts, int h_mode, long long steps, int n, int sms,
                             const double* t0, const double* t1, const double* u0, long long ld0, double* u1,
                             long long ld1, cudaStream_t st) {
  const int threads = ((npts / (2 * TY) + 31) / 32) * 32;
  const size_t smem = 2 * sizeof(double) * 2 * npts;

  const int per_launch = 2 * sms;
  const char* force = getenv("NNGP_RK_CHUNKS");  // experiments: 0 = never chunk
  if (A.traj != nullptr) {  // every step stored (run_F_full): one launch
    rk_fhn_tile_kernel<S, TY, TB, true, SHX><<<n, threads, smem, st>>>(A, h_mode, steps, n, 0, 1, t0, t1, u0, ld0, u1, ld1);
    return 1;
  }
  if (TB > 64 || n <= per_launch || steps < 4096 || (force && force[0] == '0')) {
    rk_fhn_tile_kernel<S, TY, TB, false, SHX><<<n, threads, smem, st>>>(A, h_mode, steps, n, 0, 1, t0, t1, u0, ld0, u1, ld1);
    return 1;
  }
  // chunks: the smallest count >= 24 that fills the last launch, else 32
  int chunks = 32;
  for (int c = 24; c <= 64; c++)
    if (((long long)n * c) % per_launch == 0) {
      chunks = c;
      break;
    }
  const size_t smem2 = 80 * 1024;  // > 1/3 of the SM's shared memory: at most two CTAs per SM
  // per device, so set on every fine step (64 launches follow): a process may hold handles on several GPUs
  cudaFuncSetAttribute(rk_fhn_tile_kernel<S, TY, TB, false, SHX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
  const long long total = (long long)n * chunks;
  int launches = 0;
  for (long long task0 = 0; task0 < total; task0 += per_launch) {
    const int grid = (int)((total - task0 < per_launch) ? total - task0 : per_launch);
    rk_fhn_tile_kernel<S, TY, TB, false, SHX><<<grid, threads, smem2, st>>>(A, h_mode, steps, n, task0, chunks, t0, t1, u0, ld0, u1, ld1);
    launches++;
  }
  return launches;
}

template <int S, int TY, int TB>
static int launch_fhn_tile_s(const SysArgs& A, int npts, int h_mode, long long steps, int n, int sms,
                             const double* t0, const double* t1, const double* u0, long long ld0, double* u1,
                             long long ld1, cudaStream_t st) {
  // horizontal neighbours by shuffle when a block row is a power-of-two number of consecutive lanes and every warp is full
  const int hx_ = (int)A.p[0] >> 1;
  // Measured (profiles/r02/rk_sweep_shuffle.log): by shuffle a LONE slice (<= 1 per SM, a rank of a 4-8 GPU run) steps 6 %
  // (2x2 blocks) to 11 % (1x2) faster -- the shuffles leave before the barrier and shorten the per-stage dependency chain --
  // while with several slices per SM the 16 shuffles per thread and stage cost more shared-pipe cycles than the 8 column
  // loads they replace (512 slices on one GPU: 627 vs 562 ms).  So: shuffle only when the GPU holds at most one slice per SM.
  // Re-measured with conflict-free column loads (profiles/r04/rk_layout_sweep.log, 64 and 148 slices): the shuffle form
  // still wins, 1x2 257.0 against 268.7 ms, 2x2 278.0 against 288.8 ms.
  const bool shx = getenv("NNGP_RK_NO_SHFL") == nullptr && hx_ >= 1 && hx_ <= 32 && (hx_ & (hx_ - 1)) == 0 &&
                   (npts / (2 * TY)) % 32 == 0 && n <= sms;
  if (shx) return launch_fhn_tile_x<S, TY, TB, true>(A, npts, h_mode, steps, n, sms, t0, t1, u0, ld0, u1, ld1, st);
  return launch_fhn_tile_x<S, TY, TB, false>(A, npts, h_mode, steps, n, sms, t0, t1, u0, ld0, u1, ld1, st);
}

template <int TY, int TB>
static int launch_fhn_tile(const SysArgs& A, int npts, int method, int h_mode, long long steps, int n, int sms,
                           const double* t0, const double* t1, const double* u0, long long ld0, double* u1,
                           long long ld1, cudaStream_t st) {
  switch (method) {
    case 1: return launch_fhn_tile_s<1, TY, TB>(A, npts, h_mode, steps, n, sms, t0, t1, u0, ld0, u1, ld1, st);
    case 2: return launch_fhn_tile_s<2, TY, TB>(A, npts, h_mode, steps, n, sms, t0, t1, u0, ld0, u1, ld1, st);
    case 4: return launch_fhn_tile_s<4, TY, TB>(A, npts, h_mode, steps, n, sms, t0, t1, u0, ld0, u1, ld1, st);
    default: return launch_fhn_tile_s<11, TY, TB>(A, npts, h_mode, steps, n, sms, t0, t1, u0, ld0, u1, ld1, st);
  }
}

template <class RHS>
__global__ void rhs_pde_kernel(SysArgs A, const double* __restrict__ uin,
                               double* __restrict__ out) {
  constexpr int NC = RHS::NC;
  extern __shared__ double sm[];
  const int npts = RHS::points(A);
  const int p = threadIdx.x;
  const bool active = p < npts;
  const int pp = active ? p : 0;
  const long long s = blockIdx.x;
  RHS rhs;
  rhs.setup(A, pp);
  double v[NC], f[NC], rg[NC];
#pragma unroll
  for (int c = 0; c < NC; c++) {
    const double w = uin[s * A.d + c * npts + pp];
    const double mn = A.normalize ? A.mn[c * npts + pp] : 0.0;
    rg[c] = A.normalize ? (A.mx[c * npts + pp] - A.mn[c * npts + pp]) : 2.0;
    v[c] = A.normalize ? (((w + 1.0) / 2.0) * rg[c] + mn) : w;
    if (active) sm[c * npts + p] = v[c];
  }
  __syncthreads();
  rhs.eval(A, sm, pp, v, f);
  if (active) {
#pragma unroll
    for (int c = 0; c < NC; c++)
      out[s * A.d + c * npts + p] = A.normalize ? f[c] * (2.0 / rg[c]) : f[c];
  }
}

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
SysArgs nngp_sys_args(const SystemDesc& s) {
  SysArgs A;
  A.system_id = s.system_id;
  A.d = s.d;
  A.normalize = s.normalize;
  for (int i = 0; i < NNGP_MAX_PARAMS; i++) A.p[i] = s.params[i];
  for (int i = 0; i < 4; i++) A.q[i] = 0.0;
  A.traj = nullptr;
  if (s.system_id == NNGP_SYS_FHN_PDE) {  // see FhnPde::eval_k
    A.q[0] = s.params[1] + 1.0;
    A.q[1] = s.params[4] * s.params[6];
    A.q[2] = (s.params[3] - 1.0) * s.params[6];
  }
  A.mn = s.d_mn;
  A.mx = s.d_mx;
  return A;
}

template <int SYS>
static void launch_small(const SysArgs& A, int method, int h_mode, long long steps,
                         int n, const double* t0, const double* t1, const double* u0,
                         long long ld0, double* u1, long long ld1, cudaStream_t st) {
  const int threads = 32;
  const int blocks = (n + threads - 1) / threads;
  switch (method) {
    case 1: rk_small_kernel<SYS, 1><<<blocks, threads, 0, st>>>(A, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1); break;
    case 2: rk_small_kernel<SYS, 2><<<blocks, threads, 0, st>>>(A, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1); break;
    case 4: rk_small_kernel<SYS, 4><<<blocks, threads, 0, st>>>(A, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1); break;
    default: rk_small_kernel<SYS, 11><<<blocks, threads, 0, st>>>(A, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1); break;
  }
}

template <class RHS, int TB, bool NORM>
static void launch_pde_tb(const SysArgs& A, int npts, int method, int h_mode, long long steps,
                          int n, const double* t0, const double* t1, const double* u0,
                          long long ld0, double* u1, long long ld1, cudaStream_t st) {
  const int threads = ((npts + 31) / 32) * 32;
  const size_t smem = 2 * sizeof(double) * RHS::NC * npts;
  switch (method) {
    case 1: rk_pde_kernel<RHS, 1, TB, NORM><<<n, threads, smem, st>>>(A, h_mode, steps, t0, t1, u0, ld0, u1, ld1); break;
    case 2: rk_pde_kernel<RHS, 2, TB, NORM><<<n, threads, smem, st>>>(A, h_mode, steps, t0, t1, u0, ld0, u1, ld1); break;
    case 4: rk_pde_kernel<RHS, 4, TB, NORM><<<n, threads, smem, st>>>(A, h_mode, steps, t0, t1, u0, ld0, u1, ld1); break;
    default: rk_pde_kernel<RHS, 11, TB, NORM><<<n, threads, smem, st>>>(A, h_mode, steps, t0, t1, u0, ld0, u1, ld1); break;
  }
}

template <class RHS>
static void launch_pde(const SysArgs& A, int npts, int method, int h_mode, long long steps,
                       int n, const double* t0, const double* t1, const double* u0,
                       long long ld0, double* u1, long long ld1, cudaStream_t st) {
  if (npts <= 256) {
    if (A.normalize) launch_pde_tb<RHS, 256, true>(A, npts, method, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1, st);
    else launch_pde_tb<RHS, 256, false>(A, npts, method, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1, st);
  } else {
    if (A.normalize) launch_pde_tb<RHS, 1024, true>(A, npts, method, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1, st);
    else launch_pde_tb<RHS, 1024, false>(A, npts, method, h_mode, steps, n, t0, t1, u0, ld0, u1, ld1, st);
  }
}

static int check_system(nngp_handle_t h, const SystemDesc& s, int* npts) {
  *npts = 0;
  switch (s.system_id) {
    case NNGP_SYS_FHN_ODE: case NNGP_SYS_BRUSSELATOR:
      if (s.d != 2) return nngp_fail(h, "system %d needs d=2, got %d", s.system_id, s.d);
      return 0;
    case NNGP_SYS_ROSSLER: case NNGP_SYS_HOPF: case NNGP_SYS_LORENZ: case NNGP_SYS_THOMAS:
      if (s.d != 3) return nngp_fail(h, "system %d needs d=3, got %d", s.system_id, s.d);
      return 0;
    case NNGP_SYS_DBLPEND:
      if (s.d != 4) return nngp_fail(h, "system %d needs d=4, got %d", s.system_id, s.d);
      return 0;
    case NNGP_SYS_FHN_PDE: {
      const int dx = (int)s.params[0];
      if (dx < 3 || 2 * dx * dx != s.d) return nngp_fail(h, "FHN_PDE: d=%d is not 2*d_x^2 (d_x=%d)", s.d, dx);
      if (dx * dx > 1024) return nngp_fail(h, "FHN_PDE: d_x^2=%d > 1024 grid points per CTA", dx * dx);
      *npts = dx * dx;
      return 0;
    }
    case NNGP_SYS_BURGERS:
      if (s.d < 3 || s.d > 1024) return nngp_fail(h, "Burgers: d=%d outside [3,1024]", s.d);
      *npts = s.d;
      return 0;
    default:
      return nngp_fail(h, "unknown system id %d", s.system_id);
  }
}

int rk_launch(nngp_handle_t h, const SystemDesc& s, int method, int h_mode, long long steps,
              int n_slices, const double* d_t0, const double* d_t1, const double* d_u0,
              long long ld_u0, double* d_u1, long long ld_u1, cudaStream_t st, double* d_traj) {
  const int slot = method_slot(method);
  if (slot < 0) return nngp_fail(h, "Only RK1, RK2, RK4 and RK8 are implemented (got %d)", method);
  if (steps < 1) return nngp_fail(h, "steps must be >= 1 (got %lld)", steps);
  if (h_mode != NNGP_H_LINSPACE && h_mode != NNGP_H_CONST) return nngp_fail(h, "bad h_mode %d", h_mode);
  if (n_slices <= 0) return 0;
  int npts = 0;
  if (int rc = check_system(h, s, &npts)) return rc;
  SysArgs A = nngp_sys_args(s);
  A.traj = d_traj;
  ProfScope prof(h, 0, st);
#define SMALL(SYS) launch_small<SYS>(A, method, h_mode, steps, n_slices, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st)
  switch (s.system_id) {
    case NNGP_SYS_FHN_ODE: SMALL(NNGP_SYS_FHN_ODE); break;
    case NNGP_SYS_ROSSLER: SMALL(NNGP_SYS_ROSSLER); break;
    case NNGP_SYS_HOPF: SMALL(NNGP_SYS_HOPF); break;
    case NNGP_SYS_DBLPEND: SMALL(NNGP_SYS_DBLPEND); break;
    case NNGP_SYS_BRUSSELATOR: SMALL(NNGP_SYS_BRUSSELATOR); break;
    case NNGP_SYS_LORENZ: SMALL(NNGP_SYS_LORENZ); break;
    case NNGP_SYS_THOMAS: SMALL(NNGP_SYS_THOMAS); break;
    case NNGP_SYS_FHN_PDE: {
      const int dx = (int)A.p[0];
      // NNGP_RK_TILE = 0 / 1 / 2 forces the one-point-per-thread kernel / the 2x2 blocks / the 1x2 blocks
      // (tests, experiments); default 2x2: fastest from 256 slices per GPU up and within 3 % of the 1x2
      // blocks below (a lone slice is bound by the per-stage latency chain, ~270 cycles, in every shape;
      // slice-count sweep in profiles/r01/rk_sweep.log).
      // Tried and rejected (slower): two slices per 128-thread CTA; left/right neighbours by shuffle when an SM holds
      // several slices (it wins for lone slices, see launch_fhn_tile_s).
      const char* force = getenv("NNGP_RK_TILE");
      int sms = 148;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
      // at most one slice per SM (a rank of a 4-8 GPU run): 1x2 blocks with the horizontal neighbours by shuffle are the
      // fastest lone-slice shape (257 ms per published fine step against 278 for 2x2 + shuffle, 290-295 without shuffle)
      const int hx = dx >> 1;
      int shape = (n_slices <= sms && hx >= 1 && hx <= 32 && (hx & (hx - 1)) == 0 && (npts / 2) % 32 == 0 &&
                   getenv("NNGP_RK_NO_SHFL") == nullptr) ? 1 : 2;
      if (force && force[0] >= '0' && force[0] <= '2') shape = (force[0] == '0') ? 0 : ((force[0] == '1') ? 2 : 1);
      if (!A.normalize && (dx & 1) == 0 && dx >= 4 && shape != 0) {
        int nl = 1;
        if (shape == 2) {
          if (npts / 4 <= 64)
            nl = launch_fhn_tile<2, 64>(A, npts, method, h_mode, steps, n_slices, sms, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st);
          else
            nl = launch_fhn_tile<2, 256>(A, npts, method, h_mode, steps, n_slices, sms, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st);
        } else {
          if (npts / 2 <= 128)
            nl = launch_fhn_tile<1, 128>(A, npts, method, h_mode, steps, n_slices, sms, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st);
          else
            nl = launch_fhn_tile<1, 512>(A, npts, method, h_mode, steps, n_slices, sms, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st);
        }
        h->launches += nl - 1;
      } else {
        launch_pde<FhnPde>(A, npts, method, h_mode, steps, n_slices, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st);
      }
      break;
    }
    case NNGP_SYS_BURGERS:
      launch_pde<BurgersPde>(A, npts, method, h_mode, steps, n_slices, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1, st);
      break;
  }
#undef SMALL
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

int rhs_launch(nngp_handle_t h, const SystemDesc& s, int n, const double* d_u, double* d_out,
               cudaStream_t st) {
  if (n <= 0) return 0;
  int npts = 0;
  if (int rc = check_system(h, s, &npts)) return rc;
  const SysArgs A = nngp_sys_args(s);
  const int tb = 128, nb = (n + tb - 1) / tb;
  switch (s.system_id) {
    case NNGP_SYS_FHN_ODE: rhs_small_kernel<NNGP_SYS_FHN_ODE><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_ROSSLER: rhs_small_kernel<NNGP_SYS_ROSSLER><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_HOPF: rhs_small_kernel<NNGP_SYS_HOPF><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_DBLPEND: rhs_small_kernel<NNGP_SYS_DBLPEND><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_BRUSSELATOR: rhs_small_kernel<NNGP_SYS_BRUSSELATOR><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_LORENZ: rhs_small_kernel<NNGP_SYS_LORENZ><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_THOMAS: rhs_small_kernel<NNGP_SYS_THOMAS><<<nb, tb, 0, st>>>(A, n, d_u, d_out); break;
    case NNGP_SYS_FHN_PDE: {
      const int threads = ((npts + 31) / 32) * 32;
      rhs_pde_kernel<FhnPde><<<n, threads, sizeof(double) * 2 * npts, st>>>(A, d_u, d_out);
      break;
    }
    case NNGP_SYS_BURGERS: {
      const int threads = ((npts + 31) / 32) * 32;
      rhs_pde_kernel<BurgersPde><<<n, threads, sizeof(double) * npts, st>>>(A, d_u, d_out);
      break;
    }
  }
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}
