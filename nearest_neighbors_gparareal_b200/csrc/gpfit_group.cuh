// Grouped fit kernel: SEVERAL Nelder-Mead searches per warp (included by gpfit.cu after its math helpers,
// gp_head and the Nelder-Mead constants).
//
// Why.  The one-search-per-warp kernel (gp_fit_predict_kernel) is bound by FP64 issue while executing 8.6x the
// algorithmic work of an evaluation (VERDICT round 1): 20 of 32 lanes hold rows, every lane updates the full row
// instead of its part left of the diagonal, pivots / quadratic form / determinant are accumulated in every lane.
// Here a search owns G = M/2 lanes and a warp runs NG = 32/G searches side by side (3 at the m = 20 target):
//   * lane p of a group owns the two rows p ("short") and M-1-p ("long") of the m x m kernel matrix -- together
//     M-1 off-diagonal entries left of the diagonal, the same for every lane -- so the M(M-1)/2 exponentials are
//     balanced over the lanes and land in the registers of the lane that needs them: no exchange of the matrix;
//   * the factorisation is the same right-looking square-root-free LDL^T with the same operations in the same order
//     per matrix entry as gp_core (results are bit-identical, tests/test_gpu_kernels.py), but a step costs
//     (M-1-k) + (G-1-k)^+ fused multiply-adds per WARP for NG searches instead of (M-1-k) for one;
//   * the searches of a warp advance in rounds: every group evaluates the point its own Nelder-Mead state machine
//     asks for, groups fetch their next search from the queue independently, early exits of failing
//     factorisations are taken when every group of the warp has failed.
// Selection (models.py:212-215) and the posterior mean (models.py:162-168) moved to gp_select_mean_kernel, launched
// behind the searches: one warp per (query, dimension) with the lane-per-row core gp_core<M, true>.
#pragma once

#ifdef NNGP_FIT_STATS
__device__ unsigned long long g_fail_hist[18];  // [k] first failing pivot of a wanted evaluation, [16] head failures, [17] wanted
#endif

template <int M>
struct Grp {
  static constexpr int G = M / 2;                 // lanes per search
  static constexpr int NG = 32 / G;               // searches per warp
  static constexpr int LD = Tri<M>::LD;           // row stride of a group's tile in doubles
  static constexpr int TILE = M * LD;             // column exchange tile of a group
  static constexpr int R2LD = M + 1;              // stride of a lane's slot table (M-1 used); odd: conflict-free 8-byte loads
  static constexpr int R2S = G * R2LD;            // squared distances of the group's query in slot order
  static constexpr int PER_GROUP = ((TILE + R2S + 1) / 2) * 2 + 2;  // even (16-byte aligned tiles); +2 skews the groups
  static constexpr int PER_WARP = NG * PER_GROUP;
  static constexpr int NSLOT = M - 1;
};

// exponentials of slots [T0, T0 + n) of the lane, stored to the group's tile (compile-time chunking)
template <int M, int T0>
struct BuildChunks {
  static constexpr int NS = M - 1;
  static constexpr int NCH = (NS + 7) / 8;
  static constexpr int CH = (NS + NCH - 1) / NCH;
  static constexpr int N = (NS - T0 < CH) ? (NS - T0) : CH;
  static __device__ __forceinline__ void run(double c, double amp_s, const double* __restrict__ r2s,
                                             double* __restrict__ tile, int p, int Lr, int m, bool act) {
    if constexpr (N > 0) {
      constexpr int LD = Tri<M>::LD;
      double xa[N], oa[N];
#pragma unroll
      for (int t = 0; t < N; t++) xa[t] = c * r2s[T0 + t];
      exp_neg_vec<N>(xa, oa);
#pragma unroll
      for (int t = 0; t < N; t++) {
        const bool lng = (T0 + t) < Lr;
        const int row = lng ? Lr : p, col = lng ? (T0 + t) : (T0 + t) - Lr;
        if (act) tile[row * LD + col] = (row >= m) ? 0.0 : amp_s * oa[t];
      }
      BuildChunks<M, T0 + N>::run(c, amp_s, r2s, tile, p, Lr, m, act);
    }
  }
};

struct GroupLane {
  int g, p, Lr, gbase;  // group, lane in group, long row M-1-p, first lane of the group
  bool act;             // lanes beyond NG*G mirror group 0 and never write
};

// Objective of one point per group (models.py:240-252, 86-92); `want` = the group has a point to evaluate.
// r2s: the lane's slot table (shared), tile: the group's exchange tile (shared).  All 32 lanes call it together.
template <int M>
__device__ __forceinline__ double gp_nll_grouped(double th0, double th1, double jit10, double r2_10,
                                                 const double* __restrict__ r2s, double* __restrict__ tile,
                                                 double yS, double yL, int m, const GroupLane& L, double hml,
                                                 double guard, bool want) {
  static_assert(M % 2 == 0, "M even");
  constexpr int G = Grp<M>::G, LD = Grp<M>::LD;
  const GpHead hd = gp_head(th0, th1, jit10, r2_10, m, guard);
  const double c = hd.c, sc = hd.sc, amp_s = hd.amp_s, dd0 = hd.dd0, pmin = hd.pmin;
#ifdef NNGP_FIT_STATS
  if (want && hd.fail01 && L.p == 0 && L.act) atomicAdd(g_fail_hist + 16, 1ULL);
  if (want && L.p == 0 && L.act) atomicAdd(g_fail_hist + 17, 1ULL);
#endif
  if (__all_sync(FULL, hd.fail01 || !want)) return dinf();
  const int p = L.p, Lr = L.Lr;
  // kernel entries of the lane's two rows: slot t < Lr -> (row Lr, col t), else (row p, col t - Lr);
  // exponentials interleaved in chunks of at most 8
  BuildChunks<M, 0>::run(c, amp_s, r2s, tile, p, Lr, m, L.act);
  __syncwarp();
  double aL[M], aS[G];
  {
    const double2* rl = reinterpret_cast<const double2*>(tile + Lr * LD);
#pragma unroll
    for (int j = 0; j < M; j += 2) {
      const double2 t2 = rl[j >> 1];
      aL[j] = (j < Lr) ? t2.x : 0.0;
      aL[j + 1] = (j + 1 < Lr) ? t2.y : 0.0;
    }
    const double2* rs = reinterpret_cast<const double2*>(tile + p * LD);
#pragma unroll
    for (int j = 0; j < G; j += 2) {
      const double2 t2 = rs[j >> 1];
      aS[j] = (j < p) ? t2.x : 0.0;
      if (j + 1 < G) aS[j + 1] = (j + 1 < p) ? t2.y : 0.0;
    }
  }
  __syncwarp();  // the tile is reused for the column broadcasts below
  auto load_col = [&](int k, double (&u)[M]) {
    int j = k + 1;
    if (j < M && (j & 1)) {
      u[j] = tile[k * LD + j];
      j++;
    }
#pragma unroll
    for (; j + 1 < M; j += 2) {
      const double2 u2 = *reinterpret_cast<const double2*>(&tile[k * LD + j]);
      u[j] = u2.x;
      u[j + 1] = u2.y;
    }
  };
  double ddS = dd0, ddL = dd0;
  double zS = (p < m) ? yS : 0.0, zL = (Lr < m) ? yL : 0.0;
  double quad = 0.0, prod0 = 1.0, prod1 = 1.0;
  bool ok = true;
  double u[M];
  // pivot 0 is the short row of lane 0 of the group
  double pv = __shfl_sync(FULL, ddS, L.gbase), zk = __shfl_sync(FULL, zS, L.gbase);
  // column 0: entries a_r0 of every row r > 0
  if (L.act) {
    if (p > 0) tile[p] = aS[0];
    tile[Lr] = aL[0];
  }
  __syncwarp();
  load_col(0, u);
#pragma unroll
  for (int k = 0; k < M; k++) {
#ifdef NNGP_FIT_STATS
    if (ok && !(pv > pmin) && want && L.p == 0 && L.act) atomicAdd(g_fail_hist + (k < 15 ? k : 15), 1ULL);
#endif
    ok = ok && (pv > pmin);
#ifndef NNGP_FIT_STATS
    if ((k == 1 || k == 2 || k == 4 || k == 8 || k == 14) && k < M - 1) {
      if (__all_sync(FULL, !ok || !want)) {
        __syncwarp();
        return dinf();
      }
    }
#endif
    const double ip = rcp_pos(pv);
    const double pk = pv, zkk = zk;
    // long row (exists in every lane; entries right of its diagonal are kept at zero, so w = 0 once k >= Lr)
    const double wL = aL[k] * ip;
    ddL = fma(-wL, aL[k], ddL);
    zL = fma(-wL, zk, zL);
    double wS = 0.0;
    if (k < G - 1) {
      wS = aS[k] * ip;
      ddS = fma(-wS, aS[k], ddS);
      zS = fma(-wS, zk, zS);
    }
    if (k + 1 < M) {
      // the lanes' entries of the next pivot column first, then the next pivot
      aL[k + 1] = fma(-wL, u[k + 1], aL[k + 1]);
      if (k + 1 < G) aS[k + 1] = fma(-wS, u[k + 1], aS[k + 1]);
      const int owner = (k + 1 < G) ? (k + 1) : (M - 2 - k);  // lane (in group) owning row k+1
      pv = __shfl_sync(FULL, (k + 1 < G) ? ddS : ddL, L.gbase + owner);
      zk = __shfl_sync(FULL, (k + 1 < G) ? zS : zL, L.gbase + owner);
      if (k + 2 < M) {
        if (k + 1 < G && p > k + 1 && L.act) tile[(k + 1) * LD + p] = aS[k + 1];
        if (Lr > k + 1 && L.act) tile[(k + 1) * LD + Lr] = aL[k + 1];
        __syncwarp();
      }
#pragma unroll
      for (int j = k + 2; j < M; j++) aL[j] = fma(-wL, u[j], aL[j]);
#pragma unroll
      for (int j = k + 2; j < G; j++) aS[j] = fma(-wS, u[j], aS[j]);
      if (k + 2 < M) load_col(k + 1, u);
    }
    quad = fma(zkk * zkk, ip, quad);
    if (k < M / 2) prod0 = prod0 * pk; else prod1 = prod1 * pk;
  }
  if (m < M) {
    const double id0 = rcp_pos(dd0);
    for (int r = m; r < M; r++) {
      if (r < M / 2) prod0 = prod0 * id0; else prod1 = prod1 * id0;
    }
  }
  __syncwarp();  // the next evaluation overwrites the tile
  const int h0 = __double2hiint(prod0), h1 = __double2hiint(prod1);
  const double m0 = __hiloint2double((h0 & 0x000fffff) | 0x3ff00000, __double2loint(prod0));
  const double m1 = __hiloint2double((h1 & 0x000fffff) | 0x3ff00000, __double2loint(prod1));
  const int e0 = 1023 - ((__double2hiint(sc) >> 20) & 0x7ff);
  const int esum = (h0 >> 20) + (h1 >> 20) - 2046 + m * e0;
  const double res = fma(0.5, fma(quad, sc, log_pos_plus(m0 * m1, esum)), hml);
  return (want && ok && res == res) ? res : dinf();
}

// ---- Nelder-Mead as a step function (same decisions as nelder_mead<M> above; SciPy semantics) --------------
struct NMState {
  double sx[3][2], sf[3];
  double p0, p1;            // point to evaluate next
  double xb0, xb1, xr0, xr1, fxr;
  double cx0[4], cx1[4];    // the four points of an all-inf iteration (reflection, inside contraction, 2 shrinks)
  unsigned cmask;           // which of them are known to fail at pivots 0 / 1
  int fcalls, it, phase;
  bool want_heads;          // a new all-inf iteration started: cmask has to be recomputed
};

__device__ __forceinline__ void nm_init(NMState& S, double s0, double s1) {
  S.sx[0][0] = s0; S.sx[0][1] = s1;
  S.sx[1][0] = (s0 != 0.0) ? __dmul_rn(1.05, s0) : 0.00025; S.sx[1][1] = s1;
  S.sx[2][0] = s0; S.sx[2][1] = (s1 != 0.0) ? __dmul_rn(1.05, s1) : 0.00025;
  S.sf[0] = S.sf[1] = S.sf[2] = dinf();
  S.fcalls = 0; S.it = 1; S.phase = PH_INIT0;
  S.p0 = s0; S.p1 = s1;
  S.xb0 = S.xb1 = S.xr0 = S.xr1 = S.fxr = 0.0;
  S.cmask = 0; S.want_heads = false;
#pragma unroll
  for (int j = 0; j < 4; j++) S.cx0[j] = S.cx1[j] = 0.0;
}

// consumes the objective value f of the pending point; returns true when the search has ended
__device__ __forceinline__ bool nm_step(NMState& S, double f, double fatol, double xatol, bool head_batch) {
  const int maxfun = 400, maxiter = 400;
  S.fcalls++;
  S.want_heads = false;
  bool aborted = false, do_shrink = false;
  const double p0 = S.p0, p1 = S.p1;
  if (S.phase == PH_INIT0) {
    S.sf[0] = f; S.phase = PH_INIT1; S.p0 = S.sx[1][0]; S.p1 = S.sx[1][1];
    return false;
  }
  if (S.phase == PH_INIT1) {
    S.sf[1] = f; S.phase = PH_INIT2; S.p0 = S.sx[2][0]; S.p1 = S.sx[2][1];
    return false;
  }
  const bool initial = (S.phase == PH_INIT2);
  if (initial) {
    S.sf[2] = f;
  } else if (S.phase == PH_REFLECT) {
    S.fxr = f;
    int nphase = -1;
    double q0 = 0, q1 = 0;
    const double w0 = S.sx[2][0], w1 = S.sx[2][1];
    if (f < S.sf[0]) {
      q0 = __dsub_rn(__dmul_rn(3.0, S.xb0), __dmul_rn(2.0, w0));
      q1 = __dsub_rn(__dmul_rn(3.0, S.xb1), __dmul_rn(2.0, w1));
      nphase = PH_EXPAND;
    } else if (f < S.sf[1]) {
      S.sx[2][0] = S.xr0; S.sx[2][1] = S.xr1; S.sf[2] = f;
    } else if (f < S.sf[2]) {
      q0 = __dsub_rn(__dmul_rn(1.5, S.xb0), __dmul_rn(0.5, w0));
      q1 = __dsub_rn(__dmul_rn(1.5, S.xb1), __dmul_rn(0.5, w1));
      nphase = PH_OUTC;
    } else {
      q0 = __dadd_rn(__dmul_rn(0.5, S.xb0), __dmul_rn(0.5, w0));
      q1 = __dadd_rn(__dmul_rn(0.5, S.xb1), __dmul_rn(0.5, w1));
      nphase = PH_INC;
    }
    if (nphase >= 0) {
      if (S.fcalls >= maxfun) {
        aborted = true;
      } else {
        S.phase = nphase; S.p0 = q0; S.p1 = q1;
        return false;
      }
    }
  } else if (S.phase == PH_EXPAND) {
    if (f < S.fxr) { S.sx[2][0] = p0; S.sx[2][1] = p1; S.sf[2] = f; }
    else { S.sx[2][0] = S.xr0; S.sx[2][1] = S.xr1; S.sf[2] = S.fxr; }
  } else if (S.phase == PH_OUTC) {
    if (f <= S.fxr) { S.sx[2][0] = p0; S.sx[2][1] = p1; S.sf[2] = f; }
    else do_shrink = true;
  } else if (S.phase == PH_INC) {
    if (f < S.sf[2]) { S.sx[2][0] = p0; S.sx[2][1] = p1; S.sf[2] = f; }
    else do_shrink = true;
  } else if (S.phase == PH_SHRINK1) {
    S.sf[1] = f;
    S.sx[2][0] = shrink_to(S.sx[0][0], S.sx[2][0]);
    S.sx[2][1] = shrink_to(S.sx[0][1], S.sx[2][1]);
    if (S.fcalls >= maxfun) {
      aborted = true;
    } else {
      S.phase = PH_SHRINK2; S.p0 = S.sx[2][0]; S.p1 = S.sx[2][1];
      return false;
    }
  } else {  // PH_SHRINK2
    S.sf[2] = f;
  }
  if (do_shrink) {
    S.sx[1][0] = shrink_to(S.sx[0][0], S.sx[1][0]);
    S.sx[1][1] = shrink_to(S.sx[0][1], S.sx[1][1]);
    if (S.fcalls >= maxfun) {
      aborted = true;
    } else {
      S.phase = PH_SHRINK1; S.p0 = S.sx[1][0]; S.p1 = S.sx[1][1];
      return false;
    }
  }
  if (!initial && !aborted) S.it++;
  sort3(S.sx, S.sf);
  if (!(S.fcalls < maxfun && S.it < maxiter)) return true;
  {
    const double d10 = fabs(__dsub_rn(S.sx[1][0], S.sx[0][0])), d11 = fabs(__dsub_rn(S.sx[1][1], S.sx[0][1]));
    const double d20 = fabs(__dsub_rn(S.sx[2][0], S.sx[0][0])), d21 = fabs(__dsub_rn(S.sx[2][1], S.sx[0][1]));
    const double f1 = fabs(__dsub_rn(S.sf[0], S.sf[1])), f2 = fabs(__dsub_rn(S.sf[0], S.sf[2]));
    if (d10 <= xatol && d11 <= xatol && d20 <= xatol && d21 <= xatol && f1 <= fatol && f2 <= fatol) return true;
  }
  S.xb0 = __dmul_rn(__dadd_rn(S.sx[0][0], S.sx[1][0]), 0.5);
  S.xb1 = __dmul_rn(__dadd_rn(S.sx[0][1], S.sx[1][1]), 0.5);
  S.xr0 = __dsub_rn(__dmul_rn(2.0, S.xb0), S.sx[2][0]);
  S.xr1 = __dsub_rn(__dmul_rn(2.0, S.xb1), S.sx[2][1]);
  S.phase = PH_REFLECT; S.p0 = S.xr0; S.p1 = S.xr1;
  S.cmask = 0;
  if (head_batch && S.sf[0] == dinf()) {
    S.cx0[0] = S.xr0; S.cx1[0] = S.xr1;
    S.cx0[1] = __dadd_rn(__dmul_rn(0.5, S.xb0), __dmul_rn(0.5, S.sx[2][0]));
    S.cx1[1] = __dadd_rn(__dmul_rn(0.5, S.xb1), __dmul_rn(0.5, S.sx[2][1]));
    S.cx0[2] = shrink_to(S.sx[0][0], S.sx[1][0]); S.cx1[2] = shrink_to(S.sx[0][1], S.sx[1][1]);
    S.cx0[3] = shrink_to(S.sx[0][0], S.sx[2][0]); S.cx1[3] = shrink_to(S.sx[0][1], S.sx[2][1]);
    S.want_heads = true;
  }
  return false;
}

template <int M> struct GrpOcc { static constexpr int value = (M <= 12) ? 4 : 2; };

// searches only: res[task] = (fval, theta0, theta1); selection and mean follow in gp_select_mean_kernel
template <int M>
__global__ void __launch_bounds__(GP_WARPS * 32, GrpOcc<M>::value)
gp_fit_grouped_kernel(FitArgs A) {
  extern __shared__ double sm[];
  constexpr int G = Grp<M>::G, NG = Grp<M>::NG;
  const int m = A.m, d = A.d, R = A.R, nruns = NNGP_N_JITTER * R;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  GroupLane L;
  L.act = lane < NG * G;
  L.g = L.act ? lane / G : 0;
  L.p = L.act ? lane - L.g * G : lane - NG * G;
  L.Lr = M - 1 - L.p;
  L.gbase = L.g * G;
  double* gsm = sm + (size_t)w * Grp<M>::PER_WARP + (size_t)L.g * Grp<M>::PER_GROUP;
  double* tile = gsm;
  double* r2grp = gsm + Grp<M>::TILE;
  double* r2s = r2grp + L.p * Grp<M>::R2LD;
  // lanes beyond NG*G (2 at M = 20) mirror lanes of group 0: they take part in the shuffles and votes, read group
  // 0's tile, and never store, fetch or write results
  const double hml = (m / 2.0) * 1.8378770664093453;
  const bool head_batch = (A.head_batch != 0) && (G >= 4);
  NMState S;
  nm_init(S, -1.0, -1.0);
  bool busy = false, exhausted = !L.act;
  int task = 0, q_loaded = -1, run_a = 0;
  long long gtask = 0;
  double yS = 0.0, yL = 0.0, r2_10 = 0.0, jit10 = 1e-20;
#ifdef NNGP_FIT_STATS
  unsigned long long st_rounds = 0, st_want = 0, st_ff = 0, st_busy = 0;
#endif
  for (;;) {
    const bool need = !busy && !exhausted;
    if (__any_sync(FULL, need)) {
      int t = -1;
      if (need && L.p == 0) {
        const unsigned pos = atomicAdd(A.queue, 1u);
        t = (pos < (unsigned)A.ntasks) ? (A.order ? A.order[pos] : (int)pos) : -1;
      }
      t = __shfl_sync(FULL, t, L.gbase);
      int qn = -1;
      if (need) {
        if (t < 0) {
          exhausted = true;
        } else {
          task = t;
          const int qj = task / nruns, run = task - qj * nruns;
          const int q = qj / A.dl, j = A.j0 + (qj - q * A.dl);
          const long long gqj = (long long)q * d + j;
          gtask = gqj * nruns + run;
          run_a = run / R;
          jit10 = c_jit10[run_a];
          const long long* idx = A.idx + (long long)q * m;
          yS = (L.p < m) ? A.Y[idx[L.p] * d + j] : 0.0;
          yL = (L.Lr < m) ? A.Y[idx[L.Lr] * d + j] : 0.0;
          const signed char* st = A.starts + gtask * 2;
          nm_init(S, (double)st[0], (double)st[1]);
          busy = true;
          if (q != q_loaded) qn = q;
        }
      }
      if (__any_sync(FULL, qn >= 0)) {
        if (qn >= 0) {  // squared distances of the lane's entries, slot order
          const double* r2 = A.r2 + (long long)qn * m * m;
#pragma unroll 1
          for (int s = 0; s < Grp<M>::NSLOT; s++) {
            const bool lng = s < L.Lr;
            const int row = lng ? L.Lr : L.p, col = lng ? s : s - L.Lr;
            r2s[s] = (row < m) ? __ldg(r2 + row * m + col) : 0.0;
          }
          r2_10 = (m > 1) ? __ldg(r2 + m) : 0.0;
          q_loaded = qn;
        }
        __syncwarp();
      }
    }
    if (!__any_sync(FULL, busy)) break;
    bool hit = false;
    if (busy && S.cmask) {
#pragma unroll
      for (int jj = 0; jj < 4; jj++)
        hit = hit || (((S.cmask >> jj) & 1u) && S.p0 == S.cx0[jj] && S.p1 == S.cx1[jj]);
    }
    const bool want = busy && !hit;
#ifdef NNGP_FIT_STATS
    st_rounds++;
    st_want += __popc(__ballot_sync(FULL, want && L.p == 0 && L.act));
    st_busy += __popc(__ballot_sync(FULL, busy && L.p == 0 && L.act));
#endif
    double f = gp_nll_grouped<M>(S.p0, S.p1, jit10, r2_10, r2s, tile, yS, yL, m, L, hml, A.guard, want);
    if (hit) f = dinf();
    bool fin = false;
    if (busy) fin = nm_step(S, f, A.fatol, A.xatol, head_batch);
    if (busy && !fin && S.want_heads) {
      // Every vertex of this group's simplex is +inf (identical neighbour rows at a steady state: 14 % of the
      // searches of the FHN target, each running SciPy's full 400 evaluations).  The iteration that starts now
      // evaluates four points known in advance (reflection, inside contraction, two shrunk vertices); whether each
      // fails at pivots 0 / 1 is decided by gp_head alone, here in four lanes of the group at once.  While all
      // four fail, the iteration is replayed through nm_step with f = +inf -- same decisions, no factorisation --
      // and the group does not hold the other searches of the warp to 400 full-price rounds.  Runs under
      // divergence: the vote is over the lanes of this group only.
      const unsigned gmask = ((G == 32) ? 0xffffffffu : ((1u << G) - 1u)) << L.gbase;
      for (;;) {
        const int jl = L.p & 3;
        const double t0 = (jl == 0) ? S.cx0[0] : (jl == 1) ? S.cx0[1] : (jl == 2) ? S.cx0[2] : S.cx0[3];
        const double t1 = (jl == 0) ? S.cx1[0] : (jl == 1) ? S.cx1[1] : (jl == 2) ? S.cx1[2] : S.cx1[3];
        const unsigned b = __ballot_sync(gmask, gp_head(t0, t1, jit10, r2_10, m, A.guard).fail01);
        const unsigned cm = (b >> L.gbase) & 0xFu;
        if (cm != 0xFu) {
          S.cmask = cm;
          break;
        }
        for (int e = 0; e < 4 && !fin; e++) fin = nm_step(S, dinf(), A.fatol, A.xatol, head_batch);
#ifdef NNGP_FIT_STATS
        if (L.p == 0) st_ff++;
#endif
        if (fin || !S.want_heads) break;
      }
    }
    if (fin) {
      if (L.p == 0 && L.act) {
        const double fbest = fmin(fmin(S.sf[0], S.sf[1]), S.sf[2]);
        A.res[(long long)task * 3] = fbest;
        A.res[(long long)task * 3 + 1] = S.sx[0][0];
        A.res[(long long)task * 3 + 2] = S.sx[0][1];
        atomicAdd(A.counters, 1ULL);
        atomicAdd(A.counters + 1, (unsigned long long)S.fcalls);
        if (A.nfev) A.nfev[gtask] = S.fcalls;
        if (A.fvals) A.fvals[gtask] = fbest;
        if (A.thetas) {
          A.thetas[gtask * 2] = S.sx[0][0];
          A.thetas[gtask * 2 + 1] = S.sx[0][1];
        }
      }
      busy = false;
    }
  }
#ifdef NNGP_FIT_STATS
  if (lane == 0) {
    atomicAdd(A.counters + 2, st_rounds);
    atomicAdd(A.counters + 3, st_want);
    atomicAdd(A.counters + 4, st_busy);
    atomicMax(A.counters + 6, st_rounds);
  }
  if (L.p == 0 && L.act) atomicAdd(A.counters + 5, st_ff);
#endif
}

// selection rule + posterior mean per (query, dimension) of the launch: one warp each, lane-per-row core
template <int M>
__global__ void __launch_bounds__(GP_WARPS * 32)
gp_select_mean_kernel(FitArgs A, int nqj) {
  extern __shared__ double sm[];
  const int m = A.m, d = A.d, R = A.R, nruns = NNGP_N_JITTER * R;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double* Lt = sm + w * (M * (M + 2));
  const int qj = blockIdx.x * GP_WARPS + w;
  if (qj >= nqj) return;
  const int q = qj / A.dl, j = A.j0 + (qj - q * A.dl);
  const long long gqj = (long long)q * d + j;
  const double* rf = A.res + (long long)qj * nruns * 3;
  // models.py:212-215: mask = fval < 0.9*min; empty mask -> all; first minimum in task order
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
  PairSlots<M> P;
  pair_slots_init<M>(P, lane, m);
  pair_slots_load<M>(P, A.r2 + (long long)q * m * m, m);
  const double y = (lane < m) ? A.Y[A.idx[(long long)q * m + lane] * d + j] : 0.0;
  const double kq = (lane < m) ? A.dist[(long long)q * m + lane] : 0.0;
  double mean = posterior_mean<M>(th0, th1, c_jit10[ab], P, y, kq, m, lane, Lt, A.guard);
  if (lane == 0) {
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
