/*
 * nngpara.h -- C ABI of libnngpara.so: the B200 (sm_100a) implementation of one
 * nnGParareal iteration's hot path (batched explicit Runge-Kutta propagators,
 * FP64 nearest-neighbour search over the accumulated (U, F-G) dataset, per-slice /
 * per-dimension Gaussian-process fit + predict, and the fused on-device sweep).
 *
 * The reference (Parallel-in-Time-Differential-Equations/Nearest-Neighbors-GParareal)
 * is pure Python and has no FFI; the path sits behind four duck-typed Python
 * protocols (SURVEY.md section 8b).  Each entry point below cites the reference
 * interface it replaces (file:line in the reference tree).  INTEGRATION.md shows the
 * ctypes binding a maintainer would add on the reference side.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; nngp_last_error() gives the text;
 *   - no exceptions, Python objects or torch types cross this boundary;
 *   - arrays are dense row-major FP64 unless stated; indices are int64;
 *   - names starting with d_ are DEVICE pointers on the handle's device, all others
 *     are HOST pointers; `stream` is a cudaStream_t passed as void* (NULL = default);
 *   - device-pointer entry points only enqueue work on `stream`; the *_host variants
 *     copy host<->device through the handle's pinned staging buffers and synchronise;
 *   - buffers are caller-owned; the handle owns its workspace, dataset and systems;
 *   - a handle is bound to one device and is not thread-safe: one handle per rank.
 */
#ifndef NNGPARA_H_
#define NNGPARA_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nngp_handle_s* nngp_handle_t;

#define NNGP_ABI_VERSION 2
#define NNGP_MAX_NEIGHBOURS 32 /* m <= 32: one lane per neighbour row (the fast kernels) */
#define NNGP_MAX_NEIGHBOURS_BIG 160 /* 32 < m <= 160 (nn='adaptive' past iteration 30): one CTA per search, matrix in shared memory */
#define NNGP_N_JITTER 9        /* models.py:186  jitter = arange(-20,-11) */

/* system ids: the vector fields of systems.py */
enum {
  NNGP_SYS_FHN_ODE = 0,     /* systems.py:80-106   params: -                          */
  NNGP_SYS_ROSSLER = 1,     /* systems.py:109-137                                     */
  NNGP_SYS_HOPF = 2,        /* systems.py:140-172  params: [maxtime]                  */
  NNGP_SYS_DBLPEND = 3,     /* systems.py:175-199                                     */
  NNGP_SYS_BRUSSELATOR = 4, /* systems.py:202-222                                     */
  NNGP_SYS_LORENZ = 5,      /* systems.py:225-247                                     */
  NNGP_SYS_THOMAS = 6,      /* systems.py:250-288                                     */
  NNGP_SYS_FHN_PDE = 7,     /* systems.py:291-398  params: [d_x, a*diag, a*off, b*diag, b*off, k, 1/tau] */
  NNGP_SYS_BURGERS = 8      /* systems.py:402-459  params: [Dxx_off, Dxx_diag, Dx_off] */
};

/* RK step-size convention */
enum {
  NNGP_H_LINSPACE = 0, /* RK.py:91-99,113-137 (NumPy path): h_n = t[n+1]-t[n], t = linspace */
  NNGP_H_CONST = 1     /* RK.py:101-106,146-174 (JAX path): h = (t1-t0)/steps               */
};

/* ---- lifecycle -------------------------------------------------------------------- */
int nngp_abi_version(void);
int nngp_create(int device, nngp_handle_t* out);
int nngp_destroy(nngp_handle_t h);
const char* nngp_last_error(nngp_handle_t h); /* h may be NULL: last error of a failed create */
int nngp_synchronize(nngp_handle_t h, void* stream);
/* FP64 FMA and copy-bandwidth microbenchmarks (roofline denominators; seconds per launch). */
int nngp_bench_fp64(nngp_handle_t h, int iters, double* tflops_out);
int nngp_bench_copy(nngp_handle_t h, long long bytes, double* gbs_out);

/* ---- systems: ODE.get_vector_field() + Normalize  (systems.py:32-44, utils.py:14-33) --- */
/* normalize: 0 identity, 1 '-11' (mn, mx host arrays of length d; may be NULL when 0). */
int nngp_system_create(nngp_handle_t h, int system_id, int d, const double* params, int n_params,
                       int normalize, const double* mn, const double* mx, int* sys_out);
/* f(t,u) for n state vectors: the `f` returned by ODE.get_vector_field (systems.py:32-44). */
int nngp_rhs_eval(nngp_handle_t h, int sys, int n, const double* d_u, double* d_out, void* stream);
int nngp_rhs_eval_host(nngp_handle_t h, int sys, int n, const double* u, double* out);

/* ---- propagators: RK.run_get_last (RK.py:101-109) for n_slices independent slices ----
 * replaces the task farm `pool.map(solver.run_F_timed, ...)` of parareal.py:311 (one launch
 * instead of N-I pickled tasks) and SolverRK.run_F / run_G (solver.py:102-107).
 * method: 1,2,4,8 (RK.py:30-48).  u0 rows are ld_u0 doubles apart, u1 rows ld_u1 apart. */
int nngp_rk_batch(nngp_handle_t h, int sys, int method, int h_mode, long long steps, int n_slices,
                  const double* d_t0, const double* d_t1, const double* d_u0, long long ld_u0,
                  double* d_u1, long long ld_u1, void* stream);
int nngp_rk_batch_host(nngp_handle_t h, int sys, int method, int h_mode, long long steps,
                       int n_slices, const double* t0, const double* t1, const double* u0,
                       double* u1);
/* Every step of the solve: RK.run (RK.py:91-99), what SolverRK.run_F_full / run_G_full return (solver.py:109-113).
 * d_traj[n_slices][steps+1][d] (row 0 = u0); the host variant solves one slice, traj[steps+1][d]. */
int nngp_rk_full(nngp_handle_t h, int sys, int method, int h_mode, long long steps, int n_slices,
                 const double* d_t0, const double* d_t1, const double* d_u0, long long ld_u0, double* d_traj,
                 void* stream);
int nngp_rk_full_host(nngp_handle_t h, int sys, int method, int h_mode, long long steps, double t0, double t1,
                      const double* u0, double* traj);
/* the Butcher tableau the kernels use (a[S*S] row-major, b[S], c[S]); RK.py:30-48 */
int nngp_get_tableau(int method, int* stages, double* a, double* b, double* c);

/* ---- dataset: x / D of parareal.py:336-339, held on the device ------------------------ */
int nngp_dataset_reserve(nngp_handle_t h, long long cap_rows, int d);
int nngp_dataset_reset(nngp_handle_t h);
/* keep only the first `rows` rows (a resumed / replayed iteration appends its rows again) */
int nngp_dataset_truncate(nngp_handle_t h, long long rows);
int nngp_dataset_append(nngp_handle_t h, const double* d_x, const double* d_y, long long rows,
                        void* stream);
int nngp_dataset_append_host(nngp_handle_t h, const double* x, const double* y, long long rows);
long long nngp_dataset_rows(nngp_handle_t h);
int nngp_dataset_dim(nngp_handle_t h);

/* ---- kNN: argsort(cdist(q, x, 'sqeuclidean'))[:m]  (models.py:177-179) ------------------
 * idx[nq,m] ascending in (distance, index); dist[nq,m] the squared distances, summed
 * strictly left-to-right without FMA like SciPy's cdist. Uses the first `n_rows` dataset
 * rows (n_rows<=0: all). */
int nngp_knn(nngp_handle_t h, const double* d_q, int nq, int m, long long n_rows,
             long long* d_idx, double* d_dist, void* stream);
int nngp_knn_host(nngp_handle_t h, const double* q, int nq, int m, long long n_rows,
                  long long* idx, double* dist);

/* ---- GP fit + predict: NNGP_p.get_preds (models.py:185-226) ---------------------------
 * For each query and each output dimension j: 9*R Nelder-Mead searches of the GP negative
 * log marginal likelihood (models.py:228-260, 86-92) from the host-drawn integer starts
 * d_starts[nq,d,9,R,2] (int8, models.py:192), selection (models.py:212-215) and posterior
 * mean (models.py:162-168).  Optional outputs may be NULL.
 *   pred[nq,d]  theta_opt[nq,d,2]  jitter_opt[nq,d] (log10)  fval_opt[nq,d]
 *   nfev[nq,d,9,R] (int32)  fvals[nq,d,9,R]  thetas[nq,d,9,R,2]                         */
int nngp_fit_predict(nngp_handle_t h, const double* d_q, const long long* d_idx,
                     const double* d_dist, int nq, int m, int n_restarts,
                     const signed char* d_starts, double fatol, double xatol, double* d_pred,
                     double* d_theta_opt, double* d_jitter_opt, double* d_fval_opt, int* d_nfev,
                     double* d_fvals, double* d_thetas, void* stream);
/* kNN + fit + predict with host buffers: what NNGP_p.predict (models.py:171-183) does. */
int nngp_predict_host(nngp_handle_t h, const double* q, int nq, int m, long long n_rows,
                      int n_restarts, const signed char* starts, double fatol, double xatol,
                      double* pred, long long* idx, double* theta_opt, double* jitter_opt,
                      double* fval_opt, int* nfev, double* fvals, double* thetas);
/* One rank's share of a predict: the same, fits only for the output dimensions [j0, j0+dl) of a single query
 * (dl < 0: all); pred / theta_opt / ... are written for those dimensions only.  `pred` may be a host or a device
 * pointer (copied with cudaMemcpyDefault): ranks that all-gather their blocks keep it on the device.        */
int nngp_predict_host_block(nngp_handle_t h, const double* q, int nq, int m, long long n_rows,
                            int n_restarts, const signed char* starts, double fatol, double xatol, int j0, int dl,
                            double* pred, long long* idx, double* theta_opt, double* jitter_opt,
                            double* fval_opt, int* nfev, double* fvals, double* thetas);
/* GP inputs of host-chosen neighbour lists (the listed prep of the listed sweeps, one launch): for query q (row stride
 * ld_q) and the m dataset rows d_rows[q, 0..m) (rows ld >= m apart; any order, repeats allowed),
 * dist[q, a] = ||x_rows[a] - q||^2 and r2[q, a, b] = ||x_rows[a] - x_rows[b]||^2 (rows ld apart, matrices ld x ld,
 * leading m x m block written), summed strictly left to right without FMA like nngp_knn and the fit's matrix. */
int nngp_listed_prep(nngp_handle_t h, const double* d_q, long long ld_q, int nq, int m, const long long* d_rows, int ld,
                     double* d_dist, double* d_r2, void* stream);
/* objective only: nll[nq,d,nt] at theta[nq,d,nt,2], jitter10[nq,d,nt] (= 10**jitter), the
 * `log_lik` of models.py:240-252 (+inf where the reference returns inf). */
int nngp_gp_nll(nngp_handle_t h, const long long* d_idx, int nq, int m, int nt,
                const double* d_theta, const double* d_jitter10, double* d_nll, void* stream);
/* posterior mean at given hyper-parameters (models.py:162-168): theta[nq,d,2], jitter (log10). */
int nngp_gp_mean(nngp_handle_t h, const double* d_q, const long long* d_idx, const double* d_dist,
                 int nq, int m, const double* d_theta, const double* d_jitter, double* d_pred,
                 void* stream);

/* Failure rule of the m x m factorisation (models.py:86-92 reach LAPACK potrf, whose failure becomes NaN ->
 * objective +inf, models.py:250-251): a pivot <= ulps * 2^-52 * K_rr, <= 0 or NaN fails.  Default 1 ulp (the
 * unbiased match of LAPACK's failure set, DESIGN.md section 2); 4 = the rule of the first release; values
 * below 2^-10 are clamped.  Environment override at nngp_create: NNGP_PIVOT_GUARD_ULPS.                  */
int nngp_set_pivot_guard(nngp_handle_t h, double ulps);
double nngp_get_pivot_guard(nngp_handle_t h);
/* Which search kernel nngp_fit_predict / nngp_predict_host / nngp_sweep launch: 0 auto (default), 1 one Nelder-Mead
 * search per warp, 2 several searches per warp (32 / (m/2)), 3 four warps per search (the candidate points of an
 * iteration evaluated side by side: for launches with fewer searches than warp slots, i.e. the dimension-sharded
 * sweep).  Results are bit-identical; only the speed differs (DESIGN.md section 4.5).
 * Environment override at nngp_create: NNGP_FIT_MODE=auto|warp|grouped|quad.                                    */
int nngp_set_fit_mode(nngp_handle_t h, int mode);
/* One-search-per-warp kernel only: a search still running after `evaluations` objective evaluations (0 = never, the default:
 * the continuation did not pay in the measurements of profiles/r02/fit_kernel_variants.log)
 * is continued by a second kernel in which the four warps of a CTA evaluate the candidate points of a Nelder-Mead iteration
 * side by side -- same decisions and bits, half the serial latency of the searches that end a launch.  NNGP_FIT_BUDGET. */
int nngp_set_fit_budget(nngp_handle_t h, int evaluations);

/* ---- fused on-device sweep: parareal.py:359-382 for slices i = I..N-1 -------------------
 * per slice: uG_next[i+1] = G(t_i, t_{i+1}, u_next[i]); kNN of u_next[i]; fit+predict;
 * u_next[i+1] = pred + uG_next[i+1].  No host round trip inside; d_starts holds the starts of
 * all N-I predicts in call order [(N-I), d, 9, R, 2].  d_t[N+1] slice boundaries.
 * The whole-range, all-dimension case of nngp_sweep_shard (i_first = I, i_count = N-I, j0 = 0, dl = d). */
int nngp_sweep(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g,
               const double* d_t, int N, int I, int m, int n_restarts,
               const signed char* d_starts, double fatol, double xatol, double* d_u_next,
               double* d_uG_next, int d, void* stream);
/* One rank's share of the same sweep (SURVEY.md section 8e, optional sharding of the d*9*R fits of a predict by
 * output dimension): slices i_first .. i_first+i_count-1 of the sweep that starts at slice I; G and kNN in full,
 * fits and u_next[i+1] only for dimensions [j0, j0+dl).  The caller all-gathers row i+1 of u_next over the ranks
 * (d/W doubles each) before the next slice; results are bit-identical to nngp_sweep.  So a block dl < d takes
 * i_count = 1 (rejected otherwise); with dl = d any range of slices is swept in one call.                     */
int nngp_sweep_shard(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g,
                     const double* d_t, int N, int I, int i_first, int i_count, int m, int n_restarts,
                     const signed char* d_starts, double fatol, double xatol, double* d_u_next,
                     double* d_uG_next, int d, int j0, int dl, void* stream);
/* nngp_sweep_shard for the position-based neighbour rules of the time-aware study (nnGPara_with_time.py:27-184,
 * models_alt.py): the m neighbours of the predict at slice i are the dataset rows rows[(i - I) m .. + m) that the host
 * chose, not the m nearest.  rows[(N-I), m] (host, int64, every row in [0, dataset rows), 1 <= m <= 160) covers the
 * whole sweep; a call reads the lists of its slices i_first .. i_first+i_count-1 and uploads them.  Per slice one
 * listed-prep launch forms the distances to the query and the neighbour matrix (the bits of the strict left-to-right
 * sums of the kNN path), then the same order and fit launches as nngp_sweep_shard. */
int nngp_sweep_listed_shard(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g,
                            const double* d_t, int N, int I, int i_first, int i_count, int m, const long long* rows,
                            int n_restarts, const signed char* d_starts, double fatol, double xatol,
                            double* d_u_next, double* d_uG_next, int d, int j0, int dl, void* stream);
/* parareal.py:336-339: x <- u_cur[I-1:N], D <- uF[I:N+1] - uG_cur[I:N+1] appended on device. */
int nngp_append_iteration(nngp_handle_t h, const double* d_u_cur, const double* d_uF,
                          const double* d_uG_cur, int N, int I, int d, void* stream);
/* parareal.py:402: err[p] = max_j |a[p,j]-b[p,j]| for p in [0,rows). */
int nngp_rowwise_maxabs_diff(nngp_handle_t h, const double* d_a, const double* d_b, int rows,
                             int d, double* d_err, void* stream);

/* ---- ensembles of independent runs (PararealEnsemble) -----------------------------------
 * Segmented store: E members of `cap_rows` rows each share X, Y and the transposed copy of the dataset; member e's
 * rows are the global rows [e cap, e cap + rows_e), so the GP kernels gather them by global index.  A handle holds
 * either a plain dataset (nngp_dataset_*) or a segmented store: reserving one discards the other.
 * nngp_seg_reserve: (re)lays the store out for E members of cap_rows rows; growing the capacity keeps every
 * member's rows (copied to the new layout, synchronises); changing E or d needs an empty store (nngp_seg_reset). */
int nngp_seg_reserve(nngp_handle_t h, int n_members, long long cap_rows, int d);
/* every member back to 0 rows */
int nngp_seg_reset(nngp_handle_t h);
/* rows held by `member` (-1 outside [0, E)); rows per member the store has room for */
long long nngp_seg_rows(nngp_handle_t h, int member);
long long nngp_seg_cap(nngp_handle_t h);
/* parareal.py:336-339 for n runs in one launch: position p of the state (device, member stride ld_state >= (N+1) d,
 * row stride d) appends x <- u_cur[p, I_p-1:N], D <- uF[p, I_p:N+1] - uG_cur[p, I_p:N+1] to segment members[p].
 * members[n], I[n]: host arrays, I_p in [1, N]. */
int nngp_seg_append_iteration(nngp_handle_t h, int n, const int* members, const int* I, const double* d_u_cur,
                              const double* d_uF, const double* d_uG_cur, long long ld_state, int N, int d,
                              void* stream);
/* kNN of nq queries, each in its own rows of the store: query q (device, row stride ld_q) searches global rows
 * [base[q], base[q] + rows[q]) (host arrays, rows[q] >= m).  idx[nq,m]: global indices ordered by (distance, index),
 * dist[nq,m]: squared distances -- idx - base[q] and dist equal nngp_knn on that segment alone.  r2 (optional,
 * device [nq,m,m]): the neighbour distance matrix of the GP.  Segments up to 8192 rows with m <= 32 take one fused
 * launch; larger ones or m up to 160 the distance + selection kernels. */
int nngp_knn_segmented(nngp_handle_t h, const double* d_q, long long ld_q, int nq, int m, const long long* base,
                       const long long* rows, long long* d_idx, double* d_dist, double* d_r2, void* stream);
/* dst[dst_idx[r], :] = src[src_idx[r], :] for r < rows, rows of d doubles; a NULL index list is the
 * identity.  Device pointers; gathers and scatters the rows of an ensemble's state. */
int nngp_copy_rows(nngp_handle_t h, const double* d_src, const long long* d_src_idx, double* d_dst,
                   const long long* d_dst_idx, long long rows, long long d, void* stream);
/* nngp_sweep for E runs in lockstep, slices min(I) .. N-1, enqueued with no host round trip.  Every refusal happens
 * before anything is enqueued.
 * Layout: state u_next, uG_next: device [E, N+1, d].  Position p belongs to segment members[p] (host) and sweeps
 * slices I[p] .. N-1 (host, ascending in p, so the runs active at a slice are a prefix of the positions, reached with
 * the member stride (N+1) d).  d_t_pos (device [E, N+1]): the slice boundaries of each position.  m[E] (host, each in
 * 1..160): the neighbour count of each position.  d_starts: the starts of every predict, slice-major -- for slice i the
 * [d,9,R,2] blocks of the active positions in position order.
 * Neighbours: per slice one segmented kNN over the active kNN positions at the largest m among them (the first m_p
 * neighbours of a top-m_max list are the top-m_p); a slice in which such a member holds fewer rows than that m is
 * refused.  listed (host, NULL: no position) marks with listed[p] != 0 the positions whose neighbours the host chose
 * instead (nngp_sweep_listed_shard): rows (host, int64) holds, for every listed position in position order, its lists of
 * slices I_p .. N-1, [(N - I_p), m_p], as global rows of the store (members[p] cap + a row the member holds); a row
 * outside that range is refused.  Each run's results equal its solo kNN or listed sweep, bit for bit.
 * Routes, chosen once per call from the inputs: when no swept position is listed and all share one m, per slice one
 * coarse launch over the active runs beside the kNN, and one fit over all their predicts straight into the state;
 * otherwise per slice at most one listed-prep launch (which also gathers the kNN queries when the slice has both
 * kinds), the kNN, one gather, one fit per distinct m over the runs that use it (each sees exactly the neighbour set
 * and matrix of its solo sweep) and one scatter. */
int nngp_ensemble_sweep(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g, const double* d_t_pos,
                        int N, int E, const int* members, const int* I, const int* m, const int* listed,
                        const long long* rows, int n_restarts, const signed char* d_starts, double fatol, double xatol,
                        double* d_u_next, double* d_uG_next, int d, void* stream);
/* nngp_fit_predict with one neighbour count per predict: m[nq] (host); d_idx / d_dist rows ld = max m apart, the
 * first m[q] entries of row q used; the neighbour matrix is formed at ld.  Outputs as nngp_fit_predict. */
int nngp_fit_predict_mixed(nngp_handle_t h, const double* d_q, const long long* d_idx, const double* d_dist, int nq,
                           const int* m, int n_restarts, const signed char* d_starts, double fatol, double xatol,
                           double* d_pred, double* d_theta_opt, double* d_jitter_opt, double* d_fval_opt, int* d_nfev,
                           double* d_fvals, double* d_thetas, void* stream);

/* test hook: the device exp(-|x|), 1/|x| and -- when d_exp10 (2n doubles) is not NULL -- [10**x | log|x| + 3 ln 2]
 * used inside the GP kernels */
int nngp_selftest_math(nngp_handle_t h, const double* d_x, int n, double* d_exp_neg, double* d_rcp,
                       double* d_exp10, void* stream);

/* counters of kernel launches issued through this handle (bench.py: gpu_launches) */
long long nngp_launch_count(nngp_handle_t h);
/* device-side work counters since the last reset (synchronises): Nelder-Mead searches run and
 * objective (negative log marginal likelihood) evaluations made -- models.py:254-260, 240-252 */
int nngp_counters(nngp_handle_t h, long long* nm_runs, long long* nll_evals, int reset);
/* per-kernel-class device time measured with CUDA events on the launching stream while enabled;
 * classes: 0 RK propagators, 1 kNN, 2 neighbour distance matrix, 3 GP fit+predict, 4 other.
 * nngp_profile_read synchronises; ms[5] accumulated milliseconds, counts[5] timed launches. */
int nngp_profile_enable(nngp_handle_t h, int on);
int nngp_profile_read(nngp_handle_t h, double* ms, long long* counts, int reset);

#ifdef __cplusplus
}
#endif
#endif /* NNGPARA_H_ */
