// Internal declarations shared by the translation units of libnngpara.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "nngpara.h"

#define NNGP_MAX_PARAMS 8
#define NNGP_MAX_STAGES 11
#define NNGP_PROF_CLASSES 5  // 0 rk, 1 knn, 2 gp_prep, 3 gp_fit, 4 other

struct SystemDesc {
  int system_id = -1;
  int d = 0;
  int n_params = 0;
  double params[NNGP_MAX_PARAMS] = {0};
  int normalize = 0;
  double* d_mn = nullptr;  // device [d]
  double* d_mx = nullptr;  // device [d]
};

// Passed by value to kernels.
struct SysArgs {
  int system_id;
  int d;
  int normalize;
  double p[NNGP_MAX_PARAMS];
  double q[4];  // derived parameters (rk.cu)
  double* traj;  // optional: state after every step, [n_slices][steps+1][d] (run_F_full); nullptr = last state only
  const double* mn;
  const double* mx;
};

// Where a fit block's per-(query, dim) completion counters last lived: the fit leaves them zero, so they are cleared
// only when they move (ensure_done_zero).  Owned by whoever owns the block: the handle's workspace, a fit group.
struct DoneTracker {
  const void* ptr = nullptr;
  size_t bytes = 0;
};

struct nngp_handle_s {
  int device = 0;
  std::string err;
  std::vector<SystemDesc> systems;
  long long launches = 0;
  // dataset (parareal.py:336-339): X,Y row-major [cap,d]; XT column-major copy [d,cap]
  int ds_d = 0;
  long long ds_cap = 0;
  long long ds_rows = 0;
  double* ds_x = nullptr;
  double* ds_y = nullptr;
  double* ds_xt = nullptr;
  // workspace
  void* ws = nullptr;
  size_t ws_bytes = 0;
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
  void* stage = nullptr;  // device staging for *_host variants
  size_t stage_bytes = 0;
  cudaStream_t own_stream = nullptr;
  // sweep: the coarse step of a slice runs on aux_stream beside the neighbour search (fork / join with two events)
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  unsigned int* d_ticket = nullptr;  // last-CTA-done counter of the fused sweep prologue (zero between launches)
  // a pivot <= pivot_guard * K_rr fails the factorisation (gpfit.cu::gp_head); ulps * 2^-52
  double pivot_guard = 2.220446049250313e-16;
  // per-handle (= per-device) launch state of the GP kernels, indexed by M/2: resident CTAs per SM and
  // "dynamic shared memory attribute set" flags (cudaFuncSetAttribute is per device)
  int sm_count = 148;
  int occ_fit[17] = {0};
  int occ_fit_grouped[17] = {0};
  bool attr_nll[17] = {false};
  bool attr_mean[17] = {false};
  bool attr_big = false;
  bool attr_spec[17] = {false};
  // evaluations after which a search is handed to the four-warp continuation kernel (0: never, the default: measured
  // slower than the sequential search at 1 and at 8 GPUs, profiles/r02/fit_kernel_variants.log); NNGP_FIT_BUDGET
  int fit_budget = 0;
  // which search kernel a fit launches: 0 auto (several searches per warp for batched queries, nq >= 4 and m <= 20,
  // where it is 1.4-4x faster; otherwise one search per warp, as in the serial sweep, whose searches fail early and
  // cheaply 45 % of the time -- DESIGN.md section 4.5 -- or four warps per search when such a launch has at most 3
  // searches per resident CTA), 1 always one search per warp, 2 always grouped, 3 always four warps per search.
  // NNGP_FIT_MODE=auto|warp|grouped|quad
  int fit_mode = 0;
  cudaStream_t queue_stream = nullptr;  // stream of the last fit that took a queue slot (next_queue)
  bool queue_stream_valid = false;
  bool attr_knn_tile = false;  // scan_select_tile_kernel's shared-memory attribute set on this device
  bool attr_knn_tile_seg = false;
  // segmented store (nngp_seg_reserve): seg_E members of seg_cap rows each in ds_x / ds_y / ds_xt (ds_cap = seg_E *
  // seg_cap); seg_rows[e] rows held by member e.  0 members: the handle holds a plain dataset.
  int seg_E = 0;
  long long seg_cap = 0;
  std::vector<long long> seg_rows;
  unsigned int* seg_tickets = nullptr;  // one zeroed last-CTA counter per query of the segmented kNN
  int seg_tickets_n = 0;
  // small host->device tables of the segmented entry points: pinned staging, re-used once the copy that last read it
  // has completed (event)
  struct Upload { void* host = nullptr; void* dev = nullptr; size_t bytes = 0; cudaEvent_t done = nullptr; };
  // 0 row tables, 1 segment tables, 2 copy spans of the grouped fits, 3 neighbour lists and 4 ListedQuery
  // tables of the listed sweeps
  Upload up[5];
  // device counters: [0] Nelder-Mead runs, [1] objective (nll) evaluations
  unsigned long long* d_counters = nullptr;
  // task-queue heads of the persistent fit kernel: one zeroed counter per launch
  unsigned int* d_queues = nullptr;
  int queue_next = 0;
  // where the completion counters of the last fit in the handle's workspace lived (ensure_done_zero)
  DoneTracker done;
  // optional per-kernel-class timing with CUDA events on the launching stream
  bool profiling = false;
  struct ProfRec { int cls; cudaEvent_t a, b; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_free;
  double prof_ms[NNGP_PROF_CLASSES] = {0};
  long long prof_n[NNGP_PROF_CLASSES] = {0};
};

// RAII: times the launches issued inside its scope when profiling is on
struct ProfScope {
  nngp_handle_t h;
  cudaStream_t st;
  bool on;
  ProfScope(nngp_handle_t h_, int cls, cudaStream_t st_);
  ~ProfScope();
};

int nngp_fail(nngp_handle_t h, const char* fmt, ...);
#define NNGP_CUDA(h, call)                                                                  \
  do {                                                                                      \
    cudaError_t e__ = (call);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return nngp_fail(h, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
  } while (0)

void* nngp_workspace(nngp_handle_t h, size_t bytes);  // grows, nullptr on failure
SysArgs nngp_sys_args(const SystemDesc& s);

// rk.cu
int rk_set_tableaus(nngp_handle_t h);
int rk_launch(nngp_handle_t h, const SystemDesc& s, int method, int h_mode, long long steps,
              int n_slices, const double* d_t0, const double* d_t1, const double* d_u0,
              long long ld_u0, double* d_u1, long long ld_u1, cudaStream_t st, double* d_traj = nullptr);
int rhs_launch(nngp_handle_t h, const SystemDesc& s, int n, const double* d_u, double* d_out,
               cudaStream_t st);
void rk_host_tableau(int method, int* S, double* a, double* b, double* c);

// knn.cu
size_t knn_workspace_bytes(int nq, long long n, int m);
int knn_launch(nngp_handle_t h, const double* d_q, int nq, int m, long long n_rows,
               long long* d_idx, double* d_dist, void* ws, cudaStream_t st);
bool knn_prep_fused_ok(nngp_handle_t h, long long n, int m);
int knn_prep_fused_launch(nngp_handle_t h, const double* d_q, int m, long long n, long long* d_idx, double* d_dist,
                          double* d_r2, void* ws, cudaStream_t st);
int dataset_append_launch(nngp_handle_t h, const double* d_x, const double* d_y, long long rows,
                          cudaStream_t st);
int append_iteration_launch(nngp_handle_t h, const double* d_u_cur, const double* d_uF,
                            const double* d_uG_cur, int N, int I, int d, cudaStream_t st);
size_t knn_seg_workspace_bytes(int nq, long long n_max, int m);
int knn_seg_launch(nngp_handle_t h, const double* d_q, long long ld_q, int nq, int m, const long long* d_base,
                   const long long* d_rows, long long n_max, long long* d_idx, double* d_dist, double* d_r2,
                   unsigned int* tickets, void* ws, cudaStream_t st);
int append_seg_launch(nngp_handle_t h, const double* xs, const double* ya, const double* yb, long long ld,
                      const long long* d_tab, int nsrc, long long max_rows, cudaStream_t st);
int copy_rows_launch(nngp_handle_t h, const double* src, const long long* si, double* dst, const long long* di,
                     long long rows, long long d, cudaStream_t st);
int rowwise_maxabs_launch(nngp_handle_t h, const double* a, const double* b, int rows, int d,
                          double* err, cudaStream_t st);

// One predict of a listed sweep (nngp_sweep_listed_shard, nngp_ensemble_sweep): the GP inputs of query q from
// the m dataset rows a neighbour rule chose on the host, instead of from a kNN.  m == 0: the entry only copies the
// query row to q_copy (the queries of the nearest-neighbour positions of a mixed slice, gathered to one row stride for
// the segmented kNN that follows).  All pointers are device pointers.
struct ListedQuery {
  const double* q;        // the query, d doubles
  const long long* rows;  // its m dataset rows, in the rule's order
  long long* idx;         // the rows are copied here (nullptr: the fit reads `rows` itself)
  double* dist;           // dist[a] = ||x_rows[a] - q||^2
  double* r2;             // r2[a ld + b] = ||x_rows[a] - x_rows[b]||^2 for a, b < m
  double* q_copy;
  int m, ld;
};

// gpfit.cu
size_t gp_prep_bytes(int nq, int m);
size_t gp_fit_ws_bytes(int nq, int d, int m, int R);      // [r2 | per-search results | done counters]
size_t gp_fit_done_offset(int nq, int d, int m, int R);   // byte offset of the done counters
int gp_prep_launch(nngp_handle_t h, const long long* d_idx, int nq, int m, double* d_r2,
                   cudaStream_t st);
int listed_prep_launch(nngp_handle_t h, const ListedQuery* d_lq, int n, cudaStream_t st);
int gp_order_launch(nngp_handle_t h, const signed char* d_starts, int nseg, int seg_len, int global_ids,
                    int* d_order, cudaStream_t st);
int gp_fit_predict_launch(nngp_handle_t h, const long long* d_idx, const double* d_dist, void* ws,
                          unsigned int* queue, const int* order, int nq, int m, int R, const signed char* d_starts,
                          double fatol, double xatol, double* d_pred, const double* d_add,
                          long long ld_pred, double* d_theta_opt, double* d_jitter_opt,
                          double* d_fval_opt, int* d_nfev, double* d_fvals, double* d_thetas,
                          cudaStream_t st, int j0 = 0, int dl = -1);
int gp_nll_launch(nngp_handle_t h, const long long* d_idx, const double* d_r2, int nq, int m,
                  int nt, const double* d_theta, const double* d_jitter10, double* d_nll,
                  cudaStream_t st);
int gp_mean_launch(nngp_handle_t h, const long long* d_idx, const double* d_dist,
                   const double* d_r2, int nq, int m, const double* d_theta,
                   const double* d_jitter, double* d_pred, cudaStream_t st);

int selftest_math_launch(nngp_handle_t h, const double* d_x, int n, double* d_exp, double* d_rcp,
                         double* d_exp10, cudaStream_t st);

