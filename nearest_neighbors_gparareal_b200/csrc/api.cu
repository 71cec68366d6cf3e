// extern "C" entry points of libnngpara.so (see include/nngpara.h), handle management,
// host-buffer variants, the fused on-device sweep and the roofline micro-benchmarks.
#include "common.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstring>

#define NNGP_QUEUE_SLOTS 4096

static std::string g_create_error;

int nngp_fail(nngp_handle_t h, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return -1;
}

static inline cudaStream_t as_stream(void* s) { return (cudaStream_t)s; }

// every entry point makes the handle's device current first: a process may hold handles on several devices
#define NNGP_USE_DEVICE(h)                                                                  \
  do {                                                                                      \
    if ((h) != nullptr) cudaSetDevice((h)->device);                                         \
  } while (0)

ProfScope::ProfScope(nngp_handle_t h_, int cls, cudaStream_t st_) : h(h_), st(st_), on(h_->profiling) {
  if (!on) return;
  nngp_handle_s::ProfRec r;
  r.cls = cls;
  for (cudaEvent_t* e : {&r.a, &r.b}) {
    if (!h->prof_free.empty()) {
      *e = h->prof_free.back();
      h->prof_free.pop_back();
    } else {
      cudaEventCreate(e);
    }
  }
  cudaEventRecord(r.a, st);
  h->prof_recs.push_back(r);
}

ProfScope::~ProfScope() {
  if (on) cudaEventRecord(h->prof_recs.back().b, st);
}

// a zeroed task-queue head for the next fit launch on stream st (slots are re-zeroed in bulk)
// (a fit uses up to three counters: its task queue, the number of parked long searches and their queue)
static unsigned int* next_queue(nngp_handle_t h, cudaStream_t st) {
  if (h->queue_next + 4 > NNGP_QUEUE_SLOTS) {
    // the bulk re-zeroing is ordered after the fits of `st` only: a fit still running on another stream of this
    // handle (host entry points use the handle's own stream, device entry points the caller's) must finish first
    if (h->queue_stream_valid && h->queue_stream != st) cudaStreamSynchronize(h->queue_stream);
    cudaMemsetAsync(h->d_queues, 0, NNGP_QUEUE_SLOTS * sizeof(unsigned int), st);
    h->queue_next = 0;
  }
  if (h->queue_stream_valid && h->queue_stream != st && h->queue_next != 0) {
    // the stream changed in the middle of a ring: the slots handed out so far may still be in use there, and a later
    // wrap on either stream must not overtake them -- cheap (a stream switch is rare) and keeps the invariant simple
    cudaStreamSynchronize(h->queue_stream);
  }
  h->queue_stream = st;
  h->queue_stream_valid = true;
  unsigned int* p = h->d_queues + h->queue_next;
  h->queue_next += 4;
  return p;
}

// the fit kernel leaves its completion counters zero; they only need clearing when they move (t: where they last were)
static int ensure_done_zero(nngp_handle_t h, DoneTracker& t, void* ws_fit, int nq, int d, int m, int R, cudaStream_t st) {
  const char* ptr = (const char*)ws_fit + gp_fit_done_offset(nq, d, m, R);
  const size_t bytes = sizeof(unsigned int) * (size_t)nq * d;
  if (t.ptr != ptr || t.bytes != bytes) {
    NNGP_CUDA(h, cudaMemsetAsync((void*)ptr, 0, bytes, st));
    t.ptr = ptr;
    t.bytes = bytes;
  }
  return 0;
}

void* nngp_workspace(nngp_handle_t h, size_t bytes) {
  // whoever asks for the block may overwrite the (left-zero) completion counters of an earlier fit:
  // the next fit clears them again (ensure_done_zero)
  h->done = DoneTracker{};
  if (bytes <= h->ws_bytes) return h->ws;
  // grow: work already enqueued may still use the old block
  cudaDeviceSynchronize();
  if (h->ws) cudaFree(h->ws);
  h->ws = nullptr;
  h->ws_bytes = 0;
  size_t want = bytes + bytes / 4 + (1 << 20);
  if (cudaMalloc(&h->ws, want) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  h->ws_bytes = want;
  return h->ws;
}

static void* pinned_buf(nngp_handle_t h, size_t bytes) {
  if (bytes <= h->pinned_bytes) return h->pinned;
  if (h->pinned) cudaFreeHost(h->pinned);
  h->pinned = nullptr;
  h->pinned_bytes = 0;
  size_t want = bytes + bytes / 4 + (1 << 16);
  if (cudaMallocHost(&h->pinned, want) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  h->pinned_bytes = want;
  return h->pinned;
}

static void* stage_buf(nngp_handle_t h, size_t bytes) {
  if (bytes <= h->stage_bytes) return h->stage;
  cudaDeviceSynchronize();
  if (h->stage) cudaFree(h->stage);
  h->stage = nullptr;
  h->stage_bytes = 0;
  size_t want = bytes + bytes / 4 + (1 << 16);
  if (cudaMalloc(&h->stage, want) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  h->stage_bytes = want;
  return h->stage;
}

// simple carve-out helper over a byte block (256 B aligned pieces)
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base((char*)b) {}
  template <class T> T* take(size_t count) {
    T* p = (T*)(base + off);
    off += ((count * sizeof(T) + 255) / 256) * 256;
    return p;
  }
  static size_t pad(size_t bytes) { return ((bytes + 255) / 256) * 256; }
};

// Copies `bytes` of host data to the device buffer of upload slot `slot` on stream st (pinned staging; the staging is
// overwritten only after the copy that last read it has completed).  nullptr on failure.
static void* upload_table(nngp_handle_t h, int slot, const void* src, size_t bytes, cudaStream_t st) {
  nngp_handle_s::Upload& u = h->up[slot];
  if (u.done == nullptr && cudaEventCreateWithFlags(&u.done, cudaEventDisableTiming) != cudaSuccess) return nullptr;
  if (u.host) cudaEventSynchronize(u.done);
  if (bytes > u.bytes) {
    cudaDeviceSynchronize();  // work already enqueued may still read the old device table
    if (u.host) cudaFreeHost(u.host);
    if (u.dev) cudaFree(u.dev);
    u.host = u.dev = nullptr;
    u.bytes = 0;
    const size_t want = bytes + bytes / 2 + 256;
    if (cudaMallocHost(&u.host, want) != cudaSuccess || cudaMalloc(&u.dev, want) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    u.bytes = want;
  }
  memcpy(u.host, src, bytes);
  if (cudaMemcpyAsync(u.dev, u.host, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) return nullptr;
  cudaEventRecord(u.done, st);
  return u.dev;
}

// nq zeroed last-CTA counters for the segmented kNN (the kernel leaves them zero)
static unsigned int* seg_tickets(nngp_handle_t h, int nq) {
  if (nq > h->seg_tickets_n) {
    cudaDeviceSynchronize();
    if (h->seg_tickets) cudaFree(h->seg_tickets);
    h->seg_tickets = nullptr;
    h->seg_tickets_n = 0;
    const int want = nq + 64;
    if (cudaMalloc(&h->seg_tickets, sizeof(unsigned int) * want) != cudaSuccess ||
        cudaMemset(h->seg_tickets, 0, sizeof(unsigned int) * want) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    h->seg_tickets_n = want;
  }
  return h->seg_tickets;
}

// kNN + neighbour matrix of nq queries: one launch (scan + top-m + neighbour matrix) for a single query when the
// shape allows it, otherwise the general kNN followed by gp_prep_kernel
static int knn_prep_launch(nngp_handle_t h, const double* d_q, int nq, int m, long long n, long long* idx, double* dist,
                           void* kws, void* fws, cudaStream_t st) {
  if (nq == 1 && knn_prep_fused_ok(h, n, m)) return knn_prep_fused_launch(h, d_q, m, n, idx, dist, (double*)fws, kws, st);
  if (int rc = knn_launch(h, d_q, nq, m, n, idx, dist, kws, st)) return rc;
  return gp_prep_launch(h, idx, nq, m, (double*)fws, st);
}

// Everything of a slice that precedes the fits: the coarse step gn = G(u) of nq rows (row stride ld) on the auxiliary
// stream, beside it the neighbour search `knn` on the caller's stream, which then joins the auxiliary one before the
// fit, whose epilogue adds gn to the prediction.
template <class Knn>
static int sweep_slice_prologue(nngp_handle_t h, const SystemDesc& s, int method_g, int h_mode, long long steps_g, int nq,
                                const double* t0, const double* t1, const double* u, long long ld, double* gn,
                                cudaStream_t st, Knn knn) {
  NNGP_CUDA(h, cudaEventRecord(h->ev_fork, st));
  NNGP_CUDA(h, cudaStreamWaitEvent(h->aux_stream, h->ev_fork, 0));
  if (int rc = rk_launch(h, s, method_g, h_mode, steps_g, nq, t0, t1, u, ld, gn, ld, h->aux_stream)) return rc;
  NNGP_CUDA(h, cudaEventRecord(h->ev_join, h->aux_stream));
  if (int rc = knn()) return rc;
  NNGP_CUDA(h, cudaStreamWaitEvent(st, h->ev_join, 0));
  return 0;
}

extern "C" {

int nngp_abi_version(void) { return NNGP_ABI_VERSION; }

int nngp_create(int device, nngp_handle_t* out) {
  if (!out) return nngp_fail(nullptr, "nngp_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return nngp_fail(nullptr, "nngp_create: no CUDA device (%s); this library has no CPU fallback",
                     cudaGetErrorString(e));
  if (device < 0 || device >= count) return nngp_fail(nullptr, "nngp_create: device %d of %d", device, count);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return nngp_fail(nullptr, "cudaSetDevice: %s", cudaGetErrorString(e));
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10)
    return nngp_fail(nullptr, "nngp_create: device sm_%d%d is not Blackwell sm_100a", prop.major, prop.minor);
  nngp_handle_t h = new nngp_handle_s();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  if (const char* fm = getenv("NNGP_FIT_MODE")) h->fit_mode = (strcmp(fm, "warp") == 0) ? 1 : (strcmp(fm, "grouped") == 0) ? 2 : (strcmp(fm, "quad") == 0) ? 3 : 0;
  if (const char* b = getenv("NNGP_FIT_BUDGET")) h->fit_budget = atoi(b);
  if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return nngp_fail(nullptr, "cudaStreamCreate failed");
  }
  if (cudaMalloc(&h->d_counters, 8 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(h->d_counters, 0, 8 * sizeof(unsigned long long)) != cudaSuccess) {
    delete h;
    return nngp_fail(nullptr, "cudaMalloc(counters) failed");
  }
  if (cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaMalloc(&h->d_ticket, 8 * sizeof(unsigned int)) != cudaSuccess ||
      cudaMemset(h->d_ticket, 0, 8 * sizeof(unsigned int)) != cudaSuccess) {
    delete h;
    return nngp_fail(nullptr, "nngp_create: auxiliary stream / events failed");
  }
  if (cudaMalloc(&h->d_queues, NNGP_QUEUE_SLOTS * sizeof(unsigned int)) != cudaSuccess ||
      cudaMemset(h->d_queues, 0, NNGP_QUEUE_SLOTS * sizeof(unsigned int)) != cudaSuccess) {
    delete h;
    return nngp_fail(nullptr, "cudaMalloc(queues) failed");
  }
  if (const char* g = getenv("NNGP_PIVOT_GUARD_ULPS")) {
    if (nngp_set_pivot_guard(h, atof(g)) != 0) {
      g_create_error = h->err;
      delete h;
      return -1;
    }
  }
  if (rk_set_tableaus(h) != 0) {
    g_create_error = h->err;
    delete h;
    return -1;
  }
  *out = h;
  return 0;
}

int nngp_destroy(nngp_handle_t h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (auto& s : h->systems) {
    if (s.d_mn) cudaFree(s.d_mn);
    if (s.d_mx) cudaFree(s.d_mx);
  }
  if (h->ds_x) cudaFree(h->ds_x);
  if (h->ds_y) cudaFree(h->ds_y);
  if (h->ds_xt) cudaFree(h->ds_xt);
  if (h->ws) cudaFree(h->ws);
  if (h->stage) cudaFree(h->stage);
  if (h->pinned) cudaFreeHost(h->pinned);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->d_ticket) cudaFree(h->d_ticket);
  if (h->d_counters) cudaFree(h->d_counters);
  if (h->d_queues) cudaFree(h->d_queues);
  if (h->seg_tickets) cudaFree(h->seg_tickets);
  for (auto& u : h->up) {
    if (u.host) cudaFreeHost(u.host);
    if (u.dev) cudaFree(u.dev);
    if (u.done) cudaEventDestroy(u.done);
  }
  for (auto& r : h->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto e : h->prof_free) cudaEventDestroy(e);
  delete h;
  return 0;
}

const char* nngp_last_error(nngp_handle_t h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int nngp_synchronize(nngp_handle_t h, void* stream) {
  NNGP_USE_DEVICE(h);
  NNGP_CUDA(h, cudaStreamSynchronize(as_stream(stream)));
  return 0;
}

long long nngp_launch_count(nngp_handle_t h) { return h->launches; }

int nngp_set_pivot_guard(nngp_handle_t h, double ulps) {
  if (!(ulps == ulps) || ulps < 0.0 || ulps > 1e6) return nngp_fail(h, "set_pivot_guard: ulps=%g outside [0, 1e6]", ulps);
  // below 2^-10 ulp the running product of the pivots could leave the normal range: "0" means "as small as possible"
  if (ulps < 9.765625e-4) ulps = 9.765625e-4;
  h->pivot_guard = ulps * 2.220446049250313e-16;
  return 0;
}

int nngp_set_fit_mode(nngp_handle_t h, int mode) {
  if (mode < 0 || mode > 3) return nngp_fail(h, "set_fit_mode: mode=%d outside {0 auto, 1 warp, 2 grouped, 3 quad}", mode);
  h->fit_mode = mode;
  return 0;
}

int nngp_set_fit_budget(nngp_handle_t h, int evaluations) {
  if (evaluations < 0 || evaluations > 400) return nngp_fail(h, "set_fit_budget: %d outside [0, 400]", evaluations);
  h->fit_budget = evaluations;
  return 0;
}

double nngp_get_pivot_guard(nngp_handle_t h) { return h->pivot_guard / 2.220446049250313e-16; }

int nngp_counters(nngp_handle_t h, long long* nm_runs, long long* nll_evals, int reset) {
  NNGP_USE_DEVICE(h);
  unsigned long long v[8];
  NNGP_CUDA(h, cudaDeviceSynchronize());
  NNGP_CUDA(h, cudaMemcpy(v, h->d_counters, sizeof(v), cudaMemcpyDeviceToHost));
  if (getenv("NNGP_FIT_STATS"))
    fprintf(stderr, "fit stats: searches %llu evals %llu | warp-rounds %llu wanted group-evals %llu busy group-slots %llu "
            "fast-forwarded iterations %llu max rounds of a warp (all launches) %llu\n", v[0], v[1], v[2], v[3], v[4], v[5], v[6]);
  if (nm_runs) *nm_runs = (long long)v[0];
  if (nll_evals) *nll_evals = (long long)v[1];
  if (reset) NNGP_CUDA(h, cudaMemset(h->d_counters, 0, sizeof(v)));
  return 0;
}

int nngp_profile_enable(nngp_handle_t h, int on) {
  h->profiling = (on != 0);
  return 0;
}

int nngp_profile_read(nngp_handle_t h, double* ms, long long* counts, int reset) {
  NNGP_USE_DEVICE(h);
  NNGP_CUDA(h, cudaDeviceSynchronize());
  for (auto& r : h->prof_recs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) {
      h->prof_ms[r.cls] += t;
      h->prof_n[r.cls] += 1;
    }
    h->prof_free.push_back(r.a);
    h->prof_free.push_back(r.b);
  }
  cudaGetLastError();
  h->prof_recs.clear();
  for (int i = 0; i < NNGP_PROF_CLASSES; i++) {
    if (ms) ms[i] = h->prof_ms[i];
    if (counts) counts[i] = h->prof_n[i];
    if (reset) { h->prof_ms[i] = 0; h->prof_n[i] = 0; }
  }
  return 0;
}

// ---- systems ---------------------------------------------------------------------------
int nngp_system_create(nngp_handle_t h, int system_id, int d, const double* params, int n_params,
                       int normalize, const double* mn, const double* mx, int* sys_out) {
  NNGP_USE_DEVICE(h);
  if (!sys_out) return nngp_fail(h, "system_create: sys_out is NULL");
  if (system_id < NNGP_SYS_FHN_ODE || system_id > NNGP_SYS_BURGERS)
    return nngp_fail(h, "system_create: unknown system id %d", system_id);
  if (n_params < 0 || n_params > NNGP_MAX_PARAMS) return nngp_fail(h, "system_create: n_params=%d", n_params);
  if (d < 1) return nngp_fail(h, "system_create: d=%d", d);
  if (normalize != 0 && normalize != 1) return nngp_fail(h, "Only identity and -11 are implemented");
  if (normalize && (!mn || !mx)) return nngp_fail(h, "system_create: normalize=1 needs mn and mx");
  SystemDesc s;
  s.system_id = system_id;
  s.d = d;
  s.n_params = n_params;
  for (int i = 0; i < n_params; i++) s.params[i] = params[i];
  s.normalize = normalize;
  if (normalize) {
    NNGP_CUDA(h, cudaMalloc(&s.d_mn, sizeof(double) * d));
    NNGP_CUDA(h, cudaMalloc(&s.d_mx, sizeof(double) * d));
    NNGP_CUDA(h, cudaMemcpy(s.d_mn, mn, sizeof(double) * d, cudaMemcpyHostToDevice));
    NNGP_CUDA(h, cudaMemcpy(s.d_mx, mx, sizeof(double) * d, cudaMemcpyHostToDevice));
  }
  h->systems.push_back(s);
  *sys_out = (int)h->systems.size() - 1;
  return 0;
}

static int get_sys(nngp_handle_t h, int sys, const SystemDesc** out) {
  if (sys < 0 || sys >= (int)h->systems.size()) return nngp_fail(h, "bad system handle %d", sys);
  *out = &h->systems[sys];
  return 0;
}

int nngp_rhs_eval(nngp_handle_t h, int sys, int n, const double* d_u, double* d_out, void* stream) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  return rhs_launch(h, *s, n, d_u, d_out, as_stream(stream));
}

int nngp_rhs_eval_host(nngp_handle_t h, int sys, int n, const double* u, double* out) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  const size_t bytes = sizeof(double) * (size_t)n * s->d;
  double* dev = (double*)stage_buf(h, 2 * Carver::pad(bytes));
  if (!dev) return nngp_fail(h, "rhs_eval_host: out of device memory");
  double* dout = (double*)((char*)dev + Carver::pad(bytes));
  NNGP_CUDA(h, cudaMemcpyAsync(dev, u, bytes, cudaMemcpyHostToDevice, h->own_stream));
  if (int rc = rhs_launch(h, *s, n, dev, dout, h->own_stream)) return rc;
  NNGP_CUDA(h, cudaMemcpyAsync(out, dout, bytes, cudaMemcpyDeviceToHost, h->own_stream));
  NNGP_CUDA(h, cudaStreamSynchronize(h->own_stream));
  return 0;
}

// ---- propagators -----------------------------------------------------------------------
int nngp_rk_batch(nngp_handle_t h, int sys, int method, int h_mode, long long steps, int n_slices,
                  const double* d_t0, const double* d_t1, const double* d_u0, long long ld_u0,
                  double* d_u1, long long ld_u1, void* stream) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  return rk_launch(h, *s, method, h_mode, steps, n_slices, d_t0, d_t1, d_u0, ld_u0, d_u1, ld_u1,
                   as_stream(stream));
}

int nngp_rk_batch_host(nngp_handle_t h, int sys, int method, int h_mode, long long steps,
                       int n_slices, const double* t0, const double* t1, const double* u0,
                       double* u1) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  if (n_slices <= 0) return 0;
  const int d = s->d;
  const size_t nb_t = sizeof(double) * (size_t)n_slices, nb_u = nb_t * d;
  // pinned staging: [t0 | t1 | u0] in, [u1] out
  const size_t in_bytes = 2 * Carver::pad(nb_t) + Carver::pad(nb_u);
  char* pin = (char*)pinned_buf(h, in_bytes + Carver::pad(nb_u));
  char* dev = (char*)stage_buf(h, in_bytes + Carver::pad(nb_u));
  if (!pin || !dev) return nngp_fail(h, "rk_batch_host: out of staging memory");
  Carver cp(pin), cd(dev);
  double* p_t0 = cp.take<double>(n_slices); double* p_t1 = cp.take<double>(n_slices);
  double* p_u0 = cp.take<double>((size_t)n_slices * d); double* p_u1 = cp.take<double>((size_t)n_slices * d);
  double* g_t0 = cd.take<double>(n_slices); double* g_t1 = cd.take<double>(n_slices);
  double* g_u0 = cd.take<double>((size_t)n_slices * d); double* g_u1 = cd.take<double>((size_t)n_slices * d);
  memcpy(p_t0, t0, nb_t);
  memcpy(p_t1, t1, nb_t);
  memcpy(p_u0, u0, nb_u);
  NNGP_CUDA(h, cudaMemcpyAsync(g_t0, p_t0, in_bytes, cudaMemcpyHostToDevice, h->own_stream));
  if (int rc = rk_launch(h, *s, method, h_mode, steps, n_slices, g_t0, g_t1, g_u0, d, g_u1, d, h->own_stream)) return rc;
  NNGP_CUDA(h, cudaMemcpyAsync(p_u1, g_u1, nb_u, cudaMemcpyDeviceToHost, h->own_stream));
  NNGP_CUDA(h, cudaStreamSynchronize(h->own_stream));
  memcpy(u1, p_u1, nb_u);
  return 0;
}

// every step of n_slices solves: d_traj[n_slices][steps+1][d]  (RK.run, RK.py:91-99)
int nngp_rk_full(nngp_handle_t h, int sys, int method, int h_mode, long long steps, int n_slices,
                 const double* d_t0, const double* d_t1, const double* d_u0, long long ld_u0, double* d_traj,
                 void* stream) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  if (n_slices <= 0) return 0;
  if (!d_traj) return nngp_fail(h, "rk_full: d_traj is NULL");
  if (steps < 1) return nngp_fail(h, "steps must be >= 1 (got %lld)", steps);
  // the last state also goes to the last row of each trajectory: use it as the u1 buffer
  double* u1 = d_traj + (long long)steps * s->d;
  return rk_launch(h, *s, method, h_mode, steps, n_slices, d_t0, d_t1, d_u0, ld_u0, u1, (steps + 1) * (long long)s->d,
                   as_stream(stream), d_traj);
}

int nngp_rk_full_host(nngp_handle_t h, int sys, int method, int h_mode, long long steps, double t0, double t1,
                      const double* u0, double* traj) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  if (steps < 1) return nngp_fail(h, "steps must be >= 1 (got %lld)", steps);
  const int d = s->d;
  const size_t nb_u = sizeof(double) * d, nb_tr = sizeof(double) * (size_t)(steps + 1) * d;
  char* dev = (char*)stage_buf(h, 2 * Carver::pad(sizeof(double)) + Carver::pad(nb_u) + Carver::pad(nb_tr));
  if (!dev) return nngp_fail(h, "rk_full_host: out of device memory (%zu bytes)", nb_tr);
  Carver cd(dev);
  double* g_t0 = cd.take<double>(1); double* g_t1 = cd.take<double>(1);
  double* g_u0 = cd.take<double>(d); double* g_tr = cd.take<double>((size_t)(steps + 1) * d);
  NNGP_CUDA(h, cudaMemcpyAsync(g_t0, &t0, sizeof(double), cudaMemcpyHostToDevice, h->own_stream));
  NNGP_CUDA(h, cudaMemcpyAsync(g_t1, &t1, sizeof(double), cudaMemcpyHostToDevice, h->own_stream));
  NNGP_CUDA(h, cudaMemcpyAsync(g_u0, u0, nb_u, cudaMemcpyHostToDevice, h->own_stream));
  if (int rc = nngp_rk_full(h, sys, method, h_mode, steps, 1, g_t0, g_t1, g_u0, d, g_tr, h->own_stream)) return rc;
  NNGP_CUDA(h, cudaMemcpyAsync(traj, g_tr, nb_tr, cudaMemcpyDeviceToHost, h->own_stream));
  NNGP_CUDA(h, cudaStreamSynchronize(h->own_stream));
  return 0;
}

int nngp_get_tableau(int method, int* stages, double* a, double* b, double* c) {
  if (method != 1 && method != 2 && method != 4 && method != 8) return -1;
  rk_host_tableau(method, stages, a, b, c);
  return 0;
}

// ---- dataset ---------------------------------------------------------------------------
int nngp_dataset_reserve(nngp_handle_t h, long long cap_rows, int d) {
  NNGP_USE_DEVICE(h);
  if (cap_rows < 1 || d < 1) return nngp_fail(h, "dataset_reserve: cap_rows=%lld d=%d", cap_rows, d);
  if (h->ds_x && h->ds_d == d && h->ds_cap >= cap_rows) return 0;
  if (h->ds_x && h->ds_d != d && h->ds_rows > 0)
    return nngp_fail(h, "dataset_reserve: dimension change %d -> %d with %lld rows held", h->ds_d, d, h->ds_rows);
  NNGP_CUDA(h, cudaDeviceSynchronize());
  double *nx = nullptr, *ny = nullptr, *nxt = nullptr;
  const size_t bytes = sizeof(double) * (size_t)cap_rows * d;
  NNGP_CUDA(h, cudaMalloc(&nx, bytes));
  NNGP_CUDA(h, cudaMalloc(&ny, bytes));
  NNGP_CUDA(h, cudaMalloc(&nxt, bytes));
  const long long keep = (h->ds_x && h->ds_d == d) ? h->ds_rows : 0;
  double *ox = h->ds_x, *oy = h->ds_y, *oxt = h->ds_xt;
  h->ds_x = nx; h->ds_y = ny; h->ds_xt = nxt;
  h->ds_d = d; h->ds_cap = cap_rows; h->ds_rows = 0;
  h->seg_E = 0;
  if (keep > 0) {
    if (int rc = dataset_append_launch(h, ox, oy, keep, nullptr)) return rc;
    NNGP_CUDA(h, cudaDeviceSynchronize());
  }
  if (ox) cudaFree(ox);
  if (oy) cudaFree(oy);
  if (oxt) cudaFree(oxt);
  return 0;
}

int nngp_dataset_reset(nngp_handle_t h) {
  h->ds_rows = 0;
  return 0;
}

int nngp_dataset_truncate(nngp_handle_t h, long long rows) {
  if (rows < 0 || rows > h->ds_rows) return nngp_fail(h, "dataset_truncate: rows=%lld outside [0,%lld]", rows, h->ds_rows);
  h->ds_rows = rows;
  return 0;
}

long long nngp_dataset_rows(nngp_handle_t h) { return h->ds_rows; }
int nngp_dataset_dim(nngp_handle_t h) { return h->ds_d; }

int nngp_dataset_append(nngp_handle_t h, const double* d_x, const double* d_y, long long rows,
                        void* stream) {
  NNGP_USE_DEVICE(h);
  return dataset_append_launch(h, d_x, d_y, rows, as_stream(stream));
}

int nngp_dataset_append_host(nngp_handle_t h, const double* x, const double* y, long long rows) {
  NNGP_USE_DEVICE(h);
  if (rows <= 0) return 0;
  if (!h->ds_x) return nngp_fail(h, "dataset not reserved (call nngp_dataset_reserve)");
  if (h->ds_rows + rows > h->ds_cap) {
    long long want = h->ds_cap * 2;
    if (want < h->ds_rows + rows) want = h->ds_rows + rows;
    if (int rc = nngp_dataset_reserve(h, want, h->ds_d)) return rc;
  }
  const size_t bytes = sizeof(double) * (size_t)rows * h->ds_d;
  char* dev = (char*)stage_buf(h, 2 * Carver::pad(bytes));
  if (!dev) return nngp_fail(h, "dataset_append_host: out of device memory");
  double* gx = (double*)dev;
  double* gy = (double*)(dev + Carver::pad(bytes));
  NNGP_CUDA(h, cudaMemcpyAsync(gx, x, bytes, cudaMemcpyHostToDevice, h->own_stream));
  NNGP_CUDA(h, cudaMemcpyAsync(gy, y, bytes, cudaMemcpyHostToDevice, h->own_stream));
  if (int rc = dataset_append_launch(h, gx, gy, rows, h->own_stream)) return rc;
  NNGP_CUDA(h, cudaStreamSynchronize(h->own_stream));
  return 0;
}

int nngp_append_iteration(nngp_handle_t h, const double* d_u_cur, const double* d_uF,
                          const double* d_uG_cur, int N, int I, int d, void* stream) {
  NNGP_USE_DEVICE(h);
  return append_iteration_launch(h, d_u_cur, d_uF, d_uG_cur, N, I, d, as_stream(stream));
}

int nngp_rowwise_maxabs_diff(nngp_handle_t h, const double* d_a, const double* d_b, int rows,
                             int d, double* d_err, void* stream) {
  NNGP_USE_DEVICE(h);
  return rowwise_maxabs_launch(h, d_a, d_b, rows, d, d_err, as_stream(stream));
}

// ---- kNN -------------------------------------------------------------------------------
int nngp_knn(nngp_handle_t h, const double* d_q, int nq, int m, long long n_rows,
             long long* d_idx, double* d_dist, void* stream) {
  NNGP_USE_DEVICE(h);
  const long long n = (n_rows > 0) ? n_rows : h->ds_rows;
  void* ws = nngp_workspace(h, knn_workspace_bytes(nq, n, m));
  if (!ws) return nngp_fail(h, "knn: out of device memory for %d x %lld distances", nq, n);
  return knn_launch(h, d_q, nq, m, n_rows, d_idx, d_dist, ws, as_stream(stream));
}

int nngp_knn_host(nngp_handle_t h, const double* q, int nq, int m, long long n_rows,
                  long long* idx, double* dist) {
  NNGP_USE_DEVICE(h);
  if (nq <= 0) return 0;
  const int d = h->ds_d;
  const size_t bq = Carver::pad(sizeof(double) * (size_t)nq * d);
  const size_t bi = Carver::pad(sizeof(long long) * (size_t)nq * m);
  const size_t bd = Carver::pad(sizeof(double) * (size_t)nq * m);
  char* dev = (char*)stage_buf(h, bq + bi + bd);
  if (!dev) return nngp_fail(h, "knn_host: out of device memory");
  double* gq = (double*)dev;
  long long* gi = (long long*)(dev + bq);
  double* gd = (double*)(dev + bq + bi);
  NNGP_CUDA(h, cudaMemcpyAsync(gq, q, sizeof(double) * (size_t)nq * d, cudaMemcpyHostToDevice, h->own_stream));
  if (int rc = nngp_knn(h, gq, nq, m, n_rows, gi, gd, h->own_stream)) return rc;
  NNGP_CUDA(h, cudaMemcpyAsync(idx, gi, sizeof(long long) * (size_t)nq * m, cudaMemcpyDeviceToHost, h->own_stream));
  NNGP_CUDA(h, cudaMemcpyAsync(dist, gd, sizeof(double) * (size_t)nq * m, cudaMemcpyDeviceToHost, h->own_stream));
  NNGP_CUDA(h, cudaStreamSynchronize(h->own_stream));
  return 0;
}

// ---- GP fit / predict ------------------------------------------------------------------
// workspace layout for a fit on nq queries: [knn distances nq*n | fit block (r2 | results | done)]
static int fit_workspace(nngp_handle_t h, int nq, long long n, int m, int R, void** knn_ws, void** fit_ws,
                         int** order = nullptr) {
  const size_t bk = Carver::pad(knn_workspace_bytes(nq, n, m));
  const size_t bf = Carver::pad(gp_fit_ws_bytes(nq, h->ds_d, m, R));
  const size_t bo = Carver::pad(sizeof(int) * (size_t)nq * h->ds_d * NNGP_N_JITTER * R);
  char* ws = (char*)nngp_workspace(h, bk + bf + bo);
  if (!ws) return nngp_fail(h, "fit: out of device memory (workspace %zu bytes)", bk + bf + bo);
  *knn_ws = ws;
  *fit_ws = ws + bk;
  if (order) *order = (int*)(ws + bk + bf);
  return 0;
}

int nngp_fit_predict(nngp_handle_t h, const double* d_q, const long long* d_idx,
                     const double* d_dist, int nq, int m, int n_restarts,
                     const signed char* d_starts, double fatol, double xatol, double* d_pred,
                     double* d_theta_opt, double* d_jitter_opt, double* d_fval_opt, int* d_nfev,
                     double* d_fvals, double* d_thetas, void* stream) {
  NNGP_USE_DEVICE(h);
  (void)d_q;
  if (n_restarts < 1) return nngp_fail(h, "fit: n_restarts=%d < 1", n_restarts);
  void *kws, *fws;
  int* order;
  if (int rc = fit_workspace(h, nq, h->ds_rows, m, n_restarts, &kws, &fws, &order)) return rc;
  cudaStream_t st = as_stream(stream);
  if (int rc = ensure_done_zero(h, h->done, fws, nq, h->ds_d, m, n_restarts, st)) return rc;
  if (int rc = gp_prep_launch(h, d_idx, nq, m, (double*)fws, st)) return rc;
  if (int rc = gp_order_launch(h, d_starts, nq, h->ds_d * NNGP_N_JITTER * n_restarts, 1, order, st)) return rc;
  return gp_fit_predict_launch(h, d_idx, d_dist, fws, next_queue(h, st), order, nq, m, n_restarts, d_starts, fatol,
                               xatol, d_pred, nullptr, h->ds_d, d_theta_opt, d_jitter_opt, d_fval_opt, d_nfev,
                               d_fvals, d_thetas, st);
}

int nngp_listed_prep(nngp_handle_t h, const double* d_q, long long ld_q, int nq, int m, const long long* d_rows, int ld,
                     double* d_dist, double* d_r2, void* stream) {
  NNGP_USE_DEVICE(h);
  if (nq <= 0) return 0;
  if (!h->ds_x) return nngp_fail(h, "listed_prep: dataset is empty");
  if (m < 1 || m > NNGP_MAX_NEIGHBOURS_BIG || ld < m)
    return nngp_fail(h, "listed_prep: m=%d outside [1,%d] or ld=%d < m", m, NNGP_MAX_NEIGHBOURS_BIG, ld);
  if (ld_q < h->ds_d) return nngp_fail(h, "listed_prep: ld_q=%lld < d=%d", ld_q, h->ds_d);
  std::vector<ListedQuery> lq(nq);
  for (int q = 0; q < nq; q++)
    lq[q] = ListedQuery{d_q + q * ld_q, d_rows + (size_t)q * ld, nullptr, d_dist + (size_t)q * ld,
                        d_r2 + (size_t)q * ld * ld, nullptr, m, ld};
  cudaStream_t st = as_stream(stream);
  const ListedQuery* dlq = (const ListedQuery*)upload_table(h, 4, lq.data(), sizeof(ListedQuery) * lq.size(), st);
  if (!dlq) return nngp_fail(h, "listed_prep: out of memory for the query table");
  return listed_prep_launch(h, dlq, nq, st);
}

int nngp_gp_nll(nngp_handle_t h, const long long* d_idx, int nq, int m, int nt,
                const double* d_theta, const double* d_jitter10, double* d_nll, void* stream) {
  NNGP_USE_DEVICE(h);
  void *kws, *fws;
  if (int rc = fit_workspace(h, nq, h->ds_rows, m, 1, &kws, &fws)) return rc;
  cudaStream_t st = as_stream(stream);
  if (int rc = gp_prep_launch(h, d_idx, nq, m, (double*)fws, st)) return rc;
  return gp_nll_launch(h, d_idx, (const double*)fws, nq, m, nt, d_theta, d_jitter10, d_nll, st);
}

int nngp_gp_mean(nngp_handle_t h, const double* d_q, const long long* d_idx, const double* d_dist,
                 int nq, int m, const double* d_theta, const double* d_jitter, double* d_pred,
                 void* stream) {
  NNGP_USE_DEVICE(h);
  (void)d_q;
  void *kws, *fws;
  if (int rc = fit_workspace(h, nq, h->ds_rows, m, 1, &kws, &fws)) return rc;
  cudaStream_t st = as_stream(stream);
  if (int rc = gp_prep_launch(h, d_idx, nq, m, (double*)fws, st)) return rc;
  return gp_mean_launch(h, d_idx, d_dist, (const double*)fws, nq, m, d_theta, d_jitter, d_pred, st);
}

int nngp_predict_host(nngp_handle_t h, const double* q, int nq, int m, long long n_rows,
                      int n_restarts, const signed char* starts, double fatol, double xatol,
                      double* pred, long long* idx, double* theta_opt, double* jitter_opt,
                      double* fval_opt, int* nfev, double* fvals, double* thetas) {
  return nngp_predict_host_block(h, q, nq, m, n_rows, n_restarts, starts, fatol, xatol, 0, -1, pred, idx, theta_opt,
                                 jitter_opt, fval_opt, nfev, fvals, thetas);
}

int nngp_predict_host_block(nngp_handle_t h, const double* q, int nq, int m, long long n_rows,
                            int n_restarts, const signed char* starts, double fatol, double xatol, int j0, int dl,
                            double* pred, long long* idx, double* theta_opt, double* jitter_opt,
                            double* fval_opt, int* nfev, double* fvals, double* thetas) {
  NNGP_USE_DEVICE(h);
  if (nq <= 0) return 0;
  if (!h->ds_x) return nngp_fail(h, "predict: dataset is empty");
  const int d = h->ds_d, R = n_restarts;
  if (dl < 0) {
    j0 = 0;
    dl = d;
  }
  if (j0 < 0 || dl < 1 || j0 + dl > d) return nngp_fail(h, "predict: dimension block [%d,%d) outside [0,%d)", j0, j0 + dl, d);
  if (dl != d && nq != 1) return nngp_fail(h, "predict: a dimension block needs a single query (got %d)", nq);
  const long long n = (n_rows > 0) ? n_rows : h->ds_rows;
  const size_t nqd = (size_t)nq * d, ntask = nqd * NNGP_N_JITTER * R;
  size_t total = 0;
  auto add = [&](size_t bytes) { size_t o = total; total += Carver::pad(bytes); return o; };
  const size_t o_q = add(sizeof(double) * nqd), o_st = add(ntask * 2), o_idx = add(sizeof(long long) * nq * m),
               o_dist = add(sizeof(double) * nq * m), o_pred = add(sizeof(double) * nqd),
               o_th = add(sizeof(double) * nqd * 2), o_jit = add(sizeof(double) * nqd),
               o_fv = add(sizeof(double) * nqd), o_nfev = add(sizeof(int) * ntask),
               o_fvals = add(sizeof(double) * ntask), o_thetas = add(sizeof(double) * ntask * 2);
  char* dev = (char*)stage_buf(h, total);
  if (!dev) return nngp_fail(h, "predict_host: out of device memory (%zu bytes)", total);
  cudaStream_t st = h->own_stream;
  double* gq = (double*)(dev + o_q);
  signed char* gst = (signed char*)(dev + o_st);
  long long* gidx = (long long*)(dev + o_idx);
  double* gdist = (double*)(dev + o_dist);
  if (R < 1) return nngp_fail(h, "predict: n_restarts=%d < 1", R);
  // query and starts are adjacent in the device block: one copy from the pinned staging buffer instead of two from
  // pageable memory (a single predict of the sweep is latency-bound: every call on this path counts)
  const size_t in_bytes = (o_st - o_q) + ntask * 2;
  if (in_bytes <= (1u << 20)) {
    char* pin = (char*)pinned_buf(h, in_bytes);
    if (!pin) return nngp_fail(h, "predict_host: out of pinned memory");
    memcpy(pin, q, sizeof(double) * nqd);
    memcpy(pin + (o_st - o_q), starts, ntask * 2);
    NNGP_CUDA(h, cudaMemcpyAsync(gq, pin, in_bytes, cudaMemcpyHostToDevice, st));
  } else {
    NNGP_CUDA(h, cudaMemcpyAsync(gq, q, sizeof(double) * nqd, cudaMemcpyHostToDevice, st));
    NNGP_CUDA(h, cudaMemcpyAsync(gst, starts, ntask * 2, cudaMemcpyHostToDevice, st));
  }
  void *kws, *fws;
  int* order;
  if (int rc = fit_workspace(h, nq, n, m, R, &kws, &fws, &order)) return rc;
  if (int rc = ensure_done_zero(h, h->done, fws, nq, d, m, R, st)) return rc;
  if (int rc = knn_prep_launch(h, gq, nq, m, n, gidx, gdist, kws, fws, st)) return rc;
  if (dl == d) {
    if (int rc = gp_order_launch(h, gst, nq, d * NNGP_N_JITTER * R, 1, order, st)) return rc;
  } else {  // the searches of the block are a contiguous range of the (single) query's task list
    if (int rc = gp_order_launch(h, gst + (size_t)j0 * NNGP_N_JITTER * R * 2, 1, dl * NNGP_N_JITTER * R, 0, order, st)) return rc;
  }
  if (int rc = gp_fit_predict_launch(h, gidx, gdist, fws, next_queue(h, st), order, nq, m, R, gst, fatol, xatol,
                                     (double*)(dev + o_pred), nullptr, d,
                                     theta_opt ? (double*)(dev + o_th) : nullptr,
                                     jitter_opt ? (double*)(dev + o_jit) : nullptr,
                                     fval_opt ? (double*)(dev + o_fv) : nullptr,
                                     nfev ? (int*)(dev + o_nfev) : nullptr,
                                     fvals ? (double*)(dev + o_fvals) : nullptr,
                                     thetas ? (double*)(dev + o_thetas) : nullptr, st, j0, dl))
    return rc;
  // cudaMemcpyDefault: `pred` may be a host buffer or (unified addressing) a device buffer of the caller -- the ranks of a
  // dimension-sharded host predict all-gather their blocks on the device and read the result back once
  NNGP_CUDA(h, cudaMemcpyAsync(pred, dev + o_pred, sizeof(double) * nqd, cudaMemcpyDefault, st));
  if (idx) NNGP_CUDA(h, cudaMemcpyAsync(idx, gidx, sizeof(long long) * nq * m, cudaMemcpyDeviceToHost, st));
  if (theta_opt) NNGP_CUDA(h, cudaMemcpyAsync(theta_opt, dev + o_th, sizeof(double) * nqd * 2, cudaMemcpyDeviceToHost, st));
  if (jitter_opt) NNGP_CUDA(h, cudaMemcpyAsync(jitter_opt, dev + o_jit, sizeof(double) * nqd, cudaMemcpyDeviceToHost, st));
  if (fval_opt) NNGP_CUDA(h, cudaMemcpyAsync(fval_opt, dev + o_fv, sizeof(double) * nqd, cudaMemcpyDeviceToHost, st));
  if (nfev) NNGP_CUDA(h, cudaMemcpyAsync(nfev, dev + o_nfev, sizeof(int) * ntask, cudaMemcpyDeviceToHost, st));
  if (fvals) NNGP_CUDA(h, cudaMemcpyAsync(fvals, dev + o_fvals, sizeof(double) * ntask, cudaMemcpyDeviceToHost, st));
  if (thetas) NNGP_CUDA(h, cudaMemcpyAsync(thetas, dev + o_thetas, sizeof(double) * ntask * 2, cudaMemcpyDeviceToHost, st));
  NNGP_CUDA(h, cudaStreamSynchronize(st));
  return 0;
}

// ---- fused on-device sweep (parareal.py:359-382) --------------------------------------
int nngp_sweep(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g,
               const double* d_t, int N, int I, int m, int n_restarts,
               const signed char* d_starts, double fatol, double xatol, double* d_u_next,
               double* d_uG_next, int d, void* stream) {
  return nngp_sweep_shard(h, sys, method_g, h_mode, steps_g, d_t, N, I, I, N - I, m, n_restarts, d_starts, fatol, xatol,
                          d_u_next, d_uG_next, d, 0, d, stream);
}

// Slices i_first .. i_first+i_count-1 of the sweep that starts at slice I (d_starts holds the starts of predicts I,
// I+1, ... in order): G and the neighbour search in full, the d*9*R searches only for the output dimensions
// [j0, j0+dl), and u_next[i+1] written for those dimensions only.  A block dl < d sweeps one slice per call: the
// caller all-gathers row i+1 before the neighbour search of slice i+1 reads it.
// rows == nullptr: the neighbours are the m nearest dataset rows (nngp_sweep_shard); otherwise rows[(N-I), m] (host)
// lists them per slice and one listed-prep launch replaces the kNN (nngp_sweep_listed_shard).
static int sweep_shard_impl(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g, const double* d_t,
                            int N, int I, int i_first, int i_count, int m, const long long* rows, int n_restarts,
                            const signed char* d_starts, double fatol, double xatol, double* d_u_next,
                            double* d_uG_next, int d, int j0, int dl, void* stream) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  if (d != s->d || d != h->ds_d) return nngp_fail(h, "sweep: d=%d, system d=%d, dataset d=%d", d, s->d, h->ds_d);
  if (I < 0 || I > N) return nngp_fail(h, "sweep: I=%d outside [0,%d]", I, N);
  if (i_first < I || i_count < 0 || i_first + i_count > N)
    return nngp_fail(h, "sweep: slices [%d,%d) outside [%d,%d)", i_first, i_first + i_count, I, N);
  if (j0 < 0 || dl < 1 || j0 + dl > d) return nngp_fail(h, "sweep: dimensions [%d,%d) outside [0,%d)", j0, j0 + dl, d);
  if (dl < d && i_count > 1)
    return nngp_fail(h, "sweep: a dimension block sweeps one slice per call (i_count=%d): row i+1 must be all-gathered "
                     "before the neighbour search of slice i+1", i_count);
  if (n_restarts < 1) return nngp_fail(h, "sweep: n_restarts=%d < 1", n_restarts);
  cudaStream_t st = as_stream(stream);
  const long long n = h->ds_rows;
  const ListedQuery* dlq = nullptr;
  const long long* drows = nullptr;
  if (rows) {
    if (m < 1 || m > NNGP_MAX_NEIGHBOURS_BIG)
      return nngp_fail(h, "sweep_listed: m=%d outside [1,%d]", m, NNGP_MAX_NEIGHBOURS_BIG);
    const long long* used = rows + (size_t)(i_first - I) * m;
    for (size_t a = 0; a < (size_t)i_count * m; a++)
      if (used[a] < 0 || used[a] >= n)
        return nngp_fail(h, "sweep_listed: slice %d lists row %lld, outside the dataset's %lld rows",
                         i_first + (int)(a / m), used[a], n);
    if (i_count > 0 &&
        !(drows = (const long long*)upload_table(h, 3, used, sizeof(long long) * (size_t)i_count * m, st)))
      return nngp_fail(h, "sweep_listed: out of memory for the neighbour lists");
  }
  const int nruns = NNGP_N_JITTER * n_restarts;
  const int seg_len = dl * nruns;
  const size_t per_predict = (size_t)d * nruns * 2;
  const size_t bk = rows ? 0 : Carver::pad(knn_workspace_bytes(1, n, m));
  const size_t bf = Carver::pad(gp_fit_ws_bytes(1, d, m, n_restarts));
  const size_t bi = Carver::pad(sizeof(long long) * m), bd = Carver::pad(sizeof(double) * m);
  const size_t bo = Carver::pad(sizeof(int) * (size_t)seg_len * (size_t)i_count);
  char* ws = (char*)nngp_workspace(h, bk + bf + bi + bd + bo);
  if (!ws) return nngp_fail(h, "sweep: out of device memory");
  void* kws = ws;
  void* fws = ws + bk;
  long long* idx = (long long*)(ws + bk + bf);
  double* dist = (double*)(ws + bk + bf + bi);
  int* order = (int*)(ws + bk + bf + bi + bd);
  if (drows) {
    std::vector<ListedQuery> lq(i_count);
    for (int c = 0; c < i_count; c++)
      lq[c] = ListedQuery{d_u_next + (long long)(i_first + c) * d, drows + (size_t)c * m, nullptr, dist, (double*)fws,
                          nullptr, m, m};
    if (!(dlq = (const ListedQuery*)upload_table(h, 4, lq.data(), sizeof(ListedQuery) * lq.size(), st)))
      return nngp_fail(h, "sweep_listed: out of memory for the query table");
  }
  if (int rc = ensure_done_zero(h, h->done, fws, 1, d, m, n_restarts, st)) return rc;
  // queue order of every predict of the call in one launch (the starts are all known up front); with dl = d the
  // blocks of consecutive predicts are contiguous, with dl < d there is one
  const signed char* starts_first = d_starts + (size_t)(i_first - I) * per_predict;
  if (int rc = gp_order_launch(h, starts_first + (size_t)j0 * nruns * 2, i_count, seg_len, 0, order, st)) return rc;
  for (int i = i_first; i < i_first + i_count; i++) {
    double* ui = d_u_next + (long long)i * d;
    double* un = d_u_next + (long long)(i + 1) * d;
    double* gn = d_uG_next + (long long)(i + 1) * d;
    if (int rc = sweep_slice_prologue(h, *s, method_g, h_mode, steps_g, 1, d_t + i, d_t + i + 1, ui, d, gn, st, [&] {
          if (dlq) return listed_prep_launch(h, dlq + (i - i_first), 1, st);
          return knn_prep_launch(h, ui, 1, m, n, idx, dist, kws, fws, st);
        }))
      return rc;
    const long long* nb = drows ? drows + (size_t)(i - i_first) * m : idx;
    if (int rc = gp_fit_predict_launch(h, nb, dist, fws, next_queue(h, st), order + (size_t)(i - i_first) * seg_len, 1, m,
                                       n_restarts, starts_first + (size_t)(i - i_first) * per_predict, fatol, xatol, un,
                                       gn, d, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, st, j0, dl))
      return rc;
  }
  return 0;
}

int nngp_sweep_shard(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g,
                     const double* d_t, int N, int I, int i_first, int i_count, int m, int n_restarts,
                     const signed char* d_starts, double fatol, double xatol, double* d_u_next,
                     double* d_uG_next, int d, int j0, int dl, void* stream) {
  return sweep_shard_impl(h, sys, method_g, h_mode, steps_g, d_t, N, I, i_first, i_count, m, nullptr, n_restarts,
                          d_starts, fatol, xatol, d_u_next, d_uG_next, d, j0, dl, stream);
}

int nngp_sweep_listed_shard(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g,
                            const double* d_t, int N, int I, int i_first, int i_count, int m, const long long* rows,
                            int n_restarts, const signed char* d_starts, double fatol, double xatol,
                            double* d_u_next, double* d_uG_next, int d, int j0, int dl, void* stream) {
  if (rows == nullptr) return nngp_fail(h, "sweep_listed: rows is NULL");
  return sweep_shard_impl(h, sys, method_g, h_mode, steps_g, d_t, N, I, i_first, i_count, m, rows, n_restarts,
                          d_starts, fatol, xatol, d_u_next, d_uG_next, d, j0, dl, stream);
}

// ---- ensembles: segmented store, segmented kNN, ensemble sweep -------------------------
int nngp_seg_reserve(nngp_handle_t h, int n_members, long long cap_rows, int d) {
  NNGP_USE_DEVICE(h);
  if (n_members < 1 || cap_rows < 1 || d < 1)
    return nngp_fail(h, "seg_reserve: n_members=%d cap_rows=%lld d=%d", n_members, cap_rows, d);
  const bool same = h->ds_x && h->seg_E == n_members && h->ds_d == d;
  if (same && h->seg_cap >= cap_rows) return 0;
  if (h->seg_E > 0 && !same)
    for (long long r : h->seg_rows)
      if (r > 0) return nngp_fail(h, "seg_reserve: layout change (%d members, d=%d) with rows held", n_members, d);
  NNGP_CUDA(h, cudaDeviceSynchronize());
  double *nx = nullptr, *ny = nullptr, *nxt = nullptr;
  const size_t bytes = sizeof(double) * (size_t)n_members * (size_t)cap_rows * d;
  NNGP_CUDA(h, cudaMalloc(&nx, bytes));
  NNGP_CUDA(h, cudaMalloc(&ny, bytes));
  NNGP_CUDA(h, cudaMalloc(&nxt, bytes));
  double *ox = h->ds_x, *oy = h->ds_y, *oxt = h->ds_xt;
  const long long ocap = h->seg_cap;
  h->ds_x = nx; h->ds_y = ny; h->ds_xt = nxt;
  h->ds_d = d; h->ds_cap = (long long)n_members * cap_rows; h->ds_rows = 0;
  h->seg_E = n_members; h->seg_cap = cap_rows;
  if (!same) h->seg_rows.assign(n_members, 0);
  // growth: every member's rows move to the start of its new segment (X, Y and the transposed copy)
  std::vector<long long> tab;
  long long max_rows = 0;
  for (int e = 0; same && e < n_members; e++) {
    const long long r = h->seg_rows[e];
    if (r == 0) continue;
    tab.insert(tab.end(), {(long long)e * ocap * d, (long long)e * ocap * d, r, (long long)e * cap_rows});
    max_rows = std::max(max_rows, r);
  }
  if (!tab.empty()) {
    const long long* dtab = (const long long*)upload_table(h, 0, tab.data(), sizeof(long long) * tab.size(), nullptr);
    if (!dtab) return nngp_fail(h, "seg_reserve: out of memory for the copy table");
    if (int rc = append_seg_launch(h, ox, oy, nullptr, d, dtab, (int)(tab.size() / 4), max_rows, nullptr)) return rc;
    NNGP_CUDA(h, cudaDeviceSynchronize());
  }
  if (ox) cudaFree(ox);
  if (oy) cudaFree(oy);
  if (oxt) cudaFree(oxt);
  return 0;
}

int nngp_seg_reset(nngp_handle_t h) {
  h->seg_rows.assign(h->seg_E, 0);
  return 0;
}

long long nngp_seg_rows(nngp_handle_t h, int member) {
  if (member < 0 || member >= h->seg_E) return -1;
  return h->seg_rows[member];
}

long long nngp_seg_cap(nngp_handle_t h) { return h->seg_cap; }

int nngp_seg_append_iteration(nngp_handle_t h, int n, const int* members, const int* I, const double* d_u_cur,
                              const double* d_uF, const double* d_uG_cur, long long ld_state, int N, int d,
                              void* stream) {
  NNGP_USE_DEVICE(h);
  if (n <= 0) return 0;
  if (h->seg_E < 1) return nngp_fail(h, "seg_append_iteration: no segmented store (call nngp_seg_reserve)");
  if (d != h->ds_d) return nngp_fail(h, "seg_append_iteration: d=%d but store d=%d", d, h->ds_d);
  if (ld_state < (long long)(N + 1) * d) return nngp_fail(h, "seg_append_iteration: ld_state=%lld < (N+1) d", ld_state);
  std::vector<long long> tab;
  tab.reserve(4 * (size_t)n);
  long long max_rows = 0;
  for (int p = 0; p < n; p++) {
    const int e = members[p];
    if (e < 0 || e >= h->seg_E) return nngp_fail(h, "seg_append_iteration: member %d outside [0,%d)", e, h->seg_E);
    if (I[p] < 1 || I[p] > N) return nngp_fail(h, "seg_append_iteration: I=%d outside [1,%d]", I[p], N);
    const long long rows = (long long)N - I[p] + 1;
    if (h->seg_rows[e] + rows > h->seg_cap)
      return nngp_fail(h, "seg_append_iteration: member %d: %lld + %lld rows > capacity %lld", e, h->seg_rows[e], rows,
                       h->seg_cap);
    const long long so = (long long)p * ld_state;
    tab.insert(tab.end(), {so + (long long)(I[p] - 1) * d, so + (long long)I[p] * d, rows,
                           (long long)e * h->seg_cap + h->seg_rows[e]});
    max_rows = std::max(max_rows, rows);
  }
  cudaStream_t st = as_stream(stream);
  const long long* dtab = (const long long*)upload_table(h, 0, tab.data(), sizeof(long long) * tab.size(), st);
  if (!dtab) return nngp_fail(h, "seg_append_iteration: out of memory for the row table");
  if (int rc = append_seg_launch(h, d_u_cur, d_uF, d_uG_cur, d, dtab, n, max_rows, st)) return rc;
  for (int p = 0; p < n; p++) h->seg_rows[members[p]] += (long long)N - I[p] + 1;
  return 0;
}

int nngp_knn_segmented(nngp_handle_t h, const double* d_q, long long ld_q, int nq, int m, const long long* base,
                       const long long* rows, long long* d_idx, double* d_dist, double* d_r2, void* stream) {
  NNGP_USE_DEVICE(h);
  if (nq <= 0) return 0;
  if (!h->ds_x) return nngp_fail(h, "knn_segmented: no store");
  if (ld_q < h->ds_d) return nngp_fail(h, "knn_segmented: ld_q=%lld < d=%d", ld_q, h->ds_d);
  std::vector<long long> tab(2 * (size_t)nq);
  long long n_max = 0;
  for (int q = 0; q < nq; q++) {
    if (rows[q] < m) return nngp_fail(h, "knn_segmented: query %d: segment of %lld rows, fewer than m=%d", q, rows[q], m);
    if (base[q] < 0 || base[q] + rows[q] > h->ds_cap)
      return nngp_fail(h, "knn_segmented: query %d: rows [%lld,%lld) outside the store (%lld)", q, base[q],
                       base[q] + rows[q], h->ds_cap);
    tab[q] = base[q];
    tab[nq + q] = rows[q];
    n_max = std::max(n_max, rows[q]);
  }
  cudaStream_t st = as_stream(stream);
  void* ws = nngp_workspace(h, knn_seg_workspace_bytes(nq, n_max, m));
  unsigned int* tickets = seg_tickets(h, nq);
  if (!ws || !tickets) return nngp_fail(h, "knn_segmented: out of device memory");
  const long long* dtab = (const long long*)upload_table(h, 1, tab.data(), sizeof(long long) * tab.size(), st);
  if (!dtab) return nngp_fail(h, "knn_segmented: out of memory for the segment table");
  return knn_seg_launch(h, d_q, ld_q, nq, m, dtab, dtab + nq, n_max, d_idx, d_dist, d_r2, tickets, ws, st);
}

int nngp_copy_rows(nngp_handle_t h, const double* d_src, const long long* d_src_idx, double* d_dst,
                   const long long* d_dst_idx, long long rows, long long d, void* stream) {
  NNGP_USE_DEVICE(h);
  return copy_rows_launch(h, d_src, d_src_idx, d_dst, d_dst_idx, rows, d, as_stream(stream));
}

// t_rep[i, p] = t_pos[p, i]: row i holds the slice boundaries t_i of every position, so the coarse step of the first n
// positions at slice i reads its t0 and t1 from rows i and i + 1
__global__ void transpose_t_kernel(const double* __restrict__ t_pos, int n_t, int E, double* __restrict__ t_rep) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < (long long)n_t * E) {
    const long long i = e / E, p = e - i * E;
    t_rep[e] = t_pos[p * n_t + i];
  }
}

// `rows` rows of `bytes` bytes, row r from src + r src_ld to dst + r dst_ld (strides in bytes)
struct CopySpan {
  const char* src;
  char* dst;
  long long src_ld, dst_ld;
  int bytes, rows;
};

// one warp per span; 8-byte words when every address and stride allows it
__global__ void __launch_bounds__(256) copy_spans_kernel(const CopySpan* __restrict__ sp, int n) {
  const int s = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (s >= n) return;
  const CopySpan x = sp[s];
  const bool w8 = ((((unsigned long long)x.src | (unsigned long long)x.dst | (unsigned long long)x.src_ld |
                     (unsigned long long)x.dst_ld | (unsigned long long)x.bytes) & 7ull) == 0);
  for (int r = 0; r < x.rows; r++) {
    const char* a = x.src + r * x.src_ld;
    char* b = x.dst + r * x.dst_ld;
    if (w8) {
      for (int k = lane; k < x.bytes / 8; k += 32) ((long long*)b)[k] = ((const long long*)a)[k];
    } else {
      for (int k = lane; k < x.bytes; k += 32) b[k] = a[k];
    }
  }
}

static int copy_spans_launch(nngp_handle_t h, const CopySpan* d_sp, int n, cudaStream_t st) {
  if (n <= 0) return 0;
  ProfScope prof(h, 4, st);
  copy_spans_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(d_sp, n);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

static CopySpan copy_span(const void* src, void* dst, size_t bytes, int rows = 1, long long src_ld = 0, long long dst_ld = 0) {
  return CopySpan{(const char*)src, (char*)dst, src_ld, dst_ld, (int)bytes, rows};
}

// The predicts of a fit with one neighbour count per predict, grouped by count: group g holds the positions pos[g]
// (ascending) whose count is m[g].  Each group gets compact inputs (neighbour rows, matrix, starts, the added term)
// and its own fit workspace, so its fit is an ordinary launch at m[g] over exactly what a solo fit at m[g] reads.
// One fit per distinct m, not one per template size: the objective's determinant product is split at M/2 and
// the padding rows' pivots enter it, so the bits of a search depend on the template size M as well as on m.
struct MixedGroups {
  std::vector<int> m;
  std::vector<std::vector<int>> pos;
  std::vector<int> grp, rank;  // position -> group, rank in its group
  struct Dev {
    char* fws;
    int* order;
    long long* idx;
    double *dist, *add, *pred, *theta_opt, *jitter_opt, *fval_opt, *fvals, *thetas;
    int* nfev;
    signed char* starts;
    DoneTracker done;
  };
  std::vector<Dev> dev;

  MixedGroups(const int* m_pos, int n) : grp(n), rank(n) {
    std::vector<int> ms(m_pos, m_pos + n);
    std::sort(ms.begin(), ms.end());
    ms.erase(std::unique(ms.begin(), ms.end()), ms.end());
    m = ms;
    pos.resize(m.size());
    for (int p = 0; p < n; p++) {
      const int g = (int)(std::lower_bound(m.begin(), m.end(), m_pos[p]) - m.begin());
      grp[p] = g;
      rank[p] = (int)pos[g].size();
      pos[g].push_back(p);
    }
    dev.resize(m.size());
  }
  // device bytes of every group's block (details: the per-search outputs of nngp_fit_predict too)
  size_t bytes(int d, int R, bool details) const {
    size_t t = 0;
    for (size_t g = 0; g < m.size(); g++) t += group_bytes((int)g, d, R, details, nullptr);
    return t;
  }
  void carve(char* base, int d, int R, bool details) {
    for (size_t g = 0; g < m.size(); g++) {
      dev[g].fws = base;
      base += group_bytes((int)g, d, R, details, &dev[g]);
    }
  }
  size_t group_bytes(int g, int d, int R, bool details, Dev* out) const {
    const size_t n = pos[g].size(), mg = m[g], nt = n * d * NNGP_N_JITTER * R;
    size_t off = 0;
    auto take = [&](size_t b) { const size_t o = off; off += Carver::pad(b); return o; };
    const size_t o_f = take(gp_fit_ws_bytes((int)n, d, (int)mg, R)), o_o = take(sizeof(int) * nt),
                 o_i = take(sizeof(long long) * n * mg), o_d = take(sizeof(double) * n * mg), o_s = take(2 * nt),
                 o_a = take(sizeof(double) * n * d), o_p = take(sizeof(double) * n * d);
    size_t o_th = 0, o_j = 0, o_fv = 0, o_nf = 0, o_fs = 0, o_ts = 0;
    if (details) {
      o_th = take(sizeof(double) * n * d * 2); o_j = take(sizeof(double) * n * d); o_fv = take(sizeof(double) * n * d);
      o_nf = take(sizeof(int) * nt); o_fs = take(sizeof(double) * nt); o_ts = take(sizeof(double) * nt * 2);
    }
    if (out) {
      char* b = out->fws;  // the group's base (carve)
      out->order = (int*)(b + o_o); out->idx = (long long*)(b + o_i); out->dist = (double*)(b + o_d);
      out->starts = (signed char*)(b + o_s); out->add = (double*)(b + o_a); out->pred = (double*)(b + o_p);
      out->theta_opt = details ? (double*)(b + o_th) : nullptr;
      out->jitter_opt = details ? (double*)(b + o_j) : nullptr;
      out->fval_opt = details ? (double*)(b + o_fv) : nullptr;
      out->nfev = details ? (int*)(b + o_nf) : nullptr;
      out->fvals = details ? (double*)(b + o_fs) : nullptr;
      out->thetas = details ? (double*)(b + o_ts) : nullptr;
      out->fws = b + o_f;
      out->done = DoneTracker{};
    }
    return off;
  }
};
// order + fit of the first n active predicts of group g (compact inputs already gathered); pred += add when add_on
static int mixed_fit_group(nngp_handle_t h, MixedGroups& G, int g, int n, int d, int R, double fatol, double xatol,
                           bool add_on, cudaStream_t st) {
  MixedGroups::Dev& D = G.dev[g];
  const int mg = G.m[g], seg_len = d * NNGP_N_JITTER * R;
  if (int rc = ensure_done_zero(h, D.done, D.fws, n, d, mg, R, st)) return rc;
  if (int rc = gp_order_launch(h, D.starts, n, seg_len, 1, D.order, st)) return rc;
  return gp_fit_predict_launch(h, D.idx, D.dist, D.fws, next_queue(h, st), D.order, n, mg, R, D.starts, fatol, xatol,
                               D.pred, add_on ? D.add : nullptr, d, D.theta_opt, D.jitter_opt, D.fval_opt, D.nfev,
                               D.fvals, D.thetas, st);
}

// The copies that hand predict p (rank r of group g) its inputs: the first m_g neighbours of row `src` of the kNN at
// row stride mm, the leading m_g x m_g block of its mm x mm neighbour matrix (idx == nullptr: these three are already
// in place, written by the listed prep), its starts and (optional) added term.
static void mixed_gather_spans(std::vector<CopySpan>& sp, MixedGroups& G, int p, int src, const long long* idx,
                               const double* dist, const double* r2, int mm, const signed char* starts, size_t per_predict,
                               const double* add, long long ld_add, int d) {
  const int g = G.grp[p], r = G.rank[p], mg = G.m[g];
  const MixedGroups::Dev& D = G.dev[g];
  if (idx) {
    sp.push_back(copy_span(idx + (size_t)src * mm, D.idx + (size_t)r * mg, sizeof(long long) * mg));
    sp.push_back(copy_span(dist + (size_t)src * mm, D.dist + (size_t)r * mg, sizeof(double) * mg));
    sp.push_back(copy_span(r2 + (size_t)src * mm * mm, D.fws + sizeof(double) * (size_t)r * mg * mg, sizeof(double) * mg,
                           mg, (long long)sizeof(double) * mm, (long long)sizeof(double) * mg));
  }
  sp.push_back(copy_span(starts + (size_t)p * per_predict, D.starts + (size_t)r * per_predict, per_predict));
  if (add) sp.push_back(copy_span(add + (size_t)p * ld_add, D.add + (size_t)r * d, sizeof(double) * d));
}

int nngp_fit_predict_mixed(nngp_handle_t h, const double* d_q, const long long* d_idx, const double* d_dist, int nq,
                           const int* m, int n_restarts, const signed char* d_starts, double fatol, double xatol,
                           double* d_pred, double* d_theta_opt, double* d_jitter_opt, double* d_fval_opt, int* d_nfev,
                           double* d_fvals, double* d_thetas, void* stream) {
  NNGP_USE_DEVICE(h);
  (void)d_q;
  if (nq <= 0) return 0;
  if (n_restarts < 1) return nngp_fail(h, "fit_mixed: n_restarts=%d < 1", n_restarts);
  int ld = 0;
  for (int q = 0; q < nq; q++) {
    if (m[q] < 1 || m[q] > NNGP_MAX_NEIGHBOURS_BIG)
      return nngp_fail(h, "fit_mixed: predict %d: m=%d outside [1,%d]", q, m[q], NNGP_MAX_NEIGHBOURS_BIG);
    ld = std::max(ld, m[q]);
  }
  const int d = h->ds_d, R = n_restarts, seg_len = d * NNGP_N_JITTER * R;
  const size_t per_predict = (size_t)seg_len * 2;
  MixedGroups G(m, nq);
  const size_t br = Carver::pad(gp_prep_bytes(nq, ld));
  char* ws = (char*)nngp_workspace(h, br + G.bytes(d, R, true));
  if (!ws) return nngp_fail(h, "fit_mixed: out of device memory");
  G.carve(ws + br, d, R, true);
  double* r2 = (double*)ws;
  std::vector<CopySpan> sp;
  for (int q = 0; q < nq; q++) mixed_gather_spans(sp, G, q, q, d_idx, d_dist, r2, ld, d_starts, per_predict, nullptr, 0, d);
  const size_t n_gather = sp.size();
  const size_t nd = sizeof(double) * d, nt = (size_t)seg_len;
  for (int q = 0; q < nq; q++) {
    const int r = G.rank[q];
    const MixedGroups::Dev& D = G.dev[G.grp[q]];
    sp.push_back(copy_span(D.pred + (size_t)r * d, d_pred + (size_t)q * d, nd));
    if (d_theta_opt) sp.push_back(copy_span(D.theta_opt + (size_t)r * 2 * d, d_theta_opt + (size_t)q * 2 * d, 2 * nd));
    if (d_jitter_opt) sp.push_back(copy_span(D.jitter_opt + (size_t)r * d, d_jitter_opt + (size_t)q * d, nd));
    if (d_fval_opt) sp.push_back(copy_span(D.fval_opt + (size_t)r * d, d_fval_opt + (size_t)q * d, nd));
    if (d_nfev) sp.push_back(copy_span(D.nfev + r * nt, d_nfev + q * nt, sizeof(int) * nt));
    if (d_fvals) sp.push_back(copy_span(D.fvals + r * nt, d_fvals + q * nt, sizeof(double) * nt));
    if (d_thetas) sp.push_back(copy_span(D.thetas + r * nt * 2, d_thetas + q * nt * 2, sizeof(double) * nt * 2));
  }
  cudaStream_t st = as_stream(stream);
  const CopySpan* dsp = (const CopySpan*)upload_table(h, 2, sp.data(), sizeof(CopySpan) * sp.size(), st);
  if (!dsp) return nngp_fail(h, "fit_mixed: out of memory for the copy table");
  if (int rc = gp_prep_launch(h, d_idx, nq, ld, r2, st)) return rc;
  if (int rc = copy_spans_launch(h, dsp, (int)n_gather, st)) return rc;
  for (size_t g = 0; g < G.m.size(); g++)
    if (int rc = mixed_fit_group(h, G, (int)g, (int)G.pos[g].size(), d, R, fatol, xatol, false, st)) return rc;
  return copy_spans_launch(h, dsp + n_gather, (int)(sp.size() - n_gather), st);
}

// One slice of an ensemble sweep, planned before anything is enqueued: the active positions (a prefix, n_act), the kNN
// positions among them (the first nk_act of the sweep's kNN positions, searched at their largest m, mm, over segments
// of at most n_max rows), the starts of its first predict and, on the grouped route, where its gather and scatter
// copies and its listed preps lie in the sweep's tables.
struct SlicePlan {
  int n_act, nk_act, mm;
  long long n_max;
  const signed char* starts;
  size_t gather, scatter, end;  // copies: gather [gather, scatter), scatter [scatter, end)
  size_t lq, lq_end;            // listed preps [lq, lq_end)
};

int nngp_ensemble_sweep(nngp_handle_t h, int sys, int method_g, int h_mode, long long steps_g, const double* d_t_pos,
                        int N, int E, const int* members, const int* I, const int* m, const int* listed,
                        const long long* rows, int n_restarts, const signed char* d_starts, double fatol, double xatol,
                        double* d_u_next, double* d_uG_next, int d, void* stream) {
  NNGP_USE_DEVICE(h);
  const SystemDesc* s;
  if (int rc = get_sys(h, sys, &s)) return rc;
  if (h->seg_E < 1) return nngp_fail(h, "ensemble_sweep: no segmented store (call nngp_seg_reserve)");
  if (d != s->d || d != h->ds_d) return nngp_fail(h, "ensemble_sweep: d=%d, system d=%d, store d=%d", d, s->d, h->ds_d);
  if (E < 1) return nngp_fail(h, "ensemble_sweep: E=%d < 1", E);
  if (n_restarts < 1) return nngp_fail(h, "ensemble_sweep: n_restarts=%d < 1", n_restarts);
  if (m == nullptr || d_t_pos == nullptr) return nngp_fail(h, "ensemble_sweep: m and d_t_pos are required");
  auto is_listed = [&](int p) { return listed != nullptr && listed[p] != 0; };
  // per position: the kNN positions in position order, where a listed position's block of `rows` starts, and what
  // sizes the workspace
  std::vector<int> kpos;
  std::vector<size_t> row_at(E, 0);
  size_t n_listed_rows = 0;
  int n_sw = 0, m_max = 0;  // positions that sweep at least one slice, their largest m
  long long n_max_all = 0;
  bool in_place = true;  // the route: no swept position is listed and all of them share one m
  for (int p = 0; p < E; p++) {
    const int e = members[p];
    if (m[p] < 1 || m[p] > NNGP_MAX_NEIGHBOURS_BIG)
      return nngp_fail(h, "ensemble_sweep: position %d: m=%d outside [1,%d]", p, m[p], NNGP_MAX_NEIGHBOURS_BIG);
    if (e < 0 || e >= h->seg_E) return nngp_fail(h, "ensemble_sweep: member %d outside [0,%d)", e, h->seg_E);
    if (I[p] < 0 || I[p] > N || (p > 0 && I[p] < I[p - 1]))
      return nngp_fail(h, "ensemble_sweep: I must be ascending in [0,%d] (position %d: %d)", N, p, I[p]);
    n_max_all = std::max(n_max_all, h->seg_rows[e]);
    if (is_listed(p)) {
      row_at[p] = n_listed_rows;
      n_listed_rows += (size_t)(N - I[p]) * m[p];
    } else {
      kpos.push_back(p);
    }
    if (I[p] < N) {
      n_sw++;
      m_max = std::max(m_max, m[p]);
      in_place = in_place && !is_listed(p) && m[p] == m[0];
    }
  }
  if (n_listed_rows > 0 && rows == nullptr) return nngp_fail(h, "ensemble_sweep: rows is NULL");
  if (I[0] >= N) return 0;
  const int nk = (int)kpos.size(), seg_len = d * NNGP_N_JITTER * n_restarts;
  const size_t per_predict = (size_t)seg_len * 2;
  const long long ld = (long long)(N + 1) * d;
  // in place: the kNN writes its neighbour matrices into the fit's block; grouped: they get their own block (br) and
  // the fits work in the groups' blocks
  MixedGroups G(m, in_place ? 0 : n_sw);
  const size_t bk = Carver::pad(knn_seg_workspace_bytes(E, n_max_all, m_max));
  const size_t br = Carver::pad(gp_prep_bytes(E, m_max));
  const size_t bf = in_place ? Carver::pad(gp_fit_ws_bytes(E, d, m_max, n_restarts)) : br + G.bytes(d, n_restarts, false);
  const size_t bi = Carver::pad(sizeof(long long) * (size_t)E * m_max), bd = Carver::pad(sizeof(double) * (size_t)E * m_max);
  const size_t bo = Carver::pad(sizeof(int) * (size_t)E * seg_len);
  const size_t bt = Carver::pad(sizeof(double) * (size_t)(N + 1) * E);
  const size_t bq = listed ? Carver::pad(sizeof(double) * (size_t)nk * d) : 0;  // gathered kNN queries
  char* ws = (char*)nngp_workspace(h, bk + bf + bi + bd + bo + bt + bq);
  if (!ws) return nngp_fail(h, "ensemble_sweep: out of device memory");
  void* kws = ws;
  void* fws = ws + bk;
  long long* idx = (long long*)(ws + bk + bf);
  double* dist = (double*)(ws + bk + bf + bi);
  int* order = (int*)(ws + bk + bf + bi + bd);
  double* t_rep = (double*)(ws + bk + bf + bi + bd + bo);
  double* q_knn = (double*)(ws + bk + bf + bi + bd + bo + bt);
  if (!in_place) G.carve(ws + bk + br, d, n_restarts, false);
  // The plan, in one pass over the slices.  The positions active at slice i (I <= i) are a prefix: every launch reaches
  // them with the member stride (N+1) d of the state, and their predicts' starts are consecutive in d_starts
  // (slice-major).  Grouped: every slice's gather and scatter copies go to one table for the whole sweep, its listed
  // preps (which write straight into their fit groups' inputs) to another, followed by the gathers of the kNN queries
  // when the slice has listed positions (its kNN positions are then no prefix of the state).
  std::vector<SlicePlan> plan;
  std::vector<CopySpan> sp;
  std::vector<ListedQuery> lq;  // `rows` of an entry points into the host lists until they are uploaded
  int n_act = 0, nk_act = 0, mm = 0, short_p = -1;
  long long n_max = 0;
  const signed char* starts_i = d_starts;
  for (int i = I[0]; i < N; i++) {
    for (; n_act < E && I[n_act] <= i; n_act++) {
      if (is_listed(n_act)) continue;
      const long long held = h->seg_rows[members[n_act]];
      mm = std::max(mm, m[n_act]);
      n_max = std::max(n_max, held);
      if (short_p < 0 || held < h->seg_rows[members[short_p]]) short_p = n_act;
      nk_act++;
    }
    // the kNN searches at the slice's largest m: a shorter segment would read padding indices as rows
    if (short_p >= 0 && h->seg_rows[members[short_p]] < mm)
      return nngp_fail(h, "ensemble_sweep: member %d holds %lld rows, fewer than m=%d, the largest m of slice %d",
                       members[short_p], h->seg_rows[members[short_p]], mm, i);
    SlicePlan P{n_act, nk_act, mm, n_max, starts_i, sp.size(), sp.size(), sp.size(), lq.size(), lq.size()};
    if (!in_place) {
      const double* ui = d_u_next + (long long)i * d;
      const double* gn = d_uG_next + (long long)(i + 1) * d;
      double* un = d_u_next + (long long)(i + 1) * d;
      for (int p = 0, rk = 0; p < n_act; p++) {
        if (!is_listed(p)) {
          mixed_gather_spans(sp, G, p, rk++, idx, dist, (const double*)fws, mm, starts_i, per_predict, gn, ld, d);
          continue;
        }
        const int r = G.rank[p], mg = m[p];
        const MixedGroups::Dev& D = G.dev[G.grp[p]];
        const long long base = (long long)members[p] * h->seg_cap, held = h->seg_rows[members[p]];
        const long long* lr = rows + row_at[p] + (size_t)(i - I[p]) * mg;
        for (int a = 0; a < mg; a++)
          if (lr[a] < base || lr[a] >= base + held)
            return nngp_fail(h, "ensemble_sweep: member %d, slice %d lists row %lld, outside its segment [%lld,%lld)",
                             members[p], i, lr[a], base, base + held);
        lq.push_back(ListedQuery{ui + p * ld, lr, D.idx + (size_t)r * mg, D.dist + (size_t)r * mg,
                                 (double*)D.fws + (size_t)r * mg * mg, nullptr, mg, mg});
        mixed_gather_spans(sp, G, p, 0, nullptr, nullptr, nullptr, 0, starts_i, per_predict, gn, ld, d);
      }
      if (lq.size() > P.lq)
        for (int r = 0; r < nk_act; r++)
          lq.push_back(ListedQuery{ui + kpos[r] * ld, nullptr, nullptr, nullptr, nullptr, q_knn + (size_t)r * d, 0, 0});
      P.scatter = sp.size();
      for (int p = 0; p < n_act; p++)
        sp.push_back(copy_span(G.dev[G.grp[p]].pred + (size_t)G.rank[p] * d, un + (size_t)p * ld, sizeof(double) * d));
      P.end = sp.size();
      P.lq_end = lq.size();
    }
    plan.push_back(P);
    starts_i += (size_t)n_act * per_predict;
  }
  cudaStream_t st = as_stream(stream);
  unsigned int* tickets = seg_tickets(h, E);
  if (!tickets) return nngp_fail(h, "ensemble_sweep: out of device memory");
  std::vector<long long> ktab(2 * (size_t)nk);  // [base | rows] of the kNN positions' segments
  for (int r = 0; r < nk; r++) {
    ktab[r] = (long long)members[kpos[r]] * h->seg_cap;
    ktab[nk + r] = h->seg_rows[members[kpos[r]]];
  }
  const long long* dtab = nullptr;
  if (nk > 0 && !(dtab = (const long long*)upload_table(h, 1, ktab.data(), sizeof(long long) * ktab.size(), st)))
    return nngp_fail(h, "ensemble_sweep: out of memory for the segment table");
  if (n_listed_rows > 0) {
    const long long* drows = (const long long*)upload_table(h, 3, rows, sizeof(long long) * n_listed_rows, st);
    if (!drows) return nngp_fail(h, "ensemble_sweep: out of memory for the neighbour lists");
    for (ListedQuery& q : lq)
      if (q.rows) q.rows = drows + (q.rows - rows);
  }
  const CopySpan* dsp = nullptr;
  if (!sp.empty() && !(dsp = (const CopySpan*)upload_table(h, 2, sp.data(), sizeof(CopySpan) * sp.size(), st)))
    return nngp_fail(h, "ensemble_sweep: out of memory for the copy table");
  const ListedQuery* dlq = nullptr;
  if (!lq.empty() && !(dlq = (const ListedQuery*)upload_table(h, 4, lq.data(), sizeof(ListedQuery) * lq.size(), st)))
    return nngp_fail(h, "ensemble_sweep: out of memory for the query table");
  {
    const long long tot = (long long)(N + 1) * E;
    transpose_t_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d_t_pos, N + 1, E, t_rep);
    h->launches++;
    NNGP_CUDA(h, cudaGetLastError());
  }
  for (size_t k = 0; k < plan.size(); k++) {
    const SlicePlan& P = plan[k];
    const int i = I[0] + (int)k;
    double* ui = d_u_next + (long long)i * d;
    double* un = d_u_next + (long long)(i + 1) * d;
    double* gn = d_uG_next + (long long)(i + 1) * d;
    const double* t0 = t_rep + (size_t)i * E;
    if (in_place) {
      // the queue order needs only the starts: enqueued first, it stays off the path from the kNN to the fit
      if (int rc = ensure_done_zero(h, h->done, fws, P.n_act, d, P.mm, n_restarts, st)) return rc;
      if (int rc = gp_order_launch(h, P.starts, P.n_act, seg_len, 1, order, st)) return rc;
      if (int rc = sweep_slice_prologue(h, *s, method_g, h_mode, steps_g, P.n_act, t0, t0 + E, ui, ld, gn, st, [&] {
            return knn_seg_launch(h, ui, ld, P.n_act, P.mm, dtab, dtab + nk, P.n_max, idx, dist, (double*)fws, tickets,
                                  kws, st);
          }))
        return rc;
      if (int rc = gp_fit_predict_launch(h, idx, dist, fws, next_queue(h, st), order, P.n_act, P.mm, n_restarts,
                                         P.starts, fatol, xatol, un, gn, ld, nullptr, nullptr, nullptr, nullptr, nullptr,
                                         nullptr, st))
        return rc;
      continue;
    }
    const int nl = (int)(P.lq_end - P.lq);
    if (int rc = sweep_slice_prologue(h, *s, method_g, h_mode, steps_g, P.n_act, t0, t0 + E, ui, ld, gn, st, [&] {
          if (int rc = listed_prep_launch(h, dlq + P.lq, nl, st)) return rc;
          if (P.nk_act == 0) return 0;
          return knn_seg_launch(h, nl ? q_knn : ui, nl ? d : ld, P.nk_act, P.mm, dtab, dtab + nk, P.n_max, idx, dist,
                                (double*)fws, tickets, kws, st);
        }))
      return rc;
    if (int rc = copy_spans_launch(h, dsp + P.gather, (int)(P.scatter - P.gather), st)) return rc;
    for (size_t g = 0; g < G.m.size(); g++) {
      const int n_g = (int)(std::lower_bound(G.pos[g].begin(), G.pos[g].end(), P.n_act) - G.pos[g].begin());
      if (n_g > 0)
        if (int rc = mixed_fit_group(h, G, (int)g, n_g, d, n_restarts, fatol, xatol, true, st)) return rc;
    }
    if (int rc = copy_spans_launch(h, dsp + P.scatter, (int)(P.end - P.scatter), st)) return rc;
  }
  return 0;
}

int nngp_selftest_math(nngp_handle_t h, const double* d_x, int n, double* d_exp_neg, double* d_rcp,
                       double* d_exp10, void* stream) {
  NNGP_USE_DEVICE(h);
  return selftest_math_launch(h, d_x, n, d_exp_neg, d_rcp, d_exp10, as_stream(stream));
}

// ---- roofline micro-benchmarks ---------------------------------------------------------
__global__ void fp64_fma_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5,
         x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

int nngp_bench_fp64(nngp_handle_t h, int iters, double* tflops_out) {
  NNGP_USE_DEVICE(h);
  const int blocks = 148 * 8, threads = 256;
  double* out = (double*)nngp_workspace(h, sizeof(double) * blocks * threads);
  if (!out) return nngp_fail(h, "bench_fp64: out of memory");
  cudaEvent_t e0, e1;
  NNGP_CUDA(h, cudaEventCreate(&e0));
  NNGP_CUDA(h, cudaEventCreate(&e1));
  fp64_fma_kernel<<<blocks, threads, 0, h->own_stream>>>(out, iters, 0.999999, 1e-7);
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    NNGP_CUDA(h, cudaEventRecord(e0, h->own_stream));
    fp64_fma_kernel<<<blocks, threads, 0, h->own_stream>>>(out, iters, 0.999999, 1e-7);
    NNGP_CUDA(h, cudaEventRecord(e1, h->own_stream));
    NNGP_CUDA(h, cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double tf = 2.0 * 8 * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  h->launches += 6;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *tflops_out = best;
  return 0;
}

__global__ void copy_kernel(const double2* __restrict__ src, double2* __restrict__ dst, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[i];
}

int nngp_bench_copy(nngp_handle_t h, long long bytes, double* gbs_out) {
  NNGP_USE_DEVICE(h);
  const size_t n = (size_t)bytes / sizeof(double2);
  char* ws = (char*)nngp_workspace(h, 2 * n * sizeof(double2));
  if (!ws) return nngp_fail(h, "bench_copy: out of memory");
  double2* a = (double2*)ws;
  double2* b = a + n;
  NNGP_CUDA(h, cudaMemsetAsync(a, 0, n * sizeof(double2), h->own_stream));
  cudaEvent_t e0, e1;
  NNGP_CUDA(h, cudaEventCreate(&e0));
  NNGP_CUDA(h, cudaEventCreate(&e1));
  copy_kernel<<<148 * 16, 512, 0, h->own_stream>>>(a, b, n);
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    NNGP_CUDA(h, cudaEventRecord(e0, h->own_stream));
    copy_kernel<<<148 * 16, 512, 0, h->own_stream>>>(a, b, n);
    NNGP_CUDA(h, cudaEventRecord(e1, h->own_stream));
    NNGP_CUDA(h, cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double gbs = 2.0 * n * sizeof(double2) / (ms * 1e-3) / 1e9;
    if (gbs > best) best = gbs;
  }
  h->launches += 6;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *gbs_out = best;
  return 0;
}

}  // extern "C"
