// Dataset maintenance and exact FP64 nearest-neighbour search.
//
// Replaces  s_idx = np.argsort(cdist(new_x, self.x, 'sqeuclidean')[0,:]); s_idx[:nn]
// (models.py:177-179) and the dataset growth x = vstack(x, ...), D = vstack(D, ...)
// (parareal.py:336-339).
//
// Arithmetic contract (compiled with -fmad=false): a squared distance is the strict
// left-to-right sum s = ((0 + (q_0-x_0)^2) + (q_1-x_1)^2) + ... with separately rounded
// subtract, multiply and add -- SciPy's cdist arithmetic -- so the distances, and therefore
// the index sets, are bit-exact.  Neighbours are ordered by (distance, index), i.e.
// argsort(kind='stable').
//
// Layout: the dataset is kept twice, row-major X[cap,d] (row gathers for the GP) and
// transposed XT[d,cap] so that a warp scanning 32 consecutive rows reads 32 consecutive
// doubles per coordinate.  One thread owns one row (times TQ queries; the one-query kernel
// prefetches 16 coordinates ahead of the serial addition chain); selection keeps a sorted top-m
// list spread over the lanes of a warp (lane l = l-th smallest), inserts a few survivors of a
// round with ballot + shuffle and sorts / merges many with a bitonic network; warp 0 merges the
// per-warp lists; few queries over many rows select in two levels (chunks, then candidates).
// Small datasets with one to four queries (every predict of the sweep) take scan_select_tile_kernel further down:
// 16-row tiles of the row-major copy staged through shared memory, integer images of the keys, and a level 2 that
// ranks the few keys below the m-th smallest list head instead of sorting.
#include "common.cuh"

#include <algorithm>
#include <cfloat>
#include <cstdlib>

static constexpr int KNN_SEL_THREADS = 256;

// ---------------------------------------------------------------------------------------
// dataset append: X, Y row-major; XT transposed through a 32x32 shared-memory tile
// ---------------------------------------------------------------------------------------
__global__ void append_kernel(const double* __restrict__ xs, long long ldx,
                              const double* __restrict__ ya, const double* __restrict__ yb,
                              long long ldy, long long rows, int d, long long n0, long long cap,
                              double* __restrict__ X, double* __restrict__ Y,
                              double* __restrict__ XT) {
  __shared__ double tile[32][33];
  const long long r0 = (long long)blockIdx.y * 32;
  const int j0 = blockIdx.x * 32;
  for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
    const long long r = r0 + rr;
    const int j = j0 + threadIdx.x;
    if (r < rows && j < d) {
      const double xv = xs[r * ldx + j];
      X[(n0 + r) * d + j] = xv;
      tile[rr][threadIdx.x] = xv;
      double yv = ya[r * ldy + j];
      if (yb != nullptr) yv = yv - yb[r * ldy + j];
      Y[(n0 + r) * d + j] = yv;
    }
  }
  __syncthreads();
  for (int jj = threadIdx.y; jj < 32; jj += blockDim.y) {
    const int j = j0 + jj;
    const long long r = r0 + threadIdx.x;
    if (r < rows && j < d) XT[(long long)j * cap + n0 + r] = tile[threadIdx.x][jj];
  }
}

static int append_common(nngp_handle_t h, const double* xs, long long ldx, const double* ya,
                         const double* yb, long long ldy, long long rows, cudaStream_t st) {
  if (rows <= 0) return 0;
  if (h->ds_x == nullptr) return nngp_fail(h, "dataset not reserved (call nngp_dataset_reserve)");
  if (h->ds_rows + rows > h->ds_cap)
    return nngp_fail(h, "dataset capacity exceeded: %lld + %lld > %lld", h->ds_rows, rows, h->ds_cap);
  const int d = h->ds_d;
  ProfScope prof(h, 4, st);
  dim3 block(32, 8);
  dim3 grid((d + 31) / 32, (unsigned)((rows + 31) / 32));
  append_kernel<<<grid, block, 0, st>>>(xs, ldx, ya, yb, ldy, rows, d, h->ds_rows, h->ds_cap,
                                        h->ds_x, h->ds_y, h->ds_xt);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  h->ds_rows += rows;
  return 0;
}

int dataset_append_launch(nngp_handle_t h, const double* d_x, const double* d_y, long long rows,
                          cudaStream_t st) {
  return append_common(h, d_x, h->ds_d, d_y, nullptr, h->ds_d, rows, st);
}

// parareal.py:336-339: x rows u_cur[I-1 .. N-1], D rows uF[I .. N] - uG_cur[I .. N]
int append_iteration_launch(nngp_handle_t h, const double* d_u_cur, const double* d_uF,
                            const double* d_uG_cur, int N, int I, int d, cudaStream_t st) {
  if (d != h->ds_d) return nngp_fail(h, "append_iteration: d=%d but dataset d=%d", d, h->ds_d);
  if (I < 1 || I > N) return nngp_fail(h, "append_iteration: I=%d outside [1,%d]", I, N);
  const long long rows = (long long)N - I + 1;
  return append_common(h, d_u_cur + (long long)(I - 1) * d, d, d_uF + (long long)I * d,
                       d_uG_cur + (long long)I * d, d, rows, st);
}

// ---------------------------------------------------------------------------------------
// parareal.py:402  err[p] = ||a[p,:] - b[p,:]||_inf   (one warp per row)
// ---------------------------------------------------------------------------------------
__global__ void rowwise_maxabs_kernel(const double* __restrict__ a, const double* __restrict__ b,
                                      int rows, int d, double* __restrict__ err) {
  const int row = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  double mx = 0.0;
  bool nan = false;
  for (int j = lane; j < d; j += 32) {
    const double v = fabs(a[(long long)row * d + j] - b[(long long)row * d + j]);
    nan |= (v != v);
    mx = fmax(mx, v);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nan |= __shfl_xor_sync(0xffffffffu, (int)nan, o) != 0;
  }
  if (lane == 0) err[row] = nan ? __longlong_as_double(0x7ff8000000000000LL) : mx;
}

int rowwise_maxabs_launch(nngp_handle_t h, const double* a, const double* b, int rows, int d,
                          double* err, cudaStream_t st) {
  if (rows <= 0) return 0;
  const int wpb = 8;
  rowwise_maxabs_kernel<<<(rows + wpb - 1) / wpb, wpb * 32, 0, st>>>(a, b, rows, d, err);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------
// distances: thread = one dataset row x TQ queries
// ---------------------------------------------------------------------------------------
template <int TQ>
__global__ void __launch_bounds__(128)
sqdist_kernel(const double* __restrict__ XT, long long cap, long long n, int d,
              const double* __restrict__ Q, int nq, double* __restrict__ dist) {
  extern __shared__ double qs[];  // [TQ][d]
  const int q0 = blockIdx.y * TQ;
  for (int e = threadIdx.x; e < TQ * d; e += blockDim.x) {
    const int t = e / d, j = e - t * d;
    qs[e] = (q0 + t < nq) ? Q[(long long)(q0 + t) * d + j] : 0.0;
  }
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double acc[TQ];
#pragma unroll
  for (int t = 0; t < TQ; t++) acc[t] = 0.0;
  const double* xp = XT + i;
#pragma unroll 4
  for (int j = 0; j < d; j++) {
    const double x = xp[(long long)j * cap];
#pragma unroll
    for (int t = 0; t < TQ; t++) {
      const double diff = qs[t * d + j] - x;
      acc[t] = acc[t] + diff * diff;
    }
  }
#pragma unroll
  for (int t = 0; t < TQ; t++)
    if (q0 + t < nq) dist[(long long)(q0 + t) * n + i] = acc[t];
}

// One query (the sweep's case: Q = 1, n <= a few thousand rows, so only ~100 warps exist and the scan is
// latency-bound): the strict left-to-right sum is a serial chain of d additions per row, so the loads
// must run ahead of it -- PF coordinates of the row are fetched in one batch (independent loads, L2
// hits) while the previous batch is being accumulated.
template <int PF>
__global__ void __launch_bounds__(128)
sqdist_one_kernel(const double* __restrict__ XT, long long cap, long long n, int d,
                  const double* __restrict__ Q, double* __restrict__ dist) {
  extern __shared__ double qs[];  // [d]
  const double* q = Q + (long long)blockIdx.y * d;
  for (int e = threadIdx.x; e < d; e += blockDim.x) qs[e] = q[e];
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* xp = XT + i;
  double acc = 0.0;
  double cur[PF], nxt[PF];
  const int nb = d / PF;
#pragma unroll
  for (int u = 0; u < PF; u++) cur[u] = (nb > 0) ? xp[(long long)u * cap] : 0.0;
  for (int b = 0; b < nb; b++) {
    const int j0 = b * PF;
    if (b + 1 < nb) {
#pragma unroll
      for (int u = 0; u < PF; u++) nxt[u] = xp[(long long)(j0 + PF + u) * cap];
    }
#pragma unroll
    for (int u = 0; u < PF; u++) {
      const double diff = qs[j0 + u] - cur[u];
      acc = acc + diff * diff;
    }
#pragma unroll
    for (int u = 0; u < PF; u++) cur[u] = nxt[u];
  }
  for (int j = nb * PF; j < d; j++) {
    const double diff = qs[j] - xp[(long long)j * cap];
    acc = acc + diff * diff;
  }
  dist[(long long)blockIdx.y * n + i] = acc;
}

// query coordinates straight from global memory (any d)
__global__ void __launch_bounds__(128)
sqdist_kernel_gq(const double* __restrict__ XT, long long cap, long long n, int d,
                 const double* __restrict__ Q, double* __restrict__ dist) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* q = Q + (long long)blockIdx.y * d;
  double acc = 0.0;
  for (int j = 0; j < d; j++) {
    const double diff = __ldg(q + j) - XT[(long long)j * cap + i];
    acc = acc + diff * diff;
  }
  dist[(long long)blockIdx.y * n + i] = acc;
}

// ---------------------------------------------------------------------------------------
// selection: total order (isnan, distance, index)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ bool key_less(double d1, long long i1, double d2, long long i2) {
  const bool n1 = d1 != d1, n2 = d2 != d2;
  if (n1 != n2) return n2;
  if (!n1 && d1 != d2) return d1 < d2;
  return i1 < i2;
}

__device__ __forceinline__ double shfl_d(double v, int src) {
  return __shfl_sync(0xffffffffu, v, src);
}
__device__ __forceinline__ long long shfl_ll(long long v, int src) {
  return __shfl_sync(0xffffffffu, v, src);
}

// padding entries carry the index INT64_MAX and sort after every real key (NaN distances included)
__device__ __forceinline__ bool key_less_pad(double d1, long long i1, double d2, long long i2) {
  const long long IMAX = 0x7fffffffffffffffLL;
  if (i1 == IMAX) return false;
  if (i2 == IMAX) return true;
  return key_less(d1, i1, d2, i2);
}

// bitonic sort of one key per lane, ascending over the lanes
__device__ __forceinline__ void warp_sort32(double& d, long long& i, int lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const double od = __shfl_xor_sync(0xffffffffu, d, j);
      const long long oi = __shfl_xor_sync(0xffffffffu, i, j);
      const bool take_min = ((lane & k) == 0) == ((lane & j) == 0);
      const bool less = key_less_pad(od, oi, d, i);
      if (take_min == less) {
        d = od;
        i = oi;
      }
    }
  }
}

// (d, i): a sorted list per lane; (bd, bi): another sorted list.  Leaves the 32 smallest of the union, sorted.
__device__ __forceinline__ void warp_merge32(double& d, long long& i, double bd, long long bi, int lane) {
  const double rd = shfl_d(bd, 31 - lane);
  const long long ri = shfl_ll(bi, 31 - lane);
  if (key_less_pad(rd, ri, d, i)) {  // elementwise minimum against the reversed list: a bitonic sequence
    d = rd;
    i = ri;
  }
#pragma unroll
  for (int j = 16; j > 0; j >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, d, j);
    const long long oi = __shfl_xor_sync(0xffffffffu, i, j);
    const bool less = key_less_pad(od, oi, d, i);
    if (((lane & j) == 0) == less) {
      d = od;
      i = oi;
    }
  }
}

// Top-m of the keys (dist[i], id(i)), i in this CTA's chunk of [0, n): id(i) = in_idx[i] when in_idx is
// given (second level: merging the per-chunk candidates), else i.  Grid (chunks, queries); each CTA writes
// m sorted (distance, index) pairs, padded with (+inf, INT64_MAX) when the chunk holds fewer.
// Every warp keeps a sorted list of its m best over the lanes.  A round of 32 candidates is tested against the
// list's m-th key; a few survivors are inserted one by one (ballot + shuffle), many (the first rounds) are
// sorted by a bitonic network and merged.  Warp 0 then merges the warps' lists.
template <int NW>
__device__ __forceinline__ void select_topm_cta(const double* __restrict__ dq, const long long* __restrict__ iq,
                                                long long lo, long long hi, int m, long long* __restrict__ idx_out,
                                                double* __restrict__ dist_out, double* cd, long long* ci) {
  constexpr int NT = NW * 32;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const double INF = __longlong_as_double(0x7ff0000000000000LL);
  const long long IMAX = 0x7fffffffffffffffLL;
  // lane l holds the l-th smallest key seen by this warp (l < m), padding beyond
  double bd = INF;
  long long bi = IMAX;
  // the next round's candidate is loaded while the current one is processed
  double cn = INF;
  long long cnidx = IMAX;
  {
    const long long i0 = lo + (long long)w * 32 + lane;
    if (i0 < hi) {
      cn = __ldcg(dq + i0);
      cnidx = iq ? __ldcg(iq + i0) : i0;
    }
  }
  for (long long base = lo + (long long)w * 32; base < hi; base += NT) {
    double c = cn;
    long long cidx = cnidx;
    {
      const long long i1 = base + NT + lane;
      cn = INF;
      cnidx = IMAX;
      if (i1 < hi) {
        cn = __ldcg(dq + i1);
        cnidx = iq ? __ldcg(iq + i1) : i1;
      }
    }
    const double td = shfl_d(bd, m - 1);
    const long long ti = shfl_ll(bi, m - 1);
    const bool want = key_less_pad(c, cidx, td, ti);
    unsigned pending = __ballot_sync(0xffffffffu, want);
    if (pending == 0) continue;
    if (__popc(pending) > 3) {
      if (!want) {
        c = INF;
        cidx = IMAX;
      }
      warp_sort32(c, cidx, lane);
      warp_merge32(bd, bi, c, cidx, lane);
      if (lane >= m) {
        bd = INF;
        bi = IMAX;
      }
      continue;
    }
    while (pending) {
      const int src = __ffs(pending) - 1;
      pending &= pending - 1;
      const double xd = shfl_d(c, src);
      const long long xi = shfl_ll(cidx, src);
      const unsigned below = __ballot_sync(0xffffffffu, (lane < m) && key_less_pad(bd, bi, xd, xi));
      const int pos = __popc(below);
      const double ud = __shfl_up_sync(0xffffffffu, bd, 1);
      const long long ui = __shfl_up_sync(0xffffffffu, bi, 1);
      if (pos < m) {
        if (lane > pos) {
          bd = ud;
          bi = ui;
        } else if (lane == pos) {
          bd = xd;
          bi = xi;
        }
      }
      if (lane >= m) {
        bd = INF;
        bi = IMAX;
      }
    }
  }
  cd[w * 32 + lane] = bd;
  ci[w * 32 + lane] = bi;
  __syncthreads();
  if (w != 0) return;
#pragma unroll 1
  for (int o = 1; o < NW; o++) {
    warp_merge32(bd, bi, cd[o * 32 + lane], ci[o * 32 + lane], lane);
    if (lane >= m) {
      bd = INF;
      bi = IMAX;
    }
  }
  if (lane < m) {
    idx_out[lane] = bi;
    dist_out[lane] = (bi == IMAX) ? INF : bd;
  }
}

__global__ void __launch_bounds__(KNN_SEL_THREADS)
select_kernel(const double* __restrict__ dist, const long long* __restrict__ in_idx, long long n,
              long long chunk, int m, long long* __restrict__ idx_out, double* __restrict__ dist_out) {
  constexpr int NW = KNN_SEL_THREADS / 32;
  __shared__ double cd[NW * 32];
  __shared__ long long ci[NW * 32];
  const int q = blockIdx.y;
  const double* dq = dist + (long long)q * n;
  const long long* iq = in_idx ? in_idx + (long long)q * n : nullptr;
  const long long lo = (long long)blockIdx.x * chunk, hi = min(n, lo + chunk);
  const long long ob = ((long long)q * gridDim.x + blockIdx.x) * m;
  select_topm_cta<NW>(dq, iq, lo, hi, m, idx_out + ob, dist_out + ob, cd, ci);
}

// ---------------------------------------------------------------------------------------
// Few queries (the sweep: one): distance scan, top-m selection and -- for the sweep -- the neighbour matrix in ONE
// launch (was three dependent launches, 35 + 24 + 26 us in the sweep; at n = 65 536 the scan ran at 90 % of HBM but the
// call at 40 %).  Grid (chunks of 256 rows, queries).  Every CTA scans its 256 rows, selects their m best (level 1,
// in parallel on all SMs) and writes m candidates; the CTA that finishes last for its query (ticket counter) merges
// the candidates (level 2) and, when r2 is given, forms the m x m squared-distance matrix of the selected rows (the
// r2 of the GP kernels, cdist arithmetic).
// ---------------------------------------------------------------------------------------
static constexpr int PRO_THREADS = 256;
static constexpr int PRO_JC = 64;

template <int PF>
__global__ void __launch_bounds__(PRO_THREADS)
scan_select_kernel(const double* __restrict__ XT, const double* __restrict__ X, long long cap, long long n, int d,
                   const double* __restrict__ Q, int m, double* __restrict__ dist_all, double* __restrict__ cand_d,
                   long long* __restrict__ cand_i, unsigned int* tickets, long long* __restrict__ idx_out,
                   double* __restrict__ dist_out, double* __restrict__ r2) {
  extern __shared__ double qs[];  // [d]
  constexpr int NW = PRO_THREADS / 32;
  __shared__ double cd[NW * 32];
  __shared__ long long ci[NW * 32];
  __shared__ double tile[NNGP_MAX_NEIGHBOURS][PRO_JC + 1];
  __shared__ bool last;
  const int qi = blockIdx.y;
  const double* q = Q + (long long)qi * d;
  double* dq = dist_all + (long long)qi * n;
  for (int e = threadIdx.x; e < d; e += blockDim.x) qs[e] = q[e];
  __syncthreads();
  const long long lo = (long long)blockIdx.x * PRO_THREADS, hi = min(n, lo + PRO_THREADS);
  const long long i = lo + threadIdx.x;
  if (i < n) {
    const double* xp = XT + i;
    double acc = 0.0;
    double cur[PF], nxt[PF];
    const int nb = d / PF;
#pragma unroll
    for (int u = 0; u < PF; u++) cur[u] = (nb > 0) ? xp[(long long)u * cap] : 0.0;
    for (int b = 0; b < nb; b++) {
      const int j0 = b * PF;
      if (b + 1 < nb) {
#pragma unroll
        for (int u = 0; u < PF; u++) nxt[u] = xp[(long long)(j0 + PF + u) * cap];
      }
#pragma unroll
      for (int u = 0; u < PF; u++) {
        const double diff = qs[j0 + u] - cur[u];
        acc = acc + diff * diff;
      }
#pragma unroll
      for (int u = 0; u < PF; u++) cur[u] = nxt[u];
    }
    for (int j = nb * PF; j < d; j++) {
      const double diff = qs[j] - xp[(long long)j * cap];
      acc = acc + diff * diff;
    }
    __stcg(dq + i, acc);
  }
  __syncthreads();  // the CTA's distances are visible to the CTA (global writes + barrier)
  // level 1: the m best of this CTA's rows
  const long long cbase = ((long long)qi * gridDim.x + blockIdx.x) * m;
  select_topm_cta<NW>(dq, nullptr, lo, hi, m, cand_i + cbase, cand_d + cbase, cd, ci);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(tickets + qi, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!last) return;
  __threadfence();
  // level 2: merge the candidates of all CTAs of this query
  const long long nc = (long long)gridDim.x * m;
  long long* io = idx_out + (long long)qi * m;
  select_topm_cta<NW>(cand_d + (long long)qi * nc, cand_i + (long long)qi * nc, 0, nc, m, io, dist_out + (long long)qi * m,
                      cd, ci);
  if (threadIdx.x == 0) tickets[qi] = 0;  // ready for the next launch
  if (r2 == nullptr) return;
  __syncthreads();  // idx_out written by warp 0 of this CTA
  double* r2q = r2 + (long long)qi * m * m;
  const int npairs = m * (m + 1) / 2;
  constexpr int PP = (NNGP_MAX_NEIGHBOURS * (NNGP_MAX_NEIGHBOURS + 1) / 2 + PRO_THREADS - 1) / PRO_THREADS;
  int pa[PP], pb[PP];
  double acc2[PP];
#pragma unroll
  for (int u = 0; u < PP; u++) {
    const int pidx = threadIdx.x + u * PRO_THREADS;
    int a = 0, b = 0;
    if (pidx < npairs) {
      a = (int)((sqrt(8.0 * pidx + 1.0) - 1.0) * 0.5);
      while ((a + 1) * (a + 2) / 2 <= pidx) a++;
      while (a * (a + 1) / 2 > pidx) a--;
      b = pidx - a * (a + 1) / 2;
    }
    pa[u] = a;
    pb[u] = b;
    acc2[u] = 0.0;
  }
  for (int j0 = 0; j0 < d; j0 += PRO_JC) {
    const int jn = min(PRO_JC, d - j0);
    __syncthreads();
    for (int e = threadIdx.x; e < m * PRO_JC; e += PRO_THREADS) {
      const int r = e / PRO_JC, jj = e - r * PRO_JC;
      if (jj < jn) tile[r][jj] = X[__ldcg(io + r) * d + j0 + jj];
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PP; u++) {
      if (threadIdx.x + u * PRO_THREADS < npairs) {
        double sacc = acc2[u];
        for (int jj = 0; jj < jn; jj++) {
          const double diff = tile[pa[u]][jj] - tile[pb[u]][jj];
          sacc = sacc + diff * diff;
        }
        acc2[u] = sacc;
      }
    }
  }
#pragma unroll
  for (int u = 0; u < PP; u++) {
    if (threadIdx.x + u * PRO_THREADS < npairs) {
      r2q[pa[u] * m + pb[u]] = acc2[u];
      r2q[pb[u] * m + pa[u]] = acc2[u];
    }
  }
}

// Small datasets (the sweep: 512 .. ~3000 rows): scan_select_kernel above has one thread walk one row with a fixed
// number of loads in flight, so a 512-row scan is two CTAs waiting 32 times for L2 (52 us per slice, 26 ms per iteration
// of the FHN target -- profiles/r02/launches_step_r2.summary.csv).  Here a CTA takes 32 rows: all its threads stream
// the row-major rows (coalesced), leave (q_j - x_ij)^2 in a padded shared-memory tile, and 32 threads add their row up
// in ascending j -- the same operations in the same order, so the same bits.  Level 1 is a 32-key bitonic sort in
// warp 0; level 2 and the neighbour matrix run in the CTA that takes the last ticket, the neighbour rows staged in
// the same tile, a column tile at a time.
// The kernel runs once per slice between two launches of the (large) fit kernel, so it starts with a cold instruction
// cache and executes most of its code once: in-kernel clock stamps showed 3-5x the cycles its arithmetic and memory
// latencies account for, proportional to the code size of each phase (a fully unrolled version of this kernel:
// 4 500 instructions, 60 k cycles for the last CTA).  Hence the loops below are deliberately NOT unrolled beyond what
// keeps enough loads in flight.
static constexpr int TILE_ROWS = 32;   // rows of the shared tile (the neighbour rows of the r2 phase: m <= 32)
static constexpr int SCAN_ROWS = 16;   // dataset rows scanned per CTA: with n >= 16 m there are at least m candidate
                                       // lists and level 2 is bounded by the m-th head (n = 512, m = 20: 32 lists)
static constexpr int TILE_COLS = 256;
static constexpr int TILE_LD = TILE_COLS + 1;
static constexpr long long KNN_TILE_MAX_ROWS = 8192;   // beyond: the head ranking of level 2 (lists^2 / 256 per thread) outgrows the scan; the streaming kernel takes over

#ifdef NNGP_KNN_TIMING
__device__ long long g_knn_stamps[16];
#define KNN_STAMP(k) do { if (threadIdx.x == 0 && (blockIdx.x == 0 || (k) >= 4)) g_knn_stamps[k] = clock64(); } while (0)
#else
#define KNN_STAMP(k) do {} while (0)
#endif

// The total order (isnan, distance, index) with padding last, as a pair of integers compared lexicographically:
// comparisons become predicate logic (the floating-point version compiles to divergent branches -- 40 k cycles for
// the level-2 ranks of 320 candidates, measured with in-kernel clock stamps).
typedef unsigned long long u64;
static constexpr u64 UKEY_NAN = 0xfffffffffffffffeULL, UKEY_PAD = 0xffffffffffffffffULL;
__device__ __forceinline__ u64 ukey_of(double d) {
  if (d != d) return UKEY_NAN;
  const u64 b = (u64)__double_as_longlong(d + 0.0);  // -0 -> +0: equal distances tie on the index
  return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double ukey_to_double(u64 k) {
  if (k >= UKEY_NAN) return (k == UKEY_NAN) ? __longlong_as_double(0x7ff8000000000000LL) : __longlong_as_double(0x7ff0000000000000LL);
  const u64 b = (k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k;
  return __longlong_as_double((long long)b);
}
__device__ __forceinline__ bool ukey_less(u64 k1, long long i1, u64 k2, long long i2) {
  return (k1 < k2) | ((k1 == k2) & (i1 < i2));
}

// bitonic sort of one key per lane, ascending over the lanes; the network as two rolled loops (see above)
__device__ __forceinline__ void warp_sort32_compact(u64& k, long long& i, int lane) {
#pragma unroll 1
  for (int kk = 2; kk <= 32; kk <<= 1) {
#pragma unroll 1
    for (int j = kk >> 1; j > 0; j >>= 1) {
      const u64 ok = __shfl_xor_sync(0xffffffffu, k, j);
      const long long oi = __shfl_xor_sync(0xffffffffu, i, j);
      const bool take_min = ((lane & kk) == 0) == ((lane & j) == 0);
      const bool less = ukey_less(ok, oi, k, i);
      const bool take = (take_min == less);
      k = take ? ok : k;
      i = take ? oi : i;
    }
  }
}

// rows r = wid, wid + 8, ... (< nrows) of a column tile [j0, j0 + jn) into the shared tile: warp per row, lanes over
// the columns lane + 32 k (256-byte coalesced loads, 16 of a thread in flight).  SQ: store (q_j - x)^2, else x.
template <bool SQ, int RG>
__device__ __forceinline__ void stage_rows(const double* __restrict__ X, const long long* __restrict__ rowid,
                                           long long row0, int nrows, int d, int j0, int jn,
                                           const double* __restrict__ qs, double* __restrict__ tile, int wid, int lane) {
  constexpr int NW = PRO_THREADS / 32;
  // RG row groups per warp: all their loads (8 RG per thread) in flight at once
  double xv[RG][8];
#pragma unroll
  for (int h = 0; h < RG; h++) {
    const int r = wid + h * NW;
    const long long row = (r < nrows) ? (rowid ? __ldcg(rowid + r) : row0 + r) : 0;
    const double* xr = X + row * d + j0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int c = lane + 32 * k;
      xv[h][k] = (r < nrows && c < jn) ? __ldg(xr + c) : 0.0;
    }
  }
#pragma unroll
  for (int h = 0; h < RG; h++) {
    const int r = wid + h * NW;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int c = lane + 32 * k;
      if (c < jn) {
        if (SQ) {
          const double diff = qs[j0 + c] - xv[h][k];
          tile[r * TILE_LD + c] = diff * diff;
        } else {
          tile[r * TILE_LD + c] = xv[h][k];
        }
      }
    }
  }
}

__global__ void __launch_bounds__(PRO_THREADS)
scan_select_tile_kernel(const double* __restrict__ X, long long n, int d, const double* __restrict__ Q, int m,
                        double* __restrict__ cand_d, long long* __restrict__ cand_i, unsigned int* tickets,
                        long long* __restrict__ idx_out, double* __restrict__ dist_out, double* __restrict__ r2) {
  extern __shared__ double dyn[];  // [d] query | [TILE_ROWS][TILE_LD] tile
  double* qs = dyn;
  double* tile = dyn + ((d + 1) & ~1);
  constexpr int NW = PRO_THREADS / 32;
  static_assert(TILE_ROWS % NW == 0 && SCAN_ROWS % NW == 0 && SCAN_ROWS <= 32 && TILE_COLS == 8 * 32, "row / column mapping of the tile");
  __shared__ bool last;
  __shared__ int active[NNGP_MAX_NEIGHBOURS];
  const double INF = __longlong_as_double(0x7ff0000000000000LL);
  const long long IMAX = 0x7fffffffffffffffLL;
  const int qi = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const double* q = Q + (long long)qi * d;
#pragma unroll 1
  for (int e = tid; e < d; e += PRO_THREADS) qs[e] = q[e];
  const long long lo = (long long)blockIdx.x * SCAN_ROWS;
  const int rows = (int)min((long long)SCAN_ROWS, n - lo);
  double acc = 0.0;
  KNN_STAMP(0);
  __syncthreads();
#pragma unroll 1
  for (int j0 = 0; j0 < d; j0 += TILE_COLS) {
    const int jn = min(TILE_COLS, d - j0);
    stage_rows<true, SCAN_ROWS / NW>(X, nullptr, lo, rows, d, j0, jn, qs, tile, wid, lane);
    __syncthreads();
    if (tid < rows) {
      const double* tr = tile + tid * TILE_LD;
#pragma unroll 32
      for (int c = 0; c < jn; c++) acc = acc + tr[c];
    }
    __syncthreads();
  }
  KNN_STAMP(1);
  // level 1: the CTA's rows sorted by (distance, index); the first m are its candidates
  if (tid < 32) {
    u64 kk = (lane < rows) ? ukey_of(acc) : UKEY_PAD;
    long long ki = (lane < rows) ? lo + lane : IMAX;
    warp_sort32_compact(kk, ki, lane);
    if (lane < m) {
      const long long cbase = ((long long)qi * gridDim.x + blockIdx.x) * m;
      cand_i[cbase + lane] = ki;
      reinterpret_cast<u64*>(cand_d)[cbase + lane] = kk;  // the integer key; level 2 converts back
    }
  }
  KNN_STAMP(2);
  __threadfence();
  __syncthreads();
  if (tid == 0) last = (atomicAdd(tickets + qi, 1u) == gridDim.x - 1);
  __syncthreads();
  KNN_STAMP(3);
  if (!last) return;
  __threadfence();
  KNN_STAMP(4);
  // level 2: the m smallest keys of the gridDim.x sorted candidate lists.  With at least m lists, T = the m-th smallest
  // list head bounds the answer (m heads are <= T), every key <= T sits in one of the m lists whose heads are <= T
  // ("active"), and the rank of such a key among the active lists is its rank among all candidates: each surviving
  // key finds its output position by binary searches -- no sorting network, cost independent of the number of lists.
  // With fewer than m lists all of them are active and nothing is bounded.
  const int nl = gridDim.x;
  long long* io = idx_out + (long long)qi * m;
  {
    const u64* cdq = reinterpret_cast<const u64*>(cand_d) + (long long)qi * nl * m;
    const long long* ciq = cand_i + (long long)qi * nl * m;
    u64* hd = reinterpret_cast<u64*>(tile);                 // [nl] heads
    long long* hi = reinterpret_cast<long long*>(tile + nl);
    u64* ad = reinterpret_cast<u64*>(tile + 2 * nl);        // [na][m] active lists
    long long* ai = reinterpret_cast<long long*>(tile + 2 * nl + NNGP_MAX_NEIGHBOURS * NNGP_MAX_NEIGHBOURS);
#pragma unroll 1
    for (int l = tid; l < nl; l += PRO_THREADS) {
      hd[l] = __ldcg(cdq + (long long)l * m);
      hi[l] = __ldcg(ciq + (long long)l * m);
    }
    __syncthreads();
    KNN_STAMP(8);
    const int na = min(nl, m);
#pragma unroll 1
    for (int l = tid; l < nl; l += PRO_THREADS) {
      const u64 kk = hd[l];
      const long long ki = hi[l];
      int r = 0;
#pragma unroll 4
      for (int t = 0; t < nl; t++) r += ukey_less(hd[t], hi[t], kk, ki) ? 1 : 0;
      if (r < na) active[r] = l;
    }
    __syncthreads();
    KNN_STAMP(9);
#pragma unroll 1
    for (int e = tid; e < na * m; e += PRO_THREADS) {
      const int a = e / m, pp = e - a * m;
      ad[e] = __ldcg(cdq + (long long)active[a] * m + pp);
      ai[e] = __ldcg(ciq + (long long)active[a] * m + pp);
    }
    __syncthreads();
    KNN_STAMP(10);
    const bool bounded = nl >= m;
    const u64 tk = ad[(na - 1) * m];
    const long long ti = ai[(na - 1) * m];
    // surviving keys (not padding, not above the bound) are packed, then one thread per (survivor, active list) counts
    // the list's keys below the survivor's (lower bound in a sorted list of m <= 32 entries) and adds it to the rank
    int* surv = reinterpret_cast<int*>(tile + 2 * nl + 2 * NNGP_MAX_NEIGHBOURS * NNGP_MAX_NEIGHBOURS);
    int* rankacc = surv + NNGP_MAX_NEIGHBOURS * NNGP_MAX_NEIGHBOURS;
    __shared__ int n_surv;
    if (tid == 0) n_surv = 0;
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < na * m; e += PRO_THREADS) {
      const u64 kk = ad[e];
      const long long ki = ai[e];
      if (ki == IMAX || (bounded && ukey_less(tk, ti, kk, ki))) continue;
      const int pos = atomicAdd(&n_surv, 1);
      surv[pos] = e;
      rankacc[pos] = 0;
    }
    __syncthreads();
    const int ns = n_surv;
#pragma unroll 1
    for (int t = tid; t < ns * na; t += PRO_THREADS) {
      const int sidx = t / na, a = t - sidx * na;
      const int e = surv[sidx];
      const u64 kk = ad[e];
      const long long ki = ai[e];
      int base = 0, len = m;
#pragma unroll 1
      for (int step = 0; step < 6; step++) {
        const int half = len >> 1;
        const int at = a * m + min(base + half, m - 1);
        const bool below = (len > 0) & ukey_less(ad[at], ai[at], kk, ki);
        base = below ? base + half + 1 : base;
        len = below ? len - half - 1 : half;
      }
      if (base) atomicAdd(&rankacc[sidx], base);
    }
    __syncthreads();
#pragma unroll 1
    for (int sidx = tid; sidx < ns; sidx += PRO_THREADS) {
      const int rank = rankacc[sidx];
      if (rank < m) {
        const int e = surv[sidx];
        io[rank] = ai[e];
        dist_out[(long long)qi * m + rank] = ukey_to_double(ad[e]);
      }
    }
  }
  KNN_STAMP(11);
  if (tid == 0) tickets[qi] = 0;  // ready for the next launch
  if (r2 == nullptr) return;
  __threadfence_block();
  __syncthreads();  // idx_out written by this CTA
  KNN_STAMP(5);
  // neighbour matrix: pair (a, b), a >= b, per thread (m (m + 1) / 2 <= 528 pairs: up to three per thread)
  double* r2q = r2 + (long long)qi * m * m;
  const int npairs = m * (m + 1) / 2;
  constexpr int PP = (NNGP_MAX_NEIGHBOURS * (NNGP_MAX_NEIGHBOURS + 1) / 2 + PRO_THREADS - 1) / PRO_THREADS;
  int pa[PP], pb[PP];
  double acc2[PP];
#pragma unroll
  for (int u = 0; u < PP; u++) {
    const int pidx = tid + u * PRO_THREADS;
    int a = 0, b = 0;
    if (pidx < npairs) {
      a = (int)((sqrtf(8.0f * (float)pidx + 1.0f) - 1.0f) * 0.5f);
      while ((a + 1) * (a + 2) / 2 <= pidx) a++;
      while (a * (a + 1) / 2 > pidx) a--;
      b = pidx - a * (a + 1) / 2;
    }
    pa[u] = a;
    pb[u] = b;
    acc2[u] = 0.0;
  }
  KNN_STAMP(6);
#pragma unroll 1
  for (int j0 = 0; j0 < d; j0 += TILE_COLS) {
    const int jn = min(TILE_COLS, d - j0);
    __syncthreads();
    stage_rows<false, TILE_ROWS / NW>(X, io, 0, m, d, j0, jn, nullptr, tile, wid, lane);
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PP; u++) {
      if (tid + u * PRO_THREADS < npairs) {
        const double *ta = tile + pa[u] * TILE_LD, *tb = tile + pb[u] * TILE_LD;
        double sacc = acc2[u];
#pragma unroll 16
        for (int c = 0; c < jn; c++) {
          const double diff = ta[c] - tb[c];
          sacc = sacc + diff * diff;
        }
        acc2[u] = sacc;
      }
    }
  }
  KNN_STAMP(7);
#pragma unroll
  for (int u = 0; u < PP; u++) {
    if (tid + u * PRO_THREADS < npairs) {
      r2q[pa[u] * m + pb[u]] = acc2[u];
      r2q[pb[u] * m + pa[u]] = acc2[u];
    }
  }
}

// scan_select_tile_kernel for many queries, each over its own segment of rows (the kNN of an ensemble of runs that
// share one store): query blockIdx.y searches the rows [base, base + n) of X and its candidate lists are read back from
// the nl = ceil(n / SCAN_ROWS) first of the gridDim.x slots of the query; the CTAs past the end of a short segment only
// take their ticket.  Indices are global (base + row).  The same operations in the same order as
// scan_select_tile_kernel, so the same bits; a separate copy, because folding both into one template changed the
// register allocation of the existing kernel.
__device__ __forceinline__ void scan_select_tile_seg_body(const double* __restrict__ X, long long n, long long base, int d,
                                                      const double* __restrict__ q, int m, int nl,
                                                      double* __restrict__ cand_d, long long* __restrict__ cand_i,
                                                      unsigned int* tickets, long long* __restrict__ idx_out,
                                                      double* __restrict__ dist_out, double* __restrict__ r2) {
  extern __shared__ double dyn[];  // [d] query | [TILE_ROWS][TILE_LD] tile
  double* qs = dyn;
  double* tile = dyn + ((d + 1) & ~1);
  constexpr int NW = PRO_THREADS / 32;
  static_assert(TILE_ROWS % NW == 0 && SCAN_ROWS % NW == 0 && SCAN_ROWS <= 32 && TILE_COLS == 8 * 32, "row / column mapping of the tile");
  __shared__ bool last;
  __shared__ int active[NNGP_MAX_NEIGHBOURS];
  const double INF = __longlong_as_double(0x7ff0000000000000LL);
  const long long IMAX = 0x7fffffffffffffffLL;
  const int qi = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
#pragma unroll 1
  for (int e = tid; e < d; e += PRO_THREADS) qs[e] = q[e];
  const long long lo = (long long)blockIdx.x * SCAN_ROWS;
  const int rows = (int)min((long long)SCAN_ROWS, n - lo);
  if (rows > 0) {
  double acc = 0.0;
  KNN_STAMP(0);
  __syncthreads();
#pragma unroll 1
  for (int j0 = 0; j0 < d; j0 += TILE_COLS) {
    const int jn = min(TILE_COLS, d - j0);
    stage_rows<true, SCAN_ROWS / NW>(X, nullptr, base + lo, rows, d, j0, jn, qs, tile, wid, lane);
    __syncthreads();
    if (tid < rows) {
      const double* tr = tile + tid * TILE_LD;
#pragma unroll 32
      for (int c = 0; c < jn; c++) acc = acc + tr[c];
    }
    __syncthreads();
  }
  KNN_STAMP(1);
  // level 1: the CTA's rows sorted by (distance, index); the first m are its candidates
  if (tid < 32) {
    u64 kk = (lane < rows) ? ukey_of(acc) : UKEY_PAD;
    long long ki = (lane < rows) ? base + lo + lane : IMAX;
    warp_sort32_compact(kk, ki, lane);
    if (lane < m) {
      const long long cbase = ((long long)qi * gridDim.x + blockIdx.x) * m;
      cand_i[cbase + lane] = ki;
      reinterpret_cast<u64*>(cand_d)[cbase + lane] = kk;  // the integer key; level 2 converts back
    }
  }
  }
  KNN_STAMP(2);
  __threadfence();
  __syncthreads();
  if (tid == 0) last = (atomicAdd(tickets + qi, 1u) == gridDim.x - 1);
  __syncthreads();
  KNN_STAMP(3);
  if (!last) return;
  __threadfence();
  KNN_STAMP(4);
  // level 2: the m smallest keys of the gridDim.x sorted candidate lists.  With at least m lists, T = the m-th smallest
  // list head bounds the answer (m heads are <= T), every key <= T sits in one of the m lists whose heads are <= T
  // ("active"), and the rank of such a key among the active lists is its rank among all candidates: each surviving
  // key finds its output position by binary searches -- no sorting network, cost independent of the number of lists.
  // With fewer than m lists all of them are active and nothing is bounded.
  long long* io = idx_out + (long long)qi * m;
  {
    const u64* cdq = reinterpret_cast<const u64*>(cand_d) + (long long)qi * gridDim.x * m;
    const long long* ciq = cand_i + (long long)qi * gridDim.x * m;
    u64* hd = reinterpret_cast<u64*>(tile);                 // [nl] heads
    long long* hi = reinterpret_cast<long long*>(tile + nl);
    u64* ad = reinterpret_cast<u64*>(tile + 2 * nl);        // [na][m] active lists
    long long* ai = reinterpret_cast<long long*>(tile + 2 * nl + NNGP_MAX_NEIGHBOURS * NNGP_MAX_NEIGHBOURS);
#pragma unroll 1
    for (int l = tid; l < nl; l += PRO_THREADS) {
      hd[l] = __ldcg(cdq + (long long)l * m);
      hi[l] = __ldcg(ciq + (long long)l * m);
    }
    __syncthreads();
    KNN_STAMP(8);
    const int na = min(nl, m);
#pragma unroll 1
    for (int l = tid; l < nl; l += PRO_THREADS) {
      const u64 kk = hd[l];
      const long long ki = hi[l];
      int r = 0;
#pragma unroll 4
      for (int t = 0; t < nl; t++) r += ukey_less(hd[t], hi[t], kk, ki) ? 1 : 0;
      if (r < na) active[r] = l;
    }
    __syncthreads();
    KNN_STAMP(9);
#pragma unroll 1
    for (int e = tid; e < na * m; e += PRO_THREADS) {
      const int a = e / m, pp = e - a * m;
      ad[e] = __ldcg(cdq + (long long)active[a] * m + pp);
      ai[e] = __ldcg(ciq + (long long)active[a] * m + pp);
    }
    __syncthreads();
    KNN_STAMP(10);
    const bool bounded = nl >= m;
    const u64 tk = ad[(na - 1) * m];
    const long long ti = ai[(na - 1) * m];
    // surviving keys (not padding, not above the bound) are packed, then one thread per (survivor, active list) counts
    // the list's keys below the survivor's (lower bound in a sorted list of m <= 32 entries) and adds it to the rank
    int* surv = reinterpret_cast<int*>(tile + 2 * nl + 2 * NNGP_MAX_NEIGHBOURS * NNGP_MAX_NEIGHBOURS);
    int* rankacc = surv + NNGP_MAX_NEIGHBOURS * NNGP_MAX_NEIGHBOURS;
    __shared__ int n_surv;
    if (tid == 0) n_surv = 0;
    __syncthreads();
#pragma unroll 1
    for (int e = tid; e < na * m; e += PRO_THREADS) {
      const u64 kk = ad[e];
      const long long ki = ai[e];
      if (ki == IMAX || (bounded && ukey_less(tk, ti, kk, ki))) continue;
      const int pos = atomicAdd(&n_surv, 1);
      surv[pos] = e;
      rankacc[pos] = 0;
    }
    __syncthreads();
    const int ns = n_surv;
#pragma unroll 1
    for (int t = tid; t < ns * na; t += PRO_THREADS) {
      const int sidx = t / na, a = t - sidx * na;
      const int e = surv[sidx];
      const u64 kk = ad[e];
      const long long ki = ai[e];
      int base = 0, len = m;
#pragma unroll 1
      for (int step = 0; step < 6; step++) {
        const int half = len >> 1;
        const int at = a * m + min(base + half, m - 1);
        const bool below = (len > 0) & ukey_less(ad[at], ai[at], kk, ki);
        base = below ? base + half + 1 : base;
        len = below ? len - half - 1 : half;
      }
      if (base) atomicAdd(&rankacc[sidx], base);
    }
    __syncthreads();
#pragma unroll 1
    for (int sidx = tid; sidx < ns; sidx += PRO_THREADS) {
      const int rank = rankacc[sidx];
      if (rank < m) {
        const int e = surv[sidx];
        io[rank] = ai[e];
        dist_out[(long long)qi * m + rank] = ukey_to_double(ad[e]);
      }
    }
  }
  KNN_STAMP(11);
  if (tid == 0) tickets[qi] = 0;  // ready for the next launch
  if (r2 == nullptr) return;
  __threadfence_block();
  __syncthreads();  // idx_out written by this CTA
  KNN_STAMP(5);
  // neighbour matrix: pair (a, b), a >= b, per thread (m (m + 1) / 2 <= 528 pairs: up to three per thread)
  double* r2q = r2 + (long long)qi * m * m;
  const int npairs = m * (m + 1) / 2;
  constexpr int PP = (NNGP_MAX_NEIGHBOURS * (NNGP_MAX_NEIGHBOURS + 1) / 2 + PRO_THREADS - 1) / PRO_THREADS;
  int pa[PP], pb[PP];
  double acc2[PP];
#pragma unroll
  for (int u = 0; u < PP; u++) {
    const int pidx = tid + u * PRO_THREADS;
    int a = 0, b = 0;
    if (pidx < npairs) {
      a = (int)((sqrtf(8.0f * (float)pidx + 1.0f) - 1.0f) * 0.5f);
      while ((a + 1) * (a + 2) / 2 <= pidx) a++;
      while (a * (a + 1) / 2 > pidx) a--;
      b = pidx - a * (a + 1) / 2;
    }
    pa[u] = a;
    pb[u] = b;
    acc2[u] = 0.0;
  }
  KNN_STAMP(6);
#pragma unroll 1
  for (int j0 = 0; j0 < d; j0 += TILE_COLS) {
    const int jn = min(TILE_COLS, d - j0);
    __syncthreads();
    stage_rows<false, TILE_ROWS / NW>(X, io, 0, m, d, j0, jn, nullptr, tile, wid, lane);
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PP; u++) {
      if (tid + u * PRO_THREADS < npairs) {
        const double *ta = tile + pa[u] * TILE_LD, *tb = tile + pb[u] * TILE_LD;
        double sacc = acc2[u];
#pragma unroll 16
        for (int c = 0; c < jn; c++) {
          const double diff = ta[c] - tb[c];
          sacc = sacc + diff * diff;
        }
        acc2[u] = sacc;
      }
    }
  }
  KNN_STAMP(7);
#pragma unroll
  for (int u = 0; u < PP; u++) {
    if (tid + u * PRO_THREADS < npairs) {
      r2q[pa[u] * m + pb[u]] = acc2[u];
      r2q[pb[u] * m + pa[u]] = acc2[u];
    }
  }
}

// query qi (row stride ld_q) searches rows [base[qi], base[qi] + rows[qi]); gridDim.x covers the longest segment
__global__ void __launch_bounds__(PRO_THREADS)
scan_select_tile_seg_kernel(const double* __restrict__ X, int d, const double* __restrict__ Q, long long ld_q,
                            const long long* __restrict__ base, const long long* __restrict__ rows, int m,
                            double* __restrict__ cand_d, long long* __restrict__ cand_i, unsigned int* tickets,
                            long long* __restrict__ idx_out, double* __restrict__ dist_out, double* __restrict__ r2) {
  const int qi = blockIdx.y;
  const long long n = rows[qi];
  scan_select_tile_seg_body(X, n, base[qi], d, Q + (long long)qi * ld_q, m, (int)((n + SCAN_ROWS - 1) / SCAN_ROWS),
                              cand_d, cand_i, tickets, idx_out, dist_out, r2);
}

#ifdef NNGP_KNN_TIMING
extern "C" void nngp_knn_stamps(long long* out) { cudaMemcpyFromSymbol(out, g_knn_stamps, sizeof(long long) * 16); }
#endif

// m > 32 (rare: nn='adaptive' past iteration 30): m passes of "smallest key above the last one" by one CTA per query
__global__ void __launch_bounds__(256)
select_big_kernel(const double* __restrict__ dist, long long n, int m, long long* __restrict__ idx_out,
                  double* __restrict__ dist_out) {
  __shared__ double sd[256];
  __shared__ long long si[256];
  const int q = blockIdx.x, tid = threadIdx.x;
  const double* dq = dist + (long long)q * n;
  const double INF = __longlong_as_double(0x7ff0000000000000LL);
  const long long IMAX = 0x7fffffffffffffffLL;
  double ld = 0.0;
  long long li = -1;
  for (int t = 0; t < m; t++) {
    double bd = INF;
    long long bi = IMAX;
    for (long long i = tid; i < n; i += 256) {
      const double v = dq[i];
      if ((t == 0 || key_less(ld, li, v, i)) && key_less_pad(v, i, bd, bi)) {
        bd = v;
        bi = i;
      }
    }
    sd[tid] = bd;
    si[tid] = bi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (tid < o && key_less_pad(sd[tid + o], si[tid + o], sd[tid], si[tid])) {
        sd[tid] = sd[tid + o];
        si[tid] = si[tid + o];
      }
      __syncthreads();
    }
    ld = sd[0];
    li = si[0];
    if (tid == 0) {
      idx_out[(long long)q * m + t] = li;
      dist_out[(long long)q * m + t] = ld;
    }
    __syncthreads();
  }
}

static constexpr long long KNN_CHUNK = 4096;  // rows up to which one CTA selects alone; chunks are >= a quarter of it

// Rows per first-level CTA: the scan of one query is split only as far as it takes to fill the GPU
// (about two CTAs per SM over all queries) -- every CTA pays the fill of its own top-m lists, so
// with many queries one CTA per query is the faster arrangement.
static long long knn_chunk_rows(int nq, long long n) {
  if (n <= KNN_CHUNK) return n > 0 ? n : 1;  // one CTA per query (the sweep's case)
  const long long want = (296 + nq - 1) / nq;  // CTAs per query
  long long chunk = (n + want - 1) / want;
  if (chunk < KNN_CHUNK / 4) chunk = KNN_CHUNK / 4;
  return chunk;
}

static inline size_t knn_pad256(size_t b) { return ((b + 255) / 256) * 256; }

// [distances nq*n | per-chunk candidate distances nq*chunks*m | candidate indices]
static constexpr int KNN_FUSED_MAX_Q = 4;  // queries per call served by scan_select_kernel (one ticket each)

size_t knn_workspace_bytes(int nq, long long n, int m) {
  const long long cr = knn_chunk_rows(nq, n);
  size_t chunks = (size_t)((n + cr - 1) / cr);
  if (nq <= KNN_FUSED_MAX_Q) chunks = (size_t)((n + 15) / 16);  // SCAN_ROWS of the small-dataset kernel (>= the 256-row chunks)
  size_t b = knn_pad256(sizeof(double) * (size_t)nq * (size_t)n);
  if (chunks > 1 || nq <= KNN_FUSED_MAX_Q) b += 2 * knn_pad256(sizeof(double) * (size_t)nq * chunks * (size_t)m);
  return b;
}

// distance scan + top-m (+ neighbour matrix when d_r2 is given) of up to KNN_FUSED_MAX_Q queries in one launch
static int scan_select_launch(nngp_handle_t h, const double* d_q, int nq, int m, long long n, long long* d_idx,
                              double* d_dist, double* d_r2, void* ws, cudaStream_t st) {
  const int d = h->ds_d;
  double* dist = (double*)ws;
  char* base = (char*)ws + knn_pad256(sizeof(double) * (size_t)nq * (size_t)n);
  const size_t tile_smem = sizeof(double) * ((size_t)((d + 1) & ~1) + (size_t)TILE_ROWS * TILE_LD);
  if (n <= KNN_TILE_MAX_ROWS && tile_smem <= 200 * 1024) {
    const unsigned tchunks = (unsigned)((n + SCAN_ROWS - 1) / SCAN_ROWS);
    double* tcand_d = (double*)base;
    long long* tcand_i = (long long*)(base + knn_pad256(sizeof(double) * (size_t)nq * tchunks * m));
    if (!h->attr_knn_tile) {
      NNGP_CUDA(h, cudaFuncSetAttribute(scan_select_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      h->attr_knn_tile = true;
    }
    scan_select_tile_kernel<<<dim3(tchunks, nq), PRO_THREADS, tile_smem, st>>>(
        h->ds_x, n, d, d_q, m, tcand_d, tcand_i, h->d_ticket, d_idx, d_dist, d_r2);
    h->launches++;
    NNGP_CUDA(h, cudaGetLastError());
    return 0;
  }
  const unsigned chunks = (unsigned)((n + PRO_THREADS - 1) / PRO_THREADS);
  double* cand_d = (double*)base;
  long long* cand_i = (long long*)(base + knn_pad256(sizeof(double) * (size_t)nq * chunks * m));
  scan_select_kernel<16><<<dim3(chunks, nq), PRO_THREADS, (size_t)d * sizeof(double), st>>>(
      h->ds_xt, h->ds_x, h->ds_cap, n, d, d_q, m, dist, cand_d, cand_i, h->d_ticket, d_idx, d_dist, d_r2);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

int knn_launch(nngp_handle_t h, const double* d_q, int nq, int m, long long n_rows,
               long long* d_idx, double* d_dist, void* ws, cudaStream_t st) {
  const long long n = (n_rows > 0) ? n_rows : h->ds_rows;
  if (nq <= 0) return 0;
  if (m < 1 || m > NNGP_MAX_NEIGHBOURS_BIG)
    return nngp_fail(h, "knn: m=%d outside [1,%d]", m, NNGP_MAX_NEIGHBOURS_BIG);
  if (n > h->ds_rows) return nngp_fail(h, "knn: n_rows=%lld > dataset rows %lld", n, h->ds_rows);
  if (n < m) return nngp_fail(h, "knn: dataset has %lld rows, fewer than m=%d", n, m);
  const int d = h->ds_d;
  double* dist = (double*)ws;
  ProfScope prof(h, 1, st);
  if (nq <= KNN_FUSED_MAX_Q && m <= NNGP_MAX_NEIGHBOURS && (size_t)d * sizeof(double) <= 48 * 1024)
    return scan_select_launch(h, d_q, nq, m, n, d_idx, d_dist, nullptr, ws, st);
  const int tb = 128;
  const unsigned gx = (unsigned)((n + tb - 1) / tb);
  const size_t qrow = (size_t)d * sizeof(double), lim = 48 * 1024;
  if (nq >= 8 && 8 * qrow <= lim) {
    sqdist_kernel<8><<<dim3(gx, (nq + 7) / 8), tb, 8 * qrow, st>>>(h->ds_xt, h->ds_cap, n, d, d_q, nq, dist);
  } else if (nq >= 4 && 4 * qrow <= lim) {
    sqdist_kernel<4><<<dim3(gx, (nq + 3) / 4), tb, 4 * qrow, st>>>(h->ds_xt, h->ds_cap, n, d, d_q, nq, dist);
  } else if (qrow <= lim) {
    // few queries: 64 rows per CTA spread the (few) warps over more SMs
    const unsigned g1 = (unsigned)((n + 63) / 64);
    sqdist_one_kernel<16><<<dim3(g1, nq), 64, qrow, st>>>(h->ds_xt, h->ds_cap, n, d, d_q, dist);
  } else {
    sqdist_kernel_gq<<<dim3(gx, nq), tb, 0, st>>>(h->ds_xt, h->ds_cap, n, d, d_q, dist);
  }
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  const long long chunk_rows = knn_chunk_rows(nq, n);
  const long long chunks = (n + chunk_rows - 1) / chunk_rows;
  if (m > NNGP_MAX_NEIGHBOURS) {
    select_big_kernel<<<nq, 256, 0, st>>>(dist, n, m, d_idx, d_dist);
    h->launches++;
  } else if (chunks == 1) {
    select_kernel<<<dim3(1, nq), KNN_SEL_THREADS, 0, st>>>(dist, nullptr, n, n, m, d_idx, d_dist);
    h->launches++;
  } else {
    // two levels: top-m of every 4096-row chunk in parallel, then top-m of the chunks' candidates
    char* base = (char*)ws + knn_pad256(sizeof(double) * (size_t)nq * (size_t)n);
    double* cand_d = (double*)base;
    long long* cand_i = (long long*)(base + knn_pad256(sizeof(double) * (size_t)nq * chunks * m));
    select_kernel<<<dim3((unsigned)chunks, nq), KNN_SEL_THREADS, 0, st>>>(dist, nullptr, n, chunk_rows, m, cand_i, cand_d);
    const long long nc = chunks * m;
    select_kernel<<<dim3(1, nq), KNN_SEL_THREADS, 0, st>>>(cand_d, cand_i, nc, nc, m, d_idx, d_dist);
    h->launches += 2;
  }
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// scan + selection + neighbour matrix of ONE query in one launch; false when the shape needs the general path
bool knn_prep_fused_ok(nngp_handle_t h, long long n, int m) {
  return m <= NNGP_MAX_NEIGHBOURS && n >= m && (size_t)h->ds_d * sizeof(double) <= 48 * 1024;
}

int knn_prep_fused_launch(nngp_handle_t h, const double* d_q, int m, long long n, long long* d_idx, double* d_dist,
                          double* d_r2, void* ws, cudaStream_t st) {
  ProfScope prof(h, 1, st);
  return scan_select_launch(h, d_q, 1, m, n, d_idx, d_dist, d_r2, ws, st);
}

// ---------------------------------------------------------------------------------------
// Segmented store (an ensemble of E runs in one handle): member e's rows live at [e cap, e cap + rows_e) of X, Y, XT
// (cap_total = E cap), so every kernel that gathers rows by a global index (gp_prep_kernel, the fits) is unchanged.
// ---------------------------------------------------------------------------------------

// Rows of several sources, one per blockIdx.z, appended in one launch.  tab[z] = {x offset, y offset, rows, first
// destination row}; offsets in doubles from xs / ya / yb, sources row-major with stride ld.  XT through a tile as in
// append_kernel.
__global__ void append_seg_kernel(const double* __restrict__ xs, const double* __restrict__ ya,
                                  const double* __restrict__ yb, long long ld, const long long* __restrict__ tab, int d,
                                  long long cap, double* __restrict__ X, double* __restrict__ Y,
                                  double* __restrict__ XT) {
  __shared__ double tile[32][33];
  const long long* t = tab + 4 * (long long)blockIdx.z;
  const long long xo = t[0], yo = t[1], rows = t[2], n0 = t[3];
  const long long r0 = (long long)blockIdx.y * 32;
  if (r0 >= rows) return;
  const int j0 = blockIdx.x * 32;
  for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
    const long long r = r0 + rr;
    const int j = j0 + threadIdx.x;
    if (r < rows && j < d) {
      const double xv = xs[xo + r * ld + j];
      X[(n0 + r) * d + j] = xv;
      tile[rr][threadIdx.x] = xv;
      double yv = ya[yo + r * ld + j];
      if (yb != nullptr) yv = yv - yb[yo + r * ld + j];
      Y[(n0 + r) * d + j] = yv;
    }
  }
  __syncthreads();
  for (int jj = threadIdx.y; jj < 32; jj += blockDim.y) {
    const int j = j0 + jj;
    const long long r = r0 + threadIdx.x;
    if (r < rows && j < d) XT[(long long)j * cap + n0 + r] = tile[threadIdx.x][jj];
  }
}

int append_seg_launch(nngp_handle_t h, const double* xs, const double* ya, const double* yb, long long ld,
                      const long long* d_tab, int nsrc, long long max_rows, cudaStream_t st) {
  if (nsrc <= 0 || max_rows <= 0) return 0;
  const int d = h->ds_d;
  ProfScope prof(h, 4, st);
  dim3 block(32, 8);
  dim3 grid((d + 31) / 32, (unsigned)((max_rows + 31) / 32), (unsigned)nsrc);
  append_seg_kernel<<<grid, block, 0, st>>>(xs, ya, yb, ld, d_tab, d, h->ds_cap, h->ds_x, h->ds_y, h->ds_xt);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// dst[di[r]] = src[si[r]] for rows of d doubles (a null index list is the identity)
__global__ void copy_rows_kernel(const double* __restrict__ src, const long long* __restrict__ si,
                                 double* __restrict__ dst, const long long* __restrict__ di, long long rows, long long d) {
  for (long long r = blockIdx.y; r < rows; r += gridDim.y) {
    const double* s = src + (si ? si[r] : r) * d;
    double* o = dst + (di ? di[r] : r) * d;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < d; j += (long long)gridDim.x * blockDim.x)
      o[j] = s[j];
  }
}

int copy_rows_launch(nngp_handle_t h, const double* src, const long long* si, double* dst, const long long* di,
                     long long rows, long long d, cudaStream_t st) {
  if (rows <= 0 || d <= 0) return 0;
  const unsigned gx = (unsigned)std::min<long long>((d + 255) / 256, 64);
  copy_rows_kernel<<<dim3(gx, (unsigned)std::min<long long>(rows, 65535)), 256, 0, st>>>(src, si, dst, di, rows, d);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  return 0;
}

// Distances of query q (row stride ld_q) to the rows of its segment, written at dist[q, 0 .. rows[q]); the rest of the
// row, up to n_max, is NaN.  select_kernel / select_big_kernel order keys by (isnan, distance, index), so a padding
// entry sorts after every row of the segment, NaN distances included (its index is larger), and with m <= rows[q]
// it is never selected.
__global__ void __launch_bounds__(128)
sqdist_seg_kernel(const double* __restrict__ XT, long long cap, int d, const double* __restrict__ Q, long long ld_q,
                  const long long* __restrict__ base, const long long* __restrict__ rows, long long n_max,
                  double* __restrict__ dist) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_max) return;
  const int qi = blockIdx.y;
  double acc = __longlong_as_double(0x7ff8000000000000LL);
  if (i < rows[qi]) {
    const double* q = Q + (long long)qi * ld_q;
    const double* xp = XT + base[qi] + i;
    acc = 0.0;
    for (int j = 0; j < d; j++) {
      const double diff = __ldg(q + j) - xp[(long long)j * cap];
      acc = acc + diff * diff;
    }
  }
  dist[(long long)qi * n_max + i] = acc;
}

__global__ void add_base_kernel(long long* __restrict__ idx, const long long* __restrict__ base, int nq, int m) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < nq * m) idx[e] += base[e / m];
}

// [distances nq*n_max | candidates]: both routes have at most ceil(n_max / SCAN_ROWS) candidate lists per query
size_t knn_seg_workspace_bytes(int nq, long long n_max, int m) {
  return knn_pad256(sizeof(double) * (size_t)nq * (size_t)n_max) +
         2 * knn_pad256(sizeof(double) * (size_t)nq * (size_t)((n_max + SCAN_ROWS - 1) / SCAN_ROWS) * m);
}

bool knn_seg_tile_ok(nngp_handle_t h, long long n_max, int m) {
  const size_t tile_smem = sizeof(double) * ((size_t)((h->ds_d + 1) & ~1) + (size_t)TILE_ROWS * TILE_LD);
  return n_max <= KNN_TILE_MAX_ROWS && m <= NNGP_MAX_NEIGHBOURS && tile_smem <= 200 * 1024;
}

// kNN of nq queries, each in its own segment: d_base / d_rows device [nq], n_max = the largest rows[q] (host), every
// rows[q] >= m.  Global indices ordered by (distance, index) and squared distances; r2 (optional, [nq, m, m]): the
// neighbour matrix of gp_prep_kernel.  tickets: nq zeroed counters (left zero).
int knn_seg_launch(nngp_handle_t h, const double* d_q, long long ld_q, int nq, int m, const long long* d_base,
                   const long long* d_rows, long long n_max, long long* d_idx, double* d_dist, double* d_r2,
                   unsigned int* tickets, void* ws, cudaStream_t st) {
  if (nq <= 0) return 0;
  if (m < 1 || m > NNGP_MAX_NEIGHBOURS_BIG) return nngp_fail(h, "knn_segmented: m=%d outside [1,%d]", m, NNGP_MAX_NEIGHBOURS_BIG);
  const int d = h->ds_d;
  ProfScope prof(h, 1, st);
  if (knn_seg_tile_ok(h, n_max, m)) {
    const unsigned tchunks = (unsigned)((n_max + SCAN_ROWS - 1) / SCAN_ROWS);
    double* tcand_d = (double*)ws;
    long long* tcand_i = (long long*)((char*)ws + knn_pad256(sizeof(double) * (size_t)nq * tchunks * m));
    const size_t tile_smem = sizeof(double) * ((size_t)((d + 1) & ~1) + (size_t)TILE_ROWS * TILE_LD);
    if (!h->attr_knn_tile_seg) {
      NNGP_CUDA(h, cudaFuncSetAttribute(scan_select_tile_seg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      h->attr_knn_tile_seg = true;
    }
    scan_select_tile_seg_kernel<<<dim3(tchunks, nq), PRO_THREADS, tile_smem, st>>>(
        h->ds_x, d, d_q, ld_q, d_base, d_rows, m, tcand_d, tcand_i, tickets, d_idx, d_dist, d_r2);
    h->launches++;
    NNGP_CUDA(h, cudaGetLastError());
    return 0;
  }
  double* dist = (double*)ws;
  sqdist_seg_kernel<<<dim3((unsigned)((n_max + 127) / 128), nq), 128, 0, st>>>(h->ds_xt, h->ds_cap, d, d_q, ld_q, d_base,
                                                                             d_rows, n_max, dist);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  const long long chunk_rows = knn_chunk_rows(nq, n_max);
  const long long chunks = (n_max + chunk_rows - 1) / chunk_rows;
  if (m > NNGP_MAX_NEIGHBOURS) {
    select_big_kernel<<<nq, 256, 0, st>>>(dist, n_max, m, d_idx, d_dist);
    h->launches++;
  } else if (chunks == 1) {
    select_kernel<<<dim3(1, nq), KNN_SEL_THREADS, 0, st>>>(dist, nullptr, n_max, n_max, m, d_idx, d_dist);
    h->launches++;
  } else {
    char* cb = (char*)ws + knn_pad256(sizeof(double) * (size_t)nq * (size_t)n_max);
    double* cand_d = (double*)cb;
    long long* cand_i = (long long*)(cb + knn_pad256(sizeof(double) * (size_t)nq * chunks * m));
    select_kernel<<<dim3((unsigned)chunks, nq), KNN_SEL_THREADS, 0, st>>>(dist, nullptr, n_max, chunk_rows, m, cand_i, cand_d);
    const long long nc = chunks * m;
    select_kernel<<<dim3(1, nq), KNN_SEL_THREADS, 0, st>>>(cand_d, cand_i, nc, nc, m, d_idx, d_dist);
    h->launches += 2;
  }
  add_base_kernel<<<(nq * m + 255) / 256, 256, 0, st>>>(d_idx, d_base, nq, m);
  h->launches++;
  NNGP_CUDA(h, cudaGetLastError());
  if (d_r2 != nullptr) return gp_prep_launch(h, d_idx, nq, m, d_r2, st);
  return 0;
}
