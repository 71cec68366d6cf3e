"""Alternative neighbour rules of the reference's "nnGParareal with time" study (nnGPara_with_time.py:27-184, `NNGP_alt`):
instead of the m nearest rows in state space, the m training pairs are picked by their position (time slice i, iteration
k) in the (N x K) grid of observations.  Only the CHOICE of rows differs; the fits, the selection and the posterior mean
are the same device launch as for the nearest-neighbour rule (nngp_fit_predict on an explicit index list).

    nntype   rule (nnGPara_with_time.py line)
    'nn'        nearest neighbours in state space (:50-53) -- the standard model
    'col+rnd'   the last min(nn, k+1) observations of slice i, filled up with random rows (:55-70)
    'col_only'  every observation of slice i so far: m = k+1 (:72-74)
    'row_col'   rows in order of |iteration - k| + |slice - i| (:76-96)
    'row'       iteration k first (slices i, i+1, i-1, i+2, ...), then k-1, ... (:98-135)
    'col_full'  slice i first (iterations k, k-1, ...), then slices i+1, i-1, ... (:137-171)

The model needs the driver's observation cube `data_x` [N, n, K] (NaN where a slice was already converged), which the
reference passes to `fit` (parareal.py:351); the host drivers of this package pass it when `wants_data_cube` is set.
The device drivers (PararealDevice, PararealEnsemble) keep only the first unconverged slice of every iteration and ask
`neighbour_table` for the lists of a whole sweep, which the listed sweeps of csrc/api.cu then run on the device.
"""
import numpy as np

from . import _lib
from .models import CudaNNGP, N_JITTER

NNTYPES = ('nn', 'col+rnd', 'col_only', 'row_col', 'row', 'col_full')


def _cycle(j, n):
    """slices j, j+1, j-1, j+2, ... as the reference's my_cycler walks them (left generator first: j, then j+1, j-1 ...)"""
    left, right = list(range(j, -1, -1)), list(range(j + 1, n))
    out = []
    for t in range(max(len(left), len(right))):
        if t < len(left):
            out.append(left[t])
        if t < len(right):
            out.append(right[t])
    return out


class CudaNNGPAlt(CudaNNGP):
    wants_data_cube = True

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.nntype = kwargs['nntype']
        if self.nntype not in NNTYPES:
            raise Exception(f'unknown nntype {self.nntype!r}')
        self.name = 'NNGP' + str(self.nntype)
        self.rng2 = np.random.default_rng(self.seed)

    def fit(self, x, y, k, *args, **kwargs):
        super().fit(x, y, k, *args, **kwargs)
        self.data_x = kwargs.get('data_x')
        if self.nntype != 'nn' and self.data_x is None:
            raise Exception("the driver must pass data_x to fit() for a position-based neighbour rule")
        if self.data_x is not None:
            N = self.data_x.shape[0]
            present = ~np.isnan(self.data_x[:, 0, :k + 1])
            self.set_positions([int(np.argmax(present[:, j])) if present[:, j].any() else N for j in range(k + 1)], k)

    def set_positions(self, first, k):
        """The position state of iteration k from first[j], the first unconverged slice of iteration j <= k: the rows of
        iteration j are the slices first[j] .. N-1, appended in that order (parareal.py:336-339).  fit() derives first
        from data_x; the device drivers, which hold no observation cube, pass the list they keep."""
        N = self.N
        self.k = k
        self._first = np.asarray(first[:k + 1], dtype=np.int64)
        self._offset = np.concatenate([[0], np.cumsum(N - self._first)])[:k + 1]
        self._present = np.arange(N)[:, None] >= self._first[None, :]

    def neighbour_table(self, first, I):
        """[N - I, m] int64: the rows neighbour_rows chooses for the predicts at slices I .. N-1 of iteration
        len(first) - 1, in slice order (so 'col+rnd' draws rng2 as the host driver does)"""
        self.set_positions(first, len(first) - 1)
        return np.array([self.neighbour_rows(i) for i in range(I, self.N)], dtype=np.int64).reshape(self.N - I, -1)

    def _row(self, i, j):
        return int(self._offset[j] + i - self._first[j])

    def neighbour_rows(self, i):
        """dataset row indices chosen by the rule for a predict at slice i of iteration self.k"""
        k, nn, nt = self.k, self.nn, self.nntype
        N = self._present.shape[0]
        have = lambda s, j: 0 <= s < N and self._present[s, j]
        if nt == 'col_only':
            return [self._row(i, j) for j in range(k + 1)]
        if nt == 'col+rnd':
            nn = max(10, k + 2) if nn == 'adaptive' else nn
            on_col = min(nn, k + 1)
            col = [self._row(i, j) for j in range(k + 1 - on_col, k + 1)]
            n_rows = int(self._offset[k] + N - self._first[k])  # the dataset's rows: iterations 0 .. k
            cands = self.rng2.permutation(np.arange(n_rows))[:nn]
            near = [int(c) for c in cands if int(c) not in col][:nn - on_col]
            rows = col + near
            assert len(rows) == nn
            return rows
        if nt == 'row_col':
            # all (slice, iteration) pairs ordered by |iteration - k| + |slice - i| (stable argsort of the flattened grid)
            it = np.arange(k + 1)[None, :] + np.zeros((N, 1))
            sl = np.arange(N)[:, None] + np.zeros((1, k + 1))
            order = np.argsort((np.abs(it - k) + np.abs(sl - i)).ravel(), kind='quicksort')
            rows = []
            for f in order:
                s, j = int(f // (k + 1)), int(f % (k + 1))
                if self._present[s, j]:
                    rows.append(self._row(s, j))
                    if len(rows) == nn:
                        break
        elif nt == 'row':
            rows = []
            for j in range(k, -1, -1):
                for s in _cycle(i, N):
                    if have(s, j):
                        rows.append(self._row(s, j))
                if len(rows) >= nn:
                    break
            rows = rows[:nn]
        else:  # col_full
            rows = []
            for s in _cycle(i, N):
                for j in range(k, -1, -1):
                    if have(s, j):
                        rows.append(self._row(s, j))
                if len(rows) >= nn:
                    break
            rows = rows[:nn]
        if len(rows) < nn:
            raise Exception(f"nntype {nt!r}: only {len(rows)} observations for nn={nn}")
        return rows

    def predict(self, new_x, prev_F=None, prev_G=None, *args, **kwargs):
        if self.nntype == 'nn':
            return super().predict(new_x, prev_F, prev_G, *args, **kwargs)
        import torch
        i = kwargs['i']
        rows = self.neighbour_rows(i)
        m = len(rows)
        if m > 160:
            raise Exception('more than 160 neighbours are not supported (include/nngpara.h: NNGP_MAX_NEIGHBOURS_BIG)')
        h = self.handle()
        dev = torch.device('cuda', h.device)
        q = np.asarray(new_x, dtype=float).reshape(1, -1)
        diff = self.x[rows] - q
        dist = np.zeros(m)
        for jj in range(diff.shape[1]):          # strict left-to-right sum, as for the nearest-neighbour rule
            dist = dist + diff[:, jj] * diff[:, jj]
        starts = self.draw_starts(1)
        t_q = torch.from_numpy(q).to(dev)
        t_idx = torch.tensor([rows], dtype=torch.int64, device=dev)
        t_dist = torch.from_numpy(dist[None]).to(dev)
        t_st = torch.from_numpy(starts).to(dev)
        pred = torch.empty((1, self.n), dtype=torch.float64, device=dev)
        h.fit_predict(t_q, t_idx, t_dist, 1, m, self.n_restarts, t_st, self.fatol, self.xatol, pred,
                      stream=torch.cuda.current_stream(dev).cuda_stream)
        self.train_count += self.n * N_JITTER * self.n_restarts
        return pred.cpu().numpy()[0]


NNGP_alt = CudaNNGPAlt
