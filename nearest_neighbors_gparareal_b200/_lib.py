"""ctypes binding of libnngpara.so (the C ABI declared in include/nngpara.h).

The library is the product: if it is missing, or there is no Blackwell GPU, every device entry
point raises -- there is deliberately no NumPy fallback."""
import ctypes
import os
import threading

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NNGPARA_LIB") or os.path.join(_PKG, "libnngpara.so")  # override: kernel-variant experiments

c_double_p = ctypes.POINTER(ctypes.c_double)
c_ll_p = ctypes.POINTER(ctypes.c_longlong)
c_int_p = ctypes.POINTER(ctypes.c_int)
c_i8_p = ctypes.POINTER(ctypes.c_byte)
vp = ctypes.c_void_p
ci = ctypes.c_int
cll = ctypes.c_longlong
cd = ctypes.c_double

# name -> (restype, argtypes); every symbol include/nngpara.h declares
SIGNATURES = {
    "nngp_abi_version": (ci, []),
    "nngp_create": (ci, [ci, ctypes.POINTER(vp)]),
    "nngp_destroy": (ci, [vp]),
    "nngp_last_error": (ctypes.c_char_p, [vp]),
    "nngp_synchronize": (ci, [vp, vp]),
    "nngp_bench_fp64": (ci, [vp, ci, c_double_p]),
    "nngp_bench_copy": (ci, [vp, cll, c_double_p]),
    "nngp_system_create": (ci, [vp, ci, ci, vp, ci, ci, vp, vp, c_int_p]),
    "nngp_rhs_eval": (ci, [vp, ci, ci, vp, vp, vp]),
    "nngp_rhs_eval_host": (ci, [vp, ci, ci, vp, vp]),
    "nngp_rk_batch": (ci, [vp, ci, ci, ci, cll, ci, vp, vp, vp, cll, vp, cll, vp]),
    "nngp_rk_batch_host": (ci, [vp, ci, ci, ci, cll, ci, vp, vp, vp, vp]),
    "nngp_rk_full": (ci, [vp, ci, ci, ci, cll, ci, vp, vp, vp, cll, vp, vp]),
    "nngp_rk_full_host": (ci, [vp, ci, ci, ci, cll, cd, cd, vp, vp]),
    "nngp_get_tableau": (ci, [ci, c_int_p, vp, vp, vp]),
    "nngp_dataset_reserve": (ci, [vp, cll, ci]),
    "nngp_dataset_reset": (ci, [vp]),
    "nngp_dataset_truncate": (ci, [vp, cll]),
    "nngp_dataset_append": (ci, [vp, vp, vp, cll, vp]),
    "nngp_dataset_append_host": (ci, [vp, vp, vp, cll]),
    "nngp_dataset_rows": (cll, [vp]),
    "nngp_dataset_dim": (ci, [vp]),
    "nngp_knn": (ci, [vp, vp, ci, ci, cll, vp, vp, vp]),
    "nngp_knn_host": (ci, [vp, vp, ci, ci, cll, vp, vp]),
    "nngp_fit_predict": (ci, [vp, vp, vp, vp, ci, ci, ci, vp, cd, cd, vp, vp, vp, vp, vp, vp, vp, vp]),
    "nngp_predict_host": (ci, [vp, vp, ci, ci, cll, ci, vp, cd, cd, vp, vp, vp, vp, vp, vp, vp, vp]),
    "nngp_predict_host_block": (ci, [vp, vp, ci, ci, cll, ci, vp, cd, cd, ci, ci, vp, vp, vp, vp, vp, vp, vp, vp]),
    "nngp_gp_nll": (ci, [vp, vp, ci, ci, ci, vp, vp, vp, vp]),
    "nngp_gp_mean": (ci, [vp, vp, vp, vp, ci, ci, vp, vp, vp, vp]),
    "nngp_sweep": (ci, [vp, ci, ci, ci, cll, vp, ci, ci, ci, ci, vp, cd, cd, vp, vp, ci, vp]),
    "nngp_sweep_shard": (ci, [vp, ci, ci, ci, cll, vp, ci, ci, ci, ci, ci, ci, vp, cd, cd, vp, vp, ci, ci, ci, vp]),
    "nngp_append_iteration": (ci, [vp, vp, vp, vp, ci, ci, ci, vp]),
    "nngp_rowwise_maxabs_diff": (ci, [vp, vp, vp, ci, ci, vp, vp]),
    "nngp_selftest_math": (ci, [vp, vp, ci, vp, vp, vp, vp]),
    "nngp_launch_count": (cll, [vp]),
    "nngp_set_pivot_guard": (ci, [vp, cd]),
    "nngp_get_pivot_guard": (cd, [vp]),
    "nngp_set_fit_mode": (ci, [vp, ci]),
    "nngp_set_fit_budget": (ci, [vp, ci]),
    "nngp_counters": (ci, [vp, c_ll_p, c_ll_p, ci]),
    "nngp_profile_enable": (ci, [vp, ci]),
    "nngp_profile_read": (ci, [vp, vp, vp, ci]),
    "nngp_seg_reserve": (ci, [vp, ci, cll, ci]),
    "nngp_seg_reset": (ci, [vp]),
    "nngp_seg_rows": (cll, [vp, ci]),
    "nngp_seg_cap": (cll, [vp]),
    "nngp_seg_append_iteration": (ci, [vp, ci, vp, vp, vp, vp, vp, cll, ci, ci, vp]),
    "nngp_knn_segmented": (ci, [vp, vp, cll, ci, ci, vp, vp, vp, vp, vp, vp]),
    "nngp_copy_rows": (ci, [vp, vp, vp, vp, vp, cll, cll, vp]),
    "nngp_ensemble_sweep": (ci, [vp, ci, ci, ci, cll, vp, ci, ci, vp, vp, vp, vp, vp, ci, vp, cd, cd, vp, vp, ci, vp]),
    "nngp_fit_predict_mixed": (ci, [vp, vp, vp, vp, ci, vp, ci, vp, cd, cd, vp, vp, vp, vp, vp, vp, vp, vp]),
    "nngp_listed_prep": (ci, [vp, vp, cll, ci, ci, vp, ci, vp, vp, vp]),
    "nngp_sweep_listed_shard": (ci, [vp, ci, ci, ci, cll, vp, ci, ci, ci, ci, ci, vp, ci, vp, cd, cd, vp, vp, ci, ci, ci,
                                     vp]),
}

SYSTEM_IDS = {"FHN_ODE": 0, "Rossler": 1, "Hopf": 2, "DblPend": 3, "Brusselator": 4, "Lorenz": 5,
              "ThomasLabyrinth": 6, "FHN_PDE": 7, "Burgers": 8}
METHODS = {"RK1": 1, "RK2": 2, "RK4": 4, "RK8": 8}
H_LINSPACE, H_CONST = 0, 1

_lib = None
_lock = threading.Lock()


class NNGPError(RuntimeError):
    pass


def load_library():
    """dlopen libnngpara.so and declare every prototype; raises if it was not built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH) and "NNGPARA_LIB" not in os.environ:
                # not built yet (fresh checkout): compile in-tree with nvcc -- never a CPU fallback
                try:
                    from .build import build
                    build()
                except Exception as exc:
                    raise NNGPError(f"{LIB_PATH} is missing and could not be built ({exc}); run "
                                    "`python __graft_entry__.py` (build()) first; there is no CPU fallback")
            if not os.path.exists(LIB_PATH):
                raise NNGPError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first; "
                                "there is no CPU fallback")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def _ptr(a):
    """host ndarray / device tensor / int address / None -> void*"""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):  # torch tensor (device buffer)
        return a.data_ptr()
    raise TypeError(f"cannot take the address of {type(a)}")


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Handle:
    """One library handle per process / device (nngp_create)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = vp()
        rc = self.lib.nngp_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise NNGPError(self.lib.nngp_last_error(None).decode())
        self.h = h
        self.device = device
        self._systems = {}

    def check(self, rc):
        if rc != 0:
            raise NNGPError(self.lib.nngp_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.nngp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- thin wrappers; array arguments may be host ndarrays (host variants) or device tensors
    def system_create(self, system_id, d, params, normalize, mn, mx):
        params = as_f64(params)
        out = ci(-1)
        mn_a = as_f64(mn) if normalize else None
        mx_a = as_f64(mx) if normalize else None
        self.check(self.lib.nngp_system_create(self.h, system_id, d, _ptr(params), params.size,
                                               1 if normalize else 0, _ptr(mn_a), _ptr(mx_a),
                                               ctypes.byref(out)))
        return out.value

    def rhs_eval_host(self, sys, u):
        u = as_f64(u)
        u2 = u.reshape(-1, u.shape[-1])
        out = np.empty_like(u2)
        self.check(self.lib.nngp_rhs_eval_host(self.h, sys, u2.shape[0], _ptr(u2), _ptr(out)))
        return out.reshape(u.shape)

    def rk_batch_host(self, sys, method, h_mode, steps, t0, t1, u0):
        t0, t1, u0 = as_f64(t0).ravel(), as_f64(t1).ravel(), as_f64(u0)
        u0 = u0.reshape(t0.shape[0], -1)
        u1 = np.empty_like(u0)
        self.check(self.lib.nngp_rk_batch_host(self.h, sys, method, h_mode, int(steps), t0.shape[0],
                                               _ptr(t0), _ptr(t1), _ptr(u0), _ptr(u1)))
        return u1

    def rk_full_host(self, sys, method, h_mode, steps, t0, t1, u0):
        u0 = as_f64(u0).ravel()
        traj = np.empty((int(steps) + 1, u0.shape[0]))
        self.check(self.lib.nngp_rk_full_host(self.h, sys, method, h_mode, int(steps), float(t0), float(t1),
                                              _ptr(u0), _ptr(traj)))
        return traj

    def rk_batch(self, sys, method, h_mode, steps, n, d_t0, d_t1, d_u0, ld0, d_u1, ld1, stream=None):
        self.check(self.lib.nngp_rk_batch(self.h, sys, method, h_mode, int(steps), int(n), _ptr(d_t0),
                                          _ptr(d_t1), _ptr(d_u0), int(ld0), _ptr(d_u1), int(ld1), stream))

    def get_tableau(self, method):
        S = ci(0)
        a = np.zeros(121)
        b = np.zeros(11)
        c = np.zeros(11)
        rc = self.lib.nngp_get_tableau(method, ctypes.byref(S), _ptr(a), _ptr(b), _ptr(c))
        if rc != 0:
            raise NotImplementedError("Only RK1, RK2, RK4 and RK8 are implemented")
        s = S.value
        return a[:s * s].reshape(s, s).copy(), b[:s].copy(), c[:s].copy()

    def dataset_reserve(self, cap_rows, d):
        self.check(self.lib.nngp_dataset_reserve(self.h, int(cap_rows), int(d)))

    def dataset_reset(self):
        self.check(self.lib.nngp_dataset_reset(self.h))

    def dataset_rows(self):
        return int(self.lib.nngp_dataset_rows(self.h))

    def dataset_dim(self):
        return int(self.lib.nngp_dataset_dim(self.h))

    def dataset_append_host(self, x, y):
        x, y = as_f64(x), as_f64(y)
        self.check(self.lib.nngp_dataset_append_host(self.h, _ptr(x), _ptr(y), x.shape[0]))

    def dataset_append(self, d_x, d_y, rows, stream=None):
        self.check(self.lib.nngp_dataset_append(self.h, _ptr(d_x), _ptr(d_y), int(rows), stream))

    def knn_host(self, q, m, n_rows=0):
        q = as_f64(q)
        q = q.reshape(-1, q.shape[-1])
        idx = np.empty((q.shape[0], m), dtype=np.int64)
        dist = np.empty((q.shape[0], m))
        self.check(self.lib.nngp_knn_host(self.h, _ptr(q), q.shape[0], int(m), int(n_rows), _ptr(idx), _ptr(dist)))
        return idx, dist

    def knn(self, d_q, nq, m, n_rows, d_idx, d_dist, stream=None):
        self.check(self.lib.nngp_knn(self.h, _ptr(d_q), int(nq), int(m), int(n_rows), _ptr(d_idx), _ptr(d_dist), stream))

    def predict_host(self, q, m, starts, n_restarts, fatol, xatol, n_rows=0, details=False, block=None, pred_out=None):
        q = as_f64(q)
        q = q.reshape(-1, q.shape[-1])
        nq, d = q.shape
        starts = np.ascontiguousarray(starts, dtype=np.int8)
        assert starts.size == nq * d * 9 * n_restarts * 2, "starts must be [nq,d,9,R,2]"
        # pred_out: a caller-owned float64 buffer of nq*d values, host ndarray or device tensor (see nngpara.h)
        pred = np.empty((nq, d)) if pred_out is None else pred_out
        out = dict(pred=pred)
        idx = th = jit = fv = nfev = fvals = thetas = None
        if details:
            idx = np.empty((nq, m), dtype=np.int64)
            th = np.empty((nq, d, 2))
            jit = np.empty((nq, d))
            fv = np.empty((nq, d))
            nfev = np.empty((nq, d, 9, n_restarts), dtype=np.int32)
            fvals = np.empty((nq, d, 9, n_restarts))
            thetas = np.empty((nq, d, 9, n_restarts, 2))
            out.update(idx=idx, theta_opt=th, jitter_opt=jit, fval_opt=fv, nfev=nfev, fvals=fvals, thetas=thetas)
        j0, dl = block if block is not None else (0, -1)  # block: (first dim, count) -- only those dims are fitted
        self.check(self.lib.nngp_predict_host_block(self.h, _ptr(q), nq, int(m), int(n_rows), int(n_restarts),
                                                    _ptr(starts), float(fatol), float(xatol), int(j0), int(dl),
                                                    _ptr(pred), _ptr(idx), _ptr(th), _ptr(jit), _ptr(fv), _ptr(nfev),
                                                    _ptr(fvals), _ptr(thetas)))
        return out

    def fit_predict(self, d_q, d_idx, d_dist, nq, m, n_restarts, d_starts, fatol, xatol, d_pred,
                    d_theta=None, d_jit=None, d_fval=None, d_nfev=None, d_fvals=None, d_thetas=None, stream=None):
        self.check(self.lib.nngp_fit_predict(self.h, _ptr(d_q), _ptr(d_idx), _ptr(d_dist), int(nq), int(m),
                                             int(n_restarts), _ptr(d_starts), float(fatol), float(xatol),
                                             _ptr(d_pred), _ptr(d_theta), _ptr(d_jit), _ptr(d_fval),
                                             _ptr(d_nfev), _ptr(d_fvals), _ptr(d_thetas), stream))

    def fit_predict_mixed(self, d_q, d_idx, d_dist, m, n_restarts, d_starts, fatol, xatol, d_pred, d_theta=None,
                          d_jit=None, d_fval=None, d_nfev=None, d_fvals=None, d_thetas=None, stream=None):
        """fit_predict with one neighbour count m[q] per predict; idx / dist rows max(m) apart"""
        m = np.ascontiguousarray(m, dtype=np.int32)
        self.check(self.lib.nngp_fit_predict_mixed(self.h, _ptr(d_q), _ptr(d_idx), _ptr(d_dist), m.size, _ptr(m),
                                                   int(n_restarts), _ptr(d_starts), float(fatol), float(xatol),
                                                   _ptr(d_pred), _ptr(d_theta), _ptr(d_jit), _ptr(d_fval),
                                                   _ptr(d_nfev), _ptr(d_fvals), _ptr(d_thetas), stream))

    def listed_prep(self, d_q, ld_q, nq, m, d_rows, ld, d_dist, d_r2, stream=None):
        self.check(self.lib.nngp_listed_prep(self.h, _ptr(d_q), int(ld_q), int(nq), int(m), _ptr(d_rows), int(ld),
                                             _ptr(d_dist), _ptr(d_r2), stream))

    def gp_nll(self, d_idx, nq, m, nt, d_theta, d_jitter10, d_nll, stream=None):
        self.check(self.lib.nngp_gp_nll(self.h, _ptr(d_idx), int(nq), int(m), int(nt), _ptr(d_theta),
                                        _ptr(d_jitter10), _ptr(d_nll), stream))

    def gp_mean(self, d_q, d_idx, d_dist, nq, m, d_theta, d_jitter, d_pred, stream=None):
        self.check(self.lib.nngp_gp_mean(self.h, _ptr(d_q), _ptr(d_idx), _ptr(d_dist), int(nq), int(m),
                                         _ptr(d_theta), _ptr(d_jitter), _ptr(d_pred), stream))

    def sweep(self, sys, method_g, h_mode, steps_g, d_t, N, I, m, n_restarts, d_starts, fatol, xatol,
              d_u_next, d_uG_next, d, stream=None):
        self.check(self.lib.nngp_sweep(self.h, sys, method_g, h_mode, int(steps_g), _ptr(d_t), int(N), int(I),
                                       int(m), int(n_restarts), _ptr(d_starts), float(fatol), float(xatol),
                                       _ptr(d_u_next), _ptr(d_uG_next), int(d), stream))

    def sweep_shard(self, sys, method_g, h_mode, steps_g, d_t, N, I, i_first, i_count, m, n_restarts, d_starts, fatol,
                    xatol, d_u_next, d_uG_next, d, j0, dl, stream=None):
        self.check(self.lib.nngp_sweep_shard(self.h, sys, method_g, h_mode, int(steps_g), _ptr(d_t), int(N), int(I),
                                             int(i_first), int(i_count), int(m), int(n_restarts), _ptr(d_starts),
                                             float(fatol), float(xatol), _ptr(d_u_next), _ptr(d_uG_next), int(d),
                                             int(j0), int(dl), stream))

    def sweep_listed_shard(self, sys, method_g, h_mode, steps_g, d_t, N, I, i_first, i_count, rows, n_restarts, d_starts,
                           fatol, xatol, d_u_next, d_uG_next, d, j0, dl, stream=None):
        """sweep_shard with host-chosen neighbours: rows [(N-I), m] (host int64) lists the dataset rows of each slice"""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        assert rows.ndim == 2 and rows.shape[0] == N - I, "rows must be [(N-I), m]"
        self.check(self.lib.nngp_sweep_listed_shard(self.h, sys, method_g, h_mode, int(steps_g), _ptr(d_t), int(N),
                                                    int(I), int(i_first), int(i_count), rows.shape[1], _ptr(rows),
                                                    int(n_restarts), _ptr(d_starts), float(fatol), float(xatol),
                                                    _ptr(d_u_next), _ptr(d_uG_next), int(d), int(j0), int(dl), stream))

    def append_iteration(self, d_u_cur, d_uF, d_uG_cur, N, I, d, stream=None):
        self.check(self.lib.nngp_append_iteration(self.h, _ptr(d_u_cur), _ptr(d_uF), _ptr(d_uG_cur), int(N),
                                                  int(I), int(d), stream))

    def rowwise_maxabs_diff(self, d_a, d_b, rows, d, d_err, stream=None):
        self.check(self.lib.nngp_rowwise_maxabs_diff(self.h, _ptr(d_a), _ptr(d_b), int(rows), int(d), _ptr(d_err), stream))

    # -- segmented store and ensemble sweep (host int arrays are converted here)
    def seg_reserve(self, n_members, cap_rows, d):
        self.check(self.lib.nngp_seg_reserve(self.h, int(n_members), int(cap_rows), int(d)))

    def seg_reset(self):
        self.check(self.lib.nngp_seg_reset(self.h))

    def seg_rows(self, member):
        return int(self.lib.nngp_seg_rows(self.h, int(member)))

    def seg_cap(self):
        return int(self.lib.nngp_seg_cap(self.h))

    def seg_append_iteration(self, members, I, d_u_cur, d_uF, d_uG_cur, ld_state, N, d, stream=None):
        members, I = np.ascontiguousarray(members, dtype=np.int32), np.ascontiguousarray(I, dtype=np.int32)
        self.check(self.lib.nngp_seg_append_iteration(self.h, members.size, _ptr(members), _ptr(I), _ptr(d_u_cur),
                                                      _ptr(d_uF), _ptr(d_uG_cur), int(ld_state), int(N), int(d), stream))

    def knn_segmented(self, d_q, ld_q, nq, m, base, rows, d_idx, d_dist, d_r2=None, stream=None):
        base, rows = np.ascontiguousarray(base, dtype=np.int64), np.ascontiguousarray(rows, dtype=np.int64)
        assert base.size == nq and rows.size == nq
        self.check(self.lib.nngp_knn_segmented(self.h, _ptr(d_q), int(ld_q), int(nq), int(m), _ptr(base), _ptr(rows),
                                               _ptr(d_idx), _ptr(d_dist), _ptr(d_r2), stream))

    def copy_rows(self, d_src, d_src_idx, d_dst, d_dst_idx, rows, d, stream=None):
        self.check(self.lib.nngp_copy_rows(self.h, _ptr(d_src), _ptr(d_src_idx), _ptr(d_dst), _ptr(d_dst_idx),
                                           int(rows), int(d), stream))

    def ensemble_sweep(self, sys, method_g, h_mode, steps_g, d_t_pos, N, members, I, m, n_restarts, d_starts, fatol,
                       xatol, d_u_next, d_uG_next, d, listed=None, rows=None, stream=None):
        """Position p sweeps member members[p] from slice I[p] with m[p] neighbours on its grid d_t_pos[p] (device
        [E, N+1]).  listed (None: no position) marks the positions that take the host lists rows[p] ([N - I[p], m[p]]
        global store rows; None for the others) instead of the segmented kNN."""
        members, I = np.ascontiguousarray(members, dtype=np.int32), np.ascontiguousarray(I, dtype=np.int32)
        m = np.ascontiguousarray(m, dtype=np.int32)
        assert m.size == members.size
        flat = None
        if listed is not None:
            listed = np.ascontiguousarray(listed, dtype=np.int32)
            assert listed.size == members.size and len(rows) == members.size
            blocks = []
            for p in range(members.size):
                if listed[p]:
                    b = np.asarray(rows[p], dtype=np.int64).reshape(-1, int(m[p]))
                    assert b.shape[0] == N - I[p], "the lists of position p must be [N - I[p], m[p]]"
                    blocks.append(b.ravel())
            flat = np.ascontiguousarray(np.concatenate(blocks) if blocks else np.zeros(0, np.int64))
        self.check(self.lib.nngp_ensemble_sweep(self.h, sys, method_g, h_mode, int(steps_g), _ptr(d_t_pos), int(N),
                                                members.size, _ptr(members), _ptr(I), _ptr(m), _ptr(listed), _ptr(flat),
                                                int(n_restarts), _ptr(d_starts), float(fatol), float(xatol),
                                                _ptr(d_u_next), _ptr(d_uG_next), int(d), stream))

    def selftest_math(self, d_x, n, d_exp, d_rcp, d_exp10=None, stream=None):
        self.check(self.lib.nngp_selftest_math(self.h, _ptr(d_x), int(n), _ptr(d_exp), _ptr(d_rcp),
                                               _ptr(d_exp10) if d_exp10 is not None else None, stream))

    def synchronize(self, stream=None):
        self.check(self.lib.nngp_synchronize(self.h, stream))

    def dataset_truncate(self, rows):
        self.check(self.lib.nngp_dataset_truncate(self.h, int(rows)))

    def launch_count(self):
        return int(self.lib.nngp_launch_count(self.h))

    def set_pivot_guard(self, ulps):
        """failed-pivot threshold of the GP factorisation in ulps of the diagonal (default 1; round 1 used 4)"""
        self.check(self.lib.nngp_set_pivot_guard(self.h, float(ulps)))

    def set_fit_mode(self, mode):
        """'auto' | 'warp' (one search per warp) | 'grouped' (several searches per warp); same bits either way"""
        self.check(self.lib.nngp_set_fit_mode(self.h, {"auto": 0, "warp": 1, "grouped": 2, "quad": 3}[mode]))

    def set_fit_budget(self, evaluations):
        """evaluations after which a search moves to the four-warp continuation kernel (0: never); same bits"""
        self.check(self.lib.nngp_set_fit_budget(self.h, int(evaluations)))

    def get_pivot_guard(self):
        return float(self.lib.nngp_get_pivot_guard(self.h))

    def counters(self, reset=False):
        """(Nelder-Mead runs, objective evaluations) since the last reset"""
        a, b = cll(0), cll(0)
        self.check(self.lib.nngp_counters(self.h, ctypes.byref(a), ctypes.byref(b), 1 if reset else 0))
        return a.value, b.value

    def profile_enable(self, on=True):
        self.check(self.lib.nngp_profile_enable(self.h, 1 if on else 0))

    def profile_read(self, reset=True):
        """{class: (milliseconds, launches)} for rk / knn / gp_prep / gp_fit / other"""
        ms = np.zeros(5)
        cnt = np.zeros(5, dtype=np.int64)
        self.check(self.lib.nngp_profile_read(self.h, _ptr(ms), _ptr(cnt), 1 if reset else 0))
        names = ("rk", "knn", "gp_prep", "gp_fit", "other")
        return {n: (float(ms[i]), int(cnt[i])) for i, n in enumerate(names)}

    def bench_fp64(self, iters=20000):
        out = cd(0.0)
        self.check(self.lib.nngp_bench_fp64(self.h, int(iters), ctypes.byref(out)))
        return out.value

    def bench_copy(self, nbytes=1 << 30):
        out = cd(0.0)
        self.check(self.lib.nngp_bench_copy(self.h, int(nbytes), ctypes.byref(out)))
        return out.value


_default = {}


def default_handle(device=None):
    """Process-wide handle for `device` (default: LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _default:
        _default[device] = Handle(device)
    return _default[device]
