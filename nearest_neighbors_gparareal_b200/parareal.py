"""Host mirror of the reference driver (parareal.py:26-471, 812-1060).

`Parareal` / `PararealLight` run the reference's outer loop on the host against the solver /
model / executor protocols, so any `SolverAbstr` / `ModelAbstr` plugs in; with `CudaSolverRK`,
`CudaNNGP` and `CudaPool` every arithmetic step is a C-ABI call on host buffers (this is the
end-to-end path bench.py reports as `e2e`).

`PararealDevice` keeps the whole iteration resident on the GPU: one batched RK launch for the
fine solves (sharded by time slice across ranks, exchanged with a single all-gather), a device
dataset append, the fused on-device sweep (nngp_sweep) and one small device->host read of the
per-slice errors per iteration.
"""
import os
import pickle
import time

import numpy as np

from . import _lib
from .models import BareParareal, CudaNNGP, ModelAbstr, N_JITTER
from .pool import CudaPool, MyPool
from .solver import CudaSolverRK, SolverAbstr
from .systems import ODE
from .utils import dim_block
from .checkpoint import RunHistory, adopt_model, state_from_objs


def slice_block(I, N, rank, world):
    """Contiguous block of the unconverged slices I..N-1 owned by `rank`: (chunk, first, count)."""
    n_act = N - I
    chunk = (n_act + world - 1) // world
    lo = min(I + rank * chunk, N)
    cnt = max(0, min(chunk, N - lo))
    return chunk, lo, cnt


def gather_fine_rows(uF, I, chunk, rank, world, group=None):
    """The one collective of an iteration: every rank wrote rows uF[lo+1 : lo+1+cnt] of its block;
    afterwards all ranks hold uF[I+1 : N+1].  uF needs world*chunk rows after row I."""
    import torch.distributed as dist
    view = uF[I + 1:I + 1 + world * chunk]
    mine = view[rank * chunk:(rank + 1) * chunk]
    if dist.get_backend(group) != 'nccl':
        mine = mine.clone()  # gloo (CPU tests) does not take an input aliasing the output
    dist.all_gather_into_tensor(view, mine, group=group)


def advance(err_k, I, eps):
    """parareal.py:402-416 for one run: err_k[I] = 0, then I moves over the slices whose error is below eps"""
    err_k[I] = 0
    N = err_k.shape[0] - 1
    for p in range(I + 1, N + 1):
        if err_k[p] < eps:
            I += 1
        else:
            break
    return I


class Parareal():
    def __init__(self, ode, solver, tspan, N, epsilon=5e-7, verbose='v', **kwargs):
        if not isinstance(ode, ODE):
            raise Exception('ode must be an instance of the ODE class, see systems.py file.')
        if not isinstance(solver, SolverAbstr):
            raise Exception('solver must be an instance of the SolverAbstr class, see solver.py file.')
        self.tspan = tspan
        self.N = N
        self.epsilon = epsilon
        self.runs = dict()
        self.fine = None
        self.ode_name = ode.name
        self.n = ode.get_dim()
        self.ode = ode
        self.solver = solver
        self.f = ode.get_vector_field()
        self.u0 = ode.get_init_cond()
        self.verbose = verbose

    keep_history = True  # Parareal returns u[N+1, d, K]; PararealLight only the last iterate

    def _get_pool(self, *args, **kwargs):
        pool = kwargs.get('pool', None)
        if isinstance(pool, int) or pool is None:
            # the reference spawns `pool` CPU worker processes (parareal.py:60-61); here the GPU
            # is the worker pool whatever the requested count
            pool = CudaPool()
        return pool

    def run(self, *args, _run_from_int=False, **kwargs):
        pool = self._get_pool(*args, **kwargs)
        kwargs['pool'] = pool
        try:
            if _run_from_int:
                out = self._run_from_int(*args, **kwargs)
            else:
                out = self._run(*args, **kwargs)
        except Exception:
            pool.shutdown()
            raise
        pool.shutdown()
        return out

    # ---- continuous trajectory (parareal.py:487-508) --------------------------------------------
    def build_cont_traj(self, key=None):
        """The fine solver's full trajectory through the slices of a finished run: vstack of
        solver.run_F_full(t_i, t_{i+1}, u_i) for the last iterate (parareal.py:487-508)."""
        if key is None:
            if len(self.runs) != 1:
                raise Exception('Multiple runs, must specify key')
            key = list(self.runs.keys())[0]
        if isinstance(key, dict) and 't' in key and 'u' in key:
            t, u = key['t'], key['u']
        else:
            t, u = self.runs[key]['t'], self.runs[key]['u']
        return self._build_cont_traj(t, u)

    def _build_cont_traj(self, t, u):
        u = np.asarray(u)
        last = u[:, :, -1] if u.ndim == 3 else u  # Parareal keeps u[N+1, d, K], the light drivers u[N+1, d]
        return np.vstack([self.solver.run_F_full(t[i], t[i + 1], last[i]) for i in range(self.N)])

    def clear_plot_obj(self):
        self.runs = dict()

    # ---- intermediate checkpoints (parareal.py:114-209, 420-431) -------------------------------
    def store(self, name, path='', mdl=None, objs=None):
        """Pickles the driver without its ODE / solver (device handles do not pickle), with the model copy
        `mdl.store()` and the loop state `objs` -- parareal.py:114-139."""
        if len(path) > 0 and not os.path.exists(path):
            os.makedirs(path)
        ode, solver, f = self.ode, self.solver, self.f
        self.ode = self.solver = self.f = None
        pool = None
        if objs is not None:
            pool = objs['kwargs'].get('pool', None)
            objs['kwargs']['pool'] = None
            self.objs = objs
        if mdl is not None:
            self.mdl = mdl.store()
        try:
            with open(os.path.join(path, name), 'wb') as _file:
                pickle.dump(self, _file, pickle.HIGHEST_PROTOCOL)
        finally:
            self.ode, self.solver, self.f = ode, solver, f
            if objs is not None:
                self.objs = None
                objs['kwargs']['pool'] = pool
            if mdl is not None:
                self.mdl = None

    def load_int_dump(self, other, cstm_mdl_name=None, add_model=False, **kwargs):
        """Resumes the run stored in `other` (an unpickled intermediate dump) -- parareal.py:141-189.  `ode`,
        `solver` and `pool` come from this object / kwargs (they are not in the dump)."""
        self.tspan, self.n, self.N, self.epsilon = other.tspan, other.n, other.N, other.epsilon
        self.runs, self.fine, self.ode_name, self.verbose = other.runs, other.fine, other.ode_name, other.verbose
        self.ode = kwargs.pop('ode', self.ode)
        self.solver = kwargs.pop('solver', self.solver)
        if self.ode is None or self.solver is None:
            raise Exception('ode and solver must be given to resume: they are not stored in the dump')
        if self.ode_name != self.ode.name or self.n != self.ode.get_dim():
            raise Exception('Input and previous ODEs do not match')
        self.f = self.ode.get_vector_field()
        self.u0 = self.ode.get_init_cond()
        objs = other.objs
        run_kwargs = {k: v for k, v in dict(objs['kwargs']).items() if k not in ('_reload_objs', '_run_from_int')}
        run_kwargs.update(kwargs)
        mdl = adopt_model(other.mdl, self.n, self.N)  # also dumps written by the reference (checkpoint.py)
        base_time = objs['F_time'] + objs['G_time'] + mdl.get_times()['mdl_tot_t']
        return self.run(mdl, base_time, cstm_mdl_name, add_model, _run_from_int=True, _reload_objs=objs, **run_kwargs)

    def _run_from_int(self, mdl, base_time, cstm_mdl_name, add_model, **kwargs):
        """parareal.py:192-209"""
        mdl.restore_attrs(kwargs['pool'])
        s_time = time.time()
        out = self._parareal(mdl, _load_mdl=True, **kwargs)
        elap_time = time.time() - s_time + base_time
        out['timings']['runtime'] = elap_time
        if add_model:
            out['mdl'] = mdl.store()
        self.runs[mdl.name if cstm_mdl_name is None else cstm_mdl_name] = out
        return out

    def _make_model(self, model, **kwargs):
        if isinstance(model, ModelAbstr):
            return model
        name = model.lower()
        if name == 'parareal':
            return BareParareal(N=self.N, **kwargs)
        if name == 'nngp':
            if 'pool' not in kwargs:
                raise Exception('A worker pool must be provided to run NNGP in parallel')
            kw = dict(kwargs)
            pool = kw.pop('pool')
            if kw.get('nntype', 'nn') != 'nn':   # position-based neighbour rules (nnGPara_with_time.py:27-184)
                from .models_alt import CudaNNGPAlt
                return CudaNNGPAlt(n=self.n, N=self.N, worker_pool=pool, **kw)
            return CudaNNGP(n=self.n, N=self.N, worker_pool=pool, **kw)
        if name == 'gpjax':
            if 'pool' not in kwargs:
                raise Exception('A worker pool must be provided to run NNGP in parallel')
            from .gp_full import CudaGP
            kw = dict(kwargs)
            pool = kw.pop('pool')
            return CudaGP(n=self.n, N=self.N, worker_pool=pool, **kw)
        # 'elm' is outside the scope (SURVEY.md section 2: not in the paper's results or configurations)
        raise Exception('Not implemented')

    def _run(self, model='parareal', cstm_mdl_name=None, add_model=False, **kwargs):
        mdl = self._make_model(model, **kwargs)
        s_time = time.time()
        out = self._parareal(mdl, **kwargs)
        elap_time = time.time() - s_time
        out['timings']['runtime'] = elap_time
        if self.verbose == 'v':
            print(f'Elapsed Parareal time: {elap_time:0.2f}s')
        if add_model:
            out['mdl'] = mdl.store()
        if cstm_mdl_name is None:
            cstm_mdl_name = mdl.name
        self.runs[cstm_mdl_name] = out
        return out

    # the iteration of parareal.py:212-471, state kept as in PararealLight (:851-862)
    def _parareal(self, model, debug=False, early_stop=None, parall='Serial', store_int=False, _load_mdl=False,
                  _reload_objs=None, **kwargs):
        N, eps, n = self.N, self.epsilon, self.n
        solver = self.solver
        t = np.linspace(self.tspan[0], self.tspan[1], num=N + 1)
        parall = parall.lower()
        pool = kwargs.get('pool', None)
        if parall == 'mpi' and pool is None:
            raise Exception('MPI parallel backend requested but no pool of worker provided')
        verbose = kwargs.get('verbose', self.verbose)
        I = 0
        conv_int = []
        err = np.full((N + 1, N), np.nan)
        cur = {key: np.full((N + 1, n), np.nan) for key in ('u', 'uG', 'uF')}
        for a in cur.values():
            a[0] = self.u0
        G_time = F_time = F_time_serial = 0
        k0 = 0
        if _load_mdl:
            # resume (parareal.py:279-297): state after iteration k of the stored run
            o = state_from_objs(_reload_objs)
            I, conv_int, err = o['I'], o['conv_int'], o['err']
            cur = {key: o[key] for key in ('u', 'uG', 'uF')}
            nxt = {key: a.copy() for key, a in cur.items()}
            rec = RunHistory.from_objs(_reload_objs)
            history = [h.copy() for h in rec.u]
            x, D = o['x'], o['D']
            G_time, F_time, F_time_serial = o['G_time'], o['F_time'], _reload_objs.get('F_time_serial', 0)
            k0 = o['k'] + 1
        else:
            # coarse initialisation (parareal.py:264-277)
            state = self.u0
            for i in range(N):
                state, secs = solver.run_G_timed(t[i], t[i + 1], state)
                G_time += secs
                cur['uG'][i + 1] = state
            cur['u'][:] = cur['uG']
            nxt = {key: a.copy() for key, a in cur.items()}
            history = [cur['u'].copy()]
            x = np.zeros((0, n))
            D = np.zeros((0, n))
            rec = RunHistory(N, n, cur['u'], cur['uG']) if store_int else None
        cube = getattr(model, 'wants_data_cube', False)
        if cube:  # data_x / data_D of parareal.py:243-247, only for the models that look observations up by position
            data_x = np.full((N, n, N), np.nan)
            data_D = np.full((N, n, N), np.nan)
            if _load_mdl:
                kk = _reload_objs['data_x'].shape[2]
                data_x[:, :, :kk], data_D[:, :, :kk] = _reload_objs['data_x'], _reload_objs['data_D']
        k = max(k0 - 1, 0)
        for k in range(k0, N):
            if verbose == 'v':
                print(f'{self.ode_name} {model.name} iteration number (out of {N}): {k+1} ')
            s_time = time.time()
            # fine solves of the unconverged slices (parareal.py:309-329)
            if parall in ('mpi', 'joblib'):
                res = list(pool.map(solver.run_F_timed, t[I:N], t[I + 1:N + 1], [cur['u'][i] for i in range(I, N)]))
                cur['uF'][I + 1:N + 1] = np.array([r[0] for r in res])
                F_time_serial += np.array([r[1] for r in res]).mean()
            else:
                last = 0
                for i in range(I, N):
                    cur['uF'][i + 1], last = solver.run_F_timed(t[i], t[i + 1], cur['u'][i])
                F_time_serial += last / (N - I)
            F_time += time.time() - s_time
            # slice I+1 is exact now (parareal.py:331-334)
            nxt['uG'][I + 1] = cur['uG'][I + 1]
            nxt['uF'][I + 1] = cur['uF'][I + 1]
            nxt['u'][I + 1] = cur['uF'][I + 1]
            I += 1
            # training data (parareal.py:336-339)
            x = np.vstack([x, cur['u'][I - 1:N]])
            D = np.vstack([D, cur['uF'][I:N + 1] - cur['uG'][I:N + 1]])
            if store_int and rec is not None:
                rec.add_fine(cur['uF'], I, cur['u'][I - 1:N], cur['uF'][I:N + 1] - cur['uG'][I:N + 1])
            if I == N:
                if verbose == 'v':
                    print('WARNING: early stopping')
                err[:, k] = np.linalg.norm(nxt['u'] - cur['u'], np.inf, 1)
                err[-1, k] = np.nextafter(eps, 0)
                history.append(nxt['u'].copy())
                break
            if cube:
                data_x[I - 1:N, :, k] = cur['u'][I - 1:N]
                data_D[I - 1:N, :, k] = cur['uF'][I:N + 1] - cur['uG'][I:N + 1]
                model.fit_timed(x, D, k=k, data_x=data_x, data_y=data_D)
            else:
                model.fit_timed(x, D, k=k)
            # serial sweep (parareal.py:359-382)
            for i in range(I, N):
                nxt['uG'][i + 1], secs = solver.run_G_timed(t[i], t[i + 1], nxt['u'][i])
                G_time += secs
                preds = model.predict_timed(nxt['u'][i].reshape(1, -1), cur['uF'][i + 1], cur['uG'][i + 1], i=i)
                nxt['u'][i + 1] = preds + nxt['uG'][i + 1]
            if np.any(np.isnan(nxt['uG'])):
                raise Exception("NaN values in initial coarse solve - increase Ng!")
            # convergence bookkeeping (parareal.py:402-416)
            err[:, k] = np.linalg.norm(nxt['u'] - cur['u'], np.inf, 1)
            err[I, k] = 0
            cur['u'][:] = nxt['u']
            cur['uG'][:] = nxt['uG']
            for p in range(I + 1, N + 1):
                if err[p, k] < eps:
                    nxt['uF'][p] = cur['uF'][p]
                    I += 1
                else:
                    break
            cur['uF'][:] = nxt['uF']
            history.append(cur['u'].copy())
            if verbose == 'v':
                print('--> Converged:', I)
            conv_int.append(I)
            if store_int:
                # parareal.py:420-431, the reference's key set and array layout (checkpoint.py)
                rec.add_iterate(cur['u'], cur['uG'])
                name_base = kwargs.get('int_name', f'{self.ode_name}_{self.N}_{model.name}_int')
                int_dir = kwargs.get('int_dir', '')
                u3, uG3, uF3, data_x, data_D = rec.arrays(k, I)
                run_kw = {kk: vv for kk, vv in kwargs.items() if kk not in ('_reload_objs',)}
                _objs = {'t': t, 'I': I, 'verbose': verbose, 'u': u3, 'uG': uG3, 'uF': uF3, 'err': err[:, :k + 2],
                         'x': x, 'D': D, 'data_x': data_x, 'data_D': data_D, 'G_time': G_time, 'F_time': F_time,
                         'F_time_serial': F_time_serial, 'debug': debug, 'early_stop': early_stop, 'parall': parall,
                         'store_int': store_int, 'kwargs': run_kw, 'k': k, 'conv_int': conv_int}
                self.store(path=os.path.join(int_dir, name_base), name=f'{name_base}_{k}', mdl=model, objs=_objs)
            if I == N:
                break
            if (early_stop is not None) and k == (early_stop - 1):
                if verbose == 'v':
                    print('Early stopping due to user condition.')
                break
        timings = {'F_time': F_time, 'G_time': G_time, 'F_time_serial_avg': F_time_serial}
        timings.update(model.get_times())
        u_out = np.stack(history[:k + 1], axis=2) if self.keep_history else history[-1]
        return {'t': t, 'u': u_out, 'u_last': history[-1], 'err': err[:, :k + 1], 'x': x, 'D': D, 'k': k + 1,
                'timings': timings, 'debug_dict': {}, 'converged': I == N, 'conv_int': conv_int}


class PararealLight(Parareal):
    """parareal.py:782-1060: same loop, returns only the last iterate u[N+1, d]."""
    keep_history = False


class PararealDevice(Parareal):
    """Device-resident nnGParareal: the whole iteration of parareal.py:301-439 on the GPU.

    Needs a CudaSolverRK and either the 'nngp' or the 'parareal' model; 'nngp' with a position-based `nntype`
    (models_alt.py) builds each iteration's neighbour lists on the host with the model's own rules and sweeps them
    with nngp_sweep_listed_shard.  With an initialised
    torch.distributed process group of W>1 ranks (one per GPU) the fine solves are sharded by
    time slice: rank r propagates a contiguous block of the unconverged slices, writing straight
    into its part of the gather buffer, and ONE all-gather per iteration makes every rank hold
    all uF rows; the serial sweep is replicated on every rank (bit-identical results).
    """
    keep_history = False

    def __init__(self, ode, solver, tspan, N, epsilon=5e-7, verbose='v', group=None, shard_sweep=True, **kwargs):
        super().__init__(ode, solver, tspan, N, epsilon=epsilon, verbose=verbose, **kwargs)
        if not isinstance(solver, CudaSolverRK):
            raise Exception('PararealDevice needs a CudaSolverRK')
        self.group = group
        # W > 1 ranks: split the d*9*R fits of every predict by output dimension over the ranks and
        # all-gather the d/W predictions per slice (SURVEY.md section 8e, "optional -- measure first":
        # measured in profiles/); needs d % W == 0, otherwise the sweep is replicated
        self.shard_sweep = shard_sweep
        self.events = []

    def _world(self):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(self.group), dist.get_world_size(self.group)
        return 0, 1

    # ---- device state ------------------------------------------------------------------
    def device_setup(self, model, max_rows=None):
        """Allocates the device-resident state and runs the coarse initialisation
        (parareal.py:233-277).  Returns a dict that `device_iteration` advances."""
        import torch
        if not isinstance(model, (CudaNNGP, BareParareal)):
            raise Exception('PararealDevice supports the nngp and parareal models')
        N, n = self.N, self.n
        solver = self.solver
        h, sysid = solver.device()
        dev = torch.device('cuda', h.device)
        rank, world = self._world()
        if max(solver.Nf, solver.Ng) > solver.thresh:
            raise Exception('steps > thresh (RK paging, solver.py:89-96) is only supported by the host driver')
        f64 = dict(dtype=torch.float64, device=dev)
        st = dict(h=h, sys=sysid, dev=dev, rank=rank, world=world, model=model,
                  mF=_lib.METHODS[solver.F], mG=_lib.METHODS[solver.G],
                  stream=torch.cuda.current_stream(dev).cuda_stream, is_gp=isinstance(model, CudaNNGP))
        st['t_host'] = np.linspace(self.tspan[0], self.tspan[1], num=N + 1)
        st['t'] = torch.from_numpy(st['t_host']).to(dev)
        u0 = torch.from_numpy(self.u0).to(dev)
        st['u_cur'] = torch.zeros((N + 1, n), **f64)
        st['uG_cur'] = torch.zeros((N + 1, n), **f64)
        # rows past N are scratch for the in-place all-gather of the last rank's padded block
        st['uF'] = torch.zeros((N + 1 + N + world, n), **f64)
        st['err'] = torch.zeros(N + 1, **f64)
        for key in ('u_cur', 'uG_cur', 'uF'):
            st[key][0] = u0
        # position-based neighbour rule (models_alt.py): the host chooses each predict's rows from the first unconverged
        # slice of every iteration so far, kept here as the dataset grows
        st['listed'] = st['is_gp'] and getattr(model, 'nntype', 'nn') != 'nn'
        st['first'] = []
        if st['is_gp']:
            model._handle = h
            h.dataset_reset()
            st['cap'] = max_rows or min(N * (N + 3) // 2 + 1, N * 16)
            h.dataset_reserve(st['cap'], n)
            model._n_dev = 0
        for i in range(N):  # N dependent one-slice launches
            h.rk_batch(sysid, st['mG'], solver.h_mode, solver.Ng, 1, st['t'][i:], st['t'][i + 1:],
                       st['uG_cur'][i], n, st['uG_cur'][i + 1], n, st['stream'])
        st['u_cur'].copy_(st['uG_cur'])
        st['u_next'] = st['u_cur'].clone()
        st['uG_next'] = st['uG_cur'].clone()
        st['I'] = 0
        st['times'] = dict(F=0.0, sweep=0.0)
        return st

    def device_fine_step(self, st):
        """parareal.py:309-334: fine solves of slices I..N-1 (sharded by slice over the ranks, one
        all-gather), then slice I+1 becomes exact."""
        N, n, solver = self.N, self.n, self.solver
        h, I, rank, world = st['h'], st['I'], st['rank'], st['world']
        if world == 1:
            h.rk_batch(st['sys'], st['mF'], solver.h_mode, solver.Nf, N - I, st['t'][I:], st['t'][I + 1:],
                       st['u_cur'][I], n, st['uF'][I + 1], n, st['stream'])
        else:
            chunk, lo, cnt = slice_block(I, N, rank, world)
            if cnt > 0:
                h.rk_batch(st['sys'], st['mF'], solver.h_mode, solver.Nf, cnt, st['t'][lo:], st['t'][lo + 1:],
                           st['u_cur'][lo], n, st['uF'][lo + 1], n, st['stream'])
            gather_fine_rows(st['uF'], I, chunk, rank, world, self.group)
        st['u_next'][I + 1].copy_(st['uF'][I + 1])
        st['uG_next'][I + 1].copy_(st['uG_cur'][I + 1])
        st['I'] = I + 1

    def device_sweep(self, st, k, starts=None):
        """parareal.py:336-382: dataset append + the serial sweep, all on the device.
        `starts` (device int8 [(N-I), d, 9, R, 2]) may be passed in when already resident."""
        import torch
        N, n, solver = self.N, self.n, self.solver
        h, I, model = st['h'], st['I'], st['model']
        if st['is_gp']:
            if h.dataset_rows() + (N - I + 1) > st['cap']:
                st['cap'] = 2 * st['cap'] + N
                h.dataset_reserve(st['cap'], n)
            h.append_iteration(st['u_cur'], st['uF'], st['uG_cur'], N, I, n, st['stream'])
            model._n_dev = h.dataset_rows()
            st['first'].append(I - 1)
        if I == N:
            return
        if st['is_gp']:
            model.k = k
            model.time_k = k
            rows = None
            if st['listed']:
                rows = model.neighbour_table(st['first'], I)
                m = rows.shape[1]
            else:
                m = min(model.neighbours(k), h.dataset_rows())
            if m > 160:
                raise Exception('nn > 160 neighbours is not supported (include/nngpara.h: NNGP_MAX_NEIGHBOURS_BIG)')
            if starts is None:
                starts = torch.from_numpy(model.draw_starts(N - I)).to(st['dev'])
            st['starts'] = starts  # keep alive until the stream has consumed it
            world = st['world']
            if world > 1 and self.shard_sweep and n % world == 0:
                import torch.distributed as dist
                j0, dl = dim_block(n, st['rank'], world)
                for i in range(I, N):
                    if rows is None:
                        h.sweep_shard(st['sys'], st['mG'], solver.h_mode, solver.Ng, st['t'], N, I, i, 1, m,
                                      model.n_restarts, starts, model.fatol, model.xatol, st['u_next'], st['uG_next'],
                                      n, j0, dl, st['stream'])
                    else:
                        h.sweep_listed_shard(st['sys'], st['mG'], solver.h_mode, solver.Ng, st['t'], N, I, i, 1, rows,
                                             model.n_restarts, starts, model.fatol, model.xatol, st['u_next'],
                                             st['uG_next'], n, j0, dl, st['stream'])
                    row = st['u_next'][i + 1]
                    dist.all_gather_into_tensor(row, row[j0:j0 + dl], group=self.group)
            elif rows is None:
                h.sweep(st['sys'], st['mG'], solver.h_mode, solver.Ng, st['t'], N, I, m, model.n_restarts, starts,
                        model.fatol, model.xatol, st['u_next'], st['uG_next'], n, st['stream'])
            else:
                h.sweep_listed_shard(st['sys'], st['mG'], solver.h_mode, solver.Ng, st['t'], N, I, I, N - I, rows,
                                     model.n_restarts, starts, model.fatol, model.xatol, st['u_next'], st['uG_next'],
                                     n, 0, n, st['stream'])
            model.train_count += (N - I) * n * N_JITTER * model.n_restarts
        else:
            for i in range(I, N):
                h.rk_batch(st['sys'], st['mG'], solver.h_mode, solver.Ng, 1, st['t'][i:], st['t'][i + 1:],
                           st['u_next'][i], n, st['uG_next'][i + 1], n, st['stream'])
                torch.add(st['uF'][i + 1] - st['uG_cur'][i + 1], st['uG_next'][i + 1], out=st['u_next'][i + 1])

    def device_errors(self, st):
        """parareal.py:402: per-slice max-norm of u^{k+1}-u^k; the one device->host read of an iteration"""
        st['h'].rowwise_maxabs_diff(st['u_next'], st['u_cur'], self.N + 1, self.n, st['err'], st['stream'])
        return st['err'].cpu().numpy()

    def device_advance(self, st, err_k):
        """parareal.py:402-416 after a sweep: the new iterate becomes the current one, `I` moves over the slices whose
        error is below epsilon.  err_k = the per-slice errors of this iteration (host array); returns the new I."""
        st['u_cur'].copy_(st['u_next'])
        st['uG_cur'].copy_(st['uG_next'])
        st['I'] = advance(err_k, st['I'], self.epsilon)
        return st['I']

    def _parareal(self, model, early_stop=None, parall='Serial', store_int=False, max_rows=None,
                  iteration_hook=None, **kwargs):
        import torch
        N, eps = self.N, self.epsilon
        verbose = kwargs.get('verbose', self.verbose)
        if store_int and getattr(model, 'nntype', 'nn') != 'nn':
            raise Exception(f"PararealDevice does not write intermediate checkpoints of the position-based neighbour rule "
                            f"nntype={model.nntype!r} (store_int=True): run it with the host driver Parareal")
        tic = time.time()
        st = self.device_setup(model, max_rows=max_rows)
        torch.cuda.synchronize(st['dev'])
        G_time = time.time() - tic
        F_time = sweep_time = 0.0
        rank = st['rank']
        conv_int = []
        err = np.full((N + 1, N), np.nan)
        # store_int: the reference's per-iteration dumps (parareal.py:420-431) -- the device state of every iteration is
        # copied to the host (3 x (N+1) x n doubles) and written in the reference's layout (checkpoint.py); rank 0 only
        rec = xs = Ds = None
        if store_int:
            rec = RunHistory(N, self.n, st['u_cur'].cpu().numpy(), st['uG_cur'].cpu().numpy())
            xs, Ds = [], []
        k = 0
        for k in range(N):
            if verbose == 'v' and rank == 0:
                print(f'{self.ode_name} {model.name} iteration number (out of {N}): {k+1} ')
            tic = time.time()
            self.device_fine_step(st)
            torch.cuda.synchronize(st['dev'])
            F_time += time.time() - tic
            if store_int:
                I1 = st['I']
                uc, uf, ug = st['u_cur'].cpu().numpy(), st['uF'][:N + 1].cpu().numpy(), st['uG_cur'].cpu().numpy()
                xs.append(uc[I1 - 1:N])
                Ds.append(uf[I1:N + 1] - ug[I1:N + 1])
                rec.add_fine(uf, I1, xs[-1], Ds[-1])
            tic = time.time()
            self.device_sweep(st, k)
            I = st['I']
            if I == N:
                if verbose == 'v' and rank == 0:
                    print('WARNING: early stopping')
                err[:, k] = self.device_errors(st)
                err[-1, k] = np.nextafter(eps, 0)
                st['u_cur'].copy_(st['u_next'])
                break
            err[:, k] = self.device_errors(st)
            if iteration_hook is not None:  # (k, device state after the sweep of iteration k) -- diagnostics / replay dumps
                iteration_hook(k, st)
            dt_sweep = time.time() - tic
            sweep_time += dt_sweep
            if st['is_gp']:
                model.pred_time += dt_sweep
                model.pred_times[k] += dt_sweep
                model.tot_train_t += dt_sweep
            if np.any(np.isnan(err[:, k])) and bool(torch.isnan(st['uG_next']).any()):
                raise Exception("NaN values in initial coarse solve - increase Ng!")
            I = self.device_advance(st, err[:, k])  # parareal.py:402-416
            if verbose == 'v' and rank == 0:
                print('--> Converged:', I)
            conv_int.append(I)
            if store_int:
                rec.add_iterate(st['u_cur'].cpu().numpy(), st['uG_cur'].cpu().numpy())
                if rank == 0:
                    name_base = kwargs.get('int_name', f'{self.ode_name}_{self.N}_{model.name}_int')
                    u3, uG3, uF3, data_x, data_D = rec.arrays(k, I)
                    x_all, D_all = np.vstack(xs), np.vstack(Ds)
                    if st['is_gp']:
                        model.x, model.y = x_all, D_all   # the resumed run re-uploads the dataset from the model copy
                    run_kw = {kk: vv for kk, vv in kwargs.items() if kk not in ('_reload_objs',)}
                    _objs = {'t': st['t_host'], 'I': I, 'verbose': verbose, 'u': u3, 'uG': uG3, 'uF': uF3, 'err': err[:, :k + 2],
                             'x': x_all, 'D': D_all, 'data_x': data_x, 'data_D': data_D, 'G_time': G_time, 'F_time': F_time,
                             'debug': False, 'early_stop': early_stop, 'parall': parall, 'store_int': store_int,
                             'kwargs': run_kw, 'k': k, 'conv_int': conv_int}
                    self.store(path=os.path.join(kwargs.get('int_dir', ''), name_base), name=f'{name_base}_{k}', mdl=model,
                               objs=_objs)
            if I == N:
                break
            if (early_stop is not None) and k == (early_stop - 1):
                break
        timings = {'F_time': F_time, 'G_time': G_time, 'F_time_serial_avg': F_time / max(N, 1), 'sweep_time': sweep_time}
        timings.update(model.get_times())
        u = st['u_cur'].cpu().numpy()
        out = {'t': st['t_host'], 'u': u, 'u_last': u, 'err': err[:, :k + 1], 'k': k + 1, 'timings': timings,
               'debug_dict': {}, 'converged': st['I'] == N, 'conv_int': conv_int}
        if st['is_gp']:
            out['n_rows'] = st['h'].dataset_rows()
        return out
