"""Many independent nnGParareal runs as one device-resident ensemble.

`PararealEnsemble.run(seeds=[...])` runs E solves of the same system, solver, N, `n_restarts`, `fatol` and `xatol` in
lockstep; the runs may differ in seed, initial condition, epsilon, early_stop, neighbour count `nn`, neighbour rule
`nntype` (models_alt.py) and time span.  Every iteration makes the launches of one `PararealDevice` iteration, each
over all runs at once: one fine-step launch, one dataset append and one nngp_ensemble_sweep, which per slice makes one
coarse step, one kNN (each run searches its own rows of a segmented store, csrc/knn.cu; the runs with a position rule
take the host's neighbour lists instead) and one fit over all the runs' predicts -- one fit per distinct neighbour
count when the runs' counts differ.  Run e's output dict equals, bit for bit, what
`PararealDevice(...).run(model='nngp', seed=seeds[e], ...)` returns with its settings.

Layout: the state is [E, N+1, d] per array.  At the start of every iteration the member axis is re-ordered by
(finished, I), so the runs still going are a prefix, sorted by their first unconverged slice: at slice i of the sweep
the runs with I <= i are a prefix too, and every launch of the sweep reaches them with the member stride (N+1) d --
no gather or scatter per slice.  Only the fine step, whose slices I_e..N-1 differ per run, gathers its rows into one
batch (nngp_copy_rows) once per iteration.
"""
import time

import numpy as np

from . import _lib
from .models import CudaNNGP, N_JITTER
from .models_alt import NNTYPES, CudaNNGPAlt
from .parareal import advance
from .solver import CudaSolverRK
from .systems import ODE

MAX_NEIGHBOURS = 160  # include/nngpara.h: NNGP_MAX_NEIGHBOURS_BIG


def _check_nn(nn):
    if isinstance(nn, str):
        if nn != 'adaptive':
            raise ValueError(f"nn={nn!r}: 'adaptive' or 1 to {MAX_NEIGHBOURS} neighbours")
        return
    if isinstance(nn, bool) or int(nn) != nn or not (1 <= int(nn) <= MAX_NEIGHBOURS):
        raise ValueError(f'nn={nn}: 1 to {MAX_NEIGHBOURS} neighbours are supported')


def check_run_args(E_lists, model='nngp', store_int=False, nn='adaptive', nntype='nn'):
    """Validates the per-member lists of `PararealEnsemble.run` (dict name -> list or None); returns E.
    `nn` and `nntype` are one value for every member or a list with one per member; E_lists['tspans'] entries are
    [t0, t1] or None."""
    if not isinstance(model, str) or model.lower() != 'nngp':
        raise ValueError(f"PararealEnsemble runs the 'nngp' model only (got {model!r})")
    if store_int:
        raise ValueError('PararealEnsemble does not write intermediate checkpoints (store_int=True)')
    seeds = E_lists.get('seeds')
    if seeds is None or len(seeds) == 0:
        raise ValueError('PararealEnsemble.run needs a non-empty list of seeds')
    E = len(seeds)
    lists = dict(E_lists)
    if isinstance(nn, (list, tuple, np.ndarray)):
        lists['nn'] = nn
    if isinstance(nntype, (list, tuple, np.ndarray)):
        lists['nntype'] = nntype
    for name, v in lists.items():
        if v is not None and len(v) != E:
            raise ValueError(f'{name} has {len(v)} entries, seeds has {E}: give one per member')
    for v in (nn if isinstance(nn, (list, tuple, np.ndarray)) else [nn]):
        _check_nn(v)
    nns = list(nn) if isinstance(nn, (list, tuple, np.ndarray)) else [nn] * E
    rules = list(nntype) if isinstance(nntype, (list, tuple, np.ndarray)) else [nntype] * E
    for e, (rule, v) in enumerate(zip(rules, nns)):
        if rule not in NNTYPES:
            raise ValueError(f'member {e}: unknown nntype {rule!r} (one of {", ".join(NNTYPES)})')
        if rule in ('row_col', 'row', 'col_full') and v == 'adaptive':
            raise ValueError(f"member {e}: nntype {rule!r} needs an integer nn, not 'adaptive'")
    for ts in E_lists.get('tspans') or []:
        if ts is not None and not (len(ts) == 2 and float(ts[1]) > float(ts[0])):
            raise ValueError(f'tspan {list(ts)}: give [t0, t1] with t1 > t0')
    return E


def listed_rows(mdl, e, first, I, base):
    """Member e's neighbour lists [N - I, m] for the sweep of iteration len(first) - 1, as global store rows (base = e
    cap): CudaNNGPAlt.neighbour_table, the rules of the member's solo run; a refusal names the member."""
    try:
        return mdl.neighbour_table(first, I) + base
    except Exception as exc:
        raise ValueError(f'member {e}: {exc}') from exc


def sweep_tables(m_members, sw):
    """Per-position neighbour counts of a sweep over the members sw (state order)."""
    return np.asarray(m_members, dtype=np.int32)[np.asarray(sw, dtype=np.int64)]


def launch_sweep(h, t_dev, sysid, mG, hm, steps, N, sw, I_sw, m_pos, listed_sw, lists, mdl0, starts, u_next, uG_next, n,
                 stream):
    """The sweep over the members sw (state order).  t_dev: the members' grids [E, N+1], uploaded once per run; the
    swept members' rows are selected on the device.  listed_sw: which of them take the neighbour lists `lists`."""
    import torch
    rows = torch.from_numpy(np.asarray(sw, dtype=np.int64)).to(t_dev.device)
    if not np.any(listed_sw):
        listed_sw = lists = None
    h.ensemble_sweep(sysid, mG, hm, steps, t_dev.index_select(0, rows), N, sw, I_sw, m_pos, mdl0.n_restarts, starts,
                     mdl0.fatol, mdl0.xatol, u_next, uG_next, n, listed_sw, lists, stream)


def member_order(I, done):
    """Members in state order for the next iteration: running ones first, by ascending I (stable)."""
    I = np.asarray(I)
    return np.lexsort((np.arange(I.size), I, np.asarray(done, dtype=bool)))


def fine_rows(I_pos, N):
    """(flat state row, slice) of every fine solve of the runs at positions 0..len(I_pos)-1: slices I_p..N-1 of each"""
    rows, sl = [], []
    for p, I in enumerate(I_pos):
        s = np.arange(I, N)
        rows.append(p * (N + 1) + s)
        sl.append(s)
    if not rows:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(rows).astype(np.int64), np.concatenate(sl).astype(np.int64)


def pack_starts(blocks, I_pos, N):
    """The starts of the sweep in the order nngp_ensemble_sweep reads them: slice-major, and within slice i the blocks of
    the positions with I_p <= i in position order.  blocks[p] = [N - I_p, d, 9, R, 2], the run's solo draw for this
    sweep (its block j belongs to slice I_p + j).  I_pos ascending."""
    out = []
    for i in range(min(I_pos), N):
        for p, I in enumerate(I_pos):
            if I > i:
                break
            out.append(blocks[p][i - I])
    return np.ascontiguousarray(np.stack(out))


class PararealEnsemble:
    """E independent device-resident nnGParareal runs in lockstep (see the module docstring).

    The ensemble owns its own library handle, so its segmented dataset never meets the dataset of a solo run on the
    default handle.  Per-member timings are the ensemble's shared wall times: F_time, G_time and sweep_time of every
    member are the times of the launches that served all members together.
    """

    def __init__(self, ode, solver, tspan, N, epsilon=5e-7, verbose='v', device=None):
        if not isinstance(ode, ODE):
            raise Exception('ode must be an instance of the ODE class, see systems.py file.')
        if not isinstance(solver, CudaSolverRK):
            raise Exception('PararealEnsemble needs a CudaSolverRK')
        self.ode, self.solver, self.tspan, self.N = ode, solver, tspan, N
        self.epsilon = epsilon
        self.verbose = verbose
        self.n = ode.get_dim()
        self.u0 = ode.get_init_cond()
        self._device = device
        self._h = None

    def handle(self):
        if self._h is None:
            import os
            dev = self._device if self._device is not None else int(os.environ.get("LOCAL_RANK", "0"))
            self._h = _lib.Handle(dev)
        return self._h

    def run(self, model='nngp', seeds=None, nn='adaptive', n_restarts=1, fatol=None, xatol=None, epsilons=None,
            early_stops=None, init_conds=None, tspans=None, max_rows=None, store_int=False, nntype='nn'):
        """Returns one output dict per seed (the keys of PararealDevice.run, n_rows included).

        nn: 'adaptive', an int in 1..160, or a list with one of those per member.  nntype: the neighbour rule of
        models_alt.py ('nn', 'col+rnd', 'col_only', 'row_col', 'row', 'col_full') or a list with one per member; a
        position-based member equals PararealDevice(...).run(model='nngp', nntype=..., seed=...).  tspans: None or a
        list with one [t0, t1] (or None: the ensemble's tspan) per member; member e's output 't' is its own grid.
        n_restarts, fatol and xatol are common to all members."""
        E = check_run_args(dict(seeds=seeds, epsilons=epsilons, early_stops=early_stops, init_conds=init_conds,
                                tspans=tspans), model=model, store_int=store_int, nn=nn, nntype=nntype)
        solver = self.solver
        if max(solver.Nf, solver.Ng) > solver.thresh:
            raise Exception('steps > thresh (RK paging, solver.py:89-96) is only supported by the host driver')
        eps = [self.epsilon if epsilons is None or epsilons[e] is None else epsilons[e] for e in range(E)]
        stops = [None if early_stops is None else early_stops[e] for e in range(E)]
        u0s = np.stack([self.u0 if init_conds is None or init_conds[e] is None else self.ode.get_init_cond(u0=init_conds[e])
                        for e in range(E)])
        nns = list(nn) if isinstance(nn, (list, tuple, np.ndarray)) else [nn] * E
        spans = [self.tspan if tspans is None or tspans[e] is None else tspans[e] for e in range(E)]
        t_members = np.stack([np.linspace(ts[0], ts[1], num=self.N + 1) for ts in spans])
        rules = list(nntype) if isinstance(nntype, (list, tuple, np.ndarray)) else [nntype] * E
        h = self.handle()
        models = []
        for s, v, rule in zip(seeds, nns, rules):
            kw = dict(n=self.n, N=self.N, seed=s, nn=v if v == 'adaptive' else int(v), n_restarts=n_restarts,
                      fatol=fatol, xatol=xatol, handle=h)
            models.append(CudaNNGP(**kw) if rule == 'nn' else CudaNNGPAlt(nntype=rule, **kw))
        return self._run(h, models, eps, stops, u0s, max_rows, t_members)

    def _run(self, h, models, eps, stops, u0s, max_rows, t_members):
        import torch
        N, n, solver = self.N, self.n, self.solver
        E = len(models)
        verbose = self.verbose
        _, sysid = self.ode.device_system(h)
        dev = torch.device('cuda', h.device)
        stream = torch.cuda.current_stream(dev).cuda_stream
        mF, mG, hm = _lib.METHODS[solver.F], _lib.METHODS[solver.G], solver.h_mode
        f64 = dict(dtype=torch.float64, device=dev)
        ld = (N + 1) * n
        tic = time.time()
        t_dev = torch.from_numpy(t_members).to(dev)  # [E, N+1], member order
        t_rep = t_dev.t().contiguous().view(-1)  # t_rep[i E + p] = t_p[i]
        st = {key: torch.zeros((E, N + 1, n), **f64) for key in ('u_cur', 'uG_cur', 'uF')}
        for a in st.values():
            a[:, 0] = torch.from_numpy(u0s).to(dev)
        for i in range(N):  # coarse initialisation: N dependent launches over all members
            h.rk_batch(sysid, mG, hm, solver.Ng, E, t_rep[i * E:], t_rep[(i + 1) * E:], st['uG_cur'][:, i], ld,
                       st['uG_cur'][:, i + 1], ld, stream)
        st['u_cur'].copy_(st['uG_cur'])
        st['u_next'] = st['u_cur'].clone()
        st['uG_next'] = st['uG_cur'].clone()
        scratch = torch.empty_like(st['u_cur'])
        err_dev = torch.zeros(E * (N + 1), **f64)
        cap = max_rows or min(N * (N + 3) // 2 + 1, N * 16)
        h.seg_reset()
        h.seg_reserve(E, cap, n)
        cap = h.seg_cap()
        torch.cuda.synchronize(dev)
        G_time = time.time() - tic
        F_time = sweep_time = 0.0

        I = np.zeros(E, dtype=np.int64)
        done = np.zeros(E, dtype=bool)
        rows = np.zeros(E, dtype=np.int64)
        last_k = np.zeros(E, dtype=np.int64)
        conv_int = [[] for _ in range(E)]
        first = [[] for _ in range(E)]  # first unconverged slice of every iteration a member appended (listed rules)
        listed = np.array([getattr(mdl, 'nntype', 'nn') != 'nn' for mdl in models])
        err = [np.full((N + 1, N), np.nan) for _ in range(E)]
        pos = np.arange(E)  # pos[p] = member at state position p
        for k in range(N):
            # state order: running members first, by ascending I
            order = member_order(I[pos], done[pos])
            if not np.array_equal(order, np.arange(E)):
                perm = torch.from_numpy(order.astype(np.int64)).to(dev)
                for key in ('u_cur', 'uG_cur', 'uF', 'u_next', 'uG_next'):
                    h.copy_rows(st[key], perm, scratch, None, E, ld, stream)
                    st[key], scratch = scratch, st[key]
                pos = pos[order]
            n_live = int(np.count_nonzero(~done[pos]))
            if n_live == 0:
                break
            live = pos[:n_live]
            if verbose == 'v':
                print(f'{self.ode.name} ensemble of {E} iteration number (out of {N}): {k+1}, {n_live} running')
            tic = time.time()
            # fine solves of every running member's unconverged slices in one launch (parareal.py:309-334)
            fr, fs = fine_rows(I[live], N)
            idx = torch.from_numpy(np.concatenate([fr, fr + 1, np.arange(n_live) * (N + 1) + I[live] + 1])).to(dev)
            fm = np.repeat(live, N - I[live])  # member of every fine solve
            tt = torch.from_numpy(np.concatenate([t_members[fm, fs], t_members[fm, fs + 1]])).to(dev)
            nf = fr.size
            buf = torch.empty((2, nf, n), **f64)
            h.copy_rows(st['u_cur'], idx[:nf], buf[0], None, nf, n, stream)
            h.rk_batch(sysid, mF, hm, solver.Nf, nf, tt[:nf], tt[nf:], buf[0], n, buf[1], n, stream)
            h.copy_rows(buf[1], None, st['uF'], idx[nf:2 * nf], nf, n, stream)
            exact = idx[2 * nf:]
            h.copy_rows(st['uF'], exact, st['u_next'], exact, n_live, n, stream)
            h.copy_rows(st['uG_cur'], exact, st['uG_next'], exact, n_live, n, stream)
            torch.cuda.synchronize(dev)
            F_time += time.time() - tic
            I[live] += 1
            tic = time.time()
            # dataset append of every running member, before the early-stop check as in PararealDevice.device_sweep
            need = rows[live] + (N - I[live] + 1)
            if need.max() > cap:
                while need.max() > cap:
                    cap = 2 * cap + N
                h.seg_reserve(E, cap, n)
            h.seg_append_iteration(live, I[live], st['u_cur'], st['uF'], st['uG_cur'], ld, N, n, stream)
            rows[live] = need
            for e in live:
                first[e].append(int(I[e]) - 1)
            n_sweep = int(np.count_nonzero(I[live] < N))  # the members with I == N sort last among the running ones
            if n_sweep > 0:
                sw = live[:n_sweep]
                mdl0 = models[sw[0]]
                lists = [listed_rows(models[e], e, first[e], I[e], e * cap) if listed[e] else None for e in sw]
                m_members = [mdl.neighbours(k) for mdl in models]
                for e, tab in zip(sw, lists):
                    if tab is not None:
                        m_members[e] = tab.shape[1]
                m_pos = sweep_tables(m_members, sw)
                if m_pos.max() > MAX_NEIGHBOURS:
                    raise Exception('nn > 160 neighbours is not supported (include/nngpara.h: NNGP_MAX_NEIGHBOURS_BIG)')
                blocks = []
                for e in sw:
                    mdl = models[e]
                    mdl.k = mdl.time_k = k
                    blocks.append(mdl.draw_starts(N - I[e]))
                    mdl.train_count += (N - I[e]) * n * N_JITTER * mdl.n_restarts
                starts = torch.from_numpy(pack_starts(blocks, I[sw], N)).to(dev)
                launch_sweep(h, t_dev, sysid, mG, hm, solver.Ng, N, sw, I[sw], m_pos, listed[sw], lists, mdl0, starts,
                             st['u_next'], st['uG_next'], n, stream)
            # parareal.py:402: one error launch over the running members and ONE device->host read
            h.rowwise_maxabs_diff(st['u_next'], st['u_cur'], n_live * (N + 1), n, err_dev, stream)
            errs = err_dev[:n_live * (N + 1)].cpu().numpy().reshape(n_live, N + 1)
            dt_sweep = time.time() - tic
            sweep_time += dt_sweep
            for p, e in enumerate(live):
                err[e][:, k] = errs[p]
                last_k[e] = k
                if I[e] == N:  # early stopping (parareal.py:341-347)
                    err[e][-1, k] = np.nextafter(eps[e], 0)
                    done[e] = True
                    continue
                mdl = models[e]
                mdl.pred_time += dt_sweep
                mdl.pred_times[k] += dt_sweep
                mdl.tot_train_t += dt_sweep
                if np.any(np.isnan(err[e][:, k])) and bool(torch.isnan(st['uG_next'][p]).any()):
                    raise Exception("NaN values in initial coarse solve - increase Ng!")
                I[e] = advance(err[e][:, k], I[e], eps[e])
                conv_int[e].append(int(I[e]))
                if I[e] == N or (stops[e] is not None and k == stops[e] - 1):
                    done[e] = True
            st['u_cur'].copy_(st['u_next'])
            st['uG_cur'].copy_(st['uG_next'])
        u_all = st['u_cur'].cpu().numpy()
        where = np.empty(E, dtype=np.int64)
        where[pos] = np.arange(E)
        outs = []
        for e in range(E):
            timings = {'F_time': F_time, 'G_time': G_time, 'F_time_serial_avg': F_time / max(N, 1),
                       'sweep_time': sweep_time}
            timings.update(models[e].get_times())
            u = u_all[where[e]].copy()
            kk = int(last_k[e])
            outs.append({'t': t_members[e], 'u': u, 'u_last': u, 'err': err[e][:, :kk + 1], 'k': kk + 1, 'timings': timings,
                         'debug_dict': {}, 'converged': bool(I[e] == N), 'conv_int': conv_int[e],
                         'n_rows': int(h.seg_rows(e))})
        return outs
