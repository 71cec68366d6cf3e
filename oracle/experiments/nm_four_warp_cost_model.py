"""TEST INFRASTRUCTURE / STUDY ONLY.  Cost model of one search per warp (serial evaluations) against four warps
per search (candidate points of an iteration evaluated side by side) on a replayed FHN d=512 predict: finite
evaluation 3 300 cycles, failing evaluation 800, CTA barrier 150.  Strategies: A = {reflection, expansion, outside,
inside contraction}; B = {reflection, inside contraction, both shrunk vertices}; C = B after an iteration that
contracted inside or shrank (or when every vertex is +inf), else A  (= csrc/gpfit.cu gp_fit_spec_kernel);
S6 = all six points an iteration can ask for (six warps per search: every iteration is one round).
Result (profiles/r02/nm_moves.log): longest search 695 -> 336 us for 1.8x the evaluations (strategy C).
usage: python oracle/experiments/nm_four_warp_cost_model.py [predict id = 3] [dimension stride = 8]"""
import os, sys, collections, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import nngp as onn
z = np.load(os.path.join(ROOT, 'tests', 'golden', 'run_fhn_d512_replay_k2.npz'))
CF, CI, SYNC = 3300.0, 800.0, 150.0
cost = lambda f: CI if not np.isfinite(f) else CF

def run(func, x0, strategy, xatol=0.1, fatol=0.1):
    """returns serial cycles, quad cycles, nfev"""
    maxfun = 400
    calls = [0]; serial = [0.0]
    class B(Exception): pass
    cache = {}
    def f(x):
        if calls[0] >= maxfun: raise B()
        calls[0] += 1
        v = float(func(np.copy(x))); serial[0] += cost(v); cache[tuple(x)] = v
        return v
    def peek(x):  # speculative evaluation (not counted by SciPy)
        return float(func(np.copy(x)))
    quad = 0.0
    sim = np.empty((3, 2)); sim[0] = x0
    for k in range(2):
        y = np.array(x0, float); y[k] = 1.05 * y[k] if y[k] != 0 else 0.00025; sim[k + 1] = y
    fsim = np.full(3, np.inf)
    for k in range(3): fsim[k] = f(sim[k])
    quad += max(cost(v) for v in fsim) + SYNC
    o = np.argsort(fsim, kind='stable'); sim, fsim = sim[o], fsim[o]
    it = 1; last = 'E'
    while calls[0] < maxfun and it < 400:
        try:
            if np.max(np.abs(sim[1:] - sim[0])) <= xatol and np.max(np.abs(fsim[0] - fsim[1:])) <= fatol: break
            xbar = (sim[0] + sim[1]) / 2; worst = sim[2].copy()
            pts = {'xr': 2 * xbar - worst, 'xe': 3 * xbar - 2 * worst, 'xoc': 1.5 * xbar - 0.5 * worst,
                   'xic': 0.5 * xbar + 0.5 * worst, 's1': sim[0] + 0.5 * (sim[1] - sim[0]), 's2': sim[0] + 0.5 * (sim[2] - sim[0])}
            if strategy == 'S6': cand = ['xr', 'xe', 'xoc', 'xic', 's1', 's2']
            elif strategy == 'A': cand = ['xr', 'xe', 'xoc', 'xic']
            elif strategy == 'B': cand = ['xr', 'xic', 's1', 's2']
            else: cand = ['xr', 'xic', 's1', 's2'] if (last in ('IC', 'ICS', 'OCS', 'INF') or np.isinf(fsim[0])) else ['xr', 'xe', 'xoc', 'xic']
            used = []
            xr = pts['xr']; fxr = f(xr); used.append('xr'); shrink = False
            if fxr < fsim[0]:
                fxe = f(pts['xe']); used.append('xe')
                if fxe < fxr: sim[2], fsim[2] = pts['xe'], fxe; mv = 'E'
                else: sim[2], fsim[2] = xr, fxr; mv = 'E'
            elif fxr < fsim[1]: sim[2], fsim[2] = xr, fxr; mv = 'R'
            elif fxr < fsim[2]:
                fxc = f(pts['xoc']); used.append('xoc')
                if fxc <= fxr: sim[2], fsim[2] = pts['xoc'], fxc; mv = 'OC'
                else: shrink = True; mv = 'OCS'
            else:
                fxcc = f(pts['xic']); used.append('xic')
                if fxcc < fsim[2]: sim[2], fsim[2] = pts['xic'], fxcc; mv = 'IC'
                else: shrink = True; mv = 'ICS'
            if shrink:
                for j in (1, 2):
                    sim[j] = sim[0] + 0.5 * (sim[j] - sim[0]); fsim[j] = f(sim[j]); used.append(f's{j}')
            # quad cost: round 1 evaluates cand; points used but not in cand need another round (together)
            r1 = max(cost(cache.get(tuple(pts[c]), None) if tuple(pts[c]) in cache else peek(pts[c])) for c in cand)
            quad += r1 + SYNC
            miss = [u for u in used if u not in cand]
            if miss: quad += max(cost(cache[tuple(pts[u])]) for u in miss) + SYNC
            last = mv; it += 1
        except B:
            quad += CF + SYNC
        o = np.argsort(fsim, kind='stable'); sim, fsim = sim[o], fsim[o]
    return serial[0], quad, calls[0]

pid = int(sys.argv[1]) if len(sys.argv) > 1 else 3
step = int(sys.argv[2]) if len(sys.argv) > 2 else 8
xm, ym, starts = z[f'p{pid}_xm'], z[f'p{pid}_ym'], z[f'p{pid}_starts']
r2 = onn.pairwise_sqdist(xm, xm)
import warnings; warnings.filterwarnings('ignore')
for strat in (sys.argv[3].split(',') if len(sys.argv) > 3 else ('A', 'B', 'C')):
    S, Q, NF = [], [], []
    for j in range(0, 512, step):
        for a in range(9):
            f = lambda th: onn.neg_log_lik(r2, ym[:, j], th, onn.JITTERS[a])
            s, q, n = run(f, starts[j, a, 0].astype(float), strat)
            S.append(s); Q.append(q); NF.append(n)
    S, Q = np.array(S), np.array(Q)
    print(f'p{pid} strategy {strat}: serial max {S.max()/1.9e3:.0f} us mean {S.mean()/1.9e3:.0f} us | quad max {Q.max()/1.9e3:.0f} us mean {Q.mean()/1.9e3:.0f} us | sum ratio warps*rounds/serial {(6 if strat == 'S6' else 4)*Q.sum()/S.sum():.2f}', flush=True)
