"""TEST INFRASTRUCTURE / STUDY ONLY.  Which moves do the Nelder-Mead searches of a steady-state predict make?
Traces SciPy's algorithm (oracle restatement) with the oracle objective on a replayed FHN d=512 predict
(tests/golden/run_fhn_d512_replay_k2.npz) and prints move counts for all searches and for the long finite ones.
Result (profiles/r02/nm_moves.log): the long searches are runs of inside contraction + shrink (4 evaluations per
iteration, all four points known when the iteration starts) -- the basis of the four-warp search kernel.
usage: python oracle/experiments/nm_move_study.py [predict id = 3] [dimension stride = 8]"""
import os, sys, collections, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import nngp as onn
z = np.load(os.path.join(ROOT, 'tests', 'golden', 'run_fhn_d512_replay_k2.npz'))

def trace(func, x0, xatol=0.1, fatol=0.1):
    n = 2; maxfun = 400
    calls = [0]
    class B(Exception): pass
    def f(x):
        if calls[0] >= maxfun: raise B()
        calls[0] += 1
        return float(func(np.copy(x)))
    sim = np.empty((3, 2)); sim[0] = x0
    for k in range(2):
        y = np.array(x0, float); y[k] = 1.05 * y[k] if y[k] != 0 else 0.00025; sim[k + 1] = y
    fsim = np.full(3, np.inf)
    for k in range(3): fsim[k] = f(sim[k])
    o = np.argsort(fsim, kind='stable'); sim, fsim = sim[o], fsim[o]
    it = 1; moves = []
    while calls[0] < maxfun and it < 400:
        try:
            if np.max(np.abs(sim[1:] - sim[0])) <= xatol and np.max(np.abs(fsim[0] - fsim[1:])) <= fatol: break
            allinf = np.isinf(fsim[0])
            xbar = (sim[0] + sim[1]) / 2; worst = sim[2]
            xr = 2 * xbar - worst; fxr = f(xr); shrink = False
            if fxr < fsim[0]:
                fxe = f(3 * xbar - 2 * worst)
                if fxe < fxr: sim[2], fsim[2] = 3 * xbar - 2 * worst, fxe; mv = 'E+'
                else: sim[2], fsim[2] = xr, fxr; mv = 'E-'
            elif fxr < fsim[1]: sim[2], fsim[2] = xr, fxr; mv = 'R'
            elif fxr < fsim[2]:
                xc = 1.5 * xbar - 0.5 * worst; fxc = f(xc)
                if fxc <= fxr: sim[2], fsim[2] = xc, fxc; mv = 'OC'
                else: shrink = True; mv = 'OCS'
            else:
                xcc = 0.5 * xbar + 0.5 * worst; fxcc = f(xcc)
                if fxcc < fsim[2]: sim[2], fsim[2] = xcc, fxcc; mv = 'IC'
                else: shrink = True; mv = 'ICS'
            if shrink:
                for j in (1, 2):
                    sim[j] = sim[0] + 0.5 * (sim[j] - sim[0]); fsim[j] = f(sim[j])
            if allinf: mv = 'INF'
            moves.append(mv); it += 1
        except B:
            moves.append('ABORT')
        o = np.argsort(fsim, kind='stable'); sim, fsim = sim[o], fsim[o]
    return calls[0], moves

pid = int(sys.argv[1]) if len(sys.argv) > 1 else 3
step = int(sys.argv[2]) if len(sys.argv) > 2 else 8
xm, ym, starts = z[f'p{pid}_xm'], z[f'p{pid}_ym'], z[f'p{pid}_starts']
r2 = onn.pairwise_sqdist(xm, xm)
allm = []
for j in range(0, 512, step):
    for a in range(9):
        f = lambda th: onn.neg_log_lik(r2, ym[:, j], th, onn.JITTERS[a])
        nf, mv = trace(f, starts[j, a, 0].astype(float))
        allm.append((nf, mv))
nf = np.array([a[0] for a in allm])
print('searches', len(allm), 'nfev mean', nf.mean(), 'max', nf.max(), 'pctl 90/99', np.percentile(nf, [90, 99]))
tot = collections.Counter(); 
for n_, mv in allm: tot.update(mv)
print('all moves', dict(tot))
long = [a for a in allm if a[0] >= 150 and 'INF' not in a[1][:5]]
print('long finite searches', len(long))
tl = collections.Counter()
for n_, mv in long: tl.update(mv)
print('moves of long finite searches', dict(tl))
for n_, mv in sorted(long, key=lambda a: -a[0])[:6]:
    print(n_, ' '.join(mv[:80]))
