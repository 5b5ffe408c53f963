"""cost of the field statistics accumulated inside the device loop

Headline workload of bench.py (cylinder_4, 64 members, Re 60..150, CNAB,
dt = 1/2048, tol 1e-12, 16 spin-up steps), two arms alternated on one
trajectory and repeated so that the spread shows:

  off  no statistics
  on   means and second moments of every member at every level
       (`DeviceImex.set_statistics`), read once at the end of the run

Per arm: device ms/step (`dnsb_imex_last_run_ms`, median / min / max over the
repetitions).  Then, in a run of its own, the mean time of `k_imex_stats` from
the library's CUDA-event profile, its algorithmic bytes per level
(8 nb (nvf + nv + np) read + 2 * 8 nb (5 nnodes + 2 np + nv) read and
written) and their rate as a fraction of the HBM peak of the data sheet
(7.7 TB/s).  Prints one JSON line (card name and power limit included).

usage: python tools/bench_statistics.py [--steps 128] [--reps 7] [--json FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

HBM_PEAK = 7.7e12


def stats_bytes(nb, nnodes, nv, np_):
    """algorithmic bytes of one k_imex_stats level"""
    return 8*nb*(2*nnodes + nv + np_) + 2*8*nb*(5*nnodes + 2*np_ + nv)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--members', type=int, default=64)
    ap.add_argument('--mesh', type=int, default=4)
    ap.add_argument('--nts', type=int, default=2048)
    ap.add_argument('--tol', type=float, default=1e-12)
    ap.add_argument('--guess', type=int, default=24)
    ap.add_argument('--spinup', type=int, default=16)
    ap.add_argument('--steps', type=int, default=128)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--json', metavar='FILE')
    args = ap.parse_args()
    from bench import ensemble_initial_state
    from bench_outputs import card
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import ensemble as ens

    ctx = _lib.default_context(0)
    nb, K = args.members, args.steps
    ntimes = args.spinup + (2*args.reps + 3)*K + 8
    integ, info = ens.cylinder_ensemble(N=args.mesh, nmembers=nb, dt=1./args.nts,
                                        ntimes=ntimes, ctx=ctx)
    NV, NP = info['NV'], info['NP']
    nnodes = integ.dev.nvf//2
    v0, p0 = ensemble_initial_state(info, nb)
    runkw = dict(tol=args.tol, guess=args.guess, ntimeslices=0, maxit=400)
    integ.set_state(v0, p0)
    integ.run(args.spinup, **runkw)

    def arm(which):
        integ.set_statistics(which == 'on')
        integ.run(K, **runkw)
        ok = True
        if which == 'on':
            st = integ.statistics()
            ok = bool((st['count'] == K + 1).all() and np.isfinite(st['v_mean']).all()
                      and np.isfinite(st['c_mean']).all())
        return dict(dev_ms=integ.engine.last_run_ms()/K, ok=ok)

    for which in ('off', 'on'):                           # warm both paths
        arm(which)
    reps = {w: [] for w in ('off', 'on')}
    for r in range(args.reps):
        for which in ('off', 'on'):
            reps[which].append(arm(which))
    # the kernel's device time, in a run of its own (profiling serialises the launches)
    integ.set_statistics(True)
    ctx.profile_begin()
    integ.run(K, **runkw)
    prof = ctx.profile_end()
    names = [k for k in prof if k.startswith('k_imex_stats')]
    cnt = sum(prof[k][0] for k in names)
    ms = sum(prof[k][1] for k in names)
    step_ms = sum(t for _, t in prof.values())/K
    integ.close()
    name, plim = card()
    nbytes = stats_bytes(nb, nnodes, NV, NP)
    mean_s = ms*1e-3/cnt
    res = dict(tool='bench_statistics', gpu=name, power_limit=plim, mesh=args.mesh,
               members=nb, dt=1./args.nts, tol=args.tol, steps_per_rep=K, reps=args.reps,
               kernel=dict(names=names, launches=cnt, mean_us=mean_s*1e6, bytes=nbytes,
                           tb_per_s=nbytes/mean_s/1e12, hbm_fraction=nbytes/mean_s/HBM_PEAK,
                           share_of_profiled_step=ms/K/step_ms))
    for which, rs in reps.items():
        v = np.array([x['dev_ms'] for x in rs])
        res['arm_' + which] = dict(dev_ms=dict(median=float(np.median(v)), min=float(v.min()),
                                               max=float(v.max())),
                                   ok=all(x['ok'] for x in rs))
    line = json.dumps(res)
    print(line)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
