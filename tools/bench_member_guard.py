"""cost and effect of the per-member blow-up guard

1. Headline workload of bench.py (cylinder_4, 64 members, Re 60..150, CNAB,
   dt = 1/2048, tol 1e-12, 16 spin-up steps), guard checks on (maxv 1e8, 10
   slices): the stop-all guard against the per-member guard with no member
   retired, alternated on one trajectory, `--reps` repetitions of `--steps`
   steps each.  Both arms launch the same kernels, so the difference is noise.
2. The same ensemble at dt = 1/512 (the Robin-control script's step size),
   maxv 1e8, 120 steps in member mode.  With 10 slices: which members retire
   and at which level, and which blow up after the last check.  With a check
   before every step: the same, device ms/step and FGMRES iterations/step of a run up to the
   first retirement and of a run after it (retired lanes masked); the relative
   v / p error of the lowest-Re and highest-Re surviving members against the
   oracle's CNAB from the same initial state after the 120 steps.

Device ms/step from `dnsb_imex_last_run_ms` (CUDA events).  Prints one JSON
line with the card name and power limit read in the same call.

usage: python tools/bench_member_guard.py [--steps 128] [--reps 7] [--json FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit',
                            '--format=csv,noheader'], capture_output=True, text=True,
                           timeout=30).stdout.strip()
        name, plim = [s.strip() for s in q.split(',')]
        return name, plim
    except Exception:                                     # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), 'unknown'


def _spread(v):
    v = np.asarray(v)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))


def headline(args, ctx):
    from bench import ensemble_initial_state
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, K = args.members, args.steps
    ntimes = args.spinup + (2*args.reps + 2)*K + 8
    integ, info = ens.cylinder_ensemble(N=args.mesh, nmembers=nb, dt=1./2048,
                                        ntimes=ntimes, ctx=ctx)
    runkw = dict(tol=args.tol, guess=args.guess, ntimeslices=10, check_ff_maxv=1e8, maxit=400)
    v0, p0 = ensemble_initial_state(info, nb)
    integ.set_state(v0, p0)
    integ.run(args.spinup, **runkw)
    ms = {False: [], True: []}
    for r in range(args.reps + 1):                        # the first pair warms both arms
        for mg in (False, True):
            integ.set_member_guard(mg)
            ff = integ.run(K, **runkw)
            assert ff == 0 and integ.member_status()['alive'].all()
            if r > 0:
                ms[mg].append(integ.engine.last_run_ms()/K)
    integ.close()
    return dict(dt=1./2048, steps_per_rep=K, reps=args.reps,
                stop_all_ms_per_step=_spread(ms[False]), member_ms_per_step=_spread(ms[True]))


def unstable(args, ctx):
    from bench import ensemble_initial_state, _cpu_parity_worker
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, nsteps, dt = args.members, 120, 1./512
    after = args.steps
    integ, info = ens.cylinder_ensemble(N=args.mesh, nmembers=nb, dt=dt, ctx=ctx,
                                        ntimes=nsteps + after + 8, member_guard=True)
    runkw = dict(tol=args.tol, guess=args.guess, ntimeslices=10, check_ff_maxv=1e8, maxit=400)
    v0, p0 = ensemble_initial_state(info, nb)
    # (a) 10 slices: a member that blows up after the last check is live at the end with a non-finite
    # state, and the run reports that as not converged
    integ.set_state(v0, p0)
    ff = integ.run(nsteps, allow_unconverged=True, **runkw)
    st = integ.member_status()
    v, _ = integ.state()
    s = integ.stats()
    res = dict(dt=dt, steps=nsteps, slices10=dict(
        ffflag=ff, retired={int(m): int(st['trip_level'][m]) for m in np.flatnonzero(~st['alive'])},
        live_non_finite=[int(m) for m in np.flatnonzero(st['alive'] & ~np.isfinite(v).all(axis=0))],
        max_relres_live=s['max_relres']))
    # (b) a check before every step: nothing blows up unseen
    runkw['ntimeslices'] = nsteps - 1
    integ.set_state(v0, p0)
    ff = integ.run(nsteps, **runkw)
    st = integ.member_status()
    full_ms = integ.engine.last_run_ms()/nsteps
    v, p = integ.state()
    live = np.flatnonzero(st['alive'])
    retired = np.flatnonzero(~st['alive'])
    res['every_step'] = dict(ffflag=ff, ms_per_step_120=full_ms,
                             retired={int(m): int(st['trip_level'][m]) for m in retired})
    # ms/step after the retirements: the same integrator continues with the retired lanes masked
    # (no guard checks in this run and the next, so that both time the step alone)
    runkw['ntimeslices'] = 0
    integ.run(after, allow_unconverged=True, **runkw)
    s = integ.stats()
    res['every_step']['after'] = dict(steps=after, ms_per_step=integ.engine.last_run_ms()/after,
                                      iters_per_step=s['iters']/max(s['solves'], 1),
                                      max_relres_live=s['max_relres'])
    # ms/step before the first retirement: a fresh run from the initial state up to that level
    if retired.size:
        t1 = int(st['trip_level'][retired].min())
        integ.set_state(v0, p0)
        integ.run(t1, **runkw)
        s = integ.stats()
        res['every_step']['before'] = dict(steps=t1, ms_per_step=integ.engine.last_run_ms()/t1,
                                           iters_per_step=s['iters']/max(s['solves'], 1),
                                           note='includes the Heun start-up step')
    integ.close()
    errs = []
    for m in (live[0], live[-1]):
        ov, op = _cpu_parity_worker((args.mesh, float(info['nus'][m]), dt, nsteps, 1e-5,
                                     v0[:, m], p0[:, m]))
        errs.append(dict(member=int(m), Re=float(info['Re'][m]),
                         v_rel=float(np.linalg.norm(v[:, m] - ov.ravel())/np.linalg.norm(ov)),
                         p_rel=float(np.linalg.norm(p[:, m] - op.ravel())/np.linalg.norm(op))))
    res['every_step']['live_vs_oracle'] = errs
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--members', type=int, default=64)
    ap.add_argument('--mesh', type=int, default=4)
    ap.add_argument('--tol', type=float, default=1e-12)
    ap.add_argument('--guess', type=int, default=24)
    ap.add_argument('--spinup', type=int, default=16)
    ap.add_argument('--steps', type=int, default=128)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--json', metavar='FILE')
    args = ap.parse_args()
    from dolfin_navier_scipy_b200 import _lib
    ctx = _lib.default_context(0)
    name, plim = card()
    res = dict(tool='bench_member_guard', gpu=name, power_limit=plim, mesh=args.mesh,
               members=args.members, tol=args.tol, guess=args.guess,
               headline=headline(args, ctx), unstable=unstable(args, ctx))
    line = json.dumps(res)
    print(line)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
