"""cost of the output functionals recorded inside the device loop

Headline workload of bench.py (cylinder_4, 64 members, Re 60..150, CNAB,
dt = 1/2048, tol 1e-12, 16 spin-up steps), three arms alternated on one
trajectory and repeated so that the spread shows:

  a  nothing recorded
  b  drag + lift + 16 velocity probes + the pressure difference across the
     cylinder at every step (`DeviceImex.set_outputs`), read once at the end
  c  the full state of every member at every step through the pinned snapshot
     mirror, the way to get the same numbers without (b)

Per arm: device ms/step (`dnsb_imex_last_run_ms`), end-to-end ms/step with the
final read of what was recorded, bytes moved to the host per step; then, in a
run of its own, the mean time of the output kernel from the library's
CUDA-event profile.  Prints one JSON line (card name and power limit included).

usage: python tools/bench_outputs.py [--steps 128] [--reps 7] [--json FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def probes(femp, NV, NP):
    """16 velocity dofs in the wake and p(front) - p(back) of the cylinder"""
    V = femp['V']
    xy = np.asarray(V.tabulate_dof_coordinates())[np.asarray(femp['invinds'])]
    cand = np.flatnonzero((xy[:, 0] > 0.3) & (xy[:, 0] < 1.5) &
                          (np.abs(xy[:, 1] - 0.2) < 0.1))
    pick = cand[np.linspace(0, cand.size - 1, 16).astype(int)]
    Cv = sps.csr_matrix((np.ones(16), (np.arange(16), pick)), shape=(17, NV))
    pxy = np.asarray(V.mesh().coords)
    front = np.argmin(np.hypot(pxy[:, 0] - 0.15, pxy[:, 1] - 0.2))
    back = np.argmin(np.hypot(pxy[:, 0] - 0.25, pxy[:, 1] - 0.2))
    Cp = sps.csr_matrix(([1., -1.], ([16, 16], [front, back])), shape=(17, NP))
    return Cv, Cp


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
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import ensemble as ens

    ctx = _lib.default_context(0)
    nb, K = args.members, args.steps
    ntimes = args.spinup + (3*args.reps + 2)*K + 8
    integ, info = ens.cylinder_ensemble(N=args.mesh, nmembers=nb, dt=1./args.nts,
                                        ntimes=ntimes, ctx=ctx)
    sm, femp = info['sm'], info['femp']
    NV, NP = info['NV'], info['NP']
    Cv, Cp = probes(femp, NV, NP)
    ny = Cv.shape[0]
    ops = dict(M=sm['Mfull'], A=sm['Afull'], JT=sm['JTfull'])
    v0, p0 = ensemble_initial_state(info, nb)
    runkw = dict(tol=args.tol, guess=args.guess, ntimeslices=0, maxit=400)
    integ.set_state(v0, p0)
    integ.run(args.spinup, **runkw)
    integ.reserve_snapshots(K + 2)

    def arm(which):
        if which == 'b':
            integ.set_outputs(Cv, Cp, force_dofs=femp['ldsbcinds'], force_ops=ops)
        else:
            integ.set_outputs()
        integ.engine.reset_snapshots()
        ctx.sync()
        t0 = time.perf_counter()
        integ.run(K, snap_stride=1 if which == 'c' else 0, **runkw)
        if which == 'b':
            out = integ.outputs()
            nbytes = out['y'].nbytes + out['force'].nbytes
            ok = bool(np.isfinite(out['force'][2:]).all() and np.isfinite(out['y']).all())
        elif which == 'c':
            vs, ps = integ.snapshots(copy=False)       # views of the pinned mirror
            nbytes = vs.nbytes + ps.nbytes
            ok = bool(np.isfinite(vs[-1]).all())
        else:
            nbytes, ok = 0, True
        wall = time.perf_counter() - t0
        return dict(dev_ms=integ.engine.last_run_ms()/K, e2e_ms=wall*1e3/K,
                    host_bytes_per_step=nbytes/K, ok=ok)

    for which in 'abc':                                   # warm every arm's path
        arm(which)
    reps = {w: [] for w in 'abc'}
    for r in range(args.reps):
        for which in 'abc':
            reps[which].append(arm(which))
    # the output kernel's device time, in a run of its own (profiling serialises the launches)
    integ.set_outputs(Cv, Cp, force_dofs=femp['ldsbcinds'], force_ops=ops)
    ctx.profile_begin()
    integ.run(K, **runkw)
    prof = ctx.profile_end()
    cnt, ms = prof['k_imex_outputs']
    step_ms = sum(t for _, t in prof.values())/K
    integ.close()
    name, plim = card()
    res = dict(tool='bench_outputs', gpu=name, power_limit=plim, mesh=args.mesh, members=nb,
               dt=1./args.nts, tol=args.tol, steps_per_rep=K, reps=args.reps, outputs=ny, forces=2,
               kernel=dict(name='k_imex_outputs', launches=cnt, mean_us=ms*1e3/cnt,
                           share_of_profiled_step=ms/K/step_ms))
    for which, rs in reps.items():
        d = {}
        for key in ('dev_ms', 'e2e_ms'):
            v = np.array([x[key] for x in rs])
            d[key] = dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))
        d['host_bytes_per_step'] = rs[-1]['host_bytes_per_step']
        d['ok'] = all(x['ok'] for x in rs)
        res['arm_' + which] = d
    line = json.dumps(res)
    print(line)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
