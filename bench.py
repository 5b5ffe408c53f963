#!/usr/bin/env python
"""bench.py -- cylinder-wake DoF.steps/s on N B200 vs. the host CPU.

Workload (BASELINE.json config 5 on the finest `cylinderwake` mesh, the
configuration the headline metric is quoted on): an ensemble of Robin
boundary-control trajectories of the cylinder wake, Reynolds numbers swept over
[60, 150], Taylor-Hood P2-P1 on `cylinder_4` (28 970 + 3 836 condensed DoFs per
member), CNAB (Crank-Nicolson / Adams-Bashforth-2) with dt = 1/2048, members
sharded over the GPUs (`--members` per GPU, weak scaling, no collective on the
step path).  One "step" = one time step of all members of the batch:
convection re-evaluation (K1a), right-hand side (K2), saddle-point solve (K3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--members B]
                    [--mesh 4] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU restatement of
the reference's scipy path (oracle/: SuperLU + compiled cell loop) on the box's
host cores for the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'cylinder-wake DoF*steps/s'
UNIT = 'DoF*steps/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--warmup', type=int, default=6)
    ap.add_argument('--members', type=int, default=64,
                    help='ensemble members per GPU')
    ap.add_argument('--mesh', type=int, default=4)
    ap.add_argument('--nts', type=int, default=2048, help='steps per time unit')
    ap.add_argument('--tol', type=float, default=1e-12)
    ap.add_argument('--guess', type=int, default=24)
    ap.add_argument('--cheb', type=int, default=4)
    ap.add_argument('--schur-poly', type=int, default=2)
    ap.add_argument('--coarse-max', type=int, default=4096)
    ap.add_argument('--spinup', type=int, default=16,
                    help='untimed steps before the W warm-up steps: the solver recycles the last 16 '
                         'solutions for its initial guesses; a run reaches that operating point after 16 steps')
    ap.add_argument('--schur-precision', default='tc', choices=['f64', 'tf32x3', 'tf32x2', 'tf32', 'tc'],
                    help='dense Schur block of the preconditioner: tc = tcgen05 TF32 with TMEM accumulators '
                         '(default), f64 = fp64 DMMA, tf32* = legacy mma.sync variants; FGMRES '
                         'bases, residuals and stopping test stay fp64 in every case')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cpu-seconds', type=float, default=12.)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-profile', action='store_true')
    ap.add_argument('--no-secondary', action='store_true',
                    help='skip the secondary records (configs 1, 3, 4, dt = 1/512)')
    ap.add_argument('--no-strong', action='store_true',
                    help='N > 1: skip the strong-scaling record (64 members split over the GPUs)')
    ap.add_argument('--no-bind', action='store_true',
                    help='do not pin the ranks of a multi-GPU run to the cores next to their GPU')
    ap.add_argument('--no-parity', action='store_true',
                    help='skip the CPU-oracle check of the measured trajectory')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the state (v, p of every member) after the last timed step as DIR/v.npy, '
                         'DIR/p.npy (float64, at most 64 MB together), to compare builds output for output')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the device path computed: use it with --impl ours')
    return args


# --------------------------------------------------------------------------
# clocks (sampled DURING the timed region)
# --------------------------------------------------------------------------
class ClockSampler(object):
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,'
         'clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:                       # CUDA ordinal -> NVML handle through the UUID
            import torch
            uuid = 'GPU-' + str(torch.cuda.get_device_properties(self.device).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.device)

    def _nvml_loop(self):
        nv, h = self.nvml
        masks = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40),
                 ('sw_thermal_slowdown', 0x20), ('sw_power_cap', 0x4))
        while not self.halt.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append([str(self.device), str(sm), str(self.smax), '',
                                  ] + ['Active' if bits & m else 'Not Active'
                                       for _, m in masks])
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        # NVML polled from a thread (the library calls release the GIL): a few
        # hundred samples over a 0.1 s timed region; nvidia-smi as the fallback
        try:
            self.nvml = self._nvml_handle()
            nv, h = self.nvml
            self.smax = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.halt = threading.Event()
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            self.source = 'nvml'
            return
        except Exception:
            self.nvml = None
        self.source = 'nvidia-smi'
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.device), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '20'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if getattr(self, 'nvml', None) is not None:
            self.halt.set()
            self.thread.join(timeout=2)
        elif self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['unavailable'])
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[4 + k].lower().startswith('active'):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        return dict(sm_mhz=float(np.median(sm)) if sm else None,
                    sm_max_mhz=max(smax) if smax else None,
                    samples=len(sm), source=self.source, reasons=sorted(reasons))


# --------------------------------------------------------------------------
# CPU restatement of the reference (oracle) -- baseline / reference arm
# --------------------------------------------------------------------------
def _cpu_member_worker(args):
    """CNAB steps of ONE member with the oracle (SuperLU + compiled cell loop);
    returns (steps done, seconds in the step loop)."""
    (N, Re, nts, palpha, seconds, maxsteps, nwarm) = args
    sys.stdout = sys.stderr        # worker process: keep the parent's stdout clean
    import scipy.sparse as sps
    import scipy.sparse.linalg as spsla
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from oracle.cconv import CConv
    from oracle.snu import append_bcs_vec
    from oracle.lau import solve_sadpnt_smw
    femp, sm, rv, rb = dnsps.get_sysmats(
        problem='cylinderwake', Re=Re, bccontrol=True, scheme='TH',
        meshparams=dict(refinement_level=N))
    M, J = sm['M'], sm['J']
    A = sm['A'] + sm['Arob']/palpha                # `time_dep_nse_bcrob.py:27`
    Brob = sm['Brob']/palpha
    bdiff = Brob[:, :1] - Brob[:, 1:]
    fv = rb['fv'] + rv['fv']
    fp = rb['fp'] + rv['fp']
    NP, NV = J.shape
    V, inv = femp['V'], femp['invinds']
    cc = CConv(V)
    dt = 1./nts

    def nfc(v):
        vf = append_bcs_vec(v, V.dim(), inv, femp['dbcinds'], femp['dbcvals'])
        return -cc.convvec(vf)[inv].reshape(-1, 1)
    # set-up (not timed): Stokes start, factorisation (`tiu:89-91`)
    v = solve_sadpnt_smw(amat=A, jmat=J, rhsv=fv, rhsp=fp)[:NV]
    K = sps.vstack([sps.hstack([M + .5*dt*A, J.T]),
                    sps.hstack([J, sps.csr_matrix((NP, NP))])], format='csc')
    lu = spsla.factorized(K)
    nfc_c = nfc(v)
    t, n = 0., -nwarm
    tic = time.perf_counter()
    while n < maxsteps and time.perf_counter() - tic < seconds:
        if n == 0:
            tic = time.perf_counter()          # warm-up steps are not timed
        # loop body of `time_int_utils.py:104-143`
        nfc_o, nfc_c = nfc_c, nfc(v)
        rhs = M@v - .5*dt*(A@v) + .5*dt*(3*nfc_c - nfc_o) \
            + .5*dt*(2*fv + (np.sin(t) + np.sin(t + dt))*bdiff)
        vp = lu(np.vstack([rhs, fp]).flatten())
        v = vp[:NV].reshape((NV, 1))
        t += dt
        n += 1
    return n, time.perf_counter() - tic


def _cpu_parity_worker(args):
    """the oracle's CNAB (`oracle.tiu.cnab` = `tiu:23-145`, pinned to the
    reference by tests/test_reference_pin.py) for ONE member of the measured
    ensemble from the same initial state over the same steps; returns the
    final (v, p).  Convection through the compiled cell loop."""
    (N, nu, dt, nsteps, palpha, v0, p0) = args
    sys.stdout = sys.stderr
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from oracle.cconv import CConv
    from oracle.snu import append_bcs_vec
    from oracle import tiu as otiu
    femp, sm, rv, rb = dnsps.get_sysmats(
        problem='cylinderwake', nu=1., bccontrol=True, scheme='TH',
        meshparams=dict(refinement_level=N))
    M, J = sm['M'], sm['J']
    A = nu*sm['A'] + sm['Arob']/palpha
    Brob = sm['Brob']/palpha
    bdiff = np.asarray(Brob[:, :1] - Brob[:, 1:]).reshape(-1, 1)
    fv = nu*(rb['fv'] + rv['fv'])
    fp = rb['fp'] + rv['fp']
    V, inv = femp['V'], femp['invinds']
    cc = CConv(V)

    def appndbcs(v):
        return append_bcs_vec(v, V.dim(), inv, femp['dbcinds'], femp['dbcvals'])

    def f_vdp(vfull):
        return -cc.convvec(np.asarray(vfull).reshape(-1))[inv].reshape(-1, 1)
    trange = dt*np.arange(nsteps + 1)
    v, p, ff = otiu.cnab(trange=trange, inivel=v0.reshape(-1, 1),
                         inip=p0.reshape(-1, 1), M=M, A=A, J=J, f_vdp=f_vdp,
                         f_tdp=lambda t: fv + np.sin(t)*bdiff,
                         g_tdp=lambda t: fp, appndbcs=appndbcs,
                         savevp=lambda *a, **k: None)
    return v, p


def parity_check(job):
    """rel. L2 error of the MEASURED trajectory's state (after the timed
    steps) against the CPU oracle, for the first and the last member"""
    import multiprocessing as mp
    jobs = [(job['mesh'], float(job['nus'][k]), job['dt'], job['nsteps'], 1e-5,
             job['v0'][:, k], job['p0'][:, k]) for k in range(len(job['nus']))]
    with mp.get_context('spawn').Pool(len(jobs)) as pool:
        res = pool.map(_cpu_parity_worker, jobs)
    ev = [float(np.linalg.norm(job['vd'][:, k] - r[0].ravel())/np.linalg.norm(r[0]))
          for k, r in enumerate(res)]
    ep = [float(np.linalg.norm(job['pd'][:, k] - r[1].ravel())/np.linalg.norm(r[1]))
          for k, r in enumerate(res)]
    return dict(v_rel=max(ev), p_rel=max(ep), members=job['members'],
                steps=job['nsteps'], tol_bar=1e-8,
                against='oracle CNAB (tiu:23-145 restated, pinned to the '
                'reference run) from the same initial state, state after '
                'the timed steps')


def cpu_reference(args, nworkers, seconds, maxsteps=10**9, nwarm=3):
    """all host cores: one member per worker process, Re spread over [60,150]"""
    import multiprocessing as mp
    Res = np.linspace(60., 150., max(nworkers, 2))[:nworkers]
    jobs = [(args.mesh, float(Re), args.nts, 1e-5, seconds, maxsteps, nwarm)
            for Re in Res]
    if nworkers == 1:
        res = [_cpu_member_worker(jobs[0])]
    else:
        with mp.get_context('spawn').Pool(nworkers) as pool:
            res = pool.map(_cpu_member_worker, jobs)
    return res


def dofs_of(mesh_level):
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    femp, sm, rv, rb = dnsps.get_sysmats(
        problem='cylinderwake', Re=100., bccontrol=True, scheme='TH',
        meshparams=dict(refinement_level=mesh_level))
    NP, NV = sm['J'].shape
    return NV, NP


def run_reference(args, rank, world):
    if rank != 0:
        return None
    ncores = os.cpu_count() or 1
    NV, NP = dofs_of(args.mesh)
    # W untimed warm-up steps, then K timed "steps"; each step is a bounded
    # sample of the workload: one CNAB step of `ncores` of the 64 members (one
    # per core) -- throughput per member-step, so it extrapolates linearly;
    # the LU factorisation is set-up (`tiu:89-91`), not timed
    res = cpu_reference(args, ncores, seconds=120., maxsteps=args.steps,
                        nwarm=max(args.warmup, 1))
    nsteps = min(r[0] for r in res)
    tmax = max(r[1] for r in res)
    members = len(res)
    value = members*(NV + NP)*nsteps/tmax
    line = dict(metric=METRIC, value=value, unit=UNIT, impl='reference',
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3*tmax/max(nsteps, 1), higher_is_better=True,
                scaling='weak', vs_baseline=None, dtype='f64',
                data='synthetic',
                config=workload_config(args, args.members*world, world),
                cpu_baseline=dict(value=value, unit=UNIT, cores=ncores,
                                  kind='port',
                                  sample='{0} of the {1} members (one per core) '
                                  'x {2} CNAB steps after {3} warm-up steps: '
                                  'SuperLU solve of the prefactorised matrix + '
                                  'compiled cell loop; factorisation excluded'.
                                  format(members, args.members*world, nsteps,
                                         max(args.warmup, 1))),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0,
                         d2h_bytes_per_step=0))
    return line


def workload_config(args, members_total, world):
    return dict(workload='cylinderwake Robin-control ensemble, Re in [60,150], '
                'mesh cylinder_%d, Taylor-Hood P2-P1, CNAB dt=1/%d, '
                '%d members per GPU' % (args.mesh, args.nts, args.members),
                members_total=members_total, members_per_gpu=args.members,
                mesh='cylinder_%d' % args.mesh, scheme='cnab',
                parallelism='ensemble-sharded x%d, no step-path collective'
                % world,
                tol=args.tol, guess=args.guess, cheb_steps=args.cheb,
                schur_poly=args.schur_poly,
                schur_precision=args.schur_precision,
                spinup_steps=max(args.spinup, 0),
                l2_note='ensemble working set (vectors %d members) exceeds L2'
                % args.members)


# --------------------------------------------------------------------------
# secondary records: the other BASELINE configs, device + CPU + parity each
# --------------------------------------------------------------------------
def _cpu_single_worker(args):
    """oracle CNAB (`tiu:23-145`) for ONE plain cylinder-wake trajectory;
    returns (final v, final p, seconds per loop step)"""
    (N, Re, dt, nsteps, v0, p0) = args
    sys.stdout = sys.stderr
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from oracle.cconv import CConv
    from oracle.snu import append_bcs_vec
    from oracle import tiu as otiu
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=Re, scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=N))
    V, inv = femp['V'], femp['invinds']
    cc = CConv(V)
    stamps = []

    def appndbcs(v):
        return append_bcs_vec(v, V.dim(), inv, femp['dbcinds'], femp['dbcvals'])

    def f_vdp(vfull):
        return -cc.convvec(np.asarray(vfull).reshape(-1))[inv].reshape(-1, 1)

    def savevp(v, p, time=None):
        stamps.append(__import__('time').perf_counter())
    trange = dt*np.arange(nsteps + 1)
    v, p, ff = otiu.cnab(trange=trange, inivel=v0.reshape(-1, 1), inip=p0.reshape(-1, 1),
                         M=sm['M'], A=sm['A'], J=sm['J'], f_vdp=f_vdp, f_tdp=lambda t: rhsd['fv'],
                         g_tdp=lambda t: rhsd['fp'], appndbcs=appndbcs, savevp=savevp)
    # loop steps only (the LU factorisation sits between stamps 1 and 2)
    per = (stamps[-1] - stamps[3])/max(len(stamps) - 4, 1) if len(stamps) > 5 else float('nan')
    return v, p, per


def _cpu_sweep_worker(args):
    """oracle Picard + Newton sweeps with the trapezoidal rule (`snu:1304-1587`)"""
    (N, Re, dt, nsteps, iniv, inip) = args
    sys.stdout = sys.stderr
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from oracle import snu as osnu
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=Re, scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=N))
    sd = dict(A=sm['A'], M=sm['M'], J=sm['J'], JT=sm['JT'], fv=rhsd['fv'], fp=rhsd['fp'], V=femp['V'],
              invinds=femp['invinds'], dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'],
              t0=0., tE=nsteps*dt, Nts=nsteps, iniv=iniv, inip=inip)
    traj = osnu.solve_nse(return_dictofvelstrs=True, **sd)
    t0 = time.perf_counter()
    v, p = osnu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False, vel_pcrd_stps=1, vel_nwtn_stps=1,
                          return_final_vp=True, **sd)
    return v, p, (time.perf_counter() - t0)/(2.*nsteps)


def _rel(a, b):
    return float(np.linalg.norm(np.ravel(a) - np.ravel(b))/np.linalg.norm(b))


def ensemble_initial_state(info, nb):
    """steady Stokes solution (`start_ssstokes`, snu:903-908) for the mean
    viscosity, shared by the members of the shard; solved on the device
    (velocity AMG + LSC Schur FGMRES)"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    sm, inv = info['sm'], np.asarray(info['femp']['invinds'])
    NV = info['NV']
    numean = float(np.mean(info['nus']))
    Ast = numean*sm['A'] if info['Arob'] is None else \
        numean*sm['A'] + info['Arob']
    vp = lau.solve_sadpnt_smw(amat=Ast, jmat=sm['J'], jmatT=sm['JT'],
                              rhsv=numean*info['B'][:, :1], rhsp=info['fp'],
                              krylov='gmres', vgroups=(inv//2, inv % 2),
                              mass_diag=sm['M'].diagonal(),
                              krpslvprms=dict(tol=1e-10, maxiter=1500))
    return np.repeat(vp[:NV], nb, axis=1), np.repeat(-vp[NV:], nb, axis=1)


def secondary_records(args, ctx):
    """BASELINE configs 1/3 (single trajectory, IMEX), 3 (Newton/CN sweeps), 4
    (Krylov tolerance of `tests/time_dep_nse_krylov.py:4-7`) on cylinder_4 at
    Re = 100, dt = 1/2048, and the headline ensemble at the reference script's
    dt = 1/512 -- each with the device time, the CPU oracle's time on one host
    core for the same work and the rel. L2 error against it."""
    import multiprocessing as mp
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from dolfin_navier_scipy_b200 import ensemble as ens
    N, Re, dt = args.mesh, 100., 1./args.nts
    out = []
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=Re, scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=N))
    inv = np.asarray(femp['invinds'])
    NP, NV = sm['J'].shape
    vp = lau.solve_sadpnt_smw(amat=sm['A'], jmat=sm['J'], jmatT=sm['JT'], rhsv=rhsd['fv'], rhsp=rhsd['fp'],
                              krylov='gmres', vgroups=(inv//2, inv % 2), mass_diag=sm['M'].diagonal(),
                              krpslvprms=dict(tol=1e-11, maxiter=1500))
    v0 = vp[:NV]
    p0 = snu.get_pfromv(v=v0, V=femp['V'], M=sm['M'], A=sm['M'], J=sm['J'], fv=rhsd['fv'], fp=rhsd['fp'],
                        dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'], invinds=inv)
    pool = mp.get_context('spawn').Pool(2)
    nsingle, nsweep, nsweep_long = 48, 2, 24
    vfull0 = snu.dts.append_bcs_vec(v0, V=femp['V'], invinds=inv, bcinds=femp['dbcinds'],
                                    bcvals=femp['dbcvals'])
    cpu_single = pool.apply_async(_cpu_single_worker, ((N, Re, dt, nsingle, v0, p0),))
    cpu_sweep = pool.apply_async(_cpu_sweep_worker, ((N, Re, dt, nsweep, vfull0, p0),))
    # ---- configs 1/3, IMEX part: one trajectory, tol 1e-12 and the Krylov tolerance 1e-3 ----
    for tol, name in ((args.tol, 'single trajectory CNAB (configs 1/3, IMEX)'),
                      (1e-3, 'single trajectory CNAB, Krylov tol 1e-3 (config 4, '
                       'tests/time_dep_nse_krylov.py:4-7)')):
        integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv, femp['dbcinds'], femp['dbcvals'],
                               dt, fv=rhsd['fv'], fp=rhsd['fp'], ctx=ctx)
        integ.set_state(v0, p0)
        integ.run(nsingle, tol=tol, ntimeslices=0)
        vd, pd = integ.state()
        st0 = integ.stats()
        integ.run(200, tol=tol, ntimeslices=0)      # throughput: later in the same trajectory
        ms = integ.engine.last_run_ms()/200.
        st = integ.stats()
        integ.close()
        out.append(dict(name=name, mesh='cylinder_%d' % N, Re=Re, dt='1/%d' % args.nts, tol=tol,
                        dofs=NV + NP, ms_per_step=ms, value=(NV + NP)/(ms*1e-3), unit=UNIT,
                        fgmres_iters_per_step=st['iters']/float(max(st['solves'], 1)),
                        max_relres=max(st0['max_relres'], st['max_relres']), _vd=vd, _pd=pd))
    # ---- config 3: Picard + Newton sweep with Crank-Nicolson ----
    # parity on a short sweep (the CPU needs 1.5 s per sweep step), throughput on a longer one,
    # timed around dnsb_cnsweep_run (upload of the linearisation trajectory, the device-resident
    # sweep, download of the new trajectory); the host set-up of the solver is reported beside it
    from dolfin_navier_scipy_b200 import _lib
    sweep_calls = []
    _run = _lib.CnSweep.run

    def timed_run(self, *a, **k):
        t = time.perf_counter()
        res = _run(self, *a, **k)
        sweep_calls.append(time.perf_counter() - t)
        return res
    sd = dict(A=sm['A'], M=sm['M'], J=sm['J'], JT=sm['JT'], fv=rhsd['fv'], fp=rhsd['fp'], V=femp['V'],
              invinds=inv, dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'], t0=0., iniv=vfull0, inip=p0)
    swkw = dict(treat_nonl_explicit=False, vel_pcrd_stps=1, vel_nwtn_stps=1, verbose=False)
    traj = snu.solve_nse(return_dictofvelstrs=True, tE=nsweep*dt, Nts=nsweep, **sd)
    vs, ps = snu.solve_nse(lin_vel_point=traj, return_final_vp=True, tE=nsweep*dt, Nts=nsweep,
                           **dict(sd, **swkw))
    trajl = snu.solve_nse(return_dictofvelstrs=True, tE=nsweep_long*dt, Nts=nsweep_long, **sd)
    its = []
    _lib.CnSweep.run = timed_run
    try:
        t0 = time.perf_counter()
        snu.solve_nse(lin_vel_point=trajl, return_final_vp=True, tE=nsweep_long*dt, Nts=nsweep_long,
                      krpslvprms=dict(convstatsl=its), **dict(sd, **swkw))
        sweep_total = time.perf_counter() - t0
    finally:
        _lib.CnSweep.run = _run
    sweep_ms = 1e3*sum(sweep_calls)/(len(sweep_calls)*nsweep_long)
    # ---- CPU legs and parity ----
    vo, po, per = cpu_single.get()
    for k in (0, 1):
        r = out[k]
        vd, pd = r.pop('_vd'), r.pop('_pd')
        r['cpu'] = dict(ms_per_step=1e3*per, cores=1, kind='port',
                        sample='%d CNAB steps, SuperLU solve + compiled cell loop' % nsingle)
        r['speedup_vs_1_core'] = 1e3*per/r['ms_per_step']
        r['parity'] = dict(v_rel=_rel(vd, vo), p_rel=_rel(pd, po), steps=nsingle,
                           note='relative residual 1e-3 (the reference script\'s setting): the recycled guesses already '
                           'meet it, FGMRES does no iteration and the trajectory drifts -- a like-for-like timing, '
                           'not a usable tolerance' if k else
                           'bar 1e-8')
    vso, pso, sper = cpu_sweep.get()
    pool.close()
    out.append(dict(name='Picard + Newton sweep with Crank-Nicolson (config 3, snu:1304-1587)',
                    mesh='cylinder_%d' % N, Re=Re, dt='1/%d' % args.nts, steps=nsweep_long, sweeps=2,
                    ms_per_sweep_step=sweep_ms,
                    fgmres_iters_per_step=float(np.mean(its)) if its else None,
                    call_seconds_with_host_setup=sweep_total,
                    cpu=dict(ms_per_sweep_step=1e3*sper, cores=1, kind='port',
                             sample='2 sweeps x %d steps: K1b in numpy + SuperLU factorisation '
                             'per step' % nsweep),
                    speedup_vs_1_core=1e3*sper/sweep_ms,
                    parity=dict(v_rel=_rel(vs, vso), p_rel=_rel(ps, pso), steps=nsweep,
                                note='final state of the short sweep, bar 1e-8')))
    # ---- the headline ensemble at the reference script's step size ----
    # dt = 1/512 (tests/time_dep_nse_bcrob.py:66 is written for cylinder_2); on cylinder_4 the
    # explicit convection blows up there for the members of highest Re (SURVEY 8d: "halve dt until
    # check_ff stays 0"): the record names the largest power-of-two step that integrates all members
    nb = args.members
    for nts in (512, 1024):
        integ, info = ens.cylinder_ensemble(N=N, nmembers=nb, dt=1./nts, ntimes=200, ctx=ctx,
                                            cheb_steps=args.cheb, schur_poly=args.schur_poly,
                                            coarse_max=args.coarse_max)
        NVe, NPe = info['NV'], info['NP']
        integ.set_state(*ensemble_initial_state(info, nb))
        rec = dict(name='headline ensemble at dt = 1/%d' % nts, members=nb)
        try:
            ff = integ.run(120, tol=args.tol, check_ff_maxv=1e8, ntimeslices=10)
            if ff:
                rec['blow_up'] = 'check_ff guard (tiu:94-103) tripped within 120 steps'
            else:
                integ.run(40, tol=args.tol, ntimeslices=0)
                ms = integ.engine.last_run_ms()/40.
                st = integ.stats()
                rec.update(ms_per_step=ms, value=(NVe + NPe)*nb/(ms*1e-3), unit=UNIT,
                           fgmres_iters_per_step=st['iters']/float(max(st['solves'], 1)),
                           max_relres=st['max_relres'])
        except Exception as ex:
            rec['blow_up'] = repr(ex)[:200]
        integ.close()
        out.append(rec)
        if 'ms_per_step' in rec:
            break
    return out


# --------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------
DUMP_BYTES = 64*10**6


def gather_members(a, world):
    """(n, members of this rank) -> (n, members of every rank) in rank order;
    every rank holds the same number of members"""
    if world == 1:
        return a
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t)
    return torch.cat(parts, dim=1).cpu().numpy()


def dump_outputs(dirname, arrays):
    """``arrays``: name -> (n, members) float64.  Above DUMP_BYTES in all, a
    fixed seeded sample of the members (the same columns of every array) is
    written, so that runs with the same arguments write the same entries."""
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BYTES - 4096             # room for the .npy headers
    ncols = next(iter(arrays.values())).shape[1]
    cols = slice(None)
    if total > budget:
        keep = max(1, ncols*budget//total)
        cols = np.sort(np.random.default_rng(0).choice(ncols, keep, replace=False))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        out = np.ascontiguousarray(a[:, cols], dtype=np.float64)
        np.save(os.path.join(dirname, name + '.npy'), out)
        print('dump-outputs: %s.npy %s' % (name, out.shape), file=sys.stderr)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import ensemble as ens

    torch.cuda.set_device(local_rank)
    if args.schur_precision == 'tc':       # read when the context is created
        os.environ['DNSB_SCHUR_TC'] = '1'
    elif args.schur_precision == 'f64':
        os.environ['DNSB_SCHUR_TC'] = '0'
    else:
        os.environ['DNSB_SCHUR_TF32'] = dict(tf32x3='1', tf32x2='2', tf32='3')[args.schur_precision]
    ctx = _lib.default_context(local_rank)
    nmembers = args.members*world
    ntimes = max(args.warmup, 3) + max(args.spinup, 0) + 4*args.steps + 8
    integ, info = ens.cylinder_ensemble(
        N=args.mesh, nmembers=nmembers, rank=rank, world=world,
        dt=1./args.nts, ntimes=ntimes, ctx=ctx, cheb_steps=args.cheb,
        schur_poly=args.schur_poly, coarse_max=args.coarse_max)
    NV, NP, nb = info['NV'], info['NP'], integ.nb
    v0, p0 = ensemble_initial_state(info, nb)
    runkw = dict(tol=args.tol, guess=args.guess, ntimeslices=0, maxit=400)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    # ---- warm-up ------------------------------------------------------------
    integ.set_state(v0, p0)
    nwarm = max(args.warmup, 3) + max(args.spinup, 0)   # spin-up + W warm-up steps, all untimed
    integ.run(nwarm, **runkw)
    # ---- timed: device-resident steps (inputs already in HBM) ---------------
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ctx.reset_launch_count()
    # ncu --profile-from-start off captures exactly the timed region
    torch.cuda.cudart().cudaProfilerStart()
    t0 = time.perf_counter()
    integ.run(args.steps, **runkw)
    dev_ms = integ.engine.last_run_ms()
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    wall = time.perf_counter() - t0
    launches = ctx.launch_count()
    clocks = sampler.stop()
    st = integ.stats()
    tt = torch.tensor([dev_ms, wall*1e3], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms_max, wall_ms_max = float(tt[0]), float(tt[1])
    units = (NV + NP)*args.members*world*args.steps
    value = units/(dev_ms_max*1e-3)
    # state after spin-up + warm-up + timed steps: checked against the CPU
    # oracle (first and last member of rank 0's shard) once the timing is over
    if args.dump_outputs or (rank == 0 and not args.no_parity):
        Vd, Pd = integ.state()
    if args.dump_outputs:
        Vall, Pall = gather_members(Vd, world), gather_members(Pd, world)
        if rank == 0:
            dump_outputs(args.dump_outputs, dict(v=Vall, p=Pall))
    parity_job = None
    if rank == 0 and not args.no_parity:
        sel = [0, nb - 1] if nb > 1 else [0]
        parity_job = dict(mesh=args.mesh, dt=1./args.nts, nsteps=nwarm + args.steps,
                          nus=[float(info['nus'][k]) for k in sel],
                          members=[int(info['members'][0] + k) for k in sel],
                          v0=v0[:, sel].copy(), p0=p0[:, sel].copy(),
                          vd=Vd[:, sel].copy(), pd=Pd[:, sel].copy())

    # ---- e2e: through the public API with host buffers ----------------------
    # per step the host supplies the boundary-control signal (H2D, host numpy
    # buffers) and receives the (v, p) state of every member (D2H): the
    # running integration is fed the next chunk of the control series and the
    # full trajectory is read back
    B = info['B']
    integ.reserve_snapshots(args.steps + 2)     # pinned mirror, allocated once
    e2e_s = None
    for rep in range(2):     # first pass warms the e2e path up (untimed)
        Urep = np.ascontiguousarray(
            info['U'][nwarm + (1 + rep)*args.steps:
                      nwarm + (2 + rep)*args.steps + 1])
        integ.engine.reset_snapshots()
        barrier()
        t0 = time.perf_counter()
        integ.set_forcing(B, Urep)
        integ.run(args.steps, snap_stride=1, **runkw)
        vs, ps = integ.snapshots(copy=False)    # views of the pinned mirror
        chk = float(np.abs(vs[-1]).sum() + np.abs(ps[-1]).sum())  # host reads
        barrier()
        e2e_s = time.perf_counter() - t0
    U = Urep
    st1 = integ.stats()      # counters of the last run
    e2e_its = st1['iters']/float(max(st1['solves'], 1))
    te = torch.tensor([e2e_s], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = units/float(te[0])
    h2d = (B.nbytes + U.nbytes)/float(args.steps)
    d2h = (vs.nbytes + ps.nbytes)/float(max(vs.shape[0], 1))
    finite = bool(np.isfinite(chk))

    # ---- per-kernel device times (CUDA events on the library's stream) ------
    roofline = None
    kern = {}
    if not args.no_profile:
        ctx.profile_begin(400000)
        integ.run(args.steps, **runkw)
        kern = ctx.profile_end()
        roofline = roofline_of(kern, info, integ, args)

    # ---- POD Gram matrix: the one collective (not on the step path) ---------
    G = ens.gram_allreduce(integ)
    gram = dict(ns=int(G.shape[0]), trace=float(torch.trace(G)),
                symmetric=bool(torch.allclose(G, G.T, rtol=1e-10, atol=0)))

    # ---- strong scaling: the 64-member ensemble of BASELINE config 5 split over the GPUs ----
    strong = None
    if world > 1 and not args.no_strong and args.members % world == 0:
        integ.close()
        sint, sinfo = ens.cylinder_ensemble(
            N=args.mesh, nmembers=args.members, rank=rank, world=world,
            dt=1./args.nts, ntimes=ntimes, ctx=ctx, cheb_steps=args.cheb,
            schur_poly=args.schur_poly, coarse_max=args.coarse_max)
        sint.set_state(*ensemble_initial_state(sinfo, sint.nb))
        sint.run(nwarm, **runkw)
        barrier()
        sint.run(args.steps, **runkw)
        sms = sint.engine.last_run_ms()
        barrier()
        sst = sint.stats()
        ts = torch.tensor([sms, sst['iters']/float(max(sst['solves'], 1))], dtype=torch.float64, device='cuda')
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        strong = dict(scaling='strong', members_total=args.members, members_per_gpu=sint.nb,
                      ms_per_step=float(ts[0])/args.steps,
                      value=(NV + NP)*args.members*args.steps/(float(ts[0])*1e-3), unit=UNIT,
                      fgmres_iters_per_step_max_over_ranks=float(ts[1]),
                      note='the SAME 64 members as at N = 1, %d per GPU; device time, max over ranks; '
                      'parallel efficiency = value / (N x the N = 1 value)' % sint.nb)
        sint.close()

    if rank != 0:
        return None
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world,
                steps=args.steps, warmup=args.warmup,
                ms_per_step=dev_ms_max/args.steps, higher_is_better=True,
                scaling='weak', vs_baseline=None, dtype='f64',
                data='synthetic', impl='ours',
                config=workload_config(args, args.members*world, world),
                clocks=clocks,
                e2e=dict(value=e2e_value, unit=UNIT,
                         h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                         ms_per_step=1e3*float(te[0])/args.steps,
                         fgmres_iters_per_step=e2e_its,
                         note='control-signal chunk H2D (host numpy), K steps, (v,p) '
                         'of every step D2H (async, pinned mirror, caller '
                         'numbering) through DeviceImex; host reads the last '
                         'state'),
                gpu_launches=int(launches),
                wall_ms_per_step=wall_ms_max/args.steps,
                solver=dict(fgmres_iters_per_step=st['iters']/max(st['solves'], 1),
                            max_relres=st['max_relres'],
                            unconverged=st['unconverged'], finite=finite),
                dofs_per_member=NV + NP, gram=gram)
    line['_parity_job'] = parity_job
    if strong is not None:
        line['strong'] = strong
    if world == 1 and not args.no_secondary:
        try:
            line['secondary'] = secondary_records(args, ctx)
        except Exception as ex:      # the headline must survive a failing side record
            line['secondary'] = dict(error=repr(ex))
    if roofline is not None:
        line['roofline'] = roofline
        tot = sum(v[1] for v in kern.values())
        line['kernel_share'] = {k: round(v[1]/tot, 4) for k, v in
                                sorted(kern.items(), key=lambda kv: -kv[1][1])[:8]}
        # name: [launches per step, mean us] (CUDA events around each launch)
        line['kernels'] = {k: [round(v[0]/float(args.steps), 2),
                               round(1e3*v[1]/v[0], 2)] for k, v in
                           sorted(kern.items(), key=lambda kv: -kv[1][1])[:16]}
    return line


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured'
    return 6650., 'fallback'


def _kname(name):
    return name.strip('()').replace('k_cheb_step_b2', 'k_cheb_step') \
        .replace('k_cheb_step_b', 'k_cheb_step')


def kernel_bytes(name, info, integ, mean_work=0.):
    """ALGORITHMIC bytes of one launch (DESIGN.md section 5); None if the
    kernel has no fixed byte count.  ``mean_work``: average number of basis
    vectors a Gram-Schmidt launch read (reported by the library's profiler)"""
    nb = integ.nb
    host = integ._host
    nnzF, n = host['M'].nnz, host['M'].shape[0]
    J = host['J']
    npp = J.shape[0]
    name = name.strip('()')
    if name.startswith('k_cheb_step'):
        flags = name.split('<')[1].rstrip('>').split(', ')
        tiled = name.startswith('k_cheb_step_tile')        # <FIRST, LAST>, packed entries
        first, last = (flags[0] == 'true', flags[1] == 'true') if tiled \
            else (flags[1] == 'true', flags[2] == 'true')
        passes = 7 - (1 if first else 0) - (2 if last else 0)
        if name.startswith('k_cheb_step_tilef'):   # fp32 smoother: 4 floats + 1 offset per pair entry
            return 10.*nnzF + 4.*(n + 1) + 4.*passes*n*nb + (4.*n*nb if last else 0.)
        if tiled:    # 4 values + 1 offset per column of a row pair: 18 B per CSR entry
            return 18.*nnzF + 4.*(n + 1) + 8.*passes*n*nb
        return 20.*nnzF + 4.*(n + 1) + 8.*passes*n*nb
    if name.startswith('k_spmm_b2'):
        # the unpaired divergence rows J of K beside k_spmm_tile: entries, gather of x_v, y_p out
        return 20.*J.nnz + 4.*(npp + 1) + 8.*(n + npp)*nb
    if name.startswith('k_spmm_tile'):
        # paired rows of K = [F JT]: packed entries (18 B per CSR entry) + x in, y out
        # + the unpaired rows J served by the kernel's tail warps: entries, y_p out
        return 18.*(nnzF + J.nnz) + 8.*(n + npp)*nb + 8.*n*nb \
            + 20.*J.nnz + 4.*(npp + 1) + 8.*npp*nb
    if name.startswith('k_spmm'):
        # the block matrix K = [F JT; J 0] (two value arrays): gather + store
        nnzK = nnzF + 2*J.nnz
        nt = n + npp
        return 20.*nnzK + 4.*(nt + 1) + 16.*nt*nb
    if name.startswith('k_gs_tma<false>') or name.startswith('k_mdot_b'):
        return 8.*(n + npp)*nb*(mean_work + 1.)           # basis vectors + w
    if name.startswith('k_gs_tma<true>') or name.startswith('k_gs_update_b'):
        return 8.*(n + npp)*nb*(mean_work + 2.)           # basis vectors + w in, vnext out
    if name.startswith(('k_cheb_init_p2f', 'k_cheb_init_tilef')):
        # JT entries, zp and rv (fp64) in, dinv (fp32) in, res and d (fp32) out
        return 12.*J.nnz + 4.*(n + 1) + 8.*npp*nb + 20.*n*nb
    if name.startswith('k_cheb_init'):
        return 12.*J.nnz + 4.*(n + 1) + 8.*npp*nb + 32.*n*nb
    if name.startswith(('k_dense_gemm', 'k_dense_dmma')):
        return 8.*npp*npp + 16.*npp*nb
    if name.startswith('k_schur_tc'):
        return 4.*npp*npp + 8.*npp*nb
    if name.startswith('k_scale_member'):
        return 16.*(n + npp)*nb
    if name.startswith('k_convvec'):
        return None
    return None


def roofline_of(kern, info, integ, args):
    """roofline of the dominant HBM-bound kernel: algorithmic bytes (DESIGN.md
    section 5) / mean CUDA-event duration of its launches in the timed step.
    The dense Schur solve is a DFMA (fp64 CUDA core) kernel: its TFLOP/s are
    reported beside it."""
    peak, which = measured_peak()
    J = integ._host['J']
    npp, nb = J.shape[0], integ.nb
    # template instantiations of one kernel (FIRST/LAST variants of the
    # Chebyshev step) are one kernel family: launches, time and bytes add up
    fam = {}
    work = getattr(integ.ctx, 'last_work', {})
    for name, (cnt, ms) in kern.items():
        b = kernel_bytes(name, info, integ, work.get(name, 0)/float(max(cnt, 1)))
        base = name.strip('()')
        if b is None or base.startswith('k_dense_'):
            continue
        f = fam.setdefault(base.split('<')[0], dict(cnt=0, ms=0., bytes=0., names=[]))
        f['cnt'] += cnt
        f['ms'] += ms
        f['bytes'] += cnt*b
        f['names'].append((base, cnt))
    key = max(fam.items(), key=lambda kv: kv[1]['ms'])[0]
    families = [dict(kernel=k, launches=v['cnt'], mean_us=1e3*v['ms']/v['cnt'],
                     bytes_per_launch=v['bytes']/v['cnt'],
                     achieved_gbs=v['bytes']/(v['ms']*1e-3)/1e9,
                     frac=v['bytes']/(v['ms']*1e-3)/1e9/peak)
                for k, v in sorted(fam.items(), key=lambda kv: -kv[1]['ms'])]
    f = fam[key]
    cnt, ms = f['cnt'], f['ms']
    bytes_ = f['bytes']/cnt
    dur = ms*1e-3/cnt
    ach = bytes_/dur/1e9
    # DRAM traffic per launch of the same kernels from the committed ncu
    # `--set full` capture (profiles/ncu_traffic.json, written by
    # tools/ncu_summary.py), weighted like the launches; None if not captured
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.isfile(tpath):
        with open(tpath) as fh:
            tr = json.load(fh)
        tot, n = 0., 0
        for nm, c in f['names']:
            t = tr.get(nm.replace('true', '1').replace('false', '0'), {})
            if 'traffic_bytes' in t:
                tot += c*t['traffic_bytes']
                n += c
        traffic = tot/n if n else None
    out = dict(bound='hbm', kernel=key + ('<...>' if len(f['names']) > 1 else ''),
               variants=[nm for nm, _ in f['names']],
               achieved=ach, peak=peak,
               peak_source=which, unit='GB/s', frac=ach/peak, traffic=traffic,
               launches=cnt, mean_us=dur*1e6, bytes_per_launch=bytes_)
    # every HBM-class kernel family of the step, largest first (same arithmetic as the headline entry)
    out['families'] = families
    # where the step goes: the six largest kernels of the timed region by summed event time
    tot_ms = sum(ms for _, ms in kern.values()) or 1.
    out['kernel_shares'] = [dict(kernel=k.strip('()'), launches=c, mean_us=1e3*m/c, share=m/tot_ms)
                            for k, (c, m) in sorted(kern.items(), key=lambda kv: -kv[1][1])[:6]]
    tf = [k for k in kern if k.strip('()').startswith('k_dense_tf32')]
    if tf:
        c, m = kern[tf[0]]
        out['dense_schur'] = dict(kernel=tf[0], mean_us=1e3*m/c,
                                  tf32_tflops=3*2.*npp*npp*nb/(m*1e-3/c)/1e12,
                                  note='3xTF32 mma.sync (fp32 copy of the inverse), '
                                  'preconditioner block only; FGMRES residuals fp64')
    tc = [k for k in kern if k.strip('()').startswith('k_schur_tc')]
    if tc:
        c, m = kern[tc[0]]
        byts = 4.*npp*npp + 8.*npp*nb
        out['dense_schur'] = dict(kernel=tc[0], mean_us=1e3*m/c, bytes_per_launch=byts,
                                  achieved_gbs=byts/(m*1e-3/c)/1e9,
                                  frac_of_hbm_peak=byts/(m*1e-3/c)/1e9/peak,
                                  tf32_tflops=2.*npp*npp*nb/(m*1e-3/c)/1e12,
                                  note='tcgen05.mma kind::tf32 (TMA-fed, TMEM accumulators) on '
                                  'a TF32-rounded fp32 copy of the inverse: HBM bound; '
                                  'preconditioner block only, FGMRES bases/residuals fp64')
    dn = [k for k in kern if k.strip('()').startswith(('k_dense_gemm', 'k_dense_dmma'))]
    if dn:
        c, m = kern[dn[0]]
        flops = 2.*npp*npp*nb
        out['dense_schur'] = dict(kernel=dn[0], mean_us=1e3*m/c,
                                  fp64_tflops=flops/(m*1e-3/c)/1e12,
                                  fp64_peak_tflops=37.2,
                                  note='fp64 pipe bound (148 SM x 64 FMA/clk x '
                                  '1.965 GHz; DMMA m8n8k4 kernel, no '
                                  'tcgen05 kind for fp64)')
    return out


def main():
    # the JSON line must be the only thing on stdout: library notes (e.g. the
    # reference's own "Note: ..." prints, `dts:236-252`) go to stderr
    # -- at the file-descriptor level too: NCCL prints its version banner on
    # fd 1 from C when the first communicator is created
    import contextlib
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        with contextlib.redirect_stdout(sys.stderr):
            line = _main()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    if line is not None:
        print(json.dumps(line), flush=True)


def _main():
    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        return run_reference(args, rank, world)
    if world > 1 and not args.no_bind:
        # NUMA-local pinned snapshot mirrors (see ensemble.bind_to_gpu_cpus)
        from dolfin_navier_scipy_b200 import ensemble as _ens
        _ens.bind_to_gpu_cpus(local_rank)
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', rank=rank, world_size=world,
                                device_id=torch.device('cuda', local_rank))
    line = run_ours(args, rank, world, local_rank)
    if world > 1:
        # the CPU legs below run on rank 0 only: leave the process group first
        # so that the other ranks exit instead of spinning in a NCCL barrier
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return None
    job = line.pop('_parity_job', None)
    if job is not None:
        line['parity'] = parity_check(job)
    if not args.no_cpu_baseline:
        res = cpu_reference(args, 1, seconds=args.cpu_seconds)
        n, t = res[0]
        line['cpu_baseline'] = dict(
            value=line['dofs_per_member']*n/t, unit=UNIT, cores=1,
            kind='port',
            sample='1 member (Re=60), {0} CNAB steps in {1:.1f} s: SuperLU '
            'solve + compiled cell loop, factorisation excluded'.format(n, t))
    return line


if __name__ == '__main__':
    main()
