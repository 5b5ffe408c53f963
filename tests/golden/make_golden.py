#!/usr/bin/env python
"""Generate the golden fixtures of tests/golden/ with the CPU oracle.

The reference itself cannot run in this container (dolfin, krypy and
sadptprj_riclyap_adi are absent and un-installable, SURVEY.md 8c), and it ships
no stored vectors for this path -- its tests are identities plus the printed
DFG 2D-1 literature values (`tests/steadystate_schaefer-turek_2D-1.py:112-114`).
These fixtures therefore pin the *oracle* (restatement with SuperLU, numpy
quadrature): they are produced once, committed, and checked (a) against the
oracle on every CPU run -- so the oracle cannot drift silently -- and (b)
against the CUDA path on the GPU.  The physical known answers (Cd, Cl, dP) tie
the whole chain to the literature values the reference prints.

    python tests/golden/make_golden.py        # rewrites tests/golden/*.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from dolfin_navier_scipy_b200 import problem_setups as dnsps   # noqa: E402
from oracle import convection as oconv                          # noqa: E402
from oracle import snu as osnu                                  # noqa: E402


def soldict(femp, sm, rhsd, **kw):
    d = dict(A=sm['A'], M=sm['M'], J=sm['J'], JT=sm['JT'], fv=rhsd['fv'],
             fp=rhsd['fp'], V=femp['V'], invinds=femp['invinds'],
             dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'])
    d.update(kw)
    return d


def cyl(level, Re):
    return dnsps.get_sysmats(problem='cylinderwake', Re=Re, scheme='TH',
                             mergerhs=True,
                             meshparams=dict(refinement_level=level))


def golden_convection():
    """K1a/K1b: c(u), c(u, w), N1, N2, f3 for seeded fields on cylinder_1"""
    femp, sm, rhsd = cyl(1, 60)
    V = femp['V']
    rng = np.random.default_rng(20261018)
    u = rng.standard_normal(V.dim())
    w = rng.standard_normal(V.dim())
    N1, N2, f3 = oconv.convmats(V, u)
    np.savez_compressed(
        os.path.join(HERE, 'convection_cyl1.npz'), seed=20261018,
        c_uu=oconv.convvec(V, u), c_uw=oconv.convvec(V, u, w),
        n1_data=N1.tocsr().data, n1_indices=N1.tocsr().indices,
        n1_indptr=N1.tocsr().indptr,
        n2_times_w=N2@w, n1_times_w=N1@w, f3=np.ravel(f3))


def golden_cnab():
    """config 1: cylinder wake Re=60, CNAB, 16 steps of dt=1/512 from Stokes"""
    femp, sm, rhsd = cyl(1, 60)
    sd = soldict(femp, sm, rhsd, t0=0., tE=16./512, Nts=16,
                 start_ssstokes=True, return_vp_dict=True)
    ref = osnu.solve_nse(**sd)
    ts = sorted(ref.keys())
    keep = [ts[k] for k in (0, 1, 2, 8, 16)]      # start-up, Heun, AB2, later
    np.savez_compressed(
        os.path.join(HERE, 'cnab_cyl1_re60.npz'), t=np.array(keep),
        v=np.hstack([ref[t]['v'] for t in keep]),
        p=np.hstack([ref[t]['p'] for t in keep]))
    sd.update(time_int_scheme='sbdf2')
    ref = osnu.solve_nse(**sd)
    np.savez_compressed(
        os.path.join(HERE, 'sbdf2_cyl1_re60.npz'), t=np.array(ts),
        v=np.hstack([ref[t]['v'] for t in (ts[4], ts[-1])]),
        p=np.hstack([ref[t]['p'] for t in (ts[4], ts[-1])]))


def golden_newton_cn():
    """config 3 (small): Picard + Newton sweeps with Crank-Nicolson about the
    IMEX trajectory (two-call recipe), cylinder_1, Re=100, 6 steps"""
    femp, sm, rhsd = cyl(1, 100)
    sd = soldict(femp, sm, rhsd, t0=0., tE=6./512, Nts=6, start_ssstokes=True)
    traj = osnu.solve_nse(return_dictofvelstrs=True, **sd)
    out = osnu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                         vel_pcrd_stps=1, vel_nwtn_stps=2,
                         return_dictofvelstrs=True, verbose=False, **sd)
    ts = sorted(out.keys())
    np.savez_compressed(os.path.join(HERE, 'newtoncn_cyl1_re100.npz'),
                        t=np.array(ts),
                        v=np.hstack([out[t] for t in ts]))


def golden_dfg():
    """config 2: DFG 2D-1 steady state on karman2D-rotcyl_lvl1"""
    femp, sm, rhsd = dnsps.get_sysmats(
        problem='gen_bccont', nu=1e-3, charvel=.2, scheme='TH', mergerhs=True,
        meshparams=dict(strtomeshfile='mesh/karman2D-rotcyl_lvl1.xml.gz',
                        movingwallcntrl=False,
                        strtophysicalregions='mesh/karman2D-rotcyl_lvl1_'
                        'facet_region.xml.gz',
                        strtobcsobs='mesh/karman2D-rotcyl-bm_geo_cntrlbc.json'))
    v, p = osnu.solve_steadystate_nse(return_vp=True,
                                      **soldict(femp, sm, rhsd))
    cd, cl = osnu.drag_lift(sm['Afull'], sm['JTfull'], femp['V'], v, p,
                            femp['ldsbcinds'])
    dp = femp['Q'].eval_at(p, (.15, .2)) - femp['Q'].eval_at(p, (.25, .2))
    np.savez_compressed(os.path.join(HERE, 'dfg2d1_lvl1.npz'),
                        cd=-cd, cl=-cl, dp=dp, v=v, p=p,
                        literature=np.array([5.57953523384, 0.010618948146,
                                             0.11752016697]))


def golden_live_cases():
    """what the oracle and the package return for the inputs of the tests
    that run the live reference (`tests/live_cases.py`): the always-run part
    of those tests compares with these, the live part with the reference"""
    sys.path.insert(0, os.path.dirname(HERE))
    import live_cases as lc
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    out = osnu.solve_nse(**dict(lc.bcrob_soldict(1, lc.CNAB_RE), **lc.CNAB_KW))
    ts = sorted(out.keys())
    femp, sm, rhsd = cyl(1, 60)
    (vb, pb), ffb = osnu.solve_nse(**soldict(femp, sm, rhsd, **lc.BLOWUP_KW))
    inp = lc.observer_inputs()
    ab, abkeys = lc.observer_trail(tiu.get_heunab_lti, inp)
    tz, tzkeys = lc.observer_trail(tiu.get_heuntrpz_lti, inp,
                                   constdt=inp['ts'][1] - inp['ts'][0])
    np.savez_compressed(
        os.path.join(HERE, 'live_cases_cyl1.npz'), cnab_t=np.array(ts),
        cnab_v=np.hstack([out[t]['v'] for t in ts]),
        cnab_p=np.hstack([out[t]['p'] for t in ts]),
        blowup_ff=np.array(ffb), blowup_v=vb, blowup_p=pb,
        heunab_out=ab, heunab_keys=np.array(abkeys),
        heuntrpz_out=tz, heuntrpz_keys=np.array(tzkeys))


if __name__ == '__main__':
    golden_convection()
    golden_cnab()
    golden_newton_cn()
    golden_dfg()
    golden_live_cases()
    for f in sorted(os.listdir(HERE)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(HERE, f)), 'bytes')
