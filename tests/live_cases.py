"""Inputs of the cases that `tests/test_reference_pin.py` runs beside the live
reference, shared with `tests/golden/make_golden.py`, which stores what the
oracle and the package return for them (`tests/golden/live_cases_cyl1.npz`)."""
import numpy as np

# Robin control at a Reynolds number that is in no other fixture, fresh step count
CNAB_RE = 87.
CNAB_KW = dict(t0=0., tE=9./256, Nts=9, start_ssstokes=True,
               return_vp_dict=True)
# `check_ff` / `check_ff_maxv` (`tiu:94-103`): the guard trips
BLOWUP_KW = dict(t0=0., tE=24./512, Nts=24, start_ssstokes=True,
                 return_final_vp=True, check_ff=True, check_ff_maxv=1e-3)
OBSERVER_SEQ = ['init', 'heunpred', 'heuncorr'] + ['abtwo']*4


def bcrob_soldict(level, Re, palpha=1e-5):
    """`tests/time_dep_nse_bcrob.py:14-34` on the host shim's operators"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    femp, sm, rv, rb = dnsps.get_sysmats(
        problem='cylinderwake', Re=Re, bccontrol=True, scheme='TH',
        meshparams=dict(refinement_level=level))
    Brob = sm['Brob']/palpha
    bdiff = np.asarray(Brob[:, :1] - Brob[:, 1:]).reshape(-1, 1)
    return dict(A=sm['A'] + sm['Arob']/palpha, M=sm['M'], J=sm['J'],
                JT=sm['JT'], fv=rb['fv'] + rv['fv'], fp=rb['fp'] + rv['fp'],
                fvtd=lambda t: np.sin(t)*bdiff, V=femp['V'],
                invinds=femp['invinds'], dbcinds=femp['dbcinds'],
                dbcvals=femp['dbcvals'])


def observer_inputs():
    """a 4-state observer of 2 inputs and 3 outputs, seeded"""
    rng = np.random.default_rng(3)
    ha = -2.*np.eye(4) + rng.standard_normal((4, 4))
    hb, hc = rng.standard_normal((4, 2)), rng.standard_normal((3, 4))
    x0 = rng.standard_normal((4, 1))
    ts = np.linspace(0., .5, 6)
    ys = np.stack([rng.standard_normal((2, 1)) for _ in ts])
    return dict(ha=ha, hb=hb, hc=hc, x0=x0, ts=ts, ys=ys)


def observer_trail(get_observer, inp, **extra):
    """outputs and memory keys of an observer discretisation (`tiu:148-257`)
    called in the order the integrators call it; -> (outputs (k, 3, 1),
    ['key,key,..' per call])"""
    ts, ys = inp['ts'], inp['ys']
    obs = get_observer(hb=inp['hb'], ha=inp['ha'], hc=inp['hc'],
                       inihx=inp['x0'],
                       drift=lambda t: np.full((4, 1), np.sin(t)), **extra)
    times = [ts[0], ts[1], ts[1]] + list(ts[2:])
    outs, keys, mem = [], [], {}
    for k, (t, mode) in enumerate(zip(times, OBSERVER_SEQ)):
        u, mem = obs(t, vc=ys[min(k, 5)], memory=mem, mode=mode)
        outs.append(np.asarray(u, dtype=float))
        keys.append(','.join(sorted(mem.keys())))
    return np.stack(outs), keys
