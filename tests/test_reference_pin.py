"""The oracle is pinned to outputs of the reference's OWN code.

Two layers:

 * `tests/golden/ref_*.npz` were written by `tests/golden/
   make_reference_golden.py`, which executes the unmodified reference modules
   (`time_int_utils.py`, `stokes_navier_utils.py`, the condensation helpers of
   `dolfin_to_sparrays.py`) through `tests/refharness.py`.  The oracle must
   reproduce them -- always checked, also where the reference is absent.
 * where ``DNS_REFERENCE_ROOT`` names a checkout of the reference, the
   reference is run LIVE beside the oracle on fresh inputs, so neither the
   fixtures nor the oracle can drift.

Tolerance 1e-13 relative (measured: 0.0 -- the oracle performs the same
floating-point operations in the same order).
"""
import os

import numpy as np
import pytest

import live_cases as lc
import refharness as rh
from conftest import soldict
from live_cases import bcrob_soldict

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TOL = 1e-13

needs_ref = pytest.mark.skipif(
    not rh.available(), reason='needs a checkout of the reference '
    'dolfin_navier_scipy: set DNS_REFERENCE_ROOT to its root directory')


def _rel(a, b):
    nb = np.linalg.norm(b)
    return np.linalg.norm(np.asarray(a) - np.asarray(b))/(nb if nb > 0 else 1.)


def _gold(name):
    return np.load(os.path.join(GOLD, name))


def _cyl(level, Re):
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    return dnsps.get_sysmats(problem='cylinderwake', Re=Re, scheme='TH',
                             mergerhs=True,
                             meshparams=dict(refinement_level=level))


# ---------------------------------------------------------------------------
# oracle == committed reference-run fixtures
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('scheme', ['cnab', 'sbdf2'])
def test_oracle_imex_equals_reference_run(cyl1, scheme):
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    g = _gold('ref_%s_cyl1_re60.npz' % scheme)
    out = osnu.solve_nse(t0=0., tE=16./512, Nts=16, start_ssstokes=True,
                         return_vp_dict=True, time_int_scheme=scheme,
                         **soldict(femp, sm, rhsd))
    ts = sorted(out.keys())
    for j, k in enumerate(g['keep']):
        assert _rel(out[ts[k]]['v'], g['v'][:, j:j+1]) <= TOL, (scheme, k)
        assert _rel(out[ts[k]]['p'], g['p'][:, j:j+1]) <= TOL, (scheme, k)


def test_oracle_robin_control_equals_reference_run():
    """cfg 5 (`tests/time_dep_nse_bcrob.py:26-34`): A + Arob/alpha,
    sin(t)(B1 - B2)/alpha, three members of the Re sweep"""
    from oracle import snu as osnu
    g = _gold('ref_bcrob_cyl1.npz')
    for m, Re in enumerate(g['Re']):
        out = osnu.solve_nse(t0=0., tE=16./512, Nts=16, start_ssstokes=True,
                             return_vp_dict=True, **bcrob_soldict(1, float(Re)))
        ts = sorted(out.keys())
        for j, k in enumerate(g['keep']):
            assert _rel(out[ts[k]]['v'], g['v'][:, j:j+1, m]) <= TOL, (Re, k)
            assert _rel(out[ts[k]]['p'], g['p'][:, j:j+1, m]) <= TOL, (Re, k)


def test_oracle_newton_cn_equals_reference_run():
    from oracle import snu as osnu
    g = _gold('ref_newtoncn_cyl1_re100.npz')
    femp, sm, rhsd = _cyl(1, 100)
    sd = soldict(femp, sm, rhsd, t0=0., tE=6./512, Nts=6, start_ssstokes=True)
    traj = osnu.solve_nse(return_dictofvelstrs=True, **sd)
    out = osnu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                         vel_pcrd_stps=1, vel_nwtn_stps=2,
                         return_dictofvelstrs=True, **sd)
    for k, t in enumerate(g['t']):
        assert _rel(out[float(t)], g['v'][:, k:k+1]) <= TOL, t
    vfin, pfin = osnu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                                vel_pcrd_stps=1, vel_nwtn_stps=2,
                                return_final_vp=True, **sd)
    assert _rel(vfin, g['v'][:, -1:]) <= TOL
    assert _rel(pfin, g['p'][:, -1:]) <= TOL


def test_oracle_steady_state_equals_reference_run(cyl1_re30):
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from oracle import snu as osnu
    g = _gold('ref_dfg2d1_lvl1.npz')
    femp, sm, rhsd = dnsps.get_sysmats(
        problem='gen_bccont', nu=1e-3, charvel=.2, scheme='TH', mergerhs=True,
        meshparams=dict(strtomeshfile='mesh/karman2D-rotcyl_lvl1.xml.gz',
                        movingwallcntrl=False,
                        strtophysicalregions='mesh/karman2D-rotcyl_lvl1_'
                        'facet_region.xml.gz',
                        strtobcsobs='mesh/karman2D-rotcyl-bm_geo_cntrlbc.json'))
    (v, p), nrms = osnu.solve_steadystate_nse(
        return_vp=True, return_nwtnupd_norms=True, **soldict(femp, sm, rhsd))
    assert _rel(v, g['v']) <= TOL and _rel(p, g['p']) <= TOL
    # documented deviation: at HEAD the reference only fills
    # `norm_nwtnupd_list` when it LOADS cached data (`snu:303-318`), a fresh
    # solve returns [] (`snu:542-543`); oracle and product return the norms
    assert len(g['nwtnupd_norms']) == 0 and len(nrms) == 3
    assert nrms[-1] < 5e-15 <= nrms[-2]

    femp, sm, rhsd = cyl1_re30
    g = _gold('ref_steady_cyl1_re30.npz')
    sd = soldict(femp, sm, rhsd)
    v, p = osnu.solve_steadystate_nse(return_vp=True, **sd)
    assert _rel(v, g['v']) <= TOL and _rel(p, g['p']) <= TOL
    inv = femp['invinds']
    pfv = osnu.get_pfromv(v=g['v'][inv], V=femp['V'], M=sm['M'], A=sm['A'],
                          J=sm['J'], fv=rhsd['fv'], invinds=inv,
                          dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'])
    assert _rel(pfv, g['pfromv']) <= TOL
    cm, rc, rbc = osnu.get_v_conv_conts(
        vvec=g['v'], V=femp['V'], invinds=inv, dbcinds=femp['dbcinds'],
        dbcvals=femp['dbcvals'])
    assert _rel(cm@g['w'], g['newton_mat_w']) <= TOL
    assert _rel(rc, g['newton_rhs_con']) <= TOL
    assert _rel(rbc, g['newton_rhs_bc']) <= TOL
    pm, none, pbc = osnu.get_v_conv_conts(
        vvec=g['v'], V=femp['V'], invinds=inv, dbcinds=femp['dbcinds'],
        dbcvals=femp['dbcvals'], Picard=True)
    assert none is None
    assert _rel(pm@g['w'], g['picard_mat_w']) <= TOL
    assert _rel(pbc, g['picard_rhs_bc']) <= TOL


def test_oracle_semi_implicit_euler_equals_reference_run(cyl1):
    from oracle import snu as osnu
    from oracle import tiu as otiu
    femp, sm, rhsd = cyl1
    g = _gold('ref_sie_cyl1_re60.npz')
    inv = femp['invinds']

    def rhsv(t, v):
        _, nfc, _ = osnu.get_v_conv_conts(vvec=v, V=femp['V'], invinds=inv,
                                          dbcinds=femp['dbcinds'],
                                          dbcvals=femp['dbcvals'],
                                          semi_explicit=True)
        return rhsd['fv'] + nfc
    trange = np.linspace(0., 12./512, 13)
    vl = otiu.semi_implicit_euler(iniv=g['v'][:, :1], jmat=sm['J'],
                                  mmat=sm['M'], amat=sm['A'], rhsv=rhsv,
                                  trange=trange, fp=rhsd['fp'])
    for j, k in enumerate((0, 1, 6, 12)):
        assert _rel(vl[k], g['v'][:, j:j+1]) <= TOL, k


# ---------------------------------------------------------------------------
# live: the reference's own code beside the oracle.  The tests below that
# run everywhere compare with `tests/golden/live_cases_cyl1.npz` (what the
# oracle and the package return for the same inputs, `tests/golden/
# make_golden.py`) and, where DNS_REFERENCE_ROOT names a checkout, also with
# the reference itself
# ---------------------------------------------------------------------------
@needs_ref
def test_live_reference_modules_are_the_reference_files():
    ref = rh.load()
    for k in ('tiu', 'snu', 'dts', 'dou'):
        assert os.path.realpath(ref[k].__file__).startswith(
            os.path.realpath(rh.REFPKG))
    # only the two dolfin.assemble forms are substituted
    assert ref['dts'].condense_velmatsbybcs.__module__ == \
        'dolfin_navier_scipy.dolfin_to_sparrays'
    assert ref['snu'].get_v_conv_conts.__module__ == \
        'dolfin_navier_scipy.stokes_navier_utils'


def test_live_reference_cnab_with_time_dependent_forcing(tmp_path):
    """`snu.solve_nse` -> `tiu.cnab` of the reference, Robin control at a
    Reynolds number that is in no other fixture, fresh step count"""
    from oracle import snu as osnu
    sd, kw = bcrob_soldict(1, lc.CNAB_RE), lc.CNAB_KW
    out = osnu.solve_nse(**dict(sd, **kw))
    g = _gold('live_cases_cyl1.npz')
    ts = sorted(out.keys())
    assert np.array_equal(ts, g['cnab_t'])
    for j, t in enumerate(ts):
        assert _rel(out[t]['v'], g['cnab_v'][:, j:j+1]) <= TOL, t
        assert _rel(out[t]['p'], g['cnab_p'][:, j:j+1]) <= TOL, t
    if not rh.available():
        return
    ref = rh.load()
    got = ref['snu'].solve_nse(data_prfx=str(tmp_path/'r'), verbose=False,
                               paraviewoutput=False,
                               **rh.as_spmatrix(dict(sd, **kw)))
    assert sorted(got.keys()) == sorted(out.keys())
    for t in sorted(out.keys()):
        assert _rel(out[t]['v'], got[t]['v']) <= TOL, t
        assert _rel(out[t]['p'], got[t]['p']) <= TOL, t


def test_live_reference_blowup_flag(cyl1, tmp_path):
    """`check_ff` / `check_ff_maxv` (`tiu:94-103`)"""
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    sd = soldict(femp, sm, rhsd, **lc.BLOWUP_KW)
    (vo, po), fo = osnu.solve_nse(**sd)
    g = _gold('live_cases_cyl1.npz')
    assert fo == int(g['blowup_ff']) == 1
    assert _rel(vo, g['blowup_v']) <= TOL and _rel(po, g['blowup_p']) <= TOL
    if not rh.available():
        return
    ref = rh.load()
    (vr, pr), fr = ref['snu'].solve_nse(data_prfx=str(tmp_path/'r'),
                                        verbose=False, paraviewoutput=False,
                                        **rh.as_spmatrix(sd))
    assert fo == fr == 1
    assert _rel(vo, vr) <= TOL


@needs_ref
def test_fixtures_are_what_the_reference_returns_today(cyl1, tmp_path):
    ref = rh.load()
    femp, sm, rhsd = cyl1
    g = _gold('ref_cnab_cyl1_re60.npz')
    sd = soldict(femp, sm, rhsd, t0=0., tE=16./512, Nts=16,
                 start_ssstokes=True, return_vp_dict=True)
    got = ref['snu'].solve_nse(data_prfx=str(tmp_path/'r'), verbose=False,
                               paraviewoutput=False, **rh.as_spmatrix(sd))
    ts = sorted(got.keys())
    for j, k in enumerate(g['keep']):
        assert np.array_equal(got[ts[k]]['v'], g['v'][:, j:j+1])
        assert np.array_equal(got[ts[k]]['p'], g['p'][:, j:j+1])


# ---------------------------------------------------------------------------
# callback interface (host logic of the product, no GPU: the device solves are
# replaced by the LU oracle) and the observer discretisations
# ---------------------------------------------------------------------------
class _LuWarmSolver(object):
    """stands in for `hosthop._WarmSolver` (device FGMRES) on a CPU-only box"""

    def __init__(self, F, J, **kw):
        from oracle.lau import SadLU, saddle_matrix
        self.lu = SadLU(saddle_matrix(F, J))
        self.nv = F.shape[0]

    def __call__(self, rhsv, rhsp):
        vp = self.lu.solve(np.vstack([np.asarray(rhsv).reshape(-1, 1),
                                      np.asarray(rhsp).reshape(-1, 1)]))
        return vp[:self.nv].reshape(-1, 1), vp[self.nv:].reshape(-1, 1)

    def close(self):
        pass


@pytest.mark.parametrize('scheme', ['cnab', 'sbdf2'])
def test_host_hop_loop_equals_reference_run_with_callbacks(cyl1, scheme,
                                                           monkeypatch):
    """`hosthop.imex_with_callbacks` (custom ``f_vdp``, ``f_tvdp``, AB2
    observer as ``dynamic_rhs``) reproduces what the reference's `tiu.cnab` /
    `tiu.sbdftwo` returned for the same callbacks"""
    import callback_cases as cbc
    from dolfin_navier_scipy_b200 import hosthop
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import convection as oconv
    from oracle.snu import append_bcs_vec
    monkeypatch.setattr(hosthop, '_WarmSolver', _LuWarmSolver)
    femp, sm, rhsd = cyl1
    g = _gold('ref_callbacks_cyl1_re60.npz')
    inv = femp['invinds']

    def conv_inner(vfull):
        return oconv.convvec(femp['V'], np.ravel(vfull))[inv].reshape(-1, 1)
    kw = cbc.callback_kwargs(sm['M'], inv, conv_inner, tiu.get_heunab_lti,
                             inv.size)
    v, p, ff = hosthop.imex_with_callbacks(
        scheme, trange=g['t'], inivel=g['iniv'], inip=g['inip'], M=sm['M'],
        A=sm['A'], J=sm['J'], f_tdp=lambda t: rhsd['fv'],
        g_tdp=lambda t: rhsd['fp'], scalep=-1.,
        appndbcs=lambda vv, bcs: append_bcs_vec(vv, femp['V'].dim(), inv,
                                                femp['dbcinds'],
                                                femp['dbcvals']),
        check_ff_maxv=1e8, **kw)
    assert ff == 0
    assert _rel(v, g['v_' + scheme]) <= 1e-12
    assert _rel(p, g['p_' + scheme]) <= 1e-10


def test_observer_discretisations_equal_the_reference():
    """`tiu.get_heunab_lti` / `get_heuntrpz_lti` (`tiu:148-257`): same outputs
    and the same memory trail as the reference's closures, mode by mode"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    inp = lc.observer_inputs()
    g = _gold('live_cases_cyl1.npz')
    ref = rh.load()['tiu'] if rh.available() else None
    for name, extra in (('heunab', {}),
                        ('heuntrpz', dict(constdt=inp['ts'][1] - inp['ts'][0]))):
        mine = getattr(tiu, 'get_%s_lti' % name)
        outs, keys = lc.observer_trail(mine, inp, **extra)
        theirs = [(g[name + '_out'], list(g[name + '_keys']))]
        if ref is not None:
            theirs.append(lc.observer_trail(getattr(ref, 'get_%s_lti' % name),
                                            inp, **extra))
        for touts, tkeys in theirs:
            for k, mode in enumerate(lc.OBSERVER_SEQ):
                assert np.allclose(outs[k], touts[k], rtol=1e-14, atol=0), \
                    (name, mode, k)
                assert set(keys[k].split(',')) == set(tkeys[k].split(','))


def test_live_reference_time_sections_are_broken_at_head(tmp_path):
    """`nsects` > 1 (`snu:1076-1087`): the reference's second time section dies
    with `KeyError: None` (`snu:1425-1431`, DESIGN.md section 2) -- the
    product's `NotImplementedError` for `nsects`/`addfullsweep` mirrors a dead
    path, raised before any device work"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = _cyl(1, 100)
    sdp = soldict(femp, sm, rhsd, t0=0., tE=8./512, Nts=8, start_ssstokes=True)
    for kw in (dict(nsects=2), dict(addfullsweep=True)):
        with pytest.raises(NotImplementedError):
            snu.solve_nse(treat_nonl_explicit=False, vel_pcrd_stps=1,
                          vel_nwtn_stps=2, **kw, **sdp)
    if not rh.available():
        return
    ref = rh.load()
    sd = rh.as_spmatrix(soldict(femp, sm, rhsd, t0=0., tE=8./512, Nts=8,
                                start_ssstokes=True))
    kw = dict(verbose=False, paraviewoutput=False)
    traj = ref['snu'].solve_nse(return_dictofvelstrs=True,
                                data_prfx=str(tmp_path/'a'), **kw, **sd)
    with pytest.raises(KeyError):
        ref['snu'].solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                             vel_pcrd_stps=1, vel_nwtn_stps=2, nsects=2,
                             return_dictofvelstrs=True,
                             data_prfx=str(tmp_path/'b'), **kw, **sd)
