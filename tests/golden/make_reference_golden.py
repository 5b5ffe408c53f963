#!/usr/bin/env python
"""Reference-RUN golden vectors: outputs of the reference's own code.

Runs the UNMODIFIED modules of the reference checkout that
``DNS_REFERENCE_ROOT`` names (`time_int_utils.py`, `stokes_navier_utils.py`,
`dolfin_to_sparrays.py` condensation helpers, `data_output_utils.py`) through
`tests/refharness.py`
(stub `dolfin` carrier objects, exact sparse solve for the un-vendored
`sadptprj_riclyap_adi.lin_alg_utils.solve_sadpnt_smw`, quadrature for the two
FFC-assembled convection forms) on the operators of the package's host shim,
and stores what they return.  The reference is not part of this repository,
so these small `.npz` files are what pins (a) the oracle (`tests/
test_reference_pin.py`, CPU) and (b) the CUDA path (`tests/test_gpu_parity.py`,
GPU) to reference-run numbers.

    DNS_REFERENCE_ROOT=<checkout> python tests/golden/make_reference_golden.py
                                            # rewrites tests/golden/ref_*.npz
"""
import os
import shutil
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import refharness as rh                                         # noqa: E402
from dolfin_navier_scipy_b200 import problem_setups as dnsps   # noqa: E402

PALPHA = 1e-5            # `tests/time_dep_nse_bcrob.py:26`


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


def bcrob_problem(level, Re):
    """operators of `tests/time_dep_nse_bcrob.py:14-34`"""
    femp, sm, rv, rb = dnsps.get_sysmats(
        problem='cylinderwake', Re=Re, bccontrol=True, scheme='TH',
        meshparams=dict(refinement_level=level))
    A = sm['A'] + sm['Arob']/PALPHA                        # :27
    Brob = sm['Brob']/PALPHA                               # :31
    bdiff = np.asarray(Brob[:, :1] - Brob[:, 1:]).reshape(-1, 1)

    def fvtd(t):                                           # :33-34
        return np.sin(t)*bdiff
    sd = dict(A=A, M=sm['M'], J=sm['J'], JT=sm['JT'],
              fv=rb['fv'] + rv['fv'], fp=rb['fp'] + rv['fp'], fvtd=fvtd,
              V=femp['V'], invinds=femp['invinds'], dbcinds=femp['dbcinds'],
              dbcvals=femp['dbcvals'])
    return femp, sm, sd


class RefRun(object):
    """calls into the reference with a scratch ``data_prfx`` (the reference
    passes trajectories around as `.npy` paths, `snu:1012-1014`)"""

    def __init__(self):
        self.ref = rh.load()
        self.tmp = tempfile.mkdtemp(prefix='dnsref_')
        self.k = 0

    def close(self):
        shutil.rmtree(self.tmp, ignore_errors=True)

    def solve_nse(self, **kw):
        self.k += 1
        kw = rh.as_spmatrix(kw)
        kw.setdefault('data_prfx', os.path.join(self.tmp, 'r%d_' % self.k))
        kw.setdefault('paraviewoutput', False)
        kw.setdefault('verbose', False)
        return self.ref['snu'].solve_nse(**kw)

    def solve_steadystate_nse(self, **kw):
        self.k += 1
        kw = rh.as_spmatrix(kw)
        kw.setdefault('data_prfx', os.path.join(self.tmp, 's%d_' % self.k))
        kw.setdefault('paraviewoutput', False)
        kw.setdefault('save_data', False)
        return self.ref['snu'].solve_steadystate_nse(**kw)

    def load(self, path):
        return self.ref['dou'].load_npa(path)


def ref_imex(run, name, sd, keep, **kw):
    out = run.solve_nse(return_vp_dict=True, **dict(sd, **kw))
    ts = sorted(out.keys())
    kt = [ts[k] for k in keep]
    np.savez_compressed(os.path.join(HERE, name), t=np.array(kt),
                        keep=np.array(keep),
                        v=np.hstack([out[t]['v'] for t in kt]),
                        p=np.hstack([out[t]['p'] for t in kt]))


def golden_imex(run):
    """`snu.solve_nse` IMEX branch -> `tiu.cnab` (cfg 1), and `tiu.sbdftwo`
    called the way `snu:1136-1140,1263-1280` builds its arguments: at HEAD
    `solve_nse(time_int_scheme='sbdf2')` itself fails (`snu:1266` passes
    ``f_tvdp``, which `tiu:260-268` does not accept)"""
    femp, sm, rhsd = cyl(1, 60)
    sd = soldict(femp, sm, rhsd, t0=0., tE=16./512, Nts=16,
                 start_ssstokes=True)
    keep = (0, 1, 2, 8, 16)
    ref_imex(run, 'ref_cnab_cyl1_re60.npz', sd, keep)
    try:
        run.solve_nse(return_vp_dict=True, time_int_scheme='sbdf2', **sd)
        raise RuntimeError('the reference sbdf2 path works: use it')
    except TypeError:
        pass
    snu, tiu, dts = run.ref['snu'], run.ref['tiu'], run.ref['dts']
    spm = rh.as_spmatrix(sd)
    inv = femp['invinds']
    gold = np.load(os.path.join(HERE, 'ref_cnab_cyl1_re60.npz'))
    iniv, inip = gold['v'][inv, :1], gold['p'][:, :1]
    out = {}

    def nonlvfunc(vvec):                                   # snu:1136-1140
        _, convvec, _ = snu.get_v_conv_conts(vvec=vvec, V=femp['V'],
                                             invinds=inv, semi_explicit=True)
        return convvec

    def appndbcs(vvec, ccntrlldbcvals):                    # snu:1002-1005
        return dts.append_bcs_vec(vvec, vdim=femp['V'].dim(), invinds=inv,
                                  bcinds=[femp['dbcinds'], []],
                                  bcvals=[femp['dbcvals'], ccntrlldbcvals])
    trange = np.linspace(0., 16./512, 17)
    tiu.sbdftwo(trange=trange, inivel=iniv, inip=inip, bcs_ini=[],
                M=spm['M'], A=spm['A'], J=spm['J'], f_vdp=nonlvfunc,
                f_tdp=lambda t: sd['fv'], g_tdp=lambda t: sd['fp'],
                scalep=-1., getbcs=lambda *a, **k: [],
                applybcs=lambda bcs: (0., 0., 0.), appndbcs=appndbcs,
                savevp=lambda v, p, time=None: out.update({time: (v, p)}),
                check_ff_maxv=1e8, verbose=False)
    ts = sorted(out.keys())
    kt = [ts[k] for k in keep]
    np.savez_compressed(os.path.join(HERE, 'ref_sbdf2_cyl1_re60.npz'),
                        t=np.array(kt), keep=np.array(keep),
                        v=np.hstack([out[t][0] for t in kt]),
                        p=np.hstack([out[t][1] for t in kt]))


def golden_bcrob(run):
    """Robin boundary control, `tests/time_dep_nse_bcrob.py:26-34` with the
    IMEX integrator (cfg 5), three members of the Re sweep on cylinder_1"""
    vs, ps, Res = [], [], (60., 105., 150.)
    keep = (1, 2, 8, 16)
    for Re in Res:
        femp, sm, sd = bcrob_problem(1, Re)
        out = run.solve_nse(return_vp_dict=True, t0=0., tE=16./512, Nts=16,
                            start_ssstokes=True, **sd)
        ts = sorted(out.keys())
        vs.append(np.hstack([out[ts[k]]['v'] for k in keep]))
        ps.append(np.hstack([out[ts[k]]['p'] for k in keep]))
    np.savez_compressed(os.path.join(HERE, 'ref_bcrob_cyl1.npz'),
                        Re=np.array(Res), keep=np.array(keep),
                        v=np.stack(vs, axis=2), p=np.stack(ps, axis=2))


def golden_newton_cn(run):
    """Picard + Newton sweeps with the trapezoidal rule about the IMEX
    trajectory (`snu:1304-1587`, the two-call recipe; cfg 3 small)"""
    femp, sm, rhsd = cyl(1, 100)
    sd = soldict(femp, sm, rhsd, t0=0., tE=6./512, Nts=6, start_ssstokes=True)
    traj = run.solve_nse(return_dictofvelstrs=True, **sd)
    vd, pd = run.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                           vel_pcrd_stps=1, vel_nwtn_stps=2,
                           return_dictofvelstrs=True,
                           return_dictofpstrs=True, **sd)
    # `snu._atdct` (`snu:974-989`) consumes `datatrange` on the velocity
    # entry of every t, so the pressure dict comes back empty; the pressures
    # are in the `__p` files written beside the `__vel` ones (`snu:1544-1545`)
    assert len(pd) == 0
    ts = sorted(vd.keys())
    np.savez_compressed(os.path.join(HERE, 'ref_newtoncn_cyl1_re100.npz'),
                        t=np.array(ts),
                        v=np.hstack([run.load(vd[t]) for t in ts]),
                        p=np.hstack([run.load(vd[t].replace('__vel', '__p'))
                                     for t in ts]))


def golden_steady(run):
    """`snu.solve_steadystate_nse` on DFG 2D-1 (cfg 2) and `snu.get_pfromv`,
    `snu.get_v_conv_conts` on cylinder_1"""
    femp, sm, rhsd = dnsps.get_sysmats(
        problem='gen_bccont', nu=1e-3, charvel=.2, scheme='TH', mergerhs=True,
        meshparams=dict(strtomeshfile='mesh/karman2D-rotcyl_lvl1.xml.gz',
                        movingwallcntrl=False,
                        strtophysicalregions='mesh/karman2D-rotcyl_lvl1_'
                        'facet_region.xml.gz',
                        strtobcsobs='mesh/karman2D-rotcyl-bm_geo_cntrlbc.json'))
    (v, p), nrms = run.solve_steadystate_nse(
        return_vp=True, return_nwtnupd_norms=True, **soldict(femp, sm, rhsd))
    np.savez_compressed(os.path.join(HERE, 'ref_dfg2d1_lvl1.npz'), v=v, p=p,
                        nwtnupd_norms=np.array(nrms, dtype=float))

    # Re = 30: on this coarse mesh the Galerkin convection of Re = 60 has
    # element Peclet numbers beyond what the device's multigrid-preconditioned
    # Krylov solve covers (it then raises NotConverged, DESIGN.md section 4)
    femp, sm, rhsd = cyl(1, 30)
    sd = soldict(femp, sm, rhsd)
    vss, pss = run.solve_steadystate_nse(return_vp=True, **sd)
    snu = run.ref['snu']
    inv = femp['invinds']
    spm = rh.as_spmatrix(sd)
    pfv = snu.get_pfromv(v=vss[inv], V=femp['V'], M=spm['M'], A=spm['A'],
                         J=spm['J'], fv=sd['fv'], invinds=inv,
                         dbcinds=[femp['dbcinds']], dbcvals=[femp['dbcvals']])
    cm, rc, rbc = snu.get_v_conv_conts(
        vvec=vss, V=femp['V'], invinds=inv, dbcinds=[femp['dbcinds']],
        dbcvals=[femp['dbcvals']])
    pm, _, pbc = snu.get_v_conv_conts(
        vvec=vss, V=femp['V'], invinds=inv, dbcinds=[femp['dbcinds']],
        dbcvals=[femp['dbcvals']], Picard=True)
    rng = np.random.default_rng(7)
    w = rng.standard_normal((inv.size, 1))
    np.savez_compressed(os.path.join(HERE, 'ref_steady_cyl1_re30.npz'),
                        v=vss, p=pss, pfromv=pfv, w=w,
                        newton_mat_w=cm@w, newton_rhs_con=rc, newton_rhs_bc=rbc,
                        picard_mat_w=pm@w, picard_rhs_bc=pbc)


def golden_sie(run):
    """`tiu.semi_implicit_euler` (`tiu:566-635`) with the reference's own
    ``rhsv(t, v) = fv - c(v)[inv]`` on cylinder_1 ("IMEX Euler", cfg 1)"""
    femp, sm, rhsd = cyl(1, 60)
    sd = rh.as_spmatrix(soldict(femp, sm, rhsd))
    snu, tiu = run.ref['snu'], run.ref['tiu']
    inv = femp['invinds']
    vss = run.solve_steadystate_nse(only_stokes=True, **soldict(femp, sm,
                                                                rhsd))

    def rhsv(t, v):
        _, cv, _ = snu.get_v_conv_conts(
            vvec=v, V=femp['V'], invinds=inv, dbcinds=[femp['dbcinds']],
            dbcvals=[femp['dbcvals']], semi_explicit=True)
        return sd['fv'] + cv
    trange = np.linspace(0., 12./512, 13)
    vl = tiu.semi_implicit_euler(iniv=vss[inv], jmat=sd['J'], mmat=sd['M'],
                                 amat=sd['A'], rhsv=rhsv, trange=trange,
                                 fp=sd['fp'])
    np.savez_compressed(os.path.join(HERE, 'ref_sie_cyl1_re60.npz'),
                        t=trange[[0, 1, 6, 12]],
                        v=np.hstack([vl[k] for k in (0, 1, 6, 12)]))


def golden_callbacks(run):
    """`tiu.cnab` / `tiu.sbdftwo` with the reference's callback interface
    (custom ``f_vdp``, ``f_tvdp``, an AB2 observer as ``dynamic_rhs``) and
    `tiu.semi_implicit_euler` with its opaque ``rhsv(t, v)``"""
    import callback_cases as cbc
    from oracle import convection as oconv
    femp, sm, rhsd = cyl(1, 60)
    tiu, dts = run.ref['tiu'], run.ref['dts']
    sd = rh.as_spmatrix(soldict(femp, sm, rhsd))
    inv = femp['invinds']
    NV = inv.size
    gold = np.load(os.path.join(HERE, 'ref_cnab_cyl1_re60.npz'))
    iniv, inip = gold['v'][inv, :1], gold['p'][:, :1]

    def conv_inner(vfull):
        return oconv.convvec(femp['V'], np.ravel(vfull))[inv].reshape(-1, 1)

    def appndbcs(vvec, bcs):
        return dts.append_bcs_vec(vvec, vdim=femp['V'].dim(), invinds=inv,
                                  bcinds=[femp['dbcinds'], []],
                                  bcvals=[femp['dbcvals'], bcs])
    trange = np.linspace(0., 10./512, 11)
    res = {}
    for name, integ in (('cnab', tiu.cnab), ('sbdf2', tiu.sbdftwo)):
        kw = cbc.callback_kwargs(sd['M'], inv, conv_inner, tiu.get_heunab_lti,
                                 NV)
        if name == 'sbdf2':        # `tiu:260-268` has no `f_tvdp`: fold it in
            ftv, dyn = kw.pop('f_tvdp'), kw['dynamic_rhs']

            def dynamic_rhs(t, vc=None, memory={}, mode=None, _d=dyn, _f=ftv):
                val, memory = _d(t, vc=vc, memory=memory, mode=mode)
                return val + _f(t, vc), memory
            kw['dynamic_rhs'] = dynamic_rhs
        v, p, ff = integ(trange=trange, inivel=iniv, inip=inip, bcs_ini=[],
                         M=sd['M'], A=sd['A'], J=sd['J'],
                         f_tdp=lambda t: sd['fv'], g_tdp=lambda t: sd['fp'],
                         scalep=-1., getbcs=lambda *a, **k: [],
                         applybcs=lambda bcs: (0., 0., 0.), appndbcs=appndbcs,
                         savevp=lambda *a, **k: None, dynamic_rhs_memory={},
                         check_ff_maxv=1e8, verbose=False, **kw)
        res['v_' + name], res['p_' + name] = v, p
    np.savez_compressed(os.path.join(HERE, 'ref_callbacks_cyl1_re60.npz'),
                        iniv=iniv, inip=inip, t=trange, **res)


if __name__ == '__main__':
    run = RefRun()
    try:
        golden_callbacks(run)
        golden_imex(run)
        golden_bcrob(run)
        golden_newton_cn(run)
        golden_steady(run)
        golden_sie(run)
    finally:
        run.close()
    for f in sorted(os.listdir(HERE)):
        if f.startswith('ref_') and f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(HERE, f)), 'bytes')
