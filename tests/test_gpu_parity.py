"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle
on the same inputs.  Tolerances follow BASELINE.json: relative L2 error of
velocity and pressure <= 1e-8 per step in fp64."""
import numpy as np
import pytest
import scipy.sparse as sps

from conftest import soldict
from kernel_refs import cheb_np as _cheb_np
from kernel_refs import ctx_with_env as _ctx_with_env

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def ctx():
    from dolfin_navier_scipy_b200 import _lib
    return _lib.default_context(0)


def _rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b))/np.linalg.norm(b)


def test_device_is_b200_class(ctx):
    info = ctx.info()
    assert info['cc'] >= 100, info
    assert info['sm_count'] >= 100


def test_convvec_matches_oracle(cyl1, ctx):
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    from oracle import convection as oconv
    femp, sm, rhsd = cyl1
    V = femp['V']
    rng = np.random.default_rng(0)
    u = rng.standard_normal(V.dim())
    w = rng.standard_normal(V.dim())
    c = dts.get_convvec(V=V, u0_vec=u)
    assert c.shape == (V.dim(), 1)
    assert _rel(c.ravel(), oconv.convvec(V, u)) < 1e-13
    c2 = dts.get_convvec(V=V, u0_vec=u, uone_utwo_same=False, utwo_vec=w)
    assert _rel(c2.ravel(), oconv.convvec(V, u, w)) < 1e-13
    # inner-node interface (`dts:466-467`)
    inv = femp['invinds']
    ci = dts.get_convvec(V=V, u0_vec=u, invinds=inv)
    assert np.array_equal(ci, c[inv])


def test_convvec_batched_and_deterministic(cyl1, ctx):
    from dolfin_navier_scipy_b200 import _lib
    from oracle import convection as oconv
    femp = cyl1[0]
    V = femp['V']
    dev = _lib.device_for(V)
    rng = np.random.default_rng(1)
    U = rng.standard_normal((V.dim(), 5))
    C = dev.convvec(U)
    for m in range(5):
        assert _rel(C[:, m], oconv.convvec(V, U[:, m])) < 1e-13
    assert np.array_equal(C, dev.convvec(U))       # bit-reproducible


def test_convmats_match_oracle(cyl1, ctx):
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    from oracle import convection as oconv
    femp = cyl1[0]
    V = femp['V']
    rng = np.random.default_rng(2)
    u = rng.standard_normal(V.dim())
    N1, N2, f3 = dts.get_convmats(u0_vec=u, V=V)
    O1, O2, o3 = oconv.convmats(V, u)
    assert abs(N1 - O1).max() < 1e-13*abs(O1).max()
    assert abs(N2 - O2).max() < 1e-13*abs(O2).max()
    assert _rel(f3, o3) < 1e-13
    # `tests/test_units_fenicsci.py:84-85`
    assert _rel(N1@u, f3.ravel()) < 1e-12 and _rel(N2@u, f3.ravel()) < 1e-12


def test_spmm_matches_scipy(cyl1, ctx):
    femp, sm, rhsd = cyl1
    A = sps.csr_matrix(sm['A'])
    rng = np.random.default_rng(3)
    mat = ctx.csr(A)
    x = rng.standard_normal(A.shape[1])
    assert _rel(mat.spmm(x), A@x) < 1e-14
    X = rng.standard_normal((A.shape[1], 7))
    Y0 = rng.standard_normal((A.shape[0], 7))
    Y = mat.spmm(X, alpha=-.5, beta=2., y=Y0)
    assert _rel(Y, -.5*(A@X) + 2*Y0) < 1e-14
    # two value arrays with per-member coefficients
    M = sps.csr_matrix(sm['M'])
    from dolfin_navier_scipy_b200.time_int_utils import _on_pattern, _union_pattern
    pat = _union_pattern([M, A])
    Mp, Ap = _on_pattern(M, pat), _on_pattern(A, pat)
    m2 = ctx.csr(Mp, Ap.data)
    coef = np.array([0., 1., .25, -2., 3., .5, 7.])
    Y = m2.spmm(X, coef=coef)
    for k in range(7):
        assert _rel(Y[:, k], M@X[:, k] + coef[k]*(A@X[:, k])) < 1e-13
    # rectangular
    J = sps.csr_matrix(sm['J'])
    assert _rel(ctx.csr(J).spmm(x), J@x) < 1e-14


def test_saddle_solver_matches_lu(cyl1, ctx):
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from oracle.lau import solve_sadpnt_smw as olu
    femp, sm, rhsd = cyl1
    dt = 1./512
    F = (sm['M'] + .5*dt*sm['A']).tocsr()
    rng = np.random.default_rng(4)
    b = sm['M']@rng.standard_normal((F.shape[0], 2))
    g = np.zeros((sm['J'].shape[0], 2))
    stats = []
    vp = lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b,
                              rhsp=g, krylov='gmres',
                              krpslvprms=dict(tol=1e-12, maxiter=200,
                                              convstatsl=stats))
    ref = olu(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b, rhsp=g)
    NV = F.shape[0]
    assert vp.shape == ref.shape
    assert _rel(vp[:NV], ref[:NV]) < 1e-9
    assert _rel(vp[NV:], ref[NV:]) < 1e-8
    assert 0 < stats[0] < 80


@pytest.mark.parametrize('ncols', [12, 20, 70])
def test_saddle_solver_many_columns(cyl1, ctx, ncols):
    """batched right-hand sides: dense Schur solve as split-K GEMM (16/32/64
    member tiles), staged SpMM, fused Gram-Schmidt"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from oracle.lau import solve_sadpnt_smw as olu
    femp, sm, rhsd = cyl1
    dt = 1./512
    F = (sm['M'] + .5*dt*sm['A']).tocsr()
    rng = np.random.default_rng(40 + ncols)
    b = sm['M']@rng.standard_normal((F.shape[0], ncols))
    g = sm['J']@rng.standard_normal((F.shape[0], ncols))*1e-3
    vp = lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b,
                              rhsp=g, krylov='gmres',
                              krpslvprms=dict(tol=1e-12, maxiter=200))
    ref = olu(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b, rhsp=g)
    NV = F.shape[0]
    for k in range(ncols):
        assert _rel(vp[:NV, k], ref[:NV, k]) < 1e-9, k
        assert _rel(vp[NV:, k], ref[NV:, k]) < 1e-8, k


def test_imex_cnab_parity_per_step(cyl1, ctx):
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    sd = soldict(femp, sm, rhsd, t0=0., tE=24./512, Nts=24,
                 start_ssstokes=True, return_vp_dict=True)
    got = snu.solve_nse(**sd)
    ref = osnu.solve_nse(**sd)
    assert sorted(got.keys()) == sorted(float(t) for t in ref.keys())
    tr = sorted(ref.keys())
    for t in tr[1:]:
        assert _rel(got[float(t)]['v'], ref[t]['v']) < 1e-8, t
        assert _rel(got[float(t)]['p'], ref[t]['p']) < 1e-8, t


def test_imex_sbdf2_final_state(cyl1, ctx):
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    sd = soldict(femp, sm, rhsd, t0=0., tE=20./512, Nts=20,
                 start_ssstokes=True, return_final_vp=True,
                 time_int_scheme='sbdf2')
    v, p = snu.solve_nse(**sd)
    vo, po = osnu.solve_nse(**sd)
    assert _rel(v, vo) < 1e-8 and _rel(p, po) < 1e-8


def test_ensemble_members_equal_single_runs(cyl1, ctx):
    """batched trajectories (shared pattern, different nu) == individual runs"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    nu0 = femp['nu']
    A0 = sm['A']/nu0
    nus = np.array([nu0, .5*nu0, 2*nu0])
    dt, nsteps = 1./512, 10
    # boundary contribution of A scales with nu: fv_m = nu_m/nu0 * fv
    inv = femp['invinds']
    v0 = osnu.solve_nse(t0=0, tE=dt, Nts=1, start_ssstokes=True,
                        return_vp_dict=True, **soldict(femp, sm, rhsd))
    v_ini = v0[0.0]['v'][inv]
    # per-member forcing through the input interface: fv_m = (nu_m/nu0) fv
    integ = tiu.DeviceImex(sm['M'], A0, sm['J'], femp['V'], inv,
                           femp['dbcinds'], femp['dbcvals'], dt, nus=nus,
                           fp=rhsd['fp'])
    U = np.broadcast_to((nus/nu0)[None, None, :], (nsteps + 1, 1, 3))
    integ.set_forcing(rhsd['fv'], U)
    integ.set_state(v_ini, v0[0.0]['p'])
    integ.run(nsteps, tol=1e-12)
    V, P = integ.state()
    integ.close()
    for m, nu in enumerate(nus):
        sd = soldict(femp, sm, rhsd)
        sd.update(A=nu*A0, fv=nu/nu0*rhsd['fv'])
        ref = osnu.solve_nse(t0=0, tE=nsteps*dt, Nts=nsteps, iniv=v0[0.0]['v'],
                             inip=v0[0.0]['p'], return_final_vp=True, **sd)
        assert _rel(V[:, m:m+1], ref[0]) < 1e-8, m
        assert _rel(P[:, m:m+1], ref[1]) < 1e-8, m


# ---------------------------------------------------------------------------
# committed golden fixtures (tests/golden/, generated by make_golden.py)
# ---------------------------------------------------------------------------
import os                                                    # noqa: E402
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def test_golden_convection_device(cyl1, ctx):
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    g = np.load(os.path.join(GOLD, 'convection_cyl1.npz'))
    V = cyl1[0]['V']
    rng = np.random.default_rng(int(g['seed']))
    u = rng.standard_normal(V.dim())
    w = rng.standard_normal(V.dim())
    assert _rel(dts.get_convvec(V=V, u0_vec=u).ravel(), g['c_uu']) < 1e-13
    c2 = dts.get_convvec(V=V, u0_vec=u, uone_utwo_same=False, utwo_vec=w)
    assert _rel(c2.ravel(), g['c_uw']) < 1e-13
    N1, N2, f3 = dts.get_convmats(u0_vec=u, V=V)
    assert _rel(N1@w, g['n1_times_w']) < 1e-13
    assert _rel(N2@w, g['n2_times_w']) < 1e-13
    assert _rel(np.ravel(f3), g['f3']) < 1e-13


def test_golden_cnab_and_sbdf2_device(cyl1, ctx):
    """BASELINE config 1 against the committed trajectory (tol 1e-8 per step)"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = cyl1
    g = np.load(os.path.join(GOLD, 'cnab_cyl1_re60.npz'))
    got = snu.solve_nse(t0=0., tE=16./512, Nts=16, start_ssstokes=True,
                        return_vp_dict=True, **soldict(femp, sm, rhsd))
    for k, t in enumerate(g['t']):
        assert _rel(got[float(t)]['v'], g['v'][:, k:k+1]) < 1e-8, t
        if k > 0:
            assert _rel(got[float(t)]['p'], g['p'][:, k:k+1]) < 1e-8, t
    g = np.load(os.path.join(GOLD, 'sbdf2_cyl1_re60.npz'))
    got = snu.solve_nse(t0=0., tE=16./512, Nts=16, start_ssstokes=True,
                        return_vp_dict=True, time_int_scheme='sbdf2',
                        **soldict(femp, sm, rhsd))
    for k, t in enumerate((4./512, 16./512)):
        assert _rel(got[float(t)]['v'], g['v'][:, k:k+1]) < 1e-8, t
        assert _rel(got[float(t)]['p'], g['p'][:, k:k+1]) < 1e-8, t


def test_golden_newton_cn_sweeps_device(cyl1, ctx):
    """BASELINE config 3 (small): Picard + Newton sweeps with Crank-Nicolson"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    g = np.load(os.path.join(GOLD, 'newtoncn_cyl1_re100.npz'))
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=100,
                                       scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=1))
    sd = soldict(femp, sm, rhsd, t0=0., tE=6./512, Nts=6, start_ssstokes=True)
    traj = snu.solve_nse(return_dictofvelstrs=True, **sd)
    out = snu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                        vel_pcrd_stps=1, vel_nwtn_stps=2,
                        return_dictofvelstrs=True, verbose=False, **sd)
    for k, t in enumerate(g['t']):
        assert _rel(out[float(t)], g['v'][:, k:k+1]) < 1e-8, t


def test_golden_dfg_steady_state_device(ctx):
    """BASELINE config 2: Stokes -> Picard -> Newton on karman2D-rotcyl_lvl1;
    drag/lift within 1e-6 relative of the oracle, dP likewise"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from oracle import snu as osnu
    g = np.load(os.path.join(GOLD, 'dfg2d1_lvl1.npz'))
    femp, sm, rhsd = dnsps.get_sysmats(
        problem='gen_bccont', nu=1e-3, charvel=.2, scheme='TH', mergerhs=True,
        meshparams=dict(strtomeshfile='mesh/karman2D-rotcyl_lvl1.xml.gz',
                        movingwallcntrl=False,
                        strtophysicalregions='mesh/karman2D-rotcyl_lvl1_'
                        'facet_region.xml.gz',
                        strtobcsobs='mesh/karman2D-rotcyl-bm_geo_cntrlbc.json'))
    v, p = snu.solve_steadystate_nse(return_vp=True, verbose=False,
                                     **soldict(femp, sm, rhsd))
    assert _rel(v, g['v']) < 1e-8
    assert _rel(p, g['p']) < 1e-8
    cd, cl = osnu.drag_lift(sm['Afull'], sm['JTfull'], femp['V'], v, p,
                            femp['ldsbcinds'])
    dp = femp['Q'].eval_at(p, (.15, .2)) - femp['Q'].eval_at(p, (.25, .2))
    # the product's functional (`residual_checks`, convection term on the device)
    from dolfin_navier_scipy_b200 import residual_checks as rck
    ssres = rck.get_steady_state_res(V=femp['V'], gradvsymmtrc=True, outflowds=femp['outflowds'], nu=1e-3)
    cd2, cl2 = rck.lift_drag_via_residual(ssres, v, p, femp['ldsbcinds'])
    assert abs(cd2 - cd) < 1e-10*abs(cd) and abs(cl2 - cl) < 1e-10*abs(cl)
    res = ssres(v, p)
    assert np.linalg.norm(res[femp['invinds']]) < 1e-8*np.linalg.norm(sm['Afull']@v.reshape(-1))
    assert abs(-cd - float(g['cd'])) < 1e-6*abs(float(g['cd']))
    assert abs(-cl - float(g['cl'])) < 1e-6*abs(float(g['cl']))
    assert abs(dp - float(g['dp'])) < 1e-6*abs(float(g['dp']))


# ---------------------------------------------------------------------------
# remaining rows of the scope table (SURVEY.md 8a) and edge cases
# ---------------------------------------------------------------------------
def test_semi_implicit_euler_matches_oracle(cyl1, ctx):
    """a8: `tiu.semi_implicit_euler` (`tiu:566-635`) with rhs fv - N(v)v"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import tiu as otiu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    sd = soldict(femp, sm, rhsd)
    v0 = osnu.solve_nse(t0=0, tE=1./512, Nts=1, start_ssstokes=True,
                        return_vp_dict=True, **sd)[0.0]['v'][inv]
    trange = np.linspace(0., 12./512, 13)

    def rhsv(t, v):
        _, nfc, _ = osnu.get_v_conv_conts(vvec=v, V=femp['V'], invinds=inv,
                                          dbcinds=femp['dbcinds'],
                                          dbcvals=femp['dbcvals'],
                                          semi_explicit=True)
        return rhsd['fv'] + nfc
    ref = otiu.semi_implicit_euler(iniv=v0, jmat=sm['J'], mmat=sm['M'],
                                   amat=sm['A'], rhsv=rhsv, trange=trange,
                                   fp=rhsd['fp'])
    got = tiu.semi_implicit_euler(iniv=v0, jmat=sm['J'], mmat=sm['M'],
                                  amat=sm['A'], trange=trange, fp=rhsd['fp'],
                                  V=femp['V'], invinds=inv,
                                  dbcinds=femp['dbcinds'],
                                  dbcvals=femp['dbcvals'], fv=rhsd['fv'])
    assert len(got) == len(ref)
    for a, b in zip(got[1:], ref[1:]):
        assert _rel(a, b) < 1e-8


def test_get_pfromv_matches_oracle(cyl1, ctx):
    """a12: `snu.get_pfromv` (`snu:1602-1633`)"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    rng = np.random.default_rng(5)
    v = 0.1*rng.standard_normal((inv.size, 1))
    kw = dict(v=v, V=femp['V'], M=sm['M'], A=sm['A'], J=sm['J'],
              fv=rhsd['fv'], dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'],
              invinds=inv)
    assert _rel(snu.get_pfromv(**kw), osnu.get_pfromv(**kw)) < 1e-8


def test_blowup_guard_sets_ffflag(cyl1, ctx):
    """`check_ff` (`tiu:94-103`, `snu:1281-1285`): an unstable step size must
    trip the guard, a stable one must not"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = cyl1
    sd = soldict(femp, sm, rhsd, start_ssstokes=True, return_final_vp=True,
                 check_ff=True, check_ff_maxv=1e3)
    (v, p), ff = snu.solve_nse(t0=0., tE=40./512, Nts=40, **sd)
    assert ff == 0 and np.all(np.isfinite(v))
    # explicit convection with a huge step: CFL violated by orders of magnitude
    _, ff = snu.solve_nse(t0=0., tE=400., Nts=40, **sd)
    assert ff == 1


def test_krylov_statistics_and_tolerance(cyl1, ctx):
    """config 4 (`tests/time_dep_nse_krylov.py:4-7,47`): `krpslvprms` tol /
    maxiter are honoured, `convstatsl` collects the iteration counts"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from oracle.lau import solve_sadpnt_smw as olu
    femp, sm, rhsd = cyl1
    F = (sm['M'] + .5/512*sm['A']).tocsr()
    b = sm['M']@np.random.default_rng(6).standard_normal((F.shape[0], 1))
    ref = olu(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b)
    its = []
    for tol in (1e-3, 1e-8, 1e-12):
        vp = lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b,
                                  krylov='Gmres',
                                  krpslvprms=dict(tol=tol, maxiter=800,
                                                  convstatsl=its))
        assert _rel(vp[:F.shape[0]], ref[:F.shape[0]]) < 50*tol
    assert its[0] < its[1] < its[2]


@pytest.mark.parametrize('nb', [1, 3, 4, 33])
def test_spmm_all_batch_widths(cyl1, ctx, nb):
    """every kernel family: nb = 1 (lanes per row), odd (one member per
    thread), even (member pairs / row pairs), > 32"""
    femp, sm, rhsd = cyl1
    from dolfin_navier_scipy_b200.time_int_utils import _on_pattern, _union_pattern
    M, A = sps.csr_matrix(sm['M']), sps.csr_matrix(sm['A'])
    pat = _union_pattern([M, A])
    Mp, Ap = _on_pattern(M, pat), _on_pattern(A, pat)
    m2 = ctx.csr(Mp, Ap.data)
    rng = np.random.default_rng(nb)
    X = rng.standard_normal((A.shape[1], nb))
    coef = rng.standard_normal(nb)
    Y = m2.spmm(X, coef=coef)
    for k in range(nb):
        assert _rel(Y[:, k], M@X[:, k] + coef[k]*(A@X[:, k])) < 1e-13
    JT = sps.csr_matrix(sm['JT'])
    P = rng.standard_normal((JT.shape[1], nb))
    assert _rel(ctx.csr(JT).spmm(P), JT@P) < 1e-13


@pytest.mark.parametrize('kind', ['stokes', 'picard'])
def test_preconditioner_matches_numpy_restatement(cyl1, ctx, kind):
    """one application of the block-triangular preconditioner with the LSC
    Schur approximation and the 2-level SA-AMG V-cycle (`dnsb_solver_apply_prec`)
    against a numpy restatement built from the SAME host-side hierarchy"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from oracle import convection as oconv
    from oracle import snu as osnu
    from oracle.lau import solve_sadpnt_smw as olu
    femp, sm, rhsd = cyl1
    A, M, J = sm['A'].tocsr(), sm['M'].tocsr(), sm['J'].tocsr()
    NP, NV = J.shape
    inv = np.asarray(femp['invinds'])
    F = A
    if kind == 'picard':
        ref = olu(amat=A, jmat=J, jmatT=J.T, rhsv=rhsd['fv'], rhsp=rhsd['fp'])
        vfull = osnu.append_bcs_vec(ref[:NV], femp['V'].dim(), inv,
                                    femp['dbcinds'], femp['dbcvals'])
        N1, _, _ = oconv.convmats(femp['V'], vfull.ravel())
        F = (A + N1[inv][:, inv]).tocsr()
    op = lau.SadpntOperator(F, J, J.T.tocsr(), vgroups=(inv//2, inv % 2),
                            mass_diag=M.diagonal())
    info = op.info
    assert info['velocity_amg']
    kF = 2 if kind == 'picard' else 3
    vlevels, vdense = info['vhierarchy']
    slevels, sdense = info['hierarchy']
    assert len(vlevels) == 1 and len(slevels) == 0
    lmin0, lmax0 = info['spectrum']
    du_inv = 1./M.diagonal()
    r = np.random.default_rng(11).standard_normal(NV + NP)
    z = op.solver.apply_prec(r).ravel()
    rv, rp = r[:NV], r[NV:]
    t = sdense@rp                                    # LSC: L^-1 (J D F D JT) L^-1
    t = du_inv*(J.T@t)
    t = du_inv*(F@t)
    zp = -(sdense@(J@t))
    b = rv - J.T@zp
    dinv = 1./F.diagonal()
    x = _cheb_np(F, dinv, b, kF, lmin0, lmax0)       # V-cycle, 2 levels
    x = x + vlevels[0]['P']@(vdense@(vlevels[0]['R']@(b - F@x)))
    zv = x + _cheb_np(F, dinv, b - F@x, kF, lmin0, lmax0)
    op.close()
    assert _rel(z[NV:], zp) < 1e-11
    assert _rel(z[:NV], zv) < 1e-11


def test_cnab_with_multilevel_schur_hierarchy(cyl1, ctx):
    """pressure meshes beyond the dense-inverse limit use a smoothed-aggregation
    V-cycle for the Schur approximation: force that path (coarse_max=200) on
    the small mesh, single trajectory and a 64-member batch (row-pair kernels,
    DMMA coarse solve), and check CNAB against the LU oracle"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    sd = soldict(femp, sm, rhsd)
    nsteps, dt = 8, 1./512
    v0d = osnu.solve_nse(t0=0, tE=dt, Nts=1, start_ssstokes=True,
                         return_vp_dict=True, **sd)[0.0]
    ref = osnu.solve_nse(t0=0, tE=nsteps*dt, Nts=nsteps, iniv=v0d['v'],
                         inip=v0d['p'], return_final_vp=True, **sd)
    for nb in (1, 64):
        integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv,
                               femp['dbcinds'], femp['dbcvals'], dt,
                               nus=np.ones(nb), fv=rhsd['fv'], fp=rhsd['fp'],
                               coarse_max=200)
        assert integ.infos[0]['schur_levels'] >= 2
        integ.set_state(v0d['v'][inv], v0d['p'])
        integ.run(nsteps, tol=1e-12)
        V, P = integ.state()
        integ.close()
        for m in (0, nb - 1):
            assert _rel(V[:, m:m+1], ref[0]) < 1e-8, (nb, m)
            assert _rel(P[:, m:m+1], ref[1]) < 1e-8, (nb, m)


@pytest.fixture
def staged_ctx():
    """a context with the TMA-staged SpMM forced on for every matrix size
    (DNSB_TMA_MIN_ROWS is read when a context is created)"""
    import os
    from dolfin_navier_scipy_b200 import _lib
    old = os.environ.get('DNSB_TMA_MIN_ROWS')
    os.environ['DNSB_TMA_MIN_ROWS'] = '0'
    yield _lib.Context(0)
    os.environ['DNSB_TMA_MIN_ROWS'] = old if old is not None else '65536'
    _lib.Context(0)
    if old is None:
        del os.environ['DNSB_TMA_MIN_ROWS']


@pytest.mark.parametrize('nb', [1, 2])
def test_staged_spmv_matches_scipy(cyl1, staged_ctx, nb):
    """k_spmv_tma (bulk-copy staged row tiles, nb = 1; nb = 2 checks that the
    dispatch leaves the other widths alone): operators of the mesh, two value
    arrays, alpha/beta, a row count that is not a tile multiple"""
    femp, sm, rhsd = cyl1
    from dolfin_navier_scipy_b200.time_int_utils import _on_pattern, _union_pattern
    ctx = staged_ctx
    M, A = sps.csr_matrix(sm['M']), sps.csr_matrix(sm['A'])
    assert A.shape[0] % 128 != 0
    rng = np.random.default_rng(100 + nb)
    X = rng.standard_normal((A.shape[1], nb))
    Y0 = rng.standard_normal((A.shape[0], nb))
    Y = ctx.csr(A).spmm(X, alpha=-.5, beta=2., y=Y0)
    assert _rel(Y, -.5*(A@X) + 2*Y0) < 1e-14
    pat = _union_pattern([M, A])
    Mp, Ap = _on_pattern(M, pat), _on_pattern(A, pat)
    coef = rng.standard_normal(nb)
    Y = ctx.csr(Mp, Ap.data).spmm(X, coef=coef)
    for k in range(nb):
        assert _rel(Y[:, k], M@X[:, k] + coef[k]*(A@X[:, k])) < 1e-13
    J = sps.csr_matrix(sm['J'])
    assert _rel(ctx.csr(J).spmm(X), J@X) < 1e-14
    # more tiles than CTAs: every stage of the ring is reused
    big = sps.block_diag([A]*4, format='csr')
    assert big.shape[0] > 148*128
    Xb = rng.standard_normal((big.shape[1], nb))
    assert _rel(ctx.csr(big).spmm(Xb), big@Xb) < 1e-14


def test_staged_spmv_ragged_rows(staged_ctx):
    """empty rows, an empty leading tile, one long row, a single row"""
    ctx = staged_ctx
    rng = np.random.default_rng(7)
    n = 1000
    R = sps.random(n, 300, density=.03, random_state=3, format='lil')
    R[0:200, :] = 0
    R[555, :] = rng.standard_normal(300)
    R[700:720, :] = 0
    R = sps.csr_matrix(R)
    R.eliminate_zeros()
    for nb in (1, 1, 4):
        X = rng.standard_normal((300, nb))
        assert _rel(ctx.csr(R).spmm(X), R@X) < 1e-14
    one = sps.csr_matrix(rng.standard_normal((1, 300)))
    x = rng.standard_normal(300)
    assert _rel(ctx.csr(one).spmm(x), one@x) < 1e-14


def test_schur_tf32_variant_meets_the_fp64_tolerance(cyl1):
    """DNSB_SCHUR_TF32=1: the dense Schur block of the preconditioner applied
    in 3xTF32 (fp32 copy of the inverse).  FGMRES is flexible and keeps its
    residuals in fp64: same solution to the same tolerance, iteration count
    within one of the fp64 preconditioner."""
    import os
    from dolfin_navier_scipy_b200 import _lib, lin_alg_utils as lau
    from oracle.lau import solve_sadpnt_smw as olu
    femp, sm, rhsd = cyl1
    dt = 1./512
    F = (sm['M'] + .5*dt*sm['A']).tocsr()
    ncols = 64
    rng = np.random.default_rng(11)
    b = sm['M']@rng.standard_normal((F.shape[0], ncols))
    g = sm['J']@rng.standard_normal((F.shape[0], ncols))*1e-3
    ref = olu(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b, rhsp=g)
    NV = F.shape[0]
    its = {}
    try:
        for flag in ('0', '1'):
            os.environ['DNSB_SCHUR_TF32'] = flag
            ctx = _lib.Context(0)
            op = lau.SadpntOperator(F, sm['J'], sm['JT'], ncols=ncols, ctx=ctx)
            vp = op.solve(b, g, tol=1e-12, maxit=200)
            its[flag] = op.last_iters.copy()
            for k in range(ncols):
                assert _rel(vp[:NV, k], ref[:NV, k]) < 1e-9, (flag, k)
                assert _rel(vp[NV:, k], ref[NV:, k]) < 1e-8, (flag, k)
            op.close()
    finally:
        os.environ['DNSB_SCHUR_TF32'] = '0'
        _lib.Context(0)
        del os.environ['DNSB_SCHUR_TF32']
    assert abs(int(np.max(its['1'])) - int(np.max(its['0']))) <= 1, its


def test_tma_gram_schmidt_is_bit_identical(cyl1):
    """k_gs_tma (basis vectors streamed through a shared-memory ring by bulk
    copies) keeps the thread mapping and summation order of the
    register-pipelined kernels: same iteration counts, bit-identical solution"""
    import os
    from dolfin_navier_scipy_b200 import _lib, lin_alg_utils as lau
    femp, sm, rhsd = cyl1
    dt = 1./512
    F = (sm['M'] + .5*dt*sm['A']).tocsr()
    ncols = 64
    rng = np.random.default_rng(12)
    b = sm['M']@rng.standard_normal((F.shape[0], ncols))
    g = sm['J']@rng.standard_normal((F.shape[0], ncols))*1e-3
    out = {}
    try:
        for flag in ('0', '1'):
            os.environ['DNSB_GS_TMA'] = flag
            ctx = _lib.Context(0)
            op = lau.SadpntOperator(F, sm['J'], sm['JT'], ncols=ncols, ctx=ctx)
            vp = op.solve(b, g, tol=1e-12, maxit=200)
            out[flag] = (vp.copy(), op.last_iters.copy())
            op.close()
    finally:
        os.environ['DNSB_GS_TMA'] = '1'
        _lib.Context(0)
        del os.environ['DNSB_GS_TMA']
    assert np.array_equal(out['0'][1], out['1'][1])
    assert np.array_equal(out['0'][0], out['1'][0])


@pytest.mark.parametrize('symm', [True, False])
def test_device_assembly_of_the_constant_operators(ctx, symm):
    """SURVEY 8f-1: M, A, J, JT, MP assembled on the device (per-cell kernel +
    gather into fixed patterns) against the host assembly of the FEM shim
    (`dts:236-275`), cylinder mesh and a unit square"""
    from dolfin_navier_scipy_b200 import fem, dolfin_to_sparrays as dts
    for mesh in (fem.load_mesh('cylinder_1'), fem.unit_square_mesh(5, 3)):
        V, Q = fem.VectorP2Space(mesh), fem.P1Space(mesh)
        host = fem.assemble_stokes_operators(V, Q, nu=.37, gradvsymmtrc=symm)
        from dolfin_navier_scipy_b200 import _lib
        dev = _lib.device_for(V, ctx).assemble_stokes(Q, nu=.37,
                                                      gradvsymmtrc=symm)
        for key in ('M', 'A', 'J', 'JT', 'MP'):
            h, d = host[key].tocsr(), dev[key].tocsr()
            assert h.shape == d.shape
            diff = abs(h - d)
            assert diff.max() <= 1e-13*abs(h).max(), key
    # through the reference-facing function, outflow correction included
    mesh = fem.load_mesh('cylinder_1')
    V, Q = fem.VectorP2Space(mesh), fem.P1Space(mesh)
    mask = np.zeros(mesh.bnd_edge.shape[0], dtype=bool)
    mask[::7] = True
    a = dts.get_stokessysmats(V, Q, nu=1e-2, gradvsymmtrc=symm, outflowds=mask)
    b = dts.get_stokessysmats(V, Q, nu=1e-2, gradvsymmtrc=symm, outflowds=mask,
                              device=True)
    for key in ('M', 'A', 'J', 'JT', 'MP'):
        assert abs(a[key] - b[key]).max() <= 1e-13*abs(a[key]).max(), key


def test_paraviewoutput_of_the_solvers(cyl1, cyl1_re30, ctx, tmp_path):
    """`paraviewoutput=True` (`snu:817-821,1091-1098`, `snu:348-357`) writes
    `<prfx>__timestep.pvd` / `__steadystates.pvd` without dolfin; the last
    piece holds the returned velocity"""
    import xml.etree.ElementTree as ET
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = cyl1
    V, Q = femp['V'], femp['Q']

    def _last_piece(pvd, name, ncomp):
        sets = ET.parse(pvd).getroot().find('Collection').findall('DataSet')
        root = ET.parse(os.path.join(os.path.dirname(pvd), sets[-1].get('file'))).getroot()
        arr = [a for a in root.iter('DataArray') if a.get('Name') == name][0]
        return len(sets), np.array(arr.text.split(), dtype=float).reshape(-1, ncomp)

    vprfx, pprfx = str(tmp_path / 'v'), str(tmp_path / 'p')
    vfin, pfin = snu.solve_nse(t0=0., tE=4./512, Nts=4, start_ssstokes=True, return_final_vp=True,
                               paraviewoutput=True, vfileprfx=vprfx, pfileprfx=pprfx, verbose=False,
                               Q=Q, **soldict(femp, sm, rhsd))
    nsets, v = _last_piece(vprfx + '__timestep.pvd', 'v', 3)
    assert nsets == 5
    vfull = np.asarray(vfin).reshape(-1)
    if vfull.size != V.dim():
        vfull = dts_full(vfull, femp)
    assert np.allclose(v[:, 0], vfull[0::2], rtol=0, atol=1e-15)
    assert np.allclose(v[:, 1], vfull[1::2], rtol=0, atol=1e-15)
    _, p = _last_piece(pprfx + '__timestep.pvd', 'p', 1)
    assert np.allclose(p[:, 0], np.asarray(pfin).reshape(-1), rtol=0, atol=1e-15)
    # steady solver: Stokes + 1 Picard + 1 Newton iterate
    sprfx = str(tmp_path / 's')
    vss = snu.solve_steadystate_nse(vel_pcrd_stps=1, vel_nwtn_stps=1, vel_nwtn_tol=1., verbose=False,
                                    paraviewoutput=True, vfileprfx=sprfx, pfileprfx=sprfx + 'p', Q=Q,
                                    **soldict(*cyl1_re30))
    nsets, v = _last_piece(sprfx + '__steadystates.pvd', 'v', 3)
    assert nsets == 3
    assert np.allclose(v[:, 0], np.asarray(vss).reshape(-1)[0::2], rtol=0, atol=1e-15)


def dts_full(vinner, femp):
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    return dts.append_bcs_vec(vinner, V=femp['V'], invinds=femp['invinds'], bcinds=femp['dbcinds'],
                              bcvals=femp['dbcvals']).reshape(-1)


def test_imex_residual_of_an_ab2_step(cyl1, ctx):
    """`residual_checks.get_imex_res` (`rck:59-103`) on a device CNAB run: the
    Crank-Nicolson/AB2 residual of the third state vanishes on the inner dofs
    (`tests/test_units_residuals.py:117-134`)"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from dolfin_navier_scipy_b200 import residual_checks as rck
    femp, sm, rhsd = cyl1
    dt = 1./512
    vpd = snu.solve_nse(t0=0., tE=2*dt, Nts=2, start_ssstokes=True, return_vp_dict=True, verbose=False,
                        **soldict(femp, sm, rhsd))
    ts = sorted(vpd.keys())
    assert len(ts) == 3
    v0, vm, vE = (vpd[t]['v'] for t in ts)
    crnires = rck.get_imex_res(V=femp['V'], nu=femp['nu'], gradvsymmtrc=True, outflowds=femp.get('outflowds'),
                               explscheme='abtw')
    res = crnires(vE, vpd[ts[2]]['p'], dt, lastvel=vm, othervel=v0)
    inv = np.asarray(femp['invinds'])
    scale = np.linalg.norm((sm['Mfull']@(vE - vm).reshape(-1))[inv])/dt
    assert np.linalg.norm(res[inv]) < 1e-8*scale
    # tested with a single basis function: the scalar form of the same residual
    phi = np.zeros(femp['V'].dim())
    phi[inv[7]] = 1.
    assert crnires(vE, vpd[ts[2]]['p'], dt, lastvel=vm, othervel=v0, phi=phi) == pytest.approx(res[inv[7]])


# ---------------------------------------------------------------------------
# reference-RUN fixtures (tests/golden/ref_*.npz: outputs of the reference's
# own code, written by tests/golden/make_reference_golden.py)
# ---------------------------------------------------------------------------
def _dfg_lvl1():
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    return dnsps.get_sysmats(
        problem='gen_bccont', nu=1e-3, charvel=.2, scheme='TH', mergerhs=True,
        meshparams=dict(strtomeshfile='mesh/karman2D-rotcyl_lvl1.xml.gz',
                        movingwallcntrl=False,
                        strtophysicalregions='mesh/karman2D-rotcyl_lvl1_'
                        'facet_region.xml.gz',
                        strtobcsobs='mesh/karman2D-rotcyl-bm_geo_cntrlbc.json'))


@pytest.mark.parametrize('scheme', ['cnab', 'sbdf2'])
def test_reference_run_imex_device(cyl1, ctx, scheme):
    """`snu.solve_nse` -> `tiu.cnab` / `tiu.sbdftwo` as run by the reference
    itself: v and p at the start-up, Heun, first multistep and later steps"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = cyl1
    g = np.load(os.path.join(GOLD, 'ref_%s_cyl1_re60.npz' % scheme))
    got = snu.solve_nse(t0=0., tE=16./512, Nts=16, start_ssstokes=True,
                        return_vp_dict=True, time_int_scheme=scheme,
                        **soldict(femp, sm, rhsd))
    for j, t in enumerate(g['t']):
        assert _rel(got[float(t)]['v'], g['v'][:, j:j+1]) < 1e-8, (scheme, t)
        assert _rel(got[float(t)]['p'], g['p'][:, j:j+1]) < 1e-8, (scheme, t)


def test_reference_run_robin_control_ensemble_device(ctx):
    """cfg 5 on cylinder_1 against the reference's own runs of
    `tests/time_dep_nse_bcrob.py:26-34` (A + Arob/alpha, sin(t)(B1-B2)/alpha)
    for Re = 60, 105, 150: the three trajectories as ONE batched ensemble"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    g = np.load(os.path.join(GOLD, 'ref_bcrob_cyl1.npz'))
    nsteps, dt = 16, 1./512
    integ, info = ens.cylinder_ensemble(N=1, Res=(60., 150.), nmembers=3,
                                        dt=dt, ntimes=nsteps + 1, ctx=ctx)
    assert np.allclose(info['Re'], g['Re'])
    inv = np.asarray(info['femp']['invinds'])
    # the reference starts every member from its own Stokes state; state at t1
    # (first fixture column) is the earliest one stored for all members, so
    # start from the stored initial values of a separate oracle-free source:
    # the fixture of step 1 cannot seed a multistep run -- solve the Stokes
    # problems on the device instead (`start_ssstokes`, snu:903-908)
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    sm, femp = info['sm'], info['femp']
    v0 = np.zeros((info['NV'], 3))
    p0 = np.zeros((info['NP'], 3))
    for m, nu in enumerate(info['nus']):
        Am = (nu*sm['A'] + info['Arob']).tocsr()
        fvm = nu*info['B'][:, :1]
        vp = lau.solve_sadpnt_smw(amat=Am, jmat=sm['J'], jmatT=sm['JT'],
                                  rhsv=fvm, rhsp=info['fp'], krylov='gmres',
                                  vgroups=(inv//2, inv % 2),
                                  mass_diag=sm['M'].diagonal(),
                                  krpslvprms=dict(tol=1e-13, maxiter=2000))
        v0[:, m] = vp[:info['NV'], 0]
        p0[:, m:m+1] = snu.get_pfromv(
            v=v0[:, m:m+1], V=femp['V'], M=sm['M'], A=sm['M'], J=sm['J'],
            fv=fvm, fp=info['fp'], dbcinds=femp['dbcinds'],
            dbcvals=femp['dbcvals'], invinds=inv)
    integ.set_state(v0, p0)
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    integ.close()
    for j, k in enumerate(g['keep']):
        for m in range(3):
            assert _rel(vs[k, :, m], g['v'][inv, j, m]) < 1e-8, (k, m)
            assert _rel(ps[k, :, m], g['p'][:, j, m]) < 1e-8, (k, m)


def test_reference_run_newton_cn_device(ctx):
    """Picard + Newton sweeps with the trapezoidal rule as run by the
    reference (`snu:1304-1587`): velocity AND pressure of every step"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    g = np.load(os.path.join(GOLD, 'ref_newtoncn_cyl1_re100.npz'))
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=100,
                                       scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=1))
    sd = soldict(femp, sm, rhsd, t0=0., tE=6./512, Nts=6, start_ssstokes=True)
    traj = snu.solve_nse(return_dictofvelstrs=True, **sd)
    vd, pd = snu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                           vel_pcrd_stps=1, vel_nwtn_stps=2,
                           return_dictofvelstrs=True, return_dictofpstrs=True,
                           verbose=False, **sd)
    for k, t in enumerate(g['t']):
        assert _rel(vd[float(t)], g['v'][:, k:k+1]) < 1e-8, t
        assert _rel(pd[float(t)], g['p'][:, k:k+1]) < 1e-8, t


def test_reference_run_steady_state_device(cyl1_re30, ctx):
    """`snu.solve_steadystate_nse` (DFG 2D-1 and cylinder_1), `snu.get_pfromv`
    and `snu.get_v_conv_conts` as returned by the reference"""
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    g = np.load(os.path.join(GOLD, 'ref_dfg2d1_lvl1.npz'))
    femp, sm, rhsd = _dfg_lvl1()
    v, p = snu.solve_steadystate_nse(return_vp=True, verbose=False,
                                     **soldict(femp, sm, rhsd))
    assert _rel(v, g['v']) < 1e-8 and _rel(p, g['p']) < 1e-8
    femp, sm, rhsd = cyl1_re30
    g = np.load(os.path.join(GOLD, 'ref_steady_cyl1_re30.npz'))
    sd = soldict(femp, sm, rhsd)
    v, p = snu.solve_steadystate_nse(return_vp=True, verbose=False, **sd)
    assert _rel(v, g['v']) < 1e-8 and _rel(p, g['p']) < 1e-8
    inv = femp['invinds']
    pfv = snu.get_pfromv(v=g['v'][inv], V=femp['V'], M=sm['M'], A=sm['A'],
                         J=sm['J'], fv=rhsd['fv'], invinds=inv,
                         dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'])
    assert _rel(pfv, g['pfromv']) < 1e-8
    cm, rc, rbc = snu.get_v_conv_conts(
        vvec=g['v'], V=femp['V'], invinds=inv, dbcinds=femp['dbcinds'],
        dbcvals=femp['dbcvals'])
    assert _rel(cm@g['w'], g['newton_mat_w']) < 1e-12
    assert _rel(rc, g['newton_rhs_con']) < 1e-12
    assert _rel(rbc, g['newton_rhs_bc']) < 1e-12
    pm, none, pbc = snu.get_v_conv_conts(
        vvec=g['v'], V=femp['V'], invinds=inv, dbcinds=femp['dbcinds'],
        dbcvals=femp['dbcvals'], Picard=True)
    assert none is None
    assert _rel(pm@g['w'], g['picard_mat_w']) < 1e-12
    assert _rel(pbc, g['picard_rhs_bc']) < 1e-12


def test_reference_run_semi_implicit_euler_device(cyl1, ctx):
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = cyl1
    g = np.load(os.path.join(GOLD, 'ref_sie_cyl1_re60.npz'))
    trange = np.linspace(0., 12./512, 13)
    got = tiu.semi_implicit_euler(iniv=g['v'][:, :1], jmat=sm['J'],
                                  mmat=sm['M'], amat=sm['A'], trange=trange,
                                  fp=rhsd['fp'], V=femp['V'],
                                  invinds=femp['invinds'],
                                  dbcinds=femp['dbcinds'],
                                  dbcvals=femp['dbcvals'], fv=rhsd['fv'])
    for j, k in enumerate((0, 1, 6, 12)):
        assert _rel(got[k], g['v'][:, j:j+1]) < 1e-8, k


# ---------------------------------------------------------------------------
# the BENCHMARKED workload at its own size: cylinder_4 (28 970 + 3 836 DoFs)
# ---------------------------------------------------------------------------
def _bcrob_soldict(level, Re, palpha=1e-5):
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


def _oracle_member(args):
    level, Re, nsteps, dt = args
    from oracle import snu as osnu
    out = osnu.solve_nse(t0=0., tE=nsteps*dt, Nts=nsteps, start_ssstokes=True,
                         return_vp_dict=True, **_bcrob_soldict(level, Re))
    ts = sorted(out.keys())
    return (np.hstack([out[t]['v'] for t in ts]),
            np.hstack([out[t]['p'] for t in ts]))


def test_bench_workload_parity_per_step_cylinder4(ctx):
    """BASELINE config 5 as benchmarked: Robin-control ensemble on cylinder_4,
    8 members across Re 60..150, sin(t) control, CNAB dt = 1/2048, 16 steps.
    Velocity and pressure of EVERY step and member against the oracle's CNAB
    (`tiu:104-143` with `A + Arob/alpha`), rel. L2 error <= 1e-8; then the POD
    Gram matrix of the device (`dnsb_imex_gram`) against numpy."""
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, nsteps, dt = 8, 16, 1./2048
    integ, info = ens.cylinder_ensemble(N=4, Res=(60., 150.), nmembers=nb,
                                        dt=dt, ntimes=nsteps + 1, ctx=ctx)
    inv = np.asarray(info['femp']['invinds'])
    import multiprocessing as mp
    jobs = [(4, float(Re), nsteps, dt) for Re in info['Re']]
    with mp.get_context('spawn').Pool(min(nb, os.cpu_count() or 1)) as pool:
        ref = pool.map(_oracle_member, jobs)
    v0 = np.hstack([r[0][inv, :1] for r in ref])
    p0 = np.hstack([r[1][:, :1] for r in ref])
    integ.set_state(v0, p0)
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    st = integ.stats()
    assert st['max_relres'] <= 1e-12
    worst = 0.
    for k in range(1, nsteps + 1):
        for m in range(nb):
            ev = _rel(vs[k, :, m], ref[m][0][inv, k])
            ep = _rel(ps[k, :, m], ref[m][1][:, k])
            worst = max(worst, ev, ep)
            assert ev < 1e-8 and ep < 1e-8, (k, m, ev, ep)
    print('cylinder_4 ensemble: worst rel. error over steps/members', worst)
    # ---- POD snapshot Gram matrix G = sum_m X_m^T M X_m ----------------------
    G = integ.gram()
    M = info['sm']['M']
    Gn = np.zeros_like(G)
    for m in range(nb):
        X = vs[:, :, m].T
        Gn += X.T@(M@X)
    assert G.shape == (nsteps + 1, nsteps + 1)
    assert np.linalg.norm(G - Gn) <= 1e-12*np.linalg.norm(Gn)
    assert np.array_equal(G, integ.gram())          # deterministic
    integ.close()


def test_newton_cn_sweeps_cylinder4_with_pressure(ctx):
    """BASELINE config 3 on its own mesh: cylinder_4, Re = 100, Picard +
    Newton sweeps with Crank-Nicolson about the IMEX trajectory; velocity and
    pressure of every step against the oracle (`snu:1304-1587`)"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from oracle import snu as osnu
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=100,
                                       scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=4))
    nsteps = 4
    sd = soldict(femp, sm, rhsd, t0=0., tE=nsteps/2048., Nts=nsteps)
    o0 = osnu.solve_nse(start_ssstokes=True, return_vp_dict=True, **sd)
    t0 = sorted(o0.keys())[0]
    ini = dict(iniv=o0[t0]['v'], inip=o0[t0]['p'])
    otraj = {t: d['v'] for t, d in o0.items()}
    oref = osnu.solve_nse(lin_vel_point=otraj, treat_nonl_explicit=False,
                          vel_pcrd_stps=1, vel_nwtn_stps=1,
                          return_dictofvelstrs=True, **dict(sd, **ini))
    ovf, opf = osnu.solve_nse(lin_vel_point=otraj, treat_nonl_explicit=False,
                              vel_pcrd_stps=1, vel_nwtn_stps=1,
                              return_final_vp=True, **dict(sd, **ini))
    traj = snu.solve_nse(return_dictofvelstrs=True, **dict(sd, **ini))
    for t in sorted(otraj.keys()):
        assert _rel(traj[float(t)], otraj[t]) < 1e-8, t
    vd, pd = snu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                           vel_pcrd_stps=1, vel_nwtn_stps=1,
                           return_dictofvelstrs=True, return_dictofpstrs=True,
                           verbose=False, **dict(sd, **ini))
    for t in sorted(oref.keys()):
        assert _rel(vd[float(t)], oref[t]) < 1e-8, t
    tE = sorted(oref.keys())[-1]
    assert _rel(vd[float(tE)], ovf) < 1e-8
    assert _rel(pd[float(tE)], opf) < 1e-8


def test_unconverged_solves_are_reported(cyl1, ctx):
    """the FGMRES solve stands in for an exact sparse LU: stopping at `maxit`
    above `tol` must never pass silently (single solves, the IMEX loop, the
    Newton/CN sweep)"""
    from dolfin_navier_scipy_b200 import _lib, lin_alg_utils as lau
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = cyl1
    F = (sm['M'] + .5/512*sm['A']).tocsr()
    b = sm['M']@np.random.default_rng(8).standard_normal((F.shape[0], 1))
    op = lau.SadpntOperator(F, sm['J'], sm['JT'])
    with pytest.raises(_lib.NotConverged):
        op.solve(b, tol=1e-12, maxit=1)
    vp = op.solve(b, tol=1e-12, maxit=1, allow_unconverged=True)
    assert op.last_relres.max() > 1e-12 and np.all(np.isfinite(vp))
    op.solve(b, tol=1e-12, maxit=200)
    assert op.last_relres.max() <= 1e-12
    op.close()
    with pytest.raises(_lib.NotConverged):
        lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b,
                             krylov='gmres',
                             krpslvprms=dict(tol=1e-12, maxiter=1))
    # IMEX loop: guess=0 (previous solution) needs several iterations per step
    inv = femp['invinds']
    integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv,
                           femp['dbcinds'], femp['dbcvals'], 1./512,
                           fv=rhsd['fv'], fp=rhsd['fp'])
    integ.set_state(np.zeros((inv.size, 1)), np.zeros((sm['J'].shape[0], 1)))
    with pytest.raises(_lib.NotConverged):
        integ.run(4, tol=1e-12, maxit=1, guess=0)
    st = integ.stats()
    assert st['unconverged'] >= 1 and st['max_relres'] > 1e-12
    integ.run(4, tol=1e-12, maxit=1, guess=0, allow_unconverged=True)
    integ.run(4, tol=1e-12, maxit=200, guess=0)
    st = integ.stats()
    assert st['unconverged'] == 0 and 0 < st['max_relres'] <= 1e-12
    integ.close()


def test_steady_solver_outside_its_envelope_fails_loudly(cyl1, ctx):
    """cylinder_1 at Re = 60: the unstabilised Galerkin convection has element
    Peclet numbers (eigenvalues of D^-1 F at 0.8 +- 3i) on which the Jacobi-
    Chebyshev smoothed V-cycle is no contraction; the Oseen solve stagnates.
    The reference's sparse LU does not care -- the device path must say so
    instead of handing back an unconverged iterate (DESIGN.md section 4)."""
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = cyl1
    with pytest.raises(_lib.NotConverged):
        snu.solve_steadystate_nse(vel_pcrd_stps=1, vel_nwtn_stps=1,
                                  vel_nwtn_tol=1., verbose=False,
                                  **soldict(femp, sm, rhsd))


@pytest.fixture
def tc_ctx():
    """the tcgen05 Schur block (the default for nb >= 8) switched on explicitly"""
    return _ctx_with_env('DNSB_SCHUR_TC', '1')


@pytest.fixture
def f64_ctx():
    """every block of the preconditioner in fp64 (DNSB_SCHUR_TC=0)"""
    return _ctx_with_env('DNSB_SCHUR_TC', '0')


@pytest.mark.parametrize('ncols', [256, 128, 64, 24, 8])
def test_schur_tensor_core_block_against_numpy(cyl1, tc_ctx, ncols):
    """k_schur_tc (tcgen05.mma kind::tf32, TMA-fed, TMEM accumulators): the
    pressure part of one preconditioner application, z_p = -D r_p, against the
    fp64 product with the same inverse.  TF32 operands: rel. error of a few
    1e-4 (and NOT 1e-16: the fp64 path would hide a dispatch mistake)"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    femp, sm, rhsd = cyl1
    F = (sm['M'] + .5/512*sm['A']).tocsr()
    NP, NV = sm['J'].shape
    op = lau.SadpntOperator(F, sm['J'], sm['JT'], ncols=ncols, ctx=tc_ctx)
    levels, dense = op.info['hierarchy']
    assert len(levels) == 0 and dense.shape == (NP, NP) and NP % 128 != 0
    rng = np.random.default_rng(ncols)
    R = rng.standard_normal((NV + NP, ncols))
    Z = op.solver.apply_prec(R)
    ref = -dense@R[NV:]
    # forward error bound of a product with both operands rounded to TF32
    # (unit round-off 2^-11 each) and fp32 accumulation: |err| <= 2^-10 |D||x|
    bound = 2.**-10*(np.abs(dense)@np.abs(R[NV:]))
    for m in range(ncols):
        err = _rel(Z[NV:, m], ref[:, m])
        assert 1e-9 < err < 1e-2, (m, err)
        assert np.linalg.norm(Z[NV:, m] - ref[:, m]) <= np.linalg.norm(bound[:, m]), m
    # rows beyond a 128-row tile and K beyond a 32-column block are zero-filled
    # by TMA: a right-hand side concentrated on the last rows must come through
    R2 = np.zeros_like(R)
    R2[-3:, :] = rng.standard_normal((3, ncols))
    Z2 = op.solver.apply_prec(R2)
    ref2 = -dense@R2[NV:]
    assert _rel(Z2[NV:], ref2) < 1e-2
    op.close()


def test_schur_tensor_core_block_keeps_iterations_and_parity(cyl1, tc_ctx, f64_ctx):
    """the TF32 tensor-core block is a preconditioner detail: same FGMRES
    iteration counts (+-1), the solution meets the fp64 tolerance against LU,
    and a CNAB run stays within 1e-8 of the oracle per step"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle.lau import solve_sadpnt_smw as olu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    dt = 1./512
    F = (sm['M'] + .5*dt*sm['A']).tocsr()
    ncols = 64
    rng = np.random.default_rng(21)
    b = sm['M']@rng.standard_normal((F.shape[0], ncols))
    g = sm['J']@rng.standard_normal((F.shape[0], ncols))*1e-3
    ref = olu(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b, rhsp=g)
    NV = F.shape[0]
    its = {}
    for name, c in (('f64', f64_ctx), ('tc', tc_ctx)):
        op = lau.SadpntOperator(F, sm['J'], sm['JT'], ncols=ncols, ctx=c)
        vp = op.solve(b, g, tol=1e-12, maxit=200)
        its[name] = int(op.last_iters.max())
        for k in range(ncols):
            assert _rel(vp[:NV, k], ref[:NV, k]) < 1e-9, (name, k)
            assert _rel(vp[NV:, k], ref[NV:, k]) < 1e-8, (name, k)
        op.close()
    assert abs(its['tc'] - its['f64']) <= 1, its
    # CNAB, 3 members, per-step parity
    inv = femp['invinds']
    sd = soldict(femp, sm, rhsd)
    nsteps = 8
    o = osnu.solve_nse(t0=0, tE=nsteps*dt, Nts=nsteps, start_ssstokes=True,
                       return_vp_dict=True, **sd)
    ts = sorted(o.keys())
    integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv,
                           femp['dbcinds'], femp['dbcvals'], dt,
                           nus=np.ones(16), fv=rhsd['fv'], fp=rhsd['fp'],
                           ctx=tc_ctx)
    integ.set_state(o[ts[0]]['v'][inv], o[ts[0]]['p'])
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    integ.close()
    for k in range(1, nsteps + 1):
        for m in (0, 15):
            assert _rel(vs[k, :, m], o[ts[k]]['v'][inv, 0]) < 1e-8, (k, m)
            assert _rel(ps[k, :, m], o[ts[k]]['p'][:, 0]) < 1e-8, (k, m)


def test_tiled_chebyshev_is_bit_identical(cyl1):
    """k_cheb_step_tile (matrix entries, update operands and the unique x rows
    of a tile all staged by TMA bulk copies, gathers from shared memory) keeps
    the summation order of the row-pair kernel: a 64-member ensemble run is
    bit-identical with DNSB_TILE=0 and =1, iteration counts included"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    nu0 = femp['nu']
    A0 = sm['A']/nu0
    nus = nu0*np.linspace(.5, 2., 64)
    dt, nsteps = 1./512, 6
    v0 = osnu.solve_nse(t0=0, tE=dt, Nts=1, start_ssstokes=True,
                        return_vp_dict=True, **soldict(femp, sm, rhsd))[0.0]
    out = {}
    for flag in ('0', '1'):
        c = _ctx_with_env('DNSB_TILE', flag, DNSB_CHEB_F32='0')   # the fp64 tile kernel
        integ = tiu.DeviceImex(sm['M'], A0, sm['J'], femp['V'], inv,
                               femp['dbcinds'], femp['dbcvals'], dt, nus=nus,
                               fp=rhsd['fp'], ctx=c)
        U = np.broadcast_to((nus/nu0)[None, None, :], (nsteps + 1, 1, 64))
        integ.set_forcing(rhsd['fv'], U)
        integ.set_state(v0['v'][inv], v0['p'])
        integ.run(nsteps, tol=1e-12)
        out[flag] = integ.state() + (integ.stats()['iters'],)
        integ.close()
    assert out['0'][2] == out['1'][2]
    assert np.array_equal(out['0'][0], out['1'][0])
    assert np.array_equal(out['0'][1], out['1'][1])


# ---------------------------------------------------------------------------
# the reference's callback interface: per-step host hop, device solves
# ---------------------------------------------------------------------------
@pytest.mark.parametrize('scheme', ['cnab', 'sbdf2'])
def test_reference_run_callbacks_device(cyl1, ctx, scheme):
    """`tiu.cnab` / `tiu.sbdftwo` with a custom ``f_vdp``, ``f_tvdp(t, v)`` and
    an AB2 observer as ``dynamic_rhs`` against what the reference returned for
    the same callbacks (`tests/golden/ref_callbacks_cyl1_re60.npz`)"""
    import callback_cases as cbc
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = cyl1
    g = np.load(os.path.join(GOLD, 'ref_callbacks_cyl1_re60.npz'))
    inv = femp['invinds']

    def conv_inner(vfull):          # the device kernel K1a
        return dts.get_convvec(V=femp['V'], u0_vec=np.ravel(vfull), invinds=inv)
    kw = cbc.callback_kwargs(sm['M'], inv, conv_inner, tiu.get_heunab_lti,
                             inv.size)
    integ = dict(cnab=tiu.cnab, sbdf2=tiu.sbdftwo)[scheme]
    v, p, ff = integ(trange=g['t'], inivel=g['iniv'], inip=g['inip'],
                     M=sm['M'], A=sm['A'], J=sm['J'],
                     f_tdp=lambda t: rhsd['fv'], g_tdp=lambda t: rhsd['fp'],
                     scalep=-1.,
                     appndbcs=lambda vv, bcs: dts_full(vv, femp).reshape(-1, 1),
                     check_ff_maxv=1e8, **kw)
    assert ff == 0
    assert _rel(v, g['v_' + scheme]) < 1e-8
    assert _rel(p, g['p_' + scheme]) < 1e-8


def test_solve_nse_with_callbacks_and_output_feedback(cyl1, ctx):
    """`snu.solve_nse(fvtvd=, closed_loop=True, dynamic_feedback=True,
    dyn_fb_disc='AB2', b_mat=, cv_mat=)` (`snu:1129-1140,1224-1247`) routes
    through the host hop: equals a direct `tiu.cnab` call with the same
    callbacks, and `semi_implicit_euler` takes the reference's ``rhsv(t, v)``"""
    import callback_cases as cbc
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = cyl1
    g = np.load(os.path.join(GOLD, 'ref_callbacks_cyl1_re60.npz'))
    inv = femp['invinds']
    om = cbc.observer_matrices(inv.size, sm['M'])

    def fvtvd(t, vc):
        return .2*np.sin(40.*t)*(sm['M']@np.asarray(vc).reshape(-1, 1))
    trange = g['t'][:7]
    iniv_full = dts_full(g['iniv'], femp).reshape(-1, 1)
    v1, p1 = snu.solve_nse(
        trange=trange, iniv=iniv_full, inip=g['inip'], fvtvd=fvtvd,
        closed_loop=True, dynamic_feedback=True, dyn_fb_disc='AB2',
        dyn_fb_dict=dict(ha=om['ha'], hb=om['hb'], hc=om['hc'],
                         inihx=om['inihx'], drift=om['drift']),
        b_mat=om['bmat'], cv_mat=om['cmat'], return_final_vp=True,
        **soldict(femp, sm, rhsd))
    observer = tiu.get_heunab_lti(hb=om['hb'], ha=om['ha'], hc=om['hc'],
                                  inihx=om['inihx'], drift=om['drift'])

    def dynamic_rhs(t, vc=None, memory={}, mode=None):
        u, memory = observer(t, vc=om['cmat']@vc, memory=memory, mode=mode)
        return om['bmat']@u, memory
    v2, p2, _ = tiu.cnab(
        trange=trange, inivel=g['iniv'], inip=g['inip'], M=sm['M'], A=sm['A'],
        J=sm['J'], f_tdp=lambda t: rhsd['fv'], g_tdp=lambda t: rhsd['fp'],
        f_vdp=lambda vf: -dts.get_convvec(V=femp['V'], u0_vec=np.ravel(vf),
                                          invinds=inv),
        f_tvdp=fvtvd, dynamic_rhs=dynamic_rhs, dynamic_rhs_memory={},
        appndbcs=lambda vv, bcs: dts_full(vv, femp).reshape(-1, 1))
    assert _rel(v1, v2) < 1e-9 and _rel(p1, p2) < 1e-8
    # opaque rhsv(t, v) of `tiu.semi_implicit_euler` against the reference run
    gs = np.load(os.path.join(GOLD, 'ref_sie_cyl1_re60.npz'))

    def rhsv(t, v):
        return rhsd['fv'] - dts.get_convvec(
            V=femp['V'], u0_vec=dts_full(v, femp), invinds=inv)
    got = tiu.semi_implicit_euler(iniv=gs['v'][:, :1], jmat=sm['J'],
                                  mmat=sm['M'], amat=sm['A'], rhsv=rhsv,
                                  trange=np.linspace(0., 12./512, 13),
                                  fp=rhsd['fp'])
    for j, k in enumerate((0, 1, 6, 12)):
        assert _rel(got[k], gs['v'][:, j:j+1]) < 1e-8, k


def test_low_rank_update_and_krylovini(cyl1, ctx):
    """`lau.solve_sadpnt_smw(umat=, vmat=)` (Sherman-Morrison-Woodbury,
    `snu:1505-1512`) against a direct solve of the updated matrix, and the
    `krylovini` initial-guess modes of the Newton sweeps (`snu:1493-1503`)"""
    import scipy.sparse.linalg as spsla
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import stokes_navier_utils as snu
    femp, sm, rhsd = cyl1
    F = (sm['M'] + .5/512*sm['A']).tocsr()
    NP, NV = sm['J'].shape
    rng = np.random.default_rng(9)
    U = np.asarray(sm['M']@rng.standard_normal((NV, 3)))
    V = rng.standard_normal((3, NV))/NV
    b = np.asarray(sm['M']@rng.standard_normal((NV, 1)))
    got = lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=b,
                               umat=U, vmat=V)
    K = sps.bmat([[F + sps.csr_matrix(U@V), sm['J'].T], [sm['J'], None]],
                 format='csc')
    ref = spsla.spsolve(K, np.vstack([b, np.zeros((NP, 1))]).ravel())
    assert _rel(got[:NV, 0], ref[:NV]) < 1e-9
    assert _rel(got[NV:, 0], ref[NV:]) < 1e-8
    # krylovini: same sweep result, previous-solution guesses need more iterations
    femp, sm, rhsd = dnsps.get_sysmats(problem='cylinderwake', Re=100,
                                       scheme='TH', mergerhs=True,
                                       meshparams=dict(refinement_level=1))
    g = np.load(os.path.join(GOLD, 'ref_newtoncn_cyl1_re100.npz'))
    sd = soldict(femp, sm, rhsd, t0=0., tE=6./512, Nts=6, start_ssstokes=True)
    traj = snu.solve_nse(return_dictofvelstrs=True, **sd)
    its = {}
    for mode in ('old', 'upd'):
        st = []
        vd = snu.solve_nse(lin_vel_point=traj, treat_nonl_explicit=False,
                           vel_pcrd_stps=1, vel_nwtn_stps=2, verbose=False,
                           return_dictofvelstrs=True, krylov='Gmres',
                           krpslvprms=dict(krylovini=mode, convstatsl=st), **sd)
        its[mode] = np.mean(st)
        assert _rel(vd[float(g['t'][-1])], g['v'][:, -1:]) < 1e-8, mode
    assert its['upd'] < its['old']


def test_minres_on_the_symmetric_imex_matrix_matches_lu(cyl1, ctx):
    """`north_star` K3: MINRES for the symmetric saddle-point matrix of the IMEX
    schemes, with the device's preconditioner in its symmetric positive
    definite (block diagonal) form; products with K and the preconditioner
    run on the device, the three-term recurrence on the host.  Parity against
    the sparse LU (`oracle.lau`, what the reference calls) at 1e-9; a
    nonsymmetric block is refused"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from oracle import lau as olau
    femp, sm, rhsd = cyl1
    dt = 1./512
    F = (sm['M'] + .5*dt*sm['A']).tocsr()
    rng = np.random.default_rng(3)
    rhsv = sm['M']@rng.standard_normal((F.shape[0], 1)) + dt*rhsd['fv']
    rhsp = rhsd['fp']
    ref = olau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'],
                                rhsv=rhsv, rhsp=rhsp)
    st = []
    vp = lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=rhsv,
                              rhsp=rhsp, krylov='minres',
                              krpslvprms=dict(tol=1e-11, maxiter=600,
                                              convstatsl=st))
    nv = F.shape[0]
    assert _rel(vp[:nv], ref[:nv]) < 1e-9
    assert _rel(vp[nv:], ref[nv:]) < 1e-8
    assert 0 < st[0] < 300
    # the same system by the device FGMRES: fewer iterations (block triangular form)
    st2 = []
    lau.solve_sadpnt_smw(amat=F, jmat=sm['J'], jmatT=sm['JT'], rhsv=rhsv,
                         rhsp=rhsp, krylov='gmres',
                         krpslvprms=dict(tol=1e-11, maxiter=600,
                                         convstatsl=st2))
    assert st2[0] < st[0]
    with pytest.raises(ValueError):
        N1 = sps.random(nv, nv, 1e-3, random_state=1, format='csr')
        lau.solve_sadpnt_smw(amat=F + N1, jmat=sm['J'], jmatT=sm['JT'],
                             rhsv=rhsv, rhsp=rhsp, krylov='minres')


def test_switches_belong_to_their_context(cyl1, ctx):
    """the DNSB_* switches are read when a context is created and stay with
    it: a context made under DNSB_TILE=0 runs the row-pair kernels, the
    default context created before it keeps running the tile kernels, also
    when the two are used alternately in one process (the switch tests above
    rely on this)"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    other = _ctx_with_env('DNSB_TILE', '0')

    def kernels_of(c):
        integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv,
                               femp['dbcinds'], femp['dbcvals'], 1./512,
                               nus=np.ones(64), fv=rhsd['fv'], fp=rhsd['fp'],
                               ctx=c)
        integ.set_state(np.zeros((sm['M'].shape[0], 1)),
                        np.zeros((sm['J'].shape[0], 1)))
        c.profile_begin()
        integ.run(3, tol=1e-10)
        names = ' '.join(c.profile_end().keys())
        integ.close()
        return names
    for c, tiled in ((ctx, True), (other, False), (ctx, True), (other, False)):
        names = kernels_of(c)
        assert ('k_cheb_step_tile' in names) == tiled, names
        assert ('k_cheb_step_p2' in names) == (not tiled), names


def test_programmatic_launch_is_bitwise_reproducible():
    """kernels are launched with programmatic stream serialization (every
    kernel starts with `griddepcontrol.wait`; DNSB_PDL=1, default).  That only
    changes WHEN a kernel's CTAs become resident, never what it reads: a
    64-member run on the finest mesh (multi-wave grids, where launching the
    TMA-streamed Gram-Schmidt kernels this way was measured NOT to be
    reproducible -- they are excluded, DESIGN.md section 5) gives the same bits as
    plain stream order, three times over"""
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = dnsps.get_sysmats(
        problem='cylinderwake', Re=80., scheme='TH', mergerhs=True,
        meshparams=dict(refinement_level=4))
    inv = femp['invinds']
    nus = femp['nu']*np.linspace(.6, 1.6, 64)
    out = []
    for flag in ('0', '1', '1', '1'):
        c = _ctx_with_env('DNSB_PDL', flag)
        integ = tiu.DeviceImex(sm['M'], sm['A']/femp['nu'], sm['J'], femp['V'],
                               inv, femp['dbcinds'], femp['dbcvals'], 1./1024,
                               nus=nus, fv=rhsd['fv'], fp=rhsd['fp'], ctx=c)
        integ.set_state(np.zeros((sm['M'].shape[0], 1)),
                        np.zeros((sm['J'].shape[0], 1)))
        integ.run(30, tol=1e-12, guess=24)
        out.append(integ.state() + (integ.stats()['iters'],))
        integ.close()
    for v, p, its in out[1:]:
        assert its == out[0][2]
        assert np.array_equal(v, out[0][0])
        assert np.array_equal(p, out[0][1])


def test_projection_space_forms_agree_across_rebuilds(cyl1, ctx):
    """the recycled-solution space in its implicit form (raw directions + a
    triangular factor per member, DNSB_PROJ_T=1, default) against the explicit
    form (both sides orthogonalised): a short space (6 pairs, rebuilt from 3
    raw solutions every few steps) over 24 steps gives the same trajectory,
    the same iteration count within 10 %, and the LU oracle's states"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    dt, nsteps = 1./512, 24
    sd = soldict(femp, sm, rhsd)
    o = osnu.solve_nse(t0=0, tE=nsteps*dt, Nts=nsteps, start_ssstokes=True,
                       return_vp_dict=True, **sd)
    ts = sorted(o.keys())
    out = {}
    for label, c in (('implicit', ctx),
                     ('explicit', _ctx_with_env('DNSB_PROJ_T', '0'))):
        integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv,
                               femp['dbcinds'], femp['dbcvals'], dt,
                               nus=np.ones(64), fv=rhsd['fv'], fp=rhsd['fp'],
                               ctx=c)
        integ.set_state(o[ts[0]]['v'][inv], o[ts[0]]['p'])
        integ.run(nsteps, tol=1e-12, guess=6)
        out[label] = integ.state() + (integ.stats()['iters'],)
        integ.close()
    v, p, its = out['implicit']
    assert _rel(v, out['explicit'][0]) < 1e-9
    assert _rel(p, out['explicit'][1]) < 1e-9
    assert abs(its - out['explicit'][2]) <= 0.1*out['explicit'][2] + 1
    for m in (0, 63):
        assert _rel(v[:, m], o[ts[-1]]['v'][inv, 0]) < 1e-8
        assert _rel(p[:, m], o[ts[-1]]['p'][:, 0]) < 1e-8


@pytest.mark.parametrize('switch', ['DNSB_CONV_COLOURS=1', 'DNSB_GRAPHS=0',
                                    'DNSB_DMMA=0', 'DNSB_PAIR=0',
                                    'DNSB_ROWPAIR=0', 'DNSB_GS_TMA=0',
                                    'DNSB_TILE=0', 'DNSB_SCHUR_TC=0',
                                    'DNSB_GS_PYTH=0', 'DNSB_CHEB_F32=0',
                                    'DNSB_PROJ_T=0', 'DNSB_TAIL_WARPS=0',
                                    'DNSB_PDL=0', 'DNSB_INIT_TILE=0',
                                    'DNSB_TILEF_CTAS=1', 'DNSB_TILE_STAGES=2',
                                    'DNSB_TILE_STAGES_F=2', 'DNSB_TC_CTAS=2'])
def test_every_tuning_switch_gives_the_same_trajectory(cyl1, ctx, switch):
    """the environment switches select kernel VARIANTS of the same arithmetic
    (coloured scatter vs gather assembly -- the form `north_star` names --,
    graphs on/off, DFMA vs DMMA, member/row pairing, TMA staging, fp64 vs
    tensor-core Schur block): a 64-member CNAB run under each of them agrees
    with the default path to 1e-9 and with the LU oracle to 1e-8"""
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    from oracle import snu as osnu
    femp, sm, rhsd = cyl1
    inv = femp['invinds']
    dt, nsteps = 1./512, 5
    sd = soldict(femp, sm, rhsd)
    o = osnu.solve_nse(t0=0, tE=nsteps*dt, Nts=nsteps, start_ssstokes=True,
                       return_vp_dict=True, **sd)
    ts = sorted(o.keys())
    name, val = switch.split('=')
    out = {}
    for label, c in (('default', ctx), (switch, _ctx_with_env(name, val))):
        integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'], inv,
                               femp['dbcinds'], femp['dbcvals'], dt,
                               nus=np.ones(64), fv=rhsd['fv'], fp=rhsd['fp'],
                               ctx=c)
        integ.set_state(o[ts[0]]['v'][inv], o[ts[0]]['p'])
        integ.run(nsteps, tol=1e-12)
        out[label] = integ.state()
        integ.close()
    v, p = out[switch]
    assert _rel(v, out['default'][0]) < 1e-9
    assert _rel(p, out['default'][1]) < 1e-9
    for m in (0, 63):
        assert _rel(v[:, m], o[ts[-1]]['v'][inv, 0]) < 1e-8
        assert _rel(p[:, m], o[ts[-1]]['p'][:, 0]) < 1e-8
