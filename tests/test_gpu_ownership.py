"""Every handle frees what it allocated: create, use and destroy each handle
type and compare `dnsb_live_bytes` (the bytes of device and pinned host memory
the library holds in this process) with the value before, exactly.

A cycle runs twice and the baseline is taken after the first: the first run
lets the buffers a context keeps between calls (mesh data, element and staging
vectors) reach their size.  The free memory of the device is no measure here:
other processes share it."""
import numpy as np
import pytest
import scipy.sparse as sps

pytestmark = pytest.mark.gpu

DT = 1./512


@pytest.fixture(scope='module')
def ctx():
    from dolfin_navier_scipy_b200 import _lib
    c = _lib.Context(0)
    yield c
    c.close()


def _live():
    from dolfin_navier_scipy_b200 import _lib
    return _lib.live_bytes()


def _returns_to_baseline(cycle):
    """``cycle()`` creates handles, uses them, destroys them and returns what
    `_live` read while they were alive"""
    cycle()
    base = _live()
    alive = cycle()
    assert alive[0] > base[0], 'the handles held no device memory'
    assert _live() == base, (base, _live())
    return alive[1] - base[1]


def _close_solver(s):
    """a solver of `make_saddle_solver` and its matrices"""
    s.close()
    for m in s._keepalive:
        m.close()


def test_csr(ctx, cyl1):
    M = cyl1[1]['M']

    def cycle():
        m = ctx.csr(M, 2.*M.data)
        alive = _live()
        m.close()
        return alive
    _returns_to_baseline(cycle)


@pytest.mark.parametrize('nb', [1, 64])
def test_solver_with_schur_levels(ctx, cyl1, nb):
    """nb = 1: AMG Schur levels over a dense coarse inverse, solved twice (the
    second solve runs the captured Arnoldi graphs); nb = 64: the ensemble's
    tensor-core dense Schur level and tile plans"""
    from dolfin_navier_scipy_b200 import hostsetup
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    sm = cyl1[1]
    M, A, J = sps.csr_matrix(sm['M']), sps.csr_matrix(sm['A']), sm['J']
    if nb == 1:
        kw = dict(F1=(M + .5*DT*A).tocsr(), coarse_max=200)
    else:
        pat = tiu._union_pattern([M, A])
        JT = sps.csr_matrix(J.T)
        kw = dict(F1=tiu._on_pattern(M, pat), F2=tiu._on_pattern(A, pat),
                  coef=.5*DT*np.linspace(.5, 2., nb),
                  JT=tiu._on_pattern(JT, hostsetup.pad_row_pairs(JT)))
    rng = np.random.default_rng(nb)
    nv, np_ = M.shape[0], J.shape[0]
    names = {}

    def cycle():
        s, info = hostsetup.make_saddle_solver(ctx, J=J, nb=nb, restart=40,
                                               schur='lumped', **kw)
        if nb == 1:
            assert info['schur_levels'] > 1
            rhs = rng.standard_normal(nv)
            s.solve(rhs, tol=1e-10)
            s.solve(rhs, tol=1e-10)
        else:
            ctx.profile_begin()
            s.apply_prec(rng.standard_normal((nv + np_, nb)))
            names.update(ctx.profile_end())
        alive = _live()
        _close_solver(s)
        return alive
    pinned = _returns_to_baseline(cycle)
    assert pinned > 0               # the solver's flag word is pinned
    if nb == 64:
        assert '(k_schur_tc)' in names or 'k_schur_tc' in names, names


def test_failed_solver_create_leaves_nothing(ctx, cyl1):
    """nb = 8 reduces over 256-thread blocks: restart 120 exceeds the
    Gram-Schmidt shared memory, a check that runs after K, the Krylov bases
    and the Chebyshev vectors were allocated"""
    from dolfin_navier_scipy_b200 import _lib
    sm = cyl1[1]
    mats = [ctx.csr(sm['M']), ctx.csr(sm['J']), ctx.csr(sm['JT'])]
    try:
        for _ in range(2):
            base = _live()
            with pytest.raises(_lib.DnsbError,
                               match='Gram-Schmidt shared memory'):
                _lib.SaddleSolver(ctx, *mats, nb=8, restart=120,
                                  cheb_steps=2, lmin=.5, lmax=2.)
            assert _live() == base
    finally:
        for m in mats:
            m.close()


def test_imex_engine_with_snapshots_and_outputs(ctx):
    """the whole ensemble integrator (engine, its three solvers, matrices):
    a run with device snapshots, the pinned mirror, linear outputs and
    forces, then the Gram matrix"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    femp, sm = dnsps.get_sysmats(problem='cylinderwake', nu=1.,
                                 scheme='TH', bccontrol=True,
                                 meshparams=dict(refinement_level=1))[:2]
    NP, NV = sm['J'].shape
    Cv = sps.csr_matrix((np.ones(4), (np.arange(4), np.arange(0, NV, NV//4)[:4])),
                        shape=(4, NV))

    def cycle():
        integ, info = ens.cylinder_ensemble(N=1, nmembers=8, dt=DT, ntimes=16,
                                            ctx=ctx, force=True, cv_mat=Cv)
        integ.set_state(np.zeros((NV, 8)))
        integ.run(6, snap_stride=1, tol=1e-10)
        assert integ.snapshots()[0].shape[0] == 7
        assert integ.outputs()['y'].shape == (7, 4, 8)
        assert integ.gram().shape == (7, 7)
        alive = _live()
        integ.close()
        for s in integ.solvers:
            for m in s._keepalive:
                m.close()
        for m in (integ.mmat, integ.amat, integ.jmat, integ.jtmat):
            m.close()
        return alive
    pinned = _returns_to_baseline(cycle)
    assert pinned > 0               # the snapshot mirror is pinned


def test_cnsweep_after_a_sweep(ctx, cyl1):
    """the device Picard + Crank-Nicolson sweep as `solve_nse` builds it"""
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, rhsd = cyl1
    M, A, J = sps.csr_matrix(sm['M']), sps.csr_matrix(sm['A']), sm['J']
    V, invinds = femp['V'], np.asarray(femp['invinds'])
    nv, nvf = M.shape[0], V.dim()
    aux = dict(zip(map(int, femp['dbcinds']), femp['dbcvals']))
    bci = np.array(sorted(aux), dtype=np.int32)
    bcv = np.array([aux[i] for i in bci])
    ubc = np.zeros(nvf)
    ubc[bci] = bcv

    def cycle():
        dev = _lib.ConvDevice(V, ctx)
        cip, cix = dev.pattern
        Pc = sps.csr_matrix((np.arange(1, cix.size + 1, dtype=float), cix, cip),
                            shape=(nvf, nvf))[invinds, :][:, invinds].tocsr()
        Pc.sort_indices()
        pat = tiu._union_pattern([M, A, Pc])
        pos = tiu._on_pattern(sps.csr_matrix(
            (np.arange(1, Pc.nnz + 1, dtype=float), Pc.indices, Pc.indptr),
            shape=Pc.shape), pat)
        convpos = np.nonzero(pos.data)[0]
        Mv, Av = tiu._on_pattern(M, pat).data, tiu._on_pattern(A, pat).data
        op = lau.SadpntOperator(
            sps.csr_matrix((Mv + .5*DT*Av, pat.indices, pat.indptr),
                           shape=pat.shape), J, sm['JT'], ncols=1, ctx=ctx,
            velocity_amg=False, schur='lumped', cheb_steps=3)
        mmat = ctx.csr(M)
        sweep = _lib.CnSweep(op.solver, mmat, Mv, Av,
                             Pc.data.astype(np.int64) - 1, convpos, invinds,
                             bci, bcv, rhsd['fv'], rhsd['fp'], nvf)
        sweep.run(np.full(3, DT), np.tile(ubc, (4, 1)), np.zeros(nv), None,
                  True, tol=1e-10)
        alive = _live()
        sweep.close()
        mmat.close()
        _close_solver(op.solver)
        return alive
    _returns_to_baseline(cycle)


def test_second_context(cyl1):
    """a context with a mesh bound and its convection buffers in use"""
    from dolfin_navier_scipy_b200 import _lib
    V = cyl1[0]['V']
    u = np.random.default_rng(0).standard_normal(V.dim())

    def cycle():
        c = _lib.Context(0)
        _lib.ConvDevice(V, c).convvec(u)
        alive = _live()
        c.close()
        return alive
    _returns_to_baseline(cycle)
