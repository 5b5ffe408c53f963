"""Output functionals recorded inside the device time loop
(`DeviceImex.set_outputs`, `dnsb_imex_set_outputs` / `_set_force`): linear
outputs ``Cv v + Cp p`` and the CNAB drag/lift residual of every member at
every time level, against the snapshots of the same run and the host residual
`residual_checks.get_imex_res` evaluated on them."""
import numpy as np
import pytest
import scipy.sparse as sps

from kernel_refs import ctx_with_env as _ctx_with_env

pytestmark = pytest.mark.gpu

DT = 1./2048


@pytest.fixture(scope='module')
def ctx():
    from dolfin_navier_scipy_b200 import _lib
    return _lib.default_context(0)


def _initial_state(info, nb):
    """steady Stokes state of the mean viscosity, shared by the members"""
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    sm, inv = info['sm'], np.asarray(info['femp']['invinds'])
    numean = float(np.mean(info['nus']))
    Ast = numean*sm['A'] + info['Arob']
    vp = lau.solve_sadpnt_smw(amat=Ast, jmat=sm['J'], jmatT=sm['JT'],
                              rhsv=numean*info['B'][:, :1], rhsp=info['fp'],
                              krylov='gmres', vgroups=(inv//2, inv % 2),
                              mass_diag=sm['M'].diagonal(),
                              krpslvprms=dict(tol=1e-10, maxiter=1500))
    NV = info['NV']
    return np.repeat(vp[:NV], nb, axis=1), np.repeat(-vp[NV:], nb, axis=1)


def _probes(femp, NV, NP):
    """17 outputs: 16 velocity probes (one inner dof each, in the wake) and
    the pressure difference across the cylinder (front minus back node)"""
    V = femp['V']
    xy = np.asarray(V.tabulate_dof_coordinates())[np.asarray(femp['invinds'])]
    cand = np.flatnonzero((xy[:, 0] > 0.3) & (xy[:, 0] < 1.5) &
                          (np.abs(xy[:, 1] - 0.2) < 0.1))
    pick = cand[np.linspace(0, cand.size - 1, 16).astype(int)]
    Cv = sps.csr_matrix((np.ones(16), (np.arange(16), pick)), shape=(17, NV))
    pxy = np.asarray(V.mesh().coords)
    front = np.argmin(np.hypot(pxy[:, 0] - 0.15, pxy[:, 1] - 0.2))
    back = np.argmin(np.hypot(pxy[:, 0] - 0.25, pxy[:, 1] - 0.2))
    Cp = sps.csr_matrix(([1., -1.], ([16, 16], [front, back])),
                        shape=(17, NP))
    return Cv, Cp


def _ensemble(N, nb, ctx, nsteps=40, **kw):
    from dolfin_navier_scipy_b200 import ensemble as ens
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    femp_only = dnsps.get_sysmats(problem='cylinderwake', nu=1.,
                                  scheme='TH', bccontrol=True,
                                  meshparams=dict(refinement_level=N))
    NP, NV = femp_only[1]['J'].shape
    Cv, Cp = _probes(femp_only[0], NV, NP)
    integ, info = ens.cylinder_ensemble(N=N, nmembers=nb, dt=DT,
                                        ntimes=nsteps + 8, ctx=ctx, force=True,
                                        cv_mat=Cv, cp_mat=Cp, **kw)
    v0, p0 = _initial_state(info, nb)
    return integ, info, Cv, Cp, v0, p0


def _full(v, femp):
    aux = dict(zip(map(int, femp['dbcinds']), femp['dbcvals']))
    out = np.zeros(femp['V'].dim())
    out[np.asarray(femp['invinds'])] = v
    bci = np.array(sorted(aux))
    out[bci] = [aux[i] for i in bci]
    return out


def _check_y(y, vs, ps, Cv, Cp):
    ref = np.einsum('rk,lkm->lrm', Cv.toarray(), vs) + \
        np.einsum('rk,lkm->lrm', Cp.toarray(), ps)
    assert y.shape == ref.shape
    for r in range(ref.shape[1]):
        err = np.linalg.norm(y[:, r] - ref[:, r])
        assert err <= 1e-13*np.linalg.norm(ref[:, r]), (r, err)


def _check_force(force, vs, ps, info, levels):
    """F of every member at ``levels`` against `get_imex_res(nu=nu_m)` on the
    snapshots (Dirichlet values appended); returns the worst relative error"""
    from dolfin_navier_scipy_b200 import residual_checks as rck
    femp = info['femp']
    ld = np.asarray(femp['ldsbcinds'])
    phis = []
    for c in range(2):
        phi = np.zeros(femp['V'].dim())
        phi[ld[ld % 2 == c]] = 1.
        phis.append(phi)
    worst = 0.
    for m, nu in enumerate(info['nus']):
        res = rck.get_imex_res(V=femp['V'], nu=float(nu), implscheme='crni',
                               explscheme='abtw')
        full = {}

        def vf(n):
            if n not in full:
                full[n] = _full(vs[n, :, m], femp)
            return full[n]
        ref = np.zeros((len(levels), 2))
        for j, n in enumerate(levels):
            r = res(vf(n), ps[n, :, m], DT, vf(n - 1), vf(n - 2))
            ref[j] = [phis[0]@r, phis[1]@r]
        got = force[levels, :, m]
        scale = np.abs(ref).max()
        err = np.abs(got - ref).max()/scale
        assert err <= 1e-10, (m, err)
        worst = max(worst, err)
    return worst


@pytest.mark.parametrize('N,nb', [(1, 8), (4, 64)])
def test_outputs_match_snapshots_and_leave_the_trajectory(ctx, N, nb):
    """N = 1 / 8 members (row-pair kernels), N = 4 / 64 members (tile kernels,
    the benchmarked workload), 40 CNAB steps: y against ``Cv v + Cp p`` of the
    snapshots, the force against `get_imex_res` on them, NaN at levels 0 and
    1; the trajectory is the same bits with the outputs switched off"""
    nsteps = 40
    integ, info, Cv, Cp, v0, p0 = _ensemble(N, nb, ctx, nsteps)
    integ.set_state(v0, p0)
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    out = integ.outputs()
    assert out['y'].shape == (nsteps + 1, 17, nb)
    assert out['force'].shape == (nsteps + 1, 2, nb)
    _check_y(out['y'], vs, ps, Cv, Cp)
    assert np.isnan(out['force'][:2]).all()
    assert np.isfinite(out['force'][2:]).all()
    worst = _check_force(out['force'], vs, ps, info, list(range(2, nsteps + 1)))
    print('N={0} nb={1}: worst force error rel. to the member max {2:.2e}'.
          format(N, nb, worst))
    integ.close()
    # the same run by an integrator without outputs (a fresh one: a second run
    # of one integrator starts its solves from the last run's iteration count)
    from dolfin_navier_scipy_b200 import ensemble as ens
    plain, _ = ens.cylinder_ensemble(N=N, nmembers=nb, dt=DT,
                                     ntimes=nsteps + 8, ctx=ctx)
    plain.set_state(v0, p0)
    plain.run(nsteps, snap_stride=1, tol=1e-12)
    vs2, ps2 = plain.snapshots()
    assert plain.outputs()['force'].shape[0] == 0
    plain.close()
    assert np.array_equal(vs, vs2) and np.array_equal(ps, ps2)


def test_split_run_continues_the_record(ctx):
    """``run(20); run(20)``: 41 levels, the forces at the chunk boundary come
    from the convection term saved between the runs; ``set_state`` starts a
    new record"""
    integ, info, Cv, Cp, v0, p0 = _ensemble(1, 8, ctx, 40)
    integ.set_state(v0, p0)
    integ.run(20, snap_stride=1, tol=1e-12)
    integ.run(20, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    out = integ.outputs()
    assert out['y'].shape[0] == 41 and vs.shape[0] == 41
    assert np.isfinite(out['force'][2:]).all()
    _check_y(out['y'], vs, ps, Cv, Cp)
    _check_force(out['force'], vs, ps, info, [20, 21, 22, 40])
    integ.set_state(v0, p0)
    assert integ.outputs()['y'].shape[0] == 0
    integ.run(3, tol=1e-12)
    f = integ.outputs()['force']
    assert f.shape[0] == 4 and np.isnan(f[:2]).all() and np.isfinite(f[2:]).all()
    integ.reset_outputs()
    integ.run(2, tol=1e-12)
    f = integ.outputs()['force']
    assert f.shape[0] == 3 and np.isnan(f[0]).all() and np.isfinite(f[1:]).all()
    integ.close()


@pytest.mark.parametrize('switch', ['DNSB_CONV_COLOURS=1', 'DNSB_TILE=0',
                                    'DNSB_PDL=0'])
def test_outputs_under_switches_profiled_and_not(switch):
    """64 members on cylinder_1: the outputs of the coloured convection
    (`cfull` source), of the untiled kernels and of plain stream order meet
    the same checks against their own snapshots; the profile names the output
    kernel, and a profiled run gives the same bits"""
    name, val = switch.split('=')
    c = _ctx_with_env(name, val)
    nsteps = 12
    integ, info, Cv, Cp, v0, p0 = _ensemble(1, 64, c, nsteps)
    integ.set_state(v0, p0)
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    out = integ.outputs()
    _check_y(out['y'], vs, ps, Cv, Cp)
    _check_force(out['force'], vs, ps, info, list(range(2, nsteps + 1)))
    integ.close()
    again, _, _, _, _, _ = _ensemble(1, 64, c, nsteps)
    again.set_state(v0, p0)
    c.profile_begin()
    again.run(nsteps, tol=1e-12)
    prof = c.profile_end()
    assert prof['k_imex_outputs'][0] == nsteps + 2     # levels + Heun capture
    out2 = again.outputs()
    again.close()
    assert np.array_equal(out['y'], out2['y'])
    assert np.array_equal(out['force'], out2['force'], equal_nan=True)


@pytest.mark.parametrize('scheme', ['sbdf2', 'imexeuler'])
def test_linear_outputs_of_other_schemes_and_refusals(ctx, scheme):
    """SBDF2 / IMEX Euler record the linear outputs; a force request, wrong
    column counts and out-of-range force dofs raise before any device work"""
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import ensemble as ens
    from dolfin_navier_scipy_b200 import residual_checks as rck
    integ, info = ens.cylinder_ensemble(N=1, nmembers=4, dt=DT, ntimes=16,
                                        ctx=ctx, scheme=scheme)
    femp, sm = info['femp'], info['sm']
    NV, NP = info['NV'], info['NP']
    Cv, Cp = _probes(femp, NV, NP)
    ld = femp['ldsbcinds']
    with pytest.raises(NotImplementedError):
        integ.set_outputs(Cv, Cp, force_dofs=ld)
    with pytest.raises(ValueError):
        integ.set_outputs(sps.csr_matrix((2, NV + 1)))
    with pytest.raises(ValueError):
        integ.set_outputs(Cv, sps.csr_matrix((17, NP - 1)))
    # the C-ABI refuses the same on its own
    rows = rck.get_imex_force_rows(
        invinds=femp['invinds'], dbcinds=femp['dbcinds'],
        dbcvals=femp['dbcvals'], ldsbcinds=ld,
        force_ops=dict(M=sm['Mfull'], A=sm['Afull'], JT=sm['JTfull']))
    fm = ctx.csr(rows['fm'][:, integ.pv])
    fa = ctx.csr(rows['fa'][:, integ.pv])
    fj = ctx.csr(rows['fj'][:, integ.pp])
    bad = ctx.csr(sps.csr_matrix((3, NV + 2)))
    with pytest.raises(_lib.DnsbError):
        integ.engine.set_force(rows['dofs'], fm, fa, fj, fa_bc=rows['fa_bc'])
    with pytest.raises(_lib.DnsbError):
        integ.engine.set_outputs(bad)
    integ.set_outputs(Cv, Cp)
    v0, p0 = _initial_state(info, 4)
    integ.set_state(v0, p0)
    integ.run(10, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    out = integ.outputs()
    _check_y(out['y'], vs, ps, Cv, Cp)
    assert np.isnan(out['force']).all()
    integ.close()
    for m in (fm, fa, fj, bad):
        m.close()


def test_force_dofs_out_of_range_raise(ctx):
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import ensemble as ens
    integ, info = ens.cylinder_ensemble(N=1, nmembers=2, dt=DT, ntimes=8,
                                        ctx=ctx)
    femp, sm = info['femp'], info['sm']
    nvf = femp['V'].dim()
    with pytest.raises(ValueError):
        integ.set_outputs(force_dofs=[0, nvf])
    NV, NP = info['NV'], info['NP']
    z = ctx.csr(sps.csr_matrix((2, NV)))
    zp = ctx.csr(sps.csr_matrix((2, NP)))
    with pytest.raises(_lib.DnsbError):
        integ.engine.set_force([0, nvf], z, z, zp, fa_bc=np.zeros(2))
    with pytest.raises(_lib.DnsbError):
        integ.engine.set_force([-1], z, z, zp, fa_bc=np.zeros(2))
    integ.close()
    z.close()
    zp.close()
