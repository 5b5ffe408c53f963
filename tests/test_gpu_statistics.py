"""Field statistics accumulated inside the device time loop
(`DeviceImex.set_statistics`, `dnsb_imex_set_statistics`): means and second
moments of every member against numpy over the snapshots of the same run, the
mean convection against the oracle's convection of each snapshot, the
window's continuation across runs, the per-member guard, and the summed CNAB
step equations of the mean flow."""
import numpy as np
import pytest

from kernel_refs import ctx_with_env as _ctx_with_env

pytestmark = pytest.mark.gpu

DT = 1./2048
FIELDS = ('v_mean', 'uu', 'vv', 'uv', 'p_mean', 'p_var', 'c_mean')


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


def _full_levels(vs, femp):
    """(levels, NVf, nb) full velocities of the snapshots (Dirichlet values
    set)"""
    aux = dict(zip(map(int, femp['dbcinds']), femp['dbcvals']))
    bci = np.array(sorted(aux))
    out = np.zeros((vs.shape[0], femp['V'].dim(), vs.shape[2]))
    out[:, np.asarray(femp['invinds'])] = vs
    out[:, bci] = np.array([aux[i] for i in bci])[None, :, None]
    return out


class _Conv(object):
    """oracle convection c(V)[invinds] of full velocities, member by member"""

    def __init__(self, femp):
        from oracle.cconv import CConv
        self.cc = CConv(femp['V'])
        self.inv = np.asarray(femp['invinds'])

    def __call__(self, vfull):          # (NVf, nb) -> (NV, nb)
        return np.stack([self.cc.convvec(vfull[:, m])[self.inv]
                         for m in range(vfull.shape[1])], axis=1)


def _numpy_stats(vf, ps, cs):
    """the statistics over the given levels: vf (L, NVf), ps (L, NP),
    cs (L, NV) of one member"""
    u, v = vf[:, 0::2], vf[:, 1::2]
    du, dv = u - u.mean(0), v - v.mean(0)
    return dict(v_mean=vf.mean(0), uu=(du*du).mean(0), vv=(dv*dv).mean(0),
                uv=(du*dv).mean(0), p_mean=ps.mean(0), p_var=ps.var(0),
                c_mean=cs.mean(0))


def _check(st, vf, ps, cs, levels, members=None, tol=1e-12):
    """every field of the members against numpy over ``levels`` (a list per
    member, or one list for all); returns the worst relative error"""
    nb = vf.shape[2]
    worst = 0.
    for m in range(nb) if members is None else members:
        lv = levels[m] if isinstance(levels, dict) else levels
        assert st['count'][m] == len(lv)
        ref = _numpy_stats(vf[lv, :, m], ps[lv, :, m], cs[lv, :, m])
        for key in FIELDS:
            scale = max(np.abs(ref[key]).max(), 1e-300)
            err = np.abs(st[key][:, m] - ref[key]).max()/scale
            assert err <= tol, (m, key, err)
            worst = max(worst, err)
    return worst


def _conv_levels(conv, vf):
    return np.stack([conv(vf[n]) for n in range(vf.shape[0])])


@pytest.mark.parametrize('N,nb,nsteps', [(1, 8, 40), (4, 64, 24)])
def test_statistics_match_numpy_and_leave_the_trajectory(ctx, N, nb, nsteps):
    """N = 1 / 8 members (row-pair kernels), N = 4 / 64 members (tile kernels,
    the benchmarked workload), CNAB, every level from 0 to the last against
    numpy over the snapshots and the oracle convection of each; the
    trajectory, the snapshots and the output record are the same bits with
    the statistics off"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    integ, info = ens.cylinder_ensemble(N=N, nmembers=nb, dt=DT,
                                        ntimes=nsteps + 8, ctx=ctx, force=True,
                                        statistics=True)
    v0, p0 = _initial_state(info, nb)
    integ.set_state(v0, p0)
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    st = integ.statistics()
    out = integ.outputs()
    state = integ.state()
    integ.close()
    assert st['first_level'] == 0 and st['last_level'] == nsteps
    femp = info['femp']
    vf = _full_levels(vs, femp)
    cs = _conv_levels(_Conv(femp), vf)
    worst = _check(st, vf, ps, cs, list(range(nsteps + 1)))
    print('N={0} nb={1}: worst error rel. to the member max {2:.2e}'.format(
        N, nb, worst))
    plain, _ = ens.cylinder_ensemble(N=N, nmembers=nb, dt=DT,
                                     ntimes=nsteps + 8, ctx=ctx, force=True)
    plain.set_state(v0, p0)
    plain.run(nsteps, snap_stride=1, tol=1e-12)
    vs2, ps2 = plain.snapshots()
    out2 = plain.outputs()
    state2 = plain.state()
    plain.close()
    assert np.array_equal(vs, vs2) and np.array_equal(ps, ps2)
    assert np.array_equal(state[0], state2[0])
    assert np.array_equal(state[1], state2[1])
    assert np.array_equal(out['force'], out2['force'], equal_nan=True)


def _same_bits(a, b):
    for key in FIELDS + ('count',):
        assert np.array_equal(a[key], b[key], equal_nan=True), key


def test_split_reset_and_set_state(ctx):
    """``run(20); run(20)`` gives the bits of one 40-step run;
    `reset_statistics` after 10 steps gives the statistics of levels 10..40;
    `set_state` restarts the window at level 0"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, nsteps = 8, 40
    runs = {}
    for split in ('one', 'two', 'reset'):
        integ, info = ens.cylinder_ensemble(N=1, nmembers=nb, dt=DT,
                                            ntimes=nsteps + 8, ctx=ctx,
                                            statistics=True)
        v0, p0 = _initial_state(info, nb)
        integ.set_state(v0, p0)
        if split == 'one':
            integ.run(nsteps, snap_stride=1, tol=1e-12)
        elif split == 'two':
            integ.run(20, snap_stride=1, tol=1e-12)
            st20 = integ.statistics()
            assert st20['last_level'] == 20
            integ.run(20, snap_stride=1, tol=1e-12)
        else:
            integ.run(10, snap_stride=1, tol=1e-12)
            integ.reset_statistics()
            st = integ.statistics()
            assert st['first_level'] == 10 and st['last_level'] == 9
            assert (st['count'] == 0).all() and np.isnan(st['v_mean']).all()
            integ.run(30, snap_stride=1, tol=1e-12)
        runs[split] = (integ.statistics(), integ.snapshots())
        if split == 'reset':
            integ.set_state(v0, p0)
            st = integ.statistics()
            assert st['first_level'] == 0 and st['last_level'] == -1
            integ.run(3, snap_stride=1, tol=1e-12)
            st = integ.statistics()
            assert st['first_level'] == 0 and st['last_level'] == 3
            assert (st['count'] == 4).all()
        integ.close()
    femp = info['femp']
    (s1, (vs1, ps1)), (s2, (vs2, ps2)) = runs['one'], runs['two']
    assert np.array_equal(vs1, vs2) and np.array_equal(ps1, ps2)
    _same_bits(s1, s2)
    sr, (vs, ps) = runs['reset']
    assert sr['first_level'] == 10 and sr['last_level'] == 40
    vf = _full_levels(vs, femp)
    cs = _conv_levels(_Conv(femp), vf[10:])
    lv = list(range(10, 41))
    full_cs = np.zeros((41,) + cs.shape[1:])
    full_cs[10:] = cs
    _check(sr, vf, ps, full_cs, lv)


@pytest.mark.parametrize('scheme', ['sbdf2', 'imexeuler'])
def test_other_schemes_against_numpy(ctx, scheme):
    """SBDF2 (Heun levels 0 and 1 included) and IMEX Euler on cylinder_1"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, nsteps = 4, 16
    integ, info = ens.cylinder_ensemble(N=1, nmembers=nb, dt=DT,
                                        ntimes=nsteps + 8, ctx=ctx,
                                        scheme=scheme, statistics=True)
    integ.set_state(*_initial_state(info, nb))
    integ.run(nsteps, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    st = integ.statistics()
    integ.close()
    femp = info['femp']
    vf = _full_levels(vs, femp)
    _check(st, vf, ps, _conv_levels(_Conv(femp), vf), list(range(nsteps + 1)))


def test_member_guard_counts_and_fields(ctx):
    """a threshold that retires some members mid-run: a retired member counts
    its levels up to its trip level and its fields are numpy's over them; a
    member retired before a reset window has count 0 and NaN fields"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, nsteps = 8, 41
    kw = dict(N=1, nmembers=nb, dt=DT, ntimes=nsteps + 16, ctx=ctx)
    plain, info = ens.cylinder_ensemble(**kw)
    v0, p0 = _initial_state(info, nb)
    plain.set_state(v0, p0)
    plain.run(nsteps, snap_stride=1, tol=1e-12)
    vs, _ = plain.snapshots()
    plain.close()
    # the guard checks every level 1..41 (40 slices of one step + the
    # remainder); a threshold halfway between two norms of the unguarded run
    nrm = np.linalg.norm(vs[1:], axis=1)                    # (41, nb)
    cand = np.unique(nrm)
    pick = None
    for c in 0.5*(cand[1:] + cand[:-1]):
        over = nrm > c
        trips = np.where(over.any(0), over.argmax(0) + 1, -1)
        if 2 <= (trips >= 0).sum() <= nb - 2 and (trips > 2).any() and \
                np.min(np.abs(nrm - c)) > 1e-9*c:
            pick = c
            break
    assert pick is not None
    integ, _ = ens.cylinder_ensemble(member_guard=True, statistics=True, **kw)
    integ.set_state(v0, p0)
    assert integ.run(nsteps, snap_stride=1, tol=1e-12, check_ff_maxv=pick,
                     ntimeslices=nsteps - 1) == 1
    trip = integ.member_status()['trip_level']
    print('member guard: threshold {0:.6g}, trips {1}'.format(pick, trip))
    assert (trip >= 0).any() and (trip < 0).any()
    vs, ps = integ.snapshots()
    st = integ.statistics()
    femp = info['femp']
    vf = _full_levels(vs, femp)
    conv = _Conv(femp)
    cs = np.stack([conv(np.nan_to_num(vf[n])) for n in range(nsteps + 1)])
    levels = {m: list(range((trip[m] if trip[m] >= 0 else nsteps) + 1))
              for m in range(nb)}
    _check(st, vf, ps, cs, levels)
    # a window that starts after the trips: the retired members have none
    integ.reset_statistics()
    integ.run(4, tol=1e-12, check_ff_maxv=1e300, ntimeslices=4)
    st = integ.statistics()
    assert st['first_level'] == nsteps
    want = np.where(trip < 0, 5, np.clip(trip - nsteps + 1, 0, 5))
    assert np.array_equal(st['count'], want)
    dead = want == 0
    assert dead.any()
    for key in FIELDS:
        assert np.isnan(st[key][:, dead]).all(), key
        assert np.isfinite(st[key][:, ~dead]).all(), key
    integ.close()


def test_mean_flow_identity(ctx):
    """CNAB, window a..b with a >= 1: the step equations summed over
    n = a+1..b,
      M (V_b - V_a)/dt + A_m (sum V - (V_a + V_b)/2)
      + sum c - c_b + (c_{b-1} - c_{a-1})/2 - J^T sum_{a+1..b} p = sum f,
    evaluated with the device statistics (sum c from `mean_flow_forcing` and
    c(v_mean)), the end snapshots and the forcing"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb, a, b = 8, 6, 40
    integ, info = ens.cylinder_ensemble(N=1, nmembers=nb, dt=DT,
                                        ntimes=b + 8, ctx=ctx, statistics=True)
    integ.set_state(*_initial_state(info, nb))
    integ.run(a, snap_stride=1, tol=1e-12)
    integ.reset_statistics()
    integ.run(b - a, snap_stride=1, tol=1e-12)
    vs, ps = integ.snapshots()
    st = integ.statistics()
    fm = integ.mean_flow_forcing(st)
    integ.close()
    assert st['first_level'] == a and st['last_level'] == b
    femp, sm = info['femp'], info['sm']
    inv = np.asarray(femp['invinds'])
    vf = _full_levels(vs, femp)
    conv = _Conv(femp)
    cnt = b - a + 1
    cbar = conv(st['v_mean'])
    sum_c = cnt*(fm + cbar)
    sum_v = cnt*st['v_mean'][inv]
    sum_p = cnt*st['p_mean'] - ps[a]
    c_b, c_b1, c_a1 = conv(vf[b]), conv(vf[b - 1]), conv(vf[a - 1])
    B, U = info['B'], info['U']
    sum_f = sum(B@(0.5*(U[n - 1] + U[n])) for n in range(a + 1, b + 1))
    M, J = sm['M'], sm['J']
    for m, nu in enumerate(info['nus']):
        Am = nu*sm['A'] + info['Arob']
        terms = [M@(vs[b, :, m] - vs[a, :, m])/DT,
                 Am@(sum_v[:, m] - 0.5*(vs[a, :, m] + vs[b, :, m])),
                 sum_c[:, m] - c_b[:, m] + 0.5*(c_b1[:, m] - c_a1[:, m]),
                 -(J.T@sum_p[:, m]), -sum_f[:, m]]
        res = np.linalg.norm(sum(terms))
        scale = sum(np.linalg.norm(t) for t in terms)
        print('member {0}: identity residual {1:.2e} of {2:.2e}'.format(
            m, res, scale))
        assert res <= 1e-9*scale, (m, res, scale)


@pytest.mark.parametrize('switch', ['DNSB_CONV_COLOURS=1', 'DNSB_TILE=0',
                                    'DNSB_PDL=0'])
def test_statistics_under_switches_profiled_and_not(ctx, switch):
    """64 members on cylinder_1: the statistics under each switch meet the
    numpy checks and are the bits of the default path where the trajectory
    is; the profile names the kernel once per level, a profiled run gives the
    same bits, and with the statistics off no such kernel runs"""
    from dolfin_navier_scipy_b200 import ensemble as ens
    name, val = switch.split('=')
    c = _ctx_with_env(name, val)
    nb, nsteps = 64, 12
    kw = dict(N=1, nmembers=nb, dt=DT, ntimes=nsteps + 8)
    res = {}
    for key, cx, prof in (('default', ctx, False), ('switch', c, False),
                          ('profiled', c, True), ('off', c, True)):
        integ, info = ens.cylinder_ensemble(ctx=cx, statistics=key != 'off',
                                            **kw)
        integ.set_state(*_initial_state(info, nb))
        if prof:
            cx.profile_begin()
        integ.run(nsteps, snap_stride=1, tol=1e-12)
        p = cx.profile_end() if prof else None
        st = integ.statistics() if key != 'off' else None
        res[key] = (st, integ.snapshots(), p)
        integ.close()
    names = [k for k in res['profiled'][2] if k.startswith('k_imex_stats')]
    assert sum(res['profiled'][2][k][0] for k in names) == nsteps + 1
    assert not [k for k in res['off'][2] if k.startswith('k_imex_stats')]
    _same_bits(res['switch'][0], res['profiled'][0])
    st, (vs, ps), _ = res['switch']
    femp = info['femp']
    vf = _full_levels(vs, femp)
    _check(st, vf, ps, _conv_levels(_Conv(femp), vf), list(range(nsteps + 1)))
    (vd, pd) = res['default'][1]
    if np.array_equal(vs, vd) and np.array_equal(ps, pd):
        _same_bits(st, res['default'][0])


def test_ownership_and_refusals(ctx):
    """the accumulators are the integrator's: switching the statistics off
    frees exactly their bytes, and create / run / off / on / destroy returns
    `dnsb_live_bytes` to its baseline (taken after a first cycle, which sizes
    the buffers the context keeps); get / reset before set and null handles
    are refused"""
    import ctypes
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import ensemble as ens
    nb = 4
    lib = ctx.lib
    assert lib.dnsb_imex_set_statistics(None, 1) == -2
    assert lib.dnsb_imex_reset_statistics(None) == -2
    assert lib.dnsb_imex_get_statistics(None, None, None, None, None, None,
                                        None, None, None) == -2

    def cycle():
        integ, info = ens.cylinder_ensemble(N=1, nmembers=nb, dt=DT,
                                            ntimes=16, ctx=ctx)
        with pytest.raises(_lib.DnsbError):
            integ.statistics()
        with pytest.raises(_lib.DnsbError):
            integ.reset_statistics()
        integ.set_state(np.zeros((info['NV'], nb)))
        integ.set_statistics(True)
        integ.run(5, tol=1e-12)
        assert (integ.statistics()['count'] == 6).all()
        first = ctypes.c_longlong(-7)
        assert lib.dnsb_imex_get_statistics(
            integ.engine.h, ctypes.byref(first), None, None, None, None, None,
            None, None) == 0
        assert first.value == 0
        on = _lib.live_bytes()
        integ.set_statistics(False)
        nvf, NV, NP = integ.dev.nvf, info['NV'], info['NP']
        assert on[0] - _lib.live_bytes()[0] == \
            8*nb*(nvf + 3*(nvf//2) + 2*NP + NV)
        with pytest.raises(_lib.DnsbError):
            integ.statistics()
        integ.set_statistics(True)
        integ.run(2, tol=1e-12)
        assert integ.statistics()['first_level'] == 5
        alive = _lib.live_bytes()
        integ.close()
        for s in integ.solvers:
            for m in s._keepalive:
                m.close()
        for m in (integ.mmat, integ.amat, integ.jmat, integ.jtmat):
            m.close()
        return alive
    cycle()
    base = _lib.live_bytes()
    alive = cycle()
    assert alive[0] > base[0]
    assert _lib.live_bytes() == base
