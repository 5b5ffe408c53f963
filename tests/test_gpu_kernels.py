"""The 64-member operator kernels, one application at a time, against the fp64
restatements of `kernel_refs.py`.

The fp32 tile smoother (`k_cheb_init_tilef`, `k_cheb_step_tilef`) and the
tcgen05 Schur block (`k_tc_pack_x`, `k_schur_tc`, `k_tc_epilogue`) sit inside
the preconditioner of a flexible GMRES: an error there costs iterations, not
accuracy, so the trajectory tests cannot see it.  Here each reduced-precision
block is compared on its own, against a bound derived for it, member by member
and tile by tile, on the real operators of the ensemble (cylinder_1 and the
benchmarked cylinder_4), under every tuning switch, and on small synthetic
systems at the limits of the tile planner.  The profile names the kernels that
ran, so a silent fall-back fails too."""
import numpy as np
import pytest
import scipy.sparse as sps

import kernel_refs as kr

pytestmark = pytest.mark.gpu

NB = kr.TILE_NB
F32_TOL = 2e-6        # rel. L2 per member of the fp32 smoother (test_kernel_refs_cpu)
F64_TOL = 1e-13       # fp64 smoother, other summation order
K_TOL = 1e-14         # fp64 operator products


def _rel_cols(a, b):
    return np.linalg.norm(a - b, axis=0)/np.linalg.norm(b, axis=0)


def _names(prof):
    return {k.strip('()').replace(' ', '') for k in prof}


def _profiled(ctx, fn, *args):
    """(result, kernel names) of a profiled call, after checking that it is
    bit-identical to two unprofiled calls (the profile turns programmatic
    launch off) and that those two agree"""
    ctx.profile_begin()
    y0 = fn(*args)
    names = _names(ctx.profile_end())
    y1 = fn(*args)
    y2 = fn(*args)
    assert np.array_equal(y1, y2), 'two calls in a row differ'
    assert np.array_equal(y0, y1), 'profiled and unprofiled calls differ'
    return y0, names


def _close(s):
    """free a solver made by `make_saddle_solver` and its matrices"""
    s.close()
    for m in s._keepalive:
        m.close()


def _step_kernels(k, f32=True):
    base = 'k_cheb_step_tilef' if f32 else 'k_cheb_step_tile'
    return {'{0}<{1},{2}>'.format(base, str(i == 0).lower(),
                                  str(i + 2 == k).lower())
            for i in range(k - 1)}


def _check_tc(zp, ref, dense, rp):
    """TF32 operands (unit round-off 2^-11 each), fp32 accumulation:
    |err| <= 2^-10 |D||x| per member; and not fp64-exact"""
    bound = 2.**-10*(np.abs(dense)@np.abs(rp))
    err = _rel_cols(zp, ref)
    assert np.all(err > 1e-9) and np.all(err < 1e-2), err
    assert np.all(np.linalg.norm(zp - ref, axis=0) <=
                  np.linalg.norm(bound, axis=0))
    return float(err.max())


def _check_velocity(zv, ref, f32):
    """per member rel. L2 and, per tile of 8 row pairs and member, the max
    error against the member's max-norm: a single wrong row pair, tile or
    member lane fails locally"""
    err = _rel_cols(zv, ref)
    tol = F32_TOL if f32 else F64_TOL
    assert np.all(err <= tol), (err.max(), int(err.argmax()))
    if f32:
        assert np.all(err > 1e-10), 'the fp32 smoother did not run'
    n = zv.shape[0]
    pad = (-n) % 16
    e = np.abs(zv - ref)
    e = np.vstack([e, np.zeros((pad, e.shape[1]))]).reshape(-1, 16, e.shape[1])
    local = e.max(axis=1)/np.abs(ref).max(axis=0)[None, :]
    assert np.all(local <= tol), np.unravel_index(local.argmax(), local.shape)
    return float(err.max())


# ---------------------------------------------------------------------------
# the ensemble's own solvers
# ---------------------------------------------------------------------------
class _Ensemble(object):
    """`cylinder_ensemble(N, nmembers=64)` and, per solver (loop tau = dt/2,
    Heun predictor tau = dt, corrector tau = 0), the host operators it was
    built from"""

    def __init__(self, N):
        from dolfin_navier_scipy_b200 import ensemble as ens
        from dolfin_navier_scipy_b200 import time_int_utils as tiu
        self.N = N
        self.integ, _ = ens.cylinder_ensemble(N, nmembers=NB)
        integ = self.integ
        h = integ._host
        M, Ar = h['M'], h['Arob']
        self.J = h['J']
        self.JT = sps.csr_matrix(self.J.T)
        self.F2 = h['A0']
        theta = tiu._THETA[integ.scheme]
        self.cases = []
        for tau, s, info in zip((theta*integ.dt, integ.dt, 0.),
                                integ.solvers, integ.infos):
            F1 = sps.csr_matrix((M.data + tau*Ar.data, M.indices, M.indptr),
                                shape=M.shape)
            levels, dense = info['hierarchy']
            assert len(levels) == 0 and not info['velocity_amg']
            self.cases.append(dict(tau=tau, solver=s, info=info, F1=F1,
                                   coef=tau*integ.nus, dense=dense))

    def solver(self, case, k, ctx=None):
        """a further solver with ``k`` Chebyshev steps (the host set-up of
        the ensemble's solver is reused)"""
        from dolfin_navier_scipy_b200 import hostsetup
        from dolfin_navier_scipy_b200 import time_int_utils as tiu
        if ctx is None and k == 4:
            return case['solver'], False
        ctx = self.integ.ctx if ctx is None else ctx
        JT = tiu._on_pattern(self.JT, hostsetup.pad_row_pairs(self.JT))
        s, _ = hostsetup.make_saddle_solver(
            ctx, case['F1'], self.J, JT, F2=self.F2, coef=case['coef'], nb=NB,
            restart=40, cheb_steps=k, hierarchy=case['info']['hierarchy'],
            spectrum=case['info']['spectrum'], velocity_amg=False)
        return s, True

    def close(self):
        self.integ.close()


@pytest.fixture(scope='module')
def ensembles():
    built = {}

    def get(N):
        if N not in built:
            built[N] = _Ensemble(N)
        return built[N]
    yield get
    for e in built.values():
        e.close()


MESHES = [1, 4]


@pytest.mark.parametrize('N', MESHES)
def test_k_times_x_member_by_member(ensembles, N):
    """`apply_k` (k_spmm_tile<false> with the tail warps serving the
    divergence rows) against scipy per member, every solver"""
    e = ensembles(N)
    nv, np_ = e.F2.shape[0], e.J.shape[0]
    X = np.random.default_rng(N).standard_normal((nv + np_, NB))
    for c in e.cases:
        s = c['solver']
        Y, names = _profiled(s.ctx, s.apply_k, X)
        assert names == {'k_spmm_tile<false>'}, names
        ref = kr.apply_k(c['F1'], e.F2, c['coef'], e.J, e.JT, X)
        err = _rel_cols(Y, ref)
        print('cylinder_%d tau=%g K x: %.3g' % (N, c['tau'], err.max()))
        assert np.all(err <= K_TOL), (c['tau'], err.max())
        # the divergence rows (tail warps) on their own
        assert np.all(_rel_cols(Y[nv:], ref[nv:]) <= K_TOL), c['tau']
        # the last divergence row alone (a row the tail warps could skip)
        assert np.all(np.abs(Y[-1] - ref[-1]) <=
                      K_TOL*np.abs(e.J[-1]).sum()*np.abs(X[:nv]).max(axis=0))


@pytest.mark.parametrize('N', MESHES)
def test_f_times_x_with_beta(ensembles, N):
    """y = alpha F_m x + beta y through the solver's own F (k_spmm_tile<true>)"""
    e = ensembles(N)
    nv = e.F2.shape[0]
    rng = np.random.default_rng(10 + N)
    X, Y0 = rng.standard_normal((nv, NB)), rng.standard_normal((nv, NB))
    for c in e.cases:
        fmat = c['solver'].fmat
        Y, names = _profiled(fmat.ctx, lambda: fmat.spmm(X, coef=c['coef'],
                                                         alpha=-.75, beta=1.5,
                                                         y=Y0))
        assert names == {'k_spmm_tile<true>'}, names
        ref = -.75*(c['F1']@X + (e.F2@X)*c['coef'][None, :]) + 1.5*Y0
        assert np.all(_rel_cols(Y, ref) <= K_TOL), c['tau']


def _check_prec(s, F1, F2, coef, J, JT, dense, spectrum, k, rng, tc=True,
                f32=True):
    """one `apply_prec` against the restatement; returns (errors, kernels)"""
    nv, np_ = F1.shape[0], J.shape[0]
    R = rng.standard_normal((nv + np_, NB))
    Z, names = _profiled(s.ctx, s.apply_prec, R)
    zp, zv = Z[nv:], Z[:nv]
    ref_p = kr.prec_pressure(dense, R[nv:])
    if tc:
        ep = _check_tc(zp, ref_p, dense, R[nv:])
    else:
        ep = float(_rel_cols(zp, ref_p).max())
        assert ep <= F64_TOL, ep
    # the velocity part from the device's zp: no TF32 error leaks in
    lmin, lmax = spectrum
    ref_v = kr.cheb_batched(F1, F2, coef, R[:nv], k, lmin, lmax, JT=JT, zp=zp)
    ev = _check_velocity(zv, ref_v, f32 and k >= 2)
    return (ep, ev), names


@pytest.mark.parametrize('k', [1, 2, 3, 4, 5])
@pytest.mark.parametrize('N', MESHES)
def test_preconditioner_per_step_count(ensembles, N, k):
    """`apply_prec` with k Chebyshev steps on every solver of the ensemble:
    pressure part against -D rp within the TF32 bound, velocity part against
    the fp64 smoother fed with the device's pressure part (fp32 kernel: every
    FIRST/LAST instantiation; k = 1: the fp64 start alone)"""
    e = ensembles(N)
    rng = np.random.default_rng(100*N + k)
    for c in e.cases:
        s, own = e.solver(c, k)
        try:
            errs, names = _check_prec(s, c['F1'], e.F2, c['coef'], e.J,
                                      e.JT, c['dense'],
                                      c['info']['spectrum'], k, rng)
            print('cylinder_%d tau=%g k=%d: pressure %.3g, velocity %.3g'
                  % ((N, c['tau'], k) + errs))
        finally:
            if own:
                _close(s)
        want = {'k_tc_pack_x', 'k_schur_tc', 'k_tc_epilogue'}
        want |= {'k_cheb_init_tilef'} | _step_kernels(k) if k >= 2 \
            else {'k_cheb_init_p2'}
        assert names == want, (c['tau'], names)


def test_cylinder4_ends_on_a_partial_tile():
    """the tile kernels above ran on a plan whose last tile holds 5 pairs"""
    h = kr.device_numbering(4)
    for P in (h['M'], h['JT'], kr.block_k(h['M'], h['JT'], h['J'])):
        plan = kr.tile_plan(P)
        assert plan['ok'] and plan['last'] == 5


# ---------------------------------------------------------------------------
# every tuning switch at the operator level (cylinder_4, loop solver)
# ---------------------------------------------------------------------------
_DEFAULT = dict(init='k_cheb_init_tilef', f32=True, tile=True, tc=True,
                tail=True)
SWITCHES = {
    'DNSB_INIT_TILE=0': dict(init='k_cheb_init_p2f'),
    'DNSB_TILEF_CTAS=1': {},
    'DNSB_TILE_STAGES_F=2': {},
    'DNSB_TILE_STAGES_F=8': {},
    'DNSB_TILE_STAGES=2': {},
    'DNSB_CHEB_F32=0': dict(init='k_cheb_init_p2', f32=False),
    'DNSB_TILE=0': dict(init='k_cheb_init_p2', f32=False, tile=False),
    'DNSB_TAIL_WARPS=0': dict(tail=False),
    'DNSB_TAIL_WARPS=1': {},
    'DNSB_TAIL_WARPS=8': {},
    'DNSB_TC_CTAS=2': {},
    'DNSB_SCHUR_TC=0': dict(tc=False),
    'DNSB_PDL=0': {},
}


@pytest.mark.parametrize('switch', sorted(SWITCHES))
def test_every_switch_at_the_operator_level(ensembles, switch):
    """one context per setting: `apply_prec` (4 steps) and `apply_k` of the
    cylinder_4 loop solver against the restatement at the setting's own
    precision, and the setting's kernels in the profile"""
    e = ensembles(4)
    c = e.cases[0]
    name, val = switch.split('=')
    ctx = kr.ctx_with_env(name, val)
    x = dict(_DEFAULT, **SWITCHES[switch])
    s, _ = e.solver(c, 4, ctx=ctx)
    rng = np.random.default_rng(7)
    try:
        errs, names = _check_prec(s, c['F1'], e.F2, c['coef'], e.J, e.JT,
                                  c['dense'], c['info']['spectrum'], 4, rng,
                                  tc=x['tc'], f32=x['f32'])
        print('%s: pressure %.3g, velocity %.3g' % ((switch,) + errs))
        nv, np_ = e.F2.shape[0], e.J.shape[0]
        X = rng.standard_normal((nv + np_, NB))
        Y, knames = _profiled(ctx, s.apply_k, X)
        ref = kr.apply_k(c['F1'], e.F2, c['coef'], e.J, e.JT, X)
        assert np.all(_rel_cols(Y, ref) <= K_TOL)
    finally:
        _close(s)
        ctx.close()
    assert x['init'] in names, names
    if x['f32']:
        assert _step_kernels(4) <= names, names
    elif x['tile']:
        assert _step_kernels(4, f32=False) <= names, names
    else:
        assert any(n.startswith('k_cheb_step_p2<') for n in names), names
    assert ('k_schur_tc' in names) == x['tc'], names
    if not x['tc']:
        assert 'k_dense_dmma_streamk' in names, names
    if not x['tile']:
        assert knames == {'k_spmm_k2<true>'}, knames
    elif x['tail']:
        assert knames == {'k_spmm_tile<false>'}, knames
    else:
        assert knames == {'k_spmm_tile<false>', 'k_spmm_b2<true>'}, knames


# ---------------------------------------------------------------------------
# synthetic systems at the limits of the tile planner
# ---------------------------------------------------------------------------
SYN_SPECTRUM = (.3, 2.)      # D^-1 F of a diagonally dominant F: (0, 2)


@pytest.mark.parametrize('name', sorted(kr.SYNTHETIC))
def test_synthetic_tile_edges(name):
    """nb = 64 with per-member coefficients straight through
    `_lib.SaddleSolver`: K x, F x with beta, and the preconditioner (3 steps)
    against the restatement; the kernels that ran are the ones the planner's
    restatement predicts (tile kernels, or the row-pair fall-back)"""
    from dolfin_navier_scipy_b200 import _lib
    kw, _ = kr.SYNTHETIC[name]
    F1, F2, J, JT = kr.paired_system(**kw)
    pf, pj = kr.tile_plan(F1), kr.tile_plan(JT)
    pk = kr.tile_plan(kr.block_k(F1, JT, J))
    nv, np_ = F1.shape[0], J.shape[0]
    rng = np.random.default_rng(len(name))
    coef = np.linspace(0., 1., NB)
    dense = rng.standard_normal((np_, np_))/np.sqrt(np_)
    ctx = _lib.default_context()
    fmat, jmat, jtmat = ctx.csr(F1, F2.data), ctx.csr(J), ctx.csr(JT)
    s = _lib.SaddleSolver(ctx, fmat, jmat, jtmat, coef=coef, nb=NB, restart=4,
                          cheb_steps=3, lmin=SYN_SPECTRUM[0],
                          lmax=SYN_SPECTRUM[1])
    try:
        s.add_schur_level(dense_inv=dense)
        errs, names = _check_prec(s, F1, F2, coef, J, JT, dense,
                                  SYN_SPECTRUM, 3, rng, tc=np_ >= 128,
                                  f32=pf['ok'])
        print('%s: pressure %.3g, velocity %.3g' % ((name,) + errs))
        X = rng.standard_normal((nv + np_, NB))
        Y, knames = _profiled(ctx, s.apply_k, X)
        assert np.all(_rel_cols(Y, kr.apply_k(F1, F2, coef, J, JT, X)) <=
                      K_TOL)
        Xv, Y0 = X[:nv], rng.standard_normal((nv, NB))
        Yf, fnames = _profiled(ctx, lambda: fmat.spmm(Xv, coef=coef,
                                                      alpha=2., beta=-1.,
                                                      y=Y0))
        ref = 2.*(F1@Xv + (F2@Xv)*coef[None, :]) - Y0
        assert np.all(_rel_cols(Yf, ref) <= K_TOL)
    finally:
        s.close()
        for m in (fmat, jmat, jtmat):
            m.close()
    if pf['ok']:
        assert _step_kernels(3) <= names, names
        assert ('k_cheb_init_tilef' if pj['ok'] else 'k_cheb_init_p2f') \
            in names, names
        assert fnames == {'k_spmm_tile<true>'}, fnames
    else:
        assert 'k_cheb_step_p2<true,true,false>' in names, names
        assert 'k_cheb_init_p2' in names, names
        assert fnames == {'k_spmm_p2<true>'}, fnames
    if pk['ok']:
        assert knames == {'k_spmm_tile<false>'}, knames
    else:
        assert knames == {'k_spmm_k2<true>'}, knames


# ---------------------------------------------------------------------------
# tensor-core Schur block with an arbitrary inverse
# ---------------------------------------------------------------------------
@pytest.fixture(scope='module')
def tc_ctxs():
    out = {n: kr.ctx_with_env('DNSB_TC_CTAS', str(n)) for n in (1, 2)}
    yield out
    for c in out.values():
        c.close()


def _schur_solver(ctx, np_, nb, dense, mass=None):
    from dolfin_navier_scipy_b200 import _lib
    F1, F2, J, JT = kr.paired_system(24, np_=np_, seed=np_)
    mats = [ctx.csr(F1, F2.data), ctx.csr(J), ctx.csr(JT)]
    s = _lib.SaddleSolver(ctx, *mats, coef=np.linspace(0., 1., nb), nb=nb,
                          restart=4, cheb_steps=2, lmin=SYN_SPECTRUM[0],
                          lmax=SYN_SPECTRUM[1])
    s.add_schur_level(dense_inv=dense)
    if mass is not None:
        s.set_schur_mass(*mass)
    return s, mats, F1.shape[0]


def _schur_apply(ctx, np_, nb, dense, rp, mass=None):
    s, mats, nv = _schur_solver(ctx, np_, nb, dense, mass)
    R = np.zeros((nv + np_, nb))
    R[nv:] = rp
    try:
        Z, names = _profiled(ctx, s.apply_prec, R)
    finally:
        s.close()
        for m in mats:
            m.close()
    return Z[nv:], names


TC_NAMES = {'k_tc_pack_x', 'k_schur_tc', 'k_tc_epilogue'}


@pytest.mark.parametrize('ctas', [1, 2])
@pytest.mark.parametrize('np_', [127, 128, 129, 160, 3836])
def test_schur_block_sizes(tc_ctxs, np_, ctas):
    """the 128-row threshold of the tensor-core block: 127 rows go to the
    fp64 kernels (no k_schur_tc, fp64-tight), from 128 on the TF32 bound"""
    rng = np.random.default_rng(np_)
    dense = rng.standard_normal((np_, np_))/np.sqrt(np_)
    rp = rng.standard_normal((np_, NB))
    zp, names = _schur_apply(tc_ctxs[ctas], np_, NB, dense, rp)
    ref = -dense@rp
    if np_ < 128:
        assert not names & TC_NAMES, names
        assert np.all(_rel_cols(zp, ref) <= 1e-14)
    else:
        assert TC_NAMES <= names, names
        _check_tc(zp, ref, dense, rp)


@pytest.mark.parametrize('ctas', [1, 2])
@pytest.mark.parametrize('nb', [8, 16, 24, 40, 64, 128, 256])
def test_schur_block_batch_widths(tc_ctxs, nb, ctas):
    """members padded to 16 columns, TMEM allocations of 32 to 256 columns"""
    np_ = 160
    rng = np.random.default_rng(nb)
    dense = rng.standard_normal((np_, np_))/np.sqrt(np_)
    rp = rng.standard_normal((np_, nb))
    zp, names = _schur_apply(tc_ctxs[ctas], np_, nb, dense, rp)
    assert TC_NAMES <= names, names
    _check_tc(zp, -dense@rp, dense, rp)


STRUCT = [(160, 64), (129, 256), (3836, 40)]


@pytest.mark.parametrize('ctas', [1, 2])
@pytest.mark.parametrize('np_,nb', STRUCT)
def test_schur_block_identity_and_permutation(tc_ctxs, np_, nb, ctas):
    """D = I gives -tf32(float(rp)) bit for bit; a permutation D moves every
    row and member to exactly where it belongs"""
    rng = np.random.default_rng(np_ + nb)
    rp = rng.standard_normal((np_, nb))
    want = -kr.tf32(rp).astype(np.float64)
    zp, names = _schur_apply(tc_ctxs[ctas], np_, nb, np.eye(np_), rp)
    assert TC_NAMES <= names, names
    assert np.array_equal(zp, want)
    perm = rng.permutation(np_)
    zp, _ = _schur_apply(tc_ctxs[ctas], np_, nb, np.eye(np_)[perm], rp)
    assert np.array_equal(zp, want[perm])


@pytest.mark.parametrize('ctas', [1, 2])
@pytest.mark.parametrize('np_,nb', STRUCT)
def test_schur_block_mass_term(tc_ctxs, np_, nb, ctas):
    """D = 0 with the Cahouet-Chabard mass term: what remains is the fp64 term
    k_tc_epilogue adds, zp = -scale_m mp_dinv_i rp (FMA contraction may move
    the last bit)"""
    rng = np.random.default_rng(3*np_ + nb)
    rp = rng.standard_normal((np_, nb))
    mp_dinv = rng.uniform(.5, 2., np_)
    scale = rng.uniform(.1, 1., nb)
    zp, names = _schur_apply(tc_ctxs[ctas], np_, nb, np.zeros((np_, np_)), rp,
                             mass=(mp_dinv, scale))
    assert TC_NAMES <= names, names
    ref = kr.prec_pressure(np.zeros((np_, np_)), rp, mp_dinv=mp_dinv,
                           mp_scale=scale)
    assert np.all(_rel_cols(zp, ref) <= 1e-15)
    assert np.all(np.abs(zp - ref) <= 1e-15*np.abs(ref))
