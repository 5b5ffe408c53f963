"""CPU pins of the restatements in `kernel_refs.py` that the kernel tests
(`test_gpu_kernels.py`) compare the 64-member CUDA kernels with: the
Chebyshev restatement against its closed form, the float32 emulation against
the tolerance the kernel tests use, and the synthetic systems against the
planner edges they are built to reach."""
import numpy as np
import pytest
import scipy.sparse as sps

import kernel_refs as kr

# relative L2 error per member the fp32 smoother is allowed (test_gpu_kernels)
F32_TOL = 2e-6


@pytest.mark.parametrize('k', [1, 2, 3, 4, 5])
def test_chebyshev_restatement_against_closed_form(k):
    """z = V diag((1 - P_k(l))/l) V^-1 D^-1 r with the Chebyshev residual
    polynomial P_k(l) = T_k((th - l)/de)/T_k(th/de) of D^-1 F"""
    rng = np.random.default_rng(k)
    n = 40
    B = rng.standard_normal((n, n))
    F = B@B.T + n*np.eye(n)
    dinv = 1./np.diag(F)
    lam, V = np.linalg.eig(dinv[:, None]*F)
    lam, V = lam.real, V.real
    lmin, lmax = .9*lam.min(), 1.05*lam.max()
    th, de = .5*(lmax + lmin), .5*(lmax - lmin)

    def T(x):
        return np.cosh(k*np.arccosh(x)) if np.all(x >= 1) else \
            np.cos(k*np.arccos(np.clip(x, -1, 1)))
    Pk = np.cos(k*np.arccos((th - lam)/de))/T(np.array(th/de))
    r = rng.standard_normal(n)
    ref = V@(((1. - Pk)/lam)*np.linalg.solve(V, dinv*r))
    z = kr.cheb_np(sps.csr_matrix(F), dinv, r, k, lmin, lmax)
    assert np.linalg.norm(z - ref) <= 1e-12*np.linalg.norm(ref)
    # the batched restatement is the same thing member by member
    F2 = sps.csr_matrix(F)
    coef = np.array([0., .5])
    zb = kr.cheb_batched(sps.csr_matrix(F), F2, coef, np.stack([r, r], 1), k,
                         lmin, lmax)
    assert np.array_equal(zb[:, 0], z)


def test_tf32_rounding():
    """round to nearest on the 13 dropped bits, ties away from zero"""
    one = np.float32(1.)
    ulp = np.float32(2.**-10)
    assert kr.tf32(one + np.float32(2.**-12)) == one
    assert kr.tf32(one + np.float32(2.**-11)) == one + ulp          # tie: away
    assert kr.tf32(-(one + np.float32(2.**-11))) == -(one + ulp)
    assert kr.tf32(one + np.float32(3*2.**-12)) == one + ulp
    x = np.random.default_rng(0).standard_normal(1000).astype(np.float32)
    assert np.all(np.abs(kr.tf32(x) - x) <= 2.**-11*np.abs(x))
    assert np.all((kr.tf32(x).view(np.uint32) & 0x1FFF) == 0)


def test_float32_emulation_is_well_inside_the_kernel_tolerance():
    """on the benchmarked mesh (cylinder_4, device numbering, the 64 Robin
    control members at tau = dt/2, the fp32 start from r - JT zp) the float32
    emulation of the smoother stays 10x below the tolerance the kernel tests
    allow the fp32 tile kernels, for every step count they run"""
    from dolfin_navier_scipy_b200 import hostsetup
    h = kr.device_numbering(4)
    tau = .5/512
    M, Ar = h['M'], h['Arob']
    F1 = sps.csr_matrix((M.data + tau*Ar.data, M.indices, M.indptr),
                        shape=M.shape)
    F2, coef = h['A0'], tau*h['nus']
    lo = [hostsetup.jacobi_spectrum(kr.member_matrix(F1, F2, c))
          for c in (coef.max(), coef.mean())]
    lmin, lmax = min(a for a, _ in lo), max(b for _, b in lo)
    rng = np.random.default_rng(4)
    r = rng.standard_normal((F1.shape[0], 64))
    zp = rng.standard_normal((h['J'].shape[0], 64))
    for k in (2, 3, 4, 5):
        z = kr.cheb_batched(F1, F2, coef, r, k, lmin, lmax, JT=h['JT'], zp=zp)
        zf = kr.cheb_batched(F1, F2, coef, r, k, lmin, lmax, JT=h['JT'],
                             zp=zp, f32=True)
        err = np.linalg.norm(zf - z, axis=0)/np.linalg.norm(z, axis=0)
        assert np.all(err < F32_TOL/10), (k, err.max())
        assert np.all(err > 1e-9), k          # it is float32 arithmetic
        emax = np.abs(zf - z).max(axis=0)/np.abs(z).max(axis=0)
        assert np.all(emax < F32_TOL/2), (k, emax.max())


def test_tile_plans_of_the_cylinder_meshes():
    """cylinder_1 fills its last tile, cylinder_4 (the benchmarked mesh) ends
    on a tile of 5 row pairs; F, JT and K all get a 3-stage plan"""
    for N, npairs, last in ((1, 2912, 8), (4, 14485, 5)):
        h = kr.device_numbering(N)
        pf = kr.tile_plan(h['M'])
        assert pf['ok'] and pf['npairs'] == npairs and pf['last'] == last
        assert pf['stages'] == pf['stages_f'] == 3 and pf['fp32_ctas'] == 2
        assert pf['rmax'] <= 32
        pj = kr.tile_plan(h['JT'])
        assert pj['ok'] and pj['npairs'] == npairs
        pk = kr.tile_plan(kr.block_k(h['M'], h['JT'], h['J']))
        assert pk['ok'] and pk['npairs'] == npairs and pk['last'] == last


@pytest.mark.parametrize('name', sorted(kr.SYNTHETIC))
def test_synthetic_systems_reach_their_planner_edges(name):
    kw, want = kr.SYNTHETIC[name]
    F1, F2, J, JT = kr.paired_system(**kw)
    plan = kr.tile_plan(F1)
    want = dict(want)
    want.setdefault('ok', True)
    for key, val in want.items():
        assert plan[key] == val, (key, plan)
    if plan['ok']:
        assert plan['rmax'] <= 32 and plan['stages'] >= 2
    # every row of F and of JT is paired (the fp32 smoother needs that)
    assert kr.paired_rows(F1) == F1.shape[0]
    assert kr.paired_rows(JT) == JT.shape[0]
    # F1 + c F2 is diagonally dominant for c >= 0
    for F in (F1, F2):
        d = F.diagonal()
        assert np.all(d > np.asarray(abs(F).sum(axis=1)).ravel() - d)
    pj = kr.tile_plan(JT)
    assert pj['ok'] == (not kw.get('jt_scatter', False)), pj
    ip = F1.indptr
    if kw.get('odd'):
        lens = np.diff(ip)[::2]
        assert np.any(lens % 2 == 1) and np.any(lens % 2 == 0)
        starts = ip[2*np.arange(0, plan['npairs'], kr.TILE_RP)]//2
        assert np.any(starts % 4 != 0)
    if kw.get('last_col'):
        # a run of every tile ends at the last row of x
        nv = F1.shape[0]
        for t in range(plan['ntiles']):
            assert F1.indices[ip[16*t]:ip[16*t + 1]].max() == nv - 1
        K = kr.block_k(F1, JT, J)
        assert K.indices[K.indptr[nv - 2]:K.indptr[nv - 1]].max() == \
            K.shape[1] - 1
