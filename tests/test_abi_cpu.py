"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every
symbol `include/dnsb.h` declares; host-side setup logic."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import scipy.sparse as sps

import __graft_entry__ as ge
from dolfin_navier_scipy_b200 import _lib, fem, hostsetup
from dolfin_navier_scipy_b200 import time_int_utils as tiu
from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    with open(os.path.join(ROOT, 'include', 'dnsb.h')) as f:
        txt = re.sub(r'/\*.*?\*/', '', f.read(), flags=re.S)
    return sorted(set(re.findall(r'\b(dnsb_[a-z0-9_]+)\s*\(', txt)))


def test_library_builds_and_exports_every_declared_symbol():
    lib = ge.build()
    dll = ctypes.CDLL(lib)
    names = _declared()
    assert len(names) >= 30
    for n in names:
        assert hasattr(dll, n), n
    # the ctypes table mirrors the header one to one
    assert sorted(_lib.SIGNATURES.keys()) == names
    assert dll.dnsb_version() >= 100


def test_colouring_is_valid_and_balanced():
    for lvl in (1, 2):
        m = fem.load_mesh('cylinder_%d' % lvl)
        ncol, col = fem.colour_cells(m)
        for c in range(ncol):
            verts = m.cells[col == c].ravel()
            assert verts.size == np.unique(verts).size   # no shared vertex
        counts = np.bincount(col, minlength=ncol)
        assert counts.max() <= 2.5*counts.mean()


def test_lowrank_forcing_is_exact_for_separable_inputs():
    rng = np.random.default_rng(0)
    b = rng.standard_normal((50, 2))
    tr = np.linspace(0, 1, 17)
    B, U = tiu.lowrank_forcing(
        lambda t: np.sin(t)*b[:, :1] + t*t*b[:, 1:], tr, 50)
    assert B.shape[1] == 2 and U.shape == (17, 2)
    for k, t in enumerate(tr):
        assert np.allclose(B@U[k], np.sin(t)*b[:, 0] + t*t*b[:, 1], atol=1e-12)


def test_lowrank_forcing_samples_in_chunks_and_fails_early():
    """round-1 advisor finding: the sampler worked on a dense NV x steps
    matrix and reported a rank > 64 only after every sample was evaluated.
    It now grows its basis chunk by chunk: a forcing whose later chunks add
    directions is still exact, and a full-rank one stops at the first chunks"""
    rng = np.random.default_rng(1)
    nv = 300
    b = rng.standard_normal((3, nv, 1))

    def f(t):
        return np.sin(t)*b[0] + np.cos(3*t)*b[1] + (t > .5)*b[2]
    tr = np.linspace(0, 1, 1000)
    B, U = tiu.lowrank_forcing(f, tr, nv, chunk=64)
    F = np.hstack([f(t) for t in tr])
    assert B.shape == (nv, 3) and U.shape == (1000, 3)
    assert np.linalg.norm(F - B@U.T) < 1e-13*np.linalg.norm(F)
    B0, U0 = tiu.lowrank_forcing(lambda t: np.zeros((nv, 1)), tr, nv)
    assert not B0.any() and not U0.any() and U0.shape == (1000, 1)
    calls = [0]

    def noise(t):
        calls[0] += 1
        return rng.standard_normal((nv, 1))
    with pytest.raises(NotImplementedError):
        tiu.lowrank_forcing(noise, tr, nv, chunk=64)
    assert calls[0] <= 128


class _FakeDeviceSolver(object):
    """what `SadpntOperator.solve_minres` needs from `_lib.Solver`, in scipy:
    the product with K and the block-diagonal preconditioner"""

    def __init__(self, F, J, exact_schur=True):
        import scipy.sparse.linalg as spsla
        self.nv, self.np_, self.nb = F.shape[0], J.shape[0], 1
        self.K = sps.bmat([[F, J.T], [J, None]], format='csr')
        self.Finv = spsla.factorized(sps.csc_matrix(F))
        S = (J@sps.diags(1./F.diagonal())@J.T).toarray()
        self.Sinv = np.linalg.inv(S)
        self.mode = []

    def set_prec_mode(self, flag):
        self.mode.append(bool(flag))

    def apply_k(self, x):
        return self.K@np.asarray(x).reshape(-1, 1)

    def apply_prec(self, r):
        assert self.mode and self.mode[-1], 'MINRES must ask for the SPD form'
        r = np.asarray(r).ravel()
        return np.concatenate([self.Finv(r[:self.nv]), self.Sinv@r[self.nv:]])


def _minres_operator(F, J):
    from dolfin_navier_scipy_b200 import lin_alg_utils as lau
    op = lau.SadpntOperator.__new__(lau.SadpntOperator)
    op.NP, op.NV = J.shape
    op.ncols = 1
    op.solver = _FakeDeviceSolver(F, J)
    return op


def test_minres_host_recurrence_checks_the_true_residual(cyl1):
    """the host side of `krylov='minres'`: scipy's recurrence over the device's
    operators (here replaced by scipy ones), the SPD preconditioner mode
    switched on for the solve and off again afterwards, the TRUE relative
    residual checked against the tolerance, `NotConverged` when the iteration
    budget does not reach it"""
    from dolfin_navier_scipy_b200 import _lib
    from oracle import lau as olau
    femp, sm, rhsd = cyl1
    F = (sm['M'] + .5/512*sm['A']).tocsr()
    J = sm['J'].tocsr()
    rng = np.random.default_rng(5)
    rhsv = rng.standard_normal((F.shape[0], 1))
    op = _minres_operator(F, J)
    vp = op.solve_minres(rhsv, rhsd['fp'], tol=1e-10, maxit=400)
    ref = olau.solve_sadpnt_smw(amat=F, jmat=J, jmatT=J.T, rhsv=rhsv,
                                rhsp=rhsd['fp'])
    assert np.linalg.norm(vp - ref) < 1e-8*np.linalg.norm(ref)
    assert op.last_relres[0] <= 1e-10 and 0 < op.last_iters[0] <= 400
    assert op.solver.mode[0] is True and op.solver.mode[-1] is False
    op2 = _minres_operator(F, J)
    with pytest.raises(_lib.NotConverged):
        op2.solve_minres(rhsv, rhsd['fp'], tol=1e-12, maxit=3)
    assert op2.solver.mode[-1] is False          # switched back on the error path too
    op3 = _minres_operator(F, J)
    op3.ncols = 2
    with pytest.raises(NotImplementedError):
        op3.solve_minres(np.hstack([rhsv, rhsv]))


def test_cpu_binding_helper_never_raises():
    """`ensemble.bind_to_gpu_cpus` pins a rank next to its GPU when NVML can
    say where that is, and is a no-op (None) everywhere else -- e.g. here"""
    import os
    from dolfin_navier_scipy_b200 import ensemble
    before = os.sched_getaffinity(0)
    got = ensemble.bind_to_gpu_cpus(0)
    assert got is None or set(got) <= before
    os.sched_setaffinity(0, before)


def test_pattern_embedding_keeps_explicit_zeros():
    A = sps.random(20, 20, .3, random_state=1, format='csr') + sps.identity(20)
    M = sps.identity(20, format='csr')
    pat = tiu._union_pattern([M, A])
    Mp = tiu._on_pattern(M, pat)
    assert Mp.nnz == pat.nnz and abs(Mp - M).max() == 0
    assert np.array_equal(Mp.indices, pat.indices)


def test_sa_amg_two_grid_converges_on_lumped_schur(cyl1):
    # host set-up sanity: V-cycle (numpy emulation of the device cycle) as a
    # stationary iteration contracts the error of the pressure operator
    femp, sm, rhsd = cyl1
    F = sm['M'] + .5/512*sm['A']
    S = hostsetup.lumped_schur(F.diagonal(), sm['J'])
    levels, dense = hostsetup.sa_amg_hierarchy(S, coarse_max=200)
    assert len(levels) >= 1 and dense.shape[0] <= 200

    def cheb(A, dinv, r, k, lmin, lmax):
        th, de = .5*(lmax + lmin), .5*(lmax - lmin)
        sg = th/de
        rho = 1/sg
        z, res = np.zeros_like(r), r.copy()
        d = dinv*res/th
        for i in range(k):
            z += d
            if i == k - 1:
                break
            res -= A@d
            rn = 1/(2*sg - rho)
            d = rn*rho*d + 2*rn/de*(dinv*res)
            rho = rn
        return z

    def vcyc(l, b):
        if l == len(levels):
            return dense@b
        lv = levels[l]
        dinv = 1/lv['A'].diagonal()
        x = cheb(lv['A'], dinv, b, 2, lv['lmin'], lv['lmax'])
        x = x + lv['P']@vcyc(l + 1, lv['R']@(b - lv['A']@x))
        return x + cheb(lv['A'], dinv, b - lv['A']@x, 2, lv['lmin'], lv['lmax'])
    rng = np.random.default_rng(0)
    xex = rng.standard_normal(S.shape[0])
    b = S@xex
    x = np.zeros_like(b)
    for _ in range(12):
        x = x + vcyc(0, b - S@x)
    assert np.linalg.norm(x - xex) < 1e-3*np.linalg.norm(xex)


def test_condense_and_append_roundtrip(cyl1):
    femp, sm, rhsd = cyl1
    V, inv = femp['V'], femp['invinds']
    v = np.arange(inv.size, dtype=float).reshape(-1, 1)
    vf = dts.append_bcs_vec(v, V=V, invinds=inv, bcinds=femp['dbcinds'],
                            bcvals=femp['dbcvals'])
    assert vf.shape == (V.dim(), 1) and not np.any(np.isnan(vf))
    assert np.array_equal(vf[inv], v)
    Ac, fvbc = dts.condense_velmatsbybcs(sm['Afull'], invinds=inv,
                                         dbcinds=femp['dbcinds'],
                                         dbcvals=femp['dbcvals'])
    assert abs(Ac - sm['A']).max() < 1e-15


def test_device_path_fails_loudly_without_a_gpu():
    """no CPU fallback: without a CUDA device the context cannot be created and
    every device entry point of the Python mirror raises"""
    import torch
    if torch.cuda.is_available():
        pytest.skip('a CUDA device is present')
    from dolfin_navier_scipy_b200 import _lib
    from dolfin_navier_scipy_b200 import dolfin_to_sparrays as dts
    from dolfin_navier_scipy_b200 import fem
    with pytest.raises(_lib.DnsbError):
        _lib.Context(0)
    assert _lib.live_bytes() == (0, 0)     # the failed context was destroyed
    V = fem.VectorP2Space(fem.unit_square_mesh(2))
    with pytest.raises(RuntimeError):
        dts.get_convvec(V=V, u0_vec=np.zeros(V.dim()))


def test_missing_library_is_an_error(tmp_path):
    from dolfin_navier_scipy_b200 import _lib
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        _lib.load(str(tmp_path / 'libdnsb200.so'))


def test_stokes_slot_patterns_reproduce_the_host_assembly():
    """host side of the device assembly (`dnsb_assemble_stokes`): the patterns
    of J and MP built from the connectivity equal the host shim's, and summing
    per-cell element entries through the slots equals the COO assembly"""
    mesh = fem.unit_square_mesh(4, 3)
    V, Q = fem.VectorP2Space(mesh), fem.P1Space(mesh)
    host = fem.assemble_stokes_operators(V, Q, nu=1.)
    cn, c3 = V.cell_nodes.astype(np.int64), mesh.cells.astype(np.int64)
    jk, jslots, pk, pslots = _lib.stokes_slot_patterns(cn, c3, V.dim(), Q.dim())
    for keys, slots, per, ref in ((jk, jslots, 36, host['J']), (pk, pslots, 9, host['MP'])):
        ref = ref.tocsr()
        ref.sort_indices()
        pat = _lib._csr_from_keys(keys, ref.shape[0], ref.shape[1], np.ones(keys.size))
        assert np.array_equal(pat.indptr, ref.indptr)
        assert np.array_equal(pat.indices, ref.indices)
        assert slots.size == per*mesh.num_cells and slots.min() == 0 and slots.max() == keys.size - 1
    # scatter of random element entries through the slots == COO assembly
    rng = np.random.default_rng(5)
    E = rng.standard_normal((mesh.num_cells, 3, 12))
    vals = np.zeros(jk.size)
    np.add.at(vals, jslots, E.ravel())
    vd = np.stack([2*cn, 2*cn + 1], axis=2).reshape(-1, 12)
    ref = fem._coo_to_csr(np.repeat(c3[:, :, None], 12, axis=2), np.repeat(vd[:, None, :], 3, axis=1), E,
                          (Q.dim(), V.dim()))
    got = _lib._csr_from_keys(jk, Q.dim(), V.dim(), vals)
    assert abs(got - ref).max() < 1e-14


def test_bench_byte_formulas_cover_the_kernels_of_a_step(cyl1):
    """`bench.kernel_bytes` (the ALGORITHMIC bytes behind `roofline`): every
    HBM-class kernel that the committed bench line of the final state lists
    has a formula, the fp32 variants count fewer bytes than the fp64 ones
    they replace, and the Gram-Schmidt count grows with the vectors read"""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    femp, sm, rhsd = cyl1

    class _Integ(object):
        nb = 64
        _host = dict(M=sm['M'].tocsr(), J=sm['J'].tocsr())
    with open(os.path.join(root, 'profiles', 'r2f_bench.json')) as fh:
        line = json.loads([ln for ln in fh if ln.startswith('{')][-1])
    names = [k.strip('()') for k in line['kernels']]
    assert any(n.startswith('k_gs_tma') for n in names)
    by = {n: bench.kernel_bytes(n, None, _Integ, 8.) for n in names}
    for n, b in by.items():
        if n.startswith(('k_gs_tma', 'k_cheb_step_tilef', 'k_cheb_init', 'k_spmm',
                         'k_schur_tc', 'k_scale_member')):
            assert b is not None and b > 0, n
    f64 = bench.kernel_bytes('k_cheb_step_tile<false, false>', None, _Integ)
    f32 = bench.kernel_bytes('k_cheb_step_tilef<false, false>', None, _Integ)
    assert f32 < f64 < bench.kernel_bytes('k_cheb_step_p2<true, false, false>', None, _Integ)
    assert bench.kernel_bytes('k_cheb_init_tilef', None, _Integ) == \
        bench.kernel_bytes('k_cheb_init_p2f', None, _Integ) < \
        bench.kernel_bytes('k_cheb_init_p2', None, _Integ)
    assert bench.kernel_bytes('k_gs_tma<false>', None, _Integ, 20.) > \
        2*bench.kernel_bytes('k_gs_tma<false>', None, _Integ, 8.)


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours):
    exactly one JSON line on stdout with the contract's keys; everything else
    (library notes, worker output) goes to stderr"""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '2',
                        '--warmup', '1', '--mesh', '1', '--members', '2'],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'cylinder-wake DoF*steps/s'
    assert d['higher_is_better'] is True and d['value'] > 0 and d['steps'] == 2
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['value'] == d['value']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert 'workload' in d['config']
