"""Plain restatements of the 64-member operator kernels, for the kernel tests.

Everything here runs on the host in numpy/scipy: the batched Jacobi-Chebyshev
smoother in fp64 and as a float32 emulation of the fp32 tile kernels
(`dnsb_tile.cuh`), the block-triangular preconditioner built on it, the
planner of the tile kernels (`tile_setup` in `dnsb_api.cu`), the TF32 rounding
of the tensor-core Schur block (`dnsb_tc.cuh`) and generators of small
row-paired systems that put the planner at its limits.
"""
import os

import numpy as np
import scipy.sparse as sps

TILE_RP = 8                    # row pairs per tile
TILE_NB = 64                   # members of the tile kernels
TILE_SMEM_OPTIN = 220*1024     # dynamic shared memory a tile kernel may use
TILE_MAX_STAGES = 8
SM_SMEM = 227*1024             # shared memory of an SM (B200)


# ---------------------------------------------------------------------------
# Jacobi-Chebyshev smoother (zero initial guess)
# ---------------------------------------------------------------------------
def _coefs(k, lmin, lmax):
    """per step i = 1..k-1: (c1, c2) of  d <- c1*d + c2*dinv*res"""
    th, de = .5*(lmax + lmin), .5*(lmax - lmin)
    sigma = th/de
    rho = 1./sigma
    out = []
    for _ in range(k - 1):
        rho_n = 1./(2*sigma - rho)
        out.append((rho_n*rho, 2*rho_n/de))
        rho = rho_n
    return th, out


def cheb_np(Fm, dinv, r, k, lmin, lmax):
    """k-step Jacobi-Chebyshev approximation of ``Fm^-1 r`` in fp64
    (``Fm``: one matrix, ``r``: a vector or a block of vectors)"""
    th, steps = _coefs(k, lmin, lmax)
    res = np.array(r, dtype=float)
    d = dinv*res/th
    z = d.copy()
    for c1, c2 in steps:
        res = res - Fm@d
        d = c1*d + c2*(dinv*res)
        z = z + d
    return z


def member_matrix(F1, F2, c, dtype=np.float64):
    """``F1 + c*F2`` on the shared pattern; float32: the entries the fp32
    kernel forms (values and coefficient rounded to float32 first)"""
    if F2 is None:
        data = F1.data.astype(dtype)
    elif dtype == np.float32:
        data = (np.float32(c)*F2.data.astype(np.float32) +
                F1.data.astype(np.float32))
    else:
        data = F1.data + c*F2.data
    return sps.csr_matrix((data, F1.indices, F1.indptr), shape=F1.shape)


def member_dinv(F1, F2, coef):
    """(n, nb) inverse diagonals of the members (fp64, as `k_diag_inv`)"""
    d1 = F1.diagonal()
    d2 = np.zeros_like(d1) if F2 is None else F2.diagonal()
    return 1./(d1[:, None] + d2[:, None]*np.asarray(coef)[None, :])


def cheb_batched(F1, F2, coef, r, k, lmin, lmax, JT=None, zp=None, f32=False):
    """the smoother of every member: ``z_m = cheb(F1 + coef_m*F2)(r_m - JT zp_m)``

    ``f32=True`` emulates the fp32 tile kernels: the start ``res = r - JT zp``
    is summed in fp64 and stored as float32 (`k_cheb_init_tilef`), every later
    operand -- matrix entries, inverse diagonal, residual, direction, sum -- is
    float32 with float32 sparse products; the result is returned in fp64."""
    coef = np.asarray(coef, dtype=float)
    nb = coef.size
    b = np.array(r, dtype=float).reshape(F1.shape[0], nb)
    if JT is not None:
        b = b - JT@zp
    dinv = member_dinv(F1, F2, coef)
    if not f32:
        z = np.empty_like(b)
        for m in range(nb):
            z[:, m] = cheb_np(member_matrix(F1, F2, coef[m]), dinv[:, m],
                              b[:, m], k, lmin, lmax)
        return z
    th, steps = _coefs(k, lmin, lmax)
    f = np.float32
    inv_th = f(1./th)
    res = b.astype(f)
    dv = dinv.astype(f)
    d = dv*res*inv_th
    z = d.copy()
    for m in range(nb):
        Fm = member_matrix(F1, F2, coef[m], np.float32)
        rm, dm, zm, dvm = res[:, m].copy(), d[:, m].copy(), z[:, m].copy(), dv[:, m]
        for c1, c2 in steps:
            rm = rm - Fm@dm
            dm = (f(c2)*dvm)*rm + f(c1)*dm
            zm = zm + dm
        z[:, m] = zm
    return z.astype(np.float64)


def prec_pressure(dense, rp, alpha=-1., mp_dinv=None, mp_scale=None):
    """``zp = alpha*(D rp + scale_m*mp_dinv*rp)`` (the dense Schur block)"""
    zp = dense@rp
    if mp_dinv is not None:
        zp = zp + np.asarray(mp_scale)[None, :]*np.asarray(mp_dinv)[:, None]*rp
    return alpha*zp


def apply_k(F1, F2, coef, J, JT, X):
    """``K_m x_m`` for ``K_m = [[F1 + coef_m*F2, JT], [J, 0]]``"""
    nv = F1.shape[0]
    xv, xp = X[:nv], X[nv:]
    yv = F1@xv + JT@xp
    if F2 is not None:
        yv = yv + (F2@xv)*np.asarray(coef)[None, :]
    return np.vstack([yv, J@xv])


# ---------------------------------------------------------------------------
# TF32
# ---------------------------------------------------------------------------
def tf32(x):
    """``cvt.rna.tf32.f32`` of ``float32(x)``: round to nearest, ties away
    from zero, to 10 mantissa bits; returned as float32"""
    b = np.asarray(x, dtype=np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


# ---------------------------------------------------------------------------
# planner of the tile kernels
# ---------------------------------------------------------------------------
def paired_rows(P):
    """leading rows of ``P`` that pair up as (2k, 2k+1) with the same
    non-empty column list (`csr_build`)"""
    P = sps.csr_matrix(P)
    ip, ix = P.indptr, P.indices
    n = 0
    for r in range(0, P.shape[0] - 1, 2):
        a0, a1, a2 = ip[r], ip[r + 1], ip[r + 2]
        if a1 - a0 != a2 - a1 or a1 == a0 or \
                not np.array_equal(ix[a0:a1], ix[a1:a2]):
            break
        n = r + 2
    return n


def tile_plan(P, stages=3, stages_f=3, tilef_ctas=2):
    """the tile plan `tile_setup` makes for the paired rows of ``P``

    Returns a dict: ``npairs``, ``ntiles``, ``last`` (row pairs in the last
    tile), ``rmax`` (runs of consecutive columns per tile), ``umax`` (unique
    columns per tile), ``cap`` (aligned entry span per tile), the fp64 / fp32
    stage bytes, ring depths and ring bytes, ``fp32_ctas`` (CTAs per SM of the
    fp32 smoother) and ``ok`` / ``refused`` (why the row-pair kernels serve
    the matrix instead)."""
    P = sps.csr_matrix(P)
    P.sort_indices()
    ip, ix = P.indptr, P.indices
    npairs = paired_rows(P)//2
    out = dict(npairs=npairs, ok=False, refused=None)
    if npairs < 1:
        out['refused'] = 'no paired rows'
        return out
    ntiles = (npairs + TILE_RP - 1)//TILE_RP
    rmax = umax = cap = 0
    for t in range(ntiles):
        p0, p1 = t*TILE_RP, min(npairs, (t + 1)*TILE_RP)
        cols = np.unique(np.concatenate([ix[ip[2*q]:ip[2*q + 1]]
                                         for q in range(p0, p1)]))
        umax = max(umax, cols.size)
        rmax = max(rmax, 1 + int(np.count_nonzero(np.diff(cols) != 1)))
        pe0, pe1 = ip[2*p0]//2, ip[2*p1]//2
        cap = max(cap, ((pe1 + 3) & ~3) - (pe0 & ~3))
    sb = (umax*TILE_NB*8 + cap*36 + 127) & ~127
    sbf = (umax*TILE_NB*4 + cap*20 + 127) & ~127
    st = min(stages, TILE_SMEM_OPTIN//sb)
    stf = min(stages_f, TILE_SMEM_OPTIN//sbf)
    out.update(ntiles=ntiles, last=npairs - (ntiles - 1)*TILE_RP, rmax=rmax,
               umax=umax, cap=cap, stage_bytes=sb, stage_bytes_f=sbf,
               stages=st, stages_f=stf, smem=st*sb, smem_f=stf*sbf)
    out['fp32_ctas'] = 2 if tilef_ctas >= 2 and \
        2*(stf*sbf + 2048) <= SM_SMEM else 1
    if st < 2 or stf < 2:
        out['refused'] = 'ring of fewer than 2 stages'
    elif rmax > 32:
        out['refused'] = 'more than 32 runs per tile'
    else:
        out['ok'] = True
    return out


def block_k(F1, JT, J):
    """pattern of ``K = [[F, JT], [J, 0]]`` as the solver assembles it"""
    return sps.bmat([[F1, JT], [J, None]], format='csr')


# ---------------------------------------------------------------------------
# synthetic row-paired systems
# ---------------------------------------------------------------------------
def paired_system(npairs, runs=0, run_len=4, share=False, odd=False,
                  last_col=False, np_=160, jt_scatter=False, seed=0):
    """a small saddle-point system ``F1, F2, J, JT`` with row-paired F and JT

    The velocity unknowns are ``npairs`` nodes of two components.  The pairs
    of a tile (8 consecutive nodes) couple to the columns of all the nodes of
    the tile, plus ``runs`` extra runs of ``run_len`` consecutive columns
    elsewhere (scattered, never adjacent: each one a separate bulk copy of the
    tile kernels).  ``share``: every pair of the tile takes every extra run
    (rows as long as the tile's column set), else the runs are dealt out to
    the pairs in turn.  ``odd``: every second pair drops one column, so rows
    have odd and even lengths and tile spans start unaligned.  ``last_col``:
    one extra run of every tile ends at the last column.  Both rows of a pair
    have the same columns and their own values; ``F1 + c*F2`` is diagonally
    dominant for c >= 0.  JT couples every pair to three consecutive pressure
    nodes (``jt_scatter``: to five scattered ones), the last pair to the last
    pressure node; ``J = JT.T``."""
    rng = np.random.default_rng(seed)
    nv = 2*npairs
    rows, cols = [], []
    for t in range(0, npairs, TILE_RP):
        p1 = min(npairs, t + TILE_RP)
        own = np.arange(2*t, 2*p1)
        # free run starts: runs separated by at least one column from each
        # other and from the tile's own block
        extra = []
        if runs:
            taken = np.zeros(nv + 1, dtype=bool)
            taken[max(0, 2*t - 1):min(nv, 2*p1 + 1)] = True
            if last_col:
                s = nv - run_len
                if s > 2*p1 or s + run_len < 2*t - 1:
                    extra.append(np.arange(s, nv))
                    taken[max(0, s - 1):nv] = True
            starts = rng.permutation(nv - run_len + 1)
            for s in starts:
                if len(extra) == runs:
                    break
                if not taken[max(0, s - 1):s + run_len + 1].any():
                    extra.append(np.arange(s, s + run_len))
                    taken[max(0, s - 1):s + run_len + 1] = True
            assert len(extra) == runs, 'too few columns for the runs'
        for j, q in enumerate(range(t, p1)):
            mine = extra if share else extra[j::TILE_RP]
            c = np.concatenate([own] + mine) if mine else own
            if odd and j % 2 == 1:
                # drop the first column of another node of the tile
                c = c[c != own[0 if q != t else 2]]
            c = np.sort(c)
            for r in (2*q, 2*q + 1):
                rows.append(np.full(c.size, r))
                cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    off = rows != cols

    def values(scale, shift):
        v = rng.uniform(-1., 1., rows.size)*scale
        v[~off] = 0.
        M = sps.csr_matrix((v, (rows, cols)), shape=(nv, nv))
        d = np.asarray(abs(M).sum(axis=1)).ravel() + shift
        v[~off] = d[rows[~off]]
        M = sps.csr_matrix((v, (rows, cols)), shape=(nv, nv))
        M.sort_indices()
        return M
    F1 = values(1., 1.)
    F2 = values(.5, .5)
    assert np.array_equal(F1.indices, F2.indices)
    jr, jc = [], []
    for q in range(npairs):
        if jt_scatter:
            pc = rng.choice(np_//2, 5, replace=False)*2
        else:
            b = min(np_ - 3, (q*np_)//npairs)
            pc = np.arange(b, b + 3)
        if q == npairs - 1:
            pc = np.union1d(pc, [np_ - 1])
        for r in (2*q, 2*q + 1):
            jr.append(np.full(pc.size, r))
            jc.append(pc)
    jr, jc = np.concatenate(jr), np.concatenate(jc)
    JT = sps.csr_matrix((rng.uniform(-1., 1., jr.size), (jr, jc)),
                        shape=(nv, np_))
    JT.sort_indices()
    J = JT.T.tocsr()
    J.sort_indices()
    return F1, F2, J, JT


# synthetic cases of the kernel tests:
# name: (arguments of `paired_system`, what `tile_plan` of its F must show)
SYNTHETIC = {
    'pairs_8q_plus_1': (dict(npairs=8*5 + 1, runs=2), dict(last=1)),
    'pairs_8q_plus_7': (dict(npairs=8*5 + 7, runs=2), dict(last=7)),
    'fewer_than_8_pairs': (dict(npairs=5), dict(ntiles=1, last=5)),
    'tiles_below_148': (dict(npairs=800, runs=3), dict(ntiles=100)),
    'tiles_148_to_296': (dict(npairs=1600, runs=3), dict(ntiles=200)),
    'tiles_far_above_296': (dict(npairs=9600, runs=2), dict(ntiles=1200)),
    'runs_32': (dict(npairs=800, runs=31, run_len=1), dict(rmax=32)),
    'runs_33': (dict(npairs=800, runs=32, run_len=1),
                dict(rmax=33, ok=False)),
    'fp64_ring_2_stages': (dict(npairs=400, runs=8, run_len=16),
                           dict(stages=2, stages_f=3)),
    'fp32_one_cta_per_sm': (dict(npairs=400, runs=4, run_len=19, share=True),
                            dict(stages=3, stages_f=3, fp32_ctas=1)),
    'ring_refused': (dict(npairs=400, runs=14, run_len=16),
                     dict(stages=1, ok=False)),
    'run_ends_at_last_column': (dict(npairs=203, runs=2, last_col=True),
                                dict(last=3)),
    'odd_rows_unaligned_spans': (dict(npairs=203, runs=3, run_len=3,
                                      odd=True), dict(last=3)),
    'gradient_without_plan': (dict(npairs=400, runs=2, jt_scatter=True,
                                   np_=400), dict(ntiles=50)),
}


def device_numbering(N=4, palpha=1e-5):
    """the loop operators of `ensemble.cylinder_ensemble(N)` in the device
    numbering (Hilbert order, padded row pairs) as `DeviceImex` builds them:
    ``dict(M, A0, Arob, J, JT, nus)`` (nu = 1 operators, Robin control)"""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    from dolfin_navier_scipy_b200 import hostsetup
    from dolfin_navier_scipy_b200 import problem_setups as dnsps
    from dolfin_navier_scipy_b200 import time_int_utils as tiu
    femp, sm, _, _ = dnsps.get_sysmats(
        problem='cylinderwake', nu=1., bccontrol=True, scheme='TH',
        meshparams=dict(refinement_level=N))
    V, inv = femp['V'], np.asarray(femp['invinds'])
    pv = hostsetup.locality_perm(np.asarray(V.tabulate_dof_coordinates())[inv],
                                 comp=inv % 2)
    J = sps.csr_matrix(sm['J'])
    pxy = np.asarray(V.mesh().coords)
    pp = hostsetup.locality_perm(pxy) if pxy.shape[0] == J.shape[0] else \
        hostsetup.locality_perm(pattern=abs(J)@abs(J).T)

    def _pvv(X):
        return sps.csr_matrix(X)[pv][:, pv].tocsr()
    M, A0, Arob = _pvv(sm['M']), _pvv(sm['A']), _pvv(sm['Arob']/palpha)
    pat = hostsetup.pad_row_pairs(tiu._union_pattern([M, A0, Arob]))
    J = sps.csr_matrix(sm['J'])[pp][:, pv].tocsr()
    JT = J.T.tocsr()
    JT.sort_indices()
    JT = tiu._on_pattern(JT, hostsetup.pad_row_pairs(JT))
    return dict(M=tiu._on_pattern(M, pat), A0=tiu._on_pattern(A0, pat),
                Arob=tiu._on_pattern(Arob, pat), J=J, JT=JT,
                nus=femp['charlen']/np.linspace(60., 150., 64))


def ctx_with_env(name, value, **more):
    """a device context created under environment switches (the DNSB_*
    switches are read when a context is created and stay with it)"""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    from dolfin_navier_scipy_b200 import _lib
    env = dict(more)
    env[name] = value
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return _lib.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v
