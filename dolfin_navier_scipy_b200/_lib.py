"""ctypes binding of ``libdnsb200.so`` (C ABI declared in ``include/dnsb.h``).

There is no CPU fallback: if the library is missing or no CUDA device is
available, every entry point raises ``RuntimeError``.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.path.join(_HERE, 'libdnsb200.so')

c_int_p = ctypes.POINTER(ctypes.c_int32)
c_dbl_p = ctypes.POINTER(ctypes.c_double)
c_void_pp = ctypes.POINTER(ctypes.c_void_p)

_lib = None

# name: (restype, argtypes) -- mirrors include/dnsb.h one to one
_vp, _i, _d, _ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_longlong
SIGNATURES = {
    'dnsb_ctx_create': (_i, [_i, c_void_pp]),
    'dnsb_ctx_destroy': (None, [_vp]),
    'dnsb_last_error': (ctypes.c_char_p, [_vp]),
    'dnsb_version': (_i, []),
    'dnsb_device_info': (_i, [_vp, ctypes.POINTER(_i),
                              ctypes.POINTER(ctypes.c_size_t),
                              ctypes.POINTER(_i)]),
    'dnsb_sync': (_i, [_vp]),
    'dnsb_launch_count': (_ll, [_vp]),
    'dnsb_launch_count_reset': (None, [_vp]),
    'dnsb_profile_begin': (_i, [_vp, _i]),
    'dnsb_profile_end': (_i, [_vp, ctypes.c_char_p, _i]),
    'dnsb_live_bytes': (None, [ctypes.POINTER(_ll), ctypes.POINTER(_ll)]),
    'dnsb_set_mesh': (_i, [_vp, _i, _i, c_int_p, c_dbl_p, _i, c_int_p]),
    'dnsb_set_conv_pattern': (_i, [_vp, c_int_p, c_int_p, c_int_p]),
    'dnsb_convvec': (_i, [_vp, c_dbl_p, c_dbl_p, c_dbl_p, _i]),
    'dnsb_convmats': (_i, [_vp, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    'dnsb_csr_create': (_i, [_vp, _i, _i, c_int_p, c_int_p, c_dbl_p, c_dbl_p,
                             c_void_pp]),
    'dnsb_csr_destroy': (None, [_vp]),
    'dnsb_assemble_stokes': (_i, [_vp, _d, _i, _i, c_int_p, _i, c_int_p,
                                  c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    'dnsb_spmm': (_i, [_vp, c_dbl_p, c_dbl_p, c_dbl_p, _i, _d, _d]),
    'dnsb_spmm_dev': (_i, [_vp, _vp, _vp, _vp, _i, _d, _d]),
    'dnsb_solver_create': (_i, [_vp, _vp, _vp, _vp, c_dbl_p, _i, _i, _i, _d,
                                _d, c_void_pp]),
    'dnsb_solver_destroy': (None, [_vp]),
    'dnsb_solver_add_schur_level': (_i, [_vp, _vp, _vp, _vp, _i, _d, _d,
                                         c_dbl_p]),
    'dnsb_solver_set_velocity_transfer': (_i, [_vp, _vp, _vp]),
    'dnsb_solver_add_velocity_level': (_i, [_vp, _vp, _vp, _vp, _i, _d, _d,
                                            c_dbl_p]),
    'dnsb_solver_set_schur_mass': (_i, [_vp, c_dbl_p, c_dbl_p]),
    'dnsb_solver_set_schur_lsc': (_i, [_vp, c_dbl_p]),
    'dnsb_solver_solve': (_i, [_vp, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, _d, _i,
                               c_int_p, c_dbl_p]),
    'dnsb_solver_update_fvalues': (_i, [_vp, c_dbl_p]),
    'dnsb_solver_apply_prec': (_i, [_vp, c_dbl_p, c_dbl_p]),
    'dnsb_solver_set_prec_mode': (_i, [_vp, _i]),
    'dnsb_solver_apply_k': (_i, [_vp, c_dbl_p, c_dbl_p]),
    'dnsb_cnsweep_create': (_i, [_vp, _vp, c_dbl_p, c_dbl_p, _i, c_int_p, c_int_p,
                                 c_int_p, _i, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p,
                                 c_void_pp]),
    'dnsb_cnsweep_destroy': (None, [_vp]),
    'dnsb_cnsweep_run': (_i, [_vp, _i, c_dbl_p, _i, c_dbl_p, c_dbl_p, c_dbl_p, _d,
                              _i, c_dbl_p, c_dbl_p, c_dbl_p,
                              ctypes.POINTER(_ll)]),
    'dnsb_imex_create': (_i, [_vp, _i, _i, _d, _vp, _vp, _vp, _vp, c_dbl_p,
                              c_int_p, _i, _i, c_int_p, c_dbl_p, c_dbl_p,
                              c_dbl_p, c_void_pp]),
    'dnsb_imex_destroy': (None, [_vp]),
    'dnsb_imex_set_solvers': (_i, [_vp, _vp, _vp, _vp]),
    'dnsb_imex_set_forcing': (_i, [_vp, _i, c_dbl_p, _i, c_dbl_p]),
    'dnsb_imex_set_state': (_i, [_vp, c_dbl_p, c_dbl_p]),
    'dnsb_imex_run': (_i, [_vp, _i, _i, _d, _i, _i, _d, _i,
                           ctypes.POINTER(_i)]),
    'dnsb_imex_set_member_guard': (_i, [_vp, _i]),
    'dnsb_imex_member_status': (_i, [_vp, c_int_p]),
    'dnsb_imex_set_statistics': (_i, [_vp, _i]),
    'dnsb_imex_reset_statistics': (_i, [_vp]),
    'dnsb_imex_get_statistics': (_i, [_vp, ctypes.POINTER(_ll),
                                      ctypes.POINTER(_ll), ctypes.POINTER(_ll),
                                      c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p,
                                      c_dbl_p]),
    'dnsb_imex_last_run_ms': (_d, [_vp]),
    'dnsb_imex_get_state': (_i, [_vp, c_dbl_p, c_dbl_p]),
    'dnsb_imex_num_snapshots': (_i, [_vp]),
    'dnsb_imex_reset_snapshots': (_i, [_vp]),
    'dnsb_imex_get_snapshots': (_i, [_vp, c_dbl_p]),
    'dnsb_imex_set_output_order': (_i, [_vp, c_int_p, c_int_p]),
    'dnsb_imex_reserve_snapshots': (_i, [_vp, _i]),
    'dnsb_imex_snapshots_host': (_i, [_vp, ctypes.POINTER(c_dbl_p),
                                      ctypes.POINTER(_i)]),
    'dnsb_imex_set_outputs': (_i, [_vp, _vp, _vp]),
    'dnsb_imex_set_force': (_i, [_vp, _i, c_int_p, _vp, _vp, _vp, c_dbl_p]),
    'dnsb_imex_num_output_levels': (_i, [_vp]),
    'dnsb_imex_get_outputs': (_i, [_vp, c_dbl_p, c_dbl_p]),
    'dnsb_imex_reset_outputs': (_i, [_vp]),
    'dnsb_imex_stats': (_i, [_vp, ctypes.POINTER(_ll), ctypes.POINTER(_ll),
                             c_dbl_p]),
    'dnsb_imex_gram_dev': (_i, [_vp, _vp]),
    'dnsb_imex_gram': (_i, [_vp, c_dbl_p]),
    'dnsb_imex_unconverged': (_ll, [_vp]),
    'dnsb_cnsweep_stats': (_i, [_vp, c_dbl_p, ctypes.POINTER(_ll)]),
    'dnsb_cnsweep_set_guess': (_i, [_vp, _i]),
}

E_NOT_CONVERGED = -3


def load(path=None):
    """load the shared library and declare every symbol of ``dnsb.h``"""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = LIBPATH if path is None else path
    if not os.path.isfile(path):
        raise RuntimeError(
            'libdnsb200.so not found at {0}: build it with '
            '`python -c "import __graft_entry__ as g; g.build()"` -- there is '
            'no CPU fallback for the device path'.format(path))
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError if a symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(c_dbl_p)


def _ip(a):
    return None if a is None else a.ctypes.data_as(c_int_p)


def _f64(a, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


def _i32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int32)


class DnsbError(RuntimeError):
    pass


class NotConverged(DnsbError):
    """an iterative solve stopped at ``maxit`` above ``tol`` (the reference's
    sparse-LU solve cannot fail this way: never ignored silently)"""


class Context(object):
    """one device + one stream (``dnsb_ctx``)"""

    def __init__(self, device=0):
        self.lib = load()
        h = ctypes.c_void_p()
        rc = self.lib.dnsb_ctx_create(int(device), ctypes.byref(h))
        if rc != 0:
            # a failed create still returns its context, for the message
            msg = self.lib.dnsb_last_error(h).decode() if h else 'no context'
            self.lib.dnsb_ctx_destroy(h)
            raise DnsbError('dnsb_ctx_create(device={0}) failed: {1}'.
                            format(device, msg))
        self.h = h
        self.device = int(device)
        self._keep = []

    def check(self, rc):
        if rc == E_NOT_CONVERGED:
            raise NotConverged(self.lib.dnsb_last_error(self.h).decode())
        if rc != 0:
            raise DnsbError(self.lib.dnsb_last_error(self.h).decode())

    def info(self):
        sm, mem, cc = ctypes.c_int(), ctypes.c_size_t(), ctypes.c_int()
        self.check(self.lib.dnsb_device_info(self.h, ctypes.byref(sm),
                                             ctypes.byref(mem),
                                             ctypes.byref(cc)))
        return dict(sm_count=sm.value, mem_bytes=mem.value, cc=cc.value)

    def sync(self):
        self.check(self.lib.dnsb_sync(self.h))

    def launch_count(self):
        return int(self.lib.dnsb_launch_count(self.h))

    def reset_launch_count(self):
        self.lib.dnsb_launch_count_reset(self.h)

    def profile_begin(self, max_records=200000):
        self.check(self.lib.dnsb_profile_begin(self.h, int(max_records)))

    def profile_end(self):
        """{kernel: (count, total_ms)} measured with CUDA events; the summed
        per-launch work some kernels report is kept in ``self.last_work``"""
        buf = ctypes.create_string_buffer(1 << 16)
        n = self.lib.dnsb_profile_end(self.h, buf, len(buf))
        if n < 0:
            self.check(n)
        out, self.last_work = {}, {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms, work = line.rsplit(' ', 3)
            out[name] = (int(cnt), float(ms))
            self.last_work[name] = int(work)
        return out

    def close(self):
        if self.h:
            self.lib.dnsb_ctx_destroy(self.h)
            self.h = ctypes.c_void_p()

    # -- CSR ----------------------------------------------------------------
    def csr(self, mat, vals2=None):
        return Csr(self, mat, vals2)


def live_bytes():
    """``(device, pinned)`` bytes the library holds in this process"""
    lib = load()
    dev, pinned = _ll(), _ll()
    lib.dnsb_live_bytes(ctypes.byref(dev), ctypes.byref(pinned))
    return dev.value, pinned.value


_CTX = {}


def default_context(device=None):
    if device is None:
        device = int(os.environ.get('LOCAL_RANK', '0'))
    if device not in _CTX:
        _CTX[device] = Context(device)
    return _CTX[device]


class Csr(object):
    """device CSR matrix (``dnsb_csr``); ``vals2`` shares the pattern"""

    def __init__(self, ctx, mat, vals2=None):
        import scipy.sparse as sps
        mat = sps.csr_matrix(mat)
        mat.sort_indices()
        self.ctx = ctx
        self.shape = mat.shape
        self.nnz = mat.nnz
        indptr, indices = _i32(mat.indptr), _i32(mat.indices)
        v1 = _f64(mat.data)
        v2 = _f64(vals2)
        if v2 is not None and v2.size != v1.size:
            raise ValueError('vals2 must match the pattern of the matrix')
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.dnsb_csr_create(ctx.h, mat.shape[0], mat.shape[1],
                                          _ip(indptr), _ip(indices), _dp(v1),
                                          _dp(v2), ctypes.byref(h)))
        self.h = h
        self.has2 = v2 is not None

    def spmm(self, x, coef=None, alpha=1.0, beta=0.0, y=None):
        """``alpha*A@x + beta*y`` for x of shape (ncols,) or (ncols, nb)"""
        x = _f64(x)
        nb = 1 if x.ndim == 1 else x.shape[1]
        out = np.zeros((self.shape[0],) + x.shape[1:]) if y is None \
            else _f64(y).copy()
        coef = _f64(coef)
        self.ctx.check(self.ctx.lib.dnsb_spmm(self.h, _dp(coef), _dp(x),
                                              _dp(out), nb, alpha, beta))
        return out

    def close(self):
        if self.h:
            self.ctx.lib.dnsb_csr_destroy(self.h)
            self.h = ctypes.c_void_p()


def _key_pattern(rows, cols, ncols):
    """sorted unique (row, col) keys of a pattern and, per element entry, its CSR slot"""
    keys = (rows*ncols + cols).reshape(-1)
    ukeys = np.unique(keys)
    return ukeys, np.searchsorted(ukeys, keys).astype(np.int32)


def _csr_from_keys(ukeys, nrows, ncols, vals):
    import scipy.sparse as sps
    r = ukeys // ncols
    ip = np.zeros(nrows + 1, dtype=np.int64)
    np.add.at(ip, r + 1, 1)
    return sps.csr_matrix((vals, (ukeys % ncols).astype(np.int32),
                           np.cumsum(ip).astype(np.int32)),
                          shape=(nrows, ncols))


def stokes_slot_patterns(cn, c3, NV, NQ):
    """patterns of J (P1 x P2-vector) and MP (P1 x P1) from the connectivity:
    ``(jkeys, jslots, pkeys, pslots)`` with ``jslots[c*36 + k*12 + 2m+b]`` /
    ``pslots[c*9 + k*3 + l]`` the CSR slot of the element entries of cell c
    (the layout `dnsb_assemble_stokes` expects)"""
    cn, c3 = np.asarray(cn, dtype=np.int64), np.asarray(c3, dtype=np.int64)
    nc = cn.shape[0]
    vd = np.stack([2*cn, 2*cn + 1], axis=2).reshape(nc, 12)
    return (_key_pattern(np.repeat(c3[:, :, None], 12, axis=2),
                         np.repeat(vd[:, None, :], 3, axis=1), NV) +
            _key_pattern(np.repeat(c3[:, :, None], 3, axis=2),
                         np.repeat(c3[:, None, :], 3, axis=1), NQ))


class ConvDevice(object):
    """mesh + convection kernels (K1a/K1b) bound to a P2 vector space

    A context holds ONE mesh at a time (``dnsb_set_mesh``); several function
    spaces may share a context, so every entry point re-binds its own mesh
    first if another space used the context in between.
    """

    def __init__(self, V, ctx=None):
        self.ctx = default_context() if ctx is None else ctx
        self.V = V
        mesh = V.mesh()
        gl, detj = V.geometry()
        geom = np.stack([gl[:, 1, 0], gl[:, 1, 1], gl[:, 2, 0], gl[:, 2, 1],
                         detj], axis=1)
        ncol, colour = V.colouring()
        self._cn = _i32(V.cell_nodes)
        self._geom = _f64(geom)
        self._colour = _i32(colour)
        self._ncell, self._nnodes = mesh.num_cells, V.num_nodes
        self.ncolours = ncol
        self.nvf = V.dim()
        self._pattern = None
        self._slots = None
        self.bind()

    def bind(self):
        """make this space's mesh (and pattern) the context's current one"""
        if getattr(self.ctx, '_mesh_owner', None) is self:
            return
        self.ctx.check(self.ctx.lib.dnsb_set_mesh(
            self.ctx.h, self._ncell, self._nnodes, _ip(self._cn),
            _dp(self._geom), self.ncolours, _ip(self._colour)))
        if self._pattern is not None:
            indptr, indices = self._pattern
            self.ctx.check(self.ctx.lib.dnsb_set_conv_pattern(
                self.ctx.h, _ip(indptr), _ip(indices), _ip(self._slots)))
        self.ctx._mesh_owner = self

    @property
    def pattern(self):
        """(indptr, indices) of the P2 vector space; uploads the cell slots"""
        if self._pattern is None:
            cn = self.V.cell_nodes.astype(np.int64)
            nc = cn.shape[0]
            NV = self.nvf
            vd = np.stack([2*cn, 2*cn + 1], axis=2).reshape(nc, 12)
            keys = (vd[:, :, None]*NV + vd[:, None, :]).reshape(-1)
            ukeys = np.unique(keys)
            rows = ukeys // NV
            indices = (ukeys % NV).astype(np.int32)
            indptr = np.zeros(NV + 1, dtype=np.int64)
            np.add.at(indptr, rows + 1, 1)
            indptr = np.cumsum(indptr).astype(np.int32)
            self._slots = np.searchsorted(ukeys, keys).astype(np.int32)
            self._pattern = (indptr, indices)
            self.ctx._mesh_owner = None      # force the upload of the pattern
        self.bind()
        return self._pattern

    def convvec(self, u1, u2=None):
        self.bind()
        u1 = _f64(u1)
        nb = 1 if u1.ndim == 1 else u1.shape[1]
        if u1.shape[0] != self.nvf:
            raise ValueError('convvec needs full vectors of size V.dim()')
        u2 = _f64(u2)
        out = np.empty_like(u1)
        self.ctx.check(self.ctx.lib.dnsb_convvec(self.ctx.h, _dp(u1), _dp(u2),
                                                 _dp(out), nb))
        return out

    def assemble_stokes(self, Q, nu=1., gradvsymmtrc=True):
        """M, A, J, JT, MP of `fem.assemble_stokes_operators` (no outflow
        correction) assembled on the device: per-cell kernel + gather into the
        fixed patterns (`dnsb_assemble_stokes`); zeros are kept"""
        import scipy.sparse as sps
        indptr, indices = self.pattern
        mesh = self.V.mesh()
        cn = self.V.cell_nodes.astype(np.int64)
        c3 = mesh.cells.astype(np.int64)
        NV, NQ = self.nvf, Q.dim()
        if getattr(self, '_stokes_slots', None) is None:   # once per mesh
            self._stokes_slots = stokes_slot_patterns(cn, c3, NV, NQ)
        jk, jslots, pk, pslots = self._stokes_slots
        _csr = _csr_from_keys
        mv, av = np.empty(indices.size), np.empty(indices.size)
        jv, pv = np.empty(jk.size), np.empty(pk.size)
        self.ctx.check(self.ctx.lib.dnsb_assemble_stokes(
            self.ctx.h, float(nu), int(bool(gradvsymmtrc)), jk.size,
            _ip(jslots), pk.size, _ip(pslots), _dp(mv), _dp(av), _dp(jv),
            _dp(pv)))
        # private copies of the pattern: callers compact the matrices in place
        # (`eliminate_zeros`, `dts:80`)
        M = sps.csr_matrix((mv, indices.copy(), indptr.copy()), shape=(NV, NV))
        A = sps.csr_matrix((av, indices.copy(), indptr.copy()), shape=(NV, NV))
        J = _csr(jk, NQ, NV, jv)
        JT = J.T.tocsr()
        JT.sort_indices()
        return dict(M=M, A=A, J=J, JT=JT, MP=_csr(pk, NQ, NQ, pv))

    def convmats(self, u0):
        indptr, indices = self.pattern
        u0 = _f64(u0).reshape(-1)
        n1 = np.empty(indices.size)
        n2 = np.empty(indices.size)
        f3 = np.empty(self.nvf)
        self.ctx.check(self.ctx.lib.dnsb_convmats(self.ctx.h, _dp(u0), _dp(n1),
                                                  _dp(n2), _dp(f3)))
        return n1, n2, f3


def device_for(V, ctx=None):
    """the (cached) device object of a function space, bound to its context"""
    dev = getattr(V, '_dnsb_dev', None)
    if dev is None or (ctx is not None and dev.ctx is not ctx):
        dev = ConvDevice(V, ctx)
        V._dnsb_dev = dev
    dev.bind()
    return dev


class SaddleSolver(object):
    """``dnsb_solver``: FGMRES for [[F_m, JT], [J, 0]] (see ``dnsb.h``)"""

    def __init__(self, ctx, fmat, jmat, jtmat, coef=None, nb=1, restart=40,
                 cheb_steps=3, lmin=None, lmax=None):
        self.ctx = ctx
        self.fmat, self.jmat, self.jtmat = fmat, jmat, jtmat
        self.nb = nb
        self.nv, self.np_ = fmat.shape[0], jmat.shape[0]
        coef = _f64(coef)
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.dnsb_solver_create(
            ctx.h, fmat.h, jmat.h, jtmat.h, _dp(coef), nb, restart, cheb_steps,
            float(lmin), float(lmax), ctypes.byref(h)))
        self.h = h
        self._levels = []

    def add_schur_level(self, amat=None, pmat=None, rmat=None, nsmooth=2,
                        lmin=0.0, lmax=0.0, dense_inv=None):
        dense_inv = _f64(dense_inv)
        self._levels.append((amat, pmat, rmat))
        self.ctx.check(self.ctx.lib.dnsb_solver_add_schur_level(
            self.h, amat.h if amat is not None else None,
            pmat.h if pmat is not None else None,
            rmat.h if rmat is not None else None, nsmooth, float(lmin),
            float(lmax), _dp(dense_inv)))

    def set_velocity_transfer(self, pmat, rmat):
        self._levels.append((pmat, rmat))
        self.ctx.check(self.ctx.lib.dnsb_solver_set_velocity_transfer(
            self.h, pmat.h, rmat.h))

    def add_velocity_level(self, amat=None, pmat=None, rmat=None, nsmooth=2,
                           lmin=0.0, lmax=0.0, dense_inv=None):
        dense_inv = _f64(dense_inv)
        self._levels.append((amat, pmat, rmat))
        self.ctx.check(self.ctx.lib.dnsb_solver_add_velocity_level(
            self.h, amat.h if amat is not None else None,
            pmat.h if pmat is not None else None,
            rmat.h if rmat is not None else None, nsmooth, float(lmin),
            float(lmax), _dp(dense_inv)))

    def set_schur_mass(self, mp_dinv, mp_scale):
        mp_dinv, mp_scale = _f64(mp_dinv), _f64(mp_scale)
        self.ctx.check(self.ctx.lib.dnsb_solver_set_schur_mass(
            self.h, _dp(mp_dinv), _dp(mp_scale)))

    def apply_prec(self, r):
        r = _f64(r).reshape(self.nv + self.np_, self.nb)
        z = np.empty_like(r)
        self.ctx.check(self.ctx.lib.dnsb_solver_apply_prec(self.h, _dp(r),
                                                           _dp(z)))
        return z

    def set_prec_mode(self, block_diagonal):
        self.ctx.check(self.ctx.lib.dnsb_solver_set_prec_mode(
            self.h, int(bool(block_diagonal))))

    def apply_k(self, x):
        """``K @ x`` for ``K = [[F, JT], [J, 0]]`` on the device"""
        x = _f64(x).reshape(self.nv + self.np_, self.nb)
        y = np.empty_like(x)
        self.ctx.check(self.ctx.lib.dnsb_solver_apply_k(self.h, _dp(x), _dp(y)))
        return y

    def update_fvalues(self, vals1):
        vals1 = _f64(vals1)
        if vals1.size != self.fmat.nnz:
            raise ValueError('values do not match the pattern of F')
        self.ctx.check(self.ctx.lib.dnsb_solver_update_fvalues(self.h,
                                                               _dp(vals1)))

    def set_schur_lsc(self, du_inv):
        du_inv = _f64(du_inv)
        self.ctx.check(self.ctx.lib.dnsb_solver_set_schur_lsc(self.h,
                                                              _dp(du_inv)))

    def solve(self, rhsv, rhsp=None, x0=None, tol=1e-11, maxit=400):
        """returns ``(vp, iters, relres)``; arrays are (n, nb) or (n,)"""
        rhsv = _f64(rhsv)
        flat = rhsv.ndim == 1
        rhsv = rhsv.reshape(self.nv, self.nb)
        rhsp = _f64(rhsp, (self.np_, self.nb)) if rhsp is not None else None
        x0 = _f64(x0, (self.nv + self.np_, self.nb)) if x0 is not None \
            else None
        vp = np.empty((self.nv + self.np_, self.nb))
        iters = np.zeros(self.nb, dtype=np.int32)
        relres = np.zeros(self.nb)
        self.ctx.check(self.ctx.lib.dnsb_solver_solve(
            self.h, _dp(rhsv), _dp(rhsp), _dp(x0), _dp(vp), float(tol),
            int(maxit), _ip(iters), _dp(relres)))
        return (vp.reshape(-1) if flat else vp), iters, relres

    def close(self):
        if self.h:
            self.ctx.lib.dnsb_solver_destroy(self.h)
            self.h = ctypes.c_void_p()


class ImexEngine(object):
    """``dnsb_imex``: device-resident CNAB / SBDF2 / IMEX-Euler loop"""
    SCHEMES = dict(cnab=0, sbdf2=1, imexeuler=2)

    def __init__(self, ctx, scheme, nb, dt, mmat, amat, jmat, jtmat, nu,
                 invinds, bcinds, bcvals, fv=None, fp=None):
        self.ctx = ctx
        self.nb = nb
        self.nv, self.np_ = mmat.shape[0], jmat.shape[0]
        self._keep = (mmat, amat, jmat, jtmat)
        nu = _f64(np.broadcast_to(np.asarray(nu, dtype=float), (nb,)))
        invinds, bcinds = _i32(invinds), _i32(bcinds)
        bcvals = _f64(bcvals)
        fv = _f64(fv, (-1,)) if fv is not None else None
        fp = _f64(fp, (-1,)) if fp is not None else None
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.dnsb_imex_create(
            ctx.h, self.SCHEMES[scheme], nb, float(dt), mmat.h, amat.h, jmat.h,
            jtmat.h, _dp(nu), _ip(invinds), invinds.size, bcinds.size,
            _ip(bcinds), _dp(bcvals), _dp(fv), _dp(fp), ctypes.byref(h)))
        self.h = h

    def set_solvers(self, loop, pred=None, corr=None):
        self._solvers = (loop, pred, corr)
        self.ctx.check(self.ctx.lib.dnsb_imex_set_solvers(
            self.h, loop.h, pred.h if pred else None, corr.h if corr else None))

    def set_forcing(self, bvecs, useries):
        """``f(t_n) = sum_k useries[n, k, m]*bvecs[:, k]``"""
        bvecs = _f64(bvecs).reshape(self.nv, -1)
        nk = bvecs.shape[1]
        useries = np.asarray(useries, dtype=float)
        if useries.ndim == 2:       # (ntimes, nk): shared by all members
            useries = useries[:, :, None]
        useries = _f64(np.broadcast_to(useries,
                                       (useries.shape[0], nk, self.nb)))
        self.ctx.check(self.ctx.lib.dnsb_imex_set_forcing(
            self.h, nk, _dp(bvecs), useries.shape[0], _dp(useries)))

    def set_state(self, v0, p0=None):
        v0 = _f64(np.broadcast_to(np.asarray(v0, dtype=float).
                                  reshape(self.nv, -1), (self.nv, self.nb)))
        if p0 is not None:
            p0 = _f64(np.broadcast_to(np.asarray(p0, dtype=float).
                                      reshape(self.np_, -1),
                                      (self.np_, self.nb)))
        self.ctx.check(self.ctx.lib.dnsb_imex_set_state(self.h, _dp(v0),
                                                        _dp(p0)))

    def run(self, nsteps, snap_stride=0, tol=1e-12, maxit=400, guess=16,
            check_ff_maxv=1e8, ntimeslices=10, allow_unconverged=False):
        """raises `NotConverged` if a solve of the run stopped at ``maxit``
        above ``tol`` (``allow_unconverged=True``: only `stats()` tells)"""
        ff = ctypes.c_int(0)
        rc = self.ctx.lib.dnsb_imex_run(
            self.h, int(nsteps), int(snap_stride), float(tol), int(maxit),
            int(guess), float(check_ff_maxv), int(ntimeslices),
            ctypes.byref(ff))
        if not (allow_unconverged and rc == E_NOT_CONVERGED):
            self.ctx.check(rc)
        return ff.value

    def set_member_guard(self, on):
        """per-member blow-up guard (``dnsb_imex_set_member_guard``)"""
        self.ctx.check(self.ctx.lib.dnsb_imex_set_member_guard(self.h,
                                                               int(bool(on))))

    def member_status(self):
        """trip level of every member, -1 while it is live"""
        t = np.empty(self.nb, dtype=np.int32)
        self.ctx.check(self.ctx.lib.dnsb_imex_member_status(self.h, _ip(t)))
        return t

    def set_statistics(self, on):
        """in-loop field statistics (``dnsb_imex_set_statistics``)"""
        self.ctx.check(self.ctx.lib.dnsb_imex_set_statistics(self.h,
                                                             int(bool(on))))

    def reset_statistics(self):
        self.ctx.check(self.ctx.lib.dnsb_imex_reset_statistics(self.h))

    def statistics(self, nnodes):
        """``dnsb_imex_get_statistics`` in the device numbering: dict of
        ``first``, ``last``, ``count`` (nb,), ``v_mean`` (nvf, nb), ``uvcov``
        (3, nnodes, nb), ``p_mean`` / ``p_var`` (np, nb), ``c_mean`` (nv, nb)"""
        nb = self.nb
        first, last = _ll(), _ll()
        count = np.empty(nb, dtype=np.int64)
        out = dict(v_mean=np.empty((2*nnodes, nb)),
                   uvcov=np.empty((3, nnodes, nb)),
                   p_mean=np.empty((self.np_, nb)),
                   p_var=np.empty((self.np_, nb)),
                   c_mean=np.empty((self.nv, nb)))
        self.ctx.check(self.ctx.lib.dnsb_imex_get_statistics(
            self.h, ctypes.byref(first), ctypes.byref(last),
            count.ctypes.data_as(ctypes.POINTER(_ll)), _dp(out['v_mean']),
            _dp(out['uvcov']), _dp(out['p_mean']), _dp(out['p_var']),
            _dp(out['c_mean'])))
        out.update(first=first.value, last=last.value, count=count)
        return out

    def last_run_ms(self):
        return float(self.ctx.lib.dnsb_imex_last_run_ms(self.h))

    def state(self):
        v = np.empty((self.nv, self.nb))
        p = np.empty((self.np_, self.nb))
        self.ctx.check(self.ctx.lib.dnsb_imex_get_state(self.h, _dp(v),
                                                        _dp(p)))
        return v, p

    def snapshots(self):
        ns = self.ctx.lib.dnsb_imex_num_snapshots(self.h)
        out = np.empty((ns, self.nv + self.np_, self.nb))
        if ns > 0:
            self.ctx.check(self.ctx.lib.dnsb_imex_get_snapshots(self.h,
                                                                _dp(out)))
        return out

    def set_output_order(self, vmap, pmap):
        vmap, pmap = _i32(vmap), _i32(pmap)
        self.ctx.check(self.ctx.lib.dnsb_imex_set_output_order(
            self.h, _ip(vmap), _ip(pmap)))

    def reserve_snapshots(self, nsnap):
        self.ctx.check(self.ctx.lib.dnsb_imex_reserve_snapshots(self.h,
                                                                int(nsnap)))

    def snapshots_view(self):
        """zero-copy (nsnap, nv+np, nb) view of the pinned host mirror; valid
        until the next run / reserve / close"""
        ptr, ns = c_dbl_p(), ctypes.c_int(0)
        self.ctx.check(self.ctx.lib.dnsb_imex_snapshots_host(
            self.h, ctypes.byref(ptr), ctypes.byref(ns)))
        if ns.value == 0:
            return np.empty((0, self.nv + self.np_, self.nb))
        return np.ctypeslib.as_array(ptr, shape=(ns.value, self.nv + self.np_,
                                                 self.nb))

    def reset_snapshots(self):
        self.ctx.check(self.ctx.lib.dnsb_imex_reset_snapshots(self.h))

    def set_outputs(self, cv=None, cp=None):
        """linear output rows (`Csr`, device column numbering) or None; the
        engine copies them"""
        self.ctx.check(self.ctx.lib.dnsb_imex_set_outputs(
            self.h, cv.h if cv is not None else None,
            cp.h if cp is not None else None))

    def set_force(self, dofs=None, fm=None, fa=None, fj=None, fa_bc=None):
        """force rows (`Csr`) on the full-numbering ``dofs``; None: off"""
        dofs = _i32(np.zeros(0) if dofs is None else dofs)
        fa_bc = _f64(fa_bc, (-1,))
        self.ctx.check(self.ctx.lib.dnsb_imex_set_force(
            self.h, dofs.size, _ip(dofs), fm.h if fm is not None else None,
            fa.h if fa is not None else None, fj.h if fj is not None else None,
            _dp(fa_bc)))

    def outputs(self, ny):
        """``(y (levels, ny, nb), force (levels, 2, nb))``"""
        nl = self.ctx.lib.dnsb_imex_num_output_levels(self.h)
        y = np.empty((nl, ny, self.nb))
        f = np.empty((nl, 2, self.nb))
        if nl > 0:
            self.ctx.check(self.ctx.lib.dnsb_imex_get_outputs(self.h, _dp(y),
                                                              _dp(f)))
        return y, f

    def reset_outputs(self):
        self.ctx.check(self.ctx.lib.dnsb_imex_reset_outputs(self.h))

    def stats(self):
        it, ns, rr = _ll(), _ll(), ctypes.c_double()
        self.ctx.check(self.ctx.lib.dnsb_imex_stats(
            self.h, ctypes.byref(it), ctypes.byref(ns), ctypes.byref(rr)))
        unc = int(self.ctx.lib.dnsb_imex_unconverged(self.h))
        return dict(iters=it.value, solves=ns.value, max_relres=rr.value,
                    last_relres=rr.value, unconverged=unc)

    def gram(self):
        """local POD Gram matrix ``sum_m X_m^T M X_m`` as a numpy array"""
        ns = self.ctx.lib.dnsb_imex_num_snapshots(self.h)
        g = np.empty((ns, ns))
        self.ctx.check(self.ctx.lib.dnsb_imex_gram(self.h, _dp(g)))
        return g

    def gram_dev(self, g_dev_ptr):
        self.ctx.check(self.ctx.lib.dnsb_imex_gram_dev(
            self.h, ctypes.c_void_p(int(g_dev_ptr))))

    def close(self):
        if self.h:
            self.ctx.lib.dnsb_imex_destroy(self.h)
            self.h = ctypes.c_void_p()


class CnSweep(object):
    """``dnsb_cnsweep``: device-resident Picard/Newton + Crank-Nicolson sweep"""

    def __init__(self, solver, mmat, mvals, avals, src, pos, invinds, bcinds,
                 bcvals, fv, fp, nvf):
        self.ctx = solver.ctx
        self.solver, self.mmat = solver, mmat
        self.nv, self.np_, self.nvf = solver.nv, solver.np_, int(nvf)
        mvals, avals = _f64(mvals), _f64(avals)
        src, pos = _i32(src), _i32(pos)
        invinds, bcinds = _i32(invinds), _i32(bcinds)
        bcvals = _f64(bcvals)
        fv, fp = _f64(fv, (-1,)), _f64(fp, (-1,))
        h = ctypes.c_void_p()
        self.ctx.check(self.ctx.lib.dnsb_cnsweep_create(
            solver.h, mmat.h, _dp(mvals), _dp(avals), src.size, _ip(src),
            _ip(pos), _ip(invinds), bcinds.size, _ip(bcinds), _dp(bcvals),
            _dp(fv), _dp(fp), ctypes.byref(h)))
        self.h = h

    def run(self, dts, linpoint, v0, p0, picard, tol=1e-12, maxit=2000):
        """returns ``(vtraj (n+1, V.dim()), ptraj (n+1, NP), upd_norm, iters)``"""
        dts = _f64(dts)
        n = dts.size
        linpoint = _f64(linpoint, (n + 1, self.nvf))
        v0 = _f64(v0, (-1,))
        p0 = _f64(p0, (-1,)) if p0 is not None else None
        vtraj = np.empty((n + 1, self.nvf))
        ptraj = np.empty((n + 1, self.np_))
        nrm, its = ctypes.c_double(0.), _ll(0)
        self.ctx.check(self.ctx.lib.dnsb_cnsweep_run(
            self.h, n, _dp(dts), int(bool(picard)), _dp(linpoint), _dp(v0),
            _dp(p0), float(tol), int(maxit), _dp(vtraj), _dp(ptraj),
            ctypes.byref(nrm), ctypes.byref(its)))
        return vtraj, ptraj, nrm.value, its.value

    def set_guess(self, krylovini):
        """``'old'``: previous solution, ``'upd'`` / None: extrapolation
        (`snu:1493-1503`)"""
        mode = dict(old=0, upd=1)[krylovini or 'upd']
        self.ctx.check(self.ctx.lib.dnsb_cnsweep_set_guess(self.h, mode))

    def stats(self):
        rr, unc = ctypes.c_double(0.), _ll(0)
        self.ctx.check(self.ctx.lib.dnsb_cnsweep_stats(
            self.h, ctypes.byref(rr), ctypes.byref(unc)))
        return dict(max_relres=rr.value, unconverged=unc.value)

    def close(self):
        if self.h:
            self.ctx.lib.dnsb_cnsweep_destroy(self.h)
            self.h = ctypes.c_void_p()
