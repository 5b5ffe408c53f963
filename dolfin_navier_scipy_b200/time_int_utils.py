"""IMEX time integration on the device.

Mirrors `dolfin_navier_scipy/time_int_utils.py`: `cnab` (`tiu:23-145`),
`sbdftwo` (`tiu:260-355`), `semi_implicit_euler` (`tiu:566-635`).  The whole
loop body of `tiu:104-143` -- convection re-evaluation, right-hand side, saddle
point solve, blow-up guard -- runs inside ``libdnsb200`` (``dnsb_imex_run``);
the host only sets up operators and preconditioners once.

The reference passes the convection term as an opaque Python callback
(``f_vdp``).  The device loop needs to know what that callback does, so the
integrators take the function space and boundary data instead (``V``,
``invinds``, ``dbcinds``, ``dbcvals``), which is what `snu.solve_nse` has at
hand when it builds the callback (`stokes_navier_utils.py:1136-1140`).
"""
import numpy as np
import scipy.sparse as sps

from . import _lib
from . import hostsetup

__all__ = ['cnab', 'sbdftwo', 'semi_implicit_euler', 'DeviceImex',
           'lowrank_forcing', 'get_heunab_lti', 'get_heuntrpz_lti']

_THETA = dict(cnab=.5, sbdf2=2./3, imexeuler=1.)


def _on_pattern(X, pat):
    """values of ``X`` on the (larger) CSR pattern of ``pat`` (explicit zeros)"""
    pat = sps.csr_matrix(pat)
    X = sps.coo_matrix(X)
    pc = pat.tocoo()
    rows = np.concatenate([pc.row, X.row])
    cols = np.concatenate([pc.col, X.col])
    vals = np.concatenate([np.zeros(pc.nnz), X.data])
    out = sps.coo_matrix((vals, (rows, cols)), shape=pat.shape).tocsr()
    out.sum_duplicates()
    out.sort_indices()
    if out.nnz != pat.nnz:
        raise ValueError('matrix does not fit the given pattern')
    return out


def _union_pattern(mats):
    acc = None
    for m in mats:
        m = sps.csr_matrix(m)
        p = sps.csr_matrix((np.ones(m.nnz), m.indices, m.indptr),
                           shape=m.shape)
        acc = p if acc is None else acc + p
    acc = acc.tocsr()
    acc.sort_indices()
    return acc


def lowrank_forcing(fvtd, trange, nv, maxrank=64, tol=1e-13, chunk=256):
    """sample ``fvtd(t)`` on ``trange`` and factor it as ``B @ U``

    The device loop evaluates ``f(t_n) = sum_k U[k, n] B[:, k]``; separable
    forcings such as ``sin(t)*b`` (`tests/time_dep_nse_bcrob.py:33-34`) have
    rank 1.  The samples are taken ``chunk`` time levels at a time against an
    orthonormal basis that grows with what the chunk adds, so the memory is
    ``nv*(rank + chunk)`` whatever the number of steps, and a forcing of rank
    > ``maxrank`` raises ``NotImplementedError`` at the first chunk that shows
    it, not after all samples have been evaluated.
    """
    trange = np.asarray(trange, dtype=float)
    nt = trange.size
    Q = np.zeros((nv, 0))
    coeffs = []            # per chunk: (rank at that time, chunk length)
    scale = 0.
    for c0 in range(0, nt, chunk):
        Fc = np.hstack([np.asarray(fvtd(t), dtype=float).reshape(nv, 1)
                        for t in trange[c0:c0 + chunk]])
        scale = max(scale, np.abs(Fc).max() if Fc.size else 0.)
        C = Q.T@Fc
        R = Fc - Q@C
        C2 = Q.T@R                      # second pass: keeps Q orthonormal
        R -= Q@C2
        C += C2
        # what the chunk adds: left singular vectors of the remainder
        if R.size and np.abs(R).max() > 0.:
            uu, ss, vv = np.linalg.svd(R, full_matrices=False)
            ref = max(ss[0], np.linalg.norm(C, 2) if C.size else 0.)
            r = int(np.sum(ss > tol*ref))
            if Q.shape[1] + r > maxrank:
                raise NotImplementedError(
                    'time dependent forcing of rank > {0} (seen after {1} of '
                    '{2} time levels)'.format(maxrank, min(nt, c0 + chunk), nt))
            if r:
                Q = np.hstack([Q, uu[:, :r]])
                C = np.vstack([C, ss[:r, None]*vv[:r, :]])
        coeffs.append(C)
    if scale == 0.:
        return np.zeros((nv, 1)), np.zeros((nt, 1))
    r = Q.shape[1]
    U = np.zeros((r, nt))
    c0 = 0
    for C in coeffs:
        U[:C.shape[0], c0:c0 + C.shape[1]] = C
        c0 += C.shape[1]
    # rotate to the principal directions and drop what is numerically zero
    uu, ss, vv = np.linalg.svd(U, full_matrices=False)
    keep = int(np.sum(ss > tol*ss[0]))
    B = Q@uu[:, :keep]
    return B, (ss[:keep, None]*vv[:keep, :]).T.copy()


class DeviceImex(object):
    """device-resident IMEX integrator for ``nb`` trajectories on one mesh

    ``A_m = nus[m]*A0 + Arob``; all members share M, J, the mesh, the pattern
    and the boundary data.  For a single trajectory pass ``A0=A, nus=[1.]``.
    """

    def __init__(self, M, A0, J, V, invinds, dbcinds, dbcvals, dt,
                 scheme='cnab', nus=(1.,), Arob=None, fv=None, fp=None,
                 ctx=None, cheb_steps=4, restart=40, coarse_max=4096,
                 mp_diag=None, reorder=True, schur_poly=2):
        self.ctx = _lib.default_context() if ctx is None else ctx
        self.scheme = scheme
        self.dt = float(dt)
        self.nus = np.atleast_1d(np.asarray(nus, dtype=float))
        self.nb = self.nus.size
        self.V = V
        self.invinds = np.asarray(invinds, dtype=np.int32)
        M, A0, J = sps.csr_matrix(M), sps.csr_matrix(A0), sps.csr_matrix(J)
        self.NP, self.NV = J.shape
        # ---- device numbering: Hilbert order of the mesh nodes (locality of
        # the SpMM gathers); all inputs/outputs are permuted at this boundary
        reorder = reorder and hasattr(V, 'tabulate_dof_coordinates')
        if reorder:
            xy = np.asarray(V.tabulate_dof_coordinates())[self.invinds]
            self.pv = hostsetup.locality_perm(xy, comp=self.invinds % 2)
            pxy = np.asarray(V.mesh().coords)
            if pxy.shape[0] == self.NP:
                self.pp = hostsetup.locality_perm(pxy)
            else:
                self.pp = hostsetup.locality_perm(pattern=abs(J)@abs(J).T)
        else:
            self.pv, self.pp = np.arange(self.NV), np.arange(self.NP)
        pv, pp = self.pv, self.pp
        self.ipv, self.ipp = np.argsort(pv), np.argsort(pp)

        def _pvv(X):
            return sps.csr_matrix(X)[pv][:, pv].tocsr()
        M, A0 = _pvv(M), _pvv(A0)
        J = J[pp][:, pv].tocsr()
        Arob = None if Arob is None else _pvv(Arob)
        mats = [M, A0] + ([] if Arob is None else [Arob])
        pat = _union_pattern(mats)
        if reorder:
            pat = hostsetup.pad_row_pairs(pat)
        Mp, A0p = _on_pattern(M, pat), _on_pattern(A0, pat)
        Arp = _on_pattern(sps.csr_matrix(pat.shape) if Arob is None else Arob,
                          pat)
        self._host = dict(M=Mp, A0=A0p, Arob=Arp, J=J)
        # Dirichlet data: unique indices, last write wins (`dts:534-535`)
        aux = {}
        for i, v in zip(dbcinds, dbcvals):
            aux[int(i)] = float(v)
        bci = np.array(sorted(aux.keys()), dtype=np.int32)
        bcv = np.array([aux[i] for i in bci], dtype=float)
        self._bcs = (bci, bcv)
        self.ny = 0
        self.dev = _lib.device_for(V, self.ctx)
        ctx = self.ctx
        self.mmat = ctx.csr(Mp)
        self.amat = ctx.csr(Arp, A0p.data)
        JT = J.T.tocsr()
        JT.sort_indices()
        if reorder:
            JT = _on_pattern(JT, hostsetup.pad_row_pairs(JT))
        self.jmat, self.jtmat = ctx.csr(J), ctx.csr(JT)
        if fv is not None:
            fv = np.asarray(fv, dtype=float).reshape(self.NV, -1)[pv]
        if fp is not None:
            fp = np.asarray(fp, dtype=float).reshape(self.NP, -1)[pp]
        self.engine = _lib.ImexEngine(ctx, scheme, self.nb, self.dt,
                                      self.mmat, self.amat, self.jmat,
                                      self.jtmat, self.nus,
                                      self.invinds[pv], bci, bcv, fv=fv, fp=fp)
        self.engine.set_output_order(pv, pp)
        # ---- solvers: loop (tau = theta*dt), Heun predictor (dt), corr (0) --
        theta = _THETA[scheme]
        taus = [theta*self.dt] if scheme == 'imexeuler' \
            else [theta*self.dt, self.dt, 0.]
        self.solvers, self.infos = [], []
        hierarchy = None
        numean = float(np.mean(self.nus))
        for tau in taus:
            F1 = sps.csr_matrix((Mp.data + tau*Arp.data, Mp.indices,
                                 Mp.indptr), shape=Mp.shape)
            mpd = None if mp_diag is None or tau == 0. else \
                np.asarray(mp_diag)[pp]
            if hierarchy is None:
                # Schur approximation J Z J.T of the mean member's loop matrix
                Fm = sps.csr_matrix((F1.data + tau*numean*A0p.data,
                                     F1.indices, F1.indptr), shape=F1.shape)
                S = hostsetup.poly_schur(Fm, J, k=schur_poly)
                hierarchy = hostsetup.sa_amg_hierarchy(S,
                                                       coarse_max=coarse_max)
            s, info = hostsetup.make_saddle_solver(
                ctx, F1, J, JT, F2=A0p, coef=tau*self.nus, nb=self.nb,
                restart=restart, cheb_steps=cheb_steps, hierarchy=hierarchy,
                mp_diag=mpd,
                mp_scale=None if mpd is None else tau*self.nus)
            self.solvers.append(s)
            self.infos.append(info)
        self.engine.set_solvers(*self.solvers)

    def set_forcing(self, B, U):
        B = np.asarray(B, dtype=float).reshape(self.NV, -1)
        self.engine.set_forcing(B[self.pv], U)

    def set_state(self, v0, p0=None):
        v0 = np.asarray(v0, dtype=float).reshape(self.NV, -1)[self.pv]
        if p0 is not None:
            p0 = np.asarray(p0, dtype=float).reshape(self.NP, -1)[self.pp]
        self.engine.set_state(v0, p0)

    def run(self, nsteps, **kw):
        self.dev.bind()       # the loop assembles the convection on this mesh
        return self.engine.run(nsteps, **kw)

    def state(self):
        v, p = self.engine.state()
        return v[self.ipv], p[self.ipp]

    def snapshots(self, copy=True):
        """(nsnap, NV, nb) velocities and (nsnap, NP, nb) pressures in the
        caller's numbering; ``copy=False``: views of the pinned host mirror
        (valid until the next run)"""
        s = self.engine.snapshots() if copy else self.engine.snapshots_view()
        return s[:, :self.NV, :], s[:, self.NV:, :]

    def set_outputs(self, cv_mat=None, cp_mat=None, force_dofs=None,
                    force_ops=None):
        """record output functionals at every time level inside the loop

        ``y_n = cv_mat v_n + cp_mat p_n`` (``cv_mat`` ny x NV on the inner
        velocity, ``cp_mat`` ny x NP, the caller's numbering; the reference's
        ``cv_mat.dot(v)``) and, with ``force_dofs`` (full velocity dofs such
        as ``ldsbcinds``; CNAB only), the raw x / y force: the CNAB residual
        of `residual_checks.get_imex_res` with ``nu = nus[m]`` tested with
        their indicator.  ``force_ops``: the uncondensed nu = 1 ``M``, ``A``,
        ``JT`` (`dts.get_stokessysmats`), built from ``V`` if omitted.  No
        argument switches the outputs off.  Read them with `outputs`.
        """
        from . import residual_checks
        cv = None if cv_mat is None else sps.csr_matrix(cv_mat)
        cp = None if cp_mat is None else sps.csr_matrix(cp_mat)
        if cv is not None and cv.shape[1] != self.NV:
            raise ValueError('cv_mat must have NV = {0} columns, not {1}'.
                             format(self.NV, cv.shape[1]))
        if cp is not None and cp.shape[1] != self.NP:
            raise ValueError('cp_mat must have NP = {0} columns, not {1}'.
                             format(self.NP, cp.shape[1]))
        if cv is not None and cp is not None and cv.shape[0] != cp.shape[0]:
            raise ValueError('cv_mat and cp_mat must have the same rows')
        if force_dofs is not None and self.scheme != 'cnab':
            raise NotImplementedError(
                'forces are the CNAB residual (`get_imex_res`, crni/abtw); '
                'scheme {0!r} has none'.format(self.scheme))
        rows = None
        if force_dofs is not None:
            rows = residual_checks.get_imex_force_rows(
                V=self.V, invinds=self.invinds, dbcinds=self._bcs[0],
                dbcvals=self._bcs[1], ldsbcinds=force_dofs,
                force_ops=force_ops)
        ctx, pv, pp = self.ctx, self.pv, self.pp
        mats = [None if cv is None else ctx.csr(cv[:, pv]),
                None if cp is None else ctx.csr(cp[:, pp])]
        if rows is not None:
            mats += [ctx.csr(rows['fm'][:, pv]), ctx.csr(rows['fa'][:, pv]),
                     ctx.csr(rows['fj'][:, pp])]
        try:
            self.engine.set_outputs(*mats[:2])
            if rows is None:
                self.engine.set_force()
            else:
                self.engine.set_force(rows['dofs'], *mats[2:],
                                      fa_bc=rows['fa_bc'])
        finally:
            for m in mats:              # the engine keeps its own copy
                if m is not None:
                    m.close()
        self.ny = 0 if cv is None and cp is None else \
            (cv if cv is not None else cp).shape[0]

    def outputs(self):
        """``dict(y=(levels, ny, nb), force=(levels, 2, nb))`` recorded since
        `set_state` / `reset_outputs` (members in the order of ``nus``; the
        force is NaN at levels 0 and 1)"""
        y, f = self.engine.outputs(self.ny)
        return dict(y=y, force=f)

    def reset_outputs(self):
        """start a new record (the next run first records the current state)"""
        self.engine.reset_outputs()

    def reserve_snapshots(self, nsnap):
        self.engine.reserve_snapshots(nsnap)

    def stats(self):
        return self.engine.stats()

    def gram(self):
        """POD snapshot Gram matrix ``sum_m X_m^T M X_m`` of this shard (numpy)"""
        return self.engine.gram()

    def close(self):
        self.engine.close()
        for s in self.solvers:
            s.close()


def _run_imex(scheme, trange=None, inivel=None, inip=None, M=None, A=None,
              J=None, f_tdp=None, g_tdp=None, scalep=-1., V=None,
              invinds=None, dbcinds=None, dbcvals=None, savevp=None,
              check_ff_maxv=1e8, ntimeslices=10, tol=1e-12, maxit=400,
              guess=16, cheb_steps=4, f_vdp='convection', ctx=None,
              return_engine=False, **kw):
    if f_vdp != 'convection' and f_vdp is not None:
        raise NotImplementedError(
            'the device loop assembles the P2 convection itself; a foreign '
            '`f_vdp` callback cannot run on the device')
    if scalep != -1.:
        raise NotImplementedError('scalep != -1')
    trange = np.asarray(trange, dtype=float)
    dtv = np.diff(trange)
    if not np.allclose(np.linalg.norm(np.diff(dtv)), 0):
        raise NotImplementedError()                      # `tiu:358-363`
    dt = trange[1] - trange[0]
    NP, NV = J.shape
    fv0 = np.zeros((NV, 1)) if f_tdp is None else None
    B = U = None
    if f_tdp is not None:
        B, U = lowrank_forcing(f_tdp, trange, NV)
    fp = np.zeros((NP, 1)) if g_tdp is None else \
        np.asarray(g_tdp(trange[0]), dtype=float).reshape(NP, 1)
    if g_tdp is not None:
        # the reference evaluates `g_tdp(ctime)` every step (`tiu:120,337,391`);
        # the device loop holds ONE continuity right-hand side
        for t in trange[1:]:
            if not np.array_equal(np.asarray(g_tdp(t), dtype=float).
                                  reshape(NP, 1), fp):
                raise NotImplementedError(
                    'time dependent continuity right-hand side `g_tdp`')
    integ = DeviceImex(M, A, J, V, invinds, dbcinds, dbcvals, dt,
                       scheme=scheme, nus=(1.,), fv=fv0, fp=fp, ctx=ctx,
                       cheb_steps=cheb_steps)
    if B is not None:
        integ.set_forcing(B, U)
    integ.set_state(inivel, inip)
    nsteps = trange.size - 1
    stride = 1 if savevp is not None else 0
    ffflag = integ.run(nsteps, snap_stride=stride, tol=tol, maxit=maxit,
                       guess=guess, check_ff_maxv=check_ff_maxv,
                       ntimeslices=ntimeslices)
    v_n, p_n = integ.state()
    if savevp is not None:
        from .dolfin_to_sparrays import append_bcs_vec
        vs, ps = integ.snapshots()
        for k in range(vs.shape[0]):
            vfull = append_bcs_vec(vs[k, :, :1], V=V, invinds=invinds,
                                   bcinds=dbcinds, bcvals=dbcvals)
            savevp(vfull, ps[k, :, :1], time=trange[k])
    if return_engine:
        return v_n, p_n, ffflag, integ
    integ.close()
    return v_n, p_n, ffflag


def _needs_host_hop(kw):
    """opaque callbacks (`tiu:23-38`: ``f_vdp``, ``f_tvdp``, ``dynamic_rhs``,
    ``getbcs`` / ``applybcs``) cannot run inside the CUDA loop"""
    if callable(kw.get('f_vdp', 'convection')) or \
            kw.get('f_vdp', 'convection') is None:
        return True
    if any(kw.get(k) is not None for k in ('f_tvdp', 'dynamic_rhs', 'getbcs',
                                           'applybcs')):
        return True
    return kw.get('V') is None


def cnab(**kw):
    """Crank-Nicolson/Adams-Bashforth -- `tiu:23-145`

    ``cnab(trange=, inivel=, inip=, M=, A=, J=, f_tdp=, g_tdp=, V=, invinds=,
    dbcinds=, dbcvals=, savevp=, check_ff_maxv=, ntimeslices=)`` runs the whole
    loop on the device (the convection is the P2 form of ``V``) and returns
    ``(v_n, p_n, ffflag)`` like the reference.  With the reference's callback
    arguments (``f_vdp`` callable or ``None`` = no nonlinearity, ``f_tvdp``,
    ``dynamic_rhs``, ``getbcs``/``applybcs``/``appndbcs``) the loop runs on the
    host with every solve on the device (`hosthop.imex_with_callbacks`).
    """
    if _needs_host_hop(kw):
        from . import hosthop
        return hosthop.imex_with_callbacks('cnab', **kw)
    return _run_imex('cnab', **kw)


def sbdftwo(**kw):
    """SBDF2 -- `tiu:260-355` (device loop or host hop like `cnab`)"""
    if _needs_host_hop(kw):
        from . import hosthop
        return hosthop.imex_with_callbacks('sbdf2', **kw)
    return _run_imex('sbdf2', **kw)


def get_heunab_lti(hb=None, ha=None, hc=None, inihx=None, drift=None):
    """Heun/AB2 discretisation of a linear observer ``hx' = ha hx + hb y +
    drift(t)``, ``u = hc hx`` as a ``dynamic_rhs`` callback (`tiu:148-198`)

    The returned function is called by the integrators with
    ``mode in {'init', 'heunpred', 'heuncorr', 'abtwo'}`` and threads its state
    through ``memory`` exactly like the reference's.
    """
    def f(x, y, t):
        return ha@x + hb@y + drift(t)

    def observer(t, vc=None, memory={}, mode='abtwo'):
        if mode == 'init':
            memory.update(lastt=t, lasthx=inihx)
            return hc@inihx, memory
        h = t - memory['lastt']
        if mode == 'heunpred':                 # explicit Euler from the start value
            rate = f(inihx, vc, memory['lastt'])
            x = inihx + h*rate
            memory.update(lastrhs=rate, hphx=x)
        elif mode == 'heuncorr':               # trapezoidal average of the two rates
            x = inihx + .5*h*(f(memory['hphx'], vc, t) + memory['lastrhs'])
            memory.update(lastt=t, lasthx=x, lastdt=h)
        else:                                  # AB2 on a (possibly) varying step
            rate = f(memory['lasthx'], vc, memory['lastt'])
            x = memory['lasthx'] + 1.5*h*rate \
                - .5*memory['lastdt']*memory['lastrhs']
            memory.update(lastt=t, lasthx=x, lastrhs=rate, lastdt=h)
        return hc@x, memory
    return observer


def get_heuntrpz_lti(hb=None, ha=None, hc=None, inihx=None, drift=None,
                     constdt=None):
    """Heun / implicit trapezoidal discretisation of the same observer on a
    uniform grid (`tiu:201-257`): ``(I - dt/2 ha) x+ = x + dt/2 (ha x + r + r-)``
    with ``r = hb y + drift(t)``"""
    if constdt is None:
        raise NotImplementedError()
    dt = constdt
    step = np.linalg.inv(np.eye(ha.shape[0]) - .5*dt*ha)

    def observer(t, vc=None, memory={}, mode='abtwo'):
        if mode == 'init':
            memory.update(lastt=t, lasthx=inihx)
            return hc@inihx, memory
        r = hb@vc + drift(t)
        if mode == 'heunpred':
            x = inihx + dt*(ha@inihx + r)
            memory.update(lastrhs=r, lasthx=inihx, hphx=x)
        elif mode == 'heuncorr':
            x = inihx + .5*dt*(ha@(memory['hphx'] + memory['lasthx'])
                               + r + memory['lastrhs'])
            memory.update(lastt=t, hchx=x)
        else:
            x0 = memory['lasthx']
            x = step@(x0 + .5*dt*(ha@x0 + r + memory['lastrhs']))
            memory.update(lasthx=x, lastrhs=r)
        return hc@x, memory
    return observer


def semi_implicit_euler(iniv=None, jmat=None, mmat=None, amat=None, rhsv=None,
                        trange=None, data_trange=None, fp=None, V=None,
                        invinds=None, dbcinds=None, dbcvals=None, fv=None,
                        fvtd=None, **kw):
    """IMEX Euler with the P2 convection treated explicitly -- `tiu:566-635`

    The reference takes an opaque ``rhsv(t, v)``; on the device the right hand
    side is ``fv + fvtd(t) - N(v)v`` (pass ``fv``/``fvtd``), the use the
    reference's scripts make of it.  Returns the list of velocities at
    ``data_trange``.
    """
    if rhsv is not None:
        # the reference's interface: an opaque right-hand side, per-step host hop
        from . import hosthop
        return hosthop.euler_with_callbacks(
            iniv=iniv, jmat=jmat, mmat=mmat, amat=amat, rhsv=rhsv,
            trange=trange, data_trange=data_trange, fp=fp,
            **{k: v for k, v in kw.items() if k in ('tol', 'maxit', 'ctx')})
    trange = np.asarray(trange, dtype=float)
    NP, NV = jmat.shape
    integ = DeviceImex(mmat, amat, jmat, V, invinds, dbcinds, dbcvals,
                       trange[1] - trange[0], scheme='imexeuler', nus=(1.,),
                       fv=np.zeros((NV, 1)) if fv is None else fv,
                       fp=np.zeros((NP, 1)) if fp is None else fp)
    if fvtd is not None:
        integ.set_forcing(*lowrank_forcing(fvtd, trange, NV))
    integ.set_state(iniv)
    integ.run(trange.size - 1, snap_stride=1, ntimeslices=0,
              **{k: v for k, v in kw.items() if k in ('tol', 'maxit', 'guess')})
    vs, _ = integ.snapshots()
    integ.close()
    dtr = trange if data_trange is None else np.asarray(data_trange)
    idx = [int(np.argmin(np.abs(trange - t))) for t in dtr]
    return [vs[k, :, :1] for k in idx]
