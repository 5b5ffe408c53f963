"""weak residuals of the discrete Navier-Stokes equations -- mirrors
`dolfin_navier_scipy/residual_checks.py` (`rck:40-103`) without dolfin.

The reference assembles UFL forms of dolfin functions; here velocities,
pressures and test functions are coefficient vectors on ALL dofs (boundary
values included) and the forms are evaluated as

    diffusion   nu*(grad v + grad v^T, grad phi) - outflow correction  =  phi^T A_full v
    convection  ((v.grad) v, phi)                                      =  phi^T c(v)   (device, K1a)
    pressure    (p, div phi)                                           =  phi^T JT_full p
    mass        (v, phi)                                               =  phi^T M_full v

with the uncondensed operators of `dts.get_stokessysmats`.  Testing with the
indicator of the obstacle's dofs gives drag and lift
(`tests/steadystate_schaefer-turek_2D-1.py:71-85`).
"""
import numpy as np
import scipy.sparse as sps

from . import dolfin_to_sparrays as dts
from . import fem

__all__ = ['get_steady_state_res', 'get_imex_res', 'get_imex_force_rows',
           'lift_drag_via_residual']


def _flat(vec):
    return np.asarray(vec, dtype=float).reshape(-1)


def _operators(V, outflowds, gradvsymmtrc, nu, device):
    Q = fem.P1Space(V.mesh())
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):       # the notes of `dts:231-235`
        sm = dts.get_stokessysmats(V, Q, nu=nu, gradvsymmtrc=gradvsymmtrc,
                                   outflowds=outflowds, device=device)
    return sm


def _conv(V, vel):
    return _flat(dts.get_convvec(u0_vec=_flat(vel).reshape(-1, 1), V=V))


def _test(res, phi):
    return res if phi is None else float(_flat(phi)@res)


def get_steady_state_res(V=None, outflowds=None, gradvsymmtrc=True, nu=None,
                         device=False):
    """``steady_state_res(vel, pres, phi=None)``: ``diffrm + cnvfrm - pfrm``
    (`rck:40-56`) as a vector over all velocity dofs, or tested with ``phi``"""
    sm = _operators(V, outflowds, gradvsymmtrc, nu, device)

    def steady_state_res(vel, pres, phi=None):
        res = sm['A']@_flat(vel) + _conv(V, vel) - sm['JT']@_flat(pres)
        return _test(res, phi)

    return steady_state_res


def get_imex_res(V=None, outflowds=None, gradvsymmtrc=True, nu=None,
                 implscheme='crni', explscheme='abtw', device=False):
    """``imex_res(vel, pres, dt, lastvel, othervel, phi=None)`` for
    Crank-Nicolson + {AB2 'abtw', Heun 'heun', Euler 'eule'} (`rck:59-103`)"""
    if not implscheme == 'crni':
        raise NotImplementedError()
    sm = _operators(V, outflowds, gradvsymmtrc, nu, device)

    if explscheme == 'abtw':
        def convform(cvo, cvt):
            return 1.5*_conv(V, cvo) - .5*_conv(V, cvt)
    elif explscheme == 'heun':
        def convform(cvo, cvt):
            return .5*_conv(V, cvo) + .5*_conv(V, cvt)
    elif explscheme == 'eule':
        def convform(cvo, cvt):
            return _conv(V, cvo)
    else:
        raise NotImplementedError(explscheme)

    def imex_res(vel, pres, dt, lastvel=None, othervel=None, phi=None):
        vel, lastvel = _flat(vel), _flat(lastvel)
        res = sm['A']@(.5*(vel + lastvel)) + convform(lastvel, othervel) \
            - sm['JT']@_flat(pres) + 1./dt*(sm['M']@(vel - lastvel))
        return _test(res, phi)

    return imex_res


def get_imex_force_rows(V=None, invinds=None, dbcinds=None, dbcvals=None,
                        ldsbcinds=None, force_ops=None, outflowds=None,
                        gradvsymmtrc=True):
    """the drag/lift functional of `get_imex_res` (crni/abtw) as fixed rows

    Testing the residual with the indicator ``phi`` of the x (row 0) and y
    (row 1) components of the dofs ``ldsbcinds`` gives, for full velocities
    whose Dirichlet values ``u_bc`` are the same at every level,

        F = fm (v - vl)/dt + nu (fa (v + vl)/2 + fa_bc) - fj p
            + phi^T (3/2 c(vl) - 1/2 c(vo))

    with ``v``, ``vl`` the inner velocities (``invinds`` order) of the current
    and the last level: ``fm = phi^T M[:, inv]``, ``fa = phi^T A[:, inv]``
    (2 x NV), ``fj = phi^T JT`` (2 x NP), ``fa_bc = phi^T A[:, bc] u_bc`` (the
    mass part of the boundary values cancels).  ``force_ops``: the uncondensed
    nu = 1 operators ``dict(M=, A=, JT=)`` of `dts.get_stokessysmats`, built
    from ``V`` if omitted.  Only the convection depends on the state nonlinearly;
    it stays a vector.  Returns ``dict(fm, fa, fj, fa_bc, dofs, phi)``.
    """
    sm = force_ops if force_ops is not None else \
        _operators(V, outflowds, gradvsymmtrc, 1., False)
    M, A, JT = (sps.csr_matrix(sm[k]) for k in ('M', 'A', 'JT'))
    nvf = M.shape[0]
    dofs = np.unique(np.asarray(ldsbcinds, dtype=np.int64).reshape(-1))
    if dofs.size and (dofs[0] < 0 or dofs[-1] >= nvf):
        raise ValueError('force dofs out of range (full velocity numbering, '
                         '{0} dofs)'.format(nvf))
    phi = sps.csr_matrix((np.ones(dofs.size), (dofs % 2, dofs)),
                         shape=(2, nvf))
    aux = {}                    # Dirichlet data: last write wins (`dts:534-535`)
    for i, v in zip(dbcinds, dbcvals):
        aux[int(i)] = float(v)
    bci = np.array(sorted(aux.keys()), dtype=np.int64)
    ubc = np.array([aux[i] for i in bci], dtype=float)
    inv = np.asarray(invinds, dtype=np.int64)
    pM, pA = (phi@M).tocsc(), (phi@A).tocsc()
    return dict(fm=pM[:, inv].tocsr(), fa=pA[:, inv].tocsr(),
                fj=(phi@JT).tocsr(), fa_bc=pA[:, bci]@ubc, dofs=dofs,
                phi=phi)


def lift_drag_via_residual(steady_state_res, vel, pres, ldsbcinds, rho=1.,
                           L=0.1, Um=0.2):
    """``(Cd, Cl)`` by testing the residual with the indicator of the dofs in
    ``ldsbcinds`` (x components: drag, y: lift), scaled with
    ``2/(rho*L*Um**2)`` -- `tests/steadystate_schaefer-turek_2D-1.py:71-85`"""
    res = steady_state_res(vel, rho*_flat(pres))
    ld = np.asarray(ldsbcinds)
    fac = 2./(rho*L*Um**2)
    return fac*res[ld[ld % 2 == 0]].sum(), fac*res[ld[ld % 2 == 1]].sum()
