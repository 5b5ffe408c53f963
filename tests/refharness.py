"""Run the UNMODIFIED reference modules of a `dolfin_navier_scipy` checkout.

The checkout is not part of this repository: ``DNS_REFERENCE_ROOT`` names its
root directory (the one that holds the `dolfin_navier_scipy` package).

TEST INFRASTRUCTURE.  The reference is pure Python, but its modules import
three things that are not installable here: `dolfin` (FEniCS), the un-vendored
`sadptprj_riclyap_adi` and `krypy`.  What the hot path needs from them is tiny:

 * `dolfin`: ``Function(V).vector().set_local(ve)`` as a carrier of the
   coefficient vector (`snu:92-101`), ``File(..)`` handles that are never
   written to with ``paraviewoutput=False`` (`snu:1091-1092`) and the names
   ``dx, grad, div, inner`` at import time (`dts:6`);
 * `sadptprj_riclyap_adi.lin_alg_utils.solve_sadpnt_smw`: the exact sparse
   solve of the saddle-point system (contract fixed by the call sites, see
   `oracle/lau.py`);
 * `dolfin.assemble` of the convection forms inside `dts.get_convvec` /
   `dts.get_convmats` (`dts:325-376,427-472`) -- FFC-generated C++ that cannot
   be rebuilt.  These two functions (and only these) are served by the
   quadrature restatement `oracle/convection.py`.

Everything else -- `time_int_utils.cnab/sbdftwo/_onestepheun/
semi_implicit_euler`, `stokes_navier_utils.solve_nse/solve_steadystate_nse/
get_v_conv_conts/get_pfromv/m_innerproduct`, `dolfin_to_sparrays.
condense_velmatsbybcs/condense_sysmatsbybcs/append_bcs_vec/unroll_dlfn_dbcs`,
`data_output_utils.save_npa/load_npa` -- is the reference's own code, loaded
from the files where they lie and executed unchanged.  `load()` returns the
modules; `tests/golden/make_reference_golden.py` uses them to write the
reference-run fixtures, `tests/test_reference_pin.py` to compare the oracle
with the live reference whenever ``DNS_REFERENCE_ROOT`` is set.

Nothing here is imported by the product or by the `-m gpu` tests.
"""
import importlib
import importlib.util
import os
import sys
import types

import numpy as np

REFROOT = os.environ.get('DNS_REFERENCE_ROOT', '')
REFPKG = os.path.join(REFROOT, 'dolfin_navier_scipy')


def available():
    return bool(REFROOT) and \
        os.path.isfile(os.path.join(REFPKG, 'time_int_utils.py'))


class _Vector(object):
    def __init__(self, n):
        self.arr = np.zeros(n)

    def set_local(self, values):
        self.arr = np.array(values, dtype=float).reshape(-1)

    def get_local(self):
        return self.arr.copy()


class _Function(object):
    """carrier of a coefficient vector, the part of `dolfin.Function` that
    `snu.get_v_conv_conts` touches"""

    def __init__(self, V):
        self.V = V
        self._vector = _Vector(V.dim())

    def vector(self):
        return self._vector


class _File(object):
    def __init__(self, path):
        self.path = path

    def __lshift__(self, other):
        raise RuntimeError('the harness runs with paraviewoutput=False')


def _dolfin_stub():
    m = types.ModuleType('dolfin')
    m.Function = _Function
    m.File = _File
    for name in ('dx', 'grad', 'div', 'inner', 'nabla_grad', 'ds'):
        setattr(m, name, None)
    m.parameters = {}          # `dts:8` sets the linear algebra backend
    m.__stub__ = True
    return m


def _lau_stub():
    from oracle import lau as olau
    pkg = types.ModuleType('sadptprj_riclyap_adi')
    pkg.__path__ = []
    pkg.__stub__ = True
    m = types.ModuleType('sadptprj_riclyap_adi.lin_alg_utils')
    m.solve_sadpnt_smw = olau.solve_sadpnt_smw

    class SpslaKrylovCounter(object):
        def __init__(self, *a, **kw):
            pass
    m.SpslaKrylovCounter = SpslaKrylovCounter
    m.app_prj_via_sadpnt = None
    pkg.lin_alg_utils = m
    return pkg, m


_loaded = {}


def load():
    """-> dict(tiu=, snu=, dts=, dou=) of reference modules (cached)"""
    if _loaded:
        return _loaded
    if not available():
        raise FileNotFoundError(REFPKG)
    from oracle import convection as oconv

    # the reference was written for numpy < 1.24 (`snu:1560` uses `np.float`,
    # `snu:1413` `time.clock`): restore the removed aliases, as the numpy of
    # its own requirements would provide them
    for alias, typ in (('float', float), ('int', int)):
        if alias not in np.__dict__:
            setattr(np, alias, typ)
    import time
    if not hasattr(time, 'clock'):
        time.clock = time.perf_counter

    # the stubs stay installed: the reference imports `lau` inside its
    # functions (`snu:291,723,1614`); none of the names shadows a real module
    for k in ('dolfin', 'sadptprj_riclyap_adi', 'dolfin_navier_scipy'):
        if k in sys.modules and not getattr(sys.modules[k], '__stub__', 0):
            raise RuntimeError('a real `{0}` is importable: use it instead '
                               'of this harness'.format(k))
    sys.modules['dolfin'] = _dolfin_stub()
    pkg, lau = _lau_stub()
    sys.modules['sadptprj_riclyap_adi'] = pkg
    sys.modules['sadptprj_riclyap_adi.lin_alg_utils'] = lau
    # the package object without running its __init__ (which would pull
    # problem_setups and with it the whole of dolfin)
    refpkg = types.ModuleType('dolfin_navier_scipy')
    refpkg.__path__ = [REFPKG]
    refpkg.__stub__ = True
    sys.modules['dolfin_navier_scipy'] = refpkg
    dts = importlib.import_module('dolfin_navier_scipy.dolfin_to_sparrays')
    dou = importlib.import_module('dolfin_navier_scipy.data_output_utils')
    tiu = importlib.import_module('dolfin_navier_scipy.time_int_utils')
    snu = importlib.import_module('dolfin_navier_scipy.stokes_navier_utils')
    for mod in (dts, dou, tiu, snu):
        assert os.path.realpath(mod.__file__).startswith(
            os.path.realpath(REFPKG)), mod.__file__

    # the two FFC-assembled forms, served by the quadrature restatement
    def _coeffs(u0_dolfun, u0_vec, V, invinds, dbcinds, dbcvals):
        if u0_dolfun is not None:
            return u0_dolfun.vector().get_local()
        u0 = np.asarray(u0_vec, dtype=float).reshape(-1)
        if u0.size == V.dim():
            return u0
        return dts.append_bcs_vec(u0.reshape(-1, 1), vdim=V.dim(),
                                  invinds=invinds, bcinds=dbcinds,
                                  bcvals=dbcvals).reshape(-1)

    def get_convvec(u0_dolfun=None, V=None, u0_vec=None, femp=None,
                    uone_utwo_same=True, utwo_dolfun=None, utwo_vec=None,
                    dbcvals=None, dbcinds=None, diribcs=None, invinds=None):
        uone = _coeffs(u0_dolfun, u0_vec, V, invinds, dbcinds, dbcvals)
        if uone_utwo_same:
            cv = oconv.convvec(V, uone)
        else:
            utwo = _coeffs(utwo_dolfun, utwo_vec, V, invinds, dbcinds,
                           dbcvals)
            cv = oconv.convvec(V, uone, utwo)
        cv = cv[invinds] if invinds is not None else cv
        return cv.reshape(len(cv), 1)

    def get_convmats(u0_dolfun=None, u0_vec=None, V=None, invinds=None,
                     dbcvals=None, dbcinds=None, diribcs=None):
        u0 = _coeffs(u0_dolfun, u0_vec, V, invinds, dbcinds, dbcvals)
        N1, N2, fv = oconv.convmats(V, u0)
        import scipy.sparse as sps
        N1, N2 = sps.csr_matrix(N1), sps.csr_matrix(N2)
        N1.eliminate_zeros()
        N2.eliminate_zeros()
        return N1, N2, np.asarray(fv).reshape(-1, 1)

    dts.get_convvec = get_convvec
    dts.get_convmats = get_convmats
    _loaded.update(dict(tiu=tiu, snu=snu, dts=dts, dou=dou))
    return _loaded


def as_spmatrix(d):
    """the reference multiplies with ``*`` (`snu:1035`, `tiu:399`): hand it
    `scipy.sparse` *matrices*, never sparse arrays"""
    import scipy.sparse as sps
    out = dict(d)
    for k, v in d.items():
        if sps.issparse(v):
            out[k] = sps.csr_matrix(v)
    return out
