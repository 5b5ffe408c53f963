"""Host side of the output functionals of the device time loop: the sparse rows
the drag/lift functional reduces to (`residual_checks.get_imex_force_rows`)
against the residual they are cut from (`get_imex_res`), and the all-gather of
the recorded outputs over uneven member shards (gloo, world size 2)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dolfin_navier_scipy_b200 import ensemble as ens
from dolfin_navier_scipy_b200 import problem_setups as dnsps
from dolfin_navier_scipy_b200 import residual_checks as rck
from oracle import convection as oconv


def _cyl1(bccontrol):
    return dnsps.get_sysmats(problem='cylinderwake', nu=1., scheme='TH',
                             bccontrol=bccontrol,
                             meshparams=dict(refinement_level=1))


@pytest.mark.parametrize('bccontrol', [False, True])
def test_force_rows_reproduce_the_cnab_residual(bccontrol, monkeypatch):
    """``fm (v - vl)/dt + nu (fa (v + vl)/2 + fa_bc) - fj p + phi^T (3/2 c(vl)
    - 1/2 c(vo))`` equals ``get_imex_res(nu)(v, p, dt, vl, vo, phi)`` for the
    x and y indicator of ``ldsbcinds`` on random states with the same
    Dirichlet values (the convection from the oracle's independent rule)"""
    monkeypatch.setattr(rck, '_conv',
                        lambda V, vel: oconv.convvec(V, rck._flat(vel)))
    femp, sm, rhs_vf, rhs_bc = _cyl1(bccontrol)
    V, inv = femp['V'], np.asarray(femp['invinds'])
    ops = dict(M=sm['Mfull'], A=sm['Afull'], JT=sm['JTfull'])
    rows = rck.get_imex_force_rows(
        V=V, invinds=inv, dbcinds=femp['dbcinds'], dbcvals=femp['dbcvals'],
        ldsbcinds=femp['ldsbcinds'], force_ops=ops if bccontrol else None)
    nvf, NP = V.dim(), sm['J'].shape[0]
    rng = np.random.default_rng(3 + bccontrol)
    aux = dict(zip(map(int, femp['dbcinds']), femp['dbcvals']))
    bci = np.array(sorted(aux))
    vel, lastvel, othervel = rng.standard_normal((3, nvf))
    for v in (vel, lastvel):
        v[bci] = [aux[i] for i in bci]
    pres = rng.standard_normal(NP)
    nu, dt = 0.1/75., 1./2048
    res = rck.get_imex_res(V=V, nu=nu, implscheme='crni', explscheme='abtw')
    cl, co = oconv.convvec(V, lastvel), oconv.convvec(V, othervel)
    F = rows['fm']@(vel - lastvel)[inv]/dt \
        + nu*(rows['fa']@(.5*(vel + lastvel))[inv] + rows['fa_bc']) \
        - rows['fj']@pres + rows['phi']@(1.5*cl - .5*co)
    ld = np.asarray(femp['ldsbcinds'])
    assert np.array_equal(rows['dofs'], np.unique(ld))
    for c in range(2):
        phi = np.zeros(nvf)
        phi[ld[ld % 2 == c]] = 1.
        ref = res(vel, pres, dt, lastvel, othervel, phi)
        assert abs(F[c] - ref) <= 1e-13*abs(ref), (c, F[c], ref)


@pytest.mark.parametrize('bccontrol', [False, True])
def test_condensed_stiffness_is_the_inner_block_of_the_full_one(bccontrol):
    """the loop operator A0 (`get_sysmats(nu=1)`) is ``A_full[inv][:, inv]``:
    the rows ``phi^T A_full[:, inv]`` act on the velocity the loop advances"""
    femp, sm, _, _ = _cyl1(bccontrol)
    inv = np.asarray(femp['invinds'])
    for key in ('A', 'M'):
        d = sm[key] - sm[key + 'full'][inv][:, inv]
        assert abs(d).max() == 0., key


def test_force_rows_refuse_out_of_range_dofs():
    femp, sm, _, _ = _cyl1(False)
    ops = dict(M=sm['Mfull'], A=sm['Afull'], JT=sm['JTfull'])
    with pytest.raises(ValueError):
        rck.get_imex_force_rows(invinds=femp['invinds'],
                                dbcinds=femp['dbcinds'],
                                dbcvals=femp['dbcvals'],
                                ldsbcinds=[0, femp['V'].dim()], force_ops=ops)


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _records(nmembers, levels=6, ny=3):
    rng = np.random.default_rng(11)
    return (rng.standard_normal((levels, ny, nmembers)),
            rng.standard_normal((levels, 2, nmembers)))


class _Shard(object):
    """stands in for a `DeviceImex` with its shard's recorded outputs"""

    def __init__(self, y, force):
        self.y, self.force = y, force

    def outputs(self):
        return dict(y=self.y, force=self.force)


def _worker(rank, world, port, nmembers, out):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    Y, F = _records(nmembers)
    lo, hi = ens.shard_members(nmembers, rank, world)
    got = ens.gather_outputs(_Shard(Y[:, :, lo:hi], F[:, :, lo:hi]))
    out[rank] = (got['y'].copy(), got['force'].copy())
    dist.barrier()
    dist.destroy_process_group()


def test_gather_outputs_two_ranks_uneven_shards_gloo():
    world, nmembers = 2, 5
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, nmembers, out), nprocs=world,
             join=True)
    Y, F = _records(nmembers)
    for r in range(world):
        y, f = out[r]
        assert np.array_equal(y, Y) and np.array_equal(f, F)


def test_gather_outputs_single_process_is_the_shard():
    Y, F = _records(4)
    got = ens.gather_outputs(_Shard(Y, F))
    assert got['y'] is Y and got['force'] is F
    assert not torch.distributed.is_initialized()
