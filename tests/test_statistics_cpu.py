"""In-loop field statistics without a device: `ensemble.gather_statistics`
over uneven member shards (gloo, world size 2), the numbering bookkeeping of
`DeviceImex.statistics` / `mean_flow_forcing` on a stand-in engine, and a
numpy restatement of the kernel's elementwise Welford update against
``np.mean`` / ``np.cov``."""
import os
import socket

import numpy as np
import torch.distributed as dist
import torch.multiprocessing as mp

from dolfin_navier_scipy_b200 import ensemble as ens
from dolfin_navier_scipy_b200 import time_int_utils as tiu

KEYS = ('v_mean', 'uu', 'vv', 'uv', 'p_mean', 'p_var', 'c_mean')


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _stats(nmembers, nnodes=5, NV=7, NP=3):
    """statistics of a whole ensemble, member m's entries tagged with m"""
    rng = np.random.default_rng(3)
    s = dict(first_level=4, last_level=19,
             count=np.arange(nmembers, dtype=np.int64) + 1)
    shapes = dict(v_mean=2*nnodes, uu=nnodes, vv=nnodes, uv=nnodes,
                  p_mean=NP, p_var=NP, c_mean=NV)
    for k, n in shapes.items():
        s[k] = rng.standard_normal((n, nmembers)) + np.arange(nmembers)
    return s


class _Shard(object):
    def __init__(self, s, lo, hi):
        self.s = {k: (v[..., lo:hi] if isinstance(v, np.ndarray) else v)
                  for k, v in s.items()}

    def statistics(self):
        return self.s


def _worker(rank, world, port, nmembers, out):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    lo, hi = ens.shard_members(nmembers, rank, world)
    got = ens.gather_statistics(_Shard(_stats(nmembers), lo, hi))
    out[rank] = {k: (v.copy() if isinstance(v, np.ndarray) else v)
                 for k, v in got.items()}
    dist.barrier()
    dist.destroy_process_group()


def test_gather_statistics_two_ranks_uneven_shards_gloo():
    world, nmembers = 2, 5
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, nmembers, out), nprocs=world,
             join=True)
    ref = _stats(nmembers)
    for r in range(world):
        got = out[r]
        assert got['first_level'] == 4 and got['last_level'] == 19
        assert got['count'].dtype == np.int64
        assert np.array_equal(got['count'], ref['count'])
        for k in KEYS:
            assert np.array_equal(got[k], ref[k]), k


def test_gather_statistics_single_process_is_the_shard():
    ref = _stats(3)
    got = ens.gather_statistics(_Shard(ref, 0, 3))
    for k in KEYS + ('count',):
        assert np.array_equal(got[k], ref[k])


class _Engine(object):
    """returns fixed statistics in the device numbering"""

    def __init__(self, dev):
        self.dev = dev

    def statistics(self, nnodes):
        assert nnodes == self.dev['v_mean'].shape[0]//2
        return self.dev


class _Conv(object):
    nvf = 12

    def convvec(self, u):
        return 3.*u + 1.


def test_statistics_un_permutes_p_and_c_and_the_forcing():
    """device row i of p / c is the caller's row pp[i] / pv[i] (as in
    `DeviceImex.state`); v_mean and the node moments are already in the
    caller's full numbering; the forcing is c_mean - c(v_mean)[invinds]"""
    rng = np.random.default_rng(5)
    nb, nnodes, NV, NP = 3, 6, 8, 4
    truth = dict(v_mean=rng.standard_normal((2*nnodes, nb)),
                 uvcov=rng.standard_normal((3, nnodes, nb)),
                 p_mean=rng.standard_normal((NP, nb)),
                 p_var=rng.standard_normal((NP, nb)),
                 c_mean=rng.standard_normal((NV, nb)))
    integ = object.__new__(tiu.DeviceImex)
    integ.pv, integ.pp = rng.permutation(NV), rng.permutation(NP)
    integ.ipv, integ.ipp = np.argsort(integ.pv), np.argsort(integ.pp)
    integ.invinds = np.array([0, 2, 3, 5, 6, 8, 9, 11], dtype=np.int32)
    integ.dev = _Conv()
    dev = dict(truth, p_mean=truth['p_mean'][integ.pp],
               p_var=truth['p_var'][integ.pp],
               c_mean=truth['c_mean'][integ.pv], first=2, last=9,
               count=np.array([8, 8, 0]))
    integ.engine = _Engine(dev)
    st = integ.statistics()
    assert st['first_level'] == 2 and st['last_level'] == 9
    assert np.array_equal(st['count'], [8, 8, 0])
    assert np.array_equal(st['v_mean'], truth['v_mean'])
    for i, k in enumerate(('uu', 'vv', 'uv')):
        assert np.array_equal(st[k], truth['uvcov'][i])
    for k in ('p_mean', 'p_var', 'c_mean'):
        assert np.array_equal(st[k], truth[k]), k
    fm = integ.mean_flow_forcing(st)
    want = truth['c_mean'] - (3.*truth['v_mean'] + 1.)[integ.invinds]
    assert np.array_equal(fm, want)
    assert np.array_equal(integ.mean_flow_forcing(), want)


def _welford(X, trip=None, first=0):
    """numpy restatement of k_imex_stats: X (levels, n, 2, nb) pairs (u, v)
    of consecutive levels first, first+1, ...; member m skips the levels
    after trip[m] >= 0.  Returns means (n, 2, nb) and co-moments (3, n, nb)."""
    L, n, _, nb = X.shape
    trip = np.full(nb, -1) if trip is None else np.asarray(trip)
    mean = np.full((n, 2, nb), np.nan)
    C = np.full((3, n, nb), np.nan)
    for j in range(L):
        level, k = first + j, j + 1
        live = (trip < 0) | (trip >= level)
        x = X[j]
        if k == 1:
            mean[:, :, live] = x[:, :, live]
            C[:, :, live] = 0.
            continue
        d = x - mean
        mnew = mean + d*(1./k)
        e = x - mnew
        Cn = C + np.stack([d[:, 0]*e[:, 0], d[:, 1]*e[:, 1], d[:, 0]*e[:, 1]])
        mean[:, :, live] = mnew[:, :, live]
        C[:, :, live] = Cn[:, :, live]
    return mean, C


def test_welford_restatement_against_numpy():
    """the elementwise update with count 1/k gives np.mean and the
    population np.cov of every node and member, over all levels and, for a
    retired member, over the levels up to its trip"""
    rng = np.random.default_rng(11)
    L, n, nb, first = 57, 9, 4, 3
    X = 2. + rng.standard_normal((L, n, 2, nb))*np.array([1., 1e-3])[None, None, :, None]
    trip = np.array([-1, first + 20, -1, first + L + 5])
    mean, C = _welford(X, trip, first)
    for m in range(nb):
        last = L if trip[m] < 0 else min(L, trip[m] - first + 1)
        Y = X[:last, :, :, m]
        assert np.allclose(mean[:, :, m], Y.mean(0), rtol=0, atol=1e-14)
        for i in range(n):
            cov = np.cov(Y[:, i, 0], Y[:, i, 1], bias=True)
            got = C[:, i, m]/last
            ref = np.array([cov[0, 0], cov[1, 1], cov[0, 1]])
            scale = np.array([cov[0, 0], cov[1, 1],
                              np.sqrt(cov[0, 0]*cov[1, 1])])
            assert np.all(np.abs(got - ref) <= 1e-12*scale), (m, i)
