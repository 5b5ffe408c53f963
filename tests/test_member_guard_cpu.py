"""`ensemble.gather_member_status`: the trip levels of the per-member blow-up
guard put together over uneven member shards (gloo, world size 2) and in a
single process."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dolfin_navier_scipy_b200 import ensemble as ens


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _levels(nmembers):
    """live members (-1) and members retired at assorted levels"""
    t = np.full(nmembers, -1, dtype=np.int32)
    t[1::3] = 11 + 10*np.arange(t[1::3].size)
    return t


class _Shard(object):
    """stands in for a `DeviceImex` with its shard's member status"""

    def __init__(self, trip):
        self.trip = trip

    def member_status(self):
        return dict(trip_level=self.trip, alive=self.trip < 0)


def _worker(rank, world, port, nmembers, out):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    lo, hi = ens.shard_members(nmembers, rank, world)
    got = ens.gather_member_status(_Shard(_levels(nmembers)[lo:hi]))
    out[rank] = (got['trip_level'].copy(), got['alive'].copy())
    dist.barrier()
    dist.destroy_process_group()


def test_gather_member_status_two_ranks_uneven_shards_gloo():
    world, nmembers = 2, 5
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, nmembers, out), nprocs=world,
             join=True)
    T = _levels(nmembers)
    for r in range(world):
        t, alive = out[r]
        assert np.array_equal(t, T)
        assert np.array_equal(alive, T < 0)


def test_gather_member_status_single_process_is_the_shard():
    T = _levels(7)
    got = ens.gather_member_status(_Shard(T))
    assert np.array_equal(got['trip_level'], T)
    assert np.array_equal(got['alive'], T < 0)
    assert not torch.distributed.is_initialized()
