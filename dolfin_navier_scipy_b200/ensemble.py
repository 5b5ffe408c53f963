"""Batched ensembles of trajectories that share one mesh and sparsity pattern.

BASELINE config 5: Reynolds-number / boundary-control sweeps of the cylinder
wake with penalised Robin control (`tests/time_dep_nse_bcrob.py:26-34`):
``A_m = nu_m*A0 + Arob/palpha``, ``f_m(t) = nu_m*fv_bc + u(t)*(B_1 - B_2)/palpha``.
Members are independent: they are sharded over the GPUs with *no* collective
on the step path; the only exchange is the all-reduce of the POD snapshot Gram
matrix ``G = sum_m X_m^T M X_m`` (additive over members, SURVEY.md 8e),
and the one-off all-gathers of the recorded output functionals
(`gather_outputs`), of the members' trip levels (`gather_member_status`) and
of their field statistics (`gather_statistics`).
"""
import numpy as np

from . import problem_setups as dnsps
from . import time_int_utils as tiu

__all__ = ['cylinder_ensemble', 'shard_members', 'bind_to_gpu_cpus',
           'gram_allreduce', 'gather_outputs', 'gather_member_status',
           'gather_statistics',
           'allreduce_gram', 'pod_from_gram', 'pod_modes']


def bind_to_gpu_cpus(device=0):
    """pin the calling process to the CPU cores closest to ``device`` (NVML's
    affinity mask) and return them, or ``None`` if that is not possible

    One process per GPU streams every step's state into its own pinned host
    mirror (16.8 MB per step for 64 members on `cylinder_4`).  Pinned memory
    is placed on the NUMA node of the allocating thread, so a rank that floats
    across sockets sends its snapshots over the inter-socket link; with eight
    ranks on one box that link, not PCIe, bounds the end-to-end rate.  Call
    before the context (and with it the pinned buffers) is created."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(device))
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63)//64)
        cpus = [64*w + b for w, word in enumerate(words) for b in range(64)
                if (int(word) >> b) & 1 and 64*w + b < ncpu]
        allowed = set(os.sched_getaffinity(0))
        cpus = sorted(set(cpus) & allowed)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:                                     # noqa: BLE001
        return None


def shard_members(nmembers, rank, world):
    """contiguous slice of the members owned by ``rank``"""
    per = nmembers // world
    rem = nmembers % world
    lo = rank*per + min(rank, rem)
    return lo, lo + per + (1 if rank < rem else 0)


def cylinder_ensemble(N=4, Res=(60., 150.), nmembers=64, rank=0, world=1,
                      dt=1./512, scheme='cnab', palpha=1e-5, bccontrol=True,
                      control=np.sin, ntimes=513, t0=0., ctx=None, mesh=None,
                      cheb_steps=4, restart=40, schur_poly=2, coarse_max=4096,
                      force=False, cv_mat=None, cp_mat=None,
                      member_guard=False, statistics=False):
    """device integrator for this rank's shard of a Re-sweep ensemble

    Returns ``(integ, info)``; ``integ`` is a `time_int_utils.DeviceImex` with
    forcing and members set, ``info`` holds sizes and the host operators.
    ``force=True`` records the raw drag/lift on the whole cylinder
    (``ldsbcinds``, control patches included) and ``cv_mat`` / ``cp_mat`` the
    linear outputs at every time level (`DeviceImex.set_outputs`); the drag
    coefficient is ``2/(rho L Um^2)`` times the x force
    (`residual_checks.lift_drag_via_residual`).  ``member_guard=True``
    retires a member that trips the blow-up guard and integrates the others
    on (`DeviceImex.set_member_guard`).  ``statistics=True`` accumulates
    the mean flow, the velocity and pressure fluctuation intensities and the
    mean convection of every member inside the loop
    (`DeviceImex.set_statistics`).
    """
    Re_all = np.linspace(Res[0], Res[1], nmembers)
    lo, hi = shard_members(nmembers, rank, world)
    Re = Re_all[lo:hi]
    meshparams = dict(refinement_level=N)
    if mesh is not None:
        meshparams['mesh'] = mesh
    # operators for nu = 1: A = nu*A0, boundary rhs = nu*fv_bc
    femp, sm, rhs_vf, rhs_bc = dnsps.get_sysmats(
        problem='cylinderwake', nu=1., bccontrol=bccontrol, scheme='TH',
        meshparams=meshparams)
    charlen = femp['charlen']
    nus = charlen/Re                                   # `dnsps:138-141`
    NP, NV = sm['J'].shape
    Arob = sm['Arob']/palpha if bccontrol else None
    integ = tiu.DeviceImex(sm['M'], sm['A'], sm['J'], femp['V'],
                           femp['invinds'], femp['dbcinds'], femp['dbcvals'],
                           dt, scheme=scheme, nus=nus, Arob=Arob,
                           fp=rhs_bc['fp'] + rhs_vf['fp'], ctx=ctx,
                           cheb_steps=cheb_steps, restart=restart,
                           schur_poly=schur_poly, coarse_max=coarse_max)
    trange = t0 + dt*np.arange(ntimes)
    cols = [rhs_bc['fv'].reshape(NV, 1)]
    if bccontrol:
        Brob = sm['Brob']/palpha
        cols.append(Brob[:, :1] - Brob[:, 1:])
    B = np.hstack(cols)
    U = np.zeros((ntimes, B.shape[1], nus.size))
    U[:, 0, :] = nus[None, :]
    if bccontrol:
        U[:, 1, :] = control(trange)[:, None]
    integ.set_forcing(B, U)
    if member_guard:
        integ.set_member_guard(True)
    if statistics:
        integ.set_statistics(True)
    if force or cv_mat is not None or cp_mat is not None:
        integ.set_outputs(cv_mat, cp_mat,
                          force_dofs=femp['ldsbcinds'] if force else None,
                          force_ops=dict(M=sm['Mfull'], A=sm['Afull'],
                                         JT=sm['JTfull']))
    info = dict(femp=femp, sm=sm, nus=nus, Re=Re, NV=NV, NP=NP, B=B, U=U,
                Arob=Arob, fp=rhs_bc['fp'] + rhs_vf['fp'], trange=trange,
                members=(lo, hi))
    return integ, info


def allreduce_gram(G, group=None):
    """sum the per-rank partial Gram matrices in place (NCCL on the device,
    gloo on the host); a no-op for a single process"""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() \
            and dist.get_world_size(group) > 1:
        dist.all_reduce(G, op=dist.ReduceOp.SUM, group=group)
    return G


def gram_allreduce(integ, group=None):
    """POD snapshot Gram matrix of the whole ensemble

    Each rank computes ``sum_{m in shard} X_m^T M X_m`` on its device
    (``dnsb_imex_gram_dev``); one ``all_reduce(SUM)`` over NCCL finishes it.
    Returns a (ns, ns) torch tensor on the device (identical on all ranks).
    """
    import torch
    ns = integ.engine.ctx.lib.dnsb_imex_num_snapshots(integ.engine.h)
    dev = torch.device('cuda', integ.ctx.device)
    G = torch.zeros((ns, ns), dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)
    integ.engine.gram_dev(G.data_ptr())
    return allreduce_gram(G, group)


def gather_outputs(integ, group=None):
    """output functionals of the whole ensemble on every rank

    ``integ.outputs()`` of each rank's shard (`DeviceImex.outputs`), put
    together along the member axis in rank order -- the contiguous, possibly
    uneven shards of `shard_members` -- by one ``all_gather`` (NCCL on the
    device, gloo on the host).  Returns ``dict(y=(levels, ny, nmembers),
    force=(levels, 2, nmembers))`` as numpy arrays; every rank must have
    recorded the same levels.
    """
    out = integ.outputs()
    return {key: _gather_members(np.asarray(out[key], dtype=float), group)
            for key in ('y', 'force')}


def _gather_members(a, group):
    """all-gather ``a`` (..., nb) of every rank's shard along the last axis
    in rank order (the contiguous, possibly uneven shards of
    `shard_members`); ``a`` itself for a single process"""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) \
            or dist.get_world_size(group) == 1:
        return a
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    dev = torch.device('cuda', torch.cuda.current_device()) \
        if dist.get_backend(group) == 'nccl' else torch.device('cpu')
    nb = a.shape[-1]
    cnt = torch.tensor([nb], dtype=torch.int64, device=dev)
    dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)
    nmembers = int(cnt.item())
    sizes = [hi - lo for lo, hi in (shard_members(nmembers, r, world)
                                    for r in range(world))]
    if sizes[rank] != nb:
        raise ValueError('rank {0} holds {1} members, shard_members gives it '
                         '{2}'.format(rank, nb, sizes[rank]))
    pad = np.zeros(a.shape[:-1] + (max(sizes),), dtype=a.dtype)
    pad[..., :nb] = a
    t = torch.from_numpy(pad).to(dev)
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t, group=group)
    return np.concatenate([p.cpu().numpy()[..., :sizes[r]]
                           for r, p in enumerate(parts)], axis=-1)


def gather_member_status(integ, group=None):
    """trip levels of the whole ensemble on every rank, in member order

    ``integ.member_status()['trip_level']`` of each rank's shard
    (`DeviceImex.member_status`; -1 = live), put together by one
    ``all_gather`` like `gather_outputs`.  Returns ``dict(trip_level=
    (nmembers,) int, alive=(nmembers,) bool)``.
    """
    t = np.asarray(integ.member_status()['trip_level'], dtype=np.int64)
    t = _gather_members(t, group)
    return dict(trip_level=t, alive=t < 0)


def gather_statistics(integ, group=None):
    """field statistics of the whole ensemble on every rank, in member order

    ``integ.statistics()`` of each rank's shard (`DeviceImex.statistics`),
    every per-member array put together along the member axis by one
    ``all_gather`` like `gather_outputs`; ``first_level`` and ``last_level``
    are this rank's (every rank must have run the same levels).
    """
    s = integ.statistics()
    out = dict(first_level=s['first_level'], last_level=s['last_level'])
    out['count'] = _gather_members(np.asarray(s['count'], dtype=np.int64),
                                   group)
    for key in ('v_mean', 'uu', 'vv', 'uv', 'p_mean', 'p_var', 'c_mean'):
        out[key] = _gather_members(np.asarray(s[key], dtype=float), group)
    return out


def pod_from_gram(G, energy=0.9999, kmax=None):
    """method of snapshots on the (all-reduced) Gram matrix
    ``G = sum_m X_m^T M X_m``: eigenvalues (descending), the temporal modes
    ``W`` (ns x r, scaled so that the spatial modes ``Phi_m = X_m W`` satisfy
    ``sum_m Phi_m^T M Phi_m = I``) and the rank ``r`` that captures ``energy``
    of the trace.  ``G`` is tiny (ns x ns): plain host ``eigh``."""
    G = np.asarray(G.cpu() if hasattr(G, 'cpu') else G, dtype=float)
    lam, Q = np.linalg.eigh(.5*(G + G.T))
    lam, Q = lam[::-1], Q[:, ::-1]
    lam = np.maximum(lam, 0.)
    frac = np.cumsum(lam)/max(lam.sum(), 1e-300)
    r = int(np.searchsorted(frac, energy) + 1)
    r = min(r, int(np.sum(lam > 1e-14*lam[0])))
    if kmax is not None:
        r = min(r, kmax)
    W = Q[:, :r]/np.sqrt(lam[:r])[None, :]
    return lam, W, r


def pod_modes(snapshots, W):
    """spatial POD modes of every member: ``snapshots`` (ns, NV, nb) as
    returned by `DeviceImex.snapshots()[0]`, ``W`` from `pod_from_gram` ->
    (NV, r, nb).  The reduced coordinates of member ``m`` at snapshot ``s``
    are ``(W^T G)[:, s]`` -- shared by all members by construction."""
    return np.einsum('snm,sr->nrm', np.asarray(snapshots), W)
