"""Sharded-frame logic on CPU: world_size 2 (and 3) over gloo. Each rank owns a contiguous leaf range plus ghost leaves, runs the
frame's steps on its LOCAL leaves with the CPU oracle as the per-step kernel, and exchanges ghost bricks through the same
ShardPlan / HaloExchanger code the GPU path uses. The owned results, concatenated in rank order, must equal the single-domain
frame bit for bit."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from helpers import PARTITIONS, partition_origins  # noqa: E402

from hnanosolver_b200 import dist as hdist  # noqa: E402
from hnanosolver_b200 import synth  # noqa: E402

CATALOGUE = [(name, world) for name, (_, worlds) in PARTITIONS.items() for world, reach in worlds.items() if reach is not None]


def _check_plan(origins, world):
    plans = [hdist.make_plan(origins, world, r) for r in range(world)]
    L = origins.shape[0]
    owned = np.concatenate([p.local_ids[p.owned_local] for p in plans])
    assert np.array_equal(owned, np.arange(L))                                    # a partition, in order
    assert all(p.n_owned > 0 for p in plans)
    lut = {tuple(o): i for i, o in enumerate(origins.tolist())}
    for p in plans:
        mine = set(p.local_ids[p.owned_local].tolist())
        want = set()
        for l in mine:
            o = origins[l]
            for dx in (-8, 0, 8):
                for dy in (-8, 0, 8):
                    for dz in (-8, 0, 8):
                        m = lut.get((o[0] + dx, o[1] + dy, o[2] + dz))
                        if m is not None and m not in mine:
                            want.add(m)
        if p.rank > 0:
            want.add(0)                                                           # + global leaf 0 ("element 0" of advect_scalars)
            assert p.local_ids[0] == 0 and 0 in p.local_ids[p.recv[0]]
        assert set(p.local_ids[~p.owned_local].tolist()) == want                 # ghosts == 26-neighbours owned elsewhere
        assert np.all(np.diff(p.local_ids) > 0)                                   # local order == global NanoVDB order
        for q, ids in p.send.items():                                             # my send list == the peer's recv list
            assert np.array_equal(p.local_ids[ids], plans[q].local_ids[plans[q].recv[p.rank]])
        for q, ids in p.recv.items():                                             # and every recv list has its send list
            assert p.rank in plans[q].send and len(plans[q].send[p.rank]) == len(ids)
            assert not p.owned_local[ids].any()                                   # nothing owned is overwritten by a ghost


def test_plan_partitions_and_ghosts_are_consistent():
    _check_plan(synth.smoke_sphere(48, 3).origins, 3)


@pytest.mark.parametrize("name, world", CATALOGUE, ids=[f"{n}@{w}" for n, w in CATALOGUE])
def test_plan_partitions_and_ghosts_are_consistent_on_partitions(name, world):
    _check_plan(partition_origins(name), world)


def _frame_workload(case):
    """the sphere, or a partition of the catalogue with the sparse-smoke swirl on it and 0.625 in every scalar's element 0 (the
    "inactive" value of advect_scalars, which ranks other than 0 read from their ghost copy of global leaf 0)"""
    if case == "sphere":
        return synth.smoke_sphere(40, 5)
    o = partition_origins(case)
    vel, den, tem = synth._swirl_fields(64)
    w = synth._finish(case, o, vel, [den, tem], ["density", "temperature"], 40, 5)
    for a in w.scalars:
        a[0] = np.float32(0.625)
    return w


def _worker(rank, world, port, tmp, case):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import oracle as O

    w = _frame_workload(case)
    I, dt, h = 5, w.dt, w.voxel_size
    plan = hdist.make_plan(w.origins, world, rank)
    lo = np.repeat(plan.local_ids, 512) * 512 + np.tile(np.arange(512), plan.n_local)   # local voxel -> global voxel
    coords = w.coords[lo]
    ix = O.OracleIndex(coords)
    # local fields in the same "field id" space as the GPU path; pressure / divergence are kept in brick order here and the
    # colour halves are emulated by exchanging whole bricks (ids 6/7 -> p, 8/9 unused)
    F = {0: w.velocity[lo, 0].copy(), 1: w.velocity[lo, 1].copy(), 2: w.velocity[lo, 2].copy()}
    for i, s in enumerate(w.scalars):
        F[10 + i] = s[lo].copy()
    n = coords.shape[0]
    for k in (3, 4, 5, 6):
        F[k] = np.zeros(n, np.float32)

    def pack(field, ids, out):
        f = F[6 if field == 7 else field].reshape(-1, 512)
        fpl = hdist.floats_per_leaf(field)
        out.view(-1, fpl)[:] = torch.from_numpy(f[ids.numpy()][:, :fpl] if fpl == 512 else _half(f[ids.numpy()], field))

    def unpack(field, ids, src):
        f = F[6 if field == 7 else field].reshape(-1, 512)
        fpl = hdist.floats_per_leaf(field)
        if fpl == 512:
            f[ids.numpy()] = src.view(-1, 512).numpy()
        else:
            _set_half(f, ids.numpy(), field, src.view(-1, 256).numpy())

    par = (np.add.outer(np.add.outer(np.arange(8), np.arange(8)), np.arange(8)) & 1).reshape(512).astype(bool)  # True = black

    def _half(bricks, field):
        return bricks[:, par] if field == 7 else bricks[:, ~par]

    def _set_half(f, ids, field, vals):
        sel = par if field == 7 else ~par
        tmpb = f[ids]
        tmpb[:, sel] = vals
        f[ids] = tmpb

    ex = hdist.HaloExchanger(plan, torch.device("cpu"), pack, unpack, max_fields=3 + len(w.scalars))
    vel = lambda: np.stack([F[0], F[1], F[2]], 1)
    ex.exchange(hdist.F_VEL)
    adv = ix.advect_vector(vel(), dt, h)
    F[3], F[4], F[5] = adv[:, 0].copy(), adv[:, 1].copy(), adv[:, 2].copy()
    ex.exchange(hdist.F_ADV)
    adv = np.stack([F[3], F[4], F[5]], 1)
    div = ix.divergence(adv, h)
    F[6][:] = 0
    omega = O.omega_compute(h)
    for _ in range(I):
        ix.rbgs_color(div, F[6], h, 0, omega)
        ex.exchange([hdist.F_P_RED])
        ix.rbgs_color(div, F[6], h, 1, omega)
        ex.exchange([hdist.F_P_BLK])
    v = ix.subtract_gradient(adv, F[6], h)
    F[0], F[1], F[2] = v[:, 0].copy(), v[:, 1].copy(), v[:, 2].copy()
    ex.exchange(list(hdist.F_VEL) + [10 + i for i in range(len(w.scalars))])
    outs = ix.advect_scalars(vel(), [F[10 + i] for i in range(len(w.scalars))], dt, h)
    m = np.repeat(plan.owned_local, 512)
    np.savez(os.path.join(tmp, f"rank{rank}.npz"), vel=vel()[m], p=F[6][m], s=np.stack(outs)[:, m], exchanges=ex.exchanges)
    dist.barrier()
    dist.destroy_process_group()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# the sphere; three_blobs at 3 ranks (ranks 1 and 2 exchange nothing but their ghost of leaf 0); block8 at 4 ranks (no interior leaf)
@pytest.mark.parametrize("case, world", [pytest.param("sphere", 2, id="2"), pytest.param("sphere", 3, id="3"),
                                         pytest.param("three_blobs", 3, id="three_blobs@3"), pytest.param("block8", 4, id="block8@4")])
def test_sharded_frame_equals_single_domain_frame(tmp_path, case, world):
    from oracle import oracle as O

    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    mp.spawn(_worker, args=(world, port, str(tmp_path), case), nprocs=world, join=True)
    w = _frame_workload(case)
    want = O.OracleIndex(w.coords).frame(w.velocity, w.scalars, 5, w.dt, w.voxel_size)
    parts = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    assert np.array_equal(_bits(np.concatenate([p["vel"] for p in parts])), _bits(want["vel"]))
    assert np.array_equal(_bits(np.concatenate([p["p"] for p in parts])), _bits(want["p"]))
    for i in range(len(w.scalars)):
        assert np.array_equal(_bits(np.concatenate([p["s"][i] for p in parts])), _bits(want["scalars"][i])), f"scalar {i}"
    assert int(parts[0]["exchanges"]) == 3 + 2 * 5                                # vel, adv, 2 per iteration, vel+scalars
