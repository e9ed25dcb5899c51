"""The sharded frame on partitions that reach every branch of its plan (dist.make_plan, hns_dist_set_plan's boundary / interior split)
and of its ghost-exchange protocol (hns_dist_ipc_finish's push CSR and flag slots, dist_frame's choice between the fused pressure
pipeline and pipelined_sweeps), bit for bit against the single-GPU frame.

The partitions and what each reaches are tests/helpers.py PARTITIONS; the CPU test below pins that reach, so the GPU runs keep
testing what their names say. The GPU runs share cuda:0 between the ranks when there are fewer GPUs than ranks (gloo process group,
peer-memory exchange through CUDA IPC), like tests/test_sharded_gpu.py. The GPU tests of this file take about 1 min 45 s on one
B200 with the ranks sharing it (twelve torchrun launches)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from helpers import PARTITION_DOMAINS, PARTITIONS, cube, partition_domain, partition_origins, partition_reach  # noqa: E402

from hnanosolver_b200 import dist as hdist  # noqa: E402

PAIRS = [(name, world) for name, (_, worlds) in PARTITIONS.items() for world in worlds]


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name, world", PAIRS, ids=[f"{n}@{w}" for n, w in PAIRS])
def test_partition_reaches_its_branches(name, world):
    o = partition_origins(name)
    assert partition_domain(o) == PARTITION_DOMAINS[name]
    want = PARTITIONS[name][1][world]
    if want is None:
        return   # the refusal, tested below
    plans = [hdist.make_plan(o, world, r) for r in range(world)]
    got = partition_reach(o, plans)
    assert got == want, f"{name} at {world} ranks no longer reaches what its row claims:\n got  {got}\n want {want}"


def test_make_plan_refuses_fewer_leaves_than_ranks_on_every_rank():
    o = partition_origins("too_few")
    for world in (3, 4):
        for rank in range(world):
            with pytest.raises(ValueError, match=rf"{o.shape[0]} leaves .* {world} ranks"):
                hdist.make_plan(o, world, rank)
    for rank in range(2):   # as many leaves as ranks: one each, leaf 0 a ghost of rank 1
        p = hdist.make_plan(o, 2, rank)
        assert p.n_owned == 1 and p.local_ids.tolist() == [0, 1]
    empty = hdist.make_plan(np.zeros((0, 3), np.int32), 3, 1)   # an empty domain: an empty plan on every rank
    assert empty.n_local == 0 and not empty.send and not empty.recv


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
DEFAULT = dict()                                          # two red-black frames
COLLISION = dict(collision=True, vorticity=[0.8, 7.9])    # |(int)factorScale| = 7: the vorticity stencil reaches the last ghost voxel
VORT_NEG = dict(vorticity=[0.8, -7.9])
COOK = dict(cook=True)
MG_THEN_RB = dict(multigrid=dict(red_black_frames=2))     # multigrid frames, then red-black: the flag numberings carry over
MG_ONE_LEVEL = dict(multigrid=dict(max_levels=1))         # sharded_mg_pressure's one-level branch
SOURCE = dict(source=True)
ELEMENT0 = dict(element0=0.625)                           # a wrong or stale ghost of global leaf 0 shows in advect_scalars
NO_SCALARS = dict(scalars=0, combustion=False)
ONE_SCALAR = dict(scalars=1, combustion=False)
SIXTEEN_FIELDS = dict(scalars=15, collision=True)
ALL_MODES = [DEFAULT, COLLISION, VORT_NEG, COOK, MG_THEN_RB, MG_ONE_LEVEL, SOURCE, ELEMENT0, NO_SCALARS, ONE_SCALAR, SIXTEEN_FIELDS]

# (partition, world) -> modes. Every mode runs on three_blobs at 3 ranks (boundary-free ranks beside a fused one) and on one block8
# world (no interior leaves on any rank).
GPU_RUNS = {
    ("three_blobs", 3): ALL_MODES,
    ("three_blobs", 2): [DEFAULT, ELEMENT0, MG_THEN_RB, COOK],
    ("three_blobs", 1): [DEFAULT, ELEMENT0, NO_SCALARS, MG_ONE_LEVEL],
    ("block8", 2): [DEFAULT, COLLISION, VORT_NEG, COOK],
    ("block8", 3): [DEFAULT, MG_THEN_RB, MG_ONE_LEVEL, SOURCE, ELEMENT0],
    ("block8", 4): [DEFAULT, NO_SCALARS, ONE_SCALAR, SIXTEEN_FIELDS],
    ("diagonal", 2): [DEFAULT, ELEMENT0, COOK, COLLISION],
    ("diagonal", 3): [DEFAULT, MG_THEN_RB, SIXTEEN_FIELDS],
    ("multitile_negative", 3): [DEFAULT, SOURCE, COLLISION, ELEMENT0],
    ("multitile_negative", 4): [DEFAULT, MG_THEN_RB, COOK, VORT_NEG],
    ("isolated_leaf0", 2): [DEFAULT, ELEMENT0, MG_ONE_LEVEL, ONE_SCALAR],
    ("isolated_leaf0", 4): [DEFAULT, ELEMENT0, SOURCE, COLLISION],
}
# the ncclSend / ncclRecv fallback, where there is one GPU per rank
NCCL_RUNS = {("three_blobs", 3), ("block8", 2)}


def test_gpu_runs_cover_every_mode_on_both_kinds_of_rank():
    blocks = [m for (name, _), modes in GPU_RUNS.items() if name == "block8" for m in modes]
    for m in ALL_MODES:
        assert m in GPU_RUNS[("three_blobs", 3)] and m in blocks, m
    assert {pair for pair in GPU_RUNS if pair[1] > 1} == {pair for pair in PAIRS if PARTITIONS[pair[0]][1][pair[1]] is not None}


@pytest.mark.gpu
@pytest.mark.parametrize("name, world", list(GPU_RUNS), ids=[f"{n}@{w}" for n, w in GPU_RUNS])
def test_sharded_frame_on_partition_is_bitwise_the_single_gpu_frame(name, world):
    from test_sharded_gpu import _gpus, _run

    origins = partition_origins(name).tolist()
    modes = [dict(m, origins=origins) for m in GPU_RUNS[(name, world)]]
    if (name, world) in NCCL_RUNS and _gpus() >= world:
        modes += [dict(DEFAULT, origins=origins, env=dict(HNS_P2P=0)), dict(COLLISION, origins=origins, env=dict(HNS_P2P=0))]
    share = world == 1 or _gpus() < world
    reports = _run(world, modes, share)
    for mode, rep in zip(modes, reports):
        assert rep["leaves"] == len(origins) and rep["world"] == world, rep
        assert rep["p2p"] == (world > 1 and "env" not in mode), rep
        assert rep["scalars"] == mode.get("scalars", 5), rep
        assert len(rep["fields"]) == 2 + rep["scalars"] + int(mode.get("collision", False)), rep
        mg = mode.get("multigrid")
        if mg is not None:
            if mg.get("max_levels") == 1:
                assert rep["mg_levels"] == 1 and rep["mg_gathers"] == 0, rep   # plain red-black sweeps on flag channels 8 / 9
            else:
                assert rep["mg_gathers"] == (rep["multigrid"]["cycles"] * rep["frames"] if rep["mg_levels"] > 1 else 0), rep
        if mode.get("source"):
            assert rep["sources"] == 4, rep


@pytest.mark.gpu
def test_vorticity_offset_beyond_one_ghost_leaf_is_refused():
    """dist_frame reads the advected velocity |(int)factorScale| voxels away: 7 still lies in the one-leaf ghost layer, 8 does not"""
    from hnanosolver_b200 import _lib
    from hnanosolver_b200 import launchers as H

    L = _lib.lib()
    go = cube((2, 2, 2))
    g = H.create_index_grid_from_origins(go, 0.5)
    sim = H.Simulation(g, 5)
    rng = np.random.default_rng(3)
    sim.upload(rng.random((sim.n, 3), np.float32) - np.float32(0.5), [rng.random(sim.n, np.float32) for _ in range(5)])
    owned = np.ascontiguousarray(np.arange(go.shape[0]), np.int32)
    h = C.c_void_p()
    _lib.check(L.hns_dist_create(None, 0, 1, C.byref(h)))
    try:
        _lib.check(L.hns_dist_set_plan(h, sim._h, 0, None, None, None, None, None, len(owned), owned.ctypes.data_as(_lib.c_i32p)))
        for factor, refused in ((7.9, False), (-7.9, False), (8.0, True), (-8.0, True)):
            sim.set_combustion(True, 1, 2, 3, 4, H.CombustionParams(0.5, 2.0, 1.5, 0.1, 0.8, factor))
            assert L.hns_state_vorticity_active(sim._h) == 1
            rc = L.hns_dist_frame(h, sim._h, 2, 0.1, None)
            sim.sync()
            if refused:
                assert rc == -5 and "one ghost leaf layer" in L.hns_last_error().decode(), (factor, rc)
            else:
                assert rc == 0, (factor, rc, L.hns_last_error().decode())
    finally:
        L.hns_dist_destroy(h)
    del sim
