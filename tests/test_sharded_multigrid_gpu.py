"""The sharded multigrid pressure solve (csrc/dist.cu, sharded_mg_pressure: level 0 sharded, levels >= 1 replicated, the level-1
right-hand side gathered into every rank through peer memory) must give the owned voxels of the single-GPU multigrid frame
(Simulation.set_pressure_solver) bit for bit: velocity, every scalar and pressure.

The ranks share cuda:0 on a one-GPU box (gloo process group, CUDA IPC between the processes), like tests/test_sharded_gpu.py."""
import ctypes as C
import json
import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hnanosolver_b200 import dist as hdist  # noqa: E402

# sharded_parity_check's default box
BOX, FILL, SEED = (256, 128, 128), 0.35, 7

MG_MODES = [
    dict(multigrid=dict(cycles=2, nu_pre=2, nu_post=2)),                 # V(2,2) x 2 over two frames
    dict(multigrid=dict(cycles=3, nu_pre=1, nu_post=0)),                 # no post-smoothing: the exchange after the prolongation feeds the
    dict(multigrid=dict(cycles=3, nu_pre=0, nu_post=1)),                 # next residual / gradient; no pre-smoothing: it feeds the red sweep
    dict(multigrid=dict(max_levels=2)),                                  # level 1 is the last level (smoothed, not solved in one CTA)
    dict(multigrid=dict(), env=dict(HNS_MG_GRAPH=0)),                     # coarse levels launched directly instead of a CUDA graph
    dict(multigrid=dict(), cook=True),                                   # host-buffer entry point (hns_dist_cook)
    dict(multigrid=dict(), collision=True, vorticity=[0.8, 2.0]),
    dict(multigrid=dict(), combustion=False, frames=3),
    dict(multigrid=dict(red_black_frames=2)),                            # then back to the red-black sharded frame
]


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(world: int, script: str, env: dict, timeout: int = 900):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), script]
    return subprocess.run(cmd, env=dict(os.environ, MASTER_ADDR="127.0.0.1", **env), cwd=ROOT, stdout=subprocess.PIPE,
                          stderr=subprocess.STDOUT, text=True, timeout=timeout)


def _gpus() -> int:
    import torch

    return torch.cuda.device_count()


def _pairs_without_shared_leaf(world: int):
    """rank pairs (a, b) of make_plan's partition of the test box in which neither holds a leaf of the other"""
    go = hdist.global_sparse_origins(BOX, FILL, SEED)
    plans = [hdist.make_plan(go, world, r) for r in range(world)]
    return [(a, b) for a in range(world) for b in range(a + 1, world)
            if b not in plans[a].send and b not in plans[a].recv and a not in plans[b].send and a not in plans[b].recv]


def test_a_world_has_ranks_that_share_no_ghost_leaf():
    # the gather reaches ranks that are not ghost-exchange peers, and its ordering flags are what keeps such a pair in step
    assert _pairs_without_shared_leaf(4), "no rank pair without a shared leaf at 4 ranks: the all-rank gather would go untested"


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_sharded_multigrid_frame_is_bitwise_the_single_gpu_multigrid_frame(world):
    share = world == 1 or _gpus() < world or bool(int(os.environ.get("HNS_TEST_FORCE_SHARE", "0")))
    r = _torchrun(world, os.path.join(ROOT, "tests", "sharded_worker.py"),
                  dict(HNS_TEST_MODES=json.dumps(MG_MODES), HNS_TEST_SHARE_GPU="1" if share else "0"))
    reports = [json.loads(l.split(" ", 1)[1]) for l in r.stdout.splitlines() if l.startswith("SHARDED_PARITY {")]
    assert r.returncode == 0 and "SHARDED_PARITY_SUMMARY OK" in r.stdout, r.stdout[-6000:]
    assert len(reports) == len(MG_MODES)
    for rep in reports:
        assert rep["ok"] and all("bitwise ok" in f for f in rep["fields"]), rep
        # the sharded path ran: one gather per V-cycle of every multigrid frame (not of the red-black frames after the switch back)
        assert rep["mg_gathers"] == rep["multigrid"]["cycles"] * rep["frames"], rep
        assert rep["mg_levels"] >= 2, rep
        assert (rep["mg_gather_bytes"] > 0) == (world > 1), rep
        assert rep["p2p"] == (world > 1), rep
    if world == 4:
        assert _pairs_without_shared_leaf(world)


def _state(origins, voxel_size=0.5, n_scalars=1):
    from hnanosolver_b200 import launchers as H

    g = H.create_index_grid_from_origins(origins, voxel_size)
    return g, H.Simulation(g, n_scalars)


@pytest.mark.gpu
def test_sharded_multigrid_refusals():
    from hnanosolver_b200 import _lib
    from hnanosolver_b200 import launchers as H

    L = _lib.lib()
    go = hdist.global_sparse_origins((64, 64, 64), 0.5, 3)
    plan = hdist.make_plan(go, 2, 0)
    local = np.ascontiguousarray(go[plan.local_ids])
    g, sim = _state(local)
    sim.upload(np.zeros((sim.n, 3), np.float32), [np.zeros(sim.n, np.float32)])
    G = H.create_index_grid_from_origins(go, 0.5)
    mg = H.Multigrid(G)
    assert mg.num_levels >= 2
    owned = np.ascontiguousarray(np.arange(local.shape[0]), np.int32)
    l2g = np.ascontiguousarray(plan.local_ids, np.int32)
    ip = lambda a: a.ctypes.data_as(_lib.c_i32p)  # noqa: E731
    handle = (C.c_uint8 * 64)()

    def plan_dist(world):
        h = C.c_void_p()
        _lib.check(L.hns_dist_create(None, 0, world, C.byref(h)))
        _lib.check(L.hns_dist_set_plan(h, sim._h, 0, None, None, None, None, None, len(owned), ip(owned)))
        return h

    def code(rc):
        return rc, L.hns_last_error().decode()

    d1 = plan_dist(1)
    try:
        def setp(m=mg, ids=l2g, cycles=2, nu_pre=2, nu_post=2, omega=1.15, state=sim):
            return code(L.hns_dist_set_pressure_solver(d1, state._h, m._h if m is not None else None, ip(ids), cycles, nu_pre, nu_post, omega, handle))

        for kw in (dict(cycles=0), dict(nu_pre=-1), dict(nu_post=-1), dict(nu_pre=0, nu_post=0), dict(omega=0.0), dict(omega=2.5)):
            assert setp(**kw)[0] == -1, kw
        bad = l2g.copy()
        bad[-1] = G.num_leaves
        rc, msg = setp(ids=bad)
        assert rc == -1 and "not a leaf of the hierarchy" in msg
        dup = l2g.copy()
        dup[1] = dup[0]
        assert setp(ids=dup)[0] == -1
        # a hierarchy whose level 0 has fewer leaves than the shard, and one over a grid of the right size in the wrong place
        small = H.create_index_grid_from_origins(go[: local.shape[0] - 1], 0.5)
        mg_small = H.Multigrid(small)
        rc, msg = setp(m=mg_small)
        assert rc == -1 and "not built over the global grid" in msg
        shifted = H.create_index_grid_from_origins(go + np.int32(8), 0.5)
        mg_shifted = H.Multigrid(shifted)
        rc, msg = setp(m=mg_shifted)
        assert rc == -1 and "built over another grid" in msg
        g2, other = _state(local)
        assert setp(state=other)[0] == -1
        # accepted, but a frame before hns_dist_mg_finish is refused; connecting to oneself is refused
        assert setp()[0] == 0
        rc, msg = code(L.hns_dist_frame(d1, sim._h, 4, 0.1, None))
        assert rc == -2 and "not connected" in msg
        assert L.hns_dist_mg_connect(d1, 0, handle) == -1
        assert L.hns_dist_mg_finish(d1) == 0
        assert setp(m=None)[0] == 0                       # back to red-black
    finally:
        L.hns_dist_destroy(d1)
    # more than one rank without the peer-memory exchange: nothing can carry the gather
    d2 = plan_dist(2)
    try:
        rc = L.hns_dist_set_pressure_solver(d2, sim._h, mg._h, ip(l2g), 2, 2, 2, 1.15, handle)
        assert rc == -5 and "peer memory" in L.hns_last_error().decode()
    finally:
        L.hns_dist_destroy(d2)
    del sim, other


_NCCL_WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, os.environ["HNS_ROOT"])
    import numpy as np, torch, torch.distributed as dist
    from hnanosolver_b200 import _lib, dist as hdist
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    _lib.lib().hns_set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    go = hdist.global_sparse_origins((64, 64, 64), 0.5, 3)
    plan = hdist.make_plan(go, world, rank)
    sh = hdist.ShardedSimulation(plan, np.ascontiguousarray(go[plan.local_ids]), 0.5, 1, torch.device("cuda", lr))
    try:
        sh.set_pressure_solver(go)
    except _lib.HnsError as e:
        ok = e.code == -5 and "peer memory" in e.message
    else:
        ok = False
    sh.close()
    dist.destroy_process_group()
    print("REFUSED" if ok else "NOT REFUSED", flush=True)
    sys.exit(0 if ok else 1)
""")


@pytest.mark.gpu
def test_sharded_multigrid_refused_on_the_nccl_fallback(tmp_path):
    if _gpus() < 2:
        pytest.skip("the ncclSend/ncclRecv fallback needs one GPU per rank")
    script = tmp_path / "nccl_refusal.py"
    script.write_text(_NCCL_WORKER)
    r = _torchrun(2, str(script), dict(HNS_P2P="0", HNS_ROOT=ROOT), timeout=300)
    assert r.returncode == 0 and r.stdout.count("REFUSED") == 2 and "NOT REFUSED" not in r.stdout, r.stdout[-4000:]
