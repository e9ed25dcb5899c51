"""The sharded frame (csrc/dist.cu: ghost exchange by peer-memory stores + flags, boundary/interior pipeline, velocity-ghost reuse,
background scalar exchange) must equal the single-GPU frame bit for bit on the owned voxels of every rank -- which in turn is the
reference's Compute() order (reference src/Cuda/HNanoSolver.cu:159-356; single-GPU parity: tests/test_gpu_parity.py).

With two or more GPUs the ranks get a GPU each and both data paths run (peer memory and the ncclSend/ncclRecv fallback). On a
single-GPU box the ranks share cuda:0: NCCL refuses that, CUDA IPC does not, so the peer-memory protocol is still exercised."""
import json
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

P2P_MODES = [
    dict(),                                                       # fused boundary sweep + push, two frames (velocity-ghost reuse)
    dict(vorticity=[0.8, 2.0]),                                   # vorticity confinement with the |curl| ghost exchange
    dict(collision=True),                                         # SDF collision path
    dict(cook=True),                                              # host-buffer entry point (hns_dist_cook), garbage in the ghost entries
    dict(cook=True, collision=True, vorticity=[0.8, 2.0]),
    dict(combustion=False, frames=3, iterations=3),
]
NCCL_MODES = [
    dict(env=dict(HNS_P2P=0)),
    dict(env=dict(HNS_P2P=0), vorticity=[0.8, 2.0], collision=True),
    dict(env=dict(HNS_P2P=0), cook=True),
    dict(env=dict(HNS_P2P=0), native=False, combustion=False),    # exchanges driven from Python through torch.distributed
]


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(world: int, modes, share_gpu: bool, timeout: int = 600):
    env = dict(os.environ, HNS_TEST_MODES=json.dumps(modes), HNS_TEST_SHARE_GPU="1" if share_gpu else "0", MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "sharded_worker.py")]
    r = subprocess.run(cmd, env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    reports = [json.loads(l.split(" ", 1)[1]) for l in r.stdout.splitlines() if l.startswith("SHARDED_PARITY {")]
    assert r.returncode == 0 and "SHARDED_PARITY_SUMMARY OK" in r.stdout, r.stdout[-6000:]
    assert len(reports) == len(modes)
    for rep in reports:
        assert rep["ok"] and all("bitwise ok" in f for f in rep["fields"]), rep
    return reports


def _gpus() -> int:
    import torch

    return torch.cuda.device_count()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_frame_is_bitwise_the_single_gpu_frame_peer_memory(world):
    share = _gpus() < world or bool(int(os.environ.get("HNS_TEST_FORCE_SHARE", "0")))
    reports = _run(world, P2P_MODES, share)
    assert all(r["p2p"] for r in reports)
    assert reports[0]["exchanges_per_frame"] >= 2 * 12       # the pressure ghosts travel after every half-sweep
    # the sharded frame runs the packed (third-generation) advection kernels too: advect_scalars in both frames, advect_vector in the
    # second one (velocity ghosts and group 0 carried over); none with collision data
    assert reports[0]["packed_advection_launches"] == 3 and reports[2]["packed_advection_launches"] == 0


def test_sharded_frame_is_bitwise_the_single_gpu_frame_nccl():
    if _gpus() < 2:
        pytest.skip("the ncclSend/ncclRecv fallback needs one GPU per rank")
    reports = _run(2, NCCL_MODES, False)
    assert not any(r["p2p"] for r in reports)


def test_sharded_frame_four_ranks():
    if _gpus() < 4:
        pytest.skip("needs 4 GPUs")
    _run(4, P2P_MODES[:1] + P2P_MODES[1:4] + NCCL_MODES[:1], False)
