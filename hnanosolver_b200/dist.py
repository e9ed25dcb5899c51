"""Spatially sharded frames: one process per GPU, leaves partitioned into contiguous ranges of the NanoVDB-ordered leaf list,
ghost leaves (26-neighbourhood) exchanged over NCCL between the steps that need them.

The reference is single-GPU (SURVEY.md 2.1: no NCCL/MPI anywhere); this module is new. What it must preserve is the result:
the concatenation of the ranks' owned leaves equals the single-GPU frame bit for bit (tests/test_dist_cpu.py checks the
decomposition logic with world_size 2 over gloo, the GPU scaling run checks it over NCCL).

Exchange points of one frame (ghost depth = one leaf = 8 voxels; valid for back-traces up to 3 voxels + the BFECC forward step):
    velocity                       -> advect_vector
    advected velocity              -> divergence
    red pressure after a red sweep, black pressure after a black sweep     (2 x iterations, half bricks: 1 KB per ghost leaf)
    projected velocity + scalars   -> advect_scalars
Divergence needs no exchange (a half-sweep reads it only at the voxels it updates). Ghost leaves are swept like owned leaves;
what a rank computes on them is overwritten by the owner's values at the next exchange.
"""
from __future__ import annotations

import time
from dataclasses import dataclass

import numpy as np

from . import synth

# field ids of hns_state_pack_leaves / hns_state_unpack_leaves (include/hns_b200.h)
F_VEL, F_ADV, F_P_RED, F_P_BLK, F_DIV_RED, F_DIV_BLK, F_SCALAR0 = (0, 1, 2), (3, 4, 5), 6, 7, 8, 9, 10


import os as _os

_DEBUG_SYNC = bool(int(_os.environ.get("HNS_DEBUG_SYNC", "0")))


def floats_per_leaf(field: int) -> int:
    return 256 if 6 <= field <= 9 else 512


# ------------------------------------------------------------------------------------------------------------------
# partition (pure numpy: runs identically on every rank)
# ------------------------------------------------------------------------------------------------------------------
def _coord_keys(origins: np.ndarray) -> np.ndarray:
    o = (origins.astype(np.int64) >> 3) + (1 << 20)
    return (o[:, 0] << 42) | (o[:, 1] << 21) | o[:, 2]


@dataclass
class ShardPlan:
    rank: int
    world: int
    ranges: np.ndarray            # [world+1] leaf-range boundaries in the global NanoVDB-ordered list
    local_ids: np.ndarray         # global leaf ids present on this rank (owned + ghost), ascending == NanoVDB order
    owned_local: np.ndarray       # bool [n_local]
    send: dict                    # peer -> local indices of owned leaves the peer holds as ghosts (ascending global id)
    recv: dict                    # peer -> local indices of ghost leaves owned by the peer   (ascending global id)

    @property
    def n_owned(self) -> int:
        return int(self.owned_local.sum())

    @property
    def n_local(self) -> int:
        return int(self.local_ids.shape[0])


def make_plan(global_origins: np.ndarray, world: int, rank: int) -> ShardPlan:
    """Contiguous, count-balanced ranges of the sorted leaf list; ghosts = 26-neighbours owned by another rank, plus global leaf 0
    on every rank: advect_scalars reads "array element 0" for inactive voxels (reference src/Cuda/Kernel.cu:192,225), and with
    leaf 0 held as a ghost (it sorts first, so it is LOCAL leaf 0 too) the local element 0 IS the global one after the exchange
    that precedes advect_scalars -- no broadcast, no special case in the kernels."""
    L = global_origins.shape[0]
    ranges = np.array([(L * r) // world for r in range(world + 1)], np.int64)
    owner = np.searchsorted(ranges, np.arange(L), side="right") - 1
    keys = _coord_keys(global_origins)
    order = np.argsort(keys, kind="stable")
    skeys = keys[order]
    lo, hi = int(ranges[rank]), int(ranges[rank + 1])
    mine = np.arange(lo, hi)
    send = {}
    recv = {}
    ghost = set()
    for dx in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dz in (-1, 0, 1):
                if dx == dy == dz == 0:
                    continue
                q = keys[mine] + (np.int64(dx) << 42) + (np.int64(dy) << 21) + np.int64(dz)
                pos = np.searchsorted(skeys, q)
                pos[pos >= L] = L - 1 if L else 0
                ok = skeys[pos] == q
                nbr = order[pos[ok]]
                src = mine[ok]
                far = owner[nbr] != rank
                for peer in np.unique(owner[nbr[far]]):
                    sel = far & (owner[nbr] == peer)
                    send.setdefault(int(peer), set()).update(src[sel].tolist())   # my leaves the peer needs
                    recv.setdefault(int(peer), set()).update(nbr[sel].tolist())   # the peer's leaves I need
                ghost.update(nbr[far].tolist())
    if L and world > 1:
        if rank == 0:
            for peer in range(1, world):
                if ranges[peer + 1] > ranges[peer]:      # a rank without leaves holds nothing
                    send.setdefault(peer, set()).add(0)
        elif hi > lo:
            recv.setdefault(0, set()).add(0)
            ghost.add(0)
    local_ids = np.array(sorted(set(mine.tolist()) | ghost), np.int64)
    owned_local = (local_ids >= lo) & (local_ids < hi)
    to_local = {int(g): i for i, g in enumerate(local_ids.tolist())}
    send = {p: np.array([to_local[g] for g in sorted(v)], np.int32) for p, v in sorted(send.items())}
    recv = {p: np.array([to_local[g] for g in sorted(v)], np.int32) for p, v in sorted(recv.items())}
    return ShardPlan(rank, world, ranges, local_ids, owned_local, send, recv)


# ------------------------------------------------------------------------------------------------------------------
# halo exchange over torch.distributed (NCCL on GPUs, gloo in the CPU tests)
# ------------------------------------------------------------------------------------------------------------------
class HaloExchanger:
    """pack(field, local_ids_tensor, out_tensor) / unpack(field, local_ids_tensor, in_tensor) are supplied by the owner of the
    fields (CUDA kernels of libhns_b200 on the GPU; numpy indexing in the CPU tests)."""

    def __init__(self, plan: ShardPlan, device, pack, unpack, max_fields: int = 8):
        import torch

        self.plan, self.pack, self.unpack = plan, pack, unpack
        self.device = device
        self.ids_send = {p: torch.as_tensor(v, dtype=torch.int32, device=device) for p, v in plan.send.items()}
        self.ids_recv = {p: torch.as_tensor(v, dtype=torch.int32, device=device) for p, v in plan.recv.items()}
        self.buf_send = {p: torch.empty(len(v) * 512 * max_fields, dtype=torch.float32, device=device) for p, v in plan.send.items()}
        self.buf_recv = {p: torch.empty(len(v) * 512 * max_fields, dtype=torch.float32, device=device) for p, v in plan.recv.items()}
        self.max_fields = max_fields
        self.bytes_sent = 0
        self.exchanges = 0

    def exchange(self, fields) -> None:
        import torch.distributed as dist

        fields = list(fields)
        assert len(fields) <= self.max_fields
        ops, views = [], {}
        for p in sorted(set(self.ids_send) | set(self.ids_recv)):
            ns, nr = len(self.plan.send.get(p, ())), len(self.plan.recv.get(p, ()))
            off_s = off_r = 0
            vs, vr = [], []
            for f in fields:
                fpl = floats_per_leaf(f)
                if ns:
                    seg = self.buf_send[p][off_s:off_s + ns * fpl]
                    self.pack(f, self.ids_send[p], seg)
                    off_s += ns * fpl
                if nr:
                    vr.append((f, self.buf_recv[p][off_r:off_r + nr * fpl]))
                    off_r += nr * fpl
            if ns:
                ops.append(dist.P2POp(dist.isend, self.buf_send[p][:off_s], p))
                self.bytes_sent += off_s * 4
            if nr:
                ops.append(dist.P2POp(dist.irecv, self.buf_recv[p][:off_r], p))
            views[p] = vr
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        if _DEBUG_SYNC:
            import torch

            torch.cuda.synchronize()
        for p, vr in views.items():
            for f, seg in vr:
                self.unpack(f, self.ids_recv[p], seg)
        self.exchanges += 1


# ------------------------------------------------------------------------------------------------------------------
# GPU driver
# ------------------------------------------------------------------------------------------------------------------
class ShardedSimulation:
    """Device-resident state of this rank's shard (owned + ghost leaves) and the frame with ghost exchanges.

    native=True (default): the frame is ONE call into libhns_b200 (hns_dist_frame): kernels and NCCL send/recv are issued from
    C++ on one stream. native=False drives the same steps from Python through HaloExchanger / torch.distributed (slower: a
    trip through the interpreter per exchange); kept as an independent cross-check."""

    def __init__(self, plan: ShardPlan, local_origins: np.ndarray, voxel_size: float, n_scalars: int, device, native: bool = True):
        import ctypes as C

        import torch
        import torch.distributed as tdist

        from . import _lib
        from . import launchers as H

        self.plan, self.device = plan, device
        self.grid = H.create_index_grid_from_origins(local_origins, voxel_size)
        self.sim = H.Simulation(self.grid, n_scalars)
        self.voxel_size = voxel_size
        self.n_scalars = n_scalars
        self.omega = H.omega_compute(voxel_size)
        self.full = False
        self.native = native
        self._torch = torch

        def stream():
            return torch.cuda.current_stream(device).cuda_stream

        self._stream = stream
        self._dist = None
        if native:
            L = _lib.lib()
            # NCCL carries the ghost bricks only in the fallback mode (HNS_P2P=0). Without it -- a gloo process group, e.g. two
            # ranks time-sharing ONE GPU in the tests, which NCCL refuses -- the peer-memory exchange is the only data path.
            use_nccl = plan.world > 1 and tdist.get_backend() == "nccl" and not bool(int(_os.environ.get("HNS_NO_NCCL", "0")))
            h = C.c_void_p()
            if use_nccl:
                uid = (C.c_uint8 * 128)()
                if plan.rank == 0:
                    _lib.check(L.hns_dist_unique_id(uid))
                box = [bytes(uid)]
                tdist.broadcast_object_list(box, src=0)
                uid = (C.c_uint8 * 128).from_buffer_copy(box[0])
                _lib.check(L.hns_dist_create(uid, plan.rank, plan.world, C.byref(h)))
            else:
                _lib.check(L.hns_dist_create(None, plan.rank, plan.world, C.byref(h)))
            self._dist = h
            peers = sorted(set(plan.send) | set(plan.recv))
            n = len(peers)
            empty = np.zeros(0, np.int32)
            snd = [np.ascontiguousarray(plan.send.get(p, empty), np.int32) for p in peers]
            rcv = [np.ascontiguousarray(plan.recv.get(p, empty), np.int32) for p in peers]
            owned = np.ascontiguousarray(np.nonzero(plan.owned_local)[0], np.int32)
            self._keep = (snd, rcv, owned)
            _lib.check(L.hns_dist_set_plan(
                h, self.sim._h, n, (C.c_int * max(n, 1))(*peers), (C.c_uint64 * max(n, 1))(*[len(a) for a in snd]),
                (_lib.c_i32p * max(n, 1))(*[a.ctypes.data_as(_lib.c_i32p) for a in snd]), (C.c_uint64 * max(n, 1))(*[len(a) for a in rcv]),
                (_lib.c_i32p * max(n, 1))(*[a.ctypes.data_as(_lib.c_i32p) for a in rcv]), len(owned), owned.ctypes.data_as(_lib.c_i32p)))
            self.ex = None
            self.p2p = False
            if plan.world > 1 and (not use_nccl or bool(int(_os.environ.get("HNS_P2P", "1")))):
                # direct peer-memory exchange: all-gather every rank's IPC handle and region offsets, connect to the peers
                handle = (C.c_uint8 * 192)()
                offs = (C.c_uint64 * max(n, 1))()
                _lib.check(L.hns_dist_ipc_prepare(h, handle, offs))
                mine = (bytes(handle), {p: int(offs[i]) for i, p in enumerate(peers)}, {p: np.asarray(v, np.int32) for p, v in plan.recv.items()})
                allinfo = [None] * plan.world
                tdist.all_gather_object(allinfo, mine)
                for i, p in enumerate(peers):
                    ph, poffs, precv = allinfo[p]
                    # the peer's recv list for me lists, in the same (global id) order as my send list, its local ids of my leaves
                    theirs = np.ascontiguousarray(precv.get(plan.rank, empty), np.int32)
                    assert len(theirs) == len(snd[i])
                    _lib.check(L.hns_dist_ipc_connect(h, i, (C.c_uint8 * 192).from_buffer_copy(ph), poffs.get(plan.rank, 0),
                                                      theirs.ctypes.data_as(_lib.c_i32p)))
                _lib.check(L.hns_dist_ipc_finish(h))
                tdist.barrier()
                self.p2p = True
        else:
            def pack(field, ids, out):
                self.sim.pack_leaves(field, ids.data_ptr(), ids.numel(), out.data_ptr(), stream())

            def unpack(field, ids, src):
                self.sim.unpack_leaves(field, ids.data_ptr(), ids.numel(), src.data_ptr(), stream())

            self.ex = HaloExchanger(plan, device, pack, unpack, max_fields=3 + n_scalars)

    def check_errors(self) -> None:
        """raises if a peer-flag wait timed out on the device (the frame then ran on stale ghosts)"""
        if self._dist is not None:
            import ctypes as C

            from . import _lib

            e = C.c_uint32()
            _lib.check(_lib.lib().hns_dist_error(self._dist, C.byref(e)))
            if e.value & 0xff == 11:
                raise RuntimeError("the multigrid level-1 gather timed out waiting for a rank: the frame ran on a stale coarse right-hand side")
            if e.value & 0xff:
                raise RuntimeError(f"ghost exchange timed out waiting for a peer on channel {(e.value & 0xff) - 1}: the frame ran on stale ghosts")
            if e.value & 0x100:
                raise RuntimeError("a semi-Lagrangian sample landed beyond the shard's one-leaf ghost layer (CFL too large for a sharded run)")

    def close(self):
        if self._dist is not None:
            from . import _lib

            self._torch.cuda.synchronize()
            if self.plan.world > 1:
                import torch.distributed as tdist

                tdist.barrier()  # nobody unmaps a block a peer may still be writing to
            _lib.lib().hns_dist_destroy(self._dist)
            self._dist = None

    @property
    def exchanges(self) -> int:
        from . import _lib

        return int(_lib.lib().hns_dist_exchanges(self._dist)) if self.native else self.ex.exchanges

    @property
    def bytes_sent(self) -> int:
        from . import _lib

        return int(_lib.lib().hns_dist_bytes_sent(self._dist)) if self.native else self.ex.bytes_sent

    def set_pressure_solver(self, global_origins, cycles: int = 2, nu_pre: int = 2, nu_post: int = 2, omega_smooth: float = 1.15,
                            max_levels: int = 0) -> None:
        """Collective. frame() / cook() / frame_timed() then solve the pressure with `cycles` sharded V(nu_pre, nu_post) multigrid cycles
        (hns_dist_set_pressure_solver) instead of the red-black sweeps: level 0 is this shard, the coarse levels -- a Multigrid over the
        GLOBAL leaf origins `global_origins` (NanoVDB order, as given to make_plan) -- are replicated on every rank. The owned voxels equal
        Simulation.set_pressure_solver(Multigrid(global grid, max_levels), ...) on one GPU bit for bit. global_origins=None switches
        back to red-black. Needs the native frame and, with more than one rank, the peer-memory exchange."""
        import ctypes as C

        from . import _lib
        from . import launchers as H

        if not self.native:
            raise NotImplementedError("the sharded multigrid solve needs the native sharded frame (native=True)")
        L = _lib.lib()
        if global_origins is None:
            _lib.check(L.hns_dist_set_pressure_solver(self._dist, self.sim._h, None, None, 0, 0, 0, 0.0, None))
            self._mg = None
            return
        grid = H.create_index_grid_from_origins(global_origins, self.voxel_size)
        mg = H.Multigrid(grid, max_levels)
        l2g = np.ascontiguousarray(self.plan.local_ids, np.int32)
        handle = (C.c_uint8 * 64)()
        _lib.check(L.hns_dist_set_pressure_solver(self._dist, self.sim._h, mg._h, l2g.ctypes.data_as(_lib.c_i32p), int(cycles), int(nu_pre),
                                                  int(nu_post), float(omega_smooth), handle))
        self._mg = (grid, mg)   # the library uses the hierarchy (and it the grid) until the next call
        if self.plan.world > 1:
            import torch.distributed as tdist

            handles = [None] * self.plan.world
            tdist.all_gather_object(handles, bytes(handle))
            for r, hb in enumerate(handles):
                if r != self.plan.rank:
                    _lib.check(L.hns_dist_mg_connect(self._dist, r, (C.c_uint8 * 64).from_buffer_copy(hb)))
        _lib.check(L.hns_dist_mg_finish(self._dist))
        if self.plan.world > 1:
            tdist.barrier()

    @property
    def mg_gathers(self) -> tuple[int, int]:
        """(V-cycles that gathered the level-1 right-hand side, bytes this rank stored into the other ranks' copies)"""
        from . import _lib

        return int(_lib.lib().hns_dist_mg_gathers(self._dist)), int(_lib.lib().hns_dist_mg_gather_bytes(self._dist))

    def set_combustion(self, names, params):
        self.sim.set_combustion(True, names.index("fuel"), names.index("waste"), names.index("temperature"), names.index("flame"), params)
        self.full = True

    def upload(self, velocity, scalars):
        self.sim.upload(velocity, scalars)

    def frame(self, iterations: int, dt: float) -> None:
        if self.native:
            import ctypes as C

            from . import _lib

            _lib.check(_lib.lib().hns_dist_frame(self._dist, self.sim._h, iterations, dt, C.c_void_p(self._stream())))
            return
        s, ex, st = self.sim, self.ex, self._stream()
        from . import _lib

        if _lib.lib().hns_state_vorticity_active(s._h) or _lib.lib().hns_state_collision_active(s._h):
            raise NotImplementedError("vorticity confinement / SDF collision are only wired into the native sharded frame (native=True)")
        ex.exchange(F_VEL)
        s.advect_velocity(dt, st)
        ex.exchange(F_ADV)
        s.divergence(True, st)
        if self.full:
            s.combustion_buoyancy(dt, st)
        s.pressure_init(st)
        for _ in range(iterations):
            s.pressure_half_sweep(0, self.omega, False, st)
            ex.exchange([F_P_RED])
            s.pressure_half_sweep(1, self.omega, True, st)
            ex.exchange([F_P_BLK])
        s.subtract_gradient(True, st)
        ex.exchange(list(F_VEL) + [F_SCALAR0 + i for i in range(self.n_scalars)])
        s.advect_scalars(dt, 0, st)   # "inactive -> element 0": global leaf 0 is local leaf 0 on every rank (make_plan)

    def cook(self, velocity: np.ndarray, scalars, iterations: int, dt: float) -> None:
        """One sharded cook on this rank's HOST arrays (local voxels: owned + ghost leaves), in place, synchronous: the per-rank
        counterpart of Compute_Sim (hns_dist_cook). velocity float32 (n, 3), scalars a list of float32 (n,); pinned memory recommended."""
        import ctypes as C

        from . import _lib

        if not self.native:
            raise NotImplementedError("cook() needs the native sharded frame")
        assert velocity.dtype == np.float32 and velocity.flags.c_contiguous and velocity.size == 3 * self.sim.n
        ptrs = (_lib.c_f32p * max(1, len(scalars)))()
        for i, a in enumerate(scalars):
            assert a.dtype == np.float32 and a.flags.c_contiguous and a.size == self.sim.n
            ptrs[i] = a.ctypes.data_as(_lib.c_f32p)
        _lib.check(_lib.lib().hns_dist_cook(self._dist, self.sim._h, velocity.ctypes.data_as(_lib.c_f32p), len(scalars), ptrs, iterations, dt,
                                            C.c_void_p(self._stream())))

    PHASES = ("exch_vel", "advect_vector", "exch_adv", "div+comb", "pressure", "gradient", "exch_final", "advect_scalars")

    def frame_timed(self, iterations: int, dt: float) -> dict:
        import ctypes as C

        from . import _lib

        ms = (C.c_float * 8)()
        _lib.check(_lib.lib().hns_dist_frame_timed(self._dist, self.sim._h, iterations, dt, C.c_void_p(self._stream()), ms))
        return dict(zip(self.PHASES, [float(x) for x in ms]))

    def owned(self, arr: np.ndarray) -> np.ndarray:
        """Rows of a per-voxel local array that belong to owned leaves."""
        m = np.repeat(self.plan.owned_local, 512)
        return arr[m]


# ------------------------------------------------------------------------------------------------------------------
# sharded frame == single-GPU frame, bit for bit (run by tests/test_sharded_gpu.py and by bench.py --gpus N before it times anything)
# ------------------------------------------------------------------------------------------------------------------
def sharded_parity_check(rank: int, world: int, device, *, box=(256, 128, 128), fill: float = 0.35, seed: int = 7, iterations: int = 12,
                         frames: int = 2, collision: bool = False, vorticity=(0.0, 1.0), cook: bool = False, combustion: bool = True,
                         native: bool = True, multigrid: dict | None = None):
    """Collective. Runs `frames` sharded frames of a small sparse box and, on rank 0, the same frames on ONE GPU over the whole
    domain; compares the owned voxels of every rank (velocity, every scalar, pressure) with np.array_equal.
    Returns (ok, report) on rank 0 and (None, None) elsewhere. Two frames exercise the reuse of the velocity ghosts across frames.
    multigrid = dict(cycles, nu_pre, nu_post, omega, max_levels, red_black_frames): both sides solve the pressure with that many V-cycles
    (ShardedSimulation.set_pressure_solver against Simulation.set_pressure_solver over the whole domain); red_black_frames > 0 then
    switches both back to red-black for that many more frames."""
    import torch
    import torch.distributed as tdist

    from . import _lib
    from . import launchers as H

    go = global_sparse_origins(box, fill, seed)
    vel, den, tem = synth._swirl_fields(max(box))
    wg = synth._finish("parity", go, vel, [den, tem], ["density", "temperature"], 40, seed, with_coords=False)
    plan = make_plan(go, world, rank)
    lo = np.repeat(plan.local_ids, 512) * 512 + np.tile(np.arange(512), plan.n_local)
    comb = synth.combustion_fields(wg)
    names = ["density", "fuel", "waste", "temperature", "flame"]
    gfields = [wg.scalars[0]] + [comb[k] for k in names[1:]]
    if collision:  # a sphere collider as the last scalar, hasCollision path on
        off = np.stack(np.unravel_index(np.arange(512), (8, 8, 8)), 1)
        gc = (np.repeat(go, 512, axis=0) + off[np.tile(np.arange(512), go.shape[0])]).astype(np.float32)
        centre = np.array([box[0] / 2, box[1] / 2, box[2] / 2], np.float32)
        sdf = (0.05 * (np.sqrt(((gc - centre) ** 2).sum(1)) - 20.0)).astype(np.float32)
        sdf[0] = 0.0
        names, gfields = names + ["collision_sdf"], gfields + [sdf]
    NS = len(gfields)
    P = H.CombustionParams(0.5, 2.0, 1.5, 0.1, float(vorticity[0]), float(vorticity[1]))
    mgc = None
    if multigrid is not None:
        mgc = dict(cycles=2, nu_pre=2, nu_post=2, omega=1.15, max_levels=0, red_black_frames=0)
        mgc.update(multigrid)
    sh = ShardedSimulation(plan, np.ascontiguousarray(go[plan.local_ids]), wg.voxel_size, NS, device, native=native)
    try:
        if collision:
            sh.sim.set_collision(NS - 1)
        if combustion:
            sh.set_combustion(names, P)
        if mgc is not None:
            sh.set_pressure_solver(go, mgc["cycles"], mgc["nu_pre"], mgc["nu_post"], mgc["omega"], mgc["max_levels"])
        gathers_before = sh.mg_gathers if native else (0, 0)
        rb_frames = mgc["red_black_frames"] if mgc is not None else 0
        m = np.repeat(plan.owned_local, 512)
        lv, lf = np.ascontiguousarray(wg.velocity[lo]), [np.ascontiguousarray(f[lo]) for f in gfields]
        packed_before = _lib.lib().hns_packed_advection_launches()
        if cook:
            # ghost entries of the host inputs are deliberately garbage: hns_dist_cook's contract says they need not be valid
            lv[~m] = np.float32(1e30)
            for i, a in enumerate(lf):
                a[~m] = np.float32(-7.0)
            for _ in range(frames):
                sh.cook(lv, lf, iterations, wg.dt)
            if rb_frames:
                sh.set_pressure_solver(None)
                for _ in range(rb_frames):
                    sh.cook(lv, lf, iterations, wg.dt)
            mine = [lv[m]] + [a[m] for a in lf] + [sh.sim.aux(1)[m]]
        else:
            sh.upload(lv, lf)
            for _ in range(frames):
                sh.frame(iterations, wg.dt)
            if rb_frames:
                torch.cuda.synchronize()
                sh.check_errors()
                sh.set_pressure_solver(None)
                for _ in range(rb_frames):
                    sh.frame(iterations, wg.dt)
            torch.cuda.synchronize()
            sh.check_errors()
            mine = [sh.sim.velocity()[m]] + [sh.sim.scalar(i)[m] for i in range(NS)] + [sh.sim.aux(1)[m]]
        packed_launches = int(_lib.lib().hns_packed_advection_launches() - packed_before)   # third-generation advection launches of this rank
        gathers = [a - b for a, b in zip(sh.mg_gathers, gathers_before)] if native else [0, 0]
        gathered = [None] * world
        tdist.all_gather_object(gathered, mine)
        ok, report = None, None
        if rank == 0:
            g = H.create_index_grid_from_origins(go, wg.voxel_size)
            sim = H.Simulation(g, NS)
            sim.upload(wg.velocity, gfields)
            if collision:
                sim.set_collision(NS - 1)
            if combustion:
                sim.set_combustion(True, 1, 2, 3, 4, P)
            ref_mg = None
            if mgc is not None:
                ref_mg = H.Multigrid(g, mgc["max_levels"])
                sim.set_pressure_solver(ref_mg, mgc["cycles"], mgc["nu_pre"], mgc["nu_post"], mgc["omega"])
            for _ in range(frames):
                sim.step(iterations, wg.dt)
            if rb_frames:
                sim.set_pressure_solver(None)
                for _ in range(rb_frames):
                    sim.step(iterations, wg.dt)
            sim.sync()
            ref = [sim.velocity()] + [sim.scalar(i) for i in range(NS)] + [sim.aux(1)]
            if cook and collision:
                ref[NS] = gfields[-1]   # the resident state keeps the SDF; hns_dist_cook hands the caller's block back untouched
            ok, lines = True, []
            for k, nm in enumerate(["velocity"] + names + ["pressure"]):
                got = np.concatenate([gathered[r][k] for r in range(world)])
                same = bool(np.array_equal(got, ref[k]))
                ok &= same
                bad = np.nonzero((got != ref[k]).reshape(got.shape[0], -1).any(1))[0]
                lines.append(f"{nm}: bitwise {'ok' if same else 'MISMATCH'} ({bad.size}/{got.shape[0]} voxels differ"
                             + (f", max|diff| {np.abs(got.astype(np.float64) - ref[k]).max():.3e}, first leaves {np.unique(bad // 512)[:6].tolist()}" if bad.size else "") + ")")
            report = dict(ok=ok, leaves=int(go.shape[0]), world=world, frames=frames, iterations=iterations, p2p=bool(getattr(sh, "p2p", False)),
                          native=native, collision=collision, vorticity=list(vorticity), cook=cook, exchanges_per_frame=sh.exchanges // max(frames, 1),
                          packed_advection_launches=packed_launches, multigrid=mgc, mg_gathers=gathers[0], mg_gather_bytes=gathers[1],
                          mg_levels=ref_mg.num_levels if ref_mg is not None else 0, fields=lines)
            del sim
        tdist.barrier()
        return ok, report
    finally:
        sh.close()


# ------------------------------------------------------------------------------------------------------------------
# weak-scaling workload: the bounding box grows with the number of ranks
# ------------------------------------------------------------------------------------------------------------------
WEAK_BOX = {1: (512, 512, 512), 2: (1024, 512, 512), 4: (1024, 1024, 512), 8: (1024, 1024, 1024)}


def global_sparse_origins(box, fill: float = 0.30, seed: int = 4) -> np.ndarray:
    """Leaf origins of the blobby sparse smoke (config 4 recipe) inside an arbitrary box, NanoVDB order. For (512,512,512) this is
    exactly synth.sparse_smoke(512)."""
    n = tuple(b // 8 for b in box)
    noise = synth.smooth_lattice_noise(n, tuple(max(2, k // 8) for k in n), seed)
    mask = noise > np.quantile(noise, 1.0 - fill)
    return synth.origins_from_mask(mask)


def build_sharded_workload(name: str, rank: int, world: int, scaling: str = "weak"):
    """(workload of the LOCAL leaves, field names, fields, frame kind); the plan is attached as workload.meta['plan'].
    c4, scaling "weak": the sparse-smoke box grows with the number of ranks (512^3 per GPU); c4, "strong": BASELINE.json config 4 as
    stated -- the 512^3 box split over the ranks; c5: the 1024^3 narrow band (~2e8 voxels) split over the ranks (a fixed total)."""
    if name == "c5":
        R = 1024
        gorigins, half_width = synth.narrow_band_origins(R, 2.0e8)
        box, label, scaling = (R, R, R), f"c5 narrow band (half width {half_width:.1f} voxels) in a {R}^3 box", "strong"
    elif name == "c4":
        if scaling == "strong":
            box = (512, 512, 512)
        else:
            box = WEAK_BOX.get(world)
            if box is None:
                raise SystemExit(f"no weak-scaling box defined for {world} ranks (1, 2, 4, 8)")
        gorigins = global_sparse_origins(box)
        label = f"c4 {scaling} scaling: sparse smoke ~30% of a {box[0]}x{box[1]}x{box[2]} box"
    else:
        raise SystemExit("multi-GPU bench: --workload c4 (weak: 512^3 of sparse smoke per GPU; --scaling strong: the 512^3 box split) or c5")
    plan = make_plan(gorigins, world, rank)
    local = np.ascontiguousarray(gorigins[plan.local_ids])
    vel, density, temperature = synth._swirl_fields(max(box))
    w = synth._finish(f"{name}/{box[0]}x{box[1]}x{box[2]}/rank{rank}", local, vel, [density, temperature], ["density", "temperature"], 40, 4,
                      with_coords=False, meta=dict(box=box, global_leaves=int(gorigins.shape[0]), label=label, scaling=scaling))
    w.meta["plan"] = plan
    fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
    return w, list(fields), list(fields.values()), "full"


def run_sharded_bench(w, names, fields, full, args, iterations, params6, rank, world, local_rank):
    """Timed region per the bench contract: W warm-up frames, K frames bracketed by barrier + synchronize, max over ranks."""
    import torch
    import torch.distributed as dist

    from . import _lib
    from . import launchers as H

    plan: ShardPlan = w.meta["plan"]
    dev = torch.device("cuda", local_rank)
    # Before anything is timed: the sharded frame must equal the single-GPU frame bit for bit on a small box (two frames, full
    # frame; then the host-buffer cook with vorticity confinement and the collision path on). A mismatch ends the run.
    parity = []
    for mode in (dict(), dict(cook=True, collision=True, vorticity=(0.8, 2.0))):
        ok, report = sharded_parity_check(rank, world, dev, **mode)
        if rank == 0:
            print(f"[sharded parity] {report}", file=__import__("sys").stderr, flush=True)
            parity.append(report)
            if not ok:
                raise SystemExit("sharded frame != single-GPU frame: refusing to time a wrong result")
    sh = ShardedSimulation(plan, w.origins, w.voxel_size, len(fields), dev)
    if full:
        sh.set_combustion(names, H.CombustionParams(*params6))
    vel_pinned = torch.from_numpy(w.velocity).pin_memory()
    sc_pinned = [torch.from_numpy(a).pin_memory() for a in fields]

    def restore():
        sh.upload(vel_pinned.numpy(), [t.numpy() for t in sc_pinned])

    restore()
    dist.barrier()  # pinning and uploading take a different time on every rank; a frame's flag waits give up after ~4 s
    for _ in range(args.warmup):
        sh.frame(iterations, w.dt)
    torch.cuda.synchronize()
    restore()
    # K timed frames on the evolving state (every frame does the same amount of work), device time from CUDA events on the launch stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _lib.lib().hns_launch_count_reset()
    dist.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.time()
    packed0 = _lib.lib().hns_packed_advection_launches()
    e0.record()
    for _ in range(args.steps):
        sh.frame(iterations, w.dt)
    e1.record()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    packed_launches = int(_lib.lib().hns_packed_advection_launches() - packed0)   # this rank's third-generation advection launches
    dist.barrier()
    phases = sh.frame_timed(iterations, w.dt) if sh.native else {}
    sh.check_errors()
    pr = torch.tensor([float(phases.get("pressure", 0.0)), float(plan.n_owned * 512)], device=dev)
    pr_all = [torch.zeros_like(pr) for _ in range(world)]
    dist.all_gather(pr_all, pr)
    slowest = max(pr_all, key=lambda t: float(t[0]))
    log = __import__("sys").stderr
    print(f"[rank {rank}] owned {plan.n_owned} ghost {plan.n_local - plan.n_owned} peers { {p: len(v) for p, v in plan.send.items()} } "
          f"phases(ms) { {k: (round(v, 3) if isinstance(v, float) else v) for k, v in phases.items()} }", file=log, flush=True)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = torch.tensor([float(_lib.lib().hns_launch_count())], device=dev)
    dist.all_reduce(launches, op=dist.ReduceOp.SUM)
    owned = torch.tensor([float(plan.n_owned * 512), float(plan.n_local * 512), float(sh.bytes_sent)], device=dev)
    dist.all_reduce(owned, op=dist.ReduceOp.SUM)
    sh.check_errors()
    ms_step = float(ms.item()) / args.steps
    n_owned_total, n_local_total = int(owned[0].item()), int(owned[1].item())

    # end to end: one sharded cook per step on this rank's pinned host arrays, in place (hns_dist_cook: upload, frame, download)
    restore()
    torch.cuda.synchronize()
    vel_np, sc_np = vel_pinned.numpy(), [t.numpy() for t in sc_pinned]

    def cook():
        sh.cook(vel_np, sc_np, iterations, w.dt)

    cook()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        cook()
    torch.cuda.synchronize()
    dist.barrier()
    e2e = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.e2e_steps], device=dev)
    dist.all_reduce(e2e, op=dist.ReduceOp.MAX)
    # the floor of that call contract: the same bytes up and down over every rank's PCIe link at the same time, no kernels in between
    dev_bufs = [torch.empty_like(t, device=dev) for t in [vel_pinned] + sc_pinned]
    host_bufs = [vel_pinned] + sc_pinned

    def copies():
        for dbuf, hbuf in zip(dev_bufs, host_bufs):
            dbuf.copy_(hbuf, non_blocking=True)
        for dbuf, hbuf in zip(dev_bufs, host_bufs):
            hbuf.copy_(dbuf, non_blocking=True)

    copies()
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        copies()
    torch.cuda.synchronize()
    floor = torch.tensor([(time.perf_counter() - t0) * 1e3 / 3], device=dev)
    dist.all_reduce(floor, op=dist.ReduceOp.MAX)
    del dev_bufs
    S = len(fields)
    box = w.meta["box"]
    return {"metric": "active voxel-updates/s per advect+project frame", "value": n_owned_total / (ms_step * 1e-3), "unit": "voxel-updates/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": w.meta["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{w.meta['label']}, {n_owned_total} active voxels over "
                                   f"{world} GPUs (+{n_local_total - n_owned_total} ghost voxels), frame=full, I={iterations}, S={S}",
                       "parallelism": f"spatial leaf-range sharding x{world}, ghost-leaf exchange by " + ("direct peer-memory stores + flags over NVLink (CUDA IPC)" if getattr(sh, "p2p", False) else "ncclSend/ncclRecv") + f", issued from C++, boundary sweeps + exchange pipelined against interior sweeps ({sh.exchanges // (args.steps + args.warmup + args.e2e_steps + 1)} exchanges/frame)",
                       "l2": "per-rank fields larger than L2; no flush"},
            "e2e": {"value": n_owned_total / (float(e2e.item()) * 1e-3), "unit": "voxel-updates/s", "ms_per_step": float(e2e.item()),
                    "h2d_bytes_per_step": int(n_local_total * (12 + 4 * S)), "d2h_bytes_per_step": int(n_local_total * (12 + 4 * S)),
                    "copy_floor_ms": float(floor.item()),
                    "call": "ShardedSimulation.cook (hns_dist_cook) per rank on pinned host arrays of its shard, in place, synchronous; "
                            "copy_floor_ms = the same bytes up then down on all ranks at once without any kernel"},
            "gpu_launches": int(launches.item()), "packed_advection_launches_rank0": packed_launches,
            "sharded_parity": "bitwise-ok" if parity and all(r["ok"] for r in parity) else None,
            "sharded_parity_detail": [{k: r[k] for k in ("leaves", "world", "frames", "iterations", "p2p", "collision", "vorticity", "cook")} for r in parity],
            "_timed_wall": (t_wall0, t_wall1), "_pressure": (float(slowest[0]), float(slowest[1])),
            "halo_bytes_per_frame": int(owned[2].item() / (args.steps + args.warmup + args.e2e_steps + 1))}
