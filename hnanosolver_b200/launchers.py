"""Host-side mirror of the reference's launcher interface on top of the C ABI (include/hns_b200.h).

Same names, argument meaning and error behaviour as the reference's extern "C" entry points:

    CreateIndexGrid          src/Cuda/HNanoSolver.cu:387-390
    Compute_Sim              src/Cuda/HNanoSolver.cu:393-396
    AdvectIndexGrid          src/Cuda/Advection.cu:169-171
    AdvectIndexGridVelocity  src/Cuda/Advection.cu:173-175
    ProjectNonDivergent      src/Cuda/PressureProjection.cu:132-135
    Divergence               src/Cuda/PressureProjection.cu:127-129
    CombustionKernel         src/Cuda/Combustion.cu:67-70

They operate in place on a GridIndexedData host sidecar and are synchronous, like the reference. std::invalid_argument maps
to ValueError (HnsInvalidArgument), std::runtime_error to RuntimeError (HnsError). `Simulation` is the device-resident
variant used by the headless driver and bench.py: state stays in HBM across frames instead of crossing PCIe every frame.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import CombustionParams, HnsError, check, c_f32p, c_i32p, c_u64p
from .grid_data import FLOAT, VEC3F, GridIndexedData

__all__ = ["CreateIndexGrid", "Compute_Sim", "AdvectIndexGrid", "AdvectIndexGridVelocity", "ProjectNonDivergent", "Divergence",
           "CombustionKernel", "IndexGridHandle", "Simulation", "Multigrid", "Source", "ValueGrid", "build_domain", "CombustionParams"]


def _fp(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags.c_contiguous
    return a.ctypes.data_as(c_f32p)


def _ip(a: np.ndarray):
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(c_i32p)


def omega_compute(voxel_size: float) -> float:
    """omega of the all-in-one frame: 2/(1+sinf(float(3.14159)*h)) in float (reference src/Cuda/HNanoSolver.cu:257)"""
    return float(_lib.lib().hns_omega_compute(voxel_size))


def _stream(stream) -> C.c_void_p:
    if stream is None:
        return C.c_void_p(0)
    if hasattr(stream, "cuda_stream"):  # torch.cuda.Stream
        return C.c_void_p(stream.cuda_stream)
    return C.c_void_p(int(stream))


class IndexGridHandle:
    """Stands where nanovdb::GridHandle<nanovdb::cuda::DeviceBuffer> stands in the reference: owns the device-side
    NanoVDB ValueOnIndex buffer (plus the leaf tables the kernels use)."""

    def __init__(self, ptr: int | None = None):
        self._h = C.c_void_p(ptr) if ptr else None

    def isEmpty(self) -> bool:
        return not self._h

    def reset(self) -> None:
        if self._h:
            _lib.lib().hns_grid_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.reset()
        except Exception:
            pass

    # --- introspection -----------------------------------------------------------------------------------
    @property
    def num_leaves(self) -> int:
        return _lib.lib().hns_grid_num_leaves(self._h)

    @property
    def num_voxels(self) -> int:
        return _lib.lib().hns_grid_num_voxels(self._h)

    def nanovdb_buffer(self) -> np.ndarray:
        """The NanoVDB 32.7 ValueOnIndex buffer, downloaded to the host."""
        buf = np.empty(_lib.lib().hns_grid_nanovdb_bytes(self._h), np.uint8)
        check(_lib.lib().hns_grid_nanovdb_download(self._h, buf.ctypes.data_as(C.c_void_p)))
        return buf

    def deviceData(self) -> int:
        return _lib.lib().hns_grid_nanovdb_device_ptr(self._h) or 0

    def get_values(self, ijk) -> np.ndarray:
        ijk = np.ascontiguousarray(np.asarray(ijk, np.int32).reshape(-1, 3))
        out = np.empty(ijk.shape[0], np.uint64)
        check(_lib.lib().hns_grid_get_values(self._h, _ip(ijk), ijk.shape[0], out.ctypes.data_as(c_u64p)))
        return out

    def neighbors(self) -> np.ndarray:
        out = np.empty((self.num_leaves, 27), np.int32)
        check(_lib.lib().hns_grid_neighbors_download(self._h, _ip(out)))
        return out


def CreateIndexGrid(data: GridIndexedData, voxelSize: float, validate: bool = False) -> IndexGridHandle:
    """CreateIndexGrid(data, handle, voxelSize): returns the handle instead of filling an out-parameter."""
    h = C.c_void_p()
    coords = data.pCoords()
    n = data.size()
    check(_lib.lib().hns_grid_create_from_coords(_ip(coords) if n else None, n, voxelSize, int(validate), C.byref(h)))
    return IndexGridHandle(h.value)


def create_index_grid_from_origins(origins: np.ndarray, voxelSize: float) -> IndexGridHandle:
    origins = np.ascontiguousarray(np.asarray(origins, np.int32).reshape(-1, 3))
    h = C.c_void_p()
    check(_lib.lib().hns_grid_create_from_origins(_ip(origins) if len(origins) else None, origins.shape[0], voxelSize, C.byref(h)))
    return IndexGridHandle(h.value)


def Compute_Sim(data: GridIndexedData, handle: IndexGridHandle, iteration: int, dt: float, voxelSize: float, params: CombustionParams,
                hasCollision: bool, stream=None) -> None:
    # Compute()'s validation order (HNanoSolver.cu:12-83); the C ABI re-checks the same conditions
    if not voxelSize > 0.0:
        raise _lib.HnsInvalidArgument(-1, "voxelSize must be positive.")
    if dt < 0.0:
        raise _lib.HnsInvalidArgument(-1, "dt (time step) cannot be negative.")
    if iteration <= 0:
        raise _lib.HnsInvalidArgument(-1, "Number of pressure iterations must be positive.")
    if handle is None or handle.isEmpty():
        raise _lib.HnsInvalidArgument(-1, "Invalid nanovdb::GridHandle provided (null grid).")
    if data.size() == 0:
        return
    vec = data.getBlocksOfType(VEC3F)
    floats = data.getBlocksOfType(FLOAT)
    L = _lib.lib()
    if len(vec) != 1:
        raise HnsError(-2, f"Expected exactly one Vec3f block (velocity), found {len(vec)}")
    if not floats:
        raise HnsError(-2, "No float blocks found in input data.")
    vel = data.pValues(VEC3F, vec[0])
    names = (C.c_char_p * len(floats))(*[s.encode() for s in floats])
    ptrs = (c_f32p * len(floats))(*[_fp(data.pValues(FLOAT, s)) for s in floats])
    check(L.hns_compute_sim(handle._h, _fp(vel), len(floats), names, ptrs,
                            iteration, dt, voxelSize, C.byref(params), int(bool(hasCollision)), _stream(stream)))


def AdvectIndexGrid(data: GridIndexedData, dt: float, voxelSize: float, stream=None) -> None:
    vec = data.getBlocksOfType(VEC3F)
    if len(vec) != 1:
        raise HnsError(-2, "Expected exactly one Vec3f block (velocity)")
    floats = data.getBlocksOfType(FLOAT)
    if not floats:
        raise HnsError(-2, "No float blocks found")
    ptrs = (c_f32p * len(floats))(*[_fp(data.pValues(FLOAT, s)) for s in floats])
    n = data.size()
    check(_lib.lib().hns_advect_index_grid(_ip(data.pCoords()) if n else None, n, _fp(data.pValues(VEC3F, vec[0])), len(floats), ptrs, dt,
                                           voxelSize, _stream(stream)))


def AdvectIndexGridVelocity(data: GridIndexedData, dt: float, voxelSize: float, stream=None) -> None:
    vec = data.getBlocksOfType(VEC3F)
    if len(vec) != 1:
        raise HnsError(-2, "Expected exactly one Vec3f block (velocity)")
    n = data.size()
    check(_lib.lib().hns_advect_index_grid_velocity(_ip(data.pCoords()) if n else None, n, _fp(data.pValues(VEC3F, vec[0])), dt, voxelSize,
                                                    _stream(stream)))


def ProjectNonDivergent(data: GridIndexedData, iterations: int, voxelSize: float, stream=None) -> None:
    vec = data.getBlocksOfType(VEC3F)
    if len(vec) != 1:
        raise HnsError(-2, "Expected exactly one Vec3f block (velocity)")
    n = data.size()
    check(_lib.lib().hns_project_non_divergent(_ip(data.pCoords()) if n else None, n, _fp(data.pValues(VEC3F, vec[0])), int(iterations),
                                               voxelSize, _stream(stream)))


def Divergence(data: GridIndexedData, voxelSize: float, stream=None) -> None:
    vec = data.getBlocksOfType(VEC3F)
    if len(vec) != 1:
        raise HnsError(-2, "Expected exactly one Vec3f block (velocity)")
    div = data.pValues(FLOAT, "divergence")
    n = data.size()
    check(_lib.lib().hns_divergence(_ip(data.pCoords()) if n else None, n, _fp(data.pValues(VEC3F, vec[0])),
                                    _fp(div) if div is not None else None, voxelSize, _stream(stream)))


def CombustionKernel(data: GridIndexedData, handle: IndexGridHandle, dt: float, voxelSize: float, stream=None) -> None:
    vec = data.getBlocksOfType(VEC3F)
    if len(vec) != 1:
        raise HnsError(-2, "Expected exactly one Vec3f block (velocity)")
    check(_lib.lib().hns_combustion_kernel(handle._h, _fp(data.pValues(VEC3F, vec[0])), data.size(), dt, voxelSize, _stream(stream)))


def build_domain(vel_origins, vel_masks=None, padding: int = 0, sdf_origins=None) -> np.ndarray:
    """The simulation domain's leaf origins (NanoVDB order), built on the device: leaf nodes of the velocity grid, leaves its active
    voxels reach when dilated `padding` times (26-neighbourhood), leaf nodes of the collision SDF grid -- what
    SOP_HNanoSolverVerb::cook computes with OpenVDB every cook (src/SOP/HNanoSolver/SOP_HNanoSolver.cpp:188-199).
    vel_masks: uint64 (n, 8) voxel masks of the velocity leaves (word x, bit y*8+z) or None = all voxels active."""
    vo = np.ascontiguousarray(np.asarray(vel_origins, np.int32).reshape(-1, 3))
    vm = None if vel_masks is None else np.ascontiguousarray(np.asarray(vel_masks, np.uint64).reshape(-1, 8))
    assert vm is None or vm.shape[0] == vo.shape[0]
    so = np.zeros((0, 3), np.int32) if sdf_origins is None else np.ascontiguousarray(np.asarray(sdf_origins, np.int32).reshape(-1, 3))
    h = C.c_void_p()
    L = _lib.lib()
    check(L.hns_domain_build(_ip(vo) if len(vo) else None, vm.ctypes.data_as(c_u64p) if vm is not None and len(vo) else None, vo.shape[0], int(padding),
                             _ip(so) if len(so) else None, so.shape[0], C.byref(h)))
    try:
        out = np.empty((L.hns_domain_num_leaves(h), 3), np.int32)
        check(L.hns_domain_origins(h, _ip(out) if len(out) else None))
    finally:
        L.hns_domain_destroy(h)
    return out


class Multigrid:
    """Coarse-level hierarchy over an index grid (hns_mg_create): level k+1 has cells twice the size, 2x2x2 leaves -> one leaf."""

    def __init__(self, grid: IndexGridHandle, max_levels: int = 0):
        self.grid = grid
        h = C.c_void_p()
        check(_lib.lib().hns_mg_create(grid._h, max_levels, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().hns_mg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_levels(self) -> int:
        return int(_lib.lib().hns_mg_num_levels(self._h))

    def level_leaves(self, k: int) -> int:
        return int(_lib.lib().hns_mg_level_leaves(self._h, k))

    def level_cells(self, k: int) -> int:
        return int(_lib.lib().hns_mg_level_cells(self._h, k))

    def set_coarsest_iterations(self, iterations: int):
        check(_lib.lib().hns_mg_set_coarsest_iterations(self._h, iterations))


class Source:
    """A NanoVDB float or Vec3f grid (uint8 host buffer: io.read_nvdb, io.grid_from_sidecar) on the current device, to be added to
    resident fields with Simulation.add_source: openvdb::tools::compSum as the SOP does every cook (SOP_HNanoSolver.cpp:159-181),
    bit for bit io.comp_sum. The buffer is validated on the host; a malformed one raises before anything reaches the GPU."""

    def __init__(self, buffer: np.ndarray):
        buf = np.ascontiguousarray(buffer, np.uint8)
        h = C.c_void_p()
        check(_lib.lib().hns_source_create(buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().hns_source_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def components(self) -> int:
        """1 (float grid) or 3 (Vec3f grid)"""
        return int(_lib.lib().hns_source_components(self._h))

    @property
    def num_leaves(self) -> int:
        return int(_lib.lib().hns_source_num_leaves(self._h))

    def leaves_outside(self, grid: IndexGridHandle) -> int:
        """source leaves whose origin is not a leaf of `grid`: their values reach no field (the domain stays fixed)"""
        n = C.c_uint64()
        check(_lib.lib().hns_source_leaves_outside(self._h, grid._h, C.byref(n)))
        return int(n.value)


class ValueGrid:
    """A NanoVDB float or Vec3f grid in device memory, written by Simulation.export_grid (include/hns_b200.h, export). Every export
    into it replaces the grid; its device block only grows, so a per-frame export into one ValueGrid allocates nothing in steady state."""

    def __init__(self):
        h = C.c_void_p()
        check(_lib.lib().hns_value_grid_create(C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().hns_value_grid_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def nbytes(self) -> int:
        return int(_lib.lib().hns_value_grid_bytes(self._h))

    @property
    def num_leaves(self) -> int:
        return int(_lib.lib().hns_value_grid_num_leaves(self._h))

    @property
    def device_ptr(self) -> int:
        """device address of the grid (GridData first); 0 before the first export"""
        return int(_lib.lib().hns_value_grid_device_ptr(self._h) or 0)

    def download(self) -> np.ndarray:
        """the grid as a uint8 host buffer (io.write_nvdb, io.sidecar_from_grid and Source take it)"""
        out = np.empty(self.nbytes, np.uint8)
        check(_lib.lib().hns_value_grid_download(self._h, out.ctypes.data_as(C.c_void_p), out.size))
        return out


class Simulation:
    """Device-resident state of one simulation: velocity + n_scalars float fields on an index grid."""

    AUX_DIVERGENCE, AUX_PRESSURE, AUX_ADVECTED = 0, 1, 2
    FLAG_FORWARD_ONLY = 2  # every pressure half-sweep walks the leaves front to back (default: black sweeps run back to front)

    def __init__(self, grid: IndexGridHandle, n_scalars: int):
        self.grid = grid
        self.n = grid.num_voxels
        self.n_scalars = n_scalars
        h = C.c_void_p()
        check(_lib.lib().hns_state_create(grid._h, n_scalars, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().hns_state_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, velocity: np.ndarray | None = None, scalars=()):
        if velocity is not None:
            v = np.ascontiguousarray(velocity, np.float32).reshape(-1, 3)
            assert v.shape[0] == self.n
            check(_lib.lib().hns_state_upload_velocity(self._h, _fp(v)))
        for i, a in enumerate(scalars):
            a = np.ascontiguousarray(a, np.float32).reshape(-1)
            assert a.shape[0] == self.n
            check(_lib.lib().hns_state_upload_scalar(self._h, i, _fp(a)))

    def add_source(self, target, source: Source, stream=None):
        """compSum of `source` into the velocity (target "velocity", a Vec3f source) or into scalar `target` (an int, a float source):
        every voxel of the grid gets value + the source's value there, +0.0 where the source has no leaf. Asynchronous on `stream`."""
        if isinstance(target, str):
            if target != "velocity":
                raise ValueError(f'target must be "velocity" or a scalar index, not {target!r}')
            check(_lib.lib().hns_state_add_source_velocity(self._h, source._h, _stream(stream)))
        else:
            check(_lib.lib().hns_state_add_source_scalar(self._h, int(target), source._h, _stream(stream)))

    def export_grid(self, target, name: str, tolerance: float = -1.0, out: ValueGrid | None = None, stream=None) -> ValueGrid:
        """writeIndexGrid on the device: the velocity (target "velocity") as a Vec3f grid of class Staggered or scalar `target` (an int)
        as a float grid of class FogVolume, into `out` (a new ValueGrid when None), which is returned. tolerance < 0: every leaf, every
        voxel active; tolerance >= 0: only voxels with !(|v| <= tolerance) are active and leaves without one are left out. Ordered after
        earlier work on `stream`; returns when the grid is complete. The state is not changed."""
        vg = ValueGrid() if out is None else out
        if isinstance(target, str):
            if target != "velocity":
                raise ValueError(f'target must be "velocity" or a scalar index, not {target!r}')
            check(_lib.lib().hns_state_export_velocity(self._h, float(tolerance), name.encode(), vg._h, _stream(stream)))
        else:
            check(_lib.lib().hns_state_export_scalar(self._h, int(target), float(tolerance), name.encode(), vg._h, _stream(stream)))
        return vg

    def redomain(self, tolerance: float, padding: int, sources=(), sdf_origins=None, stream=None) -> "Simulation":
        """The SOP's domain step for a resident state: a new Simulation on a new grid whose leaves are the velocity's leaf topology at
        `tolerance` (as export_grid("velocity", tolerance) writes it; tolerance < 0: every leaf, every voxel) united with the leaves of
        `sources` (Source objects), dilated by `padding` voxels, plus the collider's leaf origins `sdf_origins`. The velocity and every
        scalar are carried over bit for bit where the old grid has the leaf; new leaves hold 0, or bytes 0x01 in the collision SDF.
        Combustion, vorticity and the collision scalar are carried over, a multigrid solver is not (the new state solves red-black).
        Work on `stream` is finished first; `stream` is synchronised before returning, so this object may be dropped at once."""
        L = _lib.lib()
        so = np.zeros((0, 3), np.int32) if sdf_origins is None else np.ascontiguousarray(np.asarray(sdf_origins, np.int32).reshape(-1, 3))
        srcs = (C.c_void_p * max(1, len(sources)))(*[s._h.value for s in sources])
        self.sync(stream)
        d = C.c_void_p()
        check(L.hns_state_domain_build(self._h, float(tolerance), int(padding), len(sources), srcs, _ip(so) if len(so) else None, so.shape[0],
                                       C.byref(d)))
        try:
            g = C.c_void_p()
            check(L.hns_domain_create_grid(d, L.hns_grid_voxel_size(self.grid._h), C.byref(g)))
        finally:
            L.hns_domain_destroy(d)
        grid = IndexGridHandle(g.value)
        h = C.c_void_p()
        check(L.hns_state_create_remapped(self._h, grid._h, _stream(stream), C.byref(h)))
        out = Simulation.__new__(Simulation)
        out.grid, out.n, out.n_scalars, out._h = grid, grid.num_voxels, self.n_scalars, h
        out.sync(stream)
        return out

    def velocity(self) -> np.ndarray:
        out = np.empty((self.n, 3), np.float32)
        check(_lib.lib().hns_state_download_velocity(self._h, _fp(out)))
        return out

    def scalar(self, i: int) -> np.ndarray:
        out = np.empty(self.n, np.float32)
        check(_lib.lib().hns_state_download_scalar(self._h, i, _fp(out)))
        return out

    def aux(self, which: int) -> np.ndarray:
        out = np.empty((self.n, 3) if which == self.AUX_ADVECTED else self.n, np.float32)
        check(_lib.lib().hns_state_download_aux(self._h, which, _fp(out)))
        return out

    def set_combustion(self, enabled: bool, fuel=0, waste=0, temperature=0, flame=0, params: CombustionParams | None = None):
        check(_lib.lib().hns_state_set_combustion(self._h, int(enabled), fuel, waste, temperature, flame,
                                                  C.byref(params) if params is not None else None))

    def step(self, iterations: int, dt: float, flags: int = 0, stream=None):
        check(_lib.lib().hns_state_step(self._h, iterations, dt, flags, _stream(stream)))

    def advect_velocity(self, dt, stream=None):
        check(_lib.lib().hns_state_advect_velocity(self._h, dt, _stream(stream)))

    def set_collision(self, sdf_scalar_index: int = -1):
        """scalar `sdf_scalar_index` becomes the collision SDF of the hasCollision path (-1: off)"""
        check(_lib.lib().hns_state_set_collision(self._h, int(sdf_scalar_index)))

    def enforce_collision(self, stream=None):
        """enforceCollisionBoundaries (reference Kernel.cu:77-116) on the velocity"""
        check(_lib.lib().hns_state_enforce_collision(self._h, _stream(stream)))

    def vorticity_confinement(self, dt, scale, factor_scale, stream=None):
        """vorticityConfinement (reference Kernel.cu:969-1025) on the advected velocity, out of place"""
        check(_lib.lib().hns_state_vorticity_confinement(self._h, dt, scale, factor_scale, _stream(stream)))

    def divergence(self, of_advected=True, stream=None):
        check(_lib.lib().hns_state_divergence(self._h, int(of_advected), _stream(stream)))

    def pressure_solve(self, iterations, omega, flags=0, stream=None):
        check(_lib.lib().hns_state_pressure_solve(self._h, iterations, omega, flags, _stream(stream)))

    def pressure_init(self, stream=None):
        check(_lib.lib().hns_state_pressure_init(self._h, _stream(stream)))

    def pressure_half_sweep(self, color: int, omega: float, reverse: bool = False, stream=None):
        check(_lib.lib().hns_state_pressure_half_sweep(self._h, color, omega, int(reverse), _stream(stream)))

    def combustion_buoyancy(self, dt: float, stream=None):
        check(_lib.lib().hns_state_combustion_buoyancy(self._h, dt, _stream(stream)))

    def subtract_gradient(self, from_advected=True, stream=None):
        check(_lib.lib().hns_state_subtract_gradient(self._h, int(from_advected), _stream(stream)))

    def advect_scalars(self, dt, sampler_semantics=0, stream=None):
        check(_lib.lib().hns_state_advect_scalars(self._h, dt, sampler_semantics, _stream(stream)))

    def sync(self, stream=None):
        check(_lib.lib().hns_state_sync(self._h, _stream(stream)))

    # --- device-side norms and the multigrid solve (the reference declares compute_residual / restrict / prolongate but never
    #     defines them, src/Cuda/Kernels.cuh:38-49) ------------------------------------------------------------------------
    def residual_sums(self, stream=None) -> tuple[float, float]:
        """(sum (div - L p)^2, sum div^2) of the current pressure and divergence, fp64 on the device"""
        out = (C.c_double * 2)()
        check(_lib.lib().hns_state_residual_sums(self._h, out, _stream(stream)))
        return float(out[0]), float(out[1])

    def relative_residual(self, stream=None) -> float:
        a, b = self.residual_sums(stream)
        return float(np.sqrt(a / b)) if b > 0 else 0.0

    def divergence_sum_squares(self, of_advected=False, stream=None) -> float:
        """sum of squares of the divergence of the (advected) velocity; overwrites the state's divergence field"""
        out = C.c_double()
        check(_lib.lib().hns_state_divergence_sum_squares(self._h, int(of_advected), C.byref(out), _stream(stream)))
        return float(out.value)

    def pressure_solve_mg(self, mg: "Multigrid", max_cycles: int, rel_tol: float = 0.0, nu_pre: int = 2, nu_post: int = 2,
                          omega_smooth: float = 1.15, stream=None) -> tuple[int, float]:
        """p = 0, then V-cycles until the relative residual <= rel_tol (or exactly max_cycles when rel_tol <= 0); (cycles, residual or -1)"""
        check(_lib.lib().hns_state_pressure_solve_mg(self._h, mg._h, max_cycles, rel_tol, nu_pre, nu_post, omega_smooth, _stream(stream)))
        return int(_lib.lib().hns_mg_last_cycles(mg._h)), float(_lib.lib().hns_mg_last_relative_residual(mg._h))

    def set_pressure_solver(self, mg: "Multigrid | None", cycles: int = 2, nu_pre: int = 2, nu_post: int = 2, omega_smooth: float = 1.15):
        """step()/time_frames() then run `cycles` V-cycles instead of the reference's red-black SOR sweeps (None switches back)"""
        check(_lib.lib().hns_state_set_pressure_solver(self._h, mg._h if mg is not None else None, cycles, nu_pre, nu_post, omega_smooth))
        self._mg = mg

    def time_frames(self, frames: int, iterations: int, dt: float, flags: int = 0, stream=None) -> tuple[float, float]:
        """(total ms, ms inside the pressure solve) over `frames` identical frames, CUDA events on the launch stream."""
        a, b = C.c_float(), C.c_float()
        check(_lib.lib().hns_state_time_frames(self._h, frames, iterations, dt, flags, _stream(stream), C.byref(a), C.byref(b)))
        return a.value, b.value

    def field_ptr(self, field: int) -> int:
        return _lib.lib().hns_state_field_device_ptr(self._h, field) or 0

    def pack_leaves(self, field: int, ids_dev_ptr: int, n_ids: int, dst_dev_ptr: int, stream=None):
        check(_lib.lib().hns_state_pack_leaves(self._h, field, C.c_void_p(ids_dev_ptr), n_ids, C.c_void_p(dst_dev_ptr), _stream(stream)))

    def unpack_leaves(self, field: int, ids_dev_ptr: int, n_ids: int, src_dev_ptr: int, stream=None):
        check(_lib.lib().hns_state_unpack_leaves(self._h, field, C.c_void_p(ids_dev_ptr), n_ids, C.c_void_p(src_dev_ptr), _stream(stream)))
