"""Synthetic sparse smoke domains for the BASELINE.json configs (SURVEY.md §8d). Pure numpy, deterministic.

Every generator returns a `Workload`: leaf origins in NanoVDB order, the dense-leaf coords exactly as
HNS::IndexGridBuilder::build emits them (reference src/Utils/GridBuilder.hpp:156-166), a collocated velocity field
float[N][3] and S scalar fields float[N]. Velocities are specified as per-step displacement in voxels
(d = u*dt/h) and clamped to |d| <= cfl_max per component so that the benchmark inputs have a stated CFL bound
(the reference itself has none).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

VOXEL_SIZE = 0.1
DT = 1.0 / 24.0


@dataclass
class Workload:
    name: str
    origins: np.ndarray            # int32 [L,3], NanoVDB order
    coords: np.ndarray | None      # int32 [N,3] (None when built with with_coords=False)
    velocity: np.ndarray           # float32 [N,3]
    scalars: list[np.ndarray]      # S x float32 [N]
    scalar_names: list[str]
    voxel_size: float = VOXEL_SIZE
    dt: float = DT
    iterations: int = 40
    meta: dict = field(default_factory=dict)

    @property
    def num_leaves(self) -> int:
        return int(self.origins.shape[0])

    @property
    def num_voxels(self) -> int:
        return self.num_leaves * 512


# --------------------------------------------------------------------------------------------------------------
# ordering / coords
# --------------------------------------------------------------------------------------------------------------
def nanovdb_order(origins: np.ndarray) -> np.ndarray:
    """argsort of leaf origins in NanoVDB order: root tile (signed lexicographic x,y,z of the 4096^3 tile), then the upper
    offset (x,y,z of the 128^3 block inside the tile), then the lower offset (x,y,z of the 8^3 leaf inside the block).
    reference: externals/nanovdb/tools/cuda/PointsToGrid.cuh:596-602, 640-645."""
    o = origins.astype(np.int64)
    tile = [(o[:, d] + (1 << 31)) >> 12 for d in range(3)]
    up = [(o[:, d] & 4095) >> 7 for d in range(3)]
    lo = [(o[:, d] & 127) >> 3 for d in range(3)]
    keys = (lo[2], lo[1], lo[0], up[2], up[1], up[0], tile[2], tile[1], tile[0])  # np.lexsort: last key is primary
    return np.lexsort(keys)


_LOCAL = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(8), indexing="ij"), -1).reshape(512, 3).astype(np.int32)


def dense_coords(origins: np.ndarray) -> np.ndarray:
    """coords[l*512 + (x<<6|y<<3|z)] = origin[l] + (x,y,z)  (leaf.offsetToGlobalCoord order)."""
    return (origins[:, None, :].astype(np.int32) + _LOCAL[None, :, :]).reshape(-1, 3)


def dilate_leaves(mask: np.ndarray, n: int = 1) -> np.ndarray:
    """26-neighbourhood dilation of a boolean leaf-lattice mask."""
    m = mask.copy()
    for _ in range(n):
        p = np.pad(m, 1)
        out = np.zeros_like(m)
        for dx in range(3):
            for dy in range(3):
                for dz in range(3):
                    out |= p[dx:dx + m.shape[0], dy:dy + m.shape[1], dz:dz + m.shape[2]]
        m = out
    return m


def origins_from_mask(mask: np.ndarray, offset=(0, 0, 0)) -> np.ndarray:
    o = (np.argwhere(mask).astype(np.int32) * 8) + np.asarray(offset, np.int32)
    return np.ascontiguousarray(o[nanovdb_order(o)])


# --------------------------------------------------------------------------------------------------------------
# hash noise: splitmix64 of (seed, i, j, k, channel) -> uniform [0,1)
# --------------------------------------------------------------------------------------------------------------
def _splitmix64(x: np.ndarray) -> np.ndarray:
    x = (x + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def hash_noise(seed: int, ijk: np.ndarray, channel: int) -> np.ndarray:
    with np.errstate(over="ignore"):
        h = np.full(ijk.shape[0], np.uint64(seed) * np.uint64(0x2545F4914F6CDD1D) + np.uint64(channel), np.uint64)
        for d in range(3):
            h = _splitmix64(h ^ ijk[:, d].astype(np.int64).astype(np.uint64))
    return ((h >> np.uint64(40)).astype(np.float64) / float(1 << 24)).astype(np.float32)


def smooth_lattice_noise(shape, cells, seed: int) -> np.ndarray:
    """Trilinear value noise on a lattice of `shape`, `cells` random cells per axis (an int, or one count per axis)."""
    rng = np.random.default_rng(seed)
    cells = (cells,) * 3 if np.isscalar(cells) else tuple(cells)
    g = rng.random(tuple(c + 1 for c in cells))
    ax = [np.linspace(0, c, s, endpoint=False) for c, s in zip(cells, shape)]
    i = [np.floor(a).astype(int) for a in ax]
    f = [a - ii for a, ii in zip(ax, i)]
    f = [t * t * (3 - 2 * t) for t in f]
    out = np.zeros(shape)
    for dx in (0, 1):
        wx = (f[0] if dx else 1 - f[0])[:, None, None]
        for dy in (0, 1):
            wy = (f[1] if dy else 1 - f[1])[None, :, None]
            for dz in (0, 1):
                wz = (f[2] if dz else 1 - f[2])[None, None, :]
                out += wx * wy * wz * g[np.ix_(i[0] + dx, i[1] + dy, i[2] + dz)]
    return out


def _to_velocity(disp: np.ndarray, h: float, dt: float, cfl_max: float) -> np.ndarray:
    d = np.clip(disp, -cfl_max, cfl_max).astype(np.float32)
    return (d * np.float32(h / dt)).astype(np.float32)


def _finish(name, origins, vel_fn, scalar_fns, scalar_names, iterations, seed, with_coords=True, cfl_max=2.5, chunk_leaves=8192, meta=None):
    """Evaluates the analytic fields leaf-chunk by leaf-chunk to bound temporary memory."""
    L = origins.shape[0]
    N = L * 512
    vel = np.empty((N, 3), np.float32)
    scal = [np.empty(N, np.float32) for _ in scalar_fns]
    coords = np.empty((N, 3), np.int32) if with_coords else None
    for a in range(0, L, chunk_leaves):
        b = min(L, a + chunk_leaves)
        c = dense_coords(origins[a:b])
        if with_coords:
            coords[a * 512:b * 512] = c
        vel[a * 512:b * 512] = _to_velocity(vel_fn(c, seed), VOXEL_SIZE, DT, cfl_max)
        for s, fn in enumerate(scalar_fns):
            scal[s][a * 512:b * 512] = fn(c, seed)
    for s in scal:
        if N:
            s[0] = 0.0  # element 0 doubles as the "inactive" value of advect_scalars (reference Kernel.cu:192,225)
    return Workload(name, origins, coords, vel, scal, list(scalar_names), VOXEL_SIZE, DT, iterations, dict(meta or {}, seed=seed, cfl_max=cfl_max))


# --------------------------------------------------------------------------------------------------------------
# the five configs
# --------------------------------------------------------------------------------------------------------------
def smoke_sphere(R: int = 64, seed: int = 1, with_coords=True) -> Workload:
    """C1: 64^3 smoke sphere: leaves intersecting the ball of radius 0.4375 R around the centre, dilated by one leaf."""
    n = R // 8
    c, rad = R / 2.0, 0.4375 * R
    g = (np.arange(n) * 8)
    lo = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).astype(np.float64)
    nearest = np.clip(c, lo, lo + 7)
    mask = ((nearest - c) ** 2).sum(-1) <= rad * rad
    origins = origins_from_mask(dilate_leaves(mask, 1) if n > 2 else mask)

    def vel(cd, seed):
        x, y = cd[:, 0].astype(np.float32), cd[:, 1].astype(np.float32)
        d = np.zeros((cd.shape[0], 3), np.float32)
        d[:, 0] = -0.02 * (y - c)
        d[:, 1] = 0.02 * (x - c)
        for ch in range(3):
            d[:, ch] += 0.02 * (hash_noise(seed, cd, ch) - 0.5)
        return d

    def density(cd, seed):
        r = np.sqrt(((cd.astype(np.float32) - np.float32(c)) ** 2).sum(-1))
        return np.clip(1.0 - r / np.float32(rad), 0.0, 1.0).astype(np.float32)

    return _finish(f"sphere{R}", origins, vel, [density], ["density"], 40, seed, with_coords, meta=dict(R=R))


def smoke_plume(R: int = 128, seed: int = 2, with_coords=True, iterations: int = 40) -> Workload:
    """C2 / C3: plume around the axis x = z = R/2: radius (8 + 0.25 y) * R/128 for y in [R/16, 15R/16], dilated by one leaf."""
    n = R // 8
    sc = R / 128.0
    g = (np.arange(n) * 8)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    cx = R / 2.0
    # leaf box vs cone: test the closest point of the leaf's xz footprint to the axis at the leaf's top y (widest radius)
    nx = np.clip(cx, X, X + 7) - cx
    nz = np.clip(cx, Z, Z + 7) - cx
    ytop = np.clip(Y + 7, R / 16.0, 15 * R / 16.0)
    rad = (8 * sc + 0.25 * ytop)
    mask = (nx * nx + nz * nz <= rad * rad) & (Y + 7 >= R / 16.0) & (Y <= 15 * R / 16.0)
    origins = origins_from_mask(dilate_leaves(mask, 1))

    def radial(cd):
        x, y, z = (cd[:, d].astype(np.float32) for d in range(3))
        r2 = (x - np.float32(cx)) ** 2 + (z - np.float32(cx)) ** 2
        w = (np.float32(8 * sc) + np.float32(0.25) * y)
        return r2, w, y

    def vel(cd, seed):
        r2, w, y = radial(cd)
        d = np.zeros((cd.shape[0], 3), np.float32)
        d[:, 1] = 1.5 * np.exp(-r2 / (w * w))
        for ch in range(3):
            d[:, ch] += 0.3 * (hash_noise(seed, cd, ch) - 0.5)
        return d

    def density(cd, seed):
        r2, w, y = radial(cd)
        return (np.exp(-r2 / (w * w)) * np.clip(1.0 - y / np.float32(R), 0, 1)).astype(np.float32)

    def temperature(cd, seed):
        r2, w, y = radial(cd)
        return (np.exp(-r2 / (0.5 * w * w)) * np.clip(1.0 - y / np.float32(R), 0, 1)).astype(np.float32)

    return _finish(f"plume{R}", origins, vel, [density, temperature], ["density", "temperature"], iterations, seed, with_coords,
                   meta=dict(R=R))


def _swirl_fields(R, cells=8):
    def vel(cd, seed):
        p = cd.astype(np.float32) * np.float32(2 * np.pi / R)
        d = np.empty((cd.shape[0], 3), np.float32)
        d[:, 0] = 1.2 * np.sin(p[:, 1]) * np.cos(p[:, 2])
        d[:, 1] = 1.2 * np.sin(p[:, 2]) * np.cos(p[:, 0]) + 0.8
        d[:, 2] = 1.2 * np.sin(p[:, 0]) * np.cos(p[:, 1])
        for ch in range(3):
            d[:, ch] += 0.3 * (hash_noise(seed, cd, ch) - 0.5)
        return d

    def density(cd, seed):
        p = cd.astype(np.float32) * np.float32(4 * np.pi / R)
        return (0.5 + 0.5 * np.sin(p[:, 0]) * np.sin(p[:, 1]) * np.sin(p[:, 2])).astype(np.float32)

    def temperature(cd, seed):
        p = cd.astype(np.float32) * np.float32(2 * np.pi / R)
        return (0.5 + 0.5 * np.cos(p[:, 0] + p[:, 1]) * np.cos(p[:, 2])).astype(np.float32)

    return vel, density, temperature


def sparse_smoke(R: int = 512, fill: float = 0.30, seed: int = 4, with_coords=True, x_range=None) -> Workload:
    """C4: R^3-bounded blobby sparse smoke: a leaf is kept iff smooth lattice noise exceeds the (1 - fill) quantile, so that
    `fill` of the (R/8)^3 leaves are active. x_range = (lo, hi) in leaf units restricts generation to a slab (sharded runs)."""
    n = R // 8
    noise = smooth_lattice_noise((n, n, n), max(2, n // 8), seed)
    tau = np.quantile(noise, 1.0 - fill)
    mask = noise > tau
    if x_range is not None:
        keep = np.zeros_like(mask)
        keep[x_range[0]:x_range[1]] = True
        mask &= keep
    origins = origins_from_mask(mask)
    vel, density, temperature = _swirl_fields(R)
    return _finish(f"sparse{R}", origins, vel, [density, temperature], ["density", "temperature"], 40, seed, with_coords,
                   meta=dict(R=R, fill=fill, active_leaf_fraction=float(mask.mean())))


def narrow_band_origins(R: int = 1024, target_voxels: float = 2.0e8, x_range=None):
    """leaf origins (NanoVDB order) of the C5 shell and its half width in voxels"""
    n = R // 8
    c = R / 2.0
    g = np.arange(n) * 8 + 3.5
    d2 = ((g - c) ** 2)
    dist = np.sqrt(d2[:, None, None] + d2[None, :, None] + d2[None, None, :])
    band = np.abs(dist - 0.39 * R)
    w = np.quantile(band, min(1.0, target_voxels / 512.0 / n ** 3))
    mask = band <= w
    if x_range is not None:
        keep = np.zeros_like(mask)
        keep[x_range[0]:x_range[1]] = True
        mask &= keep
    return origins_from_mask(mask), float(w)


def narrow_band(R: int = 1024, target_voxels: float = 2.0e8, seed: int = 5, with_coords=False, x_range=None) -> Workload:
    """C5: R^3-bounded spherical shell | |x - c| - 0.39 R | < w with w chosen for ~target_voxels active voxels."""
    origins, w = narrow_band_origins(R, target_voxels, x_range)
    vel, density, temperature = _swirl_fields(R)
    return _finish(f"band{R}", origins, vel, [density, temperature], ["density", "temperature"], 40, seed, with_coords,
                   meta=dict(R=R, half_width_voxels=float(w)))


def random_leaves(n_leaves: int = 40, extent: int = 6, seed: int = 0, offset=(0, 0, 0), with_coords=True, cfl: float = 1.5, S: int = 2) -> Workload:
    """Small random leaf soup (many missing neighbours, optional negative / multi-tile offsets) for edge-case parity tests."""
    rng = np.random.default_rng(seed)
    cells = rng.integers(0, extent, size=(n_leaves * 3, 3))
    cells = np.unique(cells, axis=0)
    rng.shuffle(cells)
    cells = cells[:n_leaves]
    o = (cells * 8 + np.asarray(offset)).astype(np.int32)
    origins = np.ascontiguousarray(o[nanovdb_order(o)])

    def vel(cd, seed):
        return np.stack([2 * cfl * (hash_noise(seed, cd, ch) - 0.5) for ch in range(3)], -1)

    fns = [lambda cd, seed, k=k: hash_noise(seed, cd, 10 + k) for k in range(S)]
    return _finish(f"random{n_leaves}", origins, vel, fns, [f"s{k}" for k in range(S)], 8, seed, with_coords, cfl_max=cfl)


WORKLOADS = {
    "c1": lambda **kw: smoke_sphere(64, 1, **kw),
    "c2": lambda **kw: smoke_plume(128, 2, **kw),
    "c3": lambda **kw: smoke_plume(256, 3, **kw),
    "c4": lambda **kw: sparse_smoke(512, 0.30, 4, **kw),
    "c5": lambda **kw: narrow_band(1024, 2.0e8, 5, **kw),
}


def combustion_fields(w: Workload, seed: int = 123, chunk_leaves: int = 8192) -> dict:
    """fuel / waste / temperature / flame for the all-in-one frame (reference src/Cuda/HNanoSolver.cu:193): hash noise,
    fuel present in ~40 % of the voxels. Returned in the insertion order the frame uses."""
    L, N = w.num_leaves, w.num_voxels
    out = {k: np.empty(N, np.float32) for k in ("fuel", "waste", "temperature", "flame")}
    for a in range(0, L, chunk_leaves):
        b = min(L, a + chunk_leaves)
        c = dense_coords(w.origins[a:b])
        sl = slice(a * 512, b * 512)
        out["fuel"][sl] = hash_noise(seed, c, 20) * (hash_noise(seed, c, 21) < 0.4)
        out["waste"][sl] = 0.3 * hash_noise(seed, c, 22)
        out["temperature"][sl] = hash_noise(seed, c, 23)
        out["flame"][sl] = 0.2 * hash_noise(seed, c, 24)
    for a in out.values():
        if N:
            a[0] = 0.0
    return out


def emitter(origins: np.ndarray, fraction: float = 0.05, n_outside: int = 4, speed: float = 1.0, seed: int = 11):
    """A smoke emitter for sourcing (SOP_HNanoSolver.cpp:159-181): the `fraction` of the domain's leaves lowest in y -- the base of a
    plume rising in +y -- plus `n_outside` leaves in another root tile beside the domain, which a fixed domain drops.
    -> (source leaf origins (NanoVDB order), {"density", "temperature", "fuel": float32 (n * 512,), "velocity": float32 (n * 512, 3)});
    the velocity pushes upward at up to `speed`. io.grid_from_sidecar turns each into a NanoVDB grid."""
    o = np.asarray(origins, np.int32).reshape(-1, 3)
    k = min(len(o), max(1, int(round(fraction * len(o))))) if len(o) else 0
    base = o[np.argsort(o[:, 1], kind="stable")[:k]]
    lo = o.min(0) if len(o) else np.zeros(3, np.int32)
    outside = np.array([[lo[0] - 4096 - 8 * i, lo[1], lo[2]] for i in range(n_outside)], np.int32).reshape(-1, 3)
    so = np.concatenate([base, outside])
    so = np.ascontiguousarray(so[nanovdb_order(so)])
    c = dense_coords(so)
    values = {"density": 0.5 * hash_noise(seed, c, 30), "temperature": hash_noise(seed, c, 31), "fuel": 0.8 * hash_noise(seed, c, 32)}
    vel = np.zeros((len(c), 3), np.float32)
    vel[:, 1] = speed * hash_noise(seed, c, 33)
    values["velocity"] = vel
    return so, {name: np.ascontiguousarray(v, np.float32) for name, v in values.items()}
