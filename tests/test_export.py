"""Export of resident fields as NanoVDB grids built on the device (hns_value_grid_*, hns_state_export_*; Simulation.export_grid): the
contract is the host writer hns_sidecar_to_nanovdb (io.grid_from_sidecar) byte for byte -- over every leaf with every voxel active
(tolerance < 0), or over the leaves that keep an active voxel, !(|v| <= tolerance), with those masks (tolerance >= 0)."""
import ctypes as C

import numpy as np
import pytest

import hnanosolver_b200 as H
from hnanosolver_b200 import _lib, dist, synth
from hnanosolver_b200 import io as hio

PARAMS6 = [0.5, 2.0, 1.5, 0.1, 0.0, 1.0]
TINY = np.float32(np.ldexp(1.0, -140))  # a subnormal
EMPTY = {1: 800, 3: 832}                # bytes of a grid without leaves


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ---- host side: no GPU needed ------------------------------------------------------------------------------------------------------
def test_export_refusals_before_touching_cuda():
    L = _lib.lib()
    vg = H.ValueGrid()
    assert vg.nbytes == 0 and vg.num_leaves == 0 and vg.device_ptr == 0 and vg.download().size == 0
    nan = float("nan")
    assert L.hns_state_export_scalar(None, 0, nan, b"density", vg._h, None) == -1
    assert "NaN" in L.hns_last_error().decode()                        # the tolerance is checked first: no state needed to refuse it
    assert L.hns_state_export_velocity(None, nan, b"vel", vg._h, None) == -1
    assert "NaN" in L.hns_last_error().decode()
    assert L.hns_state_export_scalar(None, 0, 0.0, b"density", vg._h, None) == -1
    assert "null" in L.hns_last_error().decode()
    assert L.hns_state_export_velocity(None, -1.0, None, None, None) == -1
    assert L.hns_value_grid_create(None) == -1
    assert L.hns_value_grid_download(None, None, 0) == -1
    vg.close()


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
def _domain():
    """leaves in two root tiles, one of them at negative coordinates"""
    a = synth.random_leaves(40, 5, 3, with_coords=False).origins
    b = synth.random_leaves(20, 4, 4, offset=(-4096 - 64, -32, -8), with_coords=False).origins
    o = np.concatenate([a, b])
    return np.ascontiguousarray(o[synth.nanovdb_order(o)])


def _special(n, rng, comps=1):
    """random values with planted -0.0, +0.0, subnormals, +-inf and NaN"""
    v = (rng.random((n, comps)) - 0.5).astype(np.float32)
    flat = v.reshape(-1)
    k = flat.size
    flat[rng.integers(0, k, k // 8)] = np.float32(-0.0)
    flat[rng.integers(0, k, k // 16)] = np.float32(0.0)
    flat[rng.integers(0, k, k // 16)] = TINY * rng.integers(1, 5, k // 16).astype(np.float32)
    flat[rng.integers(0, k, k // 16)] = -TINY
    flat[rng.integers(0, k, 7)] = np.float32(np.inf)
    flat[rng.integers(0, k, 7)] = np.float32(-np.inf)
    flat[rng.integers(0, k, 7)] = np.float32(np.nan)
    return v if comps == 3 else v.reshape(-1)


def _sparse(domain, rng, comps):
    """a field most of whose leaves carry nothing: all-+-0 leaves, a whole lower node and the whole negative root tile of zeros, a leaf
    whose only nonzero voxel is a NaN, and (Vec3f) voxels with one nonzero component"""
    Lc = len(domain)
    v = _special(Lc * 512, rng, comps).reshape(Lc, 512, -1)
    zero = rng.random(Lc) < 0.4
    zero |= domain[:, 0] < 0                                                   # the negative root tile vanishes
    lower = domain >> 7
    first = lower[0]
    zero |= (lower == first).all(1)                                            # so does the first lower node
    keep_some = np.nonzero(~zero)[0]
    v[zero] = np.where(rng.random(v[zero].shape) < 0.5, np.float32(0.0), np.float32(-0.0))
    nan_leaf = keep_some[0]
    v[nan_leaf] = np.float32(-0.0)
    v[nan_leaf, 77, 0] = np.float32(np.nan)
    if comps == 3:
        one = keep_some[1]
        v[one] = np.float32(0.0)
        v[one, 5, 1] = np.float32(0.5)                                         # y alone
        v[one, 300, 2] = -TINY                                                 # z alone, a subnormal
    return v.reshape(-1, 3) if comps == 3 else v.reshape(-1)


def _masks(values, tol, comps):
    """-> (keep per leaf, masks uint64 (L, 8)) as the export defines them: active iff !(|v| <= tol), any component"""
    v = values.reshape(-1, 512, comps)
    act = ~(np.abs(v) <= np.float32(tol))
    act = act.any(2)
    masks = np.packbits(act.reshape(-1, 8, 64), axis=2, bitorder="little").view(np.uint64).reshape(-1, 8)
    return act.any(1), np.ascontiguousarray(masks)


def _host_pruned(origins, values, tol, comps, h, name):
    keep, masks = _masks(values, tol, comps)
    v = values.reshape(len(origins), 512, -1)[keep].reshape((-1, 3) if comps == 3 else -1)
    return hio.grid_from_sidecar(np.ascontiguousarray(origins[keep]), v, h, name, masks[keep]), keep


def _export(sim, target, name, tol, out=None, stream=None):
    vg = sim.export_grid(target, name, tol, out, stream)
    return vg.download(), vg


@pytest.mark.gpu
def test_whole_domain_export_is_the_host_writer():
    rng = np.random.default_rng(11)
    domain = _domain()
    n = len(domain) * 512
    sim = H.Simulation(H.create_index_grid_from_origins(domain, 0.1), 2)
    vel, s0, s1 = _special(n, rng, 3), _special(n, rng), _special(n, rng)
    sim.upload(vel, [s0, s1])
    long_name = "d" * 300                                                      # truncated to 255 bytes, as by the host writer
    for target, name, want_field in ((0, "density", s0), (1, long_name, s1), ("velocity", "vel", vel)):
        got, vg = _export(sim, target, name, -1.0)
        want = hio.grid_from_sidecar(domain, sim.velocity() if target == "velocity" else sim.scalar(target), 0.1, name)
        assert np.array_equal(got, want), target
        assert vg.nbytes == want.size and vg.num_leaves == len(domain) and vg.device_ptr != 0
        assert np.array_equal(_bits(hio.sidecar_from_grid(got, domain)), _bits(want_field))
    assert hio.grid_info(got)["grid_class"] == hio.GRID_CLASS_STAGGERED
    assert np.isnan(s0).any() and np.isinf(s0).any() and (np.signbit(s0) & (s0 == 0)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("comps", [1, 3])
def test_pruned_export_is_the_host_writer_over_the_kept_leaves(comps):
    rng = np.random.default_rng(12 + comps)
    domain = _domain()
    field = _sparse(domain, rng, comps)
    sim = H.Simulation(H.create_index_grid_from_origins(domain, 0.1), 1)
    sim.upload(field if comps == 3 else None, [] if comps == 3 else [field])
    target = "velocity" if comps == 3 else 0
    vg = H.ValueGrid()
    for tol in (0.0, 0.25, np.inf):
        got, _ = _export(sim, target, "f", tol, vg)
        want, keep = _host_pruned(domain, field, tol, comps, 0.1, "f")
        assert np.array_equal(got, want), tol
        assert vg.num_leaves == int(keep.sum())
        if tol == 0.0:
            assert 0 < keep.sum() < len(domain) and not keep[domain[:, 0] < 0].any()
            assert hio.grid_info(got)["num_leaves"] == keep.sum()
            # round trip: the field again, except that dropped leaves (all +-0) come back as +0.0
            dropped = np.repeat(~keep, 512)
            back = hio.sidecar_from_grid(got, domain)
            expect = field.copy()
            expect[dropped] = np.float32(0.0)
            assert np.array_equal(_bits(back), _bits(expect))
            assert (np.signbit(field[dropped]) & (field[dropped] == 0)).any()
            # Source(download) added to a zeroed state gives 0 + field (NaN stays NaN)
            zero = H.Simulation(sim.grid, 1)
            zero.upload(np.zeros((len(field), 3), np.float32), [np.zeros(len(domain) * 512, np.float32)])
            zero.add_source(target, H.Source(got))
            zero.sync()
            added = zero.velocity() if comps == 3 else zero.scalar(0)
            ref = np.float32(0.0) + expect
            nan = np.isnan(ref)
            assert nan.any() and np.array_equal(np.isnan(added), nan) and np.array_equal(_bits(added[~nan]), _bits(ref[~nan]))
        if tol == np.inf:                                                      # only NaN voxels stay active
            assert vg.num_leaves == int(np.isnan(field.reshape(len(domain), -1)).any(1).sum())
    # everything dropped: the empty grid
    sim.upload(np.zeros((len(domain) * 512, 3), np.float32) * np.float32(-1.0), [np.full(len(domain) * 512, -0.0, np.float32)])
    got, _ = _export(sim, target, "f", 0.0, vg)
    assert got.size == EMPTY[comps] and vg.num_leaves == 0
    none = np.zeros((0, 3), np.int32)
    assert np.array_equal(got, hio.grid_from_sidecar(none, np.zeros((0, 3) if comps == 3 else 0, np.float32), 0.1, "f"))


@pytest.mark.gpu
@pytest.mark.parametrize("comps", [1, 3])
def test_exported_grid_is_read_by_nanovdb(comps, tmp_path):
    from oracle import oracle as O

    if not O.ref_host_available():
        pytest.skip("needs oracle/_ref/libref_host.so, built only from the original project's sources (oracle/Makefile REF)")
    from test_nvdb_io import _refvalue

    L = _refvalue()
    rng = np.random.default_rng(21)
    domain = _domain()
    field = _sparse(domain, rng, comps)
    field[np.isnan(field)] = np.float32(1.0)
    sim = H.Simulation(H.create_index_grid_from_origins(domain, 0.1), 1)
    sim.upload(field if comps == 3 else None, [] if comps == 3 else [field])
    got, _ = _export(sim, "velocity" if comps == 3 else 0, "f", 0.0)
    path = str(tmp_path / "e.nvdb")
    hio.write_nvdb(path, got)
    n = L.refhost_read_nvdb(path.encode(), None, 0)
    back = np.empty(n, np.uint8)
    L.refhost_read_nvdb(path.encode(), back.ctypes.data_as(C.c_void_p), n)
    assert np.array_equal(back, got)
    coords = np.ascontiguousarray(synth.dense_coords(domain), np.int32)
    vals = np.empty((len(coords), comps) if comps == 3 else len(coords), np.float32)
    act = np.empty(len(coords), np.uint8)
    assert L.refhost_query_grid(back.ctypes.data_as(C.c_void_p), coords.ctypes.data_as(C.c_void_p), len(coords), comps,
                                vals.ctypes.data_as(C.c_void_p), act.ctypes.data_as(C.c_void_p)) == 0
    keep, _ = _masks(field, 0.0, comps)
    kept = np.repeat(keep, 512)
    assert np.array_equal(_bits(vals[kept]), _bits(field[kept]))
    want_act = ~(np.abs(field.reshape(len(coords), -1)) <= 0).all(1) if comps == 3 else ~(np.abs(field) <= 0)
    assert np.array_equal(act.astype(bool), want_act)


def _plume_sim(w, fields, sdf):
    grid = H.create_index_grid_from_origins(w.origins, w.voxel_size)
    sim = H.Simulation(grid, len(fields) + 1)
    sim.upload(w.velocity, list(fields.values()) + [sdf])
    sim.set_combustion(True, 1, 2, 3, 4, H.CombustionParams(*PARAMS6))
    sim.set_collision(len(fields))
    return sim


@pytest.mark.gpu
def test_export_after_real_frames_changes_nothing():
    import torch

    w = synth.smoke_plume(128, 2, with_coords=False)
    fields = dict(density=w.scalars[0], **synth.combustion_fields(w))
    c = synth.dense_coords(w.origins).astype(np.float32)
    sdf = (0.05 * (np.sqrt(((c - np.float32(64.0)) ** 2).sum(1)) - 12.0)).astype(np.float32)
    lib = _lib.lib()
    stream = torch.cuda.Stream()
    a, b = _plume_sim(w, fields, sdf), _plume_sim(w, fields, sdf)
    a.step(12, w.dt, stream=stream)
    vg = H.ValueGrid()
    got_v, _ = _export(a, "velocity", "vel", -1.0, vg, stream)                # no sync between the step and the export
    assert np.array_equal(got_v, hio.grid_from_sidecar(w.origins, a.velocity(), w.voxel_size, "vel"))
    size_v = vg.nbytes
    got_d, _ = _export(a, 0, "density", 0.01, vg, stream)                      # the same ValueGrid, a smaller grid
    want_d, keep = _host_pruned(w.origins, a.scalar(0), 0.01, 1, w.voxel_size, "density")
    assert np.array_equal(got_d, want_d) and vg.nbytes == want_d.size < size_v and 0 < keep.sum() < len(keep)
    p0 = lib.hns_packed_advection_launches()
    a.step(12, w.dt, stream=stream)
    a.sync(stream)
    packed_a = lib.hns_packed_advection_launches() - p0
    b.step(12, w.dt)
    p0 = lib.hns_packed_advection_launches()
    b.step(12, w.dt)
    b.sync()
    packed_b = lib.hns_packed_advection_launches() - p0
    assert packed_a == packed_b
    assert np.array_equal(_bits(a.velocity()), _bits(b.velocity()))
    for i in range(len(fields) + 1):
        assert np.array_equal(_bits(a.scalar(i)), _bits(b.scalar(i))), i
    assert np.array_equal(_bits(a.aux(H.Simulation.AUX_PRESSURE)), _bits(b.aux(H.Simulation.AUX_PRESSURE)))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_export_is_the_owned_part_of_the_single_gpu_export(world):
    L = _lib.lib()
    rng = np.random.default_rng(30 + world)
    go = _domain()
    h = 0.1
    dens = _sparse(go, rng, 1)
    vel = _sparse(go, rng, 3)
    single = H.Simulation(H.create_index_grid_from_origins(go, h), 1)
    single.upload(vel, [dens])
    ref = {t: _export(single, t, "f", 0.0)[0] for t in (0, "velocity")}
    parts = {0: [], "velocity": []}
    for rank in range(world):
        plan = dist.make_plan(go, world, rank)
        lo = go[plan.local_ids]
        sim = H.Simulation(H.create_index_grid_from_origins(np.ascontiguousarray(lo), h), 1)
        lv = vel.reshape(len(go), 512, 3)[plan.local_ids].reshape(-1, 3)
        ld = dens.reshape(len(go), 512)[plan.local_ids].reshape(-1)
        sim.upload(lv, [ld])
        owned = np.ascontiguousarray(np.nonzero(plan.owned_local)[0], np.int32)
        d = C.c_void_p()
        _lib.check(L.hns_dist_create(None, rank, world, C.byref(d)))
        try:
            _lib.check(L.hns_dist_set_plan(d, sim._h, 0, None, None, None, None, None, len(owned), owned.ctypes.data_as(_lib.c_i32p)))
            oo = np.ascontiguousarray(lo[owned])
            for t, comps, values in ((0, 1, ld), ("velocity", 3, lv)):
                whole, _ = _export(sim, t, "f", -1.0)
                v = values.reshape(len(lo), 512, -1)[owned].reshape((-1, 3) if comps == 3 else -1)
                assert np.array_equal(whole, hio.grid_from_sidecar(oo, v, h, "f")), (rank, t)
                origins, _ = hio.leaf_topology(whole)
                assert (origins == go[0]).all(1).any() == (rank == 0)          # global leaf 0: a ghost on every other rank
                pruned, _ = _export(sim, t, "f", 0.0)
                assert np.array_equal(pruned, _host_pruned(oo, v, 0.0, comps, h, "f")[0]), (rank, t)
                parts[t].append(pruned)
        finally:
            L.hns_dist_destroy(d)
        del sim
    for t, bufs in parts.items():
        o_ref, m_ref = hio.leaf_topology(ref[t])
        tops = [hio.leaf_topology(b) for b in bufs]
        o_cat = np.concatenate([o for o, _ in tops])
        assert np.array_equal(o_cat, o_ref) and np.array_equal(np.concatenate([m for _, m in tops]), m_ref)
        vals = np.concatenate([hio.sidecar_from_grid(b, o) for b, (o, _) in zip(bufs, tops)])
        assert np.array_equal(_bits(vals), _bits(hio.sidecar_from_grid(ref[t], o_ref)))


@pytest.mark.gpu
def test_export_refusals():
    domain = _domain()
    sim = H.Simulation(H.create_index_grid_from_origins(domain, 0.1), 2)
    L = _lib.lib()
    for target in (-1, 2):
        with pytest.raises(_lib.HnsInvalidArgument):
            sim.export_grid(target, "f")
    for target in (0, "velocity"):
        with pytest.raises(_lib.HnsInvalidArgument):
            sim.export_grid(target, "f", float("nan"))
    with pytest.raises(ValueError):
        sim.export_grid("density", "f")
    vg = H.ValueGrid()
    assert L.hns_state_export_scalar(sim._h, 0, 0.0, None, vg._h, None) == -1
    assert L.hns_state_export_velocity(sim._h, 0.0, b"f", None, None) == -1
    assert vg.nbytes == 0
    import torch

    if torch.cuda.device_count() < 2:
        return
    sim.export_grid(0, "f", out=vg)
    L.hns_set_device(1)
    try:
        other = H.Simulation(H.create_index_grid_from_origins(domain, 0.1), 1)
        with pytest.raises(_lib.HnsInvalidArgument):
            other.export_grid(0, "f", out=vg)
        del other
    finally:
        L.hns_set_device(0)
