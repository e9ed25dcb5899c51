"""NanoVDB file round trip of the index grid (host only; SURVEY.md 8f rank 3): the product's writer / reader against NanoVDB's own
dependency-free file IO (writeUncompressedGrid / readUncompressedGrids in the vendored NanoVDB.h, compiled into
oracle/_ref/libref_host.so) and against itself. No GPU: the grids come from the oracle's CPU emitter and from NanoVDB's host builder."""
import ctypes as C
import os

import numpy as np
import pytest

from hnanosolver_b200 import io as hio
from hnanosolver_b200 import synth
from hnanosolver_b200.grid_data import FLOAT, VEC3F, GridIndexedData
from oracle import oracle as O

needs_refhost = pytest.mark.skipif(not O.ref_host_available(), reason="needs oracle/_ref/libref_host.so, built only from the original project's sources (oracle/Makefile REF)")


def _cases():
    return {"soup": synth.random_leaves(28, 4, 7, offset=(-24, 4096 - 16, -16), cfl=1.8, S=2), "sphere": synth.smoke_sphere(32, 1),
            "single": synth.random_leaves(1, 1, 1, S=1)}


@pytest.fixture(scope="module", params=list(_cases()))
def w(request):
    return _cases()[request.param]


def _refhost():
    L = O.refhost()
    L.refhost_write_nvdb.argtypes = [C.c_char_p, C.c_void_p, C.c_int]
    L.refhost_write_nvdb.restype = C.c_int
    L.refhost_read_nvdb.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64]
    L.refhost_read_nvdb.restype = C.c_uint64
    return L


def test_round_trip_and_leaf_origins(w, tmp_path):
    buf = O.OracleIndex(w.coords).nanovdb_buffer(w.voxel_size)
    path = str(tmp_path / "grid.nvdb")
    hio.write_nvdb(path, buf)
    back = hio.read_nvdb(path)
    assert np.array_equal(back, buf)
    assert os.path.getsize(path) == 16 + 176 + 1 + buf.size          # FileHeader + FileMetaData + empty name + grid
    origins, h = hio.leaf_origins(back)
    assert np.array_equal(origins, w.origins) and h == np.float32(w.voxel_size)
    # a raw dump of the buffer (what GridHandle::write produces since 32.6) is accepted too
    raw = str(tmp_path / "raw.nvdb")
    buf.tofile(raw)
    assert np.array_equal(hio.read_nvdb(raw), buf)


@needs_refhost
def test_writer_matches_nanovdb_byte_for_byte(w, tmp_path):
    buf = O.OracleIndex(w.coords).nanovdb_buffer(w.voxel_size)
    mine, theirs = str(tmp_path / "mine.nvdb"), str(tmp_path / "theirs.nvdb")
    hio.write_nvdb(mine, buf)
    assert _refhost().refhost_write_nvdb(theirs.encode(), buf.ctypes.data_as(C.c_void_p), 0) == 0
    assert open(mine, "rb").read() == open(theirs, "rb").read()


@needs_refhost
def test_nanovdb_reads_what_the_product_writes_and_vice_versa(w, tmp_path):
    R = _refhost()
    # a grid made by NanoVDB's own host builder, written by NanoVDB, read by the product
    g = O.RefHostGrid(w.coords)
    theirs = str(tmp_path / "theirs.nvdb")
    native = g.buffer()
    assert R.refhost_write_nvdb(theirs.encode(), native.ctypes.data_as(C.c_void_p), 0) == 0
    got = hio.read_nvdb(theirs)
    assert np.array_equal(got, native)
    origins, _ = hio.leaf_origins(got)
    assert np.array_equal(origins, w.origins)
    # ... and as a raw dump
    raw = str(tmp_path / "theirs_raw.nvdb")
    assert R.refhost_write_nvdb(raw.encode(), native.ctypes.data_as(C.c_void_p), 1) == 0
    assert np.array_equal(hio.read_nvdb(raw), native)
    # written by the product, read by NanoVDB
    mine = str(tmp_path / "mine.nvdb")
    hio.write_nvdb(mine, native)
    out = np.empty_like(native)
    assert R.refhost_read_nvdb(mine.encode(), out.ctypes.data_as(C.c_void_p), out.size) == native.size
    assert np.array_equal(out, native)


def test_errors(tmp_path):
    from hnanosolver_b200._lib import HnsError

    junk = str(tmp_path / "junk.nvdb")
    open(junk, "wb").write(b"not a nanovdb file" * 50)
    with pytest.raises(HnsError):
        hio.read_nvdb(junk)
    with pytest.raises(HnsError):
        hio.read_nvdb(str(tmp_path / "missing.nvdb"))
    with pytest.raises(HnsError):
        hio.write_nvdb(str(tmp_path / "x.nvdb"), np.zeros(100, np.uint8))
    w = synth.random_leaves(1, 1, 1, S=1)
    buf = O.OracleIndex(w.coords).nanovdb_buffer(w.voxel_size)
    short = str(tmp_path / "short.nvdb")
    hio.write_nvdb(short, buf)
    data = open(short, "rb").read()
    open(short, "wb").write(data[:-100])
    with pytest.raises(HnsError):
        hio.read_nvdb(short)
    wrong = buf.copy()
    wrong[636] = 1                                                   # GridType::Float
    with pytest.raises(HnsError):
        hio.leaf_origins(wrong)


def test_cache_round_trip(w, tmp_path):
    d = GridIndexedData()
    d.allocateCoords(w.num_voxels)
    d.pCoords()[:] = w.coords
    d.addValueBlock(VEC3F, "vel")
    d.pValues(VEC3F, "vel")[:] = w.velocity
    for n, s in zip(w.scalar_names, w.scalars):
        d.addValueBlock(FLOAT, n)
        d.pValues(FLOAT, n)[:] = s
    hio.save_cache(str(tmp_path / "frame0001"), O.OracleIndex(w.coords).nanovdb_buffer(w.voxel_size), d)
    origins, h, back = hio.load_cache(str(tmp_path / "frame0001"))
    assert np.array_equal(origins, w.origins) and h == np.float32(w.voxel_size)
    assert np.array_equal(back.pCoords(), w.coords)
    assert back.getBlocksOfType(FLOAT) == list(w.scalar_names) and back.getBlocksOfType(VEC3F) == ["vel"]
    assert np.array_equal(back.pValues(VEC3F, "vel"), w.velocity)
    for n, s in zip(w.scalar_names, w.scalars):
        assert np.array_equal(back.pValues(FLOAT, n), s)


# ------------------------------------------------------------------------------------------------------------------
# value grids <-> sidecar blocks (IndexGridBuilder::build / writeIndexGrid, reference src/Utils/GridBuilder.hpp:87-216) over NanoVDB
# float / Vec3f grids, against NanoVDB's own host builder, accessor and file IO
# ------------------------------------------------------------------------------------------------------------------
def _refvalue():
    L = _refhost()
    L.refhost_value_grid_create.restype = C.c_void_p
    L.refhost_value_grid_create.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_double, C.c_char_p, C.c_int]
    L.refhost_value_grid_destroy.argtypes = [C.c_void_p]
    L.refhost_value_grid_bytes.restype = C.c_uint64
    L.refhost_value_grid_bytes.argtypes = [C.c_void_p]
    L.refhost_value_grid_data.restype = C.c_void_p
    L.refhost_value_grid_data.argtypes = [C.c_void_p]
    L.refhost_query_grid.restype = C.c_int
    L.refhost_query_grid.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p]
    L.refhost_grid_meta.restype = C.c_int
    L.refhost_grid_meta.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.POINTER(C.c_double), C.c_void_p]
    return L


def _nanovdb_grid(coords, values, comps, h, name, cls):
    """a float / Vec3f grid made by NanoVDB's own builder (tools::build::Grid + createNanoGrid) -> uint8 buffer"""
    L = _refvalue()
    c = np.ascontiguousarray(coords, np.int32)
    v = np.ascontiguousarray(values, np.float32)
    g = L.refhost_value_grid_create(c.ctypes.data_as(C.c_void_p), v.ctypes.data_as(C.c_void_p), c.shape[0], comps, float(h), name.encode(), cls)
    try:
        n = L.refhost_value_grid_bytes(g)
        return np.ctypeslib.as_array(C.cast(L.refhost_value_grid_data(g), C.POINTER(C.c_uint8)), shape=(n,)).copy()
    finally:
        L.refhost_value_grid_destroy(g)


@needs_refhost
@pytest.mark.parametrize("comps", [1, 3])
def test_sidecar_block_from_a_nanovdb_grid_is_indexgridbuilder_build(w, comps, tmp_path):
    """build(): leaves the grid has are copied whole, the others filled with bytes 0 (or 1 for the SDF)"""
    rng = np.random.default_rng(5)
    keep = rng.random(w.num_leaves) < 0.7 if w.num_leaves > 1 else np.ones(1, bool)      # the grid lacks some of the domain's leaves
    leaf_of_voxel = np.repeat(np.arange(w.num_leaves), 512)
    active = keep[leaf_of_voxel] & (rng.random(w.num_voxels) < 0.6)                      # ... and has inactive voxels inside its leaves
    active[np.nonzero(keep)[0] * 512] = True                                             # every kept leaf exists
    vals = rng.standard_normal((w.num_voxels, comps) if comps == 3 else w.num_voxels).astype(np.float32)
    buf = _nanovdb_grid(w.coords[active], vals[active], comps, w.voxel_size, "density", hio.GRID_CLASS_FOG_VOLUME)
    path = str(tmp_path / "in.nvdb")
    assert _refhost().refhost_write_nvdb(path.encode(), buf.ctypes.data_as(C.c_void_p), 0) == 0      # NanoVDB writes the file ...
    got_buf = hio.read_nvdb(path)                                                                    # ... the product reads it
    info = hio.grid_info(got_buf)
    assert info["name"] == "density" and info["grid_type"] == (hio.GRID_TYPE_VEC3F if comps == 3 else hio.GRID_TYPE_FLOAT)
    assert info["num_leaves"] == int(keep.sum()) and info["voxel_size"] == np.float32(w.voxel_size)
    for fill in (0, 1):
        block = hio.sidecar_from_grid(got_buf, w.origins, fill)
        want = np.where(active.reshape(-1, *([1] * (vals.ndim - 1))), vals, np.float32(0))           # inactive voxels of a NanoVDB leaf hold the background
        missing = ~keep[leaf_of_voxel]
        want[missing] = np.frombuffer(bytes([fill]) * 4, np.float32)[0]
        assert np.array_equal(block.view(np.uint32), want.astype(np.float32).view(np.uint32))
    origins, masks = hio.leaf_topology(got_buf)
    assert np.array_equal(origins, w.origins[keep])
    bits = ((masks[:, :, None] >> np.arange(64, dtype=np.uint64)[None, None, :]) & np.uint64(1)).astype(bool).reshape(-1, 512)
    assert np.array_equal(bits, active.reshape(-1, 512)[keep])


@needs_refhost
@pytest.mark.parametrize("comps", [1, 3])
def test_grid_written_from_a_sidecar_block_is_read_by_nanovdb(w, comps, tmp_path):
    """writeIndexGrid(): FogVolume float / Staggered Vec3f grid over the domain's leaves, values = the block, readable by stock NanoVDB"""
    L = _refvalue()
    rng = np.random.default_rng(6)
    vals = rng.standard_normal((w.num_voxels, 3) if comps == 3 else w.num_voxels).astype(np.float32)
    name = "vel" if comps == 3 else "temperature"
    buf = hio.grid_from_sidecar(w.origins, vals, w.voxel_size, name)
    path = str(tmp_path / "out.nvdb")
    hio.write_nvdb(path, buf)
    n = L.refhost_read_nvdb(path.encode(), None, 0)                                                  # NanoVDB's reader accepts the file
    assert n == buf.size
    back = np.empty(n, np.uint8)
    L.refhost_read_nvdb(path.encode(), back.ctypes.data_as(C.c_void_p), n)
    assert np.array_equal(back, buf)
    meta, nm, h, bbox = np.zeros(6, np.uint64), C.create_string_buffer(256), C.c_double(), np.zeros(6, np.int32)
    assert L.refhost_grid_meta(back.ctypes.data_as(C.c_void_p), meta.ctypes.data_as(C.c_void_p), nm, C.byref(h), bbox.ctypes.data_as(C.c_void_p)) == 0
    assert nm.value.decode() == name and h.value == float(np.float32(w.voxel_size))
    assert meta[0] == (hio.GRID_CLASS_STAGGERED if comps == 3 else hio.GRID_CLASS_FOG_VOLUME)        # GridBuilder.hpp:181-186
    assert meta[1] == (hio.GRID_TYPE_VEC3F if comps == 3 else hio.GRID_TYPE_FLOAT)
    assert meta[2] == w.num_leaves and meta[5] == w.num_voxels
    assert bbox[:3].tolist() == w.origins.min(0).tolist() and bbox[3:].tolist() == (w.origins.max(0) + 7).tolist()
    # every voxel of the domain through NanoVDB's accessor, plus probes outside it
    probe = np.concatenate([w.coords, w.coords[:: max(1, w.num_voxels // 500)] + np.array([4096, -64, 9])]).astype(np.int32)
    got = np.empty((probe.shape[0], comps) if comps == 3 else probe.shape[0], np.float32)
    act = np.empty(probe.shape[0], np.uint8)
    assert L.refhost_query_grid(back.ctypes.data_as(C.c_void_p), np.ascontiguousarray(probe).ctypes.data_as(C.c_void_p), probe.shape[0], comps,
                                got.ctypes.data_as(C.c_void_p), act.ctypes.data_as(C.c_void_p)) == 0
    assert np.array_equal(got[:w.num_voxels], vals) and act[:w.num_voxels].all()
    inside = O.OracleIndex(w.coords).get_values(probe[w.num_voxels:]) != 0
    assert not act[w.num_voxels:][~inside].any() and not got[w.num_voxels:][~inside].any()
    # and back into a block through the product's reader: the round trip is the identity
    assert np.array_equal(hio.sidecar_from_grid(back, w.origins), vals)


def test_sidecar_round_trip_without_nanovdb(w, tmp_path):
    """build_sidecar(write_index_grids(data)) == data, collision SDF fill included; runs without the reference build"""
    data = GridIndexedData()
    data.allocateCoords(w.num_voxels)
    data.pCoords()[:] = w.coords
    data.addValueBlock(VEC3F, "vel")
    data.pValues(VEC3F, "vel")[:] = w.velocity
    for nm, a in zip(w.scalar_names, w.scalars):
        data.addValueBlock(FLOAT, nm)
        data.pValues(FLOAT, nm)[:] = a
    paths = hio.write_index_grids(str(tmp_path), w.origins, data, w.voxel_size)
    grids = [(os.path.basename(p)[:-5], hio.read_nvdb(p), False) for p in paths]
    back = hio.build_sidecar(w.origins, grids)
    assert back.getBlocksOfType(VEC3F) == ["vel"] and back.getBlocksOfType(FLOAT) == list(w.scalar_names)
    assert np.array_equal(back.pValues(VEC3F, "vel"), w.velocity)
    for nm, a in zip(w.scalar_names, w.scalars):
        assert np.array_equal(back.pValues(FLOAT, nm), a)
    assert np.array_equal(back.pCoords(), w.coords)
    # an SDF grid that covers only part of the domain: the rest reads as bytes 0x01 (GridBuilder.hpp:108)
    half = max(1, w.num_leaves // 2)
    sdf = hio.grid_from_sidecar(w.origins[:half], np.full(half * 512, 0.25, np.float32), w.voxel_size, "collision_sdf")
    block = hio.build_sidecar(w.origins, [("collision_sdf", sdf, True)]).pValues(FLOAT, "collision_sdf")
    assert np.all(block[:half * 512] == np.float32(0.25))
    assert np.all(block[half * 512:].view(np.uint32) == 0x01010101)
    with pytest.raises(Exception):
        hio.grid_from_sidecar(w.origins[::-1] if w.num_leaves > 1 else np.array([[1, 0, 0]], np.int32), np.zeros(w.num_leaves * 512, np.float32), 0.1, "x")


# ------------------------------------------------------------------------------------------------------------------
# sourcing (compSum, reference src/SOP/HNanoSolver/SOP_HNanoSolver.cpp:159-181) over NanoVDB value grids and sidecar blocks
# ------------------------------------------------------------------------------------------------------------------
def test_sourcing_adds_the_source_grids_over_the_union_topology():
    rng = np.random.default_rng(5)
    state_leaves = np.array([[0, 0, 0], [0, 0, 8], [8, 0, 0]], np.int32)
    source_leaves = np.array([[16, -8, 0], [0, 0, 8]], np.int32)                  # one new leaf (another root tile: sorts first), one in common
    assert np.array_equal(synth.nanovdb_order(state_leaves), np.arange(3)) and np.array_equal(synth.nanovdb_order(source_leaves), np.arange(2))
    state_mask = np.full((3, 8), np.uint64(0xFFFFFFFFFFFFFFFF))
    source_mask = np.zeros((2, 8), np.uint64)
    source_mask[:, 0] = np.uint64(0xFF)                                           # the source only activates x = 0, y = 0
    dens, src = rng.random(3 * 512).astype(np.float32), rng.random(2 * 512).astype(np.float32)
    vel, vsrc = rng.random((3 * 512, 3)).astype(np.float32), rng.random((2 * 512, 3)).astype(np.float32)
    g_dens = hio.grid_from_sidecar(state_leaves, dens, 0.1, "density", state_mask)
    g_src = hio.grid_from_sidecar(source_leaves, src, 0.1, "density", source_mask)
    g_vel = hio.grid_from_sidecar(state_leaves, vel, 0.1, "vel", state_mask)
    g_vsrc = hio.grid_from_sidecar(source_leaves, vsrc, 0.1, "vel", source_mask)
    # topology: union of leaves, masks OR-ed where the leaves coincide
    o, m = hio.union_topology(hio.leaf_topology(g_vel), hio.leaf_topology(g_vsrc))
    assert sorted(map(tuple, o.tolist())) == sorted({tuple(x) for x in state_leaves.tolist()} | {tuple(x) for x in source_leaves.tolist()})
    by_leaf = {tuple(k): v for k, v in zip(o.tolist(), m)}
    assert by_leaf[(0, 0, 8)][0] == np.uint64(0xFFFFFFFFFFFFFFFF) and by_leaf[(16, -8, 0)][0] == np.uint64(0xFF) and by_leaf[(16, -8, 0)][1] == 0
    # values: state + source over the union domain (padding 0: the domain is the union's leaf set, in NanoVDB order)
    domain = synth.nanovdb_order(o)
    domain = np.ascontiguousarray(o[domain])
    data = hio.build_sidecar(domain, [("density", g_dens, False), ("vel", g_vel, False)])
    hio.comp_sum(domain, data, [("density", g_src), ("vel", g_vsrc)])
    want_d, want_v = np.zeros(domain.shape[0] * 512, np.float32), np.zeros((domain.shape[0] * 512, 3), np.float32)
    for leaves, vals, vvals in ((state_leaves, dens, vel), (source_leaves, src, vsrc)):
        for k, leaf in enumerate(leaves.tolist()):
            at = [tuple(x) for x in domain.tolist()].index(tuple(leaf)) * 512
            want_d[at:at + 512] += vals[k * 512:(k + 1) * 512]
            want_v[at:at + 512] += vvals[k * 512:(k + 1) * 512]
    assert np.array_equal(data.pValues(FLOAT, "density"), want_d)
    assert np.array_equal(data.pValues(VEC3F, "vel").reshape(-1, 3), want_v)
