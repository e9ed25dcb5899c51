"""The oracle's index-grid restatement against (a) the vendored NanoVDB unit-test vectors and (b) a real NanoVDB host grid."""
import numpy as np
import pytest

from oracle import oracle as O

needs_refhost = pytest.mark.skipif(not O.ref_host_available(), reason="needs oracle/_ref/libref_host.so, built only from the original project's sources (oracle/Makefile REF)")


def test_nanovdb_unittest_vector():
    # externals/nanovdb/unittest/TestNanoVDB.cu:302-398 (Basic_CudaPointsToGrid_ValueOnIndex)
    ix = O.OracleIndex([[1, 2, 3], [1, 2, 4], [8, 2, 3]])
    assert ix.num_leaves == 2
    assert ix.num_active + 1 == 4                                   # valueCount == 4
    assert ix.get_values([[1, 2, 3], [1, 2, 4], [8, 2, 3], [0, 2, 3]]).tolist() == [1, 2, 3, 0]
    buf = ix.nanovdb_buffer(1.0)
    assert buf.size == 672 + 64 + (96 + 32 * 1) + 270400 + 33856 + 2 * 96   # grid + tree + root(1 tile) + upper + lower + 2 leaves
    assert buf[:8].tobytes() == b"NanoVDB0"
    assert int(np.frombuffer(buf[32:40].tobytes(), np.uint64)[0]) == buf.size


def test_unsorted_and_duplicate_input_is_sorted_like_voxelsToGrid():
    pts = np.array([[8, 2, 3], [1, 2, 4], [1, 2, 3], [1, 2, 4]], np.int32)
    ix = O.OracleIndex(pts)
    assert ix.num_active == 3
    assert ix.get_values([[1, 2, 3], [1, 2, 4], [8, 2, 3]]).tolist() == [1, 2, 3]


def test_dense_leaf_indexing_contract():
    # sidecar slot of voxel (x,y,z) in leaf l = l*512 + (x&7)<<6 | (y&7)<<3 | (z&7); NanoVDB index = slot + 1 (SURVEY 8 a-0)
    from hnanosolver_b200 import synth

    w = synth.random_leaves(30, 5, 3, offset=(-40, 4096 - 16, -4096 * 2 + 8))
    ix = O.OracleIndex(w.coords)
    assert np.array_equal(ix.leaf_origins(), w.origins)
    assert np.array_equal(ix.get_values(w.coords), np.arange(1, w.num_voxels + 1, dtype=np.uint64))
    # prefix sum word of a dense leaf (SURVEY Appendix C)
    buf = ix.nanovdb_buffer(0.1)
    leaf0 = buf.size - 96 * w.num_leaves
    assert int(np.frombuffer(buf[leaf0 + 88:leaf0 + 96].tobytes(), np.uint64)[0]) == 0x7030140803010040


@needs_refhost
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_get_value_matches_real_nanovdb(seed):
    rng = np.random.default_rng(seed)
    pts = np.concatenate([rng.integers(-6000, 6000, size=(1500, 3)), rng.integers(-20, 20, size=(2500, 3))]).astype(np.int32)
    ix, rh = O.OracleIndex(pts), O.RefHostGrid(pts)
    assert ix.num_leaves == rh.leaf_count
    assert ix.num_active + 1 == rh.value_count
    q = np.concatenate([pts, pts + rng.integers(-2, 3, size=pts.shape), rng.integers(-7000, 7000, size=(4000, 3))]).astype(np.int32)
    assert np.array_equal(ix.get_values(q), rh.get_values(q))


@needs_refhost
def test_tree_structure_matches_real_nanovdb_host_builder():
    """Node hierarchy emitted by the oracle == the one nanovdb::tools::createNanoGrid builds (child masks, child offsets,
    leaf masks / mOffset / mPrefixSum, root tile keys). Flags / bbox / stats fields legitimately differ between the host
    builder and voxelsToGrid and are not compared here (they are compared against voxelsToGrid itself on the GPU)."""
    rng = np.random.default_rng(5)
    pts = np.concatenate([rng.integers(-5000, 5000, size=(300, 3)), rng.integers(0, 40, size=(4000, 3))]).astype(np.int32)
    ix, rh = O.OracleIndex(pts), O.RefHostGrid(pts)
    a, b = ix.nanovdb_buffer(0.1), rh.buffer()
    assert a.size == b.size
    tree = 672
    assert np.array_equal(a[tree:tree + 44], b[tree:tree + 44])  # node offsets + node counts (mTileCount is builder specific:
    #                                                              voxelsToGrid sets it equal to mNodeCount, PointsToGrid.cuh:792-794)
    T = int(np.frombuffer(a[tree + 40:tree + 44].tobytes(), np.uint32)[0])
    nLo = int(np.frombuffer(a[tree + 36:tree + 40].tobytes(), np.uint32)[0])
    L = int(np.frombuffer(a[tree + 32:tree + 36].tobytes(), np.uint32)[0])
    root = tree + 64
    for t in range(T):
        tile = root + 96 + 32 * t
        assert np.array_equal(a[tile:tile + 16], b[tile:tile + 16])  # key + child offset
    up0 = root + 96 + 32 * T
    for u in range(T):
        o = up0 + 270400 * u
        assert np.array_equal(a[o + 4128:o + 8224], b[o + 4128:o + 8224])      # child mask
        cm = np.unpackbits(a[o + 4128:o + 8224], bitorder="little").astype(bool)
        ta = np.frombuffer(a[o + 8256:o + 270400].tobytes(), np.int64)
        tb = np.frombuffer(b[o + 8256:o + 270400].tobytes(), np.int64)
        assert np.array_equal(ta[cm], tb[cm])
    lo0 = up0 + 270400 * T
    for l in range(nLo):
        o = lo0 + 33856 * l
        assert np.array_equal(a[o + 544:o + 1056], b[o + 544:o + 1056])
        cm = np.unpackbits(a[o + 544:o + 1056], bitorder="little").astype(bool)
        ta = np.frombuffer(a[o + 1088:o + 33856].tobytes(), np.int64)
        tb = np.frombuffer(b[o + 1088:o + 33856].tobytes(), np.int64)
        assert np.array_equal(ta[cm], tb[cm])
    lf0 = lo0 + 33856 * nLo
    la = a[lf0:lf0 + 96 * L].reshape(L, 96)
    lb = b[lf0:lf0 + 96 * L].reshape(L, 96)
    assert np.array_equal(la[:, 16:96], lb[:, 16:96])               # value mask, mOffset, mPrefixSum
    assert np.array_equal(la[:, 0:15], lb[:, 0:15])                 # bbox min + dif
