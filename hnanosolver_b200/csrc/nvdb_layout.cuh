// Node layout of NanoVDB 32.7 float / Vec3f / ValueOnIndex grids, and the grid-level header every value grid starts with: shared by the
// host writer (nvdb_io.cu, hns_sidecar_to_nanovdb) and the device export (export.cu). Restated from externals/nanovdb/NanoVDB.h
// (LeafData :3660-3742, InternalData :3125-3200, RootData :2620-2700); tests/test_nvdb_io.py pins it to NanoVDB's own builder and reader.
#pragma once
#include <cstdint>

namespace hns {
namespace vgrid {

struct ValueLayout {
	uint32_t grid_type;      // GridType: Float 1, Vec3f 6, OnIndex 20
	uint64_t root, tile, upper, lower, leaf;             // node sizes in bytes
	uint64_t upper_table, lower_table, table_stride;     // InternalData::mTable and the size of its Tile union
	uint64_t leaf_values;    // LeafData::mValues (0: none, index grids)
	int components;
};
constexpr ValueLayout kFloatLayout{1, 64, 32, 270400, 33856, 2144, 8256, 1088, 8, 96, 1};
constexpr ValueLayout kVec3fLayout{6, 96, 32, 532544, 66624, 6272, 8256, 1088, 16, 128, 3};
constexpr ValueLayout kIndexLayout{20, 96, 32, 270400, 33856, 96, 8256, 1088, 8, 0, 0};
constexpr uint64_t kUpperChildMask = 4128, kLowerChildMask = 544, kLeafValueMask = 16, kRootTableSize = 24;
constexpr uint64_t kHeadBytes = 672 + 64;  // GridData + TreeData: the root follows

// components 1 -> float, 3 -> Vec3f, else null
inline const ValueLayout* value_layout(int components) { return components == 1 ? &kFloatLayout : components == 3 ? &kVec3fLayout : nullptr; }

// Byte offsets of a breadth-first grid with T root tiles (= upper nodes), nLower lower nodes and L leaves:
// [GridData | TreeData | RootData | tiles | upper nodes | lower nodes | leaves]
struct GridOffsets {
	uint64_t root, upper, lower, leaf, end;
	GridOffsets(const ValueLayout& lay, uint64_t L, uint64_t nLower, uint64_t T)
	    : root(kHeadBytes), upper(root + lay.root + lay.tile * T), lower(upper + lay.upper * T), leaf(lower + lay.lower * nLower), end(leaf + lay.leaf * L) {}
};

// Writes GridData, TreeData and the root's own fields (its bbox and tile count: the first kHeadBytes + lay.root bytes of the grid) of a
// float (class FogVolume) or Vec3f (class Staggered) grid as writeIndexGrid leaves it: background 0, no statistics, checksum disabled,
// the map of voxel size `voxel_size`, `name` truncated to 255 bytes (null: empty). [lo, hi] is the root's index bbox (inclusive; with
// L = 0 it is CoordBBox()'s empty box, INT32_MAX / INT32_MIN), `active` the number of active voxels. Those bytes must be zero on entry.
void write_grid_header(uint8_t* buf, const ValueLayout& lay, uint64_t L, uint64_t nLower, uint64_t T, float voxel_size, const char* name,
                       const int32_t lo[3], const int32_t hi[3], uint64_t active);

}  // namespace vgrid
}  // namespace hns
