// Host-only NanoVDB file IO for index grids (SURVEY.md 8f rank 3: round trip of the topology without Houdini / OpenVDB).
//
// Format: NanoVDB's uncompressed single-grid segment (reference externals/nanovdb/NanoVDB.h:6252-6299, writer :6316-6341, reader
// :6369-6422): FileHeader (16 B: magic, version, gridCount = 1, codec NONE = 0) | FileMetaData (176 B) | grid name incl. '\0' | the
// raw grid buffer. Files written here are read by stock NanoVDB tools (io::readGrid, nanovdb_print), and the reader accepts both that
// layout and a raw buffer dump (which starts with GridData itself, :6375-6386). Everything is restated from the documented layout:
// no NanoVDB header is included. Nothing here touches the GPU.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"
#include "nvdb_layout.cuh"

namespace {

constexpr uint64_t kMagicNumb = 0x304244566f6e614eull, kMagicGrid = 0x314244566f6e614eull, kMagicFile = 0x324244566f6e614eull;
// GridData (672 B): magic 0, checksum 8, version 16, flags 20, gridIndex 24, gridCount 28, gridSize 32, gridName[256] 40, map 296,
// worldBBox 560 (6 doubles), voxelSize 608 (3 doubles), gridClass 632, gridType 636, blind metadata 640...
constexpr size_t kOffVersion = 16, kOffGridIndex = 24, kOffGridCount = 28, kOffGridSize = 32, kOffName = 40, kNameMax = 256, kOffWorldBBox = 560,
                 kOffVoxelSize = 608, kOffGridClass = 632, kOffGridType = 636;
// TreeData (64 B) behind it: nodeOffset[4] (leaf, lower, upper, root; bytes from the tree) 0, nodeCount[3] 32, tileCount[3] 44, voxelCount 56
constexpr size_t kTree = hns::nvdb::kGrid, kOffNodeOffset = 0, kOffNodeCount = 32, kOffTileCount = 44, kOffVoxelCount = 56;
constexpr uint32_t kGridTypeOnIndex = 20;  // GridType::OnIndex

#pragma pack(push, 1)
struct FileHeader {
	uint64_t magic;
	uint32_t version;
	uint16_t gridCount;
	uint16_t codec;
};
struct FileMetaData {
	uint64_t gridSize, fileSize, nameKey, voxelCount;
	uint32_t gridType, gridClass;
	double worldBBox[6];
	int32_t indexBBox[6];
	double voxelSize[3];
	uint32_t nameSize;
	uint32_t nodeCount[4];
	uint32_t tileCount[3];
	uint16_t codec, padding;
	uint32_t version;
};
#pragma pack(pop)
static_assert(sizeof(FileHeader) == 16 && sizeof(FileMetaData) == 176, "NanoVDB file structures");

template <typename T>
T rd(const uint8_t* p) {
	T v;
	std::memcpy(&v, p, sizeof(T));
	return v;
}

// a buffer that can be a single ValueOnIndex grid: long enough, known magic, sizes consistent
int check_grid(const uint8_t* g, uint64_t bytes, bool need_index_grid) {
	using namespace hns;
	// 64: the RootData of a float grid, the smallest there is -- an empty float grid is nothing else (open_grid checks the grid's own)
	if (!g || bytes < nvdb::kGrid + nvdb::kTree + 64) return fail(HNS_ERR_INVALID_ARGUMENT, "buffer is too small for a NanoVDB grid");
	const uint64_t magic = rd<uint64_t>(g);
	if (magic != kMagicNumb && magic != kMagicGrid) return fail(HNS_ERR_INVALID_ARGUMENT, "buffer does not start with a NanoVDB grid magic number");
	if (rd<uint64_t>(g + kOffGridSize) > bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "grid size in the header exceeds the buffer");
	if (need_index_grid && rd<uint32_t>(g + kOffGridType) != kGridTypeOnIndex)
		return fail(HNS_ERR_UNSUPPORTED, "not a ValueOnIndex grid (grid type " + std::to_string(rd<uint32_t>(g + kOffGridType)) + ")");
	return HNS_OK;
}

// Does a file start with GridData itself (a raw buffer dump) rather than with a FileHeader? NanoVDB's own test (GridData::isValid,
// NanoVDB.h:1864-1875): grid magic, or the 32.6 marker in mData2, or the shared magic with gridIndex < gridCount and sane class / type
// -- in a segment those bytes hold FileMetaData::fileSize, whose upper half (read as gridCount) is 0 for files below 4 GB.
bool starts_with_grid(const uint8_t* first, size_t got) {
	if (got < hns::nvdb::kGrid) return false;
	const uint64_t magic = rd<uint64_t>(first);
	if (magic == kMagicGrid || rd<uint64_t>(first + 664) == kMagicGrid) return true;
	if (magic != kMagicNumb) return false;
	const uint32_t major = rd<uint32_t>(first + kOffVersion) >> 21, index = rd<uint32_t>(first + kOffGridIndex), count = rd<uint32_t>(first + kOffGridCount);
	return major == 32 && count > 0 && index < count && rd<uint32_t>(first + kOffGridClass) < 10 && rd<uint32_t>(first + kOffGridType) < 27;
}

struct File {
	FILE* f = nullptr;
	explicit File(const char* path, const char* mode) : f(std::fopen(path, mode)) {}
	~File() {
		if (f) std::fclose(f);
	}
};

}  // namespace

extern "C" {

// Writes one grid (host copy of a NanoVDB buffer, e.g. from hns_grid_nanovdb_download) as an uncompressed .nvdb file.
int hns_nvdb_write(const char* path, const void* nanovdb_buffer, uint64_t bytes) {
	using namespace hns;
	if (!path) return fail(HNS_ERR_INVALID_ARGUMENT, "path is null");
	const uint8_t* g = static_cast<const uint8_t*>(nanovdb_buffer);
	int rc = check_grid(g, bytes, false);
	if (rc) return rc;
	const uint8_t* tree = g + kTree;
	const uint64_t grid_size = rd<uint64_t>(g + kOffGridSize);
	const char* name = reinterpret_cast<const char*>(g + kOffName);
	const uint32_t name_size = uint32_t(strnlen(name, kNameMax - 1)) + 1;  // including the terminator
	FileHeader head{kMagicNumb, rd<uint32_t>(g + kOffVersion), 1, 0};       // NANOVDB_USE_NEW_MAGIC_NUMBERS is off in 32.7 (NanoVDB.h:142)
	FileMetaData meta{};
	meta.gridSize = meta.fileSize = grid_size;
	meta.nameKey = 0;  // as writeUncompressedGrid does
	meta.voxelCount = rd<uint64_t>(tree + kOffVoxelCount);
	meta.gridType = rd<uint32_t>(g + kOffGridType), meta.gridClass = rd<uint32_t>(g + kOffGridClass);
	std::memcpy(meta.worldBBox, g + kOffWorldBBox, sizeof(meta.worldBBox));
	const uint64_t root_off = rd<uint64_t>(tree + kOffNodeOffset + 3 * 8);  // TreeData::bbox() = the root's bbox, its first member (:2281)
	if (root_off) {
		if (kTree + root_off + sizeof(meta.indexBBox) > bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "root offset points outside the buffer");
		std::memcpy(meta.indexBBox, tree + root_off, sizeof(meta.indexBBox));
	} else {  // CoordBBox(): an empty box
		for (int i = 0; i < 3; ++i) meta.indexBBox[i] = INT32_MAX, meta.indexBBox[3 + i] = INT32_MIN;
	}
	std::memcpy(meta.voxelSize, g + kOffVoxelSize, sizeof(meta.voxelSize));
	meta.nameSize = name_size;
	for (int i = 0; i < 3; ++i) meta.nodeCount[i] = rd<uint32_t>(tree + kOffNodeCount + 4 * i), meta.tileCount[i] = rd<uint32_t>(tree + kOffTileCount + 4 * i);
	meta.nodeCount[3] = 1;
	meta.codec = 0, meta.padding = 0, meta.version = head.version;
	File out(path, "wb");
	if (!out.f) return fail(HNS_ERR_RUNTIME, std::string("cannot open for writing: ") + path);
	std::string name_bytes(name, name_size - 1);
	name_bytes.push_back('\0');
	if (std::fwrite(&head, sizeof(head), 1, out.f) != 1 || std::fwrite(&meta, sizeof(meta), 1, out.f) != 1 ||
	    std::fwrite(name_bytes.data(), 1, name_size, out.f) != name_size || std::fwrite(g, 1, grid_size, out.f) != grid_size)
		return fail(HNS_ERR_RUNTIME, std::string("short write: ") + path);
	return HNS_OK;
}

// Size of the first grid stored in `path` (segment layout or raw buffer dump), so that the caller can allocate.
int hns_nvdb_file_grid_bytes(const char* path, uint64_t* bytes_out) {
	using namespace hns;
	if (!path || !bytes_out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	*bytes_out = 0;
	File in(path, "rb");
	if (!in.f) return fail(HNS_ERR_RUNTIME, std::string("cannot open: ") + path);
	uint8_t first[nvdb::kGrid] = {};
	const size_t got = std::fread(first, 1, sizeof(first), in.f);
	if (starts_with_grid(first, got)) {
		*bytes_out = rd<uint64_t>(first + kOffGridSize);
		return HNS_OK;
	}
	if (got < sizeof(FileHeader) + sizeof(FileMetaData)) return fail(HNS_ERR_INVALID_ARGUMENT, "file is too short for a NanoVDB grid");
	const FileHeader head = rd<FileHeader>(first);
	const FileMetaData meta = rd<FileMetaData>(first + sizeof(FileHeader));
	if (head.magic != kMagicNumb && head.magic != kMagicFile) return fail(HNS_ERR_INVALID_ARGUMENT, "not a NanoVDB file (magic number)");
	if (head.gridCount < 1) return fail(HNS_ERR_INVALID_ARGUMENT, "NanoVDB file segment holds no grid");
	if (head.codec != 0 || meta.codec != 0) return fail(HNS_ERR_UNSUPPORTED, "compressed NanoVDB files (ZIP / BLOSC) are not supported");
	*bytes_out = meta.gridSize;
	return HNS_OK;
}

// Reads the first grid of `path` into `dst` (capacity `capacity` bytes, see hns_nvdb_file_grid_bytes).
int hns_nvdb_read(const char* path, void* dst, uint64_t capacity) {
	using namespace hns;
	uint64_t need = 0;
	int rc = hns_nvdb_file_grid_bytes(path, &need);
	if (rc) return rc;
	if (!dst || capacity < need) return fail(HNS_ERR_INVALID_ARGUMENT, "destination buffer is too small");
	File in(path, "rb");
	if (!in.f) return fail(HNS_ERR_RUNTIME, std::string("cannot open: ") + path);
	uint8_t first[nvdb::kGrid] = {};
	const size_t got = std::fread(first, 1, sizeof(first), in.f);
	long skip = 0;
	if (!starts_with_grid(first, got)) skip = long(sizeof(FileHeader) + sizeof(FileMetaData) + rd<FileMetaData>(first + sizeof(FileHeader)).nameSize);
	if (std::fseek(in.f, skip, SEEK_SET) != 0) return fail(HNS_ERR_RUNTIME, "seek failed");
	if (std::fread(dst, 1, need, in.f) != need) return fail(HNS_ERR_RUNTIME, "short read: file ends inside the grid");
	return check_grid(static_cast<const uint8_t*>(dst), need, false);
}

// Leaf origins (int32[L][3], in the buffer's leaf order = NanoVDB order) and voxel size of a ValueOnIndex grid buffer on the host:
// what hns_grid_create_from_origins needs to rebuild the device grid. origins_out may be null to query the count.
int hns_nvdb_leaf_origins(const void* nanovdb_buffer, uint64_t bytes, int32_t* origins_out, uint64_t* num_leaves_out, float* voxel_size_out) {
	using namespace hns;
	const uint8_t* g = static_cast<const uint8_t*>(nanovdb_buffer);
	int rc = check_grid(g, bytes, true);
	if (rc) return rc;
	const uint8_t* tree = g + kTree;
	const uint64_t leaf_off = rd<uint64_t>(tree + kOffNodeOffset), L = rd<uint32_t>(tree + kOffNodeCount);
	if (L && kTree + leaf_off + L * nvdb::kLeaf > bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "leaf nodes lie outside the buffer");
	if (num_leaves_out) *num_leaves_out = L;
	if (voxel_size_out) *voxel_size_out = float(rd<double>(g + kOffVoxelSize));
	if (origins_out)
		for (uint64_t l = 0; l < L; ++l) std::memcpy(origins_out + 3 * l, tree + leaf_off + l * nvdb::kLeaf, 12);  // LeafData starts with mBBoxMin
	return HNS_OK;
}

}  // extern "C"

// =====================================================================================================================================
// Value grids: NanoVDB float / Vec3f grids <-> the dense-leaf sidecar blocks of HNS::GridIndexedData.
//
// Reference: IndexGridBuilder::build (src/Utils/GridBuilder.hpp:87-166) fills a block per input grid by walking the DOMAIN's leaves: a
// leaf the grid has at that origin is memcpy'd whole (all 512 values, active or not), a missing one is memset -- with byte 0 for float /
// vector grids (:124,:145) and with byte 0x01 for the collision SDF (:108, i.e. 2.4e-38, "on the surface"). writeIndexGrid (:168-216)
// goes back: a grid with the domain's topology, every leaf buffer memcpy'd from the block, class FOG_VOLUME for float grids and
// STAGGERED (+ VEC_CONTRAVARIANT_RELATIVE, an OpenVDB-only tag) for vector grids. The reference does this over OpenVDB grids; OpenVDB
// is not vendored, NanoVDB is (externals/nanovdb), and its float / Vec3f grids carry the same leaf buffers, so the headless path reads
// and writes those. Node layouts: nvdb_layout.cuh (shared with the device export, export.cu); tests/test_nvdb_io.py reads and writes
// the same grids with NanoVDB's own builder, accessor and file IO (oracle/_ref/libref_host.so).
// =====================================================================================================================================
using namespace hns::vgrid;

namespace {

const ValueLayout* layout_of(uint32_t grid_type) {
	return grid_type == 1 ? &kFloatLayout : grid_type == 6 ? &kVec3fLayout : grid_type == 20 ? &kIndexLayout : nullptr;
}

struct GridWalk {
	const uint8_t* g;
	uint64_t bytes;
	const ValueLayout* lay;
	const uint8_t* root;
	uint32_t tiles;
	// leaf record containing voxel (x, y, z), or null: root tile scan, upper, lower (ReadAccessor::probeLeaf, NanoVDB.h:5683-5698)
	const uint8_t* probe_leaf(int32_t x, int32_t y, int32_t z) const {
		const uint64_t key = (uint64_t(uint32_t(z) >> 12)) | (uint64_t(uint32_t(y) >> 12) << 21) | (uint64_t(uint32_t(x) >> 12) << 42);
		const uint8_t* upper = nullptr;
		for (uint32_t t = 0; t < tiles; ++t) {
			const uint8_t* tile = root + lay->root + lay->tile * t;
			if (rd<uint64_t>(tile) == key) {
				const int64_t child = rd<int64_t>(tile + 8);
				if (child) upper = root + child;
				break;
			}
		}
		if (!upper) return nullptr;
		const uint32_t uo = uint32_t(((x & 4095) >> 7) << 10 | ((y & 4095) >> 7) << 5 | ((z & 4095) >> 7));
		if (!((rd<uint64_t>(upper + kUpperChildMask + 8 * (uo >> 6)) >> (uo & 63)) & 1)) return nullptr;
		const uint8_t* lower = upper + rd<int64_t>(upper + lay->upper_table + lay->table_stride * uo);
		const uint32_t lo = uint32_t(((x & 127) >> 3) << 8 | ((y & 127) >> 3) << 4 | ((z & 127) >> 3));
		if (!((rd<uint64_t>(lower + kLowerChildMask + 8 * (lo >> 6)) >> (lo & 63)) & 1)) return nullptr;
		const uint8_t* leaf = lower + rd<int64_t>(lower + lay->lower_table + lay->table_stride * lo);
		return leaf + lay->leaf <= g + bytes ? leaf : nullptr;
	}
};

int open_grid(const void* buffer, uint64_t bytes, GridWalk& w) {
	using namespace hns;
	const uint8_t* g = static_cast<const uint8_t*>(buffer);
	int rc = check_grid(g, bytes, false);
	if (rc) return rc;
	const uint32_t type = rd<uint32_t>(g + kOffGridType);
	const ValueLayout* lay = layout_of(type);
	if (!lay) return fail(HNS_ERR_UNSUPPORTED, "grid type " + std::to_string(type) + " is not float, Vec3f or ValueOnIndex");
	const uint64_t root_off = rd<uint64_t>(g + kTree + kOffNodeOffset + 3 * 8);
	if (kTree + root_off + lay->root > bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "root offset points outside the buffer");
	w = GridWalk{g, bytes, lay, g + kTree + root_off, 0};
	w.tiles = rd<uint32_t>(w.root + kRootTableSize);
	if (kTree + root_off + lay->root + uint64_t(w.tiles) * lay->tile > bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "root tiles lie outside the buffer");
	return HNS_OK;
}

}  // namespace

extern "C" {

// type / class / leaf count / voxel size / name (char[256]) of the grid in `buffer`; any out pointer may be null
int hns_nvdb_grid_info(const void* buffer, uint64_t bytes, uint32_t* grid_type, uint32_t* grid_class, uint64_t* num_leaves, float* voxel_size, char* name256) {
	using namespace hns;
	const uint8_t* g = static_cast<const uint8_t*>(buffer);
	int rc = check_grid(g, bytes, false);
	if (rc) return rc;
	if (grid_type) *grid_type = rd<uint32_t>(g + kOffGridType);
	if (grid_class) *grid_class = rd<uint32_t>(g + kOffGridClass);
	if (num_leaves) *num_leaves = rd<uint32_t>(g + kTree + kOffNodeCount);
	if (voxel_size) *voxel_size = float(rd<double>(g + kOffVoxelSize));
	if (name256) {
		std::memcpy(name256, g + kOffName, kNameMax);
		name256[kNameMax - 1] = '\0';
	}
	return HNS_OK;
}

// Leaf origins (int32[L][3]) and active-voxel masks (uint64[L][8], bit x<<6 | y<<3 | z) of a float / Vec3f / index grid, in the buffer's
// leaf order: the topology arguments of hns_domain_build. Either output may be null.
int hns_nvdb_leaf_topology(const void* buffer, uint64_t bytes, int32_t* origins_out, uint64_t* masks_out, uint64_t* num_leaves_out) {
	using namespace hns;
	GridWalk w{};
	int rc = open_grid(buffer, bytes, w);
	if (rc) return rc;
	const uint8_t* tree = w.g + kTree;
	const uint64_t leaf_off = rd<uint64_t>(tree + kOffNodeOffset), L = rd<uint32_t>(tree + kOffNodeCount);
	if (L && kTree + leaf_off + L * w.lay->leaf > bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "leaf nodes lie outside the buffer");
	if (num_leaves_out) *num_leaves_out = L;
	for (uint64_t l = 0; l < L; ++l) {
		const uint8_t* leaf = tree + leaf_off + l * w.lay->leaf;
		if (origins_out) {
			std::memcpy(origins_out + 3 * l, leaf, 12);
			for (int a = 0; a < 3; ++a) origins_out[3 * l + a] &= ~7;  // LeafData::mBBoxMin is the origin only when the bbox was never tightened
		}
		if (masks_out) std::memcpy(masks_out + 8 * l, leaf + kLeafValueMask, 64);
	}
	return HNS_OK;
}

// IndexGridBuilder::build for one block (GridBuilder.hpp:94-150): for every domain leaf, the grid's leaf buffer at that origin (512 values,
// active or not) or 512 values whose bytes are all `fill_byte` (0 for float / vector blocks, 1 for the collision SDF, :108).
// out: float[n_leaves * 512] for a float grid, float[n_leaves * 512][3] for a Vec3f grid.
int hns_sidecar_from_nanovdb(const void* buffer, uint64_t bytes, const int32_t* domain_origins, uint64_t n_leaves, int fill_byte, void* out) {
	using namespace hns;
	GridWalk w{};
	int rc = open_grid(buffer, bytes, w);
	if (rc) return rc;
	if (!w.lay->leaf_values) return fail(HNS_ERR_UNSUPPORTED, "an index grid holds no values");
	if (n_leaves && (!domain_origins || !out)) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	const size_t leaf_bytes = size_t(512) * 4 * w.lay->components;
	for (uint64_t l = 0; l < n_leaves; ++l) {
		const int32_t* o = domain_origins + 3 * l;
		uint8_t* dst = static_cast<uint8_t*>(out) + l * leaf_bytes;
		if (const uint8_t* leaf = w.probe_leaf(o[0], o[1], o[2])) std::memcpy(dst, leaf + w.lay->leaf_values, leaf_bytes);
		else std::memset(dst, fill_byte, leaf_bytes);
	}
	return HNS_OK;
}

// size of the grid hns_sidecar_to_nanovdb emits for these leaves (components: 1 float, 3 Vec3f); 0 on a bad argument
uint64_t hns_sidecar_nanovdb_bytes(const int32_t* domain_origins, uint64_t n_leaves, int components) {
	const ValueLayout* lay = value_layout(components);
	if (!lay || (n_leaves && !domain_origins)) return 0;
	uint64_t T = 0, nLower = 0;
	for (uint64_t l = 0; l < n_leaves; ++l) {
		const int32_t *o = domain_origins + 3 * l, *p = o - 3;
		const bool newTile = l == 0 || (o[0] >> 12) != (p[0] >> 12) || (o[1] >> 12) != (p[1] >> 12) || (o[2] >> 12) != (p[2] >> 12);
		const bool newLower = newTile || (o[0] >> 7) != (p[0] >> 7) || (o[1] >> 7) != (p[1] >> 7) || (o[2] >> 7) != (p[2] >> 7);
		T += newTile, nLower += newLower;
	}
	return GridOffsets(*lay, n_leaves, nLower, T).end;
}

// IndexGridBuilder::writeIndexGrid (GridBuilder.hpp:168-216) over NanoVDB: a float (class FogVolume) or Vec3f (class Staggered) grid with
// a leaf at every domain origin (NanoVDB order, as hns_grid_create_from_origins takes them), leaf buffers = the block's values, value
// masks = `masks` (uint64[n][8]; null = every voxel active), background 0, no statistics. out_buf: hns_sidecar_nanovdb_bytes bytes.
int hns_sidecar_to_nanovdb(const int32_t* domain_origins, uint64_t n_leaves, const uint64_t* masks, const void* values, int components, float voxel_size,
                           const char* name, void* out_buf, uint64_t capacity) {
	using namespace hns;
	const ValueLayout* lay = value_layout(components);
	if (!lay) return fail(HNS_ERR_INVALID_ARGUMENT, "components must be 1 (float) or 3 (Vec3f)");
	if (!(voxel_size > 0.0f)) return fail(HNS_ERR_INVALID_ARGUMENT, "voxelSize must be positive.");
	if (n_leaves && (!domain_origins || !values)) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	const uint64_t bytes = hns_sidecar_nanovdb_bytes(domain_origins, n_leaves, components);
	if (!out_buf || capacity < bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "output buffer is too small");
	for (uint64_t l = 1; l < n_leaves; ++l) {  // strictly increasing NanoVDB order: (tile, upper offset, lower offset)
		const int32_t *a = domain_origins + 3 * (l - 1), *b = domain_origins + 3 * l;
		if (!key_less(nvdb_leaf_key(a[0], a[1], a[2]), nvdb_leaf_key(b[0], b[1], b[2])))
			return fail(HNS_ERR_TOPOLOGY, "leaves are not in strictly increasing NanoVDB order at leaf " + std::to_string(l));
	}
	uint8_t* buf = static_cast<uint8_t*>(out_buf);
	std::memset(buf, 0, bytes);
	auto put = [](uint8_t* p, auto v) { std::memcpy(p, &v, sizeof(v)); };
	uint64_t T = 0, nLower = 0;
	for (uint64_t l = 0; l < n_leaves; ++l) {
		const int32_t *o = domain_origins + 3 * l, *p = o - 3;
		const bool newTile = l == 0 || (o[0] >> 12) != (p[0] >> 12) || (o[1] >> 12) != (p[1] >> 12) || (o[2] >> 12) != (p[2] >> 12);
		T += newTile, nLower += newTile || (o[0] >> 7) != (p[0] >> 7) || (o[1] >> 7) != (p[1] >> 7) || (o[2] >> 7) != (p[2] >> 7);
	}
	const GridOffsets off(*lay, n_leaves, nLower, T);
	const uint64_t oRoot = off.root, oUpper = off.upper, oLower = off.lower, oLeaf = off.leaf;
	uint64_t active = 0;
	// nodes, walking the sorted leaf list once
	struct Box {
		int32_t lo[3] = {INT32_MAX, INT32_MAX, INT32_MAX}, hi[3] = {INT32_MIN, INT32_MIN, INT32_MIN};
		void add(const int32_t* a, const int32_t* b) {
			for (int d = 0; d < 3; ++d) lo[d] = std::min(lo[d], a[d]), hi[d] = std::max(hi[d], b[d]);
		}
		void store(uint8_t* p) const { std::memcpy(p, lo, 12), std::memcpy(p + 12, hi, 12); }
	} rootBox, upBox, loBox;
	uint8_t *U = nullptr, *Lo = nullptr;
	int64_t iu = -1, il = -1;
	const size_t leaf_bytes = size_t(512) * 4 * components;
	for (uint64_t l = 0; l < n_leaves; ++l) {
		const int32_t *o = domain_origins + 3 * l, *p = o - 3;
		if ((o[0] | o[1] | o[2]) & 7) return fail(HNS_ERR_TOPOLOGY, "leaf origin is not a multiple of 8 at leaf " + std::to_string(l));
		const bool newUpper = l == 0 || (o[0] >> 12) != (p[0] >> 12) || (o[1] >> 12) != (p[1] >> 12) || (o[2] >> 12) != (p[2] >> 12);
		const bool newLower = newUpper || (o[0] >> 7) != (p[0] >> 7) || (o[1] >> 7) != (p[1] >> 7) || (o[2] >> 7) != (p[2] >> 7);
		if (newLower && Lo) loBox.store(Lo), upBox.add(loBox.lo, loBox.hi);
		if (newUpper && U) upBox.store(U), rootBox.add(upBox.lo, upBox.hi);
		if (newUpper) {
			++iu;
			U = buf + oUpper + lay->upper * uint64_t(iu);
			upBox = Box();
			uint8_t* tile = buf + oRoot + lay->root + lay->tile * uint64_t(iu);
			put(tile, uint64_t(uint32_t(o[2]) >> 12) | uint64_t(uint32_t(o[1]) >> 12) << 21 | uint64_t(uint32_t(o[0]) >> 12) << 42);
			put(tile + 8, int64_t(U - (buf + oRoot)));
		}
		const uint32_t uo = uint32_t(((o[0] & 4095) >> 7) << 10 | ((o[1] & 4095) >> 7) << 5 | ((o[2] & 4095) >> 7));
		if (newLower) {
			++il;
			Lo = buf + oLower + lay->lower * uint64_t(il);
			loBox = Box();
			uint64_t word = rd<uint64_t>(U + kUpperChildMask + 8 * (uo >> 6)) | (uint64_t(1) << (uo & 63));
			put(U + kUpperChildMask + 8 * (uo >> 6), word);
			put(U + lay->upper_table + lay->table_stride * uo, int64_t(Lo - U));
		}
		const uint32_t lo = uint32_t(((o[0] & 127) >> 3) << 8 | ((o[1] & 127) >> 3) << 4 | ((o[2] & 127) >> 3));
		uint8_t* F = buf + oLeaf + lay->leaf * l;
		put(Lo + kLowerChildMask + 8 * (lo >> 6), rd<uint64_t>(Lo + kLowerChildMask + 8 * (lo >> 6)) | (uint64_t(1) << (lo & 63)));
		put(Lo + lay->lower_table + lay->table_stride * lo, int64_t(F - Lo));
		std::memcpy(F, o, 12);
		F[12] = F[13] = F[14] = 7;
		F[15] = 0x02;                                           // bbox valid; no min/max, no average / deviation
		if (masks) std::memcpy(F + kLeafValueMask, masks + 8 * l, 64);
		else std::memset(F + kLeafValueMask, 0xFF, 64);
		for (int k = 0; k < 8; ++k) active += uint64_t(__builtin_popcountll(rd<uint64_t>(F + kLeafValueMask + 8 * k)));
		std::memcpy(F + lay->leaf_values, static_cast<const uint8_t*>(values) + l * leaf_bytes, leaf_bytes);
		const int32_t hi[3] = {o[0] + 7, o[1] + 7, o[2] + 7};
		loBox.add(o, hi);
	}
	if (Lo) loBox.store(Lo), upBox.add(loBox.lo, loBox.hi);
	if (U) upBox.store(U), rootBox.add(upBox.lo, upBox.hi);
	write_grid_header(buf, *lay, n_leaves, nLower, T, voxel_size, name, rootBox.lo, rootBox.hi, active);
	return HNS_OK;
}

}  // extern "C"

namespace hns::vgrid {

void write_grid_header(uint8_t* buf, const ValueLayout& lay, uint64_t L, uint64_t nLower, uint64_t T, float voxel_size, const char* name,
                       const int32_t lo[3], const int32_t hi[3], uint64_t active) {
	auto put = [](uint8_t* p, auto v) { std::memcpy(p, &v, sizeof(v)); };
	const GridOffsets off(lay, L, nLower, T);
	const uint64_t oTree = nvdb::kGrid, bytes = off.end;
	const double s = double(voxel_size);
	// GridData (GridData::init, NanoVDB.h:1834-1862)
	uint8_t* g = buf;
	put(g + 0, kMagicNumb);
	put(g + 8, ~uint64_t(0));                                   // checksum: disabled
	put(g + kOffVersion, uint32_t((32u << 21) | (7u << 10)));
	put(g + 20, uint32_t(0x22));                                // HasBBox | IsBreadthFirst; no min/max, average, std deviation
	put(g + kOffGridIndex, uint32_t(0));
	put(g + kOffGridCount, uint32_t(1));
	put(g + kOffGridSize, bytes);
	if (name) std::strncpy(reinterpret_cast<char*>(g + kOffName), name, kNameMax - 1);
	uint8_t* m = g + 296;                                       // Map: matF[9] invMatF[9] vecF[3] taperF matD[9] invMatD[9] vecD[3] taperD
	for (int d = 0; d < 3; ++d) {
		put(m + 16 * d, float(s));
		put(m + 36 + 16 * d, 1.0f / float(s));
		put(m + 88 + 32 * d, s);
		put(m + 160 + 32 * d, 1.0 / s);
	}
	put(m + 84, 1.0f);
	put(m + 256, 1.0);
	for (int d = 0; d < 3; ++d) put(g + kOffVoxelSize + 8 * d, s);
	put(g + kOffGridClass, uint32_t(lay.components == 1 ? 2 : 3));  // GridClass::FogVolume / Staggered (GridBuilder.hpp:181-186)
	put(g + kOffGridType, lay.grid_type);
	put(g + 640, int64_t(bytes));                               // blind metadata: none, offset = end of the grid
	put(g + 656, uint64_t(0));
	put(g + 664, kMagicGrid);
	// TreeData
	uint8_t* t = buf + oTree;
	put(t + 0, int64_t(off.leaf - oTree));
	put(t + 8, int64_t(off.lower - oTree));
	put(t + 16, int64_t(off.upper - oTree));
	put(t + 24, int64_t(off.root - oTree));
	put(t + 32, uint32_t(L)), put(t + 36, uint32_t(nLower)), put(t + 40, uint32_t(T));   // node counts; tile counts stay 0: no active tiles
	put(t + 56, active);
	// RootData: bbox, tile count; background and statistics stay 0
	uint8_t* r = buf + off.root;
	std::memcpy(r, lo, 12), std::memcpy(r + 12, hi, 12);
	put(r + kRootTableSize, uint32_t(T));
	for (int d = 0; d < 3; ++d) {                               // world bbox = index bbox (inclusive max + 1 voxel) x scale, as NanoVDB's builders set it
		const double a = double(lo[d]) * s, b = double(L ? hi[d] + 1 : hi[d]) * s;
		put(g + kOffWorldBBox + 8 * d, L ? std::min(a, b) : 0.0);
		put(g + kOffWorldBBox + 24 + 8 * d, L ? std::max(a, b) : 0.0);
	}
}

}  // namespace hns::vgrid

namespace hns {

// The source of compSum (SOP_HNanoSolver.cpp:159-181) as flat tables: the float / Vec3f grid's leaf records -- all inside the buffer,
// their origins (bboxMin & ~7, as hns_nvdb_leaf_topology reads them) distinct -- sorted by nvdb_leaf_key, with the 512 values of each.
// Host only and before any CUDA call: a malformed buffer is refused here, and the device indexes these tables, never an offset read
// from the buffer.
int source_tables(const void* buffer, uint64_t bytes, SourceTables& out) {
	GridWalk w{};
	int rc = open_grid(buffer, bytes, w);
	if (rc) return rc;
	if (!w.lay->leaf_values) return fail(HNS_ERR_UNSUPPORTED, "an index grid holds no values to add");
	const uint8_t* tree = w.g + kTree;
	const uint64_t leaf_off = rd<uint64_t>(tree + kOffNodeOffset), L = rd<uint32_t>(tree + kOffNodeCount);
	if (L && (leaf_off > bytes - kTree || L * w.lay->leaf > bytes - kTree - leaf_off))
		return fail(HNS_ERR_INVALID_ARGUMENT, "leaf nodes lie outside the buffer");
	std::vector<int4> origins(L);
	std::vector<ulonglong2> keys(L);
	std::vector<uint32_t> order(L);
	for (uint64_t l = 0; l < L; ++l) {
		int32_t o[3];
		std::memcpy(o, tree + leaf_off + l * w.lay->leaf, 12);
		origins[l] = make_int4(o[0] & ~7, o[1] & ~7, o[2] & ~7, 0);
		keys[l] = nvdb_leaf_key(origins[l].x, origins[l].y, origins[l].z);
		order[l] = uint32_t(l);
	}
	std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return key_less(keys[a], keys[b]); });
	for (uint64_t i = 1; i < L; ++i)
		if (!key_less(keys[order[i - 1]], keys[order[i]])) {
			const int4 o = origins[order[i]];
			return fail(HNS_ERR_INVALID_ARGUMENT, "two leaves of the source have the origin (" + std::to_string(o.x) + ", " + std::to_string(o.y) + ", " +
			                                          std::to_string(o.z) + ")");
		}
	const int C = w.lay->components;
	const size_t leaf_floats = size_t(512) * C;
	out.components = C;
	out.keys.resize(L), out.origins.resize(L), out.values.resize(L * leaf_floats), out.masks.resize(L * 8);
	for (uint64_t i = 0; i < L; ++i) {
		const uint32_t l = order[i];
		out.keys[i] = keys[l], out.origins[i] = origins[l];
		std::memcpy(out.values.data() + i * leaf_floats, tree + leaf_off + l * w.lay->leaf + w.lay->leaf_values, leaf_floats * sizeof(float));
		std::memcpy(out.masks.data() + i * 8, tree + leaf_off + l * w.lay->leaf + kLeafValueMask, 64);
	}
	return HNS_OK;
}

}  // namespace hns
