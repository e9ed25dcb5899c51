// Shared declarations for libhns_b200: error handling, launch accounting, device-side grid view.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/hns_b200.h"

namespace hns {

// ---- errors -------------------------------------------------------------------------------------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

#define HNS_CUDA(call)                                                                                           \
	do {                                                                                                         \
		cudaError_t e_ = (call);                                                                                 \
		if (e_ != cudaSuccess)                                                                                   \
			return ::hns::fail(HNS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
	} while (0)

void release_grid_pool();  // topology.cu: device blocks of destroyed index grids kept for reuse

// ---- launch accounting (hns_launch_count) ---------------------------------------------------------------
extern std::atomic<uint64_t> g_launches;
#define HNS_LAUNCH(kernel, grid, block, smem, stream, ...)              \
	do {                                                                \
		kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);     \
		::hns::g_launches.fetch_add(1, std::memory_order_relaxed);      \
	} while (0)

// ---- NanoVDB 32.7 ValueOnIndex buffer layout (own POD mirror; SURVEY.md Appendix B/C) -------------------
// [GridData 672][TreeData 64][RootData 96][Tile 32 x T][Upper 270400 x T][Lower 33856 x nLower][Leaf 96 x L]
namespace nvdb {
constexpr uint64_t kGrid = 672, kTree = 64, kRoot = 96, kTile = 32, kUpper = 270400, kLower = 33856, kLeaf = 96;
constexpr uint64_t kUpperChildMask = 4128, kUpperTable = 8256;  // InternalData<.,5>: bbox 0, flags 24, valueMask 32, childMask 4128, stats 8224.., table 8256
constexpr uint64_t kLowerChildMask = 544, kLowerTable = 1088;   // InternalData<.,4>: bbox 0, flags 24, valueMask 32, childMask 544, stats 1056.., table 1088
constexpr uint64_t kLeafMask = 16, kLeafOffset = 80, kLeafPrefix = 88;  // LeafData<ValueOnIndex>: bboxMin 0, bboxDif 12, flags 15, mask 16, mOffset 80, mPrefixSum 88
constexpr uint64_t kRootTableSize = 24;
}  // namespace nvdb

// Device view of an index grid.
struct GridView {
	const uint8_t* nvdb;      // the NanoVDB buffer
	const int4* origin;       // [L] leaf origins (x, y, z, 0)
	const int32_t* nbr;       // [L][27] neighbour leaf ids, -1 = none; slot (dx+1)*9+(dy+1)*3+(dz+1)
	uint32_t num_leaves;
	uint32_t num_tiles;
	uint64_t off_root, off_leaf;  // byte offsets of RootData and of the first leaf inside nvdb
	// optional work list: when set, a launch processes leaves list[0..num_list) instead of 0..num_leaves (sharded runs: owned leaves
	// only, or the boundary / interior split that lets a ghost exchange overlap the interior sweep)
	const int32_t* list;
	uint32_t num_list;
	// optional companion of `list`: the neighbour rows gathered in list order, [num_list][27] with slot 13 = the leaf id itself. One
	// dependent load then yields the leaf id AND its neighbours (list -> nbr -> data would be three hops; this is two, like no list).
	const int32_t* list_nbr;
	// optional (sharded runs): bit 8 is set when a semi-Lagrangian sample leaves the 3x3x3 leaf neighbourhood, i.e. may land beyond
	// the shard's ghost layer where the local tree knows nothing about leaves other ranks own
	uint32_t* far_flag;
	__host__ __device__ uint32_t count() const { return list ? num_list : num_leaves; }
#ifdef __CUDACC__
	__device__ __forceinline__ uint32_t leaf_at(uint32_t i) const { return list ? uint32_t(__ldg(list + i)) : i; }
#endif
};

// A packed float4 group of the advection kernels (kernels.cuh, advect.cu; api.cu, "packed groups"): lane k mirrors the brick field
// src[k] (null: the lane holds 0) as it was when the state's version counters stood at vel_version / sc_version.
struct PackedGroup {
	float4* buf = nullptr;  // float4[n], allocated on first use
	const float* src[4] = {};
	uint64_t vel_version = 0, sc_version = 0;
};

// slot ids of the six face neighbours
constexpr int kSlotXm = 4, kSlotXp = 22, kSlotYm = 10, kSlotYp = 16, kSlotZm = 12, kSlotZp = 14, kSlotSelf = 13;

// Position of leaf origin (x, y, z) in NanoVDB's leaf order as a pair compared lexicographically: x = the root tile key with the sign
// bias that makes it increase with signed coordinates, y = upper-node offset << 12 | lower-node offset.
__host__ __device__ inline ulonglong2 nvdb_leaf_key(int32_t x, int32_t y, int32_t z) {
	const uint64_t bx = uint32_t(x) ^ 0x80000000u, by = uint32_t(y) ^ 0x80000000u, bz = uint32_t(z) ^ 0x80000000u;
	const uint64_t tile = (bz >> 12) | (by >> 12) << 21 | (bx >> 12) << 42;
	const uint64_t node = uint64_t(((x & 4095) >> 7) << 10 | ((y & 4095) >> 7) << 5 | ((z & 4095) >> 7)) << 12 |
	                      uint64_t(((x & 127) >> 3) << 8 | ((y & 127) >> 3) << 4 | ((z & 127) >> 3));
	return make_ulonglong2(tile, node);
}
__host__ __device__ inline bool key_less(const ulonglong2& a, const ulonglong2& b) { return a.x < b.x || (a.x == b.x && a.y < b.y); }

// A source grid's leaves on the host, validated and sorted by nvdb_leaf_key (nvdb_io.cu, source_tables): what hns_source_create copies
// to the device. values: float[L][512 * components], each leaf's 512 values as the grid stores them (Vec3f: AoS); masks: uint64[L][8], each
// leaf's value mask (word x, bit y * 8 + z), the source's topology for hns_state_domain_build.
struct SourceTables {
	int components = 0;
	std::vector<ulonglong2> keys;
	std::vector<int4> origins;  // (x, y, z, 0)
	std::vector<float> values;
	std::vector<uint64_t> masks;
};
int source_tables(const void* buffer, uint64_t bytes, SourceTables& out);

#ifdef __CUDACC__
// Leaf ordinal containing voxel (x,y,z), or -1: the ReadAccessor walk (root tile scan -> upper -> lower) on the emitted buffer.
__device__ __forceinline__ int probe_leaf(const GridView& g, int x, int y, int z) {
	const uint8_t* root = g.nvdb + g.off_root;
	const uint64_t key = (uint64_t(uint32_t(z) >> 12)) | (uint64_t(uint32_t(y) >> 12) << 21) | (uint64_t(uint32_t(x) >> 12) << 42);
	const uint8_t* upper = nullptr;
	for (uint32_t t = 0; t < g.num_tiles; ++t) {
		const uint8_t* tile = root + nvdb::kRoot + nvdb::kTile * t;
		if (*reinterpret_cast<const uint64_t*>(tile) == key) {
			upper = root + *reinterpret_cast<const int64_t*>(tile + 8);
			break;
		}
	}
	if (!upper) return -1;
	const uint32_t uo = uint32_t(((x & 4095) >> 7) << 10 | ((y & 4095) >> 7) << 5 | ((z & 4095) >> 7));
	if (!((*reinterpret_cast<const uint64_t*>(upper + nvdb::kUpperChildMask + 8 * (uo >> 6)) >> (uo & 63)) & 1)) return -1;
	const uint8_t* lower = upper + *reinterpret_cast<const int64_t*>(upper + nvdb::kUpperTable + 8ull * uo);
	const uint32_t lo = uint32_t(((x & 127) >> 3) << 8 | ((y & 127) >> 3) << 4 | ((z & 127) >> 3));
	if (!((*reinterpret_cast<const uint64_t*>(lower + nvdb::kLowerChildMask + 8 * (lo >> 6)) >> (lo & 63)) & 1)) return -1;
	const uint8_t* leaf = lower + *reinterpret_cast<const int64_t*>(lower + nvdb::kLowerTable + 8ull * lo);
	return int((leaf - (g.nvdb + g.off_leaf)) / nvdb::kLeaf);
}
#endif

}  // namespace hns

struct hns_mg;
struct hns_state;
namespace hns {
// ghost-exchange fields of a state (api.cu; ids as for hns_state_pack_leaves): the device pointer, or null for a bad id
float* field_ptr(hns_state* s, int field, int* floats_per_leaf);
void field_written(hns_state* s, int field);  // bumps the version counter a write into `field` invalidates
// packed advection groups (api.cu, "packed groups")
void group_wants(const hns_state* s, int j, const float* want[4]);
const float4* group_if_current(const hns_state* s, int j, const float* const want[4]);
void group_written(hns_state* s, int j, const float* const src[4]);
int mg_pressure_solve(hns_state* s, hns_mg* mg, int max_cycles, double rel_tol, int nu_pre, int nu_post, float omega, cudaStream_t st);  // multigrid.cu
void mg_coarse_cycle(hns_mg* mg, float* const rhs1[2], int nu_pre, int nu_post, float omega, cudaStream_t st);
cudaGraphExec_t mg_capture_coarse(hns_mg* mg, float* const rhs1[2], int nu_pre, int nu_post, float omega, uint64_t* launches);
}
// ---- opaque handle definitions ----------------------------------------------------------------------------
struct hns_grid {
	int device = 0;
	float voxel_size = 0.f;
	uint64_t num_leaves = 0, num_lower = 0, num_upper = 0;
	uint64_t nvdb_bytes = 0;
	uint8_t* d_block = nullptr;  // one allocation: [NanoVDB buffer | origins | neighbour table] (topology.cu)
	uint64_t block_bytes = 0;
	uint8_t* d_nvdb = nullptr;
	int4* d_origin = nullptr;
	int32_t* d_nbr = nullptr;
	hns::GridView view{};
};

// multigrid hierarchy (multigrid.cu; a sharded run reads levels >= 1 of a hierarchy over the global grid, dist.cu)
struct hns_mg {
	struct Level {
		hns_grid* grid = nullptr;     // level 0: the caller's grid (borrowed)
		bool own_grid = false;
		float* p[2] = {nullptr, nullptr};    // levels >= 1 (level 0 uses the state's pressure / divergence)
		float* rhs[2] = {nullptr, nullptr};
		float* diag[2] = {nullptr, nullptr};  // colour-split diagonal of the level's operator, 0 = cell outside the domain; null on level 0
		const float* const* diag_or_null() const { return diag[0] ? diag : nullptr; }
		int32_t* parent = nullptr;    // [L] leaf id on the next level; null on the last
		float dx = 0.f;
		uint64_t cells = 0;           // cells inside the domain
	};
	std::vector<Level> lv;
	double* d_sums = nullptr;         // device double[2]
	double* h_sums = nullptr;         // pinned
	uint64_t last_nonempty_count = 0;  // of the last level: non-empty leaves, and (when that is 1) which one
	int64_t last_nonempty_leaf = -1;
	int coarsest_iterations = 32;
	float coarsest_omega = 1.5f;      // a one-leaf last level is solved, not smoothed: SOR near its optimum for 8 cells per axis
	// statistics of the last solve
	int last_cycles = 0;
	double last_rel_residual = -1.0;
	// One V-cycle is ~10 launches per level, most of them on levels far too small to fill the GPU: issued one by one they cost their
	// launch latency (measured: 1.27 of the 2.13 ms of two cycles on the 512^3 workload). The cycle is therefore captured once into a
	// CUDA graph (on a private stream: capture executes nothing) and replayed; the key is everything the captured launches depend on.
	struct CycleGraph {
		cudaGraphExec_t exec = nullptr;
		const void* state = nullptr;
		hns::GridView view{};  // the fine level's view (pointers, counts, work list)
		const void *p = nullptr, *rhs = nullptr;
		int nu_pre = -1, nu_post = -1, coarsest_iterations = -1;
		float omega = 0.f;
		uint64_t launches = 0;
	} graph;
	cudaStream_t capture_stream = nullptr;
	bool use_graph = true;  // HNS_MG_GRAPH=0: issue every launch directly (A/B switch)
};

struct hns_state {
	const hns_grid* grid = nullptr;
	uint64_t n = 0;  // voxels
	int n_scalars = 0;
	float* vel[3] = {};   // current velocity, SoA bricks float[L][512]
	float* adv[3] = {};   // advected velocity
	float* div[2] = {};   // divergence, colour-split: [0] red = (x+y+z) even, [1] black; float[L][256] each
	float* p[2] = {};     // pressure, colour-split like div
	float* sc[16] = {};   // scalar fields (current)
	float* sc_out[16] = {};
	float* aos = nullptr; // staging float[N][3] for host <-> device velocity transfers
	uint8_t* cold = nullptr;  // [L] leaf flags of the advection kernels (advect.cu), zero between launches
	// the packed groups the advection kernels stage from: {u, v, w, first advected scalar} and {fuel, waste, temperature, flame}
	hns::PackedGroup grp[2];
	uint64_t sc_version = 1;  // bumped by every entry point that (may) overwrite a scalar field, like vel_version for the velocity
	float* burn = nullptr;  // float[n], allocated on first use: combustion's burn per voxel from advect_vector to the divergence (api.cu, frame)
	float* vort[4] = {nullptr, nullptr, nullptr, nullptr};  // vorticity confinement scratch, allocated on first use: output planes u, v, w and |curl|
	// optional combustion + buoyancy stage of the all-in-one frame
	bool comb_enabled = false;
	int comb_idx[4] = {-1, -1, -1, -1};  // fuel, waste, temperature, flame
	hns_combustion_params comb{};
	int skip_scalar = -1;  // scalar that is carried but not advected ("collision_sdf")
	bool collision = false;  // hasCollision with collision data: scalar `skip_scalar` is the SDF the kernels collide against
	const float* collision_sdf() const { return collision && skip_scalar >= 0 ? sc[skip_scalar] : nullptr; }
	uint64_t vel_version = 1;  // bumped by every entry point that (may) overwrite the velocity planes; lets a sharded run skip a ghost exchange of unchanged data
	const int32_t* active = nullptr;  // device list of the leaves the kernels process (sharded runs: the owned leaves), null = all
	uint32_t n_active = 0;
	uint32_t* far_flag = nullptr;  // GridView::far_flag
	// optional multigrid pressure solve of the frame (hns_state_set_pressure_solver); null = the reference's fixed-count red-black SOR
	struct hns_mg* mg = nullptr;
	int mg_cycles = 0, mg_nu[2] = {2, 2};
	float mg_omega = 1.0f;
	double* d_sums = nullptr;  // device double[2] of the norm reductions, allocated on first use
	// The reference's solve is 2 x iterations dependent launches; on grids of a few thousand leaves each one is launch latency, not
	// work (4.4 us per launch for 0.9 us of sweep at 1.2 k leaves). The sequence is captured once into a CUDA graph and replayed.
	struct SolveGraph {
		cudaGraphExec_t exec = nullptr;
		hns::GridView view{};  // everything the captured launches depend on: the grid view (pointers, counts, work list) ...
		const void *p = nullptr, *div = nullptr;  // ... the fields ...
		int iterations = -1;                      // ... and the solve's parameters
		unsigned flags = 0;
		float omega = 0.f, dx = 0.f;
		uint64_t launches = 0;
	} solve_graph;
	cudaStream_t capture_stream = nullptr;
	hns::GridView view() const {
		hns::GridView v = grid->view;
		v.list = active, v.num_list = n_active, v.far_flag = far_flag;
		return v;
	}
};

// a source grid on the device (hns_source_create): the host tables of source_tables, copied
struct hns_source {
	int device = 0;
	int components = 0;
	uint64_t num_leaves = 0;
	ulonglong2* keys = nullptr;  // [L], ascending
	int4* origins = nullptr;     // [L]
	float* values = nullptr;     // [L][512 * components]
	uint64_t* masks = nullptr;   // [L][8] value masks
};
