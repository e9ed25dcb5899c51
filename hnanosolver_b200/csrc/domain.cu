// Device-side construction of the simulation domain: which 8^3 leaves the sidecar covers this frame.
//
// Reference: SOP_HNanoSolverVerb::cook builds it on the CPU with OpenVDB every cook (src/SOP/HNanoSolver/SOP_HNanoSolver.cpp:188-199):
//     domain = MaskGrid; domain.topologyUnion(velocity tree)
//     Morphology(domain).dilateVoxels(padding, NN_FACE_EDGE_VERTEX, IGNORE_TILES)
//     if (has_collision && sdf) domain.topologyUnion(sdf tree)
// and IndexGridBuilder then treats every leaf NODE of that tree as a dense brick (src/Utils/GridBuilder.hpp:221-239, LeafManager order).
// So the result is a leaf list: every leaf node of the velocity tree, every leaf an active velocity voxel reaches when it is dilated
// `padding` times with the 26-neighbourhood (= by `padding` in the Chebyshev metric), every leaf node of the SDF tree -- in NanoVDB /
// LeafManager order. With the step itself at a few milliseconds this CPU pass is what a cook would wait for, hence on the device:
//   1. one thread per (velocity leaf, candidate neighbour leaf within ceil(padding / 8) leaves): the candidate is reached iff the leaf's
//      512-bit voxel mask has a bit inside the box of voxels whose +-padding cube overlaps the candidate (three interval tests);
//      reached candidates emit their 63-bit NanoVDB-order key, the others a sentinel
//   2. radix sort (CUB), unique, decode.
// Coordinates are limited to |c| < 2^23 voxels so that root tile, upper and lower offsets of a leaf fit one 64-bit key in NanoVDB order.
// OpenVDB is not vendored with the reference, so this block is pinned to a host restatement (oracle/oracle.py domain_leaves), not to
// OpenVDB itself: PARITY UNPINNED at the OpenVDB boundary (SURVEY.md 8c).
//
// Re-domaining a resident state (hns_state_domain_build, hns_state_create_remapped) runs the same steps on device inputs: the state's
// leaves with the pruned export's masks and keep flags (k_export_classify<3>) and each source's leaves and masks go through step 1 into
// one key array before the single sort (dilation distributes over union); then one launch moves every field onto the new leaves.
#include <cub/cub.cuh>

#include <cmath>
#include <cstring>
#include <vector>

#include "classify.cuh"
#include "common.cuh"

namespace hns {
// named, not anonymous: the anonymous namespace at file scope holds k_export_classify (classify.cuh)
namespace domain {

constexpr int kBias = 1 << 23;
constexpr uint64_t kNoKey = ~uint64_t(0);

// key of the leaf with origin (x, y, z) (multiples of 8): tile (12 bits per axis), upper offset (5 per axis), lower offset (4 per axis)
__host__ __device__ inline uint64_t leaf_key(int x, int y, int z) {
	const uint32_t bx = uint32_t(x + kBias), by = uint32_t(y + kBias), bz = uint32_t(z + kBias);
	const uint64_t tile = (uint64_t(bx >> 12) << 24) | (uint64_t(by >> 12) << 12) | uint64_t(bz >> 12);
	const uint64_t up = (uint64_t((bx >> 7) & 31u) << 10) | (uint64_t((by >> 7) & 31u) << 5) | uint64_t((bz >> 7) & 31u);
	const uint64_t lo = (uint64_t((bx >> 3) & 15u) << 8) | (uint64_t((by >> 3) & 15u) << 4) | uint64_t((bz >> 3) & 15u);
	return (tile << 27) | (up << 12) | lo;
}
__host__ __device__ inline void key_origin(uint64_t k, int* o) {
	const uint32_t lo = uint32_t(k & 4095u), up = uint32_t((k >> 12) & 32767u);
	const uint64_t tile = k >> 27;
	const uint32_t t[3] = {uint32_t((tile >> 24) & 4095u), uint32_t((tile >> 12) & 4095u), uint32_t(tile & 4095u)};
	const uint32_t u[3] = {(up >> 10) & 31u, (up >> 5) & 31u, up & 31u}, l[3] = {(lo >> 8) & 15u, (lo >> 4) & 15u, lo & 15u};
	for (int a = 0; a < 3; ++a) o[a] = int((t[a] << 12) | (u[a] << 7) | (l[a] << 3)) - kBias;
}

// voxels v in [0, 8) of a leaf whose dilation by p reaches the leaf d leaves away along one axis: [lo, hi], empty when lo > hi
__device__ inline void reach(int d, int p, int& lo, int& hi) {
	lo = 0, hi = 7;
	if (d > 0) lo = max(0, 8 * d - p);
	else if (d < 0) hi = min(7, p + 8 * d + 7);
}

// Leaves on the device that take part in a domain: every leaf i with keep[i] != 0 (keep null: every leaf) is a node of the domain whatever
// its mask, and its active voxels dilate. masks: [n][8], word x holds bit (y * 8 + z) (NanoVDB / OpenVDB leaf mask order: bit
// n = x<<6 | y<<3 | z); null = every voxel active.
struct LeafSet {
	const int4* origin;
	const uint64_t* masks;
	const uint32_t* keep;
	uint64_t n;
};

// one thread per (leaf, candidate); the (0, 0, 0) candidate also flags an origin beyond +-(2^23 - 128) in *out_of_range
__global__ void __launch_bounds__(256) k_dilate_candidates(LeafSet s, int padding, int R, uint64_t* __restrict__ keys, uint32_t* out_of_range) {
	const int side = 2 * R + 1, per = side * side * side;
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= s.n * uint64_t(per)) return;
	const uint64_t leaf = t / uint64_t(per);
	const int c = int(t % uint64_t(per));
	const int dx = c / (side * side) - R, dy = (c / side) % side - R, dz = c % side - R;
	const int4 o = __ldg(s.origin + leaf);
	bool hit = (dx | dy | dz) == 0;  // the leaf node itself is part of the domain whatever its mask (topologyUnion copies nodes)
	if (hit && (max(max(o.x, o.y), o.z) >= kBias - 128 || min(min(o.x, o.y), o.z) < -kBias + 128)) atomicOr(out_of_range, 1u);
	if (s.keep && !__ldg(s.keep + leaf)) hit = false;  // a dropped leaf: not a node, nothing to dilate
	else if (!hit) {
		int xl, xh, yl, yh, zl, zh;
		reach(dx, padding, xl, xh), reach(dy, padding, yl, yh), reach(dz, padding, zl, zh);
		if (xl <= xh && yl <= yh && zl <= zh) {
			uint64_t any = 0;
			for (int x = xl; x <= xh; ++x) any |= s.masks ? s.masks[leaf * 8 + x] : ~uint64_t(0);
			uint64_t box = 0;
			const uint64_t zbits = (uint64_t(0xff) >> (7 - zh)) & (uint64_t(0xff) << zl) & 0xffu;
			for (int y = yl; y <= yh; ++y) box |= zbits << (8 * y);
			hit = (any & box) != 0;
		}
	}
	const int X = o.x + 8 * dx, Y = o.y + 8 * dy, Z = o.z + 8 * dz;
	const bool in_range = X >= -kBias && X < kBias && Y >= -kBias && Y < kBias && Z >= -kBias && Z < kBias;
	keys[t] = hit && in_range ? leaf_key(X, Y, Z) : kNoKey;
}
__global__ void __launch_bounds__(256) k_leaf_keys(const int4* __restrict__ origins, uint64_t n, uint64_t* __restrict__ keys) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t < n) {
		const int4 o = __ldg(origins + t);
		keys[t] = leaf_key(o.x, o.y, o.z);
	}
}
__global__ void __launch_bounds__(256) k_decode_keys(const uint64_t* __restrict__ keys, uint64_t n, int32_t* __restrict__ origins) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	int o[3];
	key_origin(keys[t], o);
	origins[3 * t] = o[0], origins[3 * t + 1] = o[1], origins[3 * t + 2] = o[2];
}

// Remap of a state's fields onto a new grid: one warp per new leaf finds the old grid's leaf at its origin once (probe_leaf, the NanoVDB
// walk of the old index buffer), then moves each of the 3 + S planes, 2 KB per leaf, in 128-bit loads and stores: the old leaf's values
// bit for bit, or 512 copies of the plane's fill word where the old grid has no leaf.
struct RemapPlanes {
	const float* src[3 + 16];
	float* dst[3 + 16];
	uint32_t fill[3 + 16];
	int n;
};
__global__ void __launch_bounds__(256) k_remap(GridView old_grid, const int4* __restrict__ origin, uint32_t n_new, RemapPlanes p) {
	const uint32_t leaf = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
	if (leaf >= n_new) return;  // the whole warp
	const int4 o = __ldg(origin + leaf);
	const int j = probe_leaf(old_grid, o.x, o.y, o.z);  // warp-uniform
	for (int f = 0; f < p.n; ++f) {
		float4 v[4];
		if (j >= 0) {
			const float4* src = reinterpret_cast<const float4*>(p.src[f]) + uint64_t(j) * 128u;
#pragma unroll
			for (int k = 0; k < 4; ++k) v[k] = __ldg(src + k * 32 + lane);
		} else {
			const float x = __uint_as_float(p.fill[f]);
#pragma unroll
			for (int k = 0; k < 4; ++k) v[k] = make_float4(x, x, x, x);
		}
		float4* dst = reinterpret_cast<float4*>(p.dst[f]) + uint64_t(leaf) * 128u;
#pragma unroll
		for (int k = 0; k < 4; ++k) dst[k * 32 + lane] = v[k];
	}
}

struct DevBuf {
	void* p = nullptr;
	~DevBuf() { cudaFree(p); }
	template <typename T>
	T* as() {
		return static_cast<T*>(p);
	}
};

int check_origins(const int32_t* o, uint64_t n, const char* what) {
	for (uint64_t i = 0; i < n; ++i)
		for (int a = 0; a < 3; ++a) {
			const int32_t c = o[3 * i + a];
			if (c & 7) return fail(HNS_ERR_TOPOLOGY, std::string(what) + ": leaf origin is not a multiple of 8");
			if (c < -kBias + 128 || c >= kBias - 128) return fail(HNS_ERR_UNSUPPORTED, std::string(what) + ": leaf origin beyond +-(2^23 - 128) voxels");
		}
	return HNS_OK;
}

// host int32[n][3] -> device int4[n] in `buf`
cudaError_t upload_origins(const int32_t* o, uint64_t n, DevBuf& buf) {
	std::vector<int4> h(n);
	for (uint64_t i = 0; i < n; ++i) h[i] = make_int4(o[3 * i], o[3 * i + 1], o[3 * i + 2], 0);
	cudaError_t e = cudaMalloc(&buf.p, n * sizeof(int4));
	return e == cudaSuccess ? cudaMemcpy(buf.p, h.data(), n * sizeof(int4), cudaMemcpyHostToDevice) : e;
}

// The device part of every domain build: each set through the candidate kernel and the collider's leaves through k_leaf_keys into one
// key array (dilation distributes over union), one radix sort, unique, decode; the result in NanoVDB order. Synchronous (the count is
// read back). HNS_ERR_UNSUPPORTED when a set holds an origin beyond +-(2^23 - 128) voxels.
int build_leaves(const std::vector<LeafSet>& sets, int padding, const int4* d_sdf, uint64_t n_sdf, std::vector<int32_t>& origins) {
	const int R = (padding + 7) / 8, side = 2 * R + 1;
	const uint64_t per = uint64_t(side) * side * side;
	uint64_t n_keys = n_sdf;
	for (const LeafSet& s : sets) n_keys += s.n * per;
	origins.clear();
	if (!n_keys) return HNS_OK;
	DevBuf d_keys, d_sorted, d_unique, d_count, d_tmp, d_out;
	HNS_CUDA(cudaMalloc(&d_keys.p, n_keys * 8));
	HNS_CUDA(cudaMalloc(&d_sorted.p, n_keys * 8));
	HNS_CUDA(cudaMalloc(&d_unique.p, n_keys * 8));
	HNS_CUDA(cudaMalloc(&d_count.p, 16));  // [unique count, out-of-range flag]
	HNS_CUDA(cudaMemset(d_count.p, 0, 16));
	uint32_t* d_flag = reinterpret_cast<uint32_t*>(d_count.as<uint64_t>() + 1);
	uint64_t at = 0;
	for (const LeafSet& s : sets) {
		if (!s.n) continue;
		const uint64_t threads = s.n * per;
		HNS_LAUNCH(k_dilate_candidates, unsigned((threads + 255) / 256), 256, 0, 0, s, padding, R, d_keys.as<uint64_t>() + at, d_flag);
		at += threads;
	}
	if (n_sdf) HNS_LAUNCH(k_leaf_keys, unsigned((n_sdf + 255) / 256), 256, 0, 0, d_sdf, n_sdf, d_keys.as<uint64_t>() + at);
	size_t tmp_sort = 0, tmp_unique = 0;
	HNS_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_sort, d_keys.as<uint64_t>(), d_sorted.as<uint64_t>(), n_keys, 0, 64));
	HNS_CUDA(cub::DeviceSelect::Unique(nullptr, tmp_unique, d_sorted.as<uint64_t>(), d_unique.as<uint64_t>(), d_count.as<uint64_t>(), n_keys));
	HNS_CUDA(cudaMalloc(&d_tmp.p, std::max(tmp_sort, tmp_unique) + 16));
	HNS_CUDA(cub::DeviceRadixSort::SortKeys(d_tmp.p, tmp_sort, d_keys.as<uint64_t>(), d_sorted.as<uint64_t>(), n_keys, 0, 64));
	HNS_CUDA(cub::DeviceSelect::Unique(d_tmp.p, tmp_unique, d_sorted.as<uint64_t>(), d_unique.as<uint64_t>(), d_count.as<uint64_t>(), n_keys));
	uint64_t head[2] = {0, 0};
	HNS_CUDA(cudaMemcpy(head, d_count.p, 16, cudaMemcpyDeviceToHost));
	if (head[1]) return fail(HNS_ERR_UNSUPPORTED, "leaf origin beyond +-(2^23 - 128) voxels");
	uint64_t n_unique = head[0];
	if (n_unique) {  // the sentinel sorts last
		uint64_t last = 0;
		HNS_CUDA(cudaMemcpy(&last, d_unique.as<uint64_t>() + (n_unique - 1), 8, cudaMemcpyDeviceToHost));
		if (last == kNoKey) --n_unique;
	}
	origins.resize(3 * n_unique);
	if (n_unique) {
		HNS_CUDA(cudaMalloc(&d_out.p, n_unique * 12));
		HNS_LAUNCH(k_decode_keys, unsigned((n_unique + 255) / 256), 256, 0, 0, d_unique.as<uint64_t>(), n_unique, d_out.as<int32_t>());
		HNS_CUDA(cudaMemcpy(origins.data(), d_out.p, n_unique * 12, cudaMemcpyDeviceToHost));
	}
	return HNS_OK;
}

}  // namespace domain
}  // namespace hns

using namespace hns;
using namespace hns::domain;

struct hns_domain {
	std::vector<int32_t> origins;  // [L][3], NanoVDB order
};

extern "C" {

void hns_domain_destroy(hns_domain* d) { delete d; }
uint64_t hns_domain_num_leaves(const hns_domain* d) { return d ? d->origins.size() / 3 : 0; }
int hns_domain_origins(const hns_domain* d, int32_t* origins_out) {
	if (!d || (!origins_out && !d->origins.empty())) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	if (!d->origins.empty()) std::memcpy(origins_out, d->origins.data(), d->origins.size() * sizeof(int32_t));
	return HNS_OK;
}
int hns_domain_create_grid(const hns_domain* d, float voxel_size, hns_grid** out) {
	if (!d) return fail(HNS_ERR_INVALID_ARGUMENT, "null domain");
	return hns_grid_create_from_origins(d->origins.data(), d->origins.size() / 3, voxel_size, out);
}

int hns_domain_build(const int32_t* vel_origins, const uint64_t* vel_masks, uint64_t n_vel, int padding, const int32_t* sdf_origins, uint64_t n_sdf,
                     hns_domain** out) {
	if (!out) return fail(HNS_ERR_INVALID_ARGUMENT, "out is null");
	*out = nullptr;
	if ((n_vel && !vel_origins) || (n_sdf && !sdf_origins)) return fail(HNS_ERR_INVALID_ARGUMENT, "null origins");
	if (padding < 0 || padding > 64) return fail(HNS_ERR_INVALID_ARGUMENT, "padding must be in [0, 64] voxels");
	int rc;
	if ((rc = check_origins(vel_origins, n_vel, "velocity topology"))) return rc;
	if ((rc = check_origins(sdf_origins, n_sdf, "sdf topology"))) return rc;
	DevBuf d_org, d_mask, d_sorg;
	std::vector<LeafSet> sets;
	if (n_vel) {
		HNS_CUDA(upload_origins(vel_origins, n_vel, d_org));
		if (vel_masks) {
			HNS_CUDA(cudaMalloc(&d_mask.p, n_vel * 64));
			HNS_CUDA(cudaMemcpy(d_mask.p, vel_masks, n_vel * 64, cudaMemcpyHostToDevice));
		}
		sets.push_back(LeafSet{d_org.as<int4>(), d_mask.as<uint64_t>(), nullptr, n_vel});
	}
	if (n_sdf) HNS_CUDA(upload_origins(sdf_origins, n_sdf, d_sorg));
	auto* dom = new hns_domain();
	if ((rc = build_leaves(sets, padding, d_sorg.as<int4>(), n_sdf, dom->origins))) {
		delete dom;
		return rc;
	}
	*out = dom;
	return HNS_OK;
}

int hns_state_domain_build(const hns_state* s, float tolerance, int padding, int n_sources, const hns_source* const* sources, const int32_t* sdf_origins,
                           uint64_t n_sdf, hns_domain** out) {
	if (!out) return fail(HNS_ERR_INVALID_ARGUMENT, "out is null");
	*out = nullptr;
	if (std::isnan(tolerance)) return fail(HNS_ERR_INVALID_ARGUMENT, "the tolerance is NaN");
	if (padding < 0 || padding > 64) return fail(HNS_ERR_INVALID_ARGUMENT, "padding must be in [0, 64] voxels");
	if (!s || n_sources < 0 || (n_sources && !sources) || (n_sdf && !sdf_origins)) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	for (int i = 0; i < n_sources; ++i)
		if (!sources[i]) return fail(HNS_ERR_INVALID_ARGUMENT, "null source entry");
	int rc;
	if ((rc = check_origins(sdf_origins, n_sdf, "sdf topology"))) return rc;
	if (s->active) return fail(HNS_ERR_UNSUPPORTED, "a sharded state (hns_dist_set_plan) cannot be re-domained");
	for (int i = 0; i < n_sources; ++i)
		if (sources[i]->device != s->grid->device) return fail(HNS_ERR_INVALID_ARGUMENT, "a source lives on another device than the state");
	const uint64_t L = s->grid->num_leaves;
	DevBuf d_masks, d_keep, d_sorg;
	std::vector<LeafSet> sets;
	if (L) {  // the velocity's topology as hns_state_export_velocity(s, tolerance) writes it
		LeafSet v{s->grid->view.origin, nullptr, nullptr, L};
		if (tolerance >= 0.0f) {
			HNS_CUDA(cudaMalloc(&d_masks.p, L * 64));
			HNS_CUDA(cudaMalloc(&d_keep.p, L * 4));
			HNS_LAUNCH(k_export_classify<3>, unsigned((L + 7) / 8), 256, 0, 0, s->vel[0], s->vel[1], s->vel[2], nullptr, uint32_t(L), tolerance,
			           d_masks.as<uint64_t>(), d_keep.as<uint32_t>());
			v.masks = d_masks.as<uint64_t>(), v.keep = d_keep.as<uint32_t>();
		}
		sets.push_back(v);
	}
	for (int i = 0; i < n_sources; ++i) sets.push_back(LeafSet{sources[i]->origins, sources[i]->masks, nullptr, sources[i]->num_leaves});
	if (n_sdf) HNS_CUDA(upload_origins(sdf_origins, n_sdf, d_sorg));
	auto* dom = new hns_domain();
	if ((rc = build_leaves(sets, padding, d_sorg.as<int4>(), n_sdf, dom->origins))) {
		delete dom;
		return rc;
	}
	*out = dom;
	return HNS_OK;
}

int hns_state_create_remapped(const hns_state* src, const hns_grid* g, void* stream, hns_state** out) {
	if (!src || !g || !out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	*out = nullptr;
	if (src->active) return fail(HNS_ERR_UNSUPPORTED, "a sharded state (hns_dist_set_plan) cannot be re-domained");
	if (g->device != src->grid->device) return fail(HNS_ERR_INVALID_ARGUMENT, "the grid lives on another device than the state");
	hns_state* s = nullptr;
	int rc = hns_state_create(g, src->n_scalars, &s);
	if (rc) return rc;
	// the configuration that does not depend on the grid; a multigrid hierarchy does, so the new state solves red-black
	s->comb_enabled = src->comb_enabled;
	std::copy(src->comb_idx, src->comb_idx + 4, s->comb_idx);
	s->comb = src->comb;
	s->skip_scalar = src->skip_scalar, s->collision = src->collision;
	const cudaStream_t st = static_cast<cudaStream_t>(stream);
	cudaError_t e = cudaSuccess;
	if (g->num_leaves) {
		RemapPlanes p{};
		for (int c = 0; c < 3; ++c) p.src[c] = src->vel[c], p.dst[c] = s->vel[c];
		for (int i = 0; i < src->n_scalars; ++i)  // new leaves: bytes 0, or 0x01 for the collision SDF (GridBuilder.hpp:108)
			p.src[3 + i] = src->sc[i], p.dst[3 + i] = s->sc[i], p.fill[3 + i] = i == src->skip_scalar ? 0x01010101u : 0u;
		p.n = 3 + src->n_scalars;
		// hns_state_create zeroes the fields on the legacy default stream: the remap's stores go after those
		cudaEvent_t zeroed = nullptr;
		if ((e = cudaEventCreateWithFlags(&zeroed, cudaEventDisableTiming)) == cudaSuccess && (e = cudaEventRecord(zeroed, 0)) == cudaSuccess)
			e = cudaStreamWaitEvent(st, zeroed, 0);
		if (zeroed) cudaEventDestroy(zeroed);
		if (e == cudaSuccess) {
			HNS_LAUNCH(k_remap, unsigned((g->num_leaves + 7) / 8), 256, 0, st, src->grid->view, g->view.origin, uint32_t(g->num_leaves), p);
			e = cudaGetLastError();
		}
	}
	if (e != cudaSuccess) {
		hns_state_destroy(s);
		return fail(HNS_ERR_CUDA, std::string("hns_state_create_remapped: ") + cudaGetErrorString(e));
	}
	field_written(s, 0);
	if (s->n_scalars) field_written(s, 10);
	*out = s;
	return HNS_OK;
}

}  // extern "C"
