// Export of resident fields as NanoVDB float / Vec3f grids built on the device (include/hns_b200.h, "Export"): writeIndexGrid
// (reference src/Utils/GridBuilder.hpp:168-216) without the download, whole-domain or pruned to a tolerance. The bytes are those of the
// host writer hns_sidecar_to_nanovdb (nvdb_io.cu) over the kept leaves, which tests/test_export.py checks byte for byte.
//
// The state's leaves are NanoVDB-ordered 8^3 bricks, so the output tree is the state's own, or an ordered subset of it:
//   classify  (pruned only) one warp per listed leaf: active-voxel masks and a keep flag
//   select    the kept leaves in list order (an exclusive scan of the keep flags, then a scatter)
//   number    per kept leaf: "new root tile" / "new lower node" against the previous kept leaf (the host writer's tests), the root bbox
//             and the active-voxel count (integer atomics: deterministic); inclusive scans of the two flags give every kept leaf its
//             upper and lower node
//   -- one readback of the counts; the header (GridData, TreeData, root) is written on the host by the host writer's own function --
//   leaves    one warp per kept leaf writes the whole leaf record (the hot path, at copy rate), lane 0 links it into its lower node
//             and, for a node's first leaf, the lower node into its upper node and the upper node into its root tile
//   bboxes    lower nodes over their leaves, upper nodes over their lower nodes: min / max over contiguous children
#include <cmath>
#include <cstring>
#include <string>

#include <cub/cub.cuh>

#include "classify.cuh"
#include "common.cuh"
#include "nvdb_layout.cuh"

using namespace hns;
using namespace hns::vgrid;

namespace {

// what the pre-readback kernels leave for the host; zeroed before each export. The bbox is stored order-preserving as unsigned so
// that zero is the neutral element of both atomicMax's: lo_enc = ~(x ^ 0x80000000) (max of it = min of x), hi_enc = x ^ 0x80000000.
struct Summary {
	uint32_t kept, lower, upper, pad;
	uint32_t lo_enc[3], hi_enc[3];
	unsigned long long active;
};

struct Tables {             // device scratch, per listed leaf
	uint32_t* keep;         // [n] classify's keep flag
	uint32_t* pos;          // [n] exclusive sum of keep: the kept leaf's rank
	uint64_t* masks;        // [n][8] classify's masks (null: whole domain, every voxel active)
	uint32_t* kept;         // [n] list positions of the kept leaves (null: whole domain, every listed leaf kept)
	uint32_t* tflag;        // [n] per kept leaf: starts a new root tile (= upper node)
	uint32_t* lflag;        // [n] per kept leaf: starts a new lower node (a new tile does)
	uint32_t* tscan;        // [n] inclusive sums of tflag / lflag: upper / lower node index + 1
	uint32_t* lscan;
	uint32_t* lower_first;  // [nLower] first kept leaf of each lower node
	uint32_t* upper_first;  // [T] first lower node of each upper node
};

__device__ __forceinline__ uint32_t leaf_of(const int32_t* list, const uint32_t* kept, uint32_t j) {
	const uint32_t i = kept ? __ldg(kept + j) : j;
	return list ? uint32_t(__ldg(list + i)) : i;
}

// ---- classify: k_export_classify (classify.cuh), one warp per listed leaf

__global__ void __launch_bounds__(256) k_export_scatter(const uint32_t* __restrict__ keep, const uint32_t* __restrict__ pos, uint32_t n,
                                                        uint32_t* __restrict__ kept, Summary* sum) {
	const uint32_t i = blockIdx.x * 256u + threadIdx.x;
	if (i >= n) return;
	const uint32_t k = keep[i], p = pos[i];
	if (k) kept[p] = i;
	if (i == n - 1) sum->kept = p + k;
}

// ---- number: one thread per kept leaf (nk = sum->kept when selected, else n)
__global__ void __launch_bounds__(256) k_export_number(const int4* __restrict__ origin, const int32_t* __restrict__ list, Tables t, uint32_t n,
                                                       Summary* sum) {
	const uint32_t j = blockIdx.x * 256u + threadIdx.x, lane = threadIdx.x & 31u;
	const uint32_t nk = t.kept ? sum->kept : n;
	const bool valid = j < nk;
	int4 o = make_int4(INT32_MAX, INT32_MAX, INT32_MAX, 0);
	uint32_t active = 0;
	if (valid) {
		const uint32_t i = t.kept ? t.kept[j] : j;
		o = __ldg(origin + (list ? __ldg(list + i) : int32_t(i)));
		bool newTile = j == 0, newLower = j == 0;
		if (j) {
			const int4 p = __ldg(origin + leaf_of(list, t.kept, j - 1));
			newTile = (o.x >> 12) != (p.x >> 12) || (o.y >> 12) != (p.y >> 12) || (o.z >> 12) != (p.z >> 12);
			newLower = newTile || (o.x >> 7) != (p.x >> 7) || (o.y >> 7) != (p.y >> 7) || (o.z >> 7) != (p.z >> 7);
		}
		t.tflag[j] = newTile, t.lflag[j] = newLower;
		if (t.masks) {
			const uint64_t* m = t.masks + uint64_t(i) * 8u;
#pragma unroll
			for (int w = 0; w < 8; ++w) active += __popcll(m[w]);
		} else {
			active = 512;
		}
	} else if (j < n) {
		t.tflag[j] = t.lflag[j] = 0;
	}
	const uint32_t warp_active = __reduce_add_sync(0xffffffffu, active);
	const int lo[3] = {__reduce_min_sync(0xffffffffu, o.x), __reduce_min_sync(0xffffffffu, o.y), __reduce_min_sync(0xffffffffu, o.z)};
	const int hx = valid ? o.x + 7 : INT32_MIN, hy = valid ? o.y + 7 : INT32_MIN, hz = valid ? o.z + 7 : INT32_MIN;
	const int hi[3] = {__reduce_max_sync(0xffffffffu, hx), __reduce_max_sync(0xffffffffu, hy), __reduce_max_sync(0xffffffffu, hz)};
	if (lane == 0 && warp_active) {
		atomicAdd(&sum->active, (unsigned long long)warp_active);
		for (int d = 0; d < 3; ++d) {
			atomicMax(&sum->lo_enc[d], ~(uint32_t(lo[d]) ^ 0x80000000u));
			atomicMax(&sum->hi_enc[d], uint32_t(hi[d]) ^ 0x80000000u);
		}
	}
}

__global__ void k_export_counts(Tables t, uint32_t n, Summary* sum) {
	const uint32_t nk = t.kept ? sum->kept : n;
	sum->kept = nk;
	sum->upper = nk ? t.tscan[nk - 1] : 0, sum->lower = nk ? t.lscan[nk - 1] : 0;
}

struct Out {
	uint8_t* buf;
	uint64_t root, upper, lower, leaf;  // offsets (GridOffsets)
};

// ---- leaves: one warp per kept leaf. Header (16 B per lane, lanes 0 .. H/16 - 1): bboxMin, bboxDif 7,7,7, flags 0x02 (bbox valid),
// value mask, then zeroed statistics and padding. Values: a float leaf is a 2 KB copy; a Vec3f leaf turns the three SoA planes into AoS,
// per quad of voxels three float4 loads into three float4 stores (the inverse of k_add_source<3>). Leaf records start 32-byte aligned
// and their values 16-byte aligned: every node size is a multiple of 32.
template <int C>
__global__ void __launch_bounds__(256) k_export_leaves(const float* f0, const float* f1, const float* f2, const int4* __restrict__ origin,
                                                       const int32_t* __restrict__ list, Tables t, uint32_t nk, Out out) {
	constexpr ValueLayout lay = C == 1 ? kFloatLayout : kVec3fLayout;
	const uint32_t j = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
	if (j >= nk) return;  // the whole warp
	const uint32_t i = t.kept ? __ldg(t.kept + j) : j;
	const uint32_t leaf = list ? uint32_t(__ldg(list + i)) : i;
	const int4 o = __ldg(origin + leaf);
	uint8_t* F = out.buf + out.leaf + lay.leaf * uint64_t(j);
	const float4* plane[3] = {reinterpret_cast<const float4*>(f0) + uint64_t(leaf) * 128u, reinterpret_cast<const float4*>(f1) + uint64_t(leaf) * 128u,
	                          reinterpret_cast<const float4*>(f2) + uint64_t(leaf) * 128u};
	float4* dst = reinterpret_cast<float4*>(F + lay.leaf_values);
#pragma unroll
	for (int k = 0; k < 4; ++k) {
		const uint32_t q = k * 32 + lane;
		if constexpr (C == 1) {
			dst[q] = __ldg(plane[0] + q);
		} else {  // voxels 4q .. 4q+3 -> (x0 y0 z0 x1) (y1 z1 x2 y2) (z2 x3 y3 z3)
			const float4 x = __ldg(plane[0] + q), y = __ldg(plane[1] + q), z = __ldg(plane[2] + q);
			dst[3 * q] = make_float4(x.x, y.x, z.x, x.y);
			dst[3 * q + 1] = make_float4(y.y, z.y, x.z, y.z);
			dst[3 * q + 2] = make_float4(z.z, x.w, y.w, z.w);
		}
	}
	if (lane < lay.leaf_values / 16) {
		uint4 h = make_uint4(0u, 0u, 0u, 0u);
		if (lane == 0) {
			h = make_uint4(uint32_t(o.x), uint32_t(o.y), uint32_t(o.z), 0x02070707u);
		} else if (lane <= 4) {
			if (t.masks) {
				const ulonglong2 m = __ldg(reinterpret_cast<const ulonglong2*>(t.masks + uint64_t(i) * 8u) + (lane - 1));
				h = make_uint4(uint32_t(m.x), uint32_t(m.x >> 32), uint32_t(m.y), uint32_t(m.y >> 32));
			} else {
				h = make_uint4(~0u, ~0u, ~0u, ~0u);
			}
		}
		reinterpret_cast<uint4*>(F)[lane] = h;
	}
	if (lane == 0) {  // the links: the node regions were zeroed, child-mask words are shared with siblings
		const uint32_t iu = __ldg(t.tscan + j) - 1u, il = __ldg(t.lscan + j) - 1u;
		uint8_t* R = out.buf + out.root;
		uint8_t* U = out.buf + out.upper + lay.upper * uint64_t(iu);
		uint8_t* Lo = out.buf + out.lower + lay.lower * uint64_t(il);
		const uint32_t lo = uint32_t(((o.x & 127) >> 3) << 8 | ((o.y & 127) >> 3) << 4 | ((o.z & 127) >> 3));
		atomicOr(reinterpret_cast<unsigned long long*>(Lo + kLowerChildMask) + (lo >> 6), 1ull << (lo & 63));
		*reinterpret_cast<int64_t*>(Lo + lay.lower_table + lay.table_stride * lo) = int64_t(F - Lo);
		if (__ldg(t.lflag + j)) {
			t.lower_first[il] = j;
			const uint32_t uo = uint32_t(((o.x & 4095) >> 7) << 10 | ((o.y & 4095) >> 7) << 5 | ((o.z & 4095) >> 7));
			atomicOr(reinterpret_cast<unsigned long long*>(U + kUpperChildMask) + (uo >> 6), 1ull << (uo & 63));
			*reinterpret_cast<int64_t*>(U + lay.upper_table + lay.table_stride * uo) = int64_t(Lo - U);
		}
		if (__ldg(t.tflag + j)) {
			t.upper_first[iu] = il;
			uint8_t* tile = R + lay.root + lay.tile * uint64_t(iu);
			*reinterpret_cast<uint64_t*>(tile) = uint64_t(uint32_t(o.z) >> 12) | uint64_t(uint32_t(o.y) >> 12) << 21 | uint64_t(uint32_t(o.x) >> 12) << 42;
			*reinterpret_cast<int64_t*>(tile + 8) = int64_t(U - R);
		}
	}
}

// ---- bboxes: one warp per node over its children [first[node], first[node + 1]) (the last node's end: n_children)
__device__ __forceinline__ void store_box(uint8_t* node, int lo[3], int hi[3], uint32_t lane) {
	for (int d = 0; d < 3; ++d) lo[d] = __reduce_min_sync(0xffffffffu, lo[d]), hi[d] = __reduce_max_sync(0xffffffffu, hi[d]);
	if (lane < 3) reinterpret_cast<int32_t*>(node)[lane] = lane == 0 ? lo[0] : lane == 1 ? lo[1] : lo[2];
	else if (lane < 6) reinterpret_cast<int32_t*>(node)[lane] = lane == 3 ? hi[0] : lane == 4 ? hi[1] : hi[2];
}
template <int C>
__global__ void __launch_bounds__(256) k_export_lower_bbox(const int4* __restrict__ origin, const int32_t* __restrict__ list, Tables t,
                                                           uint32_t nLower, uint32_t nk, Out out) {
	constexpr ValueLayout lay = C == 1 ? kFloatLayout : kVec3fLayout;
	const uint32_t il = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
	if (il >= nLower) return;
	const uint32_t b = t.lower_first[il], e = il + 1 < nLower ? t.lower_first[il + 1] : nk;
	int lo[3] = {INT32_MAX, INT32_MAX, INT32_MAX}, hi[3] = {INT32_MIN, INT32_MIN, INT32_MIN};
	for (uint32_t j = b + lane; j < e; j += 32) {
		const int4 o = __ldg(origin + leaf_of(list, t.kept, j));
		lo[0] = min(lo[0], o.x), lo[1] = min(lo[1], o.y), lo[2] = min(lo[2], o.z);
		hi[0] = max(hi[0], o.x + 7), hi[1] = max(hi[1], o.y + 7), hi[2] = max(hi[2], o.z + 7);
	}
	store_box(out.buf + out.lower + lay.lower * uint64_t(il), lo, hi, lane);
}
template <int C>
__global__ void __launch_bounds__(256) k_export_upper_bbox(Tables t, uint32_t T, uint32_t nLower, Out out) {
	constexpr ValueLayout lay = C == 1 ? kFloatLayout : kVec3fLayout;
	const uint32_t iu = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
	if (iu >= T) return;
	const uint32_t b = t.upper_first[iu], e = iu + 1 < T ? t.upper_first[iu + 1] : nLower;
	int lo[3] = {INT32_MAX, INT32_MAX, INT32_MAX}, hi[3] = {INT32_MIN, INT32_MIN, INT32_MIN};
	for (uint32_t il = b + lane; il < e; il += 32) {
		const int32_t* box = reinterpret_cast<const int32_t*>(out.buf + out.lower + lay.lower * uint64_t(il));
		for (int d = 0; d < 3; ++d) lo[d] = min(lo[d], box[d]), hi[d] = max(hi[d], box[3 + d]);
	}
	store_box(out.buf + out.upper + lay.upper * uint64_t(iu), lo, hi, lane);
}

uint64_t align256(uint64_t b) { return (b + 255) & ~uint64_t(255); }

}  // namespace

// a NanoVDB float / Vec3f grid in device memory (hns_state_export_*), with the scratch its exports need; both only grow
struct hns_value_grid {
	int device = -1;  // bound by the first export
	uint8_t* d_buf = nullptr;
	uint64_t capacity = 0, bytes = 0, num_leaves = 0;
	uint8_t* d_scratch = nullptr;
	uint64_t scratch_bytes = 0;
	Summary* h_sum = nullptr;  // pinned
};

namespace {

int export_field(hns_state* s, const float* const planes[3], int C, float tolerance, const char* name, hns_value_grid* vg, cudaStream_t st) {
	const ValueLayout& lay = *value_layout(C);
	const bool pruned = tolerance >= 0.0f;
	const uint32_t n = s->active ? s->n_active : uint32_t(s->grid->num_leaves);
	const int32_t* list = s->active;
	const int4* origin = s->grid->view.origin;
	// scratch: [Summary | 9 uint32 tables of n | masks | cub temp]
	size_t tmp_scan = 0, tmp_ex = 0;
	if (n) {
		HNS_CUDA(cub::DeviceScan::InclusiveSum(nullptr, tmp_scan, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), int(n), st));
		HNS_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_ex, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), int(n), st));
	}
	const uint64_t table = align256(uint64_t(n) * 4), o_tables = align256(sizeof(Summary)), o_masks = o_tables + 9 * table,
	               o_tmp = o_masks + align256(uint64_t(n) * 64), need = o_tmp + align256(std::max(tmp_scan, tmp_ex));
	if (vg->scratch_bytes < need) {
		cudaFree(vg->d_scratch);
		vg->d_scratch = nullptr, vg->scratch_bytes = 0;
		HNS_CUDA(cudaMalloc(&vg->d_scratch, need));
		vg->scratch_bytes = need;
	}
	if (!vg->h_sum) HNS_CUDA(cudaMallocHost(&vg->h_sum, sizeof(Summary)));
	uint8_t* sc = vg->d_scratch;
	Summary* d_sum = reinterpret_cast<Summary*>(sc);
	auto u32 = [&](int k) { return reinterpret_cast<uint32_t*>(sc + o_tables + k * table); };
	Tables t{u32(0), u32(1), pruned ? reinterpret_cast<uint64_t*>(sc + o_masks) : nullptr, pruned ? u32(2) : nullptr, u32(3), u32(4), u32(5), u32(6), u32(7), u32(8)};
	HNS_CUDA(cudaMemsetAsync(d_sum, 0, sizeof(Summary), st));
	if (n) {
		const unsigned warps = (n + 7u) / 8u, threads = (n + 255u) / 256u;
		if (pruned) {
			if (C == 3) HNS_LAUNCH(k_export_classify<3>, warps, 256, 0, st, planes[0], planes[1], planes[2], list, n, tolerance, t.masks, t.keep);
			else HNS_LAUNCH(k_export_classify<1>, warps, 256, 0, st, planes[0], planes[0], planes[0], list, n, tolerance, t.masks, t.keep);
			size_t b = tmp_ex;
			HNS_CUDA(cub::DeviceScan::ExclusiveSum(sc + o_tmp, b, t.keep, t.pos, int(n), st));
			HNS_LAUNCH(k_export_scatter, threads, 256, 0, st, t.keep, t.pos, n, t.kept, d_sum);
		}
		HNS_LAUNCH(k_export_number, threads, 256, 0, st, origin, list, t, n, d_sum);
		size_t b = tmp_scan;
		HNS_CUDA(cub::DeviceScan::InclusiveSum(sc + o_tmp, b, t.tflag, t.tscan, int(n), st));
		b = tmp_scan;
		HNS_CUDA(cub::DeviceScan::InclusiveSum(sc + o_tmp, b, t.lflag, t.lscan, int(n), st));
		HNS_LAUNCH(k_export_counts, 1, 1, 0, st, t, n, d_sum);
	}
	HNS_CUDA(cudaMemcpyAsync(vg->h_sum, d_sum, sizeof(Summary), cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	const Summary sum = *vg->h_sum;
	const uint32_t nk = n ? sum.kept : 0, nLower = sum.lower, T = sum.upper;
	const GridOffsets off(lay, nk, nLower, T);
	if (vg->capacity < off.end) {
		cudaFree(vg->d_buf);
		vg->d_buf = nullptr, vg->capacity = vg->bytes = vg->num_leaves = 0;
		HNS_CUDA(cudaMalloc(&vg->d_buf, off.end));
		vg->capacity = off.end;
	}
	int32_t lo[3], hi[3];
	for (int d = 0; d < 3; ++d) lo[d] = int32_t(~sum.lo_enc[d] ^ 0x80000000u), hi[d] = int32_t(sum.hi_enc[d] ^ 0x80000000u);
	const uint64_t head = off.root + lay.root;
	std::vector<uint8_t> h(head, 0);
	write_grid_header(h.data(), lay, nk, nLower, T, s->grid->voxel_size, name, lo, hi, sum.active);
	HNS_CUDA(cudaMemcpyAsync(vg->d_buf, h.data(), head, cudaMemcpyHostToDevice, st));
	HNS_CUDA(cudaMemsetAsync(vg->d_buf + head, 0, off.leaf - head, st));
	if (nk) {
		const Out out{vg->d_buf, off.root, off.upper, off.lower, off.leaf};
		if (C == 3) {
			HNS_LAUNCH(k_export_leaves<3>, (nk + 7u) / 8u, 256, 0, st, planes[0], planes[1], planes[2], origin, list, t, nk, out);
			HNS_LAUNCH(k_export_lower_bbox<3>, (nLower + 7u) / 8u, 256, 0, st, origin, list, t, nLower, nk, out);
			HNS_LAUNCH(k_export_upper_bbox<3>, (T + 7u) / 8u, 256, 0, st, t, T, nLower, out);
		} else {
			HNS_LAUNCH(k_export_leaves<1>, (nk + 7u) / 8u, 256, 0, st, planes[0], planes[0], planes[0], origin, list, t, nk, out);
			HNS_LAUNCH(k_export_lower_bbox<1>, (nLower + 7u) / 8u, 256, 0, st, origin, list, t, nLower, nk, out);
			HNS_LAUNCH(k_export_upper_bbox<1>, (T + 7u) / 8u, 256, 0, st, t, T, nLower, out);
		}
	}
	HNS_CUDA(cudaGetLastError());
	HNS_CUDA(cudaStreamSynchronize(st));  // also keeps `h` alive until its copy has run
	vg->device = s->grid->device, vg->bytes = off.end, vg->num_leaves = nk;
	return HNS_OK;
}

int check_export(const hns_state* s, float tolerance, const char* name, const hns_value_grid* vg) {
	if (std::isnan(tolerance)) return fail(HNS_ERR_INVALID_ARGUMENT, "the tolerance is NaN");
	if (!s || !name || !vg) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	if (vg->device >= 0 && vg->device != s->grid->device) return fail(HNS_ERR_INVALID_ARGUMENT, "the value grid lives on another device than the state");
	return HNS_OK;
}

}  // namespace

extern "C" {

int hns_value_grid_create(hns_value_grid** out) {
	if (!out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	*out = new hns_value_grid();
	return HNS_OK;
}
void hns_value_grid_destroy(hns_value_grid* vg) {
	if (!vg) return;
	cudaFree(vg->d_buf), cudaFree(vg->d_scratch);
	if (vg->h_sum) cudaFreeHost(vg->h_sum);
	delete vg;
}
uint64_t hns_value_grid_bytes(const hns_value_grid* vg) { return vg ? vg->bytes : 0; }
uint64_t hns_value_grid_num_leaves(const hns_value_grid* vg) { return vg ? vg->num_leaves : 0; }
const void* hns_value_grid_device_ptr(const hns_value_grid* vg) { return vg && vg->bytes ? vg->d_buf : nullptr; }
int hns_value_grid_download(const hns_value_grid* vg, void* dst_host, uint64_t capacity) {
	if (!vg || (!dst_host && vg->bytes)) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	if (capacity < vg->bytes) return fail(HNS_ERR_INVALID_ARGUMENT, "destination buffer is too small");
	if (vg->bytes) HNS_CUDA(cudaMemcpy(dst_host, vg->d_buf, vg->bytes, cudaMemcpyDeviceToHost));
	return HNS_OK;
}

int hns_state_export_velocity(hns_state* s, float tolerance, const char* name, hns_value_grid* out, void* stream) {
	int rc = check_export(s, tolerance, name, out);
	if (rc) return rc;
	const float* const planes[3] = {s->vel[0], s->vel[1], s->vel[2]};
	return export_field(s, planes, 3, tolerance, name, out, static_cast<cudaStream_t>(stream));
}
int hns_state_export_scalar(hns_state* s, int index, float tolerance, const char* name, hns_value_grid* out, void* stream) {
	int rc = check_export(s, tolerance, name, out);
	if (rc) return rc;
	if (index < 0 || index >= s->n_scalars) return fail(HNS_ERR_INVALID_ARGUMENT, "scalar index out of range");
	const float* const planes[3] = {s->sc[index], nullptr, nullptr};
	return export_field(s, planes, 1, tolerance, name, out, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
