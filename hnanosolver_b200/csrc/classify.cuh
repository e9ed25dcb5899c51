// Active-voxel classification of a resident field's leaves, shared by the pruned export (export.cu) and the re-domaining of a state
// (domain.cu, hns_state_domain_build): a voxel is active iff !(|v| <= tol) in any of the C components (NaN is active), and a leaf is
// kept iff it has an active voxel. Internal linkage: each translation unit that launches it has its own instance.
#pragma once
#include <cstdint>

namespace {

// One warp per listed leaf; lane t holds the voxel quads q = k * 32 + t (k = 0..3). Voxel 4q + e is bit 4 (t & 15) + e of mask word
// 2k + (t >> 4), so each half-warp's nibbles make one word, OR-reduced over the warp per 32-bit half. list: leaf ids or null = 0 .. n-1.
// masks: [n][8] (NanoVDB leaf mask order: word x, bit y * 8 + z); keep: [n].
template <int C>
__global__ void __launch_bounds__(256) k_export_classify(const float* f0, const float* f1, const float* f2, const int32_t* __restrict__ list,
                                                         uint32_t n, float tol, uint64_t* __restrict__ masks, uint32_t* __restrict__ keep) {
	const uint32_t i = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
	if (i >= n) return;  // the whole warp
	const uint32_t leaf = list ? uint32_t(__ldg(list + i)) : i;
	const float4* plane[3] = {reinterpret_cast<const float4*>(f0) + uint64_t(leaf) * 128u, reinterpret_cast<const float4*>(f1) + uint64_t(leaf) * 128u,
	                          reinterpret_cast<const float4*>(f2) + uint64_t(leaf) * 128u};
	float4 v[C][4];
#pragma unroll
	for (int c = 0; c < C; ++c)
#pragma unroll
		for (int k = 0; k < 4; ++k) v[c][k] = __ldg(plane[c] + k * 32 + lane);
	auto on = [tol](float x) { return !(fabsf(x) <= tol); };  // NaN is active
	uint64_t mine = 0;  // lane w < 8: mask word w
#pragma unroll
	for (int k = 0; k < 4; ++k) {
		uint32_t nib = 0;
#pragma unroll
		for (int c = 0; c < C; ++c)
			nib |= uint32_t(on(v[c][k].x)) | uint32_t(on(v[c][k].y)) << 1 | uint32_t(on(v[c][k].z)) << 2 | uint32_t(on(v[c][k].w)) << 3;
		const uint32_t part = nib << (4 * (lane & 7)), hi_half = lane & 8, odd = lane & 16;
		const uint32_t e_lo = __reduce_or_sync(0xffffffffu, !odd && !hi_half ? part : 0u), e_hi = __reduce_or_sync(0xffffffffu, !odd && hi_half ? part : 0u);
		const uint32_t o_lo = __reduce_or_sync(0xffffffffu, odd && !hi_half ? part : 0u), o_hi = __reduce_or_sync(0xffffffffu, odd && hi_half ? part : 0u);
		if (lane == 2u * k) mine = uint64_t(e_hi) << 32 | e_lo;
		if (lane == 2u * k + 1u) mine = uint64_t(o_hi) << 32 | o_lo;
	}
	if (lane < 8) masks[uint64_t(i) * 8u + lane] = mine;
	const bool any = __any_sync(0xffffffffu, mine != 0);
	if (lane == 0) keep[i] = any;
}

}  // namespace
