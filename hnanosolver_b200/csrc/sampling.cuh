// Device helpers shared by the advection kernels (kernels.cu, advect.cu): the generic per-voxel samplers that resolve every fetch
// through the leaf's 27-neighbour table (or, farther away, by walking the NanoVDB buffer). The staged kernels use them only for what
// does not fit their shared-memory region; the "cold" kernels use them for everything.
// Reference semantics: src/Utils/Stencils.hpp:25-173 (Floor, IndexSampler<T,0/1>, TrilinearSampler), src/Cuda/Kernel.cu:163-206.
#pragma once
#include "common.cuh"

namespace hns {

// Resolves voxel (i,j,k) (global coordinates) to a sidecar index, or -1 when inactive. The 3x3x3 leaf neighbourhood of the
// current leaf comes from its 27-entry table; anything farther away walks the NanoVDB buffer. Cold path only.
struct LeafFrame {
	int ox, oy, oz;
	const int32_t* nbr;  // this leaf's row of the neighbour table (global memory)
};
__device__ __forceinline__ int64_t voxel_index(const GridView& g, const LeafFrame& f, int i, int j, int k) {
	const int rx = i - f.ox, ry = j - f.oy, rz = k - f.oz;
	const int dx = rx >> 3, dy = ry >> 3, dz = rz >> 3;
	int32_t l;
	if (((dx + 1) | (dy + 1) | (dz + 1)) & ~3 || dx == 2 || dy == 2 || dz == 2) {  // outside the 3x3x3 neighbourhood
		if (g.far_flag) atomicOr(g.far_flag, 0x100u);
		l = probe_leaf(g, i, j, k);
	} else {
		l = __ldg(f.nbr + (dx + 1) * 9 + (dy + 1) * 3 + (dz + 1));
	}
	return l < 0 ? int64_t(-1) : int64_t(uint64_t(l) * 512u + uint32_t(((rx & 7) << 6) | ((ry & 7) << 3) | (rz & 7)));
}
__device__ __forceinline__ float lerpf(float a, float b, float w) { return fmaf(w, b - a, a); }

// TrilinearSampler<Vec3f>::sample: Floor (round down, fractional part in place), 8 nearest fetches (inactive -> 0),
// lerp z, then y, then x (Stencils.hpp:96-157)
static __device__ __noinline__ void trilinear_vec(const GridView& g, const LeafFrame& f, const float* __restrict__ u, const float* __restrict__ v,
                                              const float* __restrict__ w, float px, float py, float pz, float& ru, float& rv, float& rw) {
	const int i = __float2int_rd(px), j = __float2int_rd(py), k = __float2int_rd(pz);
	const float fx = px - float(i), fy = py - float(j), fz = pz - float(k);
	float cu[8], cv[8], cw[8];
#pragma unroll
	for (int q = 0; q < 8; ++q) {  // q = a*4 + b*2 + c  <->  v[a][b][c]
		const int64_t idx = voxel_index(g, f, i + (q >> 2), j + ((q >> 1) & 1), k + (q & 1));
		cu[q] = idx < 0 ? 0.f : __ldg(u + idx);
		cv[q] = idx < 0 ? 0.f : __ldg(v + idx);
		cw[q] = idx < 0 ? 0.f : __ldg(w + idx);
	}
	ru = lerpf(lerpf(lerpf(cu[0], cu[1], fz), lerpf(cu[2], cu[3], fz), fy), lerpf(lerpf(cu[4], cu[5], fz), lerpf(cu[6], cu[7], fz), fy), fx);
	rv = lerpf(lerpf(lerpf(cv[0], cv[1], fz), lerpf(cv[2], cv[3], fz), fy), lerpf(lerpf(cv[4], cv[5], fz), lerpf(cv[6], cv[7], fz), fy), fx);
	rw = lerpf(lerpf(lerpf(cw[0], cw[1], fz), lerpf(cw[2], cw[3], fz), fy), lerpf(lerpf(cw[4], cw[5], fz), lerpf(cw[6], cw[7], fz), fy), fx);
}
static __device__ __noinline__ float trilinear_f(const GridView& g, const LeafFrame& f, const float* __restrict__ a, float px, float py, float pz) {
	const int i = __float2int_rd(px), j = __float2int_rd(py), k = __float2int_rd(pz);
	const float fx = px - float(i), fy = py - float(j), fz = pz - float(k);
	float c[8];
#pragma unroll
	for (int q = 0; q < 8; ++q) {
		const int64_t idx = voxel_index(g, f, i + (q >> 2), j + ((q >> 1) & 1), k + (q & 1));
		c[q] = idx < 0 ? 0.f : __ldg(a + idx);
	}
	return lerpf(lerpf(lerpf(c[0], c[1], fz), lerpf(c[2], c[3], fz), fy), lerpf(lerpf(c[4], c[5], fz), lerpf(c[6], c[7], fz), fy), fx);
}

// advect_scalars (Kernel.cu:118-266): explicit corner weights, fma accumulation in corner order (i0j0k0),(i1j0k0),(i0j1k0),(i1j1k0),(i0j0k1),...
__device__ __forceinline__ void corner_weights(float tx, float ty, float tz, float (&w)[8]) {  // :169-183
	const float itx = 1.0f - tx, ity = 1.0f - ty, itz = 1.0f - tz;
	const float w00 = itx * ity, w10 = tx * ity, w01 = itx * ty, w11 = tx * ty;
	w[0] = w00 * itz, w[1] = w10 * itz, w[2] = w01 * itz, w[3] = w11 * itz;
	w[4] = w00 * tz, w[5] = w10 * tz, w[6] = w01 * tz, w[7] = w11 * tz;
}
// cold path: weighted 8-corner sums through the leaf table / tree walk, for samples outside the staged region; inactive corners read
// array element 0
static __device__ __noinline__ float far_weighted(const GridView& g, const LeafFrame& f, const float* __restrict__ a, int i0, int j0, int k0, float tx,
                                           float ty, float tz) {
	float wt[8];
	corner_weights(tx, ty, tz, wt);
	float acc = 0.f;
#pragma unroll 1
	for (int q = 0; q < 8; ++q) {
		const int64_t t = voxel_index(g, f, i0 + (q & 1), j0 + ((q >> 1) & 1), k0 + (q >> 2));
		acc = fmaf(t < 0 ? __ldg(a) : __ldg(a + t), wt[q], acc);
	}
	return acc;
}


}  // namespace hns
