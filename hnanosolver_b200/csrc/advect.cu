// Semi-Lagrangian BFECC advection (reference src/Cuda/Kernel.cu:118-266 advect_scalars, :269-352 advect_scalar, :354-453
// advect_vector; samplers src/Utils/Stencils.hpp:25-173).
//
// Persistent CTAs of 512 threads (one per voxel of a leaf), two per SM, walk the leaf list. For every leaf the CTA needs the field
// values of the region x, y in [-3, 11), z in [-4, 12) (leaf-local; 14 x 14 rows of 16 floats, from up to 27 leaves) in shared memory:
// every trilinear / nearest fetch whose 2x2x2 footprint lies inside it is then a shared-memory read -- no per-sample leaf lookup, no
// scattered global loads. The region of the NEXT stage is copied with 16-byte cp.async into the second half of a double buffer while
// the current one is sampled ("the staged region" below has the shared-memory layout). This is the second generation of these kernels; the first (round 1, profiles/r1e_advect_ncu.txt: 1535 instructions per
// voxel in advect_scalars at S = 5, issue slots 63 % busy) was instruction bound, so the per-voxel instruction stream was cut to what
// the arithmetic needs (profiles/r2a_*: 2.65 -> 2.21 ms and 1.13 -> 0.97 ms, now bound by shared-memory wavefronts):
//   * the staging plan of a thread (which two quads of the region it copies, from which neighbour slot and leaf offset) depends on
//     the thread only: decoded once per kernel instead of once per leaf (it contained an integer division);
//   * a leaf's metadata (27 neighbour ids, origin, id) travels through a shared-memory ring one leaf ahead, so no stage starts with a
//     dependent chain of global loads;
//   * the values "inactive" cells take (0, or array element 0 for advect_scalars) are read once per kernel, not once per stage;
//   * the shared trace of advect_scalars keeps 6 weight factors per sample (4 xy products, 2 z factors) instead of recomputing all 8
//     corner weights from the fractions for every field; a corner weight is one more multiply, rounded exactly like the reference's
//     two-step product (Kernel.cu:169-183);
//   * scalar stages are compiled for 1, 2 and 3 fields (no run-time loop over fields, no run-time-indexed pointer tables);
//   * there is NO cold path inside the hot kernels: a voxel whose sample footprint leaves the region (back-trace longer than 3 voxels;
//     the reference has no CFL limit) only raises its leaf's flag, and a second kernel redoes flagged leaves voxel by voxel through
//     the neighbour table / tree walk (sampling.cuh). With CFL <= 2.5 no leaf is flagged and that kernel is a few microseconds of
//     flag reads. Results do not depend on which kernel produced a voxel: both evaluate the reference's expressions in its order.
// The hasCollision variants keep their two SDF samples per voxel as global gathers (sampling.cuh), as before.
#include <cassert>
#include <cstdlib>

#include "kernels.cuh"
#include "sampling.cuh"

namespace hns {
namespace {

__device__ __forceinline__ void cp16(float* smem_dst, const float* gsrc) {
	const uint32_t d = uint32_t(__cvta_generic_to_shared(smem_dst));
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp4(int* smem_dst, const int* gsrc) {
	const uint32_t d = uint32_t(__cvta_generic_to_shared(smem_dst));
	asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

constexpr int kMeta = 32, kMetaOx = 27, kMetaLeaf = 30;  // ring slot: nbr[27], origin x y z, leaf id

// metadata of work item `w` into a ring slot: asynchronously (rides in the caller's cp.async group) or right now
__device__ __forceinline__ void meta_fetch(const GridView& g, int* slot, uint32_t w, bool async) {
	const int t = threadIdx.x;
	if (t < 31) {
		const uint32_t leaf = g.leaf_at(w);
		if (t < 27) {
			if (async) cp4(slot + t, g.nbr + uint64_t(leaf) * 27u + t);
			else slot[t] = __ldg(g.nbr + uint64_t(leaf) * 27u + t);
		} else if (t < 30) {
			if (async) cp4(slot + t, reinterpret_cast<const int*>(g.origin + leaf) + (t - 27));
			else slot[t] = __ldg(reinterpret_cast<const int*>(g.origin + leaf) + (t - 27));
		} else {
			slot[kMetaLeaf] = int(leaf);
		}
	}
}

// ---- the staged region --------------------------------------------------------------------------------------------------------------
// x, y in [-3, 11), z in [-4, 12) around the leaf: 14 x 14 rows of 16 floats per field. Row pitch 16 floats with NO padding; instead the
// two 8-float halves of a row trade places in every other pair of rows (physical z = z ^ 8 when bit 1 of the row index is set):
//   * the 4 (y) x 8 (z) lanes of a warp still hit 32 distinct banks when they read one displaced copy of their own cells -- rows y and
//     y + 1 use different 16-bank halves, rows y and y + 2 use complementary 8-bank halves of the same half;
//   * an x-plane is 14 * 16 = 224 floats = 7 * 32 banks, so a lane whose sample straddles an integer x reads the SAME bank one plane
//     further: lanes of one warp that disagree about floor(x) no longer conflict (with the padded 24-float pitch of the first version the
//     plane pitch was 16 banks off and every such warp paid two wavefronts per gather; ncu: 33-38 % of all shared wavefronts were
//     conflicts);
//   * a field takes 12.25 KB instead of 18.4 KB, so a stage holds FOUR fields in less shared memory than three took: the shared trace of
//     advect_scalars rides with the first scalar field and the remaining fields go four at a time (S = 5: two stages per leaf, not three).
constexpr int kRX = 14, kRZ = 16, kHaloXY = 3, kHaloZ = 4;
constexpr int kPitch = 16, kPlane = kRX * kPitch, kRegionFloats = kRX * kPlane;  // 224 floats per x-plane, 3136 per field
constexpr int kStageFields = 4, kStageFloats = kStageFields * kRegionFloats;     // 49 KB per pipeline stage
constexpr size_t kAdvectSmem = 2 * kStageFloats * sizeof(float);                 // double buffer: 98 KB per CTA, two CTAs per SM
static_assert(2 * (kAdvectSmem + 2048) <= 233472, "two CTAs of the advection pipeline must fit one SM's shared memory");

__device__ __forceinline__ int swz(int ry) { return (ry & 2) << 2; }  // 8 for rows 2, 3, 6, 7, 10, 11
__device__ __forceinline__ int cell(int rx, int ry, int rz) { return rx * kPlane + ry * kPitch + (rz ^ swz(ry)); }

// Thread-constant staging plan. The region has 14 planes x 4 groups of (up to) 4 rows x 4 quads; item `it` = group * 16 + sub copies quad
// ((sub >> 3) << 1 | (sub >> 2) & 1) of row (sub & 3) of its group, so that 8 consecutive lanes cover 4 rows x 2 quads: eight 16-byte
// stores on 32 distinct banks. A thread handles items threadIdx.x and threadIdx.x + 512 (896 items, 784 of them real).
struct Stager {
	int dst[2];   // float offset in the region; -1: nothing to copy
	int slot[2];  // neighbour slot of the source leaf
	int src[2];   // float offset inside the source leaf
};
__device__ __forceinline__ Stager make_stager() {
	Stager p;
#pragma unroll
	for (int k = 0; k < 2; ++k) {
		const int it = threadIdx.x + 512 * k;
		const int group = it >> 4, sub = it & 15;
		const int rx = group >> 2, ry = (group & 3) * 4 + (sub & 3), q = ((sub >> 3) << 1) | ((sub >> 2) & 1);
		p.dst[k] = -1, p.slot[k] = kSlotSelf, p.src[k] = 0;
		if (rx < kRX && ry < kRX) {
			const int lx = rx - kHaloXY, ly = ry - kHaloXY;  // leaf-local x, y in [-3, 11)
			const int dz = q == 0 ? -1 : (q == 3 ? 1 : 0);   // z in [-4,0) | [0,4) | [4,8) | [8,12)
			p.dst[k] = rx * kPlane + ry * kPitch + ((q * 4) ^ swz(ry));
			p.slot[k] = ((lx >> 3) + 1) * 9 + ((ly >> 3) + 1) * 3 + dz + 1;
			p.src[k] = ((lx & 7) << 6) | ((ly & 7) << 3) | ((q == 1 || q == 3) ? 0 : 4);
		}
	}
	return p;
}
// starts the fill of NF regions (consecutive in shared memory) from NF brick fields; cells of missing leaves get fill[k]
template <int NF>
__device__ __forceinline__ void stage(const Stager& p, const int* __restrict__ meta, const float* const (&f)[NF], float* __restrict__ dst,
                                      const float* __restrict__ fill) {
#pragma unroll
	for (int k = 0; k < 2; ++k) {
		if (p.dst[k] < 0) continue;
		const int l = meta[p.slot[k]];
		float* d = dst + p.dst[k];
		if (l >= 0) {
			const uint32_t s = uint32_t(l) * 512u + uint32_t(p.src[k]);
#pragma unroll
			for (int i = 0; i < NF; ++i) cp16(d + i * kRegionFloats, f[i] + s);
		} else {
#pragma unroll
			for (int i = 0; i < NF; ++i) {
				const float v = fill[i];
				*reinterpret_cast<float4*>(d + i * kRegionFloats) = make_float4(v, v, v, v);
			}
		}
	}
}

// The 2x2x2 footprint of a sample whose first cell is (ri, rj, rk) relative to the leaf origin: region offsets of its four (y, z) corners
// in the plane x (the plane x + 1 is kPlane further). false when the footprint leaves the region.
struct Foot {
	int a00, a01, a10, a11;  // (y, z), (y, z+1), (y+1, z), (y+1, z+1)
};
__device__ __forceinline__ bool footprint(int ri, int rj, int rk, Foot& f) {
	const int rx = ri + kHaloXY, ry = rj + kHaloXY, rz = rk + kHaloZ;
	if (unsigned(rx) >= unsigned(kRX - 1) || unsigned(ry) >= unsigned(kRX - 1) || unsigned(rz) >= unsigned(kRZ - 1)) return false;
	const int r0 = rx * kPlane + ry * kPitch, s0 = swz(ry), s1 = swz(ry + 1);
	f.a00 = r0 + (rz ^ s0), f.a01 = r0 + ((rz + 1) ^ s0);
	f.a10 = r0 + kPitch + (rz ^ s1), f.a11 = r0 + kPitch + ((rz + 1) ^ s1);
	return true;
}
// TrilinearSampler: lerp z, then y, then x (Stencils.hpp:144-152)
__device__ __forceinline__ float tri_lerp(const float* __restrict__ r, const Foot& f, float fx, float fy, float fz) {
	const float z0 = lerpf(r[f.a00], r[f.a01], fz), z1 = lerpf(r[f.a10], r[f.a11], fz);
	const float z2 = lerpf(r[f.a00 + kPlane], r[f.a01 + kPlane], fz), z3 = lerpf(r[f.a10 + kPlane], r[f.a11 + kPlane], fz);
	return lerpf(lerpf(z0, z1, fy), lerpf(z2, z3, fy), fx);
}
// advect_scalars' weighted sum (Kernel.cu:186-206, 239-243): corners in the order (i0j0k0),(i1j0k0),(i0j1k0),(i1j1k0),(i0j0k1),...;
// wxy = {itx*ity, tx*ity, itx*ty, tx*ty}, wz = {itz, tz}; corner weight = wxy * wz, one rounding each like the reference's products
struct Weights {
	float xy[4], z[2];
};
__device__ __forceinline__ Weights make_weights(float tx, float ty, float tz) {
	const float itx = 1.0f - tx, ity = 1.0f - ty;
	return Weights{{itx * ity, tx * ity, itx * ty, tx * ty}, {1.0f - tz, tz}};
}
__device__ __forceinline__ float tri_weighted(const float* __restrict__ r, const Foot& f, const Weights& w) {
	float acc = 0.f;
	acc = fmaf(r[f.a00], w.xy[0] * w.z[0], acc);
	acc = fmaf(r[f.a00 + kPlane], w.xy[1] * w.z[0], acc);
	acc = fmaf(r[f.a10], w.xy[2] * w.z[0], acc);
	acc = fmaf(r[f.a10 + kPlane], w.xy[3] * w.z[0], acc);
	acc = fmaf(r[f.a01], w.xy[0] * w.z[1], acc);
	acc = fmaf(r[f.a01 + kPlane], w.xy[1] * w.z[1], acc);
	acc = fmaf(r[f.a11], w.xy[2] * w.z[1], acc);
	acc = fmaf(r[f.a11 + kPlane], w.xy[3] * w.z[1], acc);
	return acc;
}
// a voxel's own cell and its y / z neighbours in the region (the x neighbours are +-kPlane): thread constants
struct Own {
	int c, ym, yp, zm, zp;
};
__device__ __forceinline__ Own make_own(int x, int y, int z) {
	const int rx = x + kHaloXY, ry = y + kHaloXY, rz = z + kHaloZ;
	return Own{cell(rx, ry, rz), cell(rx, ry - 1, rz), cell(rx, ry + 1, rz), cell(rx, ry, rz - 1), cell(rx, ry, rz + 1)};
}
// min / max over the cell and its six face neighbours (Kernel.cu:250-258, 402-421)
__device__ __forceinline__ void clamp_range(const float* __restrict__ r, const Own& o, float own, float& mn, float& mx) {
	const float a = r[o.c - kPlane], b = r[o.c + kPlane], c = r[o.ym], d = r[o.yp], e = r[o.zm], f = r[o.zp];
	mn = fminf(fminf(fminf(own, a), fminf(b, c)), fminf(fminf(d, e), f));
	mx = fmaxf(fmaxf(fmaxf(own, a), fmaxf(b, c)), fmaxf(fmaxf(d, e), f));
}

struct Items {
	uint32_t base, stride, count;
	__device__ __forceinline__ uint32_t at(uint32_t k) const { return base + k * stride; }
};
// CTA b takes work items b, b + G, b + 2G, ...: the whole grid advances through the leaf list together, so the x-neighbour planes a
// region needs are still in the L2 from the CTAs that staged them a moment ago (measured in round 1: with one contiguous range per CTA
// every leaf was fetched from HBM about three times)
__device__ __forceinline__ Items cta_items2(const GridView& g) {
	Items it;
	it.base = blockIdx.x, it.stride = gridDim.x;
	it.count = it.base < g.count() ? (g.count() - it.base + gridDim.x - 1) / gridDim.x : 0u;
	return it;
}

// ---------------------------------------------------------------------------------------------------------------------------------
// advect_vector
// ---------------------------------------------------------------------------------------------------------------------------------
template <bool kCollision>
__global__ void __launch_bounds__(512, 2) k_advect_vector2(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                           const float* __restrict__ w, float* __restrict__ ou, float* __restrict__ ov,
                                                           float* __restrict__ ow, float sdt, const float* __restrict__ sdf,
                                                           uint8_t* __restrict__ cold) {
	extern __shared__ __align__(16) float region[];
	__shared__ int meta[3][kMeta];
	__shared__ float fill[3];
	const Items items = cta_items2(g);
	if (!items.count) return;
	const int tid = threadIdx.x;
	const int x = tid >> 6, y = (tid >> 3) & 7, z = tid & 7;
	const Own own = make_own(x, y, z);
	const Stager stg = make_stager();
	const float* const fields[3] = {u, v, w};
	if (tid < 3) fill[tid] = 0.f;
	meta_fetch(g, meta[0], items.at(0), false);
	__syncthreads();
	auto issue = [&](uint32_t k) {  // stage item k (its metadata is in the ring); the next item's metadata rides along
		stage<3>(stg, meta[k % 3], fields, region + (k & 1) * kStageFloats, fill);
		if (k + 1 < items.count) meta_fetch(g, meta[(k + 1) % 3], items.at(k + 1), true);
		cp_commit();
	};
	issue(0);
	for (uint32_t k = 0; k < items.count; ++k) {
		cp_wait_all();
		__syncthreads();  // item k's region and item k+1's metadata have landed for every thread; nobody reads the other buffer any more
		if (k + 1 < items.count) issue(k + 1);
		const float* __restrict__ ru = region + (k & 1) * kStageFloats;
		const float* __restrict__ rv = ru + kRegionFloats;
		const float* __restrict__ rw = rv + kRegionFloats;
		const int* m = meta[k % 3];
		const uint32_t leaf = uint32_t(m[kMetaLeaf]);
		const float u0 = ru[own.c], v0 = rv[own.c], w0 = rw[own.c];
		const int ox = m[kMetaOx], oy = m[kMetaOx + 1], oz = m[kMetaOx + 2];
		const float px = float(ox + x), py = float(oy + y), pz = float(oz + z);
		float bx = fmaf(-sdt, u0, px), by = fmaf(-sdt, v0, py), bz = fmaf(-sdt, w0, pz);  // Kernel.cu:374
		LeafFrame lf{ox, oy, oz, g.nbr + uint64_t(leaf) * 27u};
		if (kCollision && trilinear_f(g, lf, sdf, bx, by, bz) < 0.0f) bx = px, by = py, bz = pz;  // :377-382
		const int bi = __float2int_rd(bx), bj = __float2int_rd(by), bk = __float2int_rd(bz);
		Foot fb;
		if (!footprint(bi - ox, bj - oy, bk - oz, fb)) {
			cold[leaf] = 1;
			continue;
		}
		const float tx = bx - float(bi), ty = by - float(bj), tz = bz - float(bk);
		const float uf = tri_lerp(ru, fb, tx, ty, tz), vf = tri_lerp(rv, fb, tx, ty, tz), wf = tri_lerp(rw, fb, tx, ty, tz);
		float fx = fmaf(sdt, uf, bx), fy = fmaf(sdt, vf, by), fz = fmaf(sdt, wf, bz);  // :387
		if (kCollision && trilinear_f(g, lf, sdf, fx, fy, fz) < 0.0f) fx = bx, fy = by, fz = bz;  // :390-394
		const int fi = __float2int_rd(fx), fj = __float2int_rd(fy), fk = __float2int_rd(fz);
		Foot ff;
		if (!footprint(fi - ox, fj - oy, fk - oz, ff)) {
			cold[leaf] = 1;
			continue;
		}
		const float sx = fx - float(fi), sy = fy - float(fj), sz = fz - float(fk);
		const float ub = tri_lerp(ru, ff, sx, sy, sz), vb = tri_lerp(rv, ff, sx, sy, sz), wb = tri_lerp(rw, ff, sx, sy, sz);
		const float cu = fmaf(0.5f, u0 - ub, uf), cv = fmaf(0.5f, v0 - vb, vf), cw = fmaf(0.5f, w0 - wb, wf);  // :399-400
		float mn, mx;
		const uint32_t self = leaf * 512u + uint32_t(tid);
		clamp_range(ru, own, u0, mn, mx);
		ou[self] = fmaxf(fminf(mn, uf), fminf(cu, fmaxf(mx, uf)));  // :402-429
		clamp_range(rv, own, v0, mn, mx);
		ov[self] = fmaxf(fminf(mn, vf), fminf(cv, fmaxf(mx, vf)));
		clamp_range(rw, own, w0, mn, mx);
		ow[self] = fmaxf(fminf(mn, wf), fminf(cw, fmaxf(mx, wf)));
	}
}

// thread (coalesced), so an unflagged grid costs one load per leaf, not one dependent round trip per leaf and CTA.
__device__ __forceinline__ void collect_flagged(const GridView& g, uint8_t* cold, uint32_t chunk, uint32_t* todo, uint32_t& n_todo) {
	if (threadIdx.x == 0) n_todo = 0;
	__syncthreads();
	const uint32_t i = chunk + threadIdx.x;
	if (i < g.count()) {
		const uint32_t leaf = g.leaf_at(i);
		if (cold[leaf]) {
			cold[leaf] = 0;
			todo[atomicAdd(&n_todo, 1u)] = leaf;
		}
	}
	__syncthreads();
}

// Flagged leaves again, voxel by voxel through the neighbour table / tree walk: the reference's expressions with IndexSampler
// semantics (inactive -> 0). One CTA per flagged leaf, grid-stride over the work list.
template <bool kCollision>
__global__ void __launch_bounds__(512) k_advect_vector_cold(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                            const float* __restrict__ w, float* __restrict__ ou, float* __restrict__ ov,
                                                            float* __restrict__ ow, float sdt, const float* __restrict__ sdf, uint8_t* cold) {
	const int tid = threadIdx.x;
	const int x = tid >> 6, y = (tid >> 3) & 7, z = tid & 7;
	__shared__ uint32_t todo[512], n_todo;
	for (uint32_t chunk = blockIdx.x * 512u; chunk < g.count(); chunk += gridDim.x * 512u) {
	collect_flagged(g, cold, chunk, todo, n_todo);
	for (uint32_t q = 0; q < n_todo; ++q) {
		const uint32_t leaf = todo[q];
		const int4 o = __ldg(g.origin + leaf);
		const LeafFrame f{o.x, o.y, o.z, g.nbr + uint64_t(leaf) * 27u};
		const uint64_t self = uint64_t(leaf) * 512u + uint32_t(tid);
		const int ci = o.x + x, cj = o.y + y, ck = o.z + z;
		const float u0 = __ldg(u + self), v0 = __ldg(v + self), w0 = __ldg(w + self);
		float bx = fmaf(-sdt, u0, float(ci)), by = fmaf(-sdt, v0, float(cj)), bz = fmaf(-sdt, w0, float(ck));
		if (kCollision && trilinear_f(g, f, sdf, bx, by, bz) < 0.0f) bx = float(ci), by = float(cj), bz = float(ck);
		float uf, vf, wf, ub, vb, wb;
		trilinear_vec(g, f, u, v, w, bx, by, bz, uf, vf, wf);
		float fx = fmaf(sdt, uf, bx), fy = fmaf(sdt, vf, by), fz = fmaf(sdt, wf, bz);
		if (kCollision && trilinear_f(g, f, sdf, fx, fy, fz) < 0.0f) fx = bx, fy = by, fz = bz;
		trilinear_vec(g, f, u, v, w, fx, fy, fz, ub, vb, wb);
		const float cu = fmaf(0.5f, u0 - ub, uf), cv = fmaf(0.5f, v0 - vb, vf), cw = fmaf(0.5f, w0 - wb, wf);
		float mnu = u0, mxu = u0, mnv = v0, mxv = v0, mnw = w0, mxw = w0;
#pragma unroll 1
		for (int q = 0; q < 6; ++q) {
			const int d = (q & 1) ? 1 : -1;
			const int64_t t = voxel_index(g, f, ci + (q < 2 ? d : 0), cj + ((q >> 1) == 1 ? d : 0), ck + (q >= 4 ? d : 0));
			const float nu = t < 0 ? 0.f : __ldg(u + t), nv = t < 0 ? 0.f : __ldg(v + t), nw = t < 0 ? 0.f : __ldg(w + t);
			mnu = fminf(mnu, nu), mxu = fmaxf(mxu, nu), mnv = fminf(mnv, nv), mxv = fmaxf(mxv, nv), mnw = fminf(mnw, nw), mxw = fmaxf(mxw, nw);
		}
		ou[self] = fmaxf(fminf(mnu, uf), fminf(cu, fmaxf(mxu, uf)));
		ov[self] = fmaxf(fminf(mnv, vf), fminf(cv, fmaxf(mxv, vf)));
		ow[self] = fmaxf(fminf(mnw, wf), fminf(cw, fmaxf(mxw, wf)));
	}
	__syncthreads();  // the list is rebuilt for the next chunk
	}
}

// ---------------------------------------------------------------------------------------------------------------------------------
// advect_scalars (kSem 0: Kernel.cu:118-266, inactive -> array element 0) / advect_scalar per field (kSem 1: :269-352, inactive -> 0)
// ---------------------------------------------------------------------------------------------------------------------------------
struct Trace {  // of one voxel, shared by all its scalar fields
	Foot fb, ff;         // footprints of the back-traced / forward-traced sample
	Weights wb, wf;      // kSem 0
	float tb[3], tf[3];  // kSem 1: fractions
};

template <int kSem, int NS>
__device__ __forceinline__ void scalar_fields(const float* __restrict__ base, const Own& own, const Trace& t, float* const (&out)[NS], uint32_t self) {
#pragma unroll
	for (int k = 0; k < NS; ++k) {
		const float* __restrict__ r = base + k * kRegionFloats;
		const float phi0 = r[own.c];
		float phiF, phiB;
		if (kSem == 0) {
			phiF = tri_weighted(r, t.fb, t.wb);  // Kernel.cu:239-243
			phiB = tri_weighted(r, t.ff, t.wf);
		} else {
			phiF = tri_lerp(r, t.fb, t.tb[0], t.tb[1], t.tb[2]);
			phiB = tri_lerp(r, t.ff, t.tf[0], t.tf[1], t.tf[2]);
		}
		const float corr = fmaf(0.5f, phi0 - phiB, phiF);  // :246-247
		float mn, mx;
		clamp_range(r, own, phi0, mn, mx);  // :253-258
		out[k][self] = fmaxf(fminf(mn, phiF), fminf(corr, fmaxf(mx, phiF)));  // :264
	}
}

// Stages of a leaf: A = the velocity (the shared trace) + scalar field 0; then the remaining fields four at a time.
template <int kSem, bool kCollision>
__global__ void __launch_bounds__(512, 2) k_advect_scalars2(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                            const float* __restrict__ w, const __grid_constant__ ScalarPtrs sp, int S, float sdt,
                                                            const float* __restrict__ sdf, uint8_t* __restrict__ cold) {
	extern __shared__ __align__(16) float region[];
	__shared__ int meta[3][kMeta];
	__shared__ float fill[3 + 16];
	const Items items = cta_items2(g);
	if (!items.count) return;
	const int tid = threadIdx.x;
	const int x = tid >> 6, y = (tid >> 3) & 7, z = tid & 7;
	const Own own = make_own(x, y, z);
	const Stager stg = make_stager();
	// what inactive cells hold: advect_scalars reads array element 0, advect_scalar reads 0
	if (tid < 3 + S) {
		float f = 0.f;
		if (kSem == 0) f = tid == 0 ? __ldg(u) : tid == 1 ? __ldg(v) : tid == 2 ? __ldg(w) : __ldg(sp.in[tid - 3]);
		fill[tid] = f;
	}
	const int jobs_per_leaf = 1 + (S - 1 + 3) / 4;
	const uint32_t n_jobs = items.count * uint32_t(jobs_per_leaf);
	meta_fetch(g, meta[0], items.at(0), false);
	__syncthreads();
	uint32_t issue_item = 0;
	int issue_jj = 0;  // the job to issue next: (item, stage within the item)
	auto issue = [&](uint32_t job) {
		float* dst = region + (job & 1) * kStageFloats;
		const int* m = meta[issue_item % 3];
		if (issue_jj == 0) {
			const float* const f4[4] = {u, v, w, sp.in[0]};
			stage<4>(stg, m, f4, dst, fill);
			if (issue_item + 1 < items.count) meta_fetch(g, meta[(issue_item + 1) % 3], items.at(issue_item + 1), true);
		} else {
			const int s0 = 1 + 4 * (issue_jj - 1), ns = min(4, S - s0);
			if (ns == 4) {
				const float* const f4[4] = {sp.in[s0], sp.in[s0 + 1], sp.in[s0 + 2], sp.in[s0 + 3]};
				stage<4>(stg, m, f4, dst, fill + 3 + s0);
			} else if (ns == 3) {
				const float* const f3[3] = {sp.in[s0], sp.in[s0 + 1], sp.in[s0 + 2]};
				stage<3>(stg, m, f3, dst, fill + 3 + s0);
			} else if (ns == 2) {
				const float* const f2[2] = {sp.in[s0], sp.in[s0 + 1]};
				stage<2>(stg, m, f2, dst, fill + 3 + s0);
			} else {
				const float* const f1[1] = {sp.in[s0]};
				stage<1>(stg, m, f1, dst, fill + 3 + s0);
			}
		}
		cp_commit();
		if (++issue_jj == jobs_per_leaf) issue_jj = 0, ++issue_item;
	};
	Trace t;
	bool is_cold = false;
	uint32_t item = 0;
	int jj = 0;
	issue(0);
	for (uint32_t job = 0; job < n_jobs; ++job) {
		cp_wait_all();
		__syncthreads();
		if (job + 1 < n_jobs) issue(job + 1);
		const float* __restrict__ base = region + (job & 1) * kStageFloats;
		const int* m = meta[item % 3];
		const uint32_t leaf = uint32_t(m[kMetaLeaf]);
		const uint32_t self = leaf * 512u + uint32_t(tid);
		if (jj == 0) {
			// ---- the shared trace through the staged velocity (Kernel.cu:126-214), then the first scalar field ----
			const float *ru = base, *rv = base + kRegionFloats, *rw = base + 2 * kRegionFloats;
			const int ox = m[kMetaOx], oy = m[kMetaOx + 1], oz = m[kMetaOx + 2];
			const float px = float(ox + x), py = float(oy + y), pz = float(oz + z);
			float bx = fmaf(-sdt, ru[own.c], px), by = fmaf(-sdt, rv[own.c], py), bz = fmaf(-sdt, rw[own.c], pz);
			LeafFrame lf{ox, oy, oz, g.nbr + uint64_t(leaf) * 27u};
			// hasCollision (:142-155): the reference tests the back-traced position twice; the second test sees either the same position
			// or the voxel itself and resets to the voxel again, so one test decides
			if (kCollision && trilinear_f(g, lf, sdf, bx, by, bz) < 0.0f) bx = px, by = py, bz = pz;
			const int bi = __float2int_rd(bx), bj = __float2int_rd(by), bk = __float2int_rd(bz);
			is_cold = !footprint(bi - ox, bj - oy, bk - oz, t.fb);
			if (!is_cold) {
				const float tx = bx - float(bi), ty = by - float(bj), tz = bz - float(bk);
				float uf, vf, wf;
				if (kSem == 0) {
					t.wb = make_weights(tx, ty, tz);
					uf = tri_weighted(ru, t.fb, t.wb), vf = tri_weighted(rv, t.fb, t.wb), wf = tri_weighted(rw, t.fb, t.wb);  // :201-206
				} else {
					t.tb[0] = tx, t.tb[1] = ty, t.tb[2] = tz;
					uf = tri_lerp(ru, t.fb, tx, ty, tz), vf = tri_lerp(rv, t.fb, tx, ty, tz), wf = tri_lerp(rw, t.fb, tx, ty, tz);
				}
				float fx = fmaf(sdt, uf, bx), fy = fmaf(sdt, vf, by), fz = fmaf(sdt, wf, bz);  // :208
				if (kCollision && trilinear_f(g, lf, sdf, fx, fy, fz) < 0.0f) fx = bx, fy = by, fz = bz;  // :211-214
				const int fi = __float2int_rd(fx), fj = __float2int_rd(fy), fk = __float2int_rd(fz);
				is_cold = !footprint(fi - ox, fj - oy, fk - oz, t.ff);
				const float sx = fx - float(fi), sy = fy - float(fj), sz = fz - float(fk);
				if (kSem == 0) t.wf = make_weights(sx, sy, sz);
				else t.tf[0] = sx, t.tf[1] = sy, t.tf[2] = sz;
			}
			if (is_cold) {
				cold[leaf] = 1;
			} else {
				float* const o1[1] = {sp.out[0]};
				scalar_fields<kSem, 1>(base + 3 * kRegionFloats, own, t, o1, self);
			}
		} else if (!is_cold) {
			const int s0 = 1 + 4 * (jj - 1), ns = min(4, S - s0);
			if (ns == 4) {
				float* const o4[4] = {sp.out[s0], sp.out[s0 + 1], sp.out[s0 + 2], sp.out[s0 + 3]};
				scalar_fields<kSem, 4>(base, own, t, o4, self);
			} else if (ns == 3) {
				float* const o3[3] = {sp.out[s0], sp.out[s0 + 1], sp.out[s0 + 2]};
				scalar_fields<kSem, 3>(base, own, t, o3, self);
			} else if (ns == 2) {
				float* const o2[2] = {sp.out[s0], sp.out[s0 + 1]};
				scalar_fields<kSem, 2>(base, own, t, o2, self);
			} else {
				float* const o1[1] = {sp.out[s0]};
				scalar_fields<kSem, 1>(base, own, t, o1, self);
			}
		}
		if (++jj == jobs_per_leaf) jj = 0, ++item;
	}
}

template <int kSem, bool kCollision>
__global__ void __launch_bounds__(512) k_advect_scalars_cold(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                             const float* __restrict__ w, const __grid_constant__ ScalarPtrs sp, int S, float sdt,
                                                             const float* __restrict__ sdf, uint8_t* cold) {
	const int tid = threadIdx.x;
	const int x = tid >> 6, y = (tid >> 3) & 7, z = tid & 7;
	__shared__ uint32_t todo[512], n_todo;
	for (uint32_t chunk = blockIdx.x * 512u; chunk < g.count(); chunk += gridDim.x * 512u) {
	collect_flagged(g, cold, chunk, todo, n_todo);
	for (uint32_t q = 0; q < n_todo; ++q) {
		const uint32_t leaf = todo[q];
		const int4 o = __ldg(g.origin + leaf);
		const LeafFrame f{o.x, o.y, o.z, g.nbr + uint64_t(leaf) * 27u};
		const uint64_t self = uint64_t(leaf) * 512u + uint32_t(tid);
		const int ci = o.x + x, cj = o.y + y, ck = o.z + z;
		float bx = fmaf(-sdt, __ldg(u + self), float(ci)), by = fmaf(-sdt, __ldg(v + self), float(cj)), bz = fmaf(-sdt, __ldg(w + self), float(ck));
		if (kCollision && trilinear_f(g, f, sdf, bx, by, bz) < 0.0f) bx = float(ci), by = float(cj), bz = float(ck);
		const int bi = __float2int_rd(bx), bj = __float2int_rd(by), bk = __float2int_rd(bz);
		const float btx = bx - float(bi), bty = by - float(bj), btz = bz - float(bk);
		float uf, vf, wf;
		if (kSem == 0) {
			uf = far_weighted(g, f, u, bi, bj, bk, btx, bty, btz);
			vf = far_weighted(g, f, v, bi, bj, bk, btx, bty, btz);
			wf = far_weighted(g, f, w, bi, bj, bk, btx, bty, btz);
		} else {
			trilinear_vec(g, f, u, v, w, bx, by, bz, uf, vf, wf);
		}
		float fx = fmaf(sdt, uf, bx), fy = fmaf(sdt, vf, by), fz = fmaf(sdt, wf, bz);
		if (kCollision && trilinear_f(g, f, sdf, fx, fy, fz) < 0.0f) fx = bx, fy = by, fz = bz;
		const int fi = __float2int_rd(fx), fj = __float2int_rd(fy), fk = __float2int_rd(fz);
		const float ftx = fx - float(fi), fty = fy - float(fj), ftz = fz - float(fk);
		int64_t nb[6];
#pragma unroll
		for (int q = 0; q < 6; ++q) {
			const int d = (q & 1) ? 1 : -1;
			nb[q] = voxel_index(g, f, ci + (q < 2 ? d : 0), cj + ((q >> 1) == 1 ? d : 0), ck + (q >= 4 ? d : 0));
		}
#pragma unroll 1
		for (int k = 0; k < S; ++k) {
			const float* __restrict__ a = sp.in[k];
			const float phi0 = __ldg(a + self);
			float phiF, phiB;
			if (kSem == 0) {
				phiF = far_weighted(g, f, a, bi, bj, bk, btx, bty, btz);
				phiB = far_weighted(g, f, a, fi, fj, fk, ftx, fty, ftz);
			} else {
				phiF = trilinear_f(g, f, a, bx, by, bz);
				phiB = trilinear_f(g, f, a, fx, fy, fz);
			}
			const float corr = fmaf(0.5f, phi0 - phiB, phiF);
			float mn = phi0, mx = phi0;
#pragma unroll
			for (int q = 0; q < 6; ++q) {
				const float val = nb[q] < 0 ? (kSem == 0 ? __ldg(a) : 0.f) : __ldg(a + nb[q]);
				mn = fminf(mn, val), mx = fmaxf(mx, val);
			}
			sp.out[k][self] = fmaxf(fminf(mn, phiF), fminf(corr, fmaxf(mx, phiF)));
		}
	}
	__syncthreads();
	}
}

// =================================================================================================================================
// Third generation: the staged region holds FOUR fields per cell (float4), fetched with one 128-bit shared-memory load.
//
// ncu on the second generation (profiles/r2d_advect_final_ncu.txt): 142 32-bit shared loads per voxel at S = 5, a quarter to a third of
// their wavefronts bank conflicts between lanes that disagree about floor(y), `mio_throttle` + `short_scoreboard` the top stalls with
// the shared pipe only 59 % busy. With the fields of a group interleaved per cell -- {u, v, w, scalar 0} and {scalar 1..4} --
//   * one LDS.128 brings the four fields of a corner: 23 loads per voxel and group instead of 92, and a corner weight is computed once
//     per corner, not once per corner and field;
//   * a 128-bit load is served a quarter-warp at a time, and a quarter-warp is one z-row of 8 voxels: its eight cells are 128 contiguous
//     bytes whatever the row or plane they sit in, so lanes that disagree about floor(x) or floor(y) never conflict and no swizzle is
//     needed (cell = rx * 224 + ry * 16 + rz; the 2x2x2 footprint is the cell + {0, 1, 16, 17, 224, 225, 240, 241}: one register);
//   * staging is one 16-byte cp.async per cell from the packed group in global memory, with thread-constant addressing: thread t copies
//     cell (ry, rz) = t & 255 of the planes rx = 2k + (t >> 8), so source and destination of the seven copies are immediates off three
//     neighbour-leaf pointers.
// The packed groups (float4[L][512], same voxel order as the brick fields) are produced by the kernel that writes the fields anyway
// (subtractPressureGradient writes {u, v, w, scalar 0}, combustion writes {fuel, waste, temperature, flame}) or by k_pack4.
// Arithmetic, operand order and the cold path are those of the second generation: results are bit-identical.
// In the frame with combustion, k_advect_vector4 also carries the combustion field update and writes group 1 itself (kCombustion).
// =================================================================================================================================
constexpr int kCells = kRX * kRX * kRZ;                         // 3136 cells, 49 KB per group
constexpr size_t kRegions4 = 2 * kCells * sizeof(float4);        // double buffer: 98 KB per CTA, two CTAs per SM
// The regions come first in the dynamic allocation and the small tables behind them -- no static shared memory in these kernels, so a
// region starts on a 128-byte line: with 464 bytes of static tables in front (80 bytes off a line) every 16-byte cp.async of a warp
// straddled two lines and cost 14 shared-memory wavefronts instead of 7 (ncu source page, profiles/r2e_*).
constexpr size_t kAdvect4Smem = kRegions4 + 3 * kMeta * sizeof(int) + 2 * sizeof(float4);
constexpr int kCX = kRX * kRZ, kCY = kRZ;                        // cell strides: x 224, y 16, z 1
static_assert(2 * (kAdvect4Smem + 2048) <= 233472, "two CTAs must fit one SM's shared memory");

__device__ __forceinline__ void cp16v(float4* smem_dst, const float4* gsrc) {
	const uint32_t d = uint32_t(__cvta_generic_to_shared(smem_dst));
	asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc) : "memory");
}

struct Stager4 {
	int cell;     // ry * 16 + rz of the cells this thread copies; -1: idle (32 of 256 lanes)
	int slot_yz;  // neighbour slot of the source leaves without its x part: (sy) * 3 + (sz)
	int src_yz;   // voxel offset inside the source leaf without its x part
	int xh;       // odd or even planes
};
__device__ __forceinline__ Stager4 make_stager4() {
	Stager4 p;
	const int c = threadIdx.x & 255, ry = c >> 4, rz = c & 15;
	const int ly = ry - kHaloXY, lz = rz - kHaloZ;
	p.cell = ry < kRX ? c : -1;
	p.slot_yz = ((ly >> 3) + 1) * 3 + ((lz >> 3) + 1);
	p.src_yz = ((ly & 7) << 3) | (lz & 7);
	p.xh = threadIdx.x >> 8;
	return p;
}
template <int XH>
__device__ __forceinline__ void stage4_planes(const Stager4& p, const int* __restrict__ meta, const float4* __restrict__ src, float4* __restrict__ dst,
                                              const float4 fill) {
	const int l0 = meta[p.slot_yz], l1 = meta[p.slot_yz + 9], l2 = meta[p.slot_yz + 18];
	const float4* const s[3] = {src + (uint32_t(l0) * 512u + uint32_t(p.src_yz)), src + (uint32_t(l1) * 512u + uint32_t(p.src_yz)),
	                            src + (uint32_t(l2) * 512u + uint32_t(p.src_yz))};
	const bool have[3] = {l0 >= 0, l1 >= 0, l2 >= 0};
	float4* d = dst + p.cell;
#pragma unroll
	for (int k = 0; k < kRX / 2; ++k) {
		const int rx = 2 * k + XH, lx = rx - kHaloXY;
		const int sx = lx < 0 ? 0 : (lx < 8 ? 1 : 2), xoff = (lx & 7) << 6;
		if (have[sx]) cp16v(d + rx * kCX, s[sx] + xoff);
		else d[rx * kCX] = fill;
	}
}
__device__ __forceinline__ void stage4(const Stager4& p, const int* __restrict__ meta, const float4* __restrict__ src, float4* __restrict__ dst,
                                       const float4 fill) {
	if (p.cell < 0) return;
	if (p.xh) stage4_planes<1>(p, meta, src, dst, fill);
	else stage4_planes<0>(p, meta, src, dst, fill);
}
// first cell of the 2x2x2 footprint of a sample; false when the footprint leaves the region
__device__ __forceinline__ bool footprint4(int ri, int rj, int rk, int& c) {
	const int rx = ri + kHaloXY, ry = rj + kHaloXY, rz = rk + kHaloZ;
	c = rx * kCX + ry * kCY + rz;
	return unsigned(rx) < unsigned(kRX - 1) && unsigned(ry) < unsigned(kRX - 1) && unsigned(rz) < unsigned(kRZ - 1);
}
__device__ __forceinline__ float4 lerp4(const float4 a, const float4 b, float w) {
	return make_float4(lerpf(a.x, b.x, w), lerpf(a.y, b.y, w), lerpf(a.z, b.z, w), lerpf(a.w, b.w, w));
}
// TrilinearSampler on the four fields of a group: lerp z, then y, then x (Stencils.hpp:144-152)
__device__ __forceinline__ float4 tri_lerp4(const float4* __restrict__ r, int c, float fx, float fy, float fz) {
	const float4 y0 = lerp4(lerp4(r[c], r[c + 1], fz), lerp4(r[c + kCY], r[c + kCY + 1], fz), fy);
	const float4 y1 = lerp4(lerp4(r[c + kCX], r[c + kCX + 1], fz), lerp4(r[c + kCX + kCY], r[c + kCX + kCY + 1], fz), fy);
	return lerp4(y0, y1, fx);
}
__device__ __forceinline__ void fma4(float4& acc, const float4 v, float w) {
	acc.x = fmaf(v.x, w, acc.x), acc.y = fmaf(v.y, w, acc.y), acc.z = fmaf(v.z, w, acc.z), acc.w = fmaf(v.w, w, acc.w);
}
// advect_scalars' weighted sum on the four fields of a group, corners in the reference's order (Kernel.cu:186-206, 239-243)
__device__ __forceinline__ float4 tri_weighted4(const float4* __restrict__ r, int c, const Weights& w) {
	float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
	fma4(acc, r[c], w.xy[0] * w.z[0]);
	fma4(acc, r[c + kCX], w.xy[1] * w.z[0]);
	fma4(acc, r[c + kCY], w.xy[2] * w.z[0]);
	fma4(acc, r[c + kCX + kCY], w.xy[3] * w.z[0]);
	fma4(acc, r[c + 1], w.xy[0] * w.z[1]);
	fma4(acc, r[c + kCX + 1], w.xy[1] * w.z[1]);
	fma4(acc, r[c + kCY + 1], w.xy[2] * w.z[1]);
	fma4(acc, r[c + kCX + kCY + 1], w.xy[3] * w.z[1]);
	return acc;
}
// the same two samplers on the fourth field only (32-bit loads: a 16-byte cell stride costs the four wavefronts a 128-bit load costs)
__device__ __forceinline__ float tri_lerp_w(const float4* __restrict__ r, int c, float fx, float fy, float fz) {
	const float z0 = lerpf(r[c].w, r[c + 1].w, fz), z1 = lerpf(r[c + kCY].w, r[c + kCY + 1].w, fz);
	const float z2 = lerpf(r[c + kCX].w, r[c + kCX + 1].w, fz), z3 = lerpf(r[c + kCX + kCY].w, r[c + kCX + kCY + 1].w, fz);
	return lerpf(lerpf(z0, z1, fy), lerpf(z2, z3, fy), fx);
}
__device__ __forceinline__ float tri_weighted_w(const float4* __restrict__ r, int c, const Weights& w) {
	float acc = 0.f;
	acc = fmaf(r[c].w, w.xy[0] * w.z[0], acc);
	acc = fmaf(r[c + kCX].w, w.xy[1] * w.z[0], acc);
	acc = fmaf(r[c + kCY].w, w.xy[2] * w.z[0], acc);
	acc = fmaf(r[c + kCX + kCY].w, w.xy[3] * w.z[0], acc);
	acc = fmaf(r[c + 1].w, w.xy[0] * w.z[1], acc);
	acc = fmaf(r[c + kCX + 1].w, w.xy[1] * w.z[1], acc);
	acc = fmaf(r[c + kCY + 1].w, w.xy[2] * w.z[1], acc);
	acc = fmaf(r[c + kCX + kCY + 1].w, w.xy[3] * w.z[1], acc);
	return acc;
}
__device__ __forceinline__ float min7(float o, float a, float b, float c, float d, float e, float f) {
	return fminf(fminf(fminf(o, a), fminf(b, c)), fminf(fminf(d, e), f));
}
__device__ __forceinline__ float max7(float o, float a, float b, float c, float d, float e, float f) {
	return fmaxf(fmaxf(fmaxf(o, a), fmaxf(b, c)), fmaxf(fmaxf(d, e), f));
}
// the limiter of the BFECC result (Kernel.cu:250-264, 402-429)
__device__ __forceinline__ float limited(float mn, float mx, float first, float corrected) {
	return fmaxf(fminf(mn, first), fminf(corrected, fmaxf(mx, first)));
}

// kCombustion: combustion_oxygen rides along (the frame's own pass would stream 2.5 GB through HBM at 40 M voxels, while this kernel,
// bound by the shared-memory pipe, leaves about 70 % of the HBM bandwidth idle): for every work item each thread also updates its own
// voxel of the leaf from the frame's input fields (combustion_voxel, kernels.cuh). The loads are issued before the sampling and consumed
// after it, on every path through the item, the cold exits included.
template <bool kCombustion>
__global__ void __launch_bounds__(512, 2) k_advect_vector4(GridView g, const float4* __restrict__ vel4, float* __restrict__ ou, float* __restrict__ ov,
                                                           float* __restrict__ ow, float sdt, uint8_t* __restrict__ cold,
                                                           const __grid_constant__ CombustionJob cj) {
	extern __shared__ __align__(128) float4 region4[];
	int(*meta)[kMeta] = reinterpret_cast<int(*)[kMeta]>(region4 + 2 * kCells);
	const Items items = cta_items2(g);
	if (!items.count) return;
	const int tid = threadIdx.x;
	const int x = tid >> 6, y = (tid >> 3) & 7, z = tid & 7;
	const int oc = (x + kHaloXY) * kCX + (y + kHaloXY) * kCY + (z + kHaloZ);
	const Stager4 stg = make_stager4();
	const float4 fill = make_float4(0.f, 0.f, 0.f, 0.f);
	meta_fetch(g, meta[0], items.at(0), false);
	__syncthreads();
	auto issue = [&](uint32_t k) {
		stage4(stg, meta[k % 3], vel4, region4 + (k & 1) * kCells, fill);
		if (k + 1 < items.count) meta_fetch(g, meta[(k + 1) % 3], items.at(k + 1), true);
		cp_commit();
	};
	issue(0);
	for (uint32_t k = 0; k < items.count; ++k) {
		cp_wait_all();
		__syncthreads();
		if (k + 1 < items.count) issue(k + 1);
		const float4* __restrict__ r = region4 + (k & 1) * kCells;
		const int* m = meta[k % 3];
		const uint32_t leaf = uint32_t(m[kMetaLeaf]);
		const uint32_t self = leaf * 512u + uint32_t(tid);
		float4 comb_in;
		if constexpr (kCombustion) comb_in = make_float4(__ldg(cj.in[0] + self), __ldg(cj.in[1] + self), __ldg(cj.in[2] + self), __ldg(cj.in[3] + self));
		auto combust = [&] {
			if constexpr (kCombustion) {
				float4 o;
				const float burn = combustion_voxel(comb_in, cj.temp_gain, o);
				cj.out[0][self] = o.x, cj.out[1][self] = o.y, cj.out[2][self] = o.z, cj.out[3][self] = o.w;
				cj.grp1[self] = o;
				cj.burn[self] = burn;
			}
		};
		const float4 c0 = r[oc];
		const int ox = m[kMetaOx], oy = m[kMetaOx + 1], oz = m[kMetaOx + 2];
		const float px = float(ox + x), py = float(oy + y), pz = float(oz + z);
		const float bx = fmaf(-sdt, c0.x, px), by = fmaf(-sdt, c0.y, py), bz = fmaf(-sdt, c0.z, pz);  // Kernel.cu:374
		const int bi = __float2int_rd(bx), bj = __float2int_rd(by), bk = __float2int_rd(bz);
		int cb;
		if (!footprint4(bi - ox, bj - oy, bk - oz, cb)) {
			cold[leaf] = 1;
			combust();
			continue;
		}
		const float4 f = tri_lerp4(r, cb, bx - float(bi), by - float(bj), bz - float(bk));
		const float fx = fmaf(sdt, f.x, bx), fy = fmaf(sdt, f.y, by), fz = fmaf(sdt, f.z, bz);  // :387
		const int fi = __float2int_rd(fx), fj = __float2int_rd(fy), fk = __float2int_rd(fz);
		int cf;
		if (!footprint4(fi - ox, fj - oy, fk - oz, cf)) {
			cold[leaf] = 1;
			combust();
			continue;
		}
		const float4 b = tri_lerp4(r, cf, fx - float(fi), fy - float(fj), fz - float(fk));
		const float cu = fmaf(0.5f, c0.x - b.x, f.x), cv = fmaf(0.5f, c0.y - b.y, f.y), cw = fmaf(0.5f, c0.z - b.z, f.z);  // :399-400
		const float4 n0 = r[oc - kCX], n1 = r[oc + kCX], n2 = r[oc - kCY], n3 = r[oc + kCY], n4 = r[oc - 1], n5 = r[oc + 1];
		combust();
		ou[self] = limited(min7(c0.x, n0.x, n1.x, n2.x, n3.x, n4.x, n5.x), max7(c0.x, n0.x, n1.x, n2.x, n3.x, n4.x, n5.x), f.x, cu);  // :402-429
		ov[self] = limited(min7(c0.y, n0.y, n1.y, n2.y, n3.y, n4.y, n5.y), max7(c0.y, n0.y, n1.y, n2.y, n3.y, n4.y, n5.y), f.y, cv);
		ow[self] = limited(min7(c0.z, n0.z, n1.z, n2.z, n3.z, n4.z, n5.z), max7(c0.z, n0.z, n1.z, n2.z, n3.z, n4.z, n5.z), f.z, cw);
	}
}

// advect_scalars / advect_scalar on packed groups, for S = 1 or S = 5 scalars: job 0 of a leaf = group 0 {u, v, w, scalar 0} (the shared
// trace and the first field), job 1 (S = 5) = group 1 {scalars 1..4}
struct GroupPtrs {
	const float4* g[2];
};
struct Trace4 {
	int cb, cf;          // first cells of the back-traced / forward-traced footprints
	Weights wb, wf;      // kSem 0
	float tb[3], tf[3];  // kSem 1: fractions
};
template <int kSem>
__global__ void __launch_bounds__(512, 2) k_advect_scalars4(GridView g, const __grid_constant__ GroupPtrs gp, const __grid_constant__ ScalarPtrs sp, int S,
                                                            float sdt, uint8_t* __restrict__ cold) {
	extern __shared__ __align__(128) float4 region4[];
	int(*meta)[kMeta] = reinterpret_cast<int(*)[kMeta]>(region4 + 2 * kCells);
	float4* fill = reinterpret_cast<float4*>(meta + 3);
	const Items items = cta_items2(g);
	if (!items.count) return;
	const int tid = threadIdx.x;
	const int x = tid >> 6, y = (tid >> 3) & 7, z = tid & 7;
	const int oc = (x + kHaloXY) * kCX + (y + kHaloXY) * kCY + (z + kHaloZ);
	const Stager4 stg = make_stager4();
	const int jobs_per_leaf = S == 1 ? 1 : 2;
	// what inactive cells hold: advect_scalars reads array element 0, advect_scalar reads 0
	if (tid < 4 * jobs_per_leaf) {
		float f = 0.f;
		if (kSem == 0) f = __ldg(reinterpret_cast<const float*>(gp.g[tid >> 2]) + (tid & 3));
		reinterpret_cast<float*>(fill)[tid] = f;
	}
	const uint32_t n_jobs = items.count * uint32_t(jobs_per_leaf);
	meta_fetch(g, meta[0], items.at(0), false);
	__syncthreads();
	uint32_t issue_item = 0;
	int issue_jj = 0;
	auto issue = [&](uint32_t job) {
		stage4(stg, meta[issue_item % 3], gp.g[issue_jj], region4 + (job & 1) * kCells, fill[issue_jj]);
		if (issue_jj == 0 && issue_item + 1 < items.count) meta_fetch(g, meta[(issue_item + 1) % 3], items.at(issue_item + 1), true);
		cp_commit();
		if (++issue_jj == jobs_per_leaf) issue_jj = 0, ++issue_item;
	};
	Trace4 t;
	bool is_cold = false;
	uint32_t item = 0;
	int jj = 0;
	issue(0);
	for (uint32_t job = 0; job < n_jobs; ++job) {
		cp_wait_all();
		__syncthreads();
		if (job + 1 < n_jobs) issue(job + 1);
		const float4* __restrict__ r = region4 + (job & 1) * kCells;
		const int* m = meta[item % 3];
		const uint32_t leaf = uint32_t(m[kMetaLeaf]);
		const uint32_t self = leaf * 512u + uint32_t(tid);
		if (jj == 0) {
			// ---- the shared trace through the staged velocity (Kernel.cu:126-214) and, with the same loads, the first scalar field ----
			const float4 c0 = r[oc];
			const int ox = m[kMetaOx], oy = m[kMetaOx + 1], oz = m[kMetaOx + 2];
			const float px = float(ox + x), py = float(oy + y), pz = float(oz + z);
			const float bx = fmaf(-sdt, c0.x, px), by = fmaf(-sdt, c0.y, py), bz = fmaf(-sdt, c0.z, pz);
			const int bi = __float2int_rd(bx), bj = __float2int_rd(by), bk = __float2int_rd(bz);
			is_cold = !footprint4(bi - ox, bj - oy, bk - oz, t.cb);
			if (!is_cold) {
				const float tx = bx - float(bi), ty = by - float(bj), tz = bz - float(bk);
				float4 f;  // velocity and scalar 0 at the back-traced position
				if (kSem == 0) {
					t.wb = make_weights(tx, ty, tz);
					f = tri_weighted4(r, t.cb, t.wb);  // :201-206, :239-243
				} else {
					t.tb[0] = tx, t.tb[1] = ty, t.tb[2] = tz;
					f = tri_lerp4(r, t.cb, tx, ty, tz);
				}
				const float fx = fmaf(sdt, f.x, bx), fy = fmaf(sdt, f.y, by), fz = fmaf(sdt, f.z, bz);  // :208
				const int fi = __float2int_rd(fx), fj = __float2int_rd(fy), fk = __float2int_rd(fz);
				is_cold = !footprint4(fi - ox, fj - oy, fk - oz, t.cf);
				const float sx = fx - float(fi), sy = fy - float(fj), sz = fz - float(fk);
				if (kSem == 0) t.wf = make_weights(sx, sy, sz);
				else t.tf[0] = sx, t.tf[1] = sy, t.tf[2] = sz;
				if (!is_cold) {
					const float phiB = kSem == 0 ? tri_weighted_w(r, t.cf, t.wf) : tri_lerp_w(r, t.cf, sx, sy, sz);
					const float corr = fmaf(0.5f, c0.w - phiB, f.w);  // :246-247
					const float a = r[oc - kCX].w, b = r[oc + kCX].w, c = r[oc - kCY].w, d = r[oc + kCY].w, e = r[oc - 1].w, h = r[oc + 1].w;
					sp.out[0][self] = limited(min7(c0.w, a, b, c, d, e, h), max7(c0.w, a, b, c, d, e, h), f.w, corr);  // :253-264
				}
			}
			if (is_cold) cold[leaf] = 1;
		} else if (!is_cold) {
			const float4 c0 = r[oc];
			float4 f, b;
			if (kSem == 0) {
				f = tri_weighted4(r, t.cb, t.wb);
				b = tri_weighted4(r, t.cf, t.wf);
			} else {
				f = tri_lerp4(r, t.cb, t.tb[0], t.tb[1], t.tb[2]);
				b = tri_lerp4(r, t.cf, t.tf[0], t.tf[1], t.tf[2]);
			}
			const float4 n0 = r[oc - kCX], n1 = r[oc + kCX], n2 = r[oc - kCY], n3 = r[oc + kCY], n4 = r[oc - 1], n5 = r[oc + 1];
			sp.out[1][self] = limited(min7(c0.x, n0.x, n1.x, n2.x, n3.x, n4.x, n5.x), max7(c0.x, n0.x, n1.x, n2.x, n3.x, n4.x, n5.x), f.x,
			                          fmaf(0.5f, c0.x - b.x, f.x));
			sp.out[2][self] = limited(min7(c0.y, n0.y, n1.y, n2.y, n3.y, n4.y, n5.y), max7(c0.y, n0.y, n1.y, n2.y, n3.y, n4.y, n5.y), f.y,
			                          fmaf(0.5f, c0.y - b.y, f.y));
			sp.out[3][self] = limited(min7(c0.z, n0.z, n1.z, n2.z, n3.z, n4.z, n5.z), max7(c0.z, n0.z, n1.z, n2.z, n3.z, n4.z, n5.z), f.z,
			                          fmaf(0.5f, c0.z - b.z, f.z));
			sp.out[4][self] = limited(min7(c0.w, n0.w, n1.w, n2.w, n3.w, n4.w, n5.w), max7(c0.w, n0.w, n1.w, n2.w, n3.w, n4.w, n5.w), f.w,
			                          fmaf(0.5f, c0.w - b.w, f.w));
		}
		if (++jj == jobs_per_leaf) jj = 0, ++item;
	}
}

// four brick fields -> one packed group (null field: zeros); a thread moves four consecutive voxels
__global__ void __launch_bounds__(256) k_pack4(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c,
                                               const float* __restrict__ d, float4* __restrict__ out, uint64_t n_quads) {
	const uint64_t q = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (q >= n_quads) return;
	const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
	const float4 va = a ? __ldg(reinterpret_cast<const float4*>(a) + q) : zero, vb = b ? __ldg(reinterpret_cast<const float4*>(b) + q) : zero;
	const float4 vc = c ? __ldg(reinterpret_cast<const float4*>(c) + q) : zero, vd = d ? __ldg(reinterpret_cast<const float4*>(d) + q) : zero;
	float4* o = out + 4 * q;
	o[0] = make_float4(va.x, vb.x, vc.x, vd.x);
	o[1] = make_float4(va.y, vb.y, vc.y, vd.y);
	o[2] = make_float4(va.z, vb.z, vc.z, vd.z);
	o[3] = make_float4(va.w, vb.w, vc.w, vd.w);
}

// ---- launch plumbing -------------------------------------------------------------------------------------------------------------
struct DeviceInfo {
	int sms = 0;
	bool attrs = false;
};
DeviceInfo& device_info() {  // per device: function attributes and the SM count belong to a device, not to the process
	static DeviceInfo info[64];
	int dev = 0;
	cudaGetDevice(&dev);
	DeviceInfo& d = info[dev & 63];
	if (!d.sms) {
		cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev);
		if (d.sms <= 0) d.sms = 148;
	}
	return d;
}
template <typename K>
void opt_in(K kernel, size_t smem = kAdvectSmem) {
	cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
	cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
void ensure_attrs(DeviceInfo& d) {
	if (d.attrs) return;
	opt_in(k_advect_vector2<false>), opt_in(k_advect_vector2<true>);
	opt_in(k_advect_scalars2<0, false>), opt_in(k_advect_scalars2<1, false>);
	opt_in(k_advect_scalars2<0, true>), opt_in(k_advect_scalars2<1, true>);
	static_assert(kAdvect4Smem >= kAdvectSmem, "opt_in asks for the second generation's size");
	opt_in(k_advect_vector4<false>, kAdvect4Smem), opt_in(k_advect_vector4<true>, kAdvect4Smem);
	opt_in(k_advect_scalars4<0>, kAdvect4Smem), opt_in(k_advect_scalars4<1>, kAdvect4Smem);
	d.attrs = true;
}

std::atomic<int>& packed_switch() {  // HNS_ADVECT4=0 / hns_set_packed_advection(0): the second-generation kernels on the brick fields
	static std::atomic<int> on{[] {
		const char* e = std::getenv("HNS_ADVECT4");
		return (!e || std::atoi(e) != 0) ? 1 : 0;
	}()};
	return on;
}
// the same for whole leaves picked by id (sharded runs: the ghost leaves after an exchange); 128 threads per leaf
__global__ void __launch_bounds__(128) k_pack4_leaves(const int32_t* __restrict__ ids, const float* __restrict__ a, const float* __restrict__ b,
                                                      const float* __restrict__ c, const float* __restrict__ d, float4* __restrict__ out) {
	const uint64_t q = uint64_t(uint32_t(__ldg(ids + blockIdx.x))) * 128u + threadIdx.x;
	const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
	const float4 va = a ? __ldg(reinterpret_cast<const float4*>(a) + q) : zero, vb = b ? __ldg(reinterpret_cast<const float4*>(b) + q) : zero;
	const float4 vc = c ? __ldg(reinterpret_cast<const float4*>(c) + q) : zero, vd = d ? __ldg(reinterpret_cast<const float4*>(d) + q) : zero;
	float4* o = out + 4 * q;
	o[0] = make_float4(va.x, vb.x, vc.x, vd.x);
	o[1] = make_float4(va.y, vb.y, vc.y, vd.y);
	o[2] = make_float4(va.z, vb.z, vc.z, vd.z);
	o[3] = make_float4(va.w, vb.w, vc.w, vd.w);
}

std::atomic<uint64_t> g_packed_launches{0};
void pack4(const float* a, const float* b, const float* c, const float* d, float4* out, uint64_t n, cudaStream_t st) {
	HNS_LAUNCH(k_pack4, unsigned((n / 4 + 255) / 256), 256, 0, st, a, b, c, d, out, n / 4);
}

}  // namespace

void launch_pack4(const float* a, const float* b, const float* c, const float* d, float4* out, uint64_t n, cudaStream_t st) {
	if (n) pack4(a, b, c, d, out, n, st);
}
void launch_pack4_leaves(const int32_t* ids, uint64_t n_ids, const float* a, const float* b, const float* c, const float* d, float4* out,
                         cudaStream_t st) {
	if (n_ids) HNS_LAUNCH(k_pack4_leaves, unsigned(n_ids), 128, 0, st, ids, a, b, c, d, out);
}
bool packed_advection_enabled() { return packed_switch().load(std::memory_order_relaxed) != 0; }
int set_packed_advection(int on) { return packed_switch().exchange(on ? 1 : 0); }
uint64_t packed_advection_launches() { return g_packed_launches.load(); }

void launch_advect_vector(const GridView& g, const float* const vel[3], float* const out[3], float dt, float inv_dx, cudaStream_t st, const float* sdf,
                          uint8_t* cold, const float4* grp0, const CombustionJob* comb) {
	if (!g.count()) return;
	DeviceInfo& d = device_info();
	ensure_attrs(d);
	const int grid = int(std::min<uint32_t>(uint32_t(2 * d.sms), g.count()));
	const float sdt = dt * inv_dx;
	const int cold_grid = int(std::min<uint32_t>(uint32_t(4 * d.sms), (g.count() + 511u) / 512u));
	if (grp0) {  // group 0 holds this velocity: the third generation
		assert(!sdf);
		g_packed_launches.fetch_add(1, std::memory_order_relaxed);
		if (comb) HNS_LAUNCH(k_advect_vector4<true>, grid, 512, kAdvect4Smem, st, g, grp0, out[0], out[1], out[2], sdt, cold, *comb);
		else HNS_LAUNCH(k_advect_vector4<false>, grid, 512, kAdvect4Smem, st, g, grp0, out[0], out[1], out[2], sdt, cold, CombustionJob{});
	} else {
		assert(!comb);
		auto hot = sdf ? k_advect_vector2<true> : k_advect_vector2<false>;
		HNS_LAUNCH(hot, grid, 512, kAdvectSmem, st, g, vel[0], vel[1], vel[2], out[0], out[1], out[2], sdt, sdf, cold);
	}
	auto cold_k = sdf ? k_advect_vector_cold<true> : k_advect_vector_cold<false>;
	HNS_LAUNCH(cold_k, cold_grid, 512, 0, st, g, vel[0], vel[1], vel[2], out[0], out[1], out[2], sdt, sdf, cold);
	if (sdf) launch_collision_boundary(g, out, out, sdf, inv_dx, 1.5f, 1, st);  // the boundary tail of the kernel, Kernel.cu:432-450
}

void launch_advect_scalars(const GridView& g, const float* const vel[3], const ScalarPtrs& sp, int S, float dt, float inv_dx, int sampler_semantics,
                           cudaStream_t st, const float* sdf, uint8_t* cold, const float4* const grp[2]) {
	if (!g.count() || S <= 0) return;
	DeviceInfo& d = device_info();
	ensure_attrs(d);
	const int grid = int(std::min<uint32_t>(uint32_t(2 * d.sms), g.count()));
	const float sdt = dt * inv_dx;
	const int cold_grid = int(std::min<uint32_t>(uint32_t(4 * d.sms), (g.count() + 511u) / 512u));
	if (grp) {  // the packed groups of these fields: the third generation
		assert(!sdf && grp[0] && (S == 1 || (S == 5 && grp[1])));
		g_packed_launches.fetch_add(1, std::memory_order_relaxed);
		const GroupPtrs gp{{grp[0], grp[1]}};
		auto hot4 = sampler_semantics == 0 ? k_advect_scalars4<0> : k_advect_scalars4<1>;
		HNS_LAUNCH(hot4, grid, 512, kAdvect4Smem, st, g, gp, sp, S, sdt, cold);
	} else {
		auto hot = sampler_semantics == 0 ? (sdf ? k_advect_scalars2<0, true> : k_advect_scalars2<0, false>)
		                                  : (sdf ? k_advect_scalars2<1, true> : k_advect_scalars2<1, false>);
		HNS_LAUNCH(hot, grid, 512, kAdvectSmem, st, g, vel[0], vel[1], vel[2], sp, S, sdt, sdf, cold);
	}
	auto cold_k = sampler_semantics == 0 ? (sdf ? k_advect_scalars_cold<0, true> : k_advect_scalars_cold<0, false>)
	                                     : (sdf ? k_advect_scalars_cold<1, true> : k_advect_scalars_cold<1, false>);
	HNS_LAUNCH(cold_k, cold_grid, 512, 0, st, g, vel[0], vel[1], vel[2], sp, S, sdt, sdf, cold);
}

}  // namespace hns
