// Hand-written sm_100a kernels of the HNanoSolver hot path.
//
// Design (DESIGN.md §3): the reference runs one thread per voxel and resolves every neighbour with a three-level
// NanoVDB tree walk (externals/nanovdb/NanoVDB.h:5683-5698). Here the work unit is the 8^3 leaf brick: fields are
// brick-major float[L][512] (velocity as three planes), neighbour bricks come from a per-leaf 27-entry table, rows
// of eight z-consecutive voxels move as two 128-bit accesses, and the pressure sweep stages brick + halo in shared memory
// so that a red and a black half-sweep cost one pass over HBM. Arithmetic follows the reference kernels operation by
// operation, with the multiply-adds ptxas fuses in the reference build written as explicit fmaf (see oracle/hns_oracle.c).
#include <algorithm>

#include "kernels.cuh"
#include "sampling.cuh"

namespace hns {

std::atomic<uint64_t> g_launches{0};

// =============================================================================================================
// small helpers
// =============================================================================================================
struct Row8 {
	float v[8];
};
__device__ __forceinline__ Row8 ld_row(const float* __restrict__ f, uint64_t idx) {
	const float4 a = __ldg(reinterpret_cast<const float4*>(f + idx));
	const float4 b = __ldg(reinterpret_cast<const float4*>(f + idx) + 1);
	return Row8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
// plain (coherent) loads for fields that other CTAs of the same launch write (in-place half-sweeps)
__device__ __forceinline__ Row8 ld_row_coherent(const float* f, uint64_t idx) {
	const float4 a = *reinterpret_cast<const float4*>(f + idx);
	const float4 b = *(reinterpret_cast<const float4*>(f + idx) + 1);
	return Row8{{a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}};
}
__device__ __forceinline__ void st_row(float* __restrict__ f, uint64_t idx, const Row8& r) {
	reinterpret_cast<float4*>(f + idx)[0] = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
	reinterpret_cast<float4*>(f + idx)[1] = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
}
__device__ __forceinline__ Row8 zero_row() { return Row8{{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}}; }

// Row-per-thread addressing: 64 threads per leaf, thread r owns voxels (x = r>>3, y = r&7, z = 0..7).
struct RowCtx {
	uint32_t leaf;
	int x, y;
	const int32_t* nbr;  // this leaf's 27-entry table
	__device__ __forceinline__ uint64_t self() const { return uint64_t(leaf) * 512u + uint32_t(x * 64 + y * 8); }
	// index of row (x+dx, y+dy) with dx,dy in {-1,0,1} (one of them 0), or -1 when it lies in a missing leaf
	__device__ __forceinline__ int64_t row(int dx, int dy) const {
		int xx = x + dx, yy = y + dy;
		int slot = kSlotSelf;
		if (xx < 0) slot = kSlotXm, xx = 7;
		else if (xx > 7) slot = kSlotXp, xx = 0;
		if (yy < 0) slot = kSlotYm, yy = 7;
		else if (yy > 7) slot = kSlotYp, yy = 0;
		const int32_t l = slot == kSlotSelf ? int32_t(leaf) : __ldg(nbr + slot);
		return l < 0 ? int64_t(-1) : int64_t(uint64_t(l) * 512u + uint32_t(xx * 64 + yy * 8));
	}
	// index of voxel (x, y, z = 7) of the -z neighbour leaf / (x, y, z = 0) of the +z neighbour leaf, or -1
	__device__ __forceinline__ int64_t zminus() const {
		const int32_t l = __ldg(nbr + kSlotZm);
		return l < 0 ? int64_t(-1) : int64_t(uint64_t(l) * 512u + uint32_t(x * 64 + y * 8 + 7));
	}
	__device__ __forceinline__ int64_t zplus() const {
		const int32_t l = __ldg(nbr + kSlotZp);
		return l < 0 ? int64_t(-1) : int64_t(uint64_t(l) * 512u + uint32_t(x * 64 + y * 8));
	}
	// The same addresses in a colour-split half-brick field (float index of the row's quad: leaf*256 + x*32 + y*4), computed directly
	// and in 32 bits (grids are limited to 2^24 leaves, topology.cu): halving a 64-bit brick index costs six instructions per neighbour
	// row, a 64-bit index three more per address, in the hottest kernel. kNoRow marks a row in a missing leaf.
	static constexpr uint32_t kNoRow = 0xffffffffu;
	__device__ __forceinline__ uint32_t self_q() const { return leaf * 256u + uint32_t(x * 32 + y * 4); }
	__device__ __forceinline__ uint32_t row_q(int dx, int dy) const {
		int xx = x + dx, yy = y + dy;
		int slot = kSlotSelf;
		if (xx < 0) slot = kSlotXm, xx = 7;
		else if (xx > 7) slot = kSlotXp, xx = 0;
		if (yy < 0) slot = kSlotYm, yy = 7;
		else if (yy > 7) slot = kSlotYp, yy = 0;
		const int32_t l = slot == kSlotSelf ? int32_t(leaf) : __ldg(nbr + slot);
		return l < 0 ? kNoRow : uint32_t(l) * 256u + uint32_t(xx * 32 + yy * 4);
	}
	// quad of row (x, y) in the -z / +z neighbour leaf, or kNoRow
	__device__ __forceinline__ uint32_t z_q(int slot) const {
		const int32_t l = __ldg(nbr + slot);
		return l < 0 ? kNoRow : uint32_t(l) * 256u + uint32_t(x * 32 + y * 4);
	}
};
__device__ __forceinline__ bool make_row_ctx(const GridView& g, RowCtx& c) {
	const uint32_t i = blockIdx.x * (blockDim.x >> 6) + (threadIdx.x >> 6);
	if (i >= g.count()) return false;
	const uint32_t leaf = g.leaf_at(i);
	const int r = threadIdx.x & 63;
	c.leaf = leaf, c.x = r >> 3, c.y = r & 7, c.nbr = g.nbr + uint64_t(leaf) * 27u;
	return true;
}


// ---- colour-split brick fields (pressure, divergence) ----------------------------------------------------------
// A scalar field F is stored as two half-bricks per leaf: F_red[l][256] holds the voxels with (x+y+z) even, F_blk[l][256] the
// odd ones; inside a half-brick, row (x,y) owns four consecutive floats j = z>>1. A red/black half-sweep then reads and writes
// whole 16-byte quads of exactly the colour it needs (8 B/voxel of HBM traffic per half-sweep instead of 12).
// For row (x,y) with s = (x+y)&1: red voxels are z = 2j+s, black voxels z = 2j+1-s.
__device__ __forceinline__ float4 ldg4(const float* __restrict__ f, uint64_t idx) { return __ldg(reinterpret_cast<const float4*>(f + idx)); }
__device__ __forceinline__ float4 ld4(const float* f, uint64_t idx) { return *reinterpret_cast<const float4*>(f + idx); }
__device__ __forceinline__ uint64_t split_idx(uint64_t row_idx) { return row_idx >> 1; }  // brick row index (floats) -> half-brick quad index
__device__ __forceinline__ void st_split(float* __restrict__ red, float* __restrict__ blk, const RowCtx& c, const Row8& o) {
	const uint64_t q = split_idx(c.self());
	const float4 even = make_float4(o.v[0], o.v[2], o.v[4], o.v[6]), odd = make_float4(o.v[1], o.v[3], o.v[5], o.v[7]);
	const bool s = (c.x + c.y) & 1;
	*reinterpret_cast<float4*>(red + q) = s ? odd : even;
	*reinterpret_cast<float4*>(blk + q) = s ? even : odd;
}
// full 8-voxel row from the two half-bricks; row_idx as returned by RowCtx::row()/self(), parity s of that row
__device__ __forceinline__ Row8 ld_split_row(const float* __restrict__ red, const float* __restrict__ blk, uint64_t row_idx, bool s) {
	const float4 r = ldg4(red, split_idx(row_idx)), b = ldg4(blk, split_idx(row_idx));
	const float4 even = s ? b : r, odd = s ? r : b;
	return Row8{{even.x, odd.x, even.y, odd.y, even.z, odd.z, even.w, odd.w}};
}

// =============================================================================================================
// layout conversion
// =============================================================================================================
__global__ void __launch_bounds__(256) k_aos_to_soa(const float* __restrict__ aos, float* __restrict__ u, float* __restrict__ v,
                                                    float* __restrict__ w, uint64_t n) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	u[t] = __ldg(aos + 3 * t), v[t] = __ldg(aos + 3 * t + 1), w[t] = __ldg(aos + 3 * t + 2);
}
__global__ void __launch_bounds__(256) k_soa_to_aos(const float* __restrict__ u, const float* __restrict__ v, const float* __restrict__ w,
                                                    float* __restrict__ aos, uint64_t n) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	aos[3 * t] = __ldg(u + t), aos[3 * t + 1] = __ldg(v + t), aos[3 * t + 2] = __ldg(w + t);
}
void launch_aos_to_soa(const float* aos, float* u, float* v, float* w, uint64_t n, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_aos_to_soa, unsigned((n + 255) / 256), 256, 0, st, aos, u, v, w, n);
}
void launch_soa_to_aos(const float* u, const float* v, const float* w, float* aos, uint64_t n, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_soa_to_aos, unsigned((n + 255) / 256), 256, 0, st, u, v, w, aos, n);
}

// =============================================================================================================
// divergence  (reference Kernel.cu:499-519)
//   xp = (c.x + u(+x).x) * 0.5 ... ; div = (xp - xm + yp - ym + zp - zm) * inv_dx ; inactive neighbour -> 0
// =============================================================================================================
// kBurn: combustion's expansion term too (reference Kernel.cu:963), from the burn values the combustion side job of advect_vector wrote
// (advect.cu): d = fma(burn, expansion, d) on the divergence rounded to float, as when combustion_oxygen reads it back; burn = -1 (no
// oxygen) leaves d alone, so an exact -0.0 stays -0.0 there
template <bool kBurn>
__global__ void __launch_bounds__(256) k_divergence(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                    const float* __restrict__ w, float* __restrict__ div_red, float* __restrict__ div_blk,
                                                    float inv_dx, const float* __restrict__ burn, float expansion) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint64_t self = c.self();
	const Row8 cu = ld_row(u, self), cv = ld_row(v, self), cw = ld_row(w, self);
	int64_t i;
	const Row8 uxp = (i = c.row(1, 0)) >= 0 ? ld_row(u, i) : zero_row();
	const Row8 uxm = (i = c.row(-1, 0)) >= 0 ? ld_row(u, i) : zero_row();
	const Row8 vyp = (i = c.row(0, 1)) >= 0 ? ld_row(v, i) : zero_row();
	const Row8 vym = (i = c.row(0, -1)) >= 0 ? ld_row(v, i) : zero_row();
	const float wzm = (i = c.zminus()) >= 0 ? __ldg(w + i) : 0.f;
	const float wzp = (i = c.zplus()) >= 0 ? __ldg(w + i) : 0.f;
	Row8 o;
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const float xp = (cu.v[z] + uxp.v[z]) * 0.5f, xm = (cu.v[z] + uxm.v[z]) * 0.5f;
		const float yp = (cv.v[z] + vyp.v[z]) * 0.5f, ym = (cv.v[z] + vym.v[z]) * 0.5f;
		const float zp = (cw.v[z] + (z < 7 ? cw.v[z < 7 ? z + 1 : 7] : wzp)) * 0.5f;
		const float zm = (cw.v[z] + (z > 0 ? cw.v[z > 0 ? z - 1 : 0] : wzm)) * 0.5f;
		if constexpr (kBurn) o.v[z] = __fmul_rn(xp - xm + yp - ym + zp - zm, inv_dx);  // not contracted into the fma below
		else o.v[z] = (xp - xm + yp - ym + zp - zm) * inv_dx;
	}
	if constexpr (kBurn) {
		const Row8 b = ld_row(burn, self);
#pragma unroll
		for (int z = 0; z < 8; ++z)
			if (b.v[z] != -1.0f) o.v[z] = fmaf(b.v[z], expansion, o.v[z]);
	}
	st_split(div_red, div_blk, c, o);
}
void launch_divergence(const GridView& g, const float* const vel[3], float* const div[2], float inv_dx, cudaStream_t st, const float* burn,
                       float expansion) {
	if (!g.count()) return;
	HNS_LAUNCH((burn ? k_divergence<true> : k_divergence<false>), (g.count() + 3) / 4, 256, 0, st, g, vel[0], vel[1], vel[2], div[0], div[1], inv_dx, burn,
	           expansion);
}

// =============================================================================================================
// subtractPressureGradient  (reference Kernel.cu:765-829): u - ((p(+1) - p(-1)) * 0.5) * inv_dx, fused as in the reference SASS
// =============================================================================================================
// kGroup: the projected velocity also goes, together with the scalar field `s0` (or 0), into the packed group the advection kernels
// stage from (advect.cu, third generation): float4 {u, v, w, s0} per voxel.
// kBuoyancy: temperature_buoyancy first, on the v this thread reads: the value its own pass would have stored, with the same two
// roundings; that v also goes back to by.vy (= v: a thread reads and writes only its own row).
template <bool kGroup, bool kBuoyancy>
__global__ void __launch_bounds__(256) k_subtract_gradient(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                           const float* __restrict__ w, const float* __restrict__ p_red,
                                                           const float* __restrict__ p_blk, float* __restrict__ ou, float* __restrict__ ov,
                                                           float* __restrict__ ow, float inv_dx, float4* __restrict__ grp0,
                                                           const float* __restrict__ s0, const Buoyancy by) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint64_t self = c.self();
	const bool s = (c.x + c.y) & 1;
	const Row8 cp = ld_split_row(p_red, p_blk, self, s);
	int64_t i;
	const Row8 pxp = (i = c.row(1, 0)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const Row8 pxm = (i = c.row(-1, 0)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const Row8 pyp = (i = c.row(0, 1)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const Row8 pym = (i = c.row(0, -1)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	// z = 7 of the -z leaf has parity (x+y+7): colour red iff s is odd; z = 0 of the +z leaf is red iff s is even
	const float pzm = (i = c.zminus()) >= 0 ? __ldg((s ? p_red : p_blk) + (split_idx(uint64_t(i) & ~uint64_t(7)) + 3)) : 0.f;
	const float pzp = (i = c.zplus()) >= 0 ? __ldg((s ? p_blk : p_red) + split_idx(uint64_t(i))) : 0.f;
	const Row8 cu = ld_row(u, self), cw = ld_row(w, self);
	Row8 cv = ld_row(v, self);
	if constexpr (kBuoyancy) {
		const Row8 T = ld_row(by.temp, self);
#pragma unroll
		for (int z = 0; z < 8; ++z)
			if (T.v[z] > by.ambient) cv.v[z] = fmaf(fmaxf(0.0f, (T.v[z] - by.ambient) * by.strength), by.dt, cv.v[z]);
		st_row(by.vy, self, cv);
	}
	Row8 a, b, d;
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const float zp = z < 7 ? cp.v[z < 7 ? z + 1 : 7] : pzp;
		const float zm = z > 0 ? cp.v[z > 0 ? z - 1 : 0] : pzm;
		a.v[z] = fmaf(-((pxp.v[z] - pxm.v[z]) * 0.5f), inv_dx, cu.v[z]);
		b.v[z] = fmaf(-((pyp.v[z] - pym.v[z]) * 0.5f), inv_dx, cv.v[z]);
		d.v[z] = fmaf(-((zp - zm) * 0.5f), inv_dx, cw.v[z]);
	}
	st_row(ou, self, a);
	st_row(ov, self, b);
	st_row(ow, self, d);
	if constexpr (kGroup) {
		// A thread owns 8 consecutive voxels = 128 contiguous bytes of the group; stored directly, the lanes of a warp would write 16-byte
		// pieces 128 bytes apart. The 32 rows of a warp are 256 consecutive voxels (4 of the 8 x-planes of one leaf), so they trade
		// places through a warp-private tile and every store instruction writes 512 contiguous bytes. The tile is swizzled
		// (z ^ row) so that both the row-wise writes and the voxel-wise reads of a quarter-warp touch eight distinct 16-byte bank groups.
		__shared__ float4 tile[8][256];
		const Row8 q = s0 ? ld_row(s0, self) : zero_row();
		const int lane = threadIdx.x & 31;
		float4* t = tile[threadIdx.x >> 5];
#pragma unroll
		for (int z = 0; z < 8; ++z) t[lane * 8 + (z ^ (lane & 7))] = make_float4(a.v[z], b.v[z], d.v[z], q.v[z]);
		__syncwarp();
		float4* o = grp0 + (self - uint32_t(lane) * 8u);  // first voxel of the warp's 256
#pragma unroll
		for (int i = 0; i < 8; ++i) {
			const int r = 4 * i + (lane >> 3), z = lane & 7;
			o[32 * i + lane] = t[r * 8 + (z ^ (r & 7))];
		}
	}
}
void launch_subtract_gradient(const GridView& g, const float* const vel[3], const float* const p[2], float* const out[3], float inv_dx,
                              cudaStream_t st, float4* grp0, const float* s0, const Buoyancy* buoy) {
	if (!g.count()) return;
	auto k = grp0 ? (buoy ? k_subtract_gradient<true, true> : k_subtract_gradient<true, false>)
	              : (buoy ? k_subtract_gradient<false, true> : k_subtract_gradient<false, false>);
	HNS_LAUNCH(k, (g.count() + 3) / 4, 256, 0, st, g, vel[0], vel[1], vel[2], p[0], p[1], out[0], out[1], out[2], inv_dx, grp0, s0,
	           buoy ? *buoy : Buoyancy{});
}

// =============================================================================================================
// collision boundary treatment (reference Kernel.cu:77-116 enforceCollisionBoundaries; :432-450 tail of advect_vector; :808-826 tail
// of subtractPressureGradient): sdf at the voxel < 0 -> velocity 0; sdf < 0.1 -> blend towards the velocity with its normal component
// removed, blend = 1 - sdf / blend_divisor; normal = normalised central difference of the sdf (inactive neighbour -> 0).
// Per voxel, so in place is safe. Contraction as compiled in the reference (settled bit for bit against its kernels, see
// oracle/hns_oracle.c): |g|^2 = fma(gz,gz, fma(gx,gx, rnd(gy*gy))), v.n = fma(vz,nz, fma(vx,nx, rnd(vy*ny))), tangent = fma(-v.n, n, v),
// result = fma(1-b, v, rnd(b*t)) -- except in advect_vector's tail (mixed_sum), where y and z are fma(b, t, rnd((1-b)*v)).
// =============================================================================================================
__global__ void __launch_bounds__(256) k_collision_boundary(GridView g, const float* u, const float* v, const float* w, float* ou, float* ov,
                                                            float* ow, const float* __restrict__ sdf, float inv_dx, float blend_divisor,
                                                            int mixed_sum) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint64_t self = c.self();
	const Row8 sd = ld_row(sdf, self);
	Row8 a = ld_row_coherent(u, self), b = ld_row_coherent(v, self), d = ld_row_coherent(w, self);
	bool any = false;
#pragma unroll
	for (int z = 0; z < 8; ++z) any |= sd.v[z] < 0.1f;
	if (any) {
		int64_t i;
		const Row8 sxp = (i = c.row(1, 0)) >= 0 ? ld_row(sdf, i) : zero_row(), sxm = (i = c.row(-1, 0)) >= 0 ? ld_row(sdf, i) : zero_row();
		const Row8 syp = (i = c.row(0, 1)) >= 0 ? ld_row(sdf, i) : zero_row(), sym = (i = c.row(0, -1)) >= 0 ? ld_row(sdf, i) : zero_row();
		const float szm = (i = c.zminus()) >= 0 ? __ldg(sdf + i) : 0.f, szp = (i = c.zplus()) >= 0 ? __ldg(sdf + i) : 0.f;
		const float s = 0.5f * inv_dx;
#pragma unroll
		for (int z = 0; z < 8; ++z) {
			const float sv = sd.v[z];
			if (sv < 0.0f) {
				a.v[z] = b.v[z] = d.v[z] = 0.0f;
			} else if (sv < 0.1f) {
				const float zp = z < 7 ? sd.v[z < 7 ? z + 1 : 7] : szp, zm = z > 0 ? sd.v[z > 0 ? z - 1 : 0] : szm;
				const float gx = __fmul_rn(s, sxp.v[z] - sxm.v[z]), gy = __fmul_rn(s, syp.v[z] - sym.v[z]), gz = __fmul_rn(s, zp - zm);
				const float len = sqrtf(fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy))));
				float nx = 0.f, ny = 0.f, nz = 0.f;
				if (len > 1e-6f) {
					const float r = __fdiv_rn(1.0f, len);
					nx = __fmul_rn(r, gx), ny = __fmul_rn(r, gy), nz = __fmul_rn(r, gz);
				}
				const float blend = __fsub_rn(1.0f, __fdiv_rn(sv, blend_divisor)), keep = __fsub_rn(1.0f, blend);
				const float vx = a.v[z], vy = b.v[z], vz = d.v[z];
				const float vdotn = fmaf(vz, nz, fmaf(vx, nx, __fmul_rn(vy, ny)));
				const float tx = fmaf(-vdotn, nx, vx), ty = fmaf(-vdotn, ny, vy), tz = fmaf(-vdotn, nz, vz);
				a.v[z] = fmaf(keep, vx, __fmul_rn(blend, tx));
				b.v[z] = mixed_sum ? fmaf(blend, ty, __fmul_rn(keep, vy)) : fmaf(keep, vy, __fmul_rn(blend, ty));
				d.v[z] = mixed_sum ? fmaf(blend, tz, __fmul_rn(keep, vz)) : fmaf(keep, vz, __fmul_rn(blend, tz));
			}
		}
	}
	if (any || ou != u) {
		st_row(ou, self, a);
		st_row(ov, self, b);
		st_row(ow, self, d);
	}
}
void launch_collision_boundary(const GridView& g, const float* const vel[3], float* const out[3], const float* sdf, float inv_dx,
                               float blend_divisor, int mixed_sum, cudaStream_t st) {
	if (g.count())
		HNS_LAUNCH(k_collision_boundary, (g.count() + 3) / 4, 256, 0, st, g, vel[0], vel[1], vel[2], out[0], out[1], out[2], sdf, inv_dx, blend_divisor,
		           mixed_sum);
}

// =============================================================================================================
// red-black Gauss-Seidel / SOR  (reference Kernel.cu:591-623)
//   s = (pxp + pxm + pyp + pym + pzp + pzm) - div*dx^2 ; pGS = s/6 ; p = pOld + omega*(pGS - pOld)
//   as compiled in the reference: s = fma(-div, dx2, sum); d = fma(s, 1/6, -pOld); p = fma(d, omega, pOld)
// =============================================================================================================
__device__ __forceinline__ float sor_update(float pxp, float pxm, float pyp, float pym, float pzp, float pzm, float dv, float pOld, float dx2,
                                            float omega) {
	const float s = fmaf(-dv, dx2, ((((pxp + pxm) + pyp) + pym) + pzp) + pzm);
	const float d = fmaf(s, 0.166666667f, -pOld);
	return fmaf(d, omega, pOld);
}

// the same relaxation with a per-cell diagonal (coarse multigrid levels): pGS = s / diag
__device__ __forceinline__ float sor_update_diag(float pxp, float pxm, float pyp, float pym, float pzp, float pzm, float dv, float pOld, float dx2,
                                                 float omega, float diag) {
	const float s = fmaf(-dv, dx2, ((((pxp + pxm) + pyp) + pym) + pzp) + pzm);
	return fmaf(__fdiv_rn(s, diag) - pOld, omega, pOld);
}

// One colour per launch, in place, on the colour-split layout. Thread per row (x,y): the four voxels of the swept colour are
// one float4; their x/y neighbours are the same-index float4 of the other colour in the four adjacent rows, their z neighbours
// the other-colour quad of the own row shifted by one, plus one scalar from the leaf above/below. Per half-sweep the HBM
// traffic is: other-colour p (read), this-colour p (read + write), this-colour div (read) = 8 B per voxel of the grid.
// `reverse` walks the leaves back to front: consecutive launches alternate direction so that each one starts on the bricks the
// previous launch touched last, which are still resident in the 126 MB L2.
// kPush: the sharded run's boundary sweep -- every freshly swept quad is also stored straight into the ghost copy of the leaf on
// each peer GPU that holds one (NVLink peer memory, CUDA IPC): nothing is packed, sent or unpacked afterwards; the caller raises the
// peers' arrival flags from a follow-up kernel.
// kMask: a coarse level of the multigrid solve -- `diag_c` holds the operator's diagonal of every cell of the swept colour: 6 plus a
// boundary term per face neighbour outside the domain (multigrid.cu), 0 for a cell that is itself outside. Such cells keep the value 0
// they were initialised with, which is the Dirichlet condition of the reference's solve (inactive -> 0); the update divides by the
// diagonal instead of multiplying by the reference's 0.166666667f.
template <bool kPush, bool kMask = false>
__global__ void __launch_bounds__(256) k_rbgs_split(GridView g, const float* __restrict__ div_c, float* __restrict__ p_c, const float* p_o,
                                                    float dx2, int color, float omega, int reverse, RbgsPush push,
                                                    const float* __restrict__ diag_c = nullptr) {
	RowCtx c;
	uint32_t i = blockIdx.x * 4u + (threadIdx.x >> 6);
	if (i >= g.count()) return;
	if (reverse) i = g.count() - 1u - i;
	const int r = threadIdx.x & 63;
	c.x = r >> 3, c.y = r & 7;
	if (g.list_nbr) {
		c.nbr = g.list_nbr + uint64_t(i) * 27u;
		c.leaf = uint32_t(__ldg(c.nbr + kSlotSelf));
	} else {
		c.leaf = g.leaf_at(i);
		c.nbr = g.nbr + uint64_t(c.leaf) * 27u;
	}
	const uint32_t q = c.self_q();
	const int sc = (c.x + c.y + color) & 1;  // swept voxels of this row are z = 2j + sc
	const float4 C = ld4(p_c, q);            // old values of the swept colour (only this thread writes them)
	// other colour: plain (coherent) loads when peers write ghost values into this array, read-only path otherwise
	auto ldo = [&](uint64_t idx) { return kPush ? ld4(p_o, idx) : ldg4(p_o, idx); };
	const float4 O = ldo(q);                 // own row: the z neighbours
	uint32_t t;
	const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
	const float4 Oxp = (t = c.row_q(1, 0)) != RowCtx::kNoRow ? ldo(t) : zero4;
	const float4 Oxm = (t = c.row_q(-1, 0)) != RowCtx::kNoRow ? ldo(t) : zero4;
	const float4 Oyp = (t = c.row_q(0, 1)) != RowCtx::kNoRow ? ldo(t) : zero4;
	const float4 Oym = (t = c.row_q(0, -1)) != RowCtx::kNoRow ? ldo(t) : zero4;
	// the divergence is read once per sweep and not again before 2 x 240 MB of pressure have passed through the L2: load it
	// with the streaming (evict-first) policy so that it does not displace pressure lines the next, reversed sweep starts on
	const float4 D = __ldcs(reinterpret_cast<const float4*>(div_c + q));
	// z neighbours: sc == 0: voxel j (z = 2j) has below = O[j-1] (j = 0: last other-colour voxel of the -z leaf), above = O[j]
	//               sc == 1: voxel j (z = 2j+1) has below = O[j], above = O[j+1] (j = 3: first other-colour voxel of the +z leaf)
	float halo = 0.f;
	if (sc == 0) {
		if ((t = c.z_q(kSlotZm)) != RowCtx::kNoRow) halo = p_o[t + 3u];
	} else {
		if ((t = c.z_q(kSlotZp)) != RowCtx::kNoRow) halo = p_o[t];
	}
	const float b0 = sc ? O.x : halo, b1 = sc ? O.y : O.x, b2 = sc ? O.z : O.y, b3 = sc ? O.w : O.z;  // below (z-1)
	const float a0 = sc ? O.y : O.x, a1 = sc ? O.z : O.y, a2 = sc ? O.w : O.z, a3 = sc ? halo : O.w;  // above (z+1)
	float4 n;
	n.x = sor_update(Oxp.x, Oxm.x, Oyp.x, Oym.x, a0, b0, D.x, C.x, dx2, omega);
	n.y = sor_update(Oxp.y, Oxm.y, Oyp.y, Oym.y, a1, b1, D.y, C.y, dx2, omega);
	n.z = sor_update(Oxp.z, Oxm.z, Oyp.z, Oym.z, a2, b2, D.z, C.z, dx2, omega);
	n.w = sor_update(Oxp.w, Oxm.w, Oyp.w, Oym.w, a3, b3, D.w, C.w, dx2, omega);
	if (kMask) {
		const float4 W = ldg4(diag_c, q);
		n.x = W.x != 0.f ? sor_update_diag(Oxp.x, Oxm.x, Oyp.x, Oym.x, a0, b0, D.x, C.x, dx2, omega, W.x) : 0.f;
		n.y = W.y != 0.f ? sor_update_diag(Oxp.y, Oxm.y, Oyp.y, Oym.y, a1, b1, D.y, C.y, dx2, omega, W.y) : 0.f;
		n.z = W.z != 0.f ? sor_update_diag(Oxp.z, Oxm.z, Oyp.z, Oym.z, a2, b2, D.z, C.z, dx2, omega, W.z) : 0.f;
		n.w = W.w != 0.f ? sor_update_diag(Oxp.w, Oxm.w, Oyp.w, Oym.w, a3, b3, D.w, C.w, dx2, omega, W.w) : 0.f;
	}
	*reinterpret_cast<float4*>(p_c + q) = n;
	if (kPush) {
		const uint32_t row4 = q & 255u;  // quad offset inside the half-brick
		// bit f of this row's face membership: 0 x==0, 1 x==7, 2 y==0, 3 y==7; a z face (bits 4, 5) involves every row
		const int mine = (c.x == 0 ? 1 : 0) | (c.x == 7 ? 2 : 0) | (c.y == 0 ? 4 : 0) | (c.y == 7 ? 8 : 0) | 0x30;
		for (uint32_t e = __ldg(push.dst_off + i), e1 = __ldg(push.dst_off + i + 1); e < e1; ++e) {
			const int pm = __ldg(push.dst_peer + e);  // peer index | face mask << 8
			if ((pm >> 8) & mine)
				*reinterpret_cast<float4*>(push.remote_pc[pm & 255] + (uint64_t(__ldg(push.dst_leaf + e)) * 256u + row4)) = n;
		}
	}
}
void launch_rbgs_color(const GridView& g, const float* const div[2], float* const p[2], float dx, int color, float omega, int reverse,
                       cudaStream_t st) {
	if (g.count())
		HNS_LAUNCH(k_rbgs_split<false>, (g.count() + 3) / 4, 256, 0, st, g, div[color], p[color], p[color ^ 1], dx * dx, color, omega, reverse,
		           RbgsPush{});
}
void launch_rbgs_color_masked(const GridView& g, const float* const rhs[2], float* const p[2], float dx, int color, float omega,
                              const float* const diag[2], cudaStream_t st) {
	if (g.count())
		HNS_LAUNCH((k_rbgs_split<false, true>), (g.count() + 3) / 4, 256, 0, st, g, rhs[color], p[color], p[color ^ 1], dx * dx, color, omega, 0, RbgsPush{},
		           diag[color]);
}
void launch_rbgs_color_push(const GridView& g, const float* const div[2], float* const p[2], float dx, int color, float omega, int reverse,
                            const RbgsPush& push, cudaStream_t st) {
	if (g.count())
		HNS_LAUNCH(k_rbgs_split<true>, (g.count() + 3) / 4, 256, 0, st, g, div[color], p[color], p[color ^ 1], dx * dx, color, omega, reverse, push);
}

// rows of the neighbour table in work-list order, slot 13 = the leaf id (GridView::list_nbr)
__global__ void k_gather_nbr_rows(const int32_t* __restrict__ nbr, const int32_t* __restrict__ list, uint32_t n, int32_t* __restrict__ out) {
	const uint64_t t = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
	if (t >= uint64_t(n) * 27u) return;
	const uint32_t i = uint32_t(t / 27u), k = uint32_t(t % 27u);
	const int32_t leaf = list[i];
	out[t] = k == uint32_t(kSlotSelf) ? leaf : nbr[uint64_t(leaf) * 27u + k];
}
void launch_gather_nbr_rows(const int32_t* nbr, const int32_t* list, uint32_t n, int32_t* out, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_gather_nbr_rows, uint32_t((uint64_t(n) * 27u + 255u) / 256u), 256, 0, st, nbr, list, n, out);
}

// (the advection kernels live in advect.cu)

// =============================================================================================================
// combustion_oxygen / temperature_buoyancy  (reference Kernel.cu:923-966, 831-847) -- element-wise
// =============================================================================================================
__global__ void __launch_bounds__(256) k_combustion_oxygen(const float* __restrict__ fuel, const float* __restrict__ waste,
                                                           const float* __restrict__ temp, float* __restrict__ div_red, float* __restrict__ div_blk,
                                                           const float* __restrict__ flame, float* __restrict__ oFuel,
                                                           float* __restrict__ oWaste, float* __restrict__ oTemp, float* __restrict__ oFlame,
                                                           float temp_gain, float expansion, uint64_t n, bool update_div) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	float f = fuel[t];
	const float wv = waste[t], T = temp[t], fl = flame[t];
	if (f < 0.001f) f = 0.0f;
	const float oxygen = 1.0f - f - wv;
	if (oxygen < 0.0f) {
		oFuel[t] = f, oWaste[t] = wv, oTemp[t] = T, oFlame[t] = fl;
		return;
	}
	const float burn = fminf(oxygen, f);
	oFuel[t] = f - burn;
	oWaste[t] = fmaf(burn, 2.0f, wv);
	oFlame[t] = fmaxf(fl, fminf(1.0f, burn * 10.0f));
	oTemp[t] = fmaf(burn, temp_gain, T);
	if (!update_div) return;
	// voxel t = leaf*512 + (x<<6 | y<<3 | z) lives in the colour-split divergence at quad (t>>3), lane z>>1 of its colour
	const uint32_t o = uint32_t(t) & 511u;
	const bool black = (((o >> 6) + (o >> 3) + o) & 1u) != 0;
	float* d = (black ? div_blk : div_red) + ((t >> 3) << 2) + ((o & 7u) >> 1);
	*d = fmaf(burn, expansion, *d);
}
void launch_combustion_oxygen(const float* fuel, const float* waste, const float* temp, float* const div[2], const float* flame, float* oFuel,
                              float* oWaste, float* oTemp, float* oFlame, float temp_gain, float expansion, uint64_t n, cudaStream_t st,
                              bool update_div) {
	if (n)
		HNS_LAUNCH(k_combustion_oxygen, unsigned((n + 255) / 256), 256, 0, st, fuel, waste, temp, div[0], div[1], flame, oFuel, oWaste, oTemp,
		           oFlame, temp_gain, expansion, n, update_div);
}
// Only the expansion term combustion_oxygen adds to the divergence (Kernel.cu:963): it depends on fuel and waste alone, so a cook whose
// inputs are still arriving over PCIe can start the pressure solve before temperature and flame have landed (hns_compute_sim); the
// field updates follow with update_div = false. Same expressions, same rounding.
__global__ void __launch_bounds__(256) k_combustion_divergence(const float* __restrict__ fuel, const float* __restrict__ waste,
                                                               float* __restrict__ div_red, float* __restrict__ div_blk, float expansion, uint64_t n) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	float f = fuel[t];
	const float wv = waste[t];
	if (f < 0.001f) f = 0.0f;
	const float oxygen = 1.0f - f - wv;
	if (oxygen < 0.0f) return;
	const float burn = fminf(oxygen, f);
	const uint32_t o = uint32_t(t) & 511u;
	const bool black = (((o >> 6) + (o >> 3) + o) & 1u) != 0;
	float* d = (black ? div_blk : div_red) + ((t >> 3) << 2) + ((o & 7u) >> 1);
	*d = fmaf(burn, expansion, *d);
}
void launch_combustion_divergence(const float* fuel, const float* waste, float* const div[2], float expansion, uint64_t n, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_combustion_divergence, unsigned((n + 255) / 256), 256, 0, st, fuel, waste, div[0], div[1], expansion, n);
}
// combustion_oxygen + temperature_buoyancy in one pass, the four outputs also written as one float4 {fuel, waste, temperature, flame}
// into the packed group advect_scalars stages from (advect.cu, third generation). Same expressions as the two kernels above and below;
// the buoyancy term uses the temperature this thread just computed instead of reading it back.
__global__ void __launch_bounds__(256) k_combustion_buoyancy_packed(const float* __restrict__ fuel, const float* __restrict__ waste,
                                                                    const float* __restrict__ temp, float* __restrict__ div_red,
                                                                    float* __restrict__ div_blk, const float* __restrict__ flame,
                                                                    float* __restrict__ oFuel, float* __restrict__ oWaste, float* __restrict__ oTemp,
                                                                    float* __restrict__ oFlame, float4* __restrict__ grp, float* __restrict__ vy,
                                                                    float temp_gain, float expansion, float dt, float ambient, float strength,
                                                                    uint64_t n, bool update_div, bool buoyancy) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	float4 o;
	const float burn = combustion_voxel(make_float4(fuel[t], waste[t], temp[t], flame[t]), temp_gain, o);
	if (update_div && burn != -1.0f) {
		const uint32_t v = uint32_t(t) & 511u;
		const bool black = (((v >> 6) + (v >> 3) + v) & 1u) != 0;
		float* d = (black ? div_blk : div_red) + ((t >> 3) << 2) + ((v & 7u) >> 1);
		*d = fmaf(burn, expansion, *d);
	}
	oFuel[t] = o.x, oWaste[t] = o.y, oTemp[t] = o.z, oFlame[t] = o.w;
	grp[t] = o;
	if (buoyancy && o.z > ambient) vy[t] = fmaf(fmaxf(0.0f, (o.z - ambient) * strength), dt, vy[t]);
}
void launch_combustion_buoyancy_packed(const float* fuel, const float* waste, const float* temp, float* const div[2], const float* flame, float* oFuel,
                                       float* oWaste, float* oTemp, float* oFlame, float4* grp, float* const vel[3], float temp_gain, float expansion,
                                       float dt, float ambient, float strength, uint64_t n, cudaStream_t st, bool update_div, bool buoyancy) {
	if (n)
		HNS_LAUNCH(k_combustion_buoyancy_packed, unsigned((n + 255) / 256), 256, 0, st, fuel, waste, temp, div[0], div[1], flame, oFuel, oWaste, oTemp,
		           oFlame, grp, vel[1], temp_gain, expansion, dt, ambient, strength, n, update_div, buoyancy);
}
// temperature_buoyancy (Kernel.cu:831-847) with the temperature combustion_oxygen is about to write, recomputed from its inputs
// (Kernel.cu:941-960): lets a cook fed over PCIe project and send back its velocity before the flame field has even arrived.
__global__ void __launch_bounds__(256) k_buoyancy_from_inputs(const float* __restrict__ fuel, const float* __restrict__ waste,
                                                              const float* __restrict__ temp, float* __restrict__ vy, float temp_gain, float dt,
                                                              float ambient, float strength, uint64_t n) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	float f = fuel[t];
	const float wv = waste[t];
	float T = temp[t];
	if (f < 0.001f) f = 0.0f;
	const float oxygen = 1.0f - f - wv;
	if (!(oxygen < 0.0f)) T = fmaf(fminf(oxygen, f), temp_gain, T);
	if (T > ambient) vy[t] = fmaf(fmaxf(0.0f, (T - ambient) * strength), dt, vy[t]);
}
void launch_buoyancy_from_inputs(const float* fuel, const float* waste, const float* temp, float* const vel[3], float temp_gain, float dt,
                                 float ambient, float strength, uint64_t n, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_buoyancy_from_inputs, unsigned((n + 255) / 256), 256, 0, st, fuel, waste, temp, vel[1], temp_gain, dt, ambient, strength, n);
}
// The reference adds Vec3f(0, b, 0) * dt to all three components (Kernel.cu:844-846); adding 0*dt only turns a -0.0 into +0.0,
// so only the y plane is touched here (x and z stay bit-identical except for the sign of an exact zero).
__global__ void __launch_bounds__(256) k_buoyancy(float* __restrict__ v, const float* __restrict__ temp, float dt, float ambient, float strength,
                                                  uint64_t n) {
	const uint64_t t = (blockIdx.x * uint64_t(256) + threadIdx.x) * 4;
	if (t >= n) return;
	const float4 T = __ldg(reinterpret_cast<const float4*>(temp + t));
	float4 y = *reinterpret_cast<float4*>(v + t);
	if (T.x > ambient) y.x = fmaf(fmaxf(0.0f, (T.x - ambient) * strength), dt, y.x);
	if (T.y > ambient) y.y = fmaf(fmaxf(0.0f, (T.y - ambient) * strength), dt, y.y);
	if (T.z > ambient) y.z = fmaf(fmaxf(0.0f, (T.z - ambient) * strength), dt, y.z);
	if (T.w > ambient) y.w = fmaf(fmaxf(0.0f, (T.w - ambient) * strength), dt, y.w);
	*reinterpret_cast<float4*>(v + t) = y;
}
void launch_buoyancy(float* const vel[3], const float* temp, float dt, float ambient, float strength, uint64_t n, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_buoyancy, unsigned((n / 4 + 255) / 256), 256, 0, st, vel[1], temp, dt, ambient, strength, n);
}

// colour-split <-> brick order (parity checks and host round trips of pressure / divergence)
__global__ void __launch_bounds__(256) k_split_to_brick(const float* __restrict__ red, const float* __restrict__ blk, float* __restrict__ out, uint64_t n) {
	const uint64_t t = blockIdx.x * uint64_t(256) + threadIdx.x;
	if (t >= n) return;
	const uint32_t o = uint32_t(t) & 511u;
	const bool black = (((o >> 6) + (o >> 3) + o) & 1u) != 0;
	out[t] = __ldg((black ? blk : red) + ((t >> 3) << 2) + ((o & 7u) >> 1));
}
void launch_split_to_brick(const float* const f[2], float* out, uint64_t n, cudaStream_t st) {
	if (n) HNS_LAUNCH(k_split_to_brick, unsigned((n + 255) / 256), 256, 0, st, f[0], f[1], out, n);
}

// =============================================================================================================
// vorticity confinement  (reference Kernel.cu:969-1025, computeVorticityMag Utils.cuh:226-243), out of place
//   w = curl(u) by central differences * (0.5*inv_dx);  m(c) = |w(c)|;  g = ((m(c+fs) - m(c-fs)) * 0.5) * inv_dx per axis, fs = (int)factorScale;
//   N = g / (|g| + 1e-5);  u += scale * (N x w) * dt.   Inactive velocity samples are 0, and m is ALSO evaluated at inactive
//   positions (from whatever active voxels surround them).
// The reference evaluates 42 index-grid lookups per voxel, in place (a race, HNanoSolver.cu:174). Here: pass 1 writes m for every
// active voxel (one row per thread, like the divergence), pass 2 recomputes the voxel's own w from the same rows, reads m at the six
// offset positions from the m plane and only falls back to evaluating the curl at a position when that position is inactive (or
// |fs| > 8, beyond the neighbour table). Arithmetic and FMA contraction as in the reference SASS (see oracle/hns_oracle.c).
// =============================================================================================================
struct CurlRows {
	Row8 wx, wy, wz;
};
// curl * factor of the eight voxels of row c; cu, cv = the row's own u and v (also needed by the caller)
__device__ __forceinline__ CurlRows curl_rows(const RowCtx& c, const float* __restrict__ u, const float* __restrict__ v, const float* __restrict__ w,
                                              const Row8& cu, const Row8& cv, float factor) {
	int64_t i;
	Row8 w_xp = zero_row(), v_xp = zero_row(), w_xm = zero_row(), v_xm = zero_row();
	Row8 w_yp = zero_row(), u_yp = zero_row(), w_ym = zero_row(), u_ym = zero_row();
	if ((i = c.row(1, 0)) >= 0) w_xp = ld_row(w, i), v_xp = ld_row(v, i);
	if ((i = c.row(-1, 0)) >= 0) w_xm = ld_row(w, i), v_xm = ld_row(v, i);
	if ((i = c.row(0, 1)) >= 0) w_yp = ld_row(w, i), u_yp = ld_row(u, i);
	if ((i = c.row(0, -1)) >= 0) w_ym = ld_row(w, i), u_ym = ld_row(u, i);
	float u_zm = 0.f, v_zm = 0.f, u_zp = 0.f, v_zp = 0.f;
	if ((i = c.zminus()) >= 0) u_zm = __ldg(u + i), v_zm = __ldg(v + i);
	if ((i = c.zplus()) >= 0) u_zp = __ldg(u + i), v_zp = __ldg(v + i);
	CurlRows r;
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const float up = z < 7 ? cu.v[z < 7 ? z + 1 : 7] : u_zp, um = z > 0 ? cu.v[z > 0 ? z - 1 : 0] : u_zm;
		const float vp = z < 7 ? cv.v[z < 7 ? z + 1 : 7] : v_zp, vm = z > 0 ? cv.v[z > 0 ? z - 1 : 0] : v_zm;
		r.wx.v[z] = ((w_yp.v[z] - w_ym.v[z]) - (vp - vm)) * factor;
		r.wy.v[z] = ((up - um) - (w_xp.v[z] - w_xm.v[z])) * factor;
		r.wz.v[z] = ((v_xp.v[z] - v_xm.v[z]) - (u_yp.v[z] - u_ym.v[z])) * factor;
	}
	return r;
}
// |w| and |g| as the reference compiles them (checked bit for bit against its kernel): the sums of squares contract differently
__device__ __forceinline__ float vort_norm(float wx, float wy, float wz) { return sqrtf(fmaf(wz, wz, fmaf(wy, wy, __fmul_rn(wx, wx)))); }
__device__ __forceinline__ float grad_norm(float gx, float gy, float gz) { return sqrtf(fmaf(gz, gz, fmaf(gx, gx, __fmul_rn(gy, gy)))); }

__global__ void __launch_bounds__(256) k_vorticity_mag(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                       const float* __restrict__ w, float* __restrict__ mag, float factor) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint64_t self = c.self();
	const Row8 cu = ld_row(u, self), cv = ld_row(v, self);
	const CurlRows r = curl_rows(c, u, v, w, cu, cv, factor);
	Row8 m;
#pragma unroll
	for (int z = 0; z < 8; ++z) m.v[z] = vort_norm(r.wx.v[z], r.wy.v[z], r.wz.v[z]);
	st_row(mag, self, m);
}

// |curl| at an arbitrary position (i,j,k), evaluated from the velocity planes: the cold path of pass 2 (inactive positions, far offsets)
__device__ __noinline__ float vorticity_mag_at(const GridView& g, const LeafFrame& f, const float* __restrict__ u, const float* __restrict__ v,
                                               const float* __restrict__ w, int i, int j, int k, float factor) {
	float s[6][3];
#pragma unroll
	for (int q = 0; q < 6; ++q) {  // +x, -x, +y, -y, +z, -z
		const int d = (q & 1) ? -1 : 1;
		const int64_t idx = voxel_index(g, f, i + (q < 2 ? d : 0), j + ((q >> 1) == 1 ? d : 0), k + (q >= 4 ? d : 0));
		s[q][0] = idx < 0 ? 0.f : __ldg(u + idx);
		s[q][1] = idx < 0 ? 0.f : __ldg(v + idx);
		s[q][2] = idx < 0 ? 0.f : __ldg(w + idx);
	}
	const float wx = ((s[2][2] - s[3][2]) - (s[4][1] - s[5][1])) * factor;
	const float wy = ((s[4][0] - s[5][0]) - (s[0][2] - s[1][2])) * factor;
	const float wz = ((s[0][1] - s[1][1]) - (s[2][0] - s[3][0])) * factor;
	return vort_norm(wx, wy, wz);
}

// row of m at (x + dx, y + dy) of the leaf neighbourhood, |dx|, |dy| <= 8 (one of them 0); -1 when that leaf is missing
__device__ __forceinline__ int64_t row_far(const RowCtx& c, int dx, int dy) {
	int xx = c.x + dx, yy = c.y + dy;
	int slot = kSlotSelf;
	if (xx < 0) slot = kSlotXm, xx += 8;
	else if (xx > 7) slot = kSlotXp, xx -= 8;
	if (yy < 0) slot = kSlotYm, yy += 8;
	else if (yy > 7) slot = kSlotYp, yy -= 8;
	const int32_t l = slot == kSlotSelf ? int32_t(c.leaf) : __ldg(c.nbr + slot);
	return l < 0 ? int64_t(-1) : int64_t(uint64_t(l) * 512u + uint32_t(xx * 64 + yy * 8));
}

__global__ void __launch_bounds__(256) k_vorticity_force(GridView g, const float* __restrict__ u, const float* __restrict__ v,
                                                         const float* __restrict__ w, const float* __restrict__ mag, float* __restrict__ ou,
                                                         float* __restrict__ ov, float* __restrict__ ow, float factor, float inv_dx, float scale,
                                                         float dt, int fs) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint64_t self = c.self();
	const int4 o = __ldg(g.origin + c.leaf);
	const LeafFrame f{o.x, o.y, o.z, c.nbr};
	const int gx = o.x + c.x, gy = o.y + c.y;
	const bool far = fs > 8 || fs < -8;
	// m at the six offset positions, then the gradient ((m+ - m-) * 0.5) * inv_dx per axis
	Row8 G[3];
#pragma unroll
	for (int axis = 0; axis < 2; ++axis) {
		Row8 mp, mm;
		const int64_t ip = far ? -1 : row_far(c, axis == 0 ? fs : 0, axis == 1 ? fs : 0);
		const int64_t im = far ? -1 : row_far(c, axis == 0 ? -fs : 0, axis == 1 ? -fs : 0);
		if (ip >= 0) {
			mp = ld_row(mag, ip);
		} else {
			for (int z = 0; z < 8; ++z) mp.v[z] = vorticity_mag_at(g, f, u, v, w, gx + (axis == 0 ? fs : 0), gy + (axis == 1 ? fs : 0), o.z + z, factor);
		}
		if (im >= 0) {
			mm = ld_row(mag, im);
		} else {
			for (int z = 0; z < 8; ++z) mm.v[z] = vorticity_mag_at(g, f, u, v, w, gx - (axis == 0 ? fs : 0), gy - (axis == 1 ? fs : 0), o.z + z, factor);
		}
#pragma unroll
		for (int z = 0; z < 8; ++z) G[axis].v[z] = ((mp.v[z] - mm.v[z]) * 0.5f) * inv_dx;
	}
	{
		// z axis: the own row of m shifted by fs, continued into the rows (x, y) of the -z / +z leaves (scalar loads, L1-resident rows)
		const int32_t lzm = __ldg(c.nbr + kSlotZm), lzp = __ldg(c.nbr + kSlotZp);
		const uint32_t rxy = uint32_t(c.x * 64 + c.y * 8);
		auto m_at = [&](int zz) -> float {  // m at (x, y, zz) relative to this leaf, zz in [-8, 16)
			if (!far && zz >= 0 && zz < 8) return __ldg(mag + self + zz);
			if (!far && zz < 0 && lzm >= 0) return __ldg(mag + uint64_t(lzm) * 512u + rxy + uint32_t(zz + 8));
			if (!far && zz >= 8 && lzp >= 0) return __ldg(mag + uint64_t(lzp) * 512u + rxy + uint32_t(zz - 8));
			return vorticity_mag_at(g, f, u, v, w, gx, gy, o.z + zz, factor);
		};
#pragma unroll
		for (int z = 0; z < 8; ++z) G[2].v[z] = ((m_at(z + fs) - m_at(z - fs)) * 0.5f) * inv_dx;
	}
	const Row8 cu = ld_row(u, self), cv = ld_row(v, self), cw = ld_row(w, self);
	const CurlRows r = curl_rows(c, u, v, w, cu, cv, factor);
	Row8 a, b, d;
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const float g0 = G[0].v[z], g1 = G[1].v[z], g2 = G[2].v[z];
		const float len = grad_norm(g0, g1, g2) + 1e-5f;
		const float Nx = __fdiv_rn(g0, len), Ny = __fdiv_rn(g1, len), Nz = __fdiv_rn(g2, len);
		const float fx = fmaf(Ny, r.wz.v[z], -__fmul_rn(Nz, r.wy.v[z]));  // a*b - c*d = fma(a, b, -rnd(c*d))
		const float fy = fmaf(Nz, r.wx.v[z], -__fmul_rn(Nx, r.wz.v[z]));
		const float fz = fmaf(Nx, r.wy.v[z], -__fmul_rn(Ny, r.wx.v[z]));
		a.v[z] = fmaf(__fmul_rn(scale, fx), dt, cu.v[z]);
		b.v[z] = fmaf(__fmul_rn(scale, fy), dt, cv.v[z]);
		d.v[z] = fmaf(__fmul_rn(scale, fz), dt, cw.v[z]);
	}
	st_row(ou, self, a);
	st_row(ov, self, b);
	st_row(ow, self, d);
}
void launch_vorticity_mag(const GridView& g, const float* const vel[3], float* mag, float inv_dx, cudaStream_t st) {
	if (g.count()) HNS_LAUNCH(k_vorticity_mag, (g.count() + 3) / 4, 256, 0, st, g, vel[0], vel[1], vel[2], mag, 0.5f * inv_dx);
}
void launch_vorticity_force(const GridView& g, const float* const vel[3], const float* mag, float* const out[3], float dt, float inv_dx, float scale,
                            float factor_scale, cudaStream_t st) {
	const int fs = int(factor_scale);  // Coord's int constructor truncates (F2I.TRUNC in the reference SASS)
	if (g.count())
		HNS_LAUNCH(k_vorticity_force, (g.count() + 3) / 4, 256, 0, st, g, vel[0], vel[1], vel[2], mag, out[0], out[1], out[2], 0.5f * inv_dx, inv_dx, scale,
		           dt, fs);
}

// =============================================================================================================
// multigrid V-cycle pieces. The reference only sketches them: restrict_to_4x4x4 / restrict_to_2x2x2 / prolongate / compute_residual
// are declared (src/Cuda/Kernels.cuh:38-49) and called from a commented-out v_cycle (src/Cuda/HNanoSolver.cu:399-507), never defined.
// Built here on the same bricks: level k+1 has cells of twice the size, its leaves are 2x2x2 leaves of level k, cell-centred
// coarsening (8 children -> 1 parent), the same 7-point operator and red-black sweep on every level, p = 0 outside the domain.
//   residual   r = rhs - (sum of the 6 neighbours - 6 p) / dx^2          (the equation the reference's sweep relaxes, Kernel.cu:621)
//   restrict   parent rhs = mean of the 8 children's residuals           (summed z pair, then y pair, then x pair)
//   prolong    p += trilinear interpolation of the parents' correction   (weights 3/4, 1/4 per axis; z, then y, then x)
// =============================================================================================================
// kNorm: also accumulates sum r^2 and sum rhs^2 in fp64 (per-thread partial sums, warp shuffles, one atomic per warp).
// kGather (with kRestrict, sharded runs): the restricted octant goes to n_gather colour-split arrays, gather[2 t] / gather[2 t + 1] = red /
// black of target t -- every rank's copy of the level-1 right-hand side, peers' ones mapped over NVLink -- instead of crhs. Plain stores:
// the flag that publishes them is raised by a later kernel in the same stream.
template <bool kMask, bool kRestrict, bool kNorm, bool kGather = false>
__global__ void __launch_bounds__(256) k_mg_residual(GridView g, const float* __restrict__ p_red, const float* __restrict__ p_blk,
                                                     const float* __restrict__ rhs_red, const float* __restrict__ rhs_blk, float inv_dx2,
                                                     const float* __restrict__ diag_red, const float* __restrict__ diag_blk,
                                                     const int32_t* __restrict__ parent,
                                                     float* __restrict__ crhs_red, float* __restrict__ crhs_blk, double* __restrict__ sums,
                                                     float* const* __restrict__ gather, int n_gather) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint64_t self = c.self();
	const bool s = (c.x + c.y) & 1;
	const Row8 cp = ld_split_row(p_red, p_blk, self, s);
	int64_t i;
	const Row8 pxp = (i = c.row(1, 0)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const Row8 pxm = (i = c.row(-1, 0)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const Row8 pyp = (i = c.row(0, 1)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const Row8 pym = (i = c.row(0, -1)) >= 0 ? ld_split_row(p_red, p_blk, i, !s) : zero_row();
	const float pzm = (i = c.zminus()) >= 0 ? __ldg((s ? p_red : p_blk) + (split_idx(uint64_t(i) & ~uint64_t(7)) + 3)) : 0.f;
	const float pzp = (i = c.zplus()) >= 0 ? __ldg((s ? p_blk : p_red) + split_idx(uint64_t(i))) : 0.f;
	const Row8 f = ld_split_row(rhs_red, rhs_blk, self, s);
	Row8 dg;
	if (kMask) dg = ld_split_row(diag_red, diag_blk, self, s);
	float r[8];
	double a = 0.0, b = 0.0;
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const float zp = z < 7 ? cp.v[z < 7 ? z + 1 : 7] : pzp;
		const float zm = z > 0 ? cp.v[z > 0 ? z - 1 : 0] : pzm;
		const float sum = ((((pxp.v[z] + pxm.v[z]) + pyp.v[z]) + pym.v[z]) + zp) + zm;
		const float lap = fmaf(kMask ? -dg.v[z] : -6.0f, cp.v[z], sum);
		r[z] = fmaf(-lap, inv_dx2, f.v[z]);
		if (kMask && dg.v[z] == 0.f) r[z] = 0.f;
		if (kNorm) a = fma(double(r[z]), double(r[z]), a), b = fma(double(f.v[z]), double(f.v[z]), b);
	}
	if (kNorm) {
#pragma unroll
		for (int o = 16; o; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o), b += __shfl_down_sync(0xffffffffu, b, o);
		if ((threadIdx.x & 31) == 0) atomicAdd(sums, a), atomicAdd(sums + 1, b);
	}
	if (kRestrict) {
		float q[4];
#pragma unroll
		for (int k = 0; k < 4; ++k) {
			q[k] = r[2 * k] + r[2 * k + 1];
			q[k] += __shfl_xor_sync(0xffffffffu, q[k], 1);  // the row at y ^ 1
			q[k] += __shfl_xor_sync(0xffffffffu, q[k], 8);  // the rows at x ^ 1
			q[k] *= 0.125f;
		}
		if (!((c.x | c.y) & 1)) {
			const int4 o = __ldg(g.origin + c.leaf);
			const int X = ((o.x >> 3) & 1) * 4 + (c.x >> 1), Y = ((o.y >> 3) & 1) * 4 + (c.y >> 1), oz = (o.z >> 3) & 1;
			const uint32_t base = uint32_t(__ldg(parent + c.leaf)) * 256u + uint32_t(X * 32 + Y * 4 + 2 * oz);
			const bool sp = (X + Y) & 1;  // parent cells z = 4 oz + k have colour (X + Y + k) & 1
			if (kGather) {
				for (int t = 0; t < n_gather; ++t) {
					float* const gr = gather[2 * t];
					float* const gb = gather[2 * t + 1];
					*reinterpret_cast<float2*>((sp ? gb : gr) + base) = make_float2(q[0], q[2]);
					*reinterpret_cast<float2*>((sp ? gr : gb) + base) = make_float2(q[1], q[3]);
				}
			} else {
				*reinterpret_cast<float2*>((sp ? crhs_blk : crhs_red) + base) = make_float2(q[0], q[2]);
				*reinterpret_cast<float2*>((sp ? crhs_red : crhs_blk) + base) = make_float2(q[1], q[3]);
			}
		}
	}
}
void launch_mg_residual(const GridView& g, const float* const p[2], const float* const rhs[2], float dx, const float* const diag[2], const int32_t* parent,
                        float* const coarse_rhs[2], double* sums, cudaStream_t st) {
	if (!g.count()) return;
	const float inv_dx2 = 1.0f / (dx * dx);
	const unsigned grid = (g.count() + 3) / 4;
	float* cr = coarse_rhs ? coarse_rhs[0] : nullptr;
	float* cb = coarse_rhs ? coarse_rhs[1] : nullptr;
	const float* dr = diag ? diag[0] : nullptr;
	const float* db = diag ? diag[1] : nullptr;
#define HNS_MG_RES(M, R, N) HNS_LAUNCH((k_mg_residual<M, R, N>), grid, 256, 0, st, g, p[0], p[1], rhs[0], rhs[1], inv_dx2, dr, db, parent, cr, cb, sums, nullptr, 0)
	const bool R = coarse_rhs != nullptr, N = sums != nullptr;
	if (diag) {
		if (R && N) HNS_MG_RES(true, true, true);
		else if (R) HNS_MG_RES(true, true, false);
		else HNS_MG_RES(true, false, true);
	} else {
		if (R && N) HNS_MG_RES(false, true, true);
		else if (R) HNS_MG_RES(false, true, false);
		else HNS_MG_RES(false, false, true);
	}
#undef HNS_MG_RES
}
void launch_mg_restrict_gather(const GridView& g, const float* const p[2], const float* const rhs[2], float dx, const int32_t* parent,
                               float* const* gather, int n_gather, cudaStream_t st) {
	if (!g.count() || n_gather <= 0) return;
	HNS_LAUNCH((k_mg_residual<false, true, false, true>), (g.count() + 3) / 4, 256, 0, st, g, p[0], p[1], rhs[0], rhs[1], 1.0f / (dx * dx), nullptr,
	           nullptr, parent, nullptr, nullptr, nullptr, gather, n_gather);
}

// sum of squares of a colour-split field over the listed leaves (fp64)
__global__ void __launch_bounds__(256) k_sum_squares(GridView g, const float* __restrict__ red, const float* __restrict__ blk, double* __restrict__ sum) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	const uint32_t q = c.self_q();
	const float4 r = ldg4(red, q), k = ldg4(blk, q);
	double a = 0.0;
	a = fma(double(r.x), double(r.x), a), a = fma(double(r.y), double(r.y), a), a = fma(double(r.z), double(r.z), a), a = fma(double(r.w), double(r.w), a);
	a = fma(double(k.x), double(k.x), a), a = fma(double(k.y), double(k.y), a), a = fma(double(k.z), double(k.z), a), a = fma(double(k.w), double(k.w), a);
#pragma unroll
	for (int o = 16; o; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
	if ((threadIdx.x & 31) == 0) atomicAdd(sum, a);
}
void launch_sum_squares(const GridView& g, const float* const f[2], double* sum, cudaStream_t st) {
	if (g.count()) HNS_LAUNCH(k_sum_squares, (g.count() + 3) / 4, 256, 0, st, g, f[0], f[1], sum);
}

// p_fine += P e_coarse. Four leaves per CTA; each stages the 6^3 parent cells around its octant of the parent leaf (4^3 + one cell of
// halo, fetched through the parent grid's neighbour table; cells outside the domain hold 0) in shared memory.
template <bool kMask>
__global__ void __launch_bounds__(256) k_mg_prolong(GridView g, float* __restrict__ p_red, float* __restrict__ p_blk, const float* __restrict__ diag_red,
                                                    const float* __restrict__ diag_blk, const int32_t* __restrict__ parent, const int32_t* __restrict__ cnbr,
                                                    const float* __restrict__ e_red, const float* __restrict__ e_blk) {
	__shared__ float tile[4][216];
	const int slot = threadIdx.x >> 6, r = threadIdx.x & 63;
	const uint32_t i = blockIdx.x * 4u + slot;
	const bool active = i < g.count();
	uint32_t leaf = 0;
	if (active) {
		leaf = g.leaf_at(i);
		const int4 o = __ldg(g.origin + leaf);
		const int bx = ((o.x >> 3) & 1) * 4 - 1, by = ((o.y >> 3) & 1) * 4 - 1, bz = ((o.z >> 3) & 1) * 4 - 1;
		const int32_t cl = __ldg(parent + leaf);
		for (int t = r; t < 216; t += 64) {
			const int X = bx + t / 36, Y = by + (t / 6) % 6, Z = bz + t % 6;  // parent-leaf-local, in [-1, 8]
			const int sl = ((X >> 3) + 1) * 9 + ((Y >> 3) + 1) * 3 + ((Z >> 3) + 1);
			const int32_t l = sl == kSlotSelf ? cl : __ldg(cnbr + uint64_t(cl) * 27u + sl);
			float v = 0.f;
			if (l >= 0) v = __ldg((((X + Y + Z) & 1) ? e_blk : e_red) + (uint32_t(l) * 256u + uint32_t((X & 7) * 32 + (Y & 7) * 4 + ((Z & 7) >> 1))));
			tile[slot][t] = v;
		}
	}
	__syncthreads();
	if (!active) return;
	const int x = r >> 3, y = r & 7;
	const float* T = tile[slot];
	const int X0 = (x >> 1) + 1, X1 = X0 + ((x & 1) ? 1 : -1), Y0 = (y >> 1) + 1, Y1 = Y0 + ((y & 1) ? 1 : -1);
	float v[8];
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const int Z0 = (z >> 1) + 1, Z1 = Z0 + ((z & 1) ? 1 : -1);
		auto zl = [&](int X, int Y) { return fmaf(0.25f, T[X * 36 + Y * 6 + Z1], 0.75f * T[X * 36 + Y * 6 + Z0]); };
		const float a0 = fmaf(0.25f, zl(X0, Y1), 0.75f * zl(X0, Y0)), a1 = fmaf(0.25f, zl(X1, Y1), 0.75f * zl(X1, Y0));
		v[z] = fmaf(0.25f, a1, 0.75f * a0);
	}
	const uint32_t q = leaf * 256u + uint32_t(x * 32 + y * 4);
	const bool s = (x + y) & 1;  // red cells of this row are z = 2j + s
	float4 R = *reinterpret_cast<const float4*>(p_red + q), B = *reinterpret_cast<const float4*>(p_blk + q);
	float4 dR = make_float4(v[s ? 1 : 0], v[s ? 3 : 2], v[s ? 5 : 4], v[s ? 7 : 6]), dB = make_float4(v[s ? 0 : 1], v[s ? 2 : 3], v[s ? 4 : 5], v[s ? 6 : 7]);
	if (kMask) {  // cells outside the domain stay 0
		const float4 WR = ldg4(diag_red, q), WB = ldg4(diag_blk, q);
		dR.x = WR.x != 0.f ? dR.x : 0.f, dR.y = WR.y != 0.f ? dR.y : 0.f, dR.z = WR.z != 0.f ? dR.z : 0.f, dR.w = WR.w != 0.f ? dR.w : 0.f;
		dB.x = WB.x != 0.f ? dB.x : 0.f, dB.y = WB.y != 0.f ? dB.y : 0.f, dB.z = WB.z != 0.f ? dB.z : 0.f, dB.w = WB.w != 0.f ? dB.w : 0.f;
	}
	R.x += dR.x, R.y += dR.y, R.z += dR.z, R.w += dR.w;
	B.x += dB.x, B.y += dB.y, B.z += dB.z, B.w += dB.w;
	*reinterpret_cast<float4*>(p_red + q) = R;
	*reinterpret_cast<float4*>(p_blk + q) = B;
}
void launch_mg_prolong(const GridView& g, float* const p[2], const float* const diag[2], const int32_t* parent, const GridView& coarse,
                       const float* const e[2], cudaStream_t st) {
	if (!g.count()) return;
	if (diag) HNS_LAUNCH(k_mg_prolong<true>, (g.count() + 3) / 4, 256, 0, st, g, p[0], p[1], diag[0], diag[1], parent, coarse.nbr, e[0], e[1]);
	else HNS_LAUNCH(k_mg_prolong<false>, (g.count() + 3) / 4, 256, 0, st, g, p[0], p[1], nullptr, nullptr, parent, coarse.nbr, e[0], e[1]);
}

// Diagonal of the operator on a coarse level from its row masks (one byte per row (x, y), bit z = cell inside the domain): 6 + extra for
// every face neighbour outside the domain, 0 for a cell outside. Why `extra`: the fine level puts p = 0 at the centre of the first
// outside voxel, i.e. one voxel beyond the last inside centre. Seen from level k that plane lies theta_k = 1/2 + 2^-(k+1) cells beyond
// the last inside centre, not one cell; a ghost value extrapolated linearly through p = 0 at that distance is p_own (1 - 1/theta_k),
// which moves extra = 1/theta_k - 1 onto the diagonal. Without it the coarse problems solve for a domain that is too large and the
// V-cycle converges at 0.5 per cycle instead of 0.05 (measured, DESIGN.md).
__global__ void __launch_bounds__(256) k_mg_diag(GridView g, const uint8_t* __restrict__ mask, float extra, float* __restrict__ diag_red,
                                                 float* __restrict__ diag_blk) {
	RowCtx c;
	if (!make_row_ctx(g, c)) return;
	auto row_mask = [&](int dx, int dy) -> uint32_t {
		const int64_t i = c.row(dx, dy);
		return i < 0 ? 0u : uint32_t(__ldg(mask + (i >> 3)));
	};
	const uint32_t m = row_mask(0, 0), mxp = row_mask(1, 0), mxm = row_mask(-1, 0), myp = row_mask(0, 1), mym = row_mask(0, -1);
	int64_t i;
	const uint32_t mzm = (i = c.zminus()) >= 0 ? (uint32_t(__ldg(mask + (i >> 3))) >> 7) & 1u : 0u;
	const uint32_t mzp = (i = c.zplus()) >= 0 ? uint32_t(__ldg(mask + (i >> 3))) & 1u : 0u;
	const uint32_t up = (m >> 1) | (mzp << 7), down = ((m << 1) & 0xffu) | mzm;  // bit z: the cell above / below z is inside
	Row8 o;
#pragma unroll
	for (int z = 0; z < 8; ++z) {
		const int outside = 6 - int(((mxp >> z) & 1u) + ((mxm >> z) & 1u) + ((myp >> z) & 1u) + ((mym >> z) & 1u) + ((up >> z) & 1u) + ((down >> z) & 1u));
		o.v[z] = ((m >> z) & 1u) ? __fadd_rn(6.0f, __fmul_rn(float(outside), extra)) : 0.f;
	}
	st_split(diag_red, diag_blk, c, o);
}
void launch_mg_diag(const GridView& g, const uint8_t* mask, float extra, float* const diag[2], cudaStream_t st) {
	if (g.count()) HNS_LAUNCH(k_mg_diag, (g.count() + 3) / 4, 256, 0, st, g, mask, extra, diag[0], diag[1]);
}

// The coarsest level when it is a single leaf: `iterations` red-black sweeps in one CTA, the brick in shared memory with a one-cell
// rim of zeros (nothing lies outside a one-leaf level). Same update as k_rbgs_split.
__global__ void __launch_bounds__(512) k_mg_coarsest(float* __restrict__ p_red, float* __restrict__ p_blk, const float* __restrict__ rhs_red,
                                                     const float* __restrict__ rhs_blk, const float* __restrict__ diag_red,
                                                     const float* __restrict__ diag_blk, float dx2, float omega, int iterations) {
	__shared__ float P[10][10][10];
	const int t = threadIdx.x, x = t >> 6, y = (t >> 3) & 7, z = t & 7;
	for (int k = t; k < 1000; k += 512) (&P[0][0][0])[k] = 0.f;
	__syncthreads();
	const int color = (x + y + z) & 1;
	const uint32_t q = uint32_t(x * 32 + y * 4 + (z >> 1));
	const float f = color ? rhs_blk[q] : rhs_red[q];
	const float dg = color ? diag_blk[q] : diag_red[q];
	const bool on = dg != 0.f;
	P[x + 1][y + 1][z + 1] = color ? p_blk[q] : p_red[q];
	__syncthreads();
	for (int it = 0; it < 2 * iterations; ++it) {
		if (on && color == (it & 1)) {
			const float v = sor_update_diag(P[x + 2][y + 1][z + 1], P[x][y + 1][z + 1], P[x + 1][y + 2][z + 1], P[x + 1][y][z + 1], P[x + 1][y + 1][z + 2],
			                                P[x + 1][y + 1][z], f, P[x + 1][y + 1][z + 1], dx2, omega, dg);
			P[x + 1][y + 1][z + 1] = v;
		}
		__syncthreads();
	}
	(color ? p_blk : p_red)[q] = P[x + 1][y + 1][z + 1];
}
void launch_mg_coarsest(float* const p[2], const float* const rhs[2], const float* const diag[2], float dx, float omega, int iterations, cudaStream_t st) {
	HNS_LAUNCH(k_mg_coarsest, 1, 512, 0, st, p[0], p[1], rhs[0], rhs[1], diag[0], diag[1], dx * dx, omega, iterations);
}

// =============================================================================================================
// brick gather / scatter for ghost-leaf exchange
// =============================================================================================================
// qshift = log2(float4 per leaf): 7 for a brick field (512 floats), 6 for one half of a colour-split field (256 floats).
// Grid-stride over all quads of all listed leaves; `dst` of the pack kernel may be a peer GPU's memory (direct ghost exchange):
// plain 16-byte stores, no fence here -- the flag that publishes them is raised by a later kernel in the same stream.
__global__ void __launch_bounds__(256) k_pack_leaves(const float* __restrict__ field, const int32_t* __restrict__ ids, float* __restrict__ dst,
                                                     uint32_t total_quads, int qshift) {
	for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < total_quads; i += gridDim.x * 256u) {
		const int32_t l = __ldg(ids + (i >> qshift));
		reinterpret_cast<float4*>(dst)[i] = __ldg(reinterpret_cast<const float4*>(field) + ((uint64_t(l) << qshift) | (i & ((1u << qshift) - 1u))));
	}
}
__global__ void __launch_bounds__(256) k_unpack_leaves(float* __restrict__ field, const int32_t* __restrict__ ids, const float* __restrict__ src,
                                                       uint32_t total_quads, int qshift) {
	for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < total_quads; i += gridDim.x * 256u) {
		const int32_t l = __ldg(ids + (i >> qshift));
		reinterpret_cast<float4*>(field)[(uint64_t(l) << qshift) | (i & ((1u << qshift) - 1u))] = reinterpret_cast<const float4*>(src)[i];
	}
}
static unsigned copy_grid(uint32_t total_quads, int max_blocks) {
	return std::min<unsigned>((total_quads + 255u) / 256u, max_blocks > 0 ? unsigned(max_blocks) : 4u * 148u);
}
void launch_pack_leaves(const float* field, const int32_t* ids, uint64_t n_ids, float* dst, int floats_per_leaf, cudaStream_t st, int max_blocks) {
	if (!n_ids) return;
	const int qshift = floats_per_leaf == 512 ? 7 : 6;
	const uint32_t total = uint32_t(n_ids) << qshift;
	HNS_LAUNCH(k_pack_leaves, copy_grid(total, max_blocks), 256, 0, st, field, ids, dst, total, qshift);
}
void launch_unpack_leaves(float* field, const int32_t* ids, uint64_t n_ids, const float* src, int floats_per_leaf, cudaStream_t st, int max_blocks) {
	if (!n_ids) return;
	const int qshift = floats_per_leaf == 512 ? 7 : 6;
	const uint32_t total = uint32_t(n_ids) << qshift;
	HNS_LAUNCH(k_unpack_leaves, copy_grid(total, max_blocks), 256, 0, st, field, ids, src, total, qshift);
}

}  // namespace hns
