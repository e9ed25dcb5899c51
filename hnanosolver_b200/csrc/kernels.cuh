// Kernel launch wrappers of libhns_b200 (definitions in kernels.cu). Velocity and the advected scalars are brick fields: float[L][512],
// voxel (x,y,z) of leaf l at l*512 + (x<<6 | y<<3 | z), velocity as three such planes (SoA). Pressure and divergence are colour-split:
// two half-brick fields float[L][256] (red = (x+y+z) even, black = odd), row (x,y) owning the quad j = z>>1.
#pragma once
#include "common.cuh"

namespace hns {

struct ScalarPtrs {
	const float* in[16];
	float* out[16];
};

// AoS float[N][3] <-> three brick fields
void launch_aos_to_soa(const float* aos, float* u, float* v, float* w, uint64_t n, cudaStream_t st);
void launch_soa_to_aos(const float* u, const float* v, const float* w, float* aos, uint64_t n, cudaStream_t st);

// Packed groups of the advection kernels (advect.cu, third generation): float4[n] per group in brick voxel order, group 0 =
// {u, v, w, first advected scalar}, group 1 = {scalars 1..4} of the list handed to launch_advect_scalars. Owned and kept current by
// the caller (struct PackedGroup, common.cuh; api.cu, "packed groups"): the launchers run the packed kernels exactly when they are
// handed groups, and never pack one themselves.
void launch_pack4(const float* a, const float* b, const float* c, const float* d, float4* out, uint64_t n, cudaStream_t st);
void launch_pack4_leaves(const int32_t* ids, uint64_t n_ids, const float* a, const float* b, const float* c, const float* d, float4* out,
                         cudaStream_t st);
bool packed_advection_enabled();  // HNS_ADVECT4=0 / hns_set_packed_advection(0) switch the third generation off (A/B)
int set_packed_advection(int on);
uint64_t packed_advection_launches();

// combustion_oxygen's field update (reference Kernel.cu:923-966) as a side job of another kernel: inputs {fuel, waste, temperature,
// flame}, their outputs, the packed group 1 and `burn`, what the expansion term of the divergence needs: burn per voxel, or -1 where
// there is no oxygen (that voxel's divergence stays as it is)
struct CombustionJob {
	const float* in[4];
	float* out[4];
	float4* grp1;
	float* burn;
	float temp_gain;
};
// temperature_buoyancy (Kernel.cu:831-847) applied by the gradient pass to the advected v it reads: temp = the combusted temperature;
// the buoyant v also goes back to `vy` (the advected velocity's y plane, as the stage of its own leaves it)
struct Buoyancy {
	const float* temp;
	float* vy;
	float dt, ambient, strength;
};
#ifdef __CUDACC__
// One voxel of combustion_oxygen: in = {fuel, waste, temperature, flame} -> out; returns burn, or -1 where oxygen < 0 (fields unchanged)
__device__ __forceinline__ float combustion_voxel(const float4 in, float temp_gain, float4& out) {
	float f = in.x;
	if (f < 0.001f) f = 0.0f;
	const float oxygen = 1.0f - f - in.y;
	out = make_float4(f, in.y, in.z, in.w);
	if (oxygen < 0.0f) return -1.0f;
	const float burn = fminf(oxygen, f);
	out.x = f - burn;
	out.y = fmaf(burn, 2.0f, in.y);
	out.w = fmaxf(in.w, fminf(1.0f, burn * 10.0f));
	out.z = fmaf(burn, temp_gain, in.z);
	return burn;
}
#endif

// advect_vector (reference src/Cuda/Kernel.cu:354-453)
// cold: device uint8[num_leaves of the grid], zero between launches -- scratch in which the staged kernel flags the leaves whose samples
// left its shared-memory region; a follow-up kernel redoes those leaves through the neighbour table and clears the flags (advect.cu)
// sdf != null: the hasCollision variant incl. its boundary tail; second generation only
// grp0 != null: the third generation, staging from packed group 0 (it holds this velocity; needs sdf == null)
// comb: the staged kernel also runs combustion_oxygen on every voxel of the grid (needs grp0)
void launch_advect_vector(const GridView& g, const float* const vel[3], float* const out[3], float dt, float inv_dx, cudaStream_t st,
                          const float* sdf, uint8_t* cold, const float4* grp0 = nullptr, const CombustionJob* comb = nullptr);

// advect_scalars (Kernel.cu:118-266) when sampler_semantics == 0; advect_scalar (Kernel.cu:269-352) per field when == 1
// advect_scalars reads element 0 of the arrays passed in for inactive voxels (a shard's local leaf 0 is global leaf 0, dist.py::make_plan)
// grp != null: the third generation, staging from packed groups 0 (S == 1) or 0 and 1 (S == 5) of these fields; needs sdf == null
void launch_advect_scalars(const GridView& g, const float* const vel[3], const ScalarPtrs& sp, int S, float dt, float inv_dx,
                           int sampler_semantics, cudaStream_t st, const float* sdf, uint8_t* cold, const float4* const grp[2] = nullptr);
// enforceCollisionBoundaries (Kernel.cu:77-116; blend_divisor 0.1, mixed_sum 0) and the boundary tails of advect_vector (:432-450;
// 1.5, 1) and subtractPressureGradient (:808-826; 0.1, 0): vel -> out (may alias), per voxel
void launch_collision_boundary(const GridView& g, const float* const vel[3], float* const out[3], const float* sdf, float inv_dx,
                               float blend_divisor, int mixed_sum, cudaStream_t st);
// divergence (Kernel.cu:499-519); burn != null: plus combustion's expansion term, div = fma(burn, expansion, div) where burn != -1
void launch_divergence(const GridView& g, const float* const vel[3], float* const div[2], float inv_dx, cudaStream_t st, const float* burn = nullptr,
                       float expansion = 0.f);
// redBlackGaussSeidelUpdate (Kernel.cu:591-623): one colour per launch, in place, on the colour-split layout (p[0] red, p[1] black)
void launch_rbgs_color(const GridView& g, const float* const div[2], float* const p[2], float dx, int color, float omega, int reverse,
                       cudaStream_t st);
// Boundary sweep of a sharded run with the ghost exchange fused in: besides writing p[color] locally, every swept quad of work item i
// is stored into the ghost copies listed in dst_peer/dst_leaf[dst_off[i] .. dst_off[i+1]) (peer index | face mask << 8 -- only rows on
// a face the peer's stencil reads are stored: bits 0..3 = x==0, x==7, y==0, y==7, bits 4..5 = a z face = every row --, leaf id in that peer's local
// numbering) through remote_pc[peer] = that peer's p[color] array mapped over NVLink. The caller raises the peers' arrival flags from
// a follow-up kernel.
struct RbgsPush {
	const uint32_t* dst_off = nullptr;
	const int32_t* dst_peer = nullptr;
	const int32_t* dst_leaf = nullptr;
	float* const* remote_pc = nullptr;
};
void launch_rbgs_color_push(const GridView& g, const float* const div[2], float* const p[2], float dx, int color, float omega, int reverse,
                            const RbgsPush& push, cudaStream_t st);
// multigrid pieces (kernels.cu, "multigrid V-cycle pieces"). Coarse levels carry `diag`, the colour-split diagonal of their operator
// (0 = cell outside the domain; launch_mg_diag builds it from row masks); diag == null means the fine level (diagonal 6, every cell
// of a leaf inside). Residual: optionally restricted into the parent level's right-hand side and/or summed in fp64 into
// sums[0..1] = {sum r^2, sum rhs^2}.
void launch_rbgs_color_masked(const GridView& g, const float* const rhs[2], float* const p[2], float dx, int color, float omega,
                              const float* const diag[2], cudaStream_t st);
void launch_mg_residual(const GridView& g, const float* const p[2], const float* const rhs[2], float dx, const float* const diag[2], const int32_t* parent,
                        float* const coarse_rhs[2], double* sums, cudaStream_t st);
// the fine level's residual restricted, as launch_mg_residual with a parent level, but stored into n_gather colour-split arrays: gather[2 t],
// gather[2 t + 1] = red / black half of target t (a sharded run's level-1 right-hand side on every rank, dist.cu)
void launch_mg_restrict_gather(const GridView& g, const float* const p[2], const float* const rhs[2], float dx, const int32_t* parent,
                               float* const* gather, int n_gather, cudaStream_t st);
void launch_sum_squares(const GridView& g, const float* const f[2], double* sum, cudaStream_t st);
void launch_mg_prolong(const GridView& g, float* const p[2], const float* const diag[2], const int32_t* parent, const GridView& coarse,
                       const float* const e[2], cudaStream_t st);
void launch_mg_diag(const GridView& g, const uint8_t* mask, float extra, float* const diag[2], cudaStream_t st);
void launch_mg_coarsest(float* const p[2], const float* const rhs[2], const float* const diag[2], float dx, float omega, int iterations, cudaStream_t st);
// subtractPressureGradient (Kernel.cu:765-829)
// grp0 != null: the result also goes into the packed advection group 0 as float4 {u, v, w, s0 (or 0)} per voxel
// buoy != null: the buoyancy force is added to vel[1] first (vel = the advected velocity, out of place)
void launch_subtract_gradient(const GridView& g, const float* const vel[3], const float* const p[2], float* const out[3], float inv_dx,
                              cudaStream_t st, float4* grp0 = nullptr, const float* s0 = nullptr, const Buoyancy* buoy = nullptr);
// vorticityConfinement (Kernel.cu:969-1025), out of place, in two launches: |curl| of every listed leaf into the plane `mag`, then
// vel -> out using mag at the six offset positions (a sharded run exchanges the ghost leaves of `mag` in between)
void launch_vorticity_mag(const GridView& g, const float* const vel[3], float* mag, float inv_dx, cudaStream_t st);
void launch_vorticity_force(const GridView& g, const float* const vel[3], const float* mag, float* const out[3], float dt, float inv_dx, float scale,
                            float factor_scale, cudaStream_t st);
// combustion_oxygen (Kernel.cu:923-966) and temperature_buoyancy (Kernel.cu:831-847, in place on the y component)
// update_div = false: the field updates only; the expansion term has already gone into the divergence (launch_combustion_divergence)
void launch_combustion_oxygen(const float* fuel, const float* waste, const float* temp, float* const div[2], const float* flame, float* oFuel,
                              float* oWaste, float* oTemp, float* oFlame, float temp_gain, float expansion, uint64_t n, cudaStream_t st,
                              bool update_div = true);
// div += burn * expansion alone (Kernel.cu:963): needs only fuel and waste
void launch_combustion_divergence(const float* fuel, const float* waste, float* const div[2], float expansion, uint64_t n, cudaStream_t st);
void launch_buoyancy(float* const vel[3], const float* temp, float dt, float ambient, float strength, uint64_t n, cudaStream_t st);
// both in one pass; the four outputs additionally as float4 {fuel, waste, temperature, flame} into a packed advection group
void launch_combustion_buoyancy_packed(const float* fuel, const float* waste, const float* temp, float* const div[2], const float* flame, float* oFuel,
                                       float* oWaste, float* oTemp, float* oFlame, float4* grp, float* const vel[3], float temp_gain, float expansion,
                                       float dt, float ambient, float strength, uint64_t n, cudaStream_t st, bool update_div = true,
                                       bool buoyancy = true);
// the buoyancy force from the temperature combustion_oxygen WILL write, recomputed from fuel, waste and temperature
void launch_buoyancy_from_inputs(const float* fuel, const float* waste, const float* temp, float* const vel[3], float temp_gain, float dt,
                                 float ambient, float strength, uint64_t n, cudaStream_t st);
// GridView::list_nbr for a work list: out[n][27]
void launch_gather_nbr_rows(const int32_t* nbr, const int32_t* list, uint32_t n, int32_t* out, cudaStream_t st);
// whole-brick gather / scatter by leaf id (ghost exchange)
// max_blocks > 0 caps the grid: a background exchange then never takes more than that many CTA slots from a concurrent sweep
void launch_pack_leaves(const float* field, const int32_t* ids, uint64_t n_ids, float* dst, int floats_per_leaf, cudaStream_t st, int max_blocks = 0);
void launch_unpack_leaves(float* field, const int32_t* ids, uint64_t n_ids, const float* src, int floats_per_leaf, cudaStream_t st, int max_blocks = 0);
// colour-split (red, black) -> brick order
void launch_split_to_brick(const float* const f[2], float* out, uint64_t n, cudaStream_t st);
// compSum of a source grid (struct hns_source: keys, values, components) into brick fields, field[0..components): every voxel of every
// leaf of g -- its work list is ignored -- becomes value + s, s = the source's value where it has a leaf at that origin and +0.0f
// elsewhere (which turns -0.0 into +0.0, as compSum against a background tile does)
void launch_add_source(const GridView& g, const hns_source& src, float* const field[3], cudaStream_t st);
// adds to *count the source leaves whose origin is not a leaf of g
void launch_count_leaves_outside(const GridView& g, const hns_source& src, unsigned long long* count, cudaStream_t st);

}  // namespace hns
