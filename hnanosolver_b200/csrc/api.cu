// C ABI of libhns_b200 (include/hns_b200.h): resident simulation state, the frame, and the one-shot host-sidecar launchers.
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "kernels.cuh"

namespace hns {

static thread_local std::string t_error;
void set_error(const std::string& msg) { t_error = msg; }
int fail(int code, const std::string& msg) {
	t_error = msg;
	return code;
}

// omega exactly as Compute() evaluates it (reference src/Cuda/HNanoSolver.cu:257): float sinf of float(3.14159)*voxelSize
static inline float omega_compute(float voxelSize) { return 2.0f / (1.0f + sinf(static_cast<float>(3.14159) * voxelSize)); }
// ... and as pressure_projection_idx does (reference src/Cuda/PressureProjection.cu:53): double sin, narrowed at the kernel call
static inline float omega_project(float voxelSize) { return float(2.0f / (1.0f + sin(3.14159 * voxelSize))); }

static void pressure_sweeps(hns_state* s, int iterations, float dx, float omega, unsigned flags, cudaStream_t st) {
	const GridView g = s->view();
	cudaMemsetAsync(s->p[0], 0, (s->n / 2) * sizeof(float), st);  // initial guess 0 (HNanoSolver.cu:113)
	cudaMemsetAsync(s->p[1], 0, (s->n / 2) * sizeof(float), st);
	const bool alternate = !(flags & 2u);  // red sweeps walk the leaves front to back, black sweeps back to front (L2 reuse)
	for (int it = 0; it < iterations; ++it) {
		launch_rbgs_color(g, s->div, s->p, dx, 0, omega, 0, st);
		launch_rbgs_color(g, s->div, s->p, dx, 1, omega, alternate ? 1 : 0, st);
	}
}

static int pressure_solve(hns_state* s, int iterations, float dx, float omega, unsigned flags, cudaStream_t st) {
	auto& G = s->solve_graph;
	const bool want_graph = iterations > 0;
	const GridView view = s->view();
	if (want_graph && !(G.exec && std::memcmp(&G.view, &view, sizeof(view)) == 0 && G.p == s->p[0] && G.div == s->div[0] && G.iterations == iterations &&
	                    G.flags == flags && G.omega == omega && G.dx == dx)) {
		if (G.exec) cudaGraphExecDestroy(G.exec), G.exec = nullptr;
		if (!s->capture_stream && cudaStreamCreateWithFlags(&s->capture_stream, cudaStreamNonBlocking) != cudaSuccess) cudaGetLastError();
		cudaGraph_t graph = nullptr;
		if (s->capture_stream && cudaStreamBeginCapture(s->capture_stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
			const uint64_t before = g_launches.load();
			pressure_sweeps(s, iterations, dx, omega, flags, s->capture_stream);  // capture executes nothing
			const cudaError_t e = cudaStreamEndCapture(s->capture_stream, &graph);
			G.launches = g_launches.load() - before;
			g_launches.fetch_sub(G.launches);  // every replay counts them
			if (e != cudaSuccess || !graph || cudaGraphInstantiate(&G.exec, graph, 0) != cudaSuccess) G.exec = nullptr;
			if (graph) cudaGraphDestroy(graph);
		}
		cudaGetLastError();
		std::memcpy(&G.view, &view, sizeof(view));
		G.p = s->p[0], G.div = s->div[0], G.iterations = iterations, G.flags = flags, G.omega = omega, G.dx = dx;
	}
	if (want_graph && G.exec) {
		HNS_CUDA(cudaGraphLaunch(G.exec, st));
		g_launches.fetch_add(G.launches, std::memory_order_relaxed);
	} else {
		pressure_sweeps(s, iterations, dx, omega, flags, st);
	}
	return HNS_OK;
}

// ---- packed groups of the advection kernels (advect.cu, third generation) ------------------------------------------------------------
// The kernels that write the velocity and the scalars right before an advection pass also write them as float4 groups:
// subtractPressureGradient -> group 0 {u, v, w, first advected scalar}, combustion -> group 1 {fuel, waste, temperature, flame}.
// Every producer records what it wrote with group_written: the brick field behind each lane and the version counters
// (hns_state::vel_version / sc_version, bumped by every entry point that may overwrite the brick fields). A consumer asks
// group_if_current for the fields it is about to read and gets the group only while those lanes mirror exactly those buffers and the
// counters the lanes depend on have not moved since; otherwise it runs the second-generation kernels on the brick fields. Not used
// with collision data (the boundary pass rewrites the velocity after the gradient). In a sharded frame the kernels write the groups of
// the owned leaves only; dist.cu re-packs the ghost leaves after the exchange in front of the advection pass and records them again.
static bool groups_allowed(const hns_state* s) { return s->n && !s->collision_sdf() && packed_advection_enabled(); }
static bool ensure_group(hns_state* s, int j) {
	float4*& buf = s->grp[j].buf;
	if (!buf && cudaMalloc(&buf, s->n * sizeof(float4)) != cudaSuccess) {
		cudaGetLastError();
		buf = nullptr;
	}
	return buf != nullptr;
}
// The scalars an advection pass moves, in the order it moves them: every scalar except the one marked as not advected
// ("collision_sdf", HNanoSolver.cu:327). When the state carries exactly one scalar besides the four combustion fields -- the
// reference's all-in-one frame: density + fuel, waste, temperature, flame -- that one goes first and the combustion fields follow in
// the order combustion packs them, so that they form group 1 (the fields are advected independently: the order changes no value).
// A sharded run keeps the state's own order (its exchanges go by position); it packs when that order already fits.
static int advect_list(const hns_state* s, int* idx) {
	int S = 0;
	for (int i = 0; i < s->n_scalars; ++i)
		if (i != s->skip_scalar) idx[S++] = i;
	if (S == 5 && s->comb_enabled && !s->active && groups_allowed(s)) {
		int other = -1, n_other = 0;
		for (int k = 0; k < S; ++k) {
			bool comb = false;
			for (int c : s->comb_idx) comb |= c == idx[k];
			if (!comb) other = idx[k], ++n_other;
		}
		if (n_other == 1) {
			idx[0] = other;
			for (int c = 0; c < 4; ++c) idx[1 + c] = s->comb_idx[c];
		}
	}
	return S;
}
static bool combustion_packs(const hns_state* s) {  // will advect_scalars find the combustion fields as its scalars 1..4?
	int idx[16];
	if (!s->comb_enabled || !groups_allowed(s) || advect_list(s, idx) != 5) return false;
	for (int c = 0; c < 4; ++c)
		if (idx[1 + c] != s->comb_idx[c]) return false;
	return true;
}

// The fields the advection passes read from group j, which are also what its producers pack: {u, v, w, first advected scalar} and
// {advected scalars 1..4}; a lane past the end of the list is null.
void group_wants(const hns_state* s, int j, const float* want[4]) {
	int idx[16];
	const int S = advect_list(s, idx);
	for (int k = 0; k < 4; ++k) {
		const int i = j == 0 ? k - 3 : k + 1;  // position in the list; lanes 0..2 of group 0 are the velocity
		want[k] = i < 0 ? s->vel[k] : i < S ? s->sc[idx[i]] : nullptr;
	}
}
// Group j if every non-null lane of `want` is the field the group mirrors and that field's counter has not moved since the group was
// written: vel_version for lanes 0..2 of group 0, sc_version for every other lane. Null otherwise.
const float4* group_if_current(const hns_state* s, int j, const float* const want[4]) {
	const PackedGroup& g = s->grp[j];
	if (!groups_allowed(s) || !g.buf) return nullptr;
	for (int k = 0; k < 4; ++k) {
		const bool velocity = j == 0 && k < 3;
		if (want[k] && (g.src[k] != want[k] || (velocity ? g.vel_version != s->vel_version : g.sc_version != s->sc_version))) return nullptr;
	}
	return g.buf;
}
// after a producer has written group j from `src` and bumped the counters of the fields it wrote
void group_written(hns_state* s, int j, const float* const src[4]) {
	PackedGroup& g = s->grp[j];
	std::copy(src, src + 4, g.src);
	g.vel_version = s->vel_version, g.sc_version = s->sc_version;
}

static const float4* velocity_group(const hns_state* s) {  // group 0 as advect_vector reads it: the velocity lanes only
	const float* const want[4] = {s->vel[0], s->vel[1], s->vel[2], nullptr};
	return group_if_current(s, 0, want);
}
static int stage_advect_velocity(hns_state* s, float dt, float inv, cudaStream_t st, const CombustionJob* comb = nullptr) {
	launch_advect_vector(s->view(), s->vel, s->adv, dt, inv, st, s->collision_sdf(), s->cold, velocity_group(s), comb);
	return HNS_OK;
}
// the combustion fields' outputs become the current fields (HNanoSolver.cu:239-246); `packed`: group 1 was written along with them
static void combustion_swap(hns_state* s, bool packed) {
	const int* ci = s->comb_idx;
	for (int c = 0; c < 4; ++c) std::swap(s->sc[ci[c]], s->sc_out[ci[c]]);
	++s->sc_version;
	if (packed) {
		const float* const src[4] = {s->sc[ci[0]], s->sc[ci[1]], s->sc[ci[2]], s->sc[ci[3]]};
		group_written(s, 1, src);
	}
}
// update_div / buoyancy = false: the expansion term is already in the divergence (launch_combustion_divergence), the buoyancy force
// already in the advected velocity (launch_buoyancy_from_inputs): frames fed over PCIe, see frame()
static int stage_combustion_buoyancy(hns_state* s, float dt, cudaStream_t st, bool update_div = true, bool buoyancy = true) {
	const int iF = s->comb_idx[0], iW = s->comb_idx[1], iT = s->comb_idx[2], iL = s->comb_idx[3];
	const bool packed = combustion_packs(s) && ensure_group(s, 1);
	if (packed) {
		launch_combustion_buoyancy_packed(s->sc[iF], s->sc[iW], s->sc[iT], s->div, s->sc[iL], s->sc_out[iF], s->sc_out[iW], s->sc_out[iT], s->sc_out[iL],
		                                  s->grp[1].buf, s->adv, s->comb.temperatureRelease, s->comb.expansionRate, dt, s->comb.ambientTemp,
		                                  s->comb.buoyancyStrength, s->n, st, update_div, buoyancy);
	} else {
		launch_combustion_oxygen(s->sc[iF], s->sc[iW], s->sc[iT], s->div, s->sc[iL], s->sc_out[iF], s->sc_out[iW], s->sc_out[iT], s->sc_out[iL],
		                         s->comb.temperatureRelease, s->comb.expansionRate, s->n, st, update_div);
		if (buoyancy) launch_buoyancy(s->adv, s->sc_out[iT], dt, s->comb.ambientTemp, s->comb.buoyancyStrength, s->n, st);
	}
	combustion_swap(s, packed);
	return HNS_OK;
}
// adv - grad p -> vel (from_advected), or in place on vel (the stand-alone projection; every thread reads only its own velocity row)
// buoy: the buoyancy force goes onto the advected velocity in the same pass (frame() with the fused combustion pass)
static int stage_subtract_gradient(hns_state* s, bool from_advected, float inv, cudaStream_t st, bool allow_group = true, const Buoyancy* buoy = nullptr) {
	const bool packed = allow_group && from_advected && groups_allowed(s) && ensure_group(s, 0);
	const float* src[4];
	group_wants(s, 0, src);
	launch_subtract_gradient(s->view(), from_advected ? s->adv : s->vel, s->p, s->vel, inv, st, packed ? s->grp[0].buf : nullptr,
	                         packed ? src[3] : nullptr, buoy);
	++s->vel_version;
	if (packed) group_written(s, 0, src);
	return HNS_OK;
}
static int stage_advect_scalars(hns_state* s, float dt, float inv, int sampler_semantics, cudaStream_t st) {
	int idx[16];
	const int S = advect_list(s, idx);
	if (!S || !s->n) return HNS_OK;
	ScalarPtrs sp{};
	for (int k = 0; k < S; ++k) sp.in[k] = s->sc[idx[k]], sp.out[k] = s->sc_out[idx[k]];
	// the packed kernels move one scalar (group 0) or five (groups 0 and 1)
	const int n_groups = S == 1 ? 1 : S == 5 ? 2 : 0;
	const float4* grp[2] = {};
	bool packed = n_groups > 0;
	for (int j = 0; j < n_groups; ++j) {
		const float* want[4];
		group_wants(s, j, want);
		packed &= (grp[j] = group_if_current(s, j, want)) != nullptr;
	}
	launch_advect_scalars(s->view(), s->vel, sp, S, dt, inv, sampler_semantics, st, s->collision_sdf(), s->cold, packed ? grp : nullptr);
	for (int k = 0; k < S; ++k) std::swap(s->sc[idx[k]], s->sc_out[idx[k]]);
	++s->sc_version;
	return HNS_OK;
}

static ScalarPtrs scalar_ptrs(const hns_state* s) {
	ScalarPtrs sp{};
	for (int i = 0; i < s->n_scalars; ++i) sp.in[i] = s->sc[i], sp.out[i] = s->sc_out[i];
	return sp;
}

// One frame on resident state = Compute() (reference src/Cuda/HNanoSolver.cu:159-356) without the host copies:
//   advect_vector -> [vorticityConfinement, out of place] -> divergence -> [combustion_oxygen -> temperature_buoyancy] ->
//   iterations x (red, black) -> subtractPressureGradient -> advect_scalars over all scalar fields.
// `voxel_size` is the launcher argument (the reference's kernels use it, not the grid's map).
// Optional stream dependencies of a frame whose inputs arrive / outputs leave on a copy stream while it runs (hns_compute_sim):
// the frame waits for `combustion_inputs` before the combustion stage and for `scalar_inputs` before advect_scalars, and records
// `velocity_done` once the projected velocity is final.
// vorticityConfinement on the advected velocity (reference HNanoSolver.cu:172-176), out of place into scratch planes that then trade
// places with s->adv. A zero scale, or a factorScale that truncates to a zero offset (the SOP's default 0.5), makes the force
// (+-0) * dt: the pass is skipped (identical values; only the sign of an exact zero could differ).
static bool vorticity_active(float scale, float factor_scale) { return scale != 0.0f && int(factor_scale) != 0; }
static int vorticity_scratch(hns_state* s, cudaStream_t st) {
	for (float*& v : s->vort)
		if (!v) {
			HNS_CUDA(cudaMalloc(&v, std::max<size_t>(s->n, 1) * sizeof(float)));
			HNS_CUDA(cudaMemsetAsync(v, 0, std::max<size_t>(s->n, 1) * sizeof(float), st));
		}
	return HNS_OK;
}
static int vorticity_mag(hns_state* s, float inv_dx, cudaStream_t st) {
	int rc = vorticity_scratch(s, st);
	if (rc) return rc;
	launch_vorticity_mag(s->view(), s->adv, s->vort[3], inv_dx, st);
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
static int vorticity_force(hns_state* s, float dt, float inv_dx, float scale, float factor_scale, cudaStream_t st) {
	int rc = vorticity_scratch(s, st);
	if (rc) return rc;
	launch_vorticity_force(s->view(), s->adv, s->vort[3], s->vort, dt, inv_dx, scale, factor_scale, st);
	for (int c = 0; c < 3; ++c) std::swap(s->adv[c], s->vort[c]);
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
static int vorticity_pass(hns_state* s, float dt, float inv_dx, float scale, float factor_scale, cudaStream_t st) {
	if (!vorticity_active(scale, factor_scale) || !s->n) return HNS_OK;
	int rc = vorticity_mag(s, inv_dx, st);
	return rc ? rc : vorticity_force(s, dt, inv_dx, scale, factor_scale, st);
}

struct FrameDeps {
	cudaEvent_t fuel_waste_inputs = nullptr, temperature_input = nullptr, combustion_inputs = nullptr, scalar_inputs = nullptr, velocity_done = nullptr;
};
// HNS_FUSED_COMBUSTION=0: the combustion stage as a pass of its own (A/B switch, read at every frame)
static bool fused_combustion_enabled() {
	const char* e = std::getenv("HNS_FUSED_COMBUSTION");
	return !e || std::atoi(e) != 0;
}
// Combustion without a pass of its own: its field update rides in the packed advect_vector kernel (bound by the shared-memory pipe,
// with most of the HBM bandwidth idle), which also writes the burn per voxel; the expansion term goes into the divergence pass, the
// buoyancy force into the gradient pass. Same arithmetic on the same values. Only for the frame on resident fields (no collision data,
// no work list) whose advect_vector takes the packed path and whose advect_scalars finds the combustion fields as group 1.
static bool fused_combustion(hns_state* s, const FrameDeps* deps) {
	if (deps || !s->comb_enabled || s->active || !fused_combustion_enabled() || !combustion_packs(s) || !velocity_group(s) || !ensure_group(s, 1))
		return false;
	if (!s->burn && cudaMalloc(&s->burn, s->n * sizeof(float)) != cudaSuccess) {
		cudaGetLastError();
		s->burn = nullptr;
	}
	return s->burn != nullptr;
}
static int frame(hns_state* s, int iterations, float dt, float voxel_size, unsigned flags, cudaStream_t st, cudaEvent_t ev_p0 = nullptr,
                 cudaEvent_t ev_p1 = nullptr, const FrameDeps* deps = nullptr) {
	const GridView g = s->view();
	const float h = voxel_size, inv = 1.0f / h;
	const float* sdf = s->collision_sdf();
	if (sdf) launch_collision_boundary(g, s->vel, s->vel, sdf, inv, 0.1f, 0, st);  // enforceCollisionBoundaries, HNanoSolver.cu:153-157
	const bool fused = fused_combustion(s, deps);
	if (fused) {
		const int* ci = s->comb_idx;
		const CombustionJob job{{s->sc[ci[0]], s->sc[ci[1]], s->sc[ci[2]], s->sc[ci[3]]},
		                        {s->sc_out[ci[0]], s->sc_out[ci[1]], s->sc_out[ci[2]], s->sc_out[ci[3]]}, s->grp[1].buf, s->burn,
		                        s->comb.temperatureRelease};
		stage_advect_velocity(s, dt, inv, st, &job);
		combustion_swap(s, true);
	} else {
		stage_advect_velocity(s, dt, inv, st);
	}
	if (s->comb_enabled) {
		const int rc = vorticity_pass(s, dt, inv, s->comb.vorticityScale, s->comb.factorScale, st);
		if (rc) return rc;
	}
	launch_divergence(g, s->adv, s->div, inv, st, fused ? s->burn : nullptr, s->comb.expansionRate);
	// Inputs still arriving (hns_compute_sim). What the projected velocity -- the first result that can leave again -- depends on:
	// the pressure solve needs of the combustion stage only the term it adds to the divergence, i.e. fuel and waste; the gradient pass
	// needs the buoyancy force, i.e. the temperature combustion will write, i.e. fuel, waste and temperature. So: expansion term as soon
	// as fuel and waste have landed, solve, buoyancy from the three inputs, gradient, velocity on its way back; the field updates
	// themselves (they need the flame field too) and advect_scalars (every scalar) follow while the velocity is already crossing PCIe in
	// the other direction. Same arithmetic on the same values, another order of independent steps.
	const bool split_combustion = s->comb_enabled && deps && deps->fuel_waste_inputs && deps->temperature_input;
	if (split_combustion) {
		HNS_CUDA(cudaStreamWaitEvent(st, deps->fuel_waste_inputs, 0));
		launch_combustion_divergence(s->sc[s->comb_idx[0]], s->sc[s->comb_idx[1]], s->div, s->comb.expansionRate, s->n, st);
	} else {
		if (deps && deps->combustion_inputs) HNS_CUDA(cudaStreamWaitEvent(st, deps->combustion_inputs, 0));
		if (s->comb_enabled && !fused) stage_combustion_buoyancy(s, dt, st);
	}
	if (ev_p0) cudaEventRecord(ev_p0, st);
	// the reference's solve, or -- opted in with hns_state_set_pressure_solver -- a fixed number of multigrid V-cycles
	int rc = s->mg ? mg_pressure_solve(s, s->mg, s->mg_cycles, 0.0, s->mg_nu[0], s->mg_nu[1], s->mg_omega, st)
	               : pressure_solve(s, iterations, h, omega_compute(h), flags, st);
	if (rc) return rc;
	if (ev_p1) cudaEventRecord(ev_p1, st);
	if (split_combustion) {
		HNS_CUDA(cudaStreamWaitEvent(st, deps->temperature_input, 0));
		launch_buoyancy_from_inputs(s->sc[s->comb_idx[0]], s->sc[s->comb_idx[1]], s->sc[s->comb_idx[2]], s->adv, s->comb.temperatureRelease, dt,
		                            s->comb.ambientTemp, s->comb.buoyancyStrength, s->n, st);
	} else if (deps && deps->scalar_inputs && groups_allowed(s)) {
		// with packed groups the gradient pass also reads the first advected scalar: it has to have landed by now, not only by advect_scalars
		HNS_CUDA(cudaStreamWaitEvent(st, deps->scalar_inputs, 0));
	}
	Buoyancy buoy{};
	if (fused) buoy = Buoyancy{s->sc[s->comb_idx[2]], s->adv[1], dt, s->comb.ambientTemp, s->comb.buoyancyStrength};
	stage_subtract_gradient(s, true, inv, st, !split_combustion, fused ? &buoy : nullptr);  // split: group 0 is packed below, once its scalar has landed
	if (sdf) {
		launch_collision_boundary(g, s->vel, s->vel, sdf, inv, 0.1f, 0, st);  // the tail of subtractPressureGradient, Kernel.cu:808-826
		launch_collision_boundary(g, s->vel, s->vel, sdf, inv, 0.1f, 0, st);  // enforceCollisionBoundaries again, HNanoSolver.cu:292-296
	}
	if (deps && deps->velocity_done) {
		launch_soa_to_aos(s->vel[0], s->vel[1], s->vel[2], s->aos, s->n, st);
		HNS_CUDA(cudaEventRecord(deps->velocity_done, st));
	}
	if (split_combustion) {
		if (deps->combustion_inputs) HNS_CUDA(cudaStreamWaitEvent(st, deps->combustion_inputs, 0));
		stage_combustion_buoyancy(s, dt, st, false, false);
	}
	if (deps && deps->scalar_inputs) HNS_CUDA(cudaStreamWaitEvent(st, deps->scalar_inputs, 0));
	if (split_combustion && !sdf && groups_allowed(s) && ensure_group(s, 0)) {
		const float* src[4];
		group_wants(s, 0, src);
		launch_pack4(src[0], src[1], src[2], src[3], s->grp[0].buf, s->n, st);  // 0.2 ms behind 40 ms of transfers
		group_written(s, 0, src);
	}
	stage_advect_scalars(s, dt, inv, 0, st);
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

// field ids of the ghost-exchange interface: 0..2 velocity, 3..5 advected velocity, 6/7 pressure red/black, 8/9 divergence red/black,
// 10+i scalar i. Pressure and divergence halves hold 256 floats per leaf, everything else 512.
float* field_ptr(hns_state* s, int field, int* floats_per_leaf) {
	*floats_per_leaf = (field >= 6 && field <= 9) ? 256 : 512;
	if (field >= 0 && field < 3) return s->vel[field];
	if (field >= 3 && field < 6) return s->adv[field - 3];
	if (field == 6 || field == 7) return s->p[field - 6];
	if (field == 8 || field == 9) return s->div[field - 8];
	if (field >= 10 && field < 10 + s->n_scalars) return s->sc[field - 10];
	if (field == 26) return s->vort[3];  // |curl| plane of the vorticity confinement (null until first used)
	return nullptr;
}
void field_written(hns_state* s, int field) {
	if (field >= 0 && field < 3) ++s->vel_version;
	if (field >= 10) ++s->sc_version;
}

}  // namespace hns

using namespace hns;

#define HNS_REQUIRE(cond, msg) \
	if (!(cond)) return fail(HNS_ERR_INVALID_ARGUMENT, msg)

extern "C" {

int hns_abi_version(void) { return HNS_B200_ABI_VERSION; }
const char* hns_last_error(void) { return t_error.c_str(); }
uint64_t hns_launch_count(void) { return g_launches.load(); }
void hns_launch_count_reset(void) { g_launches.store(0); }
int hns_set_packed_advection(int on) { return set_packed_advection(on); }
uint64_t hns_packed_advection_launches(void) { return packed_advection_launches(); }
int hns_set_device(int device) {
	HNS_CUDA(cudaSetDevice(device));
	return HNS_OK;
}

// ---- resident state ---------------------------------------------------------------------------------------------
int hns_state_create(const hns_grid* g, int n_scalars, hns_state** out) {
	HNS_REQUIRE(g && out, "null argument");
	HNS_REQUIRE(n_scalars >= 0 && n_scalars <= 16, "n_scalars must be in [0, 16]");
	*out = nullptr;
	auto* s = new hns_state();
	s->grid = g;
	s->n = g->num_leaves * 512;
	s->n_scalars = n_scalars;
	const size_t fb = std::max<size_t>(s->n, 1) * sizeof(float);
	std::vector<float**> all;
	for (int c = 0; c < 3; ++c) all.push_back(&s->vel[c]), all.push_back(&s->adv[c]);
	std::vector<float**> halves = {&s->div[0], &s->div[1]};
	for (int i = 0; i < n_scalars; ++i) all.push_back(&s->sc[i]), all.push_back(&s->sc_out[i]);
	for (int pass = 0; pass < 2; ++pass)
		for (float** p : pass ? halves : all) {
			const size_t bytes = pass ? std::max<size_t>(fb / 2, 4) : fb;
			const cudaError_t e = cudaMalloc(p, bytes);
			if (e != cudaSuccess) {
				const std::string msg = std::string("cudaMalloc(field): ") + cudaGetErrorString(e);
				hns_state_destroy(s);
				return fail(HNS_ERR_CUDA, msg);
			}
			cudaMemset(*p, 0, bytes);
		}
	{
		const size_t nb = std::max<size_t>(g->num_leaves, 1);
		if (cudaMalloc(&s->cold, nb) != cudaSuccess) {
			hns_state_destroy(s);
			return fail(HNS_ERR_CUDA, "cudaMalloc(leaf flags)");
		}
		cudaMemset(s->cold, 0, nb);
	}
	{
		// red and black pressure halves in ONE allocation: a single L2 access-policy window (and a single IPC handle) covers both
		const cudaError_t e = cudaMalloc(&s->p[0], fb);
		if (e != cudaSuccess) {
			const std::string msg = std::string("cudaMalloc(pressure): ") + cudaGetErrorString(e);
			hns_state_destroy(s);
			return fail(HNS_ERR_CUDA, msg);
		}
		cudaMemset(s->p[0], 0, fb);
		s->p[1] = s->p[0] + s->n / 2;
	}
	*out = s;
	return HNS_OK;
}

void hns_state_destroy(hns_state* s) {
	if (!s) return;
	for (int c = 0; c < 3; ++c) cudaFree(s->vel[c]), cudaFree(s->adv[c]);
	cudaFree(s->div[0]), cudaFree(s->div[1]), cudaFree(s->p[0]);  // p[1] lives in p[0]'s allocation
	for (int i = 0; i < 16; ++i) cudaFree(s->sc[i]), cudaFree(s->sc_out[i]);
	cudaFree(s->aos);
	cudaFree(s->cold);
	for (const PackedGroup& g : s->grp) cudaFree(g.buf);
	cudaFree(s->burn);
	cudaFree(s->d_sums);
	if (s->solve_graph.exec) cudaGraphExecDestroy(s->solve_graph.exec);
	if (s->capture_stream) cudaStreamDestroy(s->capture_stream);
	for (float* v : s->vort) cudaFree(v);
	delete s;
}

static int ensure_aos(hns_state* s) {
	if (!s->aos) HNS_CUDA(cudaMalloc(&s->aos, std::max<size_t>(s->n, 1) * 3 * sizeof(float)));
	return HNS_OK;
}

int hns_state_upload_velocity(hns_state* s, const float* host) {
	HNS_REQUIRE(s && host, "null argument");
	int rc = ensure_aos(s);
	if (rc) return rc;
	HNS_CUDA(cudaMemcpy(s->aos, host, s->n * 12, cudaMemcpyHostToDevice));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], s->n, 0);
	HNS_CUDA(cudaDeviceSynchronize());
	++s->vel_version;
	return HNS_OK;
}
int hns_state_download_velocity(hns_state* s, float* host) {
	HNS_REQUIRE(s && host, "null argument");
	int rc = ensure_aos(s);
	if (rc) return rc;
	launch_soa_to_aos(s->vel[0], s->vel[1], s->vel[2], s->aos, s->n, 0);
	HNS_CUDA(cudaMemcpy(host, s->aos, s->n * 12, cudaMemcpyDeviceToHost));
	return HNS_OK;
}
int hns_state_upload_scalar(hns_state* s, int i, const float* host) {
	HNS_REQUIRE(s && host && i >= 0 && i < s->n_scalars, "bad argument");
	HNS_CUDA(cudaMemcpy(s->sc[i], host, s->n * 4, cudaMemcpyHostToDevice));
	++s->sc_version;
	return HNS_OK;
}
int hns_state_download_scalar(hns_state* s, int i, float* host) {
	HNS_REQUIRE(s && host && i >= 0 && i < s->n_scalars, "bad argument");
	HNS_CUDA(cudaMemcpy(host, s->sc[i], s->n * 4, cudaMemcpyDeviceToHost));
	return HNS_OK;
}
int hns_state_download_aux(hns_state* s, int which, float* host) {
	HNS_REQUIRE(s && host, "null argument");
	if (which == 0 || which == 1) {
		int rc = ensure_aos(s);  // staging buffer doubles as scratch for the colour-split -> brick-order conversion
		if (rc) return rc;
		launch_split_to_brick(which == 0 ? s->div : s->p, s->aos, s->n, 0);
		HNS_CUDA(cudaMemcpy(host, s->aos, s->n * 4, cudaMemcpyDeviceToHost));
	} else if (which == 2) {
		int rc = ensure_aos(s);
		if (rc) return rc;
		launch_soa_to_aos(s->adv[0], s->adv[1], s->adv[2], s->aos, s->n, 0);
		HNS_CUDA(cudaMemcpy(host, s->aos, s->n * 12, cudaMemcpyDeviceToHost));
	} else {
		return fail(HNS_ERR_INVALID_ARGUMENT, "which must be 0, 1 or 2");
	}
	return HNS_OK;
}

int hns_state_set_combustion(hns_state* s, int enabled, int i_fuel, int i_waste, int i_temperature, int i_flame, const hns_combustion_params* params) {
	HNS_REQUIRE(s, "null state");
	if (!enabled) {
		s->comb_enabled = false;
		return HNS_OK;
	}
	HNS_REQUIRE(params, "null params");
	const int idx[4] = {i_fuel, i_waste, i_temperature, i_flame};
	for (int a = 0; a < 4; ++a) {
		HNS_REQUIRE(idx[a] >= 0 && idx[a] < s->n_scalars, "combustion field index out of range");
		for (int b = 0; b < a; ++b) HNS_REQUIRE(idx[a] != idx[b], "combustion field indices must be distinct");
	}
	std::memcpy(s->comb_idx, idx, sizeof(idx));
	s->comb = *params;
	s->comb_enabled = true;
	return HNS_OK;
}

int hns_state_step(hns_state* s, int iterations, float dt, unsigned flags, void* stream) {
	HNS_REQUIRE(s, "null state");
	HNS_REQUIRE(iterations > 0, "Number of pressure iterations must be positive.");
	HNS_REQUIRE(dt >= 0.0f, "dt (time step) cannot be negative.");
	if (!s->n) return HNS_OK;
	return frame(s, iterations, dt, s->grid->voxel_size, flags, static_cast<cudaStream_t>(stream));  // bumps vel_version where it writes the velocity
}
int hns_state_advect_velocity(hns_state* s, float dt, void* stream) {
	HNS_REQUIRE(s, "null state");
	stage_advect_velocity(s, dt, 1.0f / s->grid->voxel_size, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_vorticity_confinement(hns_state* s, float dt, float scale, float factor_scale, void* stream) {
	HNS_REQUIRE(s, "null state");
	return vorticity_pass(s, dt, 1.0f / s->grid->voxel_size, scale, factor_scale, static_cast<cudaStream_t>(stream));
}
int hns_state_vorticity_active(const hns_state* s) {
	return s && s->comb_enabled && vorticity_active(s->comb.vorticityScale, s->comb.factorScale) ? 1 : 0;
}
int hns_state_vorticity_mag(hns_state* s, void* stream) {
	HNS_REQUIRE(s, "null state");
	return vorticity_mag(s, 1.0f / s->grid->voxel_size, static_cast<cudaStream_t>(stream));
}
int hns_state_vorticity_force(hns_state* s, float dt, float scale, float factor_scale, void* stream) {
	HNS_REQUIRE(s, "null state");
	return vorticity_force(s, dt, 1.0f / s->grid->voxel_size, scale, factor_scale, static_cast<cudaStream_t>(stream));
}
int hns_state_divergence(hns_state* s, int of_advected, void* stream) {
	HNS_REQUIRE(s, "null state");
	launch_divergence(s->view(), of_advected ? s->adv : s->vel, s->div, 1.0f / s->grid->voxel_size, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_pressure_solve(hns_state* s, int iterations, float omega, unsigned flags, void* stream) {
	HNS_REQUIRE(s && iterations >= 0, "bad argument");
	if (!s->n) return HNS_OK;
	int rc = pressure_solve(s, iterations, s->grid->voxel_size, omega, flags, static_cast<cudaStream_t>(stream));
	if (rc) return rc;
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_pressure_init(hns_state* s, void* stream) {
	HNS_REQUIRE(s, "null state");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	HNS_CUDA(cudaMemsetAsync(s->p[0], 0, (s->n / 2) * sizeof(float), st));
	HNS_CUDA(cudaMemsetAsync(s->p[1], 0, (s->n / 2) * sizeof(float), st));
	return HNS_OK;
}
int hns_state_pressure_half_sweep(hns_state* s, int color, float omega, int reverse, void* stream) {
	HNS_REQUIRE(s && (color == 0 || color == 1), "bad argument");
	launch_rbgs_color(s->view(), s->div, s->p, s->grid->voxel_size, color, omega, reverse, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_combustion_buoyancy(hns_state* s, float dt, void* stream) {
	HNS_REQUIRE(s, "null state");
	if (!s->comb_enabled) return fail(HNS_ERR_RUNTIME, "combustion stage not configured (hns_state_set_combustion)");
	stage_combustion_buoyancy(s, dt, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
float hns_omega_compute(float voxel_size) { return omega_compute(voxel_size); }
float hns_omega_project(float voxel_size) { return omega_project(voxel_size); }

int hns_state_subtract_gradient(hns_state* s, int from_advected, void* stream) {
	HNS_REQUIRE(s, "null state");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	stage_subtract_gradient(s, from_advected != 0, 1.0f / s->grid->voxel_size, st);  // in place when !from_advected (PressureProjection.cu:64)
	if (const float* sdf = s->collision_sdf())  // the collision tail of the kernel, Kernel.cu:808-826
		launch_collision_boundary(s->view(), s->vel, s->vel, sdf, 1.0f / s->grid->voxel_size, 0.1f, 0, st);
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_set_collision(hns_state* s, int sdf_scalar_index) {
	HNS_REQUIRE(s, "null state");
	HNS_REQUIRE(sdf_scalar_index >= -1 && sdf_scalar_index < s->n_scalars, "sdf scalar index out of range");
	s->skip_scalar = sdf_scalar_index;
	s->collision = sdf_scalar_index >= 0;
	return HNS_OK;
}
int hns_state_collision_active(const hns_state* s) { return s && s->collision_sdf() ? 1 : 0; }
int hns_state_enforce_collision(hns_state* s, void* stream) {
	HNS_REQUIRE(s, "null state");
	const float* sdf = s->collision_sdf();
	if (!sdf) return HNS_OK;
	++s->vel_version;
	launch_collision_boundary(s->view(), s->vel, s->vel, sdf, 1.0f / s->grid->voxel_size, 0.1f, 0, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_advect_scalars(hns_state* s, float dt, int sampler_semantics, void* stream) {
	HNS_REQUIRE(s, "null state");
	if (!s->n_scalars || !s->n) return HNS_OK;
	stage_advect_scalars(s, dt, 1.0f / s->grid->voxel_size, sampler_semantics, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_sync(hns_state* s, void* stream) {
	(void)s;
	HNS_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
	return HNS_OK;
}

int hns_state_time_frames(hns_state* s, int frames, int iterations, float dt, unsigned flags, void* stream, float* ms_total, float* ms_pressure) {
	HNS_REQUIRE(s && frames > 0 && iterations > 0, "bad argument");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	++s->vel_version;
	// Every frame must do identical work on identical data: keep a pristine copy of the inputs and restore it (outside
	// the per-frame events would need a sync per frame; instead the restore copies are timed separately and subtracted).
	const size_t fb = s->n * sizeof(float);
	std::vector<float*> keep;
	auto snap = [&](float* src) {
		float* d = nullptr;
		if (cudaMalloc(&d, std::max<size_t>(fb, 4)) != cudaSuccess) return false;
		cudaMemcpyAsync(d, src, fb, cudaMemcpyDeviceToDevice, st);
		keep.push_back(d);
		return true;
	};
	bool ok = true;
	for (int c = 0; c < 3 && ok; ++c) ok = snap(s->vel[c]);
	for (int i = 0; i < s->n_scalars && ok; ++i) ok = snap(s->sc[i]);
	if (!ok) {
		for (float* d : keep) cudaFree(d);
		return fail(HNS_ERR_CUDA, "cudaMalloc(snapshot)");
	}
	std::vector<cudaEvent_t> ev(4 * size_t(frames));
	for (auto& e : ev) cudaEventCreate(&e);
	int rc = HNS_OK;
	for (int f = 0; f < frames && rc == HNS_OK; ++f) {
		for (int c = 0; c < 3; ++c) cudaMemcpyAsync(s->vel[c], keep[c], fb, cudaMemcpyDeviceToDevice, st);
		for (int i = 0; i < s->n_scalars; ++i) cudaMemcpyAsync(s->sc[i], keep[3 + i], fb, cudaMemcpyDeviceToDevice, st);
		++s->vel_version, ++s->sc_version;
		// A frame of a running simulation finds the velocity the previous frame's gradient pass wrote -- brick planes and packed group 0
		// alike (every timed frame pays for that second copy in its own gradient pass). The restored input stands in for that velocity,
		// so it is packed here, outside the events, like the restore copies themselves.
		if (groups_allowed(s) && ensure_group(s, 0)) {
			const float* const src[4] = {s->vel[0], s->vel[1], s->vel[2], nullptr};
			launch_pack4(src[0], src[1], src[2], src[3], s->grp[0].buf, s->n, st);
			group_written(s, 0, src);
		}
		cudaEventRecord(ev[4 * f + 0], st);
		rc = frame(s, iterations, dt, s->grid->voxel_size, flags, st, ev[4 * f + 1], ev[4 * f + 2]);
		cudaEventRecord(ev[4 * f + 3], st);
	}
	cudaStreamSynchronize(st);
	float tot = 0.f, pr = 0.f;
	if (rc == HNS_OK)
		for (int f = 0; f < frames; ++f) {
			float a = 0.f, b = 0.f;
			cudaEventElapsedTime(&a, ev[4 * f + 0], ev[4 * f + 3]);
			cudaEventElapsedTime(&b, ev[4 * f + 1], ev[4 * f + 2]);
			tot += a, pr += b;
		}
	for (auto& e : ev) cudaEventDestroy(e);
	for (float* d : keep) cudaFree(d);
	if (ms_total) *ms_total = tot;
	if (ms_pressure) *ms_pressure = pr;
	if (rc) return rc;
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

void* hns_state_field_device_ptr(hns_state* s, int field) {
	if (!s) return nullptr;
	field_written(s, field);  // the caller may write through the pointer
	int fpl;
	return field_ptr(s, field, &fpl);
}
int hns_state_field_floats_per_leaf(int field) { return (field >= 6 && field <= 9) ? 256 : 512; }
int hns_state_pack_leaves(hns_state* s, int field, const int32_t* ids, uint64_t n_ids, float* dst, void* stream) {
	HNS_REQUIRE(s, "null state");
	int fpl;
	float* f = field_ptr(s, field, &fpl);
	HNS_REQUIRE(f, "bad field id");
	launch_pack_leaves(f, ids, n_ids, dst, fpl, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
int hns_state_unpack_leaves(hns_state* s, int field, const int32_t* ids, uint64_t n_ids, const float* src, void* stream) {
	HNS_REQUIRE(s, "null state");
	int fpl;
	float* f = field_ptr(s, field, &fpl);
	HNS_REQUIRE(f, "bad field id");
	field_written(s, field);
	launch_unpack_leaves(f, ids, n_ids, src, fpl, static_cast<cudaStream_t>(stream));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

// ---- one-shot launchers on host sidecar arrays --------------------------------------------------------------------
// The reference allocates and frees every device buffer on every call (HNanoSolver.cu:87-106; cudaMalloc/cudaFree of a few GB cost
// milliseconds). The one-shot launchers here keep ONE scratch state per process and reuse it while the voxel count and the
// number of float blocks stay the same (the usual case: a simulation is cooked frame after frame); hns_release_scratch() frees it.
namespace {
std::mutex g_scratch_mu;
hns_state* g_scratch = nullptr;
int g_scratch_device = -1;
struct Streams {
	cudaStream_t copy = nullptr, copy_out = nullptr;  // uploads / downloads on streams of their own: PCIe carries both directions at once
	cudaEvent_t ev[8] = {};
	int device = -1;
} g_streams;

int acquire_scratch(const hns_grid* g, int n_scalars, hns_state** out) {
	int dev = 0;
	HNS_CUDA(cudaGetDevice(&dev));
	if (g_scratch && (g_scratch_device != dev || g_scratch->n != g->num_leaves * 512 || g_scratch->n_scalars != n_scalars)) {
		hns_state_destroy(g_scratch);
		g_scratch = nullptr;
	}
	if (!g_scratch) {
		int rc = hns_state_create(g, n_scalars, &g_scratch);
		if (rc) return rc;
		g_scratch_device = dev;
	}
	g_scratch->grid = g;
	++g_scratch->vel_version, ++g_scratch->sc_version;  // whatever the packed advection groups mirror belongs to an earlier call
	g_scratch->mg = nullptr;
	g_scratch->comb_enabled = false, g_scratch->skip_scalar = -1, g_scratch->collision = false, g_scratch->active = nullptr, g_scratch->n_active = 0;
	*out = g_scratch;
	return HNS_OK;
}
int acquire_streams(Streams** out) {
	int dev = 0;
	HNS_CUDA(cudaGetDevice(&dev));
	if (g_streams.device != dev) {
		if (g_streams.copy) {
			cudaStreamDestroy(g_streams.copy);
			cudaStreamDestroy(g_streams.copy_out);
			for (auto& e : g_streams.ev) cudaEventDestroy(e);
		}
		HNS_CUDA(cudaStreamCreateWithFlags(&g_streams.copy, cudaStreamNonBlocking));
		HNS_CUDA(cudaStreamCreateWithFlags(&g_streams.copy_out, cudaStreamNonBlocking));
		for (auto& e : g_streams.ev) HNS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		g_streams.device = dev;
	}
	*out = &g_streams;
	return HNS_OK;
}
}  // namespace

void hns_release_scratch(void) {
	std::lock_guard<std::mutex> lk(g_scratch_mu);
	hns_state_destroy(g_scratch);
	g_scratch = nullptr;
	release_grid_pool();
}

// Shared helper: a temporary grid for the stand-alone launchers + the process-wide scratch state.
struct Scoped {
	hns_grid* grid = nullptr;
	hns_state* state = nullptr;  // borrowed from the scratch cache
	bool own_grid = false;
	std::unique_lock<std::mutex> lock{g_scratch_mu};
	~Scoped() {
		if (state) state->grid = nullptr;
		if (own_grid) hns_grid_destroy(grid);
	}
};

int hns_compute_sim(const hns_grid* g, float* velocity, int n_float, const char* const* names, float* const* fields, int iterations, float dt,
                    float voxel_size, const hns_combustion_params* params, int has_collision, void* stream) {
	// validation in the reference's order (HNanoSolver.cu:12-35)
	if (!(voxel_size > 0.0f)) return fail(HNS_ERR_INVALID_ARGUMENT, "voxelSize must be positive.");
	if (dt < 0.0f) return fail(HNS_ERR_INVALID_ARGUMENT, "dt (time step) cannot be negative.");
	if (iterations <= 0) return fail(HNS_ERR_INVALID_ARGUMENT, "Number of pressure iterations must be positive.");
	if (!g) return fail(HNS_ERR_INVALID_ARGUMENT, "Invalid nanovdb::GridHandle provided (null grid).");
	const uint64_t n = g->num_leaves * 512;
	if (n == 0) return HNS_OK;  // :26-28
	if (!velocity) return fail(HNS_ERR_RUNTIME, "Host velocity data pointer is null");
	if (n_float <= 0) return fail(HNS_ERR_RUNTIME, "No float blocks found in input data.");
	if (n_float > 16) return fail(HNS_ERR_UNSUPPORTED, "more than 16 float blocks");
	if (!names || !fields || !params) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	int iF = -1, iW = -1, iT = -1, iL = -1, iSdf = -1;
	for (int i = 0; i < n_float; ++i) {
		if (!fields[i]) return fail(HNS_ERR_RUNTIME, std::string("Host float data pointer is null for block: ") + names[i]);
		if (!std::strcmp(names[i], "fuel")) iF = i;
		if (!std::strcmp(names[i], "waste")) iW = i;
		if (!std::strcmp(names[i], "temperature")) iT = i;
		if (!std::strcmp(names[i], "flame")) iL = i;
		if (!std::strcmp(names[i], "collision_sdf")) iSdf = i;
	}
	for (const char* req : {"fuel", "waste", "temperature", "flame"}) {  // :193-201
		bool found = false;
		for (int i = 0; i < n_float; ++i) found |= !std::strcmp(names[i], req);
		if (!found) return fail(HNS_ERR_RUNTIME, std::string("Missing required input field for combustion: ") + req);
	}
	Scoped sc;
	int rc = acquire_scratch(g, n_float, &sc.state);
	if (rc) return rc;
	hns_state* s = sc.state;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	if ((rc = hns_state_set_combustion(s, 1, iF, iW, iT, iL, params))) return rc;
	++s->vel_version, ++s->sc_version;  // every field is about to be overwritten from the host
	s->skip_scalar = iSdf;
	s->collision = has_collision && iSdf >= 0;  // hasCollisionData, HNanoSolver.cu:65-76
	if ((rc = ensure_aos(s))) return rc;
	Streams* ss = nullptr;
	if ((rc = acquire_streams(&ss))) return rc;
	cudaStream_t cs = ss->copy;
	cudaEvent_t e_start = ss->ev[0], e_vel_in = ss->ev[1], e_comb_in = ss->ev[2], e_all_in = ss->ev[3], e_vel_out = ss->ev[4], e_done = ss->ev[5];
	cudaEvent_t e_fw_in = ss->ev[6], e_t_in = ss->ev[7];
	// The whole state crosses PCIe in both directions (HNanoSolver.cu:120-133, 361-369; the coords are not needed on the device
	// here). Transfers run on a copy stream and overlap the kernels: velocity first (advect_vector + divergence start as soon as
	// it has landed), then fuel and waste -- all the pressure solve needs of the combustion stage --, then the temperature (the
	// buoyancy force the gradient pass needs), then flame and the remaining scalars; the projected velocity goes back on a second copy
	// stream while those are still arriving and advect_scalars runs (PCIe is full duplex). See frame(). Critical path on the 512^3
	// workload: 14.6 of the 23.5 ms of uploads, the solve, the 24 ms of downloads.
	HNS_CUDA(cudaEventRecord(e_start, st));
	HNS_CUDA(cudaStreamWaitEvent(cs, e_start, 0));  // everything the caller queued on `stream` before this call stays ordered
	HNS_CUDA(cudaMemcpyAsync(s->aos, velocity, n * 12, cudaMemcpyHostToDevice, cs));
	if (s->collision) HNS_CUDA(cudaMemcpyAsync(s->sc[iSdf], fields[iSdf], n * 4, cudaMemcpyHostToDevice, cs));  // the first kernel reads it
	HNS_CUDA(cudaEventRecord(e_vel_in, cs));
	for (int i : {iF, iW}) HNS_CUDA(cudaMemcpyAsync(s->sc[i], fields[i], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_fw_in, cs));
	HNS_CUDA(cudaMemcpyAsync(s->sc[iT], fields[iT], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_t_in, cs));
	HNS_CUDA(cudaMemcpyAsync(s->sc[iL], fields[iL], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_comb_in, cs));
	for (int i = 0; i < n_float; ++i)
		if (i != iF && i != iW && i != iT && i != iL && !(s->collision && i == iSdf))
			HNS_CUDA(cudaMemcpyAsync(s->sc[i], fields[i], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_all_in, cs));
	HNS_CUDA(cudaStreamWaitEvent(st, e_vel_in, 0));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], n, st);
	FrameDeps deps;
	deps.fuel_waste_inputs = e_fw_in, deps.temperature_input = e_t_in, deps.combustion_inputs = e_comb_in, deps.scalar_inputs = e_all_in, deps.velocity_done = e_vel_out;
	if ((rc = frame(s, iterations, dt, voxel_size, 0u, st, nullptr, nullptr, &deps))) return rc;
	// results back into the same host arrays (HNanoSolver.cu:361-369); a collision_sdf block comes back zeroed like the
	// reference's never-written output buffer
	cudaStream_t co = ss->copy_out;  // the projected velocity leaves while the last inputs are still arriving on `cs`
	HNS_CUDA(cudaStreamWaitEvent(co, e_vel_out, 0));
	HNS_CUDA(cudaMemcpyAsync(velocity, s->aos, n * 12, cudaMemcpyDeviceToHost, co));
	if (iSdf >= 0) HNS_CUDA(cudaMemsetAsync(s->sc[iSdf], 0, n * 4, st));
	HNS_CUDA(cudaEventRecord(e_done, st));
	HNS_CUDA(cudaStreamWaitEvent(co, e_done, 0));
	for (int i = 0; i < n_float; ++i) HNS_CUDA(cudaMemcpyAsync(fields[i], s->sc[i], n * 4, cudaMemcpyDeviceToHost, co));
	HNS_CUDA(cudaStreamSynchronize(co));
	HNS_CUDA(cudaStreamSynchronize(cs));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

static int temp_grid(const int32_t* coords, uint64_t n, float voxel_size, Scoped& sc, int n_scalars) {
	int rc = hns_grid_create_from_coords(coords, n, voxel_size, 0, &sc.grid);
	if (rc) return rc;
	sc.own_grid = true;
	return acquire_scratch(sc.grid, n_scalars, &sc.state);
}

int hns_advect_index_grid(const int32_t* coords, uint64_t n, const float* velocity, int n_float, float* const* fields, float dt, float voxel_size,
                          void* stream) {
	if (!velocity) return fail(HNS_ERR_RUNTIME, "Velocity data not found");
	if (n_float <= 0 || !fields) return fail(HNS_ERR_RUNTIME, "No float blocks found");
	if (n_float > 16) return fail(HNS_ERR_UNSUPPORTED, "more than 16 float blocks");
	if (n == 0) return HNS_OK;
	Scoped sc;
	int rc = temp_grid(coords, n, voxel_size, sc, n_float);
	if (rc) return rc;
	hns_state* s = sc.state;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	if ((rc = ensure_aos(s))) return rc;
	HNS_CUDA(cudaMemcpyAsync(s->aos, velocity, n * 12, cudaMemcpyHostToDevice, st));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], n, st);
	for (int i = 0; i < n_float; ++i) {
		if (!fields[i]) return fail(HNS_ERR_RUNTIME, "Block not found or type mismatch");
		HNS_CUDA(cudaMemcpyAsync(s->sc[i], fields[i], n * 4, cudaMemcpyHostToDevice, st));
	}
	launch_advect_scalars(sc.grid->view, s->vel, scalar_ptrs(s), n_float, dt, 1.0f / voxel_size, 1, st, nullptr, s->cold);  // advect_scalar semantics (Advection.cu:89)
	for (int i = 0; i < n_float; ++i) HNS_CUDA(cudaMemcpyAsync(fields[i], s->sc_out[i], n * 4, cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

int hns_advect_index_grid_velocity(const int32_t* coords, uint64_t n, float* velocity, float dt, float voxel_size, void* stream) {
	if (!velocity) return fail(HNS_ERR_RUNTIME, "Velocity data not found");
	if (n == 0) return HNS_OK;
	Scoped sc;
	int rc = temp_grid(coords, n, voxel_size, sc, 0);
	if (rc) return rc;
	hns_state* s = sc.state;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	if ((rc = ensure_aos(s))) return rc;
	HNS_CUDA(cudaMemcpyAsync(s->aos, velocity, n * 12, cudaMemcpyHostToDevice, st));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], n, st);
	launch_advect_vector(sc.grid->view, s->vel, s->adv, dt, 1.0f / voxel_size, st, nullptr, s->cold);
	launch_soa_to_aos(s->adv[0], s->adv[1], s->adv[2], s->aos, n, st);
	HNS_CUDA(cudaMemcpyAsync(velocity, s->aos, n * 12, cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

int hns_project_non_divergent(const int32_t* coords, uint64_t n, float* velocity, uint64_t iterations, float voxel_size, void* stream) {
	if (!velocity) return fail(HNS_ERR_RUNTIME, "Velocity data not found");
	if (n == 0) return HNS_OK;
	Scoped sc;
	int rc = temp_grid(coords, n, voxel_size, sc, 0);
	if (rc) return rc;
	hns_state* s = sc.state;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	const float inv = 1.0f / voxel_size;
	if ((rc = ensure_aos(s))) return rc;
	HNS_CUDA(cudaMemcpyAsync(s->aos, velocity, n * 12, cudaMemcpyHostToDevice, st));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], n, st);
	launch_divergence(sc.grid->view, s->vel, s->div, inv, st);
	if ((rc = pressure_solve(s, int(iterations), voxel_size, omega_project(voxel_size), 0u, st))) return rc;
	launch_subtract_gradient(sc.grid->view, s->vel, s->p, s->vel, inv, st);
	launch_soa_to_aos(s->vel[0], s->vel[1], s->vel[2], s->aos, n, st);
	HNS_CUDA(cudaMemcpyAsync(velocity, s->aos, n * 12, cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

int hns_divergence(const int32_t* coords, uint64_t n, const float* velocity, float* divergence_out, float voxel_size, void* stream) {
	if (!velocity) return fail(HNS_ERR_RUNTIME, "Velocity data not found");
	if (!divergence_out) return fail(HNS_ERR_RUNTIME, "float block 'divergence' not found");
	if (n == 0) return HNS_OK;
	Scoped sc;
	int rc = temp_grid(coords, n, voxel_size, sc, 0);
	if (rc) return rc;
	hns_state* s = sc.state;
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	if ((rc = ensure_aos(s))) return rc;
	HNS_CUDA(cudaMemcpyAsync(s->aos, velocity, n * 12, cudaMemcpyHostToDevice, st));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], n, st);
	launch_divergence(sc.grid->view, s->vel, s->div, 1.0f / voxel_size, st);
	launch_split_to_brick(s->div, s->adv[0], n, st);  // adv[0] is free scratch here
	HNS_CUDA(cudaMemcpyAsync(divergence_out, s->adv[0], n * 4, cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

int hns_combustion_kernel(const hns_grid* g, float* velocity, uint64_t n_voxels, float dt, float voxel_size, void* stream) {
	(void)dt, (void)voxel_size, (void)stream;
	if (!g) return fail(HNS_ERR_INVALID_ARGUMENT, "null grid");
	if (!velocity && n_voxels) return fail(HNS_ERR_RUNTIME, "Velocity data not found");
	return HNS_OK;  // validated no-op: see header
}

}  // extern "C"
