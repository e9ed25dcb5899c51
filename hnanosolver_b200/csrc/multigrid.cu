// Geometric multigrid for the pressure Poisson equation on the sparse brick grid, and the device-side residual / divergence norms.
//
// Reference: the all-in-one node only ever runs `iteration` red-black SOR sweeps (src/Cuda/HNanoSolver.cu:252-285). A V-cycle is
// sketched but dead: v_cycle is commented out (src/Cuda/HNanoSolver.cu:399-507) and its kernels restrict_to_4x4x4, restrict_to_2x2x2,
// prolongate, update_pressure, compute_residual are declared without a definition (src/Cuda/Kernels.cuh:38-49). There is therefore no
// reference output to be bit-exact with; what is kept is the equation (7-point operator, p = 0 outside the domain, Kernel.cu:591-623),
// the smoother (the same red-black update) and the acceptance gates of SURVEY.md Appendix A-9: relative Poisson residual and the
// divergence of the projected velocity against what the reference's fixed-count solve reaches.
//
// Hierarchy: level k + 1 has cells of twice the size; a cell is inside the domain iff all 8 of its children are. Leaves of level k + 1
// are 2x2x2 leaves of level k, so every level is again a set of dense 8^3 bricks with a NanoVDB-ordered leaf list, a neighbour table
// (topology.cu builds both) and colour-split p / rhs arrays -- the fine-level sweep kernel runs unchanged on every level, plus a
// per-row byte mask for the cells of a coarse brick that lie outside the domain. The last level is a single leaf (or `max_levels`).
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "kernels.cuh"

using namespace hns;

namespace {

struct KeyLess {
	bool operator()(const std::array<int32_t, 3>& a, const std::array<int32_t, 3>& b) const {
		// NanoVDB leaf order: root tile (signed, lexicographic x, y, z), then upper offset, then lower offset (topology.cu leaf_key)
		auto tile = [](const std::array<int32_t, 3>& o) {
			const int64_t bias = int64_t(1) << 31;
			return (uint64_t(uint32_t(int64_t(o[2]) + bias) >> 12)) | (uint64_t(uint32_t(int64_t(o[1]) + bias) >> 12) << 21) |
			       (uint64_t(uint32_t(int64_t(o[0]) + bias) >> 12) << 42);
		};
		auto node = [](const std::array<int32_t, 3>& o) {
			const uint32_t up = uint32_t(((o[0] & 4095) >> 7) << 10 | ((o[1] & 4095) >> 7) << 5 | ((o[2] & 4095) >> 7));
			const uint32_t lo = uint32_t(((o[0] & 127) >> 3) << 8 | ((o[1] & 127) >> 3) << 4 | ((o[2] & 127) >> 3));
			return up << 12 | lo;
		};
		const uint64_t ta = tile(a), tb = tile(b);
		return ta != tb ? ta < tb : node(a) < node(b);
	}
};

int alloc_level_fields(hns_mg::Level& L) {
	const size_t half = std::max<size_t>(L.grid->num_leaves * 256, 4) * sizeof(float);
	HNS_CUDA(cudaMalloc(&L.p[0], 2 * half));
	L.p[1] = L.p[0] + L.grid->num_leaves * 256;
	HNS_CUDA(cudaMalloc(&L.rhs[0], 2 * half));
	L.rhs[1] = L.rhs[0] + L.grid->num_leaves * 256;
	HNS_CUDA(cudaMemset(L.p[0], 0, 2 * half));
	HNS_CUDA(cudaMemset(L.rhs[0], 0, 2 * half));
	return HNS_OK;
}

}  // namespace

extern "C" {

void hns_mg_destroy(hns_mg* mg) {
	if (!mg) return;
	for (auto& L : mg->lv) {
		cudaFree(L.p[0]), cudaFree(L.rhs[0]), cudaFree(L.diag[0]), cudaFree(L.parent);
		if (L.own_grid) hns_grid_destroy(L.grid);
	}
	cudaFree(mg->d_sums);
	if (mg->h_sums) cudaFreeHost(mg->h_sums);
	if (mg->graph.exec) cudaGraphExecDestroy(mg->graph.exec);
	if (mg->capture_stream) cudaStreamDestroy(mg->capture_stream);
	delete mg;
}

int hns_mg_create(const hns_grid* fine, int max_levels, hns_mg** out) {
	if (!fine || !out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	*out = nullptr;
	if (max_levels <= 0) max_levels = 16;
	auto* mg = new hns_mg();
	auto bail = [&](int rc) {
		const std::string keep = hns_last_error();
		hns_mg_destroy(mg);
		set_error(keep);
		return rc;
	};
	hns_mg::Level l0;
	l0.grid = const_cast<hns_grid*>(fine), l0.dx = fine->voxel_size, l0.cells = fine->num_leaves * 512;
	mg->lv.push_back(l0);
	// host copies of the current level: leaf origins (in cells of that level) and row masks
	uint64_t L = fine->num_leaves;
	std::vector<int4> org4(L);
	if (L && cudaMemcpy(org4.data(), fine->d_origin, L * sizeof(int4), cudaMemcpyDeviceToHost) != cudaSuccess) return bail(fail(HNS_ERR_CUDA, "cudaMemcpy(origins)"));
	std::vector<std::array<int32_t, 3>> org(L);
	for (uint64_t l = 0; l < L; ++l) org[l] = {org4[l].x, org4[l].y, org4[l].z};
	std::vector<uint8_t> mask(L * 64, 0xff);
	uint64_t non_empty = L;  // leaves of the current level that hold at least one cell of the domain
	while (non_empty > 1 && int(mg->lv.size()) < max_levels) {
		// parents of this level's leaves, in NanoVDB order
		std::map<std::array<int32_t, 3>, int32_t, KeyLess> ids;
		auto parent_origin = [](const std::array<int32_t, 3>& o) { return std::array<int32_t, 3>{(o[0] >> 4) * 8, (o[1] >> 4) * 8, (o[2] >> 4) * 8}; };
		for (uint64_t l = 0; l < L; ++l) ids.emplace(parent_origin(org[l]), 0);
		std::vector<std::array<int32_t, 3>> corg;
		corg.reserve(ids.size());
		for (auto& kv : ids) kv.second = int32_t(corg.size()), corg.push_back(kv.first);
		const uint64_t Lc = corg.size();
		std::vector<int32_t> parent(L);
		std::vector<uint8_t> cmask(Lc * 64, 0);
		uint64_t cells = 0;
		for (uint64_t l = 0; l < L; ++l) {
			const int32_t pl = ids[parent_origin(org[l])];
			parent[l] = pl;
			const int bx = ((org[l][0] >> 3) & 1) * 4, by = ((org[l][1] >> 3) & 1) * 4, bz = ((org[l][2] >> 3) & 1) * 4;
			// A cell belongs to the next level iff ALL 8 of its children belong to this one (they lie in this one leaf). Levels 1-3
			// then cover the domain exactly (a leaf is 8^3 voxels); deeper levels keep only what is fully covered. The opposite rule
			// ("any child") makes the coarse domains too large around thin features: the coarse correction overshoots there and
			// V(1,1) cycles diverge on the 512^3 sparse smoke (measured; the "all" rule converges at ~0.1 per V(2,2) cycle).
			for (int X = 0; X < 4; ++X)
				for (int Y = 0; Y < 4; ++Y) {
					const uint8_t m = mask[l * 64 + (2 * X) * 8 + 2 * Y] & mask[l * 64 + (2 * X) * 8 + 2 * Y + 1] & mask[l * 64 + (2 * X + 1) * 8 + 2 * Y] &
					                  mask[l * 64 + (2 * X + 1) * 8 + 2 * Y + 1];
					uint8_t pm = 0;  // children z = 2k, 2k + 1 -> parent cell bz + k
					for (int k = 0; k < 4; ++k)
						if (((m >> (2 * k)) & 3u) == 3u) pm |= uint8_t(1u << (bz + k));
					cmask[uint64_t(pl) * 64 + (bx + X) * 8 + (by + Y)] |= pm;
				}
		}
		for (uint8_t b : cmask) cells += uint64_t(__builtin_popcount(b));
		if (!cells) break;  // nothing is fully covered any more: the current level is the last
		// upload: parent table of the current level, then the new level
		hns_mg::Level& cur = mg->lv.back();
		if (cudaMalloc(&cur.parent, L * sizeof(int32_t)) != cudaSuccess || cudaMemcpy(cur.parent, parent.data(), L * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess)
			return bail(fail(HNS_ERR_CUDA, "cudaMalloc/cudaMemcpy(parent table)"));
		hns_mg::Level nl;
		std::vector<int32_t> flat(3 * Lc);
		for (uint64_t l = 0; l < Lc; ++l) flat[3 * l] = corg[l][0], flat[3 * l + 1] = corg[l][1], flat[3 * l + 2] = corg[l][2];
		int rc = hns_grid_create_from_origins(flat.data(), Lc, cur.dx * 2.0f, &nl.grid);
		if (rc) return bail(rc);
		nl.own_grid = true, nl.dx = cur.dx * 2.0f, nl.cells = cells;
		mg->lv.push_back(nl);
		hns_mg::Level& added = mg->lv.back();
		if ((rc = alloc_level_fields(added))) return bail(rc);
		{
			// the level's diagonal from its row masks, on the device (kernels.cu k_mg_diag explains the boundary term)
			uint8_t* d_mask = nullptr;
			if (cudaMalloc(&d_mask, Lc * 64) != cudaSuccess || cudaMemcpy(d_mask, cmask.data(), Lc * 64, cudaMemcpyHostToDevice) != cudaSuccess ||
			    cudaMalloc(&added.diag[0], Lc * 512 * sizeof(float)) != cudaSuccess) {
				cudaFree(d_mask);
				return bail(fail(HNS_ERR_CUDA, "cudaMalloc/cudaMemcpy(level mask)"));
			}
			added.diag[1] = added.diag[0] + Lc * 256;
			const int k = int(mg->lv.size()) - 1;
			const double theta = 0.5 + std::ldexp(1.0, -(k + 1));
			launch_mg_diag(added.grid->view, d_mask, float(1.0 / theta - 1.0), added.diag, nullptr);
			const cudaError_t e = cudaDeviceSynchronize();
			cudaFree(d_mask);
			if (e != cudaSuccess) return bail(fail(HNS_ERR_CUDA, std::string("k_mg_diag: ") + cudaGetErrorString(e)));
		}
		L = Lc, org.swap(corg), mask.swap(cmask);
		non_empty = 0;
		for (uint64_t l = 0; l < L; ++l) {
			bool any = false;
			for (int r = 0; r < 64 && !any; ++r) any = mask[l * 64 + r] != 0;
			if (any) ++non_empty, mg->last_nonempty_leaf = int64_t(l);
		}
		mg->last_nonempty_count = non_empty;
	}
	if (cudaMalloc(&mg->d_sums, 2 * sizeof(double)) != cudaSuccess || cudaMallocHost(&mg->h_sums, 2 * sizeof(double)) != cudaSuccess)
		return bail(fail(HNS_ERR_CUDA, "cudaMalloc(norm sums)"));
	if (const char* e = std::getenv("HNS_MG_GRAPH")) mg->use_graph = std::atoi(e) != 0;
	*out = mg;
	return HNS_OK;
}

int hns_mg_num_levels(const hns_mg* mg) { return mg ? int(mg->lv.size()) : 0; }
uint64_t hns_mg_level_leaves(const hns_mg* mg, int level) { return mg && level >= 0 && level < int(mg->lv.size()) ? mg->lv[level].grid->num_leaves : 0; }
uint64_t hns_mg_level_cells(const hns_mg* mg, int level) { return mg && level >= 0 && level < int(mg->lv.size()) ? mg->lv[level].cells : 0; }
int hns_mg_set_coarsest_iterations(hns_mg* mg, int iterations) {
	if (!mg || iterations <= 0) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	mg->coarsest_iterations = iterations;
	return HNS_OK;
}
int hns_mg_last_cycles(const hns_mg* mg) { return mg ? mg->last_cycles : 0; }
double hns_mg_last_relative_residual(const hns_mg* mg) { return mg ? mg->last_rel_residual : -1.0; }

}  // extern "C"

namespace hns {

// {sum (rhs - L p)^2, sum rhs^2} of the fine level into mg-independent device sums; asynchronous
static void residual_sums_async(const GridView& g, const float* const p[2], const float* const rhs[2], float dx, double* d_sums, cudaStream_t st) {
	cudaMemsetAsync(d_sums, 0, 2 * sizeof(double), st);
	launch_mg_residual(g, p, rhs, dx, nullptr, nullptr, nullptr, d_sums, st);
}

// Levels 1 .. n-1 of one V(nu_pre, nu_post) cycle (n > 1): the right-hand side of level 1 is `rhs1` (the hierarchy's own array, or a sharded
// run's gathered copy, dist.cu); the correction starts from 0 on every level and ends up in lv[1].p, ready for the prolongation to level 0.
void mg_coarse_cycle(hns_mg* mg, float* const rhs1[2], int nu_pre, int nu_post, float omega, cudaStream_t st) {
	const int n = int(mg->lv.size());
	auto P = [&](int k) -> float* const* { return mg->lv[k].p; };
	auto F = [&](int k) -> float* const* { return k == 1 ? rhs1 : mg->lv[k].rhs; };
	auto smooth = [&](int k, int iters) {
		const GridView g = mg->lv[k].grid->view;
		for (int it = 0; it < iters; ++it)
			for (int color = 0; color < 2; ++color) launch_rbgs_color_masked(g, F(k), P(k), mg->lv[k].dx, color, omega, mg->lv[k].diag, st);
	};
	cudaMemsetAsync(mg->lv[1].p[0], 0, mg->lv[1].grid->num_leaves * 512 * sizeof(float), st);
	for (int k = 1; k + 1 < n; ++k) {  // down
		smooth(k, nu_pre);
		hns_mg::Level& c = mg->lv[k + 1];
		const size_t bytes = c.grid->num_leaves * 512 * sizeof(float);
		cudaMemsetAsync(c.p[0], 0, bytes, st);
		cudaMemsetAsync(c.rhs[0], 0, bytes, st);
		launch_mg_residual(mg->lv[k].grid->view, P(k), F(k), mg->lv[k].dx, mg->lv[k].diag_or_null(), mg->lv[k].parent, c.rhs, nullptr, st);
	}
	{  // coarsest
		hns_mg::Level& c = mg->lv[n - 1];
		if (mg->last_nonempty_count == 1) {
			// the whole level is one brick (its other leaves, if any, hold no cell of the domain and stay 0): solved inside one CTA
			const uint64_t off = uint64_t(mg->last_nonempty_leaf) * 256u;
			float* const p1[2] = {c.p[0] + off, c.p[1] + off};
			const float* const f1[2] = {F(n - 1)[0] + off, F(n - 1)[1] + off};
			const float* const d1[2] = {c.diag[0] + off, c.diag[1] + off};
			launch_mg_coarsest(p1, f1, d1, c.dx, mg->coarsest_omega, mg->coarsest_iterations, st);
		}
		else smooth(n - 1, mg->coarsest_iterations);
	}
	for (int k = n - 2; k >= 1; --k) {  // up
		launch_mg_prolong(mg->lv[k].grid->view, P(k), mg->lv[k].diag_or_null(), mg->lv[k].parent, mg->lv[k + 1].grid->view, mg->lv[k + 1].p, st);
		smooth(k, nu_post);
	}
}

// One V(nu_pre, nu_post) cycle on the state's divergence / pressure. Level 0 relaxes the caller's p in place; the coarser levels are
// mg_coarse_cycle.
static void v_cycle(hns_mg* mg, hns_state* s, int nu_pre, int nu_post, float omega, cudaStream_t st) {
	const int n = int(mg->lv.size());
	const GridView g = s->view();
	const float dx = mg->lv[0].dx;
	auto smooth = [&](int iters) {
		for (int it = 0; it < iters; ++it)
			for (int color = 0; color < 2; ++color) launch_rbgs_color(g, s->div, s->p, dx, color, omega, color, st);
	};
	if (n == 1) {  // a one-level hierarchy: plain red-black sweeps
		smooth(nu_pre + nu_post);
		return;
	}
	smooth(nu_pre);
	hns_mg::Level& c = mg->lv[1];
	cudaMemsetAsync(c.rhs[0], 0, c.grid->num_leaves * 512 * sizeof(float), st);
	launch_mg_residual(g, s->p, s->div, dx, nullptr, mg->lv[0].parent, c.rhs, nullptr, st);
	mg_coarse_cycle(mg, c.rhs, nu_pre, nu_post, omega, st);
	launch_mg_prolong(g, s->p, nullptr, mg->lv[0].parent, c.grid->view, c.p, st);
	smooth(nu_post);
}

// mg_coarse_cycle captured into a CUDA graph on the hierarchy's private stream (the caller owns the result; null when capture is not
// possible); *launches = the kernels one replay runs
cudaGraphExec_t mg_capture_coarse(hns_mg* mg, float* const rhs1[2], int nu_pre, int nu_post, float omega, uint64_t* launches) {
	*launches = 0;
	if (!mg->capture_stream && cudaStreamCreateWithFlags(&mg->capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
		cudaGetLastError();
		return nullptr;
	}
	cudaGraph_t graph = nullptr;
	const uint64_t before = g_launches.load();
	if (cudaStreamBeginCapture(mg->capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
		cudaGetLastError();
		return nullptr;
	}
	mg_coarse_cycle(mg, rhs1, nu_pre, nu_post, omega, mg->capture_stream);
	const cudaError_t e = cudaStreamEndCapture(mg->capture_stream, &graph);
	*launches = g_launches.load() - before;
	g_launches.fetch_sub(*launches);  // nothing ran yet: every replay counts them
	if (e != cudaSuccess || !graph) {
		cudaGetLastError();
		return nullptr;
	}
	cudaGraphExec_t exec = nullptr;
	if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) exec = nullptr, cudaGetLastError();
	cudaGraphDestroy(graph);
	return exec;
}

// the captured cycle for this (state, parameters), or null when graphs are off / capture is not possible
static cudaGraphExec_t cycle_graph(hns_mg* mg, hns_state* s, int nu_pre, int nu_post, float omega) {
	if (!mg->use_graph) return nullptr;
	auto& g = mg->graph;
	const GridView view = s->view();
	if (g.exec && g.state == s && std::memcmp(&g.view, &view, sizeof(view)) == 0 && g.p == s->p[0] && g.rhs == s->div[0] && g.nu_pre == nu_pre &&
	    g.nu_post == nu_post && g.omega == omega && g.coarsest_iterations == mg->coarsest_iterations)
		return g.exec;
	if (g.exec) cudaGraphExecDestroy(g.exec), g.exec = nullptr;
	if (!mg->capture_stream && cudaStreamCreateWithFlags(&mg->capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
		cudaGetLastError();
		return nullptr;
	}
	cudaGraph_t graph = nullptr;
	const uint64_t before = g_launches.load();
	if (cudaStreamBeginCapture(mg->capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
		cudaGetLastError();
		return nullptr;
	}
	v_cycle(mg, s, nu_pre, nu_post, omega, mg->capture_stream);
	const cudaError_t e = cudaStreamEndCapture(mg->capture_stream, &graph);
	const uint64_t launches = g_launches.load() - before;
	g_launches.fetch_sub(launches);  // nothing ran yet: every replay counts them
	if (e != cudaSuccess || !graph) {
		cudaGetLastError();
		return nullptr;
	}
	if (cudaGraphInstantiate(&g.exec, graph, 0) != cudaSuccess) g.exec = nullptr, cudaGetLastError();
	cudaGraphDestroy(graph);
	std::memcpy(&g.view, &view, sizeof(view));
	g.state = s, g.p = s->p[0], g.rhs = s->div[0], g.nu_pre = nu_pre, g.nu_post = nu_post, g.omega = omega;
	g.coarsest_iterations = mg->coarsest_iterations, g.launches = launches;
	return g.exec;
}

int mg_pressure_solve(hns_state* s, hns_mg* mg, int max_cycles, double rel_tol, int nu_pre, int nu_post, float omega, cudaStream_t st) {
	if (mg->lv.empty() || mg->lv[0].grid != s->grid) return fail(HNS_ERR_INVALID_ARGUMENT, "the multigrid hierarchy was built for another grid");
	HNS_CUDA(cudaMemsetAsync(s->p[0], 0, s->n * sizeof(float), st));  // initial guess 0, like the reference's solve (HNanoSolver.cu:113)
	mg->last_cycles = 0, mg->last_rel_residual = -1.0;
	const cudaGraphExec_t exec = cycle_graph(mg, s, nu_pre, nu_post, omega);
	for (int c = 0; c < max_cycles; ++c) {
		if (exec) {
			HNS_CUDA(cudaGraphLaunch(exec, st));
			g_launches.fetch_add(mg->graph.launches, std::memory_order_relaxed);
		} else {
			v_cycle(mg, s, nu_pre, nu_post, omega, st);
		}
		mg->last_cycles = c + 1;
		if (rel_tol > 0.0) {
			residual_sums_async(s->view(), s->p, s->div, s->grid->voxel_size, mg->d_sums, st);
			HNS_CUDA(cudaMemcpyAsync(mg->h_sums, mg->d_sums, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
			HNS_CUDA(cudaStreamSynchronize(st));
			mg->last_rel_residual = mg->h_sums[1] > 0.0 ? std::sqrt(mg->h_sums[0] / mg->h_sums[1]) : 0.0;
			if (mg->last_rel_residual <= rel_tol) break;
		}
	}
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

}  // namespace hns

extern "C" {

int hns_state_pressure_solve_mg(hns_state* s, hns_mg* mg, int max_cycles, double rel_tol, int nu_pre, int nu_post, float omega_smooth, void* stream) {
	if (!s || !mg || max_cycles <= 0 || nu_pre < 0 || nu_post < 0 || nu_pre + nu_post == 0) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	if (s->active) return fail(HNS_ERR_UNSUPPORTED, "this entry point solves single-GPU states (a sharded state has ghost leaves): sharded frames take a multigrid solver through hns_dist_set_pressure_solver");
	if (!s->n) return HNS_OK;
	return mg_pressure_solve(s, mg, max_cycles, rel_tol, nu_pre, nu_post, omega_smooth, static_cast<cudaStream_t>(stream));
}

int hns_state_set_pressure_solver(hns_state* s, hns_mg* mg, int cycles, int nu_pre, int nu_post, float omega_smooth) {
	if (!s) return fail(HNS_ERR_INVALID_ARGUMENT, "null state");
	if (mg && (cycles <= 0 || nu_pre < 0 || nu_post < 0 || nu_pre + nu_post == 0)) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	if (mg && (mg->lv.empty() || mg->lv[0].grid != s->grid)) return fail(HNS_ERR_INVALID_ARGUMENT, "the multigrid hierarchy was built for another grid");
	s->mg = mg, s->mg_cycles = cycles, s->mg_nu[0] = nu_pre, s->mg_nu[1] = nu_post, s->mg_omega = omega_smooth;
	return HNS_OK;
}

// {sum over voxels of (div - L p)^2, sum of div^2} with L p = (sum of the 6 neighbours - 6 p) / dx^2, accumulated in fp64 on the device over the
// leaves the state's kernels process (all, or the owned leaves of a shard). Synchronises `stream`.
int hns_state_residual_sums(hns_state* s, double* out2, void* stream) {
	if (!s || !out2) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	out2[0] = out2[1] = 0.0;
	if (!s->n) return HNS_OK;
	if (!s->d_sums) HNS_CUDA(cudaMalloc(&s->d_sums, 2 * sizeof(double)));
	residual_sums_async(s->view(), s->p, s->div, s->grid->voxel_size, s->d_sums, st);
	HNS_CUDA(cudaMemcpyAsync(out2, s->d_sums, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

// sum of squares of the divergence (reference kernel `divergence`, Kernel.cu:499-519) of the current (which = 0) or advected (1) velocity,
// fp64, over the leaves the state's kernels process. OVERWRITES the state's divergence field. Synchronises `stream`.
int hns_state_divergence_sum_squares(hns_state* s, int of_advected, double* out, void* stream) {
	if (!s || !out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	*out = 0.0;
	if (!s->n) return HNS_OK;
	if (!s->d_sums) HNS_CUDA(cudaMalloc(&s->d_sums, 2 * sizeof(double)));
	launch_divergence(s->view(), of_advected ? s->adv : s->vel, s->div, 1.0f / s->grid->voxel_size, st);
	HNS_CUDA(cudaMemsetAsync(s->d_sums, 0, 2 * sizeof(double), st));
	launch_sum_squares(s->view(), s->div, s->d_sums, st);
	HNS_CUDA(cudaMemcpyAsync(out, s->d_sums, sizeof(double), cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

}  // extern "C"
