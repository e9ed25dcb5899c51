/*
 * hns_b200.h -- C ABI of the B200-native HNanoSolver hot path (libhns_b200.so).
 *
 * Plain C: opaque handles, raw pointers, sizes, int error codes. No C++ types, no torch types, no exceptions
 * cross this boundary. Every entry point names the reference interface it replaces (paths relative to the
 * reference repository root). The C++ adapter that re-exports the reference's own seven launcher symbols on
 * top of this ABI is compat/hns_compat.cu (see INTEGRATION.md).
 *
 * Data contract (reference src/Utils/GridBuilder.hpp:156-166,221-239; src/Utils/GridData.hpp:16-166):
 *   - N = L * 512 voxels, L leaves (8^3 bricks). Host arrays are leaf-major; inside a leaf the voxel at local
 *     (x,y,z) is at offset (x<<6 | y<<3 | z). Leaves are in NanoVDB order (root tile, upper offset, lower offset).
 *   - coords:   int32[N][3]   (openvdb::Coord)
 *   - velocity: float[N][3]   (openvdb::Vec3f, AoS)
 *   - every scalar field: float[N]
 *   - NanoVDB value index of a voxel = 1 + its position in these arrays; 0 = background.
 *
 * All functions return HNS_OK (0) or a negative hns_status; hns_last_error() gives the message for the calling
 * thread. There is no CPU fallback: without a CUDA device every compute entry point fails with HNS_ERR_CUDA.
 */
#ifndef HNS_B200_H
#define HNS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HNS_B200_ABI_VERSION 1

typedef enum hns_status {
	HNS_OK = 0,
	HNS_ERR_INVALID_ARGUMENT = -1, /* reference: std::invalid_argument (src/Cuda/HNanoSolver.cu:12-23) */
	HNS_ERR_RUNTIME = -2,          /* reference: std::runtime_error   (src/Cuda/HNanoSolver.cu:34,44,62,196) */
	HNS_ERR_CUDA = -3,             /* reference: CUDA_CHECK throw     (src/Cuda/Utils.cuh:10-18) */
	HNS_ERR_TOPOLOGY = -4,         /* coords are not the dense, NanoVDB-ordered leaf blocks the kernels assume */
	HNS_ERR_UNSUPPORTED = -5
} hns_status;

typedef struct hns_grid hns_grid;   /* device index grid + leaf tables; replaces nanovdb::GridHandle<DeviceBuffer> */
typedef struct hns_state hns_state; /* device-resident fields of one simulation (persistent across frames)        */

/* reference: struct CombustionParams, src/Cuda/Kernels.cuh:6-13 (same field order) */
typedef struct hns_combustion_params {
	float expansionRate;
	float temperatureRelease;
	float buoyancyStrength;
	float ambientTemp;
	float vorticityScale;
	float factorScale;
} hns_combustion_params;

/* ---------------------------------------------------------------------------------------------------------
 * Library
 * ------------------------------------------------------------------------------------------------------- */
int hns_abi_version(void);
const char* hns_last_error(void);
/* Number of kernels of this library launched by the calling process since load / since the last reset. */
uint64_t hns_launch_count(void);
void hns_launch_count_reset(void);
/* Select the CUDA device used by subsequently created grids/states of the calling thread (cudaSetDevice). */
int hns_set_device(int device);
/* Packed advection (default on, or the environment variable HNS_ADVECT4): the gradient and combustion passes of a resident state also
 * write the fields they produce as float4 groups, and advect_vector / advect_scalars stage from those groups with 128-bit shared-memory
 * loads (advect.cu, third generation). Off = the kernels that stage the brick fields directly. Results are bit-identical either way;
 * the switch exists for A/B measurements and for the test that asserts exactly that. Returns the previous setting. */
int hns_set_packed_advection(int on);
/* Launches of the third-generation advection kernels so far in this process (they replace their second-generation counterparts one for
 * one, so hns_launch_count cannot tell them apart). */
uint64_t hns_packed_advection_launches(void);

/* ---------------------------------------------------------------------------------------------------------
 * Index grid -- replaces CreateIndexGrid (src/Cuda/HNanoSolver.cu:375-390), i.e.
 * nanovdb::tools::cuda::voxelsToGrid<ValueOnIndex>(coords, N, voxelSize) for HNS's dense-leaf sidecar.
 * ------------------------------------------------------------------------------------------------------- */
/* coords: HOST int32[n_voxels][3] exactly as HNS::GridIndexedData::pCoords() holds them. Only the first coord of
 * every 512-block is needed to build the grid. validate = 1 additionally checks (on the host) that every block is the dense brick in
 * offset order, validate = 2 spot-checks eight voxels per block (O(leaves): the drop-in CreateIndexGrid does this on every cook);
 * a violation is HNS_ERR_TOPOLOGY (the reference silently produces inconsistent results for such input). */
int hns_grid_create_from_coords(const int32_t* coords, uint64_t n_voxels, float voxel_size, int validate, hns_grid** out);
/* origins: HOST int32[n_leaves][3], multiples of 8, in NanoVDB order. */
int hns_grid_create_from_origins(const int32_t* origins, uint64_t n_leaves, float voxel_size, hns_grid** out);
void hns_grid_destroy(hns_grid* g);
uint64_t hns_grid_num_leaves(const hns_grid* g);
uint64_t hns_grid_num_voxels(const hns_grid* g);
float hns_grid_voxel_size(const hns_grid* g);
/* The NanoVDB 32.7 ValueOnIndex buffer (what voxelsToGrid emits; SURVEY.md Appendix C). */
uint64_t hns_grid_nanovdb_bytes(const hns_grid* g);
const void* hns_grid_nanovdb_device_ptr(const hns_grid* g);
int hns_grid_nanovdb_download(const hns_grid* g, void* dst_host);
/* getValue(ijk) for n HOST coordinates, evaluated on the device by walking the emitted NanoVDB buffer
 * (root tile scan -> upper -> lower -> leaf), i.e. nanovdb::ReadAccessor::getValue (externals/nanovdb/NanoVDB.h:5683-5698). */
int hns_grid_get_values(const hns_grid* g, const int32_t* ijk_host, uint64_t n, uint64_t* out_host);
/* Per-leaf 27-neighbour table (int32[L][27], -1 = no leaf; slot = (dx+1)*9 + (dy+1)*3 + (dz+1)) to HOST. */
int hns_grid_neighbors_download(const hns_grid* g, int32_t* dst_host);

/* ---------------------------------------------------------------------------------------------------------
 * Domain construction on the device -- replaces the per-cook OpenVDB pass of SOP_HNanoSolverVerb::cook
 * (src/SOP/HNanoSolver/SOP_HNanoSolver.cpp:188-199): topologyUnion(velocity tree), dilateVoxels(padding, NN_FACE_EDGE_VERTEX),
 * topologyUnion(sdf tree); the leaf nodes of the result are the bricks of the sidecar (src/Utils/GridBuilder.hpp:221-239).
 * vel_origins: HOST int32[n_vel][3] leaf origins of the velocity grid (any order); vel_masks: HOST uint64[n_vel][8] active-voxel masks
 * of those leaves (bit x<<6 | y<<3 | z, i.e. word x, bit y*8+z -- the leaf mask layout of OpenVDB and NanoVDB) or NULL = every voxel
 * active; padding in voxels (0..64); sdf_origins: HOST int32[n_sdf][3] leaf origins of the collision SDF grid (n_sdf = 0 without one).
 * Result: the domain's leaf origins in NanoVDB order = the `origins` argument of hns_grid_create_from_origins.
 * Coordinates must lie within +-(2^23 - 128) voxels.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct hns_domain hns_domain;
int hns_domain_build(const int32_t* vel_origins, const uint64_t* vel_masks, uint64_t n_vel, int padding, const int32_t* sdf_origins, uint64_t n_sdf,
                     hns_domain** out);
void hns_domain_destroy(hns_domain* d);
uint64_t hns_domain_num_leaves(const hns_domain* d);
int hns_domain_origins(const hns_domain* d, int32_t* origins_out);       /* HOST int32[num_leaves][3] */
int hns_domain_create_grid(const hns_domain* d, float voxel_size, hns_grid** out);

/* ---------------------------------------------------------------------------------------------------------
 * NanoVDB files (host only, no GPU): the index grid as an uncompressed .nvdb segment -- FileHeader, FileMetaData, name, raw grid;
 * reference externals/nanovdb/NanoVDB.h:6252-6422 -- readable by stock NanoVDB tools, and back. The sidecar arrays are plain
 * float arrays in leaf order and are stored by the caller next to it (hnanosolver_b200/io.py uses .npy).
 * ------------------------------------------------------------------------------------------------------- */
int hns_nvdb_write(const char* path, const void* nanovdb_buffer, uint64_t bytes);   /* e.g. the bytes of hns_grid_nanovdb_download */
int hns_nvdb_file_grid_bytes(const char* path, uint64_t* bytes_out);                /* size of the first grid in the file */
int hns_nvdb_read(const char* path, void* dst, uint64_t capacity);                  /* segment files and raw buffer dumps, codec NONE */
/* leaf origins (int32[L][3], NanoVDB order; may be NULL to query L) and voxel size of a ValueOnIndex grid buffer on the host:
 * the arguments of hns_grid_create_from_origins */
int hns_nvdb_leaf_origins(const void* nanovdb_buffer, uint64_t bytes, int32_t* origins_out, uint64_t* num_leaves_out, float* voxel_size_out);

/* Value grids <-> sidecar blocks (host only): what IndexGridBuilder::build / writeIndexGrid do over OpenVDB grids
 * (src/Utils/GridBuilder.hpp:87-166, 168-216), over NanoVDB float (GridType 1) and Vec3f (GridType 6) grids, which carry the same
 * 512-value leaf buffers. `buffer` is a host copy of one grid (hns_nvdb_read). */
int hns_nvdb_grid_info(const void* buffer, uint64_t bytes, uint32_t* grid_type, uint32_t* grid_class, uint64_t* num_leaves, float* voxel_size,
                       char* name256);
/* leaf origins (int32[L][3]) and active-voxel masks (uint64[L][8], bit x<<6|y<<3|z) in the buffer's leaf order: the topology inputs of
 * hns_domain_build; either may be NULL */
int hns_nvdb_leaf_topology(const void* buffer, uint64_t bytes, int32_t* origins_out, uint64_t* masks_out, uint64_t* num_leaves_out);
/* build(): per domain leaf the grid's whole leaf buffer at that origin, or 512 values whose bytes are `fill_byte` where the grid has no
 * leaf (0 for float / vector blocks; 1 for the collision SDF, GridBuilder.hpp:108). out: float[n_leaves*512] or float[n_leaves*512][3] */
int hns_sidecar_from_nanovdb(const void* buffer, uint64_t bytes, const int32_t* domain_origins, uint64_t n_leaves, int fill_byte, void* out);
/* writeIndexGrid(): a float grid of class FogVolume (components 1) or a Vec3f grid of class Staggered (components 3) named `name` with
 * a leaf at every domain origin (NanoVDB order) holding the block's values; masks: uint64[n_leaves][8] or NULL = every voxel active.
 * out_buf must hold hns_sidecar_nanovdb_bytes(...) bytes; write it with hns_nvdb_write. */
uint64_t hns_sidecar_nanovdb_bytes(const int32_t* domain_origins, uint64_t n_leaves, int components);
int hns_sidecar_to_nanovdb(const int32_t* domain_origins, uint64_t n_leaves, const uint64_t* masks, const void* values, int components,
                           float voxel_size, const char* name, void* out_buf, uint64_t capacity);

/* ---------------------------------------------------------------------------------------------------------
 * One-shot launchers on HOST sidecar arrays, in place, synchronous -- the drop-in equivalents of the reference's
 * extern "C" launchers. `stream` is a cudaStream_t passed as void* (may be NULL).
 * ------------------------------------------------------------------------------------------------------- */
/* The one-shot launchers keep one scratch set of device buffers per process and reuse it while the problem size stays the same
 * (the reference allocates and frees everything on every call), and hns_grid_destroy keeps the device block of up to four destroyed
 * index grids for the next hns_grid_create_* of similar size; this frees both. */
void hns_release_scratch(void);
/* Compute_Sim (src/Cuda/HNanoSolver.cu:9-372,393-396): advect velocity -> [vorticity] -> divergence -> combustion ->
 * buoyancy -> iterations x (red, black) -> gradient subtract -> advect all float fields. float_names/float_fields are
 * the float blocks in insertion order (GridData.hpp:136-145); fuel, waste, temperature, flame must be among them.
 * A block named "collision_sdf" is never advected and comes back zeroed (the reference copies back an output buffer it never
 * writes, :361-369); with has_collision != 0 it is the SDF of the collision path (enforceCollisionBoundaries before the advection
 * and after the projection, collision tests of the traced positions, boundary tails of advect_vector and the gradient subtract).
 * The host arrays cross PCIe on two copy streams while the kernels run: uploads in the order the projected velocity depends on them
 * (velocity; fuel and waste -> the solve can start; temperature -> the gradient pass; flame and the other blocks), downloads as soon
 * as a result is final. The independent steps of the combustion stage run in that order too; every value is the reference's. */
int hns_compute_sim(const hns_grid* g, float* velocity, int n_float, const char* const* float_names, float* const* float_fields,
                    int iterations, float dt, float voxel_size, const hns_combustion_params* params, int has_collision, void* stream);
/* AdvectIndexGrid (src/Cuda/Advection.cu:13-112,169-171): BFECC advection of every float block by the velocity block. */
int hns_advect_index_grid(const int32_t* coords, uint64_t n_voxels, const float* velocity, int n_float, float* const* float_fields,
                          float dt, float voxel_size, void* stream);
/* AdvectIndexGridVelocity (src/Cuda/Advection.cu:114-166,173-175): BFECC self-advection of the velocity block. */
int hns_advect_index_grid_velocity(const int32_t* coords, uint64_t n_voxels, float* velocity, float dt, float voxel_size, void* stream);
/* ProjectNonDivergent (src/Cuda/PressureProjection.cu:9-78,132-135). */
int hns_project_non_divergent(const int32_t* coords, uint64_t n_voxels, float* velocity, uint64_t iterations, float voxel_size,
                              void* stream);
/* Divergence (src/Cuda/PressureProjection.cu:81-129): writes the "divergence" float block. */
int hns_divergence(const int32_t* coords, uint64_t n_voxels, const float* velocity, float* divergence_out, float voxel_size, void* stream);
/* CombustionKernel (src/Cuda/Combustion.cu:9-70): the reference's kernel launch is commented out (:55) and it copies an
 * unwritten buffer over the host velocity (:57). Exported for symbol parity as a validated no-op. */
int hns_combustion_kernel(const hns_grid* g, float* velocity, uint64_t n_voxels, float dt, float voxel_size, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Device-resident simulation state: what the reference re-uploads every frame (src/Cuda/HNanoSolver.cu:87-133)
 * lives on the device across frames here. Used by the headless driver, bench.py and the multi-GPU runner.
 * ------------------------------------------------------------------------------------------------------- */
int hns_state_create(const hns_grid* g, int n_scalars, hns_state** out);
void hns_state_destroy(hns_state* s);
/* HOST <-> device, converting between the sidecar layout (AoS Vec3f, float[N]) and the internal brick layout. */
int hns_state_upload_velocity(hns_state* s, const float* velocity_host);
int hns_state_download_velocity(hns_state* s, float* velocity_host);
int hns_state_upload_scalar(hns_state* s, int index, const float* host);
int hns_state_download_scalar(hns_state* s, int index, float* host);
/* intermediate fields of the last step, for parity checks: which = 0 divergence, 1 pressure, 2 advected velocity (float[N][3]) */
int hns_state_download_aux(hns_state* s, int which, float* host);

/* Enables the combustion_oxygen + temperature_buoyancy stage of the all-in-one frame (src/Cuda/HNanoSolver.cu:190-250) on the
 * scalar fields with the given indices, and the vorticityConfinement pass (Kernel.cu:969-1025) between advect_vector and the
 * divergence when params->vorticityScale != 0 and (int)params->factorScale != 0. The reference runs that kernel in place
 * (HNanoSolver.cu:174), which races; here it is evaluated out of place (what the kernel computes when given two buffers). */
int hns_state_set_combustion(hns_state* s, int enabled, int i_fuel, int i_waste, int i_temperature, int i_flame,
                             const hns_combustion_params* params);

/* One frame on resident state: advect_vector -> divergence -> iterations x (red, black) -> gradient subtract ->
 * advect_scalars (all n_scalars fields); with hns_state_set_combustion the combustion + buoyancy stage runs after the divergence,
 * exactly as in Compute(). Same arithmetic as the corresponding steps of Compute() (HNanoSolver.cu:159-356);
 * omega = 2/(1+sinf(3.14159f*voxel_size)) (HNanoSolver.cu:257). Asynchronous on `stream`.
 * flags: bit 1 = walk the leaves front to back in every pressure half-sweep (default: black sweeps run back to front so that each
 * launch starts on the bricks still resident in L2). */
int hns_state_step(hns_state* s, int iterations, float dt, unsigned flags, void* stream);
/* Individual steps on resident state (asynchronous). */
int hns_state_advect_velocity(hns_state* s, float dt, void* stream);                 /* vel -> adv              */
/* Collision path (reference hasCollision): scalar `sdf_scalar_index` is the collision SDF (-1 switches the path off). The scalar
 * is then never advected, hns_state_step / hns_state_advect_velocity / _subtract_gradient / _advect_scalars apply the reference's
 * collision handling, and hns_state_enforce_collision is enforceCollisionBoundaries (Kernel.cu:77-116) on the velocity, which
 * hns_state_step runs before the advection and after the projection (HNanoSolver.cu:153-157, 292-296). */
int hns_state_set_collision(hns_state* s, int sdf_scalar_index);
int hns_state_collision_active(const hns_state* s);
int hns_state_enforce_collision(hns_state* s, void* stream);
int hns_state_vorticity_confinement(hns_state* s, float dt, float scale, float factor_scale, void* stream); /* adv -> adv, out of place */
/* the same in its two launches (a sharded run exchanges the ghost leaves of field 26 = |curl| in between); _active: does the
 * configured frame (hns_state_set_combustion) contain the pass at all? */
int hns_state_vorticity_active(const hns_state* s);
int hns_state_vorticity_mag(hns_state* s, void* stream);                                        /* adv -> |curl| (field 26) */
int hns_state_vorticity_force(hns_state* s, float dt, float scale, float factor_scale, void* stream); /* adv, |curl| -> adv */
int hns_state_divergence(hns_state* s, int of_advected, void* stream);               /* adv|vel -> div          */
int hns_state_pressure_solve(hns_state* s, int iterations, float omega, unsigned flags, void* stream); /* p = 0; RBGS   */
int hns_state_subtract_gradient(hns_state* s, int from_advected, void* stream);      /* adv|vel, p -> vel       */
/* Pieces of the pressure solve and of the combustion stage, for drivers that interleave ghost exchanges (sharded runs). */
int hns_state_pressure_init(hns_state* s, void* stream);                              /* p = 0                   */
int hns_state_pressure_half_sweep(hns_state* s, int color, float omega, int reverse, void* stream); /* one red (0) / black (1) sweep */
int hns_state_combustion_buoyancy(hns_state* s, float dt, void* stream);              /* combustion_oxygen + temperature_buoyancy */
/* omega exactly as Compute() (src/Cuda/HNanoSolver.cu:257, float sinf) and pressure_projection_idx (PressureProjection.cu:53, double sin) evaluate it */
float hns_omega_compute(float voxel_size);
float hns_omega_project(float voxel_size);
int hns_state_advect_scalars(hns_state* s, float dt, int sampler_semantics, void* stream); /* 0: advect_scalars, 1: advect_scalar */
int hns_state_sync(hns_state* s, void* stream);
/* Timed run of `frames` identical frames (state is restored between frames) with CUDA events on `stream`;
 * ms_total = whole loop, ms_pressure = time inside the pressure solve only. */
int hns_state_time_frames(hns_state* s, int frames, int iterations, float dt, unsigned flags, void* stream, float* ms_total,
                          float* ms_pressure);

/* ---------------------------------------------------------------------------------------------------------
 * Device-side norms (fp64; per-thread partial sums, warp shuffles, one atomic per warp) and the multigrid pressure solve.
 * Reference: compute_residual, restrict_to_4x4x4, restrict_to_2x2x2, prolongate are declared but never defined
 * (src/Cuda/Kernels.cuh:38-49) and their caller v_cycle is commented out (src/Cuda/HNanoSolver.cu:399-507): the reference never
 * evaluates a residual. These entry points provide what that sketch intends, on the same equation as its red-black sweep
 * (src/Cuda/Kernel.cu:591-623): (sum of the 6 neighbours - 6 p) / dx^2 = div, p = 0 outside the domain.
 * ------------------------------------------------------------------------------------------------------- */
/* out2[0] = sum over voxels of (div - L p)^2, out2[1] = sum of div^2, for the state's current pressure and divergence; over the leaves the
 * state's kernels process (all of them, or the owned leaves of a shard: add the ranks' sums with hns_dist_allreduce_sum). Synchronous. */
int hns_state_residual_sums(hns_state* s, double* out2, void* stream);
/* *out = sum of squares of the divergence (reference kernel `divergence`, src/Cuda/Kernel.cu:499-519) of the current velocity
 * (of_advected = 0) or of the advected velocity (1). OVERWRITES the state's divergence field. Synchronous. */
int hns_state_divergence_sum_squares(hns_state* s, int of_advected, double* out, void* stream);
/* Multigrid hierarchy over an index grid: level k+1 has cells twice the size of level k, a cell belongs to the domain iff all 8 of its
 * children do, leaves of level k+1 are 2x2x2 leaves of level k; coarsening stops at a single leaf, when no cell is fully covered any
 * more, or after max_levels (<= 0: no cap). The grid must outlive the hierarchy. */
typedef struct hns_mg hns_mg;
int hns_mg_create(const hns_grid* g, int max_levels, hns_mg** out);
void hns_mg_destroy(hns_mg* mg);
int hns_mg_num_levels(const hns_mg* mg);
uint64_t hns_mg_level_leaves(const hns_mg* mg, int level);
uint64_t hns_mg_level_cells(const hns_mg* mg, int level);   /* cells inside the domain on that level */
int hns_mg_set_coarsest_iterations(hns_mg* mg, int iterations); /* red-black iterations on the last level (default 32) */
/* p = 0, then V(nu_pre, nu_post) cycles (red-black sweeps with relaxation factor omega_smooth on every level, full-weighting
 * restriction of the residual, trilinear prolongation of the correction) until the relative residual
 * sqrt(sum (div - L p)^2 / sum div^2) <= rel_tol or max_cycles cycles have run; rel_tol <= 0: exactly max_cycles cycles and no residual
 * evaluation (asynchronous). Single-GPU states only. */
int hns_state_pressure_solve_mg(hns_state* s, hns_mg* mg, int max_cycles, double rel_tol, int nu_pre, int nu_post, float omega_smooth, void* stream);
int hns_mg_last_cycles(const hns_mg* mg);
double hns_mg_last_relative_residual(const hns_mg* mg);     /* -1 when the last solve did not evaluate it */
/* Makes hns_state_step / hns_state_time_frames solve the pressure with `cycles` V-cycles instead of the reference's `iterations`
 * red-black SOR sweeps (mg = NULL switches back). Not the reference's arithmetic: results then differ from Compute_Sim's by the
 * difference in how far the two solves converge. */
int hns_state_set_pressure_solver(hns_state* s, hns_mg* mg, int cycles, int nu_pre, int nu_post, float omega_smooth);

/* Ghost-leaf exchange support for spatially sharded runs (one process per GPU): pack/unpack whole bricks of one
 * internal field by leaf id list into/from a contiguous device buffer (float[n_ids][512]).
 * field: 0..2 velocity components, 3..5 advected velocity components, 6/7 pressure red/black half, 8/9 divergence red/black half,
 * 10+i scalar i. Pressure and divergence are stored colour-split (red = (x+y+z) even): 256 floats per leaf and half; every other
 * field has 512 floats per leaf (hns_state_field_floats_per_leaf). */
int hns_state_field_floats_per_leaf(int field);
/* advect_scalars reads "array element 0" for inactive voxels (reference src/Cuda/Kernel.cu:192,225). A shard's plan
 * (hnanosolver_b200/dist.py::make_plan) makes global leaf 0 local leaf 0 on every rank, so a shard's element 0 is the global one. */
int hns_state_pack_leaves(hns_state* s, int field, const int32_t* leaf_ids_dev, uint64_t n_ids, float* dst_dev, void* stream);
int hns_state_unpack_leaves(hns_state* s, int field, const int32_t* leaf_ids_dev, uint64_t n_ids, const float* src_dev, void* stream);
void* hns_state_field_device_ptr(hns_state* s, int field);

/* ---------------------------------------------------------------------------------------------------------
 * Spatially sharded runs (one process per GPU). New: the reference is single-GPU. The partition (contiguous leaf ranges of the
 * NanoVDB-ordered leaf list + 26-neighbour ghost leaves) is computed by the caller; a rank's hns_grid / hns_state cover its owned
 * + ghost leaves. NCCL (bound at run time) carries the ghost bricks on the same stream as the kernels.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct hns_dist hns_dist;
int hns_dist_unique_id(uint8_t* out128);                                  /* rank 0: ncclGetUniqueId; ship the 128 bytes to all ranks */
/* ncclCommInitRank on the current device. id128 == NULL: no communicator at all -- the peer-memory exchange (hns_dist_ipc_*) is then
 * the only data path and must be connected before the first frame (this also lets several ranks share one GPU, which NCCL refuses). */
int hns_dist_create(const uint8_t* id128, int rank, int world, hns_dist** out);
/* Lifetime: hns_dist_set_plan points the state at work lists owned by the hns_dist (owned leaves); after
 * hns_dist_destroy the state must be destroyed too or re-planned before it launches anything. Synchronise with the peers first:
 * destroying unmaps memory a peer may still be storing into. */
void hns_dist_destroy(hns_dist* d);
/* per peer: LOCAL leaf ids (HOST arrays) of the owned leaves it holds as ghosts (send) and of the ghost leaves it owns (recv),
 * both in ascending global leaf order so that the two sides agree; owned_ids: LOCAL ids of all owned leaves (kernels skip the
 * ghost leaves). Installs the owned-leaf work list on `s`. */
int hns_dist_set_plan(hns_dist* d, hns_state* s, int n_peers, const int* peer_ranks, const uint64_t* n_send, const int32_t* const* send_ids,
                      const uint64_t* n_recv, const int32_t* const* recv_ids, uint64_t n_owned, const int32_t* owned_ids);
/* Direct peer-memory ghost exchange (CUDA IPC over NVLink/NVSwitch) instead of ncclSend/ncclRecv: bricks are stored straight into
 * the peer's landing block and a flag is raised; in the pressure solve the boundary sweep kernel itself stores every swept quad into
 * the peers' ghost copies (their pressure arrays mapped over NVLink) and a one-warp kernel behind it raises the flag -- no pack / send /
 * unpack at all.
 * Setup: every rank calls _prepare (192 opaque bytes: IPC handles of the landing block and of the pressure allocation, offsets of the
 * red and black halves inside it; plus the byte offset of
 * each peer's region inside the block, in the order of hns_dist_set_plan's peers), the caller all-gathers them together with its recv
 * leaf lists, calls _connect once per peer with that peer's 192 handle bytes, the offset of ITS OWN region inside the peer's block and,
 * for every leaf of its send list to that peer, the leaf's id in the peer's local numbering (= the peer's recv list for this rank),
 * then _finish. hns_dist_error reports a flag wait that timed out (0 = none). */
int hns_dist_ipc_prepare(hns_dist* d, uint8_t* handle_out64, uint64_t* region_offsets_out);
int hns_dist_ipc_connect(hns_dist* d, int peer_index, const uint8_t* peer_handles192, uint64_t my_region_offset_in_peer_block,
                         const int32_t* peer_leaf_ids);
int hns_dist_ipc_finish(hns_dist* d);
/* device-side error word, sticky until reset: 0 = clean; low byte = 1 + the channel of a peer-flag wait that gave up after ~4 s (the
 * frame then ran on stale ghosts); bit 8 = a semi-Lagrangian sample of advect_vector / advect_scalars landed outside the 3x3x3 leaf
 * neighbourhood of its leaf, i.e. possibly beyond the shard's one-leaf ghost layer (more than ~8 voxels of back-trace), where the
 * sharded result can differ from the single-GPU one. hns_dist_cook and hns_dist_frame_timed return HNS_ERR_RUNTIME when it is set;
 * after the asynchronous hns_dist_frame the caller polls it at its next synchronisation point. */
int hns_dist_error(hns_dist* d, uint32_t* out);
int hns_dist_reset_error(hns_dist* d);
/* ghost exchange of the given fields (ids as for hns_state_pack_leaves): pack, grouped ncclSend/ncclRecv, unpack; asynchronous */
int hns_dist_exchange(hns_dist* d, hns_state* s, int n_fields, const int* fields, void* stream);
/* the whole sharded frame (same steps as hns_state_step) with its 3 + 2*iterations ghost exchanges; the exchange of a swept
 * pressure colour overlaps the sweep of the interior leaves, the scalars' exchange hides behind the pressure solve (peer-memory
 * mode); asynchronous. COLLECTIVE: every rank calls it, and every call that overwrites the state's velocity between two frames
 * (hns_state_upload_velocity, hns_state_step, ...) must be made on all ranks alike -- a frame whose velocity is untouched since the
 * previous sharded frame skips the leading velocity-ghost exchange (those ghosts are still current), and the ranks must agree on
 * that; a disagreement surfaces as a flag time-out in hns_dist_error, not as wrong values. */
int hns_dist_frame(hns_dist* d, hns_state* s, int iterations, float dt, void* stream);
/* the sharded cook on HOST arrays of this rank's local voxels (owned + ghost leaves; velocity float[n][3] and the state's scalar
 * fields float[n] in index order), in place, synchronous: upload, hns_dist_frame, download. Collective. Pinned host memory lets the
 * copies run at PCIe rate; the ranks' transfers go over their own links in parallel. Ghost entries of the inputs need not be valid
 * (every field's ghosts, the collision SDF's included, are exchanged before they are read). */
int hns_dist_cook(hns_dist* d, hns_state* s, float* velocity, int n_float, float* const* fields, int iterations, float dt, void* stream);
/* the same frame with CUDA events between its phases (ms_out[8]: exchange velocity, advect_vector, exchange advected velocity,
 * divergence + combustion, pressure solve incl. exchanges, gradient, final exchange, advect_scalars); synchronises the stream */
int hns_dist_frame_timed(hns_dist* d, hns_state* s, int iterations, float dt, void* stream, float* ms_out);
/* in-place sum over all ranks of n <= 16 HOST doubles (ncclAllReduce, fp64): the global residual / divergence norms of a sharded solve
 * from the ranks' hns_state_residual_sums / hns_state_divergence_sum_squares. Synchronous, collective. HNS_ERR_UNSUPPORTED without a
 * communicator (hns_dist_create with a NULL id). */
int hns_dist_allreduce_sum(hns_dist* d, double* inout_host, int n, void* stream);
uint64_t hns_dist_bytes_sent(const hns_dist* d);
uint64_t hns_dist_exchanges(const hns_dist* d);
/* Sharded multigrid pressure solve: hns_dist_frame / _cook / _frame_timed then run `cycles` V(nu_pre, nu_post) cycles instead of the
 * red-black solve (`iterations` is then unused). Level 0 is the shard (sweeps on the owned leaves with their ghost exchanges), levels >= 1
 * are replicated: the ranks' restricted residuals are gathered into every rank's level-1 right-hand side through peer memory, and
 * every rank runs the coarse levels itself. The owned voxels equal those of hns_state_set_pressure_solver's single-GPU frame bit for
 * bit. `mg` is an hns_mg over the GLOBAL grid (its levels >= 1 are the single-GPU hierarchy; its coarse arrays are used by this
 * solver, so do not solve with it elsewhere at the same time; it must outlive the setting); local_to_global[i] = the global leaf id
 * of local leaf i (every leaf of the bound state, owned and ghost). mg = NULL switches back to red-black (other arguments ignored);
 * so does a refused call (bad cycles / nu / omega, ids out of range or not matching the hierarchy's level-0 leaves).
 * Setup, collective: every rank calls _set_pressure_solver (64 opaque bytes out: the IPC handle of its level-1 block; may be NULL with
 * one rank), the caller all-gathers them, calls _mg_connect with the handle of every OTHER rank, then _mg_finish; the solver takes
 * effect at _mg_finish. HNS_ERR_UNSUPPORTED with more than one rank and no peer-memory exchange (the NCCL fallback). A gather that
 * waits for a rank longer than ~4 s sets the error word (hns_dist_error: low byte 11). */
int hns_dist_set_pressure_solver(hns_dist* d, hns_state* s, hns_mg* mg, const int32_t* local_to_global, int cycles, int nu_pre, int nu_post,
                                 float omega_smooth, uint8_t* handle_out64);
int hns_dist_mg_connect(hns_dist* d, int rank, const uint8_t* handle64);
int hns_dist_mg_finish(hns_dist* d);
/* V-cycles that gathered a level-1 right-hand side, and the bytes this rank stored into the other ranks' copies, since hns_dist_create */
uint64_t hns_dist_mg_gathers(const hns_dist* d);
uint64_t hns_dist_mg_gather_bytes(const hns_dist* d);

#ifdef __cplusplus
}
#endif
#endif /* HNS_B200_H */
