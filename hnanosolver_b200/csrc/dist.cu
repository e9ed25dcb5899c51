// Spatially sharded frame, one process per GPU: the whole frame with its ghost-leaf exchanges as ONE library call, NCCL issued
// from C++ on the same stream as the kernels (no Python between the launches: a pressure half-sweep takes ~60 us, a round trip
// through the interpreter per exchange more than that).
//
// The reference is single-GPU (no NCCL/MPI anywhere, SURVEY.md 2.1); this is new code. The decomposition itself -- contiguous
// ranges of the NanoVDB-ordered leaf list, 26-neighbour ghost leaves, per-peer send/recv leaf lists -- is computed on the host
// (hnanosolver_b200/dist.py::make_plan) and handed in through hns_dist_set_plan.
//
// NCCL is bound at run time (dlopen "libnccl.so.2") so that libhns_b200.so has no link-time dependency on it and shares the
// NCCL instance torch has already loaded in the same process.
#include <dlfcn.h>

#include <cstring>
#include <string>
#include <vector>

#include "kernels.cuh"

namespace hns {

// ---- minimal NCCL binding ------------------------------------------------------------------------------------------
typedef struct ncclComm* ncclComm_t;
struct ncclUniqueId {
	char internal[128];
};
enum { ncclSuccess = 0 };
enum { ncclFloat = 7, ncclDouble = 8 };  // ncclFloat32, ncclFloat64
enum { ncclSum = 0 };
struct Nccl {
	void* lib = nullptr;
	int (*GetUniqueId)(ncclUniqueId*) = nullptr;
	int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
	int (*CommDestroy)(ncclComm_t) = nullptr;
	int (*Send)(const void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*Recv)(void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
	int (*GroupStart)() = nullptr;
	int (*GroupEnd)() = nullptr;
	const char* (*GetErrorString)(int) = nullptr;
};
static Nccl g_nccl;
static int load_nccl() {
	if (g_nccl.lib) return HNS_OK;
	void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
	if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
	if (!h) return fail(HNS_ERR_RUNTIME, std::string("cannot load NCCL: ") + dlerror());
#define HNS_SYM(field, name)                                                                 \
	*reinterpret_cast<void**>(&g_nccl.field) = dlsym(h, name);                               \
	if (!g_nccl.field) return fail(HNS_ERR_RUNTIME, std::string("NCCL symbol missing: ") + name);
	HNS_SYM(GetUniqueId, "ncclGetUniqueId")
	HNS_SYM(CommInitRank, "ncclCommInitRank")
	HNS_SYM(CommDestroy, "ncclCommDestroy")
	HNS_SYM(Send, "ncclSend")
	HNS_SYM(Recv, "ncclRecv")
	HNS_SYM(AllReduce, "ncclAllReduce")
	HNS_SYM(GroupStart, "ncclGroupStart")
	HNS_SYM(GroupEnd, "ncclGroupEnd")
	HNS_SYM(GetErrorString, "ncclGetErrorString")
#undef HNS_SYM
	g_nccl.lib = h;
	return HNS_OK;
}
#define HNS_NCCL(call)                                                                                              \
	do {                                                                                                            \
		const int r_ = (call);                                                                                      \
		if (r_ != ncclSuccess) return ::hns::fail(HNS_ERR_RUNTIME, std::string(#call) + ": " + g_nccl.GetErrorString(r_)); \
	} while (0)

}  // namespace hns

using namespace hns;

struct hns_dist {
	ncclComm_t comm = nullptr;
	int rank = 0, world = 1;
	struct Peer {
		int rank;
		uint64_t n_send, n_recv;
		int32_t *d_send = nullptr, *d_recv = nullptr;  // local leaf ids
		float *buf_send = nullptr, *buf_recv = nullptr;
		// direct peer-memory path: where this peer's bricks land in MY block, and where mine land in ITS block
		uint64_t region_off = 0;
		uint8_t* remote_region = nullptr;
		void* ipc_base = nullptr;
		void* ipc_pbase = nullptr;                // the peer's pressure allocation mapped into this process
		void* ipc_p[2] = {nullptr, nullptr};      // the peer's p[red], p[black] inside it
		std::vector<int32_t> peer_leaf;            // for each entry of my send list: that leaf's id in the PEER's local numbering
	};
	std::vector<Peer> peers;
	int max_fields = 0;
	double* d_reduce = nullptr;  // staging of hns_dist_allreduce_sum
	uint64_t bytes_sent = 0, exchanges = 0;
	// work lists (local leaf ids, device): owned = boundary (sent to some peer) + interior
	int32_t *d_owned = nullptr, *d_boundary = nullptr, *d_interior = nullptr;
	int32_t *d_boundary_nbr = nullptr, *d_interior_nbr = nullptr;  // GridView::list_nbr of the two pressure work lists
	uint32_t n_owned = 0, n_boundary = 0, n_interior = 0;
	cudaStream_t comm_stream = nullptr;  // boundary sweeps + ghost exchange run here, next to the interior sweep on the caller's stream
	cudaEvent_t ev_exchanged = nullptr;
	cudaStream_t aux_stream = nullptr;  // the scalars' ghost exchange, hidden behind the pressure solve
	cudaEvent_t ev_scalars_final = nullptr, ev_scalars_exchanged = nullptr;
	uint64_t vel_exchanged_version = ~uint64_t(0);  // hns_state::vel_version whose velocity ghosts are current on every rank
	cudaEvent_t ev_I[2] = {}, ev_B[2] = {};
	// direct peer-memory ghost exchange (CUDA IPC over NVLink): one block of device memory per rank holding, per peer, five
	// channels of landing space + their arrival flags. Peers store bricks straight into it and then raise the channel's flag.
	bool p2p = false;
	uint8_t* block = nullptr;
	uint64_t block_bytes = 0;
	uint32_t** d_remote_flags = nullptr;  // [n_peers] flag words in the peers' blocks
	uint32_t** d_local_flags = nullptr;   // [n_peers] flag words in my block
	uint32_t seq[16] = {};  // per flag channel (kCh* below)
	uint32_t* d_err = nullptr;
	int n_scalars = 0;
	// fused boundary sweep + push: CSR over the boundary work list -> (peer index, leaf id on that peer)
	uint32_t* d_push_off = nullptr;
	int32_t *d_push_peer = nullptr, *d_push_leaf = nullptr;
	float** d_remote_p[2] = {nullptr, nullptr};  // [n_peers] per colour
	std::vector<int32_t> h_boundary;             // host copy of the boundary work list
	const hns_state* bound_state = nullptr;
	uint64_t push_bytes_per_sweep = 0;
	uint32_t* d_seq_base = nullptr;  // device [3]: sequence bases of the red pushes, black pushes, frames
	cudaStream_t copy_stream = nullptr;  // hns_dist_cook: host <-> device transfers overlapping the frame
	cudaEvent_t ev_copy[6] = {};
	// Sharded multigrid pressure solve (hns_dist_set_pressure_solver): level 0 is this rank's shard, levels >= 1 of `mg` (a hierarchy
	// over the GLOBAL grid) are replicated -- every rank runs the coarse part of every cycle itself on the gathered level-1 rhs.
	struct ShardedMg {
		hns_mg* mg = nullptr;          // null: the red-black solve
		bool ready = false;            // hns_dist_mg_finish has connected every rank
		int cycles = 0, nu_pre = 0, nu_post = 0;
		float omega = 1.f;
		int32_t* d_parent = nullptr;   // [local leaves] level-1 leaf of each local leaf (global level-1 numbering)
		uint8_t* block = nullptr;      // exposed to every rank: [flag words][level-1 rhs, cycle parity 0 (red | black)][parity 1]
		uint64_t flag_bytes = 0, rhs_floats = 0;  // rhs_floats: one colour-split array, both halves
		std::vector<void*> ipc;        // [world] the other ranks' blocks mapped into this process
		float** d_gather[2] = {nullptr, nullptr};  // per parity: [world][2] red / black of every rank's level-1 rhs
		uint32_t** d_sig = nullptr;    // [world - 1] my flag words in the other ranks' blocks
		uint32_t** d_wait = nullptr;   // [world - 1] the other ranks' flag words in my block
		uint32_t seq = 0;              // number of the last gather (cycles since set-up, across frames)
		uint64_t gathers = 0, gather_bytes = 0;
		cudaGraphExec_t graph[2] = {nullptr, nullptr};  // the coarse part, one per parity (its level-1 rhs pointer differs)
		uint64_t graph_launches[2] = {0, 0};
		int graph_coarsest[2] = {0, 0};
	} smg;
};

// CTA cap of the background scalar exchange: it must not starve the pressure sweeps it runs beside
constexpr int kAuxBlocks = 148;

// flag channels: 0..7 of the ghost exchanges (see dist_frame), 8 / 9 the red / black pressure exchanges of the sharded multigrid solve
// (landing in the regions of channels 2 / 3), 10 the level-1 gather. k_wait reports a time-out as 1 + channel in the error word.
constexpr int kChMgPressure = 8, kChMgGather = 10;

// ---- layout of one peer region: [flags 128 B][ch0 velocity 3 x 512n][ch1 advected velocity 3 x 512n][ch2 red p 256n][ch3 black p 256n]
//      [ch4 velocity + scalars (3+S) x 512n][ch5 |curl| 512n] floats, n = number of ghost leaves exchanged with that peer.
//      A region is only reused after a later handshake with the same peer, so a push can never overtake the unpack of the previous use.
static uint64_t channel_floats(int ch, uint64_t n, int S) {
	switch (ch) {
		case 0:
		case 1: return 3 * 512 * n;
		case 2:
		case 3: return 256 * n;
		case 5: return 512 * n;
		default: return uint64_t(3 + S) * 512 * n;
	}
}
static uint64_t channel_offset(int ch, uint64_t n, int S) {  // bytes from the region start
	uint64_t off = 128;
	for (int c = 0; c < ch; ++c) off += channel_floats(c, n, S) * sizeof(float);
	return off;
}
static uint64_t region_bytes(uint64_t n, int S) { return (channel_offset(6, n, S) + 255) & ~uint64_t(255); }

namespace hns {
// raise channel `ch` of every peer to `seq`: everything this stream wrote into the peers' blocks before is visible first
__global__ void k_signal(uint32_t* const* __restrict__ flags, int n, int ch, uint32_t seq) {
	__threadfence_system();
	const int t = threadIdx.x;
	if (t < n && flags[t]) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flags[t] + ch), "r"(seq) : "memory");
}
// wait until every peer has raised channel `ch` of my block to `seq` (bounded: ~4 s, then the error word is set instead of hanging)
__global__ void k_wait(uint32_t* const* __restrict__ flags, int n, int ch, uint32_t seq, uint32_t* __restrict__ err) {
	const int t = threadIdx.x;
	if (t < n && flags[t]) {
		uint32_t v = 0;
		const long long t0 = clock64();
		for (;;) {
			asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags[t] + ch) : "memory");
			if (int32_t(v - seq) >= 0) break;
			if (clock64() - t0 > 8000000000ll) {
				atomicExch(err, 1u + uint32_t(ch));
				break;
			}
			__nanosleep(64);
		}
	}
}
// The sequence numbers of the fused pressure pipeline's flags are *base + offset with the bases in device memory (base[0] red pushes,
// base[1] black pushes, base[2] frames), advanced by the pipeline's last kernel: every frame issues identical launches.
__global__ void k_signal_rel(uint32_t* const* __restrict__ flags, int n, int ch, const uint32_t* __restrict__ base, uint32_t offset) {
	__threadfence_system();
	const int t = threadIdx.x;
	if (t < n && flags[t]) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flags[t] + ch), "r"(*base + offset) : "memory");
}
__global__ void k_wait_rel(uint32_t* const* __restrict__ flags, int n, int ch, const uint32_t* __restrict__ base, uint32_t offset,
                           uint32_t* __restrict__ err) {
	const int t = threadIdx.x;
	if (t < n && flags[t]) {
		const uint32_t seq = *base + offset;
		uint32_t v = 0;
		const long long t0 = clock64();
		for (;;) {
			asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags[t] + ch) : "memory");
			if (int32_t(v - seq) >= 0) break;
			if (clock64() - t0 > 8000000000ll) {
				atomicOr(err, 1u + uint32_t(ch));
				break;
			}
			__nanosleep(64);
		}
	}
}
__global__ void k_advance_bases(uint32_t* base, uint32_t iterations) {
	if (threadIdx.x == 0) base[0] += iterations, base[1] += iterations, base[2] += 1u;
}
}  // namespace hns

extern "C" {

int hns_dist_unique_id(uint8_t* out128) {
	if (!out128) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	int rc = load_nccl();
	if (rc) return rc;
	ncclUniqueId id;
	HNS_NCCL(g_nccl.GetUniqueId(&id));
	std::memcpy(out128, id.internal, 128);
	return HNS_OK;
}

int hns_dist_create(const uint8_t* id128, int rank, int world, hns_dist** out) {
	if (!out || world < 1 || rank < 0 || rank >= world) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	if (!id128) {  // peer-memory only: no communicator; every exchange goes through the CUDA IPC path (hns_dist_ipc_*)
		auto* d = new hns_dist();
		d->rank = rank, d->world = world;
		*out = d;
		return HNS_OK;
	}
	int rc = load_nccl();
	if (rc) return rc;
	auto* d = new hns_dist();
	d->rank = rank, d->world = world;
	ncclUniqueId id;
	std::memcpy(id.internal, id128, 128);
	const int r = g_nccl.CommInitRank(&d->comm, world, id, rank);
	if (r != ncclSuccess) {
		delete d;
		return fail(HNS_ERR_RUNTIME, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r));
	}
	*out = d;
	return HNS_OK;
}

static void mg_release(hns_dist* d);

void hns_dist_destroy(hns_dist* d) {
	if (!d) return;
	mg_release(d);
	for (auto& p : d->peers) cudaFree(p.d_send), cudaFree(p.d_recv), cudaFree(p.buf_send), cudaFree(p.buf_recv);
	cudaFree(d->d_reduce);
	cudaFree(d->d_owned), cudaFree(d->d_boundary), cudaFree(d->d_interior);
	cudaFree(d->d_boundary_nbr), cudaFree(d->d_interior_nbr);
	for (auto& p : d->peers) {
		if (p.ipc_base) cudaIpcCloseMemHandle(p.ipc_base);
		if (p.ipc_pbase) cudaIpcCloseMemHandle(p.ipc_pbase);
	}
	cudaFree(d->d_push_off), cudaFree(d->d_push_peer), cudaFree(d->d_push_leaf), cudaFree(d->d_remote_p[0]), cudaFree(d->d_remote_p[1]);
	cudaFree(d->block), cudaFree(d->d_remote_flags), cudaFree(d->d_local_flags), cudaFree(d->d_err);
	for (auto& e : d->ev_I)
		if (e) cudaEventDestroy(e);
	for (auto& e : d->ev_B)
		if (e) cudaEventDestroy(e);
	cudaFree(d->d_seq_base);
	if (d->copy_stream) cudaStreamDestroy(d->copy_stream);
	for (auto& e : d->ev_copy)
		if (e) cudaEventDestroy(e);
	if (d->comm_stream) cudaStreamDestroy(d->comm_stream);
	if (d->aux_stream) cudaStreamDestroy(d->aux_stream);
	if (d->ev_scalars_final) cudaEventDestroy(d->ev_scalars_final);
	if (d->ev_scalars_exchanged) cudaEventDestroy(d->ev_scalars_exchanged);
	if (d->ev_exchanged) cudaEventDestroy(d->ev_exchanged);
	if (d->comm) g_nccl.CommDestroy(d->comm);
	delete d;
}

int hns_dist_set_plan(hns_dist* d, hns_state* s, int n_peers, const int* peer_ranks, const uint64_t* n_send, const int32_t* const* send_ids,
                      const uint64_t* n_recv, const int32_t* const* recv_ids, uint64_t n_owned, const int32_t* owned_ids) {
	if (!d || !s || n_peers < 0 || (n_owned && !owned_ids)) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	mg_release(d);  // its parent table is per local leaf of the previous plan
	{
		// owned = boundary (in some send list) + interior; kernels then skip the ghost leaves altogether
		std::vector<char> is_boundary(s->grid->num_leaves, 0);
		for (int i = 0; i < n_peers; ++i)
			for (uint64_t k = 0; k < n_send[i]; ++k) is_boundary[send_ids[i][k]] = 1;
		std::vector<int32_t> bnd, inter;
		for (uint64_t k = 0; k < n_owned; ++k) (is_boundary[owned_ids[k]] ? bnd : inter).push_back(owned_ids[k]);
		cudaFree(d->d_owned), cudaFree(d->d_boundary), cudaFree(d->d_interior);
		d->d_owned = d->d_boundary = d->d_interior = nullptr;
		d->n_owned = uint32_t(n_owned), d->n_boundary = uint32_t(bnd.size()), d->n_interior = uint32_t(inter.size());
		auto up = [](const std::vector<int32_t>& v, int32_t** dst) {
			if (v.empty()) return cudaSuccess;
			cudaError_t e = cudaMalloc(dst, v.size() * sizeof(int32_t));
			return e != cudaSuccess ? e : cudaMemcpy(*dst, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
		};
		HNS_CUDA(up(std::vector<int32_t>(owned_ids, owned_ids + n_owned), &d->d_owned));
		HNS_CUDA(up(bnd, &d->d_boundary));
		d->h_boundary = bnd;
		HNS_CUDA(up(inter, &d->d_interior));
		cudaFree(d->d_boundary_nbr), cudaFree(d->d_interior_nbr);
		d->d_boundary_nbr = d->d_interior_nbr = nullptr;
		HNS_CUDA(cudaMalloc(&d->d_boundary_nbr, std::max<size_t>(bnd.size(), 1) * 27 * sizeof(int32_t)));
		HNS_CUDA(cudaMalloc(&d->d_interior_nbr, std::max<size_t>(inter.size(), 1) * 27 * sizeof(int32_t)));
		launch_gather_nbr_rows(s->grid->view.nbr, d->d_boundary, d->n_boundary, d->d_boundary_nbr, nullptr);
		launch_gather_nbr_rows(s->grid->view.nbr, d->d_interior, d->n_interior, d->d_interior_nbr, nullptr);
		HNS_CUDA(cudaDeviceSynchronize());
		s->active = d->d_owned, s->n_active = d->n_owned;
		if (!d->comm_stream) {
			int prio_lo = 0, prio_hi = 0;  // the exchange kernels are tiny and latency-critical: let their CTAs overtake the queued interior sweep
			cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
			HNS_CUDA(cudaStreamCreateWithPriority(&d->comm_stream, cudaStreamNonBlocking, prio_hi));
			HNS_CUDA(cudaStreamCreateWithFlags(&d->aux_stream, cudaStreamNonBlocking));
			HNS_CUDA(cudaEventCreateWithFlags(&d->ev_scalars_final, cudaEventDisableTiming));
			HNS_CUDA(cudaEventCreateWithFlags(&d->ev_scalars_exchanged, cudaEventDisableTiming));
			HNS_CUDA(cudaEventCreateWithFlags(&d->ev_exchanged, cudaEventDisableTiming));
			for (auto& e : d->ev_I) HNS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
			for (auto& e : d->ev_B) HNS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
		}
	}
	for (auto& p : d->peers) cudaFree(p.d_send), cudaFree(p.d_recv), cudaFree(p.buf_send), cudaFree(p.buf_recv);
	d->peers.clear();
	d->max_fields = 3 + s->n_scalars;
	for (int i = 0; i < n_peers; ++i) {
		hns_dist::Peer p{};
		p.rank = peer_ranks[i], p.n_send = n_send[i], p.n_recv = n_recv[i];
		if (p.n_send) {
			HNS_CUDA(cudaMalloc(&p.d_send, p.n_send * sizeof(int32_t)));
			HNS_CUDA(cudaMemcpy(p.d_send, send_ids[i], p.n_send * sizeof(int32_t), cudaMemcpyHostToDevice));
			HNS_CUDA(cudaMalloc(&p.buf_send, p.n_send * 512 * sizeof(float) * d->max_fields));
		}
		if (p.n_recv) {
			HNS_CUDA(cudaMalloc(&p.d_recv, p.n_recv * sizeof(int32_t)));
			HNS_CUDA(cudaMemcpy(p.d_recv, recv_ids[i], p.n_recv * sizeof(int32_t), cudaMemcpyHostToDevice));
			HNS_CUDA(cudaMalloc(&p.buf_recv, p.n_recv * 512 * sizeof(float) * d->max_fields));
		}
		d->peers.push_back(p);
	}
	// advect_scalars' "inactive -> element 0": the plan keeps global leaf 0 on every rank as LOCAL leaf 0 (a ghost fed by rank 0 in the
	// exchange before advect_scalars), so element 0 of the local arrays is the global one
	if (!d->d_err) {
		HNS_CUDA(cudaMalloc(&d->d_err, sizeof(uint32_t)));
		HNS_CUDA(cudaMemset(d->d_err, 0, sizeof(uint32_t)));
	}
	s->far_flag = d->d_err;  // a semi-Lagrangian sample beyond the ghost layer is reported, not silently treated as inactive
	d->n_scalars = s->n_scalars;
	d->bound_state = s;
	d->vel_exchanged_version = ~uint64_t(0);
	if (!d->d_seq_base) {
		HNS_CUDA(cudaMalloc(&d->d_seq_base, 3 * sizeof(uint32_t)));
		HNS_CUDA(cudaMemset(d->d_seq_base, 0, 3 * sizeof(uint32_t)));
	}
	return HNS_OK;
}

int hns_dist_exchange(hns_dist* d, hns_state* s, int n_fields, const int* fields, void* stream);

// ---- direct peer-memory exchange: setup -------------------------------------------------------------------------------
// 1. every rank: hns_dist_ipc_prepare -> its block's IPC handle + the offset of each peer's region inside it
// 2. the caller all-gathers (handle, offsets);  3. per peer: hns_dist_ipc_connect(handle of that peer, offset of MY region in ITS block)
// 4. hns_dist_ipc_finish switches the exchanges from NCCL send/recv to peer stores + flags
int hns_dist_ipc_prepare(hns_dist* d, uint8_t* handle_out64, uint64_t* region_offsets_out) {
	if (!d || !handle_out64 || (!region_offsets_out && !d->peers.empty()) || !d->bound_state) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
	uint64_t total = 256;
	for (size_t i = 0; i < d->peers.size(); ++i) {
		d->peers[i].region_off = total;
		region_offsets_out[i] = total;
		total += region_bytes(d->peers[i].n_recv, d->n_scalars);
	}
	cudaFree(d->block);
	d->block = nullptr;
	HNS_CUDA(cudaMalloc(&d->block, total));
	HNS_CUDA(cudaMemset(d->block, 0, total));
	d->block_bytes = total;
	cudaIpcMemHandle_t h;
	HNS_CUDA(cudaIpcGetMemHandle(&h, d->block));
	std::memcpy(handle_out64, &h, 64);
	// bytes 64..127: the pressure allocation (peers store swept ghost values straight into it); 128..143: byte offsets of the red and
	// black halves inside it; the rest of the 192 bytes is reserved
	HNS_CUDA(cudaIpcGetMemHandle(&h, d->bound_state->p[0]));
	std::memcpy(handle_out64 + 64, &h, 64);
	std::memset(handle_out64 + 128, 0, 64);
	const uint64_t off[2] = {0, uint64_t(reinterpret_cast<const uint8_t*>(d->bound_state->p[1]) - reinterpret_cast<const uint8_t*>(d->bound_state->p[0]))};
	std::memcpy(handle_out64 + 128, off, sizeof(off));
	return HNS_OK;
}
int hns_dist_ipc_connect(hns_dist* d, int peer_index, const uint8_t* peer_handles192, uint64_t my_region_offset_in_peer_block,
                         const int32_t* peer_leaf_ids) {
	if (!d || peer_index < 0 || peer_index >= int(d->peers.size()) || !peer_handles192) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	auto& p = d->peers[peer_index];
	if (p.n_send && !peer_leaf_ids) return fail(HNS_ERR_INVALID_ARGUMENT, "peer_leaf_ids is null");
	cudaIpcMemHandle_t h;
	std::memcpy(&h, peer_handles192, 64);
	if (p.ipc_base) cudaIpcCloseMemHandle(p.ipc_base), p.ipc_base = nullptr;
	HNS_CUDA(cudaIpcOpenMemHandle(&p.ipc_base, h, cudaIpcMemLazyEnablePeerAccess));
	p.remote_region = static_cast<uint8_t*>(p.ipc_base) + my_region_offset_in_peer_block;
	std::memcpy(&h, peer_handles192 + 64, 64);
	if (p.ipc_pbase) cudaIpcCloseMemHandle(p.ipc_pbase), p.ipc_pbase = nullptr;
	HNS_CUDA(cudaIpcOpenMemHandle(&p.ipc_pbase, h, cudaIpcMemLazyEnablePeerAccess));
	uint64_t off[2];
	std::memcpy(off, peer_handles192 + 128, sizeof(off));
	for (int c = 0; c < 2; ++c) p.ipc_p[c] = static_cast<uint8_t*>(p.ipc_pbase) + off[c];
	p.peer_leaf.assign(peer_leaf_ids, peer_leaf_ids + p.n_send);
	return HNS_OK;
}
int hns_dist_ipc_finish(hns_dist* d) {
	if (!d || !d->block) return fail(HNS_ERR_INVALID_ARGUMENT, "hns_dist_ipc_prepare has not been called");
	const size_t n = d->peers.size();
	std::vector<uint32_t*> rem(std::max<size_t>(n, 1), nullptr), loc(std::max<size_t>(n, 1), nullptr);
	for (size_t i = 0; i < n; ++i) {
		if (!d->peers[i].remote_region) return fail(HNS_ERR_RUNTIME, "peer " + std::to_string(d->peers[i].rank) + " is not connected");
		// Every exchange is a handshake with every peer, also with one this rank only sends to or only receives from: a region is
		// written again only after a later flag of the rank that unpacks it, so a rank that only sends cannot run a frame ahead and
		// overwrite ghost bricks its receivers have not unpacked yet (a region without bricks still has its flag words).
		rem[i] = reinterpret_cast<uint32_t*>(d->peers[i].remote_region);
		loc[i] = reinterpret_cast<uint32_t*>(d->block + d->peers[i].region_off);
	}
	if (n > 32) return fail(HNS_ERR_UNSUPPORTED, "more than 32 peers");
	cudaFree(d->d_remote_flags), cudaFree(d->d_local_flags);
	HNS_CUDA(cudaMalloc(&d->d_remote_flags, rem.size() * sizeof(uint32_t*)));
	HNS_CUDA(cudaMalloc(&d->d_local_flags, loc.size() * sizeof(uint32_t*)));
	HNS_CUDA(cudaMemcpy(d->d_remote_flags, rem.data(), rem.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice));
	HNS_CUDA(cudaMemcpy(d->d_local_flags, loc.data(), loc.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice));
	{
		// CSR over the boundary work list: which peers hold a ghost copy of boundary leaf i, under which leaf id, and which of its
		// faces touch leaves that peer owns. The 7-point stencil (sweeps, gradient) only ever reads the face layer of a ghost leaf, so
		// only those rows are pushed: the 8 rows of an x or y face (128 B per colour), every row for a z face (one float of each
		// quad); a leaf that touches the peer's leaves only across an edge or a corner is not pushed at all.
		const hns_grid* grid = d->bound_state->grid;
		const uint64_t L = grid->num_leaves;
		std::vector<int32_t> nbr(L * 27);
		if (L) HNS_CUDA(cudaMemcpy(nbr.data(), grid->d_nbr, nbr.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
		std::vector<int32_t> owner(L, -1);  // peer index owning a ghost leaf, -1 = this rank
		std::vector<int32_t> host_ids;
		for (size_t i = 0; i < n; ++i) {
			const auto& p = d->peers[i];
			host_ids.resize(p.n_recv);
			if (p.n_recv) HNS_CUDA(cudaMemcpy(host_ids.data(), p.d_recv, p.n_recv * sizeof(int32_t), cudaMemcpyDeviceToHost));
			for (int32_t id : host_ids) owner[id] = int32_t(i);
		}
		static const int face_slot[6] = {kSlotXm, kSlotXp, kSlotYm, kSlotYp, kSlotZm, kSlotZp};
		std::vector<std::vector<std::pair<int32_t, int32_t>>> per_leaf(L);
		uint64_t quads = 0;
		for (size_t i = 0; i < n; ++i) {
			const auto& p = d->peers[i];
			host_ids.resize(p.n_send);
			if (p.n_send) HNS_CUDA(cudaMemcpy(host_ids.data(), p.d_send, p.n_send * sizeof(int32_t), cudaMemcpyDeviceToHost));
			for (uint64_t k = 0; k < p.n_send; ++k) {
				const int32_t leaf = host_ids[k];
				int mask = 0;
				for (int f = 0; f < 6; ++f) {
					const int32_t nb = nbr[uint64_t(leaf) * 27 + face_slot[f]];
					if (nb >= 0 && owner[nb] == int32_t(i)) mask |= 1 << f;
				}
				if (!mask) continue;
				per_leaf[leaf].push_back({int32_t(i) | (mask << 8), p.peer_leaf[k]});
				int rows = 64;
				if (!(mask & 0x30)) {
					rows = 0;
					for (int x = 0; x < 8; ++x)
						for (int y = 0; y < 8; ++y) rows += ((mask & 1) && x == 0) || ((mask & 2) && x == 7) || ((mask & 4) && y == 0) || ((mask & 8) && y == 7);
				}
				quads += rows;
			}
		}
		d->push_bytes_per_sweep = quads * 16;
		std::vector<uint32_t> off(d->h_boundary.size() + 1, 0);
		std::vector<int32_t> peer, leaf;
		for (size_t b = 0; b < d->h_boundary.size(); ++b) {
			for (const auto& e : per_leaf[d->h_boundary[b]]) peer.push_back(e.first), leaf.push_back(e.second);
			off[b + 1] = uint32_t(peer.size());
		}
		cudaFree(d->d_push_off), cudaFree(d->d_push_peer), cudaFree(d->d_push_leaf);
		HNS_CUDA(cudaMalloc(&d->d_push_off, off.size() * sizeof(uint32_t)));
		HNS_CUDA(cudaMemcpy(d->d_push_off, off.data(), off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
		HNS_CUDA(cudaMalloc(&d->d_push_peer, std::max<size_t>(peer.size(), 1) * sizeof(int32_t)));
		HNS_CUDA(cudaMalloc(&d->d_push_leaf, std::max<size_t>(leaf.size(), 1) * sizeof(int32_t)));
		if (!peer.empty()) {
			HNS_CUDA(cudaMemcpy(d->d_push_peer, peer.data(), peer.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
			HNS_CUDA(cudaMemcpy(d->d_push_leaf, leaf.data(), leaf.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
		}
		for (int c = 0; c < 2; ++c) {
			std::vector<float*> rp(std::max<size_t>(n, 1), nullptr);
			for (size_t i = 0; i < n; ++i) rp[i] = static_cast<float*>(d->peers[i].ipc_p[c]);
			cudaFree(d->d_remote_p[c]);
			HNS_CUDA(cudaMalloc(&d->d_remote_p[c], rp.size() * sizeof(float*)));
			HNS_CUDA(cudaMemcpy(d->d_remote_p[c], rp.data(), rp.size() * sizeof(float*), cudaMemcpyHostToDevice));
		}
	}
	d->p2p = true;
	return HNS_OK;
}
// 0 = clean; low byte: 1 + the channel of a flag wait that timed out; bit 8: a semi-Lagrangian sample landed beyond the ghost layer
// (the leaf may exist on another rank, so the sharded result would differ from the single-GPU one). Sticky until _reset_error.
int hns_dist_error(hns_dist* d, uint32_t* out) {
	if (!d || !out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	*out = 0;
	if (d->d_err) HNS_CUDA(cudaMemcpy(out, d->d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost));
	return HNS_OK;
}
int hns_dist_reset_error(hns_dist* d) {
	if (!d) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	if (d->d_err) HNS_CUDA(cudaMemset(d->d_err, 0, sizeof(uint32_t)));
	return HNS_OK;
}
// after a stream sync: turn a recorded device-side error into a status
static int check_device_error(hns_dist* d) {
	uint32_t e = 0;
	if (d->d_err) HNS_CUDA(cudaMemcpy(&e, d->d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost));
	if ((e & 0xffu) == 1u + kChMgGather) return fail(HNS_ERR_RUNTIME, "the multigrid level-1 gather timed out waiting for a rank: the frame ran on a stale coarse right-hand side");
	if (e & 0xffu) return fail(HNS_ERR_RUNTIME, "ghost exchange timed out waiting for a peer on channel " + std::to_string((e & 0xffu) - 1) + ": the frame ran on stale ghosts");
	if (e & 0x100u)
		return fail(HNS_ERR_RUNTIME, "a semi-Lagrangian sample landed beyond the one-leaf ghost layer of this shard (CFL too large for a sharded run): the result may differ from the single-GPU frame");
	return HNS_OK;
}

// Ghost exchange through peer memory: every owned boundary brick is stored straight into the peer's landing region over NVLink
// (the pack kernel with a remote destination), the channel flag is raised, the peers' flags are awaited, the landed bricks are
// scattered into the ghost leaves. Four small launches, no library call, NVLink bandwidth instead of NCCL's p2p channel bandwidth.
// `channel` selects the arrival flag; the bricks land in region `region_ch` starting `skip_fields` whole fields in, so two exchanges
// with different flags can share one region (velocity and scalars of channel 4).
static int exchange_p2p(hns_dist* d, hns_state* s, int channel, int n_fields, const int* fields, cudaStream_t st, int region_ch = -1,
                        int skip_fields = 0, int max_blocks = 0) {
	const int S = d->n_scalars;
	if (region_ch < 0) region_ch = channel;
	for (auto& p : d->peers) {
		if (!p.n_send) continue;
		float* dst = reinterpret_cast<float*>(p.remote_region + channel_offset(region_ch, p.n_send, S)) + uint64_t(skip_fields) * 512u * p.n_send;
		for (int k = 0; k < n_fields; ++k) {
			int fpl;
			const float* f = field_ptr(s, fields[k], &fpl);
			if (!f) return fail(HNS_ERR_INVALID_ARGUMENT, "bad field id");
			launch_pack_leaves(f, p.d_send, p.n_send, dst, fpl, st, max_blocks);
			dst += p.n_send * fpl;
			d->bytes_sent += p.n_send * fpl * 4;
		}
	}
	const uint32_t seq = ++d->seq[channel];
	const int np = int(d->peers.size());
	HNS_LAUNCH(k_signal, 1, 32, 0, st, d->d_remote_flags, np, channel, seq);
	HNS_LAUNCH(k_wait, 1, 32, 0, st, d->d_local_flags, np, channel, seq, d->d_err);
	for (auto& p : d->peers) {
		if (!p.n_recv) continue;
		const float* src = reinterpret_cast<const float*>(d->block + p.region_off + channel_offset(region_ch, p.n_recv, S)) + uint64_t(skip_fields) * 512u * p.n_recv;
		for (int k = 0; k < n_fields; ++k) {
			int fpl;
			float* f = field_ptr(s, fields[k], &fpl);
			field_written(s, fields[k]);
			launch_unpack_leaves(f, p.d_recv, p.n_recv, src, fpl, st, max_blocks);
			src += p.n_recv * fpl;
		}
	}
	++d->exchanges;
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}
static int exchange_channel(hns_dist* d, hns_state* s, int channel, int n_fields, const int* fields, cudaStream_t st) {
	return d->p2p ? exchange_p2p(d, s, channel, n_fields, fields, st) : hns_dist_exchange(d, s, n_fields, fields, st);
}

// pack -> grouped send/recv -> unpack of the given fields' ghost bricks, all on `stream`
int hns_dist_exchange(hns_dist* d, hns_state* s, int n_fields, const int* fields, void* stream) {
	if (!d || !s || n_fields <= 0 || n_fields > d->max_fields) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	if (!d->comm && d->world > 1) return fail(HNS_ERR_RUNTIME, "no NCCL communicator (hns_dist_create without an id) and the peer-memory exchange is not connected");
	if (d->peers.empty()) return HNS_OK;  // a single rank (or one that shares no leaf): nothing to send or receive
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	float* f[3 + 16];  // n_fields <= max_fields = 3 + n_scalars
	int fpl[3 + 16];
	uint64_t leaf_floats = 0;  // of all the fields
	for (int k = 0; k < n_fields; ++k) {
		if (!(f[k] = field_ptr(s, fields[k], &fpl[k]))) return fail(HNS_ERR_INVALID_ARGUMENT, "bad field id");
		leaf_floats += fpl[k];
	}
	for (auto& p : d->peers) {
		uint64_t off = 0;
		for (int k = 0; k < n_fields && p.n_send; ++k) {
			launch_pack_leaves(f[k], p.d_send, p.n_send, p.buf_send + off, fpl[k], st);
			off += p.n_send * fpl[k];
		}
	}
	HNS_NCCL(g_nccl.GroupStart());
	for (auto& p : d->peers) {
		const uint64_t cs = p.n_send * leaf_floats, cr = p.n_recv * leaf_floats;
		if (cs) HNS_NCCL(g_nccl.Send(p.buf_send, cs, ncclFloat, p.rank, d->comm, st));
		if (cr) HNS_NCCL(g_nccl.Recv(p.buf_recv, cr, ncclFloat, p.rank, d->comm, st));
		d->bytes_sent += cs * 4;
	}
	HNS_NCCL(g_nccl.GroupEnd());
	for (auto& p : d->peers) {
		uint64_t off = 0;
		for (int k = 0; k < n_fields && p.n_recv; ++k) {
			field_written(s, fields[k]);
			launch_unpack_leaves(f[k], p.d_recv, p.n_recv, p.buf_recv + off, fpl[k], st);
			off += p.n_recv * fpl[k];
		}
	}
	++d->exchanges;
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

// The sharded frame: Compute()'s step order (reference src/Cuda/HNanoSolver.cu:159-356) with a ghost exchange in front of every step
// that reads a neighbour leaf. Asynchronous on `stream`.
// optional stream dependencies of a frame whose inputs arrive / outputs leave on a copy stream while it runs (hns_dist_cook): waited for
// before the combustion stage / before the scalars are first read by a ghost exchange; recorded once the projected velocity (ghosts
// included) is final and converted to the host layout
struct DistDeps {
	cudaEvent_t combustion_inputs = nullptr, scalar_inputs = nullptr, velocity_done = nullptr;
};
static int dist_frame(hns_dist* d, hns_state* s, int iterations, float dt, void* stream, cudaEvent_t* marks, const DistDeps* deps = nullptr);

int hns_dist_frame(hns_dist* d, hns_state* s, int iterations, float dt, void* stream) { return dist_frame(d, s, iterations, dt, stream, nullptr); }

// The sharded cook on HOST arrays of this rank's local voxels (owned + ghost leaves, local sidecar order), in place and synchronous:
// the per-rank equivalent of hns_compute_sim. Every rank moves its own shard over its own PCIe link, so the transfers of the N ranks
// run in parallel; ghost entries of the inputs need not be valid (every field's ghosts are exchanged before they are read) and ghost
// entries of the outputs are whatever the last exchange left there.
int hns_dist_cook(hns_dist* d, hns_state* s, float* velocity, int n_float, float* const* fields, int iterations, float dt, void* stream) {
	if (!d || !s || !velocity || n_float != s->n_scalars || (n_float && !fields)) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	const uint64_t n = s->n;
	if (!n) return HNS_OK;
	for (int i = 0; i < n_float; ++i)
		if (!fields[i]) return fail(HNS_ERR_INVALID_ARGUMENT, "null field pointer");
	if (!s->aos) HNS_CUDA(cudaMalloc(&s->aos, n * 3 * sizeof(float)));
	if (!d->copy_stream) {
		HNS_CUDA(cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking));
		for (auto& e : d->ev_copy) HNS_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
	}
	// Like hns_compute_sim (api.cu): the shard crosses PCIe on a copy stream while the kernels run. Velocity (and the collision SDF) first
	// -- advect_vector and the divergence start as soon as they have landed --, the four combustion inputs next, the remaining scalars
	// behind them (they are needed by the scalars' ghost exchange behind the pressure solve); the projected velocity goes back while
	// advect_scalars runs, the scalars when it is done.
	cudaStream_t cs = d->copy_stream;
	cudaEvent_t e_start = d->ev_copy[0], e_vel_in = d->ev_copy[1], e_comb_in = d->ev_copy[2], e_all_in = d->ev_copy[3], e_vel_out = d->ev_copy[4],
	            e_done = d->ev_copy[5];
	HNS_CUDA(cudaEventRecord(e_start, st));
	HNS_CUDA(cudaStreamWaitEvent(cs, e_start, 0));
	HNS_CUDA(cudaMemcpyAsync(s->aos, velocity, n * 12, cudaMemcpyHostToDevice, cs));
	const bool coll = hns_state_collision_active(s);
	if (coll) HNS_CUDA(cudaMemcpyAsync(s->sc[s->skip_scalar], fields[s->skip_scalar], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_vel_in, cs));
	auto is_comb = [&](int i) { return s->comb_enabled && (i == s->comb_idx[0] || i == s->comb_idx[1] || i == s->comb_idx[2] || i == s->comb_idx[3]); };
	for (int i = 0; i < n_float; ++i)
		if (is_comb(i)) HNS_CUDA(cudaMemcpyAsync(s->sc[i], fields[i], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_comb_in, cs));
	for (int i = 0; i < n_float; ++i)
		if (!is_comb(i) && !(coll && i == s->skip_scalar)) HNS_CUDA(cudaMemcpyAsync(s->sc[i], fields[i], n * 4, cudaMemcpyHostToDevice, cs));
	HNS_CUDA(cudaEventRecord(e_all_in, cs));
	HNS_CUDA(cudaStreamWaitEvent(st, e_vel_in, 0));
	launch_aos_to_soa(s->aos, s->vel[0], s->vel[1], s->vel[2], n, st);
	++s->vel_version, ++s->sc_version;
	DistDeps deps;
	deps.combustion_inputs = e_comb_in, deps.scalar_inputs = e_all_in, deps.velocity_done = e_vel_out;
	int rc = dist_frame(d, s, iterations, dt, stream, nullptr, &deps);
	if (rc) return rc;
	HNS_CUDA(cudaStreamWaitEvent(cs, e_vel_out, 0));
	HNS_CUDA(cudaMemcpyAsync(velocity, s->aos, n * 12, cudaMemcpyDeviceToHost, cs));
	HNS_CUDA(cudaEventRecord(e_done, st));
	HNS_CUDA(cudaStreamWaitEvent(cs, e_done, 0));
	for (int i = 0; i < n_float; ++i) HNS_CUDA(cudaMemcpyAsync(fields[i], s->sc[i], n * 4, cudaMemcpyDeviceToHost, cs));
	HNS_CUDA(cudaStreamSynchronize(cs));
	HNS_CUDA(cudaStreamSynchronize(st));
	HNS_CUDA(cudaGetLastError());
	return check_device_error(d);
}

// Same frame with CUDA events between the phases; ms_out[8] = exchange velocity, advect_vector, exchange advected, divergence(+combustion),
// pressure solve incl. its exchanges, gradient, final exchange, advect_scalars. Synchronises the stream.
int hns_dist_frame_timed(hns_dist* d, hns_state* s, int iterations, float dt, void* stream, float* ms_out) {
	if (!ms_out) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	cudaEvent_t ev[9];
	for (auto& e : ev) cudaEventCreate(&e);
	int rc = dist_frame(d, s, iterations, dt, stream, ev);
	cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
	if (rc == HNS_OK)
		for (int i = 0; i < 8; ++i) cudaEventElapsedTime(&ms_out[i], ev[i], ev[i + 1]);
	for (auto& e : ev) cudaEventDestroy(e);
	return rc ? rc : check_device_error(d);
}

// The pressure solve of the peer-memory mode: interior sweeps on `st`, boundary sweeps (which store every swept quad into the peers'
// ghost copies) + flag signal / wait on the comm stream.
// (Replaying this pipeline as a CUDA graph -- two captured streams, which is why the sequence numbers live in device memory -- was
// measured at 2 GPUs: 8.75 ms per frame against 8.54 ms launched directly; the graph's two branches do not overlap the way the
// high-priority comm stream does. Removed; profiles/r2d_tune2_dist_graph.txt.)
static int fused_pressure(hns_dist* d, hns_state* s, int iterations, float omega, cudaStream_t st) {
	GridView vb = s->grid->view, vi = s->grid->view;
	vb.list = d->d_boundary, vb.num_list = d->n_boundary, vb.list_nbr = d->d_boundary_nbr;
	vi.list = d->d_interior, vi.num_list = d->n_interior, vi.list_nbr = d->d_interior_nbr;
	const float dx = s->grid->voxel_size;
	const int np = int(d->peers.size());
	const uint32_t* base = d->d_seq_base;
	cudaStream_t bs = d->comm_stream;
	// "my pressure arrays are zeroed and nobody reads last frame's ghosts any more": peers may start pushing into them
	HNS_LAUNCH(k_signal_rel, 1, 32, 0, st, d->d_remote_flags, np, 5, base + 2, 1u);
	HNS_CUDA(cudaEventRecord(d->ev_I[1], st));  // "I_0": everything before the solve
	int k = 0;
	for (int it = 0; it < iterations; ++it)
		for (int color = 0; color < 2; ++color, ++k) {
			const int cur = k & 1, prev = cur ^ 1;
			HNS_CUDA(cudaStreamWaitEvent(bs, d->ev_I[prev], 0));
			// ghosts of the colour this sweep reads: pushed by the peers' previous boundary sweep (first sweep: their "zeroed" signal).
			// Red sweep of iteration `it` reads black pushes up to number `it`; black reads red pushes up to `it + 1`.
			if (k == 0) HNS_LAUNCH(k_wait_rel, 1, 32, 0, bs, d->d_local_flags, np, 5, base + 2, 1u, d->d_err);
			else HNS_LAUNCH(k_wait_rel, 1, 32, 0, bs, d->d_local_flags, np, 2 + (color ^ 1), base + (color ^ 1), uint32_t(it + color), d->d_err);
			RbgsPush push;
			push.dst_off = d->d_push_off, push.dst_peer = d->d_push_peer, push.dst_leaf = d->d_push_leaf, push.remote_pc = d->d_remote_p[color];
			launch_rbgs_color_push(vb, s->div, s->p, dx, color, omega, color, push, bs);
			HNS_LAUNCH(k_signal_rel, 1, 32, 0, bs, d->d_remote_flags, np, 2 + color, base + color, uint32_t(it) + 1u);
			HNS_CUDA(cudaEventRecord(d->ev_B[cur], bs));
			if (k > 0) HNS_CUDA(cudaStreamWaitEvent(st, d->ev_B[prev], 0));
			if (d->n_interior) launch_rbgs_color(vi, s->div, s->p, dx, color, omega, color, st);
			HNS_CUDA(cudaEventRecord(d->ev_I[cur], st));
		}
	HNS_LAUNCH(k_wait_rel, 1, 32, 0, bs, d->d_local_flags, np, 3, base + 1, uint32_t(iterations), d->d_err);  // the peers' last black push
	HNS_CUDA(cudaEventRecord(d->ev_exchanged, bs));
	HNS_CUDA(cudaStreamWaitEvent(st, d->ev_exchanged, 0));
	HNS_LAUNCH(k_advance_bases, 1, 32, 0, st, d->d_seq_base, uint32_t(iterations));
	d->bytes_sent += d->push_bytes_per_sweep * 2u * uint64_t(iterations);
	d->exchanges += 2u * uint64_t(iterations);
	return HNS_OK;
}

// `iterations` red-black iterations on the owned leaves with the ghost exchange of each swept colour, in two software-pipelined streams.
// Interior leaves (no ghost neighbour) are swept on the caller's stream, boundary leaves and the exchange of their freshly swept colour
// on comm_stream:
//   caller's stream:  I_1        I_2        I_3   ...      I_k needs I_{k-1} (in order) and B_{k-1} (event)
//   comm_stream:      B_1 x_1    B_2 x_2    B_3 x_3 ...    B_k needs B_{k-1}, x_{k-1} (in order) and I_{k-1} (event)
// Half-sweep k reads colour c_{k-1} and writes colour c_k, so I_k and B_k/x_k never touch the same colour of the same leaf at the same
// time, and the exchange latency disappears behind the interior sweep as long as B + x is the shorter chain. On return the caller's
// stream has joined the exchanges: the ghosts of both colours are current. mg_flags: the multigrid solve's flag channels (peer memory).
// The red-black solve of the NCCL fallback and of a rank without boundary leaves, and the smoother of the sharded multigrid solve.
static int pipelined_sweeps(hns_dist* d, hns_state* s, int iterations, float omega, bool mg_flags, cudaStream_t st) {
	GridView vb = s->grid->view, vi = s->grid->view;
	vb.list = d->d_boundary, vb.num_list = d->n_boundary, vb.list_nbr = d->d_boundary_nbr;
	vi.list = d->d_interior, vi.num_list = d->n_interior, vi.list_nbr = d->d_interior_nbr;
	const float dx = s->grid->voxel_size;
	const int fred[1] = {6}, fblk[1] = {7};
	cudaStream_t bs = d->comm_stream;
	int rc;
	HNS_CUDA(cudaEventRecord(d->ev_I[1], st));  // "I_0": everything before the solve
	HNS_CUDA(cudaEventRecord(d->ev_B[1], bs));  // "B_0": nothing
	int k = 0;
	for (int it = 0; it < iterations; ++it)
		for (int color = 0; color < 2; ++color, ++k) {
			const int cur = k & 1, prev = cur ^ 1;
			HNS_CUDA(cudaStreamWaitEvent(bs, d->ev_I[prev], 0));
			if (d->n_boundary) launch_rbgs_color(vb, s->div, s->p, dx, color, omega, color, bs);
			HNS_CUDA(cudaEventRecord(d->ev_B[cur], bs));
			HNS_CUDA(cudaStreamWaitEvent(st, d->ev_B[prev], 0));
			if (d->n_interior) launch_rbgs_color(vi, s->div, s->p, dx, color, omega, color, st);
			HNS_CUDA(cudaEventRecord(d->ev_I[cur], st));
			if (!mg_flags) rc = exchange_channel(d, s, 2 + color, 1, color ? fblk : fred, bs);
			else rc = d->peers.empty() ? HNS_OK : exchange_p2p(d, s, kChMgPressure + color, 1, color ? fblk : fred, bs, 2 + color, 0);
			if (rc) return rc;
		}
	HNS_CUDA(cudaEventRecord(d->ev_exchanged, bs));
	HNS_CUDA(cudaStreamWaitEvent(st, d->ev_exchanged, 0));
	return HNS_OK;
}

// The multigrid solve of a sharded frame: `cycles` V(nu_pre, nu_post) cycles whose level 0 is this rank's shard and whose levels >= 1 are
// replicated. Every kernel sees the inputs it sees in the single-GPU v_cycle (multigrid.cu), so the owned voxels come out bit for bit
// the same:
//   1. pre-smoothing: pipelined_sweeps, ghosts of both colours current afterwards;
//   2. residual + restriction over the owned leaves, stored straight into every rank's level-1 rhs (k_mg_residual<..., kGather>). A
//      level-1 cell is 2x2x2 fine voxels of ONE fine leaf, and every fine leaf has one owner, so the ranks write disjoint octants whose
//      union is the single-GPU level-1 rhs; octants without a fine leaf stay 0 from the allocation on (so nothing clears the array);
//   3. signal "gather c done" to every rank, wait for every rank's;
//   4. levels 1 .. n-1 locally (mg_coarse_cycle, a CUDA graph per parity);
//   5. prolongation over the owned leaves (it reads only level-1 corrections, which every rank has computed identically);
//   6. exchange of both pressure colours: the prolongation changed the owned leaves' values the peers hold as ghosts (the next red sweep
//      reads black ghosts; with nu_post = 0 the next residual, or the gradient pass, reads both);
//   7. post-smoothing: pipelined_sweeps.
// Ordering of the gather (c = the global gather number, which continues across frames). The level-1 rhs is double-buffered by the
// parity of c. Rank A stores gather c + 2 into rank B's buffer c & 1 only after A has waited for every rank's flag c + 1 (A's wait of
// cycle c + 1 precedes its coarse solve of c + 1, which precedes its restriction of c + 2, all on one stream). B raises flag c + 1 from
// its stream after its restriction of c + 1, which follows its coarse solve of cycle c -- the last reader of buffer c & 1. So no store
// into a buffer can overtake the coarse solve still reading it, also between two ranks that share no ghost leaf and are otherwise not
// held back by each other's sweeps. The flag a rank waits for in cycle c is raised after the stores of cycle c (k_signal fences them).
// The pressure exchanges of steps 1, 6, 7 alternate red, black, red, ... on flag channels 8 / 9, so a landing region is reused only
// after the peer has signalled the other colour, which it does after unpacking the previous use (as in the red-black solve).
static int sharded_mg_pressure(hns_dist* d, hns_state* s, cudaStream_t st) {
	auto& m = d->smg;
	if (!m.ready) return fail(HNS_ERR_RUNTIME, "the sharded multigrid solver is set but not connected (hns_dist_mg_connect, hns_dist_mg_finish)");
	hns_mg* mg = m.mg;
	const int n = int(mg->lv.size());
	const GridView g = s->view();
	const float dx = s->grid->voxel_size;
	const int np = d->world - 1;
	const int fp[2] = {6, 7};
	int rc;
	for (int c = 0; c < m.cycles; ++c) {
		if (n == 1) {  // a one-level hierarchy: plain red-black sweeps, like v_cycle
			if ((rc = pipelined_sweeps(d, s, m.nu_pre + m.nu_post, m.omega, true, st))) return rc;
			continue;
		}
		if ((rc = pipelined_sweeps(d, s, m.nu_pre, m.omega, true, st))) return rc;
		const uint32_t seq = ++m.seq;
		const int par = int(seq & 1u);
		launch_mg_restrict_gather(g, s->p, s->div, dx, m.d_parent, m.d_gather[par], d->world, st);
		if (np > 0) {
			HNS_LAUNCH(k_signal, 1, 32, 0, st, m.d_sig, np, kChMgGather, seq);
			HNS_LAUNCH(k_wait, 1, 32, 0, st, m.d_wait, np, kChMgGather, seq, d->d_err);
		}
		float* const base = reinterpret_cast<float*>(m.block + m.flag_bytes) + uint64_t(par) * m.rhs_floats;
		float* const rhs1[2] = {base, base + m.rhs_floats / 2};
		if (mg->use_graph) {
			cudaGraphExec_t& G = m.graph[par];
			if (G && m.graph_coarsest[par] != mg->coarsest_iterations) cudaGraphExecDestroy(G), G = nullptr;
			if (!G) G = mg_capture_coarse(mg, rhs1, m.nu_pre, m.nu_post, m.omega, &m.graph_launches[par]), m.graph_coarsest[par] = mg->coarsest_iterations;
			if (G) {
				HNS_CUDA(cudaGraphLaunch(G, st));
				g_launches.fetch_add(m.graph_launches[par], std::memory_order_relaxed);
			} else {
				mg_coarse_cycle(mg, rhs1, m.nu_pre, m.nu_post, m.omega, st);
			}
		} else {
			mg_coarse_cycle(mg, rhs1, m.nu_pre, m.nu_post, m.omega, st);
		}
		launch_mg_prolong(g, s->p, nullptr, m.d_parent, mg->lv[1].grid->view, mg->lv[1].p, st);
		for (int color = 0; color < 2 && !d->peers.empty(); ++color)
			if ((rc = exchange_p2p(d, s, kChMgPressure + color, 1, fp + color, st, 2 + color, 0))) return rc;
		if ((rc = pipelined_sweeps(d, s, m.nu_post, m.omega, true, st))) return rc;
		++m.gathers;
		m.gather_bytes += uint64_t(d->n_owned) * 256u * uint64_t(np);
	}
	HNS_CUDA(cudaGetLastError());
	return HNS_OK;
}

static int dist_frame(hns_dist* d, hns_state* s, int iterations, float dt, void* stream, cudaEvent_t* marks, const DistDeps* deps) {
	if (!d || !s || iterations <= 0 || dt < 0.f) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	int rc;
	int mark_i = 0;
	auto mark = [&]() {
		if (marks) cudaEventRecord(marks[mark_i++], static_cast<cudaStream_t>(stream));
	};
	mark();
	const int fvel[3] = {0, 1, 2}, fadv[3] = {3, 4, 5};
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	if (s->skip_scalar >= 0 && s->skip_scalar != s->n_scalars - 1)
		return fail(HNS_ERR_UNSUPPORTED, "sharded frames need the non-advected scalar (collision_sdf) to be the last scalar field");
	// collision path: enforceCollisionBoundaries and the collision tests of advect_vector read the SDF in ghost leaves (neighbour rows
	// of the normal, trilinear samples at the traced positions), so its ghosts are exchanged first -- the caller's ghost entries need
	// not be valid (hns_dist_cook's contract). The landing region is the |curl| one (flag 7), free at this point of a frame.
	// enforceCollisionBoundaries is per voxel on the owned leaves (it bumps the velocity version, so the velocity ghosts below are
	// exchanged, never reused).
	if (hns_state_collision_active(s)) {
		const int fsdf[1] = {10 + s->skip_scalar};
		if (d->p2p) {
			if ((rc = exchange_p2p(d, s, 7, 1, fsdf, st, 5, 0))) return rc;
		} else if ((rc = hns_dist_exchange(d, s, 1, fsdf, st))) {
			return rc;
		}
		if ((rc = hns_state_enforce_collision(s, stream))) return rc;
	}
	// the velocity ghosts are still current when the last thing that wrote the velocity was the previous sharded frame (its final
	// exchange refreshed them and advect_scalars does not touch the velocity)
	if (d->vel_exchanged_version != s->vel_version && (rc = exchange_channel(d, s, 0, 3, fvel, st))) return rc;
	mark();
	if ((rc = hns_state_advect_velocity(s, dt, stream))) return rc;
	mark();
	if ((rc = exchange_channel(d, s, 1, 3, fadv, st))) return rc;
	if (hns_state_vorticity_active(s)) {
		// vorticity confinement reads the advected velocity 1 + |offset| voxels away: |curl| of the owned leaves, its ghost leaves from
		// the peers, the force on the owned leaves, and the advected velocity's ghosts once more because it has changed
		const int off = int(s->comb.factorScale);
		if (off > 7 || off < -7)
			return fail(HNS_ERR_UNSUPPORTED, "sharded vorticity confinement needs |(int)factorScale| <= 7 (one ghost leaf layer)");
		const int fmag[1] = {26};
		if ((rc = hns_state_vorticity_mag(s, stream))) return rc;
		if (d->p2p) {
			if ((rc = exchange_p2p(d, s, 7, 1, fmag, st, 5, 0))) return rc;
		} else if ((rc = hns_dist_exchange(d, s, 1, fmag, st))) {
			return rc;
		}
		if ((rc = hns_state_vorticity_force(s, dt, s->comb.vorticityScale, s->comb.factorScale, stream))) return rc;
		if ((rc = exchange_channel(d, s, 1, 3, fadv, st))) return rc;
	}
	mark();
	if ((rc = hns_state_divergence(s, 1, stream))) return rc;
	if (deps && deps->combustion_inputs) HNS_CUDA(cudaStreamWaitEvent(st, deps->combustion_inputs, 0));
	if (s->comb_enabled && (rc = hns_state_combustion_buoyancy(s, dt, stream))) return rc;
	// Packed advection groups (api.cu): the combustion pass has just written group 1 for every voxel, the gradient pass below writes
	// group 0 for the owned leaves; the exchanges that follow refresh the ghost leaves of the brick fields only (and bump the version
	// counters), so what is current now is noted here and the groups' ghost leaves are re-packed in front of advect_scalars.
	const float* want[2][4];
	bool packed[2];
	group_wants(s, 1, want[1]);
	packed[1] = group_if_current(s, 1, want[1]) != nullptr;
	if (deps && deps->scalar_inputs) HNS_CUDA(cudaStreamWaitEvent(st, deps->scalar_inputs, 0));
	// The scalars are final until advect_scalars: exchange their ghosts now, on a third stream, behind the pressure solve.
	const bool scalars_early = d->p2p && s->n_scalars > 0;
	if (scalars_early) {
		std::vector<int> fsc;
		for (int i = 0; i < s->n_scalars; ++i) fsc.push_back(10 + i);
		HNS_CUDA(cudaEventRecord(d->ev_scalars_final, st));
		HNS_CUDA(cudaStreamWaitEvent(d->aux_stream, d->ev_scalars_final, 0));
		if ((rc = exchange_p2p(d, s, 6, int(fsc.size()), fsc.data(), d->aux_stream, 4, 3, kAuxBlocks))) return rc;
		HNS_CUDA(cudaEventRecord(d->ev_scalars_exchanged, d->aux_stream));
	}
	mark();
	if ((rc = hns_state_pressure_init(s, stream))) return rc;
	if (d->smg.mg) {
		if ((rc = sharded_mg_pressure(d, s, st))) return rc;
	} else {
		const float omega = hns_omega_compute(s->grid->voxel_size);
		if (d->p2p && d->n_boundary > 0) {
			if ((rc = fused_pressure(d, s, iterations, omega, st))) return rc;
		} else {
			// a rank without boundary leaves: its fused peers wait for its "pressure zeroed" flag of this frame as for each other's
			if (d->p2p) HNS_LAUNCH(k_signal, 1, 32, 0, st, d->d_remote_flags, int(d->peers.size()), 5, ++d->seq[5]);
			if ((rc = pipelined_sweeps(d, s, iterations, omega, false, st))) return rc;
		}
	}
	mark();
	if ((rc = hns_state_subtract_gradient(s, 1, stream))) return rc;
	if (hns_state_collision_active(s) && (rc = hns_state_enforce_collision(s, stream))) return rc;  // HNanoSolver.cu:292-296
	group_wants(s, 0, want[0]);
	packed[0] = group_if_current(s, 0, want[0]) != nullptr;
	mark();
	std::vector<int> last = {0, 1, 2};
	if (!scalars_early)
		for (int i = 0; i < s->n_scalars; ++i) last.push_back(10 + i);
	if ((rc = exchange_channel(d, s, 4, int(last.size()), last.data(), st))) return rc;
	if (deps && deps->velocity_done) {
		launch_soa_to_aos(s->vel[0], s->vel[1], s->vel[2], s->aos, s->n, st);
		HNS_CUDA(cudaEventRecord(deps->velocity_done, st));
	}
	if (scalars_early) HNS_CUDA(cudaStreamWaitEvent(st, d->ev_scalars_exchanged, 0));
	for (auto& p : d->peers)
		for (int j = 0; j < 2; ++j)
			if (packed[j]) launch_pack4_leaves(p.d_recv, p.n_recv, want[j][0], want[j][1], want[j][2], want[j][3], s->grp[j].buf, st);
	for (int j = 0; j < 2; ++j)
		if (packed[j]) group_written(s, j, want[j]);
	// advect_scalars' "inactive -> element 0" value (reference Kernel.cu:192,225) is global voxel 0's = local voxel 0's: that exchange
	// has just refreshed it on every rank
	mark();
	rc = hns_state_advect_scalars(s, dt, 0, stream);
	d->vel_exchanged_version = s->vel_version;
	mark();
	return rc;
}

// ---- sharded multigrid solver: setup ------------------------------------------------------------------------------------------
// 1. every rank: hns_dist_set_pressure_solver -> the IPC handle of its block (flag words + the two level-1 rhs arrays)
// 2. the caller all-gathers the handles;  3. hns_dist_mg_connect for every other rank;  4. hns_dist_mg_finish
static void mg_release(hns_dist* d) {
	auto& m = d->smg;
	for (void*& p : m.ipc)
		if (p) cudaIpcCloseMemHandle(p), p = nullptr;
	for (auto& g : m.graph)
		if (g) cudaGraphExecDestroy(g), g = nullptr;
	cudaFree(m.d_parent), cudaFree(m.block), cudaFree(m.d_gather[0]), cudaFree(m.d_gather[1]), cudaFree(m.d_sig), cudaFree(m.d_wait);
	const uint64_t gathers = m.gathers, bytes = m.gather_bytes;
	m = hns_dist::ShardedMg{};
	m.gathers = gathers, m.gather_bytes = bytes;  // counters of the run, not of one set-up
}

int hns_dist_set_pressure_solver(hns_dist* d, hns_state* s, hns_mg* mg, const int32_t* local_to_global, int cycles, int nu_pre, int nu_post,
                                 float omega_smooth, uint8_t* handle_out64) {
	if (!d || !s) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	if (s != d->bound_state) return fail(HNS_ERR_INVALID_ARGUMENT, "the state is not the one hns_dist_set_plan was given");
	HNS_CUDA(cudaDeviceSynchronize());  // a frame in flight may still use what is released here
	mg_release(d);
	if (!mg) return HNS_OK;  // back to the red-black solve
	if (cycles <= 0 || nu_pre < 0 || nu_post < 0 || nu_pre + nu_post == 0)
		return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument: cycles must be > 0, nu_pre and nu_post >= 0 and not both 0");
	if (!(omega_smooth > 0.f && omega_smooth < 2.f)) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument: omega_smooth must lie in (0, 2)");
	if (d->world > 1 && !d->p2p)
		return fail(HNS_ERR_UNSUPPORTED, "the sharded multigrid solve gathers the level-1 right-hand side through peer memory: connect the "
		                                 "peer-memory exchange (hns_dist_ipc_*) first; the NCCL fallback has no such path");
	if (d->world - 1 > 32) return fail(HNS_ERR_UNSUPPORTED, "the sharded multigrid solve supports at most 33 ranks");
	if (d->world > 1 && !handle_out64) return fail(HNS_ERR_INVALID_ARGUMENT, "handle_out64 is null");
	const hns_grid* local = s->grid;
	const uint64_t Ll = local->num_leaves;
	if (mg->lv.empty()) return fail(HNS_ERR_INVALID_ARGUMENT, "empty multigrid hierarchy");
	const hns_grid* global = mg->lv[0].grid;
	const uint64_t Lg = global->num_leaves;
	if (Ll && !local_to_global) return fail(HNS_ERR_INVALID_ARGUMENT, "local_to_global is null");
	if (global->voxel_size != local->voxel_size) return fail(HNS_ERR_INVALID_ARGUMENT, "the hierarchy's voxel size differs from the shard's");
	if (Ll > Lg)
		return fail(HNS_ERR_INVALID_ARGUMENT, "the hierarchy's level 0 has " + std::to_string(Lg) + " leaves, fewer than the shard's " + std::to_string(Ll) +
		                                          ": it was not built over the global grid");
	std::vector<char> seen(Lg, 0);
	for (uint64_t i = 0; i < Ll; ++i) {
		const int32_t id = local_to_global[i];
		if (id < 0 || uint64_t(id) >= Lg)
			return fail(HNS_ERR_INVALID_ARGUMENT, "local_to_global[" + std::to_string(i) + "] = " + std::to_string(id) + " is not a leaf of the hierarchy's level 0 (" +
			                                          std::to_string(Lg) + " leaves)");
		if (seen[id]++) return fail(HNS_ERR_INVALID_ARGUMENT, "local_to_global lists global leaf " + std::to_string(id) + " twice");
	}
	{
		// every local leaf must BE the global leaf it is mapped to: same origin
		std::vector<int4> go(Lg), lo(Ll);
		if (Lg) HNS_CUDA(cudaMemcpy(go.data(), global->d_origin, Lg * sizeof(int4), cudaMemcpyDeviceToHost));
		if (Ll) HNS_CUDA(cudaMemcpy(lo.data(), local->d_origin, Ll * sizeof(int4), cudaMemcpyDeviceToHost));
		for (uint64_t i = 0; i < Ll; ++i) {
			const int4 a = lo[i], b = go[local_to_global[i]];
			if (a.x != b.x || a.y != b.y || a.z != b.z)
				return fail(HNS_ERR_INVALID_ARGUMENT, "local leaf " + std::to_string(i) + " lies at (" + std::to_string(a.x) + ", " + std::to_string(a.y) + ", " +
				                                          std::to_string(a.z) + ") but global leaf " + std::to_string(local_to_global[i]) +
				                                          " of the hierarchy does not: it was built over another grid");
		}
	}
	auto& m = d->smg;
	const int n = int(mg->lv.size());
	const uint64_t L1 = n > 1 ? mg->lv[1].grid->num_leaves : 0;
	if (n > 1 && Ll) {
		std::vector<int32_t> gp(Lg), lp(Ll);
		HNS_CUDA(cudaMemcpy(gp.data(), mg->lv[0].parent, Lg * sizeof(int32_t), cudaMemcpyDeviceToHost));
		for (uint64_t i = 0; i < Ll; ++i) lp[i] = gp[local_to_global[i]];
		HNS_CUDA(cudaMalloc(&m.d_parent, Ll * sizeof(int32_t)));
		HNS_CUDA(cudaMemcpy(m.d_parent, lp.data(), Ll * sizeof(int32_t), cudaMemcpyHostToDevice));
	}
	// flag word of rank r in every block: word 16 r + kChMgGather (k_signal / k_wait address flags[t] + channel)
	m.flag_bytes = (uint64_t(d->world) * 16u * sizeof(uint32_t) + 255u) & ~uint64_t(255);
	m.rhs_floats = L1 * 512u;
	const uint64_t bytes = m.flag_bytes + 2u * m.rhs_floats * sizeof(float);
	HNS_CUDA(cudaMalloc(&m.block, bytes));
	HNS_CUDA(cudaMemset(m.block, 0, bytes));  // once: octants without a fine leaf stay 0, and the peers write into it from now on
	if (handle_out64) {
		cudaIpcMemHandle_t h;
		HNS_CUDA(cudaIpcGetMemHandle(&h, m.block));
		std::memcpy(handle_out64, &h, 64);
	}
	m.ipc.assign(size_t(d->world), nullptr);
	m.mg = mg, m.cycles = cycles, m.nu_pre = nu_pre, m.nu_post = nu_post, m.omega = omega_smooth;
	return HNS_OK;
}

int hns_dist_mg_connect(hns_dist* d, int rank, const uint8_t* handle64) {
	if (!d || !handle64 || rank < 0 || rank >= d->world || rank == d->rank) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	auto& m = d->smg;
	if (!m.block) return fail(HNS_ERR_INVALID_ARGUMENT, "hns_dist_set_pressure_solver has not been called");
	cudaIpcMemHandle_t h;
	std::memcpy(&h, handle64, 64);
	if (m.ipc[rank]) cudaIpcCloseMemHandle(m.ipc[rank]), m.ipc[rank] = nullptr;
	HNS_CUDA(cudaIpcOpenMemHandle(&m.ipc[rank], h, cudaIpcMemLazyEnablePeerAccess));
	return HNS_OK;
}

int hns_dist_mg_finish(hns_dist* d) {
	if (!d) return fail(HNS_ERR_INVALID_ARGUMENT, "null argument");
	auto& m = d->smg;
	if (!m.block) return fail(HNS_ERR_INVALID_ARGUMENT, "hns_dist_set_pressure_solver has not been called");
	const int W = d->world;
	std::vector<float*> gat[2] = {std::vector<float*>(2 * W), std::vector<float*>(2 * W)};
	std::vector<uint32_t*> sig, wait;
	for (int r = 0; r < W; ++r) {
		uint8_t* b = r == d->rank ? m.block : static_cast<uint8_t*>(m.ipc[r]);
		if (!b) return fail(HNS_ERR_RUNTIME, "rank " + std::to_string(r) + " is not connected (hns_dist_mg_connect)");
		for (int par = 0; par < 2; ++par) {
			float* rhs = reinterpret_cast<float*>(b + m.flag_bytes) + uint64_t(par) * m.rhs_floats;
			gat[par][2 * r] = rhs, gat[par][2 * r + 1] = rhs + m.rhs_floats / 2;
		}
		if (r == d->rank) continue;
		sig.push_back(reinterpret_cast<uint32_t*>(b) + 16 * d->rank);
		wait.push_back(reinterpret_cast<uint32_t*>(m.block) + 16 * r);
	}
	for (int par = 0; par < 2; ++par) {
		cudaFree(m.d_gather[par]);
		m.d_gather[par] = nullptr;
		HNS_CUDA(cudaMalloc(&m.d_gather[par], gat[par].size() * sizeof(float*)));
		HNS_CUDA(cudaMemcpy(m.d_gather[par], gat[par].data(), gat[par].size() * sizeof(float*), cudaMemcpyHostToDevice));
	}
	cudaFree(m.d_sig), cudaFree(m.d_wait);
	m.d_sig = m.d_wait = nullptr;
	if (!sig.empty()) {
		HNS_CUDA(cudaMalloc(&m.d_sig, sig.size() * sizeof(uint32_t*)));
		HNS_CUDA(cudaMalloc(&m.d_wait, wait.size() * sizeof(uint32_t*)));
		HNS_CUDA(cudaMemcpy(m.d_sig, sig.data(), sig.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice));
		HNS_CUDA(cudaMemcpy(m.d_wait, wait.data(), wait.size() * sizeof(uint32_t*), cudaMemcpyHostToDevice));
	}
	m.seq = 0;  // the blocks are fresh on every rank
	m.ready = true;
	return HNS_OK;
}

// global sums of the ranks' fp64 partial sums (residual / divergence norms): ncclAllReduce(sum, fp64), SURVEY.md 8e
int hns_dist_allreduce_sum(hns_dist* d, double* inout_host, int n, void* stream) {
	if (!d || !inout_host || n <= 0 || n > 16) return fail(HNS_ERR_INVALID_ARGUMENT, "bad argument");
	if (d->world == 1) return HNS_OK;
	if (!d->comm) return fail(HNS_ERR_UNSUPPORTED, "no NCCL communicator (hns_dist_create without an id): reduce the sums with the caller's own collective");
	cudaStream_t st = static_cast<cudaStream_t>(stream);
	if (!d->d_reduce) HNS_CUDA(cudaMalloc(&d->d_reduce, 16 * sizeof(double)));
	HNS_CUDA(cudaMemcpyAsync(d->d_reduce, inout_host, size_t(n) * sizeof(double), cudaMemcpyHostToDevice, st));
	HNS_NCCL(g_nccl.AllReduce(d->d_reduce, d->d_reduce, size_t(n), ncclDouble, ncclSum, d->comm, st));
	HNS_CUDA(cudaMemcpyAsync(inout_host, d->d_reduce, size_t(n) * sizeof(double), cudaMemcpyDeviceToHost, st));
	HNS_CUDA(cudaStreamSynchronize(st));
	return HNS_OK;
}
uint64_t hns_dist_bytes_sent(const hns_dist* d) { return d ? d->bytes_sent : 0; }
uint64_t hns_dist_mg_gathers(const hns_dist* d) { return d ? d->smg.gathers : 0; }
uint64_t hns_dist_mg_gather_bytes(const hns_dist* d) { return d ? d->smg.gather_bytes : 0; }
uint64_t hns_dist_exchanges(const hns_dist* d) { return d ? d->exchanges : 0; }

}  // extern "C"
