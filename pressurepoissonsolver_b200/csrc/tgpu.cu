// tgpu.cu - C-ABI implementation (include/tgpu.h) on top of the kernels in kernels.cuh.
// Host-side structure: context (stream, scratch), hierarchy (device neighbour tables, per-level
// work vectors and face buffers, tridiagonal multiplier table), vectors, cycle driver with CUDA-graph replay.
#include <algorithm>
#include <dlfcn.h>
#include <nccl.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/tgpu.h"
#include "kernels.cuh"
#include "mesh.h"

using namespace tgpu;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static int fail(int code, const std::string &msg)
{
	g_last_error = msg;
	return code;
}
#define CU(call)                                                                                           \
	do {                                                                                                   \
		cudaError_t e_ = (call);                                                                           \
		if (e_ != cudaSuccess)                                                                             \
			return fail(TGPU_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" \
			                           + std::to_string(__LINE__) + ")");                                  \
	} while (0)
#define TRY(expr)                   \
	do {                            \
		int rc_ = (expr);           \
		if (rc_ != TGPU_OK) return rc_; \
	} while (0)
#define API_BEGIN try {
#define API_END                                            \
	}                                                      \
	catch (const std::exception &ex)                       \
	{                                                      \
		return fail(TGPU_ERR_ARG, ex.what());              \
	}                                                      \
	catch (...)                                            \
	{                                                      \
		return fail(TGPU_ERR_ARG, "unknown C++ exception"); \
	}

extern "C" const char *tgpu_last_error(void) { return g_last_error.c_str(); }
extern "C" const char *tgpu_version(void) { return "tgpu 0.1 (sm_100a, fp64)"; }

// ------------------------------------------------------------------------------------------
// NCCL, resolved at run time
// ------------------------------------------------------------------------------------------
namespace
{
struct NcclApi {
	void *lib = nullptr;
	ncclResult_t (*GetUniqueId)(ncclUniqueId *)                                                              = nullptr;
	ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int)                                       = nullptr;
	ncclResult_t (*CommDestroy)(ncclComm_t)                                                                  = nullptr;
	ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t)                = nullptr;
	ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t)                      = nullptr;
	ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t)            = nullptr;
	ncclResult_t (*GroupStart)()                                                                             = nullptr;
	ncclResult_t (*GroupEnd)()                                                                               = nullptr;
	const char *(*GetErrorString)(ncclResult_t)                                                              = nullptr;
};
NcclApi g_nccl;
int     load_nccl()
{
	if (g_nccl.lib) return TGPU_OK;
	const char *names[] = {"libnccl.so.2", "libnccl.so"};
	for (const char *nm : names) {
		g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
		if (g_nccl.lib) break;
	}
	if (!g_nccl.lib) return fail(TGPU_ERR_COMM, std::string("cannot dlopen libnccl.so.2: ") + dlerror());
#define NCCL_SYM(field, name)                                                                      \
	*(void **) (&g_nccl.field) = dlsym(g_nccl.lib, name);                                          \
	if (!g_nccl.field) return fail(TGPU_ERR_COMM, std::string("libnccl is missing symbol ") + name);
	NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
	NCCL_SYM(CommInitRank, "ncclCommInitRank")
	NCCL_SYM(CommDestroy, "ncclCommDestroy")
	NCCL_SYM(Send, "ncclSend")
	NCCL_SYM(Recv, "ncclRecv")
	NCCL_SYM(AllReduce, "ncclAllReduce")
	NCCL_SYM(AllGather, "ncclAllGather")
	NCCL_SYM(GroupStart, "ncclGroupStart")
	NCCL_SYM(GroupEnd, "ncclGroupEnd")
	NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef NCCL_SYM
	return TGPU_OK;
}
} // namespace
#define NC(call)                                                                                         \
	do {                                                                                                 \
		ncclResult_t r_ = (call);                                                                        \
		if (r_ != ncclSuccess) return fail(TGPU_ERR_COMM, std::string(#call) + ": " + g_nccl.GetErrorString(r_)); \
	} while (0)


// ------------------------------------------------------------------------------------------
// objects
// ------------------------------------------------------------------------------------------
// Owners of what the library creates, one deleter per release call: every allocation, stream, event, graph and IPC
// mapping is stored in one of these as it is created, so an error return releases it.  Kernels take .get().
struct CudaFree { void operator()(void *p) const { cudaFree(p); } };
struct CudaFreeHost { void operator()(const volatile void *p) const { cudaFreeHost((void *) p); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct GraphDestroy { void operator()(cudaGraph_t g) const { cudaGraphDestroy(g); } };
struct GraphExecDestroy { void operator()(cudaGraphExec_t g) const { cudaGraphExecDestroy(g); } };
struct IpcClose { void operator()(void *p) const { cudaIpcCloseMemHandle(p); } };
struct VecDestroy { void operator()(tgpu_vec *v) const { tgpu_vec_destroy(v); } };
template <typename T> using DevPtr  = std::unique_ptr<T, CudaFree>;
template <typename T> using HostPtr = std::unique_ptr<T, CudaFreeHost>;
using EventPtr     = std::unique_ptr<CUevent_st, EventDestroy>;
using StreamPtr    = std::unique_ptr<CUstream_st, StreamDestroy>;
using GraphPtr     = std::unique_ptr<CUgraph_st, GraphDestroy>;
using GraphExecPtr = std::unique_ptr<CUgraphExec_st, GraphExecDestroy>;
using IpcPtr       = std::unique_ptr<void, IpcClose>;
using VecPtr       = std::unique_ptr<tgpu_vec, VecDestroy>;
template <typename T> static cudaError_t dev_malloc(DevPtr<T> &p, size_t bytes)
{
	T *raw = nullptr;
	const cudaError_t e = cudaMalloc(&raw, bytes);
	if (e == cudaSuccess) p.reset(raw);
	return e;
}
template <typename T> static cudaError_t host_alloc(HostPtr<T> &p, size_t bytes, unsigned flags = cudaHostAllocDefault)
{
	T *raw = nullptr;
	const cudaError_t e = cudaHostAlloc(&raw, bytes, flags);
	if (e == cudaSuccess) p.reset(raw);
	return e;
}
static cudaError_t event_create(EventPtr &p, unsigned flags = cudaEventDefault)
{
	cudaEvent_t raw = nullptr;
	const cudaError_t e = cudaEventCreateWithFlags(&raw, flags);
	if (e == cudaSuccess) p.reset(raw);
	return e;
}
static cudaError_t stream_create(StreamPtr &p)
{
	cudaStream_t raw = nullptr;
	const cudaError_t e = cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking);
	if (e == cudaSuccess) p.reset(raw);
	return e;
}

struct tgpu_ctx {
	int          device     = 0;
	cudaStream_t stream     = nullptr;
	StreamPtr    own_stream;           // the stream tgpu_init created, until tgpu_set_stream replaces it
	int          sm_count   = 148;
	DevPtr<double>  d_partial; // [MAX_PARTIAL]
	DevPtr<double>  d_result;  // [8]
	HostPtr<double> h_result;  // pinned [8]
	EventPtr     ev0, ev1;
	int64_t      launches  = 0;
	bool         capturing = false;
	bool         last_small = false;
	int64_t      captured  = 0;
	// multi-GPU
	ncclComm_t   comm        = nullptr;
	int          rank        = 0;
	int          nranks      = 1;
	StreamPtr    comm_stream; // halo exchanges run here, concurrently with interior sweeps
	// set by p2p_wait_kernel when a peer's flag never arrives (pinned, mapped host memory: the kernel writes it, the host
	// reads it after every synchronisation point, see check_comm)
	HostPtr<volatile int> p2p_err;
	// per-launch profiling
	bool                          profiling = false;
	const char *                  tag_name  = "kernel";
	int                           tag_level = -1;
	std::vector<EventPtr>         prof_events;
	std::vector<TgpuProfileEntry> prof_entries;
	~tgpu_ctx()
	{
		cudaSetDevice(device);
		cudaStreamSynchronize(stream);
		if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
	}
};
struct Tag {
	tgpu_ctx *  ctx;
	const char *old_name;
	int         old_level;
	Tag(tgpu_ctx *c, const char *name, int level) : ctx(c), old_name(c->tag_name), old_level(c->tag_level)
	{
		c->tag_name  = name;
		c->tag_level = level;
	}
	~Tag()
	{
		ctx->tag_name  = old_name;
		ctx->tag_level = old_level;
	}
};
static constexpr int MAX_PARTIAL = 2048;
// Called after every host synchronisation point of a multi-GPU context: a halo exchange whose peer never signalled
// (crashed or stalled rank) has consumed stale faces, so everything computed since is invalid.
static int check_comm(tgpu_ctx *ctx)
{
	if (ctx->p2p_err && *ctx->p2p_err)
		return fail(TGPU_ERR_COMM, "peer-to-peer halo exchange timed out waiting for rank " + std::to_string(*ctx->p2p_err - 1)
		                           + " (results since the last successful synchronisation are invalid; the context must be torn down)");
	return TGPU_OK;
}

struct tgpu_mesh {
	Mesh                       mesh;
	std::vector<HostLevel>     levels;
	std::vector<TgpuLevelDesc> descs;
};

struct tgpu_part {
	Partition                  part;
	std::vector<TgpuLevelDesc> descs;
};

struct PeerDev {
	int    peer = -1;
	size_t send_off = 0, send_n = 0, recv_off = 0, recv_n = 0; // in faces
};
struct LevelDev {
	int        P      = 0; // owned patches (kernel loop bound, vector length)
	int64_t    global_P = 0; // patches of the level over all ranks (Domain::getNumGlobalPatches)
	int        slots  = 0; // owned + halo face slots
	bool       distributed = false;
	int        n_interior  = 0;
	EventPtr   ev[4]; // fork/join points of the overlapped exchange
	std::vector<PeerDev> peers;
	DevPtr<int32_t> send_patch, send_side, recv_slot, recv_side;
	DevPtr<double>  sendbuf, recvbuf;
	size_t     nsend = 0, nrecv = 0;
	size_t     ncells = 0, nface = 0;
	DevPtr<PatchMeta> meta;
	DevPtr<double>    starts;
	DevPtr<double>    spacing;
	double *   Fa = nullptr, *Fb = nullptr; // face buffers: Fa_own / Fb_own, or views into the peer-to-peer arena (setup_p2p)
	DevPtr<double> Fa_own, Fb_own;
	DevPtr<double> G; // 32^3 levels: [nslots][M] interface terms of the sweeps that do not start from zero (iface_rhs32_kernel)
	DevPtr<int32_t> gslot, gowner;                 // with G: the slot table (IfaceSlots32), device [P][6] and [nslots]
	std::vector<int32_t> gbegin;                   // with G: IfaceSlots32::begin on the host (slot range of a patch range)
	DevPtr<double> u, f, r; // cycle work vectors (lazily allocated)
	DevPtr<double> bnd;     // levels >= 1: Dirichlet data of the full-multigrid right-hand side, [slot][side][M] (lazily allocated)
	bool       has_neumann = false;
	DevPtr<int32_t> neu_list;               // device: owned patches with Neumann domain sides, ascending (smooth3d16_kernel<.., NEU>)
	std::vector<int32_t> neu_host;          // the same list on the host (sub-ranges are found by binary search)
	// peer-to-peer halo exchange: peers' face buffers and flags mapped with CUDA IPC (see setup_p2p)
	bool       p2p = false;
	DevPtr<int32_t> send_peer, send_ridx, peer_rank;             // device: per send face / per peer
	DevPtr<double *> peerFa, peerFb;                             // device [npeers]: the peers' Fa / Fb
	DevPtr<uint64_t *> peer_data_flag, peer_ack_flag;            // device [npeers]: my entry of the peers' flag rows
	uint64_t * data_flags = nullptr, *ack_flags = nullptr;       // my flag rows [nranks] (in the arena, written by peers)
	DevPtr<uint64_t> cnt;                                        // generation counters: data sent / awaited, ack sent / awaited
	DevPtr<unsigned> tickets;                                    // [2] finished-CTA counters of the fused push / consumer kernels
	DevPtr<PushDesc> push_desc;                                  // device [4]: (Fa | Fb) x (plain | + prolonged correction), see ensure_push_desc
	const double *push_uc = nullptr;                             // the coarse vector the descriptors were built with
};

struct GraphEntry {
	bool    want_faces = false;
	bool    guess      = false;
	double *faces      = nullptr;
	const double *faces_old = nullptr, *faces_uc = nullptr;
	const double *  f;
	double *        u;
	const double *  b          = nullptr; // full multigrid: the boundary data
	int             fmg_cycles = 0;       // full multigrid: cycles per level (0: a cycle)
	TgpuCycleOpts   opts;
	GraphExecPtr    exec;
	int64_t         kernels;
};

struct tgpu_hier {
	tgpu_ctx *            ctx = nullptr;
	int                   D = 0, N = 0;
	std::vector<LevelDev> levels;
	DevPtr<double>        scratch32; // smooth3d32n_kernel (32^3 levels with Neumann sides): one 256 KB block per CTA
	double *              cycle_faces = nullptr; // boundary slices of the last cycle's result (level 0), if it was asked to emit them
	// ... and of the iterate before its last sweep: cycle_faces_old, plus P cycle_uc on the boundary cells if that sweep was
	// the first post-sweep (cycle_uc == nullptr otherwise); see k_face_residual_norm
	const double *        cycle_faces_old = nullptr, *cycle_uc = nullptr;
	double *              visit_faces = nullptr; // the slices of the result of the last fused_visit that was asked to emit them
	DevPtr<double>        tri; // [table][N/2 + 1][N^(D-1)] tridiagonal multipliers (TriSolve), one table per distinct h
	std::vector<double>   tab_h2;          // h^2 of each table (PatchMeta::tab)
	bool                  tab_overflow = false; // more than 256 cell sizes: one table index cannot name them all
	double                tab_shift = 0.0; // the shift the tables were built with (upload_tri)
	DevPtr<double>        mats, lam; // Neumann patches: transform matrices [6][N][N], 1-D eigenvalues [3][N]
	std::vector<GraphEntry> graphs;
	std::vector<VecPtr>   krylov_ws;
	std::vector<VecPtr>   gmg_ws; // stationary solve: residual and correction of the schedules without a start from a guess
	std::vector<VecPtr>   fmg_ws; // full multigrid, schedules without a start from a guess: residual and correction of each level
	// domain-boundary sides of level 0's owned patches, ascending (patch, side) (tgpu_boundary_sides), and on the device the
	// same list with bnd_index [P][2D]: position in the list, -1 for the other sides
	std::vector<int32_t>  bnd_patch;
	std::vector<int8_t>   bnd_side;
	DevPtr<int32_t>       bnd_patch_d, bnd_index;
	DevPtr<int8_t>        bnd_side_d;
	DevPtr<double>        krylov_sc; // BiCGStab scalars on the device
	VecPtr                host_f, host_u;
	// pipelined host-buffer path (tgpu_vcycle_host_async): two slots, copy-in / copy-out streams
	VecPtr                pipe_f[2], pipe_u[2];
	StreamPtr             s_in, s_out;
	EventPtr              ev_in[2], ev_cyc[2], ev_out[2];
	uint64_t              pipe_count = 0;
	bool                  generic_kernels = false; // test hook: force the size-generic smoother
	double                lambda = 0.0;            // the patch solver's shift (tgpu_hierarchy_set_lambda / _set_helmholtz)
	double                op_shift = 0.0;          // the operator's shift: A + op_shift I (tgpu_hierarchy_set_helmholtz)
	int                   last_level = 0;          // coarsest level the running cycle visits (CycleOpts max_levels / patches_per_proc)
	// peer-to-peer arena: flag rows + the face buffers of the distributed levels, one IPC-exported allocation
	DevPtr<void>          arena;
	std::vector<IpcPtr>   ipc_opened;
	DevPtr<int>           p2p_abort; // device flag: a wait of this hierarchy has timed out (p2p_wait_kernel)

	// the cached graphs and the vectors the hierarchy created for itself; tgpu_vec_destroy needs the hierarchy intact
	void release_workspace()
	{
		graphs.clear();
		krylov_ws.clear();
		gmg_ws.clear();
		fmg_ws.clear();
		for (LevelDev &L : levels) L.bnd.reset();
		host_f.reset(), host_u.reset();
		for (int k = 0; k < 2; k++) pipe_f[k].reset(), pipe_u[k].reset();
	}
	~tgpu_hier()
	{
		cudaSetDevice(ctx->device);
		if (s_in) cudaStreamSynchronize(s_in.get()); // pending copies of the pipelined host path still use the slot vectors
		if (s_out) cudaStreamSynchronize(s_out.get());
		cudaStreamSynchronize(ctx->stream);
		release_workspace();
	}
};

// level of a boundary-data vector (tgpu_boundary_vec_create): no level operation accepts it
static constexpr int BOUNDARY_LEVEL = -1;
struct tgpu_vec {
	tgpu_hier *h     = nullptr;
	int        level = 0;
	double *   d     = nullptr;
	size_t     n     = 0;
};

// ------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------
// brackets stream work (a kernel launch, NCCL calls) with profiling events
struct ProfSpan {
	tgpu_ctx *ctx;
	ProfSpan(tgpu_ctx *c, const char *name, int level) : ctx(c)
	{
		if (!c->profiling) return;
		EventPtr e0, e1;
		event_create(e0);
		event_create(e1);
		cudaEventRecord(e0.get(), c->stream);
		c->prof_events.push_back(std::move(e0));
		c->prof_events.push_back(std::move(e1));
		c->prof_entries.push_back(TgpuProfileEntry{name, level, 0.f});
	}
	~ProfSpan()
	{
		if (ctx->profiling) cudaEventRecord(ctx->prof_events.back().get(), ctx->stream);
	}
};
template <typename... KArgs, typename... Args>
static int launch(tgpu_ctx *ctx, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args)
{
	cudaLaunchConfig_t  cfg = {};
	cudaLaunchAttribute at[1];
	cfg.gridDim          = grid;
	cfg.blockDim         = block;
	cfg.dynamicSmemBytes = smem;
	cfg.stream           = ctx->stream;
	// programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream drains
	// (every kernel of the library begins with griddepcontrol.launch_dependents + griddepcontrol.wait)
	at[0].id                                         = cudaLaunchAttributeProgrammaticStreamSerialization;
	at[0].val.programmaticStreamSerializationAllowed = 1;
	cfg.attrs                                        = at;
	// only between kernels that leave most of the GPU idle (the coarse levels): early-resident blocks of a
	// dependent grid take shared memory and warp slots away from a predecessor that fills the machine
	const bool small = (int) (grid.x * grid.y) <= ctx->sm_count;
	cfg.numAttrs     = small && ctx->last_small ? 1 : 0;
	ctx->last_small  = small;
	{
		ProfSpan span(ctx, ctx->tag_name, ctx->tag_level);
		cudaLaunchKernelEx(&cfg, kernel, args...);
	}
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return fail(TGPU_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e));
	if (ctx->capturing) ctx->captured++;
	else ctx->launches++;
	return TGPU_OK;
}
// launch() of a kernel that takes the HaloSync hs.  A launch that also pushes this rank's faces (hs.push, halo_push_cta) has its
// grid clamped to what is resident at once: every CTA must be able to become resident without another CTA of the grid retiring.
template <typename... KArgs, typename... Args>
static int halo_launch(tgpu_ctx *ctx, const HaloSync &hs, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args)
{
	if (hs.push) {
		int nb = 0;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, (int) (block.x * block.y * block.z), smem) != cudaSuccess || nb < 1)
			return fail(TGPU_ERR_CUDA, "kernel launch: occupancy query failed");
		const unsigned cap = (unsigned) nb * (unsigned) ctx->sm_count;
		if (grid.y != 1 || grid.z != 1) return fail(TGPU_ERR_ARG, "kernel launch: resident clamp needs a 1D grid");
		if (grid.x > cap) grid.x = cap; // (cap is a multiple of the SM count: even, as the 2-CTA cluster kernel needs)
	}
	return launch(ctx, kernel, grid, block, smem, args...);
}
static int grid_for(tgpu_ctx *ctx, size_t n, int block = 256, int per_sm = 8)
{
	size_t want = (n + block - 1) / block;
	size_t cap  = (size_t) ctx->sm_count * per_sm;
	return (int) std::max<size_t>(1, std::min(want, cap));
}

#define DISPATCH_DN(D_, N_, ...)                                                      \
	do {                                                                                \
		if ((D_) == 2 && (N_) == 4) { constexpr int DD = 2, NN = 4; __VA_ARGS__; }             \
		else if ((D_) == 2 && (N_) == 8) { constexpr int DD = 2, NN = 8; __VA_ARGS__; }        \
		else if ((D_) == 2 && (N_) == 16) { constexpr int DD = 2, NN = 16; __VA_ARGS__; }      \
		else if ((D_) == 2 && (N_) == 32) { constexpr int DD = 2, NN = 32; __VA_ARGS__; }      \
		else if ((D_) == 3 && (N_) == 4) { constexpr int DD = 3, NN = 4; __VA_ARGS__; }        \
		else if ((D_) == 3 && (N_) == 8) { constexpr int DD = 3, NN = 8; __VA_ARGS__; }        \
		else if ((D_) == 3 && (N_) == 16) { constexpr int DD = 3, NN = 16; __VA_ARGS__; }      \
		else return fail(TGPU_ERR_UNSUPPORTED, "unsupported (D, n) combination");       \
	} while (0)

// grid-stride kernels also exist for 32^3 patches; the tile kernels have their own (patch3d32.cuh)
#define DISPATCH_DN_ALL(D_, N_, ...)                                                  \
	do {                                                                                \
		if ((D_) == 3 && (N_) == 32) { constexpr int DD = 3, NN = 32; __VA_ARGS__; }          \
		else DISPATCH_DN(D_, N_, __VA_ARGS__);                                          \
	} while (0)
static bool is_3d32(const tgpu_hier *h) { return h->D == 3 && h->N == 32; }

static bool supported_dn(int D, int N)
{
	return (D == 2 && (N == 4 || N == 8 || N == 16 || N == 32)) || (D == 3 && (N == 4 || N == 8 || N == 16 || N == 32));
}

// specialised smoothers exist for this hierarchy's (D, n), with the face-residual kernels that can take a halo hand-over:
// always for 32^3 patches, and for 16^3 and 2-D 32^2 patches unless the size-generic kernels are forced
static bool specialised(const tgpu_hier *h)
{
	return is_3d32(h) || (((h->D == 3 && h->N == 16) || (h->D == 2 && h->N == 32)) && !h->generic_kernels);
}
// The operator carries the patch solver's shift, so the face identity of DESIGN §3 holds after a sweep: the schedules and
// kernels that work from face buffers apply.  Always so without a shift.
static bool consistent(const tgpu_hier *h) { return h->op_shift == h->lambda; }
// A smoother-only shift (tgpu_hierarchy_set_lambda): every patch takes the general transform path
static bool shifted_smoother(const tgpu_hier *h) { return h->lambda != 0.0 && !consistent(h); }
// A Helmholtz problem (tgpu_hierarchy_set_helmholtz): the Dirichlet patch solves read shifted multiplier tables, and the
// general path solves the shifted problem of an all-Neumann patch with its zero mode
static int helmholtz(const tgpu_hier *h) { return consistent(h) && h->lambda != 0.0; }

// Calls fn with one std::integral_constant<bool, ...> argument per run-time template flag.
template <class Fn> static int flag_variant(bool a, Fn &&fn) { return a ? fn(std::true_type{}) : fn(std::false_type{}); }
template <class Fn> static int flag_variant(bool a, bool b, Fn &&fn)
{
	return flag_variant(a, [&](auto A) { return flag_variant(b, [&](auto B) { return fn(A, B); }); });
}
// The variants a sweep is instantiated for: Z = zero guess, E = emit the faces, PR = fused prolongation, W = write u.  There is
// no prolongation into a sweep from a zero guess, and a sweep that emits no faces writes u: nine variants.
static constexpr bool is_sweep_variant(bool z, bool e, bool pr, bool w) { return !(z && pr) && (e || w); }
// Calls fn(Z, E, PR, W) with std::integral_constant<bool, ...> arguments for the run-time variant of a sweep.
template <class Fn> static int smooth_variant(bool zero_guess, bool emit, bool prolong, bool write_u, Fn &&fn)
{
	return flag_variant(zero_guess, emit, [&](auto Z, auto E) {
		return flag_variant(prolong, write_u, [&](auto PR, auto W) -> int {
			if constexpr (is_sweep_variant(Z, E, PR, W)) return fn(Z, E, PR, W);
			else return fail(TGPU_ERR_ARG, "k_smooth: bad variant");
		});
	});
}
// fn for each of the nine variants, through smooth_variant
template <class Fn> static int each_smooth_variant(Fn &&fn)
{
	for (int v = 0; v < 16; v++)
		if (is_sweep_variant(v & 8, v & 4, v & 2, v & 1)) TRY(smooth_variant(v & 8, v & 4, v & 2, v & 1, fn));
	return TGPU_OK;
}
// G of the 32^3 levels whose sweeps can reach smooth3d32c_kernel from a non-zero guess (iface_rhs32_kernel): no smoother-only
// shift (it sends every patch through smooth3d32n_kernel) and at least one owned patch without Neumann sides.
template <typename T> static int dev_upload(DevPtr<T> &dst, const T *src, size_t count);
// G holds one term per interface slot (IfaceSlots32, built from the owned patches' metadata with the table).  Called at
// creation and when lambda changes (never during a graph capture); the graphs are freed before G is.
static int update_iface_buffers(tgpu_hier *h)
{
	if (!is_3d32(h)) return TGPU_OK;
	for (LevelDev &L : h->levels) {
		const bool want = !shifted_smoother(h) && L.neu_host.size() < (size_t) L.P;
		if (want && !L.G) {
			std::vector<PatchMeta> meta(L.P);
			CU(cudaMemcpy(meta.data(), L.meta.get(), meta.size() * sizeof(PatchMeta), cudaMemcpyDeviceToHost));
			const IfaceSlots32 t = build_iface_slots32(meta.data(), L.P);
			TRY(dev_upload(L.gslot, t.gslot.data(), t.gslot.size()));
			TRY(dev_upload(L.gowner, t.owner.data(), t.owner.size()));
			CU(dev_malloc(L.G, std::max<size_t>(t.owner.size(), 1) * 1024 * sizeof(double)));
			L.gbegin = t.begin;
		}
		if (!want && L.G) {
			CU(cudaDeviceSynchronize());
			L.G.reset(), L.gslot.reset(), L.gowner.reset();
			L.gbegin.clear();
		}
	}
	return TGPU_OK;
}
// smooth3d32n_kernel's scratch, one 256 KB block per CTA: 32^3 hierarchies whose sweeps take the general patch solve (a level
// with Neumann sides, or a smoother-only shift)
static int ensure_scratch32(tgpu_hier *h)
{
	bool want = shifted_smoother(h);
	for (const LevelDev &L : h->levels) want = want || L.has_neumann;
	if (is_3d32(h) && want && !h->scratch32) CU(dev_malloc(h->scratch32, (size_t) h->ctx->sm_count * 2 * 32768 * sizeof(double)));
	return TGPU_OK;
}
static constexpr size_t FRR32_SMEM = 6 * 1024 * 8; // face_residual_restrict_big_kernel<3, 32>: dynamic shared memory
template <typename... A> static int set_smem(void (*kernel)(A...), size_t bytes)
{
	CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes));
	return TGPU_OK;
}
// Opt-in shared memory sizes of every instantiation the launches of this hierarchy's (D, n) can reach, each family over the
// variants of its launch dispatch.  Set at creation: the first launch may be inside a graph capture.
static int set_kernel_attrs(const tgpu_hier *h)
{
	if (is_3d32(h)) {
		TRY(each_smooth_variant([](auto Z, auto E, auto, auto W) { return set_smem(smooth3d32c_kernel<Z, E, W>, smooth3d32c_smem_bytes<Z>()); }));
		for (bool a : {false, true})
			for (bool b : {false, true}) {
				TRY(flag_variant(a, b, [](auto PR, auto HALO) { return set_smem(iface_rhs32_kernel<PR, HALO>, iface_rhs32_smem_bytes()); }));
				TRY(flag_variant(a, b, [](auto FOLD, auto HALO) { return set_smem(face_residual_restrict_big_kernel<3, 32, FOLD, HALO>, FRR32_SMEM); }));
				TRY(flag_variant(a, [](auto UC) { return set_smem(face_residual_norm_kernel<3, 32, UC ? FV_PROLONG_DIFF : FV_DIFF>, frn_smem_bytes<3, 32>()); }));
			}
		TRY(set_smem(apply3d32_tma_kernel<0>, apply3d32_tma_smem_bytes()));
		TRY(set_smem(apply3d32_tma_kernel<1>, apply3d32_tma_smem_bytes()));
		return set_smem(apply3d32_tma_kernel<3>, apply3d32_tma_smem_bytes());
	}
	DISPATCH_DN(h->D, h->N, {
		TRY(each_smooth_variant([&](auto Z, auto E, auto PR, auto) { return set_smem(smooth_kernel<DD, NN, Z, E, PR>, smooth_smem_bytes<DD, NN, true>()); }));
		TRY(set_smem(apply_tma_kernel<DD, NN, 0>, apply_tma_smem_bytes<DD, NN>()));
		TRY(set_smem(apply_tma_kernel<DD, NN, 1>, apply_tma_smem_bytes<DD, NN>()));
		TRY(set_smem(apply_tma_kernel<DD, NN, 2>, apply_tma_smem_bytes<DD, NN>()));
		TRY(set_smem(apply_tma_kernel<DD, NN, 3>, apply_tma_smem_bytes<DD, NN>()));
	});
	if (h->D == 3 && h->N == 16) // as launch_smooth3d16 launches them: plain, with the hand-over, Neumann
		return each_smooth_variant([](auto Z, auto E, auto PR, auto W) {
			TRY(set_smem(smooth3d16_kernel<Z, E, PR, W>, smooth3d16_smem_bytes()));
			TRY(set_smem(smooth3d16_kernel<Z, E, PR, W, !Z>, smooth3d16_smem_bytes()));
			return set_smem(smooth3d16_kernel<Z, E, PR, W, false, true>, smooth3d16_smem_bytes());
		});
	if (h->D == 2 && h->N == 32) // without and with the hand-over and Neumann skip (EXTRA)
		return each_smooth_variant([](auto Z, auto E, auto PR, auto W) {
			TRY(set_smem(smooth2d32_kernel<Z, E, PR, W, false>, smooth2d32_smem_bytes()));
			return set_smem(smooth2d32_kernel<Z, E, PR, W, true>, smooth2d32_smem_bytes());
		});
	return TGPU_OK;
}

// transform tables, evaluated exactly like DftPatchSolver.h:237-289 (M_PI / n * (...))
static int init_constant_tables()
{
	for (int n : {4, 8, 16, 32}) {
		const int           H = n / 2;
		std::vector<double> fwd((size_t) n * H), inv((size_t) H * n);
		for (int k = 0; k < n; k++)
			for (int j = 0; j < H; j++) fwd[(size_t) k * H + j] = sin(M_PI / n * ((k + 1) * (j + 0.5)));
		for (int i = 0; i < H; i++) {
			for (int j = 0; j < n - 1; j++) inv[(size_t) i * n + j] = sin(M_PI / n * ((i + 0.5) * (j + 1)));
			inv[(size_t) i * n + n - 1] = (i % 2 == 0) ? 0.5 : -0.5;
		}
		std::vector<double> mag(n + 1);
		for (int i = 0; i <= n; i++) mag[i] = sin(M_PI / (2.0 * n) * i);
		mag[n] = 1.0;
		if (n == 4) CU(cudaMemcpyToSymbol(c_mag4, mag.data(), mag.size() * 8));
		else if (n == 8) CU(cudaMemcpyToSymbol(c_mag8, mag.data(), mag.size() * 8));
		else if (n == 16) CU(cudaMemcpyToSymbol(c_mag16, mag.data(), mag.size() * 8));
		else CU(cudaMemcpyToSymbol(c_mag32, mag.data(), mag.size() * 8));
		if (n == 4) {
			CU(cudaMemcpyToSymbol(c_fwd4, fwd.data(), fwd.size() * 8));
			CU(cudaMemcpyToSymbol(c_inv4, inv.data(), inv.size() * 8));
		} else if (n == 8) {
			CU(cudaMemcpyToSymbol(c_fwd8, fwd.data(), fwd.size() * 8));
			CU(cudaMemcpyToSymbol(c_inv8, inv.data(), inv.size() * 8));
		} else if (n == 16) {
			CU(cudaMemcpyToSymbol(c_fwd16, fwd.data(), fwd.size() * 8));
			CU(cudaMemcpyToSymbol(c_inv16, inv.data(), inv.size() * 8));
		} else {
			CU(cudaMemcpyToSymbol(c_fwd32, fwd.data(), fwd.size() * 8));
			CU(cudaMemcpyToSymbol(c_inv32, inv.data(), inv.size() * 8));
		}
	}
	return TGPU_OK;
}

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
extern "C" int tgpu_init(int device, tgpu_ctx **out)
{
	API_BEGIN
	if (!out) return fail(TGPU_ERR_ARG, "tgpu_init: null output pointer");
	int ndev = 0;
	cudaError_t e = cudaGetDeviceCount(&ndev);
	if (e != cudaSuccess || ndev == 0)
		return fail(TGPU_ERR_CUDA, std::string("tgpu_init: no CUDA device available (") + cudaGetErrorString(e)
		                           + "); this library has no CPU fallback");
	if (device < 0 || device >= ndev) return fail(TGPU_ERR_ARG, "tgpu_init: device index out of range");
	CU(cudaSetDevice(device));
	std::unique_ptr<tgpu_ctx> ctx(new tgpu_ctx());
	ctx->device = device;
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, device));
	ctx->sm_count = prop.multiProcessorCount;
	CU(stream_create(ctx->own_stream));
	ctx->stream = ctx->own_stream.get();
	CU(dev_malloc(ctx->d_partial, MAX_PARTIAL * sizeof(double)));
	CU(dev_malloc(ctx->d_result, 8 * sizeof(double)));
	CU(host_alloc(ctx->h_result, 8 * sizeof(double)));
	CU(event_create(ctx->ev0));
	CU(event_create(ctx->ev1));
	{ // vector storage pool (tgpu_vec_create): keep freed blocks across synchronisations; tgpu_hierarchy_trim releases them
		cudaMemPool_t pool = nullptr;
		CU(cudaDeviceGetDefaultMemPool(&pool, device));
		uint64_t keep = ~0ull;
		CU(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
	}
	TRY(init_constant_tables());
	*out = ctx.release();
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_finalize(tgpu_ctx *ctx)
{
	delete ctx;
	return TGPU_OK;
}
extern "C" int tgpu_set_stream(tgpu_ctx *ctx, void *s)
{
	if (!ctx) return fail(TGPU_ERR_ARG, "null context");
	CU(cudaStreamSynchronize(ctx->stream));
	ctx->own_stream.reset();
	ctx->stream = (cudaStream_t) s;
	return TGPU_OK;
}
extern "C" int tgpu_sync(tgpu_ctx *ctx)
{
	if (!ctx) return fail(TGPU_ERR_ARG, "null context");
	CU(cudaStreamSynchronize(ctx->stream));
	return check_comm(ctx);
}
extern "C" int tgpu_kernel_launches(tgpu_ctx *ctx, int64_t *count)
{
	if (!ctx || !count) return fail(TGPU_ERR_ARG, "null argument");
	*count = ctx->launches;
	return TGPU_OK;
}
extern "C" int tgpu_timer_start(tgpu_ctx *ctx)
{
	if (!ctx) return fail(TGPU_ERR_ARG, "null context");
	CU(cudaEventRecord(ctx->ev0.get(), ctx->stream));
	return TGPU_OK;
}
extern "C" int tgpu_timer_stop(tgpu_ctx *ctx, double *ms)
{
	if (!ctx || !ms) return fail(TGPU_ERR_ARG, "null argument");
	CU(cudaEventRecord(ctx->ev1.get(), ctx->stream));
	CU(cudaEventSynchronize(ctx->ev1.get()));
	float f = 0;
	CU(cudaEventElapsedTime(&f, ctx->ev0.get(), ctx->ev1.get()));
	*ms = f;
	return check_comm(ctx);
}

extern "C" int tgpu_profile_begin(tgpu_ctx *ctx)
{
	if (!ctx) return fail(TGPU_ERR_ARG, "null context");
	CU(cudaStreamSynchronize(ctx->stream));
	ctx->prof_events.clear();
	ctx->prof_entries.clear();
	ctx->profiling = true;
	return TGPU_OK;
}
extern "C" int tgpu_profile_end(tgpu_ctx *ctx, int *n, const TgpuProfileEntry **entries)
{
	if (!ctx || !n || !entries) return fail(TGPU_ERR_ARG, "null argument");
	ctx->profiling = false;
	CU(cudaStreamSynchronize(ctx->stream));
	for (size_t i = 0; i < ctx->prof_entries.size(); i++)
		CU(cudaEventElapsedTime(&ctx->prof_entries[i].ms, ctx->prof_events[2 * i].get(), ctx->prof_events[2 * i + 1].get()));
	*n       = (int) ctx->prof_entries.size();
	*entries = ctx->prof_entries.data();
	return TGPU_OK;
}

// ------------------------------------------------------------------------------------------
// mesh
// ------------------------------------------------------------------------------------------
extern "C" int tgpu_mesh_load(const char *path, int D, tgpu_mesh **out)
{
	API_BEGIN
	if (!path || !out) return fail(TGPU_ERR_ARG, "tgpu_mesh_load: null argument");
	std::unique_ptr<tgpu_mesh> m(new tgpu_mesh());
	try {
		m->mesh = Mesh::load(path, D);
	} catch (const std::exception &ex) {
		return fail(TGPU_ERR_IO, ex.what());
	}
	*out = m.release();
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_mesh_uniform(int D, int num_levels, tgpu_mesh **out)
{
	API_BEGIN
	if (!out || num_levels < 1) return fail(TGPU_ERR_ARG, "tgpu_mesh_uniform: bad argument");
	std::unique_ptr<tgpu_mesh> m(new tgpu_mesh());
	m->mesh = Mesh::uniform(D, num_levels);
	*out    = m.release();
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_mesh_refine_leaves(tgpu_mesh *m)
{
	API_BEGIN
	if (!m) return fail(TGPU_ERR_ARG, "null mesh");
	m->mesh.refineLeaves();
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_mesh_refine_box(tgpu_mesh *m, const double *lo, const double *hi)
{
	API_BEGIN
	if (!m || !lo || !hi) return fail(TGPU_ERR_ARG, "null argument");
	m->mesh.refineBox(lo, hi);
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_mesh_set_neumann(tgpu_mesh *m, int on)
{
	if (!m) return fail(TGPU_ERR_ARG, "null mesh");
	m->mesh.neumann = on != 0;
	return TGPU_OK;
}
extern "C" int tgpu_mesh_destroy(tgpu_mesh *m)
{
	delete m;
	return TGPU_OK;
}
extern "C" int tgpu_mesh_info(const tgpu_mesh *m, int *D, int *num_levels, int *num_nodes)
{
	if (!m) return fail(TGPU_ERR_ARG, "null mesh");
	if (D) *D = m->mesh.D;
	if (num_levels) *num_levels = m->mesh.num_levels;
	if (num_nodes) *num_nodes = m->mesh.numNodes();
	return TGPU_OK;
}
extern "C" int tgpu_mesh_extract_levels(tgpu_mesh *m, int n, int *nlevels, const TgpuLevelDesc **levels)
{
	API_BEGIN
	if (!m || !nlevels || !levels) return fail(TGPU_ERR_ARG, "null argument");
	if (n < 2 || (n & 1)) return fail(TGPU_ERR_ARG, "n must be even and >= 2");
	m->levels = m->mesh.extractLevels(n);
	m->descs.clear();
	for (const HostLevel &L : m->levels) m->descs.push_back(L.desc());
	*nlevels = (int) m->descs.size();
	*levels  = m->descs.data();
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_mesh_level_ids(const tgpu_mesh *m, int level, const int32_t **ids, const int32_t **parent_ids,
                                   const int32_t **refine_levels)
{
	if (!m || level < 0 || level >= (int) m->levels.size()) return fail(TGPU_ERR_ARG, "bad level");
	if (ids) *ids = m->levels[level].ids.data();
	if (parent_ids) *parent_ids = m->levels[level].parent_ids.data();
	if (refine_levels) *refine_levels = m->levels[level].refine_levels.data();
	return TGPU_OK;
}

// ------------------------------------------------------------------------------------------
// hierarchy
// ------------------------------------------------------------------------------------------
template <typename T> static int dev_upload(DevPtr<T> &dst, const T *src, size_t count)
{
	CU(dev_malloc(dst, std::max<size_t>(1, count) * sizeof(T)));
	if (count) CU(cudaMemcpy(dst.get(), src, count * sizeof(T), cudaMemcpyHostToDevice));
	return TGPU_OK;
}

// Multipliers of the two-sided tridiagonal elimination along the axis that is not transformed, for every pencil of the other
// axes' transform indices (TriSolve, kernels.cuh): one table [n/2 + 1][n^(D-1)] per cell size h of the hierarchy (h->tab_h2),
// with the diagonal shifted by lambda h^2 in the Helmholtz state and unshifted otherwise.  Unshifted tables are all equal.
// Rebuilt when the shift changes; the caller has dropped the graphs that could still be reading them.
static int upload_tri(tgpu_hier *h)
{
	const double shift = helmholtz(h) ? h->lambda : 0.0;
	if (h->tri && shift == h->tab_shift) return TGPU_OK;
	const int    D = h->D, n = h->N, H = n / 2;
	const size_t M = D == 2 ? n : (size_t) n * n, T = (size_t) (H + 1) * M;
	std::vector<double>      tri(T * h->tab_h2.size());
	std::vector<long double> ll(n);
	for (int k = 0; k < n; k++) {
		const long double sn = sinl((k + 1) * 3.141592653589793238462643383279502884L / (2 * n));
		ll[k]                = -4.0L * sn * sn;
	}
	for (size_t t = 0; t < h->tab_h2.size(); t++) {
		const long double lh2 = (long double) shift * h->tab_h2[t];
		double *const     tab = tri.data() + t * T;
		for (size_t m = 0; m < M; m++) {
			const long double mu = (D == 2) ? ll[m] : ll[m % n] + ll[m / n];
			long double       a  = 0.0L;
			for (int j = 0; j < H; j++) {
				const long double d = mu - (j == 0 ? 3.0L : 2.0L) + lh2;
				a                   = 1.0L / (d - (j == 0 ? 0.0L : a));
				tab[(size_t) j * M + m] = (double) a;
			}
			tab[(size_t) H * M + m] = (double) (1.0L / (1.0L - a * a));
		}
	}
	if (!h->tri) TRY(dev_upload(h->tri, tri.data(), tri.size()));
	else {
		CU(cudaStreamSynchronize(h->ctx->stream)); // sweeps still in flight read the old tables
		CU(cudaMemcpy(h->tri.get(), tri.data(), tri.size() * sizeof(double), cudaMemcpyHostToDevice));
	}
	h->tab_shift = shift;
	return TGPU_OK;
}

// n_owned == nullptr: every patch of every level is owned (single GPU).  Otherwise level l has n_owned[l]
// owned patches followed by halo face slots (multi-GPU, see tgpu_hierarchy_create_distributed).
static int hierarchy_create_impl(tgpu_ctx *ctx, int D, int n, int nlevels, const TgpuLevelDesc *levels, const int32_t *n_owned,
                                 std::unique_ptr<tgpu_hier> &out)
{
	API_BEGIN
	if (!ctx || !levels || nlevels < 1) return fail(TGPU_ERR_ARG, "tgpu_hierarchy_create: bad argument");
	if (!supported_dn(D, n))
		return fail(TGPU_ERR_UNSUPPORTED, "tgpu_hierarchy_create: (D, n) must be one of 2D n=4/8/16/32, 3D n=4/8/16/32");
	CU(cudaSetDevice(ctx->device));
	std::unique_ptr<tgpu_hier> h(new tgpu_hier());
	h->ctx = ctx;
	h->D   = D;
	h->N   = n;
	const int S = 2 * D, Q = 1 << (D - 1);
	size_t    M = 1;
	for (int i = 0; i < D - 1; i++) M *= n;
	const size_t NC = M * n;
	// h^2 -> multiplier table (PatchMeta::tab).  Sizes within the isotropy check's relative 1e-12 share a table.  Past 256
	// sizes the extra ones point at table 0: unshifted tables are all equal, and tgpu_hierarchy_set_helmholtz refuses a
	// shift on such a hierarchy.
	std::map<double, int> tab_of;
	for (int l = 0; l < nlevels; l++) {
		const TgpuLevelDesc &d = levels[l];
		if (d.npatch < 1) return fail(TGPU_ERR_ARG, "level without patches");
		LevelDev L;
		L.P      = n_owned ? n_owned[l] : d.npatch;
		L.global_P = L.P;
		L.slots  = d.npatch;
		L.ncells = (size_t) L.P * NC;
		L.nface  = (size_t) d.npatch * S * M;
		if (L.P < 0 || L.P > d.npatch) return fail(TGPU_ERR_ARG, "owned patch count out of range");
		// the 16^3 smoother's gather descriptors (GDesc16, smooth3d16.cuh) hold 32-bit element offsets into the face
		// buffer ((slot * 6 + side) * 256) and into the coarser level's vector (parent * 4096)
		if (D == 3 && n == 16 && ((uint64_t) d.npatch * 6 * 256 > 0xffffffffull || (l > 0 && (uint64_t) d.npatch * 4096 > 0xffffffffull)))
			return fail(TGPU_ERR_UNSUPPORTED, "tgpu_hierarchy_create: more than 2.7 M patches of 16^3 on one level of one GPU (1 M on a coarser level) exceed the 32-bit gather offsets");
		std::vector<PatchMeta> meta(d.npatch);
		const int              Pc = (l + 1 < nlevels) ? levels[l + 1].npatch : 0;
		for (int p = 0; p < d.npatch; p++) {
			PatchMeta &pm = meta[p];
			memset(&pm, 0, sizeof(pm));
			const double hx = d.spacing[(size_t) p * D];
			for (int a = 1; a < D; a++)
				if (std::fabs(d.spacing[(size_t) p * D + a] - hx) > 1e-12 * std::fabs(hx))
					return fail(TGPU_ERR_UNSUPPORTED, "patches must be cubic with isotropic spacing (SURVEY App. A.1)");
			pm.h2             = hx * hx;
			pm.inv_h2         = 1.0 / (hx * hx);
			{
				const auto near = tab_of.lower_bound(pm.h2 * (1.0 - 1e-12));
				int        tab  = (int) tab_of.size();
				if (near != tab_of.end() && near->first <= pm.h2 * (1.0 + 1e-12)) tab = near->second;
				else {
					tab_of.emplace(pm.h2, tab);
					if (tab < 256) h->tab_h2.push_back(pm.h2);
				}
				pm.tab = (uint8_t) (tab < 256 ? tab : 0);
			}
			pm.neumann        = d.neumann_bits ? d.neumann_bits[p] : 0;
			if (pm.neumann) L.has_neumann = true;
			if (pm.neumann && p < L.P) L.neu_host.push_back(p);
			pm.parent_idx     = d.parent_idx ? d.parent_idx[p] : -1;
			pm.orth_on_parent = d.orth_on_parent ? d.orth_on_parent[p] : -1;
			if (l + 1 < nlevels && p < L.P) {
				if (pm.parent_idx < 0 || pm.parent_idx >= Pc) return fail(TGPU_ERR_ARG, "parent_idx out of range");
				if (pm.orth_on_parent >= (1 << D)) return fail(TGPU_ERR_ARG, "orth_on_parent out of range");
			}
			for (int s = 0; s < 6; s++) {
				pm.nbr_type[s]       = NBR_NONE;
				pm.orth_on_coarse[s] = -1;
				pm.nbr_parent[s]     = 0;
				pm.nbr_orth[s]       = -1;
				for (int q = 0; q < 4; q++) pm.nbr_idx[s][q] = -1;
			}
			for (int s = 0; s < S; s++) {
				const int t    = d.nbr_type[(size_t) p * S + s];
				pm.nbr_type[s] = (int8_t) t;
				if (t == NBR_NONE) continue;
				if (t < 0 || t > 2) return fail(TGPU_ERR_ARG, "bad neighbour type");
				const int cnt = (t == NBR_FINE) ? Q : 1;
				for (int q = 0; q < cnt; q++) {
					const int j = d.nbr_idx[((size_t) p * S + s) * Q + q];
					if (j < 0 || j >= d.npatch) return fail(TGPU_ERR_ARG, "nbr_idx out of range");
					pm.nbr_idx[s][q] = j;
				}
				if (d.parent_idx) pm.nbr_parent[s] = d.parent_idx[pm.nbr_idx[s][0]];
				if (d.orth_on_parent) pm.nbr_orth[s] = d.orth_on_parent[pm.nbr_idx[s][0]];
				if (t == NBR_COARSE) {
					const int o = d.orth_on_coarse[(size_t) p * S + s];
					if (o < 0 || o >= Q) return fail(TGPU_ERR_ARG, "orth_on_coarse out of range");
					pm.orth_on_coarse[s] = (int8_t) o;
				}
			}
			// a Neumann bit means a domain side: on a side with a neighbour the smoother would pick a Neumann transform that
			// the operator (which reads the neighbour) does not match, and bits past side 2D - 1 name no side
			if (p < L.P) {
				if (pm.neumann >> S) return fail(TGPU_ERR_ARG, "neumann_bits: bit set past side 2D - 1");
				for (int s = 0; s < S; s++)
					if (((pm.neumann >> s) & 1) && pm.nbr_type[s] != NBR_NONE)
						return fail(TGPU_ERR_ARG, "neumann_bits: Neumann bit on a side with a neighbour");
			}
		}
		TRY(dev_upload(L.meta, meta.data(), meta.size()));
		if (!L.neu_host.empty()) TRY(dev_upload(L.neu_list, L.neu_host.data(), L.neu_host.size()));
		TRY(dev_upload(L.spacing, d.spacing, (size_t) d.npatch * D));
		if (d.starts) TRY(dev_upload(L.starts, d.starts, (size_t) d.npatch * D));
		CU(dev_malloc(L.Fa_own, L.nface * sizeof(double)));
		CU(dev_malloc(L.Fb_own, L.nface * sizeof(double)));
		L.Fa = L.Fa_own.get(), L.Fb = L.Fb_own.get();
		h->levels.push_back(std::move(L));
	}
	h->tab_overflow = tab_of.size() > 256;
	TRY(upload_tri(h.get()));
	// general transform path (patches with Neumann domain sides): the six matrices of DftPatchSolver.h:237-289,
	// M[k][j] such that y_k = sum_j M[k][j] x_j, order TK_*; 1-D eigenvalues -4 sin^2((k + shift) pi / 2n), shift 1, 0, 1/2
	{
		std::vector<double> mats((size_t) 6 * n * n), lam((size_t) 3 * n);
		auto M = [&](int kind, int k, int j) -> double & { return mats[((size_t) kind * n + k) * n + j]; };
		for (int k = 0; k < n; k++)
			for (int j = 0; j < n; j++) {
				M(0, k, j) = sin(M_PI / n * ((k + 1) * (j + 0.5)));
				M(1, k, j) = (j == n - 1) ? ((k % 2 == 0) ? 0.5 : -0.5) : sin(M_PI / n * ((k + 0.5) * (j + 1)));
				M(2, k, j) = cos(M_PI / n * (k * (j + 0.5)));
				M(3, k, j) = (j == 0) ? 0.5 : cos(M_PI / n * ((k + 0.5) * j));
				M(4, k, j) = cos(M_PI / n * ((k + 0.5) * (j + 0.5)));
				M(5, k, j) = sin(M_PI / n * ((k + 0.5) * (j + 0.5)));
			}
		const double shift[3] = {1.0, 0.0, 0.5};
		for (int t = 0; t < 3; t++)
			for (int k = 0; k < n; k++) lam[(size_t) t * n + k] = -4.0 * pow(sin((k + shift[t]) * M_PI / (2 * n)), 2);
		TRY(dev_upload(h->mats, mats.data(), mats.size()));
		TRY(dev_upload(h->lam, lam.data(), lam.size()));
	}
	{ // the domain-boundary sides of level 0 (tgpu_boundary_sides)
		const int            P0 = h->levels[0].P;
		std::vector<int32_t> index((size_t) P0 * S, -1);
		for (int p = 0; p < P0; p++)
			for (int s = 0; s < S; s++)
				if (levels[0].nbr_type[(size_t) p * S + s] == NBR_NONE) {
					index[(size_t) p * S + s] = (int32_t) h->bnd_patch.size();
					h->bnd_patch.push_back(p);
					h->bnd_side.push_back((int8_t) s);
				}
		TRY(dev_upload(h->bnd_patch_d, h->bnd_patch.data(), h->bnd_patch.size()));
		TRY(dev_upload(h->bnd_side_d, h->bnd_side.data(), h->bnd_side.size()));
		TRY(dev_upload(h->bnd_index, index.data(), index.size()));
	}
	TRY(set_kernel_attrs(h.get()));
	TRY(ensure_scratch32(h.get()));
	TRY(update_iface_buffers(h.get()));
	out = std::move(h);
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_hierarchy_create(tgpu_ctx *ctx, int D, int n, int nlevels, const TgpuLevelDesc *levels, tgpu_hier **out)
{
	if (!out) return fail(TGPU_ERR_ARG, "tgpu_hierarchy_create: bad argument");
	std::unique_ptr<tgpu_hier> h;
	TRY(hierarchy_create_impl(ctx, D, n, nlevels, levels, nullptr, h));
	*out = h.release();
	return TGPU_OK;
}

// ------------------------------------------------------------------------------------------
// multi-GPU: partition ABI, NCCL (resolved at run time with dlopen so that libtgpu.so itself has
// no link-time NCCL dependency), distributed hierarchy
// ------------------------------------------------------------------------------------------
extern "C" int tgpu_mesh_partition(tgpu_mesh *m, int n, int rank, int nranks, int min_patches_per_rank, tgpu_part **out)
{
	API_BEGIN
	if (!m || !out) return fail(TGPU_ERR_ARG, "null argument");
	if (n < 2 || (n & 1)) return fail(TGPU_ERR_ARG, "n must be even and >= 2");
	std::unique_ptr<tgpu_part> p(new tgpu_part());
	std::vector<HostLevel>     global = m->mesh.extractLevels(n);
	p->part                           = partitionLevels(global, m->mesh.D, n, rank, nranks, min_patches_per_rank);
	for (const PartLevel &L : p->part.levels) p->descs.push_back(L.local.desc());
	*out = p.release();
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_part_destroy(tgpu_part *p)
{
	delete p;
	return TGPU_OK;
}
extern "C" int tgpu_part_info(const tgpu_part *p, int *nlevels, int *ndist)
{
	if (!p) return fail(TGPU_ERR_ARG, "null partition");
	if (nlevels) *nlevels = (int) p->part.levels.size();
	if (ndist) *ndist = p->part.ndist;
	return TGPU_OK;
}
extern "C" int tgpu_part_level(const tgpu_part *p, int level, TgpuLevelDesc *desc, int32_t *n_owned, int32_t *n_halo,
                               const int32_t **owned_global, const int32_t **halo_global, const int32_t **halo_owner, int32_t *npeers)
{
	if (!p || level < 0 || level >= (int) p->part.levels.size()) return fail(TGPU_ERR_ARG, "bad level");
	const PartLevel &L = p->part.levels[level];
	if (desc) *desc = p->descs[level];
	if (n_owned) *n_owned = L.n_owned;
	if (n_halo) *n_halo = L.n_halo;
	if (owned_global) *owned_global = L.owned_global.data();
	if (halo_global) *halo_global = L.halo_global.data();
	if (halo_owner) *halo_owner = L.halo_owner.data();
	if (npeers) *npeers = (int32_t) L.peers.size();
	return TGPU_OK;
}
extern "C" int tgpu_part_level_interior(const tgpu_part *p, int level, int32_t *n_interior)
{
	if (!p || !n_interior || level < 0 || level >= (int) p->part.levels.size()) return fail(TGPU_ERR_ARG, "bad argument");
	*n_interior = p->part.levels[level].n_interior;
	return TGPU_OK;
}
extern "C" int tgpu_part_peer(const tgpu_part *p, int level, int k, int32_t *peer, int32_t *nsend, const int32_t **send_patch,
                              const int32_t **send_side, int32_t *nrecv, const int32_t **recv_slot, const int32_t **recv_side)
{
	if (!p || level < 0 || level >= (int) p->part.levels.size()) return fail(TGPU_ERR_ARG, "bad level");
	const PartLevel &L = p->part.levels[level];
	if (k < 0 || k >= (int) L.peers.size()) return fail(TGPU_ERR_ARG, "bad peer index");
	const PeerExchange &x = L.peers[k];
	if (peer) *peer = x.peer;
	if (nsend) *nsend = (int32_t) x.send_patch.size();
	if (send_patch) *send_patch = x.send_patch.data();
	if (send_side) *send_side = x.send_side.data();
	if (nrecv) *nrecv = (int32_t) x.recv_slot.size();
	if (recv_slot) *recv_slot = x.recv_slot.data();
	if (recv_side) *recv_side = x.recv_side.data();
	return TGPU_OK;
}

extern "C" int tgpu_comm_unique_id(void *id128)
{
	API_BEGIN
	if (!id128) return fail(TGPU_ERR_ARG, "null argument");
	TRY(load_nccl());
	static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
	ncclUniqueId id;
	NC(g_nccl.GetUniqueId(&id));
	memcpy(id128, &id, sizeof(id));
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_comm_init(tgpu_ctx *ctx, const void *id128, int rank, int nranks)
{
	API_BEGIN
	if (!ctx || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(TGPU_ERR_ARG, "tgpu_comm_init: bad argument");
	TRY(load_nccl());
	CU(cudaSetDevice(ctx->device));
	ncclUniqueId id;
	memcpy(&id, id128, sizeof(id));
	NC(g_nccl.CommInitRank(&ctx->comm, nranks, id, rank));
	if (!ctx->comm_stream) CU(stream_create(ctx->comm_stream));
	if (!ctx->p2p_err) {
		CU(host_alloc(ctx->p2p_err, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
		*ctx->p2p_err = 0;
	}
	ctx->rank   = rank;
	ctx->nranks = nranks;
	return TGPU_OK;
	API_END
}

// ------------------------------------------------------------------------------------------
// peer-to-peer set-up: one IPC-exported arena per rank holds the flag rows and the face buffers of the
// distributed levels; every rank maps the arenas of its neighbours and learns into which of their halo
// slots each of its boundary faces goes.  NCCL is used here once, as the bootstrap transport.
// ------------------------------------------------------------------------------------------
struct P2PPack {
	cudaIpcMemHandle_t handle;
	int32_t            ok;                 // this rank could allocate and export its arena
	uint64_t           base_off;           // arena - allocation base
	uint64_t           flags_off;          // flag rows: [level][kind: data, ack][rank]
	uint64_t           fa_off[16], fb_off[16];
};
static size_t align256(size_t x) { return (x + 255) & ~(size_t) 255; }
static int alloc_base_of(void *ptr, void **base)
{
	typedef int (*fn_t)(unsigned long long *, size_t *, unsigned long long);
	void *                          fn = nullptr;
	cudaDriverEntryPointQueryResult qr;
	CU(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qr));
	if (!fn || qr != cudaDriverEntryPointSuccess) return fail(TGPU_ERR_CUDA, "cuMemGetAddressRange is not available");
	unsigned long long b  = 0;
	size_t             sz = 0;
	if (((fn_t) fn)(&b, &sz, (unsigned long long) (uintptr_t) ptr) != 0) return fail(TGPU_ERR_CUDA, "cuMemGetAddressRange failed");
	*base = (void *) (uintptr_t) b;
	return TGPU_OK;
}
static int setup_p2p(tgpu_hier *h, const Partition &pt)
{
	tgpu_ctx *ctx = h->ctx;
	const int nl = (int) h->levels.size(), nr = ctx->nranks, me = ctx->rank;
	if (nl > 16) return fail(TGPU_ERR_UNSUPPORTED, "peer-to-peer exchange supports at most 16 levels");
	const int S = 2 * h->D;
	size_t    M = 1;
	for (int i = 0; i < h->D - 1; i++) M *= h->N;
	// ---- arena layout ----
	P2PPack mine;
	memset(&mine, 0, sizeof(mine));
	size_t off      = 0;
	mine.flags_off  = off;
	off += align256((size_t) nl * 2 * nr * sizeof(uint64_t));
	for (int l = 0; l < nl; l++) {
		LevelDev &L = h->levels[l];
		if (!L.distributed || (L.nsend == 0 && L.nrecv == 0)) continue;
		mine.fa_off[l] = off, off += align256(L.nface * sizeof(double));
		mine.fb_off[l] = off, off += align256(L.nface * sizeof(double));
	}
	// Everything that can fail on ONE rank only (allocation, IPC export, mapping a peer) is recorded in `ok` instead of
	// returned: the ranks then agree on the outcome with an all-reduce, and if any of them cannot map its peers every
	// rank keeps the NCCL send/recv exchange (k_exchange), so nobody is left waiting in a collective.
	int         ok = 1;
	std::string why;
	auto        soft = [&](cudaError_t e, const char *what) {
        if (e != cudaSuccess && ok) {
            ok  = 0;
            why = std::string(what) + ": " + cudaGetErrorString(e);
            cudaGetLastError();
        }
	};
	soft(dev_malloc(h->arena, off), "cudaMalloc(arena)");
	if (ok) soft(cudaMemset(h->arena.get(), 0, off), "cudaMemset(arena)");
	if (ok) {
		void *base = nullptr;
		if (alloc_base_of(h->arena.get(), &base) != TGPU_OK) ok = 0, why = "cuMemGetAddressRange failed";
		else {
			mine.base_off = (uint64_t) ((char *) h->arena.get() - (char *) base);
			soft(cudaIpcGetMemHandle(&mine.handle, base), "cudaIpcGetMemHandle");
		}
	}
	mine.ok = ok;
	// ---- all-gather the packs ----
	std::vector<P2PPack> all(nr);
	{
		DevPtr<P2PPack> d_mine, d_all;
		CU(dev_malloc(d_mine, sizeof(P2PPack)));
		CU(dev_malloc(d_all, sizeof(P2PPack) * nr));
		CU(cudaMemcpy(d_mine.get(), &mine, sizeof(P2PPack), cudaMemcpyHostToDevice));
		NC(g_nccl.AllGather(d_mine.get(), d_all.get(), sizeof(P2PPack), ncclChar, ctx->comm, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
		CU(cudaMemcpy(all.data(), d_all.get(), sizeof(P2PPack) * nr, cudaMemcpyDeviceToHost));
	}
	for (int r = 0; r < nr; r++)
		if (!all[r].ok && ok) ok = 0, why = "rank " + std::to_string(r) + " could not export its arena";
	// ---- map the arenas of the ranks I exchange with ----
	std::vector<char *> rarena(nr, nullptr);
	rarena[me] = (char *) h->arena.get();
	for (int l = 0; l < nl && ok; l++)
		for (const PeerDev &pd : h->levels[l].peers) {
			if (rarena[pd.peer] || !ok) continue;
			void *rb = nullptr;
			soft(cudaIpcOpenMemHandle(&rb, all[pd.peer].handle, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
			if (!ok) break;
			h->ipc_opened.emplace_back(rb);
			rarena[pd.peer] = (char *) rb + all[pd.peer].base_off;
		}
	if (ok) soft(dev_malloc(h->p2p_abort, sizeof(int)), "cudaMalloc(abort flag)");
	if (ok) soft(cudaMemset(h->p2p_abort.get(), 0, sizeof(int)), "cudaMemset(abort flag)");
	{ // agreement: peer-to-peer only if every rank mapped everything it needs
		DevPtr<int> d;
		CU(dev_malloc(d, sizeof(int)));
		CU(cudaMemcpy(d.get(), &ok, sizeof(int), cudaMemcpyHostToDevice));
		NC(g_nccl.AllReduce(d.get(), d.get(), 1, ncclInt32, ncclMin, ctx->comm, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
		int all_ok = 0;
		CU(cudaMemcpy(&all_ok, d.get(), sizeof(int), cudaMemcpyDeviceToHost));
		if (!all_ok) {
			if (!ok) fprintf(stderr, "tgpu: rank %d cannot use the peer-to-peer halo exchange (%s)\n", me, why.c_str());
			if (me == 0) fprintf(stderr, "tgpu: peer-to-peer mapping unavailable on at least one rank: using the NCCL send/recv halo exchange\n");
			h->ipc_opened.clear();
			h->arena.reset();
			h->p2p_abort.reset();
			return TGPU_OK; // L.p2p stays false on every level
		}
	}
	// ---- per level: move the face buffers into the arena, exchange the halo-slot numbering, build the tables ----
	for (int l = 0; l < nl; l++) {
		LevelDev &       L  = h->levels[l];
		const PartLevel &PL = pt.levels[l];
		if (!L.distributed || (L.nsend == 0 && L.nrecv == 0)) continue;
		L.Fa_own.reset(), L.Fb_own.reset();
		L.Fa         = (double *) ((char *) h->arena.get() + mine.fa_off[l]);
		L.Fb         = (double *) ((char *) h->arena.get() + mine.fb_off[l]);
		L.data_flags = (uint64_t *) ((char *) h->arena.get() + mine.flags_off) + ((size_t) l * 2 + 0) * nr;
		L.ack_flags  = (uint64_t *) ((char *) h->arena.get() + mine.flags_off) + ((size_t) l * 2 + 1) * nr;
		CU(dev_malloc(L.cnt, 4 * sizeof(uint64_t)));
		CU(cudaMemset(L.cnt.get(), 0, 4 * sizeof(uint64_t)));
		CU(dev_malloc(L.tickets, 2 * sizeof(unsigned)));
		CU(cudaMemset(L.tickets.get(), 0, 2 * sizeof(unsigned)));
		const int np = (int) L.peers.size();
		// my halo slots as the peers see them: they send (slot, side) lists in the agreed order
		DevPtr<int32_t> d_rslot;
		CU(dev_malloc(d_rslot, std::max<size_t>(1, L.nsend) * sizeof(int32_t)));
		NC(g_nccl.GroupStart());
		for (const PeerDev &pd : L.peers) {
			if (pd.recv_n) NC(g_nccl.Send(L.recv_slot.get() + pd.recv_off, pd.recv_n, ncclInt32, pd.peer, ctx->comm, ctx->stream));
			if (pd.send_n) NC(g_nccl.Recv(d_rslot.get() + pd.send_off, pd.send_n, ncclInt32, pd.peer, ctx->comm, ctx->stream));
		}
		NC(g_nccl.GroupEnd());
		CU(cudaStreamSynchronize(ctx->stream));
		std::vector<int32_t> rslot(L.nsend), ridx(L.nsend), speer(L.nsend), prank(np);
		if (L.nsend) CU(cudaMemcpy(rslot.data(), d_rslot.get(), L.nsend * sizeof(int32_t), cudaMemcpyDeviceToHost));
		std::vector<double *>   pfa(np), pfb(np);
		std::vector<uint64_t *> pdf(np), paf(np);
		size_t                  k = 0;
		for (int i = 0; i < np; i++) {
			const PeerDev &     pd = L.peers[i];
			const PeerExchange &x  = PL.peers[i];
			prank[i]               = pd.peer;
			char *ra               = rarena[pd.peer];
			pfa[i]                 = (double *) (ra + all[pd.peer].fa_off[l]);
			pfb[i]                 = (double *) (ra + all[pd.peer].fb_off[l]);
			uint64_t *rflags       = (uint64_t *) (ra + all[pd.peer].flags_off);
			pdf[i]                 = rflags + ((size_t) l * 2 + 0) * nr + me;
			paf[i]                 = rflags + ((size_t) l * 2 + 1) * nr + me;
			for (size_t j = 0; j < pd.send_n; j++, k++) {
				speer[k] = i;
				ridx[k]  = rslot[k] * S + x.send_side[j];
			}
		}
		TRY(dev_upload(L.send_peer, speer.data(), speer.size()));
		TRY(dev_upload(L.send_ridx, ridx.data(), ridx.size()));
		TRY(dev_upload(L.peer_rank, prank.data(), prank.size()));
		TRY(dev_upload(L.peerFa, pfa.data(), pfa.size()));
		TRY(dev_upload(L.peerFb, pfb.data(), pfb.size()));
		TRY(dev_upload(L.peer_data_flag, pdf.data(), pdf.size()));
		TRY(dev_upload(L.peer_ack_flag, paf.data(), paf.size()));
		L.p2p = true;
	}
	// nobody may push before everybody has finished mapping
	{
		DevPtr<int> d;
		CU(dev_malloc(d, sizeof(int)));
		CU(cudaMemset(d.get(), 0, sizeof(int)));
		NC(g_nccl.AllReduce(d.get(), d.get(), 1, ncclInt32, ncclSum, ctx->comm, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
	}
	return TGPU_OK;
}
extern "C" int tgpu_hierarchy_create_distributed(tgpu_ctx *ctx, const tgpu_part *part, tgpu_hier **out)
{
	API_BEGIN
	if (!ctx || !part || !out) return fail(TGPU_ERR_ARG, "null argument");
	const Partition &pt = part->part;
	if (pt.nranks > 1 && (!ctx->comm || ctx->nranks != pt.nranks || ctx->rank != pt.rank))
		return fail(TGPU_ERR_ARG, "tgpu_hierarchy_create_distributed: call tgpu_comm_init with the partition's rank/nranks first");
	std::vector<int32_t> owned;
	for (const PartLevel &L : pt.levels) owned.push_back(L.n_owned);
	std::unique_ptr<tgpu_hier> h;
	TRY(hierarchy_create_impl(ctx, pt.D, pt.n, (int) pt.levels.size(), part->descs.data(), owned.data(), h));
	size_t M = 1;
	for (int i = 0; i < pt.D - 1; i++) M *= pt.n;
	for (size_t l = 0; l < pt.levels.size(); l++) {
		const PartLevel &PL = pt.levels[l];
		LevelDev &       L  = h->levels[l];
		L.distributed       = PL.distributed;
		L.n_interior        = PL.n_interior;
		if (PL.distributed && l < pt.owner.size()) L.global_P = (int64_t) pt.owner[l].size();
		for (int e = 0; e < 4; e++) CU(event_create(L.ev[e], cudaEventDisableTiming));
		std::vector<int32_t> sp, ss, rs, rsd;
		for (const PeerExchange &x : PL.peers) {
			PeerDev pd;
			pd.peer     = x.peer;
			pd.send_off = sp.size(), pd.send_n = x.send_patch.size();
			pd.recv_off = rs.size(), pd.recv_n = x.recv_slot.size();
			sp.insert(sp.end(), x.send_patch.begin(), x.send_patch.end());
			ss.insert(ss.end(), x.send_side.begin(), x.send_side.end());
			rs.insert(rs.end(), x.recv_slot.begin(), x.recv_slot.end());
			rsd.insert(rsd.end(), x.recv_side.begin(), x.recv_side.end());
			L.peers.push_back(pd);
		}
		L.nsend = sp.size(), L.nrecv = rs.size();
		if (L.nsend) {
			TRY(dev_upload(L.send_patch, sp.data(), sp.size()));
			TRY(dev_upload(L.send_side, ss.data(), ss.size()));
			CU(dev_malloc(L.sendbuf, L.nsend * M * sizeof(double)));
		}
		if (L.nrecv) {
			TRY(dev_upload(L.recv_slot, rs.data(), rs.size()));
			TRY(dev_upload(L.recv_side, rsd.data(), rsd.size()));
			CU(dev_malloc(L.recvbuf, L.nrecv * M * sizeof(double)));
		}
		// halo slots must never hold NaN garbage before the first exchange
		CU(cudaMemset(L.Fa, 0, L.nface * sizeof(double)));
		CU(cudaMemset(L.Fb, 0, L.nface * sizeof(double)));
	}
	// TGPU_P2P=0 keeps the NCCL send/recv exchange (pack, ncclSend/ncclRecv, unpack)
	const char *e = getenv("TGPU_P2P");
	if (pt.nranks > 1 && !(e && atoi(e) == 0)) TRY(setup_p2p(h.get(), pt));
	*out = h.release();
	return TGPU_OK;
	API_END
}

extern "C" int tgpu_hierarchy_destroy(tgpu_hier *h)
{
	delete h;
	return TGPU_OK;
}
// Gives the memory of everything the library allocated lazily on behalf of earlier calls back to the device: Krylov work
// vectors, the host-buffer slots of tgpu_vcycle_host / _async, cached cycle graphs, the vector pool's free blocks.  The
// neighbour tables, face buffers and per-level cycle vectors stay.
extern "C" int tgpu_hierarchy_trim(tgpu_hier *h)
{
	API_BEGIN
	if (!h) return fail(TGPU_ERR_ARG, "null hierarchy");
	tgpu_ctx *ctx = h->ctx;
	CU(cudaSetDevice(ctx->device));
	if (h->s_in) CU(cudaStreamSynchronize(h->s_in.get()));
	if (h->s_out) CU(cudaStreamSynchronize(h->s_out.get()));
	CU(cudaStreamSynchronize(ctx->stream));
	h->release_workspace();
	h->pipe_count = 0;
	CU(cudaStreamSynchronize(ctx->stream));
	cudaMemPool_t pool = nullptr;
	CU(cudaDeviceGetDefaultMemPool(&pool, ctx->device));
	CU(cudaMemPoolTrimTo(pool, 0));
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_hierarchy_info(const tgpu_hier *h, int *D, int *n, int *nlevels)
{
	if (!h) return fail(TGPU_ERR_ARG, "null hierarchy");
	if (D) *D = h->D;
	if (n) *n = h->N;
	if (nlevels) *nlevels = (int) h->levels.size();
	return TGPU_OK;
}
// After either call: the cached graphs are dropped, the multiplier tables follow the Helmholtz state (upload_tri), and the
// buffers of the patch solve paths the new state takes exist.
static int shifts_changed(tgpu_hier *h)
{
	h->graphs.clear();
	TRY(ensure_scratch32(h));
	TRY(upload_tri(h));
	return update_iface_buffers(h);
}
// FftwPatchSolver(domain, lambda) / DftPatchSolver(domain, lambda) (PatchSolvers/FftwPatchSolver.h:66,170,
// DftPatchSolver.h:78,168): the block-Jacobi patch problems become (Laplacian + lambda) u = rhs.  As in the reference the
// shift lives in the patch solver only; the operator (StarPatchOp) keeps the shift of tgpu_hierarchy_set_helmholtz.
extern "C" int tgpu_hierarchy_set_lambda(tgpu_hier *h, double lambda)
{
	if (!h) return fail(TGPU_ERR_ARG, "null argument");
	if (!(lambda == lambda)) return fail(TGPU_ERR_ARG, "tgpu_hierarchy_set_lambda: lambda is NaN");
	h->lambda = lambda;
	return shifts_changed(h);
}
// Helmholtz operator A + lambda I on every level, with the same patch solver shift: the sweeps solve the shifted patch
// problems exactly, so every kernel and schedule of the Poisson problem applies (DESIGN §3.8).
extern "C" int tgpu_hierarchy_set_helmholtz(tgpu_hier *h, double lambda)
{
	if (!std::isfinite(lambda) || lambda > 0.0)
		return fail(TGPU_ERR_ARG, "tgpu_hierarchy_set_helmholtz: lambda must be finite and <= 0");
	if (!h) return fail(TGPU_ERR_ARG, "null argument");
	if (lambda != 0.0 && h->tab_overflow)
		return fail(TGPU_ERR_UNSUPPORTED, "tgpu_hierarchy_set_helmholtz: the hierarchy has more than 256 distinct cell sizes");
	h->op_shift = h->lambda = lambda;
	return shifts_changed(h);
}
extern "C" int tgpu_hierarchy_force_generic_kernels(tgpu_hier *h, int on)
{
	if (!h) return fail(TGPU_ERR_ARG, "null argument");
	h->generic_kernels = on != 0;
	h->graphs.clear();
	return TGPU_OK;
}
extern "C" int tgpu_level_npatch(const tgpu_hier *h, int level, int64_t *npatch, int64_t *ncells)
{
	if (!h || level < 0 || level >= (int) h->levels.size()) return fail(TGPU_ERR_ARG, "bad level");
	if (npatch) *npatch = h->levels[level].P;
	if (ncells) *ncells = (int64_t) h->levels[level].ncells;
	return TGPU_OK;
}

// ------------------------------------------------------------------------------------------
// vectors
// ------------------------------------------------------------------------------------------
// Vector storage comes from the device's stream-ordered pool (cudaMallocAsync / cudaFreeAsync on the library's stream):
// creating and destroying temporaries - the reference allocates three vectors per level per cycle (GMG/Cycle.h:59-64)
// and a caller driving the API-granular plugin classes does the same - costs neither a device synchronisation nor a
// trip to the driver's allocator once the pool is warm.
extern "C" int tgpu_vec_create(tgpu_hier *h, int level, tgpu_vec **out)
{
	if (!h || !out || level < 0 || level >= (int) h->levels.size()) return fail(TGPU_ERR_ARG, "tgpu_vec_create: bad argument");
	CU(cudaSetDevice(h->ctx->device));
	std::unique_ptr<tgpu_vec> v(new tgpu_vec());
	v->h     = h;
	v->level = level;
	v->n     = h->levels[level].ncells;
	CU(cudaMallocAsync(&v->d, std::max<size_t>(1, v->n) * sizeof(double), h->ctx->stream));
	CU(cudaMemsetAsync(v->d, 0, v->n * sizeof(double), h->ctx->stream));
	*out = v.release();
	return TGPU_OK;
}
// tgpu_vec_create into an owner: the work vectors a hierarchy keeps for itself
static int vec_create(tgpu_hier *h, int level, VecPtr &v)
{
	tgpu_vec *raw = nullptr;
	TRY(tgpu_vec_create(h, level, &raw));
	v.reset(raw);
	return TGPU_OK;
}
extern "C" int tgpu_vec_destroy(tgpu_vec *v)
{
	if (!v) return TGPU_OK;
	tgpu_hier *h = v->h;
	// cached cycle graphs that were captured on this storage are dropped; graphs of other vectors stay
	for (size_t i = 0; i < h->graphs.size();) {
		if (h->graphs[i].f == v->d || h->graphs[i].u == v->d || h->graphs[i].b == v->d) h->graphs.erase(h->graphs.begin() + i);
		else i++;
	}
	cudaFreeAsync(v->d, h->ctx->stream); // stream-ordered: work already queued on the vector completes first
	delete v;
	return TGPU_OK;
}
extern "C" int tgpu_vec_upload(tgpu_vec *v, const double *host)
{
	if (!v || !host) return fail(TGPU_ERR_ARG, "null argument");
	CU(cudaMemcpyAsync(v->d, host, v->n * sizeof(double), cudaMemcpyHostToDevice, v->h->ctx->stream));
	CU(cudaStreamSynchronize(v->h->ctx->stream));
	return TGPU_OK;
}
extern "C" int tgpu_vec_download(const tgpu_vec *v, double *host)
{
	if (!v || !host) return fail(TGPU_ERR_ARG, "null argument");
	CU(cudaMemcpyAsync(host, v->d, v->n * sizeof(double), cudaMemcpyDeviceToHost, v->h->ctx->stream));
	CU(cudaStreamSynchronize(v->h->ctx->stream));
	return check_comm(v->h->ctx);
}
extern "C" int tgpu_vec_upload_async(tgpu_vec *v, const double *host)
{
	if (!v || !host) return fail(TGPU_ERR_ARG, "null argument");
	CU(cudaMemcpyAsync(v->d, host, v->n * sizeof(double), cudaMemcpyHostToDevice, v->h->ctx->stream));
	return TGPU_OK;
}
extern "C" int tgpu_vec_download_async(const tgpu_vec *v, double *host)
{
	if (!v || !host) return fail(TGPU_ERR_ARG, "null argument");
	CU(cudaMemcpyAsync(host, v->d, v->n * sizeof(double), cudaMemcpyDeviceToHost, v->h->ctx->stream));
	return TGPU_OK;
}
extern "C" int tgpu_vec_device_ptr(const tgpu_vec *v, void **dptr, int64_t *ncells)
{
	if (!v) return fail(TGPU_ERR_ARG, "null vector");
	if (dptr) *dptr = v->d;
	if (ncells) *ncells = (int64_t) v->n;
	return TGPU_OK;
}
extern "C" int tgpu_host_alloc(size_t bytes, void **p)
{
	if (!p) return fail(TGPU_ERR_ARG, "null argument");
	CU(cudaMallocHost(p, bytes));
	return TGPU_OK;
}
extern "C" int tgpu_host_free(void *p)
{
	CU(cudaFreeHost(p));
	return TGPU_OK;
}

static int same_shape(const tgpu_vec *a, const tgpu_vec *b)
{
	if (!a || !b) return fail(TGPU_ERR_ARG, "null vector");
	if (a->h != b->h || a->level != b->level || a->n != b->n)
		return fail(TGPU_ERR_ARG, "vectors belong to different levels/hierarchies");
	return TGPU_OK;
}
template <int OP>
static int blas1(tgpu_vec *v, const tgpu_vec *a, const tgpu_vec *b, double alpha, double beta, double gamma)
{
	if (!v) return fail(TGPU_ERR_ARG, "null vector");
	if (a) TRY(same_shape(v, a));
	if (b) TRY(same_shape(v, b));
	tgpu_ctx *ctx = v->h->ctx;
	Tag       tg(ctx, "blas1", v->level);
	return launch(ctx, blas1_kernel<OP>, dim3(grid_for(ctx, v->n)), dim3(256), 0, v->n, v->d, a ? a->d : (const double *) nullptr,
	              b ? b->d : (const double *) nullptr, alpha, beta, gamma);
}
extern "C" int tgpu_vec_set(tgpu_vec *v, double alpha) { return blas1<B_SET>(v, nullptr, nullptr, alpha, 0, 0); }
extern "C" int tgpu_vec_scale(tgpu_vec *v, double alpha) { return blas1<B_SCALE>(v, nullptr, nullptr, alpha, 0, 0); }
extern "C" int tgpu_vec_shift(tgpu_vec *v, double delta) { return blas1<B_SHIFT>(v, nullptr, nullptr, delta, 0, 0); }
extern "C" int tgpu_vec_copy(tgpu_vec *v, const tgpu_vec *b) { return b ? blas1<B_COPY>(v, b, nullptr, 0, 0, 0) : fail(TGPU_ERR_ARG, "null vector"); }
extern "C" int tgpu_vec_add(tgpu_vec *v, const tgpu_vec *b) { return b ? blas1<B_ADD>(v, b, nullptr, 0, 0, 0) : fail(TGPU_ERR_ARG, "null vector"); }
extern "C" int tgpu_vec_add_scaled(tgpu_vec *v, double alpha, const tgpu_vec *b)
{
	return b ? blas1<B_AXPY>(v, b, nullptr, alpha, 0, 0) : fail(TGPU_ERR_ARG, "null vector");
}
extern "C" int tgpu_vec_add_scaled2(tgpu_vec *v, double alpha, const tgpu_vec *a, double beta, const tgpu_vec *b)
{
	return (a && b) ? blas1<B_AXPBY2>(v, a, b, alpha, beta, 0) : fail(TGPU_ERR_ARG, "null vector");
}
extern "C" int tgpu_vec_scale_then_add(tgpu_vec *v, double alpha, const tgpu_vec *b)
{
	return b ? blas1<B_SCALE_ADD>(v, b, nullptr, alpha, 0, 0) : fail(TGPU_ERR_ARG, "null vector");
}
extern "C" int tgpu_vec_scale_then_add_scaled(tgpu_vec *v, double alpha, double beta, const tgpu_vec *b)
{
	return b ? blas1<B_SCALE_ADDS>(v, b, nullptr, alpha, beta, 0) : fail(TGPU_ERR_ARG, "null vector");
}
extern "C" int tgpu_vec_scale_then_add_scaled2(tgpu_vec *v, double alpha, double beta, const tgpu_vec *b, double gamma,
                                               const tgpu_vec *c)
{
	return (b && c) ? blas1<B_SCALE_ADDS2>(v, b, c, alpha, beta, gamma) : fail(TGPU_ERR_ARG, "null vector");
}

template <int OP> static int reduce(const tgpu_vec *a, const tgpu_vec *b, double *result)
{
	if (!a || !b || !result) return fail(TGPU_ERR_ARG, "null argument");
	TRY(same_shape(a, b));
	tgpu_ctx *ctx = a->h->ctx;
	const int nb  = std::min(MAX_PARTIAL, grid_for(ctx, a->n, 256, 8));
	Tag       tg(ctx, "reduce", a->level);
	TRY(launch(ctx, reduce_stage1<OP>, dim3(nb), dim3(256), 0, a->n, (const double *) a->d, (const double *) b->d, ctx->d_partial.get()));
	TRY(launch(ctx, reduce_stage2<OP>, dim3(1), dim3(256), 0, nb, (const double *) ctx->d_partial.get(), ctx->d_result.get()));
	// (boundary data is split over the ranks like level 0)
	if (ctx->nranks > 1 && a->h->levels[std::max(a->level, 0)].distributed)
		NC(g_nccl.AllReduce(ctx->d_result.get(), ctx->d_result.get(), 1, ncclDouble, OP == 0 ? ncclSum : ncclMax, ctx->comm, ctx->stream));
	CU(cudaMemcpyAsync(ctx->h_result.get(), ctx->d_result.get(), sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	*result = ctx->h_result.get()[0];
	return check_comm(ctx);
}
extern "C" int tgpu_vec_dot(const tgpu_vec *v, const tgpu_vec *b, double *result) { return reduce<0>(v, b, result); }
extern "C" int tgpu_vec_two_norm(const tgpu_vec *v, double *result)
{
	double s = 0;
	TRY(reduce<0>(v, v, &s));
	*result = sqrt(s);
	return TGPU_OK;
}
extern "C" int tgpu_vec_inf_norm(const tgpu_vec *v, double *result) { return reduce<1>(v, v, result); }

// ------------------------------------------------------------------------------------------
// level operators (raw-pointer versions used by the cycle + vector-checked API wrappers)
// ------------------------------------------------------------------------------------------
static int check_level_vec(const tgpu_hier *h, int level, const tgpu_vec *v, const char *what)
{
	if (!h || !v) return fail(TGPU_ERR_ARG, std::string(what) + ": null argument");
	if (level < 0 || level >= (int) h->levels.size()) return fail(TGPU_ERR_ARG, std::string(what) + ": bad level");
	if (v->h != h || v->level != level) return fail(TGPU_ERR_ARG, std::string(what) + ": vector does not live on this level");
	return TGPU_OK;
}

// consumer side of the hand-over for kernels that poll the DATA flags themselves and acknowledge from their last CTA
static bool halo_in_kernel(const tgpu_hier *h, int l)
{
	static const bool off = getenv("TGPU_HALO_IN_KERNEL") && atoi(getenv("TGPU_HALO_IN_KERNEL")) == 0;
	const LevelDev &  L   = h->levels[l];
	return !off && L.p2p && specialised(h) && !h->generic_kernels && !L.has_neumann && consistent(h);
}
// producer side folded into the consumer kernel as well (halo_push_cta): no separate push launch
static bool push_in_kernel(const tgpu_hier *h, int l)
{
	static const bool off = getenv("TGPU_PUSH_IN_KERNEL") && atoi(getenv("TGPU_PUSH_IN_KERNEL")) == 0;
	return !off && halo_in_kernel(h, l);
}
// the four push descriptors of a level: index (F == Fb ? 2 : 0) + (with the prolonged correction of level l + 1's u ? 1 : 0)
static int ensure_push_desc(tgpu_hier *h, int l)
{
	LevelDev &L = h->levels[l];
	const double *ucv = l + 1 < (int) h->levels.size() ? h->levels[l + 1].u.get() : nullptr;
	if (!L.p2p || (L.push_desc && L.push_uc == ucv)) return TGPU_OK;
	PushDesc d[4];
	for (int i = 0; i < 4; i++) {
		d[i].patch          = L.send_patch.get();
		d[i].side           = L.send_side.get();
		d[i].peer_of        = L.send_peer.get();
		d[i].ridx           = L.send_ridx.get();
		d[i].F              = (i & 2) ? L.Fb : L.Fa;
		d[i].uc             = (i & 1) ? ucv : nullptr;
		d[i].peerF          = (i & 2) ? L.peerFb.get() : L.peerFa.get();
		d[i].ack_flags      = L.ack_flags;
		d[i].peer_rank      = L.peer_rank.get();
		d[i].peer_data_flag = L.peer_data_flag.get();
		d[i].cnt            = L.cnt.get();
		d[i].ticket         = L.tickets.get();
		d[i].abort          = h->p2p_abort.get();
		d[i].host_err       = (int *) h->ctx->p2p_err.get();
		d[i].nfaces         = (int) L.nsend;
		d[i].npeers         = (int) L.peers.size();
	}
	if (!L.push_desc) CU(dev_malloc(L.push_desc, sizeof(d)));
	CU(cudaMemcpy(L.push_desc.get(), d, sizeof(d), cudaMemcpyHostToDevice));
	L.push_uc = ucv;
	return TGPU_OK;
}
// pushF != nullptr: the consumer launch first pushes this rank's faces pushF (+ the prolonged correction if with_uc)
static HaloSync halo_sync(tgpu_hier *h, int l, const double *pushF = nullptr, bool with_uc = false)
{
	LevelDev &L = h->levels[l];
	HaloSync  hs;
	if (pushF && L.push_desc) hs.push = L.push_desc.get() + ((pushF == L.Fb ? 2 : 0) + (with_uc ? 1 : 0));
	hs.data_flags       = L.data_flags;
	hs.peer_rank        = L.peer_rank.get();
	hs.peer_ack_flag    = L.peer_ack_flag.get();
	hs.cnt              = L.cnt.get();
	hs.ticket           = L.tickets.get() + 1;
	hs.abort            = h->p2p_abort.get();
	hs.host_err         = (int *) h->ctx->p2p_err.get();
	hs.npeers           = (int) L.peers.size();
	hs.first_halo_patch = L.n_interior;
	hs.enabled          = 1;
	return hs;
}
static int k_extract_faces(tgpu_hier *h, int l, const double *u, double *F)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, "extract_faces", l);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, extract_faces_kernel<DD, NN>, dim3(grid_for(h->ctx, L.nface)), dim3(256), 0, L.P, u, F));
}
// mode 0: out = A u; 1: out = f - A u; 2: coarse = R (f - A u).  F must hold the faces of u.
// mode 3: out = A u with the block partial sums of out . f and out . out written to ctx->d_partial.get() ([0..nb),
// [MAX_PARTIAL / 2 ..)); *nb_out = number of partials
static int k_apply(tgpu_hier *h, int l, int mode, const double *u, const double *f, const double *F, double *out, double *coarse,
                   int p0 = 0, int p1 = -1, int *nb_out = nullptr)
{
	LevelDev &L = h->levels[l];
	if (p1 < 0) p1 = L.P;
	if (p1 <= p0) return TGPU_OK;
	Tag       tg(h->ctx, mode == 0 ? "apply" : (mode == 1 ? "residual" : (mode == 2 ? "residual_restrict" : "apply_dots")), l);
	double *const  part    = h->ctx->d_partial.get();
	constexpr int  pstride = MAX_PARTIAL / 2;
	if (is_3d32(h)) { // mode 2: f - A u into L.r.get(), then the restriction
		if (mode == 2 && (p0 != 0 || p1 != L.P)) return fail(TGPU_ERR_UNSUPPORTED, "residual+restrict on a patch range is not available for 32^3 patches");
		const dim3 grid(std::min((p1 - p0) * 4, h->ctx->sm_count * 2));
		if (nb_out) *nb_out = (int) grid.x;
		auto go = [&](auto kernel, double *o) {
			return launch(h->ctx, kernel, grid, dim3(TGPU_THREADS), apply3d32_tma_smem_bytes(), (const PatchMeta *) L.meta.get(), p0, p1, u, f, F, o, part, pstride, h->op_shift);
		};
		if (mode == 0) return go(apply3d32_tma_kernel<0>, out);
		if (mode == 3) return go(apply3d32_tma_kernel<3>, out);
		if (mode == 1) return go(apply3d32_tma_kernel<1>, out);
		TRY(go(apply3d32_tma_kernel<1>, L.r.get()));
		return launch(h->ctx, restrict_kernel<3, 32>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, (const double *) L.r.get(), coarse);
	}
	DISPATCH_DN(h->D, h->N, {
		using G        = Geo<DD, NN>;
		const int nblk = (p1 - p0 + G::PPB - 1) / G::PPB;
		const int grid = std::min(nblk, h->ctx->sm_count * 2);
		if (nb_out) *nb_out = grid;
		auto go = [&](auto kernel) {
			return launch(h->ctx, kernel, dim3(grid), dim3(TGPU_THREADS), apply_tma_smem_bytes<DD, NN>(), (const PatchMeta *) L.meta.get(), p0, p1, u, f, F, out, coarse, part, pstride, h->op_shift);
		};
		if (mode == 0) return go(apply_tma_kernel<DD, NN, 0>);
		if (mode == 1) return go(apply_tma_kernel<DD, NN, 1>);
		if (mode == 3) return go(apply_tma_kernel<DD, NN, 3>);
		return go(apply_tma_kernel<DD, NN, 2>);
	});
}
// zero_guess: gamma = 0 (Fin unused); emit: write the faces of the new u to Fout;
// uc != nullptr: face values are Fin + (P uc) on the boundary cells (fused prolongation);
// write_u = false (needs emit): only the faces of the new u are wanted (the generic kernel still writes u)
// neu: the instantiation for the patches with Neumann domain sides (it sweeps exactly those of the range)
template <bool Z, bool E, bool PR, bool W>
static int launch_smooth3d16(tgpu_hier *h, const LevelDev &L, int p0, int p1, const double *f, double *u, const double *Fin, double *Fout,
                             const double *uc, HaloSync hs = HaloSync{}, int skip_neumann = 0, bool neu = false)
{
	if (neu) {
		if (hs.enabled) return fail(TGPU_ERR_ARG, "smooth3d16: the Neumann instantiation is single-GPU");
		// the patches of [p0, p1) with Neumann sides: a contiguous piece of the level's (ascending) list
		const auto b0 = std::lower_bound(L.neu_host.begin(), L.neu_host.end(), p0), b1 = std::lower_bound(L.neu_host.begin(), L.neu_host.end(), p1);
		const int  nn = (int) (b1 - b0);
		if (nn == 0) return TGPU_OK;
		const dim3 gridn(std::min(nn, h->ctx->sm_count * s16_ctas_per_sm(Z, true))), blockn(S16_BLOCK);
		return launch(h->ctx, smooth3d16_kernel<Z, E, PR, W, false, true>, gridn, blockn, smooth3d16_smem_bytes(), (const PatchMeta *) L.meta.get(), p0,
		              p1, f, u, Fin, Fout, (const double *) h->tri.get(), uc, HaloSync{}, 0,
		              NeuTabs{h->mats.get(), h->lam.get(), L.neu_list.get() + (b0 - L.neu_host.begin()), nn, helmholtz(h), h->lambda});
	}
	const dim3 grid(std::min(p1 - p0, h->ctx->sm_count * s16_ctas_per_sm(Z))), block(S16_BLOCK);
	if (hs.enabled) {
		if (Z) return fail(TGPU_ERR_ARG, "smooth3d16: no halo hand-over in a zero-guess sweep");
		return halo_launch(h->ctx, hs, smooth3d16_kernel<Z, E, PR, W, !Z>, grid, block, smooth3d16_smem_bytes(), (const PatchMeta *) L.meta.get(), p0, p1,
		                   f, u, Fin, Fout, (const double *) h->tri.get(), uc, hs, skip_neumann, NeuTabs{});
	}
	return launch(h->ctx, smooth3d16_kernel<Z, E, PR, W>, grid, block, smooth3d16_smem_bytes(), (const PatchMeta *) L.meta.get(), p0, p1, f, u, Fin,
	              Fout, (const double *) h->tri.get(), uc, hs, skip_neumann, NeuTabs{});
}
// hsp != nullptr (multi-GPU, kernels that support it: halo_in_kernel): the launch covers interior and boundary patches and
// does the halo hand-over itself
static int k_smooth(tgpu_hier *h, int l, bool zero_guess, bool emit, const double *f, double *u, const double *Fin, double *Fout,
                    const double *uc = nullptr, int p0 = 0, int p1 = -1, bool write_u = true, const HaloSync *hsp = nullptr)
{
	const HaloSync hs = hsp ? *hsp : HaloSync{};
	if (hsp && !halo_in_kernel(h, l)) return fail(TGPU_ERR_ARG, "k_smooth: in-kernel halo hand-over is not available for this level");
	LevelDev &L = h->levels[l];
	if (p1 < 0) p1 = L.P;
	if (p1 <= p0) return hs.push ? fail(TGPU_ERR_ARG, "k_smooth: a launch that pushes faces needs patches") : TGPU_OK;
	if (!emit) write_u = true;
	Tag tg(h->ctx, zero_guess ? (write_u ? "smooth_zero_guess" : "smooth_zero_guess_faces")
	                          : (uc ? (write_u ? "smooth_prolong" : "smooth_prolong_faces") : (write_u ? "smooth" : "smooth_faces")),
	       l);
	const bool prolong = uc != nullptr;
	const PatchMeta *meta = L.meta.get();
	// A mixed level: the general path sweeps the patches of the range with Neumann domain sides, the specialised kernel skips
	// them and sweeps the others (two launches, disjoint patches).  A smoother-only shift sends every patch through the general
	// path; in the Helmholtz state the Dirichlet patches read their shifted tables.
	const bool mixed = specialised(h) && L.has_neumann && !shifted_smoother(h) && !hsp;
	if (!specialised(h) || L.has_neumann || shifted_smoother(h)) { // the size's general path: the whole range, or its Neumann patches
		if (is_3d32(h)) { // general transform path through an L2-resident scratch block
			const int nblk = std::min(p1 - p0, h->ctx->sm_count * 2);
			if (!h->scratch32) return fail(TGPU_ERR_ARG, "k_smooth: scratch for the general 32^3 patch solve missing");
			TRY(launch(h->ctx, smooth3d32n_kernel, dim3(nblk), dim3(TGPU_THREADS), 0, meta, p0, p1, f, u, Fin, Fout, uc, (const double *) h->mats.get(),
			           (const double *) h->lam.get(), h->scratch32.get(), (int) zero_guess, (int) emit, (int) prolong, (int) write_u, h->lambda, (int) mixed,
			           helmholtz(h)));
		} else if (mixed && h->D == 3 && h->N == 16) { // the Neumann instantiation of the specialised kernel
			TRY(smooth_variant(zero_guess, emit, prolong, write_u, [&](auto Z, auto E, auto PR, auto W) {
				return launch_smooth3d16<Z, E, PR, W>(h, L, p0, p1, f, u, Fin, Fout, uc, HaloSync{}, 0, true);
			}));
		} else { // smooth_kernel (size-generic; it always writes u)
			DISPATCH_DN(h->D, h->N, {
				using G          = Geo<DD, NN>;
				const int    nblk = (p1 - p0 + G::PPB - 1) / G::PPB;
				const dim3   grid(std::min(nblk, h->ctx->sm_count * smooth_min_blocks<NN>())), block(TGPU_THREADS);
				const size_t sm = smooth_smem_bytes<DD, NN, true>();
				TRY(smooth_variant(zero_guess, emit, prolong, write_u, [&](auto Z, auto E, auto PR, auto) {
					return launch(h->ctx, smooth_kernel<DD, NN, Z, E, PR>, grid, block, sm, meta, p0, p1, f, u, Fin, Fout, (const double *) h->tri.get(), uc,
					              (const double *) h->mats.get(), (const double *) h->lam.get(), h->lambda, (int) mixed, helmholtz(h));
				}));
			});
		}
		if (!mixed) return TGPU_OK;
		if (is_3d32(h) && L.neu_host.size() == (size_t) L.P) return TGPU_OK; // (every owned patch has Neumann sides: nothing left)
	}
	const int skipn = mixed ? 1 : 0;
	if (is_3d32(h)) {
		if (!zero_guess) {
			// the interface part of the right-hand side, transformed for the sweep (and the halo hand-over, which it consumes)
			if (!L.G) return fail(TGPU_ERR_ARG, "k_smooth: interface-term buffer of the 32^3 level missing");
			// over the slots the patches [p0, p1) own (IfaceSlots32), one warp per slot; at least one CTA, which does the
			// hand-over when the range owns none
			Tag          ti(h->ctx, "iface_rhs", l);
			const int    k0 = L.gbegin[p0], k1 = L.gbegin[p1];
			const dim3   gi(std::max(1, std::min((k1 - k0 + IR32_WARPS - 1) / IR32_WARPS, h->ctx->sm_count * IR32_CTAS_PER_SM))), bi(IR32_THREADS);
			const int32_t *own = L.gowner.get();
			TRY(flag_variant(prolong, hs.enabled, [&](auto PR, auto HALO) {
				return halo_launch(h->ctx, hs, iface_rhs32_kernel<PR, HALO>, gi, bi, iface_rhs32_smem_bytes(), meta, own, k0, k1, Fin, uc, L.G.get(), hs);
			}));
		} else if (hs.enabled) {
			return fail(TGPU_ERR_ARG, "smooth3d32c: no halo hand-over in a zero-guess sweep");
		}
		// one cluster of two CTAs (two SMs) per patch, see smooth3d32c_kernel
		const dim3 grid(2 * std::min(p1 - p0, h->ctx->sm_count / 2)), block(C32_THREADS);
		return smooth_variant(zero_guess, emit, prolong, write_u, [&](auto Z, auto E, auto, auto W) {
			return launch(h->ctx, smooth3d32c_kernel<Z, E, W>, grid, block, smooth3d32c_smem_bytes<Z>(), meta, p0, p1, f, u,
			              (const double *) L.G.get(), Fout, (const double *) h->tri.get(), skipn, (const int32_t *) L.gslot.get());
		});
	}
	if (h->D == 3)
		return smooth_variant(zero_guess, emit, prolong, write_u, [&](auto Z, auto E, auto PR, auto W) {
			return launch_smooth3d16<Z, E, PR, W>(h, L, p0, p1, f, u, Fin, Fout, uc, hs, skipn);
		});
	// 2-D 32^2: one warp per patch, see smooth2d32.cuh
	const int  nblk = (p1 - p0 + Q32_WARPS - 1) / Q32_WARPS;
	const dim3 grid(std::min(nblk, h->ctx->sm_count * 2)), block(TGPU_THREADS);
	return smooth_variant(zero_guess, emit, prolong, write_u, [&](auto Z, auto E, auto PR, auto W) {
		return flag_variant(mixed || hs.enabled, [&](auto EXTRA) {
			return halo_launch(h->ctx, hs, smooth2d32_kernel<Z, E, PR, W, EXTRA>, grid, block, smooth2d32_smem_bytes(), meta, p0, p1, f, u, Fin, Fout,
			                   (const double *) h->tri.get(), uc, hs, skipn);
		});
	});
}
// coarse = R (f - A u) for a u that a block-Jacobi sweep has just produced: needs only the faces of the new
// (Fnew) and, unless the sweep started from zero (Fold == nullptr), the previous (Fold) iterate
static int k_face_residual_restrict(tgpu_hier *h, int l, const double *Fnew, const double *Fold, double *coarse, int p0 = 0, int p1 = -1,
                                    const HaloSync *hsp = nullptr)
{
	LevelDev &L = h->levels[l];
	const HaloSync hs = hsp ? *hsp : HaloSync{};
	if (hsp && !halo_in_kernel(h, l)) return fail(TGPU_ERR_ARG, "k_face_residual_restrict: in-kernel halo hand-over is not available for this level");
	if (p1 < 0) p1 = L.P;
	if (p1 <= p0) return hs.push ? fail(TGPU_ERR_ARG, "k_face_residual_restrict: a launch that pushes faces needs patches") : TGPU_OK;
	Tag tg(h->ctx, "face_residual_restrict", l);
	const PatchMeta *meta = L.meta.get();
	if (is_3d32(h)) {
		const dim3 grid(std::min(p1 - p0, h->ctx->sm_count * 4)), block(TGPU_THREADS);
		return flag_variant(Fold != nullptr, hs.enabled, [&](auto FOLD, auto HALO) {
			return halo_launch(h->ctx, hs, face_residual_restrict_big_kernel<3, 32, FOLD, HALO>, grid, block, FRR32_SMEM, meta, p0, p1, Fnew, Fold, coarse, hs);
		});
	}
	if (specialised(h) && h->D == 3) { // 16^3 (2-D 32^2 takes the size-generic kernel, with the hand-over)
		const dim3 grid(std::min(p1 - p0, h->ctx->sm_count * 8)), block(TGPU_THREADS);
		return flag_variant(Fold != nullptr, hs.enabled, [&](auto FOLD, auto HALO) {
			return halo_launch(h->ctx, hs, face_residual_restrict16_kernel<FOLD, HALO>, grid, block, 0, meta, p0, p1, Fnew, Fold, coarse, hs);
		});
	}
	DISPATCH_DN(h->D, h->N, {
		using G        = Geo<DD, NN>;
		const int nblk = (p1 - p0 + G::PPB - 1) / G::PPB;
		const dim3 grid(std::min(nblk, h->ctx->sm_count * 8)), block(TGPU_THREADS);
		return flag_variant(Fold != nullptr, hs.enabled, [&](auto FOLD, auto HALO) -> int {
			if constexpr (HALO && !(DD == 2 && NN == 32)) // 2-D 32^2 is the only size-generic instantiation with the hand-over
				return fail(TGPU_ERR_ARG, "k_face_residual_restrict: no in-kernel hand-over for this patch size");
			else
				return halo_launch(h->ctx, hs, face_residual_restrict_kernel<DD, NN, FOLD, HALO>, grid, block, 0, meta, p0, p1, Fnew, Fold, coarse, hs);
		});
	});
}
static int k_restrict(tgpu_hier *h, int l, const double *fine, double *coarse)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, "restrict", l);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, restrict_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, fine, coarse));
}
static int k_prolong_add(tgpu_hier *h, int l, const double *coarse, double *fine)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, "prolong_add", l);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, prolong_add_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, coarse, fine));
}
static int k_prolong_linear_add(tgpu_hier *h, int l, const double *coarse, double *fine)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, "prolong_linear_add", l);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, prolong_linear_add_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, coarse, fine));
}
static int k_prolong_faces(tgpu_hier *h, int l, const double *coarse, double *F)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, "prolong_faces", l);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, prolong_faces_kernel<DD, NN>, dim3(grid_for(h->ctx, L.nface)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, coarse, F));
}
static int k_set(tgpu_hier *h, double *v, size_t n, double alpha)
{
	return launch(h->ctx, blas1_kernel<B_SET>, dim3(grid_for(h->ctx, n)), dim3(256), 0, n, v, (const double *) nullptr, (const double *) nullptr, alpha, 0.0, 0.0);
}

// ---- peer-to-peer halo exchange (see kernels.cuh: push_faces_kernel, p2p_signal_kernel, p2p_wait_kernel) ----
// Per level two generation counters per peer, both in the receiver's memory: DATA (my faces have landed in
// your halo slots) and ACK (I have consumed the halo you pushed).  Generation g is pushed once every peer has
// acknowledged g - 1, consumed after every peer's DATA has reached g, and acknowledged right after its
// consumers were enqueued (k_exchange_done).  Every step is a kernel on the library's stream, so the whole
// protocol is captured in the cycle's CUDA graph.
enum { P2P_DATA = 0, P2P_ACK = 1 };
static int p2p_signal(tgpu_hier *h, int l, int kind)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, kind == P2P_DATA ? "p2p_signal_data" : "p2p_signal_ack", l);
	return launch(h->ctx, p2p_signal_kernel, dim3(1), dim3(32), 0, (uint64_t *const *) (kind == P2P_DATA ? L.peer_data_flag.get() : L.peer_ack_flag.get()),
	              (int) L.peers.size(), L.cnt.get() + (kind == P2P_DATA ? 0 : 2));
}
static int p2p_wait(tgpu_hier *h, int l, int kind, int lag)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, kind == P2P_DATA ? "p2p_wait_data" : "p2p_wait_ack", l);
	return launch(h->ctx, p2p_wait_kernel, dim3(1), dim3(32), 0, (const uint64_t *) (kind == P2P_DATA ? L.data_flags : L.ack_flags),
	              (const int32_t *) L.peer_rank.get(), (int) L.peers.size(), L.cnt.get() + (kind == P2P_DATA ? 1 : 3), lag, h->p2p_abort.get(), (int *) h->ctx->p2p_err.get());
}
// store my boundary faces (F, or F + P uc on the boundary cells) into the peers' halo slots and publish them: one kernel
// that waits for the peers' ACK of the previous generation, pushes, and signals DATA from its last block (PushSync)
static int p2p_push(tgpu_hier *h, int l, double *F, const double *uc)
{
	LevelDev &L   = h->levels[l];
	tgpu_ctx *ctx = h->ctx;
	if (F != L.Fa && F != L.Fb) return fail(TGPU_ERR_ARG, "p2p_push: not a face buffer of this level");
	size_t M = 1;
	for (int i = 0; i < h->D - 1; i++) M *= h->N;
	if (!L.nsend) { // nothing of mine is needed by anybody, but the protocol's generations still advance
		TRY(p2p_wait(h, l, P2P_ACK, 1));
		return p2p_signal(h, l, P2P_DATA);
	}
	PushSync ps;
	ps.ack_flags      = L.ack_flags;
	ps.peer_rank      = L.peer_rank.get();
	ps.peer_data_flag = L.peer_data_flag.get();
	ps.cnt            = L.cnt.get();
	ps.ticket         = L.tickets.get();
	ps.abort          = h->p2p_abort.get();
	ps.host_err       = (int *) ctx->p2p_err.get();
	ps.npeers         = (int) L.peers.size();
	ps.enabled        = 1;
	Tag             tg(ctx, "p2p_push_faces", l);
	double *const *pf = (F == L.Fa) ? L.peerFa.get() : L.peerFb.get();
	DISPATCH_DN_ALL(h->D, h->N, return flag_variant(uc != nullptr, [&](auto PR) {
		return launch(ctx, push_faces_kernel<DD, NN, PR>, dim3(grid_for(ctx, L.nsend * M)), dim3(256), 0, (const PatchMeta *) L.meta.get(), (int) L.nsend, (const int32_t *) L.send_patch.get(), (const int32_t *) L.send_side.get(), (const int32_t *) L.send_peer.get(), (const int32_t *) L.send_ridx.get(), (const double *) F, uc, pf, ps);
	}));
}
static bool exchanges(const tgpu_hier *h, int l)
{
	const LevelDev &L = h->levels[l];
	return L.distributed && h->ctx->nranks > 1 && (L.nsend || L.nrecv);
}
// halo exchange of one distributed level.  Peer-to-peer: push + wait.  NCCL fallback (TGPU_P2P=0): pack the
// faces every peer needs, grouped ncclSend/ncclRecv, scatter what arrived into the halo slots of F.
// uc != nullptr sends F + (P uc) on the boundary cells (the receiver must not add the correction again:
// halo slots have no parent, see FaceVals).  Every k_exchange is followed, after the kernels that read the
// halo, by k_exchange_done.
static int k_exchange(tgpu_hier *h, int l, double *F, const double *uc)
{
	LevelDev &L   = h->levels[l];
	tgpu_ctx *ctx = h->ctx;
	if (!exchanges(h, l)) return TGPU_OK;
	if (L.p2p) {
		TRY(p2p_push(h, l, F, uc));
		return p2p_wait(h, l, P2P_DATA, 0);
	}
	size_t M = 1;
	for (int i = 0; i < h->D - 1; i++) M *= h->N;
	Tag tg(ctx, "halo_exchange", l);
	if (L.nsend) {
		DISPATCH_DN_ALL(h->D, h->N, TRY(flag_variant(uc != nullptr, [&](auto PR) {
			return launch(ctx, pack_faces_kernel<DD, NN, PR>, dim3(grid_for(ctx, L.nsend * M)), dim3(256), 0, (const PatchMeta *) L.meta.get(), (int) L.nsend, (const int32_t *) L.send_patch.get(), (const int32_t *) L.send_side.get(), (const double *) F, uc, L.sendbuf.get());
		})));
	}
	{
	ProfSpan span(ctx, "nccl_sendrecv", l);
	NC(g_nccl.GroupStart());
	for (const PeerDev &pd : L.peers) {
		if (pd.send_n) NC(g_nccl.Send(L.sendbuf.get() + pd.send_off * M, pd.send_n * M, ncclDouble, pd.peer, ctx->comm, ctx->stream));
		if (pd.recv_n) NC(g_nccl.Recv(L.recvbuf.get() + pd.recv_off * M, pd.recv_n * M, ncclDouble, pd.peer, ctx->comm, ctx->stream));
	}
	NC(g_nccl.GroupEnd());
	}
	if (L.nrecv) {
		DISPATCH_DN_ALL(h->D, h->N, TRY(launch(ctx, unpack_faces_kernel<DD, NN>, dim3(grid_for(ctx, L.nrecv * M)), dim3(256), 0, (int) L.nrecv, (const int32_t *) L.recv_slot.get(), (const int32_t *) L.recv_side.get(), (const double *) L.recvbuf.get(), F)));
	}
	return TGPU_OK;
}
// the kernels that read the halo of the last exchange on level l have been enqueued
static int k_exchange_done(tgpu_hier *h, int l)
{
	if (!exchanges(h, l) || !h->levels[l].p2p) return TGPU_OK;
	return p2p_signal(h, l, P2P_ACK);
}
// sum a replicated level vector over the ranks (every cell is written by exactly one rank, the others hold 0)
static int k_allreduce_sum(tgpu_hier *h, double *v, size_t n)
{
	tgpu_ctx *ctx = h->ctx;
	if (ctx->nranks == 1) return TGPU_OK;
	ProfSpan span(ctx, "nccl_allreduce", -1);
	NC(g_nccl.AllReduce(v, v, n, ncclDouble, ncclSum, ctx->comm, ctx->stream));
	return TGPU_OK;
}
// true if level l is distributed and level l + 1 is replicated (the restriction crosses the boundary)
static bool crosses_replication(const tgpu_hier *h, int l)
{
	return h->ctx->nranks > 1 && l + 1 < (int) h->levels.size() && h->levels[l].distributed && !h->levels[l + 1].distributed;
}

extern "C" int tgpu_apply(tgpu_hier *h, int level, const tgpu_vec *u, tgpu_vec *out)
{
	API_BEGIN
	TRY(check_level_vec(h, level, u, "tgpu_apply"));
	TRY(check_level_vec(h, level, out, "tgpu_apply"));
	if (u == out) return fail(TGPU_ERR_ARG, "tgpu_apply: in-place apply is not supported");
	TRY(k_extract_faces(h, level, u->d, h->levels[level].Fa));
	TRY(k_exchange(h, level, h->levels[level].Fa, nullptr));
	TRY(k_apply(h, level, 0, u->d, nullptr, h->levels[level].Fa, out->d, nullptr));
	return k_exchange_done(h, level);
	API_END
}
extern "C" int tgpu_residual(tgpu_hier *h, int level, const tgpu_vec *f, const tgpu_vec *u, tgpu_vec *r)
{
	API_BEGIN
	TRY(check_level_vec(h, level, f, "tgpu_residual"));
	TRY(check_level_vec(h, level, u, "tgpu_residual"));
	TRY(check_level_vec(h, level, r, "tgpu_residual"));
	if (u == r) return fail(TGPU_ERR_ARG, "tgpu_residual: r must not alias u");
	TRY(k_extract_faces(h, level, u->d, h->levels[level].Fa));
	TRY(k_exchange(h, level, h->levels[level].Fa, nullptr));
	TRY(k_apply(h, level, 1, u->d, f->d, h->levels[level].Fa, r->d, nullptr));
	return k_exchange_done(h, level);
	API_END
}
extern "C" int tgpu_smooth(tgpu_hier *h, int level, const tgpu_vec *f, tgpu_vec *u)
{
	API_BEGIN
	TRY(check_level_vec(h, level, f, "tgpu_smooth"));
	TRY(check_level_vec(h, level, u, "tgpu_smooth"));
	if (f == u) return fail(TGPU_ERR_ARG, "tgpu_smooth: f must not alias u");
	TRY(k_extract_faces(h, level, u->d, h->levels[level].Fa));
	TRY(k_exchange(h, level, h->levels[level].Fa, nullptr));
	TRY(k_smooth(h, level, false, false, f->d, u->d, h->levels[level].Fa, nullptr));
	return k_exchange_done(h, level);
	API_END
}
static int ensure_work(tgpu_hier *h, int l, bool need_r)
{
	LevelDev &L = h->levels[l];
	// the finest level works on the caller's f and u; r only exists for the API-granular schedule (GMG/Cycle.h:59)
	if (l > 0 && !L.u) CU(dev_malloc(L.u, L.ncells * sizeof(double)));
	if (l > 0 && !L.f) CU(dev_malloc(L.f, L.ncells * sizeof(double)));
	if (need_r && !L.r) CU(dev_malloc(L.r, L.ncells * sizeof(double)));
	return TGPU_OK;
}
extern "C" int tgpu_smooth_jacobi(tgpu_hier *h, int level, const tgpu_vec *f, tgpu_vec *u, double omega)
{
	API_BEGIN
	TRY(check_level_vec(h, level, f, "tgpu_smooth_jacobi"));
	TRY(check_level_vec(h, level, u, "tgpu_smooth_jacobi"));
	TRY(ensure_work(h, level, true));
	LevelDev &L = h->levels[level];
	TRY(k_extract_faces(h, level, u->d, L.Fa));
	TRY(k_exchange(h, level, L.Fa, nullptr));
	TRY(k_apply(h, level, 1, u->d, f->d, L.Fa, L.r.get(), nullptr));
	TRY(k_exchange_done(h, level));
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, jacobi_update_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, (const double *) L.r.get(), u->d, omega, h->op_shift));
	API_END
}
extern "C" int tgpu_restrict(tgpu_hier *h, int fine_level, const tgpu_vec *fine, tgpu_vec *coarse)
{
	API_BEGIN
	TRY(check_level_vec(h, fine_level, fine, "tgpu_restrict"));
	TRY(check_level_vec(h, fine_level + 1, coarse, "tgpu_restrict"));
	if (crosses_replication(h, fine_level)) {
		TRY(k_set(h, coarse->d, coarse->n, 0.0));
		TRY(k_restrict(h, fine_level, fine->d, coarse->d));
		return k_allreduce_sum(h, coarse->d, coarse->n);
	}
	return k_restrict(h, fine_level, fine->d, coarse->d);
	API_END
}
extern "C" int tgpu_prolong_add(tgpu_hier *h, int fine_level, const tgpu_vec *coarse, tgpu_vec *fine)
{
	API_BEGIN
	TRY(check_level_vec(h, fine_level, fine, "tgpu_prolong_add"));
	TRY(check_level_vec(h, fine_level + 1, coarse, "tgpu_prolong_add"));
	return k_prolong_add(h, fine_level, coarse->d, fine->d);
	API_END
}
extern "C" int tgpu_prolong_add_linear(tgpu_hier *h, int fine_level, const tgpu_vec *coarse, tgpu_vec *fine)
{
	API_BEGIN
	TRY(check_level_vec(h, fine_level, fine, "tgpu_prolong_add_linear"));
	TRY(check_level_vec(h, fine_level + 1, coarse, "tgpu_prolong_add_linear"));
	return k_prolong_linear_add(h, fine_level, coarse->d, fine->d);
	API_END
}
extern "C" int tgpu_residual_restrict(tgpu_hier *h, int fine_level, const tgpu_vec *f, const tgpu_vec *u, tgpu_vec *coarse_f)
{
	API_BEGIN
	TRY(check_level_vec(h, fine_level, f, "tgpu_residual_restrict"));
	TRY(check_level_vec(h, fine_level, u, "tgpu_residual_restrict"));
	TRY(check_level_vec(h, fine_level + 1, coarse_f, "tgpu_residual_restrict"));
	TRY(k_extract_faces(h, fine_level, u->d, h->levels[fine_level].Fa));
	TRY(k_exchange(h, fine_level, h->levels[fine_level].Fa, nullptr));
	if (crosses_replication(h, fine_level)) TRY(k_set(h, coarse_f->d, coarse_f->n, 0.0));
	if (is_3d32(h)) TRY(ensure_work(h, fine_level, true));
	TRY(k_apply(h, fine_level, 2, u->d, f->d, h->levels[fine_level].Fa, nullptr, coarse_f->d));
	TRY(k_exchange_done(h, fine_level));
	if (crosses_replication(h, fine_level)) TRY(k_allreduce_sum(h, coarse_f->d, coarse_f->n));
	return TGPU_OK;
	API_END
}

// ------------------------------------------------------------------------------------------
// cycle
// ------------------------------------------------------------------------------------------
extern "C" int tgpu_cycle_opts_default(TgpuCycleOpts *o)
{
	if (!o) return fail(TGPU_ERR_ARG, "null argument");
	o->pre_sweeps = o->post_sweeps = o->mid_sweeps = o->coarse_sweeps = 1;
	o->cycle_type                                                   = 0;
	o->fused                                                        = 1;
	o->use_graph                                                    = 1;
	o->max_levels                                                   = 0;
	o->interpolator                                                 = 0;
	o->reserved_                                                    = 0;
	o->patches_per_proc                                             = 0.0;
	return TGPU_OK;
}

// API-granular schedule, statement for statement GMG/Cycle.h:56-126 + VCycle.h:44-62 / WCycle.h:45-68
static int generic_smooth(tgpu_hier *h, int l, const double *f, double *u)
{
	TRY(k_extract_faces(h, l, u, h->levels[l].Fa));
	TRY(k_exchange(h, l, h->levels[l].Fa, nullptr));
	TRY(k_smooth(h, l, false, false, f, u, h->levels[l].Fa, nullptr));
	return k_exchange_done(h, l);
}
static int generic_prep_coarser(tgpu_hier *h, int l, const double *f, const double *u)
{
	LevelDev &L = h->levels[l], &C = h->levels[l + 1];
	TRY(k_extract_faces(h, l, u, L.Fa));
	TRY(k_exchange(h, l, L.Fa, nullptr));
	TRY(k_apply(h, l, 1, u, f, L.Fa, L.r.get(), nullptr)); // r = A u; r = -r + f
	TRY(k_exchange_done(h, l));
	TRY(k_set(h, C.u.get(), C.ncells, 0.0));               // new_u (zero-initialised Vec)
	if (crosses_replication(h, l)) TRY(k_set(h, C.f.get(), C.ncells, 0.0));
	TRY(k_restrict(h, l, L.r.get(), C.f.get()));                 // new_f = R r
	if (crosses_replication(h, l)) TRY(k_allreduce_sum(h, C.f.get(), C.ncells));
	return TGPU_OK;
}
static int generic_visit(tgpu_hier *h, const TgpuCycleOpts &o, int l, const double *f, double *u)
{
	const int last = h->last_level;
	if (l == last) {
		for (int i = 0; i < o.coarse_sweeps; i++) TRY(generic_smooth(h, l, f, u));
	} else {
		LevelDev &C = h->levels[l + 1];
		for (int i = 0; i < o.pre_sweeps; i++) TRY(generic_smooth(h, l, f, u));
		TRY(generic_prep_coarser(h, l, f, u));
		auto prolong = [&]() { return o.interpolator == 1 ? k_prolong_linear_add(h, l, C.u.get(), u) : k_prolong_add(h, l, C.u.get(), u); };
		TRY(generic_visit(h, o, l + 1, C.f.get(), C.u.get()));
		TRY(prolong());
		if (o.cycle_type == 1) {
			for (int i = 0; i < o.mid_sweeps; i++) TRY(generic_smooth(h, l, f, u));
			TRY(generic_prep_coarser(h, l, f, u));
			TRY(generic_visit(h, o, l + 1, C.f.get(), C.u.get()));
			TRY(prolong());
		}
		for (int i = 0; i < o.post_sweeps; i++) TRY(generic_smooth(h, l, f, u));
	}
	return TGPU_OK;
}
// fork: the comm stream waits for everything queued on the main stream so far, runs the exchange, and
// records `done`; the main stream carries on with patches that need no halo data and waits on `done` later.
static int exchange_async(tgpu_hier *h, int l, double *F, const double *uc, cudaEvent_t fork, cudaEvent_t done)
{
	tgpu_ctx *   ctx  = h->ctx;
	cudaStream_t main = ctx->stream;
	CU(cudaEventRecord(fork, main));
	CU(cudaStreamWaitEvent(ctx->comm_stream.get(), fork, 0));
	ctx->stream = ctx->comm_stream.get();
	int rc      = k_exchange(h, l, F, uc);
	ctx->stream = main;
	TRY(rc);
	CU(cudaEventRecord(done, ctx->comm_stream.get()));
	return TGPU_OK;
}
// Fused schedule for V cycles with >= 1 pre and post sweep.  Per level visit:
//   smooth(zero guess) -> faces | residual+restrict from the faces -> f_coarse | (coarser) |
//   smooth(f, faces + P u_coarse on the boundary cells) -> u
// A block-Jacobi sweep depends on the previous iterate only through its boundary-cell slices
// (SchurHelper.h:319-331), and right after a sweep the residual is (2/h^2) E^T (gamma(u_old) - gamma(u_new))
// (see face_residual_restrict_kernel).  So, compared with the generic schedule, the dead stores are never
// materialised: the zero fill of u, the pre-smoothed u itself, the fine residual vector and the interior
// of the prolonged u; only the last sweep of a level visit writes u.  opts.fused = 2 keeps the PR-1 form
// of the middle step (residual evaluated from u and f by apply_tma_kernel<2>) for cross-checking.
// guess (level 0 of a cycle with coarser levels): start from the iterate in u instead of zero.  The first pre-sweep needs
// only u's boundary slices, extracted into Fcur; from there every pre-sweep is the non-zero-guess sweep of i > 0, so
// one cycle computes u + Cycle(f - A u) (the smoother is linear and stationary).  Coarser levels start from zero.
// faces (with guess): L.Fa or L.Fb already holds u's boundary slices, no extraction (full multigrid: fmg_interp_kernel or
// the previous cycle's last sweep wrote them).  want_faces on a level above the coarsest: h->visit_faces is the face buffer
// that holds the slices of the result afterwards.
static int fused_visit(tgpu_hier *h, const TgpuCycleOpts &o, int l, const double *f, double *u, bool want_faces, bool guess = false,
                       const double *faces = nullptr)
{
	const int last = h->last_level;
	LevelDev &L    = h->levels[l];
	double *  Fcur = L.Fa, *Falt = L.Fb;
	if (faces == L.Fb) std::swap(Fcur, Falt);
	if (l == last) {
		for (int i = 0; i < o.coarse_sweeps; i++) {
			const bool emit = (i + 1 < o.coarse_sweeps);
			if (i > 0) TRY(k_exchange(h, l, Fcur, nullptr));
			TRY(k_smooth(h, l, i == 0, emit, f, u, Fcur, i == 0 ? Fcur : Falt, nullptr, 0, -1, !emit));
			if (i > 0) TRY(k_exchange_done(h, l));
			if (i > 0 && emit) std::swap(Fcur, Falt);
		}
		return TGPU_OK;
	}
	const bool from_faces = (o.fused != 2);
	LevelDev & C          = h->levels[l + 1];
	if (guess && !faces) TRY(k_extract_faces(h, l, u, Fcur));
	for (int i = 0; i < o.pre_sweeps; i++) {
		const bool nonzero = guess || i > 0;
		if (nonzero) TRY(k_exchange(h, l, Fcur, nullptr));
		TRY(k_smooth(h, l, !nonzero, true, f, u, Fcur, nonzero ? Falt : Fcur, nullptr, 0, -1, !from_faces));
		if (nonzero) TRY(k_exchange_done(h, l));
		if (nonzero) std::swap(Fcur, Falt);
	}
	// Fcur: faces of the pre-smoothed u; Falt: faces of the iterate before the last pre-sweep (if it did not start from zero)
	const double *Fold    = (guess || o.pre_sweeps > 1) ? Falt : nullptr;
	const bool    overlap = exchanges(h, l);
	auto residual_restrict = [&](int p0, int p1) {
		if (from_faces) return k_face_residual_restrict(h, l, Fcur, Fold, C.f.get(), p0, p1);
		return k_apply(h, l, 2, u, f, Fcur, nullptr, C.f.get(), p0, p1);
	};
	if (crosses_replication(h, l)) TRY(k_set(h, C.f.get(), C.ncells, 0.0));
	if (overlap && L.p2p && from_faces && halo_in_kernel(h, l)) {
		// the faces of the pre-smoothed u go straight into the neighbours' halo slots; theirs arrive while the patches
		// without off-rank neighbours are swept: ONE launch over all owned patches whose CTAs poll the peers' flags
		// before their first boundary patch and whose last CTA acknowledges the halo (HaloSync, kernels.cuh)
		// (push_in_kernel: the same launch pushes this rank's faces first, halo_push_cta)
		const HaloSync hs = halo_sync(h, l, push_in_kernel(h, l) ? Fcur : nullptr, false);
		if (!hs.push) TRY(p2p_push(h, l, Fcur, nullptr));
		TRY(k_face_residual_restrict(h, l, Fcur, Fold, C.f.get(), 0, L.P, &hs));
	} else if (overlap && L.p2p) {
		TRY(p2p_push(h, l, Fcur, nullptr));
		TRY(residual_restrict(0, L.n_interior));
		TRY(p2p_wait(h, l, P2P_DATA, 0));
		TRY(residual_restrict(L.n_interior, L.P));
		TRY(k_exchange_done(h, l));
	} else if (overlap) {
		// faces of the pre-smoothed u travel on the comm stream while the interior patches are swept
		TRY(exchange_async(h, l, Fcur, nullptr, L.ev[0].get(), L.ev[1].get()));
		TRY(residual_restrict(0, L.n_interior));
		CU(cudaStreamWaitEvent(h->ctx->stream, L.ev[1].get(), 0));
		TRY(residual_restrict(L.n_interior, L.P));
	} else {
		TRY(residual_restrict(0, L.P));
	}
	if (crosses_replication(h, l)) TRY(k_allreduce_sum(h, C.f.get(), C.ncells));
	TRY(fused_visit(h, o, l + 1, C.f.get(), C.u.get(), false));
	if (o.cycle_type == 1) {
		// W cycle (GMG/WCycle.h:57-63; one GPU, mid_sweeps >= 1): the second coarse-grid correction.  The iterate before the
		// mid sweeps is u_pre + P u_c, seen only through its boundary slices: Fcur += (P u_c) on the boundary cells; every
		// mid sweep emits the slices of its result, and the residual after the last one is again supported on the faces
		// (old slices - new slices), so neither u_pre + P u_c nor the mid-smoothed u is ever written.
		TRY(k_prolong_faces(h, l, C.u.get(), Fcur));
		for (int i = 0; i < o.mid_sweeps; i++) {
			TRY(k_smooth(h, l, false, true, f, u, Fcur, Falt, nullptr, 0, -1, !from_faces));
			std::swap(Fcur, Falt);
		}
		Fold = Falt;
		TRY(residual_restrict(0, L.P));
		TRY(fused_visit(h, o, l + 1, C.f.get(), C.u.get(), false));
	}
	// same faces + prolonged correction for the neighbours on other GPUs (owned faces add it on the fly)
	const bool push_folded = overlap && L.p2p && o.post_sweeps >= 1 && push_in_kernel(h, l) && L.push_desc && L.push_uc == C.u.get();
	if (push_folded) {} // the first post-sweep's launch pushes them itself
	else if (overlap && L.p2p) TRY(p2p_push(h, l, Fcur, C.u.get()));
	else if (overlap) TRY(exchange_async(h, l, Fcur, C.u.get(), L.ev[2].get(), L.ev[3].get()));
	for (int i = 0; i < o.post_sweeps; i++) {
		const bool lastsweep = (i + 1 == o.post_sweeps);
		const bool emit      = !lastsweep || want_faces;
		// first post-sweep: boundary values = faces of the pre-smoothed u + prolonged coarse correction
		if (i > 0) TRY(k_exchange(h, l, Fcur, nullptr));
		if (i == 0 && overlap && L.p2p && halo_in_kernel(h, l)) {
			const HaloSync hs = halo_sync(h, l, push_folded ? Fcur : nullptr, true);
			TRY(k_smooth(h, l, false, emit, f, u, Fcur, Falt, C.u.get(), 0, L.P, lastsweep, &hs));
		} else if (i == 0 && overlap) {
			TRY(k_smooth(h, l, false, emit, f, u, Fcur, Falt, C.u.get(), 0, L.n_interior, lastsweep));
			if (L.p2p) TRY(p2p_wait(h, l, P2P_DATA, 0));
			else CU(cudaStreamWaitEvent(h->ctx->stream, L.ev[3].get(), 0));
			TRY(k_smooth(h, l, false, emit, f, u, Fcur, Falt, C.u.get(), L.n_interior, L.P, lastsweep));
			TRY(k_exchange_done(h, l));
		} else {
			TRY(k_smooth(h, l, false, emit, f, u, Fcur, Falt, i == 0 ? C.u.get() : nullptr, 0, -1, lastsweep));
			if (i > 0) TRY(k_exchange_done(h, l));
		}
		std::swap(Fcur, Falt);
	}
	if (want_faces) h->visit_faces = Fcur;
	if (l == 0 && want_faces) { // the last sweep emitted the slices of u here; Falt holds those of its input
		h->cycle_faces     = Fcur;
		h->cycle_faces_old = Falt;
		h->cycle_uc        = o.post_sweeps == 1 ? C.u.get() : nullptr;
	}
	return TGPU_OK;
}
// the fused schedule covers cycles with at least one sweep everywhere and the piecewise-constant interpolator: V cycles on
// any number of GPUs, W cycles (with at least one mid sweep) on one GPU
static bool fused_schedule(const TgpuCycleOpts &o, int nranks)
{
	if (!o.fused || o.interpolator != 0 || o.pre_sweeps < 1 || o.post_sweeps < 1 || o.coarse_sweeps < 1) return false;
	return o.cycle_type == 0 || (o.cycle_type == 1 && o.mid_sweeps >= 1 && nranks == 1);
}
// want_faces: the caller applies the operator to the result next (BiCGStab: v = A M^-1 p), so the last sweep also
// writes the result's boundary slices (h->cycle_faces != nullptr afterwards) and no extraction pass is needed
// guess: start from the iterate in u (guess_schedule must hold)
static int run_cycle(tgpu_hier *h, const TgpuCycleOpts &o, const double *f, double *u, bool want_faces = false, bool guess = false)
{
	const bool fused = fused_schedule(o, h->ctx->nranks);
	h->cycle_faces   = nullptr;
	h->cycle_faces_old = h->cycle_uc = nullptr;
	if (fused) return fused_visit(h, o, 0, f, u, want_faces && h->last_level > 0, guess);
	if (guess) return fail(TGPU_ERR_ARG, "run_cycle: this schedule cannot start from a guess");
	TRY(k_set(h, u, h->levels[0].ncells, 0.0)); // Cycle::apply: u->set(0)
	return generic_visit(h, o, 0, f, u);
}
static bool same_opts(const TgpuCycleOpts &a, const TgpuCycleOpts &b) { return memcmp(&a, &b, sizeof(a)) == 0; }

// the options a cycle runs with (opts == NULL: defaults), checked, and the coarsest level it visits (h->last_level)
static int cycle_opts(tgpu_hier *h, const TgpuCycleOpts *opts, TgpuCycleOpts &o)
{
	if (opts) o = *opts;
	else tgpu_cycle_opts_default(&o);
	o.reserved_ = 0;
	// With a patch solver shift the operator does not carry, the sweep solves (A_p + lambda) u = ..., so the residual of the
	// operator right after a sweep is no longer supported on the patch boundaries: the face-only residual schedule does not apply
	if (!consistent(h) && o.fused == 1) o.fused = 2;
	if (o.pre_sweeps < 0 || o.post_sweeps < 0 || o.coarse_sweeps < 0 || o.mid_sweeps < 0 || (o.cycle_type != 0 && o.cycle_type != 1)
	    || (o.interpolator != 0 && o.interpolator != 1))
		return fail(TGPU_ERR_ARG, "tgpu_vcycle: bad cycle options"); /* reference: throw 3, GMG/CycleFactory3d.cpp:131 */
	tgpu_ctx *ctx = h->ctx;
	// the level list the reference's factory would build for these options (GMG/CycleFactory3d.cpp:99-104): at most
	// max_levels levels (0 = no limit), and no level with fewer than patches_per_proc patches per rank
	if (o.max_levels < 0 || !(o.patches_per_proc >= 0.0)) return fail(TGPU_ERR_ARG, "tgpu_vcycle: bad max_levels / patches_per_proc");
	h->last_level = 0;
	for (int l = 1; l < (int) h->levels.size() && (o.max_levels <= 0 || l < o.max_levels); l++) {
		if ((double) h->levels[l].global_P / ctx->nranks < o.patches_per_proc) break;
		h->last_level = l;
	}
	return TGPU_OK;
}
// the fused schedule starts from a guess on level 0 when the face identity holds for its sweeps (consistent shifts)
// and there is a coarser level; cycle_opts must have run
static bool guess_schedule(const tgpu_hier *h, const TgpuCycleOpts &o)
{
	return fused_schedule(o, h->ctx->nranks) && consistent(h) && h->last_level > 0;
}
// Runs run() once, through the hierarchy's cached CUDA graph of key (its f, u, b, fmg_cycles, want_faces, guess and opts):
// replayed when one was captured before, captured and launched otherwise.  o.use_graph = 0, profiling and several GPUs
// (unless use_graph >= 2) run it directly.
template <class Fn> static int graph_run(tgpu_hier *h, const TgpuCycleOpts &o, GraphEntry key, Fn &&run)
{
	tgpu_ctx *ctx = h->ctx;
	if (!o.use_graph || ctx->profiling || (ctx->nranks > 1 && o.use_graph < 2)) return run();
	for (GraphEntry &g : h->graphs)
		if (g.f == key.f && g.u == key.u && g.b == key.b && g.fmg_cycles == key.fmg_cycles && g.want_faces == key.want_faces
		    && g.guess == key.guess && same_opts(g.opts, o)) {
			h->cycle_faces     = g.faces;
			h->cycle_faces_old = g.faces_old;
			h->cycle_uc        = g.faces_uc;
			CU(cudaGraphLaunch(g.exec.get(), ctx->stream));
			ctx->launches += g.kernels;
			return TGPU_OK;
		}
	// capture
	ctx->capturing = true;
	ctx->captured  = 0;
	CU(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
	int         rc  = run();
	cudaGraph_t raw = nullptr;
	cudaError_t e   = cudaStreamEndCapture(ctx->stream, &raw);
	GraphPtr    graph(raw);
	ctx->capturing = false;
	TRY(rc);
	if (e != cudaSuccess) return fail(TGPU_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
	GraphEntry &g = key;
	g.opts = o, g.kernels = ctx->captured;
	g.faces = h->cycle_faces, g.faces_old = h->cycle_faces_old, g.faces_uc = h->cycle_uc;
	cudaGraphExec_t exec = nullptr;
	CU(cudaGraphInstantiate(&exec, graph.get(), 0));
	g.exec.reset(exec);
	if (h->graphs.size() >= 8) h->graphs.erase(h->graphs.begin());
	h->graphs.push_back(std::move(g));
	CU(cudaGraphLaunch(h->graphs.back().exec.get(), ctx->stream));
	ctx->launches += h->graphs.back().kernels;
	return TGPU_OK;
}
static int cycle_ptr(tgpu_hier *h, const TgpuCycleOpts *opts, const double *f, double *u, bool want_faces = false, bool guess = false)
{
	TgpuCycleOpts o;
	TRY(cycle_opts(h, opts, o));
	tgpu_ctx *ctx = h->ctx;
	if (guess && !guess_schedule(h, o)) return fail(TGPU_ERR_ARG, "cycle_ptr: this schedule cannot start from a guess");
	for (size_t l = 0; l <= (size_t) h->last_level; l++) {
		const bool fused_sched = fused_schedule(o, ctx->nranks);
		TRY(ensure_work(h, (int) l, !fused_sched || (o.fused == 2 && is_3d32(h))));
	}
	for (int l = 0; l <= h->last_level; l++) TRY(ensure_push_desc(h, l));
	GraphEntry key;
	key.f = f, key.u = u, key.want_faces = want_faces, key.guess = guess;
	return graph_run(h, o, std::move(key), [&] { return run_cycle(h, o, f, u, want_faces, guess); });
}
extern "C" int tgpu_vcycle(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, f, "tgpu_vcycle"));
	TRY(check_level_vec(h, 0, u, "tgpu_vcycle"));
	if (f == u) return fail(TGPU_ERR_ARG, "tgpu_vcycle: f must not alias u");
	return cycle_ptr(h, opts, f->d, u->d);
	API_END
}
extern "C" int tgpu_vcycle_host(tgpu_hier *h, const TgpuCycleOpts *opts, const double *f_host, double *u_host)
{
	API_BEGIN
	if (!h || !f_host || !u_host) return fail(TGPU_ERR_ARG, "tgpu_vcycle_host: null argument");
	if (!h->host_f) TRY(vec_create(h, 0, h->host_f));
	if (!h->host_u) TRY(vec_create(h, 0, h->host_u));
	TRY(tgpu_vec_upload_async(h->host_f.get(), f_host));
	TRY(cycle_ptr(h, opts, h->host_f->d, h->host_u->d));
	TRY(tgpu_vec_download_async(h->host_u.get(), u_host));
	CU(cudaStreamSynchronize(h->ctx->stream));
	return check_comm(h->ctx);
	API_END
}

// the copy-in / copy-out streams of the pipelined host path and their events, created on first use
static int ensure_pipe_streams(tgpu_hier *h)
{
	for (StreamPtr *s : {&h->s_in, &h->s_out})
		if (!*s) CU(stream_create(*s));
	for (int k = 0; k < 2; k++)
		for (EventPtr *e : {&h->ev_in[k], &h->ev_cyc[k], &h->ev_out[k]})
			if (!*e) CU(event_create(*e, cudaEventDisableTiming));
	return TGPU_OK;
}
// Pipelined form of tgpu_vcycle_host for a stream of independent right-hand sides: the upload of call k + 1
// runs on a copy-in stream while cycle k is on the main stream and result k - 1 travels back on a copy-out
// stream (PCIe is full duplex), with two device slots.  The caller owns the pinned buffers; u_pinned of call k
// is valid after tgpu_vcycle_host_wait, or after call k + 2 has returned and been waited for.
extern "C" int tgpu_vcycle_host_async(tgpu_hier *h, const TgpuCycleOpts *opts, const double *f_host, double *u_host)
{
	API_BEGIN
	if (!h || !f_host || !u_host) return fail(TGPU_ERR_ARG, "tgpu_vcycle_host_async: null argument");
	tgpu_ctx *ctx = h->ctx;
	TRY(ensure_pipe_streams(h));
	if (!h->pipe_f[0]) { // first call, or the first one after tgpu_hierarchy_trim
		for (int k = 0; k < 2; k++) {
			TRY(vec_create(h, 0, h->pipe_f[k]));
			TRY(vec_create(h, 0, h->pipe_u[k]));
		}
		CU(cudaStreamSynchronize(ctx->stream)); // the zero fills of the new vectors
	}
	const int    k     = (int) (h->pipe_count & 1);
	const bool   first = h->pipe_count < 2;
	const size_t bytes = h->pipe_f[k]->n * sizeof(double);
	h->pipe_count++;
	// copy-in: the cycle that last read this slot's f must be done
	if (!first) CU(cudaStreamWaitEvent(h->s_in.get(), h->ev_cyc[k].get(), 0));
	CU(cudaMemcpyAsync(h->pipe_f[k]->d, f_host, bytes, cudaMemcpyHostToDevice, h->s_in.get()));
	CU(cudaEventRecord(h->ev_in[k].get(), h->s_in.get()));
	// cycle: needs this slot's f, and its u must have left for the host
	CU(cudaStreamWaitEvent(ctx->stream, h->ev_in[k].get(), 0));
	if (!first) CU(cudaStreamWaitEvent(ctx->stream, h->ev_out[k].get(), 0));
	TRY(cycle_ptr(h, opts, h->pipe_f[k]->d, h->pipe_u[k]->d));
	CU(cudaEventRecord(h->ev_cyc[k].get(), ctx->stream));
	// copy-out
	CU(cudaStreamWaitEvent(h->s_out.get(), h->ev_cyc[k].get(), 0));
	CU(cudaMemcpyAsync(u_host, h->pipe_u[k]->d, bytes, cudaMemcpyDeviceToHost, h->s_out.get()));
	CU(cudaEventRecord(h->ev_out[k].get(), h->s_out.get()));
	return TGPU_OK;
	API_END
}
// The copies of one tgpu_vcycle_host_async step and nothing else: host -> dst_dev on the copy-in stream and src_dev -> host
// on the copy-out stream at the same time, then both are waited for.  Measures what the host link gives the e2e path.
extern "C" int tgpu_vec_transfer_pair(tgpu_hier *h, tgpu_vec *dst_dev, const double *src_pinned, const tgpu_vec *src_dev, double *dst_pinned)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, dst_dev, "tgpu_vec_transfer_pair"));
	TRY(check_level_vec(h, 0, src_dev, "tgpu_vec_transfer_pair"));
	if (!src_pinned || !dst_pinned) return fail(TGPU_ERR_ARG, "tgpu_vec_transfer_pair: null host buffer");
	TRY(ensure_pipe_streams(h));
	CU(cudaStreamSynchronize(h->ctx->stream));
	CU(cudaMemcpyAsync(dst_dev->d, src_pinned, dst_dev->n * sizeof(double), cudaMemcpyHostToDevice, h->s_in.get()));
	CU(cudaMemcpyAsync(dst_pinned, src_dev->d, src_dev->n * sizeof(double), cudaMemcpyDeviceToHost, h->s_out.get()));
	CU(cudaStreamSynchronize(h->s_in.get()));
	CU(cudaStreamSynchronize(h->s_out.get()));
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_vcycle_host_wait(tgpu_hier *h)
{
	API_BEGIN
	if (!h) return fail(TGPU_ERR_ARG, "null hierarchy");
	if (h->s_out) CU(cudaStreamSynchronize(h->s_out.get()));
	CU(cudaStreamSynchronize(h->ctx->stream));
	return check_comm(h->ctx);
	API_END
}

// BiCGStab<D>::solve (BiCGStab.h:45-106, right-preconditioned) with the BLAS-1 work of an iteration fused into three passes and
// the scalars kept on the device (bicg_*_kernel in kernels.cuh): 20 vector passes per iteration instead of 30, one host read
// instead of six.
static int bicgstab_fused(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *b, tgpu_vec *x, double tol, int max_it,
                          int *iterations, double *rel_residual)
{
	tgpu_ctx *ctx = h->ctx;
	while (h->krylov_ws.size() < 8) {
		VecPtr v;
		TRY(vec_create(h, 0, v));
		h->krylov_ws.push_back(std::move(v));
	}
	if (!h->krylov_sc) CU(dev_malloc(h->krylov_sc, 8 * sizeof(double)));
	tgpu_vec *resid = h->krylov_ws[0].get(), *rhat = h->krylov_ws[1].get(), *p = h->krylov_ws[2].get(), *ap = h->krylov_ws[3].get();
	tgpu_vec *as = h->krylov_ws[4].get(), *s = h->krylov_ws[5].get(), *ms = h->krylov_ws[6].get(), *mp = h->krylov_ws[7].get();
	const bool   prec   = opts != nullptr;
	const bool   dist   = ctx->nranks > 1 && h->levels[0].distributed;
	const size_t n      = resid->n;
	const int    stride = MAX_PARTIAL / 2;
	const int    nb     = std::min(stride, grid_for(ctx, n, 256, 8));
	double *     sc     = h->krylov_sc.get();
	auto A = [&](const tgpu_vec *in, tgpu_vec *out) { return tgpu_apply(h, 0, in, out); };
	// the preconditioner's last sweep emits the boundary slices of its result, which is all A needs besides the result
	auto M = [&](const tgpu_vec *in, tgpu_vec *out) { return cycle_ptr(h, opts, in->d, out->d, true); };
	// out = A in for in = the vector M has just produced (its boundary slices are in h->cycle_faces), with the dot products the
	// iteration needs next (out . dotv, out . out) formed by the same kernel: *nbp block partials in ctx->d_partial.get()
	auto AM = [&](const tgpu_vec *in, tgpu_vec *out, const tgpu_vec *dotv, int *nbp) {
		double *F = h->cycle_faces;
		if (!F) {
			F = h->levels[0].Fa;
			TRY(k_extract_faces(h, 0, in->d, F));
		}
		TRY(k_exchange(h, 0, F, nullptr));
		TRY(k_apply(h, 0, 3, in->d, dotv->d, F, out->d, nullptr, 0, -1, nbp));
		return k_exchange_done(h, 0);
	};
	auto finish = [&](int step, int nparts) {
		Tag tg(ctx, "bicg_scalars", 0);
		TRY(launch(ctx, bicg_finish_kernel, dim3(1), dim3(256), 0, nparts, stride, (const double *) ctx->d_partial.get(), sc, step, dist ? 0 : 1));
		if (dist) {
			NC(g_nccl.AllReduce(sc + SC_SUM0, sc + SC_SUM0, 2, ncclDouble, ncclSum, ctx->comm, ctx->stream));
			TRY(launch(ctx, bicg_scalars_kernel, dim3(1), dim3(32), 0, sc, step));
		}
		return (int) TGPU_OK;
	};
	auto dots = [&](const tgpu_vec *a, const tgpu_vec *c, int step) {
		Tag tg(ctx, "bicg_dots", 0);
		TRY(launch(ctx, bicg_dots_kernel, dim3(nb), dim3(256), 0, n, (const double *) a->d, (const double *) c->d, ctx->d_partial.get(), stride));
		return finish(step, nb);
	};
	auto read_rnorm = [&](double *out) {
		CU(cudaMemcpyAsync(ctx->h_result.get(), sc + SC_RNORM, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
		CU(cudaStreamSynchronize(ctx->stream));
		*out = ctx->h_result.get()[0];
		return check_comm(ctx);
	};
	TRY(A(x, resid));
	TRY(tgpu_vec_scale_then_add(resid, -1, b));
	TRY(tgpu_vec_copy(rhat, resid));
	TRY(tgpu_vec_copy(p, resid));
	TRY(dots(resid, rhat, 0)); // rho = rhat . r, |r|
	double r0_norm, rn;
	TRY(read_rnorm(&r0_norm));
	rn      = r0_norm;
	int its = 0;
	while (rn / r0_norm > tol && its < max_it) {
		const tgpu_vec *pp = p, *ss = s;
		int             nparts = nb;
		if (prec) {
			TRY(M(p, mp));
			pp = mp;
			TRY(AM(pp, ap, rhat, &nparts)); // ap = A mp, ap . rhat riding along
			TRY(finish(1, nparts));         // alpha
		} else {
			TRY(A(pp, ap));
			TRY(dots(rhat, ap, 1)); // alpha
		}
		{
			Tag tg(ctx, "bicg_s", 0);
			TRY(launch(ctx, bicg_s_kernel, dim3(grid_for(ctx, n)), dim3(256), 0, n, (const double *) resid->d, (const double *) ap->d, s->d, (const double *) sc));
		}
		if (prec) {
			TRY(M(s, ms));
			ss = ms;
			TRY(AM(ss, as, s, &nparts)); // as = A ms, as . s and as . as riding along
			TRY(finish(2, nparts));      // omega
		} else {
			TRY(A(ss, as));
			TRY(dots(as, s, 2)); // omega
		}
		{
			Tag tg(ctx, "bicg_xr", 0);
			TRY(launch(ctx, bicg_xr_kernel, dim3(nb), dim3(256), 0, n, x->d, (const double *) pp->d, (const double *) ss->d, resid->d, (const double *) ap->d, (const double *) as->d, (const double *) rhat->d, (const double *) sc, ctx->d_partial.get(), stride));
		}
		TRY(finish(3, nb)); // rho, beta, |r|
		{
			Tag tg(ctx, "bicg_p", 0);
			TRY(launch(ctx, bicg_p_kernel, dim3(grid_for(ctx, n)), dim3(256), 0, n, p->d, (const double *) ap->d, (const double *) resid->d, (const double *) sc));
		}
		its++;
		TRY(read_rnorm(&rn));
	}
	if (iterations) *iterations = its;
	if (rel_residual) *rel_residual = rn / r0_norm;
	return TGPU_OK;
}
extern "C" int tgpu_bicgstab(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *b, tgpu_vec *x, double tol, int max_it,
                             int *iterations, double *rel_residual)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, b, "tgpu_bicgstab"));
	TRY(check_level_vec(h, 0, x, "tgpu_bicgstab"));
	if (b == x) return fail(TGPU_ERR_ARG, "tgpu_bicgstab: b must not alias x");
	return bicgstab_fused(h, opts, b, x, tol, max_it, iterations, rel_residual);
	API_END
}

// ------------------------------------------------------------------------------------------
// stationary multigrid: u <- u + Cycle(f - A u), from the iterate in u
// ------------------------------------------------------------------------------------------
// sum of squares of level vector v into ctx->d_result.get()[0] (all ranks), no host read
static int k_sumsq(tgpu_hier *h, const double *v, size_t n)
{
	tgpu_ctx *ctx = h->ctx;
	const int nb  = std::min(MAX_PARTIAL, grid_for(ctx, n, 256, 8));
	Tag       tg(ctx, "reduce", 0);
	TRY(launch(ctx, reduce_stage1<0>, dim3(nb), dim3(256), 0, n, v, v, ctx->d_partial.get()));
	TRY(launch(ctx, reduce_stage2<0>, dim3(1), dim3(256), 0, nb, (const double *) ctx->d_partial.get(), ctx->d_result.get()));
	if (ctx->nranks > 1 && h->levels[0].distributed) NC(g_nccl.AllReduce(ctx->d_result.get(), ctx->d_result.get(), 1, ncclDouble, ncclSum, ctx->comm, ctx->stream));
	return TGPU_OK;
}
// ||f - A u||^2 of the full residual (r: work vector) into ctx->d_result.get()[0]
static int k_residual_sumsq(tgpu_hier *h, const double *f, const double *u, double *r)
{
	LevelDev &L = h->levels[0];
	TRY(k_extract_faces(h, 0, u, L.Fa));
	TRY(k_exchange(h, 0, L.Fa, nullptr));
	TRY(k_apply(h, 0, 1, u, f, L.Fa, r, nullptr));
	TRY(k_exchange_done(h, 0));
	return k_sumsq(h, r, L.ncells);
}
// ||f - A u||^2 into ctx->d_result.get()[0] right after a cycle that emitted the slices of its result u and kept those of the
// input of its last sweep (h->cycle_faces, h->cycle_faces_old, h->cycle_uc): face_residual_norm_kernel.  Reads S x M
// values of two face buffers per patch; neither u nor f.  The neighbours' new slices reach the halo slots first.
static int k_face_residual_norm(tgpu_hier *h)
{
	LevelDev &L   = h->levels[0];
	tgpu_ctx *ctx = h->ctx;
	double *  Fnew = h->cycle_faces;
	const double *Fold = h->cycle_faces_old, *uc = h->cycle_uc;
	if (!Fnew || !Fold) return fail(TGPU_ERR_ARG, "k_face_residual_norm: the cycle kept no boundary slices");
	TRY(k_exchange(h, 0, Fnew, nullptr));
	const int nb = std::max(1, std::min({L.P, ctx->sm_count * 8, MAX_PARTIAL}));
	{
		Tag tg(ctx, "face_residual_norm", 0);
		DISPATCH_DN_ALL(h->D, h->N, {
			const dim3   block(frn_threads<DD, NN>());
			const size_t sm = frn_smem_bytes<DD, NN>();
			TRY(flag_variant(uc != nullptr, [&](auto UC) {
				return launch(ctx, face_residual_norm_kernel<DD, NN, UC ? FV_PROLONG_DIFF : FV_DIFF>, dim3(nb), block, sm, (const PatchMeta *) L.meta.get(), L.P, (const double *) Fnew, Fold, uc, ctx->d_partial.get());
			}));
		});
		TRY(launch(ctx, reduce_stage2<0>, dim3(1), dim3(256), 0, nb, (const double *) ctx->d_partial.get(), ctx->d_result.get()));
	}
	TRY(k_exchange_done(h, 0));
	if (ctx->nranks > 1 && L.distributed) NC(g_nccl.AllReduce(ctx->d_result.get(), ctx->d_result.get(), 1, ncclDouble, ncclSum, ctx->comm, ctx->stream));
	return TGPU_OK;
}
// host read of ctx->d_result.get()[0 .. n)
static int read_result(tgpu_ctx *ctx, double *out, int n = 1)
{
	CU(cudaMemcpyAsync(ctx->h_result.get(), ctx->d_result.get(), n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
	CU(cudaStreamSynchronize(ctx->stream));
	for (int i = 0; i < n; i++) out[i] = ctx->h_result.get()[i];
	return check_comm(ctx);
}
static int check_stationary_args(tgpu_hier *h, const tgpu_vec *f, const tgpu_vec *u, const char *what)
{
	TRY(check_level_vec(h, 0, f, what));
	TRY(check_level_vec(h, 0, u, what));
	if (f == u) return fail(TGPU_ERR_ARG, std::string(what) + ": f must not alias u");
	return TGPU_OK;
}
static int ensure_gmg_ws(tgpu_hier *h)
{
	while (h->gmg_ws.size() < 2) {
		VecPtr v;
		TRY(vec_create(h, 0, v));
		h->gmg_ws.push_back(std::move(v));
	}
	return TGPU_OK;
}
// one update u <- u + Cycle(f - A u); want_norm: ||f - A u_new||^2 in ctx->d_result.get()[0] afterwards.  The fused schedule
// starts from u (guess_schedule) and takes the norm from the faces; every other schedule runs the loop it replaces:
// residual into a work vector, the cycle from zero, add, and (want_norm) a full residual of the result.
static int update_once(tgpu_hier *h, const TgpuCycleOpts *opts, const TgpuCycleOpts &o, const tgpu_vec *f, tgpu_vec *u, bool want_norm)
{
	if (guess_schedule(h, o)) {
		TRY(cycle_ptr(h, opts, f->d, u->d, want_norm, true));
		return want_norm ? k_face_residual_norm(h) : TGPU_OK;
	}
	TRY(ensure_gmg_ws(h));
	tgpu_vec *r = h->gmg_ws[0].get(), *e = h->gmg_ws[1].get();
	TRY(tgpu_residual(h, 0, f, u, r));
	TRY(cycle_ptr(h, opts, r->d, e->d));
	TRY(tgpu_vec_add(u, e));
	return want_norm ? k_residual_sumsq(h, f->d, u->d, r->d) : TGPU_OK;
}
extern "C" int tgpu_vcycle_update(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u, double *rel_residual)
{
	API_BEGIN
	TRY(check_stationary_args(h, f, u, "tgpu_vcycle_update"));
	TgpuCycleOpts o;
	TRY(cycle_opts(h, opts, o));
	TRY(update_once(h, opts, o, f, u, rel_residual != nullptr));
	if (!rel_residual) return TGPU_OK;
	double rr[2];
	CU(cudaMemcpyAsync(h->ctx->d_result.get() + 1, h->ctx->d_result.get(), sizeof(double), cudaMemcpyDeviceToDevice, h->ctx->stream));
	TRY(k_sumsq(h, f->d, f->n));
	TRY(read_result(h->ctx, rr, 2)); // ||f||^2, ||f - A u||^2
	*rel_residual = rr[0] > 0.0 ? sqrt(rr[1] / rr[0]) : sqrt(rr[1]);
	return TGPU_OK;
	API_END
}
// Stationary iteration of update_once.  The fused schedule iterates on the face norm and reports convergence only after a
// full residual confirms it (the face norm leaves out the patch solve's rounding noise, ~1e-16 relative); one host read of
// one double per cycle.
extern "C" int tgpu_gmg_solve(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u, double tol, int max_it,
                              int *iterations, double *rel_residual, double *history)
{
	API_BEGIN
	TRY(check_stationary_args(h, f, u, "tgpu_gmg_solve"));
	if (!(tol >= 0.0) || max_it < 0) return fail(TGPU_ERR_ARG, "tgpu_gmg_solve: tol and max_it must not be negative");
	TgpuCycleOpts o;
	TRY(cycle_opts(h, opts, o));
	tgpu_ctx *ctx = h->ctx;
	TRY(ensure_gmg_ws(h));
	double *r = h->gmg_ws[0]->d;
	double  fsq, rsq;
	TRY(k_sumsq(h, f->d, f->n));
	TRY(read_result(ctx, &fsq));
	const double scale = fsq > 0.0 ? 1.0 / sqrt(fsq) : 1.0; // f = 0: absolute residuals
	TRY(k_residual_sumsq(h, f->d, u->d, r));
	TRY(read_result(ctx, &rsq));
	double rel = sqrt(rsq) * scale;
	if (history) history[0] = rel;
	bool converged = rel <= tol;
	int  its       = 0;
	const bool fused = guess_schedule(h, o);
	while (!converged && its < max_it) {
		if (fused) {
			TRY(update_once(h, opts, o, f, u, true));
			TRY(read_result(ctx, &rsq));
			rel = sqrt(rsq) * scale;
			if (rel <= tol) { // confirmation by the full residual
				TRY(k_residual_sumsq(h, f->d, u->d, r));
				TRY(read_result(ctx, &rsq));
				rel = sqrt(rsq) * scale;
			}
		} else { // the loop: cycle from zero on the residual in gmg_ws[0], add, residual (also the convergence test)
			tgpu_vec *rv = h->gmg_ws[0].get(), *e = h->gmg_ws[1].get();
			TRY(cycle_ptr(h, opts, rv->d, e->d));
			TRY(tgpu_vec_add(u, e));
			TRY(k_residual_sumsq(h, f->d, u->d, rv->d));
			TRY(read_result(ctx, &rsq));
			rel = sqrt(rsq) * scale;
		}
		its++;
		if (history) history[its] = rel;
		converged = rel <= tol;
	}
	if (iterations) *iterations = its;
	if (rel_residual) *rel_residual = rel;
	return TGPU_OK;
	API_END
}

// ------------------------------------------------------------------------------------------
// boundary data and full multigrid
// ------------------------------------------------------------------------------------------
extern "C" int tgpu_boundary_sides(const tgpu_hier *h, int64_t *count, const int32_t **patch, const int8_t **side)
{
	if (!h || !count) return fail(TGPU_ERR_ARG, "tgpu_boundary_sides: null argument");
	*count = (int64_t) h->bnd_patch.size();
	if (patch) *patch = h->bnd_patch.data();
	if (side) *side = h->bnd_side.data();
	return TGPU_OK;
}
static size_t face_size(const tgpu_hier *h)
{
	size_t M = 1;
	for (int i = 0; i < h->D - 1; i++) M *= h->N;
	return M;
}
extern "C" int tgpu_boundary_vec_create(tgpu_hier *h, tgpu_vec **out)
{
	if (!h || !out) return fail(TGPU_ERR_ARG, "tgpu_boundary_vec_create: null argument");
	CU(cudaSetDevice(h->ctx->device));
	std::unique_ptr<tgpu_vec> v(new tgpu_vec());
	v->h     = h;
	v->level = BOUNDARY_LEVEL;
	v->n     = h->bnd_patch.size() * face_size(h);
	CU(cudaMallocAsync(&v->d, std::max<size_t>(1, v->n) * sizeof(double), h->ctx->stream));
	CU(cudaMemsetAsync(v->d, 0, v->n * sizeof(double), h->ctx->stream));
	*out = v.release();
	return TGPU_OK;
}
static int check_boundary_vec(const tgpu_hier *h, const tgpu_vec *b, const char *what)
{
	if (!b || b->h != h || b->level != BOUNDARY_LEVEL || b->n != h->bnd_patch.size() * face_size(h))
		return fail(TGPU_ERR_ARG, std::string(what) + ": not a boundary-data vector of this hierarchy");
	return TGPU_OK;
}
extern "C" int tgpu_fold_boundary(tgpu_hier *h, const tgpu_vec *b, tgpu_vec *f)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, f, "tgpu_fold_boundary"));
	TRY(check_boundary_vec(h, b, "tgpu_fold_boundary"));
	if (b->n == 0) return TGPU_OK;
	LevelDev &L = h->levels[0];
	Tag       tg(h->ctx, "fold_boundary", 0);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, fold_boundary_kernel<DD, NN>, dim3(grid_for(h->ctx, b->n)), dim3(256), 0, (const PatchMeta *) L.meta.get(), (int) h->bnd_patch.size(), (const int32_t *) h->bnd_patch_d.get(), (const int8_t *) h->bnd_side_d.get(), (const int32_t *) h->bnd_index.get(), (const double *) L.spacing.get(), (const double *) b->d, f->d));
	API_END
}
// level l + 1's right-hand side from level l's: coarse = R fine, and with boundary data bf (level 0: the caller's list
// layout, else level l's bnd) the Dirichlet folds re-posed for the coarse spacing, the coarse data into level l + 1's bnd
static int k_restrict_rhs(tgpu_hier *h, int l, const double *fine, const double *bf, double *coarse)
{
	LevelDev &L = h->levels[l], &C = h->levels[l + 1];
	double *  bc = bf ? C.bnd.get() : nullptr;
	const bool cross = crosses_replication(h, l);
	if (cross) {
		TRY(k_set(h, coarse, C.ncells, 0.0));
		if (bc) TRY(k_set(h, bc, C.nface, 0.0));
	}
	{
		Tag tg(h->ctx, "restrict_rhs", l);
		DISPATCH_DN_ALL(h->D, h->N, TRY(launch(h->ctx, restrict_rhs_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, fine, coarse, bf, l == 0 ? (const int32_t *) h->bnd_index.get() : (const int32_t *) nullptr, bc)));
	}
	if (cross) {
		TRY(k_allreduce_sum(h, coarse, C.ncells));
		if (bc) TRY(k_allreduce_sum(h, bc, C.nface));
	}
	return TGPU_OK;
}
static int k_fmg_interp(tgpu_hier *h, int l, const double *coarse, double *fine, double *F)
{
	LevelDev &L = h->levels[l];
	Tag       tg(h->ctx, "fmg_interp", l);
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, fmg_interp_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, coarse, fine, F));
}
// u = Cycle(f) from zero, starting on level l (run_cycle's schedules)
static int visit_from_zero(tgpu_hier *h, const TgpuCycleOpts &o, int l, const double *f, double *u)
{
	if (fused_schedule(o, h->ctx->nranks)) return fused_visit(h, o, l, f, u, false);
	TRY(k_set(h, u, h->levels[l].ncells, 0.0));
	return generic_visit(h, o, l, f, u);
}
// Full multigrid over levels 0 .. last_level: the right-hand sides restricted down (levels[l].f), the coarsest level's
// sweeps from zero, then per level the linear interpolation of the coarser solution as the guess (levels[l].u; level 0:
// the caller's f and u) and `cycles` cycles from it.  A cycle from level l uses only levels[k], k > l, as work space, whose
// right-hand sides and solutions have been consumed by then.  The fused schedule starts the first cycle of a level from
// the slices fmg_interp_kernel wrote; the others compute r = f - A u, a cycle from zero on r and the sum (update_once).
static int fmg_run(tgpu_hier *h, const TgpuCycleOpts &o, int cycles, const double *f, const double *b, double *u)
{
	const int last = h->last_level;
	auto fl = [&](int l) { return l == 0 ? f : (const double *) h->levels[l].f.get(); };
	auto ul = [&](int l) { return l == 0 ? u : h->levels[l].u.get(); };
	for (int l = 0; l < last; l++) TRY(k_restrict_rhs(h, l, fl(l), b ? (l == 0 ? b : (const double *) h->levels[l].bnd.get()) : nullptr, h->levels[l + 1].f.get()));
	TRY(visit_from_zero(h, o, last, fl(last), ul(last)));
	const bool guess = guess_schedule(h, o);
	for (int l = last - 1; l >= 0; l--) {
		LevelDev &L = h->levels[l];
		TRY(k_fmg_interp(h, l, ul(l + 1), ul(l), L.Fa));
		const double *faces = L.Fa;
		for (int c = 0; c < cycles; c++) {
			if (guess) { // every cycle but the last emits its result's slices for the next one
				const bool emit = c + 1 < cycles;
				TRY(fused_visit(h, o, l, fl(l), ul(l), emit, true, faces));
				faces = h->visit_faces;
				continue;
			}
			double *r = h->fmg_ws[2 * l]->d, *e = h->fmg_ws[2 * l + 1]->d;
			TRY(k_extract_faces(h, l, ul(l), L.Fa));
			TRY(k_exchange(h, l, L.Fa, nullptr));
			TRY(k_apply(h, l, 1, ul(l), fl(l), L.Fa, r, nullptr));
			TRY(k_exchange_done(h, l));
			TRY(visit_from_zero(h, o, l, r, e));
			Tag tg(h->ctx, "blas1", l);
			TRY(launch(h->ctx, blas1_kernel<B_ADD>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, L.ncells, ul(l), (const double *) e, (const double *) nullptr, 0.0, 0.0, 0.0));
		}
	}
	return TGPU_OK;
}
extern "C" int tgpu_fmg(tgpu_hier *h, const TgpuCycleOpts *opts, int cycles, const tgpu_vec *f, const tgpu_vec *b, tgpu_vec *u)
{
	API_BEGIN
	TRY(check_stationary_args(h, f, u, "tgpu_fmg"));
	if (b) TRY(check_boundary_vec(h, b, "tgpu_fmg"));
	if (cycles < 1) return fail(TGPU_ERR_ARG, "tgpu_fmg: cycles must be at least 1");
	TgpuCycleOpts o;
	TRY(cycle_opts(h, opts, o));
	tgpu_ctx * ctx   = h->ctx;
	const bool fused = fused_schedule(o, ctx->nranks);
	for (int l = 0; l <= h->last_level; l++) {
		TRY(ensure_work(h, l, !fused || (o.fused == 2 && is_3d32(h))));
		TRY(ensure_push_desc(h, l));
		if (b && l > 0 && !h->levels[l].bnd) CU(dev_malloc(h->levels[l].bnd, h->levels[l].nface * sizeof(double)));
	}
	if (!guess_schedule(h, o))
		for (int l = (int) h->fmg_ws.size() / 2; l < h->last_level; l++)
			for (int k = 0; k < 2; k++) {
				VecPtr v;
				TRY(vec_create(h, l, v));
				h->fmg_ws.push_back(std::move(v));
			}
	GraphEntry key;
	key.f = f->d, key.u = u->d, key.b = b ? b->d : nullptr, key.fmg_cycles = cycles;
	return graph_run(h, o, std::move(key), [&] {
		h->cycle_faces     = nullptr;
		h->cycle_faces_old = h->cycle_uc = nullptr;
		const int rc       = fmg_run(h, o, cycles, f->d, b ? b->d : nullptr, u->d);
		h->cycle_faces     = nullptr; // (a cycle of level 0 may have recorded its slices; FMG reports none)
		h->cycle_faces_old = h->cycle_uc = nullptr;
		return rc;
	});
	API_END
}

extern "C" int tgpu_init_neumann_rhs(tgpu_hier *h, int problem, tgpu_vec *f, tgpu_vec *exact)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, f, "tgpu_init_neumann_rhs"));
	if (exact) TRY(check_level_vec(h, 0, exact, "tgpu_init_neumann_rhs"));
	if (problem != 0 && problem != 1) return fail(TGPU_ERR_ARG, "tgpu_init_neumann_rhs: problem must be 0 (trig) or 1 (gauss)");
	if (h->D == 2 && problem != 0) return fail(TGPU_ERR_UNSUPPORTED, "tgpu_init_neumann_rhs: 2D has the trig problem only");
	LevelDev &L = h->levels[0];
	if (!L.starts) return fail(TGPU_ERR_ARG, "tgpu_init_neumann_rhs: hierarchy was created without patch starts");
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, init_neumann_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, (const double *) L.starts.get(), (const double *) L.spacing.get(), f->d, exact ? exact->d : (double *) nullptr, problem));
	API_END
}
extern "C" int tgpu_vec_integrate(tgpu_hier *h, const tgpu_vec *v, double *integral, double *volume)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, v, "tgpu_vec_integrate"));
	if (!integral && !volume) return fail(TGPU_ERR_ARG, "tgpu_vec_integrate: nothing asked for");
	LevelDev &L      = h->levels[0];
	const int owned  = L.P; // owned patches come first
	DevPtr<double> d_part;
	CU(dev_malloc(d_part, sizeof(double) * (size_t) std::max(owned, 1)));
	{
		Tag tg(h->ctx, "patch_integrals", 0);
		DISPATCH_DN_ALL(h->D, h->N, TRY(launch(h->ctx, patch_integrals_kernel<DD, NN>, dim3(std::min(std::max(owned, 1), h->ctx->sm_count * 8)), dim3(256), 0, owned, (const double *) L.spacing.get(), (const double *) v->d, d_part.get())));
	}
	std::vector<double> part((size_t) owned), sp((size_t) owned * h->D);
	CU(cudaMemcpyAsync(part.data(), d_part.get(), sizeof(double) * owned, cudaMemcpyDeviceToHost, h->ctx->stream));
	CU(cudaMemcpyAsync(sp.data(), L.spacing.get(), sizeof(double) * owned * h->D, cudaMemcpyDeviceToHost, h->ctx->stream));
	CU(cudaStreamSynchronize(h->ctx->stream));
	double res[2] = {0.0, 0.0};
	for (int p = 0; p < owned; p++) {
		res[0] += part[p];
		double vol = 1.0;
		for (int a = 0; a < h->D; a++) vol *= sp[(size_t) p * h->D + a] * h->N;
		res[1] += vol;
	}
	if (h->ctx->nranks > 1 && h->levels[0].distributed) { // a replicated level: every rank already holds the global sums
		DevPtr<double> d2;
		CU(dev_malloc(d2, 2 * sizeof(double)));
		CU(cudaMemcpyAsync(d2.get(), res, 2 * sizeof(double), cudaMemcpyHostToDevice, h->ctx->stream));
		TRY(k_allreduce_sum(h, d2.get(), 2));
		CU(cudaMemcpyAsync(res, d2.get(), 2 * sizeof(double), cudaMemcpyDeviceToHost, h->ctx->stream));
		CU(cudaStreamSynchronize(h->ctx->stream));
	}
	if (integral) *integral = res[0];
	if (volume) *volume = res[1];
	return TGPU_OK;
	API_END
}
extern "C" int tgpu_init_trig_rhs(tgpu_hier *h, tgpu_vec *f, tgpu_vec *exact)
{
	API_BEGIN
	TRY(check_level_vec(h, 0, f, "tgpu_init_trig_rhs"));
	if (exact) TRY(check_level_vec(h, 0, exact, "tgpu_init_trig_rhs"));
	LevelDev &L = h->levels[0];
	if (!L.starts) return fail(TGPU_ERR_ARG, "tgpu_init_trig_rhs: hierarchy was created without patch starts");
	DISPATCH_DN_ALL(h->D, h->N, return launch(h->ctx, init_trig_kernel<DD, NN>, dim3(grid_for(h->ctx, L.ncells)), dim3(256), 0, (const PatchMeta *) L.meta.get(), L.P, (const double *) L.starts.get(), (const double *) L.spacing.get(), f->d, exact ? exact->d : (double *) nullptr));
	API_END
}
