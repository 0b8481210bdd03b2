// kernels.cuh - hand-written sm_100a kernels of the GMG hot path (fp64, patch-contiguous storage).
//
// Kernel inventory (reference function each one replaces; paths relative to src/Thunderegg/):
//   smooth_kernel        SchurHelper::solveWithSolution (SchurHelper.h:319-331) =
//                        interface interpolation (TriLinInterp.cpp:60-172 / BilinearInterpolator.cpp:61-117)
//                        + StarPatchOp::addInterfaceToRHS (StarPatchOp.h:185-203)
//                        + patch solve (PatchSolvers/FftwPatchSolver.h:174-206, DftPatchSolver.h:173-216)
//                        size-generic form (and the path for patches with Neumann sides); specialised forms with the same
//                        arithmetic: smooth3d16_kernel (smooth3d16.cuh), smooth3d32c_kernel / smooth3d32n_kernel
//                        (patch3d32.cuh), smooth2d32_kernel (smooth2d32.cuh).  Patch solve = Dst2 / Dst3 transforms on
//                        D - 1 axes (dense halves: generated dst4_fast.cuh) + TriSolve on the remaining axis
//   face_residual_restrict_kernel / face_residual_restrict16_kernel   r = f - A u right after a sweep, from face data,
//                        fused with AvgRstr::restrict (GMG/Cycle.h:59-66, GMG/AvgRstr.h:78-113)
//   apply_tma_kernel / apply3d32_tma_kernel (apply_tma.cuh)   SchurHelper::apply (SchurHelper.h:361-376) +
//                        StarPatchOp::applyWithInterface (StarPatchOp.h:28-184), optionally fused with r = f - Au
//                        (GMG/Cycle.h:59-61) and AvgRstr::restrict (GMG/AvgRstr.h:78-113)
//   extract_faces_kernel the boundary-cell slices LocalData::getSliceOnSide yields (Vector.h:153-177)
//   prolong_faces_kernel / prolong_add_kernel   DrctIntp::interpolate (GMG/DrctIntp.h:80-113)
//   restrict_kernel      AvgRstr::restrict (GMG/AvgRstr.h:78-113)
//   blas1 / reduce       Vector<D> ops (Vector.h:190-321); bicg_* fused passes of BiCGStab.h:45-106
//   init_trig_kernel / init_neumann_kernel / patch_integrals_kernel   apps/shared/Init.cpp, Domain::integrate
//
// Ghost fill: the reference couples patches through interface values gamma (SURVEY App. A.2).
// Here every kernel that produces a level vector also emits the 2D boundary-cell slices of each
// patch into a contiguous "face buffer" F[patch][side][N^(D-1)]; gamma for a patch side is then
// evaluated on the fly from the patch's own face and its neighbours' opposite faces (normal,
// coarse and fine neighbours) with the reference's weights.  No interface vector is stored.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "dst4_fast.cuh"

namespace tgpu
{
enum { NBR_NONE = -1, NBR_NORMAL = 0, NBR_COARSE = 1, NBR_FINE = 2 };

// Device-side neighbour table entry: everything a kernel needs to know about one patch.
struct __align__(16) PatchMeta {
	double  inv_h2; // 1 / h^2
	double  h2;     // h^2
	int32_t parent_idx;
	int8_t  orth_on_parent; // -1: same patch on the coarser level
	uint8_t neumann;
	int8_t  nbr_type[6];
	int8_t  orth_on_coarse[6];
	int8_t  pad_[2];
	int32_t nbr_idx[6][4];
	int32_t nbr_parent[6]; // parent_idx of nbr_idx[s][0] (normal neighbours; lets the post-smoother fold the
	int8_t  nbr_orth[6];   // prolongation into its face reads without a dependent table lookup)
	int8_t  pad2_[6];
};

constexpr int TGPU_THREADS = 256;
// Programmatic dependent launch: every kernel of the library starts with this pair.  launch_dependents
// lets the next kernel of the stream be scheduled (its blocks become resident and run up to their own
// wait) while this grid is still running; wait blocks until the grids this one depends on have
// completed and flushed.  Both are no-ops for launches without the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
__device__ __forceinline__ void st_release_sys(uint64_t *p, uint64_t v)
{
	asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t *p)
{
	uint64_t v;
	asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
	return v;
}

// ---------------------------------------------------------------------------------------------
// Halo hand-over inside the compute kernels (multi-GPU, peer-to-peer exchange; protocol: tgpu.cu, "peer-to-peer halo
// exchange").  A kernel that consumes halo faces is launched over ALL owned patches of the level - interior patches
// first - and every CTA polls the peers' DATA flags itself right before the first patch that needs them (patch index >=
// first_halo_patch), so the patches without off-rank neighbours are swept while the faces are still in flight and no
// separate wait / signal launches (and no second, short launch for the boundary patches) are needed.  The last CTA to
// finish advances the generation counter and acknowledges the halo to the peers (ACK flags).
// cnt[]: 0 data sent, 1 data awaited, 2 ack sent, 3 ack awaited (generation counters of the level, device memory).
// ---------------------------------------------------------------------------------------------
struct PushDesc;
struct HaloSync {
	const PushDesc *  push          = nullptr; // != nullptr: the kernel also pushes this rank's faces first (halo_push_cta)
	const uint64_t *  data_flags    = nullptr; // my DATA flag row [nranks], written by the peers
	const int32_t *   peer_rank     = nullptr; // [npeers]
	uint64_t *const * peer_ack_flag = nullptr; // [npeers] my entry of each peer's ACK row
	uint64_t *        cnt           = nullptr;
	unsigned *        ticket        = nullptr; // CTAs that have finished
	int *             abort         = nullptr; // device flag: a wait of this hierarchy timed out
	int *             host_err      = nullptr; // mapped host flag (rank + 1 that was waited for)
	int               npeers           = 0;
	int               first_halo_patch = 0;
	int               enabled          = 0;
};
// one thread: wait until every peer's faces of the generation after "data awaited" have landed (bounded, see
// p2p_wait_kernel).  The counter is only advanced by the last CTA to finish (halo_finish), i.e. after every CTA has polled.
// (scalar arguments: a struct reference would put a copy of HaloSync on every caller's stack)
__device__ __noinline__ void halo_poll(const uint64_t *data_flags, const int32_t *peer_rank, int npeers, const uint64_t *cnt, int *abort, int *host_err)
{
	if (*abort) return;
	const uint64_t expected = cnt[1] + 1;
	for (int k = 0; k < npeers; k++) {
		const uint64_t *f = data_flags + peer_rank[k];
		unsigned long long t0;
		asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
		while (ld_acquire_sys(f) < expected) {
			unsigned long long t1;
			asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
			if (t1 - t0 > 20000000000ull) { // 20 s
				atomicExch(abort, 1);
				*(volatile int *) host_err = peer_rank[k] + 1;
				__threadfence_system();
				return;
			}
			__nanosleep(100);
		}
	}
}
// CTA-wide (every thread calls; ends with a barrier): make the halo of this level visible before patch p is gathered
__device__ __forceinline__ void halo_wait_cta(const HaloSync &hs, int p, bool &waited)
{
	if (!hs.enabled || waited || p < hs.first_halo_patch) return; // CTA-uniform
	if (threadIdx.x == 0) halo_poll(hs.data_flags, hs.peer_rank, hs.npeers, hs.cnt, hs.abort, hs.host_err);
	__syncthreads();
	waited = true;
}
// warp-wide form for kernels whose warps work on patches independently (every lane of the warp calls)
__device__ __forceinline__ void halo_wait_warp(const HaloSync &hs, int p, bool &waited)
{
	if (!hs.enabled || waited || p < hs.first_halo_patch) return; // warp-uniform
	if ((threadIdx.x & 31) == 0) halo_poll(hs.data_flags, hs.peer_rank, hs.npeers, hs.cnt, hs.abort, hs.host_err);
	__syncwarp();
	waited = true;
}
// end of the kernel: the last CTA to finish advances "data awaited" and acknowledges the halo to the peers (one thread; out
// of line, the fences and the release stores are cold code)
__device__ __noinline__ void halo_finish_thread0(unsigned *ticket, unsigned nctas, int *abort, uint64_t *cnt, uint64_t *const *peer_ack_flag, int npeers)
{
	__threadfence();
	const unsigned done = atomicAdd(ticket, 1u);
	if (done != nctas - 1) return;
	__threadfence();
	*ticket = 0;
	if (*abort) return; // the protocol stays where it broke
	cnt[1] += 1;
	const uint64_t v = cnt[2] + 1;
	__threadfence_system();
#pragma unroll 1
	for (int k = 0; k < npeers; k++) st_release_sys(peer_ack_flag[k], v);
	cnt[2] = v;
}
// (every thread calls)
__device__ __forceinline__ void halo_finish(const HaloSync &hs)
{
	if (!hs.enabled) return;
	__syncthreads();
	if (threadIdx.x == 0) halo_finish_thread0(hs.ticket, gridDim.x * gridDim.y, hs.abort, hs.cnt, hs.peer_ack_flag, hs.npeers);
}
// resident smoother CTAs per SM the register budget is tuned for (N = 32 pencils need > 128 registers)
template <int N> constexpr int smooth_min_blocks() { return N >= 32 ? 1 : 3; }

template <int D, int N> struct Geo {
	static constexpr int M   = (D == 2) ? N : N * N;     // pencils per patch = face size
	static constexpr int NC  = M * N;                    // cells per patch
	static constexpr int S   = 2 * D;                    // sides
	static constexpr int Q   = 1 << (D - 1);             // fine neighbours per side
	static constexpr int PPB = TGPU_THREADS / M;         // patches per block
	static constexpr int ROW = N + 1;                    // padded row (bank-conflict-free pencils)
	static constexpr int SP  = M * ROW;                  // padded patch size in smem (doubles)
	static constexpr int NG  = N + 2;                    // row with ghosts
	static constexpr int GP  = (D == 2) ? NG * NG : NG * NG * NG;
};

// ---------------------------------------------------------------------------------------------
// transform tables (DftPatchSolver.h:237-289), symmetric halves only.
//   fwd[k*H + j] = sin(pi/N (k+1)(j+1/2)),            k < N, j < H = N/2      (DST-II rows)
//   inv[i*N + j] = sin(pi/N (i+1/2)(j+1)), j < N-1;  inv[i*N + N-1] = 0.5 (-1)^i,  i < H  (DST-III rows)
// No kernel reads them (the transforms take their coefficients from Mags below).  They stay because they sit in front of
// c_mag* in constant bank 3: removing them moves every c_mag32 operand and so changes the machine code of the 32^3 kernels.
// ---------------------------------------------------------------------------------------------
__constant__ double c_fwd4[4 * 2], c_inv4[2 * 4];
__constant__ double c_fwd8[8 * 4], c_inv8[4 * 8];
__constant__ double c_fwd16[16 * 8], c_inv16[8 * 16];
__constant__ double c_fwd32[32 * 16], c_inv32[16 * 32];

// Every entry of the DST-II / DST-III matrices is +-sin(i pi / 2N), i = 1..N: N distinct magnitudes.
// For N <= 16 they live in registers for the whole kernel (loaded once from c_mag*), so the
// transforms are pure register DFMA/DADD streams with no constant fetches; the sign is folded into
// the DFMA operand modifier.  N = 32 (66 registers of magnitudes) keeps the constant-bank tables.
__constant__ double c_mag4[5], c_mag8[9], c_mag16[17], c_mag32[33];
template <int N> struct Mags {
	static constexpr bool IN_REGS = (N <= 16);
	double                m[IN_REGS ? N + 1 : 1];
	__device__ __forceinline__ void load()
	{
		if (IN_REGS) {
#pragma unroll
			for (int i = 0; i <= N; i++) m[i] = (N == 4) ? c_mag4[i] : (N == 8) ? c_mag8[i] : c_mag16[i];
		}
	}
	// sin(pi a / 2N) for a compile-time (after unrolling) integer a
	__device__ __forceinline__ double sinq(int a) const
	{
		a %= 4 * N;
		const bool neg = a >= 2 * N;
		if (neg) a -= 2 * N;
		if (a > N) a = 2 * N - a;
		const double mag = IN_REGS ? m[IN_REGS ? a : 0] : c_mag32[a]; // N = 32: constant-bank operand (compile-time index)
		return neg ? -mag : mag;
	}
};

template <int H> __device__ __forceinline__ void dst4_fast(const double (&x)[H], double (&y)[H])
{
	if constexpr (H == 32) dst4_32(x, y);
	else if constexpr (H == 16) dst4_16(x, y);
	else if constexpr (H == 8) dst4_8(x, y);
}
// DST-II of a register pencil.  S[k][j] = sin(pi (k+1)(2j+1) / 2n)  (DftPatchSolver.h:262-268).
// Symmetry S[k][n-1-j] = (-1)^k S[k][j] splits the transform into
//   even k = 2m:   sum_j sin(pi (2m+1)(2j+1) / 2n) e_j        (dense n/2 x n/2, a DST-IV)
//   odd  k = 2m+1: sum_j sin(pi (m+1)(2j+1) / n)   o_j        (= DST-II of size n/2 on o -> recursion)
// with e_j = x_j + x_{n-1-j}, o_j = x_j - x_{n-1-j}.  Cost for n = 16: 116 fp64 ops instead of 256.
// NT is the top-level pencil length (owner of the magnitude table), n the current size.
template <int NT, int n> struct Dst2 {
	static constexpr int SC = NT / n; // sin(pi a / 2n) = sinq_NT(SC a)
	__device__ static __forceinline__ void run(double (&v)[n], const Mags<NT> &mg)
	{
		constexpr int H = n / 2;
		double        e[H], o[H];
#pragma unroll
		for (int j = 0; j < H; j++) {
			e[j] = v[j] + v[n - 1 - j];
			o[j] = v[j] - v[n - 1 - j];
		}
		// the even outputs are a DST-IV of e; dense halves of size 8 and 16 go through the FFT-based straight-line code of
		// dst4_fast.cuh (45 / 119 instructions instead of 64 / 256)
		if (H == 16 || H == 8) {
			double y[H];
			dst4_fast<H>(e, y);
#pragma unroll
			for (int mm = 0; mm < H; mm++) v[2 * mm] = y[mm];
		} else {
#pragma unroll
			for (int mm = 0; mm < H; mm++) {
				double acc = 0.0;
#pragma unroll
				for (int j = 0; j < H; j++) acc = fma(mg.sinq(SC * (2 * mm + 1) * (2 * j + 1)), e[j], acc);
				v[2 * mm] = acc;
			}
		}
		Dst2<NT, H>::run(o, mg);
#pragma unroll
		for (int mm = 0; mm < H; mm++) v[2 * mm + 1] = o[mm];
	}
};
template <int NT> struct Dst2<NT, 1> {
	__device__ static __forceinline__ void run(double (&v)[1], const Mags<NT> &) { /* sin(pi/2) x_0 */ }
};
// DST-III of a register pencil.  T[i][j] = sin(pi (2i+1)(j+1) / 2n), T[i][n-1] = 0.5 (-1)^i
// (DftPatchSolver.h:269-281).  T[n-1-i][j] = (-1)^j T[i][j]  =>  y_i = E_i + O_i, y_{n-1-i} = E_i - O_i with
//   E_i = sum_{j even} T[i][j] x_j                  (dense n/2 x n/2)
//   O_i = sum_{l} sin(pi (2i+1)(l+1) / n) x_{2l+1}  (= DST-III of size n/2 on the odd inputs -> recursion)
template <int NT, int n> struct Dst3 {
	static constexpr int SC = NT / n;
	__device__ static __forceinline__ void run(double (&v)[n], const Mags<NT> &mg)
	{
		constexpr int H = n / 2;
		double        E[H], O[H];
#pragma unroll
		for (int l = 0; l < H; l++) O[l] = v[2 * l + 1];
		if (H == 16 || H == 8) { // E is a DST-IV of the even inputs (dst4_fast.cuh, as in Dst2)
			double x[H];
#pragma unroll
			for (int l = 0; l < H; l++) x[l] = v[2 * l];
			dst4_fast<H>(x, E);
		} else {
#pragma unroll
			for (int i = 0; i < H; i++) {
				double acc = 0.0;
#pragma unroll
				for (int l = 0; l < H; l++) acc = fma(mg.sinq(SC * (2 * i + 1) * (2 * l + 1)), v[2 * l], acc);
				E[i] = acc;
			}
		}
		Dst3<NT, H>::run(O, mg);
#pragma unroll
		for (int i = 0; i < H; i++) {
			v[i]         = E[i] + O[i];
			v[n - 1 - i] = E[i] - O[i];
		}
	}
};
template <int NT> struct Dst3<NT, 1> {
	__device__ static __forceinline__ void run(double (&v)[1], const Mags<NT> &) { v[0] *= 0.5; }
};

// Tridiagonal solve along one axis once the other axes are diagonalised ("matrix decomposition": two transform
// pairs + one Thomas solve instead of three transform pairs; same patch solve as FftwPatchSolver.h:174-206 /
// DftPatchSolver.h:173-216 in exact arithmetic, 56 fp64 operations per pencil instead of 248).
// For the pencil with transform indices (k_a, k_b) the remaining system is  M y = h^2 r,
//   M = tridiag(1, d_j, 1),  d_j = mu - 2 (mu - 3 at both ends: the Dirichlet closure of StarPatchOp.h:46-64),
//   mu = -4 sin^2((k_a+1) pi/2n) - 4 sin^2((k_b+1) pi/2n).
// M is symmetric under j -> n-1-j, so it is eliminated from both ends towards the middle with ONE set of
// multipliers a_0 = 1/d_0, a_j = 1/(d_j - a_{j-1}) (two independent dependency chains of n/2), leaving
//   y_j + a_j y_{j+1} = rho_j (j < n/2),  y_{n-1-j} + a_j y_{n-2-j} = rho'_j,  and a 2 x 2 system in the middle.
// tab[j * STRIDE + pencil] = a_j (j < n/2), tab[(n/2) * STRIDE + pencil] = 1 / (1 - a_{n/2-1}^2); the (2/n)^(D-1) of
// the transform pairs (DftPatchSolver.h:214) and h^2 are folded into the right-hand side.  (2D: mu has one term.)
template <int N, int STRIDE = 256> struct TriSolve { // STRIDE: pencils per table row
	static constexpr int H = N / 2;
	// v -> (rho_0..rho_{H-1}, rho'_{H-1}..rho'_0), both scaled
	// hs = h^2 (2/n)^(D-1): the scaling of the D-1 transform pairs (DftPatchSolver.h:214)
	__device__ static __forceinline__ void forward(double (&v)[N], const double *__restrict__ tab, double hs)
	{
		double       a  = __ldg(tab);
		double       sa = hs * a;
		v[0]            = v[0] * sa;
		v[N - 1]        = v[N - 1] * sa;
#pragma unroll
		for (int j = 1; j < H; j++) {
			a            = __ldg(tab + j * STRIDE);
			sa           = hs * a;
			v[j]         = fma(-a, v[j - 1], v[j] * sa);
			v[N - 1 - j] = fma(-a, v[N - j], v[N - 1 - j] * sa);
		}
	}
	__device__ static __forceinline__ void backward(double (&v)[N], const double *__restrict__ tab)
	{
		const double a = __ldg(tab + (H - 1) * STRIDE), kap = __ldg(tab + H * STRIDE);
		const double yt = kap * fma(-a, v[H], v[H - 1]), yb = kap * fma(-a, v[H - 1], v[H]);
		v[H - 1] = yt;
		v[H]     = yb;
#pragma unroll
		for (int j = H - 2; j >= 0; j--) {
			const double aj = __ldg(tab + j * STRIDE);
			v[j]            = fma(-aj, v[j + 1], v[j]);
			v[N - 1 - j]    = fma(-aj, v[N - 2 - j], v[N - 1 - j]);
		}
	}
};


// cp.async (LDGSTS) 8-byte copy global -> shared; !valid zero-fills (src-size 0)
__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gsrc, bool valid)
{
	const unsigned s  = (unsigned) __cvta_generic_to_shared(smem_dst);
	const int      sz = valid ? 8 : 0;
	asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int PENDING> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(PENDING) : "memory"); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p)); }

// cell index inside a patch of face entry m on side s (Vector.h:153-177: the slice drops axis s/2
// and keeps the remaining axes in order)
template <int D, int N> __device__ __forceinline__ void face_cell(int s, int m, int (&c)[3])
{
	const int ax  = s >> 1;
	const int pos = (s & 1) ? N - 1 : 0;
	if (D == 2) {
		c[ax]     = pos;
		c[1 - ax] = m;
		c[2]      = 0;
	} else {
		const int i = m % N, j = m / N;
		if (ax == 0) c[0] = pos, c[1] = i, c[2] = j;
		else if (ax == 1) c[0] = i, c[1] = pos, c[2] = j;
		else c[0] = i, c[1] = j, c[2] = pos;
	}
}

// coarse cell that fine cell c of a patch with orthant `orth` on its parent lies in (DrctIntp.h:92-111)
template <int D, int N> __device__ __forceinline__ int parent_cell(int orth, const int (&c)[3])
{
	if (orth < 0) return (c[2] * N + c[1]) * N + c[0];
	const int cx = (c[0] + (orth & 1) * N) / 2, cy = (c[1] + ((orth >> 1) & 1) * N) / 2;
	const int cz = (D == 2) ? 0 : (c[2] + ((orth >> 2) & 1) * N) / 2;
	return (cz * N + cy) * N + cx;
}
// ---------------------------------------------------------------------------------------------
// Producer side of the halo hand-over inside the consumer kernel: before a CTA of a sweep / face-residual launch touches
// its patches it stores its share of this rank's boundary faces (optionally + the prolonged coarse correction, as
// push_faces_kernel) into the peers' halo slots; the last CTA to finish publishes DATA.  The stores then overlap the
// launch's work on the patches without off-rank neighbours and no separate push launch sits on the critical path.
// Needs every CTA of the grid to become resident without waiting for another CTA of the same grid to retire (the
// host clamps the grid to the occupancy, see halo_launch, tgpu.cu): CTAs poll for the peers' faces later on, and the
// peers' faces are published by the last of THEIR CTAs.
// Lives in device memory, one per (level, face buffer, with / without prolongation); written once at set-up.
// ---------------------------------------------------------------------------------------------
struct PushDesc {
	const int32_t *   patch, *side, *peer_of, *ridx; // [nfaces] send list (LevelDev)
	const double *    F;                              // face buffer the faces are read from
	const double *    uc;                             // != nullptr: + (P uc) on the boundary cells
	double *const *   peerF;                          // [nranks] the peers' mapping of the same face buffer
	const uint64_t *  ack_flags;                      // my ACK flag row [nranks]
	const int32_t *   peer_rank;                      // [npeers]
	uint64_t *const * peer_data_flag;                 // [npeers] my entry of each peer's DATA row
	uint64_t *        cnt;                            // generation counters of the level (HaloSync)
	unsigned *        ticket;
	int *             abort;
	int *             host_err;
	int               nfaces, npeers;
};
// every thread of every CTA of the launch calls this once, before any halo wait (contains CTA barriers)
template <int D, int N> __device__ __noinline__ void halo_push_cta(const PatchMeta *__restrict__ meta, const PushDesc *__restrict__ pd)
{
	using G             = Geo<D, N>;
	const unsigned nctas = gridDim.x * gridDim.y * gridDim.z;
	const unsigned cta   = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
	const unsigned nthr  = blockDim.x * blockDim.y * blockDim.z;
	const unsigned tid   = (threadIdx.z * blockDim.y + threadIdx.y) * blockDim.x + threadIdx.x;
	int *const     abort = pd->abort;
	uint64_t *const cnt  = pd->cnt;
	const int      npeers = pd->npeers;
	if (tid == 0 && !*abort) { // the peers must have consumed the previous generation of my faces before their slots are rewritten
		const uint64_t expected = cnt[3];
		for (int k = 0; k < npeers; k++) {
			const uint64_t *f = pd->ack_flags + pd->peer_rank[k];
			unsigned long long t0;
			asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
			while (ld_acquire_sys(f) < expected) {
				unsigned long long t1;
				asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
				if (t1 - t0 > 20000000000ull) { // 20 s
					atomicExch(abort, 1);
					*(volatile int *) pd->host_err = pd->peer_rank[k] + 1;
					__threadfence_system();
					break;
				}
				__nanosleep(100);
			}
		}
	}
	__syncthreads();
	const int32_t *patch = pd->patch, *side = pd->side, *peer_of = pd->peer_of, *ridx = pd->ridx;
	const double * F = pd->F, *uc = pd->uc;
	double *const *peerF = pd->peerF;
	const size_t   total = (size_t) pd->nfaces * G::M;
	for (size_t i = (size_t) cta * nthr + tid; i < total; i += (size_t) nctas * nthr) {
		const int m = (int) (i % G::M), k = (int) (i / G::M);
		const int p = patch[k], s = side[k];
		double    v = F[((size_t) p * G::S + s) * G::M + m];
		if (uc) {
			int c[3];
			face_cell<D, N>(s, m, c);
			v += __ldg(uc + (size_t) meta[p].parent_idx * G::NC + parent_cell<D, N>(meta[p].orth_on_parent, c));
		}
		peerF[peer_of[k]][(size_t) ridx[k] * G::M + m] = v;
	}
	__syncthreads();
	if (tid == 0) { // the last CTA publishes the faces: DATA generation + 1 in every peer's flag row
		__threadfence_system();
		if (atomicAdd(pd->ticket, 1u) == nctas - 1) {
			__threadfence_system();
			*pd->ticket = 0;
			if (!*abort) {
				cnt[3] += 1;
				const uint64_t v = cnt[0] + 1;
				for (int k = 0; k < npeers; k++) st_release_sys(pd->peer_data_flag[k], v);
				cnt[0] = v;
			}
		}
	}
}
template <int D, int N> __device__ __forceinline__ void halo_push(const HaloSync &hs, const PatchMeta *__restrict__ meta)
{
	if (hs.enabled && hs.push) halo_push_cta<D, N>(meta, hs.push); // grid-uniform
}
// Accessor for "boundary value idx on side s of patch q".  Plain: the face buffer entry.  With a
// coarse vector attached (post-smoothing right after the coarse-grid correction) the piecewise
// constant prolongation of the correction, DrctIntp.h:92-111, is added on the fly, so the
// prolonged fine vector is never materialised: F holds the faces of the pre-smoothed u.
enum { FV_PLAIN = 0, FV_PROLONG = 1, FV_DIFF = 2, FV_NEG = 3, FV_PROLONG_DIFF = 4 };
// FV_DIFF: F2 - F (old minus new boundary values) and FV_NEG: -F; gamma is linear in the boundary
// values, so these give gamma(u_old) - gamma(u_new) directly (face-supported residual, see
// face_residual_restrict_kernel).  FV_PROLONG_DIFF: (Fold + P uc) - F, the same difference when the old
// iterate is the input of a first post-sweep (pre-smoothed u plus the prolonged correction, formed on the fly).
template <int D, int N, int MODE> struct FaceVals {
	using G = Geo<D, N>;
	const double *__restrict__ F;
	const double *__restrict__ uc; // FV_PROLONG, FV_PROLONG_DIFF: coarse vector; FV_DIFF: the old face buffer F2
	const PatchMeta *__restrict__ meta;
	const double *__restrict__ Fold = nullptr; // FV_PROLONG_DIFF: faces of the pre-smoothed u
	__device__ __forceinline__ double get(int q, int par, int orth, int s, int idx) const
	{
		const size_t o = ((size_t) q * G::S + s) * G::M + idx;
		double       v = __ldg(F + o);
		if (MODE == FV_NEG) v = -v;
		if (MODE == FV_DIFF) v = __ldg(uc + o) - v;
		if (MODE == FV_PROLONG && par >= 0) { // par < 0: halo slot whose face already arrived with the correction added
			int c[3];
			face_cell<D, N>(s, idx, c);
			v += __ldg(uc + (size_t) par * G::NC + parent_cell<D, N>(orth, c));
		}
		if (MODE == FV_PROLONG_DIFF) {
			double w = __ldg(Fold + o);
			if (par >= 0) {
				int c[3];
				face_cell<D, N>(s, idx, c);
				w += __ldg(uc + (size_t) par * G::NC + parent_cell<D, N>(orth, c));
			}
			v = w - v;
		}
		return v;
	}
	// slow-path variant: looks the parent of q up in the neighbour table
	__device__ __forceinline__ double get(int q, int s, int idx) const
	{
		int par = 0, orth = -1;
		if (MODE == FV_PROLONG || MODE == FV_PROLONG_DIFF) {
			par  = meta[q].parent_idx;
			orth = meta[q].orth_on_parent;
		}
		return get(q, par, orth, s, idx);
	}
};

// ---------------------------------------------------------------------------------------------
// interface value gamma for entry m of side s of patch p (general version, all neighbour types).
// Weights: SURVEY App. A.2 (TriLinInterp.cpp:60-172, BilinearInterpolator.cpp:61-117);
// which contributions meet on an interface: SchurInfo.h:141-150,253-259,363-370.
// ---------------------------------------------------------------------------------------------
template <int D, int N, int MODE>
__device__ __forceinline__ double iface_gamma(const PatchMeta &pm, int p, int s, int m, const FaceVals<D, N, MODE> &fv)
{
	const int    po = pm.parent_idx, oo = pm.orth_on_parent;
	const double a  = fv.get(p, po, oo, s, m);
	const int    t  = pm.nbr_type[s];
	if (t == NBR_NORMAL) return 0.5 * a + 0.5 * fv.get(pm.nbr_idx[s][0], s ^ 1, m);
	if (t == NBR_COARSE) {
		const int orth = pm.orth_on_coarse[s];
		const int nb   = pm.nbr_idx[s][0];
		if (D == 2) {
			const double f2f = 5.0 / 6 * a - 1.0 / 6 * fv.get(p, po, oo, s, m ^ 1);
			return f2f + 2.0 / 6 * fv.get(nb, s ^ 1, (m + (orth & 1) * N) / 2);
		} else {
			const int    i = m % N, j = m / N;
			const int    i0 = i & ~1, j0 = j & ~1;
			const int    self = (i & 1) | ((j & 1) << 1);
			double       acc  = 11 * a;
#pragma unroll
			for (int q = 0; q < 4; q++)
				if (q != self) acc -= fv.get(p, po, oo, s, (j0 + (q >> 1)) * N + i0 + (q & 1));
			const int ci = (i + (orth & 1) * N) / 2, cj = (j + ((orth >> 1) & 1) * N) / 2;
			return acc / 12.0 + 4.0 * fv.get(nb, s ^ 1, cj * N + ci) / 12.0;
		}
	}
	// NBR_FINE: I am the coarse side
	if (D == 2) {
		const int q  = m >= N / 2;
		const int fi = 2 * (m % (N / 2));
		const int nb = pm.nbr_idx[s][q];
		return 1.0 / 3 * a + (1.0 / 3 * fv.get(nb, s ^ 1, fi) + 1.0 / 3 * fv.get(nb, s ^ 1, fi + 1));
	} else {
		const int i = m % N, j = m / N;
		const int q  = (i >= N / 2) | ((j >= N / 2) << 1);
		const int fi = 2 * (i % (N / 2)), fj = 2 * (j % (N / 2));
		const int nb = pm.nbr_idx[s][q];
		double    g  = 2.0 / 6.0 * a;
		g += 1.0 / 6.0 * fv.get(nb, s ^ 1, fj * N + fi);
		g += 1.0 / 6.0 * fv.get(nb, s ^ 1, fj * N + fi + 1);
		g += 1.0 / 6.0 * fv.get(nb, s ^ 1, (fj + 1) * N + fi);
		g += 1.0 / 6.0 * fv.get(nb, s ^ 1, (fj + 1) * N + fi + 1);
		return g;
	}
}

// gamma of entry m on all sides at once.  The own-face and (first) neighbour-face loads of all sides
// are issued back to back without control flow in between, so a patch costs two dependent memory
// round trips (neighbour table, faces) instead of one per side; only refinement-boundary sides take
// the slow path through iface_gamma.  a[s] returns the patch's own boundary value.
template <int D, int N, int MODE>
__device__ __forceinline__ void gamma_all_sides(const PatchMeta &pm, int p, int m, const FaceVals<D, N, MODE> &fv,
                                                int (&ty)[2 * D], double (&a)[2 * D], double (&gam)[2 * D])
{
	using G = Geo<D, N>;
	double b[G::S];
	int    q[G::S], qp[G::S], qo[G::S];
	const int po = pm.parent_idx, oo = pm.orth_on_parent;
#pragma unroll
	for (int s = 0; s < G::S; s++) {
		ty[s] = pm.nbr_type[s];
		q[s]  = ty[s] == NBR_NONE ? p : pm.nbr_idx[s][0];
		qp[s] = ty[s] == NBR_NORMAL ? pm.nbr_parent[s] : po; // any valid index keeps the load harmless
		qo[s] = ty[s] == NBR_NORMAL ? pm.nbr_orth[s] : oo;
	}
#pragma unroll
	for (int s = 0; s < G::S; s++) a[s] = fv.get(p, po, oo, s, m);
#pragma unroll
	for (int s = 0; s < G::S; s++) b[s] = fv.get(q[s], qp[s], qo[s], s ^ 1, m);
#pragma unroll
	for (int s = 0; s < G::S; s++) {
		gam[s] = 0.5 * a[s] + 0.5 * b[s];
		if (ty[s] > NBR_NORMAL) gam[s] = iface_gamma<D, N, MODE>(pm, p, s, m, fv);
	}
}

// L2 prefetch of everything iface_gamma will read for patch p (own faces and the neighbours' opposite
// faces), one 128-byte line per call slot; the M threads of a patch share the work.  Issued one
// persistent-loop iteration ahead so that the demand loads of the next iteration hit L2.
template <int D, int N>
__device__ __forceinline__ void prefetch_faces_l2(const PatchMeta *__restrict__ meta, int p, int m, const double *__restrict__ F)
{
	using G              = Geo<D, N>;
	constexpr int LPF    = (G::M * 8 + 127) / 128; // lines per face
	constexpr int ITEMS  = G::S * (1 + G::Q) * LPF;
	const PatchMeta &pm  = meta[p];
	for (int i = m; i < ITEMS; i += G::M) {
		const int line = i % LPF, j = (i / LPF) % (1 + G::Q), s = i / (LPF * (1 + G::Q));
		const int t    = pm.nbr_type[s];
		if (j == 0) {
			prefetch_l2(F + ((size_t) p * G::S + s) * G::M + line * 16);
		} else if (t != NBR_NONE && (j == 1 || t == NBR_FINE)) {
			prefetch_l2(F + ((size_t) pm.nbr_idx[s][j - 1] * G::S + (s ^ 1)) * G::M + line * 16);
		}
	}
}
template <int D, int N> __device__ __forceinline__ void prefetch_patch_l2(const double *__restrict__ v, int p, int m)
{
	using G = Geo<D, N>;
	for (int i = m * 16; i < G::NC; i += G::M * 16) prefetch_l2(v + (size_t) p * G::NC + i);
}

// ---------------------------------------------------------------------------------------------
// Patches with Neumann domain sides (PatchSolvers/FftwPatchSolver.h:115-127, DftPatchSolver.h:115-127,150-165):
// per axis the transform pair and eigenvalues depend on the two closures,
//   Dirichlet/Dirichlet DST-II / DST-III, -4 sin^2((k+1) pi/2n)     Neumann/Neumann  DCT-II / DCT-III, -4 sin^2(k pi/2n)
//   Neumann/Dirichlet   DCT-IV / DCT-IV,  -4 sin^2((k+1/2) pi/2n)   Dirichlet/Neumann DST-IV / DST-IV, same
// They take a general path: dense n x n transforms with the matrices of DftPatchSolver.h:237-289 read from
// a table (mats[kind][k][j], kinds in the order below) and the eigenvalue sum formed on the fly from
// lam[shift kind][k]; an all-Neumann patch gets its zero mode removed (FftwPatchSolver.h:197).
// ---------------------------------------------------------------------------------------------
enum { TK_DST_II = 0, TK_DST_III = 1, TK_DCT_II = 2, TK_DCT_III = 3, TK_DCT_IV = 4, TK_DST_IV = 5 };
struct AxisKind {
	int fwd, inv, lam;
};
__device__ __forceinline__ AxisKind axis_kind(int neumann_bits, int axis)
{
	const bool lo = (neumann_bits >> (2 * axis)) & 1, hi = (neumann_bits >> (2 * axis + 1)) & 1;
	if (lo && hi) return {TK_DCT_II, TK_DCT_III, 1};
	if (lo) return {TK_DCT_IV, TK_DCT_IV, 2};
	if (hi) return {TK_DST_IV, TK_DST_IV, 2};
	return {TK_DST_II, TK_DST_III, 0};
}
// y_k = sum_j T[k][j] v_j, written straight into the pencil's shared-memory slots q[k * step]
template <int N>
__device__ __forceinline__ void dense_to_smem(const double *__restrict__ T, const double (&v)[N], double *q, int step)
{
	// two rows per trip, matrix rows read 16 bytes at a time (every thread of the patch reads the same address: one
	// broadcast request per load); the sums run over j in the same order as the scalar form
#pragma unroll 1
	for (int k = 0; k < N; k += 2) {
		const double2 *r0 = reinterpret_cast<const double2 *>(T + k * N), *r1 = reinterpret_cast<const double2 *>(T + (k + 1) * N);
		double         a0 = 0.0, a1 = 0.0;
#pragma unroll
		for (int j = 0; j < N / 2; j++) {
			const double2 t0 = __ldg(r0 + j), t1 = __ldg(r1 + j);
			a0 = fma(t0.x, v[2 * j], a0);
			a0 = fma(t0.y, v[2 * j + 1], a0);
			a1 = fma(t1.x, v[2 * j], a1);
			a1 = fma(t1.y, v[2 * j + 1], a1);
		}
		q[k * step]       = a0;
		q[(k + 1) * step] = a1;
	}
}

// One axis of the general patch solve: y = T_kind v, stored to q[k * step].  The four kinds that occur on a patch with at
// most one Neumann side per axis have fast forms: DST-II / DST-III (the Dirichlet transforms of the plain path) and, for
// n = 8, 16 and 32, DST-IV (generated FFT-based code, dst4_fast.cuh) and DCT-IV = DST-IV of the reversed input with alternating
// signs (cos(pi (2k+1)(2j+1) / 4n) = (-1)^k sin(pi (2k+1)(2(n-1-j)+1) / 4n)).  DCT-II / DCT-III (Neumann on both sides of an
// axis: patches that span the whole domain) and the other sizes keep the dense matrix (DftPatchSolver.h:237-289).
template <int N>
__device__ __forceinline__ void general_transform(const double *__restrict__ mats, int kind, double (&v)[N], double *q, int step, const Mags<N> &mg)
{
	constexpr bool FAST4 = N == 32 || N == 16 || N == 8;
	if (kind == TK_DST_II || kind == TK_DST_III) {
		if (kind == TK_DST_II) Dst2<N, N>::run(v, mg);
		else Dst3<N, N>::run(v, mg);
#pragma unroll
		for (int k = 0; k < N; k++) q[k * step] = v[k];
	} else if (FAST4 && (kind == TK_DST_IV || kind == TK_DCT_IV)) {
		const bool c4 = kind == TK_DCT_IV;
		double     x[N], y[N];
#pragma unroll
		for (int j = 0; j < N; j++) x[j] = c4 ? v[N - 1 - j] : v[j];
		dst4_fast<N>(x, y);
#pragma unroll
		for (int k = 0; k < N; k++) q[k * step] = (c4 && (k & 1)) ? -y[k] : y[k];
	} else {
		dense_to_smem<N>(mats + kind * N * N, v, q, step);
	}
}

// ---------------------------------------------------------------------------------------------
// block-Jacobi smoother: u_p <- S_p^-1 (f_p - (2/h^2) E^T gamma(F_in)),  one exact DST patch solve
// per patch, all in shared memory / registers.  256 threads handle PPB = 256 / N^(D-1) patches.
//   ZERO_GUESS: gamma == 0 (first sweep of a cycle, GMG/Cycle.h:118 u->set(0)), F_in is not read.
//   EMIT:       also write the new boundary-cell slices to F_out.
//   PROLONG:    face values are F_in + (P u_coarse) on the boundary cells (see FaceVals).
// tri: TriSolve's multiplier table for the x axis, [j][row m] (rows m = (k_y, k_z) after the transforms along y and z)
// ---------------------------------------------------------------------------------------------
template <int D, int N, bool ZERO_GUESS, bool EMIT, bool PROLONG>
__global__ void __launch_bounds__(TGPU_THREADS, smooth_min_blocks<N>())
smooth_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ f, double *__restrict__ u,
              const double *__restrict__ Fin, double *__restrict__ Fout, const double *__restrict__ tri,
              const double *__restrict__ uc, const double *__restrict__ mats, const double *__restrict__ lam, double lam_shift,
              int only_neumann = 0)
{
	// only_neumann != 0: only patches with Neumann domain sides are swept - the others of the range belong to a specialised
	// kernel launched over the same range (smooth3d16_kernel / smooth2d32_kernel with skip_neumann)
	// lam_shift: the patch solver's "lambda" (FftwPatchSolver.h:66,170, DftPatchSolver.h:78,168): the patch problems are
	// (Laplacian + lambda) u = rhs; != 0 sends every patch through the general transform path, whose eigenvalue sums are
	// formed on the fly
	// works on patches [p0, P) (multi-GPU: interior and boundary patches are separate launches)
	// Persistent CTAs: each loops over groups of PPB patches (group g = blockIdx.x + k gridDim.x).
	// The right-hand side of the NEXT group streams into the second shared-memory buffer with
	// cp.async while the current group is being solved (double buffering).
	using G = Geo<D, N>;
	static_assert(G::M <= TGPU_THREADS, "patch face larger than the block");
	pdl_launch_dependents();
	pdl_wait();
	extern __shared__ double smem[];
	double *Sbuf0 = smem;                      // [PPB][SP]
	double *Sbuf1 = smem + G::PPB * G::SP;     // [PPB][SP]

	const int t    = threadIdx.x;
	const int pp   = t / G::M;
	const int m    = t % G::M;
	const int nblk = (P - p0 + G::PPB - 1) / G::PPB;

	Mags<N> mg;
	mg.load();

	auto mine = [&](int g) { // does this CTA sweep group g at all?  (CTA-uniform: any patch of the group with Neumann sides)
		if (!only_neumann) return true;
		bool any = false;
		for (int k = 0; k < G::PPB; k++) any = any || (p0 + g * G::PPB + k < P && meta[p0 + g * G::PPB + k].neumann != 0);
		return any;
	};
	auto prefetch = [&](int g, double *Sdst) {
		const int pb = p0 + g * G::PPB;
		if (!mine(g)) return;
#pragma unroll
		for (int k = 0; k < N; k++) {
			const int  e  = t + TGPU_THREADS * k;
			const int  lp = e / G::NC, c = e % G::NC;
			const bool ok = pb + lp < P;
			cp_async8(Sdst + lp * G::SP + (c / N) * G::ROW + (c % N), ok ? f + (size_t) (pb + lp) * G::NC + c : f, ok);
		}
	};

	int g = blockIdx.x;
	if (g < nblk) prefetch(g, Sbuf0);
	cp_async_commit();

	for (int it = 0; g < nblk; g += gridDim.x, it++) {
		double *   Sall  = (it & 1) ? Sbuf1 : Sbuf0;
		const int  p     = p0 + g * G::PPB + pp;
		const bool valid = p < P && (!only_neumann || meta[p].neumann != 0); // only_neumann: the other patches of the group idle
		// the other buffer was last read in the previous iteration, before its closing barrier
		if (g + (int) gridDim.x < nblk) {
			prefetch(g + gridDim.x, (it & 1) ? Sbuf0 : Sbuf1);
			if (!ZERO_GUESS && mine(g + gridDim.x)) { // pull the faces the next group's gamma needs into L2 one iteration ahead
				const int pn = p0 + (g + gridDim.x) * G::PPB + pp;
				if (pn < P) prefetch_faces_l2<D, N>(meta, pn, m, Fin);
			}
		}
		cp_async_commit();
		if (!mine(g)) continue; // (no barrier has been passed in this iteration; the buffers alternate as before)

		double *S = Sall + pp * G::SP;
		double  cfac = 0.0, h2 = 0.0;
		int     neu  = 0; // Neumann domain sides of this patch: != 0 takes the general transform path
		bool    general = false;
		int8_t  ntype[6] = {-1, -1, -1, -1, -1, -1};
		double  gam[6]   = {0, 0, 0, 0, 0, 0}; // (2/h^2) gamma of entry m on each side
		if (valid) {
			const PatchMeta &pm = meta[p];
			cfac                = 2.0 * pm.inv_h2;
			h2                  = pm.h2;
			neu                 = pm.neumann;
			general             = neu != 0 || lam_shift != 0.0;
			if (!ZERO_GUESS) {
				// entry m of every side is both produced and consumed by thread m: no staging needed
				int    ty[G::S];
				double own[G::S], gm[G::S];
				const FaceVals<D, N, PROLONG ? FV_PROLONG : FV_PLAIN> fvals{Fin, uc, meta};
				gamma_all_sides(pm, p, m, fvals, ty, own, gm);
#pragma unroll
				for (int s = 0; s < G::S; s++) {
					ntype[s] = (int8_t) ty[s];
					gam[s]   = cfac * gm[s];
				}
			}
		}
		cp_async_wait<1>(); // this group's f has landed (only the newest prefetch may still be in flight)
		__syncthreads();

		if (!ZERO_GUESS) {
			// x faces: face entry m <-> row m (2D: y; 3D: y + N z)
			if (ntype[0] != NBR_NONE) S[m * G::ROW] -= gam[0];
			if (ntype[1] != NBR_NONE) S[m * G::ROW + N - 1] -= gam[1];
			__syncthreads();
			if (D == 3) {
				// y faces: entry m = x + N z
				const int x = m % N, z = m / N;
				if (ntype[2] != NBR_NONE) S[(z * N) * G::ROW + x] -= gam[2];
				if (ntype[3] != NBR_NONE) S[(z * N + N - 1) * G::ROW + x] -= gam[3];
				__syncthreads();
			}
		}

		double v[N];
		// ---- forward along the last axis (pencil = plane index m) ----
		{
			const int base = (D == 2) ? m : (m / N) * G::ROW + (m % N);
			const int step = (D == 2) ? G::ROW : N * G::ROW;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = S[base + k * step];
			if (!ZERO_GUESS) {
				if (ntype[G::S - 2] != NBR_NONE) v[0] -= gam[G::S - 2];
				if (ntype[G::S - 1] != NBR_NONE) v[N - 1] -= gam[G::S - 1];
			}
			if (general) {
				general_transform<N>(mats, axis_kind(neu, D - 1).fwd, v, S + base, step, mg);
			} else {
				Dst2<N, N>::run(v, mg);
#pragma unroll
				for (int k = 0; k < N; k++) S[base + k * step] = v[k];
			}
		}
		__syncthreads();
		if (D == 3) { // forward along y: pencil (x, z)
			const int base = (m / N) * N * G::ROW + (m % N);
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = S[base + k * G::ROW];
			if (general) {
				general_transform<N>(mats, axis_kind(neu, 1).fwd, v, S + base, G::ROW, mg);
			} else {
				Dst2<N, N>::run(v, mg);
#pragma unroll
				for (int k = 0; k < N; k++) S[base + k * G::ROW] = v[k];
			}
			__syncthreads();
		}
		// ---- x: forward, divide by the eigenvalues, inverse (pencil = row m) ----
		{
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = S[m * G::ROW + k];
			if (general) {
				const AxisKind kx = axis_kind(neu, 0), ky = axis_kind(neu, 1), kz = axis_kind(neu, 2);
				general_transform<N>(mats, kx.fwd, v, S + m * G::ROW, 1, mg);
				// eigenvalue sum of row m = (k_y, k_z) (2D: k_y) on the fly; scale (2/N)^D as in DftPatchSolver.h:214
				const double rest  = (D == 2) ? __ldg(lam + ky.lam * N + m) : __ldg(lam + ky.lam * N + m % N) + __ldg(lam + kz.lam * N + m / N);
				double       scale = h2;
#pragma unroll
				for (int a = 0; a < D; a++) scale *= 2.0 / N;
				const bool singular = neu == (1 << (2 * D)) - 1;
#pragma unroll
				for (int k = 0; k < N; k++) {
					const double sum = __ldg(lam + kx.lam * N + k) + rest + lam_shift * h2;
					v[k]             = (singular && k == 0 && m == 0) ? 0.0 : S[m * G::ROW + k] * scale / sum;
				}
				general_transform<N>(mats, kx.inv, v, S + m * G::ROW, 1, mg);
			} else {
				// the other axes are diagonalised: row m is a tridiagonal system along x (TriSolve)
				TriSolve<N, G::M>::forward(v, tri + m, h2 * ((D == 2) ? 2.0 / N : 4.0 / (N * N)));
				TriSolve<N, G::M>::backward(v, tri + m);
#pragma unroll
				for (int k = 0; k < N; k++) S[m * G::ROW + k] = v[k];
			}
		}
		__syncthreads();
		if (D == 3) { // inverse along y
			const int base = (m / N) * N * G::ROW + (m % N);
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = S[base + k * G::ROW];
			if (general) {
				general_transform<N>(mats, axis_kind(neu, 1).inv, v, S + base, G::ROW, mg);
			} else {
				Dst3<N, N>::run(v, mg);
#pragma unroll
				for (int k = 0; k < N; k++) S[base + k * G::ROW] = v[k];
			}
			__syncthreads();
		}
		// ---- inverse along the last axis, write u (and the new faces) ----
		{
			const int base = (D == 2) ? m : (m / N) * G::ROW + (m % N);
			const int step = (D == 2) ? G::ROW : N * G::ROW;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = S[base + k * step];
			if (general) { // general path: transform through the pencil's own slots, then pick the result up again
				general_transform<N>(mats, axis_kind(neu, D - 1).inv, v, S + base, step, mg);
#pragma unroll
				for (int k = 0; k < N; k++) v[k] = S[base + k * step];
			}
			__syncthreads(); // all reads of this buffer are done: the next iteration may refill it
			if (!general) Dst3<N, N>::run(v, mg);
			if (valid) {
				double *up = u + (size_t) p * G::NC + m;
#pragma unroll
				for (int k = 0; k < N; k++) up[k * G::M] = v[k];
				if (EMIT) {
					double *Fp = Fout + (size_t) p * G::S * G::M;
					Fp[(G::S - 2) * G::M + m] = v[0];
					Fp[(G::S - 1) * G::M + m] = v[N - 1];
					if (D == 2) {
						if (m == 0) {
#pragma unroll
							for (int k = 0; k < N; k++) Fp[0 * G::M + k] = v[k];
						}
						if (m == N - 1) {
#pragma unroll
							for (int k = 0; k < N; k++) Fp[1 * G::M + k] = v[k];
						}
					} else {
						const int x = m % N, y = m / N;
						if (x == 0) {
#pragma unroll
							for (int k = 0; k < N; k++) Fp[0 * G::M + k * N + y] = v[k];
						}
						if (x == N - 1) {
#pragma unroll
							for (int k = 0; k < N; k++) Fp[1 * G::M + k * N + y] = v[k];
						}
						if (y == 0) {
#pragma unroll
							for (int k = 0; k < N; k++) Fp[2 * G::M + k * N + x] = v[k];
						}
						if (y == N - 1) {
#pragma unroll
							for (int k = 0; k < N; k++) Fp[3 * G::M + k * N + x] = v[k];
						}
					}
				}
			}
		}
	}
	cp_async_wait<0>();
}
template <int D, int N, bool ZERO_GUESS> constexpr size_t smooth_smem_bytes()
{
	using G = Geo<D, N>;
	return sizeof(double) * (size_t) (2 * G::PPB * G::SP);
}

// ---------------------------------------------------------------------------------------------
// Residual + restriction right after a block-Jacobi sweep, from face data alone.
// The sweep solves A_p u_new = f - (2/h^2) E^T gamma(u_old) exactly on every patch
// (SchurHelper.h:319-331) and the composite operator is (A u)_p = A_p u_p + (2/h^2) E^T gamma(u)
// (StarPatchOp.h:46-64 with the interface values of SURVEY App. A.2), hence
//     r = f - A u_new = (2/h^2) E^T (gamma(u_old) - gamma(u_new)):
// zero away from the patch boundary cells and a function of the boundary-cell slices only.  The
// kernel evaluates it from the face buffers (DIFF = false: u_old = 0, first sweep of a cycle) and
// applies AvgRstr (GMG/AvgRstr.h:88-107) on the fly, coarse = R r.  Neither u nor f is read and no
// fine residual is written; the only difference to GMG/Cycle.h:59-66 is the rounding noise of the patch
// solve (~1e-16 relative) that the reference's r carries in the patch interiors.
// ---------------------------------------------------------------------------------------------
// one patch (all G::M threads of its slot; every thread of the CTA must call): Rp = the slot's [S][M] staging
template <int D, int N, bool DIFF>
__device__ __forceinline__ void frr_patch(const PatchMeta *__restrict__ meta, int p, bool valid, int m, double (*Rp)[Geo<D, N>::M],
                                          const double *__restrict__ Fnew, const double *__restrict__ Fold, double *__restrict__ coarse)
{
	using G         = Geo<D, N>;
	constexpr int H = N / 2;
	int           orth = -1, parent = 0;
	if (valid) {
		const PatchMeta &pm = meta[p];
		orth                = pm.orth_on_parent;
		parent              = pm.parent_idx;
		const double cfac   = 2.0 * pm.inv_h2;
		int          ty[G::S];
		double       own[G::S], gm[G::S];
		const FaceVals<D, N, DIFF ? FV_DIFF : FV_NEG> fv{Fnew, Fold, meta};
		gamma_all_sides(pm, p, m, fv, ty, own, gm);
#pragma unroll
		for (int s = 0; s < G::S; s++) Rp[s][m] = (ty[s] == NBR_NONE) ? 0.0 : cfac * gm[s];
	}
	__syncthreads();
	if (valid) {
		double *dst = coarse + (size_t) parent * G::NC;
		if (orth < 0) { // patch present on both levels: coarse = r (dense, zero in the interior)
			const int x = m % N, y = (D == 2) ? 0 : m / N;
#pragma unroll 4
			for (int k = 0; k < N; k++) {
				double v = 0.0;
				if (D == 2) {
					if (x == 0) v += Rp[0][k];
					if (x == N - 1) v += Rp[1][k];
					if (k == 0) v += Rp[2][x];
					if (k == N - 1) v += Rp[3][x];
				} else {
					if (x == 0) v += Rp[0][y + N * k];
					if (x == N - 1) v += Rp[1][y + N * k];
					if (y == 0) v += Rp[2][x + N * k];
					if (y == N - 1) v += Rp[3][x + N * k];
					if (k == 0) v += Rp[4][m];
					if (k == N - 1) v += Rp[5][m];
				}
				dst[k * G::M + m] = v;
			}
		} else {
			const int ox = (orth & 1) * H, oy = ((orth >> 1) & 1) * H, oz = (D == 2) ? 0 : ((orth >> 2) & 1) * H;
			constexpr int CC = G::NC >> D; // coarse cells under this fine patch
			for (int c = m; c < CC; c += G::M) {
				const int X = c % H, Y = (c / H) % H, Z = (D == 2) ? 0 : c / (H * H);
				double    v = 0.0;
				if (D == 2) {
					auto blk = [&](int s, int I) { return (Rp[s][2 * I] + Rp[s][2 * I + 1]) / 4.0; };
					if (X == 0) v += blk(0, Y);
					if (X == H - 1) v += blk(1, Y);
					if (Y == 0) v += blk(2, X);
					if (Y == H - 1) v += blk(3, X);
					dst[(Y + oy) * N + (X + ox)] = v;
				} else {
					auto blk = [&](int s, int I, int J) {
						const double *q = &Rp[s][2 * I + N * 2 * J];
						return ((q[0] + q[1]) + (q[N] + q[N + 1])) / 8.0;
					};
					if (X == 0) v += blk(0, Y, Z);
					if (X == H - 1) v += blk(1, Y, Z);
					if (Y == 0) v += blk(2, X, Z);
					if (Y == H - 1) v += blk(3, X, Z);
					if (Z == 0) v += blk(4, X, Y);
					if (Z == H - 1) v += blk(5, X, Y);
					dst[((Z + oz) * N + (Y + oy)) * N + (X + ox)] = v;
				}
			}
		}
	}
	__syncthreads();
}
template <int D, int N, bool DIFF, bool HALO = false>
__global__ void __launch_bounds__(TGPU_THREADS)
face_residual_restrict_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ Fnew,
                              const double *__restrict__ Fold, double *__restrict__ coarse, HaloSync hs = HaloSync{})
{
	using G = Geo<D, N>;
	pdl_launch_dependents();
	pdl_wait();
	if (HALO) halo_push<D, N>(hs, meta);
	__shared__ double R[G::PPB][G::S][G::M];
	const int t = threadIdx.x, pp = t / G::M, m = t % G::M;
	const int nblk = (P - p0 + G::PPB - 1) / G::PPB;
	bool      halo_ok = false;
	for (int g = blockIdx.x; g < nblk; g += gridDim.x) {
		const int p = p0 + g * G::PPB + pp;
		if (HALO) halo_wait_cta(hs, p0 + g * G::PPB + G::PPB - 1, halo_ok); // the last patch of the group decides for the whole CTA
		frr_patch<D, N, DIFF>(meta, p, p < P, m, R[pp], Fnew, Fold, coarse);
	}
	if (HALO) halo_finish(hs);
}
// D = 3, N = 16: refined patches whose six sides have same-level neighbours (or none) -- every patch of a uniform
// level -- go through a leaner path: one thread per COARSE face entry (6 x 64 per patch) loads its 2 x 2 block of the
// patch's and the neighbour's slices with four 128-bit loads and stores the block average; the 512 coarse cells are
// then assembled two per thread and stored as double2.  Same expressions and summation order as frr_patch (the
// results are bit-identical); other patches take frr_patch.
constexpr int FRR16_CTAS_PER_SM = 8; // 32 registers: every CTA of the grid (8 per SM) resident at once; the kernel is latency bound
template <bool DIFF, bool HALO = false>
__global__ void __launch_bounds__(TGPU_THREADS, FRR16_CTAS_PER_SM)
face_residual_restrict16_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ Fnew,
                                const double *__restrict__ Fold, double *__restrict__ coarse, HaloSync hs = HaloSync{})
{
	using G = Geo<3, 16>;
	pdl_launch_dependents();
	pdl_wait();
	if (HALO) halo_push<3, 16>(hs, meta);
	__shared__ __align__(16) double R[G::S][G::M]; // fast path uses the first 6 x 64 entries as Rc[s][c]
	const int      t        = threadIdx.x;
	bool           halo_ok  = false;
	for (int g = blockIdx.x; g < P - p0; g += gridDim.x) {
		const int        p  = p0 + g;
		if (HALO) halo_wait_cta(hs, p, halo_ok);
		const PatchMeta &pm = meta[p];
		bool             fast = pm.orth_on_parent >= 0;
#pragma unroll
		for (int s = 0; s < 6; s++) fast = fast && pm.nbr_type[s] <= NBR_NORMAL;
		if (!fast) { // CTA-uniform
			frr_patch<3, 16, DIFF>(meta, p, true, t, R, Fnew, Fold, coarse);
			continue;
		}
		const double cfac = 2.0 * pm.inv_h2;
		double *     Rc   = &R[0][0];
		for (int e = t; e < 6 * 64; e += TGPU_THREADS) {
			const int s = e >> 6, c = e & 63, m0 = 2 * (c & 7) + 32 * (c >> 3);
			double    val = 0.0;
			if (pm.nbr_type[s] == NBR_NORMAL) {
				const size_t oa = ((size_t) p * 6 + s) * 256 + m0, ob = ((size_t) pm.nbr_idx[s][0] * 6 + (s ^ 1)) * 256 + m0;
				auto ld = [&](size_t o) {
					double2 v = __ldg(reinterpret_cast<const double2 *>(Fnew + o));
					if (DIFF) {
						const double2 w = __ldg(reinterpret_cast<const double2 *>(Fold + o));
						v.x = w.x - v.x, v.y = w.y - v.y;
					} else {
						v.x = -v.x, v.y = -v.y;
					}
					return v;
				};
				const double2 a0 = ld(oa), a1 = ld(oa + 16), b0 = ld(ob), b1 = ld(ob + 16);
				const double  r00 = cfac * (0.5 * a0.x + 0.5 * b0.x), r01 = cfac * (0.5 * a0.y + 0.5 * b0.y);
				const double  r10 = cfac * (0.5 * a1.x + 0.5 * b1.x), r11 = cfac * (0.5 * a1.y + 0.5 * b1.y);
				val               = ((r00 + r01) + (r10 + r11)) / 8.0;
			}
			Rc[e] = val;
		}
		__syncthreads();
		{
			const int orth = pm.orth_on_parent;
			const int ox = (orth & 1) * 8, oy = ((orth >> 1) & 1) * 8, oz = ((orth >> 2) & 1) * 8;
			const int X = (t & 3) * 2, Y = (t >> 2) & 7, Z = t >> 5; // cells (X, Y, Z) and (X + 1, Y, Z) of the octant
			double    v[2];
#pragma unroll
			for (int i = 0; i < 2; i++) {
				const int x = X + i;
				double    a = 0.0;
				if (x == 0) a += Rc[0 * 64 + Y + 8 * Z];
				if (x == 7) a += Rc[1 * 64 + Y + 8 * Z];
				if (Y == 0) a += Rc[2 * 64 + x + 8 * Z];
				if (Y == 7) a += Rc[3 * 64 + x + 8 * Z];
				if (Z == 0) a += Rc[4 * 64 + x + 8 * Y];
				if (Z == 7) a += Rc[5 * 64 + x + 8 * Y];
				v[i] = a;
			}
			double *dst = coarse + (size_t) pm.parent_idx * G::NC + ((Z + oz) * 16 + (Y + oy)) * 16 + (X + ox);
			*reinterpret_cast<double2 *>(dst) = make_double2(v[0], v[1]);
		}
		__syncthreads();
	}
	if (HALO) halo_finish(hs);
}

// ---------------------------------------------------------------------------------------------
// face buffer helpers
// ---------------------------------------------------------------------------------------------
template <int D, int N>
__global__ void extract_faces_kernel(int P, const double *__restrict__ u, double *__restrict__ F)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) P * G::S * G::M;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int    m = (int) (i % G::M), s = (int) ((i / G::M) % G::S);
		const size_t p = i / ((size_t) G::M * G::S);
		int          c[3];
		face_cell<D, N>(s, m, c);
		F[i] = __ldg(u + p * G::NC + (c[2] * N + c[1]) * N + c[0]);
	}
}
// F_fine += (P u_coarse) restricted to the boundary cells: all the post-smoother ever reads of the
// prolonged correction (SchurHelper.h:319-331 only uses u through its face slices).
template <int D, int N>
__global__ void prolong_faces_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ uc,
                                     double *__restrict__ F)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) P * G::S * G::M;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int    m = (int) (i % G::M), s = (int) ((i / G::M) % G::S);
		const size_t p = i / ((size_t) G::M * G::S);
		int          c[3];
		face_cell<D, N>(s, m, c);
		const PatchMeta &pm = meta[p];
		F[i] += __ldg(uc + (size_t) pm.parent_idx * G::NC + parent_cell<D, N>(pm.orth_on_parent, c));
	}
}
template <int D, int N>
__global__ void prolong_add_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ uc,
                                   double *__restrict__ uf)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) P * G::NC;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int    ci = (int) (i % G::NC);
		const size_t p  = i / G::NC;
		const int    c[3] = {ci % N, (ci / N) % N, (D == 2) ? 0 : ci / (N * N)};
		const PatchMeta &pm = meta[p];
		uf[i] += __ldg(uc + (size_t) pm.parent_idx * G::NC + parent_cell<D, N>(pm.orth_on_parent, c));
	}
}
// uf += P uc with the piecewise (bi/tri)linear interpolator (the intent of the reference's GMG/TriLinIntp.cpp:110-190, dead
// code upstream; known answer test/GMG.cpp:465-600: linear fields are reproduced exactly): tensor product of the 1-D rule
//   fine cell i -> coarse cell c = (i + offset) / 2 and its neighbour towards the fine cell: 3/4 u_c + 1/4 u_nbr
//   (3D interior weights 27/9/9/3/9/3/3/1 over 64); where that neighbour lies outside the parent patch the value is
//   extrapolated from inside, 5/4 u_c - 1/4 u_(neighbour on the other side) (face weights 45/15/15/5/-9/-3/-3/-1 over 64).
// Patches present on both levels are copied.  Evaluated axis by axis (x, y, z) like oracle/gmg_oracle.py.
template <int D, int N>
__global__ void prolong_linear_add_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ uc,
                                          double *__restrict__ uf)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) P * G::NC;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int        ci = (int) (i % G::NC);
		const size_t     p  = i / G::NC;
		const PatchMeta &pm = meta[p];
		const double *   src = uc + (size_t) pm.parent_idx * G::NC;
		const int        orth = pm.orth_on_parent;
		if (orth < 0) {
			uf[i] += __ldg(src + ci);
			continue;
		}
		const int c[3] = {ci % N, (ci / N) % N, (D == 2) ? 0 : ci / (N * N)};
		int       cc[3] = {0, 0, 0}, cq[3] = {0, 0, 0};
		double    wc[3] = {1, 1, 1}, wq[3] = {0, 0, 0};
		for (int a = 0; a < D; a++) {
			const int  off = ((orth >> a) & 1) * (N / 2), k = off + c[a] / 2, odd = c[a] & 1;
			const int  nb = odd ? k + 1 : k - 1;
			const bool in = nb >= 0 && nb < N;
			cc[a] = k;
			cq[a] = in ? nb : (odd ? k - 1 : k + 1);
			wc[a] = in ? 0.75 : 1.25;
			wq[a] = in ? 0.25 : -0.25;
		}
		auto at = [&](int x, int y, int z) { return __ldg(src + (z * N + y) * N + x); };
		auto line = [&](int y, int z) { return at(cc[0], y, z) * wc[0] + at(cq[0], y, z) * wq[0]; };
		auto plane = [&](int z) { return line(cc[1], z) * wc[1] + line(cq[1], z) * wq[1]; };
		uf[i] += (D == 2) ? plane(0) : plane(cc[2]) * wc[2] + plane(cq[2]) * wq[2];
	}
}
// thread per destination (coarse-resolution) cell of every fine patch; bit-exact w.r.t. AvgRstr.h:88-107
template <int D, int N>
__global__ void restrict_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ fine,
                                double *__restrict__ coarse)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	constexpr int H    = N / 2;
	constexpr int CC   = G::NC >> D;
	const size_t total = (size_t) P * G::NC;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int        c = (int) (i % G::NC);
		const size_t     p = i / G::NC;
		const PatchMeta &pm = meta[p];
		const int        orth = pm.orth_on_parent;
		double *         dst  = coarse + (size_t) pm.parent_idx * G::NC;
		const double *   src  = fine + p * G::NC;
		if (orth < 0) {
			dst[c] = src[c];
		} else if (c < CC) {
			const int cx = c % H, cy = (c / H) % H, cz = (D == 2) ? 0 : c / (H * H);
			double    acc = 0.0;
			for (int dz = 0; dz < (D == 2 ? 1 : 2); dz++)
				for (int dy = 0; dy < 2; dy++)
					for (int dx = 0; dx < 2; dx++)
						acc += src[((2 * cz + dz) * N + (2 * cy + dy)) * N + (2 * cx + dx)] / (1 << D);
			const int ox = (orth & 1) * H, oy = ((orth >> 1) & 1) * H, oz = (D == 2) ? 0 : ((orth >> 2) & 1) * H;
			dst[((cz + oz) * N + (cy + oy)) * N + (cx + ox)] = acc;
		}
	}
}

// weighted point-Jacobi sweep u <- u + omega D^-1 (f - A u); the residual comes from apply_tma_kernel MODE 1.  D is the
// diagonal of the ghost-eliminated composite operator: -(2 D)/h^2 per cell plus, per patch side the cell touches, the
// cell's own coefficient in the ghost value 2 gamma - u (StarPatchOp.h:46-64, interface weights SURVEY App. A.2):
// domain side -1 (Dirichlet) / +1 (Neumann), same-level neighbour 0, coarse neighbour 5/6 (3D) or 2/3 (2D), fine
// neighbours -1/3.  The "weighted-Jacobi option" of the north star (no reference counterpart; oracle: gmg_oracle.jacobi).
template <int D, int N>
__global__ void jacobi_update_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ r,
                                     double *__restrict__ u, double omega)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) P * G::NC;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int        ci = (int) (i % G::NC);
		const size_t     p  = i / G::NC;
		const PatchMeta &pm = meta[p];
		const int        c[3] = {ci % N, (ci / N) % N, (D == 2) ? 0 : ci / (N * N)};
		double           diag = -2.0 * D;
		auto side = [&](int s) {
			const int ty = pm.nbr_type[s];
			if (ty == NBR_NONE) return ((pm.neumann >> s) & 1) ? 1.0 : -1.0;
			if (ty == NBR_COARSE) return (D == 3) ? 5.0 / 6.0 : 2.0 / 3.0;
			if (ty == NBR_FINE) return -1.0 / 3.0;
			return 0.0;
		};
		for (int a = 0; a < D; a++) {
			if (c[a] == 0) diag += side(2 * a);
			if (c[a] == N - 1) diag += side(2 * a + 1);
		}
		u[i] += omega * r[i] / (diag * pm.inv_h2);
	}
}

// ---------------------------------------------------------------------------------------------
// multi-GPU halo exchange: gather the faces a peer needs into a contiguous send buffer (optionally
// with the prolonged coarse correction added, see FaceVals) / scatter received faces into halo slots
// ---------------------------------------------------------------------------------------------
template <int D, int N, bool PROLONG>
__global__ void pack_faces_kernel(const PatchMeta *__restrict__ meta, int nfaces, const int32_t *__restrict__ patch,
                                  const int32_t *__restrict__ side, const double *__restrict__ F, const double *__restrict__ uc,
                                  double *__restrict__ buf)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) nfaces * G::M;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int m = (int) (i % G::M), k = (int) (i / G::M);
		const int p = patch[k], s = side[k];
		double    v = F[((size_t) p * G::S + s) * G::M + m];
		if (PROLONG) {
			int c[3];
			face_cell<D, N>(s, m, c);
			v += __ldg(uc + (size_t) meta[p].parent_idx * G::NC + parent_cell<D, N>(meta[p].orth_on_parent, c));
		}
		buf[i] = v;
	}
}
template <int D, int N>
__global__ void unpack_faces_kernel(int nfaces, const int32_t *__restrict__ slot, const int32_t *__restrict__ side,
                                    const double *__restrict__ buf, double *__restrict__ F)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) nfaces * G::M;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int m = (int) (i % G::M), k = (int) (i / G::M);
		F[((size_t) slot[k] * G::S + side[k]) * G::M + m] = buf[i];
	}
}

// ---------------------------------------------------------------------------------------------
// Peer-to-peer halo exchange over NVLink (one process per GPU, peer buffers mapped with CUDA IPC):
// push_faces_kernel stores the faces a neighbouring rank needs straight into the halo slots of that
// rank's face buffer; p2p_signal_kernel / p2p_wait_kernel hand the data over with system-scope
// release/acquire on per-peer generation counters.  Replaces pack + ncclSend/ncclRecv + unpack
// (and with it the reference's interface VecScatters, SchurHelper.h:123-150).
// ---------------------------------------------------------------------------------------------
// hand-over state of a push (see HaloSync for the consumer side): ACK flags to wait for before the peers' halo slots may be
// overwritten, DATA flags to publish afterwards
struct PushSync {
	const uint64_t *  ack_flags      = nullptr; // my ACK flag row [nranks], written by the peers
	const int32_t *   peer_rank      = nullptr; // [npeers]
	uint64_t *const * peer_data_flag = nullptr; // [npeers] my entry of each peer's DATA row
	uint64_t *        cnt            = nullptr; // generation counters of the level (HaloSync)
	unsigned *        ticket         = nullptr;
	int *             abort          = nullptr;
	int *             host_err       = nullptr;
	int               npeers         = 0;
	int               enabled        = 0;       // 0: plain push (separate wait / signal kernels around it)
};
template <int D, int N, bool PROLONG>
__global__ void push_faces_kernel(const PatchMeta *__restrict__ meta, int nfaces, const int32_t *__restrict__ patch,
                                  const int32_t *__restrict__ side, const int32_t *__restrict__ peer_of,
                                  const int32_t *__restrict__ ridx, const double *__restrict__ F, const double *__restrict__ uc,
                                  double *const *__restrict__ peerF, PushSync ps = PushSync{})
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	if (ps.enabled) { // the peers must have consumed the previous generation of my faces (ACK) before their slots are rewritten
		if (threadIdx.x == 0 && !*ps.abort) {
			const uint64_t expected = ps.cnt[3];
			for (int k = 0; k < ps.npeers; k++) {
				const uint64_t *f = ps.ack_flags + ps.peer_rank[k];
				unsigned long long t0;
				asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
				while (ld_acquire_sys(f) < expected) {
					unsigned long long t1;
					asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
					if (t1 - t0 > 20000000000ull) { // 20 s
						atomicExch(ps.abort, 1);
						*(volatile int *) ps.host_err = ps.peer_rank[k] + 1;
						__threadfence_system();
						break;
					}
					__nanosleep(100);
				}
			}
		}
		__syncthreads();
	}
	const size_t total = (size_t) nfaces * G::M;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int m = (int) (i % G::M), k = (int) (i / G::M);
		const int p = patch[k], s = side[k];
		double    v = F[((size_t) p * G::S + s) * G::M + m];
		if (PROLONG) {
			int c[3];
			face_cell<D, N>(s, m, c);
			v += __ldg(uc + (size_t) meta[p].parent_idx * G::NC + parent_cell<D, N>(meta[p].orth_on_parent, c));
		}
		peerF[peer_of[k]][(size_t) ridx[k] * G::M + m] = v;
	}
	if (ps.enabled) { // the last block publishes the faces: DATA generation + 1 in every peer's flag row
		__syncthreads();
		if (threadIdx.x == 0) {
			__threadfence_system();
			if (atomicAdd(ps.ticket, 1u) == gridDim.x - 1) {
				__threadfence_system();
				*ps.ticket = 0;
				if (!*ps.abort) {
					ps.cnt[3] += 1;
					const uint64_t v = ps.cnt[0] + 1;
					for (int k = 0; k < ps.npeers; k++) st_release_sys(ps.peer_data_flag[k], v);
					ps.cnt[0] = v;
				}
			}
		}
	}
}
// generation = ++counter; every peer's flag (in the peer's memory) is set to it.  Runs after the kernels
// whose stores it publishes (stream order), so their peer writes have been performed.
__global__ void p2p_signal_kernel(uint64_t *const *__restrict__ remote_flags, int npeers, uint64_t *__restrict__ counter)
{
	pdl_launch_dependents();
	pdl_wait();
	const uint64_t v = *counter + 1;
	__syncthreads();
	for (int k = threadIdx.x; k < npeers; k += blockDim.x) {
		__threadfence_system();
		st_release_sys(remote_flags[k], v);
	}
	if (threadIdx.x == 0) *counter = v;
}
// waits until every peer's flag has reached generation counter + 1 - lag, then counter += 1.
// A peer that never arrives (crashed rank) trips the timeout instead of hanging the GPU: the generation counter is NOT
// advanced (the protocol stays where it broke), *abort (device) makes every later wait of the hierarchy return at
// once, and *host_err (mapped host memory, read by the host after its next synchronisation, see check_comm in tgpu.cu)
// receives the rank that was waited for + 1.
__global__ void p2p_wait_kernel(const uint64_t *__restrict__ local_flags, const int32_t *__restrict__ peer_rank, int npeers,
                                uint64_t *__restrict__ counter, int lag, int *__restrict__ abort, int *__restrict__ host_err)
{
	pdl_launch_dependents();
	pdl_wait();
	__shared__ int failed;
	if (threadIdx.x == 0) failed = *abort;
	const uint64_t expected = *counter + 1 - lag;
	__syncthreads();
	if (failed) return;
	for (int k = threadIdx.x; k < npeers; k += blockDim.x) {
		const uint64_t *f = local_flags + peer_rank[k];
		unsigned long long t0;
		asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
		while (ld_acquire_sys(f) < expected) {
			unsigned long long t1;
			asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
			if (t1 - t0 > 20000000000ull) { // 20 s
				failed = 1;
				atomicExch(abort, 1);
				*(volatile int *) host_err = peer_rank[k] + 1;
				__threadfence_system();
				break;
			}
			__nanosleep(200);
		}
	}
	__syncthreads();
	if (threadIdx.x == 0 && !failed) *counter += 1;
}

// ---------------------------------------------------------------------------------------------
// BLAS-1 (Vector.h:190-262) and reductions (Vector.h:283-321, warp-shuffle + block partials)
// ---------------------------------------------------------------------------------------------
enum Blas1Op { B_SET, B_SCALE, B_SHIFT, B_COPY, B_ADD, B_AXPY, B_AXPBY2, B_SCALE_ADD, B_SCALE_ADDS, B_SCALE_ADDS2 };
template <int OP>
__global__ void blas1_kernel(size_t n, double *__restrict__ v, const double *__restrict__ a, const double *__restrict__ b,
                             double alpha, double beta, double gamma)
{
	pdl_launch_dependents();
	pdl_wait();
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
		if (OP == B_SET) v[i] = alpha;
		else if (OP == B_SCALE) v[i] *= alpha;
		else if (OP == B_SHIFT) v[i] += alpha;
		else if (OP == B_COPY) v[i] = a[i];
		else if (OP == B_ADD) v[i] += a[i];
		else if (OP == B_AXPY) v[i] += a[i] * alpha;
		else if (OP == B_AXPBY2) v[i] += a[i] * alpha + b[i] * beta;
		else if (OP == B_SCALE_ADD) v[i] = alpha * v[i] + a[i];
		else if (OP == B_SCALE_ADDS) v[i] = alpha * v[i] + beta * a[i];
		else if (OP == B_SCALE_ADDS2) v[i] = alpha * v[i] + beta * a[i] + gamma * b[i];
	}
}
__device__ __forceinline__ double warp_sum(double x)
{
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
	return x;
}
__device__ __forceinline__ double warp_max(double x)
{
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
	return x;
}
// OP 0: sum a*b, 1: max |a|.  Stage 1 writes one partial per block; stage 2 (one block) finishes.
template <int OP>
__global__ void reduce_stage1(size_t n, const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ partial)
{
	pdl_launch_dependents();
	pdl_wait();
	double acc = 0.0;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
		if (OP == 0) acc = fma(a[i], b[i], acc);
		else acc = fmax(acc, fabs(a[i]));
	}
	__shared__ double ws[32];
	acc = OP == 0 ? warp_sum(acc) : warp_max(acc);
	if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
	__syncthreads();
	if (threadIdx.x < 32) {
		double x = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0.0;
		x        = OP == 0 ? warp_sum(x) : warp_max(x);
		if (threadIdx.x == 0) partial[blockIdx.x] = x;
	}
}
template <int OP> __global__ void reduce_stage2(int nb, const double *__restrict__ partial, double *__restrict__ result)
{
	pdl_launch_dependents();
	pdl_wait();
	double acc = 0.0;
	for (int i = threadIdx.x; i < nb; i += blockDim.x) {
		if (OP == 0) acc += partial[i];
		else acc = fmax(acc, partial[i]);
	}
	__shared__ double ws[32];
	acc = OP == 0 ? warp_sum(acc) : warp_max(acc);
	if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
	__syncthreads();
	if (threadIdx.x < 32) {
		double x = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0.0;
		x        = OP == 0 ? warp_sum(x) : warp_max(x);
		if (threadIdx.x == 0) *result = x;
	}
}

// ---------------------------------------------------------------------------------------------
// ||f - A u_new||^2 right after a sweep, from face data: by the identity of face_residual_restrict_kernel the residual
// is (2/h^2) E^T (gamma(u_old) - gamma(u_new)), zero away from the patch boundary cells, so only the S x M entries of
// the sides are evaluated.  A cell on several sides (edges, corners) takes the sum of their terms in side order (as
// frr_patch) and is counted once, by the first side it lies on.  MODE: FV_DIFF (u_old's slices in Fold) or
// FV_PROLONG_DIFF (u_old = Fold + P uc on the boundary cells: the input of a first post-sweep).  One patch per CTA
// iteration, [S][M] terms staged in shared memory; one partial sum per CTA in partial[blockIdx.x].
// ---------------------------------------------------------------------------------------------
template <int D, int N> constexpr int frn_threads()
{
	return 2 * D * Geo<D, N>::M >= TGPU_THREADS ? TGPU_THREADS : (2 * D * Geo<D, N>::M + 31) / 32 * 32;
}
template <int D, int N> constexpr size_t frn_smem_bytes() { return (size_t) 2 * D * Geo<D, N>::M * sizeof(double); }
// index of cell c in the slice of side s (face_cell inverted)
template <int D, int N> __device__ __forceinline__ int face_index(int s, const int (&c)[3])
{
	const int ax = s >> 1;
	if (D == 2) return c[1 - ax];
	if (ax == 0) return c[1] + N * c[2];
	if (ax == 1) return c[0] + N * c[2];
	return c[0] + N * c[1];
}
template <int D, int N, int MODE>
__global__ void __launch_bounds__(TGPU_THREADS)
face_residual_norm_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ Fnew, const double *__restrict__ Fold,
                          const double *__restrict__ uc, double *__restrict__ partial)
{
	using G = Geo<D, N>;
	pdl_launch_dependents();
	pdl_wait();
	extern __shared__ double Rs[]; // [S][M]
	const FaceVals<D, N, MODE> fv{Fnew, MODE == FV_DIFF ? Fold : uc, meta, Fold};
	double acc = 0.0;
	for (int p = blockIdx.x; p < P; p += gridDim.x) {
		const PatchMeta &pm   = meta[p];
		const double     cfac = 2.0 * pm.inv_h2;
		for (int m = threadIdx.x; m < G::M; m += blockDim.x) {
			int    ty[G::S];
			double own[G::S], gm[G::S];
			gamma_all_sides(pm, p, m, fv, ty, own, gm);
#pragma unroll
			for (int s = 0; s < G::S; s++) Rs[s * G::M + m] = (ty[s] == NBR_NONE) ? 0.0 : cfac * gm[s];
		}
		__syncthreads();
		for (int e = threadIdx.x; e < G::S * G::M; e += blockDim.x) {
			const int s = e / G::M;
			int       c[3];
			face_cell<D, N>(s, e % G::M, c);
			double v     = 0.0;
			int    first = -1;
#pragma unroll
			for (int s2 = 0; s2 < G::S; s2++) {
				if (c[s2 >> 1] != ((s2 & 1) ? N - 1 : 0)) continue;
				if (first < 0) first = s2;
				v += Rs[s2 * G::M + face_index<D, N>(s2, c)];
			}
			if (first == s) acc = fma(v, v, acc);
		}
		__syncthreads();
	}
	__shared__ double ws[32];
	acc = warp_sum(acc);
	if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = acc;
	__syncthreads();
	if (threadIdx.x < 32) {
		double x = threadIdx.x < (blockDim.x >> 5) ? ws[threadIdx.x] : 0.0;
		x        = warp_sum(x);
		if (threadIdx.x == 0) partial[blockIdx.x] = x;
	}
}

// ---------------------------------------------------------------------------------------------
// BiCGStab (BiCGStab.h:45-106) with device-resident scalars: the vector updates of one iteration are fused
// into three passes and the dot products ride along; the host reads one number (the residual norm) per
// iteration.  Element-wise expressions are those of the Vector<D> ops the reference calls (Vector.h:218-262),
// so the iterates match the op-by-op version up to the order of the reductions.
//   sc[]: 0 rho, 1 alpha, 2 omega, 3 beta, 4 |r|, 5/6 reduction results
// ---------------------------------------------------------------------------------------------
enum { SC_RHO = 0, SC_ALPHA = 1, SC_OMEGA = 2, SC_BETA = 3, SC_RNORM = 4, SC_SUM0 = 5, SC_SUM1 = 6 };
__device__ __forceinline__ void block_partials2(double a0, double a1, double *__restrict__ partial, int stride)
{
	__shared__ double ws[2][32];
	a0 = warp_sum(a0);
	a1 = warp_sum(a1);
	if ((threadIdx.x & 31) == 0) {
		ws[0][threadIdx.x >> 5] = a0;
		ws[1][threadIdx.x >> 5] = a1;
	}
	__syncthreads();
	if (threadIdx.x < 32) {
		double x0 = threadIdx.x < (blockDim.x >> 5) ? ws[0][threadIdx.x] : 0.0;
		double x1 = threadIdx.x < (blockDim.x >> 5) ? ws[1][threadIdx.x] : 0.0;
		x0        = warp_sum(x0);
		x1        = warp_sum(x1);
		if (threadIdx.x == 0) {
			partial[blockIdx.x]          = x0;
			partial[stride + blockIdx.x] = x1;
		}
	}
}
// partial[0][b] = sum a b, partial[1][b] = sum a a
__global__ void bicg_dots_kernel(size_t n, const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ partial, int stride)
{
	pdl_launch_dependents();
	pdl_wait();
	double d0 = 0.0, d1 = 0.0;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
		const double x = a[i];
		d0             = fma(x, b[i], d0);
		d1             = fma(x, x, d1);
	}
	block_partials2(d0, d1, partial, stride);
}
// s = r + ap (-alpha)      (s->copy(resid); s->addScaled(-alpha, ap))
__global__ void bicg_s_kernel(size_t n, const double *__restrict__ r, const double *__restrict__ ap, double *__restrict__ s,
                              const double *__restrict__ sc)
{
	pdl_launch_dependents();
	pdl_wait();
	const double na = -sc[SC_ALPHA];
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
		double v = r[i];
		v += ap[i] * na;
		s[i] = v;
	}
}
// x += alpha mp + omega ms;  r += -alpha ap - omega as;  partial sums of r.rhat and r.r
__global__ void bicg_xr_kernel(size_t n, double *__restrict__ x, const double *__restrict__ mp, const double *__restrict__ ms,
                               double *__restrict__ r, const double *__restrict__ ap, const double *__restrict__ as,
                               const double *__restrict__ rhat, const double *__restrict__ sc, double *__restrict__ partial, int stride)
{
	pdl_launch_dependents();
	pdl_wait();
	const double alpha = sc[SC_ALPHA], omega = sc[SC_OMEGA], na = -alpha, no = -omega;
	double       d0 = 0.0, d1 = 0.0;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
		double xv = x[i];
		xv += mp[i] * alpha + ms[i] * omega;
		x[i]      = xv;
		double rv = r[i];
		rv += ap[i] * na + as[i] * no;
		r[i] = rv;
		d0   = fma(rv, rhat[i], d0);
		d1   = fma(rv, rv, d1);
	}
	block_partials2(d0, d1, partial, stride);
}
// p += -omega ap;  p = beta p + r
__global__ void bicg_p_kernel(size_t n, double *__restrict__ p, const double *__restrict__ ap, const double *__restrict__ r,
                              const double *__restrict__ sc)
{
	pdl_launch_dependents();
	pdl_wait();
	const double no = -sc[SC_OMEGA], beta = sc[SC_BETA];
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
		double v = p[i];
		v += ap[i] * no;
		p[i] = beta * v + r[i];
	}
}
// finishes the two reductions (-> sc[SC_SUM0/1]) and, unless an all-reduce over the ranks has to come first,
// updates the scalars of the given step (bicg_scalars)
__device__ __forceinline__ void bicg_scalars(int step, double *sc)
{
	const double s0 = sc[SC_SUM0], s1 = sc[SC_SUM1];
	if (step == 1) sc[SC_ALPHA] = sc[SC_RHO] / s0;                // alpha = rho / (rhat . ap)
	else if (step == 2) sc[SC_OMEGA] = s0 / s1;                    // omega = (as . s) / (as . as)
	else if (step == 3) {                                           // rho_new = r . rhat, beta, |r|
		sc[SC_BETA]  = s0 * sc[SC_ALPHA] / (sc[SC_RHO] * sc[SC_OMEGA]);
		sc[SC_RHO]   = s0;
		sc[SC_RNORM] = sqrt(s1);
	} else if (step == 0) {                                         // set-up: rho = rhat . r, |r|
		sc[SC_RHO]   = s0;
		sc[SC_RNORM] = sqrt(s1);
	}
}
__global__ void bicg_finish_kernel(int nb, int stride, const double *__restrict__ partial, double *__restrict__ sc, int step, int update)
{
	pdl_launch_dependents();
	pdl_wait();
	double a0 = 0.0, a1 = 0.0;
	for (int i = threadIdx.x; i < nb; i += blockDim.x) {
		a0 += partial[i];
		a1 += partial[stride + i];
	}
	__shared__ double ws[2][32];
	a0 = warp_sum(a0);
	a1 = warp_sum(a1);
	if ((threadIdx.x & 31) == 0) {
		ws[0][threadIdx.x >> 5] = a0;
		ws[1][threadIdx.x >> 5] = a1;
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		double x0 = 0.0, x1 = 0.0;
		for (int w = 0; w < (int) (blockDim.x >> 5); w++) x0 += ws[0][w], x1 += ws[1][w];
		sc[SC_SUM0] = x0;
		sc[SC_SUM1] = x1;
		if (update) bicg_scalars(step, sc);
	}
}
__global__ void bicg_scalars_kernel(double *__restrict__ sc, int step)
{
	pdl_launch_dependents();
	pdl_wait();
	if (threadIdx.x == 0) bicg_scalars(step, sc);
}

// manufactured trig problem (apps/3d/steady.cpp:253-265, apps/2d/steady.cpp:314-316) with the
// Dirichlet data folded into f on domain-boundary cells (apps/shared/Init.cpp:183-241,329-357)
template <int D> __device__ __forceinline__ double trig_exact(double x, double y, double z)
{
	if (D == 2) return sin(M_PI * y) * cos(2 * M_PI * x);
	x += .3, y += .3, z += .3;
	return sin(M_PI * x) * cos(2.0 / 3 * M_PI * y) * sin(5.0 / 6 * M_PI * z);
}
template <int D> __device__ __forceinline__ double trig_rhs(double x, double y, double z)
{
	if (D == 2) return -5 * M_PI * M_PI * sin(M_PI * y) * cos(2 * M_PI * x);
	x += .3, y += .3, z += .3;
	return -77.0 / 36 * M_PI * M_PI * sin(M_PI * x) * cos(2.0 / 3 * M_PI * y) * sin(5.0 / 6 * M_PI * z);
}
template <int D, int N>
__global__ void init_trig_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ starts,
                                 const double *__restrict__ spacing, double *__restrict__ f, double *__restrict__ exact)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const size_t total = (size_t) P * G::NC;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int        ci = (int) (i % G::NC);
		const size_t     p  = i / G::NC;
		const PatchMeta &pm = meta[p];
		const int        c[3] = {ci % N, (ci / N) % N, (D == 2) ? 0 : ci / (N * N)};
		double           h[3] = {0, 0, 0}, st[3] = {0, 0, 0}, x[3] = {0, 0, 0};
		for (int a = 0; a < D; a++) {
			h[a]  = spacing[p * D + a];
			st[a] = starts[p * D + a];
			x[a]  = st[a] + h[a] / 2.0 + h[a] * c[a];
		}
		double val = trig_rhs<D>(x[0], x[1], x[2]);
		for (int a = 0; a < D; a++) {
			double xb[3] = {x[0], x[1], x[2]};
			if (c[a] == 0 && pm.nbr_type[2 * a] == NBR_NONE) {
				xb[a] = st[a];
				val -= 2 * trig_exact<D>(xb[0], xb[1], xb[2]) / (h[a] * h[a]);
			}
			if (c[a] == N - 1 && pm.nbr_type[2 * a + 1] == NBR_NONE) {
				xb[a] = st[a] + h[a] * N;
				val -= 2 * trig_exact<D>(xb[0], xb[1], xb[2]) / (h[a] * h[a]);
			}
		}
		f[i] = val;
		if (exact) exact[i] = trig_exact<D>(x[0], x[1], x[2]);
	}
}
// Neumann form of the right-hand side (Init::initNeumann, apps/shared/Init.cpp:57-151) for the 3D manufactured problems
// of apps/3d/steady.cpp:230-282: problem 0 = trig (the one above), 1 = "gauss".  On a domain side without a neighbour the
// boundary cell gets +dg/dx_a (lower side) / -dg/dx_a (upper side), evaluated on the face, divided by h_a.
struct Problem3 {
	int kind;
	__device__ __forceinline__ double g(double x, double y, double z) const
	{
		if (kind == 1) return exp(cos(10 * M_PI * x)) - exp(cos(11 * M_PI * y)) + exp(cos(12 * M_PI * z));
		return trig_exact<3>(x, y, z);
	}
	__device__ __forceinline__ double f(double x, double y, double z) const
	{
		if (kind == 1)
			return -M_PI * M_PI
			       * (100 * exp(cos(10 * M_PI * x)) * cos(10 * M_PI * x) - 100 * exp(cos(10 * M_PI * x)) * pow(sin(10 * M_PI * x), 2)
			          - 121 * exp(cos(11 * M_PI * y)) * cos(11 * M_PI * y) + 121 * exp(cos(11 * M_PI * y)) * pow(sin(11 * M_PI * y), 2)
			          + 144 * exp(cos(12 * M_PI * z)) * cos(12 * M_PI * z) - 144 * exp(cos(12 * M_PI * z)) * pow(sin(12 * M_PI * z), 2));
		return trig_rhs<3>(x, y, z);
	}
	__device__ __forceinline__ double dg(int axis, double x, double y, double z) const
	{
		if (kind == 1) {
			if (axis == 0) return -10 * M_PI * sin(10 * M_PI * x) * exp(cos(10 * M_PI * x));
			if (axis == 1) return 11 * M_PI * sin(11 * M_PI * y) * exp(cos(11 * M_PI * y));
			return -12 * M_PI * sin(12 * M_PI * z) * exp(cos(12 * M_PI * z));
		}
		x += .3, y += .3, z += .3;
		if (axis == 0) return M_PI * cos(M_PI * x) * cos(2.0 / 3 * M_PI * y) * sin(5.0 / 6 * M_PI * z);
		if (axis == 1) return -2.0 / 3 * M_PI * sin(M_PI * x) * sin(2.0 / 3 * M_PI * y) * sin(5.0 / 6 * M_PI * z);
		return 5.0 / 6 * M_PI * sin(M_PI * x) * cos(2.0 / 3 * M_PI * y) * cos(5.0 / 6 * M_PI * z);
	}
};
// 2D: the trig problem of apps/2d/steady.cpp:314-318 (Init::initNeumann2d, apps/shared/Init.cpp:246-303)
__device__ __forceinline__ double trig2_dg(int axis, double x, double y)
{
	return axis == 0 ? -2 * M_PI * sin(M_PI * y) * sin(2 * M_PI * x) : M_PI * cos(M_PI * y) * cos(2 * M_PI * x);
}
template <int D, int N>
__global__ void init_neumann_kernel(const PatchMeta *__restrict__ meta, int P, const double *__restrict__ starts,
                                    const double *__restrict__ spacing, double *__restrict__ f, double *__restrict__ exact, int problem)
{
	pdl_launch_dependents();
	pdl_wait();
	using G            = Geo<D, N>;
	const Problem3 pr{problem};
	const size_t   total = (size_t) P * G::NC;
	for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
		const int        ci = (int) (i % G::NC);
		const size_t     p  = i / G::NC;
		const PatchMeta &pm = meta[p];
		const int        c[3] = {ci % N, (ci / N) % N, (D == 2) ? 0 : ci / (N * N)};
		double           h[3] = {0, 0, 0}, st[3] = {0, 0, 0}, x[3] = {0, 0, 0};
		for (int a = 0; a < D; a++) {
			h[a]  = spacing[p * D + a];
			st[a] = starts[p * D + a];
			x[a]  = st[a] + h[a] / 2.0 + h[a] * c[a];
		}
		double val = (D == 2) ? trig_rhs<2>(x[0], x[1], 0.0) : pr.f(x[0], x[1], x[2]);
		for (int a = 0; a < D; a++) { // west, east, south, north, bottom, top (the order of Init.cpp:90-148, 270-299)
			double xb[3] = {x[0], x[1], x[2]};
			if (c[a] == 0 && pm.nbr_type[2 * a] == NBR_NONE) {
				xb[a] = st[a];
				val += ((D == 2) ? trig2_dg(a, xb[0], xb[1]) : pr.dg(a, xb[0], xb[1], xb[2])) / h[a];
			}
			if (c[a] == N - 1 && pm.nbr_type[2 * a + 1] == NBR_NONE) {
				xb[a] = st[a] + h[a] * N;
				val -= ((D == 2) ? trig2_dg(a, xb[0], xb[1]) : pr.dg(a, xb[0], xb[1], xb[2])) / h[a];
			}
		}
		f[i] = val;
		if (exact) exact[i] = (D == 2) ? trig_exact<2>(x[0], x[1], 0.0) : pr.g(x[0], x[1], x[2]);
	}
}
// per-patch sums times the cell volume (Domain::integrate, Domain.h:258-278): out[p] = prod_a h_a * sum of the patch
template <int D, int N>
__global__ void patch_integrals_kernel(int P, const double *__restrict__ spacing, const double *__restrict__ v, double *__restrict__ out)
{
	pdl_launch_dependents();
	pdl_wait();
	using G = Geo<D, N>;
	__shared__ double part[8];
	for (int p = blockIdx.x; p < P; p += gridDim.x) {
		double acc = 0.0;
		for (int i = threadIdx.x; i < G::NC; i += blockDim.x) acc += v[(size_t) p * G::NC + i];
		for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
		if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
		__syncthreads();
		if (threadIdx.x == 0) {
			double s = 0.0;
			for (int w = 0; w < (int) (blockDim.x >> 5); w++) s += part[w];
			for (int a = 0; a < D; a++) s *= spacing[(size_t) p * D + a];
			out[p] = s;
		}
		__syncthreads();
	}
}
} // namespace tgpu
#include "smooth3d16.cuh"
#include "patch3d32.cuh"
#include "apply_tma.cuh"
#include "smooth2d32.cuh"
