// smooth2d32.cuh - block-Jacobi smoother specialised for D = 2, N = 32 (BASELINE configs A and E: 32 x 32 patches).
// Included by kernels.cuh.
//
// Same arithmetic as the generic smooth_kernel (SchurHelper::solveWithSolution, SchurHelper.h:319-331; interface
// values of BilinearInterpolator.cpp:61-117; patch solve of FftwPatchSolver.h:174-206 in the form of kernels.cuh,
// TriSolve: DST-II / DST-III along y, tridiagonal elimination along x).  A patch has 32 pencils, i.e. it is exactly
// one warp's work, so here ONE WARP OWNS ONE PATCH from load to store and no CTA barrier exists:
//   * lane x loads column x of f straight from memory (a warp's load = one 256-byte row), transforms it along y,
//     stores it into the warp's private 32 x 34 tile; lane k_y then reads row k_y (128-bit), eliminates along x,
//     writes it back; lane x reads column x, transforms back and stores u (and the boundary slices) to memory;
//   * the eight warps of a CTA drift apart freely, so the fp64, shared-memory and load phases of different
//     patches overlap on the SM; with 4 shared-memory accesses and 20 fp64 operations per cell (16^3 kernel: 8 and
//     33) the kernel ends up bound by HBM;
//   * the interface values of the warp's next patch are gathered in two batches of two sides, issued before a
//     transform and combined after it; x-face values (needed by lanes 0 and 31 for every y) pass through a
//     64-double staging row, y-face values stay in two registers.
#pragma once

namespace tgpu
{
constexpr int    Q32_ROW = 34, Q32_TILE = 32 * Q32_ROW, Q32_WARP = Q32_TILE + 64 + 64, Q32_WARPS = TGPU_THREADS / 32;
constexpr size_t smooth2d32_smem_bytes() { return sizeof(double) * Q32_WARPS * Q32_WARP; }

template <bool PROLONG>
__device__ __noinline__ double gamma_entry2d32(const PatchMeta *__restrict__ meta, int p, int s, int m, const double *__restrict__ F,
                                               const double *__restrict__ uc)
{
	const FaceVals<2, 32, PROLONG ? FV_PROLONG : FV_PLAIN> fv{F, uc, meta};
	return gamma_entry(meta[p], p, s, m, fv);
}
// one interface value split into "issue the loads" and "combine" (same-level neighbours inline, same expressions
// as gamma_entry; anything else through the general code at combine time)
template <bool PROLONG> struct Gam2d32 {
	double a0, b0, a1, b1;
	int    slow;
	__device__ __forceinline__ void issue(const PatchMeta &pm, int p, int s, int m, const double *__restrict__ F, const double *__restrict__ uc)
	{
		constexpr int N = 32, NC = N * N;
		const int     ty = pm.nbr_type[s];
		slow             = ty > NBR_NORMAL;
		a0 = b0 = a1 = b1 = 0.0;
		if (ty == NBR_NORMAL) {
			a0 = __ldg(F + ((size_t) p * 4 + s) * N + m);
			b0 = __ldg(F + ((size_t) pm.nbr_idx[s][0] * 4 + (s ^ 1)) * N + m);
			if (PROLONG) {
				int c[3];
				if (pm.parent_idx >= 0) {
					face_cell<2, N>(s, m, c);
					a1 = __ldg(uc + (size_t) pm.parent_idx * NC + parent_cell<2, N>(pm.orth_on_parent, c));
				}
				const int qp = pm.nbr_parent[s];
				if (qp >= 0) { // < 0: halo slot whose face arrived with the correction added
					face_cell<2, N>(s ^ 1, m, c);
					b1 = __ldg(uc + (size_t) qp * NC + parent_cell<2, N>(pm.nbr_orth[s], c));
				}
			}
		}
	}
	__device__ __forceinline__ double finish(const PatchMeta *__restrict__ meta, int p, int s, int m, const double *__restrict__ F,
	                                         const double *__restrict__ uc, double cfac) const
	{
		if (slow) return cfac * gamma_entry2d32<PROLONG>(meta, p, s, m, F, uc);
		return cfac * (0.5 * (a0 + a1) + 0.5 * (b0 + b1));
	}
};

// EXTRA = false compiles the halo hand-over and the Neumann skip out (single GPU, all-Dirichlet levels: the calls and the
// extra live values cost ~5 % of the sweep through spills otherwise)
template <bool ZERO_GUESS, bool EMIT, bool PROLONG, bool WRITE_U, bool EXTRA = false>
__global__ void __launch_bounds__(TGPU_THREADS, 2)
smooth2d32_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ f, double *__restrict__ u,
                  const double *__restrict__ Fin, double *__restrict__ Fout, const double *__restrict__ tri,
                  const double *__restrict__ uc, HaloSync hs = HaloSync{}, int skip_neumann = 0)
{
	// skip_neumann != 0: patches with Neumann domain sides are left to the general path of smooth_kernel (launched over
	// the same range with only_neumann); the warp still gathers its next patch's interface values
	constexpr int N = 32, ROW = Q32_ROW, NC = N * N;
	static_assert(WRITE_U || EMIT, "a sweep must produce something");
	extern __shared__ __align__(16) double smem[];
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	double *  S  = smem + w * Q32_WARP; // the warp's tile [y or k_y][x], row stride 34
	double *  GX = S + Q32_TILE;        // (2/h^2) gamma on the x faces of the patch about to be solved, [2][32]
	double *  EX = GX + 64;             // staging of the new x-face slices, [2][32]
	Mags<N>   mg;
	mg.load();
	pdl_launch_dependents();
	pdl_wait();
	if (EXTRA && !ZERO_GUESS) halo_push<2, 32>(hs, meta);
	const int npatch = P - p0, nw = gridDim.x * Q32_WARPS;
	int       g = blockIdx.x * Q32_WARPS + w;
	double    gy0 = 0.0, gy1 = 0.0; // (2/h^2) gamma of entry x = lane on the two y faces
	bool      halo_ok = false;      // multi-GPU: the warp polls the peers' flags before its first patch that needs halo faces
	if (!ZERO_GUESS && g < npatch) { // the warp's first patch: nothing to hide the gathers behind
		const int    p    = p0 + g;
		if (EXTRA) halo_wait_warp(hs, p, halo_ok);
		const double cfac = 2.0 * meta[p].inv_h2;
		GX[lane]      = cfac * gamma_entry2d32<PROLONG>(meta, p, 0, lane, Fin, uc);
		GX[32 + lane] = cfac * gamma_entry2d32<PROLONG>(meta, p, 1, lane, Fin, uc);
		gy0           = cfac * gamma_entry2d32<PROLONG>(meta, p, 2, lane, Fin, uc);
		gy1           = cfac * gamma_entry2d32<PROLONG>(meta, p, 3, lane, Fin, uc);
		__syncwarp();
	}
	for (; g < npatch; g += nw) {
		const int    p    = p0 + g;
		const bool   next = g + nw < npatch;
		const int    pn   = p + nw;
		const double h2   = meta[p].h2;
		const double *tb  = tri + (size_t) meta[p].tab * (17 * 32) + lane; // the patch's table [17][32] (TriSolve)
		double       v[N];
		if (EXTRA && !ZERO_GUESS && next) halo_wait_warp(hs, pn, halo_ok); // gamma of patch pn is gathered during this iteration
		if (EXTRA && skip_neumann && meta[p].neumann) { // warp-uniform
			if (!ZERO_GUESS && next) {
				const double cf = 2.0 * meta[pn].inv_h2;
				__syncwarp(); // GX of the skipped patch is not needed
				GX[lane]      = cf * gamma_entry2d32<PROLONG>(meta, pn, 0, lane, Fin, uc);
				GX[32 + lane] = cf * gamma_entry2d32<PROLONG>(meta, pn, 1, lane, Fin, uc);
				gy0           = cf * gamma_entry2d32<PROLONG>(meta, pn, 2, lane, Fin, uc);
				gy1           = cf * gamma_entry2d32<PROLONG>(meta, pn, 3, lane, Fin, uc);
				__syncwarp();
			}
			continue;
		}
		Gam2d32<PROLONG> ga, gb;
		double           cfn = 0.0;
		{ // y forward: column x = lane, straight from memory
			const double *fp = f + (size_t) p * NC + lane;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = __ldcs(fp + k * N);
			if (next) { // the warp's next patch -> L2 (64 lines)
				const double *fn = f + (size_t) pn * NC + lane * 32;
				prefetch_l2(fn);
				prefetch_l2(fn + 16);
			}
			if (!ZERO_GUESS) {
				v[0] -= gy0;
				v[N - 1] -= gy1;
				if (lane == 0 || lane == N - 1) { // x faces: entry y belongs to the columns x = 0 / 31
					const double *q = GX + (lane ? 32 : 0);
#pragma unroll
					for (int k = 0; k < N; k++) v[k] -= q[k];
				}
				__syncwarp(); // GX is consumed
				if (next) {
					const PatchMeta &pq = meta[pn];
					cfn                 = 2.0 * pq.inv_h2;
					ga.issue(pq, pn, 0, lane, Fin, uc);
					gb.issue(pq, pn, 1, lane, Fin, uc);
				}
			}
			Dst2<N, N>::run(v, mg);
			double *col = S + lane;
#pragma unroll
			for (int k = 0; k < N; k++) col[k * ROW] = v[k];
			if (!ZERO_GUESS && next) {
				GX[lane]      = ga.finish(meta, pn, 0, lane, Fin, uc, cfn);
				GX[32 + lane] = gb.finish(meta, pn, 1, lane, Fin, uc, cfn);
			}
		}
		__syncwarp();
		{ // x: row k_y = lane is a tridiagonal system (TriSolve, kernels.cuh); tri = multiplier table [17][32]
			double2 *rowp = reinterpret_cast<double2 *>(S + lane * ROW);
#pragma unroll
			for (int j = 0; j < N / 2; j++) {
				const double2 d = rowp[j];
				v[2 * j]        = d.x;
				v[2 * j + 1]    = d.y;
			}
			TriSolve<N, N>::forward(v, tb, h2 * (2.0 / N));
			TriSolve<N, N>::backward(v, tb);
#pragma unroll
			for (int j = 0; j < N / 2; j++) rowp[j] = make_double2(v[2 * j], v[2 * j + 1]);
		}
		__syncwarp();
		{ // y inverse: column x = lane, straight to memory
			const double *col = S + lane;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = col[k * ROW];
			if (!ZERO_GUESS && next) {
				const PatchMeta &pq = meta[pn];
				ga.issue(pq, pn, 2, lane, Fin, uc);
				gb.issue(pq, pn, 3, lane, Fin, uc);
			}
			Dst3<N, N>::run(v, mg);
			if (!ZERO_GUESS && next) {
				gy0 = ga.finish(meta, pn, 2, lane, Fin, uc, cfn);
				gy1 = gb.finish(meta, pn, 3, lane, Fin, uc, cfn);
			}
			if (WRITE_U) {
				double *up = u + (size_t) p * NC + lane;
#pragma unroll
				for (int k = 0; k < N; k++) __stcs(up + k * N, v[k]);
			}
			if (EMIT) {
				double *Fp = Fout + (size_t) p * 4 * N;
				Fp[2 * N + lane] = v[0]; // y faces: entry x
				Fp[3 * N + lane] = v[N - 1];
				if (lane == 0 || lane == N - 1) { // x faces: entries y, held by lanes 0 and 31
					double *q = EX + (lane ? 32 : 0);
#pragma unroll
					for (int k = 0; k < N; k++) q[k] = v[k];
				}
				__syncwarp();
				Fp[0 * N + lane] = EX[lane];
				Fp[1 * N + lane] = EX[32 + lane];
			}
		}
		__syncwarp();
	}
	if (EXTRA && !ZERO_GUESS) halo_finish(hs);
}
} // namespace tgpu
