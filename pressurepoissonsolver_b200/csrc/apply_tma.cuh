// apply_tma.cuh - operator apply / residual / residual+restriction with the patch staged in shared memory by the TMA
// engine (BASELINE north star (1): "patch plus ghost layer staged in shared memory via TMA").  Included by kernels.cuh.
//
// SchurHelper::apply (SchurHelper.h:361-376) + StarPatchOp::applyWithInterface (StarPatchOp.h:28-184): ghost = 2 gamma - a
// on sides with a neighbour, -a on Dirichlet and +a on Neumann domain sides (StarPatchOp.h:46-64).  How the tile moves:
//   * a patch is contiguous in memory (PetscVector.h:75-90), so ONE bulk copy per group of patches
//     (cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes, SASS UBLKCP: up to 64 KB per instruction, issued by
//     one thread) replaces the 4096 8-byte LDGSTS per 16^3 patch that a ghosted tile (rows not 16-byte aligned) would
//     take.  Two tiles alternate; completion is tracked by one mbarrier per tile (expect_tx = bytes).
//   * the tile therefore carries NO ghost layer: the 2D ghost faces (computed from the face buffers, they are not a copy
//     of anything in memory) live in a separate small array G[side][entry], and every thread picks "tile or ghost array"
//     for its four in-plane neighbours ONCE (pointer + stride) before it marches along the last axis - the inner loop is
//     the same seven loads as with a ghosted tile.
#pragma once

namespace tgpu
{
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned) __cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned) __cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
	const unsigned a = (unsigned) __cvta_generic_to_shared(bar);
	asm volatile(
	"{\n"
	".reg .pred p;\n"
	"WAIT_%=:\n"
	"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
	"@p bra DONE_%=;\n"
	"bra WAIT_%=;\n"
	"DONE_%=:\n"
	"}\n" ::"r"(a),
	"r"(parity)
	: "memory");
}
// generic-proxy accesses to a tile (the stencil's reads) are ordered before the async-proxy write that refills it
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
// 1-D bulk copy global -> shared through the TMA engine; dst, src and bytes are multiples of 16
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gsrc, unsigned bytes, uint64_t *bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"((unsigned) __cvta_generic_to_shared(smem_dst)),
	             "l"(gsrc), "r"(bytes), "r"((unsigned) __cvta_generic_to_shared(bar))
	             : "memory");
}

// MODE 0: out = A u, 1: out = f - A u, 2: coarse = AvgRstr(f - A u) (GMG/AvgRstr.h:88-107; the fine residual is never written),
// 3: out = A u and, riding along, the block partial sums of out . f and out . out (f = the vector the Krylov iteration dots A u
//    with next, BiCGStab.h:77,89: one pass over memory less per operator application; partial[b], partial[pstride + b])
template <int D, int N, int MODE>
__global__ void __launch_bounds__(TGPU_THREADS, 2)
apply_tma_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ u, const double *__restrict__ f,
                 const double *__restrict__ F, double *__restrict__ out, double *__restrict__ coarse, double *__restrict__ partial = nullptr,
                 int pstride = 0)
{
	using G = Geo<D, N>;
	pdl_launch_dependents();
	pdl_wait();
	extern __shared__ __align__(16) double smem[];
	double *                 Ut = smem;                        // [2][PPB][NC] two tiles of PPB whole patches each
	double *                 Gh = smem + 2 * G::PPB * G::NC;   // [PPB][S][M] ghost faces of the current group
	__shared__ uint64_t      bar[2];
	const int                t = threadIdx.x, pp = t / G::M, m = t % G::M;
	const int                nblk = (P - p0 + G::PPB - 1) / G::PPB;
	const int                x = m % N, y = (D == 2) ? 0 : m / N;
	if (t == 0) {
		mbar_init(&bar[0], 1);
		mbar_init(&bar[1], 1);
		mbar_fence_init();
	}
	__syncthreads();
	auto issue = [&](int g, int buf) { // one thread: the patches of group g -> tile buf
		const int      pb    = p0 + g * G::PPB;
		const int      np    = min(G::PPB, P - pb);
		const unsigned bytes = (unsigned) (np * G::NC * sizeof(double));
		fence_proxy_async();
		mbar_expect_tx(&bar[buf], bytes);
		tma_load_1d(Ut + (size_t) buf * G::PPB * G::NC, u + (size_t) pb * G::NC, bytes, &bar[buf]);
	};
	int    g  = blockIdx.x;
	double d0 = 0.0, d1 = 0.0;
	if (t == 0 && g < nblk) issue(g, 0);
	for (int it = 0; g < nblk; g += gridDim.x, it++) {
		const int     buf   = it & 1;
		const double *U     = Ut + ((size_t) buf * G::PPB + pp) * G::NC;
		double *      Gp    = Gh + (size_t) pp * G::S * G::M;
		const int     p     = p0 + g * G::PPB + pp;
		const bool    valid = p < P;
		// the other tile was last read in the previous iteration, before its closing barrier
		if (t == 0 && g + (int) gridDim.x < nblk) issue(g + gridDim.x, buf ^ 1);
		if (g + (int) gridDim.x < nblk) {
			const int pn = p0 + (g + gridDim.x) * G::PPB + pp;
			if (pn < P) { // pull the next patch's f and faces into L2 now; they are demanded next iteration
				if (MODE != 0) prefetch_patch_l2<D, N>(f, pn, m);
				prefetch_faces_l2<D, N>(meta, pn, m, F);
			}
		}
		double r[N];
		if (MODE != 0) {
#pragma unroll
			for (int k = 0; k < N; k++) r[k] = valid ? __ldg(f + (size_t) p * G::NC + k * G::M + m) : 0.0;
		}
		// ---- ghost faces of this patch: entry m of every side (independent of the tile, overlaps the bulk copy) ----
		double inv_h2 = 0.0;
		int    orth = -1, parent = 0;
		if (valid) {
			const PatchMeta &pm = meta[p];
			inv_h2              = pm.inv_h2;
			orth                = pm.orth_on_parent;
			parent              = pm.parent_idx;
			int    ty[G::S];
			double own[G::S], gm[G::S];
			const FaceVals<D, N, FV_PLAIN> fvals{F, nullptr, meta};
			gamma_all_sides(pm, p, m, fvals, ty, own, gm);
#pragma unroll
			for (int s = 0; s < G::S; s++) {
				double gh;
				if (ty[s] == NBR_NONE) gh = ((pm.neumann >> s) & 1) ? own[s] : -own[s];
				else gh = 2.0 * gm[s] - own[s];
				Gp[s * G::M + m] = gh;
			}
		}
		__syncthreads();                 // ghost faces visible
		mbar_wait(&bar[buf], (it >> 1) & 1); // the tile has landed
		// ---- stencil, marching along the last axis; in-plane neighbours come from the tile or from a ghost face ----
		{
			constexpr int ST = G::M; // tile stride along the last axis
			const double *cp = U + m;
			const double *wp, *ep;
			int           ws, es;
			if (D == 2) { // x-face entries are indexed by y = k
				wp = x > 0 ? cp - 1 : Gp + 0 * G::M, ws = x > 0 ? ST : 1;
				ep = x < N - 1 ? cp + 1 : Gp + 1 * G::M, es = x < N - 1 ? ST : 1;
			} else { // x-face entries (y, z = k): y + N k
				wp = x > 0 ? cp - 1 : Gp + 0 * G::M + y, ws = x > 0 ? ST : N;
				ep = x < N - 1 ? cp + 1 : Gp + 1 * G::M + y, es = x < N - 1 ? ST : N;
			}
			const double *sp = nullptr, *np_ = nullptr;
			int           ss = 0, ns = 0;
			if (D == 3) { // y-face entries (x, z = k): x + N k
				sp = y > 0 ? cp - N : Gp + 2 * G::M + x, ss = y > 0 ? ST : N;
				np_ = y < N - 1 ? cp + N : Gp + 3 * G::M + x, ns = y < N - 1 ? ST : N;
			}
			double lo = Gp[(G::S - 2) * G::M + m]; // ghost below the first cell of the pencil
			double ce = cp[0];
#pragma unroll
			for (int k = 0; k < N; k++) {
				const double hi = (k + 1 < N) ? cp[(k + 1) * ST] : Gp[(G::S - 1) * G::M + m];
				double       acc;
				if (D == 2) acc = (wp[k * ws] - 2 * ce + ep[k * es]) + (lo - 2 * ce + hi);
				else acc = (wp[k * ws] - 2 * ce + ep[k * es]) + (sp[k * ss] - 2 * ce + np_[k * ns]) + (lo - 2 * ce + hi);
				if (MODE == 3) {
					const double o = acc * inv_h2;
					d0             = fma(o, r[k], d0);
					d1             = fma(o, o, d1);
					r[k]           = o;
				} else {
					r[k] = (MODE == 0) ? acc * inv_h2 : r[k] - acc * inv_h2;
				}
				lo = ce;
				ce = hi;
			}
		}
		__syncthreads(); // all reads of this tile and of the ghost faces are done
		if (MODE != 2) {
			if (valid) {
				double *op = out + (size_t) p * G::NC + m;
#pragma unroll
				for (int k = 0; k < N; k++) op[k * G::M] = r[k];
			}
		} else {
			// restriction straight from registers: pairs along the last axis in-thread, x (and y) partners through shuffles
			constexpr int H = N / 2;
			double        a[H];
#pragma unroll
			for (int j = 0; j < H; j++) {
				a[j] = r[2 * j] / (1 << D) + r[2 * j + 1] / (1 << D);
				a[j] += __shfl_xor_sync(0xffffffffu, a[j], 1);
				if (D == 3) a[j] += __shfl_xor_sync(0xffffffffu, a[j], N);
			}
			if (valid) {
				double *dst = coarse + (size_t) parent * G::NC;
				if (orth < 0) { // patch present on both levels: copy
#pragma unroll
					for (int k = 0; k < N; k++) dst[k * G::M + m] = r[k];
				} else if ((x & 1) == 0 && (y & 1) == 0) {
					const int ox = (orth & 1) * H, oy = ((orth >> 1) & 1) * H, oz = ((orth >> (D - 1)) & 1) * H;
					if (D == 2) {
#pragma unroll
						for (int j = 0; j < H; j++) dst[(j + oy) * N + (x / 2 + ox)] = a[j];
					} else {
#pragma unroll
						for (int j = 0; j < H; j++) dst[((j + oz) * N + (y / 2 + oy)) * N + (x / 2 + ox)] = a[j];
					}
				}
			}
		}
	}
	if (MODE == 3) block_partials2(d0, d1, partial, pstride);
}
template <int D, int N> constexpr size_t apply_tma_smem_bytes()
{
	using G = Geo<D, N>;
	return sizeof(double) * (size_t) (2 * G::PPB * G::NC + G::PPB * G::S * G::M);
}

// ---------------------------------------------------------------------------------------------
// 32^3 patches: one (patch, slab of 8 z planes) item per iteration.  The slab and the planes below / above it that lie
// inside the patch are contiguous in memory: one bulk copy of 64-80 KB into a tile of ten planes [10][32][32] (plane 0 /
// plane 9 hold the z ghost plane at the bottom / top slab of a patch instead, written by the threads).  The x / y ghost
// faces of the slab live in GX[2][8][32], GY[2][8][32].
// ---------------------------------------------------------------------------------------------
constexpr size_t apply3d32_tma_smem_bytes() { return sizeof(double) * (10 * 1024 + 4 * 256); }
template <int MODE>
__global__ void __launch_bounds__(TGPU_THREADS, 2)
apply3d32_tma_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ u, const double *__restrict__ f,
                     const double *__restrict__ F, double *__restrict__ out, double *__restrict__ partial = nullptr, int pstride = 0)
{
	constexpr int N = 32, M = N * N, NC = N * N * N;
	extern __shared__ __align__(16) double U[]; // [10][32][32], then GX[2][256], GY[2][256]
	double *            GX = U + 10 * M;
	double *            GY = GX + 2 * 256;
	__shared__ uint64_t bar;
	const int           t = threadIdx.x, lo = t & 31, hi = t >> 5;
	pdl_launch_dependents();
	pdl_wait();
	if (t == 0) {
		mbar_init(&bar, 1);
		mbar_fence_init();
	}
	__syncthreads();
	const int nitems = (P - p0) * 4;
	int       n      = 0;
	double    d0 = 0.0, d1 = 0.0; // MODE 3: partial sums of out . f and out . out
	for (int it = blockIdx.x; it < nitems; it += gridDim.x, n++) {
		const int        p  = p0 + (it >> 2), zs = it & 3;
		const PatchMeta &pm = meta[p];
		const double *   up = u + (size_t) p * NC;
		if (t == 0) { // planes zs*8 - 1 .. zs*8 + 8 that exist inside the patch -> tile planes 0 .. 9
			const int      z0 = max(zs * 8 - 1, 0), z1 = min(zs * 8 + 8, N - 1);
			const unsigned bytes = (unsigned) ((z1 - z0 + 1) * M * sizeof(double));
			fence_proxy_async();
			mbar_expect_tx(&bar, bytes);
			tma_load_1d(U + (size_t) (z0 - (zs * 8 - 1)) * M, up + (size_t) z0 * M, bytes, &bar);
		}
		const FaceVals<3, N, FV_PLAIN> fv{F, nullptr, meta};
		auto ghost = [&](int s, int m) {
			const double a = fv.get(p, 0, -1, s, m);
			if (pm.nbr_type[s] == NBR_NONE) return ((pm.neumann >> s) & 1) ? a : -a;
			return 2.0 * gamma_entry(pm, p, s, m, fv) - a;
		};
		{
			const int zl = hi, m = lo + N * (zs * 8 + zl);
			GX[zl * 32 + lo]       = ghost(0, m); // x faces: entry (y, z)
			GX[256 + zl * 32 + lo] = ghost(1, m);
			GY[zl * 32 + lo]       = ghost(2, m); // y faces: entry (x, z)
			GY[256 + zl * 32 + lo] = ghost(3, m);
			if (zs == 0 || zs == 3) { // the z ghost plane goes into the tile plane the bulk copy leaves alone
				const int s = zs == 0 ? 4 : 5, gp = zs == 0 ? 0 : 9;
#pragma unroll
				for (int i = 0; i < 4; i++) {
					const int mm    = t + TGPU_THREADS * i;
					U[gp * M + mm] = ghost(s, mm);
				}
			}
		}
		__syncthreads();
		mbar_wait(&bar, n & 1);
		const double inv_h2 = pm.inv_h2;
#pragma unroll
		for (int j = 0; j < 4; j++) {
			const int     x = lo, y = hi + 8 * j;
			const double *cp = U + M + y * N + x; // cell (x, y) of the slab's first plane (tile plane 1)
			const double *wp = x > 0 ? cp - 1 : GX + y, *ep = x < N - 1 ? cp + 1 : GX + 256 + y;
			const int     ws = x > 0 ? M : 32, es = x < N - 1 ? M : 32;
			const double *sp = y > 0 ? cp - N : GY + x, *np_ = y < N - 1 ? cp + N : GY + 256 + x;
			const int     ss = y > 0 ? M : 32, ns = y < N - 1 ? M : 32;
			double        lo_v = cp[-M], ce = cp[0];
#pragma unroll
			for (int k = 0; k < 8; k++) {
				const double hi_v = cp[(k + 1) * M];
				const double acc  = (wp[k * ws] - 2 * ce + ep[k * es]) + (sp[k * ss] - 2 * ce + np_[k * ns]) + (lo_v - 2 * ce + hi_v);
				const size_t o    = (size_t) p * NC + (size_t) (zs * 8 + k) * M + y * N + x;
				if (MODE == 3) {
					const double v = acc * inv_h2;
					d0             = fma(v, __ldg(f + o), d0);
					d1             = fma(v, v, d1);
					out[o]         = v;
				} else {
					out[o] = (MODE == 0) ? acc * inv_h2 : __ldg(f + o) - acc * inv_h2;
				}
				lo_v              = ce;
				ce                = hi_v;
			}
		}
		__syncthreads();
	}
	if (MODE == 3) block_partials2(d0, d1, partial, pstride);
}
} // namespace tgpu
