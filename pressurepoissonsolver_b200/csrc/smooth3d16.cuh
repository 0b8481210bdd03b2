// smooth3d16.cuh - block-Jacobi smoother specialised for the flagship geometry D = 3, N = 16
// (one patch = 256 pencils = one 256-thread CTA).  Included by kernels.cuh.
//
// Same arithmetic as the generic smooth_kernel (SchurHelper::solveWithSolution, SchurHelper.h:319-331:
// interface values + StarPatchOp::addInterfaceToRHS, StarPatchOp.h:185-203 + the DST patch solve of
// PatchSolvers/FftwPatchSolver.h:174-206 / DftPatchSolver.h:173-216); what changes is how the tile moves:
//   * tile layout x + 18 y + 290 z (rows 16-byte aligned): z- and y-pencil accesses are conflict-free
//     64-bit, x-row accesses are conflict-free 128-bit (half the LDS/STS count), column accesses
//     (x fixed, y varying) are 2-way conflicted at worst;
//   * transform order z, x, (y forward, eigenvalues, y inverse), x, z with warp w owning the rows
//     y in {2w, 2w+1}: the z<->x transposes stay inside a warp (__syncwarp instead of a CTA barrier),
//     leaving two CTA barriers around the y phase (+1 when gamma has to be subtracted first);
//   * f is loaded straight from memory into the z pencils (a warp's load covers two whole 128-byte lines) while
//     a prefetch pulls the next patch into L2: no staging tile, one tile per CTA; sweeps from a zero guess fit
//     64 registers and run four CTAs per SM, the others three;
//   * the y axis is not transformed: with z and x diagonalised each (k_x, k_z) pencil is a tridiagonal system,
//     solved by a two-sided elimination with tabulated multipliers (TriSolve, 56 operations instead of 248);
//   * the interface values gamma of the NEXT patch are gathered one side per transform: the four loads
//     of a side (own face, neighbour face, and the coarse correction under both when the prolongation
//     is fused in) are issued before a transform and combined after it, so their L2/HBM latency hides
//     behind the transform instead of stalling the whole CTA at the top of an iteration; x- and y-face
//     values wait in a 8 KB shared-memory face buffer and are subtracted from the boundary pencils right
//     after the next patch's load, z-face values wait in two registers;
//   * WRITE_U = false (sweeps whose u is only ever seen through its boundary slices: every sweep but
//     the last of a level visit in the fused cycle): the last inverse transform is evaluated in full
//     only for the 60 pencils on the patch boundary (warps 0-1); the other pencils compute just their
//     two z-face values (16 DFMA instead of 116) and nothing but the face buffer is written.
#pragma once

namespace tgpu
{
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

constexpr int    S16_BLOCK = TGPU_THREADS; // threads per CTA (the host launches with this)
constexpr int    S16_ROW = 18, S16_PL = 290, S16_TILE = 16 * S16_PL;
// f is loaded straight into the z pencils (the next patch is pulled into L2 meanwhile): one tile per CTA.  Sweeps
// from a zero guess fit 64 registers and run four CTAs per SM, the others three.
__host__ __device__ constexpr int    s16_ctas_per_sm(bool zero_guess, bool neu = false)
{
	return neu ? 2 : (zero_guess ? 4 : 3); // (the Neumann variant's general transforms need the registers)
}
constexpr size_t smooth3d16_smem_bytes() { return sizeof(double) * S16_TILE; }

// refinement-boundary sides are rare: keep their (large) code out of line
template <bool PROLONG>
__device__ __noinline__ double iface_gamma_slow16(const PatchMeta *__restrict__ meta, int p, int s, int m,
                                                  const double *__restrict__ F, const double *__restrict__ uc)
{
	const FaceVals<3, 16, PROLONG ? FV_PROLONG : FV_PLAIN> fv{F, uc, meta};
	return iface_gamma<3, 16, PROLONG ? FV_PROLONG : FV_PLAIN>(meta[p], p, s, m, fv);
}
// Gather descriptor of one patch side: everything that is uniform over the 256 face entries, resolved
// once per patch by one thread, so that an entry's four loads are "base + per-thread constant offset":
//   (2/h^2) gamma = c (0.5 (a0[t] + a1[o]) + 0.5 (b0[t] + wb b1[o])),  o = the entry's offset on the coarse plane
// a0/b0: own / neighbour face slice (FaceVals), a1/b1: the parent patches' cells under them
// (DrctIntp.h:92-111; only read when the prolongation is fused in), c = 0 on sides without a neighbour,
// wb = 0 for halo faces that already carry the correction.  sa/sb: 1 = the parent is a refined patch (two
// entries per coarse cell, o = entry >> 1 per axis), 0 = the "parent" is the same patch on the coarser level
// (leaves of an adaptive mesh that are not at the finest tree level: copy-add, DrctIntp.h:107-110).
// Sides that need the general code (coarse/fine neighbours) are flagged in `slow`.
struct __align__(16) GDesc16 {
	unsigned a0, b0, a1, b1; // element offsets into F (a0, b0) and into uc (a1, b1; F when no prolongation is fused in)
	double   c;
	int      flags, pad;
};
enum { GD_SA = 1, GD_SB = 2, GD_WB = 4, GD_SLOW = 8 };
struct GPatch16 {
	GDesc16 d[6];
	double  h2;
	int     neu, pad; // Neumann bits of the patch (a level with Neumann patches: this kernel skips them, see skip_neumann)
};
template <bool PROLONG>
__device__ __forceinline__ void make_gdesc16(const PatchMeta &pm, int p, int s, GPatch16 &out)
{
	GDesc16 &  d   = out.d[s];
	const int  ty  = pm.nbr_type[s];
	const int  ax  = s >> 1;
	const int  st  = (ax == 0) ? 1 : (ax == 1 ? 16 : 256); // stride of the face-normal axis
	bool       slow = ty > NBR_NORMAL;
	d.a0 = d.b0 = ((unsigned) p * 6 + s) * 256;
	d.a1 = d.b1 = 0;
	d.c         = (ty == NBR_NONE) ? 0.0 : 2.0 * pm.inv_h2;
	int fl      = GD_SA | GD_SB | GD_WB;
	if (ty == NBR_NORMAL) {
		d.b0 = ((unsigned) pm.nbr_idx[s][0] * 6 + (s ^ 1)) * 256;
		if (PROLONG) {
			const int o = pm.orth_on_parent, qp = pm.nbr_parent[s], qo = pm.nbr_orth[s];
			if (o >= 0) d.a1 = (unsigned) pm.parent_idx * 4096 + 8 * ((o & 1) + 16 * ((o >> 1) & 1) + 256 * ((o >> 2) & 1)) + ((s & 1) ? 7 * st : 0);
			else d.a1 = (unsigned) pm.parent_idx * 4096 + ((s & 1) ? 15 * st : 0), fl &= ~GD_SA;
			if (qp < 0) d.b1 = d.a1, fl = (fl & ~(GD_SB | GD_WB)) | ((fl & GD_SA) ? GD_SB : 0);
			else if (qo >= 0) d.b1 = (unsigned) qp * 4096 + 8 * ((qo & 1) + 16 * ((qo >> 1) & 1) + 256 * ((qo >> 2) & 1)) + ((s & 1) ? 0 : 7 * st);
			else d.b1 = (unsigned) qp * 4096 + ((s & 1) ? 0 : 15 * st), fl &= ~GD_SB;
		}
	}
	if (slow) {
		d.a0 = d.b0 = ((unsigned) p * 6 + s) * 256; // harmless addresses; the value comes from iface_gamma_slow16
		d.a1 = d.b1 = 0;
		fl          = GD_SA | GD_SB | GD_WB | GD_SLOW;
	}
	d.flags = fl;
}
template <bool PROLONG> struct SideGamma16 {
	double a0, a1, b0, b1;
	// AX: face-normal axis; entry t = (lo, hi) lies over cell (lo >> s) * A + (hi >> s) * B of the parent's plane
	template <int AX>
	__device__ __forceinline__ void issue(const GDesc16 &d, int t, int lo, int hi, const double *__restrict__ F, const double *__restrict__ uc)
	{
		constexpr int A = (AX == 0) ? 16 : 1, B = (AX == 2) ? 16 : 256;
		const uint4   o = *reinterpret_cast<const uint4 *>(&d);
		a0 = __ldg(F + o.x + t);
		b0 = __ldg(F + o.y + t);
		a1 = b1 = 0.0;
		if (PROLONG) {
			const int fl = d.flags, sa = fl & GD_SA, sb = (fl >> 1) & 1;
			a1 = __ldg(uc + o.z + ((lo >> sa) * A + (hi >> sa) * B));
			b1 = __ldg(uc + o.w + ((lo >> sb) * A + (hi >> sb) * B));
		}
	}
	__device__ __forceinline__ double finish(const GPatch16 &gp, int s, const PatchMeta *__restrict__ meta, int p, int t,
	                                         const double *__restrict__ F, const double *__restrict__ uc) const
	{
		const GDesc16 &d  = gp.d[s];
		const double   c  = d.c;
		const int      fl = d.flags;
		double         g  = c * (0.5 * (a0 + a1) + 0.5 * (b0 + ((fl & GD_WB) ? b1 : 0.0)));
		if (fl & GD_SLOW) g = c * iface_gamma_slow16<PROLONG>(meta, p, s, t, F, uc);
		return g;
	}
};

// tables of the general patch solve (smooth_kernel's): dense transform matrices by kind and the eigenvalue rows
struct NeuTabs {
	const double * mats = nullptr, *lam = nullptr;
	const int32_t *list = nullptr; // the patches the launch sweeps (those of the range with Neumann sides), ascending
	int            n    = 0;
};
// HALO = false compiles the multi-GPU hand-over (HaloSync / halo_push_cta) out: the single-GPU instantiations carry none of it
// NEU = true: the instantiation for the patches WITH Neumann domain sides of a level (it sweeps exactly those of the range,
// from the list in NeuTabs; the plain instantiation launched with skip_neumann sweeps the others): same pipeline - f straight into the z
// pencils, interface values of the next patch gathered behind the transforms, slices emitted from registers - with the
// transform of each axis chosen by the patch's boundary kinds (general_transform: DST-II/III, DST-IV / DCT-IV in generated
// fast form, DCT-II/III dense) and the y axis transformed and divided by the eigenvalue sums like the others instead of the
// tridiagonal solve (whose multiplier table is the all-Dirichlet one).  Same arithmetic per patch as smooth_kernel's
// general path (DftPatchSolver.h:173-216 with the kinds of DftPatchSolver.h:237-289).
template <bool ZERO_GUESS, bool EMIT, bool PROLONG, bool WRITE_U, bool HALO = false, bool NEU = false>
__global__ void __launch_bounds__(TGPU_THREADS, s16_ctas_per_sm(ZERO_GUESS, NEU))
smooth3d16_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ f, double *__restrict__ u,
                  const double *__restrict__ Fin, double *__restrict__ Fout, const double *__restrict__ tri,
                  const double *__restrict__ uc, HaloSync hs = HaloSync{}, int skip_neumann = 0, NeuTabs nt = NeuTabs{})
{
	static_assert(!NEU || !HALO, "the Neumann instantiation is single-GPU");
	// skip_neumann != 0: patches with Neumann domain sides are left alone (their patch solve is not the plain Dirichlet
	// one; the general path of smooth_kernel sweeps them in a second launch over the same range); the interface values of
	// the next patch are still gathered while one is skipped
	constexpr int N = 16, ROW = S16_ROW, PL = S16_PL;
	using G = Geo<3, 16>;
	static_assert(WRITE_U || EMIT, "a sweep must produce something");
	extern __shared__ __align__(16) double S[];
	// neighbour-table entry of the patch after the next (staged with cp.async) and the gather descriptors
	// of the current / next patch derived from it
	constexpr int                   MW = (int) (sizeof(PatchMeta) / sizeof(double));
	__shared__ __align__(16) double metaS[MW];
	__shared__ GPatch16             GD[2];
	// (2/h^2) gamma on the x and y faces of the patch about to be solved, entry t of side s at Gs[s * 256 + t]
	// (the z-face values stay in the registers of the thread that needs them)
	__shared__ double Gs[ZERO_GUESS ? 1 : 4 * 256];
	const int t = threadIdx.x, lo = t & 15, hi = t >> 4;
	const int npatch = NEU ? nt.n : P - p0;
	auto      pid    = [&](int gg) { return NEU ? (int) __ldg(nt.list + gg) : p0 + gg; }; // patch of work item gg (CTA-uniform)
	Mags<N> mg;
	mg.load();
	pdl_launch_dependents();
	pdl_wait();
	if (!ZERO_GUESS) if (HALO) halo_push<3, 16>(hs, meta);

	// one thread per side (lane 31 of warps 0-5) resolves the descriptors of patch q into GD[slot]
	auto describe = [&](const PatchMeta &pm, int q, int slot) {
		if ((t & 31) == 31 && t < 6 * 32) make_gdesc16<PROLONG>(pm, q, t >> 5, GD[slot]);
		if (t == 6 * 32 + 31) GD[slot].h2 = pm.h2, GD[slot].neu = pm.neumann;
	};

	int g = blockIdx.x;
	// multi-GPU: the CTA polls the peers' flags itself before the first patch whose gamma needs halo faces (HaloSync)
	bool halo_ok = false;
	if (g >= npatch) {
		if (!ZERO_GUESS) if (HALO) halo_finish(hs);
		return;
	}
	double gz0 = 0.0, gz1 = 0.0; // (2/h^2) gamma of entry t on the two z faces of the current patch
	SideGamma16<PROLONG> sg;
	if (!ZERO_GUESS) {
		// first patch of this CTA: nothing to hide the gathers behind
		const int p = pid(g);
		if (HALO) halo_wait_cta(hs, p, halo_ok);
		describe(meta[p], p, 0);
		if (g + (int) gridDim.x < npatch) {
			const int p2 = pid(g + gridDim.x);
			describe(meta[p2], p2, 1);
		}
		__syncthreads();
		// all six sides' loads in flight at once (no transform registers are live yet): one memory round trip instead
		// of six, which is most of the latency of a coarse level where every CTA solves a single patch
		SideGamma16<PROLONG> s6[6];
		s6[0].template issue<0>(GD[0].d[0], t, lo, hi, Fin, uc);
		s6[1].template issue<0>(GD[0].d[1], t, lo, hi, Fin, uc);
		s6[2].template issue<1>(GD[0].d[2], t, lo, hi, Fin, uc);
		s6[3].template issue<1>(GD[0].d[3], t, lo, hi, Fin, uc);
		s6[4].template issue<2>(GD[0].d[4], t, lo, hi, Fin, uc);
		s6[5].template issue<2>(GD[0].d[5], t, lo, hi, Fin, uc);
#pragma unroll
		for (int s = 0; s < 4; s++) Gs[s * 256 + t] = s6[s].finish(GD[0], s, meta, p, t, Fin, uc);
		gz0 = s6[4].finish(GD[0], 4, meta, p, t, Fin, uc);
		gz1 = s6[5].finish(GD[0], 5, meta, p, t, Fin, uc);
	}
	for (int it = 0; g < npatch; g += gridDim.x, it++) {
		const int       b    = it & 1;
		const int       p    = pid(g);
		const int       gn   = g + gridDim.x;
		const bool      next = gn < npatch;
		const int       pn   = NEU ? (next ? pid(gn) : p) : p0 + gn; // patch whose gamma is gathered during this iteration
		const int       pnn  = (gn + (int) gridDim.x < npatch) ? pid(gn + gridDim.x) : p; // the one after it
		const GPatch16 &gp   = GD[b ^ 1]; // its descriptors
		int             neu_p = 0; // Neumann bits of patch p
		// the previous patch's last stage has read the tile; Gs and the descriptors written during the
		// previous iteration become visible
		__syncthreads();
		if (HALO && !ZERO_GUESS && next) halo_wait_cta(hs, pn, halo_ok); // gamma of patch pn is gathered during this iteration
		const double h2 = ZERO_GUESS ? meta[p].h2 : GD[b].h2;
		// table entry of the patch after the next -> metaS (read by describe() after the next barrier but one)
		if (!ZERO_GUESS && t < MW && gn + (int) gridDim.x < npatch)
			cp_async8(&metaS[t], reinterpret_cast<const double *>(meta + pnn) + t, true);
		if (NEU || skip_neumann) neu_p = ZERO_GUESS ? meta[p].neumann : GD[b].neu;
		if (NEU ? neu_p == 0 : (skip_neumann && neu_p)) { // CTA-uniform: this patch belongs to the other launch
			if (!ZERO_GUESS) {
				// keep the pipeline of the next patch's interface values going: all six sides at once, nothing to hide behind
				SideGamma16<PROLONG> s6[6];
				if (next) {
					s6[0].template issue<0>(gp.d[0], t, lo, hi, Fin, uc);
					s6[1].template issue<0>(gp.d[1], t, lo, hi, Fin, uc);
					s6[2].template issue<1>(gp.d[2], t, lo, hi, Fin, uc);
					s6[3].template issue<1>(gp.d[3], t, lo, hi, Fin, uc);
					s6[4].template issue<2>(gp.d[4], t, lo, hi, Fin, uc);
					s6[5].template issue<2>(gp.d[5], t, lo, hi, Fin, uc);
				}
				cp_async_wait_all();
				__syncthreads(); // metaS has landed
				if (next) {
#pragma unroll
					for (int s = 0; s < 4; s++) Gs[s * 256 + t] = s6[s].finish(gp, s, meta, pn, t, Fin, uc);
					gz0 = s6[4].finish(gp, 4, meta, pn, t, Fin, uc);
					gz1 = s6[5].finish(gp, 5, meta, pn, t, Fin, uc);
					if (gn + (int) gridDim.x < npatch) describe(*reinterpret_cast<const PatchMeta *>(metaS), pnn, b);
				}
			}
			continue;
		}
		double v[N];
		{ // z forward: pencil (x, y) = (lo, hi)
			double *      q  = S + lo + hi * ROW;
			const double *fp = f + (size_t) p * G::NC + t;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = __ldcs(fp + k * G::M);
			if (next) { // pull the next patch into L2 while this one is transformed: 256 lines of 128 bytes
				prefetch_l2(f + (size_t) pn * G::NC + t * 16);
			}
			if (!ZERO_GUESS) {
				v[0] -= gz0;
				v[N - 1] -= gz1;
				// x faces: entry (y, z) belongs to the pencils x = 0 / 15; y faces: entry (x, z) to y = 0 / 15
				// (edge pencils take both, like StarPatchOp::addInterfaceToRHS visiting every side)
				if (lo == 0 || lo == N - 1) {
					const double *gq = Gs + (lo == 0 ? 0 : 256) + hi;
#pragma unroll
					for (int k = 0; k < N; k++) v[k] -= gq[16 * k];
				}
				if (hi == 0 || hi == N - 1) {
					const double *gq = Gs + (hi == 0 ? 512 : 768) + lo;
#pragma unroll
					for (int k = 0; k < N; k++) v[k] -= gq[16 * k];
				}
				if (next) sg.template issue<2>(gp.d[4], t, lo, hi, Fin, uc);
			}
			if (NEU) {
				general_transform<N>(nt.mats, axis_kind(neu_p, 2).fwd, v, q, PL, mg);
			} else {
				Dst2<N, N>::run(v, mg);
#pragma unroll
				for (int k = 0; k < N; k++) q[k * PL] = v[k];
			}
			if (!ZERO_GUESS && next) gz0 = sg.finish(gp, 4, meta, pn, t, Fin, uc);
		}
		__syncwarp(); // rows (y, k_z) with y in {2w, 2w+1} were produced by this warp
		double2 *rowp = reinterpret_cast<double2 *>(S + hi * ROW + lo * PL); // row (y, k_z) = (hi, lo)
		{
#pragma unroll
			for (int j = 0; j < N / 2; j++) {
				const double2 d = rowp[j];
				v[2 * j]        = d.x;
				v[2 * j + 1]    = d.y;
			}
			if (!ZERO_GUESS && next) sg.template issue<2>(gp.d[5], t, lo, hi, Fin, uc);
			if (NEU) {
				general_transform<N>(nt.mats, axis_kind(neu_p, 0).fwd, v, reinterpret_cast<double *>(rowp), 1, mg);
			} else {
				Dst2<N, N>::run(v, mg);
#pragma unroll
				for (int j = 0; j < N / 2; j++) rowp[j] = make_double2(v[2 * j], v[2 * j + 1]);
			}
			if (!ZERO_GUESS && next) gz1 = sg.finish(gp, 5, meta, pn, t, Fin, uc);
		}
		if (!ZERO_GUESS) cp_async_wait_all(); // metaS has landed (made visible by the barrier)
		__syncthreads();
		{ // y: pencil (k_x, k_z) = (lo, hi)
			double *q = S + lo + hi * PL;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = q[k * ROW];
			if (!ZERO_GUESS && next) sg.template issue<0>(gp.d[0], t, lo, hi, Fin, uc);
			if (NEU) {
				// transform along y as well and divide by the eigenvalue sum of (k_x, k_y, k_z) = (lo, k, hi)
				const AxisKind kx = axis_kind(neu_p, 0), ky = axis_kind(neu_p, 1), kz = axis_kind(neu_p, 2);
				general_transform<N>(nt.mats, ky.fwd, v, q, ROW, mg);
				const double rest     = __ldg(nt.lam + kx.lam * N + lo) + __ldg(nt.lam + kz.lam * N + hi);
				const double scale    = h2 * (8.0 / (N * N * N));
				const bool   singular = neu_p == 63 && t == 0; // all-Neumann patch: the constant mode is left out
#pragma unroll
				for (int k = 0; k < N; k++) v[k] = (singular && k == 0) ? 0.0 : q[k * ROW] * scale / (__ldg(nt.lam + ky.lam * N + k) + rest);
			} else {
				// z and x are diagonalised: what is left per (k_x, k_z) is a tridiagonal system along y
				TriSolve<N>::forward(v, tri + t, h2 * (4.0 / (N * N)));
			}
			double gx0 = 0.0, gx1 = 0.0;
			if (!ZERO_GUESS && next) {
				gx0 = sg.finish(gp, 0, meta, pn, t, Fin, uc);
				sg.template issue<0>(gp.d[1], t, lo, hi, Fin, uc);
			}
			if (NEU) {
				general_transform<N>(nt.mats, axis_kind(neu_p, 1).inv, v, q, ROW, mg);
			} else {
				TriSolve<N>::backward(v, tri + t);
#pragma unroll
				for (int k = 0; k < N; k++) q[k * ROW] = v[k];
			}
			if (!ZERO_GUESS && next) {
				gx1 = sg.finish(gp, 1, meta, pn, t, Fin, uc);
				Gs[t]       = gx0; // (this patch's values were consumed before the barrier above)
				Gs[256 + t] = gx1;
				// descriptors of the patch after the next; GD[b] was last read before this iteration's first barrier
				if (gn + (int) gridDim.x < npatch) describe(*reinterpret_cast<const PatchMeta *>(metaS), pnn, b);
			}
		}
		__syncthreads();
		double gy0 = 0.0;
		{ // x inverse
#pragma unroll
			for (int j = 0; j < N / 2; j++) {
				const double2 d = rowp[j];
				v[2 * j]        = d.x;
				v[2 * j + 1]    = d.y;
			}
			if (!ZERO_GUESS && next) sg.template issue<1>(gp.d[2], t, lo, hi, Fin, uc);
			if (NEU) {
				general_transform<N>(nt.mats, axis_kind(neu_p, 0).inv, v, reinterpret_cast<double *>(rowp), 1, mg);
			} else {
				Dst3<N, N>::run(v, mg);
#pragma unroll
				for (int j = 0; j < N / 2; j++) rowp[j] = make_double2(v[2 * j], v[2 * j + 1]);
			}
			if (!ZERO_GUESS && next) gy0 = sg.finish(gp, 2, meta, pn, t, Fin, uc);
		}
		if (WRITE_U || NEU) { // (the Neumann instantiation has no slices-only shortcut: full inverse, u stored only if wanted)
			__syncwarp();
			double *q = S + lo + hi * ROW; // z inverse: pencil (x, y) = (lo, hi)
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = q[k * PL];
			if (!ZERO_GUESS && next) sg.template issue<1>(gp.d[3], t, lo, hi, Fin, uc);
			if (NEU) {
				general_transform<N>(nt.mats, axis_kind(neu_p, 2).inv, v, q, PL, mg);
#pragma unroll
				for (int k = 0; k < N; k++) v[k] = q[k * PL];
			} else {
				Dst3<N, N>::run(v, mg);
			}
			double *up = u + (size_t) p * G::NC + t;
			if (WRITE_U) {
#pragma unroll
				for (int k = 0; k < N; k++) __stcs(up + k * G::M, v[k]); // streaming store: u is not read again soon, the face buffers should stay in L2
			}
			if (EMIT) {
				double *Fp       = Fout + (size_t) p * G::S * G::M;
				Fp[4 * G::M + t] = v[0];
				Fp[5 * G::M + t] = v[N - 1];
				if (lo == 0) {
#pragma unroll
					for (int k = 0; k < N; k++) Fp[0 * G::M + k * N + hi] = v[k];
				}
				if (lo == N - 1) {
#pragma unroll
					for (int k = 0; k < N; k++) Fp[1 * G::M + k * N + hi] = v[k];
				}
				if (hi == 0) {
#pragma unroll
					for (int k = 0; k < N; k++) Fp[2 * G::M + k * N + lo] = v[k];
				}
				if (hi == N - 1) {
#pragma unroll
					for (int k = 0; k < N; k++) Fp[3 * G::M + k * N + lo] = v[k];
				}
			}
		} else {
			__syncthreads();
			if (!ZERO_GUESS && next) sg.template issue<1>(gp.d[3], t, lo, hi, Fin, uc);
			// Only the boundary-cell slices of u are needed.  Warp 0: the x = 0 and x = 15 columns, warp 1:
			// the y = 0 and y = 15 rows (+ 4 interior pencils): full inverse transform; warps 2-7: the other
			// 192 interior pencils, z-face values only:
			//   u_0 = sum_j T[0][j] v_j,  u_15 = sum_j (-1)^j T[0][j] v_j,
			//   T[0][j] = sin(pi (j+1) / 32), T[0][15] = 1/2   (DftPatchSolver.h:269-281)
			double *  Fp   = Fout + (size_t) p * G::S * G::M;
			const int lane = t & 31;
			if (t < 64) {
				int x, y;
				if (t < 32) {
					x = (lane < 16) ? 0 : N - 1;
					y = lane & 15;
				} else if (lane < 28) {
					x = 1 + lane % 14;
					y = (lane < 14) ? 0 : N - 1;
				} else {
					x = 11 + (lane - 28); // interior pencils 192..195 = (11..14, 14)
					y = 14;
				}
				const double *q = S + x + y * ROW;
#pragma unroll
				for (int k = 0; k < N; k++) v[k] = q[k * PL];
				Dst3<N, N>::run(v, mg);
				Fp[4 * G::M + x + N * y] = v[0];
				Fp[5 * G::M + x + N * y] = v[N - 1];
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
			} else {
				const int     idx = t - 64, x = 1 + idx % 14, y = 1 + idx / 14;
				const double *q   = S + x + y * ROW;
				double        E = 0.0, O = 0.0;
#pragma unroll
				for (int j = 0; j < N; j += 2) {
					E = fma(mg.sinq(j + 1), q[j * PL], E);
					O = fma((j + 1 == N - 1) ? 0.5 : mg.sinq(j + 2), q[(j + 1) * PL], O);
				}
				double *fz = &Fp[4 * G::M + x + N * y]; // z faces: entry (x, y) on side 4, then on side 5
				*fz        = E + O;
				fz[G::M]   = E - O;
			}
		}
		if (!ZERO_GUESS && next) {
			Gs[512 + t] = gy0;
			Gs[768 + t] = sg.finish(gp, 3, meta, pn, t, Fin, uc);
		}
	}
	if (!ZERO_GUESS) if (HALO) halo_finish(hs);
}
} // namespace tgpu
