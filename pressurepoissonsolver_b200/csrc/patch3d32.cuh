// patch3d32.cuh - kernels for D = 3, N = 32 patches (BASELINE config D).  Included by kernels.cuh.
//
// A 32^3 patch is 256 KB of fp64: more than one SM's shared memory, so the one-CTA-one-tile scheme of the
// smaller sizes does not apply.
//   smooth3d32c_kernel  the smoother the library uses: a thread-block cluster of two CTAs holds the whole patch in the
//                       shared memory of two SMs; x and y are transformed, z is a two-sided tridiagonal elimination split
//                       over the pair (see the comment above the kernel)
//   iface_rhs32_kernel  the interface part of the right-hand side of the sweeps that do not start from zero, transformed
//                       for smooth3d32c_kernel
//   smooth3d32n_kernel  levels with Neumann domain sides: general dense-transform path through an L2-resident scratch block
//   face_residual_restrict_big_kernel   residual + restriction from face data (see kernels.cuh)
// The operator apply for 32^3 patches is apply3d32_tma_kernel (apply_tma.cuh).
// Reference functions replaced: same as smooth_kernel / face_residual_restrict_kernel.
#pragma once
#include <vector>

namespace tgpu
{
// interface value gamma of entry m on side s (0 on sides without a neighbour); same expressions as
// gamma_all_sides / iface_gamma
template <int D, int N, int MODE>
__device__ __forceinline__ double gamma_entry(const PatchMeta &pm, int p, int s, int m, const FaceVals<D, N, MODE> &fv)
{
	const int ty = pm.nbr_type[s];
	if (ty == NBR_NONE) return 0.0;
	if (ty == NBR_NORMAL) {
		const double a = fv.get(p, pm.parent_idx, pm.orth_on_parent, s, m);
		const double b = fv.get(pm.nbr_idx[s][0], pm.nbr_parent[s], pm.nbr_orth[s], s ^ 1, m);
		return 0.5 * a + 0.5 * b;
	}
	return iface_gamma<D, N, MODE>(pm, p, s, m, fv);
}

// ---------------------------------------------------------------------------------------------
// smooth3d32c_kernel: the 32^3 patch solve on a pair of SMs (thread-block cluster of two CTAs), whole patch
// resident in shared memory, no scratch block.
//   The z axis is not transformed (TriSolve, kernels.cuh): with x and y diagonalised, every (k_x, k_y) pencil
//   is a tridiagonal system along z whose two-sided elimination runs from z = 0 upwards and from z = 31
//   downwards with the same multipliers.  That is exactly a split over two CTAs: CTA 0 owns the planes
//   z = 0..15, CTA 1 the planes z = 31..16 (local plane j <-> elimination step j in both), and the only data the
//   halves exchange is the last plane of eliminated right-hand sides (8 KB each way, read through distributed
//   shared memory after one cluster barrier) for the 2 x 2 system in the middle.
//   Per CTA: 512 threads = 16 warps, warp w owns local plane w for the y and x transforms (warp-local
//   transposes), the z recurrences are element-wise over the planes (two pencils per thread).
//   f goes straight from memory into the y pencils (a warp's load = one 256-byte row) and u straight from the
//   y pencils back to memory: HBM sees f once and u once, shared memory holds the 16 planes (136 KB).
//   Sweeps that do not start from zero read the interface part of their right-hand side, already transformed, from the
//   output of iface_rhs32_kernel (below).
// Same arithmetic as smooth_kernel (SchurHelper.h:319-331, FftwPatchSolver.h:174-206).
// ---------------------------------------------------------------------------------------------
constexpr int    C32_THREADS = 512, C32_ROW = 34, C32_PL = 32 * C32_ROW, C32_TILE = 16 * C32_PL;
constexpr int    C32_FV = 65; // row pitch of the face-vector staging [32][65] (faces-only sweeps, see the tail of the kernel)
// tile + two exchange planes (double buffered) + x-face output staging, and for the faces-only sweeps from a zero guess the
// face-vector staging (a 24 KB region, 188 KB in all: the carve-out step below 228 KB, which would leave the L1 28 KB instead
// of 60 KB - measured 4-7 % slower).  The other sweeps take 160 KB and leave the L1 92 KB.
template <bool ZERO_GUESS> constexpr size_t smooth3d32c_smem_bytes()
{
	return sizeof(double) * (C32_TILE + 2 * 1024 + 16 * 64 + (ZERO_GUESS ? 1024 + 16 * 128 : 0));
}
static_assert(32 * C32_FV <= 1024 + 16 * 128, "the face-vector staging of sweeps from a zero guess");
__device__ __forceinline__ unsigned cluster_ctarank()
{
	unsigned r;
	asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
	return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
	asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// value at the same shared-memory address in CTA `rank` of the cluster
__device__ __forceinline__ double ld_dsmem(const double *local, unsigned rank)
{
	unsigned a = (unsigned) __cvta_generic_to_shared(local), ra;
	double   v;
	asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(ra) : "r"(a), "r"(rank));
	asm volatile("ld.shared::cluster.f64 %0, [%1];\n" : "=d"(v) : "r"(ra) : "memory");
	return v;
}
template <bool PROLONG>
__device__ __noinline__ double gamma_entry32(const PatchMeta *__restrict__ meta, int p, int s, int m, const double *__restrict__ F,
                                             const double *__restrict__ uc)
{
	const FaceVals<3, 32, PROLONG ? FV_PROLONG : FV_PLAIN> fv{F, uc, meta};
	return gamma_entry(meta[p], p, s, m, fv);
}
// Gather descriptor of one patch side (the 32^3 analogue of GDesc16, smooth3d16.cuh): everything that is uniform over the
// 1024 face entries, resolved once per patch by one thread, so that an entry's four loads are "base + per-thread constant":
//   (2/h^2) gamma = c (0.5 (a0[m] + a1[o]) + 0.5 (b0[m] + wb b1[o])),  o = the entry's offset on the parent's plane
// a0 / b0: own / neighbour face slice, a1 / b1: the parents' cells under them (DrctIntp.h:92-111, only with the prolongation
// fused in), c = 0 on sides without a neighbour, wb = 0 for halo faces that already carry the correction, SA / SB: the
// parent is a refined patch (two entries per coarse cell) or the same patch one level up (copy-add).  Sides with coarse /
// fine neighbours are flagged GD_SLOW and take gamma_entry32.
struct __align__(16) GDesc32 {
	unsigned a0, b0, a1, b1; // element offsets into F (a0, b0) and into uc (a1, b1)
	double   c;
	int      flags, pad;
};
struct GPatch32 {
	GDesc32 d[6];
};
template <bool PROLONG>
__device__ __forceinline__ void make_gdesc32(const PatchMeta &pm, int p, int s, GPatch32 &out)
{
	GDesc32 & d  = out.d[s];
	const int ty = pm.nbr_type[s];
	const int ax = s >> 1;
	const int st = (ax == 0) ? 1 : (ax == 1 ? 32 : 1024); // stride of the face-normal axis
	d.a0 = d.b0 = ((unsigned) p * 6 + s) * 1024;
	d.a1 = d.b1 = 0;
	d.c         = (ty == NBR_NONE) ? 0.0 : 2.0 * pm.inv_h2;
	int fl      = GD_SA | GD_SB | GD_WB;
	if (ty == NBR_NORMAL) {
		d.b0 = ((unsigned) pm.nbr_idx[s][0] * 6 + (s ^ 1)) * 1024;
		if (PROLONG) {
			const int o = pm.orth_on_parent, qp = pm.nbr_parent[s], qo = pm.nbr_orth[s];
			if (o >= 0) d.a1 = (unsigned) pm.parent_idx * 32768 + 16 * ((o & 1) + 32 * ((o >> 1) & 1) + 1024 * ((o >> 2) & 1)) + ((s & 1) ? 15 * st : 0);
			else d.a1 = (unsigned) pm.parent_idx * 32768 + ((s & 1) ? 31 * st : 0), fl &= ~GD_SA;
			if (qp < 0) d.b1 = d.a1, fl = (fl & ~(GD_SB | GD_WB)) | ((fl & GD_SA) ? GD_SB : 0);
			else if (qo >= 0) d.b1 = (unsigned) qp * 32768 + 16 * ((qo & 1) + 32 * ((qo >> 1) & 1) + 1024 * ((qo >> 2) & 1)) + ((s & 1) ? 0 : 15 * st);
			else d.b1 = (unsigned) qp * 32768 + ((s & 1) ? 0 : 31 * st), fl &= ~GD_SB;
		}
	} else if (ty > NBR_NORMAL) {
		fl = GD_SA | GD_SB | GD_WB | GD_SLOW; // harmless addresses; the value comes from gamma_entry32
	}
	d.flags = fl;
}
template <bool PROLONG> struct SideGamma32 {
	double a0, a1, b0, b1;
	// AX: face-normal axis; entry m = lo + 32 hi lies over cell (lo >> s) * A + (hi >> s) * B of the parent's plane
	template <int AX>
	__device__ __forceinline__ void issue(const GDesc32 &d, int m, int lo, int hi, const double *__restrict__ F, const double *__restrict__ uc)
	{
		constexpr int A = (AX == 0) ? 32 : 1, B = (AX == 2) ? 32 : 1024;
		const uint4   o = *reinterpret_cast<const uint4 *>(&d);
		a0 = __ldg(F + o.x + m);
		b0 = __ldg(F + o.y + m);
		a1 = b1 = 0.0;
		if (PROLONG) {
			const int fl = d.flags, sa = fl & GD_SA, sb = (fl >> 1) & 1;
			a1 = __ldg(uc + o.z + ((lo >> sa) * A + (hi >> sa) * B));
			b1 = __ldg(uc + o.w + ((lo >> sb) * A + (hi >> sb) * B));
		}
	}
	// the value of a side without the GD_SLOW flag
	__device__ __forceinline__ double combine(const GDesc32 &d) const
	{
		return d.c * (0.5 * (a0 + a1) + 0.5 * (b0 + ((d.flags & GD_WB) ? b1 : 0.0)));
	}
	__device__ __forceinline__ double finish(const GDesc32 &d, const PatchMeta *__restrict__ meta, int p, int s, int m, const double *__restrict__ F,
	                                         const double *__restrict__ uc) const
	{
		double g = combine(d);
		if (d.flags & GD_SLOW) g = d.c * gamma_entry32<PROLONG>(meta, p, s, m, F, uc);
		return g;
	}
};

// ---------------------------------------------------------------------------------------------
// iface_rhs32_kernel: the interface part of the right-hand side of a 32^3 sweep that does not start from zero.
//   A block-Jacobi sweep solves S u = f - b on each patch, b = (2/h^2) E^T gamma: non-zero on boundary cells only and a sum
//   of six face terms.  The patch solve is linear, so each face term can enter smooth3d32c_kernel where it is uniform over the
//   sweep's threads: the y faces before the y transform (as they are), the x faces at x = 0 / 31 of the rows of the x
//   transform (transformed along y), the z faces at elimination step 0 (transformed along y, then x - the sweep's order).
//   This kernel forms those terms in the face shape G[slot][1024] (slots: IfaceSlots32 below):
//     s = 0, 1 (x faces): Dst2_y(c(., z))[k_y]       at k_y + 32 z
//     s = 2, 3 (y faces): c(x, z)                    at x + 32 z
//     s = 4, 5 (z faces): Dst2_x(Dst2_y(c))[k_x, k_y] at k_x + 32 k_y
//   with c = (2/h^2) gamma from the gathers of GDesc32 / SideGamma32 (gamma_entry32 on sides with coarse / fine neighbours),
//   so the values of c are those the sweep subtracted when it gathered them itself; only where they enter moved.
//   One warp per slot, the warps of a CTA independent of each other, a padded 32 x 33 tile per warp for the transposes.  On
//   several GPUs this kernel is the consumer of the halo hand-over of the first post-sweep (halo_push / halo_wait_warp /
//   halo_finish, as face_residual_restrict_big_kernel): the sweep after it reads no face data.
// ---------------------------------------------------------------------------------------------
constexpr int    IR32_THREADS = 192, IR32_WARPS = IR32_THREADS / 32, IR32_CTAS_PER_SM = 2, IR32_TP = 33;
constexpr size_t iface_rhs32_smem_bytes() { return sizeof(double) * IR32_WARPS * 32 * IR32_TP; }

// Interface slots of a 32^3 level: where G holds the term of each patch side.  Two same-level neighbours p, q see the same
// term on their common interface: c = 2/h^2 is the same for both, the gather of p's side s loads the four values of q's side
// s ^ 1 with the halves swapped (c (0.5 (a0 + a1) + 0.5 (b0 + b1)), the sum is commutative), and x, y and z terms use the same
// layout on both sides.  Such an interface gets one slot, gathered for the lower patch index (its owner), when
//   - p's side s is NBR_NORMAL to q != p and q's side s ^ 1 is NBR_NORMAL back to p,
//   - both are owned (index < P: no halo neighbour, so GD_WB stays set on both sides), neither has Neumann sides and both
//     have the same h.
// Every other side with a neighbour (coarse / fine / halo / not mutual) has a slot of its own; domain-boundary sides (the term
// is zero) and patches with Neumann sides (smooth3d32n_kernel gathers for itself) have none.  Slots are numbered in the
// order of their owner, so the patches [p0, p1) own the slots [begin[p0], begin[p1]); with the lower index as owner, a launch
// over [p0, p1) after one over [0, p0) (interior patches first, then the ones with halo neighbours) reads only slots written
// by itself or before.
struct IfaceSlots32 {
	std::vector<int32_t> gslot; // [P][6]: slot of side s of patch p, -1: no term
	std::vector<int32_t> owner; // [nslots]: 6 p + s of the side whose gather produces the slot
	std::vector<int32_t> begin; // [P + 1]
};
inline bool iface_shared32(const PatchMeta *meta, int P, int p, int s)
{
	const PatchMeta &a = meta[p];
	if (a.neumann || a.nbr_type[s] != NBR_NORMAL) return false;
	const int q = a.nbr_idx[s][0];
	if (q == p || q < 0 || q >= P) return false;
	const PatchMeta &b = meta[q];
	return !b.neumann && b.nbr_type[s ^ 1] == NBR_NORMAL && b.nbr_idx[s ^ 1][0] == p && a.inv_h2 == b.inv_h2;
}
inline IfaceSlots32 build_iface_slots32(const PatchMeta *meta, int P)
{
	IfaceSlots32 t;
	t.gslot.assign((size_t) P * 6, -1);
	t.begin.resize((size_t) P + 1);
	for (int p = 0; p < P; p++) {
		t.begin[p] = (int32_t) t.owner.size();
		if (meta[p].neumann) continue;
		for (int s = 0; s < 6; s++) {
			if (meta[p].nbr_type[s] == NBR_NONE) continue;
			const bool shared = iface_shared32(meta, P, p, s);
			const int  q      = meta[p].nbr_idx[s][0];
			if (shared && q < p) continue; // q's slot, set when q was visited
			const int32_t k = (int32_t) t.owner.size();
			t.owner.push_back(p * 6 + s);
			t.gslot[(size_t) p * 6 + s] = k;
			if (shared) t.gslot[(size_t) q * 6 + (s ^ 1)] = k;
		}
	}
	t.begin[P] = (int32_t) t.owner.size();
	return t;
}
// c of side s of patch p: entry m = lane + 32 i to out[i * stride + lane]; AX = face-normal axis.  Sides with coarse / fine
// neighbours go entry by entry through the out-of-line gamma_entry32 (SideGamma32::finish); the others keep IR32_BATCH entries'
// loads in flight per lane and need no call, so that no in-flight load is held across one.
constexpr int IR32_BATCH = 16;
template <bool PROLONG, int AX>
__device__ __forceinline__ void side_gamma32(const GDesc32 &d, const PatchMeta *__restrict__ meta, int p, int s, int lane, const double *__restrict__ F,
                                             const double *__restrict__ uc, double *out, int stride)
{
	if (d.flags & GD_SLOW) { // warp-uniform
#pragma unroll 1
		for (int i = 0; i < 32; i++) {
			SideGamma32<PROLONG> sg;
			sg.template issue<AX>(d, lane + 32 * i, lane, i, F, uc);
			out[i * stride + lane] = sg.finish(d, meta, p, s, lane + 32 * i, F, uc);
		}
		return;
	}
	constexpr int B = IR32_BATCH;
#pragma unroll
	for (int i0 = 0; i0 < 32; i0 += B) {
		SideGamma32<PROLONG> sg[B];
#pragma unroll
		for (int j = 0; j < B; j++) sg[j].template issue<AX>(d, lane + 32 * (i0 + j), lane, i0 + j, F, uc);
#pragma unroll
		for (int j = 0; j < B; j++) out[(i0 + j) * stride + lane] = sg[j].combine(d);
	}
}
// slots [k0, k1) of owner (6 p + s, IfaceSlots32::owner) into G[k]
template <bool PROLONG, bool HALO>
__global__ void __launch_bounds__(IR32_THREADS, IR32_CTAS_PER_SM)
iface_rhs32_kernel(const PatchMeta *__restrict__ meta, const int32_t *__restrict__ owner, int k0, int k1, const double *__restrict__ Fin,
                   const double *__restrict__ uc, double *__restrict__ Gout, HaloSync hs = HaloSync{})
{
	constexpr int N = 32, M = N * N, TP = IR32_TP;
	extern __shared__ __align__(16) double T[]; // [IR32_WARPS][32][TP]
	__shared__ GPatch32 GD[IR32_WARPS];         // GD[w].d[s]: written and read by warp w only
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	double *  tw   = T + w * N * TP;
	Mags<N>   mg;
	mg.load();
	pdl_launch_dependents();
	pdl_wait();
	if (HALO) halo_push<3, 32>(hs, meta);
	bool halo_ok = false;
	for (int k = k0 + blockIdx.x * IR32_WARPS + w; k < k1; k += gridDim.x * IR32_WARPS) {
		const int ps = __ldg(owner + k), p = ps / 6, s = ps - 6 * p;
		if (HALO) halo_wait_warp(hs, p, halo_ok);
		if (lane == 0) make_gdesc32<PROLONG>(meta[p], p, s, GD[w]);
		__syncwarp();
		const GDesc32 &d  = GD[w].d[s];
		double *       Gp = Gout + (size_t) k * M;
		double         v[N];
		if (s < 2) { // x faces: entry (y, z) = (lane, i) -> tile row z; transform along y, pencil z = lane
			side_gamma32<PROLONG, 0>(d, meta, p, s, lane, Fin, uc, tw, TP);
			__syncwarp();
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = tw[lane * TP + k];
			Dst2<N, N>::run(v, mg);
#pragma unroll
			for (int k = 0; k < N; k++) tw[lane * TP + k] = v[k];
			__syncwarp();
#pragma unroll
			for (int i = 0; i < N; i++) Gp[lane + N * i] = tw[i * TP + lane];
		} else if (s < 4) { // y faces: entry (x, z) = (lane, i), as they are
			side_gamma32<PROLONG, 1>(d, meta, p, s, lane, Fin, uc, Gp, N);
		} else { // z faces: entry (x, y) = (lane, i) -> tile row y; transform along y (pencil x = lane), then along x (pencil k_y = lane)
			side_gamma32<PROLONG, 2>(d, meta, p, s, lane, Fin, uc, tw, TP);
			__syncwarp();
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = tw[k * TP + lane];
			Dst2<N, N>::run(v, mg);
#pragma unroll
			for (int k = 0; k < N; k++) tw[k * TP + lane] = v[k];
			__syncwarp();
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = tw[lane * TP + k];
			Dst2<N, N>::run(v, mg);
#pragma unroll
			for (int k = 0; k < N; k++) tw[lane * TP + k] = v[k];
			__syncwarp();
#pragma unroll
			for (int i = 0; i < N; i++) Gp[lane + N * i] = tw[i * TP + lane];
		}
		__syncwarp(); // GD[w] and the tile are rewritten for the next slot
	}
	if (HALO) halo_finish(hs);
}

// Sweeps that do not start from zero take the interface part of the right-hand side from G (iface_rhs32_kernel, launched
// right before over the same patches or, for slots owned by a lower patch, earlier): up to six coalesced loads per thread and
// patch, G[gslot[p][s]], issued with the loads of f; sides without a slot (domain boundary) load and subtract nothing.
template <bool ZERO_GUESS, bool EMIT, bool WRITE_U>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(C32_THREADS, 1)
smooth3d32c_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ f, double *__restrict__ u,
                   const double *__restrict__ G, double *__restrict__ Fout, const double *__restrict__ tri, int skip_neumann = 0,
                   const int32_t *__restrict__ gslot = nullptr)
{
	// skip_neumann != 0: patches with Neumann domain sides are left to smooth3d32n_kernel (launched over the same range
	// with only_neumann); both CTAs of the cluster skip together
	constexpr int N = 32, ROW = C32_ROW, PL = C32_PL, M = N * N, NC = N * N * N;
	extern __shared__ __align__(16) double S[];
	double *       X    = S + C32_TILE;  // [2][M] last eliminated plane, for the peer
	double *       FV   = X + 2 * M;     // [32][C32_FV] faces-only sweeps from a zero guess: partially transformed face
	                                     // vectors, entry j of vector i at j * C32_FV + i
	double *       EX   = FV + (ZERO_GUESS ? 1024 + 16 * 128 : 0); // [16 warps][2][32] staging of the new x-face slices
	const int      t = threadIdx.x, lane = t & 31, w = t >> 5;
	const unsigned rank = cluster_ctarank();
	const int      z    = rank == 0 ? w : N - 1 - w; // plane of the patch behind local plane w
	const int      sz   = rank == 0 ? 4 : 5;         // the z side this half touches
	const int      ncl = gridDim.x / 2, npatch = P - p0;
	const int      mf   = lane + N * z; // x faces: entry (y, z) = (lane, z); y faces: entry (x, z) = (lane, z)
	Mags<N>        mg;
	mg.load();
	pdl_launch_dependents();
	pdl_wait();
	int g = blockIdx.x / 2;
	for (int it = 0; g < npatch; g += ncl, it++) {
		const int    p    = p0 + g;
		const bool   next = g + ncl < npatch;
		const int    pn   = p + ncl;
		const double h2   = meta[p].h2;
		const double *tp  = tri + (size_t) meta[p].tab * (17 * M); // the patch's multiplier table [17][M] (TriSolve)
		double       v[N];
		if (skip_neumann && meta[p].neumann) { // cluster-uniform: this patch belongs to the general path
			cluster_sync_all(); // keeps the pair in step: the exchange planes alternate by iteration parity
			continue;
		}
		// interface terms (see iface_rhs32_kernel): y faces of pencil (x, z) = (lane, z), x faces of row (k_y, z) = (lane, z),
		// this half's z face at pencils (k_x, k_y) = (lane, w), (lane, w + 16)
		double gy0 = 0.0, gy1 = 0.0, gx0 = 0.0, gx1 = 0.0, gz0 = 0.0, gz1 = 0.0;
		if (!ZERO_GUESS) { // slot conditions are uniform over the cluster
			const int2 *gs = reinterpret_cast<const int2 *>(gslot + (size_t) p * 6);
			const int2  kx = __ldg(gs), ky = __ldg(gs + 1), kz = __ldg(gs + 2);
			const int   ks = rank == 0 ? kz.x : kz.y;
			if (ky.x >= 0) gy0 = __ldcs(G + (size_t) ky.x * M + mf);
			if (ky.y >= 0) gy1 = __ldcs(G + (size_t) ky.y * M + mf);
			if (kx.x >= 0) gx0 = __ldcs(G + (size_t) kx.x * M + mf);
			if (kx.y >= 0) gx1 = __ldcs(G + (size_t) kx.y * M + mf);
			if (ks >= 0) {
				gz0 = __ldcs(G + (size_t) ks * M + lane + N * w);
				gz1 = __ldcs(G + (size_t) ks * M + lane + N * (w + 16));
			}
		}
		{ // y forward: pencil (x, z) = (lane, z), straight from memory
			const double *fp = f + (size_t) p * NC + (size_t) z * M + lane;
#pragma unroll
			for (int k = 0; k < N; k++) v[k] = __ldcs(fp + k * N);
			if (next) { // the same plane of the next patch -> L2 (64 lines), and what this warp reads of its G (12 lines)
				const double *fn = f + (size_t) pn * NC + (size_t) z * M + lane * 32;
				prefetch_l2(fn);
				prefetch_l2(fn + 16);
				if (!ZERO_GUESS && lane < 12) {
					const int kn = __ldg(gslot + (size_t) pn * 6 + (lane < 8 ? lane >> 1 : sz));
					if (kn >= 0) {
						const double *Gn = G + (size_t) kn * M + 16 * (lane & 1);
						prefetch_l2(lane < 8 ? Gn + N * z : Gn + N * (w + 16 * ((lane >> 1) & 1)));
					}
				}
			}
			if (!ZERO_GUESS) {
				v[0] -= gy0;
				v[N - 1] -= gy1;
			}
			Dst2<N, N>::run(v, mg);
			double *col = S + w * PL + lane;
#pragma unroll
			for (int k = 0; k < N; k++) col[k * ROW] = v[k];
		}
		__syncwarp();
		double2 *rowp = reinterpret_cast<double2 *>(S + w * PL + lane * ROW); // row (k_y, plane) = (lane, w)
		{ // x forward
#pragma unroll
			for (int j = 0; j < N / 2; j++) {
				const double2 d = rowp[j];
				v[2 * j]        = d.x;
				v[2 * j + 1]    = d.y;
			}
			if (!ZERO_GUESS) {
				v[0] -= gx0;
				v[N - 1] -= gx1;
			}
			Dst2<N, N>::run(v, mg);
#pragma unroll
			for (int j = 0; j < N / 2; j++) rowp[j] = make_double2(v[2 * j], v[2 * j + 1]);
		}
		__syncthreads();
		// z: elimination step j on local plane j, in place; pencils (k_x, k_y) = (lane, w) and (lane, w + 16)
		const double hsc = h2 * (4.0 / (N * N));
		double *     Xo = X + (it & 1) * M;
#pragma unroll
		for (int q = 0; q < 2; q++) {
			const int     ky = w + 16 * q;
			const double *zp = S + ky * ROW + lane;
			const double *tb = tp + ky * N + lane;
			double        rho = 0.0;
#pragma unroll
			for (int j = 0; j < 16; j++) {
				const double a = __ldg(tb + j * M);
				const double x = (!ZERO_GUESS && j == 0) ? zp[0] - (q ? gz1 : gz0) : zp[j * PL]; // this half's z face
				const double r = x * (hsc * a);
				rho            = (j == 0) ? r : fma(-a, rho, r);
				const_cast<double *>(zp)[j * PL] = rho;
			}
			Xo[ky * N + lane] = rho;
		}
		cluster_sync_all(); // both halves are eliminated; the peer's last plane is readable
#pragma unroll
		for (int q = 0; q < 2; q++) {
			const int     ky = w + 16 * q;
			double *      zp = S + ky * ROW + lane;
			const double *tb = tp + ky * N + lane;
			const double  a15 = __ldg(tb + 15 * M), kap = __ldg(tb + 16 * M);
			double        y   = kap * fma(-a15, ld_dsmem(Xo + ky * N + lane, rank ^ 1), zp[15 * PL]);
			zp[15 * PL]       = y;
#pragma unroll
			for (int j = 14; j >= 0; j--) {
				y          = fma(-__ldg(tb + j * M), y, zp[j * PL]);
				zp[j * PL] = y;
			}
		}
		__syncthreads();
		// faces-only sweeps from a zero guess: dot products + 60 one-dimensional transforms instead of full inverse transforms
		constexpr bool FACE_TAIL = ZERO_GUESS && !WRITE_U;
		if (!FACE_TAIL || w == 0) {
			// full inverse transforms: every plane of a sweep that writes u; in a faces-only sweep only the plane that is
			// this half's z face (local plane 0)
			{ // x inverse
#pragma unroll
				for (int j = 0; j < N / 2; j++) {
					const double2 d = rowp[j];
					v[2 * j]        = d.x;
					v[2 * j + 1]    = d.y;
				}
				Dst3<N, N>::run(v, mg);
#pragma unroll
				for (int j = 0; j < N / 2; j++) rowp[j] = make_double2(v[2 * j], v[2 * j + 1]);
			}
			__syncwarp();
			{ // y inverse: pencil (x, z) = (lane, z), straight to memory
				const double *col = S + w * PL + lane;
#pragma unroll
				for (int k = 0; k < N; k++) v[k] = col[k * ROW];
				Dst3<N, N>::run(v, mg);
				if (WRITE_U) {
					double *up = u + (size_t) p * NC + (size_t) z * M + lane;
#pragma unroll
					for (int k = 0; k < N; k++) __stcs(up + k * N, v[k]);
				}
				if (EMIT) {
					double *Fp = Fout + (size_t) p * 6 * M;
					Fp[2 * M + mf] = v[0]; // y faces: entry (x, z)
					Fp[3 * M + mf] = v[N - 1];
					if (w == 0) { // z face of this half: entries (x, y)
						double *Fz = Fp + sz * M + lane;
#pragma unroll
						for (int k = 0; k < N; k++) Fz[N * k] = v[k];
					}
					double *ex = EX + w * 64;
					if (lane == 0 || lane == N - 1) { // x faces: entries (y, z), held by lanes 0 and 31
						double *q = ex + (lane ? 32 : 0);
#pragma unroll
						for (int k = 0; k < N; k++) q[k] = v[k];
					}
					__syncwarp();
					Fp[0 * M + mf] = ex[lane];
					Fp[1 * M + mf] = ex[32 + lane];
				}
			}
		} else {
			// Faces-only sweep, planes other than the z face: only u(0 | 31, y, z) and u(x, 0 | 31, z) are wanted.  With
			// T = the DST-III matrix (DftPatchSolver.h:269-281), T[0][j] = sin(pi (j+1) / 2n), T[0][n-1] = 1/2 and
			// T[n-1][j] = (-1)^j T[0][j], contract the axis normal to the face first - two dot products per row / column of
			// the plane instead of a transform - and leave the 4 x 15 remaining 1-D transforms of the CTA to two warps.
			double E = 0.0, O = 0.0;
#pragma unroll
			for (int j = 0; j < N / 2; j++) { // row (k_y, plane) = (lane, w): contract k_x
				const double2 d = rowp[j];
				E               = fma(mg.sinq(2 * j + 1), d.x, E);
				O               = fma((2 * j + 1 == N - 1) ? 0.5 : mg.sinq(2 * j + 2), d.y, O);
			}
			const int vi = 4 * (w - 1); // vectors 4 (w - 1) + {0: x = 0, 1: x = 31, 2: y = 0, 3: y = 31}, entry index = lane
			FV[lane * C32_FV + vi]     = E + O;
			FV[lane * C32_FV + vi + 1] = E - O;
			const double *col = S + w * PL + lane; // column (k_x, plane) = (lane, w): contract k_y
			E = O = 0.0;
#pragma unroll
			for (int k = 0; k < N; k += 2) {
				E = fma(mg.sinq(k + 1), col[k * ROW], E);
				O = fma((k + 1 == N - 1) ? 0.5 : mg.sinq(k + 2), col[(k + 1) * ROW], O);
			}
			FV[lane * C32_FV + vi + 2] = E + O;
			FV[lane * C32_FV + vi + 3] = E - O;
		}
		if (FACE_TAIL) {
			__syncthreads();
			const int vec = (w - 1) * 32 + lane; // warps 1 and 2: one face vector per lane
			if ((w == 1 || w == 2) && vec < 60) {
#pragma unroll
				for (int j = 0; j < N; j++) v[j] = FV[j * C32_FV + vec];
				Dst3<N, N>::run(v, mg);
				const int lp = 1 + (vec >> 2), kind = vec & 3;             // local plane, which face
				const int zz = rank == 0 ? lp : N - 1 - lp;
				double *  Fq = Fout + (size_t) p * 6 * M + kind * M + N * zz; // x faces: entries (y, z); y faces: entries (x, z)
#pragma unroll
				for (int j = 0; j < N / 2; j++) *reinterpret_cast<double2 *>(Fq + 2 * j) = make_double2(v[2 * j], v[2 * j + 1]);
			}
		}
		__syncwarp();
	}
	cluster_sync_all(); // a CTA must not exit while its peer may still read its exchange plane
}

// ---------------------------------------------------------------------------------------------
// smooth3d32n_kernel: 32^3 levels that contain patches with Neumann domain sides (PatchSolvers/FftwPatchSolver.h:
// 115-127,197; DftPatchSolver.h:115-127,150-165).  General path, same arithmetic as the Neumann branch of
// smooth_kernel: per axis the transform pair and eigenvalues follow the two closures (axis_kind), dense 32 x 32
// transforms with the matrices of DftPatchSolver.h:237-289 (mats), eigenvalue sums formed on the fly (lam), zero mode
// removed on an all-Neumann patch.  One CTA per patch, the patch lives in a CTA-private 256 KB block of `scratch`
// (L2-resident: the block is reused for every patch of the CTA); the variant switches are run-time arguments.
// Correctness path, not a fast one: 6 x 1024 multiply-adds per cell.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TGPU_THREADS)
smooth3d32n_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ f, double *__restrict__ u,
                   const double *__restrict__ Fin, double *__restrict__ Fout, const double *__restrict__ uc,
                   const double *__restrict__ mats, const double *__restrict__ lam, double *__restrict__ scratch, int zero_guess,
                   int emit, int prolong, int write_u, double lam_shift, int only_neumann = 0, int helm = 0)
{
	// only_neumann != 0: only patches with Neumann domain sides are swept (the others of the range belong to
	// smooth3d32c_kernel, skip_neumann)
	constexpr int N = 32, M = N * N, NC = M * N;
	const int     t = threadIdx.x;
	double *      W = scratch + (size_t) blockIdx.x * NC;
	Mags<N>       mg;
	mg.load();
	pdl_launch_dependents();
	pdl_wait();
	for (int g = blockIdx.x; g < P - p0; g += gridDim.x) {
		const int        p    = p0 + g;
		const PatchMeta &pm   = meta[p];
		const int        neu  = pm.neumann;
		if (only_neumann && !neu) continue; // CTA-uniform
		const double     cfac = 2.0 * pm.inv_h2, h2 = pm.h2;
		for (int i = t; i < NC; i += TGPU_THREADS) W[i] = __ldg(f + (size_t) p * NC + i);
		__syncthreads();
		if (!zero_guess) { // f - (2/h^2) E^T gamma, side by side (edge cells belong to several sides)
			for (int s = 0; s < 6; s++) {
				if (pm.nbr_type[s] != NBR_NONE) {
					for (int m = t; m < M; m += TGPU_THREADS) {
						const double gm = prolong ? gamma_entry32<true>(meta, p, s, m, Fin, uc) : gamma_entry32<false>(meta, p, s, m, Fin, uc);
						int          c[3];
						face_cell<3, N>(s, m, c);
						W[(c[2] * N + c[1]) * N + c[0]] -= cfac * gm;
					}
				}
				__syncthreads();
			}
		}
		double v[N];
		// forward along z, y, x; then inverse along x, y, z (pass 2 also divides by the eigenvalue sums first)
		for (int pass = 0; pass < 6; pass++) {
			const int      axis = pass < 3 ? 2 - pass : pass - 3;
			const AxisKind ak   = axis_kind(neu, axis);
				const int      step = axis == 0 ? 1 : (axis == 1 ? N : M);
			if (pass == 3) {
				const AxisKind kx = axis_kind(neu, 0), ky = axis_kind(neu, 1), kz = axis_kind(neu, 2);
				const double   scale = h2 * (2.0 / N) * (2.0 / N) * (2.0 / N);
				const bool     singular = neu == 63 && !helm; // (helm: a Helmholtz operator, the zero mode is solved for)
				for (int i = t; i < NC; i += TGPU_THREADS) {
					const double sum = __ldg(lam + kx.lam * N + i % N) + (__ldg(lam + ky.lam * N + (i / N) % N) + __ldg(lam + kz.lam * N + i / M)) + lam_shift * h2;
					W[i]             = (singular && i == 0) ? 0.0 : W[i] * scale / sum;
				}
				__syncthreads();
			}
			for (int q = t; q < M; q += TGPU_THREADS) {
				const int base = axis == 0 ? q * N : (axis == 1 ? (q % N) + (q / N) * M : q);
#pragma unroll
				for (int j = 0; j < N; j++) v[j] = W[base + j * step];
				// fast forms for DST-II / III and DST-IV / DCT-IV, the dense matrix for DCT-II / III (kernels.cuh)
				general_transform<N>(mats, pass < 3 ? ak.fwd : ak.inv, v, W + base, step, mg);
			}
			__syncthreads();
		}
		if (write_u)
			for (int i = t; i < NC; i += TGPU_THREADS) u[(size_t) p * NC + i] = W[i];
		if (emit)
			for (int i = t; i < 6 * M; i += TGPU_THREADS) {
				int c[3];
				face_cell<3, N>(i / M, i % M, c);
				Fout[(size_t) p * 6 * M + i] = W[(c[2] * N + c[1]) * N + c[0]];
			}
		__syncthreads(); // the block is refilled next
	}
}

// ---------------------------------------------------------------------------------------------
// residual + restriction from face data for patches whose face (M entries) is larger than the block
// (see face_residual_restrict_kernel for the identity used); one patch per CTA, R[6][M] in dynamic smem
// ---------------------------------------------------------------------------------------------
// one patch, general form (any neighbour types, patches present on both levels); R = [S][M] staging in shared memory;
// every thread of the CTA calls; ends with a barrier
template <int D, int N, bool DIFF>
__device__ __forceinline__ void frr_big_patch(const PatchMeta *__restrict__ meta, int p, double *R, const double *__restrict__ Fnew,
                                              const double *__restrict__ Fold, double *__restrict__ coarse)
{
	using G         = Geo<D, N>;
	constexpr int H = N / 2, M = G::M;
	const int        t      = threadIdx.x;
	const PatchMeta &pm     = meta[p];
	const int        orth   = pm.orth_on_parent;
	const double     cfac   = 2.0 * pm.inv_h2;
	double *         dst    = coarse + (size_t) pm.parent_idx * G::NC;
	const FaceVals<D, N, DIFF ? FV_DIFF : FV_NEG> fv{Fnew, Fold, meta};
	for (int i = t; i < G::S * M; i += TGPU_THREADS) {
		const int s = i / M, m = i % M;
		R[i]        = cfac * gamma_entry(pm, p, s, m, fv);
	}
	__syncthreads();
	auto Rp = [&](int s, int m) { return R[s * M + m]; };
	if (orth < 0) { // patch present on both levels: coarse = r (dense, zero in the interior)
		for (int c = t; c < G::NC; c += TGPU_THREADS) {
			const int x = c % N, y = (c / N) % N, k = (D == 2) ? 0 : c / (N * N);
			double    v = 0.0;
			if (D == 2) {
				if (x == 0) v += Rp(0, y);
				if (x == N - 1) v += Rp(1, y);
				if (y == 0) v += Rp(2, x);
				if (y == N - 1) v += Rp(3, x);
			} else {
				if (x == 0) v += Rp(0, y + N * k);
				if (x == N - 1) v += Rp(1, y + N * k);
				if (y == 0) v += Rp(2, x + N * k);
				if (y == N - 1) v += Rp(3, x + N * k);
				if (k == 0) v += Rp(4, x + N * y);
				if (k == N - 1) v += Rp(5, x + N * y);
			}
			dst[c] = v;
		}
	} else {
		const int     ox = (orth & 1) * H, oy = ((orth >> 1) & 1) * H, oz = (D == 2) ? 0 : ((orth >> 2) & 1) * H;
		constexpr int CC = G::NC >> D;
		for (int c = t; c < CC; c += TGPU_THREADS) {
			const int X = c % H, Y = (c / H) % H, Z = (D == 2) ? 0 : c / (H * H);
			double    v = 0.0;
			if (D == 2) {
				auto blk = [&](int s, int I) { return (Rp(s, 2 * I) + Rp(s, 2 * I + 1)) / 4.0; };
				if (X == 0) v += blk(0, Y);
				if (X == H - 1) v += blk(1, Y);
				if (Y == 0) v += blk(2, X);
				if (Y == H - 1) v += blk(3, X);
				dst[(Y + oy) * N + (X + ox)] = v;
			} else {
				auto blk = [&](int s, int I, int J) {
					const int b = 2 * I + N * 2 * J;
					return ((Rp(s, b) + Rp(s, b + 1)) + (Rp(s, b + N) + Rp(s, b + N + 1))) / 8.0;
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
	__syncthreads();
}
template <int D, int N, bool DIFF, bool HALO = false>
__global__ void __launch_bounds__(TGPU_THREADS)
face_residual_restrict_big_kernel(const PatchMeta *__restrict__ meta, int p0, int P, const double *__restrict__ Fnew,
                                  const double *__restrict__ Fold, double *__restrict__ coarse, HaloSync hs = HaloSync{})
{
	using G = Geo<D, N>;
	extern __shared__ __align__(16) double R[]; // [S][M]
	const int t = threadIdx.x;
	pdl_launch_dependents();
	pdl_wait();
	if (HALO) halo_push<D, N>(hs, meta);
	bool halo_ok = false;
	for (int g = blockIdx.x; g < P - p0; g += gridDim.x) {
		const int p = p0 + g;
		if (HALO) halo_wait_cta(hs, p, halo_ok);
		if (D == 3 && N == 32) {
			// Refined patches whose six sides have same-level neighbours (or none) - every patch of a uniform level - take a
			// leaner path, like face_residual_restrict16_kernel: one thread per COARSE face entry (6 x 256 per patch) loads
			// its 2 x 2 block of the patch's and the neighbour's slices with four 128-bit loads and stores the block
			// average; the 16^3 coarse cells under the patch are then assembled two per thread and stored as double2.
			// Same expressions and summation order as frr_big_patch.
			const PatchMeta &pm   = meta[p];
			bool             fast = pm.orth_on_parent >= 0;
#pragma unroll
			for (int s = 0; s < 6; s++) fast = fast && pm.nbr_type[s] <= NBR_NORMAL;
			if (fast) { // CTA-uniform
				const double cfac = 2.0 * pm.inv_h2;
				double *     Rc   = R; // [6][256]
#pragma unroll
				for (int k = 0; k < 6; k++) {
					const int e = t + TGPU_THREADS * k, s = k, c = t, m0 = 2 * (c & 15) + 64 * (c >> 4);
					double    val = 0.0;
					if (pm.nbr_type[s] == NBR_NORMAL) {
						const size_t oa = ((size_t) p * 6 + s) * 1024 + m0, ob = ((size_t) pm.nbr_idx[s][0] * 6 + (s ^ 1)) * 1024 + m0;
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
						const double2 a0 = ld(oa), a1 = ld(oa + 32), b0 = ld(ob), b1 = ld(ob + 32);
						const double  r00 = cfac * (0.5 * a0.x + 0.5 * b0.x), r01 = cfac * (0.5 * a0.y + 0.5 * b0.y);
						const double  r10 = cfac * (0.5 * a1.x + 0.5 * b1.x), r11 = cfac * (0.5 * a1.y + 0.5 * b1.y);
						val               = ((r00 + r01) + (r10 + r11)) / 8.0;
					}
					Rc[e] = val;
				}
				__syncthreads();
				const int orth = pm.orth_on_parent;
				const int ox = (orth & 1) * 16, oy = ((orth >> 1) & 1) * 16, oz = ((orth >> 2) & 1) * 16;
				double *  dst = coarse + (size_t) pm.parent_idx * G::NC;
#pragma unroll
				for (int k = 0; k < 8; k++) {
					const int q = t + TGPU_THREADS * k;                          // pair index: cells (X, Y, Z), (X + 1, Y, Z)
					const int X = (q & 7) * 2, Y = (q >> 3) & 15, Z = q >> 7;
					double    v[2];
#pragma unroll
					for (int i = 0; i < 2; i++) {
						const int x = X + i;
						double    a = 0.0;
						if (x == 0) a += Rc[0 * 256 + Y + 16 * Z];
						if (x == 15) a += Rc[1 * 256 + Y + 16 * Z];
						if (Y == 0) a += Rc[2 * 256 + x + 16 * Z];
						if (Y == 15) a += Rc[3 * 256 + x + 16 * Z];
						if (Z == 0) a += Rc[4 * 256 + x + 16 * Y];
						if (Z == 15) a += Rc[5 * 256 + x + 16 * Y];
						v[i] = a;
					}
					*reinterpret_cast<double2 *>(dst + ((Z + oz) * 32 + (Y + oy)) * 32 + (X + ox)) = make_double2(v[0], v[1]);
				}
				__syncthreads();
				continue;
			}
		}
		frr_big_patch<D, N, DIFF>(meta, p, R, Fnew, Fold, coarse);
	}
	if (HALO) halo_finish(hs);
}
} // namespace tgpu
