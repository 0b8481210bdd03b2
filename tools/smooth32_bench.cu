// tools/smooth32_bench.cu - stand-alone timing harness for the D = 3, n = 32 smoother (development aid, not part of the
// product): the cluster-pair kernel (smooth3d32c_kernel) and the interface terms of the sweeps that do not start from zero
// (iface_rhs32_kernel) on a uniform G^3 grid of patches with parents on a (G/2)^3 grid and random data.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -I pressurepoissonsolver_b200/csrc \
//        tools/smooth32_bench.cu -o tools/smooth32_bench && tools/smooth32_bench [G=8] [reps=10]
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <algorithm>
#include "kernels.cuh"
using namespace tgpu;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)
constexpr int N = 32, NC = N * N * N, M = N * N;

// LOCAL != 0 (experiment): every neighbour is the patch itself and every parent is coarse patch 0, so that the gathered
// interface data comes from lines the kernel has just touched / from one L2-resident patch: separates the instruction and
// latency cost of the gathers from their memory traffic
static int LOCAL = 0;
static std::vector<PatchMeta> build_meta(int G)
{
	std::vector<PatchMeta> m((size_t) G * G * G);
	auto id  = [&](int x, int y, int z) { return (z * G + y) * G + x; };
	auto pid = [&](int x, int y, int z) { return ((z / 2) * (G / 2) + (y / 2)) * (G / 2) + (x / 2); };
	const double h = 1.0 / (G * N);
	for (int z = 0; z < G; z++)
		for (int y = 0; y < G; y++)
			for (int x = 0; x < G; x++) {
				PatchMeta &pm     = m[id(x, y, z)];
				pm                = PatchMeta{};
				pm.inv_h2         = 1.0 / (h * h);
				pm.h2             = h * h;
				pm.parent_idx     = G > 1 ? (LOCAL ? 0 : pid(x, y, z)) : 0;
				pm.orth_on_parent = G > 1 ? ((x & 1) | ((y & 1) << 1) | ((z & 1) << 2)) : -1;
				for (int s = 0; s < 6; s++) {
					int n[3] = {x, y, z};
					n[s >> 1] += (s & 1) ? 1 : -1;
					const bool in = n[s >> 1] >= 0 && n[s >> 1] < G;
					pm.nbr_type[s] = in ? NBR_NORMAL : NBR_NONE;
					for (int q = 0; q < 4; q++) pm.nbr_idx[s][q] = in ? (LOCAL ? id(x, y, z) : id(n[0], n[1], n[2])) : 0;
					pm.nbr_parent[s] = in && G > 1 ? (LOCAL ? 0 : pid(n[0], n[1], n[2])) : 0;
					pm.nbr_orth[s]   = in && G > 1 ? ((n[0] & 1) | ((n[1] & 1) << 1) | ((n[2] & 1) << 2)) : -1;
				}
			}
	return m;
}
template <typename F> static float time_it(const char *name, int reps, double bytes, F launch)
{
	cudaEvent_t e0, e1;
	cudaEventCreate(&e0), cudaEventCreate(&e1);
	for (int i = 0; i < 3; i++) launch();
	CK(cudaDeviceSynchronize());
	cudaEventRecord(e0);
	for (int i = 0; i < reps; i++) launch();
	cudaEventRecord(e1);
	CK(cudaDeviceSynchronize());
	float ms;
	cudaEventElapsedTime(&ms, e0, e1);
	ms /= reps;
	printf("%-52s %8.2f us   %7.1f GB/s (algorithmic)\n", name, ms * 1e3, bytes / ms / 1e6);
	return ms;
}

int main(int argc, char **argv)
{
	const int G = argc > 1 ? atoi(argv[1]) : 8, reps = argc > 2 ? atoi(argv[2]) : 10;
	LOCAL = argc > 3 ? atoi(argv[3]) : 0;
	const int P = G * G * G, Pc = std::max(1, P / 8);
	const size_t nc = (size_t) P * NC, ncc = (size_t) Pc * NC, nf = (size_t) P * 6 * M;
	std::vector<PatchMeta> hm = build_meta(G);
	PatchMeta *meta;
	CK(cudaMalloc(&meta, hm.size() * sizeof(PatchMeta)));
	CK(cudaMemcpy(meta, hm.data(), hm.size() * sizeof(PatchMeta), cudaMemcpyHostToDevice));
	double *f, *u, *uc, *Fa, *Fb, *tri;
	CK(cudaMalloc(&f, nc * 8)); CK(cudaMalloc(&u, nc * 8)); CK(cudaMalloc(&uc, ncc * 8));
	CK(cudaMalloc(&Fa, nf * 8)); CK(cudaMalloc(&Fb, nf * 8)); CK(cudaMalloc(&tri, 17 * M * 8));
	int sms = 148;
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
	{
		std::vector<double> h(nc);
		for (size_t i = 0; i < nc; i++) h[i] = (double) rand() / RAND_MAX - 0.5;
		CK(cudaMemcpy(f, h.data(), nc * 8, cudaMemcpyHostToDevice));
		CK(cudaMemcpy(uc, h.data() + 7, ncc * 8, cudaMemcpyHostToDevice));
		CK(cudaMemcpy(Fa, h.data() + 13, nf * 8, cudaMemcpyHostToDevice));
		std::vector<double> tb(17 * M);
		for (int m = 0; m < M; m++) {
			auto lam = [&](int k) { const long double s = sinl((k + 1) * 3.141592653589793238462643383279502884L / 64); return -4.0L * s * s; };
			const long double mu = lam(m % N) + lam(m / N);
			long double       a  = 0;
			for (int j = 0; j < 16; j++) {
				a = 1.0L / (mu - (j == 0 ? 3.0L : 2.0L) - (j == 0 ? 0.0L : a));
				tb[(size_t) j * M + m] = (double) a;
			}
			tb[(size_t) 16 * M + m] = (double) (1.0L / (1.0L - a * a));
		}
		CK(cudaMemcpy(tri, tb.data(), tb.size() * 8, cudaMemcpyHostToDevice));
		std::vector<double> mag(33);
		for (int i = 0; i <= 32; i++) mag[i] = sin(M_PI / 64.0 * i);
		CK(cudaMemcpyToSymbol(c_mag32, mag.data(), 33 * 8));
	}
	const size_t smZ = smooth3d32c_smem_bytes<true>(), smC = smooth3d32c_smem_bytes<false>(), smI = iface_rhs32_smem_bytes();
	const int    gridC = 2 * std::min(P, sms / 2);
	printf("G=%d P=%d cells=%zu cluster grid=%d smem %zu / %zu (zero guess / not), iface_rhs32 smem %zu\n", G, P, nc, gridC, smZ, smC, smI);
	const double b16 = 16.0 * nc;
	// interface slots: the library's table (one term per same-level interface, none on domain-boundary sides) and, for
	// comparison, one slot per side with a neighbour
	const IfaceSlots32 ts = build_iface_slots32(hm.data(), P);
	IfaceSlots32       tu;
	tu.gslot.assign((size_t) P * 6, -1);
	for (int p = 0; p < P; p++)
		for (int s = 0; s < 6; s++)
			if (hm[p].nbr_type[s] != NBR_NONE) tu.gslot[(size_t) p * 6 + s] = (int32_t) tu.owner.size(), tu.owner.push_back(p * 6 + s);
	const int nsh = (int) ts.owner.size(), nun = (int) tu.owner.size();
	printf("interface slots: %d shared, %d one per side (%d sides)\n", nsh, nun, 6 * P);
	int32_t *gslot_s, *gslot_u, *own_s, *own_u;
	CK(cudaMalloc(&gslot_s, ts.gslot.size() * 4)); CK(cudaMalloc(&gslot_u, tu.gslot.size() * 4));
	CK(cudaMalloc(&own_s, std::max(nsh, 1) * 4)); CK(cudaMalloc(&own_u, std::max(nun, 1) * 4));
	CK(cudaMemcpy(gslot_s, ts.gslot.data(), ts.gslot.size() * 4, cudaMemcpyHostToDevice));
	CK(cudaMemcpy(gslot_u, tu.gslot.data(), tu.gslot.size() * 4, cudaMemcpyHostToDevice));
	CK(cudaMemcpy(own_s, ts.owner.data(), nsh * 4, cudaMemcpyHostToDevice));
	CK(cudaMemcpy(own_u, tu.owner.data(), nun * 4, cudaMemcpyHostToDevice));
	double *Gv;
	CK(cudaMalloc(&Gv, std::max<size_t>(nun, 1) * M * 8));
	CK(cudaFuncSetAttribute(iface_rhs32_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smI));
	CK(cudaFuncSetAttribute(iface_rhs32_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smI));
	bool          shared = true; // which table iface() and the sweeps use
	const int32_t *gslot = gslot_s;
	auto iface = [&](bool prolong) {
		const int      n     = shared ? nsh : nun;
		const int32_t *own   = shared ? own_s : own_u;
		const int      gridI = std::max(1, std::min((n + IR32_WARPS - 1) / IR32_WARPS, sms * IR32_CTAS_PER_SM));
		if (prolong) iface_rhs32_kernel<true, false><<<gridI, IR32_THREADS, smI>>>(meta, own, 0, n, Fa, uc, Gv);
		else iface_rhs32_kernel<false, false><<<gridI, IR32_THREADS, smI>>>(meta, own, 0, n, Fa, uc, Gv);
	};
#define VARIANT(NAME, Z, E, W, PRE)                                                                                              \
	{                                                                                                                            \
		const size_t sm_ = smooth3d32c_smem_bytes<Z>();                                                                          \
		CK(cudaFuncSetAttribute(smooth3d32c_kernel<Z, E, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sm_));            \
		CK(cudaMemset(u, 0, nc * 8)); CK(cudaMemset(Fb, 0, nf * 8));                                                             \
		time_it(NAME, reps, b16, [&] { PRE; smooth3d32c_kernel<Z, E, W><<<gridC, C32_THREADS, sm_>>>(meta, 0, P, f, u, Gv, Fb, tri, 0, gslot); }); \
		CK(cudaGetLastError());                                                                                                  \
	}
	VARIANT("zero_guess faces-only", true, true, false, )
	VARIANT("zero_guess write_u", true, false, true, )
	VARIANT("zero_guess write_u+faces", true, true, true, )
	// sweeps that do not start from zero: the interface terms (iface_rhs32_kernel) alone, the sweep alone (reading the terms
	// left by the previous launch), and the two back to back as the library launches them; with the shared slots, then with
	// one slot per side
	for (int sh = 1; sh >= 0; sh--) {
		shared = sh != 0;
		gslot  = shared ? gslot_s : gslot_u;
		const char *tag = shared ? "[shared]  " : "[per side]";
		char        name[96];
		const double bi = 8.0 * M * (shared ? nsh : nun);
		snprintf(name, sizeof name, "%s iface_rhs32 plain", tag);
		time_it(name, reps, bi, [&] { iface(false); });
		snprintf(name, sizeof name, "%s sweep write_u+faces", tag);
		VARIANT(name, false, true, true, )
		snprintf(name, sizeof name, "%s iface_rhs32 plain + sweep write_u+faces", tag);
		VARIANT(name, false, true, true, iface(false))
		if (G > 1) {
			snprintf(name, sizeof name, "%s iface_rhs32 prolong", tag);
			time_it(name, reps, bi, [&] { iface(true); });
			snprintf(name, sizeof name, "%s sweep write_u", tag);
			VARIANT(name, false, false, true, )
			snprintf(name, sizeof name, "%s iface_rhs32 prolong + sweep write_u", tag);
			VARIANT(name, false, false, true, iface(true))
		}
	}
	return 0;
}
