// tools/smooth_bench.cu - stand-alone timing harness for the D = 3, n = 16 kernels (development aid, not part
// of the product).  Builds the neighbour table of a uniform G^3 grid of patches with parents on a (G/2)^3
// grid, fills the vectors with noise and times each kernel variant with CUDA events.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -I pressurepoissonsolver_b200/csrc \
//        tools/smooth_bench.cu -o tools/smooth_bench && tools/smooth_bench [G=16] [reps=20]
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include "kernels.cuh"
using namespace tgpu;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)

static std::vector<PatchMeta> build_meta(int G)
{
	std::vector<PatchMeta> m((size_t) G * G * G);
	auto id  = [&](int x, int y, int z) { return (z * G + y) * G + x; };
	auto pid = [&](int x, int y, int z) { return ((z / 2) * (G / 2) + (y / 2)) * (G / 2) + (x / 2); };
	const double h = 1.0 / (G * 16);
	for (int z = 0; z < G; z++)
		for (int y = 0; y < G; y++)
			for (int x = 0; x < G; x++) {
				PatchMeta &pm     = m[id(x, y, z)];
				pm                = PatchMeta{};
				pm.inv_h2         = 1.0 / (h * h);
				pm.h2             = h * h;
				pm.parent_idx     = G > 1 ? pid(x, y, z) : 0;
				pm.orth_on_parent = G > 1 ? ((x & 1) | ((y & 1) << 1) | ((z & 1) << 2)) : -1;
				const int c[3]    = {x, y, z};
				for (int s = 0; s < 6; s++) {
					int n[3] = {x, y, z};
					n[s >> 1] += (s & 1) ? 1 : -1;
					const bool in = n[s >> 1] >= 0 && n[s >> 1] < G;
					pm.nbr_type[s] = in ? NBR_NORMAL : NBR_NONE;
					for (int q = 0; q < 4; q++) pm.nbr_idx[s][q] = in ? id(n[0], n[1], n[2]) : 0;
					pm.nbr_parent[s] = in && G > 1 ? pid(n[0], n[1], n[2]) : 0;
					pm.nbr_orth[s]   = in && G > 1 ? ((n[0] & 1) | ((n[1] & 1) << 1) | ((n[2] & 1) << 2)) : -1;
					(void) c;
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
	printf("%-34s %8.2f us   %7.1f GB/s (algorithmic)\n", name, ms * 1e3, bytes / ms / 1e6);
	return ms;
}

int main(int argc, char **argv)
{
	const int G = argc > 1 ? atoi(argv[1]) : 16, reps = argc > 2 ? atoi(argv[2]) : 20;
	const int P = G * G * G, Pc = std::max(1, P / 8);
	const size_t nc = (size_t) P * 4096, ncc = (size_t) Pc * 4096, nf = (size_t) P * 6 * 256;
	std::vector<PatchMeta> hm = build_meta(G);
	PatchMeta *meta;
	CK(cudaMalloc(&meta, hm.size() * sizeof(PatchMeta)));
	CK(cudaMemcpy(meta, hm.data(), hm.size() * sizeof(PatchMeta), cudaMemcpyHostToDevice));
	double *f, *u, *uc, *Fa, *Fb, *tri, *coarse;
	CK(cudaMalloc(&f, nc * 8)); CK(cudaMalloc(&u, nc * 8)); CK(cudaMalloc(&uc, ncc * 8)); CK(cudaMalloc(&coarse, ncc * 8));
	CK(cudaMalloc(&Fa, nf * 8)); CK(cudaMalloc(&Fb, nf * 8)); CK(cudaMalloc(&tri, 4096 * 8));
	{
		std::vector<double> h(nc);
		for (size_t i = 0; i < nc; i++) h[i] = (double) rand() / RAND_MAX - 0.5;
		CK(cudaMemcpy(f, h.data(), nc * 8, cudaMemcpyHostToDevice));
		CK(cudaMemcpy(uc, h.data(), ncc * 8, cudaMemcpyHostToDevice));
		CK(cudaMemcpy(Fa, h.data(), nf * 8, cudaMemcpyHostToDevice));
		std::vector<double> e(4096);
		for (int i = 0; i < 4096; i++) e[i] = -1.0 / (1 + i % 7);
		CK(cudaMemcpy(tri, e.data(), 4096 * 8, cudaMemcpyHostToDevice));
		std::vector<double> mag(17);
		for (int i = 0; i <= 16; i++) mag[i] = sin(M_PI / 32.0 * i);
		CK(cudaMemcpyToSymbol(c_mag16, mag.data(), 17 * 8));
	}
	int sms = 148;
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
	const size_t sm = smooth3d16_smem_bytes();
	auto attr = [&](auto k) { CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sm)); };
	attr(smooth3d16_kernel<true, true, false, false>);
	attr(smooth3d16_kernel<true, false, false, true>);
	attr(smooth3d16_kernel<false, false, true, true>);
	attr(smooth3d16_kernel<false, false, false, true>);
	attr(smooth3d16_kernel<false, true, false, false>);
	const int grid = std::min(P, sms * s16_ctas_per_sm(false));
	const dim3 blk(S16_BLOCK);
	printf("G=%d P=%d cells=%zu grid=%d\n", G, P, nc, grid);
	const double b16 = 16.0 * nc;
	const int    gridz = std::min(P, sms * s16_ctas_per_sm(true));
	time_it("zero_guess faces-only", reps, b16, [&] { smooth3d16_kernel<true, true, false, false><<<gridz, blk, sm>>>(meta, 0, P, f, u, Fa, Fb, tri, uc); });
	time_it("zero_guess write_u", reps, b16, [&] { smooth3d16_kernel<true, false, false, true><<<gridz, blk, sm>>>(meta, 0, P, f, u, Fa, Fb, tri, uc); });
	time_it("plain gamma write_u", reps, b16, [&] { smooth3d16_kernel<false, false, false, true><<<grid, blk, sm>>>(meta, 0, P, f, u, Fa, Fb, tri, uc); });
	time_it("plain gamma faces-only", reps, b16, [&] { smooth3d16_kernel<false, true, false, false><<<grid, blk, sm>>>(meta, 0, P, f, u, Fa, Fb, tri, uc); });
	if (G > 1) time_it("prolong gamma write_u", reps, b16, [&] { smooth3d16_kernel<false, false, true, true><<<grid, blk, sm>>>(meta, 0, P, f, u, Fa, Fb, tri, uc); });
	if (G > 1) time_it("face_residual_restrict", reps, b16, [&] { face_residual_restrict_kernel<3, 16, false><<<std::min(P, sms * 8), 256>>>(meta, 0, P, Fa, nullptr, coarse); });
	if (G > 1) {
		double *coarse2;
		CK(cudaMalloc(&coarse2, ncc * 8));
		time_it("face_residual_restrict16", reps, b16, [&] { face_residual_restrict16_kernel<false><<<std::min(P, sms * 8), 256>>>(meta, 0, P, Fa, nullptr, coarse2); });
		std::vector<double> a(ncc), b(ncc);
		CK(cudaMemcpy(a.data(), coarse, ncc * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(b.data(), coarse2, ncc * 8, cudaMemcpyDeviceToHost));
		size_t bad = 0;
		for (size_t i = 0; i < ncc; i++) bad += a[i] != b[i];
		printf("   coarse right-hand side: %zu of %zu entries differ\n", bad, ncc);
	}
	CK(cudaGetLastError());
	return 0;
}
