// apps/steady.cpp - the GMG path of the reference's apps/3d/steady.cpp / apps/2d/steady.cpp
// (mesh load, --divide, manufactured trig RHS, BiCGStab with a GMG cycle as right preconditioner,
// error / residual report, apps/3d/steady.cpp:211-215,292-322,453-567) written against the
// mirrored plugin surface in include/tgpu_plugin.hpp.  Every numerical step runs on the GPU.
//
// usage: steady D mesh.bin divide n [--cycle V|W] [--plugin] [--pre k] [--post k] [--mid k] [--coarse k] [--max-levels k]
//               [--patches-per-proc x] [--lambda x] [--out u.bin] [--neumann] [--problem trig|gauss]
//               [--solver bicgstab|gmg] [--tol x]
//   --solver gmg  stationary multigrid (GMGSolve, one cycle per iteration) to ||f - A u|| <= tol ||f|| (--tol, default
//                 1e-10) from u = 0, instead of BiCGStab preconditioned by the cycle (tolerance 1e-12, relative to r0)
//   --max-levels / --patches-per-proc   GMG::CycleOpts (GMG/CycleOpts.h:55,59, honoured as in GMG/CycleFactory3d.cpp:101-104)
//   --lambda  the patch solver's shift (FftwPatchSolver(domain, lambda), PatchSolvers/FftwPatchSolver.h:66)
//   --neumann Neumann domain boundaries (ThundereggDomGen(..., neumann = true), Init::initNeumann, right-hand-side mean
//             removed as in apps/3d/steady.cpp:301,316-334; 3D); --problem gauss: the app's second manufactured problem
//   --plugin  drive the cycle through the virtual Level/Smoother/Operator/Restrictor/Interpolator
//             objects (one ABI call per step, like the reference) instead of the fused tgpu_vcycle
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>

#include "tgpu_plugin.hpp"

template <size_t D> static int run(int argc, char **argv)
{
	using namespace tgpu;
	const std::string mesh_file = argv[2];
	const int         divide = atoi(argv[3]), n = atoi(argv[4]);
	GMG::CycleOpts    copts;
	bool              plugin = false, neumann = false;
	double            lambda = 0.0;
	std::string       out, problem = "trig", solver = "bicgstab";
	double            tol = 1e-10;
	for (int a = 5; a < argc; a++) {
		if (!strcmp(argv[a], "--cycle") && a + 1 < argc) copts.cycle_type = argv[++a];
		else if (!strcmp(argv[a], "--pre") && a + 1 < argc) copts.pre_sweeps = atoi(argv[++a]);
		else if (!strcmp(argv[a], "--post") && a + 1 < argc) copts.post_sweeps = atoi(argv[++a]);
		else if (!strcmp(argv[a], "--mid") && a + 1 < argc) copts.mid_sweeps = atoi(argv[++a]);
		else if (!strcmp(argv[a], "--coarse") && a + 1 < argc) copts.coarse_sweeps = atoi(argv[++a]);
		else if (!strcmp(argv[a], "--max-levels") && a + 1 < argc) copts.max_levels = atoi(argv[++a]);
		else if (!strcmp(argv[a], "--patches-per-proc") && a + 1 < argc) copts.patches_per_proc = atof(argv[++a]);
		else if (!strcmp(argv[a], "--lambda") && a + 1 < argc) lambda = atof(argv[++a]);
		else if (!strcmp(argv[a], "--plugin")) plugin = true;
		else if (!strcmp(argv[a], "--neumann")) neumann = true;
		else if (!strcmp(argv[a], "--problem") && a + 1 < argc) problem = argv[++a];
		else if (!strcmp(argv[a], "--out") && a + 1 < argc) out = argv[++a];
		else if (!strcmp(argv[a], "--solver") && a + 1 < argc) solver = argv[++a];
		else if (!strcmp(argv[a], "--tol") && a + 1 < argc) tol = atof(argv[++a]);
	}
	if (solver != "bicgstab" && solver != "gmg") throw Error(TGPU_ERR_ARG, "unknown solver " + solver);
	auto ctx = std::make_shared<Context>(0);
	Mesh mesh(mesh_file, (int) D);
	for (int i = 0; i < divide; i++) mesh.refineLeaves();
	if (neumann) mesh.setNeumann(true);
	auto h = std::make_shared<Hierarchy>(ctx, mesh, n);
	if (lambda != 0.0) check(tgpu_hierarchy_set_lambda(h->p, lambda));

	std::shared_ptr<VectorGenerator<D>> vg(new DeviceVG<D>(h, 0));
	auto u = vg->getNewVector(), exact = vg->getNewVector(), f = vg->getNewVector(), au = vg->getNewVector();
	if (neumann) {
		check(tgpu_init_neumann_rhs(h->p, problem == "gauss" ? 1 : 0, DeviceVector<D>::raw(f), DeviceVector<D>::raw(exact)));
		double integral = 0, volume = 1;
		check(tgpu_vec_integrate(h->p, DeviceVector<D>::raw(f), &integral, &volume));
		std::cout << "Fdiff: " << integral / volume << "\n";
		f->shift(-integral / volume);
	} else {
		check(tgpu_init_trig_rhs(h->p, DeviceVector<D>::raw(f), DeviceVector<D>::raw(exact)));
	}

	std::shared_ptr<Operator<D>> A(new DeviceOperator<D>(h, 0));
	std::shared_ptr<Operator<D>> M;
	if (plugin) M = GMG::CycleFactory<D>::getCycle(copts, h);
	else M = GMG::CycleFactory<D>::getFusedCycle(copts, h);

	ctx->sync();
	auto t0  = std::chrono::steady_clock::now();
	int  its = solver == "gmg" ? GMGSolve<D>::solve(M, u, f, tol) : BiCGStab<D>::solve(vg, A, u, f, M);
	ctx->sync();
	double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();

	A->apply(u, au);
	auto resid = vg->getNewVector(), error = vg->getNewVector();
	resid->addScaled(-1, au, 1, f);
	error->addScaled(-1, exact, 1, u);
	if (neumann) { // the solution is determined up to a constant (apps/3d/steady.cpp:539-548 shifts the error by the difference of the two averages)
		double ie = 0, vol = 1;
		check(tgpu_vec_integrate(h->p, DeviceVector<D>::raw(error), &ie, &vol));
		error->shift(-ie / vol);
	}
	std::cout.precision(13);
	std::cout << "Iterations: " << its << "\n";
	std::cout << "Error (2-norm):   " << error->twoNorm() / exact->twoNorm() << "\n";
	std::cout << "Error (inf-norm): " << error->infNorm() << "\n";
	std::cout << "Residual: " << resid->twoNorm() / f->twoNorm() << "\n";
	std::cout << "Number of cells: " << h->numCells(0) << "  patches: " << h->numPatches(0) << "  levels: " << h->nlevels << "\n";
	std::cout << "Linear Solve time (s): " << sec << "\n";
	if (!out.empty()) {
		std::vector<double> host((size_t) h->numCells(0));
		std::dynamic_pointer_cast<DeviceVector<D>>(u)->download(host.data());
		std::ofstream o(out, std::ios::binary);
		o.write((const char *) host.data(), host.size() * 8);
	}
	return 0;
}

int main(int argc, char **argv)
{
	if (argc < 5) {
		std::cerr << "usage: steady D mesh.bin divide n [--cycle V|W] [--plugin] [--pre k] [--post k] [--mid k] [--coarse k] [--max-levels k] "
		             "[--patches-per-proc x] [--lambda x] [--out u.bin] [--neumann] [--problem trig|gauss] [--solver bicgstab|gmg] [--tol x]\n";
		return 2;
	}
	try {
		return atoi(argv[1]) == 2 ? run<2>(argc, argv) : run<3>(argc, argv);
	} catch (const tgpu::Error &e) {
		std::cerr << "tgpu error " << e.code << ": " << e.what() << "\n";
		return 1;
	}
}
