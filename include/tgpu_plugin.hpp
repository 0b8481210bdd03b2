// tgpu_plugin.hpp - C++ host side above the C ABI (tgpu.h), mirroring ThunderEgg's GMG plugin
// surface class for class so that code written against the reference's interfaces (BiCGStab,
// apps/*/steady.cpp, GMG::Cycle) can drive the B200 kernels unchanged apart from the namespace.
// Interfaces and thin delegates only: no algorithm of the reference is restated here.  The adaptors that derive from the
// reference's OWN headers (so that its unmodified GMG::VCycle / WCycle / BiCGStab templates run on the GPU) are in
// include/tgpu_thunderegg.hpp.
//
//   reference (src/Thunderegg/...)                         here (namespace tgpu)
//   Vector<D>                     Vector.h:179-322         Vector<D>  (same virtual ops)  -> DeviceVector<D>
//   VectorGenerator<D>            Vector.h:323-327         VectorGenerator<D>             -> DeviceVG<D>
//   Operator<D>                   Operators/Operator.h:37  Operator<D>                    -> DeviceOperator<D>
//   GMG::Smoother<D>              GMG/Smoother.h:39        GMG::Smoother<D>               -> DeviceSmoother<D>, DeviceJacobiSmoother<D>
//   GMG::Restrictor<D>            GMG/Restrictor.h:39-40   GMG::Restrictor<D>             -> DeviceRestrictor<D>
//   GMG::Interpolator<D>          GMG/Interpolator.h:39-40 GMG::Interpolator<D>           -> DeviceInterpolator<D>
//   GMG::Cycle/VCycle/WCycle<D>   GMG/Cycle.h, VCycle.h, WCycle.h   GMG::FusedCycle<D> (one tgpu_vcycle call: fused schedule with
//                                                          CUDA-graph replay, or the reference's call-by-call sequence)
//   GMG::CycleOpts                GMG/CycleOpts.h:51-80    GMG::CycleOpts
//   GMG::CycleFactory{2,3}d       GMG/CycleFactory3d.cpp:69-134     GMG::CycleFactory<D>::getCycle
//   BiCGStab<D>::solve            BiCGStab.h:45-106        BiCGStab<D>::solve (same signature; delegates to tgpu_bicgstab)
//   (no reference counterpart)                             GMGSolve<D>::solve (stationary multigrid from a guess, tgpu_gmg_solve)
//   Tree<D> + ThundereggDomGen<D> OctTree.h, ThundereggDomGen.h     Mesh, Hierarchy (RAII over tgpu_mesh / tgpu_hier)
//
// Error behaviour: the reference throws an int (`throw 3;`) on type mismatches
// (SchurHelper.h:129, GMG/InterLevelComm.h:175); here every non-zero ABI return code becomes a
// tgpu::Error (std::runtime_error) carrying tgpu_last_error().
#pragma once
#include <cmath>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "tgpu.h"

namespace tgpu
{
struct Error : std::runtime_error {
	int code;
	Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};
inline void check(int rc)
{
	if (rc != TGPU_OK) throw Error(rc, tgpu_last_error());
}

class Context
{
	public:
	tgpu_ctx *p = nullptr;
	explicit Context(int device = 0) { check(tgpu_init(device, &p)); }
	~Context() { tgpu_finalize(p); }
	Context(const Context &) = delete;
	Context &operator=(const Context &) = delete;
	void     sync() { check(tgpu_sync(p)); }
};

class Mesh
{
	public:
	tgpu_mesh *p = nullptr;
	Mesh(const std::string &file, int D) { check(tgpu_mesh_load(file.c_str(), D, &p)); }
	Mesh(int D, int num_levels) { check(tgpu_mesh_uniform(D, num_levels, &p)); }
	~Mesh() { tgpu_mesh_destroy(p); }
	Mesh(const Mesh &) = delete;
	Mesh &operator=(const Mesh &) = delete;
	void  refineLeaves() { check(tgpu_mesh_refine_leaves(p)); }
	/* ThundereggDomGen(tree, ns, neumann = true) (ThundereggDomGen.h:92): Neumann conditions on the domain boundary */
	void  setNeumann(bool on = true) { check(tgpu_mesh_set_neumann(p, on ? 1 : 0)); }
};

// the device-resident level hierarchy = what the reference's DomainGenerator + CycleFactory produce
class Hierarchy
{
	public:
	tgpu_hier *             p = nullptr;
	std::shared_ptr<Context> ctx;
	int                     D = 0, n = 0, nlevels = 0;
	Hierarchy(std::shared_ptr<Context> ctx, Mesh &mesh, int n) : ctx(ctx), n(n)
	{
		const TgpuLevelDesc *descs = nullptr;
		int                  num_nodes;
		check(tgpu_mesh_info(mesh.p, &D, nullptr, &num_nodes));
		check(tgpu_mesh_extract_levels(mesh.p, n, &nlevels, &descs));
		check(tgpu_hierarchy_create(ctx->p, D, n, nlevels, descs, &p));
	}
	// for callers that already hold Domain/PatchInfo metadata (the drop-in path)
	Hierarchy(std::shared_ptr<Context> ctx, int D, int n, const std::vector<TgpuLevelDesc> &levels)
	: ctx(ctx), D(D), n(n), nlevels((int) levels.size())
	{
		check(tgpu_hierarchy_create(ctx->p, D, n, nlevels, levels.data(), &p));
	}
	~Hierarchy() { tgpu_hierarchy_destroy(p); }
	Hierarchy(const Hierarchy &) = delete;
	Hierarchy &operator=(const Hierarchy &) = delete;
	long long  numCells(int level = 0) const
	{
		int64_t np, nc;
		check(tgpu_level_npatch(p, level, &np, &nc));
		return nc;
	}
	long long numPatches(int level = 0) const
	{
		int64_t np, nc;
		check(tgpu_level_npatch(p, level, &np, &nc));
		return np;
	}
};

// ---- Vector<D>: every op virtual, as in Vector.h:186-321 ----
template <size_t D> class Vector
{
	public:
	virtual ~Vector() {}
	virtual void   set(double alpha)                                                                              = 0;
	virtual void   scale(double alpha)                                                                            = 0;
	virtual void   shift(double delta)                                                                            = 0;
	virtual void   copy(std::shared_ptr<const Vector<D>> b)                                                       = 0;
	virtual void   add(std::shared_ptr<const Vector<D>> b)                                                        = 0;
	virtual void   addScaled(double alpha, std::shared_ptr<const Vector<D>> b)                                    = 0;
	virtual void   addScaled(double alpha, std::shared_ptr<const Vector<D>> a, double beta,
	                         std::shared_ptr<const Vector<D>> b)                                                  = 0;
	virtual void   scaleThenAdd(double alpha, std::shared_ptr<const Vector<D>> b)                                 = 0;
	virtual void   scaleThenAddScaled(double alpha, double beta, std::shared_ptr<const Vector<D>> b)              = 0;
	virtual void   scaleThenAddScaled(double alpha, double beta, std::shared_ptr<const Vector<D>> b, double gamma,
	                                  std::shared_ptr<const Vector<D>> c)                                         = 0;
	virtual double twoNorm() const                                                                                = 0;
	virtual double infNorm() const                                                                                = 0;
	virtual double dot(std::shared_ptr<const Vector<D>> b) const                                                  = 0;
};

template <size_t D> class DeviceVector : public Vector<D>
{
	public:
	tgpu_vec *                 v = nullptr;
	std::shared_ptr<Hierarchy> h;
	int                        level;
	DeviceVector(std::shared_ptr<Hierarchy> h, int level) : h(h), level(level) { check(tgpu_vec_create(h->p, level, &v)); }
	~DeviceVector() { tgpu_vec_destroy(v); }
	static const tgpu_vec *raw(const std::shared_ptr<const Vector<D>> &b)
	{
		auto d = dynamic_cast<const DeviceVector<D> *>(b.get());
		if (d == nullptr) throw Error(TGPU_ERR_ARG, "vector is not a tgpu::DeviceVector"); // reference: throw 3
		return d->v;
	}
	static tgpu_vec *raw(const std::shared_ptr<Vector<D>> &b)
	{
		auto d = dynamic_cast<DeviceVector<D> *>(b.get());
		if (d == nullptr) throw Error(TGPU_ERR_ARG, "vector is not a tgpu::DeviceVector");
		return d->v;
	}
	void upload(const double *host) { check(tgpu_vec_upload(v, host)); }
	void download(double *host) const { check(tgpu_vec_download(v, host)); }
	void set(double a) override { check(tgpu_vec_set(v, a)); }
	void scale(double a) override { check(tgpu_vec_scale(v, a)); }
	void shift(double d) override { check(tgpu_vec_shift(v, d)); }
	void copy(std::shared_ptr<const Vector<D>> b) override { check(tgpu_vec_copy(v, raw(b))); }
	void add(std::shared_ptr<const Vector<D>> b) override { check(tgpu_vec_add(v, raw(b))); }
	void addScaled(double a, std::shared_ptr<const Vector<D>> b) override { check(tgpu_vec_add_scaled(v, a, raw(b))); }
	void addScaled(double a, std::shared_ptr<const Vector<D>> x, double b, std::shared_ptr<const Vector<D>> y) override
	{
		check(tgpu_vec_add_scaled2(v, a, raw(x), b, raw(y)));
	}
	void scaleThenAdd(double a, std::shared_ptr<const Vector<D>> b) override { check(tgpu_vec_scale_then_add(v, a, raw(b))); }
	void scaleThenAddScaled(double a, double b, std::shared_ptr<const Vector<D>> x) override
	{
		check(tgpu_vec_scale_then_add_scaled(v, a, b, raw(x)));
	}
	void scaleThenAddScaled(double a, double b, std::shared_ptr<const Vector<D>> x, double g,
	                        std::shared_ptr<const Vector<D>> y) override
	{
		check(tgpu_vec_scale_then_add_scaled2(v, a, b, raw(x), g, raw(y)));
	}
	double twoNorm() const override
	{
		double r;
		check(tgpu_vec_two_norm(v, &r));
		return r;
	}
	double infNorm() const override
	{
		double r;
		check(tgpu_vec_inf_norm(v, &r));
		return r;
	}
	double dot(std::shared_ptr<const Vector<D>> b) const override
	{
		double r;
		check(tgpu_vec_dot(v, raw(b), &r));
		return r;
	}
};

template <size_t D> class VectorGenerator
{
	public:
	virtual ~VectorGenerator() {}
	virtual std::shared_ptr<Vector<D>> getNewVector() = 0;
};
template <size_t D> class DeviceVG : public VectorGenerator<D>
{
	std::shared_ptr<Hierarchy> h;
	int                        level;

	public:
	DeviceVG(std::shared_ptr<Hierarchy> h, int level) : h(h), level(level) {}
	std::shared_ptr<Vector<D>> getNewVector() override { return std::make_shared<DeviceVector<D>>(h, level); }
};

template <size_t D> class Operator
{
	public:
	virtual ~Operator() {}
	virtual void apply(std::shared_ptr<const Vector<D>> x, std::shared_ptr<Vector<D>> b) const = 0;
};
// SchurDomainOp / DomainWrapOp (Operators/SchurDomainOp.h:51-54): b = A x on one level
template <size_t D> class DeviceOperator : public Operator<D>
{
	public:
	std::shared_ptr<Hierarchy> h;
	int                        level;
	DeviceOperator(std::shared_ptr<Hierarchy> h, int level) : h(h), level(level) {}
	void apply(std::shared_ptr<const Vector<D>> x, std::shared_ptr<Vector<D>> b) const override
	{
		check(tgpu_apply(h->p, level, DeviceVector<D>::raw(x), DeviceVector<D>::raw(b)));
	}
};

namespace GMG
{
struct CycleOpts { // GMG/CycleOpts.h:51-80
	int         max_levels       = 0;
	double      patches_per_proc = 0;
	int         pre_sweeps       = 1;
	int         post_sweeps      = 1;
	int         mid_sweeps       = 1;
	int         coarse_sweeps    = 1;
	std::string cycle_type       = "V";
};
template <size_t D> class Smoother
{
	public:
	virtual ~Smoother() {}
	virtual void smooth(std::shared_ptr<const Vector<D>> f, std::shared_ptr<Vector<D>> u) const = 0;
};
template <size_t D> class Restrictor
{
	public:
	virtual ~Restrictor() {}
	virtual void restrict(std::shared_ptr<Vector<D>> coarse, std::shared_ptr<const Vector<D>> fine) const = 0;
};
template <size_t D> class Interpolator
{
	public:
	virtual ~Interpolator() {}
	virtual void interpolate(std::shared_ptr<const Vector<D>> coarse, std::shared_ptr<Vector<D>> fine) const = 0;
};
// FFTBlockJacobiSmoother (GMG/FFTBlockJacobiSmoother.h:55-58)
template <size_t D> class DeviceSmoother : public Smoother<D>
{
	std::shared_ptr<Hierarchy> h;
	int                        level;

	public:
	DeviceSmoother(std::shared_ptr<Hierarchy> h, int level) : h(h), level(level) {}
	void smooth(std::shared_ptr<const Vector<D>> f, std::shared_ptr<Vector<D>> u) const override
	{
		check(tgpu_smooth(h->p, level, DeviceVector<D>::raw(f), DeviceVector<D>::raw(u)));
	}
};
// the north star's weighted-Jacobi option (no reference counterpart)
template <size_t D> class DeviceJacobiSmoother : public Smoother<D>
{
	std::shared_ptr<Hierarchy> h;
	int                        level;
	double                     omega;

	public:
	DeviceJacobiSmoother(std::shared_ptr<Hierarchy> h, int level, double omega) : h(h), level(level), omega(omega) {}
	void smooth(std::shared_ptr<const Vector<D>> f, std::shared_ptr<Vector<D>> u) const override
	{
		check(tgpu_smooth_jacobi(h->p, level, DeviceVector<D>::raw(f), DeviceVector<D>::raw(u), omega));
	}
};
// AvgRstr (GMG/AvgRstr.h:78-113)
template <size_t D> class DeviceRestrictor : public Restrictor<D>
{
	std::shared_ptr<Hierarchy> h;
	int                        fine_level;

	public:
	DeviceRestrictor(std::shared_ptr<Hierarchy> h, int fine_level) : h(h), fine_level(fine_level) {}
	void restrict(std::shared_ptr<Vector<D>> coarse, std::shared_ptr<const Vector<D>> fine) const override
	{
		check(tgpu_restrict(h->p, fine_level, DeviceVector<D>::raw(fine), DeviceVector<D>::raw(coarse)));
	}
};
// DrctIntp (GMG/DrctIntp.h:80-113): fine += P coarse
template <size_t D> class DeviceInterpolator : public Interpolator<D>
{
	std::shared_ptr<Hierarchy> h;
	int                        fine_level;

	public:
	DeviceInterpolator(std::shared_ptr<Hierarchy> h, int fine_level) : h(h), fine_level(fine_level) {}
	void interpolate(std::shared_ptr<const Vector<D>> coarse, std::shared_ptr<Vector<D>> fine) const override
	{
		check(tgpu_prolong_add(h->p, fine_level, DeviceVector<D>::raw(coarse), DeviceVector<D>::raw(fine)));
	}
};

// GMG::Cycle<D> (GMG/Cycle.h:34,116-126, with VCycle.h:44-62 / WCycle.h:45-68) as ONE ABI call.  `granular = false`: the fused
// kernel schedule with CUDA-graph replay; `granular = true`: the library replays the reference's sequence call by call
// (zero fill, smooth, residual, restrict, ... one kernel launch per plugin call of the reference: TgpuCycleOpts.fused = 0).
// The host recursion over Level objects itself is not restated here: where the reference's own GMG::VCycle / WCycle
// classes should drive the kernels, include/tgpu_thunderegg.hpp derives adaptors from the reference's real headers.
template <size_t D> class FusedCycle : public Operator<D>
{
	public:
	std::shared_ptr<Hierarchy> h;
	TgpuCycleOpts              o;
	FusedCycle(std::shared_ptr<Hierarchy> h, const CycleOpts &opts, bool granular = false) : h(h)
	{
		tgpu_cycle_opts_default(&o);
		o.max_levels       = opts.max_levels;
		o.patches_per_proc = opts.patches_per_proc;
		o.pre_sweeps       = opts.pre_sweeps;
		o.post_sweeps      = opts.post_sweeps;
		o.mid_sweeps       = opts.mid_sweeps;
		o.coarse_sweeps    = opts.coarse_sweeps;
		if (granular) o.fused = 0;
		if (opts.cycle_type == "V") o.cycle_type = 0;
		else if (opts.cycle_type == "W") o.cycle_type = 1;
		else throw Error(TGPU_ERR_ARG, "unknown cycle type " + opts.cycle_type); // reference: throw 3
	}
	void apply(std::shared_ptr<const Vector<D>> f, std::shared_ptr<Vector<D>> u) const override
	{
		check(tgpu_vcycle(h->p, &o, DeviceVector<D>::raw(f), DeviceVector<D>::raw(u)));
	}
};
// GMG::CycleFactory{2,3}d::getCycle (GMG/CycleFactory3d.cpp:69-134): the level list lives in the Hierarchy; max_levels and
// patches_per_proc (:101-104) are honoured per cycle call by the library
template <size_t D> struct CycleFactory {
	// the reference's call-by-call sequence (one kernel launch per Smoother / Operator / Restrictor / Interpolator call)
	static std::shared_ptr<Operator<D>> getCycle(const CycleOpts &opts, std::shared_ptr<Hierarchy> h)
	{
		return std::make_shared<FusedCycle<D>>(h, opts, true);
	}
	static std::shared_ptr<Operator<D>> getFusedCycle(const CycleOpts &opts, std::shared_ptr<Hierarchy> h)
	{
		return std::make_shared<FusedCycle<D>>(h, opts, false);
	}
};
} // namespace GMG

// BiCGStab<D>::solve (BiCGStab.h:45-106): same signature and meaning; the iteration itself runs inside the library
// (tgpu_bicgstab: device-resident scalars, fused vector passes).  A must be the finest-level DeviceOperator, Mr a cycle
// from GMG::CycleFactory or null.  (The reference's own BiCGStab template runs unchanged over include/tgpu_thunderegg.hpp.)
template <size_t D> class BiCGStab
{
	public:
	static int solve(std::shared_ptr<VectorGenerator<D>> vg, std::shared_ptr<const Operator<D>> A, std::shared_ptr<Vector<D>> x,
	                 std::shared_ptr<const Vector<D>> b, std::shared_ptr<const Operator<D>> Mr = nullptr, int max_it = 1000,
	                 double tolerance = 1e-12)
	{
		(void) vg; // work vectors belong to the hierarchy
		auto op = dynamic_cast<const DeviceOperator<D> *>(A.get());
		if (op == nullptr || op->level != 0) throw Error(TGPU_ERR_ARG, "BiCGStab: A must be the finest-level DeviceOperator");
		const GMG::FusedCycle<D> *cyc = nullptr;
		if (Mr != nullptr) {
			cyc = dynamic_cast<const GMG::FusedCycle<D> *>(Mr.get());
			if (cyc == nullptr) throw Error(TGPU_ERR_ARG, "BiCGStab: Mr must come from GMG::CycleFactory");
		}
		int its = 0;
		check(tgpu_bicgstab(op->h->p, cyc ? &cyc->o : nullptr, DeviceVector<D>::raw(b), DeviceVector<D>::raw(x), tolerance, max_it, &its, nullptr));
		return its;
	}
};
// Stationary multigrid u <- u + M(f - A u) from the initial guess in u until ||f - A u|| <= tol ||f|| (relative to f,
// not to the initial residual as BiCGStab) or max_it cycles; returns the number of cycles.  M is a cycle from
// GMG::CycleFactory on the hierarchy of u (tgpu_gmg_solve: one cycle per iteration on the fused schedule).
template <size_t D> class GMGSolve
{
	public:
	static int solve(std::shared_ptr<const Operator<D>> M, std::shared_ptr<Vector<D>> u, std::shared_ptr<const Vector<D>> f,
	                 double tol = 1e-10, int max_it = 100)
	{
		auto cyc = dynamic_cast<const GMG::FusedCycle<D> *>(M.get());
		if (cyc == nullptr) throw Error(TGPU_ERR_ARG, "GMGSolve: M must come from GMG::CycleFactory");
		int its = 0;
		check(tgpu_gmg_solve(cyc->h->p, &cyc->o, DeviceVector<D>::raw(f), DeviceVector<D>::raw(u), tol, max_it, &its, nullptr, nullptr));
		return its;
	}
};
} // namespace tgpu
