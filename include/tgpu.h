/* tgpu.h - C ABI of the B200-native geometric-multigrid (FAC V-cycle) hot path.
 *
 * Drop-in boundary for ThunderEgg's GMG plugin surface (all citations relative to the
 * reference tree, src/Thunderegg/...):
 *   Operator<D>::apply            Operators/Operator.h:37      -> tgpu_apply
 *   GMG::Smoother<D>::smooth      GMG/Smoother.h:39            -> tgpu_smooth
 *   GMG::Restrictor<D>::restrict  GMG/Restrictor.h:39-40       -> tgpu_restrict
 *   GMG::Interpolator<D>::interpolate GMG/Interpolator.h:39-40 -> tgpu_prolong_add
 *   GMG::Cycle<D>::apply          GMG/Cycle.h:116-126          -> tgpu_vcycle
 *   Vector<D> BLAS-1 + norms      Vector.h:190-321             -> tgpu_vec_* ops
 *   VectorGenerator<D>::getNewVector Vector.h:323-327          -> tgpu_vec_create
 *   BiCGStab<D>::solve            BiCGStab.h:45-106            -> tgpu_bicgstab
 *   Domain<D>/PatchInfo<D>/NbrInfo metadata (Domain.h, PatchInfo.h) -> TgpuLevelDesc
 *   Tree<D> / ThundereggDomGen<D> (OctTree.h, ThundereggDomGen.h)  -> tgpu_mesh_*
 *
 * Conventions: every entry point returns 0 on success and a non-zero code on failure
 * (message via tgpu_last_error()); nothing throws across the ABI.  All arithmetic is IEEE
 * fp64 on the device; there is NO CPU fallback - without a CUDA device tgpu_init fails.
 * One host thread per context.  Patch data is patch-contiguous, x fastest, no ghost cells
 * (PetscVector.h:75-90), ordered by PatchInfo::local_index.
 */
#ifndef TGPU_H
#define TGPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct tgpu_ctx  tgpu_ctx;  /* device + stream + scratch */
typedef struct tgpu_mesh tgpu_mesh; /* host octree/quadtree (Tree<D>) */
typedef struct tgpu_hier tgpu_hier; /* device-resident level hierarchy (neighbour tables) */
typedef struct tgpu_vec  tgpu_vec;  /* device patch vector of one level */

enum { TGPU_OK = 0, TGPU_ERR_ARG = 1, TGPU_ERR_CUDA = 2, TGPU_ERR_IO = 3, TGPU_ERR_UNSUPPORTED = 4, TGPU_ERR_COMM = 5 };
/* neighbour types on a patch side (PatchInfo.h:40-44 NbrType + "no neighbour") */
enum { TGPU_NBR_NONE = -1, TGPU_NBR_NORMAL = 0, TGPU_NBR_COARSE = 1, TGPU_NBR_FINE = 2 };

/* One level of the hierarchy in local_index order; all arrays are host pointers and are copied.
 * Sides: west,east,south,north,bottom,top = 0..2D-1 (Side.h:51-56).  Q = 2^(D-1). */
typedef struct TgpuLevelDesc {
	int32_t        npatch;
	const double  *spacing;        /* [npatch][D]   cell size h; patches must be cubic/isotropic */
	const double  *starts;         /* [npatch][D]   lower corner (only used for the manufactured RHS) */
	const uint8_t *neumann_bits;   /* [npatch]      bit s set: side s is a Neumann domain boundary */
	const int8_t  *nbr_type;       /* [npatch][2D]  TGPU_NBR_* */
	const int32_t *nbr_idx;        /* [npatch][2D][Q] local index of the neighbour patch(es): normal/coarse use
	                                  slot 0, fine uses all Q slots ordered by Orthant<D-1> on the face */
	const int8_t  *orth_on_coarse; /* [npatch][2D]  for a coarse neighbour: which quadrant of its face I cover */
	const int32_t *parent_idx;     /* [npatch]      local index of the parent patch on the next coarser level */
	const int8_t  *orth_on_parent; /* [npatch]      orthant on the parent, -1 = same patch on both levels (copy) */
} TgpuLevelDesc;

/* GMG::CycleOpts (GMG/CycleOpts.h:51-80) */
typedef struct TgpuCycleOpts {
	int32_t pre_sweeps;    /* default 1 */
	int32_t post_sweeps;   /* default 1 */
	int32_t mid_sweeps;    /* default 1 (W cycle) */
	int32_t coarse_sweeps; /* default 1 */
	int32_t cycle_type;    /* 0 = V, 1 = W */
	int32_t fused;         /* 1 (default) = fused kernel schedule (face-only residual), 2 = fused schedule with the residual
	                          evaluated from u and f, 0 = API-granular sequence as GMG/Cycle.h */
	int32_t use_graph;     /* 1 (default) = replay the cycle as a CUDA graph */
	int32_t max_levels;    /* GMG/CycleOpts.h:55: the cycle uses at most this many levels, counted from the finest; 0 = all */
	int32_t interpolator;  /* 0 (default) = piecewise constant, GMG::DrctIntp (the one CycleFactory builds, GMG/CycleFactory3d.cpp:60);
	                          1 = piecewise (bi/tri)linear (GMG/TriLinIntp.cpp, unused upstream); cycles with 1 run the
	                          API-granular schedule */
	int32_t reserved_;     /* keeps the struct free of implicit padding; must be 0 */
	double  patches_per_proc; /* GMG/CycleOpts.h:59: coarsening stops before a level with fewer patches per rank than this
	                             (GMG/CycleFactory3d.cpp:101-104); 0 = never */
} TgpuCycleOpts;

const char *tgpu_last_error(void);
const char *tgpu_version(void);

/* ---- context ---- */
int tgpu_init(int device, tgpu_ctx **ctx);
int tgpu_finalize(tgpu_ctx *ctx);
int tgpu_set_stream(tgpu_ctx *ctx, void *cuda_stream); /* cudaStream_t the library launches on */
int tgpu_sync(tgpu_ctx *ctx);
int tgpu_kernel_launches(tgpu_ctx *ctx, int64_t *count); /* kernels launched (or graph-replayed) so far */
/* device-side timing helpers (CUDA events on the library's stream) */
int tgpu_timer_start(tgpu_ctx *ctx);
int tgpu_timer_stop(tgpu_ctx *ctx, double *milliseconds);

/* per-launch profiling: between begin and end every kernel launch is bracketed by CUDA events
 * (CUDA-graph replay is bypassed while profiling) */
typedef struct TgpuProfileEntry {
	const char *kernel; /* "smooth", "residual_restrict", "prolong_faces", ... */
	int32_t     level;  /* hierarchy level the launch worked on, -1 if none */
	float       ms;
} TgpuProfileEntry;
int tgpu_profile_begin(tgpu_ctx *ctx);
int tgpu_profile_end(tgpu_ctx *ctx, int *n, const TgpuProfileEntry **entries);

/* ---- mesh ingest (host): Tree<D>(file) OctTree.h:90-118, refineLeaves OctTree.h:119-179,
 *      level extraction ThundereggDomGen.h:127-222 + local indexing Domain.h:281-376 ---- */
int tgpu_mesh_load(const char *path, int D, tgpu_mesh **mesh);
int tgpu_mesh_uniform(int D, int num_levels, tgpu_mesh **mesh); /* unit domain, root = level 1 */
int tgpu_mesh_refine_leaves(tgpu_mesh *mesh);
int tgpu_mesh_refine_box(tgpu_mesh *mesh, const double *lo, const double *hi); /* refine leaves with centre in [lo, hi) */
/* Neumann instead of Dirichlet conditions on every domain-boundary side of the levels extracted afterwards
 * (ThundereggDomGen(tree, ns, neumann = true), ThundereggDomGen.h:92,216-220) */
int tgpu_mesh_set_neumann(tgpu_mesh *mesh, int on);
int tgpu_mesh_destroy(tgpu_mesh *mesh);
int tgpu_mesh_info(const tgpu_mesh *mesh, int *D, int *num_levels, int *num_nodes);
/* Extract every level (finest first) for n cells per patch side.  The returned descriptors stay
 * owned by the mesh and valid until the next extract/destroy. */
int tgpu_mesh_extract_levels(tgpu_mesh *mesh, int n, int *nlevels, const TgpuLevelDesc **levels);
/* patch ids (Tree node ids) of one extracted level, for cross-checking against the reference */
int tgpu_mesh_level_ids(const tgpu_mesh *mesh, int level, const int32_t **ids, const int32_t **parent_ids,
                        const int32_t **refine_levels);

/* ---- hierarchy (device neighbour tables; replaces SchurHelper's interface indexing,
 *      InterLevelComm and the PatchSolver plan caches) ---- */
int tgpu_hierarchy_create(tgpu_ctx *ctx, int D, int n, int nlevels, const TgpuLevelDesc *levels, tgpu_hier **h);
int tgpu_hierarchy_destroy(tgpu_hier *h);
int tgpu_hierarchy_info(const tgpu_hier *h, int *D, int *n, int *nlevels);
/* frees what earlier calls allocated lazily (Krylov and full-multigrid work vectors, full-multigrid boundary data,
 * host-buffer slots, cached cycle graphs, pooled vector storage); tables, face buffers and per-level cycle vectors stay */
int tgpu_hierarchy_trim(tgpu_hier *h);
int tgpu_level_npatch(const tgpu_hier *h, int level, int64_t *npatch, int64_t *ncells);
/* the patch solver's shift, FftwPatchSolver(domain, lambda) (PatchSolvers/FftwPatchSolver.h:66,170): block-Jacobi patch
 * problems (Laplacian + lambda) u = rhs; default 0.  Non-zero values take the general (dense-transform) patch solve. */
int tgpu_hierarchy_set_lambda(tgpu_hier *h, double lambda);
/* test hook: on != 0 routes every smoother launch through the size-generic kernel even where a
 * specialised one exists (D = 3, n = 16), so that the two can be compared */
int tgpu_hierarchy_force_generic_kernels(tgpu_hier *h, int on);

/* ---- vectors ---- */
int tgpu_vec_create(tgpu_hier *h, int level, tgpu_vec **v); /* zero-initialised like a new PETSc Vec */
int tgpu_vec_destroy(tgpu_vec *v);
int tgpu_vec_upload(tgpu_vec *v, const double *host);   /* host: ncells doubles */
int tgpu_vec_download(const tgpu_vec *v, double *host);
int tgpu_vec_upload_async(tgpu_vec *v, const double *pinned_host);
int tgpu_vec_download_async(const tgpu_vec *v, double *pinned_host);
int tgpu_vec_device_ptr(const tgpu_vec *v, void **dptr, int64_t *ncells);
int tgpu_host_alloc(size_t bytes, void **pinned);       /* pinned staging memory for e2e paths */
int tgpu_host_free(void *pinned);
/* Vector<D> ops, Vector.h:190-321 */
int tgpu_vec_set(tgpu_vec *v, double alpha);
int tgpu_vec_scale(tgpu_vec *v, double alpha);
int tgpu_vec_shift(tgpu_vec *v, double delta);
int tgpu_vec_copy(tgpu_vec *v, const tgpu_vec *b);
int tgpu_vec_add(tgpu_vec *v, const tgpu_vec *b);
int tgpu_vec_add_scaled(tgpu_vec *v, double alpha, const tgpu_vec *b);                              /* v += alpha b */
int tgpu_vec_add_scaled2(tgpu_vec *v, double alpha, const tgpu_vec *a, double beta, const tgpu_vec *b); /* v += alpha a + beta b */
int tgpu_vec_scale_then_add(tgpu_vec *v, double alpha, const tgpu_vec *b);                          /* v = alpha v + b */
int tgpu_vec_scale_then_add_scaled(tgpu_vec *v, double alpha, double beta, const tgpu_vec *b);      /* v = alpha v + beta b */
int tgpu_vec_scale_then_add_scaled2(tgpu_vec *v, double alpha, double beta, const tgpu_vec *b, double gamma,
                                    const tgpu_vec *c);                                              /* v = alpha v + beta b + gamma c */
int tgpu_vec_two_norm(const tgpu_vec *v, double *result);
int tgpu_vec_inf_norm(const tgpu_vec *v, double *result);
int tgpu_vec_dot(const tgpu_vec *v, const tgpu_vec *b, double *result);

/* ---- per-level operators ---- */
int tgpu_apply(tgpu_hier *h, int level, const tgpu_vec *u, tgpu_vec *out);             /* out = A u */
int tgpu_residual(tgpu_hier *h, int level, const tgpu_vec *f, const tgpu_vec *u, tgpu_vec *r); /* r = f - A u */
int tgpu_smooth(tgpu_hier *h, int level, const tgpu_vec *f, tgpu_vec *u);               /* block-Jacobi sweep */
int tgpu_smooth_jacobi(tgpu_hier *h, int level, const tgpu_vec *f, tgpu_vec *u, double omega); /* weighted point Jacobi */
int tgpu_restrict(tgpu_hier *h, int fine_level, const tgpu_vec *fine, tgpu_vec *coarse);
int tgpu_prolong_add(tgpu_hier *h, int fine_level, const tgpu_vec *coarse, tgpu_vec *fine); /* fine += P coarse */
int tgpu_prolong_add_linear(tgpu_hier *h, int fine_level, const tgpu_vec *coarse, tgpu_vec *fine); /* fine += P_linear coarse */
int tgpu_residual_restrict(tgpu_hier *h, int fine_level, const tgpu_vec *f, const tgpu_vec *u, tgpu_vec *coarse_f);

/* ---- cycle / Krylov ---- */
int tgpu_cycle_opts_default(TgpuCycleOpts *opts);
int tgpu_vcycle(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u); /* u = Cycle(f), zero guess */
/* BiCGStab with the cycle as right preconditioner (opts == NULL: unpreconditioned). */
int tgpu_bicgstab(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u, double tol, int max_it,
                  int *iterations, double *rel_residual);
/* Stationary multigrid from the initial guess in u (a warm start: the previous time step's solution).  Residuals are
 * relative to ||f||_2 (absolute if f = 0), not to the initial residual as in tgpu_bicgstab.  f aliasing u, a vector of
 * another level or hierarchy, tol < 0 or max_it < 0 give TGPU_ERR_ARG and leave u untouched.
 * u <- u + Cycle(f - A u): one cycle from the guess u (opts as tgpu_vcycle; NULL = defaults).  The fused schedule
 * starts the finest level's pre-sweep from u's boundary slices; the others (fused = 0, interpolator = 1, W cycles on
 * several GPUs, no post-sweep, one level, lambda != 0) compute the residual, a cycle from zero and the sum.
 * rel_residual (nullable): ||f - A u_new||_2 / ||f||_2 of the result (fused: from the boundary slices, see DESIGN). */
int tgpu_vcycle_update(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u, double *rel_residual);
/* cycles of tgpu_vcycle_update until ||f - A u||_2 <= tol ||f||_2 (confirmed by a full residual) or max_it cycles.
 * iterations, rel_residual (nullable): cycles run, relative residual of the result.  history (nullable, max_it + 1
 * doubles): the relative residual before the first cycle and after each one (iterations + 1 entries are written). */
int tgpu_gmg_solve(tgpu_hier *h, const TgpuCycleOpts *opts, const tgpu_vec *f, tgpu_vec *u, double tol, int max_it,
                   int *iterations, double *rel_residual, double *history);
/* ---- boundary data (level 0) ----
 * The domain-boundary sides of level 0 (nbr_type TGPU_NBR_NONE) of the owned patches, in ascending (patch, side) order.
 * patch, side (nullable): host arrays of count entries, owned by the hierarchy. */
int tgpu_boundary_sides(const tgpu_hier *h, int64_t *count, const int32_t **patch, const int8_t **side);
/* A zero-initialised vector of count * n^(D-1) doubles: side k's values in the library's face order (the two or one
 * remaining axes, lower axis fastest).  upload / download / device_ptr / set / scale / copy / add / norms / destroy work
 * as for any vector; no level operation accepts it. */
int tgpu_boundary_vec_create(tgpu_hier *h, tgpu_vec **b);
/* f (level 0) -= the boundary terms of b: 2 b / h^2 on Dirichlet sides (b = the boundary value on the face), b / h on
 * Neumann sides (b = the outward normal derivative).  Edge and corner cells take every side's term, as
 * tgpu_init_trig_rhs and tgpu_init_neumann_rhs fold their data. */
int tgpu_fold_boundary(tgpu_hier *h, const tgpu_vec *b, tgpu_vec *f);
/* Full multigrid: u <- FMG(f).  f is level 0 with boundary data folded in, as for every other solver.  b (nullable)
 * holds the Dirichlet values folded into f (tgpu_boundary_vec_create layout); NULL means homogeneous Dirichlet data.
 * Neumann entries of b are not read: R f already carries Neumann folds consistently.  opts as tgpu_vcycle
 * (NULL = defaults); FMG starts on the coarsest level the options select (max_levels / patches_per_proc) with
 * coarse_sweeps sweeps from zero, interpolates each level's result linearly to the next finer level and runs
 * cycles >= 1 cycles from it there (one level: the coarse sweeps only).  u is overwritten.  f aliasing u, vectors of
 * another level or hierarchy, a b that is not a boundary vector of h, cycles < 1 or bad options give TGPU_ERR_ARG and
 * leave u untouched. */
int tgpu_fmg(tgpu_hier *h, const TgpuCycleOpts *opts, int cycles, const tgpu_vec *f, const tgpu_vec *b, tgpu_vec *u);
/* host-buffer convenience (the e2e path): f_host -> device, one cycle, u -> u_host */
int tgpu_vcycle_host(tgpu_hier *h, const TgpuCycleOpts *opts, const double *f_pinned, double *u_pinned);
/* pipelined form for a stream of independent right-hand sides: returns once the work is enqueued; upload of
 * call k + 1, cycle k and download of result k - 1 overlap (two device slots, copy-in / copy-out streams).
 * u_pinned of a call is valid after tgpu_vcycle_host_wait. */
int tgpu_vcycle_host_async(tgpu_hier *h, const TgpuCycleOpts *opts, const double *f_pinned, double *u_pinned);
int tgpu_vcycle_host_wait(tgpu_hier *h);
/* the two copies of one pipelined step alone (host -> dst_dev and src_dev -> host concurrently, then waited for): the
 * host-link ceiling of the e2e path */
int tgpu_vec_transfer_pair(tgpu_hier *h, tgpu_vec *dst_dev, const double *src_pinned, const tgpu_vec *src_dev, double *dst_pinned);

/* ---- multi-GPU (one process per GPU): Morton partition of the patches + NCCL halo exchange ----
 * Replaces the reference's Zoltan partition / migration (ThundereggDomGen.h:223-648), the interface
 * VecScatters (SchurHelper.h:123-150,274-276), InterLevelComm's scatters (GMG/InterLevelComm.h:151-188)
 * and the MPI_Allreduce in the norms (Vector.h:294,306,319).
 * Levels with at least nranks*min_patches_per_rank patches are distributed (owned patches + halo face
 * slots, parents live with their children); coarser levels are replicated on every rank. */
typedef struct tgpu_part tgpu_part;
int tgpu_mesh_partition(tgpu_mesh *mesh, int n, int rank, int nranks, int min_patches_per_rank, tgpu_part **part);
int tgpu_part_destroy(tgpu_part *part);
int tgpu_part_info(const tgpu_part *part, int *nlevels, int *ndistributed);
/* local tables of one level (owned patches first, then halo slots) and the owned/halo -> global maps */
int tgpu_part_level(const tgpu_part *part, int level, TgpuLevelDesc *local_desc, int32_t *n_owned, int32_t *n_halo,
                    const int32_t **owned_global, const int32_t **halo_global, const int32_t **halo_owner, int32_t *npeers);
/* k-th peer of a level: faces to send (local patch, side) and halo faces to receive (slot, side), both in the
 * order the two ranks agree on */
int tgpu_part_peer(const tgpu_part *part, int level, int k, int32_t *peer, int32_t *nsend, const int32_t **send_patch,
                   const int32_t **send_side, int32_t *nrecv, const int32_t **recv_slot, const int32_t **recv_side);
/* owned patches [0, n_interior) have no off-rank neighbour (their sweep overlaps the halo exchange) */
int tgpu_part_level_interior(const tgpu_part *part, int level, int32_t *n_interior);
int tgpu_comm_unique_id(void *id128);                                              /* ncclGetUniqueId (128 bytes) */
int tgpu_comm_init(tgpu_ctx *ctx, const void *id128, int rank, int nranks);       /* ncclCommInitRank */
int tgpu_hierarchy_create_distributed(tgpu_ctx *ctx, const tgpu_part *part, tgpu_hier **h);

/* ---- manufactured problem (apps/3d/steady.cpp:253-265, apps/2d/steady.cpp:314-316,
 *      apps/shared/Init.cpp:152-245,305-361): f with Dirichlet data folded in, exact solution ---- */
int tgpu_init_trig_rhs(tgpu_hier *h, tgpu_vec *f, tgpu_vec *exact);
/* Neumann form (Init::initNeumann / initNeumann2d, apps/shared/Init.cpp:57-151,246-303) of the manufactured problems of
 * apps/3d/steady.cpp:230-282 (problem 0 = trig, 1 = "gauss") and apps/2d/steady.cpp:314-318 (2D: trig only, otherwise
 * TGPU_ERR_UNSUPPORTED); every domain side without a neighbour gets the normal derivative of the exact solution folded
 * into f. */
int tgpu_init_neumann_rhs(tgpu_hier *h, int problem, tgpu_vec *f, tgpu_vec *exact);
/* Domain::integrate (Domain.h:258-278) and Domain::volume (Domain.h:237-256) of a finest-level vector: the app removes
 * integral / volume from a Neumann right-hand side (apps/3d/steady.cpp:330-334).  Sums over all ranks. */
int tgpu_vec_integrate(tgpu_hier *h, const tgpu_vec *v, double *integral, double *volume);

#ifdef __cplusplus
}
#endif
#endif /* TGPU_H */
