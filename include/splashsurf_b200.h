/*
 * splashsurf_b200.h -- C ABI of the B200-native surface-reconstruction hot path.
 *
 * Drop-in boundary: this library replaces the body of
 *     splashsurf_lib::reconstruct_surface_inplace::<i64, f32>()      (splashsurf_lib/src/lib.rs:340-473)
 * i.e. everything from the particle-AABB filter through
 *     reconstruction::reconstruct_surface_subdomain_grid()           (splashsurf_lib/src/reconstruction.rs:17-62)
 * (decomposition -> per-subdomain neighbourhood search + SPH densities -> cubic-spline level-set splat ->
 * per-subdomain marching cubes -> stitching), executed as CUDA kernels on sm_100a.
 *
 * A Rust front-end binds these symbols with `extern "C"` (see INTEGRATION.md for the stub); the Python
 * harness in splashsurf_b200/ binds them with ctypes.  Plain pointers and sizes only -- no CUDA, torch or
 * C++ types cross this boundary.  All entry points are thread-compatible: one context must not be used
 * from two host threads at once (the reference has the same rule for SurfaceReconstruction workspaces,
 * splashsurf_lib/src/workspace.rs:12-79).
 */
#ifndef SPLASHSURF_B200_H
#define SPLASHSURF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SS_ABI_VERSION 3   /* 3: + ss_sph_interpolator_* / ss_neighborhood_search_f32 / ss_marching_cubes_tiles_f32 (additive) */

/* Error codes.  1..7 mirror ReconstructionError / GridConstructionError
 * (splashsurf_lib/src/lib.rs:289-314, uniform_grid.rs:147-169); the reference's panics on a non-positive
 * search radius or degenerate neighbourhood-search domain (neighborhood_search.rs:354-365) map to
 * SS_ERR_INVALID_PARAMETER. */
enum {
    SS_OK = 0,
    SS_ERR_INVALID_CELL_SIZE = 1,        /* GridConstructionError::InvalidCellSize */
    SS_ERR_DEGENERATE_AABB = 2,          /* GridConstructionError::DegenerateAabb */
    SS_ERR_INCONSISTENT_AABB = 3,        /* GridConstructionError::InconsistentAabb */
    SS_ERR_INDEX_TOO_SMALL = 4,          /* IndexTypeTooSmall*: a dimension exceeds what the device path indexes */
    SS_ERR_REAL_TOO_SMALL = 5,           /* RealTypeTooSmallDomainSize */
    SS_ERR_INVALID_PARAMETER = 6,        /* reference: assert!/panic on bad radius, support, subdomain size */
    SS_ERR_UNSUPPORTED = 7,              /* feature not provided by this build (global_neighborhood_list) */
    SS_ERR_INVALID_DOMAIN = 8,           /* DensityMapError::InvalidDomain (density_map.rs:48-61) */
    SS_ERR_CUDA = 100,                   /* CUDA runtime failure; see ss_last_error() */
    SS_ERR_NO_DEVICE = 101,              /* no CUDA device: the product never falls back to a CPU path */
    SS_ERR_OUT_OF_MEMORY = 102,
    SS_ERR_IO = 103                      /* a mesh file could not be opened or written (anyhow errors of the reference's writers) */
};

/* Mirrors splashsurf_lib::Parameters<f32> (lib.rs:158-189) + GridDecompositionParameters (lib.rs:140-145).
 * All lengths are ABSOLUTE (the CLI / Python front-ends multiply their relative -l/-c values by the
 * particle radius before this point: splashsurf/src/reconstruct.rs:628-629). */
typedef struct ss_params_f32 {
    float particle_radius;
    float rest_density;
    float compact_support_radius;
    float cube_size;
    float iso_surface_threshold;
    int32_t has_particle_aabb;           /* Parameters::particle_aabb is Some(..) */
    float particle_aabb_min[3];
    float particle_aabb_max[3];
    int32_t enable_multi_threading;      /* accepted for signature parity; the device path is always parallel */
    int32_t enable_simd;                 /* 1: arithmetic of the reference's AVX2+FMA grid loop (its x86 default);
                                            0: arithmetic of its scalar grid loop */
    int32_t spatial_decomposition;       /* 0: SpatialDecomposition::None, 1: UniformGrid */
    uint32_t subdomain_num_cubes_per_dim;
    int32_t auto_disable;                /* GridDecompositionParameters::auto_disable */
    int32_t global_neighborhood_list;    /* Parameters::global_neighborhood_list: also return the per-particle neighbour lists */
} ss_params_f32;

/* Mirrors UniformCartesianCubeGrid3d<i64, f32> (uniform_grid.rs:132-142). */
typedef struct ss_grid_f32 {
    float aabb_min[3];
    float aabb_max[3];
    float cell_size;
    int64_t points_per_dim[3];
    int64_t cells_per_dim[3];
} ss_grid_f32;

/* Device-side stage times of the last reconstruction on a context, in milliseconds (CUDA events).
 * Stage names follow the reference's profiling scopes (README.md:198-231). */
typedef struct ss_timings {
    float upload;                /* host -> device copy of the particles (0 when the input was device memory) */
    float aabb_and_grid;         /* "compute minimum enclosing aabb" + grid setup */
    float decomposition;         /* "decomposition": classification, membership sort */
    float density;               /* "compute_global_density_vector": cell lists + SPH densities */
    float binning;               /* splat bin sort + particle records */
    float levelset;              /* "density grid loop" over all subdomains */
    float marching_cubes;        /* "mc triangulation loop": classify, scan, emit */
    float stitching;             /* "stitching": boundary-vertex weld, compaction, index remap */
    float total_device;          /* first kernel to last kernel */
    uint64_t kernel_launches;    /* kernels of this library launched (cub passes included) */
    uint64_t levelset_launches;  /* launches of the level-set kernel */
    uint64_t levelset_fixup_points; /* certified points re-evaluated exactly because they touch the surface */
    double levelset_pairs;       /* in-support particle-gridpoint evaluations (only with ss_context_set_count_pairs) */
    uint64_t bricks_total;       /* 8^3-point bricks of all processed tiles */
    uint64_t bricks_levelset;    /* non-empty bricks evaluated by the level-set kernel (CTAs launched) */
    uint64_t bricks_mc;          /* bricks swept by marching cubes (can hold surface) */
    uint64_t bricks_fixscan;     /* bricks swept for certified points next to outside points */
    double levelset_cert_evals;  /* lower-bound evaluations (particle x grid point) of the certification pass (count_pairs, variant 2) */
    double tile_setup;           /* ms between the end of binning and the first level-set kernel, summed over the tile batches: buffer
                                    (re)allocation, tile table upload, zero-fill of the tiles */
} ss_timings;

typedef struct ss_context ss_context;   /* device + stream + reusable device buffers */
typedef struct ss_surface ss_surface;   /* result, mirrors SurfaceReconstruction<i64, f32> (lib.rs:247-262) */

/* Library / ABI info. */
int ss_abi_version(void);
const char *ss_last_error(void);         /* thread-local message for the last non-zero return */

/* Context = the reference's global rayon pool + ReconstructionWorkspace, for one GPU.
 * device < 0 selects the current CUDA device. */
int ss_context_create(int device, ss_context **out);
void ss_context_destroy(ss_context *ctx);

/* reconstruct_surface::<i64, f32>(particle_positions, parameters) (lib.rs:330-337).
 * `xyz` is N x 3 AoS f32 -- the layout of &[Vector3<f32>] / a C-contiguous numpy (N,3) array -- in HOST or
 * DEVICE memory (detected).  On success *out owns the result until ss_surface_free(). */
int ss_reconstruct_surface_f32(ss_context *ctx, const float *xyz, uint64_t n, const ss_params_f32 *params,
                               ss_surface **out);
void ss_surface_free(ss_surface *s);

/* grid_for_reconstruction (lib.rs:476-516) alone, for front-ends that need the grid before reconstructing. */
int ss_grid_for_reconstruction_f32(ss_context *ctx, const float *xyz, uint64_t n, const ss_params_f32 *params,
                                   ss_grid_f32 *grid_out);

/* ---- multi-GPU (one process per GPU; see splashsurf_b200/distributed.py and DESIGN.md row e) ----
 * The reference parallelises over subdomains (dense_subdomains.rs:521-526, :1581-1598); across GPUs each rank
 * owns a slab of the subdomain grid: subdomains whose index along `axis` lies in [own_lo, own_hi).  `grid` is the
 * grid of ALL particles (ss_grid_for_reconstruction_f32 of the reduced bounding box); `xyz` are the rank's particles
 * in ASCENDING GLOBAL INDEX order: every particle that is a member (owner or ghost) of a subdomain in
 * [own_lo - halo, own_hi + halo).  Subdomains of the halo layers are processed for particle densities only, so that
 * ghost particles get the same density the owning rank computes.  `global_max_particles` is the maximum particle
 * count of any subdomain over all ranks (sparse-subdomain rule, dense_subdomains.rs:1242-1251); with
 * stop_after_decomposition != 0 only the decomposition runs and ss_surface_max_subdomain_particles() reports the
 * local maximum to be max-reduced across ranks. */
int ss_reconstruct_partition_f32(ss_context *ctx, const float *xyz, uint64_t n, const ss_params_f32 *params,
                                 const ss_grid_f32 *grid, int axis, int64_t own_lo, int64_t own_hi, int64_t halo,
                                 uint64_t global_max_particles, int stop_after_decomposition, ss_surface **out);
/* Same, in ONE call: after the decomposition the library calls `max_reduce(local_max, user)`, which must return the maximum
 * over all ranks (e.g. an NCCL all-reduce issued by the caller), and continues with it. */
int ss_reconstruct_partition_cb_f32(ss_context *ctx, const float *xyz, uint64_t n, const ss_params_f32 *params,
                                    const ss_grid_f32 *grid, int axis, int64_t own_lo, int64_t own_hi, int64_t halo,
                                    uint64_t (*max_reduce)(uint64_t local_max, void *user), void *user, ss_surface **out);
uint64_t ss_surface_max_subdomain_particles(const ss_surface *s);
/* Slab-plan statistics of this rank's particles (DEVICE pointers): hist[nsd_axis] = particles per subdomain layer along `axis`,
 * occ[nsd_x * nsd_y * nsd_z] = 1 for every subdomain slot that owns a particle (x-major flat index).  The caller sums / max-reduces
 * them across ranks (NCCL) and cuts the layers into slabs. */
int ss_partition_stats_f32(ss_context *ctx, const float *xyz_dev, uint64_t n, const ss_grid_f32 *grid, uint32_t subdomain_cubes,
                           int axis, uint32_t *hist_dev, uint32_t *occ_dev);
/* Plan statistics with the exact ghost classifier (dense_subdomains.rs:1810-1905): members[slot] = how many of these particles are
 * members (owner or ghost) of subdomain `slot` (nsd_x * nsd_y * nsd_z u32, device memory); hist as in ss_partition_stats_f32.  Summed
 * over all ranks, max(members) is the global maximum subdomain population of the sparse rule (:1242-1251), so a runner can pass it
 * to ss_reconstruct_partition_f32 directly (no decomposition pre-pass, no callback), and members > 0 marks the occupied tiles. */
int ss_partition_members_f32(ss_context *ctx, const float *xyz_dev, uint64_t n, const ss_params_f32 *params, const ss_grid_f32 *grid, int axis,
                             uint32_t *hist_dev, uint32_t *members_dev);

/* Halo packing for the one exchange step: destination d receives the particles with lo[d] <= xyz[axis] < hi[d] (a particle may go
 * to several destinations), grouped by destination, ascending index inside a destination.  Call once with send_dev == NULL to
 * get counts_out[world] (host), then with a device buffer of sum(counts) * 3 floats. */
int ss_partition_pack_f32(ss_context *ctx, const float *xyz_dev, uint64_t n, int axis, const double *lo, const double *hi,
                          uint32_t world, uint64_t *counts_out, float *send_dev);
const unsigned long long *ss_surface_device_vertex_keys(const ss_surface *s);   /* nv u64 MC edge keys, device memory */
int ss_surface_copy_subdomain_owned(const ss_surface *s, uint8_t *dst);          /* 1: owned, 0: density-only halo */
/* Welds vertices with equal MC edge key in a concatenation of per-rank meshes (all pointers DEVICE memory; `cand`
 * lists the vertex ids that may be duplicated, i.e. vertices on the faces between slabs).  Compacts verts / keys in
 * place, renumbers tris, returns the vertex count in *nv_out ("stitching" across GPUs). */
int ss_weld_meshes(ss_context *ctx, float *verts, unsigned long long *keys, uint64_t nv, uint32_t *tris, uint64_t nt,
                   const uint32_t *cand, uint64_t n_cand, uint64_t *nv_out);

/* Stage-level entry: density_grid_loop_auto / density_grid_loop_scalar (dense_subdomains.rs:715-847, both `pub`
 * and driven by the reference's own bench fixture, benches/benches/bench_grid_loop.rs:203-262).  Evaluates the
 * (S+1)^3 level-set tile (i-major, f32) of ONE subdomain from an explicit particle list -- accumulated in list
 * order -- and explicit particle densities.  mode 0: arithmetic of the AVX2+FMA loop, 1: scalar loop.
 * xyz / rho / tile_out may be host or device pointers. */
int ss_levelset_tile_f32(ss_context *ctx, const float *xyz, const float *rho, uint64_t n, const float global_min[3],
                         float cube_size, const int64_t subdomain_ijk[3], uint32_t subdomain_cubes,
                         float compact_support_radius, float particle_rest_mass, int mode, float *tile_out);

/* Result copies into pageable host memory larger than four chunks are staged through page-locked buffers and scattered by several
 * host threads (parallel first touch of fresh arrays; ss_surface_copy_triangles_u64 widens on the host).  Chunk size, default and
 * maximum 32 MiB; smaller values only make sense for tests. */
int ss_context_set_copy_chunk_bytes(ss_context *ctx, uint64_t bytes);

/* Page-locked host memory (cudaHostAlloc) for callers that have no CUDA binding of their own: result copies into it run at PCIe
 * speed.  NULL on failure. */
void *ss_host_alloc_pinned(uint64_t bytes);
void ss_host_free_pinned(void *p);

/* ---- result accessors (sizes first, then copies into caller-provided HOST buffers) ---- */
uint64_t ss_surface_num_vertices(const ss_surface *s);
uint64_t ss_surface_num_triangles(const ss_surface *s);
uint64_t ss_surface_num_particles(const ss_surface *s);          /* particles after the AABB filter */
int ss_surface_used_decomposition(const ss_surface *s);
int ss_surface_grid(const ss_surface *s, ss_grid_f32 *grid_out);            /* SurfaceReconstruction::grid */
int ss_surface_subdomain_grid(const ss_surface *s, ss_grid_f32 *grid_out);  /* ::subdomain_grid */
int ss_surface_copy_vertices(const ss_surface *s, float *dst_xyz);          /* mesh.vertices, nv x 3 */
int ss_surface_copy_triangles_u32(const ss_surface *s, uint32_t *dst);      /* mesh.triangles, nt x 3 */
int ss_surface_copy_triangles_u64(const ss_surface *s, uint64_t *dst);      /* same, usize like the reference */
int ss_surface_copy_particle_densities(const ss_surface *s, float *dst);    /* ::particle_densities */
int ss_surface_copy_particle_inside_aabb(const ss_surface *s, uint8_t *dst);/* ::particle_inside_aabb (n input) */
/* SurfaceReconstruction::particle_neighbors (only with global_neighborhood_list): CSR -- offsets has num_particles + 1
 * entries, indices holds global particle indices in the reference's visiting order (neighborhood_search.rs:396-433). */
uint64_t ss_surface_num_neighbors(const ss_surface *s);
int ss_surface_copy_neighbor_lists(const ss_surface *s, uint64_t *offsets, uint32_t *indices);
/* Device-resident views (valid until ss_surface_free): vertices nv x 3 f32, triangles nt x 3 u32. */
const float *ss_surface_device_vertices(const ss_surface *s);
const uint32_t *ss_surface_device_triangles(const ss_surface *s);
const float *ss_surface_device_densities(const ss_surface *s);

/* ---- parity taps (used by tests/; cheap, no effect on the hot path unless requested) ---- */
/* Global MC edge carrying each vertex: (point i, j, k, axis), nv x 4 int64. */
int ss_surface_copy_vertex_edge_keys(const ss_surface *s, int64_t *dst);
/* Decomposition: number of non-empty subdomains, their flat indices (ascending), particle counts
 * (owned + ghost) and the sparse flag (dense_subdomains.rs:1251, :1590). */
uint64_t ss_surface_num_subdomains(const ss_surface *s);
int ss_surface_copy_subdomains(const ss_surface *s, int64_t *flat, uint64_t *count, uint8_t *sparse);
/* Request that the level-set tile ((S+1)^3 f32, i-major) of one subdomain (flat index) is kept by the next
 * reconstruction on this context; pass -1 to disable. */
int ss_context_keep_levelset_tile(ss_context *ctx, int64_t flat_subdomain);
int ss_surface_copy_levelset_tile(const ss_surface *s, float *dst);

/* Timings / launch counts of the reconstruction that produced `s`. */
int ss_surface_timings(const ss_surface *s, ss_timings *out);

/* Tuning knobs (do not change results).
 * - maximum number of subdomain tiles resident at once;
 * - level-set evaluation: by default grid points that are provably inside the fluid (a partial sum of the
 *   non-negative kernel terms already exceeds the threshold) are only classified, and every point on a
 *   surface-crossing edge is evaluated exactly; `exact_everywhere` evaluates every point exactly like the reference;
 * - count_pairs: count in-support kernel evaluations into ss_timings.levelset_pairs (instrumented kernel). */
int ss_context_set_tile_batch(ss_context *ctx, uint32_t max_tiles);
int ss_context_set_levelset_exact_everywhere(ss_context *ctx, int on);
/* Level-set launch structure (same results): 2 (default) = warp-per-brick certification kernel (bulk-copy staging, packed FP32)
 * + warp-per-brick exact pass over the boxes it could not certify; 1 = CTA-per-brick certification kernel + k_levelset exact
 * pass; 0 = fused certification + exact pass per brick (k_levelset). */
int ss_context_set_levelset_variant(ss_context *ctx, int variant);
/* Density kernel structure (same results): 0 (default) = one thread per particle over the compacted list of in-subdomain
 * memberships (k_density; 17 ms at 50 M particles); 1 / 2 = one warp per h-cell, the candidates of the 27 cells staged once per cell
 * (1: by bulk copies, 2: by 16-byte loads), ordered hit lists by ballot (csrc/ss_density.cuh) -- measured SLOWER on the B200 (36-38
 * ms: 550 warp-instructions per particle against 468; profiles/README.md) and kept as a documented experiment.  Replaces the
 * per-particle neighbour loop of neighborhood_search.rs:396-433 + density_map.rs:169-185. */
int ss_context_set_density_variant(ss_context *ctx, int variant);
/* Brick passes of the subdomain path (same mesh; vertex / triangle order inside a brick differs): 1 (default) = one warp per
 * 8x8x8-point brick, marching cubes in two launches (count, emit) and the marker fix-up sweep on row bit masks (csrc/ss_mc.cuh);
 * 0 = one CTA per brick, three marching-cubes launches.  Replaces dense_subdomains.rs:1470-1568. */
int ss_context_set_mc_variant(ss_context *ctx, int variant);
int ss_context_set_count_pairs(ss_context *ctx, int on);

/* ---- SPH normals at the mesh vertices: SphInterpolator::interpolate_normals (sph_interpolation.rs:82-133) as used by the
 * pipeline's `--sph-normals` (splashsurf/src/reconstruct.rs:1126-1129, :1287-1294): particle volume = (4/3 pi r^3 rho0) /
 * rho_j, cubic-spline gradient, normalised.  Enable on the context before reconstructing; the unit normals (nv x 3 f32)
 * are then part of the result.  Parity with the reference is to rounding (its summation follows R-tree order). */
int ss_context_set_compute_sph_normals(ss_context *ctx, int on);
int ss_surface_copy_normals(const ss_surface *s, float *dst_xyz);
const float *ss_surface_device_normals(const ss_surface *s);

/* ---- Anisotropic kernels (Yu & Turk 2013; DESIGN.md "Anisotropic kernels"), opt-in.  Every particle's kernel is stretched along
 * the principal axes of its neighbourhood's weighted covariance (radii in [R / max_ratio, R], isotropic below min_neighbors
 * neighbours) and centred at x + smoothing * (weighted neighbour mean offset).  The level set is sum_i f_i W_R(sqrt(u^T M_i u)),
 * u = x - centre_i, on the same grid and with the same threshold; marching cubes and stitching are unchanged.  NULL (the
 * default) switches it off.  Out of range (max_ratio < 1, smoothing outside [0, 1], NaN): SS_ERR_INVALID_PARAMETER.  The
 * partitioned entries return SS_ERR_UNSUPPORTED while it is on. */
typedef struct { float max_ratio; uint32_t min_neighbors; float smoothing; } ss_anisotropy_f32;
int ss_context_set_anisotropy_f32(ss_context *ctx, const ss_anisotropy_f32 *a);
/* per (filtered) particle of an anisotropic reconstruction: centres n x 3, matrices M = R^2 A n x 6 (xx, xy, xz, yy, yz, zz),
 * factors f = (m / rho) R^3 / (a1 a2 a3) n; any pointer may be NULL */
int ss_surface_copy_anisotropy_f32(const ss_surface *s, float *centers, float *matrices, float *factors);
/* device ms of the anisotropic stages -- ms2[0] moments + eigen-decomposition, ms2[1] decomposition and binning of the centres (the
 * level set and marching cubes are in ss_timings) -- and the most Jacobi sweeps one particle's eigen-decomposition took (cap 8);
 * either pointer may be NULL */
int ss_surface_anisotropy_stats(const ss_surface *s, float *ms2, uint32_t *max_jacobi_sweeps);

/* ---- Mesh post-processing on the device (SURVEY.md 8f; the steps of splashsurf/src/reconstruct.rs:1094-1391 that follow the
 * reconstruction).  They operate in place on the surface's device mesh; copy results out with the accessors above.
 * The entries marked [bins] query the particles through the splat bins of the reconstruction that produced the surface and
 * must therefore be called before the next reconstruction on the same context (SS_ERR_INVALID_PARAMETER otherwise); they
 * are not available on partitioned (multi-GPU) surfaces (SS_ERR_UNSUPPORTED).  Sums run in a different order than the
 * reference's R-tree / hash order: results agree to f32 round-off, not bit for bit.
 * Reference order of the steps: weights -> vertex smoothing -> normals -> normal smoothing -> attribute interpolation. */

/* [bins] SphInterpolator::interpolate_scalar_quantity / interpolate_vector_quantity (sph_interpolation.rs:141-258) at the mesh
 * vertices, interpolator as in reconstruct.rs:1094-1149 (sphere rest mass 4/3 pi r^3 rho0, the reconstruction's densities).
 * values: [num_particles * dim] of the FILTERED particles, dim = 1 or 3; out: [num_vertices * dim]; host or device pointers. */
int ss_surface_interpolate_quantity_f32(ss_surface *s, const float *values, uint32_t dim, int first_order_correction, float *out);

/* [bins] Smoothing weights (reconstruct.rs:1159-1258): distance-weighted neighbour count per particle, SPH-interpolated to the
 * vertices ("wnn"), min(max(n, 0) / normalization, 1) through the smooth-step 6x^5 - 15x^4 + 10x^3 ("sw").  The weights stay
 * on the device for ss_surface_laplacian_smoothing_f32; wnn_out / weights_out ([num_vertices]) may be NULL. */
int ss_surface_compute_smoothing_weights_f32(ss_surface *s, float normalization, float *wnn_out, float *weights_out);

/* splashsurf_lib::postprocessing::par_laplacian_smoothing_inplace (postprocessing.rs:17-53), including its buffer swap (the
 * blended vertex is the one of two iterations ago).  weights: [num_vertices] or NULL = the weights computed by
 * ss_surface_compute_smoothing_weights_f32 on this surface, 1 if it was not called. */
int ss_surface_laplacian_smoothing_f32(ss_surface *s, uint32_t iterations, float beta, const float *weights);

/* Vertex normals at the current (possibly smoothed) vertices, readable with ss_surface_copy_normals:
 * sph != 0: [bins] SphInterpolator::interpolate_normals (sph_interpolation.rs:82-133);
 * sph == 0: TriMesh3d::par_vertex_normals, area-weighted triangle normals (mesh.rs:799-906). */
int ss_surface_compute_normals_f32(ss_surface *s, int sph);

/* par_laplacian_smoothing_normals_inplace (postprocessing.rs:56-97) on the surface's normals. */
int ss_surface_smooth_normals_f32(ss_surface *s, uint32_t iterations);

/* ---- splashsurf_lib::sph_interpolation::SphInterpolator at arbitrary points (sph_interpolation.rs:22-258; pysplashsurf.SphInterpolator).
 * ss_sph_interpolator_create_f32 = SphInterpolator::new (:40-80): particle positions (n x 3), their densities (n), the particle rest
 * mass and the compact support radius; host or device pointers.  The handle is a surface without a mesh (free it with ss_surface_free);
 * its particle bins live in the context's scratch, so -- like the [bins] entries above -- it must be used before the next reconstruction or
 * interpolator on the same context (SS_ERR_INVALID_PARAMETER otherwise).  Sums run in bin order, not in the reference's R-tree order:
 * results agree to f32 round-off. */
int ss_sph_interpolator_create_f32(ss_context *ctx, const float *xyz, uint64_t n, const float *densities, float particle_rest_mass,
                                   float compact_support_radius, ss_surface **out);
/* interpolate_scalar_quantity / interpolate_vector_quantity (:141-258): values [n * dim] (dim = 1 or 3), points [m * 3], out [m * dim]. */
int ss_sph_interpolate_quantity_at_f32(ss_surface *interpolator, const float *values, uint32_t dim, const float *points, uint64_t m,
                                       int first_order_correction, float *out);
/* interpolate_normals (:82-133): unit SPH normals at the points, out [m * 3] (NaN where no particle lies within the support). */
int ss_sph_interpolate_normals_at_f32(ss_surface *interpolator, const float *points, uint64_t m, float *out);

/* splashsurf_lib::neighborhood_search::neighborhood_search_spatial_hashing_parallel (neighborhood_search.rs:444-588; Python function of the
 * same name): for every particle the indices of all OTHER particles with squared distance < search_radius^2, found on the cell lattice of
 * UniformGrid::from_aabb(domain, search_radius).  The result is a surface without a mesh: read the CSR lists with
 * ss_surface_num_neighbors / ss_surface_copy_neighbor_lists, free it with ss_surface_free.  The order inside a list is this library's
 * (cells x-major, ascending index inside a cell); the reference's depends on its hash map.  A particle outside of the domain's lattice is
 * SS_ERR_INVALID_PARAMETER (reference: panic). */
int ss_neighborhood_search_f32(ss_context *ctx, const float *xyz, uint64_t n, const float domain_min[3], const float domain_max[3],
                               float search_radius, ss_surface **out);

/* marching_cubes::triangulate_density_map (marching_cubes.rs:61-127; Python: pysplashsurf.marching_cubes on a dense array) on level-set
 * tiles the caller provides: `tiles` = ntiles x 65^3 floats (host or device), tile t holding the global points tile_ijk[3t..] * 64 .. + 64
 * per axis (neighbouring tiles repeat their shared face planes), point (i, j, k) at grid_min + index * cube_size.  Inside / outside and
 * the vertex interpolation follow the reference's global path (value > threshold is inside; vertices from the point >= threshold towards
 * its neighbour below).  The mesh is welded across tiles; ss_surface_copy_vertex_edge_keys tells which grid edge a vertex lies on, so a
 * caller that padded its array to whole tiles can drop the cells of the padding. */
int ss_marching_cubes_tiles_f32(ss_context *ctx, const float *tiles, uint32_t ntiles, const int32_t *tile_ijk, const float grid_min[3],
                                float cube_size, float iso_surface_threshold, ss_surface **out);

/* A surface around a caller-supplied mesh (verts nv x 3 f32, tris nt x 3 u32; host or device pointers), so that the mesh-only
 * entries (laplacian smoothing with explicit / unit weights, area-weighted normals, normal smoothing, connectivity) serve the
 * reference's free functions of postprocessing.rs / mesh.rs on any mesh.  No particles: the [bins] entries are rejected. */
int ss_surface_from_mesh_f32(ss_context *ctx, const float *verts, uint64_t nv, const uint32_t *tris, uint64_t nt, ss_surface **out);

/* Replaces the mesh of a surface (host or device arrays) and keeps its link to the reconstruction it came from, so that the
 * particle-based entries above (smoothing weights, SPH normals, attribute interpolation) run on the new vertices -- the hook for
 * the host-side steps below inside the pipeline (reconstruct.rs:1058-1092 runs them before everything else).  Cached adjacency,
 * weights and normals are dropped; marching-cubes edge keys no longer apply. */
int ss_surface_replace_mesh_f32(ss_surface *s, const float *verts, uint64_t nv, const uint32_t *tris, uint64_t nt);

/* ---- SURVEY 8(f.4): sequential half-edge algorithms, HOST code like in the reference (no context, no device needed).
 * In place on host arrays: verts [*nv x 3] f32, tris [*nt x 3] u32; *nv / *nt are updated (never grow).  keep_vertices != 0 keeps
 * vertices that lost all their triangles (halfedge_mesh.rs:92-100, :446-497).  Optional output: the vertex-vertex connectivity of
 * the result in half-edge order as CSR (conn_offsets: nv_in + 1 entries, conn_indices: capacity 6 * nt_in = twice the edges of an
 * open mesh; 3 * nt_in suffices for a closed one), which the reference
 * returns as Vec<Vec<usize>>.
 *
 * marching_cubes_cleanup (postprocessing.rs:99-242, "mesh displacement" after Moore & Warren): every vertex is assigned its nearest
 * grid point; neighbouring vertices with the same grid point are merged by half-edge collapses (halfedge_mesh.rs:204-373) into their
 * running average, for at most max_iter sweeps.  max_rel_snap_distance < 0 = None; else only vertices within that distance (in cell
 * sizes) of the grid point take part.  `grid` is the marching-cubes grid of the reconstruction (ss_surface_grid). */
int ss_mesh_cleanup_f32(float *verts, uint64_t *nv, uint32_t *tris, uint64_t *nt, const ss_grid_f32 *grid, float max_rel_snap_distance,
                        uint64_t max_iter, int keep_vertices, uint64_t *conn_offsets, uint32_t *conn_indices);
/* decimation (postprocessing.rs:244-686): merges the single and double "barnacle" configurations of marching-cubes meshes.  The
 * reference walks hash sets / maps of candidates (std HashMap + fxhash); their iteration order is restated, so the result is the
 * reference's, vertex for vertex, also where two candidates claim the same vertex. */
int ss_mesh_decimation_f32(float *verts, uint64_t *nv, uint32_t *tris, uint64_t *nt, int keep_vertices, uint64_t *conn_offsets,
                           uint32_t *conn_indices);

/* convert_tris_to_quads (postprocessing.rs:689-910): pairs of triangles sharing an edge become quads when all four edges are within
 * [1 / limit, limit] x diagonal / sqrt(2), no interior angle exceeds max_interior_angle_rad and the two triangle normals are within
 * normal_angle_limit_rad.  Outputs: the remaining triangles (capacity nt x 3, in input order) and the quads (capacity nt / 2 x 4, in the
 * reference's order -- its hash-set iteration order is restated).  Vertices are unchanged.  Host code. */
int ss_mesh_tris_to_quads_f32(const float *verts, uint64_t nv, const uint32_t *tris, uint64_t nt, float non_squareness_limit,
                              float normal_angle_limit_rad, float max_interior_angle_rad, uint32_t *tris_out, uint64_t *nt_out,
                              uint32_t *quads_out, uint64_t *nq_out);

/* ---- SURVEY 8(f.3): the mesh writers of `splashsurf reconstruct -o <file>` (splashsurf/src/io.rs:276-316 write_mesh -> vtk_format.rs:188-211
 * write_vtk(mesh, file, "mesh"), ply_format.rs:190-267 mesh_to_ply, obj_format.rs:17-71 mesh_to_obj).  HOST code, multi-threaded formatting,
 * output byte for byte the reference CLI's file for the same mesh and attributes.  A mesh is vertices + triangles (+ quads of a
 * MixedTriQuadMesh3d: cells are the triangles followed by the quads, postprocessing.rs:901-903) with u32 or u64 indices; attributes
 * mirror OwnedAttributeData (mesh.rs): f32 scalars, f32 3-vectors, u64 scalars, one entry per vertex / per cell.
 *   .vtk  legacy BINARY unstructured grid, every attribute as SCALARS <name> float|unsigned_long 1|3 + default lookup table
 *   .ply  binary_little_endian: x y z + point attributes per vertex ("normals" as nx ny nz, u64 as uint); cell attributes are not written
 *   .obj  v / vn (a point attribute named "normals") / f lines, numbers as Rust's `{}` prints them (shortest round trip, no exponent)
 * format SS_MESH_FORMAT_AUTO picks by the extension (case-insensitive) with the reference's error messages.  threads 0 = up to 16. */
#define SS_ATTR_SCALAR_F32 0
#define SS_ATTR_VECTOR3_F32 1
#define SS_ATTR_SCALAR_U64 2
#define SS_MESH_FORMAT_AUTO 0
#define SS_MESH_FORMAT_VTK 1
#define SS_MESH_FORMAT_PLY 2
#define SS_MESH_FORMAT_OBJ 3
typedef struct ss_mesh_attribute {
    const char *name;
    int32_t kind;                        /* SS_ATTR_* */
    const void *data;
} ss_mesh_attribute;
int ss_write_mesh_f32(const char *path, int format, const float *verts, uint64_t nv, const void *tris, uint64_t nt, const void *quads,
                      uint64_t nq, int index_bytes, const ss_mesh_attribute *point_attrs, uint32_t n_point_attrs,
                      const ss_mesh_attribute *cell_attrs, uint32_t n_cell_attrs, uint32_t threads);
/* Test knob: items (vertices / cells / values) per work chunk of the writer's thread pipeline, process-wide; 0 restores the built-in sizes
 * (32 Ki lines of an OBJ, 64 Ki PLY records, 256 Ki - 1 Mi VTK values).  The file written does not depend on it. */
int ss_meshio_set_chunk_items(uint64_t items);
/* One f32 as the OBJ writer prints it (Rust `{}`), NUL-terminated; 64 bytes always suffice. */
int ss_format_f32(float value, char *out, uint64_t capacity);

/* Replaces the surface's normals by [num_vertices * 3] caller-supplied ones (then ss_surface_smooth_normals_f32 smooths any field). */
int ss_surface_set_normals_f32(ss_surface *s, const float *normals);

/* TriMesh3d::vertex_vertex_connectivity (mesh.rs:290-306) as CSR, neighbours ascending: offsets [num_vertices + 1],
 * indices [*n_indices]; pass indices = NULL to query *n_indices first. */
int ss_surface_vertex_connectivity(ss_surface *s, uint64_t *offsets, uint32_t *indices, uint64_t *n_indices);

#ifdef __cplusplus
}
#endif
#endif /* SPLASHSURF_B200_H */
