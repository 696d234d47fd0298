// ss_pipeline.cu -- host orchestration + C ABI of the B200 reconstruct path (see include/splashsurf_b200.h).
//
// Host-side mirror of splashsurf_lib::reconstruct_surface_inplace (lib.rs:340-473) and
// reconstruction::reconstruct_surface_subdomain_grid (reconstruction.rs:17-62): parameter validation, grid
// derivation in exact f32 (lib.rs:476-516, dense_subdomains.rs:89-244), then the device pipeline.  There is
// no CPU fallback: without a CUDA device every entry point fails with SS_ERR_NO_DEVICE.
#include "../../include/splashsurf_b200.h"
#include "ss_kernels.cuh"
#include "ss_certify.cuh"
#include "ss_exact.cuh"
#include "ss_density.cuh"
#include "ss_mc.cuh"
#include "ss_aniso.cuh"

#ifndef SS_HOST_EMUL               // (tests/emul/cuda_emul.h compiles this file with g++ to step the kernels on the CPU)
#include <cub/cub.cuh>
#endif
#include <cfloat>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>

// ------------------------------------------------------------------ errors ----
static thread_local std::string g_last_error;
static int ss_fail(int code, const std::string &msg) { g_last_error = msg; return code; }

struct SsCudaError { cudaError_t e; const char *what; const char *file; int line; };
#define CK(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) throw SsCudaError{ _e, #call, __FILE__, __LINE__ }; } while (0)

// ------------------------------------------------------------------ device buffers ----
// Growth slack of the pooled buffers in eighths of the request: 1 (12.5 %) for whole-domain runs; partitioned (multi-GPU) runs use 4
// (50 %), because the slab plan -- and with it every per-rank size -- moves a little from frame to frame while it balances, and
// re-allocating the scratch costs far more than the memory it saves (each rank holds 1/N of the data anyway).
static int g_devbuf_slack_eighths = 1;
struct DevBuf {
    void *p = nullptr; size_t cap = 0;
    template <typename T> T *as() const { return (T *)p; }
    void ensure(size_t bytes) {
#ifdef SS_EMUL_GUARD                      // tests/emul: exact-size allocations in front of a guard page (overrun detection)
        if (bytes == cap && p) return;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes;
#else
        if (bytes <= cap) return;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + (bytes / 8) * (size_t)g_devbuf_slack_eighths + 256;
#endif
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; throw SsCudaError{ e, "cudaMalloc", __FILE__, __LINE__ }; }
        cap = want;
    }
    // grow while preserving contents
    void grow_keep(size_t bytes, size_t used, cudaStream_t st) {
        if (bytes <= cap) return;
#ifdef SS_EMUL_GUARD
        size_t want = bytes;
#else
        size_t want = std::max(bytes + bytes / 4, cap * 2) + 256;
#endif
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, want);
        if (e != cudaSuccess) throw SsCudaError{ e, "cudaMalloc", __FILE__, __LINE__ };
        if (p && used) CK(cudaMemcpyAsync(q, p, used, cudaMemcpyDeviceToDevice, st));
        if (p) { CK(cudaStreamSynchronize(st)); cudaFree(p); }
        p = q; cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct HostGrid { float mn[3], mx[3]; float cell; int64_t np[3], nc[3]; };

// State of the most recent reconstruction that the post-processing entries (ss_post.cuh) need, and their scratch.
struct PostScratch {
    int valid = 0;                   // the splat bins in the context scratch belong to frame `ss_context::frame`
    int partitioned = 0;
    SsDev D{};
    uint32_t nsub = 0, M = 0;
    float sphere_mass = 0.f;         // 4/3 pi r^3 rho0 (reconstruct.rs:1126-1129)
    DevBuf keys_a, keys_b, flag, scan, vals, out, tmpv;
    void release_all() { for (DevBuf *b : { &keys_a, &keys_b, &flag, &scan, &vals, &out, &tmpv }) b->release(); }
};

struct ss_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[12];
    uint32_t max_tiles = 0;          // 0 = auto
    int64_t keep_tile_flat = -1;
    int ls_exact_all = 0;            // 1: evaluate every grid point exactly (no certification)
    int ls_variant = 2;              // 2 (default): warp-per-brick certification + exact kernels (ss_certify.cuh, ss_exact.cuh); 1: CTA-per-brick certification kernel; 0: fused k_levelset
    int count_pairs = 0;             // 1: count in-support evaluations (work model; slower)
    int density_variant = 0;         // 0 (default, fastest measured): thread-per-particle k_density; 1 / 2: cell-cooperative kernel (ss_density.cuh), candidates staged by bulk copies / 16-byte loads
    int mc_variant = 1;              // 1 (default): warp-per-brick marching cubes (count + emit) and fix-up sweep (ss_mc.cuh); 0: CTA-per-brick passes
    void *h_stage[2] = { nullptr, nullptr };   // page-locked staging buffers of the result copies (copy_out), allocated on first use
    size_t stage_bytes = (size_t)32 << 20;     // chunk size of the staged result copies (copies below 4 chunks are plain)
    cudaEvent_t ev_stage[2] = { nullptr, nullptr };
    int sm_count = 148;              // streaming multiprocessors of the device (persistent-kernel grid sizing)
    int sph_normals = 0;             // 1: SPH normals at the mesh vertices (sph_interpolation.rs:82-133)
    int aniso = 0;                   // 1: anisotropic kernels (ss_aniso.cuh) with parameters aniso_k
    SsAniso aniso_k{};
    cudaEvent_t ev_an[3] = { nullptr, nullptr, nullptr };   // anisotropic stages: after densities, before / after the centres' decomposition
    // bins of the anisotropic centres (the isotropic bins in key_a .. ksplit stay for the post-processing queries) + per-particle data
    DevBuf an_key_a, an_key_b, an_val_a, an_val_b, an_flags, an_scan, an_cid, an_sub_flat, an_sub_off, an_tab_a, an_tab_b, an_rec, an_ksplit,
        an_am, an_sweeps, o_an_xbar, o_an_mat, o_an_fac;
    // reusable scratch
    DevBuf xyz, xyz_f, filt_flag, filt_flag32, filt_off, aabb, cnt, off, key_a, key_b, val_a, val_b, cid, cub_tmp,
        sub_flat, sub_off, sub_sparse, sub_owned, gkey_a, gkey_b, gval_a, gval_b, flags, scan, spos, rho, tab_a, tab_b, rec, ksplit, batch_subs, tiles, vcnt,
        tcnt, vmask, voff, vblk_off, tblk_off, tile_tab, brick_rng, bstate, flag_ls, off_ls, list_ls, flag_mc, flag_fix, off_mc, off_fix, list_mc, list_fix, wflag, wstate, desc_ls, dflag, doff, dlist, fallback, fallback2, fallback3, pack_cnt, pack_off, brick_seen, fix_list, nflag, bkeys_a, bkeys_b, bids_a, bids_b, bcount, remap, keep, newid, err, pairs;
    uint64_t launches = 0;
    int big_attr_set = 0;            // dynamic shared memory opt-in of k_exact_warp_big done
    uint64_t pack_n = 0; uint32_t pack_world = 0;   // ss_partition_pack_f32: count phase the scatter phase must match
    // result buffers handed to surfaces and returned by ss_surface_free (avoids cudaMalloc/cudaFree per frame,
    // the analogue of the reference's ReconstructionWorkspace, workspace.rs:12-79)
    DevBuf o_verts, o_tris, o_vkeys, o_rho, o_verts2, o_vkeys2, o_normals;
    uint64_t hint_nv = 0, hint_nt = 0, hint_bc = 0;
    uint64_t frame = 0;              // serial of the last call that rewrote the scratch
    PostScratch post;
};

#include <mutex>
#include <set>
static std::mutex g_ctx_mutex;
static std::set<ss_context *> g_live_contexts;

struct ss_surface {
    ss_context *owner = nullptr;
    int device = 0;
    uint64_t n_in = 0, n = 0, nv = 0, nt = 0, nsub = 0;
    int used_decomposition = 0;
    HostGrid grid{}, subgrid{};
    int S = 0;
    DevBuf verts, tris, vkeys, rho, normals, nbr_off, nbr_idx;
    DevBuf weights, adj_row, adj_idx, inc_row, inc_idx;      // post-processing: smoothing weights, vertex->vertex / vertex->triangle CSR
    DevBuf an_xbar, an_mat, an_fac;                         // anisotropic reconstruction: centres, matrices, factors per particle
    int aniso = 0;
    float an_ms[2] = { 0.f, 0.f };                          // anisotropic stages (ss_surface_anisotropy_stats)
    uint32_t an_sweeps = 0;
    int has_normals = 0, has_neighbors = 0, has_weights = 0, has_adj = 0, has_inc = 0;
    uint64_t frame = 0;              // ss_context::frame of the reconstruction that produced this surface
    uint64_t n_neighbors = 0;
    std::vector<uint8_t> inside_aabb;
    std::vector<int64_t> sub_flat; std::vector<uint64_t> sub_count; std::vector<uint8_t> sub_sparse, sub_owned;
    uint64_t max_particles = 0;
    std::vector<float> tile;
    ss_timings tm{};
};

// ------------------------------------------------------------------ host grid math (exact f32) ----
// All expressions are single roundings in the order the reference evaluates them; `volatile` stores stop the
// host compiler from keeping excess precision or contracting (the TU is also built with -ffp-contract=off).
static inline float fmulr(float a, float b) { volatile float r = a * b; return r; }
static inline float faddr(float a, float b) { volatile float r = a + b; return r; }
static inline float fsubr(float a, float b) { volatile float r = a - b; return r; }
static inline float fdivr(float a, float b) { volatile float r = a / b; return r; }

static int grid_new(HostGrid &g, const float mn[3], const int64_t nc[3], float cell) {       // uniform_grid.rs:204-232
    for (int d = 0; d < 3; ++d) {
        g.mn[d] = mn[d]; g.nc[d] = nc[d]; g.np[d] = nc[d] + 1;
        g.mx[d] = faddr(mn[d], fmulr(cell, (float)nc[d]));
        if (!std::isfinite(g.mx[d])) return SS_ERR_REAL_TOO_SMALL;
    }
    g.cell = cell;
    return SS_OK;
}
static int grid_from_aabb(HostGrid &g, const float mn[3], const float mx[3], float cell) {   // uniform_grid.rs:175-201
    if (!(cell > 0.0f)) return SS_ERR_INVALID_CELL_SIZE;
    if (mn[0] == mx[0] && mn[1] == mx[1] && mn[2] == mx[2]) return SS_ERR_DEGENERATE_AABB;
    for (int d = 0; d < 3; ++d) if (!(mn[d] <= mx[d])) return SS_ERR_INCONSISTENT_AABB;
    float amin[3]; int64_t nc[3];
    for (int d = 0; d < 3; ++d) {
        amin[d] = fmulr(floorf(fdivr(mn[d], cell)), cell);
        float ncr = ceilf(fdivr(fsubr(mx[d], amin[d]), cell));
        if (!(ncr < 9.0e18f)) return SS_ERR_INDEX_TOO_SMALL;
        int64_t n = (int64_t)ncr;
        nc[d] = n > 1 ? n : 1;
    }
    return grid_new(g, amin, nc, cell);
}
static void grid_to_abi(const HostGrid &g, ss_grid_f32 *o) {
    for (int d = 0; d < 3; ++d) { o->aabb_min[d] = g.mn[d]; o->aabb_max[d] = g.mx[d]; o->points_per_dim[d] = g.np[d]; o->cells_per_dim[d] = g.nc[d]; }
    o->cell_size = g.cell;
}

static int validate_params(const ss_params_f32 *p) {
    if (!p) return ss_fail(SS_ERR_INVALID_PARAMETER, "params is NULL");
    if (!(p->cube_size > 0.0f)) return ss_fail(SS_ERR_INVALID_CELL_SIZE, "invalid cell size supplied, cell size has to be larger than zero");
    if (!(p->compact_support_radius > 0.0f)) return ss_fail(SS_ERR_INVALID_PARAMETER, "compact support radius has to be positive (search radius for neighborhood search has to be positive)");
    if (!(p->particle_radius > 0.0f)) return ss_fail(SS_ERR_INVALID_PARAMETER, "particle radius has to be positive");
    if (p->spatial_decomposition == 1 && p->subdomain_num_cubes_per_dim < 1) return ss_fail(SS_ERR_INVALID_PARAMETER, "subdomain_num_cubes_per_dim has to be >= 1");
    return SS_OK;
}

// ------------------------------------------------------------------ small launch helpers ----
static inline unsigned nblk(uint64_t n, unsigned t) { return (unsigned)((n + t - 1) / t); }
#ifndef SS_LAUNCH
#define SS_LAUNCH(kern, grid, block, stream, ...) kern<<<(grid), (block), 0, (stream)>>>(__VA_ARGS__)
#endif
#define LAUNCH(ctx, kern, grid, block, ...) do { SS_LAUNCH(kern, grid, block, (ctx)->stream, __VA_ARGS__); (ctx)->launches++; } while (0)
#ifndef SS_LAUNCH_DYN
#define SS_LAUNCH_DYN(kern, grid, block, smem, stream, ...) kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif
#define LAUNCH_DYN(ctx, kern, grid, block, smem, ...) do { SS_LAUNCH_DYN(kern, grid, block, smem, (ctx)->stream, __VA_ARGS__); (ctx)->launches++; } while (0)

static void cub_sort_pairs(ss_context *c, const uint32_t *kin, uint32_t *kout, const uint32_t *vin, uint32_t *vout,
                           uint32_t n, int end_bit) {
    size_t tmp = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, kin, kout, vin, vout, (int)n, 0, end_bit, c->stream));
    c->cub_tmp.ensure(tmp);
    CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, tmp, kin, kout, vin, vout, (int)n, 0, end_bit, c->stream));
    c->launches += 1 + (uint64_t)((end_bit + 7) / 8) * 2;   // upsweep/onesweep histogram + per-digit passes (approx.)
}
static void cub_excl_scan(ss_context *c, const uint32_t *in, uint32_t *out, uint32_t n) {
    size_t tmp = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, in, out, (int)n, c->stream));
    c->cub_tmp.ensure(tmp);
    CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp, in, out, (int)n, c->stream));
    c->launches += 2;
}
static void cub_incl_scan(ss_context *c, const uint32_t *in, uint32_t *out, uint32_t n) {
    size_t tmp = 0;
    CK(cub::DeviceScan::InclusiveSum(nullptr, tmp, in, out, (int)n, c->stream));
    c->cub_tmp.ensure(tmp);
    CK(cub::DeviceScan::InclusiveSum(c->cub_tmp.p, tmp, in, out, (int)n, c->stream));
    c->launches += 2;
}
static int bits_for(uint64_t maxval) { int b = 1; while (b < 64 && (maxval >> b)) ++b; return b; }

// ------------------------------------------------------------------ context ----
extern "C" int ss_abi_version(void) { return SS_ABI_VERSION; }
extern "C" const char *ss_last_error(void) { return g_last_error.c_str(); }

extern "C" int ss_context_create(int device, ss_context **out) {
    if (!out) return ss_fail(SS_ERR_INVALID_PARAMETER, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return ss_fail(SS_ERR_NO_DEVICE, std::string("no CUDA device available (") + cudaGetErrorString(e) + "); this library has no CPU path");
    try {
        if (device < 0) CK(cudaGetDevice(&device));
        if (device >= ndev) return ss_fail(SS_ERR_INVALID_PARAMETER, "device index out of range");
        CK(cudaSetDevice(device));
        ss_context *c = new ss_context();
        c->device = device;
        CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
#ifndef SS_HOST_EMUL
        CK(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
#else
        c->sm_count = 3;
#endif
        for (auto &ev : c->ev) CK(cudaEventCreate(&ev));
        for (auto &ev : c->ev_stage) CK(cudaEventCreate(&ev));
        {
            signed char table[256][16];
            ss_mc_unpack(table);
            CK(cudaMemcpyToSymbol(c_tri_table, table, sizeof(table)));
        }
        CK(cudaMemcpyToSymbol(c_num_tris, SS_MC_NUM_TRIS, sizeof(SS_MC_NUM_TRIS)));
        { std::lock_guard<std::mutex> lk(g_ctx_mutex); g_live_contexts.insert(c); }
        *out = c;
        return SS_OK;
    } catch (const SsCudaError &err) {
        return ss_fail(SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}

extern "C" void ss_context_destroy(ss_context *c) {
    if (!c) return;
    { std::lock_guard<std::mutex> lk(g_ctx_mutex); g_live_contexts.erase(c); }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    DevBuf *bufs[] = { &c->xyz, &c->xyz_f, &c->filt_flag, &c->filt_flag32, &c->filt_off, &c->aabb, &c->cnt, &c->off, &c->key_a, &c->key_b,
                       &c->val_a, &c->val_b, &c->cid, &c->cub_tmp, &c->sub_flat, &c->sub_off, &c->sub_sparse, &c->sub_owned, &c->gkey_a, &c->gkey_b, &c->gval_a, &c->gval_b, &c->flags, &c->scan,
                       &c->spos, &c->rho, &c->tab_a, &c->tab_b, &c->rec, &c->ksplit, &c->batch_subs, &c->tiles, &c->vcnt, &c->tcnt,
                       &c->vmask, &c->voff, &c->vblk_off, &c->tblk_off, &c->tile_tab, &c->brick_rng, &c->bstate, &c->flag_ls, &c->off_ls, &c->list_ls, &c->flag_mc, &c->flag_fix, &c->off_mc, &c->off_fix, &c->list_mc, &c->list_fix, &c->wflag, &c->wstate, &c->desc_ls, &c->dflag, &c->doff, &c->dlist, &c->fallback, &c->fallback2, &c->fallback3, &c->pack_cnt, &c->pack_off, &c->brick_seen, &c->fix_list, &c->nflag, &c->bkeys_a, &c->bkeys_b, &c->bids_a, &c->bids_b, &c->bcount, &c->remap, &c->keep, &c->newid,
                       &c->err, &c->pairs, &c->o_verts, &c->o_tris, &c->o_vkeys, &c->o_rho, &c->o_verts2, &c->o_vkeys2, &c->o_normals,
                       &c->an_key_a, &c->an_key_b, &c->an_val_a, &c->an_val_b, &c->an_flags, &c->an_scan, &c->an_cid, &c->an_sub_flat, &c->an_sub_off,
                       &c->an_tab_a, &c->an_tab_b, &c->an_rec, &c->an_ksplit, &c->an_am, &c->an_sweeps, &c->o_an_xbar, &c->o_an_mat, &c->o_an_fac };
    for (DevBuf *b : bufs) b->release();
    c->post.release_all();
    for (auto &ev : c->ev) cudaEventDestroy(ev);
    for (auto &ev : c->ev_stage) if (ev) cudaEventDestroy(ev);
    for (auto &ev : c->ev_an) if (ev) cudaEventDestroy(ev);
    for (auto &h : c->h_stage) if (h) cudaFreeHost(h);
    cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int ss_context_keep_levelset_tile(ss_context *c, int64_t flat) { if (!c) return SS_ERR_INVALID_PARAMETER; c->keep_tile_flat = flat; return SS_OK; }
extern "C" int ss_context_set_tile_batch(ss_context *c, uint32_t m) { if (!c) return SS_ERR_INVALID_PARAMETER; c->max_tiles = m; return SS_OK; }
extern "C" int ss_context_set_levelset_exact_everywhere(ss_context *c, int on) { if (!c) return SS_ERR_INVALID_PARAMETER; c->ls_exact_all = on ? 1 : 0; return SS_OK; }
extern "C" int ss_context_set_density_variant(ss_context *c, int v) {
    if (!c || v < 0 || v > 2) return ss_fail(SS_ERR_INVALID_PARAMETER, "density variant must be 0, 1 or 2");
    c->density_variant = v; return SS_OK;
}
extern "C" int ss_context_set_copy_chunk_bytes(ss_context *c, uint64_t bytes) {
    if (!c || bytes < 4096 || bytes > ((uint64_t)32 << 20) || (bytes & 3)) return ss_fail(SS_ERR_INVALID_PARAMETER, "copy chunk must be 4 KiB .. 32 MiB, a multiple of 4");
    c->stage_bytes = (size_t)bytes; return SS_OK;
}
extern "C" int ss_context_set_mc_variant(ss_context *c, int v) {
    if (!c || v < 0 || v > 1) return ss_fail(SS_ERR_INVALID_PARAMETER, "marching-cubes variant must be 0 or 1");
    c->mc_variant = v; return SS_OK;
}
extern "C" int ss_context_set_levelset_variant(ss_context *c, int v) {
    if (!c || v < 0 || v > 2) return ss_fail(SS_ERR_INVALID_PARAMETER, "level-set variant must be 0, 1 or 2");
    c->ls_variant = v; return SS_OK;
}
extern "C" int ss_context_set_compute_sph_normals(ss_context *c, int on) { if (!c) return SS_ERR_INVALID_PARAMETER; c->sph_normals = on ? 1 : 0; return SS_OK; }
extern "C" int ss_surface_copy_normals(const ss_surface *s, float *dst) {
    if (!s || !dst) return SS_ERR_INVALID_PARAMETER;
    if (!s->has_normals) return ss_fail(SS_ERR_INVALID_PARAMETER, "normals were not computed (ss_context_set_compute_sph_normals)");
    cudaSetDevice(s->device);
    cudaError_t e = cudaMemcpy(dst, s->normals.p, s->nv * 12, cudaMemcpyDeviceToHost);
    return e == cudaSuccess ? SS_OK : ss_fail(SS_ERR_CUDA, cudaGetErrorString(e));
}
extern "C" const float *ss_surface_device_normals(const ss_surface *s) { return (s && s->has_normals) ? s->normals.as<float>() : nullptr; }
extern "C" int ss_context_set_count_pairs(ss_context *c, int on) { if (!c) return SS_ERR_INVALID_PARAMETER; c->count_pairs = on ? 1 : 0; return SS_OK; }
extern "C" int ss_context_set_anisotropy_f32(ss_context *c, const ss_anisotropy_f32 *a) {
    if (!c) return ss_fail(SS_ERR_INVALID_PARAMETER, "context is NULL");
    if (!a) { c->aniso = 0; return SS_OK; }
    if (!(a->max_ratio >= 1.0f) || !(a->max_ratio < INFINITY)) return ss_fail(SS_ERR_INVALID_PARAMETER, "anisotropy max_ratio must be a finite number >= 1");
    if (!(a->smoothing >= 0.0f && a->smoothing <= 1.0f)) return ss_fail(SS_ERR_INVALID_PARAMETER, "anisotropy smoothing must lie in [0, 1]");
    c->aniso = 1; c->aniso_k.max_ratio = a->max_ratio; c->aniso_k.min_neighbors = a->min_neighbors; c->aniso_k.smoothing = a->smoothing;
    return SS_OK;
}
extern "C" int ss_surface_copy_anisotropy_f32(const ss_surface *s, float *centers, float *matrices, float *factors) {
    if (!s) return ss_fail(SS_ERR_INVALID_PARAMETER, "surface is NULL");
    if (!s->aniso) return ss_fail(SS_ERR_INVALID_PARAMETER, "not an anisotropic reconstruction (ss_context_set_anisotropy_f32)");
    if (!s->n) return SS_OK;
    cudaSetDevice(s->device);
    const void *src[3] = { s->an_xbar.p, s->an_mat.p, s->an_fac.p };
    void *dst[3] = { centers, matrices, factors };
    const size_t bytes[3] = { s->n * 12, s->n * 24, s->n * 4 };
    for (int q = 0; q < 3; ++q) if (dst[q]) {
        cudaError_t e = cudaMemcpy(dst[q], src[q], bytes[q], cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return ss_fail(SS_ERR_CUDA, cudaGetErrorString(e));
    }
    return SS_OK;
}
extern "C" int ss_surface_anisotropy_stats(const ss_surface *s, float *ms2, uint32_t *max_jacobi_sweeps) {
    if (!s) return ss_fail(SS_ERR_INVALID_PARAMETER, "surface is NULL");
    if (ms2) { ms2[0] = s->an_ms[0]; ms2[1] = s->an_ms[1]; }
    if (max_jacobi_sweeps) *max_jacobi_sweeps = s->an_sweeps;
    return SS_OK;
}

// ------------------------------------------------------------------ stage: input, filter, AABB, grid ----
struct Prepared {
    const float *d_xyz = nullptr;   // filtered particles on device
    uint64_t n = 0;
    HostGrid grid{};
    float upload_ms = 0.f;
};

// Result copies device -> host.  A plain cudaMemcpy into PAGEABLE memory is staged by the driver and, into freshly allocated arrays
// (what a numpy front end hands in), page-faults single-threaded: ~3 GB/s measured for the 2.5 GB of a 50 M-particle result.  Large
// copies therefore go through two page-locked staging buffers at PCIe speed, and a few host threads scatter each chunk into the
// destination (parallel first touch) while the next chunk is in flight; `widen` turns u32 triangle indices into the reference's
// usize on the way (half the PCIe bytes of converting on the device).  Destinations that are page-locked already take one cudaMemcpy.
#include <thread>
#define SS_STAGE_BYTES_MAX ((size_t)32 << 20)
#define SS_STAGE_THREADS 8
static void scatter_chunk(char *dst, const char *stage, size_t n_src_bytes, bool widen) {
    const size_t nthreads = n_src_bytes >= ((size_t)1 << 20) ? SS_STAGE_THREADS : 1;
    auto work = [&](size_t t) {
        const size_t per = ((n_src_bytes / 4 + nthreads - 1) / nthreads) * 4;           // multiples of one 4-byte element
        const size_t lo = std::min(n_src_bytes, t * per), hi = std::min(n_src_bytes, lo + per);
        if (!widen) { memcpy(dst + lo, stage + lo, hi - lo); return; }
        const uint32_t *in = reinterpret_cast<const uint32_t *>(stage + lo);
        uint64_t *out = reinterpret_cast<uint64_t *>(dst) + lo / 4;
        for (size_t e = 0; e < (hi - lo) / 4; ++e) out[e] = in[e];
    };
    if (nthreads == 1) { work(0); return; }
    std::thread th[SS_STAGE_THREADS];
    for (size_t t = 1; t < nthreads; ++t) th[t] = std::thread(work, t);
    work(0);
    for (size_t t = 1; t < nthreads; ++t) th[t].join();
}
// The same staging for the upload of a large PAGEABLE particle array (a numpy array handed to the front end): host threads gather a
// chunk into a page-locked buffer while the previous chunk travels; page-locked inputs take one asynchronous copy.
static void upload_particles(ss_context *c, void *dst_dev, const void *src, size_t bytes, bool pinned_src) {
    const size_t chunk = c->stage_bytes;
    if (pinned_src || bytes < 4 * chunk) { CK(cudaMemcpyAsync(dst_dev, src, bytes, cudaMemcpyHostToDevice, c->stream)); return; }
    for (int q = 0; q < 2; ++q) if (!c->h_stage[q]) {
        if (cudaHostAlloc(&c->h_stage[q], SS_STAGE_BYTES_MAX, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); c->h_stage[q] = nullptr; }
    }
    if (!c->h_stage[0] || !c->h_stage[1]) { CK(cudaMemcpyAsync(dst_dev, src, bytes, cudaMemcpyHostToDevice, c->stream)); return; }
    const size_t nchunks = (bytes + chunk - 1) / chunk;
    for (size_t k = 0; k < nchunks; ++k) {
        const size_t off = k * chunk, n = std::min(chunk, bytes - off);
        if (k >= 2) CK(cudaEventSynchronize(c->ev_stage[k & 1]));     // the copy that last read this staging buffer is done
        scatter_chunk(static_cast<char *>(c->h_stage[k & 1]), static_cast<const char *>(src) + off, n, false);
        CK(cudaMemcpyAsync(static_cast<char *>(dst_dev) + off, c->h_stage[k & 1], n, cudaMemcpyHostToDevice, c->stream));
        CK(cudaEventRecord(c->ev_stage[k & 1], c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));                             // the staging buffers are free again when this returns
}

static int prepare_particles(ss_context *c, const float *xyz, uint64_t n_in, const ss_params_f32 *p, Prepared &P,
                             std::vector<uint8_t> *inside_out, const ss_grid_f32 *given_grid = nullptr) {
    if (n_in > 0xfffffff0ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "more than 2^32 particles are not supported by one device");
    const float *d_in = nullptr;
    cudaPointerAttributes attr{};
    bool on_device = false;
    bool pinned_host = false;
    if (xyz && n_in) {
        cudaError_t e = cudaPointerGetAttributes(&attr, xyz);
        if (e == cudaSuccess && (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged)) on_device = true;
        else if (e == cudaSuccess && attr.type == cudaMemoryTypeHost) pinned_host = true;
        else cudaGetLastError();
    }
    CK(cudaEventRecord(c->ev[0], c->stream));
    if (on_device) d_in = xyz;
    else if (n_in) {
        c->xyz.ensure(n_in * 12);
        upload_particles(c, c->xyz.p, xyz, n_in * 12, pinned_host);
        d_in = c->xyz.as<float>();
    }
    CK(cudaEventRecord(c->ev[1], c->stream));
    P.d_xyz = d_in; P.n = n_in;
    // particle AABB filter, lib.rs:369-406
    if (p->has_particle_aabb && n_in) {
        c->filt_flag.ensure(n_in); c->filt_flag32.ensure(n_in * 4); c->filt_off.ensure(n_in * 4 + 4);
        float3 mn = make_float3(p->particle_aabb_min[0], p->particle_aabb_min[1], p->particle_aabb_min[2]);
        float3 mx = make_float3(p->particle_aabb_max[0], p->particle_aabb_max[1], p->particle_aabb_max[2]);
        LAUNCH(c, k_filter_flags, nblk(n_in, 256), 256, d_in, n_in, mn, mx, c->filt_flag.as<uint8_t>(), c->filt_flag32.as<uint32_t>());
        cub_excl_scan(c, c->filt_flag32.as<uint32_t>(), c->filt_off.as<uint32_t>(), (uint32_t)n_in);
        uint32_t last_off = 0, last_flag = 0;
        CK(cudaMemcpyAsync(&last_off, c->filt_off.as<uint32_t>() + (n_in - 1), 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaMemcpyAsync(&last_flag, c->filt_flag32.as<uint32_t>() + (n_in - 1), 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        uint64_t nf = (uint64_t)last_off + last_flag;
        c->xyz_f.ensure(std::max<uint64_t>(nf, 1) * 12);
        LAUNCH(c, k_filter_scatter, nblk(n_in, 256), 256, d_in, n_in, c->filt_flag.as<uint8_t>(), c->filt_off.as<uint32_t>(), c->xyz_f.as<float>());
        P.d_xyz = c->xyz_f.as<float>(); P.n = nf;
        if (inside_out) {
            inside_out->resize(n_in);
            CK(cudaMemcpyAsync(inside_out->data(), c->filt_flag.p, n_in, cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
        }
    } else if (p->has_particle_aabb && inside_out) inside_out->clear();

    if (given_grid) {   // partitioned run: the grid of ALL particles was computed by the caller
        for (int d = 0; d < 3; ++d) { P.grid.mn[d] = given_grid->aabb_min[d]; P.grid.mx[d] = given_grid->aabb_max[d]; P.grid.np[d] = given_grid->points_per_dim[d]; P.grid.nc[d] = given_grid->cells_per_dim[d]; }
        P.grid.cell = given_grid->cell_size;
        return SS_OK;
    }
    // grid_for_reconstruction, lib.rs:476-516
    float mn[3], mx[3];
    if (p->has_particle_aabb) {
        for (int d = 0; d < 3; ++d) { mn[d] = p->particle_aabb_min[d]; mx[d] = p->particle_aabb_max[d]; }
    } else {
        if (P.n == 0) { for (int d = 0; d < 3; ++d) mn[d] = mx[d] = 0.0f; }   // Aabb3d::zeros(), aabb.rs:29-30
        else {
            c->aabb.ensure(6 * sizeof(int));
            int init[6] = { INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN };
            CK(cudaMemcpyAsync(c->aabb.p, init, sizeof(init), cudaMemcpyHostToDevice, c->stream));
            unsigned blocks = std::min<uint64_t>(nblk(P.n, 256), 148 * 16);
            LAUNCH(c, k_aabb, blocks, 256, P.d_xyz, P.n, c->aabb.as<int>());
            int res[6];
            CK(cudaMemcpyAsync(res, c->aabb.p, sizeof(res), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            for (int d = 0; d < 3; ++d) { mn[d] = ss_ord2f(res[d]); mx[d] = ss_ord2f(res[3 + d]); }
        }
        for (int d = 0; d < 3; ++d) { mn[d] = fsubr(mn[d], p->particle_radius); mx[d] = faddr(mx[d], p->particle_radius); }
    }
    // compute_kernel_evaluation_radius, density_map.rs:551-580
    float half_cells = ceilf(fdivr(p->compact_support_radius, p->cube_size));
    float margin = fmulr(fmulr(p->cube_size, half_cells), faddr(1.0f, sqrtf(FLT_EPSILON)));
    for (int d = 0; d < 3; ++d) { mn[d] = fsubr(mn[d], margin); mx[d] = faddr(mx[d], margin); }
    int rc = grid_from_aabb(P.grid, mn, mx, p->cube_size);
    if (rc != SS_OK) return ss_fail(rc, rc == SS_ERR_DEGENERATE_AABB ? "degenerate AABB supplied, every dimension of the AABB has to have non-zero extents"
                                        : rc == SS_ERR_INCONSISTENT_AABB ? "inconsistent AABB supplied" : "grid construction failed");
    return SS_OK;
}

extern "C" int ss_grid_for_reconstruction_f32(ss_context *c, const float *xyz, uint64_t n, const ss_params_f32 *p, ss_grid_f32 *out) {
    if (!c || !out) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    int rc = validate_params(p);
    if (rc) return rc;
    try {
        CK(cudaSetDevice(c->device));
        Prepared P;
        rc = prepare_particles(c, xyz, n, p, P, nullptr);
        if (rc) return rc;
        grid_to_abi(P.grid, out);
        return SS_OK;
    } catch (const SsCudaError &err) {
        return ss_fail(err.e == cudaErrorMemoryAllocation ? SS_ERR_OUT_OF_MEMORY : SS_ERR_CUDA,
                       std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}


// ------------------------------------------------------------------ templated launch helpers ----
static void launch_levelset(ss_context *c, dim3 grid, const SsDev &D, const SsLsArgs &A, bool count, bool global) {
    void (*kern)(SsDev, SsLsArgs) = global ? (count ? k_levelset<true, true> : k_levelset<false, true>)
                                           : (count ? k_levelset<true, false> : k_levelset<false, false>);
    LAUNCH(c, kern, grid, SS_LS_THREADS, D, A);
}

// in-place exclusive scan of the per-particle neighbour counts (n + 1 entries, last = 0) -> CSR offsets; returns the total
static uint64_t scan_neighbor_counts(ss_context *c, unsigned long long *cnt, uint64_t n) {
    size_t tmp = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp, cnt, cnt, (int)(n + 1), c->stream));
    c->cub_tmp.ensure(tmp);
    CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, tmp, cnt, cnt, (int)(n + 1), c->stream));
    c->launches += 2;
    unsigned long long total = 0;
    CK(cudaMemcpyAsync(&total, cnt + n, 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return total;
}

// Work list of non-empty bricks for the level-set launch (k_brick_worklist + scan + compaction); returns its length.
static uint32_t build_worklist(ss_context *c, const SsDev &D, uint32_t ntiles) {
    const uint32_t nbr = ntiles * (uint32_t)(D.nb * D.nb * D.nb);
    c->flag_ls.ensure((size_t)nbr * 4); c->off_ls.ensure((size_t)nbr * 4 + 4); c->list_ls.ensure((size_t)nbr * 4);
    LAUNCH(c, k_brick_worklist, nblk(nbr, 256), 256, D, c->tile_tab.as<SsTile>(), c->brick_rng.as<int2>(), c->tab_a.as<uint32_t>(), ntiles, c->flag_ls.as<uint32_t>());
    cub_excl_scan(c, c->flag_ls.as<uint32_t>(), c->off_ls.as<uint32_t>(), nbr);
    LAUNCH(c, k_compact_list, nblk(nbr, 256), 256, c->flag_ls.as<uint32_t>(), c->off_ls.as<uint32_t>(), nbr, c->list_ls.as<uint32_t>());
    uint32_t lc[2] = { 0, 0 };
    CK(cudaMemcpyAsync(&lc[0], c->off_ls.as<uint32_t>() + (nbr - 1), 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&lc[1], c->flag_ls.as<uint32_t>() + (nbr - 1), 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return lc[0] + lc[1];
}

// kernel.rs:327-336 (AVX-path constants) and :61-66 (scalar normalisation), evaluated in f32 like the reference
static void fill_kernel_consts(SsDev &D, float h) {
    D.a_hinv = fdivr(1.0f, h);
    float rrr = fmulr(fmulr(h, h), h);
    D.a_sigma = fdivr(8.0f, fmulr(SS_PI_F, rrr));
    D.a_s2 = fmulr(2.0f, D.a_sigma); D.a_s6 = fmulr(6.0f, D.a_sigma); D.a_s12 = fmulr(12.0f, D.a_sigma);
    D.s_sigma = fdivr(8.0f, rrr);
    D.s_c_inner = fdivr(3.0f, fmulr(2.0f, SS_PI_F));
    D.s_c_outer = fdivr(1.0f, fmulr(4.0f, SS_PI_F));
    D.s_two_thirds = fdivr(2.0f, 3.0f);
}
// splat bins: cubes of `be` cells; a brick (8 points) gathers the bins overlapping [8b - R, 8b + 7 + R)
static void fill_bins(SsDev &D, float cs) {
    D.nb = (D.np + 7) / 8;
    D.ext_bricks = (D.nb >= 2 && D.np == 8 * (D.nb - 1) + 1) ? 1 : 0;
    D.be = 8 * std::max(1, (7 + 2 * D.R + 39) / 40);
    D.nlo = (D.R + D.be - 1) / D.be;
    D.nbin = ss_floor_div(D.S + D.R, D.be) + D.nlo + 1;
    D.nbin_sub = D.nbin * D.nbin * D.nbin;
    D.inv_c = (float)(1.0 / (double)cs);
    D.rr_cells = (float)D.R + 0.01f;
}

// ------------------------------------------------------------------ the subdomain-grid pipeline ----
struct Partition {
    int enabled = 0;
    int axis = 0;
    int64_t own_lo = 0, own_hi = 0;     // owned subdomain index range along `axis`
    int64_t halo = 0;                   // extra subdomain layers kept for densities only
    uint64_t global_max_particles = 0;  // max particles per subdomain over ALL ranks (0: use the local maximum)
    int stop_after_decomposition = 0;   // only report the local maximum (out->max_particles)
    uint64_t (*max_reduce)(uint64_t local_max, void *user) = nullptr;   // all-reduce(MAX) of the local maximum across ranks
    void *max_reduce_user = nullptr;
    // SphInterpolator entry (ss_sph_interpolator_create_f32): densities supplied by the caller; stop after the particle bins are built
    const float *given_rho = nullptr;
    float given_mass = 0.0f;
};

// SPH densities (and optional CSR neighbour lists) of the filtered particles: per-subdomain cell lists on the h-lattice with
// ordered neighbour sums (dense_subdomains.rs:496-646), or one cell list over the whole domain in global mode.
static int stage_densities(ss_context *c, const SsDev &D, const float *d_xyz, uint64_t n, uint32_t M, uint32_t nsub, uint64_t g_ns_cells,
                           bool global_mode, bool want_nbrs, ss_surface *out, float *d_rho) {
    cudaStream_t st = c->stream;
    if ((uint64_t)nsub * (uint64_t)D.ns_stride >= 0xffffffffull || (uint64_t)nsub * (uint64_t)D.nbin_sub >= 0xffffffffull)
        return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many non-empty subdomains for 32-bit cell keys");
    c->err.ensure(4);
    CK(cudaMemsetAsync(c->err.p, 0, 4, st));
    // membership arrays: cid (compressed subdomain), val_b (particle); keys -> key_a, sorted -> key_b? key_b is in use
    // (flat ids are no longer needed after cid): reuse key_b as sort output, val_a as sorted payload.
    if (!global_mode) {
    LAUNCH(c, k_ns_keys, nblk(M, 256), 256, D, d_xyz, M, c->cid.as<uint32_t>(), c->sub_flat.as<uint32_t>(), c->val_b.as<uint32_t>(),
           c->key_a.as<uint32_t>(), c->err.as<int>());
    const uint64_t ns_keys = (uint64_t)nsub * D.ns_stride;
    cub_sort_pairs(c, c->key_a.as<uint32_t>(), c->key_b.as<uint32_t>(), c->val_b.as<uint32_t>(), c->val_a.as<uint32_t>(), M, bits_for(ns_keys));
    c->tab_a.ensure(ns_keys * 4); c->tab_b.ensure(ns_keys * 4);
    CK(cudaMemsetAsync(c->tab_a.p, 0xff, ns_keys * 4, st));
    LAUNCH(c, k_mark_starts, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->tab_a.as<uint32_t>(), (uint32_t)ns_keys);
    LAUNCH(c, k_run_counts, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->tab_b.as<uint32_t>(), (uint32_t)ns_keys);
    c->spos.ensure((size_t)M * 16);
    LAUNCH(c, k_gather_pos, nblk(M, 256), 256, d_xyz, c->val_a.as<uint32_t>(), M, c->spos.as<float4>());
    unsigned long long *d_ncnt = nullptr;
    if (want_nbrs) { out->nbr_off.ensure((n + 1) * 8); d_ncnt = out->nbr_off.as<unsigned long long>(); CK(cudaMemsetAsync(d_ncnt, 0, (n + 1) * 8, st)); }
    // entries with the particle inside the subdomain (every particle is inside at most one: <= n of them), compacted
    c->dflag.ensure((size_t)M * 4); c->doff.ensure((size_t)M * 4 + 4); c->dlist.ensure(std::max<uint64_t>(n, 1) * 4);
    if (c->density_variant >= 1 && !want_nbrs) {
        // cell-cooperative kernel (ss_density.cuh): one warp per h-cell that holds a particle inside its subdomain (<= n cells), persistent grid
        LAUNCH(c, k_density_cell_flags, nblk(M, 256), 256, D, M, c->key_b.as<uint32_t>(), c->spos.as<float4>(), c->sub_flat.as<uint32_t>(),
               c->tab_b.as<uint32_t>(), c->dflag.as<uint32_t>());
        cub_excl_scan(c, c->dflag.as<uint32_t>(), c->doff.as<uint32_t>(), M);
        LAUNCH(c, k_compact_list, nblk(M, 256), 256, c->dflag.as<uint32_t>(), c->doff.as<uint32_t>(), M, c->dlist.as<uint32_t>());
        SsDcArgs DA{};
        DA.m = M; DA.list = c->dlist.as<uint32_t>(); DA.list_off = c->doff.as<uint32_t>(); DA.list_flag = c->dflag.as<uint32_t>();
        DA.key = c->key_b.as<uint32_t>(); DA.spos = c->spos.as<float4>(); DA.sub_flat = c->sub_flat.as<uint32_t>();
        DA.cstart = c->tab_a.as<uint32_t>(); DA.cend = c->tab_b.as<uint32_t>(); DA.rho = d_rho; DA.nbr_count = nullptr;
        const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)c->sm_count * 7u, ((uint64_t)n + SS_DC_WARPS - 1) / SS_DC_WARPS);
        if (c->density_variant == 1) LAUNCH(c, k_density_cells<true>, std::max(grid, 1u), SS_DC_WARPS * 32, D, DA);
        else LAUNCH(c, k_density_cells<false>, std::max(grid, 1u), SS_DC_WARPS * 32, D, DA);
    } else {
    LAUNCH(c, k_density_flags, nblk(M, 256), 256, D, M, c->key_b.as<uint32_t>(), c->spos.as<float4>(), c->sub_flat.as<uint32_t>(), c->dflag.as<uint32_t>());
    cub_excl_scan(c, c->dflag.as<uint32_t>(), c->doff.as<uint32_t>(), M);
    LAUNCH(c, k_compact_list, nblk(M, 256), 256, c->dflag.as<uint32_t>(), c->doff.as<uint32_t>(), M, c->dlist.as<uint32_t>());
    LAUNCH(c, k_density<false>, nblk(n, 128), 128, D, M, c->dlist.as<uint32_t>(), c->doff.as<uint32_t>(), c->dflag.as<uint32_t>(),
           c->key_b.as<uint32_t>(), c->spos.as<float4>(), c->sub_flat.as<uint32_t>(),
           c->tab_a.as<uint32_t>(), c->tab_b.as<uint32_t>(), d_rho, d_ncnt, (const unsigned long long *)nullptr, (uint32_t *)nullptr);
    }
    if (want_nbrs) {
        const uint64_t total = scan_neighbor_counts(c, d_ncnt, n);
        out->nbr_idx.ensure(std::max<uint64_t>(total, 1) * 4);
        LAUNCH(c, k_density<true>, nblk(n, 128), 128, D, M, c->dlist.as<uint32_t>(), c->doff.as<uint32_t>(), c->dflag.as<uint32_t>(),
               c->key_b.as<uint32_t>(), c->spos.as<float4>(), c->sub_flat.as<uint32_t>(),
               c->tab_a.as<uint32_t>(), c->tab_b.as<uint32_t>(), d_rho, (unsigned long long *)nullptr, (const unsigned long long *)d_ncnt, out->nbr_idx.as<uint32_t>());
        out->has_neighbors = 1; out->n_neighbors = total;
    }
    } else {
        // one cell list over the whole domain; particles (not memberships) are the entries
        const uint32_t n32 = (uint32_t)n;
        c->gkey_a.ensure((size_t)n32 * 4); c->gkey_b.ensure((size_t)n32 * 4); c->gval_a.ensure((size_t)n32 * 4); c->gval_b.ensure((size_t)n32 * 4);
        LAUNCH(c, k_ns_keys_global, nblk(n32, 256), 256, D, d_xyz, n32, c->gkey_a.as<uint32_t>(), c->gval_a.as<uint32_t>(), c->err.as<int>());
        cub_sort_pairs(c, c->gkey_a.as<uint32_t>(), c->gkey_b.as<uint32_t>(), c->gval_a.as<uint32_t>(), c->gval_b.as<uint32_t>(), n32, bits_for(g_ns_cells));
        c->tab_a.ensure(g_ns_cells * 4); c->tab_b.ensure(g_ns_cells * 4);
        CK(cudaMemsetAsync(c->tab_a.p, 0xff, g_ns_cells * 4, st));
        LAUNCH(c, k_mark_starts, nblk(n32, 256), 256, c->gkey_b.as<uint32_t>(), n32, c->tab_a.as<uint32_t>(), (uint32_t)g_ns_cells);
        LAUNCH(c, k_run_counts, nblk(n32, 256), 256, c->gkey_b.as<uint32_t>(), n32, c->tab_b.as<uint32_t>(), (uint32_t)g_ns_cells);
        c->spos.ensure((size_t)n32 * 16);
        LAUNCH(c, k_gather_pos, nblk(n32, 256), 256, d_xyz, c->gval_b.as<uint32_t>(), n32, c->spos.as<float4>());
        unsigned long long *d_ncnt = nullptr;
        if (want_nbrs) { out->nbr_off.ensure((n + 1) * 8); d_ncnt = out->nbr_off.as<unsigned long long>(); CK(cudaMemsetAsync(d_ncnt, 0, (n + 1) * 8, st)); }
        LAUNCH(c, k_density_global<false>, nblk(n32, 128), 128, D, n32, c->gkey_b.as<uint32_t>(), c->spos.as<float4>(), c->tab_a.as<uint32_t>(),
               c->tab_b.as<uint32_t>(), d_rho, d_ncnt, (const unsigned long long *)nullptr, (uint32_t *)nullptr);
        if (want_nbrs) {
            const uint64_t total = scan_neighbor_counts(c, d_ncnt, n);
            out->nbr_idx.ensure(std::max<uint64_t>(total, 1) * 4);
            LAUNCH(c, k_density_global<true>, nblk(n32, 128), 128, D, n32, c->gkey_b.as<uint32_t>(), c->spos.as<float4>(), c->tab_a.as<uint32_t>(),
                   c->tab_b.as<uint32_t>(), d_rho, (unsigned long long *)nullptr, (const unsigned long long *)d_ncnt, out->nbr_idx.as<uint32_t>());
            out->has_neighbors = 1; out->n_neighbors = total;
        }
    }
    return SS_OK;
}

// Splat bins: memberships sorted by (subdomain, 8^3-point brick bin) + the particle records (x, y, z, V) the level set gathers.
// val_b still holds the membership particle indices in subdomain order (stable input for the bin sort).
static int stage_binning(ss_context *c, const SsDev &D, const float *d_xyz, const float *d_rho, uint32_t M, uint32_t nsub, bool partitioned) {
    cudaStream_t st = c->stream;
    LAUNCH(c, k_bin_keys, nblk(M, 256), 256, D, d_xyz, M, c->cid.as<uint32_t>(), c->sub_flat.as<uint32_t>(), c->val_b.as<uint32_t>(),
           partitioned ? c->sub_owned.as<uint8_t>() : nullptr, c->key_a.as<uint32_t>());
    cub_sort_pairs(c, c->key_a.as<uint32_t>(), c->key_b.as<uint32_t>(), c->val_b.as<uint32_t>(), c->val_a.as<uint32_t>(), M, 32);
    const uint64_t bin_keys = (uint64_t)nsub * D.nbin_sub;
    c->tab_a.ensure(bin_keys * 4); c->tab_b.ensure(bin_keys * 4);
    CK(cudaMemsetAsync(c->tab_a.p, 0xff, bin_keys * 4, st));
    LAUNCH(c, k_mark_starts, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->tab_a.as<uint32_t>(), (uint32_t)bin_keys);
    LAUNCH(c, k_run_counts, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->tab_b.as<uint32_t>(), (uint32_t)bin_keys);
    c->rec.ensure((size_t)M * 16); c->ksplit.ensure((size_t)M * 4);
    LAUNCH(c, k_records, nblk(M, 256), 256, D, d_xyz, d_rho, M, c->key_b.as<uint32_t>(), c->val_a.as<uint32_t>(),
           c->sub_flat.as<uint32_t>(), c->rec.as<float4>(), c->ksplit.as<int>());
    int h_err = 0;
    CK(cudaMemcpyAsync(&h_err, c->err.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(c->ev[5], st));
    CK(cudaStreamSynchronize(st));
    if (h_err) return ss_fail(SS_ERR_INVALID_PARAMETER, "particle outside of its subdomain's neighbourhood-search grid (reference: panic)");
    return SS_OK;
}


// Exact values for the flagged boxes of `n_bricks` listed bricks.  Variant 2: warp-per-brick kernel (ss_exact.cuh), bricks it
// cannot take come back in a fallback list and go through k_levelset (SS_LS_FIX) like in the other variants.
static void launch_exact(ss_context *c, const SsDev &D, const SsLsArgs &F, uint32_t n_bricks, bool global_mode, uint64_t &ls_launches) {
    if (!n_bricks) return;
    const bool count = c->count_pairs != 0;
    if (c->ls_variant != 2) { launch_levelset(c, dim3(n_bricks), D, F, count, global_mode); ++ls_launches; return; }
    cudaStream_t st = c->stream;
    c->fallback.ensure(((size_t)n_bricks + 1) * 4);
    CK(cudaMemsetAsync(c->fallback.p, 0, 4, st));
    SsXwArgs X{};
    X.bin_start = F.bin_start; X.bin_end = F.bin_end; X.rec = F.rec; X.ksplit = F.ksplit; X.pidx = F.pidx; X.tile_tab = F.tile_tab;
    X.brick_rng = F.brick_rng; X.bricks = F.fix_bricks; X.n_bricks = n_bricks; X.wflag = F.wflag; X.tiles = F.tiles;
    X.fallback = c->fallback.as<uint32_t>(); X.pairs = F.pairs;
    const unsigned grid = (n_bricks + SS_XW_WARPS - 1) / SS_XW_WARPS;
    if (global_mode) { if (count) LAUNCH(c, (k_exact_warp<true, true>), grid, SS_XW_THREADS, D, X); else LAUNCH(c, (k_exact_warp<true, false>), grid, SS_XW_THREADS, D, X); }
    else { if (count) LAUNCH(c, (k_exact_warp<false, true>), grid, SS_XW_THREADS, D, X); else LAUNCH(c, (k_exact_warp<false, false>), grid, SS_XW_THREADS, D, X); }
    ++ls_launches;
    uint32_t n_fb = 0;
    CK(cudaMemcpyAsync(&n_fb, c->fallback.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // dense clusters: the same kernel with one warp per CTA and a larger slice -- up to 1024 candidates per brick (27 KB, static;
    // list: fallback -> leftovers in fallback2), then up to 4096 (108 KB of dynamic shared memory; leftovers in fallback3)
    for (int stage = 0; stage < 2 && n_fb; ++stage) {
        DevBuf &in = stage == 0 ? c->fallback : c->fallback2, &left = stage == 0 ? c->fallback2 : c->fallback3;
        left.ensure(((size_t)n_fb + 1) * 4);
        CK(cudaMemsetAsync(left.p, 0, 4, st));
        SsXwArgs Y = X;
        Y.bricks = in.as<uint32_t>() + 1; Y.n_bricks = n_fb; Y.fallback = left.as<uint32_t>();
        if (stage == 0) {
            if (global_mode) { if (count) LAUNCH(c, (k_exact_warp_mid<true, true>), n_fb, 32, D, Y); else LAUNCH(c, (k_exact_warp_mid<true, false>), n_fb, 32, D, Y); }
            else { if (count) LAUNCH(c, (k_exact_warp_mid<false, true>), n_fb, 32, D, Y); else LAUNCH(c, (k_exact_warp_mid<false, false>), n_fb, 32, D, Y); }
        } else {
            const size_t dyn = sizeof(SsXwSliceBig);
            if (!c->big_attr_set) {
#ifndef SS_HOST_EMUL
                CK(cudaFuncSetAttribute(k_exact_warp_big<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
                CK(cudaFuncSetAttribute(k_exact_warp_big<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
                CK(cudaFuncSetAttribute(k_exact_warp_big<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
                CK(cudaFuncSetAttribute(k_exact_warp_big<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
#endif
                c->big_attr_set = 1;
            }
            if (global_mode) { if (count) LAUNCH_DYN(c, (k_exact_warp_big<true, true>), n_fb, 32, dyn, D, Y); else LAUNCH_DYN(c, (k_exact_warp_big<true, false>), n_fb, 32, dyn, D, Y); }
            else { if (count) LAUNCH_DYN(c, (k_exact_warp_big<false, true>), n_fb, 32, dyn, D, Y); else LAUNCH_DYN(c, (k_exact_warp_big<false, false>), n_fb, 32, dyn, D, Y); }
        }
        ++ls_launches;
        CK(cudaMemcpyAsync(&n_fb, left.p, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    if (n_fb) {
        // beyond 4096 candidates: k_levelset's O(C^2) selection path (extreme clustering only)
        SsLsArgs G = F;
        G.fix_bricks = c->fallback3.as<uint32_t>() + 1;
        launch_levelset(c, dim3(n_fb), D, G, count, global_mode);
        ++ls_launches;
    }
}

// Bricks that can carry surface (for marching cubes: c->list_mc, n_mc) / markers next to outside points (for the fix-up sweep:
// c->list_fix, n_fixscan), from the per-brick states the level-set kernels recorded.
static void list_bricks(ss_context *c, const SsDev &D, uint32_t nbr_b, bool zero_untouched, uint32_t &n_mc, uint32_t &n_fixscan) {
    cudaStream_t st = c->stream;
    c->flag_mc.ensure((size_t)nbr_b * 4); c->flag_fix.ensure((size_t)nbr_b * 4); c->off_mc.ensure((size_t)nbr_b * 4 + 4); c->off_fix.ensure((size_t)nbr_b * 4 + 4);
    c->list_mc.ensure((size_t)nbr_b * 4); c->list_fix.ensure((size_t)nbr_b * 4);
    LAUNCH(c, k_brick_classify, nblk(nbr_b, 256), 256, D, c->bstate.as<uint8_t>(), nbr_b, c->flag_mc.as<uint32_t>(), c->flag_fix.as<uint32_t>());
    cub_excl_scan(c, c->flag_mc.as<uint32_t>(), c->off_mc.as<uint32_t>(), nbr_b);
    cub_excl_scan(c, c->flag_fix.as<uint32_t>(), c->off_fix.as<uint32_t>(), nbr_b);
    LAUNCH(c, k_compact_list, nblk(nbr_b, 256), 256, c->flag_mc.as<uint32_t>(), c->off_mc.as<uint32_t>(), nbr_b, c->list_mc.as<uint32_t>());
    LAUNCH(c, k_compact_list, nblk(nbr_b, 256), 256, c->flag_fix.as<uint32_t>(), c->off_fix.as<uint32_t>(), nbr_b, c->list_fix.as<uint32_t>());
    if (zero_untouched)       // the tiles were not zero-filled: untouched bricks a later pass can read
        LAUNCH(c, k_zero_untouched, nblk((uint64_t)nbr_b * 32, 256), 256, D, c->bstate.as<uint8_t>(), c->flag_mc.as<uint32_t>(), c->flag_fix.as<uint32_t>(),
               nbr_b, c->tiles.as<float>());
    uint32_t lc[4] = { 0, 0, 0, 0 };
    CK(cudaMemcpyAsync(&lc[0], c->off_mc.as<uint32_t>() + (nbr_b - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&lc[1], c->flag_mc.as<uint32_t>() + (nbr_b - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&lc[2], c->off_fix.as<uint32_t>() + (nbr_b - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&lc[3], c->flag_fix.as<uint32_t>() + (nbr_b - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    n_mc = lc[0] + lc[1]; n_fixscan = lc[2] + lc[3];
}

// Level set of one batch of tiles: work list, certification + exact values (fused kernel, or variant 1: certification kernel +
// exact pass), brick classification, fix-up sweep.  Leaves the tiles, the per-brick states and the marching-cubes brick list
// (c->list_mc, *n_mc_out entries) in the context scratch.
static int levelset_batch(ss_context *c, const SsDev &D, uint32_t nbatch, unsigned nbricks, bool exact_all, int certify_runs, bool global_mode,
                          ss_surface *out, uint64_t &ls_launches, uint64_t &fix_points, uint32_t *n_mc_out) {
    cudaStream_t st = c->stream;
    SsLsArgs A{};
    A.bin_start = c->tab_a.as<uint32_t>(); A.bin_end = c->tab_b.as<uint32_t>(); A.rec = c->rec.as<float4>();
    A.ksplit = c->ksplit.as<int>(); A.pidx = c->val_a.as<uint32_t>();
    A.tile_tab = c->tile_tab.as<SsTile>(); A.brick_rng = c->brick_rng.as<int2>(); A.tiles = c->tiles.as<float>();
    A.pairs = c->count_pairs ? c->pairs.as<unsigned long long>() : nullptr;
    A.mode = exact_all ? SS_LS_EXACT_ALL : SS_LS_CERTIFY;
    A.wflag = nullptr; A.fix_bricks = nullptr; A.bstate = c->bstate.as<uint8_t>();
    const uint32_t n_work = build_worklist(c, D, nbatch);
    A.work_list = c->list_ls.as<uint32_t>();
    const bool split_certify = c->ls_variant >= 1 && !exact_all && certify_runs <= 32;
    if (n_work && !split_certify) { launch_levelset(c, dim3(n_work), D, A, c->count_pairs != 0, global_mode); ++ls_launches; }
    if (n_work && split_certify) {
        // variant 1 (ss_certify.cuh): certification kernel, then the exact pass over the boxes it could not certify
        const uint32_t nbr_c = nbatch * nbricks;
        c->wstate.ensure((size_t)nbr_c * SS_LS_WARPS); c->wflag.ensure((size_t)nbr_c * SS_LS_WARPS); c->desc_ls.ensure((size_t)n_work * 16);
        c->flag_fix.ensure((size_t)nbr_c * 4); c->off_fix.ensure((size_t)nbr_c * 4 + 4); c->fix_list.ensure((size_t)nbr_c * 4);
        CK(cudaMemsetAsync(c->wstate.p, 0, (size_t)nbr_c * SS_LS_WARPS, st));
        LAUNCH(c, k_compact_desc, nblk(nbr_c, 256), 256, D, c->flag_ls.as<uint32_t>(), c->off_ls.as<uint32_t>(), nbr_c, c->desc_ls.as<uint4>());
        SsCertArgs CA{};
        CA.bin_start = A.bin_start; CA.bin_end = A.bin_end; CA.rec = A.rec; CA.tile_tab = A.tile_tab; CA.brick_rng = A.brick_rng;
        CA.work_desc = c->desc_ls.as<uint4>(); CA.tiles = A.tiles; CA.wstate = c->wstate.as<uint8_t>();
        if (c->ls_variant == 2) {
            // warp-per-brick certification: TMA-staged candidates, packed FP32 (ss_certify.cuh, variant 2)
            SsCwArgs W{};
            W.bin_start = A.bin_start; W.bin_end = A.bin_end; W.rec = A.rec; W.tile_tab = A.tile_tab; W.brick_rng = A.brick_rng;
            W.work_desc = c->desc_ls.as<uint4>(); W.n_work = n_work; W.tiles = A.tiles; W.wstate = c->wstate.as<uint8_t>();
            W.evals = c->count_pairs ? c->pairs.as<unsigned long long>() + 1 : nullptr;
            const double ih2 = 1.0 / ((double)D.h * (double)D.h);
            W.g1 = (float)((double)SS_G1 * ih2); W.g2 = (float)((double)SS_G2 * ih2 * ih2); W.g3 = (float)((double)SS_G3 * ih2 * ih2 * ih2);
            W.r0sq = 0.3025f * D.h2; W.r1sq = 0.58f * D.h2;
            const bool cw_small = certify_runs <= 16;            // at most 4 candidate bins per axis (3 + the extension plane)
#define SS_CW_GO(G_, C_) do { if (cw_small) LAUNCH(c, (k_certify_warp<G_, C_, SS_CW_CAP_S, SS_CW_WARPS_S>), (n_work + SS_CW_WARPS_S - 1) / SS_CW_WARPS_S, SS_CW_WARPS_S * 32, D, W); \
                                 else LAUNCH(c, (k_certify_warp<G_, C_, SS_CW_CAP_L, SS_CW_WARPS_L>), (n_work + SS_CW_WARPS_L - 1) / SS_CW_WARPS_L, SS_CW_WARPS_L * 32, D, W); } while (0)
            if (global_mode) { if (c->count_pairs) SS_CW_GO(true, true); else SS_CW_GO(true, false); }
            else { if (c->count_pairs) SS_CW_GO(false, true); else SS_CW_GO(false, false); }
#undef SS_CW_GO
        } else if (global_mode) LAUNCH(c, k_certify<true>, n_work, SS_LS_THREADS, D, CA);
        else LAUNCH(c, k_certify<false>, n_work, SS_LS_THREADS, D, CA);
        ++ls_launches;
        LAUNCH(c, k_wstate_reduce, nblk(nbr_c, 256), 256, c->wstate.as<uint8_t>(), nbr_c, c->bstate.as<uint8_t>(), c->flag_fix.as<uint32_t>(),
               c->wflag.as<uint8_t>());
        cub_excl_scan(c, c->flag_fix.as<uint32_t>(), c->off_fix.as<uint32_t>(), nbr_c);
        LAUNCH(c, k_compact_list, nblk(nbr_c, 256), 256, c->flag_fix.as<uint32_t>(), c->off_fix.as<uint32_t>(), nbr_c, c->fix_list.as<uint32_t>());
        uint32_t ln[2] = { 0, 0 };
        CK(cudaMemcpyAsync(&ln[0], c->off_fix.as<uint32_t>() + (nbr_c - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&ln[1], c->flag_fix.as<uint32_t>() + (nbr_c - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (ln[0] + ln[1]) {
            SsLsArgs F = A;
            F.mode = SS_LS_FIX; F.wflag = c->wflag.as<uint8_t>(); F.fix_bricks = c->fix_list.as<uint32_t>();
            launch_exact(c, D, F, ln[0] + ln[1], global_mode, ls_launches);
        }
    }
    out->tm.bricks_levelset += n_work;
    const uint32_t nbr_b = nbatch * nbricks;
    uint32_t n_mc = 0, n_fixscan = 0;
    list_bricks(c, D, nbr_b, c->ls_variant == 2 && split_certify && !global_mode, n_mc, n_fixscan);
    out->tm.bricks_total += nbr_b; out->tm.bricks_mc += n_mc; out->tm.bricks_fixscan += n_fixscan;
    if (!exact_all && n_fixscan) {
        // exact values for certified points that turn out to lie on a surface-crossing edge
        const size_t nbr = (size_t)nbatch * nbricks;
        c->wflag.ensure(nbr * SS_LS_WARPS); c->brick_seen.ensure(nbr * 4); c->fix_list.ensure(nbr * 4); c->nflag.ensure(8);
        CK(cudaMemsetAsync(c->wflag.p, 0, nbr * SS_LS_WARPS, st));
        CK(cudaMemsetAsync(c->brick_seen.p, 0, nbr * 4, st));
        CK(cudaMemsetAsync(c->nflag.p, 0, 8, st));
        if (c->mc_variant == 1 && !global_mode)
            LAUNCH(c, k_fixup_flags_warp, (n_fixscan + SS_MW_WARPS - 1) / SS_MW_WARPS, SS_MW_WARPS * 32, D, c->tiles.as<float>(), c->list_fix.as<uint32_t>(), n_fixscan,
                   c->wflag.as<uint8_t>(), c->fix_list.as<uint32_t>(), c->nflag.as<uint32_t>());
        else
        LAUNCH(c, k_fixup_flags, n_fixscan, SS_TP_THREADS, D, c->tiles.as<float>(), c->list_fix.as<uint32_t>(), c->wflag.as<uint8_t>(),
               c->brick_seen.as<uint32_t>(), c->fix_list.as<uint32_t>(), c->nflag.as<uint32_t>());
        uint32_t nfl[2] = { 0, 0 };
        CK(cudaMemcpyAsync(nfl, c->nflag.p, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (nfl[0]) {
            A.mode = SS_LS_FIX; A.wflag = c->wflag.as<uint8_t>(); A.fix_bricks = c->fix_list.as<uint32_t>();
            if (split_certify) launch_exact(c, D, A, nfl[0], global_mode, ls_launches);
            else { launch_levelset(c, dim3(nfl[0]), D, A, c->count_pairs != 0, global_mode); ++ls_launches; }
            fix_points += nfl[1];
        }
    }
    *n_mc_out = n_mc;
    return SS_OK;
}

// Owner + ghost memberships of the points d_xyz[0..n) (dense_subdomains.rs:1810-1905), stable-sorted by subdomain: key_b = flat
// subdomain per membership, val_b = point index (ascending inside a subdomain), cid = compressed subdomain id, sub_flat / sub_off
// per non-empty subdomain (copied to h_flat / h_off).  M = 0: nothing past the count is written.
static int decompose(ss_context *c, const SsDev &D, const float *d_xyz, uint64_t n, uint64_t nslots, uint32_t &M, uint32_t &nsub,
                     std::vector<uint32_t> &h_flat, std::vector<uint32_t> &h_off) {
    cudaStream_t st = c->stream;
    c->cnt.ensure(n * 4); c->off.ensure(n * 4 + 4);
    LAUNCH(c, k_classify_count, nblk(n, 256), 256, D, d_xyz, (uint32_t)n, c->cnt.as<uint32_t>());
    cub_excl_scan(c, c->cnt.as<uint32_t>(), c->off.as<uint32_t>(), (uint32_t)n);
    uint32_t lo = 0, lc = 0;
    CK(cudaMemcpyAsync(&lo, c->off.as<uint32_t>() + (n - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&lc, c->cnt.as<uint32_t>() + (n - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const uint64_t M64 = (uint64_t)lo + lc;
    if (M64 >= 0xfffffff0ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "more than 2^32 subdomain memberships");
    M = (uint32_t)M64; nsub = 0;
    if (M == 0) return SS_OK;
    c->key_a.ensure((size_t)M * 4); c->key_b.ensure((size_t)M * 4); c->val_a.ensure((size_t)M * 4); c->val_b.ensure((size_t)M * 4);
    LAUNCH(c, k_classify_fill, nblk(n, 256), 256, D, d_xyz, (uint32_t)n, c->off.as<uint32_t>(), c->key_a.as<uint32_t>(), c->val_a.as<uint32_t>());
    cub_sort_pairs(c, c->key_a.as<uint32_t>(), c->key_b.as<uint32_t>(), c->val_a.as<uint32_t>(), c->val_b.as<uint32_t>(), M, bits_for(nslots));
    // key_b = flat subdomain per membership (sorted), val_b = particle index (ascending inside a subdomain)
    c->flags.ensure((size_t)M * 4); c->scan.ensure((size_t)M * 4); c->cid.ensure((size_t)M * 4);
    LAUNCH(c, k_seg_flags, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->flags.as<uint32_t>());
    cub_incl_scan(c, c->flags.as<uint32_t>(), c->scan.as<uint32_t>(), M);
    CK(cudaMemcpyAsync(&nsub, c->scan.as<uint32_t>() + (M - 1), 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    c->sub_flat.ensure((size_t)nsub * 4); c->sub_off.ensure((size_t)(nsub + 1) * 4); c->sub_sparse.ensure(nsub);
    LAUNCH(c, k_seg_finish, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->scan.as<uint32_t>(), c->cid.as<uint32_t>(),
           c->sub_flat.as<uint32_t>(), c->sub_off.as<uint32_t>());
    h_flat.resize(nsub); h_off.resize(nsub + 1);
    CK(cudaMemcpyAsync(h_flat.data(), c->sub_flat.p, (size_t)nsub * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h_off.data(), c->sub_off.p, (size_t)(nsub + 1) * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SS_OK;
}

// ---- anisotropic kernels (ss_aniso.cuh)
// Moments, eigen-decomposition, centres, matrices and factors of the n particles from the neighbour lists stage_densities left in
// the scratch (subdomain path: membership cell lists; global path: the whole-domain cell list).
static void stage_aniso_moments(ss_context *c, const SsDev &D, uint64_t n, uint32_t M, bool global_mode, const float *d_rho, ss_surface *out) {
    cudaStream_t st = c->stream;
    out->an_xbar = c->o_an_xbar; c->o_an_xbar = DevBuf(); out->an_mat = c->o_an_mat; c->o_an_mat = DevBuf(); out->an_fac = c->o_an_fac; c->o_an_fac = DevBuf();
    out->an_xbar.ensure(n * 12); out->an_mat.ensure(n * 24); out->an_fac.ensure(n * 4);
    c->an_sweeps.ensure(4);
    CK(cudaMemsetAsync(c->an_sweeps.p, 0, 4, st));
    if (!global_mode)
        LAUNCH(c, k_aniso_moments, nblk(M, 128), 128, D, c->aniso_k, M, c->key_b.as<uint32_t>(), c->spos.as<float4>(), c->sub_flat.as<uint32_t>(),
               c->tab_a.as<uint32_t>(), c->tab_b.as<uint32_t>(), d_rho, out->an_xbar.as<float>(), out->an_mat.as<float>(), out->an_fac.as<float>(),
               c->an_sweeps.as<unsigned>());
    else
        LAUNCH(c, k_aniso_moments_global, nblk(n, 128), 128, D, c->aniso_k, (uint32_t)n, c->gkey_b.as<uint32_t>(), c->spos.as<float4>(),
               c->tab_a.as<uint32_t>(), c->tab_b.as<uint32_t>(), d_rho, out->an_xbar.as<float>(), out->an_mat.as<float>(), out->an_fac.as<float>(),
               c->an_sweeps.as<unsigned>());
}

// The membership and bin buffers of the centres' decomposition trade places with the particles' ones while it is built, so that
// decompose / stage_binning serve both and the particles' bins stay intact for the post-processing queries.
static void swap_aniso_bins(ss_context *c) {
    std::swap(c->key_a, c->an_key_a); std::swap(c->key_b, c->an_key_b); std::swap(c->val_a, c->an_val_a); std::swap(c->val_b, c->an_val_b);
    std::swap(c->flags, c->an_flags); std::swap(c->scan, c->an_scan); std::swap(c->cid, c->an_cid); std::swap(c->sub_flat, c->an_sub_flat);
    std::swap(c->sub_off, c->an_sub_off); std::swap(c->tab_a, c->an_tab_a); std::swap(c->tab_b, c->an_tab_b); std::swap(c->rec, c->an_rec);
    std::swap(c->ksplit, c->an_ksplit);
}

// Second decomposition + splat bins over the centres x_bar (every ellipsoid lies in the ball of radius R around its centre, so
// the ghost margin and the bins' reach hold), and the bin-sorted (M, f) records.  Returns the non-empty subdomains in h_flat.
static int stage_aniso_bins(ss_context *c, const SsDev &D, const float *d_xyz, uint64_t n, uint64_t nslots, const float *d_rho, ss_surface *out,
                            uint32_t &nsub, std::vector<uint32_t> &h_flat) {
    std::vector<uint32_t> h_off;
    uint32_t M = 0;
    swap_aniso_bins(c);
    int rc = decompose(c, D, out->an_xbar.as<float>(), n, nslots, M, nsub, h_flat, h_off);
    if (!rc && M) rc = stage_binning(c, D, out->an_xbar.as<float>(), d_rho, M, nsub, false);
    if (!rc && M) {
        c->an_am.ensure((size_t)M * 32);
        LAUNCH(c, k_aniso_records, nblk(M, 256), 256, D, M, c->key_b.as<uint32_t>(), c->val_a.as<uint32_t>(), d_xyz, out->an_mat.as<float>(),
               out->an_fac.as<float>(), c->an_am.as<float4>());
    }
    swap_aniso_bins(c);
    return rc;
}

// Level set of one batch of tiles with the anisotropic kernels: exact values at every point, then the brick lists of list_bricks.
static void aniso_levelset_batch(ss_context *c, const SsDev &D, uint32_t nbatch, unsigned nbricks, ss_surface *out, uint64_t &ls_launches, uint32_t *n_mc_out) {
    SsAwArgs W{};
    W.bin_start = c->an_tab_a.as<uint32_t>(); W.bin_end = c->an_tab_b.as<uint32_t>(); W.rec = c->an_rec.as<float4>(); W.am = c->an_am.as<float4>();
    W.tile_tab = c->tile_tab.as<SsTile>(); W.brick_rng = c->brick_rng.as<int2>(); W.n_bricks = nbatch * nbricks;
    W.tiles = c->tiles.as<float>(); W.bstate = c->bstate.as<uint8_t>();
    LAUNCH(c, k_aniso_levelset_warp, (W.n_bricks + SS_AW_WARPS - 1) / SS_AW_WARPS, SS_AW_WARPS * 32, D, W);
    ++ls_launches;
    uint32_t n_mc = 0, n_fixscan = 0;
    list_bricks(c, D, W.n_bricks, false, n_mc, n_fixscan);
    out->tm.bricks_levelset += W.n_bricks; out->tm.bricks_total += W.n_bricks; out->tm.bricks_mc += n_mc;
    *n_mc_out = n_mc;
}

// Marching cubes over the listed bricks of one batch: count, scan the brick totals, emit vertices, emit triangles; appends to
// the surface's mesh buffers and to the boundary-vertex list.
static int marching_cubes_batch(ss_context *c, const SsDev &D, bool global_mode, uint32_t n_mc, ss_surface *out, uint64_t &vtotal, uint64_t &ttotal) {
    cudaStream_t st = c->stream;
    uint64_t bv = 0, bt = 0;
    const bool warp_mc = c->mc_variant == 1 && !global_mode;       // ss_mc.cuh: one warp per brick, count + emit
    if (n_mc) {
        if (warp_mc) LAUNCH(c, k_mc_count_warp, (n_mc + SS_MW_WARPS - 1) / SS_MW_WARPS, SS_MW_WARPS * 32, D, c->tiles.as<float>(), c->list_mc.as<uint32_t>(), n_mc,
                            c->vmask.as<uint8_t>(), c->voff.as<uint32_t>(), c->vcnt.as<uint32_t>(), c->tcnt.as<uint32_t>());
        else if (global_mode) LAUNCH(c, k_mc_count<true>, n_mc, SS_TP_THREADS, D, c->tiles.as<float>(), c->list_mc.as<uint32_t>(), c->vmask.as<uint8_t>(), c->vcnt.as<uint32_t>(), c->tcnt.as<uint32_t>());
        else LAUNCH(c, k_mc_count<false>, n_mc, SS_TP_THREADS, D, c->tiles.as<float>(), c->list_mc.as<uint32_t>(), c->vmask.as<uint8_t>(), c->vcnt.as<uint32_t>(), c->tcnt.as<uint32_t>());
        cub_excl_scan(c, c->vcnt.as<uint32_t>(), c->vblk_off.as<uint32_t>(), n_mc);
        cub_excl_scan(c, c->tcnt.as<uint32_t>(), c->tblk_off.as<uint32_t>(), n_mc);
    }
    uint32_t bc = 0;
    CK(cudaMemcpyAsync(&bc, c->bcount.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (n_mc) {
        uint32_t lv[2] = { 0, 0 }, lt[2] = { 0, 0 };
        CK(cudaMemcpyAsync(&lv[1], c->vcnt.as<uint32_t>() + (n_mc - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&lt[1], c->tcnt.as<uint32_t>() + (n_mc - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&lv[0], c->vblk_off.as<uint32_t>() + (n_mc - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&lt[0], c->tblk_off.as<uint32_t>() + (n_mc - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        bv = (uint64_t)lv[0] + lv[1]; bt = (uint64_t)lt[0] + lt[1];
    }
    if (vtotal + bv >= 0xfffffff0ull || ttotal + bt >= 0xfffffff0ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "mesh too large for 32-bit vertex / triangle ids");
    if (bv || bt) {
        out->verts.grow_keep((vtotal + bv) * 12, vtotal * 12, st);
        out->vkeys.grow_keep((vtotal + bv) * 8, vtotal * 8, st);
        out->tris.grow_keep((ttotal + bt) * 12, ttotal * 12, st);
        // boundary list can hold at most every vertex of the batch
        c->bkeys_a.grow_keep(((size_t)bc + bv) * 8, (size_t)bc * 8, st);
        c->bids_a.grow_keep(((size_t)bc + bv) * 4, (size_t)bc * 4, st);
        SsMcOut O{};
        O.verts = out->verts.as<float>(); O.tris = out->tris.as<uint32_t>(); O.vkeys = out->vkeys.as<unsigned long long>();
        O.bkeys = c->bkeys_a.as<unsigned long long>(); O.bids = c->bids_a.as<uint32_t>(); O.bcount = c->bcount.as<uint32_t>();
        O.vbase = (uint32_t)vtotal; O.tbase = (uint32_t)ttotal; O.bcap = (uint32_t)std::min<size_t>((size_t)bc + bv, 0xffffffffu);
        if (warp_mc) {
            LAUNCH(c, k_mc_emit_warp, (n_mc + SS_MW_WARPS - 1) / SS_MW_WARPS, SS_MW_WARPS * 32, D, c->tiles.as<float>(), c->list_mc.as<uint32_t>(), n_mc,
                   c->vmask.as<uint8_t>(), c->voff.as<uint32_t>(), c->vcnt.as<uint32_t>(), c->tcnt.as<uint32_t>(), c->vblk_off.as<uint32_t>(),
                   c->tblk_off.as<uint32_t>(), c->flag_mc.as<uint32_t>(), c->off_mc.as<uint32_t>(), c->tile_tab.as<SsTile>(), O);
        } else if (global_mode) {
            LAUNCH(c, k_mc_verts<true>, n_mc, SS_TP_THREADS, D, c->tiles.as<float>(), c->vmask.as<uint8_t>(), c->vblk_off.as<uint32_t>(),
                   c->vcnt.as<uint32_t>(), c->voff.as<uint32_t>(), c->tile_tab.as<SsTile>(), c->list_mc.as<uint32_t>(), O);
            LAUNCH(c, k_mc_tris<true>, n_mc, SS_TP_THREADS, D, c->tiles.as<float>(), c->vmask.as<uint8_t>(), c->tblk_off.as<uint32_t>(),
                   c->tcnt.as<uint32_t>(), c->voff.as<uint32_t>(), c->list_mc.as<uint32_t>(), O);
        } else {
            LAUNCH(c, k_mc_verts<false>, n_mc, SS_TP_THREADS, D, c->tiles.as<float>(), c->vmask.as<uint8_t>(), c->vblk_off.as<uint32_t>(),
                   c->vcnt.as<uint32_t>(), c->voff.as<uint32_t>(), c->tile_tab.as<SsTile>(), c->list_mc.as<uint32_t>(), O);
            LAUNCH(c, k_mc_tris<false>, n_mc, SS_TP_THREADS, D, c->tiles.as<float>(), c->vmask.as<uint8_t>(), c->tblk_off.as<uint32_t>(),
                   c->tcnt.as<uint32_t>(), c->voff.as<uint32_t>(), c->list_mc.as<uint32_t>(), O);
        }
        vtotal += bv; ttotal += bt;
    }
    return SS_OK;
}

// Stitching: weld duplicated boundary vertices (same MC edge key), compact the vertices, remap the triangle indices.
static int weld_boundary_vertices(ss_context *c, ss_surface *out, uint64_t vtotal, uint64_t ttotal, uint64_t &nv_final_out, uint32_t &bc_out) {
    cudaStream_t st = c->stream;
    uint32_t bc = 0;
    CK(cudaMemcpyAsync(&bc, c->bcount.p, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    uint64_t nv_final = vtotal;
    if (vtotal && bc) {
        c->bkeys_b.ensure((size_t)bc * 8); c->bids_b.ensure((size_t)bc * 4);
        size_t tmp = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, c->bkeys_a.as<unsigned long long>(), c->bkeys_b.as<unsigned long long>(),
                                           c->bids_a.as<uint32_t>(), c->bids_b.as<uint32_t>(), (int)bc, 0, 64, st));
        c->cub_tmp.ensure(tmp);
        CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, tmp, c->bkeys_a.as<unsigned long long>(), c->bkeys_b.as<unsigned long long>(),
                                           c->bids_a.as<uint32_t>(), c->bids_b.as<uint32_t>(), (int)bc, 0, 64, st));
        c->launches += 17;
        c->remap.ensure(vtotal * 4); c->keep.ensure(vtotal * 4); c->newid.ensure(vtotal * 4 + 4);
        LAUNCH(c, k_iota_keep, nblk(vtotal, 256), 256, (uint32_t)vtotal, c->remap.as<uint32_t>(), c->keep.as<uint32_t>());
        LAUNCH(c, k_weld_runs, nblk(bc, 256), 256, c->bkeys_b.as<unsigned long long>(), c->bids_b.as<uint32_t>(), bc,
               c->remap.as<uint32_t>(), c->keep.as<uint32_t>());
        cub_excl_scan(c, c->keep.as<uint32_t>(), c->newid.as<uint32_t>(), (uint32_t)vtotal);
        uint32_t lk = 0, ln = 0;
        CK(cudaMemcpyAsync(&lk, c->keep.as<uint32_t>() + (vtotal - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&ln, c->newid.as<uint32_t>() + (vtotal - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        nv_final = (uint64_t)lk + ln;
        // compact into fresh buffers (swap)
        DevBuf nverts = c->o_verts2, nkeys = c->o_vkeys2;
        c->o_verts2 = DevBuf(); c->o_vkeys2 = DevBuf();
        nverts.ensure(std::max<uint64_t>(vtotal, 1) * 12); nkeys.ensure(std::max<uint64_t>(vtotal, 1) * 8);
        LAUNCH(c, k_compact_verts, nblk(vtotal, 256), 256, (uint32_t)vtotal, c->keep.as<uint32_t>(), c->newid.as<uint32_t>(),
               out->verts.as<float>(), out->vkeys.as<unsigned long long>(), nverts.as<float>(), nkeys.as<unsigned long long>());
        LAUNCH(c, k_remap_tris, nblk(ttotal * 3, 256), 256, ttotal * 3, c->remap.as<uint32_t>(), c->newid.as<uint32_t>(), out->tris.as<uint32_t>());
        CK(cudaStreamSynchronize(st));
        c->o_verts2 = out->verts; c->o_vkeys2 = out->vkeys;     // keep the pre-weld buffers for the next frame
        out->verts = nverts; out->vkeys = nkeys;
    }
    nv_final_out = nv_final; bc_out = bc;
    return SS_OK;
}

static int run_subdomain_grid(ss_context *c, const Prepared &PP, const ss_params_f32 *p, ss_surface *out, const Partition &part = Partition(),
                              bool global_mode = false) {
    const uint64_t n = PP.n;
    const float *d_xyz = PP.d_xyz;
    cudaStream_t st = c->stream;

    // ---- initialize_parameters, dense_subdomains.rs:89-244
    // global path (reconstruction.rs:65-194): tiles of 64 cells are an implementation detail, the arithmetic is global
    const int64_t S = global_mode ? 64 : (int64_t)p->subdomain_num_cubes_per_dim;
    const float h = p->compact_support_radius, cs = p->cube_size;
    const float r2 = faddr(p->particle_radius, p->particle_radius);
    const float rest_mass = fmulr(fmulr(fmulr(r2, r2), r2), p->rest_density);
    const float margin = global_mode ? fmulr(cs, ceilf(fdivr(h, cs)) + 2.0f)      // stencil reach (R + 1 cells) + slack
                                     : fmulr(fmulr(ceilf(fdivr(h, cs)), cs), 1.01f);
    int64_t nsd[3], ncg[3];
    for (int d = 0; d < 3; ++d) { nsd[d] = (PP.grid.nc[d] + S - 1) / S; ncg[d] = nsd[d] * S; }
    HostGrid gg, sg;
    int rc = grid_new(gg, PP.grid.mn, ncg, cs);
    if (rc) return ss_fail(rc, "global marching cubes grid construction failed");
    const float sub_size = fmulr(cs, (float)S);
    rc = grid_new(sg, gg.mn, nsd, sub_size);
    if (rc) return ss_fail(rc, "subdomain grid construction failed");
    out->grid = global_mode ? PP.grid : gg; out->subgrid = sg; out->S = (int)S;

    for (int d = 0; d < 3; ++d) {
        if (gg.np[d] >= (1 << 20)) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "more than 2^20 grid points per dimension are not supported by the device path");
    }
    if ((double)nsd[0] * (double)nsd[1] * (double)nsd[2] >= 2147483647.0) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many subdomain slots");
    if (S > 1024) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "subdomain_num_cubes_per_dim > 1024 is not supported");

    SsDev D{};
    for (int d = 0; d < 3; ++d) { D.gmin[d] = gg.mn[d]; D.nsd[d] = (int)nsd[d]; }
    D.c = cs; D.h = h; D.h2 = fmulr(h, h); D.h2m = fmulr(D.h2, 1.01f); D.thr = p->iso_surface_threshold;
    D.rest_mass = rest_mass; D.sub_size = sub_size; D.margin = margin; D.grow = fmulr(margin, 1.5f);
    D.S = (int)S; D.np = (int)S + 1; D.np_magic = (uint32_t)(4294967296ull / (uint64_t)D.np) + 1u;
    D.R = (int)ceilf(fdivr(h, cs));
    D.srad = (int)ceilf(fdivr(margin, sub_size));
    if (D.srad > 8) return ss_fail(SS_ERR_INVALID_PARAMETER, "ghost margin spans more than 8 subdomains; increase subdomain_num_cubes_per_dim");
    fill_kernel_consts(D, h);
    D.nsD = (int)ceil(((double)S * cs + 3.0 * (double)margin) / (double)h) + 3;
    D.ns_stride = D.nsD * D.nsD * D.nsD;
    fill_bins(D, cs);
    D.simd = p->enable_simd ? 1 : 0;
    D.gmode = global_mode ? 1 : 0;
    uint64_t g_ns_cells = 0;
    if (global_mode) {
        HostGrid ns;
        int rcn = grid_from_aabb(ns, PP.grid.mn, PP.grid.mx, h);                       // neighborhood_search.rs:172-173
        if (rcn) return ss_fail(SS_ERR_INVALID_PARAMETER, "failed to construct grid for neighborhood search");
        for (int d = 0; d < 3; ++d) { D.g_ns_amin[d] = ns.mn[d]; D.g_ns_nc[d] = (int)ns.nc[d]; }
        g_ns_cells = (uint64_t)ns.nc[0] * ns.nc[1] * ns.nc[2];
        if (g_ns_cells >= (1ull << 28)) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "domain too large for the global (non-decomposed) path");
        const float half_real = ceilf(fdivr(h, cs));
        const float rev = fmulr(fmulr(cs, half_real), faddr(1.0f, sqrtf(FLT_EPSILON)));   // density_map.rs:575-576
        D.rev2 = fmulr(rev, rev); D.sup = 2 * D.R + 2;
        for (int d = 0; d < 3; ++d) { D.g_allow_min[d] = fsubr(PP.grid.mn[d], -rev); D.g_allow_max[d] = faddr(PP.grid.mx[d], -rev); }
        bool degen = D.g_allow_min[0] == D.g_allow_max[0] && D.g_allow_min[1] == D.g_allow_max[1] && D.g_allow_min[2] == D.g_allow_max[2];
        bool cons = D.g_allow_min[0] <= D.g_allow_max[0] && D.g_allow_min[1] <= D.g_allow_max[1] && D.g_allow_min[2] <= D.g_allow_max[2];
        if (degen || !cons) return ss_fail(SS_ERR_INVALID_DOMAIN, "the allowed domain of particles is inconsistent/degenerate (DensityMapError::InvalidDomain)");
    }
    D.part_axis = part.enabled ? part.axis : 0;
    D.keep_lo = part.enabled ? (int)std::max<int64_t>(part.own_lo - part.halo, 0) : 0;
    D.keep_hi = part.enabled ? (int)std::min<int64_t>(part.own_hi + part.halo, nsd[D.part_axis]) : (int)nsd[0];
    if (!part.enabled) { D.part_axis = 0; D.keep_lo = 0; D.keep_hi = (int)nsd[0]; }
    int certify_runs = 0;              // upper bound of the candidate runs of a brick (variant 1 keeps one per lane)
    {
        int per_axis = ss_floor_div(6 + D.R, D.be) - ss_floor_div(-D.R, D.be) + 2;
        if (per_axis * per_axis > 128) return ss_fail(SS_ERR_INVALID_PARAMETER, "internal: too many candidate bin runs per brick");
        certify_runs = per_axis * per_axis;
    }

    const bool want_nbrs = p->global_neighborhood_list != 0 && !part.enabled;
    const bool aniso = c->aniso && !part.enabled && !part.given_rho;
    out->aniso = aniso ? 1 : 0;
    CK(cudaEventRecord(c->ev[2], st));
    out->nv = out->nt = 0; out->nsub = 0;
    out->owner = c;
    c->post.valid = 0; out->frame = ++c->frame;
    out->rho = c->o_rho; c->o_rho = DevBuf(); out->verts = c->o_verts; c->o_verts = DevBuf();
    out->tris = c->o_tris; c->o_tris = DevBuf(); out->vkeys = c->o_vkeys; c->o_vkeys = DevBuf();
    out->rho.ensure(std::max<uint64_t>(n, 1) * 4);
    float *d_rho = out->rho.as<float>();
    CK(cudaMemsetAsync(d_rho, 0, std::max<uint64_t>(n, 1) * 4, st));
    // NOTE (multi-GPU): the max-reduce callback is a collective -- every rank must call it exactly once per
    // reconstruction, also ranks that received no particles or own no subdomain.
    if (n == 0) {
        for (int e = 3; e <= 9; ++e) CK(cudaEventRecord(c->ev[e], st));
        CK(cudaStreamSynchronize(st));
        if (part.enabled && part.max_reduce) part.max_reduce(0, part.max_reduce_user);
        return SS_OK;
    }

    // ---- decomposition: memberships (owner + ghosts), stable sort by subdomain
    const uint64_t nslots = (uint64_t)nsd[0] * nsd[1] * nsd[2];
    uint32_t M = 0, nsub = 0;
    std::vector<uint32_t> h_flat, h_off;
    rc = decompose(c, D, d_xyz, n, nslots, M, nsub, h_flat, h_off);
    if (rc) return rc;
    if (M == 0) {
        for (int e = 3; e <= 9; ++e) CK(cudaEventRecord(c->ev[e], st));
        CK(cudaStreamSynchronize(st));
        if (part.enabled && part.max_reduce) part.max_reduce(0, part.max_reduce_user);
        return SS_OK;
    }
    // sparse classification, dense_subdomains.rs:1242-1251, :1590
    uint64_t maxp = 0;
    for (uint32_t s = 0; s < nsub; ++s) maxp = std::max<uint64_t>(maxp, h_off[s + 1] - h_off[s]);
    out->max_particles = maxp;
    if (part.enabled && part.max_reduce) maxp = std::max<uint64_t>(maxp, part.max_reduce(maxp, part.max_reduce_user));
    if (part.enabled && part.global_max_particles) maxp = std::max<uint64_t>(maxp, part.global_max_particles);
    const uint64_t sparse_limit = std::max<uint64_t>(maxp / 20, 100);
    out->nsub = nsub; out->sub_flat.resize(nsub); out->sub_count.resize(nsub); out->sub_sparse.resize(nsub);
    std::vector<uint8_t> h_owned(nsub, 1);
    std::vector<uint32_t> owned_list;
    owned_list.reserve(nsub);
    for (uint32_t s = 0; s < nsub; ++s) {
        out->sub_flat[s] = h_flat[s]; out->sub_count[s] = h_off[s + 1] - h_off[s];
        out->sub_sparse[s] = (!global_mode && out->sub_count[s] <= sparse_limit) ? 1 : 0;
        if (part.enabled) {
            const int64_t f = h_flat[s];
            int64_t ijk[3];
            ijk[0] = f / (nsd[1] * nsd[2]); ijk[1] = (f - ijk[0] * nsd[1] * nsd[2]) / nsd[2]; ijk[2] = f - ijk[0] * nsd[1] * nsd[2] - ijk[1] * nsd[2];
            h_owned[s] = (ijk[part.axis] >= part.own_lo && ijk[part.axis] < part.own_hi) ? 1 : 0;
        }
        if (h_owned[s]) owned_list.push_back(s);
    }
    out->sub_owned = h_owned;
    if (part.enabled && part.stop_after_decomposition) { for (int e = 3; e <= 9; ++e) CK(cudaEventRecord(c->ev[e], st)); CK(cudaStreamSynchronize(st)); return SS_OK; }
    c->sub_owned.ensure(nsub);
    CK(cudaMemcpyAsync(c->sub_owned.p, h_owned.data(), nsub, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->sub_sparse.p, out->sub_sparse.data(), nsub, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(c->ev[3], st));

    if (part.given_rho) {
        // SphInterpolator::new (sph_interpolation.rs:40-80): the caller's densities and the particle bins the queries of ss_post.cuh walk;
        // no density pass, no level set, no mesh
        c->err.ensure(4);
        CK(cudaMemsetAsync(c->err.p, 0, 4, st));
        CK(cudaMemcpyAsync(d_rho, part.given_rho, (size_t)n * 4, cudaMemcpyDefault, st));
        CK(cudaEventRecord(c->ev[4], st));
        rc = stage_binning(c, D, d_xyz, d_rho, M, nsub, false);
        if (rc) return rc;
        c->post.D = D; c->post.nsub = nsub; c->post.M = M; c->post.partitioned = 0; c->post.sphere_mass = part.given_mass; c->post.valid = 1;
        for (int e = 6; e <= 9; ++e) CK(cudaEventRecord(c->ev[e], st));
        CK(cudaStreamSynchronize(st));
        return SS_OK;
    }

    // ---- densities, then the splat bins
    rc = stage_densities(c, D, d_xyz, n, M, nsub, g_ns_cells, global_mode, want_nbrs, out, d_rho);
    if (rc) return rc;
    if (aniso) {
        if (!c->ev_an[0]) for (auto &ev : c->ev_an) CK(cudaEventCreate(&ev));
        CK(cudaEventRecord(c->ev_an[0], st));
        stage_aniso_moments(c, D, n, M, global_mode, d_rho, out);
    }
    CK(cudaEventRecord(c->ev[4], st));
    rc = stage_binning(c, D, d_xyz, d_rho, M, nsub, part.enabled != 0);
    if (rc) return rc;
    float binning_ms = 0.f;
    CK(cudaEventElapsedTime(&binning_ms, c->ev[4], c->ev[5]));
    // anisotropic kernels: the tiles are those of the centres' decomposition
    uint32_t an_nsub = 0;
    std::vector<uint32_t> an_flat, an_list;
    if (aniso) {
        CK(cudaEventRecord(c->ev_an[1], st));
        rc = stage_aniso_bins(c, D, d_xyz, n, nslots, d_rho, out, an_nsub, an_flat);
        if (rc) return rc;
        CK(cudaEventRecord(c->ev_an[2], st));
        an_list.resize(an_nsub);
        for (uint32_t s = 0; s < an_nsub; ++s) an_list[s] = s;
        unsigned h_sw = 0;
        CK(cudaMemcpyAsync(&h_sw, c->an_sweeps.p, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        out->an_sweeps = h_sw;
    }
    const std::vector<uint32_t> &tile_flat = aniso ? an_flat : h_flat, &tile_list = aniso ? an_list : owned_list;

    // ---- level set + marching cubes over batches of subdomain tiles
    const size_t np3 = (size_t)D.np * D.np * D.np;
    const unsigned nbricks = (unsigned)(D.nb * D.nb * D.nb);
    const size_t per_tile = np3 * (4 + 4 + 1) + (size_t)nbricks * (SS_LS_WARPS + 8 + 1 + 16) + 256;
    // as many tiles per batch as fit a third of the free memory (fewer host synchronisations per frame); the brick index
    // tile * nb^3 + ... must stay below 2^31
    const uint32_t nown = (uint32_t)tile_list.size();
    // The tile buffers of the previous frame are reused whenever they hold all tiles or at least half of what a fresh
    // allocation would get: the amount of free memory wobbles from frame to frame (result buffers in flight), and re-allocating
    // tens of GB costs ~100 ms.  The free memory is only queried when the buffers do not hold all tiles: cudaMemGetInfo takes a
    // device-wide lock, and with an `nvidia-smi -lms 200` sampler running beside the process (bench.py's clock record) it was
    // measured to stall here for up to 100 ms on every step the sampler's query fell into (tile_setup in the timings).
    const size_t have_tiles = std::min(c->tiles.cap / (np3 * 4), std::min(c->voff.cap / (np3 * 4), c->vmask.cap / np3));
    size_t max_tiles;
    if (c->max_tiles) max_tiles = c->max_tiles;
    else if (have_tiles >= nown && have_tiles) max_tiles = have_tiles;
    else {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const size_t reusable = c->tiles.cap + c->voff.cap + c->vmask.cap;
        const size_t want_tiles = std::max<size_t>(1, ((free_b + reusable) / 3) / per_tile);
        max_tiles = (have_tiles >= want_tiles / 2 && have_tiles) ? have_tiles : want_tiles;
    }
    max_tiles = std::min<size_t>(max_tiles, std::max<size_t>(1, (size_t)0x7fffffff / nbricks / 2));
    max_tiles = std::min<size_t>(max_tiles, std::max<uint32_t>(nown, 1));
    const size_t nblk_max = max_tiles * nbricks;
    c->tiles.ensure(max_tiles * np3 * 4); c->voff.ensure(max_tiles * np3 * 4); c->vmask.ensure(max_tiles * np3);
    c->vcnt.ensure(nblk_max * 4 + 4); c->tcnt.ensure(nblk_max * 4 + 4); c->vblk_off.ensure(nblk_max * 4 + 4); c->tblk_off.ensure(nblk_max * 4 + 4);
    c->tile_tab.ensure(max_tiles * sizeof(SsTile)); c->brick_rng.ensure((size_t)D.nb * sizeof(int2)); c->bstate.ensure(nblk_max);
    c->bcount.ensure(4); c->pairs.ensure(16);
    CK(cudaMemsetAsync(c->bcount.p, 0, 4, st));
    CK(cudaMemsetAsync(c->pairs.p, 0, 16, st));
    {   // candidate bin range of brick b along one axis: bins overlapping [8b - R, 8b + 7 + R)
        std::vector<int2> h_rng(D.nb);
        for (int bb = 0; bb < D.nb; ++bb) {
            h_rng[bb].x = std::max(ss_floor_div(8 * bb - D.R, D.be) + D.nlo, 0);
            h_rng[bb].y = std::min(ss_floor_div(8 * bb + 6 + D.R, D.be) + D.nlo, D.nbin - 1);
        }
        CK(cudaMemcpyAsync(c->brick_rng.p, h_rng.data(), (size_t)D.nb * sizeof(int2), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
    }
    std::vector<SsTile> h_tiles(max_tiles);
    uint64_t vtotal = 0, ttotal = 0;
    size_t bcap = std::max<size_t>(1 << 16, c->hint_bc + c->hint_bc / 8);
    c->bkeys_a.ensure(bcap * 8); c->bids_a.ensure(bcap * 4);
    size_t vcap = std::max<size_t>(1 << 16, c->hint_nv + c->hint_nv / 8), tcap = std::max<size_t>(1 << 17, c->hint_nt + c->hint_nt / 8);
    out->verts.ensure(vcap * 12); out->vkeys.ensure(vcap * 8); out->tris.ensure(tcap * 12);
    float ls_ms = 0.f, mc_ms = 0.f, setup_ms = 0.f;
    uint64_t ls_launches = 0, fix_points = 0;
    out->tile.clear();
    const bool exact_all = c->ls_exact_all || c->keep_tile_flat >= 0;
    for (uint32_t s0 = 0; s0 < nown; s0 += (uint32_t)max_tiles) {
        const uint32_t nbatch = std::min<uint32_t>((uint32_t)max_tiles, nown - s0);
        for (uint32_t q = 0; q < nbatch; ++q) {
            SsTile &T = h_tiles[q];
            const uint32_t sid = tile_list[s0 + q];
            const int64_t f = tile_flat[sid];
            int64_t ijk[3];
            ijk[0] = f / (nsd[1] * nsd[2]); ijk[1] = (f - ijk[0] * nsd[1] * nsd[2]) / nsd[2]; ijk[2] = f - ijk[0] * nsd[1] * nsd[2] - ijk[1] * nsd[2];
            for (int d = 0; d < 3; ++d) { T.gbase[d] = (int)(ijk[d] * S); T.smin[d] = faddr(gg.mn[d], fmulr((float)ijk[d], sub_size)); }
            T.s = sid; T.sparse = (aniso || out->sub_sparse[sid] || !D.simd) ? 1u : 0u;
        }
        CK(cudaMemcpyAsync(c->tile_tab.p, h_tiles.data(), (size_t)nbatch * sizeof(SsTile), cudaMemcpyHostToDevice, st));
        // level-set variant 2 writes every value a later pass reads (markers, exact values, exact zeros) and fills the untouched
        // bricks next to listed ones itself (k_zero_untouched): no zero-fill of the tiles (16 GB at 50 M particles)
        // (the anisotropic level set writes every point of the batch)
        const bool lazy_zero = aniso || (c->ls_variant == 2 && !exact_all && certify_runs <= 32 && !global_mode);
        if (!lazy_zero) CK(cudaMemsetAsync(c->tiles.p, 0, (size_t)nbatch * np3 * 4, st));
        CK(cudaMemsetAsync(c->bstate.p, 0, (size_t)nbatch * nbricks, st));
        // edge masks: the CTA-per-brick marching-cubes passes read the mask of every point of a listed brick (zero = no vertex); the
        // warp-per-brick passes only read masks their count pass wrote, so they need no zero-fill (4 GB at 50 M particles)
        if (global_mode || c->mc_variant != 1) CK(cudaMemsetAsync(c->vmask.p, 0, (size_t)nbatch * np3, st));
        CK(cudaEventRecord(c->ev[10], st));
        {   // set-up time of this batch: from the end of binning (first batch) / of the previous batch's marching cubes to here
            CK(cudaEventSynchronize(c->ev[10]));
            float su = 0.f;
            CK(cudaEventElapsedTime(&su, s0 == 0 ? (aniso ? c->ev_an[2] : c->ev[5]) : c->ev[6], c->ev[10]));
            setup_ms += su;
        }
        uint32_t n_mc = 0;
        if (aniso) aniso_levelset_batch(c, D, nbatch, nbricks, out, ls_launches, &n_mc);
        else {
            rc = levelset_batch(c, D, nbatch, nbricks, exact_all, certify_runs, global_mode, out, ls_launches, fix_points, &n_mc);
            if (rc) return rc;
        }
        CK(cudaEventRecord(c->ev[11], st));
        // optional parity tap
        if (c->keep_tile_flat >= 0) {
            for (uint32_t q = 0; q < nbatch; ++q) if ((int64_t)tile_flat[tile_list[s0 + q]] == c->keep_tile_flat) {
                out->tile.resize(np3);
                CK(cudaMemcpyAsync(out->tile.data(), c->tiles.as<float>() + (size_t)q * np3, np3 * 4, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
            }
        }
        rc = marching_cubes_batch(c, D, global_mode, n_mc, out, vtotal, ttotal);
        if (rc) return rc;
        CK(cudaEventRecord(c->ev[6], st));
        CK(cudaEventSynchronize(c->ev[6]));
        float a = 0.f, b = 0.f;
        CK(cudaEventElapsedTime(&a, c->ev[10], c->ev[11]));
        CK(cudaEventElapsedTime(&b, c->ev[11], c->ev[6]));
        ls_ms += a; mc_ms += b;
    }
    CK(cudaEventRecord(c->ev[7], st));

    // ---- stitching
    uint64_t nv_final = vtotal;
    uint32_t bc = 0;
    rc = weld_boundary_vertices(c, out, vtotal, ttotal, nv_final, bc);
    if (rc) return rc;
    out->nv = nv_final; out->nt = ttotal;
    c->hint_nv = vtotal; c->hint_nt = ttotal; c->hint_bc = bc;
    {
        // the splat bins stay in the scratch until the next call on this context: ss_post.cuh queries them
        const float r3p = fmulr(fmulr(p->particle_radius, p->particle_radius), p->particle_radius);
        c->post.D = D; c->post.nsub = nsub; c->post.M = M; c->post.partitioned = part.enabled;
        c->post.sphere_mass = fmulr(fmulr(fmulr(4.0f, 1.04719755119659774615f), r3p), p->rest_density);
        c->post.valid = 1;
    }
    if (c->sph_normals && nv_final) {
        // SPH normals at the vertices (pipeline post-processing step, splashsurf/src/reconstruct.rs:1287-1294); sphere rest mass
        // 4/3 pi r^3 rho0 as in reconstruct.rs:1126-1129
        out->normals = c->o_normals; c->o_normals = DevBuf();
        out->normals.ensure(nv_final * 12);
        SsNrmArgs NA{};
        NA.verts = out->verts.as<float>(); NA.vkeys = out->vkeys.as<unsigned long long>(); NA.nv = (uint32_t)nv_final;
        NA.sub_flat = c->sub_flat.as<uint32_t>(); NA.sub_owned = part.enabled ? c->sub_owned.as<uint8_t>() : nullptr; NA.nsub = nsub;
        NA.bin_start = c->tab_a.as<uint32_t>(); NA.bin_end = c->tab_b.as<uint32_t>(); NA.rec = c->rec.as<float4>(); NA.pidx = c->val_a.as<uint32_t>();
        NA.rho = d_rho; NA.brick_rng = c->brick_rng.as<int2>();
        const float r3 = fmulr(fmulr(p->particle_radius, p->particle_radius), p->particle_radius);
        const float frac_pi_3 = 1.04719755119659774615f;
        NA.sphere_mass = fmulr(fmulr(fmulr(4.0f, frac_pi_3), r3), p->rest_density);
        NA.normals = out->normals.as<float>();
        LAUNCH(c, k_sph_normals, nblk(nv_final, 128), 128, D, NA);
        out->has_normals = 1;
    }
    CK(cudaEventRecord(c->ev[8], st));
    CK(cudaEventRecord(c->ev[9], st));
    CK(cudaStreamSynchronize(st));

    // ---- timings
    ss_timings &T = out->tm;
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, c->ev[2], c->ev[3])); T.decomposition = ms;
    CK(cudaEventElapsedTime(&ms, c->ev[3], aniso ? c->ev_an[0] : c->ev[4])); T.density = ms;
    T.binning = binning_ms;
    if (aniso) {
        CK(cudaEventElapsedTime(&out->an_ms[0], c->ev_an[0], c->ev[4]));
        CK(cudaEventElapsedTime(&out->an_ms[1], c->ev_an[1], c->ev_an[2]));
    }
    T.levelset = ls_ms; T.marching_cubes = mc_ms; T.tile_setup = setup_ms;
    CK(cudaEventElapsedTime(&ms, c->ev[7], c->ev[8])); T.stitching = ms;
    T.levelset_launches = ls_launches; T.levelset_fixup_points = fix_points;
    unsigned long long h_pairs[2] = { 0, 0 };
    CK(cudaMemcpy(h_pairs, c->pairs.p, 16, cudaMemcpyDeviceToHost));
    T.levelset_pairs = (double)h_pairs[0]; T.levelset_cert_evals = (double)h_pairs[1];
    return SS_OK;
}

// ------------------------------------------------------------------ stage-level entry: one level-set tile ----
// density_grid_loop_auto / density_grid_loop_scalar (dense_subdomains.rs:715-847, both `pub`): the level-set tile of
// ONE subdomain from an explicit particle list (in list order == ascending index) and explicit densities.
__global__ void k_iota2(uint32_t n, uint32_t *__restrict__ a, uint32_t *__restrict__ zero) {
    uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    a[e] = e; zero[e] = 0;
}
extern "C" int ss_levelset_tile_f32(ss_context *c, const float *xyz, const float *rho, uint64_t n, const float global_min[3],
                                    float cube_size, const int64_t subdomain_ijk[3], uint32_t S, float h, float rest_mass,
                                    int mode, float *tile_out) {
    if (!c || !tile_out || !global_min || !subdomain_ijk || (n && (!xyz || !rho))) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    if (!(cube_size > 0.0f) || !(h > 0.0f) || S < 1 || S > 1024) return ss_fail(SS_ERR_INVALID_PARAMETER, "bad tile parameters");
    if (n >= 0x7fffffffull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many particles");
    for (int d = 0; d < 3; ++d) if (subdomain_ijk[d] < 0 || subdomain_ijk[d] > 1000) return ss_fail(SS_ERR_INVALID_PARAMETER, "subdomain_ijk out of range");
    try {
        CK(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        c->post.valid = 0; ++c->frame;                       // this entry rewrites the bins in the scratch
        SsDev D{};
        for (int d = 0; d < 3; ++d) { D.gmin[d] = global_min[d]; D.nsd[d] = (int)subdomain_ijk[d] + 1; }
        D.c = cube_size; D.h = h; D.h2 = fmulr(h, h); D.h2m = fmulr(D.h2, 1.01f); D.rest_mass = rest_mass;
        D.sub_size = fmulr(cube_size, (float)S); D.S = (int)S; D.np = (int)S + 1; D.np_magic = (uint32_t)(4294967296ull / (uint64_t)D.np) + 1u;
        D.R = (int)ceilf(fdivr(h, cube_size));
        fill_kernel_consts(D, h);
        fill_bins(D, cube_size);
        D.simd = mode == 0 ? 1 : 0;
        const size_t np3 = (size_t)D.np * D.np * D.np;
        c->tiles.ensure(np3 * 4);
        CK(cudaMemsetAsync(c->tiles.p, 0, np3 * 4, st));
        if (n) {
            const uint32_t M = (uint32_t)n;
            const uint32_t flat = (uint32_t)((subdomain_ijk[0] * D.nsd[1] + subdomain_ijk[1]) * D.nsd[2] + subdomain_ijk[2]);
            c->xyz.ensure(n * 12); c->rho.ensure(n * 4);
            CK(cudaMemcpyAsync(c->xyz.p, xyz, n * 12, cudaMemcpyDefault, st));
            CK(cudaMemcpyAsync(c->rho.p, rho, n * 4, cudaMemcpyDefault, st));
            c->key_a.ensure((size_t)M * 4); c->key_b.ensure((size_t)M * 4); c->val_a.ensure((size_t)M * 4); c->val_b.ensure((size_t)M * 4);
            c->cid.ensure((size_t)M * 4); c->sub_flat.ensure(4); c->sub_sparse.ensure(1); c->batch_subs.ensure(4);
            LAUNCH(c, k_iota2, nblk(M, 256), 256, M, c->val_b.as<uint32_t>(), c->cid.as<uint32_t>());
            uint32_t zero = 0; uint8_t z8 = 0;
            CK(cudaMemcpyAsync(c->sub_flat.p, &flat, 4, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(c->sub_sparse.p, &z8, 1, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(c->batch_subs.p, &zero, 4, cudaMemcpyHostToDevice, st));
            LAUNCH(c, k_bin_keys, nblk(M, 256), 256, D, c->xyz.as<float>(), M, c->cid.as<uint32_t>(), c->sub_flat.as<uint32_t>(),
                   c->val_b.as<uint32_t>(), (const uint8_t *)nullptr, c->key_a.as<uint32_t>());
            cub_sort_pairs(c, c->key_a.as<uint32_t>(), c->key_b.as<uint32_t>(), c->val_b.as<uint32_t>(), c->val_a.as<uint32_t>(), M, 32);
            const uint64_t bin_keys = (uint64_t)D.nbin_sub;
            c->tab_a.ensure(bin_keys * 4); c->tab_b.ensure(bin_keys * 4);
            CK(cudaMemsetAsync(c->tab_a.p, 0xff, bin_keys * 4, st));
            LAUNCH(c, k_mark_starts, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->tab_a.as<uint32_t>(), (uint32_t)bin_keys);
            LAUNCH(c, k_run_counts, nblk(M, 256), 256, c->key_b.as<uint32_t>(), M, c->tab_b.as<uint32_t>(), (uint32_t)bin_keys);
            c->rec.ensure((size_t)M * 16); c->ksplit.ensure((size_t)M * 4);
            LAUNCH(c, k_records, nblk(M, 256), 256, D, c->xyz.as<float>(), c->rho.as<float>(), M, c->key_b.as<uint32_t>(), c->val_a.as<uint32_t>(),
                   c->sub_flat.as<uint32_t>(), c->rec.as<float4>(), c->ksplit.as<int>());
            SsTile T{};
            for (int d = 0; d < 3; ++d) { T.gbase[d] = (int)(subdomain_ijk[d] * (int64_t)S); T.smin[d] = faddr(global_min[d], fmulr((float)subdomain_ijk[d], D.sub_size)); }
            T.s = 0; T.sparse = D.simd ? 0u : 1u;
            std::vector<int2> h_rng(D.nb);
            for (int bb = 0; bb < D.nb; ++bb) {
                h_rng[bb].x = std::max(ss_floor_div(8 * bb - D.R, D.be) + D.nlo, 0);
                h_rng[bb].y = std::min(ss_floor_div(8 * bb + 6 + D.R, D.be) + D.nlo, D.nbin - 1);
            }
            c->tile_tab.ensure(sizeof(SsTile)); c->brick_rng.ensure((size_t)D.nb * sizeof(int2));
            CK(cudaMemcpyAsync(c->tile_tab.p, &T, sizeof(SsTile), cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(c->brick_rng.p, h_rng.data(), (size_t)D.nb * sizeof(int2), cudaMemcpyHostToDevice, st));
            SsLsArgs A{};
            A.bin_start = c->tab_a.as<uint32_t>(); A.bin_end = c->tab_b.as<uint32_t>(); A.rec = c->rec.as<float4>();
            A.ksplit = c->ksplit.as<int>(); A.pidx = c->val_a.as<uint32_t>();
            A.tile_tab = c->tile_tab.as<SsTile>(); A.brick_rng = c->brick_rng.as<int2>(); A.tiles = c->tiles.as<float>();
            A.pairs = nullptr; A.wflag = nullptr; A.fix_bricks = nullptr; A.bstate = nullptr; A.mode = SS_LS_EXACT_ALL;
            const uint32_t n_work = build_worklist(c, D, 1);
            A.work_list = c->list_ls.as<uint32_t>();
            if (n_work) launch_levelset(c, dim3(n_work), D, A, false, false);
            CK(cudaStreamSynchronize(st));
        }
        CK(cudaMemcpyAsync(tile_out, c->tiles.p, np3 * 4, cudaMemcpyDefault, st));
        CK(cudaStreamSynchronize(st));
        return SS_OK;
    } catch (const SsCudaError &err) {
        cudaGetLastError();
        return ss_fail(err.e == cudaErrorMemoryAllocation ? SS_ERR_OUT_OF_MEMORY : SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}

// ------------------------------------------------------------------ multi-GPU: plan statistics + halo packing ----
// Slab plan input: particles per subdomain layer along the partition axis + occupancy of every subdomain slot (work model of
// distributed.py: particles + a fixed cost per occupied tile).  Owner cells are computed in plain f32: the plan only balances.
__global__ void k_part_stats(const float *__restrict__ xyz, uint32_t n, float3 gmin, float inv_sub, int3 nsd, int axis,
                             uint32_t *__restrict__ hist, uint32_t *__restrict__ occ) {
    __shared__ uint32_t s_hist[1024];
    const int nax = axis == 0 ? nsd.x : (axis == 1 ? nsd.y : nsd.z);
    for (int t = threadIdx.x; t < nax && t < 1024; t += blockDim.x) s_hist[t] = 0;
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int ix = min(max((int)floorf((xyz[3 * (uint64_t)i] - gmin.x) * inv_sub), 0), nsd.x - 1);
        const int iy = min(max((int)floorf((xyz[3 * (uint64_t)i + 1] - gmin.y) * inv_sub), 0), nsd.y - 1);
        const int iz = min(max((int)floorf((xyz[3 * (uint64_t)i + 2] - gmin.z) * inv_sub), 0), nsd.z - 1);
        const int ia = axis == 0 ? ix : (axis == 1 ? iy : iz);
        if (ia < 1024) atomicAdd(&s_hist[ia], 1u); else atomicAdd(&hist[ia], 1u);
        occ[(ix * nsd.y + iy) * nsd.z + iz] = 1u;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nax && t < 1024; t += blockDim.x) if (s_hist[t]) atomicAdd(&hist[t], s_hist[t]);
}
extern "C" int ss_partition_stats_f32(ss_context *c, const float *xyz, uint64_t n, const ss_grid_f32 *grid, uint32_t S, int axis,
                                      uint32_t *hist, uint32_t *occ) {
    if (!c || !grid || !hist || !occ || (n && !xyz) || axis < 0 || axis > 2 || S < 1) return ss_fail(SS_ERR_INVALID_PARAMETER, "bad argument");
    if (n >= 0xfffffff0ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many particles");
    try {
        CK(cudaSetDevice(c->device));
        int3 nsd;
        nsd.x = (int)((grid->cells_per_dim[0] + S - 1) / S); nsd.y = (int)((grid->cells_per_dim[1] + S - 1) / S); nsd.z = (int)((grid->cells_per_dim[2] + S - 1) / S);
        const int nax = axis == 0 ? nsd.x : (axis == 1 ? nsd.y : nsd.z);
        CK(cudaMemsetAsync(hist, 0, (size_t)nax * 4, c->stream));
        CK(cudaMemsetAsync(occ, 0, (size_t)nsd.x * nsd.y * nsd.z * 4, c->stream));
        if (n) {
            const float sub = fmulr(grid->cell_size, (float)S);
            const unsigned blocks = (unsigned)std::min<uint64_t>(nblk(n, 256), 148 * 8);
            LAUNCH(c, k_part_stats, blocks, 256, xyz, (uint32_t)n, make_float3(grid->aabb_min[0], grid->aabb_min[1], grid->aabb_min[2]), 1.0f / sub, nsd, axis, hist, occ);
        }
        CK(cudaStreamSynchronize(c->stream));
        return SS_OK;
    } catch (const SsCudaError &err) {
        cudaGetLastError();
        return ss_fail(SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}

// Plan statistics with the EXACT classifier: `members[slot]` = number of particles of this rank's input that are members (owner or
// ghost, dense_subdomains.rs:1810-1905) of subdomain `slot` -- summed over the ranks this is the subdomain's population, so the
// global maximum (sparse rule, dense_subdomains.rs:1242-1251) is known BEFORE any rank decomposes: the runner needs neither the
// decomposition pre-pass nor the callback.  `hist` as in ss_partition_stats_f32 (owner layer counts, for the balance only).
__global__ void k_part_members(SsDev P, const float *__restrict__ xyz, uint32_t n, int axis, uint32_t *__restrict__ hist, uint32_t *__restrict__ members) {
    __shared__ uint32_t s_hist[1024];
    const int nax = P.nsd[axis];
    for (int t = threadIdx.x; t < nax && t < 1024; t += blockDim.x) s_hist[t] = 0;
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float px = xyz[3 * (uint64_t)i], py = xyz[3 * (uint64_t)i + 1], pz = xyz[3 * (uint64_t)i + 2];
        const float pc = axis == 0 ? px : (axis == 1 ? py : pz);
        const int ia = min(max(ss_cell_of(pc, P.gmin[axis], P.sub_size), 0), nax - 1);
        if (ia < 1024) atomicAdd(&s_hist[ia], 1u); else atomicAdd(&hist[ia], 1u);
        ss_classify(P, px, py, pz, [&](int, int flat) { atomicAdd(&members[flat], 1u); });
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nax && t < 1024; t += blockDim.x) if (s_hist[t]) atomicAdd(&hist[t], s_hist[t]);
}
extern "C" int ss_partition_members_f32(ss_context *c, const float *xyz, uint64_t n, const ss_params_f32 *p, const ss_grid_f32 *grid, int axis,
                                        uint32_t *hist, uint32_t *members) {
    if (!c || !grid || !hist || !members || (n && !xyz) || axis < 0 || axis > 2) return ss_fail(SS_ERR_INVALID_PARAMETER, "bad argument");
    int rc = validate_params(p);
    if (rc) return rc;
    if (n >= 0xfffffff0ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many particles");
    try {
        CK(cudaSetDevice(c->device));
        // the decomposition parameters exactly as run_subdomain_grid derives them (dense_subdomains.rs:89-244)
        const int64_t S = (int64_t)p->subdomain_num_cubes_per_dim;
        const float h = p->compact_support_radius, cs = p->cube_size;
        SsDev D{};
        D.sub_size = fmulr(cs, (float)S);
        D.margin = fmulr(fmulr(ceilf(fdivr(h, cs)), cs), 1.01f);
        D.srad = (int)ceilf(fdivr(D.margin, D.sub_size));
        if (D.srad > 8) return ss_fail(SS_ERR_INVALID_PARAMETER, "ghost margin spans more than 8 subdomains; increase subdomain_num_cubes_per_dim");
        uint64_t nslots = 1;
        for (int d = 0; d < 3; ++d) { D.gmin[d] = grid->aabb_min[d]; D.nsd[d] = (int)((grid->cells_per_dim[d] + S - 1) / S); nslots *= (uint64_t)D.nsd[d]; }
        if (nslots >= 2147483647ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many subdomain slots");
        D.part_axis = 0; D.keep_lo = 0; D.keep_hi = 0x7fffffff;
        CK(cudaMemsetAsync(hist, 0, (size_t)D.nsd[axis] * 4, c->stream));
        CK(cudaMemsetAsync(members, 0, (size_t)nslots * 4, c->stream));
        if (n) {
            const unsigned blocks = (unsigned)std::min<uint64_t>(nblk(n, 256), (uint64_t)c->sm_count * 8);
            LAUNCH(c, k_part_members, blocks, 256, D, xyz, (uint32_t)n, axis, hist, members);
        }
        CK(cudaStreamSynchronize(c->stream));
        return SS_OK;
    } catch (const SsCudaError &err) {
        cudaGetLastError();
        return ss_fail(SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}

// Halo packing: destination d takes the particles with lo[d] <= coordinate < hi[d] along the partition axis (one particle may
// go to several destinations), ascending particle index preserved inside every destination.  One warp walks a chunk of
// SS_PACK_CHUNK particles in index order; pass 0 counts per (destination, chunk), an exclusive scan over the destination-major
// count table gives every chunk its output offset, pass 1 scatters.
#define SS_PACK_CHUNK 2048
#define SS_PACK_MAXW 64
struct SsPackIv { double lo[SS_PACK_MAXW], hi[SS_PACK_MAXW]; };
template <bool SCATTER>
__global__ void k_part_pack(const float *__restrict__ xyz, uint32_t n, int axis, SsPackIv iv, int world, uint32_t nchunks,
                            uint32_t *__restrict__ table /* [world][nchunks]: counts in, offsets for SCATTER */, float *__restrict__ send) {
    const uint32_t chunk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (chunk >= nchunks) return;
    const uint32_t first = chunk * SS_PACK_CHUNK, last = min(first + SS_PACK_CHUNK, n);
    for (int d = 0; d < world; ++d) {
        const double lo = iv.lo[d], hi = iv.hi[d];
        uint32_t run = SCATTER ? table[(size_t)d * nchunks + chunk] : 0u;
        for (uint32_t base = first; base < last; base += 32) {
            const uint32_t i = base + lane;
            bool in = false;
            float x = 0.f, y = 0.f, z = 0.f;
            if (i < last) {
                x = xyz[3 * (uint64_t)i]; y = xyz[3 * (uint64_t)i + 1]; z = xyz[3 * (uint64_t)i + 2];
                const double cax = (double)(axis == 0 ? x : (axis == 1 ? y : z));
                in = cax >= lo && cax < hi;
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, in);
            if (SCATTER && in) {
                const uint64_t o = (uint64_t)run + __popc(bal & ((1u << lane) - 1u));
                send[3 * o] = x; send[3 * o + 1] = y; send[3 * o + 2] = z;
            }
            run += __popc(bal);
        }
        if (!SCATTER && lane == 0) table[(size_t)d * nchunks + chunk] = run;
    }
}
// Two-phase: send == NULL counts (counts_out[world], host) and leaves the offset table in the context; the second call with a
// device buffer of sum(counts) * 3 floats scatters.  xyz is DEVICE memory.
extern "C" int ss_partition_pack_f32(ss_context *c, const float *xyz, uint64_t n, int axis, const double *lo, const double *hi, uint32_t world,
                                     uint64_t *counts_out, float *send) {
    if (!c || !lo || !hi || !counts_out || (n && !xyz) || axis < 0 || axis > 2 || world < 1 || world > SS_PACK_MAXW) return ss_fail(SS_ERR_INVALID_PARAMETER, "bad argument");
    if (n >= 0xfffffff0ull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "too many particles");
    try {
        CK(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        const uint32_t nchunks = (uint32_t)((n + SS_PACK_CHUNK - 1) / SS_PACK_CHUNK);
        for (uint32_t d = 0; d < world; ++d) counts_out[d] = 0;
        if (!n) return SS_OK;
        SsPackIv iv{};
        for (uint32_t d = 0; d < world; ++d) { iv.lo[d] = lo[d]; iv.hi[d] = hi[d]; }
        const size_t tab = (size_t)world * nchunks;
        c->pack_cnt.ensure(tab * 4); c->pack_off.ensure(tab * 4 + 4);
        const unsigned blocks = nblk((uint64_t)nchunks * 32, 128);
        if (!send) {
            LAUNCH(c, k_part_pack<false>, blocks, 128, xyz, (uint32_t)n, axis, iv, (int)world, nchunks, c->pack_cnt.as<uint32_t>(), (float *)nullptr);
            cub_excl_scan(c, c->pack_cnt.as<uint32_t>(), c->pack_off.as<uint32_t>(), (uint32_t)tab);
            std::vector<uint32_t> h_off(world), h_last(2);
            for (uint32_t d = 0; d < world; ++d) CK(cudaMemcpyAsync(&h_off[d], c->pack_off.as<uint32_t>() + (size_t)d * nchunks, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(&h_last[0], c->pack_off.as<uint32_t>() + (tab - 1), 4, cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(&h_last[1], c->pack_cnt.as<uint32_t>() + (tab - 1), 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            const uint64_t total = (uint64_t)h_last[0] + h_last[1];
            for (uint32_t d = 0; d < world; ++d) counts_out[d] = (d + 1 < world ? h_off[d + 1] : total) - h_off[d];
            c->pack_n = n; c->pack_world = world;
        } else {
            if (c->pack_n != n || c->pack_world != world) return ss_fail(SS_ERR_INVALID_PARAMETER, "ss_partition_pack_f32: scatter phase without a matching count phase");
            LAUNCH(c, k_part_pack<true>, blocks, 128, xyz, (uint32_t)n, axis, iv, (int)world, nchunks, c->pack_off.as<uint32_t>(), send);
            CK(cudaStreamSynchronize(st));
            c->pack_n = 0;
        }
        return SS_OK;
    } catch (const SsCudaError &err) {
        cudaGetLastError();
        return ss_fail(err.e == cudaErrorMemoryAllocation ? SS_ERR_OUT_OF_MEMORY : SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}

// ------------------------------------------------------------------ multi-GPU: one rank's slab of subdomains ----
static int reconstruct_partition_impl(ss_context *c, const float *xyz, uint64_t n_in, const ss_params_f32 *p, const ss_grid_f32 *grid,
                                      int axis, int64_t own_lo, int64_t own_hi, int64_t halo, uint64_t global_max_particles,
                                      int stop_after_decomposition, uint64_t (*max_reduce)(uint64_t, void *), void *user, ss_surface **out);
extern "C" int ss_reconstruct_partition_f32(ss_context *c, const float *xyz, uint64_t n_in, const ss_params_f32 *p, const ss_grid_f32 *grid,
                                            int axis, int64_t own_lo, int64_t own_hi, int64_t halo, uint64_t global_max_particles,
                                            int stop_after_decomposition, ss_surface **out) {
    return reconstruct_partition_impl(c, xyz, n_in, p, grid, axis, own_lo, own_hi, halo, global_max_particles, stop_after_decomposition, nullptr, nullptr, out);
}
extern "C" int ss_reconstruct_partition_cb_f32(ss_context *c, const float *xyz, uint64_t n_in, const ss_params_f32 *p, const ss_grid_f32 *grid,
                                               int axis, int64_t own_lo, int64_t own_hi, int64_t halo,
                                               uint64_t (*max_reduce)(uint64_t local_max, void *user), void *user, ss_surface **out) {
    return reconstruct_partition_impl(c, xyz, n_in, p, grid, axis, own_lo, own_hi, halo, 0, 0, max_reduce, user, out);
}
struct ReduceOnce {
    uint64_t (*fn)(uint64_t, void *); void *user; bool done = false;
    static uint64_t call(uint64_t v, void *self) { ReduceOnce *r = (ReduceOnce *)self; r->done = true; return r->fn(v, r->user); }
    ~ReduceOnce() { if (fn && !done) { done = true; fn(0, user); } }
};
static int reconstruct_partition_impl(ss_context *c, const float *xyz, uint64_t n_in, const ss_params_f32 *p, const ss_grid_f32 *grid,
                                      int axis, int64_t own_lo, int64_t own_hi, int64_t halo, uint64_t global_max_particles,
                                      int stop_after_decomposition, uint64_t (*max_reduce)(uint64_t, void *), void *user, ss_surface **out) {
    // The max-reduce callback is a collective: it runs exactly once on EVERY exit path below (argument errors, error returns and
    // CUDA failures included), so that a rank that fails cannot leave the others blocked in their all-reduce.
    ReduceOnce once{ max_reduce, user };
    if (!c || !out || !grid) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    *out = nullptr;
    int rc = validate_params(p);
    if (rc) return rc;
    if (p->has_particle_aabb) return ss_fail(SS_ERR_UNSUPPORTED, "filter particles before partitioning (particle_aabb is applied by the caller)");
    if (c->aniso) return ss_fail(SS_ERR_UNSUPPORTED, "anisotropic kernels are not available in partitioned reconstructions (the halo does not carry the kernel centres)");
    if (p->spatial_decomposition != 1) return ss_fail(SS_ERR_INVALID_PARAMETER, "partitioned reconstruction requires the subdomain grid");
    if (axis < 0 || axis > 2 || own_lo < 0 || own_hi < own_lo || halo < 0) return ss_fail(SS_ERR_INVALID_PARAMETER, "bad partition");
    if (n_in && !xyz) return ss_fail(SS_ERR_INVALID_PARAMETER, "xyz is NULL");
    ss_surface *s = nullptr;
    try {
        CK(cudaSetDevice(c->device));
        s = new ss_surface();
        s->device = c->device; s->n_in = n_in;
        c->launches = 0;
        Prepared P;
        g_devbuf_slack_eighths = 4;
        rc = prepare_particles(c, xyz, n_in, p, P, nullptr, grid);
        if (rc) { ss_surface_free(s); return rc; }
        s->n = P.n; s->grid = P.grid; s->used_decomposition = 1;
        Partition part;
        part.enabled = 1; part.axis = axis; part.own_lo = own_lo; part.own_hi = own_hi; part.halo = halo;
        part.global_max_particles = global_max_particles; part.stop_after_decomposition = stop_after_decomposition;
        part.max_reduce = max_reduce ? &ReduceOnce::call : nullptr; part.max_reduce_user = &once;
        rc = run_subdomain_grid(c, P, p, s, part);
        if (rc) { ss_surface_free(s); return rc; }
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1])); s->tm.upload = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2])); s->tm.aabb_and_grid = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[1], c->ev[9])); s->tm.total_device = ms;
        s->tm.kernel_launches = c->launches;
        *out = s;
        return SS_OK;
    } catch (const SsCudaError &err) {
        if (s) ss_surface_free(s);
        cudaGetLastError();
        char buf[512];
        snprintf(buf, sizeof(buf), "%s failed at %s:%d: %s", err.what, err.file, err.line, cudaGetErrorString(err.e));
        return ss_fail(err.e == cudaErrorMemoryAllocation ? SS_ERR_OUT_OF_MEMORY : SS_ERR_CUDA, buf);
    } catch (const std::bad_alloc &) {
        if (s) ss_surface_free(s);
        return ss_fail(SS_ERR_OUT_OF_MEMORY, "host allocation failed");
    }
}
extern "C" uint64_t ss_surface_max_subdomain_particles(const ss_surface *s) { return s ? s->max_particles : 0; }

// Welds vertices that carry the same MC edge key (duplicates on faces between ranks' slabs) in a concatenation of
// per-rank meshes.  All pointers are DEVICE memory: verts nv x 3 f32, keys nv u64 (as produced per vertex by
// ss_surface_device_vertex_keys), tris nt x 3 u32 (already offset to the concatenated numbering).  `cand` lists the
// n_cand vertex ids that may have duplicates.  Compacts verts/keys in place, rewrites tris, returns the new count.
extern "C" int ss_weld_meshes(ss_context *c, float *verts, unsigned long long *keys, uint64_t nv, uint32_t *tris, uint64_t nt,
                              const uint32_t *cand, uint64_t n_cand, uint64_t *nv_out) {
    if (!c || !nv_out) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    *nv_out = nv;
    if (!nv || !n_cand) return SS_OK;
    if (nv >= 0xfffffff0ull || n_cand >= 0x7fffffffull) return ss_fail(SS_ERR_INDEX_TOO_SMALL, "mesh too large");
    try {
        CK(cudaSetDevice(c->device));
        cudaStream_t st = c->stream;
        const uint32_t bc = (uint32_t)n_cand;
        c->bkeys_a.ensure((size_t)bc * 8); c->bkeys_b.ensure((size_t)bc * 8); c->bids_b.ensure((size_t)bc * 4);
        LAUNCH(c, k_gather_keys, nblk(bc, 256), 256, keys, cand, bc, c->bkeys_a.as<unsigned long long>());
        size_t tmp = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp, c->bkeys_a.as<unsigned long long>(), c->bkeys_b.as<unsigned long long>(),
                                           cand, c->bids_b.as<uint32_t>(), (int)bc, 0, 64, st));
        c->cub_tmp.ensure(tmp);
        CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, tmp, c->bkeys_a.as<unsigned long long>(), c->bkeys_b.as<unsigned long long>(),
                                           cand, c->bids_b.as<uint32_t>(), (int)bc, 0, 64, st));
        c->remap.ensure(nv * 4); c->keep.ensure(nv * 4); c->newid.ensure(nv * 4 + 4);
        LAUNCH(c, k_iota_keep, nblk(nv, 256), 256, (uint32_t)nv, c->remap.as<uint32_t>(), c->keep.as<uint32_t>());
        LAUNCH(c, k_weld_runs, nblk(bc, 256), 256, c->bkeys_b.as<unsigned long long>(), c->bids_b.as<uint32_t>(), bc,
               c->remap.as<uint32_t>(), c->keep.as<uint32_t>());
        cub_excl_scan(c, c->keep.as<uint32_t>(), c->newid.as<uint32_t>(), (uint32_t)nv);
        uint32_t lk = 0, ln = 0;
        CK(cudaMemcpyAsync(&lk, c->keep.as<uint32_t>() + (nv - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&ln, c->newid.as<uint32_t>() + (nv - 1), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const uint64_t nv_final = (uint64_t)lk + ln;
        DevBuf nverts, nkeys;
        nverts.ensure(nv_final * 12 + 16); nkeys.ensure(nv_final * 8 + 16);
        LAUNCH(c, k_compact_verts, nblk(nv, 256), 256, (uint32_t)nv, c->keep.as<uint32_t>(), c->newid.as<uint32_t>(), verts, keys,
               nverts.as<float>(), nkeys.as<unsigned long long>());
        if (nt) LAUNCH(c, k_remap_tris, nblk(nt * 3, 256), 256, nt * 3, c->remap.as<uint32_t>(), c->newid.as<uint32_t>(), tris);
        CK(cudaMemcpyAsync(verts, nverts.p, nv_final * 12, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(keys, nkeys.p, nv_final * 8, cudaMemcpyDeviceToDevice, st));
        CK(cudaStreamSynchronize(st));
        nverts.release(); nkeys.release();
        *nv_out = nv_final;
        return SS_OK;
    } catch (const SsCudaError &err) {
        cudaGetLastError();
        return ss_fail(err.e == cudaErrorMemoryAllocation ? SS_ERR_OUT_OF_MEMORY : SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}
extern "C" const unsigned long long *ss_surface_device_vertex_keys(const ss_surface *s) { return s ? s->vkeys.as<unsigned long long>() : nullptr; }
extern "C" int ss_surface_copy_subdomain_owned(const ss_surface *s, uint8_t *dst) {
    if (!s || !dst) return SS_ERR_INVALID_PARAMETER;
    for (uint64_t q = 0; q < s->nsub; ++q) dst[q] = s->sub_owned.empty() ? 1 : s->sub_owned[q];
    return SS_OK;
}

// ------------------------------------------------------------------ public entry ----
extern "C" int ss_reconstruct_surface_f32(ss_context *c, const float *xyz, uint64_t n_in, const ss_params_f32 *p, ss_surface **out) {
    if (!c || !out) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    *out = nullptr;
    int rc = validate_params(p);
    if (rc) return rc;
    if (n_in && !xyz) return ss_fail(SS_ERR_INVALID_PARAMETER, "xyz is NULL");
    ss_surface *s = nullptr;
    try {
        CK(cudaSetDevice(c->device));
        s = new ss_surface();
        s->device = c->device; s->n_in = n_in;
        c->launches = 0;
        Prepared P;
        rc = prepare_particles(c, xyz, n_in, p, P, &s->inside_aabb);
        if (rc) { ss_surface_free(s); return rc; }
        s->n = P.n; s->grid = P.grid;
        // decomposition decision, lib.rs:421-464
        int use_dec = 0;
        if (p->spatial_decomposition == 1) {
            if (p->auto_disable) {
                int64_t mc = std::max(P.grid.nc[0], std::max(P.grid.nc[1], P.grid.nc[2]));
                uint32_t with_margin = (uint32_t)(1.2 * (double)p->subdomain_num_cubes_per_dim);
                use_dec = (uint64_t)mc > (uint64_t)with_margin;
            } else use_dec = 1;
        }
        s->used_decomposition = use_dec;
        rc = run_subdomain_grid(c, P, p, s, Partition(), /*global_mode=*/!use_dec);
        if (rc) { ss_surface_free(s); return rc; }
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1])); s->tm.upload = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2])); s->tm.aabb_and_grid = ms;
        CK(cudaEventElapsedTime(&ms, c->ev[1], c->ev[9])); s->tm.total_device = ms;
        s->tm.kernel_launches = c->launches;
        *out = s;
        return SS_OK;
    } catch (const SsCudaError &err) {
        if (s) ss_surface_free(s);
        cudaGetLastError();
        char buf[512];
        snprintf(buf, sizeof(buf), "%s failed at %s:%d: %s", err.what, err.file, err.line, cudaGetErrorString(err.e));
        return ss_fail(err.e == cudaErrorMemoryAllocation ? SS_ERR_OUT_OF_MEMORY : SS_ERR_CUDA, buf);
    } catch (const std::bad_alloc &) {
        if (s) ss_surface_free(s);
        return ss_fail(SS_ERR_OUT_OF_MEMORY, "host allocation failed");
    }
}

static void give_back(DevBuf &slot, DevBuf &buf) {
    if (!buf.p) return;
    if (!slot.p) { slot = buf; buf.p = nullptr; buf.cap = 0; }
    else if (slot.cap < buf.cap) { cudaFree(slot.p); slot = buf; buf.p = nullptr; buf.cap = 0; }
    else buf.release();
}
extern "C" void ss_surface_free(ss_surface *s) {
    if (!s) return;
    cudaSetDevice(s->device);
    {
        std::lock_guard<std::mutex> lk(g_ctx_mutex);
        if (s->owner && g_live_contexts.count(s->owner)) {
            ss_context *c = s->owner;
            give_back(c->o_verts, s->verts); give_back(c->o_tris, s->tris); give_back(c->o_vkeys, s->vkeys); give_back(c->o_rho, s->rho);
            give_back(c->o_normals, s->normals);
            give_back(c->o_an_xbar, s->an_xbar); give_back(c->o_an_mat, s->an_mat); give_back(c->o_an_fac, s->an_fac);
        }
    }
    s->verts.release(); s->tris.release(); s->vkeys.release(); s->rho.release(); s->normals.release(); s->nbr_off.release(); s->nbr_idx.release();
    s->an_xbar.release(); s->an_mat.release(); s->an_fac.release();
    s->weights.release(); s->adj_row.release(); s->adj_idx.release(); s->inc_row.release(); s->inc_idx.release();
    delete s;
}

// ------------------------------------------------------------------ accessors ----
extern "C" uint64_t ss_surface_num_vertices(const ss_surface *s) { return s ? s->nv : 0; }
extern "C" uint64_t ss_surface_num_triangles(const ss_surface *s) { return s ? s->nt : 0; }
extern "C" uint64_t ss_surface_num_particles(const ss_surface *s) { return s ? s->n : 0; }
extern "C" uint64_t ss_surface_num_subdomains(const ss_surface *s) { return s ? s->nsub : 0; }
extern "C" int ss_surface_used_decomposition(const ss_surface *s) { return s ? s->used_decomposition : 0; }
extern "C" int ss_surface_grid(const ss_surface *s, ss_grid_f32 *o) { if (!s || !o) return SS_ERR_INVALID_PARAMETER; grid_to_abi(s->grid, o); return SS_OK; }
extern "C" int ss_surface_subdomain_grid(const ss_surface *s, ss_grid_f32 *o) {
    if (!s || !o) return SS_ERR_INVALID_PARAMETER;
    if (!s->used_decomposition) return ss_fail(SS_ERR_INVALID_PARAMETER, "no subdomain grid: decomposition was not used");
    grid_to_abi(s->subgrid, o); return SS_OK;
}
static int copy_out(const ss_surface *s, void *dst, const void *src, size_t bytes, bool widen = false) {
    if (!s || (!dst && bytes)) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    if (!bytes) return SS_OK;
    cudaSetDevice(s->device);
    ss_context *c = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_ctx_mutex);
        if (s->owner && g_live_contexts.count(s->owner)) c = s->owner;
    }
    bool pinned_dst = false;
    {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, dst) == cudaSuccess) pinned_dst = at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
        else cudaGetLastError();
    }
    const size_t SS_STAGE_BYTES = c ? c->stage_bytes : SS_STAGE_BYTES_MAX;                // chunk size (tests shrink it)
    if (!c || (pinned_dst && !widen) || bytes < 4 * SS_STAGE_BYTES) {
        if (!widen) {
            cudaError_t e = cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) return ss_fail(SS_ERR_CUDA, cudaGetErrorString(e));
            return SS_OK;
        }
        std::vector<uint32_t> tmp(bytes / 4);
        cudaError_t e = cudaMemcpy(tmp.data(), src, bytes, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return ss_fail(SS_ERR_CUDA, cudaGetErrorString(e));
        scatter_chunk(static_cast<char *>(dst), reinterpret_cast<const char *>(tmp.data()), bytes, true);
        return SS_OK;
    }
    try {
        for (int q = 0; q < 2; ++q) if (!c->h_stage[q]) {
            if (cudaHostAlloc(&c->h_stage[q], SS_STAGE_BYTES_MAX, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); c->h_stage[q] = nullptr; }
        }
        if (!c->h_stage[0] || !c->h_stage[1]) {                      // cannot page-lock: the plain copy still works
            if (widen) { std::vector<uint32_t> tmp(bytes / 4); CK(cudaMemcpy(tmp.data(), src, bytes, cudaMemcpyDeviceToHost)); scatter_chunk(static_cast<char *>(dst), reinterpret_cast<const char *>(tmp.data()), bytes, true); }
            else CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
            return SS_OK;
        }
        cudaStream_t st = c->stream;
        const size_t nchunks = (bytes + SS_STAGE_BYTES - 1) / SS_STAGE_BYTES;
        auto issue = [&](size_t k) {
            const size_t off = k * SS_STAGE_BYTES, n = std::min(SS_STAGE_BYTES, bytes - off);
            CK(cudaMemcpyAsync(c->h_stage[k & 1], static_cast<const char *>(src) + off, n, cudaMemcpyDeviceToHost, st));
            CK(cudaEventRecord(c->ev_stage[k & 1], st));
        };
        issue(0);
        for (size_t k = 0; k < nchunks; ++k) {
            if (k + 1 < nchunks) issue(k + 1);                       // its staging buffer was scattered in the previous iteration
            CK(cudaEventSynchronize(c->ev_stage[k & 1]));
            const size_t off = k * SS_STAGE_BYTES, n = std::min(SS_STAGE_BYTES, bytes - off);
            scatter_chunk(static_cast<char *>(dst) + (widen ? 2 * off : off), static_cast<const char *>(c->h_stage[k & 1]), n, widen);
        }
        return SS_OK;
    } catch (const SsCudaError &err) {
        cudaGetLastError();
        return ss_fail(SS_ERR_CUDA, std::string(err.what) + ": " + cudaGetErrorString(err.e));
    }
}
extern "C" int ss_surface_copy_vertices(const ss_surface *s, float *dst) { return copy_out(s, dst, s ? s->verts.p : nullptr, s ? s->nv * 12 : 0); }
extern "C" int ss_surface_copy_triangles_u32(const ss_surface *s, uint32_t *dst) { return copy_out(s, dst, s ? s->tris.p : nullptr, s ? s->nt * 12 : 0); }
extern "C" int ss_surface_copy_triangles_u64(const ss_surface *s, uint64_t *dst) {      /* usize like the reference: widened on the host */
    if (!s || (!dst && s->nt)) return ss_fail(SS_ERR_INVALID_PARAMETER, "NULL argument");
    return copy_out(s, dst, s->tris.p, s->nt * 12, true);
}
extern "C" int ss_surface_copy_particle_densities(const ss_surface *s, float *dst) { return copy_out(s, dst, s ? s->rho.p : nullptr, s ? s->n * 4 : 0); }
extern "C" int ss_surface_copy_particle_inside_aabb(const ss_surface *s, uint8_t *dst) {
    if (!s || !dst) return SS_ERR_INVALID_PARAMETER;
    if (s->inside_aabb.empty()) return ss_fail(SS_ERR_INVALID_PARAMETER, "no particle AABB was specified");
    memcpy(dst, s->inside_aabb.data(), s->inside_aabb.size());
    return SS_OK;
}
// Page-locked host memory for callers without a CUDA binding of their own (the Python mirror's reusable result buffers): device ->
// host copies into it run at PCIe speed and touch no fresh pages.
extern "C" void *ss_host_alloc_pinned(uint64_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void ss_host_free_pinned(void *p) { if (p) cudaFreeHost(p); }
extern "C" const float *ss_surface_device_vertices(const ss_surface *s) { return s ? s->verts.as<float>() : nullptr; }
extern "C" const uint32_t *ss_surface_device_triangles(const ss_surface *s) { return s ? s->tris.as<uint32_t>() : nullptr; }
extern "C" const float *ss_surface_device_densities(const ss_surface *s) { return s ? s->rho.as<float>() : nullptr; }

extern "C" int ss_surface_copy_vertex_edge_keys(const ss_surface *s, int64_t *dst) {
    if (!s || (!dst && s->nv)) return SS_ERR_INVALID_PARAMETER;
    std::vector<unsigned long long> k(s->nv);
    int rc = copy_out(s, k.data(), s->vkeys.p, s->nv * 8);
    if (rc) return rc;
    for (uint64_t v = 0; v < s->nv; ++v) {
        dst[4 * v] = (int64_t)((k[v] >> 42) & 0xfffff); dst[4 * v + 1] = (int64_t)((k[v] >> 22) & 0xfffff);
        dst[4 * v + 2] = (int64_t)((k[v] >> 2) & 0xfffff); dst[4 * v + 3] = (int64_t)(k[v] & 3);
    }
    return SS_OK;
}
extern "C" int ss_surface_copy_subdomains(const ss_surface *s, int64_t *flat, uint64_t *count, uint8_t *sparse) {
    if (!s) return SS_ERR_INVALID_PARAMETER;
    for (uint64_t q = 0; q < s->nsub; ++q) {
        if (flat) flat[q] = s->sub_flat[q];
        if (count) count[q] = s->sub_count[q];
        if (sparse) sparse[q] = s->sub_sparse[q];
    }
    return SS_OK;
}
extern "C" int ss_surface_copy_levelset_tile(const ss_surface *s, float *dst) {
    if (!s || !dst) return SS_ERR_INVALID_PARAMETER;
    if (s->tile.empty()) return ss_fail(SS_ERR_INVALID_PARAMETER, "no level-set tile was kept (ss_context_keep_levelset_tile)");
    memcpy(dst, s->tile.data(), s->tile.size() * 4);
    return SS_OK;
}
extern "C" uint64_t ss_surface_num_neighbors(const ss_surface *s) { return (s && s->has_neighbors) ? s->n_neighbors : 0; }
extern "C" int ss_surface_copy_neighbor_lists(const ss_surface *s, uint64_t *offsets, uint32_t *indices) {
    if (!s) return SS_ERR_INVALID_PARAMETER;
    if (!s->has_neighbors) return ss_fail(SS_ERR_INVALID_PARAMETER, "neighbor lists were not requested (Parameters::global_neighborhood_list)");
    int rc = SS_OK;
    if (offsets) rc = copy_out(s, offsets, s->nbr_off.p, (s->n + 1) * 8);
    if (!rc && indices) rc = copy_out(s, indices, s->nbr_idx.p, s->n_neighbors * 4);
    return rc;
}
extern "C" int ss_surface_timings(const ss_surface *s, ss_timings *o) { if (!s || !o) return SS_ERR_INVALID_PARAMETER; *o = s->tm; return SS_OK; }

#include "ss_post.cuh"
#include "ss_meshproc.inc"
#include "ss_meshio.inc"
