// ss_aniso.cuh -- anisotropic-kernel level set (Yu & Turk 2013, "Reconstructing Surfaces of Particle-Based Fluids Using
// Anisotropic Kernels"), the opt-in alternative to the isotropic splat of ss_kernels.cuh / ss_exact.cuh (included once by
// ss_pipeline.cu; see DESIGN.md "Anisotropic kernels").
//
//   k_aniso_moments[_global]   per particle: weighted neighbourhood mean and covariance over the density stage's neighbours,
//                              3x3 Jacobi eigen-decomposition, smoothed centre x_bar, ellipsoid matrix M = R^2 A and factor f
//   k_aniso_records            bin-sorted (M, f) next to the bin-sorted x_bar records of stage_binning
//   k_aniso_levelset_warp      one warp per 8^3-point brick: L(x) = sum_i f_i W_R(sqrt(u^T M_i u)), u = x - x_bar_i
//
// Every value is computed with explicit round-to-nearest intrinsics in a fixed order (no float atomics), so the result does not
// depend on the launch configuration and the CPU executor (tests/emul/cuda_emul.h) computes the same bits.
#pragma once
#include "ss_kernels.cuh"

struct SsAniso {
    float max_ratio;        // k_r >= 1: smallest principal radius = R / k_r
    uint32_t min_neighbors; // N_eps: fewer neighbours -> isotropic kernel
    float smoothing;        // lambda in [0, 1]: x_bar = x + lambda * mu
};

#define SS_AN_SWEEPS 8       // Jacobi sweep cap (a sweep = 3 rotations); converges to f32 precision in <= 5 on 3x3 covariances

// Symmetric 3x3 eigen-decomposition a = Q diag(ev) Q^T by cyclic Jacobi rotations, in registers.  a: xx xy xz yy yz zz.
// q[r][k]: component r of eigenvector k.  Returns the sweeps used.
__device__ __forceinline__ int ss_jacobi3(const float a_in[6], float ev[3], float q[3][3]) {
    float a[3][3] = { { a_in[0], a_in[1], a_in[2] }, { a_in[1], a_in[3], a_in[4] }, { a_in[2], a_in[4], a_in[5] } };
#pragma unroll
    for (int r = 0; r < 3; ++r) for (int k = 0; k < 3; ++k) q[r][k] = r == k ? 1.0f : 0.0f;
    int sweeps = 0;
    for (; sweeps < SS_AN_SWEEPS; ++sweeps) {
        const float off = __fadd_rn(__fadd_rn(__fmul_rn(a[0][1], a[0][1]), __fmul_rn(a[0][2], a[0][2])), __fmul_rn(a[1][2], a[1][2]));
        const float dia = __fadd_rn(__fadd_rn(__fmul_rn(a[0][0], a[0][0]), __fmul_rn(a[1][1], a[1][1])), __fmul_rn(a[2][2], a[2][2]));
        if (!(off > __fmul_rn(1.0e-14f, dia))) break;
#pragma unroll
        for (int pq = 0; pq < 3; ++pq) {
            const int p = pq == 2 ? 1 : 0, r = pq == 0 ? 1 : 2;
            const float apq = a[p][r];
            if (apq == 0.0f) continue;
            const float theta = __fdiv_rn(__fsub_rn(a[r][r], a[p][p]), __fmul_rn(2.0f, apq));
            const float at = fabsf(theta);
            float t = at > 1.0e18f ? __fdiv_rn(0.5f, at) : __fdiv_rn(1.0f, __fadd_rn(at, __fsqrt_rn(__fadd_rn(__fmul_rn(at, at), 1.0f))));
            if (theta < 0.0f) t = -t;
            const float cs = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(__fmul_rn(t, t), 1.0f)));
            const float sn = __fmul_rn(t, cs);
            // a <- J^T a J with J the rotation in the (p, r) plane
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float akp = a[k][p], akr = a[k][r];
                a[k][p] = __fsub_rn(__fmul_rn(cs, akp), __fmul_rn(sn, akr));
                a[k][r] = __fadd_rn(__fmul_rn(sn, akp), __fmul_rn(cs, akr));
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float apk = a[p][k], ark = a[r][k];
                a[p][k] = __fsub_rn(__fmul_rn(cs, apk), __fmul_rn(sn, ark));
                a[r][k] = __fadd_rn(__fmul_rn(sn, apk), __fmul_rn(cs, ark));
            }
            a[p][r] = 0.0f; a[r][p] = 0.0f;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float qkp = q[k][p], qkr = q[k][r];
                q[k][p] = __fsub_rn(__fmul_rn(cs, qkp), __fmul_rn(sn, qkr));
                q[k][r] = __fadd_rn(__fmul_rn(sn, qkp), __fmul_rn(cs, qkr));
            }
        }
    }
    ev[0] = a[0][0]; ev[1] = a[1][1]; ev[2] = a[2][2];
    return sweeps;
}

// Moment accumulator of one particle: weight sum (self included with weight 1), first and second moments of d = x_j - x_i.
struct SsAnAcc {
    float w, m[3], s[6];
    unsigned cnt;
};
__device__ __forceinline__ void ss_an_add(SsAnAcc &A, float dx, float dy, float dz, float d2, float inv_r) {
    const float q = __fmul_rn(__fsqrt_rn(d2), inv_r);
    const float w = __fsub_rn(1.0f, __fmul_rn(__fmul_rn(q, q), q));
    const float wx = __fmul_rn(w, dx), wy = __fmul_rn(w, dy), wz = __fmul_rn(w, dz);
    A.w = __fadd_rn(A.w, w);
    A.m[0] = __fadd_rn(A.m[0], wx); A.m[1] = __fadd_rn(A.m[1], wy); A.m[2] = __fadd_rn(A.m[2], wz);
    A.s[0] = __fadd_rn(A.s[0], __fmul_rn(wx, dx)); A.s[1] = __fadd_rn(A.s[1], __fmul_rn(wx, dy)); A.s[2] = __fadd_rn(A.s[2], __fmul_rn(wx, dz));
    A.s[3] = __fadd_rn(A.s[3], __fmul_rn(wy, dy)); A.s[4] = __fadd_rn(A.s[4], __fmul_rn(wy, dz)); A.s[5] = __fadd_rn(A.s[5], __fmul_rn(wz, dz));
    ++A.cnt;
}

// Steps 2-4 of the definition (DESIGN.md): x_bar, M = R^2 A (= Q diag(s1^2 / s_k^2) Q^T) and f = (m / rho) R^3 / (a1 a2 a3).
__device__ __forceinline__ void ss_an_finish(const SsDev &P, const SsAniso &K, const SsAnAcc &A, float4 pi, float rho_i,
                                             float *__restrict__ xbar, float *__restrict__ mat, float *__restrict__ fac,
                                             unsigned *__restrict__ max_sweeps) {
    const uint32_t p = __float_as_uint(pi.w);
    const float mu[3] = { __fdiv_rn(A.m[0], A.w), __fdiv_rn(A.m[1], A.w), __fdiv_rn(A.m[2], A.w) };
    const float cov[6] = {
        __fsub_rn(__fdiv_rn(A.s[0], A.w), __fmul_rn(mu[0], mu[0])), __fsub_rn(__fdiv_rn(A.s[1], A.w), __fmul_rn(mu[0], mu[1])),
        __fsub_rn(__fdiv_rn(A.s[2], A.w), __fmul_rn(mu[0], mu[2])), __fsub_rn(__fdiv_rn(A.s[3], A.w), __fmul_rn(mu[1], mu[1])),
        __fsub_rn(__fdiv_rn(A.s[4], A.w), __fmul_rn(mu[1], mu[2])), __fsub_rn(__fdiv_rn(A.s[5], A.w), __fmul_rn(mu[2], mu[2])) };
    xbar[3 * (uint64_t)p] = __fadd_rn(pi.x, __fmul_rn(K.smoothing, mu[0]));
    xbar[3 * (uint64_t)p + 1] = __fadd_rn(pi.y, __fmul_rn(K.smoothing, mu[1]));
    xbar[3 * (uint64_t)p + 2] = __fadd_rn(pi.z, __fmul_rn(K.smoothing, mu[2]));
    float ev[3], q[3][3];
    const int sweeps = ss_jacobi3(cov, ev, q);
    if (max_sweeps) atomicMax(max_sweeps, (unsigned)sweeps);     // statistic only, not part of any result
    const float s1 = fmaxf(ev[0], fmaxf(ev[1], ev[2]));
    float m6[6] = { 1.0f, 0.0f, 0.0f, 1.0f, 0.0f, 1.0f };
    float f = __fdiv_rn(P.rest_mass, rho_i);
    if (A.cnt >= K.min_neighbors && s1 > 0.0f) {
        // t_k = a_k / R = max(sigma_k, sigma_1 / k_r) / sigma_1 in [1 / k_r, 1]; M = Q diag(1 / t_k^2) Q^T
        const float floor_s = __fdiv_rn(s1, K.max_ratio);
        float inv_t2[3], prod = 1.0f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float t = __fdiv_rn(fmaxf(ev[k], floor_s), s1);
            inv_t2[k] = __fdiv_rn(1.0f, __fmul_rn(t, t));
            prod = __fmul_rn(prod, t);
        }
#pragma unroll
        for (int e = 0; e < 6; ++e) {
            const int ia = e < 3 ? 0 : (e < 5 ? 1 : 2), ib = e < 3 ? e : (e < 5 ? e - 2 : 2);
            float v = 0.0f;
#pragma unroll
            for (int k = 0; k < 3; ++k) v = __fadd_rn(v, __fmul_rn(__fmul_rn(q[ia][k], q[ib][k]), inv_t2[k]));
            m6[e] = v;
        }
        f = __fdiv_rn(f, prod);
    }
#pragma unroll
    for (int e = 0; e < 6; ++e) mat[6 * (uint64_t)p + e] = m6[e];
    fac[p] = f;
}

// Subdomain path: one thread per membership entry in neighbourhood-search order; entries whose particle lies inside the
// subdomain (one per particle, the entries k_density evaluates) walk the same 27 cells in the same order as ss_density_entry.
__global__ void __launch_bounds__(128, 1)
k_aniso_moments(SsDev P, SsAniso K, uint32_t m, const uint32_t *__restrict__ key, const float4 *__restrict__ spos,
                const uint32_t *__restrict__ sub_flat, const uint32_t *__restrict__ cstart, const uint32_t *__restrict__ cend,
                const float *__restrict__ rho, float *__restrict__ xbar, float *__restrict__ mat, float *__restrict__ fac,
                unsigned *__restrict__ max_sweeps) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const uint32_t k = key[e];
    const uint32_t s = k / (uint32_t)P.ns_stride, cell = k - s * (uint32_t)P.ns_stride;
    const float4 pi = spos[e];
    const SsSubGeom g = ss_sub_geom(P, sub_flat[s]);
    if (!((pi.x >= g.smin[0] && pi.y >= g.smin[1] && pi.z >= g.smin[2]) && (pi.x < g.smax[0] && pi.y < g.smax[1] && pi.z < g.smax[2]))) return;
    const SsNsGrid ns = ss_ns_grid(P, g);
    const int c0 = (int)cell / (P.nsD * P.nsD), c1 = ((int)cell / P.nsD) % P.nsD, c2 = (int)cell % P.nsD;
    const float inv_r = __fdiv_rn(1.0f, P.h);
    SsAnAcc A{ 1.0f, { 0.0f, 0.0f, 0.0f }, { 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f }, 0u };
    const uint32_t base = s * (uint32_t)P.ns_stride;
    for (int pass = 0; pass < 2; ++pass) {
        for (int sx = -1; sx <= 1; ++sx) for (int sy = -1; sy <= 1; ++sy) for (int sz = -1; sz <= 1; ++sz) {
            const bool self = (sx == 0 && sy == 0 && sz == 0);
            if ((pass == 0) == self) continue;
            const int q0 = c0 + sx, q1 = c1 + sy, q2 = c2 + sz;
            if (q0 < 0 || q1 < 0 || q2 < 0 || q0 >= ns.nc[0] || q1 >= ns.nc[1] || q2 >= ns.nc[2]) continue;
            const uint32_t kk = base + (uint32_t)((q0 * P.nsD + q1) * P.nsD + q2);
            const uint32_t a = cstart[kk];
            if (a == 0xffffffffu) continue;
            const uint32_t b = cend[kk];
            for (uint32_t t = a; t < b; ++t) {
                if (t == e) continue;
                const float4 pj = spos[t];
                const float dx = __fsub_rn(pj.x, pi.x), dy = __fsub_rn(pj.y, pi.y), dz = __fsub_rn(pj.z, pi.z);
                const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                if (d2 < P.h2) ss_an_add(A, dx, dy, dz, d2, inv_r);
            }
        }
    }
    ss_an_finish(P, K, A, pi, rho[__float_as_uint(pi.w)], xbar, mat, fac, max_sweeps);
}

// Global path: one thread per particle over the whole-domain cell list (the walk of k_density_global).
__global__ void __launch_bounds__(128, 1)
k_aniso_moments_global(SsDev P, SsAniso K, uint32_t n, const uint32_t *__restrict__ key, const float4 *__restrict__ spos,
                       const uint32_t *__restrict__ cstart, const uint32_t *__restrict__ cend, const float *__restrict__ rho,
                       float *__restrict__ xbar, float *__restrict__ mat, float *__restrict__ fac, unsigned *__restrict__ max_sweeps) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int cell = (int)key[e];
    const int n1 = P.g_ns_nc[1], n2 = P.g_ns_nc[2];
    const int c0 = cell / (n1 * n2), c1 = (cell / n2) % n1, c2 = cell % n2;
    const float4 pi = spos[e];
    const float inv_r = __fdiv_rn(1.0f, P.h);
    SsAnAcc A{ 1.0f, { 0.0f, 0.0f, 0.0f }, { 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f }, 0u };
    for (int pass = 0; pass < 2; ++pass) {
        for (int sx = -1; sx <= 1; ++sx) for (int sy = -1; sy <= 1; ++sy) for (int sz = -1; sz <= 1; ++sz) {
            const bool self = (sx == 0 && sy == 0 && sz == 0);
            if ((pass == 0) == self) continue;
            const int q0 = c0 + sx, q1 = c1 + sy, q2 = c2 + sz;
            if (q0 < 0 || q1 < 0 || q2 < 0 || q0 >= P.g_ns_nc[0] || q1 >= n1 || q2 >= n2) continue;
            const uint32_t kk = (uint32_t)((q0 * n1 + q1) * n2 + q2);
            const uint32_t a = cstart[kk];
            if (a == 0xffffffffu) continue;
            const uint32_t b = cend[kk];
            for (uint32_t t = a; t < b; ++t) {
                if (t == e) continue;
                const float4 pj = spos[t];
                const float dx = __fsub_rn(pj.x, pi.x), dy = __fsub_rn(pj.y, pi.y), dz = __fsub_rn(pj.z, pi.z);
                const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                if (d2 < P.h2) ss_an_add(A, dx, dy, dz, d2, inv_r);
            }
        }
    }
    ss_an_finish(P, K, A, pi, rho[__float_as_uint(pi.w)], xbar, mat, fac, max_sweeps);
}

// Bin-sorted ellipsoid data next to stage_binning's records (rec = x_bar, V): am[2e] = (Mxx, Mxy, Mxz, Myy), am[2e+1] =
// (Myz, Mzz, f, 0).  On the global path a particle outside the allowed domain (density_map.rs:606-610, tested on its original
// position) is not splatted by the isotropic path either: f = 0.
__global__ void k_aniso_records(SsDev P, uint32_t m, const uint32_t *__restrict__ key, const uint32_t *__restrict__ pidx,
                                const float *__restrict__ xyz, const float *__restrict__ mat, const float *__restrict__ fac,
                                float4 *__restrict__ am) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m || key[e] == 0xffffffffu) return;
    const uint32_t p = pidx[e];
    float f = fac[p];
    if (P.gmode) {
        bool allowed = true;
#pragma unroll
        for (int d = 0; d < 3; ++d) { const float x = xyz[3 * (uint64_t)p + d]; allowed = allowed && x >= P.g_allow_min[d] && x < P.g_allow_max[d]; }
        if (!allowed) f = 0.0f;
    }
    const float *M = mat + 6 * (uint64_t)p;
    am[2 * (uint64_t)e] = make_float4(M[0], M[1], M[2], M[3]);
    am[2 * (uint64_t)e + 1] = make_float4(M[4], M[5], f, 0.0f);
}

#define SS_AW_WARPS 4        // warps (bricks) per CTA
struct SsAwArgs {
    const uint32_t *bin_start, *bin_end;   // [nsub * nbin_sub] runs of the x_bar bins
    const float4 *rec;                      // bin-sorted (x_bar, V)
    const float4 *am;                       // bin-sorted (M, f), k_aniso_records
    const SsTile *tile_tab;
    const int2 *brick_rng;
    uint32_t n_bricks;                      // ntiles * nb^3
    float *tiles;                           // [batch][np^3]: every point is written
    uint8_t *bstate;                        // [batch][nb^3]: 2 where a candidate reaches the brick, 0 (all values zero) elsewhere
};

// One warp per brick of a batch (every brick, no work list): the candidates of the brick's bins are staged 32 at a time, culled
// against the brick's box, and every lane folds them into its 16 points in bin order.  Values are exact everywhere (the
// exact_everywhere format the marching-cubes kernels read); no certification.
__global__ void __launch_bounds__(SS_AW_WARPS * 32, 1)
k_aniso_levelset_warp(SsDev P, SsAwArgs A) {
    __shared__ float s_c[SS_AW_WARPS][32][11];      // x_bar (3), M (6), f, pad
    __shared__ uint32_t s_run[SS_AW_WARPS][128][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t brick_lin = blockIdx.x * SS_AW_WARPS + warp;
    if (brick_lin >= A.n_bricks) return;             // whole warps exit together: no collective below is divergent
    const int nb = P.nb;
    uint32_t q = brick_lin;
    const int bz = (int)(q % (uint32_t)nb); q /= (uint32_t)nb;
    const int by = (int)(q % (uint32_t)nb); q /= (uint32_t)nb;
    const int bx = (int)(q % (uint32_t)nb);
    const uint32_t tile_idx = q / (uint32_t)nb;
    const SsTile T = A.tile_tab[tile_idx];
    const int2 rx = A.brick_rng[bx], ry = A.brick_rng[by], rz = A.brick_rng[bz];
    const int nyr = ry.y - ry.x + 1, nruns = (rx.y - rx.x + 1) * nyr;    // <= 128 (host check)
    for (int r = lane; r < nruns; r += 32) {
        const int X = rx.x + r / nyr, Y = ry.x + r % nyr;
        uint32_t a = 0xffffffffu, b = 0;
        const uint32_t base = T.s * (uint32_t)P.nbin_sub + (uint32_t)((X * P.nbin + Y) * P.nbin);
        for (int Z = rz.x; Z <= rz.y; ++Z) {
            const uint32_t st = A.bin_start[base + Z];
            if (st != 0xffffffffu) { if (a == 0xffffffffu) a = st; b = A.bin_end[base + Z]; }
        }
        s_run[warp][r][0] = a; s_run[warp][r][1] = a == 0xffffffffu ? 0u : b - a;
    }
    __syncwarp();
    // brick box in world coordinates (cull only; conservative slack)
    const int i0 = bx * 8, j0 = by * 8, k0 = bz * 8;
    const int i1 = min(i0 + 7, P.np - 1), j1 = min(j0 + 7, P.np - 1), k1 = min(k0 + 7, P.np - 1);
    const float blo[3] = { __fadd_rn(__fmul_rn((float)(T.gbase[0] + i0), P.c), P.gmin[0]), __fadd_rn(__fmul_rn((float)(T.gbase[1] + j0), P.c), P.gmin[1]),
                           __fadd_rn(__fmul_rn((float)(T.gbase[2] + k0), P.c), P.gmin[2]) };
    const float bhi[3] = { __fadd_rn(__fmul_rn((float)(T.gbase[0] + i1), P.c), P.gmin[0]), __fadd_rn(__fmul_rn((float)(T.gbase[1] + j1), P.c), P.gmin[1]),
                           __fadd_rn(__fmul_rn((float)(T.gbase[2] + k1), P.c), P.gmin[2]) };
    const float cull2 = __fmul_rn(P.h2, 1.0001f);
    float phi[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) phi[t] = 0.0f;
    bool touched = false;
    for (int r = 0; r < nruns; ++r) {
        const uint32_t a = s_run[warp][r][0], len = s_run[warp][r][1];
        for (uint32_t c0 = 0; c0 < len; c0 += 32) {
            bool keep = false;
            float4 x4 = make_float4(0.f, 0.f, 0.f, 0.f), m0 = x4, m1 = x4;
            if (c0 + lane < len) {
                const uint32_t e = a + c0 + lane;
                x4 = A.rec[e]; m0 = A.am[2 * (uint64_t)e]; m1 = A.am[2 * (uint64_t)e + 1];
                const float dx = fmaxf(fmaxf(blo[0] - x4.x, x4.x - bhi[0]), 0.0f);
                const float dy = fmaxf(fmaxf(blo[1] - x4.y, x4.y - bhi[1]), 0.0f);
                const float dz = fmaxf(fmaxf(blo[2] - x4.z, x4.z - bhi[2]), 0.0f);
                keep = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)) < cull2 && m1.z != 0.0f;
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                float *d = s_c[warp][__popc(bal & ((1u << lane) - 1u))];
                d[0] = x4.x; d[1] = x4.y; d[2] = x4.z; d[3] = m0.x; d[4] = m0.y; d[5] = m0.z; d[6] = m0.w; d[7] = m1.x; d[8] = m1.y; d[9] = m1.z;
            }
            __syncwarp();
            const int nk = __popc(bal);
            touched = touched || nk > 0;
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const int idx = lane + 32 * t;
                const int i = i0 + (idx >> 6), j = j0 + ((idx >> 3) & 7), k = k0 + (idx & 7);
                const float gx = __fadd_rn(__fmul_rn((float)(T.gbase[0] + i), P.c), P.gmin[0]);
                const float gy = __fadd_rn(__fmul_rn((float)(T.gbase[1] + j), P.c), P.gmin[1]);
                const float gz = __fadd_rn(__fmul_rn((float)(T.gbase[2] + k), P.c), P.gmin[2]);
                float v = phi[t];
                for (int n = 0; n < nk; ++n) {
                    const float *d = s_c[warp][n];
                    const float ux = __fsub_rn(gx, d[0]), uy = __fsub_rn(gy, d[1]), uz = __fsub_rn(gz, d[2]);
                    const float mx = __fadd_rn(__fadd_rn(__fmul_rn(d[3], ux), __fmul_rn(d[4], uy)), __fmul_rn(d[5], uz));
                    const float my = __fadd_rn(__fadd_rn(__fmul_rn(d[4], ux), __fmul_rn(d[6], uy)), __fmul_rn(d[7], uz));
                    const float mz = __fadd_rn(__fadd_rn(__fmul_rn(d[5], ux), __fmul_rn(d[7], uy)), __fmul_rn(d[8], uz));
                    const float q2 = __fadd_rn(__fadd_rn(__fmul_rn(ux, mx), __fmul_rn(uy, my)), __fmul_rn(uz, mz));
                    if (q2 < P.h2) v = __fadd_rn(v, __fmul_rn(d[9], ss_kernel_scalar(P, __fsqrt_rn(q2))));
                }
                phi[t] = v;
            }
            __syncwarp();
        }
    }
    const size_t np = (size_t)P.np, tbase = (size_t)tile_idx * np * np * np;
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        const int idx = lane + 32 * t;
        const int i = i0 + (idx >> 6), j = j0 + ((idx >> 3) & 7), k = k0 + (idx & 7);
        if (i < P.np && j < P.np && k < P.np) A.tiles[tbase + ((size_t)i * np + j) * np + k] = phi[t];
    }
    if (lane == 0) A.bstate[brick_lin] = touched ? 2 : 0;
}
