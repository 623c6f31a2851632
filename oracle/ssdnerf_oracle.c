/*
 * ssdnerf_oracle.c -- CPU restatement of the SSDNeRF ray-march hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in ssdnerf_b200/ may link, import or call
 * this file; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference leg use it, and only as the checker / the timed CPU baseline.
 *
 * PARITY UNPINNED BY REFERENCE TESTS: the reference (Lakonik/SSDNeRF @ b9d195d)
 * ships no tests, golden vectors or CPU path for these kernels (SURVEY.md F2/F3).
 * This restatement follows the arithmetic of the reference CUDA sources line by
 * line (citations below, file = lib/ops/raymarching/src/raymarching.cu unless
 * noted).  The GPU kernels the tests hold to it are in turn compared with the
 * outputs of the reference's own kernels (compiled into oracle/_ref/ by
 * oracle/build_ref.sh), stored in tests/golden/reference_kernels_v1.npz
 * (tests/test_ref_gpu.py).
 *
 * Arithmetic notes (SURVEY.md Appendix A):
 *  - nvcc contracts `o + t*d` into one FFMA; we use fmaf() at exactly those sites.
 *  - the voxel index is computed as (int)clamp(0.5 * (x*rb + 1) * H, 0, H-1) with a
 *    DOUBLE literal 0.5: float -> double, two double multiplies, double -> float.
 *  - 1/d is an IEEE-correct float divide (no fast-math in the reference build).
 *  - __expf() in the compositors is MUFU.EX2 based; expf() here differs by ~2 ulp,
 *    which is why composited floats are compared with a tolerance, not bit-exact.
 */
#include <math.h>
#include <float.h>
#include <stdint.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

static inline float orc_clampf(float x, float lo, float hi) { /* :34-36 */
    return fminf(hi, fmaxf(lo, x));
}
static inline float orc_signf(float x) { return copysignf(1.0f, x); } /* :30-32 */

static inline uint32_t orc_expand_bits(uint32_t v) { /* :56-63 */
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
static inline uint32_t orc_morton(uint32_t x, uint32_t y, uint32_t z) { /* :65-71 */
    return orc_expand_bits(x) | (orc_expand_bits(y) << 1) | (orc_expand_bits(z) << 2);
}
static inline uint32_t orc_morton_inv(uint32_t x) { /* :73-81 */
    x &= 0x49249249u;
    x = (x | (x >> 2)) & 0xc30c30c3u;
    x = (x | (x >> 4)) & 0x0f00f00fu;
    x = (x | (x >> 8)) & 0xff0000ffu;
    x = (x | (x >> 16)) & 0x0000ffffu;
    return x;
}

/* mip_from_pos / mip_from_dt, :40-53 (always 0 when C == 1, kept for completeness) */
static inline int orc_mip_from_pos(float x, float y, float z, float max_cascade) {
    const float mx = fmaxf(fabsf(x), fmaxf(fabsf(y), fabsf(z)));
    int e; frexpf(mx, &e);
    return (int)fminf(max_cascade - 1, fmaxf(0, (float)e));
}
static inline int orc_mip_from_dt(float dt, float H, float max_cascade) {
    const float mx = (float)((double)(dt * H) * 0.5);
    int e; frexpf(mx, &e);
    return (int)fminf(max_cascade - 1, fmaxf(0, (float)e));
}

/* K1  kernel_near_far_from_aabb :92-145 */
ORC_API void orc_near_far_from_aabb(const float* rays_o, const float* rays_d, const float* aabb,
                                    uint32_t N, float min_near, float* nears, float* fars) {
    for (uint32_t n = 0; n < N; ++n) {
        const float ox = rays_o[3*n], oy = rays_o[3*n+1], oz = rays_o[3*n+2];
        const float dx = rays_d[3*n], dy = rays_d[3*n+1], dz = rays_d[3*n+2];
        const float rdx = 1.0f / dx, rdy = 1.0f / dy, rdz = 1.0f / dz;
        float near = (aabb[0] - ox) * rdx, far = (aabb[3] - ox) * rdx, tmp;
        if (near > far) { tmp = near; near = far; far = tmp; }
        float near_y = (aabb[1] - oy) * rdy, far_y = (aabb[4] - oy) * rdy;
        if (near_y > far_y) { tmp = near_y; near_y = far_y; far_y = tmp; }
        if (near > far_y || near_y > far) { nears[n] = fars[n] = FLT_MAX; continue; }
        if (near_y > near) near = near_y;
        if (far_y < far) far = far_y;
        float near_z = (aabb[2] - oz) * rdz, far_z = (aabb[5] - oz) * rdz;
        if (near_z > far_z) { tmp = near_z; near_z = far_z; far_z = tmp; }
        if (near > far_z || near_z > far) { nears[n] = fars[n] = FLT_MAX; continue; }
        if (near_z > near) near = near_z;
        if (far_z < far) far = far_z;
        if (near < min_near) near = min_near;
        nears[n] = near; fars[n] = far;
    }
}

/* K3 / K4  :214-254 */
ORC_API void orc_morton3D(const int32_t* coords, uint32_t N, int32_t* indices) {
    for (uint32_t n = 0; n < N; ++n)
        indices[n] = (int32_t)orc_morton((uint32_t)coords[3*n], (uint32_t)coords[3*n+1], (uint32_t)coords[3*n+2]);
}
ORC_API void orc_morton3D_invert(const int32_t* indices, uint32_t N, int32_t* coords) {
    for (uint32_t n = 0; n < N; ++n) {
        const int32_t ind = indices[n];
        coords[3*n]   = (int32_t)orc_morton_inv((uint32_t)(ind >> 0));
        coords[3*n+1] = (int32_t)orc_morton_inv((uint32_t)(ind >> 1));
        coords[3*n+2] = (int32_t)orc_morton_inv((uint32_t)(ind >> 2));
    }
}

/* K5  kernel_packbits :268-289 ; N = number of output bytes */
ORC_API void orc_packbits(const float* grid, uint32_t N, float thresh, uint8_t* bitfield) {
    for (uint32_t n = 0; n < N; ++n) {
        uint8_t bits = 0;
        for (int i = 0; i < 8; ++i) bits |= (grid[8*(size_t)n + i] > thresh) ? (uint8_t)(1u << i) : 0;
        bitfield[n] = bits;
    }
}

/* One occupancy probe + step, shared by K6 and K9 (:757-810 == :360-398 == :422-480). */
typedef struct { float ox, oy, oz, dx, dy, dz, rdx, rdy, rdz; } orc_ray;

typedef struct {
    float bound, dt_gamma, dt_min, dt_max, rH, H3f, Hf, Cf;
    uint32_t H;
    const uint8_t* grid;
} orc_march_cfg;

static inline void orc_cfg_init(orc_march_cfg* c, float bound, float dt_gamma, uint32_t max_steps,
                                uint32_t C, uint32_t H, const uint8_t* grid) {
    c->bound = bound; c->dt_gamma = dt_gamma; c->H = H; c->grid = grid;
    c->Hf = (float)H; c->Cf = (float)C;
    c->rH = 1.0f / (float)H;
    c->H3f = (float)(H * H * H);                                 /* :739 float H3 */
    c->dt_min = 2.0f * 1.7320508075688772f / (float)max_steps;    /* :744 */
    c->dt_max = 2.0f * 1.7320508075688772f * (float)(1u << (C - 1)) / (float)H; /* :745 */
}

/* returns 1 if the probe at t is occupied (then *px..*pdt hold the sample, t is NOT advanced),
 * 0 if empty (then *t has been advanced past the voxel). */
static inline int orc_probe(const orc_march_cfg* c, const orc_ray* r, float* t,
                            float* px, float* py, float* pz, float* pdt, uint32_t* pindex) {
    const float tt0 = *t;
    const float x = orc_clampf(fmaf(tt0, r->dx, r->ox), -c->bound, c->bound);
    const float y = orc_clampf(fmaf(tt0, r->dy, r->oy), -c->bound, c->bound);
    const float z = orc_clampf(fmaf(tt0, r->dz, r->oz), -c->bound, c->bound);
    const float dt = orc_clampf(tt0 * c->dt_gamma, c->dt_min, c->dt_max);
    int l1 = orc_mip_from_pos(x, y, z, c->Cf), l2 = orc_mip_from_dt(dt, c->Hf, c->Cf);
    const int level = l1 > l2 ? l1 : l2;
    const float mip_bound = fminf(scalbnf(1.0f, level), c->bound);
    const float mip_rbound = 1.0f / mip_bound;
    /* double literal 0.5: (float)(x*rb+1) -> double * 0.5 * (double)H -> float -> clamp -> trunc */
    const int nx = (int)orc_clampf((float)(0.5 * (double)fmaf(x, mip_rbound, 1.0f) * (double)c->Hf), 0.0f, (float)(c->H - 1));
    const int ny = (int)orc_clampf((float)(0.5 * (double)fmaf(y, mip_rbound, 1.0f) * (double)c->Hf), 0.0f, (float)(c->H - 1));
    const int nz = (int)orc_clampf((float)(0.5 * (double)fmaf(z, mip_rbound, 1.0f) * (double)c->Hf), 0.0f, (float)(c->H - 1));
    const uint32_t index = (uint32_t)((float)level * c->H3f) + orc_morton((uint32_t)nx, (uint32_t)ny, (uint32_t)nz);
    const int occ = c->grid[index / 8] & (1 << (index % 8));
    if (occ) { *px = x; *py = y; *pz = z; *pdt = dt; *pindex = index; return 1; }
    /* empty: distance to the next voxel boundary (:800-810) */
    const float tx = (fmaf(((float)nx + 0.5f + 0.5f * orc_signf(r->dx)) * c->rH * 2.0f - 1.0f, mip_bound, -x)) * r->rdx;
    const float ty = (fmaf(((float)ny + 0.5f + 0.5f * orc_signf(r->dy)) * c->rH * 2.0f - 1.0f, mip_bound, -y)) * r->rdy;
    const float tz = (fmaf(((float)nz + 0.5f + 0.5f * orc_signf(r->dz)) * c->rH * 2.0f - 1.0f, mip_bound, -z)) * r->rdz;
    const float tt = tt0 + fmaxf(0.0f, fminf(tx, fminf(ty, tz)));
    float tcur = tt0;
    do { tcur += orc_clampf(tcur * c->dt_gamma, c->dt_min, c->dt_max); } while (tcur < tt);
    *t = tcur;
    return 0;
}

static inline void orc_ray_load(orc_ray* r, const float* o, const float* d) {
    r->ox = o[0]; r->oy = o[1]; r->oz = o[2];
    r->dx = d[0]; r->dy = d[1]; r->dz = d[2];
    r->rdx = 1.0f / r->dx; r->rdy = 1.0f / r->dy; r->rdz = 1.0f / r->dz;
}

/* K9  kernel_march_rays :706-812.  Output buffers must be zero-filled by the caller
 * (raymarching.py:440-442).  `voxels` (optional, int32 [n_alive*n_step]) receives the
 * occupancy-grid bit index of every sample (-1 for unused slots): the integer trace used
 * for bit-exact parity. */
ORC_API void orc_march_rays(uint32_t n_alive, uint32_t n_step, const int32_t* rays_alive, const float* rays_t,
                            const float* rays_o, const float* rays_d, float bound, float dt_gamma,
                            uint32_t max_steps, uint32_t C, uint32_t H, const uint8_t* grid,
                            const float* nears, const float* fars,
                            float* xyzs, float* dirs, float* deltas, const float* noises, int32_t* voxels) {
    orc_march_cfg c; orc_cfg_init(&c, bound, dt_gamma, max_steps, C, H, grid);
    for (uint32_t n = 0; n < n_alive; ++n) {
        const int32_t index = rays_alive[n];
        const float noise = noises ? noises[n] : 0.0f;
        orc_ray r; orc_ray_load(&r, rays_o + 3 * (size_t)index, rays_d + 3 * (size_t)index);
        float t = rays_t[index];
        const float far = fars[index];
        (void)nears;
        float* xo = xyzs + (size_t)n * n_step * 3;
        float* dO = dirs + (size_t)n * n_step * 3;
        float* de = deltas + (size_t)n * n_step * 2;
        int32_t* vo = voxels ? voxels + (size_t)n * n_step : 0;
        if (vo) for (uint32_t s = 0; s < n_step; ++s) vo[s] = -1;
        uint32_t step = 0;
        t = fmaf(orc_clampf(t * dt_gamma, c.dt_min, c.dt_max), noise, t);   /* :751 */
        while (t < far && step < n_step) {
            float x, y, z, dt; uint32_t vi;
            if (orc_probe(&c, &r, &t, &x, &y, &z, &dt, &vi)) {
                xo[0] = x; xo[1] = y; xo[2] = z;
                dO[0] = r.dx; dO[1] = r.dy; dO[2] = r.dz;
                de[0] = dt; de[1] = t;
                if (vo) vo[step] = (int32_t)vi;
                t += dt;
                xo += 3; dO += 3; de += 2; ++step;
            }
        }
    }
}

/* K10  kernel_composite_rays :826-913 */
ORC_API void orc_composite_rays(uint32_t n_alive, uint32_t n_step, float T_thresh, int32_t* rays_alive, float* rays_t,
                                const float* sigmas, const float* rgbs, const float* deltas,
                                float* weights_sum, float* depth, float* image) {
    for (uint32_t n = 0; n < n_alive; ++n) {
        const int32_t index = rays_alive[n];
        const float* sg = sigmas + (size_t)n * n_step;
        const float* cl = rgbs + (size_t)n * n_step * 3;
        const float* de = deltas + (size_t)n * n_step * 2;
        float ws = weights_sum[index], d = depth[index];
        float r = image[3*(size_t)index], g = image[3*(size_t)index+1], b = image[3*(size_t)index+2];
        uint32_t step = 0;
        while (step < n_step) {
            if (de[0] == 0) break;
            const float alpha = 1.0f - expf(-sg[0] * de[0]);
            const float T = 1 - ws;
            const float w = alpha * T;
            ws += w;
            d = fmaf(w, de[1], d);
            r = fmaf(w, cl[0], r); g = fmaf(w, cl[1], g); b = fmaf(w, cl[2], b);
            if (T < T_thresh) break;
            sg++; cl += 3; de += 2; step++;
        }
        if (step < n_step) rays_alive[n] = -1;
        else rays_t[index] = de[-1] + de[-2];
        weights_sum[index] = ws; depth[index] = d;
        image[3*(size_t)index] = r; image[3*(size_t)index+1] = g; image[3*(size_t)index+2] = b;
    }
}

/* K6  kernel_march_rays_train :312-482, made deterministic: rays are processed in index
 * order so point offsets are the exclusive prefix sum of the per-ray counts (the reference
 * orders them by atomicAdd arrival; parity is per ray, SURVEY.md Appendix C).
 * Pass xyzs == NULL to only count (rays[] and counter[] are still written). */
ORC_API void orc_march_rays_train(const float* rays_o, const float* rays_d, const uint8_t* grid, float bound, float dt_gamma,
                                  uint32_t max_steps, uint32_t N, uint32_t C, uint32_t H, uint32_t M,
                                  const float* nears, const float* fars,
                                  float* xyzs, float* dirs, float* deltas, int32_t* rays, int32_t* counter,
                                  const float* noises, int32_t* voxels) {
    orc_march_cfg c; orc_cfg_init(&c, bound, dt_gamma, max_steps, C, H, grid);
    for (uint32_t n = 0; n < N; ++n) {
        orc_ray r; orc_ray_load(&r, rays_o + 3 * (size_t)n, rays_d + 3 * (size_t)n);
        const float near = nears[n], far = fars[n], noise = noises ? noises[n] : 0.0f;
        const float t0 = fmaf(orc_clampf(near * dt_gamma, c.dt_min, c.dt_max), noise, near);
        float t = t0; uint32_t num_steps = 0;
        while (t < far && num_steps < max_steps) {
            float x, y, z, dt; uint32_t vi;
            if (orc_probe(&c, &r, &t, &x, &y, &z, &dt, &vi)) { num_steps++; t += dt; }
        }
        const uint32_t point_index = (uint32_t)counter[0]; counter[0] += (int32_t)num_steps;
        const uint32_t ray_index = (uint32_t)counter[1]; counter[1] += 1;
        rays[3*ray_index] = (int32_t)n; rays[3*ray_index+1] = (int32_t)point_index; rays[3*ray_index+2] = (int32_t)num_steps;
        if (!xyzs || num_steps == 0 || point_index + num_steps > M) continue;
        float* xo = xyzs + (size_t)point_index * 3;
        float* dO = dirs + (size_t)point_index * 3;
        float* de = deltas + (size_t)point_index * 2;
        int32_t* vo = voxels ? voxels + point_index : 0;
        t = t0; uint32_t step = 0;
        while (t < far && step < num_steps) {
            float x, y, z, dt; uint32_t vi;
            if (orc_probe(&c, &r, &t, &x, &y, &z, &dt, &vi)) {
                xo[0] = x; xo[1] = y; xo[2] = z;
                dO[0] = r.dx; dO[1] = r.dy; dO[2] = r.dz;
                de[0] = dt; de[1] = t;
                if (vo) vo[step] = (int32_t)vi;
                t += dt; xo += 3; dO += 3; de += 2; ++step;
            }
        }
    }
}

/* K7  kernel_composite_rays_train_forward :503-581 */
ORC_API void orc_composite_rays_train_forward(const float* sigmas, const float* rgbs, const float* deltas, const int32_t* rays,
                                              uint32_t M, uint32_t N, float T_thresh,
                                              float* weights_sum, float* depth, float* image) {
    for (uint32_t n = 0; n < N; ++n) {
        const uint32_t index = (uint32_t)rays[3*n], offset = (uint32_t)rays[3*n+1], num_steps = (uint32_t)rays[3*n+2];
        if (num_steps == 0 || offset + num_steps > M) {
            weights_sum[index] = 0; depth[index] = 0;
            image[3*(size_t)index] = image[3*(size_t)index+1] = image[3*(size_t)index+2] = 0;
            continue;
        }
        const float* sg = sigmas + offset; const float* cl = rgbs + 3*(size_t)offset; const float* de = deltas + 2*(size_t)offset;
        float T = 1.0f, r = 0, g = 0, b = 0, ws = 0, d = 0;
        for (uint32_t step = 0; step < num_steps; ++step) {
            const float alpha = 1.0f - expf(-sg[0] * de[0]);
            const float w = alpha * T;
            r = fmaf(w, cl[0], r); g = fmaf(w, cl[1], g); b = fmaf(w, cl[2], b);
            d = fmaf(w, de[1], d);
            ws += w;
            T *= 1.0f - alpha;
            if (T < T_thresh) break;
            sg++; cl += 3; de += 2;
        }
        weights_sum[index] = ws; depth[index] = d;
        image[3*(size_t)index] = r; image[3*(size_t)index+1] = g; image[3*(size_t)index+2] = b;
    }
}

/* K8  kernel_composite_rays_train_backward :606-687 (grad buffers zero-filled by caller) */
ORC_API void orc_composite_rays_train_backward(const float* grad_ws, const float* grad_image, const float* sigmas, const float* rgbs,
                                               const float* deltas, const int32_t* rays, const float* weights_sum, const float* image,
                                               uint32_t M, uint32_t N, float T_thresh, float* grad_sigmas, float* grad_rgbs) {
    for (uint32_t n = 0; n < N; ++n) {
        const uint32_t index = (uint32_t)rays[3*n], offset = (uint32_t)rays[3*n+1], num_steps = (uint32_t)rays[3*n+2];
        if (num_steps == 0 || offset + num_steps > M) continue;
        const float gws = grad_ws[index];
        const float* gi = grad_image + 3*(size_t)index;
        const float r_final = image[3*(size_t)index], g_final = image[3*(size_t)index+1], b_final = image[3*(size_t)index+2];
        const float ws_final = weights_sum[index];
        const float* sg = sigmas + offset; const float* cl = rgbs + 3*(size_t)offset; const float* de = deltas + 2*(size_t)offset;
        float* gs = grad_sigmas + offset; float* gc = grad_rgbs + 3*(size_t)offset;
        float T = 1.0f, r = 0, g = 0, b = 0, ws = 0;
        for (uint32_t step = 0; step < num_steps; ++step) {
            const float alpha = 1.0f - expf(-sg[0] * de[0]);
            const float w = alpha * T;
            r = fmaf(w, cl[0], r); g = fmaf(w, cl[1], g); b = fmaf(w, cl[2], b);
            ws += w;
            T *= 1.0f - alpha;
            if (T < T_thresh) break;
            gc[0] = gi[0] * w; gc[1] = gi[1] * w; gc[2] = gi[2] * w;
            gs[0] = de[0] * (gi[0] * (T * cl[0] - (r_final - r)) +
                             gi[1] * (T * cl[1] - (g_final - g)) +
                             gi[2] * (T * cl[2] - (b_final - b)) +
                             gws * (1 - ws_final));
            sg++; cl += 3; de += 2; gs++; gc += 3;
        }
    }
}

/* K11  kernel_sh, degree <= 4  (lib/ops/shencoder/src/shencoder.cu:44-69) */
ORC_API void orc_sh_encode(const float* inputs, uint32_t B, uint32_t degree, float* outputs) {
    const uint32_t C2 = degree * degree;
    for (uint32_t bidx = 0; bidx < B; ++bidx) {
        const float x = inputs[3*bidx], y = inputs[3*bidx+1], z = inputs[3*bidx+2];
        const float xy = x*y, xz = x*z, yz = y*z, x2 = x*x, y2 = y*y, z2 = z*z;
        float* o = outputs + (size_t)bidx * C2;
        o[0] = 0.28209479177387814f;
        if (degree <= 1) continue;
        o[1] = -0.48860251190291987f * y;
        o[2] = 0.48860251190291987f * z;
        o[3] = -0.48860251190291987f * x;
        if (degree <= 2) continue;
        o[4] = 1.0925484305920792f * xy;
        o[5] = -1.0925484305920792f * yz;
        o[6] = 0.94617469575755997f * z2 - 0.31539156525251999f;
        o[7] = -1.0925484305920792f * xz;
        o[8] = 0.54627421529603959f * x2 - 0.54627421529603959f * y2;
        if (degree <= 3) continue;
        o[9]  = 0.59004358992664352f * y * (-3.0f * x2 + y2);
        o[10] = 2.8906114426405538f * xy * z;
        o[11] = 0.45704579946446572f * y * (1.0f - 5.0f * z2);
        o[12] = 0.3731763325901154f * z * (5.0f * z2 - 3.0f);
        o[13] = 0.45704579946446572f * x * (1.0f - 5.0f * z2);
        o[14] = 1.4453057213202769f * z * (x2 - y2);
        o[15] = 0.59004358992664352f * x * (-x2 + 3.0f * y2);
    }
}

/* ---------------------------------------------------------------------------------
 * Whole-ray reference of the eval host loop (lib/models/decoders/base_volume_renderer.py:79-123)
 * for the INTEGER part only: given a per-quantum schedule it returns, for every ray, the voxel
 * (bitfield bit index) sequence it would sample if never terminated by transmittance.
 * Used by tests for the bit-exact ray-index / occupancy-hit check at sizes where the Python
 * loop would be slow.  trace: int32 [N, cap] (-1 padded), counts: int32 [N].
 * --------------------------------------------------------------------------------- */
ORC_API void orc_trace_rays(const float* rays_o, const float* rays_d, const float* nears, const float* fars, uint32_t N,
                            float bound, float dt_gamma, uint32_t max_steps, uint32_t C, uint32_t H, const uint8_t* grid,
                            uint32_t cap, int32_t* trace, float* ts, int32_t* counts) {
    orc_march_cfg c; orc_cfg_init(&c, bound, dt_gamma, max_steps, C, H, grid);
    for (uint32_t n = 0; n < N; ++n) {
        orc_ray r; orc_ray_load(&r, rays_o + 3*(size_t)n, rays_d + 3*(size_t)n);
        float t = nears[n]; const float far = fars[n];
        uint32_t step = 0;
        for (uint32_t s = 0; s < cap; ++s) { trace[(size_t)n*cap + s] = -1; if (ts) ts[(size_t)n*cap + s] = 0; }
        while (t < far && step < cap) {
            float x, y, z, dt; uint32_t vi;
            if (orc_probe(&c, &r, &t, &x, &y, &z, &dt, &vi)) {
                trace[(size_t)n*cap + step] = (int32_t)vi;
                if (ts) ts[(size_t)n*cap + step] = t;
                t += dt; ++step;
            }
        }
        counts[n] = (int32_t)step;
    }
}
