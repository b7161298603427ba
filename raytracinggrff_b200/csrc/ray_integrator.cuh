// Ray integrator for sm_100a: the whole n_steps RK4 loop of one ray inside one thread.
//
// Replaces raytracingGRFF/build_rays.py:128-248 (ray_trace: rhs :158-175, rk4_step :177-182,
// pencil basis :188-201, cross-section ratio :209-239, recording :241-244) and the
// one-launch-per-step CUDA path raytracingGRFF/gpu_raytrace.py:236-315, :383-408.
//
// Design (see DESIGN.md): one thread per ray, a warp = 32 neighbouring rays so that the 8-corner
// gathers of a warp fall into a handful of 128-B lines; state and RK4 accumulation in FP64
// (1e-5 R_sun after thousands of chained steps needs it, BASELINE.md §2); the cube is ONE
// interleaved float4 {omega_pe, d/dx, d/dy, d/dz} array so a corner is one 16-B load instead of
// four 4-B loads from four cubes; records go out as SoA [rec][component][ray] (coalesced);
// a ray that stopped moving is frozen exactly as in the reference, so its remaining steps are
// skipped and its remaining records filled.
#pragma once

#include "common.cuh"

namespace rtgrff {

struct RayCube {
    const float4 *__restrict__ c;
    const float4 *__restrict__ pc;   // cell-major polynomial cube (ray_core32.cuh), 8 float4 per cell, or nullptr
    int nx, ny, nz;
    int sy, sx;  // element strides of y and x (z is contiguous)
    double x0, y0, z0, xl, yl, zl, idx, idy, idz;
};

struct State {
    double rx, ry, rz, kx, ky, kz;
};

__device__ __forceinline__ bool in_cube(const RayCube &C, double x, double y, double z)
{
    // scipy: out of bounds iff x < g[0] or x > g[-1]; NaN compares false -> outside here,
    // and f(NaN) = NaN there: both end as "invalid stage".
    return (x >= C.x0) && (x <= C.xl) && (y >= C.y0) && (y <= C.yl) && (z >= C.z0) && (z <= C.zl);
}

__device__ __forceinline__ float lerpf(float a, float b, float t) { return fmaf(t, b - a, a); }
__device__ __forceinline__ double lerpd(double a, double b, double t) { return fma(t, b - a, a); }

// One RHS evaluation (build_rays.py:158-175): trilinear arithmetic in FP32 on the FP32-stored corners;
// position, cell fraction, omega and the derivative stay FP64.
__device__ __forceinline__ void rhs_eval(const RayCube &C, const State &s, State &d)
{
    d.rx = d.ry = d.rz = d.kx = d.ky = d.kz = 0.0;
    if (!in_cube(C, s.rx, s.ry, s.rz)) return;
    const double fx = (s.rx - C.x0) * C.idx, fy = (s.ry - C.y0) * C.idy, fz = (s.rz - C.z0) * C.idz;
    const int i = min((int)fx, C.nx - 2), j = min((int)fy, C.ny - 2), k = min((int)fz, C.nz - 2);
    const double tx = fx - (double)i, ty = fy - (double)j, tz = fz - (double)k;
    const float4 *p = C.c + ((size_t)i * C.sx + (size_t)j * C.sy + (size_t)k);
    const float4 c000 = __ldg(p), c001 = __ldg(p + 1);
    const float4 c010 = __ldg(p + C.sy), c011 = __ldg(p + C.sy + 1);
    const float4 c100 = __ldg(p + C.sx), c101 = __ldg(p + C.sx + 1);
    const float4 c110 = __ldg(p + C.sx + C.sy), c111 = __ldg(p + C.sx + C.sy + 1);
    const float ftx = (float)tx, fty = (float)ty, ftz = (float)tz;
#define RT_TRI32(m)                                                                               \
    lerpf(lerpf(lerpf(c000.m, c001.m, ftz), lerpf(c010.m, c011.m, ftz), fty),                     \
          lerpf(lerpf(c100.m, c101.m, ftz), lerpf(c110.m, c111.m, ftz), fty), ftx)
    const double w = (double)RT_TRI32(x), gx = (double)RT_TRI32(y), gy = (double)RT_TRI32(z), gz = (double)RT_TRI32(w);
#undef RT_TRI32
    const double om = sqrt(w * w + ((s.kx * s.kx + s.ky * s.ky) + s.kz * s.kz));
    // valid = isfinite(omega_pe) & isfinite(omega) & (omega > 0); gradients are NOT tested (build_rays.py:169)
    if (!(isfinite(w) && isfinite(om) && om > 0.0)) return;
    const double cr_om = kC_R / om;
    const double a = -w * cr_om;
    d.rx = cr_om * s.kx; d.ry = cr_om * s.ky; d.rz = cr_om * s.kz;
    d.kx = a * gx; d.ky = a * gy; d.kz = a * gz;
}

__device__ __forceinline__ State axpy(const State &s, double h, const State &d)
{
    State o;
    o.rx = fma(h, d.rx, s.rx); o.ry = fma(h, d.ry, s.ry); o.rz = fma(h, d.rz, s.rz);
    o.kx = fma(h, d.kx, s.kx); o.ky = fma(h, d.ky, s.ky); o.kz = fma(h, d.kz, s.kz);
    return o;
}

// Classic RK4 (build_rays.py:177-182).
__device__ __forceinline__ State rk4_step(const RayCube &C, const State &s, double dt)
{
    State k1, k2, k3, k4;
    rhs_eval(C, s, k1);
    rhs_eval(C, axpy(s, 0.5 * dt, k1), k2);
    rhs_eval(C, axpy(s, 0.5 * dt, k2), k3);
    rhs_eval(C, axpy(s, dt, k3), k4);
    const double c6 = dt / 6.0;
    State o;
    o.rx = fma(c6, (k1.rx + 2.0 * k2.rx) + 2.0 * k3.rx + k4.rx, s.rx);
    o.ry = fma(c6, (k1.ry + 2.0 * k2.ry) + 2.0 * k3.ry + k4.ry, s.ry);
    o.rz = fma(c6, (k1.rz + 2.0 * k2.rz) + 2.0 * k3.rz + k4.rz, s.rz);
    o.kx = fma(c6, (k1.kx + 2.0 * k2.kx) + 2.0 * k3.kx + k4.kx, s.kx);
    o.ky = fma(c6, (k1.ky + 2.0 * k2.ky) + 2.0 * k3.ky + k4.ky, s.ky);
    o.kz = fma(c6, (k1.kz + 2.0 * k2.kz) + 2.0 * k3.kz + k4.kz, s.kz);
    return o;
}

// Cross-section ratio of one step (build_rays.py:209-239): two rays displaced by eps along the
// pencil basis (e1,e2) _|_ t_hat, same k0, one RK4 step each; S = |(d1 x d2).t_hat| / eps^2.
__device__ __forceinline__ double cross_section_ratio(const RayCube &C, const State &s0, const State &s1,
                                                      double dt, double perturb_ratio)
{
    const double dx = s1.rx - s0.rx, dy = s1.ry - s0.ry, dz = s1.rz - s0.rz;
    const double nrd = sqrt((dx * dx + dy * dy) + dz * dz);
    const double inv = 1.0 / (nrd + 1e-32);
    const double tx = dx * inv, ty = dy * inv, tz = dz * inv;
    // reference axis: z if |t_z| < 0.9 else y (build_rays.py:188-194); e1 = a x t, e2 = t x e1
    const bool use_z = fabs(tz) < 0.9;
    double e1x = use_z ? -ty : tz, e1y = use_z ? tx : 0.0, e1z = use_z ? 0.0 : -tx;
    const double n1 = 1.0 / (sqrt((e1x * e1x + e1y * e1y) + e1z * e1z) + 1e-30);
    e1x *= n1; e1y *= n1; e1z *= n1;
    double e2x = ty * e1z - tz * e1y, e2y = tz * e1x - tx * e1z, e2z = tx * e1y - ty * e1x;
    const double n2 = 1.0 / (sqrt((e2x * e2x + e2y * e2y) + e2z * e2z) + 1e-30);
    e2x *= n2; e2y *= n2; e2z *= n2;
    const double eps = perturb_ratio * nrd;
    State p1 = s0, p2 = s0;
    p1.rx = fma(eps, e1x, s0.rx); p1.ry = fma(eps, e1y, s0.ry); p1.rz = fma(eps, e1z, s0.rz);
    p2.rx = fma(eps, e2x, s0.rx); p2.ry = fma(eps, e2y, s0.ry); p2.rz = fma(eps, e2z, s0.rz);
    const State q1 = rk4_step(C, p1, dt);
    const State q2 = rk4_step(C, p2, dt);
    const double d1x = q1.rx - s1.rx, d1y = q1.ry - s1.ry, d1z = q1.rz - s1.rz;
    const double d2x = q2.rx - s1.rx, d2y = q2.ry - s1.ry, d2z = q2.rz - s1.rz;
    const double cx = d1y * d2z - d1z * d2y, cy = d1z * d2x - d1x * d2z, cz = d1x * d2y - d1y * d2x;
    return fabs((cx * tx + cy * ty) + cz * tz) / (eps * eps);
}

// kc0 = sqrt(max(omega0^2 - omega_pe(start)^2, 0)), NaN-propagating (build_rays.py:147-151).
__device__ __forceinline__ double start_kc(const RayCube &C, double x, double y, double z, double omega0)
{
    if (!in_cube(C, x, y, z)) return nan("");
    const double fx = (x - C.x0) * C.idx, fy = (y - C.y0) * C.idy, fz = (z - C.z0) * C.idz;
    const int i = min((int)fx, C.nx - 2), j = min((int)fy, C.ny - 2), k = min((int)fz, C.nz - 2);
    const double tx = fx - (double)i, ty = fy - (double)j, tz = fz - (double)k;
    const float4 *p = C.c + ((size_t)i * C.sx + (size_t)j * C.sy + (size_t)k);
    const double w = lerpd(
        lerpd(lerpd((double)p[0].x, (double)p[1].x, tz), lerpd((double)p[C.sy].x, (double)p[C.sy + 1].x, tz), ty),
        lerpd(lerpd((double)p[C.sx].x, (double)p[C.sx + 1].x, tz),
              lerpd((double)p[C.sx + C.sy].x, (double)p[C.sx + C.sy + 1].x, tz), ty), tx);
    const double arg = omega0 * omega0 - w * w;
    return (arg != arg) ? arg : sqrt(fmax(arg, 0.0));
}

__device__ __forceinline__ bool state_differs(const State &a, const State &b)
{
    return (a.rx != b.rx) | (a.ry != b.ry) | (a.rz != b.rz) | (a.kx != b.kx) | (a.ky != b.ky) | (a.kz != b.kz);
}

// SoA [rec][3][ray] -> AoS (rec, ray, 3), the reference's r_record layout (build_rays.py:248).
__global__ void records_to_aos_kernel(const double *__restrict__ soa, double *__restrict__ aos,
                                      int64_t n_rec, int64_t n_rays)
{
    const int64_t total = n_rec * n_rays * 3;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = q % 3, rr = q / 3;
        const int64_t ray = rr % n_rays, rec = rr / n_rays;
        aos[q] = soa[(rec * 3 + c) * n_rays + ray];
    }
}

// {omega_pe (f64)} -> float4 {omega_pe, d/dx, d/dy, d/dz} with numpy.gradient semantics
// (build_rays.py:136-138): central differences inside, first-order one-sided on the faces;
// differences taken in FP64, stored as FP32.
__global__ void build_ray_cube_kernel(const double *__restrict__ w, float4 *__restrict__ out,
                                      int nx, int ny, int nz, double hx, double hy, double hz)
{
    const int64_t nvox = (int64_t)nx * ny * nz;
    const int64_t sx = (int64_t)ny * nz, sy = nz;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nvox;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(q % nz), j = (int)((q / nz) % ny), i = (int)(q / sx);
        const double c = w[q];
        double gx, gy, gz;
        if (nx < 2) gx = 0.0;
        else if (i == 0) gx = (w[q + sx] - c) / hx;
        else if (i == nx - 1) gx = (c - w[q - sx]) / hx;
        else gx = (w[q + sx] - w[q - sx]) / (2.0 * hx);
        if (ny < 2) gy = 0.0;
        else if (j == 0) gy = (w[q + sy] - c) / hy;
        else if (j == ny - 1) gy = (c - w[q - sy]) / hy;
        else gy = (w[q + sy] - w[q - sy]) / (2.0 * hy);
        if (nz < 2) gz = 0.0;
        else if (k == 0) gz = (w[q + 1] - c) / hz;
        else if (k == nz - 1) gz = (c - w[q - 1]) / hz;
        else gz = (w[q + 1] - w[q - 1]) / (2.0 * hz);
        out[q] = make_float4((float)c, (float)gx, (float)gy, (float)gz);
    }
}

}  // namespace rtgrff
