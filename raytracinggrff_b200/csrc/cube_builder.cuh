// Cube builder for sm_100a: resample a variable given on a spherical (phi, theta, r) mesh onto the
// regular xyz cube the ray path consumes, then compose the device cubes — the step right before the
// hot path (SURVEY.md §8f rank 1).
//
// Replaces raytracingGRFF/build_rays.py:35-45 (cart_to_sph), :69-125 (resample_to_xyz_cube: a Python
// loop over x-slices calling psipy's Variable.sample_at_coords) and
// script/resample_with_ray_tracing.py:110-151, :263-293 (resample_var_to_cube + the unit/NaN rules
// that turn rho, te, br, bt, bp into omega_pe, n_e, T, |B|).  psipy itself is not in the reference
// tree; its sampler is restated from its published behaviour: linear interpolation on the
// (phi, latitude, r) mesh with the phi axis padded by one node on each side to wrap around.
// Semantics here (oracle: oracle/oracle_cubes.py): a point outside the latitude or radius range of
// the mesh, or below r_min, is NaN and takes the fill value — per point, where the reference loses
// the whole x-slice to psipy's bounds exception (build_rays.py:109-117).
#pragma once

#include "common.cuh"

namespace rtgrff {

struct SphMesh {
    const float *data;      // [np][nt][nr], r fastest (psipy's (phi, theta, r) order)
    const double *phi;      // [np]  longitude nodes, rad, ascending, within one turn
    const double *lat;      // [nt]  latitude nodes, rad, ascending
    const double *r;        // [nr]  radius nodes, R_sun, ascending
    int np, nt, nr;
};

// i with g[i] <= x < g[i+1], clipped to [0, n-2]; the last interval is closed on the right
// (scipy find_interval_ascending).
__device__ __forceinline__ int find_interval(const double *__restrict__ g, int n, double x)
{
    int lo = 0, hi = n - 1;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (x >= g[mid]) lo = mid; else hi = mid;
    }
    return lo;
}

// psipy-style sample: linear in (phi, lat, r), phi periodic.  NaN outside the lat / r range.
__device__ __forceinline__ double sample_spherical(const SphMesh &m, double lon, double lat, double r)
{
    if (!(lat >= m.lat[0] && lat <= m.lat[m.nt - 1] && r >= m.r[0] && r <= m.r[m.nr - 1]) || !isfinite(lon))
        return nan("");
    const double two_pi = 6.283185307179586476925286766559;
    // padded phi axis: node -1 = phi[np-1] - 2 pi, node np = phi[0] + 2 pi
    int ip0, ip1;
    double p0, p1;
    // outside the padded axis psipy's interpolator raises and the reference turns the point into NaN
    // (build_rays.py:109-117): reachable with a phi0 offset beyond about +180 deg, since cart_to_sph
    // only wraps negative longitudes
    if (lon < m.phi[m.np - 1] - two_pi || lon > m.phi[0] + two_pi) return nan("");
    if (lon < m.phi[0]) {
        ip0 = m.np - 1; ip1 = 0; p0 = m.phi[m.np - 1] - two_pi; p1 = m.phi[0];
    } else if (lon >= m.phi[m.np - 1]) {
        ip0 = m.np - 1; ip1 = 0; p0 = m.phi[m.np - 1]; p1 = m.phi[0] + two_pi;
    } else {
        ip0 = find_interval(m.phi, m.np, lon); ip1 = ip0 + 1; p0 = m.phi[ip0]; p1 = m.phi[ip1];
    }
    const int it = find_interval(m.lat, m.nt, lat), ir = find_interval(m.r, m.nr, r);
    const double tp = (lon - p0) / (p1 - p0);
    const double tt = (lat - m.lat[it]) / (m.lat[it + 1] - m.lat[it]);
    const double tr = (r - m.r[ir]) / (m.r[ir + 1] - m.r[ir]);
    const double wp[2] = {1.0 - tp, tp}, wt[2] = {1.0 - tt, tt}, wr[2] = {1.0 - tr, tr};
    const int ips[2] = {ip0, ip1};
    double v = 0.0;
    // weighted 8-corner sum in itertools.product order, weight = ((1*wp)*wt)*wr (scipy _evaluate_linear)
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const size_t o = ((size_t)ips[a] * m.nt + (size_t)(it + b)) * m.nr + (size_t)(ir + c);
                v = v + (double)m.data[o] * (((1.0 * wp[a]) * wt[b]) * wr[c]);
            }
    return v;
}

// The observer's view of the model (include/rtgrff.h, "Observer view"): sin / cos of the solar B0 and P angles.  `on`
// is 0 for B0 = P = 0, and the launch then picks the VIEW = false instantiation of a kernel: the fixed equatorial
// view's code as it was, so that its results are the same bit for bit.  (A run-time branch around the rotation is not
// enough: it changes which products the compiler contracts into FMAs elsewhere in the kernel.)
struct ViewRot {
    int on;
    double sb, cb, sp, cp;
};

// observer-frame point -> model-aligned point: undo P (a rotation about the line of sight z), then B0 (about x)
__device__ __forceinline__ void view_to_model(const ViewRot &v, double &x, double &y, double &z)
{
    const double x1 = x * v.cp + y * v.sp, y1 = -x * v.sp + y * v.cp;
    x = x1;
    y = y1 * v.cb + z * v.sb;
    z = -y1 * v.sb + z * v.cb;
}

// model-aligned vector -> observer frame: the transpose of view_to_model
__device__ __forceinline__ void model_to_view(const ViewRot &v, double &x, double &y, double &z)
{
    const double y1 = y * v.cb - z * v.sb, z1 = y * v.sb + z * v.cb;
    const double x0 = x;
    x = x0 * v.cp - y1 * v.sp;
    y = x0 * v.sp + y1 * v.cp;
    z = z1;
}

struct ResampleArgs {
    SphMesh mesh;
    int nx, ny, nz;
    const double *xg, *yg, *zg;      // the cube's node coordinates exactly as the caller holds them (an
                                     // x0 + i*dx reconstruction is 4e-16 off and flips the longitude of
                                     // nodes that sit exactly on the rotation axis)
    double phi0_offset_rad, r_min, scale, fill;
    int fill_nonfinite;              // 1: NaN/inf -> fill (fill_nan is not None); 0: keep NaN
    double *out;                     // [nx][ny][nz]
    ViewRot view;
};

// One thread per cube node.  cart_to_sph(x, -z, y, phi0) as build_rays.py:93 of the model-aligned point: the solar
// rotation axis is its +y, longitude is measured in the x / -z plane.
template <bool VIEW>
__global__ void __launch_bounds__(256) resample_spherical_kernel(const ResampleArgs a)
{
    const int64_t nvox = (int64_t)a.nx * a.ny * a.nz;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nvox;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(q % a.nz), j = (int)((q / a.nz) % a.ny), i = (int)(q / ((int64_t)a.ny * a.nz));
        double x = a.xg[i], y = a.yg[j], z = a.zg[k];
        if constexpr (VIEW) view_to_model(a.view, x, y, z);
        const double cx = x, cy = -z, cz = y;
        const double r = sqrt(cx * cx + cy * cy + cz * cz);
        const double colat = acos(fmin(1.0, fmax(-1.0, cz / r)));
        double lon = atan2(cy, cx) + a.phi0_offset_rad;
        if (lon < 0.0) lon += 6.283185307179586476925286766559;
        const double lat = 1.5707963267948966192313216916398 - colat;
        double v = nan("");
        if (isfinite(r) && r >= a.r_min) v = sample_spherical(a.mesh, lon, lat, r) * a.scale;
        if (a.fill_nonfinite && !isfinite(v)) v = a.fill;
        a.out[q] = v;
    }
}

// Straight line-of-sight sampling of one spherical variable (script/resampling_MAS_LOS.py:141-231):
// pixel (i,j) at (x[j], y[i]); the LOS starts on the solar surface (inside the disk) or on the plane
// of the sky behind the limb (:198-201) and runs towards the observer over the z offsets zc[k];
// position -> cart_to_sph(x, -z, y, phi0) (:208); r < r_min -> NaN (:210-218).
struct LosArgs {
    SphMesh mesh;
    const double *x, *y, *zc;     // R_sun: pixel columns, pixel rows, cumulative z offsets
    int nx, ny, nz;
    double phi0_offset_rad, r_min, scale, z_eps;   // z_eps = 1e-6 m in R_sun (:199, :201)
    double *out;                  // [ny][nx][nz]
    ViewRot view;
};

// The LOS geometry is spherical, so it is laid out in the observer frame; only the sample point is turned to the model.
template <bool VIEW>
__global__ void __launch_bounds__(256) los_spherical_kernel(const LosArgs a)
{
    const int64_t total = (int64_t)a.ny * a.nx * a.nz;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(q % a.nz), j = (int)((q / a.nz) % a.nx), i = (int)(q / ((int64_t)a.nx * a.nz));
        double x = a.x[j], y = a.y[i];
        const double rho2 = x * x + y * y;
        const double z0 = (sqrt(rho2) < 1.0) ? sqrt(1.0 - rho2) - a.z_eps : -sqrt(rho2 - 1.0) - a.z_eps;
        double z = z0 + a.zc[k];
        if constexpr (VIEW) view_to_model(a.view, x, y, z);
        const double cx = x, cy = -z, cz = y;
        const double r = sqrt(cx * cx + cy * cy + cz * cz);
        const double colat = acos(fmin(1.0, fmax(-1.0, cz / r)));
        double lon = atan2(cy, cx) + a.phi0_offset_rad;
        if (lon < 0.0) lon += 6.283185307179586476925286766559;
        const double lat = 1.5707963267948966192313216916398 - colat;
        double v = nan("");
        if (r >= a.r_min) v = sample_spherical(a.mesh, lon, lat, r) * a.scale;
        a.out[q] = v;
    }
}

// los_spherical_kernel's geometry, expression for expression, for the fused LOS map (los_map.cuh), so that its samples
// are the ones rtgrff_sample_spherical_los returns.
// z of the first sample of the LOS through (x, y): on the disk surface, or behind the limb on the plane of the sky
__device__ __forceinline__ double los_z0(double x, double y, double z_eps)
{
    const double rho2 = x * x + y * y;
    return (sqrt(rho2) < 1.0) ? sqrt(1.0 - rho2) - z_eps : -sqrt(rho2 - 1.0) - z_eps;
}

// cart_to_sph(x, -z, y, phi0) of a cube point: longitude, latitude [rad] and r [R_sun]
__device__ __forceinline__ void los_sph(double x, double y, double z, double phi0_offset_rad, double &lon, double &lat,
                                        double &r)
{
    const double cx = x, cy = -z, cz = y;
    r = sqrt(cx * cx + cy * cy + cz * cz);
    const double colat = acos(fmin(1.0, fmax(-1.0, cz / r)));
    lon = atan2(cy, cx) + phi0_offset_rad;
    if (lon < 0.0) lon += 6.283185307179586476925286766559;
    lat = 1.5707963267948966192313216916398 - colat;
}

// Spherical (r, theta = colatitude from +y, phi in the x / -z plane) components at cube point (x, y, z) -> cube axes
// (compose_cubes_kernel's rotation)
__device__ __forceinline__ void sph_to_cube_b(double x, double y, double z, double br, double bt, double bp, double &bx,
                                              double &by, double &bz)
{
    const double cx = x, cy = -z, cz = y;              // model frame (build_rays.py:93)
    const double rr = sqrt(cx * cx + cy * cy + cz * cz), rho_c = sqrt(cx * cx + cy * cy);
    double mx = 0.0, my = 0.0, mz = 0.0;
    if (rr > 0.0 && rho_c > 0.0) {
        const double st = rho_c / rr, ct = cz / rr, cp = cx / rho_c, sp = cy / rho_c;
        mx = br * st * cp + bt * ct * cp - bp * sp;
        my = br * st * sp + bt * ct * sp + bp * cp;
        mz = br * ct - bt * st;
    } else if (rr > 0.0) {
        mz = br * (cz > 0.0 ? 1.0 : -1.0);
    }
    bx = mx; by = mz; bz = -my;                        // model (mx,my,mz) -> cube: x = mx, z = -my, y = mz
}

// sph_to_cube_b in the observer's view: the components are taken at the model-aligned point and the vector is turned
// back to the observer frame.  (x, y, z) is the observer-frame point.  VIEW = false: sph_to_cube_b itself.
template <bool VIEW>
__device__ __forceinline__ void sph_to_view_b(const ViewRot &v, double x, double y, double z, double br, double bt,
                                              double bp, double &bx, double &by, double &bz)
{
    if constexpr (VIEW) view_to_model(v, x, y, z);
    sph_to_cube_b(x, y, z, br, bt, bp, bx, by, bz);
    if constexpr (VIEW) model_to_view(v, bx, by, bz);
}

// script/resample_with_ray_tracing.py:269-293 on device: rho -> omega_pe (f64, for the gradient
// kernel) and n_e >= 0; T NaN -> 1e4; |B| = sqrt(br^2+bt^2+bp^2); optional Cartesian B vector.
struct ComposeArgs {
    const double *ne, *te, *br, *bt, *bp;   // resampled cubes; ne already in cm^-3, te in K, B in G
    int nx, ny, nz;
    const double *xg, *yg, *zg;
    double *omega_pe;                        // out f64
    float4 *fcube, *bcube;                   // out {ne, te, |B|, 0}, {bx, by, bz, 0} (bcube may be null)
    ViewRot view;                            // the view the slots were resampled with: B is turned back with it
};

template <bool VIEW>
__global__ void __launch_bounds__(256) compose_cubes_kernel(const ComposeArgs a)
{
    const int64_t nvox = (int64_t)a.nx * a.ny * a.nz;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nvox;
         q += (int64_t)gridDim.x * blockDim.x) {
        const double rho = a.ne[q];
        double w = 8.93e3 * sqrt(fmax(rho, 0.0)) * 2.0 * 3.14159265358979323846;   // :271
        if (!isfinite(w)) w = 0.0;                                                   // :273
        a.omega_pe[q] = w;
        const double ne = fmax(rho, 0.0);                                            // :279
        double te = a.te[q];
        if (!isfinite(te)) te = 1e4;                                                 // :284
        const double br = a.br[q], bt = a.bt[q], bp = a.bp[q];
        const double b = sqrt(br * br + bt * bt + bp * bp);                          // :293
        a.fcube[q] = make_float4((float)ne, (float)te, (float)b, 0.0f);
        if (a.bcube) {
            const int k = (int)(q % a.nz), j = (int)((q / a.nz) % a.ny), i = (int)(q / ((int64_t)a.ny * a.nz));
            double bx, by, bz;
            sph_to_view_b<VIEW>(a.view, a.xg[i], a.yg[j], a.zg[k], br, bt, bp, bx, by, bz);
            a.bcube[q] = make_float4((float)bx, (float)by, (float)bz, 0.0f);
        }
    }
}

}  // namespace rtgrff
