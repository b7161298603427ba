// LOS resampler for sm_100a: n_e, T, |B| (and optionally the B vector) gathered along recorded
// paths in ONE launch from one channel-interleaved cube of field nodes, with the validity mask and
// the segment lengths ds computed on the device.
//
// Replaces raytracingGRFF/gpu_raytrace.py:539-628 (trilinear_sample_uniform, launched once per
// field with a fresh H2D of the field each time, :698-700) and the host-side per-ray Python loop
// _compute_ds_from_valid (:473-486, called even on the CUDA path at :708).  The arithmetic is
// the float32 arithmetic numpy performs in _trilinear_numpy_uniform (:489-535): explicit
// round-to-nearest intrinsics keep nvcc from contracting a*b+c into an FMA, so values are
// bit-identical to the reference CPU path.
#pragma once

#include "common.cuh"

namespace rtgrff {

struct FieldSample {
    float ne, te, b;
    bool inb;
};

__device__ __forceinline__ float lerp_np(float a, float b, float t)
{
    // a*(1-t) + b*t with every operation rounded separately (gpu_raytrace.py:528-534)
    return __fadd_rn(__fmul_rn(a, __fsub_rn(1.0f, t)), __fmul_rn(b, t));
}

// gpu_raytrace.py:495-534 for the three fields at once.
__device__ __forceinline__ bool cell_of(const GridGeomF &g, float px, float py, float pz, int &i, int &j,
                                        int &k, float &tx, float &ty, float &tz)
{
    const float fx = __fmul_rn(__fsub_rn(px, g.x0), g.idx);
    const float fy = __fmul_rn(__fsub_rn(py, g.y0), g.idy);
    const float fz = __fmul_rn(__fsub_rn(pz, g.z0), g.idz);
    const bool inb = (fx >= 0.0f) && (fy >= 0.0f) && (fz >= 0.0f) && (fx <= g.fxl) && (fy <= g.fyl) && (fz <= g.fzl);
    if (!inb) return false;
    i = min(max((int)floorf(fx), 0), g.nx - 2);
    j = min(max((int)floorf(fy), 0), g.ny - 2);
    k = min(max((int)floorf(fz), 0), g.nz - 2);
    tx = fminf(fmaxf(__fsub_rn(fx, (float)i), 0.0f), 1.0f);
    ty = fminf(fmaxf(__fsub_rn(fy, (float)j), 0.0f), 1.0f);
    tz = fminf(fmaxf(__fsub_rn(fz, (float)k), 0.0f), 1.0f);
    return true;
}

// a*(1-t) + b*t on a channel pair, every operation rounded separately (packed FP32x2, no FMA)
__device__ __forceinline__ float2 lerp_np2(float2 a, float2 b, float2 u, float2 t)
{
    return __fadd2_rn(__fmul2_rn(a, u), __fmul2_rn(b, t));
}

#define RT_TRI_NP(m)                                                                              \
    lerp_np(lerp_np(lerp_np(c000.m, c100.m, tx), lerp_np(c010.m, c110.m, tx), ty),                \
            lerp_np(lerp_np(c001.m, c101.m, tx), lerp_np(c011.m, c111.m, tx), ty), tz)

// n_e, T, |B| from the first float4 of each node; `stride` = float4 per node (1, or 2 with the B vector).
__device__ __forceinline__ FieldSample sample_fields(const float4 *__restrict__ cube, int stride, const GridGeomF &g,
                                                     float px, float py, float pz, float fill_ne,
                                                     float fill_te, float fill_b)
{
    FieldSample o;
    int i, j, k;
    float tx, ty, tz;
    o.inb = cell_of(g, px, py, pz, i, j, k, tx, ty, tz);
    if (!o.inb) {
        o.ne = fill_ne; o.te = fill_te; o.b = fill_b;
        return o;
    }
    const size_t sz = (size_t)stride, sy = (size_t)g.nz * sz, sx = (size_t)g.ny * sy;
    const float4 *p = cube + ((size_t)i * sx + (size_t)j * sy + (size_t)k * sz);
    const float4 c000 = __ldg(p), c001 = __ldg(p + sz), c010 = __ldg(p + sy), c011 = __ldg(p + sy + sz);
    const float4 c100 = __ldg(p + sx), c101 = __ldg(p + sx + sz), c110 = __ldg(p + sx + sy),
                 c111 = __ldg(p + sx + sy + sz);
    // nesting order of the reference: x first, then y, then z (gpu_raytrace.py:528-534)
    o.ne = RT_TRI_NP(x);
    o.te = RT_TRI_NP(y);
    o.b = RT_TRI_NP(z);
    return o;
}
#undef RT_TRI_NP

// n_e, T (numpy-exact, as sample_fields) and the B vector at one point for the fused map's theta-aware
// path.  The B vector has no numpy twin in the reference (theta from B.t is an extension), so its
// three channels use fused lerps a + t (b - a) — a third of the arithmetic — and |B| comes from the
// vector: the |B| channel of the field cube is not interpolated at all.  o.b = |B vector| (float32).
// `nodes`: the 32-byte nodes {ne, te, |B|, 0, bx, by, bz, 0} (32-byte aligned), one load per corner, not kept in L1.
__device__ __forceinline__ FieldSample sample_fields_bvec_fast(const float4 *__restrict__ nodes, const GridGeomF &g,
                                                               float px, float py, float pz, float fill_ne,
                                                               float fill_te, float3 &bv)
{
    FieldSample o;
    int i, j, k;
    float tx, ty, tz;
    o.inb = cell_of(g, px, py, pz, i, j, k, tx, ty, tz);
    bv = make_float3(0.f, 0.f, 0.f);
    o.b = 0.0f;
    if (!o.inb) {
        o.ne = fill_ne; o.te = fill_te;
        return o;
    }
    const size_t sy = (size_t)g.nz * 2, sx = (size_t)g.ny * sy;
    const float4 *p = nodes + ((size_t)i * sx + (size_t)j * sy + (size_t)k * 2);
    const Float4x2 c000 = ldg256_no_l1(p), c001 = ldg256_no_l1(p + 2);
    const Float4x2 c010 = ldg256_no_l1(p + sy), c011 = ldg256_no_l1(p + sy + 2);
    const Float4x2 c100 = ldg256_no_l1(p + sx), c101 = ldg256_no_l1(p + sx + 2);
    const Float4x2 c110 = ldg256_no_l1(p + sx + sy), c111 = ldg256_no_l1(p + sx + sy + 2);
    const float2 tx2 = make_float2(tx, tx), ux2 = make_float2(__fsub_rn(1.0f, tx), __fsub_rn(1.0f, tx));
    const float2 ty2 = make_float2(ty, ty), uy2 = make_float2(__fsub_rn(1.0f, ty), __fsub_rn(1.0f, ty));
    const float2 tz2 = make_float2(tz, tz), uz2 = make_float2(__fsub_rn(1.0f, tz), __fsub_rn(1.0f, tz));
#define RT_NT(c) make_float2((c).lo.x, (c).lo.y)
#define RT_BXY(c) make_float2((c).hi.x, (c).hi.y)
    const float2 nt = lerp_np2(
        lerp_np2(lerp_np2(RT_NT(c000), RT_NT(c100), ux2, tx2), lerp_np2(RT_NT(c010), RT_NT(c110), ux2, tx2), uy2, ty2),
        lerp_np2(lerp_np2(RT_NT(c001), RT_NT(c101), ux2, tx2), lerp_np2(RT_NT(c011), RT_NT(c111), ux2, tx2), uy2, ty2),
        uz2, tz2);
    o.ne = nt.x; o.te = nt.y;
#define RT_FL2(a, b, t) __ffma2_rn(t, __fadd2_rn(b, make_float2(-(a).x, -(a).y)), a)
#define RT_FL(a, b, t) fmaf(t, (b) - (a), a)
    const float2 bxy = RT_FL2(RT_FL2(RT_FL2(RT_BXY(c000), RT_BXY(c100), tx2), RT_FL2(RT_BXY(c010), RT_BXY(c110), tx2), ty2),
                              RT_FL2(RT_FL2(RT_BXY(c001), RT_BXY(c101), tx2), RT_FL2(RT_BXY(c011), RT_BXY(c111), tx2), ty2), tz2);
    bv.x = bxy.x; bv.y = bxy.y;
    bv.z = RT_FL(RT_FL(RT_FL(c000.hi.z, c100.hi.z, tx), RT_FL(c010.hi.z, c110.hi.z, tx), ty),
                 RT_FL(RT_FL(c001.hi.z, c101.hi.z, tx), RT_FL(c011.hi.z, c111.hi.z, tx), ty), tz);
#undef RT_FL2
#undef RT_FL
#undef RT_NT
#undef RT_BXY
    return o;
}

__device__ __forceinline__ bool sample_valid(float x, float y, float z, float s)
{
    // valid = isfinite(pos).all & isfinite(s) & (s > 0)   (gpu_raytrace.py:644)
    return isfinite(x) && isfinite(y) && isfinite(z) && isfinite(s) && (s > 0.0f);
}

// |a-b| in float32 as numpy's axis norm computes it (gpu_raytrace.py:484).
__device__ __forceinline__ float dist_np(float ax, float ay, float az, float bx, float by, float bz)
{
    const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
}

// The same length with fused products and MUFU.SQRT (2 ulp): for the fused map, where the segment
// length feeds the transfer (T_b tolerance 1e-4) and never leaves the kernel as a float32 `ds`.
__device__ __forceinline__ float dist_fast(float ax, float ay, float az, float bx, float by, float bz)
{
    const float dx = ax - bx, dy = ay - by, dz = az - bz;
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaf(dx, dx, fmaf(dy, dy, dz * dz))));
    return r;
}

__device__ __forceinline__ float sqrt_approx(float v)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));     // MUFU.SQRT, 2 ulp
    return r;
}

// First segment (gpu_raytrace.py:482): numpy's 1-D norm goes through BLAS sdot, which accumulates
// the float32 products in a double before rounding (see oracle/oracle_sampler.c).
__device__ __forceinline__ float dist_first_np(float ax, float ay, float az, float bx, float by, float bz)
{
    const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    const double acc = __dadd_rn(__dadd_rn((double)__fmul_rn(dx, dx), (double)__fmul_rn(dy, dy)),
                                 (double)__fmul_rn(dz, dz));
    return __fsqrt_rn((float)acc);
}

struct SampleArgs {
    const float4 *fcube;
    int field_stride;        // float4 per field node (rtgrff_ctx::field_stride)
    GridGeomF g;
    int64_t n_rec, n_rays;
    // exactly one of the two position sources is set
    const float *pos_aos;    // (rec, ray, 3) float32 — the reference's API layout
    const double *pos_soa;   // [rec][3][ray] float64 — left by trace_rays_kernel
    const float *s32;        // (rec, ray) float32 or nullptr
    const double *s64;       // [rec][ray] float64 or nullptr
    const float *ray_start;  // (ray, 3)
    float r_sun_cm, fill_ne, fill_te, fill_b;
    float *ne, *te, *b, *ds, *s_out;
    uint8_t *valid;
    int64_t q_begin, q_end;  // the samples [q_begin, q_end) of the (rec, ray) array this launch works on
                             // (q_end = 0: all) — the chunks of the pipelined host path
};

__device__ __forceinline__ void load_sample(const SampleArgs &a, int64_t rec, int64_t ray, float &x, float &y,
                                            float &z, float &s)
{
    const size_t n = (size_t)a.n_rays;
    if (a.pos_aos) {
        const float *p = a.pos_aos + ((size_t)rec * n + (size_t)ray) * 3;
        x = p[0]; y = p[1]; z = p[2];
    } else {
        const double *p = a.pos_soa + (size_t)rec * 3 * n + (size_t)ray;
        x = (float)p[0]; y = (float)p[n]; z = (float)p[2 * n];  // _as_float32_c (gpu_raytrace.py:642)
    }
    const size_t q = (size_t)rec * n + (size_t)ray;
    s = a.s32 ? a.s32[q] : (a.s64 ? (float)a.s64[q] : 1.0f);
}

// One thread per sample; consecutive threads = consecutive rays of one record (coalesced).
// ds needs the previous VALID record of the same ray: the thread walks back until it finds one
// (usually one step), which keeps the kernel fully parallel over samples.
__global__ void __launch_bounds__(256) sample_paths_kernel(const SampleArgs a)
{
    const int64_t total = a.q_end > 0 ? a.q_end : a.n_rec * a.n_rays;
    for (int64_t q = a.q_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total;
         q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t rec = q / a.n_rays, ray = q - rec * a.n_rays;
        float x, y, z, s;
        load_sample(a, rec, ray, x, y, z, s);
        const bool v = sample_valid(x, y, z, s);
        // the stride as a literal on each side: the 16-byte nodes keep the address arithmetic of a one-layout kernel
        const FieldSample f = a.field_stride == 1 ? sample_fields(a.fcube, 1, a.g, x, y, z, a.fill_ne, a.fill_te, a.fill_b)
                                                  : sample_fields(a.fcube, 2, a.g, x, y, z, a.fill_ne, a.fill_te, a.fill_b);
        float ds = 0.0f;
        if (v) {
            int64_t pr = rec - 1;
            float px = 0.f, py = 0.f, pz = 0.f, ps;
            for (; pr >= 0; --pr) {
                load_sample(a, pr, ray, px, py, pz, ps);
                if (sample_valid(px, py, pz, ps)) break;
            }
            if (pr >= 0) {
                ds = __fmul_rn(dist_np(x, y, z, px, py, pz), a.r_sun_cm);
            } else {
                const float *st = a.ray_start + (size_t)ray * 3;
                ds = __fmul_rn(dist_first_np(x, y, z, st[0], st[1], st[2]), a.r_sun_cm);
            }
        }
        a.ne[q] = f.ne; a.te[q] = f.te; a.b[q] = f.b; a.ds[q] = ds;
        a.valid[q] = v ? 1 : 0;
        if (a.s_out) a.s_out[q] = s;
    }
}

// {ne, te, b} float32 cubes -> float4 {ne, te, b, 0} at out[q * stride]; {bx,by,bz} likewise (out = nodes + 1).
__global__ void interleave3_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                   const float *__restrict__ c, float4 *__restrict__ out, int stride, int64_t n)
{
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n;
         q += (int64_t)gridDim.x * blockDim.x)
        out[q * stride] = make_float4(a[q], b[q], c[q], 0.0f);
}

// the inverse: the float4 at in[q * stride] -> three planar arrays (rtgrff_export_cubes)
__global__ void deinterleave3_kernel(const float4 *__restrict__ in, int stride, float *__restrict__ a,
                                     float *__restrict__ b, float *__restrict__ c, int64_t n)
{
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n;
         q += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = in[q * stride];
        a[q] = v.x; b[q] = v.y; c[q] = v.z;
    }
}

}  // namespace rtgrff
