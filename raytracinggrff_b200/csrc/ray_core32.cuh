// Ray stepper for sm_100a: FP64 master state, FP32 RHS relative to the CACHED CELL, the cell held in
// registers as its trilinear POLYNOMIAL (fed from a cell-major polynomial cube), packed FP32x2 (FFMA2).
//
// Same mathematics as ray_integrator.cuh (build_rays.py:158-239) reorganised around what ncu showed
// (DESIGN.md 4.1 has the sequence; profiles/r1a_*, r1d_*, r1f_*):
//
//  * The ray's position and wave vector stay FP64 (the "master" state): every step adds
//    (double)sum * (dt/6 * C_R), so the accumulation over thousands of steps is exact to 1e-16
//    and no rounded constant multiplies the accumulated path.
//  * Within a step everything is FP32 and relative to the cached cell: the master position is
//    converted once per step, the four RK4 stages and the two cross-section rays are float
//    offsets from it.  Cell fractions carry 6e-8 of a cell (~1e-9 R_sun), the corners are FP32
//    anyway, omega = sqrt(w^2+k^2) and the derivatives need 1e-7 relative: increments are
//    ~1e-3 R_sun, so the per-step error is ~1e-10 R_sun and random.
//  * The cached cell lives in 32 registers as the coefficients of its trilinear polynomial
//        f = (a0 + az z) + y (ay + ayz z) + x ((ax + axz z) + y (axy + axyz z))
//    for the channel pairs {omega_pe, d/dz} and {d/dx, d/dy}: one RHS is 14 packed FFMA2 with a
//    dependency depth of 3 (nested lerps: 14 FMUL2 + 14 FFMA2, depth 6).
//  * The x,y components of every vector of a stage (position offsets, k, v, g and the RK4 sums)
//    live in register pairs and are updated with packed FP32x2 instructions (FFMA2 / FMUL2 / FADD2
//    take a scalar broadcast operand, so nothing has to be duplicated): 15 instead of 22
//    instructions in the tail of an RHS.
//  * Fast path of an RHS = one range test (VIMNMX3.U32 + ISETP on the bit patterns: 0 <= t < 1)
//    + the evaluation, ~55 instructions.  Everything else — leaving the cell, the cube bounds,
//    the re-fetch — is the slow path (move_cell), which 1-5 of a warp's 32 lanes take at a time:
//    it is kept short by the polynomial cube (8 LDG.128 from one 128-byte line, no differencing)
//    and by a per-step `edge` flag that drops the bounds logic in the interior.
//  * One RHS body per RK4 stage (the stage loop is unrolled: constant weights), the three rays
//    of a step (central + two pencil rays) are a rolled loop, the face handling is a run-time
//    flag: the stepper is ~1500 SASS instructions where the first version (16 inlined copies of
//    the RHS, 134 KB of SASS) lost 30 % of its issue slots to instruction-cache misses.
//    render_map_kernel inlines one more copy of the central ray's stages (step32_central, ~660
//    instructions) for the steps between two records.
#pragma once

#include "ray_integrator.cuh"

namespace rtgrff {

// The cached cell: element offset of its (i,j,k) corner (-1 = empty), its integer coordinates and
// the polynomial coefficients of the channel pairs L = {omega_pe, d/dz}, H = {d/dx, d/dy}.
struct Cell {
    int off;
    int ci, cj, ck;
    float2 l0, lz, ly, lyz, lx, lxz, lxy, lxyz;
    float2 h0, hz, hy, hyz, hx, hxz, hxy, hxyz;
};

__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }

// The 8 corners of a cell -> the coefficients of its trilinear polynomial, 8 float4
// {l0,lz} {ly,lyz} {lx,lxz} {lxy,lxyz} {h0,hz} {hy,hyz} {hx,hxz} {hxy,hxyz}.
__device__ __forceinline__ void cell_poly(const float4 &c000, const float4 &c001, const float4 &c010, const float4 &c011,
                                          const float4 &c100, const float4 &c101, const float4 &c110, const float4 &c111,
                                          Cell &c)
{
#define RT_POLY(LO, a0, az, ay, ayz, ax, axz, axy, axyz)                                          \
    {                                                                                             \
        const float2 d00 = sub2(LO(c001), LO(c000)), d01 = sub2(LO(c011), LO(c010));              \
        const float2 d10 = sub2(LO(c101), LO(c100)), d11 = sub2(LO(c111), LO(c110));              \
        const float2 y0 = sub2(LO(c010), LO(c000)), y1 = sub2(LO(c110), LO(c100));                \
        const float2 yz0 = sub2(d01, d00), yz1 = sub2(d11, d10);                                  \
        c.a0 = LO(c000); c.az = d00; c.ay = y0; c.ayz = yz0;                                      \
        c.ax = sub2(LO(c100), LO(c000)); c.axz = sub2(d10, d00);                                  \
        c.axy = sub2(y1, y0); c.axyz = sub2(yz1, yz0);                                            \
    }
    // channel pairs L = {omega_pe, d/dz}, H = {d/dx, d/dy}: the x,y components of the gradient come out of the
    // evaluation as one register pair, ready for the packed (FFMA2) stage updates of step32
#define RT_LO(c) make_float2((c).x, (c).w)
#define RT_HI(c) make_float2((c).y, (c).z)
    RT_POLY(RT_LO, l0, lz, ly, lyz, lx, lxz, lxy, lxyz)
    RT_POLY(RT_HI, h0, hz, hy, hyz, hx, hxz, hxy, hxyz)
#undef RT_POLY
#undef RT_LO
#undef RT_HI
}

// The cell at `off` from the NODE cube (no polynomial cube: cubes too large to afford 128 B per cell): the 8 corners
// are fetched and differenced here.  Out of line: with the polynomial cube present this never runs, and inlined at
// every site a stage can leave the cached cell it put ~650 cold instructions into the middle of the hot loop.
__device__ __noinline__ void load_cell_nodes(const float4 *__restrict__ nodes, int sx, int sy, int off, Cell *out)
{
    const float4 *p = nodes + off;
    Cell c;
    cell_poly(__ldg(p), __ldg(p + 1), __ldg(p + sy), __ldg(p + sy + 1), __ldg(p + sx), __ldg(p + sx + 1),
              __ldg(p + sx + sy), __ldg(p + sx + sy + 1), c);
    *out = c;
}

// Make the cell at element offset `off` the cached one.  With the cell-major polynomial cube
// (build_poly_cube_kernel) that is 8 LDG.128 from one 128-byte line; without it: load_cell_nodes.
__device__ __forceinline__ void load_cell(const RayCube &C, int off, Cell &c)
{
    if (C.pc) {
        c.off = off;
        const float4 *p = C.pc + (size_t)off * 8;
        const float4 q0 = __ldg(p), q1 = __ldg(p + 1), q2 = __ldg(p + 2), q3 = __ldg(p + 3);
        const float4 q4 = __ldg(p + 4), q5 = __ldg(p + 5), q6 = __ldg(p + 6), q7 = __ldg(p + 7);
#define RT_A(q) make_float2((q).x, (q).y)
#define RT_B(q) make_float2((q).z, (q).w)
        c.l0 = RT_A(q0); c.lz = RT_B(q0); c.ly = RT_A(q1); c.lyz = RT_B(q1);
        c.lx = RT_A(q2); c.lxz = RT_B(q2); c.lxy = RT_A(q3); c.lxyz = RT_B(q3);
        c.h0 = RT_A(q4); c.hz = RT_B(q4); c.hy = RT_A(q5); c.hyz = RT_B(q5);
        c.hx = RT_A(q6); c.hxz = RT_B(q6); c.hxy = RT_A(q7); c.hxyz = RT_B(q7);
#undef RT_A
#undef RT_B
        return;
    }
    // through a temporary: passing the address of the cache itself would pin all of it in local memory
    Cell t;
    load_cell_nodes(C.c, C.sx, C.sy, off, &t);
    c.off = off;
    c.l0 = t.l0; c.lz = t.lz; c.ly = t.ly; c.lyz = t.lyz; c.lx = t.lx; c.lxz = t.lxz; c.lxy = t.lxy; c.lxyz = t.lxyz;
    c.h0 = t.h0; c.hz = t.hz; c.hy = t.hy; c.hyz = t.hyz; c.hx = t.hx; c.hxz = t.hxz; c.hxy = t.hxy; c.hxyz = t.hxyz;
}

// Node cube -> cell-major polynomial cube: cell (i,j,k), i < nx-1 etc., at [off*8, off*8+8) with the node
// cube's offset off = (i*ny + j)*nz + k (the entries of the last node of each axis stay unused).
__global__ void build_poly_cube_kernel(const float4 *__restrict__ nodes, float4 *__restrict__ pc, int nx, int ny, int nz)
{
    const int64_t nvox = (int64_t)nx * ny * nz;
    const int sy = nz, sx = ny * nz;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nvox; q += (int64_t)gridDim.x * blockDim.x) {
        const int k = (int)(q % nz), j = (int)((q / nz) % ny), i = (int)(q / sx);
        if (i >= nx - 1 || j >= ny - 1 || k >= nz - 1) continue;
        const float4 *p = nodes + q;
        Cell c;
        cell_poly(p[0], p[1], p[sy], p[sy + 1], p[sx], p[sx + 1], p[sx + sy], p[sx + sy + 1], c);
        float4 *o = pc + q * 8;
        o[0] = make_float4(c.l0.x, c.l0.y, c.lz.x, c.lz.y);     o[1] = make_float4(c.ly.x, c.ly.y, c.lyz.x, c.lyz.y);
        o[2] = make_float4(c.lx.x, c.lx.y, c.lxz.x, c.lxz.y);   o[3] = make_float4(c.lxy.x, c.lxy.y, c.lxyz.x, c.lxyz.y);
        o[4] = make_float4(c.h0.x, c.h0.y, c.hz.x, c.hz.y);     o[5] = make_float4(c.hy.x, c.hy.y, c.hyz.x, c.hyz.y);
        o[6] = make_float4(c.hx.x, c.hx.y, c.hxz.x, c.hxz.y);   o[7] = make_float4(c.hxy.x, c.hxy.y, c.hxyz.x, c.hxyz.y);
    }
}

// 0 <= t < 1 as one unsigned compare on the bit pattern (negative, NaN and -0 fail).
__device__ __forceinline__ bool in_unit(float t) { return __float_as_uint(t) < 0x3f800000u; }

// Slow path of an RHS evaluation: the point (tx,ty,tz) — coordinates relative to the cached cell —
// lies outside it.  Moves the cache to the cell that holds the point, rebases the step's base
// position (px,py,pz) and the point onto the new cell.  `edge` (per step): the cached cell is within
// three cells of a face, so a stage of this step may leave the cube — then the scipy bounds
// g[0] <= x <= g[n-1] apply (the last node belongs to cell n-2 with t = 1) and the function returns
// false, leaving everything untouched, for a point outside the cube: that stage contributes a zero
// derivative (build_rays.py:169-174).  In the interior no stage can get out (a step moves every
// stage by less than a cell, see step32) and the tests are skipped.  A NaN coordinate converts to
// shift 0: the cell stays, the evaluation yields NaN and the stage is invalid.
__device__ __forceinline__ bool move_cell(const RayCube &C, Cell &c, bool edge, float &px, float &py, float &pz,
                                          float &tx, float &ty, float &tz)
{
    const int sx = __float2int_rd(tx), sy = __float2int_rd(ty), sz = __float2int_rd(tz);   // floor
    int ni = c.ci + sx, nj = c.cj + sy, nk = c.ck + sz;
    float fx = (float)sx, fy = (float)sy, fz = (float)sz;
    float ux = tx - fx, uy = ty - fy, uz = tz - fz;
    if (edge) {
        if (ni == C.nx - 1 && ux == 0.0f) { ni = C.nx - 2; ux = 1.0f; fx -= 1.0f; }
        if (nj == C.ny - 1 && uy == 0.0f) { nj = C.ny - 2; uy = 1.0f; fy -= 1.0f; }
        if (nk == C.nz - 1 && uz == 0.0f) { nk = C.nz - 2; uz = 1.0f; fz -= 1.0f; }
        if ((unsigned)ni > (unsigned)(C.nx - 2) || (unsigned)nj > (unsigned)(C.ny - 2) ||
            (unsigned)nk > (unsigned)(C.nz - 2))
            return false;
    }
    const int off = (ni * C.ny + nj) * C.nz + nk;
    if (off != c.off) load_cell(C, off, c);
    c.ci = ni; c.cj = nj; c.ck = nk;
    px -= fx; py -= fy; pz -= fz;
    tx = ux; ty = uy; tz = uz;
    return true;
}

struct Deriv32P {
    float2 vxy; float vz;   // k / omega                          (dr/dt = C_R * v)
    float2 gxy; float gz;   // (omega_pe/omega) * grad omega_pe   (dk/dt = -C_R * g)
};

__device__ __forceinline__ float2 bc2(float v) { return make_float2(v, v); }

// One RHS evaluation at p + d, all in cell units relative to the CACHED cell: p is the step's base
// position (rebased when the cache moves), d the offset of this stage of this ray from it; the x,y
// components in register pairs.  The common case — the point is inside the cached cell — costs one
// range test; the cell change, the bounds of the cube and the re-fetch all live on the slow path.
__device__ __forceinline__ Deriv32P rhs32p(const RayCube &C, Cell &cache, bool edge, float2 &pxy, float &pz, float2 dxy, float dz,
                                           float2 kxy, float kz)
{
    Deriv32P d;
    float2 txy = __fadd2_rn(pxy, dxy);
    float tz = pz + dz;
    if (!(in_unit(txy.x) & in_unit(txy.y) & in_unit(tz))) {
        if (!move_cell(C, cache, edge, pxy.x, pxy.y, pz, txy.x, txy.y, tz)) {
            d.vxy = make_float2(0.0f, 0.0f); d.gxy = make_float2(0.0f, 0.0f); d.vz = d.gz = 0.0f;
            return d;
        }
    }
    const float2 tz2 = bc2(tz), ty2 = bc2(txy.y), tx2 = bc2(txy.x);
    // {omega_pe, d/dz}
    const float2 wz = __ffma2_rn(
        __ffma2_rn(__ffma2_rn(cache.lxyz, tz2, cache.lxy), ty2, __ffma2_rn(cache.lxz, tz2, cache.lx)), tx2,
        __ffma2_rn(__ffma2_rn(cache.lyz, tz2, cache.ly), ty2, __ffma2_rn(cache.lz, tz2, cache.l0)));
    // {d/dx, d/dy}
    const float2 gg = __ffma2_rn(
        __ffma2_rn(__ffma2_rn(cache.hxyz, tz2, cache.hxy), ty2, __ffma2_rn(cache.hxz, tz2, cache.hx)), tx2,
        __ffma2_rn(__ffma2_rn(cache.hyz, tz2, cache.hy), ty2, __ffma2_rn(cache.hz, tz2, cache.h0)));
    const float w = wz.x;
    const float om2 = fmaf(w, w, fmaf(kxy.x, kxy.x, fmaf(kxy.y, kxy.y, kz * kz)));
    float inv_om;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(inv_om) : "f"(om2));   // MUFU.RSQ, 2 ulp; omega^2 ~ 1e17
    const float a = w * inv_om;
    d.vxy = __fmul2_rn(kxy, bc2(inv_om)); d.vz = kz * inv_om;
    d.gxy = __fmul2_rn(gg, bc2(a)); d.gz = a * wz.y;
    // valid = isfinite(omega_pe) & isfinite(omega) & (omega > 0)   (build_rays.py:169); a non-finite
    // omega_pe or k makes omega^2 non-finite, so one range test on omega^2 covers all three:
    // 0 < omega^2 < inf  <=>  bit pattern in [1, 0x7f7fffff].  The invalid stage (a zero derivative) is the
    // rare case: the zeros are written on that branch only, not materialised ahead of every evaluation.
    if (__builtin_expect(__float_as_uint(om2) - 1u >= 0x7f7fffffu, 0)) {
        d.vxy = make_float2(0.0f, 0.0f); d.gxy = make_float2(0.0f, 0.0f); d.vz = d.gz = 0.0f;
    }
    return d;
}

// Largest distance, in cells, between the master position of a step and any stage of any of its
// three rays (|v| <= 1: a full step plus the pencil offset eps = perturb * step).  The FP32 stepper
// works for any value (positions are relative to the cached cell, whole-cell shifts are exact); the
// host keeps it below kMaxStageOffsetCells so that cell-relative coordinates stay small (FP32
// precision) and falls back to the FP64 stepper beyond.
constexpr double kMaxStageOffsetCells = 8.0;
__host__ __device__ inline double max_stage_offset_cells(double dt, double perturb_ratio, double idx, double idy, double idz)
{
    const double i = fmax(idx, fmax(idy, idz));
    return (1.0 + fabs(perturb_ratio)) * fabs(dt) * kC_R * i;     // dt < 0 traces backwards
}

// Per-launch float constants derived from dt and the grid (uniform across the grid).
struct StepConst {
    float hx, hy, hz;     // 0.5*dt*C_R/dx : half-step position offset per unit v, in cells
    float hk;             // 0.5*dt*C_R    : half-step k offset per unit g
    float c6r;            // dt/6*C_R      : step displacement per unit sum(v), R_sun
    float ix, iy, iz;     // 1/dx          : R_sun -> cells
    double c6;            // dt/6*C_R in double: master-state increments
    float perturb;
    int margin;           // cells around the cached cell a step can touch (see step32): 3 * ceil(max stage offset)
};

__host__ __device__ __forceinline__ StepConst make_step_const(const RayCube &C, double dt, double perturb_ratio)
{
    StepConst k;
    const double h = 0.5 * dt * kC_R;
    k.hx = (float)(h * C.idx); k.hy = (float)(h * C.idy); k.hz = (float)(h * C.idz);
    k.hk = (float)h;
    k.c6 = dt / 6.0 * kC_R;
    k.c6r = (float)k.c6;
    k.ix = (float)C.idx; k.iy = (float)C.idy; k.iz = (float)C.idz;
    k.perturb = (float)perturb_ratio;
    k.margin = 3 * (int)ceil(fmax(1e-9, max_stage_offset_cells(dt, perturb_ratio, C.idx, C.idy, C.idz)));
    return k;
}

// Before the first step of a ray: cache the cell of its start position (kept out of the step loop).  A start
// outside the cube (or NaN) leaves the cache empty: step32 then reports the ray frozen at every step.
__device__ __forceinline__ void init_cell(const RayCube &C, const State &s, Cell &cache)
{
    cache.off = -1;
    if (!in_cube(C, s.rx, s.ry, s.rz)) return;
    const double fx = (s.rx - C.x0) * C.idx, fy = (s.ry - C.y0) * C.idy, fz = (s.rz - C.z0) * C.idz;
    cache.ci = min((int)fx, C.nx - 2); cache.cj = min((int)fy, C.ny - 2); cache.ck = min((int)fz, C.nz - 2);
    load_cell(C, (cache.ci * C.ny + cache.cj) * C.nz + cache.ck, cache);
}

// Start of a step, shared by step32 and step32_central: the `edge` flag, the master position relative to
// the cached cell (FP64 -> FP32 once per step) and k in FP32.  Returns false when the ray is frozen.
__device__ __forceinline__ bool step32_begin(const RayCube &C, const StepConst &K, const Cell &cache, const State &s,
                                             bool &edge, float2 &pxy, float &pz, float2 &kxy, float &kz)
{
    const double fx = (s.rx - C.x0) * C.idx, fy = (s.ry - C.y0) * C.idy, fz = (s.rz - C.z0) * C.idz;
    if (cache.off < 0) return false;      // the ray started outside the cube (init_cell): frozen for ever
    // The cached cell is the cell of the last stage evaluated in the previous step, within m cells of
    // the previous master position (m = ceil of the largest stage offset, 1 for the usual dt); a step
    // moves the master by at most m cells and every stage of this step lies within m of the new
    // master: all cells this step can touch are within K.margin = 3 m of the cached one.  Only if
    // that reaches a face can the master or a stage be outside the cube: exact scipy tests then (a
    // frozen ray stays in this state), none in the interior.
    const int mg = K.margin;
    edge = (cache.ci < mg) | (cache.ci > C.nx - 2 - mg) | (cache.cj < mg) | (cache.cj > C.ny - 2 - mg) |
           (cache.ck < mg) | (cache.ck > C.nz - 2 - mg);
    if (edge && !in_cube(C, s.rx, s.ry, s.rz)) return false;
    pxy = make_float2((float)(fx - (double)cache.ci), (float)(fy - (double)cache.cj));
    pz = (float)(fz - (double)cache.ck);
    kxy = make_float2((float)s.kx, (float)s.ky);
    kz = (float)s.kz;
    return true;
}

// The four RK4 stages of one ray that starts (qxy, qz) cells from the step's base position: the sums
// k1 + 2 k2 + 2 k3 + k4 of v and of g.
__device__ __forceinline__ void rk4_stages32(const RayCube &C, const StepConst &K, Cell &cache, bool edge, float2 &pxy,
                                             float &pz, float2 qxy, float qz, float2 kxy, float kz, float2 &avxy,
                                             float &avz, float2 &agxy, float &agz)
{
    const float2 h1xy = make_float2(K.hx, K.hy), h2xy = make_float2(2.0f * K.hx, 2.0f * K.hy);
    float2 dxy = qxy, skxy = kxy;
    float dz = qz, skz = kz;
#pragma unroll          // the four stages unrolled (constant weights); the rays of a step are a rolled loop (step32)
    for (int st = 0; st < 4; ++st) {
        const Deriv32P d = rhs32p(C, cache, edge, pxy, pz, dxy, dz, skxy, skz);
        if (st == 0) {        // (0 + x is not x for x = -0: spelled out, the compiler would keep the FADDs)
            avxy = d.vxy; avz = d.vz; agxy = d.gxy; agz = d.gz;
        } else {
            const float w = (st == 3) ? 1.0f : 2.0f;
            avxy = __ffma2_rn(bc2(w), d.vxy, avxy); avz = fmaf(w, d.vz, avz);
            agxy = __ffma2_rn(bc2(w), d.gxy, agxy); agz = fmaf(w, d.gz, agz);
        }
        // stages 2, 3 at dt/2, stage 4 at dt (K.h* are half steps)
        dxy = __ffma2_rn((st < 2) ? h1xy : h2xy, d.vxy, qxy);
        dz = fmaf((st < 2) ? K.hz : 2.0f * K.hz, d.vz, qz);
        const float ak = (st < 2) ? -K.hk : -2.0f * K.hk;
        skxy = __ffma2_rn(bc2(ak), d.gxy, kxy); skz = fmaf(ak, d.gz, kz);
    }
}

// The central ray's sums -> the FP64 master state.  Returns whether the ray moved (some stage derivative
// is not exactly zero).
__device__ __forceinline__ bool step32_commit(const StepConst &K, State &s, float2 avxy, float avz, float2 agxy, float agz)
{
    const float avx = avxy.x, avy = avxy.y, agx = agxy.x, agy = agxy.y;
    const bool moved = (fabsf(avx) + fabsf(avy) + fabsf(avz) + fabsf(agx) + fabsf(agy) + fabsf(agz)) != 0.0f;
    s.kx = fma((double)agx, -K.c6, s.kx); s.ky = fma((double)agy, -K.c6, s.ky); s.kz = fma((double)agz, -K.c6, s.kz);
    s.rx = fma((double)avx, K.c6, s.rx); s.ry = fma((double)avy, K.c6, s.ry); s.rz = fma((double)avz, K.c6, s.rz);
    return moved;
}

// One full step of the master state `s`: classic RK4 (build_rays.py:177-182) of the central ray
// and, when `want_s` (warp-uniform), the same RK4 on the two pencil rays displaced by eps along
// (e1, e2) _|_ t_hat with the cross-section ratio of this step (build_rays.py:209-239, with
// d = r_pert' - r_central' = eps*e + c6*(sum_v_pert - sum_v_central)).  Returns false when the ray
// is frozen: outside the cube / NaN, or every stage derivative exactly zero (the reference's
// update is then exactly zero too, for ever).
template <bool CS>
__device__ __forceinline__ bool step32(const RayCube &C, const StepConst &K, Cell &cache, State &s, bool want_s,
                                       float &s_step)
{
    bool edge;
    float2 pxy, kxy;
    float pz, kz;
    if (!step32_begin(C, K, cache, s, edge, pxy, pz, kxy, kz)) return false;
    const int n_rays = (CS && want_s) ? 3 : 1;
    const float2 ixy = make_float2(K.ix, K.iy);
    float2 oxy = make_float2(0.0f, 0.0f);           // displacement of the current ray from the central one, R_sun
    float oz = 0.0f;
    float2 cvxy = make_float2(0.0f, 0.0f);          // central ray: sum of v over the stages
    float cvz = 0.0f;
    float tx = 0.0f, ty = 0.0f, tz = 0.0f, e2x = 0.0f, e2y = 0.0f, e2z = 0.0f, eps = 0.0f;
    float d1x = 0.0f, d1y = 0.0f, d1z = 0.0f;
    bool moved = false;
#pragma unroll 1
    for (int q = 0; q < n_rays; ++q) {
        const float2 qxy = __fmul2_rn(oxy, ixy);                      // start of this ray relative to p, cells
        const float qz = oz * K.iz;
        float2 avxy, agxy;
        float avz, agz;
        rk4_stages32(C, K, cache, edge, pxy, pz, qxy, qz, kxy, kz, avxy, avz, agxy, agz);
        const float avx = avxy.x, avy = avxy.y;
        if (q == 0) {
            moved = step32_commit(K, s, avxy, avz, agxy, agz);
            cvxy = avxy; cvz = avz;
            if (n_rays > 1) {
                // norms through MUFU.RSQ (2 ulp): S is held to 1e-4, and the reference's +1e-32 / +1e-30
                // guards only matter for a ray that did not move, whose S is NaN either way
                const float dx = K.c6r * avx, dy = K.c6r * avy, dz2 = K.c6r * avz;
                const float d2 = fmaf(dx, dx, fmaf(dy, dy, dz2 * dz2));
                const float inv = rsqrtf(d2);
                const float nrd = d2 * inv;
                tx = dx * inv; ty = dy * inv; tz = dz2 * inv;
                // reference axis: z if |t_z| < 0.9 else y (build_rays.py:188-194); e1 = a x t, e2 = t x e1
                const bool use_z = fabsf(tz) < 0.9f;
                float e1x = use_z ? -ty : tz, e1y = use_z ? tx : 0.0f, e1z = use_z ? 0.0f : -tx;
                const float n1 = rsqrtf(fmaf(e1x, e1x, fmaf(e1y, e1y, e1z * e1z)));
                e1x *= n1; e1y *= n1; e1z *= n1;
                e2x = ty * e1z - tz * e1y; e2y = tz * e1x - tx * e1z; e2z = tx * e1y - ty * e1x;
                const float n2 = rsqrtf(fmaf(e2x, e2x, fmaf(e2y, e2y, e2z * e2z)));
                e2x *= n2; e2y *= n2; e2z *= n2;
                eps = K.perturb * nrd;
                oxy = make_float2(eps * e1x, eps * e1y); oz = eps * e1z;
            }
        } else {
            const float ddx = fmaf(K.c6r, avx - cvxy.x, oxy.x), ddy = fmaf(K.c6r, avy - cvxy.y, oxy.y),
                        ddz = fmaf(K.c6r, avz - cvz, oz);
            if (q == 1) {
                d1x = ddx; d1y = ddy; d1z = ddz;
                oxy = make_float2(eps * e2x, eps * e2y); oz = eps * e2z;
            } else {
                const float cx = d1y * ddz - d1z * ddy, cy = d1z * ddx - d1x * ddz, cz = d1x * ddy - d1y * ddx;
                s_step = __fdividef(fabsf(fmaf(cx, tx, fmaf(cy, ty, cz * tz))), eps * eps);
            }
        }
    }
    return moved;
}

// step32 without the pencil: the central ray's step, for the steps whose cross-section ratio is never observed.
// The same operations as step32's central ray, so the master state is bit-identical (that ray starts at offset
// 0 * 1/dx = +0 cells there, the literal zero here).
__device__ __forceinline__ bool step32_central(const RayCube &C, const StepConst &K, Cell &cache, State &s)
{
    bool edge;
    float2 pxy, kxy;
    float pz, kz;
    if (!step32_begin(C, K, cache, s, edge, pxy, pz, kxy, kz)) return false;
    float2 avxy, agxy;
    float avz, agz;
    rk4_stages32(C, K, cache, edge, pxy, pz, make_float2(0.0f, 0.0f), 0.0f, kxy, kz, avxy, avz, agxy, agz);
    return step32_commit(K, s, avxy, avz, agxy, agz);
}

}  // namespace rtgrff
