// FP32 evaluation of one voxel's magneto-ionic slab for the per-ray kernels (fused map, emission on
// samples): refractive indices, free-free opacities, Kirchhoff sources and e^-tau of both modes from the
// float32 sampler outputs, ~100 FP32 instructions and 9 MUFU where the FP64 twin (grff.cuh voxel_op)
// spends ~450 instructions in software FP64 divide / sqrt / expm1 chains (r1 profile: sm_100_rt.hpp
// 10.6 % of the executed instructions and 20 % of the stall samples of render_map_kernel).
//
// Same formulas as voxel_op (DESIGN.md §5; oracle: oracle/oracle_grff.c mode_eval), reorganised so that
// nothing cancels in float32 away from the mode cut-offs:
//   su = nu_B/nu, u = su^2, v = (nu_p/nu)^2, w = 1 - v evaluated with a compensated product (relative
//   accuracy 1e-7 even where v -> 1), A = su sin^2(theta), q = sqrt(A^2 + 4 w^2 cos^2(theta)) [= sqrt(D)/su],
//   t = q - A = 4 w^2 cos^2 / (q + A),
//   d_O = 2w + su t, d_X = 2w - su (q + A), n_s^2 = 1 - 2 v w / d_s,
//   F_X = 2 (su A + 2 w^2 + su A^2 / q) / d_X^2,  F_O = 2 (su A t / q + 2 w^2) / d_O^2.
// Where a mode is close to its cut-off (n^2 < kGuard, or w < kGuard) or the X mode close to the
// gyro-resonance (d_X < 0.05 of its terms) float32 rounding is amplified beyond 1e-5 — there the caller
// falls back to the FP64 path (`ok = false`), as it does for anything non-finite.  The intensities are
// accumulated in FP64.
//
// Everything is __host__ __device__ so that tests/test_grff_fast_cpu.py can run the very same source on the
// CPU against a float64 numpy restatement (no GPU needed to pin the arithmetic).
#pragma once

#include <math.h>

#ifdef __CUDA_ARCH__
// one MUFU each (1-2 ulp): the IEEE-rounded library forms cost 4-8 instructions more per call
__device__ __forceinline__ float rtf_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rtf_sqrt(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rtf_rsqrt(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rtf_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rtf_ln(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r * 0.69314718055994531f; }
#define RTF_RCP(x) rtf_rcp(x)
#define RTF_SQRT(x) rtf_sqrt(x)
#define RTF_RSQRT(x) rtf_rsqrt(x)
#define RTF_EX2(x) rtf_ex2(x)
#define RTF_LN(x) rtf_ln(x)
#else
#define RTF_RCP(x) (1.0f / (x))
#define RTF_SQRT(x) sqrtf(x)
#define RTF_RSQRT(x) (1.0f / sqrtf(x))
#define RTF_EX2(x) exp2f(x)
#define RTF_LN(x) logf(x)
#endif

#ifndef RTF_HD
#ifdef __CUDACC__
#define RTF_HD __host__ __device__ __forceinline__
#else
#define RTF_HD static inline
#endif
#endif

namespace rtgrff {

// Per-frequency float32 constants of the fast path (prepared on the host in double).
struct FreqCF {
    float c_su;            // kNuB / nu:              su = c_su * B
    float cv_hi, cv_lo;    // kNup2 / nu^2 split:     v = (cv_hi + cv_lo) * ne
    float lnl_cold;        // 18.2   - ln(nu):        ln Lambda = 1.5 ln T + lnl_cold   (T < 2e5 K)
    float lnl_hot;         // 24.573 - ln(nu):        ln Lambda =     ln T + lnl_hot
    float kff;             // kKff * kZeta / nu^2
    float srcc;            // nu^2 * k_B / c^2
};

constexpr float kFastGuard = 0.02f;

struct FastOp {
    float aL, aR, bL, bR;
    bool ok;               // false: ill-conditioned or non-finite -> evaluate this voxel in FP64
    float tauL, tauR;      // optical depth kappa dz of the slot (+inf: evanescent); read by the map diagnostics
                           // only, dead code for every other caller
};

// 1 - e^-tau and e^-tau of a slab
RTF_HD void slab_f32(float tau, float src, float &a, float &b)
{
    float em;
    if (tau < 0.125f) {
        // truncation tau^6/5040 relative: < 8e-10
        em = tau * (1.0f - tau * (0.5f - tau * (1.0f / 6.0f - tau * (1.0f / 24.0f - tau * (1.0f / 120.0f - tau * (1.0f / 720.0f))))));
        a = 1.0f - em;
    } else {
        a = RTF_EX2(-1.4426950408889634f * tau);
        em = 1.0f - a;
    }
    b = src * em;
}

// One voxel, both modes.  Inputs as the sampler delivers them (float32); `ok_in` = the voxel passed the
// emptiness tests (dz > 0, T > 0, ne > 0, B >= 0, all finite, |cth| <= 1).
RTF_HD FastOp voxel_op_f32(const FreqCF &f, float dz, float T, float ne, float B, float cth, float sth, float scale,
                           bool ff_on)
{
    FastOp o;
    o.aL = o.aR = 1.0f; o.bL = o.bR = 0.0f; o.ok = true; o.tauL = o.tauR = 0.0f;
    // v and w = 1 - v: the product error of cv_hi * ne is recovered exactly with an FMA, 1 - v_hi is exact
    // for v_hi in [0.5, 2]
    const float v = f.cv_hi * ne;
    const float v_lo = fmaf(f.cv_lo, ne, fmaf(f.cv_hi, ne, -v));
    const float w = (1.0f - v) - v_lo;
    if (!(w >= kFastGuard)) {
        // near or beyond the plasma cut-off: beyond it (w <= 0, B = 0) both modes are evanescent, which is
        // cheap to say here; anything else goes to FP64
        o.ok = false;
        return o;
    }
    float pref = 0.0f;
    if (ff_on) {
        const float lnT = RTF_LN(T);
        const float lnL = (T < 2e5f) ? fmaf(1.5f, lnT, f.lnl_cold) : lnT + f.lnl_hot;
        const float rs = RTF_RSQRT(T);
        pref = (f.kff * ne) * (ne * lnL) * (rs * rs * rs);
    }
    const float srcb = f.srcc * T * scale;
    float aX = 0.0f, bX = 0.0f, aO = 0.0f, bO = 0.0f;
    float tX = INFINITY, tO = INFINITY;
    if (B > 0.0f) {
        const float su = f.c_su * B, u = su * su;
        const float s2 = sth * sth, c2 = cth * cth;
        const float A = su * s2;
        const float w2 = w * w;
        const float fourw2c2 = 4.0f * w2 * c2;
        const float q = RTF_SQRT(fmaf(A, A, fourw2c2));
        const float qa = q + A;
        // one reciprocal for 1/q and 1/(q + A)
        const float r1 = RTF_RCP(q * qa);
        const float inv_q = r1 * qa, inv_qa = r1 * q;
        const float t = fourw2c2 * inv_qa;               // = q - A, no cancellation
        const float dO = fmaf(su, t, 2.0f * w);
        const float dX = fmaf(-su, qa, 2.0f * w);
        const bool x_on = !(u >= 1.0f || u >= w2);       // X cut-off: nu <= nu_B or v >= 1 - sqrt(u)
        // one reciprocal for 1/dX and 1/dO (dO > 0 here; a cut-off X mode lends 1)
        const float dXs = x_on ? dX : 1.0f;
        const float r2 = RTF_RCP(dXs * dO);
        const float inv_dX = r2 * dO, inv_dO = r2 * dXs;
        const float vo2 = 2.0f * v * w + 2.0f * v_lo * w;
        const float suA = su * A, twow2 = 2.0f * w2;
        const float n2O = fmaf(-vo2, inv_dO, 1.0f);
        const float FO = 2.0f * fmaf(suA * t, inv_q, twow2) * inv_dO * inv_dO;
        if (!(n2O >= kFastGuard) || !(FO < INFINITY)) { o.ok = false; return o; }
        {
            float kap = pref * FO * RTF_RSQRT(n2O);
            if (!(kap > 0.0f) || !(kap < INFINITY)) kap = 0.0f;
            tO = kap * dz;
            slab_f32(tO, n2O * srcb, aO, bO);
        }
        if (x_on) {
            // towards the gyro-resonance (nu -> nu_B) d_X = 2w - su (q + A) is a small difference of O(1) terms and
            // the X-mode opacity ~ 1/d_X^2 inherits its relative error
            if (!(dX >= 0.1f * w)) { o.ok = false; return o; }
            const float n2X = fmaf(-vo2, inv_dX, 1.0f);
            const float FX = 2.0f * (fmaf(suA * A, inv_q, suA) + twow2) * inv_dX * inv_dX;
            if (!(n2X >= kFastGuard) || !(FX < INFINITY)) { o.ok = false; return o; }
            float kap = pref * FX * RTF_RSQRT(n2X);
            if (!(kap > 0.0f) || !(kap < INFINITY)) kap = 0.0f;
            tX = kap * dz;
            slab_f32(tX, n2X * srcb, aX, bX);
        }
    } else {
        // B = 0: one refractive index n^2 = w, unpolarised
        float kap = pref * RTF_RSQRT(w);
        if (!(kap > 0.0f) || !(kap < INFINITY)) kap = 0.0f;
        tX = kap * dz;
        slab_f32(tX, w * srcb, aX, bX);
        aO = aX; bO = bX; tO = tX;
    }
    // X is R where cos(theta) >= 0
    if (cth >= 0.0f) { o.aL = aO; o.aR = aX; o.bL = bO; o.bR = bX; o.tauL = tO; o.tauR = tX; }
    else { o.aL = aX; o.aR = aO; o.bL = bX; o.bR = bO; o.tauL = tX; o.tauR = tO; }
    o.ok = (o.bL == o.bL) && (o.bR == o.bR) && (o.aL == o.aL) && (o.aR == o.aR);
    return o;
}

}  // namespace rtgrff
