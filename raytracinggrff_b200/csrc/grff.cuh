// GRFF-style emission/transfer for sm_100a: free-free + gyroresonance emissivity/absorption per
// magneto-ionic mode and the transfer equation along one line of sight, FP64.
//
// Replaces the external GRFF_DEM_Transfer.so::PyGET_MW the reference binds at
// script/resample_with_ray_tracing.py:79-86 and calls per pixel at :502-509 (and
// script/synthetic_FF_map_single_thread.py:208), and fastGRFF.get_mw_slice (:443-446).  The
// source of either is NOT in the reference tree; the physics here follows the published
// formulation (Fleishman, Kuznetsov & Landi 2021; Fleishman & Kuznetsov 2010 App. A; Dulk 1985)
// as specified in DESIGN.md §GRFF — parity for this stage is against oracle/oracle_grff.c and
// analytic limits ("parity unpinned" against the real binary).
//
// Three consumers share the device functions: the warp-per-(pixel,frequency) kernel behind the
// PyGET_MW / get_mw_slice ABIs (lanes over voxels, warp-shuffle composition of the per-voxel
// affine maps), the thread-per-ray kernel on sampler output, and the fused map kernel.
#pragma once

#include "common.cuh"
#include "grff_fast.cuh"

namespace rtgrff {

constexpr double kPi = 3.14159265358979323846;
constexpr double kKff = 9.76981314722991795e-03;      // 8 e^6 / (3 sqrt(2 pi) c (m k)^1.5)
constexpr double kCqt = 1.45534837532918656e+17;      // e^5 / (32 pi^2 m^4 c^4)
constexpr double kNup2 = 8.06163860001142621e+07;     // e^2 / (pi m):  nu_p^2 = kNup2 n_e
constexpr double kNuB = 2.79924898723330395e+06;      // e / (2 pi m c): nu_B = kNuB B
constexpr double kBres = 3.57238675287821001e-07;     // 2 pi m c / e:  B_res = kBres nu / s
constexpr double kGrPref = 2.65400885457447444e-02;   // pi e^2 / (m c)
constexpr double kKbC2 = 1.53617918724037216e-37;     // k_B / c^2
constexpr double kBeta2 = 1.68637005266055143e-10;    // k_B / (m c^2)
constexpr double kZeta = 1.14529914529914545e+00;     // sum Z^2 n_i / n_e, H + He (He/H = 0.085)
constexpr double kAu = 1.495978707e13;
constexpr double kSfu = 1e-19;

struct Voxel {
    double dz, T, ne, B, cth, sth;   // theta enters through its cosine and sine only
    double scale;                    // source-term factor of the S input (Parms[14] / area), 1 by default
    int smax;
    bool gr_on, ff_on, ok;
};

struct Mode {
    double n2, kap, src;
    bool prop;
};

// I' = a I + b on the L and R slots.
struct DiagOp {
    double aL, aR, bL, bR;
};

__device__ __forceinline__ DiagOp diag_identity() { return DiagOp{1.0, 1.0, 0.0, 0.0}; }

// second o first
__device__ __forceinline__ DiagOp diag_then(const DiagOp &first, const DiagOp &second)
{
    return DiagOp{first.aL * second.aL, first.aR * second.aR, fma(first.bL, second.aL, second.bL),
                  fma(first.bR, second.aR, second.bR)};
}

__device__ __forceinline__ Voxel make_voxel_cs(double dz, double T, double ne, double B, double cth, double sth,
                                               int flag, int smax)
{
    Voxel v;
    v.dz = dz; v.T = T; v.ne = ne; v.B = B;
    v.cth = cth; v.sth = sth;
    v.scale = 1.0;
    v.smax = smax;
    v.gr_on = !(flag & 1);
    v.ff_on = !(flag & 2);
    v.ok = (dz > 0.0) && (T > 0.0) && (ne > 0.0) && (B >= 0.0) && isfinite(dz) && isfinite(T) &&
           isfinite(ne) && isfinite(B) && isfinite(cth);
    return v;
}

// The same voxel from the float32 sampler outputs: the range tests run on the floats (a compare pair
// each instead of FP64 classification), which is what the doubles are converted from.
__device__ __forceinline__ Voxel make_voxel_f(float dz, float T, float ne, float B, double cth, double sth, int flag,
                                              int smax)
{
    Voxel v;
    v.dz = (double)dz; v.T = (double)T; v.ne = (double)ne; v.B = (double)B;
    v.cth = cth; v.sth = sth;
    v.scale = 1.0;
    v.smax = smax;
    v.gr_on = !(flag & 1);
    v.ff_on = !(flag & 2);
    v.ok = (dz > 0.0f) & (dz < INFINITY) & (T > 0.0f) & (T < INFINITY) & (ne > 0.0f) & (ne < INFINITY) & (B >= 0.0f) &
           (B < INFINITY) & (fabs(cth) <= 1.0);
    return v;
}

__device__ __forceinline__ Voxel make_voxel(double dz, double T, double ne, double B, double th_deg,
                                            int flag, int smax)
{
    // theta = 90 deg is what every reference call site passes (script/...:495): skip the sincos;
    // the constants are sin/cos of the double nearest to pi/2
    double sth = 1.0, cth = 6.123233995736766e-17;
    if (th_deg != 90.0) sincos(th_deg * (kPi / 180.0), &sth, &cth);
    return make_voxel_cs(dz, T, ne, B, cth, sth, flag, smax);
}

// Refractive index, free-free opacity and Kirchhoff source of mode sg (-1 X, +1 O).
template <bool WANT_POL>
__device__ __forceinline__ Mode mode_eval(double nu, double ne, double B, double T, double cth, double sth,
                                          int sg, bool ff_on, double &Tpol, double &Lpol)
{
    Mode m;
    m.prop = false; m.kap = 0.0; m.src = 0.0; m.n2 = 0.0;
    Tpol = 0.0; Lpol = 0.0;
    const double nuB = kNuB * B;
    const double u = (nuB / nu) * (nuB / nu), v = kNup2 * ne / (nu * nu);
    const double s2 = sth * sth, c2 = cth * cth;
    double F = 1.0, n2;
    if (u > 0.0) {
        if (sg < 0 && (u >= 1.0 || v >= 1.0 - sqrt(u))) return m;   // X cutoff / nu <= nu_B
        if (sg > 0 && v >= 1.0) return m;                            // O cutoff
        const double omv = 1.0 - v;
        const double D = u * u * s2 * s2 + 4.0 * u * omv * omv * c2;
        const double sD = sg * sqrt(D);
        const double den = 2.0 * omv - u * s2 + sD;
        n2 = 1.0 - 2.0 * v * omv / den;
        F = 2.0 * (sD * (u * s2 + 2.0 * omv * omv) - u * u * s2 * s2) / (sD * den * den);
        if (WANT_POL) {
            const double su = sqrt(u);
            Tpol = 2.0 * su * omv * cth / (u * s2 - sD);
            Lpol = (v * su * sth + Tpol * u * v * sth * cth) / (1.0 - u - v + u * v * c2);
        }
    } else {
        if (v >= 1.0) return m;
        n2 = 1.0 - v;
    }
    if (!(n2 > 0.0) || !isfinite(n2) || !isfinite(F)) return m;
    m.prop = true;
    m.n2 = n2;
    m.src = n2 * nu * nu * kKbC2 * T;
    if (ff_on && ne > 0.0) {
        const double lnL = (T < 2e5) ? 18.2 + 1.5 * log(T) - log(nu) : 24.573 + log(T / nu);
        double kap = kKff * ne * ne * kZeta * lnL * F / (sqrt(n2) * nu * nu * T * sqrt(T));
        if (!(kap > 0.0) || !isfinite(kap)) kap = 0.0;
        m.kap = kap;
    }
    return m;
}

// slab of optical depth tau and source src as an affine map; evanescent -> I = 0.
__device__ __forceinline__ void slab_ab(bool prop, double tau, double src, double &a, double &b)
{
    if (!prop) { a = 0.0; b = 0.0; return; }
    if (tau > 0.0) {
        // 1 - e^-tau: four Taylor terms below 2e-3 (truncation < tau^5/120 = 3e-16), expm1 above
        const double em = (tau < 2e-3) ? tau * (1.0 - tau * (0.5 - tau * (1.0 / 6.0 - tau * (1.0 / 24.0))))
                                       : -expm1(-tau);
        a = 1.0 - em; b = src * em;
    } else {
        a = 1.0; b = 0.0;
    }
}

// Per-frequency constants hoisted out of the voxel loop.
struct FreqC {
    double nu, nu2, inv_nu2, ln_nu;
    double sn;    // kBres * nu: resonant field of harmonic s is sn / s
    double kff;   // kKff * kZeta / nu^2: free-free opacity prefactor
    float snf;    // sn rounded up to float32 (conservative side of between_needed_f)
    FreqCF ff;    // float32 constants of the fast voxel evaluation (grff_fast.cuh)
};

__host__ __device__ __forceinline__ FreqC make_freq(double nu)
{
    FreqC f;
    f.nu = nu; f.nu2 = nu * nu; f.inv_nu2 = 1.0 / f.nu2; f.ln_nu = log(nu);
    f.sn = kBres * nu;
    f.kff = kKff * kZeta * f.inv_nu2;
    f.snf = (float)(f.sn * (1.0 - 1e-6));
    const double cv = kNup2 * f.inv_nu2;
    f.ff.c_su = (float)(kNuB / nu);
    f.ff.cv_hi = (float)cv;
    f.ff.cv_lo = (float)(cv - (double)f.ff.cv_hi);
    f.ff.lnl_cold = (float)(18.2 - f.ln_nu);
    f.ff.lnl_hot = (float)(24.573 - f.ln_nu);
    f.ff.kff = (float)f.kff;
    f.ff.srcc = (float)(f.nu2 * kKbC2);
    return f;
}

// Uniform slab of one voxel: both magneto-ionic modes at once (same formulas as mode_eval; the
// quantities common to the two modes — u, v, D, the Coulomb logarithm, the opacity prefactor —
// are evaluated once).
// FAST_T (the per-ray kernels, tolerance 1e-4 on T_b): ln T and T^-1.5 in FP32.  The kernel behind the
// PyGET_MW / get_mw_slice ABIs keeps them FP64 (agrees with the oracle to 1e-14).
// TAU: also write the optical depth kappa dz of the L and R slot to tau[0], tau[1] (+inf where the mode is
// evanescent), for the map diagnostics; the TAU = false instantiation is the plain evaluation.
template <bool FAST_T, bool TAU = false>
__device__ __forceinline__ DiagOp voxel_op(const FreqC &f, const Voxel &v, double *tau = nullptr)
{
    const double nuB = kNuB * v.B;
    const double u = nuB * nuB * f.inv_nu2, vv = kNup2 * v.ne * f.inv_nu2;
    const double omv = 1.0 - vv;
    double pref = 0.0;
    if (v.ff_on) {
        if (FAST_T) {
            // T comes from a float32 cube: its logarithm and T^-1.5 in FP32 (1e-7 relative, unbiased) save
            // an FP64 log, sqrt and divide per voxel; everything the cut-offs depend on stays FP64
            const float Tf = (float)v.T;
            const double lnT = (double)__logf(Tf);   // MUFU.LG2: |error| < 4e-7 on ln T ~ 14
            const double lnL = (v.T < 2e5) ? 18.2 + 1.5 * lnT - f.ln_nu : 24.573 + lnT - f.ln_nu;
            const float rs = rsqrtf(Tf);
            pref = f.kff * (v.ne * v.ne) * lnL * (double)(rs * rs * rs);
        } else {
            const double lnT = log(v.T);
            const double lnL = (v.T < 2e5) ? 18.2 + 1.5 * lnT - f.ln_nu : 24.573 + lnT - f.ln_nu;
            pref = kKff * v.ne * v.ne * kZeta * lnL * f.inv_nu2 / (v.T * sqrt(v.T));
        }
    }
    const double srcb = f.nu2 * kKbC2 * v.T * v.scale;
    double aX = 0.0, bX = 0.0, aO = 0.0, bO = 0.0;
    double tX = INFINITY, tO = INFINITY;
    if (u > 0.0) {
        const double s2 = v.sth * v.sth, c2 = v.cth * v.cth;
        const double us2 = u * s2;
        const double sD = sqrt(us2 * us2 + 4.0 * u * omv * omv * c2);
        const double num0 = us2 + 2.0 * omv * omv, base = 2.0 * omv - us2;
        const double us4 = us2 * us2, vo2 = 2.0 * vv * omv;
        // n^2 = 1 - 2 v (1-v)/den,  F = 2 (num0 -+ us2^2/sD) / den^2  with den = base -+ sD.
        // X mode (sigma = -1) is cut off for nu <= nu_B or v >= 1 - sqrt(u); below v = 1 that is
        // sqrt(u) >= 1 - v  <=>  u >= (1-v)^2: no square root needed.  O mode (sigma = +1): v >= 1.
        const bool x_on = !(u >= 1.0 || vv >= 1.0 || u >= omv * omv), o_on = vv < 1.0;
        const double dX = base - sD, dO = base + sD;
        double inv_sD, inv_dX, inv_dO;
        if (FAST_T) {
            // one reciprocal of the product instead of three reciprocals (a mode that is cut off lends 1)
            const double a = x_on ? dX : 1.0, b = o_on ? dO : 1.0;
            const double ab = a * b, r = 1.0 / (ab * sD);
            inv_sD = r * ab; inv_dX = r * (b * sD); inv_dO = r * (a * sD);
        } else {
            inv_sD = 1.0 / sD;
            inv_dX = x_on ? 1.0 / dX : 0.0;
            inv_dO = o_on ? 1.0 / dO : 0.0;
        }
        if (x_on) {
            const double n2 = 1.0 - vo2 * inv_dX;
            const double F = 2.0 * (num0 + us4 * inv_sD) * inv_dX * inv_dX;
            if (n2 > 0.0 && isfinite(n2) && isfinite(F)) {
                double kap = pref * F * rsqrt(n2);
                if (!(kap > 0.0) || !isfinite(kap)) kap = 0.0;
                if constexpr (TAU) tX = kap * v.dz;
                slab_ab(true, kap * v.dz, n2 * srcb, aX, bX);
            }
        }
        if (o_on) {
            const double n2 = 1.0 - vo2 * inv_dO;
            const double F = 2.0 * (num0 - us4 * inv_sD) * inv_dO * inv_dO;
            if (n2 > 0.0 && isfinite(n2) && isfinite(F)) {
                double kap = pref * F * rsqrt(n2);
                if (!(kap > 0.0) || !isfinite(kap)) kap = 0.0;
                if constexpr (TAU) tO = kap * v.dz;
                slab_ab(true, kap * v.dz, n2 * srcb, aO, bO);
            }
        }
    } else if (vv < 1.0) {
        // B = 0: one refractive index, unpolarised
        double kap = pref * rsqrt(omv);
        if (!(kap > 0.0) || !isfinite(kap)) kap = 0.0;
        if constexpr (TAU) tX = tO = kap * v.dz;
        slab_ab(true, kap * v.dz, omv * srcb, aX, bX);
        aO = aX; bO = bX;
    }
    if constexpr (TAU) {
        tau[0] = (v.cth >= 0.0) ? tO : tX;
        tau[1] = (v.cth >= 0.0) ? tX : tO;
    }
    // X is R where cos(theta) >= 0
    return (v.cth >= 0.0) ? DiagOp{aO, aX, bO, bX} : DiagOp{aX, aO, bX, bO};
}

// The per-ray kernels' voxel evaluation: float32 where it is well conditioned (grff_fast.cuh), the FP64
// voxel_op otherwise (near the mode cut-offs and the gyro-resonance, anything non-finite).  Inputs are the
// float32 sampler outputs; the emptiness tests are those of make_voxel_f.
__device__ __forceinline__ bool voxel_nonempty_f(float dz, float T, float ne, float B, float cth)
{
    return (dz > 0.0f) & (dz < INFINITY) & (T > 0.0f) & (T < INFINITY) & (ne > 0.0f) & (ne < INFINITY) & (B >= 0.0f) &
           (B < INFINITY) & (fabsf(cth) <= 1.0f);
}

// the FP64 fallback, out of line: it runs for the few voxels near a cut-off, and inlined it would put its
// ~60 live FP64 values into the register budget of the callers' hot loops
// (the four per-frequency numbers it needs travel by value: a reference into the kernel parameters would
// make the compiler copy the whole parameter block to local memory)
__device__ __noinline__ DiagOp voxel_op_slow(double nu2, double inv_nu2, double ln_nu, double kff, float dz, float T, float ne,
                                             float B, float cth, float sth, float scale, int flag, int smax)
{
    FreqC f;
    f.nu2 = nu2; f.inv_nu2 = inv_nu2; f.ln_nu = ln_nu; f.kff = kff;
    Voxel v = make_voxel_f(dz, T, ne, B, (double)cth, (double)sth, flag, smax);
    v.scale = (double)scale;
    return voxel_op<true>(f, v);
}

__device__ __forceinline__ DiagOp voxel_op_mixed(const FreqC &f, float dz, float T, float ne, float B, float cth, float sth,
                                                 float scale, int flag, int smax, bool force64)
{
    if (!force64) {
        const FastOp o = voxel_op_f32(f.ff, dz, T, ne, B, cth, sth, scale, !(flag & 2));
        if (o.ok) return DiagOp{(double)o.aL, (double)o.aR, (double)o.bL, (double)o.bR};
    }
    return voxel_op_slow(f.nu2, f.inv_nu2, f.ln_nu, f.kff, dz, T, ne, B, cth, sth, scale, flag, smax);
}

// An operator with the optical depth kappa dz it applies to the L and R slot (+inf: evanescent mode): what the
// map diagnostics need of each voxel and gyroresonance layer.  Returned by value from the out-of-line
// evaluations, so that the hot loop keeps it in registers.
struct TauOp {
    DiagOp op;
    double tauL, tauR;
};

// The slots' optical depths of voxel_op_slow's evaluation.  A function of its own, next to voxel_op_slow rather
// than folded into a copy of it: the diagnostic kernels take the operator from the very code the plain kernels
// run, so their T_b stays the plain T_b bit for bit.
__device__ __noinline__ double2 voxel_tau_slow(double nu2, double inv_nu2, double ln_nu, double kff, float dz, float T,
                                               float ne, float B, float cth, float sth, float scale, int flag, int smax)
{
    FreqC f;
    f.nu2 = nu2; f.inv_nu2 = inv_nu2; f.ln_nu = ln_nu; f.kff = kff;
    Voxel v = make_voxel_f(dz, T, ne, B, (double)cth, (double)sth, flag, smax);
    v.scale = (double)scale;
    double t[2];
    voxel_op<true, true>(f, v, t);
    return make_double2(t[0], t[1]);
}

// voxel_op_mixed with the optical depths, taken from whichever evaluation produced the operator (never as
// -log a: in float32 a thin voxel's a rounds to 1)
__device__ __forceinline__ TauOp voxel_op_mixed_tau(const FreqC &f, float dz, float T, float ne, float B, float cth,
                                                    float sth, float scale, int flag, int smax, bool force64)
{
    if (!force64) {
        const FastOp o = voxel_op_f32(f.ff, dz, T, ne, B, cth, sth, scale, !(flag & 2));
        if (o.ok) return TauOp{DiagOp{(double)o.aL, (double)o.aR, (double)o.bL, (double)o.bR}, (double)o.tauL, (double)o.tauR};
    }
    const DiagOp op = voxel_op_slow(f.nu2, f.inv_nu2, f.ln_nu, f.kff, dz, T, ne, B, cth, sth, scale, flag, smax);
    const double2 t = voxel_tau_slow(f.nu2, f.inv_nu2, f.ln_nu, f.kff, dz, T, ne, B, cth, sth, scale, flag, smax);
    return TauOp{op, t.x, t.y};
}

// One gyroresonance layer nu = s nu_B at interpolated plasma parameters.  Rare and heavy (lgamma,
// log, exp, sincos): kept out of line (gr_layer_op, gr_layer_op_tau) so the hot loops stay small.
// TAU: tau[0], tau[1] receive the layer's optical depth on the L and R slot (+inf: evanescent mode).
template <bool TAU>
__device__ __forceinline__ DiagOp gr_layer_eval(double nu, int s, double ne, double T, double th, double LB, double scale,
                                                double *tau)
{
    double sth, cth;
    sincos(th, &sth, &cth);
    const double Bres = kBres * nu / (double)s;
    double a[2], b[2], t[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int sg = q == 0 ? -1 : 1;
        double Ts, Ls;
        const Mode m = mode_eval<true>(nu, ne, Bres, T, cth, sth, sg, false, Ts, Ls);
        double tau = 0.0;
        if (m.prop) {
            const double lg = 2.0 * s * log((double)s) - (s - 1) * 0.69314718055994530942 - lgamma(s + 1.0) +
                              (s - 1) * log(kBeta2 * T * sth * sth) + (s - 1.5) * log(m.n2);
            const double pol = Ts * cth + Ls * sth + 1.0;
            tau = kGrPref * ne * LB / nu * exp(lg) * pol * pol / (1.0 + Ts * Ts);
            if (!(tau > 0.0) || !isfinite(tau)) tau = 0.0;
        }
        if constexpr (TAU) t[q] = m.prop ? tau : INFINITY;
        slab_ab(m.prop, tau, m.src * scale, a[q], b[q]);
    }
    if constexpr (TAU) {
        tau[0] = (cth >= 0.0) ? t[1] : t[0];
        tau[1] = (cth >= 0.0) ? t[0] : t[1];
    }
    return (cth >= 0.0) ? DiagOp{a[1], a[0], b[1], b[0]} : DiagOp{a[0], a[1], b[0], b[1]};
}

__device__ __noinline__ DiagOp gr_layer_op(double nu, int s, double ne, double T, double th, double LB, double scale)
{
    return gr_layer_eval<false>(nu, s, ne, T, th, LB, scale, nullptr);
}

__device__ __noinline__ TauOp gr_layer_op_tau(double nu, int s, double ne, double T, double th, double LB, double scale)
{
    TauOp r;
    double t[2];
    r.op = gr_layer_eval<true>(nu, s, ne, T, th, LB, scale, t);
    r.tauL = t[0]; r.tauR = t[1];
    return r;
}

// Everything that happens between the centres of two consecutive non-empty voxels p -> k:
// gyroresonance layers (diagonal in L/R) before and after an optional quasi-transverse layer.
struct Between {
    DiagOp before, after;
    double Q;     // exact-coupling transmission exp(-delta)
    bool qt;
};

// Cheap test for "something happens between p and k" (a quasi-transverse layer or a gyroresonance
// layer): the per-ray kernels call between_voxels only then.  Same conditions as its early exit.
__device__ __forceinline__ bool between_needed(const FreqC &f, const Voxel &p, const Voxel &k)
{
    const bool qt = (p.cth * k.cth < 0.0);
    const double smax = (double)min(p.smax, k.smax);
    const bool gr = p.gr_on && k.gr_on && (p.B != k.B) && ((p.B * smax > f.sn) || (k.B * smax > f.sn));
    return qt || gr;
}

// The same test on the float32 values the voxels were built from (the per-ray kernels keep the previous
// voxel as six floats); the resonance test leans to the "needed" side by 1e-6, between_voxels decides.
__device__ __forceinline__ bool between_needed_f(const FreqC &f, float p_cth, float p_B, float k_cth, float k_B,
                                                 int smax, bool gr_on)
{
    const bool qt = (p_cth * k_cth < 0.0f);
    const bool gr = gr_on && (p_B != k_B) && (fmaxf(p_B, k_B) * (float)smax > f.snf);
    return qt || gr;
}

// TAU: tau[0], tau[1] accumulate the optical depth of the gyroresonance layers on the L and R slot (a
// quasi-transverse layer adds none); the TAU = false instantiation is the plain event list.
template <bool TAU = false>
__device__ __forceinline__ Between between_voxels(const FreqC &f, const Voxel &p, const Voxel &k, double *tau = nullptr)
{
    Between o;
    o.before = diag_identity(); o.after = diag_identity(); o.Q = 1.0;
    o.qt = (p.cth * k.cth < 0.0);
    const int smax = min(p.smax, k.smax);
    const double blo = fmin(p.B, k.B), bhi = fmax(p.B, k.B);
    // a layer needs the resonant field of some harmonic s <= smax inside (blo, bhi): sn/smax < bhi
    const bool gr = p.gr_on && k.gr_on && (p.B != k.B) && (bhi * (double)smax > f.sn);
    if (!o.qt && !gr) return o;                      // the common case: nothing happens in between
    const double nu = f.nu;
    const double th_p = acos(p.cth), th_k = acos(k.cth);
    const double dzm = 0.5 * (p.dz + k.dz);
    double tqt = 2.0;
    if (o.qt) {
        tqt = (0.5 * kPi - th_p) / (th_k - th_p);
        const double g = fabs(th_k - th_p) / dzm;
        const double nav = 0.5 * (p.ne + k.ne), Bav = 0.5 * (p.B + k.B);
        o.Q = exp(-kCqt * nav * Bav * Bav * Bav / (nu * nu * nu * nu * g));
    }
    if (gr) {
        const bool up = k.B > p.B;
        // harmonics whose resonant field lies strictly inside (blo, bhi): s in (sn/bhi, sn/blo);
        // the range is taken one wider than that and the sign test below decides.
        const double sn = f.sn;
        const double lo_d = floor(sn / bhi), hi_d = (blo > 0.0) ? ceil(sn / blo) : (double)smax;
        const int s_lo = lo_d > 2.0 ? (lo_d < (double)smax ? (int)lo_d : smax + 1) : 2;
        const int s_hi = hi_d < (double)smax ? (int)hi_d : smax;
        for (int q = s_lo; q <= s_hi; ++q) {
            const int s = up ? (s_hi + s_lo - q) : q;   // path order: B rising -> high harmonics first
            const double Bres = sn / (double)s;
            if (!((p.B - Bres) * (k.B - Bres) < 0.0)) continue;
            const double t = (Bres - p.B) / (k.B - p.B);
            DiagOp g;
            if constexpr (TAU) {
                const TauOp tg = gr_layer_op_tau(nu, s, p.ne + t * (k.ne - p.ne), p.T + t * (k.T - p.T),
                                                 th_p + t * (th_k - th_p), Bres * dzm / fabs(k.B - p.B),
                                                 p.scale + t * (k.scale - p.scale));
                g = tg.op;
                tau[0] += tg.tauL; tau[1] += tg.tauR;
            } else {
                g = gr_layer_op(nu, s, p.ne + t * (k.ne - p.ne), p.T + t * (k.T - p.T),
                                th_p + t * (th_k - th_p), Bres * dzm / fabs(k.B - p.B),
                                p.scale + t * (k.scale - p.scale));
            }
            if (t >= tqt) o.after = diag_then(o.after, g);
            else o.before = diag_then(o.before, g);
        }
    }
    return o;
}

// The float32 voxels of the per-ray kernels (fused map): what the transfer keeps of the previous non-empty voxel.
struct VoxLite {
    float dz, T, ne, B, cth, scale;
};

__device__ __forceinline__ Voxel voxel_of(const VoxLite &l, int flag, int smax)
{
    Voxel v = make_voxel_f(l.dz, l.T, l.ne, l.B, (double)l.cth, sqrt(fmax(0.0, 1.0 - (double)l.cth * (double)l.cth)),
                           flag, smax);
    v.scale = (double)l.scale;
    return v;
}

// between_voxels for the per-ray kernels, OUT OF LINE: it runs on a fraction of a percent of the voxels (behind
// between_needed_f), and inlined its acos / exp / lgamma chains sit in the instruction footprint and the register
// allocation of the hot record loop.  The two per-frequency numbers it needs travel by value (a reference into
// the kernel parameters would make the compiler copy the parameter block to local memory).
__device__ __noinline__ void between_voxels_cold(double nu, double sn, VoxLite p, VoxLite k, int flag, int smax, Between *out)
{
    FreqC f;
    f.nu = nu; f.sn = sn;
    *out = between_voxels(f, voxel_of(p, flag, smax), voxel_of(k, flag, smax));
}

// The optical depth of between_voxels_cold's gyroresonance layers on the L and R slot (the map diagnostics).  The
// diagnostic kernels take the events themselves from between_voxels_cold, the code the plain kernels run.
__device__ __noinline__ double2 between_tau_cold(double nu, double sn, VoxLite p, VoxLite k, int flag, int smax)
{
    FreqC f;
    f.nu = nu; f.sn = sn;
    double t[2] = {0.0, 0.0};
    between_voxels<true>(f, voxel_of(p, flag, smax), voxel_of(k, flag, smax), t);
    return make_double2(t[0], t[1]);
}

// Polarisation state for the three mode-coupling variants GRFF reports:
// {L,R} weak (RL[1],RL[2]), strong (RL[3],RL[4]), exact (RL[5],RL[6]).
template <int NVAR>
struct PolState {
    double L[NVAR], R[NVAR];   // NVAR = 3: weak, strong, exact;  NVAR = 1: exact only
    __device__ __forceinline__ void clear()
    {
#pragma unroll
        for (int q = 0; q < NVAR; ++q) { L[q] = 0.0; R[q] = 0.0; }
    }
    __device__ __forceinline__ void apply(const DiagOp &d)
    {
#pragma unroll
        for (int q = 0; q < NVAR; ++q) { L[q] = fma(L[q], d.aL, d.bL); R[q] = fma(R[q], d.aR, d.bR); }
    }
    __device__ __forceinline__ void qt(double Q)
    {
        const int e = NVAR - 1;
        const double l = L[e], r = R[e];
        L[e] = Q * l + (1.0 - Q) * r;
        R[e] = Q * r + (1.0 - Q) * l;
        if (NVAR == 3) { const double t = L[0]; L[0] = R[0]; R[0] = t; }
    }
    __device__ __forceinline__ void apply(const Between &b)
    {
        apply(b.before);
        if (b.qt) qt(b.Q);
        apply(b.after);
    }
};

// ---------------------------------------------------------------------------------------------
// Kernel A: Parms ABI.  One warp per (pixel, frequency); lanes over voxels in chunks of 32.
// Each lane turns its voxel (and the interval before it) into an affine map, the warp composes
// the 32 maps in path order with shuffles, lane 0 carries the polarisation state.
// Parms (15, Nz) column-major per pixel: element (m,k) at k*15+m  (script/...:489-501).
// ---------------------------------------------------------------------------------------------
struct SliceArgs {
    const double *parms;    // (15, Nz, Npix)
    const double *rparms;   // (3, Npix)
    double *rl;             // (7, Nf, Npix)
    int32_t *status;        // (Npix) or nullptr
    int npix, nz, nf;
};

// Parms[14] > 0 is the S input (script/resample_with_ray_tracing.py:501): the voxel's own source area
// S_k * area; its source term scales by Parms[14] / area (definition in oracle/oracle_grff.c).
__device__ __forceinline__ double load_scale(const double *P, double area)
{
    const double s = P[14];
    return s > 0.0 ? s / area : 1.0;
}

__device__ __forceinline__ Voxel load_voxel(const double *P, double area)
{
    Voxel v = make_voxel(P[0], P[1], P[2], P[3], P[4], (int)P[6], (int)P[7]);
    v.scale = load_scale(P, area);
    return v;
}

__device__ __forceinline__ DiagOp shfl_down_op(const DiagOp &d, int off)
{
    return DiagOp{__shfl_down_sync(0xffffffffu, d.aL, off), __shfl_down_sync(0xffffffffu, d.aR, off),
                  __shfl_down_sync(0xffffffffu, d.bL, off), __shfl_down_sync(0xffffffffu, d.bR, off)};
}

__global__ void __launch_bounds__(128) grff_slice_kernel(const SliceArgs a)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= (int64_t)a.npix * a.nf) return;
    const int pix = (int)(warp / a.nf), f = (int)(warp % a.nf);
    const double *R = a.rparms + (size_t)pix * 3;
    const double nu = R[1] * pow(10.0, R[2] * (double)f);
    const FreqC fq = make_freq(nu);
    const double *P = a.parms + (size_t)pix * 15 * a.nz;
    PolState<3> st;
    st.clear();
    for (int base = 0; base < a.nz; base += 32) {
        const int k = base + lane;
        DiagOp op = diag_identity();
        Between bt;
        bt.qt = false;
        bool has_bt = false;
        if (k < a.nz) {
            const Voxel v = load_voxel(P + (size_t)k * 15, R[0]);
            if (v.ok) {
                if (k > 0) {
                    // the previous voxel without its S input; that (one more scattered load) and the event
                    // list are only needed where something can happen between the two voxels
                    const double *Pp = P + (size_t)(k - 1) * 15;
                    Voxel pv = make_voxel(Pp[0], Pp[1], Pp[2], Pp[3], Pp[4], (int)Pp[6], (int)Pp[7]);
                    if (pv.ok && pv.B > 0.0 && v.B > 0.0 && between_needed(fq, pv, v)) {
                        pv.scale = load_scale(Pp, R[0]);
                        bt = between_voxels(fq, pv, v);
                        has_bt = true;
                    }
                }
                op = voxel_op<false>(fq, v);
            }
        }
        const bool any_qt = __any_sync(0xffffffffu, has_bt && bt.qt);
        if (!any_qt) {
            if (has_bt) op = diag_then(diag_then(bt.before, bt.after), op);
            // ordered composition: after the loop lane 0 holds op_31 o ... o op_0
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const DiagOp nx = shfl_down_op(op, off);
                if (lane + off < 32) op = diag_then(op, nx);
            }
            if (lane == 0) st.apply(op);
        } else {
            // a quasi-transverse layer mixes L and R: replay this chunk in order on lane 0's state
            for (int l = 0; l < 32; ++l) {
                Between b;
                b.before = DiagOp{__shfl_sync(0xffffffffu, bt.before.aL, l), __shfl_sync(0xffffffffu, bt.before.aR, l),
                                  __shfl_sync(0xffffffffu, bt.before.bL, l), __shfl_sync(0xffffffffu, bt.before.bR, l)};
                b.after = DiagOp{__shfl_sync(0xffffffffu, bt.after.aL, l), __shfl_sync(0xffffffffu, bt.after.aR, l),
                                 __shfl_sync(0xffffffffu, bt.after.bL, l), __shfl_sync(0xffffffffu, bt.after.bR, l)};
                b.Q = __shfl_sync(0xffffffffu, bt.Q, l);
                b.qt = __shfl_sync(0xffffffffu, (int)bt.qt, l) != 0;
                const bool hb = __shfl_sync(0xffffffffu, (int)has_bt, l) != 0;
                const DiagOp o = DiagOp{__shfl_sync(0xffffffffu, op.aL, l), __shfl_sync(0xffffffffu, op.aR, l),
                                        __shfl_sync(0xffffffffu, op.bL, l), __shfl_sync(0xffffffffu, op.bR, l)};
                if (lane == 0) {
                    if (hb) st.apply(b);
                    st.apply(o);
                }
            }
        }
    }
    if (lane == 0) {
        double *o = a.rl + ((size_t)pix * a.nf + f) * 7;
        const double to_sfu = R[0] / (kAu * kAu) / kSfu;
        o[0] = nu / 1e9;
        o[1] = st.L[0] * to_sfu; o[2] = st.R[0] * to_sfu;
        o[3] = st.L[1] * to_sfu; o[4] = st.R[1] * to_sfu;
        o[5] = st.L[2] * to_sfu; o[6] = st.R[2] * to_sfu;
        if (a.status && f == 0) a.status[pix] = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// Online transfer used by the thread-per-ray consumers (sampler output, fused map).
// Feeds voxels one at a time in path order; keeps the previous non-empty voxel for the
// between-voxel events.  Mirrors the packing rules of script/resample_with_ray_tracing.py:472-501:
// only samples with valid & finite(ne,te,b) are handed over, theta = 90 deg unless given.
// ---------------------------------------------------------------------------------------------
template <int NVAR>
struct OnlineTransfer {
    PolState<NVAR> st;
    Voxel prev;
    bool have_prev;
    __device__ __forceinline__ void init() { st.clear(); have_prev = false; prev.ok = false; }
    // v holds float32 sampler values widened to double: the slab operator goes through voxel_op_mixed
    __device__ __forceinline__ void push(const FreqC &f, const Voxel &v, bool force64)
    {
        if (!v.ok) { have_prev = false; return; }
        if (have_prev && prev.B > 0.0 && v.B > 0.0) st.apply(between_voxels(f, prev, v));
        st.apply(voxel_op_mixed(f, (float)v.dz, (float)v.T, (float)v.ne, (float)v.B, (float)v.cth, (float)v.sth, (float)v.scale,
                                (v.gr_on ? 0 : 1) | (v.ff_on ? 0 : 2), v.smax, force64));
        prev = v;
        have_prev = true;
    }
};

// T_b and V/I from L,R intensities exactly as the workflow converts GRFF's SFU output
// (script/resample_with_ray_tracing.py:91-94, :513-520, :530): the library-side flux uses kAu/kSfu,
// the workflow-side conversion its own rounded constants.
__device__ __forceinline__ void tb_vi(double IL, double IR, double nu, double area, double &tb, double &vi)
{
    const double to_sfu = area / (kAu * kAu) / kSfu;
    const double l = IL * to_sfu, r = IR * to_sfu;
    const double conv = (1e-19 * 2.998e10 * 2.998e10 / (2.0 * 1.38065e-16 * nu * nu) / area) * (1.49599e13 * 1.49599e13);
    tb = (l + r) * conv;
    vi = (l - r) / (l + r + 1e-30);
    if (!isfinite(tb)) tb = 0.0;   // np.nan_to_num(emission_cube, nan=0, posinf=0, neginf=0)
}

struct EmissionArgs {
    const float *ne, *te, *b, *ds;   // [rec][ray]
    const float *s;                  // [rec][ray] cross-section ratio: the S input when s_input != 0
    int s_input;
    const uint8_t *valid;
    int64_t n_rec, n_rays;
    double area, freq0, log_step;
    int n_freq, em_flag, s_max;
    int grff64;                      // 1: FP64 voxel evaluation throughout (RTGRFF_GRFF64=1)
    double *tb, *vi;                 // (ray, freq)
};

// Thread per (ray, frequency) on sampler output (staged pipeline).
__global__ void __launch_bounds__(128) emission_rays_kernel(const EmissionArgs a)
{
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.n_rays * a.n_freq) return;
    const int64_t ray = q % a.n_rays;
    const int f = (int)(q / a.n_rays);
    const double nu = a.freq0 * pow(10.0, a.log_step * (double)f);
    const FreqC fq = make_freq(nu);
    OnlineTransfer<1> tr;
    tr.init();
    for (int64_t rec = 0; rec < a.n_rec; ++rec) {
        const size_t o = (size_t)rec * a.n_rays + ray;
        if (!a.valid[o]) continue;
        const float ne = a.ne[o], te = a.te[o], b = a.b[o];
        if (!(isfinite(ne) && isfinite(te) && isfinite(b))) continue;
        Voxel v = make_voxel((double)a.ds[o], (double)te, (double)ne, (double)b, 90.0, a.em_flag, a.s_max);
        // Parms[14] = S * area (script/resample_with_ray_tracing.py:501) -> source factor S where S > 0
        if (a.s_input && a.s[o] > 0.0f) v.scale = (double)a.s[o];
        tr.push(fq, v, a.grff64 != 0);
    }
    double tb, vi;
    tb_vi(tr.st.L[0], tr.st.R[0], nu, a.area, tb, vi);
    a.tb[(size_t)ray * a.n_freq + f] = tb;
    a.vi[(size_t)ray * a.n_freq + f] = vi;
}

}  // namespace rtgrff
