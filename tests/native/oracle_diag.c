/*
 * ORACLE — TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of the map diagnostics of rtgrff_render_map_diag (definitions in include/rtgrff.h) on one
 * line of sight: oracle_get_mw's loop (oracle/oracle_grff.c, included below so that the very same functions
 * compute the transfer) with, next to the exact-coupling intensities, four weighted transfers W^c (c = x, y, z, r)
 * and the optical depths of the L and R slot.
 *   W^c:  every slab I <- I e^-tau + S (1 - e^-tau) acts on W as W <- W e^-tau + c S (1 - e^-tau), an evanescent
 *         mode resets W as it resets I, a quasi-transverse layer mixes W_L, W_R with the same Q as I_L, I_R.  c is
 *         the voxel's coordinate; a layer between two voxels (gyroresonance, quasi-transverse) takes the midpoint
 *         of the two voxels' coordinates.  EM_c = (W^c_L + W^c_R) / (I_L + I_R), NaN if that is 0 or not finite.
 *   tau:  kappa dz of every slab plus every gyroresonance layer's tau, routed to L/R like the intensity;
 *         +inf once a mode is evanescent; a quasi-transverse layer adds nothing.
 * RL is written exactly as oracle_get_mw writes it (same operations in the same order).
 */
#include <string.h>

#include "../../oracle/oracle_grff.c"

typedef struct {
    double w[2][4];     /* [L/R][x, y, z, r] of the exact-coupling slots */
    double tau[2];
} diag_t;

/* one mode's slab on the exact slot `to_R` of W, with the same e^-tau as slab() */
static void diag_mode(diag_t *d, int to_R, int prop, double tau, double src, const double *c)
{
    if (!prop) {
        for (int q = 0; q < 4; ++q) d->w[to_R][q] = 0.0;
        d->tau[to_R] = INFINITY;
        return;
    }
    if (tau > 0.0) {
        const double em = -expm1(-tau);
        for (int q = 0; q < 4; ++q) d->w[to_R][q] = d->w[to_R][q] * (1.0 - em) + src * em * c[q];
        d->tau[to_R] += tau;
    }
}

/* qt_layer with W: Q as qt_layer computes it */
static void diag_qt(double *I6, diag_t *d, double nu, const voxel_t *p, const voxel_t *k)
{
    const double dzm = 0.5 * (p->dz + k->dz);
    const double g = fabs(k->th - p->th) / dzm;
    const double nav = 0.5 * (p->ne + k->ne), Bav = 0.5 * (p->B + k->B);
    const double cq = pow(Q_EL, 5) / (32.0 * M_PI * M_PI * pow(M_EL, 4) * pow(C_L, 4));
    const double dd = cq * nav * Bav * Bav * Bav / (nu * nu * nu * nu * g);
    const double Q = exp(-dd);
    qt_layer(I6, nu, p, k);
    for (int q = 0; q < 4; ++q) {
        const double l = d->w[0][q], r = d->w[1][q];
        d->w[0][q] = Q * l + (1.0 - Q) * r;
        d->w[1][q] = Q * r + (1.0 - Q) * l;
    }
}

/* gr_layer with W and tau: the layer's tau and source as gr_layer computes them */
static void diag_gr(double *I6, diag_t *d, double nu, int s, double ne, double T, double th, double LB, double scale,
                    const double *c)
{
    const double cth = cos(th), sth = sin(th);
    const double Bres = nu * 2.0 * M_PI * M_EL * C_L / (s * Q_EL);
    const int x_to_R = cth >= 0.0;
    for (int sg = -1; sg <= 1; sg += 2) {
        mode_t m; double Ts, Ls;
        mode_eval(nu, ne, Bres, T, cth, sth, sg, 0, &m, &Ts, &Ls);
        const int to_R = (sg < 0) ? x_to_R : !x_to_R;
        if (!m.prop) { apply_mode(I6, to_R, 0, 0.0, 0.0); diag_mode(d, to_R, 0, 0.0, 0.0, c); continue; }
        const double beta2 = K_B * T / (M_EL * C_L * C_L);
        const double lg = 2.0 * s * log((double)s) - (s - 1) * log(2.0) - lgamma(s + 1.0) +
                          (s - 1) * log(beta2 * sth * sth) + (s - 1.5) * log(m.n2);
        const double pol = Ts * cth + Ls * sth + 1.0;
        double tau = M_PI * Q_EL * Q_EL * ne * LB / (M_EL * C_L * nu) * exp(lg) * pol * pol / (1.0 + Ts * Ts);
        if (!(tau > 0.0) || !isfinite(tau)) tau = 0.0;
        apply_mode(I6, to_R, 1, tau, m.src * scale);
        diag_mode(d, to_R, 1, tau, m.src * scale, c);
    }
}

/* between() with W and tau, every event at coordinate c (the midpoint of p and k) */
static void diag_between(double *I6, diag_t *d, double nu, const voxel_t *p, const voxel_t *k, const double *c)
{
    const int qt = (p->cth * k->cth < 0.0);
    const double tqt = qt ? (0.5 * M_PI - p->th) / (k->th - p->th) : 2.0;
    int qt_done = !qt;
    if (p->gr_on && k->gr_on && p->B != k->B) {
        const int smax = p->smax < k->smax ? p->smax : k->smax;
        const double dzm = 0.5 * (p->dz + k->dz);
        const int up = k->B > p->B;
        for (int q = 2; q <= smax; ++q) {
            const int s = up ? (smax + 2 - q) : q;
            const double Bres = nu * 2.0 * M_PI * M_EL * C_L / (s * Q_EL);
            if ((p->B - Bres) * (k->B - Bres) >= 0.0) continue;
            const double t = (Bres - p->B) / (k->B - p->B);
            if (!qt_done && t >= tqt) { diag_qt(I6, d, nu, p, k); qt_done = 1; }
            const double ne = p->ne + t * (k->ne - p->ne), T = p->T + t * (k->T - p->T);
            const double th = p->th + t * (k->th - p->th);
            const double LB = Bres * dzm / fabs(k->B - p->B);
            diag_gr(I6, d, nu, s, ne, T, th, LB, p->scale + t * (k->scale - p->scale), c);
        }
    }
    if (!qt_done) diag_qt(I6, d, nu, p, k);
}

/*
 * oracle_get_mw with the diagnostics: Lparms, Rparms, Parms, RL as oracle_get_mw; coords f64 (4, Nz) column-major,
 * voxel k's {x, y, z, r} at k*4; diag f64 (6, Nf) column-major: {EM_X, EM_Y, EM_Z, EM_R, TAU_L, TAU_R} at f*6.
 */
int oracle_get_mw_diag(const int32_t *Lparms, const double *Rparms, const double *Parms, const double *coords,
                       double *RL, double *diag)
{
    const int Nz = Lparms[0], Nf = Lparms[1];
    if (Nz < 0 || Nf <= 0) return 1;
    if (Lparms[2] > 0) return 2;
    const double area = Rparms[0], f0 = Rparms[1], step = Rparms[2];
    for (int f = 0; f < Nf; ++f) {
        const double nu = f0 * pow(10.0, step * f);
        double I6[6] = {0, 0, 0, 0, 0, 0};
        diag_t d;
        memset(&d, 0, sizeof(d));
        voxel_t prev; int have_prev = 0;
        const double *cprev = NULL;
        for (int k = 0; k < Nz; ++k) {
            const double *P = Parms + (size_t)k * 15;
            const double *c = coords + (size_t)k * 4;
            voxel_t vx;
            vx.dz = P[0]; vx.T = P[1]; vx.ne = P[2]; vx.B = P[3];
            vx.th = P[4] * M_PI / 180.0;
            const int flag = (int)P[6];
            vx.gr_on = !(flag & 1); vx.ff_on = !(flag & 2);
            vx.smax = (int)P[7];
            vx.scale = (P[14] > 0.0) ? P[14] / area : 1.0;
            if (!(vx.dz > 0.0) || !(vx.T > 0.0) || !(vx.ne > 0.0) || !(vx.B >= 0.0) ||
                !isfinite(vx.dz) || !isfinite(vx.T) || !isfinite(vx.ne) || !isfinite(vx.B) || !isfinite(vx.th)) {
                have_prev = 0;
                continue;
            }
            vx.cth = cos(vx.th); vx.sth = sin(vx.th);
            if (have_prev && vx.B > 0.0 && prev.B > 0.0) {
                double mid[4];
                for (int q = 0; q < 4; ++q) mid[q] = 0.5 * (cprev[q] + c[q]);
                diag_between(I6, &d, nu, &prev, &vx, mid);
            }
            const int x_to_R = vx.cth >= 0.0;
            for (int sg = -1; sg <= 1; sg += 2) {
                mode_t m;
                mode_eval(nu, vx.ne, vx.B, vx.T, vx.cth, vx.sth, sg, vx.ff_on, &m, 0, 0);
                const int to_R = (sg < 0) ? x_to_R : !x_to_R;
                apply_mode(I6, to_R, m.prop, m.kap * vx.dz, m.src * vx.scale);
                diag_mode(&d, to_R, m.prop, m.kap * vx.dz, m.src * vx.scale, c);
            }
            prev = vx; have_prev = 1; cprev = c;
        }
        double *o = RL + (size_t)f * 7;
        const double to_sfu = area / (AU_CM * AU_CM) / SFU;
        o[0] = nu / 1e9;
        for (int q = 0; q < 6; ++q) o[1 + q] = I6[q] * to_sfu;
        double *g = diag + (size_t)f * 6;
        const double I = I6[4] + I6[5];
        const int ok = I != 0.0 && isfinite(I);
        for (int q = 0; q < 4; ++q) g[q] = ok ? (d.w[0][q] + d.w[1][q]) / I : NAN;
        g[4] = d.tau[0];
        g[5] = d.tau[1];
    }
    return 0;
}
