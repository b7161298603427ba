// Fused map renderer for sm_100a: integrate the ray, sample n_e/T/|B| (and the B vector) at every
// recorded step and advance the polarised transfer equation — one thread per (pixel, frequency),
// nothing materialised: no r_record, no S array, no Parms.
//
// Equivalent to the reference chain
//   trace_ray / ray_trace                      (build_rays.py:128-248)
//   -> sample_model_with_rays                  (gpu_raytrace.py:632-651, float32 semantics)
//   -> Parms packing + GET_MW + T_b conversion (script/resample_with_ray_tracing.py:467-530)
// called once per frequency as the publication drivers do (script/pub/TbSpectra_gen.py:155-182).
// A 2048^2 x 500-record map would need 25 GB of paths per frequency if materialised
// (SURVEY.md §5); here a record lives in registers for the few hundred cycles it is needed.
// The DIAG instantiations (rtgrff_render_map_diag) also accumulate where each pixel's emission comes from: emission
// centroid and height, optical depths, the ray's turning point (DiagAcc below, definitions in include/rtgrff.h).
#pragma once

#include "grff.cuh"
#include "los_sampler.cuh"
#include "trace_kernel.cuh"

#include <type_traits>

namespace rtgrff {

// Everything that depends on the frequency only, prepared on the host and passed BY VALUE inside
// the kernel parameters: the ~20 registers these constants used to occupy per thread were spilled
// around the record-time code.  One launch per frequency, so that they sit at fixed offsets of the
// constant bank and become instruction operands.
struct FreqDev {
    double nu, omega0, dt;
    int64_t n_steps, stride;
    int out_row;          // row of this frequency in the caller's tb / vi arrays
    StepConst K;
    FreqC fq;
};

struct MapArgs {
    RayCube cube;
    const float4 *fcube, *bcube;
    GridGeomF fg;
    int64_t n_rays;
    const double *x_start, *y_start, *z_start, *kvec;
    const int *ray_order;                // thread t handles ray ray_order[t] (nullptr: t); see rtgrff.h
    FreqDev freq;                        // the frequency of this launch
    double perturb_ratio, area;
    float r_sun_cm, fill_ne, fill_te, fill_b;
    int em_flag, s_max, use_bvec, order, cs_every_step;
    int s_mode;                          // RTGRFF_S_PER_STEP / RTGRFF_S_CUMULATIVE: which S a record carries
    int s_input;                         // the record's S scales the voxel's source term (--s-input-on)
    int grff64;                          // 1: every voxel through the FP64 evaluation (RTGRFF_GRFF64=1, A/B and validation)
    double *tb, *vi;                     // [freq][ray]
    unsigned long long *active_steps;    // [0] active central steps, [1] steps with the pencil traced, [2] valid samples
    double *diag;                        // [RTGRFF_N_DIAG][freq][ray], the DIAG variants only
    int64_t diag_plane;                  // elements from one diagnostic plane to the next: n_freq * n_rays
};

// ---- map diagnostics (the DIAG variants; planes and definitions in include/rtgrff.h) ----
// Next to the transfer I four weighted transfers W^c run, c = x, y, z, |p|: every source term b enters them as
// b c, c the coordinate of the event it belongs to, and every operator acts on W as on I (slab a W + b c, the same
// L/R mixing at a quasi-transverse layer, acc += M b c in the outward fold).  W^c / I is then the exact
// contribution-weighted mean of c.  A voxel's coordinate is its record position (the float32 x, y, z the sampler
// used); an event between two voxels takes the midpoint of the two, so the centroid is resolved to the record
// spacing.  The optical depths kappa ds of the slabs and gyroresonance layers are summed per slot.
__device__ __forceinline__ float4 diag_coord(float x, float y, float z)
{
    return make_float4(x, y, z, sqrtf(fmaf(x, x, fmaf(y, y, z * z))));
}

__device__ __forceinline__ float4 diag_mid(const float4 &p, const float4 &q)
{
    return make_float4(0.5f * (p.x + q.x), 0.5f * (p.y + q.y), 0.5f * (p.z + q.z), 0.5f * (p.w + q.w));
}

struct DiagAcc {
    double wL[4], wR[4];
    double tauL, tauR;
    float4 prev;          // coordinate of the previous non-empty voxel the transfer keeps
    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int q = 0; q < 4; ++q) { wL[q] = 0.0; wR[q] = 0.0; }
        tauL = tauR = 0.0;
    }
    __device__ __forceinline__ void add_tau(double tl, double tr) { tauL += tl; tauR += tr; }
    // record order: W <- a W + b c
    __device__ __forceinline__ void apply(const DiagOp &d, const float4 &c)
    {
        const double cc[4] = {(double)c.x, (double)c.y, (double)c.z, (double)c.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) { wL[q] = fma(wL[q], d.aL, d.bL * cc[q]); wR[q] = fma(wR[q], d.aR, d.bR * cc[q]); }
    }
    __device__ __forceinline__ void qt(double Q)
    {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double l = wL[q], r = wR[q];
            wL[q] = Q * l + (1.0 - Q) * r;
            wR[q] = Q * r + (1.0 - Q) * l;
        }
    }
    // outward order: W_acc += (M b) c, before M takes the operator
    __device__ __forceinline__ void fold(double m00, double m01, double m10, double m11, const DiagOp &d, const float4 &c)
    {
        const double pL = m00 * d.bL + m01 * d.bR, pR = m10 * d.bL + m11 * d.bR;
        const double cc[4] = {(double)c.x, (double)c.y, (double)c.z, (double)c.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) { wL[q] = fma(pL, cc[q], wL[q]); wR[q] = fma(pR, cc[q], wR[q]); }
    }
    // the seven planes of one (pixel, frequency) from the exact-coupling I_L, I_R and the ray's smallest |p|
    __device__ __forceinline__ void write(double IL, double IR, float rmin, double *out, size_t plane) const
    {
        const double I = IL + IR;
        const bool ok = I != 0.0 && isfinite(I);
#pragma unroll
        for (int q = 0; q < 4; ++q) out[(size_t)(RTGRFF_DIAG_EM_X + q) * plane] = ok ? (wL[q] + wR[q]) / I : (double)NAN;
        out[(size_t)RTGRFF_DIAG_TAU_L * plane] = tauL;
        out[(size_t)RTGRFF_DIAG_TAU_R * plane] = tauR;
        out[(size_t)RTGRFF_DIAG_RAY_RMIN * plane] = rmin < INFINITY ? (double)rmin : (double)NAN;
    }
};

// Transfer accumulated from the observer outwards (RTGRFF_ORDER_REVERSED): the records arrive
// nearest-first, the radiation travels farthest-first.  I_obs = acc + M I_far with M a 2x2 matrix
// in (L,R); folding one more (farther) operator I -> A I + b gives acc += M b, M = M A.
struct OutwardTransfer {
    double m00, m01, m10, m11, accL, accR;
    VoxLite prev;
    bool have_prev;
    __device__ __forceinline__ void init()
    {
        m00 = m11 = 1.0; m01 = m10 = 0.0; accL = accR = 0.0; have_prev = false;
    }
    __device__ __forceinline__ void fold(const DiagOp &d)
    {
        accL += m00 * d.bL + m01 * d.bR;
        accR += m10 * d.bL + m11 * d.bR;
        m00 *= d.aL; m10 *= d.aL; m01 *= d.aR; m11 *= d.aR;
    }
    __device__ __forceinline__ void fold_qt(double Q)
    {
        const double p = 1.0 - Q;
        const double a = m00 * Q + m01 * p, b = m00 * p + m01 * Q;
        const double c = m10 * Q + m11 * p, d = m10 * p + m11 * Q;
        m00 = a; m01 = b; m10 = c; m11 = d;
    }
};

// NEED_BETWEEN: gyroresonance on or theta from the B vector -> the previous voxel must be kept for
// the between-voxel events; with the reference's packing (theta = 90, GR off) it is dead weight.
// A voxel arrives as the float32 values the sampler produced (VoxLite + sin theta); its slab operator is
// evaluated in float32 where that is well conditioned (voxel_op_mixed), the intensities live in FP64.
// DIAG: the diagnostics' accumulators (DiagAcc) run alongside; (x, y, z) is the record position of the voxel.
template <bool NEED_BETWEEN, bool DIAG = false>
struct RecordTransfer {
    PolState<1> st;
    VoxLite prev;
    bool have_prev;
    DiagAcc dg;
    __device__ __forceinline__ void init()
    {
        st.clear(); have_prev = false;
        if constexpr (DIAG) dg.init();
    }
    __device__ __forceinline__ void push(const FreqC &f, const VoxLite &l, float sth, int flag, int smax, bool force64,
                                         float x, float y, float z)
    {
        if (!voxel_nonempty_f(l.dz, l.T, l.ne, l.B, l.cth)) { have_prev = false; return; }
        float4 c;
        if constexpr (DIAG) c = diag_coord(x, y, z);
        if (NEED_BETWEEN) {
            if (have_prev && prev.B > 0.0f && l.B > 0.0f && between_needed_f(f, prev.cth, prev.B, l.cth, l.B, smax, !(flag & 1)))
            {
                Between b;
                between_voxels_cold(f.nu, f.sn, prev, l, flag, smax, &b);
                if constexpr (DIAG) {
                    const double2 t = between_tau_cold(f.nu, f.sn, prev, l, flag, smax);
                    dg.add_tau(t.x, t.y);
                    const float4 m = diag_mid(dg.prev, c);
                    dg.apply(b.before, m);
                    if (b.qt) dg.qt(b.Q);
                    dg.apply(b.after, m);
                }
                st.apply(b);
            }
            prev = l;
            have_prev = true;
            if constexpr (DIAG) dg.prev = c;
        }
        if constexpr (DIAG) {
            const TauOp o = voxel_op_mixed_tau(f, l.dz, l.T, l.ne, l.B, l.cth, sth, l.scale, flag, smax, force64);
            dg.add_tau(o.tauL, o.tauR);
            dg.apply(o.op, c);
            st.apply(o.op);
        } else {
            st.apply(voxel_op_mixed(f, l.dz, l.T, l.ne, l.B, l.cth, sth, l.scale, flag, smax, force64));
        }
    }
    __device__ __forceinline__ void result(double &L, double &R) const { L = st.L[0]; R = st.R[0]; }
};

template <bool NEED_BETWEEN, bool DIAG = false>
struct OutwardTransferT : OutwardTransfer {
    DiagAcc dg;
    __device__ __forceinline__ void init()
    {
        OutwardTransfer::init();
        if constexpr (DIAG) dg.init();
    }
    __device__ __forceinline__ void fold_diag(const DiagOp &d, const float4 &c)
    {
        dg.fold(m00, m01, m10, m11, d, c);
        fold(d);
    }
    __device__ __forceinline__ void push(const FreqC &f, const VoxLite &l, float sth, int flag, int smax, bool force64,
                                         float x, float y, float z)
    {
        if (!voxel_nonempty_f(l.dz, l.T, l.ne, l.B, l.cth)) { have_prev = false; return; }
        float4 c;
        if constexpr (DIAG) c = diag_coord(x, y, z);
        if (NEED_BETWEEN) {
            if (have_prev && prev.B > 0.0f && l.B > 0.0f && between_needed_f(f, l.cth, l.B, prev.cth, prev.B, smax, !(flag & 1))) {
                // radiation crosses v -> prev: between_voxels(v, prev) lists the events in that order,
                // folding outwards meets them last-first
                Between b;
                between_voxels_cold(f.nu, f.sn, l, prev, flag, smax, &b);
                if constexpr (DIAG) {
                    const double2 t = between_tau_cold(f.nu, f.sn, l, prev, flag, smax);
                    dg.add_tau(t.x, t.y);
                    const float4 m = diag_mid(dg.prev, c);
                    fold_diag(b.after, m);
                    if (b.qt) fold_qt(b.Q);
                    fold_diag(b.before, m);
                } else {
                    fold(b.after);
                    if (b.qt) fold_qt(b.Q);
                    fold(b.before);
                }
            }
            prev = l;
            have_prev = true;
            if constexpr (DIAG) dg.prev = c;
        }
        if constexpr (DIAG) {
            const TauOp o = voxel_op_mixed_tau(f, l.dz, l.T, l.ne, l.B, l.cth, sth, l.scale, flag, smax, force64);
            dg.add_tau(o.tauL, o.tauR);
            fold_diag(o.op, c);
        } else {
            fold(voxel_op_mixed(f, l.dz, l.T, l.ne, l.B, l.cth, sth, l.scale, flag, smax, force64));
        }
    }
    __device__ __forceinline__ void result(double &L, double &R) const { L = accL; R = accR; }
};

// DIAG: also write the diagnostic planes to a.diag (tb / vi are the same as without)
template <bool CS, int ORDER, bool BVEC, bool GR, int MODE, bool DIAG>
__global__ void __launch_bounds__(RT_BLOCK, RT_MINB) render_map_kernel(const MapArgs a)
{
    constexpr bool NEED_BETWEEN = BVEC || GR;
    const int64_t slot = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool has_ray = slot < a.n_rays;
    const int64_t ray = (has_ray && a.ray_order) ? (int64_t)a.ray_order[slot] : slot;
    const RayCube &C = a.cube;
    const FreqDev &fp = a.freq;
    const StepConst &K = fp.K;
    const FreqC &fq = fp.fq;
    Cell cache;
    cache.off = -1;

    State s;
    s.rx = s.ry = s.rz = s.kx = s.ky = s.kz = nan("");
    float px = 0.f, py = 0.f, pz = 0.f;   // previous VALID sample position, float32; starts at ray_start
    if (has_ray) {
        s.rx = a.x_start[ray]; s.ry = a.y_start[ray]; s.rz = a.z_start[ray];
        px = (float)s.rx; py = (float)s.ry; pz = (float)s.rz;     // _as_float32_c(ray_start), gpu_raytrace.py:650
        const double kc0 = start_kc(C, s.rx, s.ry, s.rz, fp.omega0);
        if (a.kvec) {
            s.kx = a.kvec[ray * 3 + 0] * kc0; s.ky = a.kvec[ray * 3 + 1] * kc0; s.kz = a.kvec[ray * 3 + 2] * kc0;
        } else {
            s.kx = 0.0 * kc0; s.ky = 0.0 * kc0; s.kz = -kc0;
        }
    }
    if (MODE == MODE_FAST32 && has_ray) init_cell(C, s, cache);
    bool alive = has_ray;
    float s_step = CS ? 0.0f : 1.0f;
    double s_cum = 1.0;
    // launch-uniform modes, read once
    const bool cumulative = CS && a.s_mode == RTGRFF_S_CUMULATIVE;
    const bool pencil_every_step = CS && (cumulative || a.cs_every_step);
    const bool s_input = a.s_input != 0, force64 = a.grff64 != 0;
    unsigned int n_samples = 0;
    const int n_steps = (int)fp.n_steps, stride = (int)fp.stride;     // < 2^31, checked on the host
    int next_rec = 0;
    int death = -1;                       // step at which the ray froze (-1: still moving)

    typename std::conditional<ORDER == RTGRFF_ORDER_RECORD, RecordTransfer<NEED_BETWEEN, DIAG>,
                              OutwardTransferT<NEED_BETWEEN, DIAG>>::type tr;
    tr.init();
    float rmin = INFINITY;                // DIAG: smallest |p| over the records with a finite position
    bool first = true;
    bool tail_done = !has_ray;            // a frozen ray repeats the same record: ds = 0 -> empty voxel

    // The steps go in intervals: one step with the pencil traced (CS), then up to the next such step the central
    // ray only, in a tight loop with no record bookkeeping (most steps: the record strides are 1-6).  In the per-step
    // S schedule the interval is the record stride and its first step is the recorded one.  Cumulative S and
    // RTGRFF_CS_EVERY_STEP=1 need the pencil at every step: intervals of one step, a record at every stride-th.
    const int interval = pencil_every_step ? 1 : stride;
    for (int i = 0; i < n_steps;) {
        if (alive) {
            alive = advance_ray<CS, MODE>(C, K, cache, s, fp.dt, a.perturb_ratio, CS, s_step);
            if (cumulative) s_cum *= s_step;     // gpu_raytrace.py:398-408
            if (!alive) death = i;
        }
        if (i == next_rec) {
            next_rec += stride;
            if (!tail_done) {
                // --- sampler (float32, gpu_raytrace.py:642-650) ---
                const float x = (float)s.rx, y = (float)s.ry, z = (float)s.rz, sv = cumulative ? (float)s_cum : s_step;
                if (DIAG && isfinite(x) && isfinite(y) && isfinite(z)) rmin = fminf(rmin, diag_coord(x, y, z).w);
                if (sample_valid(x, y, z, sv)) {
                    ++n_samples;
                    float3 bv = make_float3(0.f, 0.f, 0.f);
                    FieldSample f = BVEC ? sample_fields_bvec_fast(a.fcube, a.bcube, a.fg, x, y, z, a.fill_ne, a.fill_te, bv)
                                         : sample_fields(a.fcube, a.fg, x, y, z, a.fill_ne, a.fill_te, a.fill_b);
                    const float dist = first ? dist_first_np(x, y, z, px, py, pz) : dist_fast(x, y, z, px, py, pz);
                    const float ds = __fmul_rn(dist, a.r_sun_cm);
                    float cthf = 6.123233995736766e-17f, sthf = 1.0f;                       // theta = 90 deg
                    if (BVEC) {
                        // theta between the B vector and the propagation direction (towards the observer:
                        // against the tracing direction), all from float32 inputs: FP32 throughout
                        const float dx = x - px, dy = y - py, dz = z - pz;
                        const float dn2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
                        const float b2 = fmaf(bv.x, bv.x, fmaf(bv.y, bv.y, bv.z * bv.z));
                        f.b = f.inb ? sqrt_approx(b2) : a.fill_b;
                        if (b2 > 0.0f && dn2 > 0.0f) {
                            const float inv = rsqrtf(b2 * dn2);
                            const float c = -fmaf(bv.x, dx, fmaf(bv.y, dy, bv.z * dz)) * inv;
                            cthf = fminf(1.0f, fmaxf(-1.0f, c));
                            // sin from the cross product: no cancellation near theta = 0
                            const float cx = bv.y * dz - bv.z * dy, cy = bv.z * dx - bv.x * dz, cz = bv.x * dy - bv.y * dx;
                            sthf = fminf(1.0f, sqrt_approx(fmaf(cx, cx, fmaf(cy, cy, cz * cz))) * inv);
                        }
                    }
                    // --- Parms packing rules (script/resample_with_ray_tracing.py:472-501) ---
                    if (isfinite(f.ne) && isfinite(f.te) && isfinite(f.b)) {
                        // Parms[14] = S * area (script/resample_with_ray_tracing.py:501): source factor S
                        const VoxLite lite = {ds, f.te, f.ne, f.b, cthf, s_input ? sv : 1.0f};
                        tr.push(fq, lite, sthf, a.em_flag, a.s_max, force64, x, y, z);
                    }
                    px = x; py = y; pz = z;
                    first = false;
                }
                // once frozen, every later record repeats this one (ds = 0 or invalid): nothing to add
                if (!alive) tail_done = true;
            }
        }
        // a frozen ray still owes its first post-freeze record (with the cross-sections off its S is 1 and the
        // record counts, exactly as in trace -> sample -> emission): leave only when every lane has handed it over
        if (!__any_sync(0xffffffffu, alive || !tail_done)) break;
        // The rest of the interval.  Its loop carries only the interval's own moving / frozen_at: with the ray's
        // alive / death / s_step in it (live across the whole kernel, so in spill slots), every step reloaded and
        // stored them.  A ray frozen here hands its record over at the start of the next interval (it no longer moves).
        const int end = n_steps - i > interval ? i + interval : n_steps;
        bool moving = alive;
        int frozen_at = end;
        for (int j = i + 1; j < end; ++j)
            if (moving && !advance_central<MODE>(C, K, cache, s, fp.dt)) { moving = false; frozen_at = j; }
        if (frozen_at < end) {
            alive = false;
            death = frozen_at;
            if (CS) s_step = nanf("");      // as advance_ray
        }
        i = end;
    }
    if (has_ray) {
        double tb, vi, IL, IR;
        tr.result(IL, IR);
        tb_vi(IL, IR, fp.nu, a.area, tb, vi);
        a.tb[(size_t)fp.out_row * a.n_rays + ray] = tb;
        a.vi[(size_t)fp.out_row * a.n_rays + ray] = vi;
        if constexpr (DIAG) tr.dg.write(IL, IR, rmin, a.diag + (size_t)fp.out_row * a.n_rays + ray, (size_t)a.diag_plane);
    }
    if (a.active_steps) {
        // a ray moves on steps [0, death): the counters follow from where it froze
        unsigned long long moved_steps = has_ray ? (unsigned long long)(death >= 0 ? death : n_steps) : 0ull;
        const unsigned long long pencil_steps =
            !CS ? 0ull : (pencil_every_step ? moved_steps : (moved_steps + stride - 1) / stride);
        unsigned long long ps = pencil_steps, ns = n_samples;
        for (int off = 16; off > 0; off >>= 1) {
            moved_steps += __shfl_down_sync(0xffffffffu, moved_steps, off);
            ps += __shfl_down_sync(0xffffffffu, ps, off);
            ns += __shfl_down_sync(0xffffffffu, ns, off);
        }
        if ((threadIdx.x & 31) == 0) {
            if (moved_steps) atomicAdd(a.active_steps, moved_steps);
            if (ps) atomicAdd(a.active_steps + 1, ps);
            if (ns) atomicAdd(a.active_steps + 2, ns);
        }
    }
}

}  // namespace rtgrff
