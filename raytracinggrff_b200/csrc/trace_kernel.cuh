// Trace kernel: the whole n_steps loop of one ray in one thread (see ray_integrator.cuh for the
// FP64 stepper and ray_core32.cuh for the FP32 cell-relative stepper it can run on).
#pragma once

#include "ray_core32.cuh"

namespace rtgrff {

// Stepper: MODE_FAST32 = FP64 master state + FP32 cell-relative RHS + register cell cache; MODE_F64 = FP64
// state and RHS with FP32 trilinear arithmetic, which the host picks when a step plus the pencil offset
// reaches kMaxStageOffsetCells.
enum { MODE_FAST32 = 0, MODE_F64 = 1 };

// Advance one ray by one step with the selected stepper.  Returns whether the ray is still alive.
// A step that leaves the state untouched (outside the cube, NaN, omega = 0) repeats forever: the
// ray is frozen from here on (bit-identical to the reference continuing), and every later step's
// cross-section ratio is 0/0 = NaN (r_diff = 0 in build_rays.py:217-239).
//
// `want_s` (warp-uniform): the reference computes the per-step cross-section ratio at EVERY step
// but only the value of a recorded step ever leaves ray_trace (build_rays.py:241-244), so in
// per-step mode the two pencil rays are traced on recorded steps only — same output, 8 of the 12
// RHS evaluations skipped on the other steps.  Cumulative mode needs every step.
template <bool CS, int MODE>
__device__ __forceinline__ bool advance_ray(const RayCube &C, const StepConst &K, Cell &cache, State &s, double dt,
                                            double perturb_ratio, bool want_s, float &s_step)
{
    bool moved;
    if (MODE == MODE_FAST32) {
        moved = step32<CS>(C, K, cache, s, want_s, s_step);
    } else {
        const State s0 = s;
        s = rk4_step(C, s0, dt);
        if (CS && want_s) s_step = (float)cross_section_ratio(C, s0, s, dt, perturb_ratio);
        moved = in_cube(C, s0.rx, s0.ry, s0.rz) && state_differs(s, s0);
    }
    if (CS && !moved) s_step = nanf("");
    return moved;
}

// advance_ray with want_s = false, without the pencil's state: the steps whose cross-section ratio no
// record carries (render_map_kernel's steps between two records).  Returns whether the ray moved; the
// caller sets the frozen ray's S to NaN as advance_ray does.
template <int MODE>
__device__ __forceinline__ bool advance_central(const RayCube &C, const StepConst &K, Cell &cache, State &s, double dt)
{
    if (MODE == MODE_FAST32) return step32_central(C, K, cache, s);
    const State s0 = s;
    s = rk4_step(C, s0, dt);
    return in_cube(C, s0.rx, s0.ry, s0.rz) && state_differs(s, s0);
}

struct TraceArgs {
    RayCube cube;
    int64_t n_rays;
    const double *x_start, *y_start, *z_start;  // device, (n_rays)
    const double *kvec;                          // device, (n_rays,3) or nullptr -> (0,0,-1)
    double omega0, dt, perturb_ratio;
    StepConst K;                                 // host-prepared constants of the FP32 stepper (constant bank)
    int64_t n_steps, stride, n_rec;
    int s_mode;
    int cs_every_step;   // 1: trace the pencil rays at every step even when only recorded steps are kept
    double *rec_pos;  // device [rec][3][ray]
    double *rec_s;    // device [rec][ray] (only when CS)
    unsigned long long *active_steps;
};

template <bool CS, int MODE>
__global__ void __launch_bounds__(RT_BLOCK, RT_MINB) trace_rays_kernel(const TraceArgs a)
{
    const int64_t ray = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool has_ray = ray < a.n_rays;
    const RayCube &C = a.cube;
    const StepConst &K = a.K;
    Cell cache;
    cache.off = -1;
    State s;
    s.rx = s.ry = s.rz = s.kx = s.ky = s.kz = nan("");
    if (has_ray) {
        s.rx = a.x_start[ray]; s.ry = a.y_start[ray]; s.rz = a.z_start[ray];
        const double kc0 = start_kc(C, s.rx, s.ry, s.rz, a.omega0);
        if (a.kvec) {
            s.kx = a.kvec[ray * 3 + 0] * kc0; s.ky = a.kvec[ray * 3 + 1] * kc0; s.kz = a.kvec[ray * 3 + 2] * kc0;
        } else {
            s.kx = 0.0 * kc0; s.ky = 0.0 * kc0; s.kz = -kc0;
        }
    }
    if (MODE == MODE_FAST32 && has_ray) init_cell(C, s, cache);
    bool alive = has_ray;
    float s_step = 0.0f;        // the ratio is a float32 quantity (MUFU-normalised pencil basis); the sampler casts it anyway
    double s_cum = 1.0;
    unsigned long long moved_steps = 0;
    int64_t rec = 0, next_rec = 0;
    const size_t n = (size_t)a.n_rays;

    for (int64_t i = 0; i < a.n_steps; ++i) {
        if (alive) {
            const bool want_s = CS && (i == next_rec || a.s_mode == RTGRFF_S_CUMULATIVE || a.cs_every_step);
            alive = advance_ray<CS, MODE>(C, K, cache, s, a.dt, a.perturb_ratio, want_s, s_step);
            if (CS && a.s_mode == RTGRFF_S_CUMULATIVE) s_cum *= s_step;
            moved_steps += alive ? 1ull : 0ull;
        }
        if (i == next_rec) {
            if (has_ray) {
                double *o = a.rec_pos + (size_t)rec * 3 * n + (size_t)ray;
                o[0] = s.rx; o[n] = s.ry; o[2 * n] = s.rz;
                if (CS) a.rec_s[(size_t)rec * n + (size_t)ray] = (a.s_mode == RTGRFF_S_CUMULATIVE) ? s_cum : (double)s_step;
            }
            ++rec;
            next_rec += a.stride;
        }
        if (!__any_sync(0xffffffffu, alive)) break;
    }
    // frozen tail: constant records
    if (has_ray) {
        const double sv = (a.s_mode == RTGRFF_S_CUMULATIVE) ? s_cum : (double)s_step;
        for (; rec < a.n_rec; ++rec) {
            double *o = a.rec_pos + (size_t)rec * 3 * n + (size_t)ray;
            o[0] = s.rx; o[n] = s.ry; o[2 * n] = s.rz;
            if (CS) a.rec_s[(size_t)rec * n + (size_t)ray] = sv;
        }
    }
    if (a.active_steps) {
        for (int off = 16; off > 0; off >>= 1) moved_steps += __shfl_down_sync(0xffffffffu, moved_steps, off);
        if ((threadIdx.x & 31) == 0 && moved_steps) atomicAdd(a.active_steps, moved_steps);
    }
}

}  // namespace rtgrff
