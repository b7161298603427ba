/*
 * rtgrff.h — C ABI of librtgrff_b200.so: the B200 (sm_100a) implementation of the per-ray hot
 * path of peijin94/raytracingGRFF (ray integrator -> LOS resampler -> GRFF transfer).
 *
 * Plain C types, raw pointers and sizes only.  Every entry point cites the reference interface
 * it replaces (paths are inside the reference repository).  All functions return 0 on success
 * and a negative RTGRFF_E* code on failure (PyGET_MW keeps GRFF's convention: 0 ok, >0 error);
 * rtgrff_last_error() returns a thread-local message for the last failure.
 *
 * Buffers marked "host" are caller-owned host memory (pageable or pinned); device memory is
 * owned by the library behind the opaque context, one context per GPU.  A context is not
 * thread-safe; use one per thread (the reference's path is single-threaded as well).
 */
#ifndef RTGRFF_H
#define RTGRFF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTGRFF_OK 0
#define RTGRFF_EINVAL (-1)      /* bad argument / size                                   */
#define RTGRFF_ECUDA (-2)       /* CUDA runtime error (message has the cudaError string)  */
#define RTGRFF_ENOCUBE (-3)     /* the cube this call needs has not been uploaded        */
#define RTGRFF_ENOMEM (-4)
#define RTGRFF_EUNSUPPORTED (-5)

typedef struct rtgrff_ctx rtgrff_ctx;

/* Library / build identification ("rtgrff_b200 <version> sm_100a"). */
const char *rtgrff_version(void);
const char *rtgrff_last_error(void);
/* Number of CUDA devices visible; <0 on error (no driver, no GPU). */
int rtgrff_device_count(void);

/* One context per GPU.  `stream` is a cudaStream_t passed as void* (NULL = the library creates
 * its own non-blocking stream).  Passing torch's current stream makes torch CUDA events see the
 * library's kernels.  Every entry point switches to the context's device for the duration of the
 * call and restores the caller's current device before it returns. */
int rtgrff_ctx_create(int device, void *stream, rtgrff_ctx **out);
/* Same, but `stream` is always the caller's stream — including 0, the legacy default stream (which
 * is torch's default stream): all work of the context is then ordered with the caller's own work on
 * that stream, as buffers shared with the caller (out_on_device, on_device) require. */
int rtgrff_ctx_create_on_stream(int device, void *stream, rtgrff_ctx **out);
/* The calling thread's current CUDA device (module-level Python drop-ins default to it); <0 on error. */
int rtgrff_current_device(void);
int rtgrff_ctx_destroy(rtgrff_ctx *ctx);
int rtgrff_ctx_synchronize(rtgrff_ctx *ctx);
/* The per-ray kernels (rtgrff_render_map, rtgrff_emission_traced) evaluate a voxel's opacities in float32 where that
 * is well conditioned and in FP64 near the mode cut-offs (DESIGN.md 4.4).  enabled = 1 forces FP64 for every voxel
 * (default 0; env RTGRFF_GRFF64=1): A/B and validation switch.  PyGET_MW / rtgrff_get_mw_slice are always FP64. */
int rtgrff_ctx_set_grff64(rtgrff_ctx *ctx, int enabled);
/* Large host arrays travel in chunks through page-locked bounce buffers, overlapped with the kernels
 * (rtgrff_sample, rtgrff_get_mw_slice, cube uploads, image download).  enabled = 0 switches to one plain copy
 * each way, so that rtgrff_ctx_last_kernel_ms brackets the kernel alone (default 1; env RTGRFF_PIPELINE=0). */
int rtgrff_ctx_set_pipeline(rtgrff_ctx *ctx, int enabled);
/* Kernel launches issued by this context since creation (for bench.py's gpu_launches). */
int64_t rtgrff_ctx_launch_count(const rtgrff_ctx *ctx);
/* Device time in ms of the dominant kernel of the last trace/sample/get_mw_slice/emission/render
 * call, measured with CUDA events on the context's stream (-1 if none).  Synchronises on the event. */
double rtgrff_ctx_last_kernel_ms(rtgrff_ctx *ctx);

/*
 * Grid geometry of one axis: {g[0], mean step, g[n-1], g[1]-g[0]}: (g0, step) exactly as the
 * reference's _check_uniform_grid returns them (raytracingGRFF/gpu_raytrace.py:21-33), the last
 * node, which scipy's bounds test uses (build_rays.py:140), and the spacing np.gradient is given
 * (build_rays.py:132-138).  geom[12] = {x0,dx,xl,hx, y0,dy,yl,hy, z0,dz,zl,hz}.
 */

/*
 * Upload omega_pe (nx,ny,nz) C-order float64 [rad/s] and build the interleaved
 * {omega_pe, d/dx, d/dy, d/dz} float32 cube on the device with numpy.gradient semantics.
 * Replaces: build_rays.py:132-143 (np.gradient x3 + four RegularGridInterpolator) and
 * gpu_raytrace.py:354-357 (H2D + cp.gradient x3).  `omega_pe` is host memory unless
 * `on_device` != 0 (then a device pointer readable from ctx's device).
 */
int rtgrff_set_omega_cube(rtgrff_ctx *ctx, const double *omega_pe, int nx, int ny, int nz,
                          const double geom[12], int on_device);

/*
 * Upload the model fields sampled along the rays, each (nx,ny,nz) C-order float32 host arrays:
 * n_e [cm^-3], T [K], |B| [G]; bx,by,bz [G] may be NULL (then theta = 90 deg everywhere, as the
 * reference hard-codes at script/resample_with_ray_tracing.py:495).
 * Replaces: gpu_raytrace.py:681 (per-call H2D of each field) / :647-649.
 */
int rtgrff_set_field_cubes(rtgrff_ctx *ctx, const float *ne, const float *te, const float *b,
                           const float *bx, const float *by, const float *bz,
                           int nx, int ny, int nz, const double geom[12]);

/*
 * Resample one variable of a spherical (phi, latitude, r) model onto the xyz cube and keep it on
 * the device in `slot` (0 rho/n_e, 1 te, 2 br, 3 bt, 4 bp); `out` (host float64 (nx,ny,nz), may be
 * NULL) receives a copy.  Replaces resample_to_xyz_cube (build_rays.py:69-125) and
 * resample_var_to_cube (script/resample_with_ray_tracing.py:110-151): cart_to_sph(x,-z,y,phi0),
 * linear interpolation with periodic phi (psipy's sample_at_coords), r < r_min or outside the mesh
 * -> NaN -> `fill` when fill_nonfinite.  data: host float32 (np,nt,nr) C-order; phi, lat, r: host
 * float64 node coordinates (rad, rad, R_sun), ascending; value = sample * scale.  x_grid, y_grid,
 * z_grid: host float64 cube nodes (used as they are, so a node on the rotation axis stays on it).
 */
int rtgrff_resample_spherical(rtgrff_ctx *ctx, int slot, const float *data, const double *phi,
                              const double *lat, const double *r, int np, int nt, int nr,
                              const double *x_grid, const double *y_grid, const double *z_grid, int nx,
                              int ny, int nz, const double geom[12], double phi0_offset_deg, double r_min,
                              double scale, double fill, int fill_nonfinite, double *out);

/*
 * Observer view.  The rtgrff_*_view entry points take the solar B0 and P angles [deg] of the observer, right after
 * phi0_offset_deg; the entry points without _view are the same calls with B0 = P = 0 (the model's equatorial plane
 * seen edge-on, solar north along image +y), and both give bit-identical results there.
 *
 * The observer frame is the cube frame: +z towards the observer, +y image up, +x image right (solar west when
 * P = 0; longitude grows towards +x, as Carrington longitude grows towards the west).  A cube or LOS point
 * p = (x, y, z) goes to model-aligned coordinates in two steps, then through the fixed mapping:
 *   1. undo P, a rotation about the line of sight:  x1 = x cos P + y sin P,  y1 = -x sin P + y cos P,  z1 = z
 *   2. undo B0, a rotation about x:                 x2 = x1,  y2 = y1 cos B0 + z1 sin B0,  z2 = -y1 sin B0 + z1 cos B0
 *   3. cart_to_sph(x2, -z2, y2, phi0).
 * Solar north in the observer frame is n = (-sin P cos B0, cos P cos B0, sin B0): B0 > 0 tilts the north pole towards
 * the observer, P > 0 turns north from +y towards -x (east), the ephemeris convention.  phi0_offset_deg keeps its
 * meaning: the central meridian does not depend on B0 or P.  The B vector is evaluated at (x2, y2, z2) and turned
 * back to the observer frame with the transpose of the same rotation.  The straight-LOS geometry (start on the disk
 * or on the plane of the sky behind the limb) is spherical and does not change.  B0 and P must be finite and
 * |B0| <= 90 deg, else RTGRFF_EINVAL.  Multiples of 90 deg are exact (P = 90 is an exact quarter turn).
 */
int rtgrff_resample_spherical_view(rtgrff_ctx *ctx, int slot, const float *data, const double *phi,
                                   const double *lat, const double *r, int np, int nt, int nr,
                                   const double *x_grid, const double *y_grid, const double *z_grid, int nx,
                                   int ny, int nz, const double geom[12], double phi0_offset_deg, double b0_deg,
                                   double p_deg, double r_min, double scale, double fill, int fill_nonfinite,
                                   double *out);

/*
 * Sample one spherical variable along straight lines of sight (the resampler of the straight-LOS
 * workflow, script/resampling_MAS_LOS.py:141-231): pixel (i,j) at (x[j], y[i]) [R_sun]; each LOS
 * starts on the solar surface / the plane of the sky behind the limb, minus z_eps, and runs towards
 * the observer over the offsets zc[k] [R_sun]; r < r_min or outside the mesh -> NaN.
 *  out: host float64 (ny, nx, nz).
 */
int rtgrff_sample_spherical_los(rtgrff_ctx *ctx, const float *data, const double *phi, const double *lat,
                                const double *r, int np, int nt, int nr, const double *x, const double *y,
                                const double *zc, int nx, int ny, int nz, double phi0_offset_deg,
                                double r_min, double scale, double z_eps, double *out);
int rtgrff_sample_spherical_los_view(rtgrff_ctx *ctx, const float *data, const double *phi, const double *lat,
                                     const double *r, int np, int nt, int nr, const double *x, const double *y,
                                     const double *zc, int nx, int ny, int nz, double phi0_offset_deg,
                                     double b0_deg, double p_deg, double r_min, double scale, double z_eps,
                                     double *out);

/*
 * Build the device cubes of the ray path from the five resampled slots with the reference's rules
 * (script/resample_with_ray_tracing.py:269-293): omega_pe = 2 pi 8.93e3 sqrt(max(rho,0)) (NaN -> 0)
 * and its numpy.gradient, n_e = max(rho,0), T NaN -> 1e4, |B| = sqrt(br^2+bt^2+bp^2); with
 * want_bvec also the Cartesian B vector (for theta from B.t).  Equivalent to rtgrff_set_omega_cube
 * + rtgrff_set_field_cubes without the cubes ever visiting the host.  The B vector is turned to the observer frame
 * with the view the slots were resampled with; RTGRFF_EINVAL if the five slots were resampled with different views.
 */
int rtgrff_compose_cubes(rtgrff_ctx *ctx, int want_bvec);

/* How the cross-section ratio S is recorded. */
#define RTGRFF_S_PER_STEP 0     /* CPU reference: ratio of the recorded step only (build_rays.py:239-244) */
#define RTGRFF_S_CUMULATIVE 1   /* CUDA reference: running product since the start (gpu_raytrace.py:398-408) */

/*
 * Integrate n_rays rays for n_steps RK4 steps.  Replaces build_rays.ray_trace
 * (build_rays.py:128-248) and gpu_raytrace._trace_ray_gpu (gpu_raytrace.py:328-411).
 *  x_start,y_start,z_start: host float64 (n_rays); kvec: host float64 (n_rays,3) unit directions.
 *  r_record: host float64 (n_rec,n_rays,3) or NULL; s_record: host float64 (n_rec,n_rays) or NULL
 *  (ignored unless trace_cs); n_rec = ceil(n_steps/record_stride), record i taken after step
 *  i*record_stride.  The records also stay on the device for rtgrff_sample_traced().
 *  active_steps (optional, host): central-ray steps taken while the ray still moved.
 */
int rtgrff_trace(rtgrff_ctx *ctx, int64_t n_rays, const double *x_start, const double *y_start,
                 const double *z_start, const double *kvec, double freq_hz, double dt,
                 int64_t n_steps, int64_t record_stride, int trace_cs, double perturb_ratio,
                 int s_mode, double *r_record, double *s_record, int64_t *active_steps);

/*
 * Sample n_e, T, |B| along recorded paths and compute validity and segment lengths.
 * Replaces gpu_raytrace._sample_model_with_rays_cuda/_cpu (gpu_raytrace.py:632-709), including
 * the per-ray Python loop _compute_ds_from_valid (:473-486).  float32 arithmetic as numpy does it.
 *  pos: host float32 (n_rec,n_rays,3); s: host float32 (n_rec,n_rays); ray_start: host float32 (n_rays,3).
 *  Outputs, host, (n_rec,n_rays): ne,te,b,ds float32; valid uint8 (0/1).
 */
int rtgrff_sample(rtgrff_ctx *ctx, int64_t n_rec, int64_t n_rays, const float *pos, const float *s,
                  const float *ray_start, double r_sun_cm, double fill_ne, double fill_te,
                  double fill_b, float *ne, float *te, float *b, float *ds, uint8_t *valid);

/* Same, on the records left on the device by the last rtgrff_trace() (no host round trip of the
 * paths).  Positions and S are rounded to float32 first, as the reference does (gpu_raytrace.py:642-643).
 * Any output pointer may be NULL; results also stay on the device for rtgrff_emission_traced(). */
int rtgrff_sample_traced(rtgrff_ctx *ctx, const float *ray_start, double r_sun_cm, double fill_ne,
                         double fill_te, double fill_b, float *ne, float *te, float *b, float *ds,
                         uint8_t *valid, float *s);

/*
 * GRFF single line of sight.  Same symbol, argument list and array layouts as
 * GRFF_DEM_Transfer.so::PyGET_MW bound at script/resample_with_ray_tracing.py:79-86:
 *  Lparms int32[5] {Nz,Nf,NT,DEMkey,DDMkey}; Rparms f64[3] {area cm^2, f0 Hz, log10 step};
 *  Parms f64 (15,Nz) column-major; T_arr/DEM_arr/DDM_arr unused (NT must be 0);
 *  RL f64 (7,Nf) column-major, written.  Returns 0 ok, 1 bad sizes, 2 DEM/DDM requested,
 *  3 CUDA failure.  Runs on device 0 through a process-wide context.
 */
int PyGET_MW(const int32_t *Lparms, const double *Rparms, const double *Parms,
             const double *T_arr, const double *DEM_arr, const double *DDM_arr, double *RL);

/*
 * GRFF batched over pixels, fastGRFF get_mw_slice layout (script/resample_with_ray_tracing.py:404-446):
 *  Lparms_M int32[6] {Npix,Nz,Nf,NT,DEMkey,DDMkey}; Rparms_M f64 (3,Npix); Parms_M f64 (15,Nz,Npix);
 *  RL_M f64 (7,Nf,Npix) written; status int32 (Npix) written; all host, Fortran order.
 */
int rtgrff_get_mw_slice(rtgrff_ctx *ctx, const int32_t *Lparms_M, const double *Rparms_M,
                        const double *Parms_M, const double *T_arr, const double *DEM_arr,
                        const double *DDM_arr, double *RL_M, int32_t *status);

/* The same call on DEVICE arrays — what the reference actually hands fastGRFF: CuPy Rparms_M / Parms_M /
 * RL_M with RL_M written in place on the device (script/resample_with_ray_tracing.py:428-446).
 * Lparms_M is host memory (6 integers); status_dev is a device int32 (Npix) or NULL. */
int rtgrff_get_mw_slice_device(rtgrff_ctx *ctx, const int32_t *Lparms_M, const double *Rparms_M_dev,
                               const double *Parms_M_dev, double *RL_M_dev, int32_t *status_dev);

/* Device memory on the context's GPU for callers without a CUDA binding of their own (image slabs for
 * rtgrff_render_map(out_on_device) + rtgrff_gather_image, staging of the *_device variants). */
int rtgrff_device_alloc(rtgrff_ctx *ctx, void **out, size_t bytes);
int rtgrff_device_free(rtgrff_ctx *ctx, void *ptr);

/* Plain copy on the context's stream, synchronous: kind 0 host->device, 1 device->host, 2 device->device.
 * Lets a host language without its own CUDA binding stage the device-array variants above. */
int rtgrff_memcpy(rtgrff_ctx *ctx, void *dst, const void *src, size_t bytes, int kind);

/* Copies of the device cubes back to the host (any pointer may be NULL): omega_pe float64 exactly as it
 * was differenced (available after rtgrff_compose_cubes / a host rtgrff_set_omega_cube until the next
 * cube upload), n_e, T, |B| and the B vector as stored (float32), each (nx,ny,nz) C-order.  For parity
 * checks of cubes that were built on the device (rtgrff_compose_cubes) against a CPU implementation. */
int rtgrff_export_cubes(rtgrff_ctx *ctx, double *omega_pe, float *ne, float *te, float *b, float *bx,
                        float *by, float *bz);

/*
 * GRFF + T_b conversion on the samples left on the device by rtgrff_sample_traced(): the
 * per-pixel loop of script/resample_with_ray_tracing.py:467-530 (valid filter, Parms packing with
 * theta=90, flag 1+4, s_max 30; GET_MW; SFU -> T_b; V/I; nan_to_num) without materialising Parms.
 *  tb, vi: host float64 (n_rays, n_freq) (= emission_cube / emission_polVI_cube flattened over pixels).
 *  s_input_on: the reference's --s-input-on (Parms[14] = S * area, :501).  The reference leaves the
 *  meaning of that slot to a private GRFF build; this library defines it: a voxel's source term is
 *  multiplied by Parms[14] / Rparms[0] = S (its own pencil cross-section instead of the pixel area),
 *  absorption unchanged.  PyGET_MW and rtgrff_get_mw_slice honour Parms[14] > 0 the same way.
 */
int rtgrff_emission_traced(rtgrff_ctx *ctx, double pixel_area_cm2, double freq0_hz, int n_freq,
                           double freq_log_step, int em_flag, int s_max, int s_input_on, double *tb,
                           double *vi);

/* Per-frequency settings of the fused map renderer. */
typedef struct {
    double freq_hz;        /* ray frequency = emission frequency */
    double dt;             /* integrator step [s] */
    int64_t n_steps;
    int64_t record_stride;
} rtgrff_freq_params;

#define RTGRFF_ORDER_RECORD 0    /* voxels handed to GRFF in record order (observer first), as the
                                    reference does for ray-traced maps (script/...:481-501)          */
#define RTGRFF_ORDER_REVERSED 1  /* far end first, observer last (GRFF's physical convention)          */

/*
 * Fused map: for every pixel and every frequency, trace the ray, sample the fields at each record
 * and integrate the transfer equation, without materialising paths.  Equivalent to
 * run_ray_tracing_emission (script/resample_with_ray_tracing.py:295-530) called once per frequency
 * as the publication drivers do (script/pub/TbSpectra_gen.py:155-182).
 *  Rays: x_start,y_start,z_start host float64 (n_rays), direction (0,0,-1) unless kvec != NULL.
 *  ray_order (host int32 (n_rays), a permutation, or NULL): thread t works on ray ray_order[t]; inputs
 *  and outputs keep the caller's ray numbering.  Walking an image in small 2-D tiles instead of rows
 *  puts 32 neighbouring pixels into a warp and cuts the distinct cube cells it gathers from.
 *  use_bvec: 0 -> theta=90 deg (reference behaviour); 1 -> theta from B.t along the ray (needs bx,by,bz).
 *  s_mode: which cross-section ratio a record carries (RTGRFF_S_PER_STEP as the reference's CPU path,
 *  RTGRFF_S_CUMULATIVE as its CUDA path — then the pencil is traced at every step); it decides the
 *  validity of a sample (S finite and > 0) and, with s_input_on (see rtgrff_emission_traced), the
 *  factor on the voxel's source term.
 *  tb, vi: float64 (n_freq, n_rays); host, or device pointers when out_on_device != 0.
 *  stats (optional, host int64[4]): {nominal ray-steps, active ray-steps (the ray still moved),
 *  steps on which the two cross-section rays were traced, valid samples handed to the transfer}.
 */
int rtgrff_render_map(rtgrff_ctx *ctx, int64_t n_rays, const double *x_start, const double *y_start,
                      const double *z_start, const double *kvec, const int32_t *ray_order, int n_freq,
                      const rtgrff_freq_params *freqs, int trace_cs, double perturb_ratio,
                      double pixel_area_cm2, double r_sun_cm, int em_flag, int s_max, int use_bvec,
                      int voxel_order, int s_mode, int s_input_on, double *tb, double *vi,
                      int out_on_device, int64_t *stats);

/*
 * Map diagnostics: where the emission a pixel sees comes from once refraction has bent the ray.  Planes of
 * rtgrff_render_map_diag's `diag`, float64 (RTGRFF_N_DIAG, n_freq, n_rays), each plane laid out as tb / vi.
 * They describe the transfer behind T_b: the exact-coupling I_L, I_R in the voxel_order asked for.
 *  EM_X, EM_Y, EM_Z  emission centroid [R_sun]: every contribution's position weighted by its share of I_L + I_R at
 *                    the observer.  Computed exactly with weighted transfers W^c that take every source term b as
 *                    b c and every operator as I does, EM_c = (W^c_L + W^c_R) / (I_L + I_R): the centroid lies in the
 *                    convex hull of the path.  A voxel's position is its record position (the float32 x, y, z the
 *                    sampler uses); a gyroresonance or quasi-transverse layer between two voxels takes the midpoint of
 *                    the two (the previous non-empty voxel), so the centroid is resolved to the record spacing.
 *  EM_R              contribution-weighted mean of |p| [R_sun] (not |centroid|): the emission height.
 *                    EM_* are NaN where I_L + I_R is 0 or not finite.
 *  TAU_L, TAU_R      total optical depth applied to the L and R slot: kappa ds of every slab, routed to L/R by the
 *                    sign of cos(theta) like the operator, plus the gyroresonance layers; a quasi-transverse layer adds
 *                    nothing.  +inf where the mode was evanescent somewhere on the path (its intensity was reset).
 *  RAY_RMIN          smallest |p| [R_sun] over the ray's records with a finite position: the ray's turning point; NaN
 *                    if there is none.
 */
#define RTGRFF_N_DIAG 7
#define RTGRFF_DIAG_EM_X 0
#define RTGRFF_DIAG_EM_Y 1
#define RTGRFF_DIAG_EM_Z 2
#define RTGRFF_DIAG_EM_R 3
#define RTGRFF_DIAG_TAU_L 4
#define RTGRFF_DIAG_TAU_R 5
#define RTGRFF_DIAG_RAY_RMIN 6

/*
 * rtgrff_render_map with the diagnostic planes above: the same arguments and the same tb, vi, stats, plus
 * diag float64 (RTGRFF_N_DIAG, n_freq, n_rays) (plane stride n_rays as tb / vi), host, or a device pointer when
 * out_on_device != 0.  diag == NULL is RTGRFF_EINVAL.  With tb, vi and diag consecutive in one device slab, the
 * 9 n_freq planes go through rtgrff_gather_image in one call.
 */
int rtgrff_render_map_diag(rtgrff_ctx *ctx, int64_t n_rays, const double *x_start, const double *y_start,
                           const double *z_start, const double *kvec, const int32_t *ray_order, int n_freq,
                           const rtgrff_freq_params *freqs, int trace_cs, double perturb_ratio,
                           double pixel_area_cm2, double r_sun_cm, int em_flag, int s_max, int use_bvec,
                           int voxel_order, int s_mode, int s_input_on, double *tb, double *vi,
                           int out_on_device, int64_t *stats, double *diag);

/*
 * Fused straight line-of-sight map: the straight-LOS counterpart of rtgrff_render_map, which replaces the staged
 * rtgrff_sample_spherical_los x 5 + GET_MW chain (script/resampling_MAS_LOS.py resample_MAS followed by
 * script/synthetic_FF_map_single_thread.py SyntheticFF) without materialising the LOS arrays or Parms.
 *
 * rtgrff_set_spherical_model: keep one variable of a spherical (phi, latitude, r) model resident on the device in
 * `slot` (0 rho/n_e [cm^-3], 1 te [K], 2 br, 3 bt, 4 bp [G]; value = data * scale) until the slot is set again.
 * data: host float32 (np, nt, nr) C-order; phi, lat, r: host float64 node coordinates (rad, rad, R_sun), ascending,
 * >= 2 per axis.  Independent of the slots of rtgrff_resample_spherical.
 */
int rtgrff_set_spherical_model(rtgrff_ctx *ctx, int slot, const float *data, const double *phi, const double *lat,
                               const double *r, int np, int nt, int nr, double scale);

/*
 * rtgrff_render_los_map: for every pixel (i, j) at (x[j], y[i]) [R_sun] the straight LOS of
 * rtgrff_sample_spherical_los (start on the disk surface or behind the limb on the plane of the sky, minus z_eps, then
 * the offsets zc[k] [R_sun] towards the observer, r < r_min -> no sample), sampled in FP64 from the five slots; then
 * the reference's packing: a sample with NaN in n_e, T or |B| is dropped, the others keep their order and are handed
 * to the transfer Sun side first with ds = dz_cm[k] [cm].  use_bvec 0: theta = 90 deg (the reference); 1: cos theta =
 * B_z / |B| with B rotated to cube axes (the radiation travels +z).  Each voxel goes through the per-ray kernels'
 * transfer (float32 voxel inputs, FP64 near the cut-offs or with rtgrff_ctx_set_grff64; gyroresonance when
 * !(em_flag & 1)).  T_b and V/I as SyntheticFF: V/I = (L-R)/(L+R) (NaN where L+R = 0); a LOS without a valid sample
 * gives T_b = 0, V/I = 0.
 *  freq_hz: host float64 (n_freq), any n_freq >= 1, any order.
 *  tb, vi: float64 (n_freq, ny, nx); diag: NULL or float64 (RTGRFF_N_DIAG, n_freq, ny, nx), the planes of
 *  rtgrff_render_map_diag with a voxel's position its float32 sample position and RAY_RMIN the smallest |p| over
 *  the LOS samples.  Host, or device pointers when out_on_device != 0: a rank that passes its rows' y values writes
 *  the slab rtgrff_gather_image assembles.
 *  stats (optional, host int64[3]): {LOS samples, valid samples, voxel-frequency evaluations}.
 * RTGRFF_ENOCUBE when a slot has not been set.
 */
int rtgrff_render_los_map(rtgrff_ctx *ctx, int nx, int ny, const double *x, const double *y, int nz, const double *zc,
                          const double *dz_cm, double phi0_offset_deg, double r_min, double z_eps, int n_freq,
                          const double *freq_hz, double pixel_area_cm2, int em_flag, int s_max, int use_bvec, double *tb,
                          double *vi, double *diag, int out_on_device, int64_t *stats);
/* rtgrff_render_los_map from the observer view (b0_deg, p_deg) (see "Observer view" above): the sample positions and,
 * with use_bvec, the B vector whose z component gives cos theta.  The diagnostic planes stay in the observer frame. */
int rtgrff_render_los_map_view(rtgrff_ctx *ctx, int nx, int ny, const double *x, const double *y, int nz,
                               const double *zc, const double *dz_cm, double phi0_offset_deg, double b0_deg,
                               double p_deg, double r_min, double z_eps, int n_freq, const double *freq_hz,
                               double pixel_area_cm2, int em_flag, int s_max, int use_bvec, double *tb, double *vi,
                               double *diag, int out_on_device, int64_t *stats);

/*
 * Multi-GPU (one process per GPU, the cube replicated on each).  Rays are independent, so the only exchange
 * is the gather of the image at the end; this replaces the reference's ProcessPoolExecutor ray chunks and
 * their concatenate (script/resample_with_ray_tracing.py:42-61, :333-352, the `--workers` switch).
 *
 * rtgrff_shard_rows: the image rows rank `rank` of `world_size` renders — rows are dealt round-robin in
 * groups of 8 adjacent rows (one by one for small images) because disk-centre rays run much longer than
 * limb rays.  rows: int32 (n_rows) buffer receiving the row indices (may be NULL), n_local their number,
 * max_rows the largest share of any rank (the slab height of rtgrff_gather_image).  Host only, no GPU needed.
 */
int rtgrff_shard_rows(int n_rows, int world_size, int rank, int32_t *rows, int *n_local, int *max_rows);

/* NCCL communicator over the contexts of all ranks (NCCL is loaded at run time: libnccl.so.2).  Rank 0 calls
 * rtgrff_comm_unique_id and hands the 128 bytes to the other ranks by whatever channel the host has (a file,
 * MPI, torch.distributed ...); then every rank calls rtgrff_comm_init_rank (collective).  world_size 1 needs no id. */
int rtgrff_comm_unique_id(char id[128]);
int rtgrff_comm_init_rank(rtgrff_ctx *ctx, int world_size, int rank, const char id[128]);
int rtgrff_comm_destroy(rtgrff_ctx *ctx);

/*
 * Gather the ranks' image slabs on `root` and put every row at its place (collective over the communicator;
 * a single-rank context just reorders).  slab: device float64 (n_planes, max_rows, n_cols), the rank's rows in
 * the order rtgrff_shard_rows lists them, padding after — what rtgrff_render_map writes with out_on_device when
 * its rays are the rank's rows (planes = [tb | vi] x frequency).  image (root only): float64 (n_planes, n_rows,
 * n_cols), a device pointer when image_on_device, else host memory (page-locked memory is written by DMA directly).
 */
int rtgrff_gather_image(rtgrff_ctx *ctx, const double *slab, int n_planes, int n_rows, int n_cols, int root,
                        double *image, int image_on_device);

/* The root-side half of rtgrff_gather_image on its own, for hosts that move the slabs by other means (MPI, files):
 * gathered = device float64 (world_size, n_planes, max_rows, n_cols), rank r's slab at index r; image = device
 * float64 (n_planes, n_rows, n_cols) with every row at its place. */
int rtgrff_place_rows(rtgrff_ctx *ctx, const double *gathered, int world_size, int n_planes, int n_rows, int n_cols,
                      double *image);

/*
 * Gaussian beam on the image plane: scipy.ndimage.gaussian_filter(map, sigma) as the workflow
 * applies it to its T_b maps (script/resample_with_ray_tracing.py:618-624; baseline beam of
 * script/pub/compare_on_off_scaling_factor.py:51-69): separable, kernel radius
 * int(truncate*sigma+0.5) (scipy's truncate = 4.0), 'reflect' boundary, float64; NaN pixels spread
 * as they do in scipy.  img, out: host float64 (n_planes, ny, nx); planes are filtered independently.
 */
int rtgrff_gaussian_beam(rtgrff_ctx *ctx, const double *img, int ny, int nx, int n_planes,
                         double sigma_pix, double truncate, double *out);

/*
 * patch_nan_emission_map (raytracingGRFF/util.py:6-77): every non-finite pixel becomes the mean
 * of the nearest finite pixels to its left, right, below and above (those that exist), visiting
 * pixels in row-major order and patching in place, for up to max_passes sweeps (the reference's
 * max_passes = 10).  img: host float64 (n_planes, ny, nx), patched in place; n_patched (optional).
 */
int rtgrff_patch_nan(rtgrff_ctx *ctx, double *img, int ny, int nx, int n_planes, int max_passes,
                     int64_t *n_patched);

#ifdef __cplusplus
}
#endif
#endif /* RTGRFF_H */
