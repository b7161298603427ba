// Shared host/device definitions of librtgrff_b200 (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/rtgrff.h"

// Threads per block / minimum resident blocks per SM of the per-ray kernels (tuned on B200, see
// profiles/): one thread per ray, small blocks so that finished warps free their slots early.
#define RT_BLOCK 64
#define RT_MINB 8

namespace rtgrff {

// build_rays.py:29-32 (C / R_S with the reference's rounded constants)
constexpr double kC_R = 2.998e10 / 6.96e10;

// Streams the per-frequency launches of the fused map go round-robin over.  The launches must overlap: each ends
// on a tail of half-empty SMs that the next one fills (DESIGN.md 4.1: one stream 514 ms, two or more 461 ms).
constexpr int kMapForkStreams = 8;

// Uniform-grid geometry of a cube.  x0/xl are the first/last node (scipy bounds test,
// build_rays.py:140), inv_d = 1/mean step (gpu_raytrace.py:21-33).
struct GridGeom {
    int nx, ny, nz;
    double x0, y0, z0;
    double xl, yl, zl;
    double idx, idy, idz;
};

// float32 view of the same geometry, rounded the way numpy's weak-scalar promotion rounds the
// Python floats in gpu_raytrace.py:495-497, :646.
struct GridGeomF {
    int nx, ny, nz;
    float x0, y0, z0;
    float idx, idy, idz;
    float fxl, fyl, fzl;   // (float)(n - 1): the in-bounds test 0 <= f <= n-1 of gpu_raytrace.py:505-511
};

extern thread_local char g_err[512];

inline int fail(int code, const char *fmt, ...)
    __attribute__((format(printf, 2, 3)));

#define RT_CUDA(call)                                                                          \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return rtgrff::fail(RTGRFF_ECUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,     \
                                cudaGetErrorString(e__));                                      \
    } while (0)

#define RT_TRY(call)                                                                           \
    do {                                                                                       \
        int r__ = (call);                                                                      \
        if (r__ != RTGRFF_OK) return r__;                                                      \
    } while (0)

// Growable device buffer owned by a context.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);
    void release();
    template <class T> T *as() const { return static_cast<T *>(p); }
};

inline unsigned int blocks_for(int64_t n, int block)
{
    int64_t b = (n + block - 1) / block;
    if (b < 1) b = 1;
    return (unsigned int)b;
}

}  // namespace rtgrff

struct rtgrff_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    // second stream + events + pinned bounce buffers of the chunked host<->device pipelines
    // (rtgrff_sample, rtgrff_get_mw_slice): host pack / H2D / kernel / D2H / host unpack overlap
    int grff64 = 0;                  // per-ray kernels evaluate every voxel in FP64 (RTGRFF_GRFF64, rtgrff_ctx_set_grff64)
    int pipeline = 1;                // chunked pinned host pipelines on (RTGRFF_PIPELINE, rtgrff_ctx_set_pipeline)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t chunk_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // in[2], kernel[2], out[2]
    // fork / join of the per-frequency launches of the fused map: one event per fork stream, the last one forks
    cudaStream_t fstream[rtgrff::kMapForkStreams] = {};
    cudaEvent_t fev[rtgrff::kMapForkStreams + 1] = {};
    void *pinned[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t pinned_cap[4] = {0, 0, 0, 0};
    int64_t launches = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // bracket the dominant kernel of the last call
    bool ev_valid = false;

    // ray cube {omega_pe, d/dx, d/dy, d/dz}
    rtgrff::DevBuf wcube;
    rtgrff::DevBuf pcube;            // cell-major polynomial form of wcube (8 float4 per cell), optional
    bool has_pcube = false;
    rtgrff::GridGeom wgeom{};
    bool has_wcube = false;

    // field cubes {ne, te, |B|, 0} and {bx, by, bz, 0}
    rtgrff::DevBuf fcube, bcube;
    rtgrff::GridGeom fgeom{};
    rtgrff::GridGeomF fgeomf{};
    bool has_fcube = false, has_bvec = false;

    // records of the last trace: positions SoA [rec][3][ray] f64, S [rec][ray] f64
    rtgrff::DevBuf rec_pos, rec_s;
    int64_t rec_n = 0, rec_rays = 0;
    bool rec_has_s = false;

    // samples of the last sample_traced: ne, te, b, ds, s float32 [rec][ray]; valid u8
    rtgrff::DevBuf smp_ne, smp_te, smp_b, smp_ds, smp_s, smp_valid;
    int64_t smp_n = 0, smp_rays = 0;

    // cubes resampled from a spherical model (rho, te, br, bt, bp as float64) before composition
    rtgrff::DevBuf slot[5];
    bool slot_set[5] = {false, false, false, false, false};
    int slot_nx = 0, slot_ny = 0, slot_nz = 0;
    double slot_geom[12] = {0};
    double slot_geoms[5][12] = {{0}};   // geometry each slot was resampled on (compose checks they agree)
    double slot_views[5][2] = {{0}};    // the view (b0, p) [deg] each slot was resampled with (compose turns B with it)
    bool stage_has_omega = false;    // `stage` still holds the float64 omega_pe of the last compose (rtgrff_export_cubes)

    // spherical model resident for the straight-LOS map (rtgrff_set_spherical_model): slot 0..4 = rho, te, br, bt, bp,
    // float32 data on the device, the node coordinates phi, lat, r on the host (uploaded with each map)
    rtgrff::DevBuf sph_data[5];
    std::vector<double> sph_nodes[5];
    int sph_n[5][3] = {{0}};
    double sph_scale[5] = {0};
    bool sph_set[5] = {false, false, false, false, false};

    // multi-GPU image gather (rtgrff_comm_*): an ncclComm_t behind a void*, NCCL loaded at run time
    void *comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    rtgrff::DevBuf gather_buf, image_buf;
    rtgrff::DevBuf slot_grids;       // x, y, z node coordinates of the slots' cube

    // scratch
    rtgrff::DevBuf in0, in1, in2, in3, out0, out1, out2, out3, out4, out5, stage, counters;
};
