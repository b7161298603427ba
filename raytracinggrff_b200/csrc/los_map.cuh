// Fused straight line-of-sight map for sm_100a: sample the resident spherical model along every pixel's straight
// LOS and advance the polarised transfer equation for every frequency in one kernel, nothing materialised.
//
// Equivalent to the reference chain
//   resample_MAS  (script/resampling_MAS_LOS.py:141-301): rho, te, br, bt, bp along the LOS, |B|
//   SyntheticFF   (script/synthetic_FF_map_single_thread.py:108-244): NaN filter, Parms packing, GET_MW, T_b
// where the staged drop-ins (los.resample_MAS + los.SyntheticFF) hold five float64 (N_pix, N_pix, N_z) arrays and a
// float64 (15, N_z, N_pix^2) Parms array: 16 GB at 512^2 x 400.
//
// The LOS does not depend on the frequency, and sampling a point of the spherical model (five 8-corner FP64 lookups,
// binary searches on up to five meshes, FP64 atan2 / acos) costs several voxel-frequency evaluations.  So a block
// owns a 4 x 8 pixel tile and a group of frequencies (one warp per frequency, lane = pixel): its threads sample a
// chunk of the tile's LOS samples once into shared memory, then every warp pushes the chunk through its own
// per-pixel RecordTransfer (fused_map.cuh: the same FP32 / FP64 voxel evaluation, between-voxel events and
// diagnostic accumulators as the ray-traced map).  More frequencies than one group: blockIdx.y, which re-samples.
#pragma once

#include "cube_builder.cuh"
#include "fused_map.cuh"

namespace rtgrff {

constexpr int kLosTileW = 4, kLosTileH = 8;        // pixels of a block's tile: one warp
constexpr int kLosMaxFreqGroup = 8;                 // frequencies (warps) per block
constexpr int kLosChunk = 32;                       // samples per LOS staged in shared memory at a time
constexpr int kLosSlots = 5;                        // rho, te, br, bt, bp

struct LosMapArgs {
    SphMesh var[kLosSlots];              // data and sizes; the node pointers are set in shared memory
    double scale[kLosSlots];
    const double *nodes;                 // phi, lat, r of every slot, one after the other
    int node_off[kLosSlots];             // where a slot's phi starts in `nodes` (lat, r follow)
    int n_nodes;
    const double *x, *y, *zc, *dz_cm;    // pixel columns, rows, cumulative z offsets [R_sun]; segment lengths [cm]
    int nx, ny, nz, tiles_x;
    double phi0_offset_rad, r_min, z_eps;
    const FreqC *freqs;                  // [n_freq], caller's order
    int n_freq, fg;                      // fg: frequencies per block (= warps)
    double area;
    int em_flag, s_max, grff64;
    double *tb, *vi;                     // [freq][ny][nx]
    double *diag;                        // [RTGRFF_N_DIAG][freq][ny][nx], the DIAG variants only
    unsigned long long *valid_samples;
    ViewRot view;                        // the observer's B0 / P (cube_builder.cuh)
};

// dynamic shared memory: FreqC[fg] | float ne, te, b, cth, sth [kLosChunk][32] | double nodes[n_nodes]
inline size_t los_map_smem(int fg, int n_nodes)
{
    return (size_t)fg * sizeof(FreqC) + (size_t)5 * kLosChunk * 32 * sizeof(float) + (size_t)n_nodes * sizeof(double);
}

// T_b and V/I as SyntheticFF converts GET_MW's output (script/synthetic_FF_map_single_thread.py:212-221): no epsilon
// in V/I (NaN where L + R = 0), no nan_to_num; a LOS without a valid sample is 0 / 0.
__device__ __forceinline__ void tb_vi_los(double IL, double IR, double nu, double area, bool any_valid, double &tb,
                                          double &vi)
{
    if (!any_valid) { tb = 0.0; vi = 0.0; return; }
    const double to_sfu = area / (kAu * kAu) / kSfu;
    const double l = IL * to_sfu, r = IR * to_sfu;
    const double conv = (1e-19 * 2.998e10 * 2.998e10 / (2.0 * 1.38065e-16 * nu * nu) / area) * (1.49599e13 * 1.49599e13);
    tb = (l + r) * conv;
    vi = (l - r) / (l + r);
}

// NEED_BETWEEN: gyroresonance on or theta from the B vector (BVEC); DIAG: the planes of rtgrff_render_map_diag;
// VIEW: a non-zero observer view (ViewRot, cube_builder.cuh)
template <bool BVEC, bool NEED_BETWEEN, bool DIAG, bool VIEW>
__global__ void __launch_bounds__(kLosMaxFreqGroup * 32, 2) los_map_kernel(const LosMapArgs a)
{
    extern __shared__ double smem_d[];
    FreqC *s_fq = reinterpret_cast<FreqC *>(smem_d);
    float *s_ne = reinterpret_cast<float *>(s_fq + a.fg);
    float *s_te = s_ne + kLosChunk * 32, *s_b = s_te + kLosChunk * 32;
    float *s_cth = s_b + kLosChunk * 32, *s_sth = s_cth + kLosChunk * 32;
    double *s_nodes = reinterpret_cast<double *>(s_sth + kLosChunk * 32);

    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nthr = blockDim.x;
    const int f = blockIdx.y * a.fg + w;
    const int tx = blockIdx.x % a.tiles_x, ty = blockIdx.x / a.tiles_x;
    for (int q = threadIdx.x; q < a.n_nodes; q += nthr) s_nodes[q] = a.nodes[q];
    if (lane == 0 && f < a.n_freq) s_fq[w] = a.freqs[f];
    SphMesh mesh[kLosSlots];
#pragma unroll
    for (int v = 0; v < kLosSlots; ++v) {
        mesh[v] = a.var[v];
        mesh[v].phi = s_nodes + a.node_off[v];
        mesh[v].lat = mesh[v].phi + a.var[v].np;
        mesh[v].r = mesh[v].lat + a.var[v].nt;
    }

    // this thread's pixel in the transfer phase
    const int pj = tx * kLosTileW + (lane % kLosTileW), pi = ty * kLosTileH + (lane / kLosTileW);
    const bool mine = f < a.n_freq && pi < a.ny && pj < a.nx;
    double px = 0.0, py = 0.0, pz0 = 0.0;
    if (mine) { px = a.x[pj]; py = a.y[pi]; pz0 = los_z0(px, py, a.z_eps); }
    const float pxf = (float)px, pyf = (float)py;

    RecordTransfer<NEED_BETWEEN, DIAG> tr;
    tr.init();
    float rmin = INFINITY;
    bool any_valid = false;
    unsigned int n_valid = 0;
    __syncthreads();

    for (int k0 = 0; k0 < a.nz; k0 += kLosChunk) {
        const int nk = min(kLosChunk, a.nz - k0);
        // --- sampling: sample s = (k - k0) * 32 + pixel lane, consecutive threads on neighbouring pixels ---
        for (int s = threadIdx.x; s < nk * 32; s += nthr) {
            const int l = s & 31, k = k0 + (s >> 5);
            const int j = tx * kLosTileW + (l % kLosTileW), i = ty * kLosTileH + (l / kLosTileW);
            float ne = nanf(""), te = 0.0f, b = 0.0f, cth = 6.123233995736766e-17f, sth = 1.0f;
            if (i < a.ny && j < a.nx) {
                const double x = a.x[j], y = a.y[i];
                const double z = los_z0(x, y, a.z_eps) + a.zc[k];
                double lon, lat, r;
                double mx = x, my = y, mz = z;      // the sample point in model-aligned axes
                if constexpr (VIEW) view_to_model(a.view, mx, my, mz);
                los_sph(mx, my, mz, a.phi0_offset_rad, lon, lat, r);
                if (r >= a.r_min) {
                    // the values resample_MAS stores, |B| in FP64 (los.py), SyntheticFF's NaN filter
                    const double rho = sample_spherical(mesh[0], lon, lat, r) * a.scale[0];
                    const double t = sample_spherical(mesh[1], lon, lat, r) * a.scale[1];
                    const double br = sample_spherical(mesh[2], lon, lat, r) * a.scale[2];
                    const double bt = sample_spherical(mesh[3], lon, lat, r) * a.scale[3];
                    const double bp = sample_spherical(mesh[4], lon, lat, r) * a.scale[4];
                    // numpy's sqrt(br**2 + bt**2 + bp**2): every operation rounded, no FMA
                    const double bm = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(br, br), __dmul_rn(bt, bt)), __dmul_rn(bp, bp)));
                    if (!isnan(rho) && !isnan(t) && !isnan(bm)) {
                        ne = (float)rho; te = (float)t; b = (float)bm;
                        if (BVEC && bm > 0.0) {
                            // theta between B and the propagation direction +z (towards the observer)
                            double bx, by, bz;
                            sph_to_view_b<VIEW>(a.view, x, y, z, br, bt, bp, bx, by, bz);
                            cth = (float)fmin(1.0, fmax(-1.0, bz / bm));
                            sth = (float)fmin(1.0, sqrt(bx * bx + by * by) / bm);
                        }
                        if (blockIdx.y == 0) ++n_valid;
                    }
                }
            }
            s_ne[s] = ne; s_te[s] = te; s_b[s] = b;
            if (BVEC) { s_cth[s] = cth; s_sth[s] = sth; }
        }
        __syncthreads();
        // --- transfer: Sun side first, as SyntheticFF hands the voxels to GET_MW ---
        if (mine) {
            const FreqC &fq = s_fq[w];
            for (int kk = 0; kk < nk; ++kk) {
                const int k = k0 + kk, s = kk * 32 + lane;
                float zf = 0.0f;
                if (DIAG) {
                    zf = (float)(pz0 + a.zc[k]);
                    rmin = fminf(rmin, diag_coord(pxf, pyf, zf).w);
                }
                const float ne = s_ne[s];
                if (isnan(ne)) continue;
                any_valid = true;
                const VoxLite v = {(float)a.dz_cm[k], s_te[s], ne, s_b[s], BVEC ? s_cth[s] : 6.123233995736766e-17f, 1.0f};
                tr.push(fq, v, BVEC ? s_sth[s] : 1.0f, a.em_flag, a.s_max, a.grff64 != 0, pxf, pyf, zf);
            }
        }
        __syncthreads();
    }
    if (mine) {
        const size_t plane = (size_t)a.ny * a.nx, o = (size_t)f * plane + (size_t)pi * a.nx + pj;
        double IL, IR, tb, vi;
        tr.result(IL, IR);
        tb_vi_los(IL, IR, s_fq[w].nu, a.area, any_valid, tb, vi);
        a.tb[o] = tb;
        a.vi[o] = vi;
        if constexpr (DIAG) tr.dg.write(IL, IR, rmin, a.diag + o, (size_t)a.n_freq * plane);
    }
    if (a.valid_samples && blockIdx.y == 0) {
        const unsigned int tot = __reduce_add_sync(0xffffffffu, n_valid);
        if (lane == 0 && tot) atomicAdd(a.valid_samples, (unsigned long long)tot);
    }
}

}  // namespace rtgrff
