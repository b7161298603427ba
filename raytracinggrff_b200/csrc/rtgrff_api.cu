// C-ABI of librtgrff_b200.so (declared in include/rtgrff.h).  Host-side staging + launches only;
// the kernels live in the .cuh files next to this one.
#include <stdarg.h>

#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "common.cuh"
#include "comm.cuh"
#include "cube_builder.cuh"
#include "fused_map.cuh"
#include "grff.cuh"
#include "image_ops.cuh"
#include "los_map.cuh"
#include "los_sampler.cuh"
#include "ray_integrator.cuh"
#include "trace_kernel.cuh"

namespace rtgrff {

thread_local char g_err[512] = "";

inline int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int DevBuf::reserve(size_t bytes)
{
    if (bytes <= cap) return RTGRFF_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        p = nullptr;
        return fail(e == cudaErrorMemoryAllocation ? RTGRFF_ENOMEM : RTGRFF_ECUDA, "cudaMalloc(%zu) -> %s", bytes,
                    cudaGetErrorString(e));
    }
    cap = bytes;
    return RTGRFF_OK;
}

void DevBuf::release()
{
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
}

static int geom_from(const double g[12], int nx, int ny, int nz, GridGeom &o)
{
    if (nx < 2 || ny < 2 || nz < 2) return fail(RTGRFF_EINVAL, "cube needs >= 2 points per axis (%d,%d,%d)", nx, ny, nz);
    if ((int64_t)nx * ny * nz >= (int64_t)1 << 31) return fail(RTGRFF_EINVAL, "cube larger than 2^31 voxels");
    for (int a = 0; a < 3; ++a)
        if (!(g[4 * a + 1] > 0.0) || !isfinite(g[4 * a + 1])) return fail(RTGRFF_EINVAL, "axis %d has invalid spacing", a);
    o.nx = nx; o.ny = ny; o.nz = nz;
    o.x0 = g[0]; o.idx = 1.0 / g[1]; o.xl = g[2];
    o.y0 = g[4]; o.idy = 1.0 / g[5]; o.yl = g[6];
    o.z0 = g[8]; o.idz = 1.0 / g[9]; o.zl = g[10];
    return RTGRFF_OK;
}

// The float32 view of a geometry geom_from accepted, for the samplers.
static GridGeomF geomf_from(const double g[12], int nx, int ny, int nz)
{
    GridGeomF f;
    f.nx = nx; f.ny = ny; f.nz = nz;
    f.x0 = (float)g[0]; f.y0 = (float)g[4]; f.z0 = (float)g[8];
    f.idx = (float)(1.0 / g[1]); f.idy = (float)(1.0 / g[5]); f.idz = (float)(1.0 / g[9]);
    f.fxl = (float)(nx - 1); f.fyl = (float)(ny - 1); f.fzl = (float)(nz - 1);
    return f;
}

// The node coordinates of a spherical mesh must ascend strictly along every axis.
static int check_ascending_nodes(const double *phi, int np, const double *lat, int nt, const double *r, int nr)
{
    for (int i = 1; i < np; ++i) if (!(phi[i] > phi[i - 1])) return fail(RTGRFF_EINVAL, "phi nodes must ascend");
    for (int i = 1; i < nt; ++i) if (!(lat[i] > lat[i - 1])) return fail(RTGRFF_EINVAL, "latitude nodes must ascend");
    for (int i = 1; i < nr; ++i) if (!(r[i] > r[i - 1])) return fail(RTGRFF_EINVAL, "radius nodes must ascend");
    return RTGRFF_OK;
}

// sin and cos of an angle in degrees, exact at multiples of 90 deg (so that P = 90 is an exact quarter turn)
static void sincos_deg(double deg, double &s, double &c)
{
    const double q = deg / 90.0;
    if (q == floor(q) && fabs(q) < 1e15) {
        const int k = (int)(((long long)q % 4 + 4) % 4);
        s = (k == 1) ? 1.0 : (k == 3) ? -1.0 : 0.0;
        c = (k == 0) ? 1.0 : (k == 2) ? -1.0 : 0.0;
        return;
    }
    s = sin(deg * M_PI / 180.0);
    c = cos(deg * M_PI / 180.0);
}

// The observer's view (include/rtgrff.h, "Observer view"): finite angles, |B0| <= 90 deg.  B0 = P = 0 leaves the
// rotation off: the launches pick the VIEW = false kernels, the fixed equatorial view's code.
static int view_from(double b0_deg, double p_deg, ViewRot &v)
{
    if (!isfinite(b0_deg) || !isfinite(p_deg)) return fail(RTGRFF_EINVAL, "view angles must be finite (b0 %g, p %g)", b0_deg, p_deg);
    if (fabs(b0_deg) > 90.0) return fail(RTGRFF_EINVAL, "|b0| must be <= 90 deg (b0 %g)", b0_deg);
    v.on = (b0_deg != 0.0 || p_deg != 0.0) ? 1 : 0;
    sincos_deg(b0_deg, v.sb, v.cb);
    sincos_deg(p_deg, v.sp, v.cp);
    return RTGRFF_OK;
}

static RayCube ray_cube_of(const rtgrff_ctx *c)
{
    RayCube r;
    const GridGeom &g = c->wgeom;
    r.c = c->wcube.as<float4>();
    r.pc = c->has_pcube ? c->pcube.as<float4>() : nullptr;
    r.nx = g.nx; r.ny = g.ny; r.nz = g.nz;
    r.sy = g.nz; r.sx = g.ny * g.nz;
    r.x0 = g.x0; r.y0 = g.y0; r.z0 = g.z0;
    r.xl = g.xl; r.yl = g.yl; r.zl = g.zl;
    r.idx = g.idx; r.idy = g.idy; r.idz = g.idz;
    return r;
}

// Every entry point runs on the context's device and puts the caller's current device back on
// exit: a rank that works on cuda:k must not find its thread switched to another GPU after a call.
struct DeviceGuard {
    int prev = -1;
    bool restore = false;
    ~DeviceGuard()
    {
        if (restore) cudaSetDevice(prev);
    }
    int enter(const rtgrff_ctx *c)
    {
        if (!c) return fail(RTGRFF_EINVAL, "null context");
        return enter_device(c->device);
    }
    int enter_device(int device)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) {
            RT_CUDA(cudaSetDevice(device));
            restore = prev >= 0;
        }
        return RTGRFF_OK;
    }
};
#define RT_USE(c)       \
    DeviceGuard guard__; \
    RT_TRY(guard__.enter(c))

static int h2d(rtgrff_ctx *c, DevBuf &b, const void *src, size_t bytes)
{
    RT_TRY(b.reserve(bytes ? bytes : 1));
    if (bytes) RT_CUDA(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return RTGRFF_OK;
}

static int d2h(rtgrff_ctx *c, void *dst, const void *src, size_t bytes)
{
    if (bytes) RT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    return RTGRFF_OK;
}

// ---- chunked host <-> device pipelines -----------------------------------------------------------
// The reference-facing entry points take pageable host arrays (numpy).  cudaMemcpyAsync on pageable
// memory is staged by the driver and serialises with everything else (config 1: 0.45 ms of kernel
// inside 93 ms of copies).  Large calls therefore go through pinned bounce buffers in chunks: the
// host packs chunk k+1 and unpacks chunk k-1 with a few threads while the DMA engines move chunk k
// in both directions (H2D on the compute stream, D2H on the copy stream) and the kernel runs on it.
static int pipeline_default()
{
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("RTGRFF_PIPELINE");   // 0: one pageable copy each way, the kernel bracketed alone by ev0/ev1
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v;
}

static int host_threads()
{
    static int v = 0;
    if (v == 0) {
        const char *e = getenv("RTGRFF_HOST_THREADS");
        int n = e ? atoi(e) : 0;
        if (n <= 0) {
            n = (int)std::thread::hardware_concurrency();
            n = n >= 8 ? (3 * n) / 4 : (n >= 4 ? n / 2 : 1);   // leave cores to the caller's own threads
        }
        v = n > 16 ? 16 : n;
    }
    return v;
}

// memcpy split over a few persistent worker threads (one thread saturates neither the memory channels nor,
// for fresh numpy output arrays, the page-fault path; spawning threads per copy costs as much as a small copy)
class CopyPool {
public:
    explicit CopyPool(int n)
    {
        for (int t = 0; t < n; ++t) workers_.emplace_back([this] { run(); });
    }
    ~CopyPool()
    {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    int size() const { return (int)workers_.size(); }
    // the calling thread takes a share too and returns when every piece is done
    void copy(void *dst, const void *src, size_t bytes, int parts)
    {
        const size_t per = ((bytes / parts) + 4095) & ~(size_t)4095;
        int posted = 0;
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (int t = 1; t < parts; ++t) {
                const size_t o = per * t;
                if (o >= bytes) break;
                tasks_.push_back(Task{(char *)dst + o, (const char *)src + o, std::min(per, bytes - o)});
                ++posted;
            }
            pending_ += posted;
        }
        cv_.notify_all();
        memcpy(dst, src, std::min(per, bytes));
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this] { return pending_ == 0; });
    }

private:
    struct Task { char *dst; const char *src; size_t len; };
    void run()
    {
        for (;;) {
            Task t;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this] { return stop_ || !tasks_.empty(); });
                if (stop_ && tasks_.empty()) return;
                t = tasks_.back();
                tasks_.pop_back();
            }
            memcpy(t.dst, t.src, t.len);
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (--pending_ == 0) done_.notify_all();
            }
        }
    }
    std::vector<std::thread> workers_;
    std::vector<Task> tasks_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    int pending_ = 0;
    bool stop_ = false;
};

static std::mutex g_copy_mu;      // one copy at a time through the pool (contexts of several host threads share it)

static void parallel_copy(void *dst, const void *src, size_t bytes)
{
    const int nt = host_threads();
    // at least 256 KB per thread: the workers are persistent, the hand-over is a condition-variable wake-up, and the
    // unpack into fresh numpy arrays is bound by page faults per thread, so it wants every thread it can get
    const int parts = (int)std::min<size_t>((size_t)nt, bytes / ((size_t)256 << 10));
    if (parts <= 1) {
        memcpy(dst, src, bytes);
        return;
    }
    static CopyPool *pool = new CopyPool(nt - 1);      // lives for the process: workers sleep on a condition variable
    std::lock_guard<std::mutex> lk(g_copy_mu);
    pool->copy(dst, src, bytes, parts);
}

static int pin_reserve(rtgrff_ctx *c, int idx, size_t bytes)
{
    if (bytes <= c->pinned_cap[idx]) return RTGRFF_OK;
    if (c->pinned[idx]) cudaFreeHost(c->pinned[idx]);
    c->pinned[idx] = nullptr;
    c->pinned_cap[idx] = 0;
    cudaError_t e = cudaMallocHost(&c->pinned[idx], bytes);
    if (e != cudaSuccess) {
        c->pinned[idx] = nullptr;
        return fail(RTGRFF_ENOMEM, "cudaMallocHost(%zu) -> %s", bytes, cudaGetErrorString(e));
    }
    c->pinned_cap[idx] = bytes;
    return RTGRFF_OK;
}

static bool is_pinned_host(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

// Large device -> host copy: straight DMA when the destination is page-locked, else 32 MB chunks
// through the two pinned output bounce buffers, the host memcpy of one chunk overlapping the DMA of
// the next.  Waits for the context's stream first and returns with the data in place.
static int d2h_large(rtgrff_ctx *c, void *dst, const void *src, size_t bytes)
{
    if (!bytes) return RTGRFF_OK;
    if (is_pinned_host(dst) || bytes < ((size_t)8 << 20) || !c->pipeline) {
        RT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
        RT_CUDA(cudaStreamSynchronize(c->stream));
        return RTGRFF_OK;
    }
    const size_t chunk = (size_t)32 << 20;
    for (int q = 0; q < 2; ++q) RT_TRY(pin_reserve(c, 2 + q, chunk));
    cudaEvent_t *ev_out = c->chunk_ev + 4;
    const size_t n_chunk = (bytes + chunk - 1) / chunk;
    for (size_t k = 0; k <= n_chunk; ++k) {
        if (k < n_chunk) {
            const size_t o = k * chunk, len = std::min(chunk, bytes - o);
            RT_CUDA(cudaMemcpyAsync(c->pinned[2 + (k & 1)], (const char *)src + o, len, cudaMemcpyDeviceToHost, c->stream));
            RT_CUDA(cudaEventRecord(ev_out[k & 1], c->stream));
        }
        if (k >= 1) {
            const size_t o = (k - 1) * chunk, len = std::min(chunk, bytes - o);
            RT_CUDA(cudaEventSynchronize(ev_out[(k - 1) & 1]));
            parallel_copy((char *)dst + o, c->pinned[2 + ((k - 1) & 1)], len);
        }
    }
    return RTGRFF_OK;
}

// The mirror image for uploads; returns when the source buffer may be reused (not when the DMA is done).
static int h2d_large(rtgrff_ctx *c, void *dst, const void *src, size_t bytes)
{
    if (!bytes) return RTGRFF_OK;
    if (is_pinned_host(src) || bytes < ((size_t)8 << 20) || !c->pipeline) {
        RT_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
        return RTGRFF_OK;
    }
    const size_t chunk = (size_t)32 << 20;
    for (int q = 0; q < 2; ++q) RT_TRY(pin_reserve(c, q, chunk));
    cudaEvent_t *ev_in = c->chunk_ev;
    const size_t n_chunk = (bytes + chunk - 1) / chunk;
    for (size_t k = 0; k < n_chunk; ++k) {
        const size_t o = k * chunk, len = std::min(chunk, bytes - o);
        if (k >= 2) RT_CUDA(cudaEventSynchronize(ev_in[k & 1]));
        parallel_copy(c->pinned[k & 1], (const char *)src + o, len);
        RT_CUDA(cudaMemcpyAsync((char *)dst + o, c->pinned[k & 1], len, cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(cudaEventRecord(ev_in[k & 1], c->stream));
    }
    // the bounce buffers are reused by the next call: drain them before returning
    RT_CUDA(cudaEventSynchronize(ev_in[(n_chunk - 1) & 1]));
    if (n_chunk >= 2) RT_CUDA(cudaEventSynchronize(ev_in[(n_chunk - 2) & 1]));
    return RTGRFF_OK;
}

constexpr size_t kPipeMinBytes = (size_t)16 << 20;    // below this a call is one plain copy each way
constexpr size_t kPipeChunkBytes = (size_t)32 << 20;  // bounce-buffer size per direction and stage

static int launched(rtgrff_ctx *c, const char *what)
{
    c->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RTGRFF_ECUDA, "launch %s -> %s", what, cudaGetErrorString(e));
    return RTGRFF_OK;
}

// Cell-major polynomial cube for the FP32 stepper: 128 B per cell (8x the node cube).  Built when it
// fits in a third of the free device memory (RTGRFF_POLY_CUBE=0 disables it, =1 forces it); the
// stepper falls back to differencing the node cube on the fly without it.
static int build_poly_cube(rtgrff_ctx *c, int nx, int ny, int nz)
{
    c->has_pcube = false;
    const char *e = getenv("RTGRFF_POLY_CUBE");
    if (e && e[0] == '0') return RTGRFF_OK;
    const size_t bytes = (size_t)nx * ny * nz * 8 * sizeof(float4);
    if (bytes > c->pcube.cap && !(e && e[0] == '1')) {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || bytes > free_b / 3) return RTGRFF_OK;
    }
    RT_TRY(c->pcube.reserve(bytes));
    build_poly_cube_kernel<<<blocks_for((int64_t)nx * ny * nz, 256), 256, 0, c->stream>>>(c->wcube.as<float4>(),
                                                                                         c->pcube.as<float4>(), nx, ny, nz);
    RT_TRY(launched(c, "build_poly_cube_kernel"));
    c->has_pcube = true;
    return RTGRFF_OK;
}


static int cs_every_step()
{
    // RTGRFF_CS_EVERY_STEP=1: trace the two cross-section rays at every step like the reference does,
    // although only the ratio of a recorded step is ever output (A/B switch; results are identical).
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("RTGRFF_CS_EVERY_STEP");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v;
}

static int grff64()
{
    // RTGRFF_GRFF64=1: the per-ray kernels evaluate every voxel in FP64 (A/B switch; default: float32 where
    // well conditioned, see grff_fast.cuh)
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("RTGRFF_GRFF64");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v;
}

}  // namespace rtgrff

using namespace rtgrff;

extern "C" {

const char *rtgrff_version(void) { return "rtgrff_b200 0.1.0 sm_100a"; }
const char *rtgrff_last_error(void) { return g_err; }

int rtgrff_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(RTGRFF_ECUDA, "cudaGetDeviceCount -> %s", cudaGetErrorString(e));
    return n;
}

static int ctx_create(int device, void *stream, bool caller_stream, rtgrff_ctx **out)
{
    if (!out) return fail(RTGRFF_EINVAL, "out is null");
    *out = nullptr;
    int n = 0;
    RT_CUDA(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(RTGRFF_EINVAL, "device %d out of range (%d visible)", device, n);
    DeviceGuard guard;
    RT_TRY(guard.enter_device(device));
    rtgrff_ctx *c = new (std::nothrow) rtgrff_ctx();
    if (!c) return fail(RTGRFF_ENOMEM, "out of host memory");
    c->device = device;
    c->pipeline = pipeline_default();
    c->grff64 = grff64();
    cudaError_t e = cudaSuccess;
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) == cudaSuccess) {
        c->sm_count = prop.multiProcessorCount;
        if (caller_stream) {
            c->stream = (cudaStream_t)stream;      // including 0: the legacy default stream
        } else if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) == cudaSuccess) {
            c->own_stream = true;
        }
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    for (int q = 0; q < 6 && e == cudaSuccess; ++q) e = cudaEventCreateWithFlags(&c->chunk_ev[q], cudaEventDisableTiming);
    if (e != cudaSuccess) {
        rtgrff_ctx_destroy(c);
        return fail(RTGRFF_ECUDA, "rtgrff_ctx_create -> %s", cudaGetErrorString(e));
    }
    *out = c;
    return RTGRFF_OK;
}

int rtgrff_ctx_create(int device, void *stream, rtgrff_ctx **out)
{
    return ctx_create(device, stream, stream != nullptr, out);
}

int rtgrff_ctx_create_on_stream(int device, void *stream, rtgrff_ctx **out)
{
    return ctx_create(device, stream, true, out);
}

int rtgrff_current_device(void)
{
    int d = -1;
    cudaError_t e = cudaGetDevice(&d);
    if (e != cudaSuccess) return fail(RTGRFF_ECUDA, "cudaGetDevice -> %s", cudaGetErrorString(e));
    return d;
}

int rtgrff_ctx_destroy(rtgrff_ctx *c)
{
    if (!c) return RTGRFF_OK;
    DeviceGuard guard;
    guard.enter_device(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->comm) {
        NcclApi *n = nccl_api();
        if (n) n->CommDestroy((NcclComm)c->comm);
        c->comm = nullptr;
    }
    DevBuf *bufs[] = {&c->wcube, &c->pcube, &c->fcube, &c->bcube, &c->rec_pos, &c->rec_s, &c->smp_ne, &c->smp_te, &c->smp_b,
                      &c->smp_ds, &c->smp_s, &c->smp_valid, &c->in0, &c->in1, &c->in2, &c->in3, &c->out0, &c->out1,
                      &c->out2, &c->out3, &c->out4, &c->out5, &c->stage, &c->counters, &c->gather_buf, &c->image_buf};
    for (DevBuf *b : bufs) b->release();
    for (DevBuf &b : c->slot) b.release();
    for (DevBuf &b : c->sph_data) b.release();
    c->slot_grids.release();
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    for (cudaEvent_t &e : c->chunk_ev)
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t &e : c->fev)
        if (e) cudaEventDestroy(e);
    for (cudaStream_t &q : c->fstream)
        if (q) cudaStreamDestroy(q);
    for (void *&h : c->pinned)
        if (h) cudaFreeHost(h);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return RTGRFF_OK;
}

int rtgrff_ctx_synchronize(rtgrff_ctx *c)
{
    RT_USE(c);
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_ctx_set_grff64(rtgrff_ctx *c, int enabled)
{
    if (!c) return fail(RTGRFF_EINVAL, "null context");
    c->grff64 = enabled ? 1 : 0;
    return RTGRFF_OK;
}

int rtgrff_ctx_set_pipeline(rtgrff_ctx *c, int enabled)
{
    if (!c) return fail(RTGRFF_EINVAL, "null context");
    c->pipeline = enabled ? 1 : 0;
    return RTGRFF_OK;
}

int64_t rtgrff_ctx_launch_count(const rtgrff_ctx *c) { return c ? c->launches : 0; }

double rtgrff_ctx_last_kernel_ms(rtgrff_ctx *c)
{
    if (!c || !c->ev_valid) return -1.0;
    float ms = -1.0f;
    DeviceGuard guard;
    if (guard.enter_device(c->device) != RTGRFF_OK) return -1.0;
    if (cudaEventSynchronize(c->ev1) != cudaSuccess) return -1.0;
    if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) != cudaSuccess) return -1.0;
    return (double)ms;
}

int rtgrff_set_omega_cube(rtgrff_ctx *c, const double *omega_pe, int nx, int ny, int nz, const double geom[12],
                          int on_device)
{
    RT_USE(c);
    if (!omega_pe || !geom) return fail(RTGRFF_EINVAL, "null argument");
    GridGeom g;
    RT_TRY(geom_from(geom, nx, ny, nz, g));
    const size_t nvox = (size_t)nx * ny * nz;
    const double *src = omega_pe;
    if (!on_device) {
        RT_TRY(c->stage.reserve(nvox * sizeof(double)));
        RT_TRY(h2d_large(c, c->stage.p, omega_pe, nvox * sizeof(double)));
        src = c->stage.as<double>();
    }
    c->stage_has_omega = !on_device;
    RT_TRY(c->wcube.reserve(nvox * sizeof(float4)));
    build_ray_cube_kernel<<<blocks_for((int64_t)nvox, 256), 256, 0, c->stream>>>(src, c->wcube.as<float4>(), nx, ny, nz,
                                                                                 geom[3], geom[7], geom[11]);
    RT_TRY(launched(c, "build_ray_cube_kernel"));
    RT_TRY(build_poly_cube(c, nx, ny, nz));
    c->wgeom = g;
    c->has_wcube = true;
    RT_CUDA(cudaStreamSynchronize(c->stream));   // the host buffer may be reused by the caller
    return RTGRFF_OK;
}

int rtgrff_set_field_cubes(rtgrff_ctx *c, const float *ne, const float *te, const float *b, const float *bx,
                           const float *by, const float *bz, int nx, int ny, int nz, const double geom[12])
{
    RT_USE(c);
    if (!ne || !te || !b || !geom) return fail(RTGRFF_EINVAL, "null argument");
    const bool bvec = bx && by && bz;
    if ((bx || by || bz) && !bvec) return fail(RTGRFF_EINVAL, "bx, by, bz must be given together");
    GridGeom g;
    RT_TRY(geom_from(geom, nx, ny, nz, g));
    const size_t nvox = (size_t)nx * ny * nz, fb = nvox * sizeof(float);
    RT_TRY(c->stage.reserve(3 * fb));
    c->stage_has_omega = false;
    float *s0 = c->stage.as<float>(), *s1 = s0 + nvox, *s2 = s1 + nvox;
    RT_TRY(c->fcube.reserve(nvox * sizeof(float4)));
    RT_TRY(h2d_large(c, s0, ne, fb));
    RT_TRY(h2d_large(c, s1, te, fb));
    RT_TRY(h2d_large(c, s2, b, fb));
    interleave3_kernel<<<blocks_for((int64_t)nvox, 256), 256, 0, c->stream>>>(s0, s1, s2, c->fcube.as<float4>(), (int64_t)nvox);
    RT_TRY(launched(c, "interleave3_kernel"));
    if (bvec) {
        RT_TRY(c->bcube.reserve(nvox * sizeof(float4)));
        RT_TRY(h2d_large(c, s0, bx, fb));
        RT_TRY(h2d_large(c, s1, by, fb));
        RT_TRY(h2d_large(c, s2, bz, fb));
        interleave3_kernel<<<blocks_for((int64_t)nvox, 256), 256, 0, c->stream>>>(s0, s1, s2, c->bcube.as<float4>(), (int64_t)nvox);
        RT_TRY(launched(c, "interleave3_kernel"));
    }
    c->fgeom = g;
    c->fgeomf = geomf_from(geom, nx, ny, nz);
    c->has_fcube = true;
    c->has_bvec = bvec;
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_resample_spherical(rtgrff_ctx *c, int slot, const float *data, const double *phi, const double *lat,
                              const double *r, int np, int nt, int nr, const double *x_grid, const double *y_grid,
                              const double *z_grid, int nx, int ny, int nz, const double geom[12],
                              double phi0_offset_deg, double r_min, double scale, double fill, int fill_nonfinite,
                              double *out)
{
    return rtgrff_resample_spherical_view(c, slot, data, phi, lat, r, np, nt, nr, x_grid, y_grid, z_grid, nx, ny, nz, geom,
                                          phi0_offset_deg, 0.0, 0.0, r_min, scale, fill, fill_nonfinite, out);
}

int rtgrff_resample_spherical_view(rtgrff_ctx *c, int slot, const float *data, const double *phi, const double *lat,
                                   const double *r, int np, int nt, int nr, const double *x_grid, const double *y_grid,
                                   const double *z_grid, int nx, int ny, int nz, const double geom[12],
                                   double phi0_offset_deg, double b0_deg, double p_deg, double r_min, double scale,
                                   double fill, int fill_nonfinite, double *out)
{
    RT_USE(c);
    if (slot < 0 || slot > 4) return fail(RTGRFF_EINVAL, "slot %d out of range 0..4", slot);
    if (!data || !phi || !lat || !r || !geom || !x_grid || !y_grid || !z_grid) return fail(RTGRFF_EINVAL, "null argument");
    if (np < 2 || nt < 2 || nr < 2) return fail(RTGRFF_EINVAL, "spherical mesh needs >= 2 nodes per axis");
    ViewRot view;
    RT_TRY(view_from(b0_deg, p_deg, view));
    GridGeom g;
    RT_TRY(geom_from(geom, nx, ny, nz, g));
    RT_TRY(check_ascending_nodes(phi, np, lat, nt, r, nr));
    if (c->slot_nx && (c->slot_nx != nx || c->slot_ny != ny || c->slot_nz != nz))
        for (bool &b : c->slot_set) b = false;           // a new cube shape invalidates the other slots
    const size_t nvox = (size_t)nx * ny * nz, nd = (size_t)np * nt * nr;
    RT_TRY(h2d(c, c->in0, data, nd * sizeof(float)));
    RT_TRY(c->in1.reserve((size_t)(np + nt + nr) * sizeof(double)));
    double *ax = c->in1.as<double>();
    RT_CUDA(cudaMemcpyAsync(ax, phi, np * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    RT_CUDA(cudaMemcpyAsync(ax + np, lat, nt * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    RT_CUDA(cudaMemcpyAsync(ax + np + nt, r, nr * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    RT_TRY(c->slot[slot].reserve(nvox * sizeof(double)));
    RT_TRY(c->slot_grids.reserve((size_t)(nx + ny + nz) * sizeof(double)));
    double *gx = c->slot_grids.as<double>();
    RT_CUDA(cudaMemcpyAsync(gx, x_grid, nx * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    RT_CUDA(cudaMemcpyAsync(gx + nx, y_grid, ny * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    RT_CUDA(cudaMemcpyAsync(gx + nx + ny, z_grid, nz * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ResampleArgs a;
    a.mesh.data = c->in0.as<float>();
    a.mesh.phi = ax; a.mesh.lat = ax + np; a.mesh.r = ax + np + nt;
    a.mesh.np = np; a.mesh.nt = nt; a.mesh.nr = nr;
    a.nx = nx; a.ny = ny; a.nz = nz;
    a.xg = gx; a.yg = gx + nx; a.zg = gx + nx + ny;
    a.phi0_offset_rad = phi0_offset_deg * M_PI / 180.0;
    a.r_min = r_min; a.scale = scale; a.fill = fill; a.fill_nonfinite = fill_nonfinite;
    a.view = view;
    a.out = c->slot[slot].as<double>();
    unsigned int blocks = blocks_for((int64_t)nvox, 256);
    const unsigned int cap = (unsigned int)c->sm_count * 32;
    if (blocks > cap) blocks = cap;
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    if (view.on) resample_spherical_kernel<true><<<blocks, 256, 0, c->stream>>>(a);
    else resample_spherical_kernel<false><<<blocks, 256, 0, c->stream>>>(a);
    RT_TRY(launched(c, "resample_spherical_kernel"));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    if (out) RT_TRY(d2h(c, out, c->slot[slot].p, nvox * sizeof(double)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    c->slot_set[slot] = true;
    c->slot_nx = nx; c->slot_ny = ny; c->slot_nz = nz;
    memcpy(c->slot_geom, geom, sizeof(c->slot_geom));
    memcpy(c->slot_geoms[slot], geom, sizeof(c->slot_geom));
    c->slot_views[slot][0] = b0_deg; c->slot_views[slot][1] = p_deg;
    return RTGRFF_OK;
}

int rtgrff_sample_spherical_los(rtgrff_ctx *c, const float *data, const double *phi, const double *lat, const double *r,
                                int np, int nt, int nr, const double *x, const double *y, const double *zc, int nx,
                                int ny, int nz, double phi0_offset_deg, double r_min, double scale, double z_eps,
                                double *out)
{
    return rtgrff_sample_spherical_los_view(c, data, phi, lat, r, np, nt, nr, x, y, zc, nx, ny, nz, phi0_offset_deg, 0.0,
                                            0.0, r_min, scale, z_eps, out);
}

int rtgrff_sample_spherical_los_view(rtgrff_ctx *c, const float *data, const double *phi, const double *lat,
                                     const double *r, int np, int nt, int nr, const double *x, const double *y,
                                     const double *zc, int nx, int ny, int nz, double phi0_offset_deg, double b0_deg,
                                     double p_deg, double r_min, double scale, double z_eps, double *out)
{
    RT_USE(c);
    if (!data || !phi || !lat || !r || !x || !y || !zc || !out) return fail(RTGRFF_EINVAL, "null argument");
    if (np < 2 || nt < 2 || nr < 2 || nx < 1 || ny < 1 || nz < 1) return fail(RTGRFF_EINVAL, "bad sizes");
    ViewRot view;
    RT_TRY(view_from(b0_deg, p_deg, view));
    RT_TRY(check_ascending_nodes(phi, np, lat, nt, r, nr));
    const size_t total = (size_t)nx * ny * nz, nd = (size_t)np * nt * nr;
    RT_TRY(h2d(c, c->in0, data, nd * sizeof(float)));
    RT_TRY(c->in1.reserve((size_t)(np + nt + nr + nx + ny + nz) * sizeof(double)));
    double *ax = c->in1.as<double>();
    const double *src[6] = {phi, lat, r, x, y, zc};
    const int len[6] = {np, nt, nr, nx, ny, nz};
    double *dst[6];
    size_t o = 0;
    for (int q = 0; q < 6; ++q) {
        dst[q] = ax + o;
        RT_CUDA(cudaMemcpyAsync(dst[q], src[q], len[q] * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        o += len[q];
    }
    RT_TRY(c->out0.reserve(total * sizeof(double)));
    LosArgs a;
    a.mesh.data = c->in0.as<float>();
    a.mesh.phi = dst[0]; a.mesh.lat = dst[1]; a.mesh.r = dst[2];
    a.mesh.np = np; a.mesh.nt = nt; a.mesh.nr = nr;
    a.x = dst[3]; a.y = dst[4]; a.zc = dst[5];
    a.nx = nx; a.ny = ny; a.nz = nz;
    a.phi0_offset_rad = phi0_offset_deg * M_PI / 180.0;
    a.r_min = r_min; a.scale = scale; a.z_eps = z_eps;
    a.view = view;
    a.out = c->out0.as<double>();
    unsigned int blocks = blocks_for((int64_t)total, 256);
    const unsigned int cap = (unsigned int)c->sm_count * 32;
    if (blocks > cap) blocks = cap;
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    if (view.on) los_spherical_kernel<true><<<blocks, 256, 0, c->stream>>>(a);
    else los_spherical_kernel<false><<<blocks, 256, 0, c->stream>>>(a);
    RT_TRY(launched(c, "los_spherical_kernel"));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    RT_TRY(d2h(c, out, c->out0.p, total * sizeof(double)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_compose_cubes(rtgrff_ctx *c, int want_bvec)
{
    RT_USE(c);
    for (int s = 0; s < 5; ++s)
        if (!c->slot_set[s]) return fail(RTGRFF_ENOCUBE, "spherical slot %d (0 rho, 1 te, 2 br, 3 bt, 4 bp) is not set", s);
    const int nx = c->slot_nx, ny = c->slot_ny, nz = c->slot_nz;
    const double *geom = c->slot_geom;
    for (int s = 0; s < 5; ++s)
        if (memcmp(c->slot_geoms[s], geom, sizeof(c->slot_geom)) != 0)
            return fail(RTGRFF_EINVAL, "spherical slot %d was resampled on a different cube geometry than the last one", s);
    for (int s = 1; s < 5; ++s)
        if (memcmp(c->slot_views[s], c->slot_views[0], sizeof(c->slot_views[0])) != 0)
            return fail(RTGRFF_EINVAL, "spherical slot %d was resampled with view (b0 %g, p %g), slot 0 with (b0 %g, p %g)",
                        s, c->slot_views[s][0], c->slot_views[s][1], c->slot_views[0][0], c->slot_views[0][1]);
    ViewRot view;
    RT_TRY(view_from(c->slot_views[0][0], c->slot_views[0][1], view));
    GridGeom g;
    RT_TRY(geom_from(geom, nx, ny, nz, g));
    const size_t nvox = (size_t)nx * ny * nz;
    RT_TRY(c->stage.reserve(nvox * sizeof(double)));
    RT_TRY(c->fcube.reserve(nvox * sizeof(float4)));
    if (want_bvec) RT_TRY(c->bcube.reserve(nvox * sizeof(float4)));
    RT_TRY(c->wcube.reserve(nvox * sizeof(float4)));
    ComposeArgs a;
    a.ne = c->slot[0].as<double>(); a.te = c->slot[1].as<double>();
    a.br = c->slot[2].as<double>(); a.bt = c->slot[3].as<double>(); a.bp = c->slot[4].as<double>();
    a.nx = nx; a.ny = ny; a.nz = nz;
    a.xg = c->slot_grids.as<double>(); a.yg = a.xg + nx; a.zg = a.yg + ny;
    a.omega_pe = c->stage.as<double>();
    a.fcube = c->fcube.as<float4>();
    a.bcube = want_bvec ? c->bcube.as<float4>() : nullptr;
    a.view = view;
    unsigned int blocks = blocks_for((int64_t)nvox, 256);
    if (view.on) compose_cubes_kernel<true><<<blocks, 256, 0, c->stream>>>(a);
    else compose_cubes_kernel<false><<<blocks, 256, 0, c->stream>>>(a);
    RT_TRY(launched(c, "compose_cubes_kernel"));
    build_ray_cube_kernel<<<blocks, 256, 0, c->stream>>>(c->stage.as<double>(), c->wcube.as<float4>(), nx, ny, nz,
                                                          geom[3], geom[7], geom[11]);
    RT_TRY(launched(c, "build_ray_cube_kernel"));
    RT_TRY(build_poly_cube(c, nx, ny, nz));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    c->wgeom = g; c->fgeom = g;
    c->fgeomf = geomf_from(geom, nx, ny, nz);
    c->has_wcube = true; c->has_fcube = true; c->has_bvec = want_bvec != 0;
    c->stage_has_omega = true;
    return RTGRFF_OK;
}

int rtgrff_trace(rtgrff_ctx *c, int64_t n_rays, const double *x_start, const double *y_start, const double *z_start,
                 const double *kvec, double freq_hz, double dt, int64_t n_steps, int64_t record_stride, int trace_cs,
                 double perturb_ratio, int s_mode, double *r_record, double *s_record, int64_t *active_steps)
{
    RT_USE(c);
    if (!c->has_wcube) return fail(RTGRFF_ENOCUBE, "rtgrff_set_omega_cube has not been called");
    if (n_rays < 0 || n_steps < 0 || record_stride < 1) return fail(RTGRFF_EINVAL, "bad n_rays/n_steps/record_stride");
    if (n_rays > 0 && (!x_start || !y_start || !z_start)) return fail(RTGRFF_EINVAL, "null start arrays");
    const int64_t n_rec = n_steps > 0 ? (n_steps + record_stride - 1) / record_stride : 0;
    c->rec_n = n_rec; c->rec_rays = n_rays; c->rec_has_s = trace_cs != 0;
    if (active_steps) *active_steps = 0;
    if (n_rays == 0 || n_rec == 0) return RTGRFF_OK;
    const size_t nb = (size_t)n_rays * sizeof(double);
    RT_TRY(h2d(c, c->in0, x_start, nb));
    RT_TRY(h2d(c, c->in1, y_start, nb));
    RT_TRY(h2d(c, c->in2, z_start, nb));
    if (kvec) RT_TRY(h2d(c, c->in3, kvec, 3 * nb));
    RT_TRY(c->rec_pos.reserve((size_t)n_rec * 3 * nb));
    if (trace_cs) RT_TRY(c->rec_s.reserve((size_t)n_rec * nb));
    RT_TRY(c->counters.reserve(64));
    RT_CUDA(cudaMemsetAsync(c->counters.p, 0, 64, c->stream));

    TraceArgs a;
    a.cube = ray_cube_of(c);
    a.n_rays = n_rays;
    a.x_start = c->in0.as<double>(); a.y_start = c->in1.as<double>(); a.z_start = c->in2.as<double>();
    a.kvec = kvec ? c->in3.as<double>() : nullptr;
    a.omega0 = 2.0 * M_PI * freq_hz;
    a.dt = dt; a.perturb_ratio = perturb_ratio;
    a.K = make_step_const(a.cube, dt, perturb_ratio);
    a.n_steps = n_steps; a.stride = record_stride; a.n_rec = n_rec;
    a.s_mode = s_mode;
    a.cs_every_step = cs_every_step();
    a.rec_pos = c->rec_pos.as<double>();
    a.rec_s = trace_cs ? c->rec_s.as<double>() : nullptr;
    a.active_steps = c->counters.as<unsigned long long>();
    const dim3 grid(blocks_for(n_rays, RT_BLOCK)), block(RT_BLOCK);
    // the FP32 cell-relative stepper keeps every stage within a few cells of the cached cell
    const int mode =
        max_stage_offset_cells(dt, trace_cs ? perturb_ratio : 0.0, c->wgeom.idx, c->wgeom.idy, c->wgeom.idz) < kMaxStageOffsetCells
            ? MODE_FAST32 : MODE_F64;
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
#define RT_TRACE_CASE(v, CS, M) \
    case v: trace_rays_kernel<CS, M><<<grid, block, 0, c->stream>>>(a); break;
    switch ((trace_cs ? 2 : 0) + mode) {
        RT_TRACE_CASE(0, false, MODE_FAST32) RT_TRACE_CASE(1, false, MODE_F64)
        RT_TRACE_CASE(2, true, MODE_FAST32) RT_TRACE_CASE(3, true, MODE_F64)
    }
#undef RT_TRACE_CASE
    RT_TRY(launched(c, "trace_rays_kernel"));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    if (r_record) {
        RT_TRY(c->out0.reserve((size_t)n_rec * 3 * nb));
        records_to_aos_kernel<<<blocks_for(n_rec * n_rays * 3, 256), 256, 0, c->stream>>>(
            c->rec_pos.as<double>(), c->out0.as<double>(), n_rec, n_rays);
        RT_TRY(launched(c, "records_to_aos_kernel"));
        RT_TRY(d2h(c, r_record, c->out0.p, (size_t)n_rec * 3 * nb));
    }
    if (s_record && trace_cs) RT_TRY(d2h(c, s_record, c->rec_s.p, (size_t)n_rec * nb));
    unsigned long long act = 0;
    RT_TRY(d2h(c, &act, c->counters.p, sizeof(act)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    if (active_steps) *active_steps = (int64_t)act;
    return RTGRFF_OK;
}

static int prepare_sampler(rtgrff_ctx *c, SampleArgs &a, double r_sun_cm, double fill_ne, double fill_te, double fill_b)
{
    const size_t n = (size_t)a.n_rec * a.n_rays;
    RT_TRY(c->smp_ne.reserve(n * 4)); RT_TRY(c->smp_te.reserve(n * 4)); RT_TRY(c->smp_b.reserve(n * 4));
    RT_TRY(c->smp_ds.reserve(n * 4)); RT_TRY(c->smp_s.reserve(n * 4)); RT_TRY(c->smp_valid.reserve(n));
    a.fcube = c->fcube.as<float4>();
    a.g = c->fgeomf;
    a.r_sun_cm = (float)r_sun_cm;   // numpy 2: float32 array * python float stays float32 (gpu_raytrace.py:482-484)
    a.fill_ne = (float)fill_ne; a.fill_te = (float)fill_te; a.fill_b = (float)fill_b;
    a.ne = c->smp_ne.as<float>(); a.te = c->smp_te.as<float>(); a.b = c->smp_b.as<float>();
    a.ds = c->smp_ds.as<float>(); a.s_out = c->smp_s.as<float>(); a.valid = c->smp_valid.as<uint8_t>();
    a.q_begin = 0; a.q_end = 0;
    c->smp_n = a.n_rec; c->smp_rays = a.n_rays;
    return RTGRFF_OK;
}

static int launch_sampler(rtgrff_ctx *c, const SampleArgs &a, int64_t count)
{
    unsigned int blocks = blocks_for(count, 256);
    const unsigned int cap = (unsigned int)c->sm_count * 64;
    if (blocks > cap) blocks = cap;
    sample_paths_kernel<<<blocks, 256, 0, c->stream>>>(a);
    return launched(c, "sample_paths_kernel");
}

static int run_sampler(rtgrff_ctx *c, SampleArgs &a, double r_sun_cm, double fill_ne, double fill_te, double fill_b)
{
    RT_TRY(prepare_sampler(c, a, r_sun_cm, fill_ne, fill_te, fill_b));
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    RT_TRY(launch_sampler(c, a, a.n_rec * a.n_rays));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    return RTGRFF_OK;
}

static int sampler_out(rtgrff_ctx *c, size_t n, float *ne, float *te, float *b, float *ds, uint8_t *valid, float *s)
{
    if (ne) RT_TRY(d2h(c, ne, c->smp_ne.p, n * 4));
    if (te) RT_TRY(d2h(c, te, c->smp_te.p, n * 4));
    if (b) RT_TRY(d2h(c, b, c->smp_b.p, n * 4));
    if (ds) RT_TRY(d2h(c, ds, c->smp_ds.p, n * 4));
    if (valid) RT_TRY(d2h(c, valid, c->smp_valid.p, n));
    if (s) RT_TRY(d2h(c, s, c->smp_s.p, n * 4));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

// rtgrff_sample on large host arrays: record-range chunks through the pinned bounce buffers (see the
// pipeline note above).  A chunk's ds looks back at earlier records, which are on the device already
// (chunks go up in order on one stream).
static int sample_pipelined(rtgrff_ctx *c, SampleArgs &a, const float *pos, const float *s, float *ne, float *te,
                            float *b, float *ds, uint8_t *valid)
{
    const int64_t n_rec = a.n_rec, n_rays = a.n_rays;
    const size_t per_rec_in = (size_t)n_rays * 16, per_rec_out = (size_t)n_rays * 17;
    int64_t rec_per_chunk = (int64_t)(kPipeChunkBytes / per_rec_out);
    if (rec_per_chunk < 1) rec_per_chunk = 1;
    const int64_t n_chunk = (n_rec + rec_per_chunk - 1) / rec_per_chunk;
    const size_t cin = (size_t)rec_per_chunk * per_rec_in, cout = (size_t)rec_per_chunk * per_rec_out;
    for (int q = 0; q < 2; ++q) {
        RT_TRY(pin_reserve(c, q, cin));
        RT_TRY(pin_reserve(c, 2 + q, cout));
    }
    cudaEvent_t *ev_in = c->chunk_ev, *ev_k = c->chunk_ev + 2, *ev_out = c->chunk_ev + 4;
    float *d_pos = c->in0.as<float>(), *d_s = c->in1.as<float>();
    auto unpack = [&](int64_t k) {
        const int64_t r0 = k * rec_per_chunk, r1 = std::min(n_rec, r0 + rec_per_chunk);
        const size_t q0 = (size_t)r0 * n_rays, cnt = (size_t)(r1 - r0) * n_rays;
        const char *src = (const char *)c->pinned[2 + (k & 1)];
        float *outs[4] = {ne, te, b, ds};
        for (int m = 0; m < 4; ++m)
            if (outs[m]) parallel_copy(outs[m] + q0, src + (size_t)m * cnt * 4, cnt * 4);
        if (valid) parallel_copy(valid + q0, src + (size_t)4 * cnt * 4, cnt);
    };
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    for (int64_t k = 0; k < n_chunk; ++k) {
        const int bsel = (int)(k & 1);
        const int64_t r0 = k * rec_per_chunk, r1 = std::min(n_rec, r0 + rec_per_chunk);
        const size_t q0 = (size_t)r0 * n_rays, cnt = (size_t)(r1 - r0) * n_rays;
        if (k >= 2) RT_CUDA(cudaEventSynchronize(ev_in[bsel]));
        char *pin = (char *)c->pinned[bsel];
        parallel_copy(pin, pos + q0 * 3, cnt * 12);
        parallel_copy(pin + cnt * 12, s + q0, cnt * 4);
        RT_CUDA(cudaMemcpyAsync(d_pos + q0 * 3, pin, cnt * 12, cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(cudaMemcpyAsync(d_s + q0, pin + cnt * 12, cnt * 4, cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(cudaEventRecord(ev_in[bsel], c->stream));
        a.q_begin = (int64_t)q0; a.q_end = (int64_t)(q0 + cnt);
        RT_TRY(launch_sampler(c, a, (int64_t)cnt));
        RT_CUDA(cudaEventRecord(ev_k[bsel], c->stream));
        RT_CUDA(cudaStreamWaitEvent(c->copy_stream, ev_k[bsel], 0));
        char *pout = (char *)c->pinned[2 + bsel];
        const float *outs[4] = {a.ne, a.te, a.b, a.ds};
        for (int m = 0; m < 4; ++m)
            RT_CUDA(cudaMemcpyAsync(pout + (size_t)m * cnt * 4, outs[m] + q0, cnt * 4, cudaMemcpyDeviceToHost, c->copy_stream));
        RT_CUDA(cudaMemcpyAsync(pout + (size_t)4 * cnt * 4, a.valid + q0, cnt, cudaMemcpyDeviceToHost, c->copy_stream));
        RT_CUDA(cudaEventRecord(ev_out[bsel], c->copy_stream));
        if (k >= 1) {
            RT_CUDA(cudaEventSynchronize(ev_out[1 - bsel]));
            unpack(k - 1);
        }
    }
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    RT_CUDA(cudaEventSynchronize(ev_out[(n_chunk - 1) & 1]));
    unpack(n_chunk - 1);
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_sample(rtgrff_ctx *c, int64_t n_rec, int64_t n_rays, const float *pos, const float *s,
                  const float *ray_start, double r_sun_cm, double fill_ne, double fill_te, double fill_b, float *ne,
                  float *te, float *b, float *ds, uint8_t *valid)
{
    RT_USE(c);
    if (!c->has_fcube) return fail(RTGRFF_ENOCUBE, "rtgrff_set_field_cubes has not been called");
    if (n_rec < 0 || n_rays < 0) return fail(RTGRFF_EINVAL, "negative sizes");
    const size_t n = (size_t)n_rec * n_rays;
    if (n == 0) return RTGRFF_OK;
    if (!pos || !s || !ray_start) return fail(RTGRFF_EINVAL, "null input");
    SampleArgs a{};
    a.n_rec = n_rec; a.n_rays = n_rays;
    RT_TRY(c->in0.reserve(n * 3 * sizeof(float)));
    RT_TRY(c->in1.reserve(n * sizeof(float)));
    RT_TRY(h2d(c, c->in2, ray_start, (size_t)n_rays * 3 * sizeof(float)));
    a.pos_aos = c->in0.as<float>(); a.s32 = c->in1.as<float>(); a.ray_start = c->in2.as<float>();
    if (c->pipeline && n * 33 >= kPipeMinBytes) {
        RT_TRY(prepare_sampler(c, a, r_sun_cm, fill_ne, fill_te, fill_b));
        return sample_pipelined(c, a, pos, s, ne, te, b, ds, valid);
    }
    RT_TRY(h2d(c, c->in0, pos, n * 3 * sizeof(float)));
    RT_TRY(h2d(c, c->in1, s, n * sizeof(float)));
    RT_TRY(run_sampler(c, a, r_sun_cm, fill_ne, fill_te, fill_b));
    return sampler_out(c, n, ne, te, b, ds, valid, nullptr);
}

int rtgrff_sample_traced(rtgrff_ctx *c, const float *ray_start, double r_sun_cm, double fill_ne, double fill_te,
                         double fill_b, float *ne, float *te, float *b, float *ds, uint8_t *valid, float *s)
{
    RT_USE(c);
    if (!c->has_fcube) return fail(RTGRFF_ENOCUBE, "rtgrff_set_field_cubes has not been called");
    if (c->rec_n <= 0 || c->rec_rays <= 0) return fail(RTGRFF_EINVAL, "no traced records on the device");
    if (!ray_start) return fail(RTGRFF_EINVAL, "null ray_start");
    const size_t n = (size_t)c->rec_n * c->rec_rays;
    RT_TRY(h2d(c, c->in2, ray_start, (size_t)c->rec_rays * 3 * sizeof(float)));
    SampleArgs a{};
    a.n_rec = c->rec_n; a.n_rays = c->rec_rays;
    a.pos_soa = c->rec_pos.as<double>();
    a.s64 = c->rec_has_s ? c->rec_s.as<double>() : nullptr;
    a.ray_start = c->in2.as<float>();
    RT_TRY(run_sampler(c, a, r_sun_cm, fill_ne, fill_te, fill_b));
    return sampler_out(c, n, ne, te, b, ds, valid, s);
}

static int launch_slice(rtgrff_ctx *c, const double *parms, const double *rparms, double *rl, int32_t *status, int npix,
                        int nz, int nf)
{
    SliceArgs a;
    a.parms = parms; a.rparms = rparms; a.rl = rl; a.status = status;
    a.npix = npix; a.nz = nz; a.nf = nf;
    const int64_t warps = (int64_t)npix * nf;
    grff_slice_kernel<<<blocks_for(warps * 32, 128), 128, 0, c->stream>>>(a);
    return launched(c, "grff_slice_kernel");
}

// on_device: Rparms / Parms / RL / status are device pointers (the fastGRFF contract: CuPy arrays in,
// RL_M written in place on the device, script/resample_with_ray_tracing.py:428-446); else host arrays,
// large ones moved in pixel chunks through the pinned bounce buffers while earlier chunks compute.
static int run_slice(rtgrff_ctx *c, int npix, int nz, int nf, const double *rparms, const double *parms, double *rl,
                     int32_t *status, int on_device)
{
    const size_t pix_b = (size_t)15 * nz * sizeof(double);
    const size_t pb = pix_b * npix, rb = (size_t)3 * npix * sizeof(double);
    const size_t ob = (size_t)7 * nf * npix * sizeof(double);
    if (on_device) {
        if (status) RT_CUDA(cudaMemsetAsync(status, 0xff, (size_t)npix * sizeof(int32_t), c->stream));
        RT_CUDA(cudaEventRecord(c->ev0, c->stream));
        RT_TRY(launch_slice(c, parms, rparms, rl, status, npix, nz, nf));
        RT_CUDA(cudaEventRecord(c->ev1, c->stream));
        c->ev_valid = true;
        RT_CUDA(cudaStreamSynchronize(c->stream));
        return RTGRFF_OK;
    }
    RT_TRY(c->in0.reserve(pb ? pb : 1));
    RT_TRY(h2d(c, c->in1, rparms, rb));
    RT_TRY(c->out0.reserve(ob));
    RT_TRY(c->out1.reserve((size_t)npix * sizeof(int32_t)));
    RT_CUDA(cudaMemsetAsync(c->out1.p, 0xff, (size_t)npix * sizeof(int32_t), c->stream));
    double *d_parms = c->in0.as<double>();
    if (c->pipeline && pb >= kPipeMinBytes && pix_b > 0) {
        int64_t pix_per_chunk = (int64_t)(kPipeChunkBytes / pix_b);
        if (pix_per_chunk < 1) pix_per_chunk = 1;
        const int64_t n_chunk = (npix + pix_per_chunk - 1) / pix_per_chunk;
        for (int q = 0; q < 2; ++q) RT_TRY(pin_reserve(c, q, (size_t)pix_per_chunk * pix_b));
        cudaEvent_t *ev_in = c->chunk_ev;
        RT_CUDA(cudaEventRecord(c->ev0, c->stream));
        for (int64_t k = 0; k < n_chunk; ++k) {
            const int bsel = (int)(k & 1);
            const int64_t p0 = k * pix_per_chunk, p1 = std::min<int64_t>(npix, p0 + pix_per_chunk);
            const size_t bytes = (size_t)(p1 - p0) * pix_b;
            if (k >= 2) RT_CUDA(cudaEventSynchronize(ev_in[bsel]));
            parallel_copy(c->pinned[bsel], (const char *)parms + (size_t)p0 * pix_b, bytes);
            RT_CUDA(cudaMemcpyAsync((char *)d_parms + (size_t)p0 * pix_b, c->pinned[bsel], bytes, cudaMemcpyHostToDevice, c->stream));
            RT_CUDA(cudaEventRecord(ev_in[bsel], c->stream));
            RT_TRY(launch_slice(c, d_parms + (size_t)p0 * 15 * nz, c->in1.as<double>() + (size_t)p0 * 3,
                                c->out0.as<double>() + (size_t)p0 * 7 * nf, c->out1.as<int32_t>() + p0, (int)(p1 - p0), nz, nf));
        }
        RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    } else {
        if (pb) RT_CUDA(cudaMemcpyAsync(d_parms, parms, pb, cudaMemcpyHostToDevice, c->stream));
        RT_CUDA(cudaEventRecord(c->ev0, c->stream));
        RT_TRY(launch_slice(c, d_parms, c->in1.as<double>(), c->out0.as<double>(), c->out1.as<int32_t>(), npix, nz, nf));
        RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    }
    c->ev_valid = true;
    RT_TRY(d2h(c, rl, c->out0.p, ob));
    if (status) RT_TRY(d2h(c, status, c->out1.p, (size_t)npix * sizeof(int32_t)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

static int slice_sizes(const int32_t *L, int &npix, int &nz, int &nf)
{
    npix = L[0]; nz = L[1]; nf = L[2];
    if (npix < 0 || nz < 0 || nf <= 0) return fail(RTGRFF_EINVAL, "bad Lparms_M {%d,%d,%d}", npix, nz, nf);
    if (L[3] > 1 || L[4] != 0 || L[5] != 0) return fail(RTGRFF_EUNSUPPORTED, "DEM / DDM inputs are not supported (Lparms_M[3..5] = {%d,%d,%d})", L[3], L[4], L[5]);
    return RTGRFF_OK;
}

int rtgrff_get_mw_slice(rtgrff_ctx *c, const int32_t *Lparms_M, const double *Rparms_M, const double *Parms_M,
                        const double *T_arr, const double *DEM_arr, const double *DDM_arr, double *RL_M, int32_t *status)
{
    (void)T_arr; (void)DEM_arr; (void)DDM_arr;
    RT_USE(c);
    if (!Lparms_M || !Rparms_M || !Parms_M || !RL_M) return fail(RTGRFF_EINVAL, "null argument");
    int npix, nz, nf;
    RT_TRY(slice_sizes(Lparms_M, npix, nz, nf));
    if (npix == 0) return RTGRFF_OK;
    return run_slice(c, npix, nz, nf, Rparms_M, Parms_M, RL_M, status, 0);
}

int rtgrff_get_mw_slice_device(rtgrff_ctx *c, const int32_t *Lparms_M, const double *Rparms_M_dev,
                               const double *Parms_M_dev, double *RL_M_dev, int32_t *status_dev)
{
    RT_USE(c);
    if (!Lparms_M || !Rparms_M_dev || !Parms_M_dev || !RL_M_dev) return fail(RTGRFF_EINVAL, "null argument");
    int npix, nz, nf;
    RT_TRY(slice_sizes(Lparms_M, npix, nz, nf));
    if (npix == 0) return RTGRFF_OK;
    return run_slice(c, npix, nz, nf, Rparms_M_dev, Parms_M_dev, RL_M_dev, status_dev, 1);
}

int rtgrff_device_alloc(rtgrff_ctx *c, void **out, size_t bytes)
{
    RT_USE(c);
    if (!out) return fail(RTGRFF_EINVAL, "null argument");
    *out = nullptr;
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? RTGRFF_ENOMEM : RTGRFF_ECUDA, "cudaMalloc(%zu) -> %s", bytes, cudaGetErrorString(e));
    return RTGRFF_OK;
}

int rtgrff_device_free(rtgrff_ctx *c, void *p)
{
    RT_USE(c);
    if (p) RT_CUDA(cudaFree(p));
    return RTGRFF_OK;
}

int rtgrff_memcpy(rtgrff_ctx *c, void *dst, const void *src, size_t bytes, int kind)
{
    RT_USE(c);
    if ((!dst || !src) && bytes) return fail(RTGRFF_EINVAL, "null argument");
    const cudaMemcpyKind k = kind == 0 ? cudaMemcpyHostToDevice : (kind == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice);
    if (kind < 0 || kind > 2) return fail(RTGRFF_EINVAL, "kind must be 0 (H2D), 1 (D2H) or 2 (D2D)");
    if (bytes) RT_CUDA(cudaMemcpyAsync(dst, src, bytes, k, c->stream));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_export_cubes(rtgrff_ctx *c, double *omega_pe, float *ne, float *te, float *b, float *bx, float *by, float *bz)
{
    RT_USE(c);
    if (omega_pe) {
        if (!c->has_wcube) return fail(RTGRFF_ENOCUBE, "no ray cube on the device");
        if (!c->stage_has_omega) return fail(RTGRFF_EUNSUPPORTED, "the float64 omega_pe of the last cube build is no longer staged on the device");
        const size_t n = (size_t)c->wgeom.nx * c->wgeom.ny * c->wgeom.nz;
        RT_TRY(d2h(c, omega_pe, c->stage.p, n * sizeof(double)));
        RT_CUDA(cudaStreamSynchronize(c->stream));
    }
    for (int pass = 0; pass < 2; ++pass) {
        float *o[3] = {pass ? bx : ne, pass ? by : te, pass ? bz : b};
        if (!o[0] && !o[1] && !o[2]) continue;
        if (pass ? !c->has_bvec : !c->has_fcube) return fail(RTGRFF_ENOCUBE, "no %s cube on the device", pass ? "B-vector" : "field");
        const size_t n = (size_t)c->fgeom.nx * c->fgeom.ny * c->fgeom.nz;
        RT_TRY(c->out3.reserve(3 * n * sizeof(float)));
        float *d = c->out3.as<float>();
        deinterleave3_kernel<<<blocks_for((int64_t)n, 256), 256, 0, c->stream>>>((pass ? c->bcube : c->fcube).as<float4>(), d,
                                                                                  d + n, d + 2 * n, (int64_t)n);
        RT_TRY(launched(c, "deinterleave3_kernel"));
        for (int m = 0; m < 3; ++m)
            if (o[m]) RT_TRY(d2h(c, o[m], d + (size_t)m * n, n * sizeof(float)));
        RT_CUDA(cudaStreamSynchronize(c->stream));
    }
    return RTGRFF_OK;
}

static std::mutex g_default_mu;
static rtgrff_ctx *g_default_ctx[64] = {nullptr};   // one process-wide context per device, made on first use

int PyGET_MW(const int32_t *Lparms, const double *Rparms, const double *Parms, const double *T_arr,
             const double *DEM_arr, const double *DDM_arr, double *RL)
{
    (void)T_arr; (void)DEM_arr; (void)DDM_arr;
    if (!Lparms || !Rparms || !Parms || !RL) return 1;
    const int nz = Lparms[0], nf = Lparms[1];
    if (nz < 0 || nf <= 0) return 1;
    if (Lparms[2] > 0) return 2;
    std::lock_guard<std::mutex> lk(g_default_mu);
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 3;   // the caller's current device
    if (!g_default_ctx[dev] && rtgrff_ctx_create(dev, nullptr, &g_default_ctx[dev]) != RTGRFF_OK) return 3;
    return run_slice(g_default_ctx[dev], 1, nz, nf, Rparms, Parms, RL, nullptr, 0) == RTGRFF_OK ? 0 : 3;
}

int rtgrff_emission_traced(rtgrff_ctx *c, double pixel_area_cm2, double freq0_hz, int n_freq, double freq_log_step,
                           int em_flag, int s_max, int s_input_on, double *tb, double *vi)
{
    RT_USE(c);
    if (c->smp_n <= 0 || c->smp_rays <= 0) return fail(RTGRFF_EINVAL, "no samples on the device (call rtgrff_sample_traced)");
    if (n_freq <= 0 || !tb || !vi) return fail(RTGRFF_EINVAL, "bad n_freq / null output");
    const size_t n = (size_t)c->smp_rays * n_freq;
    RT_TRY(c->out0.reserve(n * sizeof(double)));
    RT_TRY(c->out1.reserve(n * sizeof(double)));
    EmissionArgs a;
    a.ne = c->smp_ne.as<float>(); a.te = c->smp_te.as<float>(); a.b = c->smp_b.as<float>(); a.ds = c->smp_ds.as<float>();
    a.valid = c->smp_valid.as<uint8_t>();
    a.s = c->smp_s.as<float>(); a.s_input = s_input_on ? 1 : 0;
    a.n_rec = c->smp_n; a.n_rays = c->smp_rays;
    a.area = pixel_area_cm2; a.freq0 = freq0_hz; a.log_step = freq_log_step;
    a.n_freq = n_freq; a.em_flag = em_flag; a.s_max = s_max;
    a.grff64 = c->grff64;
    a.tb = c->out0.as<double>(); a.vi = c->out1.as<double>();
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    emission_rays_kernel<<<blocks_for((int64_t)n, 128), 128, 0, c->stream>>>(a);
    RT_TRY(launched(c, "emission_rays_kernel"));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    RT_TRY(d2h(c, tb, c->out0.p, n * sizeof(double)));
    RT_TRY(d2h(c, vi, c->out1.p, n * sizeof(double)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

// The T_b, V/I and diagnostic outputs of a map.  The kernel writes the caller's arrays when they are device
// memory, else the context's out0 / out1 / out3, which map_outputs_read_back then copies to the caller.
struct MapOutputs {
    double *tb, *vi, *diag;      // the caller's arrays; diag may be null
    size_t bytes;                // of tb and of vi; diag holds RTGRFF_N_DIAG times that
    bool on_device;
    double *dtb, *dvi, *ddiag;   // where the kernel writes
};

static int map_outputs_on_device(rtgrff_ctx *c, MapOutputs &o)
{
    o.dtb = o.tb; o.dvi = o.vi; o.ddiag = o.diag;
    if (o.on_device) return RTGRFF_OK;
    RT_TRY(c->out0.reserve(o.bytes));
    RT_TRY(c->out1.reserve(o.bytes));
    o.dtb = c->out0.as<double>(); o.dvi = c->out1.as<double>();
    if (o.diag) {
        RT_TRY(c->out3.reserve((size_t)RTGRFF_N_DIAG * o.bytes));
        o.ddiag = c->out3.as<double>();
    }
    return RTGRFF_OK;
}

static int map_outputs_read_back(rtgrff_ctx *c, const MapOutputs &o)
{
    if (o.on_device) return RTGRFF_OK;
    RT_TRY(d2h(c, o.tb, o.dtb, o.bytes));
    RT_TRY(d2h(c, o.vi, o.dvi, o.bytes));
    if (o.diag) RT_TRY(d2h(c, o.diag, o.ddiag, (size_t)RTGRFF_N_DIAG * o.bytes));
    return RTGRFF_OK;
}

// rtgrff_render_map and rtgrff_render_map_diag: diag == nullptr launches the plain kernels, else the DIAG ones
static int render_map_impl(rtgrff_ctx *c, int64_t n_rays, const double *x_start, const double *y_start,
                           const double *z_start, const double *kvec, const int32_t *ray_order, int n_freq,
                           const rtgrff_freq_params *freqs,
                           int trace_cs, double perturb_ratio, double pixel_area_cm2, double r_sun_cm, int em_flag, int s_max,
                           int use_bvec, int voxel_order, int s_mode, int s_input_on, double *tb, double *vi, int out_on_device,
                           int64_t *stats, double *diag)
{
    RT_USE(c);
    if (!c->has_wcube) return fail(RTGRFF_ENOCUBE, "rtgrff_set_omega_cube has not been called");
    if (!c->has_fcube) return fail(RTGRFF_ENOCUBE, "rtgrff_set_field_cubes has not been called");
    if (use_bvec && !c->has_bvec) return fail(RTGRFF_ENOCUBE, "use_bvec needs bx,by,bz in rtgrff_set_field_cubes");
    if (n_rays < 0 || n_freq <= 0 || n_freq > 65535 || !freqs || !tb || !vi) return fail(RTGRFF_EINVAL, "bad arguments");
    if (voxel_order != RTGRFF_ORDER_RECORD && voxel_order != RTGRFF_ORDER_REVERSED) return fail(RTGRFF_EINVAL, "bad voxel_order");
    if (s_mode != RTGRFF_S_PER_STEP && s_mode != RTGRFF_S_CUMULATIVE) return fail(RTGRFF_EINVAL, "bad s_mode");
    if (s_input_on && !trace_cs) return fail(RTGRFF_EINVAL, "s_input_on needs the cross-sections traced (trace_cs)");
    if (n_rays > 0 && (!x_start || !y_start || !z_start)) return fail(RTGRFF_EINVAL, "null start arrays");
    if (stats) stats[0] = stats[1] = stats[2] = stats[3] = 0;
    if (n_rays == 0) return RTGRFF_OK;
    const RayCube rc = ray_cube_of(c);
    std::vector<FreqDev> fd(n_freq);
    int64_t nominal = 0;
    for (int f = 0; f < n_freq; ++f) {
        if (freqs[f].n_steps < 0 || freqs[f].record_stride < 1 || !(freqs[f].freq_hz > 0.0) ||
            freqs[f].n_steps > 2147483000 || freqs[f].record_stride > 2147483000)
            return fail(RTGRFF_EINVAL, "bad per-frequency parameters at index %d", f);
        fd[f].nu = freqs[f].freq_hz;
        fd[f].omega0 = 2.0 * M_PI * freqs[f].freq_hz;
        fd[f].dt = freqs[f].dt;
        fd[f].n_steps = freqs[f].n_steps;
        fd[f].stride = freqs[f].record_stride;
        fd[f].out_row = f;
        fd[f].K = make_step_const(rc, freqs[f].dt, perturb_ratio);
        fd[f].fq = make_freq(freqs[f].freq_hz);
        nominal += freqs[f].n_steps * n_rays;
    }
    const size_t nb = (size_t)n_rays * sizeof(double);
    RT_TRY(h2d(c, c->in0, x_start, nb));
    RT_TRY(h2d(c, c->in1, y_start, nb));
    RT_TRY(h2d(c, c->in2, z_start, nb));
    if (kvec) RT_TRY(h2d(c, c->in3, kvec, 3 * nb));
    if (ray_order) {
        if (n_rays >= ((int64_t)1 << 31)) return fail(RTGRFF_EINVAL, "ray_order needs n_rays < 2^31");
        // the kernel reads x_start[ray_order[t]] and writes tb[ray_order[t]]: anything but a permutation of
        // 0..n_rays-1 would read / write out of bounds or leave pixels unwritten
        std::vector<uint8_t> seen((size_t)n_rays, 0);
        for (int64_t t = 0; t < n_rays; ++t) {
            const int32_t r = ray_order[t];
            if (r < 0 || r >= n_rays || seen[(size_t)r])
                return fail(RTGRFF_EINVAL, "ray_order is not a permutation of 0..n_rays-1 (entry %lld = %d)", (long long)t, r);
            seen[(size_t)r] = 1;
        }
        RT_TRY(h2d(c, c->out2, ray_order, (size_t)n_rays * sizeof(int32_t)));
    }
    RT_TRY(c->counters.reserve(64));
    RT_CUDA(cudaMemsetAsync(c->counters.p, 0, 64, c->stream));
    MapOutputs out{tb, vi, diag, (size_t)n_freq * nb, out_on_device != 0};
    RT_TRY(map_outputs_on_device(c, out));
    MapArgs a;
    a.cube = rc;
    a.fcube = c->fcube.as<float4>();
    a.bcube = c->has_bvec ? c->bcube.as<float4>() : nullptr;
    a.fg = c->fgeomf;
    a.n_rays = n_rays;
    a.x_start = c->in0.as<double>(); a.y_start = c->in1.as<double>(); a.z_start = c->in2.as<double>();
    a.kvec = kvec ? c->in3.as<double>() : nullptr;
    a.ray_order = ray_order ? c->out2.as<int>() : nullptr;
    a.perturb_ratio = perturb_ratio; a.area = pixel_area_cm2;
    a.r_sun_cm = (float)r_sun_cm; a.fill_ne = 0.0f; a.fill_te = 1e4f; a.fill_b = 0.0f;
    a.em_flag = em_flag; a.s_max = s_max; a.use_bvec = use_bvec; a.order = voxel_order;
    a.cs_every_step = cs_every_step();
    a.s_mode = s_mode; a.s_input = s_input_on ? 1 : 0;
    a.grff64 = c->grff64;
    a.tb = out.dtb; a.vi = out.dvi;
    a.active_steps = c->counters.as<unsigned long long>();
    a.diag = out.ddiag;
    a.diag_plane = (int64_t)n_freq * n_rays;     // planes follow the caller's frequency order: FreqDev::out_row
    const dim3 grid(blocks_for(n_rays, RT_BLOCK)), block(RT_BLOCK);
    const bool gr = !(em_flag & 1);
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    const int variant = (trace_cs ? 8 : 0) | (voxel_order == RTGRFF_ORDER_REVERSED ? 4 : 0) | (use_bvec ? 2 : 0) | (gr ? 1 : 0);
#define RT_MAP_LAUNCH(CS, ORD, BV, GR, DG)                                                                   \
        if (mode == MODE_FAST32)                                                                             \
            render_map_kernel<CS, ORD, BV, GR, MODE_FAST32, DG><<<grid, block, 0, c->stream>>>(a);           \
        else                                                                                                 \
            render_map_kernel<CS, ORD, BV, GR, MODE_F64, DG><<<grid, block, 0, c->stream>>>(a);
#define RT_MAP_CASE(v, CS, ORD, BV, GR)                                                                      \
    case v:                                                                                                  \
        if (diag) { RT_MAP_LAUNCH(CS, ORD, BV, GR, true) } else { RT_MAP_LAUNCH(CS, ORD, BV, GR, false) }    \
        break;
    // the FP32 cell-relative stepper keeps every stage within a few cells of the cached cell
    int mode = MODE_FAST32;
    for (int f = 0; f < n_freq; ++f)
        if (!(max_stage_offset_cells(freqs[f].dt, trace_cs ? perturb_ratio : 0.0, c->wgeom.idx, c->wgeom.idy,
                                     c->wgeom.idz) < kMaxStageOffsetCells))
            mode = MODE_F64;
    // Longest frequencies first: blocks are dispatched in grid order, and a launch that ends on its
    // most expensive blocks (15 000 steps with a record at every step) idles most of the chip in its tail.
    std::stable_sort(fd.begin(), fd.end(), [&](const FreqDev &x, const FreqDev &y) {
        auto cost = [&](const FreqDev &q) {
            return (double)q.n_steps * (1.0 + ((trace_cs ? 2.0 : 0.0) + 1.0) / (double)q.stride);
        };
        return cost(x) > cost(y);
    });
    // one launch per frequency (its constants travel in the kernel parameters), round-robin over the fork streams
    const bool fork = n_freq > 1;
    cudaStream_t main_stream = c->stream;
    if (fork) {
        for (int q = 0; q < kMapForkStreams; ++q)
            if (!c->fstream[q]) RT_CUDA(cudaStreamCreateWithFlags(&c->fstream[q], cudaStreamNonBlocking));
        for (int q = 0; q <= kMapForkStreams; ++q)
            if (!c->fev[q]) RT_CUDA(cudaEventCreateWithFlags(&c->fev[q], cudaEventDisableTiming));
        RT_CUDA(cudaEventRecord(c->fev[kMapForkStreams], main_stream));
        for (int q = 0; q < kMapForkStreams; ++q) RT_CUDA(cudaStreamWaitEvent(c->fstream[q], c->fev[kMapForkStreams], 0));
    }
    for (int f = 0; f < n_freq; ++f) {
        a.freq = fd[f];
        struct StreamSwap {           // the launches below go to c->stream
            rtgrff_ctx *c; cudaStream_t keep;
            ~StreamSwap() { c->stream = keep; }
        } swap{c, main_stream};
        if (fork) c->stream = c->fstream[f % kMapForkStreams];
        switch (variant) {
            RT_MAP_CASE(0, false, 0, false, false) RT_MAP_CASE(1, false, 0, false, true)
            RT_MAP_CASE(2, false, 0, true, false) RT_MAP_CASE(3, false, 0, true, true)
            RT_MAP_CASE(4, false, 1, false, false) RT_MAP_CASE(5, false, 1, false, true)
            RT_MAP_CASE(6, false, 1, true, false) RT_MAP_CASE(7, false, 1, true, true)
            RT_MAP_CASE(8, true, 0, false, false) RT_MAP_CASE(9, true, 0, false, true)
            RT_MAP_CASE(10, true, 0, true, false) RT_MAP_CASE(11, true, 0, true, true)
            RT_MAP_CASE(12, true, 1, false, false) RT_MAP_CASE(13, true, 1, false, true)
            RT_MAP_CASE(14, true, 1, true, false) RT_MAP_CASE(15, true, 1, true, true)
        }
        RT_TRY(launched(c, "render_map_kernel"));
    }
    if (fork) {
        for (int q = 0; q < kMapForkStreams; ++q) {
            RT_CUDA(cudaEventRecord(c->fev[q], c->fstream[q]));
            RT_CUDA(cudaStreamWaitEvent(main_stream, c->fev[q], 0));
        }
    }
#undef RT_MAP_CASE
#undef RT_MAP_LAUNCH
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    RT_TRY(map_outputs_read_back(c, out));
    unsigned long long act[3] = {0, 0, 0};
    RT_TRY(d2h(c, act, c->counters.p, sizeof(act)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    if (stats) { stats[0] = nominal; stats[1] = (int64_t)act[0]; stats[2] = (int64_t)act[1]; stats[3] = (int64_t)act[2]; }
    return RTGRFF_OK;
}

int rtgrff_render_map(rtgrff_ctx *c, int64_t n_rays, const double *x_start, const double *y_start,
                      const double *z_start, const double *kvec, const int32_t *ray_order, int n_freq,
                      const rtgrff_freq_params *freqs,
                      int trace_cs, double perturb_ratio, double pixel_area_cm2, double r_sun_cm, int em_flag, int s_max,
                      int use_bvec, int voxel_order, int s_mode, int s_input_on, double *tb, double *vi, int out_on_device,
                      int64_t *stats)
{
    return render_map_impl(c, n_rays, x_start, y_start, z_start, kvec, ray_order, n_freq, freqs, trace_cs, perturb_ratio,
                           pixel_area_cm2, r_sun_cm, em_flag, s_max, use_bvec, voxel_order, s_mode, s_input_on, tb, vi,
                           out_on_device, stats, nullptr);
}

int rtgrff_render_map_diag(rtgrff_ctx *c, int64_t n_rays, const double *x_start, const double *y_start,
                           const double *z_start, const double *kvec, const int32_t *ray_order, int n_freq,
                           const rtgrff_freq_params *freqs,
                           int trace_cs, double perturb_ratio, double pixel_area_cm2, double r_sun_cm, int em_flag,
                           int s_max, int use_bvec, int voxel_order, int s_mode, int s_input_on, double *tb, double *vi,
                           int out_on_device, int64_t *stats, double *diag)
{
    if (!diag) return fail(RTGRFF_EINVAL, "rtgrff_render_map_diag needs the diag output");
    return render_map_impl(c, n_rays, x_start, y_start, z_start, kvec, ray_order, n_freq, freqs, trace_cs, perturb_ratio,
                           pixel_area_cm2, r_sun_cm, em_flag, s_max, use_bvec, voxel_order, s_mode, s_input_on, tb, vi,
                           out_on_device, stats, diag);
}

// ---- fused straight line-of-sight map ----------------------------------------------------------------
int rtgrff_set_spherical_model(rtgrff_ctx *c, int slot, const float *data, const double *phi, const double *lat,
                               const double *r, int np, int nt, int nr, double scale)
{
    RT_USE(c);
    if (slot < 0 || slot >= kLosSlots) return fail(RTGRFF_EINVAL, "slot %d out of range 0..4", slot);
    if (!data || !phi || !lat || !r) return fail(RTGRFF_EINVAL, "null argument");
    if (np < 2 || nt < 2 || nr < 2) return fail(RTGRFF_EINVAL, "spherical mesh needs >= 2 nodes per axis");
    if ((int64_t)np * nt * nr >= (int64_t)1 << 31) return fail(RTGRFF_EINVAL, "spherical mesh larger than 2^31 nodes");
    RT_TRY(check_ascending_nodes(phi, np, lat, nt, r, nr));
    c->sph_set[slot] = false;
    RT_TRY(h2d(c, c->sph_data[slot], data, (size_t)np * nt * nr * sizeof(float)));
    std::vector<double> &n = c->sph_nodes[slot];
    n.assign(phi, phi + np);
    n.insert(n.end(), lat, lat + nt);
    n.insert(n.end(), r, r + nr);
    c->sph_n[slot][0] = np; c->sph_n[slot][1] = nt; c->sph_n[slot][2] = nr;
    c->sph_scale[slot] = scale;
    RT_CUDA(cudaStreamSynchronize(c->stream));   // the host buffer may be reused by the caller
    c->sph_set[slot] = true;
    return RTGRFF_OK;
}

// rtgrff_render_los_map / diag == nullptr launches the plain kernels, else the DIAG ones
int rtgrff_render_los_map(rtgrff_ctx *c, int nx, int ny, const double *x, const double *y, int nz, const double *zc,
                          const double *dz_cm, double phi0_offset_deg, double r_min, double z_eps, int n_freq,
                          const double *freq_hz, double pixel_area_cm2, int em_flag, int s_max, int use_bvec, double *tb,
                          double *vi, double *diag, int out_on_device, int64_t *stats)
{
    return rtgrff_render_los_map_view(c, nx, ny, x, y, nz, zc, dz_cm, phi0_offset_deg, 0.0, 0.0, r_min, z_eps, n_freq,
                                      freq_hz, pixel_area_cm2, em_flag, s_max, use_bvec, tb, vi, diag, out_on_device,
                                      stats);
}

int rtgrff_render_los_map_view(rtgrff_ctx *c, int nx, int ny, const double *x, const double *y, int nz,
                               const double *zc, const double *dz_cm, double phi0_offset_deg, double b0_deg,
                               double p_deg, double r_min, double z_eps, int n_freq, const double *freq_hz,
                               double pixel_area_cm2, int em_flag, int s_max, int use_bvec, double *tb, double *vi,
                               double *diag, int out_on_device, int64_t *stats)
{
    RT_USE(c);
    if (!x || !y || !zc || !dz_cm || !freq_hz || !tb || !vi) return fail(RTGRFF_EINVAL, "null argument");
    ViewRot view;
    RT_TRY(view_from(b0_deg, p_deg, view));
    if (nx < 1 || ny < 1 || nz < 1 || n_freq < 1) return fail(RTGRFF_EINVAL, "bad sizes (nx %d, ny %d, nz %d, n_freq %d)",
                                                              nx, ny, nz, n_freq);
    if ((int64_t)nx * ny >= (int64_t)1 << 31) return fail(RTGRFF_EINVAL, "image larger than 2^31 pixels");
    for (int f = 0; f < n_freq; ++f)
        if (!(freq_hz[f] > 0.0) || !isfinite(freq_hz[f])) return fail(RTGRFF_EINVAL, "bad frequency at index %d", f);
    static const char *names[kLosSlots] = {"rho", "te", "br", "bt", "bp"};
    for (int v = 0; v < kLosSlots; ++v)
        if (!c->sph_set[v]) return fail(RTGRFF_ENOCUBE, "rtgrff_set_spherical_model has not set slot %d (%s)", v, names[v]);
    if (stats) stats[0] = stats[1] = stats[2] = 0;
    LosMapArgs a;
    int n_nodes = 0;
    for (int v = 0; v < kLosSlots; ++v) {
        a.var[v].data = c->sph_data[v].as<float>();
        a.var[v].phi = a.var[v].lat = a.var[v].r = nullptr;
        a.var[v].np = c->sph_n[v][0]; a.var[v].nt = c->sph_n[v][1]; a.var[v].nr = c->sph_n[v][2];
        a.scale[v] = c->sph_scale[v];
        a.node_off[v] = n_nodes;
        n_nodes += (int)c->sph_nodes[v].size();
    }
    // the frequencies of a block: as many groups of at most kLosMaxFreqGroup as needed, balanced
    const int groups = (n_freq + kLosMaxFreqGroup - 1) / kLosMaxFreqGroup;
    const int fg = (n_freq + groups - 1) / groups;
    if (groups > 65535) return fail(RTGRFF_EINVAL, "n_freq %d too large", n_freq);
    const size_t smem = los_map_smem(fg, n_nodes);
    int dev_smem = 0;
    RT_CUDA(cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
    if (smem > (size_t)dev_smem)
        return fail(RTGRFF_EINVAL, "spherical meshes too large: %d nodes need %zu B of shared memory (%d available)", n_nodes,
                    smem, dev_smem);
    // inputs: x | y | zc | dz_cm | mesh nodes in one buffer, the per-frequency constants in another
    std::vector<double> host((size_t)nx + ny + 2 * (size_t)nz + n_nodes);
    double *h = host.data();
    memcpy(h, x, nx * sizeof(double));
    memcpy(h + nx, y, ny * sizeof(double));
    memcpy(h + nx + ny, zc, nz * sizeof(double));
    memcpy(h + nx + ny + nz, dz_cm, nz * sizeof(double));
    for (int v = 0; v < kLosSlots; ++v)
        memcpy(h + nx + ny + 2 * (size_t)nz + a.node_off[v], c->sph_nodes[v].data(), c->sph_nodes[v].size() * sizeof(double));
    std::vector<FreqC> fq(n_freq);
    for (int f = 0; f < n_freq; ++f) fq[f] = make_freq(freq_hz[f]);
    RT_TRY(h2d(c, c->in0, h, host.size() * sizeof(double)));
    RT_TRY(h2d(c, c->in1, fq.data(), fq.size() * sizeof(FreqC)));
    const double *d = c->in0.as<double>();
    a.x = d; a.y = d + nx; a.zc = d + nx + ny; a.dz_cm = d + nx + ny + nz;
    a.nodes = d + nx + ny + 2 * (size_t)nz;
    a.n_nodes = n_nodes;
    a.nx = nx; a.ny = ny; a.nz = nz;
    a.tiles_x = (nx + kLosTileW - 1) / kLosTileW;
    a.phi0_offset_rad = phi0_offset_deg * M_PI / 180.0;
    a.r_min = r_min; a.z_eps = z_eps;
    a.view = view;
    a.freqs = c->in1.as<FreqC>();
    a.n_freq = n_freq; a.fg = fg;
    a.area = pixel_area_cm2;
    a.em_flag = em_flag; a.s_max = s_max; a.grff64 = c->grff64;
    const size_t npix = (size_t)nx * ny, nb = npix * sizeof(double);
    MapOutputs out{tb, vi, diag, (size_t)n_freq * nb, out_on_device != 0};
    RT_TRY(map_outputs_on_device(c, out));
    a.tb = out.dtb; a.vi = out.dvi; a.diag = out.ddiag;
    RT_TRY(c->counters.reserve(64));
    RT_CUDA(cudaMemsetAsync(c->counters.p, 0, 64, c->stream));
    a.valid_samples = c->counters.as<unsigned long long>();
    const int64_t tiles = (int64_t)a.tiles_x * ((ny + kLosTileH - 1) / kLosTileH);
    const dim3 grid((unsigned int)tiles, (unsigned int)groups), block(32 * fg);
    const bool gr = !(em_flag & 1);
    const int variant = (use_bvec ? 4 : 0) | (use_bvec || gr ? 2 : 0) | (diag ? 1 : 0);
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
#define RT_LOS_CASE(v, BV, NB, DG, VW)                                                                                \
    case v:                                                                                                           \
        if (smem > 48 * 1024)                                                                                         \
            RT_CUDA(cudaFuncSetAttribute(los_map_kernel<BV, NB, DG, VW>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         (int)smem));                                                                 \
        los_map_kernel<BV, NB, DG, VW><<<grid, block, smem, c->stream>>>(a);                                          \
        break;
    switch (variant | (view.on ? 8 : 0)) {
        RT_LOS_CASE(0, false, false, false, false) RT_LOS_CASE(1, false, false, true, false)
        RT_LOS_CASE(2, false, true, false, false) RT_LOS_CASE(3, false, true, true, false)
        RT_LOS_CASE(6, true, true, false, false) RT_LOS_CASE(7, true, true, true, false)
        RT_LOS_CASE(8, false, false, false, true) RT_LOS_CASE(9, false, false, true, true)
        RT_LOS_CASE(10, false, true, false, true) RT_LOS_CASE(11, false, true, true, true)
        RT_LOS_CASE(14, true, true, false, true) RT_LOS_CASE(15, true, true, true, true)
    }
#undef RT_LOS_CASE
    RT_TRY(launched(c, "los_map_kernel"));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    RT_TRY(map_outputs_read_back(c, out));
    unsigned long long n_valid = 0;
    RT_TRY(d2h(c, &n_valid, c->counters.p, sizeof(n_valid)));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    if (stats) {
        stats[0] = (int64_t)npix * nz;
        stats[1] = (int64_t)n_valid;
        stats[2] = (int64_t)n_valid * n_freq;
    }
    return RTGRFF_OK;
}

// ---- multi-GPU: row sharding + image gather ---------------------------------------------------------
int rtgrff_shard_rows(int n_rows, int world_size, int rank, int32_t *rows, int *n_local, int *max_rows)
{
    if (n_rows < 0 || world_size < 1 || rank < 0 || rank >= world_size) return fail(RTGRFF_EINVAL, "bad n_rows / world_size / rank");
    const int G = row_group_of(n_rows, world_size);
    int n = 0;
    for (int row = 0; row < n_rows; ++row)
        if ((row / G) % world_size == rank) {
            if (rows) rows[n] = row;
            ++n;
        }
    if (n_local) *n_local = n;
    if (max_rows) *max_rows = max_rows_per_rank(n_rows, world_size);
    return RTGRFF_OK;
}

int rtgrff_comm_unique_id(char id[128])
{
    if (!id) return fail(RTGRFF_EINVAL, "null id");
    NcclApi *n = nccl_api();
    if (!n) return fail(RTGRFF_EUNSUPPORTED, "libnccl.so.2 could not be loaded (%s)", dlerror() ? "dlopen failed" : "symbols missing");
    NcclUniqueId u;
    const int rc = n->GetUniqueId(&u);
    if (rc != 0) return fail(RTGRFF_ECUDA, "ncclGetUniqueId -> %s", n->GetErrorString(rc));
    memcpy(id, u.internal, 128);
    return RTGRFF_OK;
}

int rtgrff_comm_init_rank(rtgrff_ctx *c, int world_size, int rank, const char id[128])
{
    RT_USE(c);
    if (world_size < 1 || rank < 0 || rank >= world_size) return fail(RTGRFF_EINVAL, "bad world_size / rank");
    if (c->comm) return fail(RTGRFF_EINVAL, "the context already has a communicator");
    c->comm_rank = rank; c->comm_size = world_size;
    if (world_size == 1) return RTGRFF_OK;        // nothing to talk to
    if (!id) return fail(RTGRFF_EINVAL, "null id");
    NcclApi *n = nccl_api();
    if (!n) return fail(RTGRFF_EUNSUPPORTED, "libnccl.so.2 could not be loaded");
    NcclUniqueId u;
    memcpy(u.internal, id, 128);
    NcclComm comm = nullptr;
    const int rc = n->CommInitRank(&comm, world_size, u, rank);
    if (rc != 0) return fail(RTGRFF_ECUDA, "ncclCommInitRank -> %s", n->GetErrorString(rc));
    c->comm = comm;
    return RTGRFF_OK;
}

int rtgrff_comm_destroy(rtgrff_ctx *c)
{
    RT_USE(c);
    if (c->comm) {
        NcclApi *n = nccl_api();
        cudaStreamSynchronize(c->stream);
        if (n) n->CommDestroy((NcclComm)c->comm);
        c->comm = nullptr;
    }
    c->comm_rank = 0; c->comm_size = 1;
    return RTGRFF_OK;
}

int rtgrff_place_rows(rtgrff_ctx *c, const double *gathered, int world_size, int n_planes, int n_rows, int n_cols,
                      double *image)
{
    RT_USE(c);
    if (!gathered || !image || world_size < 1 || n_planes < 1 || n_rows < 1 || n_cols < 1) return fail(RTGRFF_EINVAL, "bad arguments");
    const int mr = max_rows_per_rank(n_rows, world_size), G = row_group_of(n_rows, world_size);
    const size_t img_n = (size_t)n_planes * n_rows * n_cols;
    const unsigned int blocks = (unsigned int)std::min<int64_t>(blocks_for((int64_t)img_n, 256), (int64_t)c->sm_count * 16);
    place_rows_kernel<<<blocks, 256, 0, c->stream>>>(gathered, image, n_planes, n_rows, n_cols, mr, world_size, G);
    RT_TRY(launched(c, "place_rows_kernel"));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_gather_image(rtgrff_ctx *c, const double *slab, int n_planes, int n_rows, int n_cols, int root, double *image,
                        int image_on_device)
{
    RT_USE(c);
    const int W = c->comm_size, me = c->comm_rank;
    if (!slab || n_planes < 1 || n_rows < 1 || n_cols < 1 || root < 0 || root >= W) return fail(RTGRFF_EINVAL, "bad arguments");
    if (me == root && !image) return fail(RTGRFF_EINVAL, "the root needs an image buffer");
    if (W > 1 && !c->comm) return fail(RTGRFF_EINVAL, "rtgrff_comm_init_rank has not been called");
    const int mr = max_rows_per_rank(n_rows, W), G = row_group_of(n_rows, W);
    const size_t slab_n = (size_t)n_planes * mr * n_cols, img_n = (size_t)n_planes * n_rows * n_cols;
    const double *gathered = slab;
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    if (W > 1) {
        NcclApi *n = nccl_api();
        int rc = n->GroupStart();
        if (me == root) {
            RT_TRY(c->gather_buf.reserve((size_t)W * slab_n * sizeof(double)));
            double *buf = c->gather_buf.as<double>();
            for (int r = 0; r < W && rc == 0; ++r) {
                if (r == me) continue;
                rc = n->Recv(buf + (size_t)r * slab_n, slab_n * sizeof(double), kNcclInt8, r, (NcclComm)c->comm, c->stream);
            }
            gathered = buf;
        } else if (rc == 0) {
            rc = n->Send(slab, slab_n * sizeof(double), kNcclInt8, root, (NcclComm)c->comm, c->stream);
        }
        const int rc2 = n->GroupEnd();
        if (rc != 0 || rc2 != 0) return fail(RTGRFF_ECUDA, "NCCL gather -> %s", n->GetErrorString(rc ? rc : rc2));
        if (me == root)
            RT_CUDA(cudaMemcpyAsync(c->gather_buf.as<double>() + (size_t)me * slab_n, slab, slab_n * sizeof(double),
                                    cudaMemcpyDeviceToDevice, c->stream));
    }
    if (me == root) {
        double *dimg = image;
        if (!image_on_device) {
            RT_TRY(c->image_buf.reserve(img_n * sizeof(double)));
            dimg = c->image_buf.as<double>();
        }
        const unsigned int blocks = (unsigned int)std::min<int64_t>(blocks_for((int64_t)img_n, 256), (int64_t)c->sm_count * 16);
        place_rows_kernel<<<blocks, 256, 0, c->stream>>>(gathered, dimg, n_planes, n_rows, n_cols, mr, W, G);
        RT_TRY(launched(c, "place_rows_kernel"));
        RT_CUDA(cudaEventRecord(c->ev1, c->stream));
        c->ev_valid = true;
        if (!image_on_device) return d2h_large(c, image, dimg, img_n * sizeof(double));
    }
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_gaussian_beam(rtgrff_ctx *c, const double *img, int ny, int nx, int n_planes, double sigma_pix,
                         double truncate, double *out)
{
    RT_USE(c);
    if (!img || !out || ny < 1 || nx < 1 || n_planes < 1) return fail(RTGRFF_EINVAL, "bad arguments");
    if (!(sigma_pix >= 0.0) || !isfinite(sigma_pix) || !(truncate > 0.0)) return fail(RTGRFF_EINVAL, "bad sigma/truncate");
    const size_t n = (size_t)n_planes * ny * nx, nb = n * sizeof(double);
    // scipy.ndimage._gaussian_kernel1d: radius = int(truncate*sigma + 0.5), exp(-x^2/(2 sigma^2)) / sum
    const int radius = (int)(truncate * sigma_pix + 0.5);
    std::vector<double> w(radius + 1);
    double sum = 0.0;
    for (int d = -radius; d <= radius; ++d) sum += sigma_pix > 0.0 ? exp(-0.5 / (sigma_pix * sigma_pix) * (double)d * (double)d) : (d == 0 ? 1.0 : 0.0);
    for (int d = 0; d <= radius; ++d)
        w[d] = (sigma_pix > 0.0 ? exp(-0.5 / (sigma_pix * sigma_pix) * (double)d * (double)d) : (d == 0 ? 1.0 : 0.0)) / sum;
    RT_TRY(h2d(c, c->in0, img, nb));
    RT_TRY(h2d(c, c->in1, w.data(), w.size() * sizeof(double)));
    RT_TRY(c->out0.reserve(nb));
    RT_TRY(c->out1.reserve(nb));
    const unsigned int blocks = (unsigned int)std::min<int64_t>(blocks_for((int64_t)n, 256), (int64_t)c->sm_count * 32);
    RT_CUDA(cudaEventRecord(c->ev0, c->stream));
    // gaussian_filter runs the 1-D filter axis by axis: rows direction (axis 0) first, then axis 1
    gaussian_pass_kernel<<<blocks, 256, 0, c->stream>>>(c->in0.as<double>(), c->out0.as<double>(), c->in1.as<double>(),
                                                        radius, ny, nx, n_planes, 0);
    RT_TRY(launched(c, "gaussian_pass_kernel"));
    gaussian_pass_kernel<<<blocks, 256, 0, c->stream>>>(c->out0.as<double>(), c->out1.as<double>(), c->in1.as<double>(),
                                                        radius, ny, nx, n_planes, 1);
    RT_TRY(launched(c, "gaussian_pass_kernel"));
    RT_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->ev_valid = true;
    RT_TRY(d2h(c, out, c->out1.p, nb));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    return RTGRFF_OK;
}

int rtgrff_patch_nan(rtgrff_ctx *c, double *img, int ny, int nx, int n_planes, int max_passes, int64_t *n_patched)
{
    RT_USE(c);
    if (!img || ny < 1 || nx < 1 || n_planes < 1 || max_passes < 0) return fail(RTGRFF_EINVAL, "bad arguments");
    if (n_patched) *n_patched = 0;
    const size_t n = (size_t)n_planes * ny * nx, nb = n * sizeof(double);
    RT_TRY(h2d(c, c->in0, img, nb));
    RT_TRY(c->out0.reserve(nb));
    RT_TRY(c->out1.reserve(nb));
    RT_TRY(c->out2.reserve(n));
    RT_TRY(c->counters.reserve(64 + (size_t)n_planes * sizeof(int)));
    int *d_any = c->counters.as<int>();
    int *d_fixed = reinterpret_cast<int *>(c->counters.as<char>() + 64);
    const unsigned int blocks = (unsigned int)std::min<int64_t>(blocks_for((int64_t)n, 256), (int64_t)c->sm_count * 32);
    std::vector<int> fixed(n_planes);
    int64_t total = 0;
    // _patch_nan_2d (util.py:45-76): up to max_passes sweeps; stop when nothing is left or nothing could be fixed
    for (int pass = 0; pass < max_passes; ++pass) {
        RT_CUDA(cudaMemsetAsync(c->counters.p, 0, 64 + (size_t)n_planes * sizeof(int), c->stream));
        mark_nonfinite_kernel<<<blocks, 256, 0, c->stream>>>(c->in0.as<double>(), c->out2.as<unsigned char>(), (int64_t)n, d_any);
        RT_TRY(launched(c, "mark_nonfinite_kernel"));
        int any = 0;
        RT_TRY(d2h(c, &any, d_any, sizeof(int)));
        RT_CUDA(cudaStreamSynchronize(c->stream));
        if (!any) break;
        next_finite_kernel<<<blocks_for((int64_t)n_planes * (ny + nx), 128), 128, 0, c->stream>>>(
            c->in0.as<double>(), c->out0.as<double>(), c->out1.as<double>(), ny, nx, n_planes);
        RT_TRY(launched(c, "next_finite_kernel"));
        patch_nan_pass_kernel<<<n_planes, 1024, 0, c->stream>>>(c->in0.as<double>(), c->out2.as<unsigned char>(),
                                                                c->out0.as<double>(), c->out1.as<double>(), ny, nx, d_fixed);
        RT_TRY(launched(c, "patch_nan_pass_kernel"));
        RT_TRY(d2h(c, fixed.data(), d_fixed, (size_t)n_planes * sizeof(int)));
        RT_CUDA(cudaStreamSynchronize(c->stream));
        int64_t f = 0;
        for (int v : fixed) f += v;
        total += f;
        if (f == 0) break;
    }
    RT_TRY(d2h(c, img, c->in0.p, nb));
    RT_CUDA(cudaStreamSynchronize(c->stream));
    if (n_patched) *n_patched = total;
    return RTGRFF_OK;
}

}  // extern "C"
