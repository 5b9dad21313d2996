// capi.cu — host side of librtiow_cuda.so: the C ABI of include/rtiow_cuda.h.
// Replaces the rayon row loop, collect and flip of /root/reference/src/main.rs:122-145 with
// one call that drives the sm_100a kernels in rt_render.cuh.  No CPU fallback anywhere: with no
// CUDA device every compute entry point returns RTIOW_ERR_NO_DEVICE.
#include "../../include/rtiow_cuda.h"
#include "rt_unit.cuh"

#include <nccl.h>
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>
#include <utility>

using namespace rt;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
    return code;
}
#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            cudaGetLastError();                                                                          \
            return fail(e_ == cudaErrorMemoryAllocation ? RTIOW_ERR_NOMEM : RTIOW_ERR_CUDA, "%s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                                \
    } while (0)

extern "C" int rtiow_abi_version(void) { return RTIOW_ABI_VERSION; }
extern "C" const char* rtiow_last_error(void) { return g_err.c_str(); }
extern "C" int rtiow_device_count(int* out)
{
    if (!out) return fail(RTIOW_ERR_INVALID_ARG, "out_count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
    *out = n;
    return RTIOW_OK;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
// a buffer that only grows: device memory, or page-locked host memory (the staging buffers of the H2D / D2H copies)
template <typename U, bool kHost> struct Buf {
    U* p = nullptr; size_t n = 0;
    cudaError_t resize(size_t count)
    {
        if (count <= n && p) return cudaSuccess;
        release();
        const size_t bytes = std::max<size_t>(count, 1) * sizeof(U);
        cudaError_t e = kHost ? cudaMallocHost((void**)&p, bytes) : cudaMalloc((void**)&p, bytes);
        if (e == cudaSuccess) n = count;
        return e;
    }
    void release() { if (p) { if (kHost) cudaFreeHost(p); else cudaFree(p); } p = nullptr; n = 0; }
};
template <typename U> using DevBuf = Buf<U, false>;
template <typename U> using HostBuf = Buf<U, true>;

struct DeviceState {
    int device = 0;
    int sms = 0;
    cudaStream_t stream = nullptr; bool owns_stream = true;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_done = nullptr;
    // frames enqueued without a host synchronisation (rtiow_render_rank_enqueue): one event pair per frame until rtiow_ctx_synchronize
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ring; size_t ring_used = 0;
    uint64_t enq_paths = 0; uint32_t enq_launches = 0; uint32_t enq_world = 1;
    // scene
    // every scene array lives in ONE device allocation, filled by ONE H2D copy from a page-locked staging blob (rtiow_scene_upload):
    // twelve small pageable copies cost 0.25 ms per upload, which is 2.5 % of a 10 ms frame in the end-to-end call at 8 GPUs
    DevBuf<unsigned char> scene_blob;
    SceneDev scene{};
    bool has_scene = false;
    // frame
    DevBuf<unsigned long long> accum; DevBuf<unsigned long long> counters;   // [0]=work [1]=rays
    DevBuf<uint32_t> tiles; DevBuf<uint32_t> gathered; DevBuf<uint32_t> frame;
    HostBuf<uint8_t> pinned;                           // staging of the frame's D2H copy when the caller's buffer is pageable
    HostBuf<unsigned long long> pinned_cnt;            // the counters after the frame
    DevBuf<unsigned char> cams; HostBuf<unsigned char> cams_stage;   // the cameras of a batch of views (rtiow_render_views) and their staging
    // measurement
    DevBuf<uint4> flush; DevBuf<float> probe;
    int last_backend = RTIOW_SCAN_FP32;                // which filter the last render launch used (rtiow_stats.scan_backend)
};

struct rtiow_ctx {
    std::vector<DeviceState> dev;
    int scan_backend = RTIOW_SCAN_AUTO;  // rtiow_ctx_set_scan_backend
    HostBuf<unsigned char> scene_stage;  // page-locked staging blob of rtiow_scene_upload
    bool peer_ok = true;                 // every device can store into device 0's memory (NVLink P2P): fused epilogue + gather
    // the gather of the row tiles (rtiow_ctx_set_gather)
    int gather = RTIOW_GATHER_AUTO;
    std::vector<ncclComm_t> comms;       // one process driving n GPUs: ncclCommInitAll, created on first use
    // one process per GPU (rtiow_ctx_create_rank)
    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
    int* d_flag = nullptr;               // 1-int all-reduce: the frame-complete barrier of the fused gather / agreement votes
    // fused gather across processes: rank 0's double-buffered frame, mapped into every rank through CUDA IPC
    uint32_t* ipc_frame = nullptr; size_t ipc_frame_px = 0; bool ipc_owner = false; int ipc_state = 0;   // 0 untried, 1 mapped, -1 unavailable
    uint32_t ipc_parity = 0;
    // NCCL user-buffer registration of the tile / gathered buffers (symmetric window), when the library offers it
    void* win_tiles = nullptr; void* win_gathered = nullptr; uint32_t* nccl_tiles = nullptr; uint32_t* nccl_gathered = nullptr; size_t nccl_tile_px = 0;
    bool windows_registered = false;
    std::string gather_note;
};

// is this host pointer page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory)?  Then a D2H copy can DMA straight into it.
static bool host_is_pinned(const void* p)
{
    cudaPointerAttributes pa{};
    const bool yes = cudaPointerGetAttributes(&pa, p) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    (void)cudaGetLastError();
    return yes;
}

static int init_device(DeviceState& d, int device)
{
    d.device = device;
    CU(cudaSetDevice(device));
    cudaDeviceProp p; CU(cudaGetDeviceProperties(&p, device));
    // arch-specific targets are not forward compatible: sm_100a code runs on compute capability 10.0 and nothing else
    if (p.major != 10 || p.minor != 0) return fail(RTIOW_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, p.major, p.minor);
    d.sms = p.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    CU(cudaEventCreate(&d.ev0)); CU(cudaEventCreate(&d.ev1)); CU(cudaEventCreateWithFlags(&d.ev_done, cudaEventDisableTiming));
    CU(d.counters.resize(2));
    CU(d.pinned_cnt.resize(2));
    return RTIOW_OK;
}

static int create_ctx(const std::vector<int>& devices, rtiow_ctx** out)
{
    if (!out) return fail(RTIOW_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    int n = 0; rtiow_device_count(&n);
    if (n == 0) return fail(RTIOW_ERR_NO_DEVICE, "no CUDA device visible (there is no CPU fallback)");
    for (int dv : devices) if (dv < 0 || dv >= n) return fail(RTIOW_ERR_INVALID_ARG, "device %d out of range (have %d)", dv, n);
    rtiow_ctx* c = new rtiow_ctx();
    c->dev.resize(devices.size());
    for (size_t i = 0; i < devices.size(); ++i) {
        int rc = init_device(c->dev[i], devices[i]);
        if (rc != RTIOW_OK) { rtiow_ctx_destroy(c); return rc; }
    }
    // peer access for the tile gather over NVLink (single-process multi-GPU)
    for (size_t i = 1; i < devices.size(); ++i) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, devices[i], devices[0]);
        bool ok = false;
        if (can) {
            cudaSetDevice(devices[i]);
            cudaError_t e = cudaDeviceEnablePeerAccess(devices[0], 0);
            ok = (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled);
            if (e != cudaSuccess) cudaGetLastError();
        }
        if (!ok) c->peer_ok = false;
    }
    *out = c;
    return RTIOW_OK;
}

extern "C" int rtiow_ctx_create(int n_gpus, rtiow_ctx** out)
{
    if (n_gpus < 1) return fail(RTIOW_ERR_INVALID_ARG, "n_gpus must be >= 1");
    std::vector<int> d(n_gpus);
    for (int i = 0; i < n_gpus; ++i) d[i] = i;
    return create_ctx(d, out);
}
extern "C" int rtiow_ctx_create_on_device(int device, rtiow_ctx** out) { return create_ctx(std::vector<int>{ device }, out); }

extern "C" int rtiow_ctx_set_scan_backend(rtiow_ctx* c, int backend)
{
    if (!c) return fail(RTIOW_ERR_INVALID_ARG, "ctx is NULL");
    if (backend != RTIOW_SCAN_AUTO && backend != RTIOW_SCAN_FP32 && backend != RTIOW_SCAN_TENSOR) return fail(RTIOW_ERR_INVALID_ARG, "unknown scan backend %d", backend);
    c->scan_backend = backend;
    return RTIOW_OK;
}

extern "C" void rtiow_ctx_destroy(rtiow_ctx* c);
// ------------------------------------------------------------------------------------------------
// NCCL, loaded at run time (dlopen): a single-GPU caller needs no NCCL at all, and a process that already carries one (the
// bench under torchrun: torch's bundled libnccl.so.2) shares it instead of mapping a second copy with the same soname.
// ------------------------------------------------------------------------------------------------
struct NcclApi {
    void* h = nullptr; char version[16] = "";          // "2.27.3": named in the gathers' notes (rtiow_ctx_gather_info)
    ncclResult_t (*GetVersion)(int*) = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    // optional (NCCL >= 2.27): user buffers registered as a symmetric window
    ncclResult_t (*MemAlloc)(void**, size_t) = nullptr;
    ncclResult_t (*MemFree)(void*) = nullptr;
    ncclResult_t (*CommWindowRegister)(ncclComm_t, void*, size_t, ncclWindow_t*, int) = nullptr;
    ncclResult_t (*CommWindowDeregister)(ncclComm_t, ncclWindow_t) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load()
{
    if (g_nccl.h) return RTIOW_OK;
    void* h = nullptr;
    const char* tried = "libnccl.so.2, libnccl.so";
    if (const char* p = getenv("RTIOW_NCCL_LIB")) { h = dlopen(p, RTLD_NOW | RTLD_GLOBAL); tried = p; }     // deployment knob: which NCCL to load
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(RTIOW_ERR_NCCL, "NCCL is not available (%s): %s — multi-GPU gathers need it, single-GPU rendering does not", tried, dlerror());
    NcclApi a; a.h = h;
#define SYM(field, name) *(void**)(&a.field) = dlsym(h, name)
    SYM(GetVersion, "ncclGetVersion"); SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommInitAll, "ncclCommInitAll");
    SYM(CommDestroy, "ncclCommDestroy"); SYM(AllGather, "ncclAllGather"); SYM(AllReduce, "ncclAllReduce"); SYM(Broadcast, "ncclBroadcast");
    SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd"); SYM(GetErrorString, "ncclGetErrorString");
    SYM(MemAlloc, "ncclMemAlloc"); SYM(MemFree, "ncclMemFree"); SYM(CommWindowRegister, "ncclCommWindowRegister"); SYM(CommWindowDeregister, "ncclCommWindowDeregister");
#undef SYM
    if (!a.GetVersion || !a.GetUniqueId || !a.CommInitRank || !a.CommInitAll || !a.CommDestroy || !a.AllGather || !a.AllReduce || !a.Broadcast ||
        !a.GroupStart || !a.GroupEnd || !a.GetErrorString)
        return fail(RTIOW_ERR_NCCL, "the NCCL library that was loaded lacks a required symbol");
    int v = 0; a.GetVersion(&v);
    snprintf(a.version, sizeof a.version, "%d.%d.%d", v / 10000, (v / 100) % 100, v % 100);
    g_nccl = a;
    return RTIOW_OK;
}
#define NC(call)                                                                                         \
    do {                                                                                                 \
        ncclResult_t r_ = (call);                                                                        \
        if (r_ != ncclSuccess) return fail(RTIOW_ERR_NCCL, "%s -> %s (%s:%d)", #call, g_nccl.GetErrorString(r_), __FILE__, __LINE__); \
    } while (0)

extern "C" int rtiow_nccl_unique_id(void* out_id)
{
    if (!out_id) return fail(RTIOW_ERR_INVALID_ARG, "out_id is NULL");
    static_assert(sizeof(ncclUniqueId) == RTIOW_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
    int rc = nccl_load(); if (rc) return rc;
    ncclUniqueId id;
    NC(g_nccl.GetUniqueId(&id));
    memcpy(out_id, &id, sizeof id);
    return RTIOW_OK;
}

extern "C" int rtiow_ctx_create_rank(int device, int rank, int world, const void* nccl_unique_id, rtiow_ctx** out)
{
    if (!out) return fail(RTIOW_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world) return fail(RTIOW_ERR_INVALID_ARG, "bad rank/world (%d of %d)", rank, world);
    if (world > 1 && !nccl_unique_id) return fail(RTIOW_ERR_INVALID_ARG, "nccl_unique_id is NULL (rank 0 calls rtiow_nccl_unique_id and hands the 128 bytes to every rank)");
    rtiow_ctx* c = nullptr;
    int rc = create_ctx(std::vector<int>{ device }, &c); if (rc) return rc;
    c->rank = rank; c->world = world;
    if (world > 1) {
        rc = nccl_load(); if (rc) { rtiow_ctx_destroy(c); return rc; }
        ncclUniqueId id; memcpy(&id, nccl_unique_id, sizeof id);
        cudaSetDevice(device);
        ncclResult_t r = g_nccl.CommInitRank(&c->comm, world, id, rank);
        if (r != ncclSuccess) { c->comm = nullptr; rtiow_ctx_destroy(c); return fail(RTIOW_ERR_NCCL, "ncclCommInitRank(rank %d of %d) -> %s", rank, world, g_nccl.GetErrorString(r)); }
        if (cudaMalloc(&c->d_flag, 2 * sizeof(int)) != cudaSuccess) { rtiow_ctx_destroy(c); return fail(RTIOW_ERR_NOMEM, "cudaMalloc of the barrier flag failed"); }
    }
    *out = c;
    return RTIOW_OK;
}

// A one-device ctx does all its work on `stream` from now on (a cudaStream_t the caller owns; NULL restores the ctx's own):
// the caller's events and copies on that stream are then ordered with the library's kernels and NCCL calls.
extern "C" int rtiow_ctx_set_stream(rtiow_ctx* c, void* stream)
{
    if (!c) return fail(RTIOW_ERR_INVALID_ARG, "ctx is NULL");
    if (c->dev.size() != 1) return fail(RTIOW_ERR_INVALID_ARG, "rtiow_ctx_set_stream needs a one-device ctx");
    DeviceState& d = c->dev[0];
    CU(cudaSetDevice(d.device));
    CU(cudaStreamSynchronize(d.stream));
    if (d.owns_stream && d.stream) cudaStreamDestroy(d.stream);
    if (stream) { d.stream = (cudaStream_t)stream; d.owns_stream = false; }
    else { CU(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking)); d.owns_stream = true; }
    return RTIOW_OK;
}

extern "C" int rtiow_ctx_set_gather(rtiow_ctx* c, int mode)
{
    if (!c) return fail(RTIOW_ERR_INVALID_ARG, "ctx is NULL");
    if (mode != RTIOW_GATHER_AUTO && mode != RTIOW_GATHER_NCCL && mode != RTIOW_GATHER_FUSED) return fail(RTIOW_ERR_INVALID_ARG, "unknown gather mode %d", mode);
    c->gather = mode;
    return RTIOW_OK;
}

extern "C" int rtiow_ctx_gather_info(rtiow_ctx* c, char* buf, size_t n)
{
    if (!c || !buf || n == 0) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    snprintf(buf, n, "%s", c->gather_note.empty() ? "single GPU: no gather" : c->gather_note.c_str());
    return RTIOW_OK;
}

// rank 0's frame of the fused gather: rank 0 frees what it allocated, the other ranks unmap it
static void drop_ipc_frame(rtiow_ctx* c)
{
    if (c->ipc_frame) { if (c->ipc_owner) cudaFree(c->ipc_frame); else cudaIpcCloseMemHandle(c->ipc_frame); }
    c->ipc_frame = nullptr;
}
// the ncclMemAlloc buffers of the NCCL gather and their windows; afterwards no buffers are ready (nccl_tile_px = 0)
static void drop_nccl_buffers(rtiow_ctx* c)
{
    if (c->windows_registered && g_nccl.CommWindowDeregister && c->comm) {
        if (c->win_tiles) g_nccl.CommWindowDeregister(c->comm, (ncclWindow_t)c->win_tiles);
        if (c->win_gathered) g_nccl.CommWindowDeregister(c->comm, (ncclWindow_t)c->win_gathered);
    }
    if (c->nccl_tiles && g_nccl.MemFree) g_nccl.MemFree(c->nccl_tiles);
    if (c->nccl_gathered && g_nccl.MemFree) g_nccl.MemFree(c->nccl_gathered);
    c->win_tiles = c->win_gathered = nullptr; c->windows_registered = false;
    c->nccl_tiles = c->nccl_gathered = nullptr; c->nccl_tile_px = 0;
}

static void release_gather(rtiow_ctx* c)
{
    if (c->dev.empty()) return;
    cudaSetDevice(c->dev[0].device);
    drop_nccl_buffers(c);
    drop_ipc_frame(c);
    if (c->d_flag) cudaFree(c->d_flag);
    if (c->comm) g_nccl.CommDestroy(c->comm);
    for (size_t i = 0; i < c->comms.size(); ++i) { cudaSetDevice(c->dev[i].device); if (c->comms[i]) g_nccl.CommDestroy(c->comms[i]); }
    c->comms.clear(); c->comm = nullptr; c->d_flag = nullptr;
}

extern "C" void rtiow_ctx_destroy(rtiow_ctx* c)
{
    if (!c) return;
    for (auto& d : c->dev) { cudaSetDevice(d.device); if (d.stream) cudaStreamSynchronize(d.stream); }
    release_gather(c);
    for (auto& d : c->dev) {
        cudaSetDevice(d.device);
        if (d.stream) cudaStreamSynchronize(d.stream);
        d.scene_blob.release();
        d.accum.release(); d.counters.release(); d.tiles.release(); d.gathered.release(); d.frame.release();
        d.flush.release(); d.probe.release();
        d.pinned.release(); d.pinned_cnt.release(); d.cams.release(); d.cams_stage.release();
        if (d.ev0) cudaEventDestroy(d.ev0);
        if (d.ev1) cudaEventDestroy(d.ev1);
        if (d.ev_done) cudaEventDestroy(d.ev_done);
        for (auto& ev : d.ring) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
        if (d.stream && d.owns_stream) cudaStreamDestroy(d.stream);
    }
    c->scene_stage.release();
    delete c;
}

// ------------------------------------------------------------------------------------------------
// scene upload: HittableList (shapes/mod.rs:52) -> device SoA
// ------------------------------------------------------------------------------------------------
// spheres with |r| above this go to the f64 list: for them |oc|^2 - r^2 (sphere.rs:22) and the far
// root of rays leaving the surface lose more than t_min = 1e-4 (main.rs:44) in f32.
static const double kBigRadius = 8.0;

static int check_scene(const rtiow_spheres* s, const rtiow_materials* m)
{
    if (s->n > 0 && (!s->cx || !s->cy || !s->cz || !s->radius || !s->mat_index)) return fail(RTIOW_ERR_INVALID_ARG, "NULL sphere array");
    if (m->n > 0 && (!m->kind || !m->albedo_r || !m->albedo_g || !m->albedo_b || !m->param)) return fail(RTIOW_ERR_INVALID_ARG, "NULL material array");
    if (s->n > (1u << 30)) return fail(RTIOW_ERR_INVALID_ARG, "too many spheres");
    for (int i = 0; i < (int)s->n; ++i) {
        if (s->mat_index[i] >= m->n) return fail(RTIOW_ERR_INVALID_ARG, "sphere %d: material index %u out of range (%u)", i, s->mat_index[i], m->n);
        if (m->kind[s->mat_index[i]] > RTIOW_MAT_DIELECTRIC) return fail(RTIOW_ERR_UNSUPPORTED, "sphere %d: material kind %u has no GPU implementation", i, m->kind[s->mat_index[i]]);
        if (!(std::isfinite(s->cx[i]) && std::isfinite(s->cy[i]) && std::isfinite(s->cz[i]) && std::isfinite(s->radius[i])))
            return fail(RTIOW_ERR_INVALID_ARG, "sphere %d: non-finite centre or radius", i);
    }
    // a non-finite albedo or param that a sphere's material reads would turn the reference's pixel black through NaN, while the
    // render drops the sample (to_fix); Dielectric ignores its albedo and Lambertian its param (materials.rs), so those may be anything
    for (int i = 0; i < (int)s->n; ++i) {
        const uint32_t k = s->mat_index[i], kind = m->kind[k];
        if (kind != RTIOW_MAT_DIELECTRIC && !(std::isfinite(m->albedo_r[k]) && std::isfinite(m->albedo_g[k]) && std::isfinite(m->albedo_b[k])))
            return fail(RTIOW_ERR_INVALID_ARG, "sphere %d: material %u has a non-finite albedo", i, k);
        if (kind != RTIOW_MAT_LAMBERTIAN && !std::isfinite(m->param[k]))
            return fail(RTIOW_ERR_INVALID_ARG, "sphere %d: material %u has a non-finite param", i, k);
    }
    return RTIOW_OK;
}

// The FP32 filter's table of the small spheres (rt_scene.cuh): records of 4 spheres [cx0..3][cy0..3][cz0..3][K0..3], then the
// look-ahead record.  small = the first ns entries are spheres, the rest padding; R2 = the squared bounding radius of the filter.
static std::vector<float> filter_table(const std::vector<float4>& small, int ns, double R2)
{
    const int np = (int)small.size();
    std::vector<float> table(RT_TABLE_FLOATS(np), 0.0f);
    for (int p = 0; p < np; ++p) {
        float* rec = table.data() + (size_t)(p >> 2) * 16 + (p & 3);
        if (p < ns) {
            const float4 v = small[p];
            rec[0] = v.x; rec[4] = v.y; rec[8] = v.z;
            // K = |c|^2 - r^2 + R^2 of the f32 sphere, in f64, lowered by the filter slack (RT_FILTER_SLACK, rt_scene.cuh)
            // and rounded toward -inf: the filter may only err towards keeping a sphere
            const double c2 = (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z, r2 = (double)v.w * v.w;
            const double K = c2 - r2 + R2 - (double)RT_FILTER_SLACK * (c2 + r2 + R2) - 1e-30;
            float Kf = (float)K; if ((double)Kf > K) Kf = std::nextafterf(Kf, -INFINITY);
            rec[12] = Kf;
        } else {       // padding: C = 1e30 can never be reached by hb^2
            rec[0] = 0; rec[4] = 0; rec[8] = 0; rec[12] = 1e30f;
        }
    }
    for (int k = 0; k < 4; ++k) table[(size_t)np * 4 + 12 + k] = 1e30f;        // the look-ahead record: never hit, never used
    return table;
}

// f32 fast path of the large spheres: centre as hi + lo floats, K = |c|^2 - r^2 (from f64) as hi + lo; only offered (*ok) when the
// radius is a float and the centre's lo part is one too (anything else keeps the f64 routine for every ray)
static std::vector<float4> big_sphere_records(const std::vector<double4>& big, bool* ok)
{
    const int nb = (int)big.size();
    std::vector<float4> bigf(3 * (size_t)nb); bool bigf_ok = nb > 0;
    for (int b = 0; b < nb; ++b) {
        const double4 v = big[b];
        const float hx = (float)v.x, hy = (float)v.y, hz = (float)v.z, r = (float)v.w;
        const float lx = (float)(v.x - hx), ly = (float)(v.y - hy), lz = (float)(v.z - hz);
        const double K = v.x * v.x + v.y * v.y + v.z * v.z - v.w * v.w;
        const float Kh = (float)K, Kl = (float)(K - (double)Kh);
        bigf_ok = bigf_ok && (double)r == v.w && (double)hx + (double)lx == v.x && (double)hy + (double)ly == v.y && (double)hz + (double)lz == v.z && std::isfinite(Kh);
        bigf[3 * b] = make_float4(hx, hy, hz, r); bigf[3 * b + 1] = make_float4(lx, ly, lz, Kh); bigf[3 * b + 2] = make_float4(Kl, 0.f, 0.f, 0.f);
    }
    *ok = bigf_ok;
    return bigf;
}

// Tensor-core filter (rt_umma.cuh): per small sphere the 11 features of the bilinear discriminant, scaled by powers of
// two chosen from the bounding radius, split hi/lo in fp16, in the canonical K-major layout.  S_0 carries the slack that
// bounds the 3-product split and the fp32 accumulation (tools/probe_umma_filter.cu measures 1.15e-6 R^2; 1.5625e-5 R^2 here).
// Enabled when the image fits beside the candidate lists in one CTA's shared memory and the slack stays below the
// mean r^2 (a scene spread over a huge radius would pass every sphere near the line; the FP32 filter handles those).
// Returns the padded sphere count u_npad, or 0 (and no image) when the scene does not qualify.
static int tensor_image(const std::vector<float4>& small, int ns, double R, std::vector<unsigned char>* img, umma::FeatScale* u_sc)
{
    using Shape = UmmaShape<RT_UMMA_GROUPS, RT_UMMA_CHUNK>;
    const int npad = (ns + RT_UMMA_CHUNK - 1) / RT_UMMA_CHUNK * RT_UMMA_CHUNK;
    const double Rp = std::exp2(std::ceil(std::log2(R)));
    const double slack = 1.5625e-5 * R * R;
    double mean_r2 = 0; for (int j = 0; j < ns; ++j) mean_r2 += (double)small[j].w * small[j].w;
    mean_r2 = ns ? mean_r2 / ns : 0.0;
    // fp16 accumulator: |D| <= 4 R^2 for a line that meets the bounding sphere; it must stay finite in fp16
    const bool d_fits = 4.0 * R * R < 60000.0;
    if (!(ns > 0 && npad < 65536 && Shape::smem_bytes(npad) <= 227 * 1024 && Rp <= 8192.0 && slack <= mean_r2 && d_fits)) return 0;
    *u_sc = umma::FeatScale{ (float)Rp, 1.0f, (float)(Rp * 0.5), (float)(1.0 / Rp) };
    const size_t blk = RT_UMMA_B_BLOCK_BYTES(npad);
    img->assign(2 * blk, 0);
    // sphere j of `small` sits in column col(j) of the image: with the fp16 accumulator the columns of a 32-sphere word are
    // permuted so that the packed sign collection (umma::sign_word16) returns bit 31 - k for sphere k, as the funnel shifts do
    // K slots of the two blocks: umma::b2_feature (block 0 = B1: every hi feature + the hi parts that meet the ray's lo
    // parts of features 10 and 0..3; block 1 = B2: the lo parts of features 0..9 + the hi parts that meet lo_4..lo_9)
    auto put_all = [&](int j, const double (&S)[11]) {
        const uint32_t col = ((uint32_t)j & ~31u) | umma::d16_column((uint32_t)j & 31u);
        for (int b = 0; b < 2; ++b)
            for (int s = 0; s < 16; ++s) {
                int feat; bool is_lo; umma::b2_feature(b, s, &feat, &is_lo);
                const float x = (float)S[feat]; const __half h = __float2half_rn(x); const __half l = __float2half_rn(x - __half2float(h));
                memcpy(&(*img)[b * blk + umma::b_offset(col, s)], is_lo ? &l : &h, 2);
            }
    };
    for (int j = 0; j < npad; ++j) {
        double S[11] = { 0 };
        if (j < ns) {                     // position j of `small` (list order); the f32 sphere the precise test sees
            const float4 v = small[j];
            const double x = v.x, y = v.y, z = v.z, r = v.w;
            S[0] = (r * r - (x * x + y * y + z * z) + slack) / u_sc->s0;
            S[1] = x / u_sc->s1; S[2] = y / u_sc->s1; S[3] = z / u_sc->s1;
            S[4] = x * x / u_sc->s4; S[5] = y * y / u_sc->s4; S[6] = z * z / u_sc->s4;
            S[7] = x * y / u_sc->s4; S[8] = x * z / u_sc->s4; S[9] = y * z / u_sc->s4;
        } else {
            // padding: never passes, whatever the ray.  Its D = -2 Rp^2 - |f_perp|^2 (+ sigma) stays within
            // |D| <= 2 Rp^2 + R^2 < 65504, finite in fp16 up to the largest R that d_fits admits (Rp = 128)
            S[0] = -2.0 * Rp * Rp / u_sc->s0;
        }
        S[10] = 1.0 / u_sc->s10;                              // a power of two: no lo part (the two-product form relies on it)
        put_all(j, S);
    }
    return npad;
}

// The scene's arrays in one allocation, each at a 256-byte boundary.  put() appends an array and returns its offset in the
// guise of a pointer; rebase() turns such offsets into addresses in a device's copy of the blob.
struct SceneBlob {
    struct Part { const void* src; size_t bytes, off; };
    std::vector<Part> parts; size_t bytes = 0;
    template <typename U> const U* put(const std::vector<U>& v)
    {
        const Part pt{ v.data(), v.size() * sizeof(U), bytes };
        parts.push_back(pt);
        bytes += (pt.bytes + 255) & ~(size_t)255;
        return reinterpret_cast<const U*>(pt.off);
    }
    void write(unsigned char* dst) const { for (const Part& pt : parts) if (pt.bytes) memcpy(dst + pt.off, pt.src, pt.bytes); }
};
static SceneDev rebase(SceneDev s, const unsigned char* blob)
{
    auto at = [blob](auto& p) { p = reinterpret_cast<std::remove_reference_t<decltype(p)>>(blob + reinterpret_cast<uintptr_t>(p)); };
    at(s.table); at(s.small); at(s.small_idx); at(s.big); at(s.big_idx); at(s.sph); at(s.sphd); at(s.mat); at(s.matd); at(s.kind); at(s.u_bimg); at(s.bigf);
    return s;
}

extern "C" int rtiow_scene_upload(rtiow_ctx* c, const rtiow_spheres* s, const rtiow_materials* m)
{
    if (!c || !s || !m) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_scene(s, m); if (rc) return rc;
    const int n = (int)s->n;
    std::vector<float4> sph(n), mat(n); std::vector<double4> sphd(n), matd(n); std::vector<uint8_t> kind(n);
    std::vector<int> small_idx, big_idx;
    // A sphere with a later twin (the same centre and radius) never wins: the reference computes the same root for both, and
    // the later index takes every tie (mod.rs:61-66).  It is left out of every scan.  Kept in, it would compete with the
    // twin a ray starts on, whose root the scan takes exactly (candidate_self) while its own carries the origin's rounding.
    std::vector<int> order(n);
    for (int i = 0; i < n; ++i) order[i] = i;
    const auto key = [s](int i) { return std::make_tuple(s->cx[i], s->cy[i], s->cz[i], s->radius[i]); };
    std::sort(order.begin(), order.end(), [&](int a, int b) { return key(a) < key(b) || (key(a) == key(b) && a < b); });
    std::vector<uint8_t> shadowed(n, 0);
    for (int k = 0; k + 1 < n; ++k) shadowed[order[k]] = key(order[k]) == key(order[k + 1]);
    for (int i = 0; i < n; ++i) {
        const uint32_t mi = s->mat_index[i];
        sphd[i] = make_double4(s->cx[i], s->cy[i], s->cz[i], s->radius[i]);
        sph[i] = make_float4((float)s->cx[i], (float)s->cy[i], (float)s->cz[i], (float)s->radius[i]);
        matd[i] = make_double4(m->albedo_r[mi], m->albedo_g[mi], m->albedo_b[mi], m->param[mi]);
        mat[i] = make_float4((float)m->albedo_r[mi], (float)m->albedo_g[mi], (float)m->albedo_b[mi], (float)m->param[mi]);
        kind[i] = (uint8_t)m->kind[mi];
        const double reach = std::sqrt(s->cx[i] * s->cx[i] + s->cy[i] * s->cy[i] + s->cz[i] * s->cz[i]) + std::fabs(s->radius[i]);
        if (shadowed[i]) sphd[i].w = NAN;        // the f64 scan tests every sphere: a NaN root loses every comparison in candidate
        else if (std::fabs(s->radius[i]) > kBigRadius || reach > 4096.0) big_idx.push_back(i);
        else small_idx.push_back(i);
    }
    const int ns = (int)small_idx.size(), nb = (int)big_idx.size();
    while (small_idx.size() % 32) small_idx.push_back(-1);                  // whole 32-sphere words; padding never hits
    const int np = (int)small_idx.size();
    if (np > 65535 * 32) return fail(RTIOW_ERR_UNSUPPORTED, "scene too large");
    std::vector<float4> small(np);
    for (int p = 0; p < ns; ++p) small[p] = sph[small_idx[p]];
    // R: radius of the sphere around the coordinate origin on which the filter places its line point (rt_scene.cuh);
    // it bounds every small sphere, so a line that misses it can hit none of them
    double R = 1.0, rmax = 0.0;
    for (int p = 0; p < ns; ++p) {
        const float4 v = small[p];
        R = std::max(R, std::sqrt((double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z) + std::fabs((double)v.w));
        rmax = std::max(rmax, std::fabs((double)v.w));
    }
    const float R2f = (float)(R * R * (1.0 + 1e-6));
    const std::vector<float> table = filter_table(small, ns, (double)R2f);
    std::vector<double4> big(nb); for (int b = 0; b < nb; ++b) big[b] = sphd[big_idx[b]];
    bool bigf_ok = false;
    const std::vector<float4> bigf = big_sphere_records(big, &bigf_ok);
    SceneDev sc{};
    std::vector<unsigned char> ubimg;
    sc.u_sc = umma::FeatScale{ 1.0f, 1.0f, 1.0f, 1.0f };
    sc.u_npad = tensor_image(small, ns, R, &ubimg, &sc.u_sc);
    SceneBlob blob;                      // the pointers of `sc` hold offsets into the blob until rebase()
    sc.table = blob.put(table); sc.small = blob.put(small); sc.small_idx = blob.put(small_idx); sc.big = blob.put(big); sc.big_idx = blob.put(big_idx);
    sc.sph = blob.put(sph); sc.sphd = blob.put(sphd); sc.mat = blob.put(mat); sc.matd = blob.put(matd); sc.kind = blob.put(kind);
    sc.u_bimg = blob.put(ubimg); sc.bigf = blob.put(bigf);
    sc.np = np; sc.n_rec = (ns + 3) / 4; sc.nb = nb; sc.n = n;
    sc.filter_R2 = R2f; sc.filter_sigma = (float)(16.0 * 5.9604644775390625e-08 * std::max(rmax, 1e-3));
    CU(c->scene_stage.resize(blob.bytes));
    blob.write(c->scene_stage.p);
    for (auto& d : c->dev) {
        CU(cudaSetDevice(d.device));
        CU(d.scene_blob.resize(blob.bytes));
        CU(cudaMemcpyAsync(d.scene_blob.p, c->scene_stage.p, blob.bytes, cudaMemcpyHostToDevice, d.stream));
        CU(cudaStreamSynchronize(d.stream));
        d.scene = rebase(sc, d.scene_blob.p);
        if (!bigf_ok) d.scene.bigf = nullptr;          // the records stay in the blob; the f64 routine handles every large sphere
        d.has_scene = true;
    }
    return RTIOW_OK;
}

// ------------------------------------------------------------------------------------------------
// Camera::new (camera.rs:17-45), host f64
// ------------------------------------------------------------------------------------------------
struct HV { double x, y, z; };
static HV hsub(HV a, HV b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
static HV hmul(HV a, double s) { return { a.x * s, a.y * s, a.z * s }; }
static HV hdiv(HV a, double s) { return hmul(a, 1.0 / s); }                       // vec3.rs:371-376
static double hlen(HV a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
static HV hunit(HV a) { return hdiv(a, hlen(a)); }                                // vec3.rs:107-109
static HV hcross(HV a, HV b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }

extern "C" int rtiow_camera_new(const double look_from[3], const double look_at[3], const double v_up[3], double v_fov_deg,
                                double aspect_ratio, double aperture, double focus_dist, rtiow_camera* out)
{
    if (!look_from || !look_at || !v_up || !out) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    const HV from = { look_from[0], look_from[1], look_from[2] }, at = { look_at[0], look_at[1], look_at[2] }, up = { v_up[0], v_up[1], v_up[2] };
    const double theta = v_fov_deg * (3.14159265358979323846264338327950288 / 180.0);   // f64::to_radians, camera.rs:25
    const double viewport_height = 2.0 * std::tan(theta / 2.0);
    const double viewport_width = aspect_ratio * viewport_height;
    const HV w = hunit(hsub(from, at));                                                   // camera.rs:29
    const HV u = hunit(hcross(up, w));
    const HV v = hcross(w, u);
    const HV horizontal = hmul(u, focus_dist * viewport_width);                           // camera.rs:33
    const HV vertical = hmul(v, focus_dist * viewport_height);
    const HV llc = hsub(hsub(hsub(from, hdiv(horizontal, 2.0)), hdiv(vertical, 2.0)), hmul(w, focus_dist));  // camera.rs:35
    auto put = [](double* d, HV a) { d[0] = a.x; d[1] = a.y; d[2] = a.z; };
    put(out->origin, from); put(out->lower_left_corner, llc); put(out->horizontal, horizontal); put(out->vertical, vertical);
    put(out->u, u); put(out->v, v); put(out->w, w);
    out->lens_radius = aperture / 2.0;
    return RTIOW_OK;
}

template <typename T> static CameraT<T> to_dev_camera(const rtiow_camera& c)
{
    CameraT<T> d;
    d.origin = mk<T>((T)c.origin[0], (T)c.origin[1], (T)c.origin[2]);
    d.llc_minus_origin = mk<T>((T)(c.lower_left_corner[0] - c.origin[0]), (T)(c.lower_left_corner[1] - c.origin[1]), (T)(c.lower_left_corner[2] - c.origin[2]));
    d.horizontal = mk<T>((T)c.horizontal[0], (T)c.horizontal[1], (T)c.horizontal[2]);
    d.vertical = mk<T>((T)c.vertical[0], (T)c.vertical[1], (T)c.vertical[2]);
    d.u = mk<T>((T)c.u[0], (T)c.u[1], (T)c.u[2]);
    d.v = mk<T>((T)c.v[0], (T)c.v[1], (T)c.v[2]);
    d.lens_radius = (T)c.lens_radius;
    return d;
}

extern "C" void rtiow_params_default(rtiow_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->width = 200; p->height = 133; p->spp = 100; p->max_depth = 50;     // main.rs:24-28 (200/1.5 truncates to 133)
    p->t_min = 0.0001;                                                    // main.rs:44
    p->seed = 1; p->alpha = 255;                                          // main.rs:137
    p->precision = RTIOW_PRECISION_F32; p->tile_rows = 1;
}

// ------------------------------------------------------------------------------------------------
// frame partition
// ------------------------------------------------------------------------------------------------
// tile height actually used: a tile taller than the frame is the whole frame (and (height + tile_rows - 1) cannot wrap)
static uint32_t tile_rows_of(const rtiow_params* p) { return std::min(p->tile_rows, p->height); }
static uint32_t rows_of_rank(uint32_t height, uint32_t tile_rows, uint32_t world, uint32_t rank)
{
    const uint32_t n_tiles = (height + tile_rows - 1) / tile_rows;
    uint32_t rows = 0;
    for (uint32_t tg = rank; tg < n_tiles; tg += world) rows += std::min(tile_rows, height - tg * tile_rows);
    return rows;
}
static uint32_t max_rows_per_rank(uint32_t height, uint32_t tile_rows, uint32_t world)
{
    const uint32_t n_tiles = (height + tile_rows - 1) / tile_rows;
    return ((n_tiles + world - 1) / world) * tile_rows;
}
static int check_params(const rtiow_params* p)
{
    if (!p) return fail(RTIOW_ERR_INVALID_ARG, "params is NULL");
    if (p->width < 2 || p->height < 2) return fail(RTIOW_ERR_INVALID_ARG, "width and height must be >= 2 (jitter divides by W-1, H-1: main.rs:131-132)");
    if (p->spp == 0) return fail(RTIOW_ERR_INVALID_ARG, "spp must be >= 1");
    if ((uint64_t)p->width * p->height > 0xfffffff0ull) return fail(RTIOW_ERR_INVALID_ARG, "frame too large");
    if (p->tile_rows == 0) return fail(RTIOW_ERR_INVALID_ARG, "tile_rows must be >= 1");
    if (p->precision > RTIOW_PRECISION_F64) return fail(RTIOW_ERR_INVALID_ARG, "unknown precision");
    if (!(p->t_min >= 0.0)) return fail(RTIOW_ERR_INVALID_ARG, "t_min must be >= 0");
    return RTIOW_OK;
}

extern "C" int rtiow_tile_buffer_bytes(const rtiow_params* p, int world, size_t* out)
{
    int rc = check_params(p); if (rc) return rc;
    if (world < 1 || !out) return fail(RTIOW_ERR_INVALID_ARG, "bad world/out");
    *out = (size_t)max_rows_per_rank(p->height, tile_rows_of(p), (uint32_t)world) * p->width * 4;
    return RTIOW_OK;
}

// ------------------------------------------------------------------------------------------------
// launch configuration
// ------------------------------------------------------------------------------------------------
// Which filter a scan runs.  F32: the tensor-core one when the scene qualifies (rtiow_scene_upload) and the caller did not ask
// otherwise, else the FP32 one with its table in shared memory (Smem; Wide: a table too large for 256-thread CTAs, beside the
// candidate lists of one wide CTA per SM) or read from global memory.  F64 tests every sphere.
enum class Scan { F64, Tensor, Smem, Wide, Global };
using UShape = UmmaShape<RT_UMMA_GROUPS, RT_UMMA_CHUNK>;
static size_t cand_bytes(int threads) { return (size_t)threads * RT_CAND_CAP * sizeof(uint16_t); }
struct ScanPlan {
    Scan scan;
    size_t scene_smem;      // shared memory of the scene: the FP32 table (Smem, Wide), the tensor kernels' whole layout (Tensor), else 0
    // dynamic shared memory of a CTA of `threads` threads: the FP32 filters add a candidate list per thread
    size_t smem(int threads) const { return scan == Scan::F64 || scan == Scan::Tensor ? scene_smem : scene_smem + cand_bytes(threads); }
};
static int plan_scan(const rtiow_ctx* c, const DeviceState& d, int precision, ScanPlan* plan)
{
    if (precision == RTIOW_PRECISION_F64) { *plan = { Scan::F64, 0 }; return RTIOW_OK; }
    if (d.scene.u_npad > 0 && c->scan_backend != RTIOW_SCAN_FP32) { *plan = { Scan::Tensor, UShape::smem_bytes(d.scene.u_npad) }; return RTIOW_OK; }
    if (c->scan_backend == RTIOW_SCAN_TENSOR)
        return fail(RTIOW_ERR_UNSUPPORTED, "RTIOW_SCAN_TENSOR requested but the scene does not qualify for the tensor-core filter (too many / too widely spread small spheres)");
    const size_t table = RT_TABLE_FLOATS(d.scene.np) * sizeof(float);
    if (table + cand_bytes(256) <= 56 * 1024) *plan = { Scan::Smem, table };
    else if (table + cand_bytes(512) <= 227 * 1024) *plan = { Scan::Wide, table };
    else *plan = { Scan::Global, 0 };
    return RTIOW_OK;
}

// more dynamic shared memory than the default 48 KB has to be allowed per kernel
template <typename K> static int allow_smem(K kernel, size_t smem)
{
    if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return RTIOW_OK;
}

// samples [begin, begin + count) of every pixel: the whole frame is {0, spp}; a progressive pass renders a slice and adds to the
// accumulators the earlier passes left (rtiow_render_progressive)
struct SampleRange { uint32_t begin, count; };

// Work is handed out in chunks of <= 64 samples of one pixel (two rounds of a warp's 32 lanes).  A fetch from the global
// counter takes up to 256 samples' worth of chunks, less on small frames (every warp of the persistent grid should draw
// >= 8 fetches: a 400x225@10 frame is only ~8 paths per lane) and towards the end of any frame (guided_div, rt_render.cuh).
template <typename T> static void size_fetch(RenderArgs<T>& a, int grid, int threads)
{
    const uint64_t n_warps = (uint64_t)grid * threads / 32;
    const uint64_t want = a.n_chunks / std::max<uint64_t>(1, n_warps * 8);
    const uint64_t cap = std::max<uint32_t>(1u, 256u / a.chunk_samples);
    a.chunks_per_fetch = (uint32_t)std::min<uint64_t>(cap, std::max<uint64_t>(1, want));
    a.guided_div = (uint32_t)std::max<uint64_t>(1, 2 * n_warps);
}

// a persistent render kernel: as many CTAs as fit on the SMs at once.  `views` is empty for a frame and the device array of the
// cameras for a batch of views (render_views_kernel)
template <typename T, typename K, typename... V> static int launch_persistent(K kernel, RenderArgs<T>& a, int threads, size_t smem, int sms, cudaStream_t st, V... views)
{
    int rc = allow_smem(kernel, smem); if (rc) return rc;
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) return fail(RTIOW_ERR_CUDA, "kernel does not fit on an SM (smem %zu)", smem);
    const int grid = per_sm * sms;
    size_fetch(a, grid, threads);
    kernel<<<grid, threads, smem, st>>>(a, views...);
    return RTIOW_OK;
}

// the render kernel of one scan arm: a frame's, or with kViews a batch of views' (the same loop, rt_render.cuh)
template <bool kViews, typename T, bool kSmem, int kThreads, int kMinCtas> static auto render_entry()
{
    if constexpr (kViews) return render_views_kernel<T, kSmem, kThreads, kMinCtas>;
    else return render_kernel<T, kSmem, kThreads, kMinCtas>;
}
template <bool kViews> static auto render_entry_umma()
{
    if constexpr (kViews) return render_views_kernel_umma<RT_UMMA_GROUPS, RT_UMMA_CHUNK>;
    else return render_kernel_umma<RT_UMMA_GROUPS, RT_UMMA_CHUNK>;
}

template <bool kViews, typename T, typename... V>
static int launch_render_kernel(const ScanPlan& plan, const DeviceState& d, RenderArgs<T>& a, cudaStream_t st, V... views)
{
    if constexpr (std::is_same<T, double>::value) {
        return launch_persistent(render_entry<kViews, double, false, 256, 2>(), a, 256, plan.smem(256), d.sms, st, views...);
    } else {
        switch (plan.scan) {
        case Scan::Tensor: {     // one CTA per SM (it owns all of TMEM), G groups of 128 rays + G issuer warps
            auto k = render_entry_umma<kViews>();
            const size_t smem = plan.smem(UShape::kRenderThreads);
            int rc = allow_smem(k, smem); if (rc) return rc;
            size_fetch(a, d.sms, UShape::kRayThreads);          // the work is shared among the ray threads, not the whole block
            k<<<d.sms, UShape::kRenderThreads, smem, st>>>(a, views...);
            return RTIOW_OK;
        }
        case Scan::Smem:         // 3 CTAs x 256 threads x 80 registers fills the 64K-register file
            return launch_persistent(render_entry<kViews, float, true, 256, 3>(), a, 256, plan.smem(256), d.sms, st, views...);
        case Scan::Wide:         // one CTA per SM, 24 warps at 80 registers (+2.5 % over 512 threads at 104) when their lists fit
            if (plan.smem(768) <= 227 * 1024) return launch_persistent(render_entry<kViews, float, true, 768, 1>(), a, 768, plan.smem(768), d.sms, st, views...);
            return launch_persistent(render_entry<kViews, float, true, 512, 1>(), a, 512, plan.smem(512), d.sms, st, views...);
        case Scan::Global:
            return launch_persistent(render_entry<kViews, float, false, 256, 4>(), a, 256, plan.smem(256), d.sms, st, views...);
        case Scan::F64:
            break;
        }
        return fail(RTIOW_ERR_INVALID_ARG, "an F64 scan plan for an F32 render");
    }
}

// where a device's epilogue stores its pixels: its rows in rank-local order into a tile buffer, or into their top-down places in
// a whole frame that may live on another GPU (fused quantise + gather: finalize_to_frame_kernel)
struct Dest { uint32_t* p; bool whole_frame; };

// n_views = 0: a frame (or a rank's rows of one) of camera *cam.  n_views > 0 (world 1): a batch of views, the cameras
// cam[0 .. n_views), rendered as one frame n_views * height rows tall whose epilogue writes the views' frames one after the other.
// *paths: the paths launched, local rows x width x samples.
template <typename T>
static int launch_render(const ScanPlan& plan, DeviceState& d, const rtiow_camera* cam, const rtiow_params* p, uint32_t rank, uint32_t world, SampleRange sr,
                         Dest dst, cudaStream_t st, uint32_t* launches, uint64_t* paths, uint32_t n_views)
{
    RenderArgs<T> a;
    a.scene = d.scene; a.cam = to_dev_camera<T>(*cam);
    a.width = p->width; a.height = p->height; a.spp = sr.count; a.smp_begin = sr.begin; a.max_depth = p->max_depth; a.t_min = (T)p->t_min; a.key = philox_key(p->seed);
    a.inv_wm1 = (T)(1.0 / (double)(p->width - 1)); a.inv_hm1 = (T)(1.0 / (double)(p->height - 1));
    a.rank = rank; a.world = world; a.tile_rows = tile_rows_of(p);
    a.local_rows = n_views ? n_views * p->height : rows_of_rank(p->height, tile_rows_of(p), world, rank);
    a.chunk_samples = std::min<uint32_t>(sr.count, 64u);
    a.chunks_per_pixel = (sr.count + a.chunk_samples - 1) / a.chunk_samples;
    a.chunks_per_fetch = std::max<uint32_t>(1u, 256u / a.chunk_samples);
    const uint64_t n_lp = (uint64_t)a.local_rows * p->width;
    a.n_chunks = n_lp * a.chunks_per_pixel;
    a.sample_cap = (T)std::min(1e9, (double)p->spp);        // the whole frame's spp: every pass of a progressive render adds the same
    a.saturate = p->spp > 65535u;
    *paths = n_lp * sr.count;
    CU(d.accum.resize(3 * n_lp));
    a.accum = d.accum.p; a.work_counter = d.counters.p; a.ray_counter = d.counters.p + 1;
    if (sr.begin == 0) CU(cudaMemsetAsync(d.accum.p, 0, 3 * n_lp * sizeof(unsigned long long), st));     // later passes add to the same sums
    CU(cudaMemsetAsync(d.counters.p, 0, 2 * sizeof(unsigned long long), st));
    if (n_lp == 0) return RTIOW_OK;
    d.last_backend = plan.scan == Scan::Tensor ? RTIOW_SCAN_TENSOR : RTIOW_SCAN_FP32;
    int rc;
    if (n_views) {              // the cameras go up in one copy; only a path's first ray reads its view's camera
        const size_t bytes = (size_t)n_views * sizeof(CameraT<T>);
        CU(d.cams_stage.resize(bytes)); CU(d.cams.resize(bytes));
        CameraT<T>* staged = reinterpret_cast<CameraT<T>*>(d.cams_stage.p);
        for (uint32_t v = 0; v < n_views; ++v) staged[v] = to_dev_camera<T>(cam[v]);
        CU(cudaMemcpyAsync(d.cams.p, staged, bytes, cudaMemcpyHostToDevice, st));
        rc = launch_render_kernel<true>(plan, d, a, st, reinterpret_cast<const CameraT<T>*>(d.cams.p));
    } else {
        rc = launch_render_kernel<false>(plan, d, a, st);
    }
    if (rc) return rc;
    CU(cudaGetLastError());
    if (dst.whole_frame)
        finalize_to_frame_kernel<<<(unsigned)((n_lp + 255) / 256), 256, 0, st>>>(d.accum.p, (uint32_t)n_lp, sr.begin + sr.count, p->alpha, p->width, tile_rows_of(p), world, rank, dst.p);
    else
        finalize_kernel<<<(unsigned)((n_lp + 255) / 256), 256, 0, st>>>(d.accum.p, (uint32_t)n_lp, sr.begin + sr.count, p->alpha, dst.p);
    CU(cudaGetLastError());
    *launches += 2;
    return RTIOW_OK;
}

// What one device launched for a call (render_step): where, between which events and how many paths (0 for a rank without
// rows), and the D2H copy of its frame when the call starts one.  A caller's buffer that is page-locked itself (cudaHostAlloc /
// cudaHostRegister, torch pin_memory) takes the DMA directly; pageable memory goes through the device's staging buffer, and
// finish_call copies it over after the stream synchronisation (0.3 ms for the 3.2 MB headline frame).
struct Part {
    DeviceState* d = nullptr; cudaStream_t st = nullptr; cudaEvent_t e0 = nullptr, e1 = nullptr;
    uint64_t paths = 0;
    uint8_t* out = nullptr; const uint8_t* staged = nullptr; size_t copy_bytes = 0;
    int start_copy(uint8_t* dst, const uint32_t* d_frame, size_t n)
    {
        out = dst; copy_bytes = n;
        if (!host_is_pinned(dst)) { CU(d->pinned.resize(n)); staged = d->pinned.p; }
        CU(cudaMemcpyAsync(staged ? d->pinned.p : dst, d_frame, n, cudaMemcpyDeviceToHost, st));
        return RTIOW_OK;
    }
    // the counters after the part's work into d->pinned_cnt: the last thing a call puts on the part's stream
    int read_counters() const
    {
        CU(cudaSetDevice(d->device));
        CU(cudaMemcpyAsync(d->pinned_cnt.p, d->counters.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        return RTIOW_OK;
    }
};

// One device's part of a frame: samples `sr` of the rows {y : (y / tile_rows) % world == rank}, quantised into `dst`, with the
// events e0 / e1 around the work and its kernel launches added to *launches.  n_views > 0: the batch of views cam[0 .. n_views)
// (launch_render).
static int render_step(const rtiow_ctx* c, DeviceState& d, const rtiow_camera* cam, const rtiow_params* p, uint32_t rank, uint32_t world, SampleRange sr,
                       Dest dst, cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1, uint32_t* launches, Part* part, uint32_t n_views = 0)
{
    if (!d.has_scene) return fail(RTIOW_ERR_INVALID_ARG, "no scene uploaded (call rtiow_scene_upload first)");
    CU(cudaSetDevice(d.device));
    ScanPlan plan;
    int rc = plan_scan(c, d, p->precision, &plan); if (rc) return rc;
    *part = Part{ &d, st, e0, e1 };
    CU(cudaEventRecord(e0, st));
    rc = plan.scan == Scan::F64 ? launch_render<double>(plan, d, cam, p, rank, world, sr, dst, st, launches, &part->paths, n_views)
                                : launch_render<float>(plan, d, cam, p, rank, world, sr, dst, st, launches, &part->paths, n_views);
    if (rc) return rc;
    CU(cudaEventRecord(e1, st));
    return RTIOW_OK;
}

// a frame on one device: its rank-local order IS top-down (and a batch of n_views views is their frames one after the other)
static int render_single(const rtiow_ctx* c, DeviceState& d, const rtiow_camera* cam, const rtiow_params* p, SampleRange sr, cudaStream_t st,
                         cudaEvent_t e0, cudaEvent_t e1, uint32_t* launches, Part* part, const uint32_t** d_frame, uint32_t n_views = 0)
{
    CU(d.tiles.resize((size_t)p->width * p->height * std::max<uint32_t>(n_views, 1)));
    int rc = render_step(c, d, cam, p, 0, 1, sr, Dest{ d.tiles.p, false }, st, e0, e1, launches, part, n_views); if (rc) return rc;
    *d_frame = d.tiles.p;
    return RTIOW_OK;
}

// the world tile buffers of a gather, one after the other in rank-local order, into the top-down frame
static int deinterleave(const uint32_t* gathered, const rtiow_params* p, uint32_t world, uint32_t* frame, cudaStream_t st)
{
    const size_t npx = (size_t)p->width * p->height;
    const size_t tile_px = (size_t)max_rows_per_rank(p->height, tile_rows_of(p), world) * p->width;
    deinterleave_kernel<<<(unsigned)((npx + 255) / 256), 256, 0, st>>>(gathered, p->width, p->height, tile_rows_of(p), world, tile_px, frame);
    CU(cudaGetLastError());
    return RTIOW_OK;
}

// what a render call reports; the scene's sphere count and the filter used come from device d
static rtiow_stats make_stats(const DeviceState& d, double kernel_ms, double total_ms, uint64_t paths, uint64_t rays, uint32_t launches, uint32_t n_gpus,
                              uint64_t h2d_bytes, uint64_t d2h_bytes)
{
    rtiow_stats s; memset(&s, 0, sizeof s);
    s.kernel_ms = kernel_ms; s.total_ms = total_ms; s.paths = paths; s.rays_traced = rays; s.sphere_tests = rays * (uint64_t)d.scene.n;
    s.h2d_bytes = h2d_bytes; s.d2h_bytes = d2h_bytes; s.kernel_launches = launches; s.n_gpus = n_gpus; s.scan_backend = (uint32_t)d.last_backend;
    return s;
}
static const uint64_t kCallH2D = sizeof(rtiow_camera) + sizeof(rtiow_params);     // a frame's only input: the camera and the params

static double now_ms()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// The end of a synchronous call: every part's counters are read back, its stream synchronised and its frame copy finished.
// *stats (when asked for) gets the slowest part's kernel time and the parts' summed paths and rays, and the scene and filter of
// the first part's device (make_stats).
static int finish_call(Part* parts, size_t n, double t0, uint32_t launches, uint32_t n_gpus, uint64_t h2d_bytes, uint64_t d2h_bytes, rtiow_stats* stats)
{
    for (size_t i = 0; i < n; ++i) { int rc = parts[i].read_counters(); if (rc) return rc; }
    float ms = 0; uint64_t paths = 0, rays = 0;
    for (size_t i = 0; i < n; ++i) {
        const Part& pt = parts[i];
        CU(cudaSetDevice(pt.d->device));
        CU(cudaStreamSynchronize(pt.st));
        if (pt.staged) memcpy(pt.out, pt.staged, pt.copy_bytes);
        float mp = 0; if (stats) CU(cudaEventElapsedTime(&mp, pt.e0, pt.e1));
        ms = std::max(ms, mp); paths += pt.paths; rays += pt.d->pinned_cnt.p[1];          // the slowest device's kernels
    }
    CU(cudaSetDevice(parts[0].d->device));
    if (stats) *stats = make_stats(*parts[0].d, ms, now_ms() - t0, paths, rays, launches, n_gpus, h2d_bytes, d2h_bytes);
    return RTIOW_OK;
}

// shared body of the two per-rank entry points: this rank's rows into a tile buffer (rank-local order), or — with `to_frame` —
// straight into their top-down place in a whole frame that may live on another GPU (finalize_to_frame_kernel)
static int render_rank(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, int rank, int world, void* dst, bool to_frame, void* stream,
                       rtiow_stats* stats)
{
    if (!c || !cam || !dst) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_params(p); if (rc) return rc;
    if (world < 1 || rank < 0 || rank >= world) return fail(RTIOW_ERR_INVALID_ARG, "bad rank/world");
    DeviceState& d = c->dev[0];
    CU(cudaSetDevice(d.device));
    cudaStream_t st = stream ? (cudaStream_t)stream : d.stream;
    const double t0 = now_ms();
    uint32_t launches = 0;
    Part part;
    rc = render_step(c, d, cam, p, (uint32_t)rank, (uint32_t)world, SampleRange{ 0u, p->spp }, Dest{ (uint32_t*)dst, to_frame }, st, d.ev0, d.ev1, &launches, &part);
    if (rc) return rc;
    return stats ? finish_call(&part, 1, t0, launches, 1, 0, 0, stats) : RTIOW_OK;      // without stats the call stays asynchronous
}

extern "C" int rtiow_render_tiles_device(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, int rank, int world, void* d_tiles,
                                         void* stream, rtiow_stats* stats)
{
    return render_rank(c, cam, p, rank, world, d_tiles, false, stream, stats);
}

// The gather fused into the epilogue, for one-process-per-GPU jobs: d_frame is the WHOLE top-down frame (4*width*height bytes),
// typically rank 0's buffer mapped into this process (CUDA IPC / torch symmetric memory); this rank's pixels are quantised and
// stored straight into their rows of it — over NVLink when the buffer is remote.  No tile buffer, no all-gather, no
// de-interleave; the caller only needs a barrier before rank 0 reads the frame.
extern "C" int rtiow_render_to_frame_device(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, int rank, int world, void* d_frame,
                                            void* stream, rtiow_stats* stats)
{
    return render_rank(c, cam, p, rank, world, d_frame, true, stream, stats);
}

extern "C" int rtiow_deinterleave_device(rtiow_ctx* c, const void* d_gathered, const rtiow_params* p, int world, void* d_frame, void* stream)
{
    if (!c || !d_gathered || !d_frame) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_params(p); if (rc) return rc;
    if (world < 1) return fail(RTIOW_ERR_INVALID_ARG, "bad world");
    DeviceState& d = c->dev[0];
    CU(cudaSetDevice(d.device));
    return deinterleave((const uint32_t*)d_gathered, p, (uint32_t)world, (uint32_t*)d_frame, stream ? (cudaStream_t)stream : d.stream);
}

// THE drop-in call (main.rs:122-145)
// One launch per device over the sample range `sr` + the quantise/gather epilogue + the frame to host memory.
static int render_frame(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, SampleRange sr, uint8_t* out_rgba, rtiow_stats* stats)
{
    int rc = RTIOW_OK;
    const double t0 = now_ms();
    const uint32_t world = (uint32_t)c->dev.size();
    const size_t frame_bytes = (size_t)p->width * p->height * 4;
    const size_t tile_px = (size_t)max_rows_per_rank(p->height, tile_rows_of(p), world) * p->width;
    DeviceState& d0 = c->dev[0];
    uint32_t launches = 0;
    CU(cudaSetDevice(d0.device));
    std::vector<Part> parts(world);
    const uint32_t* d_final = nullptr;
    if (world == 1) {
        rc = render_single(c, d0, cam, p, sr, d0.stream, d0.ev0, d0.ev1, &launches, &parts[0], &d_final); if (rc) return rc;
    } else {
        // interleaved row tiles on every GPU.  Three gathers:
        //   fused (default with NVLink peer access, every B200 box): each rank's epilogue stores its pixels straight into device
        //     0's top-down frame (finalize_to_frame_kernel): compute and gather are one kernel, nothing is staged;
        //   NCCL (rtiow_ctx_set_gather(RTIOW_GATHER_NCCL); SURVEY §8e): ncclCommInitAll once, then per frame one grouped
        //     ncclAllGather of the equal-size (padded) tile buffers + the de-interleave kernel on device 0;
        //   without peer access and without NCCL: tile buffers + cudaMemcpyPeerAsync + de-interleave.
        const bool use_nccl = c->gather == RTIOW_GATHER_NCCL;
        if (c->gather == RTIOW_GATHER_FUSED && !c->peer_ok) return fail(RTIOW_ERR_UNSUPPORTED, "RTIOW_GATHER_FUSED needs peer access from every device to device 0");
        const bool fused = !use_nccl && c->peer_ok;
        if (use_nccl && c->comms.empty()) {
            rc = nccl_load(); if (rc) return rc;
            std::vector<int> devs; for (auto& d : c->dev) devs.push_back(d.device);
            c->comms.assign(world, nullptr);
            ncclResult_t r = g_nccl.CommInitAll(c->comms.data(), (int)world, devs.data());
            if (r != ncclSuccess) { c->comms.clear(); return fail(RTIOW_ERR_NCCL, "ncclCommInitAll(%u devices) -> %s", world, g_nccl.GetErrorString(r)); }
        }
        CU(d0.frame.resize((size_t)p->width * p->height));
        if (!fused) CU(d0.gathered.resize(tile_px * world));
        for (uint32_t r = 0; r < world; ++r) {
            DeviceState& d = c->dev[r];
            CU(cudaSetDevice(d.device));
            Dest dst{ d0.frame.p, true };
            if (use_nccl) { CU(d.tiles.resize(tile_px)); CU(d.gathered.resize(tile_px * world)); dst = Dest{ d.tiles.p, false }; }
            else if (!fused) { if (r == 0) dst = Dest{ d0.gathered.p, false }; else { CU(d.tiles.resize(tile_px)); dst = Dest{ d.tiles.p, false }; } }
            rc = render_step(c, d, cam, p, r, world, sr, dst, d.stream, d.ev0, d.ev1, &launches, &parts[r]); if (rc) return rc;
            if (r != 0 && !use_nccl) {
                if (!fused) {
                    const size_t bytes = (size_t)rows_of_rank(p->height, tile_rows_of(p), world, r) * p->width * 4;
                    CU(cudaMemcpyPeerAsync(d0.gathered.p + tile_px * r, d0.device, d.tiles.p, d.device, bytes, d.stream));
                }
                CU(cudaEventRecord(d.ev_done, d.stream));
            }
        }
        if (use_nccl) {
            NC(g_nccl.GroupStart());
            for (uint32_t r = 0; r < world; ++r) {
                DeviceState& d = c->dev[r];
                ncclResult_t e = g_nccl.AllGather(d.tiles.p, d.gathered.p, tile_px * 4, ncclUint8, c->comms[r], d.stream);
                if (e != ncclSuccess) { g_nccl.GroupEnd(); return fail(RTIOW_ERR_NCCL, "ncclAllGather(rank %u) -> %s", r, g_nccl.GetErrorString(e)); }
            }
            NC(g_nccl.GroupEnd());
        }
        CU(cudaSetDevice(d0.device));
        if (!use_nccl) for (uint32_t r = 1; r < world; ++r) CU(cudaStreamWaitEvent(d0.stream, c->dev[r].ev_done, 0));
        if (!fused) {
            rc = deinterleave(d0.gathered.p, p, world, d0.frame.p, d0.stream); if (rc) return rc;
            ++launches;
        }
        char note[160];
        snprintf(note, sizeof note, "one process, %u GPUs: %s", world, fused ? "epilogue stores into device 0's frame over NVLink peer memory (fused gather)"
                 : use_nccl ? "tile buffers + grouped ncclAllGather (ncclCommInitAll) + de-interleave" : "tile buffers + cudaMemcpyPeerAsync + de-interleave");
        c->gather_note = note;
        d_final = d0.frame.p;
    }
    rc = parts[0].start_copy(out_rgba, d_final, frame_bytes); if (rc) return rc;
    return finish_call(parts.data(), world, t0, launches, world, kCallH2D, frame_bytes + 16, stats);
}

extern "C" int rtiow_render(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, uint8_t* out_rgba, rtiow_stats* stats)
{
    if (!c || !cam || !out_rgba) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_params(p); if (rc) return rc;
    return render_frame(c, cam, p, SampleRange{ 0u, p->spp }, out_rgba, stats);
}

// Many cameras of one scene (turntables, stereo pairs, camera sweeps) in one render launch per device: CTA start-up, the
// end-of-frame tail, the memsets, the epilogue, the copy and the synchronisation are paid once per batch instead of once per
// view.  A device renders its views as one frame n_views * height rows tall in which every row keeps its own view's pixel keys
// (rt_render.cuh, assign_work), so frame v is byte-identical to rtiow_render(cams[v]).  An n-GPU ctx gives device r the whole
// views [r K / n, (r + 1) K / n), copied straight into their place in out_rgba: no gather.
extern "C" int rtiow_render_views(rtiow_ctx* c, const rtiow_camera* cams, uint32_t n_views, const rtiow_params* p, uint8_t* out_rgba, rtiow_stats* stats)
{
    if (!c || !cams || !out_rgba) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_params(p); if (rc) return rc;
    if (n_views == 0) return fail(RTIOW_ERR_INVALID_ARG, "n_views must be >= 1");
    if ((uint64_t)n_views * p->width * p->height > 0xfffffff0ull) return fail(RTIOW_ERR_INVALID_ARG, "batch too large: n_views * width * height must be <= 0xfffffff0");
    if (c->world > 1) return fail(RTIOW_ERR_UNSUPPORTED, "rtiow_render_views: a rank ctx with world > 1 renders collective frames (rtiow_render_rank), not batches of views");
    const double t0 = now_ms();
    const uint32_t n_dev = (uint32_t)c->dev.size();
    const size_t frame_bytes = (size_t)p->width * p->height * 4;
    std::vector<Part> parts;                                // of the devices that render: the first one's scene and scan backend go into the stats
    uint32_t launches = 0;
    for (uint32_t r = 0; r < n_dev; ++r) {
        const uint32_t v0 = (uint32_t)((uint64_t)r * n_views / n_dev), v1 = (uint32_t)((uint64_t)(r + 1) * n_views / n_dev);
        if (v0 == v1) continue;                             // more devices than views
        DeviceState& d = c->dev[r];
        CU(cudaSetDevice(d.device));
        const uint32_t* d_frames = nullptr;
        Part part;
        rc = render_single(c, d, cams + v0, p, SampleRange{ 0u, p->spp }, d.stream, d.ev0, d.ev1, &launches, &part, &d_frames, v1 - v0); if (rc) return rc;
        rc = part.start_copy(out_rgba + v0 * frame_bytes, d_frames, (v1 - v0) * frame_bytes); if (rc) return rc;
        parts.push_back(part);
    }
    return finish_call(parts.data(), parts.size(), t0, launches, n_dev, (uint64_t)n_views * sizeof(rtiow_camera) + sizeof(rtiow_params),
                       (uint64_t)n_views * frame_bytes + 16 * parts.size(), stats);
}

// The per-pass preview the reference gets from its progress bar and piston window (main.rs:120-124,151-171): the spp samples
// are rendered in n_passes slices; after each, the frame so far (quantised with the samples done so far, vec3.rs:404-420)
// is handed to the callback.  The accumulators are integer sums over the same (pixel, sample) keys, so the last frame is
// bit-identical to rtiow_render's, and the frame after k passes to rtiow_render with spp = samples done.
extern "C" int rtiow_render_progressive(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, uint32_t n_passes, rtiow_progress_fn on_pass,
                                        void* user, uint8_t* out_rgba, rtiow_stats* stats)
{
    if (!c || !cam || !out_rgba) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_params(p); if (rc) return rc;
    if (n_passes == 0) return fail(RTIOW_ERR_INVALID_ARG, "n_passes must be >= 1");
    n_passes = std::min<uint32_t>(n_passes, p->spp);
    rtiow_stats total; memset(&total, 0, sizeof total);
    const double t0 = now_ms();
    uint32_t done = 0;
    for (uint32_t k = 0; k < n_passes; ++k) {
        const uint32_t upto = (uint32_t)(((uint64_t)p->spp * (k + 1)) / n_passes);      // passes differ by at most one sample
        rtiow_stats st;
        rc = render_frame(c, cam, p, SampleRange{ done, upto - done }, out_rgba, &st); if (rc) return rc;
        done = upto;
        total.kernel_ms += st.kernel_ms; total.paths += st.paths; total.rays_traced += st.rays_traced; total.sphere_tests += st.sphere_tests;
        total.h2d_bytes += st.h2d_bytes; total.d2h_bytes += st.d2h_bytes; total.kernel_launches += st.kernel_launches; total.n_gpus = st.n_gpus; total.scan_backend = st.scan_backend;
        if (on_pass && on_pass(user, k + 1, n_passes, done, out_rgba) != 0 && k + 1 < n_passes) {
            total.total_ms = now_ms() - t0;
            if (stats) *stats = total;
            return fail(RTIOW_ERR_CANCELLED, "cancelled by the progress callback after pass %u of %u (%u of %u spp)", k + 1, n_passes, done, p->spp);
        }
    }
    total.total_ms = now_ms() - t0;
    if (stats) *stats = total;
    return RTIOW_OK;
}

// ------------------------------------------------------------------------------------------------
// one process per GPU (rtiow_ctx_create_rank): render this rank's row tiles and gather INSIDE the library.  The reference's
// gather is collect() at main.rs:139 (rows are the unit of work, main.rs:122-123).
// ------------------------------------------------------------------------------------------------
// 1-int all-reduce, stream-ordered after whatever each rank enqueued before it: when it completes on a rank, every rank's
// earlier work on its stream — the peer stores of its epilogue included — has completed
static int nccl_barrier(rtiow_ctx* c, cudaStream_t st)
{
    NC(g_nccl.AllReduce(c->d_flag, c->d_flag + 1, 1, ncclInt32, ncclSum, c->comm, st));
    return RTIOW_OK;
}
// min over ranks of a host value (agreement votes; synchronises the stream)
static int nccl_vote_min(rtiow_ctx* c, int mine, int* all, cudaStream_t st)
{
    CU(cudaMemcpyAsync(c->d_flag, &mine, sizeof(int), cudaMemcpyHostToDevice, st));
    NC(g_nccl.AllReduce(c->d_flag, c->d_flag + 1, 1, ncclInt32, ncclMin, c->comm, st));
    CU(cudaMemcpyAsync(all, c->d_flag + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return RTIOW_OK;
}

// The fused gather across processes: rank 0 owns a double-buffered top-down frame; its CUDA IPC handle travels to the other
// ranks in an ncclBroadcast and they map it (NVLink peer memory).  Collective: every rank calls it with the same frame size.
static int ensure_ipc_frame(rtiow_ctx* c, size_t npx, cudaStream_t st)
{
    if (c->ipc_state == -1 || (c->ipc_state == 1 && c->ipc_frame_px == npx)) return RTIOW_OK;
    CU(cudaStreamSynchronize(st));
    drop_ipc_frame(c);
    int ok = 1;
    cudaIpcMemHandle_t h; memset(&h, 0, sizeof h);
    if (c->rank == 0) {
        if (cudaMalloc(&c->ipc_frame, 2 * npx * sizeof(uint32_t)) != cudaSuccess) { cudaGetLastError(); c->ipc_frame = nullptr; ok = 0; }
        else if (cudaIpcGetMemHandle(&h, c->ipc_frame) != cudaSuccess) { cudaGetLastError(); ok = 0; }
        c->ipc_owner = true;
    }
    unsigned char* d_h = nullptr;
    CU(cudaMalloc(&d_h, sizeof h));
    cudaMemcpyAsync(d_h, &h, sizeof h, cudaMemcpyHostToDevice, st);
    ncclResult_t r = g_nccl.Broadcast(d_h, d_h, sizeof h, ncclUint8, 0, c->comm, st);
    cudaMemcpyAsync(&h, d_h, sizeof h, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(d_h);
    if (r != ncclSuccess) return fail(RTIOW_ERR_NCCL, "ncclBroadcast(IPC handle) -> %s", g_nccl.GetErrorString(r));
    if (e != cudaSuccess) return fail(RTIOW_ERR_CUDA, "IPC handle exchange -> %s", cudaGetErrorString(e));
    if (c->rank != 0) {
        c->ipc_owner = false;
        if (cudaIpcOpenMemHandle((void**)&c->ipc_frame, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); c->ipc_frame = nullptr; ok = 0; }
    }
    int all = 0;
    int rc = nccl_vote_min(c, ok, &all, st); if (rc) return rc;
    if (!all) {         // some rank could not map the frame (no peer access / IPC across containers): every rank falls back together
        drop_ipc_frame(c);
        c->ipc_state = -1;
    } else { c->ipc_state = 1; c->ipc_frame_px = npx; c->ipc_parity = 0; }
    return RTIOW_OK;
}

// tile + gathered buffers of the NCCL gather; allocated with ncclMemAlloc and registered as a symmetric window when the
// library offers it (NCCL >= 2.27: zero-copy all-gather over NVLink), plain cudaMalloc otherwise.  Collective; once buffers of
// tile_px are ready, from either allocator, later frames of that size go straight on (no synchronisation, no vote).
static int ensure_nccl_buffers(rtiow_ctx* c, size_t tile_px, cudaStream_t st)
{
    DeviceState& d = c->dev[0];
    if (c->nccl_tile_px == tile_px) return RTIOW_OK;
    CU(cudaStreamSynchronize(st));
    drop_nccl_buffers(c);
    int ok = 0;
    if (g_nccl.MemAlloc && g_nccl.MemFree && g_nccl.CommWindowRegister && g_nccl.CommWindowDeregister) {
        ok = g_nccl.MemAlloc((void**)&c->nccl_tiles, tile_px * 4) == ncclSuccess && g_nccl.MemAlloc((void**)&c->nccl_gathered, tile_px * 4 * c->world) == ncclSuccess;
        if (!ok) cudaGetLastError();
    }
    int all = 0;
    int rc = nccl_vote_min(c, ok, &all, st); if (rc) return rc;
    if (all) {
        ncclWindow_t wt = nullptr, wg = nullptr;
        const bool reg = g_nccl.CommWindowRegister(c->comm, c->nccl_tiles, tile_px * 4, &wt, NCCL_WIN_COLL_SYMMETRIC) == ncclSuccess &&
                         g_nccl.CommWindowRegister(c->comm, c->nccl_gathered, tile_px * 4 * c->world, &wg, NCCL_WIN_COLL_SYMMETRIC) == ncclSuccess;
        c->win_tiles = wt; c->win_gathered = wg; c->windows_registered = reg && wt && wg;
        if (!reg) cudaGetLastError();
    } else {
        drop_nccl_buffers(c);
        CU(d.tiles.resize(tile_px)); CU(d.gathered.resize(tile_px * c->world));
    }
    c->nccl_tile_px = tile_px;
    return RTIOW_OK;
}

static int render_rank_impl(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, uint8_t* out_rgba, const void** d_frame_out, rtiow_stats* stats,
                            bool enqueue_only)
{
    if (!c || !cam) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    int rc = check_params(p); if (rc) return rc;
    if (c->dev.size() != 1) return fail(RTIOW_ERR_INVALID_ARG, "rtiow_render_rank needs a ctx from rtiow_ctx_create_rank (one device per process)");
    if (c->rank == 0 && !out_rgba && !d_frame_out) return fail(RTIOW_ERR_INVALID_ARG, "rank 0 needs out_rgba (host) or d_frame (device)");
    DeviceState& d = c->dev[0];
    CU(cudaSetDevice(d.device));
    cudaStream_t st = d.stream;
    const double t0 = now_ms();
    const uint32_t world = (uint32_t)c->world, rank = (uint32_t)c->rank;
    const size_t npx = (size_t)p->width * p->height, frame_bytes = npx * 4;
    const size_t tile_px = (size_t)max_rows_per_rank(p->height, tile_rows_of(p), world) * p->width;
    uint32_t launches = 0;
    const uint32_t* d_final = nullptr;
    // the events around the render kernel: the ctx's pair, or — for a frame that is only enqueued — the next pair of the ring
    cudaEvent_t e0 = d.ev0, e1 = d.ev1;
    if (enqueue_only) {
        if (d.ring_used >= 1024) return fail(RTIOW_ERR_INVALID_ARG, "1024 frames enqueued: call rtiow_ctx_synchronize before enqueuing more");
        if (d.ring_used == d.ring.size()) {
            std::pair<cudaEvent_t, cudaEvent_t> ev{ nullptr, nullptr };
            CU(cudaEventCreate(&ev.first)); CU(cudaEventCreate(&ev.second));
            d.ring.push_back(ev);
        }
        e0 = d.ring[d.ring_used].first; e1 = d.ring[d.ring_used].second;
    }
    Part part;
    bool frame_here = true;                                 // d_final holds the whole frame on THIS rank
    if (world == 1) {
        rc = render_single(c, d, cam, p, SampleRange{ 0u, p->spp }, st, e0, e1, &launches, &part, &d_final); if (rc) return rc;
        c->gather_note = "single GPU: no gather";
    } else {
        bool fused = false;
        if (c->gather != RTIOW_GATHER_NCCL) {
            rc = ensure_ipc_frame(c, npx, st); if (rc) return rc;
            fused = c->ipc_state == 1;
            if (c->gather == RTIOW_GATHER_FUSED && !fused)
                return fail(RTIOW_ERR_UNSUPPORTED, "RTIOW_GATHER_FUSED: rank 0's frame could not be mapped into every rank (CUDA IPC / peer access)");
        }
        char note[256];
        if (fused) {
            // every rank's epilogue stores its rows straight into rank 0's frame (NVLink peer memory); the 1-int all-reduce after
            // it is the frame-complete barrier.  Two frames alternate, so rank 0's copy-out of frame k is ordered (by its stream
            // and the barrier of frame k+1) before anybody writes that buffer again in frame k+2.
            uint32_t* fr = c->ipc_frame + (size_t)(c->ipc_parity & 1u) * npx; c->ipc_parity ^= 1u;
            rc = render_step(c, d, cam, p, rank, world, SampleRange{ 0u, p->spp }, Dest{ fr, true }, st, e0, e1, &launches, &part); if (rc) return rc;
            rc = nccl_barrier(c, st); if (rc) return rc;
            d_final = fr; frame_here = rank == 0;
            snprintf(note, sizeof note, "one process per GPU x%u: epilogue stores into rank 0's frame over NVLink (CUDA IPC mapping made inside librtiow_cuda.so) + "
                     "1-int ncclAllReduce as the frame-complete barrier (NCCL %s)", world, g_nccl.version);
        } else {
            rc = ensure_nccl_buffers(c, tile_px, st); if (rc) return rc;
            uint32_t* tiles = c->nccl_tiles ? c->nccl_tiles : d.tiles.p;
            uint32_t* gathered = c->nccl_gathered ? c->nccl_gathered : d.gathered.p;
            CU(d.frame.resize(npx));
            rc = render_step(c, d, cam, p, rank, world, SampleRange{ 0u, p->spp }, Dest{ tiles, false }, st, e0, e1, &launches, &part); if (rc) return rc;
            NC(g_nccl.AllGather(tiles, gathered, tile_px * 4, ncclUint8, c->comm, st));      // one per frame, equal (padded) counts: SURVEY §8(e)
            rc = deinterleave(gathered, p, world, d.frame.p, st); if (rc) return rc;
            ++launches;
            d_final = d.frame.p;
            snprintf(note, sizeof note, "one process per GPU x%u: tile buffers + ncclAllGather inside librtiow_cuda.so (NCCL %s%s) + de-interleave", world,
                     g_nccl.version, c->windows_registered ? ", buffers from ncclMemAlloc registered as a symmetric window" : "");
        }
        c->gather_note = note;
    }
    if (d_frame_out) *d_frame_out = frame_here ? d_final : nullptr;
    if (out_rgba && frame_here) { rc = part.start_copy(out_rgba, d_final, frame_bytes); if (rc) return rc; }
    if (enqueue_only) {                                     // no host synchronisation: rtiow_ctx_synchronize collects the stats
        rc = part.read_counters(); if (rc) return rc;
        ++d.ring_used;
        d.enq_paths = part.paths; d.enq_launches += launches; d.enq_world = world;
        return RTIOW_OK;
    }
    return finish_call(&part, 1, t0, launches, world, kCallH2D, part.copy_bytes + 16, stats);
}

extern "C" int rtiow_render_rank(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, uint8_t* out_rgba, rtiow_stats* stats)
{
    return render_rank_impl(c, cam, p, out_rgba, nullptr, stats, false);
}
extern "C" int rtiow_render_rank_device(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, const void** d_frame, rtiow_stats* stats)
{
    if (!d_frame) return fail(RTIOW_ERR_INVALID_ARG, "d_frame is NULL");
    return render_rank_impl(c, cam, p, nullptr, d_frame, stats, false);
}

// Frames back to back without a host round trip per frame (an animation, a bench's timed loop): the render kernel, the epilogue /
// gather and the frame-complete barrier are enqueued on the ctx's stream and the call returns.
extern "C" int rtiow_render_rank_enqueue(rtiow_ctx* c, const rtiow_camera* cam, const rtiow_params* p, const void** d_frame)
{
    if (!d_frame) return fail(RTIOW_ERR_INVALID_ARG, "d_frame is NULL");
    return render_rank_impl(c, cam, p, nullptr, d_frame, nullptr, true);
}
extern "C" int rtiow_ctx_synchronize(rtiow_ctx* c, rtiow_stats* stats)
{
    if (!c) return fail(RTIOW_ERR_INVALID_ARG, "ctx is NULL");
    if (c->dev.size() != 1) return fail(RTIOW_ERR_INVALID_ARG, "rtiow_ctx_synchronize needs a one-device ctx (rtiow_ctx_create_rank)");
    DeviceState& d = c->dev[0];
    CU(cudaSetDevice(d.device));
    CU(cudaStreamSynchronize(d.stream));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        double sum = 0;
        for (size_t i = 0; i < d.ring_used; ++i) { float ms = 0; CU(cudaEventElapsedTime(&ms, d.ring[i].first, d.ring[i].second)); sum += ms; }
        // the mean kernel time of the frames enqueued since the last synchronize; paths and rays of the last one
        if (d.ring_used)
            *stats = make_stats(d, sum / (double)d.ring_used, 0.0, d.enq_paths, d.pinned_cnt.p[1], d.enq_launches, d.enq_world, kCallH2D * d.ring_used, 16 * d.ring_used);
    }
    d.ring_used = 0; d.enq_launches = 0;
    return RTIOW_OK;
}

// ------------------------------------------------------------------------------------------------
// unit-level batches
// ------------------------------------------------------------------------------------------------
struct Scratch {
    std::vector<void*> ptrs; cudaStream_t st;
    explicit Scratch(cudaStream_t s) : st(s) {}
    ~Scratch() { for (void* p : ptrs) cudaFree(p); }
    template <typename U> cudaError_t in(const U* host, size_t n, U** dev)
    {
        *dev = nullptr;
        cudaError_t e = cudaMalloc((void**)dev, std::max<size_t>(n, 1) * sizeof(U)); if (e) return e;
        ptrs.push_back(*dev);
        if (n) e = cudaMemcpyAsync(*dev, host, n * sizeof(U), cudaMemcpyHostToDevice, st);
        return e;
    }
    template <typename U> cudaError_t out(size_t n, U** dev)
    {
        *dev = nullptr;
        cudaError_t e = cudaMalloc((void**)dev, std::max<size_t>(n, 1) * sizeof(U)); if (e) return e;
        ptrs.push_back(*dev);
        return cudaMemsetAsync(*dev, 0, std::max<size_t>(n, 1) * sizeof(U), st);
    }
    template <typename U> cudaError_t back(U* host, const U* dev, size_t n) { return n ? cudaMemcpyAsync(host, dev, n * sizeof(U), cudaMemcpyDeviceToHost, st) : cudaSuccess; }
};
#define BATCH_PROLOGUE()                                                                     \
    if (!c) return fail(RTIOW_ERR_INVALID_ARG, "ctx is NULL");                               \
    if (n < 0) return fail(RTIOW_ERR_INVALID_ARG, "n < 0");                                  \
    if (precision != RTIOW_PRECISION_F32 && precision != RTIOW_PRECISION_F64) return fail(RTIOW_ERR_INVALID_ARG, "unknown precision"); \
    DeviceState& d = c->dev[0];                                                              \
    CU(cudaSetDevice(d.device));                                                             \
    Scratch S(d.stream);                                                                     \
    const unsigned grid = (unsigned)((n + 255) / 256);                                       \
    (void)grid;
#define N3 ((size_t)n * 3)

extern "C" int rtiow_sphere_hit_batch(rtiow_ctx* c, int precision, int64_t n, const double* center, const double* radius, const double* orig,
                                      const double* dir, const double* t_min, const double* t_max, int32_t* hit, double* t, double* p,
                                      double* normal, int32_t* front_face)
{
    BATCH_PROLOGUE();
    if (!center || !radius || !orig || !dir || !t_min || !t_max || !hit || !t || !p || !normal || !front_face) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    if (n == 0) return RTIOW_OK;
    double *dc, *dr, *dor, *dd, *dtn, *dtx, *dt, *dp, *dn; int32_t *dh, *dff;
    CU(S.in(center, N3, &dc)); CU(S.in(radius, n, &dr)); CU(S.in(orig, N3, &dor)); CU(S.in(dir, N3, &dd)); CU(S.in(t_min, n, &dtn)); CU(S.in(t_max, n, &dtx));
    CU(S.out(n, &dh)); CU(S.out(n, &dt)); CU(S.out(N3, &dp)); CU(S.out(N3, &dn)); CU(S.out(n, &dff));
    if (precision == RTIOW_PRECISION_F64) sphere_hit_kernel<double><<<grid, 256, 0, d.stream>>>(n, dc, dr, dor, dd, dtn, dtx, dh, dt, dp, dn, dff);
    else sphere_hit_kernel<float><<<grid, 256, 0, d.stream>>>(n, dc, dr, dor, dd, dtn, dtx, dh, dt, dp, dn, dff);
    CU(cudaGetLastError());
    CU(S.back(hit, dh, n)); CU(S.back(t, dt, n)); CU(S.back(p, dp, N3)); CU(S.back(normal, dn, N3)); CU(S.back(front_face, dff, n));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_hitlist_batch(rtiow_ctx* c, int precision, int64_t n, const double* orig, const double* dir, double t_min, int32_t* hit,
                                   int32_t* index, double* t, double* p, double* normal, int32_t* front_face)
{
    BATCH_PROLOGUE();
    if (!d.has_scene) return fail(RTIOW_ERR_INVALID_ARG, "no scene uploaded");
    if (!orig || !dir || !hit || !index || !t || !p || !normal || !front_face) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    ScanPlan plan;
    int rc = plan_scan(c, d, precision, &plan); if (rc) return rc;
    if (n == 0) return RTIOW_OK;
    double *dor, *dd, *dt, *dp, *dn; int32_t *dh, *di, *dff;
    CU(S.in(orig, N3, &dor)); CU(S.in(dir, N3, &dd));
    CU(S.out(n, &dh)); CU(S.out(n, &di)); CU(S.out(n, &dt)); CU(S.out(N3, &dp)); CU(S.out(N3, &dn)); CU(S.out(n, &dff));
    // one ray per thread, `rays` of them in a CTA of `threads`
    auto launch = [&](auto k, int rays, int threads) -> int {
        const size_t smem = plan.smem(threads);
        int rc = allow_smem(k, smem); if (rc) return rc;
        k<<<(unsigned)((n + rays - 1) / rays), threads, smem, d.stream>>>(d.scene, n, dor, dd, t_min, dh, di, dt, dp, dn, dff);
        return RTIOW_OK;
    };
    switch (plan.scan) {
    case Scan::F64: rc = launch(hitlist_kernel<double, false, 256>, 256, 256); break;
    case Scan::Tensor: rc = launch(hitlist_kernel_umma<RT_UMMA_GROUPS, RT_UMMA_CHUNK>, UShape::kRayThreads, UShape::kThreads); break;
    case Scan::Smem: rc = launch(hitlist_kernel<float, true, 256>, 256, 256); break;
    case Scan::Wide: rc = launch(hitlist_kernel<float, true, 512>, 512, 512); break;
    case Scan::Global: rc = launch(hitlist_kernel<float, false, 256>, 256, 256); break;
    }
    if (rc) return rc;
    CU(cudaGetLastError());
    CU(S.back(hit, dh, n)); CU(S.back(index, di, n)); CU(S.back(t, dt, n)); CU(S.back(p, dp, N3)); CU(S.back(normal, dn, N3)); CU(S.back(front_face, dff, n));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_scatter_batch(rtiow_ctx* c, int precision, int64_t n, const int32_t* kind, const double* albedo, const double* param,
                                   const double* r_orig, const double* r_dir, const double* p, const double* normal, const int32_t* front_face,
                                   const double* sample, int32_t* some, double* attenuation, double* s_orig, double* s_dir)
{
    BATCH_PROLOGUE();
    if (!kind || !albedo || !param || !r_orig || !r_dir || !p || !normal || !front_face || !sample || !some || !attenuation || !s_orig || !s_dir)
        return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    if (n == 0) return RTIOW_OK;
    for (int64_t i = 0; i < n; ++i) if (kind[i] < 0 || kind[i] > RTIOW_MAT_DIELECTRIC) return fail(RTIOW_ERR_UNSUPPORTED, "item %lld: material kind %d", (long long)i, kind[i]);
    int32_t *dk, *dff, *dsome; double *da, *dpar, *dro, *drd, *dp, *dn, *dsm, *datt, *dso, *dsd;
    CU(S.in(kind, n, &dk)); CU(S.in(albedo, N3, &da)); CU(S.in(param, n, &dpar)); CU(S.in(r_orig, N3, &dro)); CU(S.in(r_dir, N3, &drd));
    CU(S.in(p, N3, &dp)); CU(S.in(normal, N3, &dn)); CU(S.in(front_face, n, &dff)); CU(S.in(sample, N3, &dsm));
    CU(S.out(n, &dsome)); CU(S.out(N3, &datt)); CU(S.out(N3, &dso)); CU(S.out(N3, &dsd));
    if (precision == RTIOW_PRECISION_F64) scatter_kernel<double><<<grid, 256, 0, d.stream>>>(n, dk, da, dpar, dro, drd, dp, dn, dff, dsm, dsome, datt, dso, dsd);
    else scatter_kernel<float><<<grid, 256, 0, d.stream>>>(n, dk, da, dpar, dro, drd, dp, dn, dff, dsm, dsome, datt, dso, dsd);
    CU(cudaGetLastError());
    CU(S.back(some, dsome, n)); CU(S.back(attenuation, datt, N3)); CU(S.back(s_orig, dso, N3)); CU(S.back(s_dir, dsd, N3));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_get_ray_batch(rtiow_ctx* c, int precision, const rtiow_camera* cam, int64_t n, const double* s, const double* t,
                                   const double* disk_xy, double* orig, double* dir)
{
    BATCH_PROLOGUE();
    if (!cam || !s || !t || !disk_xy || !orig || !dir) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    if (n == 0) return RTIOW_OK;
    double *ds, *dt, *dk, *dor, *dd;
    CU(S.in(s, n, &ds)); CU(S.in(t, n, &dt)); CU(S.in(disk_xy, (size_t)n * 2, &dk)); CU(S.out(N3, &dor)); CU(S.out(N3, &dd));
    if (precision == RTIOW_PRECISION_F64) get_ray_kernel<double><<<grid, 256, 0, d.stream>>>(to_dev_camera<double>(*cam), n, ds, dt, dk, dor, dd);
    else get_ray_kernel<float><<<grid, 256, 0, d.stream>>>(to_dev_camera<float>(*cam), n, ds, dt, dk, dor, dd);
    CU(cudaGetLastError());
    CU(S.back(orig, dor, N3)); CU(S.back(dir, dd, N3));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_to_rgba_batch(rtiow_ctx* c, int precision, int64_t n, const double* color, uint8_t alpha, uint64_t spp, uint8_t* out_rgba)
{
    BATCH_PROLOGUE();
    if (spp == 0) return fail(RTIOW_ERR_INVALID_ARG, "spp must be >= 1");
    if (!color || !out_rgba) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    if (n == 0) return RTIOW_OK;
    double* dc; uint32_t* dout;
    CU(S.in(color, N3, &dc)); CU(S.out(n, &dout));
    if (precision == RTIOW_PRECISION_F64) to_rgba_kernel<double><<<grid, 256, 0, d.stream>>>(n, dc, alpha, spp, dout);
    else to_rgba_kernel<float><<<grid, 256, 0, d.stream>>>(n, dc, alpha, spp, dout);
    CU(cudaGetLastError());
    CU(S.back((uint32_t*)out_rgba, dout, n));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_reflect_batch(rtiow_ctx* c, int precision, int64_t n, const double* v, const double* nrm, double* out)
{
    BATCH_PROLOGUE();
    if (!v || !nrm || !out) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    if (n == 0) return RTIOW_OK;
    double *dv, *dn, *dout;
    CU(S.in(v, N3, &dv)); CU(S.in(nrm, N3, &dn)); CU(S.out(N3, &dout));
    if (precision == RTIOW_PRECISION_F64) reflect_kernel<double><<<grid, 256, 0, d.stream>>>(n, dv, dn, dout);
    else reflect_kernel<float><<<grid, 256, 0, d.stream>>>(n, dv, dn, dout);
    CU(cudaGetLastError());
    CU(S.back(out, dout, N3));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_refract_batch(rtiow_ctx* c, int precision, int64_t n, const double* uv, const double* nrm, const double* eta, double* out)
{
    BATCH_PROLOGUE();
    if (!uv || !nrm || !eta || !out) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    if (n == 0) return RTIOW_OK;
    double *dv, *dn, *de, *dout;
    CU(S.in(uv, N3, &dv)); CU(S.in(nrm, N3, &dn)); CU(S.in(eta, n, &de)); CU(S.out(N3, &dout));
    if (precision == RTIOW_PRECISION_F64) refract_kernel<double><<<grid, 256, 0, d.stream>>>(n, dv, dn, de, dout);
    else refract_kernel<float><<<grid, 256, 0, d.stream>>>(n, dv, dn, de, dout);
    CU(cudaGetLastError());
    CU(S.back(out, dout, N3));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_ray_color_batch(rtiow_ctx* c, int precision, int64_t n, const double* orig, const double* dir, const uint32_t* pixel,
                                     const uint32_t* sample, uint64_t seed, int32_t max_depth, double t_min, double* color, uint64_t* rays)
{
    return rtiow_ray_color_trace_batch(c, precision, n, orig, dir, pixel, sample, seed, max_depth, t_min, color, rays, nullptr, nullptr);
}

extern "C" int rtiow_ray_color_trace_batch(rtiow_ctx* c, int precision, int64_t n, const double* orig, const double* dir, const uint32_t* pixel,
                                           const uint32_t* sample, uint64_t seed, int32_t max_depth, double t_min, double* color, uint64_t* rays,
                                           int32_t* trace_index, double* trace_ray)
{
    BATCH_PROLOGUE();
    if (!d.has_scene) return fail(RTIOW_ERR_INVALID_ARG, "no scene uploaded");
    if (!orig || !dir || !pixel || !sample || !color) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    ScanPlan plan;
    int rc = plan_scan(c, d, precision, &plan); if (rc) return rc;
    if (n == 0) return RTIOW_OK;
    double *dor, *dd, *dcol; uint32_t *dpx, *dsm; unsigned long long* dr;
    CU(S.in(orig, N3, &dor)); CU(S.in(dir, N3, &dd)); CU(S.in(pixel, n, &dpx)); CU(S.in(sample, n, &dsm));
    CU(S.out(N3, &dcol)); CU(S.out(n, &dr));
    const size_t n_tr = (size_t)n * (size_t)std::max(max_depth, 0);
    int32_t* dti = nullptr; double* dtr = nullptr;
    if (trace_index && n_tr) { CU(S.out(n_tr, &dti)); CU(cudaMemsetAsync(dti, 0xff, n_tr * sizeof(int32_t), d.stream)); }   // -1: no ray at this depth
    if (trace_ray && n_tr) CU(S.out(n_tr * 6, &dtr));
    // one path per thread, `rays` of them in a CTA of `threads`
    auto launch = [&](auto k, int rays, int threads) -> int {
        const size_t smem = plan.smem(threads);
        int rc = allow_smem(k, smem); if (rc) return rc;
        k<<<(unsigned)((n + rays - 1) / rays), threads, smem, d.stream>>>(d.scene, n, dor, dd, dpx, dsm, seed, max_depth, t_min, dcol, dr, dti, dtr);
        return RTIOW_OK;
    };
    switch (plan.scan) {
    case Scan::F64: rc = launch(ray_color_kernel<double, false, 256>, 256, 256); break;
    case Scan::Tensor: rc = launch(ray_color_kernel_umma<RT_UMMA_GROUPS, RT_UMMA_CHUNK>, UShape::kRayThreads, UShape::kThreads); break;
    case Scan::Smem: rc = launch(ray_color_kernel<float, true, 256>, 256, 256); break;
    case Scan::Wide: rc = launch(ray_color_kernel<float, true, 512>, 512, 512); break;
    case Scan::Global: rc = launch(ray_color_kernel<float, false, 256>, 256, 256); break;
    }
    if (rc) return rc;
    CU(cudaGetLastError());
    CU(S.back(color, dcol, N3));
    if (rays) CU(S.back((unsigned long long*)rays, dr, n));
    if (dti) CU(S.back(trace_index, dti, n_tr));
    if (dtr) CU(S.back(trace_ray, dtr, n_tr * 6));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

extern "C" int rtiow_sampler_batch(rtiow_ctx* c, int precision, int64_t n, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce,
                                   uint64_t seed, double* out)
{
    BATCH_PROLOGUE();
    if (!pixel || !sample || !bounce || !out) return fail(RTIOW_ERR_INVALID_ARG, "NULL array");
    if (n == 0) return RTIOW_OK;
    uint32_t *dp, *ds, *db; double* dout;
    CU(S.in(pixel, n, &dp)); CU(S.in(sample, n, &ds)); CU(S.in(bounce, n, &db)); CU(S.out((size_t)n * 12, &dout));
    if (precision == RTIOW_PRECISION_F64) sampler_kernel<double><<<grid, 256, 0, d.stream>>>(n, dp, ds, db, seed, dout);
    else sampler_kernel<float><<<grid, 256, 0, d.stream>>>(n, dp, ds, db, seed, dout);
    CU(cudaGetLastError());
    CU(S.back(out, dout, (size_t)n * 12));
    CU(cudaStreamSynchronize(d.stream));
    return RTIOW_OK;
}

// ------------------------------------------------------------------------------------------------
// measurement helpers
// ------------------------------------------------------------------------------------------------
extern "C" int rtiow_fp32_peak_probe(rtiow_ctx* c, int packed, double target_ms, double* out_tflops, double* out_ms)
{
    if (!c || !out_tflops) return fail(RTIOW_ERR_INVALID_ARG, "NULL argument");
    DeviceState& d = c->dev[0];
    CU(cudaSetDevice(d.device));
    const int threads = 256, ctas = d.sms * 8;
    CU(d.probe.resize((size_t)threads * ctas));
    auto run = [&](int iters) -> cudaError_t {
        if (packed) probe_ffma2_kernel<<<ctas, threads, 0, d.stream>>>(d.probe.p, iters, 1.0001f, 0.5f);
        else probe_ffma_kernel<<<ctas, threads, 0, d.stream>>>(d.probe.p, iters, 1.0001f, 0.5f);
        return cudaGetLastError();
    };
    const double flop_per_iter = (packed ? 4.0 : 2.0) * 64.0 * threads * ctas;
    CU(run(256)); CU(cudaStreamSynchronize(d.stream));
    CU(cudaEventRecord(d.ev0, d.stream)); CU(run(2048)); CU(cudaEventRecord(d.ev1, d.stream)); CU(cudaStreamSynchronize(d.stream));
    float ms = 0; CU(cudaEventElapsedTime(&ms, d.ev0, d.ev1));
    double want = target_ms > 0 ? target_ms : 50.0;
    long long iters = (long long)(2048.0 * want / std::max(ms, 1e-3f));
    iters = std::max<long long>(2048, std::min<long long>(iters, 1LL << 30));
    CU(cudaEventRecord(d.ev0, d.stream)); CU(run((int)iters)); CU(cudaEventRecord(d.ev1, d.stream)); CU(cudaStreamSynchronize(d.stream));
    CU(cudaEventElapsedTime(&ms, d.ev0, d.ev1));
    *out_tflops = flop_per_iter * (double)iters / (ms * 1e-3) * 1e-12;
    if (out_ms) *out_ms = ms;
    return RTIOW_OK;
}

#ifdef RT_UMMA_TRACE
// debug builds only: the clock stamps of the last render (tools/umma_trace.py); not declared in the public header
extern "C" int rtiow_debug_umma_trace(long long* out, int cap)
{
    int n = 0;
    cudaMemcpyFromSymbol(&n, rt::g_umma_trace_n, sizeof n);
    n = std::min(n, cap);
    cudaMemcpyFromSymbol(out, rt::g_umma_trace, (size_t)n * 2 * sizeof(long long));
    int zero = 0; cudaMemcpyToSymbol(rt::g_umma_trace_n, &zero, sizeof zero);
    return n;
}
#endif

extern "C" int rtiow_flush_l2(rtiow_ctx* c)
{
    if (!c) return fail(RTIOW_ERR_INVALID_ARG, "ctx is NULL");
    for (auto& d : c->dev) {
        CU(cudaSetDevice(d.device));
        const size_t n = (size_t)256 * 1024 * 1024 / sizeof(uint4);     // 256 MiB > the 126 MB L2
        CU(d.flush.resize(n));
        flush_kernel<<<d.sms * 8, 256, 0, d.stream>>>(d.flush.p, n, 0x5a5a5a5au);
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(d.stream));
    }
    return RTIOW_OK;
}
