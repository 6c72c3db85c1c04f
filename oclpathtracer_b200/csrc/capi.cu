// capi.cu -- the C-ABI of libptb200.so (include/ptb200.h): device, buffers,
// kernel table + launcher, resident scene, and the render entry points that
// drive the sm_100a kernels.  Replaces the ADL Device/Buffer/Launcher plumbing
// (Adl/Adl.h, Adl/AdlKernel.h, Adl/CL/*) for this path.  No CPU fallback.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "host_internal.h"
#include "pt_kernels.cuh"
#include "pt_wavefront.cuh"
#include "lbvh.cuh"

namespace ptb {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU_TRY(expr)                                                                                    \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess)                                                                         \
            return ptb::fail(PTB_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

}  // namespace ptb

using namespace ptb;

// ---- objects ----------------------------------------------------------------------------------

struct ptb_device {
    int index = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    cudaDeviceProp prop{};
    int live_buffers = 0;
    // scratch, grown on demand
    void* samples = nullptr; size_t samples_bytes = 0;
    void* sum = nullptr; size_t sum_bytes = 0;
    void* wf = nullptr; size_t wf_bytes = 0;  // wavefront queues
    void* isect = nullptr; size_t isect_bytes = 0;  // ptb_scene_intersect: work counter of the persistent grid
    unsigned long long* counters = nullptr;   // CTR_COUNT + wavefront queue counters
    std::map<std::string, ptb_kernel*> kernels;  // KernelManager::m_map analogue (Adl/AdlKernel.cpp:142)
    // ptb_render_host cache
    ptb_scene* host_scene = nullptr; uint64_t host_scene_hash = 0;
    ptb_buffer* host_tris = nullptr; ptb_buffer* host_mats = nullptr;
    void* pinned = nullptr; size_t pinned_bytes = 0;  // staging of the scene records
    cudaStream_t copy_stream = nullptr;               // D2H of finished frames overlaps the next render
    cudaStream_t up_stream = nullptr;                 // H2D of the caller's records, off the render stream's critical path
    struct HostSlot {
        ptb_buffer* frame = nullptr; ptb_buffer* stats = nullptr; ptb_buffer* rgb8 = nullptr;
        void* pin = nullptr; size_t pin_bytes = 0;    // staging when the caller's buffers are pageable
        cudaEvent_t ev_render = nullptr, ev_done = nullptr, ev_up = nullptr;
        bool busy = false;
        uint64_t serial = 0;
        float* out = nullptr; ptb_pixel_stats* out_stats = nullptr;
        size_t fb = 0, sb = 0;
        bool direct_frame = false, direct_stats = false;
    } slots[2];
    uint64_t jobs_submitted = 0;
    int tune[16] = {0};  // experiment knobs (ptb_device_set_tuning)
    // helpers: other devices that render part of this device's work (ptb_device_add_helper); their peer access to this device is on
    std::vector<ptb_device*> helpers;
    ptb_device* helper_of = nullptr;
    cudaEvent_t ev_multi = nullptr;                 // cross-device ordering
    ptb_buffer* multi_frame = nullptr;              // ptb_render_multi: the ONE image (on this device)
    ptb_buffer* multi_rgb8 = nullptr;
    void* multi_pin = nullptr; size_t multi_pin_bytes = 0;
    bool cumulative_counters = false;  // ptb_device_counters: do not clear the counters per render call
    uint64_t cumulative_samples = 0;
    // measurement
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;   // triples: before integrator, after integrator, after resolve
    size_t ev_used = 0;
    int integrator_launch_batches = 0;
    uint64_t kernel_launches = 0;
};

struct ptb_buffer {
    ptb_device* dev = nullptr;
    void* d_ptr = nullptr;
    size_t bytes = 0;
    bool owned = true;
    bool ipc = false;       // mapping of another process's buffer (ptb_buffer_ipc_import)
    void* h_map = nullptr;  // pinned staging for map/unmap
    uint64_t version = 0;
};

struct ptb_kernel {
    std::string name;
    int num_triangles = 36;  // GenerateColors.cl:6
    int bounces = 16;        // GenerateColors.cl:5
    int accel = PTB_ACCEL_BVH;
    int integrator = PTB_INTEGRATOR_AUTO;
    // scene cache keyed on the bound buffers
    ptb_scene* scene = nullptr;
    const ptb_buffer* key_t = nullptr; const ptb_buffer* key_m = nullptr;
    uint64_t ver_t = 0, ver_m = 0, hash = 0;
    // frame-ahead batch of the progressive loop (ptb_launch1d): samples of frames [ahead_first, ahead_first+ahead_count)
    // already traced for (ahead_w x ahead_h, ahead_cfg); consumed one resolve per launch
    void* ahead = nullptr; size_t ahead_bytes = 0;
    int ahead_first = 0, ahead_count = 0, ahead_w = 0, ahead_h = 0;
    int ahead_cfg[3] = {0, 0, 0};
    int last_frame = -2, streak = 0;
    int frame_ahead = 1;  // ptb_kernel_set_int(k, "FRAME_AHEAD", 0) restores one integrator launch per ptb_launch1d
    std::vector<ptb_scene*> helper_scenes;  // the same scene resident on the device's helpers (frame-ahead batches are dealt over them)
};

struct ptb_scene {
    ptb_device* dev = nullptr;
    std::shared_ptr<BuiltBvh> bvhp = std::make_shared<BuiltBvh>();  // shared by the per-device copies of one scene (ptb_render_multi)
    BuiltBvh& built() { return *bvhp; }
    const BuiltBvh& built() const { return *bvhp; }
    int n_tris = 0, n_mats = 0;
    float4* d_nodes = nullptr;
    uint4* d_nodesq = nullptr;            // binary scenes: the 32-byte quantised encoding of d_nodes that the kernels traverse (ptb_bvh_nodeq)
    float q_lo[3] = {0, 0, 0}, q_step[3] = {1, 1, 1};  // its grid
    float4* d_nodes4 = nullptr;           // FLAT scenes also keep their 4-wide tree resident: coherent-ray modes use it (mode_class)
    float4* d_tris = nullptr;
    float4* d_tris_orig = nullptr;
    float4* d_mats = nullptr;
    bool small = false;                   // triangles and materials are staged in shared memory (FLAT and 4-wide scenes)
    int cls = ptd::PTD_LARGE;             // scene class: PTD_LARGE | PTD_SMALL4 | PTD_FLAT
    int width = 2;                        // 1: ptb_bvh_leafbox records (FLAT), 4: ptb_bvh_node4 records (small scenes), 2: ptb_bvh_node
    int n_nodes = 0, depth = 0, bfs_nodes = 0;
    int* d_order = nullptr;               // GPU-built scenes: BVH position -> caller index (device)
    bool host_copy_valid = true;          // false until a GPU-built tree has been downloaded
    std::vector<ptb_triangle> host_tris;  // host-built scenes: the default light lookup and copies of the scene on helper devices
    std::vector<ptb_material> host_mats;
    std::vector<ptd::SceneLight> lights;  // device-built scenes: the light of each quad id in [0, n_mats) (setup_light)
};

static int set_device(ptb_device* dev) {
    CU_TRY(cudaSetDevice(dev->index));
    return PTB_OK;
}

static int ensure(void** p, size_t* cur, size_t want) {
    if (*cur >= want) return PTB_OK;
    if (*p) CU_TRY(cudaFree(*p));
    *p = nullptr; *cur = 0;
    CU_TRY(cudaMalloc(p, want));
    *cur = want;
    return PTB_OK;
}

// ---- misc ---------------------------------------------------------------------------------------

extern "C" const char* ptb_last_error(void) { return g_err; }
extern "C" int ptb_version(void) { return 100; }

extern "C" int ptb_device_count(int* count) {
    if (!count) return fail(PTB_E_INVALID, "ptb_device_count: null");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return fail(PTB_E_NODEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *count = n;
    return PTB_OK;
}

static int device_create(int device_index, void* stream, bool own, ptb_device** out) {
    if (!out) return fail(PTB_E_INVALID, "ptb_device_create: null out");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(PTB_E_NODEVICE, "ptb_device_create: no CUDA device (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "count = 0");
    if (device_index < 0) device_index = 0;
    if (device_index > n - 1) device_index = n - 1;  // Adl/CL/AdlCL.cpp:154 clamps the same way
    ptb_device* d = new ptb_device();
    d->index = device_index;
    d->own_stream = own;
    if (cudaSetDevice(device_index) != cudaSuccess || cudaGetDeviceProperties(&d->prop, device_index) != cudaSuccess) {
        delete d;
        return fail(PTB_E_CUDA, "ptb_device_create: cannot select device %d", device_index);
    }
    if (d->prop.major < 10) {
        int code = fail(PTB_E_NODEVICE, "ptb_device_create: device %d is sm_%d%d; kernels are built for sm_100a only",
                        device_index, d->prop.major, d->prop.minor);
        delete d;
        return code;
    }
    if (own) {
        if (cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete d;
            return fail(PTB_E_CUDA, "ptb_device_create: cudaStreamCreate failed");
        }
    } else {
        d->stream = static_cast<cudaStream_t>(stream);
    }
    if (cudaMalloc(&d->counters, sizeof(unsigned long long) * 64) != cudaSuccess) {
        delete d;
        return fail(PTB_E_CUDA, "ptb_device_create: cudaMalloc failed");
    }
    cudaMemsetAsync(d->counters, 0, sizeof(unsigned long long) * 64, d->stream);
    *out = d;
    return PTB_OK;
}

extern "C" int ptb_device_create(int device_index, ptb_device** out) { return device_create(device_index, nullptr, true, out); }
extern "C" int ptb_device_create_on_stream(int device_index, void* cuda_stream, ptb_device** out) {
    return device_create(device_index, cuda_stream, false, out);
}

extern "C" int ptb_device_sync(ptb_device* dev) {
    if (!dev) return fail(PTB_E_INVALID, "ptb_device_sync: null device");
    if (set_device(dev)) return PTB_E_CUDA;
    CU_TRY(cudaStreamSynchronize(dev->stream));
    return PTB_OK;
}

extern "C" int ptb_device_destroy(ptb_device* dev) {
    if (!dev) return PTB_OK;
    set_device(dev);
    cudaStreamSynchronize(dev->stream);
    if (dev->copy_stream) cudaStreamSynchronize(dev->copy_stream);
    if (dev->up_stream) cudaStreamSynchronize(dev->up_stream);
    if (dev->host_scene) ptb_scene_destroy(dev->host_scene);
    for (ptb_device* h : dev->helpers) if (h) h->helper_of = nullptr;
    if (dev->helper_of) {  // scenes that the main device's kernels keep resident here die with this device
        auto& v = dev->helper_of->helpers;
        for (size_t i = 0; i < v.size(); ++i) {
            if (v[i] != dev) continue;
            for (auto& kv : dev->helper_of->kernels)
                if (kv.second->helper_scenes.size() > i && kv.second->helper_scenes[i]) {
                    ptb_scene_destroy(kv.second->helper_scenes[i]);
                    kv.second->helper_scenes[i] = nullptr;
                }
            v[i] = nullptr;
        }
        set_device(dev);
    }
    if (dev->multi_frame) ptb_buffer_destroy(dev->multi_frame);
    if (dev->multi_rgb8) ptb_buffer_destroy(dev->multi_rgb8);
    if (dev->multi_pin) cudaFreeHost(dev->multi_pin);
    if (dev->ev_multi) cudaEventDestroy(dev->ev_multi);
    for (auto& sl : dev->slots) {
        if (sl.frame) ptb_buffer_destroy(sl.frame);
        if (sl.stats) ptb_buffer_destroy(sl.stats);
        if (sl.rgb8) ptb_buffer_destroy(sl.rgb8);
        if (sl.pin) cudaFreeHost(sl.pin);
        if (sl.ev_render) cudaEventDestroy(sl.ev_render);
        if (sl.ev_done) cudaEventDestroy(sl.ev_done);
        if (sl.ev_up) cudaEventDestroy(sl.ev_up);
    }
    if (dev->copy_stream) cudaStreamDestroy(dev->copy_stream);
    if (dev->up_stream) cudaStreamDestroy(dev->up_stream);
    for (ptb_buffer* b : {dev->host_tris, dev->host_mats})
        if (b) ptb_buffer_destroy(b);
    for (auto& kv : dev->kernels) {
        if (kv.second->scene) ptb_scene_destroy(kv.second->scene);
        for (ptb_scene* hs : kv.second->helper_scenes) if (hs) ptb_scene_destroy(hs);
        if (kv.second->ahead) { set_device(dev); cudaFree(kv.second->ahead); }
        delete kv.second;
    }
    if (dev->samples) cudaFree(dev->samples);
    if (dev->sum) cudaFree(dev->sum);
    if (dev->wf) cudaFree(dev->wf);
    if (dev->isect) cudaFree(dev->isect);
    if (dev->counters) cudaFree(dev->counters);
    if (dev->pinned) cudaFreeHost(dev->pinned);
    for (cudaEvent_t e : dev->ev_pool) cudaEventDestroy(e);
    if (dev->own_stream && dev->stream) cudaStreamDestroy(dev->stream);
    int leaked = dev->live_buffers;
    delete dev;
    // DeviceUtils::deallocate asserts (debug only) that all buffers were freed, Adl/Adl.cpp:204
    if (leaked) return fail(PTB_E_INVALID, "ptb_device_destroy: %d buffer(s) still alive", leaked);
    return PTB_OK;
}

extern "C" int ptb_device_name(ptb_device* dev, char out[128]) {
    if (!dev || !out) return fail(PTB_E_INVALID, "ptb_device_name: null argument");
    snprintf(out, 128, "%s sm_%d%d CUDA", dev->prop.name, dev->prop.major, dev->prop.minor);
    return PTB_OK;
}
extern "C" int ptb_device_sm_count(ptb_device* dev, int* sm) {
    if (!dev || !sm) return fail(PTB_E_INVALID, "ptb_device_sm_count: null argument");
    *sm = dev->prop.multiProcessorCount;
    return PTB_OK;
}
extern "C" int ptb_device_memory(ptb_device* dev, size_t* free_bytes, size_t* total_bytes) {
    if (!dev) return fail(PTB_E_INVALID, "ptb_device_memory: null device");
    if (set_device(dev)) return PTB_E_CUDA;
    size_t f = 0, t = 0;
    CU_TRY(cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    return PTB_OK;
}
extern "C" void* ptb_device_stream(ptb_device* dev) { return dev ? (void*)dev->stream : nullptr; }

// ---- buffers --------------------------------------------------------------------------------------

extern "C" int ptb_buffer_create(ptb_device* dev, size_t bytes, ptb_buffer** out) {
    if (!dev || !out) return fail(PTB_E_INVALID, "ptb_buffer_create: null argument");
    *out = nullptr;
    if (set_device(dev)) return PTB_E_CUDA;
    ptb_buffer* b = new ptb_buffer();
    b->dev = dev;
    b->bytes = bytes;
    cudaError_t e = cudaMalloc(&b->d_ptr, bytes ? bytes : 1);
    if (e != cudaSuccess) {  // ADL: m_ptr = 0, m_size = 0 + log (Adl/CL/AdlCL.inl:190-197)
        delete b;
        return fail(PTB_E_NOMEM, "ptb_buffer_create: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    dev->live_buffers++;
    *out = b;
    return PTB_OK;
}

extern "C" int ptb_buffer_wrap(ptb_device* dev, void* device_ptr, size_t bytes, ptb_buffer** out) {
    if (!dev || !out || !device_ptr) return fail(PTB_E_INVALID, "ptb_buffer_wrap: null argument");
    ptb_buffer* b = new ptb_buffer();
    b->dev = dev; b->d_ptr = device_ptr; b->bytes = bytes; b->owned = false;
    dev->live_buffers++;
    *out = b;
    return PTB_OK;
}

extern "C" int ptb_buffer_destroy(ptb_buffer* buf) {
    if (!buf) return PTB_OK;
    set_device(buf->dev);
    if (buf->h_map) cudaFreeHost(buf->h_map);
    if (buf->owned && buf->d_ptr) {
        cudaStreamSynchronize(buf->dev->stream);
        cudaFree(buf->d_ptr);
    }
    if (buf->ipc && buf->d_ptr) {
        cudaStreamSynchronize(buf->dev->stream);
        cudaIpcCloseMemHandle(buf->d_ptr);
    }
    buf->dev->live_buffers--;
    delete buf;
    return PTB_OK;
}

extern "C" int ptb_buffer_write(ptb_buffer* buf, const void* host_src, size_t bytes, size_t dst_offset) {
    if (!buf || !host_src) return fail(PTB_E_INVALID, "ptb_buffer_write: null argument");
    if (bytes > buf->bytes || dst_offset > buf->bytes - bytes) return fail(PTB_E_INVALID, "ptb_buffer_write: range exceeds buffer");
    if (set_device(buf->dev)) return PTB_E_CUDA;
    CU_TRY(cudaMemcpyAsync((char*)buf->d_ptr + dst_offset, host_src, bytes, cudaMemcpyHostToDevice, buf->dev->stream));
    buf->version++;
    return PTB_OK;
}

extern "C" int ptb_buffer_read(ptb_buffer* buf, void* host_dst, size_t bytes, size_t src_offset) {
    if (!buf || !host_dst) return fail(PTB_E_INVALID, "ptb_buffer_read: null argument");
    if (bytes > buf->bytes || src_offset > buf->bytes - bytes) return fail(PTB_E_INVALID, "ptb_buffer_read: range exceeds buffer");
    if (set_device(buf->dev)) return PTB_E_CUDA;
    CU_TRY(cudaMemcpyAsync(host_dst, (const char*)buf->d_ptr + src_offset, bytes, cudaMemcpyDeviceToHost, buf->dev->stream));
    return PTB_OK;
}

extern "C" int ptb_buffer_map(ptb_buffer* buf, void** host_ptr) {
    if (!buf || !host_ptr) return fail(PTB_E_INVALID, "ptb_buffer_map: null argument");
    if (set_device(buf->dev)) return PTB_E_CUDA;
    if (!buf->h_map) CU_TRY(cudaMallocHost(&buf->h_map, buf->bytes ? buf->bytes : 1));
    // clEnqueueMapBuffer(non-blocking, READ|WRITE): contents valid after the caller waits
    CU_TRY(cudaMemcpyAsync(buf->h_map, buf->d_ptr, buf->bytes, cudaMemcpyDeviceToHost, buf->dev->stream));
    *host_ptr = buf->h_map;
    return PTB_OK;
}

extern "C" int ptb_buffer_unmap(ptb_buffer* buf, void* host_ptr) {
    if (!buf || !host_ptr || host_ptr != buf->h_map) return fail(PTB_E_INVALID, "ptb_buffer_unmap: pointer was not mapped");
    if (set_device(buf->dev)) return PTB_E_CUDA;
    CU_TRY(cudaMemcpyAsync(buf->d_ptr, buf->h_map, buf->bytes, cudaMemcpyHostToDevice, buf->dev->stream));
    buf->version++;
    return PTB_OK;
}

extern "C" int ptb_buffer_clear(ptb_buffer* buf) {
    if (!buf) return fail(PTB_E_INVALID, "ptb_buffer_clear: null");
    if (set_device(buf->dev)) return PTB_E_CUDA;
    CU_TRY(cudaMemsetAsync(buf->d_ptr, 0, buf->bytes, buf->dev->stream));
    buf->version++;
    return PTB_OK;
}

extern "C" void* ptb_buffer_device_ptr(ptb_buffer* buf) { return buf ? buf->d_ptr : nullptr; }
extern "C" int ptb_buffer_mark_dirty(ptb_buffer* buf) {
    if (!buf) return fail(PTB_E_INVALID, "ptb_buffer_mark_dirty: null");
    buf->version++;
    return PTB_OK;
}
extern "C" size_t ptb_buffer_size(ptb_buffer* buf) { return buf ? buf->bytes : 0; }

// ---- resident scene ---------------------------------------------------------------------------------

extern "C" int ptb_scene_destroy(ptb_scene* s) {
    if (!s) return PTB_OK;
    set_device(s->dev);
    cudaStreamSynchronize(s->dev->stream);
    for (void* p : {(void*)s->d_nodes, (void*)s->d_nodesq, (void*)s->d_nodes4, (void*)s->d_tris, (void*)s->d_tris_orig, (void*)s->d_mats, (void*)s->d_order})
        if (p) cudaFree(p);
    delete s;
    return PTB_OK;
}

// Binary trees are traversed through their quantised encoding: derive it on the device from the fp32 nodes (lbvh.cuh:
// k_quant_grid / k_quant_nodes) and fetch the six grid numbers the kernels take as parameters.
static int quantize_scene(ptb_scene* s) {
    ptb_device* dev = s->dev;
    float* d_grid = nullptr;
    CU_TRY(cudaMalloc((void**)&s->d_nodesq, size_t(s->n_nodes) * 32));
    CU_TRY(cudaMalloc((void**)&d_grid, 6 * sizeof(float)));
    ptd::k_quant_grid<<<1, 32, 0, dev->stream>>>(s->d_nodes, d_grid);
    ptd::k_quant_nodes<<<(unsigned)((s->n_nodes + 255) / 256), 256, 0, dev->stream>>>(s->d_nodes, s->n_nodes, d_grid, s->d_nodesq);
    float grid[6];
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(grid, d_grid, sizeof grid, cudaMemcpyDeviceToHost, dev->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(dev->stream);
    cudaFree(d_grid);
    if (e != cudaSuccess) return fail(PTB_E_CUDA, "ptb_scene_create: node quantisation failed: %s", cudaGetErrorString(e));
    for (int a = 0; a < 3; ++a) { s->q_lo[a] = grid[a]; s->q_step[a] = grid[3 + a]; }
    dev->kernel_launches += 2;
    return PTB_OK;
}

// `share`: a scene of the SAME records on another device whose host-built tree is reused (one build, one upload per device)
static int scene_create_impl(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                             const ptb_bvh_params* bvh_params, const ptb_scene* share, ptb_scene** out) {
    if (!dev || !tris || !mats || !out || n_tris < 1 || n_mats < 1)
        return fail(PTB_E_INVALID, "ptb_scene_create: bad arguments");
    *out = nullptr;
    for (int i = 0; i < n_tris; ++i)
        if (tris[i].id < 0 || tris[i].id >= n_mats)
            return fail(PTB_E_INVALID, "ptb_scene_create: triangle %d has id %d outside [0,%d)", i, tris[i].id, n_mats);
    ptb_bvh_params bp;
    if (bvh_params) bp = *bvh_params; else ptb_bvh_params_default(&bp);
    ptb_scene* s = new ptb_scene();
    s->dev = dev; s->n_tris = n_tris; s->n_mats = n_mats;
    int rc = PTB_OK;
    if (share && share->host_copy_valid) s->bvhp = share->bvhp;
    else rc = build_bvh(tris, n_tris, bp, &s->built());
    if (rc) { delete s; return rc; }
    s->host_tris.assign(tris, tris + n_tris);
    s->host_mats.assign(mats, mats + n_mats);
    std::vector<ptb_bvh_tri> orig;
    make_edge_tris(tris, n_tris, &orig);
    std::vector<float4> m(size_t(n_mats) * 2);
    for (int i = 0; i < n_mats; ++i) {
        m[2 * i] = make_float4(mats[i].albedo.x, mats[i].albedo.y, mats[i].albedo.z, mats[i].roughness);
        float tbits;
        std::memcpy(&tbits, &mats[i].type, 4);
        m[2 * i + 1] = make_float4(mats[i].emissive.x, mats[i].emissive.y, mats[i].emissive.z, tbits);
    }
    // scene class: everything (4-wide nodes, triangles, materials) fits a 32 KB shared-memory budget -> SMALL
    const size_t staged4 = s->built().nodes4.size() * sizeof(ptb_bvh_node4) + size_t(n_tris) * 48 + size_t(n_mats) * 32;
    const bool can4 = !s->built().nodes4.empty() && staged4 <= 32 * 1024 && int(s->built().nodes4.size()) == s->built().smem_nodes4;
    const bool can_flat = !s->built().flat.empty();  // <= 32 leaves and <= 64 triangles: no tree, leaf boxes as kernel parameters
    if ((bp.force_width == 1 && !can_flat) || (bp.force_width == 4 && !can4) || (bp.force_width != 0 && bp.force_width != 1 && bp.force_width != 2 && bp.force_width != 4)) {
        delete s;
        return fail(PTB_E_INVALID, "ptb_scene_create: the scene does not qualify for force_width = %d", bp.force_width);
    }
    s->cls = bp.force_width == 1 ? ptd::PTD_FLAT : bp.force_width == 4 ? ptd::PTD_SMALL4 : bp.force_width == 2 ? ptd::PTD_LARGE
             : can_flat ? ptd::PTD_FLAT : can4 ? ptd::PTD_SMALL4 : ptd::PTD_LARGE;
    s->small = s->cls != ptd::PTD_LARGE;
    if (s->cls == ptd::PTD_FLAT) { s->width = 1; s->n_nodes = int(s->built().flat.size()); s->depth = 1; s->bfs_nodes = s->n_nodes; }
    else if (s->cls == ptd::PTD_SMALL4) { s->width = 4; s->n_nodes = int(s->built().nodes4.size()); s->depth = s->built().depth4; s->bfs_nodes = s->built().smem_nodes4; }
    else { s->width = 2; s->n_nodes = int(s->built().nodes.size()); s->depth = s->built().depth; s->bfs_nodes = s->built().smem_nodes; }
    if (set_device(dev)) { delete s; return PTB_E_CUDA; }
    auto up = [&](float4** d, const void* h, size_t bytes) -> int {
        CU_TRY(cudaMalloc((void**)d, bytes));
        CU_TRY(cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, dev->stream));
        return PTB_OK;
    };
    std::vector<ptb_bvh_leafbox> flat_padded = s->built().flat;  // staged count is even: pad with a box that never hits
    if (flat_padded.size() & 1) flat_padded.push_back(ptb_bvh_leafbox{{0.f, 0.f, 0.f}, 0u, {-1e30f, -1e30f, -1e30f}, 0u});
    if ((rc = s->cls == ptd::PTD_FLAT     ? up(&s->d_nodes, flat_padded.data(), flat_padded.size() * sizeof(ptb_bvh_leafbox))
              : s->cls == ptd::PTD_SMALL4 ? up(&s->d_nodes, s->built().nodes4.data(), s->built().nodes4.size() * sizeof(ptb_bvh_node4))
                                          : up(&s->d_nodes, s->built().nodes.data(), s->built().nodes.size() * sizeof(ptb_bvh_node))) ||
        (s->cls == ptd::PTD_FLAT && can4 && bp.force_width == 0 && (rc = up(&s->d_nodes4, s->built().nodes4.data(), s->built().nodes4.size() * sizeof(ptb_bvh_node4)))) ||
        (rc = up(&s->d_tris, s->built().tris.data(), s->built().tris.size() * 48)) ||
        (rc = up(&s->d_tris_orig, orig.data(), orig.size() * 48)) || (rc = up(&s->d_mats, m.data(), m.size() * 16))) {
        ptb_scene_destroy(s);
        return rc;
    }
    // the host vectors `orig` and `m` die at return: finish the copies now
    if (cudaError_t e = cudaStreamSynchronize(dev->stream); e != cudaSuccess) {
        ptb_scene_destroy(s);
        return fail(PTB_E_CUDA, "ptb_scene_create: upload failed: %s", cudaGetErrorString(e));
    }
    if (s->cls == ptd::PTD_LARGE)
        if ((rc = quantize_scene(s))) { ptb_scene_destroy(s); return rc; }
    *out = s;
    return PTB_OK;
}

extern "C" int ptb_scene_create(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats,
                                int n_mats, const ptb_bvh_params* bvh_params, ptb_scene** out) {
    return scene_create_impl(dev, tris, n_tris, mats, n_mats, bvh_params, nullptr, out);
}

static int check_pad_rel(const char* what, const ptb_bvh_params& bp) {
    if (!(bp.pad_rel > 0.0f) || std::isinf(bp.pad_rel))
        return fail(PTB_E_INVALID, "%s: pad_rel must be a finite number > 0, got %g (without a pad, rounding in "
                    "the box and triangle tests loses hits)", what, double(bp.pad_rel));
    return PTB_OK;
}

// The device half of both LBVH constructors (lbvh.cuh).  From n_tris caller-order triangle and n_mats material records on the
// device (read on dev->stream and not kept): the validation verdicts, the caller-order edge triangles, the packed materials,
// the light table, the tree and its quantised encoding.  The verdicts and the light table come back in the synchronisation
// that fetches the tree depth; records that fail validation leave no scene.  Only the root is guaranteed to sit at index 0, so
// one node is staged in shared memory; everything else is traversed from L2/HBM.
static int scene_create_lbvh(ptb_device* dev, const char* what, const ptb_triangle* d_tris, int n_tris, const ptb_material* d_mats,
                             int n_mats, const ptb_bvh_params& bp, ptb_scene** out) {
    ptb_scene* s = new ptb_scene();
    s->dev = dev; s->n_tris = n_tris; s->n_mats = n_mats;
    s->host_copy_valid = false;
    s->n_nodes = n_tris - 1; s->bfs_nodes = 1; s->small = false; s->width = 2;
    const size_t light_bytes = sizeof(ptd::SceneLight) * size_t(n_mats);
    std::vector<unsigned char> check(16 + light_bytes);  // the two verdicts (k_scene_tris), then the light table
    unsigned long long* d_check = nullptr;
    auto fail_out = [&](int code) { if (d_check) cudaFree(d_check); ptb_scene_destroy(s); return code; };
    if (cudaMalloc((void**)&s->d_tris_orig, size_t(n_tris) * 48) != cudaSuccess || cudaMalloc((void**)&s->d_mats, size_t(n_mats) * 32) != cudaSuccess ||
        cudaMalloc((void**)&d_check, check.size()) != cudaSuccess)
        return fail_out(fail(PTB_E_NOMEM, "%s: cudaMalloc failed", what));
    ptd::SceneLight* d_lights = reinterpret_cast<ptd::SceneLight*>(d_check + 2);
    const unsigned grid_t = unsigned((n_tris + 255) / 256), grid_m = unsigned((n_mats + 255) / 256);
    if (cudaMemsetAsync(d_check, 0xff, 16, dev->stream) != cudaSuccess || cudaMemsetAsync(d_lights, 0x7f, light_bytes, dev->stream) != cudaSuccess)
        return fail_out(fail(PTB_E_CUDA, "%s: cudaMemsetAsync failed", what));
    ptd::k_scene_tris<<<grid_t, 256, 0, dev->stream>>>(d_tris, n_tris, n_mats, d_check, s->d_tris_orig, d_lights);
    ptd::k_scene_mats<<<grid_m, 256, 0, dev->stream>>>(d_mats, n_mats, s->d_mats);
    ptd::k_scene_lights<<<grid_m, 256, 0, dev->stream>>>(d_tris, n_tris, n_mats, d_lights);
    if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) return fail_out(fail(PTB_E_CUDA, "%s: launch failed: %s", what, cudaGetErrorString(e)));
    if (int rc = ptd::build_lbvh_device(dev->stream, d_tris, n_tris, bp.max_leaf, bp.pad_rel, &s->d_nodes, &s->d_tris, &s->d_order, &s->depth,
                                        d_check, check.data(), check.size()))
        return fail_out(rc);
    unsigned long long bad[2];
    std::memcpy(bad, check.data(), sizeof bad);
    if (bad[0] != ~0ull || bad[1] != ~0ull) {  // the lowest offending index; on a tie the id is reported, as the host loop does
        const unsigned long long first_id = bad[0] >> 32;
        if (first_id <= bad[1])
            return fail_out(fail(PTB_E_INVALID, "%s: triangle %d has id %d outside [0,%d)", what, int(first_id), int(uint32_t(bad[0])), n_mats));
        return fail_out(fail(PTB_E_INVALID, "%s: triangle %d has a non-finite vertex", what, int(bad[1])));
    }
    s->lights.resize(size_t(n_mats));
    std::memcpy(s->lights.data(), check.data() + 16, light_bytes);
    cudaFree(d_check); d_check = nullptr;
    if (int rc = quantize_scene(s)) return fail_out(rc);
    *out = s;
    return PTB_OK;
}

// Scene whose BVH is built on the device from host records: checked here, uploaded, then built as ptb_scene_create_from_device
// builds it.
extern "C" int ptb_scene_create_gpu(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats,
                                    int n_mats, const ptb_bvh_params* bvh_params, ptb_scene** out) {
    if (!dev || !tris || !mats || !out || n_tris < 2 || n_mats < 1)
        return fail(PTB_E_INVALID, "ptb_scene_create_gpu: bad arguments (needs >= 2 triangles)");
    *out = nullptr;
    if (n_tris >= (1 << 28))  // a leaf reference holds first << 3 in 32 bits
        return fail(PTB_E_INVALID, "ptb_scene_create_gpu: %d triangles; the leaf encoding holds fewer than 2^28", n_tris);
    for (int i = 0; i < n_tris; ++i) {
        if (tris[i].id < 0 || tris[i].id >= n_mats)
            return fail(PTB_E_INVALID, "ptb_scene_create_gpu: triangle %d has id %d outside [0,%d)", i, tris[i].id, n_mats);
        const float* v = &tris[i].p1.x;
        for (int k = 0; k < 12; ++k)
            if (!(std::fabs(v[k]) <= 3.0e38f)) return fail(PTB_E_INVALID, "ptb_scene_create_gpu: triangle %d has a non-finite vertex", i);
    }
    ptb_bvh_params bp;
    if (bvh_params) bp = *bvh_params; else ptb_bvh_params_default(&bp);
    if (int rc = check_pad_rel("ptb_scene_create_gpu", bp)) return rc;
    if (set_device(dev)) return PTB_E_CUDA;
    ptb_triangle* d_raw = nullptr;  // the triangle records, then the material records
    if (cudaMalloc((void**)&d_raw, (size_t(n_tris) + size_t(n_mats)) * 64) != cudaSuccess)
        return fail(PTB_E_NOMEM, "ptb_scene_create_gpu: cudaMalloc failed");
    ptb_material* d_rawm = reinterpret_cast<ptb_material*>(d_raw + n_tris);
    int rc = PTB_OK;
    if (cudaMemcpyAsync(d_raw, tris, size_t(n_tris) * 64, cudaMemcpyHostToDevice, dev->stream) != cudaSuccess ||
        cudaMemcpyAsync(d_rawm, mats, size_t(n_mats) * 64, cudaMemcpyHostToDevice, dev->stream) != cudaSuccess) {
        cudaStreamSynchronize(dev->stream);
        rc = fail(PTB_E_CUDA, "ptb_scene_create_gpu: upload failed");
    } else {
        rc = scene_create_lbvh(dev, "ptb_scene_create_gpu", d_raw, n_tris, d_rawm, n_mats, bp, out);
    }
    cudaFree(d_raw);
    return rc;
}

extern "C" int ptb_scene_create_from_device(ptb_device* dev, ptb_buffer* tris, int n_tris, ptb_buffer* mats, int n_mats,
                                            const ptb_bvh_params* bvh_params, ptb_scene** out) {
    if (!dev || !tris || !mats || !out) return fail(PTB_E_INVALID, "ptb_scene_create_from_device: null device, tris, mats or out");
    *out = nullptr;
    if (n_tris < 2 || n_mats < 1)
        return fail(PTB_E_INVALID, "ptb_scene_create_from_device: needs >= 2 triangles and >= 1 material, got %d and %d", n_tris, n_mats);
    if (n_tris >= (1 << 28))  // before the sizes: nothing is read
        return fail(PTB_E_INVALID, "ptb_scene_create_from_device: %d triangles; the leaf encoding holds fewer than 2^28", n_tris);
    if (tris->dev != dev || mats->dev != dev) return fail(PTB_E_INVALID, "ptb_scene_create_from_device: buffer belongs to another device");
    if (tris->bytes < size_t(n_tris) * 64)
        return fail(PTB_E_INVALID, "ptb_scene_create_from_device: tris buffer too small (%zu < %zu)", tris->bytes, size_t(n_tris) * 64);
    if (mats->bytes < size_t(n_mats) * 64)
        return fail(PTB_E_INVALID, "ptb_scene_create_from_device: mats buffer too small (%zu < %zu)", mats->bytes, size_t(n_mats) * 64);
    if (((reinterpret_cast<uintptr_t>(tris->d_ptr) | reinterpret_cast<uintptr_t>(mats->d_ptr)) & 15u) != 0)
        return fail(PTB_E_INVALID, "ptb_scene_create_from_device: tris and mats must be 16-byte aligned (float4 loads)");
    ptb_bvh_params bp;
    if (bvh_params) bp = *bvh_params; else ptb_bvh_params_default(&bp);
    if (int rc = check_pad_rel("ptb_scene_create_from_device", bp)) return rc;
    if (bp.force_width != 0 && bp.force_width != 2)
        return fail(PTB_E_INVALID, "ptb_scene_create_from_device: force_width = %d; only the binary form (0 or 2) is built on the device",
                    bp.force_width);
    if (set_device(dev)) return PTB_E_CUDA;
    return scene_create_lbvh(dev, "ptb_scene_create_from_device", static_cast<const ptb_triangle*>(tris->d_ptr), n_tris,
                             static_cast<const ptb_material*>(mats->d_ptr), n_mats, bp, out);
}

extern "C" int ptb_bvh_build_host(const ptb_triangle* tris, int n_tris, const ptb_bvh_params* bvh_params, int width,
                                  void** nodes, int* n_nodes, int32_t** tri_order, ptb_bvh_tri** ordered_tris,
                                  int* depth, int* smem_nodes) {
    if (!tris || !nodes || !n_nodes || !tri_order) return fail(PTB_E_INVALID, "ptb_bvh_build_host: null argument");
    if (width != 2 && width != 4 && width != 1) return fail(PTB_E_INVALID, "ptb_bvh_build_host: width must be 1, 2 or 4");
    ptb_bvh_params bp;
    if (bvh_params) bp = *bvh_params; else ptb_bvh_params_default(&bp);
    BuiltBvh b;
    if (int rc = build_bvh(tris, n_tris, bp, &b)) return rc;
    if (width == 4 && b.nodes4.empty()) return fail(PTB_E_INVALID, "ptb_bvh_build_host: 4-wide trees are built for <= 2048 triangles");
    if (width == 1 && b.flat.empty()) return fail(PTB_E_INVALID, "ptb_bvh_build_host: the FLAT form needs <= 32 leaves and <= 64 triangles");
    const size_t node_bytes = width == 1 ? b.flat.size() * sizeof(ptb_bvh_leafbox)
                              : width == 4 ? b.nodes4.size() * sizeof(ptb_bvh_node4) : b.nodes.size() * sizeof(ptb_bvh_node);
    *nodes = std::malloc(node_bytes);
    *tri_order = static_cast<int32_t*>(std::malloc(b.tri_order.size() * sizeof(int32_t)));
    if (ordered_tris) *ordered_tris = nullptr;
    auto oom = [&]() {
        std::free(*nodes); std::free(*tri_order);
        *nodes = nullptr; *tri_order = nullptr;
        return fail(PTB_E_NOMEM, "ptb_bvh_build_host: out of memory");
    };
    if (!*nodes || !*tri_order) return oom();
    std::memcpy(*nodes, width == 1 ? (const void*)b.flat.data() : width == 4 ? (const void*)b.nodes4.data() : (const void*)b.nodes.data(), node_bytes);
    std::memcpy(*tri_order, b.tri_order.data(), b.tri_order.size() * sizeof(int32_t));
    if (ordered_tris) {
        *ordered_tris = static_cast<ptb_bvh_tri*>(std::malloc(b.tris.size() * sizeof(ptb_bvh_tri)));
        if (!*ordered_tris) return oom();
        std::memcpy(*ordered_tris, b.tris.data(), b.tris.size() * sizeof(ptb_bvh_tri));
    }
    *n_nodes = int(width == 1 ? b.flat.size() : width == 4 ? b.nodes4.size() : b.nodes.size());
    if (depth) *depth = width == 1 ? 1 : width == 4 ? b.depth4 : b.depth;
    if (smem_nodes) *smem_nodes = width == 1 ? int(b.flat.size()) : width == 4 ? b.smem_nodes4 : b.smem_nodes;
    return PTB_OK;
}

extern "C" int ptb_scene_info(ptb_scene* s, int* n_nodes, int* n_tris, int* depth, int* smem_nodes) {
    if (!s) return fail(PTB_E_INVALID, "ptb_scene_info: null scene");
    if (n_nodes) *n_nodes = s->n_nodes;
    if (n_tris) *n_tris = s->n_tris;
    if (depth) *depth = s->depth;
    if (smem_nodes) *smem_nodes = s->bfs_nodes;
    return PTB_OK;
}

extern "C" int ptb_scene_bvh_width(ptb_scene* s) { return s ? s->width : 0; }

extern "C" int ptb_scene_copy_bvh_quantized(ptb_scene* s, uint32_t* qnodes, float grid_lo[3], float grid_step[3]) {
    if (!s) return fail(PTB_E_INVALID, "ptb_scene_copy_bvh_quantized: null scene");
    if (!s->d_nodesq) return fail(PTB_E_INVALID, "ptb_scene_copy_bvh_quantized: the scene has no binary tree (width %d)", s->width);
    if (set_device(s->dev)) return PTB_E_CUDA;
    if (qnodes) {
        CU_TRY(cudaMemcpyAsync(qnodes, s->d_nodesq, size_t(s->n_nodes) * 32, cudaMemcpyDeviceToHost, s->dev->stream));
        CU_TRY(cudaStreamSynchronize(s->dev->stream));
    }
    for (int a = 0; a < 3; ++a) {
        if (grid_lo) grid_lo[a] = s->q_lo[a];
        if (grid_step) grid_step[a] = s->q_step[a];
    }
    return PTB_OK;
}

extern "C" int ptb_scene_copy_bvh(ptb_scene* s, void* nodes, int32_t* tri_order) {
    if (!s) return fail(PTB_E_INVALID, "ptb_scene_copy_bvh: null scene");
    if (!s->host_copy_valid) {  // GPU-built tree: download on first request
        if (set_device(s->dev)) return PTB_E_CUDA;
        s->built().nodes.resize(size_t(s->n_nodes));
        s->built().tri_order.resize(size_t(s->n_tris));
        CU_TRY(cudaMemcpyAsync(s->built().nodes.data(), s->d_nodes, size_t(s->n_nodes) * sizeof(ptb_bvh_node), cudaMemcpyDeviceToHost, s->dev->stream));
        CU_TRY(cudaMemcpyAsync(s->built().tri_order.data(), s->d_order, size_t(s->n_tris) * 4, cudaMemcpyDeviceToHost, s->dev->stream));
        CU_TRY(cudaStreamSynchronize(s->dev->stream));
        s->host_copy_valid = true;
    }
    if (nodes) {
        if (s->width == 1) std::memcpy(nodes, s->built().flat.data(), s->built().flat.size() * sizeof(ptb_bvh_leafbox));
        else if (s->width == 4) std::memcpy(nodes, s->built().nodes4.data(), s->built().nodes4.size() * sizeof(ptb_bvh_node4));
        else std::memcpy(nodes, s->built().nodes.data(), s->built().nodes.size() * sizeof(ptb_bvh_node));
    }
    if (tri_order) std::memcpy(tri_order, s->built().tri_order.data(), s->built().tri_order.size() * sizeof(int32_t));
    return PTB_OK;
}

// Which form a render mode uses.  A FLAT scene tests every leaf box for every ray: that beats the tree walk when the rays of
// a warp go different ways (PATH: C4 +26 %, AO: +5 %), but coherent rays walk the 4-wide tree in lock-step at no loss and
// touch fewer boxes (DIRECT, primary + one shadow ray towards the light: the tree is 7 % faster).  Measured on B200,
// profiles/ (round 2).  The scene keeps both forms resident; results are identical, the visit statistics follow the form.
static int mode_class(const ptb_scene* s, int mode) {
    if (s->cls == ptd::PTD_FLAT && s->d_nodes4 && mode == PTB_MODE_DIRECT) return ptd::PTD_SMALL4;
    return s->cls;
}

extern "C" int ptb_scene_mode_width(ptb_scene* s, int mode) {
    if (!s) return 0;
    const int c = mode_class(s, mode);
    return c == ptd::PTD_FLAT ? 1 : c == ptd::PTD_SMALL4 ? 4 : 2;
}

static ptd::SceneDev scene_dev(const ptb_scene* s, int cls) {
    ptd::SceneDev d;
    d.nodes = s->cls == ptd::PTD_LARGE ? reinterpret_cast<const float4*>(s->d_nodesq) : s->d_nodes;
    d.tris = s->d_tris; d.tris_orig = s->d_tris_orig; d.mats = s->d_mats;
    for (int a = 0; a < 3; ++a) { d.q_lo[a] = s->q_lo[a]; d.q_step[a] = s->q_step[a]; }
    d.n_nodes = s->n_nodes; d.n_tris = s->n_tris; d.n_mats = s->n_mats;
    if (cls == ptd::PTD_SMALL4 && s->cls == ptd::PTD_FLAT) {  // the resident 4-wide tree of a FLAT scene
        d.nodes = s->d_nodes4; d.n_nodes = int(s->built().nodes4.size());
        d.smem_nodes = s->built().smem_nodes4; d.small = 1; d.flat_n = 0; d.lstack = 0; d.ld256 = 0;
        d.stack_depth = 3 * s->built().depth4 + 1;
        return d;
    }
    // Large scenes stage nothing by default: the top of the tree stays in L1 anyway, shared memory left unused is L1 capacity
    // (which the local-memory traversal stacks need), and a node visit without the "staged or global?" fork runs free of
    // divergent paths (node_step2_bf).  tune[4] = n stages an n-node prefix (round 1 measured 1024 nodes 0.83, 256 nodes 1.81,
    // 64 nodes 2.28 Grays/s on the 2M-triangle scene; round 2: 64 -> 0 nodes +1 %).
    const int cap = s->dev->tune[4] > 0 ? s->dev->tune[4] : 0;
    d.smem_nodes = s->small ? s->bfs_nodes : (s->bfs_nodes < cap ? s->bfs_nodes : cap);
    d.small = s->small ? 1 : 0;
    d.flat_n = 0;
    if (s->cls == ptd::PTD_FLAT) {
        d.flat_n = (int(s->built().flat.size()) + 1) & ~1;
        d.smem_nodes = 0;
    }
    d.stack_depth = s->width == 4 ? 3 * s->depth + 1 : s->depth + 1;  // a 4-wide visit defers up to three children
    // scenes traversed from L2/HBM keep the stack in local memory: shared memory then holds only the node
    // prefix and occupancy is bounded by registers (C5: +2.4 %); tune[2]=2 forces the shared-memory stack
    d.lstack = (!s->small && s->dev->tune[2] != 2 && s->depth + 1 <= PTD_LSTACK_ENTRIES) ? 1 : 0;
    d.ld256 = s->dev->tune[8] == 1 ? 0 : 1;  // tune[8]=1: fetch global nodes with four 128-bit loads instead of two 256-bit ones
    return d;
}

// ---- launch helpers -----------------------------------------------------------------------------------

// Opts the kernel into `smem` dynamic bytes and asks for a shared-memory carve-out large enough for every CTA the
// register file admits: left to itself the driver picked a carve-out that capped the 2M-triangle path kernel at 7 of
// its 9 register-limited CTAs per SM (ncu: launch__occupancy_limit_shared_mem 7, 43 % warps active).  Returns that
// CTA count in *per_sm.
template <class K>
static int set_smem(K kernel, size_t smem, int block, int* per_sm = nullptr) {
    if (smem > 48 * 1024) CU_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int n = 0;
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, block, smem));
    if (n < 1) n = 1;
    const size_t want = size_t(n) * (smem + 1024);  // + the 1 KB the system reserves per CTA
    int pct = (int)((want * 100 + 228 * 1024 - 1) / (228 * 1024));
    if (pct > 100) pct = 100;
    CU_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    if (per_sm) *per_sm = n;
    return PTB_OK;
}

template <int MODE, bool BVH, int SMALL, bool STATS>
static int launch_mega_t(ptb_device* dev, const ptd::SceneDev& sc, const ptd::RenderArgs& a) {
    const int block = (a.tune[3] == 64 || a.tune[3] == 32) ? a.tune[3] : 128;
    if (MODE == PTB_MODE_PATH && a.tune[5] != 1) {  // persistent grid with path regeneration (tune[5]=1: one sample per thread)
        // tune[9] = extra KB of (unused) shared memory per CTA: lowers the occupancy for latency-sensitivity measurements
        const size_t smem = ptd::scene_smem_bytes(sc, BVH, SMALL, block) + (a.tune[9] > 0 ? size_t(a.tune[9]) * 1024 : 0);
        // Two schedules of the same per-sample arithmetic: k_path_sm (per-lane state machine, the warp votes the phase) and
        // k_mega_path_regen (while-while query inside a path segment).  tune[5] = 2 / 3 forces the latter / the former.
        bool state_machine = BVH && SMALL == ptd::PTD_LARGE;
        if (a.tune[5] == 2) state_machine = false;
        if (a.tune[5] == 3) state_machine = BVH;
        const long long total = (long long)a.frames_in_batch * a.n_local;
        const long long need = (total + block - 1) / block;
        unsigned long long* work = dev->counters + 32;
        CU_TRY(cudaMemsetAsync(work, 0, sizeof(unsigned long long), dev->stream));
        int per_sm = 0;
        if constexpr (BVH) {
            if (state_machine) {
                // Large scenes: every node comes from global memory (the top of the tree stays in L1 anyway; tune[4] = n stages
                // an n-node prefix as k_mega_path_regen does), which lets the node visit run without divergent paths.
                ptd::SceneDev sc2 = sc;
                if (SMALL == ptd::PTD_LARGE && a.tune[4] == 0) sc2.smem_nodes = 0;
                const size_t smem2 = ptd::scene_smem_bytes(sc2, BVH, SMALL, block) + (a.tune[9] > 0 ? size_t(a.tune[9]) * 1024 : 0);
                // tune[12] = 1: let ptxas use the registers it wants (7 CTAs per SM on the large-scene form) instead of capping at 64 (8 CTAs)
                // the large-scene form without statistics: registers capped at 64 (8 CTAs per SM; tune[12] = 1: uncapped, 9: 56 registers) and
                // six node visits per vote (tune[14] = 1 | 2 | 4: visits per vote, A/B runs)
                auto k = ptd::k_path_sm<SMALL, STATS, 0, SMALL == ptd::PTD_LARGE ? 6 : 1>;
                if constexpr (SMALL == ptd::PTD_LARGE && !STATS) {
                    k = ptd::k_path_sm<SMALL, STATS, 8, 6>;
                    if (a.tune[12] == 1) k = ptd::k_path_sm<SMALL, STATS, 0, 6>;
                    if (a.tune[12] == 9) k = ptd::k_path_sm<SMALL, STATS, 9, 6>;
                    if (a.tune[14] == 1) k = ptd::k_path_sm<SMALL, STATS, 8, 1>;
                    if (a.tune[14] == 2) k = ptd::k_path_sm<SMALL, STATS, 8, 2>;
                    if (a.tune[14] == 4) k = ptd::k_path_sm<SMALL, STATS, 8, 4>;
                }
                // Large scenes on the local-memory stack: the form with the path state and the box-test constants parked in shared memory
                // (k_path_sm2) without statistics: 40 registers and no spills, 12 CTAs per SM.  tune[12] = 1: the registers-only k_path_sm;
                // 28 / 29 / 30: launch bounds of 8 / 9 / 10 CTAs (46 / 46 / 44 registers, 11 resident CTAs; A/B runs).
                if constexpr (SMALL == ptd::PTD_LARGE) {
                    if (a.tune[12] != 1 && a.tune[12] != 9 && a.tune[14] == 0 && sc2.lstack && sc2.smem_nodes == 0 && total < (1ll << 31) && a.tune[9] <= 0 && block == 128) {
                        auto k2 = ptd::k_path_sm2<STATS, STATS ? 0 : 11, 6>;
                        if constexpr (!STATS) {
                            if (a.tune[12] == 28) k2 = ptd::k_path_sm2<false, 8, 6>;
                            if (a.tune[12] == 29) k2 = ptd::k_path_sm2<false, 9, 6>;
                            if (a.tune[12] == 30) k2 = ptd::k_path_sm2<false, 10, 6>;
                        }
                        ptd::RenderArgs a2 = a;  // the kernel reads its quorums as plain parameters
                        if (a2.tune[0] <= 0) a2.tune[0] = 4;
                        if (a2.tune[10] <= 0) a2.tune[10] = 20;
                        if (a2.tune[11] <= 0) a2.tune[11] = 10;
                        const size_t sm2 = ptd::path_sm2_smem_bytes(block);
                        if (int rc = set_smem(k2, sm2, block, &per_sm)) return rc;
                        long long grid2 = (long long)per_sm * dev->prop.multiProcessorCount;
                        if (grid2 > need) grid2 = need;
                        k2<<<(unsigned)grid2, block, sm2, dev->stream>>>(sc2, a2, work);
                        CU_TRY(cudaGetLastError());
                        return PTB_OK;
                    }
                }
                if (int rc = set_smem(k, smem2, block, &per_sm)) return rc;
                if (a.tune[9] < 0 && -a.tune[9] < per_sm) per_sm = -a.tune[9];  // tune[9] = -n: n resident CTAs per SM (latency-sensitivity measurements)
                long long grid = (long long)per_sm * dev->prop.multiProcessorCount;
                if (grid > need) grid = need;
                k<<<(unsigned)grid, block, smem2, dev->stream>>>(sc2, a, work);
                CU_TRY(cudaGetLastError());
                return PTB_OK;
            }
        }
        auto k = ptd::k_mega_path_regen<BVH, SMALL, STATS>;
        // FLAT scenes pool the triangle tests of a warp (flat_mt_coop); tune[13] = 2: every lane loops over its own candidates (A/B runs)
        if constexpr (BVH && SMALL == ptd::PTD_FLAT) if (a.tune[13] != 2) k = ptd::k_mega_path_regen<BVH, SMALL, STATS, true>;
        if (int rc = set_smem(k, smem, block, &per_sm)) return rc;
        long long grid = (long long)per_sm * dev->prop.multiProcessorCount;
        if (grid > need) grid = need;
        k<<<(unsigned)grid, block, smem, dev->stream>>>(sc, a, work);
        CU_TRY(cudaGetLastError());
        return PTB_OK;
    }
    const long long total = (long long)a.frames_in_batch * a.n_local;
    const unsigned grid = (unsigned)((total + block - 1) / block);
    const size_t smem = ptd::scene_smem_bytes(sc, BVH, SMALL, block);
    auto k = ptd::k_mega<MODE, BVH, SMALL, STATS>;
    if (int rc = set_smem(k, smem, block)) return rc;
    k<<<grid, block, smem, dev->stream>>>(sc, a);
    CU_TRY(cudaGetLastError());
    return PTB_OK;
}

template <int MODE>
static int launch_mega_m(ptb_device* dev, const ptd::SceneDev& sc, const ptd::RenderArgs& a, bool bvh, int small, bool stats) {
    using namespace ptd;
    if (!bvh && small == PTD_FLAT) small = PTD_SMALL4;  // brute force only needs the staged triangles
#define PTB_CASE(B, S, T) if (bvh == B && small == S && stats == T) return launch_mega_t<MODE, B, S, T>(dev, sc, a)
    PTB_CASE(true, PTD_FLAT, false); PTB_CASE(true, PTD_FLAT, true);
    PTB_CASE(true, PTD_SMALL4, false); PTB_CASE(true, PTD_SMALL4, true); PTB_CASE(true, PTD_LARGE, false); PTB_CASE(true, PTD_LARGE, true);
    PTB_CASE(false, PTD_SMALL4, false); PTB_CASE(false, PTD_SMALL4, true); PTB_CASE(false, PTD_LARGE, false); PTB_CASE(false, PTD_LARGE, true);
#undef PTB_CASE
    return fail(PTB_E_INVALID, "launch_mega: unreachable");
}

static int launch_mega(ptb_device* dev, int mode, const ptd::SceneDev& sc, const ptd::RenderArgs& a, bool bvh, int small, bool stats) {
    switch (mode) {
        case PTB_MODE_PRIMARY: return launch_mega_m<PTB_MODE_PRIMARY>(dev, sc, a, bvh, small, stats);
        case PTB_MODE_AO: return launch_mega_m<PTB_MODE_AO>(dev, sc, a, bvh, small, stats);
        case PTB_MODE_DIRECT: return launch_mega_m<PTB_MODE_DIRECT>(dev, sc, a, bvh, small, stats);
        case PTB_MODE_PATH: return launch_mega_m<PTB_MODE_PATH>(dev, sc, a, bvh, small, stats);
    }
    return fail(PTB_E_INVALID, "ptb_render: unknown mode %d", mode);
}

// ---- render ---------------------------------------------------------------------------------------------

extern "C" void ptb_render_params_default(ptb_render_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof *p);
    p->width = 512; p->height = 512;  // RaytraceTest.cpp:219
    p->first_frame = 0; p->n_frames = 1;
    p->mode = PTB_MODE_PATH;
    p->accum = PTB_ACCUM_REFERENCE;
    p->integrator = PTB_INTEGRATOR_AUTO;
    p->accel = PTB_ACCEL_BVH;
    p->max_depth = 16;  // GenerateColors.cl:5
    p->ao_samples = 16;
    p->ao_max_dist = 2.0f;
    p->light_quad = 5;
    p->shard_index = 0; p->shard_count = 1; p->shard_block = 64;
}

extern "C" int ptb_render_local_pixels(const ptb_render_params* p) {
    if (!p) return 0;
    const long long n = (long long)p->width * p->height;
    if (p->shard_count <= 1) return (int)n;
    long long c = 0;
    for (long long b = p->shard_index; b * p->shard_block < n; b += p->shard_count) {
        const long long lo = b * p->shard_block, hi = lo + p->shard_block;
        c += (hi < n ? hi : n) - lo;
    }
    return (int)c;
}

static int validate(const ptb_render_params* p) {
    if (!p) return fail(PTB_E_INVALID, "ptb_render: null params");
    if (p->width <= 0 || p->height <= 0 || (long long)p->width * p->height > (1ll << 30))
        return fail(PTB_E_INVALID, "ptb_render: bad image size %dx%d", p->width, p->height);
    if (p->n_frames <= 0 || p->first_frame < 0) return fail(PTB_E_INVALID, "ptb_render: bad frame range");
    if (p->mode < 0 || p->mode > PTB_MODE_PATH) return fail(PTB_E_INVALID, "ptb_render: bad mode %d", p->mode);
    if (p->accum != PTB_ACCUM_REFERENCE && p->accum != PTB_ACCUM_LINEAR) return fail(PTB_E_INVALID, "ptb_render: bad accum");
    if (p->max_depth < 1 || p->max_depth > 4096) return fail(PTB_E_INVALID, "ptb_render: bad max_depth");
    if (p->mode == PTB_MODE_AO && (p->ao_samples < 1 || p->ao_samples > 4096)) return fail(PTB_E_INVALID, "ptb_render: bad ao_samples");
    if (p->output != PTB_OUTPUT_FLOAT4 && p->output != PTB_OUTPUT_RGB8) return fail(PTB_E_INVALID, "ptb_render: bad output format %d", p->output);
    if (p->shard_count > 1 && (p->shard_index < 0 || p->shard_index >= p->shard_count || p->shard_block < 1))
        return fail(PTB_E_INVALID, "ptb_render: bad shard spec");
    return PTB_OK;
}

// The area light of the render args (ptb_render and ptb_scene_shade): light_p1 / ea / eb from the params, or derived from the
// triangles of light_quad when ea is all zero (DIRECT only); for DIRECT also |cross(ea, eb)| and its unit vector, the same for
// every sample.
static int setup_light(const ptb_scene* scene, const ptb_render_params* p, ptd::RenderArgs& a) {
    a.light_quad = p->light_quad;
    const bool have_light = p->light_ea[0] != 0.f || p->light_ea[1] != 0.f || p->light_ea[2] != 0.f;
    if (have_light) {
        std::memcpy(a.light_p1, p->light_p1, 12); std::memcpy(a.light_ea, p->light_ea, 12); std::memcpy(a.light_eb, p->light_eb, 12);
    } else if (p->mode == PTB_MODE_DIRECT && !scene->lights.empty()) {  // device-built scene: its light table (k_scene_lights)
        const int q = p->light_quad;
        if (q < 0 || q >= scene->n_mats || scene->lights[size_t(q)].q >= scene->n_tris)
            return fail(PTB_E_NOTFOUND, "ptb_light_from_quad: no triangle pair with id %d", q);
        const ptd::SceneLight& L = scene->lights[size_t(q)];
        std::memcpy(a.light_p1, L.p1, 12); std::memcpy(a.light_ea, L.ea, 12); std::memcpy(a.light_eb, L.eb, 12);
    } else if (p->mode == PTB_MODE_DIRECT) {
        if (int rc = ptb_light_from_quad(scene->host_tris.data(), scene->n_tris, p->light_quad, a.light_p1, a.light_ea, a.light_eb)) return rc;
    }
    if (p->mode == PTB_MODE_DIRECT) {
        // |cross(ea, eb)| and its unit vector, spelled as the kernels (and the oracle) spell them per sample: products and
        // sums rounded one by one (this file is compiled without FMA contraction), IEEE sqrt and division
        const float* ea = a.light_ea; const float* eb = a.light_eb;
        const float cx = ea[1] * eb[2] - ea[2] * eb[1], cy = ea[2] * eb[0] - ea[0] * eb[2], cz = ea[0] * eb[1] - ea[1] * eb[0];
        const float dd = (cx * cx + cy * cy) + cz * cz;
        a.light_area = std::sqrt(dd);
        const float inv = 1.0f / std::sqrt(dd);
        a.light_n[0] = cx * inv; a.light_n[1] = cy * inv; a.light_n[2] = cz * inv;
    }
    return PTB_OK;
}

// `ext_samples` + `phase` split one call for the frame-ahead batching of ptb_launch1d: PHASE_TRACE writes the samples of
// all n_frames into ext_samples and stops; PHASE_RESOLVE folds n_frames already-traced frames from ext_samples into d_frame.
enum { PHASE_BOTH = 0, PHASE_TRACE = 1, PHASE_RESOLVE = 2 };
static int render_impl(ptb_device* dev, ptb_scene* scene, const ptb_render_params* p, float4* d_frame, size_t frame_bytes,
                       ptb_pixel_stats* d_stats, size_t stats_bytes, ptb_counters* counters, float4* ext_samples = nullptr,
                       int phase = PHASE_BOTH, float4* const* peers = nullptr, int n_peers = -1) {
    if (!dev || !scene || (!d_frame && phase != PHASE_TRACE)) return fail(PTB_E_INVALID, "ptb_render: null argument");
    if (int rc = validate(p)) return rc;
    if (scene->dev != dev) return fail(PTB_E_INVALID, "ptb_render: scene belongs to another device");
    if (set_device(dev)) return PTB_E_CUDA;
    const int n_local = ptb_render_local_pixels(p);
    if (n_local <= 0) return fail(PTB_E_INVALID, "ptb_render: shard owns no pixels");
    const bool gather = n_peers >= 0;  // d_frame (and the peers) are full images indexed by global pixel id
    const size_t frame_need = gather ? size_t(p->width) * size_t(p->height) * 16 : size_t(n_local) * 16;
    if (phase != PHASE_TRACE && frame_bytes < frame_need) return fail(PTB_E_INVALID, "ptb_render: frame buffer too small (%zu < %zu)", frame_bytes, frame_need);
    if (d_stats && stats_bytes < size_t(n_local) * sizeof(ptb_pixel_stats)) return fail(PTB_E_INVALID, "ptb_render: stats buffer too small");
    if (p->mode == PTB_MODE_DIRECT && (p->light_quad < 0 || p->light_quad >= scene->n_mats))
        return fail(PTB_E_INVALID, "ptb_render: light_quad %d out of range", p->light_quad);

    const int small = mode_class(scene, p->mode);
    ptd::SceneDev sc = scene_dev(scene, small);
    const bool bvh = p->accel == PTB_ACCEL_BVH;
    const bool stats = p->collect_stats != 0;

    // batch of frames kept in flight
    int fpb = p->frames_per_batch;
    if (fpb <= 0) {
        // Sample slots in flight per launch.  A persistent path kernel ends with a tail in which the few longest walks run
        // alone (a ray grazing a tessellated wall visits hundreds of nodes): with one 4K frame per launch that tail was
        // 11 % of the 2M-triangle scene's time (16 frames per launch: 3.35 -> 3.76 Grays/s; Cornell box at 4K +2.6 %).
        // 128 Mi slots = 2 GB of samples; the wavefront integrator, which keeps ~150 bytes of queues per slot, stays at 32 Mi.
        // tune[15] = log2 of the slot target overrides (A/B runs).
        const bool wavefront = p->integrator == PTB_INTEGRATOR_WAVEFRONT;
        long long target = p->mode == PTB_MODE_PATH ? (wavefront ? 32ll << 20 : 128ll << 20) : 4ll << 20;
        if (dev->tune[15] > 0 && dev->tune[15] < 31) target = 1ll << dev->tune[15];
        fpb = (int)((target + n_local - 1) / n_local);
    }
    if (fpb > p->n_frames) fpb = p->n_frames;
    if (fpb < 1) fpb = 1;
    if (ext_samples) fpb = p->n_frames;  // the caller sized ext_samples for the whole range
    else if (int rc = ensure(&dev->samples, &dev->samples_bytes, size_t(fpb) * n_local * 16)) return rc;
    if (p->accum == PTB_ACCUM_LINEAR)
        if (int rc = ensure(&dev->sum, &dev->sum_bytes, size_t(n_local) * 16)) return rc;
    if (!dev->cumulative_counters) CU_TRY(cudaMemsetAsync(dev->counters, 0, sizeof(unsigned long long) * 64, dev->stream));
    else if (phase != PHASE_RESOLVE) dev->cumulative_samples += (uint64_t)n_local * (uint64_t)p->n_frames;

    ptd::RenderArgs a;
    std::memset(&a, 0, sizeof a);
    a.width = p->width; a.height = p->height;
    a.n_local = n_local;
    a.max_depth = p->max_depth; a.ao_samples = p->ao_samples; a.ao_max_dist = p->ao_max_dist;
    if (int rc = setup_light(scene, p, a)) return rc;
    a.cam_inv_w = 1.0f / (float)p->width; a.cam_inv_h = 1.0f / (float)p->height;  // GenerateColors.cl:265
    a.cam_aspect = (float)p->width / (float)p->height;                            // :266
    a.shard.index = p->shard_index; a.shard.count = p->shard_count < 1 ? 1 : p->shard_count; a.shard.block = p->shard_block < 1 ? 1 : p->shard_block;
    a.samples = ext_samples ? ext_samples : static_cast<float4*>(dev->samples);
    // One frame with accum = LINEAR: the mean of one sample is the sample (0 + c = c and c / 1 = c exactly, w = 1), and without image
    // sharding a pixel's slot in the batch IS its place in the frame -- the integrator writes the frame itself and the resolve
    // launch is dropped (C1: one launch instead of two on a 30 us step).  Bit-identical by construction.
    const bool direct = phase == PHASE_BOTH && !ext_samples && p->accum == PTB_ACCUM_LINEAR && p->n_frames == 1 && p->shard_count <= 1 && n_peers <= 0;
    if (direct) a.samples = d_frame;
    a.stats = stats ? d_stats : nullptr;
    a.stats_frame = p->first_frame + p->n_frames - 1;
    a.counters = dev->counters;
    for (int k = 0; k < 16; ++k) a.tune[k] = dev->tune[k];

    // AUTO = the faster integrator as measured on B200 (DESIGN.md section 5).  With 4-wide nodes for
    // shared-memory-resident scenes and path regeneration, the megakernel wins every BASELINE configuration
    // (C4: 11.3 vs 10.7 Grays/s, C2: 31.0 vs 25.9, C5: 2.9 vs 2.0); the wavefront integrator stays selectable.
    int integrator = p->integrator;
    if (integrator == PTB_INTEGRATOR_AUTO) integrator = PTB_INTEGRATOR_MEGAKERNEL;

    for (int f0 = 0; f0 < p->n_frames; f0 += fpb) {
        const int nb = (p->n_frames - f0 < fpb) ? p->n_frames - f0 : fpb;
        a.first_frame = p->first_frame + f0;
        a.frames_in_batch = nb;
        cudaEvent_t* ev = nullptr;
        if (dev->profiling) {
            if (dev->ev_used + 3 > dev->ev_pool.size()) {
                for (int k = 0; k < 3; ++k) {
                    cudaEvent_t e;
                    CU_TRY(cudaEventCreate(&e));
                    dev->ev_pool.push_back(e);
                }
            }
            ev = &dev->ev_pool[dev->ev_used];
            dev->ev_used += 3;
            CU_TRY(cudaEventRecord(ev[0], dev->stream));
        }
        if (phase == PHASE_RESOLVE) {
        } else if (integrator == PTB_INTEGRATOR_WAVEFRONT) {
            if (int rc = ptd::wavefront_render(dev->stream, &dev->wf, &dev->wf_bytes, dev->counters, p->mode, sc, a, bvh, small, stats,
                                               dev->prop.multiProcessorCount, &dev->kernel_launches))
                return rc;
        } else {
            if (int rc = launch_mega(dev, p->mode, sc, a, bvh, small, stats)) return rc;
            dev->kernel_launches += 1;
        }
        if (ev) CU_TRY(cudaEventRecord(ev[1], dev->stream));
        if (phase != PHASE_RESOLVE) dev->integrator_launch_batches++;
        if (phase == PHASE_TRACE) continue;
        if (direct) {
            if (ev) CU_TRY(cudaEventRecord(ev[2], dev->stream));
            continue;
        }
        ptd::ResolveArgs r;
        r.samples = a.samples; r.n_local = n_local; r.frames_in_batch = nb; r.first_frame = a.first_frame;
        r.accum = p->accum; r.first_batch = f0 == 0; r.last_batch = f0 + nb >= p->n_frames;
        r.total_frames = p->n_frames;
        r.sum = static_cast<float4*>(dev->sum); r.frame = d_frame;
        r.gather = gather ? 1 : 0; r.n_peers = gather ? n_peers : 0; r.shard = a.shard;
        for (int k = 0; k < PTB_MAX_PEERS; ++k) r.peers[k] = (gather && k < n_peers) ? peers[k] : nullptr;
        ptd::k_resolve<<<(n_local + 255) / 256, 256, 0, dev->stream>>>(r);
        CU_TRY(cudaGetLastError());
        dev->kernel_launches += 1;
        if (ev) CU_TRY(cudaEventRecord(ev[2], dev->stream));
    }
    if (counters) {
        unsigned long long h[ptd::CTR_COUNT];
        CU_TRY(cudaMemcpyAsync(h, dev->counters, sizeof h, cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        std::memset(counters, 0, sizeof *counters);
        counters->rays_closest = h[ptd::CTR_CLOSEST]; counters->rays_any = h[ptd::CTR_ANY];
        counters->nodes = h[ptd::CTR_NODES]; counters->tri_tests = h[ptd::CTR_TESTS];
        counters->samples = (uint64_t)n_local * (uint64_t)p->n_frames;
    }
    return PTB_OK;
}

extern "C" int ptb_render(ptb_device* dev, ptb_scene* scene, const ptb_render_params* params, ptb_buffer* frame,
                          ptb_buffer* stats, ptb_counters* counters) {
    if (!frame) return fail(PTB_E_INVALID, "ptb_render: null frame buffer");
    return render_impl(dev, scene, params, static_cast<float4*>(frame->d_ptr), frame->bytes,
                       stats ? static_cast<ptb_pixel_stats*>(stats->d_ptr) : nullptr, stats ? stats->bytes : 0, counters);
}

// ---- scene queries on caller-owned device ray buffers -------------------------------------------------------------
// k_intersect: tree forms run a persistent grid (resident CTAs, rays fetched from a work counter in device scratch); FLAT scenes
// one thread per ray.

template <bool ANY, int SMALL, bool STATS>
static int launch_intersect_t(ptb_device* dev, const ptd::SceneDev& sc, const float4* rays, float4* hits, uint2* stats, int n) {
    const int block = 128;
    const size_t smem = ptd::scene_smem_bytes(sc, true, SMALL, block);
    auto k = ptd::k_intersect<ANY, SMALL, STATS>;
    int per_sm = 0;
    if (int rc = set_smem(k, smem, block, &per_sm)) return rc;
    long long grid = ((long long)n + block - 1) / block;
    unsigned int* work = static_cast<unsigned int*>(dev->isect);
    if (SMALL != ptd::PTD_FLAT) {
        const long long resident = (long long)per_sm * dev->prop.multiProcessorCount;
        if (grid > resident) grid = resident;
        CU_TRY(cudaMemsetAsync(work, 0, sizeof(unsigned int), dev->stream));
    }
    k<<<(unsigned)grid, block, smem, dev->stream>>>(sc, rays, hits, stats, (unsigned int)n, work, dev->counters);
    CU_TRY(cudaGetLastError());
    dev->kernel_launches += 1;
    return PTB_OK;
}

extern "C" int ptb_scene_intersect(ptb_device* dev, ptb_scene* scene, int query, ptb_buffer* rays, int n_rays, ptb_buffer* hits,
                                   ptb_buffer* stats, ptb_counters* counters) {
    if (!dev || !scene || !rays || !hits) return fail(PTB_E_INVALID, "ptb_scene_intersect: null device, scene, rays or hits");
    if (n_rays < 0) return fail(PTB_E_INVALID, "ptb_scene_intersect: n_rays %d < 0", n_rays);
    if (query != PTB_QUERY_CLOSEST && query != PTB_QUERY_ANY) return fail(PTB_E_INVALID, "ptb_scene_intersect: unknown query %d", query);
    if (scene->dev != dev) return fail(PTB_E_INVALID, "ptb_scene_intersect: scene belongs to another device");
    if (rays->dev != dev || hits->dev != dev || (stats && stats->dev != dev))
        return fail(PTB_E_INVALID, "ptb_scene_intersect: buffer belongs to another device");
    const size_t n = size_t(n_rays);
    if (rays->bytes < n * sizeof(ptb_ray)) return fail(PTB_E_INVALID, "ptb_scene_intersect: rays buffer too small (%zu < %zu)", rays->bytes, n * sizeof(ptb_ray));
    if (hits->bytes < n * sizeof(ptb_hit)) return fail(PTB_E_INVALID, "ptb_scene_intersect: hits buffer too small (%zu < %zu)", hits->bytes, n * sizeof(ptb_hit));
    if (stats && stats->bytes < n * 8) return fail(PTB_E_INVALID, "ptb_scene_intersect: stats buffer too small (%zu < %zu)", stats->bytes, n * 8);
    if ((reinterpret_cast<uintptr_t>(rays->d_ptr) & 31u) != 0)
        return fail(PTB_E_INVALID, "ptb_scene_intersect: rays must be 32-byte aligned (one 256-bit load per ray)");
    if ((reinterpret_cast<uintptr_t>(hits->d_ptr) & 15u) != 0 || (stats && (reinterpret_cast<uintptr_t>(stats->d_ptr) & 7u) != 0))
        return fail(PTB_E_INVALID, "ptb_scene_intersect: hits must be 16-byte and stats 8-byte aligned");
    if (n_rays == 0) {
        if (counters) std::memset(counters, 0, sizeof *counters);
        return PTB_OK;
    }
    if (set_device(dev)) return PTB_E_CUDA;
    if (!dev->cumulative_counters) CU_TRY(cudaMemsetAsync(dev->counters, 0, sizeof(unsigned long long) * ptd::CTR_COUNT, dev->stream));
    {
        if (int rc = ensure(&dev->isect, &dev->isect_bytes, 256)) return rc;
        const ptd::SceneDev sc = scene_dev(scene, scene->cls);
        const float4* r = static_cast<const float4*>(rays->d_ptr);
        float4* h = static_cast<float4*>(hits->d_ptr);
        uint2* s = stats ? static_cast<uint2*>(stats->d_ptr) : nullptr;
        const bool any = query == PTB_QUERY_ANY, st = s != nullptr;
        const int cls = scene->cls;
        int rc = fail(PTB_E_INVALID, "ptb_scene_intersect: unreachable");
#define PTB_ISECT_CASE(A, S, T) if (any == A && cls == S && st == T) rc = launch_intersect_t<A, S, T>(dev, sc, r, h, s, n_rays)
        PTB_ISECT_CASE(false, ptd::PTD_FLAT, false); PTB_ISECT_CASE(false, ptd::PTD_FLAT, true);
        PTB_ISECT_CASE(true, ptd::PTD_FLAT, false); PTB_ISECT_CASE(true, ptd::PTD_FLAT, true);
        PTB_ISECT_CASE(false, ptd::PTD_SMALL4, false); PTB_ISECT_CASE(false, ptd::PTD_SMALL4, true);
        PTB_ISECT_CASE(true, ptd::PTD_SMALL4, false); PTB_ISECT_CASE(true, ptd::PTD_SMALL4, true);
        PTB_ISECT_CASE(false, ptd::PTD_LARGE, false); PTB_ISECT_CASE(false, ptd::PTD_LARGE, true);
        PTB_ISECT_CASE(true, ptd::PTD_LARGE, false); PTB_ISECT_CASE(true, ptd::PTD_LARGE, true);
#undef PTB_ISECT_CASE
        if (rc) return rc;
    }
    if (counters) {
        unsigned long long hc[ptd::CTR_COUNT];
        CU_TRY(cudaMemcpyAsync(hc, dev->counters, sizeof hc, cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        std::memset(counters, 0, sizeof *counters);
        counters->rays_closest = hc[ptd::CTR_CLOSEST]; counters->rays_any = hc[ptd::CTR_ANY];
        counters->nodes = hc[ptd::CTR_NODES]; counters->tri_tests = hc[ptd::CTR_TESTS];
    }
    return PTB_OK;
}

// ---- render-mode samples along caller-owned device rays -----------------------------------------------------------------
// The kernels ptb_render's megakernel path launches for the mode's scene form, with their default selection, and the ray
// source ptd::SampleRays in place of the camera: PRIMARY / AO / DIRECT run k_mega (one thread per ray); PATH runs k_path_sm2 on
// large scenes with the local-memory stack and k_mega_path_regen elsewhere (FLAT scenes with the warp-pooled triangle phase).

template <int MODE, int SMALL, bool STATS>
static int launch_shade_t(ptb_device* dev, const ptd::SceneDev& sc, const ptd::ShadeArgs& a) {
    const int block = 128;
    const long long n = a.n_local;
    int per_sm = 0;
    if constexpr (MODE == PTB_MODE_PATH) {
        const long long need = (n + block - 1) / block;
        unsigned long long* work = dev->counters + 32;  // the path kernels' work counter
        CU_TRY(cudaMemsetAsync(work, 0, sizeof(unsigned long long), dev->stream));
        if (SMALL == ptd::PTD_LARGE && sc.lstack) {
            ptd::SceneDev sc2 = sc;
            sc2.smem_nodes = 0;  // k_path_sm2 fetches every node from global memory
            auto k2 = ptd::k_path_sm2_rays<STATS, STATS ? 0 : 11, 6>;
            ptd::ShadeArgs a2 = a;  // quorums resolved as for ptb_render
            if (a2.tune[0] <= 0) a2.tune[0] = 4;
            if (a2.tune[10] <= 0) a2.tune[10] = 20;
            if (a2.tune[11] <= 0) a2.tune[11] = 10;
            const size_t sm2 = ptd::path_sm2_smem_bytes(block);
            if (int rc = set_smem(k2, sm2, block, &per_sm)) return rc;
            long long grid = (long long)per_sm * dev->prop.multiProcessorCount;
            if (grid > need) grid = need;
            k2<<<(unsigned)grid, block, sm2, dev->stream>>>(sc2, a2, work);
        } else {
            auto k = ptd::k_mega_path_regen<true, SMALL, STATS, SMALL == ptd::PTD_FLAT, ptd::SampleRays>;
            const size_t smem = ptd::scene_smem_bytes(sc, true, SMALL, block);
            if (int rc = set_smem(k, smem, block, &per_sm)) return rc;
            long long grid = (long long)per_sm * dev->prop.multiProcessorCount;
            if (grid > need) grid = need;
            k<<<(unsigned)grid, block, smem, dev->stream>>>(sc, a, work);
        }
    } else {
        auto k = ptd::k_mega<MODE, true, SMALL, STATS, ptd::SampleRays>;
        const size_t smem = ptd::scene_smem_bytes(sc, true, SMALL, block);
        if (int rc = set_smem(k, smem, block)) return rc;
        k<<<(unsigned)((n + block - 1) / block), block, smem, dev->stream>>>(sc, a);
    }
    CU_TRY(cudaGetLastError());
    dev->kernel_launches += 1;
    return PTB_OK;
}

template <int MODE>
static int launch_shade_m(ptb_device* dev, const ptd::SceneDev& sc, const ptd::ShadeArgs& a, int small, bool stats) {
#define PTB_SHADE_CASE(S, T) if (small == S && stats == T) return launch_shade_t<MODE, S, T>(dev, sc, a)
    PTB_SHADE_CASE(ptd::PTD_FLAT, false); PTB_SHADE_CASE(ptd::PTD_FLAT, true);
    PTB_SHADE_CASE(ptd::PTD_SMALL4, false); PTB_SHADE_CASE(ptd::PTD_SMALL4, true);
    PTB_SHADE_CASE(ptd::PTD_LARGE, false); PTB_SHADE_CASE(ptd::PTD_LARGE, true);
#undef PTB_SHADE_CASE
    return fail(PTB_E_INVALID, "ptb_scene_shade: unreachable");
}

extern "C" int ptb_scene_shade(ptb_device* dev, ptb_scene* scene, const ptb_render_params* p, ptb_buffer* rays, int n_rays,
                               ptb_buffer* radiance, ptb_buffer* stats, ptb_counters* counters) {
    if (!dev || !scene || !p || !rays || !radiance)
        return fail(PTB_E_INVALID, "ptb_scene_shade: null device, scene, params, rays or radiance");
    if (n_rays < 0) return fail(PTB_E_INVALID, "ptb_scene_shade: n_rays %d < 0", n_rays);
    if (p->mode < 0 || p->mode > PTB_MODE_PATH) return fail(PTB_E_INVALID, "ptb_scene_shade: bad mode %d", p->mode);
    if (p->max_depth < 1 || p->max_depth > 4096) return fail(PTB_E_INVALID, "ptb_scene_shade: bad max_depth %d", p->max_depth);
    if (p->mode == PTB_MODE_AO && (p->ao_samples < 1 || p->ao_samples > 4096))
        return fail(PTB_E_INVALID, "ptb_scene_shade: bad ao_samples %d", p->ao_samples);
    if (p->accel != PTB_ACCEL_BVH) return fail(PTB_E_INVALID, "ptb_scene_shade: accel %d: only PTB_ACCEL_BVH is available", p->accel);
    if (p->integrator != PTB_INTEGRATOR_AUTO && p->integrator != PTB_INTEGRATOR_MEGAKERNEL)
        return fail(PTB_E_INVALID, "ptb_scene_shade: integrator %d: only the megakernel integrator is available", p->integrator);
    if (scene->dev != dev) return fail(PTB_E_INVALID, "ptb_scene_shade: scene belongs to another device");
    if (rays->dev != dev || radiance->dev != dev || (stats && stats->dev != dev))
        return fail(PTB_E_INVALID, "ptb_scene_shade: buffer belongs to another device");
    if (p->mode == PTB_MODE_DIRECT && (p->light_quad < 0 || p->light_quad >= scene->n_mats))
        return fail(PTB_E_INVALID, "ptb_scene_shade: light_quad %d out of range", p->light_quad);
    const size_t n = size_t(n_rays);
    if (rays->bytes < n * sizeof(ptb_sample_ray))
        return fail(PTB_E_INVALID, "ptb_scene_shade: rays buffer too small (%zu < %zu)", rays->bytes, n * sizeof(ptb_sample_ray));
    if (radiance->bytes < n * 16) return fail(PTB_E_INVALID, "ptb_scene_shade: radiance buffer too small (%zu < %zu)", radiance->bytes, n * 16);
    if (stats && stats->bytes < n * sizeof(ptb_pixel_stats))
        return fail(PTB_E_INVALID, "ptb_scene_shade: stats buffer too small (%zu < %zu)", stats->bytes, n * sizeof(ptb_pixel_stats));
    if ((reinterpret_cast<uintptr_t>(rays->d_ptr) & 31u) != 0)
        return fail(PTB_E_INVALID, "ptb_scene_shade: rays must be 32-byte aligned (one 256-bit load per ray)");
    if ((reinterpret_cast<uintptr_t>(radiance->d_ptr) & 15u) != 0 || (stats && (reinterpret_cast<uintptr_t>(stats->d_ptr) & 15u) != 0))
        return fail(PTB_E_INVALID, "ptb_scene_shade: radiance and stats must be 16-byte aligned");
    if (n_rays == 0) {
        if (counters) std::memset(counters, 0, sizeof *counters);
        return PTB_OK;
    }
    if (set_device(dev)) return PTB_E_CUDA;
    const int small = mode_class(scene, p->mode);
    const ptd::SceneDev sc = scene_dev(scene, small);
    ptd::ShadeArgs a;
    std::memset(&a, 0, sizeof a);
    a.frames_in_batch = 1;
    a.n_local = n_rays;  // sample slot i = ray i
    a.max_depth = p->max_depth; a.ao_samples = p->ao_samples; a.ao_max_dist = p->ao_max_dist;
    if (int rc = setup_light(scene, p, a)) return rc;
    a.samples = static_cast<float4*>(radiance->d_ptr);
    a.stats = stats ? static_cast<ptb_pixel_stats*>(stats->d_ptr) : nullptr;
    a.counters = dev->counters;
    for (int k = 0; k < 16; ++k) a.tune[k] = dev->tune[k];
    a.rays = static_cast<const float4*>(rays->d_ptr);
    if (!dev->cumulative_counters) CU_TRY(cudaMemsetAsync(dev->counters, 0, sizeof(unsigned long long) * ptd::CTR_COUNT, dev->stream));
    else dev->cumulative_samples += n;
    const bool st = stats != nullptr;
    int rc = PTB_OK;
    switch (p->mode) {
        case PTB_MODE_PRIMARY: rc = launch_shade_m<PTB_MODE_PRIMARY>(dev, sc, a, small, st); break;
        case PTB_MODE_AO: rc = launch_shade_m<PTB_MODE_AO>(dev, sc, a, small, st); break;
        case PTB_MODE_DIRECT: rc = launch_shade_m<PTB_MODE_DIRECT>(dev, sc, a, small, st); break;
        default: rc = launch_shade_m<PTB_MODE_PATH>(dev, sc, a, small, st); break;
    }
    if (rc) return rc;
    if (counters) {
        unsigned long long hc[ptd::CTR_COUNT];
        CU_TRY(cudaMemcpyAsync(hc, dev->counters, sizeof hc, cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        std::memset(counters, 0, sizeof *counters);
        counters->rays_closest = hc[ptd::CTR_CLOSEST]; counters->rays_any = hc[ptd::CTR_ANY];
        counters->nodes = hc[ptd::CTR_NODES]; counters->tri_tests = hc[ptd::CTR_TESTS];
        counters->samples = n;
    }
    return PTB_OK;
}

// ---- image-sharded render that delivers straight into the full images of this rank and its peers ----------------
// Buffers of other processes are mapped with CUDA IPC (NVLink / NVSwitch peer memory); k_resolve stores every finished
// pixel at its global position in each image, so the exchange step of image sharding (SURVEY 8e) needs no collective
// and no un-interleave pass: only a barrier before the images are read.

extern "C" int ptb_buffer_ipc_export(ptb_buffer* buf, void* handle64) {
    if (!buf || !handle64) return fail(PTB_E_INVALID, "ptb_buffer_ipc_export: null argument");
    if (!buf->owned) return fail(PTB_E_INVALID, "ptb_buffer_ipc_export: only buffers created by ptb_buffer_create can be exported");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    if (set_device(buf->dev)) return PTB_E_CUDA;
    cudaIpcMemHandle_t h;
    CU_TRY(cudaIpcGetMemHandle(&h, buf->d_ptr));
    std::memcpy(handle64, &h, sizeof h);
    return PTB_OK;
}

extern "C" int ptb_buffer_ipc_import(ptb_device* dev, const void* handle64, size_t bytes, ptb_buffer** out) {
    if (!dev || !handle64 || !out) return fail(PTB_E_INVALID, "ptb_buffer_ipc_import: null argument");
    *out = nullptr;
    if (set_device(dev)) return PTB_E_CUDA;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle64, sizeof h);
    void* p = nullptr;
    CU_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ptb_buffer* b = new ptb_buffer();
    b->dev = dev; b->d_ptr = p; b->bytes = bytes; b->owned = false; b->ipc = true;
    dev->live_buffers++;
    *out = b;
    return PTB_OK;
}

extern "C" int ptb_render_gather(ptb_device* dev, ptb_scene* scene, const ptb_render_params* params, ptb_buffer* full_frame,
                                 ptb_buffer* const* peer_frames, int n_peers, ptb_counters* counters) {
    if (!full_frame || n_peers < 0 || n_peers > PTB_MAX_PEERS || (n_peers && !peer_frames))
        return fail(PTB_E_INVALID, "ptb_render_gather: bad arguments (0..%d peers)", PTB_MAX_PEERS);
    float4* pp[PTB_MAX_PEERS] = {};
    const size_t need = params ? size_t(params->width) * size_t(params->height) * 16 : 0;
    for (int k = 0; k < n_peers; ++k) {
        if (!peer_frames[k] || peer_frames[k]->bytes < need) return fail(PTB_E_INVALID, "ptb_render_gather: peer image %d is missing or too small", k);
        pp[k] = static_cast<float4*>(peer_frames[k]->d_ptr);
    }
    return render_impl(dev, scene, params, static_cast<float4*>(full_frame->d_ptr), full_frame->bytes, nullptr, 0, counters,
                       nullptr, PHASE_BOTH, pp, n_peers);
}

// content hash of the caller's records (decides whether the resident scene must be rebuilt).  Four independent
// multiply-xorshift lanes over 32-byte stripes: the 2M-triangle scene is 128 MB and is hashed on every call.
static uint64_t content_hash(const void* p, size_t n, uint64_t h) {
    const unsigned char* b = static_cast<const unsigned char*>(p);
    uint64_t l0 = h ^ 0x9E3779B97F4A7C15ull, l1 = h ^ 0xC2B2AE3D27D4EB4Full, l2 = h ^ 0x165667B19E3779F9ull, l3 = h ^ 0x27D4EB2F165667C5ull;
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        uint64_t w[4];
        std::memcpy(w, b + i, 32);
        l0 = (l0 ^ w[0]) * 0x100000001B3ull; l0 ^= l0 >> 29;
        l1 = (l1 ^ w[1]) * 0x100000001B3ull; l1 ^= l1 >> 29;
        l2 = (l2 ^ w[2]) * 0x100000001B3ull; l2 ^= l2 >> 29;
        l3 = (l3 ^ w[3]) * 0x100000001B3ull; l3 ^= l3 >> 29;
    }
    h = (((l0 * 31 + l1) * 31 + l2) * 31 + l3) ^ (uint64_t)n;
    for (; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
    return h;
}

static int ensure_buffer(ptb_device* dev, ptb_buffer** b, size_t bytes) {
    if (*b && (*b)->bytes >= bytes) return PTB_OK;
    if (*b) ptb_buffer_destroy(*b);
    *b = nullptr;
    return ptb_buffer_create(dev, bytes, b);
}

static bool is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

extern "C" int ptb_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(PTB_E_INVALID, "ptb_host_alloc: null out");
    *out = nullptr;
    CU_TRY(cudaMallocHost(out, bytes ? bytes : 1));
    return PTB_OK;
}
extern "C" int ptb_host_free(void* p) {
    if (p) CU_TRY(cudaFreeHost(p));
    return PTB_OK;
}

struct ptb_job {
    ptb_device* dev;
    int slot;
    uint64_t serial;
};

extern "C" int ptb_job_wait(ptb_job* job) {
    if (!job) return fail(PTB_E_INVALID, "ptb_job_wait: null job");
    ptb_device* dev = job->dev;
    auto& sl = dev->slots[job->slot];
    int rc = PTB_OK;
    if (!sl.busy || sl.serial != job->serial) {  // a handle that was already waited for (the slot may serve a newer job by now)
        delete job;
        return fail(PTB_E_INVALID, "ptb_job_wait: this job has already been waited for");
    }
    {
        if (set_device(dev)) rc = PTB_E_CUDA;
        cudaError_t e = cudaEventSynchronize(sl.ev_done);
        if (e != cudaSuccess) rc = fail(PTB_E_CUDA, "ptb_job_wait: %s", cudaGetErrorString(e));
        if (rc == PTB_OK) {
            char* pin = static_cast<char*>(sl.pin);
            if (!sl.direct_frame) std::memcpy(sl.out, pin, sl.fb);
            if (sl.sb && !sl.direct_stats) std::memcpy(sl.out_stats, pin + sl.fb, sl.sb);
        }
        sl.busy = false;
    }
    delete job;
    return rc;
}

// Asynchronous end-to-end render with HOST buffers.  Two slots are double-buffered: while the
// frame of job j travels device->host on the copy stream, job j+1 renders on the main stream.
extern "C" int ptb_render_host_async(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats,
                                     int n_mats, const ptb_render_params* params, float* out_rgba,
                                     ptb_pixel_stats* out_stats, ptb_job** job_out) {
    if (!dev || !tris || !mats || !out_rgba || !job_out) return fail(PTB_E_INVALID, "ptb_render_host_async: null argument");
    *job_out = nullptr;
    if (int rc = validate(params)) return rc;
    if (set_device(dev)) return PTB_E_CUDA;
    const int n_local = ptb_render_local_pixels(params);
    const size_t tb = size_t(n_tris) * sizeof(ptb_triangle), mb = size_t(n_mats) * sizeof(ptb_material);
    const size_t fb = size_t(n_local) * 16, sb = out_stats ? size_t(n_local) * sizeof(ptb_pixel_stats) : 0;
    const bool rgb8 = params->output == PTB_OUTPUT_RGB8;
    if (rgb8 && params->accum == PTB_ACCUM_REFERENCE && params->first_frame > 0)
        return fail(PTB_E_INVALID, "ptb_render_host: RGB8 output cannot carry the gamma-space state of accum=REFERENCE across calls "
                                   "(first_frame > 0); use FLOAT4 output (accum=LINEAR carries nothing across calls: it is the mean of this call's frames)");
    const size_t cb = rgb8 ? size_t(n_local) * 3 : fb;  // bytes of the image that travel to the host
    const int si = !dev->slots[0].busy ? 0 : (!dev->slots[1].busy ? 1 : -1);  // any free slot
    if (si < 0) return fail(PTB_E_INVALID, "ptb_render_host_async: two jobs are in flight; wait for one first");
    auto& sl = dev->slots[si];
    // The gamma-space running mean of accum=REFERENCE continues from the caller's out_rgba, which is uploaded NOW: with a job still
    // in flight that state may not have reached the host yet (its D2H is asynchronous, pageable buffers land at ptb_job_wait), and
    // the frames in between would silently drop out of the mean.  A progressive REFERENCE loop is sequential by its definition
    // (GenerateColors.cl:318-321 reads the previous frame's gDst): wait for the previous job first.
    if (params->accum == PTB_ACCUM_REFERENCE && params->first_frame > 0 && (dev->slots[0].busy || dev->slots[1].busy))
        return fail(PTB_E_INVALID, "ptb_render_host_async: accum=REFERENCE with first_frame > 0 continues from out_rgba; "
                                   "wait for the job in flight before submitting the next frame range");
    int rc;
    if (!dev->copy_stream) CU_TRY(cudaStreamCreateWithFlags(&dev->copy_stream, cudaStreamNonBlocking));
    if (!dev->up_stream) CU_TRY(cudaStreamCreateWithFlags(&dev->up_stream, cudaStreamNonBlocking));
    if (!sl.ev_render) {
        CU_TRY(cudaEventCreateWithFlags(&sl.ev_up, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&sl.ev_render, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
    }
    // 1. H2D of the caller's records, as the reference flow uploads tBuffer / materialBuffer (RaytraceTest.cpp:222-246)
    if ((rc = ensure_buffer(dev, &dev->host_tris, tb)) || (rc = ensure_buffer(dev, &dev->host_mats, mb)) ||
        (rc = ensure_buffer(dev, &sl.frame, fb)) || (sb && (rc = ensure_buffer(dev, &sl.stats, sb))) ||
        (rgb8 && (rc = ensure_buffer(dev, &sl.rgb8, (cb + 15) & ~size_t(15)))))
        return rc;
    // 2. resident scene (BVH + relaid records) is rebuilt only when the records changed
    uint64_t h = content_hash(tris, tb, 1469598103934665603ull);
    h = content_hash(mats, mb, h);
    const bool scene_changed = !dev->host_scene || dev->host_scene_hash != h;
    const void* src_t = tris;
    const void* src_m = mats;
    if (!is_pinned(tris) || !is_pinned(mats)) {  // pageable records go through pinned staging
        if (dev->pinned_bytes < tb + mb) {
            CU_TRY(cudaStreamSynchronize(dev->up_stream));
            if (dev->pinned) cudaFreeHost(dev->pinned);
            dev->pinned = nullptr; dev->pinned_bytes = 0;
            CU_TRY(cudaMallocHost(&dev->pinned, tb + mb));
            dev->pinned_bytes = tb + mb;
        } else {
            CU_TRY(cudaStreamSynchronize(dev->up_stream));  // the previous upload must have left the staging area
        }
        std::memcpy(dev->pinned, tris, tb);
        std::memcpy(static_cast<char*>(dev->pinned) + tb, mats, mb);
        src_t = dev->pinned;
        src_m = static_cast<char*>(dev->pinned) + tb;
    }
    // The device copies of the records are the caller-visible upload (and what a device-side rebuild would read); the
    // render itself reads the resident scene, so the copies run on their own stream and only the job's completion
    // event waits for them.
    CU_TRY(cudaMemcpyAsync(dev->host_tris->d_ptr, src_t, tb, cudaMemcpyHostToDevice, dev->up_stream));
    CU_TRY(cudaMemcpyAsync(dev->host_mats->d_ptr, src_m, mb, cudaMemcpyHostToDevice, dev->up_stream));
    dev->host_tris->version++; dev->host_mats->version++;
    CU_TRY(cudaEventRecord(sl.ev_up, dev->up_stream));
    if (scene_changed) {
        if (dev->host_scene) ptb_scene_destroy(dev->host_scene);
        dev->host_scene = nullptr;
        if ((rc = ptb_scene_create(dev, tris, n_tris, mats, n_mats, nullptr, &dev->host_scene))) return rc;
        dev->host_scene_hash = h;
    }
    // 3. output staging
    sl.direct_frame = is_pinned(out_rgba);
    sl.direct_stats = sb ? is_pinned(out_stats) : true;
    const size_t need_pin = (sl.direct_frame ? 0 : cb) + (sl.direct_stats ? 0 : sb);
    if (need_pin && sl.pin_bytes < cb + sb) {
        if (sl.pin) cudaFreeHost(sl.pin);
        sl.pin = nullptr; sl.pin_bytes = 0;
        CU_TRY(cudaMallocHost(&sl.pin, cb + sb));
        sl.pin_bytes = cb + sb;
    }
    // the slot's device frame may still be read by an older copy
    CU_TRY(cudaStreamWaitEvent(dev->stream, sl.ev_done, 0));
    if (params->accum == PTB_ACCUM_REFERENCE && params->first_frame > 0)  // in/out state of the gamma-space mean
        if ((rc = ptb_buffer_write(sl.frame, out_rgba, fb, 0))) return rc;
    // 4. render on the main stream
    if ((rc = render_impl(dev, dev->host_scene, params, static_cast<float4*>(sl.frame->d_ptr), sl.frame->bytes,
                          sb ? static_cast<ptb_pixel_stats*>(sl.stats->d_ptr) : nullptr, sb ? sl.stats->bytes : 0, nullptr)))
        return rc;
    if (rgb8) {  // the reference's output transform (RaytraceTest.cpp:78-83,:283) on the device: 3 bytes per pixel travel
        ptd::k_to_rgb8<<<((n_local + 3) / 4 + 255) / 256, 256, 0, dev->stream>>>(static_cast<const float4*>(sl.frame->d_ptr), n_local,
                                                                                static_cast<uint8_t*>(sl.rgb8->d_ptr));
        CU_TRY(cudaGetLastError());
        dev->kernel_launches += 1;
    }
    CU_TRY(cudaEventRecord(sl.ev_render, dev->stream));
    // 5. D2H on the copy stream
    CU_TRY(cudaStreamWaitEvent(dev->copy_stream, sl.ev_render, 0));
    char* pin = static_cast<char*>(sl.pin);
    CU_TRY(cudaMemcpyAsync(sl.direct_frame ? (void*)out_rgba : (void*)pin, rgb8 ? sl.rgb8->d_ptr : sl.frame->d_ptr, cb, cudaMemcpyDeviceToHost, dev->copy_stream));
    if (sb) CU_TRY(cudaMemcpyAsync(sl.direct_stats ? (void*)out_stats : (void*)(pin + cb), sl.stats->d_ptr, sb, cudaMemcpyDeviceToHost, dev->copy_stream));
    CU_TRY(cudaStreamWaitEvent(dev->copy_stream, sl.ev_up, 0));
    CU_TRY(cudaEventRecord(sl.ev_done, dev->copy_stream));
    sl.busy = true; sl.serial = dev->jobs_submitted; sl.out = out_rgba; sl.out_stats = out_stats; sl.fb = cb; sl.sb = sb;
    ptb_job* job = new ptb_job{dev, si, dev->jobs_submitted};
    dev->jobs_submitted++;
    *job_out = job;
    return PTB_OK;
}

extern "C" int ptb_render_host(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats,
                               int n_mats, const ptb_render_params* params, float* out_rgba,
                               ptb_pixel_stats* out_stats, ptb_counters* counters) {
    if (!dev) return fail(PTB_E_INVALID, "ptb_render_host: null argument");
    for (auto& sl : dev->slots)
        if (sl.busy) return fail(PTB_E_INVALID, "ptb_render_host: asynchronous jobs are still in flight");
    ptb_job* job = nullptr;
    int rc = ptb_render_host_async(dev, tris, n_tris, mats, n_mats, params, out_rgba, out_stats, &job);
    if (rc) return rc;
    rc = ptb_job_wait(job);
    if (rc) return rc;
    if (counters) {
        unsigned long long hc[ptd::CTR_COUNT];
        CU_TRY(cudaMemcpyAsync(hc, dev->counters, sizeof hc, cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        std::memset(counters, 0, sizeof *counters);
        counters->rays_closest = hc[ptd::CTR_CLOSEST]; counters->rays_any = hc[ptd::CTR_ANY];
        counters->nodes = hc[ptd::CTR_NODES]; counters->tri_tests = hc[ptd::CTR_TESTS];
        counters->samples = (uint64_t)ptb_render_local_pixels(params) * (uint64_t)params->n_frames;
    }
    return PTB_OK;
}

// ---- several GPUs in one process (BUILD-DEFINED; the reference is single-device: Adl/CL/AdlCL.cpp:154 picks ONE) ---------
// A device can be given HELPERS: other devices of the box that render part of its work.  Pixels are independent and a
// sample depends on (scene, W, H, pixel, frame) only (GenerateColors.cl:305-308), so the work is dealt without changing a
// bit of the result: ptb_render_multi shards the image (64-pixel blocks round-robin) and every device's resolve kernel stores
// its pixels straight into the ONE image on the main device over NVLink peer memory; ptb_launch1d deals the frames of its
// frame-ahead batch.  One host thread: work is enqueued asynchronously on each device's own stream and ordered with events.

static int ensure_event(ptb_device* d) {
    if (d->ev_multi) return PTB_OK;
    if (set_device(d)) return PTB_E_CUDA;
    CU_TRY(cudaEventCreateWithFlags(&d->ev_multi, cudaEventDisableTiming));
    return PTB_OK;
}

extern "C" int ptb_device_add_helper(ptb_device* dev, ptb_device* helper) {
    if (!dev || !helper || dev == helper) return fail(PTB_E_INVALID, "ptb_device_add_helper: bad arguments");
    if (helper->helper_of || !helper->helpers.empty() || dev->helper_of) return fail(PTB_E_INVALID, "ptb_device_add_helper: a helper serves one device and has no helpers of its own");
    if (int(dev->helpers.size()) >= PTB_MAX_PEERS) return fail(PTB_E_INVALID, "ptb_device_add_helper: at most %d helpers", PTB_MAX_PEERS);
    if (helper->index != dev->index) {
        int can = 0;
        CU_TRY(cudaDeviceCanAccessPeer(&can, helper->index, dev->index));
        if (!can) return fail(PTB_E_CUDA, "ptb_device_add_helper: device %d cannot access the memory of device %d", helper->index, dev->index);
        if (set_device(helper)) return PTB_E_CUDA;
        cudaError_t e = cudaDeviceEnablePeerAccess(dev->index, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(PTB_E_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
        cudaGetLastError();
    }
    if (int rc = ensure_event(dev)) return rc;
    if (int rc = ensure_event(helper)) return rc;
    dev->helpers.push_back(helper);
    helper->helper_of = dev;
    return PTB_OK;
}

extern "C" int ptb_device_helper_count(ptb_device* dev) {
    int n = 0;
    if (dev) for (ptb_device* h : dev->helpers) n += h != nullptr;
    return n;
}

extern "C" int ptb_render_multi(ptb_device* dev, const ptb_triangle* tris, int n_tris, const ptb_material* mats, int n_mats,
                                const ptb_render_params* params, float* out_rgba, ptb_counters* counters) {
    if (!dev || !tris || !mats || !out_rgba) return fail(PTB_E_INVALID, "ptb_render_multi: null argument");
    if (int rc = validate(params)) return rc;
    if (params->shard_count > 1) return fail(PTB_E_INVALID, "ptb_render_multi: the call shards the image itself (shard_count must be <= 1)");
    const bool rgb8 = params->output == PTB_OUTPUT_RGB8;
    if (rgb8 && params->accum == PTB_ACCUM_REFERENCE && params->first_frame > 0)
        return fail(PTB_E_INVALID, "ptb_render_multi: RGB8 output cannot carry the gamma-space state of accum=REFERENCE across calls (first_frame > 0)");
    std::vector<ptb_device*> devs{dev};
    for (ptb_device* h : dev->helpers) if (h) devs.push_back(h);
    const int n = int(devs.size());
    const size_t npix = size_t(params->width) * size_t(params->height);
    if (npix < size_t(n) * 64) devs.resize(1);  // fewer 64-pixel blocks than devices: one device renders it all
    const int nd = int(devs.size());
    // resident copies of the scene: rebuilt only when the records changed; the host-built tree is shared
    const size_t tb = size_t(n_tris) * sizeof(ptb_triangle), mb = size_t(n_mats) * sizeof(ptb_material);
    uint64_t h = content_hash(tris, tb, 1469598103934665603ull);
    h = content_hash(mats, mb, h);
    const ptb_scene* fresh = nullptr;
    for (ptb_device* d : devs)
        if (d->host_scene && d->host_scene_hash == h) { fresh = d->host_scene; break; }
    for (ptb_device* d : devs) {
        if (d->host_scene && d->host_scene_hash == h) continue;
        if (d->host_scene) ptb_scene_destroy(d->host_scene);
        d->host_scene = nullptr;
        if (int rc = scene_create_impl(d, tris, n_tris, mats, n_mats, nullptr, fresh, &d->host_scene)) return rc;
        d->host_scene_hash = h;
        if (!fresh) fresh = d->host_scene;
    }
    int rc;
    if ((rc = ensure_buffer(dev, &dev->multi_frame, npix * 16)) || (rgb8 && (rc = ensure_buffer(dev, &dev->multi_rgb8, (npix * 3 + 15) & ~size_t(15))))) return rc;
    if ((rc = ensure_event(dev))) return rc;
    if (set_device(dev)) return PTB_E_CUDA;
    if (params->accum == PTB_ACCUM_REFERENCE && params->first_frame > 0) {  // in/out state of the gamma-space running mean
        if ((rc = ptb_buffer_write(dev->multi_frame, out_rgba, npix * 16, 0))) return rc;
        CU_TRY(cudaStreamSynchronize(dev->stream));
    }
    CU_TRY(cudaEventRecord(dev->ev_multi, dev->stream));
    float4* image = static_cast<float4*>(dev->multi_frame->d_ptr);
    for (int j = 0; j < nd; ++j) {
        ptb_device* d = devs[j];
        ptb_render_params pj = *params;
        pj.shard_index = j; pj.shard_count = nd; pj.shard_block = 64;
        if (d != dev) {
            if ((rc = ensure_event(d))) return rc;
            if (set_device(d)) return PTB_E_CUDA;
            CU_TRY(cudaStreamWaitEvent(d->stream, dev->ev_multi, 0));  // the image (and its state) is ready on the main device
        }
        if ((rc = render_impl(d, d->host_scene, &pj, image, npix * 16, nullptr, 0, nullptr, nullptr, PHASE_BOTH, nullptr, 0))) return rc;
        if (d != dev) CU_TRY(cudaEventRecord(d->ev_multi, d->stream));
    }
    if (set_device(dev)) return PTB_E_CUDA;
    for (int j = 1; j < nd; ++j) CU_TRY(cudaStreamWaitEvent(dev->stream, devs[j]->ev_multi, 0));
    const size_t cb = rgb8 ? npix * 3 : npix * 16;
    if (rgb8) {
        ptd::k_to_rgb8<<<unsigned(((npix + 3) / 4 + 255) / 256), 256, 0, dev->stream>>>(image, int(npix), static_cast<uint8_t*>(dev->multi_rgb8->d_ptr));
        CU_TRY(cudaGetLastError());
        dev->kernel_launches += 1;
    }
    const bool direct = is_pinned(out_rgba);
    if (!direct && dev->multi_pin_bytes < cb) {
        if (dev->multi_pin) cudaFreeHost(dev->multi_pin);
        dev->multi_pin = nullptr; dev->multi_pin_bytes = 0;
        CU_TRY(cudaMallocHost(&dev->multi_pin, cb));
        dev->multi_pin_bytes = cb;
    }
    CU_TRY(cudaMemcpyAsync(direct ? (void*)out_rgba : dev->multi_pin, rgb8 ? dev->multi_rgb8->d_ptr : (void*)image, cb, cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaStreamSynchronize(dev->stream));
    if (!direct) std::memcpy(out_rgba, dev->multi_pin, cb);
    if (counters) {
        std::memset(counters, 0, sizeof *counters);
        for (ptb_device* d : devs) {
            unsigned long long hc[ptd::CTR_COUNT];
            if (set_device(d)) return PTB_E_CUDA;
            CU_TRY(cudaMemcpyAsync(hc, d->counters, sizeof hc, cudaMemcpyDeviceToHost, d->stream));
            CU_TRY(cudaStreamSynchronize(d->stream));
            counters->rays_closest += hc[ptd::CTR_CLOSEST]; counters->rays_any += hc[ptd::CTR_ANY];
            counters->nodes += hc[ptd::CTR_NODES]; counters->tri_tests += hc[ptd::CTR_TESTS];
        }
        counters->samples = (uint64_t)npix * (uint64_t)params->n_frames;
    }
    return PTB_OK;
}

// ---- kernel table + launcher (drop-in for Device::getKernel / Launcher) -------------------------------------

static std::string base_name(const char* path) {
    std::string s = path ? path : "";
    size_t k = s.find_last_of("/\\");
    if (k != std::string::npos) s = s.substr(k + 1);
    if (s.size() > 3 && s.compare(s.size() - 3, 3, ".cl") == 0) s.resize(s.size() - 3);
    return s;
}

extern "C" int ptb_kernel_get(ptb_device* dev, const char* file_name, const char* func_name, ptb_kernel** out) {
    if (!dev || !func_name || !out) return fail(PTB_E_INVALID, "ptb_kernel_get: null argument");
    *out = nullptr;
    const std::string file = base_name(file_name);
    if (std::strcmp(func_name, "GenerateColors") != 0 || (!file.empty() && file != "GenerateColors"))
        return fail(PTB_E_NOTFOUND, "ptb_kernel_get: no kernel %s in %s (known: GenerateColors)", func_name, file.c_str());
    const std::string key = file + "::" + func_name;
    auto it = dev->kernels.find(key);
    if (it == dev->kernels.end()) {
        ptb_kernel* k = new ptb_kernel();
        k->name = func_name;
        it = dev->kernels.emplace(key, k).first;
    }
    *out = it->second;
    return PTB_OK;
}

extern "C" int ptb_kernel_set_int(ptb_kernel* k, const char* name, int value) {
    if (!k || !name) return fail(PTB_E_INVALID, "ptb_kernel_set_int: null argument");
    if (!std::strcmp(name, "NUM_TRIANGLES")) { if (value < 1) return fail(PTB_E_INVALID, "NUM_TRIANGLES must be >= 1"); k->num_triangles = value; k->key_t = nullptr; }
    else if (!std::strcmp(name, "BOUNCES")) { if (value < 1) return fail(PTB_E_INVALID, "BOUNCES must be >= 1"); k->bounces = value; }
    else if (!std::strcmp(name, "ACCEL")) k->accel = value;
    else if (!std::strcmp(name, "INTEGRATOR")) k->integrator = value;
    else if (!std::strcmp(name, "FRAME_AHEAD")) { k->frame_ahead = value != 0; k->ahead_count = 0; }
    else return fail(PTB_E_NOTFOUND, "ptb_kernel_set_int: unknown option %s", name);
    return PTB_OK;
}

extern "C" int ptb_launch1d(ptb_device* dev, ptb_kernel* k, ptb_buffer* const* bufs, int n_bufs, const void* consts,
                            size_t const_bytes, int n_threads, int local_size) {
    (void)local_size;  // ADL_DEFAULT_LOCAL_SIZE_1D 64 (Adl/AdlKernel.h:71); the CUDA launch shape is ours
    if (!dev || !k || !bufs || !consts) return fail(PTB_E_INVALID, "ptb_launch1d: null argument");
    if (n_bufs != 3 || const_bytes != sizeof(ptb_int4))
        return fail(PTB_E_INVALID, "ptb_launch1d: GenerateColors takes 3 buffers + one int4 (got %d, %zu B)", n_bufs, const_bytes);
    ptb_buffer* tb = bufs[0]; ptb_buffer* mb = bufs[1]; ptb_buffer* fb = bufs[2];
    if (!tb || !mb || !fb) return fail(PTB_E_INVALID, "ptb_launch1d: null buffer");
    ptb_int4 res;
    std::memcpy(&res, consts, sizeof res);
    if (res.x <= 0 || res.y <= 0 || res.z < 0) return fail(PTB_E_INVALID, "ptb_launch1d: bad cRes {%d,%d,%d}", res.x, res.y, res.z);
    if ((long long)res.x * res.y != n_threads)
        return fail(PTB_E_INVALID, "ptb_launch1d: n_threads %d != W*H %lld", n_threads, (long long)res.x * res.y);
    const int nt = k->num_triangles;
    if (size_t(nt) * sizeof(ptb_triangle) > tb->bytes) return fail(PTB_E_INVALID, "ptb_launch1d: tBuffer holds fewer than NUM_TRIANGLES=%d records", nt);
    if (set_device(dev)) return PTB_E_CUDA;
    // resident scene for the bound buffers; rebuilt when their contents changed
    const bool tracked = tb->owned && mb->owned;
    bool scene_rebuilt = false;
    if (!k->scene || !tracked || k->key_t != tb || k->key_m != mb || k->ver_t != tb->version || k->ver_m != mb->version) {
        std::vector<ptb_triangle> ht(nt);
        CU_TRY(cudaMemcpyAsync(ht.data(), tb->d_ptr, size_t(nt) * sizeof(ptb_triangle), cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        int max_id = 0;
        for (const auto& t : ht) if (t.id > max_id) max_id = t.id;
        const int nm = max_id + 1;
        if (max_id < 0 || size_t(nm) * sizeof(ptb_material) > mb->bytes) return fail(PTB_E_INVALID, "ptb_launch1d: matBuffer too small for triangle ids");
        std::vector<ptb_material> hm(nm);
        CU_TRY(cudaMemcpyAsync(hm.data(), mb->d_ptr, size_t(nm) * sizeof(ptb_material), cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        uint64_t h = content_hash(ht.data(), ht.size() * sizeof(ptb_triangle), 1469598103934665603ull);
        h = content_hash(hm.data(), hm.size() * sizeof(ptb_material), h);
        if (!k->scene || h != k->hash) {
            if (k->scene) ptb_scene_destroy(k->scene);
            k->scene = nullptr;
            for (ptb_scene*& hs : k->helper_scenes) { if (hs) ptb_scene_destroy(hs); hs = nullptr; }
            if (int rc = ptb_scene_create(dev, ht.data(), nt, hm.data(), nm, nullptr, &k->scene)) return rc;
            k->hash = h;
            scene_rebuilt = true;
        }
        k->key_t = tb; k->key_m = mb; k->ver_t = tb->version; k->ver_m = mb->version;
    }
    ptb_render_params p;
    ptb_render_params_default(&p);
    p.width = res.x; p.height = res.y;
    p.first_frame = res.z; p.n_frames = 1;  // RaytraceTest.cpp:252-253: one launch = one frame index
    p.mode = PTB_MODE_PATH; p.accum = PTB_ACCUM_REFERENCE;
    p.max_depth = k->bounces; p.accel = k->accel; p.integrator = k->integrator;
    float4* d_fb = static_cast<float4*>(fb->d_ptr);

    // Frame-ahead batching.  One 512x512 frame is under one wave of threads, so a launch-per-frame loop runs at the
    // latency of its longest path.  A sample depends only on (scene, W, H, pixel, frame) -- not on the framebuffer --
    // so once the caller is seen stepping through consecutive frame indices (the progressive loop,
    // RaytraceTest.cpp:248-262), the samples of the next frames are traced together in one full-GPU launch and each
    // later launch only folds its own frame into the caller's buffer.  Results are bit-identical to the
    // frame-by-frame path (same per-sample arithmetic, same ordered running mean); anything that could change a
    // sample (buffers rewritten, NUM_TRIANGLES/BOUNCES/ACCEL/INTEGRATOR, image size) discards the batch.
    const int z = res.z;
    const int cfg[3] = {k->bounces, k->accel, k->integrator};
    const bool same_cfg = k->ahead_w == res.x && k->ahead_h == res.y && !std::memcmp(cfg, k->ahead_cfg, sizeof cfg);
    if (!same_cfg || scene_rebuilt) k->ahead_count = 0;
    k->streak = (z == k->last_frame + 1 && same_cfg && !scene_rebuilt) ? k->streak + 1 : 0;
    k->last_frame = z;
    k->ahead_w = res.x; k->ahead_h = res.y; std::memcpy(k->ahead_cfg, cfg, sizeof cfg);
    const bool speculate = k->frame_ahead != 0;
    if (speculate && !(k->ahead_count > 0 && z >= k->ahead_first && z < k->ahead_first + k->ahead_count) && k->streak >= 1) {
        // sample slots in flight: 16 Mi per device that shares the batch (this device + its helpers), so that a 2048x2048 frame loop
        // still batches (round 2: with 4 Mi a 4 Mi-pixel frame was traced alone and eight GPUs gave nothing); tune[1] = log2 multiplier
        int n_dev = 1;
        for (ptb_device* hd : dev->helpers) n_dev += hd ? 1 : 0;
        const long long target = ((16ll << 20) * n_dev) << (dev->tune[1] > 0 && dev->tune[1] < 5 ? dev->tune[1] : 0);
        int want = (int)((target + n_threads - 1) / n_threads);
        const int ramp = k->streak >= 5 ? want : (1 << k->streak);  // 2, 4, 8, 16 ... so a short sequence wastes little
        if (want > ramp) want = ramp;
        if (want > 0x7fffffff - z) want = 0x7fffffff - z;
        k->ahead_count = 0;  // the old batch is gone whatever happens next
        if (want >= 2 && ensure(&k->ahead, &k->ahead_bytes, size_t(want) * size_t(n_threads) * 16) != PTB_OK) {
            cudaGetLastError();  // no memory for a batch: fall back to one frame per launch
            want = 0;
        }
        if (want >= 2) {
            // the frames of the batch are dealt over this device and its helpers (ptb_device_add_helper): each traces its
            // frames into its slice of the batch on THIS device (stores over NVLink peer memory); the resolves stay here
            std::vector<ptb_device*> devs{dev};
            std::vector<ptb_scene*> scs{k->scene};
            k->helper_scenes.resize(dev->helpers.size(), nullptr);
            for (size_t i = 0; i < dev->helpers.size() && int(devs.size()) < want; ++i) {
                ptb_device* hd = dev->helpers[i];
                if (!hd) continue;
                if (!k->helper_scenes[i] &&
                    scene_create_impl(hd, k->scene->host_tris.data(), k->scene->n_tris, k->scene->host_mats.data(), k->scene->n_mats, nullptr,
                                      k->scene, &k->helper_scenes[i]) != PTB_OK) {
                    k->helper_scenes[i] = nullptr;
                    continue;  // this helper cannot hold the scene: the others do the work
                }
                devs.push_back(hd); scs.push_back(k->helper_scenes[i]);
            }
            const int nd = int(devs.size());
            if (nd > 1) {
                if (set_device(dev)) return PTB_E_CUDA;
                CU_TRY(cudaEventRecord(dev->ev_multi, dev->stream));  // the previous batch has been consumed up to here
            }
            int off = 0;
            for (int j = 0; j < nd; ++j) {
                const int cnt = want / nd + (j < want % nd ? 1 : 0);
                ptb_render_params pb = p;
                pb.first_frame = z + off; pb.n_frames = cnt;
                ptb_device* d = devs[j];
                if (d != dev) {
                    if (set_device(d)) return PTB_E_CUDA;
                    CU_TRY(cudaStreamWaitEvent(d->stream, dev->ev_multi, 0));
                }
                int rc = render_impl(d, scs[j], &pb, nullptr, 0, nullptr, 0, nullptr, static_cast<float4*>(k->ahead) + size_t(off) * size_t(n_threads), PHASE_TRACE);
                if (rc == PTB_OK && d != dev && cudaEventRecord(d->ev_multi, d->stream) != cudaSuccess) rc = fail(PTB_E_CUDA, "ptb_launch1d: cudaEventRecord failed");
                if (rc) {
                    k->ahead_count = 0;
                    return rc;
                }
                off += cnt;
            }
            if (set_device(dev)) return PTB_E_CUDA;
            for (int j = 1; j < nd; ++j) CU_TRY(cudaStreamWaitEvent(dev->stream, devs[j]->ev_multi, 0));
            k->ahead_first = z; k->ahead_count = want;
        }
    }
    if (speculate && k->ahead_count > 0 && z >= k->ahead_first && z < k->ahead_first + k->ahead_count) {
        float4* smp = static_cast<float4*>(k->ahead) + size_t(z - k->ahead_first) * size_t(n_threads);
        return render_impl(dev, k->scene, &p, d_fb, fb->bytes, nullptr, 0, nullptr, smp, PHASE_RESOLVE);
    }
    return render_impl(dev, k->scene, &p, d_fb, fb->bytes, nullptr, 0, nullptr);
}

// ---- launch capture / replay (Launcher::serializeToFile / deserializeFromFile) ---------------------------------

extern "C" int ptb_launch_serialize(ptb_device* dev, const char* path, ptb_buffer* const* bufs, int n_bufs,
                                    const void* consts, size_t const_bytes, int n_threads, int local_size) {
    if (!dev || !path || !bufs || n_bufs < 0 || (!consts && const_bytes)) return fail(PTB_E_INVALID, "ptb_launch_serialize: bad arguments");
    if (const_bytes > 64) return fail(PTB_E_INVALID, "ptb_launch_serialize: constant block larger than MAX_ARG_SIZE (64)");
    if (set_device(dev)) return PTB_E_CUDA;
    FILE* f = std::fopen(path, "wb");
    if (!f) return fail(PTB_E_IO, "ptb_launch_serialize: cannot open %s", path);
    auto put_i = [&](int32_t v) { std::fwrite(&v, 4, 1, f); };
    put_i(n_bufs + (const_bytes ? 1 : 0));
    std::vector<char> host;
    for (int i = 0; i < n_bufs; ++i) {
        put_i(1);
        const size_t nb = bufs[i] ? bufs[i]->bytes : 0;
        if (nb > 0x7fffffffu) { std::fclose(f); return fail(PTB_E_INVALID, "ptb_launch_serialize: buffer %d exceeds the format's 31-bit size", i); }
        put_i((int32_t)nb);
        if (nb) {
            host.resize(nb);
            cudaError_t e = cudaMemcpyAsync(host.data(), bufs[i]->d_ptr, nb, cudaMemcpyDeviceToHost, dev->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(dev->stream);
            if (e != cudaSuccess) { std::fclose(f); return fail(PTB_E_CUDA, "ptb_launch_serialize: read-back failed: %s", cudaGetErrorString(e)); }
            std::fwrite(host.data(), 1, nb, f);
        }
    }
    if (const_bytes) {
        put_i(0);
        put_i((int32_t)const_bytes);
        std::fwrite(consts, 1, const_bytes, f);
    }
    const int32_t info[7] = {n_threads, 1, 1, local_size, 1, 1, 1};  // Launcher::ExecInfo (Adl/AdlKernel.h:139-160)
    std::fwrite(info, 4, 7, f);
    const bool ok = std::ferror(f) == 0;
    std::fclose(f);
    return ok ? PTB_OK : fail(PTB_E_IO, "ptb_launch_serialize: write error on %s", path);
}

extern "C" int ptb_launch_deserialize(ptb_device* dev, const char* path, ptb_buffer** bufs_out, int buf_cap, int* n_bufs,
                                      void* consts_out, size_t* const_bytes, int* n_threads, int* local_size) {
    if (!dev || !path || !bufs_out || !n_bufs || !consts_out || !const_bytes || !n_threads || !local_size)
        return fail(PTB_E_INVALID, "ptb_launch_deserialize: null argument");
    *n_bufs = 0; *const_bytes = 0;
    FILE* f = std::fopen(path, "rb");
    if (!f) return fail(PTB_E_IO, "ptb_launch_deserialize: cannot open %s", path);
    auto bail = [&](int code, const char* what) {
        std::fclose(f);
        for (int i = 0; i < *n_bufs; ++i) ptb_buffer_destroy(bufs_out[i]);
        *n_bufs = 0;
        return fail(code, "ptb_launch_deserialize: %s in %s", what, path);
    };
    int32_t n_args = 0;
    if (std::fread(&n_args, 4, 1, f) != 1 || n_args < 0 || n_args > 64) return bail(PTB_E_IO, "bad argument count");
    std::vector<char> data;
    for (int i = 0; i < n_args; ++i) {
        int32_t is_buf = 0, nb = 0;
        if (std::fread(&is_buf, 4, 1, f) != 1 || std::fread(&nb, 4, 1, f) != 1 || nb < 0) return bail(PTB_E_IO, "truncated argument header");
        data.resize((size_t)nb);
        if (nb && std::fread(data.data(), 1, (size_t)nb, f) != (size_t)nb) return bail(PTB_E_IO, "truncated argument data");
        if (is_buf) {
            if (*n_bufs >= buf_cap) return bail(PTB_E_INVALID, "more buffer arguments than buf_cap");
            ptb_buffer* b = nullptr;
            if (int rc = ptb_buffer_create(dev, (size_t)nb, &b)) { std::fclose(f); return rc; }
            bufs_out[(*n_bufs)++] = b;
            if (nb) {
                if (int rc = ptb_buffer_write(b, data.data(), (size_t)nb, 0)) { std::fclose(f); return rc; }
                cudaStreamSynchronize(dev->stream);  // `data` is reused for the next argument
            }
        } else {
            if (nb > 64) return bail(PTB_E_IO, "constant block larger than 64 bytes");
            std::memcpy(consts_out, data.data(), (size_t)nb);
            *const_bytes = (size_t)nb;
        }
    }
    int32_t info[7];
    if (std::fread(info, 4, 7, f) != 7) return bail(PTB_E_IO, "truncated ExecInfo");
    std::fclose(f);
    *n_threads = info[0];
    *local_size = info[3];
    return PTB_OK;
}

// ---- measurement hooks -----------------------------------------------------------------------------------------

extern "C" int ptb_device_set_tuning(ptb_device* dev, int index, int value) {
    if (!dev || index < 0 || index >= 16) return fail(PTB_E_INVALID, "ptb_device_set_tuning: bad arguments");
    dev->tune[index] = value;
    return PTB_OK;
}

extern "C" int ptb_device_counters(ptb_device* dev, int cumulative, ptb_counters* out) {
    if (!dev) return fail(PTB_E_INVALID, "ptb_device_counters: null device");
    if (set_device(dev)) return PTB_E_CUDA;
    if (out) {
        unsigned long long h[ptd::CTR_COUNT];
        CU_TRY(cudaMemcpyAsync(h, dev->counters, sizeof h, cudaMemcpyDeviceToHost, dev->stream));
        CU_TRY(cudaMemsetAsync(dev->counters, 0, sizeof(unsigned long long) * ptd::CTR_COUNT, dev->stream));
        CU_TRY(cudaStreamSynchronize(dev->stream));
        std::memset(out, 0, sizeof *out);
        out->rays_closest = h[ptd::CTR_CLOSEST]; out->rays_any = h[ptd::CTR_ANY];
        out->nodes = h[ptd::CTR_NODES]; out->tri_tests = h[ptd::CTR_TESTS];
        out->samples = dev->cumulative_samples;
        dev->cumulative_samples = 0;
    }
    if (cumulative >= 0) {
        if ((cumulative != 0) != dev->cumulative_counters) {
            CU_TRY(cudaMemsetAsync(dev->counters, 0, sizeof(unsigned long long) * ptd::CTR_COUNT, dev->stream));
            dev->cumulative_samples = 0;
        }
        dev->cumulative_counters = cumulative != 0;
    }
    return PTB_OK;
}

extern "C" int ptb_buffer_to_rgb8(ptb_buffer* frame, int n_pixels, ptb_buffer* rgb) {
    if (!frame || !rgb || n_pixels < 0) return fail(PTB_E_INVALID, "ptb_buffer_to_rgb8: bad arguments");
    if (size_t(n_pixels) * 16 > frame->bytes || size_t(n_pixels) * 3 > rgb->bytes) return fail(PTB_E_INVALID, "ptb_buffer_to_rgb8: buffer too small");
    if ((reinterpret_cast<uintptr_t>(rgb->d_ptr) & 15u) != 0) return fail(PTB_E_INVALID, "ptb_buffer_to_rgb8: rgb must be 16-byte aligned");
    if (n_pixels == 0) return PTB_OK;
    ptb_device* dev = frame->dev;
    if (set_device(dev)) return PTB_E_CUDA;
    ptd::k_to_rgb8<<<((n_pixels + 3) / 4 + 255) / 256, 256, 0, dev->stream>>>(static_cast<const float4*>(frame->d_ptr), n_pixels,
                                                                              static_cast<uint8_t*>(rgb->d_ptr));
    CU_TRY(cudaGetLastError());
    dev->kernel_launches += 1;
    return PTB_OK;
}

extern "C" int ptb_device_profile(ptb_device* dev, int enable) {
    if (!dev) return fail(PTB_E_INVALID, "ptb_device_profile: null device");
    dev->profiling = enable != 0;
    return PTB_OK;
}

extern "C" int ptb_device_profile_read(ptb_device* dev, float* integrator_ms, float* resolve_ms, int* integrator_launches,
                                       uint64_t* kernel_launches) {
    if (!dev) return fail(PTB_E_INVALID, "ptb_device_profile_read: null device");
    if (set_device(dev)) return PTB_E_CUDA;
    CU_TRY(cudaStreamSynchronize(dev->stream));
    float ti = 0.f, tr = 0.f;
    for (size_t k = 0; k + 2 < dev->ev_used + 0 && k + 2 < dev->ev_pool.size() + 0; k += 3) {
        float a = 0.f, b = 0.f;
        CU_TRY(cudaEventElapsedTime(&a, dev->ev_pool[k], dev->ev_pool[k + 1]));
        CU_TRY(cudaEventElapsedTime(&b, dev->ev_pool[k + 1], dev->ev_pool[k + 2]));
        ti += a; tr += b;
    }
    if (integrator_ms) *integrator_ms = ti;
    if (resolve_ms) *resolve_ms = tr;
    if (integrator_launches) *integrator_launches = dev->integrator_launch_batches;
    if (kernel_launches) *kernel_launches = dev->kernel_launches;
    dev->ev_used = 0;
    dev->integrator_launch_batches = 0;
    dev->kernel_launches = 0;
    return PTB_OK;
}

// ---- unit access for parity tests -----------------------------------------------------------------------------

template <class T>
struct DevArr {
    T* p = nullptr;
    ~DevArr() { if (p) cudaFree(p); }
    int alloc(size_t n) { CU_TRY(cudaMalloc((void**)&p, (n ? n : 1) * sizeof(T))); return PTB_OK; }
};

extern "C" int ptb_trace(ptb_device* dev, ptb_scene* scene, int accel, int any_hit, int n_rays, const float* o,
                         const float* d, const float* tmax, int32_t* out_tri, float* out_t, float* out_u, float* out_v,
                         uint32_t* out_visits, uint32_t* out_tests) {
    if (!dev || !scene || !o || !d || !tmax || !out_tri || n_rays < 0) return fail(PTB_E_INVALID, "ptb_trace: bad arguments");
    if (n_rays == 0) return PTB_OK;
    if (set_device(dev)) return PTB_E_CUDA;
    const size_t n = size_t(n_rays);
    DevArr<float> d_o, d_d, d_tm, d_t, d_u, d_v;
    DevArr<int> d_tri;
    DevArr<uint32_t> d_vis, d_tst;
    int rc;
    if ((rc = d_o.alloc(3 * n)) || (rc = d_d.alloc(3 * n)) || (rc = d_tm.alloc(n)) || (rc = d_t.alloc(n)) || (rc = d_u.alloc(n)) ||
        (rc = d_v.alloc(n)) || (rc = d_tri.alloc(n)) || (rc = d_vis.alloc(n)) || (rc = d_tst.alloc(n)))
        return rc;
    cudaStream_t st = dev->stream;
    CU_TRY(cudaMemcpyAsync(d_o.p, o, 12 * n, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(d_d.p, d, 12 * n, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(d_tm.p, tmax, 4 * n, cudaMemcpyHostToDevice, st));
    ptd::SceneDev sc = scene_dev(scene, scene->cls);
    ptd::TraceArgs a{n_rays, d_o.p, d_d.p, d_tm.p, d_tri.p, d_t.p, d_u.p, d_v.p, d_vis.p, d_tst.p};
    const bool bvh = accel == PTB_ACCEL_BVH, any = any_hit != 0;
    const int small = (!bvh && scene->cls == ptd::PTD_FLAT) ? ptd::PTD_SMALL4 : scene->cls;
    const int block = 128;
    const unsigned grid = (unsigned)((n + block - 1) / block);
    const size_t smem = ptd::scene_smem_bytes(sc, bvh, small, block);
#define PTB_TRACE_CASE(B, A, S)                                                \
    if (bvh == B && any == A && small == S) {                                  \
        auto k = ptd::k_trace<B, A, S>;                                        \
        if ((rc = set_smem(k, smem, block))) return rc;                               \
        k<<<grid, block, smem, st>>>(sc, a);                                   \
    }
    PTB_TRACE_CASE(true, true, 2) PTB_TRACE_CASE(true, false, 2)
    PTB_TRACE_CASE(true, true, 1) PTB_TRACE_CASE(true, true, 0) PTB_TRACE_CASE(true, false, 1) PTB_TRACE_CASE(true, false, 0)
    PTB_TRACE_CASE(false, true, 1) PTB_TRACE_CASE(false, true, 0) PTB_TRACE_CASE(false, false, 1) PTB_TRACE_CASE(false, false, 0)
#undef PTB_TRACE_CASE
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(out_tri, d_tri.p, 4 * n, cudaMemcpyDeviceToHost, st));
    if (out_t) CU_TRY(cudaMemcpyAsync(out_t, d_t.p, 4 * n, cudaMemcpyDeviceToHost, st));
    if (out_u) CU_TRY(cudaMemcpyAsync(out_u, d_u.p, 4 * n, cudaMemcpyDeviceToHost, st));
    if (out_v) CU_TRY(cudaMemcpyAsync(out_v, d_v.p, 4 * n, cudaMemcpyDeviceToHost, st));
    if (out_visits) CU_TRY(cudaMemcpyAsync(out_visits, d_vis.p, 4 * n, cudaMemcpyDeviceToHost, st));
    if (out_tests) CU_TRY(cudaMemcpyAsync(out_tests, d_tst.p, 4 * n, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return PTB_OK;
}

extern "C" int ptb_test_sincos(ptb_device* dev, const float* x, int n, float* s, float* c) {
    if (!dev || !x || !s || !c || n < 0) return fail(PTB_E_INVALID, "ptb_test_sincos: bad arguments");
    if (n == 0) return PTB_OK;
    if (set_device(dev)) return PTB_E_CUDA;
    DevArr<float> dx, ds, dc;
    int rc;
    if ((rc = dx.alloc(n)) || (rc = ds.alloc(n)) || (rc = dc.alloc(n))) return rc;
    CU_TRY(cudaMemcpyAsync(dx.p, x, 4 * size_t(n), cudaMemcpyHostToDevice, dev->stream));
    ptd::k_test_sincos<<<(n + 255) / 256, 256, 0, dev->stream>>>(dx.p, n, ds.p, dc.p);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(s, ds.p, 4 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaMemcpyAsync(c, dc.p, 4 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaStreamSynchronize(dev->stream));
    return PTB_OK;
}

extern "C" int ptb_test_pow(ptb_device* dev, const float* x, int n, float y, float* out) {
    if (!dev || !x || !out || n < 0) return fail(PTB_E_INVALID, "ptb_test_pow: bad arguments");
    if (n == 0) return PTB_OK;
    if (set_device(dev)) return PTB_E_CUDA;
    DevArr<float> dx, dout;
    int rc;
    if ((rc = dx.alloc(n)) || (rc = dout.alloc(n))) return rc;
    CU_TRY(cudaMemcpyAsync(dx.p, x, 4 * size_t(n), cudaMemcpyHostToDevice, dev->stream));
    ptd::k_test_pow<<<(n + 255) / 256, 256, 0, dev->stream>>>(dx.p, n, y, dout.p);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(out, dout.p, 4 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaStreamSynchronize(dev->stream));
    return PTB_OK;
}

extern "C" int ptb_test_ieee(ptb_device* dev, const float* x, int n, float* out6n) {
    if (!dev || !x || !out6n || n < 0) return fail(PTB_E_INVALID, "ptb_test_ieee: bad arguments");
    if (n == 0) return PTB_OK;
    if (set_device(dev)) return PTB_E_CUDA;
    DevArr<float> dx, dout;
    int rc;
    if ((rc = dx.alloc(n)) || (rc = dout.alloc(6 * size_t(n)))) return rc;
    CU_TRY(cudaMemcpyAsync(dx.p, x, 4 * size_t(n), cudaMemcpyHostToDevice, dev->stream));
    ptd::k_test_ieee<<<(n + 255) / 256, 256, 0, dev->stream>>>(dx.p, n, dout.p);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(out6n, dout.p, 24 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaStreamSynchronize(dev->stream));
    return PTB_OK;
}

extern "C" int ptb_test_rng(ptb_device* dev, uint32_t gid, uint32_t frame, int n, uint32_t* states, float* values) {
    if (!dev || !states || !values || n < 0) return fail(PTB_E_INVALID, "ptb_test_rng: bad arguments");
    if (n == 0) return PTB_OK;
    if (set_device(dev)) return PTB_E_CUDA;
    DevArr<uint32_t> ds;
    DevArr<float> dv;
    int rc;
    if ((rc = ds.alloc(n)) || (rc = dv.alloc(n))) return rc;
    ptd::k_test_rng<<<1, 32, 0, dev->stream>>>(gid, frame, n, ds.p, dv.p);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(states, ds.p, 4 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaMemcpyAsync(values, dv.p, 4 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaStreamSynchronize(dev->stream));
    return PTB_OK;
}

extern "C" int ptb_test_camera(ptb_device* dev, int width, int height, int frame, int n, const int32_t* gids, float* o,
                               float* d, uint32_t* seeds) {
    if (!dev || !gids || !o || !d || !seeds || n < 0) return fail(PTB_E_INVALID, "ptb_test_camera: bad arguments");
    if (n == 0) return PTB_OK;
    if (set_device(dev)) return PTB_E_CUDA;
    DevArr<int> dg;
    DevArr<float> d_o, d_d;
    DevArr<uint32_t> ds;
    int rc;
    if ((rc = dg.alloc(n)) || (rc = d_o.alloc(3 * size_t(n))) || (rc = d_d.alloc(3 * size_t(n))) || (rc = ds.alloc(n))) return rc;
    CU_TRY(cudaMemcpyAsync(dg.p, gids, 4 * size_t(n), cudaMemcpyHostToDevice, dev->stream));
    ptd::k_test_camera<<<(n + 127) / 128, 128, 0, dev->stream>>>(width, height, frame, n, dg.p, d_o.p, d_d.p, ds.p);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(o, d_o.p, 12 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaMemcpyAsync(d, d_d.p, 12 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaMemcpyAsync(seeds, ds.p, 4 * size_t(n), cudaMemcpyDeviceToHost, dev->stream));
    CU_TRY(cudaStreamSynchronize(dev->stream));
    return PTB_OK;
}
