// api.cu — the C ABI of include/rttnw_b200.h: contexts, scene upload, kernel launches.
// No entry point computes on the CPU; without a CUDA device they fail with RTX_ERR_CUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <thread>
#include <type_traits>
#include <new>
#include <string>
#include <vector>

#include "../../include/rttnw_b200.h"
#include "flatten.hpp"
#include "adaptive.cuh"
#include "aov.cuh"
#include "denoise.cuh"
#include "kernels.cuh"
#include "lbvh.cuh"
#include "sah_build.cuh"
#include "shade2.cuh"
#include "trace2.cuh"
#include "trace3.cuh"
#include "scene_api.hpp"

namespace {

thread_local std::string g_err = "";

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return RTX_ERR_CUDA;
}
#define CU(call)                                      \
    do {                                              \
        cudaError_t e__ = (call);                     \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// Device allocations of destroyed scenes, kept for the next rtx_scene_create on the same device: a
// caller that re-uploads its scene every frame then pays two memcpys instead of cudaMalloc /
// cudaMallocArray / cudaCreateTextureObject / cudaFree (the frees stall sporadically for 0.1-1 s).
struct ArenaSlot {
    void* p;
    size_t bytes;
};
struct ArraySlot {
    cudaArray_t arr;
    cudaTextureObject_t tex;
    int w, h;
};
struct DeviceCache {
    std::mutex m;
    std::vector<ArenaSlot> arenas;
    std::vector<ArraySlot> arrays;
};
constexpr int kMaxDevices = 64;
constexpr size_t kCacheKeep = 4;
DeviceCache g_cache[kMaxDevices];

}  // namespace

struct rtx_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    unsigned int* d_work_counter = nullptr;  // render_kernel's tile dispenser
    rtx::Counters* d_counters = nullptr;
    int node_burst = 4;
    int mode = 1;  // 1: wavefront (default), 0: megakernel (RTX_MODE=mega)
    // wavefront state, allocated at the first render
    void* d_pool = nullptr;
    int pool_slots = 0, pool_slots_wanted = 1 << 19;  // 512 Ki slots x 96 B = 48 MB, in two partitions. Measured on scene 9 (M samples/s), one
                                                      // stream: 512 Ki 485, 1 Mi 508, 2 Mi 516, 4 Mi 501; two streams: 256 Ki 511, 384 Ki 571,
                                                      // 512 Ki 596, 768 Ki 590, 1 Mi 582, 2 Mi 567; three / four streams at 512 Ki: 593 / 585
    unsigned long long* d_next_item = nullptr;
    unsigned int* d_active = nullptr;            // [2]
    unsigned long long* h_status = nullptr;      // pinned: [partition][parity] x {active, next_item}
    cudaEvent_t batch_done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // [partition][parity]
    int wf_batch = 8;
    int wf_wide = 0;     // RTX_BVH_WIDE=1: the trace kernel walks the 4-wide copy of the world BVH (measured slower: DESIGN.md §4)
    int wf_streams = 2;  // pool partitions driven concurrently on their own streams (RTX_WF_STREAMS, at most 4)
    // trace kernel form (RTX_TRACE). 1 (default): one slot per thread, while-while, local-memory stack (wf_trace_kernel).
    // The others were built in round 2 to test what ncu pointed at, measured on scene 9 against 604 M samples/s for
    // form 1 and kept as opt-in, parity-tested variants (DESIGN.md §4 has the numbers): 2 = world BVH + stacks in shared
    // memory, persistent warps with voted refill (trace2.cuh; 543-572 M); 3 = rays regrouped by kind of work through
    // shared memory every few steps (trace3.cuh; 238-342 M); 4 = form 1 with a shared-memory stack and 32-byte node
    // loads (trace2.cuh, "1c"; 596 M). Forms 2-4 need a world BVH no deeper than kShortStack and fall back to 1.
    int trace_form = 1;
    int trace_threads = 896;               // CTA size of the shared-memory form, one CTA per SM (RTX_TRACE_THREADS: 896, 640, 512, 448)
    int t_leaf = 8, t_refill = 16, t_burst = 8;  // its vote thresholds (RTX_T_LEAF / RTX_T_REFILL / RTX_T_BURST); 33 / 33 / huge = plain while-while
    // RTX_ORDER=1: the trace pass takes its rays in (direction octant, record they start on) order: order.cuh
    int order_form = 0;
    int order_groups = 512;                // record groups per octant (RTX_ORDER_GROUPS, a power of two)
    void* d_order = nullptr;
    size_t order_bytes = 0;
    int smem_optin = 0;                    // cudaDevAttrMaxSharedMemoryPerBlockOptin
    int prof_stride = 8;                   // RTX_PROF_STRIDE: every n-th iteration of partition 0 is bracketed when profiling is on
    bool perlin_smem = true;               // the shade kernel stages the Perlin table (noise.rs:5-29) in shared memory when the scene has exactly one
                                           // (RTX_PERLIN_SMEM=0 reads it through L1: measured 3.4 % / 1 % / 0.3 % slower on scenes 3 / 5 / 9)
    bool debug_batches = false;            // RTX_DEBUG_BATCHES=1: one stderr line per batch and partition
    int shade_form = 2;                    // RTX_SHADE: 2 = media after the surface search + early dispenser request (shade2.cuh), 1 = first form
    std::vector<cudaStream_t> aux_streams;
    std::vector<cudaEvent_t> join_events;
    cudaEvent_t fork_event = nullptr;
    unsigned long long launches = 0;  // kernels launched by this context (rtx_ctx_kernel_launches)
    int bvh_builder = 0;              // 0: host binned SAH (default), 1: device LBVH, 2: device PLOC, 3: device binned SAH
                                      // (rtx_ctx_set_bvh_builder, RTX_BVH=lbvh|ploc|sah_device)
    int ploc_radius = 16;             // neighbours searched on each side by the PLOC builder (RTX_PLOC_RADIUS, 1..32)
    int last_build_passes = 0;        // passes the last PLOC build took (RTX_DEBUG_BUILD=1 prints it)
    uint8_t* h_stage = nullptr;       // pinned staging buffer of rtx_scene_create (every H2D copy leaves from here)
    size_t stage_bytes = 0;
    void* d_denoise = nullptr;        // rtx_denoise's per-pixel scratch (56 B a pixel), grown on demand
    size_t denoise_bytes = 0;
    // optional per-kernel timing of the wavefront driver (rtx_ctx_set_profiling): CUDA events around every launch
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;  // grows on demand; [4 * iteration + {0,1,2,3}] = shade begin/end, trace begin/end
    double prof_shade_ms = 0, prof_trace_ms = 0;
    unsigned long long prof_iterations = 0;
    int w_node = 1, w_leaf = 1, w_shade = 1;  // render_kernel phase weights (RTX_W_NODE / RTX_W_LEAF / RTX_W_SHADE override)
    // rtx_ctx_set_async: rtx_render hands the wavefront driver's submit-and-poll loop to this context's own thread and
    // returns at once; every other entry point that uses the context first waits for that thread to run dry
    bool async = false;
    std::thread worker;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<std::function<int()>> jobs;
    int jobs_open = 0;  // queued + running
    bool stop = false;
    int async_rc = RTX_OK;  // first failure of a job, reported by the next call that joins
    std::string async_err;
};

struct rtx_scene {
    int device = 0;  // not the ctx: a scene may outlive the context that created it
    rtx::SceneView view{};
    rtx::CameraView camera{};
    void* d_arena = nullptr;
    size_t arena_bytes = 0, arena_capacity = 0;
    std::vector<ArraySlot> images;
    int32_t n_nodes = 0, n_records = 0, n_xforms = 0;
    int32_t world_first_node = 0, world_node_count = 0, world_depth = 0;  // the world BVH's node range (root first) and depth
    int32_t n_perlins = 0;
    // rtx_scene_set_environment: the map (env.texels == nullptr: none, the constant background) in its own allocation
    rtx::EnvArgs env{};
    size_t env_bytes = 0;
};

// Waits until the context's worker thread has nothing queued or running; returns (once) the failure of an asynchronous
// render, if there was one. Called at the top of every entry point that uses the context's stream or state.
static int join_async(rtx_ctx* c) {
    if (!c || !c->worker.joinable()) return RTX_OK;
    std::unique_lock<std::mutex> lock(c->mu);
    c->cv.wait(lock, [&] { return c->jobs_open == 0; });
    if (c->async_rc != RTX_OK) {
        int rc = c->async_rc;
        g_err = c->async_err;
        c->async_rc = RTX_OK;
        return rc;
    }
    return RTX_OK;
}
#define JOIN(c)                          \
    do {                                 \
        int rc__ = join_async(c);        \
        if (rc__ != RTX_OK) return rc__; \
    } while (0)

static void worker_main(rtx_ctx* c) {
    for (;;) {
        std::function<int()> job;
        {
            std::unique_lock<std::mutex> lock(c->mu);
            c->cv.wait(lock, [&] { return c->stop || !c->jobs.empty(); });
            if (c->jobs.empty()) return;  // stop requested and nothing left
            job = std::move(c->jobs.front());
            c->jobs.pop_front();
        }
        g_err.clear();
        int rc = job();
        {
            std::lock_guard<std::mutex> lock(c->mu);
            if (rc != RTX_OK && c->async_rc == RTX_OK) { c->async_rc = rc; c->async_err = g_err; }
            --c->jobs_open;
        }
        c->cv.notify_all();
    }
}

extern "C" {

int rtx_abi_version(void) { return RTX_ABI_VERSION; }
const char* rtx_last_error(void) { return g_err.c_str(); }

int rtx_device_count(int* count) {
    if (!count) return fail(RTX_ERR_INVALID, "count is NULL");
    *count = 0;
    CU(cudaGetDeviceCount(count));
    return RTX_OK;
}

int rtx_ctx_create(int device, void* stream, rtx_ctx** out) {
    if (!out) return fail(RTX_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int n = 0;
    CU(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(RTX_ERR_INVALID, "no such CUDA device");
    CU(cudaSetDevice(device));
    rtx_ctx* c = new (std::nothrow) rtx_ctx();
    if (!c) return fail(RTX_ERR_NOMEM, "out of host memory");
    c->device = device;
    if (stream) {
        c->stream = (cudaStream_t)stream;
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { rtx_ctx_destroy(c); return cuda_fail(e, "cudaStreamCreate"); }
        c->own_stream = true;
    }
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { rtx_ctx_destroy(c); return cuda_fail(e, "cudaGetDeviceProperties"); }
    c->sm_count = prop.multiProcessorCount;
    e = cudaMalloc(&c->d_work_counter, sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_counters, sizeof(rtx::Counters));
    if (e != cudaSuccess) { rtx_ctx_destroy(c); return cuda_fail(e, "cudaMalloc"); }
    auto env_int = [](const char* name, int dflt) {
        const char* v = std::getenv(name);
        int x = v ? std::atoi(v) : dflt;
        return x > 0 ? x : dflt;
    };
    c->w_node = env_int("RTX_W_NODE", c->w_node);
    c->w_leaf = env_int("RTX_W_LEAF", c->w_leaf);
    c->w_shade = env_int("RTX_W_SHADE", c->w_shade);
    c->node_burst = env_int("RTX_NODE_BURST", c->node_burst);
    c->pool_slots_wanted = env_int("RTX_WF_SLOTS", c->pool_slots_wanted);
    c->wf_batch = env_int("RTX_WF_BATCH", c->wf_batch);
    c->wf_streams = std::min(4, env_int("RTX_WF_STREAMS", c->wf_streams));
    c->wf_wide = env_int("RTX_BVH_WIDE", c->wf_wide);
    c->trace_form = env_int("RTX_TRACE", c->trace_form);
    c->trace_threads = env_int("RTX_TRACE_THREADS", c->trace_threads);
    c->t_leaf = env_int("RTX_T_LEAF", c->t_leaf);
    c->t_refill = env_int("RTX_T_REFILL", c->t_refill);
    c->t_burst = env_int("RTX_T_BURST", c->t_burst);
    c->shade_form = env_int("RTX_SHADE", c->shade_form);
    c->debug_batches = env_int("RTX_DEBUG_BATCHES", 0) != 0;
    if (const char* v = std::getenv("RTX_PERLIN_SMEM")) c->perlin_smem = std::atoi(v) != 0;
    c->prof_stride = env_int("RTX_PROF_STRIDE", c->prof_stride);
    if (const char* v = std::getenv("RTX_ORDER")) c->order_form = std::atoi(v);
    c->order_groups = env_int("RTX_ORDER_GROUPS", c->order_groups);
    { int g = 8; while (g * 2 <= c->order_groups && g < (1 << 15)) g *= 2; c->order_groups = g; }
    cudaDeviceGetAttribute(&c->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (const char* m = std::getenv("RTX_MODE")) c->mode = std::strcmp(m, "mega") == 0 ? 0 : 1;
    if (const char* m = std::getenv("RTX_BVH"))
        c->bvh_builder = std::strcmp(m, "lbvh") == 0 ? 1 : (std::strcmp(m, "ploc") == 0 ? 2 : (std::strcmp(m, "sah_device") == 0 ? 3 : 0));
    c->ploc_radius = env_int("RTX_PLOC_RADIUS", c->ploc_radius);
    // the traversal stack lives in local memory: prefer L1 over shared for it
    cudaFuncSetCacheConfig(rtx::render_kernel<false>, cudaFuncCachePreferL1);
    cudaFuncSetCacheConfig(rtx::trace_rays_kernel<false>, cudaFuncCachePreferL1);
    *out = c;
    return RTX_OK;
}

int rtx_ctx_destroy(rtx_ctx* c) {
    if (!c) return RTX_OK;
    if (c->worker.joinable()) {
        join_async(c);
        { std::lock_guard<std::mutex> lock(c->mu); c->stop = true; }
        c->cv.notify_all();
        c->worker.join();
    }
    cudaSetDevice(c->device);
    if (c->stream || !c->own_stream) cudaStreamSynchronize(c->stream);
    cudaFree(c->d_work_counter);
    cudaFree(c->d_counters);
    cudaFree(c->d_pool);
    cudaFree(c->d_order);
    cudaFree(c->d_next_item);
    cudaFree(c->d_active);
    cudaFree(c->d_denoise);
    if (c->h_status) cudaFreeHost(c->h_status);
    if (c->h_stage) cudaFreeHost(c->h_stage);
    for (auto& e : c->batch_done)
        if (e) cudaEventDestroy(e);
    for (auto e : c->prof_events) cudaEventDestroy(e);
    for (auto e : c->join_events) cudaEventDestroy(e);
    for (auto st : c->aux_streams) cudaStreamDestroy(st);
    if (c->fork_event) cudaEventDestroy(c->fork_event);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return RTX_OK;
}

int rtx_ctx_set_async(rtx_ctx* c, int on) {
    if (!c) return fail(RTX_ERR_INVALID, "ctx is NULL");
    JOIN(c);
    c->async = on != 0;
    if (c->async && !c->worker.joinable()) c->worker = std::thread(worker_main, c);
    return RTX_OK;
}

int rtx_ctx_sync(rtx_ctx* c) {
    if (!c) return fail(RTX_ERR_INVALID, "ctx is NULL");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return RTX_OK;
}
void* rtx_ctx_stream(rtx_ctx* c) { return c ? (void*)c->stream : nullptr; }
int rtx_ctx_set_profiling(rtx_ctx* c, int on) {
    if (!c) return fail(RTX_ERR_INVALID, "ctx is NULL");
    c->profiling = on != 0;
    return RTX_OK;
}
int rtx_ctx_profile_read(rtx_ctx* c, double* shade_ms, double* trace_ms, unsigned long long* iterations, int reset) {
    if (!c) return fail(RTX_ERR_INVALID, "ctx is NULL");
    JOIN(c);
    if (shade_ms) *shade_ms = c->prof_shade_ms;
    if (trace_ms) *trace_ms = c->prof_trace_ms;
    if (iterations) *iterations = c->prof_iterations;
    if (reset) { c->prof_shade_ms = c->prof_trace_ms = 0; c->prof_iterations = 0; }
    return RTX_OK;
}
int rtx_ctx_measure_l2_read(rtx_ctx* c, unsigned long long bytes, int repeats, double* gbytes_per_s) {
    if (!c || !gbytes_per_s) return fail(RTX_ERR_INVALID, "NULL argument");
    if (bytes == 0) bytes = 32ull << 20;
    if (repeats <= 0) repeats = 64;
    if (bytes < (1ull << 20) || bytes > (1ull << 30)) return fail(RTX_ERR_INVALID, "bytes must be between 1 MiB and 1 GiB");
    CU(cudaSetDevice(c->device));
    const unsigned long long n_vec = bytes / 16;
    uint4* buf = nullptr;
    unsigned int* sink = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    cudaError_t err = cudaMalloc(&buf, n_vec * 16);
    if (err == cudaSuccess) err = cudaMalloc(&sink, sizeof(unsigned int));
    if (err == cudaSuccess) err = cudaMemsetAsync(buf, 0x5a, n_vec * 16, c->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(sink, 0, sizeof(unsigned int), c->stream);
    if (err == cudaSuccess) err = cudaEventCreate(&e0);
    if (err == cudaSuccess) err = cudaEventCreate(&e1);
    float best_ms = 0.f;
    if (err == cudaSuccess) {
        const unsigned grid = (unsigned)sms * 8u;
        rtx::l2_read_kernel<<<grid, 256, 0, c->stream>>>(buf, n_vec, 2, sink);  // brings the buffer into L2
        for (int attempt = 0; attempt < 3 && err == cudaSuccess; ++attempt) {
            cudaEventRecord(e0, c->stream);
            rtx::l2_read_kernel<<<grid, 256, 0, c->stream>>>(buf, n_vec, repeats, sink);
            cudaEventRecord(e1, c->stream);
            err = cudaEventSynchronize(e1);
            float ms = 0.f;
            if (err == cudaSuccess) err = cudaEventElapsedTime(&ms, e0, e1);
            if (err == cudaSuccess && (best_ms == 0.f || ms < best_ms)) best_ms = ms;
        }
        c->launches += 4;
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(buf);
    cudaFree(sink);
    if (err != cudaSuccess) return cuda_fail(err, "rtx_ctx_measure_l2_read");
    *gbytes_per_s = (double)(n_vec * 16) * (double)repeats / ((double)best_ms * 1e-3) / 1e9;
    return RTX_OK;
}
int rtx_ctx_set_bvh_builder(rtx_ctx* c, int kind) {
    if (!c || kind < 0 || kind > 3) return fail(RTX_ERR_INVALID, "bad argument");
    c->bvh_builder = kind;
    return RTX_OK;
}
int rtx_ctx_kernel_launches(rtx_ctx* c, unsigned long long* out) {
    if (!c || !out) return fail(RTX_ERR_INVALID, "NULL argument");
    *out = c->launches;
    return RTX_OK;
}

// ---- scene ----------------------------------------------------------------
int rtx_scene_create(rtx_ctx* c, const rtx_scene_desc* desc, rtx_scene** out) {
    if (!c || !desc || !out) return fail(RTX_ERR_INVALID, "NULL argument");
    JOIN(c);
    *out = nullptr;
    CU(cudaSetDevice(c->device));
    rtx::FlatScene fs;
    std::string err;
    if (!rtx::flatten_scene(*desc, fs, err, c->bvh_builder >= 1, c->wf_wide != 0)) return fail(RTX_ERR_INVALID, "scene description: " + err);
    // nodes the device builder may add behind the host-built ones (medium boundaries), and its box upload: a binary
    // tree over n items has at most n - 1 inner nodes (the binned-SAH builder's leaves of several items make fewer)
    const size_t host_nodes = fs.nodes.size();
    const size_t lbvh_nodes = fs.world_deferred ? (size_t)fs.world_count - 1 : 0;
    size_t built_nodes = lbvh_nodes;
    rtx_scene* s = new (std::nothrow) rtx_scene();
    if (!s) return fail(RTX_ERR_NOMEM, "out of host memory");
    s->device = c->device;
    auto bail = [&](int code) { rtx_scene_destroy(s); return code; };

    // pinned staging: the flattened arena and the image texels are copied H2D from page-locked memory
    size_t image_bytes = 0;
    for (int i = 0; i < desc->n_images; ++i)
        if (desc->images[i].rgba && desc->images[i].width > 0 && desc->images[i].height > 0)
            image_bytes += ((size_t)desc->images[i].width * (size_t)desc->images[i].height * 4 + 255) & ~(size_t)255;
    auto stage_reserve = [&](size_t bytes) -> cudaError_t {
        if (bytes <= c->stage_bytes) return cudaSuccess;
        if (c->h_stage) { cudaStreamSynchronize(c->stream); cudaFreeHost(c->h_stage); c->h_stage = nullptr; c->stage_bytes = 0; }
        cudaError_t err = cudaMallocHost(&c->h_stage, bytes);
        if (err == cudaSuccess) c->stage_bytes = bytes;
        return err;
    };
    const size_t arena_bound = (host_nodes + lbvh_nodes) * sizeof(rtx::BvhNode) + fs.world_boxes.size() * sizeof(float) +
                               fs.records.size() * sizeof(rtx::Record) +
                               fs.xforms.size() * sizeof(rtx::XformOp) + fs.chains.size() * sizeof(rtx::DChain) +
                               fs.materials.size() * sizeof(rtx::DMaterial) + fs.textures.size() * sizeof(rtx::DTexture) +
                               fs.perlins.size() * sizeof(rtx::DPerlin) + (size_t)desc->n_images * sizeof(rtx::DImage) +
                               fs.media.size() * sizeof(rtx::DMedium) + 16 * 256;
    {
        cudaError_t e = stage_reserve(image_bytes + arena_bound);
        if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMallocHost(staging)"));
    }
    size_t stage_used = 0;

    // images -> point-sampled texture objects (ImageTexture, texture.rs:61-107)
    std::vector<rtx::DImage> dimages((size_t)desc->n_images);
    for (int i = 0; i < desc->n_images; ++i) {
        const rtx_image& im = desc->images[i];
        rtx::DImage& di = dimages[(size_t)i];
        di.tex = 0; di.width = im.width; di.height = im.height;
        if (!im.rgba || im.width <= 0 || im.height <= 0) continue;
        ArraySlot slot{nullptr, 0, im.width, im.height};
        if (c->device < kMaxDevices) {  // an array + texture object of the same size left by a destroyed scene
            DeviceCache& dc = g_cache[c->device];
            std::lock_guard<std::mutex> lock(dc.m);
            for (size_t k = 0; k < dc.arrays.size(); ++k)
                if (dc.arrays[k].w == im.width && dc.arrays[k].h == im.height) {
                    slot = dc.arrays[k];
                    dc.arrays.erase(dc.arrays.begin() + (long)k);
                    break;
                }
        }
        cudaError_t e = cudaSuccess;
        if (!slot.arr) {
            cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
            e = cudaMallocArray(&slot.arr, &fmt, (size_t)im.width, (size_t)im.height);
            if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMallocArray"));
            cudaResourceDesc rd;
            std::memset(&rd, 0, sizeof(rd));
            rd.resType = cudaResourceTypeArray;
            rd.res.array.array = slot.arr;
            cudaTextureDesc td;
            std::memset(&td, 0, sizeof(td));
            td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
            td.filterMode = cudaFilterModePoint;  // nearest texel, no filtering, no sRGB decode (Q23)
            td.readMode = cudaReadModeElementType;
            td.normalizedCoords = 0;
            e = cudaCreateTextureObject(&slot.tex, &rd, &td, nullptr);
            if (e != cudaSuccess) { cudaFreeArray(slot.arr); return bail(cuda_fail(e, "cudaCreateTextureObject")); }
        }
        s->images.push_back(slot);
        const size_t nbytes = (size_t)im.width * (size_t)im.height * 4;
        uint8_t* staged = c->h_stage + stage_used;
        std::memcpy(staged, im.rgba, nbytes);
        stage_used += (nbytes + 255) & ~(size_t)255;
        e = cudaMemcpy2DToArrayAsync(slot.arr, 0, 0, staged, (size_t)im.width * 4, (size_t)im.width * 4, (size_t)im.height,
                                     cudaMemcpyHostToDevice, c->stream);
        if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMemcpy2DToArray"));
        cudaTextureObject_t tex = slot.tex;
        di.tex = (unsigned long long)tex;
    }

    // one arena, every array 256-byte aligned
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t off_nodes = 0;
    size_t off_records = align(off_nodes + (host_nodes + lbvh_nodes) * sizeof(rtx::BvhNode));
    size_t off_xforms = align(off_records + fs.records.size() * sizeof(rtx::Record));
    size_t off_chains = align(off_xforms + fs.xforms.size() * sizeof(rtx::XformOp));
    size_t off_mats = align(off_chains + fs.chains.size() * sizeof(rtx::DChain));
    size_t off_texs = align(off_mats + fs.materials.size() * sizeof(rtx::DMaterial));
    size_t off_perlins = align(off_texs + fs.textures.size() * sizeof(rtx::DTexture));
    size_t off_images = align(off_perlins + fs.perlins.size() * sizeof(rtx::DPerlin));
    size_t off_media = align(off_images + dimages.size() * sizeof(rtx::DImage));
    size_t off_boxes = align(off_media + fs.media.size() * sizeof(rtx::DMedium));
    size_t total = align(off_boxes + fs.world_boxes.size() * sizeof(float)) + 256;
    if (total > arena_bound) return bail(fail(RTX_ERR_NOMEM, "internal: arena larger than its bound"));
    uint8_t* host = c->h_stage + stage_used;
    std::memset(host, 0, total);
    auto put = [&](size_t off, const void* src, size_t bytes) { if (bytes) std::memcpy(host + off, src, bytes); };
    put(off_nodes, fs.nodes.data(), fs.nodes.size() * sizeof(rtx::BvhNode));
    put(off_records, fs.records.data(), fs.records.size() * sizeof(rtx::Record));
    put(off_xforms, fs.xforms.data(), fs.xforms.size() * sizeof(rtx::XformOp));
    put(off_chains, fs.chains.data(), fs.chains.size() * sizeof(rtx::DChain));
    put(off_mats, fs.materials.data(), fs.materials.size() * sizeof(rtx::DMaterial));
    put(off_texs, fs.textures.data(), fs.textures.size() * sizeof(rtx::DTexture));
    put(off_perlins, fs.perlins.data(), fs.perlins.size() * sizeof(rtx::DPerlin));
    put(off_images, dimages.data(), dimages.size() * sizeof(rtx::DImage));
    put(off_media, fs.media.data(), fs.media.size() * sizeof(rtx::DMedium));
    put(off_boxes, fs.world_boxes.data(), fs.world_boxes.size() * sizeof(float));
    if (c->device < kMaxDevices) {  // smallest cached arena that is large enough
        DeviceCache& dc = g_cache[c->device];
        std::lock_guard<std::mutex> lock(dc.m);
        size_t pick = dc.arenas.size();
        for (size_t k = 0; k < dc.arenas.size(); ++k)
            if (dc.arenas[k].bytes >= total && (pick == dc.arenas.size() || dc.arenas[k].bytes < dc.arenas[pick].bytes)) pick = k;
        if (pick < dc.arenas.size()) {
            s->d_arena = dc.arenas[pick].p;
            s->arena_capacity = dc.arenas[pick].bytes;
            dc.arenas.erase(dc.arenas.begin() + (long)pick);
        }
    }
    cudaError_t e = cudaSuccess;
    if (!s->d_arena) {
        e = cudaMalloc(&s->d_arena, total);
        if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMalloc(scene)"));
        s->arena_capacity = total;
    }
    s->arena_bytes = total;
    e = cudaMemcpyAsync(s->d_arena, host, total, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);  // the staging buffer is reused by the next call
    if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMemcpy(scene)"));
    uint8_t* base = (uint8_t*)s->d_arena;
    if (fs.world_deferred) {
        // the world BVH is built on the device, straight into the arena behind the host-built nodes
        float lo[3], ext[3];
        for (int a = 0; a < 3; ++a) { lo[a] = 3.4e38f; ext[a] = -3.4e38f; }
        for (int32_t k = 0; k < fs.world_count; ++k)
            for (int a = 0; a < 3; ++a) {
                float cc = 0.5f * (fs.world_boxes[(size_t)(6 * k + a)] + fs.world_boxes[(size_t)(6 * k + 3 + a)]);
                lo[a] = std::fmin(lo[a], cc);
                ext[a] = std::fmax(ext[a], cc);
            }
        for (int a = 0; a < 3; ++a) ext[a] -= lo[a];
        int depth = 0;
        if (c->bvh_builder == 3) {
            rtx::SahBuildStats st;
            e = rtx::sah_build(c->stream, fs.world_count, (const float*)(base + off_boxes), fs.world_first_record,
                               (rtx::Record*)(base + off_records) + fs.world_first_record, (int32_t)host_nodes,
                               (rtx::BvhNode*)(base + off_nodes) + host_nodes, rtx::BvhPolicy::from_env(), rtx::kTraversalStack - 2, &st);
            if (e != cudaSuccess) return bail(cuda_fail(e, "sah_build"));
            c->launches += st.launches;
            depth = st.depth;
            built_nodes = (size_t)st.nodes;
            if (std::getenv("RTX_DEBUG_BUILD"))
                std::fprintf(stderr, "[rtx] SAH (device): %d primitives, %d levels, depth %d, %d nodes\n", fs.world_count, st.levels, depth, st.nodes);
        } else if (c->bvh_builder == 2) {
            int passes = 0;
            e = rtx::ploc_build(c->stream, fs.world_count, (const float*)(base + off_boxes), lo, ext, fs.world_first_record, (int32_t)host_nodes,
                                (rtx::BvhNode*)(base + off_nodes) + host_nodes, &depth, c->ploc_radius, &passes);
            if (e != cudaSuccess) return bail(cuda_fail(e, "ploc_build"));
            c->last_build_passes = passes;
            c->launches += 4ull + 4ull * (unsigned long long)passes;
            if (std::getenv("RTX_DEBUG_BUILD")) std::fprintf(stderr, "[rtx] PLOC: %d primitives, radius %d, %d passes, depth %d\n", fs.world_count, c->ploc_radius, passes, depth);
        } else {
            e = rtx::lbvh_build(c->stream, fs.world_count, (const float*)(base + off_boxes), lo, ext, fs.world_first_record, (int32_t)host_nodes,
                                (rtx::BvhNode*)(base + off_nodes) + host_nodes, &depth);
            if (e != cudaSuccess) return bail(cuda_fail(e, "lbvh_build"));
            c->launches += 4;
        }
        if (1 + depth + 1 > rtx::kTraversalStack)
            return bail(fail(RTX_ERR_UNSUPPORTED, "device-built BVH deeper than the traversal stack: use the host builder"));
        fs.world_root = (int32_t)host_nodes;
        fs.world_first_node = (int32_t)host_nodes;
        fs.world_node_count = (int32_t)built_nodes;
        fs.world_depth = depth;
    }
    s->view.nodes = (const rtx::BvhNode*)(base + off_nodes);
    s->view.records = (const rtx::Record*)(base + off_records);
    s->view.xforms = (const rtx::XformOp*)(base + off_xforms);
    s->view.chains = (const rtx::DChain*)(base + off_chains);
    s->view.materials = (const rtx::DMaterial*)(base + off_mats);
    s->view.textures = (const rtx::DTexture*)(base + off_texs);
    s->view.perlins = (const rtx::DPerlin*)(base + off_perlins);
    s->view.images = (const rtx::DImage*)(base + off_images);
    s->view.media = (const rtx::DMedium*)(base + off_media);
    s->view.world_root = fs.world_root;
    s->view.wide_root = fs.world_deferred ? -1 : fs.wide_root;
    s->view.n_media = fs.n_media;
    s->camera = fs.camera;
    s->n_nodes = (int32_t)(host_nodes + built_nodes);
    s->n_records = (int32_t)fs.records.size();
    s->n_xforms = (int32_t)fs.xforms.size();
    s->world_first_node = fs.world_first_node;
    s->world_node_count = fs.world_node_count;
    s->world_depth = fs.world_depth;
    s->n_perlins = (int32_t)fs.perlins.size();
    *out = s;
    return RTX_OK;
}

int rtx_scene_destroy(rtx_scene* s) {
    if (!s) return RTX_OK;
    cudaSetDevice(s->device);
    cudaDeviceSynchronize();  // kernels still reading the arena (any stream)
    DeviceCache* dc = s->device < kMaxDevices ? &g_cache[s->device] : nullptr;
    for (auto& im : s->images) {
        bool kept = false;
        if (dc) {
            std::lock_guard<std::mutex> lock(dc->m);
            if (dc->arrays.size() < kCacheKeep) { dc->arrays.push_back(im); kept = true; }
        }
        if (!kept) { cudaDestroyTextureObject(im.tex); cudaFreeArray(im.arr); }
    }
    if (s->d_arena) {
        bool kept = false;
        if (dc) {
            std::lock_guard<std::mutex> lock(dc->m);
            if (dc->arenas.size() < kCacheKeep) { dc->arenas.push_back(ArenaSlot{s->d_arena, s->arena_capacity}); kept = true; }
        }
        if (!kept) cudaFree(s->d_arena);
    }
    if (s->env.texels) cudaFree((void*)s->env.texels);
    delete s;
    return RTX_OK;
}

int rtx_cache_trim(int device) {
    if (device < 0 || device >= kMaxDevices) return fail(RTX_ERR_INVALID, "no such device slot");
    DeviceCache& dc = g_cache[device];
    std::lock_guard<std::mutex> lock(dc.m);
    if (dc.arenas.empty() && dc.arrays.empty()) return RTX_OK;
    CU(cudaSetDevice(device));
    for (auto& a : dc.arenas) cudaFree(a.p);
    for (auto& im : dc.arrays) { cudaDestroyTextureObject(im.tex); cudaFreeArray(im.arr); }
    dc.arenas.clear();
    dc.arrays.clear();
    return RTX_OK;
}

int rtx_scene_info(const rtx_scene* s, int32_t* n_bvh_nodes, int32_t* n_records, int32_t* n_xform_ops, int64_t* device_bytes) {
    if (!s) return fail(RTX_ERR_INVALID, "scene is NULL");
    if (n_bvh_nodes) *n_bvh_nodes = s->n_nodes;
    if (n_records) *n_records = s->n_records;
    if (n_xform_ops) *n_xform_ops = s->n_xforms;
    if (device_bytes) *device_bytes = (int64_t)(s->arena_bytes + s->env_bytes);
    return RTX_OK;
}

int rtx_scene_set_environment(rtx_ctx* c, rtx_scene* s, const rtx_environment* env) {
    if (!c || !s) return fail(RTX_ERR_INVALID, "NULL argument");
    if (c->device != s->device) return fail(RTX_ERR_INVALID, "the context and the scene are on different devices");
    std::vector<float4> host;
    rtx::EnvArgs e{};
    if (env) {
        if (env->width < 1 || env->height < 1 || (int64_t)env->width * env->height > 0x7fffffff)
            return fail(RTX_ERR_INVALID, "environment size must be >= 1 x 1 and below 2^31 texels");
        if (!env->rgb) return fail(RTX_ERR_INVALID, "environment texels are NULL");
        if (!std::isfinite(env->rotation_y)) return fail(RTX_ERR_INVALID, "environment rotation must be finite");
        for (double k : env->scale)
            if (!(k >= 0.0) || !std::isfinite(k)) return fail(RTX_ERR_INVALID, "environment scale must be finite and >= 0");
        const size_t n = (size_t)env->width * env->height;
        host.resize(n + 1);
        host[0] = make_float4((float)env->scale[0], (float)env->scale[1], (float)env->scale[2], 0.f);
        for (size_t i = 0; i < n; ++i) {
            const float* t = env->rgb + 3 * i;
            for (int k = 0; k < 3; ++k)
                if (!(t[k] >= 0.f) || !std::isfinite(t[k])) return fail(RTX_ERR_INVALID, "environment texels must be finite and >= 0");
            host[i + 1] = make_float4(t[0], t[1], t[2], 0.f);
        }
        const double th = env->rotation_y * (3.14159265358979323846 / 180.0);
        e.width = env->width;
        e.height = env->height;
        e.cos_t = std::cos(th);
        e.sin_t = std::sin(th);
    }
    JOIN(c);
    CU(cudaSetDevice(s->device));
    void* d = nullptr;
    if (env) {
        CU(cudaMalloc(&d, host.size() * sizeof(float4)));
        // on the ctx stream and waited for, like the scene upload: once the call returns the texels are on the device,
        // whichever stream renders next
        cudaError_t err = cudaMemcpyAsync(d, host.data(), host.size() * sizeof(float4), cudaMemcpyHostToDevice, c->stream);
        if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
        if (err != cudaSuccess) { cudaFree(d); return cuda_fail(err, "cudaMemcpyAsync (environment)"); }
        e.texels = (const float4*)d;
    }
    // renders queued on any stream may still read the old map
    if (s->env.texels) { CU(cudaDeviceSynchronize()); CU(cudaFree((void*)s->env.texels)); }
    s->env = e;
    s->env_bytes = host.size() * sizeof(float4);
    return RTX_OK;
}

// ---- fixed rays -------------------------------------------------------------
int rtx_trace_rays_device(rtx_ctx* c, const rtx_scene* s, int64_t n, const rtx_ray* d_rays, rtx_hit* d_hits) {
    if (!c || !s || n < 0 || (n > 0 && (!d_rays || !d_hits))) return fail(RTX_ERR_INVALID, "bad argument");
    JOIN(c);
    if (n == 0) return RTX_OK;
    CU(cudaSetDevice(c->device));
    const int block = 128;
    int64_t grid = (n + block - 1) / block;
    if (grid > 0x7fffffff) return fail(RTX_ERR_INVALID, "too many rays for one launch");
    rtx::trace_rays_kernel<false><<<(unsigned)grid, block, 0, c->stream>>>(s->view, n, d_rays, d_hits, nullptr);
    c->launches += 1;
    CU(cudaGetLastError());
    return RTX_OK;
}

int rtx_trace_rays(rtx_ctx* c, const rtx_scene* s, int64_t n, const rtx_ray* rays, rtx_hit* hits) {
    if (!c || !s || n < 0 || (n > 0 && (!rays || !hits))) return fail(RTX_ERR_INVALID, "bad argument");
    if (n == 0) return RTX_OK;
    CU(cudaSetDevice(c->device));
    rtx_ray* d_rays = nullptr;
    rtx_hit* d_hits = nullptr;
    CU(cudaMalloc(&d_rays, (size_t)n * sizeof(rtx_ray)));
    cudaError_t e = cudaMalloc(&d_hits, (size_t)n * sizeof(rtx_hit));
    if (e != cudaSuccess) { cudaFree(d_rays); return cuda_fail(e, "cudaMalloc(hits)"); }
    int rc = RTX_OK;
    e = cudaMemcpyAsync(d_rays, rays, (size_t)n * sizeof(rtx_ray), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        rc = rtx_trace_rays_device(c, s, n, d_rays, d_hits);
        if (rc == RTX_OK) {
            e = cudaMemcpyAsync(hits, d_hits, (size_t)n * sizeof(rtx_hit), cudaMemcpyDeviceToHost, c->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        }
    }
    cudaFree(d_rays);
    cudaFree(d_hits);
    if (rc != RTX_OK) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "rtx_trace_rays");
    return RTX_OK;
}

// The device tallies as means per ray (the sums themselves when no ray was traced).
static void trace_stats(const rtx::Counters& h, unsigned long long rays, rtx_trace_stats* out) {
    const double dn = rays ? (double)rays : 1.0;
    out->rays = (double)rays;
    out->box_tests = (double)h.box_tests / dn;
    out->node_visits = (double)h.node_visits / dn;
    out->sphere_tests = (double)h.sphere_tests / dn;
    out->rect_tests = (double)h.rect_tests / dn;
    out->instance_enters = (double)h.instance_enters / dn;
    out->medium_tests = (double)h.medium_tests / dn;
}

int rtx_trace_rays_stats(rtx_ctx* c, const rtx_scene* s, int64_t n, const rtx_ray* d_rays, rtx_trace_stats* out) {
    if (!c || !s || n <= 0 || !d_rays || !out) return fail(RTX_ERR_INVALID, "bad argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaMemsetAsync(c->d_counters, 0, sizeof(rtx::Counters), c->stream));
    const int block = 128;
    int64_t grid = (n + block - 1) / block;
    if (grid > 0x7fffffff) return fail(RTX_ERR_INVALID, "too many rays for one launch");
    rtx::trace_rays_kernel<true><<<(unsigned)grid, block, 0, c->stream>>>(s->view, n, d_rays, nullptr, c->d_counters);
    c->launches += 1;
    CU(cudaGetLastError());
    rtx::Counters h;
    CU(cudaMemcpyAsync(&h, c->d_counters, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    trace_stats(h, (unsigned long long)n, out);
    return RTX_OK;
}

}  // extern "C"

// ---- render: frame setup shared by the render entry points ------------------------
// The refusals the render entry points share, in this order: a bad size, first sample or depth, or the entry point's own
// condition `bad`, worded `bad_text`; 2^31 pixels or more; unless count_of is null, more than 2^24 samples per pixel
// into the fp32 sample count of the buffer it names.
static int check_frame(const rtx_render_params* p, int min_depth, bool bad, const char* bad_text, const char* count_of) {
    if (p->width <= 0 || p->height <= 0 || p->spp_begin < 0 || p->max_depth < min_depth || bad) return fail(RTX_ERR_INVALID, bad_text);
    if ((int64_t)p->width * p->height > 0x7fffffff) return fail(RTX_ERR_INVALID, "image too large");
    if (count_of && p->spp_count > (1 << 24))
        return fail(RTX_ERR_INVALID, std::string("more than 2^24 samples per pixel in one call (the fp32 sample count of the ") + count_of + ")");
    return RTX_OK;
}

struct Tiles {  // a frame's 8x4-pixel tiles; inv_per_block_row = 1 / (x * kBlockH), see tile_of_order
    int32_t x, y;
    float inv_per_block_row;
};
static Tiles frame_tiles(int32_t width, int32_t height) {
    const int32_t x = (width + rtx::kTileW - 1) / rtx::kTileW;
    return {x, (height + rtx::kTileH - 1) / rtx::kTileH, 1.0f / (float)(x * rtx::kBlockH)};
}

// Fills the frame fields of WfArgs, RenderArgs and AovArgs and returns the frame's tiles. The feature pass stops at the
// first vertex and numbers its tiles in raster order, so AovArgs has no max_depth, tiles_y or inv_per_block_row.
template <class Args>
static Tiles set_frame(Args& a, const rtx_scene* s, const rtx_render_params* p) {
    const Tiles t = frame_tiles(p->width, p->height);
    a.sc = s->view;
    a.cam = s->camera;
    a.width = p->width; a.height = p->height;
    a.spp_begin = p->spp_begin; a.spp_count = p->spp_count;
    a.k0 = (uint32_t)p->seed; a.k1 = (uint32_t)(p->seed >> 32);
    a.tiles_x = t.x;
    if constexpr (!std::is_same<Args, rtx::AovArgs>::value) {
        a.max_depth = p->max_depth;
        a.tiles_y = t.y;
        a.inv_per_block_row = t.inv_per_block_row;
    }
    return t;
}

// ---- render: wavefront driver ---------------------------------------------------
// The path pool's SoA arrays, carved out of one allocation of `slots` slots (kPoolBytesPerSlot each, 8-byte arrays
// first), and the pool of a partition, the slots from `begin` on.
template <class F>
static void for_each_array(rtx::PathPool& pool, F f) {
    f(pool.ox); f(pool.oy); f(pool.oz); f(pool.dx); f(pool.dy); f(pool.dz); f(pool.time); f(pool.best_t);
    f(pool.best_rec); f(pool.best_chain); f(pool.bounce); f(pool.pixel); f(pool.sample);
    f(pool.thr_r); f(pool.thr_g); f(pool.thr_b);
}
static rtx::PathPool pool_carve(void* base, int64_t slots) {
    rtx::PathPool pool;
    uint8_t* next = (uint8_t*)base;
    for_each_array(pool, [&](auto*& arr) {
        arr = reinterpret_cast<std::remove_reference_t<decltype(arr)>>(next);
        next += (size_t)slots * sizeof(*arr);
    });
    return pool;
}
static rtx::PathPool pool_part(rtx::PathPool pool, int64_t begin) {
    for_each_array(pool, [&](auto*& arr) { arr += begin; });
    return pool;
}

// Slots of the pool for a job of `total` path samples: the configured maximum, but a small job (few pool refills) is
// all ramp-up and drain with a pool that large: keep at least ~24 refills, down to 256 Ki slots. Whole CTAs.
static int64_t pool_slots_for(const rtx_ctx* c, unsigned long long total) {
    int64_t slots = c->pool_slots_wanted;
    if ((unsigned long long)slots > total / 24) slots = (int64_t)(total / 24);
    if (slots < (256 << 10)) slots = 256 << 10;
    if (slots > c->pool_slots_wanted) slots = c->pool_slots_wanted;
    if ((unsigned long long)slots > total) slots = (int64_t)total;
    return (slots + rtx::kWfBlock - 1) / rtx::kWfBlock * rtx::kWfBlock;
}

// The scratch of ray ordering (order.cuh) for `parts` partitions of `slots` slots: per partition, hist [bins],
// offsets [bins + 1] and done in a stride of part_words; behind them, 256-byte aligned at slots_at, key_rank (8 B)
// and order (4 B) of every slot. bins (n_bins_padded) is 8 * groups + 1, rounded up to whole uint4 per shade thread.
struct OrderLayout {
    size_t bins, part_words, slots_at, bytes;
};
static OrderLayout order_layout(int groups, int parts, int64_t slots) {
    const size_t unit = 4 * (size_t)rtx::kShadeBlock;
    OrderLayout l;
    l.bins = ((size_t)8 * (size_t)groups + 1 + unit - 1) / unit * unit;
    l.part_words = 2 * l.bins + 64;
    l.slots_at = ((size_t)parts * l.part_words * 4 + 255) & ~(size_t)255;
    l.bytes = l.slots_at + (size_t)slots * 12;
    return l;
}

static int wf_prepare(rtx_ctx* c, int64_t slots) {
    if (slots > c->pool_slots) {
        if (c->d_pool) { CU(cudaStreamSynchronize(c->stream)); CU(cudaFree(c->d_pool)); c->d_pool = nullptr; c->pool_slots = 0; }
        CU(cudaMalloc(&c->d_pool, (size_t)slots * rtx::kPoolBytesPerSlot + 256));
        c->pool_slots = (int)slots;
    }
    if (c->order_form != 0) {
        const size_t need = order_layout(c->order_groups, c->wf_streams, slots).bytes;
        if (need > c->order_bytes) {
            if (c->d_order) { CU(cudaStreamSynchronize(c->stream)); CU(cudaFree(c->d_order)); c->d_order = nullptr; c->order_bytes = 0; }
            CU(cudaMalloc(&c->d_order, need));
            c->order_bytes = need;
        }
    }
    if (!c->d_next_item) CU(cudaMalloc(&c->d_next_item, sizeof(unsigned long long)));
    if (!c->d_active) CU(cudaMalloc(&c->d_active, 8 * sizeof(unsigned int)));

    if (!c->h_status) CU(cudaMallocHost(&c->h_status, 16 * sizeof(unsigned long long)));
    while ((int)c->aux_streams.size() < c->wf_streams - 1) {
        cudaStream_t st;
        cudaEvent_t ev;
        CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        c->aux_streams.push_back(st);
        c->join_events.push_back(ev);
    }
    if (!c->fork_event) CU(cudaEventCreateWithFlags(&c->fork_event, cudaEventDisableTiming));
    for (auto& e : c->batch_done)
        if (!e) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return RTX_OK;
}

// The signatures of the kernels a render call chooses among: every shade kernel; the trace kernels that take the slots
// in slot order (form 1, wide or not, and 1c); the ordered trace kernel; forms 2 and 3.
using ShadeKernel = void (*)(rtx::WfArgs, float4*, unsigned int*, rtx::Counters*);
using SlotTraceKernel = void (*)(rtx::SceneView, rtx::PathPool, int, unsigned long long*, rtx::Counters*);
using OrderedTraceKernel = void (*)(rtx::SceneView, rtx::PathPool, rtx::OrderArgs, unsigned long long*, rtx::Counters*);
using Trace2Kernel = void (*)(rtx::SceneView, rtx::PathPool, int, rtx::TraceCfg, unsigned long long*, rtx::Counters*);
using Trace3Kernel = void (*)(rtx::SceneView, rtx::PathPool, int, rtx::Trace3Cfg, unsigned long long*, rtx::Counters*);

// The instantiations of the shared-memory forms 2 and 3 for a CTA size wf_plan has snapped, counted or not, with the
// whole world BVH staged or not.
template <bool kCount, bool kAll>
static Trace2Kernel trace2_of(int threads) {
    switch (threads) {
        case 1024: return rtx::wf_trace2_kernel<kCount, 1024, kAll>;
        case 896: return rtx::wf_trace2_kernel<kCount, 896, kAll>;
        case 640: return rtx::wf_trace2_kernel<kCount, 640, kAll>;
        case 512: return rtx::wf_trace2_kernel<kCount, 512, kAll>;
        default: return rtx::wf_trace2_kernel<kCount, 448, kAll>;
    }
}
static Trace2Kernel trace2_kernel(bool counted, int threads, bool all) {
    if (counted) return all ? trace2_of<true, true>(threads) : trace2_of<true, false>(threads);
    return all ? trace2_of<false, true>(threads) : trace2_of<false, false>(threads);
}
template <bool kCount, bool kAll>
static Trace3Kernel trace3_of(int threads) {
    switch (threads) {
        case 896: return rtx::wf_trace3_kernel<kCount, 896, kAll>;
        case 768: return rtx::wf_trace3_kernel<kCount, 768, kAll>;
        case 640: return rtx::wf_trace3_kernel<kCount, 640, kAll>;
        default: return rtx::wf_trace3_kernel<kCount, 512, kAll>;
    }
}
static Trace3Kernel trace3_kernel(bool counted, int threads, bool all) {
    if (counted) return all ? trace3_of<true, true>(threads) : trace3_of<true, false>(threads);
    return all ? trace3_of<false, true>(threads) : trace3_of<false, false>(threads);
}

// A partition of the pool, driven on its own stream.
struct WfPart {
    rtx::WfArgs a;
    cudaStream_t stream;
    unsigned sgrid, tgrid;  // CTAs of its shade and trace launches
    bool done;
};

// The kernels of one render call, chosen once before its first iteration. The trace step is exactly one of the four
// trace kernels. The shared-memory forms 2 and 3 (threads > 0) run CTAs of `threads` threads with `smem` bytes of
// dynamic shared memory, one per SM at most; the others run one thread per slot in kTraceBlock-thread CTAs.
struct WfPlan {
    ShadeKernel shade = nullptr;
    bool order_pass = false;            // RTX_ORDER=1: wf_order_kernel sorts the slots between shade and trace
    rtx::Counters* counters = nullptr;  // the tallies of a counted render (rtx_render_counted)
    SlotTraceKernel trace_slots = nullptr;
    OrderedTraceKernel trace_ordered = nullptr;
    Trace2Kernel trace2 = nullptr;
    Trace3Kernel trace3 = nullptr;
    rtx::TraceCfg cfg2{};
    rtx::Trace3Cfg cfg3{};
    int threads = 0;
    size_t smem = 0;

    unsigned long long launches() const { return order_pass ? 3 : 2; }  // per iteration
    unsigned trace_grid(int64_t slots, int sm_count) const {
        if (threads == 0) return (unsigned)(slots / rtx::kTraceBlock);
        // one CTA per SM (fewer when the partition is small): each stages the BVH once and walks its share of the slots
        return (unsigned)std::max<int64_t>(1, std::min<int64_t>(sm_count, (slots + threads - 1) / threads));
    }
    void launch_shade(const WfPart& pt, float4* acc, unsigned int* active) const {
        shade<<<pt.sgrid, rtx::kShadeBlock, 0, pt.stream>>>(pt.a, acc, active, counters);
        if (order_pass) rtx::wf_order_kernel<<<(unsigned)((pt.a.n_slots + 255) / 256), 256, 0, pt.stream>>>(pt.a.order, pt.a.n_slots);
    }
    void launch_trace(const WfPart& pt, unsigned long long* rays) const {
        const rtx::WfArgs& a = pt.a;
        if (trace_ordered) trace_ordered<<<pt.tgrid, rtx::kTraceBlock, 0, pt.stream>>>(a.sc, a.pool, a.order, rays, counters);
        else if (trace2) trace2<<<pt.tgrid, threads, smem, pt.stream>>>(a.sc, a.pool, a.n_slots, cfg2, rays, counters);
        else if (trace3) trace3<<<pt.tgrid, threads, smem, pt.stream>>>(a.sc, a.pool, a.n_slots, cfg3, rays, counters);
        else trace_slots<<<pt.tgrid, rtx::kTraceBlock, 0, pt.stream>>>(a.sc, a.pool, a.n_slots, rays, counters);
    }
};

// Forms 2 and 3 stage as much of the world BVH in shared memory as fits next to `fixed` bytes of their own (stacks,
// ray state): the nodes staged, 0 when not even one fits.
static int stage_cap(const rtx_ctx* c, const rtx_scene* s, size_t fixed) {
    const size_t room = (size_t)c->smem_optin > fixed ? (size_t)c->smem_optin - fixed : 0;
    return (int)std::min<size_t>(room / rtx::kNodeStride, (size_t)s->world_node_count);
}

static WfPlan wf_plan(const rtx_ctx* c, const rtx_scene* s, bool counted, bool adaptive) {
    WfPlan pl;
    const bool env = s->env.texels != nullptr;  // (env_refusal has ruled out counting, ray ordering and the first form)
    pl.counters = counted ? c->d_counters : nullptr;
    const bool wide = c->wf_wide != 0 && s->view.wide_root >= 0;
    pl.order_pass = c->order_form != 0 && c->shade_form >= 2 && c->trace_form == 1 && !wide;
    // the shade kernel stages the Perlin table in shared memory when the scene has exactly one (not when counting)
    const bool perlin = c->perlin_smem && s->n_perlins == 1;
    if (env)
        pl.shade = adaptive ? (perlin ? rtx::wf_shade2_env_kernel<true, true> : rtx::wf_shade2_env_kernel<false, true>)
                            : (perlin ? rtx::wf_shade2_env_kernel<true, false> : rtx::wf_shade2_env_kernel<false, false>);
    else if (adaptive)  // (rtx_render_adaptive refuses the first shade form and ray ordering)
        pl.shade = perlin ? rtx::wf_shade2_kernel<false, true, false, true> : rtx::wf_shade2_kernel<false, false, false, true>;
    else if (c->shade_form < 2)
        pl.shade = counted ? rtx::wf_shade_kernel<true> : rtx::wf_shade_kernel<false>;
    else if (counted)
        pl.shade = pl.order_pass ? rtx::wf_shade2_kernel<true, false, true> : rtx::wf_shade2_kernel<true>;
    else if (pl.order_pass)
        pl.shade = perlin ? rtx::wf_shade2_kernel<false, true, true> : rtx::wf_shade2_kernel<false, false, true>;
    else
        pl.shade = perlin ? rtx::wf_shade2_kernel<false, true> : rtx::wf_shade2_kernel<false>;
    // forms 2-4 keep their stacks in shared memory: deeper world BVHs, and the wide one, fall back to form 1
    const bool short_stack = !wide && s->world_depth <= rtx::kShortStack;
    const bool staged = c->trace_form >= 2 && short_stack && s->world_node_count > 0;
    if (pl.order_pass) {
        pl.trace_ordered = counted ? rtx::wf_trace_ordered_kernel<true> : rtx::wf_trace_ordered_kernel<false>;
        return pl;
    }
    if (c->trace_form == 4 && short_stack) {  // "1c": form 1's launch shape, shared-memory stack, 32-byte node loads
        pl.trace_slots = counted ? rtx::wf_trace1c_kernel<true> : rtx::wf_trace1c_kernel<false>;
        return pl;
    }
    // form 3 (trace3.cuh: rays regrouped by the kind of work they need next) where it fits, else form 2 (trace2.cuh:
    // persistent warps with voted refill) for any form >= 2 where it fits, else form 1
    const int t3 = c->trace_threads >= 896 ? 896 : (c->trace_threads >= 768 ? 768 : (c->trace_threads >= 640 ? 640 : 512));
    const int t2 = c->trace_threads >= 1024 ? 1024 : c->trace_threads >= 896 ? 896 : (c->trace_threads >= 640 ? 640 : (c->trace_threads >= 512 ? 512 : 448));
    const size_t fixed3 = rtx::trace3_smem_bytes(t3, 0), fixed2 = (size_t)(1 + rtx::kShortStack) * (size_t)t2 * 4 + 16;
    const int cap3 = staged && c->trace_form == 3 ? stage_cap(c, s, fixed3) : 0;
    const int cap2 = staged ? stage_cap(c, s, fixed2) : 0;
    if (cap3 >= 1) {
        pl.trace3 = trace3_kernel(counted, t3, cap3 == s->world_node_count);
        pl.cfg3 = {s->world_first_node, cap3, cap3, c->t_burst};
        pl.threads = t3;
        pl.smem = rtx::trace3_smem_bytes(t3, cap3);
    } else if (cap2 >= 1) {
        pl.trace2 = trace2_kernel(counted, t2, cap2 == s->world_node_count);
        pl.cfg2 = {s->world_first_node, cap2, cap2, c->t_leaf, c->t_refill, c->t_burst};
        pl.threads = t2;
        pl.smem = (size_t)cap2 * rtx::kNodeStride + fixed2;
    } else {
        pl.trace_slots = wide ? (counted ? rtx::wf_trace_kernel<true, true> : rtx::wf_trace_kernel<false, true>)
                              : (counted ? rtx::wf_trace_kernel<true> : rtx::wf_trace_kernel<false>);
    }
    return pl;
}

// Adaptive sampling's part of a render (rtx_render_adaptive): only the n_tiles tiles of the list of dispenser order
// indices are rendered, and the samples with an odd global index also go to aux.
struct AdaptivePass {
    rtx::AdaptiveArgs args;  // tile_list, aux
    int64_t n_tiles;
};

// Submits iterations (shade, trace) in batches; after each batch the number of rays the batch's
// last shade kernel produced and the dispenser position are copied to pinned memory. The host looks
// at batch k-1 while batch k is already queued, so the GPU never waits for the host; it stops
// submitting once a batch ended with no ray in flight and no sample left (the batch queued behind it
// then runs over empty slots). The call returns when everything has been submitted AND that check
// has come back, i.e. it may block the calling thread for most of the render.
static int render_wavefront(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, float* d_accum,
                            unsigned long long* d_ray_count, bool counted, const AdaptivePass* adaptive = nullptr) {
    const WfPlan pl = wf_plan(c, s, counted, adaptive != nullptr);
    rtx::WfArgs a;
    const Tiles tiles = set_frame(a, s, p);
    const int64_t n_tiles = adaptive ? adaptive->n_tiles : (int64_t)tiles.x * tiles.y;
    const unsigned long long total = (unsigned long long)n_tiles * 32ull * (unsigned long long)p->spp_count;
    const int64_t slots = pool_slots_for(c, total);
    int rc = wf_prepare(c, slots);
    if (rc != RTX_OK) return rc;
    if (pl.trace2) CU(cudaFuncSetAttribute(pl.trace2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    if (pl.trace3) CU(cudaFuncSetAttribute(pl.trace3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    a.pool = pool_carve(c->d_pool, slots);
    a.n_slots = (int32_t)slots;
    a.total_items = total;
    a.next_item = c->d_next_item;
    a.adaptive = adaptive ? adaptive->args : rtx::AdaptiveArgs{};  // (ray ordering, the other user of this space, fills it per partition below)
    a.env = s->env;
    CU(cudaMemsetAsync(a.pool.bounce, 0xFF, (size_t)slots * 4, c->stream));  // every slot empty (-1)
    CU(cudaMemsetAsync(c->d_next_item, 0, sizeof(unsigned long long), c->stream));
    float4* acc = reinterpret_cast<float4*>(d_accum);
    const int batch = c->wf_batch;
    // P partitions of the pool, each driven on its own stream: the shade kernel of one partition (latency bound,
    // streams the pool) can share the SMs with the trace kernel of another (issue bound). Partition 0 runs on the
    // ctx stream; the others fork from it here and join it at the end.
    const int P = (slots >= (int64_t)c->wf_streams * 4 * rtx::kWfBlock) ? c->wf_streams : 1;
    const OrderLayout ol = order_layout(c->order_groups, P, slots);
    if (pl.order_pass) CU(cudaMemsetAsync(c->d_order, 0, (size_t)P * ol.part_words * 4, c->stream));
    std::vector<WfPart> parts((size_t)P);
    const int64_t per = slots / P / rtx::kWfBlock * rtx::kWfBlock;
    for (int q = 0; q < P; ++q) {
        WfPart& pt = parts[(size_t)q];
        const int64_t begin = (int64_t)q * per, count = q == P - 1 ? slots - begin : per;
        pt.a = a;
        pt.a.pool = pool_part(a.pool, begin);
        pt.a.n_slots = (int32_t)count;
        if (pl.order_pass) {
            uint32_t* w = (uint32_t*)c->d_order + (size_t)q * ol.part_words;
            uint8_t* per_slot = (uint8_t*)c->d_order + ol.slots_at;
            rtx::OrderArgs& o = pt.a.order;
            o.hist = w;
            o.offsets = w + ol.bins;
            o.done = w + 2 * ol.bins + 1;
            o.key_rank = (uint2*)per_slot + begin;
            o.order = (uint32_t*)(per_slot + (size_t)slots * 8) + begin;
            o.n_bins_padded = (int32_t)ol.bins;
            o.groups = c->order_groups;
            o.shift = 0;
            while (((s->n_records - 1) >> o.shift) >= o.groups) ++o.shift;
        }
        pt.sgrid = (unsigned)(count / rtx::kShadeBlock);
        pt.tgrid = pl.trace_grid(count, c->sm_count);
        pt.done = false;
        pt.stream = q == 0 ? c->stream : c->aux_streams[(size_t)q - 1];
    }
    if (P > 1) {
        CU(cudaEventRecord(c->fork_event, c->stream));
        for (int q = 1; q < P; ++q) CU(cudaStreamWaitEvent(parts[(size_t)q].stream, c->fork_event, 0));
    }
    size_t prof_used = 0;
    // every kProfStride-th iteration of partition 0 is bracketed (events between back-to-back launches cost ~10 %
    // when every launch has them); the accumulated times are scaled back up by the stride
    const int kProfStride = c->prof_stride;
    long long iteration = 0;
    bool prof_now = false;
    auto prof_mark = [&](void) -> cudaError_t {
        if (!prof_now) return cudaSuccess;
        if (prof_used == c->prof_events.size()) {
            cudaEvent_t e;
            cudaError_t err = cudaEventCreate(&e);
            if (err != cudaSuccess) return err;
            c->prof_events.push_back(e);
        }
        return cudaEventRecord(c->prof_events[prof_used++], c->stream);
    };
    int remaining = P;
    for (int k = 0; remaining > 0; ++k) {
        const int par = k & 1;
        for (int q = 0; q < P; ++q) {
            WfPart& pt = parts[(size_t)q];
            if (pt.done) continue;
            unsigned int* d_act = c->d_active + 2 * q + par;
            for (int it = 0; it < batch; ++it) {
                unsigned int* active = nullptr;
                if (it == batch - 1) {
                    active = d_act;
                    CU(cudaMemsetAsync(active, 0, sizeof(unsigned int), pt.stream));
                }
                prof_now = q == 0 && c->profiling && (iteration++ % kProfStride) == 0;
                CU(prof_mark());
                pl.launch_shade(pt, acc, active);
                CU(prof_mark());
                CU(prof_mark());
                pl.launch_trace(pt, d_ray_count);
                CU(prof_mark());
            }
            CU(cudaGetLastError());
            c->launches += pl.launches() * (unsigned long long)batch;
            // status of this batch -> pinned memory (active is 32-bit: widen on the host side)
            unsigned long long* hs = c->h_status + 4 * q + 2 * par;
            hs[0] = 0;
            CU(cudaMemcpyAsync(&hs[0], d_act, sizeof(unsigned int), cudaMemcpyDeviceToHost, pt.stream));
            CU(cudaMemcpyAsync(&hs[1], c->d_next_item, sizeof(unsigned long long), cudaMemcpyDeviceToHost, pt.stream));
            CU(cudaEventRecord(c->batch_done[2 * q + par], pt.stream));
        }
        if (k >= 1) {  // look at the previous batches while these run
            const int prev = par ^ 1;
            for (int q = 0; q < P; ++q) {
                WfPart& pt = parts[(size_t)q];
                if (pt.done) continue;
                CU(cudaEventSynchronize(c->batch_done[2 * q + prev]));
                const unsigned long long* hs = c->h_status + 4 * q + 2 * prev;
                if (c->debug_batches) std::fprintf(stderr, "[rtx] batch %d partition %d: %u rays written by its last shade pass, dispenser at %llu of %llu\n", k - 1, q, (unsigned int)hs[0], hs[1], total);
                if ((unsigned int)hs[0] == 0 && hs[1] >= total) { pt.done = true; --remaining; }
            }
        }
    }
    if (P > 1)
        for (int q = 1; q < P; ++q) {
            CU(cudaEventRecord(c->join_events[(size_t)q - 1], parts[(size_t)q].stream));
            CU(cudaStreamWaitEvent(c->stream, c->join_events[(size_t)q - 1], 0));
        }
    // the batch queued behind the one that ended dry runs over empty slots only; later calls on this
    // stream are ordered after it
    if (c->profiling && prof_used >= 4) {
        CU(cudaEventSynchronize(c->prof_events[prof_used - 1]));
        for (size_t q = 0; q + 3 < prof_used; q += 4) {
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, c->prof_events[q], c->prof_events[q + 1]));
            c->prof_shade_ms += ms * kProfStride;
            CU(cudaEventElapsedTime(&ms, c->prof_events[q + 2], c->prof_events[q + 3]));
            c->prof_trace_ms += ms * kProfStride;
            c->prof_iterations += kProfStride;
        }
    }
    return RTX_OK;
}

// ---- render -----------------------------------------------------------------
// The megakernel (RTX_MODE=mega): one persistent render_kernel launch over the frame.
static int render_mega(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, float* d_accum,
                       unsigned long long* d_ray_count, bool counted) {
    rtx::RenderArgs a;
    const Tiles tiles = set_frame(a, s, p);
    a.w_node = c->w_node; a.w_leaf = c->w_leaf; a.w_shade = c->w_shade;
    a.node_burst = c->node_burst;
    CU(cudaMemsetAsync(c->d_work_counter, 0, sizeof(unsigned int), c->stream));
    const auto kernel = counted ? rtx::render_kernel<true> : rtx::render_kernel<false>;
    // persistent grid: as many CTAs as fit, a whole number per SM
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, rtx::kRenderBlock, 0));
    if (per_sm < 1) per_sm = 1;
    int64_t n_tiles = (int64_t)tiles.x * tiles.y;
    int64_t grid = (int64_t)c->sm_count * per_sm;
    const int warps = rtx::kRenderBlock / 32;
    int64_t needed = (n_tiles + warps - 1) / warps;
    if (grid > needed) grid = needed;
    if (grid < 1) grid = 1;
    kernel<<<(unsigned)grid, rtx::kRenderBlock, 0, c->stream>>>(a, reinterpret_cast<float4*>(d_accum), d_ray_count, c->d_work_counter,
                                                               counted ? c->d_counters : nullptr);
    CU(cudaGetLastError());
    c->launches += 1;
    return RTX_OK;
}

// The render forms that have no environment-map variant refuse a scene that has a map.
static int env_refusal(const rtx_ctx* c, const rtx_scene* s, bool counted) {
    if (!s->env.texels) return RTX_OK;
    if (counted) return fail(RTX_ERR_UNSUPPORTED, "rtx_render_counted does not render scenes with an environment map");
    if (c->mode != 1 || c->shade_form < 2 || c->order_form != 0)
        return fail(RTX_ERR_UNSUPPORTED, "an environment map needs the wavefront driver with the default shade form and no ray ordering");
    return RTX_OK;
}

static int render_launch(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, float* d_accum,
                         unsigned long long* d_ray_count, bool counted) {
    if (!c || !s || !p || !d_accum) return fail(RTX_ERR_INVALID, "NULL argument");
    if (const int rc = env_refusal(c, s, counted); rc != RTX_OK) return rc;
    if (const int rc = check_frame(p, 0, p->spp_count < 0, "bad render parameters", "accumulator"); rc != RTX_OK) return rc;
    if (p->spp_count == 0) return RTX_OK;
    CU(cudaSetDevice(c->device));
    if (p->max_depth == 0) {  // color(.., depth = 0) is black (main.rs:27-29): only the sample counts move
        int n = p->width * p->height;
        rtx::add_black_samples_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(reinterpret_cast<float4*>(d_accum), n, (float)p->spp_count);
        c->launches += 1;
        CU(cudaGetLastError());
        return RTX_OK;
    }
    if (c->mode == 1) return render_wavefront(c, s, p, d_accum, d_ray_count, counted);
    return render_mega(c, s, p, d_accum, d_ray_count, counted);
}

extern "C" {

int rtx_render(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, float* d_accum, unsigned long long* d_ray_count) {
    if (c && c->async && s && p && d_accum) {
        if (const int rc = env_refusal(c, s, false); rc != RTX_OK) return rc;  // refused now, not from the next join
        const rtx_render_params params = *p;  // the caller's struct need not outlive the call
        {
            std::lock_guard<std::mutex> lock(c->mu);
            c->jobs.push_back([=]() { return render_launch(c, s, &params, d_accum, d_ray_count, false); });
            ++c->jobs_open;
        }
        c->cv.notify_all();
        return RTX_OK;
    }
    return render_launch(c, s, p, d_accum, d_ray_count, false);
}

int rtx_render_counted(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, float* d_accum, rtx_trace_stats* out) {
    if (!c || !out) return fail(RTX_ERR_INVALID, "NULL argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    unsigned long long* d_rays = nullptr;
    CU(cudaMalloc(&d_rays, sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(d_rays, 0, sizeof(unsigned long long), c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->d_counters, 0, sizeof(rtx::Counters), c->stream);
    int rc = e == cudaSuccess ? render_launch(c, s, p, d_accum, d_rays, true) : cuda_fail(e, "cudaMemset");
    rtx::Counters h;
    unsigned long long rays = 0;
    if (rc == RTX_OK) {
        e = cudaMemcpyAsync(&h, c->d_counters, sizeof(h), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&rays, d_rays, sizeof(rays), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "rtx_render_counted");
    }
    cudaFree(d_rays);
    if (rc != RTX_OK) return rc;
    trace_stats(h, rays, out);
    return RTX_OK;
}

// ---- adaptive sampling (adaptive.cuh) ----------------------------------------
int rtx_render_adaptive(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, const rtx_adaptive_params* ap,
                        float* d_accum, float* d_aux, rtx_adaptive_stats* stats) {
    if (!c || !s || !p || !ap || !d_accum || !d_aux) return fail(RTX_ERR_INVALID, "NULL argument");
    if (const int rc = check_frame(p, 0, (p->spp_begin & 1) != 0, "bad render parameters (spp_begin must be even)", nullptr); rc != RTX_OK)
        return rc;
    const int max_spp = p->spp_count;
    if (max_spp < 2 || (max_spp & 1) || max_spp > (1 << 24)) return fail(RTX_ERR_INVALID, "spp_count (max_spp) must be even, in [2, 2^24]");
    if (ap->min_spp < 2 || (ap->min_spp & 1) || ap->min_spp > max_spp) return fail(RTX_ERR_INVALID, "min_spp must be even, in [2, max_spp]");
    if (ap->step_spp < 2 || (ap->step_spp & 1)) return fail(RTX_ERR_INVALID, "step_spp must be even and >= 2");
    if (!(ap->threshold >= 0.0) || !std::isfinite(ap->threshold)) return fail(RTX_ERR_INVALID, "threshold must be finite and >= 0");
    if (c->mode != 1 || c->shade_form < 2 || c->order_form != 0)
        return fail(RTX_ERR_UNSUPPORTED, "adaptive sampling needs the wavefront driver with the default shade form and no ray ordering");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    const int w = p->width, h = p->height;
    const Tiles tiles = frame_tiles(w, h);
    const int n_tiles = tiles.x * tiles.y;
    // scratch: tile errors, flags, their scan, the list, the round's read-back, cub's temporary storage
    size_t scan_bytes = 0;
    CU(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, n_tiles, c->stream));
    const size_t words = ((size_t)n_tiles + 63) / 64 * 64 * 4;
    const size_t o_round = 4 * words, o_cub = o_round + 256;
    uint8_t* block = nullptr;
    CU(cudaMalloc(&block, o_cub + scan_bytes));
    float* d_err = (float*)block;
    uint32_t* d_flag = (uint32_t*)(block + words);
    uint32_t* d_pos = (uint32_t*)(block + 2 * words);
    uint32_t* d_list = (uint32_t*)(block + 3 * words);
    rtx::AdaptiveRound* d_round = (rtx::AdaptiveRound*)(block + o_round);
    float4* acc = reinterpret_cast<float4*>(d_accum);
    float4* aux = reinterpret_cast<float4*>(d_aux);
    rtx::AdaptiveRound cur{};
    rtx_adaptive_stats st{};
    st.tiles = n_tiles;
    // the tiles that keep sampling after the errors in `err` (all of them for nullptr): list + read-back
    auto select_tiles = [&](const float* err) -> int {
        const unsigned grid = (unsigned)((n_tiles + 255) / 256);
        CU(cudaMemsetAsync(d_round, 0, sizeof(rtx::AdaptiveRound), c->stream));
        rtx::adaptive_flag_kernel<<<grid, 256, 0, c->stream>>>(err, ap->threshold, tiles.x, tiles.y, tiles.inv_per_block_row, d_flag);
        size_t cb = scan_bytes;
        CU(cub::DeviceScan::ExclusiveSum(block + o_cub, cb, d_flag, d_pos, n_tiles, c->stream));
        rtx::adaptive_scatter_kernel<<<grid, 256, 0, c->stream>>>(d_flag, d_pos, w, h, tiles.x, tiles.y, tiles.inv_per_block_row, d_list, d_round);
        c->launches += 4;  // (cub's scan counts as two)
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(&cur, d_round, sizeof(cur), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        return RTX_OK;
    };
    // RTX_DEBUG_ADAPTIVE=1: one stderr line per round (the render is then synchronised before the decision, to time it)
    const bool debug = std::getenv("RTX_DEBUG_ADAPTIVE") != nullptr;
    auto ms_since = [](std::chrono::steady_clock::time_point t) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
    };
    auto run = [&]() -> int {
        CU(cudaMemsetAsync(d_accum, 0, (size_t)w * h * 16, c->stream));
        CU(cudaMemsetAsync(d_aux, 0, (size_t)w * h * 16, c->stream));
        int rc = select_tiles(nullptr);
        if (rc != RTX_OK) return rc;
        int n = 0, spp = ap->min_spp;
        for (;;) {
            const auto t_round = std::chrono::steady_clock::now();
            double render_ms = 0.0;
            if (p->max_depth == 0) {  // color(.., depth = 0) is black (main.rs:27-29): only the sample counts move
                rtx::adaptive_black_kernel<<<(unsigned)((cur.tiles * 32 + 127) / 128), 128, 0, c->stream>>>(
                    d_list, (int)cur.tiles, w, h, tiles.x, tiles.y, tiles.inv_per_block_row, p->spp_begin + n, spp, acc, aux);
                c->launches += 1;
                CU(cudaGetLastError());
            } else {
                rtx_render_params rp = *p;
                rp.spp_begin = p->spp_begin + n;
                rp.spp_count = spp;
                const AdaptivePass pass{{d_list, aux}, (int64_t)cur.tiles};
                rc = render_wavefront(c, s, &rp, d_accum, nullptr, false, &pass);
                if (rc != RTX_OK) return rc;
            }
            if (debug) {
                CU(cudaStreamSynchronize(c->stream));
                render_ms = ms_since(t_round);
            }
            n += spp;
            ++st.rounds;
            st.path_samples += (int64_t)cur.pixels * spp;
            const unsigned long long before = cur.tiles;
            if (n == max_spp) {
                st.tiles_at_max = (int32_t)cur.tiles;
                if (debug) std::fprintf(stderr, "[rtx] adaptive round %d: %llu tiles x %d spp (n = %d), %llu path samples, render %.3f ms\n",
                                        st.rounds - 1, before, spp, n, cur.pixels * (unsigned long long)spp, render_ms);
                break;
            }
            rtx::adaptive_error_kernel<<<(unsigned)(((int64_t)n_tiles * 32 + rtx::kAdaptiveBlock - 1) / rtx::kAdaptiveBlock),
                                         rtx::kAdaptiveBlock, 0, c->stream>>>(acc, aux, w, h, tiles.x, n_tiles, d_err);
            c->launches += 1;
            CU(cudaGetLastError());
            const unsigned long long pixels = cur.pixels;
            rc = select_tiles(d_err);
            if (rc != RTX_OK) return rc;
            if (debug) std::fprintf(stderr, "[rtx] adaptive round %d: %llu tiles x %d spp (n = %d), %llu path samples, render %.3f ms, decision %.3f ms\n",
                                    st.rounds - 1, before, spp, n, pixels * (unsigned long long)spp, render_ms, ms_since(t_round) - render_ms);
            st.tiles_converged += (int32_t)(before - cur.tiles);
            if (cur.tiles == 0) break;
            spp = std::min(ap->step_spp, max_spp - n);
        }
        CU(cudaStreamSynchronize(c->stream));
        return RTX_OK;
    };
    const int rc = run();
    cudaStreamSynchronize(c->stream);  // (nothing may still use the scratch block when it is freed)
    cudaFree(block);
    if (rc == RTX_OK && stats) *stats = st;
    return rc;
}

int rtx_adaptive_error(rtx_ctx* c, const float* d_accum, const float* d_aux, int32_t width, int32_t height, float* d_tile_error) {
    if (!c || !d_accum || !d_aux || !d_tile_error || width <= 0 || height <= 0) return fail(RTX_ERR_INVALID, "bad argument");
    if ((int64_t)width * height > 0x7fffffff) return fail(RTX_ERR_INVALID, "image too large");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    const Tiles tiles = frame_tiles(width, height);
    const int64_t n_tiles = (int64_t)tiles.x * tiles.y;
    rtx::adaptive_error_kernel<<<(unsigned)((n_tiles * 32 + rtx::kAdaptiveBlock - 1) / rtx::kAdaptiveBlock), rtx::kAdaptiveBlock, 0, c->stream>>>(
        reinterpret_cast<const float4*>(d_accum), reinterpret_cast<const float4*>(d_aux), width, height, tiles.x, (int)n_tiles, d_tile_error);
    c->launches += 1;
    CU(cudaGetLastError());
    return RTX_OK;
}

// ---- feature buffers (aov.cuh) -------------------------------------------------
int rtx_render_aov(rtx_ctx* c, const rtx_scene* s, const rtx_render_params* p, float* d_albedo, float* d_normal,
                   float* d_depth) {
    if (!c || !s || !p) return fail(RTX_ERR_INVALID, "NULL argument");
    if (!d_albedo && !d_normal && !d_depth) return fail(RTX_ERR_INVALID, "no feature buffer given");
    if (const int rc = check_frame(p, 1, p->spp_count < 0, "bad render parameters (the feature pass needs max_depth >= 1)", "buffers"); rc != RTX_OK)
        return rc;
    JOIN(c);
    if (p->spp_count == 0) return RTX_OK;
    CU(cudaSetDevice(c->device));
    rtx::AovArgs a;
    const Tiles tiles = set_frame(a, s, p);
    a.albedo = reinterpret_cast<float4*>(d_albedo);
    a.normal = reinterpret_cast<float4*>(d_normal);
    a.depth = reinterpret_cast<float2*>(d_depth);
    const int64_t n_tiles = (int64_t)tiles.x * tiles.y;
    const int64_t grid = (n_tiles * 32 + rtx::kAovBlock - 1) / rtx::kAovBlock;
    if (s->env.texels) rtx::aov_env_kernel<<<(unsigned)grid, rtx::kAovBlock, 0, c->stream>>>(a, s->env);
    else rtx::aov_kernel<<<(unsigned)grid, rtx::kAovBlock, 0, c->stream>>>(a);
    c->launches += 1;
    CU(cudaGetLastError());
    return RTX_OK;
}

// ---- denoiser (denoise.cuh) ----------------------------------------------------
int rtx_denoise(rtx_ctx* c, const float* d_accum, const float* d_half, const float* d_albedo, const float* d_normal,
                int32_t width, int32_t height, const rtx_denoise_params* params, float* d_out) {
    if (!c || !d_accum || !d_half || !d_albedo || !d_normal || !d_out) return fail(RTX_ERR_INVALID, "NULL argument");
    for (const float* b : {d_accum, d_half, d_albedo, d_normal, (const float*)d_out})
        if ((uintptr_t)b % 16 != 0) return fail(RTX_ERR_INVALID, "every buffer must be 16-byte aligned (float4)");
    if (width <= 0 || height <= 0) return fail(RTX_ERR_INVALID, "bad image size");
    if ((int64_t)width * height > 0x7fffffff) return fail(RTX_ERR_INVALID, "image too large");
    const rtx_denoise_params p = params ? *params : rtx_denoise_params{5, 0.25f, 0.1f, 8.f};
    if (p.iterations < 1 || p.iterations > 10) return fail(RTX_ERR_INVALID, "iterations must lie in [1, 10]");
    for (float sg : {p.sigma_normal, p.sigma_albedo, p.sigma_luminance})
        if (!(sg > 0.f) || !std::isfinite(sg)) return fail(RTX_ERR_INVALID, "every sigma must be > 0 and finite");
    // the kernels multiply by 1 / sigma^2 in fp32: an infinite factor would turn the centre tap's 0 difference into NaN
    const double inv_sn2 = 1.0 / ((double)p.sigma_normal * p.sigma_normal), inv_sa2 = 1.0 / ((double)p.sigma_albedo * p.sigma_albedo);
    if (!(inv_sn2 <= FLT_MAX) || !(inv_sa2 <= FLT_MAX))
        return fail(RTX_ERR_INVALID, "sigma_normal and sigma_albedo must be at least about 5.4e-20 (1 / sigma^2 finite in fp32)");
    const size_t n = (size_t)width * height, bytes = n * sizeof(float4);
    const uintptr_t o0 = (uintptr_t)d_out, o1 = o0 + bytes;
    for (const float* in : {d_accum, d_half, d_albedo, d_normal}) {
        const uintptr_t i0 = (uintptr_t)in;
        if (o0 < i0 + bytes && i0 < o1) return fail(RTX_ERR_INVALID, "d_out overlaps an input buffer");
    }
    JOIN(c);
    CU(cudaSetDevice(c->device));
    const size_t need = n * (sizeof(float4) + sizeof(float2) + 2 * sizeof(float4));
    if (c->denoise_bytes < need) {
        cudaFree(c->d_denoise);  // (waits for the passes of an earlier call that still read it)
        c->d_denoise = nullptr;
        c->denoise_bytes = 0;
        CU(cudaMalloc(&c->d_denoise, need));
        c->denoise_bytes = need;
    }
    float4* feat0 = reinterpret_cast<float4*>(c->d_denoise);
    float4* ev0 = feat0 + n;
    float4* ev1 = ev0 + n;
    float2* feat1 = reinterpret_cast<float2*>(ev1 + n);
    const dim3 block(rtx::kDenoiseBX, rtx::kDenoiseBY);
    const int tiles_x = (int)(((int64_t)width + rtx::kDenoiseBX - 1) / rtx::kDenoiseBX);
    const unsigned grid = (unsigned)(tiles_x * (((int64_t)height + rtx::kDenoiseBY - 1) / rtx::kDenoiseBY));  // < 2^29 tiles for < 2^31 pixels
    rtx::denoise_prepass_kernel<<<grid, block, 0, c->stream>>>(
        reinterpret_cast<const float4*>(d_accum), reinterpret_cast<const float4*>(d_half),
        reinterpret_cast<const float4*>(d_albedo), reinterpret_cast<const float4*>(d_normal), width, height, tiles_x, feat0,
        feat1, ev0);
    CU(cudaGetLastError());
    rtx::DenoisePass a;
    a.feat0 = feat0;
    a.feat1 = feat1;
    a.width = width;
    a.height = height;
    a.tiles_x = tiles_x;
    a.inv_sn2 = (float)inv_sn2;
    a.inv_sa2 = (float)inv_sa2;
    a.sigma_l = p.sigma_luminance;
    for (int i = 0; i < p.iterations; ++i) {
        a.step = 1 << i;
        a.ev_in = (i & 1) ? ev1 : ev0;
        a.ev_out = (i & 1) ? ev0 : ev1;
        a.out = i == p.iterations - 1 ? reinterpret_cast<float4*>(d_out) : nullptr;
        rtx::denoise_atrous_kernel<<<grid, block, 0, c->stream>>>(a);
        CU(cudaGetLastError());
    }
    c->launches += 1 + p.iterations;
    return RTX_OK;
}

int rtx_tonemap_rgba8(rtx_ctx* c, const float* d_accum, int32_t width, int32_t height, uint8_t* out, int out_on_device) {
    if (!c || !d_accum || !out || width <= 0 || height <= 0) return fail(RTX_ERR_INVALID, "bad argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    int n = width * height;
    uchar4* d_out = (uchar4*)out;
    if (!out_on_device) CU(cudaMalloc(&d_out, (size_t)n * 4));
    rtx::tonemap_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(reinterpret_cast<const float4*>(d_accum), n, d_out);
    c->launches += 1;
    cudaError_t e = cudaGetLastError();
    if (!out_on_device) {
        if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, (size_t)n * 4, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        cudaFree(d_out);
    }
    if (e != cudaSuccess) return cuda_fail(e, "rtx_tonemap_rgba8");
    return RTX_OK;
}

// Makes `p` (a device pointer, possibly on another device of this process) loadable from ctx's device: enables peer
// access, or — when the two devices cannot map each other — stages a copy in `scratch` (cudaMemcpyPeerAsync).
static int map_or_stage_peer(rtx_ctx* c, const float* p, size_t bytes, std::vector<void*>& scratch, const float** out) {
    *out = p;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeDevice || at.device == c->device) {
        cudaGetLastError();  // IPC-opened pointers are already mapped by rtx_ipc_open; local ones need nothing
        return RTX_OK;
    }
    int can = 0;
    cudaDeviceCanAccessPeer(&can, c->device, at.device);
    if (can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
        if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return RTX_OK; }
    }
    cudaGetLastError();
    void* tmp = nullptr;
    CU(cudaMalloc(&tmp, bytes));
    scratch.push_back(tmp);
    CU(cudaMemcpyPeerAsync(tmp, c->device, p, at.device, bytes, c->stream));
    *out = (const float*)tmp;
    return RTX_OK;
}

int rtx_reduce_tonemap_peers(rtx_ctx* c, float* d_accum, const float* const* d_peer_accums, int32_t n_peers, int32_t width,
                             int32_t height, uint8_t* d_rgba8) {
    if (!c || !d_accum || !d_rgba8 || width <= 0 || height <= 0 || n_peers < 0 || (n_peers > 0 && !d_peer_accums))
        return fail(RTX_ERR_INVALID, "bad argument");
    if (n_peers > rtx::kMaxPeers) return fail(RTX_ERR_UNSUPPORTED, "too many peers");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    const int n = width * height;
    rtx::PeerList pl;
    pl.n = n_peers;
    std::vector<void*> scratch;
    for (int i = 0; i < n_peers; ++i) {
        const float* q = nullptr;
        int rc = map_or_stage_peer(c, d_peer_accums[i], (size_t)n * 16, scratch, &q);
        if (rc != RTX_OK) { for (void* t : scratch) cudaFree(t); return rc; }
        pl.p[i] = reinterpret_cast<const float4*>(q);
    }
    rtx::reduce_tonemap_peers_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(reinterpret_cast<float4*>(d_accum), pl, n,
                                                                            reinterpret_cast<uchar4*>(d_rgba8));
    cudaError_t e = cudaGetLastError();
    if (!scratch.empty()) {  // (the staged path is the slow path: finish before the copies go away)
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        for (void* t : scratch) cudaFree(t);
    }
    if (e != cudaSuccess) return cuda_fail(e, "reduce_tonemap_peers_kernel");
    c->launches += 1;
    return RTX_OK;
}

int rtx_reduce_tonemap_slice(rtx_ctx* c, const float* const* d_accums, int32_t n_ranks, int32_t rank, int32_t width, int32_t height,
                             uint8_t* d_rgba8_root) {
    if (!c || !d_accums || !d_rgba8_root || width <= 0 || height <= 0 || n_ranks < 1 || rank < 0 || rank >= n_ranks)
        return fail(RTX_ERR_INVALID, "bad argument");
    if (n_ranks > rtx::kMaxPeers) return fail(RTX_ERR_UNSUPPORTED, "too many ranks");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    const long long n = (long long)width * height;
    const int first = (int)(n * rank / n_ranks), count = (int)(n * (rank + 1) / n_ranks) - first;
    rtx::PeerList pl;
    pl.n = n_ranks;
    for (int i = 0; i < n_ranks; ++i) {
        if (!d_accums[i]) return fail(RTX_ERR_INVALID, "NULL accumulator");
        pl.p[i] = reinterpret_cast<const float4*>(d_accums[i]);
        cudaPointerAttributes at;  // same-process peers: map the other device (IPC-opened pointers already are)
        if (cudaPointerGetAttributes(&at, d_accums[i]) == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device != c->device) {
            cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
        }
        cudaGetLastError();
    }
    if (count > 0) {
        rtx::reduce_tonemap_slice_kernel<<<(count + 255) / 256, 256, 0, c->stream>>>(pl, first, count, reinterpret_cast<uchar4*>(d_rgba8_root));
        CU(cudaGetLastError());
        c->launches += 1;
    }
    return RTX_OK;
}

// ---- NCCL combine (libnccl.so.2 opened on demand: the library itself does not link against it) ----
namespace {
struct NcclId { char internal[128]; };
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
};
NcclApi& nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (!api.lib) return;
        api.GetUniqueId = (int (*)(NcclId*))dlsym(api.lib, "ncclGetUniqueId");
        api.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(api.lib, "ncclCommInitRank");
        api.CommDestroy = (int (*)(void*))dlsym(api.lib, "ncclCommDestroy");
        api.Reduce = (int (*)(const void*, void*, size_t, int, int, int, void*, cudaStream_t))dlsym(api.lib, "ncclReduce");
        api.GetErrorString = (const char* (*)(int))dlsym(api.lib, "ncclGetErrorString");
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.Reduce && api.GetErrorString;
    });
    return api;
}
int nccl_fail(int res, const char* what) {
    g_err = std::string(what) + ": " + (nccl().GetErrorString ? nccl().GetErrorString(res) : "NCCL error");
    return RTX_ERR_CUDA;
}
}  // namespace

struct rtx_comm {
    void* comm = nullptr;  // ncclComm_t
    bool owned = false;
};

int rtx_comm_unique_id(uint8_t id_out[128]) {
    if (!id_out) return fail(RTX_ERR_INVALID, "id_out is NULL");
    if (!nccl().ok) return fail(RTX_ERR_UNSUPPORTED, "libnccl.so.2 not found");
    NcclId id;
    int r = nccl().GetUniqueId(&id);
    if (r != 0) return nccl_fail(r, "ncclGetUniqueId");
    std::memcpy(id_out, &id, 128);
    return RTX_OK;
}
int rtx_comm_create(rtx_ctx* c, int32_t n_ranks, int32_t rank, const uint8_t id[128], rtx_comm** out) {
    if (!c || !id || !out || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(RTX_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (!nccl().ok) return fail(RTX_ERR_UNSUPPORTED, "libnccl.so.2 not found");
    CU(cudaSetDevice(c->device));
    NcclId nid;
    std::memcpy(&nid, id, 128);
    void* comm = nullptr;
    int r = nccl().CommInitRank(&comm, n_ranks, nid, rank);
    if (r != 0) return nccl_fail(r, "ncclCommInitRank");
    rtx_comm* k = new (std::nothrow) rtx_comm();
    if (!k) { nccl().CommDestroy(comm); return fail(RTX_ERR_NOMEM, "out of host memory"); }
    k->comm = comm;
    k->owned = true;
    *out = k;
    return RTX_OK;
}
int rtx_comm_wrap(void* nccl_comm, rtx_comm** out) {
    if (!nccl_comm || !out) return fail(RTX_ERR_INVALID, "NULL argument");
    if (!nccl().ok) return fail(RTX_ERR_UNSUPPORTED, "libnccl.so.2 not found");
    rtx_comm* k = new (std::nothrow) rtx_comm();
    if (!k) return fail(RTX_ERR_NOMEM, "out of host memory");
    k->comm = nccl_comm;
    k->owned = false;
    *out = k;
    return RTX_OK;
}
int rtx_comm_destroy(rtx_comm* k) {
    if (!k) return RTX_OK;
    if (k->owned && k->comm && nccl().ok) nccl().CommDestroy(k->comm);
    delete k;
    return RTX_OK;
}
int rtx_accum_reduce(rtx_ctx* c, rtx_comm* k, float* d_accum, int32_t width, int32_t height, int32_t root) {
    if (!c || !k || !k->comm || !d_accum || width <= 0 || height <= 0 || root < 0) return fail(RTX_ERR_INVALID, "bad argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    const size_t count = (size_t)width * (size_t)height * 4;
    int r = nccl().Reduce(d_accum, d_accum, count, /*ncclFloat32*/ 7, /*ncclSum*/ 0, root, k->comm, c->stream);
    if (r != 0) return nccl_fail(r, "ncclReduce");
    return RTX_OK;
}

// ---- memory / IPC helpers ------------------------------------------------------
int rtx_malloc(rtx_ctx* c, size_t bytes, void** out) {
    if (!c || !out) return fail(RTX_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(c->device));
    CU(cudaMalloc(out, bytes));
    return RTX_OK;
}
int rtx_free(rtx_ctx* c, void* ptr) {
    if (!c) return fail(RTX_ERR_INVALID, "ctx is NULL");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaFree(ptr));
    return RTX_OK;
}
int rtx_memset_zero(rtx_ctx* c, void* ptr, size_t bytes) {
    if (!c || !ptr) return fail(RTX_ERR_INVALID, "NULL argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaMemsetAsync(ptr, 0, bytes, c->stream));
    return RTX_OK;
}
int rtx_memcpy_h2d(rtx_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c || !dst || !src) return fail(RTX_ERR_INVALID, "NULL argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return RTX_OK;
}
int rtx_memcpy_d2h(rtx_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c || !dst || !src) return fail(RTX_ERR_INVALID, "NULL argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return RTX_OK;
}
int rtx_memcpy_d2d(rtx_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c || !dst || !src) return fail(RTX_ERR_INVALID, "NULL argument");
    JOIN(c);
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
    return RTX_OK;
}
int rtx_ipc_export(rtx_ctx* c, void* d_ptr, uint8_t handle_out[64]) {
    if (!c || !d_ptr || !handle_out) return fail(RTX_ERR_INVALID, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, d_ptr));
    std::memcpy(handle_out, &h, 64);
    return RTX_OK;
}
int rtx_ipc_open(rtx_ctx* c, const uint8_t handle[64], void** d_ptr_out) {
    if (!c || !handle || !d_ptr_out) return fail(RTX_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    CU(cudaIpcOpenMemHandle(d_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return RTX_OK;
}
int rtx_ipc_close(rtx_ctx* c, void* d_ptr) {
    if (!c || !d_ptr) return fail(RTX_ERR_INVALID, "NULL argument");
    CU(cudaSetDevice(c->device));
    CU(cudaIpcCloseMemHandle(d_ptr));
    return RTX_OK;
}

// ---- host-side mirrors (no GPU needed) -----------------------------------------
int rtx_builtin_scene_defaults(int scene_number, rtx_scene_defaults* out) {
    if (!out) return fail(RTX_ERR_INVALID, "out is NULL");
    rttnw::SceneDefaults d;
    if (!rttnw::builtin_scene_defaults(scene_number, d)) return fail(RTX_ERR_INVALID, "There is no scene " + std::to_string(scene_number));
    out->width = d.width; out->height = d.height; out->samples = d.samples; out->max_depth = d.max_depth; out->name = d.name;
    return RTX_OK;
}

struct DescBox {  // rtx_scene_desc must be the first member: the public pointer is &box->desc
    rtx_scene_desc desc;
    rttnw::SceneBuilder builder;
};

int rtx_builtin_scene(int scene_number, uint64_t seed, const char* earth_png_path, rtx_scene_desc** out) {
    if (!out) return fail(RTX_ERR_INVALID, "out is NULL");
    *out = nullptr;
    DescBox* box = new (std::nothrow) DescBox();
    if (!box) return fail(RTX_ERR_NOMEM, "out of host memory");
    if (!rttnw::builtin_scene(scene_number, seed, earth_png_path, box->builder)) {
        delete box;
        return fail(RTX_ERR_INVALID, "There is no scene " + std::to_string(scene_number));
    }
    box->desc = box->builder.desc;
    *out = &box->desc;
    return RTX_OK;
}
int rtx_scene_desc_free(rtx_scene_desc* desc) {
    if (desc) delete reinterpret_cast<DescBox*>(desc);
    return RTX_OK;
}

int rtx_flatten_check(const rtx_scene_desc* desc, int32_t* n_bvh_nodes, int32_t* n_records, int32_t* n_prim_ids) {
    if (!desc) return fail(RTX_ERR_INVALID, "desc is NULL");
    rtx::FlatScene fs;
    std::string err;
    if (!rtx::flatten_scene(*desc, fs, err, false, true)) return fail(RTX_ERR_INVALID, "scene description: " + err);  // with the 4-wide copy, to check it too
    if (!rtx::check_flat_scene(fs, err)) return fail(RTX_ERR_INVALID, "flattened scene invariant violated: " + err);
    if (n_bvh_nodes) *n_bvh_nodes = (int32_t)fs.nodes.size();
    if (n_records) *n_records = (int32_t)fs.records.size();
    if (n_prim_ids) *n_prim_ids = fs.n_prims;
    return RTX_OK;
}

int rtx_png_read_rgba8(const char* path, int32_t* width, int32_t* height, uint8_t** rgba_out) {
    if (!path || !width || !height || !rgba_out) return fail(RTX_ERR_INVALID, "NULL argument");
    std::vector<uint8_t> px;
    std::string err;
    int w = 0, h = 0;
    if (!rttnw::png_read_rgba8(path, w, h, px, err)) return fail(RTX_ERR_IO, err);
    uint8_t* buf = (uint8_t*)std::malloc(px.size());
    if (!buf) return fail(RTX_ERR_NOMEM, "out of host memory");
    std::memcpy(buf, px.data(), px.size());
    *width = w; *height = h; *rgba_out = buf;
    return RTX_OK;
}
int rtx_png_write_rgba8(const char* path, int32_t width, int32_t height, const uint8_t* rgba) {
    if (!path || !rgba) return fail(RTX_ERR_INVALID, "NULL argument");
    std::string err;
    if (!rttnw::png_write_rgba8(path, width, height, rgba, err)) return fail(RTX_ERR_IO, err);
    return RTX_OK;
}
int rtx_pfm_write(const char* path, int32_t width, int32_t height, int32_t channels, const float* data) {
    if (!path || !data) return fail(RTX_ERR_INVALID, "NULL argument");
    if (width <= 0 || height <= 0 || (channels != 1 && channels != 3)) return fail(RTX_ERR_INVALID, "bad PFM size or channel count (1 or 3)");
    std::string err;
    if (!rttnw::pfm_write(path, width, height, channels, data, err)) return fail(RTX_ERR_IO, err);
    return RTX_OK;
}
// A reader's result as a malloc'd buffer the caller frees with rtx_buffer_free.
static int hand_over(const std::vector<float>& px, float** out) {
    float* buf = (float*)std::malloc(px.size() * sizeof(float));
    if (!buf) return fail(RTX_ERR_NOMEM, "out of host memory");
    std::memcpy(buf, px.data(), px.size() * sizeof(float));
    *out = buf;
    return RTX_OK;
}
int rtx_pfm_read(const char* path, int32_t* width, int32_t* height, int32_t* channels, float** data) {
    if (!path || !width || !height || !channels || !data) return fail(RTX_ERR_INVALID, "NULL argument");
    std::vector<float> px;
    std::string err;
    int w = 0, h = 0, ch = 0;
    if (const int rc = rttnw::pfm_read(path, w, h, ch, px, err); rc != RTX_OK) return fail(rc, err);
    if (const int rc = hand_over(px, data); rc != RTX_OK) return rc;
    *width = w; *height = h; *channels = ch;
    return RTX_OK;
}
int rtx_hdr_read(const char* path, int32_t* width, int32_t* height, float** rgb) {
    if (!path || !width || !height || !rgb) return fail(RTX_ERR_INVALID, "NULL argument");
    std::vector<float> px;
    std::string err;
    int w = 0, h = 0;
    if (const int rc = rttnw::hdr_read(path, w, h, px, err); rc != RTX_OK) return fail(rc, err);
    if (const int rc = hand_over(px, rgb); rc != RTX_OK) return rc;
    *width = w; *height = h;
    return RTX_OK;
}
int rtx_buffer_free(void* p) {
    std::free(p);
    return RTX_OK;
}

}  // extern "C"
