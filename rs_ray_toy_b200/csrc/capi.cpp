// C ABI of librrt_sm100.so (include/rrt.h): context, scene assembly, and the batch
// intersect entry points that stand where Scene::intersect / intersect_p
// (src/scene.rs:69-80) stand in the reference.  No exception leaves this file.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "aggregate.hpp"
#include "bvh_lbvh.hpp"
#include "bvh_hlbvh.hpp"
#include "halton.cuh"
#include "literal.hpp"
#include "mesh_update.hpp"
#include "png_min.hpp"
#include "rays_f32.cuh"
#include "rays_f32.hpp"
#include "render.hpp"
#include "scene_json.hpp"
#include "stratified.cuh"
#include "surface.hpp"
#include "rrt_test.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}
int cuda_fail(const char* what, cudaError_t e) {
    g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return RRT_ERR_CUDA;
}
#define CAPI_CUDA(call)                                   \
    do {                                                  \
        cudaError_t e_ = (call);                          \
        if (e_ != cudaSuccess) return cuda_fail(#call, e_); \
    } while (0)

constexpr int kSlots = 4;  // pipeline depth of the host-buffer calls: with three, the small chunks that end a batch wait for the
                           // slot of a full chunk three places earlier (profiles/r2_e2e_trace.txt); 96 MiB of device memory each
// rays per pipeline slot (64 B each); RRT_HOST_CHUNK overrides for experiments
uint64_t chunk_rays() {
    static const uint64_t v = [] {
        const char* e = std::getenv("RRT_HOST_CHUNK");
        uint64_t c = e ? std::strtoull(e, nullptr, 10) : (1ull << 20);
        return c < 4096 ? 4096 : c;
    }();
    return v;
}
#define kChunkRays (chunk_rays())
// rays per pipeline slot of the surface calls: a quarter of the chunk, so that the slots' 336-byte records take 84 MiB
// each instead of 336 MiB.  Their chunks are bound by the records' D2H, not by the walk, so a smaller chunk costs nothing
// that the four-slot pipeline does not hide.
uint64_t surface_chunk_rays() { return kChunkRays / 4; }
// The pipeline's fill (first H2D, nothing to trace yet) and drain (last kernel + D2H, nothing left to upload) are each one
// chunk long, so the chunks at both ends of a batch are small and double towards the middle: 128 Ki, 128 Ki, 256 Ki, 512 Ki,
// 1 Mi ... 1 Mi, 512 Ki, 256 Ki, 128 Ki.  Measured on a 16 Mi-ray batch: 701 -> 726 Mrays/s (profiles/r2_e2e_taper.txt); the
// link's own floor for 1 GiB up + 0.5 GiB down at once is 20.5 ms = 819 Mrays/s (profiles/r2_pcie_probe.txt), and the
// uploads run at 49.5 GB/s while hits stream down (55.5 GB/s alone): 21.7 ms + the last chunk's walk (0.5 ms: a batch of
// any size takes that long) is what is left (profiles/r2_e2e_trace.txt).  RRT_HOST_TAPER=0: off.
uint64_t tapered_chunk(uint64_t done, uint64_t n, uint64_t full) {
    static const bool taper = [] {
        const char* e = std::getenv("RRT_HOST_TAPER");
        return !(e && e[0] == '0');
    }();
    const uint64_t left = n - done;
    uint64_t c = full;
    if (taper) {
        const uint64_t floor_c = full >> 3 ? full >> 3 : 1;
        const uint64_t up = done > floor_c ? done : floor_c;               // doubling from the start
        const uint64_t down = left / 2 > floor_c ? left / 2 : floor_c;     // halving towards the end
        c = up < c ? up : c;
        c = down < c ? down : c;
    }
    return left < c ? left : c;
}

struct Slot {
    cudaStream_t stream = nullptr;
    rrt_ray* d_rays = nullptr;
    void* d_out = nullptr;  // rrt_hit[kChunkRays] (also large enough for the any-hit bytes)
    void* d_f32 = nullptr;  // fp32 calls only: the chunk's rrt_ray_f32, then its rrt_hit_f32 (the rays are dead by then)
    void* d_surf = nullptr; // surface calls only: the chunk's rrt_surface records
};

}  // namespace

struct rrt_ctx {
    int device = 0;
    std::atomic<uint64_t> launches{0};
    std::mutex host_path_mutex;  // the staging slots are shared by host-buffer calls
    Slot slots[kSlots];
    bool slots_ready = false;

    int ensure_slots() {
        if (slots_ready) return RRT_OK;
        CAPI_CUDA(cudaSetDevice(device));
        for (auto& s : slots) {
            CAPI_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
            CAPI_CUDA(cudaMalloc(&s.d_rays, kChunkRays * sizeof(rrt_ray)));
            CAPI_CUDA(cudaMalloc(&s.d_out, kChunkRays * sizeof(rrt_hit)));
        }
        slots_ready = true;
        return RRT_OK;
    }
    // added by the first fp32 call, so that callers of the f64 entries pay no memory for them
    int ensure_f32_slots() {
        for (auto& s : slots)
            if (!s.d_f32) CAPI_CUDA(cudaMalloc(&s.d_f32, kChunkRays * sizeof(rrt_ray_f32)));
        return RRT_OK;
    }
    // likewise added by the first surface call
    int ensure_surface_slots() {
        for (auto& s : slots)
            if (!s.d_surf) CAPI_CUDA(cudaMalloc(&s.d_surf, surface_chunk_rays() * sizeof(rrt_surface)));
        return RRT_OK;
    }
    ~rrt_ctx() {
        cudaSetDevice(device);
        for (auto& s : slots) {
            if (s.d_rays) cudaFree(s.d_rays);
            if (s.d_out) cudaFree(s.d_out);
            if (s.d_f32) cudaFree(s.d_f32);
            if (s.d_surf) cudaFree(s.d_surf);
            if (s.stream) cudaStreamDestroy(s.stream);
        }
    }
};

struct rrt_scene {
    rrt_ctx* ctx = nullptr;
    rrt::HostScene host;
    std::vector<rrt_material> materials;
    std::vector<rrt_light> lights;
    std::vector<rrt_texture> textures;
    std::vector<int32_t> material_slots;  // RRT_MATERIAL_SLOTS per material, or empty
    rrt::SceneExtras extras;              // images, Scene::infinite_lights
    std::unique_ptr<rrt::RayTracer> agg;  // DeviceAggregate (Tier F) or LiteralAggregate (Tier L)
    bool committed = false;
    uint32_t build_flags = 0;
    uint32_t max_prims_in_node = 4;
    std::atomic<int> live_renders{0};  // integrators made over this scene (they hold its aggregate and shading tables)

    // The device entries that run more than the walk (rrt_intersect_f32_device, rrt_intersect_p_f32_device,
    // rrt_intersect_surface_device): the promoted rays and / or the f64 hits of a batch, one set per calling stream, grown
    // to the largest batch seen there; past kMaxScratch streams the first set is shared, ordered by its event (the policy
    // of DeviceAggregate's workspaces).  acquire_scratch / release_scratch below.
    struct StreamScratch {
        rrt_ray* d_rays = nullptr;
        rrt_hit* d_hits = nullptr;
        uint64_t ray_capacity = 0, hit_capacity = 0;
        cudaEvent_t last_use = nullptr;
        bool used = false;
        void* last_stream = nullptr;
    };
    static constexpr size_t kMaxScratch = 8;
    mutable std::mutex scratch_mutex;
    mutable std::map<void*, StreamScratch> scratch;

    // the surface pass's shape tables (Tier F), uploaded by the first surface call; the literal tier reads its
    // aggregate's own
    mutable std::mutex surface_mutex;
    mutable rrt::SurfaceTables* surface_tables = nullptr;

    // the primitives baked on the device, made by the first rrt_scene_update_mesh after a commit, dropped by
    // rrt_scene_update_instances (its runs hold the instance transforms)
    std::unique_ptr<rrt::MeshImage> mesh_image;

    ~rrt_scene() {
        for (auto& kv : scratch) {
            StreamScratch& w = kv.second;
            if (w.last_use) {
                cudaEventSynchronize(w.last_use);
                cudaEventDestroy(w.last_use);
            }
            if (w.d_rays) cudaFree(w.d_rays);
            if (w.d_hits) cudaFree(w.d_hits);
        }
        rrt::surface_tables_destroy(surface_tables);
    }
};

struct rrt_render {
    rrt_scene* scene = nullptr;
    rrt::Renderer renderer;
};

namespace {

rrt::Transform xf_from(const double* m, const double* inv) {
    rrt::Transform t;
    std::memcpy(t.m.m, m, sizeof(double) * 16);
    std::memcpy(t.inv.m, inv, sizeof(double) * 16);
    return t;
}

// The surface pass's tables: the literal tier's own, or the scene's, uploaded on first use (Tier F).
int surface_tables(const rrt_scene* scene, const rrt::ShadeScene** tables, bool* literal) {
    if (scene->build_flags == RRT_BUILD_LITERAL) {
        *tables = &static_cast<const rrt::LiteralAggregate*>(scene->agg.get())->geometry_tables();
        *literal = true;
        return RRT_OK;
    }
    std::lock_guard<std::mutex> lock(scene->surface_mutex);
    if (!scene->surface_tables) {
        std::string err;
        const int rc = rrt::surface_tables_create(scene->host, &scene->surface_tables, &err);
        if (rc != RRT_OK) return fail(rc, err);
    }
    *tables = rrt::surface_tables_view(scene->surface_tables);
    *literal = false;
    return RRT_OK;
}

// The host-buffer pipeline of every record format.  F32: a chunk goes up as rrt_ray_f32 into the slot's staging
// buffer and is promoted into the slot's rrt_ray buffer; its f64 hits are compacted into the staging buffer, whose
// rays are dead by then, and go down from there.  SURF: the surface pass turns the chunk's rays and f64 hits into
// rrt_surface records in the slot's record buffer, in chunks of surface_chunk_rays().
template <bool ANY, bool F32, bool SURF = false>
int host_batch(const rrt_scene* scene, uint64_t n, const void* rays, void* out) {
    if (!scene || !scene->committed) return fail(RRT_ERR_INVALID, "scene is not committed");
    if (n == 0) return RRT_OK;
    if (!rays || !out) return fail(RRT_ERR_INVALID, "null ray / output buffer");
    rrt_ctx* ctx = scene->ctx;
    std::lock_guard<std::mutex> lock(ctx->host_path_mutex);
    int rc = ctx->ensure_slots();
    if (rc != RRT_OK) return rc;
    CAPI_CUDA(cudaSetDevice(ctx->device));
    if (F32 && (rc = ctx->ensure_f32_slots()) != RRT_OK) return rc;
    const rrt::ShadeScene* tables = nullptr;
    bool literal = false;
    if (SURF && ((rc = ctx->ensure_surface_slots()) != RRT_OK || (rc = surface_tables(scene, &tables, &literal)) != RRT_OK))
        return rc;
    const uint64_t full_chunk = SURF ? surface_chunk_rays() : kChunkRays;
    const size_t in_elem = F32 ? sizeof(rrt_ray_f32) : sizeof(rrt_ray);
    const size_t out_elem = ANY ? sizeof(uint8_t) : (F32 ? sizeof(rrt_hit_f32) : (SURF ? sizeof(rrt_surface) : sizeof(rrt_hit)));
    auto drain = [&] {  // copies of earlier chunks into the caller's buffer may still be in flight
        for (auto& t : ctx->slots) cudaStreamSynchronize(t.stream);
    };
    std::string err;
    uint64_t done = 0;
    int k = 0;
    // RRT_HOST_TRACE=1 (diagnostic): the device-side timeline of the pipeline, one line per chunk on stderr
    static const bool tracing = std::getenv("RRT_HOST_TRACE") != nullptr;
    struct Marks { cudaEvent_t e[4]; uint64_t cnt; };
    std::vector<Marks> marks;
    auto mark = [&](int which, cudaStream_t st) {
        if (!tracing) return;
        cudaEventCreate(&marks.back().e[which]);
        cudaEventRecord(marks.back().e[which], st);
    };
    while (done < n) {
        Slot& s = ctx->slots[k % kSlots];
        const uint64_t cnt = tapered_chunk(done, n, full_chunk);
        if (tracing) {
            marks.push_back(Marks{});
            marks.back().cnt = cnt;
        }
        mark(0, s.stream);
        // a slot is reused only after its previous D2H has drained (stream order)
        CAPI_CUDA(cudaMemcpyAsync(F32 ? s.d_f32 : s.d_rays, static_cast<const char*>(rays) + done * in_elem, cnt * in_elem,
                                  cudaMemcpyHostToDevice, s.stream));
        mark(1, s.stream);
        int launched = 0;
        if (F32) {
            const int e = rrt::launch_promote_rays(cnt, static_cast<const rrt_ray_f32*>(s.d_f32), s.d_rays, s.stream);
            if (e != cudaSuccess) {
                drain();
                return cuda_fail("promote_rays_kernel", (cudaError_t)e);
            }
            ++launched;
        }
        int traced = 0;
        if (ANY)
            rc = scene->agg->any_hit(cnt, s.d_rays, static_cast<uint8_t*>(s.d_out), s.stream, &err, &traced);
        else
            rc = scene->agg->closest_hit(cnt, s.d_rays, static_cast<rrt_hit*>(s.d_out), s.stream, &err, &traced);
        if (rc != RRT_OK) {
            drain();
            return fail(rc, err);
        }
        launched += traced;
        const void* d_result = s.d_out;
        if (F32 && !ANY) {
            const int e = rrt::launch_compact_hits(cnt, static_cast<const rrt_hit*>(s.d_out), static_cast<rrt_hit_f32*>(s.d_f32),
                                                   s.stream);
            if (e != cudaSuccess) {
                drain();
                return cuda_fail("compact_hits_kernel", (cudaError_t)e);
            }
            ++launched;
            d_result = s.d_f32;
        }
        if (SURF) {
            const int e = rrt::launch_surfaces(*tables, literal, cnt, s.d_rays, static_cast<const rrt_hit*>(s.d_out),
                                               static_cast<rrt_surface*>(s.d_surf), s.stream);
            if (e != cudaSuccess) {
                drain();
                return cuda_fail("surface_kernel", (cudaError_t)e);
            }
            ++launched;
            d_result = s.d_surf;
        }
        ctx->launches.fetch_add((uint64_t)launched, std::memory_order_relaxed);
        mark(2, s.stream);
        CAPI_CUDA(cudaMemcpyAsync(static_cast<char*>(out) + done * out_elem, d_result, cnt * out_elem,
                                  cudaMemcpyDeviceToHost, s.stream));
        mark(3, s.stream);
        done += cnt;
        ++k;
    }
    for (auto& s : ctx->slots) CAPI_CUDA(cudaStreamSynchronize(s.stream));
    if (tracing) {
        for (size_t i = 0; i < marks.size(); ++i) {
            float t[4];
            for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&t[j], marks[0].e[0], marks[i].e[j]);
            fprintf(stderr, "RRT_HOST_TRACE chunk %2zu %8llu rays: slot free %7.3f  h2d done %7.3f  traced %7.3f  d2h done %7.3f ms\n", i,
                    (unsigned long long)marks[i].cnt, t[0], t[1], t[2], t[3]);
            }
        for (auto& m : marks)
            for (auto& e : m.e) cudaEventDestroy(e);
    }
    return RRT_OK;
}

// The calling stream's scratch (rrt_scene::StreamScratch), with room for `n_rays` promoted rays and `n_hits` f64 hits,
// and `stream` ordered after the last call that used it.  Called with scene->scratch_mutex held, which the caller keeps
// while it enqueues its passes and until release_scratch, so that a shared scratch's event orders whole calls.
int acquire_scratch(const rrt_scene* scene, void* stream, uint64_t n_rays, uint64_t n_hits, rrt_scene::StreamScratch** out) {
    auto& pool = scene->scratch;
    rrt_scene::StreamScratch& w =
        (pool.count(stream) || pool.size() < rrt_scene::kMaxScratch) ? pool[stream] : pool.begin()->second;
    if (!w.last_use) CAPI_CUDA(cudaEventCreateWithFlags(&w.last_use, cudaEventDisableTiming));
    if (n_rays > w.ray_capacity || n_hits > w.hit_capacity) {
        // the buffers are replaced: every call that used them is ordered before the last one (same stream, or the event)
        if (w.used) CAPI_CUDA(cudaEventSynchronize(w.last_use));
        if (n_rays > w.ray_capacity) {
            if (w.d_rays) cudaFree(w.d_rays);
            w.d_rays = nullptr;
            w.ray_capacity = 0;
            CAPI_CUDA(cudaMalloc(&w.d_rays, n_rays * sizeof(rrt_ray)));
            w.ray_capacity = n_rays;
        }
        if (n_hits > w.hit_capacity) {
            if (w.d_hits) cudaFree(w.d_hits);
            w.d_hits = nullptr;
            w.hit_capacity = 0;
            CAPI_CUDA(cudaMalloc(&w.d_hits, n_hits * sizeof(rrt_hit)));
            w.hit_capacity = n_hits;
        }
    }
    if (w.used && w.last_stream != stream) CAPI_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), w.last_use, 0));
    *out = &w;
    return RRT_OK;
}
int release_scratch(rrt_scene::StreamScratch* w, void* stream) {
    CAPI_CUDA(cudaEventRecord(w->last_use, static_cast<cudaStream_t>(stream)));
    w->used = true;
    w->last_stream = stream;
    return RRT_OK;
}

// rrt_intersect_f32_device / rrt_intersect_p_f32_device: promote into the stream's scratch, walk, compact into the
// caller's buffer.
template <bool ANY>
int device_f32(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* d_rays, void* d_out, void* stream, const char* name) {
    if (!scene || !scene->committed) return fail(RRT_ERR_INVALID, std::string(name) + ": scene is not committed");
    if (n == 0) return RRT_OK;
    if (!d_rays || !d_out) return fail(RRT_ERR_INVALID, std::string(name) + ": null buffer");
    if (n >= (1ull << 32)) return fail(RRT_ERR_INVALID, std::string(name) + ": batch too large for one call (2^32 rays)");
    if ((reinterpret_cast<uintptr_t>(d_rays) | (ANY ? 0 : reinterpret_cast<uintptr_t>(d_out))) & 15u)
        return fail(RRT_ERR_INVALID, std::string(name) + ": device buffers must be 16-byte aligned");
    CAPI_CUDA(cudaSetDevice(scene->ctx->device));
    std::lock_guard<std::mutex> lock(scene->scratch_mutex);
    rrt_scene::StreamScratch* w = nullptr;
    int rc = acquire_scratch(scene, stream, n, ANY ? 0 : n, &w);
    if (rc != RRT_OK) return rc;
    int e = rrt::launch_promote_rays(n, d_rays, w->d_rays, stream);
    if (e != cudaSuccess) return cuda_fail("promote_rays_kernel", (cudaError_t)e);
    std::string err;
    int launched = 0;
    rc = ANY ? scene->agg->any_hit(n, w->d_rays, static_cast<uint8_t*>(d_out), stream, &err, &launched)
             : scene->agg->closest_hit(n, w->d_rays, w->d_hits, stream, &err, &launched);
    if (rc != RRT_OK) return fail(rc, err);
    launched += 1;
    if (!ANY) {
        e = rrt::launch_compact_hits(n, w->d_hits, static_cast<rrt_hit_f32*>(d_out), stream);
        if (e != cudaSuccess) return cuda_fail("compact_hits_kernel", (cudaError_t)e);
        launched += 1;
    }
    if ((rc = release_scratch(w, stream)) != RRT_OK) return rc;
    scene->ctx->launches.fetch_add((uint64_t)launched, std::memory_order_relaxed);
    return RRT_OK;
}

// rrt_intersect_surface_device: walk into the stream's scratch hits, then the surface pass into the caller's records.
int device_surface(const rrt_scene* scene, uint64_t n, const rrt_ray* d_rays, rrt_surface* d_out, void* stream) {
    const char* name = "rrt_intersect_surface_device";
    if (!scene || !scene->committed) return fail(RRT_ERR_INVALID, std::string(name) + ": scene is not committed");
    if (n == 0) return RRT_OK;
    if (!d_rays || !d_out) return fail(RRT_ERR_INVALID, std::string(name) + ": null buffer");
    if (n >= (1ull << 32)) return fail(RRT_ERR_INVALID, std::string(name) + ": batch too large for one call (2^32 rays)");
    CAPI_CUDA(cudaSetDevice(scene->ctx->device));
    const rrt::ShadeScene* tables = nullptr;
    bool literal = false;
    int rc = surface_tables(scene, &tables, &literal);
    if (rc != RRT_OK) return rc;
    std::lock_guard<std::mutex> lock(scene->scratch_mutex);
    rrt_scene::StreamScratch* w = nullptr;
    if ((rc = acquire_scratch(scene, stream, 0, n, &w)) != RRT_OK) return rc;
    std::string err;
    int launched = 0;
    rc = scene->agg->closest_hit(n, d_rays, w->d_hits, stream, &err, &launched);
    if (rc != RRT_OK) return fail(rc, err);
    const int e = rrt::launch_surfaces(*tables, literal, n, d_rays, w->d_hits, d_out, stream);
    if (e != cudaSuccess) return cuda_fail("surface_kernel", (cudaError_t)e);
    launched += 1;
    if ((rc = release_scratch(w, stream)) != RRT_OK) return rc;
    scene->ctx->launches.fetch_add((uint64_t)launched, std::memory_order_relaxed);
    return RRT_OK;
}

}  // namespace

extern "C" {

const char* rrt_last_error(void) { return g_last_error.c_str(); }

int rrt_create(int device_ordinal, rrt_ctx** out) {
    if (!out) return fail(RRT_ERR_INVALID, "rrt_create: out is null");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return cuda_fail("cudaGetDeviceCount", e);
    if (device_ordinal < 0 || device_ordinal >= count)
        return fail(RRT_ERR_INVALID, "rrt_create: no CUDA device " + std::to_string(device_ordinal) +
                                         " (this library has no CPU path)");
    cudaDeviceProp prop;
    CAPI_CUDA(cudaGetDeviceProperties(&prop, device_ordinal));
    if (prop.major != 10)
        return fail(RRT_ERR_UNSUPPORTED, std::string("rrt_create: built for sm_100a only, device is ") + prop.name);
    CAPI_CUDA(cudaSetDevice(device_ordinal));
    rrt_ctx* c = new (std::nothrow) rrt_ctx();
    if (!c) return fail(RRT_ERR_INVALID, "out of host memory");
    c->device = device_ordinal;
    *out = c;
    return RRT_OK;
}

void rrt_destroy(rrt_ctx* ctx) { delete ctx; }

uint64_t rrt_launch_count(const rrt_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

int rrt_host_alloc(rrt_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return fail(RRT_ERR_INVALID, "rrt_host_alloc: null argument");
    CAPI_CUDA(cudaSetDevice(ctx->device));
    CAPI_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
    return RRT_OK;
}
int rrt_host_free(rrt_ctx* ctx, void* p) {
    if (!ctx) return fail(RRT_ERR_INVALID, "rrt_host_free: null ctx");
    CAPI_CUDA(cudaFreeHost(p));
    return RRT_OK;
}

int rrt_scene_begin(rrt_ctx* ctx, rrt_scene** out) {
    if (!ctx || !out) return fail(RRT_ERR_INVALID, "rrt_scene_begin: null argument");
    rrt_scene* s = new (std::nothrow) rrt_scene();
    if (!s) return fail(RRT_ERR_INVALID, "out of host memory");
    s->ctx = ctx;
    *out = s;
    return RRT_OK;
}
void rrt_scene_destroy(rrt_scene* scene) {
    if (scene) cudaSetDevice(scene->ctx->device);
    delete scene;
}

int rrt_scene_add_mesh(rrt_scene* scene, uint32_t nv, const double* p, uint32_t ntri, const uint32_t* vi, uint32_t nn,
                       const double* n, const uint32_t* ni, uint32_t nuv, const double* uv, const uint32_t* uvi,
                       uint32_t* mesh_id) {
    if (!scene || scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_add_mesh: scene missing or committed");
    if (!p || !vi || nv == 0 || ntri == 0) return fail(RRT_ERR_INVALID, "rrt_scene_add_mesh: empty mesh");
    try {
        rrt::TriangleMesh m;
        m.p.assign(p, p + 3 * (size_t)nv);
        m.vi.assign(vi, vi + 3 * (size_t)ntri);
        for (uint32_t x : m.vi)
            if (x >= nv) return fail(RRT_ERR_INVALID, "rrt_scene_add_mesh: vertex index out of range");
        if (nn && n && ni) {
            m.n.assign(n, n + 3 * (size_t)nn);
            m.ni.assign(ni, ni + 3 * (size_t)ntri);
            for (uint32_t x : m.ni)
                if (x >= nn) return fail(RRT_ERR_INVALID, "rrt_scene_add_mesh: normal index out of range");
        }
        if (nuv && uv && uvi) {
            m.uv.assign(uv, uv + 2 * (size_t)nuv);
            m.uvi.assign(uvi, uvi + 3 * (size_t)ntri);
            for (uint32_t x : m.uvi)
                if (x >= nuv) return fail(RRT_ERR_INVALID, "rrt_scene_add_mesh: uv index out of range");
        }
        scene->host.meshes.push_back(std::move(m));
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    if (mesh_id) *mesh_id = (uint32_t)scene->host.meshes.size() - 1;
    return RRT_OK;
}

int rrt_scene_add_triangles(rrt_scene* scene, uint32_t mesh_id, uint32_t material_id, uint32_t n_instances,
                            const double* instance_m, const double* instance_minv) {
    if (!scene || scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_add_triangles: scene missing or committed");
    if (mesh_id >= scene->host.meshes.size()) return fail(RRT_ERR_INVALID, "rrt_scene_add_triangles: bad mesh id");
    if (n_instances && (!instance_m || !instance_minv))
        return fail(RRT_ERR_INVALID, "rrt_scene_add_triangles: instance matrices missing");
    try {
        const uint32_t nt = scene->host.meshes[mesh_id].n_triangles();
        auto& prims = scene->host.prims;
        if (n_instances == 0) {
            for (uint32_t t = 0; t < nt; ++t) prims.push_back({rrt::SHAPE_TRIANGLE, mesh_id, t, -1, material_id});
        } else {
            // renderprocess.rs:1265-1281: for each instance, every triangle of the mesh
            for (uint32_t i = 0; i < n_instances; ++i) {
                scene->host.instances.push_back(xf_from(instance_m + 16 * (size_t)i, instance_minv + 16 * (size_t)i));
                int32_t xi = (int32_t)scene->host.instances.size() - 1;
                for (uint32_t t = 0; t < nt; ++t) prims.push_back({rrt::SHAPE_TRIANGLE, mesh_id, t, xi, material_id});
            }
        }
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_scene_add_sphere(rrt_scene* scene, const double* obj_to_world_m, const double* obj_to_world_minv, double radius,
                         double z_min, double z_max, double phi_max_deg, uint32_t material_id, uint32_t n_instances,
                         const double* instance_m, const double* instance_minv) {
    if (!scene || scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_add_sphere: scene missing or committed");
    if (n_instances && (!instance_m || !instance_minv))
        return fail(RRT_ERR_INVALID, "rrt_scene_add_sphere: instance matrices missing");
    try {
        rrt::Sphere s;
        s.obj_to_world = (obj_to_world_m && obj_to_world_minv) ? xf_from(obj_to_world_m, obj_to_world_minv)
                                                               : rrt::Transform::identity();
        s.radius = radius;
        s.z_min = z_min;
        s.z_max = z_max;
        s.phi_max_deg = phi_max_deg;
        scene->host.spheres.push_back(s);
        uint32_t sid = (uint32_t)scene->host.spheres.size() - 1;
        auto& prims = scene->host.prims;
        if (n_instances == 0) {
            prims.push_back({rrt::SHAPE_SPHERE, sid, 0, -1, material_id});
        } else {
            for (uint32_t i = 0; i < n_instances; ++i) {
                scene->host.instances.push_back(xf_from(instance_m + 16 * (size_t)i, instance_minv + 16 * (size_t)i));
                prims.push_back({rrt::SHAPE_SPHERE, sid, 0, (int32_t)scene->host.instances.size() - 1, material_id});
            }
        }
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_scene_commit(rrt_scene* scene, uint32_t max_prims_in_node, uint32_t build_flags) {
    if (!scene) return fail(RRT_ERR_INVALID, "rrt_scene_commit: null scene");
    if (scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_commit: already committed");
    if (build_flags != RRT_BUILD_FAST && build_flags != RRT_BUILD_LITERAL && build_flags != RRT_BUILD_DEVICE_LBVH)
        return fail(RRT_ERR_INVALID, "rrt_scene_commit: unknown build flags");
    try {
        std::string err;
        int rc;
        if (build_flags == RRT_BUILD_LITERAL) {
            auto* lit = new rrt::LiteralAggregate();
            scene->agg.reset(lit);
            rc = lit->build(scene->ctx->device, scene->host, max_prims_in_node, &err);
        } else {
            auto* fast = new rrt::DeviceAggregate();
            scene->agg.reset(fast);
            rc = fast->build(scene->ctx->device, scene->host, max_prims_in_node, &err, build_flags == RRT_BUILD_DEVICE_LBVH);
        }
        if (rc != RRT_OK) {
            scene->agg.reset();
            return fail(rc, err);
        }
    } catch (const std::exception& e) {
        scene->agg.reset();
        return fail(RRT_ERR_INVALID, e.what());
    }
    scene->build_flags = build_flags;
    scene->max_prims_in_node = max_prims_in_node;
    scene->committed = true;
    return RRT_OK;
}

int rrt_scene_update_instances(rrt_scene* scene, uint32_t first_instance, uint32_t n, const double* instance_m,
                               const double* instance_minv) {
    if (!scene || (n && (!instance_m || !instance_minv))) return fail(RRT_ERR_INVALID, "rrt_scene_update_instances: null argument");
    if (!scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_update_instances: scene is not committed");
    if (scene->build_flags == RRT_BUILD_LITERAL)
        return fail(RRT_ERR_UNSUPPORTED, "rrt_scene_update_instances: the literal tier rebuilds the reference's HLBVH on the host; commit a new scene");
    if (scene->live_renders.load() != 0)
        return fail(RRT_ERR_INVALID, "rrt_scene_update_instances: destroy the integrators made over this scene first (they hold its tables)");
    if ((uint64_t)first_instance + n > scene->host.instances.size())
        return fail(RRT_ERR_INVALID, "rrt_scene_update_instances: instance range out of bounds");
    try {
        for (uint32_t i = 0; i < n; ++i)
            scene->host.instances[first_instance + i] = xf_from(instance_m + 16 * (size_t)i, instance_minv + 16 * (size_t)i);
        scene->mesh_image.reset();
        // The tree over the moved primitives is made anew on the device: keys, sort, hierarchy and boxes take a few
        // milliseconds there (DESIGN.md §4b) — a topology-preserving refit would save none of the part that costs, the
        // host-side re-bake of the moved primitives' records.
        std::unique_ptr<rrt::DeviceAggregate> fresh(new rrt::DeviceAggregate());
        std::string err;
        CAPI_CUDA(cudaSetDevice(scene->ctx->device));
        int rc = fresh->build(scene->ctx->device, scene->host, scene->max_prims_in_node, &err, true);
        if (rc != RRT_OK) return fail(rc, err);
        scene->agg = std::move(fresh);
        scene->build_flags = RRT_BUILD_DEVICE_LBVH;
        // the surface pass's tables hold the old transforms: the next surface call uploads them anew
        std::lock_guard<std::mutex> lock(scene->surface_mutex);
        rrt::surface_tables_destroy(scene->surface_tables);
        scene->surface_tables = nullptr;
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

namespace {

// rrt_scene_update_mesh and rrt_scene_update_mesh_device: d_stream is the caller's stream for device buffers, or
// nullptr for host buffers.
int update_mesh(rrt_scene* scene, const char* name, uint32_t mesh_id, uint32_t first_vertex, uint32_t n_vertices,
                const double* p, uint32_t first_normal, uint32_t n_normals, const double* nrm, bool device,
                cudaStream_t stream) {
    const std::string fn = name;
    if (!scene || (n_vertices && !p) || (n_normals && !nrm)) return fail(RRT_ERR_INVALID, fn + ": null argument");
    if (!scene->committed) return fail(RRT_ERR_INVALID, fn + ": scene is not committed");
    if (scene->build_flags == RRT_BUILD_LITERAL)
        return fail(RRT_ERR_UNSUPPORTED, fn + ": the literal tier rebuilds the reference's HLBVH on the host; commit a new scene");
    if (scene->live_renders.load() != 0)
        return fail(RRT_ERR_INVALID, fn + ": destroy the integrators made over this scene first (they hold its tables)");
    if (mesh_id >= scene->host.meshes.size()) return fail(RRT_ERR_INVALID, fn + ": bad mesh id");
    rrt::TriangleMesh& mesh = scene->host.meshes[mesh_id];
    if ((uint64_t)first_vertex + n_vertices > mesh.p.size() / 3) return fail(RRT_ERR_INVALID, fn + ": vertex range out of bounds");
    if (n_normals && mesh.n.empty()) return fail(RRT_ERR_INVALID, fn + ": the mesh has no vertex normals");
    if ((uint64_t)first_normal + n_normals > mesh.n.size() / 3) return fail(RRT_ERR_INVALID, fn + ": normal range out of bounds");
    if (n_vertices == 0 && n_normals == 0) return RRT_OK;
    try {
        std::string err;
        const int dev = scene->ctx->device;
        CAPI_CUDA(cudaSetDevice(dev));
        // a fresh RRT_BUILD_DEVICE_LBVH commit builds its tree on the device only for scenes that device_tree_fits;
        // the others get the host SAH tree, and so does the update
        const bool on_device = rrt::DeviceAggregate::device_tree_fits(scene->host.prims.size(), scene->max_prims_in_node);
        if (on_device && !scene->mesh_image) {
            std::unique_ptr<rrt::MeshImage> image(new rrt::MeshImage());
            int rc = image->create(dev, scene->host, &err);
            if (rc != RRT_OK) return fail(rc, err);
            scene->mesh_image = std::move(image);
        }
        rrt::MeshImage* image = on_device ? scene->mesh_image.get() : nullptr;
        const size_t p_bytes = 3 * (size_t)n_vertices * sizeof(double), n_bytes = 3 * (size_t)n_normals * sizeof(double);
        double* const mp = mesh.p.data() + 3 * (size_t)first_vertex;
        double* const mn = mesh.n.data() + 3 * (size_t)first_normal;
        // The host mirror (later commits, exports, instance updates, renderers and the surface tables read it) takes the
        // new values once the aggregate over them exists; the device entry reads the caller's buffers in stream order.
        auto write_mirror = [&]() -> cudaError_t {
            if (!device) {
                if (n_vertices) std::memcpy(mp, p, p_bytes);
                if (n_normals) std::memcpy(mn, nrm, n_bytes);
                return cudaSuccess;
            }
            cudaError_t e = cudaSuccess;
            if (n_vertices) e = cudaMemcpyAsync(mp, p, p_bytes, cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess && n_normals) e = cudaMemcpyAsync(mn, nrm, n_bytes, cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            return e;
        };
        std::unique_ptr<rrt::DeviceAggregate> fresh(new rrt::DeviceAggregate());
        bool built = false;
        if (image) {
            // the new positions into the image, then re-bake, frame, tree and records on the device
            int rc = RRT_OK;
            cudaError_t e = cudaSuccess;
            double* const ip = image->positions(mesh_id) + 3 * (size_t)first_vertex;
            if (n_vertices && device) {
                e = cudaMemcpyAsync(ip, p, p_bytes, cudaMemcpyDeviceToDevice, stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            } else if (n_vertices) {
                e = cudaMemcpy(ip, p, p_bytes, cudaMemcpyHostToDevice);
            }
            if (e != cudaSuccess) rc = cuda_fail("the new positions to the device", e);
            bool too_deep = false;
            if (rc == RRT_OK && (rc = image->rebake(mesh_id, &err)) != RRT_OK) fail(rc, err);
            if (rc == RRT_OK && (rc = fresh->build_from_image(dev, *image, scene->max_prims_in_node, &too_deep, &err)) != RRT_OK)
                fail(rc, err);
            built = rc == RRT_OK && !too_deep;
            if (built && (e = write_mirror()) != cudaSuccess) rc = cuda_fail("the new values to the host", e);
            if (rc != RRT_OK) {
                scene->mesh_image.reset();
                return rc;
            }
        }
        if (!built) {
            // the host SAH tree of a commit (too few primitives, or thousands with one centroid), made from the mirror
            const std::vector<double> old_p(mp, mp + 3 * (size_t)n_vertices), old_n(mn, mn + 3 * (size_t)n_normals);
            const cudaError_t e = write_mirror();
            int rc = e == cudaSuccess ? RRT_OK : cuda_fail("the new values to the host", e);
            fresh.reset(new rrt::DeviceAggregate());
            if (rc == RRT_OK && (rc = fresh->build(dev, scene->host, scene->max_prims_in_node, &err, true)) != RRT_OK) fail(rc, err);
            if (rc != RRT_OK) {
                if (n_vertices) std::memcpy(mp, old_p.data(), p_bytes);
                if (n_normals) std::memcpy(mn, old_n.data(), n_bytes);
                scene->mesh_image.reset();
                return rc;
            }
        }
        scene->agg = std::move(fresh);
        scene->build_flags = RRT_BUILD_DEVICE_LBVH;
        // the surface pass's tables hold the old positions and normals: the next surface call uploads them anew
        std::lock_guard<std::mutex> lock(scene->surface_mutex);
        rrt::surface_tables_destroy(scene->surface_tables);
        scene->surface_tables = nullptr;
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

}  // namespace

int rrt_scene_update_mesh(rrt_scene* scene, uint32_t mesh_id, uint32_t first_vertex, uint32_t n_vertices, const double* p,
                          uint32_t first_normal, uint32_t n_normals, const double* n) {
    return update_mesh(scene, "rrt_scene_update_mesh", mesh_id, first_vertex, n_vertices, p, first_normal, n_normals, n,
                       false, nullptr);
}

int rrt_scene_update_mesh_device(rrt_scene* scene, uint32_t mesh_id, uint32_t first_vertex, uint32_t n_vertices,
                                 const double* d_p, uint32_t first_normal, uint32_t n_normals, const double* d_n,
                                 void* cuda_stream) {
    return update_mesh(scene, "rrt_scene_update_mesh_device", mesh_id, first_vertex, n_vertices, d_p, first_normal, n_normals,
                       d_n, true, static_cast<cudaStream_t>(cuda_stream));
}

int rrt_scene_num_prims(const rrt_scene* scene, uint32_t* out) {
    if (!scene || !out) return fail(RRT_ERR_INVALID, "rrt_scene_num_prims: null argument");
    *out = (uint32_t)scene->host.prims.size();
    return RRT_OK;
}

int rrt_world_bound(const rrt_scene* scene, double out6[6]) {
    if (!scene || !out6) return fail(RRT_ERR_INVALID, "rrt_world_bound: null argument");
    if (scene->host.prims.empty()) return fail(RRT_ERR_EMPTY, "rrt_world_bound: no primitives");
    // BVHAccel::world_bound = root bounds (bvh.rs:177-182).  In the literal tier that is the root of
    // the reference's own tree, which may have lost primitives (Q1); otherwise the union of every
    // Primitive::world_bound.
    if (scene->committed && scene->build_flags == RRT_BUILD_LITERAL) {
        static_cast<const rrt::LiteralAggregate*>(scene->agg.get())->root_bounds(out6);
        return RRT_OK;
    }
    rrt::Aabb b;
    for (size_t i = 0; i < scene->host.prims.size(); ++i) b.grow(scene->host.reference_world_bound(i));
    for (int k = 0; k < 3; ++k) {
        out6[k] = b.lo[k];
        out6[3 + k] = b.hi[k];
    }
    return RRT_OK;
}

int rrt_hlbvh_literal_probe(uint32_t n, const double* bounds6, uint32_t max_prims_in_node, uint32_t capacity_nodes,
                            uint32_t* n_nodes, double* node_bounds6, uint32_t* node_meta3, uint32_t* ordered) {
    if (!bounds6 || !n_nodes) return fail(RRT_ERR_INVALID, "rrt_hlbvh_literal_probe: null argument");
    if (n == 0) return fail(RRT_ERR_EMPTY, "BVHAccel::new needs at least one primitive (bvh.rs:319)");
    try {
        std::vector<rrt::Aabb> b(n);
        for (uint32_t i = 0; i < n; ++i)
            for (int k = 0; k < 3; ++k) {
                b[i].lo[k] = bounds6[6 * (size_t)i + k];
                b[i].hi[k] = bounds6[6 * (size_t)i + 3 + k];
            }
        rrt::LiteralBvh tree;
        rrt::build_hlbvh_literal(b, max_prims_in_node, &tree);
        *n_nodes = (uint32_t)tree.nodes.size();
        if (tree.nodes.size() <= capacity_nodes) {
            for (size_t i = 0; i < tree.nodes.size(); ++i) {
                const rrt::LinearNode& nd = tree.nodes[i];
                if (node_bounds6)
                    for (int k = 0; k < 3; ++k) {
                        node_bounds6[6 * i + k] = nd.lo[k];
                        node_bounds6[6 * i + 3 + k] = nd.hi[k];
                    }
                if (node_meta3) {
                    node_meta3[3 * i] = nd.offset;
                    node_meta3[3 * i + 1] = nd.n_primitives;
                    node_meta3[3 * i + 2] = nd.axis;
                }
            }
            if (ordered) std::memcpy(ordered, tree.ordered.data(), tree.ordered.size() * sizeof(uint32_t));
        }
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_scene_build_info(const rrt_scene* scene, uint64_t out4[4]) {
    if (!scene || !out4 || !scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_build_info: scene not committed");
    const rrt::AggregateStats& s = scene->agg->stats();
    out4[0] = s.tree_device_usec;
    out4[1] = s.n_nodes ? (s.device_bytes - s.n_records * (s.wide_records ? 96u : 48u)) / s.n_nodes : 0;
    out4[2] = scene->build_flags == RRT_BUILD_DEVICE_LBVH ? 1 : 0;
    out4[3] = 0;
    return RRT_OK;
}

int rrt_lbvh_host_probe(uint32_t n, const double* bounds6, uint32_t max_prims_in_node, uint32_t capacity_nodes,
                        uint32_t* n_nodes, uint32_t* node_words16, uint32_t* order, uint32_t info3[3]) {
    if (!bounds6 || !n_nodes) return fail(RRT_ERR_INVALID, "rrt_lbvh_host_probe: null argument");
    try {
        std::vector<rrt::Aabb> b(n);
        rrt::Aabb world;
        for (uint32_t i = 0; i < n; ++i) {
            for (int k = 0; k < 3; ++k) {
                b[i].lo[k] = bounds6[6 * (size_t)i + k];
                b[i].hi[k] = bounds6[6 * (size_t)i + 3 + k];
            }
            world.grow(b[i]);
        }
        const rrt::NodeFrame f = rrt::make_node_frame(world);
        std::vector<uint8_t> nodes;
        std::vector<uint32_t> ord;
        uint32_t depth = 0, leaves = 0;
        const uint32_t max_leaf = max_prims_in_node == 0 ? 4 : (max_prims_in_node > 8 ? 8 : max_prims_in_node);
        int rc = rrt::lbvh_host_probe(b, max_leaf, f.delta, false, f.grid_lo, f.grid_ext, &nodes, &ord, &depth, &leaves);
        if (rc != RRT_OK) return fail(rc, "device LBVH needs more primitives than one leaf holds");
        *n_nodes = (uint32_t)(nodes.size() / 64);
        if (info3) {
            info3[0] = *n_nodes;
            info3[1] = depth;
            info3[2] = leaves;
        }
        if (*n_nodes <= capacity_nodes) {
            if (node_words16) std::memcpy(node_words16, nodes.data(), nodes.size());
            if (order) std::memcpy(order, ord.data(), ord.size() * sizeof(uint32_t));
        }
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_scene_stats(const rrt_scene* scene, uint64_t out8[8]) {
    if (!scene || !out8 || !scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_stats: scene not committed");
    const rrt::AggregateStats& s = scene->agg->stats();
    out8[0] = s.n_nodes;
    out8[1] = s.n_leaves;
    out8[2] = s.max_depth;
    out8[3] = s.device_bytes;
    out8[4] = s.build_usec;
    out8[5] = s.n_records;
    out8[6] = s.wide_records;
    out8[7] = s.n_prims;
    return RRT_OK;
}

int rrt_scene_export_tree(const rrt_scene* scene, void* buffer, uint64_t capacity, uint64_t* bytes) {
    if (!scene || !bytes) return fail(RRT_ERR_INVALID, "rrt_scene_export_tree: null argument");
    if (!scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_export_tree: scene is not committed");
    const rrt::DeviceAggregate* agg = dynamic_cast<const rrt::DeviceAggregate*>(scene->agg.get());
    if (!agg) return fail(RRT_ERR_UNSUPPORTED, "rrt_scene_export_tree: the literal tier's aggregate is not exported");
    std::string err;
    int rc = agg->export_blob(buffer, capacity, bytes, &err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}
int rrt_scene_commit_from_tree(rrt_scene* scene, const void* blob, uint64_t bytes) {
    if (!scene || !blob) return fail(RRT_ERR_INVALID, "rrt_scene_commit_from_tree: null argument");
    if (scene->committed) return fail(RRT_ERR_INVALID, "rrt_scene_commit_from_tree: scene is already committed");
    try {
        std::unique_ptr<rrt::DeviceAggregate> agg(new rrt::DeviceAggregate());
        std::string err;
        int rc = agg->import_blob(scene->ctx->device, blob, bytes, scene->host.prims.size(), &err);
        if (rc != RRT_OK) return fail(rc, err);
        scene->agg = std::move(agg);
        scene->committed = true;
        scene->build_flags = RRT_BUILD_FAST;
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_intersect_device(const rrt_scene* scene, uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, void* cuda_stream) {
    if (!scene || !scene->committed) return fail(RRT_ERR_INVALID, "rrt_intersect_device: scene is not committed");
    if (n == 0) return RRT_OK;
    if (!d_rays || !d_hits) return fail(RRT_ERR_INVALID, "rrt_intersect_device: null buffer");
    CAPI_CUDA(cudaSetDevice(scene->ctx->device));  // the scratch buffers and the grid size belong to the scene's device
    std::string err;
    int launched = 0;
    int rc = scene->agg->closest_hit(n, d_rays, d_hits, cuda_stream, &err, &launched);
    if (rc != RRT_OK) return fail(rc, err);
    scene->ctx->launches.fetch_add((uint64_t)launched, std::memory_order_relaxed);
    return RRT_OK;
}

int rrt_intersect_p_device(const rrt_scene* scene, uint64_t n, const rrt_ray* d_rays, uint8_t* d_occluded,
                           void* cuda_stream) {
    if (!scene || !scene->committed) return fail(RRT_ERR_INVALID, "rrt_intersect_p_device: scene is not committed");
    if (n == 0) return RRT_OK;
    if (!d_rays || !d_occluded) return fail(RRT_ERR_INVALID, "rrt_intersect_p_device: null buffer");
    CAPI_CUDA(cudaSetDevice(scene->ctx->device));
    std::string err;
    int launched = 0;
    int rc = scene->agg->any_hit(n, d_rays, d_occluded, cuda_stream, &err, &launched);
    if (rc != RRT_OK) return fail(rc, err);
    scene->ctx->launches.fetch_add((uint64_t)launched, std::memory_order_relaxed);
    return RRT_OK;
}

// ---- the render loop ---------------------------------------------------------------------------
int rrt_scene_set_materials(rrt_scene* scene, uint32_t n, const rrt_material* materials) {
    if (!scene || (n && !materials)) return fail(RRT_ERR_INVALID, "rrt_scene_set_materials: null argument");
    try {
        scene->materials.assign(materials, materials + n);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_scene_set_lights(rrt_scene* scene, uint32_t n, const rrt_light* lights) {
    if (!scene || (n && !lights)) return fail(RRT_ERR_INVALID, "rrt_scene_set_lights: null argument");
    try {
        scene->lights.assign(lights, lights + n);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_scene_set_infinite_lights(rrt_scene* scene, uint32_t n, const rrt_light* lights) {
    if (!scene || (n && !lights)) return fail(RRT_ERR_INVALID, "rrt_scene_set_infinite_lights: null argument");
    try {
        scene->extras.infinite_lights.assign(lights, lights + n);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_scene_add_image(rrt_scene* scene, uint32_t width, uint32_t height, const uint8_t* rgb8, uint32_t* index) {
    if (!scene || !rgb8 || !index) return fail(RRT_ERR_INVALID, "rrt_scene_add_image: null argument");
    if (width == 0 || height == 0 || width > 16384 || height > 16384) return fail(RRT_ERR_INVALID, "rrt_scene_add_image: size out of range");
    try {
        rrt::Image8 img;
        img.width = width;
        img.height = height;
        img.rgb.assign(rgb8, rgb8 + (size_t)width * height * 3);
        scene->extras.images.push_back(std::move(img));
        *index = (uint32_t)scene->extras.images.size() - 1;
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_scene_add_image_png(rrt_scene* scene, const char* path, uint32_t* index) {
    if (!scene || !path || !index) return fail(RRT_ERR_INVALID, "rrt_scene_add_image_png: null argument");
    try {
        rrt::Image8 img;
        std::string err;
        if (!rrt::read_png_rgb8(path, &img, &err)) return fail(RRT_ERR_IO, err);
        scene->extras.images.push_back(std::move(img));
        *index = (uint32_t)scene->extras.images.size() - 1;
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}

int rrt_scene_set_textures(rrt_scene* scene, uint32_t n, const rrt_texture* textures) {
    if (!scene || (n && !textures)) return fail(RRT_ERR_INVALID, "rrt_scene_set_textures: null argument");
    if (n > RRT_MAX_TEXTURES) return fail(RRT_ERR_UNSUPPORTED, "rrt_scene_set_textures: more than RRT_MAX_TEXTURES textures");
    try {
        std::string err;
        if (!rrt::validate_textures(textures, n, &err)) return fail(RRT_ERR_INVALID, "rrt_scene_set_textures: " + err);
        scene->textures.assign(textures, textures + n);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_scene_set_material_textures(rrt_scene* scene, uint32_t n_materials, const int32_t* slots) {
    if (!scene || (n_materials && !slots)) return fail(RRT_ERR_INVALID, "rrt_scene_set_material_textures: null argument");
    try {
        scene->material_slots.assign(slots, slots + (size_t)n_materials * RRT_MATERIAL_SLOTS);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_halton_host_probe(int64_t xres, int64_t yres, uint64_t seed, int use_tables, uint64_t n, const int64_t* px,
                          const int64_t* py, const uint64_t* sample, const uint32_t* dim, uint64_t* index_out, double* value_out) {
    if (n && (!px || !py || !sample || !dim || !index_out || !value_out))
        return fail(RRT_ERR_INVALID, "rrt_halton_host_probe: null argument");
    try {
        rrt::HaltonTables h = rrt::make_halton_tables(xres, yres, false);
        const std::vector<uint16_t> perms = rrt::make_halton_permutations(h, seed);
        const std::vector<rrt::HaltonDim> dims = rrt::make_halton_dims(h, perms);
        const std::vector<uint64_t> offs = rrt::make_halton_pixel_offsets(h);
        if (use_tables) {
            if (dims.empty()) return fail(RRT_ERR_INVALID, "rrt_halton_host_probe: a divider failed its check");
            h.dims = dims.data();
            h.pixel_off = offs.data();
        }
        for (uint64_t i = 0; i < n; ++i) {
            index_out[i] = rrt::halton_index(h, px[i], py[i], sample[i]);
            value_out[i] = rrt::halton_sample(h, perms.data(), index_out[i], dim[i]);
        }
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_differentials_host_probe(const double in24[24], double out10[10]) {
    if (!in24 || !out10) return fail(RRT_ERR_INVALID, "rrt_differentials_host_probe: null argument");
    rrt::differentials_host_eval(in24, out10);
    return RRT_OK;
}
int rrt_texture_host_probe(uint32_t n, const rrt_texture* textures, const double uv[2], const double p[3], const double* diff,
                           double* out) {
    if ((n && !textures) || !uv || !p || !out) return fail(RRT_ERR_INVALID, "rrt_texture_host_probe: null argument");
    if (n > RRT_MAX_TEXTURES) return fail(RRT_ERR_UNSUPPORTED, "rrt_texture_host_probe: more than RRT_MAX_TEXTURES textures");
    std::string err;
    if (!rrt::validate_textures(textures, n, &err)) return fail(RRT_ERR_INVALID, "rrt_texture_host_probe: " + err);
    rrt::texture_host_eval(textures, n, uv, p, diff, out);
    return RRT_OK;
}

int rrt_render_create(rrt_scene* scene, const rrt_render_desc* desc, rrt_render** out) {
    if (!scene || !desc || !out) return fail(RRT_ERR_INVALID, "rrt_render_create: null argument");
    *out = nullptr;
    if (!scene->committed) return fail(RRT_ERR_INVALID, "rrt_render_create: scene is not committed");
    try {
        double wb[6];
        int rc = rrt_world_bound(scene, wb);
        if (rc != RRT_OK) return rc;
        std::unique_ptr<rrt_render> r(new rrt_render());
        r->scene = scene;
        std::string err;
        rc = r->renderer.create(scene->ctx->device, scene->host, scene->agg.get(), scene->materials, scene->lights,
                                scene->textures, scene->material_slots, wb, *desc, &err, &scene->extras);
        if (rc != RRT_OK) return fail(rc, err);
        scene->ctx->launches.fetch_add(r->renderer.stats().launches, std::memory_order_relaxed);
        scene->live_renders.fetch_add(1);
        *out = r.release();
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
void rrt_render_destroy(rrt_render* render) {
    if (render && render->scene) render->scene->live_renders.fetch_sub(1);
    delete render;
}

int rrt_scene_load_json(rrt_ctx* ctx, const char* path, const char* overrides_json, uint64_t seed, rrt_scene** scene,
                        rrt_render** render) {
    return rrt_scene_load_json_tier(ctx, path, overrides_json, seed, RRT_BUILD_FAST, scene, render);
}

int rrt_scene_load_json_tier(rrt_ctx* ctx, const char* path, const char* overrides_json, uint64_t seed, uint32_t build_flags,
                             rrt_scene** scene, rrt_render** render) {
    if (!ctx || !path || !scene) return fail(RRT_ERR_INVALID, "rrt_scene_load_json: null argument");
    *scene = nullptr;
    if (render) *render = nullptr;
    rrt::LoadedScene loaded;
    try {
        rrt::load_scene_json(path, overrides_json ? overrides_json : "", seed, &loaded);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_IO, e.what());
    }
    rrt_scene* s = nullptr;
    int rc = rrt_scene_begin(ctx, &s);
    if (rc != RRT_OK) return rc;
    s->host = std::move(loaded.scene);
    s->materials = loaded.materials;
    s->lights = loaded.lights;
    s->textures = loaded.textures;
    s->material_slots = loaded.material_slots;
    s->extras.infinite_lights = loaded.infinite_lights;
    {
        // decode the images.  A texture no material reaches is never evaluated: when its file is missing (the sample
        // scene declares such an ImageTexture) it becomes a black constant instead of an error.
        std::vector<char> image_used(loaded.image_paths.size(), 0);
        for (const rrt_light& l : s->lights)
            if (l.kind == RRT_LIGHT_INFINITE) image_used[l.env_image] = 1;
        for (const rrt_light& l : s->extras.infinite_lights)
            if (l.kind == RRT_LIGHT_INFINITE) image_used[l.env_image] = 1;
        std::vector<char> reached(s->textures.size(), 0);
        for (int32_t t : s->material_slots)
            if (t >= 0) reached[(size_t)t] = 1;
        for (size_t i = s->textures.size(); i-- > 0;) {
            if (!reached[i]) continue;
            const rrt_texture& x = s->textures[i];
            const bool pair = x.kind == RRT_TEX_SCALE || x.kind == RRT_TEX_MIX || x.kind == RRT_TEX_CHECKER2D || x.kind == RRT_TEX_CHECKER3D;
            if (pair) reached[(size_t)x.t1] = reached[(size_t)x.t2] = 1;
            if (x.kind == RRT_TEX_MIX) reached[(size_t)x.amount] = 1;
            if (x.kind == RRT_TEX_IMAGE) image_used[(size_t)x.t1] = 1;
        }
        for (size_t i = 0; i < loaded.image_paths.size(); ++i) {
            rrt::Image8 img;
            std::string ierr;
            if (!rrt::read_png_rgb8(loaded.image_paths[i], &img, &ierr)) {
                if (image_used[i]) {
                    rrt_scene_destroy(s);
                    return fail(RRT_ERR_IO, ierr);
                }
                for (rrt_texture& x : s->textures)
                    if (x.kind == RRT_TEX_IMAGE && (size_t)x.t1 == i) {
                        x.kind = RRT_TEX_CONSTANT;
                        x.t1 = -1;
                        x.v[0][0] = x.v[0][1] = x.v[0][2] = 0.0;
                    }
            }
            s->extras.images.push_back(std::move(img));
        }
    }
    rc = rrt_scene_commit(s, loaded.max_prims_in_node, build_flags);
    if (rc != RRT_OK) {
        rrt_scene_destroy(s);
        return rc;
    }
    if (render) {
        loaded.desc.lens_data = loaded.lens_data.data();
        rc = rrt_render_create(s, &loaded.desc, render);
        if (rc != RRT_OK) {
            rrt_scene_destroy(s);
            return rc;
        }
    }
    *scene = s;
    return RRT_OK;
}

int rrt_scene_json_texture_probe(const char* path, const char* overrides_json, uint32_t* n_textures, rrt_texture* textures,
                                 uint32_t max_materials, uint32_t* n_materials, rrt_material* materials, int32_t* slots) {
    if (!path || !n_textures || !n_materials) return fail(RRT_ERR_INVALID, "rrt_scene_json_texture_probe: null argument");
    try {
        rrt::LoadedScene l;
        rrt::load_scene_json(path, overrides_json ? overrides_json : "", 0, &l);
        *n_textures = (uint32_t)l.textures.size();
        *n_materials = (uint32_t)l.materials.size();
        if (textures) std::copy(l.textures.begin(), l.textures.end(), textures);
        const size_t nm = std::min<size_t>(max_materials, l.materials.size());
        if (materials) std::copy(l.materials.begin(), l.materials.begin() + nm, materials);
        if (slots) std::copy(l.material_slots.begin(), l.material_slots.begin() + nm * RRT_MATERIAL_SLOTS, slots);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_IO, e.what());
    }
    return RRT_OK;
}

int rrt_scene_json_probe(const char* path, const char* overrides_json, uint64_t out8[8], rrt_render_desc* desc) {
    if (!path || !out8) return fail(RRT_ERR_INVALID, "rrt_scene_json_probe: null argument");
    try {
        rrt::LoadedScene l;
        rrt::load_scene_json(path, overrides_json ? overrides_json : "", 0, &l);
        out8[0] = l.scene.prims.size();
        out8[1] = l.scene.meshes.size();
        out8[2] = l.scene.spheres.size();
        out8[3] = l.scene.instances.size();
        out8[4] = l.materials.size();
        out8[5] = l.lights.size();
        out8[6] = l.max_prims_in_node;
        out8[7] = l.lens_data.size();
        if (desc) {
            *desc = l.desc;
            desc->lens_data = nullptr;
        }
    } catch (const std::exception& e) {
        return fail(RRT_ERR_IO, e.what());
    }
    return RRT_OK;
}

int rrt_render_run(rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, const int64_t* crop) {
    if (!render) return fail(RRT_ERR_INVALID, "rrt_render_run: null render");
    std::string err;
    const uint64_t before = render->renderer.stats().launches;
    int rc = render->renderer.run(tile_mod, tile_rank, crop, &err);
    if (rc != RRT_OK) return fail(rc, err);
    render->scene->ctx->launches.fetch_add(render->renderer.stats().launches - before, std::memory_order_relaxed);
    return RRT_OK;
}
int rrt_render_clear(rrt_render* render) {
    if (!render) return fail(RRT_ERR_INVALID, "rrt_render_clear: null render");
    std::string err;
    int rc = render->renderer.clear(&err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}
int rrt_render_read_film(rrt_render* render, double* rgb, double* raw) {
    if (!render) return fail(RRT_ERR_INVALID, "rrt_render_read_film: null render");
    std::string err;
    int rc = render->renderer.read_film(rgb, raw, &err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}
int rrt_render_read_rgba8(rrt_render* render, uint8_t* rgba8) {
    if (!render || !rgba8) return fail(RRT_ERR_INVALID, "rrt_render_read_rgba8: null argument");
    try {
        const size_t npix = (size_t)(render->renderer.film_doubles() / 4);
        std::vector<double> rgb(3 * npix);
        std::string err;
        int rc = render->renderer.read_film(rgb.data(), nullptr, &err);
        if (rc != RRT_OK) return fail(rc, err);
        rrt::rgb_to_rgba8(rgb.data(), npix, rgba8);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_render_write_png(rrt_render* render, const char* path) {
    if (!render || !path) return fail(RRT_ERR_INVALID, "rrt_render_write_png: null argument");
    try {
        const size_t npix = (size_t)(render->renderer.film_doubles() / 4);
        std::vector<uint8_t> px(4 * npix);
        int rc = rrt_render_read_rgba8(render, px.data());
        if (rc != RRT_OK) return rc;
        if (!rrt::write_png_rgba8(path, px.data(), (uint32_t)render->renderer.xres(), (uint32_t)render->renderer.yres()))
            return fail(RRT_ERR_IO, std::string("cannot write ") + path);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_rgb_to_png(const double* rgb, uint32_t xres, uint32_t yres, const char* path, uint8_t* rgba8_or_null) {
    if (!rgb || !xres || !yres) return fail(RRT_ERR_INVALID, "rrt_rgb_to_png: null argument");
    try {
        std::vector<uint8_t> px(4 * (size_t)xres * yres);
        rrt::rgb_to_rgba8(rgb, (size_t)xres * yres, px.data());
        if (rgba8_or_null) std::memcpy(rgba8_or_null, px.data(), px.size());
        if (path && !rrt::write_png_rgba8(path, px.data(), xres, yres)) return fail(RRT_ERR_IO, std::string("cannot write ") + path);
    } catch (const std::exception& e) {
        return fail(RRT_ERR_INVALID, e.what());
    }
    return RRT_OK;
}
int rrt_render_film_device(rrt_render* render, void** d_film, uint64_t* n_doubles) {
    if (!render || !d_film || !n_doubles) return fail(RRT_ERR_INVALID, "rrt_render_film_device: null argument");
    *d_film = render->renderer.film_device();
    *n_doubles = render->renderer.film_doubles();
    return RRT_OK;
}
int rrt_render_film_copy(rrt_render* render, void* d_buffer, int to_render, void* cuda_stream) {
    if (!render || !d_buffer) return fail(RRT_ERR_INVALID, "rrt_render_film_copy: null argument");
    std::string err;
    int rc = render->renderer.copy_film_device(d_buffer, to_render != 0, cuda_stream, &err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}
int rrt_render_owned_doubles(const rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, uint64_t* n_doubles) {
    if (!render || !n_doubles) return fail(RRT_ERR_INVALID, "rrt_render_owned_doubles: null argument");
    if (tile_mod == 0 || tile_rank >= tile_mod) return fail(RRT_ERR_INVALID, "rrt_render_owned_doubles: tile_rank must be < tile_mod");
    *n_doubles = render->renderer.owned_tiles(tile_mod, tile_rank) * 1024;
    return RRT_OK;
}
int rrt_render_pack_owned(rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, void* d_buffer, uint64_t capacity_doubles,
                          void* cuda_stream) {
    if (!render || !d_buffer) return fail(RRT_ERR_INVALID, "rrt_render_pack_owned: null argument");
    std::string err;
    int rc = render->renderer.pack_owned(tile_mod, tile_rank, d_buffer, capacity_doubles, false, cuda_stream, &err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}
int rrt_render_unpack_owned(rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, const void* d_buffer,
                            uint64_t capacity_doubles, void* cuda_stream) {
    if (!render || !d_buffer) return fail(RRT_ERR_INVALID, "rrt_render_unpack_owned: null argument");
    std::string err;
    int rc = render->renderer.pack_owned(tile_mod, tile_rank, const_cast<void*>(d_buffer), capacity_doubles, true, cuda_stream, &err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}
int rrt_film_gather(rrt_render* const* renders, uint32_t n, uint32_t root) {
    if (!renders || n == 0 || root >= n) return fail(RRT_ERR_INVALID, "rrt_film_gather: bad arguments");
    for (uint32_t r = 0; r < n; ++r)
        if (!renders[r]) return fail(RRT_ERR_INVALID, "rrt_film_gather: null renderer");
    rrt::Renderer& dst = renders[root]->renderer;
    for (uint32_t r = 0; r < n; ++r) {
        if (r == root) continue;
        rrt::Renderer& src = renders[r]->renderer;
        if (src.xres() != dst.xres() || src.yres() != dst.yres()) return fail(RRT_ERR_INVALID, "rrt_film_gather: films differ in size");
        const uint64_t nd = src.owned_tiles(n, r) * 1024;
        if (nd == 0) continue;
        void *d_src = nullptr, *d_dst = nullptr;
        std::string err;
        CAPI_CUDA(cudaSetDevice(src.device()));
        CAPI_CUDA(cudaMalloc(&d_src, nd * sizeof(double)));
        int rc = src.pack_owned(n, r, d_src, nd, false, nullptr, &err);
        if (rc == RRT_OK) {
            CAPI_CUDA(cudaStreamSynchronize(nullptr));
            CAPI_CUDA(cudaSetDevice(dst.device()));
            CAPI_CUDA(cudaMalloc(&d_dst, nd * sizeof(double)));
            CAPI_CUDA(cudaMemcpyPeer(d_dst, dst.device(), d_src, src.device(), nd * sizeof(double)));
            rc = dst.pack_owned(n, r, d_dst, nd, true, nullptr, &err);
            CAPI_CUDA(cudaStreamSynchronize(nullptr));
            cudaFree(d_dst);
        }
        cudaSetDevice(src.device());
        cudaFree(d_src);
        if (rc != RRT_OK) return fail(rc, err);
    }
    return RRT_OK;
}
int rrt_render_stats(const rrt_render* render, uint64_t out16[16]) {
    if (!render || !out16) return fail(RRT_ERR_INVALID, "rrt_render_stats: null argument");
    const rrt::RenderStats& s = render->renderer.stats();
    const uint64_t v[16] = {s.camera_rays, s.extension_rays, s.shadow_rays, s.bounces, s.zero_weight, s.samples,
                            s.launches, s.render_usec, s.setup_usec, s.chunks, s.f32_neighbours, s.f32_unsure, 0, 0, 0, 0};
    std::memcpy(out16, v, sizeof(v));
    return RRT_OK;
}
int rrt_render_hit_dump(rrt_render* render, int enable, double* out, uint64_t capacity, uint64_t* count) {
    if (!render) return fail(RRT_ERR_INVALID, "rrt_render_hit_dump: null render");
    std::string err;
    int rc = render->renderer.hit_dump(enable, out, capacity, count, &err);
    return rc == RRT_OK ? RRT_OK : fail(rc, err);
}

int rrt_intersect(const rrt_scene* scene, uint64_t n, const rrt_ray* rays, rrt_hit* hits) {
    return host_batch<false, false>(scene, n, rays, hits);
}
int rrt_intersect_p(const rrt_scene* scene, uint64_t n, const rrt_ray* rays, uint8_t* occluded) {
    return host_batch<true, false>(scene, n, rays, occluded);
}
int rrt_intersect_f32(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* rays, rrt_hit_f32* hits) {
    return host_batch<false, true>(scene, n, rays, hits);
}
int rrt_intersect_p_f32(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* rays, uint8_t* occluded) {
    return host_batch<true, true>(scene, n, rays, occluded);
}
int rrt_intersect_f32_device(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* d_rays, rrt_hit_f32* d_hits,
                             void* cuda_stream) {
    return device_f32<false>(scene, n, d_rays, d_hits, cuda_stream, "rrt_intersect_f32_device");
}
int rrt_intersect_p_f32_device(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* d_rays, uint8_t* d_occluded,
                               void* cuda_stream) {
    return device_f32<true>(scene, n, d_rays, d_occluded, cuda_stream, "rrt_intersect_p_f32_device");
}
int rrt_intersect_surface(const rrt_scene* scene, uint64_t n, const rrt_ray* rays, rrt_surface* surfaces) {
    return host_batch<false, false, true>(scene, n, rays, surfaces);
}
int rrt_intersect_surface_device(const rrt_scene* scene, uint64_t n, const rrt_ray* d_rays, rrt_surface* d_surfaces,
                                 void* cuda_stream) {
    return device_surface(scene, n, d_rays, d_surfaces, cuda_stream);
}
int rrt_rays_f32_host_probe(uint64_t n_rays, const rrt_ray_f32* rays, rrt_ray* promoted, uint64_t n_hits, const rrt_hit* hits,
                            rrt_hit_f32* compact) {
    if ((n_rays && (!rays || !promoted)) || (n_hits && (!hits || !compact)))
        return fail(RRT_ERR_INVALID, "rrt_rays_f32_host_probe: null argument");
    for (uint64_t i = 0; i < n_rays; ++i) promoted[i] = rrt::promote_ray(rays[i]);
    for (uint64_t i = 0; i < n_hits; ++i) compact[i] = rrt::compact_hit(hits[i]);
    return RRT_OK;
}

int rrt_stratified_host_probe(uint64_t seed, int64_t xres, int64_t px, int64_t py, uint32_t xs, uint32_t ys, uint32_t ndims,
                              int jitter, double* out1d, double* out2d, double* overflow4) {
    if (!out1d || !out2d || !overflow4) return fail(RRT_ERR_INVALID, "rrt_stratified_host_probe: null argument");
    if (xs == 0 || ys == 0 || xs * ys > rrt::kStratMaxSamples || ndims > rrt::kStratMaxDims)
        return fail(RRT_ERR_UNSUPPORTED, "rrt_stratified_host_probe: table size outside the device sampler's range");
    rrt::StratParams sp{xs, ys, ndims, jitter ? 1u : 0u, seed, xres};
    const uint32_t n = xs * ys;
    for (uint32_t d = 0; d < ndims; ++d)
        for (uint32_t i = 0; i < n; ++i) {
            out1d[d * n + i] = rrt::strat_table_1d(sp, px, py, d, i);
            const rrt::P2 p = rrt::strat_table_2d(sp, px, py, d, i);
            out2d[2 * (d * n + i)] = p.x;
            out2d[2 * (d * n + i) + 1] = p.y;
        }
    for (uint32_t k = 1; k < n; ++k) {
        uint32_t state = 0;
        for (uint32_t d = 0; d < ndims; ++d) rrt::strat_get_1d(sp, px, py, k, &state);
        for (int j = 0; j < 4; ++j) overflow4[4 * k + j] = rrt::strat_get_1d(sp, px, py, k, &state);
    }
    return RRT_OK;
}

int rrt_png_host_probe(const char* path, uint32_t* width, uint32_t* height, uint8_t* rgb8, uint64_t capacity) {
    if (!path || !width || !height) return fail(RRT_ERR_INVALID, "rrt_png_host_probe: null argument");
    rrt::Image8 img;
    std::string err;
    if (!rrt::read_png_rgb8(path, &img, &err)) return fail(RRT_ERR_IO, err);
    *width = img.width;
    *height = img.height;
    if (rgb8 && capacity >= img.rgb.size()) std::memcpy(rgb8, img.rgb.data(), img.rgb.size());
    return RRT_OK;
}

int rrt_mipmap_host_probe(uint32_t width, uint32_t height, const uint8_t* rgb8, int trilinear, double max_aniso, uint32_t wrap,
                          uint64_t n, const double* q6, double* out6, uint64_t info[32]) {
    if (!rgb8 || (n && (!q6 || !out6)) || !info) return fail(RRT_ERR_INVALID, "rrt_mipmap_host_probe: null argument");
    rrt::Image8 img;
    img.width = width;
    img.height = height;
    img.rgb.assign(rgb8, rgb8 + (size_t)width * height * 3);
    rrt::HostMipMap m;
    std::string err;
    if (!rrt::make_mipmap(img, trilinear != 0, max_aniso, wrap, &m, &err)) return fail(RRT_ERR_UNSUPPORTED, err);
    const std::vector<double> lut = rrt::mip_weight_lut();
    const rrt::MipView v = m.host_view(lut.data());
    info[0] = v.n_levels;
    for (uint32_t l = 0; l < v.n_levels && l < 15; ++l) {
        info[1 + 2 * l] = v.level[l].u_res;
        info[2 + 2 * l] = v.level[l].v_res;
    }
    for (uint64_t i = 0; i < n; ++i) {
        const double* a = q6 + 6 * i;
        const rrt::Rgb d = rrt::mip_lookup_d(v, rrt::P2{a[0], a[1]}, rrt::P2{a[2], a[3]}, rrt::P2{a[4], a[5]});
        const rrt::Rgb w = rrt::mip_lookup_w(v, rrt::P2{a[0], a[1]}, a[2]);
        out6[6 * i] = d.r; out6[6 * i + 1] = d.g; out6[6 * i + 2] = d.b;
        out6[6 * i + 3] = w.r; out6[6 * i + 4] = w.g; out6[6 * i + 5] = w.b;
    }
    return RRT_OK;
}

int rrt_envlight_host_probe(uint32_t width, uint32_t height, const uint8_t* rgb8, const double to_world16[16],
                            const double to_local16[16], double world_radius, uint64_t n, const double* in8, double* out12) {
    if (!rgb8 || !to_world16 || !to_local16 || (n && (!in8 || !out12))) return fail(RRT_ERR_INVALID, "rrt_envlight_host_probe: null argument");
    rrt::Image8 img;
    img.width = width;
    img.height = height;
    img.rgb.assign(rgb8, rgb8 + (size_t)width * height * 3);
    rrt::HostMipMap m;
    std::string err;
    if (!rrt::make_mipmap(img, false, 8.0, rrt::MIPWRAP_REPEAT, &m, &err)) return fail(RRT_ERR_UNSUPPORTED, err);
    const std::vector<double> lut = rrt::mip_weight_lut();
    rrt::EnvLightView e{};
    e.lmap = m.host_view(lut.data());
    rrt::HostDist2D dist;
    rrt::make_env_distribution(e.lmap, &dist);
    e.dist = dist.host_view();
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) {
            e.to_world.m[4 * r + c] = to_world16[4 * r + c];
            e.to_local.m[4 * r + c] = to_local16[4 * r + c];
        }
    e.world_radius = world_radius;
    for (uint64_t i = 0; i < n; ++i) {
        const double* a = in8 + 8 * i;  // ref point, u (2), direction w (3)
        double* o = out12 + 12 * i;
        rrt::V3 wi = rrt::v3(0, 0, 0), p1 = rrt::v3(0, 0, 0);
        double pdf = 0.0;
        const rrt::Rgb li = rrt::env_sample_li(e, rrt::v3(a[0], a[1], a[2]), rrt::P2{a[3], a[4]}, &wi, &pdf, &p1);
        const rrt::V3 w = rrt::v3(a[5], a[6], a[7]);
        const rrt::Rgb le = rrt::env_le(e, w);
        o[0] = li.r; o[1] = li.g; o[2] = li.b; o[3] = wi.x; o[4] = wi.y; o[5] = wi.z; o[6] = pdf;
        o[7] = rrt::env_pdf_li(e, w); o[8] = le.r; o[9] = le.g; o[10] = le.b; o[11] = p1.x;
    }
    return RRT_OK;
}

}  // extern "C"
