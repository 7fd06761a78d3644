// rt_api.cu — the C ABI of include/rt_b200.h: context, scene upload (flatten to device
// SoA + LBVH build) and the render driver.  The driver is the GPU restatement of
// Scene::renderScene (src/scene.cpp:10-59): instead of N threads pulling 2000-pixel
// blocks and recursing per pixel, the frame is cut into batches of framebuffer slots (one
// batch when the queues can hold it) and every batch runs the wavefront loop
//   trace -> Morton sort of the hits -> shade -> shadow     once per bounce level,
// with the shadow kernel of level l on its own stream beside trace/shade of level l+1.
// Every level owns a ray queue of `cap` slots and a batch never exceeds cap/2 rays, so the
// <= 2 children per hit (src/scene.cpp:127,134) can never overflow the next level.  The levels
// run in a loop over an explicit stack of pending levels (process_levels), so any bounce_depth
// up to RT_MAX_DEPTH works on any host thread.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "rt_bvh.h"
#include "rt_kernels.cuh"
#include "rt_sort.cuh"

using namespace rt;

namespace {

thread_local std::string g_error = "";

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define CU(x)                                                                                  \
    do {                                                                                       \
        cudaError_t e_ = (x);                                                                  \
        if (e_ != cudaSuccess)                                                                 \
            return fail(e_ == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA, "%s: %s", #x, \
                        cudaGetErrorString(e_));                                               \
    } while (0)

// After every kernel launch: configuration errors surface immediately (no sync); with
// RT_DEBUG_SYNC=1 in the environment the stream is also synchronised so a faulting kernel
// is reported by name.
static bool debug_sync() {
    static int v = -1;
    if (v < 0) v = getenv("RT_DEBUG_SYNC") ? 1 : 0;
    return v == 1;
}
#define LAUNCHED(name, st)                                                                      \
    do {                                                                                        \
        cudaError_t e_ = cudaPeekAtLastError();                                                 \
        if (e_ == cudaSuccess && debug_sync()) e_ = cudaStreamSynchronize(st);                  \
        if (e_ != cudaSuccess) return fail(RT_ERR_CUDA, "kernel %s: %s", name, cudaGetErrorString(e_)); \
    } while (0)

#define RT_MAX_DEPTH 65535     // bounce_depth limit (check_params); counter blocks are allocated per level actually needed
#define CTR_LEVEL0 8           // word of bounce level 0's counter block: half-way into the first 128-byte line (see CTR_*)

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    cudaError_t ensure(size_t count) {
        if (count <= n && p) return cudaSuccess;
        release();
        cudaError_t e = cudaMalloc(&p, sizeof(T) * (count ? count : 1));
        if (e == cudaSuccess) n = count;
        return e;
    }
};

struct TileLayout {
    int width = 0, height = 0, world = 1, rank = 0;
    int tiles_x = 0, tiles_y = 0;
    std::vector<int> ids;            // this rank's tiles, global row-major order
    void build(int w, int h, int rank_, int world_) {
        width = w; height = h; world = world_; rank = rank_;
        tiles_x = (w + RT_TILE_W - 1) / RT_TILE_W;
        tiles_y = (h + RT_TILE_H - 1) / RT_TILE_H;
        ids.clear();
        for (int ty = 0; ty < tiles_y; ty++)
            for (int tx = 0; tx < tiles_x; tx++)
                if ((tx + ty) % world == rank) ids.push_back(ty * tiles_x + tx);
    }
    static long long count(int w, int h, int rank, int world) {
        int tx_n = (w + RT_TILE_W - 1) / RT_TILE_W, ty_n = (h + RT_TILE_H - 1) / RT_TILE_H;
        long long c = 0;
        for (int ty = 0; ty < ty_n; ty++) {
            int first = ((rank - ty) % world + world) % world;
            if (first < tx_n) c += (tx_n - first + world - 1) / world;
        }
        return c;
    }
};

// A device array of the scene: grow-only storage and the number of elements the scene holds in it.
template <typename T>
struct SceneArray : DevBuf<T> {
    size_t used = 0;
    cudaError_t hold(size_t count) { used = count; return this->ensure(count); }
};

// The scene an rt_context holds: its device arrays, the DScene that points into them, the LBVH bookkeeping of the
// hit sort and the refit, and the structure rt_scene_refit requires unchanged.
struct SceneStore {
    DScene S{};
    SceneArray<DGeom> geoms;
    SceneArray<float4> sph_bound;
    SceneArray<DMat> mats;
    SceneArray<DLight> slights, alights;
    SceneArray<double2> face_pts, face_nrm;
    SceneArray<int> flat, all_prims;
    SceneArray<BvhNode> nodes;
    // Read only by the build and the refit, on the device that built the LBVH: its primitive codes and the wide
    // level of every node slot.
    DevBuf<int> bvh_prims, node_level;
    size_t node_count = 0;
    int bvh_levels = 0;
    SortGrid sort_grid;                     // Morton grid over the LBVH primitives' centroid bounds
    bool sort_ok = false;                   // scene has an LBVH (bounds known)
    // Structure of the uploaded scene, which rt_scene_refit requires unchanged: (type, first_face, num_faces) per
    // geometry, the face count and the FaceOwner table of k_pack_faces.  tri_pts: the six object-space points of
    // every `tri` the device holds (a refit without faces derives the padding scale from them).
    std::vector<int64_t> shape;
    int64_t shape_faces = 0;
    std::vector<FaceOwner> owners;
    std::vector<double> tri_pts;

    // Calls f(array, field) for every device array a render reads, as pointers to the SceneStore member and to the
    // DScene field that points at it: the one list of them.  Stops at the first f that does not return RT_OK.
    template <typename F>
    static int each_array(F&& f) {
        int rc = RT_OK;
        auto go = [&](auto array, auto field) { if (rc == RT_OK) rc = f(array, field); };
        go(&SceneStore::geoms, &DScene::geoms);
        go(&SceneStore::sph_bound, &DScene::sph_bound);
        go(&SceneStore::mats, &DScene::mats);
        go(&SceneStore::slights, &DScene::slights);
        go(&SceneStore::alights, &DScene::alights);
        go(&SceneStore::face_pts, &DScene::face_pts);
        go(&SceneStore::face_nrm, &DScene::face_nrm);
        go(&SceneStore::flat, &DScene::flat);
        go(&SceneStore::all_prims, &DScene::all_prims);
        go(&SceneStore::nodes, &DScene::nodes);
        return rc;
    }

    // Points S at the arrays of `from`: this store's own, or those of a store on the same device.  An array the
    // scene holds nothing in stays null, so S.nodes is null without an LBVH.
    void bind(const SceneStore& from) {
        each_array([&](auto array, auto field) {
            S.*field = (from.*array).used ? (from.*array).p : nullptr;
            return RT_OK;
        });
    }
};

}  // namespace

struct rt_context {
    int device = 0;
    int num_sms = 1;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool have_scene = false;
    SceneStore scene;
    DeviceArena scratch;                    // upload / LBVH-build temporaries
    // render state
    size_t cap = 0;                         // ray-queue capacity
    bool cap_fixed = false;                 // pinned by RT_QUEUE_CAP
    // Ray queues come from a pool: a bounce level that fits one chunk hands its queue back as soon as its
    // k_trace is enqueued, so the levels of a frame ping-pong between two queues (5.1 GB each at 8K) instead of
    // holding one per level; only levels that are processed in several chunks keep theirs while they recurse.
    struct RayQueueBuf {
        DevBuf<double> f;                   // 9*cap doubles
        DevBuf<int> i;                      // 2*cap ints
        bool busy = false;
    };
    std::vector<RayQueueBuf> qpool;
    DevBuf<double> hf[2];                   // hit queues, 13*(cap/2) each: bounce level l uses buffer l & 1
    DevBuf<int> hi[2];                      // 3*(cap/2) each
    DevBuf<double> hsf;                     // unsorted hit records of the level being traced (hit sorting)
    DevBuf<int> hsi;
    DevBuf<uint32_t> skeys[2];              // radix-sort ping-pong buffers
    DevBuf<int> svals[2];
    DevBuf<int> shist;
    cudaStream_t shadow_stream = nullptr;   // k_shadow of level l overlaps trace/shade of level l+1
    cudaEvent_t ev_hq_free[2] = {nullptr, nullptr};   // last k_shadow reading hit buffer b has been enqueued up to here
    cudaEvent_t ev_join = nullptr;
    bool hq_pending[2] = {false, false};
    DevBuf<double> fb;                      // framebuffer, slot order
    DevBuf<int> tile_ids;
    DevBuf<int> ids_geom, ids_face;
    DevBuf<unsigned long long> ctr;
    DevBuf<unsigned char> staging;          // resolve target for the host-buffer entry points
    // Device counters: [0] the intersection-only maximum, then from CTR_LEVEL0 on one CTR_COUNT block per
    // bounce level (levels_alloc of them) so that level l+1 can be enqueued while level l's shadow kernel
    // still reads its own counts.
    unsigned long long* h_ctr = nullptr;    // pinned: 4 words for the per-chunk read-back (3 used), then the mirror of the level blocks
    int levels_alloc = 0;
    cudaEvent_t ev_build = nullptr;
    // ---- multi-GPU inside one process (rt_params.n_gpus > 1): this context drives `peers`, one
    // sub-context per additional device, each with a replica of the scene (see replicate_scene)
    std::vector<rt_context*> peers;
    bool peers_stale = true;                // scene uploaded since the peers were last synchronised
    int worker_rc = RT_OK;                  // result of the last worker-thread section (peers only)
    std::string worker_err;
    std::vector<void*> ipc_opened, ipc_created;
    DevBuf<int> unpack_starts;              // rt_unpack_tiles: per-rank tile-row offsets, kept while the layout is unchanged
    int unpack_key[3] = {0, 0, 0};          // width, height, world the table was built for
    cudaStream_t copy_stream = nullptr;     // counter read-backs that must not wait for k_shadow
    cudaEvent_t ev_shade = nullptr;
    TileLayout tiles;
    rt_stats stats;
    std::vector<cudaEvent_t> evpool;        // RT_FLAG_TIME_KERNELS: (start, stop) pairs
    std::vector<int> evclass;
    size_t evused = 0;
    rt_context() { memset(&stats, 0, sizeof(stats)); }
};

extern "C" {

const char* rt_last_error(void) { return g_error.c_str(); }
int rt_abi_version(void) { return RT_ABI_VERSION; }

static int init_context(rt_context* ctx, int device, int num_sms) {
    ctx->device = device;
    ctx->num_sms = num_sms;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU(cudaEventCreate(&ctx->ev0));
    CU(cudaEventCreate(&ctx->ev1));
    CU(cudaEventCreate(&ctx->ev_build));
    CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->shadow_stream, cudaStreamNonBlocking));
    for (int b = 0; b < 2; b++) CU(cudaEventCreateWithFlags(&ctx->ev_hq_free[b], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&ctx->ev_shade, cudaEventDisableTiming));
    // RT_QUEUE_CAP pins the ray-queue capacity (development / tests of the batching logic);
    // otherwise render_core sizes it from the frame
    const char* capenv = getenv("RT_QUEUE_CAP");
    ctx->cap_fixed = capenv != nullptr;
    ctx->cap = capenv ? (size_t)atoll(capenv) : ((size_t)8 << 20);
    if (ctx->cap < 2 * RT_TILE_PIXELS) ctx->cap = 2 * RT_TILE_PIXELS;
    ctx->cap = ctx->cap / (2 * RT_TILE_PIXELS) * (2 * RT_TILE_PIXELS);
    return RT_OK;
}

// counter blocks for bounce levels 0..levels-1 (device + pinned mirror)
static int ensure_levels(rt_context* ctx, int levels) {
    if (levels <= ctx->levels_alloc) return RT_OK;
    int want = std::max(levels, 16);
    if (ctx->h_ctr) { cudaFreeHost(ctx->h_ctr); ctx->h_ctr = nullptr; }
    ctx->levels_alloc = 0;
    CU(cudaMallocHost(&ctx->h_ctr, sizeof(unsigned long long) * ((size_t)want * CTR_COUNT + 4)));
    CU(ctx->ctr.ensure(CTR_LEVEL0 + (size_t)want * CTR_COUNT));
    ctx->levels_alloc = want;
    return RT_OK;
}

int rt_create(int device, rt_context** out) {
    if (!out) return fail(RT_ERR_INVALID, "rt_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(RT_ERR_NO_DEVICE, "no usable CUDA device (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    }
    if (device >= count) return fail(RT_ERR_NO_DEVICE, "CUDA device %d does not exist (%d present)", device, count);
    CU(cudaSetDevice(device));
    // three attributes instead of cudaGetDeviceProperties (which queries everything and costs milliseconds of a
    // short run's start-up)
    int major = 0, minor = 0, sms = 0;
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    CU(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (major < 10)
        return fail(RT_ERR_NO_DEVICE, "device %d (sm_%d%d) is not sm_100-class; kernels are built for sm_100a only", device, major, minor);
    rt_context* ctx = new rt_context();
    int rc = init_context(ctx, device, sms);
    if (rc == RT_OK) rc = ensure_levels(ctx, 16);
    if (rc != RT_OK) {
        rt_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return RT_OK;
}

void rt_destroy(rt_context* ctx) {
    if (!ctx) return;
    for (rt_context* p : ctx->peers) rt_destroy(p);
    ctx->peers.clear();
    cudaSetDevice(ctx->device);
    for (void* p : ctx->ipc_opened) cudaIpcCloseMemHandle(p);
    for (void* p : ctx->ipc_created) cudaFree(p);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->shadow_stream) cudaStreamDestroy(ctx->shadow_stream);
    for (int b = 0; b < 2; b++)
        if (ctx->ev_hq_free[b]) cudaEventDestroy(ctx->ev_hq_free[b]);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->ev_shade) cudaEventDestroy(ctx->ev_shade);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_build) cudaEventDestroy(ctx->ev_build);
    for (cudaEvent_t e : ctx->evpool) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

// faces_kept: a refit that keeps the faces on the device passes no face arrays.
static int validate_scene(const rt_scene* s, bool faces_kept) {
    if (!s) return fail(RT_ERR_INVALID, "scene is NULL");
    if (s->num_geometries < 0 || s->num_lights < 0 || s->num_materials < 0 || s->num_faces < 0)
        return fail(RT_ERR_INVALID, "negative count in scene descriptor");
    if (s->num_faces > PRIM_INDEX_MASK) return fail(RT_ERR_INVALID, "too many faces (%lld)", (long long)s->num_faces);
    if ((s->num_geometries && !s->geometries) || (s->num_lights && !s->lights) ||
        (s->num_materials && !s->materials) || (s->num_faces && !faces_kept && (!s->face_points || !s->face_normals)))
        return fail(RT_ERR_INVALID, "NULL array in scene descriptor");
    for (int i = 0; i < s->num_geometries; i++) {
        const rt_geometry& g = s->geometries[i];
        if (g.type != RT_GEOM_SPHERE && g.type != RT_GEOM_TRI && g.type != RT_GEOM_MESH)
            return fail(RT_ERR_INVALID, "geometry %d: unknown type %d", i, g.type);
        if (g.material < 0 || g.material >= s->num_materials)
            return fail(RT_ERR_INVALID, "geometry %d: material index %d out of range", i, g.material);
        if (g.type != RT_GEOM_SPHERE) {
            if (g.first_face < 0 || g.num_faces < 0 || g.first_face + g.num_faces > s->num_faces)
                return fail(RT_ERR_INVALID, "geometry %d: face range out of bounds", i);
            if (g.type == RT_GEOM_TRI && g.num_faces != 2)
                return fail(RT_ERR_INVALID, "geometry %d: a `tri` must have exactly 2 faces", i);
        }
    }
    for (int i = 0; i < s->num_lights; i++) {
        int t = s->lights[i].type;
        if (t != RT_LIGHT_AMBIENT && t != RT_LIGHT_POINT && t != RT_LIGHT_DIRECTIONAL)
            return fail(RT_ERR_INVALID, "light %d: unknown type %d", i, t);
    }
    return RT_OK;
}

}  // extern "C"

namespace {

// Host-side conversion of a scene descriptor, shared by rt_scene_upload and rt_scene_refit.
struct SceneConv {
    std::vector<DGeom> geoms;
    std::vector<DMat> mats;
    std::vector<DLight> slights, alights;
    std::vector<float4> sph_bound;       // per geometry: world-space bounding sphere of a SPHERE (FP32 pre-test)
    std::vector<int> simple_codes;       // prim codes of the spheres and `tri`s, geometry order
    std::vector<double> simple_ext;      // world-space extent (largest axis) of each of them
    double simple_lo[3] = {1e300, 1e300, 1e300}, simple_hi[3] = {-1e300, -1e300, -1e300};   // union of their boxes
    std::vector<double> tri_pts;         // the six object-space points of every `tri`, geometry order
    // Every point a ray of a render can start from is the camera eye or lies on a primitive: the largest
    // |coordinate| of the eye and of the spheres and `tri`s (flat ones included; the LBVH primitives are measured
    // on the device) scales the LBVH box padding, see slab1() in rt_device.cuh.
    double origin_abs = 0;
};

// kept_tri_pts: the `tri` points to use when the descriptor carries no faces (a refit that keeps them), else null.
int convert_scene(const rt_scene* s, const std::vector<double>* kept_tri_pts, SceneConv& c) {
    const int ng = s->num_geometries;
    const bool faces_on_device = (s->flags & RT_SCENE_FACES_ON_DEVICE) != 0;
    c.geoms.resize((size_t)ng);
    c.mats.resize((size_t)s->num_materials);
    for (int i = 0; i < ng; i++) {
        const rt_geometry& g = s->geometries[i];
        DGeom& d = c.geoms[(size_t)i];
        memset(&d, 0, sizeof(d));
        memcpy(d.inv, g.inv, sizeof(d.inv));
        memcpy(d.fwd, g.fwd, sizeof(d.fwd));
        d.det = g.det;
        memcpy(d.center, g.center, sizeof(d.center));
        d.radius2 = g.radius2;
        memcpy(d.bbmin, g.bbmin, sizeof(d.bbmin));
        memcpy(d.bbmax, g.bbmax, sizeof(d.bbmax));
        d.type = g.type;
        d.mat = g.material;
        d.first_face = (int)g.first_face;
        d.num_faces = (int)g.num_faces;
        d.use_bbox = g.use_bbox;
    }
    // world-space bounding spheres of the SPHERE geometries (FP32 pre-test, rt_device.cuh)
    c.sph_bound.assign((size_t)ng, make_float4(0.f, 0.f, 0.f, 0.f));
    for (int i = 0; i < ng; i++) {
        const rt_geometry& g = s->geometries[i];
        if (g.type != RT_GEOM_SPHERE) continue;
        double cw[3], B[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};     // B = A^T A, A = linear part of fwd
        for (int a = 0; a < 3; a++) {
            cw[a] = g.fwd[4 * a] * g.center[0] + g.fwd[4 * a + 1] * g.center[1] + g.fwd[4 * a + 2] * g.center[2] + g.fwd[4 * a + 3];
            for (int i2 = 0; i2 < 3; i2++)
                for (int j2 = 0; j2 < 3; j2++) B[i2][j2] += g.fwd[4 * a + i2] * g.fwd[4 * a + j2];
        }
        // largest eigenvalue of the symmetric 3x3 B (trigonometric closed form) = sigma_max(A)^2
        double lmax;
        const double p1 = B[0][1] * B[0][1] + B[0][2] * B[0][2] + B[1][2] * B[1][2];
        if (p1 == 0) {
            lmax = std::fmax(B[0][0], std::fmax(B[1][1], B[2][2]));
        } else {
            const double q = (B[0][0] + B[1][1] + B[2][2]) / 3;
            const double p2 = (B[0][0] - q) * (B[0][0] - q) + (B[1][1] - q) * (B[1][1] - q) + (B[2][2] - q) * (B[2][2] - q) + 2 * p1;
            const double p = std::sqrt(p2 / 6);
            double C[3][3];
            for (int i2 = 0; i2 < 3; i2++)
                for (int j2 = 0; j2 < 3; j2++) C[i2][j2] = (B[i2][j2] - (i2 == j2 ? q : 0)) / p;
            double detC = C[0][0] * (C[1][1] * C[2][2] - C[1][2] * C[2][1]) - C[0][1] * (C[1][0] * C[2][2] - C[1][2] * C[2][0]) +
                          C[0][2] * (C[1][0] * C[2][1] - C[1][1] * C[2][0]);
            double r = std::fmin(1.0, std::fmax(-1.0, detC / 2));
            lmax = q + 2 * p * std::cos(std::acos(r) / 3);
        }
        // the stored centre is c rounded to FP32: grow the radius by that rounding (sum of the axes >= its length)
        const float cf[3] = {(float)cw[0], (float)cw[1], (float)cw[2]};
        double rw = std::fabs(g.radius) * std::sqrt(std::fmax(lmax, 0.0)) * (1.0 + 1e-6);
        for (int a = 0; a < 3; a++) rw += std::fabs(cw[a] - (double)cf[a]);
        c.sph_bound[(size_t)i] = make_float4(cf[0], cf[1], cf[2], std::nextafter((float)rw, INFINITY));
    }
    for (int i = 0; i < s->num_materials; i++) {
        const rt_material& m = s->materials[i];
        DMat& d = c.mats[(size_t)i];
        memset(&d, 0, sizeof(d));
        memcpy(d.ka, m.ka, sizeof(d.ka));
        memcpy(d.kd, m.kd, sizeof(d.kd));
        memcpy(d.ks, m.ks, sizeof(d.ks));
        memcpy(d.kr, m.kr, sizeof(d.kr));
        d.sp = m.sp;
        d.ior = m.ior;
        d.has_kt = !(m.kt[0] == 0 && m.kt[1] == 0 && m.kt[2] == 0);
        d.has_kr = !(m.kr[0] == 0 && m.kr[1] == 0 && m.kr[2] == 0);
    }
    for (int i = 0; i < s->num_lights; i++) {
        const rt_light& l = s->lights[i];
        DLight d;
        memset(&d, 0, sizeof(d));
        memcpy(d.v, l.v, sizeof(d.v));
        memcpy(d.color, l.color, sizeof(d.color));
        d.falloff = l.falloff;
        d.type = l.type;
        (l.type == RT_LIGHT_AMBIENT ? c.alights : c.slights).push_back(d);
    }
    // world-space extent of every sphere / `tri` (few: host side)
    for (int i = 0; i < ng; i++) {
        const rt_geometry& g = s->geometries[i];
        if (g.type == RT_GEOM_SPHERE || g.type == RT_GEOM_TRI)
            c.simple_codes.push_back(((g.type == RT_GEOM_SPHERE ? PRIM_SPHERE : PRIM_TRI) << PRIM_KIND_SHIFT) | i);
        if (g.type != RT_GEOM_TRI) continue;
        if (kept_tri_pts) continue;
        double six[18];
        if (faces_on_device) CU(cudaMemcpy(six, s->face_points + 9 * g.first_face, sizeof(six), cudaMemcpyDeviceToHost));
        else memcpy(six, s->face_points + 9 * g.first_face, sizeof(six));
        c.tri_pts.insert(c.tri_pts.end(), six, six + 18);
    }
    if (kept_tri_pts) c.tri_pts = *kept_tri_pts;
    c.simple_ext.assign(c.simple_codes.size(), 0.0);
    for (int k = 0; k < 3; k++) c.origin_abs = std::fmax(c.origin_abs, std::fabs(s->camera.eye[k]));
    size_t tri = 0;
    for (size_t k = 0; k < c.simple_codes.size(); k++) {
        const rt_geometry& g = s->geometries[c.simple_codes[k] & PRIM_INDEX_MASK];
        double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
        auto grow = [&](const double* p) {
            for (int a = 0; a < 3; a++) {
                double w = g.fwd[4 * a] * p[0] + g.fwd[4 * a + 1] * p[1] + g.fwd[4 * a + 2] * p[2] + g.fwd[4 * a + 3];
                lo[a] = std::fmin(lo[a], w);
                hi[a] = std::fmax(hi[a], w);
            }
        };
        if (g.type == RT_GEOM_SPHERE) {
            for (int v = 0; v < 8; v++) {
                double p[3] = {g.center[0] + ((v & 1) ? g.radius : -g.radius),
                               g.center[1] + ((v & 2) ? g.radius : -g.radius),
                               g.center[2] + ((v & 4) ? g.radius : -g.radius)};
                grow(p);
            }
        } else {
            for (int v = 0; v < 6; v++) grow(c.tri_pts.data() + 18 * tri + 3 * v);
            tri++;
        }
        for (int a = 0; a < 3; a++) {
            c.simple_ext[k] = std::fmax(c.simple_ext[k], hi[a] - lo[a]);
            c.origin_abs = std::fmax(c.origin_abs, std::fmax(std::fabs(lo[a]), std::fabs(hi[a])));
            c.simple_lo[a] = std::fmin(c.simple_lo[a], lo[a]);
            c.simple_hi[a] = std::fmax(c.simple_hi[a], hi[a]);
        }
    }
    return RT_OK;
}

// Arena bytes of an upload: the raw-face staging, then (reused) the LBVH build.  A refit of the same structure
// reserves the same amount, so it never reallocates.
size_t scene_scratch_bytes(const rt_scene* s, size_t n_owners, size_t n_simple, size_t n_bvh) {
    const size_t nf = (size_t)s->num_faces;
    const size_t need_faces = 2 * DeviceArena::padded(72 * nf) + DeviceArena::padded(sizeof(FaceOwner) * n_owners) +
                              2 * DeviceArena::padded(4 * n_simple) + 4096;
    return std::max(need_faces, lbvh_scratch_bytes(n_bvh));
}

// What an upload or a refit has enqueued: kernel launches and host-to-device bytes (counted by h2d).
struct SceneWork {
    int launches = 0;
    size_t h2d_bytes = 0;
};

// A host-to-device copy of an upload or a refit, counted in its rt_stats.scene_bytes_h2d.
cudaError_t h2d(SceneWork& w, void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (!bytes) return cudaSuccess;
    w.h2d_bytes += bytes;
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
}

// Raw faces (host or device memory, see RT_SCENE_FACES_ON_DEVICE) -> the 80-byte face records and the FACE codes
// of all_prims / bvh_prims (k_pack_faces).  Host faces are staged in ctx->scratch.
int pack_faces(rt_context* ctx, const rt_scene* s, const std::vector<FaceOwner>& owners, SceneWork& w) {
    cudaStream_t st = ctx->stream;
    SceneStore& sc = ctx->scene;
    const size_t nf = (size_t)s->num_faces;
    const double *raw_p = s->face_points, *raw_n = s->face_normals;
    if (!(s->flags & RT_SCENE_FACES_ON_DEVICE)) {
        double* up = ctx->scratch.take<double>(nf * 9);
        double* un = ctx->scratch.take<double>(nf * 9);
        if (!up || !un) return fail(RT_ERR_OOM, "upload scratch arena exhausted");
        CU(h2d(w, up, s->face_points, sizeof(double) * 9 * nf, st));
        CU(h2d(w, un, s->face_normals, sizeof(double) * 9 * nf, st));
        raw_p = up; raw_n = un;
    }
    FaceOwner* d_owners = ctx->scratch.take<FaceOwner>(owners.size() ? owners.size() : 1);
    if (!d_owners) return fail(RT_ERR_OOM, "upload scratch arena exhausted");
    CU(h2d(w, d_owners, owners.data(), sizeof(FaceOwner) * owners.size(), st));
    k_pack_faces<<<(unsigned)((nf + 255) / 256), 256, 0, st>>>((long long)nf, raw_p, raw_n, d_owners, (int)owners.size(),
                                                              sc.face_pts.p, sc.face_nrm.p, sc.all_prims.p, sc.bvh_prims.p);
    w.launches++;
    LAUNCHED("k_pack_faces", st);
    return RT_OK;
}

// The geometry, material and light tables to the device, and the DScene fields that count them (the material and
// light counts may change between a scene and its refit) and the camera.
int upload_tables(rt_context* ctx, const rt_scene* s, const SceneConv& c, SceneWork& w) {
    cudaStream_t st = ctx->stream;
    SceneStore& sc = ctx->scene;
    CU(sc.geoms.hold(c.geoms.size()));
    CU(sc.sph_bound.hold(c.sph_bound.size()));
    CU(sc.mats.hold(c.mats.size()));
    CU(sc.slights.hold(c.slights.size()));
    CU(sc.alights.hold(c.alights.size()));
    CU(h2d(w, sc.geoms.p, c.geoms.data(), sizeof(DGeom) * c.geoms.size(), st));
    CU(h2d(w, sc.sph_bound.p, c.sph_bound.data(), sizeof(float4) * c.sph_bound.size(), st));
    CU(h2d(w, sc.mats.p, c.mats.data(), sizeof(DMat) * c.mats.size(), st));
    CU(h2d(w, sc.slights.p, c.slights.data(), sizeof(DLight) * c.slights.size(), st));
    CU(h2d(w, sc.alights.p, c.alights.data(), sizeof(DLight) * c.alights.size(), st));
    DScene& S = sc.S;
    memcpy(&S.cam, &s->camera, sizeof(DCamera));
    S.num_geoms = (int)c.geoms.size();
    S.num_slights = (int)c.slights.size();
    S.num_alights = (int)c.alights.size();
    return RT_OK;
}

// Where the primitives of a scene go, decided on the host before anything is written: reference order (all_prims),
// then the flat / LBVH split.  Only the per-GEOMETRY bookkeeping is done here; the per-face arrays (geometry / local
// index of a face, FACE codes in reference and LBVH order) are expanded on the device by k_pack_faces from the
// FaceOwner table.
struct ScenePlan {
    std::vector<int> simple_all_pos;        // all_prims position of every sphere / `tri` code, geometry order
    std::vector<FaceOwner> owners;          // sorted by first face; no two share a face
    std::vector<int> flat_codes, bvh_codes; // bvh_codes: the spheres and `tri`s of the LBVH only
    size_t n_all = 0, n_bvh = 0;
    int group_sizes[2] = {0, 0};            // LBVH groups: those spheres and `tri`s, then the mesh faces
    int group_first_code[2] = {0, 0};       // first primitive code of each group (all build_lbvh needs from the host side)
    int single_leaf = 0;                    // an LBVH of exactly one primitive: its code
};

int plan_scene(const rt_scene* s, const SceneConv& c, ScenePlan& p) {
    const std::vector<int>& simple_codes = c.simple_codes;
    size_t n_mesh_faces = 0;
    for (int i = 0; i < s->num_geometries; i++) {
        const rt_geometry& g = s->geometries[i];
        if (g.type == RT_GEOM_SPHERE || g.type == RT_GEOM_TRI) {
            p.simple_all_pos.push_back((int)p.n_all);
            p.n_all++;
        }
        if (g.type != RT_GEOM_SPHERE && g.num_faces > 0) {
            FaceOwner o;
            o.geom = i; o.first = (int)g.first_face; o.count = (int)g.num_faces;
            o.all_off = g.type == RT_GEOM_MESH ? (int)p.n_all : -1;
            o.bvh_off = g.type == RT_GEOM_MESH ? (int)n_mesh_faces : -1;     // + n_simple_in_bvh below
            p.owners.push_back(o);
        }
        if (g.type == RT_GEOM_MESH) {
            p.n_all += (size_t)g.num_faces;
            n_mesh_faces += (size_t)g.num_faces;
        }
    }
    if (p.n_all > (size_t)INT32_MAX) return fail(RT_ERR_INVALID, "too many primitives (%zu)", p.n_all);
    int first_mesh_face_code = 0;
    for (const FaceOwner& o : p.owners)
        if (o.all_off >= 0) { first_mesh_face_code = (PRIM_FACE << PRIM_KIND_SHIFT) | o.first; break; }
    std::vector<FaceOwner>& owners = p.owners;
    std::sort(owners.begin(), owners.end(), [](const FaceOwner& a, const FaceOwner& b) { return a.first < b.first; });
    for (size_t k = 1; k < owners.size(); k++)
        if (owners[k].first < owners[k - 1].first + owners[k - 1].count)
            return fail(RT_ERR_INVALID, "geometries %d and %d share faces", owners[k - 1].geom, owners[k].geom);
    // spheres and `tri`s: few -> tested by every ray in reference order; many -> into the
    // LBVH, except giants (floors) that would bloat its upper levels.
    const size_t kFlatMax = 64, kGiantMax = 16;
    if (simple_codes.size() <= kFlatMax) {
        p.flat_codes = simple_codes;
    } else {
        double uext = 0;
        for (int a = 0; a < 3; a++) uext = std::fmax(uext, c.simple_hi[a] - c.simple_lo[a]);
        for (size_t k = 0; k < simple_codes.size(); k++) {
            if (c.simple_ext[k] > 0.5 * uext && p.flat_codes.size() < kGiantMax) p.flat_codes.push_back(simple_codes[k]);
            else p.bvh_codes.push_back(simple_codes[k]);
        }
    }
    const int n_simple_in_bvh = (int)p.bvh_codes.size();
    p.n_bvh = (size_t)n_simple_in_bvh + n_mesh_faces;
    for (FaceOwner& o : owners)
        if (o.bvh_off >= 0) o.bvh_off += n_simple_in_bvh;
    p.group_sizes[0] = n_simple_in_bvh; p.group_sizes[1] = (int)n_mesh_faces;
    p.group_first_code[0] = n_simple_in_bvh ? p.bvh_codes[0] : 0; p.group_first_code[1] = first_mesh_face_code;
    p.single_leaf = p.n_bvh == 1 ? (n_simple_in_bvh ? p.bvh_codes[0] : first_mesh_face_code) : 0;
    return RT_OK;
}

// The end of an upload or a refit, once its arrays are held and filled and ev1 is recorded: binds the DScene to the
// arrays, builds the LBVH from the upload's plan, or refits the uploaded one when plan is null, applies its padding
// scale and hit-sort grid, waits for the device, reports the times and counts, and makes the scene current.
int commit_scene(rt_context* ctx, SceneConv& c, SceneWork& w, const ScenePlan* plan) {
    SceneStore& sc = ctx->scene;
    DScene& S = sc.S;
    cudaStream_t st = ctx->stream;
    sc.bind(sc);
    float cb[6] = {0, 0, 0, 0, 0, 0}, pad_scale = 0.f;     // the LBVH primitives' centroid bounds (min xyz, max xyz)
    if (S.nodes) {
        const float extra_abs = std::nextafter((float)c.origin_abs, INFINITY);
        char err[256] = "";
        int brc = plan ? build_lbvh(S, sc.bvh_prims.p, plan->group_first_code, S.num_bvh_prims, plan->group_sizes, 2,
                                    extra_abs, st, ctx->scratch, sc.nodes.p, &sc.node_count, &w.launches, err, sizeof(err),
                                    cb, &pad_scale, sc.node_level.p, &sc.bvh_levels)
                       : refit_lbvh(S, sc.bvh_prims.p, S.num_bvh_prims, sc.node_level.p, sc.bvh_levels, sc.node_count,
                                    extra_abs, st, ctx->scratch, sc.nodes.p, &w.launches, err, sizeof(err), cb, &pad_scale);
        ctx->scratch.reset();
        if (brc != RT_OK) return fail(brc, "LBVH %s: %s", plan ? "build" : "refit", err);
    }
    S.origin_limit = S.nodes ? pad_scale : 3.0e38f;
    // Morton grid of the hit sort over the centroid bounds; none without an LBVH
    float ext = 0.f;
    for (int a = 0; a < 3; a++) ext = fmaxf(ext, cb[3 + a] - cb[a]);
    sc.sort_ok = ext > 0.f && std::isfinite(ext);
    for (int a = 0; a < 3; a++) sc.sort_grid.lo[a] = cb[a];
    sc.sort_grid.scale = sc.sort_ok ? 1024.f / ext : 0.f;
    CU(cudaEventRecord(ctx->ev_build, st));
    CU(cudaStreamSynchronize(st));
    float ms0 = 0, ms1 = 0;
    cudaEventElapsedTime(&ms0, ctx->ev0, ctx->ev1);
    cudaEventElapsedTime(&ms1, ctx->ev1, ctx->ev_build);
    sc.tri_pts = std::move(c.tri_pts);      // a refit without faces converted a copy of the ones kept
    ctx->stats.ms_upload = ms0;
    ctx->stats.ms_build = ms1;
    ctx->stats.kernel_launches = (uint64_t)w.launches;
    ctx->stats.scene_bytes_h2d = w.h2d_bytes;
    ctx->have_scene = true;
    ctx->peers_stale = true;
    return RT_OK;
}

}  // namespace

extern "C" {

int rt_scene_upload(rt_context* ctx, const rt_scene* s) {
    if (!ctx) return fail(RT_ERR_INVALID, "context is NULL");
    int rc = validate_scene(s, false);
    if (rc != RT_OK) return rc;
    CU(cudaSetDevice(ctx->device));
    ctx->have_scene = false;
    cudaStream_t st = ctx->stream;
    CU(cudaEventRecord(ctx->ev0, st));
    SceneConv c;
    if ((rc = convert_scene(s, nullptr, c)) != RT_OK) return rc;
    ScenePlan P;
    if ((rc = plan_scene(s, c, P)) != RT_OK) return rc;

    // ---- device arrays, copies and the packing kernels ----
    SceneStore& sc = ctx->scene;
    DScene& S = sc.S;
    memset(&S, 0, sizeof(S));
    SceneWork w;
    if ((rc = upload_tables(ctx, s, c, w)) != RT_OK) return rc;
    const size_t nf = (size_t)s->num_faces;
    CU(sc.flat.hold(P.flat_codes.size()));
    CU(sc.all_prims.hold(P.n_all));
    CU(sc.bvh_prims.ensure(P.n_bvh));
    CU(sc.face_pts.hold(nf * RT_FACE_D2));
    CU(sc.face_nrm.hold(nf * RT_FACE_D2));
    CU(h2d(w, sc.flat.p, P.flat_codes.data(), sizeof(int) * P.flat_codes.size(), st));
    CU(h2d(w, sc.bvh_prims.p, P.bvh_codes.data(), sizeof(int) * P.bvh_codes.size(), st));
    // one arena reservation covers the raw-face staging and (afterwards, reused) the LBVH build
    const std::vector<int>& simple_codes = c.simple_codes;
    CU(ctx->scratch.reserve(scene_scratch_bytes(s, P.owners.size(), simple_codes.size(), P.n_bvh)));
    if (!simple_codes.empty()) {
        int* d_pos = ctx->scratch.take<int>(simple_codes.size());
        int* d_code = ctx->scratch.take<int>(simple_codes.size());
        if (!d_pos || !d_code) return fail(RT_ERR_OOM, "upload scratch arena exhausted");
        CU(h2d(w, d_pos, P.simple_all_pos.data(), sizeof(int) * simple_codes.size(), st));
        CU(h2d(w, d_code, simple_codes.data(), sizeof(int) * simple_codes.size(), st));
        k_scatter_codes<<<(unsigned)((simple_codes.size() + 255) / 256), 256, 0, st>>>((int)simple_codes.size(), d_pos, d_code,
                                                                                    sc.all_prims.p);
        w.launches++;
        LAUNCHED("k_scatter_codes", st);
    }
    if (nf && (rc = pack_faces(ctx, s, P.owners, w)) != RT_OK) return rc;
    CU(cudaStreamSynchronize(st));
    ctx->scratch.reset();
    S.num_flat = (int)P.flat_codes.size();
    S.num_all = (int)P.n_all;
    S.num_bvh_prims = (int)P.n_bvh;
    S.single_leaf = P.single_leaf;
    CU(cudaEventRecord(ctx->ev1, st));
    sc.nodes.used = sc.node_count = 0;
    if (P.n_bvh >= 2) {
        CU(sc.nodes.hold(P.n_bvh + 2));
        CU(sc.node_level.ensure(P.n_bvh + 2));
    }
    sc.shape_faces = s->num_faces;
    sc.shape.clear();
    for (int i = 0; i < s->num_geometries; i++)
        sc.shape.insert(sc.shape.end(), {s->geometries[i].type, s->geometries[i].first_face, s->geometries[i].num_faces});
    sc.owners = std::move(P.owners);
    return commit_scene(ctx, c, w, &P);
}

int rt_scene_refit(rt_context* ctx, const rt_scene* s) {
    // ---- validation: nothing is written before it passes ----
    if (!ctx) return fail(RT_ERR_INVALID, "context is NULL");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, "rt_scene_refit: rt_scene_upload has not been called");
    if (s && (s->face_points == nullptr) != (s->face_normals == nullptr))
        return fail(RT_ERR_INVALID, "rt_scene_refit: face_points and face_normals must both be set or both be NULL");
    const bool keep_faces = s && s->face_points == nullptr;
    int rc = validate_scene(s, keep_faces);
    if (rc != RT_OK) return rc;
    SceneStore& sc = ctx->scene;
    const int ng = s->num_geometries;
    if ((size_t)ng * 3 != sc.shape.size())
        return fail(RT_ERR_INVALID, "rt_scene_refit: num_geometries %d differs from the uploaded scene's %zu", ng,
                    sc.shape.size() / 3);
    if (s->num_faces != sc.shape_faces)
        return fail(RT_ERR_INVALID, "rt_scene_refit: num_faces %lld differs from the uploaded scene's %lld",
                    (long long)s->num_faces, (long long)sc.shape_faces);
    for (int i = 0; i < ng; i++) {
        const rt_geometry& g = s->geometries[i];
        const int64_t* u = sc.shape.data() + 3 * (size_t)i;
        const int64_t got[3] = {g.type, g.first_face, g.num_faces};
        static const char* const field[3] = {"type", "first_face", "num_faces"};
        for (int f = 0; f < 3; f++)
            if (got[f] != u[f])
                return fail(RT_ERR_INVALID, "rt_scene_refit: geometry %d: %s %lld differs from the uploaded scene's %lld", i,
                            field[f], (long long)got[f], (long long)u[f]);
    }
    CU(cudaSetDevice(ctx->device));
    SceneConv c;
    if ((rc = convert_scene(s, keep_faces ? &sc.tri_pts : nullptr, c)) != RT_OK) return rc;

    // ---- writes: from here a failure leaves no scene, like a failed upload ----
    ctx->have_scene = false;
    cudaStream_t st = ctx->stream;
    CU(cudaEventRecord(ctx->ev0, st));
    SceneWork w;
    if ((rc = upload_tables(ctx, s, c, w)) != RT_OK) return rc;
    // the upload reserved this much already: no allocation
    CU(ctx->scratch.reserve(scene_scratch_bytes(s, sc.owners.size(), c.simple_codes.size(), (size_t)sc.S.num_bvh_prims)));
    if (!keep_faces && s->num_faces && (rc = pack_faces(ctx, s, sc.owners, w)) != RT_OK) return rc;
    ctx->scratch.reset();       // the refit's launches are stream-ordered after k_pack_faces: the staging is free
    CU(cudaEventRecord(ctx->ev1, st));
    return commit_scene(ctx, c, w, nullptr);
}

}  // extern "C"

// ---- render driver --------------------------------------------------------------
namespace {

struct RenderJob {
    rt_context* ctx;
    const rt_params* p;
    cudaStream_t st;
    bool brute, count, timed, overlap;
    bool sort;                     // Morton-sort the hits of levels with at least sort_min_rays rays
    size_t sort_min_rays;          // levels with fewer rays are not worth the extra launches
    int* ids_geom;
    int* ids_face;
    unsigned long long* maxbits;   // intersection-only
    uint64_t launches;
    int max_level;                 // deepest bounce level that held rays
    PrimaryRays primary;           // bounce level 0 without a ray queue: k_trace generates the camera rays itself
    // progress reporting (Scene::ProgressHandler, src/scene.cpp:41-47: every 100 ms on the calling thread)
    rt_progress_fn cb;
    void* cb_user;
    long long px_total, px_before_batch, px_batch, px_reported;
    std::chrono::steady_clock::time_point last_cb;
};

// Called wherever the host has just synchronised with the device anyway (the per-level counter read-back):
// reports at most every 100 ms, like the reference's polling loop.  `frac` = share of the current batch that
// is behind us (estimated from the bounce level reached); the reported value never decreases and stays below
// the total until the final (total, total) call of render_core.
void progress_tick(RenderJob& J, double frac) {
    if (!J.cb) return;
    const auto now = std::chrono::steady_clock::now();
    if (now - J.last_cb < std::chrono::milliseconds(100)) return;
    long long done = J.px_before_batch + (long long)(frac * (double)J.px_batch);
    done = std::min(done, J.px_total - 1);
    if (done <= J.px_reported) return;
    J.px_reported = done;
    J.last_cb = now;
    J.cb((int)done, (int)J.px_total, J.cb_user);
}

// RT_FLAG_TIME_KERNELS: a (start, stop) event pair around one launch of kernel class `cls`.
struct LaunchTimer {
    RenderJob& J;
    size_t idx = 0;
    bool on;
    cudaStream_t st;
    LaunchTimer(RenderJob& j, int cls, cudaStream_t stream = nullptr) : J(j), on(j.timed), st(stream ? stream : j.st) {
        if (!on) return;
        rt_context* c = J.ctx;
        if (c->evused + 2 > c->evpool.size()) {
            for (int k = 0; k < 2; k++) {
                cudaEvent_t e;
                cudaEventCreate(&e);
                c->evpool.push_back(e);
            }
            c->evclass.resize(c->evpool.size() / 2);
        }
        idx = c->evused;
        c->evclass[idx / 2] = cls;
        c->evused += 2;
        cudaEventRecord(c->evpool[idx], st);
    }
    ~LaunchTimer() {
        if (on) cudaEventRecord(J.ctx->evpool[idx + 1], st);
    }
};

RayQ pool_queue(rt_context* ctx, int qi) {
    RayQ q;
    q.f = ctx->qpool[(size_t)qi].f.p;
    q.pixel = ctx->qpool[(size_t)qi].i.p;
    q.meta = ctx->qpool[(size_t)qi].i.p + ctx->cap;
    q.cap = ctx->cap;
    return q;
}

// A free ray queue of the current capacity (allocated on first use, kept across frames).
int acquire_queue(rt_context* ctx, int* out) {
    int qi = -1;
    for (size_t k = 0; k < ctx->qpool.size(); k++)
        if (!ctx->qpool[k].busy) { qi = (int)k; break; }
    if (qi < 0) {
        ctx->qpool.emplace_back();
        qi = (int)ctx->qpool.size() - 1;
    }
    CU(ctx->qpool[(size_t)qi].f.ensure(9 * ctx->cap));
    CU(ctx->qpool[(size_t)qi].i.ensure(2 * ctx->cap));
    ctx->qpool[(size_t)qi].busy = true;
    *out = qi;
    return RT_OK;
}
void release_queue(rt_context* ctx, int qi) { ctx->qpool[(size_t)qi].busy = false; }

template <bool BRUTE, bool COUNT, bool PRIMARY = false>
int launch_trace(RenderJob& J, RayQ q, size_t off, int n, size_t nfront, HitQ h, unsigned long long* lc) {
    LaunchTimer lt(J, 0);
    k_trace<BRUTE, COUNT, PRIMARY><<<(n + RT_BLOCK - 1) / RT_BLOCK, RT_BLOCK, 0, J.st>>>(J.ctx->scene.S, q, off, n, nfront, h, lc,
                                                                                     J.ids_geom, J.ids_face, J.primary);
    J.launches++;
    LAUNCHED("k_trace", J.st);
    return RT_OK;
}
template <bool BRUTE, bool COUNT>
int launch_shadow(RenderJob& J, int n, HitQ h, unsigned long long* lc, cudaStream_t st) {
    unsigned long long threads = (unsigned long long)n * (unsigned)J.ctx->scene.S.num_slights;
    if (!threads) return RT_OK;
    LaunchTimer lt(J, 2, st);
    k_shadow<BRUTE, COUNT><<<(unsigned)((threads + RT_BLOCK - 1) / RT_BLOCK), RT_BLOCK, 0, st>>>(J.ctx->scene.S, h, lc, J.ctx->fb.p);
    J.launches++;
    LAUNCHED("k_shadow", st);
    return RT_OK;
}

// Runs the rays of one batch: bounce level 0 (n rays in ray queue q0, or generated inside k_trace when q0 < 0)
// and everything they spawn.  A level with more rays than half a queue is processed in chunks, depth-first: each
// chunk's descendants run before the level's next chunk.  The levels still to run are kept on an explicit stack,
// so the bounce depth is bounded by heap memory rather than by the calling thread's stack.  A level's queue is
// handed back to the pool once its last chunk has been traced.
int process_levels(RenderJob& J, int q0, size_t n) {
    struct Pending {
        int level, qi;             // qi < 0: level 0, rays generated inside k_trace
        size_t n, nfront, off;     // rays, of which nfront at the front of the queue; first ray of the next chunk
    };
    rt_context* ctx = J.ctx;
    const size_t maxchunk = ctx->cap / 2;
    const bool io = J.p->intersection_only != 0;
    const bool ids_only = J.ids_geom != nullptr;
    unsigned long long* h_counts = ctx->h_ctr;
    std::vector<Pending> pending{{0, q0, n, n, 0}};
    while (!pending.empty()) {
        const Pending e = pending.back();
        const int level = e.level;
        const size_t off = e.off;
        const int m = (int)std::min(maxchunk, e.n - off);
        const bool last_chunk = off + maxchunk >= e.n;
        if (last_chunk) pending.pop_back();
        else pending.back().off += maxchunk;
        J.max_level = std::max(J.max_level, level);
        // Hit queue b = level & 1.  k_shadow runs on its own stream: it only reads this level's hit
        // queue and counters and adds into the framebuffer, so the next level's k_trace / k_shade
        // (other hit buffer, other counters) run beside it and fill the tail of the small launches.
        const int b = J.overlap ? (level & 1) : 0;
        cudaStream_t sst = J.overlap ? ctx->shadow_stream : J.st;
        HitQ h;
        h.f = ctx->hf[b].p;
        h.pixel = ctx->hi[b].p;
        h.geom = ctx->hi[b].p + maxchunk;
        h.meta = ctx->hi[b].p + 2 * maxchunk;
        h.cap = maxchunk;
        // this level's counter block (CTR_HITS, CTR_NEXT, CTR_NEXT_T are reset per chunk, the rest accumulate)
        unsigned long long* lc = ctx->ctr.p + CTR_LEVEL0 + (size_t)level * CTR_COUNT;
        const bool fused_primary = e.qi < 0;
        RayQ q;
        memset(&q, 0, sizeof(q));
        if (!fused_primary) q = pool_queue(ctx, e.qi);
        if (J.overlap && ctx->hq_pending[b]) {
            // the shadow kernel that read this hit buffer (and possibly this counter block) last
            CU(cudaStreamWaitEvent(J.st, ctx->ev_hq_free[b], 0));
            ctx->hq_pending[b] = false;
        }
        static_assert(CTR_NEXT == CTR_HITS + 1 && CTR_NEXT_T == CTR_HITS + 2, "one range per chunk");
        CU(cudaMemsetAsync(lc + CTR_HITS, 0, sizeof(unsigned long long) * 3, J.st));
        int lrc;
        const bool sorting = J.sort && (size_t)m >= J.sort_min_rays;
        HitQ ht = h;               // where k_trace appends
        if (sorting) {
            ht.f = ctx->hsf.p;
            ht.pixel = ctx->hsi.p;
            ht.geom = ctx->hsi.p + maxchunk;
            ht.meta = ctx->hsi.p + 2 * maxchunk;
        }
        if (fused_primary) lrc = J.count ? launch_trace<false, true, true>(J, q, off, m, e.nfront, ht, lc) : launch_trace<false, false, true>(J, q, off, m, e.nfront, ht, lc);
        else if (J.brute) lrc = J.count ? launch_trace<true, true>(J, q, off, m, e.nfront, ht, lc) : launch_trace<true, false>(J, q, off, m, e.nfront, ht, lc);
        else lrc = J.count ? launch_trace<false, true>(J, q, off, m, e.nfront, ht, lc) : launch_trace<false, false>(J, q, off, m, e.nfront, ht, lc);
        if (lrc != RT_OK) return lrc;
        // everything enqueued on J.st from here on runs after this k_trace, the last reader of the queue
        if (last_chunk && !fused_primary) release_queue(ctx, e.qi);
        if (ids_only) continue;
        const int* sorted_order = nullptr;
        if (sorting) {
            LaunchTimer lt(J, 3);
            const unsigned sb = (unsigned)((m + 255) / 256);
            uint32_t *kin = ctx->skeys[0].p, *kout = ctx->skeys[1].p;
            int *vin = ctx->svals[0].p, *vout = ctx->svals[1].p;
            k_hit_keys<<<sb, 256, 0, J.st>>>(ht, lc, ctx->scene.sort_grid, kin, vin);
            int nl = 0;
            sort_pairs(J.st, kin, kout, vin, vout, ctx->shist.p, m, lc + CTR_HITS, &nl);
            sorted_order = vin;                 // k_shade gathers through it and writes the sorted queue
            J.launches += 1 + (uint64_t)nl;
            LAUNCHED("hit sort", J.st);
        }
        const unsigned blocks = (unsigned)((m + RT_BLOCK - 1) / RT_BLOCK);
        if (io) {
            LaunchTimer lt(J, 1);
            k_shade_io<<<blocks, RT_BLOCK, 0, J.st>>>(h, lc, ctx->fb.p, J.maxbits);
            J.launches++;
            LAUNCHED("k_shade_io", J.st);
            continue;
        }
        const bool last_level = level >= J.p->bounce_depth;
        int nqi = -1;
        RayQ next = q;                          // unused by k_shade on the last level (depth 0: nothing is spawned)
        if (last_level && fused_primary) {      // ... but it must be a valid queue descriptor all the same
            next.cap = 1;
        }
        if (!last_level) {
            int rc = acquire_queue(ctx, &nqi);
            if (rc != RT_OK) return rc;
            next = pool_queue(ctx, nqi);
        }
        {
            LaunchTimer lt(J, 1);
            k_shade<<<(unsigned)((m + RT_SHADE_BLOCK - 1) / RT_SHADE_BLOCK), RT_SHADE_BLOCK, 0, J.st>>>(
                ctx->scene.S, sorted_order ? ht : h, h, sorted_order, lc, next, ctx->fb.p);
        }
        J.launches++;
        LAUNCHED("k_shade", J.st);
        // The hit and spawn counts are final once k_shade is done: read them back on a side
        // stream while k_shadow runs, so the next level is enqueued before the GPU goes idle.
        CU(cudaEventRecord(ctx->ev_shade, J.st));
        CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_shade, 0));
        CU(cudaMemcpyAsync(h_counts, lc + CTR_HITS, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, ctx->copy_stream));
        if (J.overlap) CU(cudaStreamWaitEvent(sst, ctx->ev_shade, 0));
        if (J.brute) lrc = J.count ? launch_shadow<true, true>(J, m, h, lc, sst) : launch_shadow<true, false>(J, m, h, lc, sst);
        else lrc = J.count ? launch_shadow<false, true>(J, m, h, lc, sst) : launch_shadow<false, false>(J, m, h, lc, sst);
        if (lrc != RT_OK) return lrc;
        if (J.overlap) {
            CU(cudaEventRecord(ctx->ev_hq_free[b], sst));
            ctx->hq_pending[b] = true;
        }
        CU(cudaStreamSynchronize(ctx->copy_stream));
        const unsigned long long nhits = h_counts[0], nrefl = h_counts[1], nnext = nrefl + h_counts[2];
        ctx->stats.hits += nhits;
        ctx->stats.rays_shadow += nhits * (unsigned long long)ctx->scene.S.num_slights;
        ctx->stats.rays_secondary += nnext;
        if (level == 0) progress_tick(J, 0.5 * (double)(off + (size_t)m) / (double)e.n);
        else progress_tick(J, 1.0 - 0.5 / (double)(level + 1));
        if (nnext > 0) {
            if (last_level) return fail(RT_ERR_CUDA, "internal: rays spawned past the depth limit");
            pending.push_back({level + 1, nqi, (size_t)nnext, (size_t)nrefl, 0});
        } else if (nqi >= 0) {
            release_queue(ctx, nqi);
        }
    }
    return RT_OK;
}

int check_params(rt_context* ctx, const rt_params* p) {
    if (!ctx) return fail(RT_ERR_INVALID, "context is NULL");
    if (!p) return fail(RT_ERR_INVALID, "params is NULL");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, "rt_scene_upload has not been called");
    if (p->width <= 0 || p->height <= 0) return fail(RT_ERR_INVALID, "width and height must be positive");
    if ((long long)p->width * p->height > 2000000000ll) return fail(RT_ERR_INVALID, "frame too large");
    if (p->bounce_depth < 0 || p->bounce_depth > RT_MAX_DEPTH) return fail(RT_ERR_INVALID, "bounce_depth must be in [0,%d]", RT_MAX_DEPTH);
    if (p->tile_world < 1 || p->tile_rank < 0 || p->tile_rank >= p->tile_world)
        return fail(RT_ERR_INVALID, "tile_rank/tile_world out of range");
    if (p->samples < 0 || p->samples > RT_MAX_SAMPLES) return fail(RT_ERR_INVALID, "samples must be in [0,%d]", RT_MAX_SAMPLES);
    if (p->samples > 1 && p->intersection_only) return fail(RT_ERR_INVALID, "supersampling is not defined for intersection_only");
    if (p->n_gpus < 0 || p->n_gpus > 64) return fail(RT_ERR_INVALID, "n_gpus must be in [0,64]");
    if (p->n_gpus > 1 && p->tile_world != 1 && !(p->flags & RT_FLAG_FULL_FRAME))
        return fail(RT_ERR_INVALID, "n_gpus > 1 with tile_world > 1 needs RT_FLAG_FULL_FRAME");
    return RT_OK;
}

// Renders this rank's tiles into ctx->fb (slot order).  ids: also/only record primary hit ids.
int render_core(rt_context* ctx, const rt_params* p, cudaStream_t st, bool ids_only, rt_progress_fn cb, void* user,
                bool final_cb = true) {
    int rc = check_params(ctx, p);
    if (rc != RT_OK) return rc;
    CU(cudaSetDevice(ctx->device));
    TileLayout& T = ctx->tiles;
    if (T.width != p->width || T.height != p->height || T.rank != p->tile_rank || T.world != p->tile_world ||
        ctx->tile_ids.n != T.ids.size() || T.ids.empty()) {
        T.build(p->width, p->height, p->tile_rank, p->tile_world);
        CU(ctx->tile_ids.ensure(T.ids.size()));
        if (!T.ids.empty())
            CU(cudaMemcpyAsync(ctx->tile_ids.p, T.ids.data(), sizeof(int) * T.ids.size(), cudaMemcpyHostToDevice, st));
    }
    const long long nslots = (long long)T.ids.size() * RT_TILE_PIXELS;
    CU(ctx->fb.ensure((size_t)nslots * 3));
    if (!ctx->cap_fixed) {
        // One batch per frame when it fits: small launches end in a long latency-bound tail
        // (measured on B200, 8K synthetic frame: k_trace 52.5 ms with 8 Mi-slot queues, 44.7 ms
        // with 64 Mi).  64 Mi slots = 5.1 GB per bounce level, 3.7 GB of hit queue.
        const size_t unit = 2 * RT_TILE_PIXELS, lo = (size_t)1 << 20, hi = (size_t)64 << 20;
        const size_t ss = p->samples > 1 ? (size_t)p->samples * p->samples : 1;
        size_t want = (2 * (size_t)nslots * ss + unit - 1) / unit * unit;
        ctx->cap = std::min(std::max(want, lo), hi);
    }
    const size_t maxchunk = ctx->cap / 2;
    const bool overlap = !(p->flags & RT_FLAG_SERIAL) && !ids_only && !p->intersection_only;
    for (int b = 0; b < (overlap ? 2 : 1); b++) {
        CU(ctx->hf[b].ensure(13 * maxchunk));
        CU(ctx->hi[b].ensure(3 * maxchunk));
    }
    rc = ensure_levels(ctx, p->bounce_depth + 1);
    if (rc != RT_OK) return rc;
    // Every pool queue is free at the start of a render.  This is what lets process_levels return from an error
    // without handing back the queues it holds.
    for (auto& qb : ctx->qpool) qb.busy = false;

    RenderJob J;
    J.ctx = ctx; J.p = p; J.st = st;
    J.brute = (p->flags & RT_FLAG_BRUTE_FORCE) != 0;
    J.count = (p->flags & RT_FLAG_COUNT_WORK) != 0;
    J.timed = (p->flags & RT_FLAG_TIME_KERNELS) != 0;
    J.overlap = overlap;
    {   // Hit sorting (k_hit_keys): pays when divergence is expensive, i.e. on big LBVHs — measured on
        // B200: 1M-triangle scene at 8K 160.6 -> 107.2 ms; bunny (5k faces) at 4K 13.2 -> 12.2 ms.
        // RT_HIT_SORT_MIN_RAYS lowers the level size from which it is worth its launches (tests: 1).
        const char* mr = getenv("RT_HIT_SORT_MIN_RAYS");
        J.sort_min_rays = mr ? (size_t)atoll(mr) : 262144;
        J.sort = ctx->scene.sort_ok && !J.brute && p->bounce_depth >= 1 && !ids_only && !p->intersection_only;
    }
    if (J.sort) {
        CU(ctx->hsf.ensure(13 * maxchunk));
        CU(ctx->hsi.ensure(3 * maxchunk));
        for (int k = 0; k < 2; k++) {
            CU(ctx->skeys[k].ensure(maxchunk));
            CU(ctx->svals[k].ensure(maxchunk));
        }
        CU(ctx->shist.ensure((size_t)256 * (SORT_MAX_BLOCKS + 1)));
    }
    ctx->hq_pending[0] = ctx->hq_pending[1] = false;
    ctx->evused = 0;
    J.ids_geom = nullptr; J.ids_face = nullptr;
    J.maxbits = ctx->ctr.p;
    const size_t n_ctr = CTR_LEVEL0 + (size_t)(p->bounce_depth + 1) * CTR_COUNT;
    J.launches = 0;
    J.max_level = 0;
    J.cb = cb; J.cb_user = user;
    J.px_total = (long long)p->width * p->height;
    J.px_before_batch = J.px_batch = 0;
    J.px_reported = -1;
    J.last_cb = std::chrono::steady_clock::now();
    if (ids_only) {
        CU(ctx->ids_geom.ensure((size_t)nslots));
        CU(ctx->ids_face.ensure((size_t)nslots));
        CU(cudaMemsetAsync(ctx->ids_geom.p, 0xff, sizeof(int) * (size_t)nslots, st));
        CU(cudaMemsetAsync(ctx->ids_face.p, 0xff, sizeof(int) * (size_t)nslots, st));
        J.ids_geom = ctx->ids_geom.p;
        J.ids_face = ctx->ids_face.p;
    }
    rt_stats& stats = ctx->stats;
    stats.rays_primary = stats.rays_shadow = stats.rays_secondary = stats.hits = stats.degenerate_rays = 0;
    stats.shadow_rays_culled = 0;
    stats.ms_readback = 0;
    for (int k = 0; k < 2; k++) stats.nodes_fetched[k] = stats.tris_tested[k] = stats.spheres_tested[k] = 0;
    for (int k = 0; k < 4; k++) { stats.ms_kernel[k] = 0; stats.launches_kernel[k] = 0; }
    CU(cudaMemsetAsync(ctx->ctr.p, 0, sizeof(unsigned long long) * n_ctr, st));
    if (p->intersection_only) {
        // std::numeric_limits<double>::min() (src/scene.cpp:51)
        const unsigned long long dblmin = 0x0010000000000000ull;
        CU(cudaMemcpyAsync(J.maxbits, &dblmin, sizeof(dblmin), cudaMemcpyHostToDevice, st));
    }
    CU(cudaMemsetAsync(ctx->fb.p, 0, sizeof(double) * (size_t)nslots * 3, st));
    CU(cudaEventRecord(ctx->ev0, st));

    FrameInfo F;
    F.width = p->width; F.height = p->height; F.tiles_x = T.tiles_x; F.tiles_y = T.tiles_y; F.tile_ids = ctx->tile_ids.p;
    const long long total_px = (long long)p->width * p->height;
    const int sub = p->samples > 1 ? p->samples : 1;
    if (sub > 1 && ids_only) return fail(RT_ERR_INVALID, "primary ids are per pixel: render them with samples <= 1");
    // slots per batch: a batch's primary rays (sub^2 per slot) must fit half a queue
    const long long slots_per_batch = std::max<long long>((long long)maxchunk / (sub * sub), 1);
    for (long long first = 0; first < nslots; first += slots_per_batch) {
        const long long nslot_batch = std::min<long long>(slots_per_batch, nslots - first);
        const int n = (int)(nslot_batch * sub * sub);
        J.primary.F = F; J.primary.first_slot = first; J.primary.sub = sub; J.primary.depth = p->bounce_depth;
        int q0 = -1;                   // stays -1 when k_trace generates the camera rays itself
        if (J.brute) {
            rc = acquire_queue(ctx, &q0);
            if (rc != RT_OK) return rc;
            {
                LaunchTimer lt(J, 3);
                k_raygen<<<(n + RT_BLOCK - 1) / RT_BLOCK, RT_BLOCK, 0, st>>>(ctx->scene.S, J.primary, n, pool_queue(ctx, q0));
            }
            J.launches++;
            LAUNCHED("k_raygen", st);
        }
        // progress is counted in pixels of the WHOLE frame: this context's slots stand for tile_world times as many
        J.px_before_batch = std::min<long long>(first * (long long)p->tile_world, total_px - 1);
        J.px_batch = std::min<long long>(nslot_batch * (long long)p->tile_world, total_px - 1 - J.px_before_batch);
        rc = process_levels(J, q0, (size_t)n);
        if (rc != RT_OK) return rc;
        progress_tick(J, 1.0);
    }
    if (overlap) {      // the shadow stream's framebuffer adds must land before anything reads the frame
        CU(cudaEventRecord(ctx->ev_join, ctx->shadow_stream));
        CU(cudaStreamWaitEvent(st, ctx->ev_join, 0));
    }
    if (p->intersection_only && !ids_only && p->tile_world == 1) {
        // global max normalisation (src/scene.cpp:50-58); with tile_world > 1 the caller
        // all-reduces the max across ranks first (rt_io_get_max / rt_io_normalize)
        k_divide<<<(unsigned)(((size_t)nslots * 3 + 255) / 256), 256, 0, st>>>(ctx->fb.p, (size_t)nslots * 3, J.maxbits);
        J.launches++;
        LAUNCHED("k_divide", st);
    }
    CU(cudaEventRecord(ctx->ev1, st));
    const int used_levels = std::min(p->bounce_depth, J.max_level) + 1;
    CU(cudaMemcpyAsync(ctx->h_ctr + 4, ctx->ctr.p + CTR_LEVEL0, sizeof(unsigned long long) * (size_t)used_levels * CTR_COUNT,
                       cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    stats.ms_trace = ms;
    // primary rays == pixels of this rank's tiles that lie inside the frame
    long long prim = 0;
    for (int gt : T.ids) {
        int tx = gt % T.tiles_x, ty = gt / T.tiles_x;
        int w = std::min(RT_TILE_W, p->width - tx * RT_TILE_W), hgt = std::min(RT_TILE_H, p->height - ty * RT_TILE_H);
        prim += (long long)w * hgt;
    }
    stats.rays_primary = (uint64_t)prim * (uint64_t)(sub * sub);
    for (int l = 0; l < used_levels; l++) {
        const unsigned long long* c = ctx->h_ctr + 4 + (size_t)l * CTR_COUNT;
        stats.degenerate_rays += c[CTR_DEGENERATE];
        stats.nodes_fetched[0] += c[CTR_NODES];
        stats.tris_tested[0] += c[CTR_TRIS];
        stats.spheres_tested[0] += c[CTR_SPHERES];
        stats.nodes_fetched[1] += c[CTR_S_NODES];
        stats.tris_tested[1] += c[CTR_S_TRIS];
        stats.spheres_tested[1] += c[CTR_S_SPHERES];
        stats.shadow_rays_culled += c[CTR_S_CULLED];
    }
    stats.kernel_launches = J.launches;
    for (size_t k = 0; k + 1 < ctx->evused; k += 2) {
        float kms = 0;
        cudaEventElapsedTime(&kms, ctx->evpool[k], ctx->evpool[k + 1]);
        int cls = ctx->evclass[k / 2];
        stats.ms_kernel[cls] += kms;
        stats.launches_kernel[cls]++;
    }
    if (cb && final_cb) cb((int)total_px, (int)total_px, user);
    return RT_OK;
}

// Framebuffer (slot order) -> output.  full: `out` is the whole row-major frame and only this context's tiles
// are stored into it; otherwise the packed tile layout.  remote: `out` is not local device memory (another
// GPU's frame over NVLink, or pinned host memory over PCIe) -> row-staged word stores for RGB8.
template <bool QUANT>
int resolve_to(rt_context* ctx, const rt_params* p, void* out, cudaStream_t st, bool full, bool remote) {
    const long long nslots = (long long)ctx->tiles.ids.size() * RT_TILE_PIXELS;
    if (!nslots) return RT_OK;
    FrameInfo F;
    F.width = p->width; F.height = p->height; F.tiles_x = ctx->tiles.tiles_x; F.tiles_y = ctx->tiles.tiles_y;
    F.tile_ids = ctx->tile_ids.p;
#if RT_TILE_W == 32
    if (QUANT && full && remote) {
        k_resolve_rgb8_rows<<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(F, ctx->fb.p, nslots, (unsigned char*)out);
        ctx->stats.kernel_launches++;
        LAUNCHED("k_resolve_rgb8_rows", st);
        return RT_OK;
    }
#endif
    k_resolve<QUANT><<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(F, ctx->fb.p, nslots, full ? 1 : 0, out);
    ctx->stats.kernel_launches++;
    LAUNCHED("k_resolve", st);
    return RT_OK;
}

inline bool full_frame(const rt_params* p) { return p->tile_world == 1 || (p->flags & RT_FLAG_FULL_FRAME) != 0; }

// ---- several GPUs inside one process (rt_params.n_gpus > 1) ---------------------------------------------
// The context the caller holds drives one sub-context per additional device.  The scene is uploaded (and its
// LBVH built) once on the primary device and replicated with peer copies; a frame's tiles are interleaved over
// the devices like over the ranks of a multi-process job, one host thread per device runs the wavefront loop,
// and every device's resolve kernel stores its tiles straight into the caller's frame.

int ensure_peers(rt_context* ctx, int n) {
    if ((int)ctx->peers.size() >= n - 1) return RT_OK;
    int count = 0;
    CU(cudaGetDeviceCount(&count));
    // RT_MULTI_SAME_DEVICE=1: all sub-contexts on the primary's device (exercises the whole multi-GPU path on a
    // one-GPU box; no speed-up, of course)
    const bool same = getenv("RT_MULTI_SAME_DEVICE") != nullptr;
    if (!same && n > count)
        return fail(RT_ERR_NO_DEVICE, "n_gpus = %d but only %d CUDA device(s) are visible", n, count);
    while ((int)ctx->peers.size() < n - 1) {
        const int k = (int)ctx->peers.size() + 1;
        const int dev = same ? ctx->device : (ctx->device + k) % count;
        if (dev != ctx->device) {
            int can = 0;
            CU(cudaDeviceCanAccessPeer(&can, dev, ctx->device));
            if (!can) return fail(RT_ERR_NO_DEVICE, "device %d cannot access device %d's memory (no NVLink/P2P path)", dev, ctx->device);
            CU(cudaSetDevice(dev));
            cudaError_t e = cudaDeviceEnablePeerAccess(ctx->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
            if (e != cudaSuccess) return fail(RT_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", dev, ctx->device, cudaGetErrorString(e));
        }
        rt_context* pc = new rt_context();
        int rc = init_context(pc, dev, ctx->num_sms);
        if (rc == RT_OK) rc = ensure_levels(pc, 16);
        if (rc != RT_OK) { rt_destroy(pc); cudaSetDevice(ctx->device); return rc; }
        ctx->peers.push_back(pc);
        ctx->peers_stale = true;
    }
    CU(cudaSetDevice(ctx->device));
    return RT_OK;
}

// Copies the primary's scene into every sub-context: the scalar state, then, for a sub-context on another device,
// every scene array with a peer copy (the LBVH is built once, not once per GPU).  A sub-context on the primary's own
// device reads the primary's arrays.
int replicate_scene(rt_context* ctx, int n) {
    if (!ctx->peers_stale) return RT_OK;
    CU(cudaSetDevice(ctx->device));
    const SceneStore& src = ctx->scene;
    for (int k = 0; k < n - 1; k++) {
        rt_context* pc = ctx->peers[(size_t)k];
        SceneStore& dst = pc->scene;
        dst.S = src.S;
        dst.sort_grid = src.sort_grid;
        dst.sort_ok = src.sort_ok;
        const bool same_device = pc->device == ctx->device;
        if (!same_device) {
            int rc = SceneStore::each_array([&](auto array, auto) -> int {
                auto& to = dst.*array;
                const auto& from = src.*array;
                CU(cudaSetDevice(pc->device));
                CU(to.hold(from.used));
                CU(cudaSetDevice(ctx->device));
                if (from.used) CU(cudaMemcpyPeerAsync(to.p, pc->device, from.p, ctx->device, sizeof(*from.p) * from.used, ctx->stream));
                return RT_OK;
            });
            if (rc != RT_OK) return rc;
        }
        dst.bind(same_device ? src : dst);
        pc->have_scene = true;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->peers_stale = false;
    return RT_OK;
}

// out: the whole row-major frame, addressable from every device (the primary's device memory with peer access
// enabled, or mapped pinned host memory).  Blocks until every device has stored its tiles.
template <bool QUANT>
int render_multi(rt_context* ctx, const rt_params* p, void* out, bool out_is_primary_local, rt_progress_fn cb, void* user) {
    const int n = p->n_gpus;
    int rc = ensure_peers(ctx, n);
    if (rc != RT_OK) return rc;
    rc = replicate_scene(ctx, n);
    if (rc != RT_OK) return rc;
    const bool io = p->intersection_only != 0;
    if (io && p->tile_world > 1)
        return fail(RT_ERR_INVALID, "intersection_only with n_gpus > 1 needs tile_world == 1 (the maximum is reduced inside one process only)");
    std::vector<rt_context*> all;
    all.push_back(ctx);
    for (int k = 0; k < n - 1; k++) all.push_back(ctx->peers[(size_t)k]);
    std::vector<rt_params> sp((size_t)n, *p);
    // device k takes the tiles (tx + ty) % (tile_world * n) == tile_rank + k * tile_world: a refinement of this rank's share
    for (int k = 0; k < n; k++) {
        sp[(size_t)k].n_gpus = 1;
        sp[(size_t)k].tile_rank = p->tile_rank + k * p->tile_world;
        sp[(size_t)k].tile_world = p->tile_world * n;
    }
    // a section of work on every device: device 0 on the calling thread (progress callbacks), the others on workers
    auto on_all = [&](auto&& body) -> int {
        std::vector<std::thread> th;
        for (int k = 1; k < n; k++)
            th.emplace_back([&, k]() {
                rt_context* c = all[(size_t)k];
                c->worker_rc = body(k);
                if (c->worker_rc != RT_OK) c->worker_err = g_error;
            });
        int rc0 = body(0);
        std::string err0 = rc0 != RT_OK ? g_error : std::string();
        for (auto& t : th) t.join();
        cudaSetDevice(ctx->device);
        if (rc0 != RT_OK) return fail(rc0, "%s", err0.c_str());
        for (int k = 1; k < n; k++)
            if (all[(size_t)k]->worker_rc != RT_OK)
                return fail(all[(size_t)k]->worker_rc, "GPU %d: %s", all[(size_t)k]->device, all[(size_t)k]->worker_err.c_str());
        return RT_OK;
    };
    auto resolve = [&](int k) -> int {
        rt_context* c = all[(size_t)k];
        const bool remote = !(k == 0 && out_is_primary_local);
        int r = resolve_to<QUANT>(c, &sp[(size_t)k], out, c->stream, true, remote);
        if (r != RT_OK) return r;
        CU(cudaStreamSynchronize(c->stream));
        return RT_OK;
    };
    if (!io) {
        rc = on_all([&](int k) -> int {
            rt_context* c = all[(size_t)k];
            int r = render_core(c, &sp[(size_t)k], c->stream, false, k == 0 ? cb : nullptr, k == 0 ? user : nullptr, /*final_cb=*/false);
            if (r != RT_OK) return r;
            return resolve(k);
        });
        if (rc != RT_OK) return rc;
    } else {
        // --intersection-only divides by the GLOBAL maximum (src/scene.cpp:50-58): render, reduce the per-device
        // maxima on the host (n doubles), then divide + resolve on every device
        rc = on_all([&](int k) -> int {
            rt_context* c = all[(size_t)k];
            return render_core(c, &sp[(size_t)k], c->stream, false, k == 0 ? cb : nullptr, k == 0 ? user : nullptr, false);
        });
        if (rc != RT_OK) return rc;
        unsigned long long gmax = 0;
        for (int k = 0; k < n; k++) {
            unsigned long long bits = 0;
            CU(cudaSetDevice(all[(size_t)k]->device));
            CU(cudaMemcpy(&bits, all[(size_t)k]->ctr.p, sizeof(bits), cudaMemcpyDeviceToHost));
            gmax = std::max(gmax, bits);          // non-negative doubles order like their bit patterns
        }
        rc = on_all([&](int k) -> int {
            rt_context* c = all[(size_t)k];
            CU(cudaSetDevice(c->device));
            const size_t nv = c->tiles.ids.size() * RT_TILE_PIXELS * 3;
            CU(cudaMemcpyAsync(c->ctr.p, &gmax, sizeof(gmax), cudaMemcpyHostToDevice, c->stream));
            if (nv) {
                k_divide<<<(unsigned)((nv + 255) / 256), 256, 0, c->stream>>>(c->fb.p, nv, c->ctr.p);
                LAUNCHED("k_divide", c->stream);
            }
            return resolve(k);
        });
        if (rc != RT_OK) return rc;
    }
    // statistics of the whole frame: counts add up, times are the slowest device's
    rt_stats& st = ctx->stats;
    for (int k = 1; k < n; k++) {
        const rt_stats& o = all[(size_t)k]->stats;
        st.rays_primary += o.rays_primary; st.rays_shadow += o.rays_shadow; st.rays_secondary += o.rays_secondary;
        st.degenerate_rays += o.degenerate_rays; st.kernel_launches += o.kernel_launches; st.hits += o.hits;
        st.shadow_rays_culled += o.shadow_rays_culled;
        for (int j = 0; j < 2; j++) {
            st.nodes_fetched[j] += o.nodes_fetched[j]; st.tris_tested[j] += o.tris_tested[j]; st.spheres_tested[j] += o.spheres_tested[j];
        }
        for (int j = 0; j < 4; j++) { st.ms_kernel[j] = std::max(st.ms_kernel[j], o.ms_kernel[j]); st.launches_kernel[j] += o.launches_kernel[j]; }
        st.ms_trace = std::max(st.ms_trace, o.ms_trace);
    }
    if (cb) cb(p->width * p->height, p->width * p->height, user);
    return RT_OK;
}

// A host pointer the devices can store through (cudaHostAlloc / cudaHostRegister memory)?  Returns its device alias.
void* mapped_host_alias(void* host) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost) return nullptr;
    return at.devicePointer;
}

template <bool QUANT>
int render_device_impl(rt_context* ctx, const rt_params* p, void* d_out, void* stream) {
    if (!d_out) return fail(RT_ERR_INVALID, "d_out is NULL");
    int rc = check_params(ctx, p);
    if (rc != RT_OK) return rc;
    if (QUANT && p->intersection_only && p->tile_world > 1)
        return fail(RT_ERR_INVALID, "intersection_only over several ranks needs the FP64 frame: the global maximum is applied after the render "
                                    "(rt_intersection_max / rt_divide_device)");
    if (p->n_gpus > 1) return render_multi<QUANT>(ctx, p, d_out, true, nullptr, nullptr);
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    rc = render_core(ctx, p, st, false, nullptr, nullptr);
    if (rc != RT_OK) return rc;
    // a frame shared with other ranks is remote memory for all of them but (at most) one
    rc = resolve_to<QUANT>(ctx, p, d_out, st, full_frame(p), p->tile_world > 1 && full_frame(p));
    if (rc != RT_OK) return rc;
    CU(cudaStreamSynchronize(st));
    return RT_OK;
}

}  // namespace

extern "C" {

int rt_render_device(rt_context* ctx, const rt_params* p, double* d_out, void* stream) {
    return render_device_impl<false>(ctx, p, d_out, stream);
}
int rt_render_device_rgb8(rt_context* ctx, const rt_params* p, uint8_t* d_out, void* stream) {
    return render_device_impl<true>(ctx, p, d_out, stream);
}

static int render_host(rt_context* ctx, const rt_params* p, void* host_out, bool quant, rt_progress_fn cb, void* user) {
    if (!host_out) return fail(RT_ERR_INVALID, "output buffer is NULL");
    int rc = check_params(ctx, p);
    if (rc != RT_OK) return rc;
    const size_t px = (size_t)p->width * p->height;
    const size_t bytes = px * 3 * (quant ? 1 : sizeof(double));
    void* alias = (p->tile_world > 1 || p->n_gpus > 1) ? mapped_host_alias(host_out) : nullptr;
    if (p->tile_world > 1) {
        // several processes fill one host frame: each stores its own tiles through its own PCIe link
        if (!(p->flags & RT_FLAG_FULL_FRAME))
            return fail(RT_ERR_INVALID, "host-buffer renders with tile_world > 1 need RT_FLAG_FULL_FRAME (or use rt_render_device*)");
        if (!alias) return fail(RT_ERR_INVALID, "a host frame shared by several ranks must be page-locked (cudaHostRegister / cudaHostAlloc)");
        if (p->intersection_only) return fail(RT_ERR_INVALID, "intersection_only over several ranks: use rt_render_device + rt_intersection_max");
        rc = render_core(ctx, p, ctx->stream, false, cb, user);
        if (rc != RT_OK) return rc;
        rc = quant ? resolve_to<true>(ctx, p, alias, ctx->stream, true, true) : resolve_to<false>(ctx, p, alias, ctx->stream, true, true);
        if (rc != RT_OK) return rc;
        CU(cudaStreamSynchronize(ctx->stream));
        return RT_OK;
    }
    if (p->n_gpus > 1 && alias)      // page-locked caller frame: every device stores its tiles over its own PCIe link
        return quant ? render_multi<true>(ctx, p, alias, false, cb, user) : render_multi<false>(ctx, p, alias, false, cb, user);
    CU(cudaSetDevice(ctx->device));
    CU(ctx->staging.ensure(bytes));
    if (p->n_gpus > 1) {             // pageable caller frame: peers store into the primary's staging frame, one copy back
        rc = quant ? render_multi<true>(ctx, p, ctx->staging.p, true, cb, user) : render_multi<false>(ctx, p, ctx->staging.p, true, cb, user);
        if (rc != RT_OK) return rc;
    } else {
        rc = render_core(ctx, p, ctx->stream, false, cb, user);
        if (rc != RT_OK) return rc;
        rc = quant ? resolve_to<true>(ctx, p, ctx->staging.p, ctx->stream, true, false)
                   : resolve_to<false>(ctx, p, ctx->staging.p, ctx->stream, true, false);
        if (rc != RT_OK) return rc;
    }
    CU(cudaEventRecord(ctx->ev0, ctx->stream));
    cudaError_t e = cudaMemcpyAsync(host_out, ctx->staging.p, bytes, cudaMemcpyDeviceToHost, ctx->stream);
    CU(cudaEventRecord(ctx->ev1, ctx->stream));
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "framebuffer readback: %s", cudaGetErrorString(e));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->stats.ms_readback = ms;
    return RT_OK;
}

int rt_render(rt_context* ctx, const rt_params* p, double* rgb, rt_progress_fn cb, void* user) {
    return render_host(ctx, p, rgb, false, cb, user);
}
int rt_render_rgb8(rt_context* ctx, const rt_params* p, uint8_t* rgb8, rt_progress_fn cb, void* user) {
    return render_host(ctx, p, rgb8, true, cb, user);
}

int rt_shared_frame_create(rt_context* ctx, uint64_t bytes, void** d_ptr, unsigned char* handle) {
    if (!ctx || !d_ptr || !handle || !bytes) return fail(RT_ERR_INVALID, "rt_shared_frame_create: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == RT_SHARED_HANDLE_BYTES, "handle size");
    CU(cudaSetDevice(ctx->device));
    void* p = nullptr;
    CU(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(RT_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(handle, &h, sizeof(h));
    ctx->ipc_created.push_back(p);
    *d_ptr = p;
    return RT_OK;
}

int rt_shared_frame_open(rt_context* ctx, const unsigned char* handle, void** d_ptr) {
    if (!ctx || !d_ptr || !handle) return fail(RT_ERR_INVALID, "rt_shared_frame_open: bad argument");
    CU(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->ipc_opened.push_back(p);
    *d_ptr = p;
    return RT_OK;
}

int rt_shared_frame_close(rt_context* ctx, void* d_ptr) {
    if (!ctx || !d_ptr) return fail(RT_ERR_INVALID, "rt_shared_frame_close: bad argument");
    CU(cudaSetDevice(ctx->device));
    for (size_t k = 0; k < ctx->ipc_opened.size(); k++)
        if (ctx->ipc_opened[k] == d_ptr) {
            ctx->ipc_opened.erase(ctx->ipc_opened.begin() + (long)k);
            CU(cudaIpcCloseMemHandle(d_ptr));
            return RT_OK;
        }
    for (size_t k = 0; k < ctx->ipc_created.size(); k++)
        if (ctx->ipc_created[k] == d_ptr) {
            ctx->ipc_created.erase(ctx->ipc_created.begin() + (long)k);
            CU(cudaFree(d_ptr));
            return RT_OK;
        }
    return fail(RT_ERR_INVALID, "rt_shared_frame_close: not a shared frame of this context");
}

int64_t rt_tile_count(const rt_params* p) {
    if (!p || p->tile_world < 1) return 0;
    return TileLayout::count(p->width, p->height, p->tile_rank, p->tile_world);
}
int64_t rt_tile_count_total(const rt_params* p) {
    if (!p) return 0;
    return (int64_t)((p->width + RT_TILE_W - 1) / RT_TILE_W) * ((p->height + RT_TILE_H - 1) / RT_TILE_H);
}
int64_t rt_tile_count_max(const rt_params* p) {
    if (!p || p->tile_world < 1) return 0;
    long long m = 0;
    for (int r = 0; r < p->tile_world; r++) m = std::max(m, TileLayout::count(p->width, p->height, r, p->tile_world));
    return m;
}

}  // extern "C"

template <typename T>
static int unpack_impl(rt_context* ctx, const rt_params* p, const T* d_packed, T* d_frame, void* stream) {
    if (!ctx || !p || !d_packed || !d_frame) return fail(RT_ERR_INVALID, "rt_unpack_tiles: NULL argument");
    if (p->width <= 0 || p->height <= 0 || p->tile_world < 1) return fail(RT_ERR_INVALID, "rt_unpack_tiles: bad params");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    const int tiles_x = (p->width + RT_TILE_W - 1) / RT_TILE_W, tiles_y = (p->height + RT_TILE_H - 1) / RT_TILE_H;
    const int world = p->tile_world;
    std::vector<int> starts((size_t)world * (tiles_y + 1), 0);
    for (int r = 0; r < world; r++) {
        int acc = 0;
        for (int ty = 0; ty < tiles_y; ty++) {
            starts[(size_t)r * (tiles_y + 1) + ty] = acc;
            int first = ((r - ty) % world + world) % world;
            if (first < tiles_x) acc += (tiles_x - first + world - 1) / world;
        }
        starts[(size_t)r * (tiles_y + 1) + tiles_y] = acc;
    }
    DevBuf<int>& d_starts = ctx->unpack_starts;
    if (ctx->unpack_key[0] != p->width || ctx->unpack_key[1] != p->height || ctx->unpack_key[2] != world || !d_starts.p) {
        CU(d_starts.ensure(starts.size()));
        CU(cudaMemcpyAsync(d_starts.p, starts.data(), sizeof(int) * starts.size(), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));          // `starts` is a local
        ctx->unpack_key[0] = p->width; ctx->unpack_key[1] = p->height; ctx->unpack_key[2] = world;
    }
    const long long npx = (long long)p->width * p->height;
    k_unpack<T><<<(unsigned)((npx + 255) / 256), 256, 0, st>>>(p->width, p->height, tiles_x, world, rt_tile_count_max(p),
                                                            d_starts.p, tiles_y, d_packed, d_frame);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    return RT_OK;
}
extern "C" {

int rt_unpack_tiles_rgb8(rt_context* ctx, const rt_params* p, const uint8_t* d_packed, uint8_t* d_frame, void* stream) {
    return unpack_impl<uint8_t>(ctx, p, d_packed, d_frame, stream);
}
int rt_unpack_tiles(rt_context* ctx, const rt_params* p, const double* d_packed, double* d_frame, void* stream) {
    return unpack_impl<double>(ctx, p, d_packed, d_frame, stream);
}

int rt_primary_ids(rt_context* ctx, const rt_params* p, int32_t* geom, int32_t* face) {
    if (!geom || !face) return fail(RT_ERR_INVALID, "rt_primary_ids: NULL output");
    int rc = check_params(ctx, p);
    if (rc != RT_OK) return rc;
    if (p->tile_world != 1) return fail(RT_ERR_INVALID, "rt_primary_ids needs tile_world == 1");
    rt_stats keep = ctx->stats;
    rc = render_core(ctx, p, ctx->stream, true, nullptr, nullptr);
    ctx->stats = keep;
    if (rc != RT_OK) return rc;
    // ids are in slot order: bring them back and de-tile on the host (parity path, not timed)
    const TileLayout& T = ctx->tiles;
    const size_t nslots = T.ids.size() * RT_TILE_PIXELS;
    std::vector<int> hg(nslots), hf(nslots);
    CU(cudaMemcpy(hg.data(), ctx->ids_geom.p, sizeof(int) * nslots, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(hf.data(), ctx->ids_face.p, sizeof(int) * nslots, cudaMemcpyDeviceToHost));
    for (size_t lt = 0; lt < T.ids.size(); lt++) {
        int gt = T.ids[lt], tx = gt % T.tiles_x, ty = gt / T.tiles_x;
        for (int j = 0; j < RT_TILE_PIXELS; j++) {
            int w = j >> 5, l = j & 31;
            int px = tx * RT_TILE_W + (w % (RT_TILE_W / 8)) * 8 + (l & 7), py = ty * RT_TILE_H + (w / (RT_TILE_W / 8)) * 4 + (l >> 3);
            if (px >= p->width || py >= p->height) continue;
            size_t dst = (size_t)py * p->width + px, src = lt * RT_TILE_PIXELS + j;
            geom[dst] = hg[src];
            face[dst] = hf[src];
        }
    }
    return RT_OK;
}

int rt_cast_rays(rt_context* ctx, int64_t n, const double* org, const double* dir, const uint8_t* reverse,
                 uint32_t flags, int32_t* geom, int32_t* face, double* dist, double* point, double* normal) {
    if (!ctx) return fail(RT_ERR_INVALID, "context is NULL");
    if (!ctx->have_scene) return fail(RT_ERR_NO_SCENE, "rt_scene_upload has not been called");
    if (n < 0 || (n && (!org || !dir))) return fail(RT_ERR_INVALID, "rt_cast_rays: bad arguments");
    if (n == 0) return RT_OK;
    CU(cudaSetDevice(ctx->device));
    DevBuf<double> d_org, d_dir, d_dist, d_point, d_normal;
    DevBuf<unsigned char> d_rev;
    DevBuf<int> d_geom, d_face;
    const size_t N = (size_t)n;
    CU(d_org.ensure(3 * N)); CU(d_dir.ensure(3 * N)); CU(d_dist.ensure(N)); CU(d_point.ensure(3 * N)); CU(d_normal.ensure(3 * N));
    CU(d_geom.ensure(N)); CU(d_face.ensure(N));
    // on the query's own stream: a cudaMemcpy from pageable memory may return before its DMA has landed, and the
    // context's streams do not wait for the legacy default stream
    CU(cudaMemcpyAsync(d_org.p, org, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_dir.p, dir, sizeof(double) * 3 * N, cudaMemcpyHostToDevice, ctx->stream));
    if (reverse) {
        CU(d_rev.ensure(N));
        CU(cudaMemcpyAsync(d_rev.p, reverse, N, cudaMemcpyHostToDevice, ctx->stream));
    }
    const unsigned blocks = (unsigned)((N + RT_BLOCK - 1) / RT_BLOCK);
    if (flags & RT_FLAG_BRUTE_FORCE)
        k_query<true><<<blocks, RT_BLOCK, 0, ctx->stream>>>(ctx->scene.S, n, d_org.p, d_dir.p, reverse ? d_rev.p : nullptr, d_geom.p,
                                                           d_face.p, d_dist.p, d_point.p, d_normal.p);
    else
        k_query<false><<<blocks, RT_BLOCK, 0, ctx->stream>>>(ctx->scene.S, n, d_org.p, d_dir.p, reverse ? d_rev.p : nullptr, d_geom.p,
                                                            d_face.p, d_dist.p, d_point.p, d_normal.p);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    if (geom) CU(cudaMemcpy(geom, d_geom.p, sizeof(int) * N, cudaMemcpyDeviceToHost));
    if (face) CU(cudaMemcpy(face, d_face.p, sizeof(int) * N, cudaMemcpyDeviceToHost));
    if (dist) CU(cudaMemcpy(dist, d_dist.p, sizeof(double) * N, cudaMemcpyDeviceToHost));
    if (point) CU(cudaMemcpy(point, d_point.p, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost));
    if (normal) CU(cudaMemcpy(normal, d_normal.p, sizeof(double) * 3 * N, cudaMemcpyDeviceToHost));
    return RT_OK;
}

int rt_intersection_max(rt_context* ctx, double* out_max) {
    if (!ctx || !out_max) return fail(RT_ERR_INVALID, "rt_intersection_max: NULL argument");
    CU(cudaSetDevice(ctx->device));
    unsigned long long bits = 0;
    CU(cudaMemcpy(&bits, ctx->ctr.p, sizeof(bits), cudaMemcpyDeviceToHost));
    memcpy(out_max, &bits, sizeof(double));
    return RT_OK;
}

int rt_divide_device(rt_context* ctx, double* d_values, int64_t count, double divisor, void* stream) {
    if (!ctx || !d_values || count < 0) return fail(RT_ERR_INVALID, "rt_divide_device: bad argument");
    if (count == 0) return RT_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    unsigned long long bits;
    memcpy(&bits, &divisor, sizeof(bits));
    unsigned long long* d_bits = ctx->ctr.p;
    CU(cudaMemcpyAsync(d_bits, &bits, sizeof(bits), cudaMemcpyHostToDevice, st));
    k_divide<<<(unsigned)(((size_t)count + 255) / 256), 256, 0, st>>>(d_values, (size_t)count, d_bits);
    LAUNCHED("k_divide", st);
    CU(cudaStreamSynchronize(st));
    return RT_OK;
}

int rt_scene_device_bytes(rt_context* ctx, uint64_t* node_bytes, uint64_t* face_bytes) {
    if (!ctx) return fail(RT_ERR_INVALID, "context is NULL");
    const SceneStore& sc = ctx->scene;
    if (node_bytes) *node_bytes = sizeof(BvhNode) * sc.node_count;
    if (face_bytes) *face_bytes = sizeof(double2) * (sc.face_pts.used + sc.face_nrm.used);
    return RT_OK;
}

int rt_microbench_gather(rt_context* ctx, uint64_t array_bytes, int loads_per_thread, double* gbs) {
    if (!ctx || !gbs || loads_per_thread < 1) return fail(RT_ERR_INVALID, "rt_microbench_gather: bad argument");
    CU(cudaSetDevice(ctx->device));
    if (array_bytes < 64) array_bytes = 64;
    const unsigned long long nrec = array_bytes / 32;
    DevBuf<float4> data;
    DevBuf<float> sink;
    CU(data.ensure((size_t)nrec * 2));
    CU(sink.ensure(1));
    CU(cudaMemsetAsync(data.p, 0, (size_t)nrec * 32, ctx->stream));
    const int blocks = ctx->num_sms * 16, threads = 256;
    k_gather_probe<<<blocks, threads, 0, ctx->stream>>>(data.p, nrec, loads_per_thread, sink.p);   // warm-up
    LAUNCHED("k_gather_probe", ctx->stream);
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(ctx->ev0, ctx->stream));
        k_gather_probe<<<blocks, threads, 0, ctx->stream>>>(data.p, nrec, loads_per_thread, sink.p);
        CU(cudaEventRecord(ctx->ev1, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (ms < best) best = ms;
    }
    *gbs = (double)blocks * threads * loads_per_thread * 32.0 / (best * 1e-3) / 1e9;
    return RT_OK;
}

int rt_microbench_node_walk(rt_context* ctx, int group, int visits_per_thread, double* visits_per_s, double* bytes_per_s) {
    if (!ctx || !visits_per_s || visits_per_thread < 1 || group < 1 || group > 32 || (group & (group - 1)))
        return fail(RT_ERR_INVALID, "rt_microbench_node_walk: bad argument (group must be a power of two <= 32)");
    if (!ctx->have_scene || !ctx->scene.S.nodes) return fail(RT_ERR_NO_SCENE, "rt_microbench_node_walk needs an uploaded scene with an LBVH");
    CU(cudaSetDevice(ctx->device));
    DevBuf<float> sink;
    CU(sink.ensure(1));
    // the traversal kernels' shape: 64-thread blocks, 16 resident per SM; 8 waves of them
    const int blocks = ctx->num_sms * RT_SHADOW_MINBLOCKS * 8;
    k_node_walk<<<blocks, RT_BLOCK, 0, ctx->stream>>>(ctx->scene.S.nodes, visits_per_thread, group, sink.p);   // warm-up
    LAUNCHED("k_node_walk", ctx->stream);
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(ctx->ev0, ctx->stream));
        k_node_walk<<<blocks, RT_BLOCK, 0, ctx->stream>>>(ctx->scene.S.nodes, visits_per_thread, group, sink.p);
        CU(cudaEventRecord(ctx->ev1, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (ms < best) best = ms;
    }
    const double visits = (double)blocks * RT_BLOCK * (double)visits_per_thread;
    *visits_per_s = visits / (best * 1e-3);
    if (bytes_per_s) *bytes_per_s = *visits_per_s * 112.0;
    return RT_OK;
}

int rt_get_stats(rt_context* ctx, rt_stats* out) {
    if (!ctx || !out) return fail(RT_ERR_INVALID, "rt_get_stats: NULL argument");
    *out = ctx->stats;
    return RT_OK;
}

}  // extern "C"
