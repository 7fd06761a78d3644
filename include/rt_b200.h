/* rt_b200.h — C ABI of the B200-native trace loop.
 *
 * This is the drop-in boundary for the reference's per-pixel trace loop.  The
 * reference has no FFI; its seam is ONE C++ member call,
 *     scene.renderScene(image, updateProgress)        (src/main.cpp:72)
 * declared at src/scene.h:14.  Everything below replaces what happens behind
 * that call: Scene::renderScene (src/scene.cpp:10-59), Scene::traceRay
 * (src/scene.cpp:61-140), Scene::castRay (src/scene.cpp:142-167) and the
 * intersection routines of src/geometry.cpp:5-126.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross the boundary;
 *   - the caller owns every host buffer; the library owns device memory;
 *   - nothing throws: every entry point returns RT_OK (0) or a negative code,
 *     and rt_last_error() gives the message the host wrapper turns into the
 *     reference's "Error: ..." convention (src/main.cpp:56-61);
 *   - there is NO CPU fallback: if no sm_100-class device is usable the calls
 *     fail with RT_ERR_NO_DEVICE.
 *
 * The scene descriptor is the reference object graph (src/scene.h:35-38)
 * flattened: one rt_geometry per entry of Scene::geometries_ in insertion
 * order (this order IS the tie-break order of src/scene.cpp:154), faces in
 * Mesh::faces_ order (tie-break order of src/geometry.cpp:109).
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 2

/* ---- error codes ------------------------------------------------------- */
#define RT_OK                0
#define RT_ERR_INVALID      -1   /* bad argument / malformed descriptor        */
#define RT_ERR_NO_DEVICE    -2   /* no usable CUDA device (no CPU fallback)    */
#define RT_ERR_CUDA         -3   /* a CUDA call failed; see rt_last_error()    */
#define RT_ERR_NO_SCENE     -4   /* render requested before rt_scene_upload()  */
#define RT_ERR_OOM          -5   /* device allocation failed                   */
#define RT_ERR_LIMIT        -6   /* scene exceeds a hard limit of the device layout (see rt_last_error()) */

/* ---- geometry / light kinds ------------------------------------------- */
#define RT_GEOM_SPHERE 0   /* `sph`  : Sphere            (src/geometry.h:17-23)          */
#define RT_GEOM_TRI    1   /* `tri`  : Mesh of 2 faces displaced +-eps (src/geometry.cpp:128-143) */
#define RT_GEOM_MESH   2   /* `obj`  : Mesh of one-sided faces + object-space AABB        */

#define RT_LIGHT_AMBIENT     0   /* AmbientLight      (src/lights.h:67-75) */
#define RT_LIGHT_POINT       1   /* PointLight        (src/lights.h:15-43) */
#define RT_LIGHT_DIRECTIONAL 2   /* DirectionalLight  (src/lights.h:45-65) */

/* Material (src/rtbase.h:30-39).  kt is only a "has refraction" flag in the
 * reference (src/scene.cpp:115); it is carried verbatim. */
typedef struct rt_material {
    double ka[3];
    double kd[3];
    double ks[3];
    double kr[3];
    double kt[3];
    double sp;
    double ior;
    double reserved_;
} rt_material;

/* One entry of Scene::geometries_.  fwd/inv are rows 0..2 of the 4x4 affine
 * matrices Transformable::forwardTransform_/inverseTransform_ (row-major 3x4;
 * row 3 is 0 0 0 1), det is transformDeterminant_ (src/rtbase.h:57-63). */
typedef struct rt_geometry {
    int32_t type;          /* RT_GEOM_*                                          */
    int32_t material;      /* index into rt_scene.materials                      */
    int64_t first_face;    /* TRI/MESH: first face in face_points/face_normals   */
    int64_t num_faces;     /* TRI: 2, MESH: n, SPHERE: 0                         */
    double  fwd[12];
    double  inv[12];
    double  det;
    double  center[3];     /* SPHERE: Sphere::center_                            */
    double  radius;        /* SPHERE: (double)radius_  (radius_ is a float)      */
    double  radius2;       /* SPHERE: (double)(radius_*radius_), float product   */
    double  bbmin[3];      /* MESH: Mesh::boundingBoxMin_ (object space)         */
    double  bbmax[3];
    int32_t use_bbox;      /* MESH: bbmin!=bbmax && faces>1 (src/geometry.cpp:72) */
    int32_t reserved_;
} rt_geometry;

/* Light, already forward-transformed at flatten time (this removes the racy
 * lazy caches of src/lights.h:28-33,56-61).  v = transformed point (POINT) or
 * transformed, NOT re-normalised direction (DIRECTIONAL). */
typedef struct rt_light {
    int32_t type;
    int32_t reserved_;
    double  v[3];
    double  color[3];
    double  falloff;
} rt_light;

/* Camera points after the camera's forward transform (src/rtbase.h:86-95). */
typedef struct rt_camera {
    double eye[3];
    double ll[3];
    double lr[3];
    double ul[3];
    double ur[3];
} rt_camera;

typedef struct rt_scene {
    rt_camera          camera;
    int32_t            num_geometries;
    int32_t            num_materials;
    int32_t            num_lights;
    uint32_t           flags;          /* RT_SCENE_*                             */
    int64_t            num_faces;
    const rt_geometry* geometries;     /* [num_geometries]                       */
    const rt_material* materials;      /* [num_materials]                        */
    const rt_light*    lights;         /* [num_lights], insertion order          */
    const double*      face_points;    /* [num_faces][3 vertices][3], object space */
    const double*      face_normals;   /* [num_faces][3 vertices][3], object space */
} rt_scene;
/* face_points / face_normals are DEVICE pointers (memory of the context's device): the upload
 * packs them in place instead of copying them from the host first.  This is how a caller that
 * already holds the arrays on the device (e.g. after an NVLink all-gather of per-rank slices
 * of a scene, one slice per PCIe link) hands them over. */
#define RT_SCENE_FACES_ON_DEVICE 1u

/* ---- render parameters -------------------------------------------------- */
#define RT_FLAG_BRUTE_FORCE   1u  /* no LBVH: every ray tests every primitive (parity aid) */
#define RT_FLAG_COUNT_WORK    2u  /* instrumented build of the same kernels: count nodes /
                                     primitives fetched for the roofline (slower)          */
#define RT_FLAG_TIME_KERNELS  4u  /* bracket every launch with CUDA events (rt_stats.ms_kernel) */
#define RT_FLAG_FULL_FRAME   16u  /* tile_world > 1: the output buffer is the WHOLE row-major frame (shared
                                     by the cooperating ranks: a peer-mapped device buffer, see
                                     rt_shared_frame_*, or pinned host memory every rank has registered);
                                     this rank stores only the pixels of its own tiles into it            */
#define RT_FLAG_SERIAL        8u  /* run a frame's kernels strictly one after another: by default the
                                     shadow kernel of bounce level l runs beside the closest-hit and
                                     shading kernels of level l+1 (their event-bracketed durations
                                     then overlap and do not add up to the frame time)          */

typedef struct rt_params {
    int32_t  width;              /* programOptions.renderWidth_   (src/options.h:13) */
    int32_t  height;             /* programOptions.renderHeight_  (src/options.h:14) */
    int32_t  bounce_depth;       /* programOptions.bounceDepth_   (src/options.h:15) */
    int32_t  intersection_only;  /* programOptions.intersectionOnly_ (src/options.h:16) */
    int32_t  tile_rank;          /* this context renders the 32x32 tiles with (tx + ty) % tile_world == tile_rank */
    int32_t  tile_world;         /* number of cooperating processes (>=1), one GPU each */
    uint32_t flags;              /* RT_FLAG_*                                        */
    int32_t  samples;            /* supersampling (the reference's stated next feature, TODO:2): 0 or 1 =
                                    one ray through the pixel centre (src/scene.cpp:28-29); n > 1 = n x n
                                    rays through the centres of an n x n grid inside the pixel, averaged.
                                    n <= RT_MAX_SAMPLES; not with intersection_only / rt_primary_ids      */
    int32_t  n_gpus;             /* GPUs of THIS process used for the render (SURVEY 8b): 0 or 1 = the
                                    context's device; N > 1 = the context's device plus the next N-1
                                    visible devices, tiles interleaved over them, every device resolving
                                    its tiles straight into the caller's frame (peer stores over NVLink
                                    for a device frame, its own PCIe link for a pinned host frame).
                                    Needs tile_world == 1.                                              */
    int32_t  reserved_[3];
} rt_params;
#define RT_MAX_SAMPLES 16

/* Progress callback == Scene::ProgressHandler (src/scene.h:12).  Invoked on the
 * calling thread only, monotone, and once at the end with (total,total)
 * (src/scene.cpp:41-47; main's printer relies on that final call). */
typedef void (*rt_progress_fn)(int complete, int total, void* user);

/* Ray/work statistics of the last render (a "ray" == one reference castRay call). */
typedef struct rt_stats {
    uint64_t rays_primary;     /* src/scene.cpp:65 from :31                   */
    uint64_t rays_shadow;      /* src/scene.cpp:91                            */
    uint64_t rays_secondary;   /* src/scene.cpp:127,134                       */
    uint64_t degenerate_rays;  /* rays the reference would have aborted on (src/rtbase.h:14-22) */
    uint64_t kernel_launches;  /* kernels launched by the last render          */
    /* RT_FLAG_COUNT_WORK: work done by the closest-hit kernel [0] and the shadow kernel [1] */
    uint64_t nodes_fetched[2];   /* 32-byte BVH child boxes tested              */
    uint64_t tris_tested[2];     /* exact FP64 face tests (80-byte records)     */
    uint64_t spheres_tested[2];  /* exact sphere tests                          */
    uint64_t hits;               /* shaded hits (each casts one shadow ray per non-ambient light) */
    /* RT_FLAG_TIME_KERNELS: summed CUDA-event durations and launch counts per kernel class
     * [0] k_trace  [1] k_shade  [2] k_shadow  [3] raygen/resolve/other */
    double   ms_kernel[4];
    uint64_t launches_kernel[4];
    double   ms_upload;        /* H2D scene + flatten (last rt_scene_upload)   */
    double   ms_build;         /* LBVH build (last rt_scene_upload)            */
    double   ms_trace;         /* device time of the last render (CUDA events) */
    double   ms_readback;      /* D2H of the result (host-buffer entry points) */
    uint64_t scene_bytes_h2d;  /* bytes copied host->device by the last rt_scene_upload */
    uint64_t shadow_rays_culled; /* RT_FLAG_COUNT_WORK: shadow rays (counted in rays_shadow) whose light term is exactly
                                    zero whether or not the light is occluded (src/scene.cpp:95-106: N.L <= 0 and no
                                    specular lobe), answered without traversing the LBVH                            */
} rt_stats;

typedef struct rt_context rt_context;

/* ---- lifetime ----------------------------------------------------------- */
/* device < 0 selects the current CUDA device. */
int  rt_create(int device, rt_context** out);
void rt_destroy(rt_context* ctx);
const char* rt_last_error(void);
int  rt_abi_version(void);

/* Flatten-to-device + LBVH build.  Replaces Mesh::updateBoundingBox
 * (src/geometry.cpp:145-162) and the per-object AABB of hitsBoundingBox
 * (src/geometry.cpp:5-29) as the acceleration structure. */
int  rt_scene_upload(rt_context* ctx, const rt_scene* scene);

/* Update the uploaded scene in place and refit its LBVH instead of rebuilding it: for
 * animation (a moving camera or light, rigid motion, deforming vertices) at a fraction of the
 * cost of rt_scene_upload.
 *   - The descriptor must have the STRUCTURE of the scene last uploaded to ctx: the same
 *     num_geometries and num_faces, and per geometry the same type, first_face and num_faces.
 *     Everything else may change: fwd, inv, det, center, radius, radius2, bbmin, bbmax,
 *     use_bbox and material (range-checked); the materials and the lights, their counts
 *     included; the camera; the face points and normals.
 *   - face_points == NULL && face_normals == NULL: the faces on the device stay as they are.
 *     Mesh faces are in object space, so a rigid motion changes only the transform and no face
 *     bytes are copied.  Exactly one of the two NULL is RT_ERR_INVALID.  Otherwise the faces are
 *     read as by rt_scene_upload, RT_SCENE_FACES_ON_DEVICE included.
 *   - Errors: RT_ERR_NO_SCENE when nothing has been uploaded; RT_ERR_INVALID on a structure
 *     mismatch (rt_last_error() names the first mismatching field and geometry index) or a
 *     malformed descriptor.  Every check runs before anything is written, so after a refused
 *     refit the previous scene renders exactly as before.  A CUDA failure part-way through
 *     leaves no scene, like a failed rt_scene_upload.
 *   - Like rt_scene_upload, it must not run while a render on another stream is in flight.
 *   - The tree keeps the topology built for the uploaded scene; so does the split into the
 *     primitives every ray tests and those in the LBVH.  Results never depend on the topology,
 *     but the nodes a ray visits grow as the geometry moves away from what the tree was built
 *     for; calling rt_scene_upload again rebuilds the tree.  A refit of the unchanged scene
 *     rewrites the node array byte for byte.
 *   - rt_stats after a refit: ms_upload = conversion and copies, ms_build = the refit kernels,
 *     kernel_launches and scene_bytes_h2d = those of the refit. */
int  rt_scene_refit(rt_context* ctx, const rt_scene* scene);

/* ---- the hot path: Scene::renderScene ----------------------------------- */
/* rgb: caller-owned double[height][width][3], row 0 = top (src/scene.cpp:26-31),
 * i.e. exactly Scene::RasterImage (src/scene.h:11).  Blocking.
 * n_gpus > 1: the frame's tiles are rendered by n_gpus devices; when the buffer is page-locked
 * (cudaHostAlloc / cudaHostRegister) every device stores its tiles straight into it over its own PCIe link.
 * tile_world > 1 (several processes filling ONE host frame, e.g. in shared memory): needs RT_FLAG_FULL_FRAME
 * and a buffer every process has page-locked; this rank stores only its own tiles. */
int  rt_render(rt_context* ctx, const rt_params* p, double* rgb,
               rt_progress_fn cb, void* user);

/* Same render + the PNG writer's quantisation on device:
 * uint8 = (uint8_t)(clamp(v,0,1)*255.0), truncating (src/writers.cpp:7).
 * rgb8: caller-owned uint8[height][width][3]. */
int  rt_render_rgb8(rt_context* ctx, const rt_params* p, uint8_t* rgb8,
                    rt_progress_fn cb, void* user);

/* Device-resident variants (no host copies).  d_out is DEVICE memory.
 * When tile_world == 1 (or RT_FLAG_FULL_FRAME) the layout is the full row-major
 * frame; otherwise it is this rank's packed tiles (rt_tile_count()*RT_TILE_PIXELS
 * pixels), to be gathered by the caller (NCCL) and unpacked with rt_unpack_tiles*.
 * stream: a cudaStream_t passed as void* (0 = the context's own stream). */
#ifndef RT_TILE_W
#define RT_TILE_W      32
#endif
#ifndef RT_TILE_H
#define RT_TILE_H      RT_TILE_W
#endif
#define RT_TILE_PIXELS (RT_TILE_W * RT_TILE_H)
int     rt_render_device(rt_context* ctx, const rt_params* p, double* d_out, void* stream);
int     rt_render_device_rgb8(rt_context* ctx, const rt_params* p, uint8_t* d_out, void* stream);
int64_t rt_tile_count(const rt_params* p);            /* tiles owned by p->tile_rank  */
int64_t rt_tile_count_total(const rt_params* p);      /* tiles in the whole frame     */
/* d_packed: tile_world consecutive rank buffers, each padded to
 * rt_tile_count_max(p)*RT_TILE_PIXELS pixels (the all_gather layout). */
int64_t rt_tile_count_max(const rt_params* p);
int     rt_unpack_tiles_rgb8(rt_context* ctx, const rt_params* p, const uint8_t* d_packed,
                             uint8_t* d_frame, void* stream);
int     rt_unpack_tiles(rt_context* ctx, const rt_params* p, const double* d_packed,
                        double* d_frame, void* stream);

/* ---- one frame shared by the GPUs of several processes (fused peer-store resolve) ----
 * Rank 0 creates the frame on its device and publishes the 64-byte handle (any byte
 * transport: torch.distributed broadcast, a file, a pipe); the other ranks open it and pass
 * the returned pointer as d_out of rt_render_device[_rgb8] with RT_FLAG_FULL_FRAME: their
 * resolve kernels then store their tiles directly into rank 0's memory over NVLink, so no
 * gather collective and no unpack pass exist.  The callers' barrier after the render is the
 * only synchronisation.  (CUDA IPC; within one process use rt_params.n_gpus instead.) */
#define RT_SHARED_HANDLE_BYTES 64
int     rt_shared_frame_create(rt_context* ctx, uint64_t bytes, void** d_ptr, unsigned char* handle /*[64]*/);
int     rt_shared_frame_open(rt_context* ctx, const unsigned char* handle /*[64]*/, void** d_ptr);
int     rt_shared_frame_close(rt_context* ctx, void* d_ptr);   /* frees (creator) or unmaps (opener) */

/* --intersection-only across ranks (src/scene.cpp:50-58 divides by the GLOBAL maximum): with
 * tile_world > 1 a render leaves 1/dist^2 un-normalised; the caller max-all-reduces
 * rt_intersection_max() over the ranks and applies rt_divide_device() to its buffer. */
int     rt_intersection_max(rt_context* ctx, double* out_max);
int     rt_divide_device(rt_context* ctx, double* d_values, int64_t count, double divisor, void* stream);

/* ---- parity / measurement exports --------------------------------------- */
/* Primary-ray hit ids of the last render's camera rays (SURVEY App. A-12):
 * geom = index in Scene::geometries_, face = index in Mesh::faces_
 * (spheres 0, miss -1/-1).  Host buffers, int32[height*width] each. */
int  rt_primary_ids(rt_context* ctx, const rt_params* p, int32_t* geom, int32_t* face);

/* Closest-hit query for caller-supplied rays (== Scene::castRay,
 * src/scene.cpp:142-167).  Host buffers; org/dir are double[n][3]; dir is
 * normalised internally like the Ray constructor (src/rtbase.h:18-24).
 * reverse: uint8[n] reverseNormals flags.  Outputs may be NULL. */
int  rt_cast_rays(rt_context* ctx, int64_t n, const double* org, const double* dir,
                  const uint8_t* reverse, uint32_t flags,
                  int32_t* geom, int32_t* face, double* dist, double* point, double* normal);

int  rt_get_stats(rt_context* ctx, rt_stats* out);

/* Measured BVH-node-bandwidth roofline (BASELINE.json north_star): independent random
 * 32-byte __ldg gathers over an array of `array_bytes` (use the scene's node-array size),
 * `loads_per_thread` per thread over a full-chip grid.  Returns GB/s in *gbs. */
int  rt_microbench_gather(rt_context* ctx, uint64_t array_bytes, int loads_per_thread, double* gbs);
/* Node-visit ceiling of the uploaded scene's LBVH: a kernel with the traversal kernels' launch shape walks the
 * real 4-wide node array issuing exactly the loads of a traversal step (7 x 16 B per visit, next node = a child
 * just loaded) and nothing else.  group (1, 2, .. 32): consecutive lanes that share one path (32 = a fully
 * coherent warp, 1 = every lane its own path).  Returns per-lane wide-node visits per second and the bytes per
 * second they pull through the LSU (112 B each). */
int  rt_microbench_node_walk(rt_context* ctx, int group, int visits_per_thread, double* visits_per_s, double* bytes_per_s);
/* Size in bytes of the LBVH node array and of the face records of the uploaded scene. */
int  rt_scene_device_bytes(rt_context* ctx, uint64_t* node_bytes, uint64_t* face_bytes);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
