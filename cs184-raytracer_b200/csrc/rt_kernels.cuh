// rt_kernels.cuh — the wavefront kernels that replace the reference's recursion:
//   k_raygen    src/scene.cpp:26-30 + Camera::calculateViewingRay src/rtbase.h:74-84
//   k_trace     Scene::castRay src/scene.cpp:142-167 (closest hit) -> compacted hit queue
//   k_hit_keys  (new) Morton key of every hit point; rt_sort.cuh sorts them (coherent warps downstream)
//   k_shade     Scene::traceRay src/scene.cpp:72-85 (normal, ambient) and :114-136 (bounce spawn);
//               gathers the hit records through the sorted index and writes the sorted queue
//   k_shadow    Scene::traceRay src/scene.cpp:86-107 (one thread per hit x shadow light)
//   k_resolve   src/scene.cpp:31 (pixel store) + optional src/writers.cpp:7 quantisation
// The recursion becomes an iterative bounce loop: a queued ray carries its pixel, the RGB
// weight accumulated along its path (product of kr; refraction weight is 1,
// src/scene.cpp:127,134), the remaining depth and the fromInside flag.  Queues are
// compacted with warp-ballot + prefix-popcount appends.
#pragma once
#include "rt_device.cuh"

namespace rt {

#ifndef RT_BLOCK
#define RT_BLOCK 64
#endif
// 64-thread blocks: the deep bounce levels are small launches (10^5 rays per rank on 8 GPUs),
// and finer blocks shorten their tail (B200, 1/8 of the 8K frame: 22.21 -> 21.94 ms).
// Minimum resident blocks per SM (= 64-register cap, 1024 threads per SM) of the two traversal
// kernels: with fewer warps they stall on node fetches (k_shadow 147 ms at 768 threads/SM vs
// 111 ms at 1024), with more the node (28 registers) no longer fits and the loop spills.
#ifndef RT_SHADOW_MINBLOCKS
#define RT_SHADOW_MINBLOCKS 16
#endif
// Light-major tile of k_shadow (hits).
#ifndef RT_SHADOW_TILE
#define RT_SHADOW_TILE 4096
#endif
#ifndef RT_TRACE_MINBLOCKS
#define RT_TRACE_MINBLOCKS 16
#endif

// Ray queue, SoA over `cap` slots.
struct RayQ {
    double* f;     // 9 fields: ox oy oz dx dy dz wr wg wb
    int* pixel;    // framebuffer slot, -1 = inactive
    int* meta;     // remaining depth | fromInside << RT_META_INSIDE_SHIFT
    size_t cap;
    __device__ __forceinline__ double& fld(int k, size_t i) const { return f[(size_t)k * cap + i]; }
};
#define RT_META_INSIDE_SHIFT 30
#define RT_META_DEPTH_MASK ((1 << RT_META_INSIDE_SHIFT) - 1)
// Hit queue (compacted): P N V W + dist, SoA over `cap` slots.
struct HitQ {
    double* f;     // 13 fields: P(3) N(3) V(3) W(3) dist
    int* pixel;
    int* geom;
    int* meta;
    size_t cap;
    __device__ __forceinline__ double& fld(int k, size_t i) const { return f[(size_t)k * cap + i]; }
};

// Device counters of one bounce level: a block of CTR_COUNT words that starts half-way into a 128-byte
// L2 line.  CTR_HITS, CTR_NEXT, CTR_NEXT_T are reset and read back per chunk as one range, with a line
// boundary between CTR_NEXT and CTR_NEXT_T: every warp of k_shade appends to both, and the appends are
// slower when the two share a line (B200 at 1000 W, 8K synthetic frame: k_shade 7.46 ms on two lines, 8.0 ms on one).
enum {
    CTR_DEGENERATE = 0,
    CTR_S_CULLED = 1,                                      // shadow rays answered without a traversal (COUNT builds)
    CTR_NODES = 2, CTR_TRIS = 3, CTR_SPHERES = 4,          // closest-hit kernel
    CTR_S_DEGENERATE = 5,                                  // the shadow rays among CTR_DEGENERATE: not cast, so not in rays_shadow
    CTR_HITS = 6, CTR_NEXT = 7,                            // the last two words of the first line
    CTR_NEXT_T = 8,                                        // refracted children (stored from the END of the next queue)
    CTR_S_NODES = 9, CTR_S_TRIS = 10, CTR_S_SPHERES = 11,  // shadow kernel
    CTR_COUNT = 16                                         // 128 bytes: every block straddles a line boundary the same way
};

struct FrameInfo {
    int width, height;
    int tiles_x, tiles_y;
    const int* tile_ids;   // [local tile] -> global tile index (ty * tiles_x + tx)
};

__device__ __forceinline__ bool slot_to_pixel(const FrameInfo& F, long long slot, int& px, int& py) {
    int lt = (int)(slot / RT_TILE_PIXELS), j = (int)(slot % RT_TILE_PIXELS);
    int gt = __ldg(F.tile_ids + lt);
    int tx = gt % F.tiles_x, ty = gt / F.tiles_x;
    int w = j >> 5, l = j & 31;                     // one warp = an 8x4 pixel block
    int x = (w % (RT_TILE_W / 8)) * 8 + (l & 7), y = (w / (RT_TILE_W / 8)) * 4 + (l >> 3);
    px = tx * RT_TILE_W + x;
    py = ty * RT_TILE_H + y;
    return px < F.width && py < F.height;
}

// warp-aggregated append: returns the slot for threads with flag set
__device__ __forceinline__ unsigned warp_append(bool flag, unsigned long long* counter) {
    unsigned m = __ballot_sync(0xffffffffu, flag);
    unsigned base = 0;
    if (m) {
        int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
        if (lane == leader) base = (unsigned)atomicAdd(counter, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        base += __popc(m & ((1u << lane) - 1u));
    }
    return base;
}

template <bool COUNT>
__device__ __forceinline__ void flush_work(const WorkCounters& wc, unsigned long long* ctr /* -> nodes slot */) {
    if (!COUNT) return;
    unsigned long long a = wc.nodes, b = wc.tris, c = wc.spheres;
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_down_sync(0xffffffffu, a, o);
        b += __shfl_down_sync(0xffffffffu, b, o);
        c += __shfl_down_sync(0xffffffffu, c, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(ctr + 0, a);
        atomicAdd(ctr + 1, b);
        atomicAdd(ctr + 2, c);
    }
}

// Camera ray of queue entry i (Camera::calculateViewingRay, src/rtbase.h:74-84, from the pixel loop of
// src/scene.cpp:26-30).  sub > 1: supersampling — entry i is sample (i % sub^2) of slot first_slot + i / sub^2; its ray
// goes through the centre of cell (si, sj) of the sub x sub grid inside the pixel and carries weight 1/sub^2.
// Returns the framebuffer slot, or -1 for a slot outside the frame / a degenerate ray (the Ray ctor would throw).
struct PrimaryRays {
    FrameInfo F;
    long long first_slot;
    int sub;
    int depth;
};
__device__ __forceinline__ int primary_ray(const DScene& S, const PrimaryRays& pr, int i, d3& E, d3& d, double& w) {
    const int ss = pr.sub * pr.sub;
    const long long slot = pr.first_slot + (pr.sub > 1 ? i / ss : i);
    int px, py;
    if (!slot_to_pixel(pr.F, slot, px, py)) return -1;
    double rowFrac = (py + 0.5) / pr.F.height, colFrac = (px + 0.5) / pr.F.width;
    w = 1.0;
    if (pr.sub > 1) {
        const int k = i % ss, si = k % pr.sub, sj = k / pr.sub;
        rowFrac = (py + (sj + 0.5) / pr.sub) / pr.F.height;
        colFrac = (px + (si + 0.5) / pr.sub) / pr.F.width;
        w = 1.0 / ss;
    }
    const DCamera& c = S.cam;
    d3 LR = mk3(c.lr[0], c.lr[1], c.lr[2]), UR = mk3(c.ur[0], c.ur[1], c.ur[2]);
    d3 LL = mk3(c.ll[0], c.ll[1], c.ll[2]), UL = mk3(c.ul[0], c.ul[1], c.ul[2]);
    E = mk3(c.eye[0], c.eye[1], c.eye[2]);
    d3 right = rowFrac * LR + (1.0 - rowFrac) * UR;
    d3 left = rowFrac * LL + (1.0 - rowFrac) * UL;
    d3 ip = colFrac * right + (1.0 - colFrac) * left;
    d3 raw = ip - E;
    const bool ok = !(raw.x == 0 && raw.y == 0 && raw.z == 0);   // Ray ctor would throw (src/rtbase.h:19-20)
    d = ok ? ray_normalize(raw) : raw;
    return ok ? (int)slot : -1;
}

// Primary rays into a ray queue (only when the closest-hit kernel does not generate them itself: brute force).
__global__ void __launch_bounds__(RT_BLOCK) k_raygen(DScene S, PrimaryRays pr, int n, RayQ q) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    d3 E = mk3(0, 0, 0), d = mk3(0, 0, 1);
    double w = 1.0;
    const int slot = primary_ray(S, pr, i, E, d, w);
    q.fld(0, i) = E.x; q.fld(1, i) = E.y; q.fld(2, i) = E.z;
    q.fld(3, i) = d.x; q.fld(4, i) = d.y; q.fld(5, i) = d.z;
    q.fld(6, i) = w; q.fld(7, i) = w; q.fld(8, i) = w;
    q.pixel[i] = slot;
    q.meta[i] = pr.depth;
}

// Closest hit for every queued ray; hits are appended (compacted) to the hit queue.
// ids_geom/ids_face (optional, indexed by framebuffer slot) receive the hit ids.
// The queue holds its rays in two regions: entries [0, nfront) from the front (camera rays; reflected children) and
// the rest from the END backwards (refracted children), so a warp is one class of rays from neighbouring origins
// instead of an interleaving of the two.  Ray number g of the level sits at g (g < nfront) or cap - 1 - (g - nfront).
// PRIMARY: the rays of bounce level 0 are generated here (primary_ray) instead of being read from a queue a separate
// kernel filled — 80 B written and 80 B read per primary ray that never need to exist.
template <bool BRUTE, bool COUNT, bool PRIMARY>
__global__ void __launch_bounds__(RT_BLOCK, RT_TRACE_MINBLOCKS) k_trace(DScene S, RayQ q, size_t off, int n, size_t nfront, HitQ h,
                                                     unsigned long long* ctr, int* ids_geom, int* ids_face, PrimaryRays pr) {
    __shared__ __align__(16) unsigned char sm_stack[RT_SH_STACK_BYTES(false)];
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t g = off + (size_t)t;
    const size_t i = PRIMARY ? 0 : (g < nfront ? g : q.cap - 1 - (g - nfront));
    bool active = t < n;
    Best best;
    best.geom = -1;
    WorkCounters wc = {0, 0, 0};
    d3 o = mk3(0, 0, 0), d = mk3(0, 0, 1);
    double w0 = 1.0;
    int meta = 0, pixel = -1;
    if (PRIMARY) {
        if (active) pixel = primary_ray(S, pr, (int)g, o, d, w0);
        meta = pr.depth;
    } else {
        pixel = active ? q.pixel[i] : -1;
    }
    active = active && pixel >= 0;
    if (active) {
        if (!PRIMARY) {
            o = mk3(q.fld(0, i), q.fld(1, i), q.fld(2, i));
            d = mk3(q.fld(3, i), q.fld(4, i), q.fld(5, i));
            meta = q.meta[i];
        }
        cast_ray<false, BRUTE, COUNT>(S, o, d, (meta >> RT_META_INSIDE_SHIFT) & 1, 0.0, best, wc, stack_base<false>(sm_stack));
        if (ids_geom) { ids_geom[pixel] = best.geom; ids_face[pixel] = best.face; }
    }
    bool hit = active && best.geom >= 0;
    unsigned slot = warp_append(hit, ctr + CTR_HITS);
    if (hit) {
        h.fld(0, slot) = best.P.x; h.fld(1, slot) = best.P.y; h.fld(2, slot) = best.P.z;
        h.fld(3, slot) = best.N.x; h.fld(4, slot) = best.N.y; h.fld(5, slot) = best.N.z;
        h.fld(6, slot) = d.x; h.fld(7, slot) = d.y; h.fld(8, slot) = d.z;
        if (PRIMARY) { h.fld(9, slot) = w0; h.fld(10, slot) = w0; h.fld(11, slot) = w0; }
        else { h.fld(9, slot) = q.fld(6, i); h.fld(10, slot) = q.fld(7, i); h.fld(11, slot) = q.fld(8, i); }
        h.fld(12, slot) = best.wd;
        h.pixel[slot] = pixel;
        h.geom[slot] = best.geom;
        h.meta[slot] = meta;
    }
    flush_work<COUNT>(wc, ctr + CTR_NODES);
}

// ---- hit sorting (bounce levels >= 1) -----------------------------------------------------
// Hits of reflected / refracted rays arrive in an order that has little to do with where they
// are: ncu (round 1) shows 8 active lanes per instruction in the k_shadow launches of the
// bounce levels against 18 on the primary level.  Sorting the hit records by a Morton code of
// the hit point makes a warp 32 neighbouring origins again — for the shadow rays of this level
// and, because k_shade spawns in hit order, for the next level's rays.  It pays on the primary
// level too (neighbours on screen are not always neighbours in space).
struct SortGrid {
    float lo[3];
    float scale;      // cells per world unit (same on the three axes: cubic cells)
};
__device__ __forceinline__ uint32_t spread_bits3(uint32_t v) {   // 10 bits -> every third bit
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
__global__ void k_hit_keys(HitQ h, const unsigned long long* __restrict__ lc, SortGrid g, uint32_t* __restrict__ keys,
                           int* __restrict__ vals) {
    unsigned j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (unsigned)lc[CTR_HITS]) return;
    const float p[3] = {(float)h.fld(0, j), (float)h.fld(1, j), (float)h.fld(2, j)};
    uint32_t q[3];
    for (int a = 0; a < 3; a++) {
        float u = (p[a] - g.lo[a]) * g.scale;
        q[a] = (uint32_t)min(max((int)u, 0), 1023);
    }
    keys[j] = (spread_bits3(q[0]) << 2) | (spread_bits3(q[1]) << 1) | spread_bits3(q[2]);
    vals[j] = (int)j;
}
// --intersection-only: pixel = 1/dist^2 on all channels (src/scene.cpp:69-70)
__global__ void __launch_bounds__(RT_BLOCK) k_shade_io(HitQ h, const unsigned long long* ctr, double* fb,
                                                        unsigned long long* maxbits) {
    unsigned j = blockIdx.x * blockDim.x + threadIdx.x;
    double v = 0.0;
    if (j < (unsigned)ctr[CTR_HITS]) {
        double dist = h.fld(12, j);
        v = 1.0 / (dist * dist);
        size_t p = (size_t)h.pixel[j] * 3;
        fb[p] = v; fb[p + 1] = v; fb[p + 2] = v;
    }
    // non-negative doubles order like their bit patterns
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long x = __shfl_down_sync(0xffffffffu, b, o);
        b = x > b ? x : b;
    }
    if ((threadIdx.x & 31) == 0 && b) atomicMax(maxbits, b);
}

__global__ void k_divide(double* fb, size_t n, const unsigned long long* maxbits) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fb[i] = fb[i] / __longlong_as_double((long long)*maxbits);
}

// Normal fix-up, ambient term, and the bounce spawn.
// order != null (Morton-sorted level): hit j of this kernel is record order[j] of `src`
// (k_trace's unsorted appends); the complete record goes to h[j], so the separate permutation
// pass over the 116-byte records is folded into this kernel.  order == null: src is h itself.
#ifndef RT_SHADE_BLOCK
#define RT_SHADE_BLOCK 256     // streaming kernel: 8.8 ms with 64-thread blocks, 8.3 ms with 256 (8K synthetic frame)
#endif
__global__ void __launch_bounds__(RT_SHADE_BLOCK) k_shade(DScene S, HitQ src, HitQ h, const int* __restrict__ order,
                                                     unsigned long long* ctr, RayQ next, double* fb) {
    unsigned j = blockIdx.x * blockDim.x + threadIdx.x;
    bool active = j < (unsigned)ctr[CTR_HITS];
    bool want_t = false, want_r = false;
    d3 P = mk3(0, 0, 0), Td = P, Rd = P;
    double W[3] = {0, 0, 0}, kr[3] = {0, 0, 0};
    int pixel = 0, depth = 0, inside = 0;
    unsigned degenerate = 0;
    if (active) {
        const unsigned s = order ? (unsigned)order[j] : j;
        P = mk3(src.fld(0, s), src.fld(1, s), src.fld(2, s));
        d3 N = mk3(src.fld(3, s), src.fld(4, s), src.fld(5, s));
        d3 V = mk3(src.fld(6, s), src.fld(7, s), src.fld(8, s));
        W[0] = src.fld(9, s); W[1] = src.fld(10, s); W[2] = src.fld(11, s);
        pixel = src.pixel[s];
        int meta = src.meta[s];
        const int geom = src.geom[s];
        depth = meta & RT_META_DEPTH_MASK;
        inside = (meta >> RT_META_INSIDE_SHIFT) & 1;
        const DMat* m = S.mats + S.geoms[geom].mat;
        if (inside) N = -N;                                   // src/scene.cpp:72-73
        N = inplace_normalize(N);                             // src/scene.cpp:75
        h.fld(3, j) = N.x; h.fld(4, j) = N.y; h.fld(5, j) = N.z;
        if (order) {
            h.fld(0, j) = P.x; h.fld(1, j) = P.y; h.fld(2, j) = P.z;
            h.fld(6, j) = V.x; h.fld(7, j) = V.y; h.fld(8, j) = V.z;
            h.fld(9, j) = W[0]; h.fld(10, j) = W[1]; h.fld(11, j) = W[2];
            h.fld(12, j) = src.fld(12, s);
            h.pixel[j] = pixel;
            h.geom[j] = geom;
            h.meta[j] = meta;
        }
        // ambient lights (src/scene.cpp:80-84)
        if (S.num_alights > 0) {
            double c[3] = {0, 0, 0};
            for (int a = 0; a < S.num_alights; a++)
                for (int k = 0; k < 3; k++) c[k] += 1.0 * S.alights[a].color[k] * m->ka[k];
            for (int k = 0; k < 3; k++) atomicAdd(fb + (size_t)pixel * 3 + k, W[k] * c[k]);
        }
        // bounce (src/scene.cpp:114-136)
        kr[0] = m->kr[0]; kr[1] = m->kr[1]; kr[2] = m->kr[2];
        bool has_kr = m->has_kr != 0;
        if (depth > 0) {
            if (m->has_kt) {
                double n = m->ior;
                if (!inside) n = 1.0 / n;
                double cosI = dot4(N, V);
                double sinT2 = n * n * (1.0 - cosI * cosI);
                if (sinT2 > 1.0) {
                    kr[0] = kr[1] = kr[2] = 1.0;              // total internal reflection
                    has_kr = true;
                } else {
                    d3 T = n * V - (n * cosI + sqrt(1.0 - sinT2)) * N;
                    if (T.x == 0 && T.y == 0 && T.z == 0) degenerate++;
                    else { Td = ray_normalize(T); want_t = true; }
                }
            }
            if (has_kr) {
                d3 Rv = V - (2 * dot4(N, V)) * N;
                if (Rv.x == 0 && Rv.y == 0 && Rv.z == 0) degenerate++;
                else { Rd = ray_normalize(Rv); want_r = true; }
            }
        }
    }
    unsigned st = (unsigned)next.cap - 1u - warp_append(want_t, ctr + CTR_NEXT_T);
    if (want_t) {
        next.fld(0, st) = P.x; next.fld(1, st) = P.y; next.fld(2, st) = P.z;
        next.fld(3, st) = Td.x; next.fld(4, st) = Td.y; next.fld(5, st) = Td.z;
        next.fld(6, st) = W[0]; next.fld(7, st) = W[1]; next.fld(8, st) = W[2];   // weight 1, not kt
        next.pixel[st] = pixel;
        next.meta[st] = (depth - 1) | ((inside ^ 1) << RT_META_INSIDE_SHIFT);
    }
    unsigned sr = warp_append(want_r, ctr + CTR_NEXT);
    if (want_r) {
        next.fld(0, sr) = P.x; next.fld(1, sr) = P.y; next.fld(2, sr) = P.z;
        next.fld(3, sr) = Rd.x; next.fld(4, sr) = Rd.y; next.fld(5, sr) = Rd.z;
        next.fld(6, sr) = W[0] * kr[0]; next.fld(7, sr) = W[1] * kr[1]; next.fld(8, sr) = W[2] * kr[2];
        next.pixel[sr] = pixel;
        next.meta[sr] = (depth - 1) | (inside << RT_META_INSIDE_SHIFT);
    }
    if (degenerate) atomicAdd(ctr + CTR_DEGENERATE, (unsigned long long)degenerate);
}

// x^y of the shading terms (src/scene.cpp:103, src/lights.h:24).  These values only colour a
// pixel (gate 1e-9 on the FP64 frame; CUDA's pow already differs from glibc's in the last
// ulp), so a whole-number exponent up to 1024 — every shipped scene's `sp` — is evaluated by
// binary exponentiation (<= 20 multiplications, relative error <= y * 2^-53 <= 1.2e-13)
// instead of the ~150-instruction general pow.
__device__ __forceinline__ double pow_shading(double x, double y) {
    if (y >= 1.0 && y <= 1024.0 && y == floor(y)) {
        unsigned n = (unsigned)y;
        double r = 1.0, b = x;
        while (true) {
            if (n & 1u) r *= b;
            n >>= 1;
            if (!n) break;
            b *= b;
        }
        return r;
    }
    return pow(x, y);
}

// One thread per (hit, shadow light): occlusion query + Phong terms of that light.
template <bool BRUTE, bool COUNT>
__global__ void __launch_bounds__(RT_BLOCK, RT_SHADOW_MINBLOCKS) k_shadow(DScene S, HitQ h, unsigned long long* ctr, double* fb) {
    __shared__ __align__(16) unsigned char sm_stack[RT_SH_STACK_BYTES(true)];
    unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned nsl = (unsigned)S.num_slights;
    WorkCounters wc = {0, 0, 0};
    const unsigned long long nhits = ctr[CTR_HITS];
    if (t < nhits * nsl) {
        // light-major mapping: a warp = 32 consecutive hits (neighbouring pixels) towards the
        // SAME light, so its shadow rays are coherent; hit-record loads coalesce
        // ... in tiles of RT_SHADOW_TILE hits: all lights of one tile are processed back to
        // back, so its hit records (116 B each) are fetched from DRAM once and re-read from
        // L2 by the other lights instead of streaming the whole queue once per light
        unsigned long long tile;
        if (nhits * nsl <= 0xffffffffull) tile = (unsigned)t / (RT_SHADOW_TILE * nsl);     // 32-bit divide: ~5x cheaper
        else tile = t / ((unsigned long long)RT_SHADOW_TILE * nsl);
        const unsigned long long first = tile * RT_SHADOW_TILE;
        const unsigned w = (unsigned)min((unsigned long long)RT_SHADOW_TILE, nhits - first);   // hits in this tile
        const unsigned r = (unsigned)(t - tile * RT_SHADOW_TILE * nsl);
        const unsigned li = r / w, j = (unsigned)first + r % w;
        const DLight* l = S.slights + li;
        d3 P = mk3(h.fld(0, j), h.fld(1, j), h.fld(2, j));
        d3 N = mk3(h.fld(3, j), h.fld(4, j), h.fld(5, j));
        d3 lv = mk3(l->v[0], l->v[1], l->v[2]);
        const bool point = l->type == RT_LIGHT_POINT;
        d3 toL = point ? lv - P : -lv;                        // src/lights.h:34-37,50-53
        if (toL.x == 0 && toL.y == 0 && toL.z == 0) {
            atomicAdd(ctr + CTR_DEGENERATE, 1ull);            // reference would abort (src/rtbase.h:19-20)
            atomicAdd(ctr + CTR_S_DEGENERATE, 1ull);          // the host takes it back out of rays_shadow
        } else {
            d3 L = ray_normalize(toL);
            double ndl = dot4(N, L);
            bool lrev = ndl < 0;                              // src/scene.cpp:88
            const double INF = __longlong_as_double(0x7ff0000000000000ll);
            double dL = point ? norm4(toL) : INF;             // src/scene.cpp:89
            int inside = (h.meta[j] >> RT_META_INSIDE_SHIFT) & 1;
            // The Phong terms of this light (src/scene.cpp:95-106) BEFORE the occlusion query: when both are exactly
            // zero (light behind the surface and no specular lobe towards the viewer) the light adds +0 whether or not
            // it is occluded, so the query's answer cannot reach the frame and the traversal is skipped.  The
            // reference casts that shadow ray too; it is still counted (rays_shadow = hits x lights - degenerate ones).
            const DMat* m = S.mats + S.geoms[h.geom[j]].mat;
            d3 V = mk3(h.fld(6, j), h.fld(7, j), h.fld(8, j));
            double att[3];
            if (point) {
                // src/lights.h:23-25.  pow(x, +-0) is exactly 1 for every x (IEEE 754 / C Annex F)
                const double fo = l->falloff;
                double f = fo == 0.0 ? 1.0 : (fo == 1.0 ? 1.0 / dL : (fo == 2.0 ? 1.0 / (dL * dL) : pow(dL, -fo)));
                for (int k = 0; k < 3; k++) att[k] = f * l->color[k];
            } else {
                for (int k = 0; k < 3; k++) att[k] = l->color[k];
            }
            double di = ndl < 0.0 ? 0.0 : ndl;                // std::max(N.L, 0.0)
            d3 R = (2 * ndl) * N - L;                         // src/scene.cpp:101-102
            double mvr = -dot4(V, R);
            // std::pow(std::max(-V.R, 0.0), sp); pow(+0, y > 0) is exactly +0 (C Annex F)
            const double sp_ = m->sp;
            double si = (mvr < 0.0 && sp_ > 0.0) ? 0.0 : pow_shading(mvr < 0.0 ? 0.0 : mvr, sp_);
            double c[3];
            bool any = false;
            for (int k = 0; k < 3; k++) {
                double w = h.fld(9 + k, j);
                c[k] = w * (di * att[k] * m->kd[k]) + w * (si * att[k] * m->ks[k]);
                any = any || !(c[k] == 0.0);                  // NaN counts as a contribution (the reference would add it)
            }
            if (COUNT && !any) atomicAdd(ctr + CTR_S_CULLED, 1ull);
            if (any) {
                Best best;
                bool occluded = cast_ray<true, BRUTE, COUNT>(S, P, L, lrev != (inside != 0), dL, best, wc, stack_base<true>(sm_stack));
                if (!occluded) {
                    int pixel = h.pixel[j];
                    for (int k = 0; k < 3; k++) atomicAdd(fb + (size_t)pixel * 3 + k, c[k]);
                }
            }
        }
    }
    flush_work<COUNT>(wc, ctr + CTR_S_NODES);
}

// Framebuffer slot order -> output.  full = row-major frame (tile_world == 1), otherwise
// the packed tile layout is kept.  QUANT applies src/writers.cpp:7.
__device__ __forceinline__ unsigned char quantize(double v) {
    v = (1.0 < v) ? 1.0 : v;
    v = (v < 0.0) ? 0.0 : v;
    if (v != v) v = 0.0;
    return (unsigned char)(int)(v * 255.0);
}
template <bool QUANT>
__global__ void k_resolve(FrameInfo F, const double* __restrict__ fb, long long nslots, int full, void* out) {
    long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= nslots) return;
    int px, py;
    bool inside = slot_to_pixel(F, slot, px, py);
    size_t dst;
    if (full) {
        if (!inside) return;
        dst = ((size_t)py * F.width + px) * 3;
    } else {
        dst = (size_t)slot * 3;
    }
    for (int k = 0; k < 3; k++) {
        double v = inside ? fb[(size_t)slot * 3 + k] : 0.0;
        if (QUANT) ((unsigned char*)out)[dst + k] = quantize(v);
        else ((double*)out)[dst + k] = v;
    }
}

// Full-frame RGB8 resolve for a frame that lives on ANOTHER device (peer-mapped, NVLink) or in pinned host
// memory (PCIe): the stores are what costs there, so one block takes 256 consecutive slots = 8 rows x 32 pixels
// of one tile, stages the quantised bytes in shared memory and stores them as 4-byte words, 24 per row (96
// contiguous bytes = three whole sectors per row) instead of three single-byte stores per pixel.
#if RT_TILE_W == 32
__global__ void __launch_bounds__(256) k_resolve_rgb8_rows(FrameInfo F, const double* __restrict__ fb, long long nslots,
                                                            unsigned char* __restrict__ out) {
    __shared__ __align__(16) unsigned char rows[8][96];
    const long long slot0 = (long long)blockIdx.x * 256;
    const long long slot = slot0 + threadIdx.x;
    int px, py;
    const bool inside = slot < nslots && slot_to_pixel(F, slot, px, py);
    {
        const int j = threadIdx.x, w = j >> 5, l = j & 31;
        const int x = (w & 3) * 8 + (l & 7), y = (w >> 2) * 4 + (l >> 3);
        for (int k = 0; k < 3; k++) rows[y][3 * x + k] = inside ? quantize(fb[(size_t)slot * 3 + k]) : 0;
    }
    __syncthreads();
    // pixel of the block's first slot = upper left corner of the 32 x 8 strip
    int px0, py0;
    if (slot0 >= nslots) return;
    slot_to_pixel(F, slot0, px0, py0);
    if (threadIdx.x < 192) {
        const int r = threadIdx.x / 24, wd = threadIdx.x % 24;
        const int y = py0 + r;
        if (y < F.height) {
            const size_t base = ((size_t)y * F.width + px0) * 3;
            if (px0 + 32 <= F.width && (base & 3) == 0) {
                *reinterpret_cast<unsigned*>(out + base + 4 * wd) = *reinterpret_cast<const unsigned*>(&rows[r][4 * wd]);
            } else {
                const int nb = 3 * min(32, F.width - px0);
                for (int bidx = 4 * wd; bidx < 4 * wd + 4; bidx++)
                    if (bidx < nb) out[base + bidx] = rows[r][bidx];
            }
        }
    }
}
#endif

// Gathered packed tiles (rank-major, each rank padded to max_tiles) -> row-major frame.
template <typename T>
__global__ void k_unpack(int width, int height, int tiles_x, int world, long long max_tiles,
                         const int* __restrict__ rank_row_start /*[world][tiles_y+1]*/, int tiles_y,
                         const T* __restrict__ packed, T* __restrict__ frame) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)width * height) return;
    int px = (int)(i % width), py = (int)(i / width);
    int tx = px / RT_TILE_W, ty = py / RT_TILE_H;
    int rank = (tx + ty) % world;
    int first_tx = ((rank - ty) % world + world) % world;
    long long lt = rank_row_start[rank * (tiles_y + 1) + ty] + (tx - first_tx) / world;
    int x = px % RT_TILE_W, y = py % RT_TILE_H;
    int w = (y / 4) * (RT_TILE_W / 8) + (x / 8), l = (y % 4) * 8 + (x % 8);
    long long slot = ((long long)rank * max_tiles + lt) * RT_TILE_PIXELS + w * 32 + l;
    for (int k = 0; k < 3; k++) frame[i * 3 + k] = packed[slot * 3 + k];
}

// per-ray query (rt_cast_rays): dir normalised like the Ray ctor
template <bool BRUTE>
__global__ void __launch_bounds__(RT_BLOCK) k_query(DScene S, long long n, const double* __restrict__ org,
                                                     const double* __restrict__ dir,
                                                     const unsigned char* __restrict__ reverse, int* geom, int* face,
                                                     double* dist, double* point, double* normal) {
    __shared__ __align__(16) unsigned char sm_stack[RT_SH_STACK_BYTES(false)];
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    d3 o = mk3(org[3 * i], org[3 * i + 1], org[3 * i + 2]);
    d3 raw = mk3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
    Best best;
    best.geom = -1; best.face = -1; best.wd = 0; best.P = mk3(0, 0, 0); best.N = mk3(0, 0, 0);
    WorkCounters wc = {0, 0, 0};
    if (raw.x == 0 && raw.y == 0 && raw.z == 0) {
        best.geom = -2;
    } else {
        cast_ray<false, BRUTE, false, true>(S, o, ray_normalize(raw), reverse ? reverse[i] != 0 : false, 0.0, best, wc, stack_base<false>(sm_stack));
    }
    bool hit = best.geom >= 0;
    if (geom) geom[i] = best.geom;
    if (face) face[i] = hit ? best.face : -1;
    if (dist) dist[i] = hit ? best.wd : 0.0;
    if (point) { point[3 * i] = hit ? best.P.x : 0; point[3 * i + 1] = hit ? best.P.y : 0; point[3 * i + 2] = hit ? best.P.z : 0; }
    if (normal) { normal[3 * i] = hit ? best.N.x : 0; normal[3 * i + 1] = hit ? best.N.y : 0; normal[3 * i + 2] = hit ? best.N.z : 0; }
}

// Node-bandwidth roofline probe: every thread issues `loads` independent 32-byte gathers
// (two float4 __ldg of one 32-byte-aligned record) at hashed positions.
__global__ void k_gather_probe(const float4* __restrict__ data, unsigned long long nrec, int loads, float* sink) {
    unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long x = t * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    float acc = 0.f;
    for (int i = 0; i < loads; i++) {
        x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
        unsigned long long r = x % nrec;
        float4 a = __ldg(data + 2 * r), b = __ldg(data + 2 * r + 1);
        acc += a.x + b.w;
    }
    if (acc == 123.456f) *sink = acc;
}

// Node-visit ceiling probe (the "measured BVH-node-bandwidth roofline" of BASELINE.json): threads walk the REAL
// 4-wide node array of the uploaded scene with exactly the loads of descend() — three near planes picked by a
// direction sign, the three far planes at address ^ 64, the four child references; 7 x 16 B = 112 B per visit — and
// nothing else: no slab arithmetic, no stack, no primitive tests.  The next node is one of the internal children
// just loaded (a dependent fetch, like a traversal step), picked by a hash; a node without internal children
// restarts the walk at the root (the next ray).  `group` consecutive lanes share one path: group = 32 is a fully
// coherent warp (every load a broadcast), group = 1 gives every lane its own path.  Same block size and
// occupancy as the traversal kernels.  What it measures is the rate at which the memory system (L1TEX / L2)
// can feed node visits to this access pattern; a traversal kernel cannot visit nodes faster.
__global__ void __launch_bounds__(RT_BLOCK, RT_SHADOW_MINBLOCKS) k_node_walk(const BvhNode* __restrict__ nodes, int visits,
                                                                              int group, float* sink) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned path = t / (unsigned)group;
    unsigned long long x = (unsigned long long)path * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27;
    // per-path "direction signs": which half of the node holds the near planes (see FRay)
    const unsigned nx = (x & 1) ? 64u : 0u, ny = (x & 2) ? 80u : 16u, nz = (x & 4) ? 96u : 32u;
    float acc = 0.f;
    int cur = 0;
    const char* const nb = reinterpret_cast<const char*>(nodes);
    for (int v = 0; v < visits; v++) {
        const unsigned off = (unsigned)cur * (unsigned)sizeof(BvhNode);
        const float4* pnx = reinterpret_cast<const float4*>(nb + (off + nx));
        const float4* pny = reinterpret_cast<const float4*>(nb + (off + ny));
        const float4* pnz = reinterpret_cast<const float4*>(nb + (off + nz));
        const float4 a = __ldg(pnx), b = __ldg(pny), c = __ldg(pnz);
        const float4 d = __ldg(flip64(pnx)), e = __ldg(flip64(pny)), f = __ldg(flip64(pnz));
        const int4 ref = __ldg(reinterpret_cast<const int4*>(nb + off + 48));
        acc += a.x + b.y + c.z + d.w + e.x + f.y;
        x = x * 6364136223846793005ull + 1442695040888963407ull;
        const unsigned r = (unsigned)(x >> 33);
        // hashed pick among the internal children, first candidate by rotation
        const int cand[4] = {ref.x, ref.y, ref.z, ref.w};
        int next = 0;
#pragma unroll
        for (int k = 3; k >= 0; k--) {
            const int cc = cand[(r + k) & 3];
            next = cc >= 0 ? cc : next;
        }
        cur = next;        // 0 (the root) when every child is a leaf or empty
    }
    if (acc == 123.456f) *sink = acc;
}

// A geometry that owns faces (TRI or MESH), sorted by first_face: lets the device derive the
// per-face (geometry, local index) pair and the primitive-code lists instead of the host
// building and uploading four million-entry arrays per scene upload.
struct FaceOwner {
    int geom, first, count;
    int all_off;      // MESH: position of its first face in all_prims; -1 for a TRI
    int bvh_off;      // MESH: position of its first face in bvh_prims; -1 for a TRI
};

// Raw faces (3 points / 3 normals, 9 doubles each) -> 80-byte device records, plus the
// FACE primitive codes of mesh faces in reference order (all_prims) and LBVH order (bvh_prims).
__global__ void k_pack_faces(long long nf, const double* __restrict__ pts, const double* __restrict__ nrm,
                             const FaceOwner* __restrict__ owners, int nowners, double2* __restrict__ out_p,
                             double2* __restrict__ out_n, int* __restrict__ all_prims, int* __restrict__ bvh_prims) {
    long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nf) return;
    // owner = last entry with first <= f (if f lies inside its range)
    int lo = 0, hi = nowners;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (owners[mid].first <= (int)f) lo = mid + 1;
        else hi = mid;
    }
    int fgeom = 0, flocal = 0;
    if (lo > 0) {
        const FaceOwner o = owners[lo - 1];
        if ((int)f - o.first < o.count) {
            fgeom = o.geom;
            flocal = (int)f - o.first;
            if (o.all_off >= 0) {
                const int code = (PRIM_FACE << PRIM_KIND_SHIFT) | (int)f;
                all_prims[o.all_off + flocal] = code;
                bvh_prims[o.bvh_off + flocal] = code;
            }
        }
    }
    const double* p = pts + 9 * f;
    const double* n = nrm + 9 * f;
    d3 p0 = mk3(p[0], p[1], p[2]), p1 = mk3(p[3], p[4], p[5]), p2 = mk3(p[6], p[7], p[8]);
    d3 va = p1 - p0, vb = p2 - p0;    // the per-ray subtractions of src/geometry.cpp:80-81, done once
    double aux = __hiloint2double(flocal, fgeom);
    double2* q = out_p + f * RT_FACE_D2;
    q[0] = make_double2(p0.x, p0.y);
    q[1] = make_double2(p0.z, va.x);
    q[2] = make_double2(va.y, va.z);
    q[3] = make_double2(vb.x, vb.y);
    q[4] = make_double2(vb.z, aux);
    double2* m = out_n + f * RT_FACE_D2;
    m[0] = make_double2(n[0], n[1]);
    m[1] = make_double2(n[2], n[3]);
    m[2] = make_double2(n[4], n[5]);
    m[3] = make_double2(n[6], n[7]);
    m[4] = make_double2(n[8], 0.0);
}

// dst[pos[i]] = code[i]: the (few) sphere / `tri` codes of all_prims
__global__ void k_scatter_codes(int n, const int* __restrict__ pos, const int* __restrict__ code, int* __restrict__ dst) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[pos[i]] = code[i];
}

}  // namespace rt
