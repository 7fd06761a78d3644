// rt_bvh.cu — GPU LBVH build: primitive bounds -> 30-bit Morton codes -> hand-written
// LSD radix sort (no CUB) -> Karras hierarchy (pure integer, deterministic) -> bottom-up
// refit -> treelet restructuring -> least-cost collapse into 128-byte 4-wide nodes.  It replaces the reference's only acceleration structure,
// one object-space AABB per .obj mesh (Mesh::updateBoundingBox src/geometry.cpp:145-162,
// hitsBoundingBox src/geometry.cpp:5-29).  The boxes only CULL (FP32, padded outward);
// every hit decision is still the exact FP64 test in rt_device.cuh.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "rt_bvh.h"
#include "rt_sort.cuh"

namespace rt {

// ---- float <-> ordered int so atomicMin/atomicMax work on floats -----------------
__device__ __forceinline__ int f2ord(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__host__ __device__ __forceinline__ float ord2f(int i) {
    int j = i >= 0 ? i : i ^ 0x7fffffff;
#ifdef __CUDA_ARCH__
    return __int_as_float(j);
#else
    float f;
    memcpy(&f, &j, 4);
    return f;
#endif
}

// World-space bounds of the primitive with code `code` (FP64 math, rounded outward to FP32).  The build and the
// refit both call this, so a refit of unchanged primitives reproduces the build's boxes bit for bit.
__device__ __forceinline__ void prim_bounds(const DScene& S, int code, float lo[3], float hi[3]) {
    int kind = code >> PRIM_KIND_SHIFT, idx = code & PRIM_INDEX_MASK;
    double mn[3] = {DBL_MAX, DBL_MAX, DBL_MAX}, mx[3] = {-DBL_MAX, -DBL_MAX, -DBL_MAX};
    auto grow = [&](d3 p) {
        mn[0] = fmin(mn[0], p.x); mn[1] = fmin(mn[1], p.y); mn[2] = fmin(mn[2], p.z);
        mx[0] = fmax(mx[0], p.x); mx[1] = fmax(mx[1], p.y); mx[2] = fmax(mx[2], p.z);
    };
    auto face_bounds = [&](int gface, const DGeom* g) {
        const double2* fp = S.face_pts + (size_t)gface * RT_FACE_D2;
        double2 q0 = fp[0], q1 = fp[1], q2 = fp[2], q3 = fp[3], q4 = fp[4];
        d3 p0 = mk3(q0.x, q0.y, q1.x), va = mk3(q1.y, q2.x, q2.y), vb = mk3(q3.x, q3.y, q4.x);
        grow(xf_point(g->fwd, p0));
        grow(xf_point(g->fwd, p0 + va));
        grow(xf_point(g->fwd, p0 + vb));
    };
    if (kind == PRIM_SPHERE) {
        const DGeom* g = S.geoms + idx;
        d3 c = xf_point(g->fwd, mk3(g->center[0], g->center[1], g->center[2]));
        double r = sqrt(g->radius2) * (1.0 + 1e-7);
        double cc[3] = {c.x, c.y, c.z};
        for (int a = 0; a < 3; a++) {
            const double* row = g->fwd + 4 * a;
            double e = r * sqrt(row[0] * row[0] + row[1] * row[1] + row[2] * row[2]);
            mn[a] = cc[a] - e;
            mx[a] = cc[a] + e;
        }
    } else if (kind == PRIM_TRI) {
        const DGeom* g = S.geoms + idx;
        face_bounds(g->first_face, g);
        face_bounds(g->first_face + 1, g);
    } else {
        double2 q4 = S.face_pts[(size_t)idx * RT_FACE_D2 + 4];
        face_bounds(idx, S.geoms + __double2loint(q4.y));
    }
    for (int a = 0; a < 3; a++) {
        lo[a] = __double2float_rd(mn[a]);
        hi[a] = __double2float_ru(mx[a]);
    }
}

__global__ void k_prim_bounds(DScene S, const int* __restrict__ codes, int n, float* __restrict__ lo,
                              float* __restrict__ hi, int* __restrict__ gbounds /*[7]: cmin xyz, cmax xyz, maxabs*/) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float pl[3], ph[3];
    prim_bounds(S, codes[i], pl, ph);
    float maxabs = 0.f;
    for (int a = 0; a < 3; a++) {
        float l = pl[a], h = ph[a];
        lo[3 * (size_t)i + a] = l;
        hi[3 * (size_t)i + a] = h;
        float c = 0.5f * l + 0.5f * h;
        atomicMin(&gbounds[a], f2ord(c));
        atomicMax(&gbounds[3 + a], f2ord(c));
        maxabs = fmaxf(maxabs, fmaxf(fabsf(l), fabsf(h)));
    }
    atomicMax(&gbounds[6], f2ord(maxabs));
}

__device__ __forceinline__ uint32_t expand10(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__global__ void k_morton(const float* __restrict__ lo, const float* __restrict__ hi, int n,
                         const int* __restrict__ gbounds, uint32_t* __restrict__ keys, int* __restrict__ vals) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // Quantise all three axes with the SAME cell size (the largest centroid extent): cubic
    // Morton cells.  Normalising each axis separately would spend as many bits on the thin
    // axis of a 2.5-D scene (a height field) as on the long ones and cut it into "hills" and
    // "valleys" whose boxes overlap everywhere.
    uint32_t q[3];
    float ext = 0.f;
    for (int a = 0; a < 3; a++) ext = fmaxf(ext, ord2f(gbounds[3 + a]) - ord2f(gbounds[a]));
    for (int a = 0; a < 3; a++) {
        float cmin = ord2f(gbounds[a]);
        float c = 0.5f * lo[3 * (size_t)i + a] + 0.5f * hi[3 * (size_t)i + a];
        float u = ext > 0.f ? (c - cmin) / ext : 0.f;
        int v = (int)(u * 1024.f);
        q[a] = (uint32_t)min(max(v, 0), 1023);
    }
    keys[i] = (expand10(q[0]) << 2) | (expand10(q[1]) << 1) | expand10(q[2]);
    vals[i] = i;
}

// ---- Karras 2012 ---------------------------------------------------------------------
__device__ __forceinline__ int delta(const uint32_t* __restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    uint32_t a = keys[i], b = keys[j];
    if (a == b) return 32 + __clz(i ^ j);
    return __clz(a ^ b);
}

// child encoding inside the build: >= 0 internal node, < 0 leaf ~index (sorted position)
__global__ void k_karras(const uint32_t* __restrict__ keys, int n, int* __restrict__ left, int* __restrict__ right,
                         int* __restrict__ parent_int, int* __restrict__ parent_leaf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, n, i, j);
    int s = 0;
    int t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int lo = min(i, j), hi = max(i, j);
    int lc, rc;
    if (lo == gamma) { lc = ~gamma; parent_leaf[gamma] = i; } else { lc = gamma; parent_int[gamma] = i; }
    if (hi == gamma + 1) { rc = ~(gamma + 1); parent_leaf[gamma + 1] = i; } else { rc = gamma + 1; parent_int[gamma + 1] = i; }
    left[i] = lc;
    right[i] = rc;
    if (i == 0) parent_int[0] = -1;
}

__global__ void k_refit(int n, const int* __restrict__ vals, const float* __restrict__ plo,
                        const float* __restrict__ phi, const int* __restrict__ left, const int* __restrict__ right,
                        const int* __restrict__ parent_int, const int* __restrict__ parent_leaf,
                        float* __restrict__ ilo, float* __restrict__ ihi, int* __restrict__ flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int cur = parent_leaf[i];
    while (cur >= 0) {
        if (atomicAdd(&flags[cur], 1) == 0) return;     // first arrival waits for the sibling
        __threadfence();
        float lo[3], hi[3];
        for (int a = 0; a < 3; a++) { lo[a] = FLT_MAX; hi[a] = -FLT_MAX; }
        int ch[2] = {left[cur], right[cur]};
        for (int k = 0; k < 2; k++) {
            const float *bl, *bh;
            if (ch[k] < 0) {
                int p = vals[~ch[k]];
                bl = plo + 3 * (size_t)p; bh = phi + 3 * (size_t)p;
            } else {
                bl = ilo + 3 * (size_t)ch[k]; bh = ihi + 3 * (size_t)ch[k];
            }
            for (int a = 0; a < 3; a++) {
                lo[a] = fminf(lo[a], __ldcg(bl + a));
                hi[a] = fmaxf(hi[a], __ldcg(bh + a));
            }
        }
        for (int a = 0; a < 3; a++) { ilo[3 * (size_t)cur + a] = lo[a]; ihi[3 * (size_t)cur + a] = hi[a]; }
        __threadfence();
        cur = parent_int[cur];
    }
}

// depth of every internal node of one group's tree (root = 0) by walking the parent chain
__global__ void k_depth(int n, const int* __restrict__ parent_int, int* __restrict__ depth, int* __restrict__ max_depth) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = 0;
    for (int p = parent_int[i]; p >= 0; p = parent_int[p]) d++;
    depth[i] = d;
    // deepest internal node of this group's tree (bounds the traversal stack of the even-depth collapse, see build_lbvh)
    const unsigned act = __activemask();
    const int m = __reduce_max_sync(act, d);
    if ((int)(threadIdx.x & 31) == __ffs(act) - 1) atomicMax(max_depth, m);
}

// ---- Cost model of the tree optimisations below ----------------------------------------------------------------
// Surface-area heuristic: a ray that enters a box of area A_parent enters a child box of area A with probability
// A / A_parent.  The expected work of a ray is then C_node * sum(area of the wide nodes it may visit) + C_prim *
// sum(area of the leaf boxes), over the area of the root.  The traversal kernels are bound by the LSU write-back of
// what they load (DESIGN section 5): a wide-node visit loads 112 B, an exact face test 80 B, so C_prim / C_node is
// about 0.7.  With ONE primitive per leaf the leaf term is the same for every topology over the same primitives, so
// neither pass below depends on the two constants: the treelet pass minimises the summed area of the binary internal
// nodes, the collapse the summed area of the binary nodes chosen to be wide nodes.
__device__ __forceinline__ float box_area(const float* lo, const float* hi) {
    const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
    return ex * ey + ey * ez + ez * ex;
}

// Box of a binary-tree child reference (>= 0 internal node, < 0 leaf ~sorted position), read through L2: the
// bottom-up passes read what other threads of the same launch wrote.
__device__ __forceinline__ void child_box(int c, const int* vals, const float* plo, const float* phi, const float* ilo,
                                          const float* ihi, float lo[3], float hi[3]) {
    const float *bl, *bh;
    if (c < 0) {
        const int p = vals[~c];
        bl = plo + 3 * (size_t)p; bh = phi + 3 * (size_t)p;
    } else {
        bl = ilo + 3 * (size_t)c; bh = ihi + 3 * (size_t)c;
    }
    for (int a = 0; a < 3; a++) { lo[a] = __ldcg(bl + a); hi[a] = __ldcg(bh + a); }
}

// Treelet restructuring (Karras & Aila, HPG 2013), one bottom-up pass with k_refit's arrival counters.  The thread
// that arrives second at an internal node (both subtrees are final) grows a treelet from it by expanding the
// internal treelet leaf of largest area until TREELET_LEAVES leaves, finds the topology of least summed internal area
// over those leaves by dynamic programming over their subsets, and rewires the treelet's own internal nodes into it
// (the node keeps its index and its parent, so the set of internal indices and the root stay as k_karras made them).
// Deterministic: every comparison is strict in a fixed order (ties keep the lower slot / the first partition
// enumerated) and the boxes are min/max of primitive boxes, so scheduling cannot change the result.
#define TREELET_LEAVES 7
// Rounds of the whole pass (a later round sees the treelets the earlier one made).  Box tests per frame of the
// 1 M-triangle scene after 0 / 1 / 2 / 3 rounds (with the least-cost collapse): 24.75 / 23.34 / 22.94 / 22.81 G.
#define TREELET_ROUNDS 2
#define TREELET_THREADS 64
#define COST(s) s_cost[(s) * TREELET_THREADS + threadIdx.x]

// Best split of treelet subset s (>= 2 leaves) into two parts, the part with the lowest leaf returned; each
// partition is enumerated once, in a fixed order, and the first of equal costs wins.
__device__ __forceinline__ int treelet_split(const float* s_cost, int s, float* best_cost) {
    const int low = s & -s, rest = s ^ low;
    float best = FLT_MAX;
    int bp = low;
    for (int q = (rest - 1) & rest;; q = (q - 1) & rest) {
        const int p = q | low;
        const float c = COST(p) + COST(s ^ p);
        if (c < best) { best = c; bp = p; }
        if (q == 0) break;
    }
    *best_cost = best;
    return bp;
}

// Launched with TREELET_THREADS threads per block and TREELET_THREADS << TREELET_LEAVES floats of shared memory.
__global__ void __launch_bounds__(TREELET_THREADS, 1) k_treelet(int n, const int* __restrict__ vals, const float* __restrict__ plo, const float* __restrict__ phi,
                          int* left, int* right, int* parent_int, int* parent_leaf, float* ilo, float* ihi,
                          int* __restrict__ flags) {
    extern __shared__ float s_cost[];
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int cur = __ldcg(parent_leaf + i);
    while (cur >= 0) {
        if (atomicAdd(&flags[cur], 1) == 0) return;
        __threadfence();
        int leaf[TREELET_LEAVES], inner[TREELET_LEAVES - 1];
        float llo[TREELET_LEAVES][3], lhi[TREELET_LEAVES][3], larea[TREELET_LEAVES];
        int nl = 2, ni = 1;
        inner[0] = cur;
        leaf[0] = __ldcg(left + cur);
        leaf[1] = __ldcg(right + cur);
        float old_cost;
        {
            float lo[3], hi[3];
            child_box(cur, vals, plo, phi, ilo, ihi, lo, hi);
            old_cost = box_area(lo, hi);
        }
        for (int k = 0; k < 2; k++) {
            child_box(leaf[k], vals, plo, phi, ilo, ihi, llo[k], lhi[k]);
            larea[k] = box_area(llo[k], lhi[k]);
        }
        while (nl < TREELET_LEAVES) {
            int best = -1;
            float ba = -1.f;
            for (int k = 0; k < nl; k++)
                if (leaf[k] >= 0 && larea[k] > ba) { ba = larea[k]; best = k; }
            if (best < 0) break;
            const int c = leaf[best];
            inner[ni++] = c;
            old_cost += ba;
            leaf[best] = __ldcg(left + c);
            leaf[nl] = __ldcg(right + c);
            for (int t = 0; t < 2; t++) {
                const int k = t ? nl : best;
                child_box(leaf[k], vals, plo, phi, ilo, ihi, llo[k], lhi[k]);
                larea[k] = box_area(llo[k], lhi[k]);
            }
            nl++;
        }
        if (nl > 2) {
            // COST(s): least summed area of the internal nodes of a tree over the leaves in subset s, in shared memory
            // as [subset][thread] so that every lane reads its own bank whatever subsets the lanes look up
            const int full = (1 << nl) - 1;
            for (int s = 1; s <= full; s++) {
                if ((s & (s - 1)) == 0) { COST(s) = 0.f; continue; }
                float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
                for (int k = 0; k < nl; k++)
                    if (s >> k & 1)
                        for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], llo[k][a]); hi[a] = fmaxf(hi[a], lhi[k][a]); }
                float best;
                treelet_split(s_cost, s, &best);
                COST(s) = box_area(lo, hi) + best;
            }
            if (COST(full) < 0.9999f * old_cost) {      // not for a rounding difference of the same topology
                // rewire: subsets in creation order take the treelet's internal nodes, inner[0] (= cur) stays the root
                int stack_s[TREELET_LEAVES], stack_n[TREELET_LEAVES], sp = 0, next = 1;
                stack_s[sp] = full; stack_n[sp++] = cur;
                while (sp > 0) {
                    const int s = stack_s[--sp], node = stack_n[sp];
                    float unused;
                    const int p = treelet_split(s_cost, s, &unused);
                    const int part[2] = {p, s ^ p};
                    int ch[2];
                    for (int k = 0; k < 2; k++) {
                        const int q = part[k];
                        if ((q & (q - 1)) == 0) {
                            ch[k] = leaf[__ffs(q) - 1];
                            if (ch[k] < 0) parent_leaf[~ch[k]] = node; else parent_int[ch[k]] = node;
                        } else {
                            ch[k] = inner[next++];
                            parent_int[ch[k]] = node;
                            stack_s[sp] = q; stack_n[sp++] = ch[k];
                        }
                    }
                    left[node] = ch[0];
                    right[node] = ch[1];
                    if (node != cur) {                       // the root's box is the union of the same leaves
                        float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
                        for (int k = 0; k < nl; k++)
                            if (s >> k & 1)
                                for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], llo[k][a]); hi[a] = fmaxf(hi[a], lhi[k][a]); }
                        for (int a = 0; a < 3; a++) { ilo[3 * (size_t)node + a] = lo[a]; ihi[3 * (size_t)node + a] = hi[a]; }
                    }
                }
            }
        }
        __threadfence();
        cur = __ldcg(parent_int + cur);
    }
}

// Least-cost collapse of the binary tree into a 4-wide one (Ylitie, Karras & Laine, HPG 2017, section 3), bottom-up
// with arrival counters.  Per internal node n (areas only, see the cost model above; leaves cost nothing):
//   S(n, k)  least cost of n's subtree spread over at most k >= 2 slots of the wide node above it without a node for
//            n itself: min over i + j <= k of D(left, i) + D(right, j);
//   D(n, 1)  = area(n) + S(n, 4): n becomes a wide node (its four slots hold S(n, 4));
//   D(n, k)  = min(D(n, 1), S(n, k)) for k = 2..4.
// dcost[n] = D(n, 1..4); choice[n] packs, for k = 2..4, the split (i | j << 2) of S(n, k) in bits 4(k-2).. and in bit
// 12 + k whether D(n, k) is n itself.  Ties keep the first candidate in a fixed order: deterministic.
// wdepth[n] packs, in byte k - 1, the number of wide levels the choice behind D(n, k) puts on the deepest path of n's
// subtree (saturated at 255), so byte 0 of the root is the depth of the wide tree before any of it is written.
__global__ void k_collapse_cost(int n, const int* __restrict__ left, const int* __restrict__ right,
                                const int* __restrict__ parent_int, const int* __restrict__ parent_leaf,
                                const float* __restrict__ ilo, const float* __restrict__ ihi, float4* dcost,
                                int* __restrict__ choice, int* wdepth, int* __restrict__ flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int cur = parent_leaf[i];
    while (cur >= 0) {
        if (atomicAdd(&flags[cur], 1) == 0) return;
        __threadfence();
        float dl[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, dr[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        const int l = left[cur], r = right[cur];
        if (l >= 0) { const float4 d = __ldcg(dcost + l); dl[1] = d.x; dl[2] = d.y; dl[3] = d.z; dl[4] = d.w; }
        if (r >= 0) { const float4 d = __ldcg(dcost + r); dr[1] = d.x; dr[2] = d.y; dr[3] = d.z; dr[4] = d.w; }
        int wl[5] = {0, 0, 0, 0, 0}, wr[5] = {0, 0, 0, 0, 0};
        if (l >= 0) { const int w = __ldcg(wdepth + l); for (int k = 1; k <= 4; k++) wl[k] = w >> (8 * (k - 1)) & 255; }
        if (r >= 0) { const int w = __ldcg(wdepth + r); for (int k = 1; k <= 4; k++) wr[k] = w >> (8 * (k - 1)) & 255; }
        float s[5];
        int ws[5];                                // wide levels below the slots of S(n, k)
        int code = 0, sij = 1 | 1 << 2;
        s[2] = dl[1] + dr[1];
        ws[2] = max(wl[1], wr[1]);
        for (int k = 2; k <= 4; k++) {
            if (k > 2) { s[k] = s[k - 1]; ws[k] = ws[k - 1]; }
            for (int a = 1; a < k; a++) {
                const float c = dl[a] + dr[k - a];
                if (c < s[k]) { s[k] = c; sij = a | (k - a) << 2; ws[k] = max(wl[a], wr[k - a]); }
            }
            code |= sij << (4 * (k - 2));
        }
        float lo[3], hi[3];
        for (int a = 0; a < 3; a++) { lo[a] = ilo[3 * (size_t)cur + a]; hi[a] = ihi[3 * (size_t)cur + a]; }
        float d[5];
        d[1] = box_area(lo, hi) + s[4];
        const int w1 = min(ws[4] + 1, 255);
        int wd = w1;
        for (int k = 2; k <= 4; k++) {
            if (d[1] <= s[k]) { d[k] = d[1]; code |= 1 << (12 + k); wd |= w1 << (8 * (k - 1)); }
            else { d[k] = s[k]; wd |= ws[k] << (8 * (k - 1)); }
        }
        dcost[cur] = make_float4(d[1], d[2], d[3], d[4]);
        choice[cur] = code;
        wdepth[cur] = wd;
        __threadfence();
        cur = parent_int[cur];
    }
}

// Top-down half of the collapse, one launch per level of the wide tree: every wide node of wave w expands its S(n, 4)
// into at most four slots; the internal nodes among them are the wide nodes of wave w + 1.  wave_of[]: wave of every
// wide node (-1: none); slots4[]: its children (BVH_DONE: none).
__global__ void k_choose_children(int n, int wave, int* __restrict__ wave_of, int4* __restrict__ slots4,
                                  const int* __restrict__ left, const int* __restrict__ right,
                                  const int* __restrict__ choice) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1 || wave_of[i] != wave) return;
    int slots[4] = {BVH_DONE, BVH_DONE, BVH_DONE, BVH_DONE};
    int ns = 0;
    int st_n[4], st_k[4], sp = 0;                // (subtree, slots it may fill); at most four entries are pending
    {
        const int ij = choice[i] >> 8 & 15;      // split of S(i, 4)
        st_n[sp] = right[i]; st_k[sp++] = ij >> 2;
        st_n[sp] = left[i]; st_k[sp++] = ij & 3;
    }
    while (sp > 0) {
        const int c = st_n[--sp], k = st_k[sp];
        const int code = c >= 0 ? choice[c] : 0;
        if (c < 0 || k == 1 || (code >> (12 + k) & 1)) {
            slots[ns++] = c;
            if (c >= 0) wave_of[c] = wave + 1;
            continue;
        }
        const int ij = code >> (4 * (k - 2)) & 15;
        st_n[sp] = right[c]; st_k[sp++] = ij >> 2;
        st_n[sp] = left[c]; st_k[sp++] = ij & 3;
    }
    slots4[i] = make_int4(slots[0], slots[1], slots[2], slots[3]);
}

// Padding of every stored child box: a few FP32 ulps at the scene's largest coordinate M (covers the slab test's
// rounding), plus a relative margin.  The build and the refit share these, so equal boxes give equal bytes.
__host__ __device__ __forceinline__ float box_pad(float m) { return 2e-6f * fmaxf(m, 1e-30f); }
__host__ __device__ __forceinline__ float pad_lo(float l, float pad) { return l - pad - fabsf(l) * 2e-7f; }
__host__ __device__ __forceinline__ float pad_hi(float h, float pad) { return h + pad + fabsf(h) * 2e-7f; }

// Binary Karras nodes at EVEN depth become 4-wide nodes: each internal child (odd depth) is
// replaced by its own two children.  Wide nodes keep the binary node's index (+ offset), so
// no compaction pass is needed; odd-depth slots of the array stay unused.
//
// slots4 != null: the children were chosen by k_choose_children (wave_of[i] >= 0 marks the wide nodes) instead.
// node_level[node_offset + i]: the wide level of slot i (+ level_base), -1 for a slot that holds no node; the
// refit (k_refit_wide) visits the levels deepest first.
__global__ void k_pack_wide(int n, const int* __restrict__ vals, const int* __restrict__ codes,
                            const float* __restrict__ plo, const float* __restrict__ phi,
                            const int* __restrict__ left, const int* __restrict__ right,
                            const float* __restrict__ ilo, const float* __restrict__ ihi,
                            const int* __restrict__ depth, const int* __restrict__ gbounds,
                            BvhNode* __restrict__ nodes, int node_offset, const int* __restrict__ wave_of,
                            const int4* __restrict__ slots4, int* __restrict__ node_level, int level_base) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int level = slots4 ? wave_of[i] : ((depth[i] & 1) ? -1 : depth[i] >> 1);
    node_level[node_offset + i] = level < 0 ? -1 : level + level_base;
    if (level < 0) return;
    const float pad = box_pad(ord2f(gbounds[6]));
    int slots[4];
    int ns = 0;
    int ch[2] = {left[i], right[i]};
    if (!slots4) {
        for (int k = 0; k < 2; k++) {
            if (ch[k] < 0) slots[ns++] = ch[k];
            else { slots[ns++] = left[ch[k]]; slots[ns++] = right[ch[k]]; }
        }
    } else {
        const int4 c4 = slots4[i];
        const int c[4] = {c4.x, c4.y, c4.z, c4.w};
        for (int k = 0; k < 4; k++)
            if (c[k] != BVH_DONE) slots[ns++] = c[k];
    }
    float lo[3][4], hi[3][4];
    int ref[4];
    // empty slots get inverted boxes, which the sign-ordered slab test never hits (rt_device.cuh)
    for (int k = 0; k < 4; k++) {
        if (k >= ns) {
            for (int a = 0; a < 3; a++) { lo[a][k] = BVH_EMPTY_LO; hi[a][k] = BVH_EMPTY_HI; }
            ref[k] = BVH_DONE;
            continue;
        }
        const float *bl, *bh;
        if (slots[k] < 0) {
            int p = vals[~slots[k]];
            bl = plo + 3 * (size_t)p; bh = phi + 3 * (size_t)p;
            ref[k] = ~codes[p];
        } else {
            bl = ilo + 3 * (size_t)slots[k]; bh = ihi + 3 * (size_t)slots[k];
            ref[k] = slots[k] + node_offset;
        }
        for (int a = 0; a < 3; a++) {
            lo[a][k] = pad_lo(bl[a], pad);
            hi[a][k] = pad_hi(bh[a], pad);
        }
    }
    BvhNode nd;
    nd.lox = make_float4(lo[0][0], lo[0][1], lo[0][2], lo[0][3]);
    nd.loy = make_float4(lo[1][0], lo[1][1], lo[1][2], lo[1][3]);
    nd.loz = make_float4(lo[2][0], lo[2][1], lo[2][2], lo[2][3]);
    nd.hix = make_float4(hi[0][0], hi[0][1], hi[0][2], hi[0][3]);
    nd.hiy = make_float4(hi[1][0], hi[1][1], hi[1][2], hi[1][3]);
    nd.hiz = make_float4(hi[2][0], hi[2][1], hi[2][2], hi[2][3]);
    nd.ref = make_int4(ref[0], ref[1], ref[2], ref[3]);
    nd.pad_ = make_int4(0, 0, 0, 0);
    nodes[node_offset + i] = nd;
}

// Refit of the wide nodes of one level (node_level[i] == level), launched for the levels deepest first: every slot
// gets a new box and keeps its reference.  A leaf slot takes its primitive's bounds; an internal slot takes the
// unpadded union of its child's four slots (ubox, 6 floats per node, written by the launch of the level below),
// which covers the same leaves as the build's binary box of that child and therefore equals it bit for bit.
__global__ void k_refit_wide(DScene S, int count, int level, const int* __restrict__ node_level,
                             const int* __restrict__ gbounds, BvhNode* __restrict__ nodes, float* __restrict__ ubox) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count || node_level[i] != level) return;
    const float pad = box_pad(ord2f(gbounds[6]));
    const int4 r4 = nodes[i].ref;
    const int ref[4] = {r4.x, r4.y, r4.z, r4.w};
    float lo[3][4], hi[3][4], u[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int k = 0; k < 4; k++) {
        if (ref[k] == BVH_DONE) {
            for (int a = 0; a < 3; a++) { lo[a][k] = BVH_EMPTY_LO; hi[a][k] = BVH_EMPTY_HI; }
            continue;
        }
        float bl[3], bh[3];
        if (ref[k] < 0) {
            prim_bounds(S, ~ref[k], bl, bh);
        } else {
            for (int a = 0; a < 3; a++) { bl[a] = ubox[6 * (size_t)ref[k] + a]; bh[a] = ubox[6 * (size_t)ref[k] + 3 + a]; }
        }
        for (int a = 0; a < 3; a++) {
            u[a] = fminf(u[a], bl[a]);
            u[3 + a] = fmaxf(u[3 + a], bh[a]);
            lo[a][k] = pad_lo(bl[a], pad);
            hi[a][k] = pad_hi(bh[a], pad);
        }
    }
    for (int a = 0; a < 6; a++) ubox[6 * (size_t)i + a] = u[a];
    BvhNode nd;
    nd.lox = make_float4(lo[0][0], lo[0][1], lo[0][2], lo[0][3]);
    nd.loy = make_float4(lo[1][0], lo[1][1], lo[1][2], lo[1][3]);
    nd.loz = make_float4(lo[2][0], lo[2][1], lo[2][2], lo[2][3]);
    nd.hix = make_float4(hi[0][0], hi[0][1], hi[0][2], hi[0][3]);
    nd.hiy = make_float4(hi[1][0], hi[1][1], hi[1][2], hi[1][3]);
    nd.hiz = make_float4(hi[2][0], hi[2][1], hi[2][2], hi[2][3]);
    nd.ref = r4;
    nd.pad_ = make_int4(0, 0, 0, 0);
    nodes[i] = nd;
}

#define TAKE(var, type, count)                                                         \
    do {                                                                               \
        var = arena.take<type>((size_t)(count));                                       \
        if (!var) {                                                                    \
            snprintf(err, errlen, "LBVH scratch arena exhausted at %s", #var);         \
            goto fail;                                                                 \
        }                                                                              \
    } while (0)

#define CK(x)                                                                          \
    do {                                                                               \
        cudaError_t e_ = (x);                                                          \
        if (e_ != cudaSuccess) {                                                       \
            snprintf(err, errlen, "%s failed: %s", #x, cudaGetErrorString(e_));        \
            goto fail;                                                                 \
        }                                                                              \
    } while (0)

// One LBVH per primitive GROUP (e.g. spheres/`tri`s vs mesh faces), joined under a short
// chain of super nodes: floating spheres mixed into a height-field's Morton order would
// otherwise stretch the leaf-level boxes of the mesh over the whole air space.
int build_lbvh(const DScene& S, const int* d_codes, const int* group_first_code, int n, const int* group_sizes, int ngroups,
               float extra_abs, cudaStream_t stream, DeviceArena& arena, BvhNode* nodes, size_t* out_count,
               int* launches, char* err, int errlen, float* centroid_bounds, float* out_pad_scale, int* node_level,
               int* out_levels) {
    *out_count = 0;
    *out_levels = 0;
    float *plo = nullptr, *phi = nullptr, *ilo = nullptr, *ihi = nullptr;
    int *gb = nullptr, *vals0 = nullptr, *vals1 = nullptr, *hist = nullptr;
    int4* slots4 = nullptr;
    int *left = nullptr, *right = nullptr, *pint = nullptr, *pleaf = nullptr, *flags = nullptr, *depth = nullptr;
    uint32_t *keys0 = nullptr, *keys1 = nullptr;
    const int T = 256;
    const int nblk = (n + T - 1) / T;
    float4* dcost = nullptr;
    int *choice = nullptr, *wdepth = nullptr;
    int hb[7];
    float pad_scale = 0.f;
    struct Group { int start, n, root_ref, first_code; float box[6]; };
    Group groups[4];
    int K = 0, levels = 0;
    size_t total_nodes = 0;
    {
        if (n < 2 || ngroups > 4) return RT_OK;    // nothing to build (caller tests a single primitive directly)
        int acc = 0;
        for (int g = 0; g < ngroups; g++) {
            if (group_sizes[g] > 0) { groups[K].start = acc; groups[K].n = group_sizes[g]; groups[K].first_code = group_first_code[g]; K++; }
            acc += group_sizes[g];
        }
        const int nsuper = K > 1 ? 1 : 0;      // one 4-wide super node joins up to four trees
        total_nodes = (size_t)nsuper;
        for (int g = 0; g < K; g++) total_nodes += (size_t)(groups[g].n > 1 ? groups[g].n - 1 : 0);
        if (total_nodes > ((size_t)1 << 25)) {      // descend() addresses nodes with a 32-bit byte offset
            snprintf(err, errlen, "%zu LBVH nodes exceed the limit of 2^25 (4 GB node array)", total_nodes);
            return RT_ERR_LIMIT;
        }
        TAKE(plo, float, 3 * (size_t)n);
        TAKE(phi, float, 3 * (size_t)n);
        TAKE(gb, int, 16);
        int init[9] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000,
                       (int)0x80000000, 0, 0};
        CK(cudaMemcpyAsync(gb, init, sizeof(init), cudaMemcpyHostToDevice, stream));
        k_prim_bounds<<<nblk, T, 0, stream>>>(S, d_codes, n, plo, phi, gb);
        (*launches)++;
        CK(cudaMemcpyAsync(hb, gb, sizeof(hb), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        {   // fold the camera eye into the padding scale (positive float: ordered int == bits)
            float m = ord2f(hb[6]);
            if (extra_abs > m) m = extra_abs;
            pad_scale = m;
            int enc;
            memcpy(&enc, &m, 4);
            CK(cudaMemcpyAsync(gb + 6, &enc, sizeof(int), cudaMemcpyHostToDevice, stream));
        }
        TAKE(keys0, uint32_t, (size_t)n);
        TAKE(keys1, uint32_t, (size_t)n);
        TAKE(vals0, int, (size_t)n);
        TAKE(vals1, int, (size_t)n);
        TAKE(hist, int, 256 * (SORT_MAX_BLOCKS + 1));
        TAKE(left, int, (size_t)n);
        TAKE(right, int, (size_t)n);
        TAKE(pint, int, (size_t)n);
        TAKE(pleaf, int, (size_t)n);
        TAKE(flags, int, (size_t)n);
        TAKE(depth, int, (size_t)n);
        TAKE(ilo, float, 3 * (size_t)n);
        TAKE(ihi, float, 3 * (size_t)n);
        TAKE(slots4, int4, (size_t)n);
        TAKE(dcost, float4, (size_t)n);
        TAKE(choice, int, (size_t)n);
        TAKE(wdepth, int, (size_t)n);
        k_morton<<<nblk, T, 0, stream>>>(plo, phi, n, gb, keys0, vals0);
        (*launches)++;
        if (nsuper) CK(cudaMemsetAsync(node_level, 0, sizeof(int), stream));     // the super node: the last level refit
        size_t node_cursor = (size_t)nsuper;
        for (int g = 0; g < K; g++) {
            const int gs = groups[g].start, gn = groups[g].n;
            if (gn == 1) {
                groups[g].root_ref = ~groups[g].first_code;
                CK(cudaMemcpyAsync(groups[g].box, plo + 3 * (size_t)gs, 12, cudaMemcpyDeviceToHost, stream));
                CK(cudaMemcpyAsync(groups[g].box + 3, phi + 3 * (size_t)gs, 12, cudaMemcpyDeviceToHost, stream));
                continue;
            }
            const int gblk = (gn + T - 1) / T;
            // radix sort of this group's (key, prim index) pairs: 4 passes x 8 bits
            uint32_t *kin = keys0 + gs, *kout = keys1 + gs;
            int *vin = vals0 + gs, *vout = vals1 + gs;
            sort_pairs(stream, kin, kout, vin, vout, hist, gn, nullptr, launches);
            // kin/vin now point at the sorted data
            float *gilo = ilo + 3 * (size_t)gs, *gihi = ihi + 3 * (size_t)gs;
            int *gleft = left + gs, *gright = right + gs, *gpint = pint + gs, *gpleaf = pleaf + gs, *gflags = flags + gs;
            const size_t flag_bytes = sizeof(int) * (size_t)gn;
            // The optimised build (treelets + least-cost collapse) can be deeper than the traversal stack allows where
            // the Karras tree is not; then the group is built again as a plain Karras tree with the even-depth
            // collapse, whose wide depth is half the binary depth.
            for (int optimised = 1; optimised >= 0; optimised--) {
                k_karras<<<gblk, T, 0, stream>>>(kin, gn, gleft, gright, gpint, gpleaf);
                CK(cudaMemsetAsync(gflags, 0, flag_bytes, stream));
                k_refit<<<gblk, T, 0, stream>>>(gn, vin, plo, phi, gleft, gright, gpint, gpleaf, gilo, gihi, gflags);
                (*launches) += 2;
                if (optimised)
                    for (int r = 0; r < TREELET_ROUNDS; r++) {
                        CK(cudaMemsetAsync(gflags, 0, flag_bytes, stream));
                        k_treelet<<<(gn + TREELET_THREADS - 1) / TREELET_THREADS, TREELET_THREADS,
                                    sizeof(float) * (TREELET_THREADS << TREELET_LEAVES), stream>>>(gn, vin, plo, phi, gleft, gright, gpint, gpleaf, gilo, gihi, gflags);
                        (*launches)++;
                    }
                // The traversal defers at most 3 siblings per wide level; the stack (RT_SH_STACK shared + RT_STACK
                // local entries) must hold them all on every root-to-leaf path (+ the super node), or the build
                // fails instead of silently dropping subtrees.
                const int stack_entries = RT_STACK + RT_SH_STACK;
                int* wave_of = gflags;
                if (optimised) {
                    CK(cudaMemsetAsync(gflags, 0, flag_bytes, stream));
                    k_collapse_cost<<<gblk, T, 0, stream>>>(gn, gleft, gright, gpint, gpleaf, gilo, gihi, dcost + gs,
                                                            choice + gs, wdepth + gs, gflags);
                    (*launches)++;
                    int wide_depth = 0;
                    CK(cudaMemcpyAsync(&wide_depth, wdepth + gs, sizeof(int), cudaMemcpyDeviceToHost, stream));
                    CK(cudaStreamSynchronize(stream));
                    wide_depth &= 255;                  // D(root, 1): the group's root is a wide node
                    if (3 * (wide_depth + nsuper) > stack_entries) continue;
                    // one light launch per level of the wide tree
                    CK(cudaMemsetAsync(wave_of, 0xff, flag_bytes, stream));
                    CK(cudaMemsetAsync(wave_of, 0, sizeof(int), stream));                      // the group's root: wave 0
                    for (int w = 0; w < wide_depth; w++) {
                        k_choose_children<<<gblk, T, 0, stream>>>(gn, w, wave_of, slots4 + gs, gleft, gright, choice + gs);
                        (*launches)++;
                    }
                    k_pack_wide<<<gblk, T, 0, stream>>>(gn, vin, d_codes, plo, phi, gleft, gright, gilo, gihi, nullptr, gb,
                                                        nodes, (int)node_cursor, wave_of, slots4 + gs, node_level, nsuper);
                    (*launches)++;
                    levels = std::max(levels, nsuper + wide_depth);
                    break;
                }
                CK(cudaMemsetAsync(gb + 7, 0, sizeof(int), stream));
                k_depth<<<gblk, T, 0, stream>>>(gn, gpint, depth + gs, gb + 7);
                (*launches)++;
                int gdepth = 0;
                CK(cudaMemcpyAsync(&gdepth, gb + 7, sizeof(int), cudaMemcpyDeviceToHost, stream));
                CK(cudaStreamSynchronize(stream));
                const int wide_levels = gdepth / 2 + 1 + nsuper;
                if (3 * wide_levels > stack_entries) {
                    snprintf(err, errlen, "LBVH is %d binary levels deep: %d deferred entries exceed the traversal stack of %d",
                             gdepth + 1, 3 * wide_levels, stack_entries);
                    return RT_ERR_LIMIT;
                }
                k_pack_wide<<<gblk, T, 0, stream>>>(gn, vin, d_codes, plo, phi, gleft, gright, gilo, gihi, depth + gs, gb,
                                                    nodes, (int)node_cursor, nullptr, nullptr, node_level, nsuper);
                (*launches)++;
                levels = std::max(levels, nsuper + gdepth / 2 + 1);
            }
            groups[g].root_ref = (int)node_cursor;
            CK(cudaMemcpyAsync(groups[g].box, ilo + 3 * (size_t)gs, 12, cudaMemcpyDeviceToHost, stream));
            CK(cudaMemcpyAsync(groups[g].box + 3, ihi + 3 * (size_t)gs, 12, cudaMemcpyDeviceToHost, stream));
            node_cursor += (size_t)(gn - 1);
        }
        CK(cudaStreamSynchronize(stream));
        CK(cudaGetLastError());
        levels = std::max(levels, nsuper);
        if (nsuper > 0) {
            const float pad = box_pad(pad_scale);
            float lo[3][4], hi[3][4];
            int ref[4];
            for (int k = 0; k < 4; k++) {
                for (int a = 0; a < 3; a++) { lo[a][k] = BVH_EMPTY_LO; hi[a][k] = BVH_EMPTY_HI; }
                ref[k] = BVH_DONE;
                if (k >= K) continue;
                ref[k] = groups[k].root_ref;
                for (int a = 0; a < 3; a++) {
                    lo[a][k] = pad_lo(groups[k].box[a], pad);
                    hi[a][k] = pad_hi(groups[k].box[3 + a], pad);
                }
            }
            BvhNode nd;
            nd.lox = make_float4(lo[0][0], lo[0][1], lo[0][2], lo[0][3]);
            nd.loy = make_float4(lo[1][0], lo[1][1], lo[1][2], lo[1][3]);
            nd.loz = make_float4(lo[2][0], lo[2][1], lo[2][2], lo[2][3]);
            nd.hix = make_float4(hi[0][0], hi[0][1], hi[0][2], hi[0][3]);
            nd.hiy = make_float4(hi[1][0], hi[1][1], hi[1][2], hi[1][3]);
            nd.hiz = make_float4(hi[2][0], hi[2][1], hi[2][2], hi[2][3]);
            nd.ref = make_int4(ref[0], ref[1], ref[2], ref[3]);
            nd.pad_ = make_int4(0, 0, 0, 0);
            CK(cudaMemcpy(nodes, &nd, sizeof(BvhNode), cudaMemcpyHostToDevice));
        }
    }
    *out_count = total_nodes;
    *out_levels = levels;
    if (out_pad_scale) *out_pad_scale = pad_scale;
    if (centroid_bounds)
        for (int a = 0; a < 6; a++) centroid_bounds[a] = ord2f(hb[a]);
    return RT_OK;
fail:
    return RT_ERR_CUDA;
}

int refit_lbvh(const DScene& S, const int* d_codes, int n, const int* node_level, int levels, size_t node_count,
               float extra_abs, cudaStream_t stream, DeviceArena& arena, BvhNode* nodes, int* launches, char* err,
               int errlen, float* centroid_bounds, float* out_pad_scale) {
    float *plo = nullptr, *phi = nullptr, *ubox = nullptr;
    int* gb = nullptr;
    const int T = 256;
    int hb[7];
    float m = 0.f;
    {
        TAKE(plo, float, 3 * (size_t)n);
        TAKE(phi, float, 3 * (size_t)n);
        TAKE(gb, int, 16);
        TAKE(ubox, float, 6 * node_count);
        const int init[7] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000,
                             (int)0x80000000};
        CK(cudaMemcpyAsync(gb, init, sizeof(init), cudaMemcpyHostToDevice, stream));
        k_prim_bounds<<<(n + T - 1) / T, T, 0, stream>>>(S, d_codes, n, plo, phi, gb);
        (*launches)++;
        CK(cudaMemcpyAsync(hb, gb, sizeof(hb), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        // M as build_lbvh derives it: the primitives' largest |coordinate| folded with extra_abs
        m = ord2f(hb[6]);
        if (extra_abs > m) m = extra_abs;
        int enc;
        memcpy(&enc, &m, 4);
        CK(cudaMemcpyAsync(gb + 6, &enc, sizeof(int), cudaMemcpyHostToDevice, stream));
        const unsigned blk = (unsigned)((node_count + T - 1) / T);
        for (int l = levels - 1; l >= 0; l--) {
            k_refit_wide<<<blk, T, 0, stream>>>(S, (int)node_count, l, node_level, gb, nodes, ubox);
            (*launches)++;
        }
        CK(cudaGetLastError());
    }
    *out_pad_scale = m;
    for (int a = 0; a < 6; a++) centroid_bounds[a] = ord2f(hb[a]);
    return RT_OK;
fail:
    return RT_ERR_CUDA;
}

}  // namespace rt
