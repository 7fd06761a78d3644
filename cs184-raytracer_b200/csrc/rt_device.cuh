// rt_device.cuh — device-side data layout and the exact FP64 arithmetic of the trace loop.
//
// Everything that DECIDES a hit (object-space transforms, sphere quadratic, Cramer's rule,
// shading-normal cull, closest-distance compare) is evaluated in FP64 with exactly the
// association order of the reference build (g++ -O2, SSE2 Eigen 3.2.2, no FMA), so hit
// ids and ray counts match the reference bit for bit; this translation unit MUST be
// compiled with -fmad=false.  Only the LBVH boxes (culling, conservative) are FP32.
//
// Reference map:
//   xf_point/xf_dir      Transform4d * Vector4d           eigen/.../Transform.h:1244-1267
//   dot4/norm4           Vector4d dot / norm (SSE2 redux)  eigen/.../Redux.h:131-136,299-305
//   det3                 Matrix3d::determinant            eigen/.../LU/Determinant.h:18-23,61-69
//   sphere_object        Sphere::calculateIntNormInObjSpace  src/geometry.cpp:47-67
//   face_object          Mesh::calculateIntNormInObjSpace    src/geometry.cpp:78-123 (loop body)
//   mesh_bbox            hitsBoundingBox                     src/geometry.cpp:5-29
//   to_world             Geometry::calculateIntersectionNormal src/geometry.cpp:39-43
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "rt_b200.h"

namespace rt {

struct d3 {
    double x, y, z;
};

__device__ __forceinline__ d3 mk3(double x, double y, double z) { d3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ d3 operator+(d3 a, d3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ d3 operator-(d3 a, d3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ d3 operator-(d3 a) { return mk3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ d3 operator*(double s, d3 a) { return mk3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ d3 vdiv(d3 a, double s) { return mk3(a.x / s, a.y / s, a.z / s); }

// two 2-wide packets added lane-wise, then horizontally: (x0+x2)+(x1+x3); w product is +0
__device__ __forceinline__ double sum4(double a, double b, double c, double d) { return (a + c) + (b + d); }
__device__ __forceinline__ double dot4(d3 a, d3 b) { return sum4(a.x * b.x, a.y * b.y, a.z * b.z, 0.0); }
__device__ __forceinline__ double norm4(d3 a) { return sqrt(dot4(a, a)); }
// Ray constructor: direction / direction.norm()  (true division; src/rtbase.h:23)
__device__ __forceinline__ d3 ray_normalize(d3 a) { return vdiv(a, norm4(a)); }
// Vector4d::normalize(): multiply by the reciprocal (Eigen 3.2 operator/=)
__device__ __forceinline__ d3 inplace_normalize(d3 a) { return (1.0 / norm4(a)) * a; }

// rows 0..2 of a row-major 3x4 affine matrix
__device__ __forceinline__ d3 xf_point(const double* __restrict__ m, d3 v) {
    return mk3(((m[0] * v.x + m[1] * v.y) + m[2] * v.z) + m[3] * 1.0,
               ((m[4] * v.x + m[5] * v.y) + m[6] * v.z) + m[7] * 1.0,
               ((m[8] * v.x + m[9] * v.y) + m[10] * v.z) + m[11] * 1.0);
}
__device__ __forceinline__ d3 xf_dir(const double* __restrict__ m, d3 v) {
    return mk3(((m[0] * v.x + m[1] * v.y) + m[2] * v.z) + m[3] * 0.0,
               ((m[4] * v.x + m[5] * v.y) + m[6] * v.z) + m[7] * 0.0,
               ((m[8] * v.x + m[9] * v.y) + m[10] * v.z) + m[11] * 0.0);
}
// inverse.matrix().transpose() * N, w := 0
__device__ __forceinline__ d3 xf_normal(const double* __restrict__ inv, d3 n) {
    return mk3(sum4(inv[0] * n.x, inv[4] * n.y, inv[8] * n.z, 0.0),
               sum4(inv[1] * n.x, inv[5] * n.y, inv[9] * n.z, 0.0),
               sum4(inv[2] * n.x, inv[6] * n.y, inv[10] * n.z, 0.0));
}

__device__ __forceinline__ double det3(d3 c0, d3 c1, d3 c2) {
    double h012 = c0.x * (c1.y * c2.z - c2.y * c1.z);
    double h102 = c1.x * (c0.y * c2.z - c2.y * c0.z);
    double h201 = c2.x * (c0.y * c1.z - c1.y * c0.z);
    return h012 - h102 + h201;
}

// ---- device scene ------------------------------------------------------------
struct alignas(16) DGeom {
    double inv[12];
    double fwd[12];
    double det;
    double center[3];
    double radius2;
    double bbmin[3];
    double bbmax[3];
    int type;
    int mat;
    int first_face;
    int num_faces;
    int use_bbox;
    int pad_[3];
};

struct alignas(16) DMat {
    double ka[3], kd[3], ks[3], kr[3];
    double sp, ior;
    int has_kt;        // translucencyColor_ != 0  (src/scene.cpp:115)
    int has_kr;        // reflectiveColor_ != 0    (src/scene.cpp:130)
    int pad_[2];
};

struct alignas(16) DLight {
    double v[3];
    double color[3];
    double falloff;
    int type;
    int pad_;
};

struct DCamera {
    double eye[3], ll[3], lr[3], ul[3], ur[3];
};

// One face = 5 x double2 = 80 B: p0.xy | p0.z va.x | va.yz | vb.xy | vb.z aux
// where va = p1 - p0, vb = p2 - p0 (the subtractions src/geometry.cpp:80-81 does per ray)
// and aux packs (geometry index, face index within the geometry) as two int32.
// Normals: n0.xy | n0.z n1.x | n1.yz | n2.xy | n2.z pad.
#define RT_FACE_D2 5

// 4-wide LBVH node, 128 B = 8 x float4 (128-byte aligned): the four child boxes as SoA (FP32,
// padded outward) + four child references.  ref >= 0: wide-node index; ref < 0: leaf, prim
// code = ~ref; empty slot: ref = BVH_DONE with an INVERTED box (lo = +1e30, hi = -1e30), which
// the sign-ordered slab test below can never hit.  A wide node is a binary Karras node at even
// depth with its grandchildren pulled up, which halves the number of dependent fetches per ray.
// The lower planes sit in the first 64 bytes and the upper planes in the second, 64 bytes
// apart: a ray fetches its NEAR plane of an axis from one half and the FAR plane from the same
// offset in the other half (address ^ 64), chosen once per ray from the sign of its direction.
struct alignas(128) BvhNode {
    float4 lox, loy, loz;
    int4 ref;
    float4 hix, hiy, hiz;
    int4 pad_;
};
#define BVH_EMPTY_LO 1e30f
#define BVH_EMPTY_HI (-1e30f)
#define BVH_DONE ((int)0x80000000)     // not a valid ref (prim codes stay below 3<<29)

// prim code: kind in the top 2 bits of a 31-bit value
#define PRIM_KIND_SHIFT 29
#define PRIM_FACE 0      // index = global face index (mesh face)
#define PRIM_SPHERE 1    // index = geometry index
#define PRIM_TRI 2       // index = geometry index (tests faces first_face, first_face+1)
#define PRIM_INDEX_MASK ((1 << PRIM_KIND_SHIFT) - 1)

struct DScene {
    DCamera cam;
    const DGeom* geoms;
    const DMat* mats;
    const DLight* slights;     // non-ambient lights, insertion order (each casts a shadow ray)
    const DLight* alights;     // ambient lights, insertion order
    const double2* face_pts;
    const double2* face_nrm;
    const BvhNode* nodes;      // null when fewer than two primitives are in the BVH
    const int* flat;           // prim codes tested by every ray, in geometry order
    const int* all_prims;      // every prim code in geometry/face order (brute force)
    const float4* sph_bound;   // per geometry: world-space bounding sphere (xyz, radius) of a SPHERE, FP32
    int num_geoms;
    int num_slights;
    int num_alights;
    int num_flat;
    int num_all;
    int num_bvh_prims;
    int single_leaf;           // BVH with exactly one primitive: its prim code
    // Largest |coordinate| the LBVH box padding was derived for (every primitive's world bounds,
    // flat ones included, and the camera eye): the FP32 slab test is conservative for ray origins
    // inside it.  A ray starting further out (only possible through rt_cast_rays) takes the
    // brute-force path instead.
    float origin_limit;
};

// ---- hit bookkeeping ------------------------------------------------------------
struct Best {
    int geom;        // -1: none
    int face;
    double dobj;     // object-space distance t*|d'| (mesh) — compared within a geometry
    double wd;       // world distance |P - o| (src/scene.cpp:153) — compared across geometries
    d3 P, N;         // world-space point, un-normalised world normal (after det flip)
};

// object-space ray of the geometry currently being tested (cached across BVH leaves)
struct ObjRay {
    int geom;        // -1: nothing cached
    int box_ok;      // hitsBoundingBox verdict for MESH geometries with use_bbox
    d3 o, d, nd;     // origin, unit direction, -direction
    double dn;       // Vector3d norm of d: sqrt(dx^2 + (dy^2 + dz^2))
};

struct WorkCounters {
    unsigned long long nodes, tris, spheres;
};

// hitsBoundingBox (src/geometry.cpp:5-29): true when ANY of the six planes is crossed at t >= 0 inside the other two
// coordinate ranges.  The reference tries the planes in a fixed order and returns at the first that passes; the
// verdict is the OR over the planes, so the order is free.  A ray that starts inside the box (every shadow and
// bounce ray of a mesh scene) passes at its EXIT plane, which an FP32 estimate picks first: one exact FP64 plane
// test (the reference's own expressions) instead of 3.5 on average.  Only if that plane fails are all six
// evaluated in the reference's order.
__device__ __forceinline__ bool bbox_plane(const double* oo, const double* dd, int axis, int bn, const double* __restrict__ bbmin,
                                           const double* __restrict__ bbmax) {
    const double mag = dd[axis];
    if (mag == 0.0) return false;
    const double t = ((bn ? bbmax[axis] : bbmin[axis]) - oo[axis]) / mag;
    if (t < 0) return false;
    bool ok = true;
#pragma unroll
    for (int a2 = 0; a2 < 3; a2++) {
        if (a2 == axis) continue;
        const double ip = oo[a2] + t * dd[a2];
        if (ip < bbmin[a2] || ip > bbmax[a2]) ok = false;
    }
    return ok;
}
__device__ __forceinline__ bool mesh_bbox(d3 o, d3 d, const double* __restrict__ bbmin,
                                          const double* __restrict__ bbmax) {
    const double oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
    {   // likely exit plane: per axis the plane ahead of the ray, the nearest of the three (FP32 estimate)
        float best = 3.0e38f;
        int baxis = 0, bbn = 0;
#pragma unroll
        for (int axis = 0; axis < 3; axis++) {
            const float df = (float)dd[axis];
            if (df == 0.f) continue;
            const int bn = df > 0.f ? 1 : 0;
            const float tf = ((float)(bn ? bbmax[axis] : bbmin[axis]) - (float)oo[axis]) / df;
            if (tf >= 0.f && tf < best) { best = tf; baxis = axis; bbn = bn; }
        }
        if (best < 3.0e38f) {
            bool hit;
            if (baxis == 0) hit = bbox_plane(oo, dd, 0, bbn, bbmin, bbmax);
            else if (baxis == 1) hit = bbox_plane(oo, dd, 1, bbn, bbmin, bbmax);
            else hit = bbox_plane(oo, dd, 2, bbn, bbmin, bbmax);
            if (hit) return true;
        }
    }
#pragma unroll
    for (int axis = 0; axis < 3; axis++) {
#pragma unroll
        for (int bn = 0; bn < 2; bn++)
            if (bbox_plane(oo, dd, axis, bn, bbmin, bbmax)) return true;
    }
    return false;
}

__device__ __forceinline__ void load_objray(const DScene& S, int gi, d3 o, d3 d, ObjRay& R) {
    const DGeom* g = S.geoms + gi;
    R.geom = gi;
    R.o = xf_point(g->inv, o);
    R.d = ray_normalize(xf_dir(g->inv, d));
    R.nd = -R.d;
    R.dn = sqrt(R.d.x * R.d.x + (R.d.y * R.d.y + R.d.z * R.d.z));
    R.box_ok = 1;
    if (g->type == RT_GEOM_MESH && g->use_bbox) R.box_ok = mesh_bbox(R.o, R.d, g->bbmin, g->bbmax) ? 1 : 0;
}

// Offer a candidate (geometry gi, face f) to the running closest hit.  Within one
// geometry the reference keeps the accepted face of smallest object-space distance, first
// face on ties (src/geometry.cpp:108-110); across geometries the smallest world distance,
// first geometry on ties (src/scene.cpp:153-155).
__device__ __forceinline__ bool beats(const Best& best, int gi, int f, double dobj, double wd) {
    if (best.geom < 0) return true;
    if (gi == best.geom) return dobj < best.dobj || (dobj == best.dobj && f < best.face);
    return wd < best.wd || (wd == best.wd && gi < best.geom);
}

// World-space completion of an object-space hit (src/geometry.cpp:39-43) + world distance.
__device__ __forceinline__ void to_world(const DGeom* g, d3 Pobj, d3 Nobj, d3 o, d3& P, d3& N, double& wd) {
    P = xf_point(g->fwd, Pobj);
    N = xf_normal(g->inv, Nobj);
    if (g->det < 0) N = -N;
    wd = norm4(P - o);
}

// ANYHIT = true: shadow query — report as soon as an accepted hit has wd <= limit.
template <bool ANYHIT>
__device__ __forceinline__ bool test_sphere(const DScene& S, int gi, d3 o, d3 d, bool reverse, double limit,
                                            Best& best) {
    const DGeom* g = S.geoms + gi;
    d3 oo = xf_point(g->inv, o);
    d3 dd = ray_normalize(xf_dir(g->inv, d));
    d3 c = mk3(g->center[0], g->center[1], g->center[2]);
    d3 ocd = oo - c;
    double a = dot4(dd, dd);
    double b = 2 * dot4(dd, ocd);
    double cc = dot4(ocd, ocd) - g->radius2;
    double disc = b * b - 4 * a * cc;
    if (disc < 0) return false;
    double res = reverse ? (-b + sqrt(disc)) / (2 * a) : (-b - sqrt(disc)) / (2 * a);
    if (res < 0) return false;
    d3 Pobj = oo + res * dd;
    d3 Nobj = Pobj - c;
    d3 P, N;
    double wd;
    to_world(g, Pobj, Nobj, o, P, N, wd);
    if (ANYHIT) return wd <= limit;
    if (beats(best, gi, 0, 0.0, wd)) {
        best.geom = gi; best.face = 0; best.dobj = 0.0; best.wd = wd; best.P = P; best.N = N;
    }
    return false;
}

// One face of a TRI/MESH geometry; R must hold the object-space ray of geometry gi.
template <bool ANYHIT>
__device__ __forceinline__ bool test_face(const DScene& S, int gi, int gface, int lface, const ObjRay& R, d3 o,
                                          bool reverse, double limit, Best& best) {
    const double2* __restrict__ fp = S.face_pts + (size_t)gface * RT_FACE_D2;
    double2 q0 = __ldg(fp + 0), q1 = __ldg(fp + 1), q2 = __ldg(fp + 2), q3 = __ldg(fp + 3), q4 = __ldg(fp + 4);
    d3 p0 = mk3(q0.x, q0.y, q1.x), va = mk3(q1.y, q2.x, q2.y), vb = mk3(q3.x, q3.y, q4.x);
    d3 rhs = R.o - p0;
    double dlower = det3(va, vb, R.nd);
    if (dlower == 0) return false;
    double a = det3(rhs, vb, R.nd) / dlower;
    if (a < 0 || a > 1) return false;
    double b = det3(va, rhs, R.nd) / dlower;
    if (b < 0 || a + b > 1) return false;
    double t = det3(va, vb, rhs) / dlower;
    if (t < 0) return false;
    double dobj = t * R.dn;
    if (!ANYHIT && best.geom == gi && (dobj > best.dobj || (dobj == best.dobj && lface > best.face))) return false;
    const double2* __restrict__ fn = S.face_nrm + (size_t)gface * RT_FACE_D2;
    double2 m0 = __ldg(fn + 0), m1 = __ldg(fn + 1), m2 = __ldg(fn + 2), m3 = __ldg(fn + 3), m4 = __ldg(fn + 4);
    d3 n0 = mk3(m0.x, m0.y, m1.x), n1 = mk3(m1.y, m2.x, m2.y), n2 = mk3(m3.x, m3.y, m4.x);
    double w0 = 1.0 - a - b;
    d3 tn = (w0 * n0 + a * n1) + b * n2;
    bool front = dot4(tn, R.d) < 0;
    if ((!front) != reverse) return false;      // (!hitsFront) ^ reverseNormals -> skip
    d3 Pobj = p0 + (a * va + b * vb);
    d3 P, N;
    double wd;
    to_world(S.geoms + gi, Pobj, tn, o, P, N, wd);
    if (ANYHIT) return wd <= limit;
    if (beats(best, gi, lface, dobj, wd)) {
        best.geom = gi; best.face = lface; best.dobj = dobj; best.wd = wd; best.P = P; best.N = N;
    }
    return false;
}

// FP32 pre-test against the sphere's world-space BOUNDING sphere.  It may only say "missed"
// when the exact test would.  Skips about half of the exact tests (a sphere fills 52 % of its
// box' projected area).  Error bound, with d a unit vector:
//  * bs.xyz is the centre rounded to nearest FP32; bs.w >= the ellipsoid's largest semi-axis
//    plus |c - bs.xyz|, rounded up (rt_api.cu), so the ball (bs.xyz, bs.w) holds the ellipsoid.
//  * (float)o is within 2^-24 |o_i| of o per axis, i.e. within sqrt(3) 2^-24 |o|inf < 2^-23 |o|inf
//    in distance.  A ray from (float)o parallel to the true ray passes within that distance of
//    every point of the true ray, so growing the radius by 2^-23 |o|inf covers it.  Both terms
//    are absolute: they grow with the coordinates, not with the sphere or |c - o|.
//  * What is left is the rounding of the FP32 expressions below and of d: a few 2^-24
//    relative to |c - o|^2 and to r.  The margins are far larger (1e-4 on |c - o|^2 and 1e-3
//    on the radius).
// The test is conservative at any |coordinate| where |c - o|^2 stays finite in FP32 (below
// ~1e19); past that c2 is inf and the comparisons are false, so nothing is culled.
__device__ __forceinline__ bool sphere_certainly_missed(float4 bs, d3 o, d3 d) {
    const float ox = (float)o.x, oy = (float)o.y, oz = (float)o.z;
    float ocx = bs.x - ox, ocy = bs.y - oy, ocz = bs.z - oz;
    float dx = (float)d.x, dy = (float)d.y, dz = (float)d.z;
    float c2 = ocx * ocx + ocy * ocy + ocz * ocz;
    float b = ocx * dx + ocy * dy + ocz * dz;
    float r = (bs.w + 0x1p-23f * fmaxf(fabsf(ox), fmaxf(fabsf(oy), fabsf(oz)))) * 1.001f;
    float r2 = r * r + 1e-4f * c2 + 1e-30f;
    if (c2 - b * b > r2) return true;                       // the line passes outside the sphere
    return c2 > r2 && b < -(r + 1e-3f * sqrtf(c2));        // origin outside and the sphere entirely behind it
}

// Dispatch one prim code.  Returns true only for ANYHIT occlusion.
template <bool ANYHIT, bool COUNT>
__device__ __forceinline__ bool test_prim(const DScene& S, int code, d3 o, d3 d, bool reverse, double limit,
                                          ObjRay& R, Best& best, WorkCounters& wc) {
    const int kind = code >> PRIM_KIND_SHIFT, idx = code & PRIM_INDEX_MASK;
    if (kind == PRIM_SPHERE) {
        if (sphere_certainly_missed(__ldg(S.sph_bound + idx), o, d)) return false;
        if (COUNT) wc.spheres++;
        return test_sphere<ANYHIT>(S, idx, o, d, reverse, limit, best);
    }
    if (kind == PRIM_TRI) {
        const DGeom* g = S.geoms + idx;
        if (R.geom != idx) load_objray(S, idx, o, d, R);
        if (COUNT) wc.tris += 2;
        if (test_face<ANYHIT>(S, idx, g->first_face, 0, R, o, reverse, limit, best)) return true;
        return test_face<ANYHIT>(S, idx, g->first_face + 1, 1, R, o, reverse, limit, best);
    }
    // mesh face: geometry/local face index ride in the face record's aux slot
    double2 q4 = __ldg(S.face_pts + (size_t)idx * RT_FACE_D2 + 4);
    int gi = __double2loint(q4.y), lf = __double2hiint(q4.y);
    if (R.geom != gi) load_objray(S, gi, o, d, R);
    if (!R.box_ok) return false;
    if (COUNT) wc.tris++;
    return test_face<ANYHIT>(S, gi, idx, lf, R, o, reverse, limit, best);
}

// ---- FP32 conservative slab test -------------------------------------------------
struct FRay {
    float ix, iy, iz;      // 1/d (clamped away from 0)
    float bx, by, bz;      // -o/d, so that t = plane * (1/d) + (-o/d) is one FMA
    // byte offset, inside a node, of this ray's NEAR plane per axis (lower plane when the
    // direction component is >= 0, upper plane otherwise); the far plane is at address ^ 64
    unsigned nx, ny, nz;
};
// A direction component below `tiny` is clamped to +-tiny.  tiny >= |o_axis| 2^-126 keeps
// |b| = |o| / tiny <= 2^126, finite: with a fixed 1e-30 an axis-parallel ray from |o| > 3.4e8
// got b = +-inf, both plane distances of that axis +-inf, and missed every box.  The clamp
// tilts the ray by at most tiny per unit of distance.  A hit lies within 3.5 M of the origin
// (M: the padding's scale, see slab1), so the tilt stays <= 3.5 M max(1e-30, M 2^-126), below
// the padding's 1e-6 M slack for M < 2e31.
__device__ __forceinline__ FRay make_fray(d3 o, d3 d) {
    FRay r;
    float ox = (float)o.x, oy = (float)o.y, oz = (float)o.z;
    float dx = (float)d.x, dy = (float)d.y, dz = (float)d.z;
    const float tx = fmaxf(1e-30f, fabsf(ox) * 0x1p-126f), ty = fmaxf(1e-30f, fabsf(oy) * 0x1p-126f),
                tz = fmaxf(1e-30f, fabsf(oz) * 0x1p-126f);
    if (fabsf(dx) < tx) dx = copysignf(tx, dx);
    if (fabsf(dy) < ty) dy = copysignf(ty, dy);
    if (fabsf(dz) < tz) dz = copysignf(tz, dz);
    r.ix = 1.0f / dx; r.iy = 1.0f / dy; r.iz = 1.0f / dz;
    r.bx = -ox * r.ix; r.by = -oy * r.iy; r.bz = -oz * r.iz;
    r.nx = r.ix < 0.f ? 64u : 0u;
    r.ny = r.iy < 0.f ? 80u : 16u;
    r.nz = r.iz < 0.f ? 96u : 32u;
    // opaque, or the compiler re-derives the three offsets from the direction signs per node visit
    asm volatile("" : "+r"(r.nx), "+r"(r.ny), "+r"(r.nz));
    return r;
}
// Entry distance of four (already padded) boxes.  near/far planes are picked by the sign of
// the direction, so t_near <= t_far per axis by construction (x -> fma(x, i, b) is monotone)
// and the test is  max(t_near, 0) <= min(t_far, tlimit).  The FP32 roundings in here
// (conversion of o and d, 1/d, b = -o/d, the FMA) move a plane distance by the equivalent of
// about 2e-7 x (|plane| + |o|) in position.  The box padding (rt_bvh.cu) is 2e-6 x M + 2e-7 x
// |plane| with M = the largest |coordinate| of ANY primitive of the scene (LBVH or flat list)
// and of the camera eye, i.e. of every point a render's ray can start from; cast_ray sends rays
// from further out (DScene::origin_limit, rt_cast_rays only) down the brute-force path.  tlimit
// is already rounded up with slack (prune_limit), so rounding can only let MORE boxes through,
// never fewer.  An empty slot (inverted box) has
// t_near >= +1e30 > t_far <= -1e30 on every axis: never hit.
// (Explicit __fmaf_rn: this file is compiled with -fmad=false.)
struct Slab4 {
    float tn[4];     // entry distance (clamped to >= 0)
    bool hit[4];
};
__device__ __forceinline__ void slab1(const FRay& r, float nx, float ny, float nz, float fx, float fy, float fz,
                                      float tlimit, float& tn, bool& hit) {
    const float tnx = __fmaf_rn(nx, r.ix, r.bx), tny = __fmaf_rn(ny, r.iy, r.by), tnz = __fmaf_rn(nz, r.iz, r.bz);
    const float tfx = __fmaf_rn(fx, r.ix, r.bx), tfy = __fmaf_rn(fy, r.iy, r.by), tfz = __fmaf_rn(fz, r.iz, r.bz);
    tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, 0.f));
    const float tf = fminf(fminf(tfx, tfy), fminf(tfz, tlimit));
    hit = tn <= tf;
}

#define RT_STACK 96
// Entries of the traversal stack kept in SHARED memory per thread (interleaved by thread, so
// any mix of stack depths within a warp is bank-conflict free); deeper entries overflow to
// the local-memory array.  ncu (round 1): with the whole stack in local memory, local
// loads/stores were 2/3 of all L1 requests of k_shadow and wrote 22 GB per launch through to
// L2 — the LSU data pipe (75 % busy) was the limiter, not DRAM.
#ifndef RT_SH_STACK
#define RT_SH_STACK 12
#endif
#ifndef RT_BLOCK
#define RT_BLOCK 64
#endif

__device__ __forceinline__ float prune_limit(double x) {
    // FP32 prune limit, rounded up with slack
    if (!(x < 3.0e38)) return __int_as_float(0x7f800000);
    return __double2float_ru(x) * 1.00001f + 1e-30f;
}

// ---- traversal stack ------------------------------------------------------------------
// The first RT_SH_STACK entries of a thread's stack live in shared memory, in a column
// interleaved by thread (entry e of thread t at base + (e * RT_BLOCK + t) * entry size: no
// bank conflicts whatever the mix of depths in a warp); deeper entries overflow into a
// local-memory array (rare).  Any-hit entries are a node/leaf reference (4 B); closest-hit
// entries also carry the subtree's entry distance (8 B).  The state is the shared address of
// the next free slot (`top`) and the number of overflowed entries (`lsp`, > 0 only while the
// shared column is full), both plain registers.
#define RT_SH_ENTRY(ANYHIT) ((ANYHIT) ? 4 : 8)
#define RT_SH_STRIDE(ANYHIT) (RT_BLOCK * RT_SH_ENTRY(ANYHIT))
#define RT_SH_STACK_BYTES(ANYHIT) ((RT_SH_STACK > 0 ? RT_SH_STACK : 1) * RT_SH_STRIDE(ANYHIT))

template <bool ANYHIT>
__device__ __forceinline__ unsigned stack_base(const void* smem) {
    unsigned b = (unsigned)__cvta_generic_to_shared(smem) + threadIdx.x * RT_SH_ENTRY(ANYHIT);
    asm volatile("" : "+r"(b));     // opaque: keep it in a register instead of re-deriving it from %tid per push
    return b;
}

// overflow part (local memory) — kept apart from the scalars so that those stay in registers
template <bool ANYHIT>
struct StackSpill {
    int ref[RT_STACK];
    float t[ANYHIT ? 1 : RT_STACK];
};
template <bool ANYHIT>
struct Stack {
    // `top`: shared address of the next free slot; it keeps growing (virtually) past `lim`
    // when the shared column is full, the entries beyond living in the spill arrays
    unsigned base, top;
    StackSpill<ANYHIT>& sp;
    __device__ __forceinline__ Stack(unsigned shbase, StackSpill<ANYHIT>& spill) : base(shbase), top(shbase), sp(spill) {}
    __device__ __forceinline__ unsigned lim() const { return base + RT_SH_STACK * RT_SH_STRIDE(ANYHIT); }
    __device__ __forceinline__ static void sts(unsigned a, int ref, float t) {
        if (ANYHIT) asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(ref));
        else asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(ref), "r"(__float_as_int(t)));
    }
    // room for n more entries in the shared column?
    __device__ __forceinline__ bool roomy(int n) const { return top + n * RT_SH_STRIDE(ANYHIT) <= lim(); }
    // push when the caller has checked roomy(): straight-line, predicated by `on`
    __device__ __forceinline__ void push_fast(bool on, int ref, float t) {
        if (on) sts(top, ref, t);
        top += on ? RT_SH_STRIDE(ANYHIT) : 0;
    }
    __device__ __forceinline__ void push(int ref, float t) {
        if (top < lim()) {
            sts(top, ref, t);
        } else {
            const unsigned k = (top - lim()) / RT_SH_STRIDE(ANYHIT);
            if (k >= RT_STACK) return;            // unreachable: rt_scene_upload rejects trees deeper than the stack (RT_ERR_LIMIT)
            sp.ref[k] = ref;
            if (!ANYHIT) sp.t[k] = t;
        }
        top += RT_SH_STRIDE(ANYHIT);
    }
    // Pops the next deferred subtree; closest hit: skips those a closer hit has made obsolete.
    __device__ __forceinline__ int pop(float tlim) {
        while (top != base) {
            top -= RT_SH_STRIDE(ANYHIT);
            int ref, tb = 0;
            if (top < lim()) {
                if (ANYHIT) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(ref) : "r"(top));
                else asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(ref), "=r"(tb) : "r"(top));
            } else {
                const unsigned k = (top - lim()) / RT_SH_STRIDE(ANYHIT);
                ref = sp.ref[k];
                if (!ANYHIT) tb = __float_as_int(sp.t[k]);
            }
            if (ANYHIT || __int_as_float(tb) <= tlim) return ref;
        }
        return BVH_DONE;
    }
};

__device__ __forceinline__ const float4* flip64(const float4* p) {
    return reinterpret_cast<const float4*>(reinterpret_cast<unsigned long long>(p) ^ 64ull);
}

// Walks internal nodes of the 4-wide LBVH until `cur` is a leaf reference (< 0) or BVH_DONE.
// Leaves are deferred through the same stack as internal nodes ("while-while"): this loop
// only does cheap FP32 slab tests, so the threads of a warp reconverge before the long exact
// FP64 primitive test instead of diverging into it.
template <bool ANYHIT, bool COUNT>
__device__ __forceinline__ void descend(const DScene& S, const FRay& fr, float tlim, int& cur, Stack<ANYHIT>& st,
                                        WorkCounters& wc) {
    while (cur >= 0) {
        const char* const nb = reinterpret_cast<const char*>(S.nodes);
        const unsigned off = (unsigned)cur * (unsigned)sizeof(BvhNode);       // node arrays stay below 4 GB: rt_scene_upload rejects more than 2^25 nodes
        const float4* pnx = reinterpret_cast<const float4*>(nb + (off + fr.nx));
        const float4* pny = reinterpret_cast<const float4*>(nb + (off + fr.ny));
        const float4* pnz = reinterpret_cast<const float4*>(nb + (off + fr.nz));
        const float4 nx = __ldg(pnx), ny = __ldg(pny), nz = __ldg(pnz);
        const float4 fx = __ldg(flip64(pnx)), fy = __ldg(flip64(pny)), fz = __ldg(flip64(pnz));
        const int4 ref = __ldg(reinterpret_cast<const int4*>(nb + off + 48));
        if (COUNT) wc.nodes += 4;
        float t0, t1, t2, t3;
        bool h0, h1, h2, h3;
        slab1(fr, nx.x, ny.x, nz.x, fx.x, fy.x, fz.x, tlim, t0, h0);
        slab1(fr, nx.y, ny.y, nz.y, fx.y, fy.y, fz.y, tlim, t1, h1);
        slab1(fr, nx.z, ny.z, nz.z, fx.z, fy.z, fz.z, tlim, t2, h2);
        slab1(fr, nx.w, ny.w, nz.w, fx.w, fy.w, fz.w, tlim, t3, h3);
        if (ANYHIT) {
            // occlusion query: any order will do; take the first hit slot, defer the others
            int next = h3 ? ref.w : BVH_DONE;
            if (st.roomy(3)) {
                bool q;
                q = h2 && next != BVH_DONE; st.push_fast(q, next, 0.f); next = h2 ? ref.z : next;
                q = h1 && next != BVH_DONE; st.push_fast(q, next, 0.f); next = h1 ? ref.y : next;
                q = h0 && next != BVH_DONE; st.push_fast(q, next, 0.f); next = h0 ? ref.x : next;
            } else {
                if (h2) { if (next != BVH_DONE) st.push(next, 0.f); next = ref.z; }
                if (h1) { if (next != BVH_DONE) st.push(next, 0.f); next = ref.y; }
                if (h0) { if (next != BVH_DONE) st.push(next, 0.f); next = ref.x; }
            }
            cur = next != BVH_DONE ? next : st.pop(tlim);
            continue;
        }
        // Closest hit: descend into the NEAREST hit child; the other hit children are deferred
        // with their entry distances in slot order, not sorted (pop() skips what a closer hit has
        // made obsolete whatever the order; a full 4-key sorting network cost 4 % more in k_trace).  The slot index rides in the two low mantissa bits
        // of the distance (t >= 0: float bit patterns order like unsigned ints).
        const unsigned MISS = 0x7f800000u;
        const unsigned k0 = h0 ? ((__float_as_uint(t0) & ~3u) | 0u) : MISS, k1 = h1 ? ((__float_as_uint(t1) & ~3u) | 1u) : MISS;
        const unsigned k2 = h2 ? ((__float_as_uint(t2) & ~3u) | 2u) : MISS, k3 = h3 ? ((__float_as_uint(t3) & ~3u) | 3u) : MISS;
        const unsigned kmin = min(min(k0, k1), min(k2, k3));
        if (st.roomy(3)) {
            st.push_fast(h3 && k3 != kmin, ref.w, t3);
            st.push_fast(h2 && k2 != kmin, ref.z, t2);
            st.push_fast(h1 && k1 != kmin, ref.y, t1);
            st.push_fast(h0 && k0 != kmin, ref.x, t0);
        } else {
            if (h3 && k3 != kmin) st.push(ref.w, t3);
            if (h2 && k2 != kmin) st.push(ref.z, t2);
            if (h1 && k1 != kmin) st.push(ref.y, t1);
            if (h0 && k0 != kmin) st.push(ref.x, t0);
        }
        if (kmin < MISS) {
            const unsigned i = kmin & 3u;
            cur = i == 0 ? ref.x : (i == 1 ? ref.y : (i == 2 ? ref.z : ref.w));
        } else {
            cur = st.pop(tlim);
        }
    }
}

// The closest-hit / any-hit query == Scene::castRay (src/scene.cpp:142-167).
//   ANYHIT: returns true when an accepted hit with world distance <= limit exists.
//   BRUTE : ignore the LBVH and test every primitive (debug / parity aid).
//   FARCHECK: the origin may lie outside DScene::origin_limit (caller-supplied rays only).
template <bool ANYHIT, bool BRUTE, bool COUNT, bool FARCHECK = false>
__device__ __forceinline__ bool cast_ray(const DScene& S, d3 o, d3 d, bool reverse, double limit, Best& best,
                                         WorkCounters& wc, unsigned shbase) {
    best.geom = -1; best.face = -1; best.dobj = 0.0; best.wd = 0.0;
    ObjRay R;
    R.geom = -1; R.box_ok = 1;
    // origins outside the range the box padding covers (see slab1): no culling for this ray
    const bool far_origin = FARCHECK && !BRUTE && fmax(fabs(o.x), fmax(fabs(o.y), fabs(o.z))) > (double)S.origin_limit;
    if (BRUTE || far_origin) {
        for (int i = 0; i < S.num_all; i++)
            if (test_prim<ANYHIT, COUNT>(S, __ldg(S.all_prims + i), o, d, reverse, limit, R, best, wc)) return true;
        return false;
    }
    for (int i = 0; i < S.num_flat; i++)
        if (test_prim<ANYHIT, COUNT>(S, __ldg(S.flat + i), o, d, reverse, limit, R, best, wc)) return true;
    if (S.num_bvh_prims == 0) return false;
    if (S.num_bvh_prims == 1)
        return test_prim<ANYHIT, COUNT>(S, S.single_leaf, o, d, reverse, limit, R, best, wc);

    const FRay fr = make_fray(o, d);
    float tlim = ANYHIT ? prune_limit(limit) : __int_as_float(0x7f800000);   // shrinks as closer hits are found
    StackSpill<ANYHIT> spill;
    Stack<ANYHIT> st(shbase, spill);
    int cur = 0;                                           // node 0 is the root
    while (true) {
        descend<ANYHIT, COUNT>(S, fr, tlim, cur, st, wc);
        if (cur == BVH_DONE) break;
        if (test_prim<ANYHIT, COUNT>(S, ~cur, o, d, reverse, limit, R, best, wc)) return true;
        if (!ANYHIT && best.geom >= 0) tlim = prune_limit(best.wd);
        cur = st.pop(tlim);
        if (cur == BVH_DONE) break;
    }
    return false;
}

}  // namespace rt
