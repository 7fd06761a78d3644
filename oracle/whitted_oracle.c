/* whitted_oracle.c — TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C, CPU, FP64 restatement of the reference's per-pixel trace loop, operating on
 * the same flat scene descriptor the product receives (include/rt_b200.h).  It exists to
 * CHECK the CUDA path; nothing in the product imports, links or executes it (only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may).
 *
 * Each function cites the reference code it follows.  The floating-point association
 * order of every expression follows what the reference's Eigen 3.2.2 expression templates
 * evaluate under g++ -O2 (SSE2, no FMA): Vector4d reductions are two 2-wide packets added
 * lane-wise then horizontally, (x0+x2)+(x1+x3)  (eigen/Eigen/src/Core/Redux.h:131-136,
 * 299-305); 3-vector reductions split [0,1)+[1,3); small products accumulate left to
 * right.  Build with -ffp-contract=off.
 *
 * PARITY PINNED: tests/test_oracle_vs_reference.py checks this file against the
 * reference itself (oracle/_ref/libref.so: per-ray castRay / traceRay, bit for bit) and
 * tests/test_oracle_golden.py against the nine golden images outputs/image-0N.png.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "rt_b200.h"

typedef struct { double x, y, z; } v3;

static inline double sum4(double a, double b, double c, double d) { return (a + c) + (b + d); }
/* 4-vector dot of two DIRECTION-like vectors (w = 0): the w product is an exact +0 */
static inline double dot4(v3 a, v3 b) { return sum4(a.x * b.x, a.y * b.y, a.z * b.z, 0.0); }
static inline double norm4(v3 a) { return sqrt(dot4(a, a)); }
static inline v3 vsub(v3 a, v3 b) { v3 r = {a.x - b.x, a.y - b.y, a.z - b.z}; return r; }
static inline v3 vadd(v3 a, v3 b) { v3 r = {a.x + b.x, a.y + b.y, a.z + b.z}; return r; }
static inline v3 vscale(double s, v3 a) { v3 r = {s * a.x, s * a.y, s * a.z}; return r; }
static inline v3 vdiv(v3 a, double s) { v3 r = {a.x / s, a.y / s, a.z / s}; return r; }
static inline v3 vneg(v3 a) { v3 r = {-a.x, -a.y, -a.z}; return r; }
static inline v3 ld3(const double* p) { v3 r = {p[0], p[1], p[2]}; return r; }

/* Transform4d * Vector4d (eigen/Eigen/src/Geometry/Transform.h:1244-1267): rows 0..2 of
 * the 3x4 affine block times the homogeneous vector, accumulated left to right. */
static inline v3 xf_apply(const double* m, v3 v, double w) {
    v3 r;
    r.x = ((m[0] * v.x + m[1] * v.y) + m[2] * v.z) + m[3] * w;
    r.y = ((m[4] * v.x + m[5] * v.y) + m[6] * v.z) + m[7] * w;
    r.z = ((m[8] * v.x + m[9] * v.y) + m[10] * v.z) + m[11] * w;
    return r;
}
/* inverseTransform().matrix().transpose() * N  then w := 0 (src/geometry.cpp:40-41) */
static inline v3 xf_normal(const double* inv, v3 n) {
    v3 r;
    r.x = sum4(inv[0] * n.x, inv[4] * n.y, inv[8] * n.z, 0.0);
    r.y = sum4(inv[1] * n.x, inv[5] * n.y, inv[9] * n.z, 0.0);
    r.z = sum4(inv[2] * n.x, inv[6] * n.y, inv[10] * n.z, 0.0);
    return r;
}

/* Matrix3d::determinant (eigen/Eigen/src/LU/Determinant.h:18-23,61-69), columns c0 c1 c2 */
static inline double det3_helper(double m0a, double m1b, double m2c, double m1c, double m2b) {
    return m0a * (m1b * m2c - m1c * m2b);
}
static inline double det3(v3 c0, v3 c1, v3 c2) {
    /* helper(a,b,c) = m(0,a) * (m(1,b)*m(2,c) - m(1,c)*m(2,b)); m(r,col) */
    double h012 = det3_helper(c0.x, c1.y, c2.z, c2.y, c1.z);
    double h102 = det3_helper(c1.x, c0.y, c2.z, c2.y, c0.z);
    double h201 = det3_helper(c2.x, c0.y, c1.z, c1.y, c0.z);
    return h012 - h102 + h201;
}

typedef struct {
    int hit;
    int face;
    v3 P, N;     /* object space */
    double a, b; /* barycentrics (mesh) */
} objhit;

/* hitsBoundingBox (src/geometry.cpp:5-29) */
static int hits_bbox(v3 o, v3 d, const double* bbmin, const double* bbmax) {
    const double oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
    for (int axis = 0; axis < 3; axis++) {
        for (int bn = 0; bn < 2; bn++) {
            double mag = dd[axis];
            if (mag == 0.0) continue;
            double t = ((bn ? bbmax : bbmin)[axis] - oo[axis]) / mag;
            if (t < 0) continue;
            double ip[3] = {oo[0] + t * dd[0], oo[1] + t * dd[1], oo[2] + t * dd[2]};
            int ok = 1;
            for (int a2 = 0; a2 < 3; a2++) {
                if (a2 == axis) continue;
                if (ip[a2] < bbmin[a2] || ip[a2] > bbmax[a2]) { ok = 0; break; }
            }
            if (ok) return 1;
        }
    }
    return 0;
}

/* Sphere::calculateIntNormInObjSpace (src/geometry.cpp:47-67) */
static objhit sphere_obj(const rt_geometry* g, v3 o, v3 d, int reverse) {
    objhit h; memset(&h, 0, sizeof(h));
    v3 ocd = vsub(o, ld3(g->center));
    double a = dot4(d, d);
    double b = 2 * dot4(d, ocd);
    double c = dot4(ocd, ocd) - g->radius2;
    double disc = b * b - 4 * a * c;
    double res;
    if (disc < 0) return h;
    if (reverse) res = (-b + sqrt(disc)) / (2 * a);
    else res = (-b - sqrt(disc)) / (2 * a);
    if (res < 0) return h;
    h.hit = 1;
    h.P = vadd(o, vscale(res, d));
    h.N = vsub(h.P, ld3(g->center));
    return h;
}

/* Mesh::calculateIntNormInObjSpace (src/geometry.cpp:69-126) */
static objhit mesh_obj(const rt_scene* s, const rt_geometry* g, v3 o, v3 d, int reverse) {
    objhit h; memset(&h, 0, sizeof(h));
    h.face = -1;
    if (g->use_bbox && !hits_bbox(o, d, g->bbmin, g->bbmax)) return h;
    double closest = INFINITY;
    v3 nd = vneg(d);
    for (int64_t f = 0; f < g->num_faces; f++) {
        const double* fp = s->face_points + 9 * (g->first_face + f);
        const double* fn = s->face_normals + 9 * (g->first_face + f);
        v3 p0 = ld3(fp), p1 = ld3(fp + 3), p2 = ld3(fp + 6);
        v3 va = vsub(p1, p0), vb = vsub(p2, p0), rhs = vsub(o, p0);
        double dlower = det3(va, vb, nd);
        if (dlower == 0) continue;
        double a = det3(rhs, vb, nd) / dlower;
        if (a < 0 || a > 1) continue;
        double b = det3(va, rhs, nd) / dlower;
        if (b < 0 || a + b > 1) continue;
        double t = det3(va, vb, rhs) / dlower;
        if (t < 0) continue;
        /* Vector3d::norm: unrolled scalar redux x + (y + z) */
        double dist = t * sqrt(d.x * d.x + (d.y * d.y + d.z * d.z));
        if (dist >= closest) continue;
        v3 n0 = ld3(fn), n1 = ld3(fn + 3), n2 = ld3(fn + 6);
        double w0 = 1.0 - a - b;
        v3 tn = vadd(vadd(vscale(w0, n0), vscale(a, n1)), vscale(b, n2));
        int front = dot4(tn, d) < 0;
        if ((!front) ^ (reverse != 0)) continue;
        h.hit = 1;
        h.face = (int)f;
        closest = dist;
        h.P = vadd(p0, vadd(vscale(a, va), vscale(b, vb)));
        h.N = tn;
        h.a = a; h.b = b;
    }
    return h;
}

typedef struct {
    int hit, geom, face;
    double dist;
    v3 P, N;
} worldhit;

/* Geometry::calculateIntersectionNormal (src/geometry.cpp:31-45) for one geometry */
static int geom_query(const rt_scene* s, int gi, v3 o, v3 d, int reverse, v3* P, v3* N, int* face) {
    const rt_geometry* g = &s->geometries[gi];
    v3 oo = xf_apply(g->inv, o, 1.0);
    v3 dd = xf_apply(g->inv, d, 0.0);
    dd = vdiv(dd, norm4(dd));                     /* Ray ctor re-normalises (src/rtbase.h:23) */
    objhit h = (g->type == RT_GEOM_SPHERE) ? sphere_obj(g, oo, dd, reverse) : mesh_obj(s, g, oo, dd, reverse);
    if (!h.hit) return 0;
    *P = xf_apply(g->fwd, h.P, 1.0);
    v3 n = xf_normal(g->inv, h.N);
    if (g->det < 0) n = vneg(n);
    *N = n;
    *face = (g->type == RT_GEOM_SPHERE) ? 0 : h.face;
    return 1;
}

/* Scene::castRay (src/scene.cpp:142-167) */
static worldhit cast_ray(const rt_scene* s, v3 o, v3 d, int reverse) {
    worldhit w; memset(&w, 0, sizeof(w));
    w.geom = -1; w.face = -1;
    for (int gi = 0; gi < s->num_geometries; gi++) {
        v3 P, N; int face;
        if (!geom_query(s, gi, o, d, reverse, &P, &N, &face)) continue;
        double dist = norm4(vsub(P, o));
        if (w.hit && dist >= w.dist) continue;
        w.hit = 1; w.geom = gi; w.face = face; w.dist = dist; w.P = P; w.N = N;
    }
    return w;
}

typedef struct {
    uint64_t primary, shadow, secondary, degenerate;
} counts_t;

/* Ray constructor (src/rtbase.h:7-24): returns 0 if the reference would throw */
static int make_dir(v3 raw, v3* out) {
    if (raw.x == 0 && raw.y == 0 && raw.z == 0) return 0;
    *out = vdiv(raw, norm4(raw));
    return 1;
}

/* Scene::traceRay (src/scene.cpp:61-140) */
static void trace_ray(const rt_scene* s, const rt_params* p, v3 o, v3 d, int depth, int inside,
                      counts_t* cnt, double out[3]) {
    out[0] = out[1] = out[2] = 0.0;
    worldhit w = cast_ray(s, o, d, inside);
    if (!w.hit) return;
    if (p->intersection_only) {
        double v = 1.0 / (w.dist * w.dist);
        out[0] = out[1] = out[2] = v;
        return;
    }
    v3 N = w.N;
    if (inside) N = vneg(N);
    /* Vector4d::normalize() is `*this /= norm()`, which Eigen 3.2 evaluates as a multiply by
     * the reciprocal (eigen/Eigen/src/Core/SelfCwiseBinaryOp.h operator/=), unlike
     * normalized(), which divides */
    N = vscale(1.0 / norm4(N), N);
    const rt_material* m = &s->materials[s->geometries[w.geom].material];
    double col[3] = {0, 0, 0};
    for (int li = 0; li < s->num_lights; li++) {
        const rt_light* l = &s->lights[li];
        if (l->type == RT_LIGHT_AMBIENT) {
            for (int k = 0; k < 3; k++) col[k] += 1.0 * l->color[k] * m->ka[k];
            continue;
        }
        v3 toL; double dL;
        if (l->type == RT_LIGHT_POINT) {
            toL = vsub(ld3(l->v), w.P);
        } else {
            toL = vneg(ld3(l->v));
        }
        v3 L;
        if (!make_dir(toL, &L)) { cnt->degenerate++; continue; }
        int lrev = dot4(N, L) < 0;
        dL = (l->type == RT_LIGHT_POINT) ? norm4(toL) : INFINITY;
        cnt->shadow++;
        worldhit occ = cast_ray(s, w.P, L, lrev ^ inside);
        if (occ.hit && occ.dist <= dL) continue;
        double att[3];
        if (l->type == RT_LIGHT_POINT) {
            double f = pow(dL, -l->falloff);
            for (int k = 0; k < 3; k++) att[k] = f * l->color[k];
        } else {
            for (int k = 0; k < 3; k++) att[k] = l->color[k];
        }
        double ndl = dot4(N, L);
        /* std::max(x, 0.0) is (x < 0.0) ? 0.0 : x, which keeps x = -0.0: pow(-0.0, y) differs from pow(+0.0, y)
         * for a negative odd whole y (-inf against +inf), and -V.R is -0.0 wherever V.R is exactly zero */
        double di = ndl < 0.0 ? 0.0 : ndl;
        for (int k = 0; k < 3; k++) col[k] += di * att[k] * m->kd[k];
        v3 R = vsub(vscale(2 * dot4(N, L), N), L);
        double mvr = -dot4(d, R);
        double si = pow(mvr < 0.0 ? 0.0 : mvr, m->sp);
        for (int k = 0; k < 3; k++) col[k] += si * att[k] * m->ks[k];
    }
    double kr[3] = {m->kr[0], m->kr[1], m->kr[2]};
    if (depth > 0) {
        if (!(m->kt[0] == 0 && m->kt[1] == 0 && m->kt[2] == 0)) {
            double n = m->ior;
            if (!inside) n = 1.0 / n;
            double cosI = dot4(N, d);
            double sinT2 = n * n * (1.0 - cosI * cosI);
            if (sinT2 > 1.0) {
                kr[0] = kr[1] = kr[2] = 1.0;
            } else {
                v3 T = vsub(vscale(n, d), vscale(n * cosI + sqrt(1.0 - sinT2), N));
                v3 Td;
                if (make_dir(T, &Td)) {
                    double c2[3];
                    cnt->secondary++;
                    trace_ray(s, p, w.P, Td, depth - 1, !inside, cnt, c2);
                    for (int k = 0; k < 3; k++) col[k] += c2[k];
                } else cnt->degenerate++;
            }
        }
        if (!(kr[0] == 0 && kr[1] == 0 && kr[2] == 0)) {
            v3 Rv = vsub(d, vscale(2 * dot4(N, d), N));
            v3 Rd;
            if (make_dir(Rv, &Rd)) {
                double c2[3];
                cnt->secondary++;
                trace_ray(s, p, w.P, Rd, depth - 1, inside, cnt, c2);
                for (int k = 0; k < 3; k++) col[k] += c2[k] * kr[k];
            } else cnt->degenerate++;
        }
    }
    out[0] = col[0]; out[1] = col[1]; out[2] = col[2];
}

/* Camera::calculateViewingRay (src/rtbase.h:74-84) at pixel (r,c) (src/scene.cpp:26-30) */
/* sub > 1: the ray through the centre of cell (si, sj) of a sub x sub grid inside the pixel
 * (supersampling, the extension of src/scene.cpp:28-29 described at rt_params.samples). */
static void camera_ray_sub(const rt_scene* s, int width, int height, int r, int c, int sub, int si, int sj, v3* o, v3* d) {
    const rt_camera* cam = &s->camera;
    double rowFrac = (r + 0.5) / height, colFrac = (c + 0.5) / width;
    if (sub > 1) {
        rowFrac = (r + (sj + 0.5) / sub) / height;
        colFrac = (c + (si + 0.5) / sub) / width;
    }
    v3 LR = ld3(cam->lr), UR = ld3(cam->ur), LL = ld3(cam->ll), UL = ld3(cam->ul), E = ld3(cam->eye);
    v3 right = vadd(vscale(rowFrac, LR), vscale(1.0 - rowFrac, UR));
    v3 left = vadd(vscale(rowFrac, LL), vscale(1.0 - rowFrac, UL));
    v3 ip = vadd(vscale(colFrac, right), vscale(1.0 - colFrac, left));
    v3 raw = vsub(ip, E);
    *o = E;
    *d = vdiv(raw, norm4(raw));
}
static void camera_ray(const rt_scene* s, int width, int height, int r, int c, v3* o, v3* d) {
    camera_ray_sub(s, width, height, r, c, 1, 0, 0, o, d);
}

/* ---- public (test-only) API --------------------------------------------- */

typedef struct {
    const rt_scene* s; const rt_params* p;
    double* rgb; int32_t* geom; int32_t* face;
    int64_t* next; int64_t total; int64_t block;
    counts_t cnt;
    pthread_mutex_t* mu;
} job_t;

static void* worker(void* arg) {
    job_t* j = (job_t*)arg;
    const int W = j->p->width, H = j->p->height;
    for (;;) {
        int64_t start = __atomic_fetch_add(j->next, j->block, __ATOMIC_RELAXED);
        if (start >= j->total) break;
        int64_t end = start + j->block < j->total ? start + j->block : j->total;
        for (int64_t i = start; i < end; i++) {
            int r = (int)(i / W), c = (int)(i % W);
            v3 o, d;
            const int sub = j->p->samples > 1 ? j->p->samples : 1;
            if (sub > 1) {          /* mean of the sub x sub sample colours */
                double acc[3] = {0, 0, 0}, col[3];
                for (int sj = 0; sj < sub; sj++)
                    for (int si = 0; si < sub; si++) {
                        camera_ray_sub(j->s, W, H, r, c, sub, si, sj, &o, &d);
                        j->cnt.primary++;
                        col[0] = col[1] = col[2] = 0.0;
                        trace_ray(j->s, j->p, o, d, j->p->bounce_depth, 0, &j->cnt, col);
                        for (int k = 0; k < 3; k++) acc[k] += col[k] * (1.0 / (sub * sub));
                    }
                for (int k = 0; k < 3; k++) j->rgb[3 * i + k] = acc[k];
                continue;
            }
            camera_ray(j->s, W, H, r, c, &o, &d);
            j->cnt.primary++;
            trace_ray(j->s, j->p, o, d, j->p->bounce_depth, 0, &j->cnt, j->rgb + 3 * i);
            if (j->geom || j->face) {
                worldhit w = cast_ray(j->s, o, d, 0);
                if (j->geom) j->geom[i] = w.geom;
                if (j->face) j->face[i] = w.face;
            }
        }
    }
    return NULL;
}

/* Scene::renderScene (src/scene.cpp:10-59) with the last block clamped. */
int oracle_render(const rt_scene* s, const rt_params* p, double* rgb, int32_t* geom, int32_t* face,
                  uint64_t counts[4], int threads) {
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    int64_t next = 0, total = (int64_t)p->width * p->height;
    job_t jobs[256]; pthread_t th[256];
    /* 2000-pixel blocks like src/scene.cpp:13, smaller on small frames so all threads work */
    int64_t block = total / ((int64_t)threads * 4);
    if (block > 2000) block = 2000;
    if (block < 1) block = 1;
    for (int t = 0; t < threads; t++) {
        memset(&jobs[t], 0, sizeof(job_t));
        jobs[t].block = block;
        jobs[t].s = s; jobs[t].p = p; jobs[t].rgb = rgb; jobs[t].geom = geom; jobs[t].face = face;
        jobs[t].next = &next; jobs[t].total = total;
        pthread_create(&th[t], NULL, worker, &jobs[t]);
    }
    counts_t c; memset(&c, 0, sizeof(c));
    for (int t = 0; t < threads; t++) {
        pthread_join(th[t], NULL);
        c.primary += jobs[t].cnt.primary; c.shadow += jobs[t].cnt.shadow;
        c.secondary += jobs[t].cnt.secondary; c.degenerate += jobs[t].cnt.degenerate;
    }
    if (counts) { counts[0] = c.primary; counts[1] = c.shadow; counts[2] = c.secondary; counts[3] = c.degenerate; }
    if (p->intersection_only) {   /* src/scene.cpp:50-58 */
        double mx = 2.2250738585072014e-308;   /* std::numeric_limits<double>::min() */
        for (int64_t i = 0; i < total * 3; i++) if (rgb[i] > mx) mx = rgb[i];
        for (int64_t i = 0; i < total * 3; i++) rgb[i] /= mx;
    }
    return 0;
}

/* Scene::castRay for caller-supplied rays (dir normalised like the Ray ctor). */
int oracle_cast_rays(const rt_scene* s, int64_t n, const double* org, const double* dir, const uint8_t* reverse,
                     int32_t* geom, int32_t* face, double* dist, double* point, double* normal) {
    for (int64_t i = 0; i < n; i++) {
        v3 o = ld3(org + 3 * i), d;
        worldhit w; memset(&w, 0, sizeof(w)); w.geom = -1; w.face = -1;
        if (make_dir(ld3(dir + 3 * i), &d)) w = cast_ray(s, o, d, reverse ? reverse[i] : 0);
        else w.geom = -2;
        if (geom) geom[i] = w.geom;
        if (face) face[i] = w.face;
        if (dist) dist[i] = w.hit ? w.dist : 0.0;
        if (point) { point[3 * i] = w.hit ? w.P.x : 0; point[3 * i + 1] = w.hit ? w.P.y : 0; point[3 * i + 2] = w.hit ? w.P.z : 0; }
        if (normal) { normal[3 * i] = w.hit ? w.N.x : 0; normal[3 * i + 1] = w.hit ? w.N.y : 0; normal[3 * i + 2] = w.hit ? w.N.z : 0; }
    }
    return 0;
}

int oracle_trace_rays(const rt_scene* s, int64_t n, const double* org, const double* dir, int depth,
                      const uint8_t* from_inside, double* rgb) {
    rt_params p; memset(&p, 0, sizeof(p));
    counts_t c; memset(&c, 0, sizeof(c));
    for (int64_t i = 0; i < n; i++) {
        v3 o = ld3(org + 3 * i), d;
        if (make_dir(ld3(dir + 3 * i), &d))
            trace_ray(s, &p, o, d, depth, from_inside ? from_inside[i] : 0, &c, rgb + 3 * i);
        else rgb[3 * i] = rgb[3 * i + 1] = rgb[3 * i + 2] = NAN;
    }
    return 0;
}

int oracle_camera_rays(const rt_scene* s, int width, int height, int64_t n, const int64_t* pix, double* org, double* dir) {
    for (int64_t k = 0; k < n; k++) {
        v3 o, d;
        camera_ray(s, width, height, (int)(pix[k] / width), (int)(pix[k] % width), &o, &d);
        org[3 * k] = o.x; org[3 * k + 1] = o.y; org[3 * k + 2] = o.z;
        dir[3 * k] = d.x; dir[3 * k + 1] = d.y; dir[3 * k + 2] = d.z;
    }
    return 0;
}
