"""The shading kernels over the light and material parameters no shipped scene uses, against the FP64 oracle.

Hit finding is checked ray by ray elsewhere; here the subject is what k_shade, k_shadow, pow_shading and the
resolve kernels do with a hit: point-light falloff, specular exponents off the whole numbers 1..1024, many lights
and light counts that do not divide a warp, negative and zero colours, the zero-contribution cull, refraction
with every kind of index, degenerate shadow rays, more than 2^32 (hit, light) pairs in one launch, and the
RGB8 quantiser at its edges.  Scenes are written as .rti / .obj text with every number in %.17g.

Unless a case says otherwise, a scene is rendered with and without RT_FLAG_BRUTE_FORCE and compared with
oracle.render: primary geometry and face ids and the four ray counts exactly, the FP64 frame within
FP64_TOL * max(1, |oracle|) per value.  The bound is relative because falloff and bright lights push values far
above 1, and it covers:
  * the order of the framebuffer's atomic additions (one per light and bounce, in any order; a few ulp of the
    pixel when the terms have one sign, and the scenes keep large terms of both signs apart);
  * pow_shading's binary exponentiation for whole exponents in 1..1024, relative error <= y * 2^-53 <= 1.2e-13,
    and CUDA's pow against glibc's elsewhere (2 ulp);
  * 1/dL and 1/(dL*dL) against the oracle's pow(dL, -1) and pow(dL, -2): at most 1 and 2 ulp.
Non-finite values (negative exponents at a zero base) are legitimate frame values: NaN must sit where the
oracle has NaN, and +-inf where it has the same infinity.
"""
import numpy as np
import pytest

from conftest import quantize
from test_gpu_round2 import same_device_multi  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-9
COUNTS = ("rays_primary", "rays_shadow", "rays_secondary", "degenerate_rays")


def g(x):
    return "%.17g" % x


def line(kw, *nums):
    return kw + " " + " ".join(g(float(x)) for x in nums)


def mat(ka=(0.1, 0.1, 0.1), kd=(0.5, 0.5, 0.5), ks=(0.3, 0.3, 0.3), sp=10.0, kr=(0, 0, 0), kt=(0, 0, 0), ior=1.0):
    return line("mat", *ka, *kd, *ks, sp, *kr, *kt, ior)


def cam(eye, ll, lr, ul, ur):
    return line("cam", *eye, *ll, *lr, *ul, *ur)


def write_scene(pkg, tmp_path, name, lines, objs=None):
    """objs: {file name: .obj text} written beside the scene; `obj` lines name them without a directory."""
    for fname, text in (objs or {}).items():
        (tmp_path / fname).write_text(text)
    path = tmp_path / name
    path.write_text("\n".join(lines) + "\n")
    return pkg.HostScene.load(path), path


def octahedron(c, r):
    """Closed mesh, faces wound counter-clockwise seen from outside (outward face normals)."""
    v = [(c[0] + r, c[1], c[2]), (c[0] - r, c[1], c[2]), (c[0], c[1] + r, c[2]), (c[0], c[1] - r, c[2]),
         (c[0], c[1], c[2] + r), (c[0], c[1], c[2] - r)]
    f = [(1, 3, 5), (3, 2, 5), (2, 4, 5), (4, 1, 5), (3, 1, 6), (2, 3, 6), (4, 2, 6), (1, 4, 6)]
    return "".join(line("v", *p) + "\n" for p in v) + "".join(f"f {a} {b} {c_}\n" for a, b, c_ in f)


def cube(c, h):
    """Closed axis-aligned cube of half-size h, outward face normals."""
    v = [(c[0] + sx * h, c[1] + sy * h, c[2] + sz * h) for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)]
    # vertex k = 4 * (sx > 0) + 2 * (sy > 0) + (sz > 0), 1-based in the file
    quads = [(1, 2, 4, 3), (5, 7, 8, 6), (1, 5, 6, 2), (3, 4, 8, 7), (1, 3, 7, 5), (2, 6, 8, 4)]
    out = "".join(line("v", *p) + "\n" for p in v)
    for a, b, c_, d in quads:
        out += f"f {a} {b} {c_}\nf {a} {c_} {d}\n"
    return out


def assert_frames_close(got, want, what=""):
    """FP64 frame check: NaN where the oracle has NaN, the same infinities, finite values within the bound."""
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN positions differ"
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf), f"{what}: infinities differ"
    assert np.array_equal(got[inf], want[inf]), f"{what}: signs of infinities differ"
    fin = np.isfinite(want)
    err = np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))
    assert err.max(initial=0.0) <= FP64_TOL, f"{what}: max relative error {err.max():.3g}"


def check_scene(pkg, gpu_renderer, oracle, sc, w, h, depth, what=""):
    """The default comparison: ids, the four counts and the frame, with and without the LBVH."""
    gpu_renderer.upload(sc)
    o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, depth)
    for flags in (0, pkg.RT_FLAG_BRUTE_FORCE):
        geom, face = gpu_renderer.primary_ids(w, h, flags=flags)
        assert np.array_equal(geom, o_geom) and np.array_equal(face, o_face), what
        rgb = gpu_renderer.render(w, h, depth, flags=flags)
        st = gpu_renderer.stats()
        assert [st[k] for k in COUNTS] == counts, (what, flags, [st[k] for k in COUNTS], counts)
        assert_frames_close(rgb, o_rgb, f"{what} flags={flags}")
    return o_rgb, counts


# Camera of the perspective scenes: eye on +z looking down -z, symmetric corners.
CAM = cam((0, 0, 30), (-10, -10, 10), (10, -10, 10), (-10, 10, 10), (10, 10, 10))


# ------------------------------------------------------------------ 1. point-light falloff
FALLOFFS = [0.0, 1.0, 2.0, 0.5, 1.5, 3.0, -1.0, -2.5]


def falloff_scene(fo):
    """Sphere, `tri` floor and an octahedron mesh, lit by point lights at about 0.1, 3, 100 and 1e4 from the
    lit surfaces, all with falloff `fo`."""
    lines = [CAM, line("lta", 0.05, 0.05, 0.05),
             line("ltp", 0.5, -5.9, 8, 0.9, 0.8, 0.7, fo),          # 0.1 above the floor
             line("ltp", -6, 1, 5, 0.6, 0.7, 0.9, fo),              # a few units from sphere and floor
             line("ltp", 60, 80, 50, 0.8, 0.8, 0.8, fo),            # ~100
             line("ltp", 3000, 9000, 4000, 0.7, 0.6, 0.5, fo),      # ~1e4
             mat(kd=(0.6, 0.5, 0.4), ks=(0.3, 0.3, 0.3), sp=20, kr=(0.2, 0.2, 0.2)),
             line("tri", -40, -6, -60, 40, -6, -60, -40, -6, 40), line("tri", 40, -6, -60, 40, -6, 40, -40, -6, 40),
             mat(kd=(0.3, 0.5, 0.7), ks=(0.5, 0.5, 0.5), sp=50, kr=(0.3, 0.3, 0.3)),
             line("sph", 0, -2, 0, 3.5),
             mat(kd=(0.7, 0.3, 0.3), ks=(0.4, 0.4, 0.4), sp=8),
             'obj "oct.obj"']
    return lines, {"oct.obj": octahedron((8, -3, 2), 2.0)}


def test_point_light_falloff(pkg, gpu_renderer, oracle, tmp_path):
    """Every branch of k_shadow's falloff expression against the oracle's pow(dL, -falloff):
         fo == 0      -> 1                    (falloff 0)
         fo == 1      -> 1 / dL               (falloff 1)
         fo == 2      -> 1 / (dL * dL)        (falloff 2)
         otherwise    -> pow(dL, -fo)         (falloff 0.5, 1.5, 3, -1, -2.5)"""
    frames = {}
    for fo in FALLOFFS:
        lines, objs = falloff_scene(fo)
        sc, _ = write_scene(pkg, tmp_path, f"falloff_{fo}.rti", lines, objs)
        frames[fo], counts = check_scene(pkg, gpu_renderer, oracle, sc, 64, 48, 3, f"falloff {fo}")
        assert counts[1] > 0 and counts[2] > 0
    # the lights do reach the frame: every falloff gives its own picture
    for a in FALLOFFS:
        for b in FALLOFFS:
            if a < b:
                assert not np.array_equal(frames[a], frames[b]), (a, b)
    assert np.abs(frames[-2.5]).max() > 1e6        # the far light with a negative falloff is bright


# ------------------------------------------------------------------ 2. specular exponents
EXPONENTS = [0.0, 0.5, 1.0, 2.0, 3.0, 1023.0, 1024.0, 1024.5, 1025.0, 4096.0, -1.0, -2.0]
W_AX, H_AX = 65, 49                      # odd: the centre column's camera rays have V.x == +0 exactly


def exponent_scene(sp):
    """Axis-aligned camera looking down -z at a wall in the plane z = 0 (N = +z exactly) and a directional light
    along +x that grazes the wall: on the centre column V.R is exactly zero, so -V.R is -0.0.  A sphere and a point
    light give the usual lobes; the wall's blue ks is 0 (inf * 0 = NaN where the exponent is negative)."""
    lines = [cam((0, 0, 10), (-1, -0.75, 9), (1, -0.75, 9), (-1, 0.75, 9), (1, 0.75, 9)),
             line("lta", 0.1, 0.1, 0.1),
             line("ltd", 1, 0, 0, 0.7, 0.7, 0.7),
             line("ltp", 3, 4, 6, 0.8, 0.8, 0.8),
             line("ltd", -1, -1, -2, 0.5, 0.5, 0.5),
             mat(kd=(0.4, 0.4, 0.4), ks=(0.5, 0.3, 0.0), sp=sp, kr=(0.2, 0.2, 0.2)),
             line("tri", -20, -20, 0, 20, -20, 0, -20, 20, 0), line("tri", 20, -20, 0, 20, 20, 0, -20, 20, 0),
             mat(kd=(0.2, 0.5, 0.3), ks=(0.6, 0.6, 0.6), sp=sp, kr=(0.3, 0.3, 0.3)),
             line("sph", 2, -1, 2, 1.5)]
    return lines


def test_specular_exponents(pkg, gpu_renderer, oracle, tmp_path):
    """Every branch of pow_shading and of the specular term in k_shadow:
         mvr < 0 and sp > 0 -> +0 without pow                 (every sp > 0: the far side of each lobe)
         binary exponentiation, whole sp in 1..1024            (sp 1, 2, 3, 1023, 1024)
         pow fallback                                          (sp 0, 0.5, 1024.5, 1025, 4096, -1, -2)
         pow(-0.0, sp) at mvr = -0.0                           (every sp on the wall's centre column;
                                                                -inf for sp = -1, +inf for sp = -2)
    std::max(x, 0.0) keeps x = -0.0, so the reference's pow(std::max(-V.R, 0.0), -1) is -inf there.
    With sp = -1 and -2 most of the frame is not finite (pow(+0, sp < 0) = +inf wherever mvr < 0, and inf * 0 = NaN
    in the wall's blue channel), so these two scenes compare few finite values; the pow fallback with negative
    exponents on finite values is covered by the seeded mixed scenes with negative exponents (seeds 2, 5, 8, 11)."""
    for sp in EXPONENTS:
        sc, _ = write_scene(pkg, tmp_path, f"sp_{sp}.rti", exponent_scene(sp))
        rgb, counts = check_scene(pkg, gpu_renderer, oracle, sc, W_AX, H_AX, 2, f"sp {sp}")
        centre = rgb[:, W_AX // 2, 0]
        if sp == -1.0:
            assert (centre == -np.inf).any()
        elif sp == -2.0:
            assert (centre == np.inf).any()
        else:
            assert np.isfinite(rgb).all()


# ------------------------------------------------------------------ 3. light kinds and counts
def lights_scene(n, seed):
    """n shadow lights (point and directional, in turn) with an ambient light after every fifth, colours from
    [-1, 1] with some exactly zero; a floor and spheres that fill most of a 97 x 61 frame."""
    rng = np.random.default_rng(seed)
    lines = [cam((0, 4, 30), (-12, -9, 10), (12, -9, 10), (-12, 6, 10), (12, 6, 10))]
    for i in range(n):
        col = rng.uniform(-1, 1, 3)
        col[rng.uniform(size=3) < 0.2] = 0.0
        if i % 2 == 0:
            lines.append(line("ltp", *rng.uniform([-20, 1, -20], [20, 25, 25]), *col))
        else:
            lines.append(line("ltd", *rng.uniform([-1, -1, -1], [1, -0.1, 1]), *col))
        if i % 5 == 4:
            lines.append(line("lta", *rng.uniform(-0.1, 0.2, 3)))
    lines += [mat(ka=(0.2, 0.1, -0.1), kd=(0.6, -0.2, 0.5), ks=(0.3, 0.0, 0.4), sp=15, kr=(0.25, 0.25, 0.25)),
              line("tri", -300, -5, -300, 300, -5, -300, -300, -5, 300),
              line("tri", 300, -5, -300, 300, -5, 300, -300, -5, 300),
              mat(ka=(0.1, 0.1, 0.1), kd=(0.2, 0.7, 0.4), ks=(0.5, 0.5, 0.5), sp=30, kr=(0.4, 0.1, 0.2)),
              line("sph", -5, -1, 0, 3), line("sph", 5, 0, -3, 4)]
    return lines


@pytest.mark.parametrize("n", [1, 31, 33, 257])
def test_light_kinds_and_counts(pkg, gpu_renderer, oracle, tmp_path, n):
    """Ambient lights interleaved with the others in the file (the GPU splits them into two tables and keeps each
    one's order), negative and zero colours, light counts that do not divide a warp, and a primary level of more
    than RT_SHADOW_TILE (4096) hits that is not a multiple of it: the last, partial tile of the light-major
    mapping."""
    sc, _ = write_scene(pkg, tmp_path, f"lights_{n}.rti", lights_scene(n, 100 + n))
    w, h = 97, 61
    _, counts = check_scene(pkg, gpu_renderer, oracle, sc, w, h, 2, f"{n} lights")
    geom, _ = gpu_renderer.primary_ids(w, h)
    primary_hits = int((geom >= 0).sum())
    assert primary_hits > 4096 and primary_hits % 4096 != 0
    assert counts[1] >= primary_hits * n


# ------------------------------------------------------------------ 4. the zero-contribution cull
def cull_scene(lit_from_above):
    """A floor with ks = 0 lit only from below (N.L < 0 and no specular term) and a mirror sphere with
    kd = ks = 0: every shadow ray's light term is exactly zero.  lit_from_above adds one light that is not."""
    lines = [CAM, line("lta", 0.2, 0.3, 0.4),
             line("ltp", 3, -20, 4, 1, 1, 1), line("ltp", -30, -8, -10, 0.5, 0.9, 0.2, 1.0),
             line("ltd", 0.2, 1, -0.1, 0.7, 0.7, 0.7)]
    if lit_from_above:
        lines.append(line("ltp", 5, 20, 15, 0.8, 0.8, 0.8))
    lines += [mat(ka=(0.3, 0.2, 0.1), kd=(0.5, 0.5, 0.5), ks=(0, 0, 0), sp=10, kr=(0.3, 0.3, 0.3)),
              line("tri", -1000, -6, -1000, 1000, -6, -1000, -1000, -6, 1000),
              line("tri", 1000, -6, -1000, 1000, -6, 1000, -1000, -6, 1000),
              mat(ka=(0.1, 0.2, 0.3), kd=(0, 0, 0), ks=(0, 0, 0), sp=10, kr=(0.6, 0.6, 0.6)),
              line("sph", 0, -1, 0, 4)]
    return lines


def test_zero_contribution_cull(pkg, gpu_renderer, oracle, tmp_path):
    """k_shadow skips the occlusion query of a light whose diffuse and specular terms are both exactly zero.
    Where every term is zero, RT_FLAG_COUNT_WORK must report every shadow ray as culled; the frame is the same
    with and without the flag (bit for bit where only ambient terms reach it: their additions run in level
    order)."""
    for lit in (False, True):
        sc, _ = write_scene(pkg, tmp_path, f"cull_{lit}.rti", cull_scene(lit))
        w, h, depth = 64, 48, 3
        o_rgb, counts = check_scene(pkg, gpu_renderer, oracle, sc, w, h, depth, f"cull lit={lit}")
        for brute in (0, pkg.RT_FLAG_BRUTE_FORCE):
            plain = gpu_renderer.render(w, h, depth, flags=brute)
            counted = gpu_renderer.render(w, h, depth, flags=brute | pkg.RT_FLAG_COUNT_WORK)
            st = gpu_renderer.stats()
            assert [st[k] for k in COUNTS] == counts
            if lit:
                assert 0 < st["shadow_rays_culled"] < st["rays_shadow"]
                assert_frames_close(counted, plain, "cull, lit")
            else:
                assert st["shadow_rays_culled"] == st["rays_shadow"] > 0
                assert st["nodes_fetched"][1] == 0 and st["tris_tested"][1] == 0 and st["spheres_tested"][1] == 0
                assert np.array_equal(counted, plain)
                assert_frames_close(counted, o_rgb, "cull")


# ------------------------------------------------------------------ 5. refraction and reflection
IORS = [0.7, 1.0, 1.5, 2.4]


def refraction_scenes():
    """name -> (lines, objs).  kt without kr and kr with kt at every ior on spheres; a glass cube (closed mesh)
    whose inner faces reflect totally; 80 glass spheres (in the LBVH, so the inside flag of the rays that run
    in them goes through the LBVH traversal)."""
    head = [CAM, line("lta", 0.1, 0.1, 0.1), line("ltp", 10, 20, 25, 0.9, 0.9, 0.9), line("ltd", -0.3, -1, -0.5, 0.4, 0.4, 0.4)]
    floor = [mat(kd=(0.6, 0.6, 0.2), ks=(0.2, 0.2, 0.2), sp=10, kr=(0.1, 0.1, 0.1)),
             line("tri", -60, -8, -60, 60, -8, -60, -60, -8, 60), line("tri", 60, -8, -60, 60, -8, 60, -60, -8, 60),
             mat(kd=(0.1, 0.8, 0.3), ks=(0.1, 0.1, 0.1), sp=5), line("sph", 0, 0, -25, 7.5)]
    out = {}
    for ior in IORS:
        out[f"kt_{ior}"] = (head + floor + [mat(kd=(0.1, 0.1, 0.1), ks=(0.5, 0.5, 0.5), sp=40, kt=(0.9, 0.9, 0.9), ior=ior),
                                            line("sph", -4, 0, 4, 3.5), line("sph", 4.5, 1, 2, 2.5)], {})
        out[f"krkt_{ior}"] = (head + floor + [mat(kd=(0.1, 0.1, 0.1), ks=(0.5, 0.5, 0.5), sp=40, kr=(0.3, 0.2, 0.1),
                                                  kt=(0.8, 0.8, 0.8), ior=ior),
                                              line("sph", -4, 0, 4, 3.5), line("sph", 4.5, 1, 2, 2.5)], {})
    out["cube_tir"] = (head + floor + [mat(kd=(0.05, 0.05, 0.05), ks=(0.4, 0.4, 0.4), sp=60, kt=(1, 1, 1), ior=1.5),
                                       line("xfr", 20, 35, 10), 'obj "cube.obj"'], {"cube.obj": cube((0, 0, 0), 4.0)})
    glass = [mat(kd=(0.05, 0.05, 0.05), ks=(0.4, 0.4, 0.4), sp=60, kr=(0.1, 0.1, 0.1) if i % 3 == 0 else (0, 0, 0),
                 kt=(0.9, 0.9, 0.9), ior=(1.5, 2.4, 0.7, 1.0)[i % 4]) + "\n" +
             line("sph", -9 + 2.25 * (i % 9), -6 + 1.8 * (i // 9), 3 * ((i * 7) % 3) - 2, 0.7 + 0.05 * (i % 4))
             for i in range(80)]
    out["spheres_80"] = (head + floor + glass, {})
    return out


@pytest.mark.parametrize("name", sorted(refraction_scenes()))
def test_refraction_and_reflection(pkg, gpu_renderer, oracle, tmp_path, name):
    lines, objs = refraction_scenes()[name]
    sc, _ = write_scene(pkg, tmp_path, f"{name}.rti", lines, objs)
    _, counts = check_scene(pkg, gpu_renderer, oracle, sc, 64, 48, 6, name)
    assert counts[2] > 0


# ------------------------------------------------------------------ 6. degenerate shadow rays
DEGENERATE = [cam((0, 0, 10), (-1, -1, 9), (1, -1, 9), (-1, 1, 9), (1, 1, 9)),
              line("lta", 0.1, 0.1, 0.1), line("ltp", 0, 0, 0, 1, 1, 1), line("ltp", 3, 5, 8, 0.5, 0.5, 0.5),
              line("ltd", 0, -1, -1, 0.3, 0.3, 0.3),
              mat(kd=(0.5, 0.5, 0.5), ks=(0.3, 0.3, 0.3), sp=10, kr=(0.2, 0.2, 0.2)),
              line("sph", 0, 0, -1, 1)]


def test_degenerate_shadow_rays(pkg, gpu_renderer, oracle, tmp_path, same_device_multi):  # noqa: F811
    """A point light exactly at a hit point: the centre ray of an odd frame hits the sphere at exactly (0, 0, 0),
    where the light sits.  Its shadow ray has no direction (the reference would abort); it counts as degenerate
    and not as cast, like a degenerate secondary ray, on every render path."""
    sc, _ = write_scene(pkg, tmp_path, "degenerate.rti", DEGENERATE)
    w, h, depth = 33, 33, 2
    o_rgb, _, _, counts = oracle.render(sc.flat, w, h, depth)
    assert counts[3] >= 1
    gpu_renderer.upload(sc)
    for flags in (0, pkg.RT_FLAG_BRUTE_FORCE, pkg.RT_FLAG_SERIAL, pkg.RT_FLAG_SERIAL | pkg.RT_FLAG_BRUTE_FORCE):
        rgb = gpu_renderer.render(w, h, depth, flags=flags)
        st = gpu_renderer.stats()
        assert [st[k] for k in COUNTS] == counts, (flags, [st[k] for k in COUNTS], counts)
        assert_frames_close(rgb, o_rgb, f"flags={flags}")
    r = pkg.Renderer(0)
    try:
        r.upload(sc)
        rgb = r.render(w, h, depth, n_gpus=2)
        st = r.stats()
        assert [st[k] for k in COUNTS] == counts, ("n_gpus=2", [st[k] for k in COUNTS], counts)
        assert_frames_close(rgb, o_rgb, "n_gpus=2")
    finally:
        r.close()


# ------------------------------------------------------------------ 7. more than 2^32 (hit, light) pairs
N_LIGHTS_BIG = 4200          # x 2^20 hits = 4.40 G pairs; 4096 lights would be exactly 2^32


def big_light_scene():
    """A floor under a camera looking straight down fills every pixel.  64 lights above it with distinct colours
    at light indices spread over the whole table (first and last included); the other 4136 lie below it and,
    with the floor's ks = 0, contribute exactly zero."""
    rng = np.random.default_rng(4200)
    above = set(np.linspace(0, N_LIGHTS_BIG - 1, 64).round().astype(int).tolist())
    lines = [cam((0, 10, 0), (-1, 9, 1), (1, 9, 1), (-1, 9, -1), (1, 9, -1)), line("lta", 0.05, 0.05, 0.05)]
    for i in range(N_LIGHTS_BIG):
        if i in above:
            x, z = rng.uniform(-12, 12, 2)
            lines.append(line("ltp", x, rng.uniform(0.5, 6), z, *rng.uniform(0.01, 0.05, 3)))
        else:
            x, z = rng.uniform(-12, 12, 2)
            lines.append(line("ltp", x, rng.uniform(-6, -0.5), z, *rng.uniform(0.01, 0.05, 3)))
    lines += [mat(ka=(0.1, 0.1, 0.1), kd=(0.7, 0.6, 0.5), ks=(0, 0, 0), sp=1),
              line("tri", -50, 0, -50, -50, 0, 50, 50, 0, -50), line("tri", 50, 0, -50, -50, 0, 50, 50, 0, 50)]
    return lines


def test_shadow_pairs_beyond_32_bits(pkg, gpu_renderer, oracle, tmp_path):
    """1024 x 1024 hits x 4200 shadow lights = 4.40 G (hit, light) pairs in ONE k_shadow launch, which takes the
    64-bit thread mapping.  The ray queue holds 2 x 2^20 slots (twice the framebuffer, within [1 Mi, 64 Mi]), so
    the whole primary level is one chunk; RT_QUEUE_CAP is left alone.  Checked: 4096 seeded pixels against
    per-ray oracle traces, the full frame against the same frame from two tile ranks (2.2 G pairs each: the
    32-bit mapping), and rays_shadow == hits x 4200.
    Cost, measured on a B200 at a 1000 W power limit: the k_shadow launch takes 74.5 ms, the library holds about
    340 MiB of device memory for this frame, and the test runs in about 2.3 s, most of it the oracle's 4096 traces."""
    import torch
    sc, _ = write_scene(pkg, tmp_path, "big_lights.rti", big_light_scene())
    w = h = 1024
    depth = 0
    gpu_renderer.upload(sc)
    rgb = gpu_renderer.render(w, h, depth, flags=pkg.RT_FLAG_TIME_KERNELS)
    st = gpu_renderer.stats()
    assert st["hits"] == w * h
    assert st["rays_shadow"] == w * h * N_LIGHTS_BIG
    assert st["launches_kernel"][2] == 1                    # one k_shadow launch for the whole level
    assert st["hits"] * N_LIGHTS_BIG > 2 ** 32
    rng = np.random.default_rng(32)
    pix = rng.choice(w * h, 4096, replace=False)
    org, direction = oracle.camera_rays(sc.flat, w, h, pix)
    want = oracle.trace_rays(sc.flat, org, direction, depth)
    got = rgb.reshape(-1, 3)[pix]
    assert_frames_close(got, want, "4096 pixels")
    assert np.ptp(want) > 0.1                               # the lights above the floor do light it
    # the same frame from two tile ranks, each under 2^32 pairs
    world = 2
    p0 = pkg.make_params(w, h, depth, tile_rank=0, tile_world=world)
    _, max_tiles, _ = pkg.tile_counts(p0)
    packed = torch.zeros(world, max_tiles * pkg.RT_TILE_PIXELS * 3, dtype=torch.float64, device="cuda")
    shadow = 0
    for rank in range(world):
        p = pkg.make_params(w, h, depth, tile_rank=rank, tile_world=world)
        gpu_renderer.render_device(p, packed[rank].data_ptr(), rgb8=False)
        s = gpu_renderer.stats()
        assert s["hits"] * N_LIGHTS_BIG < 2 ** 32
        shadow += s["rays_shadow"]
    frame = torch.empty(h, w, 3, dtype=torch.float64, device="cuda")
    gpu_renderer.unpack_tiles(p0, packed.data_ptr(), frame.data_ptr(), rgb8=False)
    torch.cuda.synchronize()
    assert shadow == w * h * N_LIGHTS_BIG
    ranks = frame.cpu().numpy()
    # the same terms per pixel in another order: positive terms, a few ulp
    assert np.abs(ranks - rgb).max() <= 1e-13 * max(1.0, np.abs(rgb).max())


# ------------------------------------------------------------------ 8. RGB8 quantisation
def quant_values():
    # the neighbours of 0 are subnormal, which the scene parser refuses (strtod's ERANGE): the smallest normals instead
    tiny = np.finfo(float).tiny
    vals = [0.0, -0.0, -1e-300, -tiny, tiny, 1.0, np.nextafter(1.0, 2.0), 1e300]
    for k in range(1, 256):
        x = k / 255.0
        vals += [np.nextafter(x, -np.inf), x, np.nextafter(x, np.inf)]
    return vals


def test_rgb8_quantisation_edges(pkg, gpu_renderer, tmp_path, same_device_multi):  # noqa: F811
    """Ambient light 1 and one `tri` per pixel with its own ka: the FP64 pixel is exactly ka (depth 0, weight 1).
    The ka values sit on and next to every k/255 and around 0 and 1.  Both resolve kernels must quantise exactly
    like the reference's writer:
      * k_resolve<true>: rt_render_rgb8 of one context, into pageable or page-locked memory (both are staged on
        the device and copied back);
      * k_resolve_rgb8_rows: resolves that store into memory other than the context's own, here a page-locked
        frame filled by two tile ranks (RT_FLAG_FULL_FRAME) and by an n_gpus = 2 render.
    41 x 19 is two 32 x 32 tiles, one per rank: the row kernel takes its word stores (rows whose first byte is
    4-aligned, first tile) and its byte stores (odd rows, and the 9-column second tile)."""
    import torch
    vals = quant_values()
    w, h = 41, 19
    assert len(vals) <= w * h
    ka = np.full(w * h, 0.5)
    ka[:len(vals)] = vals
    ka = ka.reshape(h, w)
    # camera: pixel (c, r) looks at (c + 0.5 - w/2, h/2 - r - 0.5, 0) on the plane z = 0
    u = 0.1
    lines = [cam((0, 0, 10), (-w / 2 * u, -h / 2 * u, 9), (w / 2 * u, -h / 2 * u, 9), (-w / 2 * u, h / 2 * u, 9),
                 (w / 2 * u, h / 2 * u, 9)), line("lta", 1, 1, 1)]
    for r in range(h):
        for c in range(w):
            x, y = c + 0.5 - w / 2, h / 2 - r - 0.5
            a = ka[r, c]
            lines.append(mat(ka=(a, a, a), kd=(0, 0, 0), ks=(0, 0, 0), sp=1))
            lines.append(line("tri", x - 0.4, y - 0.4, 0, x + 0.4, y - 0.4, 0, x, y + 0.4, 0))
    sc, _ = write_scene(pkg, tmp_path, "quant.rti", lines)
    gpu_renderer.upload(sc)
    rgb = gpu_renderer.render(w, h, 0)
    want = np.repeat(ka[:, :, None], 3, axis=2)
    assert np.array_equal(rgb, want)                        # -0.0 == +0.0
    q = quantize(want)
    assert np.array_equal(pkg.quantize_rgb8(want), q)
    assert np.array_equal(gpu_renderer.render_rgb8(w, h, 0), q)
    pinned = torch.zeros(h, w, 3, dtype=torch.uint8).pin_memory()
    gpu_renderer.render_host_params(pkg.make_params(w, h, 0), pinned.data_ptr(), rgb8=True)
    assert np.array_equal(pinned.numpy(), q)
    # every rank stores its own tiles into the shared page-locked frame (remote memory: the row kernel)
    assert pkg.tile_counts(pkg.make_params(w, h, 0, tile_rank=0, tile_world=2))[2] == 2
    pinned.fill_(77)
    for rank in range(2):
        p = pkg.make_params(w, h, 0, tile_rank=rank, tile_world=2, flags=pkg.RT_FLAG_FULL_FRAME)
        gpu_renderer.render_host_params(p, pinned.data_ptr(), rgb8=True)
    assert np.array_equal(pinned.numpy(), q)
    # two sub-contexts store their tiles into the page-locked frame directly (the row kernel on both)
    r = pkg.Renderer(0)
    try:
        r.upload(sc)
        pinned.fill_(77)
        r.render_host_params(pkg.make_params(w, h, 0, n_gpus=2), pinned.data_ptr(), rgb8=True)
        assert np.array_equal(pinned.numpy(), q)
    finally:
        r.close()


# ------------------------------------------------------------------ 9. seeded mixed scenes
def mixed_scene(seed):
    """Spheres (some transformed; more than 64 in some seeds) each in its own cell of a grid, a `tri` floor and
    back wall, one closed mesh in a cell of its own, and materials and lights from the value sets above.  No two
    surfaces of different geometries come closer than 1e-3.  Seeds with negative exponents keep every colour and
    coefficient non-negative, so no large terms of opposite signs cancel."""
    rng = np.random.default_rng(1000 + seed)
    neg_sp = seed % 3 == 2
    sps = [s for s in EXPONENTS if s >= 0 or neg_sp]
    lo = 0.0 if neg_sp else -0.3

    def col(a, b):
        c = rng.uniform(max(a, lo) if a < 0 else a, b, 3)
        c[rng.uniform(size=3) < 0.1] = 0.0
        return c

    def material():
        kt = col(0, 0.9) if rng.uniform() < 0.35 else (0, 0, 0)
        kr = col(0, 0.6) if rng.uniform() < 0.5 else (0, 0, 0)
        return mat(ka=col(-0.1, 0.2), kd=col(-0.3, 0.8), ks=col(-0.2, 0.6), sp=rng.choice(sps), kr=kr, kt=kt,
                   ior=rng.choice(IORS))

    lines = [CAM]
    for _ in range(int(rng.integers(1, 9))):
        kind = rng.integers(0, 3)
        if kind == 0:
            lines.append(line("lta", *col(-0.05, 0.15)))
        elif kind == 1:
            lines.append(line("ltd", *rng.uniform([-1, -1, -1], [1, -0.2, 1]), *col(-0.5, 1)))
        else:
            lines.append(line("ltp", *rng.uniform([-15, 2, -10], [15, 20, 25]), *col(-0.5, 1), rng.choice(FALLOFFS)))
    lines += [material(), line("tri", -200, -10, -19, 200, -10, -19, -200, -10, 200),     # ends 1 short of the wall
              line("tri", 200, -10, -19, 200, -10, 200, -200, -10, 200),
              material(), line("tri", -200, -200, -20, 200, -200, -20, 0, 300, -20)]
    nsph = int(rng.choice([12, 40, 70, 100]))
    cells = [(i, j, k) for i in range(8) for j in range(5) for k in range(3)]
    order = rng.permutation(len(cells))
    mesh_cell = cells[order[0]]
    cell = 2.2
    centre = lambda c_: (-8 + cell * c_[0], -8 + cell * c_[1], -10 + cell * c_[2] + 2.5)
    for idx in order[1:1 + nsph]:
        c = centre(cells[idx])
        lines.append(material())
        r = rng.uniform(0.3, 0.7)
        if rng.uniform() < 0.3:
            # scale <= 1.4 about the cell centre: the ellipsoid stays inside the cell (0.7 * 1.4 < 1.1 - 1e-3)
            lines += ["xfz", line("xft", *c), line("xfr", *rng.uniform(-90, 90, 3)),
                      line("xfs", *rng.uniform(0.6, 1.4, 3)), line("sph", 0, 0, 0, r), "xfz"]
        else:
            lines.append(line("sph", *c, r))
    lines += [material(), 'obj "mesh.obj"']
    return lines, {"mesh.obj": octahedron(centre(mesh_cell), 0.9)}


@pytest.mark.parametrize("seed", range(12))
def test_seeded_mixed_scenes(pkg, gpu_renderer, oracle, tmp_path, seed):
    lines, objs = mixed_scene(seed)
    sc, _ = write_scene(pkg, tmp_path, f"mixed_{seed}.rti", lines, objs)
    check_scene(pkg, gpu_renderer, oracle, sc, 64, 48, 5, f"seed {seed}")


# ------------------------------------------------------------------ 10. the oracle against the reference
def test_oracle_matches_the_reference_on_the_new_parameters(pkg, oracle, live_reference, tmp_path):
    """oracle.trace_rays against the unmodified reference's traceRay, bit for bit, on the falloff, exponent and
    refraction scenes (camera rays and rays from surface points in random directions, both fromInside values)."""
    if live_reference is None:
        pytest.skip("oracle/_ref/libref.so not built (needs the reference sources at build time, oracle/Makefile REF=)")
    scenes = [(f"falloff_{fo}.rti", *falloff_scene(fo)) for fo in FALLOFFS]
    scenes += [(f"sp_{sp}.rti", exponent_scene(sp), {}) for sp in EXPONENTS]
    scenes += [(f"{name}.rti", lines, objs) for name, (lines, objs) in sorted(refraction_scenes().items())]
    rng = np.random.default_rng(10)
    for name, lines, objs in scenes:
        sc, path = write_scene(pkg, tmp_path, name, lines, objs)
        href = live_reference.load(path)
        org, direction = oracle.camera_rays(sc.flat, W_AX, H_AX, np.arange(W_AX * H_AX))
        g0, _, _, p0, _ = oracle.cast_rays(sc.flat, org, direction)
        org2 = np.where((g0 >= 0)[:, None], p0, org)
        dir2 = rng.normal(size=org.shape)
        orgs, dirs = np.concatenate([org, org2]), np.concatenate([direction, dir2])
        for inside in (0, 1):
            fi = np.full(orgs.shape[0], inside, np.uint8)
            a = oracle.trace_rays(sc.flat, orgs, dirs, 4, fi)
            b = live_reference.trace_rays(href, orgs, dirs, 4, fi)
            assert np.array_equal(a, b, equal_nan=True), name
            assert np.array_equal(np.signbit(a), np.signbit(b)), name
