"""The FP32 culling steps at large scene coordinates, checked against the FP64 oracle.

Two FP32 shortcuts skip exact FP64 work: the LBVH slab test and the bounding-sphere pre-test
in front of every exact sphere test.  Both must be conservative, i.e. only skip what the exact
test would reject, wherever the scene sits.  Their rounding grows with the distance from the
world origin, not with the size of what is tested, so every scene here is also moved away from
the origin: one `xft` ahead of the scene and again after every `xfz` (the camera and the lights
take the transform too), by an offset with mixed signs and no zero component.

The sphere pre-test runs on the brute-force path (RT_FLAG_BRUTE_FORCE) as well, so a
BVH-vs-brute-force comparison cannot catch it erring; every case compares with the oracle
(FP64, no culling), and also BVH with brute force.
"""
import re

import numpy as np
import pytest

from conftest import GOLDEN, scene_path
from test_gpu_parity import SCENES

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-9
DIRECTION = (0.83, -0.47, 0.31)
OBJ = re.compile(r'^(\s*)obj\s+"?([^"\s]+)"?')


def offset(T):
    """T * DIRECTION, rounded to whole units (exact in the .rti text, and axis-parallel camera rays stay exact)."""
    return np.array([float(round(T * c)) for c in DIRECTION])


def num(x):
    return repr(float(x))


def vec(v):
    return " ".join(num(x) for x in v)


def moved(text, T, scale=None, base=GOLDEN / "inputs"):
    """The scene `text` translated by offset(T) (after a uniform `scale` about the origin, if given):
    the transform goes first and after every `xfz`.  `obj` paths become absolute (relative ones are
    resolved against `base`, the directory of the scene they come from)."""
    head = [f"xft {vec(offset(T))}"] + ([f"xfs {num(scale)} {num(scale)} {num(scale)}"] if scale else [])
    out = list(head)
    for line in text.splitlines():
        m = OBJ.match(line)
        if m:
            p = m.group(2)
            line = f'{m.group(1)}obj "{p if p.startswith("/") else (base / p).resolve()}"'
        out.append(line)
        if line.split()[:1] == ["xfz"]:
            out.extend(head)
    return "\n".join(out) + "\n"


def load(pkg, tmp_path, text, name="scene.rti"):
    path = tmp_path / name
    path.write_text(text)
    return pkg.HostScene.load(path)


def unit(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1)[:, None]


def assert_cast_rays_match(pkg, gpu_renderer, oracle, sc, org, dirs, rev):
    """rt_cast_rays with and without the LBVH equals the oracle bit for bit; returns the oracle's answer."""
    og = oracle.cast_rays(sc.flat, org, dirs, rev)
    for flags in (0, pkg.RT_FLAG_BRUTE_FORCE):
        gg = gpu_renderer.cast_rays(org, dirs, rev, flags=flags)
        for k, what in enumerate(("geometry ids", "face ids", "distances", "points", "normals")):
            bad = ~(gg[k] == og[k]) if gg[k].ndim == 1 else ~(gg[k] == og[k]).all(axis=1)
            assert not bad.any(), (f"flags {flags}: {what} differ from the oracle on {int(bad.sum())} of {len(bad)} rays "
                                   f"(oracle hits there: {int((og[0][bad] >= 0).sum())}, GPU hits: {int((gg[0][bad] >= 0).sum())})")
    return og


def assert_render_matches(pkg, gpu_renderer, oracle, sc, w, h, depth):
    """Render with and without the LBVH: primary geometry/face ids, per-class ray counts and the FP64 frame
    equal the oracle's.  Returns the oracle's frame and primary ids."""
    gpu_renderer.upload(sc)
    o_rgb, o_geom, o_face, counts = oracle.render(sc.flat, w, h, depth)
    for flags in (0, pkg.RT_FLAG_BRUTE_FORCE):
        rgb = gpu_renderer.render(w, h, depth, flags=flags)
        st = gpu_renderer.stats()
        geom, face = gpu_renderer.primary_ids(w, h, flags=flags)
        assert np.array_equal(geom, o_geom), f"flags {flags}: {int((geom != o_geom).sum())} primary geometry ids differ"
        assert np.array_equal(face, o_face), f"flags {flags}: {int((face != o_face).sum())} primary face ids differ"
        got = [st["rays_primary"], st["rays_shadow"], st["rays_secondary"]]
        assert got == counts[:3], f"flags {flags}: ray counts {got} != oracle {counts[:3]}"
        err = float(np.abs(rgb - o_rgb).max())
        assert err <= FP64_TOL, f"flags {flags}: frame differs from the oracle by {err}"
    return o_rgb, o_geom


# ---- 1 and 5: clusters of spheres and ellipsoids, per ray --------------------------------------------------

SHAPES = {"r1e-3": 1e-3, "r0.05": 0.05, "r1": 1.0, "r50": 50.0, "ellipsoid": 1.0}
PLACEMENTS = {"flat": 3, "lbvh": 5}        # spheres per side of the grid: 27 stay in the flat list, 125 go into the LBVH


def cluster(shape, side, seed=184):
    """A jittered grid of side^3 spheres of similar size (radius r * [0.7, 1.3], spacing 3 r) around the origin;
    for "ellipsoid" each one under its own xfr and non-uniform xfs, the first one with a negative scale.
    Returns the .rti text, the centres, and the radii of bounding and of inscribed spheres (all before any move)."""
    rng = np.random.default_rng(seed)
    r = SHAPES[shape]
    lines = [f"cam 0 0 {num(40 * r)}  {num(-r)} {num(-r)} {num(38 * r)}  {num(r)} {num(-r)} {num(38 * r)}  "
             f"{num(-r)} {num(r)} {num(38 * r)}  {num(r)} {num(r)} {num(38 * r)}",
             f"ltp {num(30 * r)} {num(40 * r)} {num(50 * r)} 0.6 0.6 0.6", "lta 0.1 0.1 0.1",
             "mat 0.1 0.1 0.1  0.6 0.5 0.4  0.3 0.3 0.3 10  0.2 0.2 0.2"]
    idx = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
    centres = (idx - (side - 1) / 2) * 3 * r + rng.uniform(-0.3 * r, 0.3 * r, size=idx.shape)
    radii = r * rng.uniform(0.7, 1.3, len(idx))
    bounds, inner = radii.copy(), radii.copy()
    for i, (c, rad) in enumerate(zip(centres, radii)):
        if shape == "ellipsoid":
            s = rng.uniform(0.4, 1.6, 3)
            if i == 0:
                s[0] = -s[0]                          # det < 0: the normal flips, the bound uses |scale|
            bounds[i], inner[i] = rad * np.abs(s).max(), rad * np.abs(s).min()
            lines += ["xfz", f"xft {vec(c)}", f"xfr {vec(rng.uniform(-180, 180, 3))}", f"xfs {vec(s)}", f"sph 0 0 0 {num(rad)}"]
        else:
            lines.append(f"sph {vec(c)} {num(rad)}")
    return "\n".join(lines) + "\n", centres, bounds, inner


def check_sphere_rays(pkg, gpu_renderer, oracle, tmp_path, T, shape, placement, scale=None):
    text, centres, bounds, inner = cluster(shape, PLACEMENTS[placement])
    sc = load(pkg, tmp_path, moved(text, T, scale))
    gpu_renderer.upload(sc)
    node_bytes = gpu_renderer.device_bytes()[0]
    assert (node_bytes > 0) == (placement == "lbvh"), f"placement {placement}: LBVH node bytes {node_bytes}"
    s = scale or 1.0
    world = lambda p: offset(T) + s * p
    rng = np.random.default_rng(184)
    r = SHAPES[shape]
    lo = (centres - bounds[:, None]).min(0)
    hi = (centres + bounds[:, None]).max(0)
    # (a) origins 0.5-20 radii from the centre of the cluster, aimed at uniform points of its box: many graze
    n = 20000
    org_a = world((lo + hi) / 2 + unit(rng, n) * rng.uniform(0.5, 20, n)[:, None] * r)
    dir_a = world(rng.uniform(lo, hi, size=(n, 3))) - org_a
    g_a, _, _, p_a, _ = oracle.cast_rays(sc.flat, org_a, dir_a)
    assert (g_a >= 0).sum() >= n // 10, f"only {(g_a >= 0).sum()} of {n} rays hit"
    # (b) origins on the surfaces, random directions, either side of the surface
    org_b = p_a[g_a >= 0]
    dir_b = unit(rng, len(org_b))
    # (c) origins inside, looking for the surface from within
    org_c = world(centres + unit(rng, len(centres)) * 0.5 * inner[:, None])
    dir_c = unit(rng, len(org_c))
    org = np.concatenate([org_a, org_b, org_c])
    dirs = np.concatenate([dir_a, dir_b, dir_c])
    rev = np.concatenate([np.zeros(n), rng.integers(0, 2, len(org_b)), np.ones(len(org_c))]).astype(np.uint8)
    og = assert_cast_rays_match(pkg, gpu_renderer, oracle, sc, org, dirs, rev)
    hits_b = (og[0][n:n + len(org_b)] >= 0).sum()
    hits_c = (og[0][n + len(org_b):] >= 0).sum()
    assert hits_b >= len(org_b) // 10 and hits_c >= len(org_c) // 2, (hits_b, len(org_b), hits_c, len(org_c))


@pytest.mark.parametrize("placement", sorted(PLACEMENTS))
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("T", [0, 1e3, 1e4, 1e5, 1e6, 1e7])
def test_sphere_rays_match_the_oracle_far_from_the_origin(pkg, gpu_renderer, oracle, tmp_path, T, shape, placement):
    """Per ray, bit for bit: spheres of radius 1e-3 to 50 and ellipsoids (rotated, non-uniformly scaled, one
    mirrored), in the flat list and in the LBVH, seen from close by, from their surfaces and from inside."""
    check_sphere_rays(pkg, gpu_renderer, oracle, tmp_path, T, shape, placement)


@pytest.mark.parametrize("placement", sorted(PLACEMENTS))
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("T", [0, 1e5])
@pytest.mark.parametrize("scale", [1e-4, 1e4])
def test_sphere_rays_match_the_oracle_at_small_and_large_scales(pkg, gpu_renderer, oracle, tmp_path, scale, T, shape,
                                                               placement):
    """The same clusters scaled by 1e-4 and 1e4 about the origin before the move: spheres down to 1e-7 across, where
    the 1e-30 floors matter, and up to 5e5, where the relative margins do."""
    check_sphere_rays(pkg, gpu_renderer, oracle, tmp_path, T, shape, placement, scale)


# ---- 2: shadows (the any-hit path) --------------------------------------------------------------------------

SHADOW_SCENE = """\
cam 0 3 0  -0.4 2 0.3  0.4 2 0.3  -0.4 2 -0.3  0.4 2 -0.3
ltp 0.3 1.6 0.2 0.7 0.7 0.7
ltd 0.2 -1 0.1 0.4 0.4 0.4
lta 0.1 0.1 0.1
mat 0.1 0.1 0.1  0.8 0.8 0.8  0.2 0.2 0.2 8  0.1 0.1 0.1
tri -5 0 5  5 0 5  5 0 -5
tri -5 0 5  5 0 -5  -5 0 -5
mat 0.1 0.1 0.1  0.5 0.3 0.3  0.5 0.5 0.5 20  0.3 0.3 0.3
sph 0 1 0 0.05
"""


@pytest.mark.parametrize("T", [1e5, 1e6])
def test_shadows_of_a_small_sphere_far_from_the_origin(pkg, gpu_renderer, oracle, tmp_path, T):
    """Shadow rays leave the floor about 1 unit below a sphere of radius 0.05, towards a point light and a directional
    light: the occlusion test (any-hit) must see the sphere wherever the scene sits."""
    w, h, depth = 96, 72, 3
    sc = load(pkg, tmp_path, moved(SHADOW_SCENE, T))
    rgb, geom = assert_render_matches(pkg, gpu_renderer, oracle, sc, w, h, depth)
    # not vacuous: without the sphere, floor pixels change (its shadows are in the frame)
    bare = load(pkg, tmp_path, moved(SHADOW_SCENE.replace("sph 0 1 0 0.05\n", ""), T), "bare.rti")
    b_rgb, b_geom, _, _ = oracle.render(bare.flat, w, h, depth)
    floor = (geom >= 0) & (geom <= 1) & (b_geom == geom)
    changed = (np.abs(rgb - b_rgb).max(axis=2) > 1e-3) & floor
    assert changed.sum() >= 20, f"only {changed.sum()} floor pixels are shadowed by the sphere"


# ---- 3: shipped scenes, moved ---------------------------------------------------------------------------------

SPHERE_SCENES = sorted(n for n, p in SCENES.items() if re.search(r"^\s*sph\b", scene_path(p).read_text(), re.M)) + ["bunny4"]


@pytest.mark.parametrize("T", [1e5, 1e6])
@pytest.mark.parametrize("name", SPHERE_SCENES)
def test_shipped_scenes_far_from_the_origin(pkg, gpu_renderer, oracle, tmp_path, name, T):
    path = scene_path(SCENES[name])
    sc = load(pkg, tmp_path, moved(path.read_text(), T, base=path.parent))
    _, geom = assert_render_matches(pkg, gpu_renderer, oracle, sc, 64, 48, 6)
    # test.rti's camera sits inside its sphere of radius 50, which castRay only finds from outside: no primary ray
    # of it hits anything, in the reference's own frames too (tests/golden/ref/test_96x96.npz)
    assert (geom >= 0).any() == (name != "test")


# ---- 4: axis-parallel rays at |coordinates| ~ 1e9 --------------------------------------------------------------

AXIS_SCENE = """\
cam 0 0 12  -0.75 -0.5 8  0.75 -0.5 8  -0.75 0.5 8  0.75 0.5 8
ltp 4 6 10 0.6 0.6 0.6
ltd -1 -1 -2 0.3 0.3 0.3
lta 0.1 0.1 0.1
mat 0.1 0.1 0.1  0.6 0.5 0.3  0.5 0.5 0.5 10  0.3 0.3 0.3
obj "teapot.obj"
mat 0.1 0.1 0.1  0.3 0.4 0.6  0.3 0.3 0.3 10  0.2 0.2 0.2
"""


def test_axis_parallel_rays_at_large_coordinates(pkg, gpu_renderer, oracle, tmp_path):
    """Rays along +-x, +-y, +-z have exactly zero direction components, which the slab test clamps; at |coordinates|
    ~ 1e9 the clamped plane distances must stay finite.  A teapot (mesh LBVH) in front of 121 spheres (LBVH too),
    per ray and in a frame of odd width whose centre column looks exactly down -z."""
    T = 1e9
    xy = (np.stack(np.meshgrid(np.arange(11), np.arange(11), indexing="ij"), -1).reshape(-1, 2) - 5) * 0.6
    spheres = "".join(f"sph {num(x)} {num(y)} -2.0 0.25\n" for x, y in xy)
    sc = load(pkg, tmp_path, moved(AXIS_SCENE + spheres, T))
    gpu_renderer.upload(sc)
    assert gpu_renderer.device_bytes()[0] > 0
    rng = np.random.default_rng(9)
    n = 6 * 8000
    axes = np.concatenate([np.eye(3), -np.eye(3)])
    org = offset(T) + rng.uniform([-3.0, -2.5, -2.6], [3.0, 3.0, 2.0], size=(n, 3))
    dirs = np.repeat(axes, n // 6, axis=0)
    g, _, _, p, _ = oracle.cast_rays(sc.flat, org, dirs)
    hit = g >= 0
    # and from the hit points on the surfaces, along the axes again, on either side
    org2 = np.concatenate([org, p[hit]])
    dirs2 = np.concatenate([dirs, axes[rng.integers(0, 6, hit.sum())]])
    rev = np.concatenate([np.zeros(n), rng.integers(0, 2, hit.sum())]).astype(np.uint8)
    og = assert_cast_rays_match(pkg, gpu_renderer, oracle, sc, org2, dirs2, rev)
    for k in range(6):
        gk = og[0][k * (n // 6):(k + 1) * (n // 6)]
        assert (gk == 0).sum() >= 50 and (gk > 0).sum() >= 50, f"axis {k}: teapot hits {(gk == 0).sum()}, sphere hits {(gk > 0).sum()}"
    # odd width: the centre column's image-plane x is the eye's.  A power-of-two height keeps the row fractions
    # dyadic, so that x is exact in FP64 at these coordinates, and those rays have a direction x of exactly 0.
    w, h = 65, 64
    _, d = oracle.camera_rays(sc.flat, w, h, np.arange(w * h))
    assert (d.reshape(h, w, 3)[:, w // 2, 0] == 0).all()
    _, geom = assert_render_matches(pkg, gpu_renderer, oracle, sc, w, h, 3)
    assert (geom[:, w // 2] >= 0).sum() >= 10
