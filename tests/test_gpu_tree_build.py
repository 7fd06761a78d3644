"""LBVH build on the GPU: treelet restructuring and the least-cost 4-wide collapse (csrc/rt_bvh.cu).

The tree only culls (every hit is decided by the exact FP64 test), so whatever the build does, a render through the
LBVH must equal the brute-force render: ids, ray counts, FP64 frame and per-ray cast_rays.  The build must also be
deterministic (ranks of a multi-GPU job each build their own tree) and must not refuse a scene whose optimised tree is
deeper than the traversal stack when the plain Karras tree fits."""
import numpy as np
import pytest

from conftest import scene_path

pytestmark = pytest.mark.gpu
FP64_TOL = 1e-9
CAM = "cam 0 2 30  -10 -8 10  10 -8 10  -10 12 10  10 12 10\n"
HEAD = CAM + "lta 0.1 0.1 0.1\nltp 10 20 30 1 1 1\nltd -0.3 -1 -0.2 0.5 0.5 0.5\n"
MAT = "mat 0.1 0.1 0.1 0.6 0.5 0.4 0.3 0.3 0.3 10 0.3 0.3 0.3\n"


def _write_grid_obj(path, n, half, y, jitter=0.0, seed=0):
    """n x n quads (2n^2 triangles) covering [-half, half]^2 at height y (+ a deterministic height jitter)."""
    rng = np.random.default_rng(seed)
    xs = np.linspace(-half, half, n + 1)
    lines = []
    for j in range(n + 1):
        for i in range(n + 1):
            lines.append(f"v {xs[i]:.6f} {y + jitter * rng.uniform(-1, 1):.6f} {xs[j]:.6f}")
    for j in range(n):
        for i in range(n):
            a = j * (n + 1) + i + 1
            b, c, d = a + 1, a + n + 1, a + n + 2
            lines.append(f"f {a} {b} {d}")
            lines.append(f"f {a} {d} {c}")
    path.write_text("\n".join(lines) + "\n")


def _scene(pkg, tmp_path, name, text):
    rti = tmp_path / name
    rti.write_text(text)
    return pkg.HostScene.load(rti)


def _assert_matches_brute_force(pkg, r, sc, w=96, h=72, depth=4, seed=3):
    r.upload(sc)
    a = r.render(w, h, depth)
    sa = r.stats()
    b = r.render(w, h, depth, flags=pkg.RT_FLAG_BRUTE_FORCE)
    sb = r.stats()
    for k in ("rays_primary", "rays_shadow", "rays_secondary", "hits"):
        assert sa[k] == sb[k], k
    assert np.abs(a - b).max() <= FP64_TOL
    ga, fa = r.primary_ids(w, h)
    gb, fb = r.primary_ids(w, h, flags=pkg.RT_FLAG_BRUTE_FORCE)
    assert np.array_equal(ga, gb) and np.array_equal(fa, fb)
    rng = np.random.default_rng(seed)
    n = 20000
    org = rng.uniform(-40, 40, size=(n, 3))
    tgt = rng.uniform(-6, 6, size=(n, 3))
    g1 = r.cast_rays(org, tgt - org)
    g2 = r.cast_rays(org, tgt - org, flags=pkg.RT_FLAG_BRUTE_FORCE)
    for x, y in zip(g1, g2):
        assert np.array_equal(x, y)
    return sa


def test_mixed_triangle_sizes(pkg, gpu_renderer, tmp_path):
    """The teapot's small faces next to a floor mesh of faces thousands of times larger, in ONE mesh group: treelets
    mix leaves whose areas differ by orders of magnitude."""
    floor = tmp_path / "floor.obj"
    _write_grid_obj(floor, 24, 400.0, -1.0, jitter=0.5)
    text = HEAD + MAT + f'obj "{floor}"\n' + MAT + f'obj "{scene_path("inputs/teapot.obj")}"\n'
    st = _assert_matches_brute_force(pkg, gpu_renderer, _scene(pkg, tmp_path, "mixed.rti", text))
    assert st["rays_secondary"] > 0


@pytest.mark.parametrize("faces", [3, 4, 5, 6])
def test_groups_smaller_than_a_treelet(pkg, gpu_renderer, tmp_path, faces):
    """Meshes of 3..6 faces: the only treelet is smaller than its maximum of seven leaves."""
    mesh = tmp_path / "small.obj"
    verts = [f"v {-6 + 3 * k} {(-1) ** k * 2} {-k}" for k in range(faces + 2)]
    tris = [f"f {k + 1} {k + 2} {k + 3}" for k in range(faces)]
    mesh.write_text("\n".join(verts + tris) + "\n")
    _assert_matches_brute_force(pkg, gpu_renderer, _scene(pkg, tmp_path, f"small{faces}.rti", HEAD + MAT + f'obj "{mesh}"\n'))


def test_duplicate_centroids_in_meshes_and_spheres(pkg, gpu_renderer, tmp_path):
    """Every face of a mesh repeated four times (equal boxes, equal Morton codes) and 100 concentric spheres (equal
    centroids, nested boxes): zero-cost ties in the treelet and collapse choices."""
    mesh = tmp_path / "dup.obj"
    _write_grid_obj(mesh, 6, 8.0, -3.0, jitter=1.0, seed=5)
    lines = mesh.read_text().splitlines()
    faces = [ln for ln in lines if ln.startswith("f ")]
    mesh.write_text("\n".join([ln for ln in lines if ln.startswith("v ")] + faces * 4) + "\n")
    spheres = "".join(f"sph 0 4 0 {0.3 + 0.03 * i}\n" for i in range(100))
    text = HEAD + MAT + f'obj "{mesh}"\n' + MAT + spheres
    _assert_matches_brute_force(pkg, gpu_renderer, _scene(pkg, tmp_path, "dup.rti", text))


# Kernel launches of rt_scene_upload for a scene of spheres only (one LBVH group, no super node):
# k_scatter_codes, k_prim_bounds, k_morton, 4 radix passes x 4 kernels.
UPLOAD_LAUNCHES = 3 + 16
# The group's optimised attempt: k_karras, k_refit, 2 x k_treelet, k_collapse_cost; accepted, it adds one
# k_choose_children per wide level and k_pack_wide.  Rejected as too deep, the group is built again: k_karras,
# k_refit, k_depth, k_pack_wide.
OPTIMISED_ATTEMPT = 5
FALLBACK = 4


def test_deep_optimised_tree_falls_back(pkg, gpu_renderer, tmp_path):
    """A dense cluster in a wide scene: 5000 concentric spheres share one Morton code, so the Karras tree over them
    is a balanced index split 13 levels deep, but their boxes are nested and the least-area tree over nested boxes is
    a chain: the optimised wide tree is deeper than the traversal stack.  The build must fall back to the Karras tree
    with the even-depth collapse instead of refusing the scene, and render what brute force renders."""
    cluster = "".join(f"sph 0 0 0 {0.5 + 0.001 * i}\n" for i in range(5000))
    ring = "".join(f"sph {-40 + 2 * i} -9 -20 0.7\n" for i in range(40))     # spreads the centroids: one code
    sc = _scene(pkg, tmp_path, "cluster.rti", HEAD + MAT + cluster + ring)
    gpu_renderer.upload(sc)
    # an accepted optimised tree over 5040 leaves has at least 7 wide levels, so it cannot give this count
    assert gpu_renderer.stats()["kernel_launches"] == UPLOAD_LAUNCHES + OPTIMISED_ATTEMPT + FALLBACK
    _assert_matches_brute_force(pkg, gpu_renderer, sc, w=64, h=48, depth=3)


def test_shallow_tree_keeps_the_optimised_build(pkg, gpu_renderer, tmp_path):
    """The same number of spheres on a grid: the optimised tree fits the stack and is kept (one k_choose_children
    per wide level, no second build), and renders what brute force renders."""
    grid = "".join(f"sph {-12 + 0.35 * (i % 72)} {-12 + 0.35 * (i // 72)} {-(i % 7)} 0.15\n" for i in range(5040))
    sc = _scene(pkg, tmp_path, "grid.rti", HEAD + MAT + grid)
    gpu_renderer.upload(sc)
    wide_levels = gpu_renderer.stats()["kernel_launches"] - UPLOAD_LAUNCHES - OPTIMISED_ATTEMPT - 1
    assert 7 <= wide_levels <= 36, wide_levels
    _assert_matches_brute_force(pkg, gpu_renderer, sc, w=64, h=48, depth=3)


@pytest.fixture()
def same_device_multi(monkeypatch):
    import torch
    if torch.cuda.device_count() < 2:
        monkeypatch.setenv("RT_MULTI_SAME_DEVICE", "1")


def test_build_is_deterministic(pkg, same_device_multi):
    """The same scene uploaded twice, into a second context, and rendered over two sub-contexts does the same
    counted work: the node array depends on the primitives only."""
    sc = pkg.HostScene.load(scene_path("excess_inputs/bunny4.rti"))
    w, h, depth = 320, 180, 4
    counts = []
    r1, r2 = pkg.Renderer(0), pkg.Renderer(0)
    try:
        for r in (r1, r1, r2):
            r.upload(sc)
            r.render(w, h, depth, flags=pkg.RT_FLAG_COUNT_WORK)
            st = r.stats()
            counts.append((list(st["nodes_fetched"]), list(st["tris_tested"])))
        r2.render(w, h, depth, flags=pkg.RT_FLAG_COUNT_WORK, n_gpus=2)
        st = r2.stats()
        counts.append((list(st["nodes_fetched"]), list(st["tris_tested"])))
    finally:
        r1.close()
        r2.close()
    assert counts[0][0][0] > 0
    assert all(c == counts[0] for c in counts), counts
