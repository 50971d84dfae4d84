"""Any-hit rays are traced over the occlusion tree (csrc/dev_accel.cuh trace_occlusion): 4-wide nodes collapsed from the
reference-built tree, walked in no particular order, with the reference's leaves under their own boxes.  That gives the
reference's occlusion answer bit for bit because of one claim, pinned here on the CPU: when a box passes the device's slab
test (box_geom, restated in test_slab_formulations.py), every box containing it passes too, with an entry distance no
larger.  So a triangle is tested by the reference's any-hit walk exactly when its own leaf's box passes.

The GPU tests compare ptrs_intersect_p (the occlusion walk) with the oracle, and renders in stats mode (every connect ray
over the reference tree) with ordinary renders (any-hit rays over the occlusion tree)."""
import numpy as np
import pytest

from test_slab_formulations import F, device_accept, reference_accept


def _nested_inputs(rng, n):
    special = np.array([0.0, -0.0, 1.0, -1.0, 0.5, 2.0, 1e-30, -1e-30, 1e30, -1e30, 3.0, -3.0, 1.0000001, 0.99999994, np.inf, -np.inf],
                       dtype=F)
    pick = lambda shape: np.where(rng.random(shape) < 0.5, special[rng.integers(0, special.size, shape)], rng.normal(size=shape).astype(F) * F(2.0)).astype(F)
    a, b = pick((n, 3)), pick((n, 3))
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    hi = np.where(rng.random((n, 3)) < 0.15, lo, hi)  # flat inner boxes
    # the outer box: each plane equal to the inner one (shared planes) or pushed outwards, up to infinity
    grow = lambda shape: np.where(rng.random(shape) < 0.4, F(0.0), np.abs(pick(shape))).astype(F)
    with np.errstate(invalid="ignore", over="ignore"):
        olo = np.minimum(lo, (lo - grow((n, 3))).astype(F))
        ohi = np.maximum(hi, (hi + grow((n, 3))).astype(F))
    olo = np.where(np.isnan(olo), lo, olo)  # inf - inf: keep the plane
    ohi = np.where(np.isnan(ohi), hi, ohi)
    planes = np.stack([lo, hi, olo, ohi])
    o = pick((n, 3))
    which = rng.integers(0, 6, (n, 3))  # origin on a plane of either box, or anywhere
    o = np.where(which < 4, np.take_along_axis(planes, np.minimum(which, 3)[None], 0)[0], o).astype(F)
    o = np.where(np.isinf(o), F(0.5), o)
    d = pick((n, 3))
    d = np.where(rng.random((n, 3)) < 0.01, F(np.nan), d).astype(F)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = (F(1.0) / d).astype(F)  # +-inf for d = +-0
    t_ray = np.where(rng.random(n) < 0.3, F(np.inf), np.abs(pick((n,)))).astype(F)
    return (lo, hi), (olo, ohi), o, inv, t_ray


def test_a_box_accepted_implies_every_enclosing_box_accepted():
    rng = np.random.default_rng(7)
    total = accepted = nan_rays = 0
    for _ in range(40):
        (lo, hi), (olo, ohi), o, inv, t_ray = _nested_inputs(rng, 250_000)
        assert np.all(olo <= lo) and np.all(ohi >= hi)
        inner, t_inner = device_accept(lo, hi, o, inv, t_ray)
        outer, t_outer = device_accept(olo, ohi, o, inv, t_ray)
        bad = inner & ~outer
        assert not bad.any(), f"{np.count_nonzero(bad)} inner boxes accepted whose enclosing box is rejected"
        assert np.all(t_outer[inner] <= t_inner[inner])
        # the same through the reference's compare-and-select chain
        ref_inner, _ = reference_accept(lo, hi, o, inv, t_ray)
        ref_outer, _ = reference_accept(olo, ohi, o, inv, t_ray)
        assert not (ref_inner & ~ref_outer).any()
        total += inner.size
        accepted += int(np.count_nonzero(inner))
        nan_rays += int(np.count_nonzero(np.isnan(inv).any(axis=1) | np.isinf(inv).any(axis=1)))
    assert total >= 10_000_000 and accepted > total // 50 and nan_rays > total // 20


def _segments(host, oracle, flat, rays):
    """The rays as segments ending at 0.5x, 1x and 1.5x of the oracle's closest hit (rays that miss keep t_max)."""
    o, _ = oracle.intersect(flat, rays)
    hit = o["prim"] >= 0
    out = []
    for f in (0.5, 1.0, 1.5):
        r = rays.copy()
        r["t_max"][hit] = (o["t"][hit] * np.float32(f)).astype(np.float32)
        out.append(r)
    return np.concatenate(out)


def _edge_rays(host, flat):
    v = flat.prim_vertices().reshape(-1, 3)[:30000]
    bmin, bmax = (np.asarray(b, dtype=np.float32) for b in flat.world_bound())
    edge = np.zeros(len(v) + 7, dtype=host.RAY_DTYPE)
    c = (bmin + bmax) * np.float32(0.5)
    edge["o"][: len(v)] = c + (bmax - bmin) * np.float32(0.37)
    edge["d"][: len(v)] = v - edge["o"][: len(v)]  # through vertices and along edges
    edge["o"][len(v):] = c
    edge["d"][len(v):] = [[0, 0, -1], [0, 0, 1], [1, 0, 0], [0, 1, 0], [0, -1, 0], [-1, 0, 0], [1e-20, 0, -1]]  # axis-parallel
    edge["t_max"] = np.inf
    return edge


def _check_occlusion(gpu, host, oracle, flat, cam, seed):
    scene = gpu.RenderScene(flat)
    bmin, bmax = flat.world_bound()
    sets = {"coherent": host.coherent_rays(cam, 128), "incoherent": host.incoherent_rays(bmin, bmax, seed, 30000), "edge": _edge_rays(host, flat)}
    for name, rays in sets.items():
        for r in (rays, _segments(host, oracle, flat, rays)):
            g = scene.intersect_p(r)
            o, _ = oracle.intersect_p(flat, r)
            assert np.array_equal(g, o), f"{name}: {np.count_nonzero(g != o)} of {len(r)} occlusion answers differ"
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["cornell", "field_small", "terrain_small", "atrium_small"])
def test_occlusion_tree_answers_equal_the_oracle(gpu, host, oracle, request, scene_name):
    flat, cam = request.getfixturevalue(scene_name)
    _check_occlusion(gpu, host, oracle, flat, cam, 11)


@pytest.mark.gpu
def test_occlusion_tree_answers_equal_the_oracle_under_an_alpha_mask(gpu, host, oracle, tmp_path):
    from test_gltf_import import write_gltf

    path, _ = write_gltf(host, tmp_path, "glb")
    flat, cam = host.import_scene(path, res=(96, 64), default_lights=True)
    _check_occlusion(gpu, host, oracle, flat, cam, 12)


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name,spp,depth", [("cornell_env", 16, 15), ("field_small", 8, 8), ("atrium_small", 8, 8)])
def test_render_over_the_occlusion_tree_equals_the_reference_walk(gpu, request, scene_name, spp, depth):
    """Per-path radiance bit for bit; the film to the last few ulps, since film sums are float atomics in no fixed order."""
    flat, cam = request.getfixturevalue(scene_name)
    scene = gpu.RenderScene(flat)
    rng = np.random.default_rng(5)
    n = 20000
    pixels = np.stack([rng.integers(0, cam.width, n), rng.integers(0, cam.height, n)], axis=1)
    samples = rng.integers(0, spp, n)
    radiance, films = [], []
    for stats_mode in (True, False):  # stats mode: every connect ray over the reference tree
        scene.set_stats_mode(stats_mode)
        integ = gpu.PathIntegrator(gpu.SamplerBuilder(spp), max_depth=depth)
        integ.preprocess(scene)
        radiance.append(scene.path_radiance(cam, integ.params, pixels, samples))
        film = gpu.Film(cam.width, cam.height)
        integ.render(cam, scene, film)
        films.append(film.download())
    assert np.array_equal(radiance[0], radiance[1])
    assert np.count_nonzero(radiance[0]) > 0
    assert np.allclose(films[0], films[1], rtol=2e-5, atol=1e-6)
    scene.close()
