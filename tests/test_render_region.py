"""Rendering a rectangle of sample positions (ptrs_render_region, ptrs_multi_render_region) and the helper that turns a
pixel crop into the sample rectangle that completes it (ptrs_film_region_sample_rect).

The Sobol index of a sample is a function of (position, sample number) relative to the full sample bounds
(sampler/sobol.rs:169-175), so a rectangle traces exactly the paths the full render traces there; what the helper has
to get right is the film splat's footprint, which the CPU tests below restate in numpy float32."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ONE_MINUS_EPS = np.float32(1.0) - np.float32(2.0 ** -24)  # OneMinusEpsilon: the largest jitter a sample can have
RADII = (0.4, 0.5, 1.0, 1.5, 2.0, 2.5, 3.3, 7.0)
TOL = dict(rtol=2e-5, atol=1e-6)  # float atomics: same terms, another summation order


# ---- numpy restatement of accumulate_kernel's footprint (k_misc.cu) -------------------------------------------------
def _f32(v):
    return np.asarray(v, dtype=np.float32)


def sample_bounds_1d(size, r):
    """Film::get_sample_bounds along one axis (film.rs:174-185): [floor(0.5 - r), ceil(size - 0.5 + r))."""
    r = _f32(r)
    return int(np.floor(_f32(0.5) - r)), int(np.ceil(_f32(size) - _f32(0.5) + r))


def footprint_1d(fx, r, size):
    """Pixels [p0, p1) the kernel splats a sample with film coordinate fx onto: dx = fx - 0.5, ceil(dx - r),
    floor(dx + r) + 1, clamped to the film."""
    dx = _f32(fx) - _f32(0.5)
    p0 = np.ceil(dx - _f32(r)).astype(np.int64)
    p1 = (np.floor(dx + _f32(r)) + _f32(1.0)).astype(np.int64)
    return np.maximum(p0, 0), np.minimum(p1, size)


def position_fx(s, jitter):
    """film coordinates fx = float(s) + u of a sample at position s for each jitter u (as get_camera_sample rounds them)"""
    return _f32(s)[:, None] + _f32(jitter)[None, :]


def want_sample_range_1d(size, r, a, b, rng):
    """The smallest range of positions holding every sample that reaches a pixel of [a, b): every position's fx at its
    two ends (s and the clamped s + 1 - eps, SURVEY quirk 1) and at random jitters in between."""
    lo, hi = sample_bounds_1d(size, r)
    s = np.arange(lo, hi)
    jitter = np.concatenate([_f32([0.0, ONE_MINUS_EPS]), np.minimum(rng.random(6, dtype=np.float32), ONE_MINUS_EPS)])
    p0, p1 = footprint_1d(position_fx(s, jitter), r, size)
    reaches = (np.maximum(p0, a) < np.minimum(p1, b)).any(axis=1)
    hit = s[reaches]
    return int(hit.min()), int(hit.max()) + 1


def touched_1d(size, r, s0, s1):
    """film pixels a rectangle of positions [s0, s1) can change along one axis"""
    p0, _ = footprint_1d(_f32([s0]), r, size)
    _, p1 = footprint_1d(_f32([s1 - 1]) + ONE_MINUS_EPS, r, size)
    return int(p0[0]), int(p1[0])


def touched_mask(w, h, r, rect):
    x0, x1 = touched_1d(w, r[0], rect[0], rect[2])
    y0, y1 = touched_1d(h, r[1], rect[1], rect[3])
    m = np.zeros((h, w), dtype=bool)
    m[y0:y1, x0:x1] = True
    return m


def region_sample_rect(lib, w, h, r, pixel_rect):
    """(status, sample rectangle) of ptrs_film_region_sample_rect"""
    out = (C.c_int32 * 4)()
    rc = lib.ptrs_film_region_sample_rect(w, h, (C.c_float * 2)(*r), (C.c_int32 * 4)(*pixel_rect), out)
    return rc, tuple(out)


@pytest.fixture(scope="module")
def lib():
    import pathtracer_rs_b200.gpu as g

    return g.lib()  # host arithmetic: loads and answers without a device


# ---- CPU: the helper -----------------------------------------------------------------------------------------------
def _pixel_rects(w, h, rng, n_random=12):
    rects = [(0, 0, w, h), (0, 0, 1, 1), (w - 1, h - 1, w, h), (0, 3 % h, w, min(h, 3 % h + 2)), (w - 2, 0, w, h),
             (0, h - 1, w, h), (w // 2, h // 2, w // 2 + 1, h // 2 + 1)]
    for _ in range(n_random):
        x0, y0 = int(rng.integers(0, w)), int(rng.integers(0, h))
        rects.append((x0, y0, int(rng.integers(x0 + 1, w + 1)), int(rng.integers(y0 + 1, h + 1))))
    return rects


@pytest.mark.parametrize("radius", RADII)
def test_helper_matches_the_splat_footprint(lib, radius):
    rng = np.random.default_rng(int(radius * 10))
    for w, h in ((96, 54), (7, 3), (4100, 33)):  # 4100: positions where s + 1 - eps rounds to s + 1
        for rect in _pixel_rects(w, h, rng):
            for r in ((radius, radius), (radius, 2.0)):
                rc, got = region_sample_rect(lib, w, h, r, rect)
                assert rc == 0, (w, h, r, rect)
                wx = want_sample_range_1d(w, r[0], rect[0], rect[2], rng)
                wy = want_sample_range_1d(h, r[1], rect[1], rect[3], rng)
                assert got == (wx[0], wy[0], wx[1], wy[1]), (w, h, r, rect, got)


def test_helper_at_radius_two_grows_the_crop_by_two(lib):
    rng = np.random.default_rng(2)
    w, h = 96, 54
    for rect in _pixel_rects(w, h, rng, n_random=40):
        rc, got = region_sample_rect(lib, w, h, (2.0, 2.0), rect)
        assert rc == 0
        assert got == (max(rect[0] - 2, -2), max(rect[1] - 2, -2), min(rect[2] + 2, w + 2), min(rect[3] + 2, h + 2))
    assert region_sample_rect(lib, w, h, (2.0, 2.0), (0, 0, w, h))[1] == (-2, -2, w + 2, h + 2)  # the sample bounds


def test_helper_refuses_invalid_arguments(lib):
    w, h, r, ok = 96, 54, (C.c_float * 2)(2.0, 2.0), (C.c_int32 * 4)(0, 0, 4, 4)
    out = (C.c_int32 * 4)()
    assert lib.ptrs_film_region_sample_rect(w, h, r, ok, out) == 0
    assert lib.ptrs_film_region_sample_rect(w, h, None, ok, out) == -1
    assert lib.ptrs_film_region_sample_rect(w, h, r, None, out) == -1
    assert lib.ptrs_film_region_sample_rect(w, h, r, ok, None) == -1
    for bad in ((4, 0, 4, 4), (0, 4, 4, 4), (5, 0, 4, 4), (0, 0, 4, -1), (-1, 0, 4, 4), (0, -2, 4, 4), (0, 0, w + 1, 4),
                (0, 0, 4, h + 1), (w, 0, w + 1, 4)):
        assert region_sample_rect(lib, w, h, (2.0, 2.0), bad)[0] == -1, bad
    for radius in ((0.0, 2.0), (2.0, -1.0), (float("nan"), 2.0), (float("inf"), 2.0), (2.0, 4096.0)):
        assert region_sample_rect(lib, w, h, radius, (0, 0, 4, 4))[0] == -1, radius
    for size in ((0, 54), (96, 0), (-3, 54)):
        assert region_sample_rect(lib, size[0], size[1], (2.0, 2.0), (0, 0, 1, 1))[0] == -1, size


# ---- GPU ------------------------------------------------------------------------------------------------------------
SCENES = [("cornell", 15), ("cornell_env", 15), ("field_small", 8), ("atrium_small", 8)]


def _integrator(gpu, spp, depth, radius):
    integ = gpu.PathIntegrator(gpu.SamplerBuilder(spp), max_depth=depth)
    integ.params.filter_radius[0] = integ.params.filter_radius[1] = radius
    return integ


def _render(gpu, integ, cam, scene, **kw):
    film = gpu.Film(cam.width, cam.height)
    stats = integ.render(cam, scene, film, **kw)
    return film.download(), stats


def _complement(bounds, rect):
    """rectangles that, with `rect`, partition the sample bounds"""
    bx0, by0, bx1, by1 = bounds
    x0, y0, x1, y1 = rect
    parts = [(bx0, by0, x0, by1), (x1, by0, bx1, by1), (x0, by0, x1, y0), (x0, y1, x1, by1)]
    return [p for p in parts if p[0] < p[2] and p[1] < p[3]]


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name,depth", SCENES)
def test_crop_is_bit_exact_with_one_contribution_per_pixel(gpu, request, lib, scene_name, depth):
    """spp 1 and filter radius 0.4: every pixel receives at most one sample, so the crop's pixels are the full
    render's bit for bit, and nothing outside the rectangle's footprint is written."""
    flat, cam = request.getfixturevalue(scene_name)
    w, h = cam.width, cam.height
    scene = gpu.RenderScene(flat)
    integ = _integrator(gpu, 1, depth, 0.4)
    full, st_full = _render(gpu, integ, cam, scene)
    for crop in ((11, 7, 53, 31), (0, 0, 9, 5), (w - 13, h - 6, w, h), (w // 2, h // 2, w // 2 + 1, h // 2 + 1)):
        rc, rect = region_sample_rect(lib, w, h, (0.4, 0.4), crop)
        assert rc == 0
        film, st = _render(gpu, integ, cam, scene, region=rect)
        x0, y0, x1, y1 = crop
        assert np.array_equal(film[y0:y1, x0:x1], full[y0:y1, x0:x1]), (scene_name, crop)
        assert not film[~touched_mask(w, h, (0.4, 0.4), rect)].any(), (scene_name, crop)
        assert st["camera_paths"] == (rect[2] - rect[0]) * (rect[3] - rect[1])
    bx0, by0, bx1, by1 = gpu.Film(w, h).get_sample_bounds((0.4, 0.4))
    assert st_full["camera_paths"] == (bx1 - bx0) * (by1 - by0)
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name,depth", SCENES)
def test_crop_at_the_default_filter(gpu, request, lib, scene_name, depth):
    """radius 2, 8 spp: crops (interior, at each border, 1x1, the whole image) equal the full render's pixels up to
    summation order; a rectangle inside the negative border [-2, 0) writes only the pixels it reaches; every rectangle
    plus the rest of the sample bounds sums to the full film."""
    flat, cam = request.getfixturevalue(scene_name)
    w, h = cam.width, cam.height
    scene = gpu.RenderScene(flat)
    integ = _integrator(gpu, 8, depth, 2.0)
    full, st_full = _render(gpu, integ, cam, scene)
    bounds = gpu.Film(w, h).get_sample_bounds((2.0, 2.0))
    crops = [(13, 9, 45, 30), (0, 10, 17, 29), (20, 0, 41, 11), (w - 19, 5, w, 40), (6, h - 7, 50, h), (30, 20, 31, 21), (0, 0, w, h)]
    rects = [region_sample_rect(lib, w, h, (2.0, 2.0), c)[1] for c in crops] + [(-2, 10, 0, 30), (-2, -2, 0, 0)]
    assert rects[len(crops) - 1] == bounds  # the whole image needs the whole sample bounds
    for i, rect in enumerate(rects):
        film, st = _render(gpu, integ, cam, scene, region=rect)
        assert st["camera_paths"] == (rect[2] - rect[0]) * (rect[3] - rect[1]) * 8
        touched = touched_mask(w, h, (2.0, 2.0), rect)
        assert not film[~touched].any(), (scene_name, rect)
        if i < len(crops):
            x0, y0, x1, y1 = crops[i]
            assert np.allclose(film[y0:y1, x0:x1], full[y0:y1, x0:x1], **TOL), (scene_name, crops[i])
        else:
            assert (film[touched][:, 3] > 0).all(), (scene_name, rect)  # the border positions do reach these pixels
        rest = gpu.Film(w, h)
        for part in _complement(bounds, rect):
            integ.render(cam, scene, rest, region=part)
        assert np.allclose(film + rest.download(), full, **TOL), (scene_name, rect)
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name,depth", SCENES)
def test_uneven_tiles_partition_the_full_render(gpu, request, scene_name, depth):
    flat, cam = request.getfixturevalue(scene_name)
    w, h = cam.width, cam.height
    scene = gpu.RenderScene(flat)
    integ = _integrator(gpu, 4, depth, 2.0)
    full, st_full = _render(gpu, integ, cam, scene)
    bx0, by0, bx1, by1 = gpu.Film(w, h).get_sample_bounds((2.0, 2.0))

    def cuts(lo, hi, steps):  # tile sides 13, 29, 7, ... : not multiples of the 8x4 blocks
        out, k = [lo], 0
        while out[-1] < hi:
            out.append(min(hi, out[-1] + steps[k % len(steps)]))
            k += 1
        return out

    xs, ys = cuts(bx0, bx1, (13, 29, 7, 21)), cuts(by0, by1, (5, 19, 11, 3))
    film = gpu.Film(w, h)
    paths = 0
    for y0, y1 in zip(ys, ys[1:]):
        for x0, x1 in zip(xs, xs[1:]):
            paths += integ.render(cam, scene, film, region=(x0, y0, x1, y1))["camera_paths"]
    assert paths == st_full["camera_paths"]
    assert np.allclose(film.download(), full, **TOL)
    scene.close()


@pytest.mark.gpu
def test_region_composes_with_sample_selection(gpu, cornell_env):
    flat, cam = cornell_env
    scene = gpu.RenderScene(flat)
    integ = _integrator(gpu, 8, 8, 2.0)
    rect = (7, 3, 50, 41)
    whole, st = _render(gpu, integ, cam, scene, region=rect)
    assert st["camera_paths"] == 43 * 38 * 8
    parts = gpu.Film(cam.width, cam.height)
    n = integ.render(cam, scene, parts, region=rect, sample_range=(0, 3))["camera_paths"]
    n += integ.render(cam, scene, parts, region=rect, sample_range=(3, 8))["camera_paths"]
    assert n == st["camera_paths"] and np.allclose(parts.download(), whole, **TOL)
    shards = gpu.Film(cam.width, cam.height)
    n = integ.render(cam, scene, shards, region=rect, sample_stride=(3, 0))["camera_paths"]
    n += integ.render(cam, scene, shards, region=rect, sample_stride=(3, 1))["camera_paths"]
    n += integ.render(cam, scene, shards, region=rect, sample_stride=(3, 2))["camera_paths"]
    assert n == st["camera_paths"] and np.allclose(shards.download(), whole, **TOL)
    mixed, st_mixed = _render(gpu, integ, cam, scene, region=rect, sample_range=(2, 7), sample_stride=(2, 1))
    assert st_mixed["camera_paths"] == 43 * 38 * 2  # s = 3, 5
    ref = gpu.Film(cam.width, cam.height)
    integ.render(cam, scene, ref, region=rect, sample_range=(3, 4))
    integ.render(cam, scene, ref, region=rect, sample_range=(5, 6))
    assert np.allclose(mixed, ref.download(), **TOL)
    fresh = gpu.RenderScene(flat)  # a scene's workspace only grows: small batches need one that has not rendered yet
    for batch in (1000, 4096):  # batches that split the rectangle's 8x4 blocks across calls
        integ.params.paths_per_batch = batch
        small, st_small = _render(gpu, integ, cam, fresh, region=rect)
        assert st_small["batches"] > 1 and st_small["camera_paths"] == st["camera_paths"]
        assert st_small["extension_rays"] == st["extension_rays"]
        assert np.allclose(small, whole, **TOL)
    integ.params.paths_per_batch = 0
    fresh.close()
    exact_full, _ = _render(gpu, integ, cam, scene, exact_shading=True)
    exact, _ = _render(gpu, integ, cam, scene, region=rect, exact_shading=True)
    inner = (slice(rect[1] + 2, rect[3] - 2), slice(rect[0] + 2, rect[2] - 2))  # pixels the rectangle completes
    assert np.allclose(exact[inner], exact_full[inner], **TOL)
    assert not np.array_equal(exact, whole)  # the parity build shades with other arithmetic
    scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name,depth", SCENES)
def test_region_of_the_whole_sample_bounds_is_ptrs_render(gpu, request, scene_name, depth):
    flat, cam = request.getfixturevalue(scene_name)
    scene = gpu.RenderScene(flat)
    integ = _integrator(gpu, 4, depth, 2.0)
    full, st_full = _render(gpu, integ, cam, scene)
    region, st = _render(gpu, integ, cam, scene, region=gpu.Film(cam.width, cam.height).get_sample_bounds((2.0, 2.0)))
    for k in ("camera_paths", "extension_rays", "shadow_rays", "mis_rays", "batches"):
        assert st[k] == st_full[k], k
    assert np.allclose(region, full, **TOL)
    scene.close()


@pytest.mark.gpu
def test_render_region_refuses_invalid_rectangles(gpu, cornell):
    flat, cam = cornell
    w, h = cam.width, cam.height
    scene = gpu.RenderScene(flat)
    integ = _integrator(gpu, 4, 4, 2.0)
    film = gpu.Film(w, h)
    for bad in ((5, 5, 5, 9), (5, 5, 9, 5), (9, 5, 5, 9), (5, 9, 9, 5), (-3, 0, 4, 4), (0, -3, 4, 4), (0, 0, w + 3, 4),
                (0, 0, 4, h + 3), (-3, -3, w + 3, h + 3)):
        with pytest.raises(gpu.PtrsError) as e:
            integ.render(cam, scene, film, region=bad)
        assert e.value.code == -1, bad
    L = gpu.lib()
    p = integ.params
    assert L.ptrs_render_region(scene._h, C.byref(cam), C.byref(p), None, film._h, None) == -1
    rect = (C.c_int32 * 4)(0, 0, 4, 4)
    assert L.ptrs_render_region(None, C.byref(cam), C.byref(p), rect, film._h, None) == -1
    assert L.ptrs_render_region(scene._h, C.byref(cam), C.byref(p), rect, None, None) == -1
    other = gpu.Film(w + 1, h)  # the conditions of ptrs_render still apply
    assert L.ptrs_render_region(scene._h, C.byref(cam), C.byref(p), rect, other._h, None) == -1
    deep = gpu.PathIntegrator(gpu.SamplerBuilder(4), max_depth=500)
    with pytest.raises(gpu.PtrsError) as e:
        deep.render(cam, scene, film, region=(0, 0, 4, 4))
    assert e.value.code == -3
    assert not film.download().any()  # nothing was rendered by the refused calls
    scene.close()


@pytest.mark.gpu
def test_multi_render_region_equals_single_device_region(gpu, host, lib, cornell_env):
    flat, cam = cornell_env
    n = min(2, gpu.device_count())
    params = host.default_render_params(spp=16, max_depth=8)
    rc, rect = region_sample_rect(lib, cam.width, cam.height, (2.0, 2.0), (20, 10, 61, 47))
    assert rc == 0
    multi = gpu.MultiScene(flat, n)
    film, stats, ms = multi.render(cam, params, region=rect)
    scene = gpu.RenderScene(flat)
    integ = gpu.PathIntegrator(gpu.SamplerBuilder(16), max_depth=8)
    single, st = _render(gpu, integ, cam, scene, region=rect)
    assert sum(s["camera_paths"] for s in stats) == st["camera_paths"] == (rect[2] - rect[0]) * (rect[3] - rect[1]) * 16
    assert np.allclose(film[..., 3], single[..., 3], rtol=2e-5)
    assert np.allclose(film, single, rtol=2e-4, atol=1e-5 * float(single[..., :3].max()))
    assert not film[~touched_mask(cam.width, cam.height, (2.0, 2.0), rect)].any()
    p2 = host.default_render_params(spp=16, max_depth=8)
    p2.sample_stride, p2.sample_phase = 2, 1
    half, stats2, _ = multi.render(cam, p2, region=rect)
    ref, _ = _render(gpu, integ, cam, scene, region=rect, sample_stride=(2, 1))
    assert sum(s["camera_paths"] for s in stats2) == st["camera_paths"] // 2
    assert np.allclose(half, ref, rtol=2e-4, atol=1e-5 * float(single[..., :3].max()))
    with pytest.raises(gpu.PtrsError) as e:
        multi.render(cam, params, region=(0, 0, 0, 4))
    assert e.value.code == -1
    assert lib.ptrs_multi_render_region(multi._h, C.byref(cam), C.byref(params), None, None, None, None) == -1
    multi.close()
    scene.close()


@pytest.mark.gpu
def test_headless_crop_writes_the_crop_of_the_full_render(gpu, host, tmp_path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "examples", "headless")
    xml = os.path.join(root, "tests", "golden", "cornell-box.xml")
    x0, y0, x1, y1 = 17, 9, 70, 51
    r = subprocess.run([exe, xml, "-o", str(tmp_path), "--headless", "-r", "96x80", "-s", "8", "-d", "6", "--server", "127.0.0.1:1",
                        "--crop", f"{x0},{y0},{x1},{y1}"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    png = host.load_png(str(tmp_path / "render.png"))
    assert png.shape == (y1 - y0, x1 - x0, 4)
    flat, cam = host.import_scene(xml, res=(96, 80))
    scene = gpu.RenderScene(flat)
    integ = gpu.PathIntegrator(gpu.SamplerBuilder(8), max_depth=6)
    film = gpu.Film(cam.width, cam.height)
    integ.render(cam, scene, film)
    want = film.to_rgba_image()[y0:y1, x0:x1]
    diff = np.abs(png.astype(np.int32) - want.astype(np.int32))
    assert diff.max() <= 1 and (diff != 0).sum() <= 8
    bad = subprocess.run([exe, xml, "-o", str(tmp_path), "-r", "96x80", "--server", "127.0.0.1:1", "--crop", "0,0,97,10"],
                         capture_output=True, text=True, timeout=300)
    assert bad.returncode == 1 and "ptrs error -1" in bad.stderr
    scene.close()
