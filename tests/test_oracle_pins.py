"""CPU-only checks that pin the oracle and the host-side code.

The reference holds no golden vectors for the rendering path (SURVEY.md §4: 7 unit tests, none on the
path's arithmetic) and cannot be compiled here, so parity is formally UNPINNED.  What can be pinned:
  * the Sobol tables: re-derived from the Joe-Kuo direction numbers (scipy's copy) and bit-identical to
    the reference's sobolmatrices.rs (digests of its tables under tests/golden/)
  * the Sobol sequence itself against scipy.stats.qmc.Sobol (independent implementation)
  * the helper known-answer tests the reference does have (src/common/math.rs:264-299)
  * documented quirks (next_float_down, pixel-corner clamping), analytic properties of the lobes
  * committed golden vectors of the oracle (tests/golden/) so that any later drift is caught
"""
import ctypes as C
import hashlib
import json
import os
import re
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ONE_MINUS_EPS = np.float32(float.fromhex('0x1.fffffep-1'))


# ---- Sobol --------------------------------------------------------------------------------------------
def _load_blob():
    with open(os.path.join(ROOT, "pathtracer_rs_b200", "data", "sobol_tables.bin"), "rb") as f:
        raw = f.read()
    assert raw[:4] == b"SOBL"
    nd, nc, nm, nmi = struct.unpack("<4I", raw[4:20])
    off = 20
    mats = np.frombuffer(raw, dtype="<u4", count=nd * nc, offset=off).reshape(nd, nc)
    off += nd * nc * 4
    tabs = []
    for _ in range(nm + nmi):
        (ln,) = struct.unpack("<I", raw[off:off + 4])
        tabs.append(np.frombuffer(raw, dtype="<u8", count=ln, offset=off + 4))
        off += 4 + 8 * ln
    assert off == len(raw)
    return mats, tabs[:nm], tabs[nm:]


def test_sobol_tables_rederive_from_joe_kuo():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_sobol_tables as g

    mats, vdc, vdc_inv = _load_blob()
    dm, dv, di = g.derive()
    assert np.array_equal(mats, dm)
    assert all(list(a) == b for a, b in zip(vdc, dv)) and all(list(a) == b for a, b in zip(vdc_inv, di))
    assert mats.shape == (1024, 52) and len(vdc) == 25 and len(vdc_inv) == 26
    assert [len(v) for v in vdc] == [52 - 2 * m for m in range(1, 26)] and [len(v) for v in vdc_inv] == [2 * m for m in range(1, 27)]
    # the reference's own tables (src/pathtracer/sobolmatrices.rs:5-7, 53463, 54155), stored as digests
    with open(os.path.join(ROOT, "tests", "golden", "sobol_reference_tables.json")) as f:
        ref = json.load(f)

    def digest(tables):
        return hashlib.sha256(b"".join(np.asarray(t, dtype="<u8").tobytes() for t in tables)).hexdigest()

    assert hashlib.sha256(dm.astype("<u4").tobytes()).hexdigest() == ref["SOBOL_MATRICES_32"]
    assert digest(dv) == ref["VD_C_SOBOL_MATRICES"] and digest(di) == ref["VD_C_SOBOL_MATRICES_INV"]


def test_sobol_sample_matches_scipy_sequence(oracle):
    from scipy.stats import qmc

    d, n = 16, 1024
    pts = qmc.Sobol(d=d, scramble=False, bits=32).random(n)  # Gray-code order
    L = oracle.lib()
    for i in range(0, n, 7):
        a = i ^ (i >> 1)
        for k in range(d):
            v = np.uint32(round(pts[i, k] * 2.0 ** 32))
            expect = min(ONE_MINUS_EPS, np.float32(v) * np.float32(2.0 ** -32))
            assert L.oracle_sobol_sample(a, k, 0) == expect


def test_sobol_index_hits_the_requested_pixel(oracle):
    """sobol_interval_to_index must return the index whose first two (unscrambled) dimensions fall into
    the pixel — the defining property of the global sampler (lowdiscrepancy.rs:9-39)."""
    L = oracle.lib()
    rng = np.random.default_rng(0)
    for m in (1, 4, 10, 11, 12):
        res = 1 << m
        for _ in range(200):
            px, py, frame = int(rng.integers(0, res)), int(rng.integers(0, res)), int(rng.integers(0, 1024))
            idx = L.oracle_sobol_interval_to_index(m, frame, px, py)
            assert idx >> (2 * m) == frame
            x, y = L.oracle_sobol_sample(idx, 0, 0), L.oracle_sobol_sample(idx, 1, 0)
            assert int(x * res) == px and int(y * res) == py


def test_pixel_jitter_quirk(oracle, host):
    """Quirk 1 (SURVEY.md §8): the XOR scramble is applied to dims 0/1 too, so for pixels whose scramble has
    any of the top m bits set the camera sample is clamped to a pixel corner, identically for every spp."""
    cam = host.look_at_camera((0, 0, 5), (0, 0, 0), (0, 1, 0), 40.0, 512, 512)
    params = host.default_render_params(spp=16)
    xs, ys = np.meshgrid(np.arange(-2, 514, 9), np.arange(-2, 514, 9))
    px = np.stack([xs.ravel(), ys.ravel()], 1).astype(np.int32)
    clamped = []
    for s in (0, 5, 15):
        v, _ = oracle.sobol_samples(cam, params, px, np.full(len(px), s, np.int32), [0, 1])
        assert ((v >= 0) & (v < 1)).all()
        clamped.append(np.isin(v, [0.0, ONE_MINUS_EPS]).all(axis=1))
    assert np.array_equal(clamped[0], clamped[1]) and np.array_equal(clamped[0], clamped[2])
    assert 0.3 < clamped[0].mean() < 0.7  # "50 % (C1, m = 10)"


# ---- helper KATs ----------------------------------------------------------------------------------------
def test_math_known_answers(oracle):
    L = oracle.lib()
    for i in range(63):  # src/common/math.rs:266-276
        assert L.oracle_log2_int(1 << i) == i
        if i >= 1:
            assert L.oracle_log2_int((1 << i) + 1) == i

    def solve(a, b):
        x = (C.c_float * 2)()
        ok = L.oracle_solve_2x2((C.c_float * 4)(*a), (C.c_float * 2)(*b), x)
        return ok, (x[0], x[1])

    assert solve([0, 1, 1, 0], [2, 4]) == (1, (4.0, 2.0))  # math.rs:278-299
    assert solve([0, 0, 0, 0], [2, 4])[0] == 0
    assert solve([1, 1, -1, 1], [2, 2]) == (1, (0.0, 2.0))
    eps = np.float32(2.0 ** -24)
    assert L.oracle_gamma(3) == np.float32(np.float32(3) * eps) / np.float32(np.float32(1) - np.float32(3) * eps)
    assert L.oracle_cantor_pairing(3, 4) == (7 * 8) // 2 + 4
    assert L.oracle_cantor_pairing(2 ** 30 - 3, 2 ** 30 + 500) < 2 ** 63  # fits usize like the reference


def test_next_float_quirk(oracle):
    L = oracle.lib()
    one = np.float32(1.0)
    assert L.oracle_next_float_up(1.0) == np.nextafter(one, np.float32(2))
    assert L.oracle_next_float_up(-1.0) == np.nextafter(-one, np.float32(0))
    # the reference's next_float_down moves UP (math.rs:98-103 has the increments swapped)
    assert L.oracle_next_float_down(1.0) == np.nextafter(one, np.float32(2))
    assert L.oracle_next_float_down(-1.0) == np.nextafter(-one, np.float32(0))
    assert np.isnan(L.oracle_next_float_down(0.0))


# ---- camera ---------------------------------------------------------------------------------------------
def test_camera_conventions(host, oracle):
    """Raster (0, 0) is the top-left corner, +x right, camera looks down -z (common/mod.rs:33-62,
    pathtracer/mod.rs:59-81)."""
    cam = host.look_at_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 90.0, 640, 480)
    m = np.array(cam.raster_to_screen).reshape(4, 4)
    assert np.allclose(m @ [0, 0, 0, 1], [-1, 1, 0, 1]) and np.allclose(m @ [640, 480, 0, 1], [1, -1, 0, 1])
    params = host.default_render_params(spp=1)
    rays, pf, _ = oracle.generate_rays(cam, params, [[320, 240]], [0])
    d = rays["d"][0]
    assert abs(np.linalg.norm(d) - 1) < 1e-6 and d[2] < -0.99  # centre pixel looks along -z
    assert np.allclose(cam.persp[1], 1.0, atol=1e-6) and np.allclose(cam.persp[0], 0.75, atol=1e-6)  # 1/tan(45), /aspect
    c2 = host.make_scene(host.SCENE_CORNELL, res=(64, 64))[1]
    assert np.allclose(c2.trans, [0, 1, 6.8]) and abs(abs(c2.rot[3]) - 1) < 1e-6  # Cornell sensor: identity rotation


def _quat_matrix(q):
    i, j, k, w = q
    return np.array([[1 - 2 * (j * j + k * k), 2 * (i * j - k * w), 2 * (i * k + j * w)],
                     [2 * (i * j + k * w), 1 - 2 * (i * i + k * k), 2 * (j * k - i * w)],
                     [2 * (i * k - j * w), 2 * (j * k + i * w), 1 - 2 * (i * i + j * j)]], dtype=np.float64)


def test_reference_camera_unit_tests(host):
    """The reference's three camera tests (src/common/mod.rs:103-164) as known answers for look_at_camera / make_camera —
    the one reference-held check on the restated nalgebra arithmetic (Isometry3::look_at_rh(..).inverse(), Perspective3::new,
    the glm screen_to_raster product).  Each assertion is taken over where it can hold for Camera::new AS WRITTEN
    (mod.rs:33-62, the code render() runs); where the reference's expectation contradicts its own constructor the
    arithmetic is spelled out and the constructor wins:
      * test_camera_wold_to_screen (:118-140): camera-space position — taken over verbatim (epsilon 1e-6, relative).  Its
        z_screen = (z - n) f / ((f - n) z) is the [0, 1] depth convention; nalgebra's Perspective3 (m22 = (f + n)/(n - f),
        m23 = 2 f n/(n - f)) projects to [-1, 1]: ((f + n) z - 2 f n) / ((f - n) z).  Both are evaluated below; x = y = 0 holds.
      * test_camera_screen_to_raster (:142-161) expects screen (1, 1) -> raster (640, 480) and (-1, -1) -> (0, 0), but
        mod.rs:38-40 multiplies by scaling(1/2, -1/2, 1): y is flipped, (1, 1) -> (640, 0) and (-1, -1) -> (0, 480).
        The x halves of both assertions hold and are checked; y follows the constructor.
      * test_camera_raster_to_screen (:163-178) unprojects raster (640, 360) of a 640 x 480 film and expects the view
        axis: written for a 1280 x 720 default resolution; at (320, 240) the same assertion (x = y = 0, z = -near-plane
        distance of the unprojected point) holds and is checked."""
    n, f = 0.01, 1000.0
    eye = np.array([10.0, 10.0, 10.0])
    cam = host.look_at_camera(eye, (0, 0, 0), (0, 1, 0), 90.0, 640, 480)
    # cam_to_world.inverse() * origin
    R, t = _quat_matrix(list(cam.rot)), np.array(list(cam.trans), dtype=np.float64)
    p_cam = R.T @ (np.zeros(3) - t)
    z = float(np.linalg.norm(eye))
    assert np.allclose(p_cam, [0.0, 0.0, -z], rtol=1e-6, atol=1e-6)
    # Perspective3::new(640/480, pi/2, 0.01, 1000): look_at_camera uses the same near plane and 10000 as far (the importer's
    # values, common/importer/mitsuba.rs:698-703), so m00 / m11 are pinned here and the depth terms by formula below
    m00, m11, m22, m23 = list(cam.persp)
    assert abs(m11 - 1.0) < 1e-6 and abs(m00 - 0.75) < 1e-6
    inv = -1.0 / p_cam[2]
    assert abs(m00 * p_cam[0] * inv) < 1e-6 and abs(m11 * p_cam[1] * inv) < 1e-6  # screen x = y = 0
    z_gl = ((f + n) * z - 2 * f * n) / ((f - n) * z)  # nalgebra (documented matrix)
    z_01 = ((z - n) * f) / ((f - n) * z)              # what the reference's test writes down
    assert abs(z_gl - z_01) > 1e-4                    # they cannot both hold: the reference's depth assertion is stale
    # screen_to_raster = inverse of the raster_to_screen the kernels use
    cam2 = host.look_at_camera((0, 0, 0), (1, 0, 0), (0, 1, 0), 90.0, 640, 480)
    r2s = np.array(list(cam2.raster_to_screen), dtype=np.float64).reshape(4, 4)
    s2r = np.linalg.inv(r2s)
    a = s2r @ [1.0, 1.0, 0.5, 1.0]
    b = s2r @ [-1.0, -1.0, 0.5, 1.0]
    assert abs(a[0] - 640.0) < 1e-3 and abs(a[2] - 0.5) < 1e-6 and abs(b[0]) < 1e-3 and abs(b[2] - 0.5) < 1e-6  # as the reference asserts
    assert abs(a[1]) < 1e-3 and abs(b[1] - 480.0) < 1e-3  # y per mod.rs:38-40 (flipped), not per the stale test
    # unproject_point(raster_to_screen * centre): on the view axis, on the near plane
    s = r2s @ [320.0, 240.0, 0.0, 1.0]
    m00, m11, m22, m23 = list(cam2.persp)
    k = m23 / (s[2] + m22)
    p = np.array([s[0] * k / m00, s[1] * k / m11, -k])
    assert abs(p[0]) < 1e-6 and abs(p[1]) < 1e-6 and p[2] < 0


# ---- BVH ------------------------------------------------------------------------------------------------
def _check_bvh(nodes, order, bounds, max_prims=4):
    n = len(order)
    assert sorted(order.tolist()) == list(range(n))
    seen = np.zeros(n, dtype=np.int32)
    stack = [0]
    visit = []
    while stack:
        i = stack.pop()
        visit.append(i)
        nd = nodes[i]
        if nd["n_prims"] > 0:
            sl = slice(int(nd["offset"]), int(nd["offset"]) + int(nd["n_prims"]))
            seen[sl] += 1
            b = bounds[order[sl]]
            assert np.array_equal(nd["bmin"], b[:, :3].min(0)) and np.array_equal(nd["bmax"], b[:, 3:].max(0))
            if nd["n_prims"] > max_prims:  # only allowed for identical centroids (accelerator.rs:190-197)
                c = b[:, :3] + 0.5 * (b[:, 3:] - b[:, :3])
                assert (np.ptp(c, axis=0) == 0).any()
        else:
            l, r = i + 1, int(nd["offset"])
            assert r > l and nd["axis"] < 3
            assert np.array_equal(nd["bmin"], np.minimum(nodes[l]["bmin"], nodes[r]["bmin"]))
            assert np.array_equal(nd["bmax"], np.maximum(nodes[l]["bmax"], nodes[r]["bmax"]))
            stack += [r, l]
    assert visit == list(range(len(nodes)))  # DFS pre-order, first child at idx + 1 (accelerator.rs:309-346)
    assert (seen == 1).all()


def test_bvh_build_invariants(host):
    rng = np.random.default_rng(5)
    for n in (1, 2, 3, 5, 64, 5000):
        lo = rng.random((n, 3), dtype=np.float32)
        b = np.concatenate([lo, lo + rng.random((n, 3), dtype=np.float32) * 0.05], 1)
        nodes, order = host.build_bvh(b, 4, 1)
        _check_bvh(nodes, order, b)
    # degenerate: identical centroids collapse into one leaf; duplicates along one axis still split
    b = np.tile(np.array([[0, 0, 0, 1, 1, 1]], np.float32), (9, 1))
    nodes, order = host.build_bvh(b, 4, 1)
    assert len(nodes) == 1 and nodes[0]["n_prims"] == 9
    assert host.build_bvh(np.zeros((0, 6), np.float32), 4, 1)[0].shape == (0,)


def test_bvh_parallel_build_is_identical(host):
    rng = np.random.default_rng(6)
    lo = rng.random((60000, 3), dtype=np.float32)
    b = np.concatenate([lo, lo + 0.01], 1).astype(np.float32)
    n1, o1 = host.build_bvh(b, 4, 1)
    n8, o8 = host.build_bvh(b, 4, 8)
    assert np.array_equal(n1.view(np.uint8), n8.view(np.uint8)) and np.array_equal(o1, o8)


def test_bvh_build_survives_hostile_bounds(host):
    """Non-finite or coincident primitive bounds (a corrupt mesh): the reference indexes its SAH buckets out of range or
    recurses without end; the restated builder must still return a valid tree over every primitive."""
    rng = np.random.default_rng(1)
    n = 3000
    c = rng.random((n, 3)).astype(np.float32)
    base = np.concatenate([c - 0.01, c + 0.01], 1).astype(np.float32)
    for bad in (np.nan, np.inf, -np.inf, 3e38):
        b = base.copy()
        b[rng.integers(0, n, 40), rng.integers(0, 6, 40)] = bad
        nodes, order = host.build_bvh(b)
        assert np.array_equal(np.sort(order), np.arange(n))
        leaves = nodes[nodes["n_prims"] > 0]
        assert int(leaves["n_prims"].sum()) == n
    same = np.tile(base[:1], (70000, 1))  # more coincident primitives than the 16-bit leaf count holds
    nodes, order = host.build_bvh(same)
    leaves = nodes[nodes["n_prims"] > 0]
    assert int(leaves["n_prims"].astype(np.int64).sum()) == 70000 and len(nodes) == 3


def test_cornell_scene_shape(cornell):
    flat, cam = cornell
    d = flat.desc.contents
    assert (d.n_prims, d.n_lights, d.n_materials, d.n_meshes, d.n_infinite_lights) == (36, 2, 8, 8, 0)
    lights = [d.lights[i] for i in range(2)]
    assert all(l.type == 2 and list(l.color) == [0, 0, 0] for l in lights)
    assert all(d.prim_area_light[l.prim] == i for i, l in enumerate(lights))
    assert np.isclose(sum(l.area for l in lights), 0.47 * 0.38, rtol=1e-3)  # light quad 0.47 x 0.38
    bmin, bmax = flat.world_bound()
    assert np.allclose(bmin, [-1, 0, -1], atol=1e-6) and np.allclose(bmax, [1, 2, 1], atol=1e-6)


# ---- lobes: analytic properties ---------------------------------------------------------------------------
def _lobe_params(r=(0.8, 0.6, 0.4), t=(0.04, 0.04, 0.04), ax=0.2, ay=0.3, eta=(0.2, 0.92, 1.1), k=(3.9, 2.45, 2.14), metallic=0.0, d_eta=1.5):
    return (C.c_float * 16)(*r, *t, ax, ay, *eta, *k, metallic, d_eta)


@pytest.mark.parametrize("lobe", [0, 1, 2, 3, 4])
def test_lobe_sampling_consistency(oracle, lobe):
    """sample_f returns f and pdf consistent with f()/pdf(); pdf integrates to <= 1; energy is bounded."""
    L = oracle.lib()
    p = _lobe_params()
    rng = np.random.default_rng(lobe)
    wo = np.array([0.3, -0.2, 0.8], np.float32)
    wo /= np.linalg.norm(wo)
    wo_c = (C.c_float * 3)(*wo)
    est, n_ok = np.zeros(3), 0
    for _ in range(3000):
        out = (C.c_float * 7)()
        L.oracle_bxdf_sample(lobe, p, wo_c, float(rng.random()), float(rng.random()), out)
        wi, f, pdf = np.array(out[0:3]), np.array(out[3:6]), out[6]
        if pdf == 0:
            continue
        ev = (C.c_float * 4)()
        L.oracle_bxdf_eval(lobe, p, wo_c, (C.c_float * 3)(*wi), ev)
        assert np.allclose(f, ev[0:3], rtol=1e-4, atol=1e-6) and np.isclose(pdf, ev[3], rtol=1e-3)
        est += f * abs(wi[2]) / pdf
        n_ok += 1
    albedo = est / 3000
    assert n_ok > 2000 and (albedo < 1.05).all() and (albedo > 0).all()
    # quadrature of the pdf over the hemisphere
    th, ph = np.meshgrid((np.arange(200) + 0.5) / 200 * np.pi / 2, (np.arange(400) + 0.5) / 400 * 2 * np.pi)
    tot = 0.0
    for t_, p_ in zip(th.ravel()[::37], ph.ravel()[::37]):
        wi = (C.c_float * 3)(np.sin(t_) * np.cos(p_), np.sin(t_) * np.sin(p_), np.cos(t_))
        ev = (C.c_float * 4)()
        L.oracle_bxdf_eval(lobe, p, wo_c, wi, ev)
        tot += ev[3] * np.sin(t_)
    integral = tot * (np.pi / 2 / 200) * (2 * np.pi / 400) * 37
    assert 0.5 < integral < 1.08


def test_fresnel_known_answers(oracle):
    L = oracle.lib()
    assert np.isclose(L.oracle_fr_dielectric(1.0, 1.0, 1.5), 0.04, rtol=1e-5)  # ((n-1)/(n+1))^2
    assert L.oracle_fr_dielectric(0.0, 1.0, 1.5) == 1.0
    assert L.oracle_fr_dielectric(-0.3, 1.0, 1.5) == 1.0  # total internal reflection from inside: sin_t = 1.5 * 0.954 > 1
    out = (C.c_float * 3)()
    L.oracle_cosine_sample_hemisphere(0.5, 0.5, out)
    assert list(out) == [0.0, 0.0, 1.0]


# ---- C ABI ------------------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "ptrs_b200.h")).read()
    declared = set(re.findall(r"\b(ptrs_[a-z0-9_]+)\s*\(", hdr))
    import pathtracer_rs_b200.gpu as gpu

    assert declared == set(gpu.EXPORTS), declared ^ set(gpu.EXPORTS)
    lib = C.CDLL(gpu.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.ptrs_abi_version() == 1


def test_abi_struct_sizes():
    from pathtracer_rs_b200 import _abi

    sizes = {"PtrsRay": 28, "PtrsHit": 20, "PtrsBvhNode": 32, "PtrsMesh": 8, "PtrsTexture": 56, "PtrsMaterial": 32, "PtrsLight": 64,
             "PtrsMipMap": 12 + 64 + 64 + 4 + 128, "PtrsCamera": 144, "PtrsRenderParams": 9 * 4 + 8 + 1024 + 8}
    for k, v in sizes.items():
        assert C.sizeof(getattr(_abi, k)) == v, (k, C.sizeof(getattr(_abi, k)))


def test_product_package_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "pathtracer_rs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "oracle" not in txt.lower(), os.path.join(dirpath, f)


_NO_DEVICE_CHILD = """
import ctypes as C
import sys

import pytest

sys.path.insert(0, sys.argv[1])
import pathtracer_rs_b200.gpu as gpu

n = C.c_int32(-1)
rc = gpu.lib().ptrs_device_count(C.byref(n))
assert rc != 0 or n.value == 0, n.value
flat = None
with pytest.raises((gpu.PtrsError, RuntimeError)):
    import pathtracer_rs_b200.host as host

    flat, _ = host.make_scene(host.SCENE_CORNELL, res=(8, 8))
    gpu.RenderScene(flat)
"""


def test_no_cpu_fallback_without_a_device():
    """In a child process that sees no CUDA device (on a GPU machine as well), the render path raises."""
    import subprocess

    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHILD, ROOT], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
