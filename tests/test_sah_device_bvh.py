"""The reference's SAH tree built on the device (ptrs_scene_create_sah_bvh, csrc/k_sah.cu).

The device build must emit ptrs_host::build_bvh(bounds, max_prims, 1) byte for byte: the same 32-byte records in the
same depth-first preorder and the same primitive order, over the primitives in the order the caller gives them.  A scene
made from it is then the ptrs_scene_create scene of that tree: same hits, same visit counters, same occlusion answers.
"""
import ctypes as C

import numpy as np
import pytest

from pathtracer_rs_b200._abi import PtrsLight, PtrsSceneDesc

FLT_MAX = np.float32(np.finfo(np.float32).max)


def _fmin(x, y):
    """std::fmin as glibc computes it: y only when y < x or x is NaN (so the FIRST argument wins a tie of +0 and -0)."""
    return np.where((y < x) | np.isnan(x), y, x)


def _fmax(x, y):
    return np.where((y > x) | np.isnan(x), y, x)


def _tri_bounds(tri):
    """(n, 3, 3) triangle vertices -> (n, 6) Triangle::world_bound as SceneBuilder::finalize computes it."""
    a, c, d = tri[:, 0], tri[:, 1], tri[:, 2]
    return np.concatenate([_fmin(_fmin(a, c), d), _fmax(_fmax(a, c), d)], axis=1).astype(np.float32)


def _fold(bounds):
    """A node's box: the left fold from (FLT_MAX, -FLT_MAX) over the primitives in array order."""
    mn = np.full(3, FLT_MAX, dtype=np.float32)
    mx = np.full(3, -FLT_MAX, dtype=np.float32)
    for b in bounds:
        mn = _fmin(mn, b[:3])
        mx = _fmax(mx, b[3:])
    return mn.astype(np.float32), mx.astype(np.float32)


def test_host_root_box_follows_the_first_argument_tie_rule(host):
    """Pins the rule the device build restates: the root box of host.build_bvh equals the ordered fold with
    fmin(x, y) = y if y < x or isnan(x) else x, sign bits included, over bounds with +-0, NaN and +-inf."""
    rng = np.random.default_rng(3)
    special = np.float32([0.0, -0.0, np.nan, np.inf, -np.inf, 1.0, -1.0])
    for trial in range(200):
        n = int(rng.integers(1, 12))
        lo = rng.choice(special, (n, 3))
        hi = rng.choice(special, (n, 3))
        b = np.concatenate([lo, hi], axis=1).astype(np.float32)
        nodes, _ = host.build_bvh(b, 4, 1)
        mn, mx = _fold(b)
        assert np.array_equal(nodes[0]["bmin"].view(np.uint32), mn.view(np.uint32)), (trial, b)
        assert np.array_equal(nodes[0]["bmax"].view(np.uint32), mx.view(np.uint32)), (trial, b)
    # the first argument wins a tie: the sign of a zero comes from the earlier primitive
    z = np.float32([[0.0, -0.0, 0.0, 0.0, -0.0, 0.0], [-0.0, 0.0, -0.0, -0.0, 0.0, -0.0]])
    nodes, _ = host.build_bvh(z, 4, 1)
    assert np.array_equal(np.signbit(nodes[0]["bmin"]), [False, True, False])
    assert np.array_equal(np.signbit(nodes[0]["bmax"]), [False, True, False])


# ---- helpers for the GPU tests -------------------------------------------------------------------------------------

class _Desc:
    """A copy of a FlatScene's description with its primitives in another order (area lights follow their primitive)."""

    def __init__(self, flat, perm=None):
        base = flat.desc.contents
        n = base.n_prims
        perm = np.arange(n, dtype=np.int64) if perm is None else np.asarray(perm, dtype=np.int64)
        inv = np.empty(n, dtype=np.int64)
        inv[perm] = np.arange(n)
        self.pv = np.ascontiguousarray(np.ctypeslib.as_array(base.prim_vertex, shape=(n, 3))[perm], dtype=np.uint32)
        self.arrays = [np.ascontiguousarray(np.ctypeslib.as_array(getattr(base, f), shape=(n,))[perm], dtype=np.int32)
                       for f in ("prim_mesh", "prim_material", "prim_area_light")]
        self.lights = (PtrsLight * max(1, base.n_lights))()
        if base.n_lights:
            C.memmove(self.lights, base.lights, base.n_lights * C.sizeof(PtrsLight))
        for i in range(base.n_lights):
            if self.lights[i].prim >= 0:
                self.lights[i].prim = int(inv[self.lights[i].prim])
        self.desc = PtrsSceneDesc()
        C.memmove(C.byref(self.desc), C.byref(base), C.sizeof(PtrsSceneDesc))
        self.desc.prim_vertex = self.pv.ctypes.data_as(C.POINTER(C.c_uint32))
        self.desc.prim_mesh, self.desc.prim_material, self.desc.prim_area_light = (a.ctypes.data_as(C.POINTER(C.c_int32)) for a in self.arrays)
        self.desc.lights = self.lights
        self.desc.nodes, self.desc.n_nodes = None, 0
        pos = np.ctypeslib.as_array(base.pos, shape=(base.n_verts, 3))
        self.tri = pos[self.pv]
        self.flat = flat  # keeps the pools the description points into alive

    def ptr(self):
        return C.pointer(self.desc)


def _expected_layout(ref):
    """The traversal layout ptrs_scene_create makes of the reference's preorder records (root in slot 0, the children of
    the r-th interior node in slots 2 (r + 1) and 2 (r + 1) + 1), as (slot of every record, its 8 words)."""
    interior = ref["n_prims"] == 0
    rank = np.cumsum(interior) - interior
    slot = np.zeros(ref.shape[0], dtype=np.int64)
    idx = np.nonzero(interior)[0]
    slot[idx + 1] = 2 * (rank[idx] + 1)
    slot[ref["offset"][idx].astype(np.int64)] = 2 * (rank[idx] + 1) + 1
    words = ref.view(np.uint32).reshape(-1, 8).copy()
    words[interior, 6] = 2 * (rank[interior] + 1)  # an interior record points at its pair of children
    return slot, words, int(interior.sum())


def _check_tree(gpu, host, d, m):
    """Device build over d's primitive order == host.build_bvh over the same order: records (pad masked as
    pair_layout_kernel masks it) and primitive order."""
    ref, ref_order = host.build_bvh(_tri_bounds(d.tri), m, 1)
    scene = gpu.RenderScene(d.ptr(), sah_on_device=True, max_prims_in_node=m)
    nodes, order = scene.download_nodes()
    slot, words, n_interior = _expected_layout(ref)
    assert nodes.shape[0] == 2 * (n_interior + 1)
    got = nodes.view(np.uint32).reshape(-1, 8)
    mask = np.uint32(0x0003FFFF)
    words[:, 7] &= mask
    got_at = got[slot].copy()
    got_at[:, 7] &= mask
    bad = np.nonzero((got_at != words).any(axis=1))[0]
    assert bad.size == 0, f"{bad.size} of {ref.shape[0]} records differ, first at preorder {bad[0]}: {got_at[bad[0]]} vs {words[bad[0]]}"
    assert np.array_equal(order, ref_order), f"{np.count_nonzero(order != ref_order)} primitive positions differ"
    bmin, bmax = scene.world_bound()
    assert np.array_equal(bmin.view(np.uint32), ref[0]["bmin"].view(np.uint32)) and np.array_equal(bmax.view(np.uint32), ref[0]["bmax"].view(np.uint32))
    return scene, ref


def _soup_flat(host, verts):
    b = host.SceneBuilder()
    m = b.material(host.MAT_MATTE, [b.constant_texture([0.5, 0.5, 0.5])])
    verts = np.ascontiguousarray(verts, dtype=np.float32).reshape(-1, 3)
    b.mesh(verts, np.arange(verts.shape[0], dtype=np.uint32).reshape(-1, 3), material=m)
    return b.finalize()


MAX_PRIMS = [1, 4, 16]


@pytest.mark.gpu
@pytest.mark.parametrize("m", MAX_PRIMS)
@pytest.mark.parametrize("scene_name", ["cornell", "field_small", "terrain_small", "atrium_small"])
def test_tree_equals_the_host_build_on_scenes(gpu, host, request, scene_name, m):
    flat, _ = request.getfixturevalue(scene_name)
    rng = np.random.default_rng(17)
    for perm in (None, rng.permutation(flat.n_prims)):  # the importer's order, and a shuffled one (real partitions)
        scene, _ = _check_tree(gpu, host, _Desc(flat, perm), m)
        scene.close()


@pytest.mark.gpu
@pytest.mark.parametrize("m", MAX_PRIMS)
def test_tree_equals_the_host_build_on_random_soups(gpu, host, m):
    rng = np.random.default_rng(11)
    for n_tri in list(range(1, 41)) + [257, 1000]:
        c = rng.uniform(-1, 1, (n_tri, 1, 3))
        flat = _soup_flat(host, c + rng.uniform(-0.3, 0.3, (n_tri, 3, 3)))
        scene, _ = _check_tree(gpu, host, _Desc(flat, rng.permutation(n_tri)), m)
        scene.close()


def _grid_and_copies(host, rng):
    n_dup = 4096
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    copies = _soup_flat(host, np.tile(tri, (n_dup, 1)) + np.float32([0, 0, 5]))
    g = 65
    xs, ys = np.meshgrid(np.arange(g, dtype=np.float32), np.arange(g, dtype=np.float32), indexing="ij")
    v = np.stack([xs.ravel(), ys.ravel(), np.zeros(g * g, dtype=np.float32)], axis=1)
    q = (np.arange(g - 1)[:, None] * g + np.arange(g - 1)[None, :]).ravel()
    idx = np.concatenate([np.stack([q, q + g, q + 1], axis=1), np.stack([q + 1, q + g, q + g + 1], axis=1)])
    grid = _soup_flat(host, v[idx])
    return [(copies, rng.permutation(n_dup)), (grid, rng.permutation(idx.shape[0]))]


@pytest.mark.gpu
@pytest.mark.parametrize("m", MAX_PRIMS)
def test_tree_equals_the_host_build_on_ties(gpu, host, m):
    """4096 copies of one triangle (equal centroids: one leaf per 65 535 or fewer), a regular 64 x 64 grid of quads (every
    bucket boundary a tie), and 70 000 coincident triangles (more than a leaf can count: the range is halved)."""
    rng = np.random.default_rng(5)
    cases = _grid_and_copies(host, rng)
    tri = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=np.float32)
    cases.append((_soup_flat(host, np.tile(tri, (70_000, 1))), rng.permutation(70_000)))
    for flat, perm in cases:
        scene, ref = _check_tree(gpu, host, _Desc(flat, perm), m)
        scene.close()
    assert ref.shape[0] == 3 and ref[0]["n_prims"] == 0  # 70 000 coincident: halved once, two leaves of 35 000


@pytest.mark.gpu
@pytest.mark.parametrize("m", MAX_PRIMS)
def test_tree_equals_the_host_build_on_signed_zeros_and_non_finite_coordinates(gpu, host, m):
    """Coordinates of +-0, NaN and +-inf: the fold's tie rule decides the sign of zero in the boxes, NaN is ignored by the
    fold and sends a centroid to bucket 0, and non-finite bounds make the host halve ranges it cannot split."""
    rng = np.random.default_rng(23)
    special = np.float32([0.0, -0.0, np.nan, np.inf, -np.inf])
    for n_tri, p_special in ((40, 0.3), (300, 0.05), (2000, 0.01)):
        v = rng.uniform(-1, 1, (n_tri, 3, 3)).astype(np.float32)
        pick = rng.random(v.shape) < p_special
        v[pick] = rng.choice(special, int(pick.sum()))
        v[: n_tri // 4, :, 2] = rng.choice(np.float32([0.0, -0.0]), (n_tri // 4, 3))  # flat triangles on z = +-0
        flat = _soup_flat(host, v)
        scene, _ = _check_tree(gpu, host, _Desc(flat, rng.permutation(n_tri)), m)
        scene.close()


def _device_rays(rays):
    import torch

    return torch.from_numpy(rays.view(np.uint8).reshape(-1)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name", ["cornell", "field_small", "terrain_small", "atrium_small"])
def test_scene_answers_equal_the_host_built_scene(gpu, host, request, scene_name):
    """RenderScene(flat) and the device-built scene over the same primitives: closest hits (prim, t, b0..b2), any-hit
    answers of the occlusion tree, and the reference walk's visit counters, bit for bit."""
    import torch

    flat, cam = request.getfixturevalue(scene_name)
    ref = gpu.RenderScene(flat)
    dev = gpu.RenderScene(flat, sah_on_device=True)
    _, order = dev.download_nodes()
    assert np.array_equal(order, np.arange(flat.n_prims, dtype=np.uint32))  # the importer's order is already the tree's
    bmin, bmax = flat.world_bound()
    for rays in (host.coherent_rays(cam, 192), host.incoherent_rays(bmin, bmax, 7, 60000)):
        a, b = ref.intersect(rays), dev.intersect(rays)
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
        seg = rays.copy()
        hit = a["prim"] >= 0
        seg["t_max"] = np.where(hit, a["t"] * np.float32(1.5), np.float32(1.0)).astype(np.float32)
        seg["t_max"][::2] = (a["t"][::2] * np.float32(0.5)).astype(np.float32)
        assert np.array_equal(ref.intersect_p(seg), dev.intersect_p(seg))
        assert np.array_equal(ref.intersect_p(rays), dev.intersect_p(rays))
        n = rays.shape[0]
        d_rays = _device_rays(rays)
        out = []
        for s in (ref, dev):
            d_hits = torch.empty(n * 20, dtype=torch.uint8, device="cuda")
            d_occ = torch.empty(n, dtype=torch.uint8, device="cuda")
            out.append((s.intersect_counted_device(d_rays.data_ptr(), n, d_hits.data_ptr()), d_hits.cpu().numpy(),
                        s.intersect_counted_device(d_rays.data_ptr(), n, d_occ.data_ptr(), any_hit=True), d_occ.cpu().numpy()))
        assert out[0][0] == out[1][0] and out[0][2] == out[1][2], "visit counters differ"
        assert np.array_equal(out[0][1], out[1][1]) and np.array_equal(out[0][3], out[1][3])
    ref.close()
    dev.close()


@pytest.mark.gpu
def test_shuffled_scene_maps_hits_to_the_callers_order(gpu, host, cornell_env):
    """Primitives handed over in another order: hits and area lights refer to the caller's indices, and the hits are those
    of the host-built scene of the same tree."""
    flat, cam = cornell_env
    perm = np.random.default_rng(2).permutation(flat.n_prims)
    d = _Desc(flat, perm)
    dev = gpu.RenderScene(d.ptr(), sah_on_device=True)
    ref = gpu.RenderScene(flat)
    rays = host.coherent_rays(cam, 128)
    a, b = ref.intersect(rays), dev.intersect(rays)
    hit = a["prim"] >= 0
    assert np.array_equal(hit, b["prim"] >= 0)
    assert np.array_equal(perm[b["prim"][hit]], a["prim"][hit])  # caller index -> the flat scene's index
    assert np.array_equal(a["t"][hit], b["t"][hit])
    dev.close()
    ref.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_name,depth", [("cornell_env", 15), ("field_small", 8)])
def test_path_radiance_is_bit_identical(gpu, host, request, scene_name, depth):
    flat, cam = request.getfixturevalue(scene_name)
    params = host.default_render_params(spp=16, max_depth=depth)
    rng = np.random.default_rng(11)
    px = np.stack([rng.integers(0, cam.width, 20000), rng.integers(0, cam.height, 20000)], axis=1).astype(np.int32)
    sm = rng.integers(0, params.spp, 20000).astype(np.int32)
    out = []
    for kw in ({}, {"sah_on_device": True}):
        s = gpu.RenderScene(flat, **kw)
        out.append(s.path_radiance(cam, params, px, sm))
        s.close()
    assert np.array_equal(out[0].view(np.uint32), out[1].view(np.uint32))


@pytest.mark.gpu
def test_c4_terrain_tree_at_full_size(gpu, host):
    """The 10 M-triangle C4 mesh (the scene of test_c4_hit_parity_at_full_size): byte-equal tree and primitive order."""
    flat, _ = host.make_scene(host.SCENE_TERRAIN, seed=1, n_tris=10_000_000, res=(512, 512))
    scene, ref = _check_tree(gpu, host, _Desc(flat), 4)
    _, ms = scene.bvh_info()
    print(f"C4 terrain, {flat.n_prims} triangles: device SAH build {ms:.2f} ms, host SAH build {flat.bvh_seconds * 1e3:.0f} ms")
    scene.close()


@pytest.mark.gpu
def test_refusals(gpu, host, cornell):
    """max_prims_in_node outside 1..65535 is refused (PTRS_ERR_INVALID_ARGUMENT); so is a tree deeper than the 64-entry
    traversal stack, with PTRS_ERR_UNSUPPORTED, as ptrs_scene_create refuses the host-built tree of the same primitives."""
    flat, _ = cornell
    for m in (0, 65536, -1):
        with pytest.raises(gpu.PtrsError) as e:
            gpu.RenderScene(flat, sah_on_device=True, max_prims_in_node=m)
        assert e.value.code == -1
    # triangles at 16^i along each axis and a cluster at the origin: every split peels off the farthest one or two
    p = np.float32([(16.0 ** i, 0, 0) for i in range(1, 32)] + [(0, 16.0 ** i, 0) for i in range(1, 31)] +
                   [(0, 0, 16.0 ** i) for i in range(1, 30)])
    p = np.concatenate([p, np.random.default_rng(4).uniform(0, 1, (300, 3)).astype(np.float32)])
    tri = np.stack([p, p + np.float32([0, 1, 0]), p + np.float32([0, 0, 1])], axis=1)
    deep = _soup_flat(host, tri)
    assert deep.bvh_depth > 66
    with pytest.raises(gpu.PtrsError) as e:
        gpu.RenderScene(deep)
    assert e.value.code == -3
    with pytest.raises(gpu.PtrsError) as e:
        gpu.RenderScene(deep, sah_on_device=True, max_prims_in_node=1)
    assert e.value.code == -3
    # an empty scene and a single leaf behave as through ptrs_scene_create
    one = _soup_flat(host, tri[:1])
    a, b = gpu.RenderScene(one), gpu.RenderScene(one, sah_on_device=True)
    assert a.bvh_info()[0] == b.bvh_info()[0] == 2
    r = np.zeros(1, dtype=host.RAY_DTYPE)
    r["o"], r["d"], r["t_max"] = [1.2, 0.2, 0.2], [0, 0, -1], np.inf
    assert np.array_equal(a.intersect(r).view(np.uint8), b.intersect(r).view(np.uint8))
