"""ctypes binding of libptrs_b200.so (the C ABI in include/ptrs_b200.h) plus a thin mirror of the
reference's host-facing interface for this path:

    SamplerBuilder(spp, sample_bounds)            src/pathtracer/sampler/sobol.rs:35
    PathIntegrator(sampler_builder, max_depth)    src/pathtracer/integrator.rs:230
    PathIntegrator.preprocess(scene)              src/pathtracer/integrator.rs:250
    PathIntegrator.render(camera, scene)          src/pathtracer/integrator.rs:536
    RenderScene.{intersect, intersect_p, world_bound}   src/pathtracer/mod.rs:92-102
    Film.{clear, get_sample_bounds, to_rgba_image, to_channel_updates}   src/common/film.rs:164-271

There is no CPU fallback: if the library is missing or no CUDA device is usable, calls raise.
"""
import ctypes as C
import os

import numpy as np

from ._abi import *  # noqa: F401,F403
from .host import HIT_DTYPE, RAY_DTYPE, FlatScene, default_render_params

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PTRS_B200_LIB") or os.path.join(_HERE, "lib", "libptrs_b200.so")  # override: A/B another build of the library
_LIB = None

EXPORTS = [
    "ptrs_abi_version", "ptrs_last_error", "ptrs_device_count", "ptrs_set_device", "ptrs_scene_create", "ptrs_scene_destroy",
    "ptrs_scene_world_bound", "ptrs_scene_device_bytes", "ptrs_intersect", "ptrs_intersect_p", "ptrs_intersect_device",
    "ptrs_intersect_p_device", "ptrs_intersect_counted_device", "ptrs_film_create", "ptrs_film_wrap_device", "ptrs_film_destroy",
    "ptrs_film_clear", "ptrs_film_download", "ptrs_film_resolve", "ptrs_film_resolve_srgb8", "ptrs_film_device_ptr",
    "ptrs_film_sample_bounds", "ptrs_render_params_default", "ptrs_render", "ptrs_path_radiance", "ptrs_stats",
    "ptrs_set_stats_mode", "ptrs_sobol_samples", "ptrs_generate_rays", "ptrs_trim_memory", "ptrs_scene_create_device_bvh",
    "ptrs_scene_bvh_info", "ptrs_scene_download_nodes", "ptrs_read_bandwidth", "ptrs_gather_bandwidth",
    "ptrs_multi_create", "ptrs_multi_destroy", "ptrs_multi_device_count", "ptrs_multi_render", "ptrs_multi_root_film", "ptrs_multi_scene",
    "ptrs_comm_unique_id", "ptrs_comm_init_rank", "ptrs_comm_destroy", "ptrs_comm_info", "ptrs_film_reduce",
    "ptrs_bxdf_eval", "ptrs_bxdf_sample", "ptrs_light_sample", "ptrs_light_pdf", "ptrs_scene_download_mipmaps", "ptrs_scene_download_env",
    "ptrs_scene_create_sah_bvh", "ptrs_render_region", "ptrs_multi_render_region", "ptrs_film_region_sample_rect",
]


class PtrsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ptrs error {code}: {msg}")
        self.code = code


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} missing: the CUDA library was not built (run __graft_entry__.build()); "
                               "there is no CPU fallback for this path")
        L = C.CDLL(LIB_PATH)
        vp, i32, sz = C.c_void_p, C.c_int32, C.c_size_t
        fp, i32p, u64p, u8p = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)
        camp, rpp, descp = C.POINTER(PtrsCamera), C.POINTER(PtrsRenderParams), C.POINTER(PtrsSceneDesc)
        rayp, hitp = C.POINTER(PtrsRay), C.POINTER(PtrsHit)
        L.ptrs_last_error.restype = C.c_char_p
        L.ptrs_device_count.argtypes = [i32p]
        L.ptrs_set_device.argtypes = [i32]
        L.ptrs_scene_create.argtypes = [descp, C.POINTER(vp)]
        L.ptrs_scene_create_device_bvh.argtypes = [descp, C.POINTER(vp)]
        L.ptrs_scene_create_sah_bvh.argtypes = [descp, i32, C.POINTER(vp)]
        L.ptrs_scene_bvh_info.argtypes = [vp, C.POINTER(C.c_uint32), fp]
        L.ptrs_scene_download_nodes.argtypes = [vp, C.POINTER(PtrsBvhNode), C.c_uint32, C.POINTER(C.c_uint32)]
        L.ptrs_scene_destroy.argtypes = [vp]
        L.ptrs_scene_download_mipmaps.argtypes = [vp, C.POINTER(PtrsMipMap), C.c_uint32, u64p, fp, C.c_uint64]
        L.ptrs_scene_download_env.argtypes = [vp, i32, i32p, i32p, fp, fp, fp, fp, fp]
        L.ptrs_scene_world_bound.argtypes = [vp, fp]
        L.ptrs_scene_device_bytes.restype = C.c_uint64
        L.ptrs_scene_device_bytes.argtypes = [vp]
        L.ptrs_intersect.argtypes = [vp, rayp, sz, hitp]
        L.ptrs_intersect_p.argtypes = [vp, rayp, sz, u8p]
        L.ptrs_intersect_device.argtypes = [vp, vp, sz, vp, vp]
        L.ptrs_intersect_p_device.argtypes = [vp, vp, sz, vp, vp]
        L.ptrs_intersect_counted_device.argtypes = [vp, vp, sz, vp, i32, vp, u64p, u64p, vp]
        L.ptrs_film_create.argtypes = [i32, i32, C.POINTER(vp)]
        L.ptrs_film_wrap_device.argtypes = [i32, i32, vp, C.POINTER(vp)]
        L.ptrs_film_destroy.argtypes = [vp]
        L.ptrs_film_clear.argtypes = [vp, vp]
        L.ptrs_film_download.argtypes = [vp, fp]
        L.ptrs_film_resolve.argtypes = [vp, fp]
        L.ptrs_film_resolve_srgb8.argtypes = [vp, u8p]
        L.ptrs_film_device_ptr.restype = vp
        L.ptrs_film_device_ptr.argtypes = [vp]
        L.ptrs_film_sample_bounds.argtypes = [i32, i32, fp, i32p]
        L.ptrs_film_region_sample_rect.argtypes = [i32, i32, fp, i32p, i32p]
        L.ptrs_render_params_default.argtypes = [rpp]
        L.ptrs_render.argtypes = [vp, camp, rpp, vp, vp]
        L.ptrs_render_region.argtypes = [vp, camp, rpp, i32p, vp, vp]
        L.ptrs_path_radiance.argtypes = [vp, camp, rpp, i32p, i32p, sz, fp]
        L.ptrs_stats.argtypes = [vp, C.POINTER(PtrsStats)]
        L.ptrs_set_stats_mode.argtypes = [vp, i32]
        L.ptrs_read_bandwidth.argtypes = [sz, i32, fp]
        L.ptrs_gather_bandwidth.argtypes = [sz, i32, fp]
        L.ptrs_sobol_samples.argtypes = [camp, rpp, i32p, i32p, sz, i32p, sz, fp, u64p]
        L.ptrs_generate_rays.argtypes = [camp, rpp, i32p, i32p, sz, rayp, fp, fp]
        L.ptrs_multi_create.argtypes = [descp, i32, i32p, i32, C.POINTER(vp)]
        L.ptrs_multi_destroy.argtypes = [vp]
        L.ptrs_multi_device_count.argtypes = [vp, i32p]
        L.ptrs_multi_render.argtypes = [vp, camp, rpp, fp, C.POINTER(PtrsStats), fp]
        L.ptrs_multi_render_region.argtypes = [vp, camp, rpp, i32p, fp, C.POINTER(PtrsStats), fp]
        L.ptrs_multi_root_film.argtypes = [vp, C.POINTER(vp)]
        L.ptrs_multi_scene.argtypes = [vp, i32, C.POINTER(vp)]
        L.ptrs_comm_unique_id.argtypes = [u8p]
        L.ptrs_comm_init_rank.argtypes = [u8p, i32, i32, C.POINTER(vp)]
        L.ptrs_comm_destroy.argtypes = [vp]
        L.ptrs_comm_info.argtypes = [vp, i32p, i32p]
        L.ptrs_film_reduce.argtypes = [vp, vp, i32, vp]
        lobep = C.POINTER(PtrsLobeDesc)
        L.ptrs_bxdf_eval.argtypes = [lobep, fp, fp, sz, i32, fp]
        L.ptrs_bxdf_sample.argtypes = [lobep, fp, fp, sz, i32, fp]
        L.ptrs_light_sample.argtypes = [vp, i32, fp, fp, fp, sz, i32, fp]
        L.ptrs_light_pdf.argtypes = [vp, i32, fp, fp, fp, sz, i32, fp]
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise PtrsError(rc, lib().ptrs_last_error().decode(errors="replace"))


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _rect(r):
    """(x0, y0, x1, y1) -> int32_t[4]"""
    if len(r) != 4:
        raise ValueError("a rectangle is (x0, y0, x1, y1)")
    return (C.c_int32 * 4)(*(int(v) for v in r))


def device_count():
    n = C.c_int32(0)
    _check(lib().ptrs_device_count(C.byref(n)))
    return n.value


def set_device(i):
    _check(lib().ptrs_set_device(i))


def read_bandwidth(n_bytes, reps=20):
    """GB/s of `reps` streaming read passes over a device buffer of n_bytes (ptrs_read_bandwidth): L2 read bandwidth for
    a buffer that fits in L2, HBM read bandwidth for a much larger one."""
    out = C.c_float(0)
    _check(lib().ptrs_read_bandwidth(n_bytes, reps, C.byref(out)))
    return out.value


def gather_bandwidth(n_bytes, gathers_per_thread=256):
    """GB/s of independent random 64-byte gathers over a device buffer of n_bytes (ptrs_gather_bandwidth)."""
    out = C.c_float(0)
    _check(lib().ptrs_gather_bandwidth(n_bytes, gathers_per_thread, C.byref(out)))
    return out.value


def trim_memory():
    """Return the device memory cached from destroyed scenes / workspaces to the driver."""
    _check(lib().ptrs_trim_memory())


class Film:
    """W x H x (r, g, b, weight) f32 on the device (src/common/film.rs FilmPixel sums)."""

    def __init__(self, width, height, device_ptr=None):
        self.width, self.height = width, height
        h = C.c_void_p()
        if device_ptr is None:
            _check(lib().ptrs_film_create(width, height, C.byref(h)))
        else:
            _check(lib().ptrs_film_wrap_device(width, height, C.c_void_p(device_ptr), C.byref(h)))
        self._h = h

    def __del__(self):
        if getattr(self, "_h", None):
            lib().ptrs_film_destroy(self._h)
            self._h = None

    def clear(self, stream=None):  # film.rs:164-172
        _check(lib().ptrs_film_clear(self._h, C.c_void_p(stream or 0)))

    def get_sample_bounds(self, radius=(2.0, 2.0)):  # film.rs:174-185
        r = (C.c_float * 2)(*radius)
        out = (C.c_int32 * 4)()
        _check(lib().ptrs_film_sample_bounds(self.width, self.height, r, out))
        return tuple(out)

    def region_sample_rect(self, pixel_rect, radius=(2.0, 2.0)):
        """The sample rectangle whose render completes the pixels of pixel_rect (x0, y0, x1, y1), half-open
        (ptrs_film_region_sample_rect); pass it to PathIntegrator.render(..., region=...)."""
        r = (C.c_float * 2)(*radius)
        out = (C.c_int32 * 4)()
        _check(lib().ptrs_film_region_sample_rect(self.width, self.height, r, _rect(pixel_rect), out))
        return tuple(out)

    def download(self):
        """Raw (H, W, 4) sums: contrib rgb and filter weight."""
        out = np.empty((self.height, self.width, 4), dtype=np.float32)
        _check(lib().ptrs_film_download(self._h, _p(out, C.c_float)))
        return out

    def to_channel_updates(self):  # film.rs:253-271 -> (H, W, 3) f32
        out = np.empty((self.height, self.width, 3), dtype=np.float32)
        _check(lib().ptrs_film_resolve(self._h, _p(out, C.c_float)))
        return out

    def to_rgba_image(self):  # film.rs:230-251 -> (H, W, 4) u8, sRGB
        out = np.empty((self.height, self.width, 4), dtype=np.uint8)
        _check(lib().ptrs_film_resolve_srgb8(self._h, _p(out, C.c_uint8)))
        return out

    @property
    def device_ptr(self):
        return lib().ptrs_film_device_ptr(self._h)


class RenderScene:
    """Device copy of a flattened scene (src/pathtracer/mod.rs:84-106)."""

    def __init__(self, flat, device_bvh=False, device_tables=False, sah_on_device=False, max_prims_in_node=4):
        """device_bvh=True ignores the description's nodes and builds the tree on the GPU (ptrs_scene_create_device_bvh: Morton order + PLOC);
        sah_on_device=True ignores them too and builds the reference's SAH tree over the description's primitive order on the GPU
        (ptrs_scene_create_sah_bvh, leaves of at most max_prims_in_node primitives);
        device_tables=True hands over level 0 of every MIP pyramid only and no env Distribution2D: the library builds them."""
        if device_bvh and sah_on_device:
            raise ValueError("device_bvh and sah_on_device select different trees")
        desc = (flat.desc_device_tables if device_tables else flat.desc) if isinstance(flat, FlatScene) else flat
        h = C.c_void_p()
        if sah_on_device:
            _check(lib().ptrs_scene_create_sah_bvh(desc, max_prims_in_node, C.byref(h)))
        else:
            _check((lib().ptrs_scene_create_device_bvh if device_bvh else lib().ptrs_scene_create)(desc, C.byref(h)))
        self._h = h
        self.n_lights = desc.contents.n_lights
        self.n_prims = desc.contents.n_prims
        self.device_bvh = device_bvh or sah_on_device  # the scene keeps a primitive order of its own

    def bvh_info(self):
        """(device node count, device build time in ms; 0 for a host-built tree)"""
        n, ms = C.c_uint32(0), C.c_float(0)
        _check(lib().ptrs_scene_bvh_info(self._h, C.byref(n), C.byref(ms)))
        return n.value, ms.value

    def download_nodes(self):
        """Device-side tree: (nodes structured array in the traversal layout, prim_order or None)."""
        from .host import NODE_DTYPE

        n, _ = self.bvh_info()
        nodes = np.empty(n, dtype=NODE_DTYPE)
        order = np.empty(self.n_prims, dtype=np.uint32) if self.device_bvh else None
        _check(lib().ptrs_scene_download_nodes(self._h, _p(nodes, PtrsBvhNode), n, _p(order, C.c_uint32) if self.device_bvh else None))
        return nodes, order

    def download_mipmaps(self):
        """(list of PtrsMipMap headers, texel pool) as the device holds them."""
        n = C.c_uint64(0)
        _check(lib().ptrs_scene_download_mipmaps(self._h, None, 0, C.byref(n), None, 0))
        cap = 4096
        hdr = (PtrsMipMap * cap)()
        pool = np.empty(n.value, dtype=np.float32)
        _check(lib().ptrs_scene_download_mipmaps(self._h, hdr, cap, C.byref(n), _p(pool, C.c_float), n.value))
        return hdr, pool

    def download_env(self, env):
        """Distribution2D of env light `env` as the device holds it: dict of cond_func, cond_cdf, cond_func_int, marg_cdf, marg_func_int."""
        nu, nv, mi = C.c_int32(0), C.c_int32(0), C.c_float(0)
        _check(lib().ptrs_scene_download_env(self._h, env, C.byref(nu), C.byref(nv), None, None, None, None, None))
        f = np.empty((nv.value, nu.value), dtype=np.float32)
        c = np.empty((nv.value, nu.value + 1), dtype=np.float32)
        fi = np.empty(nv.value, dtype=np.float32)
        mc = np.empty(nv.value + 1, dtype=np.float32)
        _check(lib().ptrs_scene_download_env(self._h, env, C.byref(nu), C.byref(nv), _p(f, C.c_float), _p(c, C.c_float), _p(fi, C.c_float), _p(mc, C.c_float), C.byref(mi)))
        return {"cond_func": f, "cond_cdf": c, "cond_func_int": fi, "marg_cdf": mc, "marg_func_int": mi.value}

    def close(self):
        if getattr(self, "_h", None):
            lib().ptrs_scene_destroy(self._h)
            self._h = None

    __del__ = close

    def world_bound(self):
        out = (C.c_float * 6)()
        _check(lib().ptrs_scene_world_bound(self._h, out))
        return np.array(out[:3], dtype=np.float32), np.array(out[3:], dtype=np.float32)

    @property
    def device_bytes(self):
        return lib().ptrs_scene_device_bytes(self._h)

    def intersect(self, rays):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        _check(lib().ptrs_intersect(self._h, _p(rays, PtrsRay), rays.shape[0], _p(hits, PtrsHit)))
        return hits

    def intersect_p(self, rays):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        occ = np.empty(rays.shape[0], dtype=np.uint8)
        _check(lib().ptrs_intersect_p(self._h, _p(rays, PtrsRay), rays.shape[0], _p(occ, C.c_uint8)))
        return occ

    def intersect_device(self, d_rays, n, d_hits, stream=0):
        _check(lib().ptrs_intersect_device(self._h, C.c_void_p(d_rays), n, C.c_void_p(d_hits), C.c_void_p(stream)))

    def intersect_p_device(self, d_rays, n, d_occ, stream=0):
        _check(lib().ptrs_intersect_p_device(self._h, C.c_void_p(d_rays), n, C.c_void_p(d_occ), C.c_void_p(stream)))

    def intersect_counted_device(self, d_rays, n, d_out, any_hit=False, stream=0):
        nodes, tris = C.c_uint64(0), C.c_uint64(0)
        _check(lib().ptrs_intersect_counted_device(self._h, C.c_void_p(d_rays), n, None if any_hit else C.c_void_p(d_out), 1 if any_hit else 0,
                                                   C.c_void_p(d_out) if any_hit else None, C.byref(nodes), C.byref(tris), C.c_void_p(stream)))
        return nodes.value, tris.value

    def set_stats_mode(self, count_visits):
        _check(lib().ptrs_set_stats_mode(self._h, 1 if count_visits else 0))

    def stats(self):
        st = PtrsStats()
        _check(lib().ptrs_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in PtrsStats._fields_}

    def light_sample(self, light, ref_p, ref_n, u, exact=False):
        """Light::sample_li + the visibility segment for reference points (ptrs_light_sample): (n, 16) rows of
        Li rgb, wi xyz, pdf, segment origin xyz, segment direction xyz, 3 x pad."""
        p, nn, uu = (np.ascontiguousarray(a, dtype=np.float32) for a in (ref_p, ref_n, u))
        n = p.shape[0]
        out = np.empty((n, 16), dtype=np.float32)
        _check(lib().ptrs_light_sample(self._h, light, _p(p, C.c_float), _p(nn, C.c_float), _p(uu, C.c_float), n, 1 if exact else 0, _p(out, C.c_float)))
        return out

    def light_pdf(self, light, ref_p, ref_n, wi, exact=False):
        p, nn, w = (np.ascontiguousarray(a, dtype=np.float32) for a in (ref_p, ref_n, wi))
        n = p.shape[0]
        out = np.empty(n, dtype=np.float32)
        _check(lib().ptrs_light_pdf(self._h, light, _p(p, C.c_float), _p(nn, C.c_float), _p(w, C.c_float), n, 1 if exact else 0, _p(out, C.c_float)))
        return out

    def path_radiance(self, cam, params, pixels, samples):
        px = np.ascontiguousarray(pixels, dtype=np.int32).reshape(-1, 2)
        sm = np.ascontiguousarray(samples, dtype=np.int32).reshape(-1)
        out = np.empty((px.shape[0], 3), dtype=np.float32)
        _check(lib().ptrs_path_radiance(self._h, C.byref(cam), C.byref(params), _p(px, C.c_int32), _p(sm, C.c_int32), px.shape[0],
                                        _p(out, C.c_float)))
        return out


class Comm:
    """One rank of the NCCL communicator the films are reduced over when every GPU has its own process
    (ptrs_comm_*).  Rank 0 calls Comm.unique_id() and ships the 128 bytes to the others by any channel."""

    @staticmethod
    def unique_id():
        buf = (C.c_uint8 * 128)()
        _check(lib().ptrs_comm_unique_id(buf))
        return bytes(buf)

    def __init__(self, unique_id, n_ranks, rank):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        h = C.c_void_p()
        _check(lib().ptrs_comm_init_rank(buf, n_ranks, rank, C.byref(h)))
        self._h, self.n_ranks, self.rank = h, n_ranks, rank

    def reduce_film(self, film, root=0, stream=None):
        """film.rs:213-228 across ranks: sum of all ranks' films into root's, on `stream`."""
        _check(lib().ptrs_film_reduce(self._h, film._h, root, C.c_void_p(stream or 0)))

    def close(self):
        if getattr(self, "_h", None):
            lib().ptrs_comm_destroy(self._h)
            self._h = None

    __del__ = close


class MultiScene:
    """Scene replicas on several devices of this process + the films they reduce into (ptrs_multi_*)."""

    def __init__(self, flat, n_devices, devices=None, device_bvh=False, device_tables=False):
        desc = (flat.desc_device_tables if device_tables else flat.desc) if isinstance(flat, FlatScene) else flat
        h = C.c_void_p()
        dv = (C.c_int32 * n_devices)(*devices) if devices is not None else None
        _check(lib().ptrs_multi_create(desc, n_devices, dv, 1 if device_bvh else 0, C.byref(h)))
        self._h, self.n_devices = h, n_devices

    def render(self, camera, params, download=True, region=None):
        """PathIntegrator::render over all devices.  Returns (raw film sums (H, W, 4) or None, per-device stats, total ms).
        region: a rectangle of sample positions (x0, y0, x1, y1) to trace instead of the whole sample bounds
        (ptrs_multi_render_region); the film is still reduced and downloaded whole."""
        out = np.empty((camera.height, camera.width, 4), dtype=np.float32) if download else None
        st = (PtrsStats * self.n_devices)()
        ms = C.c_float(0)
        host = _p(out, C.c_float) if download else None
        if region is None:
            _check(lib().ptrs_multi_render(self._h, C.byref(camera), C.byref(params), host, st, C.byref(ms)))
        else:
            _check(lib().ptrs_multi_render_region(self._h, C.byref(camera), C.byref(params), _rect(region), host, st, C.byref(ms)))
        stats = [{k: getattr(s, k) for k, _ in PtrsStats._fields_} for s in st]
        return out, stats, ms.value

    def render_into(self, camera, params, host_rgbw):
        """Same, into a caller-owned (H, W, 4) float32 array (e.g. pinned memory)."""
        st = (PtrsStats * self.n_devices)()
        ms = C.c_float(0)
        _check(lib().ptrs_multi_render(self._h, C.byref(camera), C.byref(params), C.cast(C.c_void_p(host_rgbw), C.POINTER(C.c_float)), st, C.byref(ms)))
        return [{k: getattr(s, k) for k, _ in PtrsStats._fields_} for s in st], ms.value

    def to_channel_updates(self, width, height):
        f = C.c_void_p()
        _check(lib().ptrs_multi_root_film(self._h, C.byref(f)))
        out = np.empty((height, width, 3), dtype=np.float32)
        _check(lib().ptrs_film_resolve(f, _p(out, C.c_float)))
        return out

    def close(self):
        if getattr(self, "_h", None):
            lib().ptrs_multi_destroy(self._h)
            self._h = None

    __del__ = close


class SamplerBuilder:
    """SobolSamplerBuilder::new(log, spp, sample_bounds) — sampler/sobol.rs:35-62.  The seed is ignored
    exactly like the reference's `with_seed` (sobol.rs:75-77)."""

    def __init__(self, samples_per_pixel, sample_bounds=None):
        self.samples_per_pixel = int(samples_per_pixel)
        self.sample_bounds = sample_bounds

    def with_seed(self, _seed):
        return self


class PathIntegrator:
    """PathIntegrator::new(log, sampler_builder, max_depth, show_progress_bar) — integrator.rs:230."""

    def __init__(self, sampler_builder, max_depth=15, show_progress_bar=False):
        self.params = default_render_params(sampler_builder.samples_per_pixel, max_depth)
        self.show_progress_bar = show_progress_bar

    def preprocess(self, scene):  # integrator.rs:250-258
        self.too_many_lights = scene.n_lights > 16

    def render(self, camera, scene, film, stream=None, sample_range=None, sample_stride=(1, 0), exact_shading=False, region=None):
        """integrator.rs:536 — accumulates into `film` (the reference's camera.film).  sample_range /
        sample_stride select a shard of the Sobol sample numbers (multi-GPU); exact_shading selects the parity
        build of the shade kernels (PTRS_RENDER_EXACT_SHADING); region (x0, y0, x1, y1) traces only that rectangle of
        sample positions (ptrs_render_region; Film.region_sample_rect gives the one that completes a pixel crop)."""
        p = PtrsRenderParams.from_buffer_copy(self.params)
        if exact_shading:
            p.flags |= RENDER_EXACT_SHADING
        if sample_range is not None:
            p.sample_begin, p.sample_end = sample_range
        p.sample_stride, p.sample_phase = sample_stride
        if region is None:
            _check(lib().ptrs_render(scene._h, C.byref(camera), C.byref(p), film._h, C.c_void_p(stream or 0)))
        else:
            _check(lib().ptrs_render_region(scene._h, C.byref(camera), C.byref(p), _rect(region), film._h, C.c_void_p(stream or 0)))
        return scene.stats()


def bxdf_eval(lobe, wo, wi, exact=False):
    """BxDF::f and BxDF::pdf of one lobe (ptrs_bxdf_eval): (n, 4) rows of f rgb, pdf."""
    o, w = np.ascontiguousarray(wo, dtype=np.float32), np.ascontiguousarray(wi, dtype=np.float32)
    out = np.empty((o.shape[0], 4), dtype=np.float32)
    _check(lib().ptrs_bxdf_eval(C.byref(lobe), _p(o, C.c_float), _p(w, C.c_float), o.shape[0], 1 if exact else 0, _p(out, C.c_float)))
    return out


def bxdf_sample(lobe, wo, u, exact=False):
    """BxDF::sample_f of one lobe (ptrs_bxdf_sample): (n, 8) rows of wi xyz, f rgb, pdf, sampled type bits."""
    o, uu = np.ascontiguousarray(wo, dtype=np.float32), np.ascontiguousarray(u, dtype=np.float32)
    out = np.empty((o.shape[0], 8), dtype=np.float32)
    _check(lib().ptrs_bxdf_sample(C.byref(lobe), _p(o, C.c_float), _p(uu, C.c_float), o.shape[0], 1 if exact else 0, _p(out, C.c_float)))
    return out


def sobol_samples(cam, params, pixels, samples, dims):
    px = np.ascontiguousarray(pixels, dtype=np.int32).reshape(-1, 2)
    sm = np.ascontiguousarray(samples, dtype=np.int32).reshape(-1)
    dm = np.ascontiguousarray(dims, dtype=np.int32)
    out = np.empty((px.shape[0], dm.shape[0]), dtype=np.float32)
    idx = np.empty(px.shape[0], dtype=np.uint64)
    _check(lib().ptrs_sobol_samples(C.byref(cam), C.byref(params), _p(px, C.c_int32), _p(sm, C.c_int32), px.shape[0], _p(dm, C.c_int32),
                                    dm.shape[0], _p(out, C.c_float), _p(idx, C.c_uint64)))
    return out, idx


def generate_rays(cam, params, pixels, samples):
    px = np.ascontiguousarray(pixels, dtype=np.int32).reshape(-1, 2)
    sm = np.ascontiguousarray(samples, dtype=np.int32).reshape(-1)
    n = px.shape[0]
    rays = np.empty(n, dtype=RAY_DTYPE)
    pf = np.empty((n, 2), dtype=np.float32)
    rxry = np.empty((n, 6), dtype=np.float32)
    _check(lib().ptrs_generate_rays(C.byref(cam), C.byref(params), _p(px, C.c_int32), _p(sm, C.c_int32), n, _p(rays, PtrsRay),
                                    _p(pf, C.c_float), _p(rxry, C.c_float)))
    return rays, pf, rxry
