"""Per-path radiance of the exact-shading build (PTRS_RENDER_EXACT_SHADING) on the test scenes, written to one .npz, so
that two builds of the library can be compared bit for bit:

    PTRS_B200_LIB=/path/to/other/libptrs_b200.so python tools/shade_parity.py a.npz
    python tools/shade_parity.py b.npz
    python tools/shade_parity.py --compare a.npz b.npz

Scenes: Cornell, Cornell + the tank-farm HDR, the material field, the atrium and an alpha-masked glTF scene."""
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SPP, DEPTH, N_PATHS = 16, 15, 40000


def scenes(host):
    yield "cornell", host.make_scene(host.SCENE_CORNELL, res=(96, 96))
    yield "cornell_env", host.make_scene(host.SCENE_CORNELL_ENV, seed=1, res=(96, 96), env_hdr=host.TANK_FARM_HDR)
    yield "field", host.make_scene(host.SCENE_MATERIAL_FIELD, seed=1, n_tris=60000, res=(96, 64))
    yield "atrium", host.make_scene(host.SCENE_ATRIUM, seed=1, n_tris=40000, res=(96, 54))
    from test_gltf_import import write_gltf

    with tempfile.TemporaryDirectory() as d:
        path, _ = write_gltf(host, pathlib.Path(d), "glb")
        yield "gltf", host.import_scene(path, res=(96, 64), default_lights=True)


def dump(out):
    import pathtracer_rs_b200.gpu as gpu
    import pathtracer_rs_b200.host as host

    gpu.set_device(0)
    res = {}
    for name, (flat, cam) in scenes(host):
        scene = gpu.RenderScene(flat)
        rng = np.random.default_rng(3)
        pixels = np.stack([rng.integers(0, cam.width, N_PATHS), rng.integers(0, cam.height, N_PATHS)], axis=1)
        samples = rng.integers(0, SPP, N_PATHS)
        integ = gpu.PathIntegrator(gpu.SamplerBuilder(SPP), max_depth=DEPTH)
        integ.preprocess(scene)
        params = integ.params
        params.flags |= gpu.RENDER_EXACT_SHADING
        res[name] = scene.path_radiance(cam, params, pixels, samples)
        scene.close()
    np.savez(out, **res)
    print("wrote", out, "from", gpu.LIB_PATH)


def compare(a, b):
    A, B = np.load(a), np.load(b)
    ok = True
    for k in A.files:
        same = np.array_equal(A[k].view(np.uint32), B[k].view(np.uint32))
        ok &= same
        print(f"{k}: {'bit-identical' if same else 'DIFFERENT'} ({np.count_nonzero(A[k])} non-zero values of {A[k].size})")
    return ok


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
    dump(sys.argv[1])
