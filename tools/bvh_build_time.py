#!/usr/bin/env python
"""BVH build timing: python tools/bvh_build_time.py [--scene K] [--tris N] [--reps K]

Per scene: the host SAH build (SceneBuilder::finalize, with its thread count), the reference's SAH tree built on the
device (ptrs_scene_create_sah_bvh) with the copy-back + host collapse of its occlusion tree reported separately, and the
PLOC build (ptrs_scene_create_device_bvh).  Every device figure is the library's own event timing of the build; each
build runs once as a warm-up before the timed reps."""
import argparse
import os
import re
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pathtracer_rs_b200.gpu as gpu  # noqa: E402
import pathtracer_rs_b200.host as host  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--tris", type=int, default=10_000_000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--scene", type=int, default=host.SCENE_TERRAIN)
ap.add_argument("--threads", type=int, default=0, help="host build threads (0: all)")
a = ap.parse_args()


def collapse_ms(flat):
    """copy-back + host collapse of the occlusion tree, as the library prints it under PTRS_BVH_DEBUG (stderr of this
    process, captured through a temporary file)"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        os.environ["PTRS_BVH_DEBUG"] = "1"
        try:
            gpu.RenderScene(flat, sah_on_device=True).close()
        finally:
            del os.environ["PTRS_BVH_DEBUG"]
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        m = re.search(r"occlusion tree \(copy-back \+ host collapse\)\s+([0-9.]+) ms", f.read())
    return float(m.group(1)) if m else float("nan")


gpu.set_device(0)
flat, cam = host.make_scene(a.scene, seed=1, n_tris=a.tris, res=(256, 256), n_threads=a.threads)
threads = a.threads or len(os.sched_getaffinity(0))
print(f"tris={flat.n_prims} host SAH build {flat.bvh_seconds * 1e3:.0f} ms ({threads} threads), host-tree depth {flat.bvh_depth}")
for name, kw in (("device SAH", {"sah_on_device": True}), ("PLOC", {"device_bvh": True})):
    gpu.RenderScene(flat, **kw).close()  # warm-up
    for _ in range(a.reps):
        s = gpu.RenderScene(flat, **kw)
        n, ms = s.bvh_info()
        print(f"{name} build: nodes {n}, {ms:.2f} ms")
        s.close()
for _ in range(a.reps):
    print(f"device SAH: occlusion tree copy-back + host collapse {collapse_ms(flat):.1f} ms")
