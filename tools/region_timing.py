#!/usr/bin/env python
"""Step time of ptrs_render_region against the rectangle's area: C5's scene (the 262k-triangle atrium, 3840x2160,
max_depth 15) at 16 spp, for the full frame and for centred pixel crops of 1/4, 1/16 and 1/256 of its area, each
completed by ptrs_film_region_sample_rect.  Shows where the per-call costs that do not shrink with the area (batch
tail rounds, launches) take over.  The Sobol split tables are built by the first render of a scene and reused by
every later one; the cold first call is reported on its own line.  Prints the card's name and power limit.
usage: python tools/region_timing.py [--spp 16] [--reps 5] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import pathtracer_rs_b200.gpu as gpu  # noqa: E402
import pathtracer_rs_b200.host as host  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        raise RuntimeError("nvidia-smi query failed: " + q.stderr)
    return q.stdout.strip()


def timed(integ, cam, scene, film, region):
    film.clear()
    t0 = time.perf_counter()
    st = integ.render(cam, scene, film, region=region)  # returns after the render's final stream synchronise
    return (time.perf_counter() - t0) * 1e3, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if gpu.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to time")
    gpu.set_device(0)
    print("card (name, power limit, max SM clock):", card())
    flat, cam = host.make_scene(host.SCENE_ATRIUM, seed=1, n_tris=262144, res=(3840, 2160))
    scene = gpu.RenderScene(flat)
    integ = gpu.PathIntegrator(gpu.SamplerBuilder(a.spp), max_depth=15)
    film = gpu.Film(cam.width, cam.height)
    W, H = cam.width, cam.height
    rows = []
    for name, div in (("full", 1), ("1/4", 2), ("1/16", 4), ("1/256", 16)):
        w, h = W // div, H // div
        crop = ((W - w) // 2, (H - h) // 2, (W - w) // 2 + w, (H - h) // 2 + h)
        rect = film.region_sample_rect(crop)
        wall_cold, st = timed(integ, cam, scene, film, rect)
        if name == "full":
            print(f"cold first call (workspace allocation, split-table build, module load): {wall_cold:.1f} ms wall")
        runs = [timed(integ, cam, scene, film, rect) for _ in range(a.reps)]
        wall = np.array([r[0] for r in runs])
        dev = np.array([r[1]["ms_total"] for r in runs])
        st = runs[-1][1]
        row = {"crop": name, "pixel_rect": crop, "sample_rect": rect, "camera_paths": st["camera_paths"],
               "device_ms_median": float(np.median(dev)), "device_ms_min": float(dev.min()), "device_ms_max": float(dev.max()),
               "wall_ms_median": float(np.median(wall)), "msamples_per_s": st["camera_paths"] / float(np.median(dev)) / 1e3,
               "batches": st["batches"], "launches": st["launches"],
               "stages_ms": {k: st["ms_" + k] for k in ("generate", "extend", "shade", "shadow", "accumulate")}}
        rows.append(row)
        print(f"{name:>6} crop {crop} -> samples {rect}: {st['camera_paths']:>10} paths  device {row['device_ms_median']:8.2f} ms "
              f"(min {row['device_ms_min']:.2f}, max {row['device_ms_max']:.2f})  wall {row['wall_ms_median']:8.2f} ms  "
              f"{row['msamples_per_s']:6.1f} M samples/s  batches {st['batches']}  launches {st['launches']}  "
              + " ".join(f"{k} {v:.2f}" for k, v in row["stages_ms"].items()))
    full = rows[0]["device_ms_median"]
    for r in rows[1:]:
        share = r["camera_paths"] / rows[0]["camera_paths"]
        print(f"{r['crop']:>6}: {share:.4f} of the full frame's paths, {r['device_ms_median'] / full:.4f} of its time")
    if a.out:
        with open(a.out, "w") as f:
            json.dump({"card": card(), "spp": a.spp, "reps": a.reps, "rows": rows}, f, indent=1)
    scene.close()


if __name__ == "__main__":
    main()
