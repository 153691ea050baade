"""Scenes beside C3 that the culled sweep's block order can speed up or slow down (development aid): one JSON line per
scene with the best render time of a few and the image's sha256, for A/B runs of two builds (RTZ_LIB=<lib>).

  C5 N=512   the sphere sweep scene of 512 spheres (tools/c5_quick.py), 1920x1080, 64 spp
  cube       485 spheres of radius 0.2 scattered uniformly through the cube [-4, 4]^3 (seeded), the main camera,
             1200x675, 32 spp: a scene without a ground grid, where even regrouped blocks overlap along most rays
"""
import hashlib
import importlib
import json
import sys

import numpy as np

sys.path.insert(0, '.')
sys.path.insert(0, 'tests')
import rtzlib as R  # noqa: E402

pkg = importlib.import_module("raytracing-with-zig_b200")
host = importlib.import_module("raytracing-with-zig_b200.host_api")


def cube_scene(n=485, seed=485):
    rng = np.random.default_rng(seed)
    sp = []
    for _ in range(n):
        c = tuple(rng.uniform(-4.0, 4.0, 3))
        kind = rng.random()
        if kind < 0.6:
            sp.append(R.make_sphere(c, 0.2, R.MAT_LAMBERTIAN, tuple(0.2 + 0.6 * rng.random(3))))
        elif kind < 0.85:
            sp.append(R.make_sphere(c, 0.2, R.MAT_METAL, tuple(0.5 + 0.5 * rng.random(3)), fuzz=0.3))
        else:
            sp.append(R.make_sphere(c, 0.2, R.MAT_DIELECTRIC, ior=1.5))
    return R.sphere_array(sp), n


def timed(r, cam, reps):
    best, img = None, None
    for _ in range(reps):
        img, st = r.render(cam)
        best = st.total_ms if best is None else min(best, st.total_ms)
    return best, hashlib.sha256(img.cpu().numpy().tobytes()).hexdigest()[:16]


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    r = pkg.Renderer(0)
    sp, _ = host.generate_sweep(0xDEADBEEF, 512)
    r.upload(sp, 512)
    ms, h = timed(r, host.main_camera(1920, 64, seed=0xDEADBEEF), reps)
    print(json.dumps({"scene": "c5_n512", "ms": round(ms, 3), "sha": h}), flush=True)
    sp, n = cube_scene()
    r.upload(sp, n)
    ms, h = timed(r, R.main_camera(1200, 32, seed=0xDEADBEEF), reps)
    print(json.dumps({"scene": "cube485", "ms": round(ms, 3), "sha": h}), flush=True)
    r.close()


if __name__ == "__main__":
    main()
