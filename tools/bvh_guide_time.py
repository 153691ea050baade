"""Guides of large BVH-mode scenes: the brute-force guide pass (guide_kernel_global) against the BVH one
(guides_kernel_bvh), and the denoised BVH frame (rtz_render_denoised) before and after.

Every measurement runs in a worker process per build (RTZ_LIB), the parent build and this one alternated, `--rounds`
rounds; the best of the rounds is kept.  Times are the calls' own CUDA-event times on the context's stream:
render_guides' trace_ms (the guide kernel alone) and render_host_denoised's total_ms (render, guides and denoise).

- guide pass: 1200x675, g = 16, sweep scenes of 600, 1 024, 4 096 and 16 384 spheres; RTZ_MODE_PATH_BVH (the BVH
  kernel in this build, the global-memory sweep in the parent) and RTZ_MODE_PATH (the global-memory sweep in both);
- denoised frame: 1200x675, 16 spp, guides of 16 samples, RTZ_MODE_PATH_BVH, at 4 096 and 16 384 spheres, with the
  guides' share of the frame (guide pass / total);
- below the threshold, in BVH mode: the final scene (485 spheres, the culled constant-bank sweep) and the 512-sphere
  sweep scene (the plain one), each also with spheres added inside the radius-1000 ground sphere, where no camera
  ray reaches them (517 and 544 spheres: the BVH kernel, on the same hits).

    python tools/bvh_guide_time.py --parent <parent librtz.so> [--out profiles/bvh_guides.json]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import rtzlib as R  # noqa: E402

SWEEPS = (600, 1024, 4096, 16384)
DENOISED = (4096, 16384)
G = 16


def sweep_scene(n):
    orc = R.oracle()
    prng = orc.orc_prng_new(7)
    buf = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, buf) == n
    orc.orc_prng_free(prng)
    return buf


def with_hidden(sp, n, k):
    """sp + k spheres of radius 0.5 inside the ground sphere (centre (0, -1000, 0), radius 1000), 20 below its top"""
    hidden = [R.make_sphere((2.0 * (i % 6) - 5, -20.0, 2.0 * (i // 6) - 5), 0.5, R.MAT_LAMBERTIAN) for i in range(k)]
    return R.sphere_array(list(sp)[:n] + hidden), n + k


def worker():
    """One build's measurements (RTZ_LIB), one JSON line on stdout."""
    import torch
    pkg = importlib.import_module("raytracing-with-zig_b200")
    cam = R.main_camera(1200, 16, seed=0xDEADBEEF)
    r = pkg.Renderer(0)
    res = {}

    def guide_ms(sp, n, mode):
        cam.mode = mode
        r.upload(sp, n)
        r.render_guides(cam, G)                       # warm-up (and the BVH build)
        _, _, st = r.render_guides(cam, G)
        return st.trace_ms, st.sphere_tests

    for n in SWEEPS:
        sp = sweep_scene(n)
        for mode, name in ((R.MODE_PATH_BVH, "bvh"), (R.MODE_PATH, "path")):
            ms, tests = guide_ms(sp, n, mode)
            res[f"guides n={n} {name}"] = {"ms": ms, "sphere_tests": tests}
    _, fs, fn = R.final_scene(0xDEADBEEF)
    small = ((fs, fn, "final 485"), (sweep_scene(512), 512, "n=512"))
    for sp, n, tag in small:
        ms, tests = guide_ms(sp, n, R.MODE_PATH_BVH)
        res[f"guides {tag} bvh"] = {"ms": ms, "sphere_tests": tests}
        ms, tests = guide_ms(*with_hidden(sp, n, 32), R.MODE_PATH_BVH)
        res[f"guides {tag} + 32 hidden bvh"] = {"ms": ms, "sphere_tests": tests}
    cam.mode = R.MODE_PATH_BVH
    for sp, n, tag in [(sweep_scene(n), n, f"n={n}") for n in DENOISED] + [(fs, fn, "final 485")]:
        pkg.render_host_denoised(cam, sp, n, G)      # warm-up
        _, _, st = pkg.render_host_denoised(cam, sp, n, G)
        res[f"denoised {tag} bvh"] = {"ms": st.total_ms, "trace_ms": st.trace_ms}
    r.close()
    torch.cuda.synchronize()
    print(json.dumps(res))


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", required=True, help="librtz.so of the parent commit")
    ap.add_argument("--out", default="profiles/bvh_guides.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--worker", action="store_true")
    args = ap.parse_args()
    if args.worker:
        return worker()
    libs = {"parent": str(Path(args.parent).resolve()), "this": str(ROOT / "raytracing-with-zig_b200" / "csrc" / "librtz.so")}
    info = card()
    rows = []
    for rnd in range(args.rounds):
        for build, lib in libs.items():
            p = subprocess.run([sys.executable, __file__, "--worker", "--parent", args.parent],
                               env=dict(os.environ, RTZ_LIB=lib), capture_output=True, text=True, check=True)
            rows.append({"round": rnd, "build": build, "results": json.loads(p.stdout.strip().splitlines()[-1])})
    best = {}
    for row in rows:
        for k, v in row["results"].items():
            key = (row["build"], k)
            best[key] = min(best.get(key, v), v, key=lambda x: x["ms"])
    summary = {}
    for (build, k), v in sorted(best.items()):
        summary.setdefault(k, {})[build] = v
    for n in DENOISED:
        for build in libs:
            gk = f"guides n={n} bvh"
            dk = f"denoised n={n} bvh"
            summary[dk][build]["guide_share"] = summary[gk][build]["ms"] / summary[dk][build]["ms"]
    out = {"frame": {"width": 1200, "height": 675, "guide_samples": G, "denoised_spp": 16, "camera": "main_camera"},
           "card": info, "rounds": args.rounds, "rows": rows, "best": summary}
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"card": info, "best": summary}))


if __name__ == "__main__":
    main()
