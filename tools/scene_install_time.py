"""Scene install and BVH build times on one GPU -> profiles/scene_install.json (DESIGN.md §5 K8).

Per sweep scene of n spheres (generated on the CPU by the oracle, the same list for every build):
  - host upload (rtz_scene_upload) and device upload from a CUDA tensor (rtz_scene_upload_device), ms;
  - the host and the device BVH builder (rtz_probe_bvh without outputs), ms;
  - the first RTZ_MODE_PATH_BVH frame at 1200x675, 16 spp, from the start of the install to the bytes on the device:
    the parent build (host upload, host BVH) against this one (device upload, BVH builder chosen by size), each round
    in fresh processes, the builds alternated, best of 3, with the frames' bytes compared;
  - a steady BVH frame (scene and BVH in place), for scale.

    python tools/scene_install_time.py [--parent-lib PATH] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
SIZES = [4096, 16384, 65536, 262144, 1 << 20]


def _ms(fn, sync):
    sync()
    t = time.perf_counter()
    fn()
    sync()
    return (time.perf_counter() - t) * 1e3


def worker(mode: str, n: int) -> dict:
    """One process: mode 'parent' (host upload + host BVH, the only path the parent has) or 'this'."""
    sys.path.insert(0, str(ROOT)), sys.path.insert(0, str(ROOT / "tests"))
    import importlib

    import numpy as np
    import torch
    import rtzlib as R

    pkg = importlib.import_module("raytracing-with-zig_b200")
    orc = R.oracle()
    prng = orc.orc_prng_new(7)
    sp = (R.Sphere * n)()
    assert orc.orc_generate_sweep(prng, n, sp) == n
    orc.orc_prng_free(prng)
    t = torch.from_numpy(np.frombuffer(bytes(sp), np.float64).reshape(n, 10).copy()).cuda()
    cam = R.main_camera(1200, 16, seed=0x5EED)
    cam.mode = R.MODE_PATH_BVH
    sync = torch.cuda.synchronize
    r = pkg.Renderer(0)
    warm = R.main_camera(64, 1, seed=1)
    warm.mode = R.MODE_PATH_BVH
    r.upload(sp, n), r.render(warm)  # modules loaded, buffers sized
    if mode == "this":
        r.upload(t), r.render(warm)
    out = torch.empty((675, 1200, 3), dtype=torch.uint8, device="cuda:0")
    src = sp if mode == "parent" else t
    first = _ms(lambda: (r.upload(src, n), r.render(cam, out=out)), sync)
    digest = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()
    res = {"first_frame_ms": first, "sha256": digest}
    if mode == "this":
        l = r.lib
        res["host_upload_ms"] = min(_ms(lambda: r.upload(sp, n), sync) for _ in range(3))
        res["device_upload_ms"] = min(_ms(lambda: r.upload(t), sync) for _ in range(3))
        cnt = C.c_uint64()
        for name, b in (("host_bvh_ms", 0), ("device_bvh_ms", 1)):
            res[name] = min(_ms(lambda: l.rtz_probe_bvh(r._ctx, b, None, 0, None, None, C.byref(cnt)), sync)
                            for _ in range(3))
        res["steady_bvh_frame_ms"] = min(_ms(lambda: r.render(cam, out=out), sync) for _ in range(3))
    r.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="librtz.so of the parent build (A/B of the first frame)")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "scene_install.json"))
    ap.add_argument("--sizes", default=",".join(map(str, SIZES)))
    ap.add_argument("--worker", nargs=2, metavar=("MODE", "N"))
    a = ap.parse_args()
    if a.worker:
        print(json.dumps(worker(a.worker[0], int(a.worker[1]))))
        return
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]

    def run(mode, n):
        env = dict(os.environ)
        if mode == "parent":
            env["RTZ_LIB"] = a.parent_lib
        p = subprocess.run([sys.executable, __file__, "--worker", mode, str(n)], capture_output=True, text=True, env=env,
                           cwd=ROOT)
        if p.returncode:
            raise RuntimeError(p.stdout + p.stderr)
        return json.loads(p.stdout.strip().splitlines()[-1])

    rows = []
    for n in [int(s) for s in a.sizes.split(",")]:
        this, parent = [], []
        for _ in range(3):
            if a.parent_lib:
                parent.append(run("parent", n))
            this.append(run("this", n))
        row = {"spheres": n}
        for k in ("host_upload_ms", "device_upload_ms", "host_bvh_ms", "device_bvh_ms", "steady_bvh_frame_ms"):
            row[k] = round(min(r[k] for r in this), 3)
        row["first_bvh_frame_ms"] = round(min(r["first_frame_ms"] for r in this), 3)
        if parent:
            row["parent_first_bvh_frame_ms"] = round(min(r["first_frame_ms"] for r in parent), 3)
            row["same_frame_as_parent"] = len({r["sha256"] for r in this + parent}) == 1
        rows.append(row)
        print(json.dumps(row), flush=True)
    doc = {"gpu": gpu, "frame": "1200x675, 16 spp, RTZ_MODE_PATH_BVH, sweep scene (seed 7)",
           "method": "host clock around work ended by a device synchronise; fresh processes, parent and this build "
                     "alternated, best of 3; BVH builds through rtz_probe_bvh without outputs",
           "rows": rows}
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(doc, indent=1) + "\n")


if __name__ == "__main__":
    main()
