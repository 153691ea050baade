"""Cost of a denoised frame on N GPUs (rtz_multi_render_denoised) against the 1-GPU rtz_render_denoised.

Frames (final scene, seed 0xdeadbeef, main camera, g = 16, default params): C3 (1200x675) and C4 (3840x2160) at
16 spp, C3 at 500 spp.  For each device count the box has (1 / 2 / 4 / 8) and each transport (P2P, NCCL), in one
process:
  multi        rtz_multi_render_denoised: total_ms (first launch -> denoised bytes on device 0), trace_ms (slowest
               device's path trace), gather_ms (the denoiser's inputs on device 0, minus trace_ms), and whether the
               frame equals the 1-GPU frame bit for bit;
  per device   each rank's tiles traced (Renderer.render_linear, trace_ms) and its guide kernel
               (Renderer.render_guides(shard=...), trace_ms), each device on its own;
  denoise      the whole frame denoised on device 0 (Renderer.denoise, total_ms);
  one GPU      rtz_render_denoised: total_ms.
Best of --rounds calls after one warm-up call of every shape.  Device counts the box does not have are recorded as
not measured.

    python tools/multi_denoise_time.py [--out profiles/multi_denoise.json]
"""
import argparse
import importlib
import json
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import rtzlib as R  # noqa: E402

FRAMES = (("C3", 1200, 16), ("C4", 3840, 16), ("C3", 1200, 500))
G = 16


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "devices": torch.cuda.device_count(),
            "nvidia_smi": q.stdout.strip().splitlines()}


def best(fn, rounds):
    fn()  # warm-up of the shape
    return min((fn() for _ in range(rounds)), key=lambda v: v if isinstance(v, float) else v[0])


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/multi_denoise.json")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    pkg = importlib.import_module("raytracing-with-zig_b200")
    ngpu = torch.cuda.device_count()
    _, sp, n = R.final_scene(0xDEADBEEF)
    renderers = []
    for d in range(ngpu):
        r = pkg.Renderer(d)
        r.upload(sp, n)
        renderers.append(r)
    rows = []
    for name, width, spp in FRAMES:
        cam = R.main_camera(width, spp, seed=0xDEADBEEF)
        W, H = int(cam.width), int(cam.height)
        frame = {"frame": name, "width": W, "height": H, "spp": spp, "g": G}
        ref = {}

        def one_gpu():
            rgb, lin, st = pkg.render_host_denoised(cam, sp, n, G)
            ref["rgb"], ref["lin"] = rgb, lin
            return st.total_ms

        one_ms = best(one_gpu, args.rounds)
        r0 = renderers[0]
        lin0 = r0.render_linear(cam)[1]
        alb0, nrm0, _ = r0.render_guides(cam, G)
        denoise_ms = best(lambda: r0.denoise(lin0, alb0, nrm0)[2].total_ms, args.rounds)
        del lin0, alb0, nrm0
        rows.append(dict(frame, gpus=1, path="rtz_render_denoised", total_ms=one_ms, denoise_ms_device0=denoise_ms))
        for world in (1, 2, 4, 8):
            for gather in ("p2p", "nccl"):
                if world == 1 and gather == "nccl":
                    continue
                row = dict(frame, gpus=world, gather=gather if world > 1 else None)
                if world > ngpu:
                    rows.append(dict(row, measured=False, reason=f"the box has {ngpu} GPU(s)"))
                    continue
                m = pkg.MultiRenderer(world, gather=gather)
                m.upload(sp, n)
                out = {}

                def multi():
                    rgb, lin, st = m.render_denoised(cam, G)
                    out["equal"] = bool(np.array_equal(rgb, ref["rgb"]) and
                                        np.array_equal(lin.view(np.uint32), ref["lin"].view(np.uint32)))
                    return st.total_ms, st.trace_ms, st.gather_ms, st.kernel_launches

                total, trace, gath, launches = best(multi, args.rounds)
                m.close()
                per_dev = []
                for rank in range(world):
                    r = renderers[rank]
                    shard = pkg.rtz_shard(rank, world, 4, 4)
                    tr = best(lambda: r.render_linear(cam, shard=shard)[2].trace_ms, args.rounds)
                    gd = best(lambda: r.render_guides(cam, G, shard=shard)[2].trace_ms, args.rounds)
                    per_dev.append({"device": rank, "trace_ms": tr, "guide_ms": gd})
                rows.append(dict(row, measured=True, total_ms=total, trace_ms_slowest=trace, gather_ms=gath,
                                 kernel_launches=launches, per_device=per_dev, denoise_ms_device0=denoise_ms,
                                 denoise_share_of_total=denoise_ms / total, one_gpu_total_ms=one_ms,
                                 speedup_vs_one_gpu=one_ms / total, equals_one_gpu_frame=out["equal"]))
                print(json.dumps({k: rows[-1][k] for k in ("frame", "spp", "gpus", "gather", "total_ms",
                                                           "trace_ms_slowest", "gather_ms", "equals_one_gpu_frame")}),
                      flush=True)
    for r in renderers:
        r.close()
    res = {"card": card(), "tile": [4, 4], "rows": rows}
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "measured_rows": sum(1 for r in rows if r.get("measured", True))}))


if __name__ == "__main__":
    main()
