"""Cost and payoff of the à-trous denoiser (rtz_denoise, DESIGN.md §5 K7) on the C3 frame (final scene, seed 0xdeadbeef,
main_camera(1200, ...)), in one process on one GPU:

  times    denoise of C3 at L = 1 .. 5 and of C4 (3840x2160) at L = 5 (the calls' own total_ms: CUDA events on the
           context's stream), best of --rounds alternated rounds, beside the 500-spp render (trace_ms);
  bounds   FP32 operations and DRAM bytes counted here from the frame size and the kernels' arithmetic, against the
           FP32 pipe (rtz_measure_fp32_peak, scalar FFMA) and 7.7 TB/s of HBM; the level pass's time is the slope of
           the L = 1 .. 5 times, prepare + finish their intercept;
  quality  RMSE of the linear colour against a 4 096-spp render of another seed, for noisy 16 .. 500 spp and for
           16 and 64 spp denoised at the defaults (guides of 16 samples), with each frame's device time.

    python tools/denoise_time.py [--out profiles/denoise_c3.json]
"""
import argparse
import ctypes as C
import importlib
import json
import math
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import rtzlib as R  # noqa: E402

HBM_BPS = 7.7e12
# FP32 operations per tap (an FMA counts 2): three squared distances (3 sub, 1 mul, 2 fma = 8 each), three scalings,
# three E(x) (fma, max, six squarings = 9 each), four weight products, three (sub + fma) and one add of the sums
FLOP_PER_TAP = 3 * 8 + 3 + 3 * 9 + 4 + 3 * 3 + 1
FLOP_PER_PIXEL_LEVEL_FIXED = 3 + 3   # three divisions (counted once each) and three adds
BYTES_PER_PIXEL_LEVEL = 3 * 16 + 16  # read e, normal, albedo planes once, write e
BYTES_PREPARE = 3 * 12 + 3 * 16      # colour, albedo, normal in; e, normal, albedo planes out
BYTES_FINISH = 16 + 12 + 12 + 3      # e plane and albedo in; linear and bytes out
SPPS = (16, 64, 128, 256, 500)


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def taps(W, H, step):
    """Taps inside the image summed over all pixels at one level."""
    return sum(max(0, H - abs(i - 2) * step) * max(0, W - abs(j - 2) * step) for i in range(5) for j in range(5))


def level_flops(W, H, step):
    return taps(W, H, step) * FLOP_PER_TAP + W * H * FLOP_PER_PIXEL_LEVEL_FIXED


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/denoise_c3.json")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    pkg = importlib.import_module("raytracing-with-zig_b200")
    import torch
    _, sp, n = R.final_scene(0xDEADBEEF)
    r = pkg.Renderer(0)
    r.upload(sp, n)
    peak = C.c_double(0)
    pkg.binding.check(pkg.lib().rtz_measure_fp32_peak(0, 0, C.byref(peak)))
    fp32_flops = peak.value * 1e12

    def inputs(width, spp, seed=0xDEADBEEF, g=16):
        cam = R.main_camera(width, spp, seed=seed)
        _, lin, st = r.render_linear(cam)
        alb, nrm, gst = r.render_guides(cam, min(g, spp))
        return lin, alb, nrm, st, gst

    c3 = inputs(1200, 16)
    c4 = inputs(3840, 16)
    W3, H3 = 1200, 675
    prm = lambda L: pkg.rtz_denoise_params(L, 0, 0.25, 0.25, 0.25)  # noqa: E731  (the defaults, levels varied)
    cam500 = R.main_camera(1200, 500, seed=0xDEADBEEF)
    for L in range(1, 6):                                              # warm-up of every shape timed below
        r.denoise(*c3[:3], params=prm(L))
    r.denoise(*c4[:3], params=prm(5))
    r.render(cam500)
    rows = []
    for rnd in range(args.rounds):
        _, st = r.render(cam500)
        rows.append({"round": rnd, "pass": "render C3 500 spp", "ms": st.trace_ms})
        for L in range(1, 6):
            _, _, ds = r.denoise(*c3[:3], params=prm(L))
            rows.append({"round": rnd, "pass": f"denoise C3 L={L}", "ms": ds.total_ms, "launches": ds.kernel_launches})
        _, _, ds = r.denoise(*c4[:3], params=prm(5))
        rows.append({"round": rnd, "pass": "denoise C4 L=5", "ms": ds.total_ms, "launches": ds.kernel_launches})
    best = {}
    for row in rows:
        best[row["pass"]] = min(best.get(row["pass"], row["ms"]), row["ms"])
    t = [best[f"denoise C3 L={L}"] for L in range(1, 6)]
    slope, intercept = np.polyfit(np.arange(1, 6), t, 1)

    def bound(flops, nbytes, ms):
        tc, tm = flops / fp32_flops, nbytes / HBM_BPS
        return {"flop": flops, "bytes": nbytes, "ms": ms, "achieved_tflops": flops / ms * 1e-9,
                "achieved_tbps": nbytes / ms * 1e-9, "fp32_bound_ms": tc * 1e3, "hbm_bound_ms": tm * 1e3,
                "bound_by": "fp32" if tc > tm else "hbm", "share_of_bound": max(tc, tm) * 1e3 / ms}

    fl = [level_flops(W3, H3, 1 << k) for k in range(5)]
    bounds = {
        "level pass C3 (mean of steps 1..16; slope of L = 1..5)": bound(sum(fl) / 5, W3 * H3 * BYTES_PER_PIXEL_LEVEL,
                                                                        slope),
        "prepare + finish C3 (intercept)": bound(0, W3 * H3 * (BYTES_PREPARE + BYTES_FINISH), intercept),
        "whole denoise C3 L=5": bound(sum(fl), W3 * H3 * (5 * BYTES_PER_PIXEL_LEVEL + BYTES_PREPARE + BYTES_FINISH),
                                      best["denoise C3 L=5"]),
        "whole denoise C4 L=5": bound(sum(level_flops(3840, 2160, 1 << k) for k in range(5)),
                                      3840 * 2160 * (5 * BYTES_PER_PIXEL_LEVEL + BYTES_PREPARE + BYTES_FINISH),
                                      best["denoise C4 L=5"]),
    }

    # equal quality against a 4 096-spp frame of another seed
    _, ref, rst = r.render_linear(R.main_camera(1200, 4096, seed=0x5EED3))
    ref = ref.double()
    rmse = lambda x: float(torch.sqrt(torch.mean((x.double() - ref) ** 2)))  # noqa: E731
    qual = []
    for spp in SPPS:
        lin, alb, nrm, st, gst = inputs(1200, spp)
        qual.append({"frame": f"noisy {spp} spp", "spp": spp, "rmse": rmse(lin), "ms": st.trace_ms + st.resolve_ms})
        if spp in (16, 64):
            _, dlin, ds = r.denoise(lin, alb, nrm)
            qual.append({"frame": f"denoised {spp} spp (g = 16, defaults)", "spp": spp, "rmse": rmse(dlin),
                         "ms": st.trace_ms + st.resolve_ms + gst.total_ms + ds.total_ms,
                         "ms_parts": {"render": st.trace_ms + st.resolve_ms, "guides": gst.total_ms,
                                      "denoise": ds.total_ms}})
    noisy = [q for q in qual if q["frame"].startswith("noisy")]
    headline = {}
    for q in qual:
        if not q["frame"].startswith("denoised"):
            continue
        # noisy RMSE falls as 1/sqrt(spp): the equal-quality spp from the fit of log RMSE on log spp
        k, b = np.polyfit([math.log(x["spp"]) for x in noisy], [math.log(x["rmse"]) for x in noisy], 1)
        n_eq = math.exp((math.log(q["rmse"]) - b) / k)
        ms_per_spp = np.polyfit([x["spp"] for x in noisy], [x["ms"] for x in noisy], 1)
        headline[q["frame"]] = {"equal_noisy_spp": n_eq, "denoised_ms": q["ms"],
                                "noisy_equal_ms": float(np.polyval(ms_per_spp, n_eq))}
    r.close()
    out = {"frame": {"scene": "final, seed 0xdeadbeef", "spheres": n, "C3": [W3, H3], "C4": [3840, 2160],
                     "denoise_inputs": "16 spp render + guides g = 16, seed 0xdeadbeef",
                     "defaults": {"sigma_color": 0.25, "sigma_normal": 0.25, "sigma_albedo": 0.25}},
           "card": card(), "fp32_peak_tflops_measured": peak.value, "hbm_tbps": HBM_BPS * 1e-12,
           "flop_per_tap": FLOP_PER_TAP, "rows": rows, "best_ms": best,
           "level_fit_ms": {"per_level": slope, "prepare_finish": intercept}, "bounds": bounds,
           "target_c3_l5_ms": 0.5, "target_met": best["denoise C3 L=5"] <= 0.5,
           "quality": {"reference": "4096 spp, seed 0x5eed3", "rows": qual, "headline": headline}}
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"best_ms": best, "headline": headline, "card": out["card"], "target_met": out["target_met"]}))


if __name__ == "__main__":
    main()
