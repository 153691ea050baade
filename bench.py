#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native `Camera.render`.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one full render of the workload frame (the hot path over one batch of synthetic input).
Workload (BASELINE.json): C3 = Book-1 final random-spheres scene (485 spheres, host-generated with the
reference's Xoshiro stream, seed 0xdeadbeef), 1200x675, 500 spp, depth 50 — at every N (strong scaling:
the frame is sharded by interleaved tiles and gathered to rank 0 over NCCL).  `--workload c4` selects
BASELINE config 4 (3840x2160, 2000 spp) instead.

value  = Msamples/s, device-resident: scene already in HBM, image left in HBM, CUDA events on the
         launching stream (the Renderer's own torch stream), max over ranks.
e2e    = the same metric through the reference-facing C-ABI call with HOST buffers, host<->device copies
         inside the timed region: rtz_render at N=1; at N>1 rtz_render_multi called by rank 0 alone — ONE
         process driving all N GPUs, which is what a Zig / C host does (the other ranks wait on a CPU
         barrier).  `e2e_torchrun` keeps the one-process-per-GPU path (upload + sharded render + NCCL gather
         + download) beside it.
At N>1 the gathered image is compared with a single-GPU render of the same frame (outside the timed
regions): `image_equals_1gpu` and the frame's sha256 go into the JSON line.
roofline = FP32 CUDA-core pipe: 17 algorithmic FLOP per ray-sphere test (SURVEY.md §8d) x tests counted
         by the kernel / trace-kernel time measured with CUDA events by the library.
cpu_baseline = the oracle (CPU port of the reference; the Zig reference cannot be built here) timed on
         this box's host cores on a bounded sample of the same workload.

--dump-outputs DIR writes what the last timed step computed, so that two builds can be compared output for
output (the inputs are seeded, hence identical from run to run): DIR/image.npy, the frame a caller receives
(uint8 [H, W, 3]) as float32, or, for a frame larger than the dump budget, DIR/image_sample.npy with a fixed
seeded sample of its pixels ([k, 3], float32) and their flat pixel indices in DIR/image_sample_index.npy
(float64); and DIR/stats.npy, the frame's work counters (STAT_FIELDS, float64).  Nothing is written to the
source tree, which may be read-only.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # no __pycache__ in the tree from the modules imported below

SEED = 0xDEADBEEF
WORKLOADS = {
    # name: (width, spp, description)
    "c3": (1200, 500, "C3: Book-1 final random-spheres scene (485 spheres, seed 0xdeadbeef), 1200x675, 500 spp, depth 50"),
    "c4": (3840, 2000, "C4: Book-1 final scene (485 spheres), 3840x2160, 2000 spp, depth 50"),
    "smoke": (400, 10, "reference test render: final scene 400x225, 10 spp (dev only)"),
}
FLOP_PER_TEST = 17.0  # SURVEY.md §8d / BASELINE.md §3
TILE = (4, 4)
STAT_FIELDS = ("samples", "segments", "sphere_tests", "depth_capped", "absorbed", "nan_samples")
DUMP_BYTES = 64 << 20
DUMP_SEED = 0x5EED


def counters(stats) -> list[float]:
    """The work counters of an rtz_stats, in STAT_FIELDS order."""
    return [float(getattr(stats, f)) for f in STAT_FIELDS]


def dump_outputs(dirname: str, image, stat_counters) -> None:
    """Write one frame (uint8 [H, W, 3]) and its work counters as described in the module docstring."""
    import numpy as np
    d = Path(dirname)
    d.mkdir(parents=True, exist_ok=True)
    img = np.asarray(image, dtype=np.float32)
    budget = DUMP_BYTES - (1 << 20)                     # headroom for stats.npy and the .npy headers
    if img.nbytes <= budget:
        np.save(d / "image.npy", img)
    else:
        flat = img.reshape(-1, 3)
        k = budget // (flat.itemsize * 3 + 8)           # a float32 pixel plus its float64 index
        idx = np.sort(np.random.Generator(np.random.PCG64(DUMP_SEED)).choice(flat.shape[0], k, replace=False))
        np.save(d / "image_sample.npy", flat[idx])
        np.save(d / "image_sample_index.npy", idx.astype(np.float64))
    np.save(d / "stats.npy", np.array(stat_counters, dtype=np.float64))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    return json.loads(p.read_text()) if p.exists() else {}


class ClockSampler:
    """nvidia-smi clocks and throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])), (smax := float(r[2]))
                for k, nme in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle (only legs of this file that touch oracle/)
# ------------------------------------------------------------------------------------------------
def oracle_throughput(width: int, spp: int, threads: int | None = None):
    """Time the f64 CPU restatement of the reference on `threads` host threads (all by default) on
    the workload's scene and camera at `spp` samples per pixel.  Returns (Msamples/s, threads, samples,
    seconds, Mtests/s, image uint8 [H, W, 3], stats)."""
    import numpy as np
    sys.path.insert(0, str(ROOT / "tests"))
    import rtzlib as R
    orc = R.oracle()
    threads = threads or max(1, orc.orc_hardware_threads())
    prng, sp, n = R.final_scene(SEED)
    cam = R.main_camera(width, spp, seed=SEED)
    st = R.Stats()
    rgb = (C.c_uint8 * (3 * cam.width * cam.height))()
    t0 = time.perf_counter()
    if threads == 1:   # reference-faithful: ONE shared sequential Xoshiro stream, one thread
        rc = orc.orc_render_reference(C.byref(cam), sp, n, prng, rgb, None, C.byref(st))
    else:              # same f64 arithmetic, per-sample Philox streams, rows striped over threads
        rc = orc.orc_render_philox64(C.byref(cam), sp, n, SEED, threads, rgb, None, C.byref(st))
    dt = time.perf_counter() - t0
    assert rc == 0
    img = np.frombuffer(rgb, dtype=np.uint8).reshape(int(cam.height), int(cam.width), 3)
    return st.samples / dt / 1e6, threads, int(st.samples), dt, st.sphere_tests / dt / 1e6, img, st


def run_reference(args, rank: int):
    if rank != 0:
        return
    width, spp_full, desc = WORKLOADS[args.workload]
    spp = args.ref_spp
    vals = []
    for i in range(args.warmup + args.steps):
        v, threads, samples, dt, mt, img, st = oracle_throughput(width, spp)
        if i >= args.warmup:
            vals.append((v, dt, mt))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, img, counters(st))
    value = sum(v for v, _, _ in vals) / len(vals)
    ms = 1e3 * sum(d for _, d, _ in vals) / len(vals)
    sample = f"{desc.split(':')[0]} scene+camera at {spp} of {spp_full} spp ({samples / 1e6:.2f} M samples per step)"
    emit({
        "impl": "reference", "metric": "Msamples/s", "value": round(value, 4), "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "sample": sample},
        "cpu_baseline": {"value": round(value, 4), "unit": "Msamples/s", "cores": threads, "kind": "port",
                         "sample": sample, "mtests_per_s": round(sum(m for _, _, m in vals) / len(vals), 1)},
        "e2e": {"value": round(value, 4), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = C++ f64 restatement of the Zig renderer (oracle/, byte-exact on its chapter14.ppm); "
                "no zig toolchain in the image, so kind=port",
    })


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, rank: int, world: int, local_rank: int):
    import numpy as np
    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a GPU: the product has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    pkg = importlib.import_module("raytracing-with-zig_b200")
    host = importlib.import_module("raytracing-with-zig_b200.host_api")
    B = pkg.binding
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    width, spp, desc = WORKLOADS[args.workload]
    if args.spp:
        spp = args.spp
    spheres, n = host.generate_world(SEED)          # product host mirror (Zig-exact Xoshiro scene)
    cam = host.main_camera(width, spp, seed=SEED)
    W, H = int(cam.width), int(cam.height)
    r = pkg.Renderer(local_rank)
    r.upload(spheres, n)
    shard = B.rtz_shard(rank, world, *TILE) if world > 1 else None
    out = torch.empty((r.shard_pixels(W, H, shard), 3) if shard is not None else (H, W, 3), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    cpu_group = dist.new_group(backend="gloo") if world > 1 else None   # a barrier that keeps the GPUs idle

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step_resident():
        """Device-resident step: render this rank's share (+ gather and de-interleave at N>1)."""
        local, st = r.render(cam, shard, out)
        if world > 1:
            g = pkg.distributed.gather_tiles(local, world, rank)
            if rank == 0:
                last["img"] = r.deinterleave(g, W, H, world, *TILE)
        else:
            last["img"] = local
        return st

    # everything below is enqueued on the stream the library launches on, so the CUDA events bracket its kernels
    with torch.cuda.stream(r.stream):
        for _ in range(args.warmup):
            step_resident()
        clocks = ClockSampler(local_rank)
        barrier()
        clocks.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        stats = []
        t_wall0 = time.perf_counter()
        for s, e in ev:
            flush.fill_(1)                  # flush L2 between timed iterations (untimed)
            if world > 1:
                dist.barrier()
            s.record()
            stats.append(step_resident())
            e.record()
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
        clk = clocks.stop()
        barrier()
    if args.dump_outputs:   # before anything below renders into `out` again
        last_counters = torch.tensor(counters(stats[-1]), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(last_counters)          # each rank counted its own tiles
        if rank == 0:
            dump_outputs(args.dump_outputs, last["img"].cpu().numpy(), last_counters.tolist())
    dev_ms = sum(s.elapsed_time(e) for s, e in ev)
    samples = sum(int(st.samples) for st in stats)
    tests = sum(int(st.sphere_tests) for st in stats)
    segments = sum(int(st.segments) for st in stats)
    trace_ms = sum(st.trace_ms for st in stats)
    agg = torch.tensor([dev_ms, trace_ms, float(samples), float(tests), float(segments)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = agg.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
        dev_ms, trace_ms_max = mx[0].item(), mx[1].item()
        samples, tests, segments = int(agg[2].item()), int(agg[3].item()), int(agg[4].item())
    else:
        trace_ms_max = trace_ms
    value = samples / (dev_ms * 1e-3) / 1e6

    # ---- correctness of the N-GPU frame, outside every timed region: rank 0 renders the whole frame alone ------
    check = {}
    if rank == 0:
        import hashlib
        img = last["img"].cpu().numpy()
        check["image_sha256"] = hashlib.sha256(img.tobytes()).hexdigest()
        if world > 1:
            whole, wst = r.render(cam)
            check["image_equals_1gpu"] = bool(torch.equal(last["img"], whole))
            check["segments_equal_1gpu"] = bool(int(wst.segments) * len(stats) == segments)
            assert check["image_equals_1gpu"], "the N-GPU image differs from the single-GPU image"

    # ---- e2e: host buffers in, host buffers out, copies inside the timed region -----------------
    sph_bytes = n * C.sizeof(B.rtz_sphere)
    if world == 1:
        pkg.render_host(cam, spheres, n)    # warm the library's cached context
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            rgb, st = pkg.render_host(cam, spheres, n)   # rtz_render: H2D scene, trace, resolve, D2H image
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_samples = W * H * spp * args.steps
        h2d = 5 * ((n + 7) // 8 * 8) * 16 + n * 32
        d2h = W * H * 3 + 64
        e2e_api = "rtz_render (C ABI, host buffers)"
        e2e_torchrun = None
    else:
        # (a) the C ABI from ONE process: rank 0 drives all N GPUs through rtz_render_multi, the others keep off the GPUs
        e2e_api = "rtz_render_multi (C ABI, host buffers; rank 0 alone drives all N GPUs, NVLink peer-store gather)"
        if rank == 0:
            rgb_m, st_m = pkg.render_host_multi(cam, spheres, n, num_gpus=world)   # creates the devices' contexts
            check["cabi_image_equals_1gpu"] = bool((torch.from_numpy(rgb_m).to(dev) == whole).all().item())
            assert check["cabi_image_equals_1gpu"], "rtz_render_multi differs from the single-GPU image"
            check["cabi_gather"] = {1: "p2p (fused resolve + peer store)", 2: "nccl (grouped send/recv)"}.get(int(st_m.gather), "none")
        dist.barrier(group=cpu_group)
        e2e_s = 0.0
        if rank == 0:
            t0 = time.perf_counter()
            for _ in range(args.steps):
                rgb_m, st_m = pkg.render_host_multi(cam, spheres, n, num_gpus=world)
            e2e_s = time.perf_counter() - t0
        dist.barrier(group=cpu_group)
        e2e_samples = W * H * spp * args.steps
        h2d = world * (5 * ((n + 7) // 8 * 8) * 16 + n * 32)
        d2h = W * H * 3 + world * 64
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
        # (b) one process per GPU: upload + sharded render + NCCL gather + D2H on rank 0
        host_img = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() if rank == 0 else None
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r.upload(spheres, n)                                  # H2D of this step's inputs
            img, st = pkg.render_sharded(r, cam, TILE)            # render + NCCL gather + de-interleave
            if rank == 0:
                host_img.copy_(img, non_blocking=False)           # D2H of the step's result
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_torchrun = e2e_samples / t.item() / 1e6
    e2e_value = e2e_samples / e2e_s / 1e6

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (trace_kernel) ----------------------------------------
    peaks = measured_peaks()
    sm_max = float(peaks.get("sm_max_mhz") or clk.get("sm_max_mhz") or 1965.0)
    sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
    nominal = sm_count * 128 * 2 * sm_max * 1e6 / 1e12               # 74.4 TFLOP/s at 1965 MHz
    v = C.c_double()
    B.check(pkg.lib().rtz_measure_fp32_peak(local_rank, 0, C.byref(v)))
    ffma_measured = v.value
    launches_trace = len(stats) * world
    flop_per_launch = FLOP_PER_TEST * tests / launches_trace
    avg_trace_s = (trace_ms_max / len(stats)) * 1e-3
    achieved = flop_per_launch / avg_trace_s / 1e12
    traffic = None
    prof = ROOT / "profiles" / "trace_kernel_dram.json"
    if prof.exists():
        try:
            traffic = json.loads(prof.read_text()).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {
        "bound": "fp32", "kernel": "rtz::trace_kernel", "achieved": round(achieved, 3), "peak": round(nominal, 2),
        "unit": "TFLOP/s", "frac": round(achieved / nominal, 4), "traffic": traffic,
        "peak_kind": f"nominal FP32 pipe: {sm_count} SMs x 128 lanes x 2 x {sm_max:.0f} MHz (MEASURED_PEAKS.json clock); "
                     "MEASURED_PEAKS.json has no FP32 entry",
        "peak_measured_ffma": round(ffma_measured, 2), "frac_of_measured_ffma": round(achieved / ffma_measured, 4),
        "flop_per_test": FLOP_PER_TEST, "tests_per_launch": tests / launches_trace,
        "avg_launch_ms": round(avg_trace_s * 1e3, 4), "per_gpu": True,
    }

    # ---- CPU baseline beside it (rank 0, N=1 only; bounded sample) ------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        v_all, threads, smp, dt, mt, _, _ = oracle_throughput(width, args.ref_spp)
        v_one, _, smp1, dt1, _, _, _ = oracle_throughput(400, 10, threads=1)
        cpu = {"value": round(v_all, 4), "unit": "Msamples/s", "cores": threads, "kind": "port",
               "sample": f"{args.workload.upper()} scene+camera at {args.ref_spp} of {spp} spp ({smp / 1e6:.2f} M samples, {dt:.1f} s)",
               "mtests_per_s": round(mt, 1),
               "single_thread_reference_faithful": {"value": round(v_one, 4), "unit": "Msamples/s", "cores": 1,
                                                    "sample": f"final scene 400x225, 10 spp, sequential Xoshiro ({dt1:.1f} s)"}}

    line = {
        "metric": "Msamples/s", "value": round(value, 2), "unit": "Msamples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 4),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc if not args.spp else desc + f" [spp overridden to {spp}]", "image": [W, H], "spp": spp,
                   "spheres": n, "depth": 50, "seed": hex(SEED), "l2": "flushed between timed steps (256 MiB write)",
                   "sharding": f"interleaved {TILE[0]}x{TILE[1]} tiles, NCCL gather to rank 0" if world > 1 else "none",
                   "timing": "CUDA events on the launching stream (Renderer.stream) per step, summed; max over ranks"},
        "mray_sphere_tests_per_s": round(tests / (dev_ms * 1e-3) / 1e6, 1),
        "segments_per_sample": round(segments / samples, 4),
        "wall_s_timed_region": round(t_wall, 3),
        "clocks": clk,
        "e2e": {"value": round(e2e_value, 2), "unit": "Msamples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": e2e_api},
        "gpu_launches": int(sum(int(st.kernel_launches) for st in stats) * world + (args.steps if world > 1 else 0)),
        "roofline": roofline,
    }
    line.update(check)
    if e2e_torchrun is not None:
        line["e2e_torchrun"] = {"value": round(e2e_torchrun, 2), "unit": "Msamples/s",
                                "api": "Renderer.upload + render_sharded (torch.distributed NCCL gather) + D2H, one process per GPU"}
    if cpu:
        line["cpu_baseline"] = cpu
    if world == 1:
        # informational, outside every timed region above: the labelled extension RTZ_MODE_PATH_BVH on the same
        # frame (same bytes; NOT the reference's brute-force algorithm, so it is neither `value` nor the roofline)
        try:
            cam.mode = B.MODE_PATH_BVH
            ext_ms = min(r.render(cam, shard, out)[1].trace_ms for _ in range(2))
            line["extension_bvh"] = {"mode": "RTZ_MODE_PATH_BVH", "value": round(W * H * spp / ext_ms / 1e3, 2),
                                     "unit": "Msamples/s", "trace_ms": round(ext_ms, 3),
                                     "note": "same image through a BVH over the spheres; not the benchmarked path"}
        finally:
            cam.mode = B.MODE_PATH
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def _quiet_stdout():
    """Libraries (NCCL's version banner, torchrun's notices) write to stdout; the contract is ONE JSON line there.
    Everything that is not that line goes to stderr: fd 1 is pointed at fd 2 and the original is kept for `emit`."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()), sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (dev only; invalidates the headline)")
    ap.add_argument("--ref-spp", type=int, default=48, help="spp of the bounded CPU sample (cost per sample does not depend on spp)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as .npy files under DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        _quiet_stdout()
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # not under torchrun: re-launch ourselves one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    _quiet_stdout()
    importlib.import_module("__graft_entry__").build()
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
