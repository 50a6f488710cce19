"""Device BLAS build (idkpt_blas_build) against the host builder on the Sponza sample, the atrium at 262 k and 1 M triangles
and street_canyon (3.9 M). Per input: device kernel time (CUDA events, median of --reps after a warm-up), the per-phase
split of that time, end to end through idkpt_blas_build_read into host arrays (wall clock), the host builder with one
thread and with all cores, equality of every output, and the device memory the build holds. Writes one JSON file.

    python scripts/blas_build_bench.py --out profiles/r03_blas_build.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import numpy as np

from idkengine_b200 import host, scenes
from idkengine_b200.pathtracer import PathTracer


def build_inputs(make):
    """(positions, source triangles) that Scene.add hands to the builder for the first model."""
    jobs = []
    orig = host.build_blas

    def capture(positions, triangles, presplit=True, threads=None, settings=None):
        jobs.append((positions, triangles.copy()))
        return orig(positions, triangles, presplit, threads, settings)
    host.build_blas = capture
    try:
        make()
    finally:
        host.build_blas = orig
    return jobs[0]


def sponza_sample():
    import importlib.util
    spec = importlib.util.spec_from_file_location("g", os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "make_sponza_golden.py"))
    g = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(g)
    return build_inputs(lambda: g.sample_scene(*g.load_sample()))


def same(d, h):
    return (d["nodes"].tobytes() == h["nodes"].tobytes() and d["triangles"].tobytes() == h["triangles"].tobytes()
            and d["fragment_count"] == h["fragment_count"] and d["required_stack_size"] == h["required_stack_size"]
            and np.float64(d["sah"]).tobytes() == np.float64(h["sah"]).tobytes())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r03_blas_build.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sizes", default="sponza,262144,1048576,street")
    args = ap.parse_args()
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    cores = os.cpu_count()
    result = dict(gpu=smi[0] if smi else "unknown", host_cores=cores, reps=args.reps, warmup=args.warmup, rows=[])
    free0 = torch.cuda.mem_get_info(0)[0]
    with PathTracer(64, 48) as pt:
        for name in args.sizes.split(","):
            if name == "sponza":
                pv, tris = sponza_sample()
            elif name == "street":
                pv, tris = build_inputs(lambda: scenes.street_canyon(threads=cores))
            else:
                pv, tris = build_inputs(lambda: scenes.atrium(int(name), threads=cores))
            for presplit in (True, False):
                t0 = time.perf_counter()
                ref1 = host.build_blas(pv, tris, presplit=presplit, threads=1)
                host1 = time.perf_counter() - t0
                hostN = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    refN = host.build_blas(pv, tris, presplit=presplit, threads=cores)
                    hostN.append(time.perf_counter() - t0)
                kernel, e2e, phases = [], [], []
                for i in range(args.warmup + args.reps):
                    t0 = time.perf_counter()
                    dev = pt.BuildBlas(pv, tris, presplit=presplit)
                    t1 = time.perf_counter() - t0
                    if i >= args.warmup:
                        kernel.append(pt.last_blas_build_ms)
                        e2e.append(t1 * 1e3)
                        phases.append(pt.BlasBuildPhaseMs())
                eq = same(dev, ref1) and same(dev, refN)
                held = free0 - torch.cuda.mem_get_info(0)[0]
                row = dict(input=name, triangles=len(tris), presplit=presplit, fragments=dev["fragment_count"], nodes=len(dev["nodes"]),
                           equal_to_host=bool(eq), device_kernel_ms_median=statistics.median(kernel), device_kernel_ms_min=min(kernel),
                           device_kernel_ms_max=max(kernel), end_to_end_ms_median=statistics.median(e2e),
                           phase_ms_median={k: statistics.median(p[k] for p in phases) for k in phases[0]},
                           host_1_thread_ms=host1 * 1e3, host_all_cores_ms_median=statistics.median(hostN) * 1e3,
                           device_bytes_held_after=int(held))
                print(json.dumps(row), flush=True)
                result["rows"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    if not all(r["equal_to_host"] for r in result["rows"]):
        sys.exit("device build differs from the host build")


if __name__ == "__main__":
    main()
