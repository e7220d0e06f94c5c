"""Times fi_marching_cubes fill calls on one GPU and the CPU port on the host, one JSON line per case.

    python scripts/time_marching_cubes.py [--out profiles/mc_time.jsonl] [--reps 10]

Cases: an analytic sphere + torus SDF built on the device at 512^3 and 1024^3, and a field solved (multigrid PCG) from
the C4 cloud generator (workloads.sphere_torus_3d) at 512^3.  Each timed call is a whole fill call with device inputs
and outputs (count pass, one host sync, emit pass, triangle pass), warmed up first, timed with CUDA events.  The fields
(0.5 / 4.3 GB) are larger than the 126 MB L2, so every call reads them from HBM.  Bytes/node counts the two lattice
passes' 4 B reads each plus the mesh written (12 B per vertex, 12 B per triangle, 4 B vbase per vertex node) over the
nodes; GB/s is that over the call time, against the 6.45 TB/s copy peak measured in BASELINE.md §3.  The CPU port
(tests/mc_port.cpp, one thread) meshes the same 512^3 analytic field on the host for the copy-out comparison, and the
device-to-host copy of that field is timed too."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

COPY_PEAK_GBS = 6450.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def analytic(n):
    import torch
    a = (torch.arange(n, device="cuda", dtype=torch.float32) - (n - 1) / 2) / (n - 1)
    z, y, x = a.view(n, 1, 1), a.view(1, n, 1), a.view(1, 1, n)
    sphere = torch.sqrt(x * x + y * y + z * z) - 0.3
    q = torch.sqrt(x * x + y * y) - 0.25
    torus = torch.sqrt(q * q + z * z) - 0.10
    return (torch.minimum(sphere, torus) * (n - 1)).contiguous()


def solved(n):
    import torch
    import field_interpolation_b200 as fi
    from field_interpolation_b200 import workloads as W
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    sizes = [n, n, n]
    field = fi.sdf_from_points(sizes, fi.Weights(), W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"])
    out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
    field.solve(fi.solve_options(fi.FI_F32, 200, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
    del field
    return out.view(n, n, n)


def time_fill(values, reps, want_normals):
    import ctypes as C
    import torch
    from field_interpolation_b200 import _lib as L
    import field_interpolation_b200 as fi
    v, t = fi.marching_cubes(values, 0.0)  # sizes the outputs
    V, T = len(v), len(t)
    nrm = torch.empty_like(v) if want_normals else None
    n = values.shape
    sizes = (C.c_int32 * 3)(n[2], n[1], n[0])
    nv, nt = C.c_int64(0), C.c_int64(0)
    args = (sizes, C.c_void_p(values.data_ptr()), 0.0, L.FI_DEVICE, C.c_void_p(v.data_ptr()),
            C.c_void_p(nrm.data_ptr()) if want_normals else None, V, C.c_void_p(t.data_ptr()), T, C.byref(nv), C.byref(nt))
    dll = L.lib()
    for _ in range(3):
        L.check(dll.fi_marching_cubes(*args))
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        L.check(dll.fi_marching_cubes(*args))
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return V, T, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sizes", default="512,1024")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    gpu = card()
    rows = []

    def report(case, n, values, want_normals):
        V, T, ms = time_fill(values, args.reps, want_normals)
        nodes = n ** 3
        vbytes = 24 if want_normals else 12
        moved = 8 * nodes + vbytes * V + 12 * T + 4 * V
        best, med = min(ms), float(np.median(ms))
        row = {"case": case, "n": n, "normals": want_normals, "vertices": V, "triangles": T, "ms_median": round(med, 3),
               "ms_min": round(best, 3), "bytes_per_node": round(moved / nodes, 3), "GBps_median": round(moved / med / 1e6, 1),
               "share_of_copy_peak": round(moved / med / 1e6 / COPY_PEAK_GBS, 3), "reps": args.reps, "gpu": gpu}
        rows.append(row)
        print(json.dumps(row), flush=True)

    for n in [int(s) for s in args.sizes.split(",")]:
        f = analytic(n)
        report("analytic_sphere_torus", n, f, False)
        report("analytic_sphere_torus", n, f, True)
        if n == 512:
            host = None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host = f.cpu().numpy()
            copy_s = time.perf_counter() - t0
            from mc_port import port
            with tempfile.TemporaryDirectory() as d:
                p = port(d)
                p.marching_cubes(host[:8], 0.0)
                t0 = time.perf_counter()
                v, t = p.marching_cubes(host, 0.0)
                cpu_s = time.perf_counter() - t0
            row = {"case": "cpu_port_analytic_sphere_torus", "n": n, "vertices": len(v), "triangles": len(t), "s": round(cpu_s, 3),
                   "device_to_host_copy_s": round(copy_s, 3), "threads": 1, "cpu": os.uname().machine, "gpu": gpu}
            rows.append(row)
            print(json.dumps(row), flush=True)
        del f
        torch.cuda.empty_cache()
    f = solved(512)
    report("solved_c4_cloud", 512, f, False)
    report("solved_c4_cloud", 512, f, True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
