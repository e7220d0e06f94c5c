"""Times fi_field_error_map (generate_error_map of a field's own system) on the device.

512^3 with the bench cloud (1M sphere-and-torus points, default weights), device-resident solution and heat map:
  whole      the call on the field of sdf_from_points (model rows, then point rows);
  model      the call on a field holding only its add_field_constraints call: heat zeroed (4 B / node), then the
             model gather (x read, heat read and written: 12 B / node, the kernel's byte bound);
  points     the call on a field holding only the add_points call: ~32M triplets emitted, sorted by column, summed
             (plus the 4 B / node zeroing of the heat map).
256^3 with the same cloud, host arrays in and out: the call against the triplet route a caller has without it —
fi_field_export into host buffers, then fi_error_map on them.

Every time is the median of 10 calls after 2 warm-up calls, CUDA events around each call (the call returns after a
stream synchronise).  Bounds are byte counts over the data-sheet 7.7 TB/s.  The card's name and power limit are read
in the same run.  Usage: time_field_error_map.py [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PEAK_GBPS = 7700.0


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def sdf(n):
    import torch
    a = (torch.arange(n, device="cuda", dtype=torch.float32) + 0.5) / n - 0.5
    z, y, x = a.view(n, 1, 1), a.view(1, n, 1), a.view(1, 1, n)
    sphere = torch.sqrt(x * x + y * y + z * z) - 0.3
    q = torch.sqrt(x * x + y * y) - 0.25
    torus = torch.sqrt(q * q + z * z) - 0.10
    return (torch.minimum(sphere, torus) * (n - 1)).reshape(-1).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import field_interpolation_b200 as fi
    from field_interpolation_b200 import _lib as L
    from field_interpolation_b200 import workloads as W
    info = card()
    dll = L.lib()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lines = []

    def timed(fn, reps=10):
        for _ in range(2):
            fn()
        ts = []
        for _ in range(reps):
            start.record()
            fn()
            end.record()
            end.synchronize()
            ts.append(start.elapsed_time(end))
        return float(np.median(ts))

    def emit(line):
        line.update(info)
        lines.append(line)
        print(json.dumps(line), flush=True)

    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    w = fi.Weights()

    # ---- 512^3, device-resident ----
    n = 512
    N = n ** 3
    pos = W.to_lattice(cloud["unit_pos"], [n, n, n])
    x = sdf(n)
    heat = torch.empty_like(x)
    whole = fi.sdf_from_points([n, n, n], w, pos, cloud["normals"])
    model = fi.LatticeField([n, n, n])
    fi.add_field_constraints(model, w)
    points = fi.LatticeField([n, n, n])
    fi.add_points(points, w.data_pos, w.value_kernel, w.data_gradient, w.gradient_kernel, pos, cloud["normals"])
    point_rows, point_trips = points.counts()
    for name, f in (("whole", whole), ("model", model), ("points", points)):
        def call():
            st = dll.fi_field_error_map(f._h, C.c_void_p(x.data_ptr()), L.FI_DEVICE, C.c_void_p(heat.data_ptr()), None)
            assert st == L.FI_OK, dll.fi_last_error()
        ms = timed(call)
        line = {"what": "fi_field_error_map", "n": n, "part": name, "ms": ms, "nodes": N, "points": len(pos)}
        if name == "model":
            line.update({"call_bytes": 16 * N, "kernel_bytes": 12 * N, "bound_ms_kernel_bytes": 12 * N / PEAK_GBPS / 1e6,
                         "bound_ms_call_bytes": 16 * N / PEAK_GBPS / 1e6, "x_over_kernel_bound": ms / (12 * N / PEAK_GBPS / 1e6)})
        if name == "points":
            line.update({"point_rows": point_rows, "point_triplets": point_trips, "triplets_per_s": point_trips / ms * 1e3})
        emit(line)
    del whole, model, points, heat, x
    torch.cuda.empty_cache()
    dll.fi_trim_memory()

    # ---- 256^3, host arrays: the call against export + fi_error_map ----
    n = 256
    N = n ** 3
    pos = W.to_lattice(cloud["unit_pos"], [n, n, n])
    f = fi.sdf_from_points([n, n, n], w, pos, cloud["normals"])
    xh = sdf(n).cpu().numpy()
    hh = np.empty(N, np.float32)
    rows, trips = f.counts()
    t_buf = np.empty(trips, dtype=np.dtype([("row", np.int32), ("col", np.int32), ("value", np.float32)]))
    r_buf = np.empty(rows, np.float32)
    hr = np.empty(N, np.float32)

    def call():
        assert dll.fi_field_error_map(f._h, C.c_void_p(xh.ctypes.data), L.FI_HOST, C.c_void_p(hh.ctypes.data), None) == L.FI_OK

    def export():
        assert dll.fi_field_export(f._h, C.c_void_p(t_buf.ctypes.data), C.c_void_p(r_buf.ctypes.data)) == L.FI_OK

    def triplet_map():
        assert dll.fi_error_map(trips, C.c_void_p(t_buf.ctypes.data), N, xh.ctypes.data_as(L._pf), rows, r_buf.ctypes.data_as(L._pf),
                                hr.ctypes.data_as(L._pf)) == L.FI_OK

    ms_call = timed(call)
    ms_export = timed(export, reps=5)
    ms_map = timed(triplet_map, reps=5)
    # the two agree to rounding (fi_error_map sums with atomics); this call is bit-identical to the reference
    rel = float(np.abs(hr - hh).max() / max(np.abs(hh).max(), 1e-30))
    emit({"what": "fi_field_error_map vs triplet route", "n": n, "points": len(pos), "rows": rows, "triplets": trips, "host_arrays": True,
          "ms_call": ms_call, "ms_export": ms_export, "ms_fi_error_map": ms_map, "ms_triplet_route": ms_export + ms_map,
          "speedup": (ms_export + ms_map) / ms_call, "triplet_bytes": 12 * trips, "max_rel_diff_vs_triplet_route": rel})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as h:
            for line in lines:
                h.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
