"""Times fi_sample_field on the device: a 512^3 sphere-union-torus SDF (512 MB, larger than L2), N = 1M and 16M points
uniform in the lattice, in random order and sorted by cell, value only and value + each gradient kernel.  Device inputs
and outputs; the median of 10 CUDA-event-timed calls after 2 warm-up calls.  The same points go through
torch.nn.functional.grid_sample (5D, align_corners=True, value only), the gather users reach for without this call.

Each line reports points/s and the achieved GB/s against two byte counts:
  io_bytes      positions + outputs: 4 D + 4 (+ 4 D) B per point;
  sector_bytes  io_bytes + 32 B per distinct 32-B field sector each point touches (counted on the host from a 1M
                sample of the positions): what the call moves when no sector is reused between points.
In cell order neighbouring points share sectors, so the field is read about once and sector_bytes over-counts.
Bounds in ms are those byte counts over the measured HBM copy peak (MEASURED_PEAKS.json) when that file is present,
else over the data-sheet 7.7 TB/s; each line names which.  The card's name and power limit are read in the same run.
Usage: time_sample_field.py [--out FILE] [--n 512] [--points 1000000,16000000]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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
    return (torch.minimum(sphere, torus) * (n - 1)).contiguous()


def peak_hbm():
    """HBM bandwidth the bounds are stated against: the measured copy peak (MEASURED_PEAKS.json) when present, else
    the HGX B200 data-sheet figure for one GPU."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 7700.0, "data sheet (HGX B200, one GPU)"


def sectors_per_point(pos, n, kernel):
    """Mean number of distinct 32-B field sectors one point reads (host, from a sample of positions): the value's
    in-lattice corners of cell floor(p), plus for the gradient kernels exactly the nodes they load."""
    p = pos.astype(np.float32)
    strides = np.array([1, n, n * n], np.int64)
    cube = [np.array([(c >> 0) & 1, (c >> 1) & 1, (c >> 2) & 1]) for c in range(8)]
    idx = []

    def add(nodes, ok):
        idx.append(np.where(ok, (nodes @ strides) * 4 // 32, -1))

    base = np.floor(p).astype(np.int64)
    for o in cube:  # value (kernels 0 and 1 read a subset of the same corners)
        c = base + o
        add(c, ((c >= 0) & (c < n)).all(axis=1))
    if kernel == 2:  # kept corners of floor(p - 0.5) (c + 1 < n) and each corner's +s_d neighbour
        b2 = np.floor(p - np.float32(0.5)).astype(np.int64)
        for o in cube:
            c = b2 + o
            ok = ((c >= 0) & (c + 1 < n)).all(axis=1)
            add(c, ok)
            for d in range(3):
                add(c + np.eye(3, dtype=np.int64)[d], ok)
    s = np.sort(np.stack(idx, axis=1), axis=1)
    distinct = (s[:, :1] >= 0).astype(np.int64).ravel() + ((s[:, 1:] != s[:, :-1]) & (s[:, 1:] >= 0)).sum(axis=1)
    return float(distinct.mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--points", default="1000000,16000000")
    args = ap.parse_args()
    import torch
    from field_interpolation_b200 import _lib as L
    info = card()
    peak_gbs, peak_src = peak_hbm()
    info.update({"peak_GBps": peak_gbs, "peak_source": peak_src})
    n = args.n
    field = sdf(n)
    dll = L.lib()
    sizes = (C.c_int32 * 3)(n, n, n)
    lines = []
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        for _ in range(2):
            fn()
        ts = []
        for _ in range(10):
            start.record()
            fn()
            end.record()
            end.synchronize()
            ts.append(start.elapsed_time(end))
        return float(np.median(ts))

    for N in [int(s) for s in args.points.split(",")]:
        g = torch.Generator(device="cuda").manual_seed(N)
        pos = torch.rand(N, 3, device="cuda", generator=g) * (n - 1)
        cell = pos.floor().long()
        key = (cell[:, 2] * n + cell[:, 1]) * n + cell[:, 0]
        orders = {"random": pos, "cell_sorted": pos[torch.argsort(key)].contiguous()}
        del cell, key
        sample = pos[:1_000_000].cpu().numpy()
        vals = torch.empty(N, device="cuda")
        grads = torch.empty(N, 3, device="cuda")
        for order, p in orders.items():
            for kernel in (None, 0, 1, 2):
                gp = grads.data_ptr() if kernel is not None else None

                def call():
                    st = dll.fi_sample_field(3, sizes, field.data_ptr(), N, p.data_ptr(), kernel or 0, L.FI_DEVICE, vals.data_ptr(), gp)
                    assert st == L.FI_OK, dll.fi_last_error()
                ms = timed(call)
                io = N * (4 * 3 + 4 + (12 if kernel is not None else 0))
                spp = sectors_per_point(sample, n, kernel if kernel is not None else -1)
                sec = io + N * 32 * spp
                line = {"what": "fi_sample_field", "n": n, "points": N, "order": order,
                        "mode": "value" if kernel is None else f"value+gradient_kernel_{kernel}", "ms": ms,
                        "points_per_s": N / ms * 1e3, "io_bytes": io, "io_GBps": io / ms / 1e6,
                        "sectors_per_point": spp, "sector_bytes": sec, "sector_GBps": sec / ms / 1e6,
                        "bound_ms": {"io": io / peak_gbs / 1e6, "sector": sec / peak_gbs / 1e6}, **info}
                lines.append(line)
                print(json.dumps(line), flush=True)
            grid = ((p / (n - 1)) * 2 - 1).view(1, 1, 1, N, 3)
            inp = field.view(1, 1, n, n, n)
            ms = timed(lambda: torch.nn.functional.grid_sample(inp, grid, mode="bilinear", padding_mode="border", align_corners=True))
            io = N * (12 + 4)
            line = {"what": "torch.grid_sample", "n": n, "points": N, "order": order, "mode": "value", "ms": ms,
                    "points_per_s": N / ms * 1e3, "io_bytes": io, "io_GBps": io / ms / 1e6, **info}
            lines.append(line)
            print(json.dumps(line), flush=True)
            del grid
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as h:
            for line in lines:
                h.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
