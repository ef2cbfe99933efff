#!/usr/bin/env python
"""fyx_skin with skinned tangents off and on, in one process, on the C4 vertex set (50 000 surfaces x 5 000 vertices x 64 bones,
250 M vertices: far larger than L2).  Every surface's tangents (AnimatedVertex offset 32; scenegen writes a constant tangent,
which does not matter for bandwidth) are turned on or off between the passes, each mode is warmed up, then the modes alternate.
Reports kernel time (CUDA events of fyx_skin, fyx_get_timings), algorithmic bytes (68 B/vertex off; 92 on: 56 read + 36
written), GB/s and the fraction of the HBM peak (MEASURED_PEAKS.json hbm_gbs, else bench.py's fallback), with the card's name
and power limit read in the same run.  Usage: skin_tangents_bench.py [units] [rounds]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import bench
import fyrox_b200 as fb
from fyrox_b200 import camera
from fyrox_b200.scenegen import Scene

BYTES_PER_VERTEX = {"off": 68, "on": 92}


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    units = int(sys.argv[1]) if len(sys.argv) > 1 else 50000
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 4
    per_pass = 15
    sc = Scene(units * 200, n_units=units, verts_per_unit=5000, bones_per_unit=64, seed=bench.SEED)
    ctx = fb.Context()
    bench.load_scene(ctx, sc, fb, lambda m: None)  # surface u = unit u
    ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=camera.cube_frusta())
    nv = units * 5000

    chunk = 1024
    pin = fb.PinnedBuffer((chunk * 5000 * 68,), np.uint8)
    aabbs = np.empty((chunk, 6), np.float32)

    def set_mode(mode):
        for u0 in range(0, units, chunk):
            cnt = min(chunk, units - u0)
            if mode == "on":
                sc.units_vertices_into(u0, cnt, pin.ptr, aabbs)
            for i in range(cnt):
                ctx.set_skinned_tangents(u0 + i, pin.ptr + i * 5000 * 68 if mode == "on" else None, 32, 68)

    def run(mode, n):
        set_mode(mode)
        ctx.skin()  # commits the tile table, loads the kernel
        t = []
        for _ in range(n):
            ctx.skin()
            t.append(ctx.timings()["skin_ms"])
        return t

    hbm, hbm_src = bench.peaks()
    samples = {"off": [], "on": []}
    for mode in ("off", "on"):  # warm-up of each mode
        run(mode, 3)
    for r in range(rounds):
        for mode in (("off", "on") if r % 2 == 0 else ("on", "off")):
            samples[mode] += run(mode, per_pass)
    out = {"card": card(), "units": units, "verts": nv, "hbm_peak_gbs": hbm, "hbm_peak_source": hbm_src, "kernel_time": "CUDA events around fyx_skin"}
    for mode, t in samples.items():
        t = np.array(t)
        nbytes = BYTES_PER_VERTEX[mode] * nv
        gbs = nbytes / np.median(t) / 1e6
        out[mode] = {"ms_median": float(np.median(t)), "ms_min": float(t.min()), "ms_max": float(t.max()), "n": int(t.size),
                     "bytes": nbytes, "GBps": gbs, "frac_hbm_peak": gbs / hbm}
    # the tangents cost: same set, one more stream
    out["on_over_off_time"] = out["on"]["ms_median"] / out["off"]["ms_median"]
    print(json.dumps(out))
    pin.free()
    ctx.close()
    sc.close()


if __name__ == "__main__":
    main()
