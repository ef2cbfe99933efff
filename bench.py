#!/usr/bin/env python
"""bench.py — the render-prep hot path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps K --warmup W                 # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                         # + the last timed frame's outputs as DIR/<name>.npy
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # weak scaling, NCCL all-gather of visible lists
    python bench.py --impl reference --gpus N --steps K --warmup W # the reference's CPU algorithm (oracle port), host cores

A step = one frame of render prep over one batch of synthetic input:
  hierarchy update (every node recomputed) + world AABBs + cull against F frusta with visible-index
  compaction + bone palettes + linear-blend skinning (+ NCCL all-gather of the visible lists when N > 1).
metric = BASELINE.json's "nodes culled + verts skinned /sec"; value = (nodes + skinned vertices) per
second over all GPUs with every input resident in HBM; e2e = the same frame through fyx_render_prep with
HOST buffers (changed bone matrices uploaded from pinned memory, visible lists read back) per step.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

METRIC = "nodes culled + verts skinned /sec"
UNIT = "nodes+verts/s"
SEED = 0xF1A0C5

# BASELINE.json configs (per GPU; weak scaling multiplies by N)
WORKLOADS = {
    "C1": dict(nodes=100_000, units=0, verts_per_unit=5000, frusta=1, desc="100k static nodes, 1 camera frustum (BASELINE.json configs[0]: the reference's CPU-runnable case)"),
    "C2": dict(nodes=10_000_000, units=0, verts_per_unit=5000, frusta=1, desc="10M static nodes, 1 frustum"),
    "C3": dict(nodes=1_000_000, units=10_000, verts_per_unit=5000, frusta=1, desc="1M nodes incl. 10k skinned meshes x 64 bones x 5k verts, 1 frustum"),
    "C4": dict(nodes=10_000_000, units=50_000, verts_per_unit=5000, frusta=6, desc="10M nodes, 50k skinned meshes x 64 bones x 5k verts, 6 frusta (cube faces)"),
    "C5": dict(nodes=100_000_000, units=200_000, verts_per_unit=5000, frusta=6, desc="100M nodes, 200k skinned meshes x 64 bones x 5k verts, 6 frusta: the WHOLE job, sharded over the GPUs (strong scaling)"),
    "target": dict(nodes=10_000_000, units=10_000, verts_per_unit=5000, frusta=1, desc="10M nodes + 50M skinned verts, 1 frustum (north_star target)"),
    "tiny": dict(nodes=200_000, units=200, verts_per_unit=5000, frusta=6, desc="debug"),
}
DEFAULT_WORKLOAD = os.environ.get("FYX_BENCH_WORKLOAD", "C4")
BONES = 64

# algorithmic bytes per unit (SURVEY.md §8d / DESIGN.md §5)
B_NODE_FUSED = 188
B_VISIBLE = 4
B_BONE = 196
B_VERT = 68
UPLOAD_FIELD = {"rot": "changed_rot", "trs": "changed_trs", "m16": "changed_m16"}
UPLOAD_BYTES = {"rot": 16, "trs": 40, "m16": 64}
# --dump-outputs: how many nodes / skinned meshes of the last timed frame are written (about 30 MB at C4, under the 64 MB cap)
DUMP_NODES = 1 << 18
DUMP_UNITS = 8
DUMP_MAX_BYTES = 64 << 20


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# the reference arm / cpu_baseline: the oracle (CPU restatement of the reference algorithm), 1 thread
# --------------------------------------------------------------------------------------------------
def cpu_sample_config(w: dict) -> dict:
    """A bounded sample of the workload with the same nodes:verts ratio (about 2-5 s of CPU work per frame)."""
    if w["nodes"] <= 100_000:  # C1 is small enough to run whole
        return dict(nodes=w["nodes"], units=w["units"], verts_per_unit=w["verts_per_unit"], frusta=w["frusta"])
    scale = 10 if w["units"] >= 10_000 else 5
    nodes = max(w["nodes"] // scale, 100_000)
    units = w["units"] // scale
    if w["units"] and w["nodes"] // max(w["units"], 1) < 200:  # C3-like: vertex heavy
        nodes, units = w["nodes"] // 20, w["units"] // 20
    return dict(nodes=nodes, units=units, verts_per_unit=w["verts_per_unit"], frusta=w["frusta"])


class CpuReference:
    """Oracle port of the reference's single-threaded path (SURVEY §0 D2: the reference is not parallel):
    update_hierarchical_data + from_graph per frustum + palette + CPU LBS (mesh/mod.rs:501-522)."""

    def __init__(self, sample: dict):
        sys.path.insert(0, os.path.join(REPO, "tests"))
        import oracle_binding as ob  # the one place bench.py executes oracle/: the CPU baseline
        from fyrox_b200.scenegen import Scene

        self.ob = ob
        self.s = sample
        sc = Scene(sample["nodes"], n_units=sample["units"], verts_per_unit=sample["verts_per_unit"], bones_per_unit=BONES, seed=SEED)
        self.sc = sc
        aabb = sc.local_aabb.copy()
        self.og = ob.Graph.build(sc.parent, sc.flags, sc.render_mask, sc.local_m16, aabb)
        self.meshes = []
        for u in range(sc.n_units):
            mesh, bones, ib = sc.unit_mesh_node(u), sc.unit_bone_nodes(u), sc.unit_inv_bind(u)
            for k, b in enumerate(bones):
                self.og.set_inv_bind(int(b), ib[k])
            verts, _ = sc.unit_vertices(u)
            self.og.add_surface(mesh, bones, verts)
            self.og.recalc_local_aabb(mesh)
            self.meshes.append(mesh)
        self.og.L.orc_graph_drop_messages(self.og.h)
        # frusta through the oracle's own restatement
        self.frusta = []
        if sample["frusta"] == 1:
            view = ob.look_at_rh((0, 0, 0), (0, 0, -1), (0, 1, 0))
            proj = ob.perspective(16 / 9, float(np.deg2rad(60.0)), 0.1, 150.0)
            self.frusta.append(ob.frustum_from_vp(ob.mat4_mul(proj, view)))
        else:
            faces = [((1, 0, 0), (0, -1, 0)), ((-1, 0, 0), (0, -1, 0)), ((0, 1, 0), (0, 0, 1)), ((0, -1, 0), (0, 0, -1)), ((0, 0, 1), (0, -1, 0)), ((0, 0, -1), (0, -1, 0))]
            for look, up in faces[: sample["frusta"]]:
                view = ob.look_at_rh((0, 0, 0), look, up)
                proj = ob.perspective(1.0, float(np.pi / 2), 0.01, 120.0)
                self.frusta.append(ob.frustum_from_vp(ob.mat4_mul(proj, view)))
        self.pos = np.empty((sample["verts_per_unit"], 3), np.float32)
        self.nrm = np.empty((sample["verts_per_unit"], 3), np.float32)
        self.vis = np.empty(max(sc.capacity, 1), np.uint32)
        self.frame = 0

    def units_per_frame(self) -> int:
        return self.s["nodes"] + self.s["units"] * self.s["verts_per_unit"]

    def step(self):
        ob, og = self.ob, self.og
        import ctypes as C

        # every bone's local matrix changes each frame (set directly; the full recompute below ignores messages)
        idx, m = self.sc.animate(self.frame)
        self.frame += 1
        t0 = time.perf_counter()
        L = og.L
        for i in range(idx.size):
            L.orc_node_set_local_matrix(og.h, int(idx[i]), ob.fp(m[i]))
        L.orc_graph_drop_messages(og.h)
        t_set = time.perf_counter() - t0  # host-side scatter of changed matrices (python loop: excluded below)
        t1 = time.perf_counter()
        og.update_hierarchical_data()
        for f in self.frusta:
            L.orc_from_graph(og.h, C.byref(f), 0xFFFFFFFF, 0, self.vis.ctypes.data_as(C.c_void_p), self.vis.size)
        for mesh in self.meshes:
            L.orc_mesh_skin(og.h, mesh, 0, ob.fp(self.pos.reshape(-1)), ob.fp(self.nrm.reshape(-1)))
        dt = time.perf_counter() - t1
        return dt, t_set


class CpuMultiCore:
    """Best-effort multi-core CPU baseline ("soa-omp-NT", BASELINE.md §3): the oracle's arithmetic on flat arrays with
    OpenMP over levels / nodes / surfaces (oracle/fyrox_oracle_mt.c).  NOT how the reference runs (it is single-threaded);
    reported next to the reference-shaped number, never instead of it."""

    def __init__(self, ref: "CpuReference", threads: int):
        ob, sc = ref.ob, ref.sc
        self.ref = ref
        self.threads = threads
        self.mt = ob.MtGraph(sc.parent, sc.flags, sc.render_mask, sc.local_m16, sc.local_aabb.copy(), threads=threads)
        for u in range(sc.n_units):
            mesh, bones, ib = sc.unit_mesh_node(u), sc.unit_bone_nodes(u), sc.unit_inv_bind(u)
            for k, b in enumerate(bones):
                self.mt.set_inv_bind(int(b), ib[k])
            verts, _ = sc.unit_vertices(u)
            self.mt.add_surface(mesh, bones, verts)
        self.frame = 0

    def step(self):
        import ctypes as C

        idx, m = self.ref.sc.animate(self.frame)
        self.frame += 1
        mt, L = self.mt, self.mt.L
        t0 = time.perf_counter()
        mt.set_local_matrices(m, idx)
        mt.update()
        vis = self.ref.vis
        for f in self.ref.frusta:
            L.orc_mt_cull(mt.h, C.byref(f), 0xFFFFFFFF, 0, vis.ctypes.data_as(C.c_void_p), vis.size)
        mt.skin_all()
        return time.perf_counter() - t0


def usable_cores() -> int:
    """Host threads this process may really use: the affinity mask, capped by the cgroup CPU quota if there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:  # cgroup v2
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        try:  # cgroup v1
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0 and period > 0:
                n = max(1, min(n, quota // period))
        except Exception:
            pass
    return n


def time_multicore(ref: "CpuReference", frames: int) -> dict:
    threads = usable_cores()
    mc = CpuMultiCore(ref, threads)
    mc.step()
    t = sum(mc.step() for _ in range(frames))
    return {"value": ref.units_per_frame() * frames / t, "unit": UNIT, "cores": threads, "kind": "port-openmp", "ms_per_frame": 1e3 * t / frames,
            "note": "flat arrays + OpenMP over levels / nodes / surfaces, same arithmetic (oracle/fyrox_oracle_mt.c); best-effort CPU, not how the reference runs"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    w = WORKLOADS[args.workload]
    sample = cpu_sample_config(w)
    ref = CpuReference(sample)
    for _ in range(args.warmup):
        ref.step()
    t = 0.0
    for _ in range(args.steps):
        dt, _ = ref.step()
        t += dt
    ms = 1e3 * t / max(args.steps, 1)
    value = ref.units_per_frame() / (ms * 1e-3)
    desc = f"{sample['nodes']} nodes, {sample['units']} skinned meshes x {BONES} bones x {sample['verts_per_unit']} verts, {sample['frusta']} frusta, 1 frame per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "desc": w["desc"], "sample": desc,
                   "note": "reference = Fyrox's single-threaded CPU path restated in C (oracle/; the Rust reference is not buildable here: no cargo)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc,
                         "note": "1 thread because the reference's path is single-threaded (SURVEY §0 D2); cpu_multicore is the best-effort all-cores variant"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:
        line["cpu_multicore"] = time_multicore(ref, max(2, min(args.steps, 5)))
    except Exception as ex:
        line["cpu_multicore"] = {"value": None, "note": f"failed: {ex!r}"}
    # ONE frame of the FULL workload (the CUDA arm's exact config), so that a same-config number exists next to the
    # bounded-sample throughput above; skipped when the sample says it would take more than ~90 s
    full = dict(nodes=w["nodes"], units=w["units"], verts_per_unit=w["verts_per_unit"], frusta=w["frusta"])
    est_s = (full["nodes"] + full["units"] * full["verts_per_unit"]) / max(value, 1.0)
    setup_est_s = 0.0035 * full["units"] + 2e-6 * full["nodes"]  # measured: vertex generation + oracle surfaces dominate the set-up
    if not args.no_full_frame and args.gpus == 1 and full != sample and est_s + setup_est_s < 240.0:
        try:
            del ref
            t0 = time.perf_counter()
            big = CpuReference(full)
            setup_s = time.perf_counter() - t0
            dt, _ = big.step()
            line["full_workload_frame"] = {"value": big.units_per_frame() / dt, "unit": UNIT, "ms": 1e3 * dt, "frames": 1, "same_config_as_cuda_arm": True,
                                           "nodes": full["nodes"], "skinned_meshes": full["units"], "frusta": full["frusta"], "setup_s": round(setup_s, 1), "cores": 1, "kind": "port"}
            del big
        except Exception as ex:
            line["full_workload_frame"] = {"value": None, "note": f"failed: {ex!r}"}
    else:
        line["full_workload_frame"] = {"value": None, "note": (f"skipped (estimated {est_s:.0f} s per frame + {setup_est_s:.0f} s set-up; only run at --gpus 1)"
                                                                if full != sample else "the sample IS the full workload")}
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------------
# the CUDA arm
# --------------------------------------------------------------------------------------------------
def load_scene(ctx, sc, fb, log):
    t0 = time.time()
    ctx.set_topology(sc.parent, sc.flags, sc.render_mask, sc.local_aabb, root=0, global_index=sc.global_index)
    ctx.set_local_matrices(sc.local_m16)
    nu, V = sc.n_units, sc.verts_per_unit
    if nu:
        ctx.reserve_skinning(nu * BONES, nu * V)
        chunk = max(1, min(nu, (256 << 20) // (V * 68)))
        pin = fb.PinnedBuffer((chunk * V * 68,), np.uint8)
        aabbs = np.empty((chunk, 6), np.float32)
        mesh_nodes = np.empty(nu, np.uint32)
        all_aabb = np.empty((nu, 6), np.float32)
        for u0 in range(0, nu, chunk):
            cnt = min(chunk, nu - u0)
            sc.units_vertices_into(u0, cnt, pin.ptr, aabbs)
            for i in range(cnt):
                u = u0 + i
                mesh_nodes[u] = sc.unit_mesh_node(u)
                ctx.add_skinned_surface(int(mesh_nodes[u]), sc.unit_bone_nodes(u), sc.unit_inv_bind(u), pin.ptr + i * V * 68, n_verts=V)
            all_aabb[u0:u0 + cnt] = aabbs[:cnt]
            ctx.sync()
        ctx.set_local_aabbs(all_aabb, mesh_nodes)  # Mesh::local_bounding_box = bounds of the vertices
        ctx.commit_surfaces()
        pin.free()
    log(f"scene on device in {time.time() - t0:.1f}s: {sc.capacity} nodes, {nu} skinned meshes, {nu * V} verts")


def device_animation_mode(ctx, sc, fb, frusta, n_bones, steps, timed, log):
    """N2: one Animation per skinned mesh (64 rotation tracks of kind UnitQuaternion, 4 linear keys per curve over a
    2 s loop, built from the generator's animation frames), sampled on the device every frame.  Returns the
    end-to-end ms/frame (two frames in flight, visible lists read back, zero bytes uploaded) and the animation
    kernels' own time."""
    K, T = 4, 2.0
    idx, _ = sc.animate_trs(0)
    rots = np.stack([sc.animate_trs(k)[1][:, 3:7] for k in range(K)], axis=2)  # (bones, 4 components, K keys)
    keys = np.zeros((n_bones, 4, K), fb.Context.KEY_DTYPE)
    keys["location"] = (np.arange(K, dtype=np.float32) * np.float32(T / (K - 1)))[None, None, :]
    keys["value"] = rots
    keys["kind"] = 1  # Linear
    bones = sc.bones_per_unit
    tracks = np.zeros(n_bones, fb.Context.TRACK_DTYPE)
    tracks["target_node"] = idx
    tracks["binding"] = 2  # Rotation
    tracks["value_kind"] = 5  # UnitQuaternion
    tracks["enabled"] = 1
    tracks["n_curves"] = 4
    local = (np.arange(n_bones, dtype=np.uint32) % bones) * (4 * K)  # key offsets are relative to the animation's own keys
    tracks["first_key"] = local[:, None] + (np.arange(4, dtype=np.uint32) * K)[None, :]
    tracks["n_keys"] = K
    keys = keys.reshape(-1)
    rng = np.random.default_rng(SEED)
    phase = rng.uniform(0.0, T, sc.n_units).astype(np.float32)
    t0 = time.perf_counter()
    for u in range(sc.n_units):
        ctx.anim_add(tracks[u * bones:(u + 1) * bones], keys[u * bones * 4 * K:(u + 1) * bones * 4 * K], speed=1.0, looped=True,
                     time_slice=(0.0, T), time_position=float(phase[u]))
    dt = 1.0 / 60.0

    def frames(n):
        for i in range(n):
            ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=frusta, readback_visible=True, async_=True, animate_dt=dt)
            if i:
                ctx.frame_wait()
        ctx.frame_wait()

    frames(3)
    log(f"device animation: {sc.n_units} animations, {n_bones} tracks, {keys.size} keys added in {time.perf_counter() - t0:.1f} s")
    ms = timed(lambda: frames(steps), 1) / steps
    anim_ms = 0.0
    for _ in range(steps):
        ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=frusta, readback_visible=False, animate_dt=dt)
        anim_ms += ctx.timings()["upload_ms"] / steps  # EV_START..EV_UPLOAD brackets the animation kernels (nothing is uploaded)
    ctx.anim_clear()
    per_bone = 4 * 2 * 20 + 32 + 48 + 4 + 2 * 16 + 4 + 2 * 40 + 48 + 4  # keys of the span, hints r/w, track, value w/r, TRS r/w, L, flag
    return {"e2e_ms_per_step": ms, "h2d_bytes_per_step": 0, "animation_kernels_ms": anim_ms, "animations": int(sc.n_units), "tracks": int(n_bones),
            "keys": int(keys.size), "approx_bytes_per_bone": per_bone,
            "animation_GBps": per_bone * n_bones / max(anim_ms, 1e-6) / 1e-3 / 1e9}


def oracle_frusta(n_frusta: int):
    """The bench's observers through the oracle's own restatement (parity block only)."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import oracle_binding as ob

    if n_frusta == 1:
        view = ob.look_at_rh((0, 0, 0), (0, 0, -1), (0, 1, 0))
        return [ob.frustum_from_vp(ob.mat4_mul(ob.perspective(16 / 9, float(np.deg2rad(60.0)), 0.1, 150.0), view))]
    faces = [((1, 0, 0), (0, -1, 0)), ((-1, 0, 0), (0, -1, 0)), ((0, 1, 0), (0, 0, 1)), ((0, -1, 0), (0, 0, -1)), ((0, 0, 1), (0, -1, 0)), ((0, 0, -1), (0, -1, 0))]
    return [ob.frustum_from_vp(ob.mat4_mul(ob.perspective(1.0, float(np.pi / 2), 0.01, 120.0), ob.look_at_rh((0, 0, 0), look, up))) for look, up in faces[:n_frusta]]


def dump_outputs(ctx, sc, n_frusta, out_dir, log):
    """Write what the last timed frame computed, as a caller of fyx_render_prep receives it, to out_dir/<name>.npy (float32 or
    float64): for a fixed, seeded sample of nodes their global matrices, world boxes and per-frustum visibility; the length
    and id sum of every visible list; the palettes and skinned streams of a few skinned meshes.  The visible lists are
    compared as sets (their order is not part of the result), and two builds run with the same arguments get the same
    inputs, so their dumps compare array for array."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from sampled_parity import SortedList

    ctx.sync()
    rng = np.random.default_rng(SEED)
    nodes = np.unique(rng.integers(0, sc.capacity, DUMP_NODES)).astype(np.uint32)
    gid = sc.global_index[nodes]
    lists = [SortedList(ctx.get_visible(f, copy=False)) for f in range(n_frusta)]
    out = {
        "node_index": gid.astype(np.float64),
        "global_matrices": ctx.get_global_matrices(nodes),
        "world_aabbs": ctx.get_world_aabbs(nodes),
        "visible": np.stack([sl.contains(gid) for sl in lists], axis=1).astype(np.float32),
        "visible_counts": np.array([sl.a.size for sl in lists], np.float64),
        "visible_id_sums": np.array([sl.a.sum(dtype=np.uint64) for sl in lists], np.float64),
    }
    if sc.n_units:  # surface id = unit index (load_scene adds them in order)
        units = np.unique(np.concatenate([[0, sc.n_units - 1], rng.integers(0, sc.n_units, DUMP_UNITS - 2)]))
        skinned = [ctx.get_skinned(int(u)) for u in units]
        out["skinned_unit_index"] = units.astype(np.float64)
        out["palettes"] = np.stack([ctx.get_palette(int(u)) for u in units])
        out["skinned_positions"] = np.stack([p for p, _ in skinned])
        out["skinned_normals"] = np.stack([n for _, n in skinned])
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"dumped {len(out)} arrays ({total / 1e6:.1f} MB) of the last timed frame to {out_dir}")


def parity_block(ctx, sc, fb, frusta, upload, world, rank, dist, log):
    """Sampled-oracle check of the context that was just timed (outside every timed region; the oracle is the checker,
    never on the product path).  One more synchronous frame with animation frame 0, then per rank: >= 5 000 sampled
    nodes (global matrix and world box bit-exact, per-frustum visibility identical) incl. skinned-mesh nodes with their
    bone folds, and 4 skinned meshes bit-exact (palette, positions, normals).  N > 1: rank 0's GATHERED host lists are
    checked against every rank's sampled truth and against the checksum of every rank's own list."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import sampled_parity as sp

    t0 = time.time()
    idx0 = pay0 = None
    if sc.n_units:
        idx0, pay0 = sc.animate(0) if upload == "m16" else sc.animate_trs(0)
    out, res = sp.check_frame(ctx, sc, frusta, oracle_frusta(len(frusta)), upload, idx0, pay0, allgather=(world > 1), seed=SEED + rank)
    out["ranks"] = world
    if world > 1:
        mine = {"gid": res["sample_gid"], "vis": res["sample_vis"], "sums": res["own_sums"], "ok": out["ok"],
                "nodes": out["checked_nodes"], "verts": out["checked_verts"], "err": out["max_abs_pos_err"]}
        allp = [None] * world if rank == 0 else None
        dist.gather_object(mine, allp, dst=0)
        if rank == 0:
            gathered = [ctx.get_visible_gathered(f) for f in range(len(frusta))]
            g_ok, c_ok = True, True
            for f, lst in enumerate(gathered):
                sl = sp.SortedList(lst)
                g_ok &= sl.duplicate_free
                for p in allp:
                    g_ok &= bool(np.array_equal(sl.contains(p["gid"]), p["vis"][:, f]))
                n, sm, x = sp.list_checksum(lst)
                c_ok &= n == sum(p["sums"][f][0] for p in allp) and sm == sum(p["sums"][f][1] for p in allp) % (1 << 64)
                xr = 0
                for p in allp:
                    xr ^= p["sums"][f][2]
                c_ok &= x == xr
            out["gathered_lists_match_every_ranks_truth"] = bool(g_ok)
            out["gathered_equals_union_of_own_lists"] = bool(c_ok)
            out["all_ranks_ok"] = bool(all(p["ok"] for p in allp))
            out["checked_nodes"] = int(sum(p["nodes"] for p in allp))
            out["checked_verts"] = int(sum(p["verts"] for p in allp))
            out["max_abs_pos_err"] = float(max(p["err"] for p in allp))
            out["visible_set_equal"] = bool(out["visible_set_equal"] and g_ok and c_ok and out["all_ranks_ok"])
            out["ok"] = bool(out["ok"] and out["visible_set_equal"])
        else:
            ctx.sync()
    out["seconds"] = round(time.time() - t0, 2)
    out["how"] = "sampled oracle (tests/sampled_parity.py) on the timed context after the timed regions; bit-exact compares"
    log(f"parity: {out}")
    return out


def measure(args, wname, strong, steps, env, full, dump_dir=None):
    """All timed regions (+ the parity block) of one workload on this rank's GPU.  `strong`: the workload's sizes are
    the WHOLE job, sharded over the ranks (strong scaling); otherwise they are per GPU (weak scaling).
    `full`: also the secondary modes (static+skeletons, device animation) and the synchronous e2e.
    `dump_dir`: write the outputs of the last all-dirty timed frame there (dump_outputs) before anything else runs."""
    import torch

    import fyrox_b200 as fb
    from fyrox_b200 import camera
    from fyrox_b200.scenegen import Scene

    rank, world, local_rank, dist, log, barrier = env["rank"], env["world"], env["local_rank"], env["dist"], env["log"], env["barrier"]
    w = WORKLOADS[wname]
    mult = 1 if strong else world
    sc = Scene(w["nodes"] * mult, n_units=w["units"] * mult, verts_per_unit=w["verts_per_unit"], bones_per_unit=BONES, seed=SEED, rank=rank, nranks=world)
    tstream = env["tstream"]
    ctx = fb.Context(device=local_rank, stream=tstream.cuda_stream)
    load_scene(ctx, sc, fb, log)
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(fb.Context.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        ctx.comm_init(world, rank, bytes(uid.cpu().numpy().tobytes()))

    frusta = [camera.camera_frustum()] if w["frusta"] == 1 else camera.cube_frusta()[: w["frusta"]]
    n_local_nodes = sc.capacity
    n_local_verts = sc.n_units * sc.verts_per_unit
    n_bones = sc.n_units * BONES

    # per-frame host inputs: two animation frames in pinned memory, alternated
    # upload format of the changed bones: "rot" = the rotations the animation rewrote (16 B; position / scale stay on the
    # device), "trs" = position/rotation/scale records (40 B) — the device evaluates Transform::calculate_local_transform
    # (SURVEY §8f N1) in both — or "m16" = the 64-byte matrices
    anim = []
    if n_bones:
        for fr in range(2):
            pi = fb.PinnedBuffer((n_bones,), np.uint32)
            if args.upload == "rot":
                full_trs = fb.PinnedBuffer((n_bones, 10), np.float32)
                sc.animate_trs_into(fr, pi.ptr, full_trs.ptr)
                if fr == 0:
                    ctx.set_local_trs(full_trs.array, pi.array)  # the device keeps every bone's position / scale from here on
                pm = fb.PinnedBuffer((n_bones, 4), np.float32)
                pm.array[:] = full_trs.array[:, 3:7]
                full_trs.free()
            elif args.upload == "trs":
                pm = fb.PinnedBuffer((n_bones, 10), np.float32)
                sc.animate_trs_into(fr, pi.ptr, pm.ptr)
            else:
                pm = fb.PinnedBuffer((n_bones, 16), np.float32)
                sc.animate_into(fr, pi.ptr, pm.ptr)
            anim.append((pi, pm))

    def step_device():
        # N > 1: the all-gather of the visible lists is part of the frame (overlapped with the skinning kernel)
        ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=frusta, do_palettes=True, do_skin=True, readback_visible=False, async_=True,
                        allgather=(world > 1))

    vis_counts = [0] * len(frusta)

    def submit_e2e(i, pipelined):
        # N > 1: every rank holds the gathered lists on its device and brings its OWN lists to the host (its PCIe link);
        # fyx_get_visible_gathered then reads the whole lists from the host segment all ranks wrote into
        kw = dict(update_flags=fb.UPDATE_ALL, frusta=frusta, readback_visible=True, async_=pipelined, allgather=(world > 1))
        if anim:
            pi, pm = anim[i & 1]
            kw.update(changed_idx=pi.ptr, n_changed=n_bones, **{UPLOAD_FIELD[args.upload]: pm.ptr})
        ctx.render_prep(**kw)

    def collect_e2e():
        for f in range(len(frusta)):
            v = ctx.get_visible_gathered(f, copy=False) if world > 1 else ctx.get_visible(f, copy=False)
            vis_counts[f] = v.size

    def step_e2e(i):
        """One frame through the C ABI with host buffers, synchronous: upload -> kernels -> read-back."""
        submit_e2e(i, False)
        collect_e2e()

    def run_e2e_pipelined(n):
        """The same K frames, two in flight (FYX_FRAME_ASYNC + fyx_frame_wait): the upload of frame i+1 and
        the read-back of frame i-1 overlap the kernels of frame i.  Every frame's inputs still travel
        host->device and every frame's visible lists device->host inside the timed region."""
        submit_e2e(0, True)
        for i in range(1, n):
            submit_e2e(i, True)
            ctx.frame_wait()
            collect_e2e()
        ctx.frame_wait()
        collect_e2e()

    def timed(fn, n, pass_index=False):
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i) if pass_index else fn()
        e1.record()
        torch.cuda.synchronize()
        ctx.sync()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # warm-up (both paths), then the timed regions; inputs (>1.6 GB of node columns, vertex streams) exceed the 126 MB L2
    for i in range(max(args.warmup, 3)):
        step_device()
    ctx.sync()
    for i in range(max(args.warmup, 3)):
        step_e2e(i)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = ctx.kernel_launch_count()
    total_ms = timed(step_device, steps)
    launches = ctx.kernel_launch_count() - launches0
    if dump_dir:
        dump_outputs(ctx, sc, len(frusta), dump_dir, log)
    e2e_sync_ms = timed(step_e2e, steps, pass_index=True) if full else None
    for _ in range(2):
        run_e2e_pipelined(3)
    e2e_pipe_ms = timed(lambda: run_e2e_pipelined(steps), 1)
    e2e_ms = e2e_pipe_ms if e2e_sync_ms is None else min(e2e_sync_ms, e2e_pipe_ms)
    # per-stage device durations: a SEPARATE pass of synchronous frames (CUDA events between the kernels, recorded
    # inside fyx_render_prep on the launching stream).  Their sum exceeds ms_per_step: the timed frames above are
    # asynchronous, record no mid-frame events and overlap each kernel's prologue with its predecessor's tail (PDL).
    stage = {"update_ms": 0.0, "palette_ms": 0.0, "skin_ms": 0.0}
    for i in range(steps):
        ctx.render_prep(update_flags=fb.UPDATE_ALL, frusta=frusta, readback_visible=False)
        t = ctx.timings()
        for k in stage:
            stage[k] += t[k] / steps
    # second mode BASELINE.md asks for: "static + skeletons" — only the bones change (uploaded every frame),
    # Graph::update semantics (FYX_UPDATE_INCREMENTAL): clean sub-trees keep their matrices / boxes, everything is culled
    inc_ms = None
    if full and anim and world == 1:
        def inc_frames(n):
            for i in range(n):
                pi, pm = anim[i & 1]
                kw = {UPLOAD_FIELD[args.upload]: pm.ptr}
                ctx.render_prep(update_flags=fb.UPDATE_INCREMENTAL, changed_idx=pi.ptr, n_changed=n_bones, frusta=frusta,
                                readback_visible=True, async_=True, **kw)
                if i:
                    ctx.frame_wait()
            ctx.frame_wait()
        inc_frames(3)
        inc_ms = timed(lambda: inc_frames(steps), 1) / steps
    # third mode (N2): the animation players run on the device — the bones' rotation curves are resident in HBM, every
    # frame samples them (fyx_render_prep do_animate), nothing is uploaded; the visible lists still come down
    dev_anim = None
    if full and anim and world == 1 and not args.no_device_animation:
        dev_anim = device_animation_mode(ctx, sc, fb, frusta, n_bones, steps, timed, log)
    clk = clocks.stop() if rank == 0 else None

    parity = None
    if not args.no_parity:
        try:
            parity = parity_block(ctx, sc, fb, frusta, args.upload, world, rank, dist, log)
        except Exception as ex:  # reported, never hidden: a failed check is a failed check
            parity = {"ok": False, "error": repr(ex)}
            if world > 1:
                raise

    xstats = None
    if world > 1:
        try:  # the exchange of one more device-resident frame, timed on the collective stream (it overlaps the skinning kernel)
            step_device()
            ctx.sync()
            xs = ctx.comm_stats()
            xstats = {"device_ms": xs["device_ms"], "entries_own": int(xs["entries_own"]), "entries_gathered": int(xs["entries_total"]),
                      "nvlink_egress_bytes_per_rank": int(xs["egress_bytes"]), "algorithmic_bytes_4_N_Vvis": 4 * int(xs["entries_own"]) * world,
                      "egress_GBps": xs["egress_bytes"] / max(xs["device_ms"], 1e-6) / 1e6,
                      "note": "device_ms spans counts -> push -> wait for every peer on the collective stream, beside k_palette / k_skin"}
        except Exception as ex:
            xstats = {"error": repr(ex)}
    ms_per_step = total_ms / steps
    e2e_ms_per_step = e2e_ms / steps
    units_all = (w["nodes"] + w["units"] * w["verts_per_unit"]) * mult  # whole job
    sum_vis = sum(vis_counts)
    own_vis = sum(int(ctx.get_visible(f, copy=False).size) for f in range(len(frusta))) if not args.no_parity else sum_vis // world
    h2d = n_bones * (UPLOAD_BYTES[args.upload] + 4)  # frusta travel as kernel parameters
    d2h = 4 * len(frusta) + 4 * own_vis  # every rank brings its own lists down (N > 1: into the host segment all ranks share)

    peak, peak_src = peaks()
    # dominant kernel: k_skin when the workload skins, else the fused update+cull level kernels
    stages = {}
    if n_local_verts:
        g = B_VERT * n_local_verts / (stage["skin_ms"] * 1e-3) / 1e9
        stages["k_skin"] = {"ms": stage["skin_ms"], "algorithmic_bytes": B_VERT * n_local_verts, "GBps": g, "frac": g / peak}
    upd_bytes = B_NODE_FUSED * n_local_nodes + B_VISIBLE * own_vis
    g = upd_bytes / (stage["update_ms"] * 1e-3) / 1e9
    stages["k_update_level+cull"] = {"ms": stage["update_ms"], "algorithmic_bytes": upd_bytes, "GBps": g, "frac": g / peak}
    if n_bones:
        g = B_BONE * n_bones / max(stage["palette_ms"], 1e-6) / 1e-3 / 1e9
        stages["k_palette"] = {"ms": stage["palette_ms"], "algorithmic_bytes": B_BONE * n_bones, "GBps": g, "frac": g / peak}
    dom = "k_skin" if n_local_verts and stage["skin_ms"] >= stage["update_ms"] else "k_update_level+cull"
    traffic = None
    tpath = os.path.join(REPO, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            ent = json.load(open(tpath)).get(wname, {}).get(dom)
            traffic = ent.get("dram_bytes_per_launch") if ent else None
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": dom, "achieved": stages[dom]["GBps"], "peak": peak, "unit": "GB/s", "frac": stages[dom]["frac"],
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": stages[dom]["algorithmic_bytes"], "stages": stages,
                "stages_note": "stage times come from a separate pass of synchronous frames with events between the kernels; "
                               "ms_per_step is timed on asynchronous frames without them (PDL overlap), so the stage sum exceeds it"}
    res = dict(w=w, world=world, strong=strong, steps=steps, ms_per_step=ms_per_step, e2e_ms_per_step=e2e_ms_per_step,
               e2e_sync_ms=None if e2e_sync_ms is None else e2e_sync_ms / steps, e2e_pipe_ms=e2e_pipe_ms / steps, units_all=units_all,
               sum_vis=sum_vis, own_vis=own_vis, h2d=h2d, d2h=d2h, launches=int(launches), roofline=roofline, clocks=clk, parity=parity,
               inc_ms=inc_ms, dev_anim=dev_anim, frusta=len(frusta), n_local_nodes=n_local_nodes, n_local_verts=n_local_verts,
               exchange={"mode": ctx.comm_mode(), "last_frame": xstats} if world > 1 else None)
    for pi, pm in anim:
        pi.free()
        pm.free()
    ctx.close()
    sc.close()
    torch.cuda.empty_cache()
    return res


def run_cuda(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch N>1 with torchrun (one process per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: bench.py has no CPU fallback for the CUDA arm (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def log(msg):
        if rank == 0 and args.verbose:
            print("[bench]", msg, file=sys.stderr, flush=True)

    def barrier():
        if world > 1:
            dist.barrier()

    from fyrox_b200 import scenegen as _sg
    _sg.set_threads(max(1, (os.cpu_count() or 8) // max(world, 1)))  # torchrun exports OMP_NUM_THREADS=1
    # the contexts launch on an explicit torch stream so that torch.cuda.Event brackets exactly their work
    tstream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(tstream)
    assert tstream.cuda_stream != 0
    env = dict(rank=rank, world=world, local_rank=local_rank, dist=dist, log=log, barrier=barrier, tstream=tstream)

    w = WORKLOADS[args.workload]
    strong_main = args.workload == "C5"
    r = measure(args, args.workload, strong_main, args.steps, env, full=True, dump_dir=args.dump_outputs if rank == 0 else None)
    # BASELINE.json configs[4] / north_star: the 100 M-node config, STRONG scaling (the whole job is fixed, sharded N ways)
    c5 = None
    if args.workload == "C4" and not args.no_c5:
        try:
            c5 = measure(args, "C5", True, max(3, min(args.steps, 10)), env, full=False)
        except Exception as ex:
            if world > 1:
                raise
            c5 = {"error": repr(ex)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    ms_per_step, e2e_ms_per_step = r["ms_per_step"], r["e2e_ms_per_step"]
    value = r["units_all"] / (ms_per_step * 1e-3)
    mult = 1 if strong_main else world
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong_main else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "desc": w["desc"], "nodes_per_gpu": r["n_local_nodes"], "skinned_meshes_per_gpu": w["units"] * mult // world,
                   "bones_per_mesh": BONES, "verts_per_mesh": w["verts_per_unit"], "skinned_verts_per_gpu": r["n_local_verts"],
                   "frusta": r["frusta"], "update": "all-dirty (every node recomputed)", "parallelism": f"shard{world}" if world > 1 else "single",
                   "l2": "inputs larger than L2 (node columns + vertex streams >> 126 MB); no flush needed", "visible_entries": r["sum_vis"],
                   "exchange": r["exchange"]},
        "fps": 1e3 / ms_per_step,
        "nodes_per_s": w["nodes"] * mult / (ms_per_step * 1e-3), "verts_per_s": w["units"] * w["verts_per_unit"] * mult / (ms_per_step * 1e-3),
        "clocks": r["clocks"],
        "e2e": {"value": r["units_all"] / (e2e_ms_per_step * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_per_step, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                "api": "fyx_render_prep (C ABI) with pinned host buffers: changed bone " + {"rot": "rotations (16 B)", "trs": "TRS records (40 B)", "m16": "matrices (64 B)"}[args.upload] + " up, visible lists down"
                       + ("; per rank: its own lists, into the host segment every rank shares (rank 0 reads the whole lists there)" if world > 1 else ""),
                "mode": "pipelined (2 frames in flight, fyx_frame_wait)" if r["e2e_sync_ms"] is None or r["e2e_pipe_ms"] < r["e2e_sync_ms"] else "synchronous",
                "ms_per_step_synchronous": r["e2e_sync_ms"], "ms_per_step_pipelined": r["e2e_pipe_ms"],
                "consumer": "visible lists on the host; palettes and skinned streams stay device-resident (the consumer of seam S3 is assumed to be on the GPU)"},
        "gpu_launches": r["launches"],
        "roofline": r["roofline"],
        "parity": r["parity"],
        "modes": {"all_dirty_ms_per_step": ms_per_step, "static_plus_skeletons_e2e_ms_per_step": r["inc_ms"], "device_animation": r["dev_anim"]},
    }
    if c5 is not None:
        if "error" in c5:
            line["modes"]["strong_C5"] = c5
        else:
            line["modes"]["strong_C5"] = {
                "workload": "C5", "desc": WORKLOADS["C5"]["desc"], "scaling": "strong", "n_gpus": world, "steps": c5["steps"],
                "ms_per_step": c5["ms_per_step"], "value": c5["units_all"] / (c5["ms_per_step"] * 1e-3), "unit": UNIT,
                "e2e_ms_per_step": c5["e2e_ms_per_step"], "e2e_value": c5["units_all"] / (c5["e2e_ms_per_step"] * 1e-3),
                "h2d_bytes_per_step": c5["h2d"], "d2h_bytes_per_step": c5["d2h"], "nodes_per_gpu": c5["n_local_nodes"], "skinned_verts_per_gpu": c5["n_local_verts"],
                "visible_entries": c5["sum_vis"], "gpu_launches": c5["launches"], "roofline_stages": c5["roofline"]["stages"], "parity": c5["parity"],
                "exchange": c5["exchange"],
                "note": "whole job = 100 M nodes + 1 G skinned vertices + 6 frusta whatever N is; speed-up at N GPUs = this value / the N=1 line's value"}
    if world == 1 and not args.no_cpu_baseline:
        try:
            sample = cpu_sample_config(w)
            ref = CpuReference(sample)
            ref.step()
            t, n = 0.0, 0
            while n < 2:
                dt, _ = ref.step()
                t += dt
                n += 1
            desc = f"{sample['nodes']} nodes, {sample['units']} skinned meshes x {BONES} bones x {sample['verts_per_unit']} verts, {sample['frusta']} frusta; {n} frames"
            line["cpu_baseline"] = {"value": ref.units_per_frame() * n / t, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc,
                                    "host_cores_available": os.cpu_count()}
            try:
                line["cpu_baseline"]["multicore"] = time_multicore(ref, 3)
            except Exception as ex:
                line["cpu_baseline"]["multicore"] = {"value": None, "note": f"failed: {ex!r}"}
        except Exception as ex:  # the baseline is reported, never allowed to break the measurement
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "port", "sample": f"failed: {ex!r}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--upload", default="rot", choices=["rot", "trs", "m16"], help="per-frame upload format of the changed bones")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-device-animation", action="store_true", help="skip the extra mode that samples the bones' animation curves on the device")
    ap.add_argument("--no-full-frame", action="store_true", help="reference arm: skip the one frame of the full workload that follows the bounded sample")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled-oracle check that follows the timed regions")
    ap.add_argument("--no-c5", action="store_true", help="skip the strong-scaling C5 measurement that follows the default C4 workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                    "(a fixed, seeded sample; rank 0's context when N > 1)")
    ap.add_argument("--verbose", action="store_true")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA arm's timed path")
    # OpenMP workers (scene generator, multi-core CPU baseline) that wait at a barrier should sleep, not spin: the host is
    # shared with the other ranks and possibly quota-limited (must be set before libgomp is loaded)
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    # stdout carries exactly ONE JSON line: libraries that write to fd 1 (NCCL prints its version banner there when
    # NCCL_DEBUG=VERSION) are sent to stderr for the whole run, the line goes out through the saved descriptor
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w")
    try:
        if args.impl == "reference":
            return run_reference(args)
        return run_cuda(args)
    finally:
        sys.stdout.flush()


if __name__ == "__main__":
    sys.exit(main())
