"""ctypes binding of oracle/libfyrox_oracle.so — the CPU restatement of the reference path.

TEST INFRASTRUCTURE: imported only from tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs.  Never from fyrox_b200/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(REPO, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "libfyrox_oracle.so")

NONE = 0xFFFFFFFF
KIND_PIVOT, KIND_MESH = 0, 1

f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)


class Plane(C.Structure):
    _fields_ = [("n", C.c_float * 3), ("d", C.c_float)]


class Frustum(C.Structure):
    _fields_ = [("planes", Plane * 6), ("corners", (C.c_float * 3) * 8)]


class Aabb(C.Structure):
    _fields_ = [("min", C.c_float * 3), ("max", C.c_float * 3)]

    @staticmethod
    def make(mn, mx):
        a = Aabb()
        for i in range(3):
            a.min[i] = mn[i]
            a.max[i] = mx[i]
        return a

    def to_np(self):
        return np.array(list(self.min) + list(self.max), dtype=np.float32)


class Transform(C.Structure):
    _fields_ = [
        ("local_position", C.c_float * 3),
        ("local_rotation", C.c_float * 4),
        ("local_scale", C.c_float * 3),
        ("pre_rotation", C.c_float * 4),
        ("post_rotation_matrix", C.c_float * 9),
        ("rotation_offset", C.c_float * 3),
        ("rotation_pivot", C.c_float * 3),
        ("scaling_offset", C.c_float * 3),
        ("scaling_pivot", C.c_float * 3),
    ]


class VertexLayout(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("stride", "position_offset", "normal_offset", "bone_weights_offset", "bone_indices_offset")]


ANIMATED_VERTEX = VertexLayout(68, 0, 20, 48, 64)

_lib = None


def build():
    r = subprocess.run(["make", "-C", ORACLE_DIR, "all"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(r.stdout + r.stderr)


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    src = os.path.join(ORACLE_DIR, "fyrox_oracle.c")
    # a stale library is rebuilt only where the tree is writable: a read-only install (bench.py's CPU baseline and parity
    # block) uses what build() made, whatever mtimes a copy of the tree left on the sources
    missing = not os.path.exists(ORACLE_LIB)
    stale = not missing and os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(ORACLE_LIB)
    if missing or (stale and os.access(ORACLE_DIR, os.W_OK)):
        build()
    L = C.CDLL(ORACLE_LIB)
    vp = C.c_void_p
    sig = {
        "orc_plane_from_abcd": (C.c_int, [C.c_float] * 4 + [C.POINTER(Plane)]),
        "orc_plane_dot": (C.c_float, [C.POINTER(Plane), f32p]),
        "orc_plane_intersection_point": (None, [C.POINTER(Plane)] * 3 + [f32p]),
        "orc_frustum_from_view_projection_matrix": (C.c_int, [f32p, C.POINTER(Frustum)]),
        "orc_frustum_default": (None, [C.POINTER(Frustum)]),
        "orc_frustum_is_intersects_point_cloud": (C.c_int, [C.POINTER(Frustum), f32p, C.c_size_t]),
        "orc_frustum_is_intersects_aabb": (C.c_int, [C.POINTER(Frustum), C.POINTER(Aabb)]),
        "orc_frustum_is_intersects_aabb_offset": (C.c_int, [C.POINTER(Frustum), C.POINTER(Aabb), f32p]),
        "orc_frustum_is_contains_point": (C.c_int, [C.POINTER(Frustum), f32p]),
        "orc_aabb_default": (None, [C.POINTER(Aabb)]),
        "orc_aabb_unit": (None, [C.POINTER(Aabb)]),
        "orc_aabb_add_point": (None, [C.POINTER(Aabb), f32p]),
        "orc_aabb_add_box": (None, [C.POINTER(Aabb), C.POINTER(Aabb)]),
        "orc_aabb_corners": (None, [C.POINTER(Aabb), f32p]),
        "orc_aabb_is_valid": (C.c_int, [C.POINTER(Aabb)]),
        "orc_aabb_is_degenerate": (C.c_int, [C.POINTER(Aabb)]),
        "orc_aabb_is_contains_point": (C.c_int, [C.POINTER(Aabb), f32p]),
        "orc_aabb_transform": (None, [C.POINTER(Aabb), f32p, C.POINTER(Aabb)]),
        "orc_mat4_identity": (None, [f32p]),
        "orc_mat4_mul": (None, [f32p, f32p, f32p]),
        "orc_mat4_transform_point": (None, [f32p, f32p, f32p]),
        "orc_quat_to_rotation_matrix": (None, [f32p, f32p]),
        "orc_look_at_rh": (None, [f32p, f32p, f32p, f32p]),
        "orc_perspective": (None, [C.c_float] * 4 + [f32p]),
        "orc_orthographic": (None, [C.c_float] * 6 + [f32p]),
        "orc_transform_identity": (None, [C.POINTER(Transform)]),
        "orc_transform_calculate_local": (None, [C.POINTER(Transform), f32p]),
        "orc_calculate_sorting_index": (C.c_uint64, [f32p, f32p]),
        "orc_graph_new": (vp, []),
        "orc_graph_free": (None, [vp]),
        "orc_graph_capacity": (C.c_uint32, [vp]),
        "orc_graph_root": (C.c_uint32, [vp]),
        "orc_graph_add_node": (C.c_uint32, [vp, C.c_int]),
        "orc_graph_link_nodes": (None, [vp, C.c_uint32, C.c_uint32]),
        "orc_graph_remove_node": (None, [vp, C.c_uint32]),
        "orc_graph_build": (vp, [C.c_uint32, vp, vp, vp, vp, vp]),
        "orc_node_set_local_matrix": (None, [vp, C.c_uint32, f32p]),
        "orc_node_set_local_transform": (None, [vp, C.c_uint32, C.POINTER(Transform)]),
        "orc_node_set_visibility": (None, [vp, C.c_uint32, C.c_int]),
        "orc_node_set_enabled": (None, [vp, C.c_uint32, C.c_int]),
        "orc_node_set_frustum_culling": (None, [vp, C.c_uint32, C.c_int]),
        "orc_node_set_cast_shadows": (None, [vp, C.c_uint32, C.c_int]),
        "orc_node_set_render_mask": (None, [vp, C.c_uint32, C.c_uint32]),
        "orc_node_set_inv_bind_pose": (None, [vp, C.c_uint32, f32p]),
        "orc_mesh_set_local_aabb": (None, [vp, C.c_uint32, C.POINTER(Aabb)]),
        "orc_mesh_add_surface": (C.c_uint32, [vp, C.c_uint32, C.c_uint32, vp, C.c_uint32, vp, C.POINTER(VertexLayout)]),
        "orc_mesh_recalc_local_aabb": (None, [vp, C.c_uint32]),
        "orc_graph_update": (None, [vp]),
        "orc_graph_update_hierarchical_data": (None, [vp]),
        "orc_graph_drop_messages": (None, [vp]),
        "orc_node_global_transform": (None, [vp, C.c_uint32, f32p]),
        "orc_node_local_matrix": (None, [vp, C.c_uint32, f32p]),
        "orc_node_global_visibility": (C.c_int, [vp, C.c_uint32]),
        "orc_node_is_globally_enabled": (C.c_int, [vp, C.c_uint32]),
        "orc_node_world_bounding_box": (None, [vp, C.c_uint32, C.POINTER(Aabb)]),
        "orc_node_parent": (C.c_uint32, [vp, C.c_uint32]),
        "orc_node_should_be_rendered": (C.c_int, [vp, C.c_uint32, C.POINTER(Frustum), C.c_uint32]),
        "orc_graph_global_scale": (None, [vp, C.c_uint32, f32p, f32p]),
        "orc_from_graph": (C.c_size_t, [vp, C.POINTER(Frustum), C.c_uint32, C.c_int, vp, C.c_size_t]),
        "orc_mesh_bone_matrices": (C.c_uint32, [vp, C.c_uint32, C.c_uint32, f32p]),
        "orc_mesh_skin": (C.c_uint32, [vp, C.c_uint32, C.c_uint32, f32p, f32p]),
        "orc_wrapf": (C.c_float, [C.c_float] * 3),
        "orc_lerpf": (C.c_float, [C.c_float] * 3),
        "orc_cubicf": (C.c_float, [C.c_float] * 5),
        "orc_key_interpolate": (C.c_float, [C.POINTER(CurveKey), C.POINTER(CurveKey), C.c_float]),
        "orc_curve_value_at": (C.c_float, [vp, C.c_uint32, C.c_float, C.POINTER(C.c_uint32)]),
        "orc_quat_from_euler_xyz": (None, [f32p, f32p]),
        "orc_track_value_blend": (None, [C.c_int, f32p, f32p, C.c_float]),
        "orc_track_fetch": (C.c_int, [vp, vp, C.c_float, C.POINTER(C.c_uint32), f32p]),
        "orc_animation_new": (vp, [vp, C.c_uint32, vp, C.c_uint32]),
        "orc_animation_free": (None, [vp]),
        "orc_animation_set_time_position": (None, [vp, C.c_float]),
        "orc_animation_set_time_slice": (None, [vp, C.c_float, C.c_float]),
        "orc_animation_set_speed": (None, [vp, C.c_float]),
        "orc_animation_set_looped": (None, [vp, C.c_int]),
        "orc_animation_set_enabled": (None, [vp, C.c_int]),
        "orc_animation_set_track_enabled": (None, [vp, C.c_uint32, C.c_int]),
        "orc_animation_time_position": (C.c_float, [vp]),
        "orc_animation_is_enabled": (C.c_int, [vp]),
        "orc_update_animations": (None, [vp, C.c_uint32, C.c_float, vp, vp, C.c_uint32]),
        "orc_node_is_alive": (C.c_int, [vp, C.c_uint32]),
        "orc_blend_group_update": (None, [vp, f32p, C.c_uint32, C.c_float, vp, vp, C.c_uint32]),
        "orc_mt_new": (vp, [C.c_uint32, C.c_uint32, vp, vp, vp, vp, vp]),
        "orc_mt_free": (None, [vp]),
        "orc_mt_set_threads": (None, [vp, C.c_int]),
        "orc_mt_set_local_matrices": (None, [vp, C.c_uint32, vp, vp]),
        "orc_mt_set_inv_bind": (None, [vp, C.c_uint32, f32p]),
        "orc_mt_add_surface": (C.c_uint32, [vp, C.c_uint32, C.c_uint32, vp, C.c_uint32, vp, C.POINTER(VertexLayout)]),
        "orc_mt_update": (None, [vp]),
        "orc_mt_cull": (C.c_size_t, [vp, C.POINTER(Frustum), C.c_uint32, C.c_int, vp, C.c_size_t]),
        "orc_mt_skin_surface": (None, [vp, C.c_uint32, f32p, f32p]),
        "orc_mt_skin_all": (None, [vp]),
        "orc_mt_get": (None, [vp, C.c_uint32, f32p, C.POINTER(Aabb), C.POINTER(C.c_uint32)]),
        "orc_node_set_lod_group": (None, [vp, C.c_uint32, C.c_uint32, f32p, f32p, vp, vp]),
        "orc_lod_filter": (None, [vp, f32p, C.c_float, C.c_float, vp]),
        "orc_from_graph_lod": (C.c_size_t, [vp, C.POINTER(Frustum), C.c_uint32, C.c_int, f32p, C.c_float, C.c_float, vp, C.c_size_t]),
        "orc_select_reflection_probe": (C.c_uint32, [vp, f32p]),
        "orc_collect_lights": (C.c_size_t, [vp, C.POINTER(Frustum), vp, C.c_size_t]),
        "orc_node_instance": (C.c_uint64, [vp, C.c_uint32, f32p, f32p, f32p, f32p]),
        "orc_mesh_accurate_world_bounding_box": (None, [vp, C.c_uint32, C.POINTER(Aabb)]),
        "orc_skin_vertices": (None, [f32p, C.c_uint32, vp, C.POINTER(VertexLayout), f32p, f32p]),
        "orc_node_surface_instance": (C.c_uint64, [vp, C.c_uint32, C.c_uint32, f32p, f32p, f32p, f32p, C.POINTER(C.c_int)]),
        "orc_surface_bone_block": (C.c_int, [vp, C.c_uint32, C.c_uint32, f32p]),
        "orc_instance_bone_block": (C.c_int, [vp, C.c_uint32, f32p]),
        "orc_skin_vertices_blend": (None, [f32p, C.c_uint32, vp, C.POINTER(VertexLayout), C.c_uint32, vp, C.c_uint32, f32p, f32p, f32p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


class CurveKey(C.Structure):
    _fields_ = [("location", C.c_float), ("value", C.c_float), ("kind", C.c_uint32), ("left_tangent", C.c_float), ("right_tangent", C.c_float)]


class Track(C.Structure):
    _fields_ = [("target_node", C.c_uint32), ("binding", C.c_uint32), ("value_kind", C.c_uint32), ("enabled", C.c_uint32),
                ("n_curves", C.c_uint32), ("first_key", C.c_uint32 * 4), ("n_keys", C.c_uint32 * 4)]


KEY_CONSTANT, KEY_LINEAR, KEY_CUBIC = 0, 1, 2
TV_REAL, TV_VECTOR2, TV_VECTOR3, TV_VECTOR4, TV_QUAT_EULER, TV_QUAT = range(6)
BIND_POSITION, BIND_SCALE, BIND_ROTATION = 0, 1, 2
KEY_DTYPE = np.dtype([("location", "<f4"), ("value", "<f4"), ("kind", "<u4"), ("left_tangent", "<f4"), ("right_tangent", "<f4")])
TRACK_DTYPE = np.dtype([("target_node", "<u4"), ("binding", "<u4"), ("value_kind", "<u4"), ("enabled", "<u4"), ("n_curves", "<u4"),
                        ("first_key", "<u4", 4), ("n_keys", "<u4", 4)])


def fp(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(f32p)


def vec(*xs):
    return np.array(xs, dtype=np.float32)


# ---- convenience wrappers -------------------------------------------------------------------------
def mat4_mul(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32).reshape(16)
    b = np.ascontiguousarray(b, dtype=np.float32).reshape(16)
    out = np.empty(16, dtype=np.float32)
    lib().orc_mat4_mul(fp(a), fp(b), fp(out))
    return out


def frustum_from_vp(m16):
    m = np.ascontiguousarray(m16, dtype=np.float32).reshape(16)
    f = Frustum()
    ok = lib().orc_frustum_from_view_projection_matrix(fp(m), C.byref(f))
    return f if ok else None


def frustum_planes_corners(f: Frustum):
    planes = np.array([[p.n[0], p.n[1], p.n[2], p.d] for p in f.planes], dtype=np.float32)
    corners = np.array([[c[0], c[1], c[2]] for c in f.corners], dtype=np.float32)
    return planes, corners


def look_at_rh(eye, target, up):
    out = np.empty(16, dtype=np.float32)
    lib().orc_look_at_rh(fp(vec(*eye)), fp(vec(*target)), fp(vec(*up)), fp(out))
    return out


def perspective(aspect, fovy, znear, zfar):
    out = np.empty(16, dtype=np.float32)
    lib().orc_perspective(aspect, fovy, znear, zfar, fp(out))
    return out


def translation(x, y, z):
    m = np.eye(4, dtype=np.float32).T.reshape(16).copy()
    m[12], m[13], m[14] = x, y, z
    return m


def scaling(x, y, z):
    m = np.zeros(16, dtype=np.float32)
    m[0], m[5], m[10], m[15] = x, y, z, 1.0
    return m


class Graph:
    """orc_graph with numpy in/out."""

    def __init__(self, handle=None):
        self.L = lib()
        self.h = handle if handle is not None else self.L.orc_graph_new()

    @staticmethod
    def build(parent, flags=None, render_mask=None, local_m16=None, local_aabb=None):
        L = lib()
        parent = np.ascontiguousarray(parent, dtype=np.uint32)
        n = parent.size

        def p(a, dt):
            if a is None:
                return None, None
            a = np.ascontiguousarray(a, dtype=dt)
            return a, a.ctypes.data_as(C.c_void_p)

        flags, pf = p(flags, np.uint32)
        render_mask, pm = p(render_mask, np.uint32)
        local_m16, pl = p(local_m16, np.float32)
        local_aabb, pa = p(local_aabb, np.float32)
        h = L.orc_graph_build(n, parent.ctypes.data_as(C.c_void_p), pf, pm, pl, pa)
        return Graph(h)

    def free(self):
        if self.h:
            self.L.orc_graph_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @property
    def capacity(self):
        return self.L.orc_graph_capacity(self.h)

    def add_node(self, kind=KIND_PIVOT):
        return self.L.orc_graph_add_node(self.h, kind)

    def link_nodes(self, child, parent):
        self.L.orc_graph_link_nodes(self.h, child, parent)

    def set_local_matrix(self, n, m16):
        m = np.ascontiguousarray(m16, dtype=np.float32).reshape(16)
        self.L.orc_node_set_local_matrix(self.h, n, fp(m))

    def set_inv_bind(self, n, m16):
        m = np.ascontiguousarray(m16, dtype=np.float32).reshape(16)
        self.L.orc_node_set_inv_bind_pose(self.h, n, fp(m))

    def set_visibility(self, n, v):
        self.L.orc_node_set_visibility(self.h, n, int(v))

    def set_enabled(self, n, v):
        self.L.orc_node_set_enabled(self.h, n, int(v))

    def set_local_aabb(self, n, aabb6):
        a = Aabb.make(aabb6[:3], aabb6[3:])
        self.L.orc_mesh_set_local_aabb(self.h, n, C.byref(a))

    def add_surface(self, mesh, bones, verts=None, layout=ANIMATED_VERTEX):
        bones = np.ascontiguousarray(bones, dtype=np.uint32)
        if verts is None:
            return self.L.orc_mesh_add_surface(self.h, mesh, bones.size, bones.ctypes.data_as(C.c_void_p), 0, None, None)
        verts = np.ascontiguousarray(verts)
        nv = verts.nbytes // layout.stride
        return self.L.orc_mesh_add_surface(self.h, mesh, bones.size, bones.ctypes.data_as(C.c_void_p), nv, verts.ctypes.data_as(C.c_void_p), C.byref(layout))

    def recalc_local_aabb(self, mesh):
        self.L.orc_mesh_recalc_local_aabb(self.h, mesh)

    def update(self):
        self.L.orc_graph_update(self.h)

    def update_hierarchical_data(self):
        self.L.orc_graph_update_hierarchical_data(self.h)

    def global_transform(self, n):
        out = np.empty(16, dtype=np.float32)
        self.L.orc_node_global_transform(self.h, n, fp(out))
        return out

    def global_transforms(self, idx=None):
        idx = range(self.capacity) if idx is None else idx
        return np.stack([self.global_transform(int(i)) for i in idx])

    def global_position(self, n):
        return self.global_transform(n)[12:15]

    def global_visibility(self, n):
        return bool(self.L.orc_node_global_visibility(self.h, n))

    def is_globally_enabled(self, n):
        return bool(self.L.orc_node_is_globally_enabled(self.h, n))

    def world_bounding_box(self, n):
        a = Aabb()
        self.L.orc_node_world_bounding_box(self.h, n, C.byref(a))
        return a.to_np()

    def world_bounding_boxes(self, idx=None):
        idx = range(self.capacity) if idx is None else idx
        return np.stack([self.world_bounding_box(int(i)) for i in idx])

    def from_graph(self, frustum: Frustum, render_mask=0xFFFFFFFF, shadow_pass=False):
        cap = self.capacity
        out = np.empty(max(cap, 1), dtype=np.uint32)
        n = self.L.orc_from_graph(self.h, C.byref(frustum) if frustum is not None else None, render_mask, int(shadow_pass), out.ctypes.data_as(C.c_void_p), cap)
        return out[:n].copy()

    def set_lod_group(self, node, levels):
        """levels = [(begin, end, [object nodes]), ...] — Base::set_lod_group with LevelOfDetail ranges."""
        b = np.array([l[0] for l in levels], np.float32)
        e = np.array([l[1] for l in levels], np.float32)
        ob_begin = np.zeros(len(levels) + 1, np.uint32)
        objs = []
        for k, l in enumerate(levels):
            objs += list(l[2])
            ob_begin[k + 1] = len(objs)
        o = np.array(objs if objs else [0], np.uint32)
        self.L.orc_node_set_lod_group(self.h, int(node), len(levels), fp(b), fp(e), ob_begin.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p))

    def lod_filter(self, translation, z_near, z_far):
        t = np.ascontiguousarray(translation, dtype=np.float32)
        out = np.empty(max(self.capacity, 1), dtype=np.uint8)
        self.L.orc_lod_filter(self.h, fp(t), float(z_near), float(z_far), out.ctypes.data_as(C.c_void_p))
        return out[: self.capacity].astype(bool)

    def from_graph_lod(self, frustum: Frustum, translation, z_near, z_far, render_mask=0xFFFFFFFF, shadow_pass=False):
        t = np.ascontiguousarray(translation, dtype=np.float32)
        cap = self.capacity
        out = np.empty(max(cap, 1), dtype=np.uint32)
        n = self.L.orc_from_graph_lod(self.h, C.byref(frustum), render_mask, int(shadow_pass), fp(t), float(z_near), float(z_far), out.ctypes.data_as(C.c_void_p), cap)
        return out[:n].copy()

    def collect_lights(self, frustum: Frustum):
        out = np.empty(max(self.capacity, 1), dtype=np.uint32)
        n = self.L.orc_collect_lights(self.h, C.byref(frustum), out.ctypes.data_as(C.c_void_p), self.capacity)
        return out[:n].copy()

    def instance(self, node, view_m16, vp_m16):
        """(sort_index, world[16], wvp[16]) of what collect_render_data / write_uniforms produce for the node."""
        v = np.ascontiguousarray(view_m16, dtype=np.float32).reshape(16)
        p = np.ascontiguousarray(vp_m16, dtype=np.float32).reshape(16)
        w = np.empty(16, dtype=np.float32)
        wvp = np.empty(16, dtype=np.float32)
        si = self.L.orc_node_instance(self.h, int(node), fp(v), fp(p), fp(w), fp(wvp))
        return int(si), w, wvp

    def bone_matrices(self, mesh, surface, n_bones):
        out = np.empty((n_bones, 16), dtype=np.float32)
        n = self.L.orc_mesh_bone_matrices(self.h, mesh, surface, fp(out.reshape(-1)))
        return out[:n]

    def skin(self, mesh, surface, n_verts):
        pos = np.empty((n_verts, 3), dtype=np.float32)
        nrm = np.empty((n_verts, 3), dtype=np.float32)
        self.L.orc_mesh_skin(self.h, mesh, surface, fp(pos.reshape(-1)), fp(nrm.reshape(-1)))
        return pos, nrm


def frustum_to_fyx(f: Frustum):
    """oracle Frustum → fyrox_b200 fyx_frustum (same numbers, product struct)."""
    from fyrox_b200 import frustum_from_numpy

    planes, corners = frustum_planes_corners(f)
    return frustum_from_numpy(planes, corners)


# ---- N2: animation (fyrox_anim_oracle.c) ------------------------------------------------------------
def curve_value_at(keys: np.ndarray, location: float, hint: int = 0):
    """Curve::value_at on a KEY_DTYPE array; returns (value, new hint)."""
    keys = np.ascontiguousarray(keys, dtype=KEY_DTYPE)
    h = C.c_uint32(hint)
    v = lib().orc_curve_value_at(keys.ctypes.data_as(C.c_void_p), len(keys), float(location), C.byref(h))
    return float(np.float32(v)), h.value


class Animation:
    """Animation<Handle<Node>> of the oracle: tracks (TRACK_DTYPE) over one key array (KEY_DTYPE)."""

    def __init__(self, tracks: np.ndarray, keys: np.ndarray, speed=1.0, looped=True, time_slice=(0.0, 0.0), time_position=0.0, enabled=True):
        self.L = lib()
        tracks = np.ascontiguousarray(tracks, dtype=TRACK_DTYPE)
        keys = np.ascontiguousarray(keys, dtype=KEY_DTYPE)
        self.h = self.L.orc_animation_new(tracks.ctypes.data_as(C.c_void_p), len(tracks), keys.ctypes.data_as(C.c_void_p), len(keys))
        self.L.orc_animation_set_speed(self.h, float(speed))
        self.L.orc_animation_set_looped(self.h, int(looped))
        self.L.orc_animation_set_time_slice(self.h, float(time_slice[0]), float(time_slice[1]))
        self.L.orc_animation_set_time_position(self.h, float(time_position))
        self.L.orc_animation_set_enabled(self.h, int(enabled))

    def __del__(self):
        try:
            if self.h:
                self.L.orc_animation_free(self.h)
                self.h = None
        except Exception:
            pass

    @property
    def time_position(self):
        return float(np.float32(self.L.orc_animation_time_position(self.h)))


def update_animations(anims, dt, graph: "Graph", transforms):
    """AnimationContainer::update_animations over a list of Animation; `transforms` is a ctypes array of Transform per node."""
    arr = (C.c_void_p * max(len(anims), 1))(*[a.h for a in anims])
    lib().orc_update_animations(arr, len(anims), float(dt), graph.h, transforms, len(transforms))


def blend_group_update(anims, weights, dt, graph: "Graph", transforms):
    """One Machine (one layer, one state, BlendAnimations over PlayAnimation sources) evaluated and applied."""
    arr = (C.c_void_p * max(len(anims), 1))(*[a.h for a in anims])
    w = np.ascontiguousarray(weights, dtype=np.float32)
    lib().orc_blend_group_update(arr, fp(w), len(anims), float(dt), graph.h, transforms, len(transforms))


# ---- "soa-omp-NT" multi-core baseline (fyrox_oracle_mt.c) ---------------------------------------------------
class MtGraph:
    """Flat-array, OpenMP form of the same arithmetic (NOT how the reference runs; see fyrox_oracle_mt.c)."""

    def __init__(self, parent, flags=None, render_mask=None, local_m16=None, local_aabb=None, root=0, threads=None):
        self.L = lib()
        n = len(parent)

        def p(a, dt):
            if a is None:
                return None, None
            a = np.ascontiguousarray(a, dtype=dt)
            return a, a.ctypes.data_as(C.c_void_p)

        keep = [p(parent, np.uint32), p(flags, np.uint32), p(render_mask, np.uint32), p(local_m16, np.float32), p(local_aabb, np.float32)]
        self.h = self.L.orc_mt_new(n, root, *[k[1] for k in keep])
        self.n = n
        if threads:
            self.L.orc_mt_set_threads(self.h, int(threads))

    def __del__(self):
        try:
            if self.h:
                self.L.orc_mt_free(self.h)
                self.h = None
        except Exception:
            pass

    def set_local_matrices(self, m16, idx=None):
        m16 = np.ascontiguousarray(m16, dtype=np.float32)
        ix = None if idx is None else np.ascontiguousarray(idx, dtype=np.uint32)
        self.L.orc_mt_set_local_matrices(self.h, m16.size // 16, None if ix is None else ix.ctypes.data_as(C.c_void_p), m16.ctypes.data_as(C.c_void_p))

    def set_inv_bind(self, n, m16):
        m = np.ascontiguousarray(m16, dtype=np.float32).reshape(16)
        self.L.orc_mt_set_inv_bind(self.h, int(n), fp(m))

    def add_surface(self, mesh, bones, verts=None, layout=ANIMATED_VERTEX):
        b = np.ascontiguousarray(bones, dtype=np.uint32)
        nv = 0 if verts is None else len(verts) // layout.stride
        vptr = None if verts is None else np.ascontiguousarray(verts, dtype=np.uint8).ctypes.data_as(C.c_void_p)
        return self.L.orc_mt_add_surface(self.h, int(mesh), len(b), b.ctypes.data_as(C.c_void_p), nv, vptr, C.byref(layout))

    def update(self):
        self.L.orc_mt_update(self.h)

    def cull(self, frustum, render_mask=0xFFFFFFFF, shadow_pass=False):
        out = np.empty(max(self.n, 1), dtype=np.uint32)
        n = self.L.orc_mt_cull(self.h, C.byref(frustum) if frustum is not None else None, render_mask, int(shadow_pass), out.ctypes.data_as(C.c_void_p), self.n)
        return out[:n].copy()

    def skin(self, surface, n_verts):
        pos = np.empty((n_verts, 3), dtype=np.float32)
        nrm = np.empty((n_verts, 3), dtype=np.float32)
        self.L.orc_mt_skin_surface(self.h, surface, fp(pos.reshape(-1)), fp(nrm.reshape(-1)))
        return pos, nrm

    def skin_all(self):
        self.L.orc_mt_skin_all(self.h)

    def get(self, i):
        g = np.empty(16, dtype=np.float32)
        a = Aabb()
        f = C.c_uint32()
        self.L.orc_mt_get(self.h, int(i), fp(g), C.byref(a), C.byref(f))
        return g, a.to_np(), f.value
