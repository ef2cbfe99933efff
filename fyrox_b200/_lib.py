"""ctypes binding of libfyrox_b200.so (include/fyrox_b200.h) and libfyrox_scenegen.so.

The libraries are built in-tree by ``fyrox_b200.build.build_all()`` (``__graft_entry__.build``).  There
is no fallback: if the CUDA library is missing, importing the compute API raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libfyrox_b200.so")
SCENEGEN_PATH = os.path.join(LIB_DIR, "libfyrox_scenegen.so")

FYX_NONE = 0xFFFFFFFF
FYX_MAX_FRUSTA = 8
FYX_MAX_BONES = 255

# status codes
FYX_OK = 0
FYX_ERR_INVALID_ARGUMENT = -1
FYX_ERR_CUDA = -2
FYX_ERR_OUT_OF_MEMORY = -3
FYX_ERR_NOT_AFFINE = -4
FYX_ERR_TOPOLOGY = -5
FYX_ERR_STATE = -6
FYX_ERR_NCCL = -7
FYX_ERR_UNSUPPORTED = -8

# node flags
NODE_VISIBILITY = 1 << 0
NODE_ENABLED = 1 << 1
NODE_FRUSTUM_CULLING = 1 << 2
NODE_CAST_SHADOWS = 1 << 3
NODE_ALIVE = 1 << 4
NODE_RENDERABLE = 1 << 5
NODE_LIGHT = 1 << 6
NODE_STATIC_BATCH = 1 << 7
NODE_REFLECTION_PROBE = 1 << 15
NODE_GLOBAL_VISIBILITY = 1 << 8
NODE_GLOBAL_ENABLED = 1 << 9
NODE_REACHABLE = 1 << 10
NODE_DEFAULT = NODE_VISIBILITY | NODE_ENABLED | NODE_FRUSTUM_CULLING | NODE_CAST_SHADOWS | NODE_ALIVE

UPDATE_INCREMENTAL = 0
UPDATE_ALL = 1
PASS_SHADOW = 1
FRAME_ASYNC = 1
FRAME_ALLGATHER = 2
FRAME_READBACK_OWN = 4
COMM_NCCL, COMM_PEER_STORES, COMM_HOST_SEGMENT, COMM_UNDECIDED = 1, 2, 4, 8

u32p = C.POINTER(C.c_uint32)
f32p = C.POINTER(C.c_float)


class fyx_config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("stream", C.c_void_p), ("flags", C.c_uint32)]


class fyx_frustum(C.Structure):
    _fields_ = [("planes", (C.c_float * 4) * 6), ("corners", (C.c_float * 3) * 8)]


class fyx_vertex_layout(C.Structure):
    _fields_ = [
        ("stride", C.c_uint32),
        ("position_offset", C.c_uint32),
        ("normal_offset", C.c_uint32),
        ("bone_weights_offset", C.c_uint32),
        ("bone_indices_offset", C.c_uint32),
    ]


class fyx_comm_stats(C.Structure):
    _fields_ = [("epoch", C.c_uint64), ("entries_own", C.c_uint64), ("entries_total", C.c_uint64), ("egress_bytes", C.c_uint64),
                ("device_ms", C.c_float), ("mode", C.c_uint32)]


class fyx_timings(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("upload_ms", "update_ms", "cull_ms", "palette_ms", "skin_ms", "readback_ms", "total_ms")]


class fyx_trs(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("rotation", C.c_float * 4), ("scale", C.c_float * 3)]


class fyx_transform_statics(C.Structure):
    _fields_ = [("pre_rotation", C.c_float * 4), ("post_rotation_matrix", C.c_float * 9), ("rotation_offset", C.c_float * 3),
                ("rotation_pivot", C.c_float * 3), ("scaling_offset", C.c_float * 3), ("scaling_pivot", C.c_float * 3)]


class fyx_frame_desc(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("update_flags", C.c_uint32),
        ("n_changed", C.c_uint32),
        ("changed_idx", C.c_void_p),
        ("changed_m16", C.c_void_p),
        ("changed_trs", C.c_void_p),
        ("changed_rot", C.c_void_p),
        ("n_frusta", C.c_uint32),
        ("frusta", C.POINTER(fyx_frustum)),
        ("cam_mask", C.c_void_p),
        ("pass_flags", C.c_void_p),
        ("do_palettes", C.c_uint32),
        ("do_skin", C.c_uint32),
        ("readback_visible", C.c_uint32),
        ("flags", C.c_uint32),
        ("do_animate", C.c_uint32),
        ("animate_dt", C.c_float),
    ]


class fyx_curve_key(C.Structure):
    _fields_ = [("location", C.c_float), ("value", C.c_float), ("kind", C.c_uint32), ("left_tangent", C.c_float), ("right_tangent", C.c_float)]


class fyx_anim_track(C.Structure):
    _fields_ = [("target_node", C.c_uint32), ("binding", C.c_uint32), ("value_kind", C.c_uint32), ("enabled", C.c_uint32),
                ("n_curves", C.c_uint32), ("first_key", C.c_uint32 * 4), ("n_keys", C.c_uint32 * 4)]


class fyx_animation_desc(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("n_tracks", C.c_uint32),
        ("tracks", C.c_void_p),
        ("n_keys", C.c_uint32),
        ("keys", C.c_void_p),
        ("speed", C.c_float),
        ("time_position", C.c_float),
        ("time_slice_start", C.c_float),
        ("time_slice_end", C.c_float),
        ("looped", C.c_uint32),
        ("enabled", C.c_uint32),
    ]


KEY_CONSTANT, KEY_LINEAR, KEY_CUBIC = 0, 1, 2
TV_REAL, TV_VECTOR2, TV_VECTOR3, TV_VECTOR4, TV_QUAT_EULER, TV_QUAT = range(6)
BIND_POSITION, BIND_SCALE, BIND_ROTATION = 0, 1, 2


class fyx_observer(C.Structure):
    _fields_ = [("translation", C.c_float * 3), ("z_near", C.c_float), ("z_far", C.c_float)]


class fyx_bundle(C.Structure):
    _fields_ = [("id", C.c_uint32), ("first", C.c_uint32), ("count", C.c_uint32), ("reserved", C.c_uint32), ("sort_index", C.c_uint64)]


class fyx_instances(C.Structure):
    _fields_ = [
        ("count", C.c_uint32),
        ("n_bundles", C.c_uint32),
        ("node", C.c_void_p),
        ("sort_index", C.c_void_p),
        ("matrices", C.c_void_p),
        ("bundles", C.c_void_p),
    ]


# every symbol include/fyrox_b200.h declares: name -> (restype, argtypes)
ctx_p = C.c_void_p
SYMBOLS = {
    "fyx_abi_version": (C.c_uint32, []),
    "fyx_create": (C.c_int32, [C.POINTER(fyx_config), C.POINTER(ctx_p)]),
    "fyx_destroy": (None, [ctx_p]),
    "fyx_last_error": (C.c_char_p, [ctx_p]),
    "fyx_sync": (C.c_int32, [ctx_p]),
    "fyx_host_alloc": (C.c_void_p, [C.c_size_t]),
    "fyx_host_free": (None, [C.c_void_p]),
    "fyx_frustum_from_view_projection_matrix": (C.c_int32, [f32p, C.POINTER(fyx_frustum)]),
    "fyx_frustum_default": (None, [C.POINTER(fyx_frustum)]),
    "fyx_mat4_mul": (None, [f32p, f32p, f32p]),
    "fyx_set_topology": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fyx_set_dfs_order": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p]),
    "fyx_set_local_matrices": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_local_trs": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_local_rotations": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_transform_statics": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_flags": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_render_masks": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_local_aabbs": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_add_skinned_surface": (
        C.c_int32,
        [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(fyx_vertex_layout), u32p],
    ),
    "fyx_reserve_skinning": (C.c_int32, [ctx_p, C.c_uint64, C.c_uint64]),
    "fyx_commit_surfaces": (C.c_int32, [ctx_p]),
    "fyx_update_transforms": (C.c_int32, [ctx_p, C.c_uint32]),
    "fyx_cull": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(fyx_frustum), C.c_void_p, C.c_void_p]),
    "fyx_update_and_cull": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.POINTER(fyx_frustum), C.c_void_p, C.c_void_p]),
    "fyx_get_visible": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(u32p), u32p]),
    "fyx_get_visible_device": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "fyx_set_lod_ranges": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_set_observers": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p]),
    "fyx_cull_lights": (C.c_int32, [ctx_p]),
    "fyx_select_reflection_probes": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p]),
    "fyx_get_visible_lights": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(u32p), u32p]),
    "fyx_build_palettes": (C.c_int32, [ctx_p]),
    "fyx_skin": (C.c_int32, [ctx_p]),
    "fyx_render_prep": (C.c_int32, [ctx_p, C.POINTER(fyx_frame_desc)]),
    "fyx_frame_wait": (C.c_int32, [ctx_p]),
    "fyx_get_global_matrices": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_get_world_aabbs": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_get_global_flags": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_get_palette": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p]),
    "fyx_get_skinned": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_get_skinned_device": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "fyx_get_timings": (C.c_int32, [ctx_p, C.POINTER(fyx_timings)]),
    "fyx_kernel_launch_count": (C.c_uint64, [ctx_p]),
    "fyx_anim_add": (C.c_int32, [ctx_p, C.POINTER(fyx_animation_desc), u32p]),
    "fyx_anim_clear": (C.c_int32, [ctx_p]),
    "fyx_anim_set_enabled": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32]),
    "fyx_anim_set_track_enabled": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "fyx_anim_set_speed": (C.c_int32, [ctx_p, C.c_uint32, C.c_float]),
    "fyx_anim_set_time_position": (C.c_int32, [ctx_p, C.c_uint32, C.c_float]),
    "fyx_anim_get_time_positions": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "fyx_anim_blend_group": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p, u32p]),
    "fyx_anim_set_blend_weights": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "fyx_animate": (C.c_int32, [ctx_p, C.c_float]),
    "fyx_set_bundle_ids": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_enable_instances": (C.c_int32, [ctx_p, C.c_uint32]),
    "fyx_pack_instances": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "fyx_get_instances": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(fyx_instances)]),
    "fyx_get_instances_device": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(fyx_instances)]),
    "fyx_comm_get_unique_id": (C.c_int32, [C.c_void_p]),
    "fyx_comm_init": (C.c_int32, [ctx_p, C.c_int32, C.c_int32, C.c_void_p]),
    "fyx_set_node_surfaces": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fyx_get_instance_surfaces": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(u32p)]),
    "fyx_pack_bone_matrices": (C.c_int32, [ctx_p, C.c_uint32]),
    "fyx_get_bone_matrix_block": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32)]),
    "fyx_get_bone_matrix_blocks_device": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p]),
    "fyx_set_blend_shapes": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]),
    "fyx_set_blend_shape_weights": (C.c_int32, [ctx_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "fyx_set_skinned_tangents": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32]),
    "fyx_get_skinned_tangents": (C.c_int32, [ctx_p, C.c_uint32, C.c_void_p]),
    "fyx_get_skinned_tangents_device": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(C.c_void_p)]),
    "fyx_allgather_visible": (C.c_int32, [ctx_p]),
    "fyx_comm_mode": (C.c_uint32, [ctx_p]),
    "fyx_comm_get_stats": (C.c_int32, [ctx_p, C.c_void_p]),
    "fyx_get_visible_gathered": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(u32p), u32p]),
    "fyx_get_visible_gathered_device": (C.c_int32, [ctx_p, C.c_uint32, C.POINTER(C.c_void_p), u32p]),
}

_lib = None
_sg = None


def load() -> C.CDLL:
    """Load libfyrox_b200.so; raises (no fallback) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the render-prep path)"
            )
        lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class sg_config(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("n_nodes", C.c_uint32),
        ("n_units", C.c_uint32),
        ("bones_per_unit", C.c_uint32),
        ("verts_per_unit", C.c_uint32),
        ("rank", C.c_int32),
        ("nranks", C.c_int32),
    ]


SG_SYMBOLS = {
    "sg_create": (C.c_void_p, [C.POINTER(sg_config)]),
    "sg_free": (None, [C.c_void_p]),
    "sg_set_threads": (None, [C.c_int]),
    "sg_capacity": (C.c_uint32, [C.c_void_p]),
    "sg_n_renderable": (C.c_uint32, [C.c_void_p]),
    "sg_parent": (u32p, [C.c_void_p]),
    "sg_flags": (u32p, [C.c_void_p]),
    "sg_render_mask": (u32p, [C.c_void_p]),
    "sg_local_m16": (f32p, [C.c_void_p]),
    "sg_local_aabb": (f32p, [C.c_void_p]),
    "sg_global_index": (u32p, [C.c_void_p]),
    "sg_n_units": (C.c_uint32, [C.c_void_p]),
    "sg_unit_mesh_node": (C.c_uint32, [C.c_void_p, C.c_uint32]),
    "sg_unit_bone_nodes": (u32p, [C.c_void_p, C.c_uint32]),
    "sg_unit_inv_bind": (f32p, [C.c_void_p, C.c_uint32]),
    "sg_unit_vertices": (None, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "sg_units_vertices": (None, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "sg_animate": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "sg_animate_trs": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
}


def load_scenegen() -> C.CDLL:
    global _sg
    if _sg is None:
        if not os.path.exists(SCENEGEN_PATH):
            raise RuntimeError(f"{SCENEGEN_PATH} is missing: run __graft_entry__.build()")
        lib = C.CDLL(SCENEGEN_PATH)
        for name, (res, args) in SG_SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _sg = lib
    return _sg
